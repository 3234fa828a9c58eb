"""Load the reference's own fenced ```python blocks from pos-evolution.md (ethereum/pos-evolution; never
copied into the repo) so they can be executed against the oracle's restated helpers.  Used by
tests/golden/gen_golden.py, which records what they compute; the tests replay those vectors."""
import __future__
import re

REF_MD = None      # path of pos-evolution.md, set by the caller


def fenced_blocks():
    """-> list of (first_line_number, source) for every ```python block."""
    out, cur, start = [], None, 0
    with open(REF_MD, encoding="utf-8") as f:
        for no, line in enumerate(f, 1):
            if cur is None:
                if line.strip().startswith("```python"):
                    cur, start = [], no + 1
            elif line.strip().startswith("```"):
                out.append((start, "".join(cur)))
                cur = None
            else:
                cur.append(line)
    return out


def function_source(name: str, occurrence: int = 0) -> str:
    """Source text of ``def name`` (whole function) from the fenced blocks."""
    hits = []
    for _, src in fenced_blocks():
        m = re.search(r"^def %s\(" % re.escape(name), src, re.M)
        if m:
            body = src[m.start():]
            # cut at the next top-level statement
            lines = body.split("\n")
            keep = [lines[0]]
            in_sig = not lines[0].rstrip().endswith(":")
            for ln in lines[1:]:
                if in_sig:
                    keep.append(ln)
                    if ln.rstrip().endswith(":"):
                        in_sig = False
                    continue
                if ln.strip() == "" or ln.startswith((" ", "\t")):
                    keep.append(ln)
                else:
                    break
            hits.append("\n".join(keep))
    return hits[occurrence]


def exec_functions(names, namespace: dict):
    """exec the reference definitions of ``names`` inside ``namespace`` (annotations unevaluated)."""
    for n in names:
        occ = 0
        if isinstance(n, tuple):
            n, occ = n
        code = compile(function_source(n, occ), "%s:%s" % (REF_MD, n), "exec",
                       flags=__future__.annotations.compiler_flag, dont_inherit=True)
        exec(code, namespace)
    return namespace
