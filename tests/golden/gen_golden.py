#!/usr/bin/env python3
"""Generates tests/golden/literal_spec.json by EXECUTING THE REFERENCE'S OWN python blocks
(pos-evolution.md of ethereum/pos-evolution, loaded by tests/ref_blocks.py -- never copied) on the minimal preset.
The document is not part of this repository, so these vectors pin the oracle (tests/test_golden.py and
tests/test_oracle_literal_spec.py, CPU) and the CUDA path (tests/test_golden.py -m gpu) to what the reference's text computes.
    python tests/golden/gen_golden.py path/to/pos-evolution.md"""
import copy
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import literal  # noqa: E402
import ref_blocks  # noqa: E402
import scenarios  # noqa: E402
from oracle import spec as S  # noqa: E402


def att_json(att):
    d = att.data
    return {"bits": [bool(b) for b in att.aggregation_bits], "slot": d.slot, "index": d.index, "beacon_block_root": d.beacon_block_root.hex(),
            "source": [d.source.epoch, d.source.root.hex()], "target": [d.target.epoch, d.target.root.hex()], "signature": att.signature.hex()}


def main():
    spec, state = scenarios.minimal_state(64, slot=9)
    ns = literal.namespace(spec)
    out = {"preset": "minimal", "n_validators": 64, "state_slot": 9, "generator": "tests/golden/gen_golden.py (reference blocks executed literally)"}
    out["pubkeys"] = [v.pubkey.hex() for v in state.validators]
    # shuffle (ref :513-534)
    out["shuffle"] = []
    for n, tag in ((1, b"a"), (2, b"b"), (37, b"c"), (257, b"e"), (256, b"d"), (1000, b"f")):
        seed = hashlib.sha256(tag).digest()
        out["shuffle"].append({"n": n, "seed": seed.hex(), "rounds": 10,
                               "perm": [int(ns["compute_shuffled_index"](ns["uint64"](i), ns["uint64"](n), seed)) for i in range(n)]})
    # committees of epochs 0 and 1 (ref :461-504 + get_beacon_committee)
    out["committees"] = {}
    for slot in range(0, 16):
        for idx in range(2):
            out["committees"]["%d/%d" % (slot, idx)] = [int(v) for v in ns["get_beacon_committee"](state, slot, idx)]
    out["committee_count_per_slot"] = {str(e): int(ns["get_committee_count_per_slot"](state, e)) for e in (0, 1)}
    out["attester_seed"] = {str(e): ns["get_seed"](state, e, S.DOMAIN_BEACON_ATTESTER).hex() for e in (0, 1)}
    # process_attestation (ref :722-754)
    bad_idx = scenarios.make_attestation(spec, state, 8, 0)
    bad_idx.data = S.AttestationData(8, 2, bad_idx.data.beacon_block_root, bad_idx.data.source, bad_idx.data.target)
    cases = [
        ("valid_full", scenarios.make_attestation(spec, state, 8, 0)),
        ("valid_partial", scenarios.make_attestation(spec, state, 8, 1, bits=[True, False, True, False])),
        ("valid_prev_epoch", scenarios.make_attestation(spec, state, 5, 1)),
        ("bad_sig_bitflip", scenarios.make_attestation(spec, state, 8, 0, corrupt="flip_bit")),
        ("bad_wrong_message", scenarios.make_attestation(spec, state, 8, 0, corrupt="wrong_message")),
        ("bad_wrong_signers", scenarios.make_attestation(spec, state, 8, 1, corrupt="wrong_signer_set")),
        ("bad_empty_bits", scenarios.make_attestation(spec, state, 8, 0, bits=[False] * 4)),
        ("bad_bits_length", scenarios.make_attestation(spec, state, 8, 0, bits=[True] * 3)),
        ("bad_committee_index", bad_idx),                                                 # index >= committee count
    ]
    out["process_attestation"] = []
    for name, att in cases:
        st = copy.deepcopy(state)
        try:
            ns["process_attestation"](st, att)
            res = {"result": "ok", "balances": st.balances, "current_epoch_participation": st.current_epoch_participation,
                   "previous_epoch_participation": st.previous_epoch_participation}
        except AssertionError:
            res = {"result": "assert"}
        dom = spec.get_domain(state, S.DOMAIN_BEACON_ATTESTER, att.data.target.epoch)
        res.update(name=name, attestation=att_json(att), signing_root=spec.compute_signing_root(att.data, dom).hex())
        out["process_attestation"].append(res)
    # the first attestation included twice: its flags are already set, so the second inclusion pays no reward
    st = copy.deepcopy(state)
    ns["process_attestation"](st, cases[0][1])
    first = list(st.balances)
    ns["process_attestation"](st, cases[0][1])
    out["process_attestation_twice"] = {"name": cases[0][0], "balances_after_first": first, "balances_after_second": list(st.balances)}
    # get_head (ref :1102-1116) on a 200-block store
    st2 = copy.deepcopy(state)
    st2.validators[5].exit_epoch = 0
    store, parent, slot, roots, leaf_viable, rb = scenarios.small_store(spec, st2)
    out["get_head"] = {
        "n_blocks": len(rb), "tree_seed": 3, "inactive_validator": 5, "equivocating": sorted(store.equivocating_indices),
        "proposer_boost_root": store.proposer_boost_root.hex(),
        "latest_messages": {str(v): [m.epoch, m.root.hex()] for v, m in store.latest_messages.items()},
        "head": ns["get_head"](store).hex(),
        "weights": {rb[b].hex(): spec.get_latest_attesting_balance(store, rb[b]) for b in range(0, len(rb), 9)},
    }
    # update_latest_messages (ref :963-979) on a 50-block store: the latest messages after scenarios.LMD_UPDATES, by block index
    store, parent, slot, roots, leaf_viable, rb = scenarios.small_store(spec, state, n_blocks=50)
    for epoch, blk, idxs in scenarios.LMD_UPDATES:
        att = S.Attestation([], S.AttestationData(0, 0, rb[blk], S.Checkpoint(), S.Checkpoint(epoch, rb[0])), b"")
        ns["update_latest_messages"](store, idxs, att)
    idx_of = {r: i for i, r in enumerate(rb)}
    out["update_latest_messages"] = {"n_blocks": len(rb), "tree_seed": 3,
                                     "latest_messages": {str(v): [m.epoch, idx_of[m.root]] for v, m in sorted(store.latest_messages.items())}}
    # FFG accounting (ref :793-852): the reference's text executed on 80 generated end-of-epoch states (scenarios.ffg_case(seed))
    out["ffg"] = []
    for seed in range(80):
        st = scenarios.ffg_case(copy.deepcopy(state), seed)
        ns["process_justification_and_finalization"](st)
        out["ffg"].append(dict(scenarios.ffg_outcome(st), seed=seed))
    with open(os.path.join(HERE, "literal_spec.json"), "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote literal_spec.json")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    ref_blocks.REF_MD = sys.argv[1]
    main()
