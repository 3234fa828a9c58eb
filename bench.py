#!/usr/bin/env python3
"""bench.py -- headline benchmark of BASELINE.json:
    "attestations aggregated+verified/sec at 1M validators; get_head p50 latency".

One step = one full epoch of 2^20 validators (BASELINE.json configs[4]: 32 slots x 64 committees x 512 members):
bls.Aggregate of the 1 048 576 individual G2 signatures into 2 048 aggregates, FastAggregateVerify of the 2 048 aggregates
(registry-indexed pubkey gather staged through TMA, hash-to-G2, pairing), update_latest_messages for the accepted ones,
vote-weight scatter, get_head on a 10 000-block tree.

Multi-GPU (`--gpus N`, one rank per GPU under torchrun):
  --scaling strong (default)  ONE 2^20-validator epoch per step for the whole box -- north_star's configs 4/5.  Rank g owns the
        aggregates of slots [32g/N, 32(g+1)/N) and only THEIR individual signatures; the registry, the committees and the LMD
        table are replicated.  Exchange per epoch: one all-gather of (aggregate signature, verdict) per aggregate, then every
        rank applies update_latest_messages for all accepted aggregates; get_head: rank g scatters the votes of validators
        [gN.., (g+1)N..), one u64[10 000] all-reduce, head on every rank.  `value` = 2^20 / step: total work is fixed.
  --scaling weak              every rank owns its OWN 2^20 validators and epoch (N x 2^20 overall); the only exchange is the
        vote-weight all-reduce.  `value` = N * 2^20 / step.
`value`  = attestations/s with every input resident in HBM, K epochs through the software pipeline (EpochProcessor.submit_dev;
all K results complete inside the timed region); `e2e` = the same through EpochProcessor.submit_host with pinned HOST buffers
(H2D of this rank's signatures + the epoch's bits/messages and D2H of verdicts, head AND aggregate signatures of every epoch
inside the timed region); `ms_per_step_unpipelined` = one epoch at a time (process_epoch_dev).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--scaling strong|weak]     # this repo, on the GPU(s)
    python bench.py --impl reference [...]                                          # the CPU oracle (pyspec/py_ecc-class path)
"""
import os
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")     # 8 pipeline slots x 3 streams: must precede the first CUDA call
import argparse
import hashlib
import json
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "attestations aggregated+verified/sec at 1M validators; get_head p50 latency"
UNIT = "attestations/s"
N_VAL = 1 << 20
SLOTS, COMMITTEES_PER_SLOT, COMMITTEE_SIZE = 32, 64, 512
N_AGG = SLOTS * COMMITTEES_PER_SLOT
N_BLOCKS = 10000
R_ORDER = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
TRAFFIC_BYTES_K3 = 1.40e9      # dram read 0.17 GB + write 1.23 GB per k_g2_decompress launch (affine points + window-table evictions), ncu r1c capture
WORKLOAD = "full epoch: 32 slots x 64 committees x 512 members = 2^20 validators per rank; 10000-block fork tree"


def _h(b):
    return hashlib.sha256(b).digest()


# ----------------------------------------------------------------------------- CPU legs (the only users of oracle/)
def _cpu_one_committee(args):
    """bls.Aggregate of the individual signatures + FastAggregateVerify, pure-Python oracle, one committee."""
    from oracle import bls_sig as B
    pks, sigs, msg = args
    t0 = time.perf_counter()
    agg = B.Aggregate(sigs)
    ok = B.FastAggregateVerify(pks, msg, agg)
    return time.perf_counter() - t0, bool(ok), bytes(agg)


def _cpu_make_committee(tag):
    from oracle import synth
    return synth.committee(tag, COMMITTEE_SIZE)


def cpu_sample(pool, cores, committees):
    """Time `committees` (list of (pks, sigs, msg)) over the worker pool; -> (attestations/s, wall seconds, aggregate bytes)."""
    t0 = time.perf_counter()
    res = pool.map(_cpu_one_committee, committees)
    wall = time.perf_counter() - t0
    assert all(ok for _, ok, _ in res), "oracle rejected a valid synthetic aggregate"
    return len(committees) * COMMITTEE_SIZE / wall, wall, [a for _, _, a in res]


def host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args):
    """--impl reference: the CPU implementation of the same path (oracle = restated pyspec + py_ecc-class big-int
    arithmetic; the reference itself is Markdown and cannot be imported -- DESIGN.md), all host cores."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = min(host_cores(), 64)
    with mp.get_context("fork").Pool(cores) as pool:
        committees = pool.map(_cpu_make_committee, range(cores))
        for _ in range(args.warmup):
            cpu_sample(pool, cores, committees[:cores])
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cpu_sample(pool, cores, committees)
        wall = time.perf_counter() - t0
    value = args.steps * cores * COMMITTEE_SIZE / wall
    sample = "%d committees x %d members per step (1 per core): bls.Aggregate + FastAggregateVerify" % (cores, COMMITTEE_SIZE)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * wall / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "python int (381-bit Fp, the oracle's arbitrary-precision arithmetic)",
        "data": "synthetic", "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "cpu_model": cpu_model(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU arm
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.idx = gpu_index
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for ln in self.f.read().strip().splitlines():
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


def build_world(eng, rank, np, PS, shard=None):
    """Everything untimed: keys, registry, real 90-round committee shuffle, messages, individual signatures (all made
    with the product's own kernels -- bls.SkToPk / bls.Sign on the GPU), fork tree and a pre-existing LMD table.
    shard=(g, world): the SAME world on every rank (one validator set, seeded as rank 0), with the individual signatures of
    this rank's aggregates only (W["sigs"] = rows [m0, m1) of the epoch's signature array)."""
    t0 = time.time()
    seed_rank = 0 if shard is not None else rank
    sk0 = (int.from_bytes(_h(b"b200pos/sk0"), "big") + seed_rank * (1 << 200)) % (R_ORDER >> 1) or 1
    delta = int.from_bytes(_h(b"b200pos/skd"), "big") >> 64             # 192-bit step: sk0 + i*delta < r for i < 2^20
    sk_bytes = b"".join((sk0 + i * delta).to_bytes(32, "little") for i in range(N_VAL))
    sk8 = np.frombuffer(sk_bytes, dtype=np.uint32).reshape(N_VAL, 8)
    pk = eng.sk_to_pk(sk8)
    rng = np.random.default_rng(4 + seed_rank)
    eff = np.where(rng.random(N_VAL) < 0.9, 32, rng.integers(16, 33, size=N_VAL)).astype(np.uint64) * np.uint64(10**9)
    active = np.ones(N_VAL, dtype=np.uint8)
    valid = eng.registry_load(pk, eff, active)
    assert int(valid.sum()) == N_VAL
    seed = _h(b"b200pos/epoch-seed" + seed_rank.to_bytes(8, "little"))
    perm = eng.shuffle_committees(seed, N_VAL, 90)                      # compute_shuffled_index for all i (pos-evolution.md:513-534), on the GPU
    members = perm.astype(np.uint32)                                    # active set = all validators, committee k = members[512k : 512k+512]
    off = (np.arange(N_AGG + 1, dtype=np.uint64) * COMMITTEE_SIZE).astype(np.uint32)
    msgs = np.frombuffer(b"".join(_h(b"b200pos/signing-root" + seed_rank.to_bytes(4, "little") + a.to_bytes(4, "little")) for a in range(N_AGG)),
                         dtype=np.uint8).reshape(N_AGG, 32).copy()
    msg_idx = np.repeat(np.arange(N_AGG, dtype=np.uint32), COMMITTEE_SIZE)
    if shard is not None:
        g, world = shard
        a0, a1 = g * N_AGG // world, (g + 1) * N_AGG // world
        m0, m1 = int(off[a0]), int(off[a1])
    else:
        m0, m1 = 0, N_VAL
    sigs = eng.sign(np.ascontiguousarray(sk8[members[m0:m1]]), msg_idx[m0:m1], msgs)   # signature j belongs to member j
    # fork tree (SURVEY.md section 8d config 4) -- same on every rank
    trng = np.random.default_rng(4)
    parent = np.zeros(N_BLOCKS, dtype=np.uint32)
    slot = np.zeros(N_BLOCKS, dtype=np.uint64)
    back = trng.geometric(0.7, size=N_BLOCKS) - 1
    skip = trng.binomial(2, 0.1, size=N_BLOCKS)
    for i in range(1, N_BLOCKS):
        parent[i] = max(0, i - 1 - int(back[i]))
        slot[i] = slot[parent[i]] + 1 + int(skip[i])
    roots = np.frombuffer(b"".join(_h(i.to_bytes(8, "little")) for i in range(N_BLOCKS)), dtype=np.uint8).reshape(N_BLOCKS, 32)
    leaf_viable = (trng.random(N_BLOCKS) >= 0.05).astype(np.uint8)
    eng.tree_load(parent, slot, roots, leaf_viable)
    msg_block = (N_BLOCKS - 1 - np.minimum(N_BLOCKS - 1, rng.geometric(0.002, size=N_VAL))).astype(np.uint32)
    has_msg = (rng.random(N_VAL) >= 0.01).astype(np.uint8)
    equiv = (rng.random(N_VAL) < 0.001).astype(np.uint8)
    eng.latest_messages_load(np.ones(N_VAL, dtype=np.uint64), msg_block, has_msg, equiv)
    boost = (N_VAL // 32) * (int(eff.astype(object).sum()) // N_VAL) * 40 // 100
    return dict(pk=pk, members=members, off=off, msgs=msgs, sigs=sigs, boost=boost, setup_s=time.time() - t0, sk0=sk0, delta=delta,
                tree=(parent, roots, leaf_viable), votes=(msg_block, has_msg, equiv, eff, active))


def committee_secret_sum(W, a, bits_row=None):
    """sum of the secret keys of the selected members of committee a (mod r): sk_i = sk0 + i*delta, so the aggregate signature of
    the committee must equal Sign(that sum, msg_a) and its aggregate pubkey SkToPk(that sum) -- the linearity check of SURVEY 8(d)."""
    m = W["members"][int(W["off"][a]):int(W["off"][a + 1])]
    if bits_row is not None:
        m = [int(v) for j, v in enumerate(m) if (int(bits_row[j >> 3]) >> (j & 7)) & 1]
    return (len(m) * W["sk0"] + W["delta"] * sum(int(v) for v in m)) % R_ORDER


def participation_case(eng, W, np, frac, seed, corrupt_frac=0.01):
    """BASELINE.json config 3 input at participation `frac`: random aggregation bits, the matching aggregate signatures
    (bls.Aggregate of the SELECTED individual signatures, on the GPU), then `corrupt_frac` of the aggregates corrupted by
    flipping one aggregation bit (the signature no longer matches the selected set).  -> (bits, agg_sigs, expected verdicts)."""
    rng = np.random.default_rng(seed)
    nbytes = COMMITTEE_SIZE // 8
    if frac >= 1.0:
        bits = np.full((N_AGG, nbytes), 0xFF, dtype=np.uint8)
    else:
        sel = rng.random((N_AGG, COMMITTEE_SIZE)) < frac
        sel[:, 0] = True                                                       # no empty aggregate (that is a separate, tested, case)
        bits = np.packbits(sel, axis=1, bitorder="little")
    sel = np.unpackbits(bits, axis=1, bitorder="little").astype(bool)
    seg_off = np.concatenate([[0], np.cumsum(sel.sum(axis=1))]).astype(np.uint32)
    agg, st = eng.aggregate(W["sigs"][sel.reshape(-1)], seg_off)
    assert not st.any()
    expect = np.ones(N_AGG, dtype=np.uint8)
    bad = rng.choice(N_AGG, size=max(1, int(corrupt_frac * N_AGG)), replace=False)
    for a in bad:
        j = int(rng.integers(1, COMMITTEE_SIZE))
        bits[a, j >> 3] ^= np.uint8(1 << (j & 7))
        expect[a] = 0
    return bits, agg, expect


def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from pos_evolution_b200 import spec as PS
    from pos_evolution_b200.engine import Engine
    from pos_evolution_b200.epoch import EpochProcessor

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this benchmark has no CPU path (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    strong = args.scaling == "strong"
    shard = (rank, world) if (strong and world > 1) else None
    if args.emulate_world > 1:                          # tuning aid: ONE rank's share of an epoch sharded over emulate_world ranks, no collectives
        assert world == 1
        shard = (0, args.emulate_world)
    eff_world = args.emulate_world if args.emulate_world > 1 else world
    # depth / how many epochs at the end of a batch take the short-latency tail: tuned on 1, 2 and 8 GPUs and with --emulate-world
    # (profiles/r2c_sweep_*.json, r2d_emu_*.json)
    depth_default, team_last_default = {1: (3, 1), 2: (4, 1), 4: (8, 3)}.get(eff_world, (12, 4)) if strong else (3, 1)
    depth = args.depth or depth_default
    eng = Engine(local)
    if args.rlc:
        eng.set_verify_mode(True)                      # FastAggregateVerify in random-linear-combination batches (fresh os.urandom seed)
    W = build_world(eng, rank, np, PS, shard=shard)
    ep = EpochProcessor(eng, N_AGG, N_VAL, COMMITTEE_SIZE // 8, N_BLOCKS, process_group=pg, device=dev, depth=depth, shard=shard, n_validators=N_VAL,
                        tail_form=args.tail_form)
    ep.set_committees(W["members"], W["off"])
    ep.team_last = args.team_last if args.team_last is not None else team_last_default
    n_loc_sig = ep.n_sig_loc                                 # individual signatures this rank aggregates per step
    bits_np = np.full((N_AGG, COMMITTEE_SIZE // 8), 0xFF, dtype=np.uint8)
    blk_np = (N_BLOCKS - 1 - (np.arange(N_AGG) % 64)).astype(np.int32)
    d_sigs = torch.as_tensor(W["sigs"], device=dev)
    d_bits = torch.as_tensor(bits_np, device=dev)
    d_msgs = torch.as_tensor(W["msgs"], device=dev)
    d_epoch = torch.full((N_AGG,), 2, dtype=torch.int64, device=dev)
    d_blk = torch.as_tensor(blk_np, device=dev)
    h_sigs = torch.as_tensor(W["sigs"]).pin_memory()
    h_bits = torch.as_tensor(bits_np).pin_memory()
    h_msgs = torch.as_tensor(W["msgs"]).pin_memory()
    h_epochs = [torch.full((N_AGG,), 1000, dtype=torch.int64).pin_memory() for _ in range(depth + 2)]
    host_epoch_counter = [0]
    h_blk = torch.as_tensor(blk_np).pin_memory()
    boost_idx, boost = N_BLOCKS - 1, W["boost"]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_sync():
        d_epoch.add_(1)                                # a later target epoch each step, so update_latest_messages really writes
        return ep.process_epoch_dev(d_sigs, d_bits, d_msgs, d_epoch, d_blk, 0, boost_idx, boost)

    def run_pipelined_dev(n):
        """n epochs through the software pipeline; every epoch's result is complete (for the current stream) when this returns."""
        results = []
        for i in range(n):
            d_epoch.add_(1)
            t = ep.submit_dev(d_sigs, d_bits, d_msgs, d_epoch, d_blk, 0, boost_idx, boost, last=ep.drain_hint(n - 1 - i))
            if t is not None:
                results.append(t)
        results.extend(ep.drain())
        return results

    def run_pipelined_host(n):
        results = []
        for i in range(n):
            host_epoch_counter[0] += 1
            he = h_epochs[host_epoch_counter[0] % len(h_epochs)]   # a pinned buffer is rewritten only after the epoch that read it has completed
            he.fill_(1000 + host_epoch_counter[0])
            t = ep.submit_host(h_sigs, h_bits, h_msgs, he, h_blk, 0, boost_idx, boost, last=ep.drain_hint(n - 1 - i))
            if t is not None:
                results.append(t.wait())               # host blocks on the D2H of the epoch submitted depth-1 calls ago
        for t in ep.drain():
            results.append(t.wait())
        return results

    # ---- warm-up, correctness gate: every aggregate of the WHOLE epoch must verify on every rank, every rank must see the
    # same head (synchronous and pipelined forms)
    for _ in range(max(args.warmup, 3)):
        ok, head = step_sync()
    barrier()
    n_expect = N_AGG if args.emulate_world <= 1 else ep.n_loc       # (an emulated rank sees only its own verdicts)
    assert int(ok.sum().item()) == n_expect, "GPU rejected valid aggregates"
    head0 = int(head.item())
    if world > 1:
        hh = torch.tensor([head0, -head0], dtype=torch.int64, device=dev)
        dist.all_reduce(hh, op=dist.ReduceOp.MAX)
        assert int(hh[0]) == head0 and int(hh[1]) == -head0, "ranks disagree on the head"
    for t in run_pipelined_dev(depth):
        okp, headp = t.wait()
        assert int(okp.sum().item()) == n_expect and headp == head0, "pipelined epoch disagrees with the synchronous one"
    agg_sig_gpu = ep.d_agg_sig[(ep.k - 1) % depth].cpu().numpy()          # bls.Aggregate's result of the last epoch, all 2 048 committees

    # ---- synchronous form (one epoch at a time), for reference
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_sync = min(args.steps, 5)
    barrier()
    ev0.record()
    for _ in range(n_sync):
        step_sync()
    ev1.record()
    barrier()
    ms_sync = ev0.elapsed_time(ev1) / n_sync

    # ---- timed region 1: device-resident inputs, software-pipelined epochs (all K results complete inside the region)
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = eng.launch_count
    barrier()
    ev0.record()
    timed_results = run_pipelined_dev(args.steps)
    ev1.record()
    barrier()
    ms_dev = ev0.elapsed_time(ev1) / args.steps
    launches = (eng.launch_count - launches0) // args.steps
    clocks = sampler.stop()
    if args.dump_outputs:
        # what submit_dev's caller receives for the last timed epoch, copied now: later epochs reuse the pipeline slots
        ok_last, head_last = timed_results[-1].wait()
        dump = {"verdicts": ok_last.cpu().numpy().astype(np.float32),
                "head_index": np.array([head_last], dtype=np.float64),
                "aggregate_signatures": timed_results[-1].aggregate_signatures().cpu().numpy().astype(np.float32)}

    # ---- timed region 2: end to end through the public host API (pinned host buffers; H2D of every epoch's inputs and D2H of
    # its verdicts + head + aggregate signatures inside the region; copies of epoch k+1 overlap with the compute of epoch k)
    res = run_pipelined_host(depth)
    assert all(int(o.sum()) == n_expect for o, _ in res)
    barrier()
    ev0.record()
    res = run_pipelined_host(args.steps)
    ev1.record()
    barrier()
    ms_e2e = ev0.elapsed_time(ev1) / args.steps
    assert len(res) == args.steps and all(int(o.sum()) == n_expect and hd == res[0][1] for o, hd in res)
    assert np.array_equal(ep.h_agg_sig[(ep.k - 1) % depth].numpy(), agg_sig_gpu), "host copy of the aggregate signatures differs"

    # ---- dominant kernel alone (roofline): stage 1+2 of bls.Aggregate on this rank's signatures
    reps = 3
    d_off_loc, d_members_loc = ep.d_off_loc, ep.d_members_loc
    d_bits_loc, d_msgs_loc = d_bits[ep.a0:ep.a1], d_msgs[ep.a0:ep.a1]
    t_aggsig = torch.zeros((ep.n_loc, 96), dtype=torch.uint8, device=dev)
    t_aggst = torch.zeros(ep.n_loc, dtype=torch.int32, device=dev)
    t_ok = torch.zeros(ep.n_loc, dtype=torch.uint8, device=dev)

    def timed(fn, n=reps, flush=None):
        """mean ms of fn() over n launches, timed one by one with CUDA events on torch's current stream (the stream the *_dev
        entry points launch on); flush() (untimed) runs before each"""
        tot = []
        for _ in range(n):
            if flush is not None:
                flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            tot.append(e0.elapsed_time(e1))
        return sum(tot) / len(tot), min(tot)

    ms_agg, _ = timed(lambda: eng.aggregate_dev(d_sigs, d_off_loc, t_aggsig, t_aggst))
    ms_verify, _ = timed(lambda: eng.fast_aggregate_verify_dev(d_members_loc, d_off_loc, d_bits_loc, d_msgs_loc, t_aggsig, t_ok))
    assert int(t_ok.sum().item()) == ep.n_loc

    # ---- the pubkey gather stage alone (north_star: >= 60 % of the HBM-read roofline on the pubkey gather).  Registry 100.7 MB <
    # 126 MB L2, so the cold number needs an L2 flush (a 512 MB memset) before every launch; the warm number is reported beside it.
    d_chk = torch.zeros(ep.n_loc, dtype=torch.int32, device=dev)
    d_chk2 = torch.zeros(ep.n_loc, dtype=torch.int32, device=dev)
    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    flush = lambda: flush_buf.zero_()                                     # noqa: E731
    g_tma_cold, g_tma_cold_min = timed(lambda: eng.gather_probe_dev(d_members_loc, d_off_loc, d_bits_loc, d_chk, tma=True), 10, flush)
    g_ldg_cold, g_ldg_cold_min = timed(lambda: eng.gather_probe_dev(d_members_loc, d_off_loc, d_bits_loc, d_chk2, tma=False), 10, flush)
    g_tma_warm, _ = timed(lambda: eng.gather_probe_dev(d_members_loc, d_off_loc, d_bits_loc, d_chk, tma=True), 10)
    assert torch.equal(d_chk, d_chk2), "TMA-staged and plain-load gathers fetched different records"
    del flush_buf

    ms_overlap = None
    if args.probe_overlap:
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        ks0, ks1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ks0.record()
        for _ in range(reps):
            s1.wait_stream(torch.cuda.current_stream())
            s2.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s1):
                eng.aggregate_dev(d_sigs, d_off_loc, t_aggsig, t_aggst)
            with torch.cuda.stream(s2):
                eng.fast_aggregate_verify_dev(d_members_loc, d_off_loc, d_bits_loc, d_msgs_loc, ep.d_agg_sig[0][ep.a0:ep.a1], t_ok)
            torch.cuda.current_stream().wait_stream(s1)
            torch.cuda.current_stream().wait_stream(s2)
        ks1.record()
        torch.cuda.synchronize()
        ms_overlap = ks0.elapsed_time(ks1) / reps

    # ---- BASELINE.json configs 2 and 3 as SURVEY.md 8(d) defines them (single GPU): bls.Aggregate of 32 768 signatures -> 64
    # segments; FastAggregateVerify of 2 048 x 512 at 100 % / 99 % / 50 % participation with 1 % corrupted aggregates
    cfg = {}
    if world == 1 and not args.no_extra_configs:
        n2 = 64 * COMMITTEE_SIZE
        d_off2 = ep.d_off[:65].contiguous()
        ms_c2, _ = timed(lambda: eng.aggregate_dev(d_sigs[:n2], d_off2, t_aggsig[:64], t_aggst[:64]), 5)
        assert np.array_equal(t_aggsig[:64].cpu().numpy(), agg_sig_gpu[:64])
        cfg["config2_bls_aggregate_32768_sigs_64_segments"] = {"ms": ms_c2, "signatures_per_s": n2 / (ms_c2 * 1e-3),
                                                                "algorithmic_bytes": 96 * n2 + 96 * 64, "GBps": (96 * n2 + 96 * 64) / (ms_c2 * 1e-3) / 1e9}
        for name, frac, seed in (("100pct", 1.0, 0), ("99pct", 0.99, 1), ("50pct", 0.5, 2)):
            b_np, agg_np, expect = participation_case(eng, W, np, frac, seed)
            db, da = torch.as_tensor(b_np, device=dev), torch.as_tensor(agg_np, device=dev)
            ms_c3, _ = timed(lambda: eng.fast_aggregate_verify_dev(ep.d_members, ep.d_off, db, d_msgs, da, t_ok))
            assert np.array_equal(t_ok.cpu().numpy(), expect), "config 3 verdicts wrong at participation " + name
            k_set = int(np.unpackbits(b_np, axis=1).sum())
            cfg["config3_fast_aggregate_verify_2048x512_" + name] = {
                "ms": ms_c3, "aggregates_per_s": N_AGG / (ms_c3 * 1e-3), "attestations_per_s": k_set / (ms_c3 * 1e-3), "set_bits": k_set,
                "corrupted_aggregates": int(N_AGG - expect.sum()), "verdicts_match_expected": True}

    # ---- get_head latency.  N = 1: the C-ABI call incl. D2H of the head index.  N > 1: THROUGH the multi-rank path (vote scatter of
    # this rank's validators -> NCCL all-reduce of u64[10 000] -> head on every rank -> D2H), every rank in lockstep.
    def head_latency(fn, n=250):
        xs = []
        h = None
        for i in range(n):
            t0 = time.perf_counter()
            h = fn()
            xs.append((time.perf_counter() - t0) * 1e6)
        xs = sorted(xs[50:])
        return h, xs[len(xs) // 2], xs[int(len(xs) * 0.99) - 1]

    p50_nccl = p99_nccl = None
    fused_ok = False
    if world > 1:
        barrier()
        hd_nccl, p50_nccl, p99_nccl = head_latency(lambda: ep.get_head(0, boost_idx, boost, fused=False))    # scatter -> NCCL all-reduce -> tree -> D2H
        if shard is not None:
            barrier()
            fused_ok = ep.enable_fused_get_head()          # collective: CUDA IPC exchange blocks on every rank, or the NCCL form everywhere
            barrier()
            if fused_ok:
                hd, p50, p99 = head_latency(lambda: ep.get_head(0, boost_idx, boost, fused=True))          # one kernel per rank, reduction over NVLink peer memory
                assert hd == hd_nccl, "fused and NCCL get_head disagree"
            else:
                hd, p50, p99 = hd_nccl, p50_nccl, p99_nccl
        else:
            hd, p50, p99 = hd_nccl, p50_nccl, p99_nccl
    else:
        hd, p50, p99 = head_latency(lambda: eng.get_head(0, boost_idx, boost))
    lat_local = []
    for i in range(150):
        t0 = time.perf_counter()
        eng.get_head(0, boost_idx, boost)               # the single-GPU call (all validators of this rank's table), for comparison
        lat_local.append((time.perf_counter() - t0) * 1e6)
    p50_local = sorted(lat_local[50:])[50]

    # max over ranks
    t = torch.tensor([ms_dev, ms_e2e, ms_agg, ms_verify, p50, p99, ms_sync, g_tma_cold, g_ldg_cold, g_tma_warm, p50_nccl or 0.0, p99_nccl or 0.0],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e, ms_agg, ms_verify, p50, p99, ms_sync, g_tma_cold, g_ldg_cold, g_tma_warm, p50_nccl, p99_nccl = [float(x) for x in t.tolist()]

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        algo_bytes = 96 * n_loc_sig + 96 * ep.n_loc                        # SURVEY.md section 8d: bls.Aggregate = 96n + 96s (this rank's share)
        achieved = algo_bytes / (ms_agg * 1e-3) / 1e9
        # integer-pipe reading of the same launch: IMAD.WIDE.U32 instructions per signature, counted from the SASS of fp_sqr (222)
        # and fp_mul (288): 2 exponentiations x (380 squarings + 76 multiplications: the schedule with the a^255 run token,
        # tools/gen_consts.py) + ~60 multiplications for the curve equation, sign fix and the segment additions.  Peak = 32 wide MACs / clk / SM (one IMAD.WIDE per 4 cycles per scheduler,
        # ncu: sm__pipe_fmaheavy) x SMs x the SM clock sampled during the timed region.
        wide_per_sig = 2 * (380 * 222 + 76 * 288) + 60 * 288
        sm_mhz = clocks.get("sm_mhz") or 1965.0
        n_sm = torch.cuda.get_device_properties(local).multi_processor_count
        int_peak = 32.0 * n_sm * sm_mhz * 1e6
        int_ach = wide_per_sig * n_loc_sig / (ms_agg * 1e-3)
        # gather stage: SURVEY.md 8(d) "pubkey-gather stage alone" = 96k + 4c + c/8 per aggregate
        gather_bytes = ep.n_loc * (96 * COMMITTEE_SIZE + 4 * COMMITTEE_SIZE + COMMITTEE_SIZE // 8)
        gbps = lambda ms: gather_bytes / (ms * 1e-3) / 1e9               # noqa: E731
        total_units = (world * N_VAL) if not strong else N_VAL
        par = ("one 2^20-validator epoch sharded by slot x%d: all-gather of aggregate signatures + verdicts, LMD replicated, "
               "votes sharded by validator, one u64[10000] all-reduce" % world) if strong else ("validators sharded x%d (own epoch per rank), one u64[10000] all-reduce" % world)
        line = {
            "metric": METRIC, "value": total_units / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_dev, "ms_per_step_unpipelined": ms_sync, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "u32 limbs (381-bit Fp, Montgomery)", "data": "synthetic",
            "config": {"workload": WORKLOAD if not strong else WORKLOAD.replace(" per rank", " in total (one epoch for the whole box)"),
                       "validators_total": total_units, "aggregates_per_rank": ep.n_loc, "signatures_per_rank": n_loc_sig, "parallelism": par,
                       "pipeline_depth": depth, "pipelining": "software pipeline over pipeline_depth slots: epoch k+1's signature decompression overlaps the pairing tails of the epochs before it; all K results complete inside the timed region (fill and drain included)",
                       "tail_form": "team" if ep.always_team else "thread (team for the last epoch of the batch)",
                       "verify_mode": "rlc batches of 32 with per-aggregate fallback" if args.rlc else "per aggregate",
                       "l2": "per-step working set ~0.5 GB/world (signatures 101 MB + decompressed points 201 MB) + registry 101 MB > 126 MB L2"},
            "e2e": {"value": total_units / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": ep.h2d_bytes, "d2h_bytes_per_step": ep.d2h_bytes,
                    "d2h": "verdicts + head index + the 2048 aggregate signatures"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "get_head_p50_us": p50, "get_head_p99_us": p99, "get_head_single_gpu_call_p50_us": p50_local, "head_index": head0,
            "get_head_path": ("b2_get_head: ONE kernel (vote scatter, last CTA runs the tree phase, head written to mapped host memory)" if world == 1 else
                              ("b2_get_head_multi: ONE kernel per rank -- scatter of N/%d validators, 64-bit reductions into every rank's accumulator over NVLink peer memory, flag exchange, tree, zero-copy result" % world
                               if fused_ok else "vote scatter -> NCCL all-reduce u64[10000] -> tree -> D2H" + ("" if shard is None else " (peer-memory form unavailable: %s)" % ep.fused_head_error))),
            **({"get_head_nccl_path_p50_us": p50_nccl, "get_head_nccl_path_p99_us": p99_nccl,
                "get_head_nccl_path": "vote scatter of N/%d validators -> NCCL all-reduce u64[10000] -> tree kernel -> D2H" % world} if world > 1 else {}),
            "stage_ms": {"bls_aggregate_rank_share": ms_agg, "fast_aggregate_verify_rank_share": ms_verify,
                         **({"aggregate_and_verify_concurrent": ms_overlap} if ms_overlap is not None else {})},
            "roofline": {"bound": "hbm", "kernel": "bls.Aggregate (k_g2_decompress + k_g2_segment_sum), this rank's %d signatures" % n_loc_sig, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": TRAFFIC_BYTES_K3 * n_loc_sig / N_VAL, "peak_source": peak_src,
                         "traffic_source": "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of k_g2_decompress (profiles/)",
                         "note": "integer-pipe bound, not HBM bound (ncu: sm__pipe_fmaheavy_cycles_active ~89%, DRAM <1% of peak); see int_pipe and DESIGN.md",
                         "int_pipe": {"achieved": int_ach / 1e12, "peak": int_peak / 1e12, "unit": "T wide-MAC/s", "frac": int_ach / int_peak,
                                      "wide_mac_per_signature": wide_per_sig},
                         "gather": {"bound": "hbm", "kernel": "k_g1_gather_tma<probe>: K2's gather stage alone (bits + u32 indices + 96-B pubkey records via cp.async.bulk -> smem -> LDS.128, XOR checksum instead of the additions)",
                                    "algorithmic_bytes": gather_bytes, "achieved": gbps(g_tma_cold), "peak": peak, "unit": "GB/s", "frac": gbps(g_tma_cold) / peak,
                                    "l2": "flushed before every launch (512 MB memset): the 100.7 MB registry would otherwise stay in the 126 MB L2",
                                    "ms": g_tma_cold, "ms_best": g_tma_cold_min, "frac_best": gbps(g_tma_cold_min) / peak,
                                    "l2_warm": {"ms": g_tma_warm, "achieved": gbps(g_tma_warm), "frac": gbps(g_tma_warm) / peak},
                                    "plain_ldg_form": {"kernel": "k_g1_gather_ldg_probe: block per aggregate, six lanes per 96-B record (LDG.E.128), all loads of a thread in flight -- the fastest of the six forms of tools/gather_bench.cu (profiles/r2_gather_microbench.jsonl)",
                                                       "ms": g_ldg_cold, "ms_best": g_ldg_cold_min, "achieved": gbps(g_ldg_cold), "frac": gbps(g_ldg_cold) / peak, "frac_best": gbps(g_ldg_cold_min) / peak},
                                    "what_binds": "random 96-byte reads: HBM moves two 64-byte bursts (128 B) per record, i.e. 1.33x the algorithmic bytes, at random-access row-buffer efficiency; with the additions K2 is bound by the integer multiply pipe (34 MAC/B), not by this stage",
                                    "checksums_equal": True}},
            "setup_s": W["setup_s"],
        }
        line.update(cfg)
        if world == 1 and not args.no_cpu_baseline:
            import multiprocessing as mp
            cores = min(host_cores(), 64)
            with mp.get_context("fork").Pool(cores) as pool:
                # same workload, bounded sample: the first `cores` committees of this very epoch (GPU-made keys/signatures)
                comm = []
                for a in range(cores):
                    m = W["members"][a * COMMITTEE_SIZE:(a + 1) * COMMITTEE_SIZE]
                    comm.append(([bytes(W["pk"][v]) for v in m], [bytes(s) for s in W["sigs"][a * COMMITTEE_SIZE:(a + 1) * COMMITTEE_SIZE]], bytes(W["msgs"][a])))
                v, wall, cpu_aggs = cpu_sample(pool, cores, comm)
            # parity of the bytes, not only of the verdict: the oracle's bls.Aggregate output == the GPU's aggregate signature
            agg_match = all(cpu_aggs[a] == bytes(agg_sig_gpu[a]) for a in range(cores))
            assert agg_match, "oracle bls.Aggregate bytes differ from the GPU aggregate signatures"
            from oracle import fast
            parent, roots, leaf_viable = W["tree"]
            e, b, hmsg = eng.latest_messages_read()
            t0 = time.perf_counter()
            w = fast.ghost_weights(parent, b, hmsg, W["votes"][3], W["votes"][4], W["votes"][2], boost_idx, boost)
            hd_cpu = fast.ghost_head(parent, roots, fast.ghost_viable(parent, leaf_viable), w, 0)
            cpu_head_ms = (time.perf_counter() - t0) * 1e3
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "cpu_model": cpu_model(), "kind": "port",
                                    "sample": "%d of the 2048 committees of this epoch (512 members each), 1 per core, %.1f s wall: oracle bls.Aggregate + FastAggregateVerify" % (cores, wall),
                                    "aggregate_bytes_match_gpu": agg_match,
                                    "get_head_numpy_ms": cpu_head_ms, "get_head_matches_gpu": bool(hd_cpu == hd)}
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--depth", type=int, default=0, help="epochs in flight in the software pipeline (2..8); 0 = 3 on one GPU, 4/6/8 on 2/4/8 GPUs of a sharded epoch")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: strong = ONE 2^20-validator epoch sharded by slot over the ranks (north_star configs 4/5); weak = an own epoch per rank")
    ap.add_argument("--tail-form", default="auto", choices=["auto", "thread", "team"],
                    help="pairing kernels of the pipelined epochs: thread per aggregate (fewest instructions), 3-lane teams (shortest critical path), auto")
    ap.add_argument("--emulate-world", type=int, default=0, help="tuning aid (1 GPU): run rank 0's share of an epoch sharded over this many ranks, without collectives")
    ap.add_argument("--team-last", type=int, default=None, help="how many epochs at the end of a batch take the team-form tail (default 1)")
    ap.add_argument("--rlc", action="store_true", help="FastAggregateVerify in random-linear-combination batches (b2_set_verify_mode 1)")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the per-config numbers of BASELINE.json configs 2 and 3")
    ap.add_argument("--probe-overlap", action="store_true",
                    help="also time bls.Aggregate and FastAggregateVerify running concurrently on two streams (diagnostic)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed epoch returned (rank 0: verdicts, head index, aggregate "
                         "signatures) as DIR/<name>.npy in float32/float64; the seeded inputs make two builds comparable")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
