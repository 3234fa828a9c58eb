"""Deterministic synthetic inputs shared by the CPU and GPU tests (SURVEY.md section 8d).
Uses the oracle to make keys/signatures -- test infrastructure only."""
import copy
import hashlib

import numpy as np

from oracle import bls_sig
from oracle import spec as S
from oracle.bls12_381 import R, E1, E2, G1, g1_compress, g2_compress
from oracle.hash_to_curve import hash_to_g2


def _h(b):
    return hashlib.sha256(b).digest()


SK0 = int.from_bytes(_h(b"b200pos/sk0"), "big") % R
SKD = int.from_bytes(_h(b"b200pos/skd"), "big") % R


def secret_key(i: int) -> int:
    return (SK0 + i * SKD) % R or 1


def pubkeys(n: int):
    """pk_i = pk_0 + i*(delta*g1): n additions + one batch inversion instead of n scalar muls."""
    step = E1.mul(G1, SKD)
    cur = E1.mul(G1, SK0)
    pts = []
    for _ in range(n):
        pts.append(cur)
        cur = E1.add(cur, step)
    aff = E1.batch_to_affine(pts)
    return [g1_compress((x, y, 1)) for (x, y) in aff]


def sign_aggregate(indices, message: bytes) -> bytes:
    """Aggregate signature of validators ``indices`` on one message = (sum sk_i) * H(m)."""
    sk = sum(secret_key(i) for i in indices) % R
    return g2_compress(E2.mul(hash_to_g2(message), sk))


def individual_signatures(indices, message: bytes):
    """sig_i = sk_i * H(m) for every i, via the arithmetic progression when indices are consecutive-agnostic."""
    h = hash_to_g2(message)
    pts = [E2.mul(h, secret_key(i)) for i in indices]
    aff = E2.batch_to_affine(pts)
    return [g2_compress((a[0], a[1], (1, 0))) if a is not None else g2_compress(E2.INF) for a in aff]


def minimal_state(n_validators: int = 64, slot: int = 9, preset=S.MINIMAL, pks=None):
    spec = S.Spec(preset)
    pks = pks if pks is not None else pubkeys(n_validators)
    rng = np.random.default_rng(7)
    bal = [int(b) * 10**9 for b in rng.choice([32, 32, 32, 31, 24, 16], size=n_validators)]
    validators = [S.Validator(pubkey=pks[i], effective_balance=bal[i]) for i in range(n_validators)]
    mixes = [_h(b"b200pos/mix" + i.to_bytes(8, "little")) for i in range(preset.EPOCHS_PER_HISTORICAL_VECTOR)]
    roots = [_h(b"b200pos/blockroot" + i.to_bytes(8, "little")) for i in range(preset.SLOTS_PER_HISTORICAL_ROOT)]
    state = S.BeaconState(
        slot=slot, fork=S.Fork(bytes(4), bytes.fromhex("00000001"), 0),
        genesis_validators_root=_h(b"b200pos/gvr"), validators=validators, balances=list(bal),
        randao_mixes=mixes, block_roots=roots,
        previous_epoch_participation=[0] * n_validators, current_epoch_participation=[0] * n_validators,
        previous_justified_checkpoint=S.Checkpoint(0, _h(b"b200pos/j0")),
        current_justified_checkpoint=S.Checkpoint(0, _h(b"b200pos/j0")))
    return spec, state


def make_attestation(spec, state, slot: int, index: int, bits=None, head_root=None, corrupt=None, target_root=None):
    """A correctly-signed aggregate attestation for (slot, index); ``bits`` defaults to full participation."""
    committee = spec.get_beacon_committee(state, slot, index)
    bits = [True] * len(committee) if bits is None else list(bits)
    epoch = spec.compute_epoch_at_slot(slot)
    just = state.current_justified_checkpoint if epoch == spec.get_current_epoch(state) else state.previous_justified_checkpoint
    if target_root is None:
        target_root = spec.get_block_root(state, epoch) if spec.compute_start_slot_at_epoch(epoch) < state.slot else _h(b"t")
    head = head_root if head_root is not None else spec.get_block_root_at_slot(state, slot)
    data = S.AttestationData(slot=slot, index=index, beacon_block_root=head, source=just,
                             target=S.Checkpoint(epoch, target_root))
    domain = spec.get_domain(state, S.DOMAIN_BEACON_ATTESTER, epoch)
    msg = spec.compute_signing_root(data, domain)
    signers = [v for v, b in zip(committee, bits) if b]
    if corrupt == "wrong_signer_set" and signers:
        signers = signers[:-1] or [committee[0] ^ 1]
    if corrupt == "wrong_message":
        msg = _h(msg)
    sig = sign_aggregate(signers, msg) if signers else g2_compress(E2.INF)
    if corrupt == "flip_bit":
        b = bytearray(sig)
        b[95] ^= 1
        sig = bytes(b)
    return S.Attestation(aggregation_bits=bits, data=data, signature=sig)


def fork_tree(n_blocks: int, seed: int = 4):
    """SURVEY.md section 8d config 4: random fork tree in topological order."""
    rng = np.random.default_rng(seed)
    parent = np.zeros(n_blocks, dtype=np.uint32)
    slot = np.zeros(n_blocks, dtype=np.uint64)
    back = rng.geometric(0.7, size=n_blocks) - 1
    skip = rng.binomial(2, 0.1, size=n_blocks)
    for i in range(1, n_blocks):
        parent[i] = max(0, i - 1 - int(back[i]))
        slot[i] = slot[parent[i]] + 1 + int(skip[i])
    roots = np.frombuffer(b"".join(_h(i.to_bytes(8, "little")) for i in range(n_blocks)), dtype=np.uint8).reshape(n_blocks, 32).copy()
    leaf_viable = (rng.random(n_blocks) >= 0.05).astype(np.uint8)
    return parent, slot, roots, leaf_viable


def small_store(spec, state, n_blocks=200, seed=3):
    """An oracle Store over fork_tree(n_blocks, seed): non-viable leaves get a mismatching justified checkpoint, validators 3
    and 17 equivocate, the proposer boost sits on the last block and ~90% of the validators hold a latest message."""
    parent, slot, roots, leaf_viable = fork_tree(n_blocks, seed)
    rb = [bytes(r) for r in roots]
    just = S.Checkpoint(1, rb[0])
    fin = S.Checkpoint(1, rb[0])
    store = S.Store(time=0, genesis_time=0, justified_checkpoint=just, finalized_checkpoint=fin,
                    best_justified_checkpoint=just, proposer_boost_root=rb[n_blocks - 1], equivocating_indices={3, 17})
    has_child = set(int(p) for p in parent[1:])
    for b in range(n_blocks):
        store.blocks[rb[b]] = S.BeaconBlock(int(slot[b]), rb[parent[b]] if b else bytes(32))
        bs = copy.copy(state)
        if b not in has_child and not leaf_viable[b]:
            bs.current_justified_checkpoint = S.Checkpoint(0, b"\x01" * 32)
        else:
            bs.current_justified_checkpoint = just
        bs.finalized_checkpoint = fin
        store.block_states[rb[b]] = bs
    store.checkpoint_states[just] = state
    rng = np.random.default_rng(seed)
    n = len(state.validators)
    for v in range(n):
        if rng.random() < 0.9:
            store.latest_messages[v] = S.LatestMessage(1, rb[int(n_blocks - 1 - min(n_blocks - 1, rng.geometric(0.05)))])
    return store, parent, slot, roots, leaf_viable, rb


# (epoch, voted block, attesting validators) of the update_latest_messages sequence the golden vectors record
LMD_UPDATES = ((1, 10, [1, 2, 3, 40]), (2, 20, [2, 3, 17, 41, 63]), (1, 30, [2, 50]))


def votes(n_validators: int, n_blocks: int, seed: int = 4):
    rng = np.random.default_rng(seed + 1000)
    msg_block = (n_blocks - 1 - np.minimum(n_blocks - 1, rng.geometric(0.002, size=n_validators))).astype(np.uint32)
    has_msg = (rng.random(n_validators) >= 0.01).astype(np.uint8)
    equiv = (rng.random(n_validators) < 0.001).astype(np.uint8)
    active = (rng.random(n_validators) >= 0.01).astype(np.uint8)
    eff = np.where(rng.random(n_validators) < 0.9, 32, rng.integers(16, 33, size=n_validators)).astype(np.uint64) * np.uint64(10**9)
    return msg_block, has_msg, equiv, active, eff


def ffg_case(state, seed: int, mod=S):
    """Mutates `state` into a deterministic end-of-epoch situation for process_justification_and_finalization (ref :793-852):
    random TIMELY_TARGET participation in both tables, a few slashed / exited / not-yet-active validators, prior checkpoints and
    justification bits chosen so that over the seeds every justification branch and every finalization rule fires."""
    rng = np.random.default_rng(1000 + seed)
    n = len(state.validators)
    cur = int(rng.integers(2, 8))
    state.slot = cur * 8 + 7                                   # last slot of the epoch (minimal preset: 8 slots)
    p_cur, p_prev = (float(rng.choice([0.2, 0.6, 0.66, 0.7, 0.95])) for _ in range(2))
    state.current_epoch_participation = [int(rng.integers(0, 8)) & 5 | (2 if rng.random() < p_cur else 0) for _ in range(n)]
    state.previous_epoch_participation = [int(rng.integers(0, 8)) & 5 | (2 if rng.random() < p_prev else 0) for _ in range(n)]
    for v in state.validators:
        r = rng.random()
        v.slashed = r < 0.06
        v.activation_epoch, v.exit_epoch = 0, 2**64 - 1
        if 0.06 <= r < 0.10:
            v.exit_epoch = cur                                 # active in the previous epoch only
        elif 0.10 <= r < 0.13:
            v.activation_epoch = cur                           # active in the current epoch only
        elif 0.13 <= r < 0.15:
            v.exit_epoch = max(0, cur - 1)                     # active in neither
        v.effective_balance = int(rng.choice([32, 32, 32, 31, 24, 16])) * 10**9
    pj = int(rng.integers(max(0, cur - 3), cur))               # previous_justified epoch in [cur-3, cur-1]
    cj = int(rng.integers(max(pj, cur - 2), cur))              # current_justified epoch in [max(pj, cur-2), cur-1]
    root = lambda e: _h(b"b200pos/cp" + int(e).to_bytes(8, "little"))   # noqa: E731
    state.previous_justified_checkpoint = mod.Checkpoint(pj, root(pj))
    state.current_justified_checkpoint = mod.Checkpoint(cj, root(cj))
    state.finalized_checkpoint = mod.Checkpoint(max(0, pj - 1), root(max(0, pj - 1)))
    state.justification_bits = [int(b) for b in rng.integers(0, 2, size=4)]
    return state


def ffg_outcome(state):
    return {"previous_justified": [state.previous_justified_checkpoint.epoch, state.previous_justified_checkpoint.root.hex()],
            "current_justified": [state.current_justified_checkpoint.epoch, state.current_justified_checkpoint.root.hex()],
            "finalized": [state.finalized_checkpoint.epoch, state.finalized_checkpoint.root.hex()],
            "justification_bits": [int(b) for b in state.justification_bits]}
