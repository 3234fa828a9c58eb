"""Differential tests: what the reference's own fenced python blocks computed (pos-evolution.md, executed
literally by tests/golden/gen_golden.py and stored in tests/golden/literal_spec.json) vs the oracle's
restatement vs the numpy array form, on the same generated inputs."""
import copy
import json
import os

import numpy as np
import pytest

import scenarios
from oracle import fast
from oracle import spec as S

G = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "literal_spec.json")))


@pytest.fixture(scope="module")
def env():
    spec, state = scenarios.minimal_state(64, slot=9)
    assert [v.pubkey.hex() for v in state.validators] == G["pubkeys"]
    return spec, state


def test_shuffle_literal_vs_oracle_vs_numpy(env):
    spec, _ = env
    assert {s["n"] for s in G["shuffle"]} == {1, 2, 37, 256, 257, 1000}
    for s in G["shuffle"]:
        n, seed, lit = s["n"], bytes.fromhex(s["seed"]), s["perm"]
        assert s["rounds"] == spec.p.SHUFFLE_ROUND_COUNT
        assert lit == [spec.compute_shuffled_index(i, n, seed) for i in range(n)]
        assert lit == fast.shuffle_permutation(n, seed, spec.p.SHUFFLE_ROUND_COUNT).tolist()
        assert sorted(lit) == list(range(n))


def test_committees_literal_vs_numpy(env):
    spec, state = env
    epoch = 1
    cps = G["committee_count_per_slot"][str(epoch)]
    assert cps == 2 == spec.get_committee_count_per_slot(state, epoch)
    seed = spec.get_seed(state, epoch, S.DOMAIN_BEACON_ATTESTER)
    assert seed.hex() == G["attester_seed"][str(epoch)]
    active = np.array(spec.get_active_validator_indices(state, epoch), dtype=np.uint32)
    members, off = fast.committees_for_epoch(active, seed, spec.p.SHUFFLE_ROUND_COUNT, cps, spec.p.SLOTS_PER_EPOCH)
    seen = []
    for s in range(spec.p.SLOTS_PER_EPOCH):
        for c in range(cps):
            lit = G["committees"]["%d/%d" % (epoch * spec.p.SLOTS_PER_EPOCH + s, c)]
            k = s * cps + c
            assert lit == members[off[k]:off[k + 1]].tolist() == spec.get_beacon_committee(state, 8 + s, c)
            assert len(lit) == 4
            seen += lit
    assert sorted(seen) == list(range(64))          # committees partition the validator set (ref :455)


def _run(fn, state, att):
    st = copy.deepcopy(state)
    try:
        fn(st, att)
        return "ok", st
    except AssertionError:
        return "assert", None


def test_process_attestation_literal_vs_oracle(env):
    spec, state = env
    cases = [
        scenarios.make_attestation(spec, state, 8, 0),
        scenarios.make_attestation(spec, state, 8, 1, bits=[True, False, True, False]),
        scenarios.make_attestation(spec, state, 5, 1),                                    # previous epoch
        scenarios.make_attestation(spec, state, 8, 0, corrupt="flip_bit"),
        scenarios.make_attestation(spec, state, 8, 0, corrupt="wrong_message"),
        scenarios.make_attestation(spec, state, 8, 1, corrupt="wrong_signer_set"),
        scenarios.make_attestation(spec, state, 8, 0, bits=[False] * 4),                  # empty -> invalid
        scenarios.make_attestation(spec, state, 8, 0, bits=[True] * 3),                   # wrong bit length
    ]
    bad_idx = scenarios.make_attestation(spec, state, 8, 0)
    bad_idx.data = S.AttestationData(8, 2, bad_idx.data.beacon_block_root, bad_idx.data.source, bad_idx.data.target)
    cases.append(bad_idx)                                                                 # index >= committee count
    expect = ["ok", "ok", "ok", "assert", "assert", "assert", "assert", "assert", "assert"]
    assert len(G["process_attestation"]) == len(cases)
    for att, exp, lit in zip(cases, expect, G["process_attestation"]):
        assert lit["attestation"]["signature"] == att.signature.hex() and lit["attestation"]["index"] == att.data.index
        assert lit["attestation"]["bits"] == [bool(b) for b in att.aggregation_bits]
        r_or, st_or = _run(spec.process_attestation, state, att)
        assert lit["result"] == r_or == exp
        if exp == "ok":
            assert lit["current_epoch_participation"] == st_or.current_epoch_participation
            assert lit["previous_epoch_participation"] == st_or.previous_epoch_participation
            assert lit["balances"] == st_or.balances
            assert lit["balances"] != state.balances
    # double inclusion: flags already set -> no second reward
    twice = G["process_attestation_twice"]
    assert twice["balances_after_first"] == G["process_attestation"][0]["balances"]
    assert twice["balances_after_second"] == twice["balances_after_first"]
    st = copy.deepcopy(state)
    spec.process_attestation(st, cases[0])
    assert st.balances == twice["balances_after_first"]
    spec.process_attestation(st, cases[0])
    assert st.balances == twice["balances_after_second"]


def test_get_head_literal_vs_oracle_vs_numpy(env):
    spec, state = env
    state = copy.deepcopy(state)
    state.validators[5].exit_epoch = 0          # inactive validator is not counted
    store, parent, slot, roots, leaf_viable, rb = scenarios.small_store(spec, state)
    assert {str(v): [m.epoch, m.root.hex()] for v, m in store.latest_messages.items()} == G["get_head"]["latest_messages"]
    head_lit = bytes.fromhex(G["get_head"]["head"])
    assert head_lit == spec.get_head(store)
    n = len(state.validators)
    idx_of = {r: i for i, r in enumerate(rb)}
    msg_block = np.zeros(n, dtype=np.uint32)
    has_msg = np.zeros(n, dtype=np.uint8)
    for v, lm in store.latest_messages.items():
        msg_block[v], has_msg[v] = idx_of[lm.root], 1
    eff = np.array([v.effective_balance for v in state.validators], dtype=np.uint64)
    active = np.array([spec.is_active_validator(v, spec.get_current_epoch(state)) for v in state.validators], dtype=np.uint8)
    equiv = np.zeros(n, dtype=np.uint8)
    equiv[list(store.equivocating_indices)] = 1
    boost = fast.proposer_boost_score(eff, active, spec.p.SLOTS_PER_EPOCH, spec.p.PROPOSER_SCORE_BOOST)
    w = fast.ghost_weights(parent, msg_block, has_msg, eff, active, equiv, len(rb) - 1, boost)
    for b in range(0, len(rb), 7):
        assert int(w[b]) == spec.get_latest_attesting_balance(store, rb[b])
    keep = fast.ghost_viable(parent, leaf_viable)
    assert set(rb[b] for b in range(len(rb)) if keep[b]) == set(spec.get_filtered_block_tree(store).keys())
    assert rb[fast.ghost_head(parent, roots, keep, w, 0)] == head_lit


def test_update_latest_messages_literal_vs_numpy(env):
    spec, state = env
    g = G["update_latest_messages"]
    store, parent, slot, roots, leaf_viable, rb = scenarios.small_store(spec, state, n_blocks=g["n_blocks"], seed=g["tree_seed"])
    n = len(state.validators)
    idx_of = {r: i for i, r in enumerate(rb)}
    msg_epoch = np.zeros(n, dtype=np.uint64)
    msg_block = np.zeros(n, dtype=np.uint32)
    has_msg = np.zeros(n, dtype=np.uint8)
    for v, lm in store.latest_messages.items():
        msg_epoch[v], msg_block[v], has_msg[v] = lm.epoch, idx_of[lm.root], 1
    equiv = np.zeros(n, dtype=np.uint8)
    equiv[list(store.equivocating_indices)] = 1
    for epoch, blk, idxs in scenarios.LMD_UPDATES:
        fast.lmd_update(msg_epoch, msg_block, has_msg, equiv, idxs, epoch, blk)
    lit = {int(v): tuple(m) for v, m in g["latest_messages"].items()}
    for v in range(n):
        if has_msg[v]:
            assert lit[v] == (int(msg_epoch[v]), int(msg_block[v]))
        else:
            assert v not in lit


def test_ffg_literal_vs_oracle(env):
    """process_justification_and_finalization / weigh_justification_and_finalization: what the reference's own text (ref :793-852)
    computed against the oracle's restatement on 80 generated end-of-epoch states; every branch must have fired."""
    spec, state0 = env
    assert [c["seed"] for c in G["ffg"]] == list(range(80))
    seen = set()
    for case in G["ffg"]:
        seed = case["seed"]
        st_or = scenarios.ffg_case(copy.deepcopy(state0), seed)
        before = (scenarios.ffg_outcome(st_or)["current_justified"], scenarios.ffg_outcome(st_or)["finalized"])
        spec.process_justification_and_finalization(st_or)
        got, want = scenarios.ffg_outcome(st_or), {k: v for k, v in case.items() if k != "seed"}
        assert got == want, seed
        seen.add(("justified_changed", want["current_justified"] != before[0]))
        seen.add(("finalized_changed", want["finalized"] != before[1]))
        seen.add(("bits", tuple(want["justification_bits"][:2])))
        if want["finalized"] != before[1]:
            seen.add(("finalized_distance", spec.get_current_epoch(st_or) - want["finalized"][0]))
    assert {("justified_changed", True), ("justified_changed", False), ("finalized_changed", True), ("finalized_changed", False)} <= seen
    assert {("bits", (0, 0)), ("bits", (0, 1)), ("bits", (1, 0)), ("bits", (1, 1))} <= seen
    assert {("finalized_distance", 1), ("finalized_distance", 2), ("finalized_distance", 3)} <= seen
