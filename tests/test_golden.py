"""Golden vectors produced by executing the reference's own python blocks (tests/golden/gen_golden.py)
replayed against (a) the oracle -- CPU -- and (b) the CUDA path through the pyspec-signature layer -- GPU."""
import copy
import json
import os

import numpy as np
import pytest

import scenarios
from oracle import fast
from oracle import spec as OS

G = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "literal_spec.json")))


def _state(pks):
    spec, state = scenarios.minimal_state(64, slot=G["state_slot"], pks=pks)
    return spec, state


def _att(mod, j):
    data = mod.AttestationData(j["slot"], j["index"], bytes.fromhex(j["beacon_block_root"]),
                               mod.Checkpoint(j["source"][0], bytes.fromhex(j["source"][1])),
                               mod.Checkpoint(j["target"][0], bytes.fromhex(j["target"][1])))
    return mod.Attestation(list(j["bits"]), data, bytes.fromhex(j["signature"]))


PKS = [bytes.fromhex(p) for p in G["pubkeys"]]


def test_oracle_shuffle_and_committees_golden():
    spec, state = _state(PKS)
    for s in G["shuffle"]:
        seed = bytes.fromhex(s["seed"])
        assert [spec.compute_shuffled_index(i, s["n"], seed) for i in range(s["n"])] == s["perm"]
        assert fast.shuffle_permutation(s["n"], seed, s["rounds"]).tolist() == s["perm"]
    for key, members in G["committees"].items():
        slot, idx = map(int, key.split("/"))
        assert spec.get_beacon_committee(state, slot, idx) == members


def test_oracle_process_attestation_golden():
    spec, state = _state(PKS)
    for case in G["process_attestation"]:
        att = _att(OS, case["attestation"])
        dom = spec.get_domain(state, OS.DOMAIN_BEACON_ATTESTER, att.data.target.epoch)
        assert spec.compute_signing_root(att.data, dom).hex() == case["signing_root"]
        st = copy.deepcopy(state)
        if case["result"] == "ok":
            spec.process_attestation(st, att)
            assert st.balances == case["balances"]
            assert st.current_epoch_participation == case["current_epoch_participation"]
            assert st.previous_epoch_participation == case["previous_epoch_participation"]
        else:
            with pytest.raises(AssertionError):
                spec.process_attestation(st, att)


def _golden_store(mod, state):
    g = G["get_head"]
    parent, slot, roots, leaf_viable = scenarios.fork_tree(g["n_blocks"], g["tree_seed"])
    rb = [bytes(r) for r in roots]
    just = mod.Checkpoint(1, rb[0])
    store = mod.Store(0, 0, just, just, just, bytes.fromhex(g["proposer_boost_root"]), set(g["equivocating"]))
    has_child = set(int(p) for p in parent[1:])
    for b in range(g["n_blocks"]):
        store.blocks[rb[b]] = mod.BeaconBlock(int(slot[b]), rb[parent[b]] if b else bytes(32))
        bs = copy.copy(state)
        bad = b not in has_child and not leaf_viable[b]
        bs.current_justified_checkpoint = mod.Checkpoint(0, b"\x01" * 32) if bad else just
        bs.finalized_checkpoint = just
        store.block_states[rb[b]] = bs
    store.checkpoint_states[just] = state
    for v, (e, r) in g["latest_messages"].items():
        store.latest_messages[int(v)] = mod.LatestMessage(e, bytes.fromhex(r))
    return store


def test_oracle_get_head_golden():
    spec, state = _state(PKS)
    state.validators[G["get_head"]["inactive_validator"]].exit_epoch = 0
    store = _golden_store(OS, state)
    assert spec.get_head(store).hex() == G["get_head"]["head"]
    for r, w in G["get_head"]["weights"].items():
        assert spec.get_latest_attesting_balance(store, bytes.fromhex(r)) == w


def test_oracle_ffg_golden():
    spec, state = _state(PKS)
    for case in G["ffg"]:
        st = scenarios.ffg_case(copy.deepcopy(state), case["seed"])
        spec.process_justification_and_finalization(st)
        assert dict(scenarios.ffg_outcome(st), seed=case["seed"]) == case


# ----------------------------------------------------------------------------- the CUDA path against the same vectors
@pytest.fixture(scope="module")
def product():
    from pos_evolution_b200 import spec as PS
    from pos_evolution_b200.engine import Engine
    return PS, PS.Spec(PS.MINIMAL, engine=Engine(0))


def _pstate(PS, ostate):
    return PS.BeaconState(
        slot=ostate.slot, fork=PS.Fork(ostate.fork.previous_version, ostate.fork.current_version, ostate.fork.epoch),
        genesis_validators_root=ostate.genesis_validators_root,
        validators=[PS.Validator(v.pubkey, v.effective_balance, v.slashed, v.activation_epoch, v.exit_epoch) for v in ostate.validators],
        balances=list(ostate.balances), randao_mixes=list(ostate.randao_mixes), block_roots=list(ostate.block_roots),
        previous_epoch_participation=list(ostate.previous_epoch_participation), current_epoch_participation=list(ostate.current_epoch_participation),
        previous_justified_checkpoint=PS.Checkpoint(ostate.previous_justified_checkpoint.epoch, ostate.previous_justified_checkpoint.root),
        current_justified_checkpoint=PS.Checkpoint(ostate.current_justified_checkpoint.epoch, ostate.current_justified_checkpoint.root),
        finalized_checkpoint=PS.Checkpoint(ostate.finalized_checkpoint.epoch, ostate.finalized_checkpoint.root))


@pytest.mark.gpu
def test_gpu_process_attestation_golden(product):
    PS, pspec = product
    _, ostate = _state(PKS)
    for key, members in G["committees"].items():
        slot, idx = map(int, key.split("/"))
        assert pspec.get_beacon_committee(ostate, slot, idx) == members
    for case in G["process_attestation"]:
        att = _att(PS, case["attestation"])
        st = _pstate(PS, ostate)
        if case["result"] == "ok":
            pspec.process_attestation(st, att)
            assert st.balances == case["balances"]
            assert st.current_epoch_participation == case["current_epoch_participation"]
            assert st.previous_epoch_participation == case["previous_epoch_participation"]
        else:
            with pytest.raises(AssertionError):
                pspec.process_attestation(st, att)
            assert st.balances == ostate.balances


@pytest.mark.gpu
def test_gpu_get_head_golden(product):
    PS, pspec = product
    _, ostate = _state(PKS)
    ostate.validators[G["get_head"]["inactive_validator"]].exit_epoch = 0
    store = _golden_store(PS, _pstate(PS, ostate))
    assert pspec.get_head(store).hex() == G["get_head"]["head"]
    for r, w in G["get_head"]["weights"].items():
        assert pspec.get_weight(store, bytes.fromhex(r)) == w


@pytest.mark.gpu
def test_gpu_ffg_golden(product):
    """process_justification_and_finalization with the balance sums on the device (b2_ffg_balances) against what the reference's
    own text produced for the same generated states."""
    PS, pspec = product
    _, ostate = _state(PKS)
    for case in G["ffg"]:
        st = scenarios.ffg_case(_pstate(PS, copy.deepcopy(ostate)), case["seed"], mod=PS)
        pspec.process_justification_and_finalization(st)
        assert dict(scenarios.ffg_outcome(st), seed=case["seed"]) == case
