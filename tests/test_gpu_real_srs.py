"""GPU parity on a powers-of-tau SRS at the BASELINE size: the device prover commits against 2^16 + 3 powers read from a
ptau file in the reference's layout (conftest `ptau_2_16`; the reference's own powers are pinned at n = 2^8 by
test_pairing.py) and the proof must pass the pairing check against the matching [tau]_2 — the prover never sees tau, so
nothing but a correct KZG opening passes — with the product verifier (`b200_plonk_verify`, host pairing) and with the
independent pure-Python pairing of the oracle.  Then the `SingleProverCircuit` surface end to end on the same SRS: the restated reference statements prove, verify and link the
way circuits-core's own tests do (`singleprover_prove_and_verify`, proof_linking/*.rs prove -> link -> verify)."""
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def real_srs(ctx, ptau_2_16):
    import renegade_b200 as rb
    params = rb.parse_ptau_file(ctx, ptau_2_16, count=(1 << 16) + 3)
    return params.powers_of_g


def test_2_16_proof_on_the_reference_srs_passes_the_pairing_check(ctx, oracle, real_srs, ptau_g2):
    from renegade_b200 import synth
    from renegade_b200.backend import PlonkKzgSnark, VerifyingKey
    h, tau_h = ptau_g2
    log_n = 16
    circ = synth.synth_circuit(log_n, num_inputs=17, seed=0xB200, check=False)
    pk = PlonkKzgSnark.preprocess(ctx, real_srs, log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
    proof, _ = PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, synth.splitmix_blinders(2016))
    vk = VerifyingKey.from_proving_key(pk, h, tau_h)
    assert PlonkKzgSnark.verify(vk, circ.pub_inputs, proof)
    # a flipped evaluation or public input does not
    from renegade_b200.backend import B200Proof
    bad = B200Proof.from_buffer_copy(bytes(proof))
    bad.wires_evals[2][1] ^= 1
    assert not PlonkKzgSnark.verify(vk, circ.pub_inputs, bad)
    pi2 = circ.pub_inputs.copy()
    pi2[5, 0] ^= np.uint64(1)
    assert not PlonkKzgSnark.verify(vk, pi2, proof)
    # independent check: the oracle's verifier equation + the pure-Python pairing
    import bn254_pairing_py as pr
    raw = h.tobytes() + tau_h.tobytes()
    g2 = (pr.decode_g2_mont(raw, 0), pr.decode_g2_mont(raw, 1))
    opk = {"selector_comms": pk.selector_comms, "sigma_comms": pk.sigma_comms}
    assert oracle.plonk_verify_pairing(log_n, circ.num_inputs, circ.k, opk, circ.pub_inputs,
                                       oracle.PlonkProof.from_buffer_copy(bytes(proof)), *g2)
    pk.free()


def test_single_prover_circuit_surface_on_the_reference_srs(ctx, real_srs, ptau_g2):
    """circuits-core's own test shape: `singleprover_prove_and_verify::<C>(witness, statement)` for the restated
    statements, keys from the cache keyed by `C::name()` (traits.rs:1187-1201 checks the sharing), a wrong statement is
    refused by the verifier, an unsatisfied witness by the prover."""
    from host_circuits import statements as st
    from host_circuits import valid_balance_create as vbc
    from renegade_b200 import circuit_types as ct
    h, tau_h = ptau_g2
    ct.set_system_srs(ctx, real_srs, h, tau_h)
    try:
        w, s = vbc.create_witness_statement(7)
        ct.singleprover_prove_and_verify(st.ValidBalanceCreate, w, s)
        pk1, vk1 = ct.setup_preprocessed_keys(st.ValidBalanceCreate)
        pk2, vk2 = ct.setup_preprocessed_keys(st.ValidBalanceCreate)
        assert pk1 is pk2 and vk1 is vk2                     # one key pair per circuit name
        proof = ct.singleprover_prove(st.ValidBalanceCreate, w, s, rng=random.Random(5))
        again = ct.singleprover_prove(st.ValidBalanceCreate, w, s, rng=random.Random(5))
        assert bytes(proof) == bytes(again)                  # injected randomness makes the proof reproducible
        ct.verify_singleprover_proof(st.ValidBalanceCreate, s, proof)
        w2, s2 = vbc.create_witness_statement(8)
        with pytest.raises(ct.VerifierError):
            ct.verify_singleprover_proof(st.ValidBalanceCreate, s2, proof)
        with pytest.raises(ct.ProverError) as err:           # witness of one instance, statement of another
            ct.singleprover_prove(st.ValidBalanceCreate, w, s2)
        assert err.value.kind == "Plonk"
    finally:
        ct.clear_key_cache()


def test_private_match_bundle_through_the_surface(ctx, real_srs, ptau_g2):
    """Prove -> link -> verify for one private match (native_proof_manager.rs:526-584, 726-782) with the typed surface:
    two INTENT AND BALANCE VALIDITY, two OUTPUT BALANCE VALIDITY and the PRIVATE SETTLEMENT proof, the four link proofs,
    everything checked with the pairing against the SRS's [tau]_2."""
    from host_circuits import intent_and_balance_validity as val
    from host_circuits import output_balance_validity as obv
    from host_circuits import private_settlement as ps
    from host_circuits import statements as st
    from renegade_b200 import circuit_types as ct
    from renegade_b200.backend import GroupLayout, link_proofs, verify_link_proof
    h, tau_h = ptau_g2
    ct.set_system_srs(ctx, real_srs, h, tau_h)
    try:
        parties, _ = ps.create_witness_statement(seed=61)
        validity = [val.create_witness_statement(seed=70 + i, intent=parties[i].intent, balance=parties[i].input_balance)
                    for i in (0, 1)]
        out_validity = [obv.create_witness_statement(80 + i, parties[i].output_balance) for i in (0, 1)]
        parties, statement = ps.create_witness_statement(
            seed=61, linked=[(validity[i][0].new_amount_public_share, validity[i][0].post_match_balance_shares,
                              out_validity[i][0].post_match_balance_shares) for i in (0, 1)])
        S = st.IntentAndBalancePrivateSettlementCircuit
        sp, sh = ct.singleprover_prove_with_hint(S, parties, statement)
        ct.verify_singleprover_proof(S, statement, sp)
        layouts = S.get_circuit_layout()
        for i in (0, 1):
            for C, (w, s_), gid in ((st.IntentAndBalanceValidityCircuit, validity[i], ps.PARTY_LINKS[i]),
                                    (st.OutputBalanceValidityCircuit, out_validity[i], ps.OUTPUT_LINKS[i])):
                p, hint = ct.singleprover_prove_with_hint(C, w, s_)
                ct.verify_singleprover_proof(C, s_, p)
                lay = GroupLayout(layouts[gid].alignment, layouts[gid].offset, layouts[gid].size)
                lp, _ = link_proofs(ctx, real_srs, hint, sh, lay)
                assert verify_link_proof(hint.linking_wire_comm, sh.linking_wire_comm, lp, lay, h, tau_h)
                other = ps.PARTY_LINKS[1 - i] if gid in ps.PARTY_LINKS else ps.OUTPUT_LINKS[1 - i]
                wrong = GroupLayout(layouts[other].alignment, layouts[other].offset, layouts[other].size)
                assert not verify_link_proof(hint.linking_wire_comm, sh.linking_wire_comm, lp, wrong, h, tau_h)
    finally:
        ct.clear_key_cache()
