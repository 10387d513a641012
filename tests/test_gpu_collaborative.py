"""GPU parity of the collaborative prover (renegade_b200/collaborative.py on `DeviceBackend`: the C ABI's device-vector
primitives, NTT and MSM): with 2 and 3 parties holding additive shares of the witness table and of the blinders, the opened
proof is byte-identical to the device single-prover proof (`b200_plonk_prove`) and to the oracle's; then the
`MultiProverCircuit` surface on a powers-of-tau SRS: the VALID-MATCH-class settlement statement proved jointly by two
parties opens to a proof that the pairing verifier accepts under the single-prover circuit's verifying key
(`multiprover_prove_and_verify`, circuits-core/src/lib.rs:166-177)."""
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TAU = 0xB200B200B200


@pytest.mark.parametrize("log_n,parties", [(6, 2), (10, 2), (10, 3)])
def test_device_collaborative_proof_equals_single_prover_proof(ctx, oracle, pyoracle, log_n, parties):
    from renegade_b200 import collaborative as co
    from renegade_b200 import synth
    from renegade_b200.backend import PlonkKzgSnark
    py = pyoracle
    n = 1 << log_n
    circ = synth.synth_circuit(log_n, num_inputs=5, seed=200 + log_n, check=(log_n <= 10))
    tau = oracle.int_to_limbs(py.to_mont(TAU % py.R, py.R))
    srs = oracle.srs_from_tau(tau, n + 3)
    bases = ctx.load_bases(srs)
    bl = synth.splitmix_blinders(90 + log_n)
    pk = PlonkKzgSnark.preprocess(ctx, bases, log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
    single, shint = PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, bl)
    be = co.DeviceBackend(ctx, bases)
    cpk = co.CollaborativeProvingKey.build(be, log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
    assert (cpk.selector_comms == pk.selector_comms).all() and (cpk.sigma_comms == pk.sigma_comms).all()
    wire_shares = co.share_table(np.asarray(circ.wires, dtype=np.uint64).reshape(-1, 4), parties, seed=17)
    blinder_shares = co.share_table(np.asarray(bl, dtype=np.uint64).reshape(-1, 4), parties, seed=18)
    proof, hint, fab = co.MultiproverPlonkKzgSnark.prove_with_link_hint(be, cpk, wire_shares, circ.pub_inputs, blinder_shares)
    assert bytes(proof) == bytes(single)
    assert (hint.linking_wire_poly == shint.linking_wire_poly).all()
    opk = oracle.plonk_preprocess(log_n, circ.selectors, circ.perm, circ.k, srs)
    rc, oproof, _, _ = oracle.plonk_prove(log_n, circ.num_inputs, circ.k, opk, circ.wires, circ.pub_inputs, bl, srs)
    assert rc == 0 and bytes(proof) == bytes(oproof)
    assert fab.multiplications >= 26 * 8 * n
    pk.free()


def test_multiprover_surface_on_the_reference_srs(ctx, ptau_2_16, ptau_g2):
    import renegade_b200 as rb
    from host_circuits import private_settlement as ps
    from host_circuits import statements as st
    from renegade_b200 import circuit_types as ct
    h, tau_h = ptau_g2
    params = rb.parse_ptau_file(ctx, ptau_2_16, count=(1 << 13) + 3)
    ct.set_system_srs(ctx, params.powers_of_g, h, tau_h)
    try:
        parties, statement = ps.create_witness_statement(seed=33)
        C = st.IntentAndBalancePrivateSettlementMultiprover
        ct.multiprover_prove_and_verify(C, parties, statement, parties=2, rng=random.Random(3))
        # the opened proof is the single-prover proof of the same witness and blinders
        circ, shares = C.share_witness_table(parties, statement, 2, seed=5)
        bl = ct.draw_blinders(random.Random(9))
        from renegade_b200.collaborative import share_table
        proof, _ = ct.multiprover_prove_with_hint(C, circ, shares, share_table(bl, 2, seed=6))
        single = ct.singleprover_prove(C.BaseCircuit, parties, statement, rng=random.Random(9))
        assert bytes(proof) == bytes(single)
        ct.verify_singleprover_proof(C.BaseCircuit, statement, proof)
        # shares that are off by one in many places make the joint witness unsatisfying: refused (a single position can
        # be an unconstrained padding / dummy variable, so every 97th entry of the table is disturbed)
        from renegade_b200.fields import limbs_to_scalars, scalars_to_limbs
        bad = limbs_to_scalars(shares[1])
        for i in range(0, len(bad), 97):
            bad[i] = (bad[i] + 1) % ct.SCALAR_FIELD_MODULUS
        with pytest.raises(ct.ProverError):
            ct.multiprover_prove_with_hint(C, circ, [shares[0], scalars_to_limbs(bad)], share_table(bl, 2, seed=6))
    finally:
        ct.clear_key_cache()
