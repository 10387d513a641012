"""GPU test of the prover service end to end (SURVEY.md §8(f) f3): a client replays the requests the reference's
`ProofServiceClient` would send (prover_service_client.rs:186-205: POST JSON, basic auth `admin`), the service proves
through the pool on the device, and the returned proofs / link proofs verify with the pairing against a powers-of-tau SRS
in the reference's ptau layout."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_prove_paths_over_http(ptau_2_16, ptau_g2):
    import renegade_b200 as rb
    from host_circuits import intent_and_balance_validity as val
    from host_circuits import output_balance_validity as obv
    from host_circuits import private_settlement as ps
    from host_circuits import service_routes
    from host_circuits import statements as st
    from host_circuits import valid_balance_create as vbc
    from renegade_b200 import circuit_types as ct
    from renegade_b200 import service as sv
    from renegade_b200.backend import GroupLayout, ProverPool, verify_link_proof
    h, tau_h = ptau_g2
    pool = ProverPool(0, workers=4)
    ctx = pool.context(0)
    params = rb.parse_ptau_file(ctx, ptau_2_16, count=(1 << 14) + 3)
    ct.set_system_srs(ctx, params.powers_of_g, h, tau_h, pool=pool)
    service = sv.ProverService(service_routes.routes(), password="pw", pool=pool)
    server = service.make_server("127.0.0.1", 0)
    threading.Thread(target=server.serve_forever, daemon=True).start()
    try:
        client = sv.ProofServiceClient(f"http://127.0.0.1:{server.server_address[1]}", "pw")
        # VALID BALANCE CREATE -> ProofResponse
        w, s = vbc.create_witness_statement(21)
        code, body = client.send_request("/prove-valid-balance-create", {"statement": sv.to_json(s), "witness": sv.to_json(w)})
        assert code == 200 and set(body) == {"proof"}
        ct.verify_singleprover_proof(st.ValidBalanceCreate, s, sv.decode_proof(body["proof"]))
        # an unsatisfied instance comes back as a prover error, and the service keeps serving
        _, s_other = vbc.create_witness_statement(22)
        code, body = client.send_request("/prove-valid-balance-create", {"statement": sv.to_json(s_other), "witness": sv.to_json(w)})
        assert code == 500 and "ProverError" in body["error"]
        # the private match: validity + output-balance proofs (ProofAndHintResponse), then the settlement request carrying
        # their hints (PrivateSettlementProofResponse)
        parties, _ = ps.create_witness_statement(seed=61)
        validity = [val.create_witness_statement(seed=70 + i, intent=parties[i].intent, balance=parties[i].input_balance)
                    for i in (0, 1)]
        out_validity = [obv.create_witness_statement(80 + i, parties[i].output_balance) for i in (0, 1)]
        parties, statement = ps.create_witness_statement(
            seed=61, linked=[(validity[i][0].new_amount_public_share, validity[i][0].post_match_balance_shares,
                              out_validity[i][0].post_match_balance_shares) for i in (0, 1)])
        results = {}

        def ask(key, path, w_, s_):
            results[key] = client.send_request(path, {"statement": sv.to_json(s_), "witness": sv.to_json(w_)})
        threads = [threading.Thread(target=ask, args=(("v", i), "/prove-intent-and-balance-validity", *validity[i])) for i in (0, 1)] + \
                  [threading.Thread(target=ask, args=(("o", i), "/prove-output-balance-validity", *out_validity[i])) for i in (0, 1)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        hints = {}
        for (kind, i), (code, body) in results.items():
            assert code == 200 and set(body) == {"proof", "link_hint"}
            C, (_, s_) = (st.IntentAndBalanceValidityCircuit, validity[i]) if kind == "v" else (st.OutputBalanceValidityCircuit, out_validity[i])
            ct.verify_singleprover_proof(C, s_, sv.decode_proof(body["proof"]))
            hints[(kind, i)] = body["link_hint"]
        req = {"statement": sv.to_json(statement), "witness": sv.to_json(parties),
               "validity_link_hint_0": hints[("v", 0)], "validity_link_hint_1": hints[("v", 1)],
               "output_balance_link_hint_0": hints[("o", 0)], "output_balance_link_hint_1": hints[("o", 1)]}
        code, body = client.send_request("/prove-intent-and-balance-private-settlement", req)
        assert code == 200 and set(body) == {"proof", "validity_link_proof_0", "validity_link_proof_1",
                                             "output_balance_link_proof_0", "output_balance_link_proof_1"}
        S = st.IntentAndBalancePrivateSettlementCircuit
        sp = sv.decode_proof(body["proof"])
        ct.verify_singleprover_proof(S, statement, sp)
        layouts = S.get_circuit_layout()
        s_comm = np.array(sp.wires_poly_comms[0], dtype=np.uint64)
        for field, key, gid in (("validity_link_proof_0", ("v", 0), ps.PARTY_LINKS[0]), ("validity_link_proof_1", ("v", 1), ps.PARTY_LINKS[1]),
                                ("output_balance_link_proof_0", ("o", 0), ps.OUTPUT_LINKS[0]),
                                ("output_balance_link_proof_1", ("o", 1), ps.OUTPUT_LINKS[1])):
            lay = GroupLayout(layouts[gid].alignment, layouts[gid].offset, layouts[gid].size)
            other = sv.decode_link_hint(hints[key])
            assert verify_link_proof(other.linking_wire_comm, s_comm, sv.decode_link_proof(body[field]), lay, h, tau_h)
        assert service.stats["proofs"] >= 6 and service.stats["link_proofs"] == 4
    finally:
        server.shutdown()
        ct.clear_key_cache()
        pool.close()


def _serve(ptau_2_16, ptau_g2, flow):
    """A prover service over a 3-worker pool on device 0 with a powers-of-tau SRS; `flow(client, service)` drives it."""
    import renegade_b200 as rb
    from host_circuits import service_routes
    from renegade_b200 import circuit_types as ct
    from renegade_b200 import service as sv
    from renegade_b200.backend import ProverPool
    h, tau_h = ptau_g2
    pool = ProverPool(0, workers=3)
    ctx = pool.context(0)
    params = rb.parse_ptau_file(ctx, ptau_2_16, count=(1 << 14) + 3)
    ct.set_system_srs(ctx, params.powers_of_g, h, tau_h, pool=pool)
    service = sv.ProverService(service_routes.routes(), password="pw", pool=pool)
    server = service.make_server("127.0.0.1", 0)
    threading.Thread(target=server.serve_forever, daemon=True).start()
    try:
        flow(sv.ProofServiceClient(f"http://127.0.0.1:{server.server_address[1]}", "pw"), service)
    finally:
        server.shutdown()
        ct.clear_key_cache()
        pool.close()


def test_state_update_paths_over_http(ptau_2_16, ptau_g2):
    """VALID DEPOSIT, VALID WITHDRAWAL, VALID ORDER CANCELLATION, VALID NOTE REDEMPTION and the two PUBLIC fee payments
    (`ProofResponse` paths, prover_service_client.rs:101-147) through the service on the device: the proofs verify with the
    pairing under the circuits' cached keys; a request whose statement does not belong to its witness comes back as a
    prover error.  (The same flow runs on the CPU with the oracle prover in tests/test_service_flows_cpu.py.)"""
    import service_flows
    _serve(ptau_2_16, ptau_g2, service_flows.plain_proof_paths)


def test_intent_only_paths_over_http(ptau_2_16, ptau_g2):
    """The intent-only flow as the relayer drives it: INTENT ONLY VALIDITY and FIRST FILL VALIDITY (`ProofAndHintResponse`),
    then INTENT ONLY PUBLIC / BOUNDED SETTLEMENT with the validity proof's hint (`SettlementProofResponse {proof, link_proof}`,
    api_types.rs:97-104, 279-299); link proofs between circuits of 2^13 / 2^11 and 2^9 rows verify with the pairing."""
    import service_flows
    _serve(ptau_2_16, ptau_g2, lambda client, service: service_flows.intent_only_flow(client, service, ptau_g2))


def test_public_settlement_paths_over_http(ptau_2_16, ptau_g2):
    """INTENT AND BALANCE PUBLIC / BOUNDED SETTLEMENT with the party's validity and output-balance hints
    (`PublicSettlementProofResponse`, api_types.rs:126-137, 238-277)."""
    import service_flows
    _serve(ptau_2_16, ptau_g2, lambda client, service: service_flows.public_settlement_flow(client, service, ptau_g2))
