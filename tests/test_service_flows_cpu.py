"""CPU: the prover service's request flows for the later statements, end to end — HTTP, codec, routing, the
`SingleProverCircuit` surface with its key cache, link proofs, and the product's pairing verifier on a powers-of-tau
SRS — with the ORACLE prover standing in for the device (test infrastructure: the device prover is byte-identical to it,
tests/test_gpu_plonk.py).  The very same flows run against the device in tests/test_gpu_service.py."""
import threading

import numpy as np
import pytest

import service_flows
from renegade_b200 import _lib, backend
from renegade_b200 import circuit_types as ct
from renegade_b200 import service as sv


class _OracleKey:
    """What `circuit_types` reads off a proving key."""

    def __init__(self, log_n, num_inputs, k, opk):
        self.log_n, self.num_inputs, self.k, self.opk = log_n, num_inputs, k, opk
        self.selector_comms, self.sigma_comms = opk["selector_comms"], opk["sigma_comms"]

    def free(self):
        pass


def _oracle_snark(oracle):
    class OracleSnark:
        verify = staticmethod(backend.PlonkKzgSnark.verify)   # the product's host verifier, unchanged

        @staticmethod
        def preprocess(ctx, srs, log_n, num_inputs, selectors, perm, k):
            return _OracleKey(log_n, num_inputs, k, oracle.plonk_preprocess(log_n, selectors, perm, k, srs[:(1 << log_n) + 3]))

        @staticmethod
        def prove_with_link_hint(ctx, pk, wires, pub_inputs, blinders):
            rc, proof, _, link = oracle.plonk_prove(pk.log_n, pk.num_inputs, pk.k, pk.opk, wires, pub_inputs, blinders,
                                                    ct.system_srs().powers_of_g[:(1 << pk.log_n) + 3], True)
            if rc != 0:
                raise _lib.B200Error(-7, "oracle prover: the quotient is not a polynomial (unsatisfied circuit)")
            p = backend.B200Proof.from_buffer_copy(bytes(proof))
            return p, backend.LinkingHint(linking_wire_poly=link, linking_wire_comm=np.array(p.wires_poly_comms[0], dtype=np.uint64))
    return OracleSnark


@pytest.fixture()
def served(oracle, ptau_2_16, ptau_g2, monkeypatch):
    """(client, service): the product's service + routes + circuit surface, the oracle where the device would prove."""
    from host_circuits import service_routes
    h, tau_h = ptau_g2
    n_srs = (1 << 14) + 3
    srs = np.frombuffer(ptau_2_16[80:80 + 64 * n_srs], dtype=np.uint64).reshape(n_srs, 8).copy()
    monkeypatch.setattr(ct, "PlonkKzgSnark", _oracle_snark(oracle))

    def link_proofs(ctx, bases, a, b, layout):
        rc, lp, eta = oracle.plonk_link(a.linking_wire_poly, b.linking_wire_poly, a.linking_wire_comm, b.linking_wire_comm,
                                        layout.alignment, layout.offset, layout.size, bases)
        if rc != 0:
            raise _lib.B200Error(-7, "oracle link: the division by the group's vanishing polynomial is not exact")
        return backend.B200LinkProof.from_buffer_copy(bytes(lp)), eta
    monkeypatch.setattr(backend, "link_proofs", link_proofs)
    ct.set_system_srs(None, srs, h, tau_h, pool=None)
    service = sv.ProverService(service_routes.routes(), password="pw")
    server = service.make_server("127.0.0.1", 0)
    threading.Thread(target=server.serve_forever, daemon=True).start()
    try:
        yield sv.ProofServiceClient(f"http://127.0.0.1:{server.server_address[1]}", "pw"), service
    finally:
        server.shutdown()
        ct.clear_key_cache()
        ct._SYSTEM_SRS = None


def test_plain_proof_paths(served):
    service_flows.plain_proof_paths(*served, negatives="first")


def test_intent_only_flow(served, ptau_g2):
    service_flows.intent_only_flow(*served, ptau_g2)


def test_public_settlement_flow(served, ptau_g2):
    service_flows.public_settlement_flow(*served, ptau_g2, which=("public",))


def test_private_match_flow(served, ptau_g2):
    service_flows.private_match_flow(*served, ptau_g2)


def test_structure_fingerprint_guards_the_key_cache(served, monkeypatch):
    """Keys are cached by circuit name and, per proof, only the value tables are arithmetized (`wires_only`, SURVEY 8(f) f4).
    A synthesis that yields OTHER gates / wiring than the key was preprocessed from — same domain size, same number of
    public inputs, so the shape check alone would let it through — is refused as `ProverError::Circuit`."""
    from host_circuits import state_updates as su
    from host_circuits import statements as st
    w, s = su.create_deposit_witness_statement(71)
    proof, _ = st.ValidDeposit.prove_with_link_hint(w, s)          # sets the key and its fingerprint up, proves wires-only
    ct.verify_singleprover_proof(st.ValidDeposit, s, proof)
    assert ct._CIRCUIT_STRUCTURE[st.ValidDeposit.name()] != 0
    _, s_other = su.create_deposit_witness_statement(73)           # the right circuit with somebody else's statement: the PROVER's
    with pytest.raises(ct.ProverError) as err:                      # refusal (WrongQuotientPolyDegree), not a structure error
        st.ValidDeposit.prove_with_link_hint(w, s_other)
    assert err.value.kind == "Plonk"
    w2, s2 = su.create_withdrawal_witness_statement(72)             # 2^13 rows and 8 public inputs as well
    monkeypatch.setattr(st.ValidDeposit, "synthesize", classmethod(lambda cls, w_, s_, lay: su.ValidWithdrawal.build(w_, s_)))
    with pytest.raises(ct.ProverError, match="gates / wiring differ"):
        st.ValidDeposit.prove_with_link_hint(w2, s2)
