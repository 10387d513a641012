"""GPU tests of the batch verifier (`b200_plonk_batch_verify`, renegade_b200/csrc/batch_verify.cu): PlonK proofs and
link proofs checked on the device and folded into one pairing product.  Its per-item operands must equal the oracle's
byte for byte, its per-item verdicts must equal the single host verifiers' (`b200_plonk_verify` /
`b200_plonk_verify_link`) for every tampering those verifiers' tests use, and the random weights must be real: two
wrong openings whose errors cancel in an unweighted sum are still caught."""
import ctypes as C

import numpy as np
import pytest

from renegade_b200 import synth
from renegade_b200.backend import (B200BatchLink, B200BatchProof, B200BatchVk, B200LinkProof, B200Proof, GroupLayout,
                                   PlonkKzgSnark, VerifyingKey, link_proofs, verify_link_proof)

pytestmark = pytest.mark.gpu

LAYOUT = GroupLayout(alignment=8, offset=40, size=12)


@pytest.fixture(scope="module")
def srs(ctx, ptau_2_16):
    """The 2^16 + 3 powers of conftest's ptau file on the device (its [tau]_2 is ptau_g2's)."""
    pts = np.frombuffer(ptau_2_16[80:], dtype=np.uint64).reshape(-1, 8)
    bases = ctx.load_bases(pts)
    yield pts, bases
    bases.free()


def _prove(ctx, srs, ptau_g2, log_n, num_inputs, seed, link_vals=None):
    circ = synth.synth_circuit(log_n, num_inputs=num_inputs, seed=seed, check=False,
                               link=None if link_vals is None else (LAYOUT.alignment, LAYOUT.offset, link_vals))
    pk = PlonkKzgSnark.preprocess(ctx, srs[1], log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
    proof, hint = PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, synth.splitmix_blinders(seed))
    vk = VerifyingKey.from_proving_key(pk, *ptau_g2)
    pk.free()
    return circ, vk, proof, hint


@pytest.fixture(scope="module")
def items(ctx, srs, ptau_g2, pyoracle):
    """Two proofs of different sizes and public-input counts that share a link group, and their link proof."""
    vals = [(i * 0x9E3779B97F4A7C15 + 77) % pyoracle.R for i in range(LAYOUT.size)]
    a = _prove(ctx, srs, ptau_g2, 10, 5, 21, vals)
    b = _prove(ctx, srs, ptau_g2, 11, 3, 22, vals)
    lp, eta = link_proofs(ctx, srs[1], a[3], b[3], LAYOUT)
    link = (a[3].linking_wire_comm, b[3].linking_wire_comm, lp, LAYOUT)
    return a, b, link, eta


def _single(item, g2):
    """The single host verifiers' verdict on one ("proof", vk, pub_inputs, proof) or ("link", ...) item."""
    if item[0] == "proof":
        _, vk, pi, proof = item
        return PlonkKzgSnark.verify(vk, pi, proof)
    _, ca, cb, lp, lay = item
    return verify_link_proof(ca, cb, lp, lay, *g2)


def _batch(ctx, batch, g2):
    proofs = [it for it in batch if it[0] == "proof"]
    links = [it[1:] for it in batch if it[0] == "link"]
    return PlonkKzgSnark.batch_verify(ctx, [p[1] for p in proofs], [p[2] for p in proofs], [p[3] for p in proofs],
                                      links, g2=g2)


def _g1(pyoracle, xy):
    return pyoracle.decode_g1_mont(np.ascontiguousarray(xy, dtype=np.uint64).tobytes(), 0)


def _enc(pyoracle, p):
    return np.frombuffer(pyoracle.encode_g1_mont(p), dtype=np.uint64)


@pytest.mark.parametrize("log_n,num_inputs", [(3, 0), (3, 2), (10, 0), (10, 7), (16, 17)])
def test_plonk_operands_match_the_oracle(ctx, oracle, srs, ptau_g2, log_n, num_inputs):
    circ, vk, proof, _ = _prove(ctx, srs, ptau_g2, log_n, num_inputs, 40 + log_n + num_inputs)
    ok, ops = PlonkKzgSnark.batch_verify(ctx, [vk], [circ.pub_inputs], [proof], want_operands=True)
    assert ok.tolist() == [True]
    opk = {"selector_comms": np.ascontiguousarray(vk.selector_comms, dtype=np.uint64),
           "sigma_comms": np.ascontiguousarray(vk.sigma_comms, dtype=np.uint64)}
    (a, a_inf), (b, b_inf) = oracle.plonk_verify_operands(log_n, circ.num_inputs, circ.k, opk, circ.pub_inputs,
                                                          oracle.PlonkProof.from_buffer_copy(bytes(proof)))
    assert (ops[0, 0] == (0 if a_inf else a)).all()
    assert (ops[0, 1] == (0 if b_inf else b)).all()


def test_link_operands_match_the_oracle(ctx, oracle, pyoracle, srs, ptau_g2, items):
    """Link operands of the test's 2^10 <-> 2^11 link and of a 2^13 <-> 2^9 link: A = pi,
    B = C1 - C2 - Z_D(eta) Cq + eta pi with eta from the oracle's link prover."""
    py = pyoracle
    a, b, link, _ = items
    lay2 = GroupLayout(alignment=9, offset=3, size=17)
    vals = [(i * 7919 + 5) % py.R for i in range(lay2.size)]
    big = synth.synth_circuit(13, num_inputs=4, seed=31, link=(lay2.alignment, lay2.offset, vals))
    small = synth.synth_circuit(9, num_inputs=2, seed=32, link=(lay2.alignment, lay2.offset, vals))
    hints = []
    for circ, seed in ((big, 31), (small, 32)):
        pk = PlonkKzgSnark.preprocess(ctx, srs[1], circ.log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
        _, hint = PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, synth.splitmix_blinders(seed))
        pk.free()
        hints.append(hint)
    lp2, _ = link_proofs(ctx, srs[1], hints[0], hints[1], lay2)
    links = [link, (hints[0].linking_wire_comm, hints[1].linking_wire_comm, lp2, lay2)]
    ok, ops = PlonkKzgSnark.batch_verify(ctx, [a[1]], [a[0].pub_inputs], [a[2]], links, want_operands=True)
    assert ok.tolist() == [True, True, True]
    for j, (ca, cb, lp, lay) in enumerate(links):
        h1 = hints if j == 1 else (a[3], b[3])
        rc, olp, eta = oracle.plonk_link(h1[0].linking_wire_poly, h1[1].linking_wire_poly, ca, cb, lay.alignment,
                                         lay.offset, lay.size, srs[0])
        assert rc == 0 and (olp.to_array() == lp.to_array()).all()
        eta_i = py.from_mont(oracle.limbs_to_int(eta), py.R)
        g = py.domain_generator(lay.alignment)
        zd = 1
        for i in range(lay.size):
            zd = zd * (eta_i - pow(g, lay.offset + i, py.R)) % py.R
        pi = _g1(py, lp.opening_proof)
        want_b = py.g1_add(py.g1_add(_g1(py, ca), py.g1_neg(_g1(py, cb))),
                           py.g1_add(py.g1_mul(_g1(py, lp.quotient_commitment), (-zd) % py.R), py.g1_mul(pi, eta_i)))
        assert (ops[1 + j, 0] == np.asarray(lp.opening_proof, dtype=np.uint64)).all()
        assert (ops[1 + j, 1] == _enc(py, want_b)).all()


def test_honest_mixed_batch_is_accepted(ctx, items):
    a, b, link, _ = items
    ok = PlonkKzgSnark.batch_verify(ctx, [a[1], b[1], a[1]], [a[0].pub_inputs, b[0].pub_inputs, a[0].pub_inputs],
                                    [a[2], b[2], a[2]], [link, link])
    assert ok.tolist() == [True] * 5


def _tamperings(items, pyoracle):
    """(name, bad item) for every tampering of the single verifiers' tests; the honest items are items' proofs."""
    a, b, link, _ = items
    ca, cb, lp, lay = link
    out = []
    p = B200Proof.from_buffer_copy(bytes(a[2]))
    p.wire_sigma_evals[1][0] ^= 1
    out.append(("evaluation", ("proof", a[1], a[0].pub_inputs, p)))
    p = B200Proof.from_buffer_copy(bytes(a[2]))
    for j in range(8):
        p.wires_poly_comms[0][j], p.wires_poly_comms[1][j] = p.wires_poly_comms[1][j], p.wires_poly_comms[0][j]
    out.append(("swapped commitments", ("proof", a[1], a[0].pub_inputs, p)))
    pi = a[0].pub_inputs.copy()
    pi[2, 0] ^= np.uint64(1)
    out.append(("public input", ("proof", a[1], pi, a[2])))
    out.append(("public-input count", ("proof", a[1], a[0].pub_inputs[:-1], a[2])))
    out.append(("other circuit's key", ("proof", b[1], a[0].pub_inputs[:3], a[2])))
    p = B200Proof.from_buffer_copy(bytes(a[2]))
    p.opening_proof[0] ^= 1
    out.append(("off-curve proof point", ("proof", a[1], a[0].pub_inputs, p)))
    sel = np.array(a[1].selector_comms, dtype=np.uint64).reshape(13, 8).copy()
    sel[3, 0] ^= np.uint64(1)
    bad_vk = VerifyingKey(a[1].log_n, a[1].num_inputs, a[1].k, sel, a[1].sigma_comms, a[1].g2_h, a[1].g2_tau_h)
    out.append(("off-curve key point", ("proof", bad_vk, a[0].pub_inputs, a[2])))
    out.append(("unshared group", ("link", ca, cb, lp, GroupLayout(lay.alignment, lay.offset + 1, lay.size))))
    return out


@pytest.mark.parametrize("n", [1, 7, 64])
@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_verdicts_equal_the_single_verifiers(ctx, items, pyoracle, ptau_g2, n, where):
    a, b, link, _ = items
    honest_proofs = [("proof", a[1], a[0].pub_inputs, a[2]), ("proof", b[1], b[0].pub_inputs, b[2])]
    honest_link = ("link",) + tuple(link)
    for name, bad in _tamperings(items, pyoracle):
        kind = bad[0]
        n_links = n // 3 if kind == "proof" else n - n // 3
        n_proofs = n - n_links
        proofs = [honest_proofs[i % 2] for i in range(n_proofs)]
        links = [honest_link] * n_links
        group = proofs if kind == "proof" else links
        at = {"first": 0, "middle": len(group) // 2, "last": len(group) - 1}[where]
        group[at] = bad
        batch = proofs + links
        want = [_single(it, ptau_g2) for it in batch]
        got = _batch(ctx, batch, ptau_g2)
        assert not all(want), name
        assert got.tolist() == want, name
        assert not got.all(), name


def test_the_weights_are_real(ctx, pyoracle, items, ptau_g2):
    """pi + G and pi - G: the unweighted sums of A and B over the two items equal the honest ones (B moves by
    eta G and -eta G), so an unweighted batch would accept; the weighted one rejects both."""
    py = pyoracle
    _, _, (ca, cb, lp, lay), _ = items
    pi = _g1(py, lp.opening_proof)
    bad = []
    for s in (py.G1_GEN, py.g1_neg(py.G1_GEN)):
        q = B200LinkProof.from_buffer_copy(bytes(lp))
        enc = _enc(py, py.g1_add(pi, s))
        for j in range(8):
            q.opening_proof[j] = int(enc[j])
        bad.append(q)
    got = PlonkKzgSnark.batch_verify(ctx, [items[0][1]], [items[0][0].pub_inputs], [items[0][2]],
                                     [(ca, cb, q, lay) for q in bad])
    assert got.tolist() == [True, False, False]
    assert not verify_link_proof(ca, cb, bad[0], lay, *ptau_g2)
    assert not verify_link_proof(ca, cb, bad[1], lay, *ptau_g2)


def test_1024_items(ctx, items):
    a, b, link, _ = items
    n_proofs, n_links = 768, 256
    vks = [(a, b)[i % 2][1] for i in range(n_proofs)]
    pis = [(a, b)[i % 2][0].pub_inputs for i in range(n_proofs)]
    proofs = [(a, b)[i % 2][2] for i in range(n_proofs)]
    links = [link] * n_links
    assert PlonkKzgSnark.batch_verify(ctx, vks, pis, proofs, links).all()
    ca, cb, lp, lay = link
    bad_link = B200LinkProof.from_buffer_copy(bytes(lp))
    bad_link.quotient_commitment, bad_link.opening_proof = lp.opening_proof, lp.quotient_commitment
    links[777 - n_proofs] = (ca, cb, bad_link, lay)
    got = PlonkKzgSnark.batch_verify(ctx, vks, pis, proofs, links)
    assert np.flatnonzero(~got).tolist() == [777]


def _raw(ctx, vks, proofs, links, g2_h, g2_tau_h):
    vt = (B200BatchVk * max(len(vks), 1))(*vks)
    pt = (B200BatchProof * max(len(proofs), 1))(*proofs)
    lt = (B200BatchLink * max(len(links), 1))(*links)
    ok = C.c_int(7)
    n = C.c_size_t(0)
    rc = ctx._lib.b200_plonk_batch_verify(ctx._h, vt, len(vks), pt, len(proofs), lt, len(links),
                                          g2_h.ctypes.data_as(C.c_void_p), g2_tau_h.ctypes.data_as(C.c_void_p),
                                          C.byref(ok), None, None, C.byref(n))
    return rc, ok.value, n.value


def test_argument_errors_leave_the_context_usable(ctx, oracle, srs, ptau_g2, items):
    a, b, link, _ = items
    h, tau_h = (np.ascontiguousarray(x, dtype=np.uint64) for x in ptau_g2)
    vk = a[1]
    arrs = [np.ascontiguousarray(vk.k, dtype=np.uint64), np.ascontiguousarray(vk.selector_comms, dtype=np.uint64),
            np.ascontiguousarray(vk.sigma_comms, dtype=np.uint64)]
    pi = np.ascontiguousarray(a[0].pub_inputs, dtype=np.uint64)

    def bvk(log_n=vk.log_n):
        return B200BatchVk(log_n, vk.num_inputs, *(x.ctypes.data_as(C.c_void_p) for x in arrs))

    def bpr(idx=0):
        return B200BatchProof(idx, pi.ctypes.data_as(C.c_void_p), pi.shape[0], C.addressof(a[2]))
    ca, cb, lp, lay = link
    ca, cb = (np.ascontiguousarray(x, dtype=np.uint64) for x in (ca, cb))

    def bln(alignment=lay.alignment, size=lay.size, proof=True):
        return B200BatchLink(ca.ctypes.data_as(C.c_void_p), cb.ctypes.data_as(C.c_void_p), alignment, lay.offset, size,
                             C.addressof(lp) if proof else None)
    rc, ok, npair = _raw(ctx, [bvk()], [bpr()], [bln()], h, tau_h)
    assert (rc, ok, npair) == (0, 1, 1)
    for args in (([bvk()], [bpr(1)], []), ([bvk(29)], [bpr()], []), ([bvk()], [bpr()], [bln(alignment=29)]),
                 ([bvk()], [bpr()], [bln(size=0)]), ([bvk()], [bpr()], [bln(proof=False)]), ([bvk()], [], [])):
        assert _raw(ctx, *args, h, tau_h)[0] == -1
    bad_h = h.copy()
    bad_h[0] ^= np.uint64(1)
    assert _raw(ctx, [bvk()], [bpr()], [], bad_h, tau_h)[0] == -5
    assert _raw(ctx, [bvk()], [bpr()], [], h, bad_h)[0] == -5
    # the context still proves what the oracle proves
    log_n = 6
    circ = synth.synth_circuit(log_n, num_inputs=3, seed=5, check=True)
    n = 1 << log_n
    pk = PlonkKzgSnark.preprocess(ctx, srs[1], log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
    proof, _ = PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, synth.splitmix_blinders(5))
    pk.free()
    opk = oracle.plonk_preprocess(log_n, circ.selectors, circ.perm, circ.k, np.ascontiguousarray(srs[0][:n + 3]))
    rc, oproof, _, _ = oracle.plonk_prove(log_n, circ.num_inputs, circ.k, opk, circ.wires, circ.pub_inputs,
                                         synth.splitmix_blinders(5), np.ascontiguousarray(srs[0][:n + 3]), True)
    assert rc == 0 and bytes(proof) == bytes(oproof)


def test_private_match_bundle_in_one_call(ctx, srs, ptau_g2):
    """The 5 proofs and 4 link proofs of one private match (the flow of test_gpu_real_srs.py) in one batch."""
    from host_circuits import intent_and_balance_validity as val
    from host_circuits import output_balance_validity as obv
    from host_circuits import private_settlement as ps
    from host_circuits import statements as st
    from renegade_b200 import circuit_types as ct
    h, tau_h = ptau_g2
    ct.set_system_srs(ctx, srs[1], h, tau_h)
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
        vks, pis, proofs, links = [S.verifying_key()], [S.statement_scalars(statement)], [sp], []
        layouts = S.get_circuit_layout()
        for i in (0, 1):
            for Cc, (w, s_), gid in ((st.IntentAndBalanceValidityCircuit, validity[i], ps.PARTY_LINKS[i]),
                                     (st.OutputBalanceValidityCircuit, out_validity[i], ps.OUTPUT_LINKS[i])):
                p, hint = ct.singleprover_prove_with_hint(Cc, w, s_)
                vks.append(Cc.verifying_key())
                pis.append(Cc.statement_scalars(s_))
                proofs.append(p)
                lay = GroupLayout(layouts[gid].alignment, layouts[gid].offset, layouts[gid].size)
                lp, _ = link_proofs(ctx, srs[1], hint, sh, lay)
                links.append((hint.linking_wire_comm, sh.linking_wire_comm, lp, lay))
        assert PlonkKzgSnark.batch_verify(ctx, vks, pis, proofs, links).tolist() == [True] * 9
    finally:
        ct.clear_key_cache()


def test_mismatched_arguments_raise(ctx, items):
    a, b, link, _ = items
    with pytest.raises(ValueError):
        PlonkKzgSnark.batch_verify(ctx, [a[1]], [], [a[2]])
    other = VerifyingKey(b[1].log_n, b[1].num_inputs, b[1].k, b[1].selector_comms, b[1].sigma_comms,
                         b[1].g2_tau_h, b[1].g2_h)
    with pytest.raises(ValueError):
        PlonkKzgSnark.batch_verify(ctx, [a[1], other], [a[0].pub_inputs, b[0].pub_inputs], [a[2], b[2]])
