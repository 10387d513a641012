"""The collaborative prover on the device (`b200_mpc_prove`, `b200_mpc_link`): every party, each with its own context,
its shares and dealer preprocessing, ends with the same opened proof as `b200_plonk_prove` on the summed witness and
blinders; refusals reach every party without hanging; the communication accounting matches the protocol's shapes."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TIMEOUT_MS = 60000


@pytest.fixture(scope="module")
def party_ctxs():
    import renegade_b200 as rb
    cs = [rb.Context(0) for _ in range(3)]
    yield cs
    for c in cs:
        c.close()


@pytest.fixture(scope="module")
def srs_points(ptau_2_16):
    return np.frombuffer(ptau_2_16[80:], dtype=np.uint64).reshape(-1, 8)


_setups = {}


def setup(ctx, srs_points, log_n):
    """(circuit, bases, pk, blinders, single proof, single link poly, challenges) for a synthetic circuit of 2^log_n gates."""
    if log_n not in _setups:
        from renegade_b200 import synth
        from renegade_b200.backend import PlonkKzgSnark
        n = 1 << log_n
        circ = synth.synth_circuit(log_n, num_inputs=5, seed=300 + log_n, check=(log_n <= 10))
        bases = ctx.load_bases(srs_points[:n + 3])
        pk = PlonkKzgSnark.preprocess(ctx, bases, log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
        bl = synth.splitmix_blinders(70 + log_n)
        proof, hint, ch = PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, bl, want_challenges=True)
        _setups[log_n] = (circ, bases, pk, bl, proof, hint, ch)
    return _setups[log_n]


def shares(circ, bl, parties, seed=17):
    from renegade_b200 import collaborative as co
    ws = co.share_table(np.asarray(circ.wires, dtype=np.uint64).reshape(-1, 4), parties, seed=seed)
    bs = co.share_table(np.asarray(bl, dtype=np.uint64).reshape(-1, 4), parties, seed=seed + 1)
    return ws, bs


def sum_shares(parts):
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R, limbs_to_scalars, scalars_to_limbs
    ints = [limbs_to_scalars(np.asarray(p, dtype=np.uint64).reshape(-1, 4)) for p in parts]
    return scalars_to_limbs([sum(col) % R for col in zip(*ints)])


def codes(results):
    from renegade_b200._lib import B200Error
    return [r.code if isinstance(r, B200Error) else (0 if not isinstance(r, Exception) else "exc") for r in results]


def expected_bytes(n, nc, P=None):
    """Bytes one party sends per proof, from the protocol's shapes (32-byte header per exchange)."""
    m = nc * n
    deg = 5 * (n + 1) + 2
    payloads = [64 + 5 * 64]                                     # statement + wire commitments
    payloads += [32 * n * 2 * k for k in (4, 2, 2, 2)]          # round-2 levels (den r and num r at the last)
    payloads.append(32 * n)                                      # den r
    d = 1
    while d < n:
        payloads.append(32 * 2 * (n - d))
        d <<= 1
    payloads.append(64)                                          # z commitment
    payloads += [32 * m * k for k in (16, 10, 14, 4)]           # round-3 levels (squares open one difference)
    payloads.append(32 * (2 + m - deg - 1))                      # r' q[deg] differences + quotient tail
    payloads.append(32)                                          # r' q[deg]
    payloads += [5 * 64, 6 * 32, 2 * 64]                         # quotient commitments, evaluations, openings
    return len(payloads), sum(32 + p for p in payloads)


@pytest.mark.parametrize("log_n,parties", [(3, 2), (3, 3), (10, 2), (10, 3), (12, 2), (12, 3), (16, 2)])
def test_joint_proof_equals_single_prover(ctx, party_ctxs, srs_points, oracle, log_n, parties):
    from renegade_b200 import collaborative as co
    circ, bases, pk, bl, single, hint, ch = setup(ctx, srs_points, log_n)
    ws, bs = shares(circ, bl, parties)
    res = co.prove_jointly(party_ctxs[:parties], [pk] * parties, ws, circ.pub_inputs, bs, seed=1000 + log_n, timeout_ms=TIMEOUT_MS)
    assert codes(res) == [0] * parties, res
    for r in res:
        assert bytes(r.proof) == bytes(single)
        assert (r.challenges == ch).all()
    assert (sum_shares([r.link_poly_share for r in res]) == hint.linking_wire_poly).all()
    # accounting: triples used == the preprocessing size; bytes from the shapes
    t, _ = co.MpcPrep.size(pk)
    nc = 6 if log_n >= 4 else 8
    ex, nbytes = expected_bytes(1 << log_n, nc)
    for r in res:
        assert r.stats["triples"] == t
        assert r.stats["exchanges"] == ex and r.stats["bytes_sent"] == nbytes
    if log_n <= 12:
        opk = oracle.plonk_preprocess(log_n, circ.selectors, circ.perm, circ.k, np.ascontiguousarray(srs_points[:(1 << log_n) + 3]))
        rc, oproof, _, _ = oracle.plonk_prove(log_n, circ.num_inputs, circ.k, opk, circ.wires, circ.pub_inputs, bl,
                                              np.ascontiguousarray(srs_points[:(1 << log_n) + 3]))
        assert rc == 0 and bytes(oproof) == bytes(single)


def test_one_party_per_gpu(srs_points):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import renegade_b200 as rb
    from renegade_b200 import collaborative as co
    from renegade_b200.backend import PlonkKzgSnark
    log_n = 10
    cs = [rb.Context(d) for d in (0, 1)]
    try:
        circ, _, _, bl, single, _, _ = setup(cs[0], srs_points, log_n)
        pks = []
        for c in cs:  # parties on different devices each preprocess their own key
            b = c.load_bases(srs_points[:(1 << log_n) + 3])
            pks.append((b, PlonkKzgSnark.preprocess(c, b, log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)))
        ws, bs = shares(circ, bl, 2)
        res = co.prove_jointly(cs, [p for _, p in pks], ws, circ.pub_inputs, bs, timeout_ms=TIMEOUT_MS)
        assert codes(res) == [0, 0] and all(bytes(r.proof) == bytes(single) for r in res)
    finally:
        for c in cs:
            c.close()


def test_perturbed_shares_are_unsatisfied_everywhere(ctx, party_ctxs, srs_points):
    from renegade_b200 import collaborative as co
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R, limbs_to_scalars, scalars_to_limbs
    circ, _, pk, bl, _, _, _ = setup(ctx, srs_points, 10)
    ws, bs = shares(circ, bl, 2)
    bad = limbs_to_scalars(ws[1])
    for i in range(0, len(bad), 97):
        bad[i] = (bad[i] + 1) % R
    res = co.prove_jointly(party_ctxs[:2], [pk] * 2, [ws[0], scalars_to_limbs(bad)], circ.pub_inputs, bs, timeout_ms=TIMEOUT_MS)
    assert codes(res) == [-7, -7]


def test_disagreeing_statement_is_invalid_everywhere(ctx, party_ctxs, srs_points):
    from renegade_b200 import collaborative as co
    circ, _, pk, bl, _, _, _ = setup(ctx, srs_points, 10)
    ws, bs = shares(circ, bl, 2)
    group = co.LocalGroup(2, TIMEOUT_MS)
    preps = [co.MpcPrep.dealer(party_ctxs[p], pk, 5, p, 2) for p in range(2)]
    other = np.array(circ.pub_inputs, dtype=np.uint64).reshape(-1, 4).copy()
    other[0, 0] ^= 1
    pis = [circ.pub_inputs, other]
    res = co._run_parties([lambda p=p: co.prove_party(party_ctxs[p], pk, group.transport(p), preps[p], ws[p], pis[p], bs[p])
                           for p in range(2)])
    assert codes(res) == [-1, -1]
    for pr in preps:
        pr.free()
    group.close()


def test_preprocessing_is_single_use(ctx, party_ctxs, srs_points):
    from renegade_b200 import collaborative as co
    circ, _, pk, bl, single, _, _ = setup(ctx, srs_points, 3)
    ws, bs = shares(circ, bl, 2)
    preps = [co.MpcPrep.dealer(party_ctxs[p], pk, 9, p, 2) for p in range(2)]
    for attempt in range(2):
        group = co.LocalGroup(2, TIMEOUT_MS)
        res = co._run_parties([lambda p=p: co.prove_party(party_ctxs[p], pk, group.transport(p), preps[p], ws[p], circ.pub_inputs,
                                                          bs[p]) for p in range(2)])
        group.close()
        if attempt == 0:
            assert codes(res) == [0, 0] and bytes(res[0].proof) == bytes(single)
        else:
            assert codes(res) == [-1, -1]
    for pr in preps:
        pr.free()


def test_bad_arguments(ctx, party_ctxs, srs_points):
    import ctypes as C
    from renegade_b200 import _lib
    from renegade_b200 import collaborative as co
    lib = _lib.load()
    circ, _, pk, bl, _, _, _ = setup(ctx, srs_points, 3)
    h = C.c_void_p()
    assert lib.b200_mpc_local_group_create(1, 1000, C.byref(h)) == -1
    assert lib.b200_mpc_prep_dealer(ctx._h, pk._h, 1, 2, 2, C.byref(h)) == -1
    assert lib.b200_mpc_prep_dealer(ctx._h, pk._h, 1, 0, 1, C.byref(h)) == -1
    assert lib.b200_mpc_prove(ctx._h, pk._h, None, None, None, None, None, None, None, None) == -1
    group = co.LocalGroup(2, TIMEOUT_MS)
    t = group.transport(0)
    assert lib.b200_mpc_local_group_transport(group._h, 2, C.byref(co.MpcTransport())) == -1
    bad = co.MpcTransport(t.all_gather, t.abort, t.user, 2, 2)      # party out of range
    assert lib.b200_mpc_prove(ctx._h, pk._h, C.byref(bad), None, None, None, None, None, None, None) == -1
    bad = co.MpcTransport(t.all_gather, t.abort, t.user, 0, 1)      # parties < 2
    assert lib.b200_mpc_prove(ctx._h, pk._h, C.byref(bad), None, None, None, None, None, None, None) == -1
    group.close()
    # a preprocessing made for another key does not fit; the failing party's abort ends the other one too
    _, _, pk10, _, _, _, _ = setup(ctx, srs_points, 10)
    ws, bs = shares(circ, bl, 2)
    group = co.LocalGroup(2, TIMEOUT_MS)
    preps = [co.MpcPrep.dealer(party_ctxs[0], pk10, 3, 0, 2), co.MpcPrep.dealer(party_ctxs[1], pk, 3, 1, 2)]
    res = co._run_parties([lambda p=p: co.prove_party(party_ctxs[p], pk, group.transport(p), preps[p], ws[p], circ.pub_inputs, bs[p])
                           for p in range(2)])
    assert codes(res) == [-1, -1]
    for pr in preps:
        pr.free()
    group.close()


class Hub:
    """An all-gather between Python threads; `tamper(party, exchange, all_bytes) -> bytes` may alter what a party receives."""

    def __init__(self, parties, tamper=None, fail_at=None):
        self.P, self.tamper, self.fail_at = parties, tamper, fail_at
        self.barrier = threading.Barrier(parties, timeout=TIMEOUT_MS / 1000)
        self.slots = [None] * parties
        self.count = [0] * parties

    def transport(self, party):
        from renegade_b200 import collaborative as co

        def gather(mine):
            k = self.count[party]
            self.count[party] += 1
            if self.fail_at == (party, k):
                self.barrier.abort()
                return None
            self.slots[party] = mine
            self.barrier.wait()
            out = b"".join(self.slots)
            self.barrier.wait()
            return self.tamper(party, k, out) if self.tamper else out

        return co.callback_transport(party, self.P, gather, abort=self.barrier.abort)


def test_python_transport(ctx, party_ctxs, srs_points, ptau_g2):
    from renegade_b200 import collaborative as co
    from renegade_b200.backend import PlonkKzgSnark, VerifyingKey
    log_n = 10
    circ, _, pk, bl, single, _, _ = setup(ctx, srs_points, log_n)
    ws, bs = shares(circ, bl, 2)
    n, m = 1 << log_n, 6 << log_n
    run = lambda hub, seed: co.prove_jointly(party_ctxs[:2], [pk] * 2, ws, circ.pub_inputs, bs, seed=seed,
                                             transports=[hub.transport(p) for p in range(2)])
    res = run(Hub(2), 11)
    assert codes(res) == [0, 0] and all(bytes(r.proof) == bytes(single) for r in res)
    # exchange index of round 3's first Beaver level: statement, 4 levels + den r, log2 n prefix levels, z
    r3 = 1 + 5 + log_n + 1

    def flip(target_party, exchange, offset):
        def tamper(party, k, data):
            if party != target_party or k != exchange:
                return data
            b = bytearray(data)
            b[offset] ^= 1
            return bytes(b)
        return tamper

    msg = 32 + 32 * 16 * m  # one party's message of round 3's first level: header, 16 m differences
    res = run(Hub(2, flip(1, r3, msg + 32 + 5 * 32 + 3)), 12)   # party 1 receives a corrupted difference of its own slot
    assert codes(res) == [-7, -7]
    # a flipped byte in a round-5 partial commitment: that party's proof does not verify
    # (round-3 levels, degree check, r' q[deg], quotient commitments, evaluations: the openings are exchange r3 + 8)
    res = run(Hub(2, flip(0, r3 + 8, 32 + 64 + 7)), 13)
    assert codes(res) == [0, 0]
    h, tau_h = ptau_g2
    vk = VerifyingKey.from_proving_key(pk, h, tau_h)
    assert PlonkKzgSnark.verify(vk, circ.pub_inputs, res[1].proof)
    assert not PlonkKzgSnark.verify(vk, circ.pub_inputs, res[0].proof)
    # a wrong header (exchange index) is refused; a transport error ends every party
    res = run(Hub(2, flip(0, 3, 0)), 14)
    assert codes(res)[0] == -1 and codes(res)[1] != 0
    res = run(Hub(2, fail_at=(1, 5)), 15)
    assert all(c != 0 for c in codes(res))
    assert n  # domain size used above


def test_link_jointly(ctx, party_ctxs, srs_points):
    from renegade_b200 import collaborative as co
    from renegade_b200.backend import GroupLayout, LinkingHint, link_proofs
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R, limbs_to_scalars, scalars_to_limbs
    import random
    rnd = random.Random(4)
    # two hints that agree on the group g^(offset + i), g of order 2^alignment: a1 = a2 + Z_D u
    layout = GroupLayout(alignment=10, offset=3, size=40)
    from renegade_b200.collaborative import domain_generator
    g = domain_generator(layout.alignment)
    zd = [1]
    for i in range(layout.size):  # zd <- zd * (X - root)
        root = pow(g, layout.offset + i, R)
        zd = [((zd[j - 1] if j > 0 else 0) - root * (zd[j] if j < len(zd) else 0)) % R for j in range(len(zd) + 1)]
    len1, len2 = 1026, 514
    a2 = [rnd.randrange(R) for _ in range(len2)]
    u = [rnd.randrange(R) for _ in range(len1 - layout.size)]
    a1 = a2 + [0] * (len1 - len2)
    for i, zi in enumerate(zd):
        for j, uj in enumerate(u):
            a1[i + j] = (a1[i + j] + zi * uj) % R
    A1, A2 = scalars_to_limbs(a1), scalars_to_limbs(a2)
    bases = ctx.load_bases(srs_points[:len1 + 8])
    from renegade_b200.backend import UnivariateKzgPCS
    c1, c2 = (UnivariateKzgPCS.commit(ctx, bases, A)[0] for A in (A1, A2))
    single, eta = link_proofs(ctx, bases, LinkingHint(A1, c1), LinkingHint(A2, c2), layout)
    s1 = co.share_table(A1, 2, seed=1)
    s2 = co.share_table(A2, 2, seed=2)
    res = co.link_jointly(party_ctxs[:2], [bases] * 2, s1, s2, c1, c2, layout)
    assert codes(res) == [0, 0]
    for proof, e in res:
        assert bytes(proof) == bytes(single) and (e == eta).all()
    # one shared hint and one plaintext hint held by party 1
    res = co.link_jointly(party_ctxs[:2], [bases] * 2, s1, [np.zeros_like(A2), A2], c1, c2, layout)
    assert codes(res) == [0, 0] and all(bytes(p) == bytes(single) for p, _ in res)
    # hints that disagree on the group: refused everywhere
    bad = limbs_to_scalars(A2)
    bad[5] = (bad[5] + 1) % R
    res = co.link_jointly(party_ctxs[:2], [bases] * 2, s1, [np.zeros_like(A2), scalars_to_limbs(bad)], c1, c2, layout)
    assert codes(res) == [-7, -7]
