"""The collaborative prover on authenticated shares (`b200_mpc_prove_auth`, `b200_mpc_link_auth`): the opened proof equals
`b200_plonk_prove` on the summed witness and blinders; any deviation of one party (an error in its own message, a wrong
MAC-key share or MAC, malformed data) gives B200_ERR_MAC on every party and leaves the outputs untouched; an unsatisfied
witness with consistent MACs gives B200_ERR_UNSATISFIED; the accounting is the plain call's plus three exchanges."""
import ctypes as C
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TIMEOUT_MS = 60000
ERR_MAC, ERR_UNSAT, ERR_INVALID = -8, -7, -1
HDR = 32


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
    """(circuit, bases, pk, blinders, single proof, single link hint, challenges) for a synthetic circuit of 2^log_n gates."""
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


def ints(a):
    from renegade_b200.fields import limbs_to_scalars
    return limbs_to_scalars(np.asarray(a, dtype=np.uint64).reshape(-1, 4))


def limbs(xs):
    from renegade_b200.fields import scalars_to_limbs
    return scalars_to_limbs(xs)


def sum_ints(parts):
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R
    return [sum(col) % R for col in zip(*[ints(p) for p in parts])]


def codes(results):
    from renegade_b200._lib import B200Error
    return [r.code if isinstance(r, B200Error) else (0 if not isinstance(r, Exception) else "exc") for r in results]


def plain_bytes(n, nc):
    """Exchanges and bytes one party sends in a plain proof (as tests/test_gpu_mpc.py's expected_bytes)."""
    m = nc * n
    deg = 5 * (n + 1) + 2
    payloads = [64 + 5 * 64] + [32 * n * 2 * k for k in (4, 2, 2, 2)] + [32 * n]
    d = 1
    while d < n:
        payloads.append(32 * 2 * (n - d))
        d <<= 1
    payloads += [64] + [32 * m * k for k in (16, 10, 14, 4)] + [32 * (2 + m - deg - 1), 32, 5 * 64, 6 * 32, 2 * 64]
    return len(payloads), sum(HDR + p for p in payloads)


# the authenticated call's extra payloads: H(seed) in exchange 0, seed reveal, check commitment, check reveal
AUTH_EXTRA_EXCHANGES = 3
AUTH_EXTRA_BYTES = 32 + (HDR + 32) + (HDR + 32) + (HDR + 160)


def dealer_keys(ctxs, pk, seed, P):
    """Every party's MAC-key share from the authenticated dealer of `seed`."""
    from renegade_b200 import collaborative as co
    keys = []
    for p in range(P):
        prep, k = co.MpcPrep.dealer_auth(ctxs[p], pk, seed, p, P)
        prep.free()
        keys.append(k)
    return keys


def auth_inputs(ctxs, circ, bl, seed, P, wires=None):
    """Per party (wire_share, wire_mac, blinder_share, blinder_mac) from the device input dealer of `seed`."""
    from renegade_b200 import collaborative as co
    w = np.asarray(circ.wires if wires is None else wires, dtype=np.uint64).reshape(-1, 4)
    table = np.concatenate([w, np.asarray(bl, dtype=np.uint64).reshape(-1, 4)])
    k = w.shape[0]
    out = []
    for p in range(P):
        sh, mac = co.dealer_share_auth(ctxs[p], seed, p, P, table)
        out.append((sh[:k], mac[:k], sh[k:], mac[k:]))
    return out


def run_auth(ctxs, pk, circ, bl, P, seed, transports=None, inputs=None, keys=None, proofs=None):
    """One authenticated proof, one thread per party, dealer preprocessing and inputs from `seed`."""
    from renegade_b200 import collaborative as co
    group = co.LocalGroup(P, TIMEOUT_MS) if transports is None else None
    trs = transports if transports is not None else [group.transport(p) for p in range(P)]
    made = [co.MpcPrep.dealer_auth(ctxs[p], pk, seed, p, P) for p in range(P)]
    keys = keys if keys is not None else [k for _, k in made]
    inputs = inputs if inputs is not None else auth_inputs(ctxs, circ, bl, seed, P)
    proofs = proofs if proofs is not None else [None] * P
    try:
        return co._run_parties([lambda p=p: co.prove_party_auth(ctxs[p], pk, trs[p], made[p][0], keys[p], inputs[p][0], inputs[p][1],
                                                                circ.pub_inputs, inputs[p][2], inputs[p][3], proofs[p])
                                for p in range(P)])
    finally:
        for prep, _ in made:
            prep.free()
        if group is not None:
            group.close()


class Hub:
    """An all-gather between Python threads; `tamper(receiver, exchange, all_bytes, msg_len) -> bytes` may alter what a
    party receives."""

    def __init__(self, parties, tamper=None):
        self.P, self.tamper = parties, tamper
        self.barrier = threading.Barrier(parties, timeout=TIMEOUT_MS / 1000)
        self.slots = [None] * parties
        self.count = [0] * parties

    def transport(self, party):
        from renegade_b200 import collaborative as co

        def gather(mine):
            k = self.count[party]
            self.count[party] += 1
            self.slots[party] = mine
            self.barrier.wait()
            out = b"".join(self.slots)
            self.barrier.wait()
            return self.tamper(party, k, out, len(mine)) if self.tamper else out

        return co.callback_transport(party, self.P, gather, abort=self.barrier.abort)


def add_one(buf, at):
    """+1 on the Montgomery field element at byte offset `at` (a non-zero additive error)."""
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R
    v = int.from_bytes(bytes(buf[at:at + 32]), "little")
    buf[at:at + 32] = ((v + 1) % R).to_bytes(32, "little")


def add_g(buf, at):
    """+G on the affine G1 point (Montgomery Fq, x || y) at byte offset `at`: the result stays on the curve."""
    from renegade_b200.fields import BASE_FIELD_MODULUS as Q
    rinv = pow(1 << 256, -1, Q)
    x1 = int.from_bytes(bytes(buf[at:at + 32]), "little") * rinv % Q
    y1 = int.from_bytes(bytes(buf[at + 32:at + 64]), "little") * rinv % Q
    x2, y2 = 1, 2
    if x1 == 0 and y1 == 0:
        x3, y3 = x2, y2
    else:
        lam = (y2 - y1) * pow(x2 - x1, -1, Q) % Q
        x3 = (lam * lam - x1 - x2) % Q
        y3 = (lam * (x1 - x3) - y1) % Q
    buf[at:at + 32] = ((x3 << 256) % Q).to_bytes(32, "little")
    buf[at + 32:at + 64] = ((y3 << 256) % Q).to_bytes(32, "little")


def sender_error(sender, exchange, payload_off, op, receivers=None):
    """The sender alters its own message of `exchange` at payload offset `payload_off`, for `receivers` (all by default)."""
    def tamper(party, k, data, msg):
        if k != exchange or (receivers is not None and party not in receivers):
            return data
        b = bytearray(data)
        op(b, sender * msg + HDR + payload_off)
        return bytes(b)
    return tamper


def test_dealer_share_auth(ctx, party_ctxs, srs_points):
    """The device input dealer: shares sum to the values and MAC shares to alpha times them, alpha being the sum of the
    authenticated preprocessing dealer's key shares for the same seed."""
    from renegade_b200 import collaborative as co
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R
    _, _, pk, _, _, _, _ = setup(ctx, srs_points, 3)
    vals = limbs([3, 5, R - 1, 0, 12345678901234567890])
    P = 3
    parts = [co.dealer_share_auth(party_ctxs[p], 77, p, P, vals) for p in range(P)]
    alpha = sum(ints(k)[0] for k in dealer_keys(party_ctxs, pk, 77, P)) % R
    assert sum_ints([p[0] for p in parts]) == ints(vals)
    assert sum_ints([p[1] for p in parts]) == [alpha * v % R for v in ints(vals)]


@pytest.mark.parametrize("log_n,parties", [(3, 2), (3, 3), (10, 2), (10, 3), (12, 2), (12, 3), (16, 2)])
def test_auth_joint_proof_equals_single_prover(ctx, party_ctxs, srs_points, oracle, log_n, parties):
    from renegade_b200 import collaborative as co
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R
    circ, _, pk, bl, single, hint, ch = setup(ctx, srs_points, log_n)
    seed = 2000 + log_n
    res = co.prove_jointly_auth(party_ctxs[:parties], [pk] * parties, circ.wires, circ.pub_inputs, bl, seed=seed, timeout_ms=TIMEOUT_MS)
    assert codes(res) == [0] * parties, res
    for r in res:
        assert bytes(r.proof) == bytes(single)
        assert (r.challenges == ch).all()
    alpha = sum(ints(k)[0] for k in dealer_keys(party_ctxs, pk, seed, parties)) % R
    link = ints(hint.linking_wire_poly)
    assert sum_ints([r.link_poly_share for r in res]) == link
    assert sum_ints([r.link_poly_mac for r in res]) == [alpha * v % R for v in link]
    t, _ = co.MpcPrep.size(pk)
    nc = 6 if log_n >= 4 else 8
    ex, nbytes = plain_bytes(1 << log_n, nc)
    for r in res:
        assert r.stats["triples"] == t
        assert r.stats["exchanges"] == ex + AUTH_EXTRA_EXCHANGES
        assert r.stats["bytes_sent"] == nbytes + AUTH_EXTRA_BYTES
    if log_n <= 12:
        pts = np.ascontiguousarray(srs_points[:(1 << log_n) + 3])
        opk = oracle.plonk_preprocess(log_n, circ.selectors, circ.perm, circ.k, pts)
        rc, oproof, _, _ = oracle.plonk_prove(log_n, circ.num_inputs, circ.k, opk, circ.wires, circ.pub_inputs, bl, pts)
        assert rc == 0 and bytes(oproof) == bytes(single)


LOG_N = 10
N = 1 << LOG_N
M = 6 * N
R3 = 1 + 5 + LOG_N + 1        # first round-3 level: statement, 4 levels + den r, log2 n prefix levels, z
EX_Z = R3 - 1                  # z commitment
EX_TAIL, EX_RQ, EX_QUOT, EX_EVALS, EX_OPEN = R3 + 4, R3 + 5, R3 + 6, R3 + 7, R3 + 8
EX_SEED, EX_COMMIT, EX_REVEAL = R3 + 9, R3 + 10, R3 + 11

TAMPERS = {
    "round2_level1": (1, 0, add_one),
    "prefix_level": (6, 32 * 5, add_one),
    "den_r": (5, 32 * 3, add_one),
    "round3_level4": (R3 + 3, 32 * 7, add_one),
    "quotient_tail": (EX_TAIL, 32 * (2 + 5), add_one),
    "rq_deg": (EX_RQ, 0, add_one),
    "evaluation": (EX_EVALS, 32 * 2, add_one),
    "commit_round1": (0, 96 + 64, add_g),
    "commit_round2": (EX_Z, 0, add_g),
    "commit_round3": (EX_QUOT, 64 * 2, add_g),
    "commit_round5": (EX_OPEN, 0, add_g),
    "seed_reveal": (EX_SEED, 0, add_one),
    "sigma_reveal": (EX_REVEAL, 0, add_one),
}


@pytest.mark.parametrize("case", sorted(TAMPERS))
def test_auth_sender_error_is_caught_everywhere(ctx, party_ctxs, srs_points, case):
    circ, _, pk, bl, _, _, _ = setup(ctx, srs_points, LOG_N)
    ex, off, op = TAMPERS[case]
    hub = Hub(2, sender_error(1, ex, off, op))
    res = run_auth(party_ctxs[:2], pk, circ, bl, 2, 31, transports=[hub.transport(p) for p in range(2)])
    assert codes(res) == [ERR_MAC, ERR_MAC], case


@pytest.mark.parametrize("case", ["round2_level1", "evaluation", "commit_round5"])
def test_auth_inconsistent_views(ctx, party_ctxs, srs_points, case):
    circ, _, pk, bl, _, _, _ = setup(ctx, srs_points, LOG_N)
    ex, off, op = TAMPERS[case]
    hub = Hub(2, sender_error(0, ex, off, op, receivers={1}))
    res = run_auth(party_ctxs[:2], pk, circ, bl, 2, 32, transports=[hub.transport(p) for p in range(2)])
    c = codes(res)
    assert 0 not in c and c[1] == ERR_MAC, c


def test_auth_contrast_with_plain_mode(ctx, party_ctxs, srs_points):
    """The plain-mode tamper that yields [0, 0] and a bad proof: a flipped byte in a round-5 partial commitment."""
    from renegade_b200.backend import B200Proof

    def flip(party, k, data, msg):
        if party != 0 or k != EX_OPEN:
            return data
        b = bytearray(data)
        b[HDR + 64 + 7] ^= 1
        return bytes(b)

    circ, _, pk, bl, _, _, _ = setup(ctx, srs_points, LOG_N)
    proofs = [B200Proof() for _ in range(2)]
    for pr in proofs:
        C.memset(C.byref(pr), 0xA5, C.sizeof(pr))
    sentinel = bytes(proofs[0])
    hub = Hub(2, flip)
    res = run_auth(party_ctxs[:2], pk, circ, bl, 2, 33, transports=[hub.transport(p) for p in range(2)], proofs=proofs)
    assert codes(res) == [ERR_MAC, ERR_MAC]
    assert all(bytes(pr) == sentinel for pr in proofs)


def test_auth_malformed_data(ctx, party_ctxs, srs_points):
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R
    circ, _, pk, bl, _, _, _ = setup(ctx, srs_points, LOG_N)

    def off_curve(b, at):
        b[at] ^= 1

    def not_canonical(b, at):
        b[at:at + 32] = R.to_bytes(32, "little")

    for ex, off, op in [(0, 96 + 64 * 2, off_curve), (1, 32 * 9, not_canonical), (EX_EVALS, 0, not_canonical)]:
        hub = Hub(2, sender_error(1, ex, off, op))
        res = run_auth(party_ctxs[:2], pk, circ, bl, 2, 34, transports=[hub.transport(p) for p in range(2)])
        assert codes(res) == [ERR_MAC, ERR_MAC], (ex, off)


def test_auth_wrong_keys_and_macs(ctx, party_ctxs, srs_points):
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R
    circ, _, pk, bl, _, _, _ = setup(ctx, srs_points, LOG_N)
    seed = 35
    keys = dealer_keys(party_ctxs, pk, seed, 2)
    bad_keys = [keys[0], limbs([(ints(keys[1])[0] + 1) % R])[0]]
    assert codes(run_auth(party_ctxs[:2], pk, circ, bl, 2, seed, keys=bad_keys)) == [ERR_MAC, ERR_MAC]
    for which in (1, 3):  # a wrong MAC on one wire share, then on one blinder share
        inp = auth_inputs(party_ctxs, circ, bl, seed, 2)
        macs = ints(inp[1][which])
        macs[4] = (macs[4] + 1) % R
        inp[1] = tuple(limbs(macs) if i == which else x for i, x in enumerate(inp[1]))
        assert codes(run_auth(party_ctxs[:2], pk, circ, bl, 2, seed, inputs=inp)) == [ERR_MAC, ERR_MAC], which


def test_auth_unsatisfied_witness_with_consistent_macs(ctx, party_ctxs, srs_points):
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R
    circ, _, pk, bl, _, _, _ = setup(ctx, srs_points, LOG_N)
    w = ints(circ.wires)
    for i in range(0, len(w), 97):
        w[i] = (w[i] + 1) % R
    inp = auth_inputs(party_ctxs, circ, bl, 36, 2, wires=limbs(w))
    assert codes(run_auth(party_ctxs[:2], pk, circ, bl, 2, 36, inputs=inp)) == [ERR_UNSAT, ERR_UNSAT]


def test_auth_preprocessing_and_arguments(ctx, party_ctxs, srs_points):
    from renegade_b200 import _lib
    from renegade_b200 import collaborative as co
    lib = _lib.load()
    circ, _, pk, bl, single, _, _ = setup(ctx, srs_points, 3)
    seed = 37
    inp = auth_inputs(party_ctxs, circ, bl, seed, 2)
    made = [co.MpcPrep.dealer_auth(party_ctxs[p], pk, seed, p, 2) for p in range(2)]

    def once(preps, fn):
        group = co.LocalGroup(2, TIMEOUT_MS)
        try:
            return co._run_parties([lambda p=p: fn(p, group.transport(p), preps[p]) for p in range(2)])
        finally:
            group.close()

    auth = lambda p, t, prep: co.prove_party_auth(party_ctxs[p], pk, t, prep, made[p][1], inp[p][0], inp[p][1], circ.pub_inputs,
                                                  inp[p][2], inp[p][3])
    res = once([m[0] for m in made], auth)
    assert codes(res) == [0, 0] and bytes(res[0].proof) == bytes(single)
    assert codes(once([m[0] for m in made], auth)) == [ERR_INVALID, ERR_INVALID]  # single use
    for m in made:
        m[0].free()
    # a plain prep to the authenticated call, an authenticated prep to the plain call
    plain = [co.MpcPrep.dealer(party_ctxs[p], pk, seed, p, 2) for p in range(2)]
    assert codes(once(plain, auth)) == [ERR_INVALID, ERR_INVALID]
    made = [co.MpcPrep.dealer_auth(party_ctxs[p], pk, seed, p, 2) for p in range(2)]
    res = once([m[0] for m in made], lambda p, t, prep: co.prove_party(party_ctxs[p], pk, t, prep, inp[p][0], circ.pub_inputs, inp[p][2]))
    assert codes(res) == [ERR_INVALID, ERR_INVALID]
    # NULL MAC pointers
    group = co.LocalGroup(2, TIMEOUT_MS)
    t = group.transport(0)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    w, bsh = np.ascontiguousarray(inp[0][0]), np.ascontiguousarray(inp[0][2])
    key = np.ascontiguousarray(made[0][1])
    pi = np.ascontiguousarray(np.asarray(circ.pub_inputs, dtype=np.uint64).reshape(-1, 4))
    from renegade_b200.backend import B200Proof
    pr = B200Proof()
    assert lib.b200_mpc_prove_auth(ctx._h, pk._h, C.byref(t), made[0][0]._h, vp(key), vp(w), None, vp(pi), vp(bsh), vp(bsh),
                                   C.byref(pr), None, None, None) == ERR_INVALID
    assert lib.b200_mpc_prove_auth(ctx._h, pk._h, C.byref(t), made[0][0]._h, None, vp(w), vp(w), vp(pi), vp(bsh), vp(bsh),
                                   C.byref(pr), None, None, None) == ERR_INVALID
    group.close()
    for pp in plain:
        pp.free()
    for m in made:
        m[0].free()


def _link_setup(ctx, srs_points):
    from renegade_b200.backend import GroupLayout, LinkingHint, UnivariateKzgPCS, link_proofs
    from renegade_b200.collaborative import domain_generator
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R
    import random
    rnd = random.Random(4)
    layout = GroupLayout(alignment=10, offset=3, size=40)
    g = domain_generator(layout.alignment)
    zd = [1]
    for i in range(layout.size):
        root = pow(g, layout.offset + i, R)
        zd = [((zd[j - 1] if j > 0 else 0) - root * (zd[j] if j < len(zd) else 0)) % R for j in range(len(zd) + 1)]
    len1, len2 = 1026, 514
    a2 = [rnd.randrange(R) for _ in range(len2)]
    u = [rnd.randrange(R) for _ in range(len1 - layout.size)]
    a1 = a2 + [0] * (len1 - len2)
    for i, zi in enumerate(zd):
        for j, uj in enumerate(u):
            a1[i + j] = (a1[i + j] + zi * uj) % R
    A1, A2 = limbs(a1), limbs(a2)
    bases = ctx.load_bases(srs_points[:len1 + 8])
    c1, c2 = (UnivariateKzgPCS.commit(ctx, bases, A)[0] for A in (A1, A2))
    single, eta = link_proofs(ctx, bases, LinkingHint(A1, c1), LinkingHint(A2, c2), layout)
    return layout, A1, A2, a2, bases, c1, c2, single, eta


def test_auth_link(ctx, party_ctxs, srs_points):
    from renegade_b200 import collaborative as co
    from renegade_b200.fields import SCALAR_FIELD_MODULUS as R
    layout, A1, A2, a2, bases, c1, c2, single, eta = _link_setup(ctx, srs_points)
    keys = [limbs([1234567])[0], limbs([R - 89])[0]]
    s1 = co.auth_share_table(A1, 2, keys, seed=1)
    s2 = co.auth_share_table(A2, 2, keys, seed=2)
    pair = lambda s: [(s[0][p], s[1][p]) for p in range(2)]
    run = lambda h1, h2, hub=None: co.link_jointly_auth(party_ctxs[:2], [bases] * 2, keys, h1, h2, c1, c2, layout, TIMEOUT_MS,
                                                        transports=None if hub is None else [hub.transport(p) for p in range(2)])
    res = run(pair(s1), pair(s2))
    assert codes(res) == [0, 0]
    for proof, e in res:
        assert bytes(proof) == bytes(single) and (e == eta).all()
    # the second hint input by party 1 alone (an input protocol gives the other party a zero share with a MAC share)
    alpha = sum(ints(k)[0] for k in keys) % R
    held = [(np.zeros_like(A2), np.zeros_like(A2)), (A2, limbs([alpha * v % R for v in a2]))]
    res = run(pair(s1), held)
    assert codes(res) == [0, 0] and all(bytes(p) == bytes(single) for p, _ in res)
    # hints that disagree on the group
    bad = list(a2)
    bad[5] = (bad[5] + 1) % R
    res = run(pair(s1), pair(co.auth_share_table(limbs(bad), 2, keys, seed=3)))
    assert codes(res) == [ERR_UNSAT, ERR_UNSAT]
    # tampering: the tail, the evaluation at eta, a partial commitment
    for ex, off, op in [(0, 64 + 32 + 32 * 3, add_one), (1, 64, add_one), (1, 0, add_g), (0, 0, add_g)]:
        res = run(pair(s1), pair(s2), Hub(2, sender_error(1, ex, off, op)))
        assert codes(res) == [ERR_MAC, ERR_MAC], (ex, off)


def test_auth_one_party_per_gpu(srs_points):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import renegade_b200 as rb
    from renegade_b200 import collaborative as co
    from renegade_b200.backend import PlonkKzgSnark
    cs = [rb.Context(d) for d in (0, 1)]
    try:
        circ, _, _, bl, single, _, _ = setup(cs[0], srs_points, LOG_N)
        pks = []
        for c in cs:
            b = c.load_bases(srs_points[:N + 3])
            pks.append((b, PlonkKzgSnark.preprocess(c, b, LOG_N, circ.num_inputs, circ.selectors, circ.perm, circ.k)))
        res = co.prove_jointly_auth(cs, [p for _, p in pks], circ.wires, circ.pub_inputs, bl, timeout_ms=TIMEOUT_MS)
        assert codes(res) == [0, 0] and all(bytes(r.proof) == bytes(single) for r in res)
    finally:
        for c in cs:
            c.close()
