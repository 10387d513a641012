"""TEST INFRASTRUCTURE — pure-Python optimal-ate pairing on BN254 (alt_bn128), used only by tests/
to check KZG equations the way the reference's verifier does (`PlonkKzgSnark::verify`,
crates/circuits/circuit-types/src/traits.rs:1003-1019) and to restate the reference's own SRS unit
test (crates/circuits/circuit-types/src/primitives/srs.rs:236-266: e(tau^i G, tau H) = e(tau^(i+1) G, H)).

The arithmetic lives in ark-bn254 / ark-ec (un-vendored); this restates the standard construction:
Fq12 = Fq[w] / (w^12 - 18 w^6 + 82), G2 on the sextic twist y^2 = x^3 + 3/(9+u) mapped into
E(Fq12) by (x, y) -> (x w^2, y w^3), Miller loop over 6x+2 with x = 4965661367192848881, two
Frobenius line steps, final exponentiation (q^12 - 1)/r.  Slow (seconds per pairing) by design:
clarity over speed.  Pinned by bilinearity and by the reference's SRS file itself.
"""
from __future__ import annotations

Q = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B97091_43E1F593F0000001
ATE_LOOP_COUNT = 29793968203157093288  # 6x + 2
LOG_ATE_LOOP_COUNT = 63
# w^12 = 18 w^6 - 82
_MOD_HI, _MOD_LO = 18, -82


class Fq12:
    __slots__ = ("c",)

    def __init__(self, coeffs):
        self.c = [v % Q for v in coeffs]

    @staticmethod
    def one():
        return Fq12([1] + [0] * 11)

    @staticmethod
    def zero():
        return Fq12([0] * 12)

    @staticmethod
    def from_fq(v):
        return Fq12([v] + [0] * 11)

    def __add__(self, o):
        return Fq12([a + b for a, b in zip(self.c, o.c)])

    def __sub__(self, o):
        return Fq12([a - b for a, b in zip(self.c, o.c)])

    def __neg__(self):
        return Fq12([-a for a in self.c])

    def __eq__(self, o):
        return self.c == o.c

    def is_zero(self):
        return not any(self.c)

    def scale(self, k):
        return Fq12([a * k for a in self.c])

    def __mul__(self, o):
        a, b = self.c, o.c
        t = [0] * 23
        for i, ai in enumerate(a):
            if ai:
                for j, bj in enumerate(b):
                    t[i + j] += ai * bj
        for k in range(22, 11, -1):  # w^k = 18 w^(k-6) - 82 w^(k-12)
            v = t[k]
            if v:
                t[k - 6] += _MOD_HI * v
                t[k - 12] += _MOD_LO * v
        return Fq12(t[:12])

    def __pow__(self, e):
        result, base = Fq12.one(), self
        while e:
            if e & 1:
                result = result * base
            base = base * base
            e >>= 1
        return result

    def inv(self):
        """Extended Euclid on polynomials over Fq against the modulus w^12 - 18 w^6 + 82."""
        def deg(p):
            d = len(p) - 1
            while d and p[d] == 0:
                d -= 1
            return d

        lm, hm = [1] + [0] * 12, [0] * 13
        low = self.c + [0]
        high = [82, 0, 0, 0, 0, 0, Q - 18, 0, 0, 0, 0, 0, 1]
        while deg(low):
            # r = high / low (polynomial quotient)
            dl, dh = deg(low), deg(high)
            r = [0] * 13
            temp = list(high)
            inv_lead = pow(low[dl], -1, Q)
            for i in range(dh - dl, -1, -1):
                r[i] = temp[dl + i] * inv_lead % Q
                for k in range(dl + 1):
                    temp[k + i] = (temp[k + i] - r[i] * low[k]) % Q
            nm, new = list(hm), list(high)
            for i in range(13):
                for j in range(13 - i):
                    nm[i + j] = (nm[i + j] - lm[i] * r[j]) % Q
                    new[i + j] = (new[i + j] - low[i] * r[j]) % Q
            lm, low, hm, high = nm, new, lm, low
        inv0 = pow(low[0], -1, Q)
        return Fq12([v * inv0 for v in lm[:12]])

    def __truediv__(self, o):
        return self * o.inv()


W = Fq12([0, 1] + [0] * 10)
W2, W3 = W * W, W * W * W


def twist(g2_point):
    """((x0, x1), (y0, y1)) on the twist -> point of E(Fq12)."""
    (x0, x1), (y0, y1) = g2_point
    # Fq2 = Fq[u]/(u^2+1) -> Fq[w^6]: u = w^6 - 9
    nx = Fq12([x0 - 9 * x1] + [0] * 5 + [x1] + [0] * 5)
    ny = Fq12([y0 - 9 * y1] + [0] * 5 + [y1] + [0] * 5)
    return (nx * W2, ny * W3)


def cast_g1(p):
    return (Fq12.from_fq(p[0]), Fq12.from_fq(p[1]))


def _double(p):
    x, y = p
    m = (x * x).scale(3) / y.scale(2)
    nx = m * m - x.scale(2)
    return (nx, m * (x - nx) - y)


def _add(p1, p2):
    if p1 is None:
        return p2
    if p2 is None:
        return p1
    x1, y1 = p1
    x2, y2 = p2
    if x1 == x2:
        return _double(p1) if y1 == y2 else None
    m = (y2 - y1) / (x2 - x1)
    nx = m * m - x1 - x2
    return (nx, m * (x1 - nx) - y1)


def _linefunc(p1, p2, t):
    x1, y1 = p1
    x2, y2 = p2
    xt, yt = t
    if not (x1 == x2):
        m = (y2 - y1) / (x2 - x1)
        return m * (xt - x1) - (yt - y1)
    if y1 == y2:
        m = (x1 * x1).scale(3) / y1.scale(2)
        return m * (xt - x1) - (yt - y1)
    return xt - x1


def miller_loop(g2_point, g1_point) -> Fq12:
    """Miller function value before the final exponentiation (so several can be multiplied)."""
    q, p = twist(g2_point), cast_g1(g1_point)
    r, f = q, Fq12.one()
    for i in range(LOG_ATE_LOOP_COUNT, -1, -1):
        f = f * f * _linefunc(r, r, p)
        r = _double(r)
        if ATE_LOOP_COUNT & (1 << i):
            f = f * _linefunc(r, q, p)
            r = _add(r, q)
    q1 = (q[0] ** Q, q[1] ** Q)
    nq2 = (q1[0] ** Q, -(q1[1] ** Q))
    f = f * _linefunc(r, q1, p)
    r = _add(r, q1)
    f = f * _linefunc(r, nq2, p)
    return f


def final_exponentiation(f: Fq12) -> Fq12:
    return f ** ((Q ** 12 - 1) // R)


def pairing(g2_point, g1_point) -> Fq12:
    return final_exponentiation(miller_loop(g2_point, g1_point))


def pairing_product_is_one(pairs) -> bool:
    """prod e(P_i, Q_i) == 1 for [(g1_point, g2_point), ...] with one shared final exponentiation;
    a G1 point given as None (identity) contributes 1."""
    f = Fq12.one()
    for g1_point, g2_point in pairs:
        if g1_point is None:
            continue
        f = f * miller_loop(g2_point, g1_point)
    return final_exponentiation(f) == Fq12.one()


def decode_g2_mont(raw: bytes, i: int):
    """One 128-byte ptau G2 record (x0, x1, y0, y1; 32-byte LE Montgomery each; srs.rs:185-199)."""
    ri = pow(1 << 256, -1, Q)
    v = [int.from_bytes(raw[128 * i + 32 * k: 128 * i + 32 * k + 32], "little") * ri % Q for k in range(4)]
    return ((v[0], v[1]), (v[2], v[3]))


def encode_g2_mont(pt) -> bytes:
    """Inverse of decode_g2_mont: one 128-byte ptau G2 record."""
    (x0, x1), (y0, y1) = pt
    return b"".join((v * (1 << 256) % Q).to_bytes(32, "little") for v in (x0, x1, y0, y1))


def g2_mul(pt, k: int):
    """k * pt for an affine point of the twist (k > 0, k * pt not the identity), affine double-and-add over
    Fq2 = Fq[u]/(u^2+1): builds [tau]_2 for an SRS whose tau is known."""
    def mul(a, b):
        return ((a[0] * b[0] - a[1] * b[1]) % Q, (a[0] * b[1] + a[1] * b[0]) % Q)

    def sub(a, b):
        return ((a[0] - b[0]) % Q, (a[1] - b[1]) % Q)

    def inv(a):
        d = pow((a[0] * a[0] + a[1] * a[1]) % Q, -1, Q)
        return (a[0] * d % Q, -a[1] * d % Q)

    def add(p1, p2):
        (x1, y1), (x2, y2) = p1, p2
        if x1 == x2:
            assert y1 == y2, "P + (-P)"
            m = mul(mul((3, 0), mul(x1, x1)), inv(mul((2, 0), y1)))
        else:
            m = mul(sub(y2, y1), inv(sub(x2, x1)))
        x3 = sub(sub(mul(m, m), x1), x2)
        return (x3, sub(mul(m, sub(x1, x3)), y1))

    acc = None
    for bit in bin(k)[2:]:
        acc = None if acc is None else add(acc, acc)
        if bit == "1":
            acc = pt if acc is None else add(acc, pt)
    return acc


def g2_is_on_curve(pt) -> bool:
    """y^2 = x^3 + 3/(9+u) over Fq2 (the check srs.rs:193-194 makes)."""
    (x0, x1), (y0, y1) = pt

    def mul(a, b):
        return ((a[0] * b[0] - a[1] * b[1]) % Q, (a[0] * b[1] + a[1] * b[0]) % Q)
    x, y = (x0, x1), (y0, y1)
    lhs = mul(y, y)
    x3 = mul(mul(x, x), x)
    # 3 / (9 + u) = 3 (9 - u) / 82
    inv82 = pow(82, -1, Q)
    b = (27 * inv82 % Q, (-3 * inv82) % Q)
    return lhs == ((x3[0] + b[0]) % Q, (x3[1] + b[1]) % Q)
