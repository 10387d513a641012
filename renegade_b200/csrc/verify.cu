// Host-side verifier of libb200prover: TurboPlonk / KZG proof verification, link-proof verification and the
// BN254 optimal-ate pairing they end in.  No device work: in the reference, too, verification stays on the
// CPU (SURVEY.md §8(a) a10).
//
// Replaces what the reference reaches through
//   `SingleProverCircuit::verify` -> `PlonkKzgSnark::<Bn254>::verify::<SolidityTranscript>(&vk, &statement
//     scalars, &proof, None)` (/root/reference/crates/circuits/circuit-types/src/traits.rs:1003-1019), and
//   `validate_*_link` -> `PlonkKzgSnark::verify_link_proof` (circuits-core/src/zk_circuits/proof_linking/
//     intent_only.rs:54-85),
// and the pairing of the reference's own SRS unit test (circuit-types/src/primitives/srs.rs:236-266:
// e(tau^i G, tau H) == e(tau^(i+1) G, H)).  The upstream code (mpc-jellyfish `verifier.rs`, ark-ec's bn
// pairing) is not vendored; what is restated here is the published algorithm:
//   * verifier: recompute the six challenges from the transcript, evaluate Z_H, L_1 and the public-input
//     polynomial at zeta, assemble the linearisation commitment D, the batched commitment F and evaluation E,
//     and check   e(W_z + u W_zw, [tau]_2) == e(zeta W_z + u zeta w W_zw + F - E G + u ([z] - z_w G), [1]_2);
//   * pairing: Fq12 = Fq[w] / (w^12 - 18 w^6 + 82) (so Fq2 = Fq[u]/(u^2 + 1) sits inside as u = w^6 - 9),
//     G2 on the sextic twist y^2 = x^3 + 3 / (9 + u), Miller loop over 6x + 2 with x = 4965661367192848881 and
//     the two Frobenius line steps, lines evaluated as sparse elements -y_P + (m x_P) w + (y_R - m x_R) w^3,
//     final exponentiation split into the easy part (q^6 - 1)(q^2 + 1) and the hard part by the x-addition chain of
//     Fuentes-Castaneda et al. (three exponentiations by x and Frobenius maps).
// Clarity first: flat Fq12 arithmetic, affine Miller steps; a verification is ~6 ms of host time.
// The transcript replay and the scalar assembly are verify_algebra.cuh's (shared with the device batch verifier,
// batch_verify.cu, which also calls the pairing below through pairing.h).
#include <cstring>
#include <mutex>
#include <vector>

#include "b200prover.h"
#include "device_ctx.h"
#include "pairing.h"
#include "verify_algebra.cuh"

namespace b200 {

namespace {

using Fq = FqCfg;
using Fr = FrCfg;

// ---- Fq2 = Fq[u] / (u^2 + 1) (struct fq2 in pairing.h) -----------------------------------------------------
inline fq2 fq2_add(const fq2& x, const fq2& y) { return {fe_add<Fq>(x.a, y.a), fe_add<Fq>(x.b, y.b)}; }
inline fq2 fq2_sub(const fq2& x, const fq2& y) { return {fe_sub<Fq>(x.a, y.a), fe_sub<Fq>(x.b, y.b)}; }
inline fq2 fq2_neg(const fq2& x) { return {fe_neg<Fq>(x.a), fe_neg<Fq>(x.b)}; }
inline fq2 fq2_mul(const fq2& x, const fq2& y) {
    const fe aa = fe_mul<Fq>(x.a, y.a), bb = fe_mul<Fq>(x.b, y.b);
    const fe cross = fe_mul<Fq>(fe_add<Fq>(x.a, x.b), fe_add<Fq>(y.a, y.b));
    return {fe_sub<Fq>(aa, bb), fe_sub<Fq>(fe_sub<Fq>(cross, aa), bb)};
}
inline fq2 fq2_mul_fq(const fq2& x, const fe& s) { return {fe_mul<Fq>(x.a, s), fe_mul<Fq>(x.b, s)}; }
inline fq2 fq2_sqr(const fq2& x) { return fq2_mul(x, x); }
inline fq2 fq2_inv(const fq2& x) {  // 1 / (a + b u) = (a - b u) / (a^2 + b^2)
    const fe n = fe_inv<Fq>(fe_add<Fq>(fe_sqr<Fq>(x.a), fe_sqr<Fq>(x.b)));
    return {fe_mul<Fq>(x.a, n), fe_neg<Fq>(fe_mul<Fq>(x.b, n))};
}
inline bool fq2_is_zero(const fq2& x) { return fe_is_zero(x.a) && fe_is_zero(x.b); }
inline bool fq2_eq(const fq2& x, const fq2& y) { return fe_eq(x.a, y.a) && fe_eq(x.b, y.b); }

// ---- Fq12 = Fq[w] / (w^12 - 18 w^6 + 82), flat coefficients -----------------------------------------------
struct fq12 {
    fe c[12];
};
fq12 fq12_one() {
    fq12 r;
    for (auto& v : r.c) v = fe_zero();
    r.c[0] = fe_one<Fq>();
    return r;
}
bool fq12_is_one(const fq12& a) {
    if (!fe_eq(a.c[0], fe_one<Fq>())) return false;
    for (int i = 1; i < 12; ++i)
        if (!fe_is_zero(a.c[i])) return false;
    return true;
}
fq12 fq12_mul(const fq12& a, const fq12& b) {
    fe t[23];
    for (auto& v : t) v = fe_zero();
    for (int i = 0; i < 12; ++i) {
        if (fe_is_zero(a.c[i])) continue;
        for (int j = 0; j < 12; ++j) t[i + j] = fe_add<Fq>(t[i + j], fe_mul<Fq>(a.c[i], b.c[j]));
    }
    const fe c18 = fe_from_u32<Fq>(18), c82 = fe_from_u32<Fq>(82);
    for (int k = 22; k >= 12; --k) {  // w^k = 18 w^(k-6) - 82 w^(k-12)
        if (fe_is_zero(t[k])) continue;
        t[k - 6] = fe_add<Fq>(t[k - 6], fe_mul<Fq>(c18, t[k]));
        t[k - 12] = fe_sub<Fq>(t[k - 12], fe_mul<Fq>(c82, t[k]));
    }
    fq12 r;
    for (int i = 0; i < 12; ++i) r.c[i] = t[i];
    return r;
}
// a^2 with the symmetric products taken once: 78 field products instead of 144
fq12 fq12_sqr(const fq12& a) {
    fe t[23];
    for (auto& v : t) v = fe_zero();
    for (int i = 0; i < 12; ++i) {
        if (fe_is_zero(a.c[i])) continue;
        t[2 * i] = fe_add<Fq>(t[2 * i], fe_sqr<Fq>(a.c[i]));
        const fe twice = fe_dbl<Fq>(a.c[i]);
        for (int j = i + 1; j < 12; ++j) t[i + j] = fe_add<Fq>(t[i + j], fe_mul<Fq>(twice, a.c[j]));
    }
    const fe c18 = fe_from_u32<Fq>(18), c82 = fe_from_u32<Fq>(82);
    for (int k = 22; k >= 12; --k) {
        if (fe_is_zero(t[k])) continue;
        t[k - 6] = fe_add<Fq>(t[k - 6], fe_mul<Fq>(c18, t[k]));
        t[k - 12] = fe_sub<Fq>(t[k - 12], fe_mul<Fq>(c82, t[k]));
    }
    fq12 r;
    for (int i = 0; i < 12; ++i) r.c[i] = t[i];
    return r;
}
// a + b u placed at w^k: u = w^6 - 9
void fq12_put(fq12* f, int k, const fq2& v) {
    const fe nine_b = fe_mul<Fq>(fe_from_u32<Fq>(9), v.b);
    f->c[k] = fe_add<Fq>(f->c[k], fe_sub<Fq>(v.a, nine_b));
    f->c[k + 6] = fe_add<Fq>(f->c[k + 6], v.b);
}
// x -> x^(q^6): w -> -w
fq12 fq12_conj(const fq12& a) {
    fq12 r = a;
    for (int i = 1; i < 12; i += 2) r.c[i] = fe_neg<Fq>(a.c[i]);
    return r;
}
// inverse by the extended Euclidean algorithm on polynomials over Fq (degree <= 12)
struct poly13 {
    fe c[13];
};
int poly_deg(const poly13& p) {
    int d = 12;
    while (d > 0 && fe_is_zero(p.c[d])) --d;
    return d;
}
fq12 fq12_inv(const fq12& a) {
    poly13 lm, hm, low, high;
    for (int i = 0; i < 13; ++i) lm.c[i] = hm.c[i] = low.c[i] = high.c[i] = fe_zero();
    lm.c[0] = fe_one<Fq>();
    for (int i = 0; i < 12; ++i) low.c[i] = a.c[i];
    high.c[0] = fe_from_u32<Fq>(82);
    high.c[6] = fe_neg<Fq>(fe_from_u32<Fq>(18));
    high.c[12] = fe_one<Fq>();
    while (poly_deg(low) > 0) {
        const int dl = poly_deg(low), dh = poly_deg(high);
        poly13 r, temp = high;
        for (auto& v : r.c) v = fe_zero();
        const fe inv_lead = fe_inv<Fq>(low.c[dl]);
        for (int i = dh - dl; i >= 0; --i) {
            r.c[i] = fe_mul<Fq>(temp.c[dl + i], inv_lead);
            for (int k = 0; k <= dl; ++k) temp.c[k + i] = fe_sub<Fq>(temp.c[k + i], fe_mul<Fq>(r.c[i], low.c[k]));
        }
        poly13 nm = hm, nw = high;
        for (int i = 0; i < 13; ++i)
            for (int j = 0; j < 13 - i; ++j) {
                if (fe_is_zero(r.c[j])) continue;
                nm.c[i + j] = fe_sub<Fq>(nm.c[i + j], fe_mul<Fq>(lm.c[i], r.c[j]));
                nw.c[i + j] = fe_sub<Fq>(nw.c[i + j], fe_mul<Fq>(low.c[i], r.c[j]));
            }
        hm = lm;
        high = low;
        lm = nm;
        low = nw;
    }
    const fe inv0 = fe_inv<Fq>(low.c[0]);
    fq12 out;
    for (int i = 0; i < 12; ++i) out.c[i] = fe_mul<Fq>(lm.c[i], inv0);
    return out;
}
fq12 fq12_pow(const fq12& a, const uint64_t* e, int limbs) {
    fq12 r = fq12_one();
    bool started = false;
    for (int i = limbs * 64 - 1; i >= 0; --i) {
        if (started) r = fq12_sqr(r);
        if ((e[i >> 6] >> (i & 63)) & 1) {
            r = started ? fq12_mul(r, a) : a;
            started = true;
        }
    }
    return r;
}

// Frobenius constants: gamma = w^(q^2 - 1) (a sixth root of unity in Fq) scales the coefficients of x^(q^2);
// for the points of the twist, (x, y)^q = (conj(x) * xi^((q-1)/3), conj(y) * xi^((q-1)/2)), xi = 9 + u.
struct PairingConsts {
    fe gamma_pow[6];  // gamma^k
    fq2 twist_frob_x, twist_frob_y;
    fq2 frob1[12];    // (w^k)^q = frob1[k] w^k: powers of xi^((q-1)/6), xi = w^6 = 9 + u
};
fq2 fq2_pow(const fq2& a, const uint64_t* e, int limbs) {
    fq2 r = {fe_one<Fq>(), fe_zero()};
    for (int i = limbs * 64 - 1; i >= 0; --i) {
        r = fq2_sqr(r);
        if ((e[i >> 6] >> (i & 63)) & 1) r = fq2_mul(r, a);
    }
    return r;
}
const PairingConsts& pairing_consts() {
    static PairingConsts pc;
    static std::once_flag once;
    std::call_once(once, [] {
        // q^2 - 1, little-endian limbs
        static const uint64_t q2m1[8] = {0x3b5458a2275d69b0ULL, 0xa602072d09eac101ULL, 0x4a50189c6d96cadcULL, 0x04689e957a1242c8ULL,
                                         0x26edfa5c34c6b38dULL, 0xb00b855116375606ULL, 0x599a6f7c0348d21cULL, 0x0925c4b8763cbf9cULL};
        fq12 w;
        for (auto& v : w.c) v = fe_zero();
        w.c[1] = fe_one<Fq>();
        const fq12 g = fq12_pow(w, q2m1, 8);  // w^(q^2 - 1) = gamma, an element of Fq: w^(q^2) = gamma w
        pc.gamma_pow[0] = fe_one<Fq>();
        pc.gamma_pow[1] = g.c[0];
        for (int k = 2; k < 6; ++k) pc.gamma_pow[k] = fe_mul<Fq>(pc.gamma_pow[k - 1], pc.gamma_pow[1]);
        // (q - 1) / 3 and (q - 1) / 2 from the modulus limbs
        uint64_t qm1[4];
        for (int i = 0; i < 4; ++i) qm1[i] = (uint64_t)Fq::mod(2 * i) | ((uint64_t)Fq::mod(2 * i + 1) << 32);
        qm1[0] -= 1;  // q is odd: no borrow
        uint64_t third[4], halfe[4];
        unsigned __int128 rem = 0;
        for (int i = 3; i >= 0; --i) {
            const unsigned __int128 cur = (rem << 64) | qm1[i];
            third[i] = (uint64_t)(cur / 3);
            rem = cur % 3;
        }
        for (int i = 0; i < 4; ++i) halfe[i] = (qm1[i] >> 1) | (i < 3 ? qm1[i + 1] << 63 : 0);
        const fq2 xi = {fe_from_u32<Fq>(9), fe_one<Fq>()};
        pc.twist_frob_x = fq2_pow(xi, third, 4);
        pc.twist_frob_y = fq2_pow(xi, halfe, 4);
        uint64_t sixth[4];  // (q - 1) / 6 = ((q - 1) / 3) / 2
        for (int i = 0; i < 4; ++i) sixth[i] = (third[i] >> 1) | (i < 3 ? third[i + 1] << 63 : 0);
        pc.frob1[0] = {fe_one<Fq>(), fe_zero()};
        pc.frob1[1] = fq2_pow(xi, sixth, 4);
        for (int k = 2; k < 12; ++k) pc.frob1[k] = fq2_mul(pc.frob1[k - 1], pc.frob1[1]);
    });
    return pc;
}
// x -> x^(q^2): coefficient of w^k scaled by gamma^(k mod 6)
fq12 fq12_frob2(const fq12& a) {
    const PairingConsts& pc = pairing_consts();
    fq12 r;
    for (int k = 0; k < 12; ++k) r.c[k] = fe_mul<Fq>(a.c[k], pc.gamma_pow[k % 6]);
    return r;
}
// x -> x^q: the coefficients are in Fq, so x^q = sum_k c_k (w^q)^k = sum_k c_k frob1[k] w^k with frob1[k] in Fq2 = Fq[u],
// u = w^6 - 9; the products land on w^k and w^(k+6) and fold back with w^12 = 18 w^6 - 82
fq12 fq12_frob1(const fq12& a) {
    const PairingConsts& pc = pairing_consts();
    fe t[18];
    for (auto& v : t) v = fe_zero();
    const fe nine = fe_from_u32<Fq>(9);
    for (int k = 0; k < 12; ++k) {
        if (fe_is_zero(a.c[k])) continue;
        const fq2& g = pc.frob1[k];
        t[k] = fe_add<Fq>(t[k], fe_mul<Fq>(a.c[k], fe_sub<Fq>(g.a, fe_mul<Fq>(nine, g.b))));
        t[k + 6] = fe_add<Fq>(t[k + 6], fe_mul<Fq>(a.c[k], g.b));
    }
    const fe c18 = fe_from_u32<Fq>(18), c82 = fe_from_u32<Fq>(82);
    for (int k = 17; k >= 12; --k) {
        t[k - 6] = fe_add<Fq>(t[k - 6], fe_mul<Fq>(c18, t[k]));
        t[k - 12] = fe_sub<Fq>(t[k - 12], fe_mul<Fq>(c82, t[k]));
    }
    fq12 r;
    for (int i = 0; i < 12; ++i) r.c[i] = t[i];
    return r;
}
g2_affine g2_frobenius(const g2_affine& p) {
    const PairingConsts& pc = pairing_consts();
    g2_affine r;
    r.inf = p.inf;
    r.x = fq2_mul(fq2{p.x.a, fe_neg<Fq>(p.x.b)}, pc.twist_frob_x);
    r.y = fq2_mul(fq2{p.y.a, fe_neg<Fq>(p.y.b)}, pc.twist_frob_y);
    return r;
}

// One Miller step: multiplies f by the line through r and s (the tangent when r == s) evaluated at the G1
// point (px, py), and replaces r by r + s.
void line_and_add(fq12* f, g2_affine* r, const g2_affine& s, const fe& px, const fe& py) {
    if (r->inf || s.inf) {  // not reached for points of prime order inside the loop bounds
        if (r->inf) *r = s;
        return;
    }
    fq12 line;
    for (auto& v : line.c) v = fe_zero();
    fq2 m;
    if (fq2_eq(r->x, s.x)) {
        if (!fq2_eq(r->y, s.y) || fq2_is_zero(r->y)) {  // vertical line x_P - x_R w^2
            line.c[0] = px;
            fq12_put(&line, 2, fq2_neg(r->x));
            *f = fq12_mul(line, *f);
            r->inf = true;
            return;
        }
        const fq2 xx = fq2_sqr(r->x);
        m = fq2_mul(fq2_add(fq2_add(xx, xx), xx), fq2_inv(fq2_add(r->y, r->y)));
    } else {
        m = fq2_mul(fq2_sub(s.y, r->y), fq2_inv(fq2_sub(s.x, r->x)));
    }
    // untwisted slope = m w:  l(P) = m w (x_P - x_R w^2) - (y_P - y_R w^3) = -y_P + (m x_P) w + (y_R - m x_R) w^3
    line.c[0] = fe_neg<Fq>(py);
    fq12_put(&line, 1, fq2_mul_fq(m, px));
    fq12_put(&line, 3, fq2_sub(r->y, fq2_mul(m, r->x)));
    *f = fq12_mul(line, *f);  // sparse operand first: fq12_mul skips its zero coefficients
    const fq2 nx = fq2_sub(fq2_sub(fq2_sqr(m), r->x), s.x);
    const fq2 ny = fq2_sub(fq2_mul(m, fq2_sub(r->x, nx)), r->y);
    r->x = nx;
    r->y = ny;
}

// Product of the Miller functions of k pairs (P_i in G1, Q_i in G2) before the final exponentiation: one accumulator, so
// the 64 squarings are shared by all pairs
fq12 miller_loop_product(const g1_affine* ps, const g2_affine* qs, size_t k) {
    fq12 f = fq12_one();
    std::vector<size_t> live;
    for (size_t i = 0; i < k; ++i)
        if (!g1_affine_is_inf(ps[i]) && !qs[i].inf) live.push_back(i);  // a pair with an identity contributes 1
    if (live.empty()) return f;
    static const uint64_t ate[2] = {0x9d797039be763ba8ULL, 0x1ULL};  // 6x + 2, 65 bits
    std::vector<g2_affine> r(live.size());
    for (size_t j = 0; j < live.size(); ++j) r[j] = qs[live[j]];
    for (int i = 63; i >= 0; --i) {
        f = fq12_sqr(f);
        const bool bit = (ate[i >> 6] >> (i & 63)) & 1;
        for (size_t j = 0; j < live.size(); ++j) {
            const g1_affine& p = ps[live[j]];
            line_and_add(&f, &r[j], r[j], p.x, p.y);
            if (bit) line_and_add(&f, &r[j], qs[live[j]], p.x, p.y);
        }
    }
    for (size_t j = 0; j < live.size(); ++j) {
        const g1_affine& p = ps[live[j]];
        const g2_affine q1 = g2_frobenius(qs[live[j]]);
        g2_affine nq2 = g2_frobenius(q1);
        nq2.y = fq2_neg(nq2.y);
        line_and_add(&f, &r[j], q1, p.x, p.y);
        line_and_add(&f, &r[j], nq2, p.x, p.y);
    }
    return f;
}

// t^x for the curve parameter x = 4965661367192848881 (63 bits, 28 of them set)
fq12 fq12_pow_x(const fq12& t) {
    static const uint64_t x[1] = {0x44e992b44a6909f1ULL};
    return fq12_pow(t, x, 1);
}

fq12 final_exponentiation(const fq12& f) {
    // easy part: f^((q^6 - 1)(q^2 + 1)); afterwards t is in the cyclotomic subgroup, where the inverse is the conjugate
    fq12 t = fq12_mul(fq12_conj(f), fq12_inv(f));
    t = fq12_mul(fq12_frob2(t), t);
    // hard part (q^4 - q^2 + 1) / r by the addition chain of Fuentes-Castaneda, Knapp and Rodriguez-Henriquez ("Faster
    // hashing to G2", SAC 2011; the schedule ark-ec's bn model uses): three exponentiations by x, Frobenius maps and a
    // dozen products instead of a 762-bit square-and-multiply.  It raises t to c (q^4 - q^2 + 1) / r with a c prime to r
    // (checked on the exponents: tests/test_pairing.py), which is one exactly when the reduced pairing is.
    auto neg_x = [](const fq12& a) { return fq12_conj(fq12_pow_x(a)); };  // a^(-x)
    const fq12 y0 = neg_x(t);
    const fq12 y1 = fq12_sqr(y0);
    const fq12 y2 = fq12_sqr(y1);
    fq12 y3 = fq12_mul(y2, y1);
    const fq12 y4 = neg_x(y3);
    const fq12 y5 = fq12_sqr(y4);
    fq12 y6 = neg_x(y5);
    y3 = fq12_conj(y3);
    y6 = fq12_conj(y6);
    const fq12 y7 = fq12_mul(y6, y4);
    const fq12 y8 = fq12_mul(y7, y3);
    const fq12 y9 = fq12_mul(y8, y1);
    const fq12 y10 = fq12_mul(y8, y4);
    const fq12 y11 = fq12_mul(y10, t);
    const fq12 y13 = fq12_mul(fq12_frob1(y9), y11);
    const fq12 y14 = fq12_mul(fq12_frob2(y8), y13);
    const fq12 y15 = fq12_mul(fq12_conj(t), y9);
    return fq12_mul(fq12_frob1(fq12_frob2(y15)), y14);  // q^3 = q o q^2
}

// ---- G1 sums of the host verifiers (host XYZZ arithmetic of ec.cuh) ----------------------------------------
// sum_i s_i P_i over a term list, evaluated with ONE chain of doublings (Straus: 254 doublings in all and a mixed
// addition per set scalar bit, instead of 254 doublings per term)
g1_affine g1_sum_terms(const G1Term* terms, int n) {
    std::vector<g1_affine> pts;
    std::vector<fe> scalars;  // canonical (non-Montgomery) limbs
    for (int i = 0; i < n; ++i) {
        if (g1_affine_is_inf(terms[i].p) || fe_is_zero(terms[i].s)) continue;
        pts.push_back(terms[i].p);
        scalars.push_back(fe_from_mont<Fr>(terms[i].s));
    }
    g1_xyzz acc = g1_xyzz_inf();
    for (int bit = 253; bit >= 0; --bit) {
        acc = g1_dbl(acc);
        for (size_t i = 0; i < pts.size(); ++i)
            if ((scalars[i].l[bit >> 5] >> (bit & 31)) & 1u) acc = g1_add_mixed(acc, pts[i]);
    }
    return g1_to_affine(acc);
}

g1_affine g1_load(const uint64_t xy[8]) {
    g1_affine p;
    std::memcpy(&p, xy, 64);
    return p;
}

// e(A, [tau]_2) == e(B, [1]_2)   <=>   e(A, [tau]_2) * e(-B, [1]_2) == 1
int check_operands(const OperandTerms& t, const uint64_t g2_h[16], const uint64_t g2_tau_h[16], const char* who, int* accepted) {
    const g1_affine ps[2] = {g1_sum_terms(t.a, t.na), g1_affine_neg(g1_sum_terms(t.b, t.nb))};
    const g2_affine qs[2] = {g2_load(g2_tau_h), g2_load(g2_h)};
    if (!g2_on_curve(qs[0]) || !g2_on_curve(qs[1])) {
        set_error(std::string(who) + ": G2 point not on curve");
        return B200_ERR_NOT_ON_CURVE;
    }
    *accepted = pairing_product_is_one(ps, qs, 2) ? 1 : 0;
    return B200_OK;
}

}  // namespace

bool g2_on_curve(const g2_affine& p) {
    if (p.inf) return true;
    // b' = 3 / (9 + u) = 3 (9 - u) / 82
    const fe inv82 = fe_inv<Fq>(fe_from_u32<Fq>(82));
    const fq2 b = {fe_mul<Fq>(fe_from_u32<Fq>(27), inv82), fe_neg<Fq>(fe_mul<Fq>(fe_from_u32<Fq>(3), inv82))};
    return fq2_eq(fq2_sqr(p.y), fq2_add(fq2_mul(fq2_sqr(p.x), p.x), b));
}

g2_affine g2_load(const uint64_t rec[16]) {
    g2_affine p;
    std::memcpy(&p.x.a, rec, 32);
    std::memcpy(&p.x.b, rec + 4, 32);
    std::memcpy(&p.y.a, rec + 8, 32);
    std::memcpy(&p.y.b, rec + 12, 32);
    p.inf = fq2_is_zero(p.x) && fq2_is_zero(p.y);
    return p;
}

bool pairing_product_is_one(const g1_affine* ps, const g2_affine* qs, size_t k) {
    return fq12_is_one(final_exponentiation(miller_loop_product(ps, qs, k)));
}

}  // namespace b200

using namespace b200;

extern "C" {

int b200_pairing_check(const uint64_t* g1_points, const uint64_t* g2_points, size_t k, int* is_one) {
    B200_TRY
    if ((k && (!g1_points || !g2_points)) || !is_one) return B200_ERR_INVALID;
    std::vector<g1_affine> ps(k);
    std::vector<g2_affine> qs(k);
    for (size_t i = 0; i < k; ++i) {
        ps[i] = g1_load(g1_points + 8 * i);
        qs[i] = g2_load(g2_points + 16 * i);
        if (!g1_affine_on_curve(ps[i]) || !g2_on_curve(qs[i])) {
            set_error("pairing_check: point not on curve");
            return B200_ERR_NOT_ON_CURVE;
        }
    }
    *is_one = pairing_product_is_one(ps.data(), qs.data(), k) ? 1 : 0;
    return B200_OK;
    B200_CATCH
}

int b200_plonk_verify(unsigned log_n, size_t num_inputs, const uint64_t* k, const uint64_t* selector_comms,
                      const uint64_t* sigma_comms, const uint64_t* pub_inputs, const b200_proof* proof_in,
                      const uint64_t g2_h[16], const uint64_t g2_tau_h[16], int* accepted) {
    B200_TRY
    if (!k || !selector_comms || !sigma_comms || !proof_in || !g2_h || !g2_tau_h || !accepted || (num_inputs && !pub_inputs) ||
        log_n > 28)
        return B200_ERR_INVALID;
    *accepted = 0;
    const VkIn vk = {reinterpret_cast<const fe*>(k), reinterpret_cast<const g1_affine*>(selector_comms),
                     reinterpret_cast<const g1_affine*>(sigma_comms)};
    std::vector<uint8_t> buf(plonk_transcript_bytes(num_inputs));
    TranscriptT<ByteSpan> tr(ByteSpan{buf.data(), 0, buf.size()});
    OperandTerms t;
    if (!plonk_verify_terms(log_n, num_inputs, vk, reinterpret_cast<const fe*>(pub_inputs),
                            *reinterpret_cast<const ProofIn*>(proof_in), host_root_of_unity(log_n), tr, &t))
        return B200_OK;  // rejected
    return check_operands(t, g2_h, g2_tau_h, "verify", accepted);
    B200_CATCH
}

int b200_plonk_verify_link(const uint64_t* comm1, const uint64_t* comm2, unsigned alignment, size_t offset, size_t size,
                           const b200_link_proof* proof, const uint64_t g2_h[16], const uint64_t g2_tau_h[16], int* accepted) {
    B200_TRY
    if (!comm1 || !comm2 || !proof || !g2_h || !g2_tau_h || !accepted || alignment > 28 || size == 0) return B200_ERR_INVALID;
    *accepted = 0;
    uint8_t buf[kLinkTranscriptBytes];
    TranscriptT<ByteSpan> tr(ByteSpan{buf, 0, sizeof(buf)});
    OperandTerms t;
    if (!link_verify_terms(g1_load(comm1), g1_load(comm2), g1_load(proof->quotient_commitment), g1_load(proof->opening_proof),
                           host_root_of_unity(alignment), offset, size, tr, &t))
        return B200_OK;  // rejected
    return check_operands(t, g2_h, g2_tau_h, "verify_link", accepted);
    B200_CATCH
}

}  // extern "C"
