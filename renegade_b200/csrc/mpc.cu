// Collaborative TurboPlonk prover on the device: one party per call, additive shares over Fr, a caller-supplied
// all-gather between the parties (include/b200prover.h, "collaborative prover (device)").
//
// Each round of prove() in plonk.cu runs here on this party's shares, with the same kernels.  Linear steps (transforms,
// blinding, commitments, evaluations, opening quotients) are share-wise; the parties exchange partial commitments and
// add them.  Products of shared values are Beaver multiplications with preprocessed triples ([a], [b], [ab]): open
// d = x - a and e = y - b, then [xy] = [c] + d [b] + e [a] + d e (party 0 adds d e).  All independent products of one
// multiplicative depth share one exchange; a square uses a triple with b = a and opens one difference.  Round 2
// divides by den with a mask r: it forms [den r] and [num r] at the same level, opens den r and keeps
// [num / den] = [num r] / (den r).  The quotient runs on the key's nc resident cosets (26 products per point, 4 levels).
// Every opened value and every decision derived from it is the same on every party, so parties agree on every
// outcome.  The opened proof equals b200_plonk_prove on the summed witness and blinders, byte for byte.
#include <sys/random.h>

#include <cerrno>
#include <condition_variable>
#include <cstring>
#include <map>

#include "plonk_internal.cuh"
#include "transcript.h"

namespace b200 {

namespace {

constexpr size_t kHdr = 32;  // message header: exchange index, payload bytes, two zero words
constexpr int kMaxProd = 10;

// one multiplicative level: product k is x_k * y_k (y_k == x_k for a square) over `len` elements, triples at
// a/b/c + k * len, its differences at msg[off_k ..) (d) and, unless a square, msg[off_k + len ..) (e)
struct BeaverLevel {
    const fe* x[kMaxProd];
    const fe* y[kMaxProd];
    fe* out[kMaxProd];
    uint32_t off[kMaxProd];
    uint8_t sq[kMaxProd];
    int count;
    size_t len;
    const fe *a, *b, *c;
};

// gathers the masked differences of every product of a level into this party's (mapped, pinned) outgoing message
__global__ void k_beaver_open(BeaverLevel L, fe* __restrict__ msg) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int k = blockIdx.y;
    if (i >= L.len) return;
    const size_t t = (size_t)k * L.len + i;
    fe* dst = msg + L.off[k];
    fe_store(dst + i, FSUB(fe_load(L.x[k] + i), fe_load_ro(L.a + t)));
    if (!L.sq[k]) fe_store(dst + L.len + i, FSUB(fe_load(L.y[k] + i), fe_load_ro(L.b + t)));
}

// sums the P received messages on the fly: out = c + d b + e a (+ d e on party 0)
__global__ void k_beaver_close(BeaverLevel L, const uint8_t* __restrict__ all, size_t stride, int parties, int party0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int k = blockIdx.y;
    if (i >= L.len) return;
    const size_t t = (size_t)k * L.len + i;
    fe d = fe_zero(), e = fe_zero();
    for (int p = 0; p < parties; ++p) {
        const fe* m = reinterpret_cast<const fe*>(all + (size_t)p * stride + kHdr) + L.off[k];
        d = FADD(d, fe_load_ro(m + i));
        if (!L.sq[k]) e = FADD(e, fe_load_ro(m + L.len + i));
    }
    const fe a = fe_load_ro(L.a + t);
    fe r;
    if (L.sq[k]) {
        r = FADD(fe_load_ro(L.c + t), FMUL(FADD(d, d), a));
        if (party0) r = FADD(r, fe_sqr<Fr>(d));
    } else {
        r = FADD(fe_load_ro(L.c + t), FADD(FMUL(d, fe_load_ro(L.b + t)), FMUL(e, a)));
        if (party0) r = FADD(r, FMUL(d, e));
    }
    fe_store(L.out[k] + i, r);
}

// ---- authenticated mode: every shared x also has a MAC share [alpha x]; opened values leave gamma records ----------
// true iff the limbs are below the field's modulus (a received element must be a canonical residue)
template <class Cfg>
FF_HD bool canonical(const fe& v) {
    for (int k = 7; k >= 0; --k)
        if (v.l[k] != Cfg::mod(k)) return v.l[k] < Cfg::mod(k);
    return false;
}

// the MAC plane of one Beaver level: MAC shares of x, y, out and of the triples; gamma records in message order
struct MacLevel {
    const fe* x[kMaxProd];
    const fe* y[kMaxProd];
    fe* out[kMaxProd];
    const fe *a, *b, *c;
    fe* log;
    fe key;    // this party's share of the MAC key
    int* bad;  // set when a received difference is not canonical
};

// k_beaver_close on both planes: out = c + d b + e a (+ d e on party 0), [alpha out] = [alpha c] + d [alpha b] +
// e [alpha a] + key d e, and gamma = ([alpha x] - [alpha a]) - key d (likewise e) for every opened difference
__global__ void k_auth_beaver_close(BeaverLevel L, MacLevel M, const uint8_t* __restrict__ all, size_t stride, int parties,
                                    int party0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int k = blockIdx.y;
    if (i >= L.len) return;
    const size_t t = (size_t)k * L.len + i;
    fe d = fe_zero(), e = fe_zero();
    bool ok = true;
    for (int p = 0; p < parties; ++p) {
        const fe* m = reinterpret_cast<const fe*>(all + (size_t)p * stride + kHdr) + L.off[k];
        const fe dv = fe_load_ro(m + i);
        ok = ok && canonical<FrCfg>(dv);
        d = FADD(d, dv);
        if (!L.sq[k]) {
            const fe ev = fe_load_ro(m + L.len + i);
            ok = ok && canonical<FrCfg>(ev);
            e = FADD(e, ev);
        }
    }
    if (!ok) *M.bad = 1;
    const fe a = fe_load_ro(L.a + t), am = fe_load_ro(M.a + t);
    fe r, rm, de;
    if (L.sq[k]) {
        const fe d2 = FADD(d, d);
        r = FADD(fe_load_ro(L.c + t), FMUL(d2, a));
        rm = FADD(fe_load_ro(M.c + t), FMUL(d2, am));
        de = fe_sqr<Fr>(d);
    } else {
        r = FADD(fe_load_ro(L.c + t), FADD(FMUL(d, fe_load_ro(L.b + t)), FMUL(e, a)));
        rm = FADD(fe_load_ro(M.c + t), FADD(FMUL(d, fe_load_ro(M.b + t)), FMUL(e, am)));
        de = FMUL(d, e);
        fe_store(M.log + L.off[k] + L.len + i, FSUB(FSUB(fe_load(M.y[k] + i), fe_load_ro(M.b + t)), FMUL(M.key, e)));
    }
    fe_store(M.log + L.off[k] + i, FSUB(FSUB(fe_load(M.x[k] + i), am), FMUL(M.key, d)));
    if (party0) r = FADD(r, de);
    fe_store(L.out[k] + i, r);
    fe_store(M.out[k] + i, FADD(rm, FMUL(M.key, de)));
}

// k_sum_open with the check: out = the sum, log = mac - key out, bad set on a non-canonical element
__global__ void k_auth_sum_open(const uint8_t* __restrict__ all, size_t stride, size_t len, int parties, fe* __restrict__ out,
                                const fe* __restrict__ mac, fe key, fe* __restrict__ log, int* bad) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    fe s = fe_zero();
    bool ok = true;
    for (int p = 0; p < parties; ++p) {
        const fe v = fe_load_ro(reinterpret_cast<const fe*>(all + (size_t)p * stride + kHdr) + i);
        ok = ok && canonical<FrCfg>(v);
        s = FADD(s, v);
    }
    if (!ok) *bad = 1;
    fe_store(out + i, s);
    fe_store(log + i, FSUB(fe_load_ro(mac + i), FMUL(key, s)));
}

// gamma records of values opened on the host: log = mac - key opened
__global__ void k_auth_gamma(const fe* __restrict__ mac, const fe* __restrict__ opened, size_t len, fe key, fe* __restrict__ log) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    fe_store(log + i, FSUB(fe_load_ro(mac + i), FMUL(key, fe_load_ro(opened + i))));
}

// out[i] = sum over the P received messages of element off + i
__global__ void k_sum_open(const uint8_t* __restrict__ all, size_t stride, size_t off, size_t len, int parties, fe* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    fe s = fe_zero();
    for (int p = 0; p < parties; ++p) s = FADD(s, fe_load_ro(reinterpret_cast<const fe*>(all + (size_t)p * stride + kHdr) + off + i));
    fe_store(out + i, s);
}

// the permutation factors of rounds 2 and 3 on this party's shares: nf_j = w_j + beta k_j x + gamma and
// df_j = w_j + beta sigma_j + gamma, the public terms on party 0 only
__global__ void k_mpc_perm_factors(const fe* __restrict__ w, size_t wstride, const fe* __restrict__ pts, const fe* __restrict__ sig,
                                   size_t len, KArr k, fe beta, fe gamma, int party0, fe* __restrict__ nf, fe* __restrict__ df) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    const fe bx = FMUL(beta, fe_load_ro(pts + i));
#pragma unroll 1
    for (int j = 0; j < NW; ++j) {
        fe a = fe_load_ro(w + j * wstride + i), b = a;
        if (party0) {
            a = FADD(a, FADD(FMUL(k.v[j], bx), gamma));
            b = FADD(b, FADD(FMUL(beta, fe_load_ro(sig + j * len + i)), gamma));
        }
        fe_store(nf + j * len + i, a);
        fe_store(df + j * len + i, b);
    }
}

// both planes of k_mpc_perm_factors in one pass over the public tables: the MAC plane adds key x (public term) on every
// party
__global__ void k_auth_perm_factors(const fe* __restrict__ w, const fe* __restrict__ wm, size_t wstride, const fe* __restrict__ pts,
                                    const fe* __restrict__ sig, size_t len, KArr k, fe beta, fe gamma, int party0, fe key,
                                    fe* __restrict__ nf, fe* __restrict__ df, fe* __restrict__ nfm, fe* __restrict__ dfm) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    const fe bx = FMUL(beta, fe_load_ro(pts + i));
#pragma unroll 1
    for (int j = 0; j < NW; ++j) {
        const fe tn = FADD(FMUL(k.v[j], bx), gamma);
        const fe td = FADD(FMUL(beta, fe_load_ro(sig + j * len + i)), gamma);
        fe a = fe_load_ro(w + j * wstride + i), b = a;
        if (party0) {
            a = FADD(a, tn);
            b = FADD(b, td);
        }
        fe_store(nf + j * len + i, a);
        fe_store(df + j * len + i, b);
        const fe am = fe_load_ro(wm + j * wstride + i);
        fe_store(nfm + j * len + i, FADD(am, FMUL(key, tn)));
        fe_store(dfm + j * len + i, FADD(am, FMUL(key, td)));
    }
}

// z(w x) on the quotient domain: the next point of the same coset
__global__ void k_next_on_coset(const fe* __restrict__ z, size_t m, unsigned log_n, fe* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const size_t nmask = ((size_t)1 << log_n) - 1;
    fe_store(out + i, fe_load_ro(z + ((i & ~nmask) | ((i + 1) & nmask))));
}

struct MpcQuotArgs {
    const fe* sel;   // 13 x m resident coset evaluations
    const fe* ext;   // 7 x m: wire shares 0..4, public-input polynomial, z share
    const fe* w01;   // products of round 3: w0 w1, w2 w3, w0 w1 w2 w3 w4, w_j^5 (4 x m), z num, z(wx) den
    const fe* w23;
    const fe* w01234;
    const fe* p5;
    const fe* zn;
    const fe* zd;
    const fe* l1_inv;
    fe* out;
    size_t m;
    unsigned log_n;
    int party0;
    fe alpha, alpha2;
    fe zh_inv[8];
};
// this party's share of the quotient's evaluations (k_quotient on shares; public constants on party 0)
__global__ void __launch_bounds__(128) k_mpc_quotient(MpcQuotArgs a) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.m) return;
    const size_t m = a.m;
    fe acc = a.party0 ? FADD(fe_load_ro(a.sel + 11 * m + i), fe_load_ro(a.ext + 5 * m + i)) : fe_zero();
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        acc = FADD(acc, FMUL(fe_load_ro(a.sel + j * m + i), fe_load_ro(a.ext + j * m + i)));
        acc = FADD(acc, FMUL(fe_load_ro(a.sel + (6 + j) * m + i), fe_load_ro(a.p5 + j * m + i)));
    }
    acc = FADD(acc, FMUL(fe_load_ro(a.sel + 4 * m + i), fe_load_ro(a.w01 + i)));
    acc = FADD(acc, FMUL(fe_load_ro(a.sel + 5 * m + i), fe_load_ro(a.w23 + i)));
    acc = FADD(acc, FMUL(fe_load_ro(a.sel + 12 * m + i), fe_load_ro(a.w01234 + i)));
    acc = FSUB(acc, FMUL(fe_load_ro(a.sel + 10 * m + i), fe_load_ro(a.ext + 4 * m + i)));
    acc = FADD(acc, FMUL(a.alpha, FSUB(fe_load_ro(a.zn + i), fe_load_ro(a.zd + i))));
    acc = FMUL(acc, a.zh_inv[i >> a.log_n]);
    fe zm1 = fe_load_ro(a.ext + 6 * m + i);
    if (a.party0) zm1 = FSUB(zm1, fe_one<Fr>());
    acc = FADD(acc, FMUL(FMUL(a.alpha2, zm1), fe_load_ro(a.l1_inv + i)));
    fe_store(a.out + i, acc);
}

// the operands of one plane of the quotient
struct QuotPlane {
    const fe *ext, *w01, *w23, *w01234, *p5, *zn, *zd;
    fe* out;
};
// one plane of k_mpc_quotient: `pub` weighs the public terms (the public-input evaluations, the q_c selector, the 1
// of z - 1), [party 0] for shares and the key share for MACs
__device__ __forceinline__ void quot_plane(const MpcQuotArgs& a, const QuotPlane& q, size_t i, const fe& pub) {
    const size_t m = a.m;
    fe acc = FMUL(pub, FADD(fe_load_ro(a.sel + 11 * m + i), fe_load_ro(a.ext + 5 * m + i)));
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        acc = FADD(acc, FMUL(fe_load_ro(a.sel + j * m + i), fe_load_ro(q.ext + j * m + i)));
        acc = FADD(acc, FMUL(fe_load_ro(a.sel + (6 + j) * m + i), fe_load_ro(q.p5 + j * m + i)));
    }
    acc = FADD(acc, FMUL(fe_load_ro(a.sel + 4 * m + i), fe_load_ro(q.w01 + i)));
    acc = FADD(acc, FMUL(fe_load_ro(a.sel + 5 * m + i), fe_load_ro(q.w23 + i)));
    acc = FADD(acc, FMUL(fe_load_ro(a.sel + 12 * m + i), fe_load_ro(q.w01234 + i)));
    acc = FSUB(acc, FMUL(fe_load_ro(a.sel + 10 * m + i), fe_load_ro(q.ext + 4 * m + i)));
    acc = FADD(acc, FMUL(a.alpha, FSUB(fe_load_ro(q.zn + i), fe_load_ro(q.zd + i))));
    acc = FMUL(acc, a.zh_inv[i >> a.log_n]);
    const fe zm1 = FSUB(fe_load_ro(q.ext + 6 * m + i), pub);
    acc = FADD(acc, FMUL(FMUL(a.alpha2, zm1), fe_load_ro(a.l1_inv + i)));
    fe_store(q.out + i, acc);
}
// both planes of the quotient in one launch; the MAC plane's public terms are weighted by the key share
__global__ void __launch_bounds__(128) k_auth_quotient(MpcQuotArgs a, QuotPlane mac, fe key) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.m) return;
    const QuotPlane sh{a.ext, a.w01, a.w23, a.w01234, a.p5, a.zn, a.zd, a.out};
    quot_plane(a, sh, i, a.party0 ? fe_one<Fr>() : fe_zero());
    quot_plane(a, mac, i, key);
}

// ---- dealer (INSECURE stand-in for an offline phase) ----------------------------------------------------------------
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
// element i of stream `key` under `seed`: 254 random bits reduced once mod r (2^254 < 2 r), used as a Montgomery form
__device__ __forceinline__ fe prg_fr(uint64_t seed, uint64_t key, uint64_t i) {
    const uint64_t h = mix64(seed + 0x9E3779B97F4A7C15ULL * (key + 1));
    fe v;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint64_t x = mix64(h + 0x9E3779B97F4A7C15ULL * (4 * i + k + 1));
        v.l[2 * k] = (uint32_t)x;
        v.l[2 * k + 1] = (uint32_t)(x >> 32);
    }
    v.l[7] &= 0x3FFFFFFFu;
    bool ge = true;
    for (int k = 7; k >= 0; --k)
        if (v.l[k] != FrCfg::mod(k)) {
            ge = v.l[k] > FrCfg::mod(k);
            break;
        }
    if (ge) {
        uint64_t borrow = 0;
        for (int k = 0; k < 8; ++k) {
            const uint64_t d = (uint64_t)v.l[k] - FrCfg::mod(k) - borrow;
            v.l[k] = (uint32_t)d;
            borrow = (d >> 32) & 1u;
        }
    }
    return v;
}
struct SquareRanges {
    size_t beg[2], end[2];
};
// party p's shares of triple i (streams 0, 1, 2: a, b, c) or of mask i (stream 3).  Parties below P - 1 take their
// shares straight from the PRG; the last party computes the values and subtracts the others' shares.
__global__ void k_dealer(uint64_t seed, int party, int parties, size_t count, int masks, SquareRanges sq, fe* __restrict__ a,
                         fe* __restrict__ b, fe* __restrict__ c) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const int ns = masks ? 1 : 3;
    const uint64_t s0 = masks ? 3 : 0;
    auto key = [&](int who, int s) { return (uint64_t)who * 8 + s0 + (uint64_t)s; };
    if (party < parties - 1) {
        a[i] = prg_fr(seed, key(party, 0), i);
        if (!masks) {
            b[i] = prg_fr(seed, key(party, 1), i);
            c[i] = prg_fr(seed, key(party, 2), i);
        }
        return;
    }
    const int V = 255;  // the stream of the values themselves
    fe v[3];
    v[0] = prg_fr(seed, key(V, 0), i);
    if (!masks) {
        const bool square = (i >= sq.beg[0] && i < sq.end[0]) || (i >= sq.beg[1] && i < sq.end[1]);
        v[1] = square ? v[0] : prg_fr(seed, key(V, 1), i);
        v[2] = FMUL(v[0], v[1]);
    }
    for (int q = 0; q < parties - 1; ++q)
        for (int s = 0; s < ns; ++s) v[s] = FSUB(v[s], prg_fr(seed, key(q, s), i));
    a[i] = v[0];
    if (!masks) {
        b[i] = v[1];
        c[i] = v[2];
    }
}

// the authenticated dealer's MAC streams and input-sharing streams, disjoint from the triple streams of `seed`
__device__ __forceinline__ uint64_t mac_seed(uint64_t seed) { return mix64(seed ^ 0x6D61632D6B657921ULL); }
__device__ __forceinline__ uint64_t input_seed(uint64_t seed) { return mix64(seed ^ 0x696E7075742D7368ULL); }
// party p's share of the MAC key alpha = prg(V, 7); the last party's share completes the sum
__device__ fe dealer_key_share(uint64_t seed, int party, int parties) {
    const uint64_t sm = mac_seed(seed);
    if (party < parties - 1) return prg_fr(sm, (uint64_t)party * 8 + 7, 0);
    fe k = prg_fr(sm, 255ull * 8 + 7, 0);
    for (int q = 0; q < parties - 1; ++q) k = FSUB(k, prg_fr(sm, (uint64_t)q * 8 + 7, 0));
    return k;
}
// party p's MAC shares of triple i (alpha a, alpha b, alpha c) or of mask i, under the values k_dealer shares; thread 0
// also writes the party's key share to key_out (may be null)
__global__ void k_dealer_mac(uint64_t seed, int party, int parties, size_t count, int masks, SquareRanges sq, fe* __restrict__ am,
                             fe* __restrict__ bm, fe* __restrict__ cm, fe* __restrict__ key_out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0 && key_out) *key_out = dealer_key_share(seed, party, parties);
    if (i >= count) return;
    const int ns = masks ? 1 : 3;
    const uint64_t s0 = masks ? 3 : 0, sm = mac_seed(seed);
    auto key = [&](int who, int s) { return (uint64_t)who * 8 + s0 + (uint64_t)s; };
    fe* out[3] = {am, bm, cm};
    if (party < parties - 1) {
        for (int s = 0; s < ns; ++s) out[s][i] = prg_fr(sm, key(party, s), i);
        return;
    }
    const int V = 255;
    const fe alpha = prg_fr(sm, (uint64_t)V * 8 + 7, 0);
    fe v[3];
    v[0] = prg_fr(seed, key(V, 0), i);
    if (!masks) {
        const bool square = (i >= sq.beg[0] && i < sq.end[0]) || (i >= sq.beg[1] && i < sq.end[1]);
        v[1] = square ? v[0] : prg_fr(seed, key(V, 1), i);
        v[2] = FMUL(v[0], v[1]);
    }
    for (int s = 0; s < ns; ++s) {
        fe t = FMUL(alpha, v[s]);
        for (int q = 0; q < parties - 1; ++q) t = FSUB(t, prg_fr(sm, key(q, s), i));
        out[s][i] = t;
    }
}
// party p's authenticated shares of values the caller knows in full, under the MAC key of `seed`
__global__ void k_dealer_input(uint64_t seed, int party, int parties, size_t count, const fe* __restrict__ values,
                               fe* __restrict__ shares, fe* __restrict__ macs) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint64_t si = input_seed(seed);
    if (party < parties - 1) {
        shares[i] = prg_fr(si, (uint64_t)party * 2, i);
        macs[i] = prg_fr(si, (uint64_t)party * 2 + 1, i);
        return;
    }
    const fe v = values[i];
    fe s = v, t = FMUL(prg_fr(mac_seed(seed), 255ull * 8 + 7, 0), v);
    for (int q = 0; q < parties - 1; ++q) {
        s = FSUB(s, prg_fr(si, (uint64_t)q * 2, i));
        t = FSUB(t, prg_fr(si, (uint64_t)q * 2 + 1, i));
    }
    shares[i] = s;
    macs[i] = t;
}

}  // namespace

// ---- preprocessing -------------------------------------------------------------------------------------------------
// Triple layout of one proof (n = 2^log_n, m = nc n): round 2 takes 10 n (levels 1-4) then n - d for each doubling
// step d = 1, 2, .., n / 2; round 3 takes 26 m from R3 = that total: levels of 10, 7, 7, 2 products of m; the last
// triple is the degree check's.  Squares (b = a): [R3 + 2m, R3 + 6m) and [R3 + 11m, R3 + 15m).  Masks: n, then 1.
struct MpcLayout {
    size_t n, m, r3, triples, masks;
    SquareRanges sq;
};
static MpcLayout mpc_layout(const ProvingKey* pk) {
    MpcLayout L;
    L.n = pk->n;
    L.m = pk->m;
    size_t t = 10 * L.n;
    for (size_t d = 1; d < L.n; d <<= 1) t += L.n - d;
    L.r3 = t;
    L.triples = t + 26 * L.m + 1;
    L.masks = L.n + 1;
    L.sq.beg[0] = L.r3 + 2 * L.m;
    L.sq.end[0] = L.r3 + 6 * L.m;
    L.sq.beg[1] = L.r3 + 11 * L.m;
    L.sq.end[1] = L.r3 + 15 * L.m;
    return L;
}

struct MpcPrep {
    int device = 0;
    uint64_t pk_id = 0;
    size_t n = 0, m = 0, triples = 0, masks = 0;
    fe *a = nullptr, *b = nullptr, *c = nullptr, *mask = nullptr;
    fe *am = nullptr, *bm = nullptr, *cm = nullptr, *mask_mac = nullptr;  // MAC shares (authenticated preprocessing)
    bool auth = false;
    bool used = false;
    ~MpcPrep() {
        for (fe* p : {a, b, c, mask, am, bm, cm, mask_mac})
            if (p) cudaFree(p);
    }
};

static int prep_alloc(Context* c, const ProvingKey* pk, MpcPrep** out, bool auth = false) {
    const MpcLayout L = mpc_layout(pk);
    MpcPrep* p = new MpcPrep();
    p->device = c->device;
    p->n = L.n;
    p->m = L.m;
    p->triples = L.triples;
    p->masks = L.masks;
    int rc;
    if ((rc = alloc_fe(&p->a, L.triples)) || (rc = alloc_fe(&p->b, L.triples)) || (rc = alloc_fe(&p->c, L.triples)) ||
        (rc = alloc_fe(&p->mask, L.masks))) {
        delete p;
        return rc;
    }
    p->auth = auth;
    if (auth && ((rc = alloc_fe(&p->am, L.triples)) || (rc = alloc_fe(&p->bm, L.triples)) || (rc = alloc_fe(&p->cm, L.triples)) ||
                 (rc = alloc_fe(&p->mask_mac, L.masks)))) {
        delete p;
        return rc;
    }
    *out = p;
    return B200_OK;
}

// ---- local group: an in-process all-gather between threads --------------------------------------------------------
struct LocalGroup;
struct LocalMember {
    LocalGroup* g;
    int party;
};
struct LocalGroup {
    int parties;
    unsigned timeout_ms;
    std::mutex mu;
    std::condition_variable cv;
    bool failed = false;
    struct Round {
        std::vector<uint8_t> data;
        size_t bytes = 0;
        int arrived = 0, copied = 0, left = 0;
    };
    std::map<uint64_t, Round> rounds;
    std::vector<uint64_t> calls;
    std::vector<LocalMember> members;
};

static void local_abort(void* user) {
    LocalGroup* g = static_cast<LocalMember*>(user)->g;
    std::lock_guard<std::mutex> lk(g->mu);
    g->failed = true;
    g->cv.notify_all();
}

static int local_all_gather(void* user, const void* mine, size_t bytes, void* all) {
    LocalMember* me = static_cast<LocalMember*>(user);
    LocalGroup* g = me->g;
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(g->timeout_ms);
    std::unique_lock<std::mutex> lk(g->mu);
    auto fail = [&](const char* why) {
        g->failed = true;
        g->cv.notify_all();
        set_error(why);
        return B200_ERR_INVALID;
    };
    if (g->failed) return fail("local group: aborted");
    const uint64_t r = g->calls[me->party]++;
    LocalGroup::Round& R = g->rounds[r];
    if (R.arrived == 0) {
        R.bytes = bytes;
        R.data.resize((size_t)g->parties * bytes);
    } else if (R.bytes != bytes) {
        return fail("local group: parties sent messages of different sizes");
    }
    ++R.arrived;
    lk.unlock();
    std::memcpy(R.data.data() + (size_t)me->party * bytes, mine, bytes);  // own slot; the buffer is sized already
    lk.lock();
    ++R.copied;
    g->cv.notify_all();
    while (R.copied < g->parties && !g->failed)
        if (g->cv.wait_until(lk, deadline) == std::cv_status::timeout && R.copied < g->parties)
            return fail("local group: timed out waiting for the other parties");
    if (g->failed) return fail("local group: aborted");
    lk.unlock();
    std::memcpy(all, R.data.data(), (size_t)g->parties * bytes);
    lk.lock();
    if (++R.left == g->parties) g->rounds.erase(r);
    return B200_OK;
}

// ---- one party's run -----------------------------------------------------------------------------------------------
// `count` commitments of this party's share polynomials (`len` coefficients, `stride` apart); the identity as zeros
static int commit_partials(Context* c, const Bases* srs, const fe* d_coeffs, size_t len, size_t stride, unsigned count,
                           g1_affine* out, cudaStream_t st) {
    int inf[8];
    if (count > 8) return B200_ERR_INVALID;
    const int rc = msm_device_batch(srs, 0, d_coeffs, len, stride, count, /*montgomery=*/1, &c->msm, st, out, inf);
    if (rc != B200_OK) return rc;
    for (unsigned i = 0; i < count; ++i)
        if (inf[i]) std::memset(&out[i], 0, sizeof(out[i]));
    return B200_OK;
}

static void keccak(const void* p, size_t n, uint8_t out[32]) { Keccak256::hash(static_cast<const uint8_t*>(p), n, out); }

// G1 point received from another party: canonical coordinates on y^2 = x^3 + 3 (the identity is 64 zero bytes)
static bool point_ok(const g1_affine& q) { return canonical<FqCfg>(q.x) && canonical<FqCfg>(q.y) && g1_affine_on_curve(q); }

// State of the authenticated mode of one call.  The MAC plane of a shared workspace buffer lives `total` elements after
// it; gamma records of every opened value go to `log` in opening order; the MAC planes of the committed polynomials
// and their opened commitments are kept for the point check.
struct Auth {
    fe key;                              // this party's MAC-key share alpha_i
    const fe* ws = nullptr;              // share plane [ws, ws + total), MAC plane [ws + total, ws + 2 total)
    size_t total = 0;
    const MpcPrep* prep = nullptr;       // masks live there (MAC plane: prep->mask_mac)
    fe* log = nullptr;                   // device
    size_t log_len = 0, log_cap = 0;
    fe* stage = nullptr;                 // device staging of host-opened values (stage_cap elements)
    size_t stage_cap = 0;
    int* bad = nullptr;                  // device: a received element was not canonical
    bool reject = false;                 // host: malformed data or a reveal that does not match its commitment
    uint8_t seed[32];
    std::vector<uint8_t> seed_comms;     // H(seed_p) of every party, from exchange 0
    std::vector<const fe*> polys;        // MAC planes of the committed polynomials
    std::vector<size_t> lens;
    std::vector<g1_affine> comms;        // their opened commitments

    const fe* mac(const fe* p) const {
        if (p >= ws && p < ws + total) return p + total;
        if (prep && p >= prep->mask && p < prep->mask + prep->masks) return prep->mask_mac + (p - prep->mask);
        return nullptr;
    }
    fe* mac(fe* p) const { return const_cast<fe*>(mac(static_cast<const fe*>(p))); }
    // gamma records of `len` values opened on the host, whose MAC shares are at d_mac
    int record(const fe* d_mac, const fe* h_open, size_t len, cudaStream_t st) {
        if (len > stage_cap || log_len + len > log_cap || !d_mac) {
            set_error("collaborative prover: MAC log out of step");
            return B200_ERR_INVALID;
        }
        B200_CUDA(cudaMemcpyAsync(stage, h_open, len * sizeof(fe), cudaMemcpyHostToDevice, st));
        B200_LAUNCH(k_auth_gamma, grid_for(len, 256), 256, 0, st)(d_mac, stage, len, key, log + log_len);
        B200_CUDA(cudaStreamSynchronize(st));
        log_len += len;
        return B200_OK;
    }
};

struct Party {
    Context* c;
    const b200_mpc_transport* tr;
    int party, P;
    cudaStream_t st;
    uint64_t exchange = 0;
    double bytes = 0, ms = 0, triples = 0;
    uint8_t* send = nullptr;
    uint8_t* recv = nullptr;
    size_t stride = 0;  // bytes per party in recv of the last exchange
    Auth* au = nullptr;  // authenticated mode

    int reserve(size_t payload) {
        int rc;
        if ((rc = c->mpc_send.reserve(kHdr + payload)) != B200_OK) return rc;
        if ((rc = c->mpc_recv.reserve((size_t)P * (kHdr + payload))) != B200_OK) return rc;
        send = static_cast<uint8_t*>(c->mpc_send.p);
        recv = static_cast<uint8_t*>(c->mpc_recv.p);
        return B200_OK;
    }
    // the payload is in send + kHdr (the device work that wrote it has completed)
    int exchange_now(size_t payload) {
        uint64_t* h = reinterpret_cast<uint64_t*>(send);
        h[0] = exchange;
        h[1] = payload;
        h[2] = h[3] = 0;
        const size_t msg = kHdr + payload;
        const auto t0 = std::chrono::steady_clock::now();
        const int r = tr->all_gather(tr->user, send, msg, recv);
        ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (r != 0) {
            set_error("collaborative prover: the transport's all_gather failed (exchange " + std::to_string(exchange) + ")");
            return r < 0 ? r : B200_ERR_INVALID;
        }
        for (int p = 0; p < P; ++p) {
            const uint64_t* hp = reinterpret_cast<const uint64_t*>(recv + (size_t)p * msg);
            if (hp[0] != exchange || hp[1] != payload) {
                set_error("collaborative prover: party " + std::to_string(p) + " sent the wrong exchange or size (exchange " +
                          std::to_string(exchange) + ")");
                return B200_ERR_INVALID;
            }
        }
        stride = msg;
        bytes += (double)msg;
        ++exchange;
        return B200_OK;
    }
    const uint8_t* payload_of(int p) const { return recv + (size_t)p * stride + kHdr; }

    // sums of `count` partial commitments (64-byte affine records at byte offset `off` of every payload)
    int sum_points(size_t off, unsigned count, g1_affine* out) {
        std::vector<uint64_t> pts((size_t)P * 8);
        std::vector<int> inf(P);
        for (unsigned k = 0; k < count; ++k) {
            for (int p = 0; p < P; ++p) {
                std::memcpy(&pts[(size_t)p * 8], payload_of(p) + off + 64 * k, 64);
                if (au && !point_ok(*reinterpret_cast<const g1_affine*>(&pts[(size_t)p * 8]))) {
                    au->reject = true;  // finish the call with verdict reject; the sum is not used
                    std::memset(&pts[(size_t)p * 8], 0, 64);
                }
                bool z = true;
                for (int w = 0; w < 8; ++w) z = z && pts[(size_t)p * 8 + w] == 0;
                inf[p] = z;
            }
            int oinf = 0;
            const int rc = b200_g1_sum_affine(pts.data(), inf.data(), (size_t)P, reinterpret_cast<uint64_t*>(&out[k]), &oinf);
            if (rc != B200_OK) return rc;
            if (oinf) std::memset(&out[k], 0, sizeof(g1_affine));
        }
        return B200_OK;
    }
    // sum of `count` field elements at byte offset `off` of every payload (host)
    void sum_fe(size_t off, size_t count, fe* out) const {
        for (size_t i = 0; i < count; ++i) {
            fe s = fe_zero();
            for (int p = 0; p < P; ++p) {
                fe v;
                std::memcpy(&v, payload_of(p) + off + 32 * i, 32);
                if (au && !canonical<FrCfg>(v)) au->reject = true;
                s = FADD(s, v);
            }
            out[i] = s;
        }
    }
    // open `count` partial commitments of `count` share polynomials (`len` coefficients, `stride` apart), summed
    int open_commitments(const Bases* srs, const fe* d_coeffs, size_t len, size_t pstride, unsigned count, g1_affine* out,
                         const void* prefix = nullptr, size_t prefix_bytes = 0) {
        std::vector<g1_affine> part(count);
        int rc = commit_partials(c, srs, d_coeffs, len, pstride, count, part.data(), st);
        if (rc != B200_OK) return rc;
        const size_t payload = prefix_bytes + 64 * count;
        if ((rc = reserve(payload)) != B200_OK) return rc;
        if (prefix_bytes) std::memcpy(send + kHdr, prefix, prefix_bytes);
        std::memcpy(send + kHdr + prefix_bytes, part.data(), 64 * count);
        if ((rc = exchange_now(payload)) != B200_OK) return rc;
        if ((rc = sum_points(prefix_bytes, count, out)) != B200_OK) return rc;
        if (au)
            for (unsigned k = 0; k < count; ++k) {
                au->polys.push_back(au->mac(d_coeffs + k * pstride));
                au->lens.push_back(len);
                au->comms.push_back(out[k]);
            }
        return B200_OK;
    }
    // one Beaver level; `extra` (device, may be null): `extra_len` shares opened in the same message (summed on the host)
    int beaver(const MpcPrep* prep, size_t& t_used, BeaverLevel L, const fe* extra = nullptr, size_t extra_len = 0,
               fe* extra_sum = nullptr) {
        size_t off = 0;
        for (int k = 0; k < L.count; ++k) {
            L.off[k] = (uint32_t)off;
            off += L.sq[k] ? L.len : 2 * L.len;
        }
        const size_t used = (size_t)L.count * L.len;
        if (t_used + used > prep->triples) {
            set_error("collaborative prover: preprocessing exhausted");
            return B200_ERR_INVALID;
        }
        L.a = prep->a + t_used;
        L.b = prep->b + t_used;
        L.c = prep->c + t_used;
        const size_t payload = (off + extra_len) * sizeof(fe);
        int rc = reserve(payload);
        if (rc != B200_OK) return rc;
        fe* msg = reinterpret_cast<fe*>(send + kHdr);
        B200_LAUNCH(k_beaver_open, dim3(grid_for(L.len, 256), (unsigned)L.count), 256, 0, st)(L, msg);
        if (extra_len) B200_CUDA(cudaMemcpyAsync(msg + off, extra, extra_len * sizeof(fe), cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        if ((rc = exchange_now(payload)) != B200_OK) return rc;
        if (au) {
            MacLevel M{};
            for (int k = 0; k < L.count; ++k) {
                M.x[k] = au->mac(L.x[k]);
                M.y[k] = au->mac(L.y[k]);
                M.out[k] = au->mac(L.out[k]);
                if (!M.x[k] || !M.y[k] || !M.out[k] || au->log_len + off > au->log_cap) {
                    set_error("collaborative prover: MAC plane out of step");
                    return B200_ERR_INVALID;
                }
            }
            M.a = prep->am + t_used;
            M.b = prep->bm + t_used;
            M.c = prep->cm + t_used;
            M.log = au->log + au->log_len;
            M.key = au->key;
            M.bad = au->bad;
            B200_LAUNCH(k_auth_beaver_close, dim3(grid_for(L.len, 256), (unsigned)L.count), 256, 0, st)(L, M, recv, stride, P, party == 0);
            au->log_len += off;
        } else {
            B200_LAUNCH(k_beaver_close, dim3(grid_for(L.len, 256), (unsigned)L.count), 256, 0, st)(L, recv, stride, P, party == 0);
        }
        if (extra_len) sum_fe(off * sizeof(fe), extra_len, extra_sum);
        B200_CUDA(cudaStreamSynchronize(st));  // the next exchange reuses the receive buffer
        if (au && extra_len && (rc = au->record(au->mac(extra), extra_sum, extra_len, st)) != B200_OK) return rc;
        t_used += used;
        triples += (double)used;
        return B200_OK;
    }
    // opens `len` shares on the device: out = the sum over the parties
    int open_device(const fe* src, size_t len, fe* out) {
        int rc = reserve(len * sizeof(fe));
        if (rc != B200_OK) return rc;
        B200_CUDA(cudaMemcpyAsync(send + kHdr, src, len * sizeof(fe), cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        if ((rc = exchange_now(len * sizeof(fe))) != B200_OK) return rc;
        if (au) {
            if (!au->mac(src) || au->log_len + len > au->log_cap) {
                set_error("collaborative prover: MAC log out of step");
                return B200_ERR_INVALID;
            }
            B200_LAUNCH(k_auth_sum_open, grid_for(len, 256), 256, 0, st)(recv, stride, len, P, out, au->mac(src), au->key,
                                                                         au->log + au->log_len, au->bad);
            au->log_len += len;
        } else {
            B200_LAUNCH(k_sum_open, grid_for(len, 256), 256, 0, st)(recv, stride, 0, len, P, out);
        }
        B200_CUDA(cudaStreamSynchronize(st));
        return B200_OK;
    }
    // the three exchanges of the MAC check that end an authenticated call; `ok` is true when every party's check passed
    // and nothing malformed was received
    int auth_check(const Bases* srs, fe* lin_buf, fe* scratch, bool* ok);
    // opens `count` host values
    int open_host(const fe* vals, size_t count, fe* out) {
        int rc = reserve(count * sizeof(fe));
        if (rc != B200_OK) return rc;
        std::memcpy(send + kHdr, vals, count * sizeof(fe));
        if ((rc = exchange_now(count * sizeof(fe))) != B200_OK) return rc;
        sum_fe(0, count, out);
        return B200_OK;
    }
};

// 32 bytes from the OS's CSPRNG
static int draw_random(uint8_t* p, size_t n) {
    while (n) {
        const ssize_t r = getrandom(p, n, 0);
        if (r < 0) {
            if (errno == EINTR) continue;
            set_error("collaborative prover: getrandom failed");
            return B200_ERR_INVALID;
        }
        p += r;
        n -= (size_t)r;
    }
    return B200_OK;
}

// a challenge of the MAC check: keccak(tag || joint seed) read big-endian, reduced mod r
static fe check_challenge(const char* tag, const uint8_t joint[32]) {
    Keccak256 k;
    k.absorb(reinterpret_cast<const uint8_t*>(tag), std::strlen(tag));
    k.absorb(joint, 32);
    uint8_t h[32];
    k.finish(h);
    fe acc = fe_zero();
    const fe c256 = fe_from_u32<Fr>(256);
    for (int i = 0; i < 32; ++i) acc = FADD(FMUL(acc, c256), fe_from_u32<Fr>(h[i]));
    return acc;
}

// Three exchanges after the last opening.  (1) The seeds committed in exchange 0 are revealed and checked; the joint
// seed gives rho_s and rho_p.  (2) This party commits to H(sigma || Sigma_pt || verdict || salt), with
// sigma = rho_s Gamma(rho_s) over the gamma log and Sigma_pt = MSM(srs, sum_k rho_p^k [alpha p_k]) - key sum_k rho_p^k C_k
// over the committed polynomials.  (3) The records are revealed, checked against the commitments, and accepted when the
// sigmas sum to 0, the points to the identity and every verdict is "accept".
int Party::auth_check(const Bases* srs, fe* lin_buf, fe* scratch, bool* ok) {
    *ok = false;
    int rc;
    if ((rc = reserve(32)) != B200_OK) return rc;
    std::memcpy(send + kHdr, au->seed, 32);
    if ((rc = exchange_now(32)) != B200_OK) return rc;
    std::vector<uint8_t> seeds((size_t)P * 32);
    for (int p = 0; p < P; ++p) {
        uint8_t h[32];
        keccak(payload_of(p), 32, h);
        if (std::memcmp(h, &au->seed_comms[(size_t)p * 32], 32) != 0) au->reject = true;
        std::memcpy(&seeds[(size_t)p * 32], payload_of(p), 32);
    }
    uint8_t joint[32];
    keccak(seeds.data(), seeds.size(), joint);
    const fe rho_s = check_challenge("b200 mac check: opened scalars", joint);
    const fe rho_p = check_challenge("b200 mac check: commitments", joint);
    // scalar check
    fe sigma = fe_zero();
    if (au->log_len) {
        const fe* polys[1] = {au->log};
        const size_t lens[1] = {au->log_len};
        eval_batch(polys, lens, &rho_s, 1, au->stage, scratch, st);
        fe g;
        B200_CUDA(cudaMemcpyAsync(&g, au->stage, sizeof(fe), cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        sigma = FMUL(rho_s, g);
    }
    // point check
    const size_t K = au->polys.size();
    if (K == 0 || K > (size_t)kMaxLin) {
        set_error("collaborative prover: MAC check out of step");
        return B200_ERR_INVALID;
    }
    LinArgs la{};
    g1_xyzz csum = g1_xyzz_inf();
    fe w = fe_one<Fr>();
    size_t len = 0;
    for (size_t k = 0; k < K; ++k) {
        la.p[k] = au->polys[k];
        la.len[k] = (uint32_t)au->lens[k];
        la.s[k] = w;
        csum = g1_add(csum, g1_mul_bits(au->comms[k], fe_from_mont<Fr>(w), 254));
        len = au->lens[k] > len ? au->lens[k] : len;
        w = FMUL(w, rho_p);
    }
    la.count = (int)K;
    B200_LAUNCH(k_lincomb, grid_for(len, 128), 128, 0, st)(la, len, lin_buf);
    g1_affine mi;
    if ((rc = commit_partials(c, srs, lin_buf, len, len, 1, &mi, st)) != B200_OK) return rc;
    const g1_xyzz t = g1_mul_bits(g1_to_affine(csum), fe_from_mont<Fr>(fe_neg<Fr>(au->key)), 254);
    const g1_affine spt = g1_to_affine(g1_add_mixed(t, mi));
    int bad = 0;
    B200_CUDA(cudaMemcpy(&bad, au->bad, sizeof(int), cudaMemcpyDeviceToHost));
    const bool verdict = !au->reject && !bad;
    // commit, then reveal: sigma (32) || Sigma_pt (64) || verdict (32: 1 = accept, then zeros) || salt (32)
    uint8_t rec[160] = {};
    std::memcpy(rec, &sigma, 32);
    std::memcpy(rec + 32, &spt, 64);
    rec[96] = verdict ? 1 : 0;
    if ((rc = draw_random(rec + 128, 32)) != B200_OK) return rc;
    if ((rc = reserve(32)) != B200_OK) return rc;
    keccak(rec, sizeof(rec), send + kHdr);
    if ((rc = exchange_now(32)) != B200_OK) return rc;
    std::vector<uint8_t> comms((size_t)P * 32);
    for (int p = 0; p < P; ++p) std::memcpy(&comms[(size_t)p * 32], payload_of(p), 32);
    if ((rc = reserve(sizeof(rec))) != B200_OK) return rc;
    std::memcpy(send + kHdr, rec, sizeof(rec));
    if ((rc = exchange_now(sizeof(rec))) != B200_OK) return rc;
    bool good = verdict;
    fe ssum = fe_zero();
    g1_xyzz psum = g1_xyzz_inf();
    for (int p = 0; p < P; ++p) {
        const uint8_t* r = payload_of(p);
        uint8_t h[32];
        keccak(r, sizeof(rec), h);
        good = good && std::memcmp(h, &comms[(size_t)p * 32], 32) == 0 && r[96] == 1;
        fe s;
        g1_affine q;
        std::memcpy(&s, r, 32);
        std::memcpy(&q, r + 32, 64);
        good = good && canonical<FrCfg>(s) && point_ok(q);
        if (!good) break;
        ssum = FADD(ssum, s);
        psum = g1_add_mixed(psum, q);
    }
    *ok = good && fe_is_zero(ssum) && g1_xyzz_is_inf(psum);
    return B200_OK;
}

static BeaverLevel level(size_t len) {
    BeaverLevel L{};
    L.len = len;
    return L;
}
static void add(BeaverLevel& L, const fe* x, const fe* y, fe* out) {
    L.x[L.count] = x;
    L.y[L.count] = y ? y : x;
    L.out[L.count] = out;
    L.sq[L.count] = y == nullptr;
    ++L.count;
}

// authenticated (pt.au set): h_wire_macs / h_blinder_macs are the MAC shares of the wires and blinders, h_link_mac
// receives those of the linking polynomial, and the call ends with the MAC check (B200_ERR_MAC when it fails)
static int mpc_prove(Party& pt, const ProvingKey* pk, MpcPrep* prep, const fe* h_wires, const fe* h_pub_inputs,
                     const fe* h_blinders, ProofOut* proof, fe* h_link_share, fe* h_challenges, const fe* h_wire_macs = nullptr,
                     const fe* h_blinder_macs = nullptr, fe* h_link_mac = nullptr) {
    Context* c = pt.c;
    const size_t n = pk->n, m = pk->m;
    const unsigned log_n = pk->log_n;
    const bool p0 = pt.party == 0;
    cudaStream_t st = pt.st;
    const MpcLayout LY = mpc_layout(pk);
    const size_t S = n + 4;
    // device workspace
    const size_t hs = 4 * (S / CH + 4 * CH + 64), es = kMaxEval * (S / CH + S / CH / CH + 2 * CH + 16);
    const size_t total = NW * n + 6 * S + S + 10 * m + 14 * n + 7 * m + m + 26 * m + m + NW * S + S + 2 * (S + 8) + hs + es + 64 + 32;
    int rc;
    Auth* au = pt.au;
    // authenticated: the MAC plane, the gamma log (at most two differences per triple, den r, the tail, r' q[deg] and
    // the six evaluations), a staging area for host openings and the log's evaluation scratch
    const size_t log_cap = 2 * LY.triples + n + m + 8, stage_cap = m + 8, lscr = log_cap / CH + log_cap / CH / CH + 2 * CH + 16;
    const size_t auth_total = au ? total + log_cap + stage_cap + lscr + 1 : 0;
    if ((rc = c->mpc_ws.reserve((total + auth_total) * sizeof(fe))) != B200_OK) return rc;
    if ((rc = c->ntt_scratch.reserve((size_t)7 * m * sizeof(fe))) != B200_OK) return rc;
    fe* p = reinterpret_cast<fe*>(c->mpc_ws.p);
    fe* lscr_p = nullptr;
    if (au) {
        fe* base = p + 2 * total;
        au->ws = p;
        au->total = total;
        au->log = base;
        au->log_cap = log_cap;
        au->stage = base + log_cap;
        au->stage_cap = stage_cap;
        lscr_p = au->stage + stage_cap;
        au->bad = reinterpret_cast<int*>(lscr_p + lscr);
        B200_CUDA(cudaMemsetAsync(au->bad, 0, sizeof(int), st));
    }
    auto M = [&](const fe* x) { return au->mac(const_cast<fe*>(x)); };
    auto take = [&](size_t k) { fe* r = p; p += k; return r; };
    fe* wires_ev = take(NW * n);
    fe* wpoly = take(6 * S);  // 5 wire shares, then the public-input polynomial
    fe* pi_poly = wpoly + NW * S;
    fe* zpoly = take(S);
    fe* nf = take(5 * m);
    fe* df = take(5 * m);
    fe* r2 = take(14 * n);
    fe* ext = take(7 * m);
    fe* zw = take(m);
    fe* pr = take(26 * m);
    fe* quot = take(m);
    fe* split = take(NW * S);
    fe* lin = take(S);
    fe* sdiv = take(2 * (S + 8));
    fe* hscr = take(hs);
    fe* escr = take(es);
    fe* evals = take(64);
    fe* d_bl = take(32);
    fe* nscr = reinterpret_cast<fe*>(c->ntt_scratch.p);
    Domain* dn = nullptr;
    if ((rc = get_domain(c, log_n, &dn)) != B200_OK) return rc;
    const fe one = fe_one<Fr>();
    size_t t_used = 0;

    SolidityTranscript tr;
    tr.append_u32_be(254);
    tr.append_u64_be((uint64_t)n);
    tr.append_u64_be((uint64_t)pk->num_inputs);
    for (int i = 0; i < NW; ++i) tr.append_field_elem(pk->k.v[i]);
    for (int s = 0; s < NS; ++s) tr.append_commitment(pk->sel_comms[s]);
    for (int i = 0; i < NW; ++i) tr.append_commitment(pk->sig_comms[i]);
    for (size_t i = 0; i < pk->num_inputs; ++i) tr.append_field_elem(h_pub_inputs[i]);
    uint8_t statement[64];
    {
        SolidityTranscript probe = tr;  // the state a challenge would have now: binds the key and the public inputs
        probe.get_and_append_challenge();
        std::memcpy(statement, probe.state(), 64);
    }

    // ---- round 1 ------------------------------------------------------------------------------------------------
    B200_CUDA(cudaMemcpyAsync(wires_ev, h_wires, NW * n * sizeof(fe), cudaMemcpyDefault, st));
    B200_CUDA(cudaMemcpyAsync(d_bl, h_blinders, 17 * sizeof(fe), cudaMemcpyDefault, st));
    B200_CUDA(cudaMemsetAsync(wpoly, 0, 6 * S * sizeof(fe), st));
    if (pk->num_inputs) B200_CUDA(cudaMemcpyAsync(pi_poly, h_pub_inputs, pk->num_inputs * sizeof(fe), cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemcpy2DAsync(wpoly, S * sizeof(fe), wires_ev, n * sizeof(fe), n * sizeof(fe), NW, cudaMemcpyDeviceToDevice, st));
    if ((rc = ntt_device(dn, wpoly, nscr, 1, 0, NW + 1, S, st)) != B200_OK) return rc;
    B200_LAUNCH(k_blind_wires, 1, 32, 0, st)(wpoly, S, n, d_bl);
    if ((rc = coset_evals(pk, dn, wpoly, S, n + 2, NW + 1, ext, nscr, st)) != B200_OK) return rc;
    uint8_t prefix[96];  // the statement, then (authenticated) the commitment H(seed_i) to this party's check seed
    std::memcpy(prefix, statement, 64);
    if (au) {
        au->prep = prep;
        B200_CUDA(cudaMemcpyAsync(M(wires_ev), h_wire_macs, NW * n * sizeof(fe), cudaMemcpyDefault, st));
        B200_CUDA(cudaMemcpyAsync(M(d_bl), h_blinder_macs, 17 * sizeof(fe), cudaMemcpyDefault, st));
        B200_CUDA(cudaMemsetAsync(M(wpoly), 0, 6 * S * sizeof(fe), st));
        B200_CUDA(cudaMemcpy2DAsync(M(wpoly), S * sizeof(fe), M(wires_ev), n * sizeof(fe), n * sizeof(fe), NW, cudaMemcpyDeviceToDevice, st));
        if ((rc = ntt_device(dn, M(wpoly), nscr, 1, 0, NW, S, st)) != B200_OK) return rc;
        B200_LAUNCH(k_blind_wires, 1, 32, 0, st)(M(wpoly), S, n, M(d_bl));
        if ((rc = coset_evals(pk, dn, M(wpoly), S, n + 2, NW, M(ext), nscr, st)) != B200_OK) return rc;
        keccak(au->seed, 32, prefix + 64);
    }
    // first exchange: the statement and the 5 partial wire commitments
    if ((rc = pt.open_commitments(pk->srs, wpoly, n + 2, S, NW, proof->wires_poly_comms, prefix, au ? 96 : 64)) != B200_OK) return rc;
    for (int q = 1; q < pt.P; ++q)
        if (std::memcmp(pt.payload_of(q), pt.payload_of(0), 64) != 0) {
            set_error("collaborative prover: the parties disagree on the statement (verifying key or public inputs)");
            return B200_ERR_INVALID;
        }
    if (au) {
        au->seed_comms.resize((size_t)pt.P * 32);
        for (int q = 0; q < pt.P; ++q) std::memcpy(&au->seed_comms[(size_t)q * 32], pt.payload_of(q) + 64, 32);
        if (h_link_mac) B200_CUDA(cudaMemcpyAsync(h_link_mac, M(wpoly), (n + 2) * sizeof(fe), cudaMemcpyDeviceToHost, st));
    }
    if (h_link_share) B200_CUDA(cudaMemcpyAsync(h_link_share, wpoly, (n + 2) * sizeof(fe), cudaMemcpyDeviceToHost, st));
    for (int i = 0; i < NW; ++i) tr.append_commitment(proof->wires_poly_comms[i]);

    // ---- round 2 ------------------------------------------------------------------------------------------------
    const fe beta = tr.get_and_append_challenge();
    const fe gamma = tr.get_and_append_challenge();
    if (au)
        B200_LAUNCH(k_auth_perm_factors, grid_for(n, 128), 128, 0, st)(wires_ev, M(wires_ev), n, pk->dom, pk->sig_evals, n, pk->k, beta, gamma,
                                                                       p0 ? 1 : 0, au->key, nf, df, M(nf), M(df));
    else
        B200_LAUNCH(k_mpc_perm_factors, grid_for(n, 128), 128, 0, st)(wires_ev, n, pk->dom, pk->sig_evals, n, pk->k, beta, gamma, p0 ? 1 : 0, nf, df);
    {
        fe *n01 = r2, *n23 = r2 + n, *d01 = r2 + 2 * n, *d23 = r2 + 3 * n, *n0123 = r2 + 4 * n, *d0123 = r2 + 5 * n;
        fe *num = r2 + 6 * n, *den = r2 + 7 * n, *denr = r2 + 8 * n, *numr = r2 + 9 * n, *x = r2 + 10 * n, *x2 = r2 + 11 * n;
        fe* pub = r2 + 12 * n;  // den r, opened
        BeaverLevel L = level(n);
        add(L, nf, nf + n, n01);
        add(L, nf + 2 * n, nf + 3 * n, n23);
        add(L, df, df + n, d01);
        add(L, df + 2 * n, df + 3 * n, d23);
        if ((rc = pt.beaver(prep, t_used, L)) != B200_OK) return rc;
        L = level(n);
        add(L, n01, n23, n0123);
        add(L, d01, d23, d0123);
        if ((rc = pt.beaver(prep, t_used, L)) != B200_OK) return rc;
        L = level(n);
        add(L, n0123, nf + 4 * n, num);
        add(L, d0123, df + 4 * n, den);
        if ((rc = pt.beaver(prep, t_used, L)) != B200_OK) return rc;
        L = level(n);
        add(L, den, prep->mask, denr);
        add(L, num, prep->mask, numr);
        if ((rc = pt.beaver(prep, t_used, L)) != B200_OK) return rc;
        if ((rc = pt.open_device(denr, n, pub)) != B200_OK) return rc;
        if (au) {  // [alpha num / den] = [alpha num r] / (den r), before pub is overwritten
            B200_CUDA(cudaMemcpyAsync(M(pub), pub, n * sizeof(fe), cudaMemcpyDeviceToDevice, st));
            batch_inverse_enqueue(M(numr), M(pub), M(r2 + 13 * n), n, st);
            B200_CUDA(cudaMemcpyAsync(M(x), M(pub), n * sizeof(fe), cudaMemcpyDeviceToDevice, st));
        }
        batch_inverse_enqueue(numr, pub, r2 + 13 * n, n, st);  // pub <- [num r] / (den r) = [num / den]
        B200_CUDA(cudaMemcpyAsync(x, pub, n * sizeof(fe), cudaMemcpyDeviceToDevice, st));
        // inclusive prefix products by doubling: x'[i] = x[i] x[i - d] for i >= d
        for (size_t d = 1; d < n; d <<= 1) {
            B200_CUDA(cudaMemcpyAsync(x2, x, d * sizeof(fe), cudaMemcpyDeviceToDevice, st));
            if (au) B200_CUDA(cudaMemcpyAsync(M(x2), M(x), d * sizeof(fe), cudaMemcpyDeviceToDevice, st));
            L = level(n - d);
            add(L, x + d, x, x2 + d);
            if ((rc = pt.beaver(prep, t_used, L)) != B200_OK) return rc;
            std::swap(x, x2);
        }
        // z(w^0) = 1, z(w^(j+1)) = prod_{i<=j} ratio_i
        B200_CUDA(cudaMemsetAsync(zpoly, 0, S * sizeof(fe), st));
        if (p0) B200_CUDA(cudaMemcpyAsync(zpoly, &one, sizeof(fe), cudaMemcpyHostToDevice, st));
        B200_CUDA(cudaMemcpyAsync(zpoly + 1, x, (n - 1) * sizeof(fe), cudaMemcpyDeviceToDevice, st));
        if ((rc = ntt_device(dn, zpoly, nscr, 1, 0, 1, S, st)) != B200_OK) return rc;
        BlindArgs b{};
        b.count = 3;
        b.dyn = d_bl + 10;
        B200_LAUNCH(k_blind, 1, 32, 0, st)(zpoly, n, b);
        if (au) {  // the MAC plane of z(w^0) = 1 is the key share on every party
            B200_CUDA(cudaMemsetAsync(M(zpoly), 0, S * sizeof(fe), st));
            B200_CUDA(cudaMemcpyAsync(M(zpoly), &au->key, sizeof(fe), cudaMemcpyHostToDevice, st));
            B200_CUDA(cudaMemcpyAsync(M(zpoly) + 1, M(x), (n - 1) * sizeof(fe), cudaMemcpyDeviceToDevice, st));
            if ((rc = ntt_device(dn, M(zpoly), nscr, 1, 0, 1, S, st)) != B200_OK) return rc;
            b.dyn = M(d_bl) + 10;
            B200_LAUNCH(k_blind, 1, 32, 0, st)(M(zpoly), n, b);
        }
        B200_CUDA(cudaStreamSynchronize(st));  // the host-to-device copy of `one` above reads a stack value
    }
    if ((rc = pt.open_commitments(pk->srs, zpoly, n + 3, n + 3, 1, &proof->prod_perm_poly_comm)) != B200_OK) return rc;
    tr.append_commitment(proof->prod_perm_poly_comm);

    // ---- round 3 ------------------------------------------------------------------------------------------------
    const fe alpha = tr.get_and_append_challenge();
    if (t_used != LY.r3) {
        set_error("collaborative prover: triple schedule out of step");
        return B200_ERR_INVALID;
    }
    if ((rc = coset_evals(pk, dn, zpoly, S, n + 3, 1, ext + 6 * m, nscr, st)) != B200_OK) return rc;
    B200_LAUNCH(k_next_on_coset, grid_for(m, 256), 256, 0, st)(ext + 6 * m, m, log_n, zw);
    if (au) {
        if ((rc = coset_evals(pk, dn, M(zpoly), S, n + 3, 1, M(ext) + 6 * m, nscr, st)) != B200_OK) return rc;
        B200_LAUNCH(k_next_on_coset, grid_for(m, 256), 256, 0, st)(M(ext) + 6 * m, m, log_n, M(zw));
        B200_LAUNCH(k_auth_perm_factors, grid_for(m, 128), 128, 0, st)(ext, M(ext), m, pk->coset_pts, pk->ce_sig, m, pk->k, beta, gamma,
                                                                       p0 ? 1 : 0, au->key, nf, df, M(nf), M(df));
    } else {
        B200_LAUNCH(k_mpc_perm_factors, grid_for(m, 128), 128, 0, st)(ext, m, pk->coset_pts, pk->ce_sig, m, pk->k, beta, gamma, p0 ? 1 : 0, nf, df);
    }
    {
        auto P3 = [&](int k) { return pr + (size_t)k * m; };
        auto W = [&](int j) { return ext + (size_t)j * m; };
        auto NF = [&](int j) { return nf + (size_t)j * m; };
        auto DF = [&](int j) { return df + (size_t)j * m; };
        // level 1 -> P3(0..9): w01 w23 w0^2..w3^2 n01 n23 d01 d23
        BeaverLevel L = level(m);
        add(L, W(0), W(1), P3(0));
        add(L, W(2), W(3), P3(1));
        for (int j = 0; j < 4; ++j) add(L, W(j), nullptr, P3(2 + j));
        add(L, NF(0), NF(1), P3(6));
        add(L, NF(2), NF(3), P3(7));
        add(L, DF(0), DF(1), P3(8));
        add(L, DF(2), DF(3), P3(9));
        if ((rc = pt.beaver(prep, t_used, L)) != B200_OK) return rc;
        // level 2 -> P3(10..16): w0123, w_j^4, n0123, d0123
        L = level(m);
        add(L, P3(0), P3(1), P3(10));
        for (int j = 0; j < 4; ++j) add(L, P3(2 + j), nullptr, P3(11 + j));
        add(L, P3(6), P3(7), P3(15));
        add(L, P3(8), P3(9), P3(16));
        if ((rc = pt.beaver(prep, t_used, L)) != B200_OK) return rc;
        // level 3 -> P3(17..23): w01234, w_j^5, num, den
        L = level(m);
        add(L, P3(10), W(4), P3(17));
        for (int j = 0; j < 4; ++j) add(L, P3(11 + j), W(j), P3(18 + j));
        add(L, P3(15), NF(4), P3(22));
        add(L, P3(16), DF(4), P3(23));
        if ((rc = pt.beaver(prep, t_used, L)) != B200_OK) return rc;
        // level 4 -> P3(24, 25): z num, z(wx) den
        L = level(m);
        add(L, W(6), P3(22), P3(24));
        add(L, zw, P3(23), P3(25));
        if ((rc = pt.beaver(prep, t_used, L)) != B200_OK) return rc;
        MpcQuotArgs q;
        q.sel = pk->ce_sel;
        q.ext = ext;
        q.w01 = P3(0);
        q.w23 = P3(1);
        q.w01234 = P3(17);
        q.p5 = P3(18);
        q.zn = P3(24);
        q.zd = P3(25);
        q.l1_inv = pk->l1_inv;
        q.out = quot;
        q.m = m;
        q.log_n = log_n;
        q.party0 = p0 ? 1 : 0;
        q.alpha = alpha;
        q.alpha2 = fe_sqr<Fr>(alpha);
        for (int i = 0; i < 8; ++i) q.zh_inv[i] = pk->zh_inv[i];
        if (au) {
            const QuotPlane qm{M(ext), M(P3(0)), M(P3(1)), M(P3(17)), M(P3(18)), M(P3(24)), M(P3(25)), M(quot)};
            B200_LAUNCH(k_auth_quotient, grid_for(m, 128), 128, 0, st)(q, qm, au->key);
        } else {
            B200_LAUNCH(k_mpc_quotient, grid_for(m, 128), 128, 0, st)(q);
        }
        for (fe* qq : {quot, au ? M(quot) : nullptr}) {
            if (!qq) continue;
            if ((rc = ntt_device(dn, qq, nscr, 1, 0, (unsigned)pk->nc, n, st)) != B200_OK) return rc;
            if (pk->nc == 6) B200_LAUNCH(k_coset_combine<6>, grid_for(n, 128), 128, 0, st)(qq, n, pk->cscale_inv, pk->comb);
            else B200_LAUNCH(k_coset_combine<8>, grid_for(n, 128), 128, 0, st)(qq, n, pk->cscale_inv, pk->comb);
        }
    }
    // degree check: the coefficients above deg are opened (zero for a satisfied witness) with the Beaver differences
    // of r' q[deg]; then r' q[deg] is opened (non-zero iff q[deg] is)
    const size_t deg = NW * (n + 1) + 2;
    bool unsat = false;
    {
        fe* rq = evals + 40;
        const size_t tail = m - deg - 1;
        std::vector<fe> tail_sum(tail);
        BeaverLevel L = level(1);
        add(L, quot + deg, prep->mask + n, rq);
        if ((rc = pt.beaver(prep, t_used, L, quot + deg + 1, tail, tail_sum.data())) != B200_OK) return rc;
        fe rq_h, rq_open;
        B200_CUDA(cudaMemcpy(&rq_h, rq, sizeof(fe), cudaMemcpyDeviceToHost));
        if ((rc = pt.open_host(&rq_h, 1, &rq_open)) != B200_OK) return rc;
        if (au && (rc = au->record(M(rq), &rq_open, 1, st)) != B200_OK) return rc;
        bool bad = fe_is_zero(rq_open);
        for (const fe& v : tail_sum) bad = bad || !fe_is_zero(v);
        if (bad) {
            set_error("WrongQuotientPolyDegree: the joint witness does not satisfy the circuit");
            if (!au) return B200_ERR_UNSATISFIED;
            unsat = true;  // reported only after the MAC check passed; rounds 4 and 5 are skipped
        }
    }
    // the rest of the proof: the quotient commitments, round 4 and round 5
    auto rounds45 = [&]() -> int {
        if (t_used != LY.triples) {
            set_error("collaborative prover: triple schedule out of step");
            return B200_ERR_INVALID;
        }
        B200_LAUNCH(k_split_quotient, dim3(grid_for(n + 3, 256), NW), 256, 0, st)(quot, n, S, d_bl + 13, split);
        if (au) B200_LAUNCH(k_split_quotient, dim3(grid_for(n + 3, 256), NW), 256, 0, st)(M(quot), n, S, M(d_bl) + 13, M(split));
        if ((rc = pt.open_commitments(pk->srs, split, n + 3, S, NW, proof->split_quot_poly_comms)) != B200_OK) return rc;
        for (int i = 0; i < NW; ++i) tr.append_commitment(proof->split_quot_poly_comms[i]);

        // ---- round 4 ------------------------------------------------------------------------------------------------
        const fe zeta = tr.get_and_append_challenge();
        const fe zeta_w = FMUL(zeta, pk->group_gen);
        {
            const fe* polys[kMaxEval];
            size_t lens[kMaxEval];
            fe pts[kMaxEval];
            for (int i = 0; i < NW; ++i) { polys[i] = wpoly + (size_t)i * S; lens[i] = n + 2; pts[i] = zeta; }
            for (int i = 0; i < NW - 1; ++i) { polys[NW + i] = pk->sig_coeffs + (size_t)i * n; lens[NW + i] = n; pts[NW + i] = zeta; }
            polys[2 * NW - 1] = zpoly; lens[2 * NW - 1] = n + 3; pts[2 * NW - 1] = zeta_w;
            eval_batch(polys, lens, pts, 2 * NW, evals, escr, st);
            fe h[2 * NW], mine[NW + 1], opened[NW + 1];
            B200_CUDA(cudaMemcpyAsync(h, evals, sizeof(h), cudaMemcpyDeviceToHost, st));
            B200_CUDA(cudaStreamSynchronize(st));
            for (int i = 0; i < NW; ++i) mine[i] = h[i];
            mine[NW] = h[2 * NW - 1];
            if ((rc = pt.open_host(mine, NW + 1, opened)) != B200_OK) return rc;
            if (au) {  // the MAC shares of the six opened evaluations, at M(evals)[0..5]
                const fe* mp[NW + 1];
                size_t ml[NW + 1];
                fe mz[NW + 1];
                for (int i = 0; i < NW; ++i) { mp[i] = M(wpoly) + (size_t)i * S; ml[i] = n + 2; mz[i] = zeta; }
                mp[NW] = M(zpoly); ml[NW] = n + 3; mz[NW] = zeta_w;
                eval_batch(mp, ml, mz, NW + 1, M(evals), M(escr), st);
                if ((rc = au->record(M(evals), opened, NW + 1, st)) != B200_OK) return rc;
            }
            for (int i = 0; i < NW; ++i) proof->wires_evals[i] = opened[i];
            for (int i = 0; i < NW - 1; ++i) proof->wire_sigma_evals[i] = h[NW + i];  // public polynomials
            proof->perm_next_eval = opened[NW];
        }
        for (int i = 0; i < NW; ++i) tr.append_field_elem(proof->wires_evals[i]);
        for (int i = 0; i < NW - 1; ++i) tr.append_field_elem(proof->wire_sigma_evals[i]);
        tr.append_field_elem(proof->perm_next_eval);

        // ---- round 5 ------------------------------------------------------------------------------------------------
        const fe v = tr.get_and_append_challenge();
        {
            LinArgs la{}, lm{};  // share plane; MAC plane (public polynomials weighted by the key share)
            const fe* we = proof->wires_evals;
            const fe* se = proof->wire_sigma_evals;
            int t = 0, tm = 0;
            auto push_to = [](LinArgs& a, int& k, const fe* poly, size_t len, const fe& s) {
                a.p[k] = poly;
                a.len[k] = (uint32_t)len;
                a.s[k] = s;
                ++k;
            };
            auto push = [&](const fe* poly, size_t len, const fe& s) {
                push_to(la, t, poly, len, s);
                if (au) push_to(lm, tm, au->mac(poly), len, s);
            };
            auto pub = [&](const fe* poly, size_t len, const fe& s) {
                if (p0) push_to(la, t, poly, len, s);
                if (au) push_to(lm, tm, poly, len, FMUL(au->key, s));
            };
            auto pow5 = [&](const fe& x) { return FMUL(fe_sqr<Fr>(fe_sqr<Fr>(x)), x); };
            const fe* sel = pk->sel_coeffs;
            const fe vanish = FSUB(host_pow(zeta, n), one);
            if (p0 || au) {  // the public part of the linearisation
                for (int j = 0; j < 4; ++j) pub(sel + (size_t)j * n, n, we[j]);
                pub(sel + 4 * n, n, FMUL(we[0], we[1]));
                pub(sel + 5 * n, n, FMUL(we[2], we[3]));
                for (int j = 0; j < 4; ++j) pub(sel + (size_t)(6 + j) * n, n, pow5(we[j]));
                pub(sel + 10 * n, n, fe_neg<Fr>(we[4]));
                pub(sel + 11 * n, n, one);
                pub(sel + 12 * n, n, FMUL(FMUL(FMUL(we[0], we[1]), FMUL(we[2], we[3])), we[4]));
                fe cs = FMUL(FMUL(alpha, beta), proof->perm_next_eval);
                for (int j = 0; j < NW - 1; ++j) cs = FMUL(cs, FADD(FADD(we[j], FMUL(beta, se[j])), gamma));
                pub(pk->sig_coeffs + (size_t)(NW - 1) * n, n, fe_neg<Fr>(cs));
                fe cv = one;
                for (int i = 0; i < 2 * NW - 1; ++i) {
                    cv = FMUL(cv, v);
                    if (i >= NW) pub(pk->sig_coeffs + (size_t)(i - NW) * n, n, cv);
                }
            }
            const fe l1 = FMUL(vanish, fe_inv<Fr>(FMUL(host_from_u64(n), FSUB(zeta, one))));
            fe cz = alpha;
            for (int j = 0; j < NW; ++j) cz = FMUL(cz, FADD(FADD(we[j], FMUL(FMUL(pk->k.v[j], zeta), beta)), gamma));
            cz = FADD(cz, FMUL(fe_sqr<Fr>(alpha), l1));
            push(zpoly, n + 3, cz);
            const fe zn2 = FMUL(FMUL(FADD(vanish, one), zeta), zeta);
            fe ct = fe_neg<Fr>(vanish);
            for (int i = 0; i < NW; ++i) {
                push(split + (size_t)i * S, i < NW - 1 ? n + 3 : n, ct);
                ct = FMUL(ct, zn2);
            }
            fe cv = one;
            for (int i = 0; i < NW; ++i) {
                cv = FMUL(cv, v);
                push(wpoly + (size_t)i * S, n + 2, cv);
            }
            la.count = t;
            la.dyn = nullptr;
            B200_LAUNCH(k_lincomb, grid_for(n + 3, 128), 128, 0, st)(la, n + 3, lin);
            horner_suffix(lin, n + 3, zeta, sdiv, evals + 16, hscr, st);
            horner_suffix(zpoly, n + 3, zeta_w, sdiv + (S + 8), evals + 17, hscr, st);
            if (au) {
                lm.count = tm;
                lm.dyn = nullptr;
                B200_LAUNCH(k_lincomb, grid_for(n + 3, 128), 128, 0, st)(lm, n + 3, M(lin));
                horner_suffix(M(lin), n + 3, zeta, M(sdiv), M(evals) + 16, M(hscr), st);
                horner_suffix(M(zpoly), n + 3, zeta_w, M(sdiv) + (S + 8), M(evals) + 17, M(hscr), st);
            }
        }
        g1_affine open2[2];
        if ((rc = pt.open_commitments(pk->srs, sdiv + 1, n + 2, S + 8, 2, open2)) != B200_OK) return rc;
        proof->opening_proof = open2[0];
        proof->shifted_opening_proof = open2[1];
        if (h_challenges) {
            tr.append_commitment(proof->opening_proof);
            tr.append_commitment(proof->shifted_opening_proof);
            const fe u = tr.get_and_append_challenge();
            const fe all[6] = {beta, gamma, alpha, zeta, v, u};
            std::memcpy(h_challenges, all, sizeof(all));
        }
        return B200_OK;
    };
    if (!unsat && (rc = rounds45()) != B200_OK) return rc;
    if (au) {
        bool ok = false;
        if ((rc = pt.auth_check(pk->srs, M(lin), lscr_p, &ok)) != B200_OK) return rc;
        if (!ok) {
            set_error("collaborative prover: the MAC check failed or malformed data was received (a party deviated); nothing "
                      "opened in this call may be used");
            return B200_ERR_MAC;
        }
        if (unsat) {
            set_error("WrongQuotientPolyDegree: the joint witness does not satisfy the circuit");
            return B200_ERR_UNSATISFIED;
        }
    }
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

// link() of plonk.cu on shares: everything is linear in the hints
// authenticated (pt.au set): h_a1m / h_a2m are the MAC shares of the hints, and the call ends with the MAC check
static int mpc_link(Party& pt, const Bases* srs, const fe* h_a1, size_t len1, const fe* h_a2, size_t len2, const g1_affine& comm1,
                    const g1_affine& comm2, unsigned alignment, size_t offset, size_t size, LinkOut* out, fe* h_eta,
                    const fe* h_a1m = nullptr, const fe* h_a2m = nullptr) {
    Context* c = pt.c;
    cudaStream_t st = pt.st;
    const size_t len = len1 > len2 ? len1 : len2;
    unsigned log_N = 1;
    while (((size_t)1 << log_N) < len) ++log_N;
    const size_t N = (size_t)1 << log_N;
    const size_t L = len + 8, NL = N + 8;
    const size_t scr = 4 * (L / CH + 4 * CH + 64);
    int rc;
    Auth* au = pt.au;
    const size_t total = 5 * L + 3 * NL + scr + size + 16;
    // authenticated: the MAC plane, the gamma log (the tail and the evaluation), staging and the log's evaluation scratch
    const size_t log_cap = N + 8, lscr = log_cap / CH + log_cap / CH / CH + 2 * CH + 16;
    const size_t auth_total = au ? total + 2 * log_cap + lscr + 1 : 0;
    if ((rc = c->mpc_ws.reserve((total + auth_total) * sizeof(fe))) != B200_OK) return rc;
    if ((rc = c->ntt_scratch.reserve(N * sizeof(fe))) != B200_OK) return rc;
    Domain* dN = nullptr;
    if ((rc = get_domain(c, log_N, &dN)) != B200_OK) return rc;
    fe* base = reinterpret_cast<fe*>(c->mpc_ws.p);
    fe* lscr_p = nullptr;
    if (au) {
        au->ws = base;
        au->total = total;
        au->log = base + 2 * total;
        au->log_cap = log_cap;
        au->stage = au->log + log_cap;
        au->stage_cap = log_cap;
        lscr_p = au->stage + log_cap;
        au->bad = reinterpret_cast<int*>(lscr_p + lscr);
        B200_CUDA(cudaMemsetAsync(au->bad, 0, sizeof(int), st));
    }
    auto M = [&](const fe* x) { return au->mac(const_cast<fe*>(x)); };
    fe *d_a1 = base, *d_a2 = base + L, *d_diff = base + 2 * L, *d_ident = base + 3 * L, *d_open = base + 4 * L;
    fe *d_E = base + 5 * L, *d_Z = d_E + NL, *d_Q = d_Z + NL;
    fe* hscr = d_Q + NL;
    fe* d_roots = hscr + scr;
    fe* slot = d_roots + size;
    fe* nscr = reinterpret_cast<fe*>(c->ntt_scratch.p);
    B200_CUDA(cudaMemcpyAsync(d_a1, h_a1, len1 * sizeof(fe), cudaMemcpyDefault, st));
    B200_CUDA(cudaMemcpyAsync(d_a2, h_a2, len2 * sizeof(fe), cudaMemcpyDefault, st));
    const fe one = fe_one<Fr>();
    const fe g = host_root_of_unity(alignment);
    std::vector<fe> roots(size);
    fe root = host_pow(g, (uint64_t)offset);
    const fe root0 = root;
    for (size_t i = 0; i < size; ++i) {
        roots[i] = root;
        root = FMUL(root, g);
    }
    {
        LinArgs a{};
        a.count = 2;
        a.p[0] = d_a1; a.len[0] = (uint32_t)len1; a.s[0] = one;
        a.p[1] = d_a2; a.len[1] = (uint32_t)len2; a.s[1] = fe_neg<Fr>(one);
        B200_LAUNCH(k_lincomb, grid_for(len, 128), 128, 0, st)(a, len, d_diff);
        if (au) {
            B200_CUDA(cudaMemcpyAsync(M(d_a1), h_a1m, len1 * sizeof(fe), cudaMemcpyDefault, st));
            B200_CUDA(cudaMemcpyAsync(M(d_a2), h_a2m, len2 * sizeof(fe), cudaMemcpyDefault, st));
            a.p[0] = M(d_a1);
            a.p[1] = M(d_a2);
            B200_LAUNCH(k_lincomb, grid_for(len, 128), 128, 0, st)(a, len, M(d_diff));
        }
    }
    fill_powers(d_roots, size, g, root0, st);
    B200_CUDA(cudaMemsetAsync(d_E, 0, N * sizeof(fe), st));
    B200_CUDA(cudaMemcpyAsync(d_E, d_diff, len * sizeof(fe), cudaMemcpyDeviceToDevice, st));
    if ((rc = ntt_device(dN, d_E, nscr, 0, 1, 1, N, st)) != B200_OK) return rc;
    B200_LAUNCH(k_vanishing_on_coset, grid_for(N, 128), 128, 0, st)(dN->tw_fwd, N, fe_from_u32<Fr>(5), d_roots, size, d_Z);
    if (au) {  // the same division on the MAC plane
        B200_CUDA(cudaMemsetAsync(M(d_E), 0, N * sizeof(fe), st));
        B200_CUDA(cudaMemcpyAsync(M(d_E), M(d_diff), len * sizeof(fe), cudaMemcpyDeviceToDevice, st));
        if ((rc = ntt_device(dN, M(d_E), nscr, 0, 1, 1, N, st)) != B200_OK) return rc;
        B200_CUDA(cudaMemcpyAsync(M(d_Z), d_Z, N * sizeof(fe), cudaMemcpyDeviceToDevice, st));
        batch_inverse_enqueue(M(d_E), M(d_Z), M(d_Q), N, st);
        if ((rc = ntt_device(dN, M(d_Z), nscr, 1, 1, 1, N, st)) != B200_OK) return rc;
    }
    batch_inverse_enqueue(d_E, d_Z, d_Q, N, st);  // d_Z <- diff / Z_D on the coset
    if ((rc = ntt_device(dN, d_Z, nscr, 1, 1, 1, N, st)) != B200_OK) return rc;
    const size_t q_len = len - size;
    bool unsat = false;
    // exactness: the interpolant's coefficients from q_len on are opened (zero when the hints agree on the group),
    // together with the partial quotient commitment
    {
        g1_affine part;
        rc = commit_partials(c, srs, d_Z, q_len, q_len, 1, &part, st);
        if (rc != B200_OK) return rc;
        // authenticated: the commitment H(seed_i) to this party's check seed follows the partial commitment
        const size_t hx = au ? 32 : 0, tail = N - q_len, payload = 64 + hx + tail * sizeof(fe);
        if ((rc = pt.reserve(payload)) != B200_OK) return rc;
        std::memcpy(pt.send + kHdr, &part, 64);
        if (au) keccak(au->seed, 32, pt.send + kHdr + 64);
        B200_CUDA(cudaMemcpyAsync(pt.send + kHdr + 64 + hx, d_Z + q_len, tail * sizeof(fe), cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        if ((rc = pt.exchange_now(payload)) != B200_OK) return rc;
        std::vector<fe> t(tail);
        pt.sum_fe(64 + hx, tail, t.data());
        for (const fe& x : t)
            if (!fe_is_zero(x)) {
                set_error("link: the two wire polynomials differ on the link group (wrong layout or mismatched witnesses)");
                if (!au) return B200_ERR_UNSATISFIED;
                unsat = true;  // reported only after the MAC check passed
                break;
            }
        if ((rc = pt.sum_points(0, 1, &out->quotient_commitment)) != B200_OK) return rc;
        if (au) {
            au->seed_comms.resize((size_t)pt.P * 32);
            for (int q = 0; q < pt.P; ++q) std::memcpy(&au->seed_comms[(size_t)q * 32], pt.payload_of(q) + 64, 32);
            au->polys.push_back(M(d_Z));
            au->lens.push_back(q_len);
            au->comms.push_back(out->quotient_commitment);
            if ((rc = au->record(M(d_Z) + q_len, t.data(), tail, st)) != B200_OK) return rc;
        }
    }
    // the opening and its exchange (skipped in authenticated mode when the exactness check failed)
    auto opening = [&]() -> int {
        SolidityTranscript tr;
        tr.append_commitment(comm1);
        tr.append_commitment(comm2);
        tr.append_commitment(out->quotient_commitment);
        const fe eta = tr.get_and_append_challenge();
        if (h_eta) *h_eta = eta;
        fe zd = one;
        for (size_t i = 0; i < size; ++i) zd = FMUL(zd, FSUB(eta, roots[i]));
        {
            LinArgs a{};
            a.count = 2;
            a.p[0] = d_diff; a.len[0] = (uint32_t)len; a.s[0] = one;
            a.p[1] = d_Z; a.len[1] = (uint32_t)q_len; a.s[1] = fe_neg<Fr>(zd);
            B200_LAUNCH(k_lincomb, grid_for(len, 128), 128, 0, st)(a, len, d_ident);
            horner_suffix(d_ident, len, eta, d_open, slot, hscr, st);
            if (au) {
                a.p[0] = M(d_diff);
                a.p[1] = M(d_Z);
                B200_LAUNCH(k_lincomb, grid_for(len, 128), 128, 0, st)(a, len, M(d_ident));
                horner_suffix(M(d_ident), len, eta, M(d_open), M(slot), M(hscr), st);
            }
        }
        // the opening: the evaluation (zero for an exact division) and the partial opening commitment
        g1_affine part;
        rc = commit_partials(c, srs, d_open + 1, len - 1, len - 1, 1, &part, st);
        if (rc != B200_OK) return rc;
        if ((rc = pt.reserve(96)) != B200_OK) return rc;
        std::memcpy(pt.send + kHdr, &part, 64);
        B200_CUDA(cudaMemcpy(pt.send + kHdr + 64, d_open, sizeof(fe), cudaMemcpyDeviceToHost));
        if ((rc = pt.exchange_now(96)) != B200_OK) return rc;
        fe ev;
        pt.sum_fe(64, 1, &ev);
        if (!fe_is_zero(ev)) {
            set_error("link: the opened evaluation is not zero");
            if (!au) return B200_ERR_UNSATISFIED;
            unsat = true;
        }
        if ((rc = pt.sum_points(0, 1, &out->opening_proof)) != B200_OK) return rc;
        if (au) {
            au->polys.push_back(M(d_open) + 1);
            au->lens.push_back(len - 1);
            au->comms.push_back(out->opening_proof);
            if ((rc = au->record(M(d_open), &ev, 1, st)) != B200_OK) return rc;
        }
        return B200_OK;
    };
    if (!unsat && (rc = opening()) != B200_OK) return rc;
    if (au) {
        bool ok = false;
        if ((rc = pt.auth_check(srs, M(d_E), lscr_p, &ok)) != B200_OK) return rc;
        if (!ok) {
            set_error("link: the MAC check failed or malformed data was received (a party deviated); nothing opened in this call "
                      "may be used");
            return B200_ERR_MAC;
        }
        if (unsat) return B200_ERR_UNSATISFIED;  // the message of the failed exactness check stands
    }
    return B200_OK;
}

static bool transport_ok(const b200_mpc_transport* t) {
    return t && t->all_gather && t->parties >= 2 && t->party >= 0 && t->party < t->parties;
}

}  // namespace b200

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
using namespace b200;

struct b200_mpc_prep {
    MpcPrep p;
};
struct b200_mpc_local_group {
    LocalGroup g;
};

extern "C" {

int b200_mpc_prep_size(const b200_pk* pk, size_t* n_triples, size_t* n_masks) {
    if (!pk || !n_triples || !n_masks) return B200_ERR_INVALID;
    const MpcLayout L = mpc_layout(pk->pk);
    *n_triples = L.triples;
    *n_masks = L.masks;
    return B200_OK;
}

int b200_mpc_prep_load(b200_ctx* ctx, const b200_pk* pk, const uint64_t* a, const uint64_t* b, const uint64_t* c,
                       const uint64_t* masks, b200_mpc_prep** out) {
    B200_TRY
    if (!ctx || !pk || !a || !b || !c || !masks || !out) return B200_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    MpcPrep* p = nullptr;
    int rc = prep_alloc(&ctx->c, pk->pk, &p);
    if (rc != B200_OK) return rc;
    p->pk_id = pk->pk->id;
    const size_t tb = p->triples * sizeof(fe);
    cudaStream_t st = ctx->c.stream;
    if (cudaMemcpyAsync(p->a, a, tb, cudaMemcpyDefault, st) != cudaSuccess || cudaMemcpyAsync(p->b, b, tb, cudaMemcpyDefault, st) != cudaSuccess ||
        cudaMemcpyAsync(p->c, c, tb, cudaMemcpyDefault, st) != cudaSuccess ||
        cudaMemcpyAsync(p->mask, masks, p->masks * sizeof(fe), cudaMemcpyDefault, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
        delete p;
        return cuda_fail(cudaGetLastError(), "b200_mpc_prep_load");
    }
    *out = reinterpret_cast<b200_mpc_prep*>(p);
    return B200_OK;
    B200_CATCH
}

int b200_mpc_prep_dealer(b200_ctx* ctx, const b200_pk* pk, uint64_t seed, int party, int parties, b200_mpc_prep** out) {
    B200_TRY
    if (!ctx || !pk || !out || parties < 2 || party < 0 || party >= parties) return B200_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    MpcPrep* p = nullptr;
    int rc = prep_alloc(&ctx->c, pk->pk, &p);
    if (rc != B200_OK) return rc;
    p->pk_id = pk->pk->id;
    const MpcLayout L = mpc_layout(pk->pk);
    cudaStream_t st = ctx->c.stream;
    B200_LAUNCH(k_dealer, grid_for(p->triples, 256), 256, 0, st)(seed, party, parties, p->triples, 0, L.sq, p->a, p->b, p->c);
    B200_LAUNCH(k_dealer, grid_for(p->masks, 256), 256, 0, st)(seed, party, parties, p->masks, 1, L.sq, p->mask, nullptr, nullptr);
    if (cudaStreamSynchronize(st) != cudaSuccess) {
        delete p;
        return cuda_fail(cudaGetLastError(), "b200_mpc_prep_dealer");
    }
    *out = reinterpret_cast<b200_mpc_prep*>(p);
    return B200_OK;
    B200_CATCH
}

int b200_mpc_prep_load_auth(b200_ctx* ctx, const b200_pk* pk, const uint64_t* a, const uint64_t* b, const uint64_t* c,
                            const uint64_t* a_mac, const uint64_t* b_mac, const uint64_t* c_mac, const uint64_t* masks,
                            const uint64_t* masks_mac, b200_mpc_prep** out) {
    B200_TRY
    if (!ctx || !pk || !a || !b || !c || !a_mac || !b_mac || !c_mac || !masks || !masks_mac || !out) return B200_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    MpcPrep* p = nullptr;
    int rc = prep_alloc(&ctx->c, pk->pk, &p, /*auth=*/true);
    if (rc != B200_OK) return rc;
    p->pk_id = pk->pk->id;
    const size_t tb = p->triples * sizeof(fe), mb = p->masks * sizeof(fe);
    cudaStream_t st = ctx->c.stream;
    const std::pair<fe*, const uint64_t*> copies[8] = {{p->a, a}, {p->b, b}, {p->c, c}, {p->am, a_mac}, {p->bm, b_mac}, {p->cm, c_mac},
                                                       {p->mask, masks}, {p->mask_mac, masks_mac}};
    bool fine = true;
    for (int i = 0; i < 8; ++i) fine = fine && cudaMemcpyAsync(copies[i].first, copies[i].second, i < 6 ? tb : mb, cudaMemcpyDefault, st) == cudaSuccess;
    if (!fine || cudaStreamSynchronize(st) != cudaSuccess) {
        delete p;
        return cuda_fail(cudaGetLastError(), "b200_mpc_prep_load_auth");
    }
    *out = reinterpret_cast<b200_mpc_prep*>(p);
    return B200_OK;
    B200_CATCH
}

int b200_mpc_prep_dealer_auth(b200_ctx* ctx, const b200_pk* pk, uint64_t seed, int party, int parties, uint64_t mac_key_share[4],
                              b200_mpc_prep** out) {
    B200_TRY
    if (!ctx || !pk || !mac_key_share || !out || parties < 2 || party < 0 || party >= parties) return B200_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    MpcPrep* p = nullptr;
    int rc = prep_alloc(&ctx->c, pk->pk, &p, /*auth=*/true);
    if (rc != B200_OK) return rc;
    p->pk_id = pk->pk->id;
    const MpcLayout L = mpc_layout(pk->pk);
    cudaStream_t st = ctx->c.stream;
    fe* d_key = nullptr;
    if ((rc = alloc_fe(&d_key, 1)) != B200_OK) {
        delete p;
        return rc;
    }
    B200_LAUNCH(k_dealer, grid_for(p->triples, 256), 256, 0, st)(seed, party, parties, p->triples, 0, L.sq, p->a, p->b, p->c);
    B200_LAUNCH(k_dealer, grid_for(p->masks, 256), 256, 0, st)(seed, party, parties, p->masks, 1, L.sq, p->mask, nullptr, nullptr);
    B200_LAUNCH(k_dealer_mac, grid_for(p->triples, 256), 256, 0, st)(seed, party, parties, p->triples, 0, L.sq, p->am, p->bm, p->cm, d_key);
    B200_LAUNCH(k_dealer_mac, grid_for(p->masks, 256), 256, 0, st)(seed, party, parties, p->masks, 1, L.sq, p->mask_mac, nullptr, nullptr,
                                                                   nullptr);
    if (cudaStreamSynchronize(st) != cudaSuccess || cudaMemcpy(mac_key_share, d_key, sizeof(fe), cudaMemcpyDeviceToHost) != cudaSuccess) {
        cudaFree(d_key);
        delete p;
        return cuda_fail(cudaGetLastError(), "b200_mpc_prep_dealer_auth");
    }
    cudaFree(d_key);
    *out = reinterpret_cast<b200_mpc_prep*>(p);
    return B200_OK;
    B200_CATCH
}

int b200_mpc_dealer_share_auth(b200_ctx* ctx, uint64_t seed, int party, int parties, const uint64_t* values, size_t count,
                               uint64_t* shares, uint64_t* macs) {
    B200_TRY
    if (!ctx || !values || !shares || !macs || count == 0 || parties < 2 || party < 0 || party >= parties) return B200_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    int rc;
    if ((rc = ctx->c.mpc_ws.reserve(3 * count * sizeof(fe))) != B200_OK) return rc;
    fe* d = reinterpret_cast<fe*>(ctx->c.mpc_ws.p);
    cudaStream_t st = ctx->c.stream;
    B200_CUDA(cudaMemcpyAsync(d, values, count * sizeof(fe), cudaMemcpyDefault, st));
    B200_LAUNCH(k_dealer_input, grid_for(count, 256), 256, 0, st)(seed, party, parties, count, d, d + count, d + 2 * count);
    B200_CUDA(cudaMemcpyAsync(shares, d + count, count * sizeof(fe), cudaMemcpyDefault, st));
    B200_CUDA(cudaMemcpyAsync(macs, d + 2 * count, count * sizeof(fe), cudaMemcpyDefault, st));
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
    B200_CATCH
}

void b200_mpc_prep_free(b200_ctx* ctx, b200_mpc_prep* prep) {
    if (!prep) return;
    if (ctx) {
        std::lock_guard<std::mutex> lk(ctx->c.mu);
        cudaSetDevice(ctx->c.device);
        cudaStreamSynchronize(ctx->c.stream);
    }
    delete reinterpret_cast<MpcPrep*>(prep);
}

int b200_mpc_prove(b200_ctx* ctx, const b200_pk* pk, const b200_mpc_transport* transport, b200_mpc_prep* prep,
                   const uint64_t* wire_shares, const uint64_t* pub_inputs, const uint64_t* blinder_shares, b200_proof* proof,
                   uint64_t* link_poly_share, uint64_t* challenges) {
    B200_TRY
    if (!transport_ok(transport)) {
        set_error("b200_mpc_prove: bad transport (NULL, parties < 2 or party out of range)");
        return B200_ERR_INVALID;
    }
    auto refuse = [&](const char* why) {
        set_error(why);
        if (transport->abort) transport->abort(transport->user);
        return B200_ERR_INVALID;
    };
    if (!ctx || !pk || !prep || !wire_shares || !blinder_shares || !proof || (pk->pk->num_inputs && !pub_inputs))
        return refuse("b200_mpc_prove: NULL argument");
    MpcPrep* pp = reinterpret_cast<MpcPrep*>(prep);
    const MpcLayout L = mpc_layout(pk->pk);
    if (pp->n != L.n || pp->m != L.m || pp->triples != L.triples || pp->masks != L.masks || pp->device != ctx->c.device)
        return refuse("b200_mpc_prove: the preprocessing does not fit this key or device");
    if (pp->used) return refuse("b200_mpc_prove: this preprocessing was used already (Beaver triples are single-use)");
    if (pp->auth) return refuse("b200_mpc_prove: authenticated preprocessing belongs to b200_mpc_prove_auth");
    pp->used = true;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    Context* c = &ctx->c;
    for (double& s : c->mpc_stats) s = 0;
    int rc = cudaSetDevice(c->device) == cudaSuccess ? B200_OK : cuda_fail(cudaGetLastError(), "cudaSetDevice");
    Party pt{c, transport, transport->party, transport->parties, c->stream};
    if (rc == B200_OK)
        rc = mpc_prove(pt, pk->pk, pp, reinterpret_cast<const fe*>(wire_shares), reinterpret_cast<const fe*>(pub_inputs),
                       reinterpret_cast<const fe*>(blinder_shares), reinterpret_cast<ProofOut*>(proof),
                       reinterpret_cast<fe*>(link_poly_share), reinterpret_cast<fe*>(challenges));
    c->mpc_stats[0] = (double)pt.exchange;
    c->mpc_stats[1] = pt.bytes;
    c->mpc_stats[2] = pt.triples;
    c->mpc_stats[3] = pt.ms;
    if (rc != B200_OK) {
        cudaStreamSynchronize(c->stream);
        if (transport->abort) transport->abort(transport->user);
    }
    return rc;
    B200_CATCH
}

int b200_mpc_link(b200_ctx* ctx, const b200_bases* srs, const b200_mpc_transport* transport, const uint64_t* a1_share,
                  size_t len1, const uint64_t* a2_share, size_t len2, const uint64_t* comm1, const uint64_t* comm2,
                  unsigned alignment, size_t offset, size_t size, b200_link_proof* proof, uint64_t* eta) {
    B200_TRY
    if (!transport_ok(transport)) {
        set_error("b200_mpc_link: bad transport (NULL, parties < 2 or party out of range)");
        return B200_ERR_INVALID;
    }
    const size_t len = len1 > len2 ? len1 : len2;
    if (!ctx || !srs || !a1_share || !a2_share || !comm1 || !comm2 || !proof || size == 0 || size >= len || alignment > 28 ||
        len > srs->b->n || len > ((size_t)1 << 28)) {
        set_error("b200_mpc_link: bad argument, group layout or polynomial length");
        if (transport->abort) transport->abort(transport->user);
        return B200_ERR_INVALID;
    }
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    Context* c = &ctx->c;
    for (double& s : c->mpc_stats) s = 0;
    int rc = cudaSetDevice(c->device) == cudaSuccess ? B200_OK : cuda_fail(cudaGetLastError(), "cudaSetDevice");
    Party pt{c, transport, transport->party, transport->parties, c->stream};
    g1_affine c1, c2;
    std::memcpy(&c1, comm1, 64);
    std::memcpy(&c2, comm2, 64);
    if (rc == B200_OK)
        rc = mpc_link(pt, srs->b, reinterpret_cast<const fe*>(a1_share), len1, reinterpret_cast<const fe*>(a2_share), len2, c1, c2,
                      alignment, offset, size, reinterpret_cast<LinkOut*>(proof), reinterpret_cast<fe*>(eta));
    c->mpc_stats[0] = (double)pt.exchange;
    c->mpc_stats[1] = pt.bytes;
    c->mpc_stats[3] = pt.ms;
    if (rc != B200_OK) {
        cudaStreamSynchronize(c->stream);
        if (transport->abort) transport->abort(transport->user);
    }
    return rc;
    B200_CATCH
}

// a MAC-key share from the caller: a canonical Montgomery element
static bool key_share(const uint64_t* k, fe* out) {
    if (!k) return false;
    std::memcpy(out, k, sizeof(fe));
    return canonical<FrCfg>(*out);
}

int b200_mpc_prove_auth(b200_ctx* ctx, const b200_pk* pk, const b200_mpc_transport* transport, b200_mpc_prep* prep,
                        const uint64_t* mac_key_share, const uint64_t* wire_shares, const uint64_t* wire_macs,
                        const uint64_t* pub_inputs, const uint64_t* blinder_shares, const uint64_t* blinder_macs, b200_proof* proof,
                        uint64_t* link_poly_share, uint64_t* link_poly_mac, uint64_t* challenges) {
    B200_TRY
    if (!transport_ok(transport)) {
        set_error("b200_mpc_prove_auth: bad transport (NULL, parties < 2 or party out of range)");
        return B200_ERR_INVALID;
    }
    auto refuse = [&](const char* why) {
        set_error(why);
        if (transport->abort) transport->abort(transport->user);
        return B200_ERR_INVALID;
    };
    Auth au;
    if (!ctx || !pk || !prep || !wire_shares || !wire_macs || !blinder_shares || !blinder_macs || !proof ||
        (pk->pk->num_inputs && !pub_inputs) || !key_share(mac_key_share, &au.key))
        return refuse("b200_mpc_prove_auth: NULL argument or a MAC-key share that is not a canonical field element");
    MpcPrep* pp = reinterpret_cast<MpcPrep*>(prep);
    const MpcLayout L = mpc_layout(pk->pk);
    if (pp->n != L.n || pp->m != L.m || pp->triples != L.triples || pp->masks != L.masks || pp->device != ctx->c.device)
        return refuse("b200_mpc_prove_auth: the preprocessing does not fit this key or device");
    if (!pp->auth) return refuse("b200_mpc_prove_auth: the preprocessing has no MACs (made for b200_mpc_prove)");
    if (pp->used) return refuse("b200_mpc_prove_auth: this preprocessing was used already (Beaver triples are single-use)");
    if (draw_random(au.seed, 32) != B200_OK) return refuse("b200_mpc_prove_auth: getrandom failed");
    pp->used = true;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    Context* c = &ctx->c;
    for (double& s : c->mpc_stats) s = 0;
    int rc = cudaSetDevice(c->device) == cudaSuccess ? B200_OK : cuda_fail(cudaGetLastError(), "cudaSetDevice");
    Party pt{c, transport, transport->party, transport->parties, c->stream};
    pt.au = &au;
    // the outputs are written only after the MAC check passed
    ProofOut po;
    std::vector<fe> link(L.n + 2), link_mac(L.n + 2);
    fe ch[6];
    if (rc == B200_OK)
        rc = mpc_prove(pt, pk->pk, pp, reinterpret_cast<const fe*>(wire_shares), reinterpret_cast<const fe*>(pub_inputs),
                       reinterpret_cast<const fe*>(blinder_shares), &po, link.data(), ch, reinterpret_cast<const fe*>(wire_macs),
                       reinterpret_cast<const fe*>(blinder_macs), link_mac.data());
    c->mpc_stats[0] = (double)pt.exchange;
    c->mpc_stats[1] = pt.bytes;
    c->mpc_stats[2] = pt.triples;
    c->mpc_stats[3] = pt.ms;
    if (rc != B200_OK) {
        cudaStreamSynchronize(c->stream);
        if (transport->abort) transport->abort(transport->user);
        return rc;
    }
    std::memcpy(proof, &po, sizeof(po));
    if (link_poly_share) std::memcpy(link_poly_share, link.data(), link.size() * sizeof(fe));
    if (link_poly_mac) std::memcpy(link_poly_mac, link_mac.data(), link_mac.size() * sizeof(fe));
    if (challenges) std::memcpy(challenges, ch, sizeof(ch));
    return B200_OK;
    B200_CATCH
}

int b200_mpc_link_auth(b200_ctx* ctx, const b200_bases* srs, const b200_mpc_transport* transport, const uint64_t* mac_key_share,
                       const uint64_t* a1_share, const uint64_t* a1_mac, size_t len1, const uint64_t* a2_share, const uint64_t* a2_mac,
                       size_t len2, const uint64_t* comm1, const uint64_t* comm2, unsigned alignment, size_t offset, size_t size,
                       b200_link_proof* proof, uint64_t* eta) {
    B200_TRY
    if (!transport_ok(transport)) {
        set_error("b200_mpc_link_auth: bad transport (NULL, parties < 2 or party out of range)");
        return B200_ERR_INVALID;
    }
    const size_t len = len1 > len2 ? len1 : len2;
    Auth au;
    if (!ctx || !srs || !a1_share || !a1_mac || !a2_share || !a2_mac || !comm1 || !comm2 || !proof || size == 0 || size >= len ||
        alignment > 28 || len > srs->b->n || len > ((size_t)1 << 28) || !key_share(mac_key_share, &au.key) ||
        draw_random(au.seed, 32) != B200_OK) {
        set_error("b200_mpc_link_auth: bad argument, MAC-key share, group layout or polynomial length");
        if (transport->abort) transport->abort(transport->user);
        return B200_ERR_INVALID;
    }
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    Context* c = &ctx->c;
    for (double& s : c->mpc_stats) s = 0;
    int rc = cudaSetDevice(c->device) == cudaSuccess ? B200_OK : cuda_fail(cudaGetLastError(), "cudaSetDevice");
    Party pt{c, transport, transport->party, transport->parties, c->stream};
    pt.au = &au;
    g1_affine c1, c2;
    std::memcpy(&c1, comm1, 64);
    std::memcpy(&c2, comm2, 64);
    LinkOut lo;
    fe e;
    if (rc == B200_OK)
        rc = mpc_link(pt, srs->b, reinterpret_cast<const fe*>(a1_share), len1, reinterpret_cast<const fe*>(a2_share), len2, c1, c2,
                      alignment, offset, size, &lo, &e, reinterpret_cast<const fe*>(a1_mac), reinterpret_cast<const fe*>(a2_mac));
    c->mpc_stats[0] = (double)pt.exchange;
    c->mpc_stats[1] = pt.bytes;
    c->mpc_stats[3] = pt.ms;
    if (rc != B200_OK) {
        cudaStreamSynchronize(c->stream);
        if (transport->abort) transport->abort(transport->user);
        return rc;
    }
    std::memcpy(proof, &lo, sizeof(lo));
    if (eta) std::memcpy(eta, &e, sizeof(e));
    return B200_OK;
    B200_CATCH
}

int b200_mpc_local_group_create(int parties, unsigned timeout_ms, b200_mpc_local_group** out) {
    B200_TRY
    if (parties < 2 || !out || timeout_ms == 0) return B200_ERR_INVALID;
    b200_mpc_local_group* g = new b200_mpc_local_group();
    g->g.parties = parties;
    g->g.timeout_ms = timeout_ms;
    g->g.calls.assign(parties, 0);
    g->g.members.resize(parties);
    for (int p = 0; p < parties; ++p) g->g.members[p] = LocalMember{&g->g, p};
    *out = g;
    return B200_OK;
    B200_CATCH
}

int b200_mpc_local_group_transport(b200_mpc_local_group* group, int party, b200_mpc_transport* out) {
    if (!group || !out || party < 0 || party >= group->g.parties) return B200_ERR_INVALID;
    out->all_gather = local_all_gather;
    out->abort = local_abort;
    out->user = &group->g.members[party];
    out->party = party;
    out->parties = group->g.parties;
    return B200_OK;
}

void b200_mpc_local_group_destroy(b200_mpc_local_group* group) { delete group; }

int b200_mpc_last_stats(b200_ctx* ctx, double out[4]) {
    if (!ctx || !out) return B200_ERR_INVALID;
    for (int i = 0; i < 4; ++i) out[i] = ctx->c.mpc_stats[i];
    return B200_OK;
}

}  // extern "C"
