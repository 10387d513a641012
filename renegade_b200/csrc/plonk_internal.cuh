// Internal pieces of the TurboPlonk prover shared by plonk.cu (single prover) and mpc.cu (collaborative prover):
// the round kernels, the proving key, and the host helpers that enqueue them.  Nothing here is part of the public
// boundary.
#pragma once
#include <algorithm>
#include <chrono>
#include <cstring>
#include <vector>

#include "b200prover.h"
#include "device_ctx.h"

namespace b200 {

namespace {

constexpr int NW = 5;    // wire columns (GATE_WIDTH + 1)
constexpr int NS = 13;   // q_lc[4] q_mul[2] q_hash[4] q_o q_c q_ecc
constexpr int CH = 16;   // elements per thread in the chunked scans: every level is a chain of CH dependent products
                         // (latency-bound kernels), so short chunks and one more level beat long chunks

struct KArr {
    fe v[NW];
};

using Fr = FrCfg;
#define FMUL(a, b) fe_mul<Fr>((a), (b))
#define FADD(a, b) fe_add<Fr>((a), (b))
#define FSUB(a, b) fe_sub<Fr>((a), (b))

// ---- key setup ---------------------------------------------------------------------------------
// sigma_i(w^j) = k_{i'} * w^{j'} where (i', j') is the image of wire position (i, j)
__global__ void k_sigma_evals(const uint64_t* __restrict__ perm, const fe* __restrict__ dom, size_t n, KArr k,
                              fe* __restrict__ out) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= NW * n) return;
    const uint64_t tgt = perm[t];
    fe_store(out + t, FMUL(k.v[tgt / n], fe_load_ro(dom + tgt % n)));
}

// out[i] = n * (x_i - 1)   (inverted afterwards: L_1(x) / Z_H(x) = 1 / (n (x - 1)))
__global__ void k_l1_denominators(const fe* __restrict__ pts, size_t m, fe n_mont, fe* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    fe_store(out + i, FMUL(FSUB(fe_load_ro(pts + i), fe_one<Fr>()), n_mont));
}

// Batch inversion with ONE field inversion per block of 4096 elements (Montgomery's trick on two levels): every thread
// multiplies up its chunk of 16, the 256 chunk totals are scanned in shared memory (prefix and suffix products at once),
// thread 0 inverts the block total with the binary extended Euclid — a single lane, so its data-dependent branches have
// nobody to diverge from: ~20 us, against ~180 us for the 380 dependent products of a Fermat ladder (what a per-thread
// inversion costs whatever the batch size) — and the chunk inverses fan back out.  ~5 products per element.
// Measured against the alternatives on B200 (profiles/r2o_inverse_ab.log, round 2 of a 2^13 proof): Fermat per 16
// elements 0.68 ms, one-lane Fermat per block 0.65, block totals inverted on the host through a pinned mailbox and a host
// node 0.57, this 0.55.
// data[i] <- 1 / data[i], or num[i] / data[i] (RATIO); zeros stay zero and do not disturb their neighbours.
constexpr int kInvThreads = 256, kInvChunk = 16, kInvBlock = kInvThreads * kInvChunk;
template <bool RATIO>
__global__ void __launch_bounds__(kInvThreads) k_block_inverse(const fe* __restrict__ num, fe* __restrict__ data,
                                                               fe* __restrict__ scratch, size_t n) {
    __shared__ fe pre[kInvThreads], suf[kInvThreads];
    __shared__ fe binv;
    const unsigned t = threadIdx.x;
    const size_t beg = ((size_t)blockIdx.x * kInvThreads + t) * kInvChunk;
    const size_t end = beg + kInvChunk < n ? beg + kInvChunk : n;
    const fe one = fe_one<Fr>();
    fe run = one;
    for (size_t i = beg; i < end; ++i) {
        fe_store(scratch + i, run);
        const fe d = fe_load(data + i);
        if (!fe_is_zero(d)) run = FMUL(run, d);
    }
    fe p = run, s = run;
    pre[t] = p;
    suf[t] = s;
    __syncthreads();
#pragma unroll 1
    for (unsigned off = 1; off < kInvThreads; off <<= 1) {
        fe pp = one, ss = one;
        if (t >= off) pp = pre[t - off];
        if (t + off < kInvThreads) ss = suf[t + off];
        __syncthreads();
        if (t >= off) p = FMUL(p, pp);
        if (t + off < kInvThreads) s = FMUL(s, ss);
        pre[t] = p;
        suf[t] = s;
        __syncthreads();
    }
    if (t == 0) binv = fe_inv_euclid<Fr>(pre[kInvThreads - 1]);
    __syncthreads();
    fe inv = binv;
    if (t > 0) inv = FMUL(inv, pre[t - 1]);
    if (t + 1 < kInvThreads) inv = FMUL(inv, suf[t + 1]);
    for (size_t i = end; i-- > beg;) {
        const fe d = fe_load(data + i);
        const bool zero = fe_is_zero(d);
        fe r = FMUL(inv, fe_load(scratch + i));
        if (RATIO) r = FMUL(fe_load_ro(num + i), r);
        fe_store(data + i, zero ? fe_zero() : r);
        if (!zero) inv = FMUL(inv, d);
    }
}

// ---- round 1 / 2 helpers -------------------------------------------------------------------------
// Per-proof scalars (blinders, challenges and what the host derives from them) reach the prover's kernels through
// `dyn`: a pointer into the context's device copy of ProofParams, so that the kernel ARGUMENTS are the same for every
// proof of a key and a round can be replayed as a CUDA graph.  dyn == nullptr: the by-value fields are used (link
// proofs, the stand-alone polynomial entry points).
struct BlindArgs {
    fe b[3];
    int count;
    const fe* dyn;
};
// poly += (b0 + b1 X + ...) * (X^n - 1)
__global__ void k_blind(fe* poly, size_t n, BlindArgs a) {
    const int i = threadIdx.x;
    if (i >= a.count) return;
    const fe b = a.dyn ? fe_load_ro(a.dyn + i) : a.b[i];
    fe_store(poly + i, FSUB(fe_load(poly + i), b));
    fe_store(poly + n + i, FADD(fe_load(poly + n + i), b));
}

// the five wire polynomials in one launch: thread (i, t) adds blinder t of wire i
__global__ void k_blind_wires(fe* wpoly, size_t stride, size_t n, const fe* __restrict__ dyn /* [NW][2] */) {
    const int i = threadIdx.x >> 1, t = threadIdx.x & 1;
    if (i >= NW) return;
    fe* poly = wpoly + (size_t)i * stride;
    const fe b = fe_load_ro(dyn + 2 * i + t);
    fe_store(poly + t, FSUB(fe_load(poly + t), b));
    fe_store(poly + n + t, FADD(fe_load(poly + n + t), b));
}

// per row j: num = prod_i (w_ij + beta k_i w^j + gamma), den = prod_i (w_ij + beta sigma_ij + gamma)
__global__ void k_perm_num_den(const fe* __restrict__ wires, const fe* __restrict__ sig_evals,
                               const fe* __restrict__ dom, KArr k, const fe* __restrict__ beta_gamma, size_t n,
                               fe* __restrict__ num, fe* __restrict__ den) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const fe beta = fe_load_ro(beta_gamma), gamma = fe_load_ro(beta_gamma + 1);
    const fe bw = FMUL(beta, fe_load_ro(dom + j));
    fe a = fe_one<Fr>(), b = fe_one<Fr>();
#pragma unroll
    for (int i = 0; i < NW; ++i) {
        const fe t = FADD(fe_load_ro(wires + i * n + j), gamma);
        a = FMUL(a, FADD(t, FMUL(k.v[i], bw)));
        b = FMUL(b, FADD(t, FMUL(beta, fe_load_ro(sig_evals + i * n + j))));
    }
    fe_store(num + j, a);
    fe_store(den + j, b);
}

// exclusive multiplicative scan, chunked: data[j] <- prod_{i<j} data[i]
__global__ void k_scan_mul_local(fe* __restrict__ data, size_t n, fe* __restrict__ totals) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t beg = t * CH;
    if (beg >= n) return;
    const size_t end = beg + CH < n ? beg + CH : n;
    fe run = fe_one<Fr>();
    for (size_t i = beg; i < end; ++i) {
        const fe v = fe_load(data + i);
        fe_store(data + i, run);
        run = FMUL(run, v);
    }
    fe_store(totals + t, run);
}
__global__ void k_scan_mul_apply(fe* __restrict__ data, size_t n, const fe* __restrict__ offs) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n || j < CH) return;  // the first chunk's offset is 1
    fe_store(data + j, FMUL(fe_load(data + j), fe_load_ro(offs + j / CH)));
}

// ---- Horner suffix scan: S[j] = sum_{i >= j} p[i] z^(i-j) -------------------------------------------
// S[0] = p(z) (evaluation) and S[1..] are the coefficients of p(X) / (X - z) (synthetic division).
__global__ void k_horner_local(const fe* __restrict__ p, size_t len, fe z_val, const fe* __restrict__ z_dyn, fe* __restrict__ S,
                               fe* __restrict__ H) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t beg = t * CH;
    if (beg >= len) return;
    const size_t end = beg + CH < len ? beg + CH : len;
    const fe z = z_dyn ? fe_load_ro(z_dyn) : z_val;
    fe run = fe_zero();
    for (size_t i = end; i-- > beg;) {
        run = FADD(FMUL(run, z), fe_load_ro(p + i));
        if (S) fe_store(S + i, run);
    }
    fe_store(H + t, run);
}
// batched evaluation-only variant: blockIdx.y selects the polynomial
constexpr int kMaxEval = 10;
struct EvalArgs {
    const fe* p[kMaxEval];
    fe* H[kMaxEval];
    fe z[kMaxEval];
    uint32_t len[kMaxEval];
    const fe* dyn;  // z[] of this level in device memory, or null
};
__global__ void k_horner_local_batch(EvalArgs a) {
    const int q = blockIdx.y;
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t beg = t * CH, len = a.len[q];
    if (beg >= len) return;
    const size_t end = beg + CH < len ? beg + CH : len;
    const fe z = a.dyn ? fe_load_ro(a.dyn + q) : a.z[q];
    const fe* p = a.p[q];
    fe run = fe_zero();
    for (size_t i = end; i-- > beg;) run = FADD(FMUL(run, z), fe_load_ro(p + i));
    fe_store(a.H[q] + t, run);
}
// S[j] += z^(chunk_end - j) * T[chunk + 1], one thread per element; zpow[e] = z^e for e = 1..CH
struct ZPow {
    fe v[CH + 1];
};
__global__ void k_horner_apply(fe* __restrict__ S, size_t len, ZPow zp, const fe* __restrict__ zp_dyn, const fe* __restrict__ T,
                               size_t n_chunks) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t t = j / CH;
    if (j >= len || t + 1 >= n_chunks) return;  // the last chunk has no carry
    const size_t e = (t + 1) * CH - j;
    const fe ze = zp_dyn ? fe_load_ro(zp_dyn + e) : zp.v[e];
    fe_store(S + j, FADD(fe_load(S + j), FMUL(ze, fe_load_ro(T + t + 1))));
}

// ---- round 3: quotient over nc cosets s_j * H_n of the 8n-th roots' coset g * H_8n ---------------------
// The reference evaluates the quotient on all of g * H_8n (8n points, the next power of two above its
// degree 5n + 7) and interpolates with one size-8n inverse FFT.  g * H_8n is the union of the 8 cosets
// s_j * H_n, s_j = g * w_8n^j, and t(X) = sum_k X^(kn) t_k(X) (deg t_k < n) restricted to coset j is
// u_j = sum_k c_j^k t_k with c_j = s_j^n: nc = 6 cosets (6n > 5n + 7 points) determine t.  So every
// polynomial is evaluated on 6 cosets with size-n transforms (after folding X^n -> c_j), the quotient
// kernel runs on 6n points, and t comes back from 6 size-n inverse transforms and one 6 x 6
// inverse-Vandermonde combination per coefficient index — the same coefficients, 25 % fewer points and
// 16 instead of 19 butterfly levels.  Layout of every table: [coset j][h], point s_j * w_n^h.
struct CosetConsts {
    fe cn[8];  // c_j = s_j^n
};
// dst[(p * nc + j) * n + i] = (a_p[i] + c_j * a_p[n + i]) * s_j^i : input of the size-n transform that
// evaluates polynomial p (len <= 2n coefficients, `src_stride` apart) on coset j
__global__ void k_coset_fold(const fe* __restrict__ src, size_t src_stride, size_t len, size_t n, int nc,
                             CosetConsts cc, const fe* __restrict__ cscale, fe* __restrict__ dst) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = blockIdx.y;
    const fe* a = src + (size_t)blockIdx.z * src_stride;
    fe v = fe_load_ro(a + i);
    if (n + i < len) v = FADD(v, FMUL(cc.cn[j], fe_load_ro(a + n + i)));
    v = FMUL(v, fe_load_ro(cscale + (size_t)j * n + i));
    fe_store(dst + ((size_t)blockIdx.z * nc + j) * n + i, v);
}

constexpr int kMaxCosets = 8;
struct CombineArgs {
    fe minv[kMaxCosets * kMaxCosets];  // inverse of the Vandermonde matrix V[j][k] = c_j^k, row-major [k][j]
};
// in place: q[j * n + i] holds (n^-1-scaled) coefficient i of u_j(s_j X); afterwards q[k * n + i] = t_k[i]
template <int NC>
__global__ void k_coset_combine(fe* __restrict__ q, size_t n, const fe* __restrict__ cscale_inv, CombineArgs a) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe u[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) u[j] = FMUL(fe_load(q + (size_t)j * n + i), fe_load_ro(cscale_inv + (size_t)j * n + i));
#pragma unroll 1
    for (int k = 0; k < NC; ++k) {
        fe acc = FMUL(a.minv[k * NC], u[0]);
#pragma unroll
        for (int j = 1; j < NC; ++j) acc = FADD(acc, FMUL(a.minv[k * NC + j], u[j]));
        fe_store(q + (size_t)k * n + i, acc);
    }
}

struct QuotArgs {
    const fe* sel;   // 13 x m resident coset evaluations
    const fe* sig;   // 5 x m
    const fe* ext;   // 7 x m: wires 0..4, public-input polynomial, z
    const fe* pts;   // m evaluation points s_j * w_n^h
    const fe* l1_inv;  // 1 / (n (x_i - 1))
    fe* out;
    size_t m;        // nc * n
    unsigned log_n;
    KArr k;
    const fe* chal;  // device: beta, gamma, alpha, alpha^2
    fe zh_inv[8];    // 1 / (c_j - 1)
};
// k_quotient chains ~60 field products; fully unrolled it is ~180 KB of code and starves on the
// instruction cache (ncu: 1.9 "no instruction" stalls per issue; an out-of-line multiplier was
// slower still: 0.85 -> 0.98 ms, stack traffic).  The per-wire loops are therefore kept rolled.
__global__ void __launch_bounds__(128) k_quotient(QuotArgs a) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.m) return;
    const size_t m = a.m;
    const fe beta = fe_load_ro(a.chal), gamma = fe_load_ro(a.chal + 1);
    fe w[NW];
#pragma unroll
    for (int j = 0; j < NW; ++j) w[j] = fe_load_ro(a.ext + j * m + i);
    // gate: q_c + pi + sum q_lc w + q_mul0 w0 w1 + q_mul1 w2 w3 + q_ecc w0..w4 + sum q_hash w^5 - q_o w4
    fe acc = FADD(fe_load_ro(a.sel + 11 * m + i), fe_load_ro(a.ext + 5 * m + i));
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        acc = FADD(acc, FMUL(fe_load_ro(a.sel + j * m + i), w[j]));
        const fe w2 = fe_sqr<Fr>(w[j]);
        acc = FADD(acc, FMUL(fe_load_ro(a.sel + (6 + j) * m + i), FMUL(fe_sqr<Fr>(w2), w[j])));
    }
    const fe w01 = FMUL(w[0], w[1]), w23 = FMUL(w[2], w[3]);
    acc = FADD(acc, FMUL(fe_load_ro(a.sel + 4 * m + i), w01));
    acc = FADD(acc, FMUL(fe_load_ro(a.sel + 5 * m + i), w23));
    acc = FADD(acc, FMUL(fe_load_ro(a.sel + 12 * m + i), FMUL(FMUL(w01, w23), w[4])));
    acc = FSUB(acc, FMUL(fe_load_ro(a.sel + 10 * m + i), w[4]));
    // permutation: alpha * ( z prod(w + beta k x + gamma) - z(wx) prod(w + beta sigma + gamma) )
    const fe zx = fe_load_ro(a.ext + 6 * m + i);
    const size_t nmask = ((size_t)1 << a.log_n) - 1;
    const fe zxw = fe_load_ro(a.ext + 6 * m + ((i & ~nmask) | ((i + 1) & nmask)));  // z(w x): next point of the same coset
    const fe bx = FMUL(beta, fe_load_ro(a.pts + i));
    fe p1 = zx, p2 = zxw;
#pragma unroll 1
    for (int j = 0; j < NW; ++j) {
        const fe t = FADD(w[j], gamma);
        p1 = FMUL(p1, FADD(t, FMUL(a.k.v[j], bx)));
        p2 = FMUL(p2, FADD(t, FMUL(beta, fe_load_ro(a.sig + j * m + i))));
    }
    acc = FADD(acc, FMUL(fe_load_ro(a.chal + 2), FSUB(p1, p2)));
    acc = FMUL(acc, a.zh_inv[i >> a.log_n]);
    // alpha^2 (z - 1) L1(x) / Z_H(x)
    acc = FADD(acc, FMUL(FMUL(fe_load_ro(a.chal + 3), FSUB(zx, fe_one<Fr>())), fe_load_ro(a.l1_inv + i)));
    fe_store(a.out + i, acc);
}

// flag bit 0: a coefficient above `deg` is non-zero; bit 1: coefficient `deg` is zero
__global__ void k_check_degree(const fe* __restrict__ q, size_t deg, size_t m, uint32_t* flag) {
    const size_t i = deg + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const bool zero = fe_is_zero(fe_load_ro(q + i));
    if (i == deg) {
        if (zero) atomicOr(flag, 2u);
    } else if (!zero) {
        atomicOr(flag, 1u);
    }
}

// out[j] = prod_i (x_j - roots[i]), x_j = g * w^j the j-th point of the coset g * H_N (tw[k] = w^k, k < N/2)
__global__ void k_vanishing_on_coset(const fe* __restrict__ tw, size_t N, fe g, const fe* __restrict__ roots, size_t count,
                                     fe* __restrict__ out) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    const size_t half = N >> 1;
    fe wj = fe_load_ro(tw + (j < half ? j : j - half));
    if (j >= half) wj = fe_neg<Fr>(wj);
    const fe x = FMUL(g, wj);
    fe acc = fe_one<Fr>();
    for (size_t i = 0; i < count; ++i) acc = FMUL(acc, FSUB(x, fe_load_ro(roots + i)));
    fe_store(out + j, acc);
}

// flag |= 1 when any of the `count` elements is non-zero (single small block)
__global__ void k_any_nonzero(const fe* __restrict__ v, size_t count, uint32_t* flag) {
    for (size_t i = threadIdx.x; i < count; i += blockDim.x)
        if (!fe_is_zero(fe_load_ro(v + i))) atomicOr(flag, 1u);
}


// ---- element-wise Fr vector primitives (the collaborative prover's share arithmetic) ------------------------------
// out[i] = a[i] (op) b[i]  or  a[i] (op) b[0] when b is a scalar; op: 0 add, 1 sub, 2 mul
__global__ void k_fr_vec_op(int op, const fe* __restrict__ a, const fe* __restrict__ b, int b_scalar, size_t n, fe* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const fe x = fe_load(a + i), y = fe_load(b + (b_scalar ? 0 : i));
    fe r;
    switch (op) {
        case 0: r = FADD(x, y); break;
        case 1: r = FSUB(x, y); break;
        default: r = FMUL(x, y); break;
    }
    fe_store(out + i, r);
}


// t_i = quot[i(n+2) .. ) - b_{i-1} + b_i X^(n+2)   (the last chunk has n coefficients)
__global__ void k_split_quotient(const fe* __restrict__ quot, size_t n, size_t stride, const fe* __restrict__ dyn /* b[4] */,
                                 fe* __restrict__ out) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y;
    if (j >= n + 3) return;
    const size_t len = i < NW - 1 ? n + 2 : n;
    fe v = j < len ? fe_load_ro(quot + (size_t)i * (n + 2) + j) : fe_zero();
    if (j == 0 && i > 0) v = FSUB(v, fe_load_ro(dyn + i - 1));
    if (j == n + 2 && i < NW - 1) v = fe_load_ro(dyn + i);
    fe_store(out + (size_t)i * stride + j, v);
}

// ---- round 5: linear combination of polynomials -------------------------------------------------------
constexpr int kMaxLin = 32;
struct LinArgs {
    const fe* p[kMaxLin];
    uint32_t len[kMaxLin];
    fe s[kMaxLin];
    int count;
    const fe* dyn;  // s[] in device memory, or null
};
__global__ void k_lincomb(LinArgs a, size_t out_len, fe* __restrict__ out) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= out_len) return;
    fe acc = fe_zero();
    for (int t = 0; t < a.count; ++t)
        if (j < a.len[t]) acc = FADD(acc, FMUL(a.dyn ? fe_load_ro(a.dyn + t) : a.s[t], fe_load_ro(a.p[t] + j)));
    fe_store(out + j, acc);
}

// ---- per-proof scalars ------------------------------------------------------------------------------------
// Everything a proof's kernels need that is not a function of (context, proving key): blinders, Fiat–Shamir challenges
// and the host-side values derived from them.  The host fills the pinned copy between rounds; each round's first
// operation copies it to the device copy the kernels read (see `dyn` above).
constexpr int kLevels = 8;  // levels of the chunked Horner scans: CH^8 = 2^32 coefficients
struct OpenParams {
    fe z[kLevels];     // the point raised to CH^level
    ZPow zp[kLevels];  // powers 0..CH of z[level]
};
struct ProofParams {
    fe blind_w[NW][2];             // round 1
    fe chal[4];                    // beta, gamma (round 2), alpha, alpha^2 (round 3)
    fe blind_z[4];                 // 3 used
    fe blind_q[4];                 // round 3
    fe eval_z[kLevels][kMaxEval];  // round 4
    fe lin_s[kMaxLin];             // round 5
    OpenParams open[2];            // zeta, zeta * w
};

struct LinkParams {  // the same for a link proof
    fe lin_s[4];      // 1, -Z_D(eta)
    OpenParams open;  // eta
};

inline unsigned grid_for(size_t n, unsigned bs) { return (unsigned)((n + bs - 1) / bs); }

}  // namespace

// data[i] <- 1 / data[i] (num == nullptr) or num[i] / data[i]; enqueue only.  scratch: n elements.
static inline void batch_inverse_enqueue(const fe* num, fe* data, fe* scratch, size_t n, cudaStream_t st) {
    if (num) B200_LAUNCH(k_block_inverse<true>, grid_for(n, kInvBlock), kInvThreads, 0, st)(num, data, scratch, n);
    else B200_LAUNCH(k_block_inverse<false>, grid_for(n, kInvBlock), kInvThreads, 0, st)(nullptr, data, scratch, n);
}

// ---------------------------------------------------------------------------------------------
// host-side structures
// ---------------------------------------------------------------------------------------------
struct ProvingKey {
    uint64_t id = g_object_ids.fetch_add(1);  // never reused: what a context's captured graphs are keyed by
    unsigned log_n = 0;
    size_t n = 0, m = 0, num_inputs = 0;
    KArr k;
    const Bases* srs = nullptr;
    fe *sel_coeffs = nullptr, *sig_coeffs = nullptr, *sig_evals = nullptr;
    fe *ce_sel = nullptr, *ce_sig = nullptr;
    fe *dom = nullptr, *coset_pts = nullptr, *l1_inv = nullptr;
    // quotient domain: nc cosets s_j * H_n, m = nc * n points (see "round 3" above)
    int nc = 0;
    fe *cscale = nullptr, *cscale_inv = nullptr;  // s_j^i and s_j^-i, [j][i]
    CosetConsts cc;
    CombineArgs comb;
    fe zh_inv[8];
    fe group_gen;
    g1_affine sel_comms[NS], sig_comms[NW];
    ~ProvingKey() {
        for (fe* p : {sel_coeffs, sig_coeffs, sig_evals, ce_sel, ce_sig, dom, coset_pts, l1_inv, cscale, cscale_inv})
            if (p) cudaFree(p);
    }
};

// inverse of the nc x nc matrix a (row-major) over Fr by Gauss–Jordan elimination (host, set-up time)
static inline bool host_mat_inverse(const fe* a, int nc, fe* out) {
    const fe one = fe_one<Fr>(), zero = fe_zero();
    std::vector<fe> m((size_t)nc * 2 * nc);
    for (int r = 0; r < nc; ++r)
        for (int c = 0; c < nc; ++c) {
            m[(size_t)r * 2 * nc + c] = a[r * nc + c];
            m[(size_t)r * 2 * nc + nc + c] = r == c ? one : zero;
        }
    for (int col = 0; col < nc; ++col) {
        int piv = -1;
        for (int r = col; r < nc && piv < 0; ++r)
            if (!fe_is_zero(m[(size_t)r * 2 * nc + col])) piv = r;
        if (piv < 0) return false;
        for (int c = 0; c < 2 * nc; ++c) std::swap(m[(size_t)col * 2 * nc + c], m[(size_t)piv * 2 * nc + c]);
        const fe iv = fe_inv<Fr>(m[(size_t)col * 2 * nc + col]);
        for (int c = 0; c < 2 * nc; ++c) m[(size_t)col * 2 * nc + c] = FMUL(m[(size_t)col * 2 * nc + c], iv);
        for (int r = 0; r < nc; ++r) {
            if (r == col) continue;
            const fe f = m[(size_t)r * 2 * nc + col];
            if (fe_is_zero(f)) continue;
            for (int c = 0; c < 2 * nc; ++c)
                m[(size_t)r * 2 * nc + c] = FSUB(m[(size_t)r * 2 * nc + c], FMUL(f, m[(size_t)col * 2 * nc + c]));
        }
    }
    for (int r = 0; r < nc; ++r)
        for (int c = 0; c < nc; ++c) out[r * nc + c] = m[(size_t)r * 2 * nc + nc + c];
    return true;
}

static inline fe host_pow(fe a, uint64_t e) {
    fe r = fe_one<Fr>();
    while (e) {
        if (e & 1) r = FMUL(r, a);
        a = fe_sqr<Fr>(a);
        e >>= 1;
    }
    return r;
}
static inline fe host_from_u64(uint64_t v) {
    fe x = fe_zero();
    x.l[0] = (uint32_t)v;
    x.l[1] = (uint32_t)(v >> 32);
    return fe_to_mont<Fr>(x);
}

// Runs the enclosed launches on the context's low-priority stream (b200_init), ordered after what is
// already queued on `st` and before what `st` gets next: for the long throughput-bound kernels, so that
// other contexts' short kernels are scheduled ahead of them.
struct HeavyScope {
    Context* c;
    cudaStream_t st, run;
    HeavyScope(Context* c_, cudaStream_t st_) : c(c_), st(st_), run(c_->heavy_plonk ? c_->heavy : st_) {
        if (c->heavy_plonk) {
            cudaEventRecord(c->hv_fork, st);
            cudaStreamWaitEvent(run, c->hv_fork, 0);
        }
    }
    ~HeavyScope() {
        if (c->heavy_plonk) {
            cudaEventRecord(c->hv_join, run);
            cudaStreamWaitEvent(st, c->hv_join, 0);
        }
    }
};

// exclusive product scan of `data[0..n)` in place; scratch >= n/CH + n/CH^2 + 2*CH + 8 elements
static inline void scan_mul_exclusive(fe* data, size_t n, fe* scratch, cudaStream_t st) {
    if (n <= 1) {
        // data[0] <- 1 handled by the local kernel as well
    }
    const size_t n1 = (n + CH - 1) / CH;
    B200_LAUNCH(k_scan_mul_local, grid_for(n1, 128), 128, 0, st)(data, n, scratch);
    if (n1 > 1) {
        scan_mul_exclusive(scratch, n1, scratch + n1, st);
        B200_LAUNCH(k_scan_mul_apply, grid_for(n, 256), 256, 0, st)(data, n, scratch);
    }
}

// Horner suffix scan; S may be null (evaluation only).  The value p(z) ends up at out_total (device).
// scratch >= 2 * (len/CH + len/CH^2 + 2*CH + 8) elements
// `dyn` (device, or null): the point and its powers per level come from there instead of `z` (see ProofParams).
static inline void horner_suffix(const fe* p, size_t len, fe z, fe* S, fe* out_total, fe* scratch, cudaStream_t st,
                          const OpenParams* dyn = nullptr, int level = 0) {
    const size_t n1 = (len + CH - 1) / CH;
    fe* H = scratch;
    fe* T = scratch + n1;
    B200_LAUNCH(k_horner_local, grid_for(n1, 128), 128, 0, st)(p, len, z, dyn ? &dyn->z[level] : nullptr, S, H);
    if (n1 == 1) {
        cudaMemcpyAsync(out_total, H, sizeof(fe), cudaMemcpyDeviceToDevice, st);
        return;
    }
    const fe zc = dyn ? z : host_pow(z, CH);
    horner_suffix(H, n1, zc, S ? T : nullptr, out_total, scratch + 2 * n1, st, dyn, level + 1);
    if (S) {
        ZPow zp{};
        if (!dyn) {
            zp.v[0] = fe_one<Fr>();
            for (int e = 1; e <= CH; ++e) zp.v[e] = FMUL(zp.v[e - 1], z);
        }
        B200_LAUNCH(k_horner_apply, grid_for(len, 256), 256, 0, st)(S, len, zp, dyn ? dyn->zp[level].v : nullptr, T, n1);
    }
}

// p_q(z_q) for up to kMaxEval polynomials, written to out[q];
// scratch: count * (max_len/CH + max_len/CH^2 + 2*CH + 16)
// `dyn_z` (device, or null): [level][kMaxEval] evaluation points, points[q]^(CH^level); `points` is unused then.
static inline void eval_batch(const fe* const* polys, const size_t* lens, const fe* points, int count, fe* out, fe* scratch,
                       cudaStream_t st, const fe (*dyn_z)[kMaxEval] = nullptr) {
    EvalArgs a;
    size_t cur_len[kMaxEval], max_len = 0;
    for (int q = 0; q < count; ++q) {
        a.p[q] = polys[q];
        a.z[q] = dyn_z ? fe_zero() : points[q];
        cur_len[q] = lens[q];
        max_len = lens[q] > max_len ? lens[q] : max_len;
    }
    // two disjoint regions per polynomial (levels alternate A, B, A, ...): a level reads one and
    // writes the other
    const size_t region_a = max_len / CH + 2, region_b = max_len / CH / CH + CH + 2;
    const size_t per_poly = region_a + region_b;
    int level = 0;
    while (true) {
        bool last = true;
        size_t max_chunks = 0;
        for (int q = 0; q < count; ++q) {
            const size_t n1 = (cur_len[q] + CH - 1) / CH;
            if (n1 > 1) last = false;
            max_chunks = n1 > max_chunks ? n1 : max_chunks;
        }
        for (int q = 0; q < count; ++q) {
            a.len[q] = (uint32_t)cur_len[q];
            // levels alternate between the two halves of each polynomial's scratch slice
            a.H[q] = last ? out + q : scratch + (size_t)q * per_poly + (level & 1 ? region_a : 0);
        }
        a.dyn = dyn_z ? &dyn_z[level][0] : nullptr;
        B200_LAUNCH(k_horner_local_batch, dim3(grid_for(max_chunks, 64), count), 64, 0, st)(a);
        if (last) break;
        for (int q = 0; q < count; ++q) {
            a.p[q] = a.H[q];
            if (!dyn_z) a.z[q] = host_pow(a.z[q], CH);
            cur_len[q] = (cur_len[q] + CH - 1) / CH;
        }
        ++level;
    }
}

struct Workspace {
    fe *wires_ev, *wpoly, *pi_poly, *zpoly, *num, *den, *tmp, *scan, *ext, *quot, *split, *lin, *sdiv, *hscr, *escr, *evals;
    uint32_t* flag;
    size_t S;  // stride of the (n + 3)-coefficient polynomials
};
static inline size_t workspace_elems(size_t n) {
    const size_t S = n + 4, m = 8 * n;
    return NW * n + NW * S + S + S + 3 * n + (2 * (n / CH) + 4 * CH + 64) + 7 * m + m + NW * S + S + 2 * (S + 8) +
           4 * (S / CH + 4 * CH + 64) + kMaxEval * (S / CH + S / CH / CH + 2 * CH + 16) + 32 + 8;
}
static inline Workspace carve(fe* base, size_t n) {
    Workspace w;
    const size_t S = n + 4, m = 8 * n;
    w.S = S;
    fe* p = base;
    w.wires_ev = p; p += NW * n;
    w.wpoly = p; p += NW * S;
    w.pi_poly = p; p += S;  // directly behind the wire polynomials: one batch of 6 for the coset evaluations
    w.zpoly = p; p += S;
    w.num = p; p += n;
    w.den = p; p += n;
    w.tmp = p; p += n;
    w.scan = p; p += 2 * (n / CH) + 4 * CH + 64;  // all levels of the product scan: n / CH * (1 + 1/CH + ...)
    w.ext = p; p += 7 * m;
    w.quot = p; p += m;
    w.split = p; p += NW * S;
    w.lin = p; p += S;
    w.sdiv = p; p += 2 * (S + 8);
    w.hscr = p; p += 4 * (S / CH + 4 * CH + 64);
    w.escr = p; p += kMaxEval * (S / CH + S / CH / CH + 2 * CH + 16);
    w.evals = p; p += 32;
    w.flag = reinterpret_cast<uint32_t*>(p);
    return w;
}

// `count` commitments to polynomials `stride` coefficients apart, in one batched MSM
static inline int commit_batch(Context* c, const ProvingKey* pk, const fe* d_coeffs, size_t len, size_t stride,
                        unsigned count, g1_affine* out) {
    int inf[32];
    if (count > 32) return B200_ERR_INVALID;
    int rc = msm_device_batch(pk->srs, 0, d_coeffs, len, stride, count, /*montgomery=*/1, &c->msm, c->stream, out, inf);
    if (rc != B200_OK) return rc;
    for (unsigned i = 0; i < count; ++i)
        if (inf[i]) std::memset(&out[i], 0, sizeof(out[i]));
    return B200_OK;
}

static inline int alloc_fe(fe** p, size_t count) {
    cudaError_t e = cudaMalloc(p, count * sizeof(fe));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(proving key)");
    return B200_OK;
}

// Evaluations of `count` polynomials (`len` <= 2n coefficients each, `src_stride` apart) on the nc cosets
// of the quotient domain: dst[(p * nc + j) * n + h] = poly_p(s_j * w_n^h).  scratch: count * nc * n elements.
static inline int coset_evals(const ProvingKey* pk, const Domain* dn, const fe* src, size_t src_stride, size_t len,
                       unsigned count, fe* dst, fe* scratch, cudaStream_t st) {
    const size_t n = pk->n;
    if (len > 2 * n) {
        set_error("coset_evals: polynomial longer than 2n");
        return B200_ERR_INVALID;
    }
    B200_LAUNCH(k_coset_fold, dim3(grid_for(n, 256), (unsigned)pk->nc, count), 256, 0, st)(src, src_stride, len, n, pk->nc, pk->cc,
                                                                                 pk->cscale, dst);
    return ntt_device(dn, dst, scratch, /*inverse=*/0, /*coset=*/0, count * (unsigned)pk->nc, n, st);
}

struct ProofOut {  // same field order and layout as b200_proof / PlonkProofDef
    g1_affine wires_poly_comms[NW];
    g1_affine prod_perm_poly_comm;
    g1_affine split_quot_poly_comms[NW];
    g1_affine opening_proof;
    g1_affine shifted_opening_proof;
    fe wires_evals[NW];
    fe wire_sigma_evals[NW - 1];
    fe perm_next_eval;
};
static_assert(sizeof(ProofOut) == sizeof(b200_proof), "proof layout");

struct LinkOut {
    g1_affine quotient_commitment;
    g1_affine opening_proof;
};
static_assert(sizeof(LinkOut) == sizeof(b200_link_proof), "link proof layout");

static inline void fill_open_params(OpenParams* o, fe z) {
    for (int l = 0; l < kLevels; ++l) {
        o->z[l] = z;
        o->zp[l].v[0] = fe_one<Fr>();
        for (int e = 1; e <= CH; ++e) o->zp[l].v[e] = FMUL(o->zp[l].v[e - 1], z);
        z = o->zp[l].v[CH];
    }
}

}  // namespace b200

struct b200_pk {
    b200::ProvingKey* pk;
};
