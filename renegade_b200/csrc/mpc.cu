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
#include <condition_variable>
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
    bool used = false;
    ~MpcPrep() {
        for (fe* p : {a, b, c, mask})
            if (p) cudaFree(p);
    }
};

static int prep_alloc(Context* c, const ProvingKey* pk, MpcPrep** out) {
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
        return sum_points(prefix_bytes, count, out);
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
        B200_LAUNCH(k_beaver_close, dim3(grid_for(L.len, 256), (unsigned)L.count), 256, 0, st)(L, recv, stride, P, party == 0);
        if (extra_len) sum_fe(off * sizeof(fe), extra_len, extra_sum);
        B200_CUDA(cudaStreamSynchronize(st));  // the next exchange reuses the receive buffer
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
        B200_LAUNCH(k_sum_open, grid_for(len, 256), 256, 0, st)(recv, stride, 0, len, P, out);
        B200_CUDA(cudaStreamSynchronize(st));
        return B200_OK;
    }
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

static int mpc_prove(Party& pt, const ProvingKey* pk, MpcPrep* prep, const fe* h_wires, const fe* h_pub_inputs,
                     const fe* h_blinders, ProofOut* proof, fe* h_link_share, fe* h_challenges) {
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
    if ((rc = c->mpc_ws.reserve(total * sizeof(fe))) != B200_OK) return rc;
    if ((rc = c->ntt_scratch.reserve((size_t)7 * m * sizeof(fe))) != B200_OK) return rc;
    fe* p = reinterpret_cast<fe*>(c->mpc_ws.p);
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
    // first exchange: the statement and the 5 partial wire commitments
    if ((rc = pt.open_commitments(pk->srs, wpoly, n + 2, S, NW, proof->wires_poly_comms, statement, 64)) != B200_OK) return rc;
    for (int q = 1; q < pt.P; ++q)
        if (std::memcmp(pt.payload_of(q), pt.payload_of(0), 64) != 0) {
            set_error("collaborative prover: the parties disagree on the statement (verifying key or public inputs)");
            return B200_ERR_INVALID;
        }
    if (h_link_share) B200_CUDA(cudaMemcpyAsync(h_link_share, wpoly, (n + 2) * sizeof(fe), cudaMemcpyDeviceToHost, st));
    for (int i = 0; i < NW; ++i) tr.append_commitment(proof->wires_poly_comms[i]);

    // ---- round 2 ------------------------------------------------------------------------------------------------
    const fe beta = tr.get_and_append_challenge();
    const fe gamma = tr.get_and_append_challenge();
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
        batch_inverse_enqueue(numr, pub, r2 + 13 * n, n, st);  // pub <- [num r] / (den r) = [num / den]
        B200_CUDA(cudaMemcpyAsync(x, pub, n * sizeof(fe), cudaMemcpyDeviceToDevice, st));
        // inclusive prefix products by doubling: x'[i] = x[i] x[i - d] for i >= d
        for (size_t d = 1; d < n; d <<= 1) {
            B200_CUDA(cudaMemcpyAsync(x2, x, d * sizeof(fe), cudaMemcpyDeviceToDevice, st));
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
    B200_LAUNCH(k_mpc_perm_factors, grid_for(m, 128), 128, 0, st)(ext, m, pk->coset_pts, pk->ce_sig, m, pk->k, beta, gamma, p0 ? 1 : 0, nf, df);
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
        B200_LAUNCH(k_mpc_quotient, grid_for(m, 128), 128, 0, st)(q);
        if ((rc = ntt_device(dn, quot, nscr, 1, 0, (unsigned)pk->nc, n, st)) != B200_OK) return rc;
        if (pk->nc == 6) B200_LAUNCH(k_coset_combine<6>, grid_for(n, 128), 128, 0, st)(quot, n, pk->cscale_inv, pk->comb);
        else B200_LAUNCH(k_coset_combine<8>, grid_for(n, 128), 128, 0, st)(quot, n, pk->cscale_inv, pk->comb);
    }
    // degree check: the coefficients above deg are opened (zero for a satisfied witness) with the Beaver differences
    // of r' q[deg]; then r' q[deg] is opened (non-zero iff q[deg] is)
    const size_t deg = NW * (n + 1) + 2;
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
        bool bad = fe_is_zero(rq_open);
        for (const fe& v : tail_sum) bad = bad || !fe_is_zero(v);
        if (bad) {
            set_error("WrongQuotientPolyDegree: the joint witness does not satisfy the circuit");
            return B200_ERR_UNSATISFIED;
        }
    }
    if (t_used != LY.triples) {
        set_error("collaborative prover: triple schedule out of step");
        return B200_ERR_INVALID;
    }
    B200_LAUNCH(k_split_quotient, dim3(grid_for(n + 3, 256), NW), 256, 0, st)(quot, n, S, d_bl + 13, split);
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
        LinArgs la{};
        const fe* we = proof->wires_evals;
        const fe* se = proof->wire_sigma_evals;
        int t = 0;
        auto push = [&](const fe* poly, size_t len, const fe& s) {
            la.p[t] = poly;
            la.len[t] = (uint32_t)len;
            la.s[t] = s;
            ++t;
        };
        auto pow5 = [&](const fe& x) { return FMUL(fe_sqr<Fr>(fe_sqr<Fr>(x)), x); };
        const fe* sel = pk->sel_coeffs;
        const fe vanish = FSUB(host_pow(zeta, n), one);
        if (p0) {  // the public part of the linearisation
            for (int j = 0; j < 4; ++j) push(sel + (size_t)j * n, n, we[j]);
            push(sel + 4 * n, n, FMUL(we[0], we[1]));
            push(sel + 5 * n, n, FMUL(we[2], we[3]));
            for (int j = 0; j < 4; ++j) push(sel + (size_t)(6 + j) * n, n, pow5(we[j]));
            push(sel + 10 * n, n, fe_neg<Fr>(we[4]));
            push(sel + 11 * n, n, one);
            push(sel + 12 * n, n, FMUL(FMUL(FMUL(we[0], we[1]), FMUL(we[2], we[3])), we[4]));
            fe cs = FMUL(FMUL(alpha, beta), proof->perm_next_eval);
            for (int j = 0; j < NW - 1; ++j) cs = FMUL(cs, FADD(FADD(we[j], FMUL(beta, se[j])), gamma));
            push(pk->sig_coeffs + (size_t)(NW - 1) * n, n, fe_neg<Fr>(cs));
            fe cv = one;
            for (int i = 0; i < 2 * NW - 1; ++i) {
                cv = FMUL(cv, v);
                if (i >= NW) push(pk->sig_coeffs + (size_t)(i - NW) * n, n, cv);
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
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

// link() of plonk.cu on shares: everything is linear in the hints
static int mpc_link(Party& pt, const Bases* srs, const fe* h_a1, size_t len1, const fe* h_a2, size_t len2, const g1_affine& comm1,
                    const g1_affine& comm2, unsigned alignment, size_t offset, size_t size, LinkOut* out, fe* h_eta) {
    Context* c = pt.c;
    cudaStream_t st = pt.st;
    const size_t len = len1 > len2 ? len1 : len2;
    unsigned log_N = 1;
    while (((size_t)1 << log_N) < len) ++log_N;
    const size_t N = (size_t)1 << log_N;
    const size_t L = len + 8, NL = N + 8;
    const size_t scr = 4 * (L / CH + 4 * CH + 64);
    int rc;
    if ((rc = c->mpc_ws.reserve((5 * L + 3 * NL + scr + size + 16) * sizeof(fe))) != B200_OK) return rc;
    if ((rc = c->ntt_scratch.reserve(N * sizeof(fe))) != B200_OK) return rc;
    Domain* dN = nullptr;
    if ((rc = get_domain(c, log_N, &dN)) != B200_OK) return rc;
    fe* base = reinterpret_cast<fe*>(c->mpc_ws.p);
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
    }
    fill_powers(d_roots, size, g, root0, st);
    B200_CUDA(cudaMemsetAsync(d_E, 0, N * sizeof(fe), st));
    B200_CUDA(cudaMemcpyAsync(d_E, d_diff, len * sizeof(fe), cudaMemcpyDeviceToDevice, st));
    if ((rc = ntt_device(dN, d_E, nscr, 0, 1, 1, N, st)) != B200_OK) return rc;
    B200_LAUNCH(k_vanishing_on_coset, grid_for(N, 128), 128, 0, st)(dN->tw_fwd, N, fe_from_u32<Fr>(5), d_roots, size, d_Z);
    batch_inverse_enqueue(d_E, d_Z, d_Q, N, st);  // d_Z <- diff / Z_D on the coset
    if ((rc = ntt_device(dN, d_Z, nscr, 1, 1, 1, N, st)) != B200_OK) return rc;
    const size_t q_len = len - size;
    // exactness: the interpolant's coefficients from q_len on are opened (zero when the hints agree on the group),
    // together with the partial quotient commitment
    {
        g1_affine part;
        rc = commit_partials(c, srs, d_Z, q_len, q_len, 1, &part, st);
        if (rc != B200_OK) return rc;
        const size_t tail = N - q_len, payload = 64 + tail * sizeof(fe);
        if ((rc = pt.reserve(payload)) != B200_OK) return rc;
        std::memcpy(pt.send + kHdr, &part, 64);
        B200_CUDA(cudaMemcpyAsync(pt.send + kHdr + 64, d_Z + q_len, tail * sizeof(fe), cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        if ((rc = pt.exchange_now(payload)) != B200_OK) return rc;
        std::vector<fe> t(tail);
        pt.sum_fe(64, tail, t.data());
        for (const fe& x : t)
            if (!fe_is_zero(x)) {
                set_error("link: the two wire polynomials differ on the link group (wrong layout or mismatched witnesses)");
                return B200_ERR_UNSATISFIED;
            }
        if ((rc = pt.sum_points(0, 1, &out->quotient_commitment)) != B200_OK) return rc;
    }
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
        return B200_ERR_UNSATISFIED;
    }
    return pt.sum_points(0, 1, &out->opening_proof);
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
