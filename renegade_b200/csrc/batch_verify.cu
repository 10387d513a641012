// Batch verification of PlonK proofs and link proofs on the device with one pairing check.
//
// Every check has the KZG shape e(A_j, [tau]_2) == e(B_j, [1]_2).  With a random rho, the N checks hold (up to a
// probability of about N / r) exactly when
//     e(sum_j rho^j A_j, [tau]_2) == e(sum_j rho^j B_j, [1]_2),
// one 2-pair pairing product.  The per-item work is data parallel and runs here:
//   bv_items_kernel     one thread per item: on-curve checks, transcript replay and scalar assembly
//                       (verify_algebra.cuh, the same routines the host verifiers call) -> a list of (point, scalar)
//                       terms and the item's final transcript state;
//   bv_operands_kernel  one block per item, one thread per term: s * P by double-and-add, summed in the block
//                       -> the unweighted operands (A_j, B_j);
//   bv_weight_kernel    one thread per item: rho^j A_j, rho^j B_j;
//   bv_scan_kernel      prefix sums of the weighted operands, so that the sum over any range of items is one
//                       subtraction (bv_range_kernel).
// The host derives rho (Keccak over the items' final transcript states, see batch_challenge) and evaluates the
// pairing products (verify.cu).  When the combined check fails and per-item verdicts are wanted, contiguous ranges are
// bisected with the same weights: k bad items cost at most about 2 k log2(N) pairing products, and a range of one item
// decides that item exactly (rho^j != 0), with the same equation as b200_plonk_verify / b200_plonk_verify_link.
#include <cstring>
#include <vector>

#include "b200prover.h"
#include "device_ctx.h"
#include "pairing.h"
#include "verify_algebra.cuh"

namespace b200 {
namespace {

struct BvVk {
    fe k[kNW];
    g1_affine sel[kNS];
    g1_affine sig[kNW];
    uint64_t num_inputs;
    uint32_t log_n, pad;
};
struct BvProof {
    ProofIn proof;
    uint64_t pi_off;  // first public input in the pool
    uint64_t tr_off;  // transcript bytes of this item in the byte pool
    uint32_t vk;
    uint32_t count_ok;  // the item's public-input count equals its key's
};
struct BvLink {
    g1_affine c1, c2, cq, op;
    uint64_t offset, size;
    uint32_t alignment, pad;
};
struct Operands {
    g1_affine a, b;
};

constexpr int kItemThreads = 64;
constexpr int kTermThreads = 64;  // >= kTermsA + kTermsB
constexpr int kScanThreads = 128;
static_assert(kTermThreads >= kTermsA + kTermsB, "one thread per term");

size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

__global__ void __launch_bounds__(kItemThreads) bv_items_kernel(const BvVk* vks, const BvProof* proofs, size_t n_proofs,
                                                                const BvLink* links, size_t n_links, const fe* pis,
                                                                const fe* roots, uint8_t* tr_pool, OperandTerms* terms,
                                                                uint8_t* states, uint8_t* valid) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_proofs + n_links) return;
    OperandTerms* t = terms + j;
    t->na = t->nb = 0;  // a rejected item contributes the identity
    bool ok;
    uint8_t st[64];
    if (j < n_proofs) {
        const BvProof& it = proofs[j];
        const BvVk& vk = vks[it.vk];
        TranscriptT<ByteSpan> tr(ByteSpan{tr_pool + it.tr_off, 0, plonk_transcript_bytes(vk.num_inputs)});
        ok = it.count_ok && plonk_verify_terms(vk.log_n, (size_t)vk.num_inputs, VkIn{vk.k, vk.sel, vk.sig}, pis + it.pi_off,
                                               it.proof, roots[vk.log_n], tr, t);
        for (int i = 0; i < 64; ++i) st[i] = tr.state()[i];
    } else {
        const BvLink& l = links[j - n_proofs];
        uint8_t buf[kLinkTranscriptBytes];
        TranscriptT<ByteSpan> tr(ByteSpan{buf, 0, sizeof(buf)});
        ok = link_verify_terms(l.c1, l.c2, l.cq, l.op, roots[l.alignment], l.offset, l.size, tr, t);
        for (int i = 0; i < 64; ++i) st[i] = tr.state()[i];
    }
    for (int i = 0; i < 64; ++i) states[64 * j + i] = ok ? st[i] : 0;
    valid[j] = ok ? 1 : 0;
}

FF_D g1_xyzz term_mul(const G1Term& t) {
    const g1_affine p = t.p;
    const fe s = t.s;
    if (g1_affine_is_inf(p) || fe_is_zero(s)) return g1_xyzz_inf();
    return g1_mul_bits(p, fe_from_mont<FrCfg>(s), 254);
}

__global__ void __launch_bounds__(kTermThreads) bv_operands_kernel(const OperandTerms* terms, Operands* out) {
    __shared__ g1_xyzz part[kTermsA + kTermsB];
    const OperandTerms& t = terms[blockIdx.x];
    const int tid = threadIdx.x;
    if (tid < kTermsA) {
        part[tid] = tid < t.na ? term_mul(t.a[tid]) : g1_xyzz_inf();
    } else if (tid < kTermsA + kTermsB) {
        const int k = tid - kTermsA;
        part[tid] = k < t.nb ? term_mul(t.b[k]) : g1_xyzz_inf();
    }
    __syncthreads();
    if (tid < 2) {  // thread 0 sums A, thread 1 sums B
        const int lo = tid == 0 ? 0 : kTermsA, hi = tid == 0 ? kTermsA : kTermsA + kTermsB;
        g1_xyzz acc = g1_xyzz_inf();
        for (int i = lo; i < hi; ++i) acc = g1_add(acc, part[i]);
        const g1_affine r = g1_to_affine(acc);
        if (tid == 0)
            out[blockIdx.x].a = r;
        else
            out[blockIdx.x].b = r;
    }
}

__global__ void __launch_bounds__(kItemThreads) bv_weight_kernel(const Operands* ops, size_t n, fe rho, g1_xyzz* wa, g1_xyzz* wb) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const fe w = fe_from_mont<FrCfg>(fr_pow_u64(rho, (uint64_t)j));
    g1_xyzz_store(wa + j, g1_mul_bits(ops[j].a, w, 254));
    g1_xyzz_store(wb + j, g1_mul_bits(ops[j].b, w, 254));
}

// pa[i] = sum_{j < i} wa[j], i <= n (pa[0] the identity); same for b.  One block: each thread sums a contiguous chunk,
// the chunk totals are scanned by one thread, and each chunk adds its offset.
__global__ void __launch_bounds__(kScanThreads) bv_scan_kernel(const g1_xyzz* wa, const g1_xyzz* wb, size_t n, g1_xyzz* pa,
                                                               g1_xyzz* pb) {
    __shared__ g1_xyzz tot_a[kScanThreads], tot_b[kScanThreads];
    const int tid = threadIdx.x;
    const size_t chunk = (n + kScanThreads - 1) / kScanThreads;
    const size_t lo = (size_t)tid * chunk, hi = lo + chunk < n ? lo + chunk : n;
    g1_xyzz acc_a = g1_xyzz_inf(), acc_b = g1_xyzz_inf();
    for (size_t i = lo; i < hi; ++i) {
        acc_a = g1_add(acc_a, g1_xyzz_load(wa + i));
        acc_b = g1_add(acc_b, g1_xyzz_load(wb + i));
        g1_xyzz_store(pa + i + 1, acc_a);
        g1_xyzz_store(pb + i + 1, acc_b);
    }
    tot_a[tid] = acc_a;
    tot_b[tid] = acc_b;
    __syncthreads();
    if (tid == 0) {  // exclusive scan of the chunk totals, in place
        g1_xyzz run_a = g1_xyzz_inf(), run_b = g1_xyzz_inf();
        for (int i = 0; i < kScanThreads; ++i) {
            const g1_xyzz ta = tot_a[i], tb = tot_b[i];
            tot_a[i] = run_a;
            tot_b[i] = run_b;
            run_a = g1_add(run_a, ta);
            run_b = g1_add(run_b, tb);
        }
        g1_xyzz_store(pa, g1_xyzz_inf());
        g1_xyzz_store(pb, g1_xyzz_inf());
    }
    __syncthreads();
    const g1_xyzz off_a = tot_a[tid], off_b = tot_b[tid];
    for (size_t i = lo; i < hi; ++i) {
        g1_xyzz_store(pa + i + 1, g1_add(off_a, g1_xyzz_load(pa + i + 1)));
        g1_xyzz_store(pb + i + 1, g1_add(off_b, g1_xyzz_load(pb + i + 1)));
    }
}

// out = (pa[hi] - pa[lo], pb[hi] - pb[lo]) in affine: the weighted operands of the items [lo, hi)
__global__ void bv_range_kernel(const g1_xyzz* pa, const g1_xyzz* pb, size_t lo, size_t hi, Operands* out) {
    const g1_xyzz* p = threadIdx.x == 0 ? pa : pb;
    g1_xyzz neg = g1_xyzz_load(p + lo);
    neg.y = fe_neg<FqCfg>(neg.y);
    const g1_affine r = g1_to_affine(g1_add(g1_xyzz_load(p + hi), neg));
    if (threadIdx.x == 0)
        out->a = r;
    else
        out->b = r;
}

// The batch challenge rho: a Keccak challenge over, item by item, each PlonK item's final transcript state, each link
// item's final state, opening proof pi and group layout, then the two G2 records.  A PlonK item's final state binds
// its key, public inputs and whole proof.  The link transcript absorbs C1, C2 and Cq only: pi and (alignment, offset,
// size) are not in it, so they are hashed here explicitly, else an adversary could choose them after seeing rho.
fe batch_challenge(const uint8_t* states, size_t n_proofs, const b200_batch_link* links, size_t n_links,
                   const uint64_t g2_h[16], const uint64_t g2_tau_h[16]) {
    SolidityTranscript tr;
    for (size_t j = 0; j < n_proofs; ++j) tr.append_message(states + 64 * j, 64);
    for (size_t l = 0; l < n_links; ++l) {
        tr.append_message(states + 64 * (n_proofs + l), 64);
        g1_affine op;
        std::memcpy(&op, links[l].proof->opening_proof, 64);
        tr.append_commitment(op);
        tr.append_u32_be(links[l].alignment);
        tr.append_u64_be((uint64_t)links[l].offset);
        tr.append_u64_be((uint64_t)links[l].size);
    }
    tr.append_message(reinterpret_cast<const uint8_t*>(g2_h), 128);
    tr.append_message(reinterpret_cast<const uint8_t*>(g2_tau_h), 128);
    fe rho = tr.get_and_append_challenge();
    for (uint32_t ctr = 0; fe_is_zero(rho); ++ctr) {  // a zero weight would drop items: re-derive instead
        tr.append_u32_be(ctr);
        rho = tr.get_and_append_challenge();
    }
    return rho;
}

struct BatchRun {
    Context* c;
    g1_xyzz *pa, *pb;
    Operands* d_range;
    Operands* h_range;
    g2_affine qs[2];
    size_t pairings = 0;
    // e(A, [tau]_2) * e(-B, [1]_2) == 1 for the weighted operands of the items [lo, hi)
    int range_ok(size_t lo, size_t hi, bool* ok) {
        B200_LAUNCH(bv_range_kernel, 1, 2, 0, c->stream)(pa, pb, lo, hi, d_range);
        B200_CUDA(cudaGetLastError());
        B200_CUDA(cudaMemcpyAsync(h_range, d_range, sizeof(Operands), cudaMemcpyDeviceToHost, c->stream));
        B200_CUDA(cudaStreamSynchronize(c->stream));
        const g1_affine ps[2] = {h_range->a, g1_affine_neg(h_range->b)};
        *ok = pairing_product_is_one(ps, qs, 2);
        ++pairings;
        return B200_OK;
    }
    // [lo, hi) is known to fail: find its bad items (flags start at 1)
    int bisect(size_t lo, size_t hi, uint8_t* flags) {
        if (hi - lo == 1) {
            flags[lo] = 0;
            return B200_OK;
        }
        const size_t mid = lo + (hi - lo) / 2;
        bool left = false;
        int rc = range_ok(lo, mid, &left);
        if (rc != B200_OK) return rc;
        if (left) return bisect(mid, hi, flags);  // the product of the halves is the failing whole: the right fails
        rc = bisect(lo, mid, flags);
        if (rc != B200_OK) return rc;
        bool right = false;
        rc = range_ok(mid, hi, &right);
        if (rc != B200_OK) return rc;
        return right ? B200_OK : bisect(mid, hi, flags);
    }
};

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" int b200_plonk_batch_verify(b200_ctx* ctx, const b200_batch_vk* vks, size_t n_vks, const b200_batch_proof* proofs,
                                       size_t n_proofs, const b200_batch_link* links, size_t n_links, const uint64_t g2_h[16],
                                       const uint64_t g2_tau_h[16], int* accepted, uint8_t* item_accepted,
                                       uint64_t* operands, size_t* pairing_products) {
    B200_TRY
    const size_t n = n_proofs + n_links;
    if (!ctx || !g2_h || !g2_tau_h || !accepted || n == 0 || (n_vks && !vks) || (n_proofs && !proofs) || (n_links && !links))
        return B200_ERR_INVALID;
    for (size_t v = 0; v < n_vks; ++v)
        if (!vks[v].k || !vks[v].selector_comms || !vks[v].sigma_comms || vks[v].log_n > 28) return B200_ERR_INVALID;
    size_t n_pi = 0, tr_bytes = 0;
    for (size_t j = 0; j < n_proofs; ++j) {
        const b200_batch_proof& p = proofs[j];
        if (p.vk >= n_vks || !p.proof || (p.num_inputs && !p.pub_inputs)) return B200_ERR_INVALID;
        if (p.num_inputs == vks[p.vk].num_inputs) {
            n_pi += p.num_inputs;
            tr_bytes += plonk_transcript_bytes(p.num_inputs);
        }
    }
    for (size_t l = 0; l < n_links; ++l)
        if (!links[l].comm1 || !links[l].comm2 || !links[l].proof || links[l].alignment > 28 || links[l].size == 0)
            return B200_ERR_INVALID;
    BatchRun run;
    run.qs[0] = g2_load(g2_tau_h);
    run.qs[1] = g2_load(g2_h);
    if (!g2_on_curve(run.qs[0]) || !g2_on_curve(run.qs[1])) {
        set_error("batch_verify: G2 point not on curve");
        return B200_ERR_NOT_ON_CURVE;
    }
    *accepted = 0;
    if (pairing_products) *pairing_products = 0;

    Context& c = ctx->c;
    std::lock_guard<std::mutex> lk(c.mu);
    B200_CUDA(cudaSetDevice(c.device));
    run.c = &c;
    // ---- one staging buffer in, one device workspace ------------------------------------------------------------
    const size_t o_vk = 0, o_pr = align_up(o_vk + n_vks * sizeof(BvVk)), o_ln = align_up(o_pr + n_proofs * sizeof(BvProof)),
                 o_pi = align_up(o_ln + n_links * sizeof(BvLink)), o_rt = align_up(o_pi + n_pi * sizeof(fe)),
                 in_bytes = align_up(o_rt + 29 * sizeof(fe));
    const size_t o_tr = in_bytes, o_terms = align_up(o_tr + tr_bytes), o_st = align_up(o_terms + n * sizeof(OperandTerms)),
                 o_valid = align_up(o_st + 64 * n), o_ops = align_up(o_valid + n), o_wa = align_up(o_ops + n * sizeof(Operands)),
                 o_wb = align_up(o_wa + n * sizeof(g1_xyzz)), o_pa = align_up(o_wb + n * sizeof(g1_xyzz)),
                 o_pb = align_up(o_pa + (n + 1) * sizeof(g1_xyzz)), o_rng = align_up(o_pb + (n + 1) * sizeof(g1_xyzz)),
                 dev_bytes = o_rng + sizeof(Operands);
    // pinned: the inputs, then what comes back (states + valid flags, operands, one range's operands)
    const size_t h_st = align_up(in_bytes), h_valid = h_st + 64 * n, h_ops = align_up(h_valid + n),
                 h_rng = align_up(h_ops + n * sizeof(Operands)), host_bytes = h_rng + sizeof(Operands);
    int rc = c.bv_dev.reserve(dev_bytes);
    if (rc != B200_OK) return rc;
    rc = c.bv_host.reserve(host_bytes);
    if (rc != B200_OK) return rc;
    uint8_t* hb = static_cast<uint8_t*>(c.bv_host.p);
    uint8_t* db = static_cast<uint8_t*>(c.bv_dev.p);
    BvVk* hv = reinterpret_cast<BvVk*>(hb + o_vk);
    for (size_t v = 0; v < n_vks; ++v) {
        std::memcpy(hv[v].k, vks[v].k, sizeof(hv[v].k));
        std::memcpy(hv[v].sel, vks[v].selector_comms, sizeof(hv[v].sel));
        std::memcpy(hv[v].sig, vks[v].sigma_comms, sizeof(hv[v].sig));
        hv[v].num_inputs = vks[v].num_inputs;
        hv[v].log_n = vks[v].log_n;
        hv[v].pad = 0;
    }
    BvProof* hp = reinterpret_cast<BvProof*>(hb + o_pr);
    fe* hpi = reinterpret_cast<fe*>(hb + o_pi);
    size_t pi_at = 0, tr_at = 0;
    for (size_t j = 0; j < n_proofs; ++j) {
        const b200_batch_proof& p = proofs[j];
        std::memcpy(&hp[j].proof, p.proof, sizeof(ProofIn));
        hp[j].vk = p.vk;
        hp[j].count_ok = p.num_inputs == vks[p.vk].num_inputs;  // else a rejection, as PlonkKzgSnark::verify
        hp[j].pi_off = pi_at;
        hp[j].tr_off = tr_at;
        if (hp[j].count_ok) {
            if (p.num_inputs) std::memcpy(hpi + pi_at, p.pub_inputs, p.num_inputs * sizeof(fe));
            pi_at += p.num_inputs;
            tr_at += plonk_transcript_bytes(p.num_inputs);
        }
    }
    BvLink* hl = reinterpret_cast<BvLink*>(hb + o_ln);
    for (size_t l = 0; l < n_links; ++l) {
        std::memcpy(&hl[l].c1, links[l].comm1, 64);
        std::memcpy(&hl[l].c2, links[l].comm2, 64);
        std::memcpy(&hl[l].cq, links[l].proof->quotient_commitment, 64);
        std::memcpy(&hl[l].op, links[l].proof->opening_proof, 64);
        hl[l].offset = links[l].offset;
        hl[l].size = links[l].size;
        hl[l].alignment = links[l].alignment;
        hl[l].pad = 0;
    }
    fe* hroots = reinterpret_cast<fe*>(hb + o_rt);
    for (unsigned k = 0; k <= 28; ++k) hroots[k] = host_root_of_unity(k);

    OperandTerms* d_terms = reinterpret_cast<OperandTerms*>(db + o_terms);
    Operands* d_ops = reinterpret_cast<Operands*>(db + o_ops);
    g1_xyzz* d_wa = reinterpret_cast<g1_xyzz*>(db + o_wa);
    g1_xyzz* d_wb = reinterpret_cast<g1_xyzz*>(db + o_wb);
    run.pa = reinterpret_cast<g1_xyzz*>(db + o_pa);
    run.pb = reinterpret_cast<g1_xyzz*>(db + o_pb);
    run.d_range = reinterpret_cast<Operands*>(db + o_rng);
    run.h_range = reinterpret_cast<Operands*>(hb + h_rng);
    cudaStream_t st = c.stream;
    B200_CUDA(cudaMemcpyAsync(db, hb, in_bytes, cudaMemcpyHostToDevice, st));
    const unsigned item_blocks = (unsigned)((n + kItemThreads - 1) / kItemThreads);
    B200_LAUNCH(bv_items_kernel, item_blocks, kItemThreads, 0, st)(
        reinterpret_cast<const BvVk*>(db + o_vk), reinterpret_cast<const BvProof*>(db + o_pr), n_proofs,
        reinterpret_cast<const BvLink*>(db + o_ln), n_links, reinterpret_cast<const fe*>(db + o_pi),
        reinterpret_cast<const fe*>(db + o_rt), db + o_tr, d_terms, db + o_st, db + o_valid);
    B200_CUDA(cudaGetLastError());
    B200_CUDA(cudaMemcpyAsync(hb + h_st, db + o_st, 64 * n, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaMemcpyAsync(hb + h_valid, db + o_valid, n, cudaMemcpyDeviceToHost, st));
    cudaEvent_t items_done = nullptr;
    B200_CUDA(cudaEventCreateWithFlags(&items_done, cudaEventDisableTiming));
    struct EvGuard {
        cudaEvent_t e;
        ~EvGuard() { cudaEventDestroy(e); }
    } ev_guard{items_done};
    B200_CUDA(cudaEventRecord(items_done, st));
    B200_LAUNCH(bv_operands_kernel, (unsigned)n, kTermThreads, 0, st)(d_terms, d_ops);
    B200_CUDA(cudaGetLastError());
    // rho on the host while the operands are computed
    B200_CUDA(cudaEventSynchronize(items_done));
    const uint8_t* h_valid_p = hb + h_valid;
    const fe rho = batch_challenge(hb + h_st, n_proofs, links, n_links, g2_h, g2_tau_h);
    B200_LAUNCH(bv_weight_kernel, item_blocks, kItemThreads, 0, st)(d_ops, n, rho, d_wa, d_wb);
    B200_CUDA(cudaGetLastError());
    B200_LAUNCH(bv_scan_kernel, 1, kScanThreads, 0, st)(d_wa, d_wb, n, run.pa, run.pb);
    B200_CUDA(cudaGetLastError());
    if (operands) {
        B200_CUDA(cudaMemcpyAsync(hb + h_ops, d_ops, n * sizeof(Operands), cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        std::memcpy(operands, hb + h_ops, n * sizeof(Operands));
    }
    bool all_valid = true;
    for (size_t j = 0; j < n; ++j) all_valid = all_valid && h_valid_p[j];
    if (all_valid || item_accepted) {
        bool ok = false;
        rc = run.range_ok(0, n, &ok);
        if (rc != B200_OK) return rc;
        *accepted = ok && all_valid ? 1 : 0;
        if (item_accepted) {
            std::memset(item_accepted, 1, n);
            if (!ok) {
                rc = run.bisect(0, n, item_accepted);
                if (rc != B200_OK) return rc;
            }
            // a rejected item's operands are the identity, which passes any range: its verdict is its flag
            for (size_t j = 0; j < n; ++j) item_accepted[j] = item_accepted[j] && h_valid_p[j];
        }
    }
    if (pairing_products) *pairing_products = run.pairings;
    return B200_OK;
    B200_CATCH
}
