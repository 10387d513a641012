// TurboPlonk / KZG prover rounds on the device.
//
// Replaces what the reference calls at
//   /root/reference/crates/circuits/circuit-types/src/traits.rs:850
//       PlonkKzgSnark::<Bn254>::preprocess(&SYSTEM_SRS, &cs)            -> b200_plonk_preprocess
//   /root/reference/crates/circuits/circuit-types/src/traits.rs:996
//       PlonkKzgSnark::prove_with_link_hint::<_, _, SolidityTranscript> -> b200_plonk_prove
// (the algorithm is mpc-jellyfish's TurboPlonk prover, restated in SURVEY.md App. A: 5 wire
// columns, 13 selectors, quotient over the 8n coset, 5-way split, Keccak transcript).
//
// B200-first layout: everything a proof needs that does not depend on the witness is resident in
// HBM per proving key — selector/sigma coefficients, sigma evaluations, and the 18 coset
// evaluation vectors over the 8n domain (302 MB at n = 2^16; 180 GB of HBM holds hundreds of
// keys) — so a proof runs 7 size-8n coset NTTs instead of the reference's 25.  Polynomials never
// leave the device between rounds; the host sees 13 commitments and 10 evaluations and runs the
// (serial, few-KB) Keccak transcript between rounds.
#include <algorithm>
#include <chrono>
#include <cstring>
#include <vector>

#include "b200prover.h"
#include "device_ctx.h"
#include "plonk_internal.cuh"
#include "transcript.h"

namespace b200 {

static int preprocess(Context* c, const Bases* srs, unsigned log_n, size_t num_inputs, const fe* h_selectors,
                      const uint64_t* h_perm, const fe* h_k, ProvingKey** out) {
    const size_t n = (size_t)1 << log_n;
    // 6 cosets (6n > 5n + 7 points) from n = 16 on; all 8 for the tiny domains, where 6n would not exceed
    // the quotient's degree by enough to keep the degree check meaningful
    const int nc = log_n >= 4 ? 6 : 8;
    const size_t m = (size_t)nc * n;
    if (log_n < 2 || log_n + 3 > 28) {
        set_error("preprocess: log_n out of range");
        return B200_ERR_INVALID;
    }
    if (srs->n < n + 3) {
        set_error("preprocess: SRS shorter than n + 3 (MAX_SRS_DEGREE rule, srs.rs:44-47)");
        return B200_ERR_INVALID;
    }
    if (num_inputs > n) return B200_ERR_INVALID;
    cudaStream_t st = c->stream;
    ProvingKey* pk = new ProvingKey();
    pk->log_n = log_n;
    pk->n = n;
    pk->m = m;
    pk->nc = nc;
    pk->num_inputs = num_inputs;
    pk->srs = srs;
    for (int i = 0; i < NW; ++i) pk->k.v[i] = h_k[i];
    int rc;
    Domain* dn = nullptr;
    if ((rc = get_domain(c, log_n, &dn)) != B200_OK) {
        delete pk;
        return rc;
    }
    pk->group_gen = dn->group_gen;
    uint64_t* d_perm = nullptr;
    auto fail = [&](int code) {
        if (d_perm) cudaFree(d_perm);
        delete pk;
        return code;
    };
    if ((rc = alloc_fe(&pk->sel_coeffs, NS * n)) || (rc = alloc_fe(&pk->sig_coeffs, NW * n)) ||
        (rc = alloc_fe(&pk->sig_evals, NW * n)) || (rc = alloc_fe(&pk->ce_sel, NS * m)) ||
        (rc = alloc_fe(&pk->ce_sig, NW * m)) || (rc = alloc_fe(&pk->dom, n)) || (rc = alloc_fe(&pk->coset_pts, m)) ||
        (rc = alloc_fe(&pk->l1_inv, m)) || (rc = alloc_fe(&pk->cscale, m)) || (rc = alloc_fe(&pk->cscale_inv, m)))
        return fail(rc);
    if (cudaMalloc(&d_perm, NW * n * 8) != cudaSuccess) return fail(B200_ERR_CUDA);
    if ((rc = c->ntt_scratch.reserve((size_t)NS * m * sizeof(fe))) != B200_OK) return fail(rc);
    fe* scratch = reinterpret_cast<fe*>(c->ntt_scratch.p);

    const fe one = fe_one<Fr>();
    const fe g = fe_from_u32<Fr>(5);
    fill_powers(pk->dom, n, dn->group_gen, one, st);
    {
        const fe w8n = host_root_of_unity(log_n + 3);
        fe vand[kMaxCosets * kMaxCosets];
        for (int j = 0; j < nc; ++j) {
            const fe sj = FMUL(g, host_pow(w8n, (uint64_t)j));  // s_j = g * w_8n^j
            const fe cj = host_pow(sj, n);                       // x^n on the whole coset
            pk->cc.cn[j] = cj;
            pk->zh_inv[j] = fe_inv<Fr>(FSUB(cj, one));
            fe pw = one;
            for (int k = 0; k < nc; ++k) {
                vand[j * nc + k] = pw;
                pw = FMUL(pw, cj);
            }
            fill_powers(pk->coset_pts + (size_t)j * n, n, dn->group_gen, sj, st);  // s_j * w_n^h
            fill_powers(pk->cscale + (size_t)j * n, n, sj, one, st);               // s_j^i
            fill_powers(pk->cscale_inv + (size_t)j * n, n, fe_inv<Fr>(sj), one, st);
        }
        for (int j = nc; j < 8; ++j) {
            pk->cc.cn[j] = fe_zero();
            pk->zh_inv[j] = fe_zero();
        }
        if (!host_mat_inverse(vand, nc, pk->comb.minv)) {
            set_error("preprocess: singular coset Vandermonde matrix");
            return fail(B200_ERR_INVALID);
        }
    }
    B200_LAUNCH(k_l1_denominators, grid_for(m, 256), 256, 0, st)(pk->coset_pts, m, host_from_u64(n), pk->l1_inv);
    batch_inverse_enqueue(nullptr, pk->l1_inv, pk->ce_sel /*scratch, overwritten below*/, m, st);

    // selectors: evaluations -> coefficients -> commitments
    cudaMemcpyAsync(pk->sel_coeffs, h_selectors, NS * n * sizeof(fe), cudaMemcpyHostToDevice, st);
    if ((rc = ntt_device(dn, pk->sel_coeffs, scratch, 1, 0, NS, n, st)) != B200_OK) return fail(rc);
    // sigmas: permutation -> evaluations (kept for the grand product) -> coefficients
    cudaMemcpyAsync(d_perm, h_perm, NW * n * 8, cudaMemcpyHostToDevice, st);
    B200_LAUNCH(k_sigma_evals, grid_for(NW * n, 256), 256, 0, st)(d_perm, pk->dom, n, pk->k, pk->sig_evals);
    cudaMemcpyAsync(pk->sig_coeffs, pk->sig_evals, NW * n * sizeof(fe), cudaMemcpyDeviceToDevice, st);
    if ((rc = ntt_device(dn, pk->sig_coeffs, scratch, 1, 0, NW, n, st)) != B200_OK) return fail(rc);
    // resident evaluations of the 18 fixed polynomials on the quotient domain
    if ((rc = coset_evals(pk, dn, pk->sel_coeffs, n, n, NS, pk->ce_sel, scratch, st)) != B200_OK) return fail(rc);
    if ((rc = coset_evals(pk, dn, pk->sig_coeffs, n, n, NW, pk->ce_sig, scratch, st)) != B200_OK) return fail(rc);
    if (cudaStreamSynchronize(st) != cudaSuccess) return fail(cuda_fail(cudaGetLastError(), "preprocess"));
    cudaFree(d_perm);
    d_perm = nullptr;
    // the 18 commitments of the verifying key
    if ((rc = commit_batch(c, pk, pk->sel_coeffs, n, n, NS, pk->sel_comms)) != B200_OK) return fail(rc);
    if ((rc = commit_batch(c, pk, pk->sig_coeffs, n, n, NW, pk->sig_comms)) != B200_OK) return fail(rc);
    *out = pk;
    return B200_OK;
}


// ---- prover rounds as CUDA graphs ---------------------------------------------------------------
// The launches of a proof depend on (context, key) only — every per-proof value travels through ProofParams — so each
// segment between two host synchronisations is captured once (second proof of a key on a context; the first runs
// eagerly and sizes every buffer) and replayed as ONE submission afterwards: ~90 kernel launches per proof become 7
// graph launches.  Same kernels, same order, same bytes out.
// the addresses a captured segment refers to besides the key's: every grow-only buffer of the context
static uint64_t buffer_fingerprint(const Context* c) {
    const MsmScratch& m = c->msm;
    const void* ps[] = {c->plonk_ws.p, c->ntt_scratch.p, c->ntt_scratch2.p, c->h_small.p, c->h_params.p, c->d_params.p,
                        m.counts.p, m.offsets.p, m.cursor.p, m.entries.p, m.buckets.p, m.window_sums.p, m.scalars.p,
                        m.seg_offsets.p, m.seg_bucket.p, m.seg_sums.p, m.heavy.p, m.seg_order.p, m.scan_state.p, m.tree.p,
                        m.bit_sums.p, m.h_sums.p};
    uint64_t h = 1469598103934665603ull;
    for (const void* p : ps) {
        h ^= (uint64_t)(uintptr_t)p;
        h *= 1099511628211ull;
    }
    return h;
}

static ProofGraphSet* graph_set_for(Context* c, uint64_t key, const uint64_t* sub = nullptr) {
    int on = c->use_graphs;
    if (on < 0) {
        static const bool env_on = [] {
            const char* e = std::getenv("B200_GRAPHS");
            return !(e && e[0] == '0');
        }();
        on = env_on ? 1 : 0;
    }
    if (!on) return nullptr;
    ProofGraphSet* gs = nullptr;
    const uint64_t no_sub[6] = {};
    if (!sub) sub = no_sub;
    for (ProofGraphSet* g : c->graph_sets)
        if (g->key == key && std::memcmp(g->sub, sub, sizeof(g->sub)) == 0) gs = g;
    if (!gs) {
        if (c->graph_sets.size() >= 32) {  // keys come and go: drop the least recently used set
            size_t lru = 0;
            for (size_t i = 1; i < c->graph_sets.size(); ++i)
                if (c->graph_sets[i]->last_use < c->graph_sets[lru]->last_use) lru = i;
            delete c->graph_sets[lru];
            c->graph_sets.erase(c->graph_sets.begin() + (long)lru);
        }
        gs = new ProofGraphSet();
        gs->key = key;
        std::memcpy(gs->sub, sub, sizeof(gs->sub));
        c->graph_sets.push_back(gs);
    }
    gs->last_use = ++c->graph_clock;
    const uint64_t buffers = buffer_fingerprint(c);
    if (gs->buffers != buffers || gs->timing != c->msm.timing) {  // a buffer moved since the capture (a larger key grew
                                                                  // it), or the MSM timing events were switched
        gs->timing = c->msm.timing;
        for (auto& e : gs->exec)
            if (e) {
                cudaGraphExecDestroy(e);
                e = nullptr;
            }
        gs->buffers = buffers;
    }
    return gs;
}

// Runs `fn` (which only enqueues work on `st` and on streams it forks from / joins back to `st`): directly when `gs`
// is null, else through the segment's graph, capturing it first if need be.
template <class F>
static int run_segment(ProofGraphSet* gs, int idx, cudaStream_t st, F&& fn) {
    if (!gs) return fn();
    if (!gs->exec[idx]) {
        const uint64_t k0 = t_kernel_launches;
        cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) return cuda_fail(e, "cudaStreamBeginCapture");
        const int rc = fn();
        cudaGraph_t graph = nullptr;
        e = cudaStreamEndCapture(st, &graph);
        if (rc != B200_OK || e != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            return rc != B200_OK ? rc : cuda_fail(e, "cudaStreamEndCapture");
        }
        e = cudaGraphInstantiate(&gs->exec[idx], graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) {
            gs->exec[idx] = nullptr;
            return cuda_fail(e, "cudaGraphInstantiate");
        }
        gs->kernels[idx] = t_kernel_launches - k0;
    } else {
        g_kernel_launches.fetch_add(gs->kernels[idx], std::memory_order_relaxed);  // the kernels this submission runs
    }
    const auto t0 = std::chrono::steady_clock::now();
    const cudaError_t e = cudaGraphLaunch(gs->exec[idx], st);
    g_launch_host_ns.fetch_add(
        (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count(),
        std::memory_order_relaxed);
    g_graph_launches.fetch_add(1, std::memory_order_relaxed);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGraphLaunch");
    return B200_OK;
}

// Enqueue `count` commitments as segment `idx` (after `before`'s launches), leaving the batch pending for commit_collect.
template <class F>
static int commit_enqueue(Context* c, const Bases* srs, ProofGraphSet* gs, int idx, const fe* d_coeffs, size_t len, size_t stride,
                          unsigned count, F&& before) {
    cudaStream_t st = c->stream;
    const int r = run_segment(gs, idx, st, [&]() -> int {
        const int r2 = before();
        if (r2 != B200_OK) return r2;
        return msm_launch_batch(srs, 0, d_coeffs, len, stride, count, /*montgomery=*/1, &c->msm, st);
    });
    if (r != B200_OK) return r;
    if (gs) {  // what msm_launch_batch leaves behind when it runs outside a capture
        msm_mark_pending(srs, len, count, &c->msm);
        B200_CUDA(cudaEventRecord(c->msm.done_ev, st));
    }
    return B200_OK;
}

static int commit_collect(Context* c, unsigned count, g1_affine* out) {
    int inf[32];
    if (count > 32) return B200_ERR_INVALID;
    const int rc = msm_finish_batch(&c->msm, out, inf);
    if (rc != B200_OK) return rc;
    for (unsigned i = 0; i < count; ++i)
        if (inf[i]) std::memset(&out[i], 0, sizeof(out[i]));
    return B200_OK;
}


static int prove(Context* c, const ProvingKey* pk, const fe* h_wires, const fe* h_pub_inputs, const fe* h_blinders,
                 ProofOut* proof, fe* h_link_poly, fe* h_challenges) {
    const size_t n = pk->n, m = pk->m;
    const unsigned log_n = pk->log_n;
    cudaStream_t st = c->stream;
    int rc;
    if ((rc = c->plonk_ws.reserve(workspace_elems(n) * sizeof(fe))) != B200_OK) return rc;
    if ((rc = c->ntt_scratch.reserve((size_t)7 * m * sizeof(fe))) != B200_OK) return rc;
    if ((rc = c->ntt_scratch2.reserve((size_t)6 * m * sizeof(fe))) != B200_OK) return rc;
    if ((rc = c->h_small.reserve(4096)) != B200_OK) return rc;
    if ((rc = c->h_params.reserve(sizeof(ProofParams))) != B200_OK) return rc;
    if ((rc = c->d_params.reserve(sizeof(ProofParams))) != B200_OK) return rc;
    if (!c->stream2) {
        int prio_least = 0, prio_greatest = 0;
        cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
        B200_CUDA(cudaStreamCreateWithPriority(&c->stream2, cudaStreamNonBlocking, c->heavy ? prio_least : 0));
        B200_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        B200_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
    }
    Workspace w = carve(reinterpret_cast<fe*>(c->plonk_ws.p), n);
    fe* nscr = reinterpret_cast<fe*>(c->ntt_scratch.p);
    const size_t S = w.S;
    Domain* dn = nullptr;
    if ((rc = get_domain(c, log_n, &dn)) != B200_OK) return rc;
    const fe one = fe_one<Fr>();

    // graphs: only once a proof of this key has run eagerly on this context (every buffer has its final size then)
    ProofGraphSet* gset = graph_set_for(c, pk->id);
    ProofGraphSet* gs = gset && gset->proofs_seen > 0 ? gset : nullptr;
    c->msm.in_graph = gs != nullptr;
    struct InGraphReset {
        MsmScratch& s;
        ~InGraphReset() { s.in_graph = false; }
    } in_graph_reset{c->msm};
    ProofParams* hp = reinterpret_cast<ProofParams*>(c->h_params.p);  // pinned staging copy
    ProofParams* dp = reinterpret_cast<ProofParams*>(c->d_params.p);  // what the kernels read
    // first operation of every segment that follows a host update of *hp
    auto push_params = [&]() -> int {
        B200_CUDA(cudaMemcpyAsync(dp, hp, sizeof(ProofParams), cudaMemcpyHostToDevice, st));
        return B200_OK;
    };
    auto commit_enqueue = [&](int idx, const fe* d_coeffs, size_t len, size_t stride, unsigned count, auto&& before) -> int {
        return b200::commit_enqueue(c, pk->srs, gs, idx, d_coeffs, len, stride, count, before);
    };
    auto nothing = []() -> int { return B200_OK; };

    using clk = std::chrono::steady_clock;
    auto t_prev = clk::now();
    int phase = 0;
    auto mark = [&]() {  // wall time between sync points (every commit synchronises the stream)
        const auto now = clk::now();
        if (phase < 8) c->plonk_ms[phase++] = std::chrono::duration<float, std::milli>(now - t_prev).count();
        t_prev = now;
    };
    SolidityTranscript tr;
    tr.append_u32_be(254);  // field size in bits
    tr.append_u64_be((uint64_t)n);
    tr.append_u64_be((uint64_t)pk->num_inputs);
    for (int i = 0; i < NW; ++i) tr.append_field_elem(pk->k.v[i]);
    for (int s = 0; s < NS; ++s) tr.append_commitment(pk->sel_comms[s]);
    for (int i = 0; i < NW; ++i) tr.append_commitment(pk->sig_comms[i]);
    for (size_t i = 0; i < pk->num_inputs; ++i) tr.append_field_elem(h_pub_inputs[i]);

    // ---- round 1 ------------------------------------------------------------------------------------
    // caller-owned buffers are copied outside the graphs (their addresses change from proof to proof)
    B200_CUDA(cudaMemcpyAsync(w.wires_ev, h_wires, NW * n * sizeof(fe), cudaMemcpyDefault, st));  // host or device pointer (UVA)
    B200_CUDA(cudaMemsetAsync(w.wpoly, 0, (NW + 1) * S * sizeof(fe), st));  // wire slots and the public-input slot behind them
    if (pk->num_inputs)
        B200_CUDA(cudaMemcpyAsync(w.pi_poly, h_pub_inputs, pk->num_inputs * sizeof(fe), cudaMemcpyHostToDevice, st));
    for (int i = 0; i < NW; ++i) {
        hp->blind_w[i][0] = h_blinders[2 * i];
        hp->blind_w[i][1] = h_blinders[2 * i + 1];
    }
    rc = run_segment(gs, 0, st, [&]() -> int {
        int r = push_params();
        if (r != B200_OK) return r;
        B200_CUDA(cudaMemcpy2DAsync(w.wpoly, S * sizeof(fe), w.wires_ev, n * sizeof(fe), n * sizeof(fe), NW,
                                    cudaMemcpyDeviceToDevice, st));
        {
            // wires and public inputs: evaluations -> coefficients, one batch of 6 (pi_poly sits directly behind wpoly)
            HeavyScope hv(c, st);
            if ((r = ntt_device(dn, w.wpoly, nscr, 1, 0, NW + 1, S, hv.run)) != B200_OK) return r;
        }
        B200_LAUNCH(k_blind_wires, 1, 32, 0, st)(w.wpoly, S, n, &dp->blind_w[0][0]);
        return B200_OK;
    });
    if (rc != B200_OK) return rc;
    // Fork: the coset evaluations of the 5 wire polynomials and of the public-input polynomial do not
    // depend on any challenge, so they run on a second stream underneath the round-1/2 commitments
    // (whose bucket reduction and host round trip leave most SMs idle).
    struct Side {
        Context* c;
        bool pending = false;
        ~Side() {
            if (pending) cudaStreamSynchronize(c->stream2);  // error paths: never leave the side stream running
        }
    } side{c};
    {
        cudaStream_t s2 = c->stream2;
        B200_CUDA(cudaEventRecord(c->ev_fork, st));
        B200_CUDA(cudaStreamWaitEvent(s2, c->ev_fork, 0));
        side.pending = true;
        // 5 wire polynomials (n + 2 coefficients) and the public-input polynomial (n, zero tail) in one batch
        rc = run_segment(gs, 1, s2, [&]() -> int {
            return coset_evals(pk, dn, w.wpoly, S, n + 2, NW + 1, w.ext, reinterpret_cast<fe*>(c->ntt_scratch2.p), s2);
        });
        if (rc != B200_OK) return rc;
        B200_CUDA(cudaEventRecord(c->ev_join, s2));
    }
    if ((rc = commit_enqueue(2, w.wpoly, n + 2, S, NW, nothing)) != B200_OK) return rc;
    if ((rc = commit_collect(c, NW, proof->wires_poly_comms)) != B200_OK) return rc;
    if (h_link_poly)  // completes under round 2; the stream is synchronised several times before this call returns
        B200_CUDA(cudaMemcpyAsync(h_link_poly, w.wpoly, (n + 2) * sizeof(fe), cudaMemcpyDeviceToHost, st));
    for (int i = 0; i < NW; ++i) tr.append_commitment(proof->wires_poly_comms[i]);
    mark();  // [0] round 1

    // ---- round 2 ------------------------------------------------------------------------------------
    const fe beta = tr.get_and_append_challenge();
    const fe gamma = tr.get_and_append_challenge();
    hp->chal[0] = beta;
    hp->chal[1] = gamma;
    for (int i = 0; i < 3; ++i) hp->blind_z[i] = h_blinders[10 + i];
    rc = commit_enqueue(3, w.zpoly, n + 3, n + 3, 1, [&]() -> int {
        int r = push_params();
        if (r != B200_OK) return r;
        B200_LAUNCH(k_perm_num_den, grid_for(n, 128), 128, 0, st)(w.wires_ev, pk->sig_evals, pk->dom, pk->k, &dp->chal[0], n, w.num, w.den);
        batch_inverse_enqueue(w.num, w.den, w.tmp, n, st);
        scan_mul_exclusive(w.den, n, w.scan, st);  // z(w^j) = prod_{i<j} ratio_i
        B200_CUDA(cudaMemsetAsync(w.zpoly, 0, S * sizeof(fe), st));
        B200_CUDA(cudaMemcpyAsync(w.zpoly, w.den, n * sizeof(fe), cudaMemcpyDeviceToDevice, st));
        if ((r = ntt_device(dn, w.zpoly, nscr, 1, 0, 1, S, st)) != B200_OK) return r;
        BlindArgs b{};
        b.count = 3;
        b.dyn = &dp->blind_z[0];
        B200_LAUNCH(k_blind, 1, 32, 0, st)(w.zpoly, n, b);
        return B200_OK;
    });
    if (rc != B200_OK) return rc;
    if ((rc = commit_collect(c, 1, &proof->prod_perm_poly_comm)) != B200_OK) return rc;
    tr.append_commitment(proof->prod_perm_poly_comm);
    mark();  // [1] round 2

    // ---- round 3 ------------------------------------------------------------------------------------
    const fe alpha = tr.get_and_append_challenge();
    hp->chal[2] = alpha;
    hp->chal[3] = fe_sqr<Fr>(alpha);
    for (int i = 0; i < 4; ++i) hp->blind_q[i] = h_blinders[13 + i];
    B200_CUDA(cudaStreamWaitEvent(st, c->ev_join, 0));  // join: wire / PI coset evaluations are ready
    side.pending = false;
    const size_t deg = NW * (n + 1) + 2;
    uint32_t* h_flag = reinterpret_cast<uint32_t*>(c->h_small.p);  // pinned; read after the commitments below are in
    mark();  // [2] round 3 (host part)
    // the last chunk has n coefficients; its tail up to n + 3 is zero, so one batch length serves
    rc = commit_enqueue(4, w.split, n + 3, S, NW, [&]() -> int {
        int r = push_params();
        if (r != B200_OK) return r;
        {
            HeavyScope hv(c, st);
            if ((r = coset_evals(pk, dn, w.zpoly, S, n + 3, 1, w.ext + 6 * m, nscr, hv.run)) != B200_OK) return r;
        }
        {
            QuotArgs q;
            q.sel = pk->ce_sel;
            q.sig = pk->ce_sig;
            q.ext = w.ext;
            q.pts = pk->coset_pts;
            q.l1_inv = pk->l1_inv;
            q.out = w.quot;
            q.m = m;
            q.log_n = log_n;
            q.k = pk->k;
            q.chal = &dp->chal[0];
            for (int i = 0; i < 8; ++i) q.zh_inv[i] = pk->zh_inv[i];
            HeavyScope hv(c, st);
            B200_LAUNCH(k_quotient, grid_for(m, 128), 128, 0, hv.run)(q);
            // back to coefficients: nc size-n inverse transforms, then un-scale and un-mix the cosets
            if ((r = ntt_device(dn, w.quot, nscr, 1, 0, (unsigned)pk->nc, n, hv.run)) != B200_OK) return r;
            if (pk->nc == 6) B200_LAUNCH(k_coset_combine<6>, grid_for(n, 128), 128, 0, hv.run)(w.quot, n, pk->cscale_inv, pk->comb);
            else B200_LAUNCH(k_coset_combine<8>, grid_for(n, 128), 128, 0, hv.run)(w.quot, n, pk->cscale_inv, pk->comb);
        }
        B200_CUDA(cudaMemsetAsync(w.flag, 0, 4, st));
        B200_LAUNCH(k_check_degree, grid_for(m - deg, 256), 256, 0, st)(w.quot, deg, m, w.flag);
        B200_CUDA(cudaMemcpyAsync(h_flag, w.flag, 4, cudaMemcpyDeviceToHost, st));
        B200_LAUNCH(k_split_quotient, dim3(grid_for(n + 3, 256), NW), 256, 0, st)(w.quot, n, S, &dp->blind_q[0], w.split);
        return B200_OK;
    });
    if (rc != B200_OK) return rc;
    if ((rc = commit_collect(c, NW, proof->split_quot_poly_comms)) != B200_OK) return rc;
    if (*h_flag) {  // copied before the commitments' window sums on the same stream
        set_error("WrongQuotientPolyDegree: the witness does not satisfy the circuit");
        return B200_ERR_UNSATISFIED;
    }
    for (int i = 0; i < NW; ++i) tr.append_commitment(proof->split_quot_poly_comms[i]);
    mark();  // [3] round 3: quotient and its 5 commitments

    // ---- round 4 ------------------------------------------------------------------------------------
    const fe zeta = tr.get_and_append_challenge();
    const fe zeta_w = FMUL(zeta, pk->group_gen);
    fe* h_evals = reinterpret_cast<fe*>(reinterpret_cast<char*>(c->h_small.p) + 64);  // pinned
    {
        const fe* polys[kMaxEval];
        size_t lens[kMaxEval];
        fe pts[kMaxEval];
        for (int i = 0; i < NW; ++i) { polys[i] = w.wpoly + (size_t)i * S; lens[i] = n + 2; pts[i] = zeta; }
        for (int i = 0; i < NW - 1; ++i) { polys[NW + i] = pk->sig_coeffs + (size_t)i * n; lens[NW + i] = n; pts[NW + i] = zeta; }
        polys[2 * NW - 1] = w.zpoly; lens[2 * NW - 1] = n + 3; pts[2 * NW - 1] = zeta_w;
        for (int q = 0; q < 2 * NW; ++q) {
            fe z = pts[q];
            for (int l = 0; l < kLevels; ++l) {
                hp->eval_z[l][q] = z;
                z = host_pow(z, CH);
            }
        }
        rc = run_segment(gs, 5, st, [&]() -> int {
            int r = push_params();
            if (r != B200_OK) return r;
            eval_batch(polys, lens, pts, 2 * NW, w.evals, w.escr, st, dp->eval_z);
            B200_CUDA(cudaMemcpyAsync(h_evals, w.evals, 2 * NW * sizeof(fe), cudaMemcpyDeviceToHost, st));
            return B200_OK;
        });
        if (rc != B200_OK) return rc;
    }
    B200_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < NW; ++i) proof->wires_evals[i] = h_evals[i];
    for (int i = 0; i < NW - 1; ++i) proof->wire_sigma_evals[i] = h_evals[NW + i];
    proof->perm_next_eval = h_evals[2 * NW - 1];
    for (int i = 0; i < NW; ++i) tr.append_field_elem(proof->wires_evals[i]);
    for (int i = 0; i < NW - 1; ++i) tr.append_field_elem(proof->wire_sigma_evals[i]);
    tr.append_field_elem(proof->perm_next_eval);
    mark();  // [4] round 4

    // ---- round 5 ------------------------------------------------------------------------------------
    const fe v = tr.get_and_append_challenge();
    LinArgs la{};
    {
        const fe* we = proof->wires_evals;
        const fe* se = proof->wire_sigma_evals;
        int t = 0;
        auto push = [&](const fe* p, size_t len, const fe& s) {  // pointers and lengths: launch arguments; scalars: ProofParams
            la.p[t] = p;
            la.len[t] = (uint32_t)len;
            hp->lin_s[t] = s;
            ++t;
        };
        auto pow5 = [&](const fe& x) { return FMUL(fe_sqr<Fr>(fe_sqr<Fr>(x)), x); };
        const fe* sel = pk->sel_coeffs;
        for (int j = 0; j < 4; ++j) push(sel + (size_t)j * n, n, we[j]);
        push(sel + 4 * n, n, FMUL(we[0], we[1]));
        push(sel + 5 * n, n, FMUL(we[2], we[3]));
        for (int j = 0; j < 4; ++j) push(sel + (size_t)(6 + j) * n, n, pow5(we[j]));
        push(sel + 10 * n, n, fe_neg<Fr>(we[4]));
        push(sel + 11 * n, n, one);
        push(sel + 12 * n, n, FMUL(FMUL(FMUL(we[0], we[1]), FMUL(we[2], we[3])), we[4]));
        // z(X): alpha prod(w_i + beta k_i zeta + gamma) + alpha^2 L1(zeta)
        const fe vanish = FSUB(host_pow(zeta, n), one);
        const fe l1 = FMUL(vanish, fe_inv<Fr>(FMUL(host_from_u64(n), FSUB(zeta, one))));
        fe cz = alpha;
        for (int j = 0; j < NW; ++j) cz = FMUL(cz, FADD(FADD(we[j], FMUL(FMUL(pk->k.v[j], zeta), beta)), gamma));
        cz = FADD(cz, FMUL(fe_sqr<Fr>(alpha), l1));
        push(w.zpoly, n + 3, cz);
        // sigma_4(X): -alpha beta z(zeta w) prod_{i<4}(w_i + beta sigma_i + gamma)
        fe cs = FMUL(FMUL(alpha, beta), proof->perm_next_eval);
        for (int j = 0; j < NW - 1; ++j) cs = FMUL(cs, FADD(FADD(we[j], FMUL(beta, se[j])), gamma));
        push(pk->sig_coeffs + (size_t)(NW - 1) * n, n, fe_neg<Fr>(cs));
        // - Z_H(zeta) * sum zeta^((n+2) i) t_i(X)
        const fe zn2 = FMUL(FMUL(FADD(vanish, one), zeta), zeta);
        fe ct = fe_neg<Fr>(vanish);
        for (int i = 0; i < NW; ++i) {
            push(w.split + (size_t)i * S, i < NW - 1 ? n + 3 : n, ct);
            ct = FMUL(ct, zn2);
        }
        // batched opening at zeta: lin + v w_0 + ... + v^5 w_4 + v^6 sigma_0 + ... + v^9 sigma_3
        fe cv = one;
        for (int i = 0; i < NW; ++i) {
            cv = FMUL(cv, v);
            push(w.wpoly + (size_t)i * S, n + 2, cv);
        }
        for (int i = 0; i < NW - 1; ++i) {
            cv = FMUL(cv, v);
            push(pk->sig_coeffs + (size_t)i * n, n, cv);
        }
        la.count = t;
        la.dyn = &dp->lin_s[0];
    }
    fill_open_params(&hp->open[0], zeta);
    fill_open_params(&hp->open[1], zeta_w);
    g1_affine open2[2];
    rc = commit_enqueue(6, w.sdiv + 1, n + 2, S + 8, 2, [&]() -> int {
        int r = push_params();
        if (r != B200_OK) return r;
        B200_LAUNCH(k_lincomb, grid_for(n + 3, 128), 128, 0, st)(la, n + 3, w.lin);
        // opening proofs: commit((batch - batch(zeta)) / (X - zeta)) and commit((z - z(zeta w)) / (X - zeta w))
        horner_suffix(w.lin, n + 3, zeta, w.sdiv, w.evals + 16, w.hscr, st, &dp->open[0]);
        horner_suffix(w.zpoly, n + 3, zeta_w, w.sdiv + (S + 8), w.evals + 17, w.hscr, st, &dp->open[1]);
        return B200_OK;
    });
    if (rc != B200_OK) return rc;
    if ((rc = commit_collect(c, 2, open2)) != B200_OK) return rc;
    proof->opening_proof = open2[0];
    proof->shifted_opening_proof = open2[1];
    mark();  // [5] round 5
    if (gset && !gs) gset->proofs_seen = 1;  // this key has now run eagerly on this context: later proofs replay graphs
    if (h_challenges) {
        tr.append_commitment(proof->opening_proof);
        tr.append_commitment(proof->shifted_opening_proof);
        const fe u = tr.get_and_append_challenge();
        const fe all[6] = {beta, gamma, alpha, zeta, v, u};
        std::memcpy(h_challenges, all, sizeof(all));
    }
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------
// proof linking — replaces `PlonkKzgSnark::link_proofs::<SolidityTranscript>(hint_a, hint_b,
// &group_layout, &commit_key)` (circuits-core/src/zk_circuits/proof_linking/intent_only.rs:42-47,
// intent_and_balance.rs:66-72): q = (a1 - a2) / Z_D with Z_D = prod_{i<size} (X - g^(offset+i)),
// g the generator of the 2^alignment roots of unity (`GroupLayout`); eta from the transcript;
// opening of a1 - a2 - Z_D(eta) q at eta.  The reference divides by the `size` linear factors in turn; here the
// division runs on an evaluation domain (coset transform, pointwise division by Z_D, inverse transform): the same
// quotient, and an inexact division shows as a quotient of too high a degree.
// ---------------------------------------------------------------------------------------------
static int link(Context* c, const Bases* srs, const fe* h_a1, size_t len1, const fe* h_a2, size_t len2,
                const g1_affine& comm1, const g1_affine& comm2, unsigned alignment, size_t offset, size_t size,
                LinkOut* out, fe* h_eta) {
    const size_t len = len1 > len2 ? len1 : len2;
    if (size == 0 || size >= len || alignment > 28 || len > srs->n) {
        set_error("link: bad group layout or polynomial length");
        return B200_ERR_INVALID;
    }
    cudaStream_t st = c->stream;
    int rc;
    // Division by Z_D on an evaluation domain: N = 2^k >= len points of the coset g * H_N (Z_D has no root there).
    // diff / Z_D pointwise, back to coefficients: the quotient when the division is exact — and exact it is iff the
    // interpolant's degree is len - 1 - size (p * Z_D - diff has degree < N and vanishes on N points).  Two transforms,
    // one batch inversion and three element-wise kernels instead of `size` dependent synthetic divisions.
    unsigned log_N = 1;
    while (((size_t)1 << log_N) < len) ++log_N;
    if (log_N > 28) {
        set_error("link: polynomial too long");
        return B200_ERR_INVALID;
    }
    const size_t N = (size_t)1 << log_N;
    const size_t L = len + 8, NL = N + 8;
    const size_t scr = 4 * (L / CH + 4 * CH + 64);
    if ((rc = c->plonk_ws.reserve((5 * L + 3 * NL + scr + size + 16) * sizeof(fe))) != B200_OK) return rc;
    if ((rc = c->ntt_scratch.reserve(N * sizeof(fe))) != B200_OK) return rc;
    if ((rc = c->h_small.reserve(4096)) != B200_OK) return rc;
    if ((rc = c->h_params.reserve(sizeof(ProofParams))) != B200_OK) return rc;
    if ((rc = c->d_params.reserve(sizeof(ProofParams))) != B200_OK) return rc;
    Domain* dN = nullptr;
    if ((rc = get_domain(c, log_N, &dN)) != B200_OK) return rc;
    fe* base = reinterpret_cast<fe*>(c->plonk_ws.p);
    fe *d_a1 = base, *d_a2 = base + L, *d_diff = base + 2 * L, *d_ident = base + 3 * L, *d_open = base + 4 * L;
    fe *d_E = base + 5 * L, *d_Z = d_E + NL, *d_ZS = d_Z + NL;  // evaluations, Z_D on the coset, inversion scratch / quotient
    fe* hscr = d_ZS + NL;
    fe* d_roots = hscr + scr;    // the `size` roots of the group's vanishing polynomial
    fe* slot = d_roots + size;   // 16 spare elements: evaluation slot, then the exactness flag
    uint32_t* d_flag = reinterpret_cast<uint32_t*>(slot + 4);
    fe* nscr = reinterpret_cast<fe*>(c->ntt_scratch.p);
    uint32_t* h_flag = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(c->h_small.p) + 1024);
    // the launches depend on (context, SRS, lengths, layout) only: two graph segments, like the prover's rounds
    const uint64_t sub[6] = {srs->id, (uint64_t)len1, (uint64_t)len2, (uint64_t)alignment, (uint64_t)offset, (uint64_t)size};
    ProofGraphSet* gset = graph_set_for(c, ~(uint64_t)0, sub);
    ProofGraphSet* gs = gset && gset->proofs_seen > 0 ? gset : nullptr;
    c->msm.in_graph = gs != nullptr;
    struct InGraphReset {
        MsmScratch& s;
        ~InGraphReset() { s.in_graph = false; }
    } in_graph_reset{c->msm};
    LinkParams* hp = reinterpret_cast<LinkParams*>(c->h_params.p);
    LinkParams* dp = reinterpret_cast<LinkParams*>(c->d_params.p);
    static_assert(sizeof(LinkParams) <= sizeof(ProofParams), "one parameter block serves both");

    B200_CUDA(cudaMemcpyAsync(d_a1, h_a1, len1 * sizeof(fe), cudaMemcpyDefault, st));  // caller-owned: outside the graphs
    B200_CUDA(cudaMemcpyAsync(d_a2, h_a2, len2 * sizeof(fe), cudaMemcpyDefault, st));
    const fe one = fe_one<Fr>();
    // roots of the link group's vanishing polynomial: g_a^(offset + i), g_a the generator of the 2^alignment roots of unity
    const fe g = host_root_of_unity(alignment);
    std::vector<fe> roots(size);
    fe root = host_pow(g, (uint64_t)offset);
    const fe root0 = root;
    for (size_t i = 0; i < size; ++i) {
        roots[i] = root;
        root = FMUL(root, g);
    }
    fe* d_Q = d_ZS;  // the inversion's scratch is free again after it: quotient evaluations, then coefficients
    const size_t q_len = len - size;
    rc = commit_enqueue(c, srs, gs, 0, d_Q, q_len, q_len, 1, [&]() -> int {
        int r;
        B200_CUDA(cudaMemsetAsync(d_flag, 0, 4, st));
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
        if ((r = ntt_device(dN, d_E, nscr, /*inverse=*/0, /*coset=*/1, 1, N, st)) != B200_OK) return r;
        B200_LAUNCH(k_vanishing_on_coset, grid_for(N, 128), 128, 0, st)(dN->tw_fwd, N, fe_from_u32<Fr>(5), d_roots, size, d_Z);
        batch_inverse_enqueue(nullptr, d_Z, d_ZS, N, st);
        B200_LAUNCH(k_fr_vec_op, grid_for(N, 256), 256, 0, st)(2, d_E, d_Z, 0, N, d_Q);
        if ((r = ntt_device(dN, d_Q, nscr, /*inverse=*/1, /*coset=*/1, 1, N, st)) != B200_OK) return r;
        // a1 and a2 must agree on every root of the group, i.e. the division is exact: otherwise no link proof verifies
        // and the reference's prover output would be rejected (ADVICE r1: silent bad proof)
        B200_LAUNCH(k_any_nonzero, 1, 256, 0, st)(d_Q + q_len, N - q_len, d_flag);
        B200_CUDA(cudaMemcpyAsync(h_flag, d_flag, 4, cudaMemcpyDeviceToHost, st));
        return B200_OK;
    });
    if (rc != B200_OK) return rc;
    if ((rc = commit_collect(c, 1, &out->quotient_commitment)) != B200_OK) return rc;
    if (*h_flag) {
        set_error("link: the two wire polynomials differ on the link group (wrong layout or mismatched witnesses)");
        return B200_ERR_UNSATISFIED;
    }
    SolidityTranscript tr;
    tr.append_commitment(comm1);
    tr.append_commitment(comm2);
    tr.append_commitment(out->quotient_commitment);
    const fe eta = tr.get_and_append_challenge();
    if (h_eta) *h_eta = eta;
    fe zd = one;
    for (size_t i = 0; i < size; ++i) zd = FMUL(zd, FSUB(eta, roots[i]));
    hp->lin_s[0] = one;
    hp->lin_s[1] = fe_neg<Fr>(zd);
    fill_open_params(&hp->open, eta);
    rc = commit_enqueue(c, srs, gs, 1, d_open + 1, len - 1, len - 1, 1, [&]() -> int {
        B200_CUDA(cudaMemcpyAsync(dp, hp, sizeof(LinkParams), cudaMemcpyHostToDevice, st));
        LinArgs a{};
        a.count = 2;
        a.p[0] = d_diff; a.len[0] = (uint32_t)len;
        a.p[1] = d_Q; a.len[1] = (uint32_t)q_len;
        a.dyn = &dp->lin_s[0];
        B200_LAUNCH(k_lincomb, grid_for(len, 128), 128, 0, st)(a, len, d_ident);
        horner_suffix(d_ident, len, eta, d_open, slot, hscr, st, &dp->open);
        return B200_OK;
    });
    if (rc != B200_OK) return rc;
    if ((rc = commit_collect(c, 1, &out->opening_proof)) != B200_OK) return rc;
    if (gset && !gs) gset->proofs_seen = 1;
    return B200_OK;
}

}  // namespace b200

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
using namespace b200;

extern "C" {

int b200_plonk_preprocess(b200_ctx* ctx, const b200_bases* srs, unsigned log_n, size_t num_inputs,
                          const uint64_t* selectors_evals, const uint64_t* perm, const uint64_t* k, b200_pk** out) {
    B200_TRY
    if (!ctx || !srs || !selectors_evals || !perm || !k || !out) return B200_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    ProvingKey* pk = nullptr;
    int rc = preprocess(&ctx->c, srs->b, log_n, num_inputs, reinterpret_cast<const fe*>(selectors_evals), perm,
                        reinterpret_cast<const fe*>(k), &pk);
    if (rc != B200_OK) return rc;
    *out = new b200_pk{pk};
    return B200_OK;
    B200_CATCH
}

int b200_pk_verifying_key(const b200_pk* pk, uint64_t* selector_comms, uint64_t* sigma_comms) {
    if (!pk || !selector_comms || !sigma_comms) return B200_ERR_INVALID;
    std::memcpy(selector_comms, pk->pk->sel_comms, sizeof(pk->pk->sel_comms));
    std::memcpy(sigma_comms, pk->pk->sig_comms, sizeof(pk->pk->sig_comms));
    return B200_OK;
}

size_t b200_pk_num_inputs(const b200_pk* pk) { return pk ? pk->pk->num_inputs : 0; }
unsigned b200_pk_log_n(const b200_pk* pk) { return pk ? pk->pk->log_n : 0; }

int b200_plonk_link(b200_ctx* ctx, const b200_bases* srs, const uint64_t* a1, size_t len1, const uint64_t* a2,
                    size_t len2, const uint64_t* comm1, const uint64_t* comm2, unsigned alignment, size_t offset,
                    size_t size, b200_link_proof* proof, uint64_t* eta) {
    B200_TRY
    if (!ctx || !srs || !a1 || !a2 || !comm1 || !comm2 || !proof) return B200_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    g1_affine c1, c2;
    std::memcpy(&c1, comm1, 64);
    std::memcpy(&c2, comm2, 64);
    return link(&ctx->c, srs->b, reinterpret_cast<const fe*>(a1), len1, reinterpret_cast<const fe*>(a2), len2, c1, c2,
                alignment, offset, size, reinterpret_cast<LinkOut*>(proof), reinterpret_cast<fe*>(eta));
    B200_CATCH
}

int b200_plonk_last_timings(b200_ctx* ctx, float out_ms[8]) {
    if (!ctx || !out_ms) return B200_ERR_INVALID;
    for (int i = 0; i < 8; ++i) out_ms[i] = ctx->c.plonk_ms[i];
    return B200_OK;
}

void b200_pk_free(b200_ctx* ctx, b200_pk* pk) {
    if (!pk) return;
    if (ctx) {
        std::lock_guard<std::mutex> lk(ctx->c.mu);
        cudaSetDevice(ctx->c.device);
        cudaStreamSynchronize(ctx->c.stream);
        delete pk->pk;
    } else {
        delete pk->pk;
    }
    delete pk;
}

int b200_plonk_prove(b200_ctx* ctx, const b200_pk* pk, const uint64_t* wires, const uint64_t* pub_inputs,
                     const uint64_t* blinders, b200_proof* proof, uint64_t* link_poly, uint64_t* challenges) {
    B200_TRY
    if (!ctx || !pk || !wires || !blinders || !proof || (pk->pk->num_inputs && !pub_inputs)) return B200_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    return prove(&ctx->c, pk->pk, reinterpret_cast<const fe*>(wires), reinterpret_cast<const fe*>(pub_inputs),
                 reinterpret_cast<const fe*>(blinders), reinterpret_cast<ProofOut*>(proof),
                 reinterpret_cast<fe*>(link_poly), reinterpret_cast<fe*>(challenges));
    B200_CATCH
}


/* ---- device-vector primitives (collaborative prover) ---------------------------------------------------------- */
int b200_fr_vec_op(b200_ctx* ctx, int op, const void* d_a, const void* d_b, int b_is_scalar, size_t n, void* d_out) {
    B200_TRY
    if (!ctx || op < 0 || op > 2 || (n && (!d_a || !d_b || !d_out))) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    B200_LAUNCH(k_fr_vec_op, grid_for(n, 256), 256, 0, ctx->c.stream)(op, reinterpret_cast<const fe*>(d_a), reinterpret_cast<const fe*>(d_b),
                                                                     b_is_scalar, n, reinterpret_cast<fe*>(d_out));
    B200_CUDA(cudaGetLastError());
    B200_CUDA(cudaStreamSynchronize(ctx->c.stream));
    return B200_OK;
    B200_CATCH
}

int b200_fr_batch_inverse_device(b200_ctx* ctx, void* d_data, size_t n) {
    B200_TRY
    if (!ctx || (n && !d_data)) return B200_ERR_INVALID;
    if (n == 0) return B200_OK;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    int rc = ctx->c.ntt_scratch.reserve(n * sizeof(fe));
    if (rc != B200_OK) return rc;
    batch_inverse_enqueue(nullptr, reinterpret_cast<fe*>(d_data), reinterpret_cast<fe*>(ctx->c.ntt_scratch.p), n, ctx->c.stream);
    B200_CUDA(cudaGetLastError());
    B200_CUDA(cudaStreamSynchronize(ctx->c.stream));
    return B200_OK;
    B200_CATCH
}

int b200_fr_poly_eval_device(b200_ctx* ctx, const void* d_coeffs, size_t len, const uint64_t z[4], uint64_t out[4]) {
    B200_TRY
    if (!ctx || !z || !out || (len && !d_coeffs)) return B200_ERR_INVALID;
    if (len == 0) {
        std::memset(out, 0, 32);
        return B200_OK;
    }
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    int rc = ctx->c.plonk_ws.reserve((2 * (len / CH + len / CH / CH) + 4 * CH + 64) * sizeof(fe));
    if (rc != B200_OK) return rc;
    fe* scr = reinterpret_cast<fe*>(ctx->c.plonk_ws.p);
    fe zz;
    std::memcpy(&zz, z, 32);
    const fe* polys[1] = {reinterpret_cast<const fe*>(d_coeffs)};
    const size_t lens[1] = {len};
    eval_batch(polys, lens, &zz, 1, scr, scr + 8, ctx->c.stream);
    B200_CUDA(cudaMemcpyAsync(out, scr, 32, cudaMemcpyDeviceToHost, ctx->c.stream));
    B200_CUDA(cudaStreamSynchronize(ctx->c.stream));
    return B200_OK;
    B200_CATCH
}

int b200_fr_poly_div_linear_device(b200_ctx* ctx, const void* d_p, size_t len, const uint64_t z[4], void* d_q) {
    B200_TRY
    if (!ctx || !z || len < 2 || !d_p || !d_q) return B200_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    B200_CUDA(cudaSetDevice(ctx->c.device));
    const size_t L = len + 8;
    int rc = ctx->c.plonk_ws.reserve((L + 4 * (L / CH + 4 * CH + 64) + 16) * sizeof(fe));
    if (rc != B200_OK) return rc;
    fe* S = reinterpret_cast<fe*>(ctx->c.plonk_ws.p);
    fe* hscr = S + L;
    fe* slot = hscr + 4 * (L / CH + 4 * CH + 64);
    fe zz;
    std::memcpy(&zz, z, 32);
    horner_suffix(reinterpret_cast<const fe*>(d_p), len, zz, S, slot, hscr, ctx->c.stream);
    B200_CUDA(cudaMemcpyAsync(d_q, S + 1, (len - 1) * sizeof(fe), cudaMemcpyDeviceToDevice, ctx->c.stream));  // drop the remainder S[0]
    B200_CUDA(cudaStreamSynchronize(ctx->c.stream));
    return B200_OK;
    B200_CATCH
}

}  // extern "C"
