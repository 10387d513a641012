// Internal (C++) declarations shared by the CUDA translation units behind the C ABI in
// include/b200prover.h.  Nothing here is part of the public boundary.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cstddef>
#include <cstdint>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "ec.cuh"
#include "ff.cuh"

#include "b200prover.h"  // error codes

namespace b200 {

void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);  // records the message, returns B200_ERR_CUDA

#define B200_CUDA(expr)                                            \
    do {                                                           \
        cudaError_t _e = (expr);                                   \
        if (_e != cudaSuccess) return ::b200::cuda_fail(_e, #expr); \
    } while (0)

// Process-wide count of kernel launches made by the library (bench.py's `gpu_launches` is the difference of
// two reads around the timed region; b200_kernel_launches()).  A relaxed increment per launch.
extern std::atomic<uint64_t> g_kernel_launches;
extern std::atomic<uint64_t> g_launch_host_ns;
extern std::atomic<uint64_t> g_graph_launches;  // cudaGraphLaunch calls (a replayed prover round is one submission)
extern thread_local uint64_t t_kernel_launches; // this thread's launches (what a stream capture recorded)
// Counts the launch and the host time its submission took: the temporary lives until the end of the launch statement.
struct LaunchClock {
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    ~LaunchClock() {
        g_kernel_launches.fetch_add(1, std::memory_order_relaxed);
        ++t_kernel_launches;
        g_launch_host_ns.fetch_add((uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count(),
                                   std::memory_order_relaxed);
    }
};
#define B200_LAUNCH(kern, grid, block, smem, st) ::b200::LaunchClock(), kern<<<grid, block, smem, st>>>

// Grow-only device buffer
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return B200_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(DevBuf)");
        cap = bytes;
        return B200_OK;
    }
    ~DevBuf() {
        if (p) cudaFree(p);
    }
};

// Grow-only pinned host buffer (results the host reads right after a stream wait)
struct HostPinned {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return B200_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        if (bytes < 4096) bytes = 4096;
        cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocDefault);
        if (e != cudaSuccess) return cuda_fail(e, "cudaHostAlloc(HostPinned)");
        cap = bytes;
        return B200_OK;
    }
    ~HostPinned() {
        if (p) cudaFreeHost(p);
    }
};

// ---- NTT ------------------------------------------------------------------------------------
struct Domain {
    unsigned log_n = 0;
    fe* tw_fwd = nullptr;     // w^k,  k < n/2
    fe* tw_inv = nullptr;     // w^-k, k < n/2
    fe* coset_fwd = nullptr;  // g^i,  i < n
    fe* coset_inv = nullptr;  // g^-i * n^-1
    fe n_inv;                 // n^-1 (Montgomery)
    fe group_gen;             // w (Montgomery)
    ~Domain();
};
int domain_create(unsigned log_n, cudaStream_t st, Domain** out);
// out[i] = scale * base^i, i < n (device table, launched on st)
void fill_powers(fe* d_out, size_t n, fe base, fe scale, cudaStream_t st);
fe host_root_of_unity(unsigned log_n);
int ntt_device(const Domain* d, fe* data, fe* scratch, int inverse, int coset, unsigned batch,
               size_t stride, cudaStream_t st);

// ---- MSM ------------------------------------------------------------------------------------
struct MsmPlan {
    int c = 0;        // window bits (signed digits in [-2^(c-1), 2^(c-1)])
    int n_digits = 0; // W = ceil(255 / c)
    int n_phys = 0;   // physical bucket windows Wp
    int n_tables = 0; // F = ceil(W / Wp); table j holds 2^(c*Wp*j) * P
    int latency = 0;  // chosen for one MSM at a time (shortest dependent chains) rather than for throughput
};

extern std::atomic<uint64_t> g_object_ids;  // proving keys and base sets: never reused, what captured graphs are keyed by

struct Bases {
    uint64_t id = g_object_ids.fetch_add(1);
    size_t n = 0;
    MsmPlan plan;
    g1_affine* tables = nullptr;  // n_tables * n affine points, table-major
    ~Bases() {
        if (tables) cudaFree(tables);
    }
};

struct MsmScratch {
    DevBuf counts, offsets, cursor, entries, buckets, window_sums, scalars;
    DevBuf seg_offsets, seg_bucket, seg_sums, heavy, seg_order;
    DevBuf scan_state;  // ScanState header + tile status words of the single-pass scan (msm.cu)
    DevBuf tree;        // partial sums of the row / column reduction trees
    DevBuf bit_sums;    // per window, the c - 1 bit sums T_b of the weighted tail
    HostPinned h_sums;  // window sums land here (pinned), read by the host epilogue
    cudaEvent_t done_ev = nullptr;  // recorded after the D2H of the window sums
    // the MSM batch queued by msm_launch_batch and not yet collected by msm_finish_batch
    MsmPlan pending_plan;
    size_t pending_n = 0;
    unsigned pending_batch = 0;
    // optional per-phase device timing (CUDA events on the launching stream)
    bool timing = false;
    bool ev_init = false;
    cudaEvent_t ev[5] = {};
    float ms[4] = {0, 0, 0, 0};  // total, sort (count+scan+scatter), accumulate, reduce
    // running totals since timing was switched on: accumulate ms, (point, scalar) pairs, launches
    double tot_acc_ms = 0, tot_pairs = 0, tot_launches = 0;
    // the final weighted sum of each window's bit sums runs on the host (msm_finish_batch); false: msm_horner_kernel leaves the
    // window sums on the device (the multi-GPU path adds them there)
    bool host_horner = true;
    // set by a caller that captures / replays the launches as a CUDA graph: timing events become graph nodes, and the
    // caller records done_ev itself
    bool in_graph = false;
    // borrowed from the context: low-priority stream for the accumulation kernel (null: same stream)
    cudaStream_t hv_stream = nullptr;
    cudaEvent_t hv_fork = nullptr, hv_join = nullptr;
    ~MsmScratch() {
        if (ev_init)
            for (auto& e : ev) cudaEventDestroy(e);
        if (done_ev) cudaEventDestroy(done_ev);
    }
};

MsmPlan msm_choose_plan(size_t n, int c_override, size_t mem_budget_bytes);
int bases_create(const g1_affine* h_points, size_t n, int c_override, int check_on_curve,
                 cudaStream_t st, Bases** out);
int bases_create_device(const g1_affine* d_points, size_t n, int c_override, cudaStream_t st,
                        Bases** out);
// scalars on device (n x 32 B); result: XYZZ sums of the n_phys windows copied to host and
// combined there (Horner + one inversion).
int msm_device(const Bases* b, size_t base_off, const fe* d_scalars, size_t n, int montgomery,
               MsmScratch* s, cudaStream_t st, g1_affine* out, int* out_inf);
int msm_device_batch(const Bases* b, size_t base_off, const fe* d_scalars, size_t n, size_t stride,
                     unsigned batch, int montgomery, MsmScratch* s, cudaStream_t st, g1_affine* out,
                     int* out_inf);
// the two halves of msm_device_batch: enqueue only / wait + host epilogue (one batch pending per scratch)
int msm_launch_batch(const Bases* b, size_t base_off, const fe* d_scalars, size_t n, size_t stride,
                     unsigned batch, int montgomery, MsmScratch* s, cudaStream_t st);
int msm_finish_batch(MsmScratch* s, g1_affine* out, int* out_inf);
void msm_mark_pending(const Bases* b, size_t n, unsigned batch, MsmScratch* s);
void msm_collect_timing(MsmScratch* s, size_t n, unsigned batch);
// synthetic known-discrete-log bases P_i = a_i * G, a_i = SplitMix64-derived (SURVEY §8(d))
int g1_known_dlog_bases_device(uint64_t seed, size_t first, size_t n, g1_affine* d_out,
                               cudaStream_t st);
int splitmix_fr_device(uint64_t seed, size_t first, size_t n, int montgomery, fe* d_out,
                       cudaStream_t st);

// ---- prover rounds as CUDA graphs -----------------------------------------------------------------
// One set per (context, proving key): the launches of each prover segment, captured on the second proof of that key
// on that context (the first sizes every buffer) and replayed afterwards.  Stale when a buffer of the context moved
// (`buffers`: a fingerprint of the addresses the launches refer to).
constexpr int kProofSegs = 7;
struct ProofGraphSet {
    uint64_t key = 0, sub[6] = {}, buffers = 0, last_use = 0;  // proofs: key = the proving key's id; link proofs: see link()
    unsigned proofs_seen = 0;
    bool timing = false;  // captured with the MSM's timing events as graph nodes
    cudaGraphExec_t exec[kProofSegs] = {};
    uint64_t kernels[kProofSegs] = {};
    ~ProofGraphSet() {
        for (auto& e : exec)
            if (e) cudaGraphExecDestroy(e);
    }
};

// ---- context --------------------------------------------------------------------------------
struct Context {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::mutex mu;  // one call at a time per context; callers may hold several contexts
    std::map<unsigned, Domain*> domains;
    DevBuf ntt_data, ntt_scratch;
    cudaEvent_t ntt_ev[2] = {};
    bool ntt_ev_init = false;
    float ntt_last_ms = 0.f;  // device time of the last b200_ntt_device call (CUDA events)
    MsmScratch msm;
    DevBuf plonk_ws;  // prover workspace (plonk.cu)
    float plonk_ms[8] = {0};  // wall time of the last proof's phases
    cudaStream_t stream2 = nullptr;  // side stream of the prover (challenge-independent coset NTTs)
    // lowest-priority companion of `stream` for the long throughput-bound kernels (null: priorities off)
    cudaStream_t heavy = nullptr;
    cudaEvent_t hv_fork = nullptr, hv_join = nullptr;
    bool heavy_plonk = false;  // also route the prover's NTT passes and quotient kernel there
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    DevBuf ntt_scratch2;
    HostPinned h_small;  // pinned landing zone of the prover's small read-backs (degree flag, evaluations)
    // per-proof scalars of the prover (plonk.cu ProofParams): pinned staging copy and the device copy the kernels read
    HostPinned h_params;
    DevBuf d_params;
    int use_graphs = -1;  // 1 / 0: replay prover rounds as CUDA graphs or not; -1: B200_GRAPHS from the environment (default on)
    std::vector<ProofGraphSet*> graph_sets;
    uint64_t graph_clock = 0;
    // batch verifier (batch_verify.cu): device workspace and the pinned staging of its inputs and results
    DevBuf bv_dev;
    HostPinned bv_host;
    // collaborative prover (mpc.cu): device workspace, the pinned outgoing message and the P received ones (read by the
    // kernels through their mapped addresses), and the last call's {exchanges, bytes sent, triples used, ms in all_gather}
    DevBuf mpc_ws;
    HostPinned mpc_send, mpc_recv;
    double mpc_stats[4] = {0, 0, 0, 0};
    ~Context();
};

int get_domain(Context* c, unsigned log_n, Domain** out);

}  // namespace b200

// opaque handle types of the C ABI
struct b200_ctx {
    b200::Context c;
};
struct b200_bases {
    b200::Bases* b;
};

#define B200_TRY try {
#define B200_CATCH                                               \
    }                                                            \
    catch (const std::bad_alloc&) {                              \
        ::b200::set_error("out of host memory");                 \
        return B200_ERR_NOMEM;                                   \
    }                                                            \
    catch (const std::exception& e) {                            \
        ::b200::set_error(std::string("exception: ") + e.what()); \
        return B200_ERR_INVALID;                                 \
    }                                                            \
    catch (...) {                                                \
        ::b200::set_error("unknown exception");                  \
        return B200_ERR_INVALID;                                 \
    }
