// libprmf_b200.so -- C ABI (include/prmf_b200.h) over the sm_100a kernels in kernels.cuh, block.cuh and tf32.cuh.
// Host orchestration of one PRMF inner step (reference prmf_runner.py:419-449).  Both passes over X are TMA X-stream
// launches: skinny_tma_kernel<k,kTmaRS,EPI> at k <= 10, skinny_tma_gen_kernel<KT,FG,kTmaRS> at k > 10 (their _f32_
// twins when X is stored in fp32, PRMF_X_F32), or tc_rowdot_kernel in tf32 mode.  The four DFMA kernels wrap one device
// body (skinny_tma_body, kernels.cuh) and one lookup picks among them (xstream_kernel).  step_path chooses which of
// the sequences below a block of steps runs (StepPath).
//
// k <= 10, fp64 (fused tails, launch_xv_epi / launch_xtu_epi):
//   skinny_tma_kernel<k,8,1>   A partials = Xt^T.V, then U <- U*A/(U.Gv+U) and Gu in the last CTA of each panel   (:420-422)
//   skinny_tma_kernel<k,8,2>   B partials = X^T.U_new, then V_new, Gv/VB partials                                 (:424-444)
//   objective_(parts|deferred)_kernel   recon/manifold/ignore/fro/obj, per step or once per block                 (:336-372)
//   sharded: the pass-2 tail packs (EPI 3) for ncclAllReduce or for the V-update kernel's NVLink pull; or the whole
//   block of steps runs as one persistent launch (block_kernel<K>, block.cuh)
//
// otherwise (k > 10, tf32 mode, PRMF_EPI=0, ranks without rows):
//   X-stream pass 1 (launch_xv)   A partials = Xt^T.V                                      (:420)
//   u_update_kernel               U <- U*A/(U.Gv+U), Gu partials                          (:421-422,:425)
//   X-stream pass 2 (launch_xtu)  B partials = X^T.U_new                                  (:424)
//   reduce_pack_kernel + ncclAllReduce          only when sharded
//   v_update_objective_kernel     V_new (double-buffered), Gv/VB partials, objective     (:425-444,:336-372,:542-548)
//   (k > 16: the tiled U / V updates, gram_reduce_kernel, manifold_parts_kernel and objective_kernel instead)
#include "../../include/prmf_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include "kernels.cuh"
#include "block_params.h"
#include "tf32.cuh"
#include "nccl_dyn.h"
#include "nnls_init.cuh"

using namespace prmf;

namespace {

thread_local std::string g_create_error;
NcclApi g_nccl;

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
};

// Cache of a handle's device allocations (X, its transposed copy, the arenas of the small state) across handles of one
// process: every cudaMalloc / cudaFree costs 10-100 ms on these boxes (multi-GB ones up to a second), which is most of
// the wall time of a short solve that creates and destroys a handle (random restarts, repeated solves of one
// instance).  A freed buffer is kept (bounded count and bytes) and handed to the next request of the same size on
// the same device.  PRMF_POOL=0 disables it; prmf_release_pool() returns everything to the driver.
struct BigPool {
    struct Ent { void* p; size_t bytes; int device; };
    std::vector<Ent> free_list;
    size_t held = 0;
    static constexpr size_t kMaxEntries = 16;
    static constexpr size_t kMaxBytes = (size_t)24 << 30;
    bool enabled() const { const char* e = getenv("PRMF_POOL"); return !(e && atoi(e) == 0); }
    cudaError_t alloc(void** out, size_t bytes, int device) {
        if (enabled())
            for (size_t i = 0; i < free_list.size(); ++i)
                if (free_list[i].bytes == bytes && free_list[i].device == device) {
                    *out = free_list[i].p;
                    held -= bytes;
                    free_list.erase(free_list.begin() + i);
                    return cudaSuccess;
                }
        return cudaMalloc(out, bytes);
    }
    void release(void* p, size_t bytes, int device) {
        if (!p) return;
        if (enabled() && free_list.size() < kMaxEntries && held + bytes <= kMaxBytes) {
            free_list.push_back({p, bytes, device});
            held += bytes;
            return;
        }
        cudaFree(p);
    }
    void drain() {
        for (auto& e : free_list) { cudaSetDevice(e.device); cudaFree(e.p); }
        free_list.clear();
        held = 0;
    }
};
BigPool g_pool;

// pinned host words (one per handle) for the error word read-back: one cudaHostAlloc per process
unsigned int* pinned_word() {
    static unsigned int* slab = nullptr;
    static int next = 0;
    if (!slab && cudaHostAlloc((void**)&slab, sizeof(unsigned int) * 1024, cudaHostAllocDefault) != cudaSuccess) { slab = nullptr; return nullptr; }
    unsigned int* w = slab + (next++ % 1024);
    *w = 0;
    return w;
}


}  // namespace

// Bump allocator over ONE cudaMalloc.  All small state of a handle lives in a few contiguous 2 MB pages: after
// 2 GB of X have streamed through, every first touch of a separately allocated small buffer is a TLB miss, and the
// latency-bound tail kernels pay for each of them in sequence.
struct Arena {
    unsigned char* base = nullptr;
    size_t cap = 0, used = 0;
    int device = 0;
    cudaError_t reserve(size_t bytes, int dev) {
        device = dev; used = 0;
        cudaError_t e = g_pool.alloc((void**)&base, bytes, dev);
        cap = e == cudaSuccess ? bytes : 0;
        if (e != cudaSuccess) base = nullptr;
        return e;
    }
    template <typename T>
    T* take(size_t count) {
        const size_t bytes = ((count ? count : 1) * sizeof(T) + 255) & ~(size_t)255;
        if (used + bytes > cap) return nullptr;
        T* p = reinterpret_cast<T*>(base + used);
        used += bytes;
        return p;
    }
    void release() { if (base) g_pool.release(base, cap, device); base = nullptr; cap = used = 0; }
};

struct prmf_handle {
    int device = 0;
    int sm_count = 148;
    int64_t m = 0, m_global = 0, n = 0;
    int k = 0;
    int64_t ldx = 0, ldxt = 0;
    int n2 = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;

    // device buffers (everything but X, Xt and the peer-exchange buffer comes out of the arenas)
    Arena arena, pw_arena, as_arena;
    double *X = nullptr, *Xt = nullptr;       // samples x genes, and its transposed copy genes x samples
    double *U = nullptr, *Vbuf[2] = {nullptr, nullptr}, *Ub = nullptr, *Vb = nullptr, *Gvb = nullptr;
    double* U2 = nullptr;                     // the other U buffer: the fused U update writes U_new there
    int vcur = 0;                             // Vbuf[vcur] is the current V
    double* Apart = nullptr;                  // pass-1 partials [chunks1][m][k]
    double *Gv = nullptr, *Gu_part = nullptr, *Gv_part = nullptr, *VB_part = nullptr;
    double* Bpart = nullptr;
    double* red = nullptr;
    double *normX_sq = nullptr, *scal_part = nullptr;
    double* gd = nullptr;
    double* obj = nullptr;
    int* step_counter = nullptr;
    int obj_capacity = 0;
    int32_t *active = nullptr, *pos = nullptr;
    double* scores_buf = nullptr;             // 3 x k x P tables of prmf_scores
    // flattened normalised Laplacians of the active pathways (objective)
    ActiveSet as{};
    int64_t as_cap_diag = 0, as_cap_off = 0;
    int32_t *as_i32 = nullptr;                // [diag_gene | diag_factor | off_r | off_c | off_factor]
    double* as_f64 = nullptr;                 // [diag_coef | off_coef]
    int64_t* as_off = nullptr;                // doff[k+1] | eoff[k+1] on the device
    std::vector<int64_t> row_ptr_host;
    bool have_X = false, have_U = false, have_V = false, have_pw = false, have_active = false, pos_dirty = true;
    std::vector<int32_t> active_host;

    // pathways
    Pathways pw{};
    int64_t S = 0, E = 0;
    int64_t max_support = 0, max_edges = 0;
    std::vector<int64_t> path_ptr_host;
    std::vector<int32_t> support_host;

    // launch geometry
    int uu_grid = 0, uu_rows = 0, vu_grid = 0, vu_rows = 0;
    int nq = 1, ni = 1;
    unsigned int* ticket = nullptr;
    prmf_xstream_plan plan{};                 // both X-stream passes (prmf_plan_xstream)

    // large k (> 16): register-tiled U update, Gram partials folded by gram_reduce_kernel, objective as its own launch
    bool big_k = false;
    double* mi_part = nullptr;                // manifold | ignore partials of manifold_parts_kernel (2 x 64)
    double* Gv_red = nullptr;                 // V_new^T V_new folded by gram_reduce_kernel (the objective publishes it to Gv)
    int tiled_cpt = 0, tiled_grid = 0;
    size_t tiled_smem = 0;

    // fused tails (k <= 10, TMA path): the U / V updates run in the last CTA of each panel of the X-stream kernels
    bool use_epi = false;
    unsigned long long* epi_counters = nullptr;   // arrive | done, each [pass-1 + pass-2 panels], monotone over launches
    unsigned long long epi_seq1 = 0, epi_seq2 = 0;
    // deferred objective: per-step history [obj_capacity] of what the objective needs (one cudaMalloc)
    double* hist = nullptr;
    size_t hist_bytes = 0;
    double *hist_Gu = nullptr, *hist_Gvp = nullptr, *hist_VBp = nullptr, *hist_vh = nullptr;
    bool defer_ok = false;
    double *epi_part2 = nullptr, *epi_vb2 = nullptr;

    // persistent step kernel (block.cuh): a whole block of inner steps per cooperative launch
    bool use_block = false;                   // this rank can take it (fused-tail geometry, deferred objective, smem fits)
    bool blk_xchg = false;                    // sharded: every rank takes it with the same geometry (prmf_p2p_finalize)
    bool block_forced = false;                // PRMF_BLOCK=1: also on one GPU
    unsigned long long* blk_ctr = nullptr;    // arrive1 | done1 | arrive2 | done2 | udone | vdone | ufold | vfold
    unsigned long long blk_n1 = 0, blk_n2 = 0, blk_xseq = 0;
    size_t blk_smem = 0;
    uint32_t blk_stage_bytes = 0;
    unsigned int* err_word = nullptr;         // device: set by a bounded wait that expired
    unsigned int* err_host = nullptr;         // pinned host copy read at the end of every block
    unsigned long long spin_timeout_ns = 10000000000ull;
    bool failed = false;                      // a launch failed or a device wait expired: no further steps
    double normX_sq_host = 0.0;               // ||X||^2 (all ranks), cached by prmf_set_X
    double* xbuf = nullptr;                   // push-exchange receive buffer inside p2p_buf
    double* xsmall = nullptr;                 // receive slots of the small all-reduce (set-up scalars without NCCL)
    unsigned long long small_seq = 0;
    size_t xcount = 0;

    // Storage of X and the engine of the two products are separate properties.  x32: X, X^T kept in fp32 (X32, Xt32)
    // instead of fp64 (X, Xt), in the tf32 mode (rounded to tf32) and the f32 mode (PRMF_X_F32, exact fp32 values).
    // x_tc: both passes on the tensor cores by tc_rowdot_kernel (tf32 mode); otherwise the DFMA X streams, which read
    // fp32 tiles in the f32 mode.  Everything else is the same in every mode.
    bool x32 = false, x_tc = false;
    float *X32 = nullptr, *Xt32 = nullptr, *Vt32 = nullptr, *Ut32 = nullptr;
    int64_t ldx32 = 0, ldxt32 = 0;
    int Kp = 0;
    CUtensorMap tm_X{}, tm_Xt{}, tm_Vt{}, tm_Ut{};
    TcParams tc1{}, tc2{};                    // pass 1: M = X (m x n), W = V^T; pass 2: M = X^T (n x m), W = U^T

    // multi-GPU
    NcclComm comm = nullptr;
    int rank = 0, nranks = 1;
    // NVLink peer exchange: [red parity 0 | red parity 1 | flags | ...] (layout: prmf_p2p_export)
    double* p2p_buf = nullptr;
    size_t p2p_red_count = 0;
    bool p2p_ready = false;
    void* peer_base[kMaxPeers] = {nullptr};
    unsigned long long p2p_seq = 0;
    int p2p_parity = 0;
    double* Gu_glob = nullptr;                // large k: U^T U summed over the U-update CTAs (and over ranks when sharded)

    // Speculative pass 1: the first X.V pass (+ U update on the fused-tail path) of the NEXT inner step does not
    // depend on the active pathways, so prmf_block_end enqueues it before the host waits for the score tables;
    // the GPU streams X while the host runs restrict / sampling.  0: nothing ahead; 1: A partials ready, U
    // untouched; 2: fused-tail path, h->U already holds U_new and h->U2 the current U.
    int ahead = 0;
    cudaEvent_t ev_sync = nullptr;

    // introspection
    int64_t launches = 0;
    bool profiling = false;
    std::vector<cudaEvent_t> ev_pool;
    std::vector<std::pair<int, int>> ev_pairs;   // (phase, pool index of start event; end = start + 1)
    double phase_ms[PRMF_N_PHASES] = {0, 0, 0, 0, 0, 0};
    int64_t phase_n[PRMF_N_PHASES] = {0, 0, 0, 0, 0, 0};
};

namespace {

int fail(prmf_handle* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(h, PRMF_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                  \
    } while (0)

#define LAUNCH_CHECK(name)                                                                    \
    do {                                                                                      \
        h->launches++;                                                                        \
        cudaError_t e_ = cudaGetLastError();                                                  \
        if (e_ != cudaSuccess)                                                                \
            return fail(h, PRMF_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e_)); \
    } while (0)

template <typename T>
int dalloc(prmf_handle* h, T** p, size_t count) {
    *p = nullptr;
    if (count == 0) count = 1;
    cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
    if (e != cudaSuccess)
        return fail(h, PRMF_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", count * sizeof(T), cudaGetErrorString(e));
    return PRMF_OK;
}

int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }

int pick_nq(int k) {
    int pairs = k * k;
    int q = (pairs + 255) / 256;
    if (q <= 1) return 1;
    if (q <= 4) return 4;
    if (q <= 16) return 16;
    return 64;
}

template <typename F>
int set_smem(prmf_handle* h, F kernel, size_t bytes) {
    // static shared memory counts against the 48 KB default too, so opt in with some margin
    if (bytes > 40 * 1024) CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return PRMF_OK;
}

// ---- X-stream launches -----------------------------------------------------------------------------
// One pass over X: out[chunk][j][0:k] = sum over the rows i of the chunk of M[i][j] * W[i][0:k]
struct XStream {
    const void* M;                            // fp32 when f32, else fp64
    bool f32;
    int64_t ldm, rows, cols;
    const double* W;
    double* out;                              // per-chunk partials
    const prmf_xstream_pass& p;
};

// pass 1: A partials = Xt^T . V   (M = Xt: n rows x m cols)
XStream pass1(const prmf_handle* h) {
    return {h->x32 ? (const void*)h->Xt32 : h->Xt, h->x32, h->x32 ? h->ldxt32 : h->ldxt, h->n, h->m, h->Vbuf[h->vcur],
            h->Apart, h->plan.pass1};
}

// pass 2: B partials = X^T . U_new   (M = X: m rows x n cols)
XStream pass2(const prmf_handle* h) {
    return {h->x32 ? (const void*)h->X32 : h->X, h->x32, h->x32 ? h->ldx32 : h->ldx, h->m, h->n, h->U, h->Bpart,
            h->plan.pass2};
}

// The X-stream kernel of a pass with fused tail `epi`, or nullptr: skinny_tma_kernel<k,kTmaRS,EPI> at k <= 10,
// skinny_tma_gen_kernel<KT,FG,kTmaRS> (no fused tail) at the plan's (KT, FG) above, or their _f32_ twins.  It
// instantiates exactly the kernels prmf_plan_xstream can select.  Call with K = 1: it recurses to K = k.
template <int K = 1>
const void* xstream_kernel(int k, const prmf_xstream_plan& plan, bool f32, int epi) {
    if constexpr (K <= 10) {
        if (k != K) return xstream_kernel<K + 1>(k, plan, f32, epi);
        switch (epi) {
            case 0: return f32 ? (const void*)skinny_tma_f32_kernel<K, kTmaRS, 0> : (const void*)skinny_tma_kernel<K, kTmaRS, 0>;
            case 1: return f32 ? (const void*)skinny_tma_f32_kernel<K, kTmaRS, 1> : (const void*)skinny_tma_kernel<K, kTmaRS, 1>;
            case 2: return f32 ? (const void*)skinny_tma_f32_kernel<K, kTmaRS, 2> : (const void*)skinny_tma_kernel<K, kTmaRS, 2>;
            // no pack on fp32 storage: the f32 mode is single-rank (prmf_p2p_attach), the tf32 mode uses tc_rowdot_kernel
            case 3: return f32 ? nullptr : (const void*)skinny_tma_kernel<K, kTmaRS, 3>;
        }
    } else if (epi == 0) {
#define GEN_CASE(KT_, FG_)                                                                                   \
        if (plan.kt == KT_ && plan.fg == FG_)                                                                \
            return f32 ? (const void*)skinny_tma_gen_f32_kernel<KT_, FG_, kTmaRS> : (const void*)skinny_tma_gen_kernel<KT_, FG_, kTmaRS>;
        GEN_CASE(12, 1) GEN_CASE(16, 1) GEN_CASE(12, 2) GEN_CASE(16, 2) GEN_CASE(12, 4) GEN_CASE(16, 4) GEN_CASE(12, 8)
        GEN_CASE(16, 8)
#undef GEN_CASE
    }
    return nullptr;
}

// every launch of a pass on a fused-tail handle requests the tail's shared memory
size_t pass_smem(const prmf_handle* h, const prmf_xstream_pass& p) { return h->use_epi ? p.tail_smem : p.ring_smem; }

// EpiParams of an X-stream launch without a fused tail; the fused-tail launchers fill in the rest
EpiParams plain_epi(const prmf_handle* h) {
    EpiParams ep{};
    ep.dbg_slot = -1;
    ep.err = h->err_word; ep.timeout_ns = h->spin_timeout_ns;
    return ep;
}

// Launches pass `x` with fused tail `epi` (0: none, 1: U update, 2: V update, 3: pack for the exchange over ranks).
// The storage of M, k and the plan choose the kernel once (xstream_kernel).  The CTAs of a panel with a fused tail wait
// for each other, so that launch is cooperative (all CTAs co-resident or the launch fails).
int launch_xstream(prmf_handle* h, const XStream& x, int epi, const EpiParams& ep_in) {
    const void* fn = xstream_kernel(h->k, h->plan, x.f32, epi);
    if (!fn)
        return fail(h, PRMF_ERR_STATE, "no X-stream kernel for k=%d (KT=%d FG=%d), fused tail %d, %s storage", h->k,
                    (int)h->plan.kt, (int)h->plan.fg, epi, x.f32 ? "fp32" : "fp64");
    const prmf_xstream_pass& p = x.p;
    EpiParams ep = ep_in;
    int k = h->k, panel_w = (int)p.panel_w, stages = (int)h->plan.stages;     // the kernels' parameter types
    void* args[] = {(void*)&x.M, (void*)&x.ldm, (void*)&x.rows, (void*)&x.cols, (void*)&x.W, (void*)&k, (void*)&panel_w,
                    (void*)&p.rows_per_chunk, (void*)&stages, (void*)&x.out, (void*)&ep};
    const dim3 grid(p.panels, p.chunks);
    const size_t smem = pass_smem(h, p);
    CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (epi != 0)
        CU(cudaLaunchCooperativeKernel(fn, grid, dim3(kTmaThreads), args, smem, h->stream));
    else   // as with <<<>>>, a failure is left for the caller's LAUNCH_CHECK
        cudaLaunchKernel(fn, grid, dim3(kTmaThreads), args, smem, h->stream);
    return PRMF_OK;
}

// number of per-chunk partials the passes leave in Apart / Bpart
int a_chunks(const prmf_handle* h) { return (int)(h->x_tc ? h->plan.tc_chunks1 : h->plan.pass1.chunks); }
int b_chunks(const prmf_handle* h) { return (int)(h->x_tc ? h->plan.tc_chunks2 : h->plan.pass2.chunks); }

// TF32 mode: one tensor-core kernel serves both passes
int launch_tc(prmf_handle* h, const CUtensorMap& tmM, const CUtensorMap& tmW, const TcParams& prm, int64_t tiles,
              int64_t chunks, const char* name) {
    dim3 grid(tiles, chunks);
    tc_rowdot_kernel<<<grid, kTcThreads, h->plan.tc_smem, h->stream>>>(tmM, tmW, prm);
    LAUNCH_CHECK(name);
    return PRMF_OK;
}

// W^T operand of the tensor-core passes: Wt[f][r] = tf32(W[r][f])
int refresh_wt(prmf_handle* h, const double* W, int64_t rows, float* Wt, int64_t ld) {
    if (rows == 0) return PRMF_OK;
    dim3 grid((unsigned)((rows + 31) / 32), (unsigned)((h->Kp + 31) / 32));
    cast_transpose_w_kernel<<<grid, 256, 0, h->stream>>>(W, rows, h->k, h->Kp, Wt, ld);
    LAUNCH_CHECK("cast_transpose_w_kernel");
    return PRMF_OK;
}

// pass 1 without a fused tail
int launch_xv(prmf_handle* h) {
    if (h->m == 0) return PRMF_OK;
    if (h->x_tc)
        return launch_tc(h, h->tm_X, h->tm_Vt, h->tc1, h->plan.tc_tiles1, h->plan.tc_chunks1, "tc_rowdot_kernel(pass 1)");
    int rc = launch_xstream(h, pass1(h), 0, plain_epi(h));
    if (rc) return rc;
    LAUNCH_CHECK("skinny_tma_kernel(pass 1)");
    return PRMF_OK;
}

// pass 2 without a fused tail
int launch_xtu(prmf_handle* h) {
    if (h->m == 0) {
        CU(cudaMemsetAsync(h->Bpart, 0, sizeof(double) * b_chunks(h) * h->n * h->k, h->stream));
        return PRMF_OK;
    }
    if (h->x_tc) {
        int rc = refresh_wt(h, h->U, h->m, h->Ut32, h->ldxt32);
        if (rc) return rc;
        return launch_tc(h, h->tm_Xt, h->tm_Ut, h->tc2, h->plan.tc_tiles2, h->plan.tc_chunks2, "tc_rowdot_kernel(pass 2)");
    }
    int rc = launch_xstream(h, pass2(h), 0, plain_epi(h));
    if (rc) return rc;
    LAUNCH_CHECK("skinny_tma_kernel(pass 2)");
    return PRMF_OK;
}

#define NQ_SWITCH(nq, EXPR)                    \
    switch (nq) {                              \
        case 1: { constexpr int NQ = 1; EXPR; } break;   \
        case 4: { constexpr int NQ = 4; EXPR; } break;   \
        case 16: { constexpr int NQ = 16; EXPR; } break; \
        default: { constexpr int NQ = 64; EXPR; } break; \
    }

#define NI_SWITCH(ni, EXPR)                    \
    switch (ni) {                              \
        case 1: { constexpr int NI = 1; EXPR; } break;   \
        case 2: { constexpr int NI = 2; EXPR; } break;   \
        case 4: { constexpr int NI = 4; EXPR; } break;   \
        case 8: { constexpr int NI = 8; EXPR; } break;   \
        default: { constexpr int NI = 16; EXPR; } break; \
    }

int pick_ni(int k) {
    const int items = k * k * gram_slices(k);
    const int need = (items + kTailThreads - 1) / kTailThreads;
    return need <= 1 ? 1 : need <= 2 ? 2 : need <= 4 ? 4 : need <= 8 ? 8 : 16;
}

size_t uu_smem(const prmf_handle* h) {
    return sizeof(double) * ((size_t)h->k * h->k + std::max<size_t>((size_t)h->uu_rows * h->k, 1024));
}
size_t vu_smem(const prmf_handle* h) {
    const size_t kk2 = (size_t)h->k * h->k;
    // sGu + (sGv when k <= 64; for larger k that slot only holds the 1024-double slice buffer) + V tile
    return sizeof(double) * (kk2 + (h->k > 64 ? 1024 : kk2) + std::max<size_t>((size_t)h->vu_rows * h->k, 1024) + kVhCap);
}
size_t obj_smem(const prmf_handle* h) {
    const size_t kk2 = (size_t)h->k * h->k;
    return sizeof(double) * (kk2 + (h->k > 64 ? 1024 : kk2) + 1024 + kVhCap);
}
size_t gram_smem(const prmf_handle* h) { return sizeof(double) * ((size_t)h->vu_rows * h->k); }

int launch_u_update(prmf_handle* h) {
    if (h->m == 0) {
        CU(cudaMemsetAsync(h->Gu_part, 0, sizeof(double) * h->uu_grid * h->k * h->k, h->stream));
        if (h->big_k) CU(cudaMemsetAsync(h->Gu_glob, 0, sizeof(double) * h->k * h->k, h->stream));
        return PRMF_OK;
    }
    if (h->big_k) {
#define TILED_CASE(C)                                                                                             \
    case C:                                                                                                       \
        u_update_tiled_kernel<C, 2><<<h->tiled_grid, 256, h->tiled_smem, h->stream>>>(h->U, h->Apart, a_chunks(h), \
                                                                                      h->Gv, h->m, h->k, h->Gu_part); \
        break;
        switch (h->tiled_cpt) {
            TILED_CASE(2)
            TILED_CASE(4)
            default:
            TILED_CASE(8)
        }
#undef TILED_CASE
        LAUNCH_CHECK("u_update_tiled_kernel");
        const int kk2 = h->k * h->k;
        gram_reduce_kernel<<<(kk2 + 255) / 256, 256, 0, h->stream>>>(h->Gu_part, h->tiled_grid, kk2, h->Gu_glob);
        LAUNCH_CHECK("gram_reduce_kernel(Gu)");
        return PRMF_OK;
    }
    NI_SWITCH(h->ni, (u_update_kernel<NI><<<h->uu_grid, kTailThreads, uu_smem(h), h->stream>>>(
                         h->U, h->Apart, a_chunks(h), h->Gv, h->m, h->k, h->uu_rows, h->Gu_part)));
    LAUNCH_CHECK("u_update_kernel");
    return PRMF_OK;
}

// V update + objective.  `sharded`: B and Gu come from the all-reduced packed buffer, else straight from
// the pass-2 / U-update partials (the fixed-order sums happen inside the kernel).
int launch_v_update_objective(prmf_handle* h, bool sharded, double tradeoff) {
    const int64_t nk = h->n * h->k;
    PeerExchange px{};
    if (sharded && h->p2p_ready) {
        px.nranks = h->nranks;
        px.rank = h->rank;
        px.seq = ++h->p2p_seq;
        px.err = h->err_word; px.timeout_ns = h->spin_timeout_ns;
        for (int r = 0; r < h->nranks; ++r) {
            double* base = (double*)h->peer_base[r];
            px.red[r] = base + (size_t)h->p2p_parity * h->p2p_red_count;
            px.flags[r] = (unsigned long long*)(base + 2 * h->p2p_red_count);
        }
        h->p2p_parity ^= 1;
    }
    const double* Bsrc = sharded ? h->red : h->Bpart;
    const int bchunks = sharded ? 1 : b_chunks(h);
    const double* Gusrc = sharded ? h->red + nk : h->big_k ? h->Gu_glob : h->Gu_part;
    const int gchunks = (sharded || h->big_k) ? 1 : h->uu_grid;
    double* Gu_out = (h->big_k && sharded) ? h->Gu_glob : nullptr;
    if (h->big_k) {
#define TILED_CASE(C)                                                                                                  \
    case C:                                                                                                            \
        v_update_tiled_kernel<C, 2><<<h->vu_grid, 256, h->tiled_smem, h->stream>>>(                                     \
            h->Vbuf[h->vcur], h->Vbuf[h->vcur ^ 1], Bsrc, bchunks, nk, Gusrc, (int)h->n, h->k, h->pw, h->active, h->pos, \
            h->gd, h->Gv_part, h->VB_part, px, Gu_out);                                                                \
        break;
        switch (h->tiled_cpt) {
            TILED_CASE(2)
            TILED_CASE(4)
            default:
            TILED_CASE(8)
        }
#undef TILED_CASE
        LAUNCH_CHECK("v_update_tiled_kernel");
    } else {
        NI_SWITCH(h->ni, (v_update_objective_kernel<NI><<<h->vu_grid, kTailThreads, vu_smem(h), h->stream>>>(
                             h->Vbuf[h->vcur], h->Vbuf[h->vcur ^ 1], Bsrc, bchunks, nk, Gusrc, gchunks, (int)h->n, h->k,
                             h->pw, h->active, h->pos, h->gd, h->vu_rows, h->Gv_part, h->VB_part, h->normX_sq, h->as, h->Gv,
                             tradeoff, h->obj, h->step_counter, h->obj_capacity, h->ticket, px)));
        LAUNCH_CHECK("v_update_objective_kernel");
    }
    h->vcur ^= 1;
    if (h->big_k) {
        const int kk2 = h->k * h->k;
        gram_reduce_kernel<<<(kk2 + 255) / 256, 256, 0, h->stream>>>(h->Gv_part, h->vu_grid, kk2, h->Gv_red);
        LAUNCH_CHECK("gram_reduce_kernel(Gv)");
        constexpr int kMiBlocks = 64;
        manifold_parts_kernel<<<kMiBlocks, 256, 0, h->stream>>>(h->Vbuf[h->vcur], h->k, h->Gv_red, h->as, h->mi_part,
                                                                h->mi_part + kMiBlocks);
        LAUNCH_CHECK("manifold_parts_kernel");
        objective_kernel<<<1, kTailThreads, obj_smem(h), h->stream>>>(
            h->Vbuf[h->vcur], h->k, h->Gu_glob, h->Gv_red, h->VB_part, h->vu_grid, h->mi_part, h->mi_part + kMiBlocks, kMiBlocks,
            h->normX_sq, h->Gv, h->gd, tradeoff, h->obj, h->step_counter, h->obj_capacity);
        LAUNCH_CHECK("objective_kernel");
    }
    if (h->x_tc) return refresh_wt(h, h->Vbuf[h->vcur], h->n, h->Vt32, h->ldx32);
    return PRMF_OK;
}

// Gv = V^T V from scratch (after set_UV / restore)
int recompute_Gv(prmf_handle* h) {
    NQ_SWITCH(h->nq, (gram_rows_kernel<NQ><<<h->vu_grid, 256, gram_smem(h), h->stream>>>(
                         h->Vbuf[h->vcur], h->n, h->k, h->vu_rows, h->Gv_part)));
    LAUNCH_CHECK("gram_rows_kernel");
    const int kk2 = h->k * h->k;
    sum_gram_parts_kernel<<<(kk2 + 255) / 256, 256, 0, h->stream>>>(h->Gv_part, h->vu_grid, kk2, h->Gv);
    LAUNCH_CHECK("sum_gram_parts_kernel");
    return PRMF_OK;
}

// device arrays of the flattened active set (ActiveSet): capacity in diagonal / off-diagonal entries
int alloc_active_arena(prmf_handle* h, int64_t cap_diag, int64_t cap_off) {
    const int k = h->k;
    CU(cudaStreamSynchronize(h->stream));
    h->as_arena.release();
    h->as_cap_diag = cap_diag;
    h->as_cap_off = cap_off;
    const size_t n_i32 = (size_t)(2 * h->as_cap_diag + 5 * h->as_cap_off);
    const size_t n_f64 = (size_t)(h->as_cap_diag + h->as_cap_off);
    const size_t total = ((n_i32 * 4 + 255) & ~(size_t)255) + ((n_f64 * 8 + 255) & ~(size_t)255) +
                         ((sizeof(int64_t) * 2 * (k + 1) + 255) & ~(size_t)255);
    cudaError_t ea = h->as_arena.reserve(total, h->device);
    if (ea != cudaSuccess) return fail(h, PRMF_ERR_NOMEM, "cudaMalloc active set: %s", cudaGetErrorString(ea));
    h->as_f64 = h->as_arena.take<double>(n_f64);
    h->as_i32 = h->as_arena.take<int32_t>(n_i32);
    h->as_off = h->as_arena.take<int64_t>((size_t)2 * (k + 1));
    return PRMF_OK;
}

int ensure_pos(prmf_handle* h) {
    if (!h->pos_dirty) return PRMF_OK;
    const int k = h->k;
    // per-factor offsets into the flattened active set
    std::vector<int64_t> offs(2 * (k + 1), 0);
    for (int c = 0; c < k; ++c) {
        const int p = h->active_host[c];
        const int64_t beg = h->path_ptr_host[p], end = h->path_ptr_host[p + 1];
        offs[c + 1] = offs[c] + (end - beg);
        offs[k + 1 + c + 1] = offs[k + 1 + c] + (h->row_ptr_host[end] - h->row_ptr_host[beg]);
    }
    const int64_t nd = offs[k], no = offs[2 * k + 1];
    if (nd > h->as_cap_diag || no > h->as_cap_off || !h->as_i32) {     // (prmf_set_pathways sizes it for the k largest pathways)
        int rc = alloc_active_arena(h, std::max<int64_t>(nd * 2, 1024), std::max<int64_t>(no * 2, 4096));
        if (rc) return rc;
    }
    int32_t* dg = h->as_i32;
    int32_t* df = dg + h->as_cap_diag;
    int32_t* orr = df + h->as_cap_diag;
    int32_t* occ = orr + h->as_cap_off;
    int32_t* olr = occ + h->as_cap_off;
    int32_t* olc = olr + h->as_cap_off;
    int32_t* of = olc + h->as_cap_off;
    double* dc = h->as_f64;
    double* oc = dc + h->as_cap_diag;
    // (pageable source: the runtime stages the bytes before the call returns, so `offs` may go out of scope
    //  and the host does not wait for work still queued on the stream, e.g. a speculative pass 1)
    CU(cudaMemcpyAsync(h->as_off, offs.data(), sizeof(int64_t) * offs.size(), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemsetAsync(h->pos, 0xff, sizeof(int32_t) * h->n * h->k, h->stream));
    dim3 grid(4, h->k);
    build_active_kernel<<<grid, 128, 0, h->stream>>>(h->pw, h->active, k, h->as_off, h->as_off + (k + 1), h->pos, dg, df,
                                                     dc, orr, occ, olr, olc, of, oc);
    LAUNCH_CHECK("build_active_kernel");
    h->as.n_diag = nd; h->as.n_off = no;
    h->as.diag_gene = dg; h->as.diag_factor = df; h->as.diag_coef = dc;
    h->as.off_r = orr; h->as.off_c = occ; h->as.off_lr = olr; h->as.off_lc = olc; h->as.off_factor = of; h->as.off_coef = oc;
    h->pos_dirty = false;
    return PRMF_OK;
}

// ---- fused-tail path (use_epi): two X-stream launches per inner step do the U and V updates as well ----
// Where a sharded step packs its [X^T U | U^T U] for the sum over ranks: this rank's peer-buffer slot of the step's
// parity, which the V update pulls from every rank, or h->red for ncclAllReduce
double* exchange_dst(const prmf_handle* h) {
    return h->p2p_ready ? h->p2p_buf + (size_t)h->p2p_parity * h->p2p_red_count : h->red;
}

int launch_xv_epi(prmf_handle* h, const double* gv_src = nullptr, int gv_parts = 1) {
    EpiParams ep = plain_epi(h);
    ep.arrive = h->epi_counters;
    ep.done = h->epi_counters + h->plan.pass1.panels + h->plan.pass2.panels;
    ep.seq = ++h->epi_seq1;
    ep.dbg_slot = (int)((2 * (h->epi_seq1 - 1)) % 64);
    ep.part2 = h->epi_part2;
    ep.vb2 = h->epi_vb2;
    ep.Uold = h->U;
    ep.Unew = h->U2;
    ep.Gv = gv_src ? gv_src : h->Gv;
    ep.gv_parts = gv_src ? gv_parts : 1;
    ep.Gu_part = h->Gu_part;
    const int rc = launch_xstream(h, pass1(h), 1, ep);
    if (rc) { h->failed = true; return rc; }     // the panel counters expect this launch: no further steps on this handle
    LAUNCH_CHECK("skinny_tma_kernel(pass 1 + U update)");
    std::swap(h->U, h->U2);
    return PRMF_OK;
}

// mode 2: V update (one GPU); 3: pack into exchange_dst(h) for the sum over ranks (sharded)
int launch_xtu_epi(prmf_handle* h, int mode, int hist_slot = -1) {
    EpiParams ep = plain_epi(h);
    const int64_t panels1 = h->plan.pass1.panels, panels2 = h->plan.pass2.panels;
    ep.arrive = h->epi_counters + panels1;
    ep.done = h->epi_counters + panels1 + panels2 + panels1;
    ep.seq = ++h->epi_seq2;
    ep.dbg_slot = (int)((2 * (h->epi_seq2 - 1) + 1) % 64);
    ep.part2 = h->epi_part2;
    ep.vb2 = h->epi_vb2;
    ep.Gu_part_in = h->Gu_part;
    ep.gu_parts = (int)panels1;
    if (mode == 3) {
        ep.red = exchange_dst(h);
    } else {
        ep.Vold = h->Vbuf[h->vcur];
        ep.Vnew = h->Vbuf[h->vcur ^ 1];
        ep.pw = h->pw;
        ep.active = h->active;
        ep.pos = h->pos;
        ep.gd = h->gd;
        ep.Gv_part = h->Gv_part;
        ep.VB_part = h->VB_part;
        if (hist_slot >= 0) {                       // deferred objective: this step's slots
            const size_t kk2 = (size_t)h->k * h->k;
            ep.Gv_part = h->hist_Gvp + (size_t)hist_slot * panels2 * kk2;
            ep.VB_part = h->hist_VBp + (size_t)hist_slot * panels2;
            ep.hist_Gu = h->hist_Gu + (size_t)hist_slot * kk2;
            ep.hist_vh = h->hist_vh + (size_t)hist_slot * kVhCap;
            ep.doff = h->as_off;
        }
    }
    const int rc = launch_xstream(h, pass2(h), mode, ep);
    if (rc) { h->failed = true; return rc; }
    LAUNCH_CHECK(mode == 3 ? "skinny_tma_kernel(pass 2 + pack)" : "skinny_tma_kernel(pass 2 + V update)");
    if (mode != 3) h->vcur ^= 1;
    return PRMF_OK;
}

// fused-tail path (k <= 10): objective of the step from the per-panel partials the pass-2 kernel left
int launch_objective(prmf_handle* h, double tradeoff, const double* Gu_parts, int gu_parts) {
    objective_parts_kernel<<<1, kTailThreads, obj_smem(h), h->stream>>>(
        h->Vbuf[h->vcur], h->k, Gu_parts, gu_parts, h->Gv_part, h->VB_part, h->plan.pass2.panels, h->normX_sq, h->as,
        h->Gv, h->gd, tradeoff, h->obj, h->step_counter, h->obj_capacity);
    LAUNCH_CHECK("objective_parts_kernel");
    return PRMF_OK;
}

// k x P score tables of the current V into h->scores_buf (mass | quad_norm | quad_raw)
template <int F>
int launch_scores_t(prmf_handle* h) {
    const int tiles = (h->k + F - 1) / F;
    // staging buffers sized for the largest pathway, capped near 96 KB (larger pathways gather from global memory)
    int rows = (int)std::max<int64_t>(1, std::min<int64_t>(h->max_support, 2048));
    int edges = (int)std::max<int64_t>(1, std::min<int64_t>(h->max_edges, 16384));
    auto bytes = [&](int r, int e) {
        return sizeof(double) * ((size_t)r * (F + 2) + e) + sizeof(int32_t) * ((size_t)r + 1 + e + 1);
    };
    while (bytes(rows, edges) > 96 * 1024 && (rows > 64 || edges > 256)) {
        if (rows > 64) rows = rows * 3 / 4;
        if (edges > 256) edges = edges * 3 / 4;
    }
    edges = (edges + 1) & ~1;                       // keeps the int32 arrays 8-byte aligned behind the doubles
    const size_t smem = bytes(rows, edges);
    if (smem > 40 * 1024)
        CU(cudaFuncSetAttribute(scores_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const size_t cnt = (size_t)h->k * h->pw.P;
    double* d = h->scores_buf;
    dim3 grid((unsigned)std::min(h->pw.P, h->sm_count * 16), (unsigned)tiles);
    scores_kernel<F><<<grid, 256, smem, h->stream>>>(h->Vbuf[h->vcur], h->k, h->Gv, h->pw, rows, edges, d, d + cnt, d + 2 * cnt);
    LAUNCH_CHECK("scores_kernel");
    return PRMF_OK;
}

int launch_scores(prmf_handle* h) {
    if (h->k <= 4) return launch_scores_t<4>(h);
    if (h->k <= 8) return launch_scores_t<8>(h);
    if (h->k <= 10) return launch_scores_t<10>(h);
    return launch_scores_t<16>(h);
}

// persistent step kernel: halves [h0, h0 + nh) of a block in one cooperative launch (block.cuh / block.cu)
// Rows of X are sharded over ranks: with an NCCL communicator, or with the NVLink / IPC peer buffers alone (then every
// reduction over ranks -- the per-step one inside the persistent step kernel and the few set-up scalars -- goes through
// peer memory and NCCL is not needed at all, e.g. ranks that share one device in a test).
bool sharded(const prmf_handle* h) { return h->nranks > 1 && (h->comm != nullptr || h->p2p_ready); }

// The persistent step kernel is the default for sharded runs (there the exchange lives inside it); on one GPU it
// times like the two-launch path and draws more power in sustained runs, so it is opt-in there (PRMF_BLOCK=1).
bool block_path(const prmf_handle* h) {
    if (!h->use_block) return false;
    if (!sharded(h)) return h->block_forced;
    return h->blk_xchg;
}

int launch_block(prmf_handle* h, int h0, int nh) {
    if (nh <= 0) return PRMF_OK;
    BlockParams prm{};
    prm.X = h->X; prm.Xt = h->Xt; prm.ldx = h->ldx; prm.ldxt = h->ldxt; prm.m = h->m; prm.n = h->n;
    const prmf_xstream_pass &p1 = h->plan.pass1, &p2 = h->plan.pass2;
    prm.panels1 = p1.panels; prm.panel_w1 = p1.panel_w; prm.chunks1 = p1.chunks; prm.rpc1 = p1.rows_per_chunk;
    prm.panels2 = p2.panels; prm.panel_w2 = p2.panel_w; prm.chunks2 = p2.chunks; prm.rpc2 = p2.rows_per_chunk;
    prm.stages = h->plan.stages;
    prm.ring_stage_bytes = h->blk_stage_bytes;
    prm.U[0] = h->U; prm.U[1] = h->U2;
    prm.V[0] = h->Vbuf[h->vcur]; prm.V[1] = h->Vbuf[h->vcur ^ 1];
    prm.Apart = h->Apart; prm.Bpart = h->Bpart; prm.Gu_part = h->Gu_part;
    prm.part2 = h->epi_part2; prm.vb2 = h->epi_vb2;
    prm.Gv0 = h->Gv;
    unsigned long long* c = h->blk_ctr;
    prm.arrive1 = c; c += p1.panels;
    prm.done1 = c; c += p1.panels;
    prm.arrive2 = c; c += p2.panels;
    prm.done2 = c; c += p2.panels;
    prm.udone = c; prm.vdone = c + 1; prm.ufold = c + 2; prm.vfold = c + 3;
    prm.base1 = h->blk_n1; prm.base2 = h->blk_n2;
    prm.h0 = h0; prm.nh = nh;
    { const char* ef = getenv("PRMF_BLOCK_FLAGS"); prm.flags = ef ? (unsigned int)atoi(ef) : 0u; }
    prm.pw = h->pw; prm.active = h->active; prm.pos = h->pos; prm.gd = h->gd;
    prm.hist_Gu = h->hist_Gu; prm.hist_Gvp = h->hist_Gvp; prm.hist_VBp = h->hist_VBp; prm.hist_vh = h->hist_vh;
    prm.doff = h->as_off;
    prm.err = h->err_word; prm.timeout_ns = h->spin_timeout_ns;
    prm.nranks = sharded(h) ? h->nranks : 1; prm.rank = h->rank;
    if (prm.nranks > 1) {
        const size_t off_buf = (size_t)(h->xbuf - h->p2p_buf);                 // same layout in every rank's buffer
        for (int r = 0; r < h->nranks; ++r) prm.xbuf[r] = (ulonglong2*)((double*)h->peer_base[r] + off_buf);
        prm.xcount = h->xcount;
        prm.xbase = h->blk_xseq;
    }
    int n_p1 = 0, n_p2 = 0;
    for (int i = 0; i < nh; ++i) (((h0 + i) & 1) == 0 ? n_p1 : n_p2)++;
    const int grid = (int)std::max(p1.panels * p1.chunks, p2.panels * p2.chunks);
    cudaError_t e_ = prmf_launch_block_kernel(h->k, prm, grid, h->blk_smem, h->stream);
    if (e_ == cudaSuccess) e_ = cudaGetLastError();
    if (e_ != cudaSuccess) {                      // the counters below only move for a launch that is really queued
        h->failed = true;
        return fail(h, PRMF_ERR_CUDA, "launch of block_kernel failed: %s", cudaGetErrorString(e_));
    }
    h->launches++;
    h->blk_n1 += n_p1; h->blk_n2 += n_p2;
    if (prm.nranks > 1) h->blk_xseq += n_p2;
    if (n_p1 & 1) std::swap(h->U, h->U2);
    if (n_p2 & 1) h->vcur ^= 1;
    return PRMF_OK;
}

const double* cur_U(const prmf_handle* h) { return h->ahead == 2 ? h->U2 : h->U; }

void cancel_ahead(prmf_handle* h) {
    if (h->ahead == 2) std::swap(h->U, h->U2);
    h->ahead = 0;
}

// The launch sequence of a block of inner steps (one steps_* function each, below)
enum class StepPath {
    Persistent,        // block_kernel runs the whole block, then objective_deferred_kernel
    FusedDeferred,     // per step: pass 1 + U update, pass 2 + V update; objective_deferred_kernel after the block
    FusedPerStep,      // per step: pass 1 + U update, pass 2 + V update, objective_parts_kernel
    FusedSharded,      // per step: pass 1 + U update, pass 2 + pack, [ncclAllReduce], V update + objective (+ pull)
    Unfused,           // per step: pass 1, U update, pass 2, [pack, exchange], V update + objective
};

// The one place that chooses the path of a block of steps.  Call after ensure_pos (it reads the active set's size).
int step_path(prmf_handle* h, double tradeoff, StepPath* path) {
    // the objective of every step can wait for one launch after the block when
    const bool defer = h->defer_ok                       // the per-step history is allocated (PRMF_DEFER_OBJ != 0),
                       && h->use_epi                     // the fused V update fills it,
                       && (!sharded(h) || h->blk_xchg)   // every rank evaluates the same numbers (sharded: block_kernel),
                       && tradeoff < 0.0                 // gamma and delta stay fixed (--tradeoff updates them every step),
                       && !h->profiling                  // the objective is not timed as a phase of each step,
                       && h->as.n_diag <= kVhCap;        // and the active set's values of V_new fit a history slot
    if (block_path(h) && defer) *path = StepPath::Persistent;
    else if (sharded(h) && !h->comm)                     // without NCCL only block_kernel exchanges between ranks
        return fail(h, PRMF_ERR_STATE, "without an NCCL communicator a sharded handle can only run the persistent step kernel "
                                       "(k <= 10, fixed gamma / delta, no per-phase profiling); call prmf_comm_init for this configuration");
    else if (!h->use_epi) *path = StepPath::Unfused;
    else if (defer) *path = StepPath::FusedDeferred;
    else *path = sharded(h) ? StepPath::FusedSharded : StepPath::FusedPerStep;
    return PRMF_OK;
}

// Pass 1 (+ U update) of the next block's first step, by the kernel step_path picks for that block when its objective
// is deferred.  The block's tradeoff and active set are not known yet, so only step_path's tests of the handle decide.
int prefetch_pass1(prmf_handle* h) {
    if (h->ahead || h->profiling || h->m == 0) return PRMF_OK;
    if (!h->have_X || !h->have_U || !h->have_V) return PRMF_OK;
    int rc = 0;
    if (h->failed) return PRMF_OK;
    if (block_path(h)) {
        if ((rc = launch_block(h, 0, 1))) return rc;
        h->ahead = 2;
    } else if (h->use_epi) {
        if ((rc = launch_xv_epi(h))) return rc;
        h->ahead = 2;
    } else {
        if ((rc = launch_xv(h))) return rc;
        h->ahead = 1;
    }
    return PRMF_OK;
}

int allreduce(prmf_handle* h, double* buf, size_t count) {
    if (!h->comm) {
        if (!sharded(h)) return PRMF_OK;
        // no NCCL: the few set-up scalars (||X||^2, the agreement of prmf_p2p_finalize, a verification residual) are summed
        // over the peer buffers with the same {value, sequence} entries as the per-step exchange
        if (count > (size_t)kSmallAllreduceMax) return fail(h, PRMF_ERR_STATE, "reduction of %zu values over ranks needs NCCL", count);
        PeerSmall ps{};
        const size_t off = (size_t)(h->xsmall - h->p2p_buf);
        for (int r = 0; r < h->nranks; ++r) ps.slot[r] = (ulonglong2*)((double*)h->peer_base[r] + off);
        ps.nranks = h->nranks; ps.rank = h->rank; ps.seq = ++h->small_seq;
        ps.err = h->err_word; ps.timeout_ns = h->spin_timeout_ns;
        cudaError_t e_ = prmf_launch_small_allreduce(buf, (int)count, ps, h->stream);
        if (e_ != cudaSuccess) return fail(h, PRMF_ERR_CUDA, "peer all-reduce launch failed: %s", cudaGetErrorString(e_));
        h->launches++;
        return PRMF_OK;
    }
    int r = g_nccl.AllReduce(buf, buf, count, kNcclFloat64, kNcclSum, h->comm, h->stream);
    if (r != 0)
        return fail(h, PRMF_ERR_NCCL, "ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
    return PRMF_OK;
}

int ensure_obj_capacity(prmf_handle* h, int n_steps) {
    if (n_steps <= h->obj_capacity) return PRMF_OK;
    return fail(h, PRMF_ERR_ARG, "at most %d inner steps per prmf_step call", h->obj_capacity);
}

void harvest_events(prmf_handle* h) {
    for (auto& pr : h->ev_pairs) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->ev_pool[pr.second], h->ev_pool[pr.second + 1]) == cudaSuccess) {
            h->phase_ms[pr.first] += ms;
            h->phase_n[pr.first]++;
        }
    }
    for (auto e : h->ev_pool) cudaEventDestroy(e);
    h->ev_pool.clear();
    h->ev_pairs.clear();
}

// phase timing (profiling mode only): an event pair around each phase of the step
void tic(prmf_handle* h, int phase) {
    if (!h->profiling) return;
    cudaEvent_t e[2];
    cudaEventCreate(&e[0]);
    cudaEventCreate(&e[1]);
    h->ev_pairs.push_back({phase, (int)h->ev_pool.size()});
    h->ev_pool.insert(h->ev_pool.end(), e, e + 2);
    cudaEventRecord(e[0], h->stream);
}

void toc(prmf_handle* h) {
    if (!h->profiling) return;
    cudaEventRecord(h->ev_pool[h->ev_pairs.back().second + 1], h->stream);
}

// the objective of every step of a block from the history slots its V updates filled: one thread block per step
int launch_deferred_objective(prmf_handle* h, int n_steps) {
    objective_deferred_kernel<<<n_steps, kTailThreads, obj_smem(h), h->stream>>>(
        h->k, h->hist_Gu, h->hist_Gvp, h->hist_VBp, h->plan.pass2.panels, h->hist_vh, kVhCap, h->normX_sq, h->as, h->Gv,
        h->gd, h->obj, h->obj_capacity);
    LAUNCH_CHECK("objective_deferred_kernel");
    return PRMF_OK;
}

// ---- the launch sequence of each StepPath.  pass1_done: prmf_block_end already enqueued pass 1 (+ U update) of the
// first step (prefetch_pass1).

int steps_persistent(prmf_handle* h, int n_steps, bool pass1_done) {
    const int h0 = pass1_done ? 1 : 0;
    int rc = launch_block(h, h0, 2 * n_steps - h0);
    if (rc) return rc;
    return launch_deferred_objective(h, n_steps);
}

int steps_fused_deferred(prmf_handle* h, int n_steps, bool pass1_done) {
    const size_t kk2 = (size_t)h->k * h->k;
    const int64_t panels2 = h->plan.pass2.panels;
    for (int s = 0; s < n_steps; ++s) {
        int rc = 0;
        // pass 1 of a later step reads V^T V as the panel partials the previous step's V update left in its slot
        if (s > 0) rc = launch_xv_epi(h, h->hist_Gvp + (size_t)(s - 1) * panels2 * kk2, (int)panels2);
        else if (!pass1_done) rc = launch_xv_epi(h);
        if (rc) return rc;
        if ((rc = launch_xtu_epi(h, 2, s))) return rc;
    }
    return launch_deferred_objective(h, n_steps);
}

int steps_fused_per_step(prmf_handle* h, int n_steps, bool pass1_done, double tradeoff) {
    for (int s = 0; s < n_steps; ++s) {
        int rc = 0;
        if (s > 0 || !pass1_done) { tic(h, 0); rc = launch_xv_epi(h); toc(h); }
        if (rc) return rc;
        tic(h, 2); rc = launch_xtu_epi(h, 2); toc(h);                  // + V update
        if (rc) return rc;
        tic(h, 5); rc = launch_objective(h, tradeoff, h->Gu_part, h->plan.pass1.panels); toc(h);
        if (rc) return rc;
    }
    return PRMF_OK;
}

int steps_fused_sharded(prmf_handle* h, int n_steps, bool pass1_done, double tradeoff) {
    const size_t red_count = (size_t)h->n * h->k + (size_t)h->k * h->k + 2;
    for (int s = 0; s < n_steps; ++s) {
        int rc = 0;
        if (s > 0 || !pass1_done) { tic(h, 0); rc = launch_xv_epi(h); toc(h); }
        if (rc) return rc;
        tic(h, 2); rc = launch_xtu_epi(h, 3); toc(h);                  // + pack
        if (rc) return rc;
        if (!h->p2p_ready) {                                            // else: pulled inside the V update
            tic(h, 3); rc = allreduce(h, h->red, red_count); toc(h);
            if (rc) return rc;
        }
        tic(h, 4); rc = launch_v_update_objective(h, true, tradeoff); toc(h);
        if (rc) return rc;
    }
    return PRMF_OK;
}

int steps_unfused(prmf_handle* h, int n_steps, bool pass1_done, double tradeoff) {
    const bool is_sharded = sharded(h);
    const int64_t nk = h->n * h->k;
    const int kk2 = h->k * h->k;
    for (int s = 0; s < n_steps; ++s) {
        int rc = 0;
        if (s > 0 || !pass1_done) { tic(h, 0); rc = launch_xv(h); toc(h); }
        if (rc) return rc;
        tic(h, 1); rc = launch_u_update(h); toc(h);
        if (rc) return rc;
        tic(h, 2); rc = launch_xtu(h); toc(h);
        if (rc) return rc;
        if (is_sharded) {
            tic(h, 3);
            reduce_pack_kernel<<<(unsigned)((nk + kk2 + 2 + 255) / 256), 256, 0, h->stream>>>(
                h->Bpart, b_chunks(h), nk, h->Gu_part, h->uu_grid, h->k, exchange_dst(h));
            LAUNCH_CHECK("reduce_pack_kernel");
            if (!h->p2p_ready) rc = allreduce(h, h->red, (size_t)nk + kk2 + 2);      // else: pulled inside the V update
            toc(h);
            if (rc) return rc;
        }
        tic(h, 4); rc = launch_v_update_objective(h, is_sharded, tradeoff); toc(h);
        if (rc) return rc;
    }
    return PRMF_OK;
}

// Enqueues a block of n_steps inner steps: the launch sequence of the StepPath that step_path chooses.
int enqueue_steps(prmf_handle* h, int n_steps, double gamma, double delta, double tradeoff) {
    if (!h->have_X || !h->have_U || !h->have_V || !h->have_pw || !h->have_active)
        return fail(h, PRMF_ERR_STATE, "prmf_step needs X, U/V, pathways and the active set first");
    if (n_steps <= 0) return fail(h, PRMF_ERR_ARG, "n_steps must be positive");
    if (h->failed) return fail(h, PRMF_ERR_STATE, "the handle is in a failed state (an earlier launch failed or a device wait expired)");
    CU(cudaSetDevice(h->device));
    int rc = ensure_obj_capacity(h, n_steps);
    if (rc) return rc;
    if ((rc = ensure_pos(h))) return rc;
    const double gdh[2] = {gamma, delta};
    CU(cudaMemcpyAsync(h->gd, gdh, sizeof gdh, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemsetAsync(h->step_counter, 0, sizeof(int), h->stream));
    StepPath path;
    if ((rc = step_path(h, tradeoff, &path))) return rc;
    const bool pass1_done = h->ahead != 0;
    h->ahead = 0;
    switch (path) {
        case StepPath::Persistent: return steps_persistent(h, n_steps, pass1_done);
        case StepPath::FusedDeferred: return steps_fused_deferred(h, n_steps, pass1_done);
        case StepPath::FusedPerStep: return steps_fused_per_step(h, n_steps, pass1_done, tradeoff);
        case StepPath::FusedSharded: return steps_fused_sharded(h, n_steps, pass1_done, tradeoff);
        case StepPath::Unfused: return steps_unfused(h, n_steps, pass1_done, tradeoff);
    }
    return fail(h, PRMF_ERR_STATE, "unknown step path");
}

int check_err_word(prmf_handle* h, unsigned int errw) {
    if (errw == 0) return PRMF_OK;
    h->failed = true;
    return fail(h, PRMF_ERR_TIMEOUT, "a device-side wait expired after %.1f s (%s%s); results of this block are invalid",
                h->spin_timeout_ns * 1e-9, (errw & kErrTimeoutLocal) ? "waiting for another thread block of this GPU " : "",
                (errw & kErrTimeoutPeer) ? "waiting for a peer rank's exchange flag" : "");
}

// The hot loop takes recon^2 from the identity ||X||^2 - 2 sum(V*B) + tr(Gu Gv) (no pass over X).  When the fit is tight
// (recon^2 below 1e-8 ||X||^2, e.g. noiseless low-rank data) the cancellation leaves few correct digits, and the value
// drives the convergence test and the best-iterate choice of the driver (:745-774), which only look at the LAST step of
// a block.  For that step U and V are still on the device: redo its recon with the explicit residual pass (:337).
int refine_last_row(prmf_handle* h, int n_steps, double* obj_parts) {
    if (!obj_parts || n_steps <= 0 || h->failed) return PRMF_OK;
    double* row = obj_parts + (size_t)(n_steps - 1) * kObjStride;
    const double r2 = row[7];
    if (!(r2 < 1e-8 * h->normX_sq_host)) return PRMF_OK;
    double exact = 0.0;
    int rc = prmf_residual_sq(h, &exact);
    if (rc) return rc;
    const double recon = std::sqrt(exact > 0.0 ? exact : 0.0);
    row[4] = recon + row[5] * row[1] + row[6] * row[2] + row[3];                   // :362
    row[0] = recon;
    row[7] = exact;
    return PRMF_OK;
}

int collect(prmf_handle* h, int n_steps, double* obj_parts, double* gamma_delta_out) {
    CU(cudaSetDevice(h->device));
    if (n_steps > h->obj_capacity) return fail(h, PRMF_ERR_ARG, "collect: more steps than were run");
    if (obj_parts)
        CU(cudaMemcpyAsync(obj_parts, h->obj, sizeof(double) * n_steps * kObjStride, cudaMemcpyDeviceToHost, h->stream));
    if (gamma_delta_out)
        CU(cudaMemcpyAsync(gamma_delta_out, h->gd, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    unsigned int errw = 0;
    CU(cudaMemcpyAsync(&errw, h->err_word, sizeof errw, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (h->profiling) harvest_events(h);
    int rc_e = check_err_word(h, errw);
    if (rc_e) return rc_e;
    return refine_last_row(h, n_steps, obj_parts);
}

// ---- TF32 mode set-up ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D fp32 tensor map over a row-major matrix (rows x cols, leading dimension ld), box = box_rows x 32 columns,
// 128-byte swizzle; out-of-range elements read as zero (ragged tiles need no special case).
int make_tensor_map(prmf_handle* h, CUtensorMap* map, const float* base, int64_t rows, int64_t cols, int64_t ld,
                    int box_rows) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
            return fail(h, PRMF_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
        encode = (EncodeTiledFn)fn;
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)kTcBlockK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, PRMF_ERR_CUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
    return PRMF_OK;
}

// Tiles of 128 rows x column chunks: pick the smallest chunk count whose wave quantisation over the
// 2 x SM-count resident CTAs is within 3 % of the best one.
void plan_tc(int sm_count, int64_t R, int64_t C, int64_t* tiles, int64_t* chunks, int64_t* cols_per_chunk) {
    *tiles = std::max<int64_t>(1, (R + kTcTileRows - 1) / kTcTileRows);
    const double slots = 2.0 * sm_count;
    const int max_chunks = (int)std::max<int64_t>(1, std::min<int64_t>(64, C / 512));
    double best = 0.0;
    std::vector<double> eff(max_chunks + 1, 0.0);
    for (int c = 1; c <= max_chunks; ++c) {
        const double ctas = (double)*tiles * c;
        eff[c] = ctas / (std::ceil(ctas / slots) * slots);
        best = std::max(best, eff[c]);
    }
    int pick = 1;
    for (int c = 1; c <= max_chunks; ++c)
        if (eff[c] >= best - 0.03) { pick = c; break; }
    *cols_per_chunk = round_up(std::max<int64_t>(1, (C + pick - 1) / pick), kTcBlockK);
    *chunks = std::max<int64_t>(1, (C + *cols_per_chunk - 1) / *cols_per_chunk);
}

void setup_tf32(prmf_handle* h) {
    const prmf_xstream_plan& p = h->plan;
    h->Kp = (int)round_up(h->k, 16);
    uint32_t tcols = 32;
    while ((int)tcols < h->Kp) tcols <<= 1;
    const int stages = (int)p.tc_stages;
    h->tc1 = TcParams{h->m, h->n, h->k, h->Kp, p.tc_cols_per_chunk1, stages, tcols, nullptr};
    h->tc2 = TcParams{h->n, h->m, h->k, h->Kp, p.tc_cols_per_chunk2, stages, tcols, nullptr};
}

int finish_setup_tf32(prmf_handle* h) {
    h->tc1.Out = h->Apart;
    h->tc2.Out = h->Bpart;
    CU(cudaFuncSetAttribute(tc_rowdot_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->plan.tc_smem));
    CU(cudaFuncSetAttribute(tc_rowdot_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    int rc = 0;
    if (h->m > 0) {
        if ((rc = make_tensor_map(h, &h->tm_X, h->X32, h->m, h->n, h->ldx32, kTcTileRows))) return rc;
        if ((rc = make_tensor_map(h, &h->tm_Xt, h->Xt32, h->n, h->m, h->ldxt32, kTcTileRows))) return rc;
        if ((rc = make_tensor_map(h, &h->tm_Ut, h->Ut32, h->Kp, h->m, h->ldxt32, h->Kp))) return rc;
        if ((rc = make_tensor_map(h, &h->tm_Vt, h->Vt32, h->Kp, h->n, h->ldx32, h->Kp))) return rc;
    }
    return PRMF_OK;
}

// fp32 storage (tf32 and f32 modes): store a row block (host or device, fp64 or fp32) into the fp32 layout, rounded to
// tf32 in the tf32 mode and to the nearest fp32 value in the f32 mode (exact for fp32 input).  Host blocks go through a
// bounded device staging buffer, block after block on the handle's stream.
template <typename T, bool TF32>
void launch_store_rows(prmf_handle* h, const T* X, int64_t ld, int64_t rows, float* dst) {
    to_tf32_rows_kernel<T, TF32><<<h->sm_count * 8, 256, 0, h->stream>>>(X, ld, rows, h->n, dst, h->ldx32);
}

template <typename T>
int store_x32(prmf_handle* h, const T* X, int64_t ld, bool on_host) {
    const int64_t m = h->m, n = h->n;
    if (m == 0) return PRMF_OK;
    auto store = h->x_tc ? launch_store_rows<T, true> : launch_store_rows<T, false>;
    if (!on_host) {
        store(h, X, ld, m, h->X32);
        LAUNCH_CHECK("to_tf32_rows_kernel");
        return PRMF_OK;
    }
    const int64_t rows_blk = std::max<int64_t>(1, std::min<int64_t>(m, ((int64_t)256 << 20) / (n * (int64_t)sizeof(T))));
    T* stage = nullptr;
    int rc = dalloc(h, &stage, (size_t)rows_blk * n);
    if (rc) return rc;
    cudaError_t e = cudaSuccess;
    for (int64_t r0 = 0; r0 < m && e == cudaSuccess; r0 += rows_blk) {
        const int64_t rows = std::min(rows_blk, m - r0);
        e = cudaMemcpy2DAsync(stage, n * sizeof(T), X + r0 * ld, ld * sizeof(T), n * sizeof(T), rows,
                              cudaMemcpyHostToDevice, h->stream);
        if (e != cudaSuccess) break;
        store(h, stage, n, rows, h->X32 + r0 * h->ldx32);
        h->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(stage);
    if (e != cudaSuccess) return fail(h, PRMF_ERR_CUDA, "fp32 upload of X failed: %s", cudaGetErrorString(e));
    return PRMF_OK;
}

// The Lawson-Hanson loop of prmf_nnls_x over a workspace laid out by the caller (wk).  W: the operand of the X stream
// that computes the duals (V for A = X^T, pass 1; U for A = X, pass 2); its zero pad rows are left as they are.
template <typename T>
int nnls_loop(prmf_handle* h, int transpose, NnlsWork<T>& wk, double* rnorm_dev, std::vector<int32_t>& status) {
    const int k = wk.k;
    double* W = transpose ? h->Vbuf[h->vcur] : h->U;
    const double* part = transpose ? h->Apart : h->Bpart;
    const int chunks = transpose ? a_chunks(h) : b_chunks(h);
    const int64_t wcount = wk.nun * k;
    const dim3 rgrid((unsigned)((wk.neq + kNnlsThreads - 1) / kNnlsThreads), (unsigned)k);
    // every launch of nnls_step_kernel counts one iteration of each running problem, so the loop ends by maxiter + 1
    for (int64_t round = 0; round <= (int64_t)wk.maxiter; ++round) {
        nnls_resid_kernel<<<rgrid, kNnlsThreads, 0, h->stream>>>(wk, W, 0);
        LAUNCH_CHECK("nnls_resid_kernel");
        int rc = transpose ? launch_xv(h) : launch_xtu(h);
        if (rc) return rc;
        sum_chunks_kernel<<<(unsigned)((wcount + 255) / 256), 256, 0, h->stream>>>(part, chunks, wcount, wk.w);
        LAUNCH_CHECK("sum_chunks_kernel");
        nnls_step_kernel<<<(unsigned)k, kNnlsThreads, 0, h->stream>>>(wk);
        LAUNCH_CHECK("nnls_step_kernel");
        CU(cudaMemcpyAsync(status.data(), wk.status, sizeof(int32_t) * k, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        if (std::none_of(status.begin(), status.end(), [](int32_t s) { return s == kNnlsRunning; })) break;
    }
    nnls_resid_kernel<<<rgrid, kNnlsThreads, 0, h->stream>>>(wk, W, 1);
    LAUNCH_CHECK("nnls_resid_kernel");
    nnls_rnorm_kernel<<<(unsigned)k, kNnlsThreads, 0, h->stream>>>(W, wk.neq, k, rnorm_dev);
    LAUNCH_CHECK("nnls_rnorm_kernel");
    return PRMF_OK;
}

int finish_X(prmf_handle* h) {
    cancel_ahead(h);
    // transposed copy for pass 1, then ||X||^2 partial of this rank, all-reduced once
    const int blocks = h->sm_count * 4;
    if (h->m > 0 && h->x32) {
        dim3 tg((unsigned)((h->n + 31) / 32), (unsigned)((h->m + 31) / 32));
        transpose_f32_kernel<<<tg, 256, 0, h->stream>>>(h->X32, h->ldx32, h->m, h->n, h->Xt32, h->ldxt32);
        LAUNCH_CHECK("transpose_f32_kernel");
        if (h->x_tc) {
            sumsq_f32_kernel<<<blocks, 256, 0, h->stream>>>(h->X32, h->ldx32, h->m, h->n, h->scal_part);
            LAUNCH_CHECK("sumsq_f32_kernel");
        } else {                    // f32 mode: the order of the fp64 mode, so ||X||^2 is that of the widened matrix
            sumsq_kernel<<<blocks, 256, 0, h->stream>>>(h->X32, h->ldx32, h->m, h->n2, h->scal_part);
            LAUNCH_CHECK("sumsq_kernel");
        }
        sum_partials_kernel<<<1, 256, 0, h->stream>>>(h->scal_part, blocks, h->normX_sq);
        LAUNCH_CHECK("sum_partials_kernel");
    } else if (h->m > 0) {
        dim3 tg((unsigned)((h->n + 31) / 32), (unsigned)((h->m + 31) / 32));
        transpose_kernel<<<tg, 256, 0, h->stream>>>(h->X, h->ldx, h->m, h->n, h->Xt, h->ldxt);
        LAUNCH_CHECK("transpose_kernel");
        sumsq_kernel<<<blocks, 256, 0, h->stream>>>(h->X, h->ldx, h->m, h->n2, h->scal_part);
        LAUNCH_CHECK("sumsq_kernel");
        sum_partials_kernel<<<1, 256, 0, h->stream>>>(h->scal_part, blocks, h->normX_sq);
        LAUNCH_CHECK("sum_partials_kernel");
    } else {
        CU(cudaMemsetAsync(h->normX_sq, 0, sizeof(double), h->stream));
    }
    int rc = allreduce(h, h->normX_sq, 1);
    if (rc) return rc;
    CU(cudaMemcpyAsync(&h->normX_sq_host, h->normX_sq, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->have_X = true;
    return PRMF_OK;
}

// prmf_nnls_x after its checks, on the columns of A = Arows[j * lda ..] (rows of X or of its transposed copy)
template <typename T>
int nnls_x_run(prmf_handle* h, int transpose, const T* Arows, int64_t lda, const double* B_host, int maxiter,
               double* x_out, double* rnorm_out, int32_t* status_out, int32_t* iter_out) {
    NnlsWork<T> wk;
    wk.k = h->k;
    wk.neq = transpose ? h->n : h->m;
    wk.nun = transpose ? h->m : h->n;
    wk.Arows = Arows;
    wk.lda = lda;
    wk.cap = (int)std::min<int64_t>({wk.neq, wk.nun, (int64_t)kNnlsMaxPassive});
    wk.maxiter = maxiter > 0 ? maxiter : (int)std::min<int64_t>(3 * wk.nun, INT32_MAX - 1);   // scipy: 3 * #unknowns
    wk.tol = 10.0 * (double)std::max(wk.neq, wk.nun) * DBL_EPSILON;                          // 10 max(m, n) eps
    const int k = wk.k;
    const size_t cap = (size_t)wk.cap, kk = (size_t)k;
    auto pad = [](size_t bytes) { return (bytes + 255) & ~(size_t)255; };
    const size_t d = sizeof(double);
    const size_t b_bt = pad(d * kk * wk.neq), b_w = pad(d * kk * wk.nun), b_g = pad(d * kk * cap * cap);
    const size_t b_vec = pad(d * kk * cap), b_idx = pad(sizeof(int) * kk * cap), b_flag = pad(kk * wk.nun);
    const size_t b_small = pad(sizeof(int) * kk), b_rn = pad(d * kk);
    const size_t total = b_bt + b_w + 2 * b_g + 2 * b_vec + b_idx + b_flag + 3 * b_small + b_rn;
    unsigned char* ws = nullptr;
    cudaError_t ea = g_pool.alloc((void**)&ws, total, h->device);
    if (ea != cudaSuccess) return fail(h, PRMF_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", total, cudaGetErrorString(ea));
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* p = ws + off; off += bytes; return p; };
    wk.Bt = (const double*)take(b_bt);
    wk.w = (double*)take(b_w);
    wk.G = (double*)take(b_g);
    wk.L = (double*)take(b_g);
    wk.atb = (double*)take(b_vec);
    unsigned char* zero_from = ws + off;               // everything from here on starts at zero
    wk.xP = (double*)take(b_vec);
    wk.pidx = (int*)take(b_idx);
    wk.flag = (int8_t*)take(b_flag);
    wk.np = (int*)take(b_small);
    wk.iter = (int*)take(b_small);
    wk.status = (int*)take(b_small);
    double* rnorm_dev = (double*)take(b_rn);

    std::vector<double> Bt((size_t)k * wk.neq);
    for (int64_t e = 0; e < wk.neq; ++e)
        for (int c = 0; c < k; ++c) Bt[(size_t)c * wk.neq + e] = B_host[e * k + c];
    std::vector<int32_t> status(k, kNnlsRunning), np_h(k), pidx_h(kk * cap);
    std::vector<double> xP_h(kk * cap);
    int rc = PRMF_OK;
    cudaError_t e = cudaMemcpyAsync((void*)wk.Bt, Bt.data(), sizeof(double) * Bt.size(), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(zero_from, 0, (size_t)(ws + total - zero_from), h->stream);
    if (e != cudaSuccess) rc = fail(h, PRMF_ERR_CUDA, "prmf_nnls_x upload: %s", cudaGetErrorString(e));
    if (!rc) rc = nnls_loop(h, transpose, wk, rnorm_dev, status);
    if (!rc) {
        e = cudaMemcpyAsync(np_h.data(), wk.np, sizeof(int32_t) * k, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(pidx_h.data(), wk.pidx, sizeof(int32_t) * kk * cap, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(xP_h.data(), wk.xP, sizeof(double) * kk * cap, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(status_out, wk.status, sizeof(int32_t) * k, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(rnorm_out, rnorm_dev, sizeof(double) * k, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess && iter_out)
            e = cudaMemcpyAsync(iter_out, wk.iter, sizeof(int32_t) * k, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) rc = fail(h, PRMF_ERR_CUDA, "prmf_nnls_x read-back: %s", cudaGetErrorString(e));
    } else {
        cudaStreamSynchronize(h->stream);
    }
    g_pool.release(ws, total, h->device);
    if (rc) return rc;
    std::fill(x_out, x_out + wk.nun * k, 0.0);
    for (int c = 0; c < k; ++c)
        for (int q = 0; q < np_h[c]; ++q) x_out[(int64_t)pidx_h[c * cap + q] * k + c] = xP_h[c * cap + q];
    h->err.clear();
    for (int c = 0; c < k; ++c) {
        if (status_out[c] == kNnlsCapacity) {
            fail(h, PRMF_OK, "prmf_nnls_x: problem %d needs more than %d passive columns (the workspace capacity)", c,
                 wk.cap);
            break;
        }
        if (status_out[c] == kNnlsSingular) {
            fail(h, PRMF_OK, "prmf_nnls_x: problem %d: the Gram matrix of its passive columns lost positive definiteness", c);
            break;
        }
    }
    return PRMF_OK;
}

}  // namespace

// =====================================================================================================
extern "C" {

int prmf_abi_version(void) { return 1; }

const char* prmf_last_error(const prmf_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int prmf_plan_xstream(int64_t m_local, int64_t n, int k, int x_dtype, int sm_count, int stages_override,
                      prmf_xstream_plan* out) {
    if (!out || m_local < 0 || n <= 0 || k <= 0 || k > 128 || sm_count <= 0 ||
        (x_dtype != PRMF_X_F64 && x_dtype != PRMF_X_TF32 && x_dtype != PRMF_X_F32))
        return PRMF_ERR_ARG;
    prmf_xstream_plan p{};
    // DFMA kernels: one CTA per SM, column panels of at most 1024 / FG columns, row chunks of at least 4 stages.  The
    // panels and chunks do not depend on the storage type, which is what makes an fp32 handle bitwise equal to an fp64
    // handle on the widened matrix; only the ring differs (an fp32 stage holds half the bytes of X).
    const bool x32 = x_dtype != PRMF_X_F64;
    p.fg = 1;
    if (k > 10) {                          // general-k kernel: FG factor groups x KT factors per thread
        const int groups = (k + 15) / 16;
        p.fg = groups <= 1 ? 1 : groups <= 2 ? 2 : groups <= 4 ? 4 : 8;
        const int64_t per = (k + p.fg - 1) / p.fg;
        p.kt = per <= 12 ? 12 : 16;
    }
    const int64_t max_panel = 1024 / p.fg;
    auto plan = [&](int64_t cols, int64_t rows, prmf_xstream_pass& q) {
        q.panels = std::max<int64_t>(1, (cols + max_panel - 1) / max_panel);
        q.panel_w = round_up((std::max<int64_t>(1, cols) + q.panels - 1) / q.panels, 4);
        q.chunks = std::max<int64_t>(1, sm_count / q.panels);
        q.chunks = std::min<int64_t>(q.chunks, std::max<int64_t>(1, rows / (4 * kTmaRS)));
        // rows per chunk: even (the W rows of a chunk must start 16-byte aligned for the bulk copies), not a multiple
        // of the stage height -- a ragged last stage costs less than a last chunk that is nearly empty
        q.rows_per_chunk = round_up(std::max<int64_t>(1, (rows + q.chunks - 1) / q.chunks), 2);
        const int64_t xb = kTmaRS * q.panel_w * (x32 ? 4 : 8);
        const int64_t wb = ((kTmaRS * (int64_t)k + 16) * 8 + 127) & ~(int64_t)127;
        q.ring_smem = p.stages * (xb + wb) + 2 * p.stages * (int64_t)sizeof(uint64_t);
        // the last CTA of a panel reuses the ring for Gv/Gu, the slice sums and the panel's new rows
        const int64_t share = (q.panel_w + q.chunks - 1) / q.chunks * k;
        const int64_t tail = (int64_t)sizeof(double) * (128 + 8 * (int64_t)k * k + 3 * share);
        q.tail_smem = k <= 10 ? std::max(q.ring_smem, tail) : q.ring_smem;
    };
    auto plan_passes = [&]() {             // true when both rings fit
        plan(m_local, n, p.pass1);
        plan(n, m_local, p.pass2);
        return std::max(p.pass1.ring_smem, p.pass2.ring_smem) <= 220 * 1024;
    };
    // the default ring fits at every k <= 128 (tests/test_xstream_exact.py, tests/test_f32_storage.py); an override is
    // kept where its ring fits as well, and the default runs elsewhere.  fp32 tiles: twice the stages, the same bytes of
    // X in flight.
    const int64_t default_stages = (p.fg >= 4 ? 6 : p.fg == 2 ? 4 : 3) * (x32 ? 2 : 1);
    p.stages = stages_override >= 2 && stages_override <= 12 ? stages_override : default_stages;
    if (!plan_passes()) {
        p.stages = default_stages;
        plan_passes();
    }
    if (x_dtype == PRMF_X_TF32) {
        plan_tc(sm_count, m_local, n, &p.tc_tiles1, &p.tc_chunks1, &p.tc_cols_per_chunk1);
        plan_tc(sm_count, n, m_local, &p.tc_tiles2, &p.tc_chunks2, &p.tc_cols_per_chunk2);
        const int64_t stage = (int64_t)kTcTileRows * kTcBlockK * 4 + round_up(k, 16) * kTcBlockK * 4;
        p.tc_stages = std::max<int64_t>(2, std::min<int64_t>(8, (108 * 1024) / stage));      // two CTAs per SM
        p.tc_smem = p.tc_stages * stage + (2 * p.tc_stages + 1) * (int64_t)sizeof(uint64_t) + 16 + 1024;
    }
    *out = p;
    return PRMF_OK;
}

int prmf_create(prmf_handle** out, int device, int64_t m_local, int64_t m_global, int64_t n, int k, void* stream) {
    return prmf_create_ex(out, device, m_local, m_global, n, k, stream, PRMF_X_F64);
}

int prmf_create_ex(prmf_handle** out, int device, int64_t m_local, int64_t m_global, int64_t n, int k, void* stream,
                   int x_dtype) {
    prmf_handle* h = nullptr;
    if (x_dtype != PRMF_X_F64 && x_dtype != PRMF_X_TF32 && x_dtype != PRMF_X_F32)
        return fail(h, PRMF_ERR_ARG, "unknown x_dtype %d", x_dtype);
    if (!out) return fail(h, PRMF_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (m_local < 0 || n <= 0 || k <= 0 || m_global < m_local)
        return fail(h, PRMF_ERR_ARG, "bad shape m_local=%lld m_global=%lld n=%lld k=%d", (long long)m_local,
                    (long long)m_global, (long long)n, k);
    if (k > 128) return fail(h, PRMF_ERR_ARG, "k=%d not supported (max 128)", k);
    if (x_dtype == PRMF_X_F32 && m_local != m_global)
        return fail(h, PRMF_ERR_ARG, "PRMF_X_F32 handles are single-rank (m_local=%lld, m_global=%lld)", (long long)m_local,
                    (long long)m_global);
    if (n > (int64_t)1 << 30) return fail(h, PRMF_ERR_ARG, "n too large");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(h, PRMF_ERR_CUDA, "no CUDA device (%s); libprmf_b200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= ndev) return fail(h, PRMF_ERR_ARG, "device %d out of range (%d devices)", device, ndev);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(h, PRMF_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(h, PRMF_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major < 10)
        return fail(h, PRMF_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                    prop.minor);
    prmf_handle* hh = new prmf_handle();
    h = hh;
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    h->m = m_local; h->m_global = m_global; h->n = n; h->k = k;
    h->ldx = round_up(n, 16);        // rows start on 128-byte lines; pad columns are zero
    h->ldxt = round_up(std::max<int64_t>(1, m_local), 16);
    h->n2 = (int)round_up(n, 2);
    if (stream) { h->stream = (cudaStream_t)stream; }
    else {
        e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { delete hh; return fail(nullptr, PRMF_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
        h->own_stream = true;
    }
    // launch geometry
    h->nq = pick_nq(k);
    h->ni = pick_ni(k);
    h->uu_rows = (int)std::max<int64_t>(8, std::min<int64_t>(128, 2048 / k));
    h->uu_grid = (int)std::max<int64_t>(1, std::min<int64_t>(h->sm_count, (m_local + h->uu_rows - 1) / h->uu_rows));
    h->big_k = k > 16;
    if (h->big_k) {
        h->tiled_cpt = k <= 32 ? 2 : k <= 64 ? 4 : 8;
        const int kt = 16 * h->tiled_cpt;
        h->tiled_smem = sizeof(double) * ((size_t)kt * kt + 32 * (size_t)(kt + 2) + 32 * (size_t)k);
        h->tiled_grid = (int)std::max<int64_t>(1, std::min<int64_t>(h->sm_count, (m_local + 31) / 32));
        h->uu_grid = h->tiled_grid;              // number of U^T U partials
    }
    h->vu_rows = (int)std::max<int64_t>(8, std::min<int64_t>(128, 2048 / k));
    h->vu_grid = (int)std::max<int64_t>(1, std::min<int64_t>(h->sm_count, (n + h->vu_rows - 1) / h->vu_rows));
    if (h->big_k) {                              // tiles of 32 genes per block in the tiled V update
        h->vu_rows = 32;
        h->vu_grid = (int)std::max<int64_t>(1, std::min<int64_t>(h->sm_count, (n + 31) / 32));
    }
    h->x32 = x_dtype != PRMF_X_F64;
    h->x_tc = x_dtype == PRMF_X_TF32;
    {
        const char* es = getenv("PRMF_TMA_STAGES");
        prmf_plan_xstream(m_local, n, k, x_dtype, h->sm_count, es ? atoi(es) : 0, &h->plan);   // arguments checked above
    }
    const prmf_xstream_pass &p1 = h->plan.pass1, &p2 = h->plan.pass2;
    if (h->x32) {
        h->ldx32 = round_up(n, 32);
        h->ldxt32 = round_up(std::max<int64_t>(1, m_local), 32);
    }
    if (h->x_tc) setup_tf32(h);
    {
        const char* ee = getenv("PRMF_EPI");
        h->use_epi = !(ee && atoi(ee) == 0) && k <= 10 && m_local > 0 && !h->x_tc &&
                     p1.panels * p1.chunks <= h->sm_count && p2.panels * p2.chunks <= h->sm_count;
    }
    const int gu_parts_max = (int)std::max<int64_t>(h->uu_grid, h->use_epi ? p1.panels : 0);
    const int gv_parts_max = (int)std::max<int64_t>(h->vu_grid, h->use_epi ? p2.panels : 0);

    int rc = 0;
    const int64_t nk = n * k;
    const int kk2 = k * k;
    const int64_t pad_rows = 16;      // bulk copies of W read up to one stage past the last row
    h->obj_capacity = 256;
    {
        auto pad = [](size_t count, size_t elem) { return ((count ? count : 1) * elem + 255) & ~(size_t)255; };
        const size_t d = sizeof(double);
        size_t total = 0;
        total += 3 * pad((size_t)(m_local + pad_rows) * k, d);                                      // U, U2, Ub
        total += pad((size_t)a_chunks(h) * std::max<int64_t>(1, m_local) * k, d);                  // Apart
        total += 2 * pad((size_t)(n + pad_rows) * k, d) + pad((size_t)nk, d);                      // Vbuf[2], Vb
        total += pad(128, d) + 4 * pad(kk2, d) + pad((size_t)gu_parts_max * kk2, d) + pad((size_t)gv_parts_max * kk2, d);
        total += pad(gv_parts_max, d) + pad((size_t)b_chunks(h) * nk, d);                           // VB_part, Bpart
        total += pad(2 * ((size_t)p1.panels + p2.panels) + 2, sizeof(unsigned long long));     // fused-tail counters
        total += pad(2 * ((size_t)p1.panels + p2.panels) + 4, sizeof(unsigned long long)) + pad(1, sizeof(unsigned int));   // block kernel
        total += pad((size_t)std::max(p1.panels * p1.chunks, p2.panels * p2.chunks) * kk2, d) +
                 pad((size_t)p2.panels * p2.chunks, d);                                          // per-CTA partials
        total += pad((size_t)nk + kk2 + 2, d) + pad(1, d) + pad((size_t)h->sm_count * 8, d) + pad(2, d);
        total += pad(1, sizeof(int)) + pad(1, sizeof(unsigned int)) + pad(k, sizeof(int32_t)) + pad(nk, sizeof(int32_t));
        total += pad((size_t)h->obj_capacity * kObjStride, d);
        cudaError_t ea = h->arena.reserve(total, device);
        if (ea != cudaSuccess) rc = fail(h, PRMF_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", total, cudaGetErrorString(ea));
    }
#define ALLOC(ptr, count) if (!rc) rc = dalloc(h, &ptr, (size_t)(count))
#define TAKE(ptr, T, count) if (!rc) { ptr = h->arena.take<T>((size_t)(count)); if (!ptr) rc = fail(h, PRMF_ERR_NOMEM, "arena exhausted"); }
#define ALLOC_BIG(ptr, T, count)                                                                                   \
    if (!rc) {                                                                                                       \
        const size_t bytes_ = sizeof(T) * (size_t)(count);                                                           \
        cudaError_t eb_ = g_pool.alloc((void**)&ptr, bytes_, device);                                                \
        if (eb_ != cudaSuccess) { ptr = nullptr; rc = fail(h, PRMF_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", bytes_, cudaGetErrorString(eb_)); } \
    }
    if (h->x32) {
        ALLOC_BIG(h->X32, float, (size_t)std::max<int64_t>(1, m_local) * h->ldx32);
        ALLOC_BIG(h->Xt32, float, (size_t)n * h->ldxt32);
    }
    if (h->x_tc) {
        ALLOC(h->Vt32, (size_t)h->Kp * h->ldx32);
        ALLOC(h->Ut32, (size_t)h->Kp * h->ldxt32);
    }
    if (!h->x32) {
        ALLOC_BIG(h->X, double, (size_t)std::max<int64_t>(1, m_local) * h->ldx);
        ALLOC_BIG(h->Xt, double, (size_t)n * h->ldxt);
    }
#undef ALLOC_BIG
    TAKE(h->U, double, (m_local + pad_rows) * k);
    TAKE(h->Ub, double, (m_local + pad_rows) * k);
    TAKE(h->U2, double, (m_local + pad_rows) * k);
    TAKE(h->Apart, double, (size_t)a_chunks(h) * std::max<int64_t>(1, m_local) * k);
    TAKE(h->Vbuf[0], double, (n + pad_rows) * k); TAKE(h->Vbuf[1], double, (n + pad_rows) * k); TAKE(h->Vb, double, nk);
    TAKE(h->Gv, double, kk2); TAKE(h->Gvb, double, kk2); TAKE(h->Gu_glob, double, kk2); TAKE(h->mi_part, double, 128); TAKE(h->Gv_red, double, kk2);
    TAKE(h->Gu_part, double, (size_t)gu_parts_max * kk2);
    TAKE(h->Gv_part, double, (size_t)gv_parts_max * kk2);
    TAKE(h->VB_part, double, gv_parts_max);
    TAKE(h->epi_counters, unsigned long long, 2 * ((size_t)p1.panels + p2.panels) + 2);
    TAKE(h->blk_ctr, unsigned long long, 2 * ((size_t)p1.panels + p2.panels) + 4);
    TAKE(h->err_word, unsigned int, 1);
    TAKE(h->epi_part2, double, (size_t)std::max(p1.panels * p1.chunks, p2.panels * p2.chunks) * kk2);
    TAKE(h->epi_vb2, double, (size_t)p2.panels * p2.chunks);
    TAKE(h->Bpart, double, (size_t)b_chunks(h) * nk);
    TAKE(h->red, double, (size_t)nk + kk2 + 2);
    TAKE(h->normX_sq, double, 1);
    TAKE(h->scal_part, double, (size_t)h->sm_count * 8);
    TAKE(h->gd, double, 2);
    TAKE(h->step_counter, int, 1);
    TAKE(h->ticket, unsigned int, 1);
    TAKE(h->active, int32_t, k);
    TAKE(h->pos, int32_t, nk);
    TAKE(h->obj, double, (size_t)h->obj_capacity * kObjStride);
#undef TAKE
#undef ALLOC
    if (!rc && h->x32) cudaMemsetAsync(h->Xt32, 0, sizeof(float) * n * h->ldxt32, h->stream);
    if (!rc && h->x_tc) {
        cudaMemsetAsync(h->Vt32, 0, sizeof(float) * h->Kp * h->ldx32, h->stream);
        cudaMemsetAsync(h->Ut32, 0, sizeof(float) * h->Kp * h->ldxt32, h->stream);
        rc = finish_setup_tf32(h);
    }
    if (!rc) {
        if (h->Xt) cudaMemsetAsync(h->Xt, 0, sizeof(double) * n * h->ldxt, h->stream);
        cudaMemsetAsync(h->ticket, 0, sizeof(unsigned int), h->stream);
        cudaMemsetAsync(h->epi_counters, 0, sizeof(unsigned long long) * (2 * ((size_t)p1.panels + p2.panels) + 2), h->stream);
        cudaMemsetAsync(h->blk_ctr, 0, sizeof(unsigned long long) * (2 * ((size_t)p1.panels + p2.panels) + 4), h->stream);
        cudaMemsetAsync(h->err_word, 0, sizeof(unsigned int), h->stream);
        cudaMemsetAsync(h->U, 0, sizeof(double) * (m_local + pad_rows) * k, h->stream);
        cudaMemsetAsync(h->U2, 0, sizeof(double) * (m_local + pad_rows) * k, h->stream);
        cudaMemsetAsync(h->Vbuf[0], 0, sizeof(double) * (n + pad_rows) * k, h->stream);
        cudaMemsetAsync(h->Vbuf[1], 0, sizeof(double) * (n + pad_rows) * k, h->stream);
        cudaMemsetAsync(h->red, 0, sizeof(double) * (nk + kk2 + 2), h->stream);
        cudaMemsetAsync(h->Gu_part, 0, sizeof(double) * gu_parts_max * kk2, h->stream);
        e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) rc = fail(h, PRMF_ERR_CUDA, "init memset: %s", cudaGetErrorString(e));
    }
    if (!rc && h->use_epi) {
        const char* ed = getenv("PRMF_DEFER_OBJ");
        if (!(ed && atoi(ed) == 0)) {
            const size_t H = (size_t)h->obj_capacity, kk2s = (size_t)kk2;
            const size_t n_gu = H * kk2s, n_gvp = H * p2.panels * kk2s, n_vbp = H * p2.panels, n_vh = H * kVhCap;
            h->hist_bytes = sizeof(double) * (n_gu + n_gvp + n_vbp + n_vh);
            if (g_pool.alloc((void**)&h->hist, h->hist_bytes, device) == cudaSuccess) {
                h->hist_Gu = h->hist;
                h->hist_Gvp = h->hist_Gu + n_gu;
                h->hist_VBp = h->hist_Gvp + n_gvp;
                h->hist_vh = h->hist_VBp + n_vbp;
                h->defer_ok = true;
            }
        }
    }
    if (!rc) {
        // persistent step kernel: needs the fused-tail geometry, the per-step history of the deferred objective, and
        // ring + tail scratch within the shared memory of one CTA
        const char* eb = getenv("PRMF_BLOCK");
        const char* et = getenv("PRMF_SPIN_TIMEOUT_MS");
        if (et && atof(et) > 0) h->spin_timeout_ns = (unsigned long long)(atof(et) * 1e6);
        const size_t wb = ((size_t)kBlkRS * k * 8 + 127) & ~(size_t)127;
        h->blk_stage_bytes = (uint32_t)((size_t)kBlkRS * std::max(p1.panel_w, p2.panel_w) * 8 + wb);
        h->blk_smem = (size_t)h->plan.stages * h->blk_stage_bytes + 2 * h->plan.stages * sizeof(uint64_t) +
                      sizeof(double) * (256 + 8 * (size_t)k * k + (size_t)kBlkRowsCap * k);
        // (block_kernel streams fp64 X: not for fp32 storage, where PRMF_BLOCK=1 is ignored)
        h->use_block = h->use_epi && h->defer_ok && !h->x32 && !(eb && atoi(eb) == 0) && h->blk_smem <= 227 * 1024;
        h->block_forced = eb && atoi(eb) == 1;
        h->err_host = pinned_word();
    }
    // opt in to large dynamic shared memory where k needs it
    if (!rc && h->big_k) {
        if (h->tiled_cpt == 2) rc = set_smem(h, u_update_tiled_kernel<2, 2>, h->tiled_smem);
        else if (h->tiled_cpt == 4) rc = set_smem(h, u_update_tiled_kernel<4, 2>, h->tiled_smem);
        else rc = set_smem(h, u_update_tiled_kernel<8, 2>, h->tiled_smem);
        if (!rc && h->tiled_cpt == 2) rc = set_smem(h, v_update_tiled_kernel<2, 2>, h->tiled_smem);
        else if (!rc && h->tiled_cpt == 4) rc = set_smem(h, v_update_tiled_kernel<4, 2>, h->tiled_smem);
        else if (!rc) rc = set_smem(h, v_update_tiled_kernel<8, 2>, h->tiled_smem);
        if (!rc) rc = set_smem(h, objective_kernel, obj_smem(h));
    }
    if (!rc) {
        NQ_SWITCH(h->nq, {
            if (!rc) rc = set_smem(h, gram_rows_kernel<NQ>, gram_smem(h));
        });
        NI_SWITCH(h->ni, {
            if (!rc) rc = set_smem(h, u_update_kernel<NI>, uu_smem(h));
            if (!rc) rc = set_smem(h, v_update_objective_kernel<NI>, vu_smem(h));
        });
    }
    if (rc) {
        g_create_error = h->err;
        prmf_destroy(h);
        return rc;
    }
    *out = h;
    return PRMF_OK;
}

int prmf_destroy(prmf_handle* h) {
    if (!h) return PRMF_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    harvest_events(h);
    if (h->p2p_ready)
        for (int r = 0; r < h->nranks; ++r)
            if (r != h->rank && h->peer_base[r]) cudaIpcCloseMemHandle(h->peer_base[r]);
    if (h->ev_sync) cudaEventDestroy(h->ev_sync);
    if (h->p2p_buf) cudaFree(h->p2p_buf);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    g_pool.release(h->X, sizeof(double) * (size_t)std::max<int64_t>(1, h->m) * h->ldx, h->device);
    g_pool.release(h->Xt, sizeof(double) * (size_t)h->n * h->ldxt, h->device);
    g_pool.release(h->hist, h->hist_bytes, h->device);
    g_pool.release(h->X32, sizeof(float) * (size_t)std::max<int64_t>(1, h->m) * h->ldx32, h->device);
    g_pool.release(h->Xt32, sizeof(float) * (size_t)h->n * h->ldxt32, h->device);
    if (h->Vt32) cudaFree(h->Vt32);
    if (h->Ut32) cudaFree(h->Ut32);
    h->arena.release();
    h->pw_arena.release();
    h->as_arena.release();
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return PRMF_OK;
}

int prmf_set_X(prmf_handle* h, const double* X_host, int64_t ld) {
    if (!h) return PRMF_ERR_ARG;
    if ((!X_host && h->m > 0) || ld < h->n) return fail(h, PRMF_ERR_ARG, "prmf_set_X: bad pointer or ld < n");
    CU(cudaSetDevice(h->device));
    if (h->x32) {
        int rc = store_x32<double>(h, X_host, ld, true);
        return rc ? rc : finish_X(h);
    }
    if (h->m > 0) {
        CU(cudaMemsetAsync(h->X, 0, sizeof(double) * h->m * h->ldx, h->stream));
        CU(cudaMemcpy2DAsync(h->X, h->ldx * sizeof(double), X_host, ld * sizeof(double), h->n * sizeof(double),
                             h->m, cudaMemcpyHostToDevice, h->stream));
    }
    return finish_X(h);
}

int prmf_set_X_device(prmf_handle* h, const double* X_dev, int64_t ld) {
    if (!h) return PRMF_ERR_ARG;
    if ((!X_dev && h->m > 0) || ld < h->n) return fail(h, PRMF_ERR_ARG, "prmf_set_X_device: bad pointer or ld < n");
    CU(cudaSetDevice(h->device));
    if (h->x32) {
        int rc = store_x32<double>(h, X_dev, ld, false);
        return rc ? rc : finish_X(h);
    }
    if (h->m > 0) {
        CU(cudaMemsetAsync(h->X, 0, sizeof(double) * h->m * h->ldx, h->stream));
        CU(cudaMemcpy2DAsync(h->X, h->ldx * sizeof(double), X_dev, ld * sizeof(double), h->n * sizeof(double),
                             h->m, cudaMemcpyDeviceToDevice, h->stream));
    }
    return finish_X(h);
}

int prmf_set_X_f32(prmf_handle* h, const float* X, int64_t ld, int on_device) {
    if (!h) return PRMF_ERR_ARG;
    if (!h->x32) return fail(h, PRMF_ERR_STATE, "prmf_set_X_f32 needs a handle created with PRMF_X_TF32 or PRMF_X_F32");
    if ((!X && h->m > 0) || ld < h->n) return fail(h, PRMF_ERR_ARG, "prmf_set_X_f32: bad pointer or ld < n");
    CU(cudaSetDevice(h->device));
    int rc = store_x32<float>(h, X, ld, on_device == 0);
    return rc ? rc : finish_X(h);
}

int prmf_x_dtype(const prmf_handle* h) {
    if (!h || !h->x32) return PRMF_X_F64;
    return h->x_tc ? PRMF_X_TF32 : PRMF_X_F32;
}

int prmf_get_normX_sq(prmf_handle* h, double* out) {
    if (!h || !out) return PRMF_ERR_ARG;
    if (!h->have_X) return fail(h, PRMF_ERR_STATE, "X not set");
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(out, h->normX_sq, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return PRMF_OK;
}

int prmf_set_pathways(prmf_handle* h, int32_t P, const int64_t* path_ptr, const int32_t* support_idx,
                      const int64_t* row_ptr, const int32_t* col_local, const double* w) {
    if (!h) return PRMF_ERR_ARG;
    if (P <= 0 || !path_ptr || !row_ptr) return fail(h, PRMF_ERR_ARG, "prmf_set_pathways: P <= 0 or NULL tables");
    const int64_t S = path_ptr[P];
    if (path_ptr[0] != 0 || S < 0) return fail(h, PRMF_ERR_ARG, "path_ptr must start at 0");
    const int64_t E = row_ptr[S];
    if ((S > 0 && !support_idx) || (E > 0 && (!col_local || !w))) return fail(h, PRMF_ERR_ARG, "NULL pathway arrays");
    // validate + derive deg, diag(L), diag(L)^-1/2 on the host (pow(x,-0.5) as numpy does, :58-62)
    std::vector<double> deg(S, 0.0), ldiag(S, 0.0), isd(S, 0.0);
    for (int32_t p = 0; p < P; ++p) {
        const int64_t beg = path_ptr[p], end = path_ptr[p + 1];
        if (end < beg) return fail(h, PRMF_ERR_ARG, "path_ptr not monotone at pathway %d", p);
        const int64_t sp = end - beg;
        for (int64_t r = beg; r < end; ++r) {
            if (support_idx[r] < 0 || support_idx[r] >= h->n)
                return fail(h, PRMF_ERR_ARG, "support index %d out of range at row %lld", support_idx[r], (long long)r);
            if (row_ptr[r + 1] < row_ptr[r]) return fail(h, PRMF_ERR_ARG, "row_ptr not monotone at row %lld", (long long)r);
            double d = 0.0, self = 0.0;
            for (int64_t e2 = row_ptr[r]; e2 < row_ptr[r + 1]; ++e2) {
                if (col_local[e2] < 0 || col_local[e2] >= sp)
                    return fail(h, PRMF_ERR_ARG, "col_local out of range at entry %lld", (long long)e2);
                d += w[e2];
                if (beg + col_local[e2] == r) self += w[e2];
            }
            deg[r] = d;
            ldiag[r] = d - self;
            isd[r] = ldiag[r] != 0.0 ? std::pow(ldiag[r], -0.5) : 0.0;
        }
    }
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    h->pw_arena.release();
    {
        auto pad = [](size_t bytes) { return (bytes + 255) & ~(size_t)255; };
        const size_t total = pad(sizeof(int64_t) * (P + 1)) + pad(sizeof(int32_t) * std::max<int64_t>(1, S)) +
                             pad(sizeof(int64_t) * (S + 1)) + pad(sizeof(int32_t) * std::max<int64_t>(1, E)) +
                             pad(sizeof(double) * std::max<int64_t>(1, E)) + 3 * pad(sizeof(double) * std::max<int64_t>(1, S)) +
                             pad(sizeof(double) * 3 * (size_t)h->k * P);
        cudaError_t ea = h->pw_arena.reserve(total, h->device);
        if (ea != cudaSuccess) return fail(h, PRMF_ERR_NOMEM, "cudaMalloc pathways (%zu bytes): %s", total, cudaGetErrorString(ea));
    }
    int rc = 0;
    auto up = [&](const void* src, size_t bytes, const void** dst) -> int {
        unsigned char* d = h->pw_arena.take<unsigned char>(bytes);
        if (!d) return fail(h, PRMF_ERR_NOMEM, "pathway arena exhausted");
        if (bytes) {
            cudaError_t e = cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, h->stream);
            if (e != cudaSuccess) return fail(h, PRMF_ERR_CUDA, "copy pathways: %s", cudaGetErrorString(e));
        }
        *dst = d;
        return 0;
    };
    Pathways pw{};
    pw.P = P;
    if (!rc) rc = up(path_ptr, sizeof(int64_t) * (P + 1), (const void**)&pw.path_ptr);
    if (!rc) rc = up(support_idx, sizeof(int32_t) * S, (const void**)&pw.support_idx);
    if (!rc) rc = up(row_ptr, sizeof(int64_t) * (S + 1), (const void**)&pw.row_ptr);
    if (!rc) rc = up(col_local, sizeof(int32_t) * E, (const void**)&pw.col_local);
    if (!rc) rc = up(w, sizeof(double) * E, (const void**)&pw.w);
    if (!rc) rc = up(deg.data(), sizeof(double) * S, (const void**)&pw.deg);
    if (!rc) rc = up(ldiag.data(), sizeof(double) * S, (const void**)&pw.ldiag);
    if (!rc) rc = up(isd.data(), sizeof(double) * S, (const void**)&pw.isd);
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));
    h->scores_buf = h->pw_arena.take<double>((size_t)3 * h->k * P);
    if (!h->scores_buf) return fail(h, PRMF_ERR_NOMEM, "pathway arena exhausted (scores)");
    h->pw = pw; h->S = S; h->E = E;
    h->max_support = 0;
    h->max_edges = 0;
    for (int32_t p = 0; p < P; ++p) {
        h->max_support = std::max(h->max_support, path_ptr[p + 1] - path_ptr[p]);
        h->max_edges = std::max(h->max_edges, row_ptr[path_ptr[p + 1]] - row_ptr[path_ptr[p]]);
    }
    h->path_ptr_host.assign(path_ptr, path_ptr + P + 1);
    h->row_ptr_host.assign(row_ptr, row_ptr + S + 1);
    h->have_pw = true;
    h->have_active = false;
    h->pos_dirty = true;
    {   // every factor may pick the largest pathway: size the active-set arrays for that now, not in the middle of a block
        const int64_t nd = std::max<int64_t>((int64_t)h->k * h->max_support, 1024);
        const int64_t no = std::max<int64_t>((int64_t)h->k * h->max_edges, 4096);
        if (nd > h->as_cap_diag || no > h->as_cap_off || !h->as_i32) {
            int rc2 = alloc_active_arena(h, nd, no);
            if (rc2) return rc2;
        }
    }
    return PRMF_OK;
}

int prmf_set_UV(prmf_handle* h, const double* U_local, const double* V) {
    if (!h) return PRMF_ERR_ARG;
    CU(cudaSetDevice(h->device));
    cancel_ahead(h);
    if (U_local && h->m > 0)
        CU(cudaMemcpyAsync(h->U, U_local, sizeof(double) * h->m * h->k, cudaMemcpyHostToDevice, h->stream));
    if (V) {
        const int64_t nk = h->n * h->k;
        CU(cudaMemcpyAsync(h->Vbuf[h->vcur], V, sizeof(double) * nk, cudaMemcpyHostToDevice, h->stream));
        int rc = recompute_Gv(h);
        if (rc) return rc;
        if (h->x_tc && (rc = refresh_wt(h, h->Vbuf[h->vcur], h->n, h->Vt32, h->ldx32))) return rc;
    }
    CU(cudaStreamSynchronize(h->stream));
    if (U_local || h->m == 0) h->have_U = true;          // a handle without rows has no U to set
    if (V) h->have_V = true;
    return PRMF_OK;
}

int prmf_get_UV(prmf_handle* h, double* U_local, double* V) {
    if (!h) return PRMF_ERR_ARG;
    CU(cudaSetDevice(h->device));
    if (U_local && h->m > 0)
        CU(cudaMemcpyAsync(U_local, cur_U(h), sizeof(double) * h->m * h->k, cudaMemcpyDeviceToHost, h->stream));
    if (V) CU(cudaMemcpyAsync(V, h->Vbuf[h->vcur], sizeof(double) * h->n * h->k, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return PRMF_OK;
}

int prmf_set_active(prmf_handle* h, const int32_t* pathway_of_factor) {
    if (!h || !pathway_of_factor) return PRMF_ERR_ARG;
    if (!h->have_pw) return fail(h, PRMF_ERR_STATE, "pathways not set");
    for (int c = 0; c < h->k; ++c)
        if (pathway_of_factor[c] < 0 || pathway_of_factor[c] >= h->pw.P)
            return fail(h, PRMF_ERR_ARG, "active pathway %d of factor %d out of range", pathway_of_factor[c], c);
    CU(cudaSetDevice(h->device));
    h->active_host.assign(pathway_of_factor, pathway_of_factor + h->k);
    CU(cudaMemcpyAsync(h->active, h->active_host.data(), sizeof(int32_t) * h->k, cudaMemcpyHostToDevice, h->stream));
    h->have_active = true;
    h->pos_dirty = true;
    return PRMF_OK;
}

int prmf_step_async(prmf_handle* h, int n_steps, double gamma, double delta, double tradeoff) {
    if (!h) return PRMF_ERR_ARG;
    return enqueue_steps(h, n_steps, gamma, delta, tradeoff);
}

int prmf_step_collect(prmf_handle* h, int n_steps, double* obj_parts, double* gamma_delta_out) {
    if (!h) return PRMF_ERR_ARG;
    return collect(h, n_steps, obj_parts, gamma_delta_out);
}

int prmf_step(prmf_handle* h, int n_steps, double gamma, double delta, double tradeoff, double* obj_parts,
              double* gamma_delta_out) {
    if (!h) return PRMF_ERR_ARG;
    int rc = enqueue_steps(h, n_steps, gamma, delta, tradeoff);
    if (rc) return rc;
    return collect(h, n_steps, obj_parts, gamma_delta_out);
}

int prmf_scores(prmf_handle* h, double* mass, double* quad_norm, double* quad_raw) {
    if (!h) return PRMF_ERR_ARG;
    if (!h->have_pw || !h->have_V) return fail(h, PRMF_ERR_STATE, "prmf_scores needs pathways and V");
    CU(cudaSetDevice(h->device));
    const size_t cnt = (size_t)h->k * h->pw.P;
    double* d = h->scores_buf;
    int rc_s = launch_scores(h);
    if (rc_s) return rc_s;
    if (mass) CU(cudaMemcpyAsync(mass, d, cnt * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (quad_norm) CU(cudaMemcpyAsync(quad_norm, d + cnt, cnt * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (quad_raw) CU(cudaMemcpyAsync(quad_raw, d + 2 * cnt, cnt * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return PRMF_OK;
}

int prmf_block_end(prmf_handle* h, int n_steps, double* obj_parts, double* gamma_delta_out, int want_scores,
                   double* mass, double* quad_norm, double* quad_raw, int prefetch) {
    if (!h) return PRMF_ERR_ARG;
    CU(cudaSetDevice(h->device));
    if (n_steps > h->obj_capacity) return fail(h, PRMF_ERR_ARG, "prmf_block_end: more steps than were run");
    if (want_scores) {
        if (!h->have_pw || !h->have_V) return fail(h, PRMF_ERR_STATE, "prmf_block_end needs pathways and V for the scores");
        const size_t cnt = (size_t)h->k * h->pw.P;
        double* d = h->scores_buf;
        int rc_s = launch_scores(h);
        if (rc_s) return rc_s;
        if (mass) CU(cudaMemcpyAsync(mass, d, cnt * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (quad_norm) CU(cudaMemcpyAsync(quad_norm, d + cnt, cnt * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (quad_raw) CU(cudaMemcpyAsync(quad_raw, d + 2 * cnt, cnt * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    }
    if (obj_parts && n_steps > 0)
        CU(cudaMemcpyAsync(obj_parts, h->obj, sizeof(double) * n_steps * kObjStride, cudaMemcpyDeviceToHost, h->stream));
    if (gamma_delta_out)
        CU(cudaMemcpyAsync(gamma_delta_out, h->gd, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (h->err_host) CU(cudaMemcpyAsync(h->err_host, h->err_word, sizeof(unsigned int), cudaMemcpyDeviceToHost, h->stream));
    if (!h->ev_sync) CU(cudaEventCreateWithFlags(&h->ev_sync, cudaEventDisableTiming));
    CU(cudaEventRecord(h->ev_sync, h->stream));
    if (prefetch) {
        int rc = prefetch_pass1(h);              // streams X while the host digests the tables
        if (rc) return rc;
    }
    CU(cudaEventSynchronize(h->ev_sync));
    if (h->profiling) {
        CU(cudaStreamSynchronize(h->stream));
        harvest_events(h);
    }
    int rc_e = check_err_word(h, h->err_host ? *h->err_host : 0u);
    if (rc_e) return rc_e;
    return refine_last_row(h, n_steps, obj_parts);
}

int prmf_snapshot_best(prmf_handle* h) {
    if (!h) return PRMF_ERR_ARG;
    CU(cudaSetDevice(h->device));
    if (h->m > 0) CU(cudaMemcpyAsync(h->Ub, cur_U(h), sizeof(double) * h->m * h->k, cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaMemcpyAsync(h->Vb, h->Vbuf[h->vcur], sizeof(double) * h->n * h->k, cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaMemcpyAsync(h->Gvb, h->Gv, sizeof(double) * h->k * h->k, cudaMemcpyDeviceToDevice, h->stream));
    return PRMF_OK;
}

int prmf_restore_best(prmf_handle* h) {
    if (!h) return PRMF_ERR_ARG;
    CU(cudaSetDevice(h->device));
    cancel_ahead(h);
    if (h->m > 0) CU(cudaMemcpyAsync(h->U, h->Ub, sizeof(double) * h->m * h->k, cudaMemcpyDeviceToDevice, h->stream));
    const int64_t nk = h->n * h->k;
    CU(cudaMemcpyAsync(h->Vbuf[h->vcur], h->Vb, sizeof(double) * nk, cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaMemcpyAsync(h->Gv, h->Gvb, sizeof(double) * h->k * h->k, cudaMemcpyDeviceToDevice, h->stream));
    if (h->x_tc) {
        int rc = refresh_wt(h, h->Vbuf[h->vcur], h->n, h->Vt32, h->ldx32);
        if (rc) return rc;
    }
    CU(cudaStreamSynchronize(h->stream));
    return PRMF_OK;
}

int prmf_residual_sq(prmf_handle* h, double* out) {
    if (!h || !out) return PRMF_ERR_ARG;
    if (!h->have_X || !h->have_U || !h->have_V) return fail(h, PRMF_ERR_STATE, "prmf_residual_sq needs X and U/V");
    CU(cudaSetDevice(h->device));
    const int blocks = h->sm_count * 4;
    double* d = nullptr;
    int rc = dalloc(h, &d, 1);
    if (rc) return rc;
    if (h->m > 0) {
        if (h->x32)
            residual_f32_kernel<<<blocks, 256, 0, h->stream>>>(h->X32, h->ldx32, h->m, (int)h->n, cur_U(h), h->Vbuf[h->vcur], h->k,
                                                                h->scal_part);
        else
            residual_kernel<<<blocks, 256, 0, h->stream>>>(h->X, h->ldx, h->m, (int)h->n, cur_U(h), h->Vbuf[h->vcur], h->k, h->scal_part);
        h->launches++;
        sum_partials_kernel<<<1, 256, 0, h->stream>>>(h->scal_part, blocks, d);
        h->launches++;
    } else {
        cudaMemsetAsync(d, 0, sizeof(double), h->stream);
    }
    rc = allreduce(h, d, 1);
    cudaError_t e = cudaGetLastError();
    if (!rc && e == cudaSuccess) e = cudaMemcpyAsync(out, d, sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(h, PRMF_ERR_CUDA, "prmf_residual_sq: %s", cudaGetErrorString(e));
    return PRMF_OK;
}

int prmf_objective(prmf_handle* h, double gamma, double delta, double* out) {
    if (!h || !out) return PRMF_ERR_ARG;
    if (!h->have_X || !h->have_U || !h->have_V || !h->have_pw || !h->have_active)
        return fail(h, PRMF_ERR_STATE, "prmf_objective needs X, U/V, pathways and the active set");
    CU(cudaSetDevice(h->device));
    int rc = ensure_pos(h);
    if (rc) return rc;
    double r2 = 0.0;
    if ((rc = prmf_residual_sq(h, &r2))) return rc;                            // ||X - U V^T||^2, explicit pass (:337)
    double* d = nullptr;
    if ((rc = dalloc(h, &d, 4))) return rc;
    const int blocks = h->sm_count * 4;
    const int64_t mk = h->m * h->k;
    if (mk > 0) {                                                              // sum(U^2) (:359); U is zero padded
        sumsq_kernel<<<blocks, 256, 0, h->stream>>>(cur_U(h), mk + 2, 1, (int)round_up(mk, 2), h->scal_part);
        h->launches++;
        sum_partials_kernel<<<1, 256, 0, h->stream>>>(h->scal_part, blocks, d + 2);
        h->launches++;
    } else {
        cudaMemsetAsync(d + 2, 0, sizeof(double), h->stream);
    }
    rc = allreduce(h, d + 2, 1);
    manifold_ignore_kernel<<<1, 1024, 0, h->stream>>>(h->Vbuf[h->vcur], h->k, h->Gv, h->as, d);
    h->launches++;
    double host[3] = {0, 0, 0};
    cudaError_t e = cudaGetLastError();
    if (!rc && e == cudaSuccess) e = cudaMemcpyAsync(host, d, 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(h, PRMF_ERR_CUDA, "prmf_objective: %s", cudaGetErrorString(e));
    const double recon = std::sqrt(r2 > 0.0 ? r2 : 0.0);
    out[0] = recon; out[1] = host[0]; out[2] = host[1]; out[3] = host[2];
    out[4] = recon + gamma * host[0] + delta * host[1] + host[2];              // :362
    out[5] = gamma; out[6] = delta; out[7] = r2;
    return PRMF_OK;
}

int prmf_nccl_load(const char* libnccl_path) {
    const char* err = g_nccl.load(libnccl_path);
    if (err) return fail(nullptr, PRMF_ERR_NCCL, "%s", err);
    return PRMF_OK;
}

int prmf_comm_unique_id(uint8_t* id_out) {
    if (!id_out) return PRMF_ERR_ARG;
    if (!g_nccl.loaded()) return fail(nullptr, PRMF_ERR_NCCL, "call prmf_nccl_load first");
    NcclUniqueId id;
    int r = g_nccl.GetUniqueId(&id);
    if (r != 0) return fail(nullptr, PRMF_ERR_NCCL, "ncclGetUniqueId failed (%d)", r);
    memcpy(id_out, id.internal, PRMF_UNIQUE_ID_BYTES);
    return PRMF_OK;
}

int prmf_comm_init(prmf_handle* h, int rank, int nranks, const uint8_t* id) {
    if (!h || !id) return PRMF_ERR_ARG;
    if (h->x32 && !h->x_tc) return fail(h, PRMF_ERR_STATE, "PRMF_X_F32 handles are single-rank: no communicator");
    if (!g_nccl.loaded()) return fail(h, PRMF_ERR_NCCL, "call prmf_nccl_load first");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(h, PRMF_ERR_ARG, "bad rank %d / %d", rank, nranks);
    CU(cudaSetDevice(h->device));
    NcclUniqueId uid;
    memcpy(uid.internal, id, PRMF_UNIQUE_ID_BYTES);
    int r = g_nccl.CommInitRank(&h->comm, nranks, uid, rank);
    if (r != 0) {
        h->comm = nullptr;
        return fail(h, PRMF_ERR_NCCL, "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
    }
    h->rank = rank; h->nranks = nranks;
    return PRMF_OK;
}

int prmf_p2p_export(prmf_handle* h, uint8_t* handle_out) {
    if (!h || !handle_out) return PRMF_ERR_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == PRMF_IPC_HANDLE_BYTES, "IPC handle size");
    CU(cudaSetDevice(h->device));
    if (!h->p2p_buf) {
        // [red parity 0 | red parity 1 | 64 peer-barrier flag words | push receive slots | small all-reduce slots], in
        // doubles; it depends on n and k only, so every rank computes the same offsets into every rank's buffer
        h->p2p_red_count = (size_t)round_up(h->n * h->k + (int64_t)h->k * h->k + 2, 32);
        const size_t flags_end = 2 * h->p2p_red_count + 64;
        const size_t xbuf_at = (flags_end + 1) & ~(size_t)1;                   // 16-byte aligned
        // push exchange of the persistent step kernel: receive slots [parity][source rank][n*k + k*k] + its flags
        h->xcount = h->p2p_red_count;
        const size_t xdoubles = 2 * 2 * (size_t)kMaxPeers * h->xcount;        // 16-byte {value, sequence} entries
        const size_t sdoubles = 2 * 2 * (size_t)kMaxPeers * kSmallAllreduceMax;   // set-up scalars without NCCL
        const size_t total = xbuf_at + xdoubles + sdoubles;
        int rc = dalloc(h, &h->p2p_buf, total);
        if (rc) return rc;
        CU(cudaMemset(h->p2p_buf, 0, total * sizeof(double)));
        h->xbuf = h->p2p_buf + xbuf_at;
        h->xsmall = h->xbuf + xdoubles;
    }
    cudaIpcMemHandle_t hd;
    CU(cudaIpcGetMemHandle(&hd, h->p2p_buf));
    memcpy(handle_out, &hd, sizeof hd);
    return PRMF_OK;
}

int prmf_p2p_attach(prmf_handle* h, int rank, int nranks, const uint8_t* handles) {
    if (!h || !handles) return PRMF_ERR_ARG;
    if (h->x32 && !h->x_tc) return fail(h, PRMF_ERR_STATE, "PRMF_X_F32 handles are single-rank: no peer exchange");
    if (!h->p2p_buf) return fail(h, PRMF_ERR_STATE, "call prmf_p2p_export first");
    if (nranks < 2 || nranks > kMaxPeers || rank < 0 || rank >= nranks)
        return fail(h, PRMF_ERR_ARG, "prmf_p2p_attach: bad rank %d / %d (max %d ranks)", rank, nranks, kMaxPeers);
    if (h->comm && (h->rank != rank || h->nranks != nranks))
        return fail(h, PRMF_ERR_ARG, "prmf_p2p_attach: rank/nranks differ from prmf_comm_init");
    CU(cudaSetDevice(h->device));
    for (int r = 0; r < nranks; ++r) {
        if (r == rank) { h->peer_base[r] = h->p2p_buf; continue; }
        cudaIpcMemHandle_t hd;
        memcpy(&hd, handles + (size_t)r * PRMF_IPC_HANDLE_BYTES, sizeof hd);
        cudaError_t e = cudaIpcOpenMemHandle(&h->peer_base[r], hd, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            for (int q = 0; q < r; ++q)
                if (q != rank && h->peer_base[q]) { cudaIpcCloseMemHandle(h->peer_base[q]); h->peer_base[q] = nullptr; }
            return fail(h, PRMF_ERR_CUDA, "cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
        }
    }
    h->rank = rank; h->nranks = nranks;
    h->p2p_ready = true;
    return PRMF_OK;
}

int prmf_p2p_finalize(prmf_handle* h) {
    if (!h) return PRMF_ERR_ARG;
    if (!h->p2p_ready) return fail(h, PRMF_ERR_STATE, "prmf_p2p_finalize needs prmf_p2p_attach (and prmf_comm_init unless NCCL is not used)");
    CU(cudaSetDevice(h->device));
    // The persistent step kernel is used only if EVERY rank can take it (ranks that disagreed would wait on flags
    // nobody writes), and its push exchange pairs CTA c of every rank, so all ranks must split the genes the same
    // way: [persistent step kernel possible | pass-2 chunks | chunks^2], summed over ranks
    const double chunks = (double)h->plan.pass2.chunks;
    const double mine[3] = {h->use_block ? 1.0 : 0.0, chunks, chunks * chunks};
    CU(cudaMemcpyAsync(h->scal_part, mine, sizeof mine, cudaMemcpyHostToDevice, h->stream));
    int rc = allreduce(h, h->scal_part, 3);
    if (rc) return rc;
    double sum[3] = {0, 0, 0};
    CU(cudaMemcpyAsync(sum, h->scal_part, sizeof sum, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    const bool same_chunks = std::fabs(h->nranks * sum[2] - sum[1] * sum[1]) < 0.5;
    h->blk_xchg = sum[0] > h->nranks - 0.5 && same_chunks;
    return PRMF_OK;
}

// 0 one GPU, 1 NCCL, 2 P2P pull in the V-update kernel, 4 push inside the persistent step kernel (3, the pull inside
// the pass-2 kernel, was removed; the numbers are part of the ABI)
int prmf_exchange_mode(const prmf_handle* h) {
    if (!h || !sharded(h)) return 0;
    if (!h->p2p_ready) return 1;
    if (h->blk_xchg && h->use_block) return 4;
    return 2;
}

int64_t prmf_launch_count(const prmf_handle* h) { return h ? h->launches : 0; }

int prmf_set_profiling(prmf_handle* h, int on) {
    if (!h) return PRMF_ERR_ARG;
    h->profiling = on != 0;
    return PRMF_OK;
}

int prmf_kernel_times(prmf_handle* h, int reset, double* phase_ms, int64_t* phase_count) {
    if (!h) return PRMF_ERR_ARG;
    for (int i = 0; i < PRMF_N_PHASES; ++i) {
        if (phase_ms) phase_ms[i] = h->phase_ms[i];
        if (phase_count) phase_count[i] = h->phase_n[i];
        if (reset) { h->phase_ms[i] = 0; h->phase_n[i] = 0; }
    }
    return PRMF_OK;
}

int prmf_project(prmf_handle* h, double* A_local) {
    if (!h || (!A_local && h->m > 0)) return PRMF_ERR_ARG;
    if (!h->have_X || !h->have_V) return fail(h, PRMF_ERR_STATE, "prmf_project needs X and V");
    if (h->failed) return fail(h, PRMF_ERR_STATE, "the handle is in a failed state");
    CU(cudaSetDevice(h->device));
    if (h->m == 0) return PRMF_OK;
    cancel_ahead(h);                                   // a speculative pass left other partials in Apart
    int rc = launch_xv(h);                             // the pass-1 stream of the inner step, without its U update
    if (rc) return rc;
    const int64_t cnt = h->m * h->k;
    double* dst = h->U2;                               // scratch: the second U buffer is free between steps
    sum_chunks_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, h->stream>>>(h->Apart, a_chunks(h), cnt, dst);
    LAUNCH_CHECK("sum_chunks_kernel");
    CU(cudaMemcpyAsync(A_local, dst, sizeof(double) * cnt, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return PRMF_OK;
}

int prmf_project_t(prmf_handle* h, double* B_out) {
    if (!h || !B_out) return PRMF_ERR_ARG;
    if (!h->have_X || !h->have_U) return fail(h, PRMF_ERR_STATE, "prmf_project_t needs X and U");
    if (h->failed) return fail(h, PRMF_ERR_STATE, "the handle is in a failed state");
    if (h->m != h->m_global) return fail(h, PRMF_ERR_STATE, "prmf_project_t needs a single-rank handle (m_local != m_global)");
    CU(cudaSetDevice(h->device));
    cancel_ahead(h);
    int rc = launch_xtu(h);                            // the pass-2 stream of the inner step, without its V update
    if (rc) return rc;
    const int64_t cnt = h->n * h->k;
    double* dst = h->Vbuf[h->vcur ^ 1];                // scratch: the second V buffer is free between steps
    sum_chunks_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, h->stream>>>(h->Bpart, b_chunks(h), cnt, dst);
    LAUNCH_CHECK("sum_chunks_kernel");
    CU(cudaMemcpyAsync(B_out, dst, sizeof(double) * cnt, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return PRMF_OK;
}

int prmf_nnls_x(prmf_handle* h, int transpose, const double* B_host, int maxiter, double* x_out, double* rnorm_out,
                int32_t* status_out, int32_t* iter_out) {
    if (!h || !B_host || !x_out || !rnorm_out || !status_out) return PRMF_ERR_ARG;
    if (h->x_tc) return fail(h, PRMF_ERR_STATE, "prmf_nnls_x needs an fp64 or f32 handle (X is stored as tf32)");
    if (h->m != h->m_global) return fail(h, PRMF_ERR_STATE, "prmf_nnls_x needs a single-rank handle (m_local != m_global)");
    if (!h->have_X) return fail(h, PRMF_ERR_STATE, "prmf_nnls_x needs X");
    if (h->failed) return fail(h, PRMF_ERR_STATE, "the handle is in a failed state");
    if (h->m == 0) return fail(h, PRMF_ERR_ARG, "prmf_nnls_x needs at least one sample");
    CU(cudaSetDevice(h->device));
    cancel_ahead(h);
    h->have_U = h->have_V = false;                     // U and V serve as the residual operand from here on
    if (h->x32)
        return nnls_x_run<float>(h, transpose, transpose ? h->X32 : h->Xt32, transpose ? h->ldx32 : h->ldxt32, B_host,
                                 maxiter, x_out, rnorm_out, status_out, iter_out);
    return nnls_x_run<double>(h, transpose, transpose ? h->X : h->Xt, transpose ? h->ldx : h->ldxt, B_host, maxiter,
                              x_out, rnorm_out, status_out, iter_out);
}

int prmf_release_pool(void) {
    g_pool.drain();
    return PRMF_OK;
}

int prmf_debug_inject_fault(prmf_handle* h, int kind) {
    if (!h) return PRMF_ERR_ARG;
    if (kind == 1) h->blk_n1 += 1;            // arrival targets of the next launch are one pass ahead of the counters
    else if (kind == 2) h->blk_xseq += 1;     // this rank expects exchange flags one step ahead of what peers send
    else return fail(h, PRMF_ERR_ARG, "unknown fault kind %d", kind);
    return PRMF_OK;
}

void* prmf_stream(const prmf_handle* h) { return h ? (void*)h->stream : nullptr; }

#ifdef PRMF_TAIL_TIMING
int prmf_debug_timeline(unsigned long long* out256, int reset) {
#ifdef PRMF_EPI_TIMING
    if (reset) {
        unsigned long long init[256];
        for (int i = 0; i < 256; ++i) init[i] = (i % 4 == 0) ? ~0ull : 0ull;
        return cudaMemcpyToSymbol(g_kt_dbg, init, sizeof init) == cudaSuccess ? 0 : -1;
    }
    return cudaMemcpyFromSymbol(out256, g_kt_dbg, sizeof(unsigned long long) * 256) == cudaSuccess ? 0 : -1;
#else
    (void)out256; (void)reset;
    return -1;
#endif
}

int prmf_debug_tail_stamps(unsigned long long* out16) {
    return cudaMemcpyFromSymbol(out16, g_tail_dbg, sizeof(unsigned long long) * 16) == cudaSuccess ? 0 : -1;
}
#endif

}  // extern "C"
