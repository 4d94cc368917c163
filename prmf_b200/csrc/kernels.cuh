// PRMF hot-path kernels for sm_100a (B200).  All arithmetic is IEEE fp64; every reduction has a fixed
// order so results are bitwise reproducible from run to run.
//
// Reference lines are in /root/reference/script/prmf_runner.py.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace prmf {

constexpr double kEps = 1.1920928955078125e-07;   // np.finfo(np.float32).eps, prmf_runner.py:23
constexpr int kObjStride = 8;

__device__ __forceinline__ double2 ld_stream(const double* p) {
    // streaming 128-bit load, do not allocate in L1 (X is read once per pass)
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}

// ---- sm_100a async-copy primitives (TMA bulk copies completed on mbarriers) ------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared (TMA engine, SASS UBLKCP); dst/src 16-byte aligned, bytes % 16 == 0
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::
            "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// s = part[0] + part[stride] + ... (count terms, added in index order; loads issued 8 at a time)
__device__ __forceinline__ double sum_strided(const double* __restrict__ part, int count, int64_t stride) {
    double s = 0.0;
    int c = 0;
    for (; c + 8 <= count; c += 8) {
        double t[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) t[q] = part[(int64_t)(c + q) * stride];
#pragma unroll
        for (int q = 0; q < 8; ++q) s += t[q];
    }
    for (; c < count; ++c) s += part[(int64_t)c * stride];
    return s;
}

// Deterministic block reduction (fixed tree); result valid in thread 0.  `scratch` holds >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    const int nw = (blockDim.x + 31) >> 5;
    if (warp == 0) {
        double t = lane < nw ? scratch[lane] : 0.0;
        t = warp_sum(t);
        if (lane == 0) scratch[0] = t;
    }
    __syncthreads();
    return scratch[0];
}

// Deterministic block reduction of NV values at once (one shared-memory round instead of NV); results valid in
// thread 0.  `scratch` holds >= 32*NV doubles.
template <int NV>
__device__ __forceinline__ void block_sum_multi(double (&v)[NV], double* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
    __syncthreads();
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) scratch[i * 32 + warp] = v[i];
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            double t = lane < nw ? scratch[i * 32 + lane] : 0.0;
            v[i] = warp_sum(t);
        }
    }
}

// ----------------------------------------------------------------------------------------------------
// ||X||_F^2  (np.linalg.norm(X), :640) : per-block partials, summed in order by sum_partials_kernel
// ----------------------------------------------------------------------------------------------------
// T = double (fp64 X, and U in prmf_objective) or float (fp32 X, PRMF_X_F32: squares of widened values, same order)
__device__ __forceinline__ double2 ld_stream_pair(const double* p) { return ld_stream(p); }
__device__ __forceinline__ double2 ld_stream_pair(const float* p) {
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return make_double2((double)r.x, (double)r.y);
}

template <typename T>
static __global__ void __launch_bounds__(256) sumsq_kernel(const T* __restrict__ X, int64_t ldx, int64_t m,
                                                    int n2, double* __restrict__ part) {
    __shared__ double scratch[32];
    double acc = 0.0;
    for (int64_t row = blockIdx.x; row < m; row += gridDim.x) {
        const T* xr = X + row * ldx;
        double a = 0.0;
        for (int j = threadIdx.x * 2; j < n2; j += blockDim.x * 2) {
            double2 x = ld_stream_pair(xr + j);
            a = fma(x.x, x.x, a);
            a = fma(x.y, x.y, a);
        }
        acc += a;
    }
    double t = block_sum(acc, scratch);
    if (threadIdx.x == 0) part[blockIdx.x] = t;
}

static __global__ void sum_partials_kernel(const double* __restrict__ part, int count, double* __restrict__ out) {
    __shared__ double scratch[32];
    double a = 0.0;
    for (int i = threadIdx.x; i < count; i += blockDim.x) a += part[i];
    double t = block_sum(a, scratch);
    if (threadIdx.x == 0) out[0] = t;
}

// ----------------------------------------------------------------------------------------------------
// Gram accumulation shared by the U and V update kernels: G += T^T T for a tile T (rows x k) held in shared
// memory.  The k*k pairs are split over the 1024 threads; when k*k < 1024 the rows of the tile are also cut
// into NS slices so every thread has work (item = slice * k*k + pair).  Slices are combined in a fixed order.
// ----------------------------------------------------------------------------------------------------
constexpr int kTailThreads = 1024;
constexpr int kVhCap = 4096;          // staged (support gene, factor) values in the objective (32 KB of smem)

__host__ __device__ inline int gram_slices(int k) {
    const int kk2 = k * k;
    if (kk2 >= kTailThreads) return 1;
    int ns = kTailThreads / kk2;
    return ns > 8 ? 8 : ns;
}

// dst[e] = sum_b src[b*kk2 + e] (b < count) for a k*k matrix, using all 1024 threads: the partials are cut into
// 1024/kk2 slices that are summed concurrently, then the slice sums are added in order.  sBuf: >= 1024 doubles.
__device__ __forceinline__ void sum_gram_partials(double* __restrict__ dst, const double* __restrict__ src, int count,
                                                  int kk2, double* __restrict__ sBuf) {
    if (kk2 > 512 || count <= 8) {
        for (int e = threadIdx.x; e < kk2; e += blockDim.x) dst[e] = sum_strided(src + e, count, kk2);
        __syncthreads();
        return;
    }
    const int nsl = 1024 / kk2;
    const int per = (count + nsl - 1) / nsl;
    if (threadIdx.x < nsl * kk2) {
        const int e = threadIdx.x % kk2, sl = threadIdx.x / kk2;
        const int b0 = sl * per, cnt = max(0, min(count, b0 + per) - b0);
        sBuf[sl * kk2 + e] = sum_strided(src + (int64_t)b0 * kk2 + e, cnt, kk2);
    }
    __syncthreads();
    if (threadIdx.x < kk2) {
        double s2 = 0.0;
        for (int sl = 0; sl < nsl; ++sl) s2 += sBuf[sl * kk2 + threadIdx.x];
        dst[threadIdx.x] = s2;
    }
    __syncthreads();
}

template <int NI>
__device__ __forceinline__ void gram_accumulate(const double* __restrict__ sT, int rows, int rows_per_tile, int k,
                                                int ns, double (&gacc)[NI]) {
    const int kk2 = k * k;
    const int rps = (rows_per_tile + ns - 1) / ns;
#pragma unroll
    for (int q = 0; q < NI; ++q) {
        const int item = threadIdx.x + q * kTailThreads;
        if (item < kk2 * ns) {
            const int pair = item % kk2, sl = item / kk2;
            const int a = pair / k, b = pair - a * k;
            const int rb = sl * rps, re = min(rows, rb + rps);
            double s2 = gacc[q];
            for (int r = rb; r < re; ++r) s2 = fma(sT[r * k + a], sT[r * k + b], s2);
            gacc[q] = s2;
        }
    }
}

// Combine the slices through shared memory (sBuf: >= k*k*ns doubles) and write this block's k*k partial.
template <int NI>
__device__ __forceinline__ void gram_store(double* __restrict__ sBuf, int k, int ns, const double (&gacc)[NI],
                                           double* __restrict__ part) {
    const int kk2 = k * k;
    if (ns == 1) {
#pragma unroll
        for (int q = 0; q < NI; ++q) {
            const int item = threadIdx.x + q * kTailThreads;
            if (item < kk2) part[item] = gacc[q];
        }
        return;
    }
    __syncthreads();
    if (threadIdx.x < kk2 * ns) sBuf[threadIdx.x] = gacc[0];             // ns > 1 implies NI == 1
    __syncthreads();
    if (threadIdx.x < kk2) {
        double s2 = 0.0;
        for (int sl = 0; sl < ns; ++sl) s2 += sBuf[sl * kk2 + threadIdx.x];
        part[threadIdx.x] = s2;
    }
}

// ----------------------------------------------------------------------------------------------------
// Elementwise update rules (u_update_value here, pathway_term / v_update_value / active_slot after ActiveSet): one
// definition for every kernel that updates U or V.  Keep each expression's shape: nvcc contracts device code into
// FMAs, so a re-associated form changes bits.
// ----------------------------------------------------------------------------------------------------

// New U element from u, a = (X.V)[r][c] and ugv = (U.Gv)[r][c] (:421-422): 0/0 := 1, no clamp.  `a` is read only
// when den != 0.
__device__ __forceinline__ double u_update_value(double u, const double& a, double ugv) {
    const double den = ugv + u;
    return u * ((den != 0.0) ? a / den : 1.0);
}

// ----------------------------------------------------------------------------------------------------
// U update (u_update_value) + per-block partials of U^T U (:425).  sum(U^2) (:359) is its trace.
// Blocks of 1024 threads loop over row tiles; the tile of new U rows is staged in shared memory.
// ----------------------------------------------------------------------------------------------------
template <int NI>
__global__ void __launch_bounds__(kTailThreads)
u_update_kernel(double* __restrict__ U, const double* __restrict__ Apart, int achunks, const double* __restrict__ Gv,
                int64_t m, int k, int rows_per_tile, double* __restrict__ Gu_part) {
    extern __shared__ double sm[];
    double* sGv = sm;                  // k*k
    double* sU = sm + k * k;           // max(rows_per_tile * k, 1024)   (new U rows; slice buffer at the end)
    const int kk2 = k * k;
    const int ns = gram_slices(k);
    for (int i = threadIdx.x; i < kk2; i += blockDim.x) sGv[i] = Gv[i];
    double gacc[NI];
#pragma unroll
    for (int q = 0; q < NI; ++q) gacc[q] = 0.0;
    __syncthreads();
    const int64_t ntiles = (m + rows_per_tile - 1) / rows_per_tile;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t r0 = tile * rows_per_tile;
        const int rows = (int)min((int64_t)rows_per_tile, m - r0);
        for (int e = threadIdx.x; e < rows * k; e += blockDim.x) {
            const int r = e / k, c = e - r * k;
            const double* urow = U + (r0 + r) * k;
            double ugv = 0.0;
            for (int l = 0; l < k; ++l) ugv = fma(urow[l], sGv[l * k + c], ugv);
            const double u = urow[c];
            const double a = sum_strided(Apart + (r0 + r) * k + c, achunks, m * k);      // X.V   (:420)
            sU[e] = u_update_value(u, a, ugv);
        }
        __syncthreads();
        for (int e = threadIdx.x; e < rows * k; e += blockDim.x) U[r0 * k + e] = sU[e];
        gram_accumulate<NI>(sU, rows, rows_per_tile, k, ns, gacc);
        __syncthreads();
    }
    gram_store<NI>(sU, k, ns, gacc, Gu_part + (int64_t)blockIdx.x * kk2);
}

// ----------------------------------------------------------------------------------------------------
// Packed pathway tables (device view)
// ----------------------------------------------------------------------------------------------------
struct Pathways {
    int P;
    const int64_t* path_ptr;     // P+1
    const int32_t* support_idx;  // S
    const int64_t* row_ptr;      // S+1
    const int32_t* col_local;    // E
    const double* w;             // E
    const double* deg;           // S   column sums of W                         (:680)
    const double* ldiag;         // S   diag(L) = deg - self-loop weight          (:683)
    const double* isd;           // S   diag(L)^-1/2, 0 where diag(L) == 0        (:58-62)
};

// Normalised Laplacians of the k ACTIVE pathways, flattened for the objective (:344-352): one diagonal
// entry per support row and one off-diagonal entry per stored edge, with global gene indices, so the
// objective needs a single gather of V per entry instead of walking the packed CSR.
struct ActiveSet {
    int64_t n_diag, n_off;
    const int32_t* diag_gene;    // gene of the support row
    const int32_t* diag_factor;
    const double* diag_coef;     // isd_r * diag(L)_r * isd_r
    const int32_t* off_r;        // gene of the row
    const int32_t* off_c;        // gene of the neighbour
    const int32_t* off_lr;       // index of the row's diagonal entry (0..n_diag)
    const int32_t* off_lc;       // index of the neighbour's diagonal entry
    const int32_t* off_factor;
    const double* off_coef;      // isd_r * (-w_rc * isd_c)   (0 for a self loop: it is part of diag(L))
};

// (W v)[j][c] of the V update (:434) over packed support row pr (gene j in factor c's active pathway).  kCg: read V_old
// (leading dimension ld) through L2 only, as needed where other CTAs of the same launch wrote it.
template <bool kCg>
__device__ __forceinline__ double pathway_term(const Pathways& pw, const int32_t* active, int32_t pr, int c,
                                               const double* Vold, int ld) {
    const int64_t base = pw.path_ptr[active[c]];
    double wv = 0.0;
    for (int64_t e2 = pw.row_ptr[pr]; e2 < pw.row_ptr[pr + 1]; ++e2) {
        const double* src = Vold + (int64_t)pw.support_idx[base + pw.col_local[e2]] * ld + c;
        wv = fma(pw.w[e2], kCg ? __ldcg(src) : *src, wv);
    }
    return wv;
}

// New V element from v, b = (X^T.U)[j][c] and vgu = (V.Gu)[j][c] (:425-444).  On the support (wv = pathway_term,
// deg = column sum of W) it adds the raw W / D terms, not the objective's normalised Laplacian; clamps at float32 eps.
__device__ __forceinline__ double v_update_value(double v, double b, double vgu, bool in_support, double wv, double deg,
                                                 double gamma, double delta) {
    double num = b, den = vgu;
    if (in_support) {
        const double vp1 = v + 1.0;
        const double man = gamma * wv;                          // :434
        const double ign = delta * (1.0 / (vp1 * vp1));         // :438
        num = b + (man + ign);                                  // :440
        den = vgu + gamma * (deg * v);                          // :435, :441
    }
    if (den < kEps) den = kEps;
    double vn = v * (num / den);                                // :443
    if (vn < kEps) vn = kEps;
    return vn;
}

// Index of (support row `row`, factor c) in the ActiveSet's diagonal order, which is also the order of the per-step
// V_new values of the deferred objective (hist_vh).  path_begin = path_ptr[active[c]].
__device__ __forceinline__ int64_t active_slot(const int64_t* doff, int c, int64_t row, int64_t path_begin) {
    return doff[c] + (row - path_begin);
}

// ----------------------------------------------------------------------------------------------------
// The X-stream kernel, used for BOTH passes:   Out[chunk][j][0:KT] = sum_{i in chunk} M[i][j] * W[i][0:KT]   (KT == k)
//   pass 1  (U_up_num = X.V, :420):        M = Xt (genes x samples, the transposed copy), W = V -> A partials
//   pass 2  (V_up_num_recon = X^T.U, :424): M = X  (samples x genes),                     W = U -> B partials
// M is row-major with leading dimension ldm (a multiple of 16 doubles, pad columns zero).  The grid is (column panels)
// x (row chunks); per-chunk partials are summed in a fixed order by the consumer.  A producer warp issues 1-D bulk
// async copies (cp.async.bulk, SASS UBLKCP) of RS row pieces of M (<= 8 KB each, contiguous) plus the RS matching rows
// of W per stage into a ring of `stages` shared-memory buffers; completion is tracked with mbarrier transaction
// counts, and the 8 consumer warps release a buffer through an "empty" mbarrier.  Bytes in flight per SM are set by
// the ring (>= 100 KB), not by registers: a version that streamed M with ld.global stalled on long_scoreboard (ncu:
// 24 % warps active) and reached 84 % of the measured copy bandwidth.
// Thread t owns the double2 columns t and t + H of the panel (H = panel_w / 4), so shared-memory reads of a
// warp are contiguous 512-byte runs (conflict free); W rows are broadcast reads.
// W must be readable for RS rows past the last row of the chunk (the host pads U and V allocations).
// ----------------------------------------------------------------------------------------------------
constexpr int kTmaRS = 8;                  // rows of M per ring stage (the RS of every launched instantiation)
constexpr int kTmaConsumerWarps = 8;
constexpr int kTmaThreads = (kTmaConsumerWarps + 1) * 32;

// ----------------------------------------------------------------------------------------------------
// One-shot all-reduce over NVLink peer memory, fused into the V update (sample-sharded runs).
// Every rank leaves its locally reduced packed buffer [X^T U | U^T U] in its own HBM; after a flag barrier
// over peer memory every rank reads all ranks' buffers with plain P2P loads and adds them in rank order, so
// all ranks obtain bitwise identical sums without a separate collective launch.  The packed buffers are
// double-buffered by step parity: a rank can only write parity p again after it passed the barrier of the
// step in between, which every peer reaches only after it finished reading parity p.
// ----------------------------------------------------------------------------------------------------
constexpr int kMaxPeers = 8;

// ---- bounded device-side waits ------------------------------------------------------------------------
// Every spin wait on a counter or flag written by another thread block or another GPU has a %globaltimer deadline:
// on expiry the waiter sets an error word, stops waiting (so do all later waits of the launch) and the kernel drains;
// the host turns the word into PRMF_ERR_TIMEOUT.  A lost launch or a dead peer rank is an error code, not a hang.
constexpr unsigned int kErrTimeoutLocal = 1u;   // a wait on another CTA of this GPU expired
constexpr unsigned int kErrTimeoutPeer = 2u;    // a wait on a peer GPU's flag expired

__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long blk_gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ unsigned int ld_volatile_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// Spin until *p >= target (acquire; SYS: the writer is a peer GPU).  Gives up when the deadline passes or when
// another waiter of this kernel already gave up (err != 0), so a failed launch drains instead of hanging.
template <bool SYS>
__device__ __forceinline__ bool blk_wait_ge(const unsigned long long* p, unsigned long long target, unsigned int* err,
                                            unsigned long long timeout_ns) {
    unsigned long long t0 = 0;
    unsigned int polls = 0;
    for (;;) {
        const unsigned long long v = SYS ? ld_acquire_sys_u64(p) : ld_acquire_gpu_u64(p);
        if (v >= target) return true;
        __nanosleep(40);                          // a spinning warp costs issue slots and power on its SM
        if ((++polls & 255u) == 0u) {
            const unsigned long long now = blk_gtime();
            if (t0 == 0) t0 = now;
            if (now - t0 > timeout_ns || ld_volatile_u32(err) != 0u) {
                atomicOr(err, SYS ? kErrTimeoutPeer : kErrTimeoutLocal);
                return false;
            }
        }
    }
}





struct PeerExchange {
    int nranks;                                // 0: no exchange (one GPU, or the NCCL path)
    int rank;
    const double* red[kMaxPeers];              // rank r's packed buffer of this step's parity (P2P mapped)
    unsigned long long* flags[kMaxPeers];      // rank r's flag array: flags[r][q] = last step rank q announced
    unsigned long long seq;                    // this step's sequence number (monotone)
    unsigned int* err;                         // bounded waits: error word and deadline
    unsigned long long timeout_ns;
};

__device__ __forceinline__ double ld_peer(const double* p) {
    double v;
    asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

// Announce "my packed buffer of step seq is complete" to every rank, then wait until every rank has done so.
__device__ __forceinline__ void peer_barrier(const PeerExchange& px) {
    if (threadIdx.x < px.nranks) {
        if (blockIdx.x == 0) {
            __threadfence_system();
            asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(px.flags[threadIdx.x] + px.rank), "l"(px.seq) : "memory");
        }
        blk_wait_ge<true>(px.flags[px.rank] + threadIdx.x, px.seq, px.err, px.timeout_ns);
    }
    __syncthreads();
}

__device__ __forceinline__ double sum_peers(const PeerExchange& px, int64_t idx) {
    double s = 0.0;
    double t[kMaxPeers];
#pragma unroll
    for (int r = 0; r < kMaxPeers; ++r) t[r] = r < px.nranks ? ld_peer(px.red[r] + idx) : 0.0;
#pragma unroll
    for (int r = 0; r < kMaxPeers; ++r) s += t[r];
    return s;
}

// ----------------------------------------------------------------------------------------------------
// Fused tails of the X-stream kernel (k <= 10).  The CTAs of one column panel cover different row chunks; once
// all of them have stored their partials (a counter per panel, monotone over launches, so it never needs a
// reset) the panel's rows are complete, and the SAME CTAs split them up and update them on the spot instead of
// leaving that to a separate latency-bound launch:
//   EPI 1 (pass 1, panel = samples): A = fixed-order sum of the chunk partials, U update (:421-422) into the
//          second U buffer, partials of U_new^T U_new
//   EPI 2 (pass 2, panel = genes, one GPU): B = fixed-order sum of the chunk partials, V update (:425-444) into
//          the second V buffer, partials of V_new^T V_new and sum(V_new * B) for the objective
//   EPI 3 (pass 2, sharded): B sums and the Gu sum written to the packed buffer that the ranks sum, either with
//          ncclAllReduce or with the P2P pull of the V-update kernel
// The per-CTA Gram partials are folded per panel by the last CTA of the panel to finish (second counter), so
// the next consumer adds only `panels` terms.  All CTAs of the grid must be co-resident (they wait for each
// other): the grid never exceeds the SM count and the launch is cooperative.  Only the 8 consumer warps take
// part (the producer warp has exited): barriers are the named barrier 1.
// ----------------------------------------------------------------------------------------------------
struct EpiParams {
    unsigned long long* arrive;   // per panel: CTAs whose partials are stored (monotone)
    unsigned long long* done;     // per panel: CTAs whose share of the update is finished (monotone)
    unsigned long long seq;       // 1-based launch number of this pass on this handle
    double* part2;                // scratch: per-CTA Gram partials [panels*chunks][k*k]
    double* vb2;                  // scratch: per-CTA sum(V_new * B) [panels*chunks]
    // EPI 1
    const double* Uold;
    double* Unew;
    const double* Gv;             // V^T V of the current V: gv_parts partials of k*k, added in order
    int gv_parts;
    double* Gu_part;              // out: [panels][k*k]
    // EPI 2
    const double* Vold;
    double* Vnew;
    const double* Gu_part_in;     // [gu_parts][k*k]
    int gu_parts;
    Pathways pw;
    const int32_t* active;
    const int32_t* pos;
    const double* gd;             // gamma, delta on the device
    double* Gv_part;              // out: [panels][k*k]
    double* VB_part;              // out: [panels]
    // deferred objective (EPI 2; null when the objective is evaluated every step): what the objective of this
    // step needs, kept per step so that ONE launch at the end of the block evaluates all of them
    double* hist_Gu;              // out: U^T U of this step (k*k)
    double* hist_vh;              // out: V_new at the (support gene, factor) pairs of the active set, in its order
    const int64_t* doff;          // per-factor offsets into that order (ActiveSet)
    // EPI 3
    double* red;                  // [n*k | k*k | 2]
    int dbg_slot;                 // developer timing builds only: timeline slot of this launch (-1: none)
    unsigned int* err;            // bounded waits: error word and deadline
    unsigned long long timeout_ns;
};

__device__ __forceinline__ void cons_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

#ifdef PRMF_EPI_TIMING
// Developer instrumentation (not part of the product build): per-launch timeline of the X-stream kernels.
__device__ __forceinline__ unsigned long long epi_gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// per-launch timeline: [slot][0] first CTA start, [1] last CTA past its main loop, [2] last CTA end
__device__ unsigned long long g_kt_dbg[64 * 4];
#define KT_STAMP_MIN(slot, i) do { if (threadIdx.x == 0 && (slot) >= 0 && (slot) < 64) atomicMin(&g_kt_dbg[(slot) * 4 + (i)], epi_gtime()); } while (0)
#define KT_STAMP_MAX(slot, i) do { if (threadIdx.x == 0 && (slot) >= 0 && (slot) < 64) atomicMax(&g_kt_dbg[(slot) * 4 + (i)], epi_gtime()); } while (0)
#else
#define KT_STAMP_MIN(slot, i) do { } while (0)
#define KT_STAMP_MAX(slot, i) do { } while (0)
#endif


// fixed-order sum of `count` partials read from L2 (they were just written by other SMs)
__device__ __forceinline__ double sum_strided_cg(const double* __restrict__ part, int count, int64_t stride) {
    double s = 0.0;
    int c = 0;
    for (; c + 8 <= count; c += 8) {
        double t[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) t[q] = __ldcg(part + (int64_t)(c + q) * stride);
#pragma unroll
        for (int q = 0; q < 8; ++q) s += t[q];
    }
    for (; c < count; ++c) s += __ldcg(part + (int64_t)c * stride);
    return s;
}

// wait until every CTA of this panel has stored its partials
__device__ __forceinline__ void epi_panel_barrier(const EpiParams& ep, int panel) {
    __threadfence();
    cons_bar();
    if (threadIdx.x == 0) {
        atomicAdd(ep.arrive + panel, 1ull);
        blk_wait_ge<false>(ep.arrive + panel, ep.seq * gridDim.y, ep.err, ep.timeout_ns);
    }
    cons_bar();
}

// this CTA's share of the update is stored; true in every thread of the panel's last CTA to get here
__device__ __forceinline__ bool epi_panel_done(const EpiParams& ep, int panel, int* s_flag) {
    __threadfence();
    cons_bar();
    if (threadIdx.x == 0) {
        const unsigned long long prev = atomicAdd(ep.done + panel, 1ull);
        *s_flag = prev + 1ull == ep.seq * gridDim.y;
    }
    cons_bar();
    const bool last = *s_flag != 0;
    if (last) __threadfence();
    return last;
}

// out = T^T T for the `rows` x K tile in shared memory (256 threads; row slices combined in a fixed order)
template <int K>
__device__ __forceinline__ void epi_gram(const double* __restrict__ sT, int rows, double* __restrict__ sBuf,
                                         double* __restrict__ out) {
    constexpr int NP = K * K;
    constexpr int NS = (256 / NP) > 8 ? 8 : (256 / NP);          // K <= 10: at least 2 slices
    const int t = threadIdx.x;
    const int rps = (max(rows, 0) + NS - 1) / NS;
    if (t < NP * NS) {
        const int pair = t % NP, sl = t / NP;
        const int a = pair / K, b = pair - a * K;
        const int rb = sl * rps, re = min(rows, rb + rps);
        double g = 0.0;
        for (int r = rb; r < re; ++r) g = fma(sT[r * K + a], sT[r * K + b], g);
        sBuf[sl * NP + pair] = g;
    }
    cons_bar();
    if (t < NP) {
        double g = 0.0;
#pragma unroll
        for (int sl = 0; sl < NS; ++sl) g += sBuf[sl * NP + t];
        out[t] = g;
    }
}

// dst[e] = sum over `count` partials of src[c*stride + e] for e < n_el (contiguous elements; fixed order per
// element).  Up to 2 elements x 16 partials of a thread are in flight at once instead of one dependent chain
// per element: the tail is latency bound, so the number of L2 round trips is what counts.
__device__ __forceinline__ void epi_stage_sums(double* __restrict__ dst, const double* __restrict__ src, int n_el,
                                               int count, int64_t stride) {
    for (int e0 = threadIdx.x; e0 < n_el; e0 += 256 * 2) {
        const bool ok1 = e0 + 256 < n_el;
        double acc0 = 0.0, acc1 = 0.0;
        for (int c = 0; c < count; c += 16) {
            double v0[16], v1[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const bool in = c + i < count;
                v0[i] = in ? __ldcg(src + (int64_t)(c + i) * stride + e0) : 0.0;
                v1[i] = (in && ok1) ? __ldcg(src + (int64_t)(c + i) * stride + e0 + 256) : 0.0;
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                if (c + i < count) { acc0 += v0[i]; acc1 += v1[i]; }
            }
        }
        dst[e0] = acc0;
        if (ok1) dst[e0 + 256] = acc1;
    }
}

// rows [rb, rb + rows) of the panel belong to this CTA
__device__ __forceinline__ void epi_share(int width, int64_t cols, int64_t c0, int& rb, int& rows) {
    const int all = (int)max((int64_t)0, min((int64_t)width, cols - c0));
    const int per = (all + (int)gridDim.y - 1) / (int)gridDim.y;
    rb = (int)blockIdx.y * per;
    rows = max(0, min(all, rb + per) - rb);
}

template <int K>
__device__ __forceinline__ void epi_u_update(const EpiParams& ep, unsigned char* smem, int* s_flag, int panel, int64_t c0,
                                             int width, int64_t cols, const double* __restrict__ Apart) {
    const int t = threadIdx.x;
    const int chunks = (int)gridDim.y;
    int rb, rows;
    epi_share(width, cols, c0, rb, rows);
    const int n_el = rows * K;
    double* sG = reinterpret_cast<double*>(smem);            // K*K (Gv), padded to 128 doubles
    double* sBuf = sG + 128;                                 // 8 * K*K slice sums
    double* sT = sBuf + 8 * K * K;                           // rows x K new rows
    double* sA = sT + n_el;                                  // rows x K sums of the pass-1 partials
    double* sU = sA + n_el;                                  // rows x K old rows
    const int64_t base = (c0 + rb) * K;                      // this share is one contiguous run of rows
    if (t < K * K) sG[t] = sum_strided(ep.Gv + t, ep.gv_parts, K * K);
    for (int e = t; e < n_el; e += 256) sU[e] = ep.Uold[base + e];
    epi_panel_barrier(ep, panel);
    epi_stage_sums(sA, Apart + base, n_el, chunks, cols * K);                               // X.V   (:420)
    cons_bar();
    for (int e = t; e < n_el; e += 256) {
        const int r = e / K, c = e - r * K;
        const double* urow = sU + r * K;
        double ugv = 0.0;
#pragma unroll
        for (int l = 0; l < K; ++l) ugv = fma(urow[l], sG[l * K + c], ugv);
        const double u = urow[c];
        const double un = u_update_value(u, sA[e], ugv);
        sT[e] = un;
        ep.Unew[base + e] = un;
    }
    cons_bar();
    const int64_t me = (int64_t)panel * chunks + blockIdx.y;
    epi_gram<K>(sT, rows, sBuf, ep.part2 + me * K * K);
    if (!epi_panel_done(ep, panel, s_flag)) return;
    if (t < K * K) ep.Gu_part[(int64_t)panel * K * K + t] = sum_strided_cg(ep.part2 + (int64_t)panel * chunks * K * K + t, chunks, K * K);
}

template <int K>
__device__ __forceinline__ void epi_v_update(const EpiParams& ep, unsigned char* smem, int* s_flag, int panel, int64_t c0,
                                             int width, int64_t cols, const double* __restrict__ Bpart) {
    const int t = threadIdx.x;
    const int chunks = (int)gridDim.y;
    int rb, rows;
    epi_share(width, cols, c0, rb, rows);
    const int n_el = rows * K;
    double* sG = reinterpret_cast<double*>(smem);            // K*K (Gu)
    double* sBuf = sG + 128;
    double* sT = sBuf + 8 * K * K;                           // rows x K new rows
    double* sB = sT + n_el;                                  // rows x K sums of the pass-2 partials
    double* sV = sB + n_el;                                  // rows x K old rows
    double* sW = sG + 112;                                   // 8 warp sums (K*K <= 100 < 112)
    const int64_t base = (c0 + rb) * K;
    // Gu = sum over the sample panels of pass 1 (complete before this kernel started)
    if (t < K * K) {
        const double g = sum_strided(ep.Gu_part_in + t, ep.gu_parts, K * K);
        sG[t] = g;
        if (ep.hist_Gu != nullptr && panel == 0 && blockIdx.y == 0) ep.hist_Gu[t] = g;
    }
    for (int e = t; e < n_el; e += 256) sV[e] = ep.Vold[base + e];
    const double gamma = ep.gd[0], delta = ep.gd[1];
    epi_panel_barrier(ep, panel);
    epi_stage_sums(sB, Bpart + base, n_el, chunks, cols * K);                               // X^T U  (:424)
    cons_bar();
    double vb = 0.0;
    for (int e = t; e < n_el; e += 256) {
        const int r = e / K, c = e - r * K;
        const int64_t j = c0 + rb + r;
        const double* vrow = sV + r * K;
        const double b = sB[e];
        double cden = 0.0;
#pragma unroll
        for (int l = 0; l < K; ++l) cden = fma(vrow[l], sG[l * K + c], cden);               // V.Gu   (:425)
        const double v = vrow[c];
        const int32_t pr = ep.pos[j * K + c];
        double wv = 0.0, dg = 0.0;
        if (pr >= 0) { wv = pathway_term<false>(ep.pw, ep.active, pr, c, ep.Vold, K); dg = ep.pw.deg[pr]; }
        const double vn = v_update_value(v, b, cden, pr >= 0, wv, dg, gamma, delta);
        sT[e] = vn;
        ep.Vnew[j * K + c] = vn;
        if (pr >= 0 && ep.hist_vh != nullptr) ep.hist_vh[active_slot(ep.doff, c, pr, ep.pw.path_ptr[ep.active[c]])] = vn;
        vb = fma(vn, b, vb);
    }
    // sum(V_new * B) of this share: warp sums, then the 8 warp sums in order
    vb = warp_sum(vb);
    if ((t & 31) == 0) sW[t >> 5] = vb;
    cons_bar();
    const int64_t me = (int64_t)panel * chunks + blockIdx.y;
    if (t == 0) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += sW[w];
        ep.vb2[me] = s;
    }
    epi_gram<K>(sT, rows, sBuf, ep.part2 + me * K * K);
    if (epi_panel_done(ep, panel, s_flag)) {
        if (t < K * K) ep.Gv_part[(int64_t)panel * K * K + t] = sum_strided_cg(ep.part2 + (int64_t)panel * chunks * K * K + t, chunks, K * K);
        if (t == 128) ep.VB_part[panel] = sum_strided_cg(ep.vb2 + (int64_t)panel * chunks, chunks, 1);
    }
}

template <int K>
__device__ __forceinline__ void epi_pack(const EpiParams& ep, int panel, int64_t c0, int width, int64_t cols,
                                         const double* __restrict__ Bpart) {
    const int t = threadIdx.x;
    const int chunks = (int)gridDim.y;
    int rb, rows;
    epi_share(width, cols, c0, rb, rows);
    epi_panel_barrier(ep, panel);
    const int64_t base = (c0 + rb) * K;
    for (int e = t; e < rows * K; e += 256) ep.red[base + e] = sum_strided_cg(Bpart + base + e, chunks, cols * K);
    if (panel == 0 && blockIdx.y == 0) {
        const int64_t nk = cols * K;
        if (t < K * K) ep.red[nk + t] = sum_strided(ep.Gu_part_in + t, ep.gu_parts, K * K);
        if (t < 2) ep.red[nk + K * K + t] = 0.0;
    }
}


// ----------------------------------------------------------------------------------------------------
// X-stream kernels: out[chunk][j][0:k] = sum over the rows i of the chunk of M[i][j] * W[i][0:k].  One CTA streams the
// rows of its chunk through a TMA ring: the producer warp bulk-copies a stage of RS rows of its column panel of M and
// the RS matching rows of W, and each of the 256 consumer threads accumulates 4 columns x KT factors in registers.
//
// One body serves every kernel; a single compile-time fact, FIXED_K, separates the two families:
//  - FIXED_K (skinny_tma_kernel<K,RS,EPI>, k = K <= 10): the wrapper passes k = KT, so the W row stride, the W slot and
//    the store are compile-time; one factor group; an unrolled branch for full stages; the fused tails EPI 1 / 2 / 3
//    run behind the store.
//  - run-time k (skinny_tma_gen_kernel<KT,FG,RS>, 10 < k <= 128, no fused tail): the consumers split into FG factor
//    groups of 256/FG threads.  A thread owns 4 columns of a (1024/FG)-column panel and KT consecutive factors of its
//    group, so the X tile is fetched from HBM once and re-read from shared memory by every group -- at k = 64 the
//    kernel is FP64-FMA bound (16 flop per byte of X), not HBM bound.  Factors >= k are computed on in-bounds garbage
//    and never written.  A group reads W indices up to f0 + (RS-1) k + KT - 1, which for f0 < k is <= RS k + KT - 2,
//    inside the RS k + KT doubles of the W slot; groups with f0 >= k read group 0's columns instead.
//
// T is the storage of X: double, or float for the fp32 storage mode (the _f32_ kernels).  An fp32 element is widened to
// fp64 exactly before its DFMA, so every column runs the same fma chain in the same row order on the same values, and
// the fp32 kernel returns, bit for bit, what the fp64 kernel returns on the widened matrix under the same launch plan.
// ----------------------------------------------------------------------------------------------------
// the two consecutive elements i = 2p, 2p + 1 of a shared-memory row, as fp64
__device__ __forceinline__ double2 x_pair(const double* row, int p) { return reinterpret_cast<const double2*>(row)[p]; }
__device__ __forceinline__ double2 x_pair(const float* row, int p) {
    const float2 v = reinterpret_cast<const float2*>(row)[p];
    return make_double2((double)v.x, (double)v.y);
}

template <typename T, bool FIXED_K, int KT, int FG, int RS, int EPI>
__device__ __forceinline__ void
skinny_tma_body(const T* __restrict__ M, int64_t ldm, int64_t rows_total, int64_t cols,
                const double* __restrict__ W, int k, int panel_w, int64_t rows_per_chunk, int stages,
                double* __restrict__ OutPart, const EpiParams& ep, unsigned tid) {
    static_assert(!FIXED_K || FG == 1, "a fixed k <= 10 runs one factor group");
    static_assert(FIXED_K || EPI == 0, "the fused tails need k fixed at compile time");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr uint32_t XB = (uint32_t)sizeof(T);                          // bytes per stored element of X
    constexpr int TG = 256 / FG;                                          // threads per factor group
    constexpr uint32_t W_SLACK = FIXED_K ? 0 : KT;                        // doubles behind a stage's W rows
    const int panel = blockIdx.x;
    const int64_t chunk = blockIdx.y;
    const int64_t c0 = (int64_t)panel * panel_w;                          // first column of the panel
    const int width = (int)min((int64_t)panel_w, ldm - c0);               // columns held (multiple of 4)
    const uint32_t row_bytes = (uint32_t)width * XB;
    const uint32_t x_stage_bytes = (uint32_t)RS * (uint32_t)panel_w * XB;
    const uint32_t w_bytes = (uint32_t)RS * (uint32_t)k * 8u;
    const uint32_t w_slot = (((uint32_t)RS * (uint32_t)k + W_SLACK) * 8u + 127u) & ~127u;
    const uint32_t stage_bytes = x_stage_bytes + w_slot;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_raw + (size_t)stages * stage_bytes);
    uint64_t* empty_bar = full_bar + stages;
    const int64_t rbeg = chunk * rows_per_chunk;
    const int64_t rend = min(rows_total, rbeg + rows_per_chunk);
    const int nstage_iters = rend > rbeg ? (int)((rend - rbeg + RS - 1) / RS) : 0;
    const int warp = tid >> 5, lane = tid & 31;
    if constexpr (FIXED_K) KT_STAMP_MIN(ep.dbg_slot, 0);

    if (tid == 0) {
        for (int s2 = 0; s2 < stages; ++s2) {
            mbar_init(&full_bar[s2], 1);
            mbar_init(&empty_bar[s2], kTmaConsumerWarps);
        }
        fence_mbar_init();
    }
    // the slack behind every W slot is read (and discarded) by the last factor group: keep it finite
    if constexpr (W_SLACK > 0)
        for (int s2 = tid; s2 < stages * KT; s2 += blockDim.x)
            reinterpret_cast<double*>(smem_raw + (size_t)(s2 / KT) * stage_bytes + x_stage_bytes + w_bytes)[s2 % KT] = 0.0;
    __syncthreads();

    if (warp == kTmaConsumerWarps) {
        // ===== producer warp: lanes 0..RS-1 copy one row piece each, lane 0 also copies the W rows =====
        const uint64_t pol_x = l2_policy_evict_first();
        const uint64_t pol_w = l2_policy_evict_last();
        int s2 = 0;
        uint32_t phase = 0;
        for (int it = 0; it < nstage_iters; ++it) {
            const int64_t r0 = rbeg + (int64_t)it * RS;
            const int rows = (int)min((int64_t)RS, rend - r0);
            if (lane == 0) mbar_wait(&empty_bar[s2], phase ^ 1u);
            __syncwarp();
            unsigned char* sx = smem_raw + (size_t)s2 * stage_bytes;
            if (lane == 0) {
                mbar_arrive_expect_tx(&full_bar[s2], (uint32_t)rows * row_bytes + w_bytes);
                bulk_g2s(sx + x_stage_bytes, W + r0 * k, w_bytes, &full_bar[s2], pol_w);
            }
            __syncwarp();
            if (lane < rows)
                bulk_g2s(sx + (size_t)lane * panel_w * XB, M + (r0 + lane) * ldm + c0, row_bytes, &full_bar[s2], pol_x);
            if (++s2 == stages) { s2 = 0; phase ^= 1u; }
        }
        return;
    }

    // ===== consumer warps =====
    const int H = panel_w >> 2;                        // double2 columns per half panel
    const int fg = FIXED_K ? 0 : tid / TG, t = FIXED_K ? tid : tid % TG;   // factor group, thread within it
    const int f0 = fg * KT;                            // first factor of this thread
    // groups whose factors all lie at or beyond k (k = 33..36, 65..84, 97..112) read group 0's columns, since their
    // own can lie past the W slot; what they compute is never written.  A branch around their loop instead measured
    // 1 % slower on the k = 64 stream, where no group is idle (B200, 1000 W).
    const int fr = f0 < k ? f0 : 0;
    const bool active = t < H && (2 * t) < width;      // first pair inside the held columns
    const bool active2 = t < H && (2 * (t + H)) < width;
    double acc[4][KT];
#pragma unroll
    for (int g = 0; g < 4; ++g)
#pragma unroll
        for (int c = 0; c < KT; ++c) acc[g][c] = 0.0;
    int s2 = 0;
    uint32_t phase = 0;
    for (int it = 0; it < nstage_iters; ++it) {
        const int rows = (int)min((int64_t)RS, rend - (rbeg + (int64_t)it * RS));
        mbar_wait(&full_bar[s2], phase);
        const unsigned char* sx = smem_raw + (size_t)s2 * stage_bytes;
        const double* sw = reinterpret_cast<const double*>(sx + x_stage_bytes) + fr;
        // the same row step twice: unrolled over a full stage at fixed k, a plain loop otherwise (a helper function or
        // lambda for the step changes the fixed-k kernels' SASS)
        if (FIXED_K && rows == RS) {
#pragma unroll
            for (int r = 0; r < RS; ++r) {
                const T* xrow = reinterpret_cast<const T*>(sx + (size_t)r * panel_w * XB);
                const double2 xa = active ? x_pair(xrow, t) : make_double2(0.0, 0.0);
                const double2 xb = active2 ? x_pair(xrow, t + H) : make_double2(0.0, 0.0);
#pragma unroll
                for (int c = 0; c < KT; ++c) {
                    const double u = sw[r * k + c];
                    acc[0][c] = fma(xa.x, u, acc[0][c]);
                    acc[1][c] = fma(xa.y, u, acc[1][c]);
                    acc[2][c] = fma(xb.x, u, acc[2][c]);
                    acc[3][c] = fma(xb.y, u, acc[3][c]);
                }
            }
        } else {
            for (int r = 0; r < rows; ++r) {
                const T* xrow = reinterpret_cast<const T*>(sx + (size_t)r * panel_w * XB);
                const double2 xa = active ? x_pair(xrow, t) : make_double2(0.0, 0.0);
                const double2 xb = active2 ? x_pair(xrow, t + H) : make_double2(0.0, 0.0);
#pragma unroll
                for (int c = 0; c < KT; ++c) {
                    const double u = sw[r * k + c];
                    acc[0][c] = fma(xa.x, u, acc[0][c]);
                    acc[1][c] = fma(xa.y, u, acc[1][c]);
                    acc[2][c] = fma(xb.x, u, acc[2][c]);
                    acc[3][c] = fma(xb.y, u, acc[3][c]);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s2]);
        if (++s2 == stages) { s2 = 0; phase ^= 1u; }
    }
    // columns owned: c0 + 2t, c0 + 2t + 1, c0 + 2(t+H), c0 + 2(t+H) + 1
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const int64_t j = c0 + 2 * (int64_t)(g < 2 ? t : t + H) + (g & 1);
        const bool ok = (g < 2 ? active : active2) && j < cols;
        if (ok) {
            double* out = OutPart + ((int64_t)chunk * cols + j) * k + f0;
#pragma unroll
            for (int c = 0; c < KT; ++c)
                if (f0 + c < k) out[c] = acc[g][c];
        }
    }
    if constexpr (FIXED_K) {
        KT_STAMP_MAX(ep.dbg_slot, 1);
        if constexpr (EPI != 0) {
            __shared__ int s_last;
            if constexpr (EPI == 1) epi_u_update<KT>(ep, smem_raw, &s_last, panel, c0, width, cols, OutPart);
            if constexpr (EPI == 2) epi_v_update<KT>(ep, smem_raw, &s_last, panel, c0, width, cols, OutPart);
            if constexpr (EPI == 3) epi_pack<KT>(ep, panel, c0, width, cols, OutPart);
        }
        KT_STAMP_MAX(ep.dbg_slot, 2);
    }
}

// The four kernels share one parameter list; a fixed-k kernel ignores `k`, a general-k kernel ignores `ep`.
// fp64 X (PRMF_X_F64), k = KT <= 10
template <int KT, int RS, int EPI>
__global__ void __launch_bounds__(kTmaThreads, 1)
skinny_tma_kernel(const double* __restrict__ M, int64_t ldm, int64_t rows_total, int64_t cols,
                  const double* __restrict__ W, int k, int panel_w, int64_t rows_per_chunk, int stages,
                  double* __restrict__ OutPart, const EpiParams ep) {
    skinny_tma_body<double, true, KT, 1, RS, EPI>(M, ldm, rows_total, cols, W, KT, panel_w, rows_per_chunk, stages,
                                                 OutPart, ep, threadIdx.x);
}

// fp32 X (PRMF_X_F32), k = KT <= 10; single rank, so the fused tails are the U update (EPI 1) and the V update (EPI 2)
template <int KT, int RS, int EPI>
__global__ void __launch_bounds__(kTmaThreads, 1)
skinny_tma_f32_kernel(const float* __restrict__ M, int64_t ldm, int64_t rows_total, int64_t cols,
                      const double* __restrict__ W, int k, int panel_w, int64_t rows_per_chunk, int stages,
                      double* __restrict__ OutPart, const EpiParams ep) {
    static_assert(EPI <= 2, "the fp32 storage mode has no sharded tails");
    skinny_tma_body<float, true, KT, 1, RS, EPI>(M, ldm, rows_total, cols, W, KT, panel_w, rows_per_chunk, stages,
                                                OutPart, ep, threadIdx.x);
}

// fp64 X, 10 < k <= 128 (BASELINE configs 4 and 5)
template <int KT, int FG, int RS>
__global__ void __launch_bounds__(kTmaThreads, 1)
skinny_tma_gen_kernel(const double* __restrict__ M, int64_t ldm, int64_t rows_total, int64_t cols,
                      const double* __restrict__ W, int k, int panel_w, int64_t rows_per_chunk, int stages,
                      double* __restrict__ OutPart, const EpiParams ep) {
    skinny_tma_body<double, false, KT, FG, RS, 0>(M, ldm, rows_total, cols, W, k, panel_w, rows_per_chunk, stages,
                                                 OutPart, ep, threadIdx.x);
}

// fp32 X, 10 < k <= 128
template <int KT, int FG, int RS>
__global__ void __launch_bounds__(kTmaThreads, 1)
skinny_tma_gen_f32_kernel(const float* __restrict__ M, int64_t ldm, int64_t rows_total, int64_t cols,
                          const double* __restrict__ W, int k, int panel_w, int64_t rows_per_chunk, int stages,
                          double* __restrict__ OutPart, const EpiParams ep) {
    skinny_tma_body<float, false, KT, FG, RS, 0>(M, ldm, rows_total, cols, W, k, panel_w, rows_per_chunk, stages,
                                                OutPart, ep, threadIdx.x);
}

// Xt[j][i] = X[i][j] : the factor of 2 in HBM capacity buys a coalesced, reduction-free pass 1.
static __global__ void __launch_bounds__(256)
transpose_kernel(const double* __restrict__ X, int64_t ldx, int64_t m, int64_t n, double* __restrict__ Xt,
                 int64_t ldxt) {
    __shared__ double tile[32][33];
    const int64_t i0 = (int64_t)blockIdx.y * 32, j0 = (int64_t)blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int64_t i = i0 + r, j = j0 + tx;
        tile[r][tx] = (i < m && j < n) ? X[i * ldx + j] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int64_t j = j0 + r, i = i0 + tx;
        if (j < n && i < m) Xt[j * ldxt + i] = tile[tx][r];
    }
}

// ----------------------------------------------------------------------------------------------------
// Sum the per-chunk X^T U partials and per-block U^T U partials in a fixed order into the packed
// buffer that is all-reduced over ranks:  red = [ B (n*k) | Gu (k*k) | sum(U^2) | pad ]
// ----------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
reduce_pack_kernel(const double* __restrict__ Bpart, int chunks, int64_t nk, const double* __restrict__ Gu_part,
                   int gu_blocks, int k, double* __restrict__ red) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int kk2 = k * k;
    if (idx < nk) {
        red[idx] = sum_strided(Bpart + idx, chunks, nk);
    } else if (idx < nk + kk2) {
        red[idx] = sum_strided(Gu_part + (idx - nk), gu_blocks, kk2);
    } else if (idx < nk + kk2 + 2) {
        red[idx] = 0.0;
    }
}

// out[e] = fixed-order sum of `chunks` partials (prmf_project: A = X.V from the pass-1 partials)
static __global__ void __launch_bounds__(256)
sum_chunks_kernel(const double* __restrict__ part, int chunks, int64_t count, double* __restrict__ out) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < count) out[idx] = sum_strided(part + idx, chunks, count);
}

// pos[j*k + c] = packed row of gene j in the active pathway of factor c (or -1, preset by a memset), and
// the flattened ActiveSet.  grid = (blocks, k); doff/eoff = per-factor offsets into the flat arrays.
static __global__ void build_active_kernel(Pathways pw, const int32_t* __restrict__ active, int k,
                                    const int64_t* __restrict__ doff, const int64_t* __restrict__ eoff,
                                    int32_t* __restrict__ pos, int32_t* __restrict__ diag_gene,
                                    int32_t* __restrict__ diag_factor, double* __restrict__ diag_coef,
                                    int32_t* __restrict__ off_r, int32_t* __restrict__ off_c,
                                    int32_t* __restrict__ off_lr, int32_t* __restrict__ off_lc,
                                    int32_t* __restrict__ off_factor, double* __restrict__ off_coef) {
    const int c = blockIdx.y;
    const int p = active[c];
    const int64_t beg = pw.path_ptr[p], end = pw.path_ptr[p + 1];
    const int64_t ebeg = pw.row_ptr[beg];
    for (int64_t r = beg + blockIdx.x * blockDim.x + threadIdx.x; r < end; r += (int64_t)gridDim.x * blockDim.x) {
        const int32_t g = pw.support_idx[r];
        pos[(int64_t)g * k + c] = (int32_t)r;
        const double ir = pw.isd[r];
        const int64_t di = active_slot(doff, c, r, beg);
        diag_gene[di] = g;
        diag_factor[di] = c;
        diag_coef[di] = ir * (pw.ldiag[r] * ir);
        for (int64_t e2 = pw.row_ptr[r]; e2 < pw.row_ptr[r + 1]; ++e2) {
            const int64_t oi = eoff[c] + (e2 - ebeg);
            const int64_t rc = beg + pw.col_local[e2];
            off_r[oi] = g;
            off_c[oi] = pw.support_idx[rc];
            off_lr[oi] = (int32_t)di;
            off_lc[oi] = (int32_t)active_slot(doff, c, rc, beg);
            off_factor[oi] = c;
            off_coef[oi] = (rc == r) ? 0.0 : ir * (-pw.w[e2] * pw.isd[rc]);
        }
    }
}

#ifdef PRMF_TAIL_TIMING
// Developer instrumentation (not part of the product build): phase time stamps of the V-update kernel.
__device__ unsigned long long g_tail_dbg[16];
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define TAIL_STAMP(i, cond) do { if (threadIdx.x == 0 && (cond)) g_tail_dbg[i] = gtime(); } while (0)
#else
#define TAIL_STAMP(i, cond) do { } while (0)
#endif

// ----------------------------------------------------------------------------------------------------
// Objective of one inner step (:336-372) without a pass over X, and the tradeoff feedback (:542-548).
//   recon^2 = ||X||^2 - 2 sum(V_new*B) + sum(Gu*Gv_new)        (B = X^T U_new, Gu = U_new^T U_new)
//   manifold = sum_k vhat_k^T Lhat_{p_k} vhat_k ; ignore = sum_k sum_{i in supp} 1/(vhat_i + 1)
//   fro = trace(Gu) = sum(U^2)
// Executed by ONE block of 1024 threads (the last block of the V update to finish); every phase is one
// round of independent loads followed by a fixed-order reduction.  Publishes Gv_new = V_new^T V_new for
// the next step's U update.  Loads bypass L1 (__ldcg): the data was just written by other SMs.
// ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ void objective_block(const double* __restrict__ V, int k, const double* __restrict__ sGu,
                                                double* __restrict__ sGv, double* __restrict__ sSl,
                                                double* __restrict__ scratch, const double* __restrict__ Gv_part,
                                                const double* __restrict__ VB_part, int vblocks, int gv_parts,
                                                const double* __restrict__ normX_sq, const ActiveSet& as,
                                                double* __restrict__ Gv, double* __restrict__ gd, double tradeoff,
                                                double* __restrict__ obj_out, int* __restrict__ step_counter,
                                                int obj_capacity, double* __restrict__ sVh, int vh_cap,
                                                const double* __restrict__ vh_pre = nullptr, int row = -1,
                                                bool publish_gv = true) {
    // vh_pre: the (support gene, factor) values of V_new already gathered by the V update (deferred objective);
    // row >= 0: write that row of obj_out and leave the step counter alone; publish_gv: store Gv_new in `Gv`
    const int kk2 = k * k;
    const int t = threadIdx.x;
    // prefetch everything that does not depend on Gv_new: scalars, VB partials, the flattened-Laplacian entries
    const double gamma = gd[0], delta = gd[1], nx2 = normX_sq[0];
    double vb = 0.0;
    for (int b = t; b < vblocks; b += blockDim.x) vb += __ldcg(VB_part + b);
    // One SM runs this block, and every scattered gather costs it an L1 wavefront: gather each distinct
    // (support gene, factor) value ONCE into shared memory (n_diag of them) and let the ~5x more numerous
    // off-diagonal entries index that copy.  Falls back to global gathers when n_diag exceeds the buffer.
    const bool staged = as.n_diag <= vh_cap;
    if (staged)
        for (int64_t i = t; i < as.n_diag; i += blockDim.x)
            sVh[i] = vh_pre != nullptr ? __ldcg(vh_pre + i) : __ldcg(V + (int64_t)as.diag_gene[i] * k + as.diag_factor[i]);
    constexpr int kPre = 4;                       // entries per thread handled from registers (4096 per pass)
    int dfac[kPre], ofac[kPre];
    double dcoef[kPre], dv[kPre], ocoef[kPre], ovr[kPre], ovc[kPre];
#pragma unroll
    for (int q = 0; q < kPre; ++q) {
        const int64_t i = t + (int64_t)q * blockDim.x;
        dfac[q] = -1; ofac[q] = -1; dcoef[q] = dv[q] = ocoef[q] = ovr[q] = ovc[q] = 0.0;
        if (staged) continue;
        if (i < as.n_diag) {
            dfac[q] = as.diag_factor[i];
            dcoef[q] = as.diag_coef[i];
            dv[q] = __ldcg(V + (int64_t)as.diag_gene[i] * k + dfac[q]);
        }
        if (i < as.n_off) {
            ofac[q] = as.off_factor[i];
            ocoef[q] = as.off_coef[i];
            ovr[q] = __ldcg(V + (int64_t)as.off_r[i] * k + ofac[q]);
            ovc[q] = __ldcg(V + (int64_t)as.off_c[i] * k + ofac[q]);
        }
    }
    TAIL_STAMP(6, true);
    // Gv_new[e] = fixed-order sum of the V-update blocks' partials (slices in parallel, then slice sums in order)
    if (kk2 <= 1024) {
        const int nsl = 1024 / kk2;
        const int per = (gv_parts + nsl - 1) / nsl;
        if (t < nsl * kk2) {
            const int e = t % kk2, sl = t / kk2;
            const int b0 = sl * per, cnt = max(0, min(gv_parts, b0 + per) - b0);
            const double* src = Gv_part + (int64_t)b0 * kk2 + e;
            double s2 = 0.0;
            int b = 0;
            for (; b + 8 <= cnt; b += 8) {
                double tmp[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) tmp[q] = __ldcg(src + (int64_t)(b + q) * kk2);
#pragma unroll
                for (int q = 0; q < 8; ++q) s2 += tmp[q];
            }
            for (; b < cnt; ++b) s2 += __ldcg(src + (int64_t)b * kk2);
            sSl[sl * kk2 + e] = s2;
        }
        __syncthreads();
        if (t < kk2) {
            double s2 = 0.0;
            for (int sl = 0; sl < nsl; ++sl) s2 += sSl[sl * kk2 + t];
            sGv[t] = s2;
            if (publish_gv) Gv[t] = s2;
        }
    } else {
        for (int e = t; e < kk2; e += blockDim.x) {
            double s2 = 0.0;
            for (int b = 0; b < gv_parts; ++b) s2 += __ldcg(Gv_part + (int64_t)b * kk2 + e);
            sGv[e] = s2;
            Gv[e] = s2;
        }
    }
    __syncthreads();
    TAIL_STAMP(7, true);
    double* sNrm = scratch + 5 * 32;              // ||v_c|| per factor (:345), computed once
    for (int c = t; c < k; c += blockDim.x) sNrm[c] = sqrt(sGv[c * k + c]);
    double gg = 0.0, fr = 0.0;
    for (int e = t; e < kk2; e += blockDim.x) {
        const double gu = sGu[e];
        gg = fma(sGv[e], gu, gg);
        if (e / k == e % k) fr += gu;                                                       // :359
    }
    __syncthreads();
    double man = 0.0, ign = 0.0;
    if (staged) {
        for (int64_t i = t; i < as.n_diag; i += blockDim.x) {
            const double vr = sVh[i] / sNrm[as.diag_factor[i]];                             // :345
            sVh[i] = vr;
            man = fma(as.diag_coef[i] * vr, vr, man);
            ign += 1.0 / (vr + 1.0);                                                        // :352
        }
        __syncthreads();
        for (int64_t i = t; i < as.n_off; i += blockDim.x)
            man = fma(as.off_coef[i] * sVh[as.off_lc[i]], sVh[as.off_lr[i]], man);          // :350
    }
#pragma unroll
    for (int q = 0; q < kPre; ++q) {
        if (dfac[q] >= 0) {
            const double vr = dv[q] / sNrm[dfac[q]];                                        // :345
            man = fma(dcoef[q] * vr, vr, man);
            ign += 1.0 / (vr + 1.0);                                                        // :352
        }
        if (ofac[q] >= 0) {
            const double nrm = sNrm[ofac[q]];
            man = fma(ocoef[q] * (ovc[q] / nrm), ovr[q] / nrm, man);                        // :350
        }
    }
    for (int64_t i = t + (int64_t)kPre * blockDim.x; !staged && i < as.n_diag; i += blockDim.x) {
        const int c = as.diag_factor[i];
        const double vr = __ldcg(V + (int64_t)as.diag_gene[i] * k + c) / sNrm[c];
        man = fma(as.diag_coef[i] * vr, vr, man);
        ign += 1.0 / (vr + 1.0);
    }
    for (int64_t i = t + (int64_t)kPre * blockDim.x; !staged && i < as.n_off; i += blockDim.x) {
        const int c = as.off_factor[i];
        const double nrm = sNrm[c];
        const double vr = __ldcg(V + (int64_t)as.off_r[i] * k + c) / nrm;
        const double vc = __ldcg(V + (int64_t)as.off_c[i] * k + c) / nrm;
        man = fma(as.off_coef[i] * vc, vr, man);
    }
    TAIL_STAMP(8, true);
    double red5[5] = {gg, fr, vb, man, ign};
    block_sum_multi<5>(red5, scratch);
    TAIL_STAMP(9, true);
    if (t == 0) {
        const double GG = red5[0], FRO = red5[1], VB = red5[2], MAN = red5[3], IGN = red5[4];
        const double r2 = nx2 - 2.0 * VB + GG;
        const double recon = sqrt(r2 > 0.0 ? r2 : 0.0);
        const double obj = recon + gamma * MAN + delta * IGN + FRO;                         // :362
        const int s2 = row >= 0 ? row : *step_counter;
        if (s2 < obj_capacity) {
            double* o = obj_out + (int64_t)s2 * kObjStride;
            o[0] = recon; o[1] = MAN; o[2] = IGN; o[3] = FRO; o[4] = obj; o[5] = gamma; o[6] = delta; o[7] = r2;
        }
        if (row < 0) *step_counter = s2 + 1;
        if (tradeoff >= 0.0) {                                                              // :542-548
            const double den = tradeoff * MAN;
            const double g2 = (den == 0.0) ? 1.0 : ((1.0 - tradeoff) * recon) / den;
            gd[0] = g2; gd[1] = g2;
        }
    }
}

// ----------------------------------------------------------------------------------------------------
// V update (:425-444) fused with the objective (:336-372).
//   B  = fixed-order sum of `bchunks` partials (the pass-2 partials directly on one GPU; the all-reduced
//        packed buffer with bchunks = 1 when sharded), Gu likewise from `gchunks` partials
//   C = V.Gu ; num = B + (gamma*W v + delta*(v+1)^-2 on the support) ; den = C + gamma*deg*v
//   den < eps -> eps ; V <- V*num/den ; V < eps -> eps
// V is double-buffered: pathway neighbours of a gene may be updated by another block, so new values go to Vnew
// while every block reads the untouched Vold.  Every block leaves partials of V_new^T V_new and
// sum(V_new * B); block 0 waits for the others (atomic ticket) and evaluates the objective from them.
// ----------------------------------------------------------------------------------------------------
template <int NI>
__global__ void __launch_bounds__(kTailThreads)
v_update_objective_kernel(const double* __restrict__ Vold, double* __restrict__ Vnew,
                          const double* __restrict__ Bsrc, int bchunks, int64_t bstride,
                          const double* __restrict__ Gusrc, int gchunks, int n, int k, Pathways pw,
                          const int32_t* __restrict__ active, const int32_t* __restrict__ pos,
                          double* __restrict__ gd, int rows_per_tile, double* __restrict__ Gv_part,
                          double* __restrict__ VB_part, const double* __restrict__ normX_sq, ActiveSet as,
                          double* __restrict__ Gv, double tradeoff, double* __restrict__ obj_out,
                          int* __restrict__ step_counter, int obj_capacity, unsigned int* __restrict__ ticket,
                          PeerExchange px) {
    extern __shared__ double sm[];
    double* sGu = sm;                   // k*k
    double* sGv = sm + k * k;           // k*k   (objective)
    // Two k*k arrays do not fit for k > 64 (2 x 128 KB at k = 128): then the objective keeps Gv_new in global
    // memory and the second slot shrinks to the 1024-double slice buffer (the host sizes smem the same way).
    double* sV = sm + k * k + (k > 64 ? 1024 : k * k);   // max(rows_per_tile*k, 1024): new V rows / slice sums
    double* sVh = sV + max(rows_per_tile * k, 1024);     // kVhCap doubles: unit-vector values of the active supports
    __shared__ double scratch[5 * 32 + 128];    // block reductions + per-factor norms (k <= 128)
    const int kk2 = k * k;
    const int ns = gram_slices(k);
    const int64_t nk_all = (int64_t)n * k;
    TAIL_STAMP(0, blockIdx.x == 0);
    if (px.nranks > 0) {
        peer_barrier(px);
        for (int i = threadIdx.x; i < kk2; i += blockDim.x) sGu[i] = sum_peers(px, nk_all + i);
        __syncthreads();
    } else {
        sum_gram_partials(sGu, Gusrc, gchunks, kk2, sV);
    }
    const double gamma = gd[0], delta = gd[1];
    double gacc[NI];
#pragma unroll
    for (int q = 0; q < NI; ++q) gacc[q] = 0.0;
    double vb = 0.0;
    __syncthreads();
    TAIL_STAMP(1, blockIdx.x == 0);
    const int ntiles = (n + rows_per_tile - 1) / rows_per_tile;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int j0 = tile * rows_per_tile;
        const int rows = min(rows_per_tile, n - j0);
        for (int e = threadIdx.x; e < rows * k; e += blockDim.x) {
            const int r = e / k, c = e - r * k;
            const int j = j0 + r;
            const double* vrow = Vold + (int64_t)j * k;
            const double b = px.nranks > 0 ? sum_peers(px, (int64_t)j * k + c)
                                           : sum_strided(Bsrc + (int64_t)j * k + c, bchunks, bstride);   // X^T U  (:424)
            double cden = 0.0;
            for (int l = 0; l < k; ++l) cden = fma(vrow[l], sGu[l * k + c], cden);       // V.Gu   (:425)
            const double v = vrow[c];
            const int32_t pr = pos[(int64_t)j * k + c];
            double wv = 0.0, dg = 0.0;
            if (pr >= 0) { wv = pathway_term<false>(pw, active, pr, c, Vold, k); dg = pw.deg[pr]; }
            const double vn = v_update_value(v, b, cden, pr >= 0, wv, dg, gamma, delta);
            sV[e] = vn;
            Vnew[(int64_t)j0 * k + e] = vn;
            vb = fma(vn, b, vb);
        }
        __syncthreads();
        TAIL_STAMP(2, blockIdx.x == 0);
        gram_accumulate<NI>(sV, rows, rows_per_tile, k, ns, gacc);
        __syncthreads();
    }
    gram_store<NI>(sV, k, ns, gacc, Gv_part + (int64_t)blockIdx.x * kk2);
    const double tvb = block_sum(vb, scratch);
    if (threadIdx.x == 0) VB_part[blockIdx.x] = tvb;
    TAIL_STAMP(3, blockIdx.x == 0);
    // ---- objective: block 0 waits for the other blocks (they never wait on anything, so this cannot deadlock)
    //      and evaluates it.  Always the same block, hence the same SM from launch to launch: the objective's
    //      code stays in that SM's instruction cache (with a "last block done" scheme a random, cold SM ran it).
    __threadfence();
    __syncthreads();
    if (blockIdx.x != 0) {
        if (threadIdx.x == 0) atomicAdd(ticket, 1u);
        return;
    }
    if (threadIdx.x == 0) {
        unsigned int seen;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(ticket) : "memory");
        } while (seen < gridDim.x - 1);
    }
    __syncthreads();
    TAIL_STAMP(4, true);
    if (threadIdx.x == 0) *ticket = 0u;                 // re-arm for the next launch
    // (the other blocks' results are read with ld.global.cg from L2, where their fenced writes already are)
    objective_block(Vnew, k, sGu, k > 64 ? Gv : sGv, k > 64 ? sGv : sV, scratch, Gv_part, VB_part, (int)gridDim.x,
                    (int)gridDim.x, normX_sq, as, Gv, gd, tradeoff, obj_out, step_counter, obj_capacity, sVh, kVhCap);
    TAIL_STAMP(5, true);
}

// ----------------------------------------------------------------------------------------------------
// Large k (> 16): the k x k Grams are no longer "small state".  (1) Summing the per-block Gram partials inside
// every consumer block re-read parts x k*k doubles per block (2.9 GB of L2 traffic per step at k = 128): they are
// folded ONCE by a grid-wide kernel.  (2) The U update is two skinny GEMMs (U.Gv and U_new^T U_new, 2 m k^2 flop
// each) and gets register tiles: 256 threads = 16 x 16, a thread owns RPT rows x CPT columns of U.Gv and a
// CPT x CPT block of the Gram; column ownership is interleaved in pairs (columns 32 j + 2 tx, +1) so the shared-memory
// reads of a warp are conflict-free 128-bit accesses.
// ----------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
gram_reduce_kernel(const double* __restrict__ parts, int count, int kk2, double* __restrict__ out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < kk2) out[e] = sum_strided(parts + e, count, kk2);
}

template <int CPT>
__device__ __forceinline__ int tiled_col(int tx, int j) { return 32 * (j >> 1) + 2 * tx + (j & 1); }

template <int CPT, int RPT>
__global__ void __launch_bounds__(256)
u_update_tiled_kernel(double* __restrict__ U, const double* __restrict__ Apart, int achunks,
                      const double* __restrict__ Gv, int64_t m, int k, double* __restrict__ Gu_part) {
    constexpr int KT = 16 * CPT;          // padded factor count (k <= KT)
    constexpr int TR = 16 * RPT;          // rows per tile
    constexpr int LD = KT + 2;            // row pitch of the U tile (rows of a warp fall into different banks)
    extern __shared__ __align__(16) double sm_tiled[];
    double* sGv = sm_tiled;               // KT x KT, zero padded
    double* sU = sGv + KT * KT;           // TR x LD: old rows, then the new rows in place
    double* sA = sU + TR * LD;            // TR x k: X.V of the tile's rows (sum of the pass-1 partials)
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    for (int e = threadIdx.x; e < KT * KT; e += 256) {
        const int l = e / KT, c = e - l * KT;
        sGv[e] = (l < k && c < k) ? Gv[l * k + c] : 0.0;
    }
    double g[CPT][CPT];
#pragma unroll
    for (int i = 0; i < CPT; ++i)
#pragma unroll
        for (int j = 0; j < CPT; ++j) g[i][j] = 0.0;
    const int64_t ntiles = (m + TR - 1) / TR;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t r0 = tile * TR;
        __syncthreads();
        for (int e = threadIdx.x; e < TR * KT; e += 256) {
            const int r = e / KT, c = e - r * KT;
            sU[r * LD + c] = (r0 + r < m && c < k) ? U[(r0 + r) * k + c] : 0.0;
        }
        // the rows of a tile are one contiguous run: fixed-order sums of the partials with many loads in flight
        epi_stage_sums(sA, Apart + r0 * k, (int)min((int64_t)TR, m - r0) * k, achunks, m * k);  // X.V   (:420)
        __syncthreads();
        // den = U.Gv for RPT rows x CPT columns
        double den[RPT][CPT];
#pragma unroll
        for (int i = 0; i < RPT; ++i)
#pragma unroll
            for (int j = 0; j < CPT; ++j) den[i][j] = 0.0;
        for (int l = 0; l < k; ++l) {
            double u[RPT], gv[CPT];
#pragma unroll
            for (int i = 0; i < RPT; ++i) u[i] = sU[(ty + 16 * i) * LD + l];
#pragma unroll
            for (int j = 0; j < CPT; j += 2) {
                const double2 t2 = *reinterpret_cast<const double2*>(sGv + l * KT + tiled_col<CPT>(tx, j));
                gv[j] = t2.x; gv[j + 1] = t2.y;
            }
#pragma unroll
            for (int i = 0; i < RPT; ++i)
#pragma unroll
                for (int j = 0; j < CPT; ++j) den[i][j] = fma(u[i], gv[j], den[i][j]);
        }
        double un[RPT][CPT];
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            const int r = ty + 16 * i;
            const int64_t row = r0 + r;
#pragma unroll
            for (int j = 0; j < CPT; ++j) {
                const int c = tiled_col<CPT>(tx, j);
                double v = 0.0;
                if (row < m && c < k) {
                    v = u_update_value(sU[r * LD + c], sA[r * k + c], den[i][j]);
                    U[row * k + c] = v;
                }
                un[i][j] = v;
            }
        }
        __syncthreads();                                   // everyone is done reading the old rows
#pragma unroll
        for (int i = 0; i < RPT; ++i)
#pragma unroll
            for (int j = 0; j < CPT; ++j) sU[(ty + 16 * i) * LD + tiled_col<CPT>(tx, j)] = un[i][j];
        __syncthreads();
        // Gram: G[a][b] += sum_r Unew[r][a] Unew[r][b], a from ty's columns, b from tx's columns
        for (int r = 0; r < TR; ++r) {
            double ua[CPT], ub[CPT];
#pragma unroll
            for (int j = 0; j < CPT; j += 2) {
                const double2 a2 = *reinterpret_cast<const double2*>(sU + r * LD + tiled_col<CPT>(ty, j));
                const double2 b2 = *reinterpret_cast<const double2*>(sU + r * LD + tiled_col<CPT>(tx, j));
                ua[j] = a2.x; ua[j + 1] = a2.y; ub[j] = b2.x; ub[j + 1] = b2.y;
            }
#pragma unroll
            for (int i = 0; i < CPT; ++i)
#pragma unroll
                for (int j = 0; j < CPT; ++j) g[i][j] = fma(ua[i], ub[j], g[i][j]);
        }
    }
    double* out = Gu_part + (int64_t)blockIdx.x * k * k;
#pragma unroll
    for (int i = 0; i < CPT; ++i) {
        const int a = tiled_col<CPT>(ty, i);
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
            const int b = tiled_col<CPT>(tx, j);
            if (a < k && b < k) out[a * k + b] = g[i][j];
        }
    }
}

// V update (:425-444) for large k with the same register tiles as u_update_tiled_kernel: V.Gu and V_new^T V_new are
// the two k x k contractions; B, the pathway terms and the clamps are applied per owned element.  Leaves per-block
// partials of V_new^T V_new and sum(V_new * B); the objective is a separate launch (objective_kernel).
template <int CPT, int RPT>
__global__ void __launch_bounds__(256)
v_update_tiled_kernel(const double* __restrict__ Vold, double* __restrict__ Vnew, const double* __restrict__ Bsrc,
                      int bchunks, int64_t bstride, const double* __restrict__ Gu, int n, int k, Pathways pw,
                      const int32_t* __restrict__ active, const int32_t* __restrict__ pos,
                      const double* __restrict__ gd, double* __restrict__ Gv_part, double* __restrict__ VB_part,
                      PeerExchange px, double* __restrict__ Gu_out) {
    constexpr int KT = 16 * CPT;
    constexpr int TR = 16 * RPT;
    constexpr int LD = KT + 2;
    extern __shared__ __align__(16) double sm_tiled[];
    double* sGu = sm_tiled;               // KT x KT, zero padded
    double* sV = sGu + KT * KT;           // TR x LD: old rows, then the new rows in place
    double* sB = sV + TR * LD;            // TR x k: X^T U of the tile's genes (summed over chunks / ranks)
    __shared__ double scratch[32];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t nk_all = (int64_t)n * k;
    if (px.nranks > 0) peer_barrier(px);
    for (int e = threadIdx.x; e < KT * KT; e += 256) {
        const int l = e / KT, c = e - l * KT;
        double v = 0.0;
        if (l < k && c < k) v = px.nranks > 0 ? sum_peers(px, nk_all + l * k + c) : Gu[l * k + c];
        sGu[e] = v;
        if (Gu_out != nullptr && blockIdx.x == 0 && l < k && c < k) Gu_out[l * k + c] = v;
    }
    const double gamma = gd[0], delta = gd[1];
    double g[CPT][CPT];
#pragma unroll
    for (int i = 0; i < CPT; ++i)
#pragma unroll
        for (int j = 0; j < CPT; ++j) g[i][j] = 0.0;
    double vb = 0.0;
    const int ntiles = (n + TR - 1) / TR;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int j0 = tile * TR;
        __syncthreads();
        for (int e = threadIdx.x; e < TR * KT; e += 256) {
            const int r = e / KT, c = e - r * KT;
            sV[r * LD + c] = (j0 + r < n && c < k) ? Vold[(int64_t)(j0 + r) * k + c] : 0.0;
        }
        {
            const int n_el = min(TR, n - j0) * k;                                           // X^T U  (:424)
            if (px.nranks > 0) {
                for (int e = threadIdx.x; e < n_el; e += 256) sB[e] = sum_peers(px, (int64_t)j0 * k + e);
            } else {
                epi_stage_sums(sB, Bsrc + (int64_t)j0 * k, n_el, bchunks, bstride);
            }
        }
        __syncthreads();
        double den[RPT][CPT];
#pragma unroll
        for (int i = 0; i < RPT; ++i)
#pragma unroll
            for (int j = 0; j < CPT; ++j) den[i][j] = 0.0;
        for (int l = 0; l < k; ++l) {                                                       // V.Gu   (:425)
            double v[RPT], gu[CPT];
#pragma unroll
            for (int i = 0; i < RPT; ++i) v[i] = sV[(ty + 16 * i) * LD + l];
#pragma unroll
            for (int j = 0; j < CPT; j += 2) {
                const double2 t2 = *reinterpret_cast<const double2*>(sGu + l * KT + tiled_col<CPT>(tx, j));
                gu[j] = t2.x; gu[j + 1] = t2.y;
            }
#pragma unroll
            for (int i = 0; i < RPT; ++i)
#pragma unroll
                for (int j = 0; j < CPT; ++j) den[i][j] = fma(v[i], gu[j], den[i][j]);
        }
        double vnew[RPT][CPT];
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            const int r = ty + 16 * i;
            const int jg = j0 + r;
#pragma unroll
            for (int j = 0; j < CPT; ++j) {
                const int c = tiled_col<CPT>(tx, j);
                double vn = 0.0;
                if (jg < n && c < k) {
                    const double v = sV[r * LD + c];
                    const double b = sB[r * k + c];
                    const int32_t pr = pos[(int64_t)jg * k + c];
                    double wv = 0.0, dg = 0.0;
                    if (pr >= 0) { wv = pathway_term<false>(pw, active, pr, c, Vold, k); dg = pw.deg[pr]; }
                    vn = v_update_value(v, b, den[i][j], pr >= 0, wv, dg, gamma, delta);
                    Vnew[(int64_t)jg * k + c] = vn;
                    vb = fma(vn, b, vb);
                }
                vnew[i][j] = vn;
            }
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < RPT; ++i)
#pragma unroll
            for (int j = 0; j < CPT; ++j) sV[(ty + 16 * i) * LD + tiled_col<CPT>(tx, j)] = vnew[i][j];
        __syncthreads();
        for (int r = 0; r < TR; ++r) {
            double va[CPT], vbb[CPT];
#pragma unroll
            for (int j = 0; j < CPT; j += 2) {
                const double2 a2 = *reinterpret_cast<const double2*>(sV + r * LD + tiled_col<CPT>(ty, j));
                const double2 b2 = *reinterpret_cast<const double2*>(sV + r * LD + tiled_col<CPT>(tx, j));
                va[j] = a2.x; va[j + 1] = a2.y; vbb[j] = b2.x; vbb[j + 1] = b2.y;
            }
#pragma unroll
            for (int i = 0; i < CPT; ++i)
#pragma unroll
                for (int j = 0; j < CPT; ++j) g[i][j] = fma(va[i], vbb[j], g[i][j]);
        }
    }
    double* out = Gv_part + (int64_t)blockIdx.x * k * k;
#pragma unroll
    for (int i = 0; i < CPT; ++i) {
        const int a = tiled_col<CPT>(ty, i);
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
            const int b = tiled_col<CPT>(tx, j);
            if (a < k && b < k) out[a * k + b] = g[i][j];
        }
    }
    const double tvb = block_sum(vb, scratch);
    if (threadIdx.x == 0) VB_part[blockIdx.x] = tvb;
}

// manifold / ignore terms of the objective (:344-352) over the flattened active set, spread over the grid (large k:
// k pathways x hundreds of entries are too many gathers for one block).  Per-block partials, fixed order.
static __global__ void __launch_bounds__(256)
manifold_parts_kernel(const double* __restrict__ V, int k, const double* __restrict__ Gv, ActiveSet as,
                      double* __restrict__ man_part, double* __restrict__ ign_part) {
    __shared__ double scratch[32];
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (int64_t)gridDim.x * blockDim.x;
    double man = 0.0, ign = 0.0;
    for (int64_t i = t; i < as.n_diag; i += nt) {
        const int c = as.diag_factor[i];
        const double vr = V[(int64_t)as.diag_gene[i] * k + c] / sqrt(Gv[c * k + c]);
        man = fma(as.diag_coef[i] * vr, vr, man);
        ign += 1.0 / (vr + 1.0);
    }
    for (int64_t i = t; i < as.n_off; i += nt) {
        const int c = as.off_factor[i];
        const double nrm = sqrt(Gv[c * k + c]);
        man = fma(as.off_coef[i] * (V[(int64_t)as.off_c[i] * k + c] / nrm), V[(int64_t)as.off_r[i] * k + c] / nrm, man);
    }
    const double MAN = block_sum(man, scratch);
    const double IGN = block_sum(ign, scratch);
    if (threadIdx.x == 0) { man_part[blockIdx.x] = MAN; ign_part[blockIdx.x] = IGN; }
}

// Objective of one inner step as its own one-block launch (large k: after gram_reduce_kernel folded the Gram
// partials; Gu and Gv arrive as single k*k matrices, the sum(V_new*B) partials per V-update block).
static __global__ void __launch_bounds__(kTailThreads)
objective_kernel(const double* __restrict__ V, int k, const double* __restrict__ Gu, const double* __restrict__ Gv_in,
                 const double* __restrict__ VB_part, int vb_parts, const double* __restrict__ man_part,
                 const double* __restrict__ ign_part, int mi_parts, const double* __restrict__ normX_sq,
                 double* __restrict__ Gv, double* __restrict__ gd, double tradeoff, double* __restrict__ obj_out,
                 int* __restrict__ step_counter, int obj_capacity) {
    extern __shared__ double sm[];
    const int kk2 = k * k;
    // same shared-memory plan as the fused V-update kernel: two k*k arrays only fit up to k = 64
    double* sGu = sm;
    double* sGv = sm + kk2;                                   // k <= 64: Gv_new; else the 1024-double slice buffer
    double* sSl = sm + kk2 + (k > 64 ? 1024 : kk2);           // 1024 doubles
    double* sVh = sSl + 1024;                                 // kVhCap doubles
    __shared__ double scratch[5 * 32 + 128];
    for (int i = threadIdx.x; i < kk2; i += blockDim.x) sGu[i] = Gu[i];
    __syncthreads();
    // the manifold / ignore terms were summed by manifold_parts_kernel: hand objective_block an empty active set and
    // add them (fixed order) to what it writes
    ActiveSet none{};
    const int s0 = *step_counter;
    __syncthreads();
    objective_block(V, k, sGu, k > 64 ? Gv : sGv, k > 64 ? sGv : sSl, scratch, Gv_in, VB_part, vb_parts, 1, normX_sq, none, Gv,
                    gd, -1.0, obj_out, step_counter, obj_capacity, sVh, kVhCap);
    if (threadIdx.x == 0) {
        double MAN = 0.0, IGN = 0.0;
        for (int b = 0; b < mi_parts; ++b) { MAN += man_part[b]; IGN += ign_part[b]; }
        if (s0 < obj_capacity) {
            double* o = obj_out + (int64_t)s0 * kObjStride;
            const double gamma = o[5], delta = o[6], recon = o[0];
            o[1] = MAN; o[2] = IGN;
            o[4] = recon + gamma * MAN + delta * IGN + o[3];                                 // :362
            if (tradeoff >= 0.0) {                                                           // :542-548
                const double den = tradeoff * MAN;
                const double g2 = (den == 0.0) ? 1.0 : ((1.0 - tradeoff) * recon) / den;
                gd[0] = g2; gd[1] = g2;
            }
        }
    }
}

// Objective of one inner step from per-panel partials (fused-tail path, k <= 10: the V update ran inside the pass-2
// kernel and left `vparts` partials of V_new^T V_new and sum(V_new*B); Gu arrives as `gu_parts` partials).
static __global__ void __launch_bounds__(kTailThreads)
objective_parts_kernel(const double* __restrict__ V, int k, const double* __restrict__ Gu_part, int gu_parts,
                       const double* __restrict__ Gv_part, const double* __restrict__ VB_part, int vparts,
                       const double* __restrict__ normX_sq, ActiveSet as, double* __restrict__ Gv,
                       double* __restrict__ gd, double tradeoff, double* __restrict__ obj_out,
                       int* __restrict__ step_counter, int obj_capacity) {
    extern __shared__ double sm[];
    const int kk2 = k * k;
    double* sGu = sm;
    double* sGv = sm + kk2;
    double* sSl = sGv + kk2;            // 1024 doubles
    double* sVh = sSl + 1024;           // kVhCap doubles
    __shared__ double scratch[5 * 32 + 128];
    sum_gram_partials(sGu, Gu_part, gu_parts, kk2, sSl);
    objective_block(V, k, sGu, sGv, sSl, scratch, Gv_part, VB_part, vparts, vparts, normX_sq, as, Gv, gd, tradeoff, obj_out,
                    step_counter, obj_capacity, sVh, kVhCap);
}

// Deferred objective (fused-tail path, fixed gamma / delta): block s evaluates the objective of inner step s of
// the block from what that step's V update left behind (per-panel Gram and sum(V_new*B) partials, U^T U, the
// active-set values of V_new), so a block of n steps costs ONE launch instead of n on the critical path.  The
// last block publishes Gv_new.  Same arithmetic and summation orders as objective_parts_kernel.
static __global__ void __launch_bounds__(kTailThreads)
objective_deferred_kernel(int k, const double* __restrict__ hist_Gu, const double* __restrict__ hist_Gvp,
                          const double* __restrict__ hist_VBp, int vparts, const double* __restrict__ hist_vh,
                          int vh_stride, const double* __restrict__ normX_sq, ActiveSet as, double* __restrict__ Gv,
                          double* __restrict__ gd, double* __restrict__ obj_out, int obj_capacity) {
    extern __shared__ double sm[];
    const int kk2 = k * k;
    const int s = blockIdx.x;
    double* sGu = sm;
    double* sGv = sm + kk2;
    double* sSl = sGv + kk2;            // 1024 doubles
    double* sVh = sSl + 1024;           // kVhCap doubles
    __shared__ double scratch[5 * 32 + 128];
    for (int i = threadIdx.x; i < kk2; i += blockDim.x) sGu[i] = hist_Gu[(int64_t)s * kk2 + i];
    __syncthreads();
    objective_block(nullptr, k, sGu, sGv, sSl, scratch, hist_Gvp + (int64_t)s * vparts * kk2, hist_VBp + (int64_t)s * vparts,
                    vparts, vparts, normX_sq, as, Gv, gd, -1.0, obj_out, nullptr, obj_capacity, sVh, kVhCap,
                    hist_vh + (int64_t)s * vh_stride, s, s == (int)gridDim.x - 1);
}

// Gram of V from scratch (after prmf_set_UV): same tiling as the update kernel so partial layout matches.
template <int NQ>
__global__ void __launch_bounds__(256)
gram_rows_kernel(const double* __restrict__ M, int64_t rows_total, int k, int rows_per_tile,
                 double* __restrict__ G_part) {
    extern __shared__ double sm[];
    double* sT = sm;
    const int kk2 = k * k;
    double gacc[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) gacc[q] = 0.0;
    const int64_t ntiles = (rows_total + rows_per_tile - 1) / rows_per_tile;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t r0 = tile * rows_per_tile;
        const int rows = (int)min((int64_t)rows_per_tile, rows_total - r0);
        __syncthreads();
        for (int e = threadIdx.x; e < rows * k; e += blockDim.x) sT[e] = M[r0 * k + e];
        __syncthreads();
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const int pidx = threadIdx.x + q * 256;
            if (pidx < kk2) {
                const int a = pidx / k, b = pidx - a * k;
                double s = gacc[q];
                for (int r = 0; r < rows; ++r) s = fma(sT[r * k + a], sT[r * k + b], s);
                gacc[q] = s;
            }
        }
    }
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        const int pidx = threadIdx.x + q * 256;
        if (pidx < kk2) G_part[(int64_t)blockIdx.x * kk2 + pidx] = gacc[q];
    }
}

// G[e] = sum_b G_part[b][e]  (fixed order)
static __global__ void __launch_bounds__(256)
sum_gram_parts_kernel(const double* __restrict__ G_part, int blocks, int kk2, double* __restrict__ G) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < kk2) {
        double s = 0.0;
        for (int b = 0; b < blocks; ++b) s += G_part[(int64_t)b * kk2 + e];
        G[e] = s;
    }
}

// ----------------------------------------------------------------------------------------------------
// Factor x pathway tables (restrict :129-194 / score :115-127, force_distinct_lapls :232, find_mins :49):
//   mass[c][p]      = sum_{i in supp_p} vu_i^2                      vu = V[:,c] / ||V[:,c]||
//   quad_norm[c][p] = vu^T (D^-1/2 L_p D^-1/2) vu
//   quad_raw[c][p]  = V[:,c]^T L_p V[:,c]
// One block per (pathway, tile of F factors).  The V rows of the support are staged once in shared memory
// (coalesced row reads: F contiguous factors per gene); thread (row lane, factor) walks the packed CSR row of
// its support row for its factor, so the CSR of a pathway is read once per factor TILE (the F threads of a row
// read the same entries: a broadcast) and every neighbour gather is a shared-memory read.  The row lanes of a
// factor are combined in a fixed order.  Pathways whose support does not fit the staging buffer gather from
// global memory with the same arithmetic.
// ----------------------------------------------------------------------------------------------------
template <int F>
__global__ void __launch_bounds__(256)
scores_kernel(const double* __restrict__ V, int k, const double* __restrict__ Gv, Pathways pw, int rows_cap, int edges_cap,
              double* __restrict__ mass, double* __restrict__ quad_norm, double* __restrict__ quad_raw) {
    // staged copy of one pathway: V rows of the support (F factors), isd, ldiag, w | row offsets, neighbour indices
    extern __shared__ double s_dyn[];
    double* sV = s_dyn;                                // rows_cap x F
    double* sIsd = sV + (size_t)rows_cap * F;          // rows_cap
    double* sLd = sIsd + rows_cap;                     // rows_cap
    double* sW = sLd + rows_cap;                       // edges_cap
    int32_t* sRow = reinterpret_cast<int32_t*>(sW + edges_cap);   // rows_cap + 1 (relative to the pathway's first edge)
    int32_t* sCol = sRow + rows_cap + 1;               // edges_cap
    __shared__ double sRed[3][256];
    constexpr int RL = 256 / F;                        // row lanes
    const int t = threadIdx.x;
    const int f = t % F, rl = t / F;
    const int f0 = (int)blockIdx.y * F;
    const int c = f0 + f;
    const bool live = rl < RL && c < k;
    const double nrm = live ? sqrt(Gv[c * k + c]) : 1.0;
    for (int p = blockIdx.x; p < pw.P; p += gridDim.x) {
        const int64_t beg = pw.path_ptr[p], end = pw.path_ptr[p + 1];
        const int s = (int)(end - beg);
        const int64_t ebeg = pw.row_ptr[beg];
        const int ne = (int)(pw.row_ptr[end] - ebeg);
        const bool staged = s <= rows_cap && ne <= edges_cap;
        __syncthreads();                               // previous pathway's readers are done with the staged copy / sRed
        if (staged) {                                  // every range is contiguous in the packed tables: coalesced copies
            for (int idx = t; idx < s * F; idx += 256) {
                const int r = idx / F, ff = idx - r * F;
                sV[idx] = (f0 + ff < k) ? V[(int64_t)pw.support_idx[beg + r] * k + f0 + ff] : 0.0;
            }
            for (int r = t; r < s; r += 256) { sIsd[r] = pw.isd[beg + r]; sLd[r] = pw.ldiag[beg + r]; }
            for (int r = t; r <= s; r += 256) sRow[r] = (int32_t)(pw.row_ptr[beg + r] - ebeg);
            for (int e = t; e < ne; e += 256) { sCol[e] = pw.col_local[ebeg + e]; sW[e] = pw.w[ebeg + e]; }
        }
        __syncthreads();
        double ms = 0.0, qn = 0.0, qr = 0.0;
        if (live && staged) {
            for (int r = rl; r < s; r += RL) {
                const double v = sV[r * F + f];
                const double vu = v / nrm;
                const double ir = sIsd[r];
                const double ld = sLd[r];
                double yn = (ir * (ld * ir)) * vu;
                double yr = ld * v;
                const int e1 = sRow[r + 1];
                for (int e2 = sRow[r]; e2 < e1; ++e2) {
                    const int cl = sCol[e2];
                    if (cl == r) continue;             // a self loop is part of diag(L)
                    const double vc = sV[cl * F + f];
                    const double we = sW[e2];
                    yn = fma(ir * (-we * sIsd[cl]), vc / nrm, yn);
                    yr = fma(-we, vc, yr);
                }
                ms = fma(vu, vu, ms);
                qn = fma(yn, vu, qn);
                qr = fma(yr, v, qr);
            }
        } else if (live) {                             // support or edge list larger than the staging buffers
            for (int r = rl; r < s; r += RL) {
                const int64_t gr = beg + r;
                const double v = V[(int64_t)pw.support_idx[gr] * k + c];
                const double vu = v / nrm;
                const double ir = pw.isd[gr];
                const double ld = pw.ldiag[gr];
                double yn = (ir * (ld * ir)) * vu;
                double yr = ld * v;
                const int64_t e1 = pw.row_ptr[gr + 1];
                for (int64_t e2 = pw.row_ptr[gr]; e2 < e1; ++e2) {
                    const int cl = pw.col_local[e2];
                    if (cl == r) continue;
                    const double vc = V[(int64_t)pw.support_idx[beg + cl] * k + c];
                    const double we = pw.w[e2];
                    yn = fma(ir * (-we * pw.isd[beg + cl]), vc / nrm, yn);
                    yr = fma(-we, vc, yr);
                }
                ms = fma(vu, vu, ms);
                qn = fma(yn, vu, qn);
                qr = fma(yr, v, qr);
            }
        }
        sRed[0][t] = ms; sRed[1][t] = qn; sRed[2][t] = qr;
        __syncthreads();
        if (t < 3 * F) {                               // thread (table, factor): the row lanes in order
            const int tab = t / F, ff = t - tab * F;
            if (f0 + ff < k) {
                double a = 0.0;
#pragma unroll 5
                for (int l = 0; l < RL; ++l) a += sRed[tab][l * F + ff];
                double* dst = tab == 0 ? mass : tab == 1 ? quad_norm : quad_raw;
                dst[(int64_t)(f0 + ff) * pw.P + p] = a;
            }
        }
    }
}

// manifold / ignore terms of the objective (:344-352) for the current V, standalone (prmf_objective).
static __global__ void __launch_bounds__(1024)
manifold_ignore_kernel(const double* __restrict__ V, int k, const double* __restrict__ Gv, ActiveSet as,
                       double* __restrict__ out2) {
    __shared__ double scratch[32];
    const int t = threadIdx.x;
    double man = 0.0, ign = 0.0;
    for (int64_t i = t; i < as.n_diag; i += blockDim.x) {
        const int c = as.diag_factor[i];
        const double vr = V[(int64_t)as.diag_gene[i] * k + c] / sqrt(Gv[c * k + c]);
        man = fma(as.diag_coef[i] * vr, vr, man);
        ign += 1.0 / (vr + 1.0);
    }
    for (int64_t i = t; i < as.n_off; i += blockDim.x) {
        const int c = as.off_factor[i];
        const double nrm = sqrt(Gv[c * k + c]);
        man = fma(as.off_coef[i] * (V[(int64_t)as.off_c[i] * k + c] / nrm), V[(int64_t)as.off_r[i] * k + c] / nrm, man);
    }
    const double MAN = block_sum(man, scratch);
    const double IGN = block_sum(ign, scratch);
    if (t == 0) { out2[0] = MAN; out2[1] = IGN; }
}

// ----------------------------------------------------------------------------------------------------
// Exact residual ||X - U V^T||_F^2 (verification only; one extra pass over X).  Warp per row.
// ----------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
residual_kernel(const double* __restrict__ X, int64_t ldx, int64_t m, int n, const double* __restrict__ U,
                const double* __restrict__ V, int k, double* __restrict__ part) {
    __shared__ double scratch[32];
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double acc = 0.0;
    for (int64_t row = warp; row < m; row += nwarps) {
        const double* xr = X + row * ldx;
        const double* ur = U + row * k;
        for (int j = lane; j < n; j += 32) {
            double s = 0.0;
            for (int l = 0; l < k; ++l) s = fma(ur[l], V[(int64_t)j * k + l], s);
            const double d = xr[j] - s;
            acc = fma(d, d, acc);
        }
    }
    const double t = block_sum(acc, scratch);
    if (threadIdx.x == 0) part[blockIdx.x] = t;
}

}  // namespace prmf
