// TF32 tensor-core X streams (opt-in storage mode PRMF_X_TF32: X kept in HBM as fp32 rounded to tf32).
//
// Both products of the inner step (prmf_runner.py:420 X.V and :424 X^T.U) become one kernel,
//     Out[chunk][r][0:k] = sum_{c in chunk} M[r][c] * Wt[f][c]        (M: R x C fp32 row-major, Wt: Kp x C fp32)
// with (M, Wt) = (X, V^T) for pass 1 and (X^T, U^T) for pass 2 -- both operands K-major, so the canonical
// 128-byte-swizzled shared-memory layout serves A and B.  Per CTA: one 128-row tile of M and one column chunk.
//   warp 0 (one lane)  TMA producer: 2-D tensor-map copies (cp.async.bulk.tensor, SWIZZLE_128B) of a 128 x 32 tile
//                      of M (L2 evict_first: streamed once) and the Kp x 32 tile of Wt (evict_last: shared by all
//                      CTAs) into a ring of stages, completion on mbarriers
//   warp 1 (one lane)  tcgen05.mma.cta_group::1.kind::tf32, M = 128, N = Kp, K = 8 (4 per stage); the fp32
//                      accumulator (128 lanes x Kp columns) lives in TMEM; tcgen05.commit releases the stage
//   warps 0..3         epilogue: tcgen05.ld (32 lanes x 16 columns per warp and instruction) -> fp64 -> the SAME
//                      per-chunk partial layout the fp64 X-stream kernels write, so the U / V updates, the
//                      objective and the sharded reduction are unchanged (and stay fp64)
// At k = 128 the contraction is dense enough (64 flop per byte of X) that only the tensor cores keep the pass
// HBM-bound; at k = 10 the same kernel simply halves the bytes of the fp64 path.  Two CTAs are resident per SM so
// one CTA's epilogue overlaps the other's stream.
//
// Numerics: X, U, V are rounded to tf32 (round-to-nearest, cvt.rna) when they are stored, products are exact,
// accumulation is fp32 in TMEM; chunk partials are added in fp64 in a fixed order.  This mode is NOT the parity
// mode (tests state its tolerance against the fp64 oracle).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.cuh"

namespace prmf {

constexpr int kTcTileRows = 128;      // UMMA M
constexpr int kTcBlockK = 32;         // fp32 elements per stage row = one 128-byte swizzle atom
constexpr int kTcUmmaK = 8;           // tf32: 32 bytes of K per instruction
constexpr int kTcThreads = 128;

__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c_inner, int c_outer, uint64_t* bar,
                                            uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)),
        "r"(smem_u32(bar)), "r"(c_inner), "r"(c_outer), "l"(policy) : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format): start address >> 4 in bits [0,14),
// leading byte offset (unused for swizzled K-major, 1) in [16,30), stride byte offset = 1024 B between 8-row
// groups in [32,46), version 1 in [46,48), layout type 2 (SWIZZLE_128B) in [61,64).
__device__ __forceinline__ uint64_t umma_desc_k128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fffu);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Instruction descriptor of kind::tf32: D = f32 (bits 4-5 = 1), A = B = tf32 (bits 7-9, 10-12 = 2), both K-major,
// N >> 3 in bits [17,23), M >> 4 in bits [24,29).
__host__ __device__ inline uint32_t umma_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}

__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

struct TcParams {
    int64_t R, C;                // M is R x C
    int k, Kp;                   // factors; Kp = k rounded up to a multiple of 16 (the UMMA N)
    int64_t cols_per_chunk;      // multiple of kTcBlockK
    int stages;
    uint32_t tmem_cols;          // power of two >= max(32, Kp)
    double* Out;                 // [chunks][R][k]
};

__global__ void __launch_bounds__(kTcThreads)
tc_rowdot_kernel(const __grid_constant__ CUtensorMap tmM, const __grid_constant__ CUtensorMap tmW, const TcParams p) {
    extern __shared__ unsigned char tc_smem_raw[];
    // SWIZZLE_128B tiles need 1024-byte alignment
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)tc_smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t a_bytes = kTcTileRows * kTcBlockK * 4;                 // 16 KB
    const uint32_t b_bytes = (uint32_t)p.Kp * kTcBlockK * 4;              // Kp x 128 B
    const uint32_t stage_bytes = a_bytes + b_bytes;
    const int S = p.stages;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)S * stage_bytes);
    uint64_t* empty_bar = full_bar + S;
    uint64_t* tmem_full = empty_bar + S;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t tile = blockIdx.x, chunk = blockIdx.y;
    const int64_t r_tile = tile * kTcTileRows;
    const int64_t cbeg = chunk * p.cols_per_chunk;
    const int64_t cend = min(p.C, cbeg + p.cols_per_chunk);
    const int nkb = cend > cbeg ? (int)((cend - cbeg + kTcBlockK - 1) / kTcBlockK) : 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(tmem_full, 1);
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // ===== TMA producer =====
            const uint64_t pol_m = l2_policy_evict_first();
            const uint64_t pol_w = l2_policy_evict_last();
            int s = 0;
            uint32_t phase = 0;
            for (int kb = 0; kb < nkb; ++kb) {
                mbar_wait(&empty_bar[s], phase ^ 1u);
                unsigned char* sa = smem + (size_t)s * stage_bytes;
                mbar_arrive_expect_tx(&full_bar[s], stage_bytes);
                const int c0 = (int)(cbeg + (int64_t)kb * kTcBlockK);
                tma_load_2d(sa, &tmM, c0, (int)r_tile, &full_bar[s], pol_m);
                tma_load_2d(sa + a_bytes, &tmW, c0, 0, &full_bar[s], pol_w);
                if (++s == S) { s = 0; phase ^= 1u; }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            // ===== MMA issuer =====
            const uint32_t idesc = umma_idesc_tf32(kTcTileRows, p.Kp);
            int s = 0;
            uint32_t phase = 0;
            for (int kb = 0; kb < nkb; ++kb) {
                mbar_wait(&full_bar[s], phase);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes);
                const uint64_t da = umma_desc_k128(sa);
                const uint64_t db = umma_desc_k128(sa + a_bytes);
#pragma unroll
                for (int j = 0; j < kTcBlockK / kTcUmmaK; ++j) {
                    // advance 32 bytes along K inside the swizzle atom: +2 in the (address >> 4) field
                    umma_tf32(tmem_base, da + (uint64_t)(j * 2), db + (uint64_t)(j * 2), idesc, (kb | j) != 0 ? 1u : 0u);
                }
                umma_commit(&empty_bar[s]);                       // frees the stage when these MMAs have read it
                if (++s == S) { s = 0; phase ^= 1u; }
            }
            umma_commit(tmem_full);                               // accumulator complete
        }
        __syncwarp();
    }

    // ===== epilogue: all four warps; warp w owns TMEM lanes 32w .. 32w+31 = rows r_tile + 32w + lane =====
    if (nkb > 0) {
        mbar_wait(tmem_full, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    const int64_t row = r_tile + warp * 32 + lane;
    double* out = p.Out + ((int64_t)chunk * p.R + row) * p.k;
    for (int c0 = 0; c0 < p.Kp; c0 += 16) {
        uint32_t v[16];
        if (nkb > 0) {
            tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
        } else {
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = 0u;
        }
        if (row < p.R) {
#pragma unroll
            for (int q = 0; q < 16; ++q)
                if (c0 + q < p.k) out[c0 + q] = (double)__uint_as_float(v[q]);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
    }
}

// ---- storage conversions --------------------------------------------------------------------------------
// dst[r][c] = tf32(src[r][c]) (TF32) or the nearest fp32 value, as astype(np.float32) rounds (PRMF_X_F32), for c < n;
// 0 for n <= c < ld_dst (T = double or float source)
template <typename T, bool TF32>
__global__ void __launch_bounds__(256)
to_tf32_rows_kernel(const T* __restrict__ src, int64_t ld_src, int64_t rows, int64_t n, float* __restrict__ dst,
                    int64_t ld_dst) {
    const int64_t total = rows * ld_dst;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / ld_dst, c = i - r * ld_dst;
        if (TF32) dst[i] = c < n ? to_tf32((float)src[r * ld_src + c]) : 0.0f;
        else dst[i] = c < n ? (float)src[r * ld_src + c] : 0.0f;
    }
}

__global__ void __launch_bounds__(256)
transpose_f32_kernel(const float* __restrict__ X, int64_t ldx, int64_t m, int64_t n, float* __restrict__ Xt,
                     int64_t ldxt) {
    __shared__ float tile[32][33];
    const int64_t i0 = (int64_t)blockIdx.y * 32, j0 = (int64_t)blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int64_t i = i0 + r, j = j0 + tx;
        tile[r][tx] = (i < m && j < n) ? X[i * ldx + j] : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int64_t j = j0 + r, i = i0 + tx;
        if (j < n && i < m) Xt[j * ldxt + i] = tile[tx][r];
    }
}

// Wt[f][r] = tf32(W[r][f]) for f < k, 0 for k <= f < Kp   (W: rows x k fp64 row-major; Wt: Kp x ld fp32)
__global__ void __launch_bounds__(256)
cast_transpose_w_kernel(const double* __restrict__ W, int64_t rows, int k, int Kp, float* __restrict__ Wt, int64_t ld) {
    __shared__ float tile[32][33];
    const int64_t r0 = (int64_t)blockIdx.x * 32;
    const int f0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int q = ty; q < 32; q += 8) {
        const int64_t r = r0 + q;
        const int f = f0 + tx;
        tile[q][tx] = (r < rows && f < k) ? to_tf32((float)W[r * k + f]) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int q = ty; q < 32; q += 8) {
        const int f = f0 + q;
        const int64_t r = r0 + tx;
        if (f < Kp && r < rows) Wt[(int64_t)f * ld + r] = tile[tx][q];
    }
}

// ||X||_F^2 of the stored (rounded) fp32 matrix, per-block partials (fixed order)
__global__ void __launch_bounds__(256) sumsq_f32_kernel(const float* __restrict__ X, int64_t ldx, int64_t m, int64_t n,
                                                        double* __restrict__ part) {
    __shared__ double scratch[32];
    double acc = 0.0;
    for (int64_t row = blockIdx.x; row < m; row += gridDim.x) {
        const float* xr = X + row * ldx;
        double a = 0.0;
        for (int64_t j = threadIdx.x; j < n; j += blockDim.x) {
            const double x = (double)xr[j];
            a = fma(x, x, a);
        }
        acc += a;
    }
    const double t = block_sum(acc, scratch);
    if (threadIdx.x == 0) part[blockIdx.x] = t;
}

// exact residual ||X - U V^T||_F^2 against the stored fp32 X (verification; fp64 arithmetic)
__global__ void __launch_bounds__(256)
residual_f32_kernel(const float* __restrict__ X, int64_t ldx, int64_t m, int n, const double* __restrict__ U,
                    const double* __restrict__ V, int k, double* __restrict__ part) {
    __shared__ double scratch[32];
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double acc = 0.0;
    for (int64_t row = warp; row < m; row += nwarps) {
        const float* xr = X + row * ldx;
        const double* ur = U + row * k;
        for (int j = lane; j < n; j += 32) {
            double s = 0.0;
            for (int l = 0; l < k; ++l) s = fma(ur[l], V[(int64_t)j * k + l], s);
            const double d = (double)xr[j] - s;
            acc = fma(d, d, acc);
        }
    }
    const double t = block_sum(acc, scratch);
    if (threadIdx.x == 0) part[blockIdx.x] = t;
}

}  // namespace prmf
