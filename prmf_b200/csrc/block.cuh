// block.cuh -- the persistent step kernel (k <= 10, fp64): a whole block of inner steps in ONE cooperative launch.
//
// An inner step (reference prmf_runner.py:419-444) is two passes over X separated by full reductions:
//   half-step "pass 1":  A = X.V  (streams the transposed copy Xt)  -> U update  (:420-422) + partials of U_new^T U_new
//   half-step "pass 2":  B = X^T.U_new (streams X)                  -> V update  (:424-444) + what the objective needs
// skinny_tma_kernel runs each half as its own launch; every launch pays the ramp-up of its TMA ring, its fused tail
// with the SMs idle on HBM, and a kernel boundary.  Here one CTA per SM stays resident for `nh` consecutive halves:
//   * the producer warp runs ahead across the half boundary: while the 8 consumer warps are still in the tail of
//     half h, it has already refilled the whole ring with the X tiles of half h+1 (they depend on nothing); only
//     the small W operand (rows of V / U_new) waits for the data dependency, a monotone counter in L2;
//   * kernel boundaries are replaced by those counters: `udone` (all sample panels updated and folded) gates the
//     W rows of pass 2 and the V update; `vdone` gates the W rows of the next pass 1 and the next U update;
//   * on several GPUs the sum over ranks of [X^T U | U^T U] is part of the pass-2 tail: every thread pushes the sums it
//     owns straight into every peer's receive buffer as 16-byte {value, sequence number} entries (one NVLink store
//     each, no fence, no flag) and polls the same entries of all ranks in its OWN memory until their sequence number is
//     this step's, adding them in rank order -- one one-way hop, bitwise identical on all ranks, no collective launch.
//     U^T U is pushed at the START of pass 2 (it is complete after pass 1), so it has the whole pass to arrive.
// Every spin wait has a %globaltimer deadline: on expiry the kernel sets an error word, stops waiting and drains;
// the host reports PRMF_ERR_TIMEOUT instead of hanging (dead peer, lost launch).
// The objective is deferred exactly as on the two-launch path: every step leaves its Gram partials, U^T U and the
// active-set values of V_new in per-step slots; objective_deferred_kernel evaluates the block afterwards.
#pragma once

#include "block_params.h"

namespace prmf {

// Low-latency exchange entries (NCCL's LL protocol with 64-bit payloads): a double travels as TWO 8-byte words, each
// carrying 32 bits of the value and the low 32 bits of the step's sequence number,
//     word0 = seq32 << 32 | lo32(value)        word1 = seq32 << 32 | hi32(value)
// written by one 16-byte store.  The receiver needs neither a fence nor a separate flag: it polls the entry itself until
// BOTH words carry the expected sequence number.  Only 8-byte single-copy atomicity is assumed (the PTX memory model
// treats a .v2 access as two scalar accesses): if the halves of the 16-byte store ever became visible separately, each
// half still validates itself.  One one-way NVLink hop per exchange.
__device__ __forceinline__ void ll_store(ulonglong2* dst, double v, unsigned long long seq) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
    const unsigned long long tag = (seq & 0xffffffffull) << 32;
    const unsigned long long w0 = tag | (bits & 0xffffffffull), w1 = tag | (bits >> 32);
    asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(w0), "l"(w1) : "memory");
}
__device__ __forceinline__ bool ll_valid(unsigned long long w0, unsigned long long w1, unsigned long long seq) {
    const unsigned long long tag = seq & 0xffffffffull;
    return (w0 >> 32) == tag && (w1 >> 32) == tag;
}
__device__ __forceinline__ double ll_value(unsigned long long w0, unsigned long long w1) {
    return __longlong_as_double((long long)((w1 << 32) | (w0 & 0xffffffffull)));
}

__device__ __forceinline__ double ll_wait(const ulonglong2* src, unsigned long long seq, unsigned int* err,
                                          unsigned long long timeout_ns) {
    unsigned long long t0 = 0, w0, w1;
    unsigned int polls = 0;
    for (;;) {
        asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0), "=l"(w1) : "l"(src) : "memory");
        if (ll_valid(w0, w1, seq)) break;
        __nanosleep(20);
        if ((++polls & 255u) == 0u) {
            const unsigned long long now = blk_gtime();
            if (t0 == 0) t0 = now;
            if (now - t0 > timeout_ns || ld_volatile_u32(err) != 0u) {
                atomicOr(err, kErrTimeoutPeer);
                return 0.0;
            }
        }
    }
    return ll_value(w0, w1);
}

// Sum over ranks of one entry: the entries of ALL ranks are polled together (one round of local loads per sweep
// instead of one dependent poll per rank), then added in rank order.  Kept small on purpose: the kernel's main loop
// lives at the register limit of a 10-warp CTA (168 per thread); anything bigger here ends up as spills or register
// moves inside the stream (and a non-inlined call costs even more: the ABI pins the allocation of the whole kernel).
__device__ __forceinline__ double ll_gather(const ulonglong2* mine, size_t xpar, size_t xcount, int nranks, size_t idx,
                                            unsigned long long seq, unsigned int* err, unsigned long long timeout_ns) {
    double v[kMaxPeers];
    unsigned int pend = (1u << nranks) - 1u;
    unsigned long long t0 = 0;
    unsigned int polls = 0;
#pragma unroll
    for (int r = 0; r < kMaxPeers; ++r) v[r] = 0.0;
    while (pend) {
        unsigned long long w0[kMaxPeers], w1[kMaxPeers];
#pragma unroll
        for (int r = 0; r < kMaxPeers; ++r) {
            w0[r] = w1[r] = 0ull;
            if ((pend >> r) & 1u)
                asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0[r]), "=l"(w1[r]) : "l"(mine + (xpar + r) * xcount + idx));
        }
#pragma unroll
        for (int r = 0; r < kMaxPeers; ++r)
            if (((pend >> r) & 1u) && ll_valid(w0[r], w1[r], seq)) { v[r] = ll_value(w0[r], w1[r]); pend &= ~(1u << r); }
        if (pend) {
            __nanosleep(20);
            if ((++polls & 255u) == 0u) {
                const unsigned long long now = blk_gtime();
                if (t0 == 0) t0 = now;
                if (now - t0 > timeout_ns || ld_volatile_u32(err) != 0u) { atomicOr(err, kErrTimeoutPeer); break; }
            }
        }
    }
    double sum = 0.0;
#pragma unroll
    for (int r = 0; r < kMaxPeers; ++r) sum += v[r];          // rank order; absent ranks contribute +0.0
    return sum;
}

// per-thread running Gram accumulation over the sub-tiles of a share (thread = (pair a,b ; row slice))
template <int K>
struct BlkGram {
    static constexpr int NP = K * K;
    static constexpr int NS = (256 / NP) > 8 ? 8 : (256 / NP);
    double g = 0.0;
    __device__ __forceinline__ void add(const double* __restrict__ sT, int rows) {
        const int t = threadIdx.x;
        if (t < NP * NS) {
            const int pair = t % NP, sl = t / NP;
            const int a = pair / K, b = pair - a * K;
            const int rps = (rows + NS - 1) / NS;
            const int rb = sl * rps, re = min(rows, rb + rps);
            for (int r = rb; r < re; ++r) g = fma(sT[r * K + a], sT[r * K + b], g);
        }
    }
    // slice sums in order -> out[K*K]   (all 256 consumer threads call this)
    __device__ __forceinline__ void finish(double* __restrict__ sBuf, double* __restrict__ out) {
        const int t = threadIdx.x;
        if (t < NP * NS) sBuf[t] = g;             // sBuf[sl * NP + pair]
        cons_bar();
        if (t < NP) {
            double s = 0.0;
#pragma unroll
            for (int sl = 0; sl < NS; ++sl) s += sBuf[sl * NP + t];
            out[t] = s;
        }
    }
};

struct BlkTile {          // this CTA's tile of a pass
    bool in;              // CTA takes part in the pass
    int panel, chunk;
    int64_t c0;           // first column of the panel
    int width;            // columns held (multiple of 4)
    int64_t rbeg, rend;   // row range of the chunk
    int iters;            // ring stages this tile streams
};

__device__ __forceinline__ BlkTile blk_tile(int b, int panels, int panel_w, int chunks, int64_t rpc, int64_t rows_total,
                                            int64_t ldm) {
    BlkTile tl;
    tl.in = b < panels * chunks;
    tl.panel = b % panels;
    tl.chunk = b / panels;
    tl.c0 = (int64_t)tl.panel * panel_w;
    tl.width = (int)max((int64_t)0, min((int64_t)panel_w, ldm - tl.c0));
    tl.rbeg = (int64_t)tl.chunk * rpc;
    tl.rend = min(rows_total, tl.rbeg + rpc);
    tl.iters = (tl.in && tl.rend > tl.rbeg) ? (int)((tl.rend - tl.rbeg + kBlkRS - 1) / kBlkRS) : 0;
    return tl;
}

// rows [rb, rb + rows) of the panel's columns are this CTA's share of the update
__device__ __forceinline__ void blk_share(const BlkTile& tl, int chunks, int64_t cols, int& rb, int& rows) {
    const int all = (int)max((int64_t)0, min((int64_t)tl.width, cols - tl.c0));
    const int per = (all + chunks - 1) / chunks;
    rb = tl.chunk * per;
    rows = max(0, min(all, rb + per) - rb);
}

#ifdef PRMF_BLOCK_TIMING
// Developer instrumentation (not in the product build): %globaltimer stamps per CTA and half:
// [0] half entered  [1] first ring stage landed  [2] main loop done  [3] panel complete (arrive barrier passed)
// [4] sums over ranks done (pass 2, sharded)  [5] share updated  [6] tail done  [7] producer: W dependency satisfied
constexpr int kBlkDbgHalves = 24;
__device__ unsigned long long g_blk_dbg[160 * kBlkDbgHalves * 8];
#define BLK_STAMP(i_half, slot) do { if ((threadIdx.x & 255) == 0 && (i_half) < kBlkDbgHalves) \
        g_blk_dbg[((size_t)blockIdx.x * kBlkDbgHalves + (i_half)) * 8 + (slot)] = blk_gtime(); } while (0)
#define BLK_STAMP_P(i_half, slot) do { if (lane == 0 && (i_half) < kBlkDbgHalves) \
        g_blk_dbg[((size_t)blockIdx.x * kBlkDbgHalves + (i_half)) * 8 + (slot)] = blk_gtime(); } while (0)
#else
#define BLK_STAMP(i_half, slot) do { } while (0)
#define BLK_STAMP_P(i_half, slot) do { } while (0)
#endif

__device__ __forceinline__ void red_release_add(unsigned long long* p, unsigned long long v) {
    // release-add: the writes this CTA made before the preceding barrier are visible to whoever acquires the counter
    asm volatile("red.release.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long atom_acq_rel_add(unsigned long long* p, unsigned long long v) {
    unsigned long long old;
    asm volatile("atom.acq_rel.gpu.global.add.u64 %0, [%1], %2;" : "=l"(old) : "l"(p), "l"(v) : "memory");
    return old;
}
// consumers (256) + helper warp (32): the helper's prefetched operands are in shared memory
__device__ __forceinline__ void tail_bar() { asm volatile("bar.sync 2, 288;" ::: "memory"); }

template <int K>
__global__ void __launch_bounds__(kBlkThreads, 1)
block_kernel(const BlockParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int stages = p.stages;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_raw + (size_t)stages * p.ring_stage_bytes);
    uint64_t* empty_bar = full_bar + stages;
    double* scratch = reinterpret_cast<double*>(empty_bar + stages);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x;
    constexpr uint32_t w_bytes = (uint32_t)kBlkRS * K * 8u;
    constexpr int KK = K * K;
    __shared__ int s_last;
    // scratch: Gv | Gu (128 each) | 8 slice sums of a Gram | tail arrays
    double* sGv = scratch;                                 // V^T V of the current V (U update)
    double* sGu = scratch + 128;                           // U_new^T U_new, summed over ranks (V update)
    double* sW8 = sGu + 112;                               // 8 warp sums (K*K <= 100 < 112)
    double* sBuf = scratch + 256;                          // 8 * K*K slice sums
    // tail arrays, all views of the same kBlkRowsCap x K doubles:
    double* sR = sBuf + 8 * KK;                            // large shares: old rows, then the new ones (kBlkRowsCap x K)
    double* sT = sR;                                       // small shares: new rows | sums of the pass partials | old rows
    double* sS = sT + kBlkTile * K;                        //   (three arrays of kBlkTile x K)
    double* sO = sS + kBlkTile * K;
    double* pT = sR;                                       // pass 2 with the helper warp's prefetch (five arrays of kBlkPre x K):
    double* pS = pT + kBlkPre * K;                         //   new rows | sums | old rows | W.v of the active pathway | degree
    double* pO = pS + kBlkPre * K;
    double* pWv = pO + kBlkPre * K;
    double* pDg = pWv + kBlkPre * K;

    if (threadIdx.x == 0) {
        for (int s2 = 0; s2 < stages; ++s2) {
            mbar_init(&full_bar[s2], 1);
            mbar_init(&empty_bar[s2], kTmaConsumerWarps);
        }
        fence_mbar_init();
    }
    __syncthreads();

    const BlkTile t1 = blk_tile(b, p.panels1, p.panel_w1, p.chunks1, p.rpc1, p.n, p.ldxt);   // M = Xt: n rows, m columns
    const BlkTile t2 = blk_tile(b, p.panels2, p.panel_w2, p.chunks2, p.rpc2, p.m, p.ldx);    // M = X:  m rows, n columns
    const unsigned long long tiles1 = (unsigned long long)p.panels1 * p.chunks1;
    const unsigned long long tiles2 = (unsigned long long)p.panels2 * p.chunks2;
    int rb1, rows1, rb2, rows2;
    blk_share(t1, p.chunks1, p.m, rb1, rows1);
    blk_share(t2, p.chunks2, p.n, rb2, rows2);
    const bool helper_on = (p.flags & 1u) == 0u;
    const bool pre2 = helper_on && t2.in && rows2 <= kBlkPre;   // the helper warp prefetches the V update's operands

    if (warp == kTmaConsumerWarps) {
        // ================================= producer warp =================================
        const uint64_t pol_x = l2_policy_evict_first();
        const uint64_t pol_w = l2_policy_evict_last();
        int s2 = 0;
        uint32_t phase = 0;
        unsigned long long n1 = p.base1, n2 = p.base2;
        int ui = 0, vi = 0;                               // current U / V buffer
        for (int i = 0; i < p.nh; ++i) {
            const bool pass1 = ((p.h0 + i) & 1) == 0;
            const BlkTile& tl = pass1 ? t1 : t2;
            const double* M = pass1 ? p.Xt : p.X;
            const int64_t ldm = pass1 ? p.ldxt : p.ldx;
            const int panel_w = pass1 ? p.panel_w1 : p.panel_w2;
            // W of pass 1: the current V (that pass writes U[ui ^ 1] and flips ui); W of pass 2: the U this step's
            // pass 1 has just produced (that pass writes V[vi ^ 1] and flips vi)
            const double* Wsrc;
            if (pass1) { ++n1; Wsrc = p.V[vi]; ui ^= 1; }
            else { ++n2; Wsrc = p.U[ui]; vi ^= 1; }
            if (tl.iters > 0) {
                const uint32_t row_bytes = (uint32_t)tl.width * 8u;
                const uint32_t x_stage_bytes = (uint32_t)kBlkRS * (uint32_t)panel_w * 8u;
                // the data dependency of the W rows: every CTA of the previous half has stored its share
                const unsigned long long* dep = pass1 ? p.vdone : p.udone;
                const unsigned long long dep_target = pass1 ? n2 * tiles2 : n1 * tiles1;
                const int pre = min(stages, tl.iters);
                // X tiles of the first `pre` stages: no dependency, they go out as soon as the ring slots are free
                {
                    int s3 = s2;
                    uint32_t ph3 = phase;
                    for (int it = 0; it < pre; ++it) {
                        const int64_t r0 = tl.rbeg + (int64_t)it * kBlkRS;
                        const int rows = (int)min((int64_t)kBlkRS, tl.rend - r0);
                        if (lane == 0) {
                            mbar_wait(&empty_bar[s3], ph3 ^ 1u);
                            mbar_arrive_expect_tx(&full_bar[s3], (uint32_t)rows * row_bytes + w_bytes);
                        }
                        __syncwarp();
                        unsigned char* sx = smem_raw + (size_t)s3 * p.ring_stage_bytes;
                        if (lane < rows)
                            bulk_g2s(sx + (size_t)lane * panel_w * 8, M + (r0 + lane) * ldm + tl.c0, row_bytes, &full_bar[s3], pol_x);
                        if (++s3 == stages) { s3 = 0; ph3 ^= 1u; }
                    }
                }
                if (lane == 0) blk_wait_ge<false>(dep, dep_target, p.err, p.timeout_ns);
                BLK_STAMP_P(i, 7);
                __syncwarp();
                for (int it = 0; it < pre; ++it) {
                    const int64_t r0 = tl.rbeg + (int64_t)it * kBlkRS;
                    unsigned char* sx = smem_raw + (size_t)s2 * p.ring_stage_bytes;
                    if (lane == 0) bulk_g2s(sx + x_stage_bytes, Wsrc + r0 * K, w_bytes, &full_bar[s2], pol_w);
                    if (++s2 == stages) { s2 = 0; phase ^= 1u; }
                }
                for (int it = pre; it < tl.iters; ++it) {
                    const int64_t r0 = tl.rbeg + (int64_t)it * kBlkRS;
                    const int rows = (int)min((int64_t)kBlkRS, tl.rend - r0);
                    if (lane == 0) mbar_wait(&empty_bar[s2], phase ^ 1u);
                    __syncwarp();
                    unsigned char* sx = smem_raw + (size_t)s2 * p.ring_stage_bytes;
                    if (lane == 0) {
                        mbar_arrive_expect_tx(&full_bar[s2], (uint32_t)rows * row_bytes + w_bytes);
                        bulk_g2s(sx + x_stage_bytes, Wsrc + r0 * K, w_bytes, &full_bar[s2], pol_w);
                    }
                    __syncwarp();
                    if (lane < rows)
                        bulk_g2s(sx + (size_t)lane * panel_w * 8, M + (r0 + lane) * ldm + tl.c0, row_bytes, &full_bar[s2], pol_x);
                    if (++s2 == stages) { s2 = 0; phase ^= 1u; }
                }
            }
        }
        return;
    }

    if (warp == kTmaConsumerWarps + 1) {
        // ================================= helper warp =================================
        // While the consumer warps stream the pass, this warp fetches what their tail will need, so that the tail
        // itself is left with one round of loads (the pass partials): the Gram of the other factor matrix, and for
        // the V update the old rows of the share and the sparse terms of the active pathways (a chain of five
        // dependent gathers per entry: pos -> row_ptr -> col_local -> support_idx -> V).
        unsigned long long n1 = p.base1, n2 = p.base2;
        int vi = 0;
        for (int i = 0; i < p.nh; ++i) {
            const int half = p.h0 + i;
            const bool pass1 = (half & 1) == 0;
            const int step = half >> 1;
            if (pass1) {
                ++n1;
                if (!t1.in) continue;
                if (half == 0) {
                    for (int e = lane; e < KK; e += 32) sGv[e] = p.Gv0[e];
                } else {
                    if (lane == 0) blk_wait_ge<false>(p.vfold, n2 * (unsigned long long)p.panels2, p.err, p.timeout_ns);
                    __syncwarp();
                    for (int e = lane; e < KK; e += 32)
                        sGv[e] = sum_strided_cg(p.hist_Gvp + (size_t)(step - 1) * p.panels2 * KK + e, p.panels2, KK);
                }
                tail_bar();
                continue;
            }
            ++n2;
            const double* Vold = p.V[vi];
            vi ^= 1;
            if (!t2.in) continue;
            // U^T U: this rank's folded panel partials (complete once ufold reached this step's pass 1), then over ranks
            if (lane == 0) blk_wait_ge<false>(p.ufold, n1 * (unsigned long long)p.panels1, p.err, p.timeout_ns);
            __syncwarp();
            const unsigned long long xs = p.xbase + (n2 - p.base2);                 // this exchange's sequence number
            const size_t xpar = (size_t)(xs & 1ull) * kMaxPeers;
            if (p.nranks <= 1) {
                for (int e = lane; e < KK; e += 32) {
                    const double g = sum_strided_cg(p.Gu_part + e, p.panels1, KK);
                    sGu[e] = g;
                    if (b == 0) p.hist_Gu[(size_t)step * KK + e] = g;
                }
            } else {
                if (b == 0) {                      // CTA 0 pushes this rank's U^T U to every peer: it has the whole pass to arrive
                    const size_t slot = (xpar + p.rank) * p.xcount + (size_t)p.n * K;
                    for (int e = lane; e < KK; e += 32) {
                        const double g = sum_strided_cg(p.Gu_part + e, p.panels1, KK);
                        for (int r = 0; r < p.nranks; ++r) ll_store(p.xbuf[r] + slot + e, g, xs);
                    }
                }
                for (int e = lane; e < KK; e += 32) {
                    double g = 0.0;
                    for (int r = 0; r < p.nranks; ++r)
                        g += ll_wait(p.xbuf[p.rank] + (xpar + r) * p.xcount + (size_t)p.n * K + e, xs, p.err, p.timeout_ns);
                    sGu[e] = g;
                    if (b == 0) p.hist_Gu[(size_t)step * KK + e] = g;
                }
            }
            if (pre2) {
                // round 1: the old rows and the row map of every entry this lane owns, all loads in flight at once;
                // round 2: the few entries inside an active pathway (about 1 % of them) walk their packed CSR row
                constexpr int PER = (kBlkPre * K + 31) / 32;
                const int n_el = rows2 * K;
                const int64_t base = (t2.c0 + rb2) * K;
                double vo[PER];
                int32_t prs[PER];
#pragma unroll
                for (int q = 0; q < PER; ++q) {
                    const int e = lane + 32 * q;
                    const bool ok = e < n_el;
                    vo[q] = ok ? __ldcg(Vold + base + e) : 0.0;
                    prs[q] = ok ? __ldg(p.pos + base + e) : -1;
                }
#pragma unroll
                for (int q = 0; q < PER; ++q) {
                    const int e = lane + 32 * q;
                    if (e >= n_el) continue;
                    const int c = e % K;
                    double wv = 0.0, dg = -1.0;                                                  // dg < 0: not in the support
                    const int32_t pr = prs[q];
                    if (pr >= 0) { wv = pathway_term<true>(p.pw, p.active, pr, c, Vold, K); dg = p.pw.deg[pr]; }
                    pO[e] = vo[q];
                    pWv[e] = wv;
                    pDg[e] = dg;
                }
            }
            tail_bar();
        }
        return;
    }

    // ================================= consumer warps =================================
    const int t = threadIdx.x;                             // 0..255
    int s2 = 0;
    uint32_t phase = 0;
    unsigned long long n1 = p.base1, n2 = p.base2;
    int ui = 0, vi = 0;
    for (int i = 0; i < p.nh; ++i) {
        const int half = p.h0 + i;
        const bool pass1 = (half & 1) == 0;
        const int step = half >> 1;
        const BlkTile& tl = pass1 ? t1 : t2;
        const int panel_w = pass1 ? p.panel_w1 : p.panel_w2;
        const int chunks = pass1 ? p.chunks1 : p.chunks2;
        const int64_t cols = pass1 ? p.m : p.n;            // columns of M = rows of the matrix being updated
        double* OutPart = pass1 ? p.Apart : p.Bpart;
        if (pass1) ++n1; else ++n2;
        BLK_STAMP(i, 0);

        // ---- main loop: acc[g][c] += M[row][col g] * W[row][c] over the chunk's rows ----
        if (tl.in) {
            const int H = panel_w >> 2;
            const bool act = t < H && (2 * t) < tl.width;
            const bool act2 = t < H && (2 * (t + H)) < tl.width;
            const uint32_t x_stage_bytes = (uint32_t)kBlkRS * (uint32_t)panel_w * 8u;
            double acc[4][K];
#pragma unroll
            for (int g = 0; g < 4; ++g)
#pragma unroll
                for (int c = 0; c < K; ++c) acc[g][c] = 0.0;
            for (int it = 0; it < tl.iters; ++it) {
                const int rows = (int)min((int64_t)kBlkRS, tl.rend - (tl.rbeg + (int64_t)it * kBlkRS));
                mbar_wait(&full_bar[s2], phase);
                if (it == 0) BLK_STAMP(i, 1);
                const unsigned char* sx = smem_raw + (size_t)s2 * p.ring_stage_bytes;
                const double* sw = reinterpret_cast<const double*>(sx + x_stage_bytes);
                if (rows == kBlkRS) {
#pragma unroll
                    for (int r = 0; r < kBlkRS; ++r) {
                        const double2* xrow = reinterpret_cast<const double2*>(sx + (size_t)r * panel_w * 8);
                        const double2 xa = act ? xrow[t] : make_double2(0.0, 0.0);
                        const double2 xb = act2 ? xrow[t + H] : make_double2(0.0, 0.0);
                        // the W row as 128-bit broadcast reads (the ring stage stride is a run-time value, so the
                        // compiler cannot prove the 16-byte alignment of sw itself; K even => every row is aligned)
                        double wr[K];
                        if constexpr (K % 2 == 0) {
                            const double2* sw2 = reinterpret_cast<const double2*>(sw + r * K);
#pragma unroll
                            for (int c = 0; c < K / 2; ++c) { const double2 w2 = sw2[c]; wr[2 * c] = w2.x; wr[2 * c + 1] = w2.y; }
                        } else {
#pragma unroll
                            for (int c = 0; c < K; ++c) wr[c] = sw[r * K + c];
                        }
#pragma unroll
                        for (int c = 0; c < K; ++c) {
                            const double u = wr[c];
                            acc[0][c] = fma(xa.x, u, acc[0][c]);
                            acc[1][c] = fma(xa.y, u, acc[1][c]);
                            acc[2][c] = fma(xb.x, u, acc[2][c]);
                            acc[3][c] = fma(xb.y, u, acc[3][c]);
                        }
                    }
                } else {
                    for (int r = 0; r < rows; ++r) {
                        const double2* xrow = reinterpret_cast<const double2*>(sx + (size_t)r * panel_w * 8);
                        const double2 xa = act ? xrow[t] : make_double2(0.0, 0.0);
                        const double2 xb = act2 ? xrow[t + H] : make_double2(0.0, 0.0);
#pragma unroll
                        for (int c = 0; c < K; ++c) {
                            const double u = sw[r * K + c];
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
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const int64_t j = tl.c0 + 2 * (int64_t)(g < 2 ? t : t + H) + (g & 1);
                const bool ok = (g < 2 ? act : act2) && j < cols;
                if (ok) {
                    double* out = OutPart + ((int64_t)tl.chunk * cols + j) * K;
#pragma unroll
                    for (int c = 0; c < K; ++c) out[c] = acc[g][c];
                }
            }
        }
        BLK_STAMP(i, 2);

        // ---- tail: this CTA's share of the panel's rows ----
        // Element e = t + 256 q of a tile of <= kBlkRowsCap rows belongs to thread t (q < K): the pass partials and the old
        // rows are read as contiguous runs (fully used sectors), the sums stay in registers, the old rows go through shared
        // memory because an entry needs its whole row for the k x k contraction; the new rows replace them there for the Gram.
        if (pass1) {
            const double* Uold = p.U[ui];
            double* Unew = p.U[ui ^ 1];
            ui ^= 1;
            if (!tl.in) continue;
            const int rb = rb1, rows = rows1;
            // every CTA of the panel has stored its partials (release-add after the barrier: cumulative over the CTA's stores)
            cons_bar();
            if (t == 0) {
                red_release_add(p.arrive1 + tl.panel, 1ull);
                blk_wait_ge<false>(p.arrive1 + tl.panel, n1 * (unsigned long long)chunks, p.err, p.timeout_ns);
            }
            tail_bar();                                     // + the helper warp: sGv is ready
            BLK_STAMP(i, 3);
            BlkGram<K> gram;
            if (chunks <= 8) {
                // few chunks, large shares (1-2 GPUs): entry e = t + 256 q of a tile belongs to thread t (q < K); partials and old
                // rows are read as contiguous runs with every load of the thread in flight at once, the sums stay in registers
                for (int r0 = 0; r0 < rows; r0 += kBlkRowsCap) {
                    const int nr = min(kBlkRowsCap, rows - r0);
                    const int n_el = nr * K;
                    const int64_t base = (tl.c0 + rb + r0) * K;
                    double a[K];
    #pragma unroll
                    for (int q = 0; q < K; ++q) {
                        const int e = t + 256 * q;
                        a[q] = 0.0;
                        if (e < n_el) sR[e] = __ldcg(Uold + base + e);
                    }
    #pragma unroll 4
                    for (int ch = 0; ch < chunks; ++ch) {                                            // X.V (:420), chunk order
                        const double* src = p.Apart + (int64_t)ch * cols * K + base;
    #pragma unroll
                        for (int q = 0; q < K; ++q) {
                            const int e = t + 256 * q;
                            if (e < n_el) a[q] += __ldcg(src + e);
                        }
                    }
                    cons_bar();
                    double un[K];
    #pragma unroll
                    for (int q = 0; q < K; ++q) {
                        const int e = t + 256 * q;
                        un[q] = 0.0;
                        if (e < n_el) {
                            const int r = e / K, c = e - r * K;
                            const double* urow = sR + r * K;
                            double ugv = 0.0;
    #pragma unroll
                            for (int l = 0; l < K; ++l) ugv = fma(urow[l], sGv[l * K + c], ugv);
                            const double u = urow[c];
                            un[q] = u_update_value(u, a[q], ugv);
                            Unew[base + e] = un[q];
                        }
                    }
                    cons_bar();
                    // the share of U_new is stored: release the W rows of pass 2 (the Gram partial below is off that path)
                    if (r0 + kBlkRowsCap >= rows && t == 0) red_release_add(p.udone, 1ull);
    #pragma unroll
                    for (int q = 0; q < K; ++q) {
                        const int e = t + 256 * q;
                        if (e < n_el) sR[e] = un[q];
                    }
                    cons_bar();
                    gram.add(sR, nr);
                    cons_bar();
                }
            } else {
                // many chunks, small shares: sums staged 16 partials at a time (epi_stage_sums)
                for (int r0 = 0; r0 < rows; r0 += kBlkTile) {
                    const int nr = min(kBlkTile, rows - r0);
                    const int n_el = nr * K;
                    const int64_t base = (tl.c0 + rb + r0) * K;
                    for (int e = t; e < n_el; e += 256) sO[e] = __ldcg(Uold + base + e);
                    epi_stage_sums(sS, p.Apart + base, n_el, chunks, cols * K);                  // X.V   (:420)
                    cons_bar();
                    for (int e = t; e < n_el; e += 256) {
                        const int r = e / K, c = e - r * K;
                        const double* urow = sO + r * K;
                        double ugv = 0.0;
#pragma unroll
                        for (int l = 0; l < K; ++l) ugv = fma(urow[l], sGv[l * K + c], ugv);
                        const double u = urow[c];
                        const double un = u_update_value(u, sS[e], ugv);
                        sT[e] = un;
                        Unew[base + e] = un;
                    }
                    cons_bar();
                    if (r0 + kBlkTile >= rows && t == 0) red_release_add(p.udone, 1ull);
                    gram.add(sT, nr);
                    cons_bar();
                }
            }
            if (rows == 0 && t == 0) red_release_add(p.udone, 1ull);
            BLK_STAMP(i, 5);
            const int64_t me = (int64_t)tl.panel * chunks + tl.chunk;
            gram.finish(sBuf, p.part2 + me * KK);
            cons_bar();
            if (t == 0) {
                const unsigned long long prev = atom_acq_rel_add(p.done1 + tl.panel, 1ull);
                s_last = prev + 1ull == n1 * (unsigned long long)chunks;
            }
            cons_bar();
            if (s_last) {                                   // last CTA of the panel: fold the panel's Gram partials
                if (t < KK)
                    p.Gu_part[(int64_t)tl.panel * KK + t] = sum_strided_cg(p.part2 + (int64_t)tl.panel * chunks * KK + t, chunks, KK);
                cons_bar();
                if (t == 0) red_release_add(p.ufold, 1ull);
            }
            cons_bar();                                     // s_last / sR are rewritten by the next tail
            BLK_STAMP(i, 6);
        } else {
            const double* Vold = p.V[vi];
            double* Vnew = p.V[vi ^ 1];
            vi ^= 1;
            if (!tl.in) continue;
            const int rb = rb2, rows = rows2;
            const unsigned long long xs = p.xbase + (n2 - p.base2);                 // this exchange's sequence number
            const size_t xpar = (size_t)(xs & 1ull) * kMaxPeers;
            const double gamma = p.gd[0], delta = p.gd[1];
            cons_bar();
            if (t == 0) {
                red_release_add(p.arrive2 + tl.panel, 1ull);
                blk_wait_ge<false>(p.arrive2 + tl.panel, n2 * (unsigned long long)chunks, p.err, p.timeout_ns);
            }
            tail_bar();                                     // + the helper warp: sGu (and the prefetched operands) are ready
            BLK_STAMP(i, 3);
            BlkGram<K> gram;
            double vb = 0.0;
            const int tile = pre2 ? kBlkPre : kBlkTile;
            double* aT = pre2 ? pT : sT;
            double* aS = pre2 ? pS : sS;
            double* aO = pre2 ? pO : sO;
            for (int r0 = 0; r0 < rows; r0 += tile) {
                const int nr = min(tile, rows - r0);
                const int n_el = nr * K;
                const int64_t base = (tl.c0 + rb + r0) * K;
                if (!pre2)
                    for (int e = t; e < n_el; e += 256) aO[e] = __ldcg(Vold + base + e);
                epi_stage_sums(aS, p.Bpart + base, n_el, chunks, cols * K);                      // local X^T U  (:424)
                if (p.nranks > 1) {
                    // sum over ranks: every thread pushes the entries it owns into every rank's receive slot and then polls
                    // the same entries of all ranks in its own buffer, adding them in rank order (bitwise identical everywhere)
                    for (int e = t; e < n_el; e += 256) {
                        const double v = aS[e];
                        for (int r = 0; r < p.nranks; ++r) ll_store(p.xbuf[r] + (xpar + p.rank) * p.xcount + base + e, v, xs);
                    }
                    for (int e = t; e < n_el; e += 256)
                        aS[e] = ll_gather(p.xbuf[p.rank], xpar, p.xcount, p.nranks, (size_t)(base + e), xs, p.err, p.timeout_ns);
                    BLK_STAMP(i, 4);
                }
                cons_bar();
                for (int e = t; e < n_el; e += 256) {
                    const int r = e / K, c = e - r * K;
                    const int64_t j = tl.c0 + rb + r0 + r;
                    const double* vrow = aO + r * K;
                    const double bb = aS[e];
                    double cden = 0.0;
#pragma unroll
                    for (int l = 0; l < K; ++l) cden = fma(vrow[l], sGu[l * K + c], cden);      // V.Gu   (:425)
                    const double v = vrow[c];
                    int32_t pr = -1;
                    double wv = 0.0, dg = 0.0;
                    if (pre2) {
                        dg = pDg[e];
                        if (dg >= 0.0) { pr = p.pos[j * K + c]; wv = pWv[e]; }
                    } else {
                        pr = p.pos[j * K + c];
                        if (pr >= 0) {
                            // pathway_term<true>, written out: called here, it makes ptxas spill block_kernel<4> and <8>
                            const Pathways& pw = p.pw;
                            const int64_t pbase = pw.path_ptr[p.active[c]];
                            for (int64_t e2 = pw.row_ptr[pr]; e2 < pw.row_ptr[pr + 1]; ++e2)
                                wv = fma(pw.w[e2], __ldcg(Vold + (int64_t)pw.support_idx[pbase + pw.col_local[e2]] * K + c), wv);
                            dg = pw.deg[pr];
                        }
                    }
                    const double vn = v_update_value(v, bb, cden, pr >= 0, wv, dg, gamma, delta);
                    aT[e] = vn;
                    Vnew[j * K + c] = vn;
                    if (pr >= 0) p.hist_vh[(size_t)step * kVhCap + active_slot(p.doff, c, pr, p.pw.path_ptr[p.active[c]])] = vn;
                    vb = fma(vn, bb, vb);
                }
                cons_bar();
                // the share of V_new (and its active-set values) is stored: release the W rows of the next pass 1
                if (r0 + tile >= rows && t == 0) red_release_add(p.vdone, 1ull);
                gram.add(aT, nr);
                cons_bar();
            }
            if (rows == 0 && t == 0) red_release_add(p.vdone, 1ull);
            BLK_STAMP(i, 5);
            // sum(V_new * B) of this share: warp sums, then the 8 warp sums in order
            vb = warp_sum(vb);
            if ((t & 31) == 0) sW8[t >> 5] = vb;
            cons_bar();
            const int64_t me = (int64_t)tl.panel * chunks + tl.chunk;
            if (t == 0) {
                double s = 0.0;
#pragma unroll
                for (int w = 0; w < 8; ++w) s += sW8[w];
                p.vb2[me] = s;
            }
            gram.finish(sBuf, p.part2 + me * KK);
            cons_bar();
            if (t == 0) {
                const unsigned long long prev = atom_acq_rel_add(p.done2 + tl.panel, 1ull);
                s_last = prev + 1ull == n2 * (unsigned long long)chunks;
            }
            cons_bar();
            if (s_last) {
                if (t < KK)
                    p.hist_Gvp[((size_t)step * p.panels2 + tl.panel) * KK + t] =
                        sum_strided_cg(p.part2 + (int64_t)tl.panel * chunks * KK + t, chunks, KK);
                if (t == 128) p.hist_VBp[(size_t)step * p.panels2 + tl.panel] = sum_strided_cg(p.vb2 + (int64_t)tl.panel * chunks, chunks, 1);
                cons_bar();
                if (t == 0) red_release_add(p.vfold, 1ull);
            }
            cons_bar();
            BLK_STAMP(i, 6);
        }
    }
}

}  // namespace prmf
