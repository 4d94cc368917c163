// block_params.h -- launch parameters of the persistent step kernel (block.cuh), shared by the host orchestration
// (prmf_b200.cu) and the kernel's own translation unit (block.cu).
#pragma once

#include "kernels.cuh"

namespace prmf {

constexpr int kBlkRS = kTmaRS;       // rows of M per ring stage, as in the X-stream kernels
constexpr int kBlkRowsCap = 256;     // large shares (few chunks): rows per tile, K entries per thread, one staged array
constexpr int kBlkTile = 85;         // small shares (many chunks): rows per tile, three staged arrays share the same scratch
constexpr int kBlkPre = 51;          // largest pass-2 share the helper warp prefetches (five staged arrays share that scratch)
constexpr int kBlkThreads = 320;     // 8 consumer warps + the TMA producer warp + the helper warp


struct BlockParams {
    // X (m x n, leading dimension ldx) and its transposed copy (n x m, ldxt)
    const double* X;
    const double* Xt;
    int64_t ldx, ldxt, m, n;
    // pass 1: column panels over samples, row chunks over genes; pass 2: panels over genes, chunks over samples
    int panels1, panel_w1, chunks1;
    int panels2, panel_w2, chunks2;
    int64_t rpc1, rpc2;
    int stages;
    uint32_t ring_stage_bytes;       // max over the two passes of (RS * panel_w * 8 + W rows, 128-byte padded)
    // state: U[0] / V[0] are current at launch; every pass 1 flips U, every pass 2 flips V
    double* U[2];
    double* V[2];
    double* Apart;                   // [chunks1][m][K]
    double* Bpart;                   // [chunks2][n][K]
    double* Gu_part;                 // [panels1][K*K]   U_new^T U_new per sample panel (this rank's rows)
    double* part2;                   // scratch [tiles][K*K] per-CTA Gram partials
    double* vb2;                     // scratch [tiles]
    const double* Gv0;               // V^T V of the V at block start (for the U update of half 0)
    // monotone counters (never reset): arrive / done per panel, and the two grid-wide ones
    unsigned long long* arrive1;
    unsigned long long* done1;
    unsigned long long* arrive2;
    unsigned long long* done2;
    unsigned long long* udone;       // += 1 per CTA whose share of U_new is stored   (gates the W rows of pass 2)
    unsigned long long* vdone;       // += 1 per CTA whose share of V_new is stored   (gates the W rows of the next pass 1)
    unsigned long long* ufold;       // += 1 per sample panel whose Gram partials are folded (gates the V update's U^T U)
    unsigned long long* vfold;       // += 1 per gene panel whose Gram partials are folded   (gates the U update's V^T V)
    unsigned long long base1, base2; // pass-1 / pass-2 executions of this kernel on this handle before this launch
    unsigned int flags;              // developer switches (PRMF_BLOCK_FLAGS): 1 = no prefetch by the helper warp
    int h0, nh;                      // halves [h0, h0 + nh) of the block: even = pass 1, odd = pass 2; step = half / 2
    // V update
    Pathways pw;
    const int32_t* active;
    const int32_t* pos;
    const double* gd;
    // deferred objective: per-step slots
    double* hist_Gu;                 // [steps][K*K]
    double* hist_Gvp;                // [steps][panels2][K*K]
    double* hist_VBp;                // [steps][panels2]
    double* hist_vh;                 // [steps][kVhCap]
    const int64_t* doff;
    // bounded waits
    unsigned int* err;
    unsigned long long timeout_ns;
    // exchange over ranks (nranks <= 1: none)
    int nranks, rank;
    ulonglong2* xbuf[kMaxPeers];     // rank r's receive buffer: [parity 2][src rank kMaxPeers][xcount] LL entries (block.cuh)
    size_t xcount;                   // entries per (parity, src) slot: n*K + K*K, padded
    unsigned long long xbase;        // exchanges (= pass-2 executions of this kernel) before this launch
};

// sum over ranks of a few scalars through the peer buffers (no NCCL): [parity 2][source rank][kSmallAllreduceMax] entries
constexpr int kSmallAllreduceMax = 64;
struct PeerSmall {
    ulonglong2* slot[kMaxPeers];
    int nranks, rank;
    unsigned long long seq;
    unsigned int* err;
    unsigned long long timeout_ns;
};

}  // namespace prmf

// buf[0:count] <- sum over ranks, in rank order (count <= kSmallAllreduceMax); one small launch on `stream` (block.cu)
cudaError_t prmf_launch_small_allreduce(double* buf, int count, const prmf::PeerSmall& ps, cudaStream_t stream);
// Launches block_kernel<k> cooperatively (block.cu).  Returns cudaSuccess or the launch error.
cudaError_t prmf_launch_block_kernel(int k, const prmf::BlockParams& prm, int grid, size_t smem, cudaStream_t stream);
