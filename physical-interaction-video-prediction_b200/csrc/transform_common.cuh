// Device helpers shared by the fused transform kernels (fused_transform.cu) and the un-fused transformation lists
// (transform_unfused.cu): band staging of an image with its 2-pixel halo, the CDNA kernel normalisation and its backward.
#pragma once
#include "common.cuh"

namespace pivp {

constexpr float RELU_SHIFT = 1e-12f;       // train_model.py:42

// prev tile with a 2-pixel zero halo: tile[c][(R+4)][(W+4)], rows r0-2 .. r0+nrows+1
__device__ inline void load_prev_tile(const float* __restrict__ prev_sample, int H, int W, int r0, int nrows, float* tile) {
    // One warp per tile row (channel c, row ty), lanes walk the row: no per-element integer division (the flat i / (TH*TW), r / TW form
    // cost ~800 instructions per thread, more than the transform itself).  Every global load of the thread is issued into registers BEFORE
    // the first shared-memory store: a `smem[i] = __ldg(...)` loop issues in order, i.e. one full memory round trip per iteration.
    const int TW = W + 4, TH = nrows + 4;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    constexpr int RR = 5, JJ = 3;                        // rows per warp x 32-lane column groups held in registers
    if (TW <= 32 * JJ && 3 * TH <= RR * nw) {
        float v[RR][JJ];
#pragma unroll
        for (int rr = 0; rr < RR; ++rr) {
            const int row = warp + rr * nw;
            const int c = row / TH, ty = row - c * TH, y = r0 - 2 + ty;
            const bool ok = row < 3 * TH && y >= 0 && y < H;
            const float* src = prev_sample + (long)(c * H + y) * W - 2;
#pragma unroll
            for (int jj = 0; jj < JJ; ++jj) {
                const int tx = lane + 32 * jj;
                v[rr][jj] = (ok && tx >= 2 && tx < W + 2) ? __ldg(src + tx) : 0.f;
            }
        }
#pragma unroll
        for (int rr = 0; rr < RR; ++rr) {
            const int row = warp + rr * nw;
            if (row < 3 * TH) {
#pragma unroll
                for (int jj = 0; jj < JJ; ++jj) {
                    const int tx = lane + 32 * jj;
                    if (tx < TW) tile[row * TW + tx] = v[rr][jj];
                }
            }
        }
        return;
    }
    for (int row = warp; row < 3 * TH; row += nw) {
        const int c = row / TH, ty = row - c * TH;
        const int y = r0 - 2 + ty;
        const bool yin = y >= 0 && y < H;
        const float* src = prev_sample + (long)(c * H + y) * W - 2;
        float* dst = tile + row * TW;
        for (int tx = lane; tx < TW; tx += 32) dst[tx] = (yin && tx >= 2 && tx < W + 2) ? __ldg(src + tx) : 0.f;
    }
}

// normalised CDNA kernels of one sample: kn[m][25] = ktil / sum(ktil), ktil = relu(r - eps) + eps   (ref:326-329)
__device__ inline void cdna_normalise(const float* __restrict__ kraw_sample, int M, float* kn, float* ksum) {
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
        float s = 0.f, kt[25];
#pragma unroll
        for (int t = 0; t < 25; ++t) { kt[t] = fmaxf(kraw_sample[m * 25 + t] - RELU_SHIFT, 0.f) + RELU_SHIFT; s += kt[t]; }
#pragma unroll
        for (int t = 0; t < 25; ++t) kn[m * 25 + t] = kt[t] / s;
        if (ksum) ksum[m] = s;
    }
}

// Backward of the normalisation of ONE kernel (25 taps): d_kraw from dK = d(normalised kernel).
// dkt = (dK - sum_t K_t dK_t) / s ; d_r = dkt * [r - eps > 0]     (D.1)
__device__ __forceinline__ void cdna_kern_bwd_one(const float* kraw, const float* dK, float* d_kraw) {
    float kt[25], s = 0.f, dot = 0.f;
#pragma unroll
    for (int t = 0; t < 25; ++t) { kt[t] = fmaxf(kraw[t] - RELU_SHIFT, 0.f) + RELU_SHIFT; s += kt[t]; }
#pragma unroll
    for (int t = 0; t < 25; ++t) dot = fmaf(kt[t] / s, dK[t], dot);
#pragma unroll
    for (int t = 0; t < 25; ++t) d_kraw[t] = (kraw[t] - RELU_SHIFT > 0.f) ? (dK[t] - dot) / s : 0.f;
}

}  // namespace pivp
