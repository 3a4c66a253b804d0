// Fused transform + mask-softmax + composite kernels (the bandwidth-bound part of the path).
//
// Replaces, per time step, train_model.py:315-317,326-349 (CDNA) / :388-415 (DNA) / :454-471 (STP)
// together with the mask softmax and compositing :719-728.  Inputs are the NCHW planes written by the
// 1x1 deconvolutions and the kernel Linear; the output is gen_images[t] (boundary = SURVEY 8d).
//
// Quirks reproduced on purpose (SURVEY App. B): the softmax normalises groups of (M+1) FLAT-contiguous
// NCHW elements of a sample (B.1); the DNA taps are truncated at H/W and carry no gradient (B.2); the
// last CDNA kernel is never composited (B.3); all STP transformers share one theta (B.4).
//
// Tiling: one CTA per (sample, band of R image rows).  Phase 1 stages relu(mask logits) for the band plus
// the <= M elements of halo each softmax group needs, normalises the groups in shared memory; phase 2
// walks the band's pixels with the previous frame staged (+2 halo) in shared memory.
#include "transform_common.cuh"

namespace pivp {

constexpr int FT = 256;
constexpr int MAXM1 = 16;

struct Band {
    int H, W, M1;       // image size, masks+1
    int R;              // rows per band
    int L;              // shared row length for mu: R*W + 2*M1 (padded to odd)
};

// After the call mu[j*L + shift[j] + q] is the softmax mask of channel j at band pixel q (q = (row-r0)*W + col).
__device__ void band_softmax(const float* __restrict__ a_sample, const Band& bd, int r0, int nrows, float* mu, int* shift) {
    const int HW = bd.H * bd.W, M1 = bd.M1;
    const int p0 = r0 * bd.W, np = nrows * bd.W;
    for (int j = 0; j < M1; ++j) {
        const int f0 = j * HW + p0;                       // first flat element of the band in channel j
        const int fb = (f0 / M1) * M1;                    // start of its group
        const int fe = ((f0 + np - 1) / M1 + 1) * M1;     // one past the last group
        if (threadIdx.x == 0) shift[j] = f0 - fb;
        const int cnt = fe - fb, nt = blockDim.x;
        for (int i0 = threadIdx.x; i0 < cnt; i0 += 4 * nt) {       // four loads in flight per thread before the first store (see load_prev_tile)
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = (i0 + u * nt < cnt) ? __ldg(a_sample + fb + i0 + u * nt) : 0.f;
#pragma unroll
            for (int u = 0; u < 4; ++u) if (i0 + u * nt < cnt) mu[j * bd.L + i0 + u * nt] = fmaxf(v[u], 0.f);
        }
    }
    __syncthreads();
    for (int j = 0; j < M1; ++j) {
        const int f0 = j * HW + p0;
        const int ng = (f0 + np - 1) / M1 - f0 / M1 + 1;
        for (int g = threadIdx.x; g < ng; g += blockDim.x) {
            float* z = mu + j * bd.L + g * M1;
            float mx = z[0];
            for (int k = 1; k < M1; ++k) mx = fmaxf(mx, z[k]);
            float e[MAXM1], s = 0.f;
            for (int k = 0; k < M1; ++k) { e[k] = expf(z[k] - mx); s += e[k]; }
            const float inv = 1.f / s;
            for (int k = 0; k < M1; ++k) z[k] = e[k] * inv;
        }
    }
    __syncthreads();
}

// ====================================================================================== CDNA forward
__global__ void __launch_bounds__(FT) cdna_fwd_kernel(const float* __restrict__ prev, const float* __restrict__ e_pre,
                                                      const float* __restrict__ a_pre, const float* __restrict__ kraw,
                                                      float* __restrict__ out, Band bd, int M) {
    pdl_enter();
    extern __shared__ float sm[];
    __shared__ int shift[MAXM1];
    const int b = blockIdx.y, r0 = blockIdx.x * bd.R;
    const int nrows = min(bd.R, bd.H - r0), HW = bd.H * bd.W, W = bd.W;
    float* mu = sm;
    float* tile = mu + bd.M1 * bd.L;
    float* kn = tile + 3 * (bd.R + 4) * (W + 4);
    cdna_normalise(kraw + (long)b * M * 25, M, kn, nullptr);
    load_prev_tile(prev + (long)b * 3 * HW, bd.H, W, r0, nrows, tile);
    band_softmax(a_pre + (long)b * bd.M1 * HW, bd, r0, nrows, mu, shift);      // ends with __syncthreads()
    const int TW = W + 4, TS = (nrows + 4) * TW;
    for (int q = threadIdx.x; q < nrows * W; q += FT) {
        const int y = q / W, x = q - y * W;
        float keff[25];
#pragma unroll
        for (int t = 0; t < 25; ++t) keff[t] = 0.f;
        for (int m = 0; m < M - 1; ++m) {                                       // zip truncation: kernel M-1 unused (B.3)
            const float w = mu[(m + 2) * bd.L + shift[m + 2] + q];
#pragma unroll
            for (int t = 0; t < 25; ++t) keff[t] = fmaf(w, kn[m * 25 + t], keff[t]);
        }
        const float m0 = mu[shift[0] + q], m1 = mu[bd.L + shift[1] + q];
        const long gp = (long)b * 3 * HW + (r0 + y) * W + x;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float* tp = tile + c * TS + y * TW + x;                       // top-left of the 5x5 window
            float acc = 0.f;
#pragma unroll
            for (int u = 0; u < 5; ++u)
#pragma unroll
                for (int v = 0; v < 5; ++v) acc = fmaf(keff[u * 5 + v], tp[u * TW + v], acc);
            const float gpx = sigmoid_acc(fmaxf(__ldg(e_pre + gp + (long)c * HW), 0.f));
            out[gp + (long)c * HW] = m0 * tp[2 * TW + 2] + m1 * gpx + acc;
        }
    }
}

// ====================================================================================== CDNA backward, kernel 1
// Writes wq = mu * dmu (B,M1,H,W), d_e_pre; accumulates dK (B,M,25) with atomics (dK must be zeroed by the caller).
__global__ void __launch_bounds__(FT) cdna_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ prev,
                                                      const float* __restrict__ e_pre, const float* __restrict__ a_pre,
                                                      const float* __restrict__ kraw, float* __restrict__ wq, float* __restrict__ d_e,
                                                      float* __restrict__ dK, Band bd, int M) {
    pdl_enter();
    extern __shared__ float sm[];
    __shared__ int shift[MAXM1];
    const int b = blockIdx.y, r0 = blockIdx.x * bd.R;
    const int nrows = min(bd.R, bd.H - r0), HW = bd.H * bd.W, W = bd.W, PB = bd.R * W;
    float* mu = sm;
    float* tile = mu + bd.M1 * bd.L;
    float* kn = tile + 3 * (bd.R + 4) * (W + 4);
    float* Qs = kn + M * 25;                                                    // [25][PB]
    cdna_normalise(kraw + (long)b * M * 25, M, kn, nullptr);
    load_prev_tile(prev + (long)b * 3 * HW, bd.H, W, r0, nrows, tile);
    band_softmax(a_pre + (long)b * bd.M1 * HW, bd, r0, nrows, mu, shift);
    const int TW = W + 4, TS = (nrows + 4) * TW, np = nrows * W;
    for (int q = threadIdx.x; q < np; q += FT) {
        const int y = q / W, x = q - y * W;
        const long gp = (long)b * 3 * HW + (r0 + y) * W + x;
        float g[3], Q[25];
#pragma unroll
        for (int c = 0; c < 3; ++c) g[c] = __ldg(gout + gp + (long)c * HW);
#pragma unroll
        for (int t = 0; t < 25; ++t) Q[t] = 0.f;
        float dmu0 = 0.f, dmu1 = 0.f;
        const float m1 = mu[bd.L + shift[1] + q];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float* tp = tile + c * TS + y * TW + x;
#pragma unroll
            for (int u = 0; u < 5; ++u)
#pragma unroll
                for (int v = 0; v < 5; ++v) Q[u * 5 + v] = fmaf(g[c], tp[u * TW + v], Q[u * 5 + v]);
            dmu0 = fmaf(g[c], tp[2 * TW + 2], dmu0);
            const float ev = __ldg(e_pre + gp + (long)c * HW);
            const float gpx = sigmoid_acc(fmaxf(ev, 0.f));
            dmu1 = fmaf(g[c], gpx, dmu1);
            d_e[gp + (long)c * HW] = ev > 0.f ? m1 * g[c] * gpx * (1.f - gpx) : 0.f;
        }
#pragma unroll
        for (int t = 0; t < 25; ++t) Qs[t * PB + q] = Q[t];
        const long wp = (long)b * bd.M1 * HW + (r0 + y) * W + x;
        wq[wp] = mu[shift[0] + q] * dmu0;
        wq[wp + HW] = m1 * dmu1;
        for (int m = 0; m < M - 1; ++m) {
            float d = 0.f;
#pragma unroll
            for (int t = 0; t < 25; ++t) d = fmaf(kn[m * 25 + t], Q[t], d);
            wq[wp + (long)(m + 2) * HW] = mu[(m + 2) * bd.L + shift[m + 2] + q] * d;
        }
    }
    __syncthreads();
    // dK[m][tap] += sum_q mu_{m+2}(q) * Q[tap](q)
    for (int id = threadIdx.x; id < (M - 1) * 25; id += FT) {
        const int m = id / 25, t = id - m * 25;
        const float* mrow = mu + (m + 2) * bd.L + shift[m + 2];
        const float* qrow = Qs + t * PB;
        float acc = 0.f;
        const int lane = threadIdx.x & 31;
        for (int i = 0; i < np; ++i) {
            const int q = (i + lane) % np;
            acc = fmaf(mrow[q], qrow[q], acc);
        }
        atomicAdd(dK + ((long)b * M + m) * 25 + t, acc);
    }
}

// dprev (only when the previous frame carries gradient: feedself mode, ref:664-666):
// dP_c(p) (+)= mu0(p) g_c(p) + sum_tap Keff_s[tap] g_c(s),  s = p - (tap - centre)
__global__ void __launch_bounds__(FT) cdna_dprev_kernel(const float* __restrict__ gout, const float* __restrict__ a_pre,
                                                        const float* __restrict__ kraw, float* __restrict__ dprev, Band bd, int M,
                                                        int accumulate) {
    pdl_enter();
    extern __shared__ float sm[];
    __shared__ int shift[MAXM1];
    const int b = blockIdx.y, r0 = blockIdx.x * bd.R;
    const int nrows = min(bd.R, bd.H - r0), HW = bd.H * bd.W, W = bd.W;
    // extended band: rows [e0, e1) = [r0-2, r0+nrows+2) clipped to the image
    const int e0 = max(0, r0 - 2), e1 = min(bd.H, r0 + nrows + 2), erows = e1 - e0;
    float* mu = sm;                                                             // bd.L sized for R+4 rows by the host
    float* tile = mu + bd.M1 * bd.L;                                            // g tile [3][erows+4][W+4] anchored at e0-2
    float* kn = tile + 3 * (bd.R + 8) * (W + 4);
    cdna_normalise(kraw + (long)b * M * 25, M, kn, nullptr);
    load_prev_tile(gout + (long)b * 3 * HW, bd.H, W, e0, erows, tile);
    band_softmax(a_pre + (long)b * bd.M1 * HW, bd, e0, erows, mu, shift);
    const int TW = W + 4, TS = (erows + 4) * TW;
    for (int q = threadIdx.x; q < nrows * W; q += FT) {
        const int y = q / W, x = q - y * W, yi = r0 + y;
        float acc[3] = {0.f, 0.f, 0.f};
        for (int u = 0; u < 5; ++u) {
            const int sy = yi - u + 2;
            if (sy < 0 || sy >= bd.H) continue;
            for (int v = 0; v < 5; ++v) {
                const int sx = x - v + 2;
                if (sx < 0 || sx >= W) continue;
                const int sq = (sy - e0) * W + sx;
                float ke = 0.f;
                for (int m = 0; m < M - 1; ++m) ke = fmaf(mu[(m + 2) * bd.L + shift[m + 2] + sq], kn[m * 25 + u * 5 + v], ke);
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[c] = fmaf(ke, tile[c * TS + (sy - e0 + 2) * TW + sx + 2], acc[c]);
            }
        }
        const float m0 = mu[shift[0] + (yi - e0) * W + x];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float v = acc[c] + m0 * tile[c * TS + (yi - e0 + 2) * TW + x + 2];
            float* d = dprev + (long)b * 3 * HW + (long)c * HW + yi * W + x;
            *d = accumulate ? (*d + v) : v;
        }
    }
}

// ====================================================================================== softmax backward (shared by all three)
// thread per flat group: d_a = (wq - mu * sum(wq)) * [a > 0]
__global__ void mask_softmax_bwd_kernel(const float* __restrict__ a_pre, const float* __restrict__ wq, float* __restrict__ d_a,
                                        long ngroups, int M1) {
    pdl_enter();
    const long gidx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gidx >= ngroups) return;
    const float* a = a_pre + gidx * M1;
    const float* w = wq + gidx * M1;
    float z[MAXM1], mx = 0.f, S = 0.f;
    for (int k = 0; k < M1; ++k) { z[k] = fmaxf(a[k], 0.f); mx = fmaxf(mx, z[k]); S += w[k]; }
    float s = 0.f;
    for (int k = 0; k < M1; ++k) { z[k] = expf(z[k] - mx); s += z[k]; }
    const float inv = 1.f / s;
    for (int k = 0; k < M1; ++k) d_a[gidx * M1 + k] = a[k] > 0.f ? (w[k] - z[k] * inv * S) : 0.f;
}

// d_kraw from dK: dkt = (dK - sum_t K_t dK_t) / s ; d_r = dkt * [r - eps > 0]     (D.1)
__global__ void cdna_kern_bwd_kernel(const float* __restrict__ kraw, const float* __restrict__ dK, float* __restrict__ d_kraw, int BM_) {
    pdl_enter();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;       // over B*M kernels
    if (i >= BM_) return;
    cdna_kern_bwd_one(kraw + i * 25, dK + i * 25, d_kraw + i * 25);
}

// ====================================================================================== DNA
// tap (xk,yk) of pixel (i,j) reads prev[i+xk-2][j+yk-2] iff i+xk < H and j+yk < W (and inside the image) -- B.2
// BWD and the image width are compile-time (WC = 0: run-time width): the forward instantiation carries none of the gradient arithmetic and the
// pixel index splits into (row, column) with shifts.
template <bool BWD, int WC>
__global__ void __launch_bounds__(FT) dna_kernel(const float* __restrict__ prev, const float* __restrict__ e_pre,
                                                 const float* __restrict__ a_pre, const float* __restrict__ gout,
                                                 float* __restrict__ out, float* __restrict__ wq, float* __restrict__ d_e,
                                                 float* __restrict__ dprev, int dprev_acc, Band bd) {
    pdl_enter();
    constexpr bool backward = BWD;
    extern __shared__ float sm[];
    __shared__ int shift[MAXM1];
    const int W = WC ? WC : bd.W;
    const int b = blockIdx.y, r0 = blockIdx.x * bd.R;
    const int nrows = min(bd.R, bd.H - r0), HW = bd.H * W, H = bd.H;
    float* mu = sm;
    float* tile = mu + bd.M1 * bd.L;
    // the 25 kernel logits of this thread's first pixel are requested BEFORE the two shared-memory staging phases (each of which is a
    // global round trip followed by a barrier): three dependent memory latencies become one
    float kpre[25];
    if ((int)threadIdx.x < nrows * W) {
        const int y = threadIdx.x / W, x = threadIdx.x - y * W;
        const float* src = e_pre + (long)b * 25 * HW + (r0 + y) * W + x;
#pragma unroll
        for (int t = 0; t < 25; ++t) kpre[t] = __ldg(src + (long)t * HW);
    }
    load_prev_tile(prev + (long)b * 3 * HW, H, W, r0, nrows, tile);
    band_softmax(a_pre + (long)b * 2 * HW, bd, r0, nrows, mu, shift);
    const int TW = W + 4, TS = (nrows + 4) * TW;
    for (int q = threadIdx.x; q < nrows * W; q += FT) {
        const int y = q / W, x = q - y * W, yi = r0 + y;
        const long ep = (long)b * 25 * HW + yi * W + x;
        float k[25], s = 0.f;
#pragma unroll
        for (int t = 0; t < 25; ++t) {
            const float raw = (q == (int)threadIdx.x) ? kpre[t] : __ldg(e_pre + ep + (long)t * HW);
            k[t] = fmaxf(raw - RELU_SHIFT, 0.f) + RELU_SHIFT; s += k[t];
        }
        const float inv = 1.f / s;
        const float m0 = mu[shift[0] + q], m1 = mu[bd.L + shift[1] + q];
        const long gp = (long)b * 3 * HW + yi * W + x;
        float T[3] = {0.f, 0.f, 0.f};
        float g[3] = {0.f, 0.f, 0.f};
        float dKt[BWD ? 25 : 1];
        if (backward) {
#pragma unroll
            for (int c = 0; c < 3; ++c) g[c] = __ldg(gout + gp + (long)c * HW);
        }
        // The window is truncated at i + xkern >= H / j + ykern >= W (B.2): only pixels of the last four rows / columns lose taps, so the
        // interior runs the 75 multiply-adds without a predicate per tap; T is normalised once at the end instead of per tap.
        const float* trow = tile + y * TW + x;
        if (yi + 4 < H && x + 4 < W) {
#pragma unroll
            for (int u = 0; u < 5; ++u)
#pragma unroll
                for (int v = 0; v < 5; ++v) {
                    float dk = 0.f;
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        const float pv = trow[c * TS + u * TW + v];
                        T[c] = fmaf(k[u * 5 + v], pv, T[c]);
                        if (BWD) dk = fmaf(g[c], pv, dk);
                    }
                    if (BWD) dKt[u * 5 + v] = dk * m1;
                }
        } else {
#pragma unroll
            for (int u = 0; u < 5; ++u)
#pragma unroll
                for (int v = 0; v < 5; ++v) {
                    const bool live = (yi + u < H) && (x + v < W);
                    float dk = 0.f;
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        const float pv = live ? trow[c * TS + u * TW + v] : 0.f;
                        T[c] = fmaf(k[u * 5 + v], pv, T[c]);
                        if (BWD) dk = fmaf(g[c], pv, dk);
                    }
                    if (BWD) dKt[u * 5 + v] = dk * m1;
                }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) T[c] *= inv;
        if (!backward) {
#pragma unroll
            for (int c = 0; c < 3; ++c) out[gp + (long)c * HW] = m0 * tile[c * TS + (y + 2) * TW + x + 2] + m1 * T[c];
        } else {
            float dmu0 = 0.f, dmu1 = 0.f, dot = 0.f;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float pc = tile[c * TS + (y + 2) * TW + x + 2];
                dmu0 = fmaf(g[c], pc, dmu0);
                dmu1 = fmaf(g[c], T[c], dmu1);
                if (dprev) {
                    float* d = dprev + gp + (long)c * HW;
                    *d = dprev_acc ? (*d + m0 * g[c]) : m0 * g[c];
                }
            }
#pragma unroll
            for (int t = 0; t < 25; ++t) dot = fmaf(k[t] * inv, dKt[BWD ? t : 0], dot);
#pragma unroll
            for (int t = 0; t < 25; ++t)               // k[t] > eps  <=>  the ReLU of ref:408 let the logit through
                d_e[ep + (long)t * HW] = (k[t] > RELU_SHIFT) ? (dKt[BWD ? t : 0] - dot) * inv : 0.f;
            const long wp = (long)b * 2 * HW + yi * W + x;
            wq[wp] = m0 * dmu0;
            wq[wp + HW] = m1 * dmu1;
        }
    }
}

// ====================================================================================== STP
// theta = theta_raw + identity (ref:462-468); grid A.7; bilinear sampler with "zeros" (oob=0) or "border" (oob=1) rule.
__global__ void __launch_bounds__(FT) stp_kernel(const float* __restrict__ prev, const float* __restrict__ e_pre,
                                                 const float* __restrict__ a_pre, const float* __restrict__ theta_raw,
                                                 const float* __restrict__ gout, float* __restrict__ out, float* __restrict__ wq,
                                                 float* __restrict__ d_e, float* __restrict__ d_theta, float* __restrict__ dprev,
                                                 Band bd, int M, int oob, int backward) {
    pdl_enter();
    extern __shared__ float sm[];
    __shared__ int shift[MAXM1];
    __shared__ float red[32];
    const int b = blockIdx.y, r0 = blockIdx.x * bd.R;
    const int nrows = min(bd.R, bd.H - r0), HW = bd.H * bd.W, W = bd.W, H = bd.H;
    float* mu = sm;
    band_softmax(a_pre + (long)b * bd.M1 * HW, bd, r0, nrows, mu, shift);
    float th[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) th[i] = __ldg(theta_raw + b * 6 + i) + ((i == 0 || i == 4) ? 1.f : 0.f);
    const float* P = prev + (long)b * 3 * HW;
    const float sx = (W > 1) ? 2.f / (float)(W - 1) : 0.f, sy = (H > 1) ? 2.f / (float)(H - 1) : 0.f;
    const float hw = 0.5f * (float)(W - 1), hh = 0.5f * (float)(H - 1);
    float dth[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const int np = nrows * W;
    for (int q0 = 0; q0 < np; q0 += FT) {
        const int q = q0 + threadIdx.x;
        if (q < np) {
            const int y = q / W, x = q - y * W, yi = r0 + y;
            const float xn = -1.f + sx * (float)x, yn = -1.f + sy * (float)yi;
            float u = (th[0] * xn + th[1] * yn + th[2] + 1.f) * hw;
            float v = (th[3] * xn + th[4] * yn + th[5] + 1.f) * hh;
            bool live_u = true, live_v = true;
            if (oob == 1) {
                live_u = (u >= 0.f) && (u <= (float)(W - 1));
                live_v = (v >= 0.f) && (v <= (float)(H - 1));
                u = fminf(fmaxf(u, 0.f), (float)(W - 1));
                v = fminf(fmaxf(v, 0.f), (float)(H - 1));
            }
            // keep the integer conversion safe for wildly out-of-range coordinates
            const float uc = fminf(fmaxf(u, -2.f), (float)W + 1.f), vc = fminf(fmaxf(v, -2.f), (float)H + 1.f);
            const float fu0 = floorf(uc), fv0 = floorf(vc);
            const int u0 = (int)fu0, v0 = (int)fv0;
            const float fu = uc - fu0, fv = vc - fv0;
            const bool inside = (u == uc) && (v == vc);                  // clamped => every corner is outside anyway
            const bool ok00 = inside && v0 >= 0 && v0 < H && u0 >= 0 && u0 < W;
            const bool ok01 = inside && v0 >= 0 && v0 < H && u0 + 1 >= 0 && u0 + 1 < W;
            const bool ok10 = inside && v0 + 1 >= 0 && v0 + 1 < H && u0 >= 0 && u0 < W;
            const bool ok11 = inside && v0 + 1 >= 0 && v0 + 1 < H && u0 + 1 >= 0 && u0 + 1 < W;
            const float w00 = (1.f - fv) * (1.f - fu), w01 = (1.f - fv) * fu, w10 = fv * (1.f - fu), w11 = fv * fu;
            float msum = 0.f;
            for (int m = 2; m < bd.M1; ++m) msum += mu[m * bd.L + shift[m] + q];
            const float m0 = mu[shift[0] + q], m1 = mu[bd.L + shift[1] + q];
            const long gp = (long)b * 3 * HW + yi * W + x;
            float dmu0 = 0.f, dmu1 = 0.f, dmus = 0.f, gu = 0.f, gv = 0.f;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float* Pc = P + (long)c * HW;
                const float p00 = ok00 ? __ldg(Pc + v0 * W + u0) : 0.f;
                const float p01 = ok01 ? __ldg(Pc + v0 * W + u0 + 1) : 0.f;
                const float p10 = ok10 ? __ldg(Pc + (v0 + 1) * W + u0) : 0.f;
                const float p11 = ok11 ? __ldg(Pc + (v0 + 1) * W + u0 + 1) : 0.f;
                const float S = p00 * w00 + p01 * w01 + p10 * w10 + p11 * w11;
                const float ev = __ldg(e_pre + gp + (long)c * HW);
                const float sg = sigmoid_acc(ev);
                const float pc = __ldg(Pc + yi * W + x);
                if (!backward) {
                    out[gp + (long)c * HW] = m0 * pc + m1 * sg + msum * S;
                } else {
                    const float g = __ldg(gout + gp + (long)c * HW);
                    dmu0 = fmaf(g, pc, dmu0);
                    dmu1 = fmaf(g, sg, dmu1);
                    dmus = fmaf(g, S, dmus);
                    d_e[gp + (long)c * HW] = m1 * g * sg * (1.f - sg);
                    const float dS = msum * g;
                    gu = fmaf(dS, (p01 - p00) * (1.f - fv) + (p11 - p10) * fv, gu);
                    gv = fmaf(dS, (p10 - p00) * (1.f - fu) + (p11 - p01) * fu, gv);
                    if (dprev) {
                        float* D = dprev + (long)b * 3 * HW + (long)c * HW;
                        atomicAdd(D + yi * W + x, m0 * g);
                        if (ok00) atomicAdd(D + v0 * W + u0, dS * w00);
                        if (ok01) atomicAdd(D + v0 * W + u0 + 1, dS * w01);
                        if (ok10) atomicAdd(D + (v0 + 1) * W + u0, dS * w10);
                        if (ok11) atomicAdd(D + (v0 + 1) * W + u0 + 1, dS * w11);
                    }
                }
            }
            if (backward) {
                const long wp = (long)b * bd.M1 * HW + yi * W + x;
                wq[wp] = m0 * dmu0;
                wq[wp + HW] = m1 * dmu1;
                for (int m = 2; m < bd.M1; ++m) wq[wp + (long)m * HW] = mu[m * bd.L + shift[m] + q] * dmus;
                gu *= (live_u ? hw : 0.f);
                gv *= (live_v ? hh : 0.f);
                dth[0] += gu * xn; dth[1] += gu * yn; dth[2] += gu;
                dth[3] += gv * xn; dth[4] += gv * yn; dth[5] += gv;
            }
        }
    }
    if (backward) {
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const float s = block_sum(dth[i], red);
            if (threadIdx.x == 0) atomicAdd(d_theta + b * 6 + i, s);
        }
    }
}

static int make_band(int H, int W, int M1, int extra_rows, Band* bd, int band_pixels = 512) {
    PIVP_REQUIRE(H > 0 && W > 0 && M1 >= 2 && M1 <= MAXM1, "fused transform: bad geometry (need 2 <= masks+1 <= 16)");
    int R = band_pixels / W;
    if (R < 1) R = 1;
    if (R > H) R = H;
    bd->H = H; bd->W = W; bd->M1 = M1; bd->R = R;
    bd->L = ((R + extra_rows) * W + 2 * M1) | 1;
    return PIVP_OK;
}

// Raises the dynamic shared-memory limit of `kernel` once per (kernel type, size) so that steady-state calls -- and CUDA-graph
// capture -- issue no attribute call.  Every kernel in this file has a distinct signature, hence a distinct instantiation.
template <typename K>
static int allow_smem(K kernel, size_t bytes) {
    static PerDeviceOnce granted;              // per device and per kernel instantiation
    if (bytes > 48 * 1024 && granted.need(bytes)) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(smem=%zu): %s", bytes, cudaGetErrorString(e)); return PIVP_ECUDA; }
    }
    return PIVP_OK;
}

// fast path for the BASELINE geometry (cdna_band.cu)
bool cdna_band_supported(int H, int W, int num_masks, const void* p0, const void* p1, const void* p2, const void* p3);
int cdna_band_fwd(const float* prev, const float* e_pre, const float* a_pre, const float* kraw, float* out, int B, int H, cudaStream_t st);
size_t cdna_band_bwd_workspace_floats(int B, int H);
int cdna_band_bwd(const float* gout, const float* prev, const float* e_pre, const float* a_pre, const float* kraw, float* d_e,
                  float* d_a, float* d_kraw, float* dKp, int B, int H, cudaStream_t st);

}  // namespace pivp

using namespace pivp;

extern "C" {

int pivp_cdna_fused_fwd(const float* prev, const float* enc7_pre, const float* mask_pre, const float* kern_raw, float* out,
                        int B, int H, int W, int num_masks, void* stream) {
    PIVP_REQUIRE(prev && enc7_pre && mask_pre && kern_raw && out && B > 0 && num_masks >= 1, "cdna_fused_fwd: bad argument");
    if (cdna_band_supported(H, W, num_masks, prev, enc7_pre, mask_pre, out) && cdna_band_supported(H, W, num_masks, kern_raw, out, out, out))
        return cdna_band_fwd(prev, enc7_pre, mask_pre, kern_raw, out, B, H, (cudaStream_t)stream);
    Band bd;
    if (int e = make_band(H, W, num_masks + 1, 0, &bd)) return e;
    const size_t smem = sizeof(float) * ((size_t)bd.M1 * bd.L + 3 * (bd.R + 4) * (W + 4) + num_masks * 25);
    if (int e = allow_smem(cdna_fwd_kernel, smem)) return e;
    launch_k(cdna_fwd_kernel, dim3((H + bd.R - 1) / bd.R, B), dim3(FT), smem, (cudaStream_t)stream, prev, enc7_pre, mask_pre, kern_raw, out, bd, num_masks);
    return check_launch("cdna_fused_fwd");
}

size_t pivp_cdna_fused_bwd_workspace_bytes(int B, int H, int W, int num_masks) {
    // wq planes (B,M+1,H,W) + dK (B,M,25)
    return sizeof(float) * ((size_t)B * (num_masks + 1) * H * W + (size_t)B * num_masks * 25);
}

int pivp_cdna_fused_bwd(const float* g_out, const float* prev, const float* enc7_pre, const float* mask_pre, const float* kern_raw,
                        float* d_enc7_pre, float* d_mask_pre, float* d_kern_raw, float* d_prev, int accumulate_dprev,
                        int B, int H, int W, int num_masks, void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(g_out && prev && enc7_pre && mask_pre && kern_raw && d_enc7_pre && d_mask_pre && d_kern_raw && workspace,
                 "cdna_fused_bwd: null pointer");
    PIVP_REQUIRE(ws_bytes >= pivp_cdna_fused_bwd_workspace_bytes(B, H, W, num_masks), "cdna_fused_bwd: workspace too small");
    Band bd;
    if (int e = make_band(H, W, num_masks + 1, 0, &bd)) return e;
    cudaStream_t st = (cudaStream_t)stream;
    if (cdna_band_supported(H, W, num_masks, prev, enc7_pre, mask_pre, g_out) &&
        cdna_band_supported(H, W, num_masks, d_enc7_pre, d_mask_pre, workspace, workspace)) {
        // one pass: every input read once, every output written once; workspace holds the per-band kernel-gradient partials
        if (int e = cdna_band_bwd(g_out, prev, enc7_pre, mask_pre, kern_raw, d_enc7_pre, d_mask_pre, d_kern_raw, (float*)workspace, B, H, st))
            return e;
        if (d_prev) {
            Band be;
            if (int e = make_band(H, W, num_masks + 1, 4, &be)) return e;
            const size_t sm2 = sizeof(float) * ((size_t)be.M1 * be.L + 3 * (be.R + 8) * (W + 4) + num_masks * 25);
            if (int e = allow_smem(cdna_dprev_kernel, sm2)) return e;
            launch_k(cdna_dprev_kernel, dim3((H + be.R - 1) / be.R, B), dim3(FT), sm2, st, g_out, mask_pre, kern_raw, d_prev, be, num_masks, accumulate_dprev);
            return check_launch("cdna_fused_bwd(dprev)");
        }
        return PIVP_OK;
    }
    float* wq = (float*)workspace;
    float* dK = wq + (size_t)B * (num_masks + 1) * H * W;
    cudaMemsetAsync(dK, 0, sizeof(float) * (size_t)B * num_masks * 25, st);
    const size_t smem = sizeof(float) * ((size_t)bd.M1 * bd.L + 3 * (bd.R + 4) * (W + 4) + num_masks * 25 + 25 * (size_t)bd.R * W);
    if (int e = allow_smem(cdna_bwd_kernel, smem)) return e;
    launch_k(cdna_bwd_kernel, dim3((H + bd.R - 1) / bd.R, B), dim3(FT), smem, st, g_out, prev, enc7_pre, mask_pre, kern_raw, wq, d_enc7_pre, dK, bd, num_masks);
    if (int e = check_launch("cdna_fused_bwd(k1)")) return e;
    const long ngroups = (long)B * H * W;
    launch_k(mask_softmax_bwd_kernel, dim3((unsigned)((ngroups + 255) / 256)), dim3(256), 0, st, mask_pre, wq, d_mask_pre, ngroups, num_masks + 1);
    if (int e = check_launch("cdna_fused_bwd(softmax)")) return e;
    launch_k(cdna_kern_bwd_kernel, dim3((B * num_masks + 127) / 128), dim3(128), 0, st, kern_raw, dK, d_kern_raw, B * num_masks);
    if (int e = check_launch("cdna_fused_bwd(kern)")) return e;
    if (d_prev) {
        Band be;
        if (int e = make_band(H, W, num_masks + 1, 4, &be)) return e;
        const size_t sm2 = sizeof(float) * ((size_t)be.M1 * be.L + 3 * (be.R + 8) * (W + 4) + num_masks * 25);
        if (int e = allow_smem(cdna_dprev_kernel, sm2)) return e;
        launch_k(cdna_dprev_kernel, dim3((H + be.R - 1) / be.R, B), dim3(FT), sm2, st, g_out, mask_pre, kern_raw, d_prev, be, num_masks, accumulate_dprev);
        return check_launch("cdna_fused_bwd(dprev)");
    }
    return PIVP_OK;
}

int pivp_dna_fused_fwd(const float* prev, const float* enc7_pre, const float* mask_pre, float* out, int B, int H, int W, void* stream) {
    PIVP_REQUIRE(prev && enc7_pre && mask_pre && out && B > 0, "dna_fused_fwd: bad argument");
    Band bd;
    if (int e = make_band(H, W, 2, 0, &bd)) return e;              // (measured: 256-pixel bands -- one pixel per thread, twice the CTAs -- are 1.7x slower:
                                                                   //  the per-band staging, not the pixel loop, is what a CTA waits for)
    const size_t smem = sizeof(float) * ((size_t)2 * bd.L + 3 * (bd.R + 4) * (W + 4));
    PIVP_REQUIRE(smem <= 48 * 1024, "dna_fused_fwd: image too wide for the band staging");
    if (W == 64) launch_k(dna_kernel<false, 64>, dim3((H + bd.R - 1) / bd.R, B), dim3(FT), smem, (cudaStream_t)stream, prev, enc7_pre, mask_pre, nullptr, out,
                          nullptr, nullptr, nullptr, 0, bd);
    else launch_k(dna_kernel<false, 0>, dim3((H + bd.R - 1) / bd.R, B), dim3(FT), smem, (cudaStream_t)stream, prev, enc7_pre, mask_pre, nullptr, out,
                  nullptr, nullptr, nullptr, 0, bd);
    return check_launch("dna_fused_fwd");
}

size_t pivp_dna_fused_bwd_workspace_bytes(int B, int H, int W) { return sizeof(float) * (size_t)B * 2 * H * W; }

int pivp_dna_fused_bwd(const float* g_out, const float* prev, const float* enc7_pre, const float* mask_pre,
                       float* d_enc7_pre, float* d_mask_pre, float* d_prev, int accumulate_dprev,
                       int B, int H, int W, void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(g_out && prev && enc7_pre && mask_pre && d_enc7_pre && d_mask_pre && workspace, "dna_fused_bwd: null pointer");
    PIVP_REQUIRE(ws_bytes >= pivp_dna_fused_bwd_workspace_bytes(B, H, W), "dna_fused_bwd: workspace too small");
    Band bd;
    if (int e = make_band(H, W, 2, 0, &bd)) return e;
    cudaStream_t st = (cudaStream_t)stream;
    float* wq = (float*)workspace;
    const size_t smem = sizeof(float) * ((size_t)2 * bd.L + 3 * (bd.R + 4) * (W + 4));
    PIVP_REQUIRE(smem <= 48 * 1024, "dna_fused_bwd: image too wide for the band staging");
    if (W == 64) launch_k(dna_kernel<true, 64>, dim3((H + bd.R - 1) / bd.R, B), dim3(FT), smem, st, prev, enc7_pre, mask_pre, g_out, nullptr, wq, d_enc7_pre,
                          d_prev, accumulate_dprev, bd);
    else launch_k(dna_kernel<true, 0>, dim3((H + bd.R - 1) / bd.R, B), dim3(FT), smem, st, prev, enc7_pre, mask_pre, g_out, nullptr, wq, d_enc7_pre,
                  d_prev, accumulate_dprev, bd);
    if (int e = check_launch("dna_fused_bwd(k1)")) return e;
    const long ngroups = (long)B * H * W;
    launch_k(mask_softmax_bwd_kernel, dim3((unsigned)((ngroups + 255) / 256)), dim3(256), 0, st, mask_pre, wq, d_mask_pre, ngroups, 2);
    return check_launch("dna_fused_bwd(softmax)");
}

int pivp_stp_fused_fwd(const float* prev, const float* enc7_pre, const float* mask_pre, const float* theta_raw, float* out,
                       int B, int H, int W, int num_masks, int oob_border, void* stream) {
    PIVP_REQUIRE(prev && enc7_pre && mask_pre && theta_raw && out && B > 0 && num_masks >= 1, "stp_fused_fwd: bad argument");
    Band bd;
    if (int e = make_band(H, W, num_masks + 1, 0, &bd)) return e;
    const size_t smem = sizeof(float) * ((size_t)bd.M1 * bd.L);
    if (int e = allow_smem(stp_kernel, smem)) return e;
    launch_k(stp_kernel, dim3((H + bd.R - 1) / bd.R, B), dim3(FT), smem, (cudaStream_t)stream, prev, enc7_pre, mask_pre, theta_raw, nullptr, out, nullptr,
                                                                                  nullptr, nullptr, nullptr, bd, num_masks, oob_border, 0);
    return check_launch("stp_fused_fwd");
}

size_t pivp_stp_fused_bwd_workspace_bytes(int B, int H, int W, int num_masks) {
    return sizeof(float) * (size_t)B * (num_masks + 1) * H * W;
}

// d_theta is OVERWRITTEN; d_prev (optional) is ACCUMULATED into (scatter-add).
int pivp_stp_fused_bwd(const float* g_out, const float* prev, const float* enc7_pre, const float* mask_pre, const float* theta_raw,
                       float* d_enc7_pre, float* d_mask_pre, float* d_theta, float* d_prev,
                       int B, int H, int W, int num_masks, int oob_border, void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(g_out && prev && enc7_pre && mask_pre && theta_raw && d_enc7_pre && d_mask_pre && d_theta && workspace,
                 "stp_fused_bwd: null pointer");
    PIVP_REQUIRE(ws_bytes >= pivp_stp_fused_bwd_workspace_bytes(B, H, W, num_masks), "stp_fused_bwd: workspace too small");
    Band bd;
    if (int e = make_band(H, W, num_masks + 1, 0, &bd)) return e;
    cudaStream_t st = (cudaStream_t)stream;
    float* wq = (float*)workspace;
    cudaMemsetAsync(d_theta, 0, sizeof(float) * (size_t)B * 6, st);
    const size_t smem = sizeof(float) * ((size_t)bd.M1 * bd.L);
    if (int e = allow_smem(stp_kernel, smem)) return e;
    launch_k(stp_kernel, dim3((H + bd.R - 1) / bd.R, B), dim3(FT), smem, st, prev, enc7_pre, mask_pre, theta_raw, g_out, nullptr, wq, d_enc7_pre, d_theta,
                                                                d_prev, bd, num_masks, oob_border, 1);
    if (int e = check_launch("stp_fused_bwd(k1)")) return e;
    const long ngroups = (long)B * H * W;
    launch_k(mask_softmax_bwd_kernel, dim3((unsigned)((ngroups + 255) / 256)), dim3(256), 0, st, mask_pre, wq, d_mask_pre, ngroups, num_masks + 1);
    return check_launch("stp_fused_bwd(softmax)");
}

}  // extern "C"
