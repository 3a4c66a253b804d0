// Un-fused transformation lists of StatelessCDNA / StatelessDNA / StatelessSTP (train_model.py:293-351, 368-417, 434-475): the
// reference call surface returns (transformed_list, enc7) and lets Model.__call__ composite them (:725-728).  The training path never
// materialises these lists (fused_transform.cu / cdna_band.cu composite in the same pass); these kernels exist so that the links can
// also be called exactly like the reference's, e.g. by visualisation code that wants the individual transformed images.
//   out layout: [L][B][3][H][W], L = number of list entries; entry 0 of CDNA / STP is sigmoid(enc7) (:315-317, :454-455).
// The backward entry points take the gradient of the list as L separate planes (Chainer's grad_outputs, NULL = no gradient), so a link
// dropped into the reference Model, which composites with zip(transformed, mask_list[1:]) (:725-728), trains through the list form too.
#include "transform_common.cuh"

namespace pivp {
namespace unf {

// CDNA: thread = (b, y, x); normalised kernels of the sample in shared memory.  grid (ceil(HW/256), B)
__global__ void __launch_bounds__(256) cdna_list_kernel(const float* __restrict__ prev, const float* __restrict__ e_pre,
                                                        const float* __restrict__ kraw, float* __restrict__ out, int B, int H, int W, int M) {
    pdl_enter();
    extern __shared__ float kn[];                  // [M][25]
    const int b = blockIdx.y, HW = H * W;
    for (int m = threadIdx.x; m < M; m += 256) {
        float kt[25], s = 0.f;
#pragma unroll
        for (int t = 0; t < 25; ++t) { kt[t] = fmaxf(kraw[(long)b * 25 * M + m * 25 + t] - RELU_SHIFT, 0.f) + RELU_SHIFT; s += kt[t]; }
#pragma unroll
        for (int t = 0; t < 25; ++t) kn[m * 25 + t] = kt[t] / s;
    }
    __syncthreads();
    const int q = blockIdx.x * 256 + threadIdx.x;
    if (q >= HW) return;
    const int y = q / W, x = q - y * W;
    const long LS = (long)B * 3 * HW;              // stride between list entries
    for (int c = 0; c < 3; ++c) {
        const long p = ((long)b * 3 + c) * HW;
        out[p + q] = sigmoid_acc(fmaxf(e_pre[p + q], 0.f));                       // sigmoid(relu(enc7_pre))
        float win[25];
#pragma unroll
        for (int u = 0; u < 5; ++u)
#pragma unroll
            for (int v = 0; v < 5; ++v) {
                const int yy = y + u - 2, xx = x + v - 2;
                win[u * 5 + v] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(prev + p + yy * W + xx) : 0.f;
            }
        for (int m = 0; m < M; ++m) {
            float acc = 0.f;
#pragma unroll
            for (int t = 0; t < 25; ++t) acc = fmaf(kn[m * 25 + t], win[t], acc);    // cross-correlation, zero padding, no flip (:341)
            out[(long)(m + 1) * LS + p + q] = acc;
        }
    }
}

// DNA: one entry; tap (xk,yk) of pixel (i,j) reads prev[i+xk-2][j+yk-2] iff i+xk < H and j+yk < W (App. B.2)
__global__ void __launch_bounds__(256) dna_list_kernel(const float* __restrict__ prev, const float* __restrict__ e_pre, float* __restrict__ out,
                                                       int B, int H, int W) {
    pdl_enter();
    const int b = blockIdx.y, HW = H * W;
    const int q = blockIdx.x * 256 + threadIdx.x;
    if (q >= HW) return;
    const int y = q / W, x = q - y * W;
    float k[25], s = 0.f;
#pragma unroll
    for (int t = 0; t < 25; ++t) { k[t] = fmaxf(fmaxf(e_pre[((long)b * 25 + t) * HW + q], 0.f) - RELU_SHIFT, 0.f) + RELU_SHIFT; s += k[t]; }
    const float inv = 1.f / s;
    for (int c = 0; c < 3; ++c) {
        const long p = ((long)b * 3 + c) * HW;
        float acc = 0.f;
#pragma unroll
        for (int u = 0; u < 5; ++u)
#pragma unroll
            for (int v = 0; v < 5; ++v) {
                const int yy = y + u - 2, xx = x + v - 2;
                const bool live = (y + u < H) && (x + v < W) && yy >= 0 && xx >= 0;
                acc = fmaf(k[u * 5 + v] * inv, live ? __ldg(prev + p + yy * W + xx) : 0.f, acc);
            }
        out[p + q] = acc;
    }
}

// STP: entry 0 = sigmoid(enc7) (no ReLU, :454-455); entries 1..M-1 all sample with the SAME theta (App. B.4)
__global__ void __launch_bounds__(256) stp_list_kernel(const float* __restrict__ prev, const float* __restrict__ e_pre,
                                                       const float* __restrict__ theta_raw, float* __restrict__ out, int B, int H, int W, int M, int oob) {
    pdl_enter();
    const int b = blockIdx.y, HW = H * W;
    const int q = blockIdx.x * 256 + threadIdx.x;
    if (q >= HW) return;
    const int yi = q / W, x = q - yi * W;
    float th[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) th[i] = theta_raw[b * 6 + i] + ((i == 0 || i == 4) ? 1.f : 0.f);
    const float sx = (W > 1) ? 2.f / (float)(W - 1) : 0.f, sy = (H > 1) ? 2.f / (float)(H - 1) : 0.f;
    const float hw = 0.5f * (float)(W - 1), hh = 0.5f * (float)(H - 1);
    const float xn = -1.f + sx * (float)x, yn = -1.f + sy * (float)yi;
    float u = (th[0] * xn + th[1] * yn + th[2] + 1.f) * hw;
    float v = (th[3] * xn + th[4] * yn + th[5] + 1.f) * hh;
    if (oob == 1) { u = fminf(fmaxf(u, 0.f), (float)(W - 1)); v = fminf(fmaxf(v, 0.f), (float)(H - 1)); }
    const float uc = fminf(fmaxf(u, -2.f), (float)W + 1.f), vc = fminf(fmaxf(v, -2.f), (float)H + 1.f);
    const float fu0 = floorf(uc), fv0 = floorf(vc);
    const int u0 = (int)fu0, v0 = (int)fv0;
    const float fu = uc - fu0, fv = vc - fv0;
    const bool inside = (u == uc) && (v == vc);
    const bool ok00 = inside && v0 >= 0 && v0 < H && u0 >= 0 && u0 < W;
    const bool ok01 = inside && v0 >= 0 && v0 < H && u0 + 1 >= 0 && u0 + 1 < W;
    const bool ok10 = inside && v0 + 1 >= 0 && v0 + 1 < H && u0 >= 0 && u0 < W;
    const bool ok11 = inside && v0 + 1 >= 0 && v0 + 1 < H && u0 + 1 >= 0 && u0 + 1 < W;
    const float w00 = (1.f - fv) * (1.f - fu), w01 = (1.f - fv) * fu, w10 = fv * (1.f - fu), w11 = fv * fu;
    const long LS = (long)B * 3 * HW;
    for (int c = 0; c < 3; ++c) {
        const long p = ((long)b * 3 + c) * HW;
        const float* Pc = prev + p;
        const float S = (ok00 ? Pc[v0 * W + u0] : 0.f) * w00 + (ok01 ? Pc[v0 * W + u0 + 1] : 0.f) * w01 +
                        (ok10 ? Pc[(v0 + 1) * W + u0] : 0.f) * w10 + (ok11 ? Pc[(v0 + 1) * W + u0 + 1] : 0.f) * w11;
        out[p + q] = sigmoid_acc(e_pre[p + q]);
        for (int m = 1; m < M; ++m) out[(long)m * LS + p + q] = S;
    }
}

// ====================================================================================== backward of the lists
// Gradient of the list: one (B,3,H,W) plane per entry, NULL = that entry has no gradient (is not read).  Passed by value.
constexpr int MAXL = 65;                       // CDNA: num_masks <= 64 kernels + the sigmoid entry
struct GradList {
    const float* g[MAXL];
};

constexpr int LT = 256;                        // threads per CTA of the band kernels
constexpr int LPX = 2;                         // pixels per thread: a band holds at most LT * LPX pixels

static int list_band_rows(int H, int W) {
    int R = (LT * LPX) / W;
    if (R < 1) R = 1;
    if (R > H) R = H;
    return R;
}

// Sum of v[t] over the 32 lanes of the warp for every t < 32, returned in lane t: a reduce-scatter (31 shuffles, fixed order) instead of
// 32 butterfly sums of 5 shuffles each.  At step o every lane keeps the half of its values selected by lane bit o and adds the partner's.
__device__ __forceinline__ float warp_reduce_scatter32(float (&v)[32]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int i = 0; i < o; ++i) {
            const float send = up ? v[i] : v[i + o];
            const float keep = up ? v[i + o] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
    return v[0];
}

// CDNA: CTA = (band of R rows, sample).  prev (+2 halo) is staged once; the live gradient planes g_{m+1} are staged one after the other
// (+2 halo) into one buffer, and both products of an entry are taken from the two staged tiles:
//   dK[m][t]   = sum_c sum_q g_{m+1}[c,q] prev[c,q+off_t]       (per-band partial -> dKp[b][band][m][25], reduced by the finalize kernel)
//   d_prev[c,p] = sum_m sum_t kn[m][t] g_{m+1}[c,p-off_t]        (gather, in registers over the entries, written once)
// and d_enc7_pre = [e > 0] (g_enc7 + g_0 s (1 - s)), s = sigmoid(relu(e)).
__global__ void __launch_bounds__(LT) cdna_list_bwd_kernel(GradList gl, const float* __restrict__ g_e7, const float* __restrict__ prev,
                                                           const float* __restrict__ e_pre, const float* __restrict__ kraw,
                                                           float* __restrict__ d_e, float* __restrict__ d_prev, int acc_dprev,
                                                           float* __restrict__ dKp, int H, int W, int R, int M) {
    pdl_enter();
    extern __shared__ float sm[];
    const int b = blockIdx.y, band = blockIdx.x, nb = gridDim.x, r0 = band * R;
    const int nrows = min(R, H - r0), HW = H * W, np = nrows * W;
    const int TW = W + 4, TS = (nrows + 4) * TW;
    float* ptile = sm;                                                          // [3][R+4][W+4]
    float* gtile = ptile + 3 * (R + 4) * TW;                                    // [3][R+4][W+4]
    float* kn = gtile + 3 * (R + 4) * TW;                                       // [M][25]
    float* red = kn + M * 25;                                                   // [LT/32][25]
    const long sb = (long)b * 3 * HW, bo = sb + (long)r0 * W;                   // sample / band offsets
    cdna_normalise(kraw + (long)b * M * 25, M, kn, nullptr);
    load_prev_tile(prev + sb, H, W, r0, nrows, ptile);
    const float* g0 = gl.g[0];
    for (int q = threadIdx.x; q < np; q += LT) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const long p = bo + (long)c * HW + q;
            const float ev = __ldg(e_pre + p);
            float d = g_e7 ? __ldg(g_e7 + p) : 0.f;
            if (g0) {
                const float s = sigmoid_acc(fmaxf(ev, 0.f));
                d = fmaf(__ldg(g0 + p), s * (1.f - s), d);
            }
            d_e[p] = ev > 0.f ? d : 0.f;
        }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float dp[LPX][3];
#pragma unroll
    for (int i = 0; i < LPX; ++i)
#pragma unroll
        for (int c = 0; c < 3; ++c) dp[i][c] = 0.f;
    for (int m = 0; m < M; ++m) {
        const float* gm = gl.g[m + 1];
        float* part = dKp + (((long)b * nb + band) * M + m) * 25;
        if (!gm) {                                                              // uniform over the CTA
            if (threadIdx.x < 25) part[threadIdx.x] = 0.f;
            continue;
        }
        __syncthreads();                                                        // gtile / red of the previous entry consumed
        load_prev_tile(gm + sb, H, W, r0, nrows, gtile);
        __syncthreads();
        float acc[32];
#pragma unroll
        for (int t = 0; t < 32; ++t) acc[t] = 0.f;
        const float* km = kn + m * 25;
#pragma unroll
        for (int i = 0; i < LPX; ++i) {
            const int q = threadIdx.x + i * LT;
            if (q < np) {
                const int y = q / W, x = q - y * W;
                const float* tp = ptile + y * TW + x;                           // top-left of the 5x5 window of pixel q
                const float* gp = gtile + y * TW + x;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float gc = gp[c * TS + 2 * TW + 2];
#pragma unroll
                    for (int u = 0; u < 5; ++u)
#pragma unroll
                        for (int v = 0; v < 5; ++v) acc[u * 5 + v] = fmaf(gc, tp[c * TS + u * TW + v], acc[u * 5 + v]);
                    if (d_prev) {
                        float a = dp[i][c];
#pragma unroll
                        for (int u = 0; u < 5; ++u)
#pragma unroll
                            for (int v = 0; v < 5; ++v) a = fmaf(km[u * 5 + v], gp[c * TS + (4 - u) * TW + 4 - v], a);
                        dp[i][c] = a;
                    }
                }
            }
        }
        const float wsum = warp_reduce_scatter32(acc);
        if (lane < 25) red[warp * 25 + lane] = wsum;
        __syncthreads();
        if (threadIdx.x < 25) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < LT / 32; ++w) s += red[w * 25 + threadIdx.x];
            part[threadIdx.x] = s;
        }
    }
    if (d_prev) {
#pragma unroll
        for (int i = 0; i < LPX; ++i) {
            const int q = threadIdx.x + i * LT;
            if (q < np) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    float* d = d_prev + bo + (long)c * HW + q;
                    *d = acc_dprev ? (*d + dp[i][c]) : dp[i][c];
                }
            }
        }
    }
}

// dK = sum of the per-band partials (fixed order), then the normalisation backward: one thread per (sample, kernel)
__global__ void cdna_list_kern_bwd_kernel(const float* __restrict__ dKp, const float* __restrict__ kraw, float* __restrict__ d_kraw,
                                          int B, int M, int nb) {
    pdl_enter();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * M) return;
    const int b = i / M, m = i - b * M;
    float dK[25];
#pragma unroll
    for (int t = 0; t < 25; ++t) dK[t] = 0.f;
    for (int k = 0; k < nb; ++k) {
        const float* p = dKp + (((long)b * nb + k) * M + m) * 25;
#pragma unroll
        for (int t = 0; t < 25; ++t) dK[t] += p[t];
    }
    cdna_kern_bwd_one(kraw + (long)i * 25, dK, d_kraw + (long)i * 25);
}

// DNA: CTA = (band, sample), prev staged (+2 halo) when the entry has a gradient.  The taps are detached (ref:404): no d_prev.
//   dkhat_t = sum_c g_0[c] tap_t[c] (truncated windows of :395-405, the liveness rule of dna_list_kernel)
//   d_e_t = [e_t > 0] (g_enc7_t + [relu(e_t) > eps] (dkhat_t - sum_s khat_s dkhat_s) / S)
__global__ void __launch_bounds__(LT) dna_list_bwd_kernel(const float* __restrict__ g0, const float* __restrict__ g_e7,
                                                          const float* __restrict__ prev, const float* __restrict__ e_pre,
                                                          float* __restrict__ d_e, int H, int W, int R) {
    pdl_enter();
    extern __shared__ float sm[];
    const int b = blockIdx.y, r0 = blockIdx.x * R;
    const int nrows = min(R, H - r0), HW = H * W, np = nrows * W;
    const int TW = W + 4, TS = (nrows + 4) * TW;
    if (g0) {
        load_prev_tile(prev + (long)b * 3 * HW, H, W, r0, nrows, sm);
        __syncthreads();
    }
    for (int q = threadIdx.x; q < np; q += LT) {
        const int y = q / W, x = q - y * W, yi = r0 + y;
        const long ep = (long)b * 25 * HW + yi * W + x;
        float ev[25], k[25], s = 0.f;
#pragma unroll
        for (int t = 0; t < 25; ++t) {
            ev[t] = __ldg(e_pre + ep + (long)t * HW);
            k[t] = fmaxf(fmaxf(ev[t], 0.f) - RELU_SHIFT, 0.f) + RELU_SHIFT;
            s += k[t];
        }
        const float inv = 1.f / s;
        float dk[25], dot = 0.f;
#pragma unroll
        for (int t = 0; t < 25; ++t) dk[t] = 0.f;
        if (g0) {
            const long gp = (long)b * 3 * HW + yi * W + x;
            float g[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) g[c] = __ldg(g0 + gp + (long)c * HW);
            const float* trow = sm + y * TW + x;
#pragma unroll
            for (int u = 0; u < 5; ++u)
#pragma unroll
                for (int v = 0; v < 5; ++v) {
                    float d = 0.f;
#pragma unroll
                    for (int c = 0; c < 3; ++c) d = fmaf(g[c], trow[c * TS + u * TW + v], d);
                    dk[u * 5 + v] = (yi + u < H && x + v < W) ? d : 0.f;
                }
#pragma unroll
            for (int t = 0; t < 25; ++t) dot = fmaf(k[t] * inv, dk[t], dot);
        }
#pragma unroll
        for (int t = 0; t < 25; ++t) {
            float d = g_e7 ? __ldg(g_e7 + ep + (long)t * HW) : 0.f;
            if (k[t] > RELU_SHIFT) d += (dk[t] - dot) * inv;
            d_e[ep + (long)t * HW] = ev[t] > 0.f ? d : 0.f;
        }
    }
}

// STP: CTA = (band, sample).  The sampled entries share theta (B.4), so only their sum g_S = sum_{m>=1} g_m reaches the sampler backward
// (the grid + bilinear-sampler backward of stp_kernel, live_u / live_v included).  The sampler reads prev at arbitrary positions, so
// nothing is staged; every gradient plane is read once.  d_theta: per-band partials dthp[b][band][6] (block sums, fixed order), reduced by
// the finalize kernel.  d_prev: scatter-add (atomics), NULL when no sampled entry has a gradient.  d_e = g_enc7 + g_0 sigmoid'(e).
__global__ void __launch_bounds__(LT) stp_list_bwd_kernel(GradList gl, int L, const float* __restrict__ g_e7, const float* __restrict__ prev,
                                                          const float* __restrict__ e_pre, const float* __restrict__ theta_raw,
                                                          float* __restrict__ d_e, float* __restrict__ dthp, float* __restrict__ d_prev,
                                                          int H, int W, int R, int oob) {
    pdl_enter();
    __shared__ float red[32];
    const int b = blockIdx.y, band = blockIdx.x, nb = gridDim.x, r0 = band * R;
    const int nrows = min(R, H - r0), HW = H * W, np = nrows * W;
    float th[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) th[i] = __ldg(theta_raw + b * 6 + i) + ((i == 0 || i == 4) ? 1.f : 0.f);
    const float* P = prev + (long)b * 3 * HW;
    const float* g0 = gl.g[0];
    const float sx = (W > 1) ? 2.f / (float)(W - 1) : 0.f, sy = (H > 1) ? 2.f / (float)(H - 1) : 0.f;
    const float hw = 0.5f * (float)(W - 1), hh = 0.5f * (float)(H - 1);
    float dth[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int q = threadIdx.x; q < np; q += LT) {
        const int y = q / W, x = q - y * W, yi = r0 + y;
        const long gp = (long)b * 3 * HW + yi * W + x;
        float gS[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const long p = gp + (long)c * HW;
            float d = g_e7 ? __ldg(g_e7 + p) : 0.f;
            if (g0) {
                const float s = sigmoid_acc(__ldg(e_pre + p));
                d = fmaf(__ldg(g0 + p), s * (1.f - s), d);
            }
            d_e[p] = d;
        }
        for (int m = 1; m < L; ++m) {
            const float* gm = gl.g[m];
            if (gm) {
#pragma unroll
                for (int c = 0; c < 3; ++c) gS[c] += __ldg(gm + gp + (long)c * HW);
            }
        }
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
        const float uc = fminf(fmaxf(u, -2.f), (float)W + 1.f), vc = fminf(fmaxf(v, -2.f), (float)H + 1.f);
        const float fu0 = floorf(uc), fv0 = floorf(vc);
        const int u0 = (int)fu0, v0 = (int)fv0;
        const float fu = uc - fu0, fv = vc - fv0;
        const bool inside = (u == uc) && (v == vc);
        const bool ok00 = inside && v0 >= 0 && v0 < H && u0 >= 0 && u0 < W;
        const bool ok01 = inside && v0 >= 0 && v0 < H && u0 + 1 >= 0 && u0 + 1 < W;
        const bool ok10 = inside && v0 + 1 >= 0 && v0 + 1 < H && u0 >= 0 && u0 < W;
        const bool ok11 = inside && v0 + 1 >= 0 && v0 + 1 < H && u0 + 1 >= 0 && u0 + 1 < W;
        const float w00 = (1.f - fv) * (1.f - fu), w01 = (1.f - fv) * fu, w10 = fv * (1.f - fu), w11 = fv * fu;
        float gu = 0.f, gv = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float* Pc = P + (long)c * HW;
            const float p00 = ok00 ? __ldg(Pc + v0 * W + u0) : 0.f;
            const float p01 = ok01 ? __ldg(Pc + v0 * W + u0 + 1) : 0.f;
            const float p10 = ok10 ? __ldg(Pc + (v0 + 1) * W + u0) : 0.f;
            const float p11 = ok11 ? __ldg(Pc + (v0 + 1) * W + u0 + 1) : 0.f;
            const float dS = gS[c];
            gu = fmaf(dS, (p01 - p00) * (1.f - fv) + (p11 - p10) * fv, gu);
            gv = fmaf(dS, (p10 - p00) * (1.f - fu) + (p11 - p01) * fu, gv);
            if (d_prev) {
                float* D = d_prev + (long)b * 3 * HW + (long)c * HW;
                if (ok00) atomicAdd(D + v0 * W + u0, dS * w00);
                if (ok01) atomicAdd(D + v0 * W + u0 + 1, dS * w01);
                if (ok10) atomicAdd(D + (v0 + 1) * W + u0, dS * w10);
                if (ok11) atomicAdd(D + (v0 + 1) * W + u0 + 1, dS * w11);
            }
        }
        gu *= (live_u ? hw : 0.f);
        gv *= (live_v ? hh : 0.f);
        dth[0] += gu * xn; dth[1] += gu * yn; dth[2] += gu;
        dth[3] += gv * xn; dth[4] += gv * yn; dth[5] += gv;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const float s = block_sum(dth[i], red);
        if (threadIdx.x == 0) dthp[((long)b * nb + band) * 6 + i] = s;
    }
}

// d_theta_raw[b][i] = sum of the per-band partials (fixed order)
__global__ void stp_list_theta_bwd_kernel(const float* __restrict__ dthp, float* __restrict__ d_theta, int B, int nb) {
    pdl_enter();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * 6) return;
    const int b = i / 6, j = i - b * 6;
    float s = 0.f;
    for (int k = 0; k < nb; ++k) s += dthp[((long)b * nb + k) * 6 + j];
    d_theta[i] = s;
}

__global__ void zero_kernel(float* __restrict__ p, long n) {
    pdl_enter();
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = 0.f;
}

}  // namespace unf
}  // namespace pivp

using namespace pivp;

extern "C" {

int pivp_cdna_transform(const float* prev, const float* enc7_pre, const float* kern_raw, float* out, int B, int H, int W, int num_masks, void* stream) {
    PIVP_REQUIRE(prev && enc7_pre && kern_raw && out && B > 0 && H > 0 && W > 0 && num_masks >= 1 && num_masks <= 64, "cdna_transform: bad argument");
    dim3 grid((unsigned)((H * W + 255) / 256), (unsigned)B);
    launch_k(unf::cdna_list_kernel, grid, dim3(256), sizeof(float) * 25 * num_masks, stream, prev, enc7_pre, kern_raw, out, B, H, W, num_masks);
    return check_launch("cdna_transform");
}

int pivp_dna_transform(const float* prev, const float* enc7_pre, float* out, int B, int H, int W, void* stream) {
    PIVP_REQUIRE(prev && enc7_pre && out && B > 0 && H > 0 && W > 0, "dna_transform: bad argument");
    dim3 grid((unsigned)((H * W + 255) / 256), (unsigned)B);
    launch_k(unf::dna_list_kernel, grid, dim3(256), 0, stream, prev, enc7_pre, out, B, H, W);
    return check_launch("dna_transform");
}

int pivp_stp_transform(const float* prev, const float* enc7_pre, const float* theta_raw, float* out, int B, int H, int W, int num_masks, int oob,
                       void* stream) {
    PIVP_REQUIRE(prev && enc7_pre && theta_raw && out && B > 0 && H > 0 && W > 0 && num_masks >= 1, "stp_transform: bad argument");
    dim3 grid((unsigned)((H * W + 255) / 256), (unsigned)B);
    launch_k(unf::stp_list_kernel, grid, dim3(256), 0, stream, prev, enc7_pre, theta_raw, out, B, H, W, num_masks, oob);
    return check_launch("stp_transform");
}

static size_t cdna_list_bwd_smem(int H, int W, int M) {
    const int R = unf::list_band_rows(H, W);
    return sizeof(float) * (2 * 3 * (size_t)(R + 4) * (W + 4) + (size_t)M * 25 + (unf::LT / 32) * 25);
}

size_t pivp_cdna_transform_bwd_workspace_bytes(int B, int H, int W, int num_masks) {
    if (B <= 0 || H <= 0 || W <= 0 || num_masks < 1) return 0;
    const int R = unf::list_band_rows(H, W);
    return sizeof(float) * (size_t)B * ((H + R - 1) / R) * num_masks * 25;      // per-band partials of dK
}

int pivp_cdna_transform_bwd(const float* const* g_list, const float* g_enc7, const float* prev, const float* enc7_pre, const float* kern_raw,
                            float* d_enc7_pre, float* d_kern_raw, float* d_prev, int accumulate_dprev,
                            int B, int H, int W, int num_masks, void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(g_list && prev && enc7_pre && kern_raw && d_enc7_pre && d_kern_raw && workspace, "cdna_transform_bwd: null pointer");
    PIVP_REQUIRE(B > 0 && H > 0 && W > 0 && num_masks >= 1 && num_masks <= 64, "cdna_transform_bwd: bad geometry (need 1 <= num_masks <= 64)");
    PIVP_REQUIRE(ws_bytes >= pivp_cdna_transform_bwd_workspace_bytes(B, H, W, num_masks), "cdna_transform_bwd: workspace too small");
    const size_t smem = cdna_list_bwd_smem(H, W, num_masks);
    PIVP_REQUIRE(smem <= 48 * 1024, "cdna_transform_bwd: image too wide for the band staging");
    unf::GradList gl;
    memset(&gl, 0, sizeof(gl));
    for (int i = 0; i <= num_masks; ++i) gl.g[i] = g_list[i];
    const int R = unf::list_band_rows(H, W), nb = (H + R - 1) / R;
    float* dKp = (float*)workspace;
    launch_k(unf::cdna_list_bwd_kernel, dim3((unsigned)nb, (unsigned)B), dim3(unf::LT), smem, stream, gl, g_enc7, prev, enc7_pre, kern_raw,
             d_enc7_pre, d_prev, accumulate_dprev, dKp, H, W, R, num_masks);
    if (int e = check_launch("cdna_transform_bwd")) return e;
    launch_k(unf::cdna_list_kern_bwd_kernel, dim3((unsigned)((B * num_masks + 127) / 128)), dim3(128), 0, stream, (const float*)dKp, kern_raw,
             d_kern_raw, B, num_masks, nb);
    return check_launch("cdna_transform_bwd(kern)");
}

int pivp_dna_transform_bwd(const float* const* g_list, const float* g_enc7, const float* prev, const float* enc7_pre, float* d_enc7_pre,
                           int B, int H, int W, void* stream) {
    PIVP_REQUIRE(g_list && prev && enc7_pre && d_enc7_pre, "dna_transform_bwd: null pointer");
    PIVP_REQUIRE(B > 0 && H > 0 && W > 0, "dna_transform_bwd: bad geometry");
    const int R = unf::list_band_rows(H, W);
    const size_t smem = sizeof(float) * 3 * (size_t)(R + 4) * (W + 4);
    PIVP_REQUIRE(smem <= 48 * 1024, "dna_transform_bwd: image too wide for the band staging");
    launch_k(unf::dna_list_bwd_kernel, dim3((unsigned)((H + R - 1) / R), (unsigned)B), dim3(unf::LT), smem, stream, g_list[0], g_enc7, prev,
             enc7_pre, d_enc7_pre, H, W, R);
    return check_launch("dna_transform_bwd");
}

size_t pivp_stp_transform_bwd_workspace_bytes(int B, int H, int W, int num_masks) {
    if (B <= 0 || H <= 0 || W <= 0 || num_masks < 1) return 0;
    const int R = unf::list_band_rows(H, W);
    return sizeof(float) * (size_t)B * ((H + R - 1) / R) * 6;                     // per-band partials of d_theta
}

int pivp_stp_transform_bwd(const float* const* g_list, const float* g_enc7, const float* prev, const float* enc7_pre, const float* theta_raw,
                           float* d_enc7_pre, float* d_theta_raw, float* d_prev, int accumulate_dprev,
                           int B, int H, int W, int num_masks, int oob_border, void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(g_list && prev && enc7_pre && theta_raw && d_enc7_pre && d_theta_raw && workspace, "stp_transform_bwd: null pointer");
    PIVP_REQUIRE(B > 0 && H > 0 && W > 0 && num_masks >= 1 && num_masks <= 64, "stp_transform_bwd: bad geometry (need 1 <= num_masks <= 64)");
    PIVP_REQUIRE(ws_bytes >= pivp_stp_transform_bwd_workspace_bytes(B, H, W, num_masks), "stp_transform_bwd: workspace too small");
    unf::GradList gl;
    memset(&gl, 0, sizeof(gl));
    bool sampled = false;                                   // does any sampled entry (1 .. L-1) carry a gradient?
    for (int i = 0; i < num_masks; ++i) {
        gl.g[i] = g_list[i];
        sampled |= i > 0 && g_list[i] != nullptr;
    }
    const int R = unf::list_band_rows(H, W), nb = (H + R - 1) / R;
    float* dthp = (float*)workspace;
    if (d_prev && !accumulate_dprev) {
        const long n = (long)B * 3 * H * W;
        launch_k(unf::zero_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, stream, d_prev, n);
        if (int e = check_launch("stp_transform_bwd(zero)")) return e;
    }
    launch_k(unf::stp_list_bwd_kernel, dim3((unsigned)nb, (unsigned)B), dim3(unf::LT), 0, stream, gl, num_masks, g_enc7, prev, enc7_pre,
             theta_raw, d_enc7_pre, dthp, sampled ? d_prev : nullptr, H, W, R, oob_border);
    if (int e = check_launch("stp_transform_bwd")) return e;
    launch_k(unf::stp_list_theta_bwd_kernel, dim3((unsigned)((B * 6 + 127) / 128)), dim3(128), 0, stream, (const float*)dthp, d_theta_raw, B, nb);
    return check_launch("stp_transform_bwd(theta)");
}


}  // extern "C"
