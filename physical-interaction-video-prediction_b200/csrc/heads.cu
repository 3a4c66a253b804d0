// The two 1x1 "head" deconvolutions on enc6 (train_model.py:288/364/429 enc7 and :527 masks, applied at :315/:388/:454 and :719)
// as ONE bandwidth-bound kernel each way.  enc6 is the widest activation of the model (B*H*W x 64 fp32 = 33.5 MB at b32); the generic
// path read it three times per time step (forward, weight gradient, input gradient) through implicit-GEMM tiles sized for real
// convolutions and moved the 14 output planes through two extra NHWC<->NCHW transposes.
//
//   forward : [enc7_pre | mask_pre] (NCHW planes) = e6 (NHWC rows) . W^T + b          reads 256 B, writes 4*NH B per pixel
//   backward: d_e6 = dY . W ; dW += dY^T . e6 ; db += sum dY                          reads 256 + 4*NH B, writes 256 B per pixel
//
// CTA tile = 128 pixels staged in shared memory with coalesced 128-bit accesses (row pitch 68 floats: conflict-free for one
// row per thread).  Arithmetic is packed fp32 (FFMA2).  NH (heads: 3+11 for CDNA/STP with 10 masks, 25+2 for DNA) is a template
// parameter so every accumulator stays in a register.
#include "common.cuh"
#include <string.h>

namespace pivp {
namespace hd {

constexpr int TP = 128;              // pixels per tile = threads per CTA
constexpr int C = 64;                // enc6 channels
constexpr int XP = 68;               // smem row pitch of the pixel tile (floats)

__device__ __forceinline__ unsigned long long pk2(float2 a) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y));
    return r;
}
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b)), "l"(pk2(c)));
    float2 d;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(r));
    return d;
}

// coalesced copy of a 128-pixel x 64-channel tile between global rows (stride cs, offset co) and shared memory
template <int BATCH>
__device__ __forceinline__ void load_tile(const float* __restrict__ x, int cs, int co, long m0, long M, float* xs) {
    // BATCH loads of a thread are issued before their shared-memory stores (16 / BATCH memory round trips per tile, not sixteen)
    constexpr int NL = TP * (C / 4) / TP;
#pragma unroll
    for (int k0 = 0; k0 < NL; k0 += BATCH) {
        float4 v[BATCH];
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
            const int i = threadIdx.x + (k0 + k) * TP, r = i >> 4, c4 = i & 15;
            v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (m0 + r < M) v[k] = __ldg(reinterpret_cast<const float4*>(x + (m0 + r) * cs + co) + c4);
        }
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
            const int i = threadIdx.x + (k0 + k) * TP, r = i >> 4, c4 = i & 15;
            *reinterpret_cast<float4*>(xs + r * XP + 4 * c4) = v[k];
        }
    }
}

// LayerNorm + ReLU applied while the tile is staged (pivp_heads_fwd_ln): x is the PRE-normalisation tensor (enc6's deconvolution output),
// the (mean, M2) partials of the sample come from the deconvolution's epilogue, and the normalised tile is also written to y for the backward.
struct LnIn {
    const float* gamma; const float* beta;       // per element of a sample, [HW][64]; gamma == null: no LayerNorm (x is used as it is)
    const float2* partial; int S;                // [B][S] pairs over 4096 values each
    float eps;
    float2* stats;                               // [B] (mean, rstd) saved for the LayerNorm backward
    float* y; int y_cs, y_co;                    // normalised + ReLU output rows
};

// Chan merge of the S equal-sized chunk partials of sample b by one warp (same order as lnv::combine_warp); (mean, rstd) in every lane
__device__ __forceinline__ float2 ln_combine(const float2* __restrict__ partial, long b, int S, float eps, int lane) {
    float wsum = 0.f;
    for (int s = lane; s < S; s += 32) wsum += partial[b * S + s].x * 4096.f;
    const float n = 4096.f * (float)S;
    const float mu = warp_sum(wsum) / n;
    float m2 = 0.f;
    for (int s = lane; s < S; s += 32) {
        const float2 p = partial[b * S + s];
        const float d = p.x - mu;
        m2 += p.y + 4096.f * d * d;
    }
    m2 = warp_sum(m2);
    return make_float2(mu, 1.f / sqrtf(m2 / n + eps));
}

// Y = false: the normalised rows are not written (pivp_heads_fwd_ln with y == NULL: forward-only prediction, no backward reads them)
template <int BATCH, bool Y>
__device__ __forceinline__ void load_tile_ln(const float* __restrict__ x, int cs, int co, long m0, long M, float* xs, const LnIn& ln, float2 st,
                                             long e0) {
    constexpr int NL = TP * (C / 4) / TP;
#pragma unroll
    for (int k0 = 0; k0 < NL; k0 += BATCH) {
        float4 v[BATCH], ga[BATCH], be[BATCH];
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
            const int i = threadIdx.x + (k0 + k) * TP, r = i >> 4, c4 = i & 15;
            v[k] = ga[k] = be[k] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (m0 + r < M) {
                v[k] = __ldg(reinterpret_cast<const float4*>(x + (m0 + r) * cs + co) + c4);
                ga[k] = __ldg(reinterpret_cast<const float4*>(ln.gamma + e0) + i);       // element (pixel r, channel 4 c4) of the sample = e0 + 4 i
                be[k] = __ldg(reinterpret_cast<const float4*>(ln.beta + e0) + i);
            }
        }
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
            const int i = threadIdx.x + (k0 + k) * TP, r = i >> 4, c4 = i & 15;
            float4 o;
            o.x = fmaxf((v[k].x - st.x) * st.y * ga[k].x + be[k].x, 0.f);
            o.y = fmaxf((v[k].y - st.x) * st.y * ga[k].y + be[k].y, 0.f);
            o.z = fmaxf((v[k].z - st.x) * st.y * ga[k].z + be[k].z, 0.f);
            o.w = fmaxf((v[k].w - st.x) * st.y * ga[k].w + be[k].w, 0.f);
            *reinterpret_cast<float4*>(xs + r * XP + 4 * c4) = o;
            if (Y && m0 + r < M) *reinterpret_cast<float4*>(ln.y + (m0 + r) * ln.y_cs + ln.y_co + 4 * c4) = o;
        }
    }
}

template <int NH, bool Y>
__global__ void __launch_bounds__(TP) heads_fwd_kernel(const float* __restrict__ x, int cs, int co, const float* __restrict__ Wt,
                                                       const float* __restrict__ bias, float* __restrict__ out_a, int Na,
                                                       float* __restrict__ out_b, long M, int HW, LnIn ln) {
    pdl_enter();
    constexpr int NP = (NH + 3) / 4 * 4;                         // padded to float4
    __shared__ __align__(16) float xs[TP * XP];
    __shared__ float2 st_s;
    if (ln.gamma && threadIdx.x < 32) {                          // the tile lies inside one sample (HW is a multiple of the tile)
        const long b = ((long)blockIdx.x * TP) / HW;
        const float2 st = ln_combine(ln.partial, b, ln.S, ln.eps, threadIdx.x);
        if (threadIdx.x == 0) {
            st_s = st;
            if (((long)blockIdx.x * TP) % HW == 0) ln.stats[b] = st;
        }
    }
    __shared__ __align__(16) float wt[C * NP];                   // W transposed: wt[c][n]
    {   // W rows are contiguous ([n][64]): 128-bit loads, all in flight together with the pixel tile and the bias
        constexpr int NW = (NP * (C / 4) + TP - 1) / TP;
        float4 wv[NW];
#pragma unroll
        for (int k = 0; k < NW; ++k) {
            const int i = threadIdx.x + k * TP, n = i >> 4;
            wv[k] = (i < NP * (C / 4) && n < NH) ? __ldg(reinterpret_cast<const float4*>(Wt) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int k = 0; k < NW; ++k) {
            const int i = threadIdx.x + k * TP, n = i >> 4, c = 4 * (i & 15);
            if (i < NP * (C / 4)) { wt[c * NP + n] = wv[k].x; wt[(c + 1) * NP + n] = wv[k].y; wt[(c + 2) * NP + n] = wv[k].z; wt[(c + 3) * NP + n] = wv[k].w; }
        }
    }
    float2 acc[NP / 2];
#pragma unroll
    for (int j = 0; j < NP / 2; ++j) acc[j] = make_float2(2 * j < NH ? __ldg(bias + 2 * j) : 0.f, 2 * j + 1 < NH ? __ldg(bias + 2 * j + 1) : 0.f);
    const long m0 = (long)blockIdx.x * TP;
    if (ln.gamma) {
        __syncthreads();                                         // st_s
        load_tile_ln<8, Y>(x, cs, co, m0, M, xs, ln, st_s, (m0 % HW) * C);
    } else {
        load_tile<16>(x, cs, co, m0, M, xs);
    }
    __syncthreads();
    const float* xr = xs + threadIdx.x * XP;
#pragma unroll 4
    for (int c4 = 0; c4 < C / 4; ++c4) {
        const float4 xv = *reinterpret_cast<const float4*>(xr + 4 * c4);
        const float xa[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float4* wr = reinterpret_cast<const float4*>(wt + (4 * c4 + k) * NP);
#pragma unroll
            for (int j = 0; j < NP / 4; ++j) {
                const float4 w4 = wr[j];
                acc[2 * j] = ffma2(make_float2(xa[k], xa[k]), make_float2(w4.x, w4.y), acc[2 * j]);
                acc[2 * j + 1] = ffma2(make_float2(xa[k], xa[k]), make_float2(w4.z, w4.w), acc[2 * j + 1]);
            }
        }
    }
    const long m = m0 + threadIdx.x;
    if (m >= M) return;
    const long b = m / HW, p = m - b * HW;
    const int Nb = NH - Na;
#pragma unroll
    for (int n = 0; n < NH; ++n) {
        const float v = (n & 1) ? acc[n >> 1].y : acc[n >> 1].x;
        if (n < Na) out_a[(b * Na + n) * HW + p] = v;
        else out_b[(b * Nb + (n - Na)) * HW + p] = v;
    }
}

// Persistent: CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ...; dW / db partials live in registers across tiles.
// Weight-gradient ownership per thread: 4 channels x NB contiguous heads (n = half * NB + j) x one quarter of the tile's pixels.
template <int NH>
__global__ void __launch_bounds__(TP, 4) heads_bwd_kernel(const float* __restrict__ x, int cs, int co, const float* __restrict__ Wt,
                                                          const float* __restrict__ dy_a, int Na, const float* __restrict__ dy_b,
                                                          float* __restrict__ dx, int dcs, int dco, float* __restrict__ dW,
                                                          float* __restrict__ db, long M, int HW, int ntiles) {
    pdl_enter();
    constexpr int NB = ((NH + 1) / 2 + 3) / 4 * 4;               // heads per thread half, padded to float4 (8 for 14, 16 for 27)
    constexpr int NP = 2 * NB;                                   // dY tile pitch: [pixel][NP], heads >= NH are zero
    extern __shared__ __align__(16) float hsm[];
    float* xs = hsm;                                             // [TP][XP] pixel tile
    float* ds = xs + TP * XP;                                    // [TP][NP] dY tile
    float* dT = ds + TP * NP;                                    // [NH][TP] dY tile, head-major (the d_x phase reads 4 pixels per 128-bit load)
    float* ws = dT + NH * TP;                                    // [NH][C]  W
    for (int i = threadIdx.x; i < NH * C; i += TP) ws[i] = __ldg(Wt + i);
    const int cg = threadIdx.x & 15, half = (threadIdx.x >> 4) & 1, pq = threadIdx.x >> 5;
    float2 aw[NB][2];
    float ab[NB];
#pragma unroll
    for (int j = 0; j < NB; ++j) { aw[j][0] = aw[j][1] = make_float2(0.f, 0.f); ab[j] = 0.f; }
    const int Nb = NH - Na;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long m0 = (long)tile * TP;
        __syncthreads();                                          // previous tile's readers are done
        load_tile<8>(x, cs, co, m0, M, xs);
        {
            const long m = m0 + threadIdx.x;
            const long b = m / HW, p = m - b * HW;
            float v[NP];
#pragma unroll
            for (int n = 0; n < NP; ++n) {
                v[n] = 0.f;
                if (m < M && n < NH) v[n] = n < Na ? __ldg(dy_a + (b * Na + n) * HW + p) : __ldg(dy_b + (b * Nb + (n - Na)) * HW + p);
            }
#pragma unroll
            for (int n4 = 0; n4 < NP / 4; ++n4)
                *reinterpret_cast<float4*>(ds + threadIdx.x * NP + 4 * n4) = make_float4(v[4 * n4], v[4 * n4 + 1], v[4 * n4 + 2], v[4 * n4 + 3]);
#pragma unroll
            for (int n = 0; n < NH; ++n) dT[n * TP + threadIdx.x] = v[n];
        }
        __syncthreads();
        // ---- dW[n][c] += sum_p dY[p][n] x[p][c]   (this thread: 32 pixels, 4 channels, NB heads) -- packed FFMA2, broadcast dY
#pragma unroll 2
        for (int i = 0; i < TP / 4; ++i) {
            const int p = pq * (TP / 4) + i;
            const float4 xv = *reinterpret_cast<const float4*>(xs + p * XP + 4 * cg);
            const float2 x01 = make_float2(xv.x, xv.y), x23 = make_float2(xv.z, xv.w);
            const float4* dr = reinterpret_cast<const float4*>(ds + p * NP + half * NB);
#pragma unroll
            for (int j4 = 0; j4 < NB / 4; ++j4) {
                const float4 d4 = dr[j4];
                const float dd[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int j = 4 * j4 + k;
                    aw[j][0] = ffma2(make_float2(dd[k], dd[k]), x01, aw[j][0]);
                    aw[j][1] = ffma2(make_float2(dd[k], dd[k]), x23, aw[j][1]);
                    if (cg == 0) ab[j] += dd[k];
                }
            }
        }
        // ---- d_x[p][c] = sum_n dY[p][n] W[n][c]: thread = 4 pixels x 16 channels, so one W row quarter (4 x 128 bit) serves 4 pixels
        // (one pixel x 64 channels per thread re-read all of W per pixel: 228 shared-memory loads per thread and tile, now 70)
        {
            const int q = threadIdx.x & 3, pg = threadIdx.x >> 2;
            float2 acc[4][8];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = make_float2(0.f, 0.f);
#pragma unroll
            for (int n = 0; n < NH; ++n) {
                const float4 d4 = *reinterpret_cast<const float4*>(dT + n * TP + 4 * pg);
                const float dd[4] = {d4.x, d4.y, d4.z, d4.w};
                const float4* wr = reinterpret_cast<const float4*>(ws + n * C + 16 * q);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 w4 = wr[j];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        acc[i][2 * j] = ffma2(make_float2(dd[i], dd[i]), make_float2(w4.x, w4.y), acc[i][2 * j]);
                        acc[i][2 * j + 1] = ffma2(make_float2(dd[i], dd[i]), make_float2(w4.z, w4.w), acc[i][2 * j + 1]);
                    }
                }
            }
            __syncthreads();                                      // everyone has finished reading the x tile (weight-gradient phase)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float* xr = xs + (4 * pg + i) * XP + 16 * q;
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    *reinterpret_cast<float4*>(xr + 4 * j) = make_float4(acc[i][2 * j].x, acc[i][2 * j].y, acc[i][2 * j + 1].x, acc[i][2 * j + 1].y);
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < TP * (C / 4); i += TP) {
            const int r = i >> 4, c4 = i & 15;
            if (m0 + r < M) *(reinterpret_cast<float4*>(dx + (m0 + r) * dcs + dco) + c4) = *reinterpret_cast<const float4*>(xs + r * XP + 4 * c4);
        }
    }
    // ---- reduce the four pixel-quarter partials of dW / db inside the CTA, then one atomic per element
    __syncthreads();
    float* red = xs;                                              // [4][NP][C + 1]
    constexpr int RP = C + 1;
#pragma unroll
    for (int j = 0; j < NB; ++j) {
        float* r = red + ((pq * NP) + (half * NB + j)) * RP + 4 * cg;
        r[0] = aw[j][0].x; r[1] = aw[j][0].y; r[2] = aw[j][1].x; r[3] = aw[j][1].y;
        if (cg == 0) red[((pq * NP) + (half * NB + j)) * RP + C] = ab[j];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < NH * RP; i += TP) {
        const int n = i / RP, c = i - n * RP;
        const float v = red[(0 * NP + n) * RP + c] + red[(1 * NP + n) * RP + c] + red[(2 * NP + n) * RP + c] + red[(3 * NP + n) * RP + c];
        if (c < C) atomicAdd(dW + n * C + c, v);
        else atomicAdd(db + n, v);
    }
}

static_assert(4 * 32 * (C + 1) <= TP * XP, "weight-gradient reduction scratch must fit in the pixel tile");

static bool a16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace hd
}  // namespace pivp

using namespace pivp;

extern "C" {

/* x: NHWC rows (stride x_cs, offset x_co, 64 channels); W: [NH][64] (enc7 rows then mask rows, the internal "head" layout);
 * out_a (B,Na,H,W) and out_b (B,NH-Na,H,W) NCHW planes.  NH in {14, 27}; other head counts -> PIVP_EUNSUPPORTED (use the conv path). */
static int heads_fwd_impl(const float* x, int x_cs, int x_co, const float* W, const float* bias, float* out_a, int Na, float* out_b, int NH,
                          int B, int HW, const hd::LnIn& ln, void* stream) {
    PIVP_REQUIRE(x && W && bias && out_a && out_b && B > 0 && HW > 0 && Na > 0 && Na < NH, "heads_fwd: bad argument");
    PIVP_REQUIRE(hd::a16(x) && x_cs % 4 == 0 && x_co % 4 == 0, "heads_fwd: rows must be 16-byte aligned");
    const long M = (long)B * HW;
    const unsigned grid = (unsigned)((M + hd::TP - 1) / hd::TP);
    const bool y = !ln.gamma || ln.y;               // the LayerNorm form with y == NULL: the instantiation that does not write the normalised rows
    if (NH == 14 && y) launch_k(hd::heads_fwd_kernel<14, true>, dim3(grid), dim3(hd::TP), 0, (cudaStream_t)stream, x, x_cs, x_co, W, bias, out_a, Na, out_b, M, HW, ln);
    else if (NH == 27 && y) launch_k(hd::heads_fwd_kernel<27, true>, dim3(grid), dim3(hd::TP), 0, (cudaStream_t)stream, x, x_cs, x_co, W, bias, out_a, Na, out_b, M, HW, ln);
    else if (NH == 14) launch_k(hd::heads_fwd_kernel<14, false>, dim3(grid), dim3(hd::TP), 0, (cudaStream_t)stream, x, x_cs, x_co, W, bias, out_a, Na, out_b, M, HW, ln);
    else if (NH == 27) launch_k(hd::heads_fwd_kernel<27, false>, dim3(grid), dim3(hd::TP), 0, (cudaStream_t)stream, x, x_cs, x_co, W, bias, out_a, Na, out_b, M, HW, ln);
    else { set_error("heads_fwd: %d heads not instantiated (14 or 27)", NH); return PIVP_EUNSUPPORTED; }
    return check_launch("heads_fwd");
}

int pivp_heads_fwd(const float* x, int x_cs, int x_co, const float* W, const float* bias, float* out_a, int Na, float* out_b, int NH,
                   int B, int HW, void* stream) {
    hd::LnIn none;
    memset(&none, 0, sizeof(none));
    return heads_fwd_impl(x, x_cs, x_co, W, bias, out_a, Na, out_b, NH, B, HW, none, stream);
}

/* The heads on relu(LayerNorm(x)) in ONE launch (norm_enc6 + ReLU, train_model.py:601, 698, then enc7 / masks): x = the LayerNorm INPUT (enc6's
 * deconvolution output), partial = the [B][HW*64/4096] (mean, M2) pairs the deconvolution's epilogue wrote (pivp_tc_conv_taps_multi_ln),
 * gamma / beta [HW*64]; y receives the normalised rows (the backward reads them; NULL: not written), stats [B] the (mean, rstd) pairs
 * pivp_layernorm_bwd needs.
 * Replaces pivp_layernorm_fwd(relu | 2) + pivp_heads_fwd.  HW must be a multiple of 128 and HW*64 of 4096. */
int pivp_heads_fwd_ln(const float* x, int x_cs, int x_co, const float* gamma, const float* beta, const float* partial, float eps, float* stats,
                      float* y, int y_cs, int y_co, const float* W, const float* bias, float* out_a, int Na, float* out_b, int NH,
                      int B, int HW, void* stream) {
    PIVP_REQUIRE(gamma && beta && partial && stats, "heads_fwd_ln: null pointer");     // y may be NULL: the normalised rows are then not written
    PIVP_REQUIRE(HW % hd::TP == 0 && ((long)HW * hd::C) % 4096 == 0, "heads_fwd_ln: HW must be a multiple of 128");
    PIVP_REQUIRE(hd::a16(gamma) && hd::a16(beta) && (!y || (hd::a16(y) && y_cs % 4 == 0 && y_co % 4 == 0)), "heads_fwd_ln: rows must be 16-byte aligned");
    hd::LnIn ln{gamma, beta, reinterpret_cast<const float2*>(partial), (int)((long)HW * hd::C / 4096), eps, reinterpret_cast<float2*>(stats), y, y_cs, y_co};
    return heads_fwd_impl(x, x_cs, x_co, W, bias, out_a, Na, out_b, NH, B, HW, ln, stream);
}

/* dx is OVERWRITTEN; dW [NH][64] and db [NH] are ACCUMULATED into (atomics). */
int pivp_heads_bwd(const float* x, int x_cs, int x_co, const float* W, const float* dy_a, int Na, const float* dy_b, int NH,
                   float* dx, int dx_cs, int dx_co, float* dW, float* db, int B, int HW, void* stream) {
    PIVP_REQUIRE(x && W && dy_a && dy_b && dx && dW && db && B > 0 && HW > 0 && Na > 0 && Na < NH, "heads_bwd: bad argument");
    PIVP_REQUIRE(hd::a16(x) && hd::a16(dx) && x_cs % 4 == 0 && x_co % 4 == 0 && dx_cs % 4 == 0 && dx_co % 4 == 0, "heads_bwd: rows must be 16-byte aligned");
    const long M = (long)B * HW;
    const int ntiles = (int)((M + hd::TP - 1) / hd::TP);
    int grid = 148 * 4;
    if (grid > ntiles) grid = ntiles;
    const int NB = ((NH + 1) / 2 + 3) / 4 * 4;
    const size_t smem = sizeof(float) * ((size_t)hd::TP * hd::XP + (size_t)hd::TP * 2 * NB + (size_t)NH * hd::TP + (size_t)NH * hd::C);
    static PerDeviceOnce attr_once;            // the opt-in is per device
    if (attr_once.need()) {
        cudaFuncSetAttribute(hd::heads_bwd_kernel<14>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024);
        cudaFuncSetAttribute(hd::heads_bwd_kernel<27>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024);
    }
    if (NH == 14) launch_k(hd::heads_bwd_kernel<14>, dim3(grid), dim3(hd::TP), smem, (cudaStream_t)stream, x, x_cs, x_co, W, dy_a, Na, dy_b, dx, dx_cs, dx_co, dW, db, M, HW, ntiles);
    else if (NH == 27) launch_k(hd::heads_bwd_kernel<27>, dim3(grid), dim3(hd::TP), smem, (cudaStream_t)stream, x, x_cs, x_co, W, dy_a, Na, dy_b, dx, dx_cs, dx_co, dW, db, M, HW, ntiles);
    else { set_error("heads_bwd: %d heads not instantiated (14 or 27)", NH); return PIVP_EUNSUPPORTED; }
    return check_launch("heads_bwd");
}

}  // extern "C"
