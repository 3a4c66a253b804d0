// Epilogues shared by the tcgen05 convolution kernels (conv_tc.cu, conv_tc_halo.cu): one thread = one accumulator row (TMEM lane).
//   mode 0: D (+bias, ReLU, accumulate) -> fp32 view and / or bf16 view at output row `orow`
//   mode 1: ConvLSTM gates (train_model.py:269-272): bias + sigma/tanh + cell update + h, written for pixel row `m`
#pragma once
#include "tc_common.cuh"

namespace pivp {

__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(tanh_fast(0.5f * x), 0.5f, 0.5f); }

struct TcEpilogue {
    int mode;                    // 0: plain fp32 store (+bias), 1: ConvLSTM gates
    const float* bias;           // [N] (may be null in mode 0)
    float* out; int out_cs, out_co;              // mode 0: D -> out[row(m)*out_cs + out_co + n]  (may be null)
    __nv_bfloat16* out_bf16; int ob_cs, ob_co;   // mode 0: optional bf16 copy (next GEMM's operand), same row mapping
    int relu;                                    // mode 0: ReLU after bias
    int accumulate;                              // mode 0: out += D (fp32 view only)
    int atomic;                                  // mode 0: out += D with vector atomics (split-K CTAs of the halo kernel share an output tile)
    float* gates;                                // mode 1: activated gates [M][N] (saved for backward); bf16 storage when gates_bf16;
                                                 //   null: not stored (the launchers then pick the instantiation without the gate store)
    int gates_bf16;
    float2* ln_partial;                          // per-tile (mean, M2) of the output for the LayerNorm that follows, 4096 values each:
    int ln_S;                                    //   mode 1 (halo kernel): partial[b * ln_S + tile_in_sample * (C / 32) + n_tile];
                                                 //   mode 0 (tap kernel, deconvolution phases): one pair per (tile, phase, 32-column group)
    const float* c_prev; float* c_out;           // [M][C]  (c_prev may be null)
    float* h_out; int h_cs, h_co;                // fp32 h view (next step's xh h-slot)
    __nv_bfloat16* h_bf16; int hb_cs, hb_co;     // bf16 shadow (GEMM operand of the next step)
    __nv_bfloat16* h_t; long h_t_ld;             // optional channel-major bf16 copy  h_t[(hT_co + ch) * h_t_ld + m]  (wgrad operand)
    int hT_co;
    // mode 1, halo kernel with TMA stores only: the LayerNorm that follows the cell (train_model.py:203-208, 596-601) applied in the SAME
    // kernel.  The CTAs of a sample meet at a per-sample arrival counter once their (mean, M2) partials are written; every thread then
    // normalises the h values it still holds in registers.  ln_gamma == null: no fusion (the separate LayerNorm kernel reads ln_partial).
    const float* ln_gamma; const float* ln_beta; // per-element affine in the sample's H*W*C order
    float* ln_y; int ln_y_cs, ln_y_co;           // fp32 output view (the next layer's x slot)
    __nv_bfloat16* ln_yb; int ln_yb_cs, ln_yb_co;   // optional bf16 copy (the next GEMM's operand)
    float2* ln_stats;                            // [B] (mean, rstd) saved for the LayerNorm backward
    unsigned* ln_counter;                        // [B] arrival counters, never reset: every launch adds exactly ln_S per sample
    float ln_eps;
    int C;                                       // LSTM channels (N = 4C)
    float forget_bias;
    int accurate;                                // 1: expf/tanhf, 0: tanh.approx
};

// Gate non-linearities + cell update of 8 channels (train_model.py:269-272): gj/gi/gf/go hold the accumulator on entry and the ACTIVATED
// gates on exit.  ACC is a template parameter on purpose: with a run-time flag inside the element loop ptxas keeps one basic block per
// element (branch, 4 MUFU, branch, MUFU ...) and the eight independent dependency chains run one after the other.
template <bool ACC>
__device__ __forceinline__ void gate_math8(float (&gj)[8], float (&gi)[8], float (&gf)[8], float (&go)[8], const float* cp, const float* bias_s,
                                           int c0, float forget_bias, float (&cn)[8], float (&hn)[8]) {
    // bias one gate at a time (8 transient registers instead of 32 live ones)
    auto add_bias = [&](float (&g)[8], int off, float extra) {
        const float4 b0 = *reinterpret_cast<const float4*>(bias_s + off + c0), b1 = *reinterpret_cast<const float4*>(bias_s + off + c0 + 4);
        g[0] += b0.x + extra; g[1] += b0.y + extra; g[2] += b0.z + extra; g[3] += b0.w + extra;
        g[4] += b1.x + extra; g[5] += b1.y + extra; g[6] += b1.z + extra; g[7] += b1.w + extra;
    };
    add_bias(gj, 0, 0.f); add_bias(gi, 32, 0.f); add_bias(gf, 64, forget_bias); add_bias(go, 96, 0.f);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float j = gj[i], ii = gi[i], f = gf[i], o = go[i];
        if (ACC) { j = tanhf(j); ii = sigmoid_acc(ii); f = sigmoid_acc(f); o = sigmoid_acc(o); }
        else { j = tanh_fast(j); ii = sigmoid_fast(ii); f = sigmoid_fast(f); o = sigmoid_fast(o); }
        cn[i] = cp[i] * f + ii * j;
        hn[i] = (ACC ? tanhf(cn[i]) : tanh_fast(cn[i])) * o;
        gj[i] = j; gi[i] = ii; gf[i] = f; go[i] = o;
    }
}

__device__ __forceinline__ uint4 pack8_bf16(const float (&v)[8]) {
    __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(v[4], v[5]), p3 = __floats2bfloat162_rn(v[6], v[7]);
    uint4 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
    pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
    return pk;
}

// Plain (mode 0) epilogue, staged: tcgen05.ld hands every thread one accumulator ROW, but the output is row-major, so storing
// straight from registers writes 16-byte pieces of 32 different rows per instruction.  The rows go through shared memory instead
// (`stage`: [128][NP] floats, NP = BN + 4: conflict-free for 128-bit accesses; the operand ring is dead once the accumulator is complete)
// and leave as whole rows: consecutive lanes write consecutive 16 bytes.  `nthr` threads (thread index `t`, named barrier `bar_id`) own
// the tile; this thread converts columns [cbeg, cend) of accumulator row `row`, whose output row is `orow` (kept in a 128-entry table
// behind the staged tile, so the write-out loop does no index arithmetic beyond one 32-bit division).  Needs 128*(BN+4)*4 + 1024 bytes.
__device__ __forceinline__ void tc_epilogue_staged(const TcEpilogue& ep, uint32_t trow, float* stage, int row, long orow, int cbeg, int cend, int n0,
                                                   int BN, const float* bias_s, int t, int nthr, int bar_id) {
    const int NP = BN + 4;
    long* rowmap = reinterpret_cast<long*>(stage + 128 * NP);
    rowmap[row] = orow;
    for (int c0 = cbeg; c0 < cend; c0 += 8) {
        float v[8];
        tc_ld8(trow + (uint32_t)c0, v);
        tc_ld_wait();
        if (ep.bias) {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] += bias_s[c0 + i];
        }
        if (ep.relu) {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
        }
        float* s = stage + row * NP + c0;
        *reinterpret_cast<float4*>(s) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(s + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
    asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(nthr) : "memory");
    const int q4 = BN >> 2, total = 128 * q4;
    for (int e = t; e < total; e += nthr) {
        const int r = e / q4, c = 4 * (e - r * q4);
        float4 v = *reinterpret_cast<const float4*>(stage + r * NP + c);
        const long orow = rowmap[r];
        if (ep.out) {
            float* dst = ep.out + orow * ep.out_cs + ep.out_co + n0 + c;
            if (ep.atomic) {
                atomicAdd(reinterpret_cast<float4*>(dst), v);
            } else {
                if (ep.accumulate) {
                    const float4 o = *reinterpret_cast<const float4*>(dst);
                    v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                }
                *reinterpret_cast<float4*>(dst) = v;
            }
        }
        if (ep.out_bf16) {
            __nv_bfloat162 p0 = __floats2bfloat162_rn(v.x, v.y), p1 = __floats2bfloat162_rn(v.z, v.w);
            uint2 pk;
            pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
            *reinterpret_cast<uint2*>(ep.out_bf16 + orow * ep.ob_cs + ep.ob_co + n0 + c) = pk;
        }
    }
}

// trow: TMEM address of this thread's lane at the tile's first column; n0 = first output channel of the tile; bias_s: BN floats in smem
// Mode 0 with the statistics of the LayerNorm that follows (norm_enc6 behind enc6, train_model.py:507/601): bias + store as tc_epilogue_row,
// and for every 32-column group of the tile the warp's exact (mean, M2) over its 32 rows x 32 columns -- per chunk of 8 registers in two
// passes, chunks and lanes merged with Chan's formula -- into red[group * 4 + q] (q = the warp's TMEM lane quarter).  No ReLU, no accumulate.
__device__ __forceinline__ void tc_epilogue_row_ln(const TcEpilogue& ep, uint32_t trow, long orow, int n0, int BN, const float* bias_s,
                                                   float2* red, int q, int lane) {
    for (int g0 = 0; g0 < BN; g0 += 32) {
        float mean = 0.f, m2 = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c0 = g0 + 8 * k;
            float v[8];
            tc_ld8(trow + (uint32_t)c0, v);
            tc_ld_wait();
            if (ep.bias) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] += bias_s[c0 + i];
            }
            if (ep.out) {
                float* dst = ep.out + orow * ep.out_cs + ep.out_co + n0 + c0;
                *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
            }
            if (ep.out_bf16) *reinterpret_cast<uint4*>(ep.out_bf16 + orow * ep.ob_cs + ep.ob_co + n0 + c0) = pack8_bf16(v);
            const float cm = (((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]))) * 0.125f;
            float c2 = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float d = v[i] - cm; c2 = fmaf(d, d, c2); }
            const float d = cm - mean;                       // Chan: 8k values so far + 8 new ones
            mean += d * (1.f / (float)(k + 1));
            m2 += c2 + d * d * (8.f * (float)k / (float)(k + 1));
        }
        float cnt = 32.f;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {                   // equal counts on both sides of every merge
            const float mo = __shfl_xor_sync(0xffffffffu, mean, o), m2o = __shfl_xor_sync(0xffffffffu, m2, o);
            const float d = mo - mean;
            m2 = (m2 + m2o) + d * d * (cnt * 0.5f);
            mean = 0.5f * (mean + mo);
            cnt *= 2.f;
        }
        if (lane == 0) red[(g0 >> 5) * 4 + q] = make_float2(mean, m2);
    }
}

// Mode 0 through shared memory for a TMA store: the row's BN fp32 values (+bias, ReLU) go into BN / 32 staging tiles of 128 rows x 128 B laid
// out as the output tensor map's boxes (128-byte swizzle), one 16 KB tile per 32 columns; a per-thread global store would put 16 bytes into each of
// 32 different cache lines per instruction.  STATS: also the (mean, M2) pairs of tc_epilogue_row_ln (computed before the ReLU is applied: not combined).
// stage_b != 0: also the bf16 copy, BN / 32 tiles of 128 rows x 64 B (64-byte swizzle) at stage_b.
template <bool STATS>
__device__ __forceinline__ void tc_epilogue_row_stage(const TcEpilogue& ep, uint32_t trow, int BN, const float* bias_s, uint32_t stage, int row,
                                                      float2* red, int q, int lane, uint32_t stage_b = 0) {
    const uint32_t r128 = (uint32_t)row * 128u, rsw = (uint32_t)(row & 7);
    const uint32_t r64 = (uint32_t)row * 64u, rsw64 = (uint32_t)((row >> 1) & 3);
    for (int g0 = 0; g0 < BN; g0 += 32) {
        float mean = 0.f, m2 = 0.f;
        const uint32_t sb = stage + (uint32_t)(g0 >> 5) * 16384u + r128;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c0 = g0 + 8 * k;
            float v[8];
            tc_ld8(trow + (uint32_t)c0, v);
            tc_ld_wait();
            if (ep.bias) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] += bias_s[c0 + i];
            }
            if (STATS) {
                const float cm = (((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]))) * 0.125f;
                float c2 = 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) { const float d = v[i] - cm; c2 = fmaf(d, d, c2); }
                const float d = cm - mean;
                mean += d * (1.f / (float)(k + 1));
                m2 += c2 + d * d * (8.f * (float)k / (float)(k + 1));
            } else if (ep.relu) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
            }
            st_shared_v4(sb + (((uint32_t)(2 * k) ^ rsw) << 4), __float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
            st_shared_v4(sb + (((uint32_t)(2 * k + 1) ^ rsw) << 4), __float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7]));
            if (stage_b) {
                const uint4 pk = pack8_bf16(v);
                st_shared_v4(stage_b + (uint32_t)(g0 >> 5) * 8192u + r64 + (((uint32_t)k ^ rsw64) << 4), pk.x, pk.y, pk.z, pk.w);
            }
        }
        if (STATS) {
            float cnt = 32.f;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const float mo = __shfl_xor_sync(0xffffffffu, mean, o), m2o = __shfl_xor_sync(0xffffffffu, m2, o);
                const float d = mo - mean;
                m2 = (m2 + m2o) + d * d * (cnt * 0.5f);
                mean = 0.5f * (mean + mo);
                cnt *= 2.f;
            }
            if (lane == 0) red[(g0 >> 5) * 4 + q] = make_float2(mean, m2);
        }
    }
}

// GATES = false (mode 1, pivp_tc_conv5x5 flags bit 2): the activated gates are not stored (forward-only prediction has no reader for them).
// Each thread reads c_prev for exactly the (pixel, channel) elements it later writes to c_out, so c_prev may alias c_out.
template <bool GATES = true>
__device__ __forceinline__ void tc_epilogue_row(const TcEpilogue& ep, uint32_t trow, long m, long orow, int n0, int BN, int n_tile,
                                                const float* bias_s) {
    if (ep.mode == 0) {
        for (int c0 = 0; c0 < BN; c0 += 8) {
            float v[8];
            tc_ld8(trow + (uint32_t)c0, v);
            tc_ld_wait();
            if (ep.bias) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] += bias_s[c0 + i];
            }
            if (ep.relu) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
            }
            if (ep.out) {
                float* dst = ep.out + orow * ep.out_cs + ep.out_co + n0 + c0;
                if (ep.atomic) {
                    atomicAdd(reinterpret_cast<float4*>(dst), make_float4(v[0], v[1], v[2], v[3]));
                    atomicAdd(reinterpret_cast<float4*>(dst + 4), make_float4(v[4], v[5], v[6], v[7]));
                    continue;
                }
                if (ep.accumulate) {
                    const float4 o0 = *reinterpret_cast<const float4*>(dst), o1 = *reinterpret_cast<const float4*>(dst + 4);
                    v[0] += o0.x; v[1] += o0.y; v[2] += o0.z; v[3] += o0.w; v[4] += o1.x; v[5] += o1.y; v[6] += o1.z; v[7] += o1.w;
                }
                *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
            }
            if (ep.out_bf16) {
                __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
                __nv_bfloat162 p2 = __floats2bfloat162_rn(v[4], v[5]), p3 = __floats2bfloat162_rn(v[6], v[7]);
                uint4 pk;
                pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
                pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
                *reinterpret_cast<uint4*>(ep.out_bf16 + orow * ep.ob_cs + ep.ob_co + n0 + c0) = pk;
            }
        }
    } else {
        // tile = 32 channels x 4 gates: columns [0,32) j, [32,64) i, [64,96) f, [96,128) o
        const int ch0 = n_tile * 32;
        for (int c0 = 0; c0 < 32; c0 += 8) {
            float gj[8], gi[8], gf[8], go[8];
            tc_ld8(trow + (uint32_t)(c0), gj);
            tc_ld8(trow + (uint32_t)(32 + c0), gi);
            tc_ld8(trow + (uint32_t)(64 + c0), gf);
            tc_ld8(trow + (uint32_t)(96 + c0), go);
            tc_ld_wait();
            float cp[8], cn[8], hn[8];
            if (ep.c_prev) {
                const float4 a = *reinterpret_cast<const float4*>(ep.c_prev + m * ep.C + ch0 + c0);
                const float4 b = *reinterpret_cast<const float4*>(ep.c_prev + m * ep.C + ch0 + c0 + 4);
                cp[0] = a.x; cp[1] = a.y; cp[2] = a.z; cp[3] = a.w; cp[4] = b.x; cp[5] = b.y; cp[6] = b.z; cp[7] = b.w;
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) cp[i] = 0.f;
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float j = gj[i] + bias_s[c0 + i], ii = gi[i] + bias_s[32 + c0 + i];
                float f = gf[i] + bias_s[64 + c0 + i] + ep.forget_bias, o = go[i] + bias_s[96 + c0 + i];
                if (ep.accurate) { j = tanhf(j); ii = sigmoid_acc(ii); f = sigmoid_acc(f); o = sigmoid_acc(o); }
                else { j = tanh_fast(j); ii = sigmoid_fast(ii); f = sigmoid_fast(f); o = sigmoid_fast(o); }
                cn[i] = cp[i] * f + ii * j;
                hn[i] = (ep.accurate ? tanhf(cn[i]) : tanh_fast(cn[i])) * o;
                gj[i] = j; gi[i] = ii; gf[i] = f; go[i] = o;
            }
            if (!GATES) {
            } else if (ep.gates_bf16) {
                __nv_bfloat16* gb = reinterpret_cast<__nv_bfloat16*>(ep.gates) + m * (4 * ep.C) + n0 + c0;
                *reinterpret_cast<uint4*>(gb) = pack8_bf16(gj);
                *reinterpret_cast<uint4*>(gb + 32) = pack8_bf16(gi);
                *reinterpret_cast<uint4*>(gb + 64) = pack8_bf16(gf);
                *reinterpret_cast<uint4*>(gb + 96) = pack8_bf16(go);
            } else {
                float* gp = ep.gates + m * (4 * ep.C) + n0 + c0;
                *reinterpret_cast<float4*>(gp) = make_float4(gj[0], gj[1], gj[2], gj[3]);
                *reinterpret_cast<float4*>(gp + 4) = make_float4(gj[4], gj[5], gj[6], gj[7]);
                *reinterpret_cast<float4*>(gp + 32) = make_float4(gi[0], gi[1], gi[2], gi[3]);
                *reinterpret_cast<float4*>(gp + 36) = make_float4(gi[4], gi[5], gi[6], gi[7]);
                *reinterpret_cast<float4*>(gp + 64) = make_float4(gf[0], gf[1], gf[2], gf[3]);
                *reinterpret_cast<float4*>(gp + 68) = make_float4(gf[4], gf[5], gf[6], gf[7]);
                *reinterpret_cast<float4*>(gp + 96) = make_float4(go[0], go[1], go[2], go[3]);
                *reinterpret_cast<float4*>(gp + 100) = make_float4(go[4], go[5], go[6], go[7]);
            }
            float* cdst = ep.c_out + m * ep.C + ch0 + c0;
            *reinterpret_cast<float4*>(cdst) = make_float4(cn[0], cn[1], cn[2], cn[3]);
            *reinterpret_cast<float4*>(cdst + 4) = make_float4(cn[4], cn[5], cn[6], cn[7]);
            float* hdst = ep.h_out + m * ep.h_cs + ep.h_co + ch0 + c0;
            *reinterpret_cast<float4*>(hdst) = make_float4(hn[0], hn[1], hn[2], hn[3]);
            *reinterpret_cast<float4*>(hdst + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
            if (ep.h_bf16) {
                __nv_bfloat162 p0 = __floats2bfloat162_rn(hn[0], hn[1]), p1 = __floats2bfloat162_rn(hn[2], hn[3]);
                __nv_bfloat162 p2 = __floats2bfloat162_rn(hn[4], hn[5]), p3 = __floats2bfloat162_rn(hn[6], hn[7]);
                uint4 pk;
                pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
                pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
                *reinterpret_cast<uint4*>(ep.h_bf16 + m * ep.hb_cs + ep.hb_co + ch0 + c0) = pk;
            }
            if (ep.h_t) {
#pragma unroll
                for (int i = 0; i < 8; ++i) ep.h_t[(long)(ep.hT_co + ch0 + c0 + i) * ep.h_t_ld + m] = __float2bfloat16(hn[i]);
            }
        }
    }
}

}  // namespace pivp
