// Bandwidth-bound pieces of the training step over NHWC views / NCHW planes:
// ConvLSTM gate math (train_model.py:269-272), LayerNormalizationConv2D (:203-208) fwd/bwd,
// ReLU backward (:698), layout packing, the state predictor (:676,730-731) with the smear (:563-565),
// Linear layers (:321-322,457-466), MSE (:741,751), scheduled-sampling select (:73-122) and Adam (A.8).
#include "common.cuh"

namespace pivp {

// ----------------------------------------------------------------------------- ConvLSTM gates
// Gate buffer layout: row m holds 4*C values ordered [block of 32 channels][gate j,i,f,o][32 channels].
__device__ __forceinline__ int gate_col(int ch, int gate) { return (ch >> 5) * 128 + gate * 32 + (ch & 31); }

// c_prev may alias c_out (the cell state updated in place): each thread reads c_prev[idx] once, before it writes c_out[idx], and no other
// thread touches element idx -- hence no __restrict__ on those two.
__global__ void lstm_gates_fwd_kernel(float* __restrict__ gates, const float* c_prev, float* c_out,
                                      View h_out, __nv_bfloat16* __restrict__ h_bf16, int hb_cs, int hb_co,
                                      long M, int C, float forget_bias) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * C) return;
    const long m = idx / C;
    const int ch = (int)(idx - m * C);
    float* g = gates + m * 4 * C;
    const float j = tanhf(g[gate_col(ch, 0)]);
    const float i = sigmoid_acc(g[gate_col(ch, 1)]);
    const float f = sigmoid_acc(g[gate_col(ch, 2)] + forget_bias);
    const float o = sigmoid_acc(g[gate_col(ch, 3)]);
    const float cp = c_prev ? c_prev[idx] : 0.f;
    const float c = cp * f + i * j;
    const float h = tanhf(c) * o;
    g[gate_col(ch, 0)] = j; g[gate_col(ch, 1)] = i; g[gate_col(ch, 2)] = f; g[gate_col(ch, 3)] = o;
    c_out[idx] = c;
    h_out.p[m * h_out.cs + h_out.co + ch] = h;
    if (h_bf16) h_bf16[m * hb_cs + hb_co + ch] = __float2bfloat16(h);
}

// dh = dh_a[m][ch] (+ dh_b view), dc_next (nullable) -> d(pre-activations) written over the saved gates, dc_prev over dc.
__global__ void lstm_gates_bwd_kernel(float* __restrict__ gates, const float* __restrict__ c_prev, const float* __restrict__ c_cur,
                                      const float* __restrict__ dh_a, CView dh_b, float* __restrict__ dc, int dc_valid,
                                      __nv_bfloat16* __restrict__ dg_bf16, long M, int C) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * C) return;
    const long m = idx / C;
    const int ch = (int)(idx - m * C);
    float* g = gates + m * 4 * C;
    const float j = g[gate_col(ch, 0)], i = g[gate_col(ch, 1)], f = g[gate_col(ch, 2)], o = g[gate_col(ch, 3)];
    float dh = dh_a ? dh_a[idx] : 0.f;
    if (dh_b.p) dh += dh_b.p[m * dh_b.cs + dh_b.co + ch];
    const float tc = tanhf(c_cur[idx]);
    const float d_o = dh * tc * o * (1.f - o);
    float dcv = dh * o * (1.f - tc * tc);
    if (dc_valid) dcv += dc[idx];
    const float cp = c_prev ? c_prev[idx] : 0.f;
    const float d_f = dcv * cp * f * (1.f - f);
    const float d_i = dcv * j * i * (1.f - i);
    const float d_j = dcv * i * (1.f - j * j);
    dc[idx] = dcv * f;
    g[gate_col(ch, 0)] = d_j; g[gate_col(ch, 1)] = d_i; g[gate_col(ch, 2)] = d_f; g[gate_col(ch, 3)] = d_o;
    if (dg_bf16) {
        __nv_bfloat16* gb = dg_bf16 + m * 4 * C;
        gb[gate_col(ch, 0)] = __float2bfloat16(d_j); gb[gate_col(ch, 1)] = __float2bfloat16(d_i);
        gb[gate_col(ch, 2)] = __float2bfloat16(d_f); gb[gate_col(ch, 3)] = __float2bfloat16(d_o);
    }
}

// bf16 gate storage (tensor-core mode): activated gates bf16 in, gate pre-activation gradients bf16 out (the tcgen05 input-gradient and
// weight-gradient GEMMs only ever read the bf16 copy).  One thread = 8 channels of one pixel: four 16-byte gate loads / stores.
__device__ __forceinline__ void unpack8(const uint4& u, float (&v)[8]) {
    const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) { const float2 f = __bfloat1622float2(p[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
    uint4 u;
    __nv_bfloat162* p = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    return u;
}
__global__ void __launch_bounds__(256) lstm_gates_bwd_bf16_kernel(const __nv_bfloat16* __restrict__ gates, const float* __restrict__ c_prev,
                                                                  const float* __restrict__ c_cur, const float* __restrict__ dh_a, CView dh_b,
                                                                  float* __restrict__ dc, int dc_valid, __nv_bfloat16* __restrict__ dg,
                                                                  long M, int C) {
    pdl_enter();
    const int c8 = C >> 3;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * c8) return;
    const long m = idx / c8;
    const int ch = (int)(idx - m * c8) * 8;
    const long e = m * C + ch;
    const __nv_bfloat16* g = gates + m * 4 * C + gate_col(ch, 0);
    float j[8], i[8], f[8], o[8];
    unpack8(*reinterpret_cast<const uint4*>(g), j);
    unpack8(*reinterpret_cast<const uint4*>(g + 32), i);
    unpack8(*reinterpret_cast<const uint4*>(g + 64), f);
    unpack8(*reinterpret_cast<const uint4*>(g + 96), o);
    float dh[8], cc[8], cp[8], dcn[8];
    auto ld8 = [](const float* p, float (&v)[8]) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    };
    if (dh_a) ld8(dh_a + e, dh);
    else {
#pragma unroll
        for (int k = 0; k < 8; ++k) dh[k] = 0.f;
    }
    if (dh_b.p) {
        float t[8];
        ld8(dh_b.p + m * dh_b.cs + dh_b.co + ch, t);
#pragma unroll
        for (int k = 0; k < 8; ++k) dh[k] += t[k];
    }
    ld8(c_cur + e, cc);
    if (c_prev) ld8(c_prev + e, cp);
    else {
#pragma unroll
        for (int k = 0; k < 8; ++k) cp[k] = 0.f;
    }
    if (dc_valid) ld8(dc + e, dcn);
    else {
#pragma unroll
        for (int k = 0; k < 8; ++k) dcn[k] = 0.f;
    }
    float dj[8], di[8], df[8], dout[8], dcp[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float tc = tanhf(cc[k]);
        dout[k] = dh[k] * tc * o[k] * (1.f - o[k]);
        const float dcv = dh[k] * o[k] * (1.f - tc * tc) + dcn[k];
        df[k] = dcv * cp[k] * f[k] * (1.f - f[k]);
        di[k] = dcv * j[k] * i[k] * (1.f - i[k]);
        dj[k] = dcv * i[k] * (1.f - j[k] * j[k]);
        dcp[k] = dcv * f[k];
    }
    *reinterpret_cast<float4*>(dc + e) = make_float4(dcp[0], dcp[1], dcp[2], dcp[3]);
    *reinterpret_cast<float4*>(dc + e + 4) = make_float4(dcp[4], dcp[5], dcp[6], dcp[7]);
    __nv_bfloat16* d = dg + m * 4 * C + gate_col(ch, 0);
    *reinterpret_cast<uint4*>(d) = pack8(dj);
    *reinterpret_cast<uint4*>(d + 32) = pack8(di);
    *reinterpret_cast<uint4*>(d + 64) = pack8(df);
    *reinterpret_cast<uint4*>(d + 96) = pack8(dout);
}

// ----------------------------------------------------------------------------- LayerNorm over (H*W*C) per sample
constexpr int LN_T = 256, LN_E = 16;        // a stats CTA keeps LN_T*LN_E elements in registers

__device__ __forceinline__ long ln_addr(const CView& v, long b, int HW, int C, int e) {
    const int pix = e / C, ch = e - pix * C;
    return (b * HW + pix) * v.cs + v.co + ch;
}

__global__ void __launch_bounds__(LN_T) ln_stats_kernel(CView x, int n, int C, int chunk, float2* __restrict__ partial) {
    pdl_enter();
    __shared__ float red[32];
    const int s = blockIdx.x, S = gridDim.x;
    const long b = blockIdx.y;
    const int HW = n / C;
    const int e0 = s * chunk, e1 = min(n, e0 + chunk);
    float v[LN_E];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < LN_E; ++i) {
        const int e = e0 + i * LN_T + threadIdx.x;
        v[i] = (e < e1) ? __ldg(x.p + ln_addr(x, b, HW, C, e)) : 0.f;
        sum += v[i];
    }
    const float cnt = (float)(e1 - e0);
    const float mean = block_sum(sum, red) / cnt;
    float m2 = 0.f;
#pragma unroll
    for (int i = 0; i < LN_E; ++i) {
        const int e = e0 + i * LN_T + threadIdx.x;
        const float d = v[i] - mean;
        if (e < e1) m2 += d * d;
    }
    m2 = block_sum(m2, red);
    if (threadIdx.x == 0) partial[b * S + s] = make_float2(mean, m2);
}

__device__ __forceinline__ float2 ln_combine(const float2* __restrict__ partial, long b, int S, int n, int chunk, float eps) {
    float mu = 0.f;
    for (int s = 0; s < S; ++s) {
        const float cnt = (float)(min(n, (s + 1) * chunk) - s * chunk);
        mu += partial[b * S + s].x * cnt;
    }
    mu /= (float)n;
    float m2 = 0.f;
    for (int s = 0; s < S; ++s) {
        const float cnt = (float)(min(n, (s + 1) * chunk) - s * chunk);
        const float2 p = partial[b * S + s];
        const float d = p.x - mu;
        m2 += p.y + cnt * d * d;
    }
    return make_float2(mu, 1.f / sqrtf(m2 / (float)n + eps));
}

__global__ void __launch_bounds__(LN_T) ln_apply_kernel(CView x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        int n, int C, const float2* __restrict__ partial, int S, int chunk, float eps,
                                                        View y, View y2, __nv_bfloat16* __restrict__ y_bf16, int yb_cs, int yb_co,
                                                        int relu, float2* __restrict__ stats) {
    pdl_enter();
    const long b = blockIdx.y;
    const int HW = n / C;
    const float2 st = ln_combine(partial, b, S, n, chunk, eps);
    if (blockIdx.x == 0 && threadIdx.x == 0) stats[b] = st;
    for (int e = blockIdx.x * LN_T + threadIdx.x; e < n; e += gridDim.x * LN_T) {
        const int pix = e / C, ch = e - pix * C;
        const long row = b * HW + pix;
        float v = (__ldg(x.p + row * x.cs + x.co + ch) - st.x) * st.y * __ldg(gamma + e) + __ldg(beta + e);
        if (relu) v = fmaxf(v, 0.f);
        y.p[row * y.cs + y.co + ch] = v;
        if (y2.p) y2.p[row * y2.cs + y2.co + ch] = v;
        if (y_bf16) y_bf16[row * yb_cs + yb_co + ch] = __float2bfloat16(v);
    }
}

// partial sums of q = g*gamma and q*xhat per sample  (g = (g1+g2) * [y>0] when relu)
__global__ void __launch_bounds__(LN_T) ln_bwd_stats_kernel(CView x, CView g1, CView g2, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, const float2* __restrict__ stats,
                                                            int n, int C, int chunk, int relu, float2* __restrict__ partial) {
    pdl_enter();
    __shared__ float red[32];
    const int s = blockIdx.x, S = gridDim.x;
    const long b = blockIdx.y;
    const int HW = n / C;
    const int e0 = s * chunk, e1 = min(n, e0 + chunk);
    const float2 st = stats[b];
    float s1 = 0.f, s2 = 0.f;
    for (int e = e0 + threadIdx.x; e < e1; e += LN_T) {
        const int pix = e / C, ch = e - pix * C;
        const long row = b * HW + pix;
        const float xh = (__ldg(x.p + row * x.cs + x.co + ch) - st.x) * st.y;
        float g = __ldg(g1.p + row * g1.cs + g1.co + ch);
        if (g2.p) g += __ldg(g2.p + row * g2.cs + g2.co + ch);
        const float ga = __ldg(gamma + e);
        if (relu && xh * ga + __ldg(beta + e) <= 0.f) g = 0.f;
        const float q = g * ga;
        s1 += q;
        s2 += q * xh;
    }
    s1 = block_sum(s1, red);
    s2 = block_sum(s2, red);
    if (threadIdx.x == 0) partial[b * S + s] = make_float2(s1, s2);
}

// thread per element e, loop over the batch: dx, and dgamma[e] += sum_b g*xhat, dbeta[e] += sum_b g
__global__ void __launch_bounds__(LN_T) ln_bwd_apply_kernel(CView x, CView g1, CView g2, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, const float2* __restrict__ stats,
                                                            const float2* __restrict__ partial, int S, int B, int n, int C, int relu,
                                                            View dx, float* __restrict__ dgamma, float* __restrict__ dbeta) {
    pdl_enter();
    extern __shared__ float2 tot[];      // [B] : (mean q, mean q*xhat)
    for (int b = threadIdx.x; b < B; b += LN_T) {
        float a = 0.f, c = 0.f;
        for (int s = 0; s < S; ++s) { const float2 p = partial[(long)b * S + s]; a += p.x; c += p.y; }
        tot[b] = make_float2(a / (float)n, c / (float)n);
    }
    __syncthreads();
    const int e = blockIdx.x * LN_T + threadIdx.x;
    if (e >= n) return;
    const int HW = n / C;
    const int pix = e / C, ch = e - pix * C;
    const float ga = __ldg(gamma + e), be = relu ? __ldg(beta + e) : 0.f;
    float dg = 0.f, db = 0.f;
    for (int b = 0; b < B; ++b) {
        const long row = (long)b * HW + pix;
        const float2 st = stats[b];
        const float xh = (__ldg(x.p + row * x.cs + x.co + ch) - st.x) * st.y;
        float g = __ldg(g1.p + row * g1.cs + g1.co + ch);
        if (g2.p) g += __ldg(g2.p + row * g2.cs + g2.co + ch);
        if (relu && xh * ga + be <= 0.f) g = 0.f;
        dg += g * xh;
        db += g;
        const float2 t2 = tot[b];
        dx.p[row * dx.cs + dx.co + ch] = (g * ga - t2.x - xh * t2.y) * st.y;
    }
    dgamma[e] += dg;
    dbeta[e] += db;
}

// ----------------------------------------------------------------------------- small view kernels
// dst = (ga + gb) * [out > 0]
__global__ void relu_bwd_kernel(CView out, CView ga, CView gb, View dst, long M, int C) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * C) return;
    const long m = idx / C;
    const int ch = (int)(idx - m * C);
    float g = ga.p[m * ga.cs + ga.co + ch];
    if (gb.p) g += gb.p[m * gb.cs + gb.co + ch];
    dst.p[m * dst.cs + dst.co + ch] = out.p[m * out.cs + out.co + ch] > 0.f ? g : 0.f;
}

__global__ void copy_view_kernel(CView src, View dst, __nv_bfloat16* __restrict__ dst_bf16, int db_cs, int db_co, long M, int C) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * C) return;
    const long m = idx / C;
    const int ch = (int)(idx - m * C);
    const float v = src.p[m * src.cs + src.co + ch];
    if (dst.p) dst.p[m * dst.cs + dst.co + ch] = v;
    if (dst_bf16) dst_bf16[m * db_cs + db_co + ch] = __float2bfloat16(v);
}

// 128-bit variants of the three view kernels above: one thread = 4 consecutive channels (C, strides and offsets multiples of 4)
__device__ __forceinline__ uint2 pack4_bf16(float4 v) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<unsigned*>(&lo);
    u.y = *reinterpret_cast<unsigned*>(&hi);
    return u;
}
__global__ void relu_bwd_v4_kernel(CView out, CView ga, CView gb, View dst, long M, int C4) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * C4) return;
    const long m = idx / C4;
    const int ch = (int)(idx - m * C4) * 4;
    float4 g = __ldg(reinterpret_cast<const float4*>(ga.p + m * ga.cs + ga.co + ch));
    if (gb.p) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(gb.p + m * gb.cs + gb.co + ch));
        g.x += t.x; g.y += t.y; g.z += t.z; g.w += t.w;
    }
    const float4 o = __ldg(reinterpret_cast<const float4*>(out.p + m * out.cs + out.co + ch));
    *reinterpret_cast<float4*>(dst.p + m * dst.cs + dst.co + ch) =
        make_float4(o.x > 0.f ? g.x : 0.f, o.y > 0.f ? g.y : 0.f, o.z > 0.f ? g.z : 0.f, o.w > 0.f ? g.w : 0.f);
}
__global__ void copy_view_v4_kernel(CView src, View dst, __nv_bfloat16* __restrict__ dst_bf16, int db_cs, int db_co, long M, int C4) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * C4) return;
    const long m = idx / C4;
    const int ch = (int)(idx - m * C4) * 4;
    const float4 v = __ldg(reinterpret_cast<const float4*>(src.p + m * src.cs + src.co + ch));
    if (dst.p) *reinterpret_cast<float4*>(dst.p + m * dst.cs + dst.co + ch) = v;
    if (dst_bf16) *reinterpret_cast<uint2*>(dst_bf16 + m * db_cs + db_co + ch) = pack4_bf16(v);
}
__global__ void cast_bf16_v4_kernel(CView src, __nv_bfloat16* __restrict__ dst, int d_cs, int d_co, long M, int C4, int H, int W, int s2d, int cblk) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * C4) return;
    const long m = idx / C4;
    const int ch = (int)(idx - m * C4) * 4;
    const float4 v = __ldg(reinterpret_cast<const float4*>(src.p + m * src.cs + src.co + ch));
    long row = m;
    int cc = d_co + ch;
    if (s2d) {
        const long hw = (long)H * W;
        const long b = m / hw;
        const int r = (int)(m - b * hw), y = r / W, x = r - y * W;
        row = (b * (H >> 1) + (y >> 1)) * (W >> 1) + (x >> 1);
        cc += ((y & 1) * 2 + (x & 1)) * cblk;
    }
    *reinterpret_cast<uint2*>(dst + row * d_cs + cc) = pack4_bf16(v);
}
// Fused "gradient hand-over" between a ReLU / LayerNorm backward and a tensor-core transposed-convolution backward:
//   g = ga (+ gb), masked by [out > 0] when `out` is given;  optional fp32 copy;  optional bf16 copy (plain or space-to-depth, the
//   GEMM operand);  optional bias gradient db[c] += sum over rows of g.   One thread owns 4 channels and walks rows (grid-stride), so
//   the column sums cost one 128-bit reduction per block and channel quad instead of a separate colsum kernel.
__global__ void __launch_bounds__(256) grad_handover_kernel(CView out, CView ga, CView gb, View dst, __nv_bfloat16* __restrict__ dst_bf16,
                                                            int b_cs, int b_co, int H, int W, int s2d, int cblk, float* __restrict__ db,
                                                            long M, int C4, int RPB) {
    pdl_enter();
    __shared__ float4 red[256];
    const int c4 = threadIdx.x % C4, ty = threadIdx.x / C4;
    const int ch = c4 * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ty < RPB)
        for (long m = (long)blockIdx.x * RPB + ty; m < M; m += (long)gridDim.x * RPB) {
            float4 g = __ldg(reinterpret_cast<const float4*>(ga.p + m * ga.cs + ga.co + ch));
            if (gb.p) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(gb.p + m * gb.cs + gb.co + ch));
                g.x += t.x; g.y += t.y; g.z += t.z; g.w += t.w;
            }
            if (out.p) {
                const float4 o = __ldg(reinterpret_cast<const float4*>(out.p + m * out.cs + out.co + ch));
                g = make_float4(o.x > 0.f ? g.x : 0.f, o.y > 0.f ? g.y : 0.f, o.z > 0.f ? g.z : 0.f, o.w > 0.f ? g.w : 0.f);
            }
            if (dst.p) *reinterpret_cast<float4*>(dst.p + m * dst.cs + dst.co + ch) = g;
            if (dst_bf16) {
                long row = m;
                int cc = b_co + ch;
                if (s2d) {
                    const long hw = (long)H * W;
                    const long b = m / hw;
                    const int r = (int)(m - b * hw), y = r / W, x = r - y * W;
                    row = (b * (H >> 1) + (y >> 1)) * (W >> 1) + (x >> 1);
                    cc += ((y & 1) * 2 + (x & 1)) * cblk;
                }
                *reinterpret_cast<uint2*>(dst_bf16 + row * b_cs + cc) = pack4_bf16(g);
            }
            acc.x += g.x; acc.y += g.y; acc.z += g.z; acc.w += g.w;
        }
    if (!db) return;
    red[threadIdx.x] = acc;
    __syncthreads();
    if (ty == 0) {
        for (int r = 1; r < RPB; ++r) {
            const float4 t = red[r * C4 + c4];
            acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
        }
        atomicAdd(reinterpret_cast<float4*>(db + ch), acc);
    }
}

static inline bool v4ok(const void* p, int cs, int co) { return !p || (!((uintptr_t)p & 15) && cs % 4 == 0 && co % 4 == 0); }

// planar (B,C,HW) <-> NHWC view rows (b*HW + pix)
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, View dst, int B, int C, int HW) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;     // over B*HW pixels
    if (idx >= (long)B * HW) return;
    const long b = idx / HW;
    const int pix = (int)(idx - b * HW);
    for (int c = 0; c < C; ++c) dst.p[idx * dst.cs + dst.co + c] = __ldg(src + (b * C + c) * HW + pix);
}

__global__ void nhwc_to_nchw_kernel(CView src, float* __restrict__ dst, int B, int C, int HW, int accumulate) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long)B * HW) return;
    const long b = idx / HW;
    const int pix = (int)(idx - b * HW);
    for (int c = 0; c < C; ++c) {
        const float v = src.p[idx * src.cs + src.co + c];
        float* d = dst + (b * C + c) * HW + pix;
        *d = accumulate ? (*d + v) : v;
    }
}

// fp32 NHWC view (rows on a B x H x W grid) -> bf16.  s2d = 0: dst[m][co + ch].  s2d = 1: space-to-depth for the stride-2
// layers: dst row = (b, y/2, x/2) on the half grid, channel = co + ((y&1)*2 + (x&1))*cblk + ch  (cblk >= C, pad stays untouched).
__global__ void cast_bf16_kernel(CView src, __nv_bfloat16* __restrict__ dst, int d_cs, int d_co, long M, int C, int H, int W, int s2d, int cblk) {
    pdl_enter();
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * C) return;
    const long m = idx / C;
    const int ch = (int)(idx - m * C);
    const float v = src.p[m * src.cs + src.co + ch];
    long row = m;
    int cc = d_co + ch;
    if (s2d) {
        const long hw = (long)H * W;
        const long b = m / hw;
        const int r = (int)(m - b * hw), y = r / W, x = r - y * W;
        row = (b * (H >> 1) + (y >> 1)) * (W >> 1) + (x >> 1);
        cc += ((y & 1) * 2 + (x & 1)) * cblk;
    }
    dst[row * d_cs + cc] = __float2bfloat16(v);
}

__global__ void axpy_kernel(const float* __restrict__ x, float* __restrict__ y, long n) {
    pdl_enter();
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] += x[i];
}

// ----------------------------------------------------------------------------- state predictor + smear
// one block per sample: sa = [action, cur]; next = Wc sa + bc; smear sa over npix rows of `smear`.
__global__ void state_fwd_kernel(const float* __restrict__ action, const float* __restrict__ cur, const float* __restrict__ Wc,
                                 const float* __restrict__ bc, float* __restrict__ sa, float* __restrict__ next, View smear, int npix) {
    pdl_enter();
    __shared__ float s[10];
    const int b = blockIdx.x, t = threadIdx.x;
    if (t < 5) s[t] = action[b * 5 + t];
    else if (t < 10) s[t] = cur[b * 5 + t - 5];
    __syncthreads();
    if (t < 10) sa[b * 10 + t] = s[t];
    if (t < 5) {
        float a = bc[t];
#pragma unroll
        for (int k = 0; k < 10; ++k) a = fmaf(Wc[t * 10 + k], s[k], a);
        next[b * 5 + t] = a;
    }
    if (smear.p)
        for (int i = t; i < npix * 10; i += blockDim.x) {
            const int p = i / 10, k = i - p * 10;
            smear.p[((long)b * npix + p) * smear.cs + smear.co + k] = s[k];
        }
}

// one block (64 threads) per sample: d_next = dn_a + dn_b (either may be null); d_sa = Wc^T d_next + smear-sum;
// d_cur_prev = d_sa[5:10]; dWc / dbc accumulated with atomics (50 + 5 values per sample).
__global__ void state_bwd_kernel(const float* __restrict__ dn_a, const float* __restrict__ dn_b, const float* __restrict__ sa,
                                 const float* __restrict__ Wc, CView dsmear, int npix, int B,
                                 float* __restrict__ d_cur_prev, float* __restrict__ dWc, float* __restrict__ dbc) {
    pdl_enter();
    __shared__ float dn[5];
    __shared__ float sm[5][64];
    const int b = blockIdx.x, t = threadIdx.x;
    if (t < 5) dn[t] = (dn_a ? dn_a[b * 5 + t] : 0.f) + (dn_b ? dn_b[b * 5 + t] : 0.f);
    // smear gradient: sum over pixels of channels 5..9 of the state_action slice
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    if (dsmear.p)
        for (int p = t; p < npix; p += 64) {
            const float* row = dsmear.p + ((long)b * npix + p) * dsmear.cs + dsmear.co + 5;
#pragma unroll
            for (int k = 0; k < 5; ++k) acc[k] += row[k];
        }
#pragma unroll
    for (int k = 0; k < 5; ++k) sm[k][t] = acc[k];
    __syncthreads();
    if (t < 5) {
        float d = 0.f;
        for (int i = 0; i < 64; ++i) d += sm[t][i];
#pragma unroll
        for (int j = 0; j < 5; ++j) d = fmaf(Wc[j * 10 + 5 + t], dn[j], d);
        d_cur_prev[b * 5 + t] = d;
        atomicAdd(dbc + t, dn[t]);
    }
    if (t < 50) atomicAdd(dWc + t, dn[t / 10] * sa[b * 10 + t % 10]);
}

// ----------------------------------------------------------------------------- Linear
constexpr int LIN_BB = 8, LIN_NN = 4;
__global__ void __launch_bounds__(256) linear_fwd_kernel(const float* __restrict__ x, int xs, const float* __restrict__ W,
                                                         const float* __restrict__ bias, float* __restrict__ y, int B, int K, int N, int relu) {
    pdl_enter();
    __shared__ float red[32];
    const int n0 = blockIdx.x * LIN_NN, b0 = blockIdx.y * LIN_BB;
    float acc[LIN_NN][LIN_BB] = {};
    for (int k = threadIdx.x; k < K; k += 256) {
        float wv[LIN_NN], xv[LIN_BB];
#pragma unroll
        for (int nn = 0; nn < LIN_NN; ++nn) wv[nn] = (n0 + nn < N) ? __ldg(W + (long)(n0 + nn) * K + k) : 0.f;
#pragma unroll
        for (int bb = 0; bb < LIN_BB; ++bb) xv[bb] = (b0 + bb < B) ? __ldg(x + (long)(b0 + bb) * xs + k) : 0.f;
#pragma unroll
        for (int nn = 0; nn < LIN_NN; ++nn)
#pragma unroll
            for (int bb = 0; bb < LIN_BB; ++bb) acc[nn][bb] = fmaf(wv[nn], xv[bb], acc[nn][bb]);
    }
#pragma unroll
    for (int nn = 0; nn < LIN_NN; ++nn)
#pragma unroll
        for (int bb = 0; bb < LIN_BB; ++bb) {
            const float v = block_sum(acc[nn][bb], red);
            if (threadIdx.x == 0 && b0 + bb < B && n0 + nn < N) {
                float o = v + (bias ? bias[n0 + nn] : 0.f);
                y[(long)(b0 + bb) * N + n0 + nn] = relu ? fmaxf(o, 0.f) : o;
            }
        }
}

// dx[b][k] (+)= sum_n dy[b][n] W[n][k]
__global__ void linear_bwd_dx_kernel(const float* __restrict__ dy, const float* __restrict__ W, float* __restrict__ dx, int dxs,
                                     int B, int K, int N, int accumulate) {
    pdl_enter();
    const int k = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (k >= K) return;
    float a = 0.f;
    for (int n = 0; n < N; ++n) a = fmaf(__ldg(dy + (long)b * N + n), __ldg(W + (long)n * K + k), a);
    float* d = dx + (long)b * dxs + k;
    *d = accumulate ? (*d + a) : a;
}

// dW[n][k] += sum_b dy[b][n] x[b][k];  db[n] += sum_b dy[b][n]
__global__ void linear_bwd_dw_kernel(const float* __restrict__ dy, const float* __restrict__ x, int xs, float* __restrict__ dW,
                                     float* __restrict__ db, int B, int K, int N) {
    pdl_enter();
    const int k = blockIdx.x * blockDim.x + threadIdx.x, n = blockIdx.y;
    if (k < K) {
        float a = 0.f;
        for (int b = 0; b < B; ++b) a = fmaf(__ldg(dy + (long)b * N + n), __ldg(x + (long)b * xs + k), a);
        dW[(long)n * K + k] += a;
    }
    if (db && blockIdx.x == 0 && threadIdx.x == 0) {
        float s = 0.f;
        for (int b = 0; b < B; ++b) s += dy[(long)b * N + n];
        db[n] += s;
    }
}

// ---- wide Linear (K a multiple of 4, batch <= 32, 16-byte aligned rows): the weight matrix is streamed exactly once per kernel.
// All three keep 32 batch rows x one float4 of K per thread in registers.
constexpr int LW_T = 128, LW_B = 32;

// y partial: one WARP per (4 outputs n, K slice): lane l owns the float4 columns k = k0 + 4*(l + 32*i) and keeps 4 x 32 batch
// accumulators; the 32 lane partials of each (n, b) are combined by a warp reduce-scatter (lane b ends with batch row b).
// part[ks][b][n]; a second tiny kernel adds the slices, the bias and the ReLU.
__device__ __forceinline__ float warp_reduce_scatter32(const float (&v)[LW_B], int lane) {
    float a16[16], a8[8], a4[4], a2[2];
    {
        const bool hi = lane & 16;
#pragma unroll
        for (int k = 0; k < 16; ++k) a16[k] = (hi ? v[k + 16] : v[k]) + __shfl_xor_sync(0xffffffffu, hi ? v[k] : v[k + 16], 16);
    }
    {
        const bool hi = lane & 8;
#pragma unroll
        for (int k = 0; k < 8; ++k) a8[k] = (hi ? a16[k + 8] : a16[k]) + __shfl_xor_sync(0xffffffffu, hi ? a16[k] : a16[k + 8], 8);
    }
    {
        const bool hi = lane & 4;
#pragma unroll
        for (int k = 0; k < 4; ++k) a4[k] = (hi ? a8[k + 4] : a8[k]) + __shfl_xor_sync(0xffffffffu, hi ? a8[k] : a8[k + 4], 4);
    }
    {
        const bool hi = lane & 2;
#pragma unroll
        for (int k = 0; k < 2; ++k) a2[k] = (hi ? a4[k + 2] : a4[k]) + __shfl_xor_sync(0xffffffffu, hi ? a4[k] : a4[k + 2], 2);
    }
    const bool hi = lane & 1;
    return (hi ? a2[1] : a2[0]) + __shfl_xor_sync(0xffffffffu, hi ? a2[0] : a2[1], 1);      // lane l holds element l
}

__global__ void __launch_bounds__(128) linear_fwd_wide_kernel(const float* __restrict__ x, int xs, const float* __restrict__ W,
                                                              float* __restrict__ part, int B, int K, int N, int kchunk, int KS) {
    pdl_enter();
    const int lane = threadIdx.x & 31;
    const int wid = blockIdx.x * 4 + (threadIdx.x >> 5);           // warp id over (n group, K slice), K slice fastest
    const int ng = wid / KS, ks = wid - ng * KS;
    const int n0 = ng * 4;
    if (n0 >= N) return;
    const int k0 = ks * kchunk, k1 = min(K, k0 + kchunk);
    float acc[4][LW_B];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int b = 0; b < LW_B; ++b) acc[i][b] = 0.f;
    for (int k = k0 + 4 * lane; k < k1; k += 128) {
        float4 w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = (n0 + i < N) ? __ldg(reinterpret_cast<const float4*>(W + (long)(n0 + i) * K + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int b = 0; b < LW_B; ++b) {
            const float4 xv = b < B ? __ldg(reinterpret_cast<const float4*>(x + (long)b * xs + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                acc[i][b] = fmaf(w[i].x, xv.x, acc[i][b]); acc[i][b] = fmaf(w[i].y, xv.y, acc[i][b]);
                acc[i][b] = fmaf(w[i].z, xv.z, acc[i][b]); acc[i][b] = fmaf(w[i].w, xv.w, acc[i][b]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float v = warp_reduce_scatter32(acc[i], lane);
        if (lane < B && n0 + i < N) part[((long)ks * B + lane) * N + n0 + i] = v;
    }
}
__global__ void linear_fwd_finish_kernel(const float* __restrict__ part, const float* __restrict__ bias, float* __restrict__ y, int BN_, int N,
                                         int KS, int relu) {
    pdl_enter();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= BN_) return;
    float v = bias ? bias[i % N] : 0.f;
    for (int s = 0; s < KS; ++s) v += part[(long)s * BN_ + i];
    y[i] = relu ? fmaxf(v, 0.f) : v;
}

// dx[b][k4] += sum_{n in chunk} dy[b][n] W[n][k4]   grid (K/4/LW_T, n chunks); 128-bit reductions into a zeroed / accumulated dx
__global__ void __launch_bounds__(LW_T) linear_bwd_dx_wide_kernel(const float* __restrict__ dy, const float* __restrict__ W,
                                                                  float* __restrict__ dx, int dxs, int B, int K, int N, int nchunk) {
    pdl_enter();
    extern __shared__ __align__(16) float dys[];                 // [nchunk][LW_B]
    const int na = blockIdx.y * nchunk, nb = min(N, na + nchunk);
    for (int i = threadIdx.x; i < (nb - na) * LW_B; i += LW_T) {
        const int n = i / LW_B, b = i - n * LW_B;
        dys[i] = b < B ? __ldg(dy + (long)b * N + na + n) : 0.f;
    }
    __syncthreads();
    const int k = 4 * (blockIdx.x * LW_T + threadIdx.x);
    if (k >= K) return;
    float4 acc[LW_B];
#pragma unroll
    for (int b = 0; b < LW_B; ++b) acc[b] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
    for (int n = na; n < nb; ++n) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(W + (long)n * K + k));
        const float4* dr = reinterpret_cast<const float4*>(dys + (n - na) * LW_B);
#pragma unroll
        for (int b4 = 0; b4 < LW_B / 4; ++b4) {
            const float4 d = dr[b4];
            const float dd[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float4& a = acc[4 * b4 + j];
                a.x = fmaf(dd[j], w.x, a.x); a.y = fmaf(dd[j], w.y, a.y); a.z = fmaf(dd[j], w.z, a.z); a.w = fmaf(dd[j], w.w, a.w);
            }
        }
    }
#pragma unroll
    for (int b = 0; b < LW_B; ++b)
        if (b < B) atomicAdd(reinterpret_cast<float4*>(dx + (long)b * dxs + k), acc[b]);
}

// dW[n][k4] += sum_b dy[b][n] x[b][k4]; db[n] += sum_b dy[b][n]     grid (K/4/LW_T, n chunks)
__global__ void __launch_bounds__(LW_T) linear_bwd_dw_wide_kernel(const float* __restrict__ dy, const float* __restrict__ x, int xs,
                                                                  float* __restrict__ dW, float* __restrict__ db, int B, int K, int N,
                                                                  int nchunk) {
    pdl_enter();
    extern __shared__ __align__(16) float dys[];                 // [nchunk][LW_B]
    const int na = blockIdx.y * nchunk, nb = min(N, na + nchunk);
    for (int i = threadIdx.x; i < (nb - na) * LW_B; i += LW_T) {
        const int n = i / LW_B, b = i - n * LW_B;
        dys[i] = b < B ? __ldg(dy + (long)b * N + na + n) : 0.f;
    }
    __syncthreads();
    if (db && blockIdx.x == 0)
        for (int n = na + threadIdx.x; n < nb; n += LW_T) {
            float s = 0.f;
            for (int b = 0; b < LW_B; ++b) s += dys[(n - na) * LW_B + b];
            db[n] += s;
        }
    const int k = 4 * (blockIdx.x * LW_T + threadIdx.x);
    if (k >= K) return;
    float4 xv[LW_B];
#pragma unroll
    for (int b = 0; b < LW_B; ++b) xv[b] = b < B ? __ldg(reinterpret_cast<const float4*>(x + (long)b * xs + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int n = na; n < nb; ++n) {
        const float4* dr = reinterpret_cast<const float4*>(dys + (n - na) * LW_B);
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int b4 = 0; b4 < LW_B / 4; ++b4) {
            const float4 d = dr[b4];
            const float dd[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 v = xv[4 * b4 + j];
                a.x = fmaf(dd[j], v.x, a.x); a.y = fmaf(dd[j], v.y, a.y); a.z = fmaf(dd[j], v.z, a.z); a.w = fmaf(dd[j], v.w, a.w);
            }
        }
        float4* dst = reinterpret_cast<float4*>(dW + (long)n * K + k);
        float4 o = *dst;
        o.x += a.x; o.y += a.y; o.z += a.z; o.w += a.w;
        *dst = o;
    }
}

// The same weight gradient over S time steps in ONE pass: dW[n][k4] += sum_s sum_b dy[s][b][n] x[s][b][k4].  The per-step kernel
// re-reads and re-writes all of dW (8 MB for the 8192 -> 250 kernel Linear) every step; here a thread keeps its NCH x 4 partial sums
// in registers across the steps and touches dW once.   grid (K/4/LW_T, n chunks of NCH)
template <int NCH>
__global__ void __launch_bounds__(LW_T) linear_dw_steps_kernel(const float* __restrict__ dy, long dy_ss, const float* __restrict__ x, long x_ss,
                                                               int xs, float* __restrict__ dW, float* __restrict__ db, int S, int B, int K,
                                                               int N) {
    pdl_enter();
    extern __shared__ __align__(16) float dys[];                 // [S][NCH][LW_B]
    const int na = blockIdx.y * NCH;
    for (int i = threadIdx.x; i < S * NCH * LW_B; i += LW_T) {
        const int s = i / (NCH * LW_B), r = i - s * NCH * LW_B, n = r / LW_B, b = r - n * LW_B;
        dys[i] = (b < B && na + n < N) ? __ldg(dy + s * dy_ss + (long)b * N + na + n) : 0.f;
    }
    __syncthreads();
    if (db && blockIdx.x == 0 && threadIdx.x < NCH && na + threadIdx.x < N) {
        float sum = 0.f;
        for (int s = 0; s < S; ++s)
            for (int b = 0; b < LW_B; ++b) sum += dys[(s * NCH + threadIdx.x) * LW_B + b];
        db[na + threadIdx.x] += sum;
    }
    const int k = 4 * (blockIdx.x * LW_T + threadIdx.x);
    if (k >= K) return;
    float4 acc[NCH];
#pragma unroll
    for (int n = 0; n < NCH; ++n) acc[n] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < S; ++s) {
        float4 xv[LW_B];
#pragma unroll
        for (int b = 0; b < LW_B; ++b)
            xv[b] = b < B ? __ldg(reinterpret_cast<const float4*>(x + s * x_ss + (long)b * xs + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int n = 0; n < NCH; ++n) {
            const float4* dr = reinterpret_cast<const float4*>(dys + (s * NCH + n) * LW_B);
#pragma unroll
            for (int b4 = 0; b4 < LW_B / 4; ++b4) {
                const float4 d = dr[b4];
                const float dd[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 v = xv[4 * b4 + j];
                    acc[n].x = fmaf(dd[j], v.x, acc[n].x); acc[n].y = fmaf(dd[j], v.y, acc[n].y);
                    acc[n].z = fmaf(dd[j], v.z, acc[n].z); acc[n].w = fmaf(dd[j], v.w, acc[n].w);
                }
            }
        }
    }
#pragma unroll
    for (int n = 0; n < NCH; ++n)
        if (na + n < N) {
            float4* dst = reinterpret_cast<float4*>(dW + (long)(na + n) * K + k);
            float4 o = *dst;
            o.x += acc[n].x; o.y += acc[n].y; o.z += acc[n].z; o.w += acc[n].w;
            *dst = o;
        }
}

// relu'(y) applied in place to a dense gradient (y is the saved post-ReLU output)
__global__ void relu_mask_kernel(const float* __restrict__ y, float* __restrict__ g, long n) {
    pdl_enter();
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && y[i] <= 0.f) g[i] = 0.f;
}

// ----------------------------------------------------------------------------- loss, select, Adam
// *loss_slot += sum (a-b)^2 ; dgen = gscale * (a-b)   (a = generated, b = target)
__global__ void __launch_bounds__(256) mse_kernel(const float* __restrict__ a, const float* __restrict__ b, long n, float gscale,
                                                  float* __restrict__ dgen, float* __restrict__ loss_slot) {
    pdl_enter();
    __shared__ float red[32];
    float s = 0.f;
    for (long i = (long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long)gridDim.x * 256) {
        const float d = a[i] - b[i];
        s += d * d;
        if (dgen) dgen[i] = gscale * d;
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) atomicAdd(loss_slot, s);
}

// out[b] = take[b] ? gt[b] : gen[b]   (train_model.py:73-122 reduces to this select; SURVEY a2)
__global__ void sched_select_kernel(const float* __restrict__ gt, const float* __restrict__ gen, const int* __restrict__ take,
                                    float* __restrict__ out, int per_sample, long n) {
    pdl_enter();
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = take[i / per_sample] ? gt[i] : gen[i];
}
// the same select, also delivered as NHWC rows (the layout the first convolution reads): out_nhwc[(b * HW + p) * C + c] = out[(b * C + c) * HW + p]
__global__ void sched_select_nhwc_kernel(const float* __restrict__ gt, const float* __restrict__ gen, const int* __restrict__ take,
                                         float* __restrict__ out, float* __restrict__ out_nhwc, int C, int HW, long n) {
    pdl_enter();
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long bc = i / HW;
    const int p = (int)(i - bc * HW);
    const long b = bc / C;
    const int c = (int)(bc - b * C);
    const float v = take[b] ? gt[i] : gen[i];
    out[i] = v;
    out_nhwc[(b * HW + p) * C + c] = v;
}

// Chainer 2.0.1 AdamRule (SURVEY A.8).  step[0] holds t-1 on entry; lr computed once per block.
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, long n, const int* __restrict__ step, float alpha, float b1,
                                                   float b2, float eps, float gscale) {
    pdl_enter();
    __shared__ float lr_s;
    if (threadIdx.x == 0) {
        const double t = (double)(step[0] + 1);
        lr_s = (float)((double)alpha * sqrt(1.0 - pow((double)b2, t)) / (1.0 - pow((double)b1, t)));
    }
    __syncthreads();
    const float lr = lr_s;
    for (long i = (long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long)gridDim.x * 256) {
        const float gi = g[i] * gscale;
        const float mi = m[i] + (1.f - b1) * (gi - m[i]);
        const float vi = v[i] + (1.f - b2) * (gi * gi - v[i]);
        m[i] = mi;
        v[i] = vi;
        p[i] -= lr * mi / (sqrtf(vi) + eps);
    }
}

__global__ void counter_inc_kernel(int* c) {
    pdl_enter(); c[0] += 1; }

__global__ void fill_kernel(float* __restrict__ p, float v, long n) {
    pdl_enter();
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) p[i] = v;
}

static inline unsigned nblk(long n, int t) { return (unsigned)((n + t - 1) / t); }

// 128-bit vectorised LayerNorm kernels (layernorm_vec.cu): 1 = done, 0 = not applicable, < 0 = error
int ln_vec_fwd(const float* x, int x_cs, int x_co, const float* gamma, const float* beta, int B, int HW, int C, float eps,
               float* y, int y_cs, int y_co, float* y2, int y2_cs, int y2_co, void* y_bf16, int yb_cs, int yb_co, int relu,
               float* stats, void* workspace, int S, int chunk, cudaStream_t st, int s2d_w, int s2d_cblk);
int ln_vec_bwd(const float* x, int x_cs, int x_co, const float* g1, int g1_cs, int g1_co, const float* g2, int g2_cs, int g2_co,
               const float* gamma, const float* beta, const float* stats, int B, int HW, int C, int relu, float* dx, int dx_cs,
               int dx_co, float* dgamma, float* dbeta, void* workspace, int S, int chunk, cudaStream_t st, void* gates_bf16,
               const float* c_prev, const float* c_cur, const float* dh_b, int dhb_cs, int dhb_co, float* dc, int dc_valid,
               void* ho_bf16, int ho_cs, int ho_co, int ho_w, int ho_cblk, float* ho_db);

}  // namespace pivp

using namespace pivp;

extern "C" {

int pivp_lstm_gates_fwd(float* gates, const float* c_prev, float* c_out, float* h_out, int h_cs, int h_co,
                        void* h_bf16, int hb_cs, int hb_co, long M, int C, float forget_bias, void* stream) {
    PIVP_REQUIRE(gates && c_out && h_out && M > 0 && C > 0 && C % 32 == 0, "lstm_gates_fwd: bad argument (C must be a multiple of 32)");
    launch_k(lstm_gates_fwd_kernel, dim3(nblk(M * C, 256)), dim3(256), 0, (cudaStream_t)stream, gates, c_prev, c_out, View{h_out, h_cs, h_co},
                                                                              (__nv_bfloat16*)h_bf16, hb_cs, hb_co, M, C, forget_bias);
    return check_launch("lstm_gates_fwd");
}

int pivp_lstm_gates_bwd(float* gates, const float* c_prev, const float* c_cur, const float* dh_a,
                        const float* dh_b, int dhb_cs, int dhb_co, float* dc, int dc_valid, void* dg_bf16,
                        long M, int C, void* stream) {
    PIVP_REQUIRE(gates && c_cur && dc && (dh_a || dh_b) && M > 0 && C % 32 == 0, "lstm_gates_bwd: bad argument");
    launch_k(lstm_gates_bwd_kernel, dim3(nblk(M * C, 256)), dim3(256), 0, (cudaStream_t)stream, gates, c_prev, c_cur, dh_a, CView{dh_b, dhb_cs, dhb_co},
                                                                              dc, dc_valid, (__nv_bfloat16*)dg_bf16, M, C);
    return check_launch("lstm_gates_bwd");
}

/* Tensor-core mode: activated gates stored bf16 (pivp_tc_conv5x5 flags bit 1); writes d(pre-activations) bf16 to dg_bf16 (may alias
 * gates_bf16) and dc in place.  Same math as pivp_lstm_gates_bwd. */
int pivp_lstm_gates_bwd_bf16(const void* gates_bf16, const float* c_prev, const float* c_cur, const float* dh_a,
                             const float* dh_b, int dhb_cs, int dhb_co, float* dc, int dc_valid, void* dg_bf16,
                             long M, int C, void* stream) {
    PIVP_REQUIRE(gates_bf16 && dg_bf16 && c_cur && dc && (dh_a || dh_b) && M > 0 && C % 32 == 0, "lstm_gates_bwd_bf16: bad argument");
    PIVP_REQUIRE(!dh_b || (dhb_cs % 4 == 0 && dhb_co % 4 == 0), "lstm_gates_bwd_bf16: dh view must be 16-byte aligned");
    launch_k(lstm_gates_bwd_bf16_kernel, dim3(nblk(M * (C / 8), 256)), dim3(256), 0, (cudaStream_t)stream, 
        (const __nv_bfloat16*)gates_bf16, c_prev, c_cur, dh_a, CView{dh_b, dhb_cs, dhb_co}, dc, dc_valid, (__nv_bfloat16*)dg_bf16, M, C);
    return check_launch("lstm_gates_bwd_bf16");
}

static int ln_split(int n, int* chunk) {
    int S = (n + LN_T * LN_E - 1) / (LN_T * LN_E);
    *chunk = (n + S - 1) / S;
    return S;
}

size_t pivp_layernorm_workspace_bytes(int B, int n) {
    int chunk;
    const int S = ln_split(n, &chunk);
    return (size_t)B * S * sizeof(float2);
}

int pivp_layernorm_fwd_s2d(const float* x, int x_cs, int x_co, const float* gamma, const float* beta, int B, int HW, int C, float eps,
                           float* y, int y_cs, int y_co, float* y2, int y2_cs, int y2_co, void* y_bf16, int yb_cs, int yb_co,
                           int relu, float* stats, void* workspace, size_t ws_bytes, int s2d_w, int s2d_cblk, void* stream) {
    PIVP_REQUIRE(x && gamma && beta && y && stats && workspace, "layernorm_fwd: null pointer");
    PIVP_REQUIRE(B > 0 && HW > 0 && C > 0, "layernorm_fwd: bad shape");
    const int n = HW * C;
    int chunk;
    const int S = ln_split(n, &chunk);
    PIVP_REQUIRE(ws_bytes >= (size_t)B * S * sizeof(float2), "layernorm_fwd: workspace too small");
    PIVP_REQUIRE(!(relu & 2) || (n % 4096 == 0 && chunk == 4096), "layernorm_fwd: precomputed partials need n to be a multiple of 4096");
    PIVP_REQUIRE(s2d_w == 0 || (y_bf16 && s2d_w > 0 && s2d_w % 2 == 0 && HW % s2d_w == 0 && (HW / s2d_w) % 2 == 0 && s2d_cblk >= C && s2d_cblk % 4 == 0 &&
                                yb_cs >= yb_co + 4 * s2d_cblk),
                 "layernorm_fwd: bad space-to-depth geometry for the bf16 output");
    if (int r = ln_vec_fwd(x, x_cs, x_co, gamma, beta, B, HW, C, eps, y, y_cs, y_co, y2, y2_cs, y2_co, y_bf16, yb_cs, yb_co, relu, stats,
                           workspace, S, chunk, (cudaStream_t)stream, s2d_w, s2d_cblk))
        return r < 0 ? r : PIVP_OK;
    PIVP_REQUIRE(!(relu & 2), "layernorm_fwd: precomputed partials are only supported by the vectorised path");
    PIVP_REQUIRE(!s2d_w, "layernorm_fwd: the space-to-depth bf16 output is only supported by the vectorised path");
    launch_k(ln_stats_kernel, dim3(S, B), dim3(LN_T), 0, (cudaStream_t)stream, CView{x, x_cs, x_co}, n, C, chunk, (float2*)workspace);
    if (int e = check_launch("layernorm_fwd(stats)")) return e;
    int gx = (n + LN_T * 4 - 1) / (LN_T * 4);
    launch_k(ln_apply_kernel, dim3(gx, B), dim3(LN_T), 0, (cudaStream_t)stream, CView{x, x_cs, x_co}, gamma, beta, n, C, (const float2*)workspace, S, chunk,
                                                                     eps, View{y, y_cs, y_co}, View{y2, y2_cs, y2_co}, (__nv_bfloat16*)y_bf16,
                                                                     yb_cs, yb_co, relu, (float2*)stats);
    return check_launch("layernorm_fwd(apply)");
}

int pivp_layernorm_fwd(const float* x, int x_cs, int x_co, const float* gamma, const float* beta, int B, int HW, int C, float eps,
                       float* y, int y_cs, int y_co, float* y2, int y2_cs, int y2_co, void* y_bf16, int yb_cs, int yb_co,
                       int relu, float* stats, void* workspace, size_t ws_bytes, void* stream) {
    return pivp_layernorm_fwd_s2d(x, x_cs, x_co, gamma, beta, B, HW, C, eps, y, y_cs, y_co, y2, y2_cs, y2_co, y_bf16, yb_cs, yb_co, relu, stats,
                                  workspace, ws_bytes, 0, 0, stream);
}

int pivp_layernorm_bwd_handover(const float* x, int x_cs, int x_co, const float* g1, int g1_cs, int g1_co, const float* g2, int g2_cs, int g2_co,
                                const float* gamma, const float* beta, const float* stats, int B, int HW, int C, int relu,
                                float* dx, int dx_cs, int dx_co, float* dgamma, float* dbeta, void* workspace, size_t ws_bytes,
                                void* ho_bf16, int ho_cs, int ho_co, int ho_w, int ho_cblk, float* ho_db, void* stream) {
    PIVP_REQUIRE(x && g1 && gamma && beta && stats && (dx || ho_bf16) && dgamma && dbeta && workspace, "layernorm_bwd: null pointer");
    PIVP_REQUIRE(!ho_bf16 || (ho_db && ho_w > 0 && ho_w % 2 == 0 && HW % ho_w == 0 && (HW / ho_w) % 2 == 0 && ho_cblk >= C && ho_cblk % 4 == 0 &&
                              ho_cs % 4 == 0 && ho_co % 4 == 0 && ho_cs >= ho_co + 4 * ho_cblk && !((uintptr_t)ho_bf16 & 7) && !((uintptr_t)ho_db & 15)),
                 "layernorm_bwd: bad hand-over geometry");
    const int n = HW * C;
    int chunk;
    const int S = ln_split(n, &chunk);
    PIVP_REQUIRE(ws_bytes >= (size_t)B * S * sizeof(float2), "layernorm_bwd: workspace too small");
    PIVP_REQUIRE(B <= 4096, "layernorm_bwd: batch too large for the shared-memory totals");
    if (int r = ln_vec_bwd(x, x_cs, x_co, g1, g1_cs, g1_co, g2, g2_cs, g2_co, gamma, beta, stats, B, HW, C, relu, dx, dx_cs, dx_co, dgamma,
                           dbeta, workspace, S, chunk, (cudaStream_t)stream, nullptr, nullptr, nullptr, nullptr, 0, 0, nullptr, 0, ho_bf16, ho_cs, ho_co, ho_w,
                           ho_cblk, ho_db))
        return r < 0 ? r : PIVP_OK;
    PIVP_REQUIRE(!ho_bf16, "layernorm_bwd: the hand-over output needs the vectorised path (16-byte aligned views, C a multiple of 4 dividing 512)");
    launch_k(ln_bwd_stats_kernel, dim3(S, B), dim3(LN_T), 0, (cudaStream_t)stream, CView{x, x_cs, x_co}, CView{g1, g1_cs, g1_co}, CView{g2, g2_cs, g2_co},
                                                                        gamma, beta, (const float2*)stats, n, C, chunk, relu, (float2*)workspace);
    if (int e = check_launch("layernorm_bwd(stats)")) return e;
    launch_k(ln_bwd_apply_kernel, dim3(nblk(n, LN_T)), dim3(LN_T), (size_t)B * sizeof(float2), (cudaStream_t)stream, 
        CView{x, x_cs, x_co}, CView{g1, g1_cs, g1_co}, CView{g2, g2_cs, g2_co}, gamma, beta, (const float2*)stats,
        (const float2*)workspace, S, B, n, C, relu, View{dx, dx_cs, dx_co}, dgamma, dbeta);
    return check_launch("layernorm_bwd(apply)");
}

int pivp_layernorm_bwd(const float* x, int x_cs, int x_co, const float* g1, int g1_cs, int g1_co, const float* g2, int g2_cs, int g2_co,
                       const float* gamma, const float* beta, const float* stats, int B, int HW, int C, int relu,
                       float* dx, int dx_cs, int dx_co, float* dgamma, float* dbeta, void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(dx, "layernorm_bwd: null pointer");
    return pivp_layernorm_bwd_handover(x, x_cs, x_co, g1, g1_cs, g1_co, g2, g2_cs, g2_co, gamma, beta, stats, B, HW, C, relu, dx, dx_cs, dx_co, dgamma,
                                       dbeta, workspace, ws_bytes, nullptr, 0, 0, 0, 0, nullptr, stream);
}

/* LayerNorm backward of a ConvLSTM output h_t fused with the gate backward of that layer (tensor-core mode, bf16 gate storage):
 * instead of writing dx = d h_t, each thread adds the recurrent d h_t (dh_b view, may be NULL) and turns it into the gate
 * pre-activation gradients, written bf16 over `gates_bf16`; dc is updated in place.  x is the LayerNorm input = h_t (HW*C per sample). */
int pivp_layernorm_bwd_lstm(const float* x, int x_cs, int x_co, const float* g1, int g1_cs, int g1_co, const float* g2, int g2_cs, int g2_co,
                            const float* gamma, const float* beta, const float* stats, int B, int HW, int C,
                            float* dgamma, float* dbeta, void* gates_bf16, const float* c_prev, const float* c_cur,
                            const float* dh_b, int dhb_cs, int dhb_co, float* dc, int dc_valid, void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(x && g1 && gamma && beta && stats && dgamma && dbeta && workspace && gates_bf16 && c_cur && dc, "layernorm_bwd_lstm: null pointer");
    PIVP_REQUIRE(C % 32 == 0 && !((uintptr_t)gates_bf16 & 7) && !(((uintptr_t)c_cur | (uintptr_t)c_prev | (uintptr_t)dc) & 15) &&
                     (!dh_b || (!((uintptr_t)dh_b & 15) && dhb_cs % 4 == 0 && dhb_co % 4 == 0)),
                 "layernorm_bwd_lstm: C must be a multiple of 32 and the state tensors 16-byte aligned");
    const int n = HW * C;
    int chunk;
    const int S = ln_split(n, &chunk);
    PIVP_REQUIRE(ws_bytes >= (size_t)B * S * sizeof(float2), "layernorm_bwd_lstm: workspace too small");
    const int r = ln_vec_bwd(x, x_cs, x_co, g1, g1_cs, g1_co, g2, g2_cs, g2_co, gamma, beta, stats, B, HW, C, 0, (float*)c_cur /*unused*/, C, 0,
                             dgamma, dbeta, workspace, S, chunk, (cudaStream_t)stream, gates_bf16, c_prev, c_cur, dh_b, dhb_cs, dhb_co, dc, dc_valid,
                             nullptr, 0, 0, 0, 0, nullptr);
    if (r == 0) { set_error("layernorm_bwd_lstm: views must be 16-byte aligned with channel counts that are multiples of 4"); return PIVP_EUNSUPPORTED; }
    return r < 0 ? r : PIVP_OK;
}

int pivp_relu_bwd(const float* out, int o_cs, int o_co, const float* ga, int ga_cs, int ga_co, const float* gb, int gb_cs, int gb_co,
                  float* dst, int d_cs, int d_co, long M, int C, void* stream) {
    PIVP_REQUIRE(out && ga && dst && M > 0 && C > 0, "relu_bwd: bad argument");
    if (C % 4 == 0 && v4ok(out, o_cs, o_co) && v4ok(ga, ga_cs, ga_co) && v4ok(gb, gb_cs, gb_co) && v4ok(dst, d_cs, d_co)) {
        launch_k(relu_bwd_v4_kernel, dim3(nblk(M * (C / 4), 256)), dim3(256), 0, (cudaStream_t)stream, CView{out, o_cs, o_co}, CView{ga, ga_cs, ga_co},
                                                                                    CView{gb, gb_cs, gb_co}, View{dst, d_cs, d_co}, M, C / 4);
        return check_launch("relu_bwd");
    }
    launch_k(relu_bwd_kernel, dim3(nblk(M * C, 256)), dim3(256), 0, (cudaStream_t)stream, CView{out, o_cs, o_co}, CView{ga, ga_cs, ga_co}, CView{gb, gb_cs, gb_co},
                                                                        View{dst, d_cs, d_co}, M, C);
    return check_launch("relu_bwd");
}

/* g = ga (+ gb) [* (out > 0)] -> optional fp32 view `dst`, optional bf16 view (plain, or space-to-depth on the H x W grid with channel
 * block cblk, as pivp_cast_bf16), optional bias gradient db[C] += column sums.  Replaces relu_bwd + colsum + cast_bf16 by one launch. */
int pivp_grad_handover(const float* out, int o_cs, int o_co, const float* ga, int ga_cs, int ga_co, const float* gb, int gb_cs, int gb_co,
                       float* dst, int d_cs, int d_co, void* dst_bf16, int b_cs, int b_co, int H, int W, int s2d, int cblk,
                       float* db, long M, int C, void* stream) {
    PIVP_REQUIRE(ga && (dst || dst_bf16 || db) && M > 0 && C > 0 && C % 4 == 0 && C <= 1024, "grad_handover: bad argument (C must be a multiple of 4)");
    PIVP_REQUIRE(v4ok(out, o_cs, o_co) && v4ok(ga, ga_cs, ga_co) && v4ok(gb, gb_cs, gb_co) && v4ok(dst, d_cs, d_co) && v4ok(db, 4, 0),
                 "grad_handover: views must be 16-byte aligned");
    PIVP_REQUIRE(!dst_bf16 || (!((uintptr_t)dst_bf16 & 7) && b_cs % 4 == 0 && b_co % 4 == 0 && cblk % 4 == 0), "grad_handover: bf16 view must be 8-byte aligned");
    PIVP_REQUIRE(!s2d || (H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0 && M % ((long)H * W) == 0 && cblk >= C), "grad_handover: bad space-to-depth geometry");
    const int C4 = C / 4;
    int RPB = 256 / C4;
    if (RPB < 1) RPB = 1;
    long blocks = (M + RPB - 1) / RPB;
    if (blocks > 148 * 8) blocks = 148 * 8;
    launch_k(grad_handover_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, CView{out, o_cs, o_co}, CView{ga, ga_cs, ga_co}, CView{gb, gb_cs, gb_co},
                                                                           View{dst, d_cs, d_co}, (__nv_bfloat16*)dst_bf16, b_cs, b_co, H, W, s2d,
                                                                           cblk, db, M, C4, RPB);
    return check_launch("grad_handover");
}

int pivp_copy_view(const float* src, int s_cs, int s_co, float* dst, int d_cs, int d_co, void* dst_bf16, int db_cs, int db_co,
                   long M, int C, void* stream) {
    PIVP_REQUIRE(src && (dst || dst_bf16) && M > 0 && C > 0, "copy_view: bad argument");
    if (C % 4 == 0 && v4ok(src, s_cs, s_co) && v4ok(dst, d_cs, d_co) && (!dst_bf16 || (!((uintptr_t)dst_bf16 & 7) && db_cs % 4 == 0 && db_co % 4 == 0))) {
        launch_k(copy_view_v4_kernel, dim3(nblk(M * (C / 4), 256)), dim3(256), 0, (cudaStream_t)stream, CView{src, s_cs, s_co}, View{dst, d_cs, d_co},
                                                                                     (__nv_bfloat16*)dst_bf16, db_cs, db_co, M, C / 4);
        return check_launch("copy_view");
    }
    launch_k(copy_view_kernel, dim3(nblk(M * C, 256)), dim3(256), 0, (cudaStream_t)stream, CView{src, s_cs, s_co}, View{dst, d_cs, d_co},
                                                                         (__nv_bfloat16*)dst_bf16, db_cs, db_co, M, C);
    return check_launch("copy_view");
}

int pivp_nchw_to_nhwc(const float* src, float* dst, int d_cs, int d_co, int B, int C, int HW, void* stream) {
    PIVP_REQUIRE(src && dst && B > 0 && C > 0 && HW > 0, "nchw_to_nhwc: bad argument");
    launch_k(nchw_to_nhwc_kernel, dim3(nblk((long)B * HW, 256)), dim3(256), 0, (cudaStream_t)stream, src, View{dst, d_cs, d_co}, B, C, HW);
    return check_launch("nchw_to_nhwc");
}

int pivp_nhwc_to_nchw(const float* src, int s_cs, int s_co, float* dst, int B, int C, int HW, int accumulate, void* stream) {
    PIVP_REQUIRE(src && dst && B > 0 && C > 0 && HW > 0, "nhwc_to_nchw: bad argument");
    launch_k(nhwc_to_nchw_kernel, dim3(nblk((long)B * HW, 256)), dim3(256), 0, (cudaStream_t)stream, CView{src, s_cs, s_co}, dst, B, C, HW, accumulate);
    return check_launch("nhwc_to_nchw");
}

int pivp_cast_bf16(const float* src, int s_cs, int s_co, void* dst_bf16, int d_cs, int d_co, long M, int C, int H, int W, int s2d, int cblk,
                   void* stream) {
    PIVP_REQUIRE(src && dst_bf16 && M > 0 && C > 0, "cast_bf16: bad argument");
    PIVP_REQUIRE(!s2d || (H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0 && M % ((long)H * W) == 0 && cblk >= C), "cast_bf16: bad space-to-depth geometry");
    if (C % 4 == 0 && v4ok(src, s_cs, s_co) && !((uintptr_t)dst_bf16 & 7) && d_cs % 4 == 0 && d_co % 4 == 0 && cblk % 4 == 0) {
        launch_k(cast_bf16_v4_kernel, dim3(nblk(M * (C / 4), 256)), dim3(256), 0, (cudaStream_t)stream, CView{src, s_cs, s_co}, (__nv_bfloat16*)dst_bf16, d_cs, d_co, M,
                                                                                     C / 4, H, W, s2d, cblk);
        return check_launch("cast_bf16");
    }
    launch_k(cast_bf16_kernel, dim3(nblk(M * C, 256)), dim3(256), 0, (cudaStream_t)stream, CView{src, s_cs, s_co}, (__nv_bfloat16*)dst_bf16, d_cs, d_co, M, C, H, W, s2d, cblk);
    return check_launch("cast_bf16");
}

int pivp_axpy(const float* x, float* y, long n, void* stream) {
    PIVP_REQUIRE(x && y && n > 0, "axpy: bad argument");
    launch_k(axpy_kernel, dim3(nblk(n, 256)), dim3(256), 0, (cudaStream_t)stream, x, y, n);
    return check_launch("axpy");
}

int pivp_state_fwd(const float* action, const float* cur, const float* Wc, const float* bc, float* sa, float* next,
                   float* smear, int sm_cs, int sm_co, int npix, int B, void* stream) {
    PIVP_REQUIRE(action && cur && Wc && bc && sa && next && B > 0, "state_fwd: bad argument");
    launch_k(state_fwd_kernel, dim3(B), dim3(64), 0, (cudaStream_t)stream, action, cur, Wc, bc, sa, next, View{smear, sm_cs, sm_co}, npix);
    return check_launch("state_fwd");
}

int pivp_state_bwd(const float* dn_a, const float* dn_b, const float* sa, const float* Wc, const float* dsmear, int ds_cs, int ds_co,
                   int npix, int B, float* d_cur_prev, float* dWc, float* dbc, void* stream) {
    PIVP_REQUIRE(sa && Wc && d_cur_prev && dWc && dbc && B > 0, "state_bwd: bad argument");
    launch_k(state_bwd_kernel, dim3(B), dim3(64), 0, (cudaStream_t)stream, dn_a, dn_b, sa, Wc, CView{dsmear, ds_cs, ds_co}, npix, B, d_cur_prev, dWc, dbc);
    return check_launch("state_bwd");
}

int pivp_linear_fwd(const float* x, int xs, const float* W, const float* bias, float* y, int B, int K, int N, int relu, void* stream) {
    PIVP_REQUIRE(x && W && y && B > 0 && K > 0 && N > 0 && xs >= K, "linear_fwd: bad argument");
    launch_k(linear_fwd_kernel, dim3((N + LIN_NN - 1) / LIN_NN, (B + LIN_BB - 1) / LIN_BB), dim3(256), 0, (cudaStream_t)stream, x, xs, W, bias, y, B, K, N, relu);
    return check_launch("linear_fwd");
}

static int linear_ks(int K) { int ks = K / 512; return ks > 16 ? 16 : (ks < 1 ? 1 : ks); }

size_t pivp_linear_fwd_workspace_bytes(int B, int K, int N) { return sizeof(float) * (size_t)linear_ks(K) * B * N; }

/* Same result as pivp_linear_fwd; split-K over the caller's workspace so the weight matrix is streamed once by >= 2 CTAs per SM.
 * Falls back to the plain kernel when the wide path does not apply (batch > 32, K < 1024 or not a multiple of 4, unaligned rows). */
int pivp_linear_fwd_splitk(const float* x, int xs, const float* W, const float* bias, float* y, int B, int K, int N, int relu,
                           void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(x && W && y && B > 0 && K > 0 && N > 0 && xs >= K, "linear_fwd_splitk: bad argument");
    if (!(B <= LW_B && K >= 1024 && K % 4 == 0 && xs % 4 == 0 && !(((uintptr_t)x | (uintptr_t)W) & 15) && workspace))
        return pivp_linear_fwd(x, xs, W, bias, y, B, K, N, relu, stream);
    PIVP_REQUIRE(ws_bytes >= pivp_linear_fwd_workspace_bytes(B, K, N), "linear_fwd_splitk: workspace too small");
    const int KS = linear_ks(K);
    const int kchunk = ((K / KS) + 3) / 4 * 4;
    float* part = (float*)workspace;
    const int warps = ((N + 3) / 4) * KS;
    launch_k(linear_fwd_wide_kernel, dim3((warps + 3) / 4), dim3(128), 0, (cudaStream_t)stream, x, xs, W, part, B, K, N, kchunk, KS);
    if (int e = check_launch("linear_fwd(wide)")) return e;
    launch_k(linear_fwd_finish_kernel, dim3((B * N + 255) / 256), dim3(256), 0, (cudaStream_t)stream, part, bias, y, B * N, N, KS, relu);
    return check_launch("linear_fwd(finish)");
}

int pivp_linear_bwd(const float* dy, const float* x, int xs, const float* W, float* dx, int dxs, int accumulate_dx,
                    float* dW, float* db, int B, int K, int N, void* stream) {
    PIVP_REQUIRE(dy && x && W && (dW || dx) && B > 0 && K > 0 && N > 0, "linear_bwd: bad argument");
    if (B <= LW_B && K >= 1024 && K % 4 == 0 && xs % 4 == 0 && !(((uintptr_t)x | (uintptr_t)W | (uintptr_t)dW) & 15) &&
        (!dx || (dxs % 4 == 0 && !((uintptr_t)dx & 15)))) {
        cudaStream_t st = (cudaStream_t)stream;
        const int kblocks = (K / 4 + LW_T - 1) / LW_T;
        if (dx) {
            if (!accumulate_dx) {
                if (dxs == K) cudaMemsetAsync(dx, 0, sizeof(float) * (size_t)B * K, st);
                else cudaMemset2DAsync(dx, sizeof(float) * dxs, 0, sizeof(float) * K, B, st);
            }
            int nsplit = (296 + kblocks - 1) / kblocks;
            if (nsplit > N) nsplit = N;
            const int nchunk = (N + nsplit - 1) / nsplit;
            launch_k(linear_bwd_dx_wide_kernel, dim3(kblocks, (N + nchunk - 1) / nchunk), dim3(LW_T), sizeof(float) * nchunk * LW_B, st, dy, W, dx, dxs, B, K, N,
                                                                                                                          nchunk);
            if (int e = check_launch("linear_bwd(dx wide)")) return e;
        }
        if (!dW) return PIVP_OK;                      // weight gradient deferred (pivp_linear_wgrad_steps)
        int nsplit = (444 + kblocks - 1) / kblocks;
        if (nsplit > N) nsplit = N;
        const int nchunk = (N + nsplit - 1) / nsplit;
        launch_k(linear_bwd_dw_wide_kernel, dim3(kblocks, (N + nchunk - 1) / nchunk), dim3(LW_T), sizeof(float) * nchunk * LW_B, st, dy, x, xs, dW, db, B, K, N,
                                                                                                                      nchunk);
        return check_launch("linear_bwd(dw wide)");
    }
    if (dx) {
        launch_k(linear_bwd_dx_kernel, dim3((K + 255) / 256, B), dim3(256), 0, (cudaStream_t)stream, dy, W, dx, dxs, B, K, N, accumulate_dx);
        if (int e = check_launch("linear_bwd(dx)")) return e;
    }
    if (!dW) return PIVP_OK;
    launch_k(linear_bwd_dw_kernel, dim3((K + 255) / 256, N), dim3(256), 0, (cudaStream_t)stream, dy, x, xs, dW, db, B, K, N);
    return check_launch("linear_bwd(dw)");
}

int pivp_linear_wgrad_steps(const float* dy, long dy_step, const float* x, long x_step, int xs, float* dW, float* db, int S, int B, int K, int N,
                            void* stream) {
    PIVP_REQUIRE(dy && x && dW && S > 0 && B > 0 && K > 0 && N > 0, "linear_wgrad_steps: bad argument");
    constexpr int NCH = 9;
    if (B <= LW_B && K % 4 == 0 && xs % 4 == 0 && x_step % 4 == 0 && !(((uintptr_t)x | (uintptr_t)dW) & 15) &&
        (size_t)S * NCH * LW_B * sizeof(float) <= 48 * 1024) {
        const int kblocks = (K / 4 + LW_T - 1) / LW_T;
        launch_k(linear_dw_steps_kernel<NCH>, dim3(kblocks, (N + NCH - 1) / NCH), dim3(LW_T), sizeof(float) * S * NCH * LW_B, stream, dy, dy_step, x,
                 x_step, xs, dW, db, S, B, K, N);
        return check_launch("linear_wgrad_steps");
    }
    for (int s = 0; s < S; ++s) {                   // shapes outside the fast kernel: the per-step path
        launch_k(linear_bwd_dw_kernel, dim3((K + 255) / 256, N), dim3(256), 0, stream, dy + s * dy_step, x + s * x_step, xs, dW, db, B, K, N);
        if (int e = check_launch("linear_wgrad_steps(dw)")) return e;
    }
    return PIVP_OK;
}

int pivp_relu_mask(const float* y, float* g, long n, void* stream) {
    PIVP_REQUIRE(y && g && n > 0, "relu_mask: bad argument");
    launch_k(relu_mask_kernel, dim3(nblk(n, 256)), dim3(256), 0, (cudaStream_t)stream, y, g, n);
    return check_launch("relu_mask");
}

int pivp_mse(const float* gen, const float* target, long n, float gscale, float* dgen, float* loss_slot, void* stream) {
    PIVP_REQUIRE(gen && target && loss_slot && n > 0, "mse: bad argument");
    unsigned g = nblk(n, 256 * 4);
    if (g > 592) g = 592;
    launch_k(mse_kernel, dim3(g), dim3(256), 0, (cudaStream_t)stream, gen, target, n, gscale, dgen, loss_slot);
    return check_launch("mse");
}

int pivp_sched_select(const float* gt, const float* gen, const int* take, float* out, int B, int per_sample, void* stream) {
    PIVP_REQUIRE(gt && gen && take && out && B > 0 && per_sample > 0, "sched_select: bad argument");
    const long n = (long)B * per_sample;
    launch_k(sched_select_kernel, dim3(nblk(n, 256)), dim3(256), 0, (cudaStream_t)stream, gt, gen, take, out, per_sample, n);
    return check_launch("sched_select");
}

int pivp_sched_select_nhwc(const float* gt, const float* gen, const int* take, float* out, float* out_nhwc, int B, int C, int HW, void* stream) {
    PIVP_REQUIRE(gt && gen && take && out && out_nhwc && B > 0 && C > 0 && HW > 0, "sched_select_nhwc: bad argument");
    const long n = (long)B * C * HW;
    launch_k(sched_select_nhwc_kernel, dim3(nblk(n, 256)), dim3(256), 0, (cudaStream_t)stream, gt, gen, take, out, out_nhwc, C, HW, n);
    return check_launch("sched_select_nhwc");
}

int pivp_adam_step(float* p, const float* g, float* m, float* v, long n, int* step, float alpha, float beta1, float beta2, float eps,
                   float gscale, void* stream) {
    PIVP_REQUIRE(p && g && m && v && step && n > 0, "adam_step: bad argument");
    unsigned gb = nblk(n, 256 * 4);
    if (gb > 148 * 8) gb = 148 * 8;
    launch_k(adam_kernel, dim3(gb), dim3(256), 0, (cudaStream_t)stream, p, g, m, v, n, step, alpha, beta1, beta2, eps, gscale);
    if (int e = check_launch("adam_step")) return e;
    launch_k(counter_inc_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, step);
    return check_launch("adam_step(counter)");
}

int pivp_fill(float* p, float value, long n, void* stream) {
    PIVP_REQUIRE(p && n > 0, "fill: bad argument");
    unsigned gb = nblk(n, 256 * 4);
    if (gb > 148 * 8) gb = 148 * 8;
    launch_k(fill_kernel, dim3(gb), dim3(256), 0, (cudaStream_t)stream, p, value, n);
    return check_launch("fill");
}

}  // extern "C"
