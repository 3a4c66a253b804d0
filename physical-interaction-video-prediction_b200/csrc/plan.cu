// Cross-entropy-method (CEM) planning over the forward-only predictor: candidate sampling into the predictor's action buffer, the
// goal-image cost of the predicted frames, and the elite refit of the sampling distribution.  See include/pivp.h for the contracts.
#include "common.cuh"
#include <curand_philox4x32_x.h>   // the header-only Philox4x32-10 block of curand_kernel.h (without its generator tables)
#include <math.h>

namespace pivp {

static constexpr int kCemMaxSamples = 8192;           // keys of the shared-memory bitonic sort: 8192 * 8 B = 64 KB
static constexpr int kCostThreads = 256;
static constexpr int kRefitThreads = 1024;

struct Bounds {
    float lo[5], hi[5];
};

// ----------------------------------------------------------------------------- sample
// a[t, n, d] = clip(mean[s, d] + std[s, d] * eps, lo[d], hi[d]), t = ctx-1+s.  eps is one Box-Muller normal from the Philox4x32-10 block
// keyed by the seed at counter (element index e = (n*S + s)*5 + d, iteration): the value of element (n, s, d) depends on neither the grid
// nor Bp.
__global__ void cem_sample_kernel(float* __restrict__ a, int S, int Bp, int t0, const float* __restrict__ mean, const float* __restrict__ stdv,
                                  Bounds b, const long* __restrict__ seed, int iteration) {
    pdl_enter();
    const long total = (long)S * Bp * 5;
    const unsigned long long sd = (unsigned long long)seed[0];
    const uint2 key = make_uint2((unsigned)sd, (unsigned)(sd >> 32));
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const int d = (int)(i % 5);
        const long r = i / 5;                          // r = s * Bp + n: the layout of the action buffer's sampled rows
        const int n = (int)(r % Bp), s = (int)(r / Bp);
        const unsigned long long e = ((unsigned long long)n * S + s) * 5 + d;
        const uint4 x = curand_Philox4x32_10(make_uint4((unsigned)e, (unsigned)(e >> 32), (unsigned)iteration, 0x43454d31u), key);
        const float u1 = ((float)(x.x >> 8) + 0.5f) * (1.0f / 16777216.0f);      // (0, 1): log finite
        const float u2 = (float)(x.y >> 8) * (1.0f / 16777216.0f);
        const float eps = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
        const float v = fmaf(stdv[s * 5 + d], eps, mean[s * 5 + d]);          // std == 0: exactly mean
        float lo = b.lo[0], hi = b.hi[0];
#pragma unroll
        for (int k = 1; k < 5; ++k)                    // register select: a dynamic index into the by-value bounds would go to local memory
            if (d == k) { lo = b.lo[k]; hi = b.hi[k]; }
        a[((long)(t0 + s) * Bp + n) * 5 + d] = fminf(fmaxf(v, lo), hi);
    }
}

// ----------------------------------------------------------------------------- goal cost
// One CTA per candidate row n.  Thread k sums the squared differences of float4 chunks k, k + 256, ... of each weighted step's image and
// folds the step in as acc += w[t] * part; the block then reduces in a fixed tree.  The order depends on (H, W, T) only.
__global__ void __launch_bounds__(kCostThreads) goal_cost_kernel(const float4* __restrict__ gen, int T, int Bp, int n4,
                                                                 const float4* __restrict__ goal, int goal_per_step,
                                                                 const float* __restrict__ w, float inv, float* __restrict__ cost) {
    pdl_enter();
    __shared__ float red[32];
    const int n = blockIdx.x;
    float acc = 0.f;
    for (int t = 0; t < T - 1; ++t) {
        const float wt = w[t];
        if (wt == 0.f) continue;                       // uniform over the CTA: the step is not read
        const float4* g = gen + ((long)t * Bp + n) * n4;
        const float4* q = goal + (goal_per_step ? (long)t * n4 : 0);
        float part = 0.f;
#pragma unroll 4
        for (int i = threadIdx.x; i < n4; i += kCostThreads) {
            const float4 u = g[i], v = q[i];
            const float dx = u.x - v.x, dy = u.y - v.y, dz = u.z - v.z, dw = u.w - v.w;
            part = fmaf(dx, dx, part);
            part = fmaf(dy, dy, part);
            part = fmaf(dz, dz, part);
            part = fmaf(dw, dw, part);
        }
        acc = fmaf(wt, part, acc);
    }
    const float tot = block_sum(acc, red);
    if (threadIdx.x == 0) cost[n] = tot * inv;
}

// ----------------------------------------------------------------------------- refit
__device__ __forceinline__ unsigned long long rank_key(float c, unsigned idx) {
    unsigned u = __float_as_uint(c);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);  // order-preserving: -inf < ... < -0 < +0 < ... < +inf
    if (c != c) u = 0xffffffffu;                      // every NaN after +inf
    return ((unsigned long long)u << 32) | idx;
}

// One CTA: bitonic sort of the N keys (cost bits, index) in shared memory, the K lowest are the elites; per (s, d) one warp takes the
// elite mean and the population standard deviation (two passes, lanes stride over the elites, fixed shuffle tree, double accumulators).
__global__ void __launch_bounds__(kRefitThreads) cem_refit_kernel(const float* __restrict__ cost, const float* __restrict__ a, int T, int Bp,
                                                                  int t0, int N, int P, int K, float alpha, float min_std,
                                                                  float* __restrict__ mean, float* __restrict__ stdv,
                                                                  float* __restrict__ best_cost, float* __restrict__ best_actions,
                                                                  float* __restrict__ history, int iteration) {
    pdl_enter();
    extern __shared__ unsigned long long keys[];
    __shared__ int s_replace;
    const int tid = threadIdx.x;
    for (int i = tid; i < P; i += blockDim.x) keys[i] = i < N ? rank_key(cost[i], (unsigned)i) : ~0ull;
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < P; i += blockDim.x) {
                const int l = i ^ j;
                if (l > i) {
                    const unsigned long long x = keys[i], y = keys[l];
                    if ((x > y) == ((i & k) == 0)) { keys[i] = y; keys[l] = x; }
                }
            }
            __syncthreads();
        }
    }
    const int S = T - t0 - 1;
    const int lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
    const int best = (int)(unsigned)keys[0];
    if (tid == 0) {
        const float c0 = cost[best];
        s_replace = c0 < best_cost[0];               // strictly lower: an earlier iteration keeps a tie
        history[2 * iteration] = c0;
    }
    if (wid == 0) {                                    // mean elite cost
        double sc = 0.0;
        for (int k = lane; k < K; k += 32) sc += (double)cost[(unsigned)keys[k]];
        for (int o = 16; o > 0; o >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, o);
        if (lane == 0) history[2 * iteration + 1] = (float)(sc / K);
    }
    for (int p = wid; p < S * 5; p += nw) {
        const int s = p / 5, d = p % 5;
        const float* col = a + (long)(t0 + s) * Bp * 5 + d;
        double sm = 0.0;
        for (int k = lane; k < K; k += 32) sm += (double)col[(long)(unsigned)keys[k] * 5];
        for (int o = 16; o > 0; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
        const double mu = sm / K;
        double sq = 0.0;
        for (int k = lane; k < K; k += 32) {
            const double dv = (double)col[(long)(unsigned)keys[k] * 5] - mu;
            sq += dv * dv;
        }
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if (lane == 0) {
            const float em = (float)mu, es = (float)sqrt(sq / K);
            mean[p] = alpha * mean[p] + (1.f - alpha) * em;
            stdv[p] = fmaxf(alpha * stdv[p] + (1.f - alpha) * es, min_std);
        }
    }
    __syncthreads();
    if (s_replace) {
        if (tid == 0) best_cost[0] = cost[best];
        for (int i = tid; i < (T - 1) * 5; i += blockDim.x) best_actions[i] = a[((long)(i / 5) * Bp + best) * 5 + i % 5];
    }
}

static bool misaligned16(const void* p) { return ((uintptr_t)p & 15) != 0; }

}  // namespace pivp

using namespace pivp;

extern "C" {

int pivp_cem_max_samples(void) { return kCemMaxSamples; }

int pivp_cem_sample(float* actions, int T, int Bp, int ctx, const float* mean, const float* std_, const float* low, const float* high,
                    const long* seed, int iteration, void* stream) {
    PIVP_REQUIRE(actions && mean && std_ && seed, "cem_sample: actions, mean, std and seed are required");
    PIVP_REQUIRE(Bp >= 1 && ctx >= 1 && T - ctx >= 1 && iteration >= 0,
                 "cem_sample: need Bp >= 1, ctx >= 1, S = T - ctx >= 1, iteration >= 0 (got Bp %d, T %d, ctx %d, iteration %d)",
                 Bp, T, ctx, iteration);
    Bounds b;
    for (int d = 0; d < 5; ++d) {
        b.lo[d] = low ? low[d] : -INFINITY;
        b.hi[d] = high ? high[d] : INFINITY;
        PIVP_REQUIRE(b.lo[d] <= b.hi[d], "cem_sample: low[%d] = %g > high[%d] = %g", d, b.lo[d], d, b.hi[d]);
    }
    const int S = T - ctx;
    const long total = (long)S * Bp * 5;
    long gb = (total + 255) / 256;
    if (gb > 148 * 16) gb = 148 * 16;
    launch_k(cem_sample_kernel, dim3((unsigned)gb), dim3(256), 0, stream, actions, S, Bp, ctx - 1, mean, std_, b, seed, iteration);
    return check_launch("cem_sample");
}

int pivp_goal_cost(const float* gen, int T, int Bp, int N, int H, int W, const float* goal, int goal_per_step, const float* weights,
                   float* cost, void* stream) {
    PIVP_REQUIRE(gen && goal && weights && cost, "goal_cost: gen, goal, weights and cost are required");
    PIVP_REQUIRE(T >= 2 && N >= 1 && N <= Bp && H >= 1 && W >= 1 && (3L * H * W) % 4 == 0,
                 "goal_cost: need T >= 2, 1 <= N <= Bp, 3*H*W a multiple of 4 (got T %d, N %d, Bp %d, H %d, W %d)", T, N, Bp, H, W);
    PIVP_REQUIRE(!misaligned16(gen) && !misaligned16(goal), "goal_cost: gen and goal must be 16-byte aligned (float4 loads)");
    const int n4 = 3 * H * W / 4;
    launch_k(goal_cost_kernel, dim3(N), dim3(kCostThreads), 0, stream, (const float4*)gen, T, Bp, n4, (const float4*)goal,
             goal_per_step ? 1 : 0, weights, 1.f / (3.f * H * W), cost);
    return check_launch("goal_cost");
}

int pivp_cem_refit(const float* cost, const float* actions, int T, int Bp, int ctx, int N, int K, float alpha, float min_std,
                   float* mean, float* std_, float* best_cost, float* best_actions, float* history, int iteration, void* stream) {
    PIVP_REQUIRE(cost && actions && mean && std_ && best_cost && best_actions && history,
                 "cem_refit: cost, actions, mean, std, best_cost, best_actions and history are required");
    PIVP_REQUIRE(N >= 1 && N <= Bp && N <= kCemMaxSamples && K >= 1 && K <= N,
                 "cem_refit: need 1 <= K <= N <= min(Bp, %d) (got N %d, K %d, Bp %d)", kCemMaxSamples, N, K, Bp);
    PIVP_REQUIRE(ctx >= 1 && T - ctx >= 1 && iteration >= 0, "cem_refit: need ctx >= 1, S = T - ctx >= 1, iteration >= 0 (got T %d, ctx %d)",
                 T, ctx);
    PIVP_REQUIRE(alpha >= 0.f && alpha < 1.f && min_std >= 0.f, "cem_refit: need 0 <= alpha < 1 and min_std >= 0 (got %g, %g)", alpha, min_std);
    int P = 1;
    while (P < N) P <<= 1;
    static PerDeviceOnce once;
    if (once.need(sizeof(unsigned long long) * kCemMaxSamples))
        cudaFuncSetAttribute(cem_refit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(unsigned long long) * kCemMaxSamples));
    launch_k(cem_refit_kernel, dim3(1), dim3(kRefitThreads), sizeof(unsigned long long) * P, stream, cost, actions, T, Bp, ctx - 1, N, P, K,
             alpha, min_std, mean, std_, best_cost, best_actions, history, iteration);
    return check_launch("cem_refit");
}

}  // extern "C"
