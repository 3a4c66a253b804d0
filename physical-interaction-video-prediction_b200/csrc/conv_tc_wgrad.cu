// tcgen05 weight-gradient of the ConvLSTM 5x5 convolutions, deferred to the end of BPTT and batched over ALL time steps:
//      dW[n][tap][c] += sum_{t} sum_{p} dG_t[p][n] * XH_t[p + (dy-2, dx-2)][c]             (SURVEY D.5; train_model.py:950)
// One launch per layer contracts over K = S*B*H*W pixels (S = T-1 steps) instead of 9 launches of K = B*H*W:
// long K loops, 9x fewer launches, and the split-K partials are written once.
//
// GEMM view per CTA: D[128 n-rows][ntaps x Cx columns] in TMEM (<= 512 fp32 columns), K = pixels.
// Both operands are consumed MN-MAJOR, straight from the NHWC bf16 tensors the forward / input-gradient kernels already use
// (no transposed copies): a TMA box of 64 pixels x 64 channels lands as 64 rows (K) of 128 B (64 MN elements) with the
// 128-byte swizzle, which is the canonical MN-major SWIZZLE_128B UMMA layout (8 K-rows x 128 B atoms; SBO = 1024 B between
// 8-row K groups, LBO = 8192 B between 64-element MN chunks).
//  * A = dG   [S*P][4C] bf16 -> two 2-D boxes {64 ch, 64 px} (128 n-rows)
//  * B = XH   [T*B][H][W][Kpad] bf16 -> ceil(Cx/64) 4-D boxes {64 ch, bw, bh, 1} (bw*bh = 64 px) at the tap-shifted pixel
//    coordinate; out-of-image pixels are zero-filled by TMA (= the convolution's zero padding).  TMA cannot shift along the
//    contiguous dimension by less than 16 B, which is why the pixel shift must be on an outer dimension, i.e. NHWC.
//  * A ring (3 x 16 KB) and B ring (up to 8 slots) with full/empty mbarriers; one A tile feeds ntaps*4 MMAs.
//  * grid = (4C/128, tap groups, K splits); every CTA stores its fp32 partial tile, a second kernel sums the splits into dW.
#include "tc_common.cuh"
#include <string.h>
#include <stdlib.h>
#include <stdlib.h>

namespace pivp {

constexpr int WG_THREADS = 192;
constexpr int WG_ASTAGES = 3;

struct WgGeom {
    int H, W, bw, bh;        // image size at this level, pixel box (bw*bh = 64)
    int Cx, N4;              // channels of XH (accumulator width per tap), 4C
    int chunks;              // 64-channel chunks of XH covering Cx
    int tpg;                 // taps per group
    int kb_total, kb_per_split;
    int b_stages;
    int ntaps;               // total taps of the layer (25 for the ConvLSTM 5x5, 9 for the 3x3 stride-2 layers, 1 for 1x1)
    int Mrows;               // accumulator rows = ceil(N4/128)*128 (rows >= N4 are zero: TMA fills out-of-range channels)
    signed char dy[25], dx[25];
    short coff[25];          // channel offset of each tap inside the XH rows (space-to-depth phases)
    int tma_out;             // partial tiles leave as TMA reduce-adds straight into dW (rows >= N4 are clipped by the tensor map)
};

// MN-major, 128-byte swizzle shared-memory matrix descriptor: LBO = byte distance between 64-element MN chunks,
// SBO = 1024 B between groups of 8 K-rows.
__device__ __forceinline__ uint64_t make_mnmajor_sw128_desc(uint32_t saddr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

__global__ void __launch_bounds__(WG_THREADS, 1)
conv5x5_wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_o,
                        WgGeom g, float* __restrict__ part) {
    pdl_enter();
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t chunk_bytes = 64 * 128;                        // 64 pixel rows x 128 B
    const uint32_t a_bytes = 2 * chunk_bytes, b_bytes = (uint32_t)g.chunks * chunk_bytes;
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + WG_ASTAGES * a_bytes;
    uint64_t* bars = (uint64_t*)(smem_b + (size_t)g.b_stages * b_bytes);
    uint64_t* a_full = bars;
    uint64_t* a_empty = a_full + WG_ASTAGES;
    uint64_t* b_full = a_empty + WG_ASTAGES;
    uint64_t* b_empty = b_full + g.b_stages;
    uint64_t* accum_full = b_empty + g.b_stages;
    uint32_t* tmem_slot = (uint32_t*)(accum_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * 128;
    const int tap0 = blockIdx.y * g.tpg;
    const int ntaps = min(g.tpg, g.ntaps - tap0);
    const int split = blockIdx.z;
    const int kb0 = split * g.kb_per_split, kb1 = min(g.kb_total, kb0 + g.kb_per_split);

    if (threadIdx.x == 0) {
        for (int s = 0; s < WG_ASTAGES; ++s) { mbar_init(smem_u32(a_full + s), 1); mbar_init(smem_u32(a_empty + s), 1); }
        for (int s = 0; s < g.b_stages; ++s) { mbar_init(smem_u32(b_full + s), 1); mbar_init(smem_u32(b_empty + s), 1); }
        mbar_init(smem_u32(accum_full), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // warp-uniform producer / issuer loops, one elected lane (see conv_tc_halo.cu)
    if (warp == 0) {
        const int hw = g.H * g.W;
        const uint32_t afull0 = smem_u32(a_full), aempty0 = smem_u32(a_empty), bfull0 = smem_u32(b_full), bempty0 = smem_u32(b_empty);
        uint32_t sa = 0, pa = 1, sb = 0, pb = 1;
        for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(aempty0 + 8 * sa, pa);
            if (elect_one()) {
                mbar_expect_tx(afull0 + 8 * sa, a_bytes);
                const uint32_t adst = smem_u32(smem_a) + sa * a_bytes;
                tma_load_2d(adst, &map_a, afull0 + 8 * sa, n0, kb * 64);
                tma_load_2d(adst + chunk_bytes, &map_a, afull0 + 8 * sa, n0 + 64, kb * 64);
            }
            __syncwarp();
            if (++sa == WG_ASTAGES) { sa = 0; pa ^= 1u; }
            const long p = (long)kb * 64;
            const int bimg = (int)(p / hw), rem = (int)(p - (long)bimg * hw);
            const int y0 = rem / g.W, x0 = rem - y0 * g.W;
            for (int tl = 0; tl < ntaps; ++tl) {
                const int tap = tap0 + tl;
                mbar_wait(bempty0 + 8 * sb, pb);
                if (elect_one()) {
                    mbar_expect_tx(bfull0 + 8 * sb, b_bytes);
                    const uint32_t bdst = smem_u32(smem_b) + sb * b_bytes;
                    for (int ch = 0; ch < g.chunks; ++ch)
                        tma_load_4d(bdst + ch * chunk_bytes, &map_b, bfull0 + 8 * sb, g.coff[tap] + ch * 64, x0 + g.dx[tap], y0 + g.dy[tap], bimg);
                }
                __syncwarp();
                if (++sb == (uint32_t)g.b_stages) { sb = 0; pb ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // D=f32, A=B=bf16, BOTH MN-major (bits 15, 16), N>>3 at [17,23), M>>4 at [24,29)
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(g.Cx >> 3) << 17) |
                               ((uint32_t)(128 >> 4) << 24);
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        // MN-major SW128 descriptor halves: lo = addr >> 4 | (LBO = 8192 B between 64-element MN chunks) >> 4 << 16; hi = SBO 1024 | v1 | SW128
        const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
        const uint32_t lbo = ((chunk_bytes >> 4) & 0x3FFFu) << 16;
        const uint32_t a_lo0 = ((smem_u32(smem_a) & 0x3FFFFu) >> 4) | lbo, b_lo0 = ((smem_u32(smem_b) & 0x3FFFFu) >> 4) | lbo;
        const uint32_t a_step = a_bytes >> 4, b_step = b_bytes >> 4;
        const uint32_t afull0 = smem_u32(a_full), aempty0 = smem_u32(a_empty), bfull0 = smem_u32(b_full), bempty0 = smem_u32(b_empty);
        uint32_t sa = 0, pa = 0, sb = 0, pb = 0, a_lo = a_lo0, b_lo = b_lo0;
        for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(afull0 + 8 * sa, pa);
            const uint32_t acc0 = kb > kb0 ? 1u : 0u;
            for (int tl = 0; tl < ntaps; ++tl) {
                mbar_wait(bfull0 + 8 * sb, pb);
                tc_fence_after();
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)        // 16 pixels (K) = 16 rows x 128 B = 2048 B per MMA
                        tc_mma_lohi(tmem_u + (uint32_t)(tl * g.Cx), a_lo + 128 * k, b_lo + 128 * k, hi, hi, idesc, (k == 0) ? acc0 : 1u);
                    tc_commit(bempty0 + 8 * sb);
                    if (tl == ntaps - 1) {
                        tc_commit(aempty0 + 8 * sa);
                        if (kb == kb1 - 1) tc_commit(smem_u32(accum_full));
                    }
                }
                __syncwarp();
                b_lo += b_step;
                if (++sb == (uint32_t)g.b_stages) { sb = 0; pb ^= 1u; b_lo = b_lo0; }
            }
            a_lo += a_step;
            if (++sa == WG_ASTAGES) { sa = 0; pa ^= 1u; a_lo = a_lo0; }
        }
    } else {
        const int q = warp & 3;
        const int n = n0 + q * 32 + lane;
        mbar_wait(smem_u32(accum_full), 0);
        tc_fence_after();
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
        if (g.tma_out) {
            // dW += partial tile, added by the memory system (see conv_tc_wgrad_halo.cu): two staging buffers of Cx / 32 boxes in the dead rings
            const int row = q * 32 + lane, nbox = g.Cx >> 5;
            const uint32_t r128 = (uint32_t)row * 128u, rsw = (uint32_t)(row & 7);
            const uint32_t stage0 = smem_u32(smem), buf_bytes = (uint32_t)nbox * 16384u;
            for (int tl = 0; tl < ntaps; ++tl) {
                const uint32_t sbuf = stage0 + (uint32_t)(tl & 1) * buf_bytes;
                if (tl >= 2) {
                    if (warp == 2) { if (elect_one()) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); __syncwarp(); }
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                }
                for (int c0 = 0; c0 < g.Cx; c0 += 8) {
                    float v[8];
                    tc_ld8(trow + (uint32_t)(tl * g.Cx + c0), v);
                    tc_ld_wait();
                    const uint32_t base = sbuf + (uint32_t)(c0 >> 5) * 16384u + r128;
                    const uint32_t k4 = (uint32_t)((c0 & 31) >> 2);
                    st_shared_v4(base + ((k4 ^ rsw) << 4), __float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
                    st_shared_v4(base + (((k4 + 1u) ^ rsw) << 4), __float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7]));
                }
                fence_proxy_async();
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (warp == 2) {
                    if (elect_one()) {
                        for (int b = 0; b < nbox; ++b) tma_reduce_add_4d(&map_o, sbuf + (uint32_t)b * 16384u, 32 * b, tap0 + tl, n0, 0);
                        tma_store_commit();
                        if (tl == ntaps - 1) tma_store_wait_read();
                    }
                    __syncwarp();
                }
            }
            tc_fence_before();
        } else {
        float* dst_row = part + ((size_t)split * g.Mrows + n) * g.ntaps * g.Cx;
        for (int tl = 0; tl < ntaps; ++tl) {
            float* dst = dst_row + (size_t)(tap0 + tl) * g.Cx;
            for (int c0 = 0; c0 < g.Cx; c0 += 8) {
                float v[8];
                tc_ld8(trow + (uint32_t)(tl * g.Cx + c0), v);
                tc_ld_wait();
                *reinterpret_cast<float4*>(dst + c0) = make_float4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<float4*>(dst + c0 + 4) = make_float4(v[4], v[5], v[6], v[7]);
            }
        }
        tc_fence_before();
        }
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// dW[i] += sum_s part[s*stride + i]   (i < n: the valid rows of every split's partial tile come first).  blockIdx.y owns a chunk of
// the splits: one chunk = plain read-modify-write, several chunks (small outputs with up to 144 splits, which were latency-bound in a
// single serial loop: 31 us for 9 CTAs) add their sub-sums with vector atomics.
__global__ void splitk_reduce_kernel(const float* __restrict__ part, float* __restrict__ out, long n, long stride, int splits, int per_chunk) {
    pdl_enter();
    const long i4 = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= n) return;
    const int s0 = blockIdx.y * per_chunk, s1 = min(splits, s0 + per_chunk);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int s = s0;
    for (; s + 8 <= s1; s += 8) {                  // eight independent loads in flight
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __ldg(reinterpret_cast<const float4*>(part + (size_t)(s + j) * stride + i4));
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w; }
    }
    for (; s < s1; ++s) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(part + (size_t)s * stride + i4));
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    if (gridDim.y == 1) {
        float4 o = *reinterpret_cast<const float4*>(out + i4);
        o.x += acc.x; o.y += acc.y; o.z += acc.z; o.w += acc.w;
        *reinterpret_cast<float4*>(out + i4) = o;
    } else {
        atomicAdd(reinterpret_cast<float4*>(out + i4), acc);
    }
}

static void launch_splitk_reduce(const float* part, float* out, long n, long stride, int splits, void* stream) {
    const int per_chunk = splits > 16 ? 16 : splits;
    launch_k(splitk_reduce_kernel, dim3((unsigned)((n / 4 + 255) / 256), (unsigned)((splits + per_chunk - 1) / per_chunk)), dim3(256), 0, stream, part,
             out, n, stride, splits, per_chunk);
}

// out[c] += sum_p src[p][c]  (bf16 in, fp32 accumulate): the ConvLSTM bias gradient over all time steps.
// Thread = 8 channels (one 128-bit load per row), 256 threads = (C8 channel groups) x (256 / C8 row phases); four rows in flight.
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const __nv_bfloat16* __restrict__ src, int ld, long P, int C, long pchunk,
                                                          float* __restrict__ out) {
    pdl_enter();
    __shared__ float red[256][9];
    const int C8 = C >> 3, cg = threadIdx.x % C8, row = threadIdx.x / C8, rows = 256 / C8;
    const long p0 = (long)blockIdx.y * pchunk, p1 = min(P, p0 + pchunk);
    float s[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s[k] = 0.f;
    auto add = [&](const uint4& u) {
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
        for (int k = 0; k < 4; ++k) { const float2 f = __bfloat1622float2(h[k]); s[2 * k] += f.x; s[2 * k + 1] += f.y; }
    };
    if (row < rows) {
        long p = p0 + row;
        for (; p + 3L * rows < p1; p += 4L * rows) {
            uint4 u[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) u[j] = __ldg(reinterpret_cast<const uint4*>(src + (p + (long)j * rows) * ld + 8 * cg));
#pragma unroll
            for (int j = 0; j < 4; ++j) add(u[j]);
        }
        for (; p < p1; p += rows) add(__ldg(reinterpret_cast<const uint4*>(src + p * ld + 8 * cg)));
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) red[threadIdx.x][k] = (row < rows) ? s[k] : 0.f;
    __syncthreads();
    if (threadIdx.x < C) {                                        // channel c = 8 * cg + k: sum the row phases
        const int g8 = threadIdx.x >> 3, k = threadIdx.x & 7;
        float tot = 0.f;
        for (int r = 0; r < rows; ++r) tot += red[r * C8 + g8][k];
        atomicAdd(out + threadIdx.x, tot);
    }
}

// halo-patch variant for the 5x5 stride-1 case (conv_tc_wgrad_halo.cu)
bool wgrad_halo_supported(int H, int W, int Cx, int N4);
size_t wgrad_halo_ws_bytes(int SB, int H, int W, int Cx, int N4);
int launch_wgrad5x5_halo(const void* dg_bf16, int dg_cs, const void* xh_bf16, int xh_cs, int SB, int H, int W, int Cx, int N4, float* part,
                         size_t ws_bytes, float* dW, void* stream, const char* who);

}  // namespace pivp

using namespace pivp;

extern "C" {

int pivp_tc_colsum_bf16(const void* src_bf16, int ld, long P, int C, float* out, void* stream) {
    PIVP_REQUIRE(src_bf16 && out && P > 0 && C > 0 && C % 8 == 0 && C <= 2048 && ld % 8 == 0 && !((uintptr_t)src_bf16 & 15),
                 "tc_colsum_bf16: bad argument (C and ld must be multiples of 8, C <= 2048, rows 16-byte aligned)");
    // channel slabs of <= 256 channels (one CTA column each), row chunks over blockIdx.y
    int slab = C;
    while (slab > 256 || (256 % (slab / 8))) slab -= 8;          // largest slab whose channel groups divide the 256 threads
    PIVP_REQUIRE(C % slab == 0, "tc_colsum_bf16: %d channels cannot be cut into equal slabs of <= 256", C);
    int splits = (int)((P + 255) / 256);                          // enough CTAs to keep ~100 KB per SM in flight
    if (splits > 148 * 8) splits = 148 * 8;
    const long pchunk = (P + splits - 1) / splits;
    for (int c0 = 0; c0 < C; c0 += slab) {
        launch_k(colsum_bf16_kernel, dim3(1, (unsigned)splits), dim3(256), 0, stream, (const __nv_bfloat16*)src_bf16 + c0, ld, P, slab, pchunk,
                 out + c0);
        if (int e = check_launch("tc_colsum_bf16")) return e;
    }
    return PIVP_OK;
}

static void wgrad_plan(int Cx, int Mrows, int ntaps_total, int kb_total, int* tpg, int* groups, int* splits, int* kbps) {
    int tmax = 512 / Cx;
    if (tmax > ntaps_total) tmax = ntaps_total;
    *groups = (ntaps_total + tmax - 1) / tmax;
    *tpg = (ntaps_total + *groups - 1) / *groups;
    *groups = (ntaps_total + *tpg - 1) / *tpg;
    const int tiles = (Mrows / 128) * (*groups);
    static const int target = getenv("PIVP_TC_WGRAD_TAPS_CTAS") ? atoi(getenv("PIVP_TC_WGRAD_TAPS_CTAS")) : 0;      // 0: 2 x 148 rounded up
    int s = target > 0 ? target / tiles : (2 * 148 + tiles - 1) / tiles;
    int smax = kb_total / 8;
    if (smax < 1) smax = 1;
    if (s > smax) s = smax;
    if (s < 1) s = 1;
    *kbps = (kb_total + s - 1) / s;
    *splits = (kb_total + *kbps - 1) / *kbps;
}

static size_t wgrad_ws_bytes(int SB, int H, int W, int Cx, int N4, int ntaps) {
    const long ptot = (long)SB * H * W;
    const int Mrows = (N4 + 127) / 128 * 128;
    int tpg, groups, splits, kbps;
    wgrad_plan(Cx, Mrows, ntaps, (int)(ptot / 64), &tpg, &groups, &splits, &kbps);
    return (size_t)splits * Mrows * ntaps * Cx * sizeof(float);
}

size_t pivp_tc_wgrad_workspace_bytes(int SB, int H, int W, int Cx, int N4) {
    size_t a = wgrad_ws_bytes(SB, H, W, Cx, N4, 25);
    if (wgrad_halo_supported(H, W, Cx, N4)) {
        const size_t b = wgrad_halo_ws_bytes(SB, H, W, Cx, N4);
        if (b > a) a = b;
    }
    return a;
}
size_t pivp_tc_wgrad_taps_workspace_bytes(int SB, int H, int W, int Cx, int N4, int ntaps) { return wgrad_ws_bytes(SB, H, W, Cx, N4, ntaps); }

static int launch_wgrad(const void* dg_bf16, int dg_cs, const void* xh_bf16, int xh_cs, int SB, int H, int W, int Cx, int N4, int ntaps,
                        const int* dy, const int* dx, const int* coff, float* dW, void* workspace, size_t ws_bytes, void* stream, const char* who) {
    PIVP_REQUIRE(dg_bf16 && xh_bf16 && dW && workspace, "%s: null pointer", who);
    // the TMA reduce-add, the split-K partial tiles and splitk_reduce_kernel all move float4s
    PIVP_REQUIRE(!(reinterpret_cast<uintptr_t>(dW) & 15) && !(reinterpret_cast<uintptr_t>(workspace) & 15),
                 "%s: dW and workspace must be 16-byte aligned", who);
    PIVP_REQUIRE(ntaps >= 1 && ntaps <= 25, "%s: 1..25 taps", who);
    PIVP_REQUIRE(Cx >= 16 && Cx <= 256 && Cx % 16 == 0 && N4 >= 8 && N4 % 8 == 0 && dg_cs >= N4 && dg_cs % 8 == 0,
                 "%s: Cx must be a multiple of 16 <= 256, N4 a multiple of 8, rows 16-byte aligned", who);
    const int chunks = (Cx + 63) / 64;
    PIVP_REQUIRE(xh_cs % 8 == 0, "%s: XH rows must be 16-byte aligned", who);
    const long ptot = (long)SB * H * W;
    if ((H * W) % 64 || (W < 64 && 64 % W) || (W > 64 && W % 64)) {
        set_error("%s: cannot cut %dx%d images into 64-pixel TMA boxes", who, H, W);
        return PIVP_EUNSUPPORTED;
    }
    WgGeom g;
    g.H = H; g.W = W; g.bw = W < 64 ? W : 64; g.bh = 64 / g.bw; g.Cx = Cx; g.N4 = N4; g.chunks = chunks; g.ntaps = ntaps;
    g.Mrows = (N4 + 127) / 128 * 128;
    for (int t = 0; t < ntaps; ++t) {
        PIVP_REQUIRE(coff[t] >= 0 && coff[t] % 8 == 0 && coff[t] + chunks * 64 <= xh_cs + 56, "%s: tap %d channel offset out of range", who, t);
        g.dy[t] = (signed char)dy[t]; g.dx[t] = (signed char)dx[t]; g.coff[t] = (short)coff[t];
    }
    int groups, splits;
    g.kb_total = (int)(ptot / 64);
    wgrad_plan(Cx, g.Mrows, ntaps, g.kb_total, &g.tpg, &groups, &splits, &g.kb_per_split);
    int bst = (150 * 1024) / (chunks * 8192);
    if (bst > 8) bst = 8;
    if (bst < 2) bst = 2;
    g.b_stages = bst;
    // whole 32-channel boxes and two staging buffers fit the (dead) operand rings: reduce-add the partial tiles into dW, no workspace, no reduce launch
    static const int tma_env = getenv("PIVP_TC_WGRAD_TMA") ? atoi(getenv("PIVP_TC_WGRAD_TMA")) : 1;
    const size_t ring_bytes = (size_t)WG_ASTAGES * 16384 + (size_t)bst * chunks * 8192;
    g.tma_out = tma_env && Cx % 32 == 0 && 2 * (size_t)(Cx / 32) * 16384 <= ring_bytes;
    CUtensorMap map_o;
    memset(&map_o, 0, sizeof(map_o));
    if (g.tma_out) {
        cuuint64_t dims[4] = {(cuuint64_t)Cx, (cuuint64_t)ntaps, (cuuint64_t)N4, 1};
        cuuint64_t str[3] = {(cuuint64_t)Cx * 4, (cuuint64_t)ntaps * Cx * 4, (cuuint64_t)N4 * ntaps * Cx * 4};
        cuuint32_t box[4] = {32, 1, 128, 1};
        if (encode_tmap_ex(&map_o, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, CU_TENSOR_MAP_SWIZZLE_128B, dW, 4, dims, str, box) != CUDA_SUCCESS) g.tma_out = 0;
    }
    PIVP_REQUIRE(g.tma_out || ws_bytes >= (size_t)splits * g.Mrows * ntaps * Cx * sizeof(float), "%s: workspace too small", who);
    CUtensorMap map_a, map_b;
    {
        cuuint64_t dims[2] = {(cuuint64_t)N4, (cuuint64_t)ptot};
        cuuint64_t str[1] = {(cuuint64_t)dg_cs * 2};
        cuuint32_t box[2] = {64, 64};
        CUresult r = encode_tmap(&map_a, dg_bf16, 2, dims, str, box);
        if (r != CUDA_SUCCESS) { set_error("%s: cuTensorMapEncodeTiled(A) failed (%d)", who, (int)r); return PIVP_ECUDA; }
    }
    {
        cuuint64_t dims[4] = {(cuuint64_t)xh_cs, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)SB};
        cuuint64_t str[3] = {(cuuint64_t)xh_cs * 2, (cuuint64_t)W * xh_cs * 2, (cuuint64_t)H * W * xh_cs * 2};
        cuuint32_t box[4] = {64, (cuuint32_t)g.bw, (cuuint32_t)g.bh, 1};
        CUresult r = encode_tmap(&map_b, xh_bf16, 4, dims, str, box);
        if (r != CUDA_SUCCESS) { set_error("%s: cuTensorMapEncodeTiled(B) failed (%d)", who, (int)r); return PIVP_ECUDA; }
    }
    const size_t smem = 1024 + (size_t)WG_ASTAGES * 16384 + (size_t)bst * chunks * 8192 + (2 * WG_ASTAGES + 2 * bst + 1) * 8 + 16;
    static PerDeviceOnce attr_once;            // the opt-in is per device
    if (attr_once.need()) {
        cudaError_t e = cudaFuncSetAttribute(conv5x5_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        if (e != cudaSuccess) { set_error("%s: cudaFuncSetAttribute: %s", who, cudaGetErrorString(e)); return PIVP_ECUDA; }
    }
    dim3 grid((unsigned)(g.Mrows / 128), (unsigned)groups, (unsigned)splits);
    launch_k(conv5x5_wgrad_tc_kernel, dim3(grid), dim3(WG_THREADS), smem, (cudaStream_t)stream, map_a, map_b, map_o, g, (float*)workspace);
    if (int e = check_launch(who)) return e;
    if (g.tma_out) return PIVP_OK;
    const long n = (long)N4 * ntaps * Cx;
    const long stride = (long)g.Mrows * ntaps * Cx;
    launch_splitk_reduce((const float*)workspace, dW, n, stride, splits, stream);
    return check_launch(who);
}

// dg: [SB*H*W][N4] bf16 (NHWC, all time steps stacked), xh: [>=SB][H][W][xh_cs] bf16 (NHWC), dW: fp32 [N4][25][Cx] accumulated into.
int pivp_tc_wgrad5x5(const void* dg_bf16, const void* xh_bf16, int xh_cs, int SB, int H, int W, int Cx, int N4, float* dW,
                     void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(N4 % 128 == 0 && xh_cs >= (Cx + 63) / 64 * 64, "tc_wgrad5x5: 4C must be a multiple of 128 and XH rows hold ceil(Cx/64)*64 channels");
    if (wgrad_halo_supported(H, W, Cx, N4)) {
        PIVP_REQUIRE(dg_bf16 && xh_bf16 && dW && workspace, "tc_wgrad5x5: null pointer");
        PIVP_REQUIRE(!(reinterpret_cast<uintptr_t>(dW) & 15) && !(reinterpret_cast<uintptr_t>(workspace) & 15),
                     "tc_wgrad5x5: dW and workspace must be 16-byte aligned");
        const int splits = launch_wgrad5x5_halo(dg_bf16, N4, xh_bf16, xh_cs, SB, H, W, Cx, N4, (float*)workspace, ws_bytes, dW, stream, "tc_wgrad5x5");
        if (splits <= 0) return splits;                // 0: the kernel added its partial tiles into dW itself (TMA reduce-add)
        const long n = (long)N4 * 25 * Cx, stride = (long)((N4 + 127) / 128 * 128) * 25 * Cx;
        launch_splitk_reduce((const float*)workspace, dW, n, stride, splits, stream);
        return check_launch("tc_wgrad5x5(reduce)");
    }
    int dy[25], dx[25], co[25];
    for (int t = 0; t < 25; ++t) { dy[t] = t / 5 - 2; dx[t] = t % 5 - 2; co[t] = 0; }
    return launch_wgrad(dg_bf16, N4, xh_bf16, xh_cs, SB, H, W, Cx, N4, 25, dy, dx, co, dW, workspace, ws_bytes, stream, "tc_wgrad5x5");
}

// General form: dW[n][t][c] += sum_p A[p][n] * X[p + (dy_t,dx_t)][coff_t + c]  for n < N4 (A rows of stride a_cs), t < ntaps, c < Cx.
int pivp_tc_wgrad_taps(const void* a_bf16, int a_cs, const void* x_bf16, int x_cs, int SB, int H, int W, int Cx, int N4, int ntaps,
                       const int* dy, const int* dx, const int* coff, float* dW, void* workspace, size_t ws_bytes, void* stream) {
    PIVP_REQUIRE(dy && dx && coff, "tc_wgrad_taps: null tap list (host arrays)");
    return launch_wgrad(a_bf16, a_cs, x_bf16, x_cs, SB, H, W, Cx, N4, ntaps, dy, dx, coff, dW, workspace, ws_bytes, stream, "tc_wgrad_taps");
}

}  // extern "C"
