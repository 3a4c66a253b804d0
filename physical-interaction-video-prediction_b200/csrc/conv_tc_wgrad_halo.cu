// tcgen05 weight gradient of the ConvLSTM 5x5 convolutions with the XH operand staged once per pixel block (halo patch).
//
//      dW[n][tap][c] += sum_{images, pixels p} dG[p][n] * XH[p + (ky-2, kx-2)][c]            (SURVEY D.5; train_model.py:950)
//
// Same GEMM as conv_tc_wgrad.cu (K = pixels, both operands MN-major straight from the NHWC bf16 tensors), different operand movement:
// that kernel fetches a shifted 64-pixel box of XH for every tap and lets every tap group re-read everything, which made it
// L2 -> SMEM bound at ~23 % of the tensor peak.  Here one K step is an 8 x 8 pixel block:
//   * A = dG  : 4-D TMA box {64 n, 8, 8, 1} x 2 (128 accumulator rows)                                        16 KB
//   * B = XH  : ONE 4-D TMA box {64 c, 16, 12, 1} = the block's (8+4) x (8+4 -> 16) neighbourhood of one 64-channel chunk   24 KB
//     and the B operand of tap (ky, kx), K slice k (16 pixels = two block rows) is that patch seen through an MN-major SW128
//     descriptor starting at patch row (2k + ky) * 16 + kx with SBO = 16 * 128 B between 8-pixel K groups (the swizzle is a function
//     of the shared-memory address, see conv_tc_halo.cu).
// A CTA owns (128 n) x (one 64-channel chunk) x (up to 8 taps = 512 TMEM columns) and a slice of the pixel blocks; partial tiles go
// to the split-K workspace exactly like conv_tc_wgrad.cu (same layout, same reduce kernel).
#include "tc_common.cuh"
#include <stdlib.h>
#include <string.h>

namespace pivp {
namespace wgh {

constexpr int THREADS = 192;
constexpr int A_BYTES = 2 * 64 * 128;            // two 64-n chunks of 64 pixel rows
constexpr int PW = 16, PH = 12;
constexpr int P_BYTES = PW * PH * 128;           // 24576
constexpr int STAGE = A_BYTES + P_BYTES;         // 40960
constexpr int STAGES = 5;
constexpr int MAXTPG = 8;

struct Geom {
    int H, W, Cx, N4, Mrows;
    int chunks, tpg, groups;                     // 64-channel chunks of XH, taps per group, tap groups
    int kb_total, kb_per_split;                  // K steps = 8x8 pixel blocks over all images
    int pair;                                    // most taps issued as one MMA of N = 64 * run columns (PIVP_TC_WGRAD_PAIR = 1, 2 or 4; default 4)
    int tma_out;                                 // partial tiles leave as TMA reduce-adds straight into dW (no split-K workspace, no reduce kernel)
};

__global__ void __launch_bounds__(THREADS, 1)
wgrad5x5_halo_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_o,
                     Geom g, float* __restrict__ part) {
    pdl_enter();
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + (size_t)STAGES * STAGE);
    uint64_t* full = bars;
    uint64_t* empty = bars + STAGES;
    uint64_t* accum_full = bars + 2 * STAGES;
    uint32_t* tmem_slot = (uint32_t*)(accum_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * 128;
    const int chunk = blockIdx.y / g.groups, grp = blockIdx.y - chunk * g.groups;
    const int tap0 = grp * g.tpg, ntaps = min(g.tpg, 25 - tap0);
    const int ncol = min(64, g.Cx - chunk * 64);                  // accumulator columns per tap (channels of this chunk)
    const int split = blockIdx.z;
    const int kb0 = split * g.kb_per_split, kb1 = min(g.kb_total, kb0 + g.kb_per_split);
    const int bx_n = g.W / 8, by_n = g.H / 8;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(full + s), 1); mbar_init(smem_u32(empty + s), 1); }
        mbar_init(smem_u32(accum_full), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer (warp-uniform loop, one elected lane) =====================
        const uint32_t full0 = smem_u32(full), empty0 = smem_u32(empty), ring0 = smem_u32(smem);
        uint32_t st = 0, ph = 1;
        int bx = kb0 % bx_n, by = (kb0 / bx_n) % by_n, img = kb0 / (bx_n * by_n);
        for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(empty0 + 8 * st, ph);
            if (elect_one()) {
                const uint32_t dst = ring0 + st * STAGE;
                mbar_expect_tx(full0 + 8 * st, STAGE);
                tma_load_4d(dst, &map_a, full0 + 8 * st, n0, bx * 8, by * 8, img);
                tma_load_4d(dst + 64 * 128, &map_a, full0 + 8 * st, n0 + 64, bx * 8, by * 8, img);
                tma_load_4d(dst + A_BYTES, &map_b, full0 + 8 * st, chunk * 64, bx * 8 - 2, by * 8 - 2, img);
            }
            __syncwarp();
            if (++st == STAGES) { st = 0; ph ^= 1u; }
            if (++bx == bx_n) { bx = 0; if (++by == by_n) { by = 0; ++img; } }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        // D=f32, A=B=bf16, BOTH MN-major (bits 15, 16), N>>3 at [17,23), M>>4 at [24,29)
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(ncol >> 3) << 17) |
                               ((uint32_t)(128 >> 4) << 24);
        const int max_run = ncol == 64 ? g.pair : 1;         // taps per MMA (partial channel chunks: one, the LBO blocks are 64 wide)
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        // MN-major SW128 descriptor halves.  A: LBO = 8192 B between the two 64-n chunks, SBO = 1024 B between 8-pixel K groups.
        // B: 64-channel blocks = tap-shifted views of one patch (LBO set per MMA, see below), SBO = one patch row = 2048 B between 8-pixel K groups.
        const uint32_t hi_a = (1024u >> 4) | (1u << 14) | (2u << 29);
        const uint32_t hi_b = ((uint32_t)(PW * 128) >> 4) | (1u << 14) | (2u << 29);
        const uint32_t lbo_a = ((8192u >> 4) & 0x3FFFu) << 16;
        const uint32_t ring_lo = (smem_u32(smem) & 0x3FFFFu) >> 4, st_step = STAGE >> 4;
        const uint32_t full0 = smem_u32(full), empty0 = smem_u32(empty);
        const int ky0 = tap0 / 5, kx0 = tap0 - ky0 * 5;
        uint32_t st = 0, ph = 0, lo = ring_lo;
        for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(full0 + 8 * st, ph);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t acc0 = kb > kb0 ? 1u : 0u;
                const uint32_t a_lo = lo | lbo_a;
                int ky = ky0, kx = kx0;
                for (int tl = 0; tl < ntaps;) {
                    // A RUN of taps in one MMA of N = 64 * run columns: block j of the B operand is the SAME patch seen j taps further (LBO = the
                    // row distance between consecutive views), and the accumulators of taps tl .. tl+run-1 are adjacent column blocks.
                    // Cuts the A reads per tap: a 128 x 64 x 16 MMA reads 6 KB of shared memory in 32 tensor cycles (port-bound at 128 B/clk),
                    // 128 x 128 x 16 reads 8 KB in 64, 128 x 256 x 16 reads 12 KB in 128.  Runs of 3-4 need equal distances: taps of one
                    // kernel row (distance 1 patch row); the last tap of a row pairs with the first of the next (distance 16 - 4 rows).
                    const uint32_t row = (uint32_t)(ky * PW + kx);                    // one pixel row = 128 B = 8 descriptor units
                    int run = 1;
                    uint32_t lbo = 1;
                    if (max_run > 1) {
                        const int in_row = min(5 - kx, ntaps - tl);
                        if (in_row >= 2) run = min(in_row, max_run);
                        else if (tl + 1 < ntaps) { run = 2; lbo = (uint32_t)(PW - 4); }
                    }
                    const uint32_t b_lo = ((lo + (A_BYTES >> 4)) + row * 8u) | ((lbo * 8u) << 16);
                    const uint32_t id = (idesc & ~(0x3Fu << 17)) | ((uint32_t)((ncol * run) >> 3) << 17);
#pragma unroll
                    for (int k = 0; k < 4; ++k)        // K slice k: block rows 2k, 2k+1 -> A rows 16k.. (2048 B), patch rows +2k (2k * 16 * 8 units)
                        tc_mma_lohi(tmem_u + (uint32_t)(tl * 64), a_lo + 128 * k, b_lo + (uint32_t)(2 * k * PW * 8), hi_a, hi_b, id,
                                    (k == 0) ? acc0 : 1u);
                    tl += run;
                    kx += run;
                    if (kx >= 5) { kx -= 5; ++ky; }
                }
                tc_commit(empty0 + 8 * st);
                if (kb == kb1 - 1) tc_commit(smem_u32(accum_full));
            }
            __syncwarp();
            lo += st_step;
            if (++st == STAGES) { st = 0; ph ^= 1u; lo = ring_lo; }
        }
    } else {
        // ===================== epilogue: fp32 partial tile -> split-K workspace [split][Mrows][25][Cx] =====================
        const int q = warp & 3;
        const int n = n0 + q * 32 + lane;
        mbar_wait(smem_u32(accum_full), 0);
        tc_fence_after();
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
        if (g.tma_out) {
            // dW (fp32 [n][tap][c], zeroed by cleargrads) += this CTA's partial tiles, added by the memory system: one TMA reduce-add per
            // (tap, 32 channels) box of 128 n x 128 B.  The operand ring is dead (every MMA has retired): six staging buffers of two boxes
            // rotate through it, a buffer is rewritten once the bulk group that read it has finished reading.
            const int row = q * 32 + lane;
            const uint32_t r128 = (uint32_t)row * 128u, rsw = (uint32_t)(row & 7);
            const uint32_t stage0 = smem_u32(smem);
            for (int tl = 0; tl < ntaps; ++tl) {
                const uint32_t sb = stage0 + (uint32_t)(tl % 6) * 32768u;
                if (tl >= 6) {
                    if (warp == 2) { if (elect_one()) asm volatile("cp.async.bulk.wait_group.read 5;" ::: "memory"); __syncwarp(); }
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                }
                for (int c0 = 0; c0 < ncol; c0 += 8) {
                    float v[8];
                    tc_ld8(trow + (uint32_t)(tl * 64 + c0), v);
                    tc_ld_wait();
                    const uint32_t base = sb + (uint32_t)(c0 >> 5) * 16384u + r128;
                    const uint32_t k4 = (uint32_t)((c0 & 31) >> 2);
                    st_shared_v4(base + ((k4 ^ rsw) << 4), __float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
                    st_shared_v4(base + (((k4 + 1u) ^ rsw) << 4), __float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7]));
                }
                fence_proxy_async();
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (warp == 2) {
                    if (elect_one()) {
                        for (int b = 0; b < (ncol >> 5); ++b) tma_reduce_add_4d(&map_o, sb + (uint32_t)b * 16384u, chunk * 64 + 32 * b, tap0 + tl, n0, 0);
                        tma_store_commit();
                        if (tl == ntaps - 1) tma_store_wait_read();
                    }
                    __syncwarp();
                }
            }
            tc_fence_before();
        } else {
        float* dst_row = part + ((size_t)split * g.Mrows + n) * 25 * g.Cx + chunk * 64;
        for (int tl = 0; tl < ntaps; ++tl) {
            float* dst = dst_row + (size_t)(tap0 + tl) * g.Cx;
            for (int c0 = 0; c0 < ncol; c0 += 8) {
                float v[8];
                tc_ld8(trow + (uint32_t)(tl * 64 + c0), v);
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

static void plan(int Cx, int N4, int H, int W, int SB, Geom* g, int* splits) {
    g->H = H; g->W = W; g->Cx = Cx; g->N4 = N4; g->Mrows = (N4 + 127) / 128 * 128;
    g->chunks = (Cx + 63) / 64;
    g->groups = (25 + MAXTPG - 1) / MAXTPG;                       // 4
    g->tpg = (25 + g->groups - 1) / g->groups;                    // 7
    g->kb_total = SB * (H / 8) * (W / 8);
    static const int pair_env = getenv("PIVP_TC_WGRAD_PAIR") ? atoi(getenv("PIVP_TC_WGRAD_PAIR")) : 4;
    g->pair = pair_env < 1 ? 1 : pair_env > 4 ? 4 : pair_env;
    const int tiles = (g->Mrows / 128) * g->chunks * g->groups;
    // K splits: one CTA per SM is resident -- ONE wave (split count rounded down to <= 148 CTAs).  With the partial tiles reduce-added by TMA a
    // second wave only doubles the reduce traffic and the prologues (PIVP_TC_WGRAD_CTAS; measured per launch / per step: 148 -> 108 us, 6.80 ms;
    // 296 -> 115 us, 6.87 ms; 444 -> 120 us, 6.92 ms; 128 / 160 / 192 -> 125 / 133 / 147 us; 0 = the old rule, 2 x 148 rounded up)
    static const int target = getenv("PIVP_TC_WGRAD_CTAS") ? atoi(getenv("PIVP_TC_WGRAD_CTAS")) : 148;
    int s = target > 0 ? target / tiles : (2 * 148 + tiles - 1) / tiles;
    int smax = g->kb_total / 8;
    if (smax < 1) smax = 1;
    if (s > smax) s = smax;
    if (s < 1) s = 1;
    g->kb_per_split = (g->kb_total + s - 1) / s;
    *splits = (g->kb_total + g->kb_per_split - 1) / g->kb_per_split;
}

}  // namespace wgh

bool wgrad_halo_supported(int H, int W, int Cx, int N4) {
    const char* v = getenv("PIVP_TC_WGRAD_HALO");                 // tuning switch: 0 = always use the per-tap kernel
    if (v && atoi(v) == 0) return false;
    return H % 8 == 0 && W % 8 == 0 && Cx % 16 == 0 && Cx >= 16 && Cx <= 512 && N4 % 128 == 0;
}

size_t wgrad_halo_ws_bytes(int SB, int H, int W, int Cx, int N4) {
    wgh::Geom g;
    int splits;
    wgh::plan(Cx, N4, H, W, SB, &g, &splits);
    return (size_t)splits * g.Mrows * 25 * Cx * sizeof(float);
}

// returns the number of K splits written to `part` (>= 1; 0 when the partial tiles were reduce-added into dW directly), or a negative error code
int launch_wgrad5x5_halo(const void* dg_bf16, int dg_cs, const void* xh_bf16, int xh_cs, int SB, int H, int W, int Cx, int N4, float* part,
                         size_t ws_bytes, float* dW, void* stream, const char* who) {
    using namespace wgh;
    Geom g;
    int splits;
    plan(Cx, N4, H, W, SB, &g, &splits);
    // whole 32-channel boxes (dW is 16-byte aligned, pivp_tc_wgrad5x5 checks it): the partial tiles are reduce-added into dW directly, 0 splits returned
    static const int tma_env = getenv("PIVP_TC_WGRAD_TMA") ? atoi(getenv("PIVP_TC_WGRAD_TMA")) : 1;
    g.tma_out = tma_env && Cx % 32 == 0;
    CUtensorMap map_o;
    memset(&map_o, 0, sizeof(map_o));
    if (g.tma_out) {
        cuuint64_t dims[4] = {(cuuint64_t)Cx, 25, (cuuint64_t)N4, 1};
        cuuint64_t str[3] = {(cuuint64_t)Cx * 4, (cuuint64_t)25 * Cx * 4, (cuuint64_t)N4 * 25 * Cx * 4};
        cuuint32_t box[4] = {32, 1, 128, 1};
        if (encode_tmap_ex(&map_o, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, CU_TENSOR_MAP_SWIZZLE_128B, dW, 4, dims, str, box) != CUDA_SUCCESS) g.tma_out = 0;
    }
    PIVP_REQUIRE(g.tma_out || ws_bytes >= (size_t)splits * g.Mrows * 25 * Cx * sizeof(float), "%s(halo): workspace too small", who);
    PIVP_REQUIRE(dg_cs % 8 == 0 && xh_cs % 8 == 0, "%s(halo): rows must be 16-byte aligned", who);
    CUtensorMap map_a, map_b;
    {
        cuuint64_t dims[4] = {(cuuint64_t)N4, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)SB};
        cuuint64_t str[3] = {(cuuint64_t)dg_cs * 2, (cuuint64_t)W * dg_cs * 2, (cuuint64_t)H * W * dg_cs * 2};
        cuuint32_t box[4] = {64, 8, 8, 1};
        CUresult r = encode_tmap(&map_a, dg_bf16, 4, dims, str, box);
        if (r != CUDA_SUCCESS) { set_error("%s(halo): cuTensorMapEncodeTiled(A) failed (%d)", who, (int)r); return PIVP_ECUDA; }
    }
    {
        cuuint64_t dims[4] = {(cuuint64_t)xh_cs, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)SB};
        cuuint64_t str[3] = {(cuuint64_t)xh_cs * 2, (cuuint64_t)W * xh_cs * 2, (cuuint64_t)H * W * xh_cs * 2};
        cuuint32_t box[4] = {64, (cuuint32_t)PW, (cuuint32_t)PH, 1};
        CUresult r = encode_tmap(&map_b, xh_bf16, 4, dims, str, box);
        if (r != CUDA_SUCCESS) { set_error("%s(halo): cuTensorMapEncodeTiled(B) failed (%d)", who, (int)r); return PIVP_ECUDA; }
    }
    const size_t smem = 1024 + (size_t)STAGES * STAGE + (2 * STAGES + 1) * 8 + 16;
    static PerDeviceOnce attr_once;            // the opt-in is per device
    if (attr_once.need()) {
        cudaError_t e = cudaFuncSetAttribute(wgrad5x5_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        if (e != cudaSuccess) { set_error("%s(halo): cudaFuncSetAttribute: %s", who, cudaGetErrorString(e)); return PIVP_ECUDA; }
    }
    dim3 grid((unsigned)(g.Mrows / 128), (unsigned)(g.chunks * g.groups), (unsigned)splits);
    launch_k(wgrad5x5_halo_kernel, dim3(grid), dim3(THREADS), smem, (cudaStream_t)stream, map_a, map_b, map_o, g, part);
    if (int e = check_launch(who)) return e;
    return g.tma_out ? 0 : splits;
}

}  // namespace pivp
