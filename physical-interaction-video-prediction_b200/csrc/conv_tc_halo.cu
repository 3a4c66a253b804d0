// tcgen05 implicit-GEMM 5x5 "same" convolution with the A operand staged ONCE per 64-channel block as a halo patch in shared memory.
//
// Same GEMM and epilogues as conv_tc.cu (ConvLSTM forward with the fused gate epilogue, train_model.py:262-272; Convolution2D input
// gradient, SURVEY D.5), different operand movement.  conv_tc.cu fetches the 128-pixel A tile again for each of the 25 taps
// (25 x 16 KB per 64 channels, all of it L2 -> SMEM traffic, which is what bounds that kernel).  Here a CTA owns an 8 x 16 pixel tile
// and loads the (16+4) x (8+4 -> 16) pixel neighbourhood once (one 4-D TMA box {64 ch, 16, 20, 1} = 40 KB, zero-filled outside the
// image = the convolution's padding).  With 128-byte rows (64 bf16 channels of one pixel) and the 128-byte swizzle, the A operand of
// tap (dy, dx) is the SAME shared memory seen through a UMMA descriptor whose start address is moved by ((dy+2)*16 + (dx+2)) rows:
// an 8-pixel tile row is exactly one 8-row swizzle atom, consecutive tile rows are one patch row (SBO = 16 * 128 B) apart, and the
// swizzle is a function of the shared-memory address bits, so a row-shifted view stays consistent with what TMA wrote.
// A traffic drops 25 x 16 KB -> 40 KB per (tile, 64 channels); the weight tiles stream through the ring as before.
//
// 8 x 8 maps (ConvLSTM layer 5) use the "pair" geometry: a tile is two whole images, and the patch interleaves their rows --
// tensor-map dimensions ordered (channel, x, image, y), box {64, 16, 2, 12} = 48 KB -- so that the 16 eight-pixel groups (y, image)
// are again one uniform 2048 B apart and tap (dy, dx) is a start address moved by (2*(dy+2)*16 + (dx+2)) rows.
#include "tc_common.cuh"
#include "tc_epilogue.cuh"
#include <stdlib.h>

namespace pivp {
namespace halo {

constexpr int TW = 8, TH = 16;                    // output pixels per CTA: 8 wide x 16 tall = 128 TMEM lanes
constexpr int PW = 16, PH = TH + 4;               // patch: 16 x 20 pixels (x0-2 .. x0+13, y0-2 .. y0+17)
constexpr int PATCH_BYTES = PW * PH * 128;        // 40960
constexpr int PAIR_PATCH_BYTES = PW * 2 * 12 * 128;   // 49152: two 8x8 images, rows interleaved
constexpr int GP = 132, CP = 36;                  // padded row pitches (floats) of the epilogue staging: gates 128 + 4, c / h 32 + 4
constexpr int STG_FLOATS = 128 * (GP + 2 * CP);   // per pixel tile: 104448 bytes

struct Geom {
    int H, W, Kc, N, BN, stages, tmem_cols;
    int pair;                                     // 8 x 8 maps: one tile = two images (see the header)
    int patch_bytes;
    int cb_per_split;                             // split-K: blockIdx.z owns 64-channel blocks [z * cb_per_split, ...) and adds its partial atomically
    int npatch;                                   // patch buffers (1..3): the next 64-channel block's patch loads under this block's MMAs
    int tma_out;                                  // epilogue writes its tiles with TMA stores (OutMaps) instead of per-thread global stores
    long long* dbg;                               // optional per-CTA clock64 stamps [grid][8] (pivp_tc_set_debug_buffer), else null
};
// Output tensor maps of the TMA-store epilogues.  Every map describes the output as (channel, x, y, image) -- (channel, x, image, y) in
// the pair geometry -- with a box of {32 fp32 | 64 bf16 | 32 bf16 channels, 8, 16, 1} ({.., 8, 2, 8}): exactly one 128-pixel tile in the
// order of the accumulator rows, so a tile leaves shared memory with one instruction per 128-byte (64-byte: hb) column group.
struct OutMaps {
    CUtensorMap gates;      // mode 1: activated gates, bf16 (M, 4C), SWIZZLE_128B, two boxes of 64 columns per tile
    CUtensorMap c;          // mode 1: c_t fp32 (M, C)
    CUtensorMap h;          // mode 1: h_t fp32 view into xh[t+1]
    CUtensorMap hb;         // mode 1: bf16 shadow of h_t, SWIZZLE_64B
    CUtensorMap out;        // mode 0: fp32 output view, BN / 32 boxes per tile (plain store, or reduce-add for split-K partials)
    CUtensorMap y;          // mode 1 + fused LayerNorm: normalised h, fp32 view
    CUtensorMap yb;         // mode 1 + fused LayerNorm: its bf16 copy, SWIZZLE_64B
};
constexpr int STG_TMA = 96 * 1024;                // mode 1 staging per pixel tile: gates 2 x 16 KB | c 16 KB | h 16 KB | hb 8 KB | y 16 KB | yb 8 KB
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

#define HALO_ROW ((size_t)((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 8)
#define HALO_STAMP(i) do { if (g.dbg && lane == 0) g.dbg[HALO_ROW + (i)] = clock64(); } while (0)
__device__ __forceinline__ long long global_ns() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }

// K-major SW128 descriptor with an explicit stride between 8-row groups.  The swizzle XOR is taken from the shared-memory ADDRESS
// bits [7,10) (measured on B200: a start address moved by whole 128-byte rows needs no base-offset field; setting it breaks the result).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(sbo_bytes >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// MS = pixel tiles (of 128) per CTA: each weight stage feeds 4*MS MMAs, i.e. MS*BN/4... cycles of tensor work per 128*BN bytes fetched.
// One CTA per SM: all shared memory that the MS patches leave goes to the weight ring, deep enough to cover the L2 round trip.
// NP = patch buffers (compile-time: the buffer index and barrier parity of a block must stay on the uniform datapath, a run-time
// modulus pushes the whole issue loop back onto vector registers + per-MMA R2UR / divergence checks).
// GATES = false: the mode-1 epilogues store no activated gates (pivp_tc_conv5x5 flags bit 2: forward-only prediction, ep.gates == null).
// c_prev may alias c_out in every mode-1 epilogue: a thread loads the c_prev elements of its own pixel row and channels before the
// accumulator wait, and those elements are written (by a TMA store or the coalesced write-out) only after the barrier of the tile's warps.
template <int MS, int NP, bool GATES>
__global__ void __launch_bounds__(64 + 256 * MS, 1)
conv5x5_halo_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ OutMaps om,
                       Geom g, TcEpilogue ep) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* patch = smem;
    const uint32_t pbuf_bytes = (uint32_t)(MS * g.patch_bytes);     // one patch buffer = the MS tiles' patches of one 64-channel block
    uint8_t* bring = smem + NP * pbuf_bytes;
    const uint32_t b_bytes = (uint32_t)g.BN * 128;
    uint64_t* bars = (uint64_t*)(bring + (size_t)g.stages * b_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + g.stages;
    uint64_t* patch_full = bars + 2 * g.stages;                     // [3]
    uint64_t* patch_empty = patch_full + 3;                         // [3]
    uint64_t* accum_full = patch_full + 6;
    uint32_t* tmem_slot = (uint32_t*)(patch_full + 7);
    float* bias_s = (float*)(tmem_slot + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tile = blockIdx.y;
    const int n0 = n_tile * g.BN;
    const int cb_first = blockIdx.z * g.cb_per_split;
    const int ncb = min(g.Kc / 64 - cb_first, g.cb_per_split);        // 64-channel blocks of this CTA (local index cb, global cb_first + cb)
    const int tiles_x = g.W / TW, tiles_y = g.H / TH;
    if (warp == 0) { HALO_STAMP(0); if (g.dbg && lane == 0) g.dbg[HALO_ROW + 6] = global_ns(); }

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) { mbar_init(smem_u32(full + s), 1); mbar_init(smem_u32(empty + s), 1); }
        for (int s = 0; s < 3; ++s) { mbar_init(smem_u32(patch_full + s), 1); mbar_init(smem_u32(patch_empty + s), 1); }
        mbar_init(smem_u32(accum_full), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)g.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    pdl_wait();                                      // barrier init / TMEM allocation above overlap the previous kernel's tail
    if (warp >= 2 && ep.bias && blockIdx.z == 0) {
        for (int i = threadIdx.x - 64; i < g.BN; i += 256 * MS) bias_s[i] = ep.bias[n0 + i];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 1) HALO_STAMP(1);

    // Producer and MMA issuer run warp-uniform loops (every operand derives from kernel parameters and loop counters, the TMEM
    // base is broadcast with a shuffle) and one elected lane issues: otherwise the compiler cannot keep descriptors in uniform
    // registers and wraps every tcgen05.mma in a per-lane waterfall loop -- ~20 issue slots per MMA, which is what bounded the
    // per-tap kernel at ~25 % tensor-pipe utilisation (profiles/r01_ncu_halo_issue_bound.md).
    // (Measured and dropped in round 2: running the first `stages` iterations of the producer loop BEFORE the CTA-wide set-up barrier -- the
    // TMA issue path costs ~300 cycles per stage (try_wait + elect + expect_tx + UTMALDG), so the barrier, and with it the MMA warp, waited
    // 3.6k cycles for the producer: first operands at 5.0k cycles instead of 3.6k.  Also measured: the same loop written as a resumable
    // lambda over captured state ran at 356 instead of 294 cycles per stage and made the one-tile launches producer-bound.)
    if (warp == 0) {
        // ===================== TMA producer =====================
        const uint32_t full0 = smem_u32(full), empty0 = smem_u32(empty), ring0 = smem_u32(bring);
        uint32_t st = 0, ph = 1;                                  // waits on `empty` start with parity 1 (fresh barrier)
        const uint32_t pfull0 = smem_u32(patch_full), pempty0 = smem_u32(patch_empty);
        constexpr int np = NP;
        int next = 0;                                             // next 64-channel block whose patch has not been requested yet
        // patch n goes to buffer n % np once the MMAs of block n - np have drained it (use count u = n / np -> parity (u & 1) ^ 1)
        auto issue_patch = [&](int n) {
            const uint32_t slot = (uint32_t)(n % np);
            if (elect_one()) {
                mbar_expect_tx(pfull0 + 8 * slot, pbuf_bytes);
#pragma unroll
                for (int i = 0; i < MS; ++i) {
                    const int mt = blockIdx.x * MS + i;
                    const uint32_t dst = smem_u32(patch) + slot * pbuf_bytes + (uint32_t)(i * g.patch_bytes);
                    if (g.pair) {
                        tma_load_4d(dst, &map_a, pfull0 + 8 * slot, (cb_first + n) * 64, -2, 2 * mt, -2);
                    } else {
                        const int tx = mt % tiles_x, ty = (mt / tiles_x) % tiles_y, tb = mt / (tiles_x * tiles_y);
                        tma_load_4d(dst, &map_a, pfull0 + 8 * slot, (cb_first + n) * 64, tx * TW - 2, ty * TH - 2, tb);
                    }
                }
            }
            __syncwarp();
        };
        for (int cb = 0; cb < ncb; ++cb) {
            if (next == cb) {                                     // this block's patch must be on its way before its weights fill the ring
                mbar_wait(pempty0 + 8 * (uint32_t)(next % np), (uint32_t)((next / np) & 1) ^ 1u);
                issue_patch(next++);
            }
            for (int tap = 0; tap < 25; ++tap) {
                // prefetch later patches as soon as their buffer is free (non-blocking test), after this block's first weight tiles
                if (NP > 1 && tap >= 2 && next < ncb && next < cb + np) {
                    const int freed = (int)mbar_test(pempty0 + 8 * (uint32_t)(next % np), (uint32_t)((next / np) & 1) ^ 1u);
                    if (__all_sync(0xffffffffu, freed)) issue_patch(next++);      // a vote keeps the branch (and with it the whole kernel) warp-uniform for ptxas
                }
                mbar_wait(empty0 + 8 * st, ph);
                if (elect_one()) {
                    mbar_expect_tx(full0 + 8 * st, b_bytes);
                    tma_load_2d(ring0 + st * b_bytes, &map_b, full0 + 8 * st, tap * g.Kc + (cb_first + cb) * 64, n0);
                }
                __syncwarp();
                if (++st == (uint32_t)g.stages) { st = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(g.BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        // descriptor halves: lo = (addr >> 4) | LBO(1) << 16; hi = SBO >> 4 | version 1 (bit 46) | SWIZZLE_128B (bits 61-63)
        const uint32_t hi_b = (1024u >> 4) | (1u << 14) | (2u << 29);
        const uint32_t hi_a = ((uint32_t)(PW * 128) >> 4) | (1u << 14) | (2u << 29);
        const uint32_t ring_lo = ((smem_u32(bring) & 0x3FFFFu) >> 4) | 0x10000u, b_step = b_bytes >> 4;
        const uint32_t patch_lo = ((smem_u32(patch) & 0x3FFFFu) >> 4) | 0x10000u;
        const uint32_t full0 = smem_u32(full), empty0 = smem_u32(empty);
        const uint32_t ky_rows = g.pair ? 2u * PW : (uint32_t)PW, patch_step = (uint32_t)g.patch_bytes >> 4;
        const uint32_t pfull0 = smem_u32(patch_full), pempty0 = smem_u32(patch_empty);
        uint32_t st = 0, ph = 0, b_lo = ring_lo;
        for (int cb = 0; cb < ncb; ++cb) {
            const uint32_t slot = (uint32_t)(cb % NP), use_par = (uint32_t)((cb / NP) & 1);      // patch buffer of this block, parity of its use count
            const uint32_t pf_bar = pfull0 + 8 * slot, pe_bar = pempty0 + 8 * slot;
            const uint32_t pb_lo = patch_lo + slot * (pbuf_bytes >> 4);
            mbar_wait(pf_bar, use_par);
            if (cb == 0) HALO_STAMP(2);
            for (int ky = 0; ky < 5; ++ky) {
#pragma unroll
                for (int kx = 0; kx < 5; ++kx) {
                    mbar_wait(full0 + 8 * st, ph);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t a_lo = pb_lo + ((uint32_t)ky * ky_rows + (uint32_t)kx) * 8u;      // one pixel row = 128 B = 8 descriptor units
#pragma unroll
                        for (int i = 0; i < MS; ++i)
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                tc_mma_lohi(tmem_u + (uint32_t)(i * g.BN), a_lo + (uint32_t)i * patch_step + 2u * k, b_lo + 2 * k, hi_a, hi_b,
                                            idesc, (k == 0) ? ((cb | ky | kx) ? 1u : 0u) : 1u);
                        tc_commit(empty0 + 8 * st);
                        if (ky == 4 && kx == 4) {
                            tc_commit(pe_bar);
                            if (cb == ncb - 1) tc_commit(smem_u32(accum_full));
                        }
                    }
                    __syncwarp();
                    b_lo += b_step;
                    if (++st == (uint32_t)g.stages) { st = 0; ph ^= 1u; b_lo = ring_lo; }
                }
            }
        }
        HALO_STAMP(3);
    } else {
        // ===================== epilogue: 8 warps per pixel tile (lane quarter q x column half) =====================
        const int ew = warp - 2, sub = ew >> 3, half = (ew >> 2) & 1, q = warp & 3;       // q = TMEM lane quarter this warp may read
        const int row = q * 32 + lane;
        const int mt = blockIdx.x * MS + sub;
        const int tx = mt % tiles_x, ty = (mt / tiles_x) % tiles_y, tb = mt / (tiles_x * tiles_y);
        // NHWC pixel index of accumulator row r: tile rows are 8-pixel groups; pair geometry: group = (y, image) of two 8x8 images
        const long m00 = g.pair ? (long)mt * 128 : ((long)tb * g.H + ty * TH) * g.W + tx * TW;
        auto pixel_of = [&](int r) -> long {
            return g.pair ? m00 + ((r >> 3) & 1) * 64 + (r >> 4) * 8 + (r & 7) : m00 + (long)(r >> 3) * g.W + (r & 7);
        };
        const long m = pixel_of(row);
        const uint32_t trow = tmem_base + (uint32_t)(sub * g.BN) + ((uint32_t)(q * 32) << 16);
        const int lw = ew & 7;
        // tile coordinates of the output tensor maps
        const int oc1 = g.pair ? 0 : tx * TW, oc2 = g.pair ? 2 * mt : ty * TH, oc3 = g.pair ? 0 : tb;
        if (ep.mode == 1 && g.tma_out) {
            // ---- ConvLSTM gate epilogue with TMA stores.  Every thread owns one accumulator row (pixel) and 16 of the tile's 32 channels.
            // Results are packed to their storage type in registers and written ONCE into shared-memory tiles laid out as the output
            // tensor maps' boxes (128-byte rows, 128-byte swizzle: the 32 rows of a warp hit all banks), then five TMA stores write
            // the tile: no shared-memory read-back, no per-thread global store, no index arithmetic per row.
            const int ch0 = n_tile * 32;
            float cp[16];
            if (ep.c_prev) {                                 // issued before the accumulator wait: the main loop hides the latency
                const float4* src = reinterpret_cast<const float4*>(ep.c_prev + m * ep.C + ch0 + half * 16);
#pragma unroll
                for (int i = 0; i < 4; ++i) { const float4 v = __ldg(src + i); cp[4 * i] = v.x; cp[4 * i + 1] = v.y; cp[4 * i + 2] = v.z; cp[4 * i + 3] = v.w; }
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) cp[i] = 0.f;
            }
            mbar_wait(smem_u32(accum_full), 0);
            tc_fence_after();
            if (warp == 2) HALO_STAMP(4);
            const uint32_t sG = smem_u32(smem) + (uint32_t)(sub * STG_TMA), sC = sG + 32768u, sH = sC + 16384u, sHB = sH + 16384u;
            const uint32_t r128 = (uint32_t)row * 128u, rsw = (uint32_t)(row & 7), r64 = (uint32_t)row * 64u, rsw64 = (uint32_t)((row >> 1) & 3);
            float hv[16];
#pragma unroll
            for (int cc = 0; cc < 16; cc += 8) {
                const int c0 = half * 16 + cc;
                float gj[8], gi[8], gf[8], go[8], cn[8], hn[8];
                tc_ld8(trow + (uint32_t)(c0), gj);
                tc_ld8(trow + (uint32_t)(32 + c0), gi);
                tc_ld8(trow + (uint32_t)(64 + c0), gf);
                tc_ld8(trow + (uint32_t)(96 + c0), go);
                tc_ld_wait();
                if (ep.accurate) gate_math8<true>(gj, gi, gf, go, cp + cc, bias_s, c0, ep.forget_bias, cn, hn);
                else gate_math8<false>(gj, gi, gf, go, cp + cc, bias_s, c0, ep.forget_bias, cn, hn);
#pragma unroll
                for (int i = 0; i < 8; ++i) hv[cc + i] = hn[i];
                const uint32_t k8 = (uint32_t)(c0 >> 3), k4 = (uint32_t)(c0 >> 2);       // 16-byte chunk of this thread's columns in a bf16 / fp32 row
                uint4 pk;
                if (GATES) {
                    pk = pack8_bf16(gj); st_shared_v4(sG + r128 + ((k8 ^ rsw) << 4), pk.x, pk.y, pk.z, pk.w);                   // box 0: j | i
                    pk = pack8_bf16(gi); st_shared_v4(sG + r128 + (((4u + k8) ^ rsw) << 4), pk.x, pk.y, pk.z, pk.w);
                    pk = pack8_bf16(gf); st_shared_v4(sG + 16384u + r128 + ((k8 ^ rsw) << 4), pk.x, pk.y, pk.z, pk.w);          // box 1: f | o
                    pk = pack8_bf16(go); st_shared_v4(sG + 16384u + r128 + (((4u + k8) ^ rsw) << 4), pk.x, pk.y, pk.z, pk.w);
                }
                st_shared_v4(sC + r128 + ((k4 ^ rsw) << 4), __float_as_uint(cn[0]), __float_as_uint(cn[1]), __float_as_uint(cn[2]), __float_as_uint(cn[3]));
                st_shared_v4(sC + r128 + (((k4 + 1u) ^ rsw) << 4), __float_as_uint(cn[4]), __float_as_uint(cn[5]), __float_as_uint(cn[6]), __float_as_uint(cn[7]));
                st_shared_v4(sH + r128 + ((k4 ^ rsw) << 4), __float_as_uint(hn[0]), __float_as_uint(hn[1]), __float_as_uint(hn[2]), __float_as_uint(hn[3]));
                st_shared_v4(sH + r128 + (((k4 + 1u) ^ rsw) << 4), __float_as_uint(hn[4]), __float_as_uint(hn[5]), __float_as_uint(hn[6]), __float_as_uint(hn[7]));
                pk = pack8_bf16(hn); st_shared_v4(sHB + r64 + ((k8 ^ rsw64) << 4), pk.x, pk.y, pk.z, pk.w);
            }
            float2* red = reinterpret_cast<float2*>(smem + (size_t)MS * STG_TMA) + sub * 12;        // 8 warp pairs + the sample's (mean, rstd)
            const bool fuse_ln = ep.ln_gamma != nullptr;
            float ga[16], be[16];
            if (fuse_ln) {                                   // affine parameters of this thread's 16 elements: in flight across the barriers below
                const long e = (m - (long)tb * g.H * g.W) * ep.C + ch0 + half * 16;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 a = __ldg(reinterpret_cast<const float4*>(ep.ln_gamma + e) + i), b4 = __ldg(reinterpret_cast<const float4*>(ep.ln_beta + e) + i);
                    ga[4 * i] = a.x; ga[4 * i + 1] = a.y; ga[4 * i + 2] = a.z; ga[4 * i + 3] = a.w;
                    be[4 * i] = b4.x; be[4 * i + 1] = b4.y; be[4 * i + 2] = b4.z; be[4 * i + 3] = b4.w;
                }
            }
            if (ep.ln_partial) {
                // LayerNorm statistics of the h tile (train_model.py:203-208): every warp reduces its 32 x 16 block to (mean, M2) exactly
                // (two passes over registers), one thread merges the eight equal-sized blocks (Chan) into the tile's (mean, M2) pair
                float s = 0.f;
#pragma unroll
                for (int i = 0; i < 16; ++i) s += hv[i];
                const float mean_w = warp_sum(s) * (1.f / 512.f);
                float m2 = 0.f;
#pragma unroll
                for (int i = 0; i < 16; ++i) { const float d = hv[i] - mean_w; m2 = fmaf(d, d, m2); }
                m2 = warp_sum(m2);
                if (lane == 0) red[lw] = make_float2(mean_w, m2);
            }
            fence_proxy_async();
            asm volatile("bar.sync %0, 256;" ::"r"(1 + sub) : "memory");          // the eight warps of this pixel tile
            const int tiles_per_img = tiles_x * tiles_y;
            if (lw == 0) {
                if (elect_one()) {
                    if (GATES) {
                        tma_store_4d(&om.gates, sG, n0, oc1, oc2, oc3);
                        tma_store_4d(&om.gates, sG + 16384u, n0 + 64, oc1, oc2, oc3);
                    }
                    tma_store_4d(&om.c, sC, ch0, oc1, oc2, oc3);
                    tma_store_4d(&om.h, sH, ep.h_co + ch0, oc1, oc2, oc3);
                    tma_store_4d(&om.hb, sHB, ep.hb_co + ch0, oc1, oc2, oc3);
                    tma_store_commit();
                }
                __syncwarp();
            } else if (lw == 1 && ep.ln_partial) {
                if (lane == 0) {
                    float mean = 0.f;
#pragma unroll
                    for (int i = 0; i < 8; ++i) mean += red[i].x;
                    mean *= 0.125f;
                    float t2 = 0.f;
#pragma unroll
                    for (int i = 0; i < 8; ++i) { const float d = red[i].x - mean; t2 += red[i].y + 512.f * d * d; }
                    ep.ln_partial[(long)tb * ep.ln_S + (mt - tb * tiles_per_img) * (ep.C >> 5) + n_tile] = make_float2(mean, t2);
                    if (fuse_ln) {
                        // arrive at the sample's counter; the launch adds exactly ln_S arrivals per sample, so the target is the next multiple
                        __threadfence();
                        const unsigned old = atomicAdd(ep.ln_counter + tb, 1u);
                        const unsigned target = (old / (unsigned)ep.ln_S + 1u) * (unsigned)ep.ln_S;
                        unsigned spins = 0;
                        while ((int)(ld_acquire_u32(ep.ln_counter + tb) - target) < 0 && ++spins < (1u << 22)) { }       // bounded: never hangs the GPU
                    }
                }
                if (fuse_ln) {
                    // every tile of the sample has published its pair: lane i fetches pair i (ONE L2 round trip for the whole merge), Chan merge
                    // of the ln_S <= 32 equal-sized chunks with two warp reductions, result to shared memory for the tile's threads
                    __syncwarp();
                    const float2 p = lane < ep.ln_S ? __ldcg(ep.ln_partial + (long)tb * ep.ln_S + lane) : make_float2(0.f, 0.f);
                    const float mu = warp_sum(p.x) / (float)ep.ln_S;
                    const float d = p.x - mu;
                    const float m2 = warp_sum(lane < ep.ln_S ? p.y + 4096.f * d * d : 0.f);
                    if (lane == 0) red[8] = make_float2(mu, 1.f / sqrtf(m2 / (4096.f * (float)ep.ln_S) + ep.ln_eps));
                }
            }
            if (fuse_ln) {
                asm volatile("bar.sync %0, 256;" ::"r"(1 + sub) : "memory");      // the sample's (mean, rstd) is in shared memory
                const float mu = red[8].x, rstd = red[8].y;
                const uint32_t sY = sHB + 8192u, sYB = sY + 16384u;
                float yv[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) yv[i] = (hv[i] - mu) * rstd * ga[i] + be[i];
                const uint32_t k4 = (uint32_t)(half * 4), k8 = (uint32_t)(half * 2);
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    st_shared_v4(sY + r128 + (((k4 + (uint32_t)i) ^ rsw) << 4), __float_as_uint(yv[4 * i]), __float_as_uint(yv[4 * i + 1]),
                                 __float_as_uint(yv[4 * i + 2]), __float_as_uint(yv[4 * i + 3]));
                if (ep.ln_yb) {
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const float v8[8] = {yv[8 * i], yv[8 * i + 1], yv[8 * i + 2], yv[8 * i + 3], yv[8 * i + 4], yv[8 * i + 5], yv[8 * i + 6], yv[8 * i + 7]};
                        const uint4 pk = pack8_bf16(v8);
                        st_shared_v4(sYB + r64 + (((k8 + (uint32_t)i) ^ rsw64) << 4), pk.x, pk.y, pk.z, pk.w);
                    }
                }
                fence_proxy_async();
                asm volatile("bar.sync %0, 256;" ::"r"(1 + sub) : "memory");
                if (lw == 0) {
                    if (elect_one()) {
                        tma_store_4d(&om.y, sY, ep.ln_y_co + ch0, oc1, oc2, oc3);
                        if (ep.ln_yb) tma_store_4d(&om.yb, sYB, ep.ln_yb_co + ch0, oc1, oc2, oc3);
                        tma_store_commit();
                    }
                    __syncwarp();
                } else if (lw == 1 && lane == 0 && n_tile == 0 && mt == tb * tiles_per_img) {
                    ep.ln_stats[tb] = make_float2(mu, rstd);
                }
            }
            if (lw == 0) {
                if (elect_one()) tma_store_wait_read();      // shared memory must outlive the bulk reads
                __syncwarp();
            }
        } else if (ep.mode == 0 && g.tma_out) {
            // ---- plain epilogue with TMA stores: BN / 32 boxes of 32 fp32 columns per tile; split-K partials leave as TMA reduce-adds
            mbar_wait(smem_u32(accum_full), 0);
            tc_fence_after();
            if (warp == 2) HALO_STAMP(4);
            const int nbox = g.BN >> 5;
            const uint32_t s0 = smem_u32(smem) + (uint32_t)(sub * nbox) * 16384u;
            const uint32_t r128 = (uint32_t)row * 128u, rsw = (uint32_t)(row & 7);
            const int hc = (g.BN / 2 + 15) / 16 * 16;
            const int cbeg = half ? hc : 0, cend = half ? g.BN : hc;
            const bool has_bias = ep.bias != nullptr && blockIdx.z == 0;
            for (int c0 = cbeg; c0 < cend; c0 += 16) {
                float v[16];
                tc_ld8(trow + (uint32_t)c0, v);
                tc_ld8(trow + (uint32_t)(c0 + 8), v + 8);
                tc_ld_wait();
                if (has_bias) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] += bias_s[c0 + i];
                }
                if (ep.relu) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
                }
                const uint32_t sb = s0 + (uint32_t)(c0 >> 5) * 16384u + r128;
                const uint32_t k4 = (uint32_t)((c0 & 31) >> 2);
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    st_shared_v4(sb + (((k4 + (uint32_t)i) ^ rsw) << 4), __float_as_uint(v[4 * i]), __float_as_uint(v[4 * i + 1]), __float_as_uint(v[4 * i + 2]),
                                 __float_as_uint(v[4 * i + 3]));
            }
            fence_proxy_async();
            asm volatile("bar.sync %0, 256;" ::"r"(1 + sub) : "memory");
            if (lw == 0) {
                if (elect_one()) {
                    for (int b = 0; b < nbox; ++b) {
                        if (ep.atomic) tma_reduce_add_4d(&om.out, s0 + (uint32_t)b * 16384u, ep.out_co + n0 + 32 * b, oc1, oc2, oc3);
                        else tma_store_4d(&om.out, s0 + (uint32_t)b * 16384u, ep.out_co + n0 + 32 * b, oc1, oc2, oc3);
                    }
                    tma_store_commit();
                    tma_store_wait_read();
                }
                __syncwarp();
            }
        } else if (ep.mode == 1) {
            // ---- ConvLSTM gate epilogue, staged: every thread owns one pixel row of the accumulator (that is how tcgen05.ld hands
            // it out), but the outputs are pixel-major, so per-thread stores would scatter 16-byte pieces over 32 cache lines per
            // instruction (measured: 25.8k of the CTA's 42k cycles).  The row results go to shared memory instead -- the operand
            // ring is dead once accum_full fires -- and are written out with fully coalesced 128-bit stores.  Two warps share a
            // lane quarter (16 of the 32 channels each) so that the TMEM-load / MUFU latency chains overlap.
            const int ch0 = n_tile * 32;
            float cp[16];
            if (ep.c_prev) {                                 // issued before the accumulator wait: the main loop hides the latency
                const float4* src = reinterpret_cast<const float4*>(ep.c_prev + m * ep.C + ch0 + half * 16);
#pragma unroll
                for (int i = 0; i < 4; ++i) { const float4 v = __ldg(src + i); cp[4 * i] = v.x; cp[4 * i + 1] = v.y; cp[4 * i + 2] = v.z; cp[4 * i + 3] = v.w; }
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) cp[i] = 0.f;
            }
            mbar_wait(smem_u32(accum_full), 0);
            tc_fence_after();
            if (warp == 2) HALO_STAMP(4);
            float* G = reinterpret_cast<float*>(smem) + (size_t)sub * STG_FLOATS;     // [128][GP] gates | [128][CP] c | [128][CP] h
            float* Cc = G + 128 * GP;
            float* Hh = Cc + 128 * CP;
#pragma unroll
            for (int cc = 0; cc < 16; cc += 8) {
                const int c0 = half * 16 + cc;
                float gj[8], gi[8], gf[8], go[8], cn[8], hn[8];
                tc_ld8(trow + (uint32_t)(c0), gj);
                tc_ld8(trow + (uint32_t)(32 + c0), gi);
                tc_ld8(trow + (uint32_t)(64 + c0), gf);
                tc_ld8(trow + (uint32_t)(96 + c0), go);
                tc_ld_wait();
                if (ep.accurate) gate_math8<true>(gj, gi, gf, go, cp + cc, bias_s, c0, ep.forget_bias, cn, hn);
                else gate_math8<false>(gj, gi, gf, go, cp + cc, bias_s, c0, ep.forget_bias, cn, hn);
                if (GATES) {
                    float* gr = G + row * GP + c0;
                    *reinterpret_cast<float4*>(gr) = make_float4(gj[0], gj[1], gj[2], gj[3]);
                    *reinterpret_cast<float4*>(gr + 4) = make_float4(gj[4], gj[5], gj[6], gj[7]);
                    *reinterpret_cast<float4*>(gr + 32) = make_float4(gi[0], gi[1], gi[2], gi[3]);
                    *reinterpret_cast<float4*>(gr + 36) = make_float4(gi[4], gi[5], gi[6], gi[7]);
                    *reinterpret_cast<float4*>(gr + 64) = make_float4(gf[0], gf[1], gf[2], gf[3]);
                    *reinterpret_cast<float4*>(gr + 68) = make_float4(gf[4], gf[5], gf[6], gf[7]);
                    *reinterpret_cast<float4*>(gr + 96) = make_float4(go[0], go[1], go[2], go[3]);
                    *reinterpret_cast<float4*>(gr + 100) = make_float4(go[4], go[5], go[6], go[7]);
                }
                *reinterpret_cast<float4*>(Cc + row * CP + c0) = make_float4(cn[0], cn[1], cn[2], cn[3]);
                *reinterpret_cast<float4*>(Cc + row * CP + c0 + 4) = make_float4(cn[4], cn[5], cn[6], cn[7]);
                *reinterpret_cast<float4*>(Hh + row * CP + c0) = make_float4(hn[0], hn[1], hn[2], hn[3]);
                *reinterpret_cast<float4*>(Hh + row * CP + c0 + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
            }
            asm volatile("bar.sync %0, 256;" ::"r"(1 + sub) : "memory");          // the eight warps of this pixel tile
            if (ep.ln_partial) {
                // LayerNorm statistics of the h tile (128 pixels x 32 channels = one 4096-value chunk of the sample), two-pass in
                // shared memory, in the (mean, M2) form the LayerNorm apply kernel merges (train_model.py:203-208; layernorm_vec.cu)
                float* red = reinterpret_cast<float*>(smem) + (size_t)MS * STG_FLOATS + sub * 16;       // 8 warp sums + mean
                const int t256 = lw * 32 + lane;                                     // 0..255: row t256 >> 1, 16-channel half t256 & 1
                const float* hr = Hh + (t256 >> 1) * CP + (t256 & 1) * 16;
                float hv[16], sum = 0.f;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 v = *reinterpret_cast<const float4*>(hr + 4 * i);
                    hv[4 * i] = v.x; hv[4 * i + 1] = v.y; hv[4 * i + 2] = v.z; hv[4 * i + 3] = v.w;
                    sum += (v.x + v.y) + (v.z + v.w);
                }
                sum = warp_sum(sum);
                if (lane == 0) red[lw] = sum;
                asm volatile("bar.sync %0, 256;" ::"r"(1 + sub) : "memory");
                float tot = 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) tot += red[i];
                const float mean = tot * (1.f / 4096.f);
                float m2 = 0.f;
#pragma unroll
                for (int i = 0; i < 16; ++i) { const float d = hv[i] - mean; m2 = fmaf(d, d, m2); }
                m2 = warp_sum(m2);
                asm volatile("bar.sync %0, 256;" ::"r"(1 + sub) : "memory");          // everyone has read the sums
                if (lane == 0) red[lw] = m2;
                asm volatile("bar.sync %0, 256;" ::"r"(1 + sub) : "memory");
                if (lw == 0 && lane == 0) {
                    float t2 = 0.f;
#pragma unroll
                    for (int i = 0; i < 8; ++i) t2 += red[i];
                    const int tiles_per_img = tiles_x * tiles_y;
                    ep.ln_partial[(long)tb * ep.ln_S + (mt - tb * tiles_per_img) * (ep.C >> 5) + n_tile] = make_float2(mean, t2);
                }
            }
            if (!GATES) {
            } else if (ep.gates_bf16) {
                // bf16 gate storage: 256-byte rows, 16 lanes x 16 B per row, two rows per warp instruction
                __nv_bfloat16* gb = reinterpret_cast<__nv_bfloat16*>(ep.gates);
                const int sr = lane >> 4, l16 = lane & 15;
                for (int r0 = lw * 2; r0 < 128; r0 += 16) {
                    const int r = r0 + sr;
                    const long mr = pixel_of(r);
                    const float4 a = *reinterpret_cast<const float4*>(G + r * GP + 8 * l16), b4 = *reinterpret_cast<const float4*>(G + r * GP + 8 * l16 + 4);
                    const float v[8] = {a.x, a.y, a.z, a.w, b4.x, b4.y, b4.z, b4.w};
                    *reinterpret_cast<uint4*>(gb + mr * (4 * ep.C) + n0 + 8 * l16) = pack8_bf16(v);
                }
            } else {
                // fp32 gates: one 512-byte row per warp instruction
                for (int r = lw; r < 128; r += 8) {
                    const long mr = pixel_of(r);
                    const float4 v = *reinterpret_cast<const float4*>(G + r * GP + 4 * lane);
                    *reinterpret_cast<float4*>(ep.gates + mr * (4 * ep.C) + n0 + 4 * lane) = v;
                }
            }
            // c, h (fp32) and the bf16 shadow of h: 8 lanes per 128-byte row, four rows per warp instruction
            const int sub_r = lane >> 3, l8 = lane & 7;
            for (int r0 = lw * 4; r0 < 128; r0 += 32) {
                const int r = r0 + sub_r;
                const long mr = pixel_of(r);
                const float4 cv = *reinterpret_cast<const float4*>(Cc + r * CP + 4 * l8);
                const float4 hv = *reinterpret_cast<const float4*>(Hh + r * CP + 4 * l8);
                *reinterpret_cast<float4*>(ep.c_out + mr * ep.C + ch0 + 4 * l8) = cv;
                *reinterpret_cast<float4*>(ep.h_out + mr * ep.h_cs + ep.h_co + ch0 + 4 * l8) = hv;
                if (ep.h_bf16) {
                    __nv_bfloat162 p0 = __floats2bfloat162_rn(hv.x, hv.y), p1 = __floats2bfloat162_rn(hv.z, hv.w);
                    uint2 pk;
                    pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
                    *reinterpret_cast<uint2*>(ep.h_bf16 + mr * ep.hb_cs + ep.hb_co + ch0 + 4 * l8) = pk;
                }
                if (ep.h_t) {
                    const float hh[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) ep.h_t[(long)(ep.hT_co + ch0 + 4 * l8 + i) * ep.h_t_ld + mr] = __float2bfloat16(hh[i]);
                }
            }
        } else {
            mbar_wait(smem_u32(accum_full), 0);
            tc_fence_after();
            if (warp == 2) HALO_STAMP(4);
            // plain epilogue: the two warps of a lane quarter split the columns; rows are staged in the dead operand ring and written
            // out whole (tc_epilogue_staged).  Split-K partials (blockIdx.z > 0) carry no bias.
            const int hc = (g.BN / 2 + 7) / 8 * 8;
            const int cbeg = half ? hc : 0, cend = half ? g.BN : hc;
            TcEpilogue epz = ep;
            if (blockIdx.z != 0) epz.bias = nullptr;
            const size_t stage_floats = (size_t)128 * (g.BN + 4) + 256;           // tile + the 128-entry output-row table
            if ((size_t)MS * stage_floats * sizeof(float) <= (size_t)NP * pbuf_bytes + (size_t)g.stages * b_bytes) {
                float* stage = reinterpret_cast<float*>(smem) + (size_t)sub * stage_floats;
                tc_epilogue_staged(epz, trow, stage, row, m, cbeg, cend, n0, g.BN, bias_s, (ew & 7) * 32 + lane, 256, 1 + sub);
            } else if (cend > cbeg) {                          // two wide tiles do not fit the dead operand area: row stores
                tc_epilogue_row(epz, trow + (uint32_t)cbeg, m, m, n0 + cbeg, cend - cbeg, n_tile, bias_s + cbeg);
            }
        }
        tc_fence_before();
        if (warp == 2) HALO_STAMP(5);
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)g.tmem_cols) : "memory");
        if (g.dbg && lane == 0) g.dbg[HALO_ROW + 7] = global_ns();
    }
}

template <int MS, int NP, bool GATES>
static int launch_ms_np(const CUtensorMap& map_a, const CUtensorMap& map_b, const OutMaps& om, const Geom& g, const TcEpilogue& ep, int tiles, int splits,
                        size_t smem, void* stream, const char* who) {
    static PerDeviceOnce attr_once;            // the opt-in is per device
    if (attr_once.need()) {
        cudaError_t e = cudaFuncSetAttribute(conv5x5_halo_tc_kernel<MS, NP, GATES>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) { set_error("%s(halo): cudaFuncSetAttribute: %s", who, cudaGetErrorString(e)); return PIVP_ECUDA; }
    }
    dim3 grid((unsigned)(tiles / MS), (unsigned)(g.N / g.BN), (unsigned)splits);
    launch_k(conv5x5_halo_tc_kernel<MS, NP, GATES>, grid, dim3(64 + 256 * MS), smem, stream, map_a, map_b, om, g, ep);
    return check_launch(who);
}

template <int MS>
static int launch_ms(const CUtensorMap& map_a, const CUtensorMap& map_b, const OutMaps& om, Geom g, TcEpilogue ep, int tiles, long M, void* stream,
                     const char* who) {
    const int b_bytes = g.BN * 128;
    // one CTA per SM.  Patch buffers: up to 3 (never more than the 64-channel blocks), as long as the weight ring keeps >= 8 stages and
    // the staged gate epilogue still fits; the ring takes what the patches leave.
    // Split-K: a plain-epilogue launch that would leave most SMs idle (the 8x8-map input gradient: 16 pixel tiles, K = 25 x 512)
    // spreads its 64-channel blocks over blockIdx.z; every split adds its partial tile with vector atomics into the zeroed output.
    int ncb = g.Kc / 64, splits = 1;
    const long ctas = (long)(tiles / MS) * (g.N / g.BN);
    const char* env_sk = getenv("PIVP_TC_HALO_SPLITK");
    if (ep.mode == 0 && ep.out && !ep.out_bf16 && !ep.relu && ncb >= 4 && 2 * ctas <= 148 && (!env_sk || atoi(env_sk) != 0)) {
        splits = (int)(148 / ctas);
        if (splits > ncb / 2) splits = ncb / 2;
        if (env_sk && atoi(env_sk) > 1) splits = atoi(env_sk) < ncb ? atoi(env_sk) : ncb;
    }
    g.cb_per_split = (ncb + splits - 1) / splits;
    splits = (ncb + g.cb_per_split - 1) / g.cb_per_split;
    if (splits > 1) {
        if (!ep.accumulate) {
            cudaError_t e = cudaMemset2DAsync(ep.out + ep.out_co, (size_t)ep.out_cs * 4, 0, (size_t)g.N * 4, (size_t)M, (cudaStream_t)stream);
            if (e != cudaSuccess) { set_error("%s(halo): cudaMemset2DAsync: %s", who, cudaGetErrorString(e)); return PIVP_ECUDA; }
        }
        ep.atomic = 1;
        ncb = g.cb_per_split;
    }
    const char* env_np = getenv("PIVP_TC_HALO_NP");
    int np = env_np ? atoi(env_np) : 3;
    if (MS > 1) np = 1;                                  // two-tile CTAs: 80 KB per buffer, the ring needs the rest
    if (np > 3) np = 3;
    if (np > ncb) np = ncb;
    if (np < 1) np = 1;
    while (np > 1 && (225 * 1024 - np * MS * g.patch_bytes) / b_bytes < 8) --np;
    g.npatch = np;
    int stages = (225 * 1024 - np * MS * g.patch_bytes) / b_bytes;
    if (stages > 24) stages = 24;
    g.stages = stages;
    const int cols = MS * g.BN;
    g.tmem_cols = cols <= 32 ? 32 : cols <= 64 ? 64 : cols <= 128 ? 128 : cols <= 256 ? 256 : 512;
    const size_t smem = 1024 + (size_t)np * MS * g.patch_bytes + (size_t)stages * b_bytes + (2 * stages + 7) * 8 + 16 + (size_t)g.BN * 4;
    const size_t dead = (size_t)np * MS * g.patch_bytes + (size_t)stages * b_bytes;          // operand area, free once the accumulator is complete
    if (g.tma_out) {
        const size_t need = ep.mode == 1 ? (size_t)MS * STG_TMA + 256 : (size_t)MS * (g.BN / 32) * 16384;
        if (dead < need) g.tma_out = 0;                   // (does not happen for the ConvLSTM shapes) fall back to the register-store epilogues
    }
    PIVP_REQUIRE(!ep.ln_gamma || g.tma_out, "%s(halo): the fused LayerNorm needs the TMA-store epilogue (bf16 gate storage, bf16 h shadow, aligned views)", who);
    // the fused LayerNorm's per-sample rendezvous needs every CTA of the launch resident at once: one CTA per SM, so at most 148 of them
    PIVP_REQUIRE(!ep.ln_gamma || (long)(tiles / MS) * (g.N / g.BN) * splits <= 148, "%s(halo): fused LayerNorm with more CTAs than SMs", who);
    PIVP_REQUIRE(ep.mode != 1 || g.tma_out || dead >= (size_t)MS * STG_FLOATS * 4 + 256, "%s(halo): operand ring too small to stage the gate epilogue", who);
    if (ep.mode == 1 && !ep.gates) {                    // forward-only: the instantiation without the gate store
        if (MS == 1 && np == 3) return launch_ms_np<1, 3, false>(map_a, map_b, om, g, ep, tiles, splits, smem, stream, who);
        if (MS == 1 && np == 2) return launch_ms_np<1, 2, false>(map_a, map_b, om, g, ep, tiles, splits, smem, stream, who);
        return launch_ms_np<MS, 1, false>(map_a, map_b, om, g, ep, tiles, splits, smem, stream, who);
    }
    if (MS == 1 && np == 3) return launch_ms_np<1, 3, true>(map_a, map_b, om, g, ep, tiles, splits, smem, stream, who);
    if (MS == 1 && np == 2) return launch_ms_np<1, 2, true>(map_a, map_b, om, g, ep, tiles, splits, smem, stream, who);
    return launch_ms_np<MS, 1, true>(map_a, map_b, om, g, ep, tiles, splits, smem, stream, who);
}

}  // namespace halo

// Diagnostics (scripts/halo_timeline_all.py): while a buffer is set, launch number k since the call writes its per-CTA stamps
// ([0..5] clock64 of the phases, [6] / [7] %globaltimer at CTA start / end) to rows [256 k, 256 k + CTAs); at most 512 launches.
static long long* g_halo_dbg = nullptr;
static int g_halo_dbg_launch = 0;
void tc_halo_set_debug(long long* p) { g_halo_dbg = p; g_halo_dbg_launch = 0; }

// PIVP_TC_HALO: 0 = use the per-tap kernel of conv_tc.cu, 1 = default, 3 = always one tile per CTA, 4 = always two (tuning switches)
int tc_halo_mode() {
    const char* v = getenv("PIVP_TC_HALO");
    return v ? atoi(v) : 1;
}

bool tc_halo_supported(int B, int H, int W, int Kc, int BN) {
    const bool tiled = W % halo::TW == 0 && H % halo::TH == 0;
    const bool pair = W == 8 && H == 8 && B % 2 == 0 && tc_halo_mode() != 5;      // 5 = pair geometry off (tuning switch)
    return tc_halo_mode() != 0 && (tiled || pair) && Kc % 64 == 0 && BN % 16 == 0 && BN >= 16 && BN <= 256 && B > 0;
}

int launch_conv5x5_halo(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, const void* wt_bf16, int N, int BN, TcEpilogue ep,
                        void* stream, const char* who) {
    using namespace halo;
    PIVP_REQUIRE(in_bf16 && wt_bf16 && in_cs % 8 == 0 && N % BN == 0, "%s(halo): bad operand", who);
    Geom g;
    g.H = H; g.W = W; g.Kc = Kc; g.N = N; g.BN = BN;
    g.dbg = (g_halo_dbg && g_halo_dbg_launch < 512) ? g_halo_dbg + (size_t)256 * 8 * g_halo_dbg_launch++ : nullptr;
    g.pair = (H == 8 && W == 8) ? 1 : 0;
    g.patch_bytes = g.pair ? PAIR_PATCH_BYTES : PATCH_BYTES;
    PIVP_REQUIRE(!g.pair || !ep.ln_partial, "%s(halo): no LayerNorm partials in the 8x8 pair geometry (a tile spans two samples)", who);
    CUtensorMap map_a, map_b;
    {
        cuuint64_t dims[4] = {(cuuint64_t)in_cs, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
        cuuint64_t str[3] = {(cuuint64_t)in_cs * 2, (cuuint64_t)W * in_cs * 2, (cuuint64_t)H * W * in_cs * 2};
        cuuint32_t box[4] = {64u, (cuuint32_t)PW, (cuuint32_t)PH, 1u};
        if (g.pair) {                      // (channel, x, image, y): the two images' rows interleave in the patch
            dims[2] = (cuuint64_t)B; dims[3] = (cuuint64_t)H;
            str[1] = (cuuint64_t)H * W * in_cs * 2; str[2] = (cuuint64_t)W * in_cs * 2;
            box[2] = 2u; box[3] = 12u;
        }
        CUresult r = encode_tmap(&map_a, in_bf16, 4, dims, str, box);
        if (r != CUDA_SUCCESS) { set_error("%s(halo): cuTensorMapEncodeTiled(A) failed (%d)", who, (int)r); return PIVP_ECUDA; }
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)25 * Kc, (cuuint64_t)N};
        cuuint64_t str[1] = {(cuuint64_t)25 * Kc * 2};
        cuuint32_t box[2] = {64u, (cuuint32_t)BN};
        CUresult r = encode_tmap(&map_b, wt_bf16, 2, dims, str, box);
        if (r != CUDA_SUCCESS) { set_error("%s(halo): cuTensorMapEncodeTiled(B) failed (%d)", who, (int)r); return PIVP_ECUDA; }
    }
    // ---- output tensor maps of the TMA-store epilogues (PIVP_TC_HALO_TMA=0: per-thread stores as before)
    OutMaps om;
    memset(&om, 0, sizeof(om));
    g.tma_out = 0;
    {
        const char* env = getenv("PIVP_TC_HALO_TMA");
        const bool want = !env || atoi(env) != 0;
        auto a16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
        // (channel, x, y, image) view of an NHWC tensor with row stride cs (elements of esz bytes); pair geometry: (channel, x, image, y)
        auto enc = [&](CUtensorMap* mp, CUtensorMapDataType dt, CUtensorMapSwizzle sw, const void* base, int cs, int esz, int boxc) -> bool {
            cuuint64_t dims[4] = {(cuuint64_t)cs, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
            cuuint64_t str[3] = {(cuuint64_t)cs * esz, (cuuint64_t)W * cs * esz, (cuuint64_t)H * W * cs * esz};
            cuuint32_t box[4] = {(cuuint32_t)boxc, (cuuint32_t)TW, (cuuint32_t)TH, 1u};
            if (g.pair) {
                dims[2] = (cuuint64_t)B; dims[3] = (cuuint64_t)H;
                str[1] = (cuuint64_t)H * W * cs * esz; str[2] = (cuuint64_t)W * cs * esz;
                box[2] = 2u; box[3] = 8u;
            }
            return encode_tmap_ex(mp, dt, sw, base, 4, dims, str, box) == CUDA_SUCCESS;
        };
        // (no gate map without gate storage: forward-only launches, ep.gates == null)
        if (want && ep.mode == 1 && (!ep.gates || (ep.gates_bf16 && a16(ep.gates))) && ep.h_bf16 && !ep.h_t && a16(ep.c_out) && a16(ep.h_out) &&
            a16(ep.h_bf16) && ep.C % 4 == 0 && ep.h_cs % 4 == 0 && ep.hb_cs % 8 == 0) {
            g.tma_out = (!ep.gates || enc(&om.gates, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_128B, ep.gates, 4 * ep.C, 2, 64)) &&
                        enc(&om.c, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, CU_TENSOR_MAP_SWIZZLE_128B, ep.c_out, ep.C, 4, 32) &&
                        enc(&om.h, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, CU_TENSOR_MAP_SWIZZLE_128B, ep.h_out, ep.h_cs, 4, 32) &&
                        enc(&om.hb, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_64B, ep.h_bf16, ep.hb_cs, 2, 32);
            if (g.tma_out && ep.ln_gamma) {
                PIVP_REQUIRE(ep.ln_partial && ep.ln_beta && ep.ln_y && ep.ln_stats && ep.ln_counter && !g.pair && a16(ep.ln_y) && ep.ln_y_cs % 4 == 0 &&
                             ep.ln_y_co % 4 == 0 && a16(ep.ln_gamma) && a16(ep.ln_beta) &&
                             (!ep.ln_yb || (a16(ep.ln_yb) && ep.ln_yb_cs % 8 == 0 && ep.ln_yb_co % 8 == 0)),
                             "%s(halo): fused LayerNorm needs the statistics partials, 16-byte aligned views and the tiled geometry", who);
                const bool ok = enc(&om.y, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, CU_TENSOR_MAP_SWIZZLE_128B, ep.ln_y, ep.ln_y_cs, 4, 32) &&
                                (!ep.ln_yb || enc(&om.yb, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_64B, ep.ln_yb, ep.ln_yb_cs, 2, 32));
                PIVP_REQUIRE(ok, "%s(halo): cuTensorMapEncodeTiled failed for the fused LayerNorm outputs", who);
            }
        } else if (want && ep.mode == 0 && ep.out && !ep.out_bf16 && !ep.accumulate && BN % 32 == 0 && a16(ep.out) && ep.out_cs % 4 == 0) {
            g.tma_out = enc(&om.out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, CU_TENSOR_MAP_SWIZZLE_128B, ep.out, ep.out_cs, 4, 32);
        }
    }
    const int tiles = g.pair ? B / 2 : B * (H / TH) * (W / TW);
    // two pixel tiles per CTA halve the weight traffic per FLOP; only worth it while the grid still covers most of the SMs
    const int force = tc_halo_mode();
    const bool two = (force == 3) ? false : (tiles % 2 == 0 && 2 * BN <= 512 && ((tiles / 2) * (N / BN) >= 96 || force == 4));
    const long M = (long)B * H * W;
    return two ? launch_ms<2>(map_a, map_b, om, g, ep, tiles, M, stream, who) : launch_ms<1>(map_a, map_b, om, g, ep, tiles, M, stream, who);
}

}  // namespace pivp
