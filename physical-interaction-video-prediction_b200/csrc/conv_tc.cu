// tcgen05 / TMEM / TMA implicit-GEMM 5x5 convolution for the seven ConvLSTM layers (bf16 operands, fp32 accumulate).
//
// Replaces the `self.conv(inputs_h)` + gate math of BasicConvLSTMCell (train_model.py:262-272) in the forward pass,
// and Chainer's Convolution2D input-gradient (SURVEY D.5) in the backward pass.  Both are the same stride-1 "same"
// convolution over an NHWC bf16 tensor:
//      D[m, n] = sum_{tap=(dy,dx), c} In[pixel(m) + (dy-2, dx-2), c] * Wt[n][tap][c]
// (for the input gradient the caller passes dG as `In` and a tap-flipped, transposed weight -- see pivp_tc_prep_weights).
//
// GEMM view: M = B*H*W pixels (128 per CTA), N = output channels (BN <= 256 per CTA), K = 25 taps x Kc channels.
//  * A tile: one 4-D TMA box {64 ch, TW, TH, TB} (TW*TH*TB = 128 pixels) per (tap, 64-channel block), fetched at the
//    tap-shifted coordinate; out-of-image pixels are zero-filled by TMA, which IS the convolution's zero padding.
//    The box lands in shared memory as 128 rows x 128 B with the 128-byte swizzle = the canonical K-major UMMA layout.
//  * B tile: 2-D TMA box {64, BN} of the K-major weight matrix [N][25*Kc].
//  * tcgen05.mma (cta_group::1, kind::f16, M=128, N=BN, K=16) issued by one elected thread, accumulator in TMEM.
//  * Warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..5 = epilogue (one TMEM lane
//    quarter each).  smem ring of `stages` slots with full/empty mbarriers; tcgen05.commit frees slots.
//  * Epilogue mode 1 (ConvLSTM forward): bias + gates + cell update + h fused -- the pre-activations never reach HBM.
//    N is ordered [32-channel block][gate j,i,f,o][channel], so one 128-column tile holds all four gates of 32 channels.
//  * Two CTAs are resident per SM (<= 110 KB smem, <= 256 TMEM columns each), so one CTA's epilogue overlaps the other's
//    main loop without an in-kernel tile scheduler.
#include "tc_common.cuh"
#include "tc_epilogue.cuh"

namespace pivp {

constexpr int TC_BM = 128;          // pixels per CTA (TMEM lanes)
constexpr int TC_BK = 64;           // bf16 elements per k-block row = 128 B = one swizzle span
constexpr int TC_THREADS = 192;

constexpr int TC_MAXTAPS = 25;
struct TcGeom {
    int H, W, TW, TH, TB;        // pixel grid the M tiles walk (A-operand grid), pixel box of one M tile
    int Kc;                      // contracted channels per tap (multiple of 64)
    int N, BN;                   // output channels, tile width
    int stages;
    int tmem_cols;
    int ntaps;                   // K = ntaps * Kc
    signed char dy[TC_MAXTAPS], dx[TC_MAXTAPS];   // pixel offset of each tap on the A grid
    short coff[TC_MAXTAPS];                       // channel offset of each tap inside the A rows
    // plain-epilogue row mapping: A-grid pixel (b,i,j) -> output row ((b*OH + i*os + oa)*OW + j*os + ob)
    int OH, OW, os, oa, ob;
};

// Up to four independent tap lists ("phases": the output phases of a stride-2 transposed convolution) share one launch:
// blockIdx.z picks the weight tensor map and the geometry; the A tensor, tile counts and epilogue are common.
constexpr int TC_MAXPH = 4;
struct TcMapsB { CUtensorMap m[TC_MAXPH]; };
struct TcMapsOut { CUtensorMap m[TC_MAXPH]; };   // per phase: the output seen as (channel, x', y', image) of the A grid (strides os pixels)
struct TcGeomPack {
    TcGeom g[TC_MAXPH];
    int out_bytes;   // > 0: the epilogue stages its tile in the first out_bytes of shared memory and writes it with TMA stores (maps_o)
    int out_b_off;   // > 0: offset of the bf16 copy's staging tiles inside that region (maps_ob)
    int nloop;       // 1: one phase per CTA (blockIdx.z picks it).  n > 1: every CTA walks phases 0..n-1 of its pixel tile, one TMEM
                     // accumulator of BN columns per phase (grid z = 1) -- a quarter of the CTAs, so a 64x64 deconvolution is ONE wave
};

// GATES = false: mode 1 without the gate store (pivp_tc_conv5x5 flags bit 2, ep.gates == null)
template <bool GATES>
__global__ void __launch_bounds__(TC_THREADS, 2)
conv_taps_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ TcMapsB maps_b, const __grid_constant__ TcMapsOut maps_o,
                    const __grid_constant__ TcMapsOut maps_ob, const __grid_constant__ TcGeomPack gp, TcEpilogue ep) {
    const TcGeom& g = gp.g[blockIdx.z];            // fields common to all phases (tile geometry, Kc, BN, ring depth, TMEM columns)
    const int nloop = gp.nloop;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // carve: [output staging, out_bytes] [stages][A 16 KB | B BN*128] then barriers
    uint8_t* smem_base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* smem = smem_base + gp.out_bytes;        // the operand ring
    const uint32_t a_bytes = TC_BM * 128, b_bytes = (uint32_t)g.BN * 128, stage_bytes = a_bytes + b_bytes;
    uint64_t* bars = (uint64_t*)(smem + (size_t)g.stages * stage_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + g.stages;
    uint64_t* accum_full = bars + 2 * g.stages;     // [TC_MAXPH]: one per phase accumulator
    uint32_t* tmem_slot = (uint32_t*)(bars + 2 * g.stages + TC_MAXPH);
    float* bias_s = (float*)(tmem_slot + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tile = blockIdx.x, n_tile = blockIdx.y;
    const int n0 = n_tile * g.BN;
    const int kblocks_per_tap = g.Kc / TC_BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) { mbar_init(smem_u32(full + s), 1); mbar_init(smem_u32(empty + s), 1); }
        for (int p = 0; p < TC_MAXPH; ++p) mbar_init(smem_u32(accum_full + p), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // descriptor fetches overlap the set-up and the wait for the previous kernel instead of preceding the first operand load
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        for (int p = 0; p < nloop; ++p) asm volatile("prefetch.tensormap [%0];" ::"l"(&maps_b.m[blockIdx.z + p]) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)g.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    pdl_wait();                                      // everything above is independent of the previous kernel's output
    if (warp >= 2 && ep.bias) {
        for (int i = threadIdx.x - 64; i < g.BN; i += 128) bias_s[i] = ep.bias[n0 + i];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // Warp-uniform producer / issuer loops with one elected lane (see conv_tc_halo.cu: a `lane == 0` branch makes ptxas wrap every
    // tcgen05.mma in a per-lane waterfall loop, ~20 issue slots per MMA).
    if (warp == 0) {
        // ===================== TMA producer =====================
        // first pixel of this M tile: tiles walk x fastest, then y, then batch
        const int tiles_x = g.W / g.TW, tiles_y = g.H / g.TH;
        const int tx = m_tile % tiles_x, ty = (m_tile / tiles_x) % tiles_y, tb = m_tile / (tiles_x * tiles_y);
        const int x0 = tx * g.TW, y0 = ty * g.TH, b0 = tb * g.TB;
        const uint32_t full0 = smem_u32(full), empty0 = smem_u32(empty), ring0 = smem_u32(smem);
        uint32_t st = 0, ph = 1;
        for (int p = 0; p < nloop; ++p) {
            const TcGeom& gq = gp.g[blockIdx.z + p];
            const CUtensorMap& map_b = maps_b.m[blockIdx.z + p];
            for (int tap = 0; tap < gq.ntaps; ++tap) {
                const int cx = x0 + gq.dx[tap], cy = y0 + gq.dy[tap], cc = gq.coff[tap];
                for (int cb = 0; cb < kblocks_per_tap; ++cb) {
                    mbar_wait(empty0 + 8 * st, ph);
                    if (elect_one()) {
                        const uint32_t sa = ring0 + st * stage_bytes;
                        mbar_expect_tx(full0 + 8 * st, stage_bytes);
                        tma_load_4d(sa, &map_a, full0 + 8 * st, cc + cb * TC_BK, cx, cy, b0);
                        tma_load_2d(sa + a_bytes, &map_b, full0 + 8 * st, tap * g.Kc + cb * TC_BK, n0);
                    }
                    __syncwarp();
                    if (++st == (uint32_t)g.stages) { st = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        // instruction descriptor: D=f32, A=B=bf16, both K-major, N>>3 at [17,23), M>>4 at [24,29)
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(g.BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);           // SBO | version 1 | SWIZZLE_128B
        const uint32_t ring_lo = ((smem_u32(smem) & 0x3FFFFu) >> 4) | 0x10000u, step_lo = stage_bytes >> 4, a_lo_sz = a_bytes >> 4;
        const uint32_t full0 = smem_u32(full), empty0 = smem_u32(empty);
        uint32_t st = 0, ph = 0, lo = ring_lo;
        for (int p = 0; p < nloop; ++p) {
            const int num_kb = gp.g[blockIdx.z + p].ntaps * kblocks_per_tap;
            const uint32_t acc = tmem_u + (uint32_t)(p * g.BN);      // this phase's accumulator columns
            for (int kb = 0; kb < num_kb; ++kb) {
                mbar_wait(full0 + 8 * st, ph);
                tc_fence_after();
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < TC_BK / 16; ++k)      // advance 16 bf16 = 32 B = 2 (>>4 units) inside the swizzle span
                        tc_mma_lohi(acc, lo + 2 * k, lo + a_lo_sz + 2 * k, hi, hi, idesc, (k == 0) ? (kb ? 1u : 0u) : 1u);
                    tc_commit(empty0 + 8 * st);               // frees the smem slot when these MMAs retire
                    if (kb == num_kb - 1) tc_commit(smem_u32(accum_full + p));
                }
                __syncwarp();
                lo += step_lo;
                if (++st == (uint32_t)g.stages) { st = 0; ph ^= 1u; lo = ring_lo; }
            }
        }
    } else {
        // ===================== epilogue (warps 2..5) =====================
        const int q = warp & 3;                            // TMEM lane quarter this warp may read
        const int row = q * 32 + lane;
        const long m = (long)m_tile * TC_BM + row;
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
        // output row of this A-grid pixel (identity for stride-1 convs, phase scatter for transposed convs)
        const int hw = g.H * g.W;
        const int bi = (int)(m / hw), rem = (int)(m - (long)bi * hw);
        const int iy = rem / g.W, ix = rem - iy * g.W;
        for (int p = 0; p < nloop; ++p) {                  // phase p's epilogue overlaps phase p+1's MMAs
            const TcGeom& gq = gp.g[blockIdx.z + p];
            mbar_wait(smem_u32(accum_full + p), 0);
            tc_fence_after();
            const long orow = ((long)bi * g.OH + iy * g.os + gq.oa) * g.OW + ix * g.os + gq.ob;
            // (the staged, coalesced write-out of tc_epilogue_staged was measured here too: +0.2 ms per step -- with 4 epilogue warps and
            // rows of <= 128 channels the extra shared-memory round trip costs more than the scattered 16-byte stores)
            if (gp.out_bytes) {
                // staged tile + TMA stores (one box of 32 fp32 columns x 128 pixels per store) into phase p's strided view of the output
                float2* red = reinterpret_cast<float2*>(bias_s + g.BN) + p * 32;
                if (p > 0) {                                                   // the previous phase's stores have read the staging tile
                    if (warp == 2) { if (elect_one()) tma_store_wait_read(); __syncwarp(); }
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                }
                const uint32_t stage = smem_u32(smem_base), stage_b = gp.out_b_off ? stage + (uint32_t)gp.out_b_off : 0u;
                if (ep.ln_partial) tc_epilogue_row_stage<true>(ep, trow + (uint32_t)(p * g.BN), g.BN, bias_s, stage, row, red, q, lane, stage_b);
                else tc_epilogue_row_stage<false>(ep, trow + (uint32_t)(p * g.BN), g.BN, bias_s, stage, row, red, q, lane, stage_b);
                fence_proxy_async();
                asm volatile("bar.sync 1, 128;" ::: "memory");                 // the four epilogue warps: tile (and statistics) complete
                if (warp == 2) {
                    if (elect_one()) {
                        const int tiles_x = g.W / g.TW, tiles_y = g.H / g.TH;
                        const int tx = m_tile % tiles_x, ty = (m_tile / tiles_x) % tiles_y, tb = m_tile / (tiles_x * tiles_y);
                        for (int b = 0; b < (g.BN >> 5); ++b) {
                            tma_store_4d(&maps_o.m[blockIdx.z + p], stage + (uint32_t)b * 16384u, ep.out_co + n0 + 32 * b, tx * g.TW, ty * g.TH, tb * g.TB);
                            if (stage_b)
                                tma_store_4d(&maps_ob.m[blockIdx.z + p], stage_b + (uint32_t)b * 8192u, ep.ob_co + n0 + 32 * b, tx * g.TW, ty * g.TH, tb * g.TB);
                        }
                        tma_store_commit();
                        if (p == nloop - 1) tma_store_wait_read();             // shared memory must outlive the bulk reads
                    }
                    __syncwarp();
                }
            }
            if (ep.ln_partial) {
                // statistics of the LayerNorm behind this deconvolution: one (mean, M2) pair per (tile, phase, 32-column group)
                float2* red = reinterpret_cast<float2*>(bias_s + g.BN) + p * 32;
                if (!gp.out_bytes) {
                    tc_epilogue_row_ln(ep, trow + (uint32_t)(p * g.BN), orow, n0, g.BN, bias_s, red, q, lane);
                    asm volatile("bar.sync 1, 128;" ::: "memory");             // the four epilogue warps
                }
                const int grp = (int)threadIdx.x - 64;
                if (grp < (g.BN >> 5)) {
                    const float2 a = red[grp * 4], b = red[grp * 4 + 1], c = red[grp * 4 + 2], e = red[grp * 4 + 3];
                    const float dab = b.x - a.x, dce = e.x - c.x;                // 1024 values each, then 2048 + 2048
                    const float mab = 0.5f * (a.x + b.x), mce = 0.5f * (c.x + e.x);
                    const float sab = (a.y + b.y) + dab * dab * 512.f, sce = (c.y + e.y) + dce * dce * 512.f;
                    const float dd = mce - mab;
                    const int tiles_per_img = hw / TC_BM, nphases = nloop > 1 ? nloop : (int)gridDim.z;
                    const int tile_in = m_tile - bi * tiles_per_img;            // a tile never straddles samples (H * W is a multiple of 128)
                    ep.ln_partial[(long)bi * ep.ln_S + ((long)(tile_in * nphases + (int)blockIdx.z + p)) * (g.N >> 5) + (n0 >> 5) + grp] =
                        make_float2(0.5f * (mab + mce), (sab + sce) + dd * dd * 1024.f);
                }
            } else if (!gp.out_bytes) {
                tc_epilogue_row<GATES>(ep, trow + (uint32_t)(p * g.BN), m, orow, n0, g.BN, n_tile, bias_s);
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)g.tmem_cols) : "memory");
    }
}

// ------------------------------------------------------------------------------------------ weight preparation
// fp32 master W[n][tap][c] (c < Cx)  ->  bf16 forward operand  Wf[n][tap][Kpad]  (zero padded to Kpad channels)
//                                    ->  bf16 dgrad operand    Wd[c][tap'][n] = W[n][24 - tap'][c]
__global__ void tc_prep_weights_kernel(const float* __restrict__ W, int N, int Cx, int Kpad, __nv_bfloat16* __restrict__ Wf,
                                       __nv_bfloat16* __restrict__ Wd) {
    pdl_enter();
    const long total_f = (long)N * 25 * Kpad;
    const long total_d = (long)Cx * 25 * N;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total_f + total_d; i += (long)gridDim.x * blockDim.x) {
        if (i < total_f) {
            if (!Wf) continue;
            const int c = (int)(i % Kpad);
            const long r = i / Kpad;                    // n*25 + tap
            Wf[i] = __float2bfloat16(c < Cx ? W[r * Cx + c] : 0.f);
        } else {
            if (!Wd) continue;
            const long jx = i - total_f;
            const int n = (int)(jx % N);
            const long r = jx / N;                      // c*25 + tap'
            const int tp = (int)(r % 25), c = (int)(r / 25);
            Wd[jx] = __float2bfloat16(W[((long)n * 25 + (24 - tp)) * Cx + c]);
        }
    }
}

static int pick_pixel_box(int B, int H, int W, int* TW, int* TH, int* TB) {
    // 128 consecutive NHWC pixels that form a box: full rows (TW = W), then rows, then whole images
    if (W > 128 || 128 % W) return -1;
    *TW = W;
    int th = 128 / W;
    if (th > H) th = H;
    if (H % th) return -1;
    *TH = th;
    const int tb = 128 / (W * th);
    if (tb > 1 && th != H) return -1;
    if (B % tb) return -1;
    *TB = tb;
    return 0;
}

// dst[i] = bf16(src[idx[i]]), idx < 0 -> 0.  Builds any permuted / zero-padded bf16 weight operand from the fp32 master.
__global__ void gather_bf16_kernel(const float* __restrict__ src, const int* __restrict__ idx, long n, __nv_bfloat16* __restrict__ dst) {
    pdl_enter();
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const int j = idx[i];
        dst[i] = __float2bfloat16(j >= 0 ? src[j] : 0.f);
    }
}

struct TapPhase {
    int ntaps;
    const int *dy, *dx, *coff;
    const void* wt_bf16;
    int oa, ob;
};

static int launch_conv_taps_multi(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, int nph, const TapPhase* ph, int N, int BN,
                                  TcEpilogue ep, int OH, int OW, int os, void* stream, const char* who) {
    PIVP_REQUIRE(in_bf16 && nph >= 1 && nph <= TC_MAXPH, "%s: null operand or bad phase count", who);
    PIVP_REQUIRE(Kc > 0 && Kc % TC_BK == 0 && in_cs % 8 == 0, "%s: Kc must be a multiple of 64 and rows 16-byte aligned", who);
    PIVP_REQUIRE(BN >= 16 && BN <= 256 && BN % 16 == 0 && N % BN == 0, "%s: BN must be a multiple of 16 <= 256 dividing N", who);
    int TW, TH, TB;
    if (pick_pixel_box(B, H, W, &TW, &TH, &TB) != 0) {
        set_error("%s: cannot tile B=%d H=%d W=%d into 128-pixel boxes", who, B, H, W);
        return PIVP_EUNSUPPORTED;
    }
    const int stage_bytes = TC_BM * 128 + BN * 128;
    // ring depth: at most one CTA per SM fits anyway when the grid is <= 148 CTAs, so a small launch takes the whole shared memory
    // (the 8x8-map layers were bound by 3 stages x ~1.5 us TMA round trip, not by the MMAs); larger grids leave room for two CTAs per SM
    long ctas = ((long)B * H * W / TC_BM) * (N / BN) * nph;
    // more than one wave of two CTAs per SM and room for every phase's accumulator: let each CTA walk all phases of its tile
    static const int fuse_env = getenv("PIVP_TC_TAPS_FUSE_PH") ? atoi(getenv("PIVP_TC_TAPS_FUSE_PH")) : 1;
    const bool fuse_ph = fuse_env && nph > 1 && ctas > 2 * 148 && nph * BN <= 256;
    if (fuse_ph) ctas /= nph;
    // a plain fp32 output (no bf16 copy, no accumulate): the epilogue stages each tile in shared memory and writes it with TMA stores
    // (PIVP_TC_TAPS_TMA: 0 = per-thread stores, 1 = only the launches that walk their phases inside the CTA, 2 = every eligible launch;
    //  measured on the b32 step: 7.05 / 7.00 / 6.95 ms)
    static const int tma_env = getenv("PIVP_TC_TAPS_TMA") ? atoi(getenv("PIVP_TC_TAPS_TMA")) : 2;
    const bool bf16_ok = !ep.out_bf16 || (tma_env >= 3 && !(reinterpret_cast<uintptr_t>(ep.out_bf16) & 15) && ep.ob_cs % 8 == 0 && ep.ob_co % 8 == 0);
    const bool tma_out = tma_env && (fuse_ph || tma_env >= 2) && ep.mode == 0 && ep.out && bf16_ok && !ep.accumulate && !ep.atomic && BN % 32 == 0 &&
                         !(reinterpret_cast<uintptr_t>(ep.out) & 15) && ep.out_cs % 4 == 0 && ep.out_co % 4 == 0;
    // (two CTAs per SM share 227 KB: a staging area above 48 KB would leave the operand ring a single stage -- keep the per-thread stores there)
    const int want_bytes = (BN / 32) * 16384 + (ep.out_bf16 ? (BN / 32) * 8192 : 0);
    const bool tma_fits = ctas <= 148 || want_bytes <= 48 * 1024;
    const int out_b_off = tma_out && tma_fits && ep.out_bf16 ? (BN / 32) * 16384 : 0;
    const int out_bytes = tma_out && tma_fits ? want_bytes : 0;
    const int env_ring = getenv("PIVP_TC_TAPS_RING_KB") ? atoi(getenv("PIVP_TC_TAPS_RING_KB")) : 0;
    int stages = ((env_ring > 0 ? env_ring : ctas <= 148 ? 190 : out_bytes ? 108 : 100) * 1024 - out_bytes) / stage_bytes;      // two CTAs per SM: <= ~112 KB each
    if (stages > 8) stages = 8;
    if (stages < 2) stages = 2;
    TcGeomPack gp;                                 // by-value kernel parameters
    TcMapsB mb;
    memset(&gp, 0, sizeof(gp));
    memset(&mb, 0, sizeof(mb));
    CUtensorMap map_a;
    {
        cuuint64_t dims[4] = {(cuuint64_t)in_cs, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
        cuuint64_t str[3] = {(cuuint64_t)in_cs * 2, (cuuint64_t)W * in_cs * 2, (cuuint64_t)H * W * in_cs * 2};
        cuuint32_t box[4] = {(cuuint32_t)TC_BK, (cuuint32_t)TW, (cuuint32_t)TH, (cuuint32_t)TB};
        CUresult r = encode_tmap(&map_a, in_bf16, 4, dims, str, box);
        if (r != CUDA_SUCCESS) { set_error("%s: cuTensorMapEncodeTiled(A) failed (%d)", who, (int)r); return PIVP_ECUDA; }
    }
    for (int p = 0; p < nph; ++p) {
        const TapPhase& q = ph[p];
        PIVP_REQUIRE(q.wt_bf16 && q.ntaps >= 1 && q.ntaps <= TC_MAXTAPS, "%s: phase %d: null weights or tap count outside 1..25", who, p);
        TcGeom& g = gp.g[p];
        g.H = H; g.W = W; g.TW = TW; g.TH = TH; g.TB = TB; g.Kc = Kc; g.N = N; g.BN = BN; g.ntaps = q.ntaps;
        for (int t = 0; t < q.ntaps; ++t) {
            PIVP_REQUIRE(q.dy[t] >= -64 && q.dy[t] <= 64 && q.dx[t] >= -64 && q.dx[t] <= 64 && q.coff[t] >= 0 && q.coff[t] + Kc <= in_cs &&
                             q.coff[t] % 8 == 0,
                         "%s: phase %d tap %d out of range", who, p, t);
            g.dy[t] = (signed char)q.dy[t]; g.dx[t] = (signed char)q.dx[t]; g.coff[t] = (short)q.coff[t];
        }
        g.OH = OH; g.OW = OW; g.os = os; g.oa = q.oa; g.ob = q.ob;
        g.stages = stages;
        const int cols = fuse_ph ? nph * BN : BN;
        g.tmem_cols = cols <= 32 ? 32 : cols <= 64 ? 64 : cols <= 128 ? 128 : 256;
        cuuint64_t dims[2] = {(cuuint64_t)q.ntaps * Kc, (cuuint64_t)N};
        cuuint64_t str[1] = {(cuuint64_t)q.ntaps * Kc * 2};
        cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)BN};
        CUresult r = encode_tmap(&mb.m[p], q.wt_bf16, 2, dims, str, box);
        if (r != CUDA_SUCCESS) { set_error("%s: cuTensorMapEncodeTiled(B%d) failed (%d)", who, p, (int)r); return PIVP_ECUDA; }
    }
    gp.nloop = fuse_ph ? nph : 1;
    gp.out_bytes = out_bytes;
    gp.out_b_off = out_b_off;
    TcMapsOut mo, mob;
    memset(&mo, 0, sizeof(mo));
    memset(&mob, 0, sizeof(mob));
    if (out_bytes) {
        for (int p = 0; p < nph; ++p) {                    // phase p writes pixels (i * os + oa, j * os + ob): a strided view with its own base
            const float* base = ep.out + ((long)ph[p].oa * OW + ph[p].ob) * ep.out_cs;
            cuuint64_t dims[4] = {(cuuint64_t)ep.out_cs, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
            cuuint64_t str[3] = {(cuuint64_t)os * ep.out_cs * 4, (cuuint64_t)os * OW * ep.out_cs * 4, (cuuint64_t)OH * OW * ep.out_cs * 4};
            cuuint32_t box[4] = {32u, (cuuint32_t)TW, (cuuint32_t)TH, (cuuint32_t)TB};
            CUresult r = encode_tmap_ex(&mo.m[p], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, CU_TENSOR_MAP_SWIZZLE_128B, base, 4, dims, str, box);
            if (r != CUDA_SUCCESS) { set_error("%s: cuTensorMapEncodeTiled(out%d) failed (%d)", who, p, (int)r); return PIVP_ECUDA; }
            if (ep.out_bf16) {
                const __nv_bfloat16* bb = ep.out_bf16 + ((long)ph[p].oa * OW + ph[p].ob) * ep.ob_cs;
                cuuint64_t dimb[4] = {(cuuint64_t)ep.ob_cs, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
                cuuint64_t strb[3] = {(cuuint64_t)os * ep.ob_cs * 2, (cuuint64_t)os * OW * ep.ob_cs * 2, (cuuint64_t)OH * OW * ep.ob_cs * 2};
                r = encode_tmap_ex(&mob.m[p], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_64B, bb, 4, dimb, strb, box);
                if (r != CUDA_SUCCESS) { set_error("%s: cuTensorMapEncodeTiled(out_bf16 %d) failed (%d)", who, p, (int)r); return PIVP_ECUDA; }
            }
        }
    }
    if (ep.ln_partial) {
        PIVP_REQUIRE(ep.mode == 0 && !ep.relu && !ep.accumulate && !ep.atomic && BN % 32 == 0 && N % 32 == 0 && (H * W) % TC_BM == 0 && TB == 1,
                     "%s: LayerNorm statistics need a plain store, 32-column groups and tiles inside one sample", who);
        ep.ln_S = (H * W / TC_BM) * nph * (N / 32);
    }
    const size_t smem = 1024 + (size_t)out_bytes + (size_t)stages * stage_bytes + (2 * stages + TC_MAXPH) * 8 + 16 + (size_t)BN * 4 + TC_MAXPH * 32 * sizeof(float2);
    static PerDeviceOnce attr_once;            // the opt-in is per device
    if (attr_once.need()) {
        cudaError_t e = cudaFuncSetAttribute(conv_taps_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_taps_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) { set_error("%s: cudaFuncSetAttribute: %s", who, cudaGetErrorString(e)); return PIVP_ECUDA; }
    }
    const long M = (long)B * H * W;
    dim3 grid((unsigned)(M / TC_BM), (unsigned)(N / BN), (unsigned)(fuse_ph ? 1 : nph));
    if (ep.mode == 1 && !ep.gates) launch_k(conv_taps_tc_kernel<false>, grid, dim3(TC_THREADS), smem, stream, map_a, mb, mo, mob, gp, ep);
    else launch_k(conv_taps_tc_kernel<true>, grid, dim3(TC_THREADS), smem, stream, map_a, mb, mo, mob, gp, ep);
    return check_launch(who);
}

static int launch_conv_taps(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, int ntaps, const int* dy, const int* dx, const int* coff,
                            const void* wt_bf16, int N, int BN, TcEpilogue ep, int OH, int OW, int os, int oa, int ob, void* stream,
                            const char* who) {
    PIVP_REQUIRE(in_bf16 && wt_bf16, "%s: null operand", who);
    TapPhase ph{ntaps, dy, dx, coff, wt_bf16, oa, ob};
    return launch_conv_taps_multi(in_bf16, in_cs, B, H, W, Kc, 1, &ph, N, BN, ep, OH, OW, os, stream, who);
}

// halo-patch variant (conv_tc_halo.cu): A operand staged once per 64-channel block instead of once per tap
bool tc_halo_supported(int B, int H, int W, int Kc, int BN);
void tc_halo_set_debug(long long* p);
int launch_conv5x5_halo(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, const void* wt_bf16, int N, int BN, TcEpilogue ep,
                        void* stream, const char* who);

}  // namespace pivp

using namespace pivp;

extern "C" {

/* Debugging aid: device buffer of [CTAs][8] long long that the halo kernel fills with clock64() stamps (null = off). */
int pivp_tc_set_debug_buffer(void* p) { tc_halo_set_debug((long long*)p); return PIVP_OK; }

int pivp_tc_prep_weights(const float* W, int N, int Cx, int Kpad, void* w_fwd_bf16, void* w_dgrad_bf16, void* stream) {
    PIVP_REQUIRE(W && N > 0 && Cx > 0 && Kpad >= Cx && (w_fwd_bf16 || w_dgrad_bf16), "tc_prep_weights: bad argument");
    launch_k(tc_prep_weights_kernel, dim3(148 * 4), dim3(256), 0, (cudaStream_t)stream, W, N, Cx, Kpad, (__nv_bfloat16*)w_fwd_bf16, (__nv_bfloat16*)w_dgrad_bf16);
    return check_launch("tc_prep_weights");
}

int pivp_gather_bf16(const float* src, const int* idx, long n, void* dst_bf16, void* stream) {
    PIVP_REQUIRE(src && idx && dst_bf16 && n > 0, "gather_bf16: bad argument");
    unsigned gb = (unsigned)((n + 255) / 256);
    if (gb > 148 * 8) gb = 148 * 8;
    launch_k(gather_bf16_kernel, dim3(gb), dim3(256), 0, (cudaStream_t)stream, src, idx, n, (__nv_bfloat16*)dst_bf16);
    return check_launch("gather_bf16");
}

}  // extern "C"

struct LnFuse {                 // LayerNorm applied inside the gate epilogue (pivp_tc_conv5x5_ln); all null / zero = not fused
    const float* gamma; const float* beta; float* y; int y_cs, y_co; void* y_bf16; int yb_cs, yb_co; float* stats; unsigned* counter; float eps;
};

static int tc_conv5x5_impl(const void* in_bf16, int in_cs, int B, int H, int W, int Kc,
                    const void* wt_bf16, int N, int BN,
                    int mode, const float* bias,
                    float* out, int out_cs, int out_co,
                    float* gates, const float* c_prev, float* c_out,
                    float* h_out, int h_cs, int h_co, void* h_bf16, int hb_cs, int hb_co,
                    void* h_t, long h_t_ld, int hT_co,
                    int C, float forget_bias, int flags, float* ln_partial, const LnFuse& lf, void* stream) {
    PIVP_REQUIRE(in_cs >= Kc, "tc_conv5x5: row stride smaller than Kc");
    const bool no_gates = (flags >> 2) & 1;       // forward-only: the activated gates are not stored (nothing reads them without a backward pass)
    PIVP_REQUIRE(!no_gates || mode == 1, "tc_conv5x5: flags bit 2 (no gate storage) needs mode 1");
    if (mode == 1) {
        PIVP_REQUIRE(BN == 128 && N == 4 * C && C % 32 == 0 && (gates || no_gates) && c_out && h_out && bias,
                     "tc_conv5x5: gate epilogue needs BN=128, N=4C, bias, and gates unless flags bit 2 is set");
        PIVP_REQUIRE(h_cs % 4 == 0 && h_co % 4 == 0 && (!h_bf16 || (hb_cs % 8 == 0 && hb_co % 8 == 0)), "tc_conv5x5: h views must be 16-byte aligned");
    } else {
        PIVP_REQUIRE(mode == 0 && out && out_cs % 4 == 0 && out_co % 4 == 0, "tc_conv5x5: plain epilogue needs a 16-byte aligned fp32 view");
    }
    int dy[25], dx[25], co[25];
    for (int t = 0; t < 25; ++t) { dy[t] = t / 5 - 2; dx[t] = t % 5 - 2; co[t] = 0; }
    TcEpilogue ep;
    memset(&ep, 0, sizeof(ep));
    ep.mode = mode; ep.bias = bias; ep.out = out; ep.out_cs = out_cs; ep.out_co = out_co; ep.gates = no_gates ? nullptr : gates; ep.c_prev = c_prev;
    ep.c_out = c_out; ep.h_out = h_out; ep.h_cs = h_cs; ep.h_co = h_co; ep.h_bf16 = (__nv_bfloat16*)h_bf16; ep.hb_cs = hb_cs; ep.hb_co = hb_co;
    ep.h_t = (__nv_bfloat16*)h_t; ep.h_t_ld = h_t_ld; ep.hT_co = hT_co;
    ep.C = C; ep.forget_bias = forget_bias; ep.accurate = flags & 1; ep.gates_bf16 = (flags >> 1) & 1;
    if (ln_partial) {
        PIVP_REQUIRE(mode == 1 && tc_halo_supported(B, H, W, Kc, BN) && (H * W) % 128 == 0,
                     "tc_conv5x5: LayerNorm partials are produced by the halo-patch kernel only (H % 16 == 0, W % 8 == 0)");
        ep.ln_partial = reinterpret_cast<float2*>(ln_partial);
        ep.ln_S = (H * W / 128) * (C / 32);
    }
    if (lf.gamma) {
        PIVP_REQUIRE(ln_partial && lf.beta && lf.y && lf.stats && lf.counter, "tc_conv5x5_ln: the fused LayerNorm needs ln_partial, beta, y, stats and counter");
        ep.ln_gamma = lf.gamma; ep.ln_beta = lf.beta; ep.ln_y = lf.y; ep.ln_y_cs = lf.y_cs; ep.ln_y_co = lf.y_co;
        ep.ln_yb = (__nv_bfloat16*)lf.y_bf16; ep.ln_yb_cs = lf.yb_cs; ep.ln_yb_co = lf.yb_co;
        ep.ln_stats = reinterpret_cast<float2*>(lf.stats); ep.ln_counter = lf.counter; ep.ln_eps = lf.eps;
    }
    if (tc_halo_supported(B, H, W, Kc, BN)) return launch_conv5x5_halo(in_bf16, in_cs, B, H, W, Kc, wt_bf16, N, BN, ep, stream, "tc_conv5x5");
    PIVP_REQUIRE(!lf.gamma, "tc_conv5x5_ln: the fused LayerNorm exists in the halo-patch kernel only");
    return launch_conv_taps(in_bf16, in_cs, B, H, W, Kc, 25, dy, dx, co, wt_bf16, N, BN, ep, H, W, 1, 0, 0, stream, "tc_conv5x5");
}

extern "C" {

int pivp_tc_conv5x5(const void* in_bf16, int in_cs, int B, int H, int W, int Kc,
                    const void* wt_bf16, int N, int BN,
                    int mode, const float* bias,
                    float* out, int out_cs, int out_co,
                    float* gates, const float* c_prev, float* c_out,
                    float* h_out, int h_cs, int h_co, void* h_bf16, int hb_cs, int hb_co,
                    void* h_t, long h_t_ld, int hT_co,
                    int C, float forget_bias, int flags, float* ln_partial, void* stream) {
    LnFuse none;
    memset(&none, 0, sizeof(none));
    return tc_conv5x5_impl(in_bf16, in_cs, B, H, W, Kc, wt_bf16, N, BN, mode, bias, out, out_cs, out_co, gates, c_prev, c_out, h_out, h_cs, h_co,
                           h_bf16, hb_cs, hb_co, h_t, h_t_ld, hT_co, C, forget_bias, flags, ln_partial, none, stream);
}

/* ConvLSTM cell (mode 1 of pivp_tc_conv5x5, bf16 gate storage) with the LayerNorm of its output applied in the same kernel:
 * y = LN(h_t) * gamma + beta -> fp32 view (and optional bf16 view); stats[b] = (mean, rstd) for the backward pass.
 * counter: B unsigned ints owned by this layer, zeroed once at allocation (per-sample arrival counters, never reset). */
int pivp_tc_conv5x5_ln(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, const void* wt_bf16, int C, const float* bias,
                       void* gates_bf16, const float* c_prev, float* c_out, float* h_out, int h_cs, int h_co, void* h_bf16, int hb_cs, int hb_co,
                       float forget_bias, int flags, float* ln_partial,
                       const float* gamma, const float* beta, float eps, float* y, int y_cs, int y_co, void* y_bf16, int yb_cs, int yb_co,
                       float* stats, void* counter, void* stream) {
    LnFuse lf{gamma, beta, y, y_cs, y_co, y_bf16, yb_cs, yb_co, stats, (unsigned*)counter, eps};
    PIVP_REQUIRE(gamma, "tc_conv5x5_ln: gamma is null");
    PIVP_REQUIRE(!(flags & 4), "tc_conv5x5_ln: stores the gates always (flags bit 2 is for pivp_tc_conv5x5)");
    return tc_conv5x5_impl(in_bf16, in_cs, B, H, W, Kc, wt_bf16, 4 * C, 128, 1, bias, nullptr, 0, 0, (float*)gates_bf16, c_prev, c_out, h_out, h_cs, h_co,
                           h_bf16, hb_cs, hb_co, nullptr, 0, 0, C, forget_bias, flags | 2, ln_partial, lf, stream);
}

// General tap-list convolution with a plain epilogue:  D[m,n] = sum_t sum_c In[pixel(m)+(dy_t,dx_t), coff_t + c] * Wt[n][t*Kc + c],
// out[row(m)] = relu?(D + bias) written to an fp32 view and/or a bf16 view, row(m) = ((b*OH + i*os + oa)*OW + j*os + ob).
// One call = one output phase of a stride-2 Deconvolution2D (train_model.py:505-507), a 1x1 convolution, ...
int pivp_tc_conv_taps(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, int ntaps, const int* dy, const int* dx, const int* coff,
                      const void* wt_bf16, int N, int BN, const float* bias, int relu, int accumulate,
                      float* out, int out_cs, int out_co, void* out_bf16, int ob_cs, int ob_co,
                      int OH, int OW, int os, int oa, int ob, void* stream) {
    PIVP_REQUIRE(dy && dx && coff, "tc_conv_taps: null tap list (host arrays)");
    PIVP_REQUIRE(out || out_bf16, "tc_conv_taps: no output");
    PIVP_REQUIRE((!out || (out_cs % 4 == 0 && out_co % 4 == 0)) && (!out_bf16 || (ob_cs % 8 == 0 && ob_co % 8 == 0)),
                 "tc_conv_taps: output views must be 16-byte aligned");
    PIVP_REQUIRE(os >= 1 && oa >= 0 && ob >= 0 && OH >= (H - 1) * os + oa + 1 && OW >= (W - 1) * os + ob + 1, "tc_conv_taps: bad output mapping");
    TcEpilogue ep;
    memset(&ep, 0, sizeof(ep));
    ep.mode = 0; ep.bias = bias; ep.relu = relu; ep.accumulate = accumulate; ep.out = out; ep.out_cs = out_cs; ep.out_co = out_co;
    ep.out_bf16 = (__nv_bfloat16*)out_bf16; ep.ob_cs = ob_cs; ep.ob_co = ob_co;
    return launch_conv_taps(in_bf16, in_cs, B, H, W, Kc, ntaps, dy, dx, coff, wt_bf16, N, BN, ep, OH, OW, os, oa, ob, stream, "tc_conv_taps");
}

/* Up to four tap lists in ONE launch (blockIdx.z = phase): the output phases (oa[p], ob[p]) of a stride-2 Deconvolution2D, or of the
 * input gradient of a stride-2 Convolution2D.  ntaps[p] <= 4 taps per phase; dy / dx / coff hold 4 slots per phase; wt[p] = bf16
 * weights [N][ntaps[p] * Kc] of phase p.  Everything else as pivp_tc_conv_taps. */
/* ln_partial != null: also write the (mean, M2) partials of the LayerNorm that follows the deconvolution (norm_enc6, train_model.py:601):
 * per sample (H * W / 128) * nph * (N / 32) pairs of 4096 values each, the layout pivp_layernorm_fwd reads when its relu argument has
 * bit 1 set.  Needs relu = accumulate = 0. */
int pivp_tc_conv_taps_multi_ln(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, int nph, const int* ntaps, const int* dy,
                               const int* dx, const int* coff, const void* const* wt_bf16, int N, int BN, const float* bias, int relu,
                               int accumulate, float* out, int out_cs, int out_co, void* out_bf16, int ob_cs, int ob_co,
                               int OH, int OW, int os, const int* oa, const int* ob, float* ln_partial, void* stream) {
    PIVP_REQUIRE(ntaps && dy && dx && coff && wt_bf16 && oa && ob && nph >= 1 && nph <= TC_MAXPH, "tc_conv_taps_multi: null list or bad phase count");
    PIVP_REQUIRE(out || out_bf16, "tc_conv_taps_multi: no output");
    PIVP_REQUIRE((!out || (out_cs % 4 == 0 && out_co % 4 == 0)) && (!out_bf16 || (ob_cs % 8 == 0 && ob_co % 8 == 0)),
                 "tc_conv_taps_multi: output views must be 16-byte aligned");
    TapPhase ph[TC_MAXPH];
    for (int p = 0; p < nph; ++p) {
        PIVP_REQUIRE(ntaps[p] >= 1 && ntaps[p] <= 4, "tc_conv_taps_multi: 1..4 taps per phase");
        PIVP_REQUIRE(os >= 1 && oa[p] >= 0 && ob[p] >= 0 && OH >= (H - 1) * os + oa[p] + 1 && OW >= (W - 1) * os + ob[p] + 1,
                     "tc_conv_taps_multi: bad output mapping");
        ph[p] = TapPhase{ntaps[p], dy + 4 * p, dx + 4 * p, coff + 4 * p, wt_bf16[p], oa[p], ob[p]};
    }
    TcEpilogue ep;
    memset(&ep, 0, sizeof(ep));
    ep.mode = 0; ep.bias = bias; ep.relu = relu; ep.accumulate = accumulate; ep.out = out; ep.out_cs = out_cs; ep.out_co = out_co;
    ep.out_bf16 = (__nv_bfloat16*)out_bf16; ep.ob_cs = ob_cs; ep.ob_co = ob_co;
    ep.ln_partial = reinterpret_cast<float2*>(ln_partial);
    return launch_conv_taps_multi(in_bf16, in_cs, B, H, W, Kc, nph, ph, N, BN, ep, OH, OW, os, stream, "tc_conv_taps_multi");
}

int pivp_tc_conv_taps_multi(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, int nph, const int* ntaps, const int* dy,
                            const int* dx, const int* coff, const void* const* wt_bf16, int N, int BN, const float* bias, int relu,
                            int accumulate, float* out, int out_cs, int out_co, void* out_bf16, int ob_cs, int ob_co,
                            int OH, int OW, int os, const int* oa, const int* ob, void* stream) {
    return pivp_tc_conv_taps_multi_ln(in_bf16, in_cs, B, H, W, Kc, nph, ntaps, dy, dx, coff, wt_bf16, N, BN, bias, relu, accumulate, out, out_cs,
                                      out_co, out_bf16, ob_cs, ob_co, OH, OW, os, oa, ob, nullptr, stream);
}

}  // extern "C"
