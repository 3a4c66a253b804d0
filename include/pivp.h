/* libpivp.so -- C-ABI of the B200-native video-prediction training path.
 *
 * The reference (kristofbc/physical-interaction-video-prediction) has NO plugin / FFI layer: its hot
 * path is pure-Python Chainer links (src/models/train_model.py).  This header therefore defines the
 * boundary a maintainer would bind with ctypes + CuPy device pointers (INTEGRATION.md shows the stub);
 * every entry point cites the reference lines it replaces.
 *
 * Conventions
 *  - All pointers are CALLER-OWNED DEVICE pointers (cupy `arr.data.ptr`, torch `t.data_ptr()`); the
 *    library never allocates or frees.  Scratch is passed in as `workspace` (+ `*_workspace_bytes`).
 *  - `stream` is a cudaStream_t passed as void*; every launch goes to it, nothing synchronises.
 *  - Return 0 on success, a negative PIVP_E* code otherwise; pivp_last_error() returns a thread-local
 *    message.  Shape / pointer violations are errors, not undefined behaviour.
 *  - Trunk activations are NHWC "views": element (row m = b*H*W + y*W + x, channel c) lives at
 *    p[m*cs + co + c] (cs = row stride in elements, co = channel offset) so that the channel
 *    concatenations of the reference (F.concat, train_model.py:262,565,575) are free.
 *    Image-space tensors (frames, enc7 / mask logits) are NCHW planes exactly like the reference's.
 *  - Convolution weights are stored [N][KH][KW][C] (OHWI); a Chainer Deconvolution2D weight
 *    (in,out,kh,kw) is stored [in][KH][KW][out].  ConvLSTM gate rows are ordered
 *    [32-channel block][gate j,i,f,o][channel] (private layout; see layout.py for the bijection).
 *  - fp32 everywhere in this header; `*_bf16` pointers are optional bf16 shadows (may be NULL).
 */
#ifndef PIVP_H_
#define PIVP_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIVP_OK 0
#define PIVP_EINVAL (-1)
#define PIVP_ECUDA (-2)
#define PIVP_EUNSUPPORTED (-3)

const char* pivp_last_error(void);
int pivp_abi_version(void);
int pivp_device_sync_check(void);
/* number of CUDA kernels this library has launched in this process (every successful launch is counted once) */
long pivp_launch_count(void);
/* programmatic dependent launch (kernel N+1's CTAs become resident and run their prologue while kernel N drains; every kernel waits
 * for its predecessor before its first global access) on / off for subsequent launches; default on, PIVP_PDL=0 in the environment = off */
int pivp_set_pdl(int on);

/* ---- Convolution2D / Deconvolution2D (train_model.py:224,500-507,527; Chainer A.2/A.3) --------------- */
/* y = conv(x, w) + bias [, relu]  -- L.Convolution2D forward; Deconvolution2D input-gradient */
int pivp_conv2d_fwd(const float* x, int x_cs, int x_co, int B, int H, int W, int C,
                    const float* w, const float* bias, int N, int KH, int KW, int stride, int pad,
                    float* y, int y_cs, int y_co, int Ho, int Wo, int relu, int accumulate, void* stream);
/* dx = conv^T(dy, w) [+ bias, relu]  -- Convolution2D input-gradient; L.Deconvolution2D forward (outsize = H,W) */
int pivp_conv2d_dgrad(const float* dy, int dy_cs, int dy_co, int B, int Ho, int Wo, int N,
                      const float* w, const float* bias, int KH, int KW, int stride, int pad,
                      float* dx, int dx_cs, int dx_co, int H, int W, int C, int relu, int accumulate, void* stream);
/* dw += x (*) dy ; dbias += sum dy   (dbias may be NULL) */
int pivp_conv2d_wgrad(const float* x, int x_cs, int x_co, int B, int H, int W, int C,
                      const float* dy, int dy_cs, int dy_co, int Ho, int Wo, int N,
                      int KH, int KW, int stride, int pad, float* dw, float* dbias, void* stream);
int pivp_colsum(const float* v, int v_cs, int v_co, int P, int N, float* out, void* stream);

/* ---- BasicConvLSTMCell gate math (train_model.py:269-272; D.5) ---------------------------------------- */
/* gates: (M, 4C) pre-activations in, activated gates out (saved for backward). c_prev may be NULL (zeros).
 * c_prev == c_out is allowed (the cell state updated in place): every element of c_prev is read once, by the thread that then writes
 * the same element of c_out, before it writes it. */
int pivp_lstm_gates_fwd(float* gates, const float* c_prev, float* c_out, float* h_out, int h_cs, int h_co,
                        void* h_bf16, int hb_cs, int hb_co, long M, int C, float forget_bias, void* stream);
/* dh = dh_a (dense, may be NULL) + dh_b (view, may be NULL); dc in/out (dc_valid=0: treat incoming dc as 0);
 * gates: activated gates in, d(pre-activation) out. */
int pivp_lstm_gates_bwd(float* gates, const float* c_prev, const float* c_cur, const float* dh_a,
                        const float* dh_b, int dhb_cs, int dhb_co, float* dc, int dc_valid, void* dg_bf16,
                        long M, int C, void* stream);
/* bf16 gate storage (tensor-core mode; pivp_tc_conv5x5 flags bit 1): same math, gates read and d(pre-activations) written as bf16 */
int pivp_lstm_gates_bwd_bf16(const void* gates_bf16, const float* c_prev, const float* c_cur, const float* dh_a,
                             const float* dh_b, int dhb_cs, int dhb_co, float* dc, int dc_valid, void* dg_bf16,
                             long M, int C, void* stream);

/* ---- LayerNormalizationConv2D (train_model.py:186-208; A.4, D.4) -------------------------------------- */
size_t pivp_layernorm_workspace_bytes(int B, int n);
/* per-sample LN over HW*C with per-element gamma/beta (HWC order); stats (B,2) = mean, rstd saved for bwd.
 * relu: bit 0 = ReLU after the affine; bit 1 = the (mean, M2) chunk partials are already in `workspace` (written by the epilogue of
 * pivp_tc_conv5x5 ..., ln_partial) -- the statistics pass is skipped. */
int pivp_layernorm_fwd(const float* x, int x_cs, int x_co, const float* gamma, const float* beta, int B, int HW, int C, float eps,
                       float* y, int y_cs, int y_co, float* y2, int y2_cs, int y2_co, void* y_bf16, int yb_cs, int yb_co,
                       int relu, float* stats, void* workspace, size_t ws_bytes, void* stream);
/* The same, with the bf16 copy written in the space-to-depth layout the stride-2 convolution behind this LayerNorm contracts over
 * (hidden2 -> enc1, hidden4 -> enc2, train_model.py:597-599): s2d_w = width W of the normalised map (0 = plain rows, identical to
 * pivp_layernorm_fwd); pixel (y, x) of sample b goes to row (b, y/2, x/2) of a [B*H/2*W/2][yb_cs] matrix, columns
 * yb_co + ((y&1)*2 + (x&1)) * s2d_cblk + c.  Replaces a separate pivp_cast_bf16 launch. */
int pivp_layernorm_fwd_s2d(const float* x, int x_cs, int x_co, const float* gamma, const float* beta, int B, int HW, int C, float eps,
                           float* y, int y_cs, int y_co, float* y2, int y2_cs, int y2_co, void* y_bf16, int yb_cs, int yb_co,
                           int relu, float* stats, void* workspace, size_t ws_bytes, int s2d_w, int s2d_cblk, void* stream);
/* g = g1 + g2 (g2 may be NULL), masked by [y>0] when relu; dgamma/dbeta are accumulated into */
int pivp_layernorm_bwd(const float* x, int x_cs, int x_co, const float* g1, int g1_cs, int g1_co, const float* g2, int g2_cs, int g2_co,
                       const float* gamma, const float* beta, const float* stats, int B, int HW, int C, int relu,
                       float* dx, int dx_cs, int dx_co, float* dgamma, float* dbeta, void* workspace, size_t ws_bytes, void* stream);
/* The same, with dx delivered as the bf16 space-to-depth GEMM operand of the transposed convolution BELOW this LayerNorm and that convolution's
 * bias gradient accumulated (norm_enc6 -> enc6, train_model.py:507, 601 backward): ho_bf16 rows (b, y/2, x/2) of [B*H/2*W/2][ho_cs], column
 * ho_co + ((y&1)*2 + (x&1)) * ho_cblk + c; ho_w = width of the normalised map; ho_db [C] += sum of dx over samples and pixels.  Replaces
 * pivp_layernorm_bwd + pivp_grad_handover; dx may be NULL (the fp32 gradient is then never written).  ho_bf16 = NULL: pivp_layernorm_bwd. */
int pivp_layernorm_bwd_handover(const float* x, int x_cs, int x_co, const float* g1, int g1_cs, int g1_co, const float* g2, int g2_cs, int g2_co,
                                const float* gamma, const float* beta, const float* stats, int B, int HW, int C, int relu,
                                float* dx, int dx_cs, int dx_co, float* dgamma, float* dbeta, void* workspace, size_t ws_bytes,
                                void* ho_bf16, int ho_cs, int ho_co, int ho_w, int ho_cblk, float* ho_db, void* stream);
/* LayerNorm backward of a ConvLSTM output h_t fused with that layer's gate backward (tensor-core mode, bf16 gate storage): instead of
 * writing d h_t, each thread adds the recurrent d h_t (dh_b view, may be NULL) and produces the gate pre-activation gradients, written
 * bf16 over gates_bf16 (pivp_tc_conv5x5 flags bit 1); dc updated in place.  Replaces pivp_layernorm_bwd + pivp_lstm_gates_bwd_bf16. */
int pivp_layernorm_bwd_lstm(const float* x, int x_cs, int x_co, const float* g1, int g1_cs, int g1_co, const float* g2, int g2_cs, int g2_co,
                            const float* gamma, const float* beta, const float* stats, int B, int HW, int C,
                            float* dgamma, float* dbeta, void* gates_bf16, const float* c_prev, const float* c_cur,
                            const float* dh_b, int dhb_cs, int dhb_co, float* dc, int dc_valid, void* workspace, size_t ws_bytes, void* stream);

/* ---- small view ops (F.relu backward :698, F.concat copies, layout packing) --------------------------- */
int pivp_relu_bwd(const float* out, int o_cs, int o_co, const float* ga, int ga_cs, int ga_co, const float* gb, int gb_cs, int gb_co,
                  float* dst, int d_cs, int d_co, long M, int C, void* stream);
/* Fused gradient hand-over: g = ga (+ gb) [* (out > 0)] -> optional fp32 view, optional bf16 view (plain or space-to-depth with channel
 * block cblk on the H x W grid, as pivp_cast_bf16), optional bias gradient db[C] += column sums of g.  One launch instead of
 * relu_bwd + colsum + cast_bf16 between the ReLU / LayerNorm backward and the tensor-core transposed-convolution backward. */
int pivp_grad_handover(const float* out, int o_cs, int o_co, const float* ga, int ga_cs, int ga_co, const float* gb, int gb_cs, int gb_co,
                       float* dst, int d_cs, int d_co, void* dst_bf16, int b_cs, int b_co, int H, int W, int s2d, int cblk,
                       float* db, long M, int C, void* stream);
int pivp_copy_view(const float* src, int s_cs, int s_co, float* dst, int d_cs, int d_co, void* dst_bf16, int db_cs, int db_co,
                   long M, int C, void* stream);
int pivp_nchw_to_nhwc(const float* src, float* dst, int d_cs, int d_co, int B, int C, int HW, void* stream);
int pivp_nhwc_to_nchw(const float* src, int s_cs, int s_co, float* dst, int B, int C, int HW, int accumulate, void* stream);
int pivp_axpy(const float* x, float* y, long n, void* stream);
int pivp_relu_mask(const float* y, float* g, long n, void* stream);
int pivp_fill(float* p, float value, long n, void* stream);

/* ---- state predictor + smear (train_model.py:563-565,676,730-731) ------------------------------------- */
int pivp_state_fwd(const float* action, const float* cur, const float* Wc, const float* bc, float* sa, float* next,
                   float* smear, int sm_cs, int sm_co, int npix, int B, void* stream);
int pivp_state_bwd(const float* dn_a, const float* dn_b, const float* sa, const float* Wc, const float* dsmear, int ds_cs, int ds_co,
                   int npix, int B, float* d_cur_prev, float* dWc, float* dbc, void* stream);

/* ---- L.Linear (train_model.py:289,321-322,430-431,457-466) -------------------------------------------- */
int pivp_linear_fwd(const float* x, int xs, const float* W, const float* bias, float* y, int B, int K, int N, int relu, void* stream);
/* split-K variant for wide inputs (the 8192 -> 250 kernel Linear, train_model.py:321-322): same result, caller-provided scratch */
size_t pivp_linear_fwd_workspace_bytes(int B, int K, int N);
int pivp_linear_fwd_splitk(const float* x, int xs, const float* W, const float* bias, float* y, int B, int K, int N, int relu,
                           void* workspace, size_t ws_bytes, void* stream);
int pivp_linear_bwd(const float* dy, const float* x, int xs, const float* W, float* dx, int dxs, int accumulate_dx,
                    float* dW, float* db, int B, int K, int N, void* stream);
/* The weight / bias gradient of pivp_linear_bwd over S stacked time steps in one pass (dy [S][B][N] with step stride dy_step elements,
 * x [S][B rows of stride xs] with step stride x_step): dW [N][K] and db [N] are accumulated into.  pivp_linear_bwd with dW = NULL
 * computes dx only, so a caller can defer the weight gradient of a time loop to one launch (train_model.py:321-322 backward). */
int pivp_linear_wgrad_steps(const float* dy, long dy_step, const float* x, long x_step, int xs, float* dW, float* db, int S, int B, int K, int N,
                            void* stream);

/* ---- loss, scheduled sampling, optimizer --------------------------------------------------------------- */
/* F.mean_squared_error pieces (train_model.py:741,751): *loss_slot += sum (gen-target)^2 ; dgen = gscale*(gen-target) */
int pivp_mse(const float* gen, const float* target, long n, float gscale, float* dgen, float* loss_slot, void* stream);
/* scheduled_sample (train_model.py:73-122) as the per-sample select it reduces to */
int pivp_sched_select(const float* gt, const float* gen, const int* take, float* out, int B, int per_sample, void* stream);
/* the same select of (B, C, H*W) planes, also written as NHWC rows out_nhwc[(b*HW + p)*C + c] -- the layout enc0 (train_model.py:500) reads,
 * so the layout change costs no launch of its own */
int pivp_sched_select_nhwc(const float* gt, const float* gen, const int* take, float* out, float* out_nhwc, int B, int C, int HW, void* stream);
/* Chainer 2.0.1 AdamRule (train_model.py:860-861; A.8). step[0] = number of updates done so far (device int, incremented). */
int pivp_adam_step(float* p, const float* g, float* m, float* v, long n, int* step, float alpha, float beta1, float beta2, float eps,
                   float gscale, void* stream);

/* ---- the two 1x1 "head" deconvolutions on enc6 (train_model.py:288/364/429 + 527, applied at :315/:388/:454 and :719) fused:
 * x = NHWC rows of 64 channels, W = [NH][64] (enc7 rows, then mask rows), outputs / output gradients as NCHW planes
 * out_a (B,Na,H,W) | out_b (B,NH-Na,H,W).  NH in {14, 27}; anything else returns PIVP_EUNSUPPORTED (use pivp_conv2d_*).
 * backward: dx overwritten, dW [NH][64] and db [NH] accumulated into. */
int pivp_heads_fwd(const float* x, int x_cs, int x_co, const float* W, const float* bias, float* out_a, int Na, float* out_b, int NH,
                   int B, int HW, void* stream);
/* forward on relu(LayerNorm(x)) in one launch (norm_enc6 + ReLU `:601, 698` then the heads): x = the LayerNorm input, partial = the
 * [B][HW*64/4096] (mean, M2) pairs written by pivp_tc_conv_taps_multi_ln, y = normalised rows kept for the backward, stats [B][2] =
 * (mean, rstd) for pivp_layernorm_bwd.  HW must be a multiple of 128.
 * y == NULL: the normalised rows are not written (forward-only prediction; a kernel instantiation without that store).  stats stays
 * required. */
int pivp_heads_fwd_ln(const float* x, int x_cs, int x_co, const float* gamma, const float* beta, const float* partial, float eps, float* stats,
                      float* y, int y_cs, int y_co, const float* W, const float* bias, float* out_a, int Na, float* out_b, int NH,
                      int B, int HW, void* stream);
int pivp_heads_bwd(const float* x, int x_cs, int x_co, const float* W, const float* dy_a, int Na, const float* dy_b, int NH,
                   float* dx, int dx_cs, int dx_co, float* dW, float* db, int B, int HW, void* stream);

/* ---- fused transform + mask softmax + composite (train_model.py:315-349 / 388-415 / 454-471 + 719-728) - */
int pivp_cdna_fused_fwd(const float* prev, const float* enc7_pre, const float* mask_pre, const float* kern_raw, float* out,
                        int B, int H, int W, int num_masks, void* stream);
size_t pivp_cdna_fused_bwd_workspace_bytes(int B, int H, int W, int num_masks);
int pivp_cdna_fused_bwd(const float* g_out, const float* prev, const float* enc7_pre, const float* mask_pre, const float* kern_raw,
                        float* d_enc7_pre, float* d_mask_pre, float* d_kern_raw, float* d_prev, int accumulate_dprev,
                        int B, int H, int W, int num_masks, void* workspace, size_t ws_bytes, void* stream);
int pivp_dna_fused_fwd(const float* prev, const float* enc7_pre, const float* mask_pre, float* out, int B, int H, int W, void* stream);
size_t pivp_dna_fused_bwd_workspace_bytes(int B, int H, int W);
int pivp_dna_fused_bwd(const float* g_out, const float* prev, const float* enc7_pre, const float* mask_pre,
                       float* d_enc7_pre, float* d_mask_pre, float* d_prev, int accumulate_dprev,
                       int B, int H, int W, void* workspace, size_t ws_bytes, void* stream);
int pivp_stp_fused_fwd(const float* prev, const float* enc7_pre, const float* mask_pre, const float* theta_raw, float* out,
                       int B, int H, int W, int num_masks, int oob_border, void* stream);
size_t pivp_stp_fused_bwd_workspace_bytes(int B, int H, int W, int num_masks);
int pivp_stp_fused_bwd(const float* g_out, const float* prev, const float* enc7_pre, const float* mask_pre, const float* theta_raw,
                       float* d_enc7_pre, float* d_mask_pre, float* d_theta, float* d_prev,
                       int B, int H, int W, int num_masks, int oob_border, void* workspace, size_t ws_bytes, void* stream);

/* ---- un-fused transformation lists: the reference call surface of the Stateless* links returns (transformed_list, enc7)
 *      (train_model.py:293-351, 368-417, 434-475).  out = [L][B][3][H][W]:
 *      CDNA  L = num_masks + 1: sigmoid(relu(enc7_pre)) (:315-317), then the num_masks per-sample cross-correlations (:326-347)
 *      DNA   L = 1: the 25-tap per-pixel transform with the truncated windows of :395-405
 *      STP   L = num_masks: sigmoid(enc7_pre) (:454-455), then num_masks - 1 samplings with the one shared theta (:465-470)
 *      Model itself trains through the fused entry points above; the backward below serves a link called in its reference form. */
int pivp_cdna_transform(const float* prev, const float* enc7_pre, const float* kern_raw, float* out, int B, int H, int W, int num_masks,
                        void* stream);
int pivp_dna_transform(const float* prev, const float* enc7_pre, float* out, int B, int H, int W, void* stream);
int pivp_stp_transform(const float* prev, const float* enc7_pre, const float* theta_raw, float* out, int B, int H, int W, int num_masks,
                       int oob_border, void* stream);
/* Backward of the three lists.  g_list = HOST array of L device pointers (L as above), entry i = the gradient of list entry i,
 * (B,3,H,W) contiguous, or NULL when that entry has no gradient (it is not read; e.g. the last CDNA entry, which the reference
 * composite's zip(transformed, mask_list[1:]) never uses).  g_list itself must not be NULL.  g_enc7 = gradient of the returned enc7
 * (relu(enc7_pre) for CDNA / DNA, enc7_pre for STP), may be NULL.
 *  - d_enc7_pre, d_kern_raw (B,25*num_masks), d_theta_raw (B,6) are OVERWRITTEN.
 *  - d_prev (optional, NULL = not computed) is overwritten, or added to when accumulate_dprev != 0.  DNA has none: its taps are
 *    detached (:404).  STP with no live sampled entry (L = 1, or all of entries 1 .. L-1 NULL) only zeroes d_prev (if not accumulating).
 *  - 1 <= num_masks <= 64.  d_kern_raw, d_theta_raw and the CDNA d_prev are deterministic (per-band partials in `workspace`, no float
 *    atomics); the STP d_prev is a scatter-add.  CDNA / DNA stage bands of the image in 48 KB of shared memory: wider images than that
 *    allows (CDNA W > 345 at num_masks = 64, DNA W > 815) are PIVP_EINVAL. */
size_t pivp_cdna_transform_bwd_workspace_bytes(int B, int H, int W, int num_masks);
int pivp_cdna_transform_bwd(const float* const* g_list, const float* g_enc7, const float* prev, const float* enc7_pre, const float* kern_raw,
                            float* d_enc7_pre, float* d_kern_raw, float* d_prev, int accumulate_dprev,
                            int B, int H, int W, int num_masks, void* workspace, size_t ws_bytes, void* stream);
int pivp_dna_transform_bwd(const float* const* g_list, const float* g_enc7, const float* prev, const float* enc7_pre, float* d_enc7_pre,
                           int B, int H, int W, void* stream);
size_t pivp_stp_transform_bwd_workspace_bytes(int B, int H, int W, int num_masks);
int pivp_stp_transform_bwd(const float* const* g_list, const float* g_enc7, const float* prev, const float* enc7_pre, const float* theta_raw,
                           float* d_enc7_pre, float* d_theta_raw, float* d_prev, int accumulate_dprev,
                           int B, int H, int W, int num_masks, int oob_border, void* workspace, size_t ws_bytes, void* stream);

/* ---- inference preprocessing (predict_model.py:118-123): F.resize_images (bilinear, positions linspace(0, W-1, OW) in float64, corner
 *      indices clipped to [0, W-2]) fused with the cast and the division: y = resize(x) / scale (divide != 0) or * scale.
 *      x: (BC, H, W) float32 or uint8 planes (x_is_u8), y: (BC, OH, OW) float32. */
int pivp_resize_images(const void* x, int x_is_u8, float* y, int BC, int H, int W, int OH, int OW, float scale, int divide, void* stream);

/* ---- tcgen05 / TMEM / TMA path for the seven ConvLSTM 5x5 convolutions (bf16 operands, fp32 accumulate) ---------- */
/* fp32 master W[n][tap][c] -> bf16 forward operand Wf[n][tap][Kpad] and tap-flipped dgrad operand Wd[c][tap'][n] */
int pivp_tc_prep_weights(const float* W, int N, int Cx, int Kpad, void* w_fwd_bf16, void* w_dgrad_bf16, void* stream);
/* Debugging aid (scripts/halo_timeline_all.py): device buffer of [512 launches][256 CTAs][8] 64-bit slots; launch k after the call fills
 * rows [256 k, 256 k + CTAs) with clock64() stamps (0 launch, 1 set-up done, 2 first operands landed, 3 last MMA issued, 4 accumulator
 * ready, 5 epilogue done) and %globaltimer at CTA start / end (6, 7);
 * null switches it off.  Process-wide, not thread-safe. */
int pivp_tc_set_debug_buffer(void* device_buffer);
/* D[m,n] = sum_{tap,c} In[pixel(m)+tap-2, c] * Wt[n][tap][c]  (In bf16 NHWC with row stride in_cs; Wt bf16 [N][25][Kc]).
 * mode 0: out[m*out_cs+out_co+n] = D (+bias)                      -- Convolution2D input-gradient (D.5) with Wd
 * mode 1: bias + gates + cell + h fused (train_model.py:262-272)  -- BN must be 128, N = 4C in the gate-interleaved order;
 *         writes activated gates (M,4C), c_out, h (fp32 view + optional bf16 view + optional channel-major bf16 copy).
 *         ln_partial (optional, mode 1 on maps with H % 16 == 0, W % 8 == 0): the epilogue also writes the LayerNorm statistics of h as
 *         per-tile (mean, M2) pairs in the workspace layout of pivp_layernorm_fwd, which can then be called with relu | 2 (skip its
 *         own statistics pass).
 *         flags: bit 0 = accurate tanhf/expf instead of tanh.approx; bit 1 = `gates` points to bf16 storage (M,4C) (pivp_lstm_gates_bwd_bf16);
 *         bit 2 = no gate storage: the activated gates are not written (forward-only prediction: only the backward pass reads them) and
 *         `gates` may be NULL.  Chosen at compile time (a kernel instantiation without the gate store).  Bit 2 without mode 1, or a NULL
 *         `gates` without bit 2, returns PIVP_EINVAL before any CUDA call.
 *         c_prev == c_out is allowed in every epilogue variant (cell state updated in place): each c_prev element is read by the thread that
 *         computes c_t for the same pixel and channel, before the accumulator wait (halo kernel) or before its own store (per-tap kernel),
 *         and written only after that read.
 * Returns PIVP_EUNSUPPORTED when B*H*W cannot be cut into 128-pixel TMA boxes. */
int pivp_tc_conv5x5(const void* in_bf16, int in_cs, int B, int H, int W, int Kc,
                    const void* wt_bf16, int N, int BN,
                    int mode, const float* bias,
                    float* out, int out_cs, int out_co,
                    float* gates, const float* c_prev, float* c_out,
                    float* h_out, int h_cs, int h_co, void* h_bf16, int hb_cs, int hb_co,
                    void* h_t, long h_t_ld, int hT_co,
                    int C, float forget_bias, int flags, float* ln_partial, void* stream);

/* The ConvLSTM cell of pivp_tc_conv5x5 (mode 1, bf16 gate storage) with the LayerNormalizationConv2D that follows it (train_model.py:203-208,
 * 596-601) applied in the SAME kernel: the CTAs of a sample meet at a per-sample arrival counter once their statistics partials are
 * written, then every thread normalises the h values it still holds in registers: y = (h - mean) * rstd * gamma + beta -> fp32 view `y`
 * (+ optional bf16 view), stats[b] = (mean, rstd) for the LayerNorm backward.  gamma / beta in the sample's H*W*C order.
 * counter: B unsigned ints owned by this layer, zeroed once (never reset: every launch adds the same number of arrivals per sample).
 * Needs the halo-patch geometry (H % 16 == 0, W % 8 == 0), H*W*C % 4096 == 0 and at most 148 CTAs (all resident at once).
 * Always stores the gates: flags bit 2 is PIVP_EINVAL here. */
int pivp_tc_conv5x5_ln(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, const void* wt_bf16, int C, const float* bias,
                       void* gates_bf16, const float* c_prev, float* c_out, float* h_out, int h_cs, int h_co, void* h_bf16, int hb_cs, int hb_co,
                       float forget_bias, int flags, float* ln_partial,
                       const float* gamma, const float* beta, float eps, float* y, int y_cs, int y_co, void* y_bf16, int yb_cs, int yb_co,
                       float* stats, void* counter, void* stream);

/* dst[i] = bf16(src[idx[i]]) (idx < 0 -> 0): builds permuted / zero-padded bf16 weight operands from the fp32 master parameters */
int pivp_gather_bf16(const float* src, const int* idx, long n, void* dst_bf16, void* stream);
/* General tap-list implicit GEMM on tcgen05: D[m,n] = sum_t sum_c In[pixel(m)+(dy_t,dx_t), coff_t+c] * Wt[n][t*Kc+c];
 * out[row(m)] = relu?(D + bias) to an fp32 view and/or a bf16 view, row(m) = ((b*OH + i*os + oa)*OW + j*os + ob).
 * One call = one output phase of a stride-2 Deconvolution2D (train_model.py:505-507), a 1x1 convolution, ...
 * dy/dx/coff are HOST int arrays of length ntaps (<= 25). */
int pivp_tc_conv_taps(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, int ntaps, const int* dy, const int* dx, const int* coff,
                      const void* wt_bf16, int N, int BN, const float* bias, int relu, int accumulate,
                      float* out, int out_cs, int out_co, void* out_bf16, int ob_cs, int ob_co,
                      int OH, int OW, int os, int oa, int ob, void* stream);
/* Up to four tap lists in ONE launch (grid z = phase): the four output phases (oa[p], ob[p]) of a stride-2 Deconvolution2D
 * (train_model.py:505-507) or of the input gradient of a stride-2 Convolution2D.  ntaps[p] <= 4; dy / dx / coff hold 4 slots per phase;
 * wt_bf16[p] = bf16 weights [N][ntaps[p]*Kc] of phase p (host array of device pointers). */
int pivp_tc_conv_taps_multi(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, int nph, const int* ntaps, const int* dy,
                            const int* dx, const int* coff, const void* const* wt_bf16, int N, int BN, const float* bias, int relu,
                            int accumulate, float* out, int out_cs, int out_co, void* out_bf16, int ob_cs, int ob_co,
                            int OH, int OW, int os, const int* oa, const int* ob, void* stream);
/* Same launch, and the epilogue also delivers the statistics of the LayerNorm that follows the deconvolution (norm_enc6 behind enc6,
 * train_model.py:507, 601): ln_partial[b][(H*W/128) * nph * (N/32)] (mean, M2) pairs of 4096 outputs each -- exactly the workspace
 * pivp_layernorm_fwd reads when bit 1 of its relu argument is set (no separate statistics launch).  Needs relu = accumulate = 0,
 * N and BN multiples of 32, H*W a multiple of 128.  ln_partial = null: identical to pivp_tc_conv_taps_multi. */
int pivp_tc_conv_taps_multi_ln(const void* in_bf16, int in_cs, int B, int H, int W, int Kc, int nph, const int* ntaps, const int* dy,
                               const int* dx, const int* coff, const void* const* wt_bf16, int N, int BN, const float* bias, int relu,
                               int accumulate, float* out, int out_cs, int out_co, void* out_bf16, int ob_cs, int ob_co,
                               int OH, int OW, int os, const int* oa, const int* ob, float* ln_partial, void* stream);
/* fp32 NHWC view -> bf16 copy; s2d=1 writes the space-to-depth layout the stride-2 layers contract over
 * (row = (b, y/2, x/2), channel = d_co + ((y&1)*2 + (x&1))*cblk + ch) */
int pivp_cast_bf16(const float* src, int s_cs, int s_co, void* dst_bf16, int d_cs, int d_co, long M, int C, int H, int W, int s2d, int cblk,
                   void* stream);
size_t pivp_tc_wgrad_taps_workspace_bytes(int SB, int H, int W, int Cx, int N4, int ntaps);
/* general weight-gradient GEMM: dW[n][t][c] += sum_p A[p][n] * X[p + (dy_t,dx_t)][coff_t + c]  (n < N4, t < ntaps, c < Cx).
 * dW and workspace must be 16-byte aligned (PIVP_EINVAL otherwise). */
int pivp_tc_wgrad_taps(const void* a_bf16, int a_cs, const void* x_bf16, int x_cs, int SB, int H, int W, int Cx, int N4, int ntaps,
                       const int* dy, const int* dx, const int* coff, float* dW, void* workspace, size_t ws_bytes, void* stream);
/* out[c] += sum_p src[p][c] over a bf16 (P, ld) matrix -- the ConvLSTM bias gradient from the stacked dG of all time steps.
 * C and ld multiples of 8, rows 16-byte aligned (128-bit loads); C <= 256 or a multiple of 256 (one launch per 256-channel slab). */
int pivp_tc_colsum_bf16(const void* src_bf16, int ld, long P, int C, float* out, void* stream);
size_t pivp_tc_wgrad_workspace_bytes(int SB, int H, int W, int Cx, int N4);
/* dW[n][tap][c] += sum over all SB images (time steps x batch) and pixels p of dG[p][n] * XH[p + tap - 2][c]   (D.5).
 * dg: (SB*H*W, N4) bf16; xh: NHWC bf16 with row stride xh_cs >= ceil(Cx/64)*64 (pad channels are ignored). Both operands are
 * read MN-major by tcgen05.mma straight from these NHWC tensors.  dW and workspace must be 16-byte aligned (PIVP_EINVAL otherwise). */
int pivp_tc_wgrad5x5(const void* dg_bf16, const void* xh_bf16, int xh_cs, int SB, int H, int W, int Cx, int N4, float* dW,
                     void* workspace, size_t ws_bytes, void* stream);

/* ---- cross-entropy-method planning over the forward-only predictor (planner.py) -------------------------------------------------
 * One iteration = sample -> predictor forward -> goal cost -> refit, all stream-ordered (graph-capturable), no host synchronisation.
 * Shapes: actions (T-1, Bp, 5) with row stride Bp (the predictor's action buffer; step t of candidate n at (t*Bp + n)*5); the S = T - ctx
 * sampled steps are t = ctx-1 .. T-2 (step s of the distribution is action step ctx-1+s); mean / std (S, 5); predicted frames
 * gen (T-1, Bp, 3, H, W).  Bad arguments return PIVP_EINVAL before any CUDA call. */
/* largest N pivp_cem_refit ranks (its bitonic sort keeps the N keys in shared memory) */
int pivp_cem_max_samples(void);
/* a[t, n, d] = clip(mean[s, d] + std[s, d] * eps, low[d], high[d]) for t = ctx-1+s, every one of the Bp rows n (padding rows included);
 * rows t < ctx-1 are not written.  eps ~ N(0, 1): one Box-Muller pair from the Philox4x32-10 block of curand keyed by *seed (a device
 * int64, read at run time: a new seed needs no new capture) at counter (e = (n*S + s)*5 + d, iteration), so a value depends on neither
 * the launch geometry nor Bp.  std == 0 gives exactly clip(mean).  low / high: HOST arrays of 5 floats (read at the call, so baked into
 * a captured graph), either may be NULL (no bound on that side); low[d] > high[d] or a NaN bound is PIVP_EINVAL. */
int pivp_cem_sample(float* actions, int T, int Bp, int ctx, const float* mean, const float* std_, const float* low, const float* high,
                    const long* seed, int iteration, void* stream);
/* cost[n] = sum_t w[t] * mean_{c,y,x} (gen[t, n, c, y, x] - goal[t or 0, c, y, x])^2 for n < N (cost[n >= N] untouched).
 * goal: one image (goal_per_step = 0) or T-1 images.  weights: device (T-1,); a step with w[t] == 0 is not read.  One CTA per row with a
 * fixed reduction tree: the order depends only on (H, W, T), so the same frames give a bit-identical cost at any N and Bp.
 * gen and goal must be 16-byte aligned (float4 loads) and 3*H*W a multiple of 4 (PIVP_EINVAL otherwise). */
int pivp_goal_cost(const float* gen, int T, int Bp, int N, int H, int W, const float* goal, int goal_per_step, const float* weights,
                   float* cost, void* stream);
/* One CTA.  Ranks cost[0 .. N) by the 64-bit key (order-preserving float bits, index): ties go to the lower index, NaN after +inf.  The K
 * lowest are the elites; per (s, d) their mean and population standard deviation (ddof 0, two passes, fixed order) give
 *   mean <- alpha * mean + (1 - alpha) * elite_mean,  std <- max(alpha * std + (1 - alpha) * elite_std, min_std).
 * Best-so-far record: when the lowest cost is strictly below *best_cost, *best_cost takes it and best_actions (T-1, 5) the candidate's
 * whole action row (context steps included).  history[2*iteration .. +1] = (lowest cost, mean elite cost).
 * Needs 1 <= K <= N <= min(Bp, pivp_cem_max_samples()), 0 <= alpha < 1, min_std >= 0, ctx >= 1, T - ctx >= 1. */
int pivp_cem_refit(const float* cost, const float* actions, int T, int Bp, int ctx, int N, int K, float alpha, float min_std,
                   float* mean, float* std_, float* best_cost, float* best_actions, float* history, int iteration, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PIVP_H_ */
