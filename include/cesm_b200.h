/*
 * cesm_b200.h -- C ABI of libcesm_b200.so, the B200 (sm_100a) kernel library behind the
 * cesm_emulator_b200 PyTorch modules.
 *
 * The reference (kallenordling/cesm_emulator) has no FFI of its own: its hot path is the PyTorch
 * nn.Module tree in video_net.py / model.py, which lowers to aten/cuDNN/cuBLAS calls.  Each entry
 * point below replaces one of those lowered call groups and cites the reference lines it stands in
 * for.  Conventions shared by every function:
 *
 *   - plain C types only: raw DEVICE pointers, sizes, and an opaque `stream` (a cudaStream_t);
 *   - activations are fp16, channels-last: [N, H, W, C] with N = batch*frames (NDHWC flattened);
 *   - parameters / parameter gradients / statistics are fp32;
 *   - the library owns no tensor memory: callers (PyTorch's caching allocator) own every buffer;
 *   - no implicit synchronisation, nothing on the default stream, CUDA-graph capturable;
 *   - return 0 on success, a negative cesm_status otherwise; cesm_last_error() gives the
 *     thread-local message.  There is no CPU fallback: without a CUDA device every compute call
 *     fails with CESM_ERR_CUDA.
 */
#ifndef CESM_B200_H
#define CESM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum cesm_status {
    CESM_OK = 0,
    CESM_ERR_INVALID = -1, /* bad argument (shape not supported, misaligned pointer, ...) */
    CESM_ERR_CUDA = -2,    /* a CUDA runtime / driver call failed */
    CESM_ERR_INTERNAL = -3
} cesm_status;

/* Thread-local description of the last failing call on this thread ("" if none). */
const char* cesm_last_error(void);
/* Library version string, e.g. "cesm_b200 0.1 sm_100a". */
const char* cesm_version(void);
/* Number of CUDA kernels this library has launched in this process so far (all threads). */
long long cesm_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Dense contractions on tcgen05 tensor cores (TMA-fed, TMEM accumulators).
 * ---------------------------------------------------------------------------------------------- */

#define CESM_MAX_TAPS 16

/*
 * Implicit GEMM over pixels:
 *     out[n, oh, ow, co] = sum_t sum_ci  A[n, oh*stride + tap_dh[t], ow*stride + tap_dw[t], ci]
 *                                        * wt[co, t, ci]          (+ bias[co]) (+ residual[...])
 * A is the channel concatenation of a0 (c0 channels) and a1 (c1 channels, may be NULL/0); reads
 * outside the image are zero (conv padding).  The output pixel (n, oh, ow) is written to row
 * ((n*out_h + oh*o_sh + o_h0)*out_w + ow*o_sw + o_w0) of an [*, ldo] matrix, which lets the four
 * sub-pixel phases of a transposed conv interleave into one tensor.
 *
 * Replaces: Conv3d(1,3,3) video_net.py:215; Conv3d 1x1x1 :246; Downsample Conv3d(1,4,4)/s2 :62;
 * Upsample ConvTranspose3d(1,4,4)/s2 :66 (as 4 phase GEMMs); Conv2d 1x1 to_qkv/to_out :322-323;
 * nn.Linear to_qkv/to_out :380-381; and the data-gradient of each (same op, transformed weights).
 *
 * Constraints: c0, c1, cout multiples of 64; stride in {1, 2}; stride 2 needs c1 == 0 and even h, w.
 */
typedef struct cesm_igemm_args {
    const void* a0; /* fp16 [n, h, w, c0] */
    const void* a1; /* fp16 [n, h, w, c1] or NULL */
    int32_t c0, c1;
    int32_t n, h, w;
    int32_t stride;
    int32_t num_taps;
    int32_t tap_dh[CESM_MAX_TAPS];
    int32_t tap_dw[CESM_MAX_TAPS];
    const void* wt; /* fp16 [cout, num_taps*(c0+c1)] */
    int32_t cout;
    int32_t oh, ow; /* output pixels iterated per image */
    void* out;      /* fp16 */
    int32_t ldo;
    int32_t out_h, out_w, o_sh, o_sw, o_h0, o_w0;
    const float* bias;    /* fp32 [cout] or NULL */
    const void* residual; /* fp16, addressed like out with pitch ldr, or NULL */
    int32_t ldr;
    /* Optional fused GroupNorm statistics (video_net.py:216): if gn_sums != NULL it is zeroed and then
     * receives, per sample b = image / gn_frames and group g of cout / gn_groups channels,
     * (sum, sum of squares) of the fp16-rounded outputs: fp32 [n / gn_frames][gn_groups][2]. */
    float* gn_sums;
    int32_t gn_groups;
    int32_t gn_frames;
    /* Optional channel-LayerNorm folded into a 64 -> 64 projection with a residual -- the whole temporal-attention
     * block at ONE frame without gradients (video_net.py:78-87 + :380-453: the softmax over a single key is 1, so
     * y = x + LN(x) (W_out W_v)^T).  If ln_colsum != NULL, `a0` and `residual` must both be the [rows, 64] tensor x,
     * `wt` = W * gamma (scaled per INPUT channel) and ln_colsum[co] = sum_ci wt[co][ci] (of the fp16 values); the
     * call returns   out = x + rstd(x) * (x wt^T - mean(x) * ln_colsum) (+ bias)   with the row statistics taken
     * over the 64 channels (biased variance, + ln_eps).  Needs cout == c0 == 64, c1 == 0, one tap, stride 1. */
    const float* ln_colsum;
    float ln_eps;
    int32_t reserved_;
} cesm_igemm_args;

int cesm_igemm(const cesm_igemm_args* args, void* stream);

/*
 * Weight gradient of the implicit GEMM above, contracted over pixels on tcgen05 tensor cores:
 *     dw[co, t, ci] = sum_{n, oh, ow}  dy[n, oh, ow, co] * X[n, oh*stride + tap_dh[t], ow*stride + tap_dw[t], ci]
 * X = concat(x0, x1) as in cesm_igemm.  dy pixel (n, oh, ow) is row
 * ((n*y_h + oh*y_sh + y_h0)*y_w + ow*y_sw + y_w0) of a fp16 [*, cout] matrix (sub-pixel phases of
 * a transposed conv).  dw is fp32 [cout, num_taps, c0+c1] and is overwritten (see dw_so for the
 * accumulate-in-place form).
 *
 * Replaces the weight-gradient halves of cuDNN/cuBLAS backward for the call sites listed above.
 */
typedef struct cesm_wgrad_args {
    const void* x0;
    const void* x1;
    int32_t c0, c1;
    int32_t n, h, w;
    int32_t stride;
    int32_t num_taps;
    int32_t tap_dh[CESM_MAX_TAPS];
    int32_t tap_dw[CESM_MAX_TAPS];
    const void* dy;
    int32_t cout;
    int32_t oh, ow;
    int32_t y_h, y_w, y_sh, y_sw, y_h0, y_w0;
    float* dw;
    /* Optional destination layout: if dw_so != 0 the result is ACCUMULATED (fp32 atomics, dw is not
     * cleared) at dw[co*dw_so + ci*dw_si + dw_tap_off[t]] -- e.g. straight into a PyTorch conv-weight
     * gradient [cout][cin][kh][kw] (dw_so = cin*kh*kw, dw_si = kh*kw, dw_tap_off[t] = t).  With
     * dw_so == 0, dw is the packed fp32 [cout][num_taps][c0+c1] and is overwritten. */
    long long dw_so, dw_si;
    int32_t dw_tap_off[CESM_MAX_TAPS];
} cesm_wgrad_args;

int cesm_wgrad(const cesm_wgrad_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Weight re-layout.  dst[o][t][i] (fp16) = src[o*so + i*si + tap_off[t]] (fp32): turns a PyTorch
 * conv / linear parameter into the [cout][taps][cin] operand of cesm_igemm (forward, or flipped /
 * transposed for the data gradient).  cesm_unpack_wgrad is the inverse scatter for fp32 gradients
 * produced by cesm_wgrad (accumulate != 0 adds into dst).
 * ---------------------------------------------------------------------------------------------- */
int cesm_pack_weight(const float* src, void* dst, int O, int T, int I, long long so, long long si,
                     const int32_t* tap_off, void* stream);
/* One launch re-packs many parameters: `descs_device` is an array of n descriptors in DEVICE memory
 * (the training engine refreshes every fp16 operand copy with it once per optimizer step). */
typedef struct cesm_pack_desc {
    const float* src;
    void* dst;
    int32_t O, T, I, pad_;
    long long so, si;
    int32_t tap_off[CESM_MAX_TAPS];
} cesm_pack_desc;
int cesm_pack_weights_batched(const cesm_pack_desc* descs_device, int n, void* stream);
/* Batched inverse for gradients: for each descriptor, dst (fp32, the parameter-gradient layout)
 * += src[o][t][i] (fp32 packed scratch written by cesm_wgrad) and the scratch is zeroed. */
int cesm_unpack_wgrads_batched(const cesm_pack_desc* descs_device, int n, void* stream);
/* Backward of the q/k/v projection (to_qkv, no bias; video_net.py:322, :380) for 64 input channels: data
 * gradient and weight gradient in ONE pass over dy (the two separate calls each stream the 768-wide dy from
 * HBM).  dy: fp16 [rows][cout]; x: fp16 [rows][64] (the projection's input, LN(x)); wt: fp16 [64][cout] = W^T
 * (the data-gradient operand cesm_pack_weight produces); dx: fp16 [rows][64] (written); dw: fp32, dw[co*dw_so +
 * ci] += sum_rows dy[row][co] * x[row][ci].  cin == 64, cout a multiple of 128, <= 768. */
int cesm_qkv_bwd(const void* dy, const void* x, const void* wt, void* dx, float* dw, long long dw_so, long long rows,
                 int cin, int cout, void* stream);

/* Scratch / statistics buffers the kernels ACCUMULATE into (igemm gn_sums, cesm_gn_bwd csum, cesm_tattn_bwd
 * dbias, cesm_linattn_fwd ws, cesm_linattn_bwd scratch) are zeroed by the call itself.  A caller that hands
 * in already-zeroed memory (the training engine carves them from one arena cleared once per step) switches
 * those ~70 per-step memsets off with on != 0.  Process-wide; default off. */
void cesm_set_prezeroed_scratch(int on);

/* Optimizer step of train.py:862-867 + 1078-1084 on FLAT fp32 buffers (every parameter, its gradient and
 * both AdamW moments are views into four contiguous arrays of n floats, 16-byte aligned):
 * torch.amp.GradScaler's unscale / inf check / skip / update (the gradients arrive multiplied by the loss
 * scale S because the activations and gradient stream are fp16, as under the reference's autocast),
 * global-norm clip (torch.nn.utils.clip_grad_norm_: coef = min(1, max_norm / (|g| + 1e-6)); max_norm <= 0
 * disables it) and torch.optim.AdamW's update, all on the device so that a CUDA-graph replay advances them.
 * `partials`: fp32 scratch of cesm_adamw_partials() floats.
 * `state`: fp32[CESM_OPT_STATE_FLOATS] in device memory:
 *   [0] step count (incremented by every non-skipped call)   [1] <- unscaled pre-clip gradient norm
 *   [2] loss scale S (halved after an overflow, doubled after [8] clean steps; set 1 for unscaled gradients)
 *   [3] growth tracker   [4] <- 1 if this call found a non-finite gradient and skipped the update
 *   [5] skipped-step count   [6] learning rate   [7] weight decay   [8] growth interval (0: static scale)
 * Three launches, no host sync. */
#define CESM_OPT_STATE_FLOATS 16
int cesm_adamw_partials(void);
int cesm_adamw_step(float* p, const float* g, float* m, float* v, long long n, float* partials, float* state,
                    float beta1, float beta2, float eps, float max_norm, void* stream);
/* cesm_adamw_step plus an exponential moving average of the parameters, updated in the same pass and the same
 * three launches.  `ema`: fp32[n], 16-byte aligned, laid out like `p`.  With k = the step count after this step
 * (state[0] + 1), every non-skipped call does, after the AdamW update of p:
 *   k <= ema_start:  ema = p                                   (exact copy)
 *   otherwise:       ema = fmaf(1 - ema_decay, p - ema, ema)   (1 - ema_decay rounded once to fp32)
 * ema_start = 1 is torch.optim.swa_utils.AveragedModel(multi_avg_fn=get_ema_multi_avg_fn(ema_decay)) updated after
 * every optimizer step.  A skipped step (non-finite gradient) leaves `ema` unchanged.  Requires 0 <= ema_decay < 1
 * and ema_start >= 0. */
int cesm_adamw_ema_step(float* p, const float* g, float* m, float* v, float* ema, long long n, float* partials,
                        float* state, float beta1, float beta2, float eps, float max_norm, double ema_decay,
                        long long ema_start, void* stream);
int cesm_unpack_wgrad(const float* src, float* dst, int O, int T, int I, long long so, long long si,
                      const int32_t* tap_off, int accumulate, void* stream);
/* out[c] (+)= sum over rows of fp16 x[M][C] (bias gradients).  `accumulate` != 0 here and in the other
 * backward entry points adds into the parameter-gradient outputs instead of overwriting them, which
 * lets the caller pass the parameter's .grad buffer directly. */
int cesm_colsum(const void* x, float* out, long long M, int C, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------
 * GroupNorm + FiLM + SiLU (+ residual), video_net.py:216-227 and :265.   x: fp16 [B][P][C],
 * P = frames*H*W (statistics couple the frames of a sample, as nn.GroupNorm on a 5-D tensor does).
 *   sums  : fp32 [B][G][2]  (sum, sum of squares), written by cesm_gn_stats
 *   film  : fp32 [B][2C] = (scale | shift) from the time-embedding MLP, or NULL
 *   out   = silu(((x-mean)*rstd*gamma+beta)*(scale+1)+shift) (+ residual)
 * cesm_gn_bwd returns dx (fp16), dgamma/dbeta [C], dfilm [B][2C] (if film) and, if dconv_bias is not
 * NULL, dconv_bias[c] = sum over samples and pixels of dx -- the bias gradient of the convolution
 * that produced x (video_net.py:215), from the same per-channel sums.  csum is fp32 scratch [B][C][3].
 * ---------------------------------------------------------------------------------------------- */
int cesm_gn_stats(const void* x, float* sums, int B, long long P, int C, int G, void* stream);
int cesm_gn_apply_fwd(const void* x, const float* sums, const float* gamma, const float* beta, const float* film,
                      const void* residual, void* out, int B, long long P, int C, int G, float eps, void* stream);
int cesm_gn_bwd(const void* x, const void* dout, const float* sums, const float* gamma, const float* beta,
                const float* film, float* csum, void* dx, float* dgamma, float* dbeta, float* dfilm,
                float* dconv_bias, int B, long long P, int C, int G, float eps, int accumulate_params, void* stream);

/* Channel LayerNorm with gain only, video_net.py:78-87.  x, out, dy, dres, dx: fp16 [M][C],
 * C in {64, 128, 256, 512, 1024}.
 * bwd: dx = LN'(dy) (+ dres if not NULL); dgamma fp32 [C] is overwritten. */
int cesm_ln_fwd(const void* x, const float* gamma, void* out, long long M, int C, float eps, void* stream);
int cesm_ln_bwd(const void* x, const float* gamma, const void* dy, const void* dres, void* dx, float* dgamma,
                long long M, int C, float eps, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Temporal attention core, video_net.py:413-453 + rotary_embedding.py:29-48, fused:
 * q*scale -> RoPE(q), RoPE(k) -> q.k + rel-pos bias -> online softmax over frames -> .v
 *   qkv : fp16 [B*F*HW][3*H*32] (q | k | v), row = (b*F + f)*HW + pixel
 *   bias: fp32 [H][F][F];  cs, sn: fp32 [F][16] rotary cos / sin;  out: fp16 [B*F*HW][H*32]
 *   lse : fp32 [B*F*HW][H] log-sum-exp saved for the backward.  For F <= 4 (the training window
 *         K=3 and the one-frame sampling call) a register-resident kernel is used whose backward
 *         recomputes the softmax from qkv: lse may then be NULL in fwd, and out / lse NULL in bwd.
 * ---------------------------------------------------------------------------------------------- */
int cesm_tattn_fwd(const void* qkv, const float* bias, const float* cs, const float* sn, void* out, float* lse,
                   int B, int F, int HW, int H, int dim_head, float scale, void* stream);
int cesm_tattn_bwd(const void* qkv, const float* bias, const float* cs, const float* sn, const void* out,
                   const float* lse, const void* dout, void* dqkv, float* dbias, int B, int F, int HW, int H,
                   int dim_head, float scale, void* stream);

/* Forward only, without gradients: short windows (F <= 3) FUSED WITH THE q/k/v PROJECTION, 64 input channels,
 * 8 heads of 32 (csrc/tattn_proj.cu): out = attention(xn Wq^T, xn Wk^T, xn Wv^T) with q, k, v never written to
 * memory.  A training step projects q/k/v with cesm_igemm and runs cesm_tattn_fwd / cesm_tattn_bwd instead.
 *   xn  : fp16 [B*F*HW][64] = LayerNorm(x);  wqkv: fp16 [768][64] (to_qkv.weight as cesm_pack_weight lays it out)
 *   bias: fp32 [8][F][F];  cs, sn: fp32 [F][16];  out: fp16 [B*F*HW][256].  HW must be a multiple of 16. */
int cesm_tattn_proj_fwd(const void* xn, const void* wqkv, const float* bias, const float* cs, const float* sn, void* out,
                        int B, int F, int HW, int H, int dim_head, int cin, float scale, void* stream);

/* Long windows (F > 4, up to 128 frames; BASELINE.json configs[4]): the same computation, flash style.  A CTA
 * stages every frame of one pixel column in shared memory once and one warp per head runs the F x F attention on
 * the tensor cores (mma.sync m16n8k16), instead of each query re-reading all keys / values from global memory.
 * The relative-position bias of video_net.py:302-310 depends on (key - query) only, so it is passed by diagonal:
 *   bias_diag : fp32 [H][2F-1], bias_diag[h][d + F - 1] = bias[h][i][i + d];  dbias_diag likewise (zeroed by the call).
 * lse is always written (fwd) / read (bwd). */
int cesm_tattn_long_max_frames(void);
int cesm_tattn_long_fwd(const void* qkv, const float* bias_diag, const float* cs, const float* sn, void* out,
                        float* lse, int B, int F, int HW, int H, int dim_head, float scale, void* stream);
int cesm_tattn_long_bwd(const void* qkv, const float* bias_diag, const float* cs, const float* sn, const void* out,
                        const float* lse, const void* dout, void* dqkv, float* dbias_diag, int B, int F, int HW, int H,
                        int dim_head, float scale, void* stream);

/* Bottleneck spatial attention (use_mid_attn=True, video_net.py:713-719): per image of n pixels and per head,
 * out = softmax((q * scale) k^T) v over all n pixels, no mask, no bias, no rotary embedding; flash style on the
 * tensor cores (csrc/mid_attn.cu).  dim_head must be 32.
 *   qkv : fp16 [NI*n][3*H*32] (q | k | v, each (head, d));  out / dout: fp16 [NI*n][H*32]
 *   lse : fp32 [NI*n][H], log sum_j exp(scale q.k_j), written by fwd and read by bwd
 *   delta: fp32 [NI*n][H] scratch of the backward (rowsum(dout * out), overwritten)
 *   dqkv: fp16 [NI*n][3*H*32], every element written; no atomics, so the backward is bitwise deterministic.
 * fp16 pointers must be 16-byte aligned.  1 <= NI <= 65535, n >= 1. */
int cesm_mattn_fwd(const void* qkv, void* out, float* lse, int NI, int n, int H, int dim_head, float scale, void* stream);
int cesm_mattn_bwd(const void* qkv, const void* out, const float* lse, const void* dout, void* dqkv, float* delta, int NI,
                   int n, int H, int dim_head, float scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Spatial linear attention core, video_net.py:338-344, per image (frame) of n pixels and head:
 * qs = scale*softmax(q) over d, kh = softmax(k) over the n pixels, ctx = kh^T v, out = qs ctx.
 * Both contractions run as warp-level fp16 tensor-core tiles; the softmaxed operands are
 * recomputed from qkv where needed, so only q, k, v, out (and their gradients) touch HBM.
 *   qkv: fp16 [NI*n][3*H*32];  out: fp16 [NI*n][H*32];  1 <= H <= 8
 *   ws : fp32 [cesm_linattn_ws_floats(NI, H)], written by fwd and read by bwd; per image it
 *        holds the column maxima of k (order-encoded), Z = sum_p exp(k - max) and ctx [H][32][32]
 *   bwd: scratch fp32 [NI*H*32*32 + NI*H*32]; dqkv: fp16 [NI*n][3*H*32]
 * ---------------------------------------------------------------------------------------------- */
size_t cesm_linattn_ws_floats(int NI, int H);
int cesm_linattn_fwd(const void* qkv, float* ws, void* out, int NI, int n, int H, int dim_head, float scale,
                     void* stream);
int cesm_linattn_bwd(const void* qkv, float* ws, const void* dout, float* scratch, void* dqkv, int NI, int n, int H,
                     int dim_head, float scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Network boundary convs.
 * Input conv (video_net.py:808-815 + model.py:110-121): 7x7, the two fp32 input planes (noisy
 * target, condition) are read in place -- channel concat and frame broadcast (f0/f1 = 1 or F frames
 * per sample) are folded into the kernel.  out: fp16 [B*F][H][W][64].  Only the weight gradient
 * exists (network inputs need no gradient).
 * Output conv (video_net.py:763 + model.py:129-130): 1x1x1, 64 -> 1, evaluated on the centre
 * frame only (the reference computes every frame and then selects frame F//2).
 * ---------------------------------------------------------------------------------------------- */
/* All FiLM projections of a pass in one launch (video_net.py:238-241: SiLU -> Linear(time_dim, 2*dim_out), one
 * per ResnetBlock, all fed by the same time embedding x [B][K]).  `layers_device`: n_layers descriptors in
 * DEVICE memory; n0 = running sum of N over the preceding layers, n_total = sum of N.  Outputs and output
 * gradients are packed layer after layer: layer i owns the contiguous [B][N_i] block at float offset B*n0_i
 * of y / dy.  cesm_film_fwd: y_i = silu(x) W_i^T + bias_i.  cesm_film_bwd: dW_i, db_i (+= if accumulate) and,
 * if dx is not NULL, dx = silu'(x) * sum_i dy_i W_i. */
typedef struct cesm_film_desc {
    const float* W;      /* [N][K] */
    const float* bias;   /* [N] */
    float* dW;           /* [N][K] (backward) */
    float* db;           /* [N]    (backward) */
    int32_t N, n0;
} cesm_film_desc;
int cesm_film_fwd(const float* x, const cesm_film_desc* layers_device, float* y, int n_layers, int n_total, int B,
                  int K, void* stream);
int cesm_film_bwd(const float* x, const cesm_film_desc* layers_device, const float* dy, int n_layers, int n_total,
                  float* dx, int B, int K, int accumulate, void* stream);

/* On-device data path (dataset_single_member.py:168-196; SURVEY 8(f) rank 3).  cond, tgt: fp32 [T][M][H][W]
 * resident in device memory.  plan: int32 [B][6] = {member, first window frame, target frame, crop row,
 * crop col, time-reverse flag} in device memory.  Writes cond_out fp32 [B][K][h][w] (= the reference's
 * [B,1,K,h,w]) and x0_out fp32 [B][h][w].  With the flag the frames left and right of the centre are flipped
 * (the reference's centred time reversal). */
int cesm_gather_windows(const float* cond, const float* tgt, const int* plan, float* cond_out, float* x0_out, int B,
                        int T, int M, int H, int W, int K, int h, int w, void* stream);

/* Tensor-core form of the same input convolution.  cesm_input_patches writes the im2col matrix
 * fp16 [B*F][H][W][kpad] = [hi(x) | lo(x) | 1 | 1 | 0...] (x = the 2*ks*ks taps of the two fp32 planes, frame
 * broadcast as above; hi = fp16(x), lo = fp16(x - hi)); cesm_input_weight_pack writes the matching operand
 * fp16 [cout][kpad] = [w | w | bias_hi | bias_lo | 0].  cesm_igemm (1 tap) of the two is the convolution with
 * its bias; cesm_wgrad of (patches, dy) is [dW_hi-block | dW_lo-block | db | db | 0]: dW = sum of the two
 * blocks.  ks = 7, kpad = 256. */
int cesm_input_patches(const float* in0, const float* in1, int f0, int f1, void* out, int B, int F, int H, int W,
                       int ks, int kpad, void* stream);
/* cesm_input_patches with condition dropout: keep is an fp32 [B] device vector (NULL: keep all), and batch element b
 * reads its in1 plane as zeros where keep[b] == 0.  The GEMM and the weight gradient over these patches then see the
 * null condition; no masked copy of in1 is made. */
int cesm_input_patches_masked(const float* in0, const float* in1, int f0, int f1, const float* keep, void* out, int B,
                              int F, int H, int W, int ks, int kpad, void* stream);
int cesm_input_weight_pack(const float* w, const float* bias, void* out, int cout, int ks, int kpad, void* stream);
int cesm_input_conv_fwd(const float* in0, const float* in1, int f0, int f1, const float* w, const float* bias,
                        void* out, int B, int F, int H, int W, int ks, int cout, void* stream);
int cesm_input_conv_wgrad(const float* in0, const float* in1, int f0, int f1, const void* dy, float* dw, float* db,
                          int B, int F, int H, int W, int ks, int cout, void* stream);
/* Data gradient of the input convolution: the transposed 7x7 convolution (zero padding, fp32 accumulation) of
 * dy fp16 [B*F][H][W][cout] with the fp32 weight [cout][2][ks][ks], giving d_in0 fp32 [B][f0][H][W] and
 * d_in1 fp32 [B][f1][H][W].  A plane with one frame while F > 1 (the broadcast of cesm_input_conv_fwd) receives
 * the sum over the F frames.  out = scale * grad, or out += scale * grad with `accumulate`.  Either output may be
 * NULL (not requested), not both.  ks = 7, cout = 64, B <= 65535. */
int cesm_input_conv_dgrad(const void* dy, const float* w, float* d_in0, float* d_in1, int f0, int f1, int B, int F,
                          int H, int W, int ks, int cout, float scale, int accumulate, void* stream);
/* cesm_input_conv_dgrad of a forward made with cesm_input_patches_masked: where keep[b] == 0, d_in1 of batch element
 * b is 0 (written as 0, or nothing added with `accumulate`).  keep NULL: cesm_input_conv_dgrad. */
int cesm_input_conv_dgrad_masked(const void* dy, const float* w, float* d_in0, float* d_in1, const float* keep, int f0,
                                 int f1, int B, int F, int H, int W, int ks, int cout, float scale, int accumulate,
                                 void* stream);
int cesm_out_conv_fwd(const void* a, const float* w, const float* bias, float* eps, int B, int F, int mid,
                      long long HW, int C, void* stream);
int cesm_out_conv_bwd(const void* a, const float* w, const float* deps, void* da, float* dw, float* db, int B, int F,
                      int mid, long long HW, int C, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Time embedding and small fp32 linears (video_net.py:101-113, 651-656, 238-241).
 * small_linear: y[b][n] = sum_k act(x[b][k]) W[n][k] + bias[n], act = SiLU if act_silu_in.
 * ---------------------------------------------------------------------------------------------- */
int cesm_sinusoidal(const long long* t, float* out, int B, int dim, void* stream);
int cesm_small_linear_fwd(const float* x, const float* W, const float* bias, float* y, int B, int K, int N,
                          int act_silu_in, void* stream);
int cesm_small_linear_bwd(const float* x, const float* W, const float* dy, float* dx, float* dW, float* db, int B,
                          int K, int N, int act_silu_in, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------
 * DDPM elementwise steps (model.py:168-208); t is an int64 device vector, schedule buffers fp32 [T].
 * ---------------------------------------------------------------------------------------------- */
int cesm_q_sample(const float* x0, const float* noise, const long long* t, const float* sqrt_ac,
                  const float* sqrt_1mac, float* xt, int B, long long per_sample, void* stream);
/* Backward of cesm_q_sample: dx0 = sqrt_ac[t[b]] * g, dnoise = sqrt_1mac[t[b]] * g.  Either output may be NULL
 * (not requested), not both. */
int cesm_q_sample_bwd(const float* g, const long long* t, const float* sqrt_ac, const float* sqrt_1mac, float* dx0,
                      float* dnoise, int B, long long per_sample, void* stream);
int cesm_mse_fwd(const float* eps, const float* noise, float* diff, float* loss, long long total, void* stream);
int cesm_scale_by_scalar(const float* in, const float* gscale, float factor, float* out, long long total,
                         void* stream);
/* Diffusion objective with a per-timestep target and weight (v-prediction, Min-SNR-gamma).  Per sample b with
 * tb = t[b]: target = c_n[tb] * noise + c_x[tb] * x0 from the fp32 [T][2] rows (c_n, c_x) of tgt_coef; a NULL
 * tgt_coef is the eps target (target = noise, x0 not read, may be NULL).  diff = pred - target, and
 * *loss = sum_b w[tb] * sum diff^2 / (B * per_sample) with w = weight[T] (NULL: 1); *loss is zeroed first.  A t
 * outside [0, T) makes diff and *loss NaN.  Rejects T, B, per_sample <= 0, B > 65535 and NULL pred, noise, t, diff
 * or loss with CESM_ERR_INVALID. */
int cesm_diffusion_loss_fwd(const float* pred, const float* x0, const float* noise, const long long* t,
                            const float* tgt_coef, const float* weight, float* diff, float* loss, int B,
                            long long per_sample, int T, void* stream);
/* Backward of cesm_diffusion_loss_fwd for an incoming gradient *gscale (device scalar): dpred = factor * g * w[tb] *
 * diff, dnoise = -c_n[tb] * dpred and dx0 = -c_x[tb] * dpred (the target's share of those input gradients).  Any
 * output may be NULL, not all three.  A t outside [0, T) writes NaN. */
int cesm_diffusion_loss_bwd(const float* diff, const long long* t, const float* tgt_coef, const float* weight,
                            const float* gscale, float factor, float* dpred, float* dnoise, float* dx0, int B,
                            long long per_sample, int T, void* stream);
int cesm_p_sample(const float* xt, const float* eps, const float* z, const long long* t, const float* betas,
                  const float* sqrt_1mac, const float* sqrt_recip_a, const float* post_var, float* out, int B,
                  long long per_sample, void* stream);
/* Strided DDIM step: out = A[t]*xt + B[t]*eps + S[t]*z per sample, coef = fp32 [T][3] rows (A, B, S) computed on the
 * host in float64.  out may equal xt.  z may be NULL when every S is 0.  t_out (optional, must not alias t) receives
 * next_t[t] from the int64 [T] table.  A t outside [0, T) writes NaN.  Rejects T, B, per_sample <= 0 and NULL xt,
 * eps, t, coef or out with CESM_ERR_INVALID. */
int cesm_ddim_step(const float* xt, const float* eps, const float* z, const long long* t, const float* coef,
                   const long long* next_t, long long* t_out, float* out, int T, int B, long long per_sample,
                   void* stream);
/* DPM-Solver++(2M) step: x0 = P[t]*xt + Q[t]*eps, out = R[t]*xt + K0[t]*x0 + K1[t]*hist, then hist = x0, from the
 * fp32 [T][5] rows (P, Q, R, K0, K1) computed on the host in float64.  hist (B*per_sample floats) is read only where
 * K1 != 0.  out may equal xt.  t_out (optional, must not alias t) receives next_t[t] from the int64 [T] table.  A t
 * outside [0, T) writes NaN to out and hist.  Rejects T, B, per_sample <= 0, NULL xt, eps, hist, t, coef or out, and
 * a hist that overlaps any other buffer with CESM_ERR_INVALID. */
int cesm_dpm_step(const float* xt, const float* eps, float* hist, const long long* t, const float* coef,
                  const long long* next_t, long long* t_out, float* out, int T, int B, long long per_sample,
                  void* stream);
/* Classifier-free guidance.  The *_guided steps take eps with 2B rows of per_sample floats: rows [0, B) are the
 * network's predictions with the fields' conditions, rows [B, 2B) its predictions for the same fields with the null
 * (all-zero) condition.  They update the B fields with c + guidance * (c - u) = (1 + w) c - w u, element by element,
 * in place of eps, in the network's own output space (eps or v); nothing else changes.  guidance must be finite and
 * > 0 (CESM_ERR_INVALID otherwise); w = 0 is the unguided entry point. */
int cesm_p_sample_guided(const float* xt, const float* eps, const float* z, const long long* t, const float* betas,
                         const float* sqrt_1mac, const float* sqrt_recip_a, const float* post_var, float* out, int B,
                         long long per_sample, float guidance, void* stream);
int cesm_ddim_step_guided(const float* xt, const float* eps, const float* z, const long long* t, const float* coef,
                          const long long* next_t, long long* t_out, float* out, int T, int B, long long per_sample,
                          float guidance, void* stream);
int cesm_dpm_step_guided(const float* xt, const float* eps, float* hist, const long long* t, const float* coef,
                         const long long* next_t, long long* t_out, float* out, int T, int B, long long per_sample,
                         float guidance, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Seeded sampling noise.  Element e of field f in draw d is word e & 3 of Philox4x32-10 with counter
 * (e >> 2, d, f_lo, f_hi) and key (seed_lo, seed_hi), mapped to normals by Box-Muller on the word pairs (w0, w1) and
 * (w2, w3): u = ((w >> 9) + 0.5) * 2^-23 (exact in fp32, inside (0, 1)), r = sqrtf(-2 logf(u_a)),
 * (r cospi(2 u_b), r sinpi(2 u_b)).  A value depends
 * on (seed, field id, draw, e) only.  x_T is draw 0xFFFFFFFF; the reverse step leaving timestep t draws with d = t.
 * field_ids is an int64 [B] device vector (one id per row); rows are per_sample floats.  All three reject B outside
 * [1, 65535], per_sample outside [1, 2^34] and NULL pointers with CESM_ERR_INVALID.
 * ---------------------------------------------------------------------------------------------- */
/* out[b] = the normals of field field_ids[b] in `draw`. */
int cesm_field_normal(unsigned seed_lo, unsigned seed_hi, const long long* field_ids, unsigned draw, float* out,
                      int B, long long per_sample, void* stream);
/* cesm_p_sample with z = the field's draw t[b], made in registers: bit-identical to cesm_p_sample fed
 * cesm_field_normal(draw = t[b]).  out may equal xt.  A t outside [0, T) writes NaN; rejects T <= 0. */
int cesm_p_sample_seeded(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                         const long long* field_ids, const long long* t, const float* betas, const float* sqrt_1mac,
                         const float* sqrt_recip_a, const float* post_var, float* out, int T, int B,
                         long long per_sample, void* stream);
/* cesm_ddim_step with z = the field's draw t[b], made in registers: bit-identical to cesm_ddim_step fed
 * cesm_field_normal(draw = t[b]).  Same out / t_out / NaN contract; t_out must not alias t or field_ids. */
int cesm_ddim_step_seeded(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                          const long long* field_ids, const long long* t, const float* coef, const long long* next_t,
                          long long* t_out, float* out, int T, int B, long long per_sample, void* stream);
/* The seeded steps with classifier-free guidance (eps with 2B rows, as cesm_ddim_step_guided).  The noise is drawn for
 * the B fields only, by field id, so a guided field does not depend on its row or batch either. */
int cesm_p_sample_seeded_guided(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                                const long long* field_ids, const long long* t, const float* betas,
                                const float* sqrt_1mac, const float* sqrt_recip_a, const float* post_var, float* out,
                                int T, int B, long long per_sample, float guidance, void* stream);
int cesm_ddim_step_seeded_guided(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                                 const long long* field_ids, const long long* t, const float* coef,
                                 const long long* next_t, long long* t_out, float* out, int T, int B,
                                 long long per_sample, float guidance, void* stream);
/* Condition dropout of a training step: keep[b] = 1 if u >= p else 0, with u = ((w0 >> 9) + 0.5) * 2^-23 from word 0
 * of Philox4x32-10 with counter (g_lo, g_hi, s_lo, s_hi) and key (seed_lo, seed_hi), g = first + b the sample's index
 * in the global batch and s = *step (an int64 device counter); then *step += 1.  The masks depend on (seed, step, g)
 * only: the same for a global batch on one GPU or split over ranks.  Rejects B < 1, first < 0, p outside [0, 1) and
 * NULL pointers with CESM_ERR_INVALID. */
int cesm_cond_keep(unsigned seed_lo, unsigned seed_hi, long long* step, long long first, float p, float* keep, int B,
                   void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CESM_B200_H */
