/* flowk.h - C ABI of libflowk.so: the sm_100a kernels behind the mAR-SCF flow-step path.
 *
 * The reference has no FFI layer of its own (SURVEY.md section 8b): its boundary is the
 * torch.nn.Module contract `layer(x, logdet, reverse) -> (x', logdet')`.  Each entry point
 * below replaces the eager ATen launch sequence of one such module's forward / reverse
 * branch (cited as file:line of the reference repository) and is what a reference-side
 * binding would load (ctypes stub in INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to float32, NCHW contiguous ("HW" = H*W, flattened);
 *   - the caller owns all memory; kernels never allocate, free or keep state between calls;
 *   - work is enqueued on `stream` and the call returns immediately (stream-ordered, re-entrant);
 *   - return value: FLOWK_OK, a FLOWK_ERR_* code, or FLOWK_ERR_CUDA_BASE + cudaError_t;
 *   - `ldj_in` may be NULL (treated as zeros); `ldj_out` NULL skips the log-det output, like the
 *     reference's `logdet=None`; ldj_in == ldj_out (in place) is allowed;
 *   - `ws` is a reduction workspace of flowk_ldj_workspace_bytes(B) bytes that must be zero
 *     when first used and is left zeroed-where-needed by every call; one workspace per stream.
 *     Per-sample log-det sums are reduced in a fixed order (bit-reproducible run to run).
 */
#ifndef FLOWK_H_
#define FLOWK_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* flowk_stream_t;   /* == cudaStream_t */

enum {
  FLOWK_OK = 0,
  FLOWK_ERR_SHAPE = 1,      /* reference: AssertionError (common_modules.py:21,38) */
  FLOWK_ERR_ALIGN = 2,      /* pointer not 4-byte aligned / vector path precondition */
  FLOWK_ERR_ARG = 3,        /* NULL where data is required, unsupported K, ... */
  FLOWK_ERR_CUDA_BASE = 1000
};

int flowk_abi_version(void);
const char* flowk_error_string(int status);
size_t flowk_ldj_workspace_bytes(int B);

/* squeeze2d / unsqueeze2d, flow_modules/common_modules.py:12-42.
 * squeeze:   y[b, c*f*f + fh*f + fw, h, w] = x[b, c, h*f+fh, w*f+fw];  x is [B,C,H,W], y is [B,C*f*f,H/f,W/f].
 * unsqueeze: exact inverse; x is [B,C,H,W] with C % (f*f) == 0, y is [B,C/(f*f),H*f,W*f]. */
int flowk_squeeze2d(const float* x, float* y, int B, int C, int H, int W, int factor, flowk_stream_t stream);
int flowk_unsqueeze2d(const float* x, float* y, int B, int C, int H, int W, int factor, flowk_stream_t stream);

/* Actnormlayer data-dependent init, common_modules.py:141-151:
 * bias[c] = -mean_{b,h,w} x ; logs[c] = log(scale / (sqrt(mean((x+bias)^2)) + eps)). */
int flowk_actnorm_init(const float* x, float* bias, float* logs, int B, int C, int HW,
                       float scale, float eps, flowk_stream_t stream);

/* Per-channel affine map  y = (x + pre[c]) * mul[c] + post[c].
 * Actnormlayer forward (pre=bias, mul=e^{logs}, post=0) and reverse (pre=0, mul=e^{-logs}, post=-bias),
 * common_modules.py:153-186.  ldj_out[b] = ldj_in[b] + ldj_add[0] (device scalar, may be NULL). */
int flowk_channel_scale(const float* x, const float* pre, const float* mul, const float* post, float* y,
                        const float* ldj_in, const float* ldj_add, float* ldj_out,
                        int B, int C, int HW, flowk_stream_t stream);

/* Per-pixel channel mixing  y[b,o,p] = sum_i Wm[o*C+i] * x[b,i,p] + bias[o]   (bias may be NULL).
 * InvertibleConv1x1 forward/reverse (common_modules.py:113-127) and, with ActNorm folded into
 * Wm/bias by the caller, the fused ActNorm->InvConv step of FlowStep (marscf_main.py:64-68,95-97).
 * ldj_out[b] = ldj_in[b] + ldj_add[0].
 * in_squeeze != 0: x is the UN-squeezed tensor [B, C/4, 2H', 2W'] (H'*W' = HW, `W` = W') and the
 * squeeze2d index map is applied on load (SqueezeLayer fused into the first step of a level).
 * out_unsqueeze != 0: y is written through the unsqueeze2d map (last step of a level, reverse). */
int flowk_channel_mix(const float* x, const float* Wm, const float* bias, float* y,
                      const float* ldj_in, const float* ldj_add, float* ldj_out,
                      int B, int C, int H, int W, int in_squeeze, int out_unsqueeze,
                      flowk_stream_t stream);

/* AffineCoupling arithmetic, flow_modules/affine_coupling.py:100-124, given the conditioner output
 * h = NN_net(x[:, :C/2]) of shape [B,C,HW]: shift = h[:,0::2], scale = sigmoid(h[:,1::2] + 2).
 *   fwd: y = cat(x1, x2*scale + shift),  ldj_out = ldj_in + sum log(scale)
 *   inv: y = cat(x1, (x2 - shift)/scale), ldj_out = ldj_in - sum log(scale)
 *   bwd: given gy = dL/dy [B,C,HW] and gldj = dL/dldj_out [B] (may be NULL) of the FORWARD op,
 *        writes gx (second half only; the caller adds gy's first half) and gh [B,C,HW]. */
int flowk_affine_coupling_fwd(const float* x, const float* h, float* y, const float* ldj_in, float* ldj_out,
                              void* ws, int B, int C, int HW, flowk_stream_t stream);
int flowk_affine_coupling_inv(const float* x, const float* h, float* y, const float* ldj_in, float* ldj_out,
                              void* ws, int B, int C, int HW, flowk_stream_t stream);
int flowk_affine_coupling_bwd(const float* x, const float* h, const float* gy, const float* gldj,
                              float* gx, float* gh, int B, int C, int HW, flowk_stream_t stream);

/* MixLogCDFCoupling arithmetic, flow_modules/mixlogcdf_coupling.py:37-57 + log_dist.py, given the RAW
 * conditioner output `raw` = out_conv(...) of shape [B, (2+3K)*c, HW], c = C/2 (mixlogcdf_nn.py:69-76):
 * plane j of channel ch is raw[b, j*c+ch, p]; planes (0, 1, 2.., 2+K.., 2+2K..) = (a_raw, b, pi, mu, s);
 * a = rescale[ch] * tanh(a_raw), s = max(s, -7).  Only K == 32 is built (marscf_main.py:41).
 *   fwd: out = (logit(F(x1)) + b) * e^a,  ldj += sum(log f(x1) - log u - log(1-u) + a)
 *        y = cat(out, x2)           (flip == 0)
 *        y = cat(x2, out)           (flip != 0: TupleFlip fused, marscf_main.py:72-73)
 *   inv: input is cat(v, x2) (flip == 0) or cat(x2, v) (flip != 0, marscf_main.py:89-90);
 *        x1 = F^-1(clamp(sigmoid(v e^-a - b), 1e-5, 1-1e-5)) by bisection (log_dist.py:43-72),
 *        ldj -= sum(a + softplus(t) + softplus(-t) + log f(x1));  y = cat(x1, x2) always.
 *   bwd: gradients of the forward op given gy = dL/dy [B,C,HW] and gldj = dL/dldj_out [B] (may be NULL):
 *        gx [B,C,HW] (x2 half = gy's pass-through half; the conditioner's input gradient is added by
 *        the caller), graw [B,(2+3K)c,HW], and ga_tanh [B,c,HW] = dL/da * tanh(a_raw), whose sum over
 *        (B,HW) is the gradient of `rescale`. */
int flowk_mixlogcdf_fwd(const float* x, const float* raw, const float* rescale, float* y,
                        const float* ldj_in, float* ldj_out, void* ws,
                        int B, int C, int HW, int K, int flip, flowk_stream_t stream);
int flowk_mixlogcdf_inv(const float* x, const float* raw, const float* rescale, float* y,
                        const float* ldj_in, float* ldj_out, void* ws,
                        int B, int C, int HW, int K, int flip, flowk_stream_t stream);
int flowk_mixlogcdf_bwd(const float* x, const float* raw, const float* rescale,
                        const float* gy, const float* gldj, float* gx, float* graw, float* ga_tanh,
                        int B, int C, int HW, int K, int flip, flowk_stream_t stream);

/* log_dist.py functions on explicit parameter tensors pi/mu/s of shape [B,K,N] and x,y,out of [B,N]
 * (N = c*H*W flattened): mixture_log_cdf :34, mixture_log_pdf :25, mixture_inv_cdf :43 (bisection;
 * the (0,1) domain check of :46-47 is the caller's, it needs a host read). */
int flowk_mixture_log_cdf(const float* x, const float* pi, const float* mu, const float* s, float* out,
                          int B, int K, int N, flowk_stream_t stream);
int flowk_mixture_log_pdf(const float* x, const float* pi, const float* mu, const float* s, float* out,
                          int B, int K, int N, flowk_stream_t stream);
int flowk_mixture_inv_cdf(const float* y, const float* pi, const float* mu, const float* s, float* out,
                          int B, int K, int N, flowk_stream_t stream);

/* ---- conditioner layers on the tensor cores (tcgen05, 3xTF32 split operands) --------------------------------
 * Implicit-GEMM convolution / linear layer in NHWC:
 *     D[m, n] = sum_{tap, c} A[pos(m) + shift(tap), c] * Wt[n, tap*Cin + c]      taps = 1 (1x1 / Linear) or 9 (3x3, "same")
 * replacing F.conv2d / F.linear of flow_modules/mixlogcdf_nn.py:12-29,121-122,134,149 and affine_coupling.py:27-80.
 * Every operand is an (hi, lo) pair of fp32 arrays: hi = value with the 13 low mantissa bits cleared, lo = value - hi.
 * Constraints: Cin % 32 == 0; W divides 128 and H*W divides or is a multiple of 128.
 *
 * `pre` selects what happens to an accumulator row before it is written:
 *   FLOWK_PRE_BIAS        y = D + bias
 *   FLOWK_PRE_GLU_RES_LN  N = 2C: y = LayerNorm_C((D_a + bias_a) * sigmoid(D_b + bias_b) + res) * gamma + beta
 *                         (GatedConv / GatedAttn gate + residual + norm, mixlogcdf_nn.py:92-101,149-151,257-258)
 *   FLOWK_PRE_LSTM        N = 4 hid gate columns [i | f | g | o] of a ConvLSTM cell (the mAR channel prior,
 *                         mar_prior/convolutional_rnn/functional.py:30-52): gates = D + bias + res (res = input-to-hidden
 *                         gates [M, N] of this step), gamma = c_{t-1} [M, hid]; writes c_t = sig(f) c + sig(i) tanh(g) to
 *                         out_f32 [M, hid] and h_t = sig(o) tanh(c_t) to out_hi / out_lo [M, hid]; out_mask is ignored
 * `out_mask` selects the forms y is written in (Nout = N, or C after the GLU):
 *   FLOWK_OUT_F32        out_f32[m, Nout]
 *   FLOWK_OUT_HILO       out_hi/out_lo[m, Nout]                       operand of the next GEMM
 *   FLOWK_OUT_HILO_POS   out_hi/out_lo[m, Nout] of y + pos[m % HW]    (GatedAttn input, mixlogcdf_nn.py:130-131)
 *   FLOWK_OUT_HILO_CELU  out_hi/out_lo[m, 2*Nout] of [elu(y) | elu(-y)]   (concat_elu, mixlogcdf_nn.py:8-10)
 *   FLOWK_OUT_NCHW       out_nchw[b, n, hw]                            (raw parameter tensor for flowk_mixlogcdf_*)
 *   FLOWK_OUT_HILO_RELU  out_hi/out_lo[m, Nout] of max(y, 0)            (NN_net activations, affine_coupling.py:77-78)
 * `status` (device int, may be NULL) is set to 1 if an internal barrier wait timed out (never hangs). */
enum { FLOWK_PRE_BIAS = 0, FLOWK_PRE_GLU_RES_LN = 1, FLOWK_PRE_LSTM = 2 };
enum { FLOWK_OUT_F32 = 1, FLOWK_OUT_HILO = 2, FLOWK_OUT_HILO_POS = 4, FLOWK_OUT_HILO_CELU = 8, FLOWK_OUT_NCHW = 16,
       FLOWK_OUT_HILO_RELU = 32 };

typedef struct flowk_conv_gemm_args {
  const float* a_hi;      /* activations NHWC [B,H,W,Cin] */
  const float* a_lo;
  const float* w_hi;      /* weights [N, taps*Cin], (tap, c) order along K */
  const float* w_lo;
  const float* bias;      /* [N] or NULL */
  const float* res;       /* [B*H*W, C] residual (GLU_RES_LN) */
  const float* gamma;     /* [C] LayerNorm weight */
  const float* beta;      /* [C] LayerNorm bias */
  const float* pos;       /* [H*W, C] positional encoding (OUT_HILO_POS) */
  float* out_f32;
  float* out_hi;
  float* out_lo;
  float* out_nchw;
  int* status;
  long long* trace;       /* optional device [16]: clock64 stamps of CTA (0,0) for profiling; NULL in production */
  int B, H, W, Cin, N, taps, pre, out_mask;
  /* optional chained GEMM (FLOWK_PRE_GLU_RES_LN only, N + N2 <= 512): out2_f32[m, N2] = (y [+ pos]) . W2^T with
   * W2 = [N2, N/2] as an (hi, lo) pair - GatedAttn's in_proj applied to the normalised rows inside the same CTA
   * (mixlogcdf_nn.py:130-136).  NULL / 0 disables it. */
  const float* w2_hi;
  const float* w2_lo;
  float* out2_f32;
  int N2;
  /* optional split-K workspace (FLOWK_PRE_BIAS with out_mask == FLOWK_OUT_F32 or FLOWK_OUT_NCHW only): when non-null
   * and the layer has few 128-row tiles and a long K loop, flowk_conv_gemm_splitk_slices(args) CTAs share every output
   * tile, each writing fp32 partial rows here ([slices, B*H*W, N] floats), and a second kernel adds the slices in index
   * order plus the bias into the destination.  Serves the latency of single-stream (training) steps. */
  float* splitk_ws;
  /* Operand format of a_hi/a_lo/w_hi/w_lo and of the out_hi/out_lo the epilogue writes:
   *   FLOWK_OPERAND_TF32 (0)  fp32 arrays holding TF32 values (tcgen05 kind::tf32, 32 channels per k-block); Cin % 32 == 0
   *   FLOWK_OPERAND_F16  (1)  fp16 arrays (the pointers are reinterpreted; tcgen05 kind::f16, 64 channels per k-block):
   *                           half the operand bytes, twice the MMA rate, the same 11 + 11 significant bits as the TF32
   *                           pair.  Cin % 8 == 0; the weight rows are [taps * ceil64(Cin)] with every tap zero-padded to
   *                           whole 64-channel blocks; weights may be pre-scaled by a power of two s (|w s| < 65504) with
   *                           acc_scale = 1 / s applied to the accumulator before the bias.  Inference only: values
   *                           must stay below 65504 in magnitude. */
  int operand_format;
  float acc_scale;
  /* taps = 25 selects a 5x5 kernel; `dilation` (0 or 1 = dense) spaces the taps of 3x3 / 5x5 kernels ("same" zero padding of
   * dilation * (k - 1) / 2, mar_prior/convolutional_rnn/functional.py:248-272). */
  int dilation;
  float acc_scale2;       /* FLOWK_OPERAND_F16 with a chained GEMM: 1 / (power-of-two pre-scaling of w2) */
  const float* acc_scale_ptr;   /* non-NULL: acc_scale is read from this DEVICE float when the kernel runs (weights packed on
                                 * the device in the same stream, e.g. by flowk_weight_norm_operands_batched); acc_scale is
                                 * then only checked for being positive */
} flowk_conv_gemm_args;
enum { FLOWK_OPERAND_TF32 = 0, FLOWK_OPERAND_F16 = 1 };

int flowk_conv_gemm(const flowk_conv_gemm_args* args, flowk_stream_t stream);
/* Slices flowk_conv_gemm would use for `args` if args->splitk_ws were non-null (1 = no split-K); no pointer is read. */
int flowk_conv_gemm_splitk_slices(const flowk_conv_gemm_args* args);

/* ---- one step of ancestral sampling from the mAR channel prior (mar_prior/corr_prior.py:66-101) -------------------------
 * The implicit GEMM of flowk_conv_gemm (FLOWK_OPERAND_F16 only: a_* / w_* / dst*_ are fp16 arrays, weights
 * [N, taps * ceil64(Cin)] from flowk_pack_weight_f16 with acc_scale = 1 / their pre-scaling) with one of three epilogues.
 * Every activation row is [B*H*W, Cin] NHWC; hid = the ConvLSTM width (hid % 8 == 0, 4 hid <= 256).  A destination d is
 * the fp16 pair dst<d>_hi / dst<d>_lo written at row m, columns [dst<d>_col, dst<d>_col + width) of rows dst<d>_pitch
 * elements long.  `mode` selects:
 *   FLOWK_MAR_EMBED   N = hid: y = D + bias (conv_embed on the step input [prev sample | z1 embedding | 0]), width hid, to
 *                     dst 0
 *   FLOWK_MAR_LSTM    N = 4 hid gate columns [i | f | g | o] of one ConvLSTM layer from ONE GEMM over the rows [x_t | h_{t-1}]
 *                     (Cin = 2 hid) with weights [W_ih | W_hh] per tap and bias = b_ih + b_hh (functional.py:30-52):
 *                     c [B*H*W, hid] (fp32, c_{t-1} in, c_t out, in place), h_t = sig(o) tanh(c_t), width hid, to dst 0
 *                     and, when dst1_hi is non-NULL, to dst 1
 *   FLOWK_MAR_SAMPLE  N = 2 columns (mean, log-std) of conv_out1 (weights [0 | W_out] over [x | h] rows), never stored:
 *                     s = noise[m] * exp(log-std) + mean (fp32, accurate exp) to z[b * z_stride + hw] and, width 1, to dst 0
 * A launch must not write rows it reads (neighbouring taps belong to other CTAs): callers ping-pong buffers by step parity.
 * Returns FLOWK_ERR_ARG for a pointer the mode needs that is NULL (dst 1 is optional) or a bad mode / taps / acc_scale,
 * FLOWK_ERR_SHAPE for a bad hid, Cin, destination (column + width beyond the pitch, pitch or column not a multiple of 4)
 * or z_stride < H*W, or maps that do not tile into 128-row blocks (W | 128, and H*W | 128 or 128 | H*W) - before any launch. */
enum { FLOWK_MAR_EMBED = 0, FLOWK_MAR_LSTM = 1, FLOWK_MAR_SAMPLE = 2 };
typedef struct flowk_mar_step_args {
  const void* a_hi;       /* activation pair [B*H*W, Cin] */
  const void* a_lo;
  const void* w_hi;       /* weight pair [N, taps * ceil64(Cin)] */
  const void* w_lo;
  const float* bias;      /* [N] */
  void* dst0_hi;
  void* dst0_lo;
  void* dst1_hi;          /* FLOWK_MAR_LSTM only, optional */
  void* dst1_lo;
  float* c;               /* FLOWK_MAR_LSTM: cell state [B*H*W, hid] */
  const float* noise;     /* FLOWK_MAR_SAMPLE: [B*H*W] */
  float* z;               /* FLOWK_MAR_SAMPLE: z[b * z_stride + hw] (the caller points it at the channel) */
  long long z_stride;
  int* status;            /* device int, may be NULL: set to 1 if an internal barrier wait timed out */
  int mode, B, H, W, Cin, taps, dilation, hid;   /* taps 1, 9 or 25; dilation 0 or 1 = dense */
  int dst0_pitch, dst0_col, dst1_pitch, dst1_col;
  float acc_scale;
} flowk_mar_step_args;
int flowk_mar_step(const flowk_mar_step_args* args, flowk_stream_t stream);

/* x[b, ch, p] (NCHW, `batch_stride` floats between samples, ch < C) -> NHWC hi/lo [B*HW, C_pad], zero-padded channels. */
int flowk_nchw_to_nhwc_hilo(const float* x, long long batch_stride, int B, int C, int HW, int C_pad,
                            float* hi, float* lo, flowk_stream_t stream);
/* fp32 array -> (hi, lo) operand pair. */
int flowk_split_hilo(const float* x, float* hi, float* lo, long long n, flowk_stream_t stream);
/* The same two for FLOWK_OPERAND_F16: hi / lo are fp16 arrays (C_pad % 8 == 0); split_hilo_f16 multiplies by `scale`
 * (the power-of-two weight pre-scaling) first. */
int flowk_nchw_to_nhwc_hilo_f16(const float* x, long long batch_stride, int B, int C, int HW, int C_pad,
                                void* hi, void* lo, flowk_stream_t stream);
int flowk_split_hilo_f16(const float* x, void* hi, void* lo, long long n, float scale, flowk_stream_t stream);

/* Weight preparation for FLOWK_OPERAND_F16 in two launches (csrc/weight_pack.cu), once per weight version: w [N, cin, taps]
 * (torch conv / linear layout) times a per-output-channel gain
 *   FLOWK_PACK_PLAIN        1
 *   FLOWK_PACK_WEIGHT_NORM  gain[n] / ||w[n]||      weight_g / weight_v of mixlogcdf_nn.py:19-21
 *   FLOWK_PACK_EXP_GAIN     exp(factor * gain[n])   ActNorm / Conv2dZeros scale folded into the conv (affine_coupling.py:31-63);
 *                                                   bias_out[n] = bias_in[n] * exp(factor * gain[n]) when bias_out is given
 * -> K-major fp16 (hi, lo) rows [N, taps * cin_pad] in (tap, c) order (cin_pad % 8 == 0, zero padding), pre-scaled by the power
 * of two that puts max|w| into [2^14, 2^15).  ws: N + 2 floats {row gains [N], max bits, acc_scale}; ws[N + 1] is the
 * `acc_scale` to hand to flowk_conv_gemm. */
enum { FLOWK_PACK_PLAIN = 0, FLOWK_PACK_WEIGHT_NORM = 1, FLOWK_PACK_EXP_GAIN = 2 };
int flowk_pack_weight_f16(const float* w, const float* gain, int mode, float factor, const float* bias_in, float* bias_out,
                          int N, int cin, int taps, int cin_pad, void* hi, void* lo, float* ws, flowk_stream_t stream);

/* ActNorm followed by the LU-parametrised invertible 1x1 conv (common_modules.py:57-127,130-187; a FlowStep's first two
 * layers, marscf_main.py:64-68 / :95-97) folded into one per-pixel affine map for flowk_channel_mix_*: l, u, p [C, C],
 * log_s, sign_s [C] (InvertibleConv1x1), logs, bias [C] (Actnormlayer); assembled in fp64 by one CTA.
 *   forward (reverse = 0)  mat = P (L U) diag(e^logs),  bias_out = mat bias,  ldj[0] = sum(logs) H W + sum(log_s) W^2
 *   reverse                mat = diag(e^-logs) U^-1 L^-1 P^T,  bias_out = -bias,  ldj[0] = -(...)
 * C <= 158 (the fp64 matrix lives in shared memory). */
int flowk_fold_actnorm_invconv(const float* l, const float* u, const float* log_s, const float* p, const float* sign_s,
                               const float* logs, const float* bias, int C, int H, int W, int reverse, float* mat,
                               float* bias_out, float* ldj, flowk_stream_t stream);

/* Fused pointwise layers of the Flow++ conditioner (training path), tensors viewed as [outer, channels, inner]
 * (inner = H*W for NCHW / dim 1, inner = 1 for NHWC / last dim):
 *   concat_elu: x [outer, C, inner] -> y [outer, 2C, inner] = elu(cat(x, -x))        mixlogcdf_nn.py:8-10
 *               optional mask [outer, 2C]: per-(sample, output channel) multiplier = the nn.Dropout2d that follows
 *               concat_elu in GatedConv (mixlogcdf_nn.py:251-256), folded in (0 or 1/(1-p); nullable)
 *   glu:        x [outer, 2C, inner] -> y [outer, C, inner] = x[:, :C] * sigmoid(x[:, C:])   mixlogcdf_nn.py:149-151,257-258
 * and their backward passes (gx from x and gy). */
int flowk_concat_elu_fwd(const float* x, float* y, const float* mask, long long outer, int C, long long inner,
                         flowk_stream_t stream);
int flowk_concat_elu_bwd(const float* x, const float* gy, float* gx, const float* mask, long long outer, int C,
                         long long inner, flowk_stream_t stream);
int flowk_glu_fwd(const float* x, float* y, long long outer, int C, long long inner, flowk_stream_t stream);
int flowk_glu_bwd(const float* x, const float* gy, float* gx, long long outer, int C, long long inner,
                  flowk_stream_t stream);

/* Weight normalisation w = v * g / ||v|| (norm over all dims but 0; `weight_norm(nn.Conv2d)`, mixlogcdf_nn.py:19-21)
 * fused with building the flowk_conv_gemm weight operands.  v [N, cin, taps] (torch conv / linear weight), g [N].
 * Outputs (each pair nullable): norm [N]; w [N, cin, taps] fp32; forward operand [N, taps, cin_pad] hi/lo;
 * input-gradient operand [cin, taps, n_pad] hi/lo (taps flipped, weight transposed).  Pads are zero-filled.
 * flowk_weight_norm_bwd: from gw = dL/dw returns gv [N, cols] and gg [N]. */
int flowk_weight_norm_operands(const float* v, const float* g, int N, int cin, int taps, int cin_pad, int n_pad,
                               float* norm, float* w, float* fwd_hi, float* fwd_lo, float* dg_hi, float* dg_lo,
                               flowk_stream_t stream);
/* The same for every layer of a model in two launches (a training step re-normalises ~500 tiny weight tensors and the
 * per-layer kernels are launch-bound).  `jobs_device` is a DEVICE array of njobs entries; w / fwd_* / dg_* may be null
 * per entry; max_rows = the largest N among the jobs. */
typedef struct flowk_wn_job {
  const float* v;
  const float* g;
  float* norm;
  float* w;
  float* fwd_hi;
  float* fwd_lo;
  float* dg_hi;
  float* dg_lo;
  int N, cin, taps, cin_pad, n_pad;
  int fwd_f16;   /* 1: fwd_hi / fwd_lo are fp16 arrays [N, taps * cin_pad] (FLOWK_OPERAND_F16, cin_pad = ceil64(cin)), pre-scaled
                  * by a power of two; `norm` then has N + 2 entries, norm[N] zeroed by the caller before the call (scratch:
                  * the layer's max |w|) and norm[N + 1] receiving the acc_scale (pass it as acc_scale_ptr) */
} flowk_wn_job;
int flowk_weight_norm_operands_batched(const flowk_wn_job* jobs_device, int njobs, int max_rows, flowk_stream_t stream);
int flowk_weight_norm_bwd(const float* v, const float* g, const float* norm, const float* gw, float* gv, float* gg,
                          int N, int cols, flowk_stream_t stream);

/* Standard-normal log-likelihood of every sample, added to the running objective:
 * out[b] = (in ? in[b] : 0) - (sum_i z[b, i]^2 + n log 2 pi) / 2 with z[b, i] at z + b * sample_stride + i (a channel slice of
 * an NCHW tensor is fine).  FlowNet.encode's default prior terms (GaussianDiag.logp, common_modules.py:223-240, summed into
 * the log-det at marscf_main.py:159-164), one launch per level.  in may alias out. */
int flowk_std_normal_logp(const float* z, long long sample_stride, const float* in, float* out, int B, long long n,
                          flowk_stream_t stream);

/* Residual add + LayerNorm over channels (ConvAttnBlock, mixlogcdf_nn.py:226-234): y = LN_C(a + b) * gamma + beta.
 * M = B*HW pixel rows; a, b (b nullable) are NCHW [B, C, HW] when in_nchw else rows [M, C]; y likewise by out_nchw.
 * Forward also returns s = a + b as rows [M, C] and mean / rstd [M] for the backward pass, which yields
 * gs = dL/da = dL/db (input layout) and dgamma / dbeta [C] (deterministic two-stage sum; workspace of
 * flowk_add_layernorm_workspace_bytes(M, C) bytes, caller-owned). */
long long flowk_add_layernorm_workspace_bytes(long long M, int C);
int flowk_add_layernorm_fwd(const float* a, const float* b, const float* gamma, const float* beta, float* y, float* s,
                            float* mean, float* rstd, long long M, int C, int HW, int in_nchw, int out_nchw, float eps,
                            flowk_stream_t stream);
int flowk_add_layernorm_bwd(const float* gy, const float* s, const float* mean, const float* rstd, const float* gamma,
                            float* gs, float* dgamma, float* dbeta, void* workspace, long long M, int C, int HW,
                            int in_nchw, int out_nchw, flowk_stream_t stream);

/* Bias gradient: out[c] = sum of x[o, c, i] over o < outer, i < inner (NCHW: outer = B, inner = H*W; rows: inner = 1).
 * Deterministic two-stage sum; workspace of flowk_channel_sum_workspace_bytes(C) bytes, caller-owned. */
long long flowk_channel_sum_workspace_bytes(int C);
int flowk_channel_sum(const float* x, float* out, void* workspace, long long outer, int C, long long inner,
                      flowk_stream_t stream);

/* Weight gradient of a stride-1 "same" convolution (taps = 1 or 9) / linear layer on tcgen05 (3xTF32, fp32-accurate):
 *   partial[s][t][n][c] = sum over the s-th slice of (b, pixel) of gy[b, n, p] * x[b, c, p + shift(t)]
 * x [B, Cin, H, W] and gy [B, N, H, W] are plain fp32 channel-major (NCHW) tensors (W % 4 == 0, H*W % 32 == 0); a
 * linear layer passes its transposed operands as B = 1, H = M / 32, W = 32.  For taps = 9 the caller also passes the
 * column-shifted copies of x made by flowk_shift_columns: x_left[.., w] = x[.., w-1], x_right[.., w] = x[.., w+1],
 * zero at the image border (a TMA box cannot start at an unaligned innermost coordinate).  flowk_conv_wgrad_splits returns how many split-K slices the
 * launch writes (0: shape not supported) and whether the kernel puts x on the 128-row side of the MMA, in which case
 * the slices are stored transposed, [splits, taps, Cin, N] (*transposed = 1); the caller allocates partial
 * [splits, taps, N, Cin] floats and sums the slices in index order (flowk_weight_norm_bwd_partials does, fused with the weight-norm backward).
 * status: optional device int, set to 1 if a pipeline wait timed out (protocol bug; never hangs). */
int flowk_conv_wgrad_splits(int B, int H, int W, int Cin, int N, int taps, int* transposed);
int flowk_conv_wgrad(const float* x, const float* x_left, const float* x_right, const float* gy, float* partial,
                     int* status, int B, int H, int W, int Cin, int N, int taps, flowk_stream_t stream);
/* Same for a Linear layer with ROW-major operands x [M, K], gy [M, N] (M % 32 == 0, K % 32 == 0, N % 32 == 0): the
 * contraction index is the row, so the tiles are MN-major (transposed) tf32 operands - no transposed copies needed.
 * partial [splits, N, K] (or [splits, K, N] when *transposed). */
int flowk_linear_wgrad_splits(long long M, int K, int N, int* transposed);
int flowk_linear_wgrad(const float* x, const float* gy, float* partial, int* status, long long M, int K, int N,
                       flowk_stream_t stream);
int flowk_shift_columns(const float* x, float* x_left, float* x_right, long long total, int W, flowk_stream_t stream);
/* Same for a stride-1 "same" convolution over NHWC rows x [NB*H*W, Cin], gy [NB*H*W, N] (Cin % 32 == 0, N % 32 == 0;
 * the mAR prior's time-major tensors, NB = T*B images), taps = 1, 9 or 25 at any dilation:
 *   partial[s][t][n][c] = sum over the s-th slice of (image, pixel) of gy[., n, p] * x[., c, p + (ky, kx - k/2) * dilation]
 * with out-of-image pixels zero.  No shifted copies: the tap shift is a TMA coordinate.  Shapes: W | 32 or 32 | W, and the
 * 32-pixel k-block (min(W, 32) columns x bh rows x bb images) must tile the maps (NB % bb == 0).  Replaces the weight
 * gradients of F.conv2d in the ConvLSTM prior (mar_prior/lstm.py:33-35, 73-74; corr_prior.py:26-28). */
int flowk_conv_wgrad_nhwc_splits(int NB, int H, int W, int Cin, int N, int taps, int dilation, int* transposed);
int flowk_conv_wgrad_nhwc(const float* x, const float* gy, float* partial, int* status, int NB, int H, int W, int Cin, int N,
                          int taps, int dilation, flowk_stream_t stream);
/* Backward of one ConvLSTM cell step (mar_prior/convolutional_rnn/functional.py:30-52), one thread per (row, unit):
 * gi, hh [M, 4 hid] (gate pre-activations = gi + hh, order i, f, g, o), c_prev, c [M, hid], dh [M, hid] plus the optional
 * recurrent dh_rec and dc_next (dL/dc_t from step t+1, already times f_{t+1}) -> dgates [M, 4 hid] fp32 and as the TF32
 * (hi, lo) operand pair, dc_prev = dL/dc_{t-1} (may alias dc_next). */
int flowk_lstm_cell_bwd(const float* gi, const float* hh, const float* c_prev, const float* c, const float* dh,
                        const float* dh_rec, const float* dc_next, float* dgates, float* dg_hi, float* dg_lo, float* dc_prev,
                        long long M, int hid, flowk_stream_t stream);
/* fp16 (hi, lo) operand rows [M, C] -> fp32 rows out [M, C_out] = hi + lo, columns >= C zero (C_out >= C). */
int flowk_f16_pair_to_f32(const void* hi, const void* lo, float* out, long long M, int C, int C_out, flowk_stream_t stream);
int flowk_weight_norm_bwd_partials(const float* v, const float* g, const float* norm, const float* partial, float* gv,
                                   float* gg, int N, int cin, int taps, int splits, int transposed,
                                   flowk_stream_t stream);

/* Training-time attention core with attention-weight dropout (mixlogcdf_nn.py:134-147 with :143's F.dropout): forward and
 * backward.  qkv / dqkv rows [B*HW, 3C] in (k | v | q) order; out / dout rows [B*HW, C]; lse [B*heads, HW] (row
 * log-sum-exp, written by the forward).  The backward is two independent kernels selected by `which`: 1 = query side
 * (writes the q columns of dqkv), 2 = key side (k and v columns), 3 = both; 1 and 2 may run on different streams.  The dropout mask is a counter-based hash of
 * (*seed_device, salt, image*head, query, key): the backward regenerates it, nothing of size HW x HW touches HBM.
 * seed_device: device scalar the caller advances once per training step (so a captured graph draws fresh masks on each
 * replay); salt: per-layer constant.  HW % 8 == 0, C / heads in {8, 16, 24, 32, 40, 64}, B*heads*HW*HW < 2^32.
 * flowk_attention_dropout_mask materialises the multipliers (0 or 1/(1-p)) [B*heads, HW, HW] - for tests. */
int flowk_attention_train_fwd(const float* qkv, float* out, float* lse, const unsigned* seed_device, unsigned salt,
                              float p_drop, int B, int HW, int C, int heads, flowk_stream_t stream);
int flowk_attention_train_bwd(int which, const float* qkv, const float* out, const float* dout, const float* lse,
                              float* dqkv, const unsigned* seed_device, unsigned salt, float p_drop, int B, int HW, int C,
                              int heads, flowk_stream_t stream);
int flowk_attention_dropout_mask(const unsigned* seed_device, unsigned salt, float p_drop, int pairs, int HW, float* mask,
                                 flowk_stream_t stream);

/* The same training attention core (reference flow_modules/mixlogcdf_nn.py:139-147: q k^T / sqrt(d), softmax, dropout,
 * weight v) on tcgen05 (csrc/attention_train_tc.cu) for head dim C / heads == 64 and HW in {128, 256}: kind::tf32 MMAs on
 * (hi, lo) operand pairs (fp32 accuracy), TMEM accumulators, the dropout mask of flowk_attention_dropout_mask.  Same
 * arguments, layouts, lse and `which` as flowk_attention_train_fwd / _bwd; the two backward kernels use no atomics, so
 * results are bit-identical from call to call.  FLOWK_ERR_ARG on a NULL pointer or `which` outside 1..3; FLOWK_ERR_SHAPE
 * for C / heads != 64, HW not in {128, 256}, p_drop outside [0, 1) or B*heads*HW*HW >= 2^32 - 1. */
int flowk_attention_train_tc_fwd(const float* qkv, float* out, float* lse, const unsigned* seed_device, unsigned salt,
                                 float p_drop, int B, int HW, int C, int heads, flowk_stream_t stream);
int flowk_attention_train_tc_bwd(int which, const float* qkv, const float* out, const float* dout, const float* lse,
                                 float* dqkv, const unsigned* seed_device, unsigned salt, float p_drop, int B, int HW, int C,
                                 int heads, flowk_stream_t stream);

/* Adamax step (torch.optim.Adamax semantics, weight_decay = 0; the reference's optimizer, marscf_main.py:302) over every
 * parameter tensor of a model in one launch / one HBM pass.  `chunks_device`: DEVICE array, each tensor cut into pieces
 * (the caller chooses the size, e.g. 16 Ki elements), one CTA per piece; p, m (exp_avg), u (exp_inf) are updated in
 * place from g.  clr_device: device scalar lr / (1 - beta1^step), refreshed by the host before every (graph) launch. */
typedef struct flowk_adamax_chunk {
  float* p;
  const float* g;
  float* m;
  float* u;
  long long n;
} flowk_adamax_chunk;
int flowk_adamax_step(const flowk_adamax_chunk* chunks_device, int nchunks, const float* clr_device, float beta1,
                      float beta2, float eps, flowk_stream_t stream);

/* Self-attention core of GatedAttn (mixlogcdf_nn.py:134-147,154-173), inference: qkv = in_proj rows [B*HW, 3C] in the
 * reference's (k | v | q) column order; out_hi/out_lo [B*HW, C] = softmax(q k^T / sqrt(C/heads)) v as an operand pair.
 * C/heads in {8,16,24,32,40,64}; HW <= 256 or a multiple of 256. */
int flowk_attention(const float* qkv, float* out_hi, float* out_lo, int B, int HW, int C, int heads,
                    flowk_stream_t stream);
/* Same, writing the operand pair as fp16 arrays (FLOWK_OPERAND_F16 input of the gate GEMM). */
int flowk_attention_f16(const float* qkv, void* out_hi, void* out_lo, int B, int HW, int C, int heads,
                        flowk_stream_t stream);

/* `Transformer_attn`, the fork's invertible patch attention (reference flow_modules/transformer.py:123-326; two per FlowStep,
 * marscf_main.py:50-51,69-70), inference / sampling, one pass: x, y [B, C, H, W] fp32 (H == W even); G [C, C] =
 * sum_i Wq_i^T Wk_i; prm = device {offset, offset2, offset3, scale}; ldj_in / ldj_out [B] (NULL allowed).  Forward mixes
 * the free entries of patches (0, 2) / (1, 3) with the 2x2 attention matrices and adds (log|det M1| + log|det M2|) p (p/2) C
 * to ldj; reverse applies the closed-form inverses and subtracts. */
int flowk_patch_attention(const float* x, const float* G, const float* prm, float* y, const float* ldj_in, float* ldj_out,
                          int B, int C, int H, int W, int permute, int reverse, flowk_stream_t stream);

/* `Transformer_attn` training (reference flow_modules/transformer.py:123-326 and its autograd), forward direction only.
 * flowk_patch_attention_train_fwd is flowk_patch_attention with reverse = 0 (the same y and ldj_out, bit for bit) that also
 * writes the raw scores [B, 8] = S_0 (row-major 2x2, patches (0, 2)), S_1 (patches (1, 3)); scores must not be NULL.
 * flowk_patch_attention_bwd takes x, G, prm and those scores with gy [B, C, H, W] and gldj [B] (the gradient of ldj_out,
 * which is also that of ldj_in) and writes gx [B, C, H, W] and partials [B, C*C + 4]: per sample the gradient of G
 * (row-major) and of offset, offset2, offset3, scale; their batch sums (flowk_channel_sum over rows) are the parameter
 * gradients.  Needs (3 C H W + C^2) * 4 <= 200 KB of shared memory; FLOWK_ERR_SHAPE otherwise.  No host synchronisation
 * and no allocation (graph-capturable); every sum has a fixed order, so repeated calls are bit-identical. */
int flowk_patch_attention_train_fwd(const float* x, const float* G, const float* prm, float* y, const float* ldj_in,
                                    float* ldj_out, float* scores, int B, int C, int H, int W, int permute,
                                    flowk_stream_t stream);
int flowk_patch_attention_bwd(const float* x, const float* G, const float* prm, const float* scores, const float* gy,
                              const float* gldj, float* gx, float* partials, int B, int C, int H, int W, int permute,
                              flowk_stream_t stream);

/* The same attention core on tcgen05 (csrc/attention_tc.cu): S = Q K^T and O = P V as kind::f16 MMAs with TMEM accumulators,
 * fp16 (hi, lo) operand tiles built in shared memory, softmax between them; out_f16 selects fp16 or TF32-in-fp32 output
 * pairs.  Takes HW in {128, 256} with C/heads a multiple of 8 and <= 64; FLOWK_ERR_SHAPE otherwise (use flowk_attention).
 * `status` (device int, may be NULL) is set to 1 if an internal barrier wait timed out; `trace` (device long long[8], NULL in
 * production) receives clock64 stamps of the first CTA's phases. */
int flowk_attention_tc(const float* qkv, void* out_hi, void* out_lo, int out_f16, int B, int HW, int C, int heads,
                       int* status, long long* trace, flowk_stream_t stream);
/* The one-wave variant (csrc/attention_tc.cu, attention_tc_v2_kernel): 256 TMEM columns and < 110 KB of shared memory per
 * CTA, so two CTAs share an SM; keys in blocks of 128 with per-block softmax statistics combined exactly in the epilogue,
 * P kept in tensor memory.  Same arguments, outputs and trace slots as flowk_attention_tc; takes HW in {128, 256} with
 * C/heads in {24, 32}, FLOWK_ERR_SHAPE otherwise.
 * flowk_attention_tc_v2_occupancy reports how many of its CTAs one SM's registers, shared memory and thread slots hold at a
 * shape and, if smem_bytes is not NULL, the dynamic shared memory per CTA (the runtime's occupancy calculator answers 1 for
 * any kernel that uses tcgen05 instructions). */
int flowk_attention_tc_v2(const float* qkv, void* out_hi, void* out_lo, int out_f16, int B, int HW, int C, int heads,
                          int* status, long long* trace, flowk_stream_t stream);
int flowk_attention_tc_v2_occupancy(int HW, int C, int heads, int* blocks_per_sm, int* smem_bytes);
/* The tcgen05 attention core for long sequences (csrc/attention_long_tc.cu): one CTA per (image, head, 128-query tile), keys
 * streamed through shared memory in 128-key blocks, per-block softmax folded into a running output (online softmax), P kept
 * in tensor memory; nothing of size HW x HW leaves the SM.  Same arguments and outputs as flowk_attention_tc.  Takes HW a
 * multiple of 128 with HW >= 512 and C/heads in {24, 32, 40, 64}, any B >= 0 (B = 0: FLOWK_OK, no launch);
 * FLOWK_ERR_SHAPE otherwise, FLOWK_ERR_ARG for a NULL qkv / out_hi / out_lo.  `status` as for flowk_attention_tc;
 * `trace` (device long long[3], NULL in production): clock64 stamps of CTA 0 at start, after the key loop and at the end.
 * Deterministic: no atomics, key blocks folded in order. */
int flowk_attention_long_tc(const float* qkv, void* out_hi, void* out_lo, int out_f16, int B, int HW, int C, int heads,
                            int* status, long long* trace, flowk_stream_t stream);
/* The one-wave kernel with the in_proj GEMM fused in front: instead of the fp32 in_proj rows it takes the rows that GEMM
 * would multiply, p_hi / p_lo [B*HW, C] fp16 (the normalised rows + positional encoding, as flowk_conv_gemm's
 * OUT_HILO_POS writes them), and the in_proj weight operand w_hi / w_lo [3C, ceil64(C)] fp16 with (k | v | q) rows as
 * flowk_pack_weight_f16 packs a 1x1 weight, whose pre-scaling acc_scale undoes.  q, k and v are computed per (image, head)
 * on the tensor cores and never leave the SM.  Output: fp16 (hi, lo) pairs [B*HW, C].  Same shapes as flowk_attention_tc_v2
 * (FLOWK_ERR_SHAPE otherwise); FLOWK_ERR_ALIGN unless the four inputs are 16-byte aligned.  `trace` slots: 0 start,
 * 1 projection done, 2..7 as slots 1..6 of flowk_attention_tc.  flowk_attention_inproj_tc_occupancy: as
 * flowk_attention_tc_v2_occupancy, for this kernel. */
int flowk_attention_inproj_tc(const void* p_hi, const void* p_lo, const void* w_hi, const void* w_lo, float acc_scale,
                              void* out_hi, void* out_lo, int B, int HW, int C, int heads, int* status, long long* trace,
                              flowk_stream_t stream);
int flowk_attention_inproj_tc_occupancy(int HW, int C, int heads, int* blocks_per_sm, int* smem_bytes);
/* The attention half of a ConvAttnBlock in one launch (csrc/block_tail_tc.cu), for feature maps whose images fit whole into
 * a 128-row tile: gate GEMM -> GLU + bias + x -> LayerNorm(gamma1, beta1) = x1; in_proj of x1 + pos; softmax attention per
 * image and head; attention-gate GEMM -> GLU + bias + x1 -> LayerNorm(gamma2, beta2) = x2.  x1, q, k, v and the attention
 * output never leave the SM.  Inputs: c1_hi / c1_lo [B*HW, 2C] fp16 (the concat-ELU rows the gate multiplies), the fp16
 * weight operands as flowk_pack_weight_f16 packs 1x1 weights (gate [2C, ceil64(2C)], in_proj [3C, ceil64(C)] with
 * (k | v | q) rows, attention gate [2C, ceil64(C)]) with their acc_scale factors, fp32 biases [2C], x [B*HW, C],
 * LayerNorm parameters [C] and the positional encoding pos [HW, C].  Outputs: x2 [B*HW, C] fp32 and out_hi / out_lo fp16,
 * [B*HW, 2C] concat_elu(x2) when celu != 0, else [B*HW, C] x2.  Takes HW <= 128 with 128 % HW == 0, B*HW % 128 == 0,
 * C a multiple of 32 with 5C <= 512 and C/heads in {24, 32}; FLOWK_ERR_SHAPE otherwise, FLOWK_ERR_ARG for a NULL input or
 * output or a non-positive scale, FLOWK_ERR_ALIGN unless every pointer is 16-byte aligned.  `status` (device int, may be
 * NULL) is set to 1 if an internal barrier wait timed out; `trace` (device long long[8], NULL in production) receives
 * clock64 stamps of the first CTA: 0 start, 1 gate accumulator, 2 in_proj operand written, 3 in_proj accumulator, 4 first
 * head's S, 5 attention done, 6 attention-gate accumulator, 7 end. */
int flowk_block_tail_tc(const void* c1_hi, const void* c1_lo, const void* wg_hi, const void* wg_lo, float sc_g,
                        const float* bias_g, const float* x, const float* gamma1, const float* beta1, const float* pos,
                        const void* wi_hi, const void* wi_lo, float sc_i, const void* wa_hi, const void* wa_lo, float sc_a,
                        const float* bias_a, const float* gamma2, const float* beta2, float* x2, void* out_hi,
                        void* out_lo, int celu, int B, int HW, int C, int heads, int* status, long long* trace,
                        flowk_stream_t stream);
/* The same block tail for 16x16 maps (HW = 256), where an image spans two 128-row tiles: one cluster of two CTAs per image,
 * each CTA owning 128 of its rows, exchanging each head's K and V through distributed shared memory so that every row
 * attends over all 256 keys of its image.  Same arguments, outputs, status and error codes as flowk_block_tail_tc; takes
 * HW = 256, any B >= 0 (B = 0 returns FLOWK_OK), C a multiple of 32 with 5C <= 512 and C/heads in {24, 32}; FLOWK_ERR_SHAPE
 * otherwise.  `trace` (device long long[8], NULL in production) receives clock64 stamps of the first CTA (rank 0 of image
 * 0): 0 start, 1 gate accumulator, 2 in_proj operand written, 3 in_proj accumulator, 4 first head's S over its own keys,
 * 5 attention done, 6 attention-gate accumulator, 7 end (after the cluster's closing barrier). */
int flowk_block_tail_pair_tc(const void* c1_hi, const void* c1_lo, const void* wg_hi, const void* wg_lo, float sc_g,
                             const float* bias_g, const float* x, const float* gamma1, const float* beta1, const float* pos,
                             const void* wi_hi, const void* wi_lo, float sc_i, const void* wa_hi, const void* wa_lo,
                             float sc_a, const float* bias_a, const float* gamma2, const float* beta2, float* x2,
                             void* out_hi, void* out_lo, int celu, int B, int HW, int C, int heads, int* status,
                             long long* trace, flowk_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif  /* FLOWK_H_ */
