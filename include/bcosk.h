/* bcosk.h -- C ABI of libbcosk.so: hand-written sm_100a kernels for the B-cos forward pass and its
 * dynamic-linear explanation (explain-dgrad) pass.
 *
 * The reference (shrebox/B-cosification) is pure Python on ATen: it has no FFI of its own.  The
 * boundary a maintainer binds is therefore the arithmetic behind its torch modules; each entry
 * point below names the reference code it replaces (paths relative to the reference root).
 * INTEGRATION.md shows the ctypes stub that binds these symbols inside `bcos.modules`.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless stated; the caller owns all buffers; nothing here
 *     allocates or synchronises; all work is enqueued on `stream` (a cudaStream_t passed as void*).
 *   - activations are NHWC ("channels_last"), 16-bit (bf16 or fp16).  A tensor may carry P precision
 *     planes concatenated along the channel axis ([hi | lo | lo2], value = sum of planes); P=1 is
 *     the plain 16-bit throughput mode, P=2/3 is the parity mode (~16/24 mantissa bits).
 *   - return value: 0 ok, -1 bad argument, -2 unsupported shape / device, -3 CUDA error
 *     (text via bcosk_last_error()).
 */
#ifndef BCOSK_H_
#define BCOSK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BCOSK_OK 0
#define BCOSK_EINVAL (-1)
#define BCOSK_EUNSUPPORTED (-2)
#define BCOSK_ECUDA (-3)

#define BCOSK_DTYPE_F16 0
#define BCOSK_DTYPE_BF16 1

#define BCOSK_MAX_TAPS 64
#define BCOSK_MAX_SEGS 6

/* epilogue modes of the implicit GEMM */
#define BCOSK_MODE_FWD 0     /* B-cos forward epilogue */
#define BCOSK_MODE_EXPLAIN 1 /* explanation-dgrad epilogue */

/* scale modes (forward) */
#define BCOSK_SCALE_NONE 0 /* plain linear map (B = 1, or nn.Linear / nn.Conv2d) */
#define BCOSK_SCALE_B2 1   /* |lin| / ||patch||                       (bcosconv2d.py:186-187) */
#define BCOSK_SCALE_POW 2  /* (|lin / ||patch||| + 1e-6)^(B-1)         (bcosconv2d.py:189-190) */

/* One implicit-GEMM launch:   D[m, n] = sum_k A[m, k] * B[n, k]
 *   m = output pixel (image, p, q) of an NHWC tensor gathered by TMA im2col, k = (segment, tap, channel).
 * Forward  (replaces BcosConv2d.forward_impl bcos/modules/bcosconv2d.py:153-194, BcosifyConv2d.forward_impl
 *           bcosifyconv2d.py:50-102, BcosLinear.forward bcoslinear.py:88-130, BcosifyLinear.forward
 *           bcosifylinear.py:42-95 and, fused into the epilogue, batch_norm_uncentered_2d (eval)
 *           batchnorm_uncentered.py:49-58, the block's residual add and nn.ReLU):
 *     s    = scale(D, inv_norm[m]);  t = s * alpha[n];  v = D * t + beta[n] + res[m, n]
 *     y    = relu ? max(v, 0) : v;   gain = (relu && v <= 0) ? 0 : t;   mask bit = (v > 0)
 *     sq_out[tile_n][m] = sum_n y^2   (feeds the next layer's patch norm)
 * Explain  (replaces autograd's MulBackward * detached scale -> ConvolutionBackward(dgrad) reached from
 *           BcosUtilMixin.explain bcos/common.py:163-181):
 *     tot  = D + add[m', n];   y = tot * mul1[m, n];   out2 = tot * mul2[m, n] * mask2 bit
 */
typedef struct bcosk_igemm_params {
  /* ---- A operand: activations / output-gradients, NHWC 16-bit, total channels a_c per pixel */
  const void* a;
  int32_t a_nb, a_h, a_w, a_c;
  int32_t lo_w, lo_h;         /* im2col lower corner: -pad (fprop) or pad-(k-1) (dgrad) */
  int32_t up_w, up_h;         /* im2col upper corner: pad-(k-1)*dil (fprop) */
  int32_t stride_w, stride_h; /* traversal stride */
  int32_t op, oq;             /* output spatial extent; M = a_nb * op * oq */
  /* ---- K loop: chunk i = ((seg * num_taps) + tap) * chunks_per_tap + kc, B column = i * kch */
  int32_t kch;                /* channels per chunk: 64 (128B swizzle) or 32 (64B swizzle) */
  int32_t chunks_per_tap;
  int32_t num_taps;
  int32_t num_segs;
  int32_t seg_a_choff[BCOSK_MAX_SEGS]; /* first channel of the A plane used by segment s */
  int32_t seg_b_plane[BCOSK_MAX_SEGS]; /* precision plane of B that segment s multiplies with (informational: the B columns of
                                        * segment s already hold that plane).  With hp_accum, the canonical two-plane order
                                        * {a0 b0, a0 b1, a1 b0} lets the kernel fetch a0 once for two segments. */
  uint16_t tap_off_w[BCOSK_MAX_TAPS];
  uint16_t tap_off_h[BCOSK_MAX_TAPS];
  /* ---- B operand: packed weights [n][num_segs*num_taps*chunks_per_tap*kch], 16-bit, K-major */
  const void* b;
  int32_t n;
  int32_t dtype;   /* BCOSK_DTYPE_* of a, b, and all 16-bit epilogue tensors */
  int32_t block_n; /* CTA tile N: 32, 64, 128; 0 = choose */
  int32_t mode;    /* BCOSK_MODE_* */
  /* ---- forward epilogue */
  int32_t scale_mode; /* BCOSK_SCALE_* */
  float b_exp;        /* B (used by BCOSK_SCALE_POW) */
  int32_t relu;
  const float* inv_norm; /* [M] 1/||patch||; NULL = compute from sq_in (or scale_mode == NONE) */
  /* patch norm from the producer's per-pixel sums of squares (calc_patch_norms bcosconv2d.py:196-231):
   * 1/(sqrt(sumpool_{sq_k,sq_stride,sq_pad} sum_parts sq_in + sq_eps_in) + sq_eps_out), sq_in = [sq_parts][a_nb*sq_h*sq_w] */
  const float* sq_in;
  int32_t sq_parts, sq_h, sq_w, sq_k, sq_stride, sq_pad;
  float sq_eps_in, sq_eps_out;
  const float* alpha;    /* [n] per-channel multiplier (BN weight/sqrt(var+eps)), NULL = 1 */
  const float* beta;     /* [n] per-channel bias, NULL = 0 */
  const float* lin_bias; /* [n] bias of the linear map itself (added BEFORE the scale: nn.Conv2d/nn.Linear bias of the
                          * Bcosify modules, bcosifyconv2d.py:68), NULL = none */
  const void* res;       /* [M, res_ld] residual (16-bit planes), NULL = none */
  int32_t res_ld, res_planes, res_plane_stride;
  void* gain;            /* [M, gain_ld] d y / d lin under the detached scale; NULL = not saved */
  int32_t gain_ld, gain_f32;
  uint32_t* maskbits;    /* [M, mask_ld] ReLU mask, bit (n % 32) of word n / 32; NULL = not saved */
  int32_t mask_ld;
  float* sq_out;         /* [ceil(n / block_n)][M] partial sum_n y^2; NULL = not produced */
  /* ---- primary output (forward: y, explain: y = tot * mul1); row m=(img,p,q) is written at
   *      row  os_0 + img*os_n + p*os_p + q*os_q  (dense: os_n = op*oq, os_p = oq, os_q = 1) */
  void* y;
  int32_t y_ld, y_planes, y_plane_stride, y_f32;
  int64_t os_0, os_n, os_p, os_q;
  /* ---- explain epilogue */
  const void* add;       /* extra gradient contribution (16-bit planes), spatially sub-sampled by add_stride */
  int32_t add_ld, add_planes, add_plane_stride, add_stride, add_p, add_q;
  const void* mul1;      /* [M, mul1_ld] gain of the producer layer, NULL = 1 */
  int32_t mul1_ld, mul1_f32;
  void* out2;            /* second output [M, out2_ld] = tot * mul2 * mask2 bit (each optional), NULL = none */
  int32_t out2_ld, out2_planes, out2_plane_stride;
  const void* mul2;
  int32_t mul2_ld, mul2_f32;
  const uint32_t* mask2;
  int32_t mask2_ld;
  /* ---- accumulation: 0 = one fp32 TMEM accumulator over all of K (throughput mode); 1 = a fresh TMEM accumulator
   *      per 64-deep K stage, summed in registers with round-to-nearest fp32 adds (parity mode: 64-wide tiles, or 128-wide
   *      for forward launches with block_n = 128).
   *      The tensor core truncates when aligning addends to a large running sum (measured: relative error ~K*2^-26,
   *      biased), which random-init deep B-cos nets amplify 10^2-10^3 x. */
  int32_t hp_accum;
  /* hp_accum only: K stages (64 deep each) of the leading operand segment (a-plane 0 x b-plane 0) that one TMEM
   *      accumulation covers before the epilogue warps add it to their registers; 0 = library default
   *      (bcosk_set_hp_chunk, initially 2).  With fp16 planes the cross-term segments (a0 b1, a1 b0; each 2^-11 of the leading one) run back
   *      to back in ONE further accumulation; with bf16 planes they are chunked like the leading segment. */
  int32_t hp_chunk;
  /* ---- schedule of a block_n == 64 launch (ignored otherwise; results do not depend on it):
   *      0 and 1 = one CTA per tile (the variant follows bcosk_set_light), 2 = persistent CTAs, tiles strided over the
   *      grid, 3 = persistent CTAs, each walks all n tiles of one 128-row block back to back (the segments of an output
   *      row reach L2 together).  The host plan measures the
   *      three per launch once (engine/base.py PlanBase.autotune) - which wins depends on N/K and the epilogue streams.
   *      With hp_accum (forward launches only): 3 = three CTAs per SM (6 warps, 128 TMEM columns: one partial accumulator
   *      of the leading segment, drained before the next chunk starts; one paired stage as the ring) where the packed
   *      two-plane epilogue applies and its boxes fit that stage, else the same as 0; 4 = four CTAs per SM (the same kernel in
   *      <= 56 KB of shared memory: launches whose leading segment is ONE accumulation, K stages <= hp_chunk, with 16-bit gains),
   *      else the same as 3; any other value = two CTAs per SM (10 warps, two ping-pong partial accumulators).  All give
   *      bit-identical y planes, gains, mask bits and sums of squares; the plan measures them per launch. */
  int32_t sched;
  /* ---- flat-window gather (a_flat = 1): `a` points at pixel (0,0) of a [a_nb, a_h, a_w, a_c] VIEW into a larger
   *      zero-bordered buffer whose rows are a_wp pixels and whose images are a_hp rows apart (borders at least as wide
   *      as the padding, never written).  For stride-1 convolutions the rows of every tap are then one contiguous run of
   *      the flattened buffer, so a CTA fetches ONE window of 128 + max tap offset pixels per tile (tiled TMA) and feeds
   *      every tap's MMA from shifted shared-memory descriptors, instead of one im2col box per tap (k*k x less L2->SM
   *      traffic; the 7x7 stem and its data gradient were bound by it).  Tiles walk the flattened positions p*a_wp + x
   *      of one image; positions with x >= oq are computed and dropped.  Requires stride 1, num_segs 1,
   *      chunks_per_tap 1, n <= 64.  a_flat_rows = pixels from the window origin (a + (lo_h*a_wp + lo_w) pixels) to
   *      the end of the buffer.  Results are identical to the im2col gather.
   *      a_flat = 2: `a` is an ordinary dense [a_nb, a_h, a_w, a_c] tensor and the zero borders exist only in shared
   *      memory: each tile fetches its image rows with ONE 4-D tiled TMA box that starts at pixel lo_w (negative) and is
   *      (a_w + kw - 1 rounded up to 8) pixels wide, so the out-of-range pixels arrive as zeros (a_wp/a_hp/a_flat_rows
   *      unused). */
  int32_t a_flat, a_wp, a_hp;
  int64_t a_flat_rows;
  /* ---- explain mode: 1 = mul1 / mul2 / out2 / mask2 are addressed by the MAPPED output row
   *      (os_0 + img*os_n + p*os_p + q*os_q) like y, not by the launch's dense row.  Used by the parity-class launches
   *      of a strided k x k data gradient: class (py, px) computes the input pixels (s*i + py, s*j + px) from the taps
   *      that reach them, so the s*s launches together do k*k/(s*s) taps per pixel instead of k*k over a zero-inserted
   *      gradient.  `add` is not supported together with it. */
  int32_t side_mapped;
  /* ---- gains that are not stored.  For a B-cos conv followed by ReLU with no residual and the BN multiplier folded into
   *      the weights, y = lin |lin| / n (clamped at 0), so the gain the explanation pass needs, |lin| / n, equals
   *      sqrt(y / n): it is recomputed from the activation the next layer keeps anyway instead of being written (-1.7 GB
   *      of writes per RN50 step).  Forward: inv_norm_out [M] (optional) receives the 1/||patch|| the launch used.
   *      Explain: mul1_sqrt_scale [M] non-NULL means `mul1` holds that ReLU output y and the multiplier is
   *      sqrt(mul1 * mul1_sqrt_scale[row]).  Both are addressed like mul1 (dense row, or mapped row with side_mapped). */
  float* inv_norm_out;
  const float* mul1_sqrt_scale;
  /* ---- MaxOut in the forward epilogue (BcosConv2d.forward_impl bcosconv2d.py:166-170, BcosLinear.forward
   *      bcoslinear.py:107-110).  max_out = G > 1: the n GEMM columns are n/G groups of G ADJACENT units (unit c = o*G + k,
   *      the reference's unflatten(dim=1, (O, G))).  The epilogue keeps the largest unit of every group (the first one on
   *      ties, like torch.max), computes the B-cos scale from the kept unit and writes n/G columns per row: y (fp32 or
   *      precision planes, row pitch y_ld), gain (the scale of the kept unit, row pitch gain_ld), amax (optional, uint8
   *      [M][amax_ld]: k of the kept unit - the only unit the explanation gradient reaches), sq_out (sum of the kept
   *      outputs squared).  G in {2, 4, 8}, n % G == 0; not combined with alpha / beta / res / relu / maskbits / a_flat.
   *      0 and 1 both mean "no MaxOut". */
  uint8_t* amax;
  int32_t max_out, amax_ld;
  /* ---- activation fused behind the B-cos transform (forward launches of the one-plane 16-bit path only).
   *      act = 1: MyGELU of the ViT MLP (bcos/models/vit.py:89-113: x * Phi(x), the gate Phi(x) = (1 + erf(x / sqrt 2)) / 2
   *      detached in explanation mode): y <- y * Phi(y) and gain <- gain * Phi(y) before rounding, so y is the activation the next
   *      linear map reads (sq_out: its sums of squares) and gain is d y / d lin under the detached scale and gate.
   *      act = 2: QuickGELU of the CLIP ViT MLP (CLIP/clip/model.py:166-168: x * sigmoid(1.702 x), an ordinary torch op that is NOT
   *      detached in the explanation pass): y <- y * s, gain <- gain * (s + 1.702 y s (1 - s)), s = sigmoid(1.702 y).
   *      Not combined with relu / maskbits / max_out / lin_bias / fp32 or multi-plane outputs / hp_accum.  0 = none. */
  int32_t act, act_reserved;
} bcosk_igemm_params;

int bcosk_igemm(const bcosk_igemm_params* p, void* stream);

/* Parity-mode (hp_accum) launches: default for bcosk_igemm_params.hp_chunk == 0 (>= 1).  Returns the previous setting. */
int bcosk_set_hp_chunk(int32_t stages);
/* Parity-mode launches, A/B measurement switches.  Bit 0 (default 1): epilogue tensors move as TMA
 * boxes through shared memory instead of per-row 16-byte accesses.  Bit 1 (default 0): the generic epilogue arithmetic runs
 * even where the packed two-plane form applies.  Bit 2 (default 0): no paired stages (every segment fetches its own A plane).
 * Bits 8..: when non-zero, 1 + the number of K stages up to which the input
 * boxes are fetched at kernel start (default 4) instead of after the last MMA.  Returns the previous setting in the same
 * encoding (passing it back restores it).  Bits 0, 1 and 8.. leave y planes, gains and mask bits bit-identical (sums of squares
 * are regrouped).  Bit 2 is not bit-identical: unpaired stages accumulate the cross terms in another order (a0 b1 over all of K,
 * then a1 b0, instead of both per stage; with bf16 planes also in chunks), which moves the last bit of fp32 within the same error
 * bound (tests/test_contract_gemm_fp64_gpu.py). */
int bcosk_set_hp_boxes(int32_t enabled);
/* Parity-mode launch configuration, without launching: info[0] = CTAs per SM the chosen kernel is built for (2, 3 or 4 for
 * 64-wide tiles, see `sched`; 1 for 128-wide), info[1] = threads per CTA, info[2] = dynamic shared memory bytes,
 * info[3] = CTAs per SM cudaOccupancyMaxActiveBlocksPerMultiprocessor reports for that kernel at that size (measured on a
 * B200 with CUDA 12.9: 1 for every instance of this kernel, also at 0 bytes, though registers, threads and shared memory admit
 * 2, 3 or 4), info[4] = registers per thread, info[5] = local memory bytes per thread (spills).  Needs a current device. */
int bcosk_igemm_hp_config(const bcosk_igemm_params* p, int32_t* info);

/* 128-wide launches whose K loop has at least `min_k_stages` 64-deep stages fetch their epilogue input tile (residual /
 * producer gain) after the main loop instead of parking it in a ring slot, so the MMAs run on 3 stages instead of 2
 * (0 = never).  Returns the previous setting.  Results are identical. */
int bcosk_set_late_input(int32_t min_k_stages);

/* Bit 0: launches with block_n 64 and a K loop of <= 4 stages use the 3-CTA-per-SM variant.  Bit 1: forward launches with
 * a single K stage use the 4-CTA-per-SM variant (the gain tile is staged over the consumed residual tile).  Default 3.
 * Returns the previous setting.  Results are identical. */
int bcosk_set_light(int32_t enabled);

/* Debug aid: raw bytes of the first A chunk (tile_m, chunk) as TMA im2col lands it in shared memory
 * (128 rows x kch 16-bit values, de-swizzled) -> out[128*kch]. */
int bcosk_debug_a_tile(const bcosk_igemm_params* p, int32_t tile_m, int32_t chunk, void* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fine-tuning step (SURVEY 8f row 2, BASELINE config 5): reference bcos/training/trainer.py:666-784 (training_step:
 * forward in train mode, loss, autograd backward), bcos/training/agc.py:28-42, bcos/modules/losses.py:99-139,
 * batchnorm_uncentered.py:36-43 (batch statistics).  The gradient all-reduce is NCCL (torch.distributed) on the host side.
 * ------------------------------------------------------------------------------------------- */

/* Weight gradient of a convolution / linear map (autograd's ConvolutionBackward grad_weight):
 *   dw[o, (tap, c)] += sum_m g[m, o] * x_patch[m, (tap, c)],  m = output pixel of the forward launch, x_patch gathered by the
 * forward launch's own TMA im2col traversal (same lo / up / stride / taps).  tcgen05 implicit GEMM over MN-major operands
 * (the NHWC boxes are used as they land), split-K over the pixels with 16-byte vector reductions into dw.
 * dw is fp32 in the packed operand layout of the forward launch, [n][num_taps * chunks_per_tap * kch]; the caller zeroes it. */
typedef struct bcosk_wgrad_params {
  const void* x;              /* forward input, NHWC 16-bit */
  int32_t a_nb, a_h, a_w, a_c;
  int32_t lo_w, lo_h, up_w, up_h, stride_w, stride_h, op, oq;
  int32_t kch, chunks_per_tap, num_taps;
  uint16_t tap_off_w[BCOSK_MAX_TAPS];
  uint16_t tap_off_h[BCOSK_MAX_TAPS];
  const void* g;              /* gradient wrt the linear output, [M, g_ld] 16-bit, dense rows */
  int32_t n, g_ld;
  float* dw;
  int32_t dtype;
  int32_t split_k;            /* CTAs along the pixel axis; 0 = choose (~4 waves) */
} bcosk_wgrad_params;
int bcosk_wgrad(const bcosk_wgrad_params* p, void* stream);
int bcosk_sizeof_wgrad_params(void);

/* Uncentred batch norm with batch statistics on NHWC 16-bit rows (batchnorm_uncentered.py:36-43):
 * stats: block b of the nblk launched writes partials[b][0..c) = sum of x, partials[b][c..2c) = sum of x^2 over its rows
 *        (no atomics: the statistics are bit-reproducible; partials is [nblk][2c] fp32, nblk ~ 2 x SM count);
 * finalize: sums the partials in a fixed order (fp64); mean, rstd = 1/sqrt(E[x^2] - E[x]^2 + eps), alpha = weight * rstd, running_var EMA with the biased variance;
 * apply: y = relu?(x * alpha[c] + res), sq[row] = sum_c y^2 (feeds the next layer's patch norm). */
int bcosk_bnu_stats_nhwc(const void* x, int64_t rows, int32_t c, int32_t dtype, float* partials, int32_t nblk, void* stream);
int bcosk_bnu_finalize(const float* partials, int32_t nblk, int64_t rows, int32_t c, const float* weight, float eps, float momentum,
                       float* running_var, float* alpha, float* mean, float* rstd, void* stream);
int bcosk_bnu_apply_nhwc(const void* x, int64_t rows, int32_t c, const float* alpha, const void* res, int32_t relu, void* y,
                         float* sq, int32_t dtype, void* stream);

/* Backward of [B-cos conv -> uncentred batch norm (batch statistics) -> (+ residual) -> ReLU] between two contractions.
 * Incoming gradient of the layer's output z:  g_z = ga + gb + xpost * tn[row]  (data gradients of the consumers, and the
 * consumers' patch-norm path: d||patch|| / dx = x / ||patch||);  g_y = g_z * [xpost > 0] when relu.
 *   reduce:   partials[b][c] = sum over block b's rows of g_y * out          ([nblk][c] fp32, fixed summation order)
 *   finalize: s = sum_b partials[b];  kcoef[c] = -rstd^3 * weight * s / rows;  g_weight[c] = s * rstd;  s_out[c] = s (optional)
 *   apply:    g_out = g_y * alpha[c] + (out - mean[c]) * kcoef[c]             (alpha NULL: g_out = g_y, no norm layer)
 *             g_lin = 2 * g_out * scale        (out = lin |lin| / n: the B-cos scale is part of the graph, bcosconv2d.py:186-194)
 *             gnt[row] = -sum_c g_out * out * inv_norm[row]^2;  g_y optionally stored (identity / downsample branch)
 * ga / out may be fp32 (ga_f32 / out_f32), everything else 16-bit of `dtype`. */
int bcosk_train_bwd_reduce(const void* ga, int32_t ga_f32, const void* gb, const void* xpost, const float* tn, int32_t relu,
                           const void* out, int32_t out_f32, int64_t rows, int32_t c, float* partials, int32_t nblk, int32_t dtype,
                           void* stream);
int bcosk_bnu_bwd_finalize(const float* partials, int32_t nblk, const float* rstd, const float* weight, int64_t rows, int32_t c,
                           float* kcoef, float* g_weight, float* s_out, void* stream);
int bcosk_train_bwd_apply(const void* ga, int32_t ga_f32, const void* gb, const void* xpost, const float* tn, int32_t relu,
                          const void* out, int32_t out_f32, const void* scale, const float* alpha, const float* kcoef,
                          const float* mean, const float* inv_norm, int64_t rows, int32_t c, void* g_lin, float* gnt, void* g_y,
                          int32_t dtype, void* stream);
/* out = ga + gb + x * tn[row] (16-bit rows; gb / tn optional): gradient of a tensor that is not a norm layer's output */
int bcosk_grad_combine(const void* ga, const void* gb, const void* x, const float* tn, int64_t rows, int32_t c, void* out,
                       int32_t dtype, void* stream);
/* Backward of AvgPool2d(k) (stride k, no padding; CLIP/clip/model.py:10-55 Bottleneck.avgpool and the downsample's AvgPool2d,
 * model.py:140-145 the stem's AvgPool2d(2)) fused with the consumers' terms at the pooled resolution, which the pool's output
 * receives like any conv input (ga + gb + x * tn, see bcosk_train_bwd_reduce):
 *   gx[img, y, x, :] (+)= (ga + gb + xp * tn[row])[img, y / k, x / k, :] / k^2        (pixels past the last full window: 0)
 * ga [nb*op*oq, c] 16-bit or fp32 (ga_f32), gb / xp 16-bit (optional), tn fp32 [nb*op*oq] (optional, needs xp), op = h / k,
 * oq = w / k; gx [nb, h, w, c] 16-bit, added to when accumulate.  One writer per element: bit-reproducible. */
int bcosk_pool_bwd_norm(const void* ga, int32_t ga_f32, const void* gb, const void* xp, const float* tn, int32_t nb, int32_t h,
                        int32_t w, int32_t c, int32_t k, int32_t accumulate, void* gx, int32_t dtype, void* stream);
/* tn[img, y, x] (+)= sum of gnt over the output pixels whose k x k window (stride, pad) covers input pixel (y, x) */
int bcosk_sumpool_transpose(const float* gnt, int32_t nb, int32_t h, int32_t w, int32_t k, int32_t stride, int32_t pad,
                            int32_t op, int32_t oq, int32_t accumulate, float* tn, void* stream);
/* UniformOffLabelsBCEWithLogitsLoss (losses.py:99-139, mean reduction): loss += mean BCE(logits, clamp(one_hot, min = off_label));
 * g_fc[n, pix, c] = d loss / d logits[n, c] * inv_temp / npix * grad_scale (through LogitLayer and the global average pool). */
int bcosk_bce_uniform_off(const float* logits, const int32_t* labels, int32_t n, int32_t c, float off_label, float inv_temp,
                          int32_t npix, float grad_scale, float* loss, void* g_fc, float* g_logits, int32_t dtype, void* stream);
/* out[i] = idx[i] >= 0 ? src[idx[i]] : 0, cast to 16 bit: fp32 master weights -> packed operand layouts */
int bcosk_gather_cast(const float* src, const int32_t* idx, int64_t n, void* out, int32_t dtype, void* stream);
/* Unit-wise adaptive gradient clipping (agc.py:28-42; one unit = one row of `cols` elements, 1-D parameters are one unit)
 * followed by AdamW on fp32 master weights.  The gradient of element i is g[gidx ? gidx[i] : i] * grad_scale. */
int bcosk_agc_adamw(float* w, const float* g, const int32_t* gidx, float* m, float* v, int32_t units, int32_t cols,
                    float grad_scale, float lr, float beta1, float beta2, float eps, float weight_decay, float clip_factor,
                    float agc_eps, int32_t step, void* stream);
/* Whole-model variants, one launch each and CUDA-graph friendly.  adam_state [3] fp32 on the device = {step, 1 - beta1^step,
 * 1 - beta2^step}: bcosk_adam_state_step advances it (so a captured training-step graph can be replayed), bcosk_agc_adamw_multi
 * runs AGC + AdamW for EVERY unit of the model (unit u = unit_cols[u] consecutive master weights at unit_off[u]; gidx maps every
 * master element to its gradient slot), bcosk_gather_cast_multi refreshes every packed operand (table[p] = {int32 index pointer,
 * 16-bit output pointer, n} as int64). */
int bcosk_adam_state_step(float* state, float beta1, float beta2, void* stream);
int bcosk_agc_adamw_multi(float* w, const float* g, const int32_t* gidx, float* m, float* v, const int64_t* unit_off,
                          const int32_t* unit_cols, int32_t units, float grad_scale, float lr, float beta1, float beta2, float eps,
                          float weight_decay, float clip_factor, float agc_eps, const float* adam_state, void* stream);
int bcosk_gather_cast_multi(const float* src, const int64_t* table, int32_t npacks, int64_t max_n, int32_t dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Bandwidth kernels (coalesced, 16-byte vectorised, warp-shuffle reductions)
 * ------------------------------------------------------------------------------------------- */

/* BcosifyNetwork.forward bcosify.py:50-53 (Normalize(mean6, std6)) fused with the NCHW fp32 -> NHWC
 * 16-bit layout change and the 2x2 space-to-depth that turns the 7x7/2 stem into a 4x4/1 conv:
 *   x    [nb, 6, h, w] fp32 (un-normalised [x, 1-x])
 *   out  [nb, h/2, w/2, planes * cp]   channel (dy*2+dx)*6 + c, zero padded to cp
 *   sq   [nb, h, w] fp32  sum_c xn^2 per ORIGINAL pixel (for the stem patch norm), summed over the STORED values (the sum
 *        of the planes written for each channel, squared), so that the norm matches the operand the stem GEMM reads; may be NULL */
int bcosk_input_prep_s2d(const float* x, int32_t nb, int32_t h, int32_t w, const float* mean6, const float* inv_std6,
                         void* out, int32_t cp, int32_t planes, int32_t dtype, float* sq, int32_t out_row_pitch,
                         int32_t out_img_pitch, void* stream);
/* Same, from uint8 RGB images x [nb, 3, h, w]: x/255 and the inverse channels 1 - x/255 (AddInverse,
 * bcos/data/transforms.py:42-55) are formed on the fly (8x fewer host->device bytes than fp32 6-channel input). */
int bcosk_input_prep_s2d_u8(const uint8_t* x, int32_t nb, int32_t h, int32_t w, const float* mean6,
                            const float* inv_std6, void* out, int32_t cp, int32_t planes, int32_t dtype, float* sq,
                            int32_t out_row_pitch, int32_t out_img_pitch, void* stream);
/* out_row_pitch / out_img_pitch (both entry points): pixels between consecutive rows / images of `out`; 0 = dense
 * (w/2 and h/2*w/2).  Non-dense pitches let `out` be a view into the zero-bordered buffer of a flat-window launch. */

/* BcosConv2d.calc_patch_norms bcosconv2d.py:196-231: inv_norm[img,p,q] = 1/sqrt(sumpool_k,s,p(sq) + eps_in) (conv)
 * or 1/(sqrt(sq) + eps_out) (linear, bcoslinear.py:113).  sq holds `parts` partial maps [parts][nb*h*w]. */
int bcosk_patch_inv_norm(const float* sq, int32_t parts, int32_t nb, int32_t h, int32_t w, int32_t kh, int32_t kw,
                         int32_t stride, int32_t pad, float eps_in, float eps_out, float* inv_norm, int32_t op,
                         int32_t oq, void* stream);

/* sum_c x^2 per pixel of an NHWC 16-bit tensor with planes -> sq [rows] (module-level path). */
int bcosk_pixel_sqsum(const void* x, int64_t rows, int32_t c, int32_t planes, int32_t plane_stride, int32_t ld,
                      int32_t dtype, float* sq, void* stream);

/* nn.AvgPool2d(k, s, pad) forward on NHWC 16-bit planes (count_include_pad=True), + optional sq map. */
int bcosk_avgpool_fwd(const void* x, int32_t nb, int32_t h, int32_t w, int32_t c, int32_t planes, int32_t k,
                      int32_t stride, int32_t pad, void* y, int32_t op, int32_t oq, int32_t dtype, float* sq,
                      void* stream);

/* Explain backward of AvgPool2d fused with the producer's gain: gx = avgpool_bwd(gy) * gain.
 * gx_row_pitch / gx_img_pitch: pixels between rows / images of gx, 0 = dense (see bcosk_input_prep_s2d). */
int bcosk_avgpool_bwd_mul(const void* gy, int32_t nb, int32_t h, int32_t w, int32_t c, int32_t planes, int32_t k,
                          int32_t stride, int32_t pad, int32_t op, int32_t oq, const void* gain, int32_t gain_f32,
                          void* gx, int32_t dtype, int32_t gx_row_pitch, int32_t gx_img_pitch,
                          const float* gain_sqrt_scale, void* stream);
/* gain_sqrt_scale [nb*h*w] non-NULL: `gain` holds the producer's ReLU output y and the multiplier is
 * sqrt(gain * gain_sqrt_scale[pixel]) (see bcosk_igemm_params.mul1_sqrt_scale); single 16-bit plane only. */

/* ResNetBcos._forward_impl standard_models.py:50-52 tail + LogitLayer logitlayer.py:22-27:
 * logits[img, cls] = mean_pix fc[img, pix, cls] * inv_temp + bias; pred[img] = argmax in torch.argmax's order: the first NaN,
 * else the first maximum (a row of -inf gives 0), so pred is always in [0, ncls). */
int bcosk_gap_logits(const float* fc, int32_t nb, int32_t npix, int32_t ncls, float inv_temp, float bias,
                     float* logits, int32_t* pred, void* stream);

/* Explain seed through GAP + classifier (one-hot logit gradient; bcos/common.py:166-177):
 *   g[img,pix,c] = inv_temp/npix * gain_fc[img,pix,cls] * W_fc[cls, c],  cls = target[img]
 *   out1 = g * mul1 (gain of the producing conv), out2 = g * mask2 bit   (both 16-bit planes) */
int bcosk_fc_seed_dgrad(const int32_t* target, const void* gain_fc, int32_t gain_f32, const float* w_fc, int32_t nb,
                        int32_t npix, int32_t ncls, int32_t c, float inv_temp, float seed_scale, const void* mul1,
                        int32_t mul1_f32, void* out1, const uint32_t* mask2, void* out2, int32_t planes, int32_t dtype,
                        void* stream);

/* (in_tensor * in_tensor.grad).sum(1) bcos/common.py:181, reading the stem dgrad in its space-to-depth
 * layout g [nb, h/2, w/2, cp] fp32 and the raw input x [nb,6,h,w] fp32:
 *   grad6[img,c,y,x] = g * inv_std6[c] * out_scale (optional output), cmap[img,y,x] = sum_c x * grad6
 * h and w must be even (as for bcosk_input_prep_s2d). */
int bcosk_contrib_map_s2d(const float* g, const float* x, int32_t nb, int32_t h, int32_t w, int32_t cp,
                          const float* inv_std6, float out_scale, float* cmap, float* grad6, void* stream);
int bcosk_contrib_map_s2d_u8(const float* g, const uint8_t* x, int32_t nb, int32_t h, int32_t w, int32_t cp,
                             const float* inv_std6, float out_scale, float* cmap, float* grad6, void* stream);

/* RGBA explanation images for a batch, on the device (replaces gradient_to_image bcos/common.py:387-436, which handles
 * one image and ends in numpy): out [nb, h, w, 4] fp32 = (r, g, b, alpha).  grad6 [nb,6,h,w] = dynamic linear weights,
 * x = the network input ([nb,6,h,w] fp32, or uint8 RGB [nb,3,h,w] with the inverse channels formed on the fly).
 * smooth = odd box-filter window of the alpha channel (15 in the reference, 0 = none), percentile in [0,100] (99.5):
 * alpha is divided by that per-image percentile (torch.quantile: linear interpolation of the two neighbouring order
 * statistics, found by radix select) and clipped to [0,1] like torch.clamp, which keeps NaN: an image whose percentile is
 * 0 gets NaN where its alpha is 0 (an all-zero gradient image: NaN everywhere), as the reference does.  The quantile's
 * position q*(n-1) is formed in fp32.  tmp: 2*nb*h*w + nb floats of scratch. */
int bcosk_explanation_rgba(const float* grad6, const float* x, int32_t nb, int32_t h, int32_t w, int32_t smooth,
                           float percentile, float* tmp, float* out, void* stream);
int bcosk_explanation_rgba_u8(const float* grad6, const uint8_t* x, int32_t nb, int32_t h, int32_t w, int32_t smooth,
                              float percentile, float* tmp, float* out, void* stream);

/* Localisation scores of a grid image (interpretability/analyses/localisation.py:306-388): attr [nt, c, h, w] fp32 =
 * attributions x*grad of nt targets -> sum over c -> smooth x smooth box average (odd, 0 = none; zero padded) -> sign flip
 * when negate -> clamp(min 0) -> mean over every cell x cell region -> out [nt, (h/cell)*(w/cell)] = region / total
 * (0 where total*region <= 0), regions in COLUMN-major order like `.permute(0,1,3,2).reshape(nt,-1)`.  The localisation
 * metric of target t is out[t][t].  tmp: 2*nt*h*w + nt*regions floats of scratch. */
int bcosk_localisation_scores(const float* attr, int32_t nt, int32_t c, int32_t h, int32_t w, int32_t smooth, int32_t cell,
                              int32_t negate, float* tmp, float* out, void* stream);

/* MaxOut for the module-level path (bcosconv2d.py:166-170 `lin.unflatten(1, (O, M)).max(2)`, bcoslinear.py:107-110):
 * lin [rows, o*m] fp32 (unit c = oo*m + k) -> y [rows, o] = best * scale(best, inv_norm[row]) with the launch's scale mode
 * and B; gain [rows, o] = that scale (optional), amax [rows, o] = index of the kept unit (optional, first on ties). */
int bcosk_maxout_bcos_fwd(const float* lin, const float* inv_norm, int64_t rows, int32_t o, int32_t m, int32_t scale_mode,
                          float b_exp, float* y, float* gain, uint8_t* amax, void* stream);
/* Explanation backward of MaxOut on 16-bit planes: dst [rows, planes*o*m] gets src [rows, planes*o] at the kept unit of
 * every group and zeros elsewhere (autograd of torch.max). */
int bcosk_maxout_scatter(const void* src, const uint8_t* amax, int64_t rows, int32_t o, int32_t m, int32_t planes,
                         int32_t dtype, void* dst, void* stream);

/* Generic element-wise helpers for the module-level (un-fused) path. */
/* batch_norm_uncentered_2d eval (batchnorm_uncentered.py:49-58) / ReLU on NHWC 16-bit: y = relu?(x*alpha[c]+beta[c]) */
int bcosk_channel_affine(const void* x, int64_t rows, int32_t c, const float* alpha, const float* beta, int32_t relu,
                         void* y, int32_t dtype, void* stream);
/* out = a * b element-wise (16-bit), used for g_out * detached scale */
int bcosk_mul(const void* a, const void* b, int64_t n, void* out, int32_t dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Module-level (un-fused) path: the reference's modules exchange NCHW fp32 tensors
 * ------------------------------------------------------------------------------------------- */
/* x [nb,c,h,w] fp32 (optionally * mul[pixel, c], e.g. g_out * detached gain) -> NHWC 16-bit planes
 * out [nb,h,w,planes*cp] (channels c..cp-1 zero) + optional per-pixel sum of squares (calc_patch_norms' first step) */
int bcosk_nchw_to_nhwc16(const float* x, int32_t nb, int32_t c, int32_t h, int32_t w, void* out, int32_t cp,
                         int32_t planes, int32_t dtype, const float* mul, int32_t mul_ld, float* sq, void* stream);
/* NHWC (fp32, or 16-bit planes summed) -> NCHW fp32 */
int bcosk_nhwc_to_nchw_f32(const void* y, int32_t y_f32, int32_t nb, int32_t c, int32_t h, int32_t w, int32_t ld,
                           int32_t planes, int32_t dtype, float* out, void* stream);
/* ---------------------------------------------------------------------------------------------
 * Fused SimpleViT plan (engine/vit.py): token tensors are [rows = images * tokens][planes * d] 16-bit precision planes
 * (plane pl at column pl * d), so the linear layers run as 1x1 bcosk_igemm launches with only these kernels in between.
 * ------------------------------------------------------------------------------------------- */
/* "b c (h p1) (w p2) -> b h w (p1 p2 c)" (bcos/models/vit.py:290-294) of the normalised [x, 1-x] input (bcosify_vit.py:79-82):
 * x [nb,6,h,w] fp32 (or uint8 RGB [nb,3,h,w], inverse channels formed on the fly) -> out [nb*(h/p)*(w/p)][planes * p*p*6],
 * column (p1*p + p2)*6 + c; sq [rows] = sum of the stored values squared (the patch-embedding B-cos linear's input norm). */
int bcosk_vit_patchify(const float* x, int32_t nb, int32_t h, int32_t w, int32_t p, const float* mean6, const float* inv_std6,
                       void* out, int32_t planes, int32_t dtype, float* sq, void* stream);
int bcosk_vit_patchify_u8(const uint8_t* x, int32_t nb, int32_t h, int32_t w, int32_t p, const float* mean6, const float* inv_std6,
                          void* out, int32_t planes, int32_t dtype, float* sq, void* stream);
/* (x * grad).sum(1) (bcos/common.py:181) from the patch-embedding data gradient g [rows][p*p*6] fp32 (columns as above):
 * cmap[img,y,x] = sum_c x6[c] * g[..] * inv_std6[c] * out_scale; grad6 [nb,6,h,w] (optional) receives the dynamic linear weights */
int bcosk_vit_contrib_map(const float* g, const float* x, int32_t nb, int32_t h, int32_t w, int32_t p, const float* inv_std6,
                          float out_scale, float* cmap, float* grad6, void* stream);
int bcosk_vit_contrib_map_u8(const float* g, const uint8_t* x, int32_t nb, int32_t h, int32_t w, int32_t p, const float* inv_std6,
                             float out_scale, float* cmap, float* grad6, void* stream);
/* DetachableLayerNorm.forward (centered_norms.py:187-224, bias-free): y = (x - mean) / sqrt(var + eps) * w over d, plane rows in
 * (`planes`) and out (`out_planes`, 0 = the same: a two-plane residual stream may feed one-plane branch operands); rstd [rows] is
 * kept for the explanation pass, sq [rows] (optional) = sum of the stored outputs squared. */
int bcosk_vit_ln_fwd(const void* x, int64_t rows, int32_t d, int32_t planes, int32_t out_planes, const float* w, float eps, void* y,
                     float* rstd, float* sq, int32_t dtype, void* stream);
/* Explanation backward of that LayerNorm (variance detached, mean in the graph) fused with the residual-stream add and the gain
 * of the linear layer in front:  G_out = G_in + rstd * (g w - mean_d(g w));  ghat = G_out * gain.
 * g [rows][d] fp32 or one 16-bit plane; G_in / G_out fp32 (G_in, G_out, gain optional); ghat one 16-bit plane (optional). */
int bcosk_vit_ln_bwd(const void* g, int32_t g_f32, const float* G_in, int64_t rows, int32_t d, const float* w, const float* rstd,
                     float* G_out, const void* gain, int32_t gain_f32, void* ghat, int32_t dtype, void* stream);
/* MyGELU (bcosify_vit.py:27-32) on plane rows: a = u * Phi(u), sq [rows] = sum a^2 (optional); gain [rows][d] (optional, the
 * saved gain of the B-cos linear that produced u, 16-bit or fp32) is multiplied in place by the detached gate Phi(u). */
int bcosk_vit_gelu_fwd(const void* u, int64_t rows, int32_t d, int32_t planes, void* a, float* sq, void* gain, int32_t gain_f32,
                       int32_t dtype, void* stream);
/* Attention.forward (bcos/models/vit.py:143-158) on plane rows, one CTA per (image, head), dim_head = 64, n <= 208:
 * qkv [batch*n][planes * 3*heads*64] (q | k | v blocks per plane).  backward = 0: out [batch*n][planes * heads*64] =
 * softmax(q k^T scale) v.  backward = 1 (explanation mode: q, k frozen): out [batch*n][heads*64] one 16-bit plane = P^T g,
 * g [batch*n][heads*64] fp32, P recomputed from q, k. */
int bcosk_vit_attention(const void* qkv, int32_t planes, const float* g, int32_t batch, int32_t n, int32_t heads, int32_t dim_head,
                        float scale, int32_t backward, void* out, int32_t dtype, void* stream);

/* CLIP ViT image encoder (engine/clip_vit.py).  The reference converts only conv1 and the MLP linears of CLIP's VisionTransformer
 * (bcosify.py:74-113); LayerNorm, QuickGELU and nn.MultiheadAttention (CLIP/clip/model.py:157-204) stay stock and are differentiated
 * exactly in its explanation pass.  True backward forms:
 *   ln_bwd_full         with xh = (x - mean) rstd, gw = g w:  G_out = G_in + rstd (gw - mean(gw) - xh mean(gw xh)); ghat = G_out (* gain)
 *                       (x: the LayerNorm input as plane rows; other arguments as bcosk_vit_ln_bwd)
 *   quickgelu_fwd       a = u sigmoid(1.702 u) on plane rows, sq = sum a^2; gain *= sigmoid + 1.702 u sigmoid (1 - sigmoid)
 *   attention_bwd_full  dV = P^T g, dz = P o (g V^T - rowsum(P o g V^T)), dQ = scale dz K, dK = scale dz^T Q -> out [batch*n][3*heads*64]
 *                       one 16-bit plane (q | k | v blocks); qkv, g as bcosk_vit_attention; n <= 112 */
int bcosk_vit_ln_bwd_full(const void* g, int32_t g_f32, const void* x, int32_t planes, const float* G_in, int64_t rows, int32_t d,
                          const float* w, const float* rstd, float* G_out, const void* gain, int32_t gain_f32, void* ghat, int32_t dtype,
                          void* stream);
int bcosk_vit_quickgelu_fwd(const void* u, int64_t rows, int32_t d, int32_t planes, void* a, float* sq, void* gain, int32_t gain_f32,
                            int32_t dtype, void* stream);
int bcosk_vit_attention_bwd_full(const void* qkv, int32_t planes, const float* g, int32_t batch, int32_t n, int32_t heads, int32_t dim_head,
                                 float scale, void* out, int32_t dtype, void* stream);
/* The same attention on the tensor cores (csrc/bcosk_vit_attn.cu: TMA boxes, tcgen05.mma into TMEM for q k^T and for the
 * probability-weighted sums, softmax by the TMEM-lane threads; V and, in the backward, the probabilities and g are fed as
 * MN-major operands, so no transpose exists).  Same arguments and results as bcosk_vit_attention up to fp32 rounding;
 * n <= 256, dim_head = 64.  The explanation pass rounds the probabilities and g / row-sum to ONE 16-bit plane (its format). */
int bcosk_vit_attention_tc(const void* qkv, int32_t planes, const float* g, int32_t batch, int32_t n, int32_t heads, int32_t dim_head,
                           float scale, int32_t backward, void* out, int32_t dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused DenseNet plan (engine/densenet.py).  A dense block keeps ONE feature tensor F [pixels][planes * C_total]; every layer's
 * 3x3 launch writes its new channels into its slice of F (y pointer + column offset, y_ld = planes * C_total), so the
 * torch.cat of torchvision's _DenseLayer never copies.  Every consumer applies ITS OWN eval-mode uncentred BN + ReLU
 * (batchnorm_uncentered.py:49-58) to the channels it reads:
 * ------------------------------------------------------------------------------------------- */
/* y [rows][planes * c] = relu?(x[:, :c] * alpha[c]) (x rows [rows][x_ld], plane pl at column pl * x_plane_stride);
 * sq [rows] = sum y^2 (optional), maskbits [rows][c/32] = ReLU bits (optional, c % 32 == 0). */
int bcosk_dense_bn_relu_fwd(const void* x, int64_t rows, int32_t c, int32_t planes, int32_t x_ld, int32_t x_plane_stride,
                            const float* alpha, int32_t relu, void* y, float* sq, uint32_t* maskbits, int32_t dtype, void* stream);
/* Its (explanation / plain) backward into the fp32 feature-gradient tensor G [rows][g_ld]:
 * G[:, :c] = (accumulate ? G[:, :c] : 0) + g * alpha * mask bit;  g [rows][c] fp32 or one 16-bit plane. */
int bcosk_dense_bn_relu_bwd(const void* g, int32_t g_f32, int64_t rows, int32_t c, const float* alpha, const uint32_t* maskbits,
                            float* G, int32_t g_ld, int32_t accumulate, int32_t dtype, void* stream);
/* out [rows][c] (one 16-bit plane) = G[:, col0 : col0 + c] * gain[rows][c] (optional, 16-bit or fp32) * scale: the A operand of
 * the data gradient of the layer that produced those channels. */
int bcosk_dense_slice_cast(const float* G, int32_t g_ld, int32_t col0, int64_t rows, int32_t c, const void* gain, int32_t gain_f32,
                           float scale, void* out, int32_t dtype, void* stream);
/* Strided device-to-device copy (cudaMemcpy2DAsync): a pooled tensor into the first channels of the next block's F. */
int bcosk_copy_rows_2d(void* dst, int64_t dst_pitch_bytes, const void* src, int64_t src_pitch_bytes, int64_t width_bytes,
                       int64_t rows, void* stream);

/* DenseNet fine-tuning step (engine/train.py DenseNetTrainPlan, csrc/bcosk_dense_train.cu).  In train mode consumer l normalises
 * F[:, :C_l] with the batch statistics of those channels, which do not depend on the consumer: they are computed ONCE per slice
 * of F, when the slice is written.  In the backward pass consumer l's batch-statistics term for channel c is
 * (F[:, c] - mean[c]) * k_l[c], k_l = -rstd^3 w_l S_l / rows, S_l[c] = sum_m g_y * F: linear in (F - mean), so the block keeps
 * ONE accumulator K = sum_l k_l, applied when the producer of the slice runs its backward (all consumers of a slice run before
 * it in reverse order).  16-bit rows of `dtype`, fp32 arithmetic; every reduction is a fixed-order sum of per-block partials
 * (no atomics: bit-reproducible).  F / G rows have pitch ld (= C_total) elements; c <= 2048, c % 8 == 0, col0 % 8 == 0.
 * slice_stats:  mean / var (centred, biased) / rstd = 1/sqrt(var + eps) of F[:, col0 : col0 + c] -> mean, var, rstd [col0 ..
 *               col0 + c) (arrays of the whole block); partials [nblk][2c] fp32 scratch.
 * consumer_finalize:  alpha[:c] = weight * rstd;  running_var[:c] = (1 - momentum) running_var + momentum var  (this consumer's buffer).
 * consumer_bwd (one pass over the prefix; the consumer is a 1x1 B-cos conv, so its patch-norm vector is its own gnt):
 *               g_y = (g_t + t * gnt[row]) * [t > 0];  G[:, :c] = (accumulate ? G[:, :c] : 0) + g_y * alpha;
 *               partials[b][c] = sum over block b's rows of g_y * F      (g_t fp32 or 16-bit [rows][c], t 16-bit [rows][c])
 * consumer_bwd_finalize:  S = sum_b partials[b];  g_weight = S * rstd;  K[:c] = (accumulate ? K[:c] : 0) + k_l.
 * slice_bwd:    g_out = G[:, slice] + (F[:, slice] - mean) * K.  scale != NULL (the slice is a B-cos conv's output F = lin |lin| / n,
 *               scale = |lin| / n [rows][c]): out = 2 * scale * g_out and gnt[row] = -sum_c g_out * F * inv_norm[row]^2;
 *               scale == NULL (a block's input channels): out = g_out.  out [rows][c] dense 16-bit. */
int bcosk_dense_slice_stats(const void* F, int64_t rows, int32_t ld, int32_t col0, int32_t c, float eps, float* partials, int32_t nblk,
                            float* mean, float* var, float* rstd, int32_t dtype, void* stream);
int bcosk_dense_consumer_finalize(const float* var, const float* rstd, const float* weight, int32_t c, float momentum, float* running_var,
                                  float* alpha, void* stream);
int bcosk_dense_consumer_bwd(const void* g_t, int32_t g_t_f32, const void* t, const float* gnt, const float* alpha, const void* F, int32_t ld,
                             int64_t rows, int32_t c, float* G, int32_t accumulate, float* partials, int32_t nblk, int32_t dtype, void* stream);
int bcosk_dense_consumer_bwd_finalize(const float* partials, int32_t nblk, const float* rstd, const float* weight, int64_t rows, int32_t c,
                                      int32_t accumulate, float* K, float* g_weight, void* stream);
int bcosk_dense_slice_bwd(const float* G, const void* F, int32_t ld, int32_t col0, int64_t rows, int32_t c, const float* mean, const float* K,
                          const void* scale, const float* inv_norm, void* out, float* gnt, int32_t dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Attention-pool head of the CLIP ResNet encoders inside the fused plan (BcosAttentionPool2d.forward bcosattnpool.py:34-59, pooled
 * mode; csrc/bcosk_head.cu).  Only the mean token's output is kept, so projections commute with the pooling: scores
 * s_j = (W_k,h^T q_h) . x_j, output o_h = W_v,h (sum_j p_j x_j) - three token-equivalents of projections per image instead of 150.
 * fp32 on the CUDA cores (small: 32 GFLOP per 512 images).
 * ------------------------------------------------------------------------------------------- */
/* C[i] (m x n, row pitch ldc) = alpha * op(A[i]) (m x k) * op(B[i]) (k x n) for i < batch; row-major, operand i at base + i * stride;
 * trans_a: A is stored k x m; trans_b: B is stored n x k. */
int bcosk_sgemm_batched(int32_t trans_a, int32_t trans_b, int32_t m, int32_t n, int32_t k, const float* a, int64_t lda, int64_t stride_a,
                        const float* b, int64_t ldb, int64_t stride_b, float* c, int64_t ldc, int64_t stride_c, int32_t batch, float alpha,
                        void* stream);
/* The same, adding into C: C[i] += alpha * op(A[i]) * op(B[i]). */
int bcosk_sgemm_batched_acc(int32_t trans_a, int32_t trans_b, int32_t m, int32_t n, int32_t k, const float* a, int64_t lda,
                            int64_t stride_a, const float* b, int64_t ldb, int64_t stride_b, float* c, int64_t ldc, int64_t stride_c,
                            int32_t batch, float alpha, void* stream);
/* tokens [nb][npix + 1][c] fp32 from the trunk output planes x [nb][npix][planes * c]: token 0 = mean over the pixels
 * (bcosattnpool.py:37-38: cat([x.mean(0), x])), token j + 1 = pixel j. */
int bcosk_head_tokens(const void* x, int32_t nb, int32_t npix, int32_t c, int32_t planes, int32_t dtype, float* tokens, void* stream);
/* in-place softmax over rows of n fp32 values */
int bcosk_row_softmax(float* s, int64_t rows, int32_t n, void* stream);
/* Backward of the row softmax (the attention weights p = softmax(s), bcosattnpool.py:48-50 through F.multi_head_attention_forward,
 * with q and k in the graph as in training): ds = p * (dp - sum_j p_j dp_j) per row of n fp32 values; ds may alias dp. */
int bcosk_softmax_bwd(const float* p, const float* dp, int64_t rows, int32_t n, float* ds, void* stream);
/* Gradient wrt the tokens g_tokens [nb][npix + 1][c] fp32 -> the last trunk block's gradient tensors (see bcosk_seed_from_nchw):
 * g[pix] = g_tokens[pix + 1] + g_tokens[0] / npix;  out1 = planes(g * scale * mul1) (mul1 NULL: 1), out2 = planes(g * scale [* mul2]) under mask2. */
int bcosk_seed_from_tokens(const float* g_tokens, int32_t nb, int32_t npix, int32_t c, float scale, const void* mul1, int32_t mul1_f32,
                           void* out1, const uint32_t* mask2, const void* mul2, int32_t mul2_f32, void* out2, int32_t planes,
                           int32_t dtype, void* stream);

/* Stem patch matrix for the contract-mode plans with uint8 input.  The k x k / stride stem conv over the normalised [x, 1-x] input
 * (BcosifyNetwork.forward bcosify.py:50-53 + BcosifyConv2d) is linear in the raw byte v of every colour, so it equals a GEMM over
 * rows of (v_R, v_G, v_B, 1) per tap with folded weights (engine/pack.py stem_im2col_weight): the bytes are exact in ONE 16-bit plane
 * and the window is gathered once.  out [nb*op*oq][kp] (kp % 64 == 0, kp >= 4 k^2): column tap*4 + c = v_c * a_scale, tap*4 + 3 = 1
 * for in-image taps, zeros elsewhere; inv_norm [nb*op*oq] = 1/sqrt(sum over the window of the 6 normalised channels squared + 1e-6)
 * (calc_patch_norms bcosconv2d.py:196-231). */
int bcosk_stem_im2col_u8(const uint8_t* x, int32_t nb, int32_t h, int32_t w, int32_t k, int32_t stride, int32_t pad, const float* mean6,
                         const float* inv_std6, float a_scale, void* out, int32_t kp, float* inv_norm, int32_t dtype, void* stream);

/* Seed of a fused trunk's explanation pass from a gradient computed OUTSIDE the plan (CLIP encoders: the attention-pool head
 * bcos/modules/bcosattnpool.py:34-59 runs on the module-level path and autograd hands back d target / d trunk output):
 * g [nb, c, h, w] fp32 NCHW ->  out1[pix, pl*c + ch] = planes(g * seed_scale * mul1[pix, ch])  (mul1 = gain of the block's last conv)
 *                               out2[pix, pl*c + ch] = planes(g * seed_scale [* mul2[pix, ch]]) where bit ch of mask2[pix] is set
 * mul1 / mul2: [nb*h*w, c] 16-bit or fp32; mask2: [nb*h*w, ceil(c/32)] words (the block's ReLU bits); out1 / out2 may be NULL. */
int bcosk_seed_from_nchw(const float* g, int32_t nb, int32_t c, int32_t h, int32_t w, float seed_scale, const void* mul1,
                         int32_t mul1_f32, void* out1, const uint32_t* mask2, const void* mul2, int32_t mul2_f32, void* out2,
                         int32_t planes, int32_t dtype, void* stream);
/* Strided movers of the module-level path.  zero_insert: dst[img, s*p, s*q, :] = src[img, p, q, :] (row_elems 16-bit elements per pixel,
 * a multiple of 8; dst [nb, h, w, row_elems] is zero elsewhere and stays so): the zero-inserted gradient of a strided k x k conv.
 * nhwc_scatter_nchw_f32: out[img, ch, s*p, s*q] = y[img, p, q, ch] (y as in bcosk_nhwc_to_nchw_f32; out [nb, c, h, w] zero elsewhere):
 * the data gradient of a strided 1x1 conv.  pixel_sqsum_nchw_f32: sq[img, pix] = sum_ch x[img, ch, pix]^2 (calc_patch_norms
 * bcosconv2d.py:196-231 on the reference's own NCHW fp32 layout). */
int bcosk_zero_insert_nhwc(const void* src, int32_t nb, int32_t oh, int32_t ow, int32_t row_elems, void* dst, int32_t h, int32_t w,
                           int32_t stride, void* stream);
int bcosk_nhwc_scatter_nchw_f32(const void* y, int32_t y_f32, int32_t nb, int32_t c, int32_t oh, int32_t ow, int32_t ld, int32_t planes,
                                int32_t dtype, float* out, int32_t h, int32_t w, int32_t stride, void* stream);
int bcosk_pixel_sqsum_nchw_f32(const float* x, int32_t nb, int32_t c, int64_t hw, float* sq, void* stream);
/* out = relu?((x * alpha[c] + beta[c]) * smul + sadd) on NCHW fp32: batch_norm_uncentered_2d (eval / after statistics)
 * batchnorm_uncentered.py:45-58 and LogitLayer.forward logitlayer.py:22-27 (alpha = beta = NULL) */
int bcosk_scale_bias_nchw(const float* x, int32_t nb, int32_t c, int64_t hw, const float* alpha, const float* beta, float smul,
                          float sadd, int32_t relu, float* out, void* stream);
/* per-channel mean and biased variance over (N,H,W): x.var(dim=(0,2,3), unbiased=False) batchnorm_uncentered.py:39 */
int bcosk_channel_stats_nchw(const float* x, int32_t nb, int32_t c, int64_t hw, float* mean, float* var, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Token models (B-cosified SimpleViT), fp32 I/O
 * ------------------------------------------------------------------------------------------- */
/* DetachableLayerNorm.forward bcos/modules/norms/centered_norms.py:187-224: y = w*(x-mean)/sqrt(var+eps)+b per row of d
 * values; rstd[row] = 1/sqrt(var+eps) is saved for the explanation backward */
int bcosk_layernorm_fwd(const float* x, int64_t rows, int32_t d, const float* w, const float* b, float eps, float* y,
                        float* rstd, void* stream);
/* explanation backward of the above (variance detached :211, mean in graph): gx = (w*gy - mean_d(w*gy)) * rstd */
int bcosk_layernorm_explain_bwd(const float* gy, int64_t rows, int32_t d, const float* w, const float* rstd, float* gx,
                                void* stream);
/* attn_unpool head of BcosAttentionPool2d.forward bcos/modules/bcosattnpool.py:23-33: y = x / ||x||_2 per row (token) of d
 * values, inv[row] = 1/||x||_2 saved; with the norm detached (:30-31) the explanation backward is bcosk_row_scale(gy, inv) */
int bcosk_l2norm_rows(const float* x, int64_t rows, int32_t d, float* y, float* inv, void* stream);
/* y[row, :] = x[row, :] * s[row] */
int bcosk_row_scale(const float* x, int64_t rows, int32_t d, const float* s, float* y, void* stream);
/* MyGELU bcosify_vit.py:27-32: g == NULL: y = x * gate(x);  g != NULL (explanation backward, gate detached): y = g * gate(x) */
int bcosk_gelu_gate(const float* x, const float* g, int64_t n, float* y, void* stream);
/* Attention.forward bcos/models/vit.py:143-158 after to_qkv: qkv [batch, n, 3*heads*64] ->
 *   backward == 0: out [batch, n, heads*64] = softmax(q k^T * scale) v
 *   backward == 1: explanation backward with q, k detached (:148-150): out [batch, n, 3*heads*64] (pre-zeroed), v block =
 *                  P^T g, g [batch, n, heads*64] */
int bcosk_attention(const float* qkv, const float* g, int32_t batch, int32_t n, int32_t heads, int32_t dim_head, float scale,
                    int32_t backward, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Group / position normalisation with detachable statistics, NCHW fp32 (module-level path)
 * ------------------------------------------------------------------------------------------- */
/* group_norm_uncentered groupnorm_uncentered.py:21-61 (centred == 0) and DetachableGroupNorm2d.forward
 * centered_norms.py:93-138 (centred == 1): per (image, group) var = biased CENTRED variance over (C/groups, H, W);
 * y = w[c] * (x - centred*mean) / sqrt(var + eps) + b[c]; rstd[nb*groups] saved for the explanation backward.
 * groups == 1 is the GN-LayerNorm, groups == c the GN-InstanceNorm of the reference. */
int bcosk_groupnorm_fwd(const float* x, int32_t nb, int32_t c, int64_t hw, int32_t groups, const float* w, const float* b,
                        float eps, int32_t centred, float* y, float* rstd, void* stream);
/* explanation backward (variance detached, mean in graph): gx = (w*gy - centred*mean_group(w*gy)) * rstd */
int bcosk_groupnorm_explain_bwd(const float* gy, int32_t nb, int32_t c, int64_t hw, int32_t groups, const float* w,
                                const float* rstd, int32_t centred, float* gx, void* stream);
/* PositionNormUncentered2d.forward posnorm_uncentered.py:39-58 (centred == 0) and DetachablePositionNorm2d.forward
 * centered_norms.py:251-297 (centred == 1): the same with the statistics over the channels of one pixel; rstd[nb*hw] */
int bcosk_positionnorm_fwd(const float* x, int32_t nb, int32_t c, int64_t hw, const float* w, const float* b, float eps,
                           int32_t centred, float* y, float* rstd, void* stream);
int bcosk_positionnorm_explain_bwd(const float* gy, int32_t nb, int32_t c, int64_t hw, const float* w, const float* rstd,
                                   int32_t centred, float* gx, void* stream);

const char* bcosk_last_error(void);
int bcosk_version(void);
/* sizeof(bcosk_igemm_params) as compiled into the library (binding self-check). */
int bcosk_sizeof_igemm_params(void);
/* 1 when the current device is compute capability 10.x (sm_100a kernels can run). */
int bcosk_device_supported(void);

#ifdef __cplusplus
}
#endif
#endif /* BCOSK_H_ */
