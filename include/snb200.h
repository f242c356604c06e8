/*
 * snb200.h — C-ABI of the B200-native StereoNet hot path (libsnb200.so).
 *
 * Drop-in boundary for miloknowles/adaptive-stereo-icra-2021's StereoNet forward / online-adaptation step.
 * The reference has no native interface (it is 100 % PyTorch); every entry point below replaces the ATen/cuDNN
 * calls issued by one span of adaptive_stereo/models/stereo_net.py (cited per function, paths relative to the
 * reference checkout).  The host side (stereonet_b200/models/stereo_net.py) mirrors the reference nn.Module API
 * and calls these through ctypes with raw device pointers.
 *
 * Conventions
 *  - plain C types only: device pointers, ints, floats, an opaque cudaStream_t passed as void*.
 *  - the caller owns every buffer (inputs, outputs, workspaces); the library never allocates, frees or
 *    synchronises, and every launch is ordered on the given stream (CUDA-graph capturable).
 *  - activations are fp32 channels-last: [B,H,W,32] (2-D) or [B,D,H,W,32] (3-D); images are NCHW fp32 as the
 *    reference's callers pass them; single-channel maps are [B,H,W] / [B,D,H,W].
 *  - return value 0 on success, non-zero on failure; snb_last_error() returns a thread-local message.
 *  - re-entrant: no global mutable state (the reference may be driven from a ROS callback thread,
 *    ros/stereo_depth_node.py:113), except the mutex-guarded host-side record of the arguments of the last
 *    snb_stereonet_adapt_forward per workspace, which snb_stereonet_adapt_update checks its own against.
 */
#ifndef SNB200_H_
#define SNB200_H_

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SNB_API __attribute__((visibility("default")))
#else
#define SNB_API
#endif

#define SNB_C 32 /* channel width of every hidden activation (stereo_net.py:59,64,155) */
/* OR-ed into `passes` of the tensor-core convolutions / `mode` of snb_prep_conv_weights_tc: error-compensated split with fp16
 * operands (tcgen05.mma.kind::f16, K = 16, power-of-two weight scaling) instead of 3xTF32 — same three products, same
 * fp32-grade result, half the MMA count.  The weight image must have been prepared in the matching format. */
#define SNB_CONV_F16 0x10
/* OR-ed into `mode` of snb_prep_conv_weights_tc[_batch]: the weight image layout of snb_conv_c32_ws (fp16 split; one image per
 * (window, kw) with the three taps of the walk axis stacked along N; snb_conv_weights_ws_floats(kd) floats). */
#define SNB_CONV_WS 0x20

/* Geometry of one convolution over channels-last tensors. 2-D convs use D = OD = KD = 1, pd = 0. */
typedef struct {
  int B, D, H, W;     /* input  [B,D,H,W,C] */
  int OD, OH, OW;     /* output [B,OD,OH,OW,C] */
  int KD, KH, KW;     /* taps */
  int stride;         /* H/W stride (depth stride is always 1) */
  int dil;            /* H/W dilation (depth dilation is always 1) */
  int pd, ph, pw;     /* zero padding */
  int transposed;     /* 0: y = conv(x).  1: data gradient of that conv (x := dy [B,D,H,W], y := dx [B,OD,OH,OW]):
                         tap (kd,kh,kw) reads x at ((o + p - k*dil) / stride) when divisible; weights from
                         snb_prep_conv_weights mode 2.  Needed for the stride-2 5x5 layers (stereo_net.py:64-70). */
} snb_conv_geom;

/* Epilogue of the 32->32 convolution: z = conv + bias; stats += (sum z, sum z^2) per channel;
 * y = z*scale + shift (if scale); y = LeakyReLU_0.2(y) (if lrelu); y += residual (if residual). */
typedef struct {
  const float* bias;      /* [32] or NULL */
  const float* scale;     /* [32] or NULL : folded eval-mode BatchNorm (stereo_net.py:17,29) */
  const float* shift;     /* [32] (required when scale != NULL) */
  const float* residual;  /* channels-last tensor shaped like the output, or NULL (BasicBlock, stereo_net.py:50) */
  float* stats;           /* [ntiles][2][32] per-tile partial sums for train-mode BN, or NULL */
  int lrelu;              /* 1: LeakyReLU(0.2) (stereo_net.py:39,94,159) */
} snb_conv_epilogue;

SNB_API const char* snb_last_error(void);
SNB_API int snb_version(void);

/* Number of 128-position tiles (= rows of the `stats` partial buffer) snb_conv_c32 uses for this geometry. */
SNB_API int snb_conv_c32_num_tiles(const snb_conv_geom* g);

/* Repack a PyTorch conv weight [Cout][Cin][taps] into the kernels' [taps][Cin][Cout] layout.
 * mode 0: forward weights.  mode 1: data-gradient weights (taps flipped, Cin/Cout swapped) for a stride-1 'same' conv run as
 * a plain convolution.  mode 2: Cin/Cout swapped, taps NOT flipped, for snb_conv_geom.transposed = 1. */
SNB_API int snb_prep_conv_weights(const float* w, float* out, int cout, int cin, int taps, int mode, void* stream);

/* Difference cost volume — replaces the host-side zero+H2D+24-slice loop of stereo_net.py:173-184.
 * left/right [B,H,W,32] -> cost [B,D,H,W,32]; cost[b,d,y,x,c] = left[b,y,x,c] - right[b,y,x-d,c] (x >= d) else 0. */
SNB_API int snb_cost_volume_fwd(const float* left, const float* right, float* cost, int B, int D, int H, int W, void* stream);
/* Adjoint of the above (autograd of the slice assignments, stereo_net.py:178-182). */
SNB_API int snb_cost_volume_bwd(const float* dcost, float* dleft, float* dright, int B, int D, int H, int W, void* stream);

/* 32->32 convolution, fp32 CUDA-core (FFMA) implicit GEMM — replaces nn.Conv2d / nn.Conv3d (+ folded BN, LeakyReLU,
 * residual add) at stereo_net.py:10-17,23-29,44-51,64-70,77,81-85,185-186.  wprep from snb_prep_conv_weights. */
SNB_API int snb_conv_c32(const float* x, const float* wprep, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e, void* stream);

/* Same contract as snb_conv_c32 for stride-1 "same" 3x3 (dilated) / 3x3x3 convolutions, on the tcgen05 tensor cores
 * (TF32 operands from shared memory, fp32 accumulators in TMEM; kw folded into N = 96).  passes = 3: error-compensated
 * 3xTF32 split (fp32-grade results); passes = 1: plain single-pass TF32.  wimg from snb_prep_conv_weights_tc.
 * `stats` rows are indexed by this kernel's own tiles: snb_conv_c32_tc_num_tiles().
 * 3-D (KD = 3) runs conv3d_c32_tma.cu: one TMA tile load per (kd,kh) window of the un-padded flat index, converter warps
 * (hi/lo split -> tcgen05.st) and the A operand in TMEM; passes | 0x400 selects the older loader-warp kernel (no `stats`).
 * (A TMEM-operand variant of the loader-warp kernel was measured and dropped: with 3 warps left to load 9 windows per tile it is
 * loader-bound, 113 us vs 72 us.) */
SNB_API int snb_conv_c32_tc(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                    int passes, void* stream);
SNB_API int snb_conv_c32_tc_num_tiles(const snb_conv_geom* g);
/* Diagnostics: same launch, plus per-CTA cycle counters [grid][16] = {loader wait-empty, loader total, MMA wait-full,
 * MMA wait-tmem, MMA total, epilogue wait-tmem-full, epilogue total, epilogue barrier} (clock64 ticks). */
SNB_API int snb_conv_c32_tc_profile(const float* x, const float* wimg, float* y, const snb_conv_geom* g,
                            const snb_conv_epilogue* e, int passes, long long* counters, void* stream);
/* 2-D specialisation with the "vertical walk" schedule (consecutive tiles of a CTA step down a column block by `dil` rows
 * and share two of their three input-row windows: 3x less loader / L2 traffic).  Same weights image (kd = 1), same
 * epilogue contract; `stats` has snb_conv2d_c32_tc_num_tiles() rows (one per image row x column block). */
SNB_API int snb_conv2d_c32_tc(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                      int passes, void* stream);
SNB_API int snb_conv2d_c32_tc_num_tiles(const snb_conv_geom* g);
/* Diagnostics: same launch plus per-CTA cycle counters (layout of snb_conv_c32_tc_profile).  passes | 0x100 selects the
 * legacy path that feeds the A operand from shared memory instead of TMEM (for A/B measurements). */
SNB_API int snb_conv2d_c32_tc_profile(const float* x, const float* wimg, float* y, const snb_conv_geom* g,
                              const snb_conv_epilogue* e, int passes, long long* counters, void* stream);
/* Round-2 product kernel for the 2-D (dilated) and 3-D layers (csrc/conv_c32_ws.cu; weight image from
 * snb_prep_conv_weights_tc with mode | SNB_CONV_WS): walk along the slowest kernel axis, the kw shift applied on the way INTO the
 * tensor core (converter warps write three shifted fp16-split copies of every raw input row into TMEM), the three taps of the walk
 * axis folded into N = 96 over a ring of accumulators, all weight images resident in shared memory, one TMA tile store per output
 * tile; a residual that is the layer's own input (BasicBlock, stereo_net.py:50) comes from the rows already on chip.  Same contract
 * as snb_conv_c32_tc except: `stats` (train-mode BN partials; snb_conv_c32_ws_num_tiles() rows) may only be combined with `bias` —
 * which is how the adaptation step uses it. */
SNB_API int snb_conv_c32_ws(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                    void* stream);
SNB_API int snb_conv_c32_ws_num_tiles(const snb_conv_geom* g);
/* Reduced-precision inference variant of snb_conv_c32_ws (same arguments, same weight image, same epilogue): ONE fp16 product per
 * tap, out = 2^-s (xh . wh) with xh = fp16(x) and wh the high half of the prepared weight, fp32 accumulation.  That is about
 * 1e-3 relative error per layer, so its results are reported separately from the fp32 parity contract of every other call here.
 * Inputs below 2^-14 in magnitude are fp16 subnormals and lose relative precision (BatchNorm-normalised activations and cost-volume
 * differences sit well above that).  Inference only: `stats` must be NULL (rejected by name, nothing launched). */
SNB_API int snb_conv_c32_ws_f16(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                        void* stream);
SNB_API int snb_conv_weights_ws_floats(int kd);      /* kd = 1, 3; 5: the image set of snb_conv5x5s2_c32_ws */
/* downsample[1:] (nn.Conv2d(32, 32, 5, stride 2, padding 2), stereo_net.py:64-70) in ONE launch of the same kernel: the four
 * polyphase images of the input (snb_phase_split / snb_conv5x5s2_c3 with phases = 1; [4][B][OH][OW][32]) are four raw windows per
 * walk step feeding one accumulator ring.  wimg from snb_prep_conv5x5s2_weights_ws (or batch kind 2).  No residual input. */
SNB_API int snb_conv5x5s2_c32_ws(const float* phases, const float* wimg, float* y, int B, int OH, int OW,
                         const snb_conv_epilogue* e, void* stream);
/* The same layer straight from the un-split input x [B][H][W][32] (H, W >= 2): the polyphase images are four STRIDED TMA views
 * of x (element strides 2 in x and y, zero fill past an odd edge), so no split pass exists; y [B][ceil(H/2)][ceil(W/2)][32]. */
SNB_API int snb_conv5x5s2_c32_ws_x(const float* x, const float* wimg, float* y, int B, int H, int W,
                           const snb_conv_epilogue* e, void* stream);
SNB_API int snb_prep_conv5x5s2_weights_ws(const float* w, float* out, void* stream);
/* The refinement's input layer (upsample + scale + concat + Conv2d(4 -> 32) [+ BN + LeakyReLU], stereo_net.py:105-117) on the walk
 * kernel: snb_refine_pack_input writes x4 [B][H][W][4] = (mul * bilinear(coarse), r, g, b) and the upsampled plane up [B][H][W];
 * snb_conv_c4_ws convolves it — the three kw taps of a pixel are 48 contiguous bytes = ONE K = 16 slice, 3 MMAs per walk step.
 * wimg: snb_prep_conv_weights_tc(kd = 1, mode = SNB_CONV_WS) of W'[co][kw*4 + ch][kh][0] = w[co][ch][kh][kw] (a [32][32][3][3]
 * tensor, zero elsewhere).  Epilogue as snb_conv_c32_ws (stats rows: snb_conv_c32_ws_num_tiles of the 3x3 geometry); no residual. */
SNB_API int snb_refine_pack_input(const float* coarse, const float* rgb, float* x4, float* up, int B, int h, int w, int H, int W,
                          float mul, void* stream);
SNB_API int snb_conv_c4_ws(const float* x4, const float* wimg, float* y, int B, int H, int W, const snb_conv_epilogue* e, void* stream);
/* Diagnostics: same launch plus per-CTA cycle counters [grid][16]. */
SNB_API int snb_conv_c32_ws_profile(const float* x, const float* wimg, float* y, const snb_conv_geom* g,
                            const snb_conv_epilogue* e, long long* counters, void* stream);
/* Repack [32][32][kd*3*3] weights into the tensor-core B-operand smem image (hi/lo TF32 split, SWIZZLE_128B K-major,
 * one 24 KB block per (kd,kh) window).  kd = 1 (2-D) or 3 (3-D).  mode 0: forward, 1: data gradient. */
SNB_API int snb_prep_conv_weights_tc(const float* w, float* out, int kd, int mode, void* stream);
SNB_API int snb_conv_weights_tc_floats(int kd);
/* All weight images of a model in ONE launch (the adaptation step re-derives ~50 of them after every optimizer update).
 * table: n device-resident entries of 4 int64 = {source weight pointer, output image pointer, config, 0};
 * config = nwin | mode << 8 | kind << 16 | a << 24 | b << 28.  kind 0: a [32][32][nwin*3] weight as in
 * snb_prep_conv_weights_tc (nwin = 3 kd).  kind 1: the polyphase 3x3 sub-kernel (a, b) of a [32][32][5][5] stride-2 weight,
 * sub[i][j] = w[2i + a][2j + b] (zero outside the 5x5 support), nwin = 3 (csrc/phase.cu).  kind 2: the image set of
 * snb_conv5x5s2_c32_ws from a [32][32][5][5] weight (nwin = 10, mode = SNB_CONV_WS).  kind 3: the snb_conv_c4_ws image from the
 * refinement input layer's [32][4][3][3] weight (nwin = 3, mode = SNB_CONV_WS). */
SNB_API int snb_prep_conv_weights_tc_batch(const long long* table, int n, void* stream);

/* Polyphase helpers for the stride-2 5x5 32->32 layers (stereo_net.py:64-70): the convolution is the sum of four stride-1
 * 'same' 3x3 convolutions over the phase images P_ab[i][j] = x[2i+a][2j+b], so forward and data gradient run on
 * snb_conv2d_c32_tc.  snb_phase_split: x [B,H,W,32] -> out [4][B,ceil(H/2),ceil(W/2),32] (phase a*2+b, zero padded);
 * snb_phase_merge: the inverse interleave, in [4][B,ceil(H/2),ceil(W/2),32] -> dx [B,H,W,32]. */
SNB_API int snb_phase_split(const float* x, float* out, int B, int H, int W, void* stream);
SNB_API int snb_phase_merge(const float* in, float* dx, int B, int H, int W, void* stream);

/* Small-Cin first layers.
 * snb_conv5x5s2_c3: FeatureExtractorNetwork.downsample[0] (stereo_net.py:64-70,81): NCHW image [B,3,H,W] -> [B,OH,OW,32]. */
SNB_API int snb_conv5x5s2_c3(const float* img, const float* w /*[32][3][5][5]*/, const float* bias, float* y,
                     int B, int H, int W, void* stream);
/* Same convolution, written directly as the four polyphase images [4][B][OH/2][OW/2][32] that the following stride-2 layer
 * consumes (inference path: saves the separate snb_phase_split pass).  OH and OW must be even. */
SNB_API int snb_conv5x5s2_c3_phases(const float* img, const float* w, const float* bias, float* yph, int B, int H, int W, void* stream);
/* snb_refine_in_conv: EdgeAwareRefinement stereo_net.py:105-117 fused: bilinear upsample of coarse [B,h,w] to HxW
 * (align_corners=False), * disp_scale, concat with NCHW rgb, Conv2d(4->32,3x3,p1) + bias.  Writes the upsampled
 * disparity to up [B,H,W] and z [B,H,W,32]; epilogue fields as in snb_conv_c32 (residual unused). */
SNB_API int snb_refine_in_conv(const float* coarse, const float* rgb, const float* w /*[32][4][3][3]*/, float* up, float* z,
                       int B, int h, int w_, int H, int W, float disp_scale, const snb_conv_epilogue* e, void* stream);
SNB_API int snb_refine_in_conv_num_tiles(int B, int H, int W);

/* Channel contraction of a 32->1 convolution: taps[b,(d),t,y,x] = sum_c w[t][c] * x[b,(d),y,x,c].
 * First half of conv3d_alone (stereo_net.py:162,187) and conv2d_out (stereo_net.py:102,121). ntaps = 27 or 9.
 * npos = B*D*H*W positions, plane = H*W. */
SNB_API int snb_conv_c32_taps(const float* x, const float* w /*[1][32][ntaps]*/, float* taps, long long nslices, int plane, int ntaps, void* stream);

/* Second half of conv3d_alone fused with the soft-argmin (stereo_net.py:187-192, DisparityRegression :124-134):
 * cost[b,d,y,x] = bias + sum over the 27 shifted tap planes; p = softmax_d(+cost); pred = sum_d d * p_d.
 * cost_out may be NULL (stereo_net.py:197-198 returns it when requested). */
SNB_API int snb_tapsum_softargmin(const float* taps /*[B,D,27,H,W]*/, const float* bias /*[1]*/, float* cost_out /*[B,D,H,W]*/,
                          float* pred /*[B,H,W]*/, int B, int D, int H, int W, void* stream);

/* conv3d_alone + softmax + DisparityRegression as ONE kernel (stereo_net.py:187-198, :124-134) — the product path; the two
 * entry points above remain as the independent cross-check.  x [B,D,H,W,32] channels-last, w [1][32][3][3][3], bias [1] ->
 * pred [B,H,W] = sum_d d * softmax_d(cost), optional cost_out [B,D,H,W] (the pre-softmax cost volume adapt.py:73 asks for)
 * and optional fcs_out [B,H,W] = feature-contrast score of that cost (feature_contrast.py:12-23; same value as
 * snb_feature_contrast(cost_out)).  A CTA streams the input rows of its output band once: each activation leaves HBM once,
 * the tap sums never leave the chip; softmax / expectation / top-2 over D are warp-shuffle reductions.  D <= 64. */
SNB_API int snb_conv3d_out_softargmin(const float* x, const float* w /*[1][32][3][3][3]*/, const float* bias /*[1]*/,
                              float* cost_out, float* pred, float* fcs_out, int B, int D, int H, int W, void* stream);

/* Second half of conv2d_out fused with the residual add + ReLU (stereo_net.py:121): out = relu(up + bias + sum taps).
 * bias / up may be NULL and relu = 0 turns it into a plain 3x3 tap gather (used by the refinement-head data gradient). */
SNB_API int snb_tapsum_refine_out(const float* taps /*[B,9,H,W]*/, const float* bias, const float* up, float* out,
                          int B, int H, int W, int relu, void* stream);

/* out[b,y,x] = mul * bilinear(in[b], size (H,W), align_corners=False) — stereo_net.py:201-202 (mul = 2**k). */
SNB_API int snb_upsample_bilinear(const float* in, float* out, int B, int h, int w, int H, int W, float mul, void* stream);
/* adjoint: din[b,y,x] (+)= mul * sum of bilinear weights * dout ; din must be zeroed by the caller when accumulate=0 is not used */
SNB_API int snb_upsample_bilinear_bwd(const float* dout, float* din, int B, int h, int w, int H, int W, float mul, void* stream);

/* Train-mode BatchNorm (batch statistics, adapt.py:313-314).  Reduces the per-tile partials written by a conv epilogue,
 * updates running stats in place (momentum, unbiased variance) and emits scale = gamma*invstd, shift = beta - mean*scale,
 * plus mean / invstd for the backward pass. */
SNB_API int snb_bn_finalize(const float* stats, int ntiles, long long count, const float* gamma, const float* beta,
                    float* running_mean, float* running_var, float momentum, float eps,
                    float* scale, float* shift, float* mean, float* invstd, void* stream);
/* Same, with a caller-provided scratch of 64 x 64 floats: more than 256 partial rows are first reduced by 64 CTAs (a single
 * CTA walking ~1 MB of partials is bound by one SM's load bandwidth).  num_batches_tracked (nn.BatchNorm's int64 counter, or
 * NULL) is incremented by the same launch when the running statistics are updated. */
SNB_API int snb_bn_finalize_ws(const float* stats, int ntiles, long long count, const float* gamma, const float* beta,
                       float* running_mean, float* running_var, long long* num_batches_tracked, float momentum, float eps,
                       float* scale, float* shift, float* mean, float* invstd, float* scratch, void* stream);
/* The running-statistics half of snb_bn_finalize[_ws] for a call that was made WITHOUT running buffers: running = (1 - m) running
 * + m batch statistic (unbiased variance from invstd), num_batches_tracked += 1.  Lets the left / right feature passes of one
 * adaptation step (adapt.py:72) run on two streams and still update nn.BatchNorm's buffers in the reference's order. */
SNB_API int snb_bn_running_update(const float* mean, const float* invstd, long long count, float* running_mean, float* running_var,
                          long long* num_batches_tracked, float momentum, float eps, void* stream);
/* y = [residual +] LeakyReLU(z*scale + shift) over n positions x 32 channels. */
SNB_API int snb_bn_apply(const float* z, const float* scale, const float* shift, const float* residual, float* y,
                 long long npos, int lrelu, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Backward pass of the adaptation step (autograd of stereo_net.py:79-85,168-207, triggered at adapt.py:390).
 * Data gradients of the 3x3 / 3x3x3 convolutions reuse snb_conv_c32 / snb_conv_c32_tc with mode-1 weights; the
 * stride-2 5x5 layers use snb_conv_c32 with snb_conv_geom.transposed = 1 and mode-2 weights.
 * --------------------------------------------------------------------------------------------------------------- */
/* Number of blocks (rows of the partial buffers) the elementwise backward kernels use for npos positions. */
SNB_API int snb_bwd_num_blocks(long long npos);
/* BatchNorm(+LeakyReLU) backward, pass 1: partial[blk][0:32] = sum du, [32:64] = sum du*zhat with
 * u = z*scale + shift, du = dy * (u > 0 ? 1 : 0.2) (or dy when lrelu = 0), zhat = (z - mean) * invstd. */
SNB_API int snb_bn_lrelu_bwd_reduce(const float* z, const float* dy, const float* scale, const float* shift, const float* mean,
                            const float* invstd, float* partial, long long npos, int lrelu, void* stream);
/* pass 2: dz = scale * (du - train * (sums[0:32]/N + zhat * sums[32:64]/N)); dzpart[blk][32] = per-block sum of dz. */
SNB_API int snb_bn_lrelu_bwd_apply(const float* z, const float* dy, const float* scale, const float* shift, const float* mean,
                           const float* invstd, const float* sums, long long npos, int train, int lrelu,
                           float* dz, float* dzpart, void* stream);
/* out[j] = mul * sum_i partial[i][j], i < n, j < len (fixed order, double accumulation). */
SNB_API int snb_reduce_partials(const float* partial, int n, int len, float* out, float mul, void* stream);
/* Sum the per-CTA weight-gradient partials [n][taps][32 cin][32 cout] and write PyTorch's layout out[cout][cin][taps]
 * (fixed order, double accumulation): reduction and layout change of snb_conv_c32_wgrad[_tc] in one launch. */
SNB_API int snb_reduce_wgrad_partials(const float* partial, int n, int taps, float* out, void* stream);
/* partial[blk][32] = per-channel sums of x [npos][32] (bias gradient of a plain convolution). */
SNB_API int snb_channel_sum(const float* x, float* partial, long long npos, void* stream);
/* Weight gradient of a 32->32 convolution: partial[cta][taps][cin][cout]; sum over cta with snb_reduce_partials. */
SNB_API int snb_conv_c32_wgrad(const float* x, const float* dz, float* partial, const snb_conv_geom* g, void* stream);
SNB_API int snb_conv_c32_wgrad_num_partials(const snb_conv_geom* g);
/* Same result for the stride-1 'same' 3x3 (dilated) / 3x3x3 layers on the tcgen05 tensor cores: the reduction over
 * positions is the GEMM K dimension, both operands are MN-major SWIZZLE_128B images of the channels-last rows (no
 * transpose), kw shifts are descriptor offsets into one dz row window, each x row window is fetched once ("walk"
 * schedules).  passes = 3: 3xTF32 split (fp32-grade); 1: plain TF32.  partial[cta][taps][cin][cout] with
 * snb_conv_c32_wgrad_tc_num_partials() CTAs. */
SNB_API int snb_conv_c32_wgrad_tc(const float* x, const float* dz, float* partial, const snb_conv_geom* g, int passes, void* stream);
SNB_API int snb_conv_c32_wgrad_tc_num_partials(const snb_conv_geom* g);
/* Diagnostics: same launch plus dbg[cta][64] = {accumulator mask, slots, tiles, any, ..., raw TMEM samples}. */
SNB_API int snb_conv_c32_wgrad_tc_debug(const float* x, const float* dz, float* partial, const snb_conv_geom* g, int passes,
                                float* dbg, void* stream);
/* Weight gradients of the small-Cin layers: partial[tile][k = (ci,kh,kw)][cout]. */
SNB_API int snb_conv5x5s2_c3_wgrad(const float* img, const float* dy, float* partial, int B, int H, int W, void* stream);
SNB_API int snb_conv5x5s2_c3_num_tiles(int B, int H, int W);
SNB_API int snb_refine_in_wgrad(const float* coarse, const float* rgb, const float* dz, float* partial,
                        int B, int h, int w_, int H, int W, float disp_scale, void* stream);
/* Soft-argmin backward: dcost[b,d,y,x] = p_d * (d - pred) * dpred (+ dcost_extra), p = softmax_d(cost). */
SNB_API int snb_softargmin_bwd(const float* cost, const float* pred, const float* dpred, const float* dcost_extra, float* dcost,
                       int B, int D, int H, int W, void* stream);
/* dres = dout * (out > 0)  (ReLU of stereo_net.py:121). */
SNB_API int snb_relu_bwd(const float* out, const float* dout, float* dres, long long n, void* stream);
/* Backward of a 32->1 3x3(x3) convolution given g = d(output) [B,D,H,W]: dx [B,D,H,W,32] and per-CTA partials
 * [ceil(npos/128)][ntaps*32 + 1] holding dw[tap][c] and, last, db. */
SNB_API int snb_conv_c32_taps_bwd(const float* x, const float* w, const float* g, float* dx, float* partial,
                          int B, int D, int H, int W, int ntaps, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * SURVEY.md section 8 row f1: fused photometric loss of the adaptation step (adapt.py:78-86; LinearWarping
 * linear_warping.py:18-57; SSIM / L1 / edge-aware smoothness loss_functions.py:41-138), forward value AND gradient
 * w.r.t. the predicted disparity in three launches.  left/right [B,3,H,W] NCHW, disp [B,H,W] (full resolution),
 * loss_out [1 + B]: [0] = the masked mean over the whole batch (what adapt.py:83 returns), [1 + b] = the same masked mean
 * over sample b alone (= what StateMachine.validate, adapt.py:122-142, gets from its one-pair-at-a-time loop; row f4);
 * ddisp [B,H,W] = d loss_out[0] / d disp, workspace of snb_photo_loss_workspace_floats(B,H,W) floats.
 * smooth_w = 1e-3 in adapt.py:81-83. */
SNB_API int snb_photo_loss(const float* left, const float* right, const float* disp, float* loss_out, float* ddisp,
                   float* workspace, int B, int H, int W, float smooth_w, void* stream);
SNB_API int snb_photo_loss_workspace_floats(int B, int H, int W);
/* Row f2: feature-contrast score of a cost volume [B,D,H,W] -> [B,H,W] (feature_contrast.py:12-23, adapt.py:352-353):
 * max_d cost - mean of all but the two largest costs, without sorting. */
SNB_API int snb_feature_contrast(const float* cost, float* out, int B, int D, int H, int W, void* stream);
/* Row f3: khamis_robust_loss (loss_functions.py:6-15; the experience-replay term of adapt.py:339-349) over n elements:
 * loss_out [1] = sum_{gt > 0} (sqrt((gt - pred)^2 + 4) / 2 - 1) / max(#valid, 1), dpred [n] = d loss / d pred,
 * workspace of snb_khamis_loss_workspace_floats(n) floats.  Two launches, deterministic, no host sync. */
SNB_API int snb_khamis_loss(const float* pred, const float* gt, float* loss_out, float* dpred, float* workspace, long long n,
                    void* stream);
SNB_API int snb_khamis_loss_workspace_floats(long long n);
/* Row f4: evaluation metrics of train.py:98-107 as per-sample sums over gt > 0 (hw = H*W elements per sample):
 * out [B][6] = {sum |pred - gt|, #valid, #(|e| > 2), #(|e| > 3), #(|e| > 4), #(|e| > 5)}; EPE = out[0] / out[1],
 * D1-all_t = out[2 + t] / out[1].  One CTA per sample, deterministic. */
SNB_API int snb_eval_metrics(const float* pred, const float* gt, float* out, int B, long long hw, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Optimizer side of the adaptation step (adapt.py:391-393) and the flat gradient bucket of shared-model data parallelism
 * (SURVEY.md section 8e).
 * snb_multi_gather: n device tensors (src[i], count[i] floats; src[i] == NULL writes zeros) -> dst + dst_off[i].  src / dst_off /
 * count are HOST arrays (they travel as kernel parameters: CUDA-graph capturable, no table upload). */
SNB_API int snb_multi_gather(const float* const* src, const long long* dst_off, const long long* count, int n, float* dst, void* stream);
/* clip_grad_norm_(first n_clip elements of the bucket, max_norm; max_norm <= 0: no clipping) + Adam (no weight decay, no amsgrad)
 * over the flat bucket: g = flat_grad * grad_scale (* clip coefficient inside the clipped group); exp_avg / exp_avg_sq are flat
 * buffers laid out like the bucket; `step` is a device float incremented by the call (bias corrections are computed on the
 * device: capturable).  chunk_table: device [nchunks][3] int64 = {parameter address of the chunk, flat offset, count <= 1024}.
 * workspace: snb_adam_clip_workspace_bytes() bytes, 8-byte aligned; after the call its last four floats hold {clip coefficient,
 * lr / (1 - beta1^t), 1 / sqrt(1 - beta2^t), total norm of the clipped group}.  Three launches. */
SNB_API int snb_adam_clip_step(const long long* chunk_table, int nchunks, const float* flat_grad, float* exp_avg, float* exp_avg_sq,
                       float* step, long long n_total, long long n_clip, float max_norm, float grad_scale, double lr,
                       double beta1, double beta2, double eps, void* workspace, void* stream);
SNB_API int snb_adam_clip_workspace_bytes(void);

/* ---------------------------------------------------------------------------------------------------------------
 * Whole-model inference (eval mode): StereoNet's feature extractor on both images plus the stereo head, as the Python
 * engine runs it (stereonet_b200.runtime.StereoEngine), for hosts without Python or torch (csrc/model.cu).  Bit-identical
 * to that path.  The adaptation step (train mode, backward, clip + Adam) is the snb_stereonet_adapt_* group further below.
 *
 * params: HOST array of DEVICE pointers (contiguous fp32), one per tensor the eval forward reads, in the reference's state_dict
 * order: feature_net (downsample.i.{weight,bias}, residual_blocks.i.conv1.0.0.{weight,bias},
 * residual_blocks.i.conv1.0.1.{weight,bias,running_mean,running_var}, conv_alone.{weight,bias}), then stereo_net (filter.i.0.0 /
 * .0.1 as above, conv3d_alone, edge_aware_refinements.0.conv2d_feature.0.0 / .0.1, .residual_astrous_blocks.i.conv1.0.0 / .0.1,
 * .conv2d_out).  BasicBlock.conv2.* and num_batches_tracked are not read.  2k + 108 tensors (stereonet_b200.native.param_names).
 * --------------------------------------------------------------------------------------------------------------- */
SNB_API int snb_stereonet_num_params(int k);
/* Size of the prepared-weights buffer.  It holds everything the forward reads (tensor-core weight images, folded eval-mode
 * BatchNorm, copies of the raw biases and small weights), so the caller may free or change `params` after prepare. */
SNB_API long long snb_stereonet_weights_bytes(int k);
/* Where the tensor params[index] left its derived piece inside `weights`: byte offset and size (size 0 for the running statistics,
 * which only feed the fold).  Weight images of the 32->32 convolutions, the ten-image sets of downsample[1:], the refinement input
 * layer's four-channel image; BatchNorm weight -> folded scale [32], BatchNorm bias -> folded shift [32]; everything else a copy. */
SNB_API int snb_stereonet_weights_piece(int k, int index, long long* offset, long long* bytes);
/* Derive `weights` (device, 256-byte aligned, snb_stereonet_weights_bytes(k) bytes) from params: one launch pair, no host-to-device
 * copy (capturable).  Call again after a parameter changed. */
SNB_API int snb_stereonet_prepare(const float* const* params, int k, void* weights, void* stream);
/* Workspace of snb_stereonet_forward in bytes, or -1 (snb_last_error) for arguments the forward rejects. */
SNB_API long long snb_stereonet_workspace_bytes(int k, int input_scale, int maxdisp, int B, int H, int W);
/* images [2][B][3][H][W] fp32 NCHW (left batch, then right batch).  With D' = (maxdisp + 1) / 2^(input_scale + k) (in [1, 32])
 * and h, w the size after k stride-2 layers (h = ceil(H / 2^k) step by step):
 *   disp   [B,H,W]     = pred_disp_l/{input_scale}
 *   coarse [B,H,W]     = pred_disp_l/{input_scale + k}, or NULL
 *   cost   [B,D',h,w]  = cost_volume_l/{input_scale + k}, or NULL
 *   fcs    [B,h,w]     = feature-contrast score of that cost volume (needs cost and D' > 2), or NULL.
 * weights and workspace (snb_stereonet_workspace_bytes) 256-byte aligned, the other buffers 16-byte aligned.  Nothing outside
 * these extents is written.  Independent calls may run concurrently on separate streams with separate workspaces and outputs. */
SNB_API int snb_stereonet_forward(const void* weights, int k, int input_scale, int maxdisp, const float* images, int B, int H, int W,
                          void* workspace, float* disp, float* coarse, float* cost, float* fcs, void* stream);
/* Opt-in reduced-precision forward for throughput inference: the same arguments, weights buffer, workspace size and launch sequence
 * as snb_stereonet_forward, with the 32->32 3x3 layers of the feature extractor and the refinement and the 3x3x3 cost-filter layers
 * on snb_conv_c32_ws_f16 (one fp16 product per tap instead of the fp32-grade three).  The 5x5 stride-2 layers, the refinement's
 * input layer, the first layer and the 32->1 heads are unchanged.  Its disparities differ from snb_stereonet_forward's by far more
 * than the fp32 parity tolerance, so its numbers are reported separately from that contract (DESIGN.md section 4.2f16 lists the
 * measured errors).  Inputs below 2^-14 in magnitude lose relative precision in fp16 (see snb_conv_c32_ws_f16).  Bit-identical to
 * stereonet_b200.runtime.StereoEngine(..., precision="fp16"). */
SNB_API int snb_stereonet_forward_f16(const void* weights, int k, int input_scale, int maxdisp, const float* images, int B, int H, int W,
                              void* workspace, float* disp, float* coarse, float* cost, float* fcs, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Whole-model online adaptation, single pass (adapt.py:304-396 without experience replay: the update of the NONE / NONSTOP / VS
 * modes; the replay step of ER and VS+ER follows below), for hosts without Python or torch (csrc/adapt.cu).  Bit-identical to the Python step
 * AdaptStepper(f, s, make_optimizer(f, s, lr, fused=True), two_streams=False).  Two calls per frame, because the host decides
 * from the loss whether to update (adapt.py:381: not when the frame was just added to the OVS):
 *   snb_stereonet_adapt_forward  train-mode forward of both images (adapt.py:72-73; BatchNorm running statistics and
 *                                num_batches_tracked move, left pass, right pass, stereo head, refinement), Monodepth loss
 *                                (adapt.py:78-86, :328-337) and feature-contrast score (adapt.py:352-353);
 *   snb_stereonet_adapt_update   backward from what the forward saved in `workspace` (adapt.py:390), every gradient into the flat
 *                                bucket, clip_grad_norm_ on stereo_net (adapt.py:391-392) and Adam (adapt.py:393).
 * `params` is the list of snb_stereonet_prepare (2k + 108 tensors, stereonet_b200.native.param_names); Adam rewrites the parameters
 * in place and the forward rewrites running_mean / running_var.  `state` (snb_stereonet_adapt_state_bytes, 256-byte aligned) holds
 * the gradient bucket, Adam's moments and step, and the weight images the forward derives from the parameters.  The bucket is laid
 * out as optim.FusedAdamClip's: used parameters only, stereo_net first, then feature_net, in named_parameters() order, without
 * BasicBlock.conv2.*; so FusedAdamClip state (and adam.pth through its state_dict) converts by copying the flat buffers.
 * Contract: update follows a forward with the same workspace and arguments, and the parameter values do not change in between.
 * The library records each forward's arguments on the host, keyed by the workspace address, and the update rejects by name, before
 * any launch, a workspace no forward has run on and any k, input_scale, maxdisp, B, H, W, state or params[i] other than its
 * forward's (this holds under graph capture too, where each call runs on the host once).  The parameter addresses are those given
 * to snb_stereonet_adapt_init.  No allocation, no synchronisation, no host-to-device copy: both calls are
 * CUDA-graph capturable.
 * --------------------------------------------------------------------------------------------------------------- */
SNB_API long long snb_stereonet_adapt_state_bytes(int k);
/* what: 0 flat_grad [n] fp32, 1 exp_avg [n], 2 exp_avg_sq [n], 3 step [1] fp32 (Adam's t); byte offset and size inside `state`. */
SNB_API int snb_stereonet_adapt_state_piece(int k, int what, long long* offset, long long* bytes);
/* Element offset and count of params[index]'s slot in the bucket (count 0: a running statistic, no slot). */
SNB_API int snb_stereonet_adapt_grad_slot(int k, int index, long long* offset, long long* count);
/* Zero the bucket, the moments and step, and write Adam's per-chunk table from the parameter addresses (two launches). */
SNB_API int snb_stereonet_adapt_init(float* const* params, int k, void* state, void* stream);
/* Workspace of the forward / update pair in bytes (the activations the update reads and both calls' scratch), or -1. */
SNB_API long long snb_stereonet_adapt_workspace_bytes(int k, int input_scale, int maxdisp, int B, int H, int W);
/* images [2][B][3][H][W] as in snb_stereonet_forward.  bn_counters: the 17 num_batches_tracked int64 counters in module order
 * (feature_net's six BasicBlocks, stereo_net's four filters, the refinement's input layer and six blocks), or NULL.
 *   loss     [1 + B]  [0] = the batch's masked photometric mean (adapt.py:83), [1 + b] = sample b's
 *   disp     [B,H,W]  pred_disp_l/{input_scale}, or NULL
 *   fcs      [B,h,w]  feature-contrast score of the coarse cost volume, or NULL
 *   fcs_mean [1]      its mean (fixed-order double sum), or NULL.  fcs and fcs_mean need more than 2 coarse disparity levels.
 * state, workspace 256-byte aligned; images, disp, fcs 16-byte aligned. */
SNB_API int snb_stereonet_adapt_forward(float* const* params, long long* const* bn_counters, int k, int input_scale, int maxdisp,
                                const float* images, int B, int H, int W, void* state, void* workspace, float* loss, float* disp,
                                float* fcs, float* fcs_mean, void* stream);
/* Gradients of loss[0] into the bucket (slots of parameters without a gradient: zeros), then snb_adam_clip_step with
 * max_norm (<= 0: no clipping), lr, beta1, beta2, eps (torch.optim.Adam defaults 0.9, 0.999, 1e-8). */
SNB_API int snb_stereonet_adapt_update(float* const* params, int k, int input_scale, int maxdisp, int B, int H, int W, void* state,
                               void* workspace, float max_norm, double lr, double beta1, double beta2, double eps, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * The same step with experience replay (adapt.py:339-349, :381-394: the update of the ER and VS+ER modes), bit-identical to
 * AdaptStepper(f, s, make_optimizer(f, s, lr, fused=True), two_streams=False).step(left, right, replay=(rl, rr, gt)).  The forward
 * runs a second train-mode pass on a stored sample with ground truth and adds er_weight times its Khamis robust loss
 * (loss_functions.py:6-15) to the photometric loss of the stream frame; the update differentiates both passes and applies clip +
 * Adam once.  Choosing the sample (reservoir, OVS) stays with the host.  Same contract as the single pass above; the update must be
 * snb_stereonet_adapt_update_replay with the forward's RB (and a plain forward's update snb_stereonet_adapt_update), which the
 * update checks by name before any launch.  Both calls are CUDA-graph capturable.
 * --------------------------------------------------------------------------------------------------------------- */
/* Workspace of the replay forward / update pair in bytes (RB >= 1), or -1. */
SNB_API long long snb_stereonet_adapt_replay_workspace_bytes(int k, int input_scale, int maxdisp, int B, int H, int W, int RB);
/* As snb_stereonet_adapt_forward (images, loss, disp, fcs, fcs_mean keep their meaning: the stream frame's), then the replay pass,
 * whose BatchNorm running statistics and counters move after the stream pass's (per frame: feature_net's counters + 4, stereo_net's
 * + 2), and the Khamis loss of its disparity:
 *   replay_images  [2][RB][3][H][W]  the stored pair (same H and W as the frame, RB >= 1), 16-byte aligned
 *   replay_gt      [RB][H][W]        its ground-truth disparity, gt <= 0 marks an invalid pixel
 *   er_weight      weight of the replay term (adapt.py's 0.05), finite and >= 0
 *   loss_replay    [2]               {khamis term, total = loss[0] + er_weight * khamis} (the loss AdaptStepper.step returns) */
SNB_API int snb_stereonet_adapt_forward_replay(float* const* params, long long* const* bn_counters, int k, int input_scale,
                                       int maxdisp, const float* images, int B, int H, int W, const float* replay_images,
                                       const float* replay_gt, int RB, float er_weight, void* state, void* workspace, float* loss,
                                       float* loss_replay, float* disp, float* fcs, float* fcs_mean, void* stream);
/* Gradients of the total loss (both passes) into the bucket, then snb_adam_clip_step as snb_stereonet_adapt_update. */
SNB_API int snb_stereonet_adapt_update_replay(float* const* params, int k, int input_scale, int maxdisp, int B, int H, int W, int RB,
                                      void* state, void* workspace, float max_norm, double lr, double beta1, double beta2, double eps,
                                      void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SNB200_H_ */
