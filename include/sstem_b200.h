/*
 * sstem_b200.h -- C ABI of the B200-native (sm_100a) hot path of
 * sydeng99/ssTEM-restoration: the 51-tap adaptive separable local convolution
 * (forward, grad w.r.t. vertical / horizontal taps, grad w.r.t. input) and the
 * flow-driven bilinear backward warps.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / THC types.
 * Each entry point names the reference interface it replaces (paths relative to
 * the reference checkout).  INTEGRATION.md shows the binding a maintainer of the
 * reference would add (ctypes, as the reference bound its THC library via cffi in
 * libs/sepconv/_ext/cunnex/__init__.py:2-15).
 *
 * Conventions
 *   - every pointer is DEVICE memory on one GPU; fp32 unless stated; tensors are
 *     contiguous NCHW exactly as the reference asserts
 *     (libs/sepconv/SeparableConvolution.py:33-35);
 *   - the caller allocates every output; the callee overwrites all of it (no
 *     zero-fill needed, unlike SeparableConvolution.py:37,60-62);
 *   - `stream` is a cudaStream_t (0 = legacy default stream).  Calls are
 *     asynchronous and re-entrant; the launch happens on the device that owns
 *     the output pointer (the calling thread's current device is restored);
 *   - return 0 on success, a positive cudaError_t on a CUDA failure, a negative
 *     SSTEM_E_* on bad arguments.  sstem_error_string() explains either.
 */
#ifndef SSTEM_B200_H_
#define SSTEM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSTEM_ABI_VERSION 7

/* argument errors (negative) */
#define SSTEM_E_NULL      (-1)  /* a required pointer is NULL */
#define SSTEM_E_SHAPE     (-2)  /* non-positive size / unsupported tap count */
#define SSTEM_E_ALIGN     (-3)  /* pointer not 4-byte aligned */
#define SSTEM_E_DEVICE    (-4)  /* pointer is not device memory */
#define SSTEM_E_FLAG      (-5)  /* unknown flag / mode */

/* flags for the sepconv entry points */
#define SSTEM_SEPCONV_DEFAULT       0u
/* evaluate the forward in the reference's exact summation order (fy outer, fx
 * inner, one accumulator, (in*v) then fma with h -- kernel.cu:45-49): bit-exact
 * with the reference kernel, ~2x the arithmetic.  Verification mode. */
#define SSTEM_SEPCONV_STRICT_ORDER  1u
/* The caller asserts that all `channels` planes of `input` are identical copies -- what the
 * reference's callers feed it (grayscale sections replicated x3:
 * sff_scripts_interp/data/data_provider.py:136-137, inference.py:71-77).  The forward then
 * computes one plane and writes `channels` copies (bit-identical to the general path); the tap
 * gradients use t = (sum_c g_c) * in_0 (same value up to fp32 rounding).  51 taps only; ignored by
 * the grad_input path (its result differs per channel through grad_output). */
#define SSTEM_SEPCONV_GRAY_REPLICATED 2u
/* sstem_sepconv_forward_tiled only: output += result (the second frame of the interpolation tail); not with GRAY_REPLICATED */
#define SSTEM_SEPCONV_ACCUMULATE 4u

/*
 * out[b,c,y,x] = sum_{fy,fx} in[b,c,y+fy,x+fx] * v[b,fy,y,x] * h[b,fx,y,x]
 *
 * Replaces SeparableConvolution_cuda_forward(THCudaTensor* input, vertical,
 * horizontal, output) -- libs/sepconv/src/SeparableConvolution_cuda.h:6-11,
 * launcher libs/sepconv/src/SeparableConvolution_kernel.cu:54-73 -- and the CuPy
 * launch in sff_scripts_interp/model/sepconv.py:99-109.
 *   input      [batch, channels, out_h + taps - 1, out_w + taps - 1]
 *   vertical   [batch, taps, out_h, out_w]
 *   horizontal [batch, taps, out_h, out_w]
 *   output     [batch, channels, out_h, out_w]
 * taps: 1..64 (51 is the reference's only value and the tuned path).
 */
int sstem_sepconv_forward(const float* input, const float* vertical, const float* horizontal,
                          float* output,
                          int64_t batch, int64_t channels, int64_t out_h, int64_t out_w,
                          int32_t taps, uint32_t flags, void* stream);

/*
 * Gradients of the above given grad_output [batch, channels, out_h, out_w].
 *
 * Replaces SeparableConvolution_cuda_backward(gradLoss, input, vertical,
 * horizontal, gradInput, gradVertical, gradHorizontal) --
 * libs/sepconv/src/SeparableConvolution_cuda.h:13-21, launcher kernel.cu:152-206.
 * Differences, both deliberate: (1) the channel sum runs over all `channels`
 * (the reference hard-codes 0,1,2 -- kernel.cu:100-108); (2) grad_input is
 * actually computed when non-NULL (the reference leaves it zero --
 * kernel.cu:158 unused, SeparableConvolution.py:60).
 * Any of the three outputs may be NULL = not wanted (ctx.needs_input_grad).
 *   grad_input      [batch, channels, out_h + taps - 1, out_w + taps - 1]
 *   grad_vertical   [batch, taps, out_h, out_w]
 *   grad_horizontal [batch, taps, out_h, out_w]
 */
int sstem_sepconv_backward(const float* grad_output, const float* input,
                           const float* vertical, const float* horizontal,
                           float* grad_input, float* grad_vertical, float* grad_horizontal,
                           int64_t batch, int64_t channels, int64_t out_h, int64_t out_w,
                           int32_t taps, uint32_t flags, void* stream);

/*
 * Fused interpolation tail of the kernel-prediction network -- the expression every IFNet
 * evaluates after its tap branches (sff_scripts_interp/model/model_interp.py:90-97;
 * sp_scripts_train/networks.py:116-123 evaluates it twice):
 *
 *   y      = sepconv(ReplicationPad2d(25)(frame2), k2_vertical, k2_horizontal)
 *          + sepconv(ReplicationPad2d(25)(frame1), k1_vertical, k1_horizontal)
 *   output = mean over channels of y                                  -> [batch, 1, h, w]
 *
 * Replaces, in one launch, two nn.ReplicationPad2d (model_interp.py:46), two
 * SeparableConvolution_cuda_forward calls (SeparableConvolution_cuda.h:6-11), the add and
 * torch.mean(dim=1, keepdim=True) (model_interp.py:94,97).  The padded copies are never
 * materialised, and because the convolution is linear in the image the channel mean is taken on
 * the frames, so one plane per frame is convolved instead of `channels`.
 *   frame1, frame2   [batch, channels, h, w] UNPADDED; planes contiguous, consecutive batches
 *                    `frame_batch_stride` ELEMENTS apart (the callers pass x[:, :3] / x[:, 3:6]
 *                    views of one [batch, 6, h, w] tensor: stride 6*h*w)
 *   k*_vertical / k*_horizontal  [batch, 51, h, w]
 *   output           [batch, 1, h, w]
 * taps must be 51.  flags: SSTEM_SEPCONV_GRAY_REPLICATED = the channel planes of each frame are
 * identical copies (plane 0 is used as is); other flags are rejected.
 */
int sstem_interp_tail_forward(const float* frame1, const float* frame2, int64_t frame_batch_stride,
                              const float* k1_vertical, const float* k1_horizontal,
                              const float* k2_vertical, const float* k2_horizontal,
                              float* output,
                              int64_t batch, int64_t channels, int64_t h, int64_t w,
                              int32_t taps, uint32_t flags, void* stream);

/*
 * Tap gradients of sstem_interp_tail_forward given grad_output [batch, 1, h, w] (what autograd
 * derives from the reference expression: mean -> add -> two SeparableConvolution_cuda_backward
 * calls, SeparableConvolution_cuda.h:13-21).  Any of the four outputs may be NULL = not wanted;
 * the frames are data and get no gradient (as in the reference, whose gradInput stays zero --
 * SeparableConvolution.py:60).
 *   grad_k*_vertical / grad_k*_horizontal  [batch, 51, h, w]
 */
int sstem_interp_tail_backward(const float* grad_output,
                               const float* frame1, const float* frame2, int64_t frame_batch_stride,
                               const float* k1_vertical, const float* k1_horizontal,
                               const float* k2_vertical, const float* k2_horizontal,
                               float* grad_k1_vertical, float* grad_k1_horizontal,
                               float* grad_k2_vertical, float* grad_k2_horizontal,
                               int64_t batch, int64_t channels, int64_t h, int64_t w,
                               int32_t taps, uint32_t flags, void* stream);

/* memory layout of the warp output */
#define SSTEM_LAYOUT_NCHW 0
#define SSTEM_LAYOUT_NHWC 1  /* what the reference materialises (image_warp_torch.py:94,112) */

/*
 * Zero-padded bilinear backward warp, bit-compatible with
 * SpatialTransformation.forward(moving_image, deformation_matrix) --
 * sff_scripts_unfolding/utils/image_warp_torch.py:97-113 (interpolate :32-95):
 *   out[b,c,i,j] = bilinear(zero-padded moving[b,c], x = j + flow[b,i,j,0],
 *                                                    y = i + flow[b,i,j,1])
 * evaluated with the reference's op order and without FMA contraction.
 *   moving [batch, channels, h, w] contiguous
 *   flow   logical shape [batch, h, w, 2] addressed through flow_strides[4]
 *          (in ELEMENTS) -- every reference call site passes a permuted view of
 *          a planar [batch,2,h,w] tensor (sff_scripts_fusion/inference.py:149)
 *   out    [batch, channels, h, w] (NCHW) or [batch, h, w, channels] (NHWC)
 */
int sstem_warp_forward(const float* moving, const float* flow, const int64_t flow_strides[4],
                       float* out,
                       int64_t batch, int64_t channels, int64_t h, int64_t w,
                       int32_t out_layout, void* stream);

/* Backward of sstem_warp_forward (NCHW): the gradients autograd derives through the reference's ATen ops
 * (image_warp_torch.py:32-95; no reference call site needs them).  grad_out [B,C,H,W]; grad_moving [B,C,H,W] (nullable;
 * zero-filled here, then accumulated with atomics: the order of the <= 4 x neighbours adds on an element may vary);
 * grad_flow [B,H,W,2] CONTIGUOUS (nullable). */
int sstem_warp_backward(const float* moving, const float* flow, const int64_t flow_strides[4], const float* grad_out,
                        float* grad_moving, float* grad_flow, int64_t B, int64_t C, int64_t H, int64_t W, void* stream);

/* pixel type of the numpy-semantics warp input */
#define SSTEM_PIX_U8  0
#define SSTEM_PIX_F32 1
#define SSTEM_WARP_BILINEAR 0
#define SSTEM_WARP_NEAREST  1

/*
 * Clamp-border backward warp with the semantics of numpy
 * image_warp(im, flow, mode) -- simu_sff/image_warp.py:3-111 (identical copies
 * under sff_scripts_{unfolding,fusion}/utils/): NHWC image, x1 = clip(x0+1)
 * taken from the clipped x0 (:84-88), weights from frac(flow) (:72-82),
 * 'nearest' = floor (:67-69), result truncated to uint8 (:110).
 *   im        [batch, h, w, channels], uint8 or float32 (pix_type)
 *   flow      [batch, h, w, 2] float32 contiguous (ch0 = x, ch1 = y)
 *   out_u8    [batch, h, w, channels] uint8, may be NULL
 *   out_f32   [batch, h, w, channels] value before the uint8 cast, may be NULL
 */
int sstem_image_warp(const void* im, int32_t pix_type, const float* flow,
                     uint8_t* out_u8, float* out_f32,
                     int64_t batch, int64_t h, int64_t w, int64_t channels,
                     int32_t mode, void* stream);

/*
 * GPU-resident SFF (support-film fold) degradation -- one pass for simu_sff/simuSFF.py:113-121:
 *   flow, mask = gen_flow(h, w, k, b, line_width, fold_width, dis_k)   (simu_sff/flow_synthesis.py:27-83)
 *   deformed   = image_warp(img, flow, mode='bilinear')                (simu_sff/image_warp.py:3-111)
 *   out        = (deformed * mask).astype(np.uint8)
 * bit-equal to the reference's numpy run (FP64 distance field in numpy's operation order, float32
 * flow, numpy-semantics bilinear gather, uint8 truncation).
 *   img      [batch, h, w] uint8 (grayscale sections)
 *   params   DEVICE [batch][8] float64: k, b, sqrt(k*k+1), line_width, fold_width, dis_k,
 *            sin(atan(1/k)), cos(atan(1/k)) -- the scalars flow_synthesis.py:31,64-71 derives with
 *            Python's math module (passed in so the device never re-derives a libm result)
 *   out      [batch, h, w] uint8
 *   flow_out [batch, h, w, 2] float32 or NULL;  mask_out [batch, h, w] uint8 (0/1) or NULL
 *   flow2_out [batch, h, w, 2] float32 or NULL: the second flow of the training data providers'
 *            gen_flow variant (sff_scripts_unfolding/utils/flow_synthesis.py:44-61 -- displacement kept
 *            beyond fold_width, opposite sign; the label of sff_scripts_unfolding/data/data_provider.py:225-239)
 *   stats    DEVICE [batch][2] int64, overwritten: number of zero pixels of `out` (the accept test
 *            of simuSFF.py:125-130) and the sum of its pixels (np.mean for sstem_sff_contrast), both
 *            taken over the pixels at least `stats_border` away from the image border (0 for simuSFF;
 *            the data providers count on the centre crop, data_provider.py:231-238)
 */
int sstem_sff_degrade(const uint8_t* img, const double* params, uint8_t* out, float* flow_out,
                      float* flow2_out, uint8_t* mask_out, int64_t* stats,
                      int64_t batch, int64_t h, int64_t w, int64_t stats_border, void* stream);

/*
 * Regional-contrast step of simuSFF.py:134-144 (`noise`), in place on the image sstem_sff_degrade
 * produced: inside the box p <- uint8(ran * (p - mean) + mean) with mean = np.mean(img); pixels
 * that are 0 stay 0.
 *   img      [batch, h, w] uint8, modified in place
 *   stats    DEVICE [batch][2] int64 as written by sstem_sff_degrade for the same image
 *   params   DEVICE [batch][8] float64: ran_reginal_contrast, box row0, box col0, box height, box
 *            width, 3 unused
 *   max_box_h / max_box_w: largest box of the batch (grid size)
 */
int sstem_sff_contrast(uint8_t* img, const int64_t* stats, const double* params,
                       int64_t batch, int64_t h, int64_t w, int64_t max_box_h, int64_t max_box_w, void* stream);

/*
 * Network input from two uint8 sections, on the device -- sff_scripts_interp/inference.py:69-83:
 *   inputs = concat(repeat(section[k-1], 3), repeat(section[k+1], 3)).astype(float32) / 255.0,
 *   zero-padded by `pad` on every side (F.pad(inputs, (PAD,)*4)).
 *   section_prev, section_next  [batch, h, w] uint8
 *   inputs                      [batch, 6, h + 2*pad, w + 2*pad] float32
 * Bit-equal to the numpy expression; only the uint8 sections have to cross PCIe.
 * section_next == NULL: one section only -> inputs [batch, 3, h + 2*pad, w + 2*pad] (the correction module's
 * input_sff, sff_scripts_fusion/inference.py:127-131,145).
 */
int sstem_sections_to_input(const uint8_t* section_prev, const uint8_t* section_next, float* inputs,
                            int64_t batch, int64_t h, int64_t w, int32_t pad, void* stream);

/*
 * Network output to a uint8 section -- sff_scripts_interp/inference.py:84-88:
 *   section = (F.pad(pred, (-PAD,)*4) * 255).astype(np.uint8)
 *   pred     [batch, 1, h + 2*pad, w + 2*pad] float32
 *   section  [batch, h, w] uint8
 * Values outside [0, 256) convert as C does through int32 (what numpy does on x86-64); NaN / |v| >=
 * 2^31 are unspecified there as well.
 */
int sstem_prediction_to_u8(const float* pred, uint8_t* section, int64_t batch, int64_t h, int64_t w,
                           int32_t pad, void* stream);

/* Output assembly of the correction module -- replaces sff_scripts_fusion/inference.py:163-171:
 *   warped_sff = (warped * 255).astype(np.uint8) -> PIL convert('L');  mask = warped_sff >= 2;
 *   stitch = (img_interp * (1 - mask) + warped_sff * mask).astype(np.uint8)
 * warped: float32 [B,C,H,W] (C = 1 or 3: the SpatialTransformation output), interp: uint8 [B,H,W] (the interpolated
 * section), gray_out (nullable) / stitch_out: uint8 [B,H,W].  H*W must be a multiple of 4.  Bit-equal to numpy + PIL. */
int sstem_warp_stitch_u8(const float* warped, const uint8_t* interp, uint8_t* gray_out, uint8_t* stitch_out,
                         int64_t B, int64_t C, int64_t H, int64_t W, void* stream);

/* The two steps above in ONE kernel: SpatialTransformation(moving, flow) with the stitch assembly as its epilogue (the float32
 * warped image is neither written nor read back).  moving [B,C,H,W] float32 (C = 1 or 3), flow as sstem_warp_forward,
 * interp / gray_out (nullable) / stitch_out uint8 [B,H,W].  Bit-equal to sstem_warp_forward + sstem_warp_stitch_u8.
 * Shapes the TMA kernel does not take (W % 4 != 0, interleaved flow, H*W % 4 != 0 excluded) run the two steps through a
 * stream-ordered scratch image. */
int sstem_warp_stitch_forward(const float* moving, const float* flow, const int64_t flow_strides[4],
                              const uint8_t* interp, uint8_t* gray_out, uint8_t* stitch_out,
                              int64_t B, int64_t C, int64_t H, int64_t W, void* stream);

/*
 * Tile-major taps (SURVEY 8f N2: the layout a tap PRODUCER should emit -- the last Conv2d(51,51,3x3) of
 * IFNet._kernel_module, sff_scripts_interp/model/model_interp.py:129-137, writes [B,51,H,W] today and sepconv re-reads it
 * as 51 x 8 row segments of 32 bytes per 8x8 pixel tile):
 *
 *     tiled[b][ty][tx][tap][row][col] = taps[b][tap][8*ty + row][8*tx + col]     (0 outside the image)
 *     ty < ceil(H/8), tx < ceil(W/8), tap < 51, row < 8, col < 8
 *
 * i.e. all 51 taps of an 8x8 pixel tile are 13 056 contiguous bytes -- one bulk copy for the consuming warp.
 * sstem_taps_tiled_elems: floats to allocate.  sstem_taps_to_tiled: conversion for producers that cannot emit it directly
 * (and for the parity tests).  sstem_sepconv_forward_tiled: the forward of sstem_sepconv_forward with both tap tensors in
 * this layout (K must be 51; flags: SSTEM_SEPCONV_GRAY_REPLICATED); results are bit-identical to the [B,51,H,W] path.
 */
int64_t sstem_taps_tiled_elems(int64_t B, int64_t H, int64_t W);
int sstem_taps_to_tiled(const float* taps, float* tiled, int64_t B, int64_t H, int64_t W, void* stream);
int sstem_sepconv_forward_tiled(const float* input, const float* vertical_tiled, const float* horizontal_tiled,
                                float* output, int64_t B, int64_t C, int64_t H, int64_t W,
                                int32_t K, uint32_t flags, void* stream);

/*
 * Gradients of sstem_sepconv_forward_tiled given grad_output [B,C,H,W] (NCHW, as the forward's output).
 *   grad_vertical_tiled / grad_horizontal_tiled: tile-major like the taps, EVERY element written; entries outside the
 *     image are 0 (the forward never reads them)
 *   grad_input [B,C,H+50,W+50] or NULL (computed as sstem_sepconv_backward does; not a tuned path here: the taps are
 *     converted back to [B,51,H,W] in a stream-ordered workspace, 2 x 204 B per pixel, ~816 B per pixel of traffic)
 * Any of the three outputs may be NULL; K must be 51; flags: SSTEM_SEPCONV_GRAY_REPLICATED (same meaning as for
 * sstem_sepconv_backward: t = (sum_c g_c) * in_0).  Tiled pointers 16-byte aligned (SSTEM_E_ALIGN otherwise).
 * With [B,51,H,W] taps that run the same (third-generation) kernel, the tap gradients are bit-identical to
 * sstem_sepconv_backward's.
 */
int sstem_sepconv_backward_tiled(const float* grad_output, const float* input,
                                 const float* vertical_tiled, const float* horizontal_tiled,
                                 float* grad_input, float* grad_vertical_tiled, float* grad_horizontal_tiled,
                                 int64_t B, int64_t C, int64_t H, int64_t W, int32_t K, uint32_t flags, void* stream);

/* inverse of sstem_taps_to_tiled: tile-major -> [B,51,H,W] (the padding entries are ignored) */
int sstem_taps_from_tiled(const float* tiled, float* taps, int64_t B, int64_t H, int64_t W, void* stream);

/*
 * The one-plane frame the interpolation tail convolves when its taps are tile-major (mean_c sepconv(i_c) = sepconv(mean_c i_c);
 * sff_scripts_interp/model/model_interp.py:46, 90-97):  out[b,0,Y,X] = mean_c frame[b,c,clamp(Y-pad),clamp(X-pad)], i.e.
 * channel mean + nn.ReplicationPad2d(pad).  frame [B,C,H,W] with batch stride frame_bstride elements (a channel slice of the
 * network input); out [B,1,H+2 pad,W+2 pad].  SSTEM_SEPCONV_GRAY_REPLICATED: the planes are identical copies, plane 0 is used.
 * The tail is then two sstem_sepconv_forward_tiled calls on one-plane frames, the second with SSTEM_SEPCONV_ACCUMULATE.
 */
int sstem_frame_mean_pad(const float* frame, int64_t frame_bstride, float* out, int64_t B, int64_t C, int64_t H, int64_t W,
                         int32_t pad, uint32_t flags, void* stream);

/*
 * Tap producer (SURVEY 8f N2, producer side): the last two layers of IFNet._kernel_module,
 *     nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True) -> nn.Conv2d(51, 51, 3, 1, 1)
 * (sff_scripts_interp/model/model_interp.py:18, 130-137; four instances per forward, :34-37, :86-89), as one sm_100a
 * kernel: tcgen05 TF32 implicit GEMM (torch runs this layer in TF32 through cuDNN by default), the bilinear upsample
 * folded into the operand producer, the result written [B,cout,H,W] or directly tile-major (SSTEM_TAPCONV_TILED, the
 * layout of sstem_sepconv_forward_tiled; cout must then be 51).
 *
 *   x       [B, cin, h, w]      cin <= 52, cin * h * w < 2^31
 *   weight  [cout, cin, 3, 3]   cout <= 64 (torch's Conv2d.weight); packed once by sstem_tap_conv3x3_pack_weights into
 *                               sstem_tap_conv3x3_packed_elems() floats ([tap][cin chunk of 4 < 13][64][4] + a zero chunk, rounded to TF32)
 *   bias    [cout] or NULL
 *   out     [B, cout, H, W] or tiled; (H, W) = (2h, 2w) with SSTEM_TAPCONV_UPSAMPLE2X, else (h, w)
 *
 * Arithmetic: operands rounded to TF32 (round-to-nearest), products accumulated in fp32 -- the reference layer's own
 * precision class; tests hold it to the TF32 bound against an fp64 restatement, not to bit equality with cuDNN.
 */
#define SSTEM_TAPCONV_UPSAMPLE2X 1u
#define SSTEM_TAPCONV_TILED 2u
int64_t sstem_tap_conv3x3_packed_elems(void);
int sstem_tap_conv3x3_pack_weights(const float* weight, float* packed, int32_t cin, int32_t cout, void* stream);
int sstem_tap_conv3x3(const float* x, const float* packed_weight, const float* bias, float* out,
                      int64_t B, int32_t cin, int32_t cout, int64_t h, int64_t w, uint32_t flags, void* stream);

/*
 * Backward of the tap producer, y = conv3x3(up(x), W) + b as in sstem_tap_conv3x3 (for training IFNet with the producer
 * in the graph).  grad_out is [B,cout,H,W], or tile-major with SSTEM_TAPCONV_TILED (cout == 51: the tap gradients
 * sstem_sepconv_backward_tiled returns; entries outside the image are never read).  Each non-NULL output is overwritten:
 *
 *   grad_x       [B, cin, h, w]      up^T(conv3x3(grad_out, W')), W'[ci][co][ky][kx] = W[co][ci][2-ky][2-kx]: the forward's
 *                                    tcgen05 convolution on W' (packed by sstem_tap_conv3x3_pack_weights_adjoint into
 *                                    sstem_tap_conv3x3_packed_elems() floats), then the adjoint of the align_corners upsample
 *                                    as a gather with the forward's float32 indices and weights (no atomics)
 *   grad_weight  [cout, cin, 3, 3]   sum over pixels of grad_out x up(x) shifted per tap: a persistent tcgen05 TF32 kernel
 *   grad_bias    [cout]              fp32 sum of grad_out over pixels
 *
 * packed_adjoint may be NULL when grad_x is.  cin <= 52, cout <= 52, (cin or cout) * H * W < 2^31.  Operands are rounded to
 * TF32, sums accumulated in fp32; every gradient is run-to-run bit-identical on a given device, and identical for the
 * two layouts of grad_out.  Stream-ordered workspaces: B*cin*H*W floats (grad_x with the upsample) and
 * min(tiles, SMs) * (cout*cin*9 + cout) floats (grad_weight / grad_bias).
 */
int sstem_tap_conv3x3_pack_weights_adjoint(const float* weight, float* packed, int32_t cin, int32_t cout, void* stream);
int sstem_tap_conv3x3_backward(const float* grad_out, const float* x, const float* packed_adjoint,
                               float* grad_x, float* grad_weight, float* grad_bias,
                               int64_t B, int32_t cin, int32_t cout, int64_t h, int64_t w, uint32_t flags, void* stream);

/*
 * Tap branch convolutions: the three half-resolution layers of IFNet._kernel_module in front of the tap producer,
 *     Conv2d(cin, cout, 3, 1, 1) -> ReLU       (sff_scripts_interp/model/model_interp.py:129-137, run at :86-89)
 * as one sm_100a kernel per layer: y = relu?(conv3x3(x, W) + b), stride 1, zero padding 1, no upsample; tcgen05 TF32
 * implicit GEMM with the producer's operand encoding (same arithmetic class as sstem_tap_conv3x3).
 *
 * Chunk-major layout (the activations between the layers): [B][C8/4][h][w][4], C8 = channels rounded up to 8, i.e.
 * element (b, ch, y, x) at ((b * C8/4 + ch/4) * h + y) * w + x) * 4 + ch % 4; sstem_chunked_elems(B, c, h, w) floats.
 * Values are rounded to TF32 (cvt.rna) and the padding channels hold 0.  A chunk-major input must obey both; the kernel
 * writes its chunk-major output that way.
 *
 *   x       [B, cin, h, w] NCHW (converted to chunk-major in a stream-ordered workspace, TF32-rounded), or chunk-major
 *           with SSTEM_BRANCH_IN_CHUNKED (16-byte aligned).  Both give bit-identical results.
 *   weight  [cout, cin, 3, 3], cin <= 64, cout <= 64; packed once by sstem_branch_conv3x3_pack_weights into
 *           sstem_branch_conv3x3_packed_elems() floats ([tap][cin chunk of 4 < 16][64][4], zero padded, rounded to TF32)
 *   bias    [cout] or NULL
 *   out     [B, cout, h, w] NCHW in full fp32, or chunk-major with SSTEM_BRANCH_OUT_CHUNKED (16-byte aligned)
 * SSTEM_BRANCH_RELU applies ReLU (before the TF32 rounding of a chunk-major output).
 */
#define SSTEM_BRANCH_RELU 1u
#define SSTEM_BRANCH_IN_CHUNKED 2u
#define SSTEM_BRANCH_OUT_CHUNKED 4u
int64_t sstem_branch_conv3x3_packed_elems(void);
int sstem_branch_conv3x3_pack_weights(const float* weight, float* packed, int32_t cin, int32_t cout, void* stream);
int64_t sstem_chunked_elems(int64_t B, int64_t c, int64_t h, int64_t w);
int sstem_branch_conv3x3(const float* x, const float* packed_weight, const float* bias, float* out,
                         int64_t B, int32_t cin, int32_t cout, int64_t h, int64_t w, uint32_t flags, void* stream);

/*
 * Backward of one branch convolution, y = relu?(conv3x3(x, W) + b) as in sstem_branch_conv3x3 (for training IFNet with the
 * tap branches in the graph), with the forward's flag bits: SSTEM_BRANCH_RELU masks with y, g = (y <= 0) ? 0 : grad_out
 * (torch's threshold_backward: y == 0 gives 0, a NaN y passes the gradient); SSTEM_BRANCH_IN_CHUNKED says x is chunk-major and
 * SSTEM_BRANCH_OUT_CHUNKED that y is, i.e. the saved activations come in the layouts the forward read and wrote.
 * grad_out is [B, cout, h, w] NCHW.  Each non-NULL output is overwritten:
 *
 *   grad_x       [B, cin, h, w] NCHW   conv3x3(g, W'), W'[ci][co][ky][kx] = W[co][ci][2-ky][2-kx]: the forward's tcgen05
 *                                      convolution on W' (packed by sstem_branch_conv3x3_pack_weights_adjoint into
 *                                      sstem_branch_conv3x3_packed_elems() floats) fed g chunk-major and TF32-rounded
 *   grad_weight  [cout, cin, 3, 3]     sum over pixels of g x x shifted per tap: a persistent tcgen05 TF32 kernel
 *   grad_bias    [cout]                fp32 sum of the unrounded g over pixels
 *
 * y may be NULL without SSTEM_BRANCH_RELU; packed_adjoint may be NULL when grad_x is.  cin, cout <= 64.  Chunk-major
 * pointers 16-byte aligned.  Operands of products are rounded to TF32, sums accumulated in fp32; every gradient is
 * run-to-run bit-identical on a given device and identical for either layout of x and y.  One stream-ordered workspace of
 * B*C8out*h*w (g) + ~64*cout (bias partials) floats, plus B*C8in*h*w (NCHW x, grad_weight) and
 * min(tiles, SMs / (cin > 32 ? 2 : 1)) * cout*cin*9 (grad_weight partials).
 */
int sstem_branch_conv3x3_pack_weights_adjoint(const float* weight, float* packed, int32_t cin, int32_t cout, void* stream);
int sstem_branch_conv3x3_backward(const float* grad_out, const float* y, const float* x, const float* packed_adjoint,
                                  float* grad_x, float* grad_weight, float* grad_bias,
                                  int64_t B, int32_t cin, int32_t cout, int64_t h, int64_t w, uint32_t flags, void* stream);

/*
 * Gray x3 detection on the device, without a host round trip.  Every reference caller feeds sepconv a grayscale section
 * replicated x3 (sff_scripts_interp/data/data_provider.py:136-137, inference.py:71-77): identical channel planes, for which
 * one plane of work gives all outputs (SSTEM_SEPCONV_GRAY_REPLICATED).  These entry points decide that themselves:
 * forward_detect compares the planes with a streaming kernel, writes *gray_flag (DEVICE int32: non-zero = identical planes) and
 * launches BOTH paths, each gated on the flag -- the one that does not apply returns at its first instruction (~3 us);
 * backward_detect reads the flag the forward left.  Results equal those of sstem_sepconv_forward / _backward with the flag
 * set by hand (forward: bit-identical to the general path).  K != 51, C == 1 or STRICT_ORDER: plain general path, flag 0.
 */
int sstem_sepconv_forward_detect(const float* input, const float* vertical, const float* horizontal,
                                 float* output, int64_t B, int64_t C, int64_t H, int64_t W,
                                 int32_t K, uint32_t flags, int32_t* gray_flag, void* stream);
int sstem_sepconv_backward_detect(const float* grad_output, const float* input,
                                  const float* vertical, const float* horizontal,
                                  float* grad_input, float* grad_vertical, float* grad_horizontal,
                                  int64_t B, int64_t C, int64_t H, int64_t W,
                                  int32_t K, uint32_t flags, const int32_t* gray_flag, void* stream);

/*
 * FP32 FMA-pipe probe: runs a register-resident FFMA loop on every SM of the
 * current device and returns the sustained rate in TFLOP/s (2 flop per FMA).
 * bench.py uses it as the measured denominator of the sepconv roofline
 * (MEASURED_PEAKS.json has no fp32 row).  Synchronous.
 */
int sstem_fp32_peak_probe(double* tflops_out, double* sm_mhz_out);

/* counts kernel launches issued through this library by the calling process */
int64_t sstem_launch_count(void);

int sstem_abi_version(void);
const char* sstem_error_string(int code);

#ifdef __cplusplus
}
#endif
#endif /* SSTEM_B200_H_ */
