/*
 * nbc.h -- C-ABI of libnbc.so: the B200 (sm_100a) segmentation hot path of NeuralBarkCalculator.
 *
 * The reference (TortillasAlfred/NeuralBarkCalculator) is pure Python and has no FFI; the functions below are
 * what a ctypes binding for its hot path binds (see INTEGRATION.md).  Each entry cites the reference code it
 * replaces as  file:line  relative to  src/bark_calculator/ .
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its name ends in _host; the caller allocates everything
 *    (the library owns only the opaque nbc_plan and its packed-weight cache);
 *  - every launch function takes the CUDA stream (a cudaStream_t passed as void*) and is asynchronous;
 *  - every function returns 0 on success or a negative nbc_status; nbc_last_error() gives the text
 *    (thread-local).  There is NO CPU fallback: a missing GPU or a non-sm_100 device is an error.
 *  - activations are NHWC 16-bit floats, masks are u8 [N,H,W], logits are f32 planar [N,3,h,w].
 *  - `f16` arguments select the 16-bit storage format of activations and packed weights: 0 = bf16 (default),
 *    1 = IEEE fp16 (same tensor-core rate, 3 more mantissa bits; see DESIGN.md "Numerics").
 */
#ifndef NBC_H_
#define NBC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  NBC_OK = 0,
  NBC_ERR_INVALID = -1,      /* bad argument / unsupported shape */
  NBC_ERR_CUDA = -2,         /* CUDA runtime / driver error */
  NBC_ERR_DEVICE = -3,       /* no CUDA device or not compute capability 10.x */
  NBC_ERR_WORKSPACE = -4,    /* workspace too small */
  NBC_ERR_KERNEL = -5        /* a kernel reported an internal error (pipeline timeout) */
} nbc_status;

typedef struct nbc_plan nbc_plan;

/* ---- library ------------------------------------------------------------------------------------------- */
int nbc_version(void);
const char* nbc_last_error(void);
/* checks that `device` exists and is sm_100 (B200); must succeed before anything else is called */
int nbc_device_check(int device);
/* number of kernels launched by this library in this process since load (bench.py "gpu_launches") */
int64_t nbc_launch_count(void);

/* ---- K1: 4x cubic resize + dark-band trim  (models.py:157-166 trim_black, 191-203 _preprocess_image) ------
 * raw: H x W x 3 u8 with `pitch` bytes per row.  flags: bit0 = channels are BGR, bit1 = rows are bottom-up
 * (a 24-bit BMP pixel array is flags=3), so the BMP is consumed without a host-side decode.
 * Requires H % 4 == 0 and W % 4 == 0 (the 4096^2 -> 1024^2 scan case).  Writes the trimmed image, rows
 * [first,last) of the resized one, contiguously to out (capacity (H/4)*(W/4)*3) and {first,last} to
 * first_last (2 x int32).  Trimming is applied only when the resized image is square (models.py:200). */
size_t nbc_preprocess_workspace_bytes(int H, int W);
int nbc_preprocess_4x_u8(const uint8_t* raw, int H, int W, int64_t pitch, int flags, uint8_t* out,
                         int32_t* first_last, void* workspace, size_t workspace_bytes, void* stream);
/* Same, for a scan whose dark bands never left the host: raw_span points at memory row span_row0 and holds span_rows
 * rows (both multiples of 4); every other row of the H x W image is all zero by definition and is never read.  The
 * result is bit-identical to nbc_preprocess_4x_u8 on the full image (global min / max clip included).
 * nbc_host_zero_row_span (HOST memory, plain C++, no GPU) finds that span: the rows before the first and after the
 * last row with a non-zero byte, widened outwards to whole groups of `group` rows; rows = 0 for an all-zero image. */
int nbc_preprocess_4x_span_u8(const uint8_t* raw_span, int H, int W, int64_t pitch, int flags, int span_row0, int span_rows,
                              uint8_t* out, int32_t* first_last, void* workspace, size_t workspace_bytes, void* stream);
int nbc_host_zero_row_span(const uint8_t* raw, int H, int64_t pitch, int64_t row_bytes, int group, int32_t* row0,
                           int32_t* rows);
/* A CHUNK of n scans in three launches (what the engine issues per ragged batch; the per-scan calls above are n = 1):
 * raw_spans / span_row0 / span_rows are HOST arrays of n entries (device pointers and spans as above; the span arrays may
 * be NULL = whole scans), result i goes to out + i * out_stride_bytes, its {first,last} to first_last + 2 i.
 * workspace >= n * nbc_preprocess_workspace_bytes(H, W). */
int nbc_preprocess_4x_batch_u8(const uint8_t* const* raw_spans, const int32_t* span_row0, const int32_t* span_rows, int n, int H,
                               int W, int64_t pitch, int flags, uint8_t* out, int64_t out_stride_bytes, int32_t* first_last,
                               void* workspace, size_t workspace_bytes, void* stream);
/* General ratio: any H x W image whose larger side exceeds `target` becomes target x target (models.py:194-198,
 * skimage resize order 3, mode 'reflect', no anti-aliasing, clipped to the input range), then trim_black and the
 * float -> u8 rounding -- float64 arithmetic in the order of oracle/preprocess.py::resize_general_f64.  Same flags,
 * outputs and conventions as nbc_preprocess_4x_u8; out capacity target*target*3.
 * The Python mirror (Preprocessor) routes every size other than exactly 4 * target squared to it. */
size_t nbc_preprocess_general_workspace_bytes(int H, int W, int target);
int nbc_preprocess_general_u8(const uint8_t* raw, int H, int W, int64_t pitch, int flags, int target, uint8_t* out,
                              int32_t* first_last, void* workspace, size_t workspace_bytes, void* stream);
/* trim only, for images that need no resize (max dim <= 1024, models.py:194,200) */
int nbc_trim_u8(const uint8_t* img, int H, int W, uint8_t* out, int32_t* first_last, void* workspace,
                size_t workspace_bytes, void* stream);
/* A CHUNK of n raw images of any sizes, each routed as the Python mirror (Preprocessor.preprocess_array) routes it:
 * exactly (4 target)^2 -> the 4x kernels (the span applies); larger side above target -> the general-ratio kernel, then
 * trim; otherwise square -> trim only; otherwise copied unchanged (first = 0, last = H).  descs is a HOST array: `raw` is
 * the device address of memory row span_row0, and the buffer holds span_rows rows (a span other than (0, H) only for a
 * 4x scan; NULL with span_rows = 0 for an all-zero one).  Result i (processed width `target`, or W for an image that is
 * not resized) goes to out + i * out_stride_bytes, its {first,last} to first_last + 2 i; every result equals the
 * per-image entry's byte for byte.  Each kernel family runs once per chunk. */
typedef struct nbc_mixed_desc {
  const uint8_t* raw;
  int32_t H, W;
  int64_t pitch;
  int32_t flags;       /* bit0 = BGR, bit1 = bottom-up */
  int32_t span_row0, span_rows;
  int32_t reserved;
} nbc_mixed_desc;
size_t nbc_preprocess_mixed_workspace_bytes(const nbc_mixed_desc* descs, int n, int target);
int nbc_preprocess_mixed_batch_u8(const nbc_mixed_desc* descs, int n, int target, uint8_t* out, int64_t out_stride_bytes,
                                  int32_t* first_last, void* workspace, size_t workspace_bytes, void* stream);

/* ---- weights: BatchNorm folding + packing  (models.py:113-139; eval-mode BN of torchvision resnet50) --------
 * w: f32 OIHW [Cout,Cin,kh,kw].  gamma/beta/mean/var may be NULL (no BN: scale 1, shift = conv_bias or 0).
 * Output: bf16 [Cout][kh][kw][cin_pad] with w * gamma/sqrt(var+eps) folded in (channels >= Cin zero), and
 * f32 bias[Cout] = beta - mean*gamma/sqrt(var+eps) (+ conv_bias * scale). */
int nbc_fold_bn_pack(const float* w, const float* gamma, const float* beta, const float* mean, const float* var,
                     const float* conv_bias, float eps, int Cout, int Cin, int kh, int kw, int cin_pad, int f16,
                     void* w_packed_bf16, float* bias_out, void* stream);

/* ---- K2: one convolution layer, implicit GEMM  (every nn.Conv2d+BN(+ReLU)(+residual) of models.py:127-139) --
 * y[N,Ho,Wo,Cout] = act( conv(x[N,H,W,Cin], w) + bias (+ residual[N,Ho,Wo,Cout]) ), bf16 NHWC, f32 accumulate.
 * impl: 0 = auto (tcgen05 when the shape allows), 1 = tcgen05/TMEM/TMA kernel, 2 = mma.sync kernel. */
typedef struct {
  int32_t N, H, W, Cin, Cout;
  int32_t kh, kw, stride, pad, dil;
  int32_t relu;
  int32_t impl;
  int32_t f16;
} nbc_conv_desc;
int nbc_conv_bf16(const nbc_conv_desc* desc, const void* x, const void* w_packed, const float* bias,
                  const void* residual, void* y, void* stream);

/* Two sources, one accumulator: y = act(conv(x; w[:, :K1]) + conv1x1(x2; w[:, K1:]) + bias) -- a bottleneck's conv3 with
 * its downsample branch (torchvision Bottleneck.forward: out = conv3(...) ; identity = downsample(x); out += identity)
 * as ONE launch.  desc: the main convolution (stride 1); desc2: a 1x1 convolution (stride 1 or 2, pad 0) of x2 with the
 * same output geometry; w_cat: [Cout][K1 + Cin2] (per output channel: main weights then the second source's). tcgen05 only. */
int nbc_conv_dual_bf16(const nbc_conv_desc* desc, const void* x, const nbc_conv_desc* desc2, const void* x2,
                       const void* w_cat, const float* bias, void* y, void* stream);

/* Weight gradient of the same layer (training path, __main__.py:231-269 backward of every nn.Conv2d):
 * dw[Cout][kh][kw][Cin] (f32) += sum over output pixels of dz[N,Ho,Wo,Cout]^T * x[N,H,W,Cin] (both bf16 NHWC);
 * accumulates into dw (zero it first).  desc.impl: 0 = auto, 1 = tcgen05 (MN-major operands), 2 = mma.sync. */
int nbc_conv_wgrad_bf16(const nbc_conv_desc* desc, const void* dz, const void* x, float* dw, void* stream);

/* ---- stem: ToTensor + Normalize + conv1 7x7/2 + bn1 + relu, then maxpool 3x3/2
 *      (dataset.py:181-190, models.py:233-237, torchvision resnet50 stem) ---------------------------------------
 * img: u8 NHWC [N,H,W,3]; w_stem: f32 [64][7][7][3] BN-folded; out: bf16 NHWC [N,ceil(H/2),ceil(W/2),64]. */
int nbc_stem_u8(const uint8_t* img, int N, int H, int W, const float* mean3_host, const float* std3_host,
                const float* w_stem, const float* bias, void* out, void* stream);
/* same conv on an already normalised f32 NCHW tensor [N,3,H,W] (what nn.Module.forward receives, models.py:33) */
int nbc_stem_f32(const float* x_nchw, int N, int H, int W, const float* w_stem, const float* bias, void* out,
                 void* stream);
/* tensor-core stem (what the plan uses): the image is staged as zero-padded normalised bf16 [N][Hp][Wp][4] in the
 * workspace and the 7x7/2 conv runs as an implicit GEMM (K = 7 rows x 8 px x 4 ch = 224) on tcgen05.
 * w224: bf16 [64][7][8][4] from nbc_stem_pack_weights(w_stem f32 [64][7][7][3] BN-folded). */
size_t nbc_stem_tc_workspace_bytes(int N, int H, int W);
int nbc_stem_pack_weights(const float* w_stem_f32, int f16, void* w224_bf16, void* stream);
int nbc_stem_tc(const void* input, int input_kind, int N, int H, int W, const float* mean3_host,
                const float* std3_host, const void* w224_bf16, const float* bias, int f16, void* workspace,
                size_t workspace_bytes, void* out, void* stream);
int nbc_maxpool3x3s2_bf16(const void* x, int N, int H, int W, int C, int f16, void* y, void* stream);

/* ---- head tail: Dropout(eval)=identity + Conv2d(512,3,1)+bias  (models.py:113-124) -> f32 planar logits ------ */
int nbc_head_1x1(const void* x_bf16, int64_t pixels_per_image, int N, int Cin, int f16, const float* w3xC,
                 const float* bias3, float* logits_planar, void* stream);

/* ---- K3: bicubic upsample (A=-0.75, align_corners=False) + argmax  (models.py:38-41, 270) -----------------------
 * logits: f32 [N,3,h,w] -> mask u8 [N,H,W] (ties -> lowest class).  nbc_upsample_bicubic writes the f32
 * [N,3,H,W] logits instead (what SimpleSegmentationModel.forward returns). */
int nbc_upsample_argmax(const float* logits, int N, int h, int w, int H, int W, uint8_t* mask, void* stream);
int nbc_upsample_bicubic(const float* logits, int N, int C, int h, int w, int H, int W, float* out, void* stream);

/* ragged batch variant: mask canvas u8 [N,Hc,W], image n has heights[n] valid rows (device array); its logits
 * occupy ceil(heights[n]/8) rows of the [N,3,hc,w] logits canvas.  Rows beyond the valid height are not written. */
int nbc_upsample_argmax_ragged(const float* logits, int N, int hc, int w, int Hc, int W, const int32_t* heights,
                               uint8_t* mask, void* stream);
/* heights[n] = last - first from the {first,last}[N] pairs written by nbc_preprocess_4x_u8 (device -> device) */
int nbc_heights_from_first_last(const int32_t* first_last, int N, int32_t* heights, void* stream);

/* ---- K5: small-region removal + class counts  (utils.py:135-148, models.py:273-276, 323-332) ------------------
 * mask u8 [N,H,W] in place; 8-connected; regions with size < threshold are flipped (two-stage, see DESIGN.md).
 * exclude_nodes != 0 rewrites class 2 -> 1 afterwards.  counts: int32 [N,3] pixels per class of the result. */
size_t nbc_ccl_workspace_bytes(int N, int H, int W);
int nbc_remove_small_zones(uint8_t* mask, int N, int H, int W, int threshold, int exclude_nodes, int32_t* counts,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ragged batch variant: only rows [0, heights[n]) of image n take part (labelling, flips and counts) */
int nbc_remove_small_zones_ragged(uint8_t* mask, int N, int Hc, int W, const int32_t* heights, int threshold,
                                  int exclude_nodes, int32_t* counts, void* workspace, size_t workspace_bytes,
                                  void* stream);

/* ---- K4: max-of-class-index weighted cross entropy, forward + backward  (utils.py:151-165) ----------------------
 * logits f32 [N,3,H,W]; target u8 [N,H,W] (target_is_i64: int64); weights f32[3].  loss: f32 scalar (mean over
 * N*H*W); grad (may be NULL): d loss / d logits, f32 [N,3,H,W].  Deterministic two-stage reduction. */
size_t nbc_wce_workspace_bytes(int N, int H, int W);
int nbc_wce_fwd_bwd(const float* logits, const void* target, int target_is_i64, const float* weights3, int N, int H,
                    int W, float* loss, float* grad, void* workspace, size_t workspace_bytes, void* stream);

/* ---- N1: Lovasz-Softmax loss, forward + backward  (lovasz_losses.py:19-31, 162-218; the loss of __main__.py:239) --
 * logits f32 planar [N,3,H,W]; target u8 or int64 [N,H,W] (labels 0..2); classes='present', per_image=False.
 * loss: device scalar; grad (may be NULL): upstream * d loss / d logits, f32 [N,3,H,W].  The per-class descending
 * sort is cub::DeviceRadixSort; everything else (fused softmax + errors, Lovasz gradient, softmax backward) is ours. */
size_t nbc_lovasz_workspace_bytes(int N, int H, int W);
int nbc_lovasz_softmax_fwd_bwd(const float* logits, const void* target, int target_is_i64, int N, int H, int W,
                               float upstream, float* loss, float* grad, void* workspace, size_t workspace_bytes,
                               void* stream);

/* ---- N2: validation metrics  (lovasz_losses.py:54-77 iou / miou; utils.py:201-235 PixelWiseF1) ------------------
 * nbc_argmax3_u8: torch.argmax(logits, 1) of f32 planar [N,3,H,W] (ties -> lowest index) as u8 [N,H,W].
 * nbc_confusion_matrix: cm9[t*3+p] = number of pixels with label t and prediction p (device uint64[9], overwritten);
 * IoU_c = cm[c][c] / (row_c + col_c - cm[c][c]), F1_c = 2 cm[c][c] / (row_c + col_c) follow on the host. */
int nbc_argmax3_u8(const float* logits, int N, int H, int W, uint8_t* out, void* stream);
int nbc_confusion_matrix(const uint8_t* pred, const void* target, int target_is_i64, int64_t n_pixels, uint64_t* cm9,
                         void* stream);

/* ---- N4: training-time augmentation of a batch  (__main__.py:153-176 get_loader_for_crop_batch; dataset.py:171-193) --
 * images u8 [M,Hs,Ws,3] and their dual label images u8 [M,Hs,Ws] (0/127/255) resident on the device; for each of the B
 * output samples the caller draws the parameters: source index, crop offset (x0, y0) in the pad_resize'd (reflect-padded
 * to target_w x target_h; the differences must be even) image, flips, colour-jitter factors and their order.  One fused
 * gather: out_images u8 [B,crop,crop,3] (PIL ImageEnhance arithmetic, bit-exact), out_classes u8 [B,crop,crop] =
 * round(ToTensor(jittered dual) * 2).  duals / out_classes may both be NULL. */
typedef struct {
  int32_t src, x0, y0, hflip, vflip, order; /* order: 0 = brightness then saturation, 1 = saturation then brightness */
  float brightness, saturation;             /* factors; <= 0 disables the op */
} nbc_augment_params;
int nbc_augment_batch(const uint8_t* images, const uint8_t* duals, int M, int Hs, int Ws, int target_h, int target_w,
                      int crop, const nbc_augment_params* params, int B, uint8_t* out_images, uint8_t* out_classes,
                      void* stream);
/* Ragged sources with the full pad_resize  (__main__.py:153-176; utils.py:242-247 pad_resize = reflect pad by
 * ceil(d/2) per side, then Pillow's BILINEAR resize to the target).  Sources of different sizes in one canvas:
 * images u8 [M,Hc,Wc,3], duals u8 [M,Hc,Wc] (or NULL), dims int32 [M][2] = (height, width) of source m, which occupies
 * rows [0, height) and columns [0, width) of its slot.  Per source and axis, d = target - size: an even d is reflect
 * padding alone (as nbc_augment_batch); an odd d pads to target + 1 and resizes that axis back to target with Pillow's
 * fixed-point arithmetic (Resample.c: 22 fraction bits, horizontal pass first, the intermediate rounded to u8).
 * resize_tables: device int32 [target_h + target_w][4], the rows of the H axis then of the W axis; row i = {first padded
 * index read, three fixed-point weights} of Pillow's (target + 1 -> target) BILINEAR coefficients (float64, converted as
 * trunc(0.5 + k * 2^22)); rows of an axis no source resizes are not read.  Same params and outputs as
 * nbc_augment_batch; x0 / y0 live in the target frame.  dims is read back to the host (M x 8 bytes, which waits for the
 * stream) and a source larger than the target, or whose reflect padding is not narrower than it, is refused with
 * NBC_ERR_INVALID naming the source before anything is launched. */
int nbc_augment_ragged(const uint8_t* images, const uint8_t* duals, int M, int Hc, int Wc, const int32_t* dims, int target_h,
                       int target_w, const int32_t* resize_tables, int crop, const nbc_augment_params* params, int B,
                       uint8_t* out_images, uint8_t* out_classes, void* stream);

/* ---- the whole network  (models.py:27-43 SimpleSegmentationModel.forward, 127-139 fcn_resnet50) ------------------
 * tensors_host: host array of DEVICE pointers to the 326 f32 state_dict tensors in torchvision key order
 * (backbone.conv1.weight, backbone.bn1.{weight,bias,running_mean,running_var,num_batches_tracked}, ...).
 * The plan folds BN, packs bf16 weights (owned by the plan) and keeps nothing else. */
nbc_plan* nbc_plan_create(const void* const* tensors_host, int n_tensors, const float* mean3_host,
                          const float* std3_host, int f16);
void nbc_plan_destroy(nbc_plan* plan);
size_t nbc_plan_workspace_bytes(const nbc_plan* plan, int N, int H, int W);
/* input_kind 0: images u8 NHWC [N,H,W,3] (normalised inside with the plan's mean/std);
 * input_kind 1: f32 NCHW [N,3,H,W] already normalised.  -> lowres_logits f32 [N,3,ceil(H/8),ceil(W/8)] */
int nbc_plan_forward(nbc_plan* plan, const void* input, int input_kind, int N, int H, int W, float* lowres_logits,
                     void* workspace, size_t workspace_bytes, void* stream);
/* Ragged batch: N images of different heights in one canvas u8 [N,Hc,W,3]; image n occupies rows [0, height_n).
 * Heights are read ON THE DEVICE -- either heights[N] or the {first,last}[N] pairs written by nbc_preprocess_4x_u8
 * (exactly one of the two non-NULL) -- so a whole batch is enqueued without a host round trip.  Every layer treats
 * rows >= its per-image valid height as the conv zero padding (tiles beyond are skipped), which makes each image's
 * logits bit-identical to running it alone.  lowres_logits: f32 [N,3,ceil(Hc/8),ceil(W/8)], valid rows only. */
int nbc_plan_forward_ragged(nbc_plan* plan, const uint8_t* canvas, int N, int Hc, int W, const int32_t* heights,
                            const int32_t* first_last, float* lowres_logits, void* workspace,
                            size_t workspace_bytes, void* stream);
/* per-layer timing of the last shape (debug / profiling): runs the forward with events around every layer;
 * ms_out[n_layers] and flops_out[n_layers] (may be NULL); returns number of layers or <0 */
int nbc_plan_profile(nbc_plan* plan, const void* input, int input_kind, int N, int H, int W, float* lowres_logits,
                     void* workspace, size_t workspace_bytes, void* stream, float* ms_out, double* flops_out,
                     int max_layers);
/* conv implementation used by the plan: 0 auto, 1 force tcgen05 where legal, 2 force mma.sync */
int nbc_plan_set_impl(nbc_plan* plan, int impl);
/* Test / debug hooks.  nbc_plan_set_stop(k): the forwards that follow (nbc_plan_forward, nbc_plan_forward_ragged) run
 * steps 0..k of the launch list and return; k < 0 runs all of them (the default).  Every launch up to step k is made as
 * in a full forward, programmatic dependent launch included.  No input of a step (x, x2, residual, the stem's staging
 * image) is the buffer the step writes, so a forward stopped at k leaves step k's operands and its output in the
 * workspace.  nbc_plan_num_steps / nbc_plan_step_info describe the launch list of the most recent forward. */
typedef struct {
  char name[24];
  int32_t kind;       /* 0 stem on CUDA cores, 5 stem on tensor cores (staging pass + implicit GEMM), 1 maxpool,
                         2 conv on tcgen05, 3 conv on mma.sync, 4 head 1x1 (f32 logits) */
  /* tcgen05 kernel variant (0 for the other kinds): CTA pairs, the 64->64 3x3 halo kernel, the stem halo kernel, a second
     source (conv3 + downsample), output channels per tile, K per stage, output staging buffers */
  int32_t pair, halo3, stem_halo, dual, block_n, kblk, out_bufs;
  int32_t ragged_map; /* -1 dense batch (or no tile walk), 1 compact tile map, 0 dense tile numbering, dead tiles skipped */
  int32_t N, H, W, Cin, Cout, k, stride, pad, dil, relu;   /* input geometry of the step */
  int32_t H2, W2, Cin2, stride2;                         /* dual: the second source (1x1, pad 0); 0 otherwise */
  int32_t level;      /* ragged batch: row of the level table with the valid OUTPUT rows of the step; -1 dense */
  /* byte offsets into the workspace, -1 for none.  The stem's x is its staging image (tensor-core stem only; its
     input is the caller's image), head1x1's y is the caller's logits. */
  int64_t x, x2, residual, y, levels;
} nbc_plan_step;
int nbc_plan_set_stop(nbc_plan* plan, int k);
int nbc_plan_num_steps(const nbc_plan* plan);
int nbc_plan_step_info(const nbc_plan* plan, int i, nbc_plan_step* out);

/* ---- training step  (__main__.py:231-269: train-mode forward, loss, backward, Adam; utils.py:151-165 as the loss) ----
 * A plan is built for a fixed (N, H, W).  All state is caller-allocated and flat:
 *   params / grads / adam_m / adam_v : f32[nbc_train_param_count]   (conv weights in [Cout][kh][kw][Cin] order)
 *   stats                            : f32[nbc_train_stats_count]   (BatchNorm running mean / var)
 * nbc_train_exchange converts between the 326 state_dict tensors (torchvision order, OIHW) and the flat buffers:
 * direction 0 loads tensors -> (params, stats), 1 stores (params, stats) -> tensors.  Storing the gradient buffer
 * gives per-layer gradients in state_dict layout (stats = NULL).
 * nbc_train_forward_backward: input_kind 0 = u8 NHWC images (normalised inside), 1 = f32 NCHW; target u8 [N,H,W];
 * BatchNorm uses batch statistics and updates `stats` (momentum 0.1) unless stats is NULL; dropout_p applies to the
 * head (mask = hash(seed, index)); loss = mean weighted CE (device scalar); grads are overwritten.
 * Data-parallel training: all-reduce `grads` (sum) across ranks, then nbc_train_adam with grad_scale = 1/world.
 * nbc_train_adam follows torch.optim.Adam (L2 weight decay added to the gradient, bias correction by `step` >= 1). */
typedef struct nbc_train_plan nbc_train_plan;
nbc_train_plan* nbc_train_create(int N, int H, int W);
void nbc_train_destroy(nbc_train_plan* plan);
int64_t nbc_train_param_count(const nbc_train_plan* plan);
int64_t nbc_train_stats_count(const nbc_train_plan* plan);
size_t nbc_train_workspace_bytes(const nbc_train_plan* plan);
int nbc_train_exchange(nbc_train_plan* plan, void* const* tensors_host, int n_tensors, float* params, float* stats,
                       int direction, void* stream);
int nbc_train_forward_backward(nbc_train_plan* plan, float* params, float* stats, float* grads, const void* input,
                               int input_kind, const float* mean3_host, const float* std3_host, const uint8_t* target,
                               const float* weights3, float dropout_p, uint64_t seed, float* loss, void* workspace,
                               size_t workspace_bytes, void* stream);
/* Gradient-ready events, for overlapping the data-parallel all-reduce (SURVEY.md 8e) with the backward.  The flat
 * gradient buffer becomes final in SEGMENTS, last layer first: segment 0 = head conv + classifier, then the 16 bottleneck
 * blocks last to first, then the stem.  nbc_train_segment gives segment i's range (in floats);
 * nbc_train_wait_segment makes `stream` wait (cudaStreamWaitEvent) until segment i of the most recently enqueued
 * nbc_train_forward_backward is final -- the caller then all-reduces that range on `stream` while the backward of the
 * earlier layers is still running. */
int nbc_train_num_segments(const nbc_train_plan* plan);
int nbc_train_segment(const nbc_train_plan* plan, int i, int64_t* offset, int64_t* count);
int nbc_train_wait_segment(nbc_train_plan* plan, int i, void* stream);
/* test / debug accessors: workspace byte offset + {N,H,W,C} of an intermediate (what: 0 z of unit, 1 y of unit,
 * 2 low-res logits, 3 full-res logits, 4 dL/dfull, 5 dL/dlow); units are in state_dict order (0 = stem).
 * what 6 / 7 = dy / dz of the BatchNorm backward of unit `index` (bf16 NHWC, the geometry of z): byte offsets into the
 * CAPTURE buffer, not the workspace; they hold data only for a step run with capture on. */
int64_t nbc_train_debug_offset(const nbc_train_plan* plan, int what, int index, int32_t* dims_out);
/* Capture for tests: with a device buffer of >= nbc_train_capture_bytes set, every nbc_train_forward_backward copies the
 * dy its BatchNorm backward consumes and the dz it produces, per unit, into `buf` (cudaMemcpyAsync on the step's stream).
 * The backward reuses its gradient buffers, so these are gone otherwise.  buf = NULL turns capture off (the default). */
size_t nbc_train_capture_bytes(const nbc_train_plan* plan);
int nbc_train_set_capture(nbc_train_plan* plan, void* buf, size_t bytes);
int nbc_train_num_units(const nbc_train_plan* plan);
/* weight-gradient kernels used by the plan: 0 = tcgen05 (default), 1 = mma.sync / CUDA-core cross-check kernels */
int nbc_train_set_wgrad_impl(nbc_train_plan* plan, int impl);
/* loss of the step: 0 = CustomWeightedCrossEntropy (utils.py:151-165, default), 1 = LovaszSoftmax (__main__.py:239),
 * 2 = MixedLoss = CE / 4 + Lovasz (utils.py:185-192) */
int nbc_train_set_loss(nbc_train_plan* plan, int kind);
int nbc_train_adam(float* params, const float* grads, float* adam_m, float* adam_v, int64_t n, float lr, float beta1,
                   float beta2, float eps, float weight_decay, int step, float grad_scale, void* stream);

/* ---- result files (host side; SURVEY.md 8f N3) -----------------------------------------------------------------
 * The PNG image data of the files the hot path writes: processed/ RGB images (reference models.py:203, skimage imsave)
 * and the 0/127/255 dual images (models.py:349-356, PIL save).  nbc_png_idat produces the complete zlib stream of ONE
 * IDAT chunk (PNG filter Sub for 3 channels, None for 1; run-length matches + per-segment dynamic Huffman codes) from
 * an 8-bit image in HOST memory -- chunk framing and CRC-32 are the caller's.  Pure host code: no GPU, no stream.
 * pixels: [height][row_stride_bytes] with width*channels meaningful bytes per row (row_stride_bytes 0 = dense);
 * lut256 (1 channel only, may be NULL): every pixel goes through this 256-entry table first -- the dual image
 * 0/127/255 straight from the class mask (models.py:349-353).  out_cap >= nbc_png_idat_bound().
 * Returns the number of bytes written, or a negative NBC_ERR_* status. */
size_t nbc_png_idat_bound(int height, int width, int channels);
int64_t nbc_png_idat(const uint8_t* pixels, int height, int width, int channels, int64_t row_stride_bytes,
                     const uint8_t* lut256, uint8_t* out, size_t out_cap);
/* Stand-in for the reference's two-panel figure under results/combined_images (models.py:280-347; matplotlib is not a
 * dependency): canvas[strip_h + (height+1)/2][2*((width+1)/2) + gap][3] = the title strip the caller rendered
 * (strip[strip_h][same width][3]) above the processed image and the class mask (colours[3 classes][3]) side by side at
 * half resolution, `gap` white columns between them.  Host memory only. */
int nbc_compose_combined(const uint8_t* proc_rgb, const uint8_t* mask, int height, int width, const uint8_t* colours,
                         const uint8_t* strip, int strip_h, int gap, uint8_t* canvas);

#ifdef __cplusplus
}
#endif
#endif /* NBC_H_ */
