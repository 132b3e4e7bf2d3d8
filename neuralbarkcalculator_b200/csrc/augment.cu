// N4 -- training-time augmentation on the GPU, one fused gather pass per batch (reference __main__.py:153-176
// get_loader_for_crop_batch: pad_resize -> ColorJitter(saturation, brightness) -> RandomCrop -> RandomHorizontalFlip ->
// RandomVerticalFlip -> ToTensor, applied with the SAME random draw to the image and to its label image,
// dataset.py:171-179; then target = round(target * 2), dataset.py:184-193).
//
// The random draws are made by the caller (host); this kernel applies them.  For output sample b, pixel (y, x):
//   geometry : flips and crop offset map (y, x) to a row / column of the pad_resize'd source (utils.py:242-247).  Per
//              source and axis, d = target - size: an even d is reflect padding by d/2 alone; an odd d pads ceil(d/2)
//              on both sides (target + 1 long) and Pillow's BILINEAR resize brings the axis back to target
//              (Resample.c: fixed-point taps with 22 fraction bits, horizontal pass first -- Pillow's order unless
//              the target is over 100 times taller than wide, refused here -- the intermediate rounded to u8).  The (target + 1 -> target) tap table of each axis is computed on the host in float64 exactly as
//              Pillow does and passed in; a padded index reaches the source through reflect_index, so an output pixel
//              reads at most 3 x 3 source pixels.
//   colour   : PIL's ImageEnhance arithmetic in explicitly rounded f32 operations, in the drawn order:
//                brightness: out = blend(0, v, f)              saturation: out = blend(L, v, f),
//                L = (19595 R + 38470 G + 7471 B + 0x8000) >> 16    (PIL's ITU-R 601-2 luma)
//                blend(a, v, f) = (uint8) trunc(a + f * (v - a)), clipped to [0, 255] when f is outside [0, 1]
//   label    : the dual image value (0 / 127 / 255, any value after a resize) goes through the SAME geometry and the
//              SAME brightness blend (saturation leaves a grey image unchanged), then class = round(value / 255 * 2)
//              as dataset.py:190-193
// Bytes: reads 4 bytes per output pixel (up to 36 where an axis is resized, mostly from L1) and writes 4 -- a gather;
// the crop is tiny next to a training step.
#include <vector>

#include "common.cuh"

namespace nbc {

struct AugmentParams {   // one per output sample, in device memory (matches nbc_augment_params in nbc.h)
  int32_t src, x0, y0, hflip, vflip, order;   // order: 0 = brightness then saturation, 1 = saturation then brightness
  float brightness, saturation;               // factor; <= 0 disables (a factor of exactly 1 is applied like PIL does)
};

__device__ __forceinline__ int pil_blend(int a, int v, float f) {
  const float t = __fadd_rn(__int2float_rn(a), __fmul_rn(f, __int2float_rn(v - a)));
  if (f >= 0.f && f <= 1.f) return (int)t;          // interpolation: plain truncation (Pillow Blend.c)
  if (t <= 0.f) return 0;
  if (t >= 255.f) return 255;
  return (int)t;
}

__device__ __forceinline__ int reflect_index(int i, int n) {   // numpy / torchvision 'reflect': edge not repeated
  if (n == 1) return 0;
  const int period = 2 * (n - 1);
  i %= period;
  if (i < 0) i += period;
  return i < n ? i : period - i;
}

// Taps of one axis of one output pixel: padded coordinate q (in [0, target)) -> up to 3 source indices and their
// fixed-point weights.  Even d: the padded axis IS the target axis, one tap of weight 1 << 22 (the fixed-point identity,
// exact for any u8).  Odd d: the table row {first padded index, w0, w1, w2} of Pillow's (target + 1 -> target) resize.
struct Taps {
  int n, idx[3], w[3];
};

__device__ __forceinline__ Taps axis_taps(int q, int size, int target, const int4* __restrict__ table) {
  Taps t;
  const int d = target - size;
  if ((d & 1) == 0) {
    t.n = 1, t.idx[0] = reflect_index(q - d / 2, size), t.w[0] = 1 << 22;
  } else {
    const int4 e = table[q];
    const int pad = (d + 1) / 2;
    t.n = 3;
    t.idx[0] = reflect_index(e.x - pad, size), t.idx[1] = reflect_index(e.x + 1 - pad, size);
    t.idx[2] = reflect_index(e.x + 2 - pad, size);
    t.w[0] = e.y, t.w[1] = e.z, t.w[2] = e.w;
  }
  return t;
}

__device__ __forceinline__ int pil_round(int acc) {   // Resample.c clip8: (acc + 2^21 already added) >> 22, clipped
  const int v = acc >> 22;
  return v < 0 ? 0 : (v > 255 ? 255 : v);
}

// dims: int32 [M][2] = (height, width) of each source in the canvas, or NULL = every source is Hc x Wc.
// tables: int4 [target_h + target_w] (rows of the H axis, then of the W axis), or NULL when no axis is odd.
__global__ void __launch_bounds__(256) augment_kernel(const uint8_t* __restrict__ images, const uint8_t* __restrict__ duals,
                                                      int Hc, int Wc, const int2* __restrict__ dims, int target_h,
                                                      int target_w, const int4* __restrict__ tables, int crop,
                                                      const AugmentParams* __restrict__ params, uint8_t* __restrict__ out_img,
                                                      uint8_t* __restrict__ out_cls) {
  const int b = blockIdx.z;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= crop) return;
  const AugmentParams p = params[b];
  const int2 hw = dims != nullptr ? dims[p.src] : make_int2(Hc, Wc);
  // output (y, x) <- flipped crop coordinates <- pad_resize'd coordinates <- source taps
  const int cx = p.hflip ? crop - 1 - x : x, cy = p.vflip ? crop - 1 - y : y;
  const Taps ty = axis_taps(p.y0 + cy, hw.x, target_h, tables);
  const Taps tx = axis_taps(p.x0 + cx, hw.y, target_w, tables + target_h);
  const uint8_t* base = images + (int64_t)p.src * Hc * Wc * 3;
  const uint8_t* dbase = duals != nullptr ? duals + (int64_t)p.src * Hc * Wc : nullptr;
  // Pillow: horizontal pass per source row (rounded to u8), then the vertical pass over those rows
  int accv[4] = {1 << 21, 1 << 21, 1 << 21, 1 << 21};
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    if (j >= ty.n || ty.w[j] == 0) continue;
    int acch[4] = {1 << 21, 1 << 21, 1 << 21, 1 << 21};
    const int64_t row = (int64_t)ty.idx[j] * Wc;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      if (i >= tx.n || tx.w[i] == 0) continue;
      const uint8_t* s = base + (row + tx.idx[i]) * 3;
      acch[0] += tx.w[i] * s[0], acch[1] += tx.w[i] * s[1], acch[2] += tx.w[i] * s[2];
      if (dbase != nullptr) acch[3] += tx.w[i] * dbase[row + tx.idx[i]];
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) accv[c] += ty.w[j] * pil_round(acch[c]);
  }
  int r = pil_round(accv[0]), g = pil_round(accv[1]), bl = pil_round(accv[2]);
  int d = dbase != nullptr ? pil_round(accv[3]) : 0;
#pragma unroll
  for (int step = 0; step < 2; ++step) {
    const bool do_brightness = (step == 0) == (p.order == 0);
    if (do_brightness) {
      if (p.brightness > 0.f) {
        r = pil_blend(0, r, p.brightness), g = pil_blend(0, g, p.brightness), bl = pil_blend(0, bl, p.brightness);
        d = pil_blend(0, d, p.brightness);
      }
    } else if (p.saturation > 0.f) {
      const int L = (19595 * r + 38470 * g + 7471 * bl + 0x8000) >> 16;
      r = pil_blend(L, r, p.saturation), g = pil_blend(L, g, p.saturation), bl = pil_blend(L, bl, p.saturation);
    }
  }
  const int64_t opix = ((int64_t)b * crop + y) * crop + x;
  uint8_t* o = out_img + opix * 3;
  o[0] = (uint8_t)r, o[1] = (uint8_t)g, o[2] = (uint8_t)bl;
  if (out_cls != nullptr) {
    // ToTensor: d / 255 (f32); dataset.py:190-191: * 2, round (half to even, torch.round_)
    const float t = __fmul_rn(__fdiv_rn(__int2float_rn(d), 255.f), 2.f);
    out_cls[opix] = (uint8_t)__float2int_rn(t);
  }
}

static int launch_augment(const uint8_t* images, const uint8_t* duals, int Hc, int Wc, const int32_t* dims, int target_h,
                          int target_w, const int32_t* tables, int crop, const nbc_augment_params* params, int B,
                          uint8_t* out_images, uint8_t* out_classes, cudaStream_t stream) {
  dim3 grid(ceil_div(crop, 256), crop, B);
  augment_kernel<<<grid, 256, 0, stream>>>(images, duals, Hc, Wc, reinterpret_cast<const int2*>(dims), target_h, target_w,
                                           reinterpret_cast<const int4*>(tables), crop,
                                           reinterpret_cast<const AugmentParams*>(params), out_images, out_classes);
  NBC_CHECK_LAUNCH();
  count_launch();
  return 0;
}

}  // namespace nbc

using namespace nbc;

extern "C" int nbc_augment_batch(const uint8_t* images, const uint8_t* duals, int M, int Hs, int Ws, int target_h, int target_w,
                                 int crop, const nbc_augment_params* params, int B, uint8_t* out_images, uint8_t* out_classes,
                                 void* stream_) {
  static_assert(sizeof(nbc_augment_params) == sizeof(AugmentParams), "parameter struct mismatch");
  NBC_REQUIRE(images && params && out_images, "nbc_augment_batch: null pointer");
  NBC_REQUIRE((duals == nullptr) == (out_classes == nullptr), "nbc_augment_batch: duals and out_classes go together");
  NBC_REQUIRE(M > 0 && Hs > 0 && Ws > 0 && B > 0 && crop > 0 && B <= 65535 && crop <= 65535, "nbc_augment_batch: bad shape");
  NBC_REQUIRE(target_h >= Hs && target_w >= Ws && (target_h - Hs) % 2 == 0 && (target_w - Ws) % 2 == 0,
              "nbc_augment_batch: pad_resize(%d, %d) of a %dx%d image needs a real resize (odd or negative difference); only "
              "reflect padding is built here (nbc_augment_ragged has the resize)", target_w, target_h, Ws, Hs);
  NBC_REQUIRE(crop <= target_h && crop <= target_w, "nbc_augment_batch: crop %d larger than the padded image", crop);
  NBC_REQUIRE((target_h - Hs) / 2 < Hs && (target_w - Ws) / 2 < Ws, "nbc_augment_batch: reflect padding wider than the image");
  return launch_augment(images, duals, Hs, Ws, nullptr, target_h, target_w, nullptr, crop, params, B, out_images, out_classes,
                        reinterpret_cast<cudaStream_t>(stream_));
}

extern "C" int nbc_augment_ragged(const uint8_t* images, const uint8_t* duals, int M, int Hc, int Wc, const int32_t* dims,
                                  int target_h, int target_w, const int32_t* resize_tables, int crop,
                                  const nbc_augment_params* params, int B, uint8_t* out_images, uint8_t* out_classes,
                                  void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(images && dims && resize_tables && params && out_images, "nbc_augment_ragged: null pointer");
  NBC_REQUIRE((duals == nullptr) == (out_classes == nullptr), "nbc_augment_ragged: duals and out_classes go together");
  NBC_REQUIRE(M > 0 && Hc > 0 && Wc > 0 && B > 0 && crop > 0 && B <= 65535 && crop <= 65535 && target_h >= 2 && target_w >= 2,
              "nbc_augment_ragged: bad shape");
  NBC_REQUIRE(crop <= target_h && crop <= target_w, "nbc_augment_ragged: crop %d larger than the %dx%d target", crop, target_w,
              target_h);
  // Pillow runs the vertical pass first for targets about 128 times taller than wide; the kernel has Pillow's order
  // for everything else.
  NBC_REQUIRE(target_h < 64 * target_w, "nbc_augment_ragged: a %dx%d target is too narrow", target_w, target_h);
  // The sizes live on the device: one M x 8-byte read-back (it waits for the stream) so that a bad source is refused
  // before anything is launched.
  std::vector<int32_t> hw(2 * (size_t)M);
  NBC_CUDA(cudaMemcpyAsync(hw.data(), dims, hw.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  NBC_CUDA(cudaStreamSynchronize(stream));
  for (int m = 0; m < M; ++m) {
    const int h = hw[2 * m], w = hw[2 * m + 1];
    NBC_REQUIRE(h > 0 && w > 0 && h <= Hc && w <= Wc, "nbc_augment_ragged: source %d is %dx%d, outside the %dx%d canvas", m, w, h,
                Wc, Hc);
    NBC_REQUIRE(h <= target_h && w <= target_w, "nbc_augment_ragged: source %d (%dx%d) is larger than the %dx%d target", m, w, h,
                target_w, target_h);
    NBC_REQUIRE((target_h - h + 1) / 2 < h && (target_w - w + 1) / 2 < w,
                "nbc_augment_ragged: source %d (%dx%d) needs reflect padding of %d x %d, not narrower than the source", m, w, h,
                (target_w - w + 1) / 2, (target_h - h + 1) / 2);
  }
  return launch_augment(images, duals, Hc, Wc, dims, target_h, target_w, resize_tables, crop, params, B, out_images,
                        out_classes, stream);
}
