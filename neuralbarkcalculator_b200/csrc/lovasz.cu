// N1 -- Lovasz-Softmax loss, forward + backward (the loss the reference's training script really uses:
// __main__.py:239 `loss_function=LovaszSoftmax()`; lovasz_losses.py:19-31 lovasz_grad, 162-218 LovaszSoftmax /
// lovasz_softmax / lovasz_softmax_flat with classes='present', per_image=False), and
// N2 -- the confusion matrix behind the validation metrics iou / miou (lovasz_losses.py:54-77) and PixelWiseF1
// (utils.py:201-235).
//
// Per class c with at least one pixel of that label (over the WHOLE batch):
//   e_i = |[t_i == c] - softmax(logits_i)_c|,  sorted descending;  with fg the sorted indicator, G = sum fg,
//   J_i = 1 - (G - cumsum(fg)_i) / (G + cumsum(1 - fg)_i),  g_i = J_i - J_{i-1} (g_0 = J_0),  loss_c = sum e_i g_i
// loss = mean over present classes.  d loss / d e at the ORIGINAL pixel is g at its rank (the permutation is constant
// for autograd), d e / d p_c = -1 on foreground, +1 elsewhere, then the softmax Jacobian.
//   K_a  one pass: softmax, the three error arrays, packed (index | fg << 31) payloads, per-class label counts
//   sort : cub::DeviceRadixSort::SortPairsDescending (library primitive, one call per class)
//   scan : cub::DeviceScan::InclusiveSum of fg in sorted order (exact integer counts: the reference's f32 cumsum of
//          0/1 values is exact below 2^24 pixels, and equal to these)
//   K_c  Lovasz gradient at every rank, loss partials (deterministic two-stage sum), scatter g to the pixel
//   K_d  per pixel: recompute softmax, combine the three classes, softmax backward -> d loss / d logits (planar f32)
#include <cub/cub.cuh>
#include <thrust/iterator/transform_iterator.h>

#include "loss.cuh"

namespace nbc {

template <typename T>
__global__ void __launch_bounds__(kLvThreads) lovasz_errors_kernel(const float* __restrict__ logits, const T* __restrict__ target,
                                                                   int64_t HW, int64_t P, float* __restrict__ keys /* [3][P] */,
                                                                   uint32_t* __restrict__ vals /* [3][P] */, LovaszHeader* hdr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int t = -1;
  if (i < P) {
    const int64_t n = i / HW, hw = i - n * HW;
    const float* l = logits + n * 3 * HW + hw;
    float p[3];
    softmax3(__ldg(l), __ldg(l + HW), __ldg(l + 2 * HW), p);
    t = (int)target[i];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const bool fg = (t == c);
      keys[(int64_t)c * P + i] = lovasz_error(p[c], fg);
      vals[(int64_t)c * P + i] = (uint32_t)i | (fg ? 0x80000000u : 0u);
    }
  }
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int k = __popc(__ballot_sync(0xffffffffu, t == c));
    if (lane == 0 && k) atomicAdd(&hdr->gts[c], k);
  }
}

// rank i of class c: Lovasz gradient, loss partial, scatter to the pixel
__global__ void __launch_bounds__(kLvThreads) lovasz_grad_kernel(const float* __restrict__ e_sorted, const uint32_t* __restrict__ v_sorted,
                                                                 const uint32_t* __restrict__ cum, int64_t P, int c,
                                                                 const LovaszHeader* __restrict__ hdr, float* __restrict__ ge /* [P] of class c */,
                                                                 float* __restrict__ partial) {
  __shared__ float s_part[kLvThreads / 32];
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int G = hdr->gts[c];
  float contrib = 0.f;
  if (i < P && G > 0) {
    const uint32_t v = v_sorted[i];
    const uint32_t fg = v >> 31;
    const uint32_t cf = cum[i];
    const float g = lovasz_rank_grad(G, i, cf, fg);
    contrib = e_sorted[i] * g;
    ge[v & 0x7FFFFFFFu] = g;
  }
  const float s = lovasz_block_sum(contrib, s_part);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

// sums the block partials of one class in double (one block), fixed order
__global__ void __launch_bounds__(256) lovasz_class_sum(const float* __restrict__ partial, int nblocks, int c, LovaszHeader* hdr) {
  __shared__ double s[256];
  const float sum = lovasz_partials_sum(partial, nblocks, s);
  if (threadIdx.x == 0) hdr->loss[c] = sum;
}

__global__ void lovasz_finish(const LovaszHeader* __restrict__ hdr, float* __restrict__ loss_out) {
  *loss_out = lovasz_present_mean(hdr->gts, hdr->loss);
}

// out[i] = scale_a * a[i] + scale_b * b[i]   (MixedLoss: CE / 4 + Lovasz, utils.py:185-192)
__global__ void __launch_bounds__(256) axpby_kernel(const float* __restrict__ a, float sa, const float* __restrict__ b, float sb,
                                                    int64_t n, float* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = sa * a[i] + sb * b[i];
}

template <typename T>
__global__ void __launch_bounds__(kLvThreads) lovasz_backward_kernel(const float* __restrict__ logits, const T* __restrict__ target,
                                                                     int64_t HW, int64_t P, const float* __restrict__ ge /* [3][P] */,
                                                                     const LovaszHeader* __restrict__ hdr, float upstream,
                                                                     float* __restrict__ grad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  const int64_t n = i / HW, hw = i - n * HW;
  const float* l = logits + n * 3 * HW + hw;
  float p[3];
  softmax3(__ldg(l), __ldg(l + HW), __ldg(l + 2 * HW), p);
  const int t = (int)target[i];
  int np = 0;
#pragma unroll
  for (int c = 0; c < 3; ++c) np += hdr->gts[c] > 0 ? 1 : 0;
  const float inv = np > 0 ? upstream / (float)np : 0.f;
  float dp[3], dot = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float d = 0.f;
    if (hdr->gts[c] > 0) d = ge[(int64_t)c * P + i] * (t == c ? -inv : inv);
    dp[c] = d;
    dot = fmaf(p[c], d, dot);
  }
  float* g = grad + n * 3 * HW + hw;
#pragma unroll
  for (int c = 0; c < 3; ++c) g[(int64_t)c * HW] = p[c] * (dp[c] - dot);
}

__global__ void __launch_bounds__(256) argmax3_kernel(const float* __restrict__ logits, int64_t HW, int64_t P, uint8_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  const int64_t n = i / HW, hw = i - n * HW;
  const float* l = logits + n * 3 * HW + hw;
  const float a = __ldg(l), b = __ldg(l + HW), c = __ldg(l + 2 * HW);
  int arg = 0;
  float best = a;
  if (b > best) best = b, arg = 1;      // ties -> lowest index, as torch.argmax
  if (c > best) arg = 2;
  out[i] = (uint8_t)arg;
}

// cm[t * 3 + p] += 1 for every pixel with label t and prediction p (values > 2 are ignored)
template <typename T>
__global__ void __launch_bounds__(256) confusion_kernel(const uint8_t* __restrict__ pred, const T* __restrict__ target, int64_t P,
                                                        unsigned long long* __restrict__ cm) {
  __shared__ unsigned int s_cm[9];
  if (threadIdx.x < 9) s_cm[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x; i0 < P; i0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = i0 + threadIdx.x;
    int bin = -1;
    if (i < P) {
      const int t = (int)target[i], p = (int)pred[i];
      if (t >= 0 && t < 3 && p < 3) bin = t * 3 + p;
    }
#pragma unroll
    for (int b = 0; b < 9; ++b) {
      const int k = __popc(__ballot_sync(0xffffffffu, bin == b));
      if (lane == 0 && k) atomicAdd(&s_cm[b], (unsigned int)k);
    }
  }
  __syncthreads();
  if (threadIdx.x < 9 && s_cm[threadIdx.x]) atomicAdd(cm + threadIdx.x, (unsigned long long)s_cm[threadIdx.x]);
}

struct LovaszLayout {
  size_t hdr, keys_in, keys_out, vals_in, vals_out, cum, ge, partial, cub_temp, cub_bytes, total;
};

static LovaszLayout lovasz_layout(int64_t P) {
  LovaszLayout L;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += align_up(bytes, 256);
    return o;
  };
  L.hdr = take(sizeof(LovaszHeader));
  L.keys_in = take((size_t)3 * P * 4);
  L.vals_in = take((size_t)3 * P * 4);
  L.keys_out = take((size_t)P * 4);
  L.vals_out = take((size_t)P * 4);
  L.cum = take((size_t)P * 4);
  L.ge = take((size_t)3 * P * 4);
  L.partial = take((size_t)ceil_div64(P, kLvThreads) * 4);
  size_t sort_bytes = 0, scan_bytes = 0;
  cub::DeviceRadixSort::SortPairsDescending(nullptr, sort_bytes, (const float*)nullptr, (float*)nullptr, (const uint32_t*)nullptr,
                                            (uint32_t*)nullptr, (int)P);
  auto it = thrust::make_transform_iterator((const uint32_t*)nullptr, FgOf());
  cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, it, (uint32_t*)nullptr, (int)P);
  L.cub_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
  L.cub_temp = take(L.cub_bytes);
  L.total = off;
  return L;
}

template <typename T>
static int lovasz_impl(const float* logits, const T* target, int N, int H, int W, float upstream, float* loss, float* grad,
                       void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  const int64_t HW = (int64_t)H * W, P = (int64_t)N * HW;
  NBC_REQUIRE(P < (1ll << 31), "nbc_lovasz_softmax: N*H*W must be < 2^31");
  const LovaszLayout L = lovasz_layout(P);
  if (workspace_bytes < L.total) {
    set_error("nbc_lovasz_softmax: workspace %zu < %zu", workspace_bytes, L.total);
    return NBC_ERR_WORKSPACE;
  }
  char* ws = reinterpret_cast<char*>(workspace);
  LovaszHeader* hdr = reinterpret_cast<LovaszHeader*>(ws + L.hdr);
  float* keys_in = reinterpret_cast<float*>(ws + L.keys_in);
  uint32_t* vals_in = reinterpret_cast<uint32_t*>(ws + L.vals_in);
  float* keys_out = reinterpret_cast<float*>(ws + L.keys_out);
  uint32_t* vals_out = reinterpret_cast<uint32_t*>(ws + L.vals_out);
  uint32_t* cum = reinterpret_cast<uint32_t*>(ws + L.cum);
  float* ge = reinterpret_cast<float*>(ws + L.ge);
  float* partial = reinterpret_cast<float*>(ws + L.partial);
  const int blocks = (int)ceil_div64(P, kLvThreads);
  NBC_CUDA(cudaMemsetAsync(hdr, 0, sizeof(LovaszHeader), stream));
  lovasz_errors_kernel<T><<<blocks, kLvThreads, 0, stream>>>(logits, target, HW, P, keys_in, vals_in, hdr);
  NBC_CHECK_LAUNCH();
  for (int c = 0; c < 3; ++c) {
    size_t tb = L.cub_bytes;
    NBC_CUDA(cub::DeviceRadixSort::SortPairsDescending(ws + L.cub_temp, tb, keys_in + (int64_t)c * P, keys_out,
                                                       vals_in + (int64_t)c * P, vals_out, (int)P, 0, 32, stream));
    count_launch(4);
    auto it = thrust::make_transform_iterator((const uint32_t*)vals_out, FgOf());
    tb = L.cub_bytes;
    NBC_CUDA(cub::DeviceScan::InclusiveSum(ws + L.cub_temp, tb, it, cum, (int)P, stream));
    count_launch(2);
    lovasz_grad_kernel<<<blocks, kLvThreads, 0, stream>>>(keys_out, vals_out, cum, P, c, hdr, ge + (int64_t)c * P, partial);
    NBC_CHECK_LAUNCH();
    lovasz_class_sum<<<1, 256, 0, stream>>>(partial, blocks, c, hdr);
    NBC_CHECK_LAUNCH();
  }
  lovasz_finish<<<1, 1, 0, stream>>>(hdr, loss);
  NBC_CHECK_LAUNCH();
  if (grad != nullptr) {
    lovasz_backward_kernel<T><<<blocks, kLvThreads, 0, stream>>>(logits, target, HW, P, ge, hdr, upstream, grad);
    NBC_CHECK_LAUNCH();
  }
  return 0;
}

int axpby(const float* a, float sa, const float* b, float sb, int64_t n, float* out, cudaStream_t stream) {
  const int64_t want = ceil_div64(n, 256);
  axpby_kernel<<<(int)(want < 148 * 16 ? (want < 1 ? 1 : want) : 148 * 16), 256, 0, stream>>>(a, sa, b, sb, n, out);
  NBC_CHECK_LAUNCH();
  return 0;
}

}  // namespace nbc

using namespace nbc;

extern "C" size_t nbc_lovasz_workspace_bytes(int N, int H, int W) {
  const int64_t P = (int64_t)N * H * W;
  if (P <= 0 || P >= (1ll << 31)) return 0;
  return lovasz_layout(P).total;
}

extern "C" int nbc_lovasz_softmax_fwd_bwd(const float* logits, const void* target, int target_is_i64, int N, int H, int W,
                                          float upstream, float* loss, float* grad, void* workspace, size_t workspace_bytes,
                                          void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(logits && target && loss && workspace, "nbc_lovasz_softmax_fwd_bwd: null pointer");
  NBC_REQUIRE(N > 0 && H > 0 && W > 0, "nbc_lovasz_softmax_fwd_bwd: bad shape");
  if (target_is_i64)
    return lovasz_impl<int64_t>(logits, reinterpret_cast<const int64_t*>(target), N, H, W, upstream, loss, grad, workspace,
                                workspace_bytes, stream);
  return lovasz_impl<uint8_t>(logits, reinterpret_cast<const uint8_t*>(target), N, H, W, upstream, loss, grad, workspace,
                              workspace_bytes, stream);
}

extern "C" int nbc_argmax3_u8(const float* logits, int N, int H, int W, uint8_t* out, void* stream_) {
  NBC_REQUIRE(logits && out && N > 0 && H > 0 && W > 0, "nbc_argmax3_u8: bad argument");
  const int64_t HW = (int64_t)H * W, P = (int64_t)N * HW;
  argmax3_kernel<<<(unsigned)ceil_div64(P, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream_)>>>(logits, HW, P, out);
  NBC_CHECK_LAUNCH();
  return 0;
}

extern "C" int nbc_confusion_matrix(const uint8_t* pred, const void* target, int target_is_i64, int64_t n_pixels, uint64_t* cm9,
                                    void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(pred && target && cm9 && n_pixels > 0, "nbc_confusion_matrix: bad argument");
  NBC_CUDA(cudaMemsetAsync(cm9, 0, 9 * sizeof(uint64_t), stream));
  const int64_t want = ceil_div64(n_pixels, 256);
  const int blocks = (int)(want < 148 * 8 ? want : 148 * 8);
  if (target_is_i64)
    confusion_kernel<int64_t><<<blocks, 256, 0, stream>>>(pred, reinterpret_cast<const int64_t*>(target), n_pixels,
                                                           reinterpret_cast<unsigned long long*>(cm9));
  else
    confusion_kernel<uint8_t><<<blocks, 256, 0, stream>>>(pred, reinterpret_cast<const uint8_t*>(target), n_pixels,
                                                           reinterpret_cast<unsigned long long*>(cm9));
  NBC_CHECK_LAUNCH();
  return 0;
}
