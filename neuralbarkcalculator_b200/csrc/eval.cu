// Batched evaluation of a ragged chunk (what the reference's post-training dump computes per image,
// __main__.py:293-437): one call scores every image of a chunk from its low-resolution logits.
//
//   K3 + sink  per full-resolution pixel: bicubic logits (K3's arithmetic), argmax into the mask canvas, the confusion
//              bin (shared-memory bins, one global atomic per bin and block), the weighted-CE term, and the three Lovasz
//              errors as composite u64 keys (segment (image, class) above bit 32, ~bits of the f32 error below) with the
//              (pixel | fg << 31) payload.  The f32 logits at full resolution are never written.
//   sort       ONE cub::DeviceRadixSort::SortPairs over the chunk on 32 + ceil(log2(3N)) bits.  It is stable, errors are
//              fabsf values (no -0, no NaN), so each segment comes out in exactly the order of the per-image
//              SortPairsDescending of lovasz.cu.
//   scan       ONE cub::DeviceScan::InclusiveSum of the fg bits; a segment subtracts the count before its start (exact).
//   Lovasz     per segment, the 256-thread block decomposition of lovasz_grad_kernel relative to the segment start, then
//              lovasz_partials_sum per segment and lovasz_present_mean per image (loss.cuh, shared with lovasz.cu).
//   WCE        per image, the grid-stride double accumulation of wce_kernel on min(ceil(P_n / 256), kWceBlocks) blocks and
//              wce_finish's ordered sum (loss.cuh, shared with wce.cu).
//   K5         nbc_remove_small_zones_ragged (threshold 150, no node rewrite) on the mask canvas, then a ragged per-image
//              confusion matrix.
// Every output therefore equals, bit for bit, what the per-image ops give for that image alone.
#include <cub/cub.cuh>
#include <thrust/iterator/transform_iterator.h>

#include <vector>

#include "k3.cuh"
#include "loss.cuh"

namespace nbc {

constexpr int kEvalThreshold = 150;   // utils.py:135-148, PixelWiseF1's region removal

struct EvalSink {
  static constexpr bool kMask = true;
  const uint8_t* __restrict__ labels;   // [N,Hc,W]
  const int* __restrict__ off;          // [N+1] first compact pixel of each image
  const float* __restrict__ weights;    // [3] class weights of the weighted CE
  int losses, Hc, W;
  float* __restrict__ wce;              // [P] per-pixel weighted-CE term
  uint64_t* __restrict__ keys;          // [3P] segment-major: image n, class c at 3 off[n] + c P_n
  uint32_t* __restrict__ vals;          // [3P]
  unsigned long long* __restrict__ cm;  // [N][9]

  struct Acc {
    uint64_t bins;   // 4 bits per confusion bin: a thread scores at most kK3Rows (8) pixels
  };

  __device__ __forceinline__ void pixel(Acc& acc, int n, int H, int Y, int X, const float (&v)[3], int arg) const {
    const int t = labels[((int64_t)n * Hc + Y) * W + X];
    if (t < 3) acc.bins += 1ull << (4 * (t * 3 + arg));
    const int li = Y * W + X, g = off[n] + li;
    if (losses & 1) {
      float e0, e1, e2, s, w;
      wce[g] = wce_term(v[0], v[1], v[2], t, __ldg(weights), __ldg(weights + 1), __ldg(weights + 2), e0, e1, e2, s, w);
    }
    if (losses & 2) {
      float p[3];
      softmax3(v[0], v[1], v[2], p);
      const int64_t P = (int64_t)H * W, base = 3 * (int64_t)off[n] + li;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const bool fg = (t == c);
        const uint32_t e = __float_as_uint(lovasz_error(p[c], fg));
        keys[base + c * P] = ((uint64_t)(3 * n + c) << 32) | (uint32_t)~e;   // ascending ~e = descending e (e >= +0)
        vals[base + c * P] = (uint32_t)g | (fg ? 0x80000000u : 0u);
      }
    }
  }

  __device__ __forceinline__ void flush(Acc& acc, int n) const {
    __shared__ unsigned int s_cm[9];
    if (threadIdx.x < 9) s_cm[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int b = 0; b < 9; ++b) {
      const unsigned int k = __reduce_add_sync(0xffffffffu, (unsigned int)(acc.bins >> (4 * b)) & 15u);
      if ((threadIdx.x & 31) == 0 && k) atomicAdd(&s_cm[b], k);
    }
    __syncthreads();
    if (threadIdx.x < 9 && s_cm[threadIdx.x]) atomicAdd(cm + n * 9 + threadIdx.x, (unsigned long long)s_cm[threadIdx.x]);
  }
};

__global__ void eval_offsets_kernel(const int* __restrict__ heights, int N, int W, int* __restrict__ off) {
  int acc = 0;
  for (int n = 0; n < N; ++n) off[n] = acc, acc += heights[n] * W;
  off[N] = acc;
}

// segment s = 3 n + c, block b: lovasz_grad_kernel's block b of that image and class, forward only
__global__ void __launch_bounds__(kLvThreads) eval_lovasz_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                                 const uint32_t* __restrict__ cum, const int* __restrict__ off,
                                                                 const unsigned long long* __restrict__ cm, int nbmax,
                                                                 float* __restrict__ partial) {
  __shared__ float s_part[kLvThreads / 32];
  const int s = blockIdx.y, n = s / 3, c = s - 3 * n;
  const int64_t P = off[n + 1] - off[n];
  if ((int64_t)blockIdx.x * kLvThreads >= P) return;     // block-uniform
  const int64_t base = 3 * (int64_t)off[n] + c * P;
  const uint32_t cum0 = base > 0 ? cum[base - 1] : 0u;
  const int G = (int)(cm[n * 9 + c * 3] + cm[n * 9 + c * 3 + 1] + cm[n * 9 + c * 3 + 2]);
  const int64_t i = (int64_t)blockIdx.x * kLvThreads + threadIdx.x;
  float contrib = 0.f;
  if (i < P && G > 0) {
    const uint32_t fg = vals[base + i] >> 31;
    const float g = lovasz_rank_grad(G, i, cum[base + i] - cum0, fg);
    contrib = __uint_as_float(~(uint32_t)keys[base + i]) * g;
  }
  const float sum = lovasz_block_sum(contrib, s_part);
  if (threadIdx.x == 0) partial[(int64_t)s * nbmax + blockIdx.x] = sum;
}

__global__ void __launch_bounds__(256) eval_lovasz_sum(const float* __restrict__ partial, int nbmax, const int* __restrict__ off,
                                                       float* __restrict__ seg_loss) {
  __shared__ double s[256];
  const int seg = blockIdx.x, n = seg / 3;
  const float sum = lovasz_partials_sum(partial + (int64_t)seg * nbmax, ceil_div(off[n + 1] - off[n], kLvThreads), s);
  if (threadIdx.x == 0) seg_loss[seg] = sum;
}

__device__ __forceinline__ int wce_blocks(int P) { return min(ceil_div(P, 256), kWceBlocks); }

// image blockIdx.y: wce_kernel's accumulation on wce_fwd_bwd's grid for that image alone
__global__ void __launch_bounds__(256) eval_wce_kernel(const float* __restrict__ term, const int* __restrict__ off,
                                                       double* __restrict__ partial) {
  __shared__ double s_part[8];
  const int n = blockIdx.y;
  const int64_t P = off[n + 1] - off[n];
  const int nb = wce_blocks((int)P);
  if ((int)blockIdx.x >= nb) return;                      // block-uniform
  const float* t = term + off[n];
  double local = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < P; i += (int64_t)nb * 256) local += (double)t[i];
  const double s = wce_block_sum(local, s_part);
  if (threadIdx.x == 0) partial[(int64_t)n * kWceBlocks + blockIdx.x] = s;
}

__global__ void eval_finish(const int* __restrict__ off, int N, int losses, const unsigned long long* __restrict__ cm,
                            const float* __restrict__ seg_loss, const double* __restrict__ wce_partial,
                            float* __restrict__ loss_wce, float* __restrict__ loss_lovasz) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const int P = off[n + 1] - off[n];
  loss_wce[n] = (losses & 1) ? wce_partials_mean(wce_partial + (int64_t)n * kWceBlocks, wce_blocks(P), 1.0 / (double)P) : 0.f;
  if (losses & 2) {
    int gts[3];
    float l[3];
    for (int c = 0; c < 3; ++c) {
      gts[c] = (int)(cm[n * 9 + c * 3] + cm[n * 9 + c * 3 + 1] + cm[n * 9 + c * 3 + 2]);
      l[c] = seg_loss[3 * n + c];
    }
    loss_lovasz[n] = lovasz_present_mean(gts, l);
  } else {
    loss_lovasz[n] = 0.f;
  }
}

// cm[n][t * 3 + p] over the rows [0, H_n) of image n of the two canvases (confusion_kernel per image)
__global__ void __launch_bounds__(256) eval_confusion_kernel(const uint8_t* __restrict__ pred, const uint8_t* __restrict__ labels,
                                                             int64_t canvas, const int* __restrict__ off,
                                                             unsigned long long* __restrict__ cm) {
  __shared__ unsigned int s_cm[9];
  if (threadIdx.x < 9) s_cm[threadIdx.x] = 0;
  __syncthreads();
  const int n = blockIdx.y;
  const int64_t P = off[n + 1] - off[n];
  const uint8_t* pr = pred + n * canvas;
  const uint8_t* lb = labels + n * canvas;
  const int lane = threadIdx.x & 31;
  for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x; i0 < P; i0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = i0 + threadIdx.x;
    int bin = -1;
    if (i < P) {
      const int t = lb[i], p = pr[i];
      if (t < 3 && p < 3) bin = t * 3 + p;
    }
#pragma unroll
    for (int b = 0; b < 9; ++b) {
      const int k = __popc(__ballot_sync(0xffffffffu, bin == b));
      if (lane == 0 && k) atomicAdd(&s_cm[b], (unsigned int)k);
    }
  }
  __syncthreads();
  if (threadIdx.x < 9 && s_cm[threadIdx.x]) atomicAdd(cm + n * 9 + threadIdx.x, (unsigned long long)s_cm[threadIdx.x]);
}

static int key_bits(int N) {      // bits of the largest segment id 3N - 1
  int b = 1;
  while ((1ll << b) < 3ll * N) ++b;
  return b;
}

struct EvalLayout {
  size_t off, seg_loss, wce_part, lv_part, mask, wce, keys_in, keys_out, vals_in, vals_out, cum, cub, cub_bytes, ccl, total;
  int nbmax;
};

static EvalLayout eval_layout(int N, int Hc, int W) {
  EvalLayout L;
  const int64_t P = (int64_t)N * Hc * W, P3 = 3 * P;
  L.nbmax = ceil_div(Hc * W, kLvThreads);
  size_t o = 0;
  auto take = [&](size_t bytes) {
    const size_t at = o;
    o += align_up(bytes, 256);
    return at;
  };
  L.off = take((size_t)(N + 1) * 4);
  L.seg_loss = take((size_t)3 * N * 4);
  L.wce_part = take((size_t)N * kWceBlocks * 8);
  L.lv_part = take((size_t)3 * N * L.nbmax * 4);
  L.mask = take((size_t)P);
  L.wce = take((size_t)P * 4);
  // the loss buffers below are dead once the reductions have run: K5's workspace reuses them
  L.ccl = o;
  L.keys_in = take((size_t)P3 * 8);
  L.keys_out = take((size_t)P3 * 8);
  L.vals_in = take((size_t)P3 * 4);
  L.vals_out = take((size_t)P3 * 4);
  L.cum = take((size_t)P3 * 4);
  size_t sort_bytes = 0, scan_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr,
                                  (uint32_t*)nullptr, (int)P3, 0, 32 + key_bits(N));
  auto it = thrust::make_transform_iterator((const uint32_t*)nullptr, FgOf());
  cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, it, (uint32_t*)nullptr, (int)P3);
  L.cub_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
  L.cub = take(L.cub_bytes);
  const size_t ccl_end = L.ccl + align_up(nbc_ccl_workspace_bytes(N, Hc, W), 256);
  L.total = o > ccl_end ? o : ccl_end;
  return L;
}

static bool eval_shape_ok(int N, int Hc, int W) {
  return N >= 1 && Hc >= 1 && W >= 1 && 3ll * N <= 65535 && ceil_div(Hc, kK3Rows) <= 65535 && 3ll * N * Hc * W < (1ll << 31);
}

}  // namespace nbc

using namespace nbc;

extern "C" size_t nbc_eval_workspace_bytes(int N, int Hc, int W) {
  if (!eval_shape_ok(N, Hc, W)) return 0;
  return eval_layout(N, Hc, W).total;
}

namespace nbc {
// nbc_eval_ragged on a view set (K3Views, V = 1, 2 or 4, checked by the caller): K3's sink sees the mean of the views
static int eval_ragged_views(const K3Views& views, int V, int N, int Hc, int W, const int32_t* heights, const uint8_t* labels,
                             const float* weights3, int losses, float* loss_wce, float* loss_lovasz, uint64_t* cm_raw,
                             uint64_t* cm_rsz, int32_t* counts, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  NBC_REQUIRE(heights && labels && loss_wce && loss_lovasz && cm_raw && cm_rsz && counts && workspace,
              "nbc_eval_ragged: null pointer");
  NBC_REQUIRE(N >= 1, "nbc_eval_ragged: N must be at least 1 (got %d)", N);
  NBC_REQUIRE(eval_shape_ok(N, Hc, W),
              "nbc_eval_ragged: bad shape N=%d Hc=%d W=%d (3 N Hc W must stay below 2^31, the pixel index of the sort payload "
              "and its item count)", N, Hc, W);
  NBC_REQUIRE(losses >= 0 && losses <= 3, "nbc_eval_ragged: losses is a bitmask of 1 (weighted CE) and 2 (Lovasz), got %d", losses);
  NBC_REQUIRE(weights3 || !(losses & 1), "nbc_eval_ragged: the weighted CE needs class weights");
  const EvalLayout L = eval_layout(N, Hc, W);
  if (workspace_bytes < L.total) {
    set_error("nbc_eval_ragged: workspace %zu < %zu", workspace_bytes, L.total);
    return NBC_ERR_WORKSPACE;
  }
  std::vector<int32_t> hs(N);
  NBC_CUDA(cudaMemcpyAsync(hs.data(), heights, (size_t)N * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  NBC_CUDA(cudaStreamSynchronize(stream));
  for (int n = 0; n < N; ++n)
    NBC_REQUIRE(hs[n] >= 1 && hs[n] <= Hc, "nbc_eval_ragged: image %d has height %d, outside [1, %d]", n, hs[n], Hc);

  char* ws = reinterpret_cast<char*>(workspace);
  int* off = reinterpret_cast<int*>(ws + L.off);
  float* seg_loss = reinterpret_cast<float*>(ws + L.seg_loss);
  double* wce_part = reinterpret_cast<double*>(ws + L.wce_part);
  float* lv_part = reinterpret_cast<float*>(ws + L.lv_part);
  uint8_t* mask = reinterpret_cast<uint8_t*>(ws + L.mask);
  float* wce = reinterpret_cast<float*>(ws + L.wce);
  uint64_t* keys_in = reinterpret_cast<uint64_t*>(ws + L.keys_in);
  uint64_t* keys_out = reinterpret_cast<uint64_t*>(ws + L.keys_out);
  uint32_t* vals_in = reinterpret_cast<uint32_t*>(ws + L.vals_in);
  uint32_t* vals_out = reinterpret_cast<uint32_t*>(ws + L.vals_out);
  uint32_t* cum = reinterpret_cast<uint32_t*>(ws + L.cum);
  unsigned long long* cm0 = reinterpret_cast<unsigned long long*>(cm_raw);
  unsigned long long* cm1 = reinterpret_cast<unsigned long long*>(cm_rsz);

  NBC_CUDA(cudaMemsetAsync(cm_raw, 0, (size_t)N * 9 * sizeof(uint64_t), stream));
  NBC_CUDA(cudaMemsetAsync(cm_rsz, 0, (size_t)N * 9 * sizeof(uint64_t), stream));
  eval_offsets_kernel<<<1, 1, 0, stream>>>(heights, N, W, off);
  NBC_CHECK_LAUNCH();

  const int hc = ((((Hc - 1) / 2 + 1) - 1) / 2 + 1 - 1) / 2 + 1, w = ((((W - 1) / 2 + 1) - 1) / 2 + 1 - 1) / 2 + 1;
  EvalSink sink;
  sink.labels = labels, sink.off = off, sink.weights = weights3, sink.losses = losses, sink.Hc = Hc, sink.W = W;
  sink.wce = wce, sink.keys = keys_in, sink.vals = vals_in, sink.cm = cm0;
  launch_k3(V, views, N, hc, w, Hc, W, 0, heights, mask, sink, stream);
  NBC_CHECK_LAUNCH();

  int total = 0;
  for (int n = 0; n < N; ++n) total += hs[n] * W;
  if (losses & 2) {
    const int items = 3 * total, end_bit = 32 + key_bits(N);
    size_t tb = L.cub_bytes;
    NBC_CUDA(cub::DeviceRadixSort::SortPairs(ws + L.cub, tb, keys_in, keys_out, vals_in, vals_out, items, 0, end_bit, stream));
    count_launch(ceil_div(end_bit, 8));
    auto it = thrust::make_transform_iterator((const uint32_t*)vals_out, FgOf());
    tb = L.cub_bytes;
    NBC_CUDA(cub::DeviceScan::InclusiveSum(ws + L.cub, tb, it, cum, items, stream));
    count_launch(2);
    eval_lovasz_kernel<<<dim3(L.nbmax, 3 * N), kLvThreads, 0, stream>>>(keys_out, vals_out, cum, off, cm0, L.nbmax, lv_part);
    NBC_CHECK_LAUNCH();
    eval_lovasz_sum<<<3 * N, 256, 0, stream>>>(lv_part, L.nbmax, off, seg_loss);
    NBC_CHECK_LAUNCH();
  }
  if (losses & 1) {
    eval_wce_kernel<<<dim3(std::min(ceil_div(Hc * W, 256), kWceBlocks), N), 256, 0, stream>>>(wce, off, wce_part);
    NBC_CHECK_LAUNCH();
  }
  eval_finish<<<ceil_div(N, 128), 128, 0, stream>>>(off, N, losses, cm0, seg_loss, wce_part, loss_wce, loss_lovasz);
  NBC_CHECK_LAUNCH();

  const int rc = nbc_remove_small_zones_ragged(mask, N, Hc, W, heights, kEvalThreshold, 0, counts, ws + L.ccl,
                                               L.total - L.ccl, stream);
  if (rc != 0) return rc;
  eval_confusion_kernel<<<dim3(std::min(ceil_div(Hc * W, 256), kWceBlocks), N), 256, 0, stream>>>(mask, labels, (int64_t)Hc * W,
                                                                                                 off, cm1);
  NBC_CHECK_LAUNCH();
  return 0;
}
}  // namespace nbc

extern "C" int nbc_eval_ragged(const float* logits, int N, int Hc, int W, const int32_t* heights, const uint8_t* labels,
                               const float* weights3, int losses, float* loss_wce, float* loss_lovasz, uint64_t* cm_raw,
                               uint64_t* cm_rsz, int32_t* counts, void* workspace, size_t workspace_bytes, void* stream) {
  NBC_REQUIRE(logits, "nbc_eval_ragged: null pointer");
  return eval_ragged_views(k3_one(logits), 1, N, Hc, W, heights, labels, weights3, losses, loss_wce, loss_lovasz, cm_raw, cm_rsz,
                           counts, workspace, workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int nbc_eval_ragged_views(const float* const* logits, const int32_t* flips, int V, int N, int Hc, int W,
                                     const int32_t* heights, const uint8_t* labels, const float* weights3, int losses,
                                     float* loss_wce, float* loss_lovasz, uint64_t* cm_raw, uint64_t* cm_rsz, int32_t* counts,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  K3Views views;
  const int rc = k3_views_args(logits, flips, V, views, "nbc_eval_ragged_views");
  if (rc != 0) return rc;
  return eval_ragged_views(views, V, N, Hc, W, heights, labels, weights3, losses, loss_wce, loss_lovasz, cm_raw, cm_rsz, counts,
                           workspace, workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
}
