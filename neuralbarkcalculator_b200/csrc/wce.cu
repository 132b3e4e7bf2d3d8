// K4 -- CustomWeightedCrossEntropy forward + backward in one pass (utils.py:151-165).
//
//   ent = CE(logits, target) per pixel; w = weights[max(argmax_c logits, target)]; loss = mean(ent * w)
//   d loss / d logit_c = w * (softmax_c - [c == target]) / (N*H*W)      (w is a constant for autograd)
// The reference runs five separate full-tensor torch ops; here each pixel's three logits are read once
// (planar f32 [N,3,H,W], coalesced per class plane) and the three gradients written once: 25 B/pixel in f32.
// The loss is reduced deterministically: per-block partial sums in double, then one block sums them in order.
#include "loss.cuh"

namespace nbc {

template <typename TargetT>
__global__ void __launch_bounds__(256) wce_kernel(const float* __restrict__ logits, const TargetT* __restrict__ target,
                                                  const float* __restrict__ weights, int64_t HW, int64_t total,
                                                  float inv_total, float* __restrict__ grad,
                                                  double* __restrict__ partial) {
  const float w0 = __ldg(weights), w1 = __ldg(weights + 1), w2 = __ldg(weights + 2);
  double local = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / HW, pix = i - n * HW;
    const float* lp = logits + n * 3 * HW + pix;
    const float l0 = __ldg(lp), l1 = __ldg(lp + HW), l2 = __ldg(lp + 2 * HW);
    const int t = (int)target[i];
    float e0, e1, e2, s, w;
    local += (double)wce_term(l0, l1, l2, t, w0, w1, w2, e0, e1, e2, s, w);
    if (grad) {
      const float k = w * inv_total, inv_s = 1.f / s;
      float* gp = grad + n * 3 * HW + pix;
      gp[0] = k * (e0 * inv_s - (t == 0 ? 1.f : 0.f));
      gp[HW] = k * (e1 * inv_s - (t == 1 ? 1.f : 0.f));
      gp[2 * HW] = k * (e2 * inv_s - (t == 2 ? 1.f : 0.f));
    }
  }
  __shared__ double s_part[8];
  const double s = wce_block_sum(local, s_part);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void wce_finish(const double* __restrict__ partial, int n, double inv_total, float* __restrict__ loss) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *loss = wce_partials_mean(partial, n, inv_total);
}

}  // namespace nbc

using namespace nbc;

extern "C" size_t nbc_wce_workspace_bytes(int, int, int) { return kWceBlocks * sizeof(double); }

extern "C" int nbc_wce_fwd_bwd(const float* logits, const void* target, int target_is_i64, const float* weights3,
                               int N, int H, int W, float* loss, float* grad, void* workspace, size_t workspace_bytes,
                               void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(logits && target && weights3 && loss && workspace, "nbc_wce_fwd_bwd: null pointer");
  NBC_REQUIRE(N > 0 && H > 0 && W > 0, "nbc_wce_fwd_bwd: bad shape");
  if (workspace_bytes < nbc_wce_workspace_bytes(N, H, W)) {
    set_error("nbc_wce_fwd_bwd: workspace too small");
    return NBC_ERR_WORKSPACE;
  }
  const int64_t HW = (int64_t)H * W, total = (int64_t)N * HW;
  const int blocks = (int)(ceil_div64(total, 256) < kWceBlocks ? ceil_div64(total, 256) : kWceBlocks);
  double* partial = reinterpret_cast<double*>(workspace);
  const float inv_total = (float)(1.0 / (double)total);
  if (target_is_i64)
    wce_kernel<int64_t><<<blocks, 256, 0, stream>>>(logits, reinterpret_cast<const int64_t*>(target), weights3, HW, total, inv_total, grad, partial);
  else
    wce_kernel<uint8_t><<<blocks, 256, 0, stream>>>(logits, reinterpret_cast<const uint8_t*>(target), weights3, HW, total, inv_total, grad, partial);
  NBC_CHECK_LAUNCH();
  wce_finish<<<1, 32, 0, stream>>>(partial, blocks, 1.0 / (double)total, loss);
  NBC_CHECK_LAUNCH();
  return 0;
}
