// Internal interfaces of the training path (train_kernels.cu, train_plan.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "conv.h"

namespace nbc {

size_t bn_partial_bytes(int64_t M, int C);
// z -> batch statistics -> y = relu?(gamma (z-mean) invstd + beta (+ residual)); running stats updated like torch
int bn_forward_train(const void* z, int64_t M, int C, const float* gamma, const float* beta, float eps, float momentum,
                     float* running_mean, float* running_var, float* save_mean, float* save_invstd, float* a, float* b,
                     float* partial, const void* residual, int relu, void* y, cudaStream_t stream);
// dz from dy (ReLU mask from y when relu), accumulates dgamma / dbeta; g_out (optional) = masked dy for the skip path
int bn_backward(const void* dy, const void* y, const void* z, int64_t M, int C, const float* gamma, const float* save_mean,
                const float* save_invstd, int relu, float* partial, float* sums, float* dgamma, float* dbeta, void* dz,
                void* g_out, cudaStream_t stream);
int cast_pack(const float* w, int64_t n, void* out_bf16, cudaStream_t stream);
int dgrad_pack(const float* w_ohwi, int Cout, int Cin, int kh, int kw, void* out_bf16, cudaStream_t stream);
int oihw_ohwi(const float* src, int Cout, int Cin, int kh, int kw, float* dst, int reverse, cudaStream_t stream);
// dW[Cout][kh][kw][Cin] (f32, accumulated with atomics) += dz^T * x over all output pixels
int wgrad_mma(const ConvGeom& g, const void* dz, const void* x, float* dw, cudaStream_t stream);
// the same on the tcgen05 tensor cores (wgrad_tc.cu); Cin % 64 == 0, Cout % 64 == 0, stride 1 or 2.  Deterministic:
// with scratch (>= wgrad_tc_scratch_bytes, 16-byte aligned) the pixels are split over the SMs and the split partials
// are added in a fixed order by a second launch; with scratch == null one CTA per tile sums all pixels.  Either way
// every element of dw has one writer, dw += sum.
bool wgrad_tc_supported(const ConvGeom& g);
size_t wgrad_tc_scratch_bytes(const ConvGeom& g);
int wgrad_tc(const ConvGeom& g, const void* dz, const void* x, float* dw, void* scratch, size_t scratch_bytes,
             cudaStream_t stream);
size_t stem_wgrad_tc_scratch_bytes(int N, int Ho, int Wo);
int stem_wgrad_tc(const void* dz, const void* padded, int N, int Ho, int Wo, float* dw, void* scratch, size_t scratch_bytes,
                  cudaStream_t stream);

// 3x3/2 max pooling that records the position of the first maximum (idx: one byte per output element), and its backward
int maxpool_forward_idx(const void* x, int N, int H, int W, int C, void* y, void* idx, cudaStream_t stream);
int maxpool_backward(const void* dy, const void* idx, int N, int H, int W, int C, void* dx, cudaStream_t stream);
// stem: dW f32 [64][7][7][3] += dz^T * padded image (the bf16 staging buffer [N][2Ho+5][2Wo+6][4] of the stem)
int stem_wgrad(const void* dz, const void* padded, int N, int Ho, int Wo, float* dw, cudaStream_t stream);
int dropout_apply(const void* x, int64_t n, float p, uint64_t seed, void* y, cudaStream_t stream);
// classifier backward; dW / db get the per-block partials (partial: cls_partial_bytes) added in a fixed order
size_t cls_partial_bytes(int C);
int cls_backward(const float* dlow, const void* x, const float* w, int N, int64_t P, int C, float drop_p, uint64_t seed,
                 void* dx, float* dw, float* db, void* partial, cudaStream_t stream);
size_t upsample_bwd_workspace_bytes(int N, int C, int h, int w, int H, int W);
int upsample_backward(const float* dup, int N, int C, int h, int w, int H, int W, float* dlow, void* workspace,
                      cudaStream_t stream);
int zero_insert(const void* dz, int N, int Ho, int Wo, int H, int W, int C, void* up, cudaStream_t stream);
// out = sa * a + sb * b (lovasz.cu)
int axpby(const float* a, float sa, const float* b, float sb, int64_t n, float* out, cudaStream_t stream);
int adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float b1, float b2, float eps, float wd,
              int step, float grad_scale, cudaStream_t stream);

}  // namespace nbc
