// Internal convolution interfaces shared by conv_tc.cu (tcgen05), conv_mma.cu (mma.sync), plan.cu and api.cu.
#pragma once
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>
#include <string.h>

namespace nbc {

struct ConvGeom {
  int N, H, W, Cin, Cout;
  int kh, kw, stride, pad, dil;
  int relu;
  int f16 = 0;  // 16-bit storage format of x / w / y: 0 bf16, 1 fp16
  int Ho() const { return (H + 2 * pad - dil * (kh - 1) - 1) / stride + 1; }
  int Wo() const { return (W + 2 * pad - dil * (kw - 1) - 1) / stride + 1; }
  double flops() const { return 2.0 * N * Ho() * Wo() * (double)Cout * Cin * kh * kw; }
};

// tcgen05 path: tensor maps are encoded once per (shape, pointers) and reused across launches
struct ConvTcPrepared {
  alignas(64) unsigned char storage[1536];
};
bool conv_tc_supported(const ConvGeom& g);
// valid_h (device, int[N], optional): ragged batch -- valid OUTPUT rows per image (see conv_tc.cu)
int conv_tc_prepare(const ConvGeom& g, const void* x, const void* w, const float* bias, const void* residual, void* y,
                    ConvTcPrepared* out, const int* valid_h = nullptr);
// main convolution + a 1x1 convolution of a second tensor accumulated into the same output (see conv_tc.cu)
int conv_tc_prepare_dual(const ConvGeom& g, const void* x, const ConvGeom& g2, const void* x2, const void* w_cat,
                         const float* bias, void* y, ConvTcPrepared* out, const int* valid_h = nullptr);
int conv_tc_run(const ConvTcPrepared* prep, cudaStream_t stream);
// which kernel conv_tc_run launches for a prepared convolution (nbc_plan_step_info)
struct ConvTcVariant {
  int pair, halo3, stem_halo, dual, block_n, kblk, out_bufs;
  int ragged_map;   // -1 dense batch, 1 compact tile map, 0 dense tile numbering with dead tiles skipped
};
void conv_tc_describe(const ConvTcPrepared* prep, ConvTcVariant* v);
// stem 7x7/2 as an implicit GEMM over the padded bf16 image (see stem.cu)
int conv_tc_prepare_stem(int N, int Ho, int Wo, int Hp, int Wp, const void* padded, const void* w224, const float* bias,
                         void* y, ConvTcPrepared* out, const int* valid_h = nullptr, int f16 = 0, int relu = 1);
int conv_tc(const ConvGeom& g, const void* x, const void* w, const float* bias, const void* residual, void* y,
            cudaStream_t stream);

// mma.sync path (any stride / dilation / kernel size; Cin % 32 == 0, Cout % 64 == 0)
bool conv_mma_supported(const ConvGeom& g);
int conv_mma(const ConvGeom& g, const void* x, const void* w, const float* bias, const void* residual, void* y,
             cudaStream_t stream);

// stem staging pass (stem.cu): input (0 = u8 NHWC, 1 = f32 NCHW) -> zero-padded normalised bf16 [N][Hp][Wp][4]
int stem_tc_pad(const void* input, int input_kind, int N, int H, int W, const float* mean3, const float* std3, void* padded,
                cudaStream_t stream, const int* valid_h, int f16 = 0);
int maxpool_ragged(const void* x, int N, int H, int W, int C, void* y, const int* valid_h, cudaStream_t stream,
                   int f16 = 0);
// valid_h (optional, ragged batch): rows of image n at or beyond valid_h[n] are skipped; row_w = pixels per row
int head_1x1(const void* x16, int64_t pixels_per_image, int N, int Cin, const float* w3xC, const float* bias3,
             float* logits_planar, int f16, cudaStream_t stream, const int* valid_h = nullptr, int row_w = 1);
// levels[4][N]: valid rows per image at full, 1/2, 1/4 and 1/8 resolution, from heights[N] or K1's {first,last}[N]
int ragged_levels(const int* heights, const int* first_last, int N, int Hc, int* levels, cudaStream_t stream);

// BN fold + pack (api.cu): w f32 OIHW -> bf16 (and/or f32) [Cout][kh][kw][cin_pad], bias f32[Cout]
int fold_pack(const float* w, const float* gamma, const float* beta, const float* mean, const float* var,
              const float* cb, float eps, int Cout, int Cin, int kh, int kw, int cin_pad, void* wp_bf16, float* wp_f32,
              float* bias, cudaStream_t stream, int f16 = 0);
// count of folded weights outside the fp16 range since the last reset (fp16 packs saturate; nbc_plan_create checks this)
int fold_overflow_reset();
int fold_overflow_read(unsigned int* n);

}  // namespace nbc
