// C-ABI glue: error reporting, device check, launch accounting, BN fold / weight packing, single-layer conv entry.
#include <stdarg.h>

#include "common.cuh"
#include "conv.h"
#include "train.h"

namespace nbc {

static thread_local char g_err[1024] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  static int cached = 0;
  if (cached) return cached;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) == cudaSuccess &&
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
    cached = n;
  else
    cached = 148;
  return cached;
}

encode_tiled_fn get_encode_tiled() {
  static encode_tiled_fn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<encode_tiled_fn>(p);
  }
  return fn;
}

// number of folded weights outside the fp16 range seen by fold_pack_kernel since the last reset (nbc_plan_create refuses
// an fp16 plan when it is non-zero: a saturated WEIGHT is a wrong network, unlike a saturated activation spike)
__device__ unsigned int g_fold_overflow = 0;

int fold_overflow_reset() {
  const unsigned int z = 0;
  NBC_CUDA(cudaMemcpyToSymbol(g_fold_overflow, &z, sizeof(z)));
  return 0;
}
int fold_overflow_read(unsigned int* n) {
  NBC_CUDA(cudaMemcpyFromSymbol(n, g_fold_overflow, sizeof(*n)));
  return 0;
}

// w f32 OIHW -> bf16 [Cout][kh][kw][cin_pad] scaled by gamma/sqrt(var+eps); bias = beta - mean*scale (+cb*scale)
__global__ void __launch_bounds__(256) fold_pack_kernel(const float* __restrict__ w, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, const float* __restrict__ mean,
                                                        const float* __restrict__ var, const float* __restrict__ cb,
                                                        float eps, int Cout, int Cin, int kh, int kw, int cin_pad,
                                                        unsigned short* __restrict__ wp, float* __restrict__ bias,
                                                        float* __restrict__ wp_f32, int f16) {
  const int64_t total = (int64_t)Cout * kh * kw * cin_pad;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % cin_pad);
    int64_t t = i / cin_pad;
    const int kx = (int)(t % kw);
    t /= kw;
    const int ky = (int)(t % kh);
    const int oc = (int)(t / kh);
    const float scale = gamma ? gamma[oc] / sqrtf(var[oc] + eps) : 1.f;
    float v = 0.f;
    if (c < Cin) v = w[(((int64_t)oc * Cin + c) * kh + ky) * kw + kx] * scale;
    if (wp) wp[i] = cvt16(v, f16);
    if (wp && f16 && !(fabsf(v) <= 65504.f)) atomicAdd(&g_fold_overflow, 1u);
    if (wp_f32) wp_f32[i] = v;
    if (c == 0 && ky == 0 && kx == 0) {
      float b = gamma ? beta[oc] - mean[oc] * scale : 0.f;
      if (cb) b += cb[oc] * scale;
      bias[oc] = b;
    }
  }
}

int fold_pack(const float* w, const float* gamma, const float* beta, const float* mean, const float* var,
              const float* cb, float eps, int Cout, int Cin, int kh, int kw, int cin_pad, void* wp_bf16, float* wp_f32,
              float* bias, cudaStream_t stream, int f16) {
  const int64_t total = (int64_t)Cout * kh * kw * cin_pad;
  const int blocks = (int)(ceil_div64(total, 256) < 148 * 8 ? ceil_div64(total, 256) : 148 * 8);
  fold_pack_kernel<<<blocks, 256, 0, stream>>>(w, gamma, beta, mean, var, cb, eps, Cout, Cin, kh, kw, cin_pad,
                                               reinterpret_cast<unsigned short*>(wp_bf16), bias, wp_f32, f16);
  NBC_CHECK_LAUNCH();
  return 0;
}

}  // namespace nbc

using namespace nbc;

extern "C" int nbc_version(void) { return 100; }
extern "C" const char* nbc_last_error(void) { return g_err; }
extern "C" int64_t nbc_launch_count(void) { return g_launches.load(); }

extern "C" int nbc_device_check(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    set_error("no CUDA device available (%s); libnbc has no CPU fallback", e == cudaSuccess ? "count 0" : cudaGetErrorString(e));
    return NBC_ERR_DEVICE;
  }
  if (device < 0 || device >= n) {
    set_error("device %d out of range (have %d)", device, n);
    return NBC_ERR_DEVICE;
  }
  cudaDeviceProp prop;
  NBC_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; libnbc is built for sm_100a (B200) only", device, prop.major, prop.minor);
    return NBC_ERR_DEVICE;
  }
  NBC_CUDA(cudaSetDevice(device));
  return 0;
}

extern "C" int nbc_fold_bn_pack(const float* w, const float* gamma, const float* beta, const float* mean,
                                const float* var, const float* conv_bias, float eps, int Cout, int Cin, int kh, int kw,
                                int cin_pad, int f16, void* w_packed_bf16, float* bias_out, void* stream) {
  NBC_REQUIRE(w && w_packed_bf16 && bias_out, "nbc_fold_bn_pack: null pointer");
  NBC_REQUIRE((gamma != nullptr) == (beta != nullptr) && (gamma != nullptr) == (mean != nullptr) &&
                  (gamma != nullptr) == (var != nullptr),
              "nbc_fold_bn_pack: gamma/beta/mean/var must be all given or all NULL");
  NBC_REQUIRE(Cout > 0 && Cin > 0 && kh > 0 && kw > 0 && cin_pad >= Cin, "nbc_fold_bn_pack: bad shape");
  return fold_pack(w, gamma, beta, mean, var, conv_bias, eps, Cout, Cin, kh, kw, cin_pad, w_packed_bf16, nullptr,
                   bias_out, reinterpret_cast<cudaStream_t>(stream), f16 ? 1 : 0);
}

extern "C" int nbc_conv_bf16(const nbc_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                             const void* residual, void* y, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(d && x && w_packed && bias && y, "nbc_conv_bf16: null pointer");
  ConvGeom g{d->N, d->H, d->W, d->Cin, d->Cout, d->kh, d->kw, d->stride, d->pad, d->dil, d->relu, d->f16 ? 1 : 0};
  NBC_REQUIRE(g.N > 0 && g.H > 0 && g.W > 0 && g.Ho() > 0 && g.Wo() > 0, "nbc_conv_bf16: bad shape");
  const bool tc_ok = conv_tc_supported(g);
  if (d->impl == 1 || (d->impl == 0 && tc_ok)) return conv_tc(g, x, w_packed, bias, residual, y, stream);
  if (d->impl == 2 || d->impl == 0) return conv_mma(g, x, w_packed, bias, residual, y, stream);
  set_error("nbc_conv_bf16: unknown impl %d", d->impl);
  return NBC_ERR_INVALID;
}

extern "C" int nbc_conv_wgrad_bf16(const nbc_conv_desc* d, const void* dz, const void* x, float* dw, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(d && dz && x && dw, "nbc_conv_wgrad_bf16: null pointer");
  NBC_REQUIRE(!d->f16, "nbc_conv_wgrad_bf16: the training path is bf16 only");
  ConvGeom g{d->N, d->H, d->W, d->Cin, d->Cout, d->kh, d->kw, d->stride, d->pad, d->dil, 0, 0};
  NBC_REQUIRE(g.N > 0 && g.H > 0 && g.W > 0 && g.Ho() > 0 && g.Wo() > 0, "nbc_conv_wgrad_bf16: bad shape");
  const bool tc_ok = wgrad_tc_supported(g);
  if (d->impl == 1 || (d->impl == 0 && tc_ok)) return wgrad_tc(g, dz, x, dw, nullptr, 0, stream);
  if (d->impl == 2 || d->impl == 0) return wgrad_mma(g, dz, x, dw, stream);
  set_error("nbc_conv_wgrad_bf16: unknown impl %d", d->impl);
  return NBC_ERR_INVALID;
}

extern "C" size_t nbc_conv_wgrad_workspace_bytes(const nbc_conv_desc* d) {
  if (!d) return 0;
  const ConvGeom g{d->N, d->H, d->W, d->Cin, d->Cout, d->kh, d->kw, d->stride, d->pad, d->dil, 0, 0};
  if (g.N <= 0 || g.H <= 0 || g.W <= 0 || g.Ho() <= 0 || g.Wo() <= 0) return 0;
  return wgrad_tc_scratch_bytes(g);
}

extern "C" int nbc_conv_wgrad_bf16_ws(const nbc_conv_desc* d, const void* dz, const void* x, float* dw, void* workspace,
                                      size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(d && dz && x && dw, "nbc_conv_wgrad_bf16_ws: null pointer");
  NBC_REQUIRE(!d->f16, "nbc_conv_wgrad_bf16_ws: the training path is bf16 only");
  ConvGeom g{d->N, d->H, d->W, d->Cin, d->Cout, d->kh, d->kw, d->stride, d->pad, d->dil, 0, 0};
  NBC_REQUIRE(g.N > 0 && g.H > 0 && g.W > 0 && g.Ho() > 0 && g.Wo() > 0, "nbc_conv_wgrad_bf16_ws: bad shape");
  return wgrad_tc(g, dz, x, dw, workspace, workspace_bytes, stream);
}

extern "C" int nbc_conv_dual_bf16(const nbc_conv_desc* d, const void* x, const nbc_conv_desc* d2, const void* x2, const void* w_cat,
                                  const float* bias, void* y, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(d && d2 && x && x2 && w_cat && bias && y, "nbc_conv_dual_bf16: null pointer");
  ConvGeom g{d->N, d->H, d->W, d->Cin, d->Cout, d->kh, d->kw, d->stride, d->pad, d->dil, d->relu, d->f16 ? 1 : 0};
  ConvGeom g2{d2->N, d2->H, d2->W, d2->Cin, d2->Cout, d2->kh, d2->kw, d2->stride, d2->pad, d2->dil, 0, d->f16 ? 1 : 0};
  ConvTcPrepared prep;
  int rc = conv_tc_prepare_dual(g, x, g2, x2, w_cat, bias, y, &prep);
  if (rc) return rc;
  return conv_tc_run(&prep, stream);
}
