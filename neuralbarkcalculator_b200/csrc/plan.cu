// The whole FCN-ResNet50 forward as a native plan (models.py:27-43 SimpleSegmentationModel.forward up to the
// classifier output, models.py:127-139 fcn_resnet50; torchvision resnet50 with replace_stride_with_dilation =
// [False, True, True]).  The plan owns the BN-folded bf16 weights; activations live in the caller's workspace:
//   bufA / bufB : block input / output ping-pong (largest: layer4 output, 2048 ch at H/8 x W/8)
//   t1 / t2     : bottleneck inner tensors
// Layer list (55 convs): stem 7x7/2 (normalise + pad staging pass, then tcgen05 implicit GEMM) -> maxpool -> 16 bottlenecks
// (conv1 1x1 +ReLU, conv2 3x3 stride/dilation +ReLU, conv3 1x1 + residual + ReLU, optional downsample 1x1)
// -> FCNHead conv3x3 + ReLU -> 1x1 (512 -> 3) + bias as f32 planar logits.
#include <map>
#include <tuple>
#include <vector>

#include "common.cuh"
#include "conv.h"
#include "train.h"   // axpby

namespace nbc {

struct ConvLayer {
  int Cin, Cout, k, stride, pad, dil, relu;
  __nv_bfloat16* w = nullptr;  // [Cout][k][k][Cin], BN scale folded
  float* bias = nullptr;       // [Cout]
};

struct Block {
  ConvLayer c1, c2, c3, ds;
  bool has_ds = false;
  // conv3 and the downsample branch as ONE launch (tcgen05 path): weights [Cout][K3 + Kds], bias = b3 + bds
  __nv_bfloat16* w_cat = nullptr;
  float* bias_cat = nullptr;
};

struct Step {  // one launch of the cached forward
  int kind;    // 0 stem, 1 maxpool, 2 conv(tc), 3 conv(mma), 4 head1x1
  ConvGeom g;
  const void* x;
  const void* w;
  const float* bias;
  const void* residual;
  void* y;
  ConvTcPrepared prep;
  const char* name;
  double extra_flops = 0.0;   // fused second source
  const void* x2 = nullptr;   // fused second source (conv3 + downsample): its input and geometry
  ConvGeom g2{};
  int level = -1;             // ragged batch: row of the level table with the valid output rows
};

}  // namespace nbc

struct nbc_plan {
  float mean[3], std[3];
  float* stem_w = nullptr;  // f32 [64][7][7][3]
  float* stem_b = nullptr;
  __nv_bfloat16* stem_w224 = nullptr;  // bf16 [64][7][8][4] for the tensor-core stem
  std::vector<nbc::Block> blocks;
  nbc::ConvLayer head;
  float* cls_w = nullptr;  // f32 [3][512]
  float* cls_b = nullptr;
  std::vector<void*> allocs;
  char* slab = nullptr;       // parameter slab (see dev_alloc)
  size_t slab_used = 0;
  int impl = 0;
  int f16 = 0;   // 16-bit storage format: 0 bf16 (default), 1 fp16
  // cached launch lists (tensor maps are encoded once per shape / workspace): key = (N, H, W, workspace, impl)
  typedef std::tuple<int, int, int, void*, int, int> Key;   // N, H, W, workspace, impl, ragged
  std::map<Key, std::vector<nbc::Step>> cache;
  std::vector<nbc::Step>* steps_ptr = nullptr;
  Key steps_key;   // the key of *steps_ptr
  int stop = -1;   // nbc_plan_set_stop: last step a forward runs (< 0: all)
};

namespace nbc {

// Parameters are carved out of one slab (one cudaMalloc / cudaFree per plan instead of ~115: cudaFree synchronises the
// device and unmaps memory, which made tearing a plan down take up to a second); an allocation that does not fit --
// never for FCN-ResNet50, 66 MB of packed weights -- falls back to its own cudaMalloc.
constexpr size_t kPlanSlabBytes = 96u << 20;
static int dev_alloc(nbc_plan* p, void** ptr, size_t bytes) {
  if (p->slab == nullptr) {
    NBC_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->slab), kPlanSlabBytes));
    p->allocs.push_back(p->slab);
    p->slab_used = 0;
  }
  const size_t need = align_up(bytes, 256);
  if (p->slab_used + need <= kPlanSlabBytes) {
    *ptr = p->slab + p->slab_used;
    p->slab_used += need;
    return 0;
  }
  NBC_CUDA(cudaMalloc(ptr, bytes));
  p->allocs.push_back(*ptr);
  return 0;
}

// tensors: conv weight, then bn {weight, bias, running_mean, running_var, num_batches_tracked}
static int make_conv(nbc_plan* p, const void* const* t, int Cin, int Cout, int k, int stride, int pad, int dil, int relu,
                     ConvLayer* L) {
  L->Cin = Cin, L->Cout = Cout, L->k = k, L->stride = stride, L->pad = pad, L->dil = dil, L->relu = relu;
  int rc = dev_alloc(p, reinterpret_cast<void**>(&L->w), (size_t)Cout * k * k * Cin * 2);
  if (rc) return rc;
  rc = dev_alloc(p, reinterpret_cast<void**>(&L->bias), (size_t)Cout * 4);
  if (rc) return rc;
  return fold_pack(reinterpret_cast<const float*>(t[0]), reinterpret_cast<const float*>(t[1]),
                   reinterpret_cast<const float*>(t[2]), reinterpret_cast<const float*>(t[3]),
                   reinterpret_cast<const float*>(t[4]), nullptr, 1e-5f, Cout, Cin, k, k, Cin, L->w, nullptr, L->bias, 0,
                   p->f16);
}

// [W3 | Wds] per output channel and b3 + bds, for the fused conv3 + downsample launch
static int concat_weights(Block& B, int width, int inplanes, int outp) {
  const size_t pitch = (size_t)(width + inplanes) * 2;
  NBC_CUDA(cudaMemcpy2DAsync(B.w_cat, pitch, B.c3.w, (size_t)width * 2, (size_t)width * 2, outp, cudaMemcpyDeviceToDevice, 0));
  NBC_CUDA(cudaMemcpy2DAsync(reinterpret_cast<char*>(B.w_cat) + (size_t)width * 2, pitch, B.ds.w, (size_t)inplanes * 2,
                             (size_t)inplanes * 2, outp, cudaMemcpyDeviceToDevice, 0));
  return axpby(B.c3.bias, 1.f, B.ds.bias, 1.f, outp, B.bias_cat, 0);
}

struct Dims {
  int H2, W2, H4, W4, H8, W8;
};
static Dims dims_of(int H, int W) {
  Dims d;
  d.H2 = (H - 1) / 2 + 1, d.W2 = (W - 1) / 2 + 1;      // conv 7x7/2 pad 3
  d.H4 = (d.H2 - 1) / 2 + 1, d.W4 = (d.W2 - 1) / 2 + 1;  // maxpool 3x3/2 pad 1
  d.H8 = (d.H4 - 1) / 2 + 1, d.W8 = (d.W4 - 1) / 2 + 1;  // layer2 stride 2
  return d;
}
static void buffer_sizes(int N, int H, int W, size_t* big, size_t* small) {
  const Dims d = dims_of(H, W);
  const size_t p2 = (size_t)d.H2 * d.W2, p4 = (size_t)d.H4 * d.W4, p8 = (size_t)d.H8 * d.W8;
  size_t b = p2 * 64;
  b = b > p4 * 256 ? b : p4 * 256;
  b = b > p8 * 2048 ? b : p8 * 2048;
  size_t s = p4 * 128;
  s = s > p8 * 512 ? s : p8 * 512;
  *big = align_up(b * N * 2, 1024);
  *small = align_up(s * N * 2, 1024);
  const size_t stem_ws = nbc_stem_tc_workspace_bytes(N, H, W);   // the padded bf16 image lives in t2
  if (*small < stem_ws) *small = stem_ws;
}

// levels: device int[4][N] of a ragged batch (nullptr for a dense batch); *level = resolution level of the input
// (0 full, 1 half, 2 quarter, 3 eighth), advanced by stride-2 layers
static int add_conv(nbc_plan* p, const ConvLayer& L, int N, int H, int W, const void* x, const void* residual, void* y,
                    const char* name, int* Ho, int* Wo, const int* levels = nullptr, int* level = nullptr) {
  Step s;
  memset(&s.prep, 0, sizeof(s.prep));
  s.g = ConvGeom{N, H, W, L.Cin, L.Cout, L.k, L.k, L.stride, L.pad, L.dil, L.relu, p->f16};
  s.x = x, s.w = L.w, s.bias = L.bias, s.residual = residual, s.y = y, s.name = name;
  const bool tc = (p->impl != 2) && conv_tc_supported(s.g);
  s.kind = tc ? 2 : 3;
  const int* vh = nullptr;
  if (levels != nullptr) {
    if (!tc) {
      set_error("plan: ragged batches need the tcgen05 path (layer %s)", name);
      return NBC_ERR_INVALID;
    }
    if (L.stride == 2) ++*level;
    vh = levels + (size_t)(*level) * N;
  }
  if (tc) {
    int rc = conv_tc_prepare(s.g, x, L.w, L.bias, residual, y, &s.prep, vh);
    if (rc) return rc;
  } else if (!conv_mma_supported(s.g)) {
    set_error("plan: layer %s has no kernel (Cin=%d Cout=%d)", name, L.Cin, L.Cout);
    return NBC_ERR_INVALID;
  }
  *Ho = s.g.Ho(), *Wo = s.g.Wo();
  if (level != nullptr) s.level = *level;
  p->steps_ptr->push_back(s);
  return 0;
}

static int build_steps(nbc_plan* p, int N, int H, int W, void* workspace, bool ragged) {
  std::vector<Step>& steps = *p->steps_ptr;
  steps.clear();
  const void* images = nullptr;   // the stem input and the logits output are patched in at run time
  float* logits = nullptr;
  size_t big, small;
  buffer_sizes(N, H, W, &big, &small);
  char* ws = reinterpret_cast<char*>(workspace);
  void* bufA = ws;
  void* bufB = ws + big;
  void* t1 = ws + 2 * big;
  void* t2 = ws + 2 * big + small;
  const int* levels = ragged ? reinterpret_cast<const int*>(ws + 2 * big + 2 * small) : nullptr;
  const Dims d = dims_of(H, W);
  {
    Step s;
    memset(&s.prep, 0, sizeof(s.prep));
    s.kind = 0, s.g = ConvGeom{N, H, W, 3, 64, 7, 7, 2, 3, 1, 1}, s.x = images, s.y = bufB;
    s.name = "stem";
    s.w = p->stem_w, s.bias = p->stem_b, s.residual = t2;   // residual slot = staging buffer of the padded image
    if (ragged && p->impl == 2) {
      set_error("plan: ragged batches need the tcgen05 path");
      return NBC_ERR_INVALID;
    }
    if (p->impl != 2) {
      s.kind = 5;  // tensor-core stem
      int rc = conv_tc_prepare_stem(N, d.H2, d.W2, 2 * d.H2 + 5, 2 * d.W2 + 6, t2, p->stem_w224, p->stem_b, bufB, &s.prep,
                                    ragged ? levels + N : nullptr, p->f16);
      if (rc) return rc;
    }
    s.w = levels;   // w slot of the stem / maxpool steps = ragged level table (or nullptr)
    s.level = ragged ? 1 : -1;
    steps.push_back(s);
    Step m;
    memset(&m.prep, 0, sizeof(m.prep));
    m.kind = 1, m.g = ConvGeom{N, d.H2, d.W2, 64, 64, 3, 3, 2, 1, 1, 0}, m.x = bufB, m.y = bufA, m.name = "maxpool";
    m.w = levels, m.bias = nullptr, m.residual = nullptr;
    m.level = ragged ? 2 : -1;
    steps.push_back(m);
  }
  int h = d.H4, w = d.W4;
  int level = 2;   // the bottlenecks start at quarter resolution
  void* in = bufA;
  void* other = bufB;
  for (size_t b = 0; b < p->blocks.size(); ++b) {
    const Block& B = p->blocks[b];
    int h1, w1, h2, w2, h3, w3;
    int lv_in = level, lv = level;
    int rc = add_conv(p, B.c1, N, h, w, in, nullptr, t1, "conv1", &h1, &w1, levels, &lv);
    if (rc) return rc;
    rc = add_conv(p, B.c2, N, h1, w1, t1, nullptr, t2, "conv2", &h2, &w2, levels, &lv);
    if (rc) return rc;
    level = lv;
    if (B.has_ds && p->impl != 2) {
      // conv3 + downsample branch in one launch: out = relu(W3 * t2 + Wds * in(strided) + b3 + bds); no intermediate
      // tensor for the branch, its 1x1 convolution is just more K for the same accumulator
      Step s;
      memset(&s.prep, 0, sizeof(s.prep));
      s.g = ConvGeom{N, h2, w2, B.c3.Cin, B.c3.Cout, 1, 1, 1, 0, 1, 1, p->f16};
      const ConvGeom g2{N, h, w, B.ds.Cin, B.ds.Cout, 1, 1, B.ds.stride, 0, 1, 0, p->f16};
      s.extra_flops = g2.flops();
      s.x = t2, s.w = B.w_cat, s.bias = B.bias_cat, s.residual = nullptr, s.y = other, s.name = "conv3+downsample";
      s.kind = 2;
      s.x2 = in, s.g2 = g2, s.level = levels != nullptr ? lv : -1;
      rc = conv_tc_prepare_dual(s.g, t2, g2, in, B.w_cat, B.bias_cat, other, &s.prep, levels != nullptr ? levels + (size_t)lv * N : nullptr);
      if (rc) return rc;
      h3 = s.g.Ho(), w3 = s.g.Wo();
      p->steps_ptr->push_back(s);
      void* tmp = in;
      in = other;
      other = tmp;
    } else if (B.has_ds) {
      int hd, wd;
      rc = add_conv(p, B.ds, N, h, w, in, nullptr, other, "downsample", &hd, &wd, levels, &lv_in);
      if (rc) return rc;
      // the block input is dead after conv1 and downsample: conv3 overwrites it, residual = downsample output
      rc = add_conv(p, B.c3, N, h2, w2, t2, other, in, "conv3", &h3, &w3, levels, &lv);
      if (rc) return rc;
    } else {
      rc = add_conv(p, B.c3, N, h2, w2, t2, in, other, "conv3", &h3, &w3, levels, &lv);
      if (rc) return rc;
      void* tmp = in;
      in = other;
      other = tmp;
    }
    h = h3, w = w3;
  }
  int hh, wh;
  int rc = add_conv(p, p->head, N, h, w, in, nullptr, t1, "head3x3", &hh, &wh, levels, &level);
  if (rc) return rc;
  Step s;
  memset(&s.prep, 0, sizeof(s.prep));
  s.kind = 4, s.g = ConvGeom{N, hh, wh, 512, 3, 1, 1, 1, 0, 1, 0}, s.x = t1, s.y = logits, s.name = "head1x1";
  s.w = p->cls_w, s.bias = p->cls_b;
  s.residual = levels != nullptr ? levels + (size_t)3 * N : nullptr;      // ragged: valid rows at 1/8 resolution
  s.level = levels != nullptr ? 3 : -1;
  steps.push_back(s);
  return 0;
}

static int run_step(nbc_plan* p, const Step& s, const void* input, int input_kind, float* logits,
                    cudaStream_t stream) {
  switch (s.kind) {
    case 0:
      if (input_kind == 1)
        return nbc_stem_f32(reinterpret_cast<const float*>(input), s.g.N, s.g.H, s.g.W, p->stem_w, p->stem_b, s.y,
                            stream);
      return nbc_stem_u8(reinterpret_cast<const uint8_t*>(input), s.g.N, s.g.H, s.g.W, p->mean, p->std, p->stem_w,
                         p->stem_b, s.y, stream);
    case 5: {
      int rc = stem_tc_pad(input, input_kind, s.g.N, s.g.H, s.g.W, p->mean, p->std, const_cast<void*>(s.residual), stream,
                           reinterpret_cast<const int*>(s.w), p->f16);
      if (rc) return rc;
      return conv_tc_run(&s.prep, stream);
    }
    case 1:
      if (s.w != nullptr)
        return maxpool_ragged(s.x, s.g.N, s.g.H, s.g.W, 64, s.y, reinterpret_cast<const int*>(s.w) + 2 * (size_t)s.g.N, stream,
                              p->f16);
      return nbc_maxpool3x3s2_bf16(s.x, s.g.N, s.g.H, s.g.W, 64, p->f16, s.y, stream);
    case 2: return conv_tc_run(&s.prep, stream);
    case 3: return conv_mma(s.g, s.x, s.w, s.bias, s.residual, s.y, stream);
    case 4:
      return head_1x1(s.x, (int64_t)s.g.H * s.g.W, s.g.N, 512, p->cls_w, p->cls_b, logits, p->f16, stream,
                      reinterpret_cast<const int*>(s.residual), s.g.W);
  }
  return NBC_ERR_INVALID;
}

static int ensure_steps(nbc_plan* p, const void* images, int input_kind, int N, int H, int W, float* logits,
                        void* workspace, size_t workspace_bytes, bool ragged = false) {
  NBC_REQUIRE(p && images && logits && workspace, "nbc_plan_forward: null pointer");
  NBC_REQUIRE(N > 0 && H >= 16 && W >= 16, "nbc_plan_forward: bad shape %dx%dx%d", N, H, W);
  NBC_REQUIRE(input_kind == 0 || input_kind == 1, "nbc_plan_forward: input_kind must be 0 (u8 NHWC) or 1 (f32 NCHW)");
  if (workspace_bytes < nbc_plan_workspace_bytes(p, N, H, W)) {
    set_error("nbc_plan_forward: workspace %zu < %zu", workspace_bytes, nbc_plan_workspace_bytes(p, N, H, W));
    return NBC_ERR_WORKSPACE;
  }
  NBC_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 1024 == 0, "nbc_plan_forward: workspace must be 1024-byte aligned");
  (void)images, (void)logits;
  nbc_plan::Key key(N, H, W, workspace, p->impl, ragged ? 1 : 0);
  auto it = p->cache.find(key);
  p->steps_key = key;
  if (it != p->cache.end()) {
    p->steps_ptr = &it->second;
    return 0;
  }
  if (p->cache.size() >= 256) p->cache.clear();
  p->steps_ptr = &p->cache[key];
  int rc = build_steps(p, N, H, W, workspace, ragged);
  if (rc) {
    p->cache.erase(key);
    p->steps_ptr = nullptr;
    return rc;
  }
  return 0;
}

}  // namespace nbc

using namespace nbc;

extern "C" nbc_plan* nbc_plan_create(const void* const* t, int n_tensors, const float* mean3_host,
                                     const float* std3_host, int f16) {
  if (!t || n_tensors != 326 || !mean3_host || !std3_host) {
    set_error("nbc_plan_create: expected the 326 state_dict tensors of fcn_resnet50 (got %d)", n_tensors);
    return nullptr;
  }
  for (int i = 0; i < n_tensors; ++i)
    if (!t[i]) {
      set_error("nbc_plan_create: tensor %d is NULL", i);
      return nullptr;
    }
  nbc_plan* p = new nbc_plan();
  p->f16 = f16 ? 1 : 0;
  for (int i = 0; i < 3; ++i) p->mean[i] = mean3_host[i], p->std[i] = std3_host[i];
  int rc = 0;
  int idx = 0;
  if (p->f16) rc = fold_overflow_reset();
  // stem: f32 weights [64][7][7][3]
  if (!rc) rc = dev_alloc(p, reinterpret_cast<void**>(&p->stem_w), 64 * 147 * 4);
  if (!rc) rc = dev_alloc(p, reinterpret_cast<void**>(&p->stem_b), 64 * 4);
  if (!rc)
    rc = fold_pack(reinterpret_cast<const float*>(t[0]), reinterpret_cast<const float*>(t[1]),
                   reinterpret_cast<const float*>(t[2]), reinterpret_cast<const float*>(t[3]),
                   reinterpret_cast<const float*>(t[4]), nullptr, 1e-5f, 64, 3, 7, 7, 3, nullptr, p->stem_w, p->stem_b, 0);
  if (!rc) rc = dev_alloc(p, reinterpret_cast<void**>(&p->stem_w224), 64 * 224 * 2);
  if (!rc) rc = nbc_stem_pack_weights(p->stem_w, p->f16, p->stem_w224, 0);
  idx = 6;
  const int nblocks[4] = {3, 4, 6, 3};
  const int planes[4] = {64, 128, 256, 512};
  int inplanes = 64, dilation = 1;
  for (int li = 0; li < 4 && !rc; ++li) {
    // torchvision ResNet._make_layer with replace_stride_with_dilation = [False, True, True]
    int stride = (li == 0) ? 1 : 2;
    const int prev_dil = dilation;
    if (li >= 2) {
      dilation *= stride;
      stride = 1;
    }
    for (int b = 0; b < nblocks[li] && !rc; ++b) {
      Block B;
      const int width = planes[li], outp = planes[li] * 4;
      const int s = (b == 0) ? stride : 1;
      const int dl = (b == 0) ? prev_dil : dilation;
      rc = make_conv(p, t + idx, inplanes, width, 1, 1, 0, 1, 1, &B.c1);
      idx += 6;
      if (!rc) rc = make_conv(p, t + idx, width, width, 3, s, dl, dl, 1, &B.c2);
      idx += 6;
      if (!rc) rc = make_conv(p, t + idx, width, outp, 1, 1, 0, 1, 1, &B.c3);  // ReLU after the residual add
      idx += 6;
      if (b == 0) {  // every first block of a resnet50 layer has a downsample branch (channel count changes)
        B.has_ds = true;
        if (!rc) rc = make_conv(p, t + idx, inplanes, outp, 1, s, 0, 1, 0, &B.ds);
        idx += 6;
        // fused launch: [W3 | Wds] along K (both already carry their BN scale), bias = b3 + bds
        if (!rc) rc = dev_alloc(p, reinterpret_cast<void**>(&B.w_cat), (size_t)outp * (width + inplanes) * 2);
        if (!rc) rc = dev_alloc(p, reinterpret_cast<void**>(&B.bias_cat), (size_t)outp * 4);
        if (!rc) rc = concat_weights(B, width, inplanes, outp);
      }
      inplanes = outp;
      p->blocks.push_back(B);
    }
  }
  if (!rc) rc = make_conv(p, t + idx, 2048, 512, 3, 1, 1, 1, 1, &p->head);
  idx += 6;
  if (!rc) rc = dev_alloc(p, reinterpret_cast<void**>(&p->cls_w), 3 * 512 * 4);
  if (!rc) rc = dev_alloc(p, reinterpret_cast<void**>(&p->cls_b), 3 * 4);
  if (!rc) {
    cudaError_t e = cudaMemcpy(p->cls_w, t[idx], 3 * 512 * 4, cudaMemcpyDeviceToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(p->cls_b, t[idx + 1], 3 * 4, cudaMemcpyDeviceToDevice);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
      set_error("nbc_plan_create: %s", cudaGetErrorString(e));
      rc = NBC_ERR_CUDA;
    }
  }
  idx += 2;
  if (!rc && p->f16) {
    // fp16 storage: a BN-folded weight beyond +-65504 cannot be represented (the pack saturates) -- refuse the plan
    // instead of running a different network; bf16 storage (f16 = 0) has the f32 exponent range
    unsigned int over = 0;
    rc = fold_overflow_read(&over);
    if (!rc && over) {
      set_error("nbc_plan_create: %u BN-folded weights exceed the fp16 range (|w| > 65504); build the plan with bf16 "
                "storage (f16 = 0, precision='bf16')", over);
      rc = NBC_ERR_INVALID;
    }
  }
  if (rc || idx != 326) {
    if (!rc) set_error("nbc_plan_create: internal tensor walk ended at %d", idx);
    nbc_plan_destroy(p);
    return nullptr;
  }
  return p;
}

extern "C" void nbc_plan_destroy(nbc_plan* p) {
  if (!p) return;
  for (void* a : p->allocs) cudaFree(a);
  delete p;
}

extern "C" size_t nbc_plan_workspace_bytes(const nbc_plan*, int N, int H, int W) {
  size_t big, small;
  buffer_sizes(N, H, W, &big, &small);
  return 2 * big + 2 * small + align_up((size_t)4 * N * sizeof(int), 1024);   // + ragged level table
}

extern "C" int nbc_plan_set_impl(nbc_plan* p, int impl) {
  NBC_REQUIRE(p && impl >= 0 && impl <= 2, "nbc_plan_set_impl: bad argument");
  p->impl = impl;
  return 0;
}

extern "C" int nbc_plan_forward(nbc_plan* p, const void* input, int input_kind, int N, int H, int W,
                                float* lowres_logits, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  int rc = ensure_steps(p, input, input_kind, N, H, W, lowres_logits, workspace, workspace_bytes);
  if (rc) return rc;
  const std::vector<Step>& steps = *p->steps_ptr;
  for (int i = 0; i < (int)steps.size(); ++i) {
    rc = run_step(p, steps[i], input, input_kind, lowres_logits, stream);
    if (rc) return rc;
    if (i == p->stop) break;
  }
  return 0;
}

extern "C" int nbc_plan_forward_ragged(nbc_plan* p, const uint8_t* canvas, int N, int Hc, int W, const int32_t* heights,
                                       const int32_t* first_last, float* lowres_logits, void* workspace,
                                       size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE((heights != nullptr) != (first_last != nullptr),
              "nbc_plan_forward_ragged: give exactly one of heights / first_last");
  int rc = ensure_steps(p, canvas, 0, N, Hc, W, lowres_logits, workspace, workspace_bytes, true);
  if (rc) return rc;
  size_t big, small;
  buffer_sizes(N, Hc, W, &big, &small);
  int* levels = reinterpret_cast<int*>(reinterpret_cast<char*>(workspace) + 2 * big + 2 * small);
  rc = ragged_levels(heights, first_last, N, Hc, levels, stream);
  if (rc) return rc;
  const std::vector<Step>& steps = *p->steps_ptr;
  for (int i = 0; i < (int)steps.size(); ++i) {
    rc = run_step(p, steps[i], canvas, 0, lowres_logits, stream);
    if (rc) return rc;
    if (i == p->stop) break;
  }
  return 0;
}

extern "C" int nbc_plan_profile(nbc_plan* p, const void* input, int input_kind, int N, int H, int W,
                                float* lowres_logits, void* workspace, size_t workspace_bytes, void* stream_,
                                float* ms_out, double* flops_out, int max_layers) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  int rc = ensure_steps(p, input, input_kind, N, H, W, lowres_logits, workspace, workspace_bytes);
  if (rc) return rc;
  const std::vector<Step>& steps = *p->steps_ptr;
  const int n = (int)steps.size();
  NBC_REQUIRE(ms_out && max_layers >= n, "nbc_plan_profile: need room for %d layers", n);
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) NBC_CUDA(cudaEventCreate(&e));
  NBC_CUDA(cudaEventRecord(ev[0], stream));
  for (int i = 0; i < n; ++i) {
    rc = run_step(p, steps[i], input, input_kind, lowres_logits, stream);
    if (rc) return rc;
    NBC_CUDA(cudaEventRecord(ev[i + 1], stream));
  }
  NBC_CUDA(cudaStreamSynchronize(stream));
  for (int i = 0; i < n; ++i) {
    NBC_CUDA(cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]));
    if (flops_out) flops_out[i] = (steps[i].kind == 1) ? 0.0 : steps[i].g.flops() + steps[i].extra_flops;
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return n;
}

// Stopping after step k leaves its operands intact: in build_steps no step reads the buffer it writes.  The stem reads
// the caller's image (and, on tensor cores, its staging image in t2) and writes bufB; maxpool bufB -> bufA; each
// bottleneck conv1 in -> t1, conv2 t1 -> t2, then either the fused conv3 + downsample (t2, in) -> other, or on the
// mma.sync path downsample in -> other and conv3 (t2, residual other) -> in, or without a downsample conv3 (t2,
// residual in) -> other; head3x3 in -> t1 and head1x1 t1 -> the caller's logits.
extern "C" int nbc_plan_set_stop(nbc_plan* p, int k) {
  NBC_REQUIRE(p, "nbc_plan_set_stop: null plan");
  p->stop = k < 0 ? -1 : k;
  return 0;
}

extern "C" int nbc_plan_num_steps(const nbc_plan* p) {
  NBC_REQUIRE(p, "nbc_plan_num_steps: null plan");
  return p->steps_ptr ? (int)p->steps_ptr->size() : 0;
}

extern "C" int nbc_plan_step_info(const nbc_plan* p, int i, nbc_plan_step* out) {
  NBC_REQUIRE(p && out, "nbc_plan_step_info: null pointer");
  NBC_REQUIRE(p->steps_ptr && i >= 0 && i < (int)p->steps_ptr->size(), "nbc_plan_step_info: no step %d", i);
  const Step& s = (*p->steps_ptr)[i];
  const char* ws = reinterpret_cast<const char*>(std::get<3>(p->steps_key));
  size_t big, small;
  buffer_sizes(std::get<0>(p->steps_key), std::get<1>(p->steps_key), std::get<2>(p->steps_key), &big, &small);
  auto off = [&](const void* a) -> int64_t { return a ? (int64_t)(reinterpret_cast<const char*>(a) - ws) : -1; };
  memset(out, 0, sizeof(*out));
  snprintf(out->name, sizeof(out->name), "%s", s.name);
  out->kind = s.kind;
  out->ragged_map = -1;
  if (s.kind == 2 || s.kind == 5) {
    ConvTcVariant v;
    conv_tc_describe(&s.prep, &v);
    out->pair = v.pair, out->halo3 = v.halo3, out->stem_halo = v.stem_halo, out->dual = v.dual;
    out->block_n = v.block_n, out->kblk = v.kblk, out->out_bufs = v.out_bufs, out->ragged_map = v.ragged_map;
  }
  out->N = s.g.N, out->H = s.g.H, out->W = s.g.W, out->Cin = s.g.Cin, out->Cout = s.g.Cout, out->k = s.g.kh;
  out->stride = s.g.stride, out->pad = s.g.pad, out->dil = s.g.dil, out->relu = s.g.relu;
  if (s.x2 != nullptr) out->H2 = s.g2.H, out->W2 = s.g2.W, out->Cin2 = s.g2.Cin, out->stride2 = s.g2.stride;
  out->level = s.level;
  const bool stem = s.kind == 0 || s.kind == 5;
  out->x = stem ? (s.kind == 5 ? off(s.residual) : -1) : off(s.x);
  out->x2 = off(s.x2);
  out->residual = (s.kind == 2 || s.kind == 3) ? off(s.residual) : -1;
  out->y = s.kind == 4 ? -1 : off(s.y);
  out->levels = std::get<5>(p->steps_key) ? (int64_t)(2 * big + 2 * small) : -1;
  return 0;
}
