// C ABI + host orchestration of the DeepWMH / nnU-Net 3d_fullres inference path on one B200.
// See include/deepwmh_b200.h for the contract and the reference lines each entry point replaces.
#include "../../include/deepwmh_b200.h"

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "kernels_scan.cuh"
#include "kernels_ccl.cuh"
#include "kernels_conv_generic.cuh"
#include "conv_tcgen05.cuh"

using namespace dwmh;

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  g_err = buf;
  return 1;
}
#define CU_TRY(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) \
  return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); } while (0)
#define DW_TRY(expr) do { int r__ = (expr); if (r__) return r__; } while (0)

// Entry points run on the context's device and leave the caller's current device as they found it.
struct DevGuard {
  int prev = -1; bool ok = false;
  explicit DevGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
    if (prev == dev) prev = -1;
  }
  ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define DEV_GUARD(dev) DevGuard dev_guard__(dev); if (!dev_guard__.ok) return fail("cudaSetDevice(%d) failed", (int)(dev))

extern "C" const char* dwmh_last_error(void) { return g_err.c_str(); }
extern "C" void dwmh_internal_set_error(const char* msg) { g_err = msg ? msg : ""; }   // for the other translation units (stage1.cu)
extern "C" int dwmh_version(void) { return 100; }

// ------------------------------------------------------------------------------------------------
// network plan
// ------------------------------------------------------------------------------------------------
enum LayerKind { L_FIRST = 0, L_CONV = 1, L_TCONV = 2 };

// largest output edge of a normalised conv whose raw output is stored in fp32 (Layer::raw32)
constexpr int RAW32_MAX_EDGE = 64;

struct Layer {
  LayerKind kind;
  std::string name;                 // nnU-Net module prefix
  int c0 = 0, c1 = 0, cout = 0;     // input channels (c1 = concat partner), output channels
  int k[3] = {3, 3, 3}, s[3] = {1, 1, 1};
  int in_sp[3], out_sp[3];
  int in0 = -1, in1 = -1;           // producing layer indices (-1 = network input)
  bool has_norm = false;
  bool normalized_in_place = false; // apply kernel run after this layer
  // host copies (PyTorch layout)
  std::vector<float> w, gamma, beta;
  std::vector<int64_t> wshape;
  bool have_w = false, have_g = false, have_b = false;
  // device
  void* out = nullptr;              // [maxN][cout/8][V][8] T: normalised+activated (raw for the last conv / tconv)
  void* raw = nullptr;              // raw conv output; == out (normalised in place) unless raw32
  bool fused_norm = false;          // no norm pass: the (single) consumer applies InstanceNorm+LeakyReLU on load
  bool raw32 = false;               // raw output kept in fp32 (low-resolution layers: one rounding less per layer)
  void* s2d = nullptr;              // parity-split copy for a strided tcgen05 consumer
  int s2d_s[3] = {1, 1, 1};
  float* w_dev = nullptr;           // generic packing
  float* gamma_dev = nullptr; float* beta_dev = nullptr;
  double* sums = nullptr;           // into the stats arena: [maxN][cout][2] fp64
  bool stats_mean_var = false;      // sums hold {mean, variance} (tcgen05 path) instead of {sum, sum of squares}
  TcLayer tc;                       // tcgen05 packing / tensor maps (valid iff tc.enabled)
  int64_t vin() const { return (int64_t)in_sp[0] * in_sp[1] * in_sp[2]; }
  int64_t vout() const { return (int64_t)out_sp[0] * out_sp[1] * out_sp[2]; }
  double flops_per_sample() const {
    if (kind == L_TCONV) return 2.0 * vout() * c0 * cout;
    return 2.0 * vout() * (double)(k[0] * k[1] * k[2]) * (c0 + c1) * cout;
  }
};

struct dwmh_ctx {
  int device = 0;
  dwmh_net_desc d{};
  bool bf16 = false;
  int max_batch = 8;
  int elt = 2;
  std::vector<Layer> layers;
  int last_conv = -1;
  // head
  std::vector<float> w_head; bool have_head = false; float* w_head_dev = nullptr;
  bool committed = false;
  bool force_generic = false;
  // workspaces
  double* stats_arena = nullptr; size_t stats_bytes = 0;
  StatPartial* stat_partials = nullptr; size_t stat_partials_cap = 0;   // per-CTA Welford partials of the layer in flight
  float* probs = nullptr;            // [maxN][2][P]
  bool buffers_ready = false;
  dwmh_ctx* lender = nullptr;        // dwmh_create_like: activation workspaces are borrowed from this context
  float* gauss_dev = nullptr; std::vector<float> gauss_host; bool gauss_custom = false;
  SampleMeta* metas_dev = nullptr; size_t metas_cap = 0;
  double* zs_acc = nullptr;          // z-score: [0..2] totals for the host, [4 ...] one {sum, sum of squares, count} slot per CTA
  unsigned long long* zs_barrier = nullptr; unsigned long long zs_target = 0; int zs_grid = 0;
  int* ccl_labels = nullptr; int* ccl_sizes = nullptr; size_t ccl_cap_l = 0, ccl_cap_s = 0;   // dwmh_remove_sparks workspace
  // host-buffer path (grow only)
  float* hv_vol = nullptr; float* hv_pad = nullptr; float* hv_agg = nullptr; float* hv_wgt = nullptr; uint8_t* hv_seg = nullptr;
  size_t hv_vol_cap = 0, hv_pad_cap = 0, hv_agg_cap = 0, hv_wgt_cap = 0, hv_seg_cap = 0;
  // counters / timing
  int64_t launches = 0; double conv_flops = 0.0;
  bool stage_timing = false; float stage_ms[4] = {0, 0, 0, 0};
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  // per-launch timing by kernel class (stage timing only): 0 = conv3_tc_kernel, 1 = instnorm_lrelu_kernel, 2 = head_softmax_kernel
  std::vector<cudaEvent_t> tcev; std::vector<int> tcev_cls; int tcev_used = 0;
  double tc_ms = 0.0, tc_flops = 0.0, tc_launches = 0.0;
  double cls_ms[3] = {0, 0, 0}, cls_bytes[3] = {0, 0, 0}, cls_launches[3] = {0, 0, 0};
  int num_sms = 148;
  int64_t P() const { return (int64_t)d.patch_size[0] * d.patch_size[1] * d.patch_size[2]; }
};

static int build_plan(dwmh_ctx* c) {
  const dwmh_net_desc& d = c->d;
  const int np = d.num_pool;
  std::vector<int> f(np + 1);
  f[0] = d.base_num_features;
  for (int i = 1; i <= np; ++i) f[i] = std::min((int)std::nearbyint(f[i - 1] * 2.0), d.max_num_features);
  std::vector<std::array<int, 3>> sp(np + 1);
  sp[0] = {d.patch_size[0], d.patch_size[1], d.patch_size[2]};
  for (int i = 1; i <= np; ++i)
    for (int a = 0; a < 3; ++a) {
      const int pk = d.pool_op_kernel_sizes[i - 1][a];
      if (pk != 1 && pk != 2) return fail("pool_op_kernel_sizes[%d][%d]=%d unsupported (1 or 2)", i - 1, a, pk);
      if (sp[i - 1][a] % pk) return fail("patch_size axis %d not divisible by the pooling product", a);
      sp[i][a] = sp[i - 1][a] / pk;
    }
  for (int i = 0; i <= np; ++i) {
    if (f[i] % 32) return fail("feature count %d is not a multiple of 32 (unsupported)", f[i]);
    for (int a = 0; a < 3; ++a)
      if (d.conv_kernel_sizes[i][a] != 1 && d.conv_kernel_sizes[i][a] != 3)
        return fail("conv_kernel_sizes[%d][%d]=%d unsupported (1 or 3)", i, a, d.conv_kernel_sizes[i][a]);
  }
  auto add_conv = [&](const std::string& name, int c0, int c1, int cout, const int* k, const int* s,
                      const std::array<int, 3>& isp, const std::array<int, 3>& osp, int in0, int in1, bool first) {
    Layer L;
    L.kind = first ? L_FIRST : L_CONV; L.name = name; L.c0 = c0; L.c1 = c1; L.cout = cout;
    for (int a = 0; a < 3; ++a) { L.k[a] = k[a]; L.s[a] = s ? s[a] : 1; L.in_sp[a] = isp[a]; L.out_sp[a] = osp[a]; }
    L.in0 = in0; L.in1 = in1; L.has_norm = true;
    c->layers.push_back(L);
    return (int)c->layers.size() - 1;
  };
  char nm[128];
  int cur = -1, cin = d.in_channels;
  std::vector<int> skip(np);
  for (int e = 0; e < np; ++e) {
    snprintf(nm, sizeof nm, "conv_blocks_context.%d.blocks.0", e);
    cur = add_conv(nm, cin, 0, f[e], d.conv_kernel_sizes[e], e > 0 ? d.pool_op_kernel_sizes[e - 1] : nullptr,
                   e > 0 ? sp[e - 1] : sp[0], sp[e], cur, -1, e == 0);
    snprintf(nm, sizeof nm, "conv_blocks_context.%d.blocks.1", e);
    cur = add_conv(nm, f[e], 0, f[e], d.conv_kernel_sizes[e], nullptr, sp[e], sp[e], cur, -1, false);
    skip[e] = cur; cin = f[e];
  }
  snprintf(nm, sizeof nm, "conv_blocks_context.%d.0.blocks.0", np);
  cur = add_conv(nm, cin, 0, f[np], d.conv_kernel_sizes[np], d.pool_op_kernel_sizes[np - 1], sp[np - 1], sp[np], cur, -1, false);
  snprintf(nm, sizeof nm, "conv_blocks_context.%d.1.blocks.0", np);
  cur = add_conv(nm, f[np], 0, f[np], d.conv_kernel_sizes[np], nullptr, sp[np], sp[np], cur, -1, false);
  int ccur = f[np];
  for (int u = 0; u < np; ++u) {
    const int e = np - 1 - u, sc = f[e];
    Layer T;
    T.kind = L_TCONV; snprintf(nm, sizeof nm, "tu.%d", u); T.name = nm;
    T.c0 = ccur; T.cout = sc;
    for (int a = 0; a < 3; ++a) { T.k[a] = T.s[a] = d.pool_op_kernel_sizes[np - 1 - u][a]; T.in_sp[a] = sp[e + 1][a]; T.out_sp[a] = sp[e][a]; }
    T.in0 = cur; T.has_norm = false;
    c->layers.push_back(T);
    const int tu = (int)c->layers.size() - 1;
    snprintf(nm, sizeof nm, "conv_blocks_localization.%d.0.blocks.0", u);
    cur = add_conv(nm, sc, sc, sc, d.conv_kernel_sizes[np - u], nullptr, sp[e], sp[e], tu, skip[e], false);
    snprintf(nm, sizeof nm, "conv_blocks_localization.%d.1.blocks.0", u);
    cur = add_conv(nm, sc, 0, sc, d.conv_kernel_sizes[np - u], nullptr, sp[e], sp[e], cur, -1, false);
    ccur = sc;
  }
  c->last_conv = cur;
  if (c->layers[0].cout % 8) return fail("base_num_features must be a multiple of 8");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// life cycle
// ------------------------------------------------------------------------------------------------
// Model shapes this library runs; checked before any device work, so an unsupported model fails the same way everywhere.
static int check_model_bounds(const dwmh_net_desc* d) {
  if (d->in_channels < 1 || d->in_channels > DWMH_MAX_IN_CHANNELS)
    return fail("dwmh_create: in_channels=%d unsupported (1 <= in_channels <= %d: the first conv keeps 4 input slices and one "
                "weight tile per modality in one SM's shared memory)", d->in_channels, DWMH_MAX_IN_CHANNELS);
  if (d->num_classes < 2 || d->num_classes > DWMH_MAX_CLASSES)
    return fail("dwmh_create: num_classes=%d unsupported (2 <= num_classes <= %d: the head keeps every class's logits of two "
                "voxels in registers)", d->num_classes, DWMH_MAX_CLASSES);
  if (d->in_channels > 1 && d->base_num_features > 32)
    return fail("dwmh_create: base_num_features=%d with in_channels=%d unsupported (the multi-modality first conv has at most 32 "
                "output channels)", d->base_num_features, d->in_channels);
  return 0;
}

extern "C" int dwmh_create(dwmh_ctx** out, int device, const dwmh_net_desc* desc) {
  if (!out || !desc) return fail("dwmh_create: null argument");
  if (desc->struct_size == (int32_t)sizeof(dwmh_net_desc)) DW_TRY(check_model_bounds(desc));
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("dwmh_create: no CUDA device visible (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail("dwmh_create: device %d out of range (%d devices)", device, ndev);
  if (desc->struct_size != (int32_t)sizeof(dwmh_net_desc))
    return fail("dwmh_create: dwmh_net_desc.struct_size is %d, this library expects %d (set it to sizeof(dwmh_net_desc); "
                "a stale binding of the struct would otherwise be read past its end)", desc->struct_size, (int)sizeof(dwmh_net_desc));
  DEV_GUARD(device);
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail("dwmh_create: device %d is sm_%d%d; this build targets sm_100a (B200) only", device, prop.major, prop.minor);
  if (desc->num_pool < 1 || desc->num_pool > DWMH_MAX_POOL) return fail("num_pool out of range");
  dwmh_ctx* c = new dwmh_ctx();
  c->device = device; c->d = *desc; c->bf16 = desc->act_dtype == 1; c->num_sms = prop.multiProcessorCount;
  c->max_batch = desc->max_batch > 0 ? desc->max_batch : 8;
  if (build_plan(c)) { delete c; return 1; }
  for (int i = 0; i < 4; ++i) cudaEventCreate(&c->ev[i]);
  *out = c;
  return 0;
}

extern "C" int dwmh_create_like(dwmh_ctx** out, dwmh_ctx* parent) {
  if (!out || !parent) return fail("dwmh_create_like: null argument");
  if (parent->lender) return fail("dwmh_create_like: the parent itself borrows its workspaces; pass the owning context");
  if (!parent->buffers_ready) return fail("dwmh_create_like: commit the parent's weights first (its workspaces do not exist yet)");
  dwmh_ctx* c = nullptr;
  DW_TRY(dwmh_create(&c, parent->device, &parent->d));
  c->max_batch = parent->max_batch;
  c->lender = parent;
  *out = c;
  return 0;
}

static void free_dev(void* p) { if (p) cudaFree(p); }

extern "C" int dwmh_destroy(dwmh_ctx* c) {
  if (!c) return 0;
  DevGuard dg(c->device);
  cudaDeviceSynchronize();
  for (auto& L : c->layers) {
    if (!c->lender) { if (L.raw != L.out) free_dev(L.raw); free_dev(L.out); free_dev(L.s2d); }
    free_dev(L.w_dev); free_dev(L.gamma_dev); free_dev(L.beta_dev); tc_free(L.tc);
  }
  if (!c->lender) { free_dev(c->stats_arena); free_dev(c->probs); free_dev(c->stat_partials); }
  free_dev(c->w_head_dev); free_dev(c->gauss_dev); free_dev(c->metas_dev); free_dev(c->zs_acc); free_dev(c->zs_barrier);
  free_dev(c->hv_vol); free_dev(c->hv_pad); free_dev(c->hv_agg); free_dev(c->hv_wgt); free_dev(c->hv_seg);
  free_dev(c->ccl_labels); free_dev(c->ccl_sizes);
  for (int i = 0; i < 4; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  for (auto e : c->tcev) cudaEventDestroy(e);
  delete c;
  return 0;
}

extern "C" int dwmh_num_layers(dwmh_ctx* c) { return c ? (int)c->layers.size() : -1; }
extern "C" int dwmh_layer_kernel_kind(dwmh_ctx* c, int32_t i) {
  if (!c || i < 0 || i >= (int)c->layers.size()) return -1;
  return (c->layers[i].tc.enabled && !c->force_generic) ? 1 : 0;
}
extern "C" int dwmh_layer_norm_on_load(dwmh_ctx* c, int32_t i) {
  if (!c || i < 0 || i >= (int)c->layers.size()) return -1;
  return (c->layers[i].fused_norm && !c->force_generic) ? 1 : 0;
}
extern "C" int dwmh_set_force_generic(dwmh_ctx* c, int32_t on) { if (!c) return fail("null ctx"); c->force_generic = on != 0; return 0; }
extern "C" int dwmh_get_counters(dwmh_ctx* c, int64_t* k, double* f) { if (!c) return fail("null ctx"); if (k) *k = c->launches; if (f) *f = c->conv_flops; return 0; }
extern "C" int dwmh_set_stage_timing(dwmh_ctx* c, int32_t on) { if (!c) return fail("null ctx"); c->stage_timing = on != 0; return 0; }
extern "C" int dwmh_get_stage_timing(dwmh_ctx* c, float out[4]) { if (!c) return fail("null ctx"); memcpy(out, c->stage_ms, sizeof c->stage_ms); return 0; }
extern "C" int dwmh_get_kernel_timing(dwmh_ctx* c, double out[9]) {
  if (!c) return fail("null ctx");
  for (int i = 0; i < 3; ++i) { out[3 * i] = c->cls_ms[i]; out[3 * i + 1] = c->cls_bytes[i]; out[3 * i + 2] = c->cls_launches[i]; }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// weights
// ------------------------------------------------------------------------------------------------
static bool ends_with(const std::string& s, const char* suf) {
  const size_t n = strlen(suf);
  return s.size() >= n && s.compare(s.size() - n, n, suf) == 0;
}

extern "C" int dwmh_set_weight(dwmh_ctx* c, const char* key_c, const float* data, const int64_t* shape, int32_t ndim) {
  if (!c || !key_c || !data || !shape) return fail("dwmh_set_weight: null argument");
  std::string key(key_c);
  if (key.rfind("module.", 0) == 0) key = key.substr(7);
  int64_t numel = 1;
  for (int i = 0; i < ndim; ++i) numel *= shape[i];
  c->committed = false;
  if (key.rfind("seg_outputs.", 0) == 0) {
    const int u = atoi(key.c_str() + 12);
    if (u != c->d.num_pool - 1) return 0;                       // deep-supervision heads: discarded at inference
    const int C = c->layers[c->last_conv].cout;
    if (numel != (int64_t)c->d.num_classes * C) return fail("%s: expected %d x %d elements, got %lld", key_c, c->d.num_classes, C, (long long)numel);
    c->w_head.assign(data, data + numel); c->have_head = true;
    return 0;
  }
  for (auto& L : c->layers) {
    if (key.rfind(L.name + ".", 0) != 0) continue;
    const std::string suf = key.substr(L.name.size());
    if (L.kind == L_TCONV) {
      if (suf != ".weight") return fail("unexpected key %s", key_c);
      const int64_t want = (int64_t)L.c0 * L.cout * L.k[0] * L.k[1] * L.k[2];
      if (numel != want || ndim != 5 || shape[0] != L.c0 || shape[1] != L.cout) return fail("%s: shape mismatch (want [%d,%d,%d,%d,%d])", key_c, L.c0, L.cout, L.k[0], L.k[1], L.k[2]);
      L.w.assign(data, data + numel); L.have_w = true;
      return 0;
    }
    if (suf == ".conv.weight") {
      const int cin = L.c0 + L.c1;
      if (ndim != 5 || shape[0] != L.cout || shape[1] != cin || shape[2] != L.k[0] || shape[3] != L.k[1] || shape[4] != L.k[2])
        return fail("%s: shape mismatch (want [%d,%d,%d,%d,%d])", key_c, L.cout, cin, L.k[0], L.k[1], L.k[2]);
      L.w.assign(data, data + numel); L.have_w = true;
      return 0;
    }
    if (suf == ".conv.bias") return 0;          // cancels under InstanceNorm (SURVEY.md A1); accepted, unused
    if (suf == ".instnorm.weight") { if (numel != L.cout) return fail("%s: size", key_c); L.gamma.assign(data, data + numel); L.have_g = true; return 0; }
    if (suf == ".instnorm.bias") { if (numel != L.cout) return fail("%s: size", key_c); L.beta.assign(data, data + numel); L.have_b = true; return 0; }
    return fail("unexpected key %s", key_c);
  }
  return fail("unknown state_dict key %s", key_c);
}

static float round_act(float v, bool bf16) {
  return bf16 ? __bfloat162float(__float2bfloat16_rn(v)) : __half2float(__float2half_rn(v));
}

template <typename V>
static int upload(V** dst, const std::vector<V>& src) {
  if (*dst) { cudaFree(*dst); *dst = nullptr; }
  CU_TRY(cudaMalloc((void**)dst, src.size() * sizeof(V)));
  CU_TRY(cudaMemcpy(*dst, src.data(), src.size() * sizeof(V), cudaMemcpyHostToDevice));
  return 0;
}

extern "C" int dwmh_commit_weights(dwmh_ctx* c) {
  if (!c) return fail("null ctx");
  DEV_GUARD(c->device);
  if (!c->have_head) return fail("missing weight seg_outputs.%d.weight", c->d.num_pool - 1);
  for (auto& L : c->layers) {
    if (!L.have_w) return fail("missing weight for %s", L.name.c_str());
    if (L.has_norm && (!L.have_g || !L.have_b)) return fail("missing instnorm parameters for %s", L.name.c_str());
  }
  const int maxN = c->max_batch;
  const int nL = (int)c->layers.size();
  // ---- shared: weight packing for the CUDA-core kernels, norm parameters ----
  for (auto& L : c->layers) {
    const int taps = L.k[0] * L.k[1] * L.k[2];
    // fp32 raw storage of conv outputs (profiles/precision_full_r01.txt): those layers then round once
    // (operand) instead of twice (storage + operand)
    L.raw32 = L.kind == L_CONV && L.has_norm && (int)(&L - c->layers.data()) != c->last_conv &&
              std::max(L.out_sp[0], std::max(L.out_sp[1], L.out_sp[2])) <= RAW32_MAX_EDGE;
    std::vector<float> pk;
    if (L.kind == L_FIRST) {
      // [modality][tap][Cout] from PyTorch's [Cout][modality][tap]
      pk.resize((size_t)L.c0 * taps * L.cout);
      for (int co = 0; co < L.cout; ++co) for (int m = 0; m < L.c0; ++m) for (int t = 0; t < taps; ++t)
        pk[((size_t)m * taps + t) * L.cout + co] = L.w[((size_t)co * L.c0 + m) * taps + t];
    } else if (L.kind == L_CONV) {
      const int cin = L.c0 + L.c1, ncob = L.cout / GC_COB;
      pk.resize((size_t)cin * L.cout * taps);
      for (int co = 0; co < L.cout; ++co) for (int ci = 0; ci < cin; ++ci) for (int t = 0; t < taps; ++t) {
        const size_t dst = ((((size_t)(ci >> 3) * ncob + co / GC_COB) * taps + t) * 8 + (ci & 7)) * GC_COB + co % GC_COB;
        pk[dst] = round_act(L.w[((size_t)co * cin + ci) * taps + t], c->bf16);
      }
    } else {
      pk.resize((size_t)L.c0 * L.cout * taps);
      for (int ci = 0; ci < L.c0; ++ci) for (int co = 0; co < L.cout; ++co) for (int t = 0; t < taps; ++t) {
        const size_t dst = (((size_t)(co / GC_COB) * taps + t) * L.c0 + ci) * GC_COB + co % GC_COB;
        pk[dst] = round_act(L.w[((size_t)ci * L.cout + co) * taps + t], c->bf16);
      }
    }
    DW_TRY(upload(&L.w_dev, pk));
    if (L.has_norm) { DW_TRY(upload(&L.gamma_dev, L.gamma)); DW_TRY(upload(&L.beta_dev, L.beta)); }
  }
  DW_TRY(upload(&c->w_head_dev, c->w_head));
  // which producers need a parity-split copy (strided tcgen05 consumer)
  for (auto& L : c->layers) {
    const bool strided = L.s[0] != 1 || L.s[1] != 1 || L.s[2] != 1;
    const bool k_ok = (L.k[0] == 3 || (L.k[0] == 1 && L.s[0] == 1)) && L.k[1] == 3 && L.k[2] == 3;      // what tc_prepare accepts
    if (L.kind == L_CONV && strided && k_ok && L.c0 % 16 == 0 && L.c1 == 0 && L.cout % 16 == 0)
      for (int a_ = 0; a_ < 3; ++a_) c->layers[L.in0].s2d_s[a_] = L.s[a_];
  }
  // ---- activation buffers, statistics, probabilities (allocated once per context) ----
  size_t stat_doubles = 0;
  for (auto& L : c->layers) if (L.has_norm) stat_doubles += (size_t)maxN * L.cout * 2;
  c->stats_bytes = stat_doubles * sizeof(double);
  if (!c->buffers_ready && c->lender) {
    dwmh_ctx* o = c->lender;
    if (o->layers.size() != c->layers.size() || o->max_batch != maxN) return fail("dwmh_commit_weights: lender context does not match");
    c->stats_arena = o->stats_arena; c->probs = o->probs;
    for (int i = 0; i < nL; ++i) {
      Layer& L = c->layers[i]; const Layer& S = o->layers[i];
      if (L.raw32 != S.raw32) return fail("dwmh_commit_weights: lender context does not match (raw storage of %s)", L.name.c_str());
      L.sums = S.sums; L.out = S.out; L.raw = S.raw; L.s2d = S.s2d;
    }
    c->buffers_ready = true;
  }
  if (!c->buffers_ready) {
    CU_TRY(cudaMalloc((void**)&c->stats_arena, c->stats_bytes));
    CU_TRY(cudaMalloc((void**)&c->probs, (size_t)maxN * c->d.num_classes * c->P() * sizeof(float)));
    size_t off = 0;
    for (int i = 0; i < nL; ++i) {
      Layer& L = c->layers[i];
      if (L.has_norm) { L.sums = c->stats_arena + off; off += (size_t)maxN * L.cout * 2; }
      CU_TRY(cudaMalloc(&L.out, (size_t)maxN * L.cout * L.vout() * c->elt));
      if (L.raw32) CU_TRY(cudaMalloc(&L.raw, (size_t)maxN * L.cout * L.vout() * 4)); else L.raw = L.out;
      const bool need_s2d = L.s2d_s[0] * L.s2d_s[1] * L.s2d_s[2] > 1;
      if (need_s2d) CU_TRY(cudaMalloc(&L.s2d, (size_t)maxN * L.cout * L.vout() * c->elt));
    }
    c->buffers_ready = true;
  }
  // ---- tcgen05 packing + tensor maps ----
  for (int i = 0; i < nL; ++i) {
    Layer& L = c->layers[i];
    tc_free(L.tc);
    std::string why;
    if (L.kind == L_FIRST) {
      if (L.k[0] == 3 && L.k[1] == 3 && L.k[2] == 3 && L.c0 <= DWMH_MAX_IN_CHANNELS) {
        std::vector<float> w27((size_t)L.c0 * 27 * L.cout);      // [modality][tap][Cout]
        for (int co = 0; co < L.cout; ++co) for (int m = 0; m < L.c0; ++m) for (int t = 0; t < 27; ++t)
          w27[((size_t)m * 27 + t) * L.cout + co] = L.w[((size_t)co * L.c0 + m) * 27 + t];
        if (tc_prepare_first(L.tc, w27, L.cout, L.out_sp, c->bf16, L.raw, &why, L.c0))
          if (!why.empty()) return fail("tcgen05 setup for %s failed: %s", L.name.c_str(), why.c_str());
      }
      continue;
    }
    const void* in0 = c->layers[L.in0].out;
    const void* in1 = L.in1 >= 0 ? c->layers[L.in1].out : nullptr;
    const bool strided = L.kind == L_CONV && (L.s[0] != 1 || L.s[1] != 1 || L.s[2] != 1);
    if (strided && c->layers[L.in0].s2d) in0 = c->layers[L.in0].s2d;
    if (L.kind == L_TCONV) {
      if (tc_prepare_tconv(L.tc, L.w, L.c0, L.cout, L.s, L.in_sp, maxN, c->bf16, in0, L.out, &why))
        if (!why.empty()) return fail("tcgen05 setup for %s failed: %s", L.name.c_str(), why.c_str());
    } else if (tc_prepare(L.tc, L.w, L.c0, L.c1, L.cout, L.k, L.s, L.in_sp, L.out_sp, maxN, c->bf16, in0, in1, L.raw, L.raw32, &why)) {
      if (!why.empty()) return fail("tcgen05 setup for %s failed: %s", L.name.c_str(), why.c_str());
    }
  }
  // scratch for the per-CTA statistics partials of one launch (largest layer x batch size)
  {
    size_t need = 0;
    for (auto& L : c->layers)
      if (L.tc.enabled)
        for (int nb = 1; nb <= maxN; ++nb) need = std::max(need, tc_partials_needed(L.tc.kp, nb, c->num_sms));
    if (c->lender) {
      if (need > c->lender->stat_partials_cap) return fail("dwmh_commit_weights: lender's statistics scratch is too small");
      c->stat_partials = c->lender->stat_partials; c->stat_partials_cap = c->lender->stat_partials_cap;
    } else if (need > c->stat_partials_cap) {
      free_dev(c->stat_partials); c->stat_partials = nullptr; c->stat_partials_cap = 0;
      CU_TRY(cudaMalloc((void**)&c->stat_partials, need * sizeof(StatPartial)));
      c->stat_partials_cap = need;
    }
  }
  // norm-on-load fusion: producer P feeds exactly one consumer, a tcgen05 layer whose shape supports the in-kernel
  // transform, and P's raw output is fp16 (the consumer's loaders read it into registers and transform it there)
  {
    std::vector<int> uses(nL, 0);
    for (auto& L : c->layers) { if (L.in0 >= 0) uses[L.in0]++; if (L.in1 >= 0) uses[L.in1]++; }
    for (auto& L : c->layers) L.fused_norm = false;
    for (auto& L : c->layers) {
      if (L.kind != L_CONV || !L.tc.enabled || !L.tc.xform_ok || L.in0 < 0) continue;
      Layer& P = c->layers[L.in0];
      if (P.has_norm && !P.raw32 && uses[L.in0] == 1 && P.s2d_s[0] * P.s2d_s[1] * P.s2d_s[2] == 1 && P.cout <= 64) P.fused_norm = true;
    }
  }
  if (!c->gauss_custom) {
    c->gauss_host.resize(c->P());
    DW_TRY(dwmh_gaussian_map(c->d.patch_size, 1.0 / 8, c->gauss_host.data()));
  }
  DW_TRY(upload(&c->gauss_dev, c->gauss_host));
  // opt in to large dynamic shared memory
  const int smem_max = 100 * 1024;
  if (c->bf16) {
    CU_TRY(cudaFuncSetAttribute(conv_generic_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    CU_TRY(cudaFuncSetAttribute(tconv_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
  } else {
    CU_TRY(cudaFuncSetAttribute(conv_generic_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    CU_TRY(cudaFuncSetAttribute(tconv_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
  }
  DW_TRY(tc_init_attributes(c->bf16));
  c->committed = true;
  return 0;
}

extern "C" int dwmh_set_importance_map(dwmh_ctx* c, const float* map_host) {
  if (!c || !map_host) return fail("null argument");
  DEV_GUARD(c->device);
  c->gauss_host.assign(map_host, map_host + c->P());
  c->gauss_custom = true;
  if (c->gauss_dev) CU_TRY(cudaMemcpy(c->gauss_dev, c->gauss_host.data(), c->P() * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// a8 / a9 host helpers
// ------------------------------------------------------------------------------------------------
static int steps_1d(int patch, int image, double step_size, std::vector<int>& out) {
  if (image < patch) return fail("image extent %d smaller than patch %d (pad first)", image, patch);
  if (!(step_size > 0.0 && step_size <= 1.0)) return fail("step_size must be in (0, 1]");
  const double target = patch * step_size;
  const int n = (int)std::ceil((image - patch) / target) + 1;
  const double actual = n > 1 ? (double)(image - patch) / (n - 1) : 99999999999.0;
  out.clear();
  for (int i = 0; i < n; ++i) out.push_back((int)std::nearbyint(actual * i));     // round-half-even == np.round
  return 0;
}

extern "C" int dwmh_compute_steps(const int32_t patch[3], const int32_t image[3], double step_size,
                                  int32_t* sx, int32_t* sy, int32_t* sz, int32_t max_steps, int32_t counts[3]) {
  int32_t* dst[3] = {sx, sy, sz};
  for (int a = 0; a < 3; ++a) {
    std::vector<int> s;
    DW_TRY(steps_1d(patch[a], image[a], step_size, s));
    if ((int)s.size() > max_steps) return fail("more than max_steps steps on axis %d", a);
    for (size_t i = 0; i < s.size(); ++i) dst[a][i] = s[i];
    counts[a] = (int)s.size();
  }
  return 0;
}

extern "C" int dwmh_gaussian_map(const int32_t patch[3], double sigma_scale, float* out) {
  // scipy.ndimage.gaussian_filter of a unit impulse at patch//2 (mode constant, truncate 4.0) is the
  // outer product of the three normalised 1-D kernels, evaluated in the same association order.
  std::vector<double> w[3];
  for (int a = 0; a < 3; ++a) {
    const double sigma = patch[a] * sigma_scale;
    const int lw = (int)(4.0 * sigma + 0.5);
    std::vector<double> k(2 * lw + 1);
    double sum = 0.0;
    for (int i = -lw; i <= lw; ++i) { k[i + lw] = std::exp(-0.5 / (sigma * sigma) * (double)i * i); sum += k[i + lw]; }
    w[a].assign(patch[a], 0.0);
    const int c = patch[a] / 2;
    for (int i = 0; i < patch[a]; ++i) { const int off = i - c; if (off >= -lw && off <= lw) w[a][i] = k[off + lw] / sum; }
  }
  const int64_t P = (int64_t)patch[0] * patch[1] * patch[2];
  std::vector<double> g(P);
  double mx = 0.0;
  for (int i = 0; i < patch[0]; ++i) for (int j = 0; j < patch[1]; ++j) for (int k = 0; k < patch[2]; ++k) {
    const double v = (w[0][i] * w[1][j]) * w[2][k];
    g[((int64_t)i * patch[1] + j) * patch[2] + k] = v; if (v > mx) mx = v;
  }
  float mn = INFINITY;
  for (int64_t i = 0; i < P; ++i) { out[i] = (float)(g[i] / mx * 1); if (out[i] != 0.f && out[i] < mn) mn = out[i]; }
  for (int64_t i = 0; i < P; ++i) if (out[i] == 0.f) out[i] = mn;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// a2 z-score
// ------------------------------------------------------------------------------------------------
extern "C" int dwmh_zscore(dwmh_ctx* c, float* vol, const int8_t* seg, int64_t n, int32_t mask_mode, double* stats_out, void* stream_) {
  if (!c || !vol) return fail("dwmh_zscore: null argument");
  if (mask_mode < 0 || mask_mode > 2) return fail("dwmh_zscore: mask_mode %d", mask_mode);
  if (mask_mode == 1 && !seg) return fail("dwmh_zscore: mask_mode 1 needs seg");
  if ((reinterpret_cast<uintptr_t>(vol) & 15) || (seg && (reinterpret_cast<uintptr_t>(seg) & 3))) return fail("dwmh_zscore: buffers must be 16-byte (vol) / 4-byte (seg) aligned");
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(c->device);
  if (!c->zs_acc) {
    // one cooperative launch: every CTA must be resident at once
    int per_sm = 0;
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, zscore_fused_kernel, 256, 0));
    if (per_sm < 1) return fail("dwmh_zscore: the fused kernel does not fit an SM");
    c->zs_grid = c->num_sms * std::min(per_sm, 4);
    CU_TRY(cudaMalloc((void**)&c->zs_acc, (4 + 3 * (size_t)c->zs_grid) * sizeof(double)));
    CU_TRY(cudaMalloc((void**)&c->zs_barrier, sizeof(unsigned long long)));
    CU_TRY(cudaMemset(c->zs_barrier, 0, sizeof(unsigned long long)));
    c->zs_target = 0;
  }
  {
    double* slots = c->zs_acc + 4; double* totals = c->zs_acc;
    unsigned long long target = c->zs_target + (unsigned long long)c->zs_grid;
    void* args[] = {(void*)&vol, (void*)&seg, (void*)&n, (void*)&mask_mode, (void*)&slots, (void*)&c->zs_barrier, (void*)&target, (void*)&totals};
    CU_TRY(cudaLaunchCooperativeKernel((const void*)zscore_fused_kernel, dim3(c->zs_grid), dim3(256), args, 0, st));
    c->zs_target = target;
  }
  c->launches += 1;
  CU_TRY(cudaGetLastError());
  if (stats_out) {
    double h[3];
    CU_TRY(cudaMemcpyAsync(h, c->zs_acc, sizeof h, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    const double cnt = h[2] > 0 ? h[2] : 1.0, m = h[0] / cnt;
    double var = h[1] / cnt - m * m; if (var < 0) var = 0;
    stats_out[0] = m; stats_out[1] = std::sqrt(var); stats_out[2] = h[2];
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
// head of a model with NC = 3 .. DWMH_MAX_CLASSES classes
template <typename T>
static int launch_head_c(int NC, dim3 grid, cudaStream_t st, const T* y, NormParams np, const float* w, float* probs, int C, int64_t V) {
  const size_t smem = (size_t)(2 + NC) * C * sizeof(float);
  switch (NC) {
#define DWMH_HEAD_C(K) case K: head_softmax_c_kernel<T, K><<<grid, 256, smem, st>>>(y, np, w, probs, C, V); return 0
    DWMH_HEAD_C(3); DWMH_HEAD_C(4); DWMH_HEAD_C(5); DWMH_HEAD_C(6); DWMH_HEAD_C(7); DWMH_HEAD_C(8);
#undef DWMH_HEAD_C
    default: return fail("internal: no head for %d classes", NC);
  }
}

// One batch of forwards on one stream.  Every conv / transposed conv is a conv3_tc_kernel launch (tcgen05) unless the layer
// shape is unsupported or dwmh_set_force_generic is on (CUDA-core cross-check kernels).
template <typename T>
static int forward_impl(dwmh_ctx* c, const float* src, int patch_mode, int SX, int SY, int SZ,
                        const SampleMeta* metas, int nb, cudaStream_t st) {
  if (nb > c->max_batch) return fail("forward: batch %d > max_batch %d", nb, c->max_batch);
  CU_TRY(cudaMemsetAsync(c->stats_arena, 0, c->stats_bytes, st));
  // stage timing: CUDA events around single launches, grouped by kernel class (the stats_reduce_kernel that follows a
  // conv launch is inside the conv's pair: it is part of producing the layer)
  auto cls_timed = [&](int cls, double bytes, auto&& launch) -> int {
    const bool timed = c->stage_timing && c->tcev_used + 2 <= (int)c->tcev.size();
    if (timed) CU_TRY(cudaEventRecord(c->tcev[c->tcev_used], st));
    DW_TRY(launch());
    if (timed) {
      CU_TRY(cudaEventRecord(c->tcev[c->tcev_used + 1], st));
      c->tcev_cls[c->tcev_used / 2] = cls; c->tcev_used += 2; c->cls_bytes[cls] += bytes; c->cls_launches[cls] += 1;
    }
    return 0;
  };
  auto tc_timed = [&](Layer& L, auto&& launch) -> int {
    DW_TRY(cls_timed(0, 0.0, launch));
    if (c->stage_timing) { c->tc_flops += L.flops_per_sample() * nb; c->tc_launches += 1; }
    c->launches += L.kind == L_TCONV ? 1 : 2;      // conv3_tc_kernel (+ stats_reduce_kernel)
    return 0;
  };
  auto norm_of = [&](Layer& L) { return NormParams{L.sums, L.gamma_dev, L.beta_dev, L.stats_mean_var ? 0.0 : 1.0 / (double)L.vout()}; };
  for (size_t li = 0; li < c->layers.size(); ++li) {
    Layer& L = c->layers[li];
    const int taps = L.k[0] * L.k[1] * L.k[2];
    const bool use_tc = L.tc.enabled && !c->force_generic;
    L.stats_mean_var = use_tc && L.has_norm;
    if (L.kind == L_FIRST && use_tc) {
      TcFirstSrc fs{src, metas, patch_mode, SY, SZ, patch_mode ? c->P() : (int64_t)SX * SY * SZ};
      DW_TRY(tc_timed(L, [&] { return tc_launch<T>(L.tc, nb, L.sums, c->stat_partials, c->num_sms, st, &g_err, nullptr, &fs); }));
    } else if (L.kind == L_FIRST) {
      FirstConvParams p;
      p.src = src; p.metas = metas; p.w = L.w_dev; p.out = L.raw; p.sums = L.sums; p.patch_mode = patch_mode;
      p.SX = SX; p.SY = SY; p.SZ = SZ; p.px = L.out_sp[0]; p.py = L.out_sp[1]; p.pz = L.out_sp[2];
      p.kd = L.k[0]; p.kh = L.k[1]; p.kw = L.k[2]; p.Cout = L.cout;
      p.Cin = L.c0; p.mstride = (int64_t)SX * SY * SZ;
      dim3 grid((unsigned)((L.vout() + 256 * FC_VPT - 1) / (256 * FC_VPT)), nb);
      const size_t smem = ((size_t)L.c0 * taps * L.cout + 2 * L.cout) * sizeof(float);
      if (L.c0 > 1) {
        if (taps == 27) conv_first_mm_kernel<T, true><<<grid, 256, smem, st>>>(p);
        else conv_first_mm_kernel<T, false><<<grid, 256, smem, st>>>(p);
      } else if (taps == 27 && L.cout <= 32 && L.out_sp[2] % 2 == 0) {
        dim3 grid2((unsigned)((L.vout() / 2 + 128 * FC_VPT - 1) / (128 * FC_VPT)), nb);
        conv_first_k3x2_kernel<T><<<grid2, 128, smem, st>>>(p);
      } else if (taps == 27) conv_first_kernel<T, true><<<grid, 256, smem, st>>>(p);
      else conv_first_kernel<T, false><<<grid, 256, smem, st>>>(p);
      c->launches++;
    } else if (L.kind == L_CONV && use_tc) {
      Layer& P = c->layers[L.in0];
      NormParams pn = norm_of(P);
      TcXform xf{pn.sums, pn.gamma, pn.beta, pn.inv_count, P.out};
      DW_TRY(tc_timed(L, [&] { return tc_launch<T>(L.tc, nb, L.sums, c->stat_partials, c->num_sms, st, &g_err, P.fused_norm ? &xf : nullptr); }));
    } else if (L.kind == L_CONV) {
      ConvParams p;
      p.in0 = c->layers[L.in0].out; p.C0 = L.c0;
      p.in1 = L.in1 >= 0 ? c->layers[L.in1].out : nullptr; p.C1 = L.c1;
      p.w = L.w_dev; p.out = L.raw; p.out32 = L.raw32 ? 1 : 0; p.sums = L.sums; p.N = nb;
      p.Di = L.in_sp[0]; p.Hi = L.in_sp[1]; p.Wi = L.in_sp[2]; p.Do = L.out_sp[0]; p.Ho = L.out_sp[1]; p.Wo = L.out_sp[2];
      p.Cout = L.cout; p.kd = L.k[0]; p.kh = L.k[1]; p.kw = L.k[2]; p.sd = L.s[0]; p.sh = L.s[1]; p.sw = L.s[2];
      const int tiles = ((p.Do + GC_TD - 1) / GC_TD) * ((p.Ho + GC_TH - 1) / GC_TH) * ((p.Wo + GC_TW - 1) / GC_TW);
      const int ed = (GC_TD - 1) * p.sd + p.kd, eh = (GC_TH - 1) * p.sh + p.kh, ew = (GC_TW - 1) * p.sw + p.kw;
      const size_t smem = (size_t)ed * eh * ew * 16 + (size_t)taps * 8 * GC_COB * sizeof(float);
      dim3 grid(tiles, L.cout / GC_COB, nb);
      conv_generic_kernel<T><<<grid, 128, smem, st>>>(p);
      c->launches++;
    } else if (use_tc) {
      DW_TRY(tc_timed(L, [&] { return tc_launch<T>(L.tc, nb, nullptr, nullptr, c->num_sms, st, &g_err); }));
    } else {
      TConvParams p;
      p.in = c->layers[L.in0].out; p.out = L.out; p.w = L.w_dev; p.N = nb; p.Cin = L.c0; p.Cout = L.cout;
      p.Di = L.in_sp[0]; p.Hi = L.in_sp[1]; p.Wi = L.in_sp[2]; p.sd = L.s[0]; p.sh = L.s[1]; p.sw = L.s[2];
      dim3 grid((unsigned)((L.vin() + 127) / 128), L.cout / GC_COB, nb);
      tconv_kernel<T><<<grid, 128, (size_t)L.c0 * GC_COB * sizeof(float), st>>>(p);
      c->launches++;
    }
    c->conv_flops += L.flops_per_sample() * nb;
    if (L.has_norm && (int)li != c->last_conv && !(L.fused_norm && !c->force_generic)) {
      const int64_t V = L.vout();
      const int gx = (int)std::min<int64_t>((V / 2 + 255) / 256, 1024);      // a thread handles voxel pairs (256-bit accesses)
      dim3 grid(std::max(gx, 1), nb * (L.cout >> 3));
      S2dParams sp{L.s2d, L.out_sp[0], L.out_sp[1], L.out_sp[2], L.s2d_s[0], L.s2d_s[1], L.s2d_s[2]};
      const double bytes = (double)nb * L.cout * V * ((L.raw32 ? 4 : 2) + 2 + (L.s2d ? 2 : 0));
      const bool quad = sp.dst && sp.sw == 2 && (sp.W & 3) == 0;              // parity-split copy written with 256-bit stores
      DW_TRY(cls_timed(1, bytes, [&] {
        if (quad) instnorm_lrelu_kernel<T, true><<<grid, 256, 0, st>>>(L.raw, L.raw32 ? 1 : 0, L.out, norm_of(L), L.cout, V, sp);
        else instnorm_lrelu_kernel<T><<<grid, 256, 0, st>>>(L.raw, L.raw32 ? 1 : 0, L.out, norm_of(L), L.cout, V, sp);
        return 0; }));
      c->launches++;
    }
  }
  // head: norm-on-load + 1x1x1 + softmax
  Layer& L = c->layers[c->last_conv];
  const int64_t head_items = (L.cout == 32 && (L.vout() & 1) == 0) ? L.vout() / 2 : L.vout();      // two voxels per thread in the usual head
  dim3 grid((unsigned)((head_items + 255) / 256), nb);
  const int NC = c->d.num_classes;
  DW_TRY(cls_timed(2, (double)nb * L.vout() * (2.0 * L.cout + 4.0 * NC), [&] {
    if (NC == 2) {
      head_softmax_kernel<T><<<grid, 256, 4 * L.cout * sizeof(float), st>>>((const T*)L.out, norm_of(L), c->w_head_dev, c->probs, L.cout, L.vout());
      return 0;
    }
    return launch_head_c<T>(NC, grid, st, (const T*)L.out, norm_of(L), c->w_head_dev, c->probs, L.cout, L.vout()); }));
  c->launches++;
  c->conv_flops += 2.0 * L.vout() * L.cout * c->d.num_classes * nb;
  CU_TRY(cudaGetLastError());
  return 0;
}

static int forward(dwmh_ctx* c, const float* src, int patch_mode, int SX, int SY, int SZ, const SampleMeta* metas, int nb, cudaStream_t st) {
  return c->bf16 ? forward_impl<__nv_bfloat16>(c, src, patch_mode, SX, SY, SZ, metas, nb, st)
                 : forward_impl<__half>(c, src, patch_mode, SX, SY, SZ, metas, nb, st);
}

extern "C" int dwmh_forward_patches(dwmh_ctx* c, const float* patches, int32_t n, float* probs_out, void* stream_) {
  if (!c || !patches || !probs_out) return fail("dwmh_forward_patches: null argument");
  if (!c->committed) return fail("dwmh_forward_patches: weights not committed");
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(c->device);
  const int64_t P = c->P();
  const int NM = c->d.in_channels, NC = c->d.num_classes;
  for (int b = 0; b < n; b += c->max_batch) {
    const int nb = std::min(c->max_batch, n - b);
    DW_TRY(forward(c, patches + (size_t)b * NM * P, 1, 0, 0, 0, nullptr, nb, st));
    CU_TRY(cudaMemcpyAsync(probs_out + (size_t)b * NC * P, c->probs, (size_t)nb * NC * P * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  return 0;
}

extern "C" int dwmh_debug_layer_output(dwmh_ctx* c, int32_t li, float* out, int64_t capacity, int32_t dims[5], void* stream_) {
  if (!c || li < 0 || li >= (int)c->layers.size()) return fail("dwmh_debug_layer_output: bad layer index");
  Layer& L = c->layers[li];
  const int n = c->max_batch;
  dims[0] = n; dims[1] = L.cout; dims[2] = L.out_sp[0]; dims[3] = L.out_sp[1]; dims[4] = L.out_sp[2];
  if (!out) return 0;                         // dims query
  const int64_t need = (int64_t)n * L.cout * L.vout();
  int nn = n;
  if (capacity < need) { nn = (int)(capacity / ((int64_t)L.cout * L.vout())); dims[0] = nn; if (nn <= 0) return fail("capacity too small"); }
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(c->device);
  // the last conv is kept raw (the head normalises on load): normalise here for a uniform view
  NormParams np{nullptr, nullptr, nullptr, 0.0};
  if ((int)li == c->last_conv || (L.fused_norm && !c->force_generic)) np = NormParams{L.sums, L.gamma_dev, L.beta_dev, L.stats_mean_var ? 0.0 : 1.0 / (double)L.vout()};
  if (c->bf16) unpack_layer_kernel<__nv_bfloat16><<<c->num_sms * 4, 256, 0, st>>>((const __nv_bfloat16*)L.out, np, out, nn, L.cout, L.vout());
  else unpack_layer_kernel<__half><<<c->num_sms * 4, 256, 0, st>>>((const __half*)L.out, np, out, nn, L.cout, L.vout());
  CU_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// a7/a11/a12 tiled prediction
// ------------------------------------------------------------------------------------------------
extern "C" int dwmh_predict_3d(dwmh_ctx* c, const float* vol, int32_t X, int32_t Y, int32_t Z, double step_size,
                               int32_t do_mirroring, int32_t mirror_axes_mask, int32_t use_gaussian,
                               float* agg, float* wgt, int32_t tile_begin, int32_t tile_end, void* stream_) {
  if (!c || !vol || !agg || !wgt) return fail("dwmh_predict_3d: null argument");
  if (!c->committed) return fail("dwmh_predict_3d: weights not committed");
  if (step_size > 1.0) return fail("step_size must be smaller than 1");
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(c->device);
  const int32_t* ps = c->d.patch_size;
  std::vector<int> steps[3];
  const int img[3] = {X, Y, Z};
  for (int a = 0; a < 3; ++a) DW_TRY(steps_1d(ps[a], img[a], step_size, steps[a]));
  const int ntiles = (int)(steps[0].size() * steps[1].size() * steps[2].size());
  if (tile_end < 0 || tile_end > ntiles) tile_end = ntiles;
  if (tile_begin < 0) tile_begin = 0;
  // mirror list: index m uses z if m&1, y if m&2, x if m&4; needs those axes enabled
  std::vector<int> mirrors;
  if (do_mirroring) {
    const int zbit = (mirror_axes_mask >> 2) & 1, ybit = (mirror_axes_mask >> 1) & 1, xbit = mirror_axes_mask & 1;
    for (int m = 0; m < 8; ++m) {
      if ((m & 1) && !zbit) continue;
      if ((m & 2) && !ybit) continue;
      if ((m & 4) && !xbit) continue;
      mirrors.push_back(m);
    }
  } else mirrors.push_back(0);
  const int M = (int)mirrors.size();
  const bool gauss = use_gaussian && ntiles > 1;
  const int nt = tile_end - tile_begin;
  if (nt <= 0) return 0;
  if (M > c->max_batch) return fail("max_batch %d smaller than the mirror count %d", c->max_batch, M);
  std::vector<SampleMeta> metas((size_t)nt * M);
  for (int t = 0; t < nt; ++t) {
    int lin = tile_begin + t;
    const int iz = lin % (int)steps[2].size(); lin /= (int)steps[2].size();
    const int iy = lin % (int)steps[1].size(); lin /= (int)steps[1].size();
    const int ix = lin;
    for (int m = 0; m < M; ++m) metas[(size_t)t * M + m] = SampleMeta{steps[0][ix], steps[1][iy], steps[2][iz], mirrors[m]};
  }
  if (c->metas_cap < metas.size()) {
    free_dev(c->metas_dev); c->metas_dev = nullptr;
    CU_TRY(cudaMalloc((void**)&c->metas_dev, metas.size() * sizeof(SampleMeta)));
    c->metas_cap = metas.size();
  }
  // pageable source: the copy is staged synchronously by the runtime, so `metas` may die afterwards
  CU_TRY(cudaMemcpyAsync(c->metas_dev, metas.data(), metas.size() * sizeof(SampleMeta), cudaMemcpyHostToDevice, st));
  const int tiles_per_batch = std::max(1, c->max_batch / M);
  const int64_t P = c->P();
  const int NC = c->d.num_classes;
  float conv_ms = 0.f, agg_ms = 0.f;
  if (c->stage_timing) {
    while (c->tcev.size() < 256) { cudaEvent_t e; CU_TRY(cudaEventCreate(&e)); c->tcev.push_back(e); }
    c->tcev_cls.assign(c->tcev.size() / 2, 0);
    c->tcev_used = 0; c->tc_ms = 0; c->tc_flops = 0; c->tc_launches = 0;
    for (int i = 0; i < 3; ++i) { c->cls_ms[i] = 0; c->cls_bytes[i] = 0; c->cls_launches[i] = 0; }
  }
  // Batches of forwards and the overlap-add of their tiles alternate on the caller's stream, tiles in order (deterministic).
  for (int t0 = 0; t0 < nt; t0 += tiles_per_batch) {
    const int tb = std::min(tiles_per_batch, nt - t0);
    if (c->stage_timing) CU_TRY(cudaEventRecord(c->ev[0], st));
    DW_TRY(forward(c, vol, 0, X, Y, Z, c->metas_dev + (size_t)t0 * M, tb * M, st));
    if (c->stage_timing) CU_TRY(cudaEventRecord(c->ev[1], st));
    for (int t = 0; t < tb; ++t) {
      if (NC == 2)
        aggregate_tile_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(
            c->probs + (size_t)t * M * 2 * P, c->metas_dev + (size_t)(t0 + t) * M, M, gauss ? c->gauss_dev : nullptr,
            agg, wgt, ps[0], ps[1], ps[2], X, Y, Z);
      else
        aggregate_tile_c_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(
            c->probs + (size_t)t * M * NC * P, c->metas_dev + (size_t)(t0 + t) * M, M, NC, gauss ? c->gauss_dev : nullptr,
            agg, wgt, ps[0], ps[1], ps[2], X, Y, Z);
      c->launches++;
    }
    if (c->stage_timing) {
      CU_TRY(cudaEventRecord(c->ev[2], st));
      CU_TRY(cudaEventSynchronize(c->ev[2]));
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, c->ev[0], c->ev[1]); cudaEventElapsedTime(&b, c->ev[1], c->ev[2]);
      conv_ms += a; agg_ms += b;
      for (int i = 0; i + 1 < c->tcev_used; i += 2) {
        float t = 0; cudaEventElapsedTime(&t, c->tcev[i], c->tcev[i + 1]);
        c->cls_ms[c->tcev_cls[i / 2]] += t;
        if (c->tcev_cls[i / 2] == 0) c->tc_ms += t;
      }
      c->tcev_used = 0;
    }
  }
  CU_TRY(cudaGetLastError());
  if (c->stage_timing) { c->stage_ms[0] = conv_ms; c->stage_ms[1] = agg_ms; c->stage_ms[2] = (float)c->tc_ms; c->stage_ms[3] = (float)(c->tc_flops / 1e12); }
  return 0;
}

extern "C" int dwmh_weight_map(dwmh_ctx* c, int32_t X, int32_t Y, int32_t Z, double step_size, int32_t use_gaussian, float* wgt, void* stream_) {
  if (!c || !wgt) return fail("dwmh_weight_map: null argument");
  if (!c->gauss_dev) return fail("dwmh_weight_map: weights not committed (no importance map yet)");
  DEV_GUARD(c->device);
  const int32_t* ps = c->d.patch_size;
  const int img[3] = {X, Y, Z};
  TileSteps ts;
  int ntiles = 1;
  for (int a = 0; a < 3; ++a) {
    std::vector<int> s_;
    DW_TRY(steps_1d(ps[a], img[a], step_size, s_));
    if ((int)s_.size() > WM_MAX_STEPS) return fail("dwmh_weight_map: more than %d tiles along axis %d", WM_MAX_STEPS, a);
    ts.n[a] = (int)s_.size();
    for (size_t i = 0; i < s_.size(); ++i) ts.s[a][i] = s_[i];
    ntiles *= (int)s_.size();
  }
  const bool gauss = use_gaussian && ntiles > 1;
  weight_map_kernel<<<c->num_sms * 8, 256, 0, (cudaStream_t)stream_>>>(gauss ? c->gauss_dev : nullptr, wgt, ts, ps[0], ps[1], ps[2], X, Y, Z);
  c->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_finalize(dwmh_ctx* c, const float* agg, const float* wgt, float* softmax, uint8_t* seg,
                             int32_t X, int32_t Y, int32_t Z, void* stream_) {
  if (!c || !agg || !wgt) return fail("dwmh_finalize: null argument");
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(c->device);
  const int64_t V = (int64_t)X * Y * Z;
  if (c->d.num_classes != 2) {
    finalize_c_kernel<<<c->num_sms * 8, 256, 0, st>>>(agg, wgt, softmax, seg, c->d.num_classes, V);
    c->launches++;
    CU_TRY(cudaGetLastError());
    return 0;
  }
  const bool vec = (V & 3) == 0 && !((reinterpret_cast<uintptr_t>(agg) | reinterpret_cast<uintptr_t>(wgt) | reinterpret_cast<uintptr_t>(softmax)) & 15) &&
                   !(reinterpret_cast<uintptr_t>(seg) & 3);
  if (vec) finalize_kernel<true><<<c->num_sms * 8, 256, 0, st>>>(agg, wgt, softmax, seg, V);
  else finalize_kernel<false><<<c->num_sms * 8, 256, 0, st>>>(agg, wgt, softmax, seg, V);
  c->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_axpy(dwmh_ctx* c, float* acc, const float* x, float alpha, int64_t n, void* stream_) {
  if (!c || !acc || !x) return fail("dwmh_axpy: null argument");
  DEV_GUARD(c->device);
  axpy_kernel<<<c->num_sms * 8, 256, 0, (cudaStream_t)stream_>>>(acc, x, alpha, n);
  c->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_argmax2(dwmh_ctx* c, const float* p, uint8_t* seg, int64_t V, void* stream_) {
  if (!c || !p || !seg) return fail("dwmh_argmax2: null argument");
  DEV_GUARD(c->device);
  argmax2_kernel<<<c->num_sms * 8, 256, 0, (cudaStream_t)stream_>>>(p, seg, V);
  c->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_argmax(dwmh_ctx* c, const float* p, int32_t num_classes, uint8_t* seg, int64_t V, void* stream_) {
  if (!c || !p || !seg) return fail("dwmh_argmax: null argument");
  if (num_classes < 1 || num_classes > 255) return fail("dwmh_argmax: num_classes=%d outside 1..255 (uint8 labels)", num_classes);
  DEV_GUARD(c->device);
  argmax_c_kernel<<<c->num_sms * 8, 256, 0, (cudaStream_t)stream_>>>(p, num_classes, seg, V);
  c->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// a6 with host buffers
// ------------------------------------------------------------------------------------------------
template <typename V>
static int grow(V** p, size_t* cap, size_t need) {
  if (*cap >= need) return 0;
  if (*p) cudaFree(*p);
  *p = nullptr; *cap = 0;
  CU_TRY(cudaMalloc((void**)p, need * sizeof(V)));
  *cap = need;
  return 0;
}

// SURVEY 8f-3: checkpoint ensemble of masked background probabilities (DCNN_multistage.py:102-125)
extern "C" int dwmh_ensemble_masked_add(dwmh_ctx* c, float* acc, const float* bg_softmax, const float* valid_mask, int64_t n, void* stream_) {
  if (!c || !acc || !bg_softmax) return fail("dwmh_ensemble_masked_add: null argument");
  DEV_GUARD(c->device);
  ensemble_masked_add_kernel<<<c->num_sms * 8, 256, 0, (cudaStream_t)stream_>>>(acc, bg_softmax, valid_mask, n);
  c->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}
extern "C" int dwmh_ensemble_refine(dwmh_ctx* c, float* acc, int32_t k, uint8_t* label, int64_t n, void* stream_) {
  if (!c || !acc) return fail("dwmh_ensemble_refine: null argument");
  if (k <= 0) return fail("dwmh_ensemble_refine: k must be positive");
  DEV_GUARD(c->device);
  ensemble_refine_kernel<<<c->num_sms * 8, 256, 0, (cudaStream_t)stream_>>>(acc, (float)k, label, n);
  c->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}

// SURVEY 8f-2: remove_sparks (deepwmh/analysis/image_ops.py:325-344) on the device; seg and out may alias.
extern "C" int dwmh_remove_sparks(dwmh_ctx* c, const uint8_t* seg, int32_t X, int32_t Y, int32_t Z, int32_t min_volume,
                                  uint8_t* out, void* stream_) {
  if (!c || !seg || !out) return fail("dwmh_remove_sparks: null argument");
  if (X <= 0 || Y <= 0 || Z <= 0) return fail("dwmh_remove_sparks: empty volume");
  const int64_t V = (int64_t)X * Y * Z;
  if (V >= (int64_t)1 << 31) return fail("dwmh_remove_sparks: volume of %lld voxels exceeds the 32-bit label range", (long long)V);
  DEV_GUARD(c->device);
  DW_TRY(grow(&c->ccl_labels, &c->ccl_cap_l, (size_t)V));
  DW_TRY(grow(&c->ccl_sizes, &c->ccl_cap_s, (size_t)V));
  cudaStream_t st = (cudaStream_t)stream_;
  const int grid = c->num_sms * 8;
  ccl_init_kernel<<<grid, 256, 0, st>>>(seg, c->ccl_labels, c->ccl_sizes, V, Z);
  ccl_merge_kernel<<<grid, 256, 0, st>>>(c->ccl_labels, X, Y, Z);
  ccl_count_kernel<<<grid, 256, 0, st>>>(c->ccl_labels, c->ccl_sizes, V);
  ccl_filter_kernel<<<grid, 256, 0, st>>>(c->ccl_labels, c->ccl_sizes, out, min_volume, V);
  c->launches += 4;
  CU_TRY(cudaGetLastError());
  return 0;
}

static int predict_volume_host_impl(dwmh_ctx* c, const float* vol_host, const int8_t* seg_mask_host, int32_t X, int32_t Y, int32_t Z,
                                    int32_t zscore_mask_mode, double step_size, int32_t do_mirroring,
                                    int32_t mirror_axes_mask, int32_t use_gaussian,
                                    float* softmax_host, uint8_t* seg_host, void* stream_);

extern "C" int dwmh_predict_volume_host(dwmh_ctx* c, const float* vol_host, int32_t X, int32_t Y, int32_t Z,
                                        int32_t zscore_mask_mode, double step_size, int32_t do_mirroring,
                                        int32_t mirror_axes_mask, int32_t use_gaussian,
                                        float* softmax_host, uint8_t* seg_host, void* stream_) {
  if (zscore_mask_mode == 1) return fail("dwmh_predict_volume_host: mask_mode 1 needs the crop mask; use dwmh_predict_volume_host_masked");
  return predict_volume_host_impl(c, vol_host, nullptr, X, Y, Z, zscore_mask_mode, step_size, do_mirroring, mirror_axes_mask, use_gaussian,
                                  softmax_host, seg_host, stream_);
}

extern "C" int dwmh_predict_volume_host_masked(dwmh_ctx* c, const float* vol_host, const int8_t* seg_mask_host, int32_t X, int32_t Y, int32_t Z,
                                               double step_size, int32_t do_mirroring, int32_t mirror_axes_mask, int32_t use_gaussian,
                                               float* softmax_host, uint8_t* seg_host, void* stream_) {
  if (!seg_mask_host) return fail("dwmh_predict_volume_host_masked: null crop mask");
  return predict_volume_host_impl(c, vol_host, seg_mask_host, X, Y, Z, 1, step_size, do_mirroring, mirror_axes_mask, use_gaussian,
                                  softmax_host, seg_host, stream_);
}

static int predict_volume_host_impl(dwmh_ctx* c, const float* vol_host, const int8_t* seg_mask_host, int32_t X, int32_t Y, int32_t Z,
                                    int32_t zscore_mask_mode, double step_size, int32_t do_mirroring,
                                    int32_t mirror_axes_mask, int32_t use_gaussian,
                                    float* softmax_host, uint8_t* seg_host, void* stream_) {
  if (!c || !vol_host) return fail("dwmh_predict_volume_host: null argument");
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(c->device);
  const int64_t V = (int64_t)X * Y * Z;
  const int32_t* ps = c->d.patch_size;
  // a10 pad_nd_image: below = diff/2, above = diff/2 + diff%2
  const int PX = std::max(X, ps[0]), PY = std::max(Y, ps[1]), PZ = std::max(Z, ps[2]);
  const int bx = (PX - X) / 2, by = (PY - Y) / 2, bz = (PZ - Z) / 2;
  const bool padded = PX != X || PY != Y || PZ != Z;
  const int64_t PV = (int64_t)PX * PY * PZ;
  // modalities: vol_host [NM][X][Y][Z]; on the device each channel starts 16-byte aligned (z-score's vector accesses)
  const int NM = c->d.in_channels, NC = c->d.num_classes;
  const int64_t Vp = NM == 1 ? V : (V + 3) & ~(int64_t)3;
  DW_TRY(grow(&c->hv_vol, &c->hv_vol_cap, (size_t)NM * Vp));
  DW_TRY(grow(&c->hv_agg, &c->hv_agg_cap, (size_t)NC * PV));
  DW_TRY(grow(&c->hv_wgt, &c->hv_wgt_cap, (size_t)PV));
  DW_TRY(grow(&c->hv_seg, &c->hv_seg_cap, (size_t)PV));
  for (int m = 0; m < NM; ++m)
    CU_TRY(cudaMemcpyAsync(c->hv_vol + (size_t)m * Vp, vol_host + (size_t)m * V, V * sizeof(float), cudaMemcpyHostToDevice, st));
  const int8_t* mask_dev = nullptr;
  if (seg_mask_host) {
    // the crop mask rides in the (not yet used) label buffer: 1 byte per voxel, 4-byte aligned
    CU_TRY(cudaMemcpyAsync(c->hv_seg, seg_mask_host, V, cudaMemcpyHostToDevice, st));
    mask_dev = reinterpret_cast<const int8_t*>(c->hv_seg);
  }
  // nnU-Net normalises every modality on its own (same mask for all of them here)
  if (zscore_mask_mode >= 0)
    for (int m = 0; m < NM; ++m) DW_TRY(dwmh_zscore(c, c->hv_vol + (size_t)m * Vp, mask_dev, V, zscore_mask_mode, nullptr, st));
  const float* vol_dev = c->hv_vol;
  if (padded || Vp != V) {
    DW_TRY(grow(&c->hv_pad, &c->hv_pad_cap, (size_t)NM * PV));
    if (padded) CU_TRY(cudaMemsetAsync(c->hv_pad, 0, NM * PV * sizeof(float), st));
    for (int m = 0; m < NM; ++m) {
      cudaMemcpy3DParms cp = {};
      cp.srcPtr = make_cudaPitchedPtr(c->hv_vol + (size_t)m * Vp, Z * sizeof(float), Z, Y);
      cp.dstPtr = make_cudaPitchedPtr(c->hv_pad + (size_t)m * PV, PZ * sizeof(float), PZ, PY);
      cp.dstPos = make_cudaPos(bz * sizeof(float), by, bx);
      cp.extent = make_cudaExtent(Z * sizeof(float), Y, X);
      cp.kind = cudaMemcpyDeviceToDevice;
      CU_TRY(cudaMemcpy3DAsync(&cp, st));
    }
    vol_dev = c->hv_pad;
  }
  CU_TRY(cudaMemsetAsync(c->hv_agg, 0, NC * PV * sizeof(float), st));
  CU_TRY(cudaMemsetAsync(c->hv_wgt, 0, PV * sizeof(float), st));
  DW_TRY(dwmh_predict_3d(c, vol_dev, PX, PY, PZ, step_size, do_mirroring, mirror_axes_mask, use_gaussian, c->hv_agg, c->hv_wgt, 0, -1, st));
  DW_TRY(dwmh_finalize(c, c->hv_agg, c->hv_wgt, c->hv_agg, c->hv_seg, PX, PY, PZ, st));
  if (!padded) {
    if (softmax_host) CU_TRY(cudaMemcpyAsync(softmax_host, c->hv_agg, NC * V * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (seg_host) CU_TRY(cudaMemcpyAsync(seg_host, c->hv_seg, V, cudaMemcpyDeviceToHost, st));
  } else {
    for (int ch = 0; ch < NC && softmax_host; ++ch) {
      cudaMemcpy3DParms cp = {};
      cp.srcPtr = make_cudaPitchedPtr(c->hv_agg + (size_t)ch * PV, PZ * sizeof(float), PZ, PY);
      cp.srcPos = make_cudaPos(bz * sizeof(float), by, bx);
      cp.dstPtr = make_cudaPitchedPtr(softmax_host + (size_t)ch * V, Z * sizeof(float), Z, Y);
      cp.extent = make_cudaExtent(Z * sizeof(float), Y, X);
      cp.kind = cudaMemcpyDeviceToHost;
      CU_TRY(cudaMemcpy3DAsync(&cp, st));
    }
    if (seg_host) {
      cudaMemcpy3DParms cp = {};
      cp.srcPtr = make_cudaPitchedPtr(c->hv_seg, PZ, PZ, PY);
      cp.srcPos = make_cudaPos(bz, by, bx);
      cp.dstPtr = make_cudaPitchedPtr(seg_host, Z, Z, Y);
      cp.extent = make_cudaExtent(Z, Y, X);
      cp.kind = cudaMemcpyDeviceToHost;
      CU_TRY(cudaMemcpy3DAsync(&cp, st));
    }
  }
  CU_TRY(cudaStreamSynchronize(st));
  return 0;
}
