// api.cu -- the C ABI declared in include/ovn_b200.h: handle lifetime, weights, stage dispatch
// and the host-buffer convenience entry points.  No CPU fallback exists anywhere in this library:
// without an sm_100 device ovn_create fails with OVN_ERR_NO_DEVICE.
#include "common.cuh"
#include <math.h>
#include <string.h>

using namespace ovn;

static const char* kLegNames[] = {"s_conv1", "s_conv2", "s_conv3", "s_conv3a", "s_conv4", "s_conv5",
                                  "s_conv6", "s_conv7", "s_conv8", "s_conv9", "s_conv10"};

static void set_spec(ConvSpec& L, const char* name, int kh, int kw, int sh, int sw, int cin, int cout, int relu,
                     int h_in, int w_in) {
  memset(&L, 0, sizeof(L));
  snprintf(L.name, sizeof(L.name), "%s", name);
  L.kh = kh; L.kw = kw; L.sh = sh; L.sw = sw; L.cin = cin; L.cout = cout; L.relu = relu;
  L.h_in = h_in; L.w_in = w_in;
  L.h_out = (h_in - kh) / sh + 1;
  L.w_out = (w_in - kw) / sw + 1;
}

static __global__ void k_iota(int32_t* p, int n, int start) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = start + i;
}

static __global__ void k_sanitize_idx(const int32_t* __restrict__ in, int32_t* __restrict__ out, int n, int64_t limit,
                                      int code, int* __restrict__ err) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t v = in[i];
  if (v < 0 || v >= limit) {
    atomicCAS(err, 0, code);              // the first error wins; results of this call are poisoned by the finalize kernels
    v = v < 0 ? 0 : limit - 1;
  }
  out[i] = (int32_t)v;
}

// ---- device-side signalling between the ranks of a sharded bank (search.py transport 'symm') ----------
// Flags are int32 slots in symmetric (peer-mapped) memory holding the number of the last finished step.
// One launch signals every peer (release at system scope, after everything this stream did before),
// one launch waits for every peer (acquire at system scope, bounded).
struct PeerPtrs { int32_t* p[16]; };

static __global__ void k_peer_signal(PeerPtrs dst, int n, int value) {
  const int i = threadIdx.x;
  if (i >= n || dst.p[i] == nullptr) return;
  __threadfence_system();
  asm volatile("st.release.sys.global.s32 [%0], %1;" :: "l"(dst.p[i]), "r"(value) : "memory");
}

static __global__ void k_peer_wait(const int32_t* __restrict__ flags, int n, int skip, int value, int* __restrict__ err) {
  const int i = threadIdx.x;
  if (i >= n || i == skip) return;
  const long long t0 = clock64();
  for (;;) {
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(flags + i) : "memory");
    if (v >= value) break;
    if (clock64() - t0 > (1ll << 32)) { atomicCAS(err, 0, 950); break; }     // ~2 s: a peer died
    __nanosleep(32);
  }
}

namespace ovn {

int sanitize_indices(ovn_handle* h, const int32_t* d_in, int n, int64_t limit, int code, int32_t* d_out, cudaStream_t s) {
  if (n <= 0) return OVN_OK;
  k_sanitize_idx<<<(n + 255) / 256, 256, 0, s>>>(d_in, d_out, n, limit < 1 ? 1 : limit, code, h->d_err);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

// The caller has queued everything on `s`; this copies the flag back, synchronises `s` and maps a
// non-zero flag to a status (the flag is cleared so that the handle stays usable).
int check_device_error(ovn_handle* h, cudaStream_t s) {
  int* hp = reinterpret_cast<int*>(h->h_pinned);
  if (!hp || !h->d_err) return OVN_OK;
  OVN_CUDA(h, cudaMemcpyAsync(hp, h->d_err, sizeof(int), cudaMemcpyDeviceToHost, s));
  OVN_CUDA(h, cudaStreamSynchronize(s));
  const int e = *hp;
  if (e == 0) return OVN_OK;
  OVN_CUDA(h, cudaMemsetAsync(h->d_err, 0, sizeof(int), s));
  if (e == kErrBadIndex) OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "a pair / candidate index is outside [0, bank_size)");
  if (e == kErrRowNotPrepared)
    OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "resident bank: an indexed row was never passed to ovn_bank_prepare");
  if (e == kErrBadYawBin) OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "a yaw-bin target is outside [0, leg_output_width)");
  if (e == 950) OVN_SET_ERR(h, OVN_ERR_CUDA, "ovn_peer_wait timed out: a peer rank never signalled");
  OVN_SET_ERR(h, OVN_ERR_CUDA, "tensor-core pipeline barrier timed out (code %d); outputs of the call are poisoned (NaN / INT32_MIN)", e);
}

}  // namespace ovn

extern "C" {

int ovn_abi_version(void) { return OVN_ABI_VERSION; }

const char* ovn_status_string(int status) {
  switch (status) {
    case OVN_OK: return "OVN_OK";
    case OVN_ERR_INVALID_ARG: return "OVN_ERR_INVALID_ARG";
    case OVN_ERR_BAD_CONFIG: return "OVN_ERR_BAD_CONFIG";
    case OVN_ERR_WEIGHTS: return "OVN_ERR_WEIGHTS";
    case OVN_ERR_CUDA: return "OVN_ERR_CUDA";
    case OVN_ERR_NO_DEVICE: return "OVN_ERR_NO_DEVICE";
    case OVN_ERR_CAPACITY: return "OVN_ERR_CAPACITY";
    default: return "OVN_ERR_UNKNOWN";
  }
}

void ovn_default_config(ovn_config* c) {
  if (!c) return;
  memset(c, 0, sizeof(*c));
  c->abi_version = OVN_ABI_VERSION;
  c->proj_H = 64; c->proj_W = 900;                 // config/network.yml:75
  c->fov_up_deg = 3.0f; c->fov_down_deg = -25.0f;  // utils.py:59
  c->max_range = 50.0f;
  c->use_depth = 1; c->use_normals = 1;            // network.yml:20-24
  c->n_prob_channels = 0; c->use_intensity = 0;
  c->strides_layer1[0] = 2; c->strides_layer1[1] = 2;   // network.yml:79
  c->additional_unsymmetric_layer3a = 1;           // network.yml:82
  c->leg_output_width = 360;                       // network.yml:77
  c->conv1size = 15;                               // generateNet.py:88-89
  c->precision = OVN_PREC_F16_TC;
  c->max_batch_scans = 16;                         // network.yml:41 batch_size
  c->max_batch_pairs = 1101;
}

static thread_local std::string g_create_error;

const char* ovn_last_error(const ovn_handle* h) { return h ? h->last_error.c_str() : g_create_error.c_str(); }
int64_t ovn_launch_count(const ovn_handle* h) { return h ? h->launches : 0; }
int ovn_input_channels(const ovn_handle* h) { return h ? h->C : 0; }
int ovn_feature_width(const ovn_handle* h) { return h ? h->cfg.leg_output_width : 0; }
int ovn_feature_channels(const ovn_handle* h) { return h ? kFeatC : 0; }

#define CREATE_FAIL(code, ...)                              \
  do {                                                      \
    char _b[512];                                           \
    snprintf(_b, sizeof(_b), __VA_ARGS__);                  \
    g_create_error = _b;                                    \
    if (h) ovn_destroy(h);                                  \
    return (code);                                          \
  } while (0)

#define CREATE_CUDA(call)                                                              \
  do {                                                                                 \
    cudaError_t _e = (call);                                                           \
    if (_e != cudaSuccess) CREATE_FAIL(OVN_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(_e)); \
  } while (0)

int ovn_create(const ovn_config* cfg, ovn_handle** out) {
  ovn_handle* h = nullptr;
  if (!cfg || !out) CREATE_FAIL(OVN_ERR_INVALID_ARG, "ovn_create: NULL argument");
  *out = nullptr;
  if (cfg->abi_version != OVN_ABI_VERSION)
    CREATE_FAIL(OVN_ERR_INVALID_ARG, "ovn_create: abi_version %d != %d", cfg->abi_version, OVN_ABI_VERSION);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    CREATE_FAIL(OVN_ERR_NO_DEVICE, "ovn_create: no CUDA device visible (this library has no CPU fallback)");
  }
  int dev = 0;
  CREATE_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CREATE_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10)
    CREATE_FAIL(OVN_ERR_NO_DEVICE, "ovn_create: device %d is sm_%d%d; this build targets sm_100a only", dev,
                prop.major, prop.minor);
  h = new ovn_handle();
  h->cfg = *cfg;
  h->device = dev;
  h->sm_count = prop.multiProcessorCount;
  const ovn_config& c = h->cfg;
  if (c.proj_H <= 0 || c.proj_W <= 0 || c.max_batch_scans <= 0 || c.max_batch_pairs <= 0)
    CREATE_FAIL(OVN_ERR_BAD_CONFIG, "ovn_create: non-positive size in config");
  if (c.n_prob_channels != 0 && c.n_prob_channels != 3 && c.n_prob_channels != 20)
    CREATE_FAIL(OVN_ERR_BAD_CONFIG, "ovn_create: n_prob_channels must be 0, 3 or 20 (infer.py:68-73)");
  h->C = (c.use_depth ? 1 : 0) + (c.use_normals ? 3 : 0) + c.n_prob_channels + (c.use_intensity ? 1 : 0);
  if (h->C <= 0) CREATE_FAIL(OVN_ERR_BAD_CONFIG, "ovn_create: no input channel enabled");

  // ---- leg shape inference (generateNet.py:161-217).  A config whose leg does not reduce the image
  // to 1 x leg_output_width x 128 still gets a handle, but only the projection stages work on it.
  struct { int kh, kw, sh, sw, cout; bool opt; } T[] = {
      {5, 15, c.strides_layer1[0], c.strides_layer1[1], 16, false}, {3, 15, 2, 1, 32, false},
      {3, 15, 2, 1, 64, false},  {3, 12, 2, 1, 64, true},           {2, 9, 2, 1, 128, false},
      {1, 9, 1, 1, 128, false},  {1, 9, 1, 1, 128, false},          {1, 9, 1, 1, 128, false},
      {1, 7, 1, 1, 128, false},  {1, 5, 1, 1, 128, false},          {1, 3, 1, 1, 128, false}};
  int hh = c.proj_H, ww = c.proj_W, cc = h->C;
  h->n_leg = 0;
  h->net_ok = true;
  char nb[256];
  for (int i = 0; i < 11 && h->net_ok; ++i) {
    if (T[i].opt && !c.additional_unsymmetric_layer3a) continue;
    if (T[i].sh <= 0 || T[i].sw <= 0 || hh < T[i].kh || ww < T[i].kw) {
      snprintf(nb, sizeof(nb), "layer %s does not fit its input %dx%d", kLegNames[i], hh, ww);
      h->net_ok = false; h->net_error = nb;
      break;
    }
    set_spec(h->leg[h->n_leg], kLegNames[i], T[i].kh, T[i].kw, T[i].sh, T[i].sw, cc, T[i].cout, 1, hh, ww);
    hh = h->leg[h->n_leg].h_out; ww = h->leg[h->n_leg].w_out; cc = T[i].cout;
    h->n_leg++;
  }
  const int Wf = c.leg_output_width, s = c.conv1size;
  if (h->net_ok && (hh != 1 || ww != c.leg_output_width || cc != kFeatC)) {
    snprintf(nb, sizeof(nb), "leg output is %dx%dx%d, expected 1x%dx%d (network.yml:77)", hh, ww, cc,
             c.leg_output_width, kFeatC);
    h->net_ok = false; h->net_error = nb;
  }
  if (h->net_ok && (s <= 0 || Wf % s != 0 || Wf / s < 3)) {
    snprintf(nb, sizeof(nb), "conv1size %d must divide leg_output_width %d", s, Wf);
    h->net_ok = false; h->net_error = nb;
  }
  if (!h->net_ok) { h->n_leg = 0; *out = nullptr; }
  // ---- head shapes (generateNet.py:96-114)
  if (h->net_ok) {
    set_spec(h->head[0], "c_conv1", 1, s, 1, s, kFeatC, 64, 0, Wf, Wf);
    set_spec(h->head[1], "c_conv2", s, 1, s, 1, 64, 128, 1, h->head[0].h_out, h->head[0].w_out);
    set_spec(h->head[2], "c_conv3", 3, 3, 1, 1, 128, 256, 1, h->head[1].h_out, h->head[1].w_out);
    h->o1_h = h->head[0].h_out; h->o1_w = h->head[0].w_out;
    h->o2_h = h->head[1].h_out; h->o2_w = h->head[1].w_out;
    h->o3_h = h->head[2].h_out; h->o3_w = h->head[2].w_out;
    h->dense_in = h->o3_h * h->o3_w * h->head[2].cout;
  }

  // ---- workspaces
  const size_t HW = (size_t)c.proj_H * c.proj_W;
  CREATE_CUDA(cudaMalloc(&h->d_keys, (size_t)c.max_batch_scans * HW * sizeof(unsigned long long)));
  CREATE_CUDA(cudaMalloc(&h->d_input, (size_t)c.max_batch_scans * HW * h->C * sizeof(float)));
  size_t max_act = 1;
  for (int l = 0; l < h->n_leg; ++l) {
    size_t a = (size_t)h->leg[l].h_out * h->leg[l].w_out * h->leg[l].cout;
    if (a > max_act) max_act = a;
  }
  h->cap_act = (int64_t)max_act * c.max_batch_scans;
  CREATE_CUDA(cudaMalloc(&h->d_act[0], h->cap_act * sizeof(float)));
  CREATE_CUDA(cudaMalloc(&h->d_act[1], h->cap_act * sizeof(float)));
  CREATE_CUDA(cudaMalloc(&h->d_query_fv, (size_t)Wf * kFeatC * sizeof(float)));
  CREATE_CUDA(cudaMalloc(&h->d_idx_tmp, (size_t)2 * c.max_batch_pairs * sizeof(int32_t)));
  CREATE_CUDA(cudaMalloc(&h->d_idx_san, (size_t)3 * c.max_batch_pairs * sizeof(int32_t)));   // left, right, resident-row check
  CREATE_CUDA(cudaMalloc(&h->d_err, sizeof(int)));
  CREATE_CUDA(cudaMemset(h->d_err, 0, sizeof(int)));
  CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_bank, cudaEventDisableTiming));
  CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_train, cudaEventDisableTiming));
  // pinned staging of the host entry points: [err int, pad][offsets 2 x i64][cand idx][overlap][yaw]
  h->cap_pinned = 64 + (int64_t)c.max_batch_pairs * 12;
  CREATE_CUDA(cudaHostAlloc(&h->h_pinned, (size_t)h->cap_pinned, cudaHostAllocDefault));
  CREATE_CUDA(cudaMalloc(&h->d_logit, (size_t)c.max_batch_pairs * sizeof(float)));
  if (h->net_ok) CREATE_CUDA(cudaMalloc(&h->d_G, (size_t)c.max_batch_pairs * Wf * Wf * sizeof(float)));
  if (c.precision == OVN_PREC_FP32 && h->net_ok) {
    CREATE_CUDA(cudaMalloc(&h->d_o1, (size_t)c.max_batch_pairs * h->o1_h * h->o1_w * 64 * sizeof(float)));
    CREATE_CUDA(cudaMalloc(&h->d_o2, (size_t)c.max_batch_pairs * h->o2_h * h->o2_w * 128 * sizeof(float)));
  } else if (c.precision != OVN_PREC_F16_TC && c.precision != OVN_PREC_FP32) {
    CREATE_FAIL(OVN_ERR_BAD_CONFIG, "ovn_create: unknown precision %d", c.precision);
  }
  CREATE_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  *out = h;
  return OVN_OK;
}

int ovn_destroy(ovn_handle* h) {
  if (!h) return OVN_OK;
  DeviceGuard guard(h);
  tc_free(h);
  train_free(h);
  for (auto& p : h->d_w) if (p) cudaFree(p);
  for (auto& p : h->d_b) if (p) cudaFree(p);
  for (auto& p : h->d_w16) if (p) cudaFree(p);
  void* bufs[] = {h->d_keys, h->d_valid_words, h->d_word_prefix, h->d_scan_tmp, h->d_act[0], h->d_act[1],
                  h->d_input, h->d_o1, h->d_o2, h->d_logit, h->d_G, h->d_idx_tmp, h->d_query_fv,
                  h->d_stage_points, h->d_stage_offsets, h->d_idx_san, h->d_err};
  for (void* b : bufs) if (b) cudaFree(b);
  if (h->h_pinned) cudaFreeHost(h->h_pinned);
  if (h->ev_bank) cudaEventDestroy(h->ev_bank);
  if (h->ev_train) cudaEventDestroy(h->ev_train);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  for (auto& v : h->prof_ev) for (cudaEvent_t e : v) cudaEventDestroy(e);
  delete h;
  return OVN_OK;
}

int ovn_profile_enable(ovn_handle* h, int on) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  h->profiling = on != 0;
  return OVN_OK;
}

int ovn_profile_read(ovn_handle* h, const char* kernel, double* total_ms, int64_t* launches) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  if (!kernel || !total_ms || !launches) OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "ovn_profile_read: NULL argument");
  static const char* names[kProfKinds] = {"delta_conv1", "conv2", "conv3", "corr", "project_scatter",
                                          "project_gather", "leg"};
  int kind = -1;
  for (int i = 0; i < kProfKinds; ++i) if (strcmp(kernel, names[i]) == 0) kind = i;
  if (kind < 0) OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "ovn_profile_read: unknown kernel '%s'", kernel);
  OVN_CUDA(h, cudaDeviceSynchronize());
  { int rc = check_device_error(h, h->own_stream); if (rc != OVN_OK) return rc; }
  std::vector<cudaEvent_t>& ev = h->prof_ev[kind];
  double ms = 0;
  int64_t n = 0;
  for (size_t i = 0; i + 1 < ev.size(); i += 2) {
    float t = 0;
    if (cudaEventElapsedTime(&t, ev[i], ev[i + 1]) == cudaSuccess) { ms += t; ++n; }
  }
  for (cudaEvent_t e : ev) cudaEventDestroy(e);
  ev.clear();
  *total_ms = ms;
  *launches = n;
  return OVN_OK;
}

// ---- weights ------------------------------------------------------------------------------------
static const ConvSpec* find_layer(const ovn_handle* h, const char* name, int* slot) {
  for (int l = 0; l < h->n_leg; ++l)
    if (strcmp(h->leg[l].name, name) == 0) { *slot = l; return &h->leg[l]; }
  for (int l = 0; l < 3; ++l)
    if (strcmp(h->head[l].name, name) == 0) { *slot = kMaxLegLayers + l; return &h->head[l]; }
  return nullptr;
}

static const char* kHeadNames[4] = {"c_conv1", "c_conv2", "c_conv3", "overlap_output"};

// After Adagrad steps the device fp32 head weights (and, after full-network steps, the leg weights) are
// the newest copy: bring them back into host_w, which ovn_finalize_weights packs from.
static int sync_trained_weights(ovn_handle* h) {
  if (!h->weights_trained) return OVN_OK;
  OVN_CUDA(h, cudaEventSynchronize(h->ev_train));
  for (int l = 0; l < 4; ++l) {
    LayerWeights& w = h->host_w[kHeadNames[l]];
    OVN_CUDA(h, cudaMemcpy(w.kernel.data(), h->d_w[kMaxLegLayers + l], w.kernel.size() * sizeof(float),
                           cudaMemcpyDeviceToHost));
    OVN_CUDA(h, cudaMemcpy(w.bias.data(), h->d_b[kMaxLegLayers + l], w.bias.size() * sizeof(float),
                           cudaMemcpyDeviceToHost));
  }
  for (int l = 0; h->leg_trained && l < h->n_leg; ++l) {
    LayerWeights& w = h->host_w[h->leg[l].name];
    OVN_CUDA(h, cudaMemcpy(w.kernel.data(), h->d_w[l], w.kernel.size() * sizeof(float), cudaMemcpyDeviceToHost));
    OVN_CUDA(h, cudaMemcpy(w.bias.data(), h->d_b[l], w.bias.size() * sizeof(float), cudaMemcpyDeviceToHost));
  }
  h->weights_trained = h->leg_trained = false;
  return OVN_OK;
}

int ovn_set_weights(ovn_handle* h, const char* name, const float* k, const int64_t* dims, int32_t ndim,
                    const float* bias, int64_t bias_len) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  if (!name || !k || !dims || !bias) OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "ovn_set_weights: NULL argument");
  if (!h->net_ok) OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "ovn_set_weights: %s", h->net_error.c_str());
  int slot = -1;
  int64_t expect[4];
  int expect_nd = 0;
  int64_t expect_bias = 0;
  if (strcmp(name, "overlap_output") == 0) {
    expect[0] = h->dense_in; expect[1] = 1; expect_nd = 2; expect_bias = 1;
  } else {
    const ConvSpec* L = find_layer(h, name, &slot);
    if (!L) OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_set_weights: unknown layer name '%s'", name);
    expect[0] = L->kh; expect[1] = L->kw; expect[2] = L->cin; expect[3] = L->cout; expect_nd = 4;
    expect_bias = L->cout;
  }
  if (ndim != expect_nd || bias_len != expect_bias)
    OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_set_weights: layer %s expects a %d-d kernel and %lld biases", name,
                expect_nd, (long long)expect_bias);
  int64_t total = 1;
  for (int i = 0; i < ndim; ++i) {
    if (dims[i] != expect[i])
      OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_set_weights: layer %s kernel dim %d is %lld, expected %lld", name, i,
                  (long long)dims[i], (long long)expect[i]);
    total *= dims[i];
  }
  {
    int rc = sync_trained_weights(h);
    if (rc != OVN_OK) return rc;
  }
  train_reset_optimizer(h);                 // new weights start a new Adagrad run
  LayerWeights& w = h->host_w[name];
  w.kernel.assign(k, k + total);
  w.dims.assign(dims, dims + ndim);
  w.bias.assign(bias, bias + bias_len);
  w.set = true;
  h->weights_ready = false;
  return OVN_OK;
}

static int upload(ovn_handle* h, int slot, const LayerWeights& w) {
  if (h->d_w[slot]) { cudaFree(h->d_w[slot]); h->d_w[slot] = nullptr; }
  if (h->d_b[slot]) { cudaFree(h->d_b[slot]); h->d_b[slot] = nullptr; }
  OVN_CUDA(h, cudaMalloc(&h->d_w[slot], w.kernel.size() * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&h->d_b[slot], w.bias.size() * sizeof(float)));
  OVN_CUDA(h, cudaMemcpy(h->d_w[slot], w.kernel.data(), w.kernel.size() * sizeof(float), cudaMemcpyHostToDevice));
  OVN_CUDA(h, cudaMemcpy(h->d_b[slot], w.bias.data(), w.bias.size() * sizeof(float), cudaMemcpyHostToDevice));
  return OVN_OK;
}

int ovn_finalize_weights(ovn_handle* h) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  if (!h->net_ok) OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "ovn_finalize_weights: %s", h->net_error.c_str());
  {
    int rc = sync_trained_weights(h);
    if (rc != OVN_OK) return rc;
  }
  for (int l = 0; l < h->n_leg; ++l) {
    auto it = h->host_w.find(h->leg[l].name);
    if (it == h->host_w.end() || !it->second.set)
      OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_finalize_weights: layer %s has no weights", h->leg[l].name);
    int rc = upload(h, l, it->second);
    if (rc != OVN_OK) return rc;
  }
  for (int l = 0; l < 4; ++l) {
    auto it = h->host_w.find(kHeadNames[l]);
    if (it == h->host_w.end() || !it->second.set)
      OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_finalize_weights: layer %s has no weights", kHeadNames[l]);
    int rc = upload(h, kMaxLegLayers + l, it->second);
    if (rc != OVN_OK) return rc;
  }
  if (h->cfg.precision == OVN_PREC_F16_TC) {
    int rc = tc_pack_weights(h);
    if (rc != OVN_OK) return rc;
  }
  h->weights_ready = true;
  return OVN_OK;
}

// ---- stage entry points ---------------------------------------------------------------------------
#define REQUIRE(h, cond, msg) \
  do { if (!(cond)) OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "%s: %s", __func__, msg); } while (0)

int ovn_project_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int32_t n_scans,
                      int64_t n_total, float max_range, float* d_range, float* d_vertex, float* d_intensity,
                      int32_t* d_idx, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_scans >= 0 && n_total >= 0, "negative size");
  REQUIRE(h, n_scans == 0 || d_offsets, "d_offsets is NULL");
  REQUIRE(h, n_total == 0 || d_points, "d_points is NULL");
  return project_batch(h, d_points, d_offsets, n_scans, n_total, max_range, d_range, d_vertex, d_intensity, d_idx,
                       (cudaStream_t)stream);
}

int ovn_normals_batch(ovn_handle* h, const float* d_range, const float* d_vertex, int32_t n_scans, float* d_normal,
                      void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_scans >= 0, "negative size");
  REQUIRE(h, n_scans == 0 || (d_range && d_vertex && d_normal), "NULL image pointer");
  return normals_batch(h, d_range, d_vertex, n_scans, d_normal, (cudaStream_t)stream);
}

int ovn_semantic_batch(ovn_handle* h, const int32_t* d_idx, const float* d_probs, const int64_t* d_offsets,
                       int32_t n_scans, int32_t n_classes, float* d_out, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_scans >= 0 && n_classes > 0, "bad size");
  REQUIRE(h, n_scans == 0 || (d_idx && d_probs && d_offsets && d_out), "NULL pointer");
  return semantic_batch(h, d_idx, d_probs, d_offsets, n_scans, n_classes, d_out, (cudaStream_t)stream);
}

int ovn_gt_range_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int32_t n_scans,
                       int64_t n_total, const double* d_pose_ref, const double* d_pose_cur_inv, float max_range,
                       float* d_range, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_scans >= 0 && n_total >= 0, "negative size");
  REQUIRE(h, n_scans == 0 || (d_offsets && d_range && (d_points || n_total == 0)), "NULL pointer");
  return gt_range_batch(h, d_points, d_offsets, n_scans, n_total, d_pose_ref, d_pose_cur_inv, max_range, d_range,
                        (cudaStream_t)stream);
}

int ovn_gt_overlap_count(ovn_handle* h, const float* d_ref_ranges, const float* d_cur_range, int32_t n_scans,
                         int32_t* d_counts, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_scans >= 0, "negative size");
  REQUIRE(h, d_cur_range && d_counts && (n_scans == 0 || d_ref_ranges), "NULL pointer");
  return gt_overlap_count(h, d_ref_ranges, d_cur_range, n_scans, d_counts, (cudaStream_t)stream);
}

int ovn_gt_pair_counts(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int32_t n_scans,
                       int64_t n_points_total, const double* d_pose_ref, const double* d_pose_cur_inv,
                       const float* d_cur_ranges, int32_t n_cur, const int32_t* d_pairs, int64_t n_pairs,
                       float max_range, int32_t* d_counts, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_pairs >= 0 && n_points_total >= 0, "negative size");
  if (n_pairs == 0) return OVN_OK;
  REQUIRE(h, n_scans > 0 && n_cur > 0, "n_scans and n_cur must be positive");
  REQUIRE(h, d_offsets && d_pose_ref && d_pose_cur_inv && d_cur_ranges && d_pairs && d_counts &&
                 (d_points || n_points_total == 0), "NULL pointer");
  return gt_pair_counts(h, d_points, d_offsets, n_scans, n_points_total, d_pose_ref, d_pose_cur_inv, d_cur_ranges,
                        n_cur, d_pairs, n_pairs, max_range, d_counts, (cudaStream_t)stream);
}

int ovn_preprocess_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int32_t n_scans,
                         int64_t n_total, const float* d_probs, float* d_input, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_scans >= 0 && n_total >= 0, "negative size");
  REQUIRE(h, n_scans == 0 || (d_offsets && d_input), "NULL pointer");
  return preprocess_batch(h, d_points, d_offsets, n_scans, n_total, d_probs, d_input, (cudaStream_t)stream);
}

int ovn_pack_input(ovn_handle* h, const float* d_depth, const float* d_normal, const float* d_prob,
                   const float* d_intensity, int32_t n_scans, float* d_input, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_scans >= 0, "negative size");
  REQUIRE(h, (d_depth != nullptr) == (h->cfg.use_depth != 0), "depth pointer does not match use_depth");
  REQUIRE(h, (d_normal != nullptr) == (h->cfg.use_normals != 0), "normal pointer does not match use_normals");
  REQUIRE(h, (d_prob != nullptr) == (h->cfg.n_prob_channels != 0), "prob pointer does not match n_prob_channels");
  REQUIRE(h, (d_intensity != nullptr) == (h->cfg.use_intensity != 0), "intensity pointer does not match use_intensity");
  return pack_input(h, d_depth, d_normal, d_prob, d_intensity, n_scans, d_input, (cudaStream_t)stream);
}

int ovn_leg_forward(ovn_handle* h, const float* d_input, int32_t n_scans, float* d_fv, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_scans >= 0, "negative size");
  if (n_scans == 0) return OVN_OK;
  REQUIRE(h, d_input && d_fv, "NULL pointer");
  if (!h->net_ok) OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "ovn_leg_forward: %s", h->net_error.c_str());
  if (!h->weights_ready) OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_leg_forward: weights not finalised");
  if (h->leg_trained)
    OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_leg_forward: weights changed by training; call ovn_finalize_weights");
  const int Wf = h->cfg.leg_output_width;
  const size_t in_stride = (size_t)h->cfg.proj_H * h->cfg.proj_W * h->C;
  for (int s0 = 0; s0 < n_scans; s0 += h->cfg.max_batch_scans) {
    const int n = (n_scans - s0 < h->cfg.max_batch_scans) ? n_scans - s0 : h->cfg.max_batch_scans;
    int rc = (h->cfg.precision == OVN_PREC_F16_TC)
                 ? leg_forward_tc(h, d_input + s0 * in_stride, n, d_fv + (size_t)s0 * Wf * kFeatC, (cudaStream_t)stream)
                 : leg_forward_fp32(h, d_input + s0 * in_stride, n, d_fv + (size_t)s0 * Wf * kFeatC, (cudaStream_t)stream);
    if (rc != OVN_OK) return rc;
  }
  return OVN_OK;
}

static int heads_dispatch(ovn_handle* h, const float* d_bank, int64_t bank_size, const float* d_query,
                          const int32_t* d_left, const int32_t* d_right, int n, float* d_overlap, int32_t* d_yaw,
                          float* d_corr, cudaStream_t s) {
  if (!h->net_ok) OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "heads: %s", h->net_error.c_str());
  if (!h->weights_ready) OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "heads: weights not finalised");
  if (h->weights_trained)
    OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "heads: weights changed by training; call ovn_finalize_weights");
  if (bank_size <= 0) OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "heads: bank_size must be positive");
  // Every index list is bounds-checked on the device (no host sync): out-of-range entries are clamped,
  // the error flag is raised, the finalize kernels poison the outputs and the next synchronising
  // entry point (ovn_check, *_host, ovn_profile_read) returns OVN_ERR_INVALID_ARG.
  const int maxp = h->cfg.max_batch_pairs;
  const int Wf = h->cfg.leg_output_width;
  for (int p0 = 0; p0 < n; p0 += maxp) {
    const int np = (n - p0 < maxp) ? n - p0 : maxp;
    int32_t* l = h->d_idx_san;
    int32_t* r = d_right ? h->d_idx_san + maxp : nullptr;
    int rc = sanitize_indices(h, d_left + p0, np, bank_size, kErrBadIndex, l, s);
    if (rc == OVN_OK && d_right) rc = sanitize_indices(h, d_right + p0, np, bank_size, kErrBadIndex, r, s);
    if (rc != OVN_OK) return rc;
    float* corr = d_corr ? d_corr + (size_t)p0 * Wf : nullptr;
    rc = (h->cfg.precision == OVN_PREC_F16_TC)
             ? heads_forward_tc(h, d_bank, d_query, l, r, np, d_overlap + p0, d_yaw + p0, corr, s)
             : heads_forward_fp32(h, d_bank, d_query, l, r, np, d_overlap + p0, d_yaw + p0, corr, s);
    if (rc != OVN_OK) return rc;
  }
  return OVN_OK;
}

int ovn_heads_forward(ovn_handle* h, const float* d_bank, int64_t bank_size, const int32_t* d_left,
                      const int32_t* d_right, int32_t n_pairs, float* d_overlap, int32_t* d_yaw, float* d_corr,
                      void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_pairs >= 0 && bank_size >= 0, "negative size");
  if (n_pairs == 0) return OVN_OK;
  REQUIRE(h, d_bank && d_left && d_right && d_overlap && d_yaw, "NULL pointer");
  return heads_dispatch(h, d_bank, bank_size, nullptr, d_left, d_right, n_pairs, d_overlap, d_yaw, d_corr,
                        (cudaStream_t)stream);
}

int ovn_heads_1vsN(ovn_handle* h, const float* d_bank, int64_t bank_size, const float* d_query,
                   const int32_t* d_cand_idx, int32_t n_cand, float* d_overlap, int32_t* d_yaw, float* d_corr,
                   void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_cand >= 0 && bank_size >= 0, "negative size");
  if (n_cand == 0) return OVN_OK;
  REQUIRE(h, d_bank && d_query && d_overlap && d_yaw, "NULL pointer");
  cudaStream_t s = (cudaStream_t)stream;
  if (d_cand_idx)
    return heads_dispatch(h, d_bank, bank_size, d_query, d_cand_idx, nullptr, n_cand, d_overlap, d_yaw, d_corr, s);
  REQUIRE(h, n_cand <= bank_size, "n_cand exceeds bank_size");
  // candidates 0..n-1 in chunks of the scratch capacity
  const int maxp = h->cfg.max_batch_pairs;
  for (int p0 = 0; p0 < n_cand; p0 += maxp) {
    const int np = (n_cand - p0 < maxp) ? n_cand - p0 : maxp;
    k_iota<<<(np + 255) / 256, 256, 0, s>>>(h->d_idx_tmp, np, p0);
    OVN_LAUNCH_CHECK(h);
    int rc = heads_dispatch(h, d_bank, bank_size, d_query, h->d_idx_tmp, nullptr,
                            np, d_overlap + p0, d_yaw + p0,
                            d_corr ? d_corr + (size_t)p0 * h->cfg.leg_output_width : nullptr, s);
    if (rc != OVN_OK) return rc;
  }
  return OVN_OK;
}

int ovn_heads_rows_vs_bank(ovn_handle* h, const float* d_bank, int64_t bank_size, int64_t row_lo, int64_t row_hi,
                           float* d_overlap, int32_t* d_yaw, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, bank_size >= 0 && row_lo >= 0 && row_lo <= row_hi && row_hi <= bank_size, "bad row range");
  if (row_lo == row_hi || bank_size == 0) return OVN_OK;
  REQUIRE(h, d_bank && d_overlap && d_yaw, "NULL pointer");
  REQUIRE(h, bank_size <= INT32_MAX, "bank too large");
  const size_t vol = (size_t)h->cfg.leg_output_width * kFeatC;
  for (int64_t i = row_lo; i < row_hi; ++i) {
    int rc = ovn_heads_1vsN(h, d_bank, bank_size, d_bank + (size_t)i * vol, nullptr, (int32_t)bank_size,
                            d_overlap + (size_t)(i - row_lo) * bank_size, d_yaw + (size_t)(i - row_lo) * bank_size,
                            nullptr, stream);
    if (rc != OVN_OK) return rc;
  }
  return OVN_OK;
}

int ovn_bank_prepare(ovn_handle* h, const float* d_bank, int64_t bank_capacity, int64_t first, int64_t count,
                     void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, d_bank != nullptr, "d_bank is NULL");
  REQUIRE(h, bank_capacity > 0 && first >= 0 && count >= 0 && first + count <= bank_capacity, "bad row range");
  if (h->cfg.precision != OVN_PREC_F16_TC || count == 0) return OVN_OK;
  if (!h->weights_ready) OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_bank_prepare: weights not finalised");
  int rc = tc_bank_prepare(h, d_bank, bank_capacity, first, count, (cudaStream_t)stream);
  if (rc == OVN_OK) OVN_CUDA(h, cudaEventRecord(h->ev_bank, (cudaStream_t)stream));
  return rc;
}

int ovn_peer_signal(ovn_handle* h, const uint64_t* h_flag_ptrs, int32_t n, int32_t value, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  if (n == 0) return OVN_OK;
  REQUIRE(h, h_flag_ptrs != nullptr && n > 0 && n <= 16, "bad peer list (at most 16 peers)");
  PeerPtrs pp = {};
  for (int i = 0; i < n; ++i) pp.p[i] = reinterpret_cast<int32_t*>(h_flag_ptrs[i]);
  k_peer_signal<<<1, 32, 0, (cudaStream_t)stream>>>(pp, n, value);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

int ovn_peer_wait(ovn_handle* h, const int32_t* d_flags, int32_t n, int32_t skip, int32_t value, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  if (n == 0) return OVN_OK;
  REQUIRE(h, d_flags != nullptr && n > 0 && n <= 32, "bad flag list");
  k_peer_wait<<<1, 32, 0, (cudaStream_t)stream>>>(d_flags, n, skip, value, h->d_err);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

int ovn_check(ovn_handle* h, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  return check_device_error(h, (cudaStream_t)stream);
}

int ovn_set_feature_center(ovn_handle* h, const float* h_mu) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  if (h->cfg.precision != OVN_PREC_F16_TC) return OVN_OK;
  if (!h->weights_ready) OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_set_feature_center: weights not finalised");
  return tc_set_center(h, h_mu);
}

int ovn_calibrate(ovn_handle* h, const float* d_volume, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, d_volume != nullptr, "d_volume is NULL");
  if (h->cfg.precision != OVN_PREC_F16_TC) return OVN_OK;
  if (!h->weights_ready) OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_calibrate: weights not finalised");
  return tc_calibrate(h, d_volume, (cudaStream_t)stream);
}

int ovn_get_feature_center(ovn_handle* h, float* h_mu, int32_t* is_set) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, h_mu && is_set, "NULL pointer");
  if (h->cfg.precision != OVN_PREC_F16_TC || !h->weights_ready) {
    for (int c = 0; c < kFeatC; ++c) h_mu[c] = 0.f;
    *is_set = 0;
    return OVN_OK;
  }
  return tc_get_center(h, h_mu, is_set);
}

int ovn_bank_release(ovn_handle* h, const float* d_bank) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  if (h->cfg.precision != OVN_PREC_F16_TC) return OVN_OK;
  return tc_bank_release(h, d_bank);
}

// ---- training: heads on a frozen leg, and the full network (train.cu) ------------------------------
static int head_layer_index(const char* name) {
  for (int l = 0; l < 4; ++l)
    if (name && strcmp(name, kHeadNames[l]) == 0) return l;
  return -1;
}

int ovn_heads_backward(ovn_handle* h, const float* d_bank, int64_t bank_size, const int32_t* d_left,
                       const int32_t* d_right, int32_t n_pairs, const float* d_overlap_gt, const int32_t* d_yaw_bin_gt,
                       float min_overlap_for_angle, float* d_losses, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_pairs > 0 && bank_size > 0, "n_pairs and bank_size must be positive");
  REQUIRE(h, d_bank && d_left && d_right && d_overlap_gt && d_yaw_bin_gt && d_losses, "NULL pointer");
  if (!h->net_ok) OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "ovn_heads_backward: %s", h->net_error.c_str());
  if (!h->weights_ready) OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_heads_backward: weights not finalised");
  if (n_pairs > h->cfg.max_batch_pairs)
    OVN_SET_ERR(h, OVN_ERR_CAPACITY, "ovn_heads_backward: n_pairs=%d exceeds max_batch_pairs=%d", n_pairs,
                h->cfg.max_batch_pairs);
  int rc = train_heads_backward(h, d_bank, bank_size, d_left, d_right, n_pairs, d_overlap_gt, d_yaw_bin_gt,
                                min_overlap_for_angle, d_losses, (cudaStream_t)stream);
  if (rc == OVN_OK) OVN_CUDA(h, cudaEventRecord(h->ev_train, (cudaStream_t)stream));
  return rc;
}

int ovn_get_gradient(ovn_handle* h, const char* layer_name, float* h_kernel, float* h_bias) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  const int l = head_layer_index(layer_name);
  if (l >= 0) return train_get_gradient(h, l, h_kernel, h_bias);
  int slot = -1;
  if (layer_name && train_has_leg_gradients(h) && find_layer(h, layer_name, &slot) && slot < kMaxLegLayers)
    return train_get_gradient(h, kMaxLegLayers + slot, h_kernel, h_bias);
  OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_get_gradient: '%s' is not a trained head layer%s",
              layer_name ? layer_name : "(null)",
              train_has_leg_gradients(h) ? " or leg layer" : " (leg gradients need ovn_network_backward)");
}

int ovn_network_backward(ovn_handle* h, const float* d_inputs, int64_t n_inputs, const int32_t* d_left,
                         const int32_t* d_right, const int32_t* d_right_roll, int32_t n_pairs,
                         const float* d_overlap_gt, const int32_t* d_yaw_bin_gt, float min_overlap_for_angle,
                         float* d_losses, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_pairs > 0 && n_inputs > 0, "n_pairs and n_inputs must be positive");
  REQUIRE(h, d_inputs && d_left && d_right && d_overlap_gt && d_yaw_bin_gt && d_losses, "NULL pointer");
  if (!h->net_ok) OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "ovn_network_backward: %s", h->net_error.c_str());
  if (!h->weights_ready) OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_network_backward: weights not finalised");
  if (n_pairs > h->cfg.max_batch_pairs)
    OVN_SET_ERR(h, OVN_ERR_CAPACITY, "ovn_network_backward: n_pairs=%d exceeds max_batch_pairs=%d", n_pairs,
                h->cfg.max_batch_pairs);
  int rc = train_network_backward(h, d_inputs, n_inputs, d_left, d_right, d_right_roll, n_pairs, d_overlap_gt,
                                  d_yaw_bin_gt, min_overlap_for_angle, d_losses, (cudaStream_t)stream);
  if (rc == OVN_OK) OVN_CUDA(h, cudaEventRecord(h->ev_train, (cudaStream_t)stream));
  return rc;
}

int ovn_adagrad_step(ovn_handle* h, float lr, void* stream) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, isfinite(lr) && lr >= 0.f, "learning rate must be finite and non-negative");
  bool leg_changed = false;
  int rc = train_adagrad_step(h, lr, (cudaStream_t)stream, &leg_changed);
  if (rc == OVN_OK) {
    h->weights_trained = true;
    if (leg_changed) h->leg_trained = true;
    OVN_CUDA(h, cudaEventRecord(h->ev_train, (cudaStream_t)stream));
  }
  return rc;
}

int ovn_get_weights(ovn_handle* h, const char* layer_name, float* h_kernel, float* h_bias) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, layer_name && h_kernel && h_bias, "NULL pointer");
  auto it = h->host_w.find(layer_name);
  if (it == h->host_w.end() || !it->second.set)
    OVN_SET_ERR(h, OVN_ERR_WEIGHTS, "ovn_get_weights: layer '%s' has no weights", layer_name);
  const LayerWeights& w = it->second;
  const int l = head_layer_index(layer_name);
  int slot = l >= 0 ? kMaxLegLayers + l : -1;
  if (l < 0 && h->leg_trained) find_layer(h, layer_name, &slot);
  if (slot >= 0 && h->weights_trained) {     // the device master copy is newer than host_w
    OVN_CUDA(h, cudaEventSynchronize(h->ev_train));
    OVN_CUDA(h, cudaMemcpy(h_kernel, h->d_w[slot], w.kernel.size() * sizeof(float), cudaMemcpyDeviceToHost));
    OVN_CUDA(h, cudaMemcpy(h_bias, h->d_b[slot], w.bias.size() * sizeof(float), cudaMemcpyDeviceToHost));
    return OVN_OK;
  }
  memcpy(h_kernel, w.kernel.data(), w.kernel.size() * sizeof(float));
  memcpy(h_bias, w.bias.data(), w.bias.size() * sizeof(float));
  return OVN_OK;
}

// ---- host-buffer entry points ---------------------------------------------------------------------
static int ensure_stage(ovn_handle* h, int64_t n_points, int n_scans) {
  if (n_points > h->cap_stage_points) {
    if (h->d_stage_points) cudaFree(h->d_stage_points);
    h->d_stage_points = nullptr;
    const int64_t cap = n_points + n_points / 8 + 4096;
    OVN_CUDA(h, cudaMalloc(&h->d_stage_points, cap * 4 * sizeof(float)));
    h->cap_stage_points = cap;
  }
  if (!h->d_stage_offsets) OVN_CUDA(h, cudaMalloc(&h->d_stage_offsets, ((size_t)h->cfg.max_batch_scans + 1) * sizeof(int64_t)));
  (void)n_scans;
  return OVN_OK;
}

int ovn_encode_clouds_host(ovn_handle* h, const float* h_points, const int64_t* h_offsets, int32_t n_scans,
                           float* h_fv) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_scans >= 0, "negative size");
  if (n_scans == 0) return OVN_OK;
  REQUIRE(h, h_points && h_offsets && h_fv, "NULL pointer");
  if (h->cfg.n_prob_channels != 0)
    OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "ovn_encode_clouds_host: semantic channels need per-point probabilities; "
                "use the device-pointer stages");
  cudaStream_t s = h->own_stream;
  const int Wf = h->cfg.leg_output_width;
  float* d_fv = nullptr;
  OVN_CUDA(h, cudaMalloc(&d_fv, (size_t)h->cfg.max_batch_scans * Wf * kFeatC * sizeof(float)));
  int rc = OVN_OK;
  for (int s0 = 0; s0 < n_scans && rc == OVN_OK; s0 += h->cfg.max_batch_scans) {
    const int n = (n_scans - s0 < h->cfg.max_batch_scans) ? n_scans - s0 : h->cfg.max_batch_scans;
    const int64_t p0 = h_offsets[s0], p1 = h_offsets[s0 + n];
    rc = ensure_stage(h, p1 - p0, n);
    if (rc != OVN_OK) break;
    std::vector<int64_t> rel(n + 1);
    for (int i = 0; i <= n; ++i) rel[i] = h_offsets[s0 + i] - p0;
    cudaError_t e = cudaMemcpyAsync(h->d_stage_points, h_points + p0 * 4, (p1 - p0) * 4 * sizeof(float),
                                    cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h->d_stage_offsets, rel.data(), (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);   // rel is a stack-lifetime buffer
    if (e != cudaSuccess) { h->last_error = cudaGetErrorString(e); rc = OVN_ERR_CUDA; break; }
    rc = preprocess_batch(h, h->d_stage_points, h->d_stage_offsets, n, p1 - p0, nullptr, h->d_input, s);
    if (rc == OVN_OK) rc = ovn_leg_forward(h, h->d_input, n, d_fv, s);
    if (rc == OVN_OK) {
      e = cudaMemcpyAsync(h_fv + (size_t)s0 * Wf * kFeatC, d_fv, (size_t)n * Wf * kFeatC * sizeof(float),
                          cudaMemcpyDeviceToHost, s);
      if (e != cudaSuccess) { h->last_error = cudaGetErrorString(e); rc = OVN_ERR_CUDA; }
      else rc = check_device_error(h, s);                 // synchronises s
    }
  }
  cudaFree(d_fv);
  return rc;
}

int ovn_query_cloud_vs_bank_host(ovn_handle* h, const float* h_points, int64_t n_points, const float* d_bank,
                                 int64_t bank_size, const int32_t* h_cand_idx, int32_t n_cand, float* h_overlap,
                                 int32_t* h_yaw, float* h_query_fv) {
  if (!h) return OVN_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  REQUIRE(h, n_points >= 0 && n_cand >= 0, "negative size");
  REQUIRE(h, h_points, "h_points is NULL");
  REQUIRE(h, n_cand == 0 || (d_bank && h_overlap && h_yaw), "NULL pointer");
  REQUIRE(h, n_cand == 0 || bank_size > 0, "bank_size must be positive");
  REQUIRE(h, h_cand_idx != nullptr || n_cand <= bank_size, "n_cand exceeds bank_size");
  if (h->cfg.n_prob_channels != 0)
    OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "ovn_query_cloud_vs_bank_host: semantic channels are not supported here");
  if (n_cand > h->cfg.max_batch_pairs)
    OVN_SET_ERR(h, OVN_ERR_CAPACITY, "n_cand=%d exceeds max_batch_pairs=%d", n_cand, h->cfg.max_batch_pairs);
  cudaStream_t s = h->own_stream;
  int rc = ensure_stage(h, n_points, 1);
  if (rc != OVN_OK) return rc;
  const int Wf = h->cfg.leg_output_width;
  const int maxp = h->cfg.max_batch_pairs;
  // pinned staging: [0,64) error flag + the two offsets; then cand idx / overlap / yaw (4 B x max_batch_pairs each).
  // Everything the device reads or writes asynchronously lives there, so the call has ONE host sync.
  uint8_t* pin = reinterpret_cast<uint8_t*>(h->h_pinned);
  int64_t* p_offs = reinterpret_cast<int64_t*>(pin + 16);
  int32_t* p_idx = reinterpret_cast<int32_t*>(pin + 64);
  float* p_ov = reinterpret_cast<float*>(pin + 64 + (size_t)maxp * 4);
  int32_t* p_yaw = reinterpret_cast<int32_t*>(pin + 64 + (size_t)maxp * 8);
  p_offs[0] = 0; p_offs[1] = n_points;
  // the bank's operand copies may have been prepared on another stream (ovn_bank_prepare records ev_bank)
  OVN_CUDA(h, cudaStreamWaitEvent(s, h->ev_bank, 0));
  OVN_CUDA(h, cudaMemcpyAsync(h->d_stage_points, h_points, (size_t)n_points * 4 * sizeof(float), cudaMemcpyHostToDevice, s));
  OVN_CUDA(h, cudaMemcpyAsync(h->d_stage_offsets, p_offs, 2 * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  if (h_cand_idx && n_cand > 0) {
    memcpy(p_idx, h_cand_idx, (size_t)n_cand * sizeof(int32_t));
    OVN_CUDA(h, cudaMemcpyAsync(h->d_idx_tmp, p_idx, (size_t)n_cand * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  }
  rc = preprocess_batch(h, h->d_stage_points, h->d_stage_offsets, 1, n_points, nullptr, h->d_input, s);
  if (rc != OVN_OK) return rc;
  rc = ovn_leg_forward(h, h->d_input, 1, h->d_query_fv, s);
  if (rc != OVN_OK) return rc;
  if (n_cand > 0) {
    int32_t* d_yaw = h->d_idx_tmp + maxp;
    if (!h_cand_idx) {
      k_iota<<<(n_cand + 255) / 256, 256, 0, s>>>(h->d_idx_tmp, n_cand, 0);
      OVN_LAUNCH_CHECK(h);
    }
    rc = heads_dispatch(h, d_bank, bank_size, h->d_query_fv, h->d_idx_tmp, nullptr, n_cand, h->d_logit, d_yaw, nullptr, s);
    if (rc != OVN_OK) return rc;
    OVN_CUDA(h, cudaMemcpyAsync(p_ov, h->d_logit, (size_t)n_cand * sizeof(float), cudaMemcpyDeviceToHost, s));
    OVN_CUDA(h, cudaMemcpyAsync(p_yaw, d_yaw, (size_t)n_cand * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  }
  if (h_query_fv)
    OVN_CUDA(h, cudaMemcpyAsync(h_query_fv, h->d_query_fv, (size_t)Wf * kFeatC * sizeof(float), cudaMemcpyDeviceToHost, s));
  rc = check_device_error(h, s);            // the one synchronisation of the call
  if (n_cand > 0) {                         // results are delivered even on error (poisoned: NaN / INT32_MIN)
    memcpy(h_overlap, p_ov, (size_t)n_cand * sizeof(float));
    memcpy(h_yaw, p_yaw, (size_t)n_cand * sizeof(int32_t));
  }
  return rc;
}

}  // extern "C"
