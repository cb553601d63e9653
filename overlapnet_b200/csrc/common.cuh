// common.cuh -- handle, error plumbing and small device helpers shared by all translation units.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <map>

#include "../../include/ovn_b200.h"

namespace ovn {

constexpr int kFeatC = 128;           // leg output channels (generateNet.py:214)
constexpr int kMaxLegLayers = 12;
enum ProfKind { PROF_DELTA = 0, PROF_CONV2, PROF_CONV3, PROF_CORR, PROF_SCATTER, PROF_GATHER, PROF_LEG, kProfKinds };

struct ConvSpec {                      // one Conv2D layer (valid padding, bias)
  char name[24];
  int kh, kw, sh, sw, cin, cout;
  int relu;
  int h_in, w_in, h_out, w_out;
};

struct LayerWeights {
  std::vector<float> kernel;           // Keras layout, flattened
  std::vector<int64_t> dims;
  std::vector<float> bias;
  bool set = false;
};

}  // namespace ovn

namespace ovn { struct TcState; struct TrainState; }

struct ovn_handle {
  ovn_config cfg;
  int device = 0;
  int sm_count = 0;
  std::string last_error;
  int64_t launches = 0;

  int C = 0;                            // input channels (infer.py:61-73)
  int n_leg = 0;
  ovn::ConvSpec leg[ovn::kMaxLegLayers];
  ovn::ConvSpec head[3];                // c_conv1..3 in "delta image" coordinates
  int o1_h = 0, o1_w = 0;               // c_conv1 output (360, 24)
  int o2_h = 0, o2_w = 0;               // c_conv2 output (24, 24)
  int o3_h = 0, o3_w = 0;               // c_conv3 output (22, 22)
  int dense_in = 0;

  std::map<std::string, ovn::LayerWeights> host_w;
  bool weights_ready = false;
  bool net_ok = false;                 // leg/head shapes valid for this config (else projection only)
  std::string net_error;

  // device weights, fp32 GEMM layout [K][N] (K = kh*kw*cin, Keras HWIO flattened is already that)
  float* d_w[ovn::kMaxLegLayers + 4] = {};
  float* d_b[ovn::kMaxLegLayers + 4] = {};
  // fp16 packed weights for the tensor-core path (layout documented in network_tc.cu)
  __half* d_w16[ovn::kMaxLegLayers + 4] = {};

  // workspaces
  unsigned long long* d_keys = nullptr;      // [max_batch_scans][H*W] atomic-min keys
  uint32_t* d_valid_words = nullptr;         // validity bitmask, 1 bit per point
  uint32_t* d_word_prefix = nullptr;         // exclusive prefix of popcounts
  uint32_t* d_scan_tmp = nullptr;
  int64_t cap_points = 0;
  float* d_act[2] = {nullptr, nullptr};      // ping-pong activations for the leg
  int64_t cap_act = 0;
  float* d_input = nullptr;                  // [max_batch_scans][H][W][C]
  float* d_o1 = nullptr;                     // [max_batch_pairs][360][24][64]
  float* d_o2 = nullptr;                     // [max_batch_pairs][24][24][128]
  float* d_logit = nullptr;                  // [max_batch_pairs]
  float* d_G = nullptr;                      // [max_batch_pairs][360][360] (fp32 path corr)
  int32_t* d_idx_tmp = nullptr;              // [max_batch_pairs] x2 scratch for 1vsN index lists
  int32_t* d_idx_san = nullptr;              // [max_batch_pairs] x2 bounds-checked (clamped) copies of the caller's index lists
  int* d_err = nullptr;                      // device error flag: pipeline barrier time-outs (1xx-8xx), bad indices (9xx)
  cudaEvent_t ev_bank = nullptr;             // recorded after ovn_bank_prepare: the host entry points (own stream) wait on it
  float* d_query_fv = nullptr;               // [360][128]
  float* d_stage_points = nullptr;           // host-entry staging of clouds
  int64_t cap_stage_points = 0;
  int64_t* d_stage_offsets = nullptr;
  void* h_pinned = nullptr;                  // pinned staging for host entry points
  int64_t cap_pinned = 0;
  cudaStream_t own_stream = nullptr;
  // per-kernel profiling (ovn_profile_enable / ovn_profile_read)
  bool profiling = false;
  std::vector<cudaEvent_t> prof_ev[ovn::kProfKinds];   // start/stop pairs, in launch order
  ovn::TcState* tc = nullptr;              // tensor-core path state (network_tc.cu)
  ovn::TrainState* tr = nullptr;           // head-training buffers and Adagrad state (train.cu), allocated on first use
  bool weights_trained = false;
  bool leg_trained = false;                // an Adagrad step changed the device leg weights: ovn_leg_forward refuses
  cudaEvent_t ev_train = nullptr;         // recorded after each training call: read-backs wait on it, not on the device            // an Adagrad step changed the device head weights: packs are stale
};

#define OVN_SET_ERR(h, code, ...)                                 \
  do {                                                            \
    char _buf[512];                                               \
    snprintf(_buf, sizeof(_buf), __VA_ARGS__);                    \
    (h)->last_error = _buf;                                       \
    return (code);                                                \
  } while (0)

#define OVN_CUDA(h, call)                                                                   \
  do {                                                                                      \
    cudaError_t _e = (call);                                                                \
    if (_e != cudaSuccess) {                                                                \
      OVN_SET_ERR(h, OVN_ERR_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,     \
                  cudaGetErrorString(_e));                                                  \
    }                                                                                       \
  } while (0)

#define OVN_LAUNCH_CHECK(h)                                                                 \
  do {                                                                                      \
    (h)->launches++;                                                                        \
    cudaError_t _e = cudaGetLastError();                                                    \
    if (_e != cudaSuccess) {                                                                \
      OVN_SET_ERR(h, OVN_ERR_CUDA, "kernel launch failed at %s:%d: %s", __FILE__, __LINE__, \
                  cudaGetErrorString(_e));                                                  \
    }                                                                                       \
  } while (0)

namespace ovn {

// Every ABI entry point runs on the device its handle was created on (ADVICE r1: Engine(device=1)
// with another current device allocated on the wrong GPU).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(const ovn_handle* h) {
    if (h && cudaGetDevice(&prev) == cudaSuccess && prev != h->device) switched = cudaSetDevice(h->device) == cudaSuccess;
  }
  ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

// error codes written to ovn_handle::d_err by kernels
constexpr int kErrBadIndex = 900;        // a pair / candidate index outside [0, bank_size)
constexpr int kErrRowNotPrepared = 901;  // resident bank: the row was never passed to ovn_bank_prepare
constexpr int kErrBadYawBin = 902;       // training: a yaw-bin target outside [0, leg_output_width)

// RAII-free profiling helpers: record an event on `s` before / after a launch when enabled
inline void prof_mark(ovn_handle* h, int kind, cudaStream_t s) {
  if (!h->profiling) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, s);
  h->prof_ev[kind].push_back(e);
}

// ---- stage entry points implemented in the .cu files (called from api.cu) -------------------
int project_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int n_scans,
                  int64_t n_total, float max_range, float* d_range, float* d_vertex,
                  float* d_intensity, int32_t* d_idx, cudaStream_t s);
int normals_batch(ovn_handle* h, const float* d_range, const float* d_vertex, int n_scans,
                  float* d_normal, cudaStream_t s);
int semantic_batch(ovn_handle* h, const int32_t* d_idx, const float* d_probs,
                   const int64_t* d_offsets, int n_scans, int n_classes, float* d_out,
                   cudaStream_t s);
int preprocess_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int n_scans,
                     int64_t n_total, const float* d_probs, float* d_input, cudaStream_t s);
int gt_range_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int n_scans, int64_t n_total,
                   const double* d_pose_ref, const double* d_pose_cur_inv, float max_range, float* d_range,
                   cudaStream_t s);
int gt_overlap_count(ovn_handle* h, const float* d_ref, const float* d_cur, int n_scans, int32_t* d_counts, cudaStream_t s);
int gt_pair_counts(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int n_scans, int64_t n_total,
                   const double* d_pose_ref, const double* d_pose_cur_inv, const float* d_cur, int n_cur,
                   const int32_t* d_pairs, int64_t n_pairs, float max_range, int32_t* d_counts, cudaStream_t s);
int pack_input(ovn_handle* h, const float* d_depth, const float* d_normal, const float* d_prob,
               const float* d_intensity, int n_scans, float* d_input, cudaStream_t s);

int leg_forward_fp32(ovn_handle* h, const float* d_input, int n, float* d_fv, cudaStream_t s);
int leg_layer_fp32(ovn_handle* h, int l, const float* x, float* y, int n, cudaStream_t s);
int heads_forward_fp32(ovn_handle* h, const float* d_bank, const float* d_query,
                       const int32_t* d_left, const int32_t* d_right, int n, float* d_overlap,
                       int32_t* d_yaw, float* d_corr, cudaStream_t s);

int corr_forward_fp32(ovn_handle* h, const float* d_bank, const float* d_query, const int32_t* left,
                      const int32_t* right, int np, int32_t* d_yaw, float* d_corr, cudaStream_t s);

int leg_forward_tc(ovn_handle* h, const float* d_input, int n, float* d_fv, cudaStream_t s);
int heads_forward_tc(ovn_handle* h, const float* d_bank, const float* d_query,
                     const int32_t* d_left, const int32_t* d_right, int n, float* d_overlap,
                     int32_t* d_yaw, float* d_corr, cudaStream_t s);
int tc_pack_weights(ovn_handle* h);
int tc_bank_prepare(ovn_handle* h, const float* d_bank, int64_t capacity, int64_t first, int64_t count, cudaStream_t s);
int tc_bank_release(ovn_handle* h, const float* d_bank);
void tc_free(ovn_handle* h);
int tc_set_center(ovn_handle* h, const float* h_mu);
int tc_get_center(ovn_handle* h, float* h_mu, int32_t* is_set);
int tc_calibrate(ovn_handle* h, const float* d_volume, cudaStream_t s);
// head training (train.cu)
int train_heads_backward(ovn_handle* h, const float* d_bank, int64_t bank_size, const int32_t* d_left,
                         const int32_t* d_right, int n, const float* d_ov_gt, const int32_t* d_bin_gt,
                         float min_ov_angle, float* d_losses, cudaStream_t s);
int train_network_backward(ovn_handle* h, const float* d_inputs, int64_t n_inputs, const int32_t* d_left,
                           const int32_t* d_right, const int32_t* d_roll, int n, const float* d_ov_gt,
                           const int32_t* d_bin_gt, float min_ov_angle, float* d_losses, cudaStream_t s);
int train_adagrad_step(ovn_handle* h, float lr, cudaStream_t s, bool* leg_changed);
bool train_has_leg_gradients(const ovn_handle* h);
int train_get_gradient(ovn_handle* h, int layer, float* h_kernel, float* h_bias);
void train_reset_optimizer(ovn_handle* h);
void train_free(ovn_handle* h);
// bounds-checked copies of index lists (d_idx_san): out-of-range entries are clamped and flagged in d_err
int sanitize_indices(ovn_handle* h, const int32_t* d_in, int n, int64_t limit, int code, int32_t* d_out, cudaStream_t s);
// read (and clear) the device error flag after the caller has synchronised `s`; maps it to a status
int check_device_error(ovn_handle* h, cudaStream_t s);

}  // namespace ovn
