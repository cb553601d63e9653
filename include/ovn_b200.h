/*
 * ovn_b200.h -- C ABI of the Blackwell-native OverlapNet inference hot path (libovn_b200.so).
 *
 * The reference (PRBonn/OverlapNet) has no FFI / plugin interface: its boundary is the Python
 * class `Infer` (src/two_heads/infer.py:22-265) plus the NumPy preprocessing functions
 * (src/utils/utils.py:59-186).  This header is the native boundary a maintainer binds underneath
 * those Python entry points (ctypes stub in INTEGRATION.md); every function names the reference
 * code it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - Pointers named d_* are DEVICE pointers, h_* are HOST pointers.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Device-pointer
 *     entry points are asynchronous on that stream and never synchronise the host; host-buffer
 *     entry points (suffix _host) copy in/out and return after the result is on the host.
 *   - Every function returns an ovn_status (0 = OK, negative = error); no exception crosses the ABI.
 *     ovn_last_error(h) gives the message for the last failure on that handle.
 *   - A handle owns the packed weights and all workspaces, is bound to the CUDA device that was
 *     current at ovn_create(), and is NOT thread-safe (like `Infer`: infer.py keeps a mutable
 *     feature bank, SURVEY 8b "Threading").
 *   - Feature volumes cross the ABI as float32 [n][W_out=360][128] (what
 *     Infer.create_feature_volumes returns, infer.py:240-265, with the singleton H axis dropped).
 */
#ifndef OVN_B200_H_
#define OVN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OVN_ABI_VERSION 1

typedef enum ovn_status {
  OVN_OK = 0,
  OVN_ERR_INVALID_ARG = -1,    /* NULL pointer, bad size, bad enum */
  OVN_ERR_BAD_CONFIG = -2,     /* unsupported model wiring (config/network.yml:64-82) */
  OVN_ERR_WEIGHTS = -3,        /* unknown layer name / wrong shape / weights not finalised */
  OVN_ERR_CUDA = -4,           /* a CUDA runtime call failed; see ovn_last_error */
  OVN_ERR_NO_DEVICE = -5,      /* no sm_100 device: the library has NO CPU fallback */
  OVN_ERR_CAPACITY = -6        /* batch larger than the workspace reserved at ovn_create */
} ovn_status;

/* Arithmetic of the network kernels. */
typedef enum ovn_precision {
  OVN_PREC_FP32 = 0,           /* fp32 SIMT kernels (verification path) */
  OVN_PREC_F16_TC = 1          /* fp16 operands, fp32 accumulate in TMEM, tcgen05 tensor cores */
} ovn_precision;

/*
 * Model + projection configuration.  Mirrors the keys Infer.__init__ reads from
 * config/network.yml (infer.py:32-93) and the defaults of range_projection (utils.py:59).
 */
typedef struct ovn_config {
  int32_t abi_version;            /* must be OVN_ABI_VERSION */
  /* range projection, utils.py:59 */
  int32_t proj_H, proj_W;         /* 64, 900 (network.yml:75 inputShape) */
  float   fov_up_deg, fov_down_deg; /* 3.0, -25.0 */
  float   max_range;              /* 50.0 */
  /* input cues, network.yml:20-24, channel order ImagePairOverlapOrientationSequence.py:143-207 */
  int32_t use_depth;              /* 1 channel  */
  int32_t use_normals;            /* 3 channels */
  int32_t n_prob_channels;        /* 0, 3 (pca) or 20 */
  int32_t use_intensity;          /* 1 channel  */
  /* leg, generateNet.py:119-219 / network.yml:70-82 */
  int32_t strides_layer1[2];      /* (2,2) */
  int32_t additional_unsymmetric_layer3a; /* 1 */
  int32_t leg_output_width;       /* 360 */
  /* overlap head, generateNet.py:88-89 */
  int32_t conv1size;              /* 15 */
  /* execution */
  int32_t precision;              /* ovn_precision */
  int32_t max_batch_scans;        /* workspace: scans per ovn_leg_forward / ovn_project_batch call */
  int32_t max_batch_pairs;        /* workspace: pairs per ovn_heads_forward call */
} ovn_config;

typedef struct ovn_handle ovn_handle;

/* ---- lifetime -------------------------------------------------------------------------- */
void        ovn_default_config(ovn_config* cfg);            /* network.yml geo-only defaults */
int         ovn_create(const ovn_config* cfg, ovn_handle** out);   /* replaces Infer.__init__ model build, infer.py:86-111 */
int         ovn_destroy(ovn_handle* h);
const char* ovn_last_error(const ovn_handle* h);
const char* ovn_status_string(int status);
int         ovn_abi_version(void);
int         ovn_input_channels(const ovn_handle* h);        /* infer.py:61-73 */
int         ovn_feature_width(const ovn_handle* h);         /* 360 */
int         ovn_feature_channels(const ovn_handle* h);      /* 128 */
/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t     ovn_launch_count(const ovn_handle* h);

/* ---- per-kernel device timing (bench.py roofline): CUDA events recorded around the named kernels
 * on the launching stream while enabled.  ovn_profile_read synchronises the device, returns the
 * accumulated milliseconds / launch count since the last read and resets them.  Names:
 * "delta_conv1", "conv2", "conv3", "corr", "project_scatter", "project_gather", "leg". */
int ovn_profile_enable(ovn_handle* h, int on);
int ovn_profile_read(ovn_handle* h, const char* kernel, double* total_ms, int64_t* launches);

/* ---- weights: replaces load_weights(by_name=True), infer.py:117-120 ----------------------- */
/* kernel: Keras layout, conv (kh,kw,cin,cout) / dense (in,out), float32 host memory; bias (cout).
 * Layer names: s_conv1..s_conv10 (+s_conv3a), c_conv1..c_conv3, overlap_output
 * (generateNet.py:99-114,162-214). */
int ovn_set_weights(ovn_handle* h, const char* layer_name,
                    const float* h_kernel, const int64_t* kernel_dims, int32_t kernel_ndim,
                    const float* h_bias, int64_t bias_len);
int ovn_finalize_weights(ovn_handle* h);   /* pack + upload; every layer must have been set */

/* ---- stage 1: range projection (utils.py:59-134) ------------------------------------------ */
/* d_points: [n_total][4] float32 x,y,z,intensity of `n_scans` clouds back to back;
 * d_offsets: [n_scans+1] int64 point offsets (device).  Outputs are optional (NULL = skip):
 *   d_range [n][H][W] f32, d_vertex [n][H][W][4] f32, d_intensity [n][H][W] f32,
 *   d_idx [n][H][W] i32 (index into the FILTERED cloud, utils.py:76,117-118).
 * max_range < 0 selects the handle's configured max_range; +inf is allowed
 * (gen_semantic_data.py:39). */
int ovn_project_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int32_t n_scans,
                      int64_t n_points_total, float max_range,
                      float* d_range, float* d_vertex, float* d_intensity, int32_t* d_idx,
                      void* stream);

/* ---- stage 1b: normal map (utils.py:137-175) ---------------------------------------------- */
int ovn_normals_batch(ovn_handle* h, const float* d_range, const float* d_vertex, int32_t n_scans,
                      float* d_normal /* [n][H][W][3] */, void* stream);

/* ---- stage 1c: semantic gather (gen_semantic_data.py:41-46, incl. the filtered-index quirk) */
int ovn_semantic_batch(ovn_handle* h, const int32_t* d_idx, const float* d_probs,
                       const int64_t* d_offsets, int32_t n_scans, int32_t n_classes,
                       float* d_out /* [n][H][W][n_classes] */, void* stream);

/* ---- ground-truth generator (com_overlap_yaw.py:10-68; SURVEY 8f-2) ------------------------- */
/* Float32 range images [n][H][W] of scans moved into the current frame: every point (x, y, z, 1)
 * is multiplied, in float64, by d_pose_ref[scan] and then by d_pose_cur_inv (row-major 4x4, either
 * may be NULL = identity; com_overlap_yaw.py:39-40) and projected by range_projection evaluated in
 * FLOAT64 (the reference's load_vertex builds a float64 array, utils.py:218-231; bins utils.py:75-104),
 * nearest point per pixel, depth rounded to float32 on store, -1 where empty (utils.py:120,129).
 * max_range < 0 selects the handle's configured max_range. */
int ovn_gt_range_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int32_t n_scans,
                       int64_t n_points_total, const double* d_pose_ref /* [n][16] */,
                       const double* d_pose_cur_inv /* [16] */, float max_range,
                       float* d_range /* [n][H][W] */, void* stream);

/* d_counts[b] = #{pixels: ref_b > 0 and |ref_b - cur| < 1} for b < n_scans (com_overlap_yaw.py:44-45,
 * float32 arithmetic); d_counts[n_scans] = #{cur > 0} = the reference's valid_num (:31-32). */
int ovn_gt_overlap_count(ovn_handle* h, const float* d_ref_ranges /* [n][H][W] */,
                         const float* d_cur_range /* [H][W] */, int32_t n_scans,
                         int32_t* d_counts /* [n_scans + 1] */, void* stream);

/* For pair k (d_pairs[2k] = current frame c, d_pairs[2k+1] = reference scan r):
 * d_counts[k] = #{pixels: ref > 0 and |ref - cur_c| < 1}, where ref = scan r moved by d_pose_ref[r]
 * and then d_pose_cur_inv[c] (float64), projected as in ovn_gt_range_batch.  Equal to
 * ovn_gt_range_batch + ovn_gt_overlap_count of that pair.  com_overlap_yaw.py:35-46 for many frames.
 * Scan r is d_points[d_offsets[r] .. d_offsets[r+1]); d_cur_ranges are the current frames' images as
 * ovn_gt_range_batch makes them without poses.  One CTA builds each pair's H x W image in shared
 * memory: OVN_ERR_BAD_CONFIG when H*W*4 bytes exceed what a block may use (64 x 900 fits).  Order
 * the pairs reference-major so that concurrent CTAs share one scan's points in L2.  Indices outside
 * [0, n_cur) / [0, n_scans) are clamped, the count is poisoned (-1) and the next synchronising call
 * (ovn_check) returns OVN_ERR_INVALID_ARG.  max_range < 0 selects the handle's configured max_range. */
int ovn_gt_pair_counts(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int32_t n_scans,
                       int64_t n_points_total, const double* d_pose_ref /* [n_scans][16] */,
                       const double* d_pose_cur_inv /* [n_cur][16] */, const float* d_cur_ranges /* [n_cur][H][W] */,
                       int32_t n_cur, const int32_t* d_pairs /* [n_pairs][2] */, int64_t n_pairs,
                       float max_range, int32_t* d_counts /* [n_pairs] */, void* stream);

/* ---- stage 1d: fused raw cloud -> packed network input ------------------------------------- */
/* Projection + normals + channel packing (ImagePairOverlapOrientationSequence.py:130-207) in one
 * pass; d_probs may be NULL when n_prob_channels == 0.  d_input: [n][H][W][C] float32. */
int ovn_preprocess_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets,
                         int32_t n_scans, int64_t n_points_total, const float* d_probs,
                         float* d_input, void* stream);

/* Pack separately computed cue images into the NHWC network input (same channel order). */
int ovn_pack_input(ovn_handle* h, const float* d_depth, const float* d_normal, const float* d_prob,
                   const float* d_intensity, int32_t n_scans, float* d_input, void* stream);

/* ---- stage 2: leg encoder (generateNet.py:161-217; Infer.create_feature_volumes) ----------- */
/* d_input [n][H][W][C] f32 -> d_fv [n][360][128] f32. */
int ovn_leg_forward(ovn_handle* h, const float* d_input, int32_t n_scans, float* d_fv, void* stream);

/* ---- stage 3: heads (generateNet.py:15-116, 327-354; readout infer.py:157-158) ------------- */
/* Pair p uses LEFT = d_bank[left_idx[p]], RIGHT = d_bank[right_idx[p]]
 * (ImagePairOverlapSequenceFeatureVolume.py:44-45).  Outputs: d_overlap [n] f32,
 * d_yaw [n] i32 = 180 - argmax(corr) (first maximum), d_corr [n][360] f32 or NULL. */
int ovn_heads_forward(ovn_handle* h, const float* d_bank, int64_t bank_size,
                      const int32_t* d_left_idx, const int32_t* d_right_idx, int32_t n_pairs,
                      float* d_overlap, int32_t* d_yaw, float* d_corr, void* stream);

/* 1 query vs N candidates (Infer.infer_multiple, infer.py:162-203): RIGHT = the query volume
 * d_query [360][128] for every pair, LEFT = d_bank[cand_idx[p]] (cand_idx NULL = 0..n-1). */
int ovn_heads_1vsN(ovn_handle* h, const float* d_bank, int64_t bank_size, const float* d_query,
                   const int32_t* d_cand_idx, int32_t n_cand,
                   float* d_overlap, int32_t* d_yaw, float* d_corr, void* stream);

/* Rows [row_lo, row_hi) of the ordered all-pairs matrix of a bank (Infer.infer_multiple_vs_multiple,
 * infer.py:205-238, with every (first, second) combination; testing.py:237-272): for each row i,
 * RIGHT = d_bank[i] and LEFT = d_bank[j] for every j < bank_size.  The delta head is not symmetric in
 * (LEFT, RIGHT), so all ordered pairs are computed.  d_overlap / d_yaw: [row_hi - row_lo][bank_size].
 * The loop over rows runs inside the library (no per-row host round trip through the caller). */
int ovn_heads_rows_vs_bank(ovn_handle* h, const float* d_bank, int64_t bank_size, int64_t row_lo, int64_t row_hi,
                           float* d_overlap, int32_t* d_yaw, void* stream);

/* ---- resident bank (Infer keeps self.feature_volumes across calls, infer.py:113,184-193) ---------
 * The tensor-core heads consume fp16 / hi-lo split copies of the LEFT volumes.  Without this call
 * they are rebuilt from d_bank on every heads call; ovn_bank_prepare builds them once for rows
 * [first, first+count) of the bank that lives at d_bank (capacity = rows the bank may grow to), and
 * every later ovn_heads_forward / ovn_heads_1vsN whose d_bank is the same pointer reuses them.
 * Call it again for rows that were appended or overwritten.  No-op for precision fp32. */
int ovn_bank_prepare(ovn_handle* h, const float* d_bank, int64_t bank_capacity, int64_t first, int64_t count,
                     void* stream);
int ovn_bank_release(ovn_handle* h, const float* d_bank);

/* ---- deferred device errors ------------------------------------------------------------------
 * The device-pointer entry points never synchronise, so two classes of error can only be detected on
 * the device: an index outside [0, bank_size) (or, for a resident bank, a row that was never
 * prepared), and a bounded pipeline-barrier wait of a tensor-core kernel that timed out (GPU
 * time-slicing, debuggers).  Both raise a flag on the device; the kernels that write overlap / yaw
 * then POISON their outputs (overlap = NaN, yaw = INT32_MIN) so garbage never looks valid, indices are
 * clamped so no out-of-bounds read happens, and the flag is turned into a status by the next entry point
 * that synchronises anyway: ovn_check (synchronises `stream`), the *_host entry points and
 * ovn_profile_read.  OVN_ERR_INVALID_ARG for index errors, OVN_ERR_CUDA for time-outs; the flag is
 * cleared when it is reported. */
int ovn_check(ovn_handle* h, void* stream);

/* ---- device-side signalling between the GPUs of a sharded bank (overlapnet_b200/search.py, transport 'symm') --
 * The query volume and the result table of a sharded 1-vs-N search live in symmetric (peer-mapped) memory:
 * kernels read / write them directly over NVLink, and these two calls replace the collectives.  A flag is an
 * int32 slot in that memory holding the number of the last finished step.
 *   ovn_peer_signal: ONE launch stores `value` (release, system scope -- after everything queued on `stream`
 *                    before it) to each of the n flag addresses (host array of peer-mapped device addresses).
 *   ovn_peer_wait:   ONE launch spins (acquire, system scope, bounded) until d_flags[i] >= value for every
 *                    i < n except i == skip.  A time-out raises the handle's deferred error (ovn_check). */
int ovn_peer_signal(ovn_handle* h, const uint64_t* h_flag_ptrs, int32_t n, int32_t value, void* stream);
int ovn_peer_wait(ovn_handle* h, const int32_t* d_flags, int32_t n, int32_t skip, int32_t value, void* stream);

/* ---- feature centre of the tensor-core delta head ------------------------------------------------
 * DeltaLayer only sees |l - r| (generateNet.py:59), which is invariant to a common per-channel offset:
 * the fp16 operand copies of the volumes are stored as fp16(x - mu[c]), which shrinks their rounding
 * error (measured: 3x on leg outputs, profiles/r2_precision_budget.txt).  mu is calibrated automatically
 * on the first volume the handle sees (first ovn_bank_prepare row, else the first RIGHT volume) and
 * then frozen until ovn_finalize_weights; ovn_set_feature_center(h, mu[128]) fixes it explicitly
 * (NULL = back to automatic; not allowed while a bank is resident).  No effect for precision fp32. */
int ovn_set_feature_center(ovn_handle* h, const float* h_mu);
int ovn_get_feature_center(ovn_handle* h, float* h_mu /* [128] */, int32_t* is_set);
/* The same offset trick is applied to the two intermediate images (o1, x3: c_conv2 and c_conv3 are
 * linear, the mean's image is folded into the layer's bias with exact fp32 weights).  All three centres are
 * derived from ONE feature volume V0 with fixed summation orders: mu = channel means of V0, the o1 / x3
 * centres = channel means over the canonical pair (V0, V0 rolled by half a turn).  V0 is the first volume
 * the handle sees, or the one given here: ovn_calibrate(h, d_volume [360][128]) makes the calibration
 * explicit, so that handles on different GPUs (a sharded bank) produce bit-identical results. */
int ovn_calibrate(ovn_handle* h, const float* d_volume, void* stream);

/* ---- overlap-head training on a frozen leg (training.py with legsType 360OutputkLegsFixed,
 * generateNet.py:222-324).  The forward and all gradients but dW1 run in fp32; dW1 runs in fp32 on
 * precision fp32 handles and on tensor cores (fp16 operands, fp32 accumulation) on f16_tc handles.
 * ovn_heads_backward: for pairs LEFT = d_bank[d_left[p]], RIGHT = d_bank[d_right[p]]
 * (ImagePairOverlapOrientationSequence.py:100-112) runs both heads, the losses
 *   d_losses[0] = 5 * L_ov + L_or, d_losses[1] = L_ov (my_sigmoid_loss, training.py:71-83),
 *   d_losses[2] = L_or (my_entropy, training.py:86-92: target bin d_yaw_bin_gt[p] carries
 *   d_overlap_gt[p] and counts as positive when > min_overlap_for_angle; pos_weight = 360)
 * and OVERWRITES the gradients of c_conv1..3 and overlap_output (L_or has none) held by the handle.
 * n_pairs <= max_batch_pairs (else OVN_ERR_CAPACITY).  Indices and yaw bins are range-checked on the
 * device like ovn_heads_forward (deferred error, ovn_check; the losses are NaN).  The training
 * workspace and the Adagrad state are allocated on the first call. */
int ovn_heads_backward(ovn_handle* h, const float* d_bank, int64_t bank_size,
                       const int32_t* d_left_idx, const int32_t* d_right_idx, int32_t n_pairs,
                       const float* d_overlap_gt, const int32_t* d_yaw_bin_gt, float min_overlap_for_angle,
                       float* d_losses /* [3] */, void* stream);
/* Gradient of a head layer (c_conv1..3, overlap_output) in Keras layout; synchronises the device.  The leg
 * layers (s_conv1..s_conv10, s_conv3a) are accepted only when the last backward call was
 * ovn_network_backward. */
int ovn_get_gradient(ovn_handle* h, const char* layer_name, float* h_kernel, float* h_bias);
/* Keras 2.1.5 Adagrad (training.py:253) on the device fp32 weights of the layers the last backward call
 * produced gradients for (the four head layers; after ovn_network_backward also the leg):
 * a += g^2; w -= lr * g / (sqrt(a) + 1e-7).  Accumulators start at zero and are reset by
 * ovn_set_weights (head and leg alike).  Afterwards the inference entry points refuse (OVN_ERR_WEIGHTS) until
 * ovn_finalize_weights repacks from the trained weights (and re-calibrates the centres on next use). */
int ovn_adagrad_step(ovn_handle* h, float lr, void* stream);
/* Current weights of any layer in Keras layout (trained head weights included); synchronises. */
int ovn_get_weights(ovn_handle* h, const char* layer_name, float* h_kernel, float* h_bias);

/* ---- full-network training (training.py with legsType 360OutputkLegs, generateNet.py:119-219).
 * ovn_network_backward: the Siamese leg runs on LEFT image d_inputs[d_left_idx[p]] and RIGHT image
 * d_inputs[d_right_idx[p]] of every pair (ImagePairOverlapOrientationSequence.py:100-112), the RIGHT image
 * rolled by d_right_roll[p] columns first (np.roll along the width, any integer, taken modulo W; NULL = no
 * roll).  Both heads then run on the 2n feature volumes; the losses are those of ovn_heads_backward.  The
 * call OVERWRITES the gradients of every layer: the four head layers (bit-identical to ovn_heads_backward on
 * the same fp32 volumes) and the 11 leg layers (each the sum over both images of every pair; L_or now has
 * a gradient).  Everything but dW1 of c_conv1 is fp32 SIMT in both precisions; dW1 follows the precision as
 * in ovn_heads_backward.  n_pairs <= max_batch_pairs (else OVN_ERR_CAPACITY).  Indices and yaw bins are
 * range-checked on the device (deferred error, NaN losses).  The leg training buffers are allocated on the
 * first call and grown to the largest n_pairs seen.  Afterwards ovn_get_gradient also accepts the leg layer
 * names, and ovn_adagrad_step also updates the leg; after such a step ovn_leg_forward (and the host entry
 * points built on it) refuses with OVN_ERR_WEIGHTS until ovn_finalize_weights. */
int ovn_network_backward(ovn_handle* h, const float* d_inputs /* [n_inputs][H][W][C] */, int64_t n_inputs,
                         const int32_t* d_left_idx, const int32_t* d_right_idx,
                         const int32_t* d_right_roll /* [n_pairs] columns, NULL = none */, int32_t n_pairs,
                         const float* d_overlap_gt, const int32_t* d_yaw_bin_gt, float min_overlap_for_angle,
                         float* d_losses /* [3] */, void* stream);

/* ---- host-buffer convenience entry points (what a non-CUDA caller binds; bench.py e2e) ------ */
/* Raw clouds on the host -> feature volumes on the host. */
int ovn_encode_clouds_host(ovn_handle* h, const float* h_points, const int64_t* h_offsets,
                           int32_t n_scans, float* h_fv);
/* One raw query cloud on the host vs a device-resident bank: preprocess + leg + heads.
 * h_overlap [n_cand], h_yaw [n_cand]; h_query_fv [360][128] may be NULL. */
int ovn_query_cloud_vs_bank_host(ovn_handle* h, const float* h_points, int64_t n_points,
                                 const float* d_bank, int64_t bank_size,
                                 const int32_t* h_cand_idx, int32_t n_cand,
                                 float* h_overlap, int32_t* h_yaw, float* h_query_fv);

#ifdef __cplusplus
}
#endif
#endif /* OVN_B200_H_ */
