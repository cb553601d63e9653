// gt_overlap.cu -- ground-truth overlap generator (com_overlap_yaw.py:10-68) on the GPU.
//
// The reference projects every reference scan, moved into the current frame by two float64 matrix
// products (com_overlap_yaw.py:39-40), with range_projection running in FLOAT64 (load_vertex builds
// a float64 array, utils.py:218-231) and compares float32 range images pixel by pixel (:44-45).
// Here: one thread per point does the two 4x4 products, the float64 depth / angle / bin pipeline
// of utils.py:75-104 and a 64-bit atomicMin of the depth's bit pattern (positive doubles order
// like integers; only the range image is needed, so no point index travels with the key); a second
// kernel rounds the winners to float32 (the image dtype, utils.py:120) and a third counts pixels.
// HBM-bound byte work: 16 B read per point, 8 B atomic per valid point into an L2-resident key image.
// k_gt_pair_counts does the same per-point work for many (current, reference) pairs at once, with the
// image in shared memory and the pixel count fused; it is bound by the FP64 pipe (DESIGN.md section 11).
#include "common.cuh"

namespace ovn {

struct GtParams {
  int H, W;
  double pi, abs_fov_down, fov, max_range;
};

constexpr unsigned long long kGtEmpty = 0xFFFFFFFFFFFFFFFFull;
#ifndef OVN_GT_PAIR_THREADS
#define OVN_GT_PAIR_THREADS 1024
#endif
constexpr int kGtPairThreads = OVN_GT_PAIR_THREADS;   // one CTA per SM (the image takes the shared memory)

// row-major 4x4 times (x, y, z, w): left-to-right sums of separately rounded products, which is
// what a reference BLAS without FMA contraction produces; FMA vs non-FMA differences (<= 1 ulp of a
// coordinate) move a point across a bin edge or the |dr| < 1 threshold with probability ~1e-12.
__device__ __forceinline__ void mat4_apply(const double* __restrict__ M, double& x, double& y, double& z, double& w) {
  double r[4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
    r[i] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(M[4 * i + 0], x), __dmul_rn(M[4 * i + 1], y)),
                               __dmul_rn(M[4 * i + 2], z)), __dmul_rn(M[4 * i + 3], w));
  x = r[0]; y = r[1]; z = r[2]; w = r[3];
}

// The float64 per-point pipeline shared by k_gt_scatter_f64 and k_gt_pair_counts: the two pose
// products (either may be NULL = identity), depth, the 0 < depth < max_range filter of utils.py:76-77
// and the clamped pixel of utils.py:86-104.  Returns false for a filtered point.
__device__ __forceinline__ bool gt_point_pixel(const float4 p, const double* __restrict__ pose_ref,
                                               const double* __restrict__ pose_cur_inv, const GtParams& P,
                                               double& depth, int& pix) {
  double x = (double)p.x, y = (double)p.y, z = (double)p.z, w = 1.0;   // load_vertex: (x, y, z, 1) float64
  if (pose_ref != nullptr) mat4_apply(pose_ref, x, y, z, w);                          // com_overlap_yaw.py:39
  if (pose_cur_inv != nullptr) mat4_apply(pose_cur_inv, x, y, z, w);                  // :40
  depth = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z)));                 // utils.py:75
  if (!(depth > 0.0 && depth < P.max_range)) return false;                                               // :76-77
  const double yaw = -atan2(y, x);                                                                       // :86
  const double pitch = asin(__ddiv_rn(z, depth));                                                        // :87
  double px = __dmul_rn(0.5, __dadd_rn(__ddiv_rn(yaw, P.pi), 1.0));                                      // :90
  double py = __dsub_rn(1.0, __ddiv_rn(__dadd_rn(pitch, P.abs_fov_down), P.fov));                        // :91
  px = floor(__dmul_rn(px, (double)P.W));                                                                // :94,98
  py = floor(__dmul_rn(py, (double)P.H));
  const int bx = (int)fmax(0.0, fmin((double)(P.W - 1), px));                                            // :99-104
  const int by = (int)fmax(0.0, fmin((double)(P.H - 1), py));
  pix = by * P.W + bx;
  return true;
}

__global__ void __launch_bounds__(256)
k_gt_scatter_f64(const float4* __restrict__ pts, const int64_t* __restrict__ offsets, int n_scans, int64_t n_total,
                 const double* __restrict__ pose_ref, const double* __restrict__ pose_cur_inv, GtParams P,
                 unsigned long long* __restrict__ keys) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_total || g < offsets[0] || g >= offsets[n_scans]) return;
  int lo = 0, hi = n_scans;                      // largest b with offsets[b] <= g
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (offsets[mid] <= g) lo = mid; else hi = mid;
  }
  const int b = lo;
  double depth;
  int pix;
  if (!gt_point_pixel(__ldg(pts + g), pose_ref != nullptr ? pose_ref + (size_t)b * 16 : nullptr, pose_cur_inv, P,
                      depth, pix))
    return;
  atomicMin(keys + (size_t)b * P.H * P.W + pix, (unsigned long long)__double_as_longlong(depth));
}

// One CTA per (current frame c, reference scan r) pair: the range image of scan r moved by
// pose_ref[r] and then pose_cur_inv[c] is built in shared memory and compared with the current
// image cur[c] right there, so no reference image ever reaches global memory (com_overlap_yaw.py:35-46
// for many current frames at once).
//
// The image holds 32-bit keys: the bit pattern of the depth rounded to float32, combined by a
// shared-memory atomicMin.  This equals ovn_gt_range_batch (64-bit atomicMin of the float64 depth,
// rounded to float32 afterwards) bit for bit:
//   - round-to-nearest is monotone, so round_f32(min d) = min round_f32(d);
//   - every depth that passes the filter is > 0, so its float32 is +0 or positive, and non-negative
//     float bit patterns order like unsigned integers; the empty key 0xFFFFFFFF is above all of them
//     (and is not > 0 as a float, like the -1 the other path stores);
//   - a depth that rounds to 0.0f gives a pixel that is not > 0 in both paths, so it never counts.
// The count is the expression of k_gt_overlap_count on the same float32 values, so the counts equal
// ovn_gt_range_batch + ovn_gt_overlap_count of that pair exactly.  The pair list is built
// reference-major by the caller, so CTAs that run together read the same scan's points from L2.
// Out-of-range pair indices are clamped, raise the device flag and poison the count (-1).
__global__ void __launch_bounds__(kGtPairThreads)
k_gt_pair_counts(const float4* __restrict__ pts, const int64_t* __restrict__ offsets, int n_scans, int64_t n_total,
                 const double* __restrict__ pose_ref, const double* __restrict__ pose_cur_inv,
                 const float* __restrict__ cur, int n_cur, const int32_t* __restrict__ pairs, GtParams P,
                 int32_t* __restrict__ counts, int* __restrict__ err) {
  extern __shared__ uint32_t img[];
  __shared__ int warp_sum[kGtPairThreads / 32];
  const int64_t k = blockIdx.x;
  int c = pairs[2 * k], r = pairs[2 * k + 1];
  const bool bad = c < 0 || c >= n_cur || r < 0 || r >= n_scans;
  if (bad) {
    c = c < 0 ? 0 : (c >= n_cur ? n_cur - 1 : c);
    r = r < 0 ? 0 : (r >= n_scans ? n_scans - 1 : r);
    if (threadIdx.x == 0) atomicCAS(err, 0, kErrBadIndex);
  }
  const int HW = P.H * P.W;
  for (int i = threadIdx.x; i < HW; i += kGtPairThreads) img[i] = 0xFFFFFFFFu;
  __syncthreads();
  const int64_t p0 = min(max(offsets[r], (int64_t)0), n_total), p1 = min(max(offsets[r + 1], p0), n_total);
  const double* pr = pose_ref + (size_t)r * 16;
  const double* pc = pose_cur_inv + (size_t)c * 16;
  for (int64_t g = p0 + threadIdx.x; g < p1; g += kGtPairThreads) {
    double depth;
    int pix;
    if (gt_point_pixel(__ldg(pts + g), pr, pc, P, depth, pix)) atomicMin(img + pix, __float_as_uint(__double2float_rn(depth)));
  }
  __syncthreads();
  const float* cimg = cur + (size_t)c * HW;
  int n = 0;
  for (int i = threadIdx.x; i < HW; i += kGtPairThreads) {
    const uint32_t key = img[i];
    const float rv = key == 0xFFFFFFFFu ? -1.0f : __uint_as_float(key);
    n += (rv > 0.0f) && (fabsf(__fsub_rn(rv, __ldg(cimg + i))) < 1.0f);
  }
  n = __reduce_add_sync(0xffffffffu, n);
  if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < kGtPairThreads / 32; ++w) t += warp_sum[w];
    counts[k] = bad ? -1 : t;
  }
}

__global__ void __launch_bounds__(256)
k_gt_keys_to_range(const unsigned long long* __restrict__ keys, int64_t n, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long k = keys[i];
  out[i] = (k == kGtEmpty) ? -1.0f : __double2float_rn(__longlong_as_double((long long)k));   // float32 image, utils.py:120,129
}

// counts[b] = #{ref_b > 0 and |ref_b - cur| < 1} (float32 arithmetic, com_overlap_yaw.py:44-45);
// row b == n_scans counts the current image's valid pixels (:31-32)
__global__ void __launch_bounds__(256)
k_gt_overlap_count(const float* __restrict__ ref, const float* __restrict__ cur, int n_scans, int HW,
                   int32_t* __restrict__ counts) {
  const int b = blockIdx.y;
  int c = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += gridDim.x * blockDim.x) {
    if (b == n_scans) {
      c += cur[i] > 0.0f;
    } else {
      const float r = ref[(size_t)b * HW + i];
      c += (r > 0.0f) && (fabsf(__fsub_rn(r, cur[i])) < 1.0f);
    }
  }
  c = __reduce_add_sync(0xffffffffu, c);
  __shared__ int s[8];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int k = 0; k < 8; ++k) t += s[k];
    if (t) atomicAdd(counts + b, t);
  }
}

static GtParams gt_params(const ovn_handle* h, float max_range) {
  GtParams P;
  P.H = h->cfg.proj_H; P.W = h->cfg.proj_W;
  P.pi = 3.14159265358979323846;
  const double fu = (double)h->cfg.fov_up_deg / 180.0 * P.pi, fd = (double)h->cfg.fov_down_deg / 180.0 * P.pi;   // utils.py:70-71
  P.abs_fov_down = fabs(fd);
  P.fov = fabs(fd) + fabs(fu);                                                                                     // :72
  P.max_range = max_range < 0 ? (double)h->cfg.max_range : (double)max_range;
  return P;
}

int gt_range_batch(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int n_scans, int64_t n_total,
                   const double* d_pose_ref, const double* d_pose_cur_inv, float max_range, float* d_range,
                   cudaStream_t s) {
  if (n_scans <= 0) return OVN_OK;
  if (n_scans > h->cfg.max_batch_scans)
    OVN_SET_ERR(h, OVN_ERR_CAPACITY, "n_scans=%d exceeds max_batch_scans=%d", n_scans, h->cfg.max_batch_scans);
  const GtParams P = gt_params(h, max_range);
  const int64_t n_pix = (int64_t)n_scans * P.H * P.W;
  OVN_CUDA(h, cudaMemsetAsync(h->d_keys, 0xFF, (size_t)n_pix * sizeof(unsigned long long), s));
  if (n_total > 0) {
    k_gt_scatter_f64<<<(unsigned)((n_total + 255) / 256), 256, 0, s>>>(reinterpret_cast<const float4*>(d_points), d_offsets,
                                                                      n_scans, n_total, d_pose_ref, d_pose_cur_inv, P,
                                                                      h->d_keys);
    OVN_LAUNCH_CHECK(h);
  }
  k_gt_keys_to_range<<<(unsigned)((n_pix + 255) / 256), 256, 0, s>>>(h->d_keys, n_pix, d_range);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

int gt_overlap_count(ovn_handle* h, const float* d_ref, const float* d_cur, int n_scans, int32_t* d_counts, cudaStream_t s) {
  if (n_scans < 0) OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "n_scans < 0");
  const int HW = h->cfg.proj_H * h->cfg.proj_W;
  OVN_CUDA(h, cudaMemsetAsync(d_counts, 0, (size_t)(n_scans + 1) * sizeof(int32_t), s));
  k_gt_overlap_count<<<dim3(8, (unsigned)(n_scans + 1)), 256, 0, s>>>(d_ref, d_cur, n_scans, HW, d_counts);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

int gt_pair_counts(ovn_handle* h, const float* d_points, const int64_t* d_offsets, int n_scans, int64_t n_total,
                   const double* d_pose_ref, const double* d_pose_cur_inv, const float* d_cur, int n_cur,
                   const int32_t* d_pairs, int64_t n_pairs, float max_range, int32_t* d_counts, cudaStream_t s) {
  if (n_pairs == 0) return OVN_OK;
  const GtParams P = gt_params(h, max_range);
  const size_t smem = (size_t)P.H * P.W * sizeof(uint32_t);
  int optin = 0;
  OVN_CUDA(h, cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
  if (smem + (kGtPairThreads / 32) * sizeof(int) > (size_t)optin)
    OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "ovn_gt_pair_counts: a %dx%d image (%zu B) does not fit the %d B of shared memory "
                "a block may use", P.H, P.W, smem, optin);
  OVN_CUDA(h, cudaFuncSetAttribute(k_gt_pair_counts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  constexpr int64_t kMaxGrid = 1 << 30;
  for (int64_t k0 = 0; k0 < n_pairs; k0 += kMaxGrid) {
    const int64_t np = n_pairs - k0 < kMaxGrid ? n_pairs - k0 : kMaxGrid;
    k_gt_pair_counts<<<(unsigned)np, kGtPairThreads, smem, s>>>(
        reinterpret_cast<const float4*>(d_points), d_offsets, n_scans, n_total, d_pose_ref, d_pose_cur_inv, d_cur, n_cur,
        d_pairs + 2 * k0, P, d_counts + k0, h->d_err);
    OVN_LAUNCH_CHECK(h);
  }
  return OVN_OK;
}

}  // namespace ovn
