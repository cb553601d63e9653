// train.cu -- training of the overlap head on a frozen leg (the `360OutputkLegsFixed` leg of
// generateNet.py:222-324, fitted by training.py): forward pass with saved activations, the two
// losses, the gradients of c_conv1..3 and overlap_output, and the Keras Adagrad update.
//
// The forward pass and all gradients except dW1 are fp32 SIMT; dW1 is fp32 SIMT for precision fp32 and
// the tcgen05 kernel k_delta_wgrad_tc for precision f16_tc.  The SIMT parts reuse the operand functors of
// simt_gemm.cuh: a weight gradient
// dW[k][n] = sum_m A[m][k] * dY[m][n] is the same implicit GEMM with the reduction running over the
// rows m instead of k, so the |L - R| delta image and the im2col operands are again never
// materialised.  Every reduction over pairs or rows runs in a fixed order (per-split partial sums,
// then an ordered sum over the splits), so gradients are bit-identical from run to run.
//
// Semantics (cited from the reference):
//   pairs        LEFT = imgf1, RIGHT = imgf2            ImagePairOverlapOrientationSequence.py:100-112
//   yaw target   t[b] = y_ov, 0 elsewhere (:118-121), then t > min_overlap_for_angle (training.py:86-92)
//   overlap loss mean_p sigmoid((|yhat - y| + 0.25) * 24 - 12)                  training.py:71-83
//   yaw loss     tf.nn.weighted_cross_entropy_with_logits(t, corr, pos_weight = 360), mean over
//                the bins, then over the batch                                   training.py:86-92
//   total        5 * L_ov + 1 * L_or                                             training.py:255-257
//   Adagrad      a += g^2; p -= lr * g / (sqrt(a) + 1e-7)  (Keras 2.1.5)         training.py:253
// The correlation head has no weights and the leg is frozen, so L_or has no gradient: it is
// computed and reported only.
#include "simt_gemm.cuh"
#include "umma.cuh"
#include <math.h>

namespace ovn {

constexpr int kHeadLayers = 4;            // c_conv1, c_conv2, c_conv3, overlap_output
constexpr int kMaxSplits = 64;            // row splits of a weight-gradient GEMM
constexpr int kWgRows = 64;               // k_delta_wgrad_tc: rows (K) per shared-memory chunk
constexpr int kWgSplits = 20;             // k_delta_wgrad_tc: row splits (x conv1size CTAs)
constexpr int kErrWgradTimeout = 170;     // k_delta_wgrad_tc: MMA completion barrier timed out

struct TrainState {
  int cap = 0;                            // pairs (= max_batch_pairs)
  float *o1 = nullptr, *o2 = nullptr, *o3 = nullptr;   // saved activations [cap][...]
  float *dO3 = nullptr, *dO2 = nullptr, *dO1 = nullptr;
  float* corr = nullptr;                  // [cap][Wf] raw correlation scores (the yaw logits)
  int32_t* yaw = nullptr;                 // [cap] readout of the correlation head (unused)
  int32_t* idx = nullptr;                 // [3][cap] bounds-checked left, right, yaw bin
  float* pp = nullptr;                    // [4][cap] per pair: overlap, dL/dz, overlap loss, yaw loss
  uint32_t* scale = nullptr;              // [2] max |dO1| (float bits), power-of-two fp16 scale of dO1
  float* ws = nullptr;                    // [kMaxSplits][max K*N] partial weight gradients
  float* w3t = nullptr;                   // c_conv3 kernel as [dy][dx][cout][cin]
  float* w2t = nullptr;                   // c_conv2 kernel as [di][cout][cin]
  float* gk[kHeadLayers] = {};            // gradients (Keras layouts)
  float* gb[kHeadLayers] = {};
  float* ak[kHeadLayers] = {};            // Adagrad accumulators
  float* ab[kHeadLayers] = {};
  int64_t nk[kHeadLayers] = {}, nb[kHeadLayers] = {};
  int64_t ws_elems = 0;
  bool have_grad = false;
  bool acc_zero = true;                   // accumulators must be cleared before the next step
};

// ---- operand functors ----------------------------------------------------------------------------
// Data gradient of a stride-1 valid conv (c_conv3) as a GEMM over the zero-padded output gradient:
//   A[m, k] = dY[img, y - dy, x - dx, o],  m = (img, y, x) over the INPUT grid, k = (dy, dx, o);
// zero where (y - dy, x - dx) falls outside the Ho x Wo output.  B = the kernel as [dy][dx][o][c].
struct ConvTOperand {
  const float* dY;
  int H, W, Ho, Wo, kw, Co;
  __device__ __forceinline__ int64_t row_base(int m, int) const { return m; }
  __device__ __forceinline__ int col_off(int k) const { return k; }
  __device__ __forceinline__ float load(int64_t m64, int k, int64_t, int) const {
    const int m = (int)m64;
    const int x = m % W, t = m / W, y = t % H, img = t / H;
    const int o = k % Co, tap = k / Co, dx = tap % kw, dy = tap / kw;
    const int yo = y - dy, xo = x - dx;
    if (yo < 0 || yo >= Ho || xo < 0 || xo >= Wo) return 0.f;
    return __ldg(dY + (((int64_t)img * Ho + yo) * Wo + xo) * Co + o);
  }
  __device__ __forceinline__ int64_t row_base2(int, int) const { return 0; }
  __device__ __forceinline__ int col_off2(int) const { return 0; }
};

// ---- weight-gradient GEMM ------------------------------------------------------------------------
// ws[z][k][n] = sum over rows m of split z (in increasing order) of A[m, k] * B[m, n];  B row-major [M][N].
template <class AOp>
__global__ void __launch_bounds__(256)
k_wgrad(AOp a, const float* __restrict__ B, int M, int K, int N, int rows_per_split, float* __restrict__ ws) {
  __shared__ float As[BK][BM + 4];        // [m][k]
  __shared__ float Bs[BK][BN + 4];        // [m][n]
  __shared__ int64_t s_rb[BK], s_rb2[BK];
  const int tid = threadIdx.x;
  const int n0 = blockIdx.x * BN, k0 = blockIdx.y * BM, z = blockIdx.z;
  const int m_lo = z * rows_per_split;
  const int m_hi = min(M, m_lo + rows_per_split);
  const int ty = tid / 16, tx = tid % 16;
  float acc[4][4] = {};
  for (int m0 = m_lo; m0 < m_hi; m0 += BK) {
    if (tid < BK) {
      const int m = m0 + tid;
      s_rb[tid] = m < m_hi ? a.row_base(m, 0) : -1;
      s_rb2[tid] = m < m_hi ? a.row_base2(m, 0) : 0;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + i * 256;
      const int kk = e % BM, mm = e / BM;
      const int k = k0 + kk;
      float v = 0.f;
      if (k < K && s_rb[mm] >= 0) v = a.load(s_rb[mm], a.col_off(k), s_rb2[mm], a.col_off2(k));
      As[mm][kk] = v;
      const int n = n0 + kk;
      float w = 0.f;
      if (n < N && m0 + mm < m_hi) w = __ldg(B + (int64_t)(m0 + mm) * N + n);
      Bs[mm][kk] = w;
    }
    __syncthreads();
#pragma unroll
    for (int mm = 0; mm < BK; ++mm) {
      float av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) av[i] = As[mm][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) bv[j] = Bs[mm][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int k = k0 + ty * 4 + i;
    if (k >= K) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < N) ws[((int64_t)z * K + k) * N + n] = acc[i][j];
    }
  }
}

// out[i] = sum_{z < splits} ws[z][i], in increasing z
__global__ void k_split_reduce(const float* __restrict__ ws, int splits, int64_t kn, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kn) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += ws[(int64_t)z * kn + i];
  out[i] = s;
}

// The split depends on M only (never on the device), so two GPUs produce the same bits.
template <class AOp>
static int weight_grad(ovn_handle* h, TrainState* t, const AOp& a, const float* B, int M, int K, int N, float* out,
                       cudaStream_t s) {
  int splits = (M + 1023) / 1024;
  if (splits > kMaxSplits) splits = kMaxSplits;
  if (splits < 1) splits = 1;
  int rps = (M + splits - 1) / splits;
  rps = (rps + BK - 1) / BK * BK;
  splits = (M + rps - 1) / rps;
  if ((int64_t)splits * K * N > t->ws_elems)
    OVN_SET_ERR(h, OVN_ERR_CAPACITY, "training workspace too small for a %dx%d weight gradient", K, N);
  dim3 grid((N + BN - 1) / BN, (K + BM - 1) / BM, splits);
  k_wgrad<AOp><<<grid, 256, 0, s>>>(a, B, M, K, N, rps, t->ws);
  OVN_LAUNCH_CHECK(h);
  const int64_t kn = (int64_t)K * N;
  k_split_reduce<<<(unsigned)((kn + 255) / 256), 256, 0, s>>>(t->ws, splits, kn, out);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

// Bias gradient: db[n] = sum_m dY[m][n].  Split z sums rows [z*rps, (z+1)*rps) in increasing order
// into ws[z][n]; k_split_reduce then adds the splits in order (the split rule of weight_grad).
__global__ void k_colsum(const float* __restrict__ B, int M, int N, int rows_per_split, float* __restrict__ ws) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x, z = blockIdx.y;
  if (n >= N) return;
  const int m_hi = min(M, (z + 1) * rows_per_split);
  float acc = 0.f;
  for (int m = z * rows_per_split; m < m_hi; ++m) acc += B[(int64_t)m * N + n];
  ws[(int64_t)z * N + n] = acc;
}

static int bias_grad(ovn_handle* h, TrainState* t, const float* B, int M, int N, float* out, cudaStream_t s) {
  int splits = (M + 1023) / 1024;
  if (splits > kMaxSplits) splits = kMaxSplits;
  if (splits < 1) splits = 1;
  const int rps = (M + splits - 1) / splits;
  splits = (M + rps - 1) / rps;
  k_colsum<<<dim3((N + 63) / 64, splits), 64, 0, s>>>(B, M, N, rps, t->ws);
  OVN_LAUNCH_CHECK(h);
  k_split_reduce<<<(N + 255) / 256, 256, 0, s>>>(t->ws, splits, N, out);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

// ---- dW1 on tensor cores (precision f16_tc) ---------------------------------------------------------
// dW1[dj][c][o] = sum over rows m = (p, i, jb) of |L_p[i,c] - R_p[s*jb + dj, c]| * dO1[m][o]: for each dj
// a GEMM with M = 128 channels, N = 64, K = rows.  One CTA owns one dj and one contiguous range of
// 64-row chunks; its 128 x 64 fp32 accumulator lives in 64 TMEM columns.  Per chunk the four warps
// synthesise A = fp16 |L - R| (thread = channel; the difference is taken in fp32 from the bank and rounded
// once) and B = fp16(dO1 * scale) into K-major SWIZZLE_NONE tiles, then one thread issues
// four M128 N64 K16 MMAs (SS mode) and commits to an mbarrier that guards the tiles' reuse.
// Operand precision: |L - R| and dO1 both in fp16 (kind::f16 wants one type); dO1 is multiplied by a
// power-of-two scale so that its maximum lands in [2^13, 2^14) and no value underflows the fp16 range
// that matters; the scale is divided out exactly in the epilogue.  The partials of the splits are
// added in split order by k_split_reduce (bit-reproducible).
__global__ void k_dO1_absmax(const float* __restrict__ x, int64_t n, uint32_t* __restrict__ out) {
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(x[i]));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));     // non-negative floats order as integers
}

__global__ void k_dO1_scale(uint32_t* __restrict__ s) {
  const float m = __uint_as_float(s[0]);
  int e = 0;
  if (m > 0.f) frexpf(m, &e);                                          // m = f * 2^e, f in [0.5, 1)
  s[1] = __float_as_uint(m > 0.f ? ldexpf(1.f, 14 - e) : 1.f);
}

__global__ void __launch_bounds__(128)
k_delta_wgrad_tc(const float* __restrict__ bank, const int32_t* __restrict__ left, const int32_t* __restrict__ right,
                 const float* __restrict__ dO1, const uint32_t* __restrict__ scale, int Wf, int sz, int nb,
                 int n_chunks, int chunks_per_split, float* __restrict__ ws, int* __restrict__ err) {
  __shared__ __align__(1024) uint8_t sA[128 * kWgRows * 2];      // [c/8][k/8][c%8][k%8] fp16, 16 KB
  __shared__ __align__(1024) uint8_t sB[64 * kWgRows * 2];       // [o/8][k/8][o%8][k%8] fp16, 8 KB
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base;
  __shared__ int s_fail;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int dj = blockIdx.x, z = blockIdx.y;
  const int ch0 = z * chunks_per_split;
  const int ch1 = min(n_chunks, ch0 + chunks_per_split);
  if (warp == 0) umma::tmem_alloc(&tmem_base, 64);
  if (tid == 0) {
    umma::mbar_init(&bar, 1);
    umma::mbar_fence_init();
    s_fail = 0;
  }
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = tmem_base;
  const float sc = __uint_as_float(scale[1]);
  const uint32_t idesc = umma::make_idesc_f16(128, 64);
  const uint32_t a_addr = umma::smem_u32(sA), b_addr = umma::smem_u32(sB);
  const int64_t rows_per_pair = (int64_t)Wf * nb;
  uint32_t phase = 0;
  for (int ch = ch0; ch < ch1; ++ch) {
    const int64_t m0 = (int64_t)ch * kWgRows;
    {                                                             // A: thread = channel c
      const int c = tid;
      for (int kc = 0; kc < kWgRows / 8; ++kc) {
        uint32_t pk[4];
#pragma unroll
        for (int e = 0; e < 8; e += 2) {
          float v[2];
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const int64_t m = m0 + kc * 8 + e + q;
            const int p = (int)(m / rows_per_pair);
            const int r = (int)(m - (int64_t)p * rows_per_pair);
            const int i = r / nb, jb = r - i * nb;
            const float l = __ldg(bank + ((int64_t)left[p] * Wf + i) * kFeatC + c);
            const float rr = __ldg(bank + ((int64_t)right[p] * Wf + sz * jb + dj) * kFeatC + c);
            v[q] = fabsf(l - rr);
          }
          const __half2 hv = __floats2half2_rn(v[0], v[1]);
          pk[e / 2] = *reinterpret_cast<const uint32_t*>(&hv);
        }
        *reinterpret_cast<uint4*>(sA + (c >> 3) * 1024 + (c & 7) * 16 + kc * 128) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
    }
    {                                                             // B: thread = (o, half of the K chunks)
      const int o = tid & 63, kh = tid >> 6;
      for (int kc = kh * 4; kc < kh * 4 + 4; ++kc) {
        uint32_t pk[4];
#pragma unroll
        for (int e = 0; e < 8; e += 2) {
          const float v0 = __ldg(dO1 + (m0 + kc * 8 + e) * 64 + o) * sc;
          const float v1 = __ldg(dO1 + (m0 + kc * 8 + e + 1) * 64 + o) * sc;
          const __half2 hv = __floats2half2_rn(v0, v1);
          pk[e / 2] = *reinterpret_cast<const uint32_t*>(&hv);
        }
        *reinterpret_cast<uint4*>(sB + (o >> 3) * 1024 + (o & 7) * 16 + kc * 128) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
    }
    umma::fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
      umma::fence_after_sync();
#pragma unroll
      for (int ks = 0; ks < kWgRows / 16; ++ks) {                 // a K16 step = two 8-element K chunks
        const uint64_t ad = umma::make_desc_kmajor_noswizzle(a_addr + ks * 256, 128, 1024);
        const uint64_t bd = umma::make_desc_kmajor_noswizzle(b_addr + ks * 256, 128, 1024);
        umma::mma_ss(tmem, ad, bd, idesc, (ch > ch0 || ks > 0) ? 1u : 0u);
      }
      umma::commit(&bar);
    }
    if (!umma::mbar_wait(&bar, phase)) {
      atomicCAS(err, 0, kErrWgradTimeout);
      s_fail = 1;
    }
    phase ^= 1;
    umma::fence_after_sync();
    __syncthreads();
    if (s_fail) break;
  }
  // epilogue: warp w reads TMEM lanes (= channels) 32w..32w+31, 64 columns (= o)
  const int c = tid;
  float* dst = ws + (((int64_t)z * gridDim.x + dj) * 128 + c) * 64;
  const float inv = 1.f / sc;                                     // exact: sc is a power of two
  for (int hcol = 0; hcol < 2; ++hcol) {
    uint32_t r[32];
    umma::tmem_ld_x32(tmem + ((uint32_t)(warp * 32) << 16) + hcol * 32, r);
    umma::tmem_ld_wait();
    for (int j = 0; j < 32; ++j)
      dst[hcol * 32 + j] = s_fail ? __int_as_float(0x7fc00000) : (ch1 > ch0 ? __uint_as_float(r[j]) * inv : 0.f);
  }
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, 64);
}

static int delta_wgrad_tc(ovn_handle* h, TrainState* t, const float* d_bank, const int32_t* left,
                          const int32_t* right, int n, cudaStream_t s) {
  const int Wf = h->cfg.leg_output_width, sz = h->cfg.conv1size, nb = h->o1_w;
  const int64_t rows = (int64_t)n * Wf * nb;
  if (rows % kWgRows != 0)
    OVN_SET_ERR(h, OVN_ERR_BAD_CONFIG, "k_delta_wgrad_tc needs a multiple of %d c_conv1 output rows", kWgRows);
  const int n_chunks = (int)(rows / kWgRows);
  int splits = n_chunks < kWgSplits ? n_chunks : kWgSplits;
  const int cps = (n_chunks + splits - 1) / splits;
  splits = (n_chunks + cps - 1) / cps;
  const int64_t kn = (int64_t)sz * kFeatC * 64;
  if ((int64_t)splits * kn > t->ws_elems)
    OVN_SET_ERR(h, OVN_ERR_CAPACITY, "training workspace too small for the tensor-core dW1 partials");
  OVN_CUDA(h, cudaMemsetAsync(t->scale, 0, 2 * sizeof(uint32_t), s));
  k_dO1_absmax<<<h->sm_count * 4, 256, 0, s>>>(t->dO1, rows * 64, t->scale);
  OVN_LAUNCH_CHECK(h);
  k_dO1_scale<<<1, 1, 0, s>>>(t->scale);
  OVN_LAUNCH_CHECK(h);
  k_delta_wgrad_tc<<<dim3(sz, splits), 128, 0, s>>>(d_bank, left, right, t->dO1, t->scale, Wf, sz, nb, n_chunks, cps,
                                                   t->ws, h->d_err);
  OVN_LAUNCH_CHECK(h);
  k_split_reduce<<<(unsigned)((kn + 255) / 256), 256, 0, s>>>(t->ws, splits, kn, t->gk[0]);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

// ---- small kernels -------------------------------------------------------------------------------
// bounds-checked copies of the pair indices and yaw bins (clamped; the error flag poisons the losses)
__global__ void k_train_sanitize(const int32_t* __restrict__ left, const int32_t* __restrict__ right,
                                 const int32_t* __restrict__ bin, int n, int64_t bank_size, int n_bins,
                                 int32_t* __restrict__ out, int cap, int* __restrict__ err) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t l = left[i], r = right[i], b = bin[i];
  if (l < 0 || l >= bank_size || r < 0 || r >= bank_size) {
    atomicCAS(err, 0, kErrBadIndex);
    l = l < 0 ? 0 : (l >= bank_size ? bank_size - 1 : l);
    r = r < 0 ? 0 : (r >= bank_size ? bank_size - 1 : r);
  }
  if (b < 0 || b >= n_bins) {
    atomicCAS(err, 0, kErrBadYawBin);
    b = b < 0 ? 0 : n_bins - 1;
  }
  out[i] = (int32_t)l;
  out[cap + i] = (int32_t)r;
  out[2 * cap + i] = (int32_t)b;
}

__device__ __forceinline__ float sigmoidf(float x) { return 1.0f / (1.0f + expf(-x)); }

// One block per pair: Dense(1, sigmoid) (generateNet.py:112-114), the two per-pair loss terms and
// dL_total/dz = 5/n * dL_ov/dyhat * yhat (1 - yhat).  The dot product uses the summation order of
// k_dense_sigmoid, so the training forward reproduces the inference overlap bit for bit.
__global__ void __launch_bounds__(256)
k_dense_loss(const float* __restrict__ o3, const float* __restrict__ wd, const float* __restrict__ bd, int n_in,
             const float* __restrict__ corr, int n_bins, const float* __restrict__ y_ov,
             const int32_t* __restrict__ y_bin, float min_ov_angle, int n, float* __restrict__ pp, int cap) {
  __shared__ float red[256];
  const int p = blockIdx.x;
  const float* x = o3 + (int64_t)p * n_in;
  float acc = 0.f;
  for (int i = threadIdx.x; i < n_in; i += 256) acc = fmaf(x[i], __ldg(wd + i), acc);
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  const float z = red[0] + bd[0];
  __syncthreads();
  // yaw loss: TF's stable form (1 - t) x + (1 + (q - 1) t) (log1p(exp(-|x|)) + max(-x, 0)), q = n_bins
  const float q = (float)n_bins;
  const float yo = y_ov[p];
  const int b = y_bin[p];
  float le = 0.f;
  for (int k = threadIdx.x; k < n_bins; k += 256) {
    const float xk = corr[(int64_t)p * n_bins + k];
    const float tk = ((k == b ? yo : 0.f) > min_ov_angle) ? 1.f : 0.f;
    le += (1.f - tk) * xk + (1.f + (q - 1.f) * tk) * (log1pf(expf(-fabsf(xk))) + fmaxf(-xk, 0.f));
  }
  red[threadIdx.x] = le;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    // sigmoid'(x) = sigmoid(x) sigmoid(-x): 1 - sigmoid(x) would cancel where sigmoid(x) is near 1
    const float yh = sigmoidf(z);
    const float d = yh - yo;
    const float u = (fabsf(d) + 0.25f) * 24.f - 12.f;
    const float sl = sigmoidf(u);
    const float sgn = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);      // d|.|/d at 0 is 0, as in TF
    const float dyh = sl * sigmoidf(-u) * 24.f * sgn;
    pp[p] = yh;
    pp[cap + p] = 5.f / (float)n * dyh * yh * sigmoidf(-z);
    pp[2 * cap + p] = sl;
    pp[3 * cap + p] = red[0] / q;
  }
}

// losses = {5 L_ov + L_or, L_ov, L_or} (ordered means over the pairs) and the Dense bias gradient.
// A device error (bad index / yaw bin) poisons the losses with NaN.
__global__ void k_loss_finalize(const float* __restrict__ pp, int n, int cap, const int* __restrict__ err,
                                float* __restrict__ losses, float* __restrict__ gbd) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float sov = 0.f, sor = 0.f, sdz = 0.f;
  for (int p = 0; p < n; ++p) {
    sdz += pp[cap + p];
    sov += pp[2 * cap + p];
    sor += pp[3 * cap + p];
  }
  const float lov = sov / (float)n, lor = sor / (float)n;
  const bool bad = *err != 0;
  losses[0] = bad ? __int_as_float(0x7fc00000) : 5.f * lov + lor;
  losses[1] = bad ? __int_as_float(0x7fc00000) : lov;
  losses[2] = bad ? __int_as_float(0x7fc00000) : lor;
  *gbd = sdz;
}

// Dense backward: dwd[k] = sum_p dz_p o3[p][k] (ordered over p); dO3 = dz_p wd[k] [o3 > 0] (ReLU of c_conv3)
__global__ void k_dense_backward(const float* __restrict__ o3, const float* __restrict__ wd,
                                 const float* __restrict__ dz, int n, int n_in, float* __restrict__ gwd,
                                 float* __restrict__ dO3) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_in) return;
  const float w = __ldg(wd + k);
  float g = 0.f;
  for (int p = 0; p < n; ++p) {
    const float a = o3[(int64_t)p * n_in + k];
    const float d = dz[p];
    g = fmaf(d, a, g);
    dO3[(int64_t)p * n_in + k] = a > 0.f ? d * w : 0.f;
  }
  gwd[k] = g;
}

// x *= [act > 0]  (ReLU gradient of c_conv2)
__global__ void k_relu_mask(float* __restrict__ x, const float* __restrict__ act, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && !(act[i] > 0.f)) x[i] = 0.f;
}

// W3t[dy][dx][o][c] = W3[dy][dx][c][o]
__global__ void k_transpose_taps(const float* __restrict__ w, int taps, int ci, int co, float* __restrict__ wt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)taps * ci * co) return;
  const int c = (int)(i % ci);
  const int64_t r = i / ci;
  const int o = (int)(r % co), tap = (int)(r / co);
  wt[i] = w[((int64_t)tap * ci + c) * co + o];
}

// c_conv2 data gradient: a (s,1) conv with stride (s,1) has disjoint windows, so
//   dO1[p][s*ib + di][jb][c] = sum_o dO2[p][ib][jb][o] * W2t[di][o][c]     (W2t = W2 with c, o swapped)
// One block per (p, ib, jb); c_conv1 is linear, so this is also the gradient at c_conv1's output.
__global__ void __launch_bounds__(256)
k_conv2_dgrad(const float* __restrict__ dO2, const float* __restrict__ w2t, int s, int nb, int c1, int c2,
              float* __restrict__ dO1) {
  extern __shared__ float g[];
  const int r = blockIdx.x;                       // (p, ib, jb)
  const int jb = r % nb, t = r / nb, ib = t % nb, p = t / nb;
  for (int o = threadIdx.x; o < c2; o += blockDim.x) g[o] = dO2[(int64_t)r * c2 + o];
  __syncthreads();
  for (int e = threadIdx.x; e < s * c1; e += blockDim.x) {
    const int c = e % c1, di = e / c1;
    const float* wr = w2t + (int64_t)di * c2 * c1 + c;        // consecutive threads read consecutive c
    float acc = 0.f;
    for (int o = 0; o < c2; ++o) acc = fmaf(g[o], __ldg(wr + (int64_t)o * c1), acc);
    const int i = s * ib + di;
    dO1[((((int64_t)p * s * nb + i) * nb) + jb) * c1 + c] = acc;
  }
}

__global__ void k_adagrad(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ a, int64_t n,
                          float lr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i];
  const float ai = a[i] + gi * gi;
  a[i] = ai;
  w[i] = w[i] - lr * gi / (sqrtf(ai) + 1e-7f);
}

// ---- drivers -------------------------------------------------------------------------------------
void train_free(ovn_handle* h) {
  TrainState* t = h->tr;
  if (!t) return;
  void* bufs[] = {t->o1, t->o2, t->o3, t->dO3, t->dO2, t->dO1, t->corr, t->yaw, t->idx, t->pp, t->ws, t->w3t, t->w2t, t->scale};
  for (void* b : bufs) if (b) cudaFree(b);
  for (int l = 0; l < kHeadLayers; ++l) {
    void* lb[] = {t->gk[l], t->gb[l], t->ak[l], t->ab[l]};
    for (void* b : lb) if (b) cudaFree(b);
  }
  delete t;
  h->tr = nullptr;
}

// Allocated on the first backward call, so handles used only for inference allocate nothing.
static int train_alloc(ovn_handle* h) {
  if (h->tr) return OVN_OK;
  TrainState* t = new TrainState();
  h->tr = t;
  const int cap = h->cfg.max_batch_pairs, Wf = h->cfg.leg_output_width;
  t->cap = cap;
  const int64_t n1 = (int64_t)h->o1_h * h->o1_w * h->head[0].cout;
  const int64_t n2 = (int64_t)h->o2_h * h->o2_w * h->head[1].cout;
  const int64_t n3 = (int64_t)h->dense_in;
  OVN_CUDA(h, cudaMalloc(&t->o1, cap * n1 * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->dO1, cap * n1 * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->o2, cap * n2 * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->dO2, cap * n2 * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->o3, cap * n3 * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->dO3, cap * n3 * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->corr, (size_t)cap * Wf * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->yaw, (size_t)cap * sizeof(int32_t)));
  OVN_CUDA(h, cudaMalloc(&t->idx, (size_t)3 * cap * sizeof(int32_t)));
  OVN_CUDA(h, cudaMalloc(&t->pp, (size_t)4 * cap * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->scale, 2 * sizeof(uint32_t)));
  int64_t kn_max = 1;
  for (int l = 0; l < 3; ++l) {
    const ConvSpec& L = h->head[l];
    t->nk[l] = (int64_t)L.kh * L.kw * L.cin * L.cout;
    t->nb[l] = L.cout;
    if (t->nk[l] > kn_max) kn_max = t->nk[l];
  }
  t->nk[3] = h->dense_in;
  t->nb[3] = 1;
  t->ws_elems = kn_max * kMaxSplits;
  OVN_CUDA(h, cudaMalloc(&t->ws, t->ws_elems * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->w3t, t->nk[2] * sizeof(float)));
  OVN_CUDA(h, cudaMalloc(&t->w2t, t->nk[1] * sizeof(float)));
  for (int l = 0; l < kHeadLayers; ++l) {
    OVN_CUDA(h, cudaMalloc(&t->gk[l], t->nk[l] * sizeof(float)));
    OVN_CUDA(h, cudaMalloc(&t->gb[l], t->nb[l] * sizeof(float)));
    OVN_CUDA(h, cudaMalloc(&t->ak[l], t->nk[l] * sizeof(float)));
    OVN_CUDA(h, cudaMalloc(&t->ab[l], t->nb[l] * sizeof(float)));
  }
  t->acc_zero = true;
  return OVN_OK;
}

int train_heads_backward(ovn_handle* h, const float* d_bank, int64_t bank_size, const int32_t* d_left,
                         const int32_t* d_right, int n, const float* d_ov_gt, const int32_t* d_bin_gt,
                         float min_ov_angle, float* d_losses, cudaStream_t s) {
  int rc = train_alloc(h);
  if (rc != OVN_OK) { train_free(h); return rc; }
  TrainState* t = h->tr;
  const int Wf = h->cfg.leg_output_width, Cf = kFeatC, sz = h->cfg.conv1size, cap = t->cap;
  const int base = kMaxLegLayers;
  const ConvSpec &L1 = h->head[0], &L2 = h->head[1], &L3 = h->head[2];
  const int n3 = h->dense_in;
  const int32_t *left = t->idx, *right = t->idx + cap, *bin = t->idx + 2 * cap;
  k_train_sanitize<<<(n + 255) / 256, 256, 0, s>>>(d_left, d_right, d_bin_gt, n, bank_size, Wf, t->idx, cap, h->d_err);
  OVN_LAUNCH_CHECK(h);

  // ---- forward with saved activations (the launches of heads_forward_fp32)
  {
    DeltaOperand a{d_bank, nullptr, left, right, Wf, Cf, sz, h->o1_w};
    BOperand b{h->d_w[base + 0], nullptr, nullptr, 0, 0};
    rc = launch_gemm(h, a, b, h->d_b[base + 0], t->o1, n * h->o1_h * h->o1_w, L1.cout, sz * Cf, 1, 0, s);
    if (rc != OVN_OK) return rc;
  }
  {
    ConvOperand a{t->o1, L2.h_in, L2.w_in, L2.cin, L2.kw, L2.sh, L2.sw, L2.h_out, L2.w_out};
    BOperand b{h->d_w[base + 1], nullptr, nullptr, 0, 0};
    rc = launch_gemm(h, a, b, h->d_b[base + 1], t->o2, n * L2.h_out * L2.w_out, L2.cout, L2.kh * L2.kw * L2.cin, 1,
                     1, s);
    if (rc != OVN_OK) return rc;
  }
  {
    ConvOperand a{t->o2, L3.h_in, L3.w_in, L3.cin, L3.kw, L3.sh, L3.sw, L3.h_out, L3.w_out};
    BOperand b{h->d_w[base + 2], nullptr, nullptr, 0, 0};
    rc = launch_gemm(h, a, b, h->d_b[base + 2], t->o3, n * L3.h_out * L3.w_out, L3.cout, L3.kh * L3.kw * L3.cin, 1,
                     1, s);
    if (rc != OVN_OK) return rc;
  }
  rc = corr_forward_fp32(h, d_bank, nullptr, left, right, n, t->yaw, t->corr, s);
  if (rc != OVN_OK) return rc;

  // ---- losses, Dense
  k_dense_loss<<<n, 256, 0, s>>>(t->o3, h->d_w[base + 3], h->d_b[base + 3], n3, t->corr, Wf, d_ov_gt, bin,
                                 min_ov_angle, n, t->pp, cap);
  OVN_LAUNCH_CHECK(h);
  k_loss_finalize<<<1, 32, 0, s>>>(t->pp, n, cap, h->d_err, d_losses, t->gb[3]);
  OVN_LAUNCH_CHECK(h);
  k_dense_backward<<<(n3 + 255) / 256, 256, 0, s>>>(t->o3, h->d_w[base + 3], t->pp + cap, n, n3, t->gk[3], t->dO3);
  OVN_LAUNCH_CHECK(h);

  // ---- c_conv3: dW3 = im2col(o2)^T dO3, db3 = colsum(dO3), dX2 = full conv of dO3 with the flipped kernel
  const int M3 = n * L3.h_out * L3.w_out, K3 = L3.kh * L3.kw * L3.cin;
  {
    ConvOperand a{t->o2, L3.h_in, L3.w_in, L3.cin, L3.kw, L3.sh, L3.sw, L3.h_out, L3.w_out};
    rc = weight_grad(h, t, a, t->dO3, M3, K3, L3.cout, t->gk[2], s);
    if (rc == OVN_OK) rc = bias_grad(h, t, t->dO3, M3, L3.cout, t->gb[2], s);
    if (rc != OVN_OK) return rc;
  }
  {
    const int64_t nw = t->nk[2];
    k_transpose_taps<<<(unsigned)((nw + 255) / 256), 256, 0, s>>>(h->d_w[base + 2], L3.kh * L3.kw, L3.cin, L3.cout,
                                                                   t->w3t);
    OVN_LAUNCH_CHECK(h);
    ConvTOperand a{t->dO3, L3.h_in, L3.w_in, L3.h_out, L3.w_out, L3.kw, L3.cout};
    BOperand b{t->w3t, nullptr, nullptr, 0, 0};
    const int64_t n2 = (int64_t)n * L3.h_in * L3.w_in * L3.cin;
    rc = launch_gemm(h, a, b, nullptr, t->dO2, n * L3.h_in * L3.w_in, L3.cin, L3.kh * L3.kw * L3.cout, 1, 0, s);
    if (rc != OVN_OK) return rc;
    k_relu_mask<<<(unsigned)((n2 + 255) / 256), 256, 0, s>>>(t->dO2, t->o2, n2);
    OVN_LAUNCH_CHECK(h);
  }
  // ---- c_conv2: dW2 = im2col(o1)^T dO2, db2, dO1 (stride-s scatter)
  const int M2 = n * L2.h_out * L2.w_out, K2 = L2.kh * L2.kw * L2.cin;
  {
    ConvOperand a{t->o1, L2.h_in, L2.w_in, L2.cin, L2.kw, L2.sh, L2.sw, L2.h_out, L2.w_out};
    rc = weight_grad(h, t, a, t->dO2, M2, K2, L2.cout, t->gk[1], s);
    if (rc == OVN_OK) rc = bias_grad(h, t, t->dO2, M2, L2.cout, t->gb[1], s);
    if (rc != OVN_OK) return rc;
    k_transpose_taps<<<(unsigned)((t->nk[1] + 255) / 256), 256, 0, s>>>(h->d_w[base + 1], L2.kh * L2.kw, L2.cin,
                                                                          L2.cout, t->w2t);
    OVN_LAUNCH_CHECK(h);
    k_conv2_dgrad<<<M2, 256, L2.cout * sizeof(float), s>>>(t->dO2, t->w2t, L2.kh, L2.w_out, L2.cin, L2.cout,
                                                            t->dO1);
    OVN_LAUNCH_CHECK(h);
  }
  // ---- c_conv1: dW1 = |L - R|^T dO1 (the delta image, synthesised again), db1
  {
    const int M1 = n * h->o1_h * h->o1_w;
    DeltaOperand a{d_bank, nullptr, left, right, Wf, Cf, sz, h->o1_w};
    rc = (h->cfg.precision == OVN_PREC_F16_TC) ? delta_wgrad_tc(h, t, d_bank, left, right, n, s)
                                               : weight_grad(h, t, a, t->dO1, M1, sz * Cf, L1.cout, t->gk[0], s);
    if (rc == OVN_OK) rc = bias_grad(h, t, t->dO1, M1, L1.cout, t->gb[0], s);
    if (rc != OVN_OK) return rc;
  }
  t->have_grad = true;
  return OVN_OK;
}

int train_adagrad_step(ovn_handle* h, float lr, cudaStream_t s) {
  TrainState* t = h->tr;
  if (!t || !t->have_grad)
    OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "ovn_adagrad_step: no gradients yet (call ovn_heads_backward first)");
  if (t->acc_zero) {
    for (int l = 0; l < kHeadLayers; ++l) {
      OVN_CUDA(h, cudaMemsetAsync(t->ak[l], 0, t->nk[l] * sizeof(float), s));
      OVN_CUDA(h, cudaMemsetAsync(t->ab[l], 0, t->nb[l] * sizeof(float), s));
    }
    t->acc_zero = false;
  }
  for (int l = 0; l < kHeadLayers; ++l) {
    const int slot = kMaxLegLayers + l;
    k_adagrad<<<(unsigned)((t->nk[l] + 255) / 256), 256, 0, s>>>(h->d_w[slot], t->gk[l], t->ak[l], t->nk[l], lr);
    OVN_LAUNCH_CHECK(h);
    k_adagrad<<<(unsigned)((t->nb[l] + 255) / 256), 256, 0, s>>>(h->d_b[slot], t->gb[l], t->ab[l], t->nb[l], lr);
    OVN_LAUNCH_CHECK(h);
  }
  return OVN_OK;
}

void train_reset_optimizer(ovn_handle* h) {
  if (h->tr) h->tr->acc_zero = true;
}

int train_get_gradient(ovn_handle* h, int layer, float* h_kernel, float* h_bias) {
  TrainState* t = h->tr;
  if (!t || !t->have_grad)
    OVN_SET_ERR(h, OVN_ERR_INVALID_ARG, "ovn_get_gradient: no gradients yet (call ovn_heads_backward first)");
  OVN_CUDA(h, cudaEventSynchronize(h->ev_train));
  if (h_kernel) OVN_CUDA(h, cudaMemcpy(h_kernel, t->gk[layer], t->nk[layer] * sizeof(float), cudaMemcpyDeviceToHost));
  if (h_bias) OVN_CUDA(h, cudaMemcpy(h_bias, t->gb[layer], t->nb[layer] * sizeof(float), cudaMemcpyDeviceToHost));
  return OVN_OK;
}

}  // namespace ovn
