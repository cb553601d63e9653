// simt_gemm.cuh -- the fp32 SIMT implicit-GEMM kernel and its operand functors, shared by the
// inference path (network_fp32.cu) and the training path (train.cu).
#pragma once
#include "common.cuh"

namespace ovn {

constexpr int BM = 64, BN = 64, BK = 16;

// ---- operand functors ------------------------------------------------------------------------
// NHWC valid conv:  A[m, k] = X[img, ho*sh + dh, wo*sw + dw, c],  m = (img, ho, wo), k = (dh, dw, c)
struct ConvOperand {
  const float* X;
  int H, W, C, kw, sh, sw, Ho, Wo;
  __device__ __forceinline__ int64_t row_base(int m, int /*z*/) const {
    const int wo = m % Wo;
    const int t = m / Wo;
    const int ho = t % Ho;
    const int img = t / Ho;
    return (((int64_t)img * H + (int64_t)ho * sh) * W + (int64_t)wo * sw) * C;
  }
  __device__ __forceinline__ int col_off(int k) const {
    const int rowlen = kw * C;
    const int dh = k / rowlen;
    return dh * W * C + (k - dh * rowlen);
  }
  __device__ __forceinline__ float load(int64_t rb, int co, int64_t, int) const { return __ldg(X + rb + co); }
  __device__ __forceinline__ int64_t row_base2(int, int) const { return 0; }
  __device__ __forceinline__ int col_off2(int) const { return 0; }
};

// c_conv1 on the delta image (generateNet.py:45-59,96-100):
//   A[m, k] = | L[i, c] - R[s*jb + dj, c] |,  m = (pair, i, jb),  k = (dj, c)
struct DeltaOperand {
  const float* bank;          // [n][Wf][128]
  const float* query;         // non-null: RIGHT is this single volume for every pair
  const int32_t* left;        // [n_pairs] bank rows
  const int32_t* right;       // [n_pairs] bank rows (ignored when query != null)
  int Wf, Cf, s, nb;          // 360, 128, 15, 24
  __device__ __forceinline__ int64_t row_base(int m, int) const {          // into LEFT
    const int jb = m % nb;
    const int t = m / nb;
    const int i = t % Wf;
    const int p = t / Wf;
    (void)jb;
    return ((int64_t)left[p] * Wf + i) * Cf;
  }
  __device__ __forceinline__ int64_t row_base2(int m, int) const {         // into RIGHT
    const int jb = m % nb;
    const int p = m / (nb * Wf);
    const int64_t vol = query ? 0 : (int64_t)right[p] * Wf * Cf;
    return vol + (int64_t)(s * jb) * Cf;
  }
  __device__ __forceinline__ int col_off(int k) const { return k % Cf; }
  __device__ __forceinline__ int col_off2(int k) const { return k; }
  __device__ __forceinline__ float load(int64_t rb, int co, int64_t rb2, int co2) const {
    const float* R = query ? query : bank;
    return fabsf(__ldg(bank + rb + co) - __ldg(R + rb2 + co2));
  }
};

// correlation Gram matrix: A = LEFT volume rows (z = pair); B comes from the RIGHT volume
struct GramOperand {
  const float* bank;
  const int32_t* left;
  int Wf, Cf;
  __device__ __forceinline__ int64_t row_base(int m, int z) const { return ((int64_t)left[z] * Wf + m) * Cf; }
  __device__ __forceinline__ int col_off(int k) const { return k; }
  __device__ __forceinline__ float load(int64_t rb, int co, int64_t, int) const { return __ldg(bank + rb + co); }
  __device__ __forceinline__ int64_t row_base2(int, int) const { return 0; }
  __device__ __forceinline__ int col_off2(int) const { return 0; }
};

struct BOperand {
  const float* B;             // weights [K][N] (b_nk = 0) or per-batch [N][K] (b_nk = 1)
  const float* query;         // b_nk: RIGHT volume = query for every z when non-null
  const int32_t* right;       // b_nk: bank row of the RIGHT volume of pair z
  int64_t vol_stride;
  int b_nk;
};

// C[m, n] = act(sum_k A[m,k] * B[k,n] + bias[n]);  C row-major [z][M][N]
template <class AOp>
__global__ void __launch_bounds__(256)
k_simt_gemm(AOp a, BOperand bop, const float* __restrict__ bias, float* __restrict__ C, int M, int N, int K,
            int relu) {
  __shared__ float As[BK][BM + 4];
  __shared__ float Bs[BK][BN + 4];
  __shared__ int64_t s_rb[BM];
  __shared__ int64_t s_rb2[BM];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN, z = blockIdx.z;
  if (tid < BM) {
    const int m = m0 + tid;
    s_rb[tid] = m < M ? a.row_base(m, z) : -1;
    s_rb2[tid] = m < M ? a.row_base2(m, z) : 0;
  }
  const float* Bz = bop.B;
  if (bop.b_nk) Bz = bop.query ? bop.query : bop.B + (int64_t)bop.right[z] * bop.vol_stride;
  __syncthreads();
  const int ty = tid / 16, tx = tid % 16;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += BK) {
    // A tile: 64 x 16 elements, consecutive threads -> consecutive k (contiguous in memory)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + i * 256;
      const int kk = e % BK, mm = e / BK;
      const int k = k0 + kk;
      float v = 0.f;
      if (k < K && s_rb[mm] >= 0) v = a.load(s_rb[mm], a.col_off(k), s_rb2[mm], a.col_off2(k));
      As[kk][mm] = v;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + i * 256;
      float v = 0.f;
      if (!bop.b_nk) {
        const int nn = e % BN, kk = e / BN;
        if (k0 + kk < K && n0 + nn < N) v = __ldg(Bz + (int64_t)(k0 + kk) * N + n0 + nn);
        Bs[kk][nn] = v;
      } else {
        const int kk = e % BK, nn = e / BK;
        if (k0 + kk < K && n0 + nn < N) v = __ldg(Bz + (int64_t)(n0 + nn) * K + k0 + kk);
        Bs[kk][nn] = v;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) av[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) bv[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j] + (bias ? __ldg(bias + n) : 0.f);
      if (relu) v = fmaxf(v, 0.f);
      C[((int64_t)z * M + m) * N + n] = v;
    }
  }
}

template <class AOp>
static int launch_gemm(ovn_handle* h, const AOp& a, const BOperand& b, const float* bias, float* C, int M,
                       int N, int K, int batch, int relu, cudaStream_t s) {
  dim3 grid((N + BN - 1) / BN, (M + BM - 1) / BM, batch);
  k_simt_gemm<AOp><<<grid, 256, 0, s>>>(a, b, bias, C, M, N, K, relu);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

}  // namespace ovn
