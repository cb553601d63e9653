// network_fp32.cu -- fp32 SIMT verification path for the leg and the two heads.
//
// One tiled implicit-GEMM kernel (64x64x16 tiles, 4x4 register blocking) serves every layer; the
// A operand is produced on the fly by an "operand functor" (im2col of a valid-padded NHWC conv,
// or the |L - R| delta operand), so neither the im2col matrix nor the 66 MB delta tensor of the
// reference (generateNet.py:45-59) is ever materialised.  This path exists to (a) give a
// bit-for-bit reproducible fp32 result that the tensor-core path is validated against on the
// device and (b) serve precision=OVN_PREC_FP32.  The performance path is network_tc.cu.
//
// Replaces: generate360OutputkLegs (generateNet.py:161-217), DeltaLayer (:15-61),
// generateDeltaLayerConv1NetworkHead (:64-116), RangePadding2D.call (RangePadding2D.py:31-38),
// NormalizedCorrelation2D.call (NormalizedCorrelation2D.py:43-109), readout (infer.py:157-158).
#include "simt_gemm.cuh"

namespace ovn {

// ---- Dense(1, sigmoid) over the flattened (H,W,C) c_conv3 output (generateNet.py:112-114) -----
__global__ void __launch_bounds__(256)
k_dense_sigmoid(const float* __restrict__ o3, const float* __restrict__ wd, const float* __restrict__ bd,
                int n_in, float* __restrict__ overlap) {
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
  if (threadIdx.x == 0) {
    const float zz = red[0] + bd[0];
    overlap[p] = 1.0f / (1.0f + expf(-zz));
  }
}

// ---- circular diagonal sums of the Gram matrix + argmax readout -------------------------------
//   corr[k] = sum_j G[(k + j + W/2) mod W, j]      (RangePadding2D.py:34 + NormalizedCorrelation2D.py:96-109)
//   yaw     = W/2 - argmax_k corr[k], first maximum (infer.py:158)
__global__ void __launch_bounds__(384)
k_corr_readout(const float* __restrict__ G, int Wf, float* __restrict__ corr_out, int32_t* __restrict__ yaw) {
  extern __shared__ float s_corr[];
  const int p = blockIdx.x;
  const float* g = G + (int64_t)p * Wf * Wf;
  for (int k = threadIdx.x; k < Wf; k += blockDim.x) {
    float acc = 0.f;
    int i = k + Wf / 2;
    if (i >= Wf) i -= Wf;
    for (int j = 0; j < Wf; ++j) {
      acc += g[(int64_t)i * Wf + j];
      if (++i == Wf) i = 0;
    }
    s_corr[k] = acc;
    if (corr_out) corr_out[(int64_t)p * Wf + k] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int best = 0;
    float bv = s_corr[0];
    for (int k = 1; k < Wf; ++k)
      if (s_corr[k] > bv) { bv = s_corr[k]; best = k; }
    yaw[p] = Wf / 2 - best;
  }
}

// ---- drivers ----------------------------------------------------------------------------------
int leg_layer_fp32(ovn_handle* h, int l, const float* x, float* y, int n, cudaStream_t s) {
  const ConvSpec& L = h->leg[l];
  ConvOperand a{x, L.h_in, L.w_in, L.cin, L.kw, L.sh, L.sw, L.h_out, L.w_out};
  BOperand b{h->d_w[l], nullptr, nullptr, 0, 0};
  return launch_gemm(h, a, b, h->d_b[l], y, n * L.h_out * L.w_out, L.cout, L.kh * L.kw * L.cin, 1, L.relu, s);
}

int leg_forward_fp32(ovn_handle* h, const float* d_input, int n, float* d_fv, cudaStream_t s) {
  const float* x = d_input;
  prof_mark(h, PROF_LEG, s);
  for (int l = 0; l < h->n_leg; ++l) {
    const ConvSpec& L = h->leg[l];
    float* y = (l == h->n_leg - 1) ? d_fv : h->d_act[l & 1];
    ConvOperand a{x, L.h_in, L.w_in, L.cin, L.kw, L.sh, L.sw, L.h_out, L.w_out};
    BOperand b{h->d_w[l], nullptr, nullptr, 0, 0};
    int rc = launch_gemm(h, a, b, h->d_b[l], y, n * L.h_out * L.w_out, L.cout, L.kh * L.kw * L.cin, 1, L.relu, s);
    if (rc != OVN_OK) return rc;
    x = y;
  }
  prof_mark(h, PROF_LEG, s);
  return OVN_OK;
}

// correlation head for <= max_batch_pairs pairs: Gram matrix per pair (fp32), then circular
// diagonal sums + argmax.  LEFT = bank[left[p]], RIGHT = query or bank[right[p]].
int corr_forward_fp32(ovn_handle* h, const float* d_bank, const float* d_query, const int32_t* left,
                      const int32_t* right, int np, int32_t* d_yaw, float* d_corr, cudaStream_t s) {
  const int Wf = h->cfg.leg_output_width, Cf = kFeatC;
  GramOperand a{d_bank, left, Wf, Cf};
  BOperand b{d_bank, d_query, right, (int64_t)Wf * Cf, 1};
  int rc = launch_gemm(h, a, b, nullptr, h->d_G, Wf, Wf, Cf, np, 0, s);
  if (rc != OVN_OK) return rc;
  k_corr_readout<<<np, 384, Wf * sizeof(float), s>>>(h->d_G, Wf, d_corr, d_yaw);
  OVN_LAUNCH_CHECK(h);
  return OVN_OK;
}

int heads_forward_fp32(ovn_handle* h, const float* d_bank, const float* d_query, const int32_t* d_left,
                       const int32_t* d_right, int n, float* d_overlap, int32_t* d_yaw, float* d_corr,
                       cudaStream_t s) {
  const int Wf = h->cfg.leg_output_width, Cf = kFeatC, sz = h->cfg.conv1size;
  const int base = kMaxLegLayers;   // weight slots of c_conv1..3, overlap_output
  const int maxp = h->cfg.max_batch_pairs;
  for (int p0 = 0; p0 < n; p0 += maxp) {
    const int np = (n - p0 < maxp) ? n - p0 : maxp;
    const int32_t* left = d_left + p0;
    const int32_t* right = d_right ? d_right + p0 : nullptr;
    // c_conv1 (linear) on the implicit delta image
    {
      DeltaOperand a{d_bank, d_query, left, right, Wf, Cf, sz, h->o1_w};
      BOperand b{h->d_w[base + 0], nullptr, nullptr, 0, 0};
      prof_mark(h, PROF_DELTA, s);
      int rc = launch_gemm(h, a, b, h->d_b[base + 0], h->d_o1, np * h->o1_h * h->o1_w, h->head[0].cout,
                           sz * Cf, 1, 0, s);
      prof_mark(h, PROF_DELTA, s);
      if (rc != OVN_OK) return rc;
    }
    // c_conv2 (relu): (15,1) stride (15,1) over [p][360][24][64]
    {
      const ConvSpec& L = h->head[1];
      ConvOperand a{h->d_o1, L.h_in, L.w_in, L.cin, L.kw, L.sh, L.sw, L.h_out, L.w_out};
      BOperand b{h->d_w[base + 1], nullptr, nullptr, 0, 0};
      int rc = launch_gemm(h, a, b, h->d_b[base + 1], h->d_o2, np * L.h_out * L.w_out, L.cout,
                           L.kh * L.kw * L.cin, 1, 1, s);
      if (rc != OVN_OK) return rc;
    }
    // c_conv3 (relu) 3x3 -> reuse d_o1 as the o3 buffer (o1 is dead after c_conv2)
    float* d_o3 = h->d_o1;
    {
      const ConvSpec& L = h->head[2];
      ConvOperand a{h->d_o2, L.h_in, L.w_in, L.cin, L.kw, L.sh, L.sw, L.h_out, L.w_out};
      BOperand b{h->d_w[base + 2], nullptr, nullptr, 0, 0};
      int rc = launch_gemm(h, a, b, h->d_b[base + 2], d_o3, np * L.h_out * L.w_out, L.cout,
                           L.kh * L.kw * L.cin, 1, 1, s);
      if (rc != OVN_OK) return rc;
    }
    k_dense_sigmoid<<<np, 256, 0, s>>>(d_o3, h->d_w[base + 3], h->d_b[base + 3], h->dense_in, d_overlap + p0);
    OVN_LAUNCH_CHECK(h);
    {
      int rc = corr_forward_fp32(h, d_bank, d_query, left, right, np, d_yaw + p0,
                                 d_corr ? d_corr + (int64_t)p0 * Wf : nullptr, s);
      if (rc != OVN_OK) return rc;
    }
  }
  return OVN_OK;
}

}  // namespace ovn
