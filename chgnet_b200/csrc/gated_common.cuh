// Shared pieces of the gated-MLP kernels (FFMA: gated.cu, gated_2nd.cu; warp-specialised tcgen05: gated_ws.cu).
#pragma once
#include "common.cuh"

namespace chg {
namespace gated {

constexpr int HS = 132;    // smem stride of a 128-wide row
constexpr float LN_EPS = 1e-5f;
}  // namespace gated
// below this many rows the warp-specialised tcgen05 kernels hand the call to the FFMA kernels (launch-bound regime);
// default 4096; chg_set_option("ws_min_rows", n) changes it (abi.cu), e.g. to run the tcgen05 kernels on small test graphs
int ws_min_rows();
namespace gated {

enum Mode { ATOM = 0, BOND = 1, ANGLE = 2 };

struct FwdArgs {
  const float* p_a;     // ATOM: pcn [N][256]        BOND/ANGLE: pij [Eu][256]
  const float* p_b;     // ATOM: pe  [Eu][128]       BOND/ANGLE: px  [N][128]
  const float* p_c;     // BOND/ANGLE: pa [A][128] = angle features @ W1a (row = angle), else null
  const float* feat;    // ANGLE: angle features [A][64] (residual)
  const float* wgt;     // ATOM: wag [Eu][64]        BOND: wbg [Eu][64]
  const int32_t* idx0;  // row of p_a, first half    (center | bond i)
  const int32_t* idx1;  // row of p_a, second half   (nbr    | bond j)
  const int32_t* idx2;  // row of p_b                (d2u    | atom)
  int32_t n_rows;
  const float* w2t;    // [64][128]
  const float* b2;     // [128]
  const float* ln;     // [4][64] or null
  float* out;          // [rows][64]
  float* save_pre;     // [rows][128] or null
  float* save_p;       // [rows][128] or null
};

struct BwdArgs {
  const float* p_a;
  const float* p_b;
  const float* wgt;
  const int32_t* idx0;
  const int32_t* idx1;
  const int32_t* idx2;
  int32_t n_rows;
  const float* save_pre;  // BOND
  const float* save_p;
  const float* g_in;  // ATOM: g_agg [N][64]; BOND: g_agg [Eu][64]; ANGLE: g_ang_in [A][64] or null
  const float* w2;    // [128][64]
  const float* ln;
  float* g_pre;   // [rows][128]
  float* g_w0;    // ATOM: g_w; BOND: gw_i
  float* g_w1;    // BOND: gw_j
  // training only (parameter gradients); both null in inference
  float* g_p;     // [rows][128] dL/dp (second-layer output, before LayerNorm) or null
  double* g_ln;   // [4][64] accumulated dL/d(gamma1, beta1, gamma2, beta2) or null
};

// LayerNorm statistics of one 64-wide row spread over 16 lanes (4 values each)
__device__ __forceinline__ void ln_stats(const float (&v)[4], float (&xhat)[4], float& rstd) {
  const float mean = sum16(v[0] + v[1] + v[2] + v[3]) * (1.f / 64.f);
  float d[4], ss = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    d[j] = v[j] - mean;
    ss = fmaf(d[j], d[j], ss);
  }
  const float var = sum16(ss) * (1.f / 64.f);
  rstd = 1.f / sqrtf(var + LN_EPS);
#pragma unroll
  for (int j = 0; j < 4; ++j) xhat[j] = d[j] * rstd;
}

// pre-activation rows gathered from the per-atom / per-bond / per-angle first-layer products
template <int TMV>
__device__ __forceinline__ void gather_pre(float (&acc)[4][8], const float* __restrict__ p_a,
                                           const float* __restrict__ p_b, const float* __restrict__ p_c,
                                           const int* s_idx, int base, int n_rows, int r0, int c0) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = r0 + i;
    const float* s0 = p_a + (size_t)s_idx[row] * 256 + c0;
    const float* s1 = p_a + (size_t)s_idx[TMV + row] * 256 + 128 + c0;
    const float* s2 = p_b + (size_t)s_idx[2 * TMV + row] * 128 + c0;
    float4 vc = ldg4(s0) + ldg4(s1) + ldg4(s2);
    float4 vg = ldg4(s0 + 64) + ldg4(s1 + 64) + ldg4(s2 + 64);
    if (p_c != nullptr) {
      const float* s3 = p_c + (size_t)min(base + row, n_rows - 1) * 128 + c0;
      vc = vc + ldg4(s3);
      vg = vg + ldg4(s3 + 64);
    }
    acc[i][0] += vc.x; acc[i][1] += vc.y; acc[i][2] += vc.z; acc[i][3] += vc.w;
    acc[i][4] += vg.x; acc[i][5] += vg.y; acc[i][6] += vg.z; acc[i][7] += vg.w;
  }
}


// ---- shared by gated.cu (first order) and gated_2nd.cu (second order) ---------------------------
#ifdef __CUDACC__
constexpr int TM = 64;     // rows (edges / angles) per tile
constexpr int NTHR = 256;  // threads per CTA

__device__ __forceinline__ void copy_to_smem(float* dst, const float* src, int n_floats, int tid) {
  for (int i = tid * 4; i < n_floats; i += NTHR * 4) sts4(dst + i, ldg4(src + i));
}

// Block-diagonal pair of 64x64 products on a [64][HS] tile:
// acc[i][0..3] += sum_k T[r0+i][k]    * Bc[k][c0..]
// acc[i][4..7] += sum_k T[r0+i][64+k] * Bg[k][c0..]
// Bc row k at sBc + k*ldb, Bg row k at sBg + k*ldb.
__device__ __forceinline__ void gemm_blockdiag(float (&acc)[4][8], const float* __restrict__ sT,
                                               const float* __restrict__ sBc, const float* __restrict__ sBg,
                                               int ldb, int r0, int c0) {
#pragma unroll 2
  for (int k4 = 0; k4 < 16; ++k4) {
    float4 hc[4], hg[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      hc[i] = lds4(sT + (r0 + i) * HS + k4 * 4);
      hg[i] = lds4(sT + (r0 + i) * HS + 64 + k4 * 4);
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float4 wc = lds4(sBc + (k4 * 4 + kk) * ldb + c0);
      const float4 wg = lds4(sBg + (k4 * 4 + kk) * ldb + c0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float a = f4at(hc[i], kk);
        const float g = f4at(hg[i], kk);
        acc[i][0] = fmaf(a, wc.x, acc[i][0]);
        acc[i][1] = fmaf(a, wc.y, acc[i][1]);
        acc[i][2] = fmaf(a, wc.z, acc[i][2]);
        acc[i][3] = fmaf(a, wc.w, acc[i][3]);
        acc[i][4] = fmaf(g, wg.x, acc[i][4]);
        acc[i][5] = fmaf(g, wg.y, acc[i][5]);
        acc[i][6] = fmaf(g, wg.z, acc[i][6]);
        acc[i][7] = fmaf(g, wg.w, acc[i][7]);
      }
    }
  }
}


template <typename KernelT>
inline int resident_ctas(KernelT kernel, int smem_bytes) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, NTHR, smem_bytes) != cudaSuccess || per_sm < 1)
    per_sm = 1;
  return per_sm * sm_count();
}

#endif

// warp-specialised tcgen05 reverse kernels (gated_ws.cu): same outputs as gated_bwd_kernel<MODE, false>
int atom_conv_bwd_ws(const BwdArgs& a, cudaStream_t stream);
int bond_conv_bwd_ws(const BwdArgs& a, cudaStream_t stream);

// warp-specialised tcgen05 message + aggregation kernels (gated_ws.cu); `parts` = strip partials workspace
int atom_conv_fused_ws(const float* pcn, const float* pe, const float* wag, const int32_t* center, const int32_t* nbr,
                       const int32_t* d2u, const int32_t* ptr_c, int n_edges, int n_atoms, const float* w2t, const float* b2,
                       const float* ln, float* agg, float* save_p, float* parts, cudaStream_t stream);
int bond_conv_fused_ws(const float* pij, const float* px, const float* pa, const float* wbg, const int32_t* ang_atom,
                       const int32_t* ang_i, const int32_t* ang_j, const int32_t* ptr_i, int n_angles, int n_slots,
                       const float* w2t, const float* b2, const float* ln, float* agg, float* save_pre, float* save_p,
                       float* parts, cudaStream_t stream);

}  // namespace gated
}  // namespace chg
