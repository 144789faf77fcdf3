// Gated-MLP message kernels: AtomConv / BondConv / AngleUpdate, forward and reverse.
//
// Reference semantics: chgnet/model/layers.py:113-121 (AtomConv message),
// 238-249 (BondConv message), 348-360 (AngleUpdate), GatedMLP in
// chgnet/model/functions.py:168-183.
//
// B200 design (DESIGN.md §3): the first Linear of every GatedMLP is split by input
// block and evaluated per ATOM / per BOND / per ANGLE by chg_linear (tensor cores); the
// kernels here gather the 128-wide pre-activation rows of each edge/angle (3 for AtomConv,
// 4 for BondConv / AngleUpdate), add them, run the two 64x64 second layers, and fuse
// LayerNorm / SiLU / sigmoid / bond-weight smoothing / residual in the epilogue.
//
// This file is the FFMA implementation (64-row tiles in shared memory, register-tiled
// GEMM; measured shared-memory-bandwidth bound, profiles/SUMMARY_r01.md).  The AtomConv /
// BondConv reverse and fused message + aggregation entry points hand inference calls of at least
// ws_min_rows() rows to the warp-specialised tcgen05 kernels of gated_ws.cu; everything
// else runs here.  One persistent CTA per resident slot; weights stay in shared memory.
//
// Thread map: 256 threads = 16 (ty) x 16 (tx); a thread owns rows ty*4..+3 and, in
// each 64-wide half (core | gate), columns tx*4..+3 — so core and gate of the same
// feature live in the same thread and LayerNorm reduces over the 16 tx lanes.
#include <cstdlib>

#include "gated_common.cuh"

namespace chg {
namespace {

using namespace gated;

template <int MODE>
struct FwdSmem {
  static constexpr bool HAS_W2 = MODE != ANGLE;
  static constexpr int W2_OFF = 0;
  static constexpr int TILE_OFF = W2_OFF + (HAS_W2 ? 64 * 128 : 0);
  static constexpr int TILE_FLOATS = HAS_W2 ? TM * HS : 0;
  static constexpr int B2_OFF = TILE_OFF + TILE_FLOATS;
  static constexpr int LN_OFF = B2_OFF + 128;
  static constexpr int IDX_OFF = LN_OFF + 256;
  static constexpr int TOTAL_BYTES = (IDX_OFF + 3 * TM) * 4;
};

template <int MODE>
__global__ void __launch_bounds__(NTHR, 2) gated_fwd_kernel(const FwdArgs a) {
  using L = FwdSmem<MODE>;
  extern __shared__ __align__(16) float smem[];
  float* s_w2t = smem + L::W2_OFF;
  float* s_tile = smem + L::TILE_OFF;  // H [64][HS]
  float* s_b2 = smem + L::B2_OFF;
  float* s_ln = smem + L::LN_OFF;
  int* s_idx = reinterpret_cast<int*>(smem + L::IDX_OFF);

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int r0 = ty * 4, c0 = tx * 4;
  const bool use_ln = a.ln != nullptr;

  if (L::HAS_W2) {
    copy_to_smem(s_w2t, a.w2t, 64 * 128, tid);
    if (tid < 128) s_b2[tid] = a.b2[tid];
  }
  if (use_ln) s_ln[tid] = a.ln[tid];

  const int n_tiles = (a.n_rows + TM - 1) / TM;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int base = tile * TM;
    __syncthreads();  // previous tile is done with s_tile / s_idx (also covers the weight loads)
    if (tid < TM) {
      const int r = min(base + tid, a.n_rows - 1);
      s_idx[tid] = a.idx0[r];
      s_idx[TM + tid] = a.idx1[r];
      s_idx[2 * TM + tid] = a.idx2[r];
    }
    __syncthreads();

    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    gather_pre<TM>(acc, a.p_a, a.p_b, a.p_c, s_idx, base, a.n_rows, r0, c0);

    if (L::HAS_W2) {
      if (a.save_pre != nullptr) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int g = base + r0 + i;
          if (g < a.n_rows) {
            stg4(a.save_pre + (size_t)g * 128 + c0, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
            stg4(a.save_pre + (size_t)g * 128 + 64 + c0, make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]));
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        sts4(s_tile + (r0 + i) * HS + c0,
             make_float4(silu_f(acc[i][0]), silu_f(acc[i][1]), silu_f(acc[i][2]), silu_f(acc[i][3])));
        sts4(s_tile + (r0 + i) * HS + 64 + c0,
             make_float4(silu_f(acc[i][4]), silu_f(acc[i][5]), silu_f(acc[i][6]), silu_f(acc[i][7])));
      }
      __syncthreads();
      const float4 bc = lds4(s_b2 + c0), bg = lds4(s_b2 + 64 + c0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[i][0] = bc.x; acc[i][1] = bc.y; acc[i][2] = bc.z; acc[i][3] = bc.w;
        acc[i][4] = bg.x; acc[i][5] = bg.y; acc[i][6] = bg.z; acc[i][7] = bg.w;
      }
      gemm_blockdiag(acc, s_tile, s_w2t, s_w2t + 64, 128, r0, c0);
    }

    // ---- epilogue: p -> LayerNorm -> silu * sigmoid -> smoothing / residual -> store
    float4 g1, b1, g2, b2v;
    if (use_ln) {
      g1 = lds4(s_ln + c0);
      b1 = lds4(s_ln + 64 + c0);
      g2 = lds4(s_ln + 128 + c0);
      b2v = lds4(s_ln + 192 + c0);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int row = r0 + i;
      const int g = base + row;
      const bool valid = g < a.n_rows;
      if (a.save_p != nullptr && valid) {
        stg4(a.save_p + (size_t)g * 128 + c0, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
        stg4(a.save_p + (size_t)g * 128 + 64 + c0, make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]));
      }
      float y1[4] = {acc[i][0], acc[i][1], acc[i][2], acc[i][3]};
      float y2[4] = {acc[i][4], acc[i][5], acc[i][6], acc[i][7]};
      if (use_ln) {
        float xh[4], rstd;
        ln_stats(y1, xh, rstd);
#pragma unroll
        for (int j = 0; j < 4; ++j) y1[j] = fmaf(xh[j], f4at(g1, j), f4at(b1, j));
        ln_stats(y2, xh, rstd);
#pragma unroll
        for (int j = 0; j < 4; ++j) y2[j] = fmaf(xh[j], f4at(g2, j), f4at(b2v, j));
      }
      float4 o;
#pragma unroll
      for (int j = 0; j < 4; ++j) f4at(o, j) = silu_f(y1[j]) * sigmoid_f(y2[j]);
      if (MODE == ATOM) {
        o = o * ldg4(a.wgt + (size_t)s_idx[2 * TM + row] * 64 + c0);
      } else if (MODE == BOND) {
        o = o * ldg4(a.wgt + (size_t)s_idx[row] * 64 + c0) * ldg4(a.wgt + (size_t)s_idx[TM + row] * 64 + c0);
      } else {
        o = o + ldg4(a.feat + (size_t)min(g, a.n_rows - 1) * 64 + c0);
      }
      if (valid) stg4(a.out + (size_t)g * 64 + c0, o);
    }
  }
}

template <int MODE>
struct BwdSmem {
  static constexpr bool HAS_W2 = MODE != ANGLE;
  static constexpr int W2_OFF = 0;
  static constexpr int TILE_OFF = W2_OFF + (HAS_W2 ? 128 * 64 : 0);
  static constexpr int LN_OFF = TILE_OFF + (HAS_W2 ? TM * HS : 0);
  static constexpr int IDX_OFF = LN_OFF + 256;
  static constexpr int TOTAL_BYTES = (IDX_OFF + 3 * TM) * 4;
};

// TRAIN adds what the parameter gradients need (reference trainer.py:409 loss.backward()): dL/dp rows
// for the second-layer weight gradients and the LayerNorm affine gradients, reduced per CTA.
template <int MODE, bool TRAIN>
__global__ void __launch_bounds__(NTHR, 2) gated_bwd_kernel(const BwdArgs a) {
  using L = BwdSmem<MODE>;
  extern __shared__ __align__(16) float smem[];
  float* s_w2 = smem + L::W2_OFF;   // [128][64]
  float* s_g = smem + L::TILE_OFF;  // [64][HS]
  float* s_ln = smem + L::LN_OFF;
  int* s_idx = reinterpret_cast<int*>(smem + L::IDX_OFF);

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int r0 = ty * 4, c0 = tx * 4;
  const bool use_ln = a.ln != nullptr;

  if (L::HAS_W2) copy_to_smem(s_w2, a.w2, 128 * 64, tid);
  if (use_ln) s_ln[tid] = a.ln[tid];
  float ln_acc[16];  // TRAIN: this thread's 4 columns x (gamma1, beta1, gamma2, beta2)
#pragma unroll
  for (int j = 0; j < 16; ++j) ln_acc[j] = 0.f;

  const int n_tiles = (a.n_rows + TM - 1) / TM;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int base = tile * TM;
    __syncthreads();
    if (MODE != ANGLE && tid < TM) {
      const int r = min(base + tid, a.n_rows - 1);
      s_idx[tid] = a.idx0[r];
      s_idx[TM + tid] = a.idx1[r];
      if (MODE == ATOM) s_idx[2 * TM + tid] = a.idx2[r];
    }
    __syncthreads();

    float4 g1, g2, b1, b2v;
    if (use_ln) {
      g1 = lds4(s_ln + c0);
      b1 = lds4(s_ln + 64 + c0);
      g2 = lds4(s_ln + 128 + c0);
      b2v = lds4(s_ln + 192 + c0);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int row = r0 + i;
      const int g = base + row;
      const bool valid = g < a.n_rows;
      const int r = min(g, a.n_rows - 1);
      const float4 pc4 = ldg4(a.save_p + (size_t)r * 128 + c0);
      const float4 pg4 = ldg4(a.save_p + (size_t)r * 128 + 64 + c0);
      float y1[4] = {pc4.x, pc4.y, pc4.z, pc4.w};
      float y2[4] = {pg4.x, pg4.y, pg4.z, pg4.w};
      float xh1[4], xh2[4], rstd1 = 1.f, rstd2 = 1.f;
      if (use_ln) {
        ln_stats(y1, xh1, rstd1);
        ln_stats(y2, xh2, rstd2);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          y1[j] = fmaf(xh1[j], f4at(g1, j), f4at(b1, j));
          y2[j] = fmaf(xh2[j], f4at(g2, j), f4at(b2v, j));
        }
      }
      float s1[4], core[4], gate[4];
      float4 o;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s1[j] = sigmoid_f(y1[j]);
        core[j] = y1[j] * s1[j];
        gate[j] = sigmoid_f(y2[j]);
        f4at(o, j) = core[j] * gate[j];
      }
      float4 go;
      if (MODE == ATOM) {
        const float4 gm = ldg4(a.g_in + (size_t)s_idx[row] * 64 + c0);
        const float4 w = ldg4(a.wgt + (size_t)s_idx[2 * TM + row] * 64 + c0);
        if (valid) stg4(a.g_w0 + (size_t)g * 64 + c0, gm * o);
        go = gm * w;
      } else if (MODE == BOND) {
        const float4 gm = ldg4(a.g_in + (size_t)s_idx[row] * 64 + c0);
        const float4 wi = ldg4(a.wgt + (size_t)s_idx[row] * 64 + c0);
        const float4 wj = ldg4(a.wgt + (size_t)s_idx[TM + row] * 64 + c0);
        const float4 gmo = gm * o;
        if (valid) {
          stg4(a.g_w0 + (size_t)g * 64 + c0, gmo * wj);
          stg4(a.g_w1 + (size_t)g * 64 + c0, gmo * wi);
        }
        go = gm * wi * wj;
      } else {
        go = a.g_in != nullptr ? ldg4(a.g_in + (size_t)r * 64 + c0) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      float gy1[4], gy2[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float gj = f4at(go, j);
        gy1[j] = gj * gate[j] * (s1[j] * fmaf(y1[j], 1.f - s1[j], 1.f));
        gy2[j] = gj * core[j] * gate[j] * (1.f - gate[j]);
      }
      if (use_ln) {
        if (TRAIN && valid) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            ln_acc[j] = fmaf(gy1[j], xh1[j], ln_acc[j]);
            ln_acc[4 + j] += gy1[j];
            ln_acc[8 + j] = fmaf(gy2[j], xh2[j], ln_acc[8 + j]);
            ln_acc[12 + j] += gy2[j];
          }
        }
        // g_p = rstd * (gx - mean(gx) - xhat * mean(gx * xhat)), gx = gy * gamma
        float gx[4], sa = 0.f, sb = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          gx[j] = gy1[j] * f4at(g1, j);
          sa += gx[j];
          sb = fmaf(gx[j], xh1[j], sb);
        }
        sa = sum16(sa) * (1.f / 64.f);
        sb = sum16(sb) * (1.f / 64.f);
#pragma unroll
        for (int j = 0; j < 4; ++j) gy1[j] = rstd1 * (gx[j] - sa - xh1[j] * sb);
        sa = 0.f, sb = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          gx[j] = gy2[j] * f4at(g2, j);
          sa += gx[j];
          sb = fmaf(gx[j], xh2[j], sb);
        }
        sa = sum16(sa) * (1.f / 64.f);
        sb = sum16(sb) * (1.f / 64.f);
#pragma unroll
        for (int j = 0; j < 4; ++j) gy2[j] = rstd2 * (gx[j] - sa - xh2[j] * sb);
      }
      const float4 gpc = make_float4(gy1[0], gy1[1], gy1[2], gy1[3]);
      const float4 gpg = make_float4(gy2[0], gy2[1], gy2[2], gy2[3]);
      if (TRAIN && L::HAS_W2 && valid && a.g_p != nullptr) {
        stg4(a.g_p + (size_t)g * 128 + c0, gpc);
        stg4(a.g_p + (size_t)g * 128 + 64 + c0, gpg);
      }
      if (L::HAS_W2) {
        sts4(s_g + row * HS + c0, gpc);
        sts4(s_g + row * HS + 64 + c0, gpg);
      } else if (valid) {  // no hidden layer: dE/dpre == dE/dp
        stg4(a.g_pre + (size_t)g * 128 + c0, gpc);
        stg4(a.g_pre + (size_t)g * 128 + 64 + c0, gpg);
      }
    }

    if (L::HAS_W2) {
      __syncthreads();
      float acc[4][8];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
      // g_h = g_p . W2 (core rows 0..63, gate rows 64..127 of the stacked [128][64] matrix)
      gemm_blockdiag(acc, s_g, s_w2, s_w2 + 64 * 64, 64, r0, c0);
      float pre[4][8];
      if (MODE == ATOM) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) pre[i][j] = 0.f;
        gather_pre<TM>(pre, a.p_a, a.p_b, nullptr, s_idx, base, a.n_rows, r0, c0);
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = min(base + r0 + i, a.n_rows - 1);
          const float4 vc = ldg4(a.save_pre + (size_t)r * 128 + c0);
          const float4 vg = ldg4(a.save_pre + (size_t)r * 128 + 64 + c0);
          pre[i][0] = vc.x; pre[i][1] = vc.y; pre[i][2] = vc.z; pre[i][3] = vc.w;
          pre[i][4] = vg.x; pre[i][5] = vg.y; pre[i][6] = vg.z; pre[i][7] = vg.w;
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int g = base + r0 + i;
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] *= dsilu_f(pre[i][j]);
        if (g < a.n_rows) {
          stg4(a.g_pre + (size_t)g * 128 + c0, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
          stg4(a.g_pre + (size_t)g * 128 + 64 + c0, make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]));
        }
      }
    }
  }
  if (TRAIN && use_ln && a.g_ln != nullptr) {
    // reduce the 16 row-groups (ty) of every column in shared memory, then one fp64 atomic per column
    __syncthreads();
    float* s_red = smem;  // [16 ty][256]; the weight / tile regions are free now
#pragma unroll
    for (int which = 0; which < 4; ++which)
#pragma unroll
      for (int j = 0; j < 4; ++j) s_red[ty * 256 + which * 64 + c0 + j] = ln_acc[which * 4 + j];
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int r = 0; r < 16; ++r) tot += s_red[r * 256 + tid];
    atomicAdd(a.g_ln + tid, (double)tot);
  }
}

template <int MODE>
int launch_fwd(const FwdArgs& a, cudaStream_t stream) {
  if (a.n_rows == 0) return CHG_OK;
  constexpr int smem = FwdSmem<MODE>::TOTAL_BYTES;
  static int slots = 0;
  if (slots == 0) {
    CHG_CUDA(cudaFuncSetAttribute(gated_fwd_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    slots = resident_ctas(gated_fwd_kernel<MODE>, smem);
  }
  const int n_tiles = (a.n_rows + TM - 1) / TM;
  gated_fwd_kernel<MODE><<<min(n_tiles, slots), NTHR, smem, stream>>>(a);
  CHG_LAUNCH_END();
}

template <int MODE, bool TRAIN>
int launch_bwd_t(const BwdArgs& a, cudaStream_t stream) {
  if (a.n_rows == 0) return CHG_OK;
  // the TRAIN epilogue reduces through 16 x 256 floats of shared memory
  constexpr int smem = TRAIN ? (BwdSmem<MODE>::TOTAL_BYTES > 16 * 256 * 4 ? BwdSmem<MODE>::TOTAL_BYTES : 16 * 256 * 4)
                             : BwdSmem<MODE>::TOTAL_BYTES;
  static int slots = 0;
  if (slots == 0) {
    CHG_CUDA(cudaFuncSetAttribute(gated_bwd_kernel<MODE, TRAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    slots = resident_ctas(gated_bwd_kernel<MODE, TRAIN>, smem);
  }
  const int n_tiles = (a.n_rows + TM - 1) / TM;
  gated_bwd_kernel<MODE, TRAIN><<<min(n_tiles, slots), NTHR, smem, stream>>>(a);
  CHG_LAUNCH_END();
}

template <int MODE>
int launch_bwd(const BwdArgs& a, cudaStream_t stream) {
  if (a.g_p != nullptr || a.g_ln != nullptr) return launch_bwd_t<MODE, true>(a, stream);
  return launch_bwd_t<MODE, false>(a, stream);
}

}  // namespace
}  // namespace chg

using namespace chg;
using namespace chg::gated;

extern "C" int chg_atom_conv_fwd(const float* pcn, const float* pe, const float* wag, const int32_t* center,
                                 const int32_t* nbr, const int32_t* d2u, int32_t n_edges, const float* w2t,
                                 const float* b2, const float* ln, float* msg, float* save_p, float* save_pre,
                                 void* stream) {
  CHG_CHECK_ARG(n_edges >= 0, "negative size");
  if (n_edges == 0) return CHG_OK;
  CHG_CHECK_ARG(pcn && pe && wag && center && nbr && d2u && w2t && b2 && msg, "null pointer");
  FwdArgs a{pcn, pe, nullptr, nullptr, wag, center, nbr, d2u, n_edges, w2t, b2, ln, msg, save_pre, save_p};
  return launch_fwd<ATOM>(a, as_stream(stream));
}

extern "C" int chg_atom_conv_bwd(const float* pcn, const float* pe, const float* wag, const int32_t* center,
                                 const int32_t* nbr, const int32_t* d2u, int32_t n_edges, const float* save_p,
                                 const float* g_agg, const float* w2, const float* ln, float* g_pre, float* g_w,
                                 float* g_p, double* g_ln, void* stream) {
  CHG_CHECK_ARG(n_edges >= 0, "negative size");
  if (n_edges == 0) return CHG_OK;
  CHG_CHECK_ARG(pcn && pe && wag && center && nbr && d2u && save_p && g_agg && w2 && g_pre && g_w, "null pointer");
  BwdArgs a{pcn, pe, wag, center, nbr, d2u, n_edges, nullptr, save_p, g_agg, w2, ln, g_pre, g_w, nullptr, g_p, g_ln};
  const bool train = g_p != nullptr || g_ln != nullptr;
  if (!train && n_edges >= ws_min_rows()) return atom_conv_bwd_ws(a, as_stream(stream));  // warp-specialised tcgen05
  return launch_bwd<ATOM>(a, as_stream(stream));
}

extern "C" int chg_bond_conv_fwd(const float* pij, const float* px, const float* pa, const float* wbg,
                                 const int32_t* ang_atom, const int32_t* ang_i, const int32_t* ang_j,
                                 int32_t n_angles, const float* w2t, const float* b2, const float* ln, float* upd,
                                 float* save_pre, float* save_p, void* stream) {
  CHG_CHECK_ARG(n_angles >= 0, "negative size");
  if (n_angles == 0) return CHG_OK;
  CHG_CHECK_ARG(pij && px && pa && wbg && ang_atom && ang_i && ang_j && w2t && b2 && upd, "null pointer");
  FwdArgs a{pij, px, pa, nullptr, wbg, ang_i, ang_j, ang_atom, n_angles, w2t, b2, ln, upd, save_pre, save_p};
  return launch_fwd<BOND>(a, as_stream(stream));
}

extern "C" int chg_bond_conv_bwd(const float* save_pre, const float* save_p, const float* wbg, const int32_t* ang_i,
                                 const int32_t* ang_j, int32_t n_angles, const float* g_agg, const float* w2,
                                 const float* ln, float* g_pre, float* gw_i, float* gw_j, float* g_p, double* g_ln,
                                 void* stream) {
  CHG_CHECK_ARG(n_angles >= 0, "negative size");
  if (n_angles == 0) return CHG_OK;
  CHG_CHECK_ARG(save_pre && save_p && wbg && ang_i && ang_j && g_agg && w2 && g_pre && gw_i && gw_j, "null pointer");
  BwdArgs a{nullptr, nullptr, wbg, ang_i, ang_j, nullptr, n_angles, save_pre, save_p, g_agg, w2, ln,
            g_pre, gw_i, gw_j, g_p, g_ln};
  const bool train = g_p != nullptr || g_ln != nullptr;
  if (!train && n_angles >= ws_min_rows()) return bond_conv_bwd_ws(a, as_stream(stream));  // warp-specialised tcgen05
  return launch_bwd<BOND>(a, as_stream(stream));
}

extern "C" int chg_angle_update_fwd(const float* pij, const float* px, const float* pa, const float* ang,
                                    const int32_t* ang_atom, const int32_t* ang_i, const int32_t* ang_j,
                                    int32_t n_angles, const float* ln, float* ang_new, float* save_p, void* stream) {
  CHG_CHECK_ARG(n_angles >= 0, "negative size");
  if (n_angles == 0) return CHG_OK;
  CHG_CHECK_ARG(pij && px && pa && ang && ang_atom && ang_i && ang_j && ang_new, "null pointer");
  FwdArgs a{pij, px, pa, ang, nullptr, ang_i, ang_j, ang_atom, n_angles, nullptr, nullptr, ln, ang_new,
            nullptr, save_p};
  return launch_fwd<ANGLE>(a, as_stream(stream));
}

extern "C" int chg_angle_update_bwd(const float* save_p, const float* g_ang_in, int32_t n_angles, const float* ln,
                                    float* g_pre, double* g_ln, void* stream) {
  CHG_CHECK_ARG(n_angles >= 0, "negative size");
  if (n_angles == 0) return CHG_OK;
  CHG_CHECK_ARG(save_p && g_pre, "null pointer");
  BwdArgs a{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, n_angles, nullptr, save_p, g_ang_in,
            nullptr, ln, g_pre, nullptr, nullptr, nullptr, g_ln};
  return launch_bwd<ANGLE>(a, as_stream(stream));
}
