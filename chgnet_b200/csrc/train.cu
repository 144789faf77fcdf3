// Training-only kernels: parameter gradients, loss terms, Adam.
//
// Reference: chgnet/trainer/trainer.py:398-411 (prediction -> CombinedLoss -> loss.backward()
// -> optimizer.step()), CombinedLoss 779-869.  The reverse pass over ACTIVATIONS is the one the
// force / stress path already runs (gated.cu, segsum.cu, linear*.cu); what training adds is
//   * chg_wgrad    : dL/dW^T = act(X)^T . G for every dense layer (reduction over rows),
//   * chg_colsum   : bias / LayerNorm-affine / last-layer gradients (weighted column sums),
//   * chg_readout_bwd, chg_magmom_bwd : the two heads with a loss seed,
//   * chg_loss_terms, chg_adam_step.
// All reductions over rows go through per-CTA partials and a second pass in fp64, so the
// gradients are deterministic (no floating-point atomics on the weight gradients).
#include <algorithm>

#include "common.cuh"

namespace chg {
namespace {

// ---- wgrad: out[64][n] = act(X[xr])^T . G[gr] -----------------------------------------------
constexpr int WG_ROWS = 32;  // rows staged per step
constexpr int WG_MAX_CHUNKS = 1024;

// ACT: 0 x, 1 silu(x), 2 silu'(x) * x2 (tangent of the hidden activations; x2 shares x's rows / stride)
template <int ACT>
__global__ void __launch_bounds__(256)
wgrad_kernel(const float* __restrict__ x, const float* __restrict__ x2, int ldx, const int32_t* __restrict__ x_rows,
             const float* __restrict__ g,
             int ldg, const int32_t* __restrict__ g_rows, int m, int n, float* __restrict__ partial,
             float* __restrict__ cs_partial) {
  __shared__ __align__(16) float s_x[WG_ROWS][64];
  __shared__ __align__(16) float s_g[WG_ROWS][64];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int k0 = ty * 4, n0 = tx * 4;
  const int col_base = blockIdx.y * 64;
  const int n_chunks = gridDim.x;
  // contiguous, balanced row range of this chunk (multiples of WG_ROWS except the last)
  const int steps_total = (m + WG_ROWS - 1) / WG_ROWS;
  const int s_beg = (int)((long long)steps_total * blockIdx.x / n_chunks);
  const int s_end = (int)((long long)steps_total * (blockIdx.x + 1) / n_chunks);
  float acc[4][4], cs[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  // register-staged software pipeline: the global loads of step s+1 are in flight while step s
  // is multiplied out of shared memory
  float4 xr[2], gr[2], x2r[2];
  auto fetch = [&](int step) {
    const int base = step * WG_ROWS;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int f4 = tid + h * 256;  // 512 float4 per tile
      const int r = f4 >> 4, c = (f4 & 15) * 4;
      const int row = base + r;
      xr[h] = make_float4(0.f, 0.f, 0.f, 0.f);
      gr[h] = xr[h];
      x2r[h] = xr[h];
      if (row < m) {
        const int xi = x_rows != nullptr ? x_rows[row] : row;
        const int gi = g_rows != nullptr ? g_rows[row] : row;
        xr[h] = ldg4(x + (size_t)xi * ldx + c);
        if (ACT == 2) x2r[h] = ldg4(x2 + (size_t)xi * ldx + c);
        gr[h] = ldg4(g + (size_t)gi * ldg + col_base + c);
      }
    }
  };
  if (s_beg < s_end) fetch(s_beg);
  for (int step = s_beg; step < s_end; ++step) {
    __syncthreads();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int f4 = tid + h * 256;
      const int r = f4 >> 4, c = (f4 & 15) * 4;
      float4 xv = xr[h];
      if (ACT == 1) xv = make_float4(silu_f(xv.x), silu_f(xv.y), silu_f(xv.z), silu_f(xv.w));
      if (ACT == 2)
        xv = make_float4(dsilu_f(xv.x) * x2r[h].x, dsilu_f(xv.y) * x2r[h].y, dsilu_f(xv.z) * x2r[h].z,
                         dsilu_f(xv.w) * x2r[h].w);
      sts4(&s_x[r][c], xv);
      sts4(&s_g[r][c], gr[h]);
    }
    __syncthreads();
    if (step + 1 < s_end) fetch(step + 1);
#pragma unroll 8
    for (int r = 0; r < WG_ROWS; ++r) {
      const float4 xv = lds4(&s_x[r][k0]);
      const float4 gv = lds4(&s_g[r][n0]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float a = f4at(xv, i);
        acc[i][0] = fmaf(a, gv.x, acc[i][0]);
        acc[i][1] = fmaf(a, gv.y, acc[i][1]);
        acc[i][2] = fmaf(a, gv.z, acc[i][2]);
        acc[i][3] = fmaf(a, gv.w, acc[i][3]);
      }
      if (ty == 0) {
        cs[0] += gv.x; cs[1] += gv.y; cs[2] += gv.z; cs[3] += gv.w;
      }
    }
  }
  float* dst = partial + (size_t)blockIdx.x * 64 * n;
#pragma unroll
  for (int i = 0; i < 4; ++i)
    stg4(dst + (size_t)(k0 + i) * n + col_base + n0, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
  if (cs_partial != nullptr && ty == 0)
    stg4(cs_partial + (size_t)blockIdx.x * n + col_base + n0, make_float4(cs[0], cs[1], cs[2], cs[3]));
}

// second pass: sum the per-chunk partials in fp64 (fixed order -> deterministic).
// A block owns 32 consecutive outputs; its 8 chunk-lanes each sum every 8th chunk with independent
// loads in flight, then combine through shared memory.
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ partial, const float* __restrict__ cs_partial, int n_chunks, int n,
                    float* __restrict__ out, int ldo, float* __restrict__ colsum) {
  __shared__ double s_red[8][32];
  const int o = threadIdx.x & 31, cl = threadIdx.x >> 5;
  const int n_w = 64 * n;
  const int idx = blockIdx.x * 32 + o;  // [0, n_w) weights, [n_w, n_w + n) column sums
  const bool is_w = idx < n_w, is_c = !is_w && colsum != nullptr && idx < n_w + n;
  const float* src = is_w ? partial + idx : (is_c ? cs_partial + (idx - n_w) : nullptr);
  const size_t stride = is_w ? (size_t)n_w : (size_t)n;
  double s = 0.0;
  if (src != nullptr) {
    int c = cl;
    for (; c + 24 < n_chunks; c += 32) {
      const float v0 = src[(size_t)c * stride], v1 = src[(size_t)(c + 8) * stride];
      const float v2 = src[(size_t)(c + 16) * stride], v3 = src[(size_t)(c + 24) * stride];
      s += ((double)v0 + (double)v1) + ((double)v2 + (double)v3);
    }
    for (; c < n_chunks; c += 8) s += (double)src[(size_t)c * stride];
  }
  s_red[cl][o] = s;
  __syncthreads();
  if (cl == 0 && src != nullptr) {
#pragma unroll
    for (int q = 1; q < 8; ++q) s += s_red[q][o];
    if (is_w) out[(size_t)(idx / n) * ldo + (idx % n)] = (float)s;
    else colsum[idx - n_w] = (float)s;
  }
}

// ---- weighted column sum: out[c] += sum_r a[r][c] * b[r][c] * rowscale[r]  (fp64 accumulator) ---------
__global__ void __launch_bounds__(256)
colsum_kernel(const float* __restrict__ a, int lda, const float* __restrict__ bmul, int ldb,
              const float* __restrict__ rowscale, int m, int n, double* __restrict__ out) {
  __shared__ double s_red[256];
  const int tid = threadIdx.x;
  const int c = tid % n, rl = tid / n, lanes = 256 / n;
  const int rows_per_cta = (m + gridDim.x - 1) / gridDim.x;
  const int r_beg = blockIdx.x * rows_per_cta, r_end = min(r_beg + rows_per_cta, m);
  auto term = [&](int r) {
    float v = a[(size_t)r * lda + c];
    if (bmul != nullptr) v *= bmul[(size_t)r * ldb + c];
    if (rowscale != nullptr) v *= rowscale[r];
    return v;
  };
  double s = 0.0;
  int r = r_beg + rl;
  for (; r + 3 * lanes < r_end; r += 4 * lanes) {  // four independent loads in flight
    const float v0 = term(r), v1 = term(r + lanes), v2 = term(r + 2 * lanes), v3 = term(r + 3 * lanes);
    s += ((double)v0 + (double)v1) + ((double)v2 + (double)v3);
  }
  for (; r < r_end; r += lanes) s += (double)term(r);
  s_red[tid] = s;
  __syncthreads();
  if (rl == 0) {
    for (int q = 1; q < lanes; ++q) s += s_red[q * n + c];
    atomicAdd(out + c, s);
  }
}

// ---- readout reverse with a per-atom seed (one warp per atom; lane owns features lane, lane+32) ------
constexpr int MAX_HIDDEN = 4;

__global__ void __launch_bounds__(256)
readout_bwd_kernel(const float* __restrict__ x, int n_atoms, const float* __restrict__ ln,
                   const float* __restrict__ mlp_wt, const float* __restrict__ mlp_w,
                   const float* __restrict__ mlp_b, int n_hidden, const float* __restrict__ w_last,
                   const float* __restrict__ seed, float* __restrict__ g_x, float* __restrict__ h_all,
                   float* __restrict__ gz_all, float* __restrict__ g_h0, float* __restrict__ xhat) {
  extern __shared__ __align__(16) float smem[];
  float* s_wt = smem;                   // [L][64][64] k-major
  float* s_w = s_wt + n_hidden * 4096;  // [L][64][64] PyTorch layout
  for (int i = threadIdx.x; i < n_hidden * 4096; i += blockDim.x) {
    s_wt[i] = mlp_wt[i];
    s_w[i] = mlp_w[i];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  const float wl0 = w_last[lane], wl1 = w_last[lane + 32];
  const size_t plane = (size_t)n_atoms * 64;
  for (int atom = warp; atom < n_atoms; atom += n_warps) {
    const size_t off = (size_t)atom * 64;
    float h0 = x[off + lane], h1 = x[off + lane + 32];
    float xh0 = 0.f, xh1 = 0.f, rstd = 1.f;
    if (ln != nullptr) {
      const float mean = sum32(h0 + h1) * (1.f / 64.f);
      const float d0 = h0 - mean, d1 = h1 - mean;
      const float var = sum32(fmaf(d0, d0, d1 * d1)) * (1.f / 64.f);
      rstd = 1.f / sqrtf(var + 1e-5f);
      xh0 = d0 * rstd;
      xh1 = d1 * rstd;
      h0 = fmaf(xh0, ln[lane], ln[64 + lane]);
      h1 = fmaf(xh1, ln[lane + 32], ln[64 + lane + 32]);
      xhat[off + lane] = xh0;
      xhat[off + lane + 32] = xh1;
    }
    float za[MAX_HIDDEN], zb[MAX_HIDDEN];
#pragma unroll
    for (int l = 0; l < MAX_HIDDEN; ++l) {
      if (l < n_hidden) {
        h_all[l * plane + off + lane] = h0;
        h_all[l * plane + off + lane + 32] = h1;
        const float* wt = s_wt + l * 4096;
        float a = mlp_b[l * 64 + lane], b = mlp_b[l * 64 + lane + 32];
        for (int k = 0; k < 32; ++k) {
          const float v0 = __shfl_sync(0xffffffffu, h0, k), v1 = __shfl_sync(0xffffffffu, h1, k);
          a = fmaf(v0, wt[k * 64 + lane], a);
          b = fmaf(v0, wt[k * 64 + lane + 32], b);
          a = fmaf(v1, wt[(k + 32) * 64 + lane], a);
          b = fmaf(v1, wt[(k + 32) * 64 + lane + 32], b);
        }
        za[l] = a;
        zb[l] = b;
        h0 = silu_f(a);
        h1 = silu_f(b);
      }
    }
    h_all[n_hidden * plane + off + lane] = h0;
    h_all[n_hidden * plane + off + lane + 32] = h1;
    const float sd = seed[atom];
    float g0 = wl0 * sd, g1 = wl1 * sd;
#pragma unroll
    for (int l = MAX_HIDDEN - 1; l >= 0; --l) {
      if (l < n_hidden) {
        const float* w = s_w + l * 4096;
        const float gz0 = g0 * dsilu_f(za[l]), gz1 = g1 * dsilu_f(zb[l]);
        gz_all[l * plane + off + lane] = gz0;
        gz_all[l * plane + off + lane + 32] = gz1;
        float a = 0.f, b = 0.f;
        for (int n = 0; n < 32; ++n) {
          const float v0 = __shfl_sync(0xffffffffu, gz0, n), v1 = __shfl_sync(0xffffffffu, gz1, n);
          a = fmaf(v0, w[n * 64 + lane], a);
          b = fmaf(v0, w[n * 64 + lane + 32], b);
          a = fmaf(v1, w[(n + 32) * 64 + lane], a);
          b = fmaf(v1, w[(n + 32) * 64 + lane + 32], b);
        }
        g0 = a;
        g1 = b;
      }
    }
    g_h0[off + lane] = g0;
    g_h0[off + lane + 32] = g1;
    if (ln != nullptr) {
      const float gx0 = g0 * ln[lane], gx1 = g1 * ln[lane + 32];
      const float m1 = sum32(gx0 + gx1) * (1.f / 64.f);
      const float m2 = sum32(fmaf(gx0, xh0, gx1 * xh1)) * (1.f / 64.f);
      g0 = rstd * (gx0 - m1 - xh0 * m2);
      g1 = rstd * (gx1 - m1 - xh1 * m2);
    }
    g_x[off + lane] = g0;
    g_x[off + lane + 32] = g1;
  }
}

// ---- readout, second order: reverse of (readout, its tangent along xd) ---------------------------------
// scalar per atom:  seed * site_e + <d site_e / dx, xd>.  gz_all = adjoint of the TANGENT pre-activations
// (= dE/dz with seed 1), zbar_all = adjoint of the PRIMAL pre-activations.  (oracle/kernel_specs.py
// readout_bwd2 states the same maths.)
__device__ __forceinline__ float d2silu_r(float x) {
  const float s = sigmoid_f(x);
  return s * (1.f - s) * fmaf(x, 1.f - 2.f * s, 2.f);
}

__global__ void __launch_bounds__(256)
readout_bwd2_kernel(const float* __restrict__ x, const float* __restrict__ xd, int n_atoms,
                    const float* __restrict__ ln, const float* __restrict__ mlp_wt, const float* __restrict__ mlp_w,
                    const float* __restrict__ mlp_b, int n_hidden, const float* __restrict__ w_last,
                    const float* __restrict__ seed, float* __restrict__ bar_x, float* __restrict__ h_all,
                    float* __restrict__ hd_all, float* __restrict__ gz_all, float* __restrict__ zbar_all,
                    float* __restrict__ g_h0, float* __restrict__ hbar0, float* __restrict__ xhat,
                    float* __restrict__ xhatd) {
  extern __shared__ __align__(16) float smem[];
  float* s_wt = smem;
  float* s_w = s_wt + n_hidden * 4096;
  for (int i = threadIdx.x; i < n_hidden * 4096; i += blockDim.x) {
    s_wt[i] = mlp_wt[i];
    s_w[i] = mlp_w[i];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  const float wl0 = w_last[lane], wl1 = w_last[lane + 32];
  const size_t plane = (size_t)n_atoms * 64;
  for (int atom = warp; atom < n_atoms; atom += n_warps) {
    const size_t off = (size_t)atom * 64;
    float h0 = x[off + lane], h1 = x[off + lane + 32];
    float d0 = xd[off + lane], d1 = xd[off + lane + 32];
    const float xd0 = d0, xd1 = d1;
    float xh0 = 0.f, xh1 = 0.f, xt0 = 0.f, xt1 = 0.f, rstd = 1.f;
    if (ln != nullptr) {
      const float mean = sum32(h0 + h1) * (1.f / 64.f);
      const float c0 = h0 - mean, c1 = h1 - mean;
      const float var = sum32(fmaf(c0, c0, c1 * c1)) * (1.f / 64.f);
      rstd = 1.f / sqrtf(var + 1e-5f);
      xh0 = c0 * rstd;
      xh1 = c1 * rstd;
      const float m1 = sum32(d0 + d1) * (1.f / 64.f);
      const float m2 = sum32(fmaf(xh0, d0, xh1 * d1)) * (1.f / 64.f);
      xt0 = rstd * (d0 - m1 - xh0 * m2);
      xt1 = rstd * (d1 - m1 - xh1 * m2);
      h0 = fmaf(xh0, ln[lane], ln[64 + lane]);
      h1 = fmaf(xh1, ln[lane + 32], ln[64 + lane + 32]);
      d0 = ln[lane] * xt0;
      d1 = ln[lane + 32] * xt1;
      xhat[off + lane] = xh0;
      xhat[off + lane + 32] = xh1;
      xhatd[off + lane] = xt0;
      xhatd[off + lane + 32] = xt1;
    }
    float za[MAX_HIDDEN], zb[MAX_HIDDEN], zda[MAX_HIDDEN], zdb[MAX_HIDDEN];
#pragma unroll
    for (int l = 0; l < MAX_HIDDEN; ++l) {
      if (l < n_hidden) {
        h_all[l * plane + off + lane] = h0;
        h_all[l * plane + off + lane + 32] = h1;
        hd_all[l * plane + off + lane] = d0;
        hd_all[l * plane + off + lane + 32] = d1;
        const float* wt = s_wt + l * 4096;
        float a = mlp_b[l * 64 + lane], b = mlp_b[l * 64 + lane + 32], ad = 0.f, bd = 0.f;
        for (int k = 0; k < 32; ++k) {
          const float v0 = __shfl_sync(0xffffffffu, h0, k), v1 = __shfl_sync(0xffffffffu, h1, k);
          const float u0 = __shfl_sync(0xffffffffu, d0, k), u1 = __shfl_sync(0xffffffffu, d1, k);
          const float w00 = wt[k * 64 + lane], w01 = wt[k * 64 + lane + 32];
          const float w10 = wt[(k + 32) * 64 + lane], w11 = wt[(k + 32) * 64 + lane + 32];
          a = fmaf(v0, w00, a); b = fmaf(v0, w01, b); a = fmaf(v1, w10, a); b = fmaf(v1, w11, b);
          ad = fmaf(u0, w00, ad); bd = fmaf(u0, w01, bd); ad = fmaf(u1, w10, ad); bd = fmaf(u1, w11, bd);
        }
        za[l] = a; zb[l] = b; zda[l] = ad; zdb[l] = bd;
        h0 = silu_f(a);
        h1 = silu_f(b);
        d0 = dsilu_f(a) * ad;
        d1 = dsilu_f(b) * bd;
      }
    }
    h_all[n_hidden * plane + off + lane] = h0;
    h_all[n_hidden * plane + off + lane + 32] = h1;
    hd_all[n_hidden * plane + off + lane] = d0;
    hd_all[n_hidden * plane + off + lane + 32] = d1;
    const float sd = seed[atom];
    float hdb0 = wl0, hdb1 = wl1;            // adjoint of hd (tangent stream)
    float hb0 = wl0 * sd, hb1 = wl1 * sd;    // adjoint of h (primal stream)
#pragma unroll
    for (int l = MAX_HIDDEN - 1; l >= 0; --l) {
      if (l < n_hidden) {
        const float* w = s_w + l * 4096;
        const float ds0 = dsilu_f(za[l]), ds1 = dsilu_f(zb[l]);
        const float zdbar0 = hdb0 * ds0, zdbar1 = hdb1 * ds1;
        const float zbar0 = fmaf(hdb0 * d2silu_r(za[l]), zda[l], hb0 * ds0);
        const float zbar1 = fmaf(hdb1 * d2silu_r(zb[l]), zdb[l], hb1 * ds1);
        gz_all[l * plane + off + lane] = zdbar0;
        gz_all[l * plane + off + lane + 32] = zdbar1;
        zbar_all[l * plane + off + lane] = zbar0;
        zbar_all[l * plane + off + lane + 32] = zbar1;
        float a = 0.f, b = 0.f, ab = 0.f, bb = 0.f;
        for (int n = 0; n < 32; ++n) {
          const float v0 = __shfl_sync(0xffffffffu, zdbar0, n), v1 = __shfl_sync(0xffffffffu, zdbar1, n);
          const float u0 = __shfl_sync(0xffffffffu, zbar0, n), u1 = __shfl_sync(0xffffffffu, zbar1, n);
          const float w00 = w[n * 64 + lane], w01 = w[n * 64 + lane + 32];
          const float w10 = w[(n + 32) * 64 + lane], w11 = w[(n + 32) * 64 + lane + 32];
          a = fmaf(v0, w00, a); b = fmaf(v0, w01, b); a = fmaf(v1, w10, a); b = fmaf(v1, w11, b);
          ab = fmaf(u0, w00, ab); bb = fmaf(u0, w01, bb); ab = fmaf(u1, w10, ab); bb = fmaf(u1, w11, bb);
        }
        hdb0 = a; hdb1 = b; hb0 = ab; hb1 = bb;
      }
    }
    g_h0[off + lane] = hdb0;
    g_h0[off + lane + 32] = hdb1;
    hbar0[off + lane] = hb0;
    hbar0[off + lane + 32] = hb1;
    if (ln != nullptr) {
      const float k0 = hdb0 * ln[lane], k1 = hdb1 * ln[lane + 32];
      const float m2 = sum32(fmaf(xh0, xd0, xh1 * xd1)) * (1.f / 64.f);
      const float skx = sum32(fmaf(k0, xh0, k1 * xh1));
      const float skt = sum32(fmaf(k0, xt0, k1 * xt1));
      const float v0 = fmaf(hb0, ln[lane], rstd * (-k0 * m2 - skx * xd0 * (1.f / 64.f)));
      const float v1 = fmaf(hb1, ln[lane + 32], rstd * (-k1 * m2 - skx * xd1 * (1.f / 64.f)));
      const float mv = sum32(v0 + v1) * (1.f / 64.f);
      const float mvx = sum32(fmaf(v0, xh0, v1 * xh1)) * (1.f / 64.f);
      hb0 = rstd * (v0 - mv - xh0 * mvx) - rstd * xh0 * skt * (1.f / 64.f);
      hb1 = rstd * (v1 - mv - xh1 * mvx) - rstd * xh1 * skt * (1.f / 64.f);
    }
    bar_x[off + lane] = hb0;
    bar_x[off + lane + 32] = hb1;
  }
}

// ---- magmom head reverse: m = |x.w + b| --------------------------------------------------------
__global__ void magmom_bwd_kernel(const float* __restrict__ x, int n_atoms, const float* __restrict__ w, float b,
                                  const float* __restrict__ g_m, float* __restrict__ g_x,
                                  float* __restrict__ g_lin) {
  const int lane = threadIdx.x & 31;
  const int atom = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (atom >= n_atoms) return;
  const float* row = x + (size_t)atom * 64;
  const float w0 = w[lane], w1 = w[lane + 32];
  const float v = sum32(fmaf(row[lane], w0, row[lane + 32] * w1)) + b;
  const float sgn = v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f);
  const float gl = sgn * g_m[atom];
  if (lane == 0) g_lin[atom] = gl;
  g_x[(size_t)atom * 64 + lane] += gl * w0;
  g_x[(size_t)atom * 64 + lane + 32] += gl * w1;
}

// ---- one CombinedLoss term over a flat vector ----------------------------------------------------
__global__ void __launch_bounds__(256)
loss_terms_kernel(const float* __restrict__ pred, const float* __restrict__ target, int n, int kind, float delta,
                  float* __restrict__ g_pred, double* __restrict__ sums) {
  __shared__ double s_red[3][8];
  double sl = 0.0, sa = 0.0, sc = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float t = target[i];
    float gi = 0.f;
    if (t == t) {  // NaN target = missing label (trainer.py:803-806)
      const float err = pred[i] - t;
      const float ae = fabsf(err);
      float li;
      if (kind == 0) {
        li = err * err;
        gi = 2.f * err;
      } else if (kind == 1) {
        li = ae;
        gi = err > 0.f ? 1.f : (err < 0.f ? -1.f : 0.f);
      } else {
        const bool small = ae <= delta;
        li = small ? 0.5f * err * err : delta * (ae - 0.5f * delta);
        gi = small ? err : (err > 0.f ? delta : -delta);
      }
      sl += (double)li;
      sa += (double)ae;
      sc += 1.0;
    }
    g_pred[i] = gi;
  }
  sl = sum32d(sl), sa = sum32d(sa), sc = sum32d(sc);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) {
    s_red[0][wid] = sl;
    s_red[1][wid] = sa;
    s_red[2][wid] = sc;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int q = 0; q < 8; ++q) t += s_red[threadIdx.x][q];
    atomicAdd(sums + threadIdx.x, t);
  }
}

// ---- Adam on one flat buffer (torch.optim.Adam semantics, no amsgrad) ----------------------------------
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, float lr, float beta1, float beta2, float eps,
                            float weight_decay, float bc1, float bc2) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float pi = p[i];
    const float gi = fmaf(weight_decay, pi, g[i]);
    const float mi = fmaf(beta1, m[i], (1.f - beta1) * gi);
    const float vi = fmaf(beta2, v[i], (1.f - beta2) * gi * gi);
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi / bc2) + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

}  // namespace

// shared with wgrad_tc.cu
void wgrad_reduce_launch(const float* partial, const float* cs_partial, int n_chunks, int n, float* out, int ldo, float* colsum,
                         cudaStream_t stream) {
  const int total = 64 * n + n;
  wgrad_reduce_kernel<<<(total + 31) / 32, 256, 0, stream>>>(partial, cs_partial, n_chunks, n, out, ldo, colsum);
}
int wgrad_tc(const float* x, const float* x2, int ldx, const int32_t* x_rows, int x_silu, const float* g, int ldg,
             const int32_t* g_rows, int m, int n_out, float* out, int ldo, float* colsum, float* workspace, int max_chunks,
             cudaStream_t stream);  // wgrad_tc.cu: returns 1 when it does not take the call
}  // namespace chg

using namespace chg;

extern "C" int64_t chg_wgrad_workspace_floats(int32_t n_out) {
  // chunks(n) * (64 n + n) with chunks(n) <= min(WG_MAX_CHUNKS, 2 * 256 / n * SMs): largest at n = 256 on 148+ SMs
  const int64_t chunks = std::min<int64_t>(WG_MAX_CHUNKS, (int64_t)sm_count() * 2 * std::max(1, 256 / n_out));
  return chunks * (64 * (int64_t)n_out + n_out);
}

extern "C" int chg_wgrad(const float* x, const float* x2, int32_t ldx, const int32_t* x_rows, int32_t x_silu, const float* g,
                         int32_t ldg, const int32_t* g_rows, int32_t m, int32_t n_out, float* out, int32_t ldo,
                         float* colsum, float* workspace, void* stream) {
  CHG_CHECK_ARG(m >= 0, "negative size");
  CHG_CHECK_ARG(n_out > 0 && n_out % 64 == 0, "n_out must be a positive multiple of 64");
  CHG_CHECK_ARG(x && g && out && workspace, "null pointer");
  CHG_CHECK_ARG(ldx >= 64 && ldx % 4 == 0 && ldg >= n_out && ldg % 4 == 0 && ldo >= n_out, "bad leading dimension");
  CHG_CHECK_ARG((((uintptr_t)x | (uintptr_t)x2 | (uintptr_t)g | (uintptr_t)workspace) & 15) == 0,
                "x, x2, g, workspace must be 16-byte aligned");
  // tensor cores (3xTF32) for the large reductions; same partial buffer, same fp64 second pass
  const int64_t cap = std::min<int64_t>(WG_MAX_CHUNKS, (int64_t)sm_count() * 2 * std::max(1, 256 / n_out));
  const int rc = wgrad_tc(x, x2, ldx, x_rows, x_silu, g, ldg, g_rows, m, n_out, out, ldo, colsum, workspace, (int)cap,
                          as_stream(stream));
  if (rc != 1) return rc;  // 1: not taken (small reduction): the FFMA kernel below
  const int steps = (m + WG_ROWS - 1) / WG_ROWS;
  // narrow outputs get more row chunks (more CTAs per SM in flight: the kernel is latency bound)
  const int n_chunks = max(1, min(min(steps, sm_count() * 2 * max(1, 256 / n_out)), WG_MAX_CHUNKS));
  float* partial = workspace;
  float* cs_partial = colsum != nullptr ? workspace + (size_t)n_chunks * 64 * n_out : nullptr;
  dim3 grid(n_chunks, n_out / 64);
  if (x2 != nullptr)
    wgrad_kernel<2><<<grid, 256, 0, as_stream(stream)>>>(x, x2, ldx, x_rows, g, ldg, g_rows, m, n_out, partial, cs_partial);
  else if (x_silu)
    wgrad_kernel<1><<<grid, 256, 0, as_stream(stream)>>>(x, x2, ldx, x_rows, g, ldg, g_rows, m, n_out, partial, cs_partial);
  else
    wgrad_kernel<0><<<grid, 256, 0, as_stream(stream)>>>(x, x2, ldx, x_rows, g, ldg, g_rows, m, n_out, partial, cs_partial);
  {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      set_error("chg_wgrad: launch failed: %s", cudaGetErrorString(e));
      return CHG_ERR_CUDA;
    }
    count_launch();
  }
  const int total = 64 * n_out + n_out;
  wgrad_reduce_kernel<<<(total + 31) / 32, 256, 0, as_stream(stream)>>>(partial, cs_partial, n_chunks, n_out, out, ldo,
                                                                      colsum);
  CHG_LAUNCH_END();
}

extern "C" int chg_colsum(const float* a, int32_t lda, const float* bmul, int32_t ldb, const float* rowscale, int32_t m,
                          int32_t n, double* out, void* stream) {
  CHG_CHECK_ARG(m >= 0, "negative size");
  CHG_CHECK_ARG(n == 64 || n == 128 || n == 256, "n must be 64, 128 or 256");
  if (m == 0) return CHG_OK;
  CHG_CHECK_ARG(a && out, "null pointer");
  const int blocks = max(1, min((m + 63) / 64, sm_count() * 8));
  colsum_kernel<<<blocks, 256, 0, as_stream(stream)>>>(a, lda, bmul, ldb, rowscale, m, n, out);
  CHG_LAUNCH_END();
}

extern "C" int chg_readout_bwd(const float* x, int32_t n_atoms, const float* ln, const float* mlp_wt,
                               const float* mlp_w, const float* mlp_b, int32_t n_hidden, const float* w_last,
                               const float* seed, float* g_x, float* h_all, float* gz_all, float* g_h0, float* xhat,
                               void* stream) {
  CHG_CHECK_ARG(n_atoms >= 0, "negative size");
  CHG_CHECK_ARG(n_hidden >= 1 && n_hidden <= MAX_HIDDEN, "n_hidden must be in [1, 4]");
  if (n_atoms == 0) return CHG_OK;
  CHG_CHECK_ARG(x && mlp_wt && mlp_w && mlp_b && w_last && seed && g_x && h_all && gz_all && g_h0, "null pointer");
  CHG_CHECK_ARG(ln == nullptr || xhat != nullptr, "xhat is required with LayerNorm");
  const int smem = 2 * n_hidden * 4096 * 4;
  static int max_smem_set = 0;
  if (smem > max_smem_set) {
    CHG_CUDA(cudaFuncSetAttribute(readout_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    max_smem_set = smem;
  }
  const int blocks = max(1, min((n_atoms + 7) / 8, sm_count() * 2));
  readout_bwd_kernel<<<blocks, 256, smem, as_stream(stream)>>>(x, n_atoms, ln, mlp_wt, mlp_w, mlp_b, n_hidden, w_last,
                                                               seed, g_x, h_all, gz_all, g_h0, xhat);
  CHG_LAUNCH_END();
}

extern "C" int chg_magmom_bwd(const float* x, int32_t n_atoms, const float* w, float b, const float* g_m, float* g_x,
                              float* g_lin, void* stream) {
  CHG_CHECK_ARG(n_atoms >= 0, "negative size");
  if (n_atoms == 0) return CHG_OK;
  CHG_CHECK_ARG(x && w && g_m && g_x && g_lin, "null pointer");
  const int blocks = (n_atoms * 32 + 255) / 256;
  magmom_bwd_kernel<<<blocks, 256, 0, as_stream(stream)>>>(x, n_atoms, w, b, g_m, g_x, g_lin);
  CHG_LAUNCH_END();
}

extern "C" int chg_loss_terms(const float* pred, const float* target, int32_t n, int32_t kind, float delta,
                              float* g_pred, double* sums, void* stream) {
  CHG_CHECK_ARG(n >= 0, "negative size");
  CHG_CHECK_ARG(kind >= 0 && kind <= 2, "kind must be 0 (MSE), 1 (MAE) or 2 (Huber)");
  if (n == 0) return CHG_OK;
  CHG_CHECK_ARG(pred && target && g_pred && sums, "null pointer");
  const int blocks = max(1, min((n + 255) / 256, sm_count() * 2));
  loss_terms_kernel<<<blocks, 256, 0, as_stream(stream)>>>(pred, target, n, kind, delta, g_pred, sums);
  CHG_LAUNCH_END();
}

extern "C" int chg_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                             float beta2, float eps, float weight_decay, int32_t step, void* stream) {
  CHG_CHECK_ARG(n >= 0 && step >= 1, "bad size or step");
  if (n == 0) return CHG_OK;
  CHG_CHECK_ARG(p && g && m && v, "null pointer");
  const float bc1 = (float)(1.0 - pow((double)beta1, (double)step)), bc2 = (float)(1.0 - pow((double)beta2, (double)step));
  const int blocks = (int)max((int64_t)1, min((n + 255) / 256, (int64_t)sm_count() * 4));
  adam_kernel<<<blocks, 256, 0, as_stream(stream)>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, bc1, bc2);
  CHG_LAUNCH_END();
}

extern "C" int chg_readout_bwd2(const float* x, const float* xd, int32_t n_atoms, const float* ln, const float* mlp_wt,
                                const float* mlp_w, const float* mlp_b, int32_t n_hidden, const float* w_last,
                                const float* seed, float* bar_x, float* h_all, float* hd_all, float* gz_all,
                                float* zbar_all, float* g_h0, float* hbar0, float* xhat, float* xhatd, void* stream) {
  CHG_CHECK_ARG(n_atoms >= 0, "negative size");
  CHG_CHECK_ARG(n_hidden >= 1 && n_hidden <= MAX_HIDDEN, "n_hidden must be in [1, 4]");
  if (n_atoms == 0) return CHG_OK;
  CHG_CHECK_ARG(x && xd && mlp_wt && mlp_w && mlp_b && w_last && seed && bar_x && h_all && hd_all && gz_all && zbar_all &&
                    g_h0 && hbar0, "null pointer");
  CHG_CHECK_ARG(ln == nullptr || (xhat != nullptr && xhatd != nullptr), "xhat / xhatd are required with LayerNorm");
  const int smem = 2 * n_hidden * 4096 * 4;
  static int max_smem_set = 0;
  if (smem > max_smem_set) {
    CHG_CUDA(cudaFuncSetAttribute(readout_bwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    max_smem_set = smem;
  }
  const int blocks = max(1, min((n_atoms + 7) / 8, sm_count() * 2));
  readout_bwd2_kernel<<<blocks, 256, smem, as_stream(stream)>>>(x, xd, n_atoms, ln, mlp_wt, mlp_w, mlp_b, n_hidden, w_last,
                                                                seed, bar_x, h_all, hd_all, gz_all, zbar_all, g_h0, hbar0,
                                                                xhat, xhatd);
  CHG_LAUNCH_END();
}
