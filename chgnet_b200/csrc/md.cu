// Device-resident molecular dynamics / relaxation updates (SURVEY.md §8 row f2).
//
// The reference keeps positions in an ase.Atoms object on the host and calls the model once per step through
// CHGNetCalculator.calculate (chgnet/model/dynamics.py:129-181): structure -> graph on the CPU -> H2D -> model -> D2H.
// Here positions, velocities and forces stay on the device in fp64; these kernels are the integrator halves that sit
// on either side of chg_forward inside ONE CUDA graph per step (chgnet_b200/dynamics_device.py):
//   chg_md_kick_drift : v += dt/2 F/m ; x += dt v ; frac = x L^-1 (fp64 for the graph builder, fp32 for the model);
//                       max |x - x_ref|^2 for the neighbour-list skin test
//   chg_md_kick       : v += dt/2 F/m ; kinetic energy
//   chg_fire_step     : FIRE (Bitzek et al. 2006; the reference's default optimizer, dynamics.py:190-204) with its
//                       state (dt, alpha, counters) in device memory: two launches, no host decision in the loop
//
// Berendsen NVT / NPT (the reference's MolecularDynamics ensembles, dynamics.py:595-715) with the cell in device
// memory, so a captured step reads the cell, the targets and the couplings from buffers, never from launch arguments:
//   chg_md_cell_step      : ONE block: K from the per-block partials (fixed order) -> thermostat lambda -> pressure
//                           -> barostat mu -> L_new, L_new^-1, V, fp32 lattice, strain of the lists
//   chg_md_kick_drift_cell: [v *= lambda; x = (x L_old^-1) L_new; v += dt/2 F/m; partials of sum m v]
//                           -> [v -= p_mean/m; x += dt v; frac; max displacement in the build frame]
//   chg_md_kick_partials  : v += dt/2 F/m; per-block partials of K_aa and K_tr (deterministic: no atomics)
#include "common.cuh"

namespace chg {
namespace {

struct Mat3 {
  double m[9];
};

__device__ __forceinline__ void atomic_max_nonneg(double* addr, double v) {
  // non-negative doubles order like their bit patterns
  atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

__global__ void md_kick_drift_kernel(double* __restrict__ x, double* __restrict__ v, const double* __restrict__ f,
                                     const double* __restrict__ inv_mass, int n, double dt, Mat3 inv_l,
                                     double* __restrict__ frac64, float* __restrict__ frac32, const double* __restrict__ x_ref,
                                     double* __restrict__ max_disp2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double im = inv_mass[i];
  double xi[3], d2 = 0.0;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const double vj = v[3 * i + j] + 0.5 * dt * f[3 * i + j] * im;
    v[3 * i + j] = vj;
    xi[j] = x[3 * i + j] + dt * vj;
    x[3 * i + j] = xi[j];
    if (x_ref != nullptr) {
      const double d = xi[j] - x_ref[3 * i + j];
      d2 += d * d;
    }
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const double fj = xi[0] * inv_l.m[j] + xi[1] * inv_l.m[3 + j] + xi[2] * inv_l.m[6 + j];
    frac64[3 * i + j] = fj;
    frac32[3 * i + j] = (float)fj;
  }
  if (max_disp2 != nullptr) atomic_max_nonneg(max_disp2, d2);
}

__global__ void md_kick_kernel(double* __restrict__ v, const double* __restrict__ f, const double* __restrict__ inv_mass, int n,
                               double dt, double* __restrict__ e_kin) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double ke = 0.0;
  if (i < n) {
    const double im = inv_mass[i];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double vj = v[3 * i + j] + 0.5 * dt * f[3 * i + j] * im;
      v[3 * i + j] = vj;
      ke += vj * vj;
    }
    ke *= 0.5 / im;
  }
  ke = sum32d(ke);
  if (e_kin != nullptr && (threadIdx.x & 31) == 0 && ke != 0.0) atomicAdd(e_kin, ke);
}

// FIRE state in device memory: [0] dt, [1] alpha, [2] n_pos (as double), [3] power, [4] |v|^2, [5] |f|^2, [6] max |f_i|^2,
// [7] max step^2 of the last update
__global__ void fire_reduce_kernel(const double* __restrict__ v, const double* __restrict__ f, int n, double* __restrict__ st) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double p = 0.0, vv = 0.0, ff = 0.0;
  if (i < n) {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double vj = v[3 * i + j], fj = f[3 * i + j];
      p += fj * vj;
      vv += vj * vj;
      ff += fj * fj;
    }
    atomic_max_nonneg(st + 6, ff);
  }
  p = sum32d(p);
  vv = sum32d(vv);
  ff = sum32d(ff);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(st + 3, p);
    atomicAdd(st + 4, vv);
    atomicAdd(st + 5, ff);
  }
}

__global__ void fire_update_kernel(double* __restrict__ x, double* __restrict__ v, const double* __restrict__ f, int n,
                                   double* __restrict__ st, Mat3 inv_l, double* __restrict__ frac64, float* __restrict__ frac32,
                                   double dt_max, double max_step) {
  // every thread derives the same scalars from the reduced state (written by the previous launch)
  const double n_min = 5.0, f_inc = 1.1, f_dec = 0.5, alpha_start = 0.1, f_alpha = 0.99;
  double dt = st[0], alpha = st[1], n_pos = st[2];
  const double power = st[3], vnorm = sqrt(st[4]), fnorm = sqrt(st[5]);
  const bool uphill = !(power > 0.0);
  if (!uphill) {
    n_pos += 1.0;
    if (n_pos > n_min) {
      dt = fmin(dt * f_inc, dt_max);
      alpha *= f_alpha;
    }
  } else {
    dt *= f_dec;
    alpha = alpha_start;
    n_pos = 0.0;
  }
  const double mix = uphill ? 0.0 : st[1] * vnorm / fmax(fnorm, 1e-30);
  const double keep = uphill ? 0.0 : 1.0 - st[1];
  // the largest displacement of this update bounds the step (ase's maxstep): |dr_i| <= dt |v_i| with
  // |v_new| <= |v| + dt |f|; use the exact per-atom value via a two-phase trick: scale computed from the global maxima
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    double dr[3], vn[3], d2 = 0.0;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      vn[j] = keep * v[3 * i + j] + mix * f[3 * i + j] + dt * f[3 * i + j];
      dr[j] = dt * vn[j];
      d2 += dr[j] * dr[j];
    }
    // per-atom clamp to max_step (a conservative form of ase's global rescaling: never moves an atom further)
    const double s = d2 > max_step * max_step ? max_step / sqrt(d2) : 1.0;
    double xi[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      v[3 * i + j] = vn[j];
      xi[j] = x[3 * i + j] + s * dr[j];
      x[3 * i + j] = xi[j];
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double fj = xi[0] * inv_l.m[j] + xi[1] * inv_l.m[3 + j] + xi[2] * inv_l.m[6 + j];
      frac64[3 * i + j] = fj;
      frac32[3 * i + j] = (float)fj;
    }
  }
  __syncthreads();
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
    // last block publishes the new scalars for the host / the next step; the sums are re-zeroed by the caller
    st[8] = dt;
    st[9] = alpha;
    st[10] = n_pos;
    st[11] = st[6];  // max |f_i|^2 seen by this step
  }
}

// commits the scalars of fire_update (a separate tiny launch: every block of the update must have read the old ones)
__global__ void fire_commit_kernel(double* __restrict__ st) {
  st[0] = st[8];
  st[1] = st[9];
  st[2] = st[10];
  st[3] = st[4] = st[5] = st[6] = 0.0;
}

inline unsigned blocks(int n) { return (unsigned)((n + 255) / 256); }

// ---- Berendsen ensembles --------------------------------------------------------------------------------------------
// cell state (64 doubles; rows of L = lattice vectors, row-major):
enum : int {
  CS_L = 0,         // current cell
  CS_LINV = 9,      // its inverse
  CS_LOLD_INV = 18, // inverse of the cell at the start of the step (positions are rescaled from it)
  CS_LREF = 27,     // cell at the last neighbour-list build
  CS_LREF_INV = 36, // its inverse
  CS_VOL = 45,      // |det L|
  CS_LAMBDA = 46,   // thermostat factor of the last step
  CS_TEMP = 47,     // temperature the last thermostat saw (K)
  CS_D2 = 52,       // max_i |(s_i - s_ref,i) L_ref|^2 (reset by chg_md_cell_step)
  CS_EPS = 53,      // || L_ref^-1 L - I ||_F
};
// parameters: [0] T0 (K), [1] P0 (eV/A^3), [2] dt / tau_t, [3] dt beta / (3 tau_p), [4..6] mask, [7] k_B (eV/K)
enum : int { MD_THERMO = 1, MD_BARO_ISO = 2, MD_BARO_ANISO = 4, MD_FIX_COM = 8 };

__device__ __forceinline__ void mat3_inv(const double* a, double* r) {
  const double c00 = a[4] * a[8] - a[5] * a[7], c01 = a[5] * a[6] - a[3] * a[8], c02 = a[3] * a[7] - a[4] * a[6];
  const double det = a[0] * c00 + a[1] * c01 + a[2] * c02, id = 1.0 / det;
  r[0] = c00 * id;
  r[1] = (a[2] * a[7] - a[1] * a[8]) * id;
  r[2] = (a[1] * a[5] - a[2] * a[4]) * id;
  r[3] = c01 * id;
  r[4] = (a[0] * a[8] - a[2] * a[6]) * id;
  r[5] = (a[2] * a[3] - a[0] * a[5]) * id;
  r[6] = c02 * id;
  r[7] = (a[1] * a[6] - a[0] * a[7]) * id;
  r[8] = (a[0] * a[4] - a[1] * a[3]) * id;
}

// y = x M for a row vector x and a row-major 3x3 M
__device__ __forceinline__ void row_times(const double* x, const double* m, double* y) {
#pragma unroll
  for (int j = 0; j < 3; ++j) y[j] = x[0] * m[j] + x[1] * m[3 + j] + x[2] * m[6 + j];
}

// sum over the threads of a block in a fixed order (warp trees, then the warps in order); the result is valid in thread 0
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double (*sh)[K]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = sum32d(v[k]);
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) sh[warp][k] = v[k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < nw; ++w) {
#pragma unroll
      for (int k = 0; k < K; ++k) v[k] += sh[w][k];
    }
  }
}

__global__ void __launch_bounds__(256) md_cell_kernel(const double* __restrict__ par, double* __restrict__ cs,
                                                      const double* __restrict__ k_part, int nblk,
                                                      const double* __restrict__ virial, float* __restrict__ lat32, int n,
                                                      int flags) {
  __shared__ double sh[8][4];
  double k[4] = {0.0, 0.0, 0.0, 0.0};
  for (int b = threadIdx.x; b < nblk; b += blockDim.x) {
#pragma unroll
    for (int c = 0; c < 4; ++c) k[c] += k_part[4 * b + c];
  }
  block_sum<4>(k, sh);
  if (threadIdx.x != 0) return;
  double lam = 1.0;
  if (flags & MD_THERMO) {
    // NVTBerendsen.scale_velocities: lambda = sqrt(1 + (T0 / T - 1) dt / tau_t), clamped to [0.9, 1.1]
    const double t = k[3] / (3.0 * n * par[7]);
    cs[CS_TEMP] = t;
    if (t == 0.0) {
      lam = 1.1;
    } else {
      const double a = 1.0 + (par[0] / t - 1.0) * par[2];
      lam = a <= 0.81 ? 0.9 : fmin(fmax(sqrt(a), 0.9), 1.1);
    }
  }
  cs[CS_LAMBDA] = lam;
  double* L = cs + CS_L;
#pragma unroll
  for (int j = 0; j < 9; ++j) cs[CS_LOLD_INV + j] = cs[CS_LINV + j];
  if (flags & (MD_BARO_ISO | MD_BARO_ANISO)) {
    // pressure with the ideal-gas term and the momenta after the thermostat: P_a = -sigma_aa + lambda^2 K_aa / V
    const double vol = cs[CS_VOL];
    double p[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) p[a] = (lam * lam * k[a] - virial[4 * a]) / vol;
    if (flags & MD_BARO_ISO) {
      const double mu = 1.0 - par[3] * (par[1] - (p[0] + p[1] + p[2]) / 3.0);
#pragma unroll
      for (int j = 0; j < 9; ++j) L[j] *= mu;
    } else {
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const double mu = 1.0 - par[3] * (par[1] - p[a]) * par[4 + a];
#pragma unroll
        for (int j = 0; j < 3; ++j) L[3 * a + j] *= mu;
      }
    }
    mat3_inv(L, cs + CS_LINV);
    const double det = L[0] * (L[4] * L[8] - L[5] * L[7]) - L[1] * (L[3] * L[8] - L[5] * L[6]) + L[2] * (L[3] * L[7] - L[4] * L[6]);
    cs[CS_VOL] = fabs(det);
    double e2 = 0.0;  // || L_ref^-1 L - I ||_F^2
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      double row[3];
      row_times(cs + CS_LREF_INV + 3 * r, L, row);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double e = row[c] - (r == c ? 1.0 : 0.0);
        e2 += e * e;
      }
    }
    cs[CS_EPS] = sqrt(e2);
  }
#pragma unroll
  for (int j = 0; j < 9; ++j) lat32[j] = (float)L[j];
  cs[CS_D2] = 0.0;
}

__global__ void __launch_bounds__(256) md_scale_kick_kernel(double* __restrict__ x, double* __restrict__ v,
                                                            const double* __restrict__ f, const double* __restrict__ inv_mass,
                                                            int n, double dt, const double* __restrict__ cs,
                                                            double* __restrict__ mom_part, int flags) {
  __shared__ double sh[8][3];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double p[3] = {0.0, 0.0, 0.0};
  if (i < n) {
    const double im = inv_mass[i], lam = cs[CS_LAMBDA];
    double xi[3], vi[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) xi[j] = x[3 * i + j], vi[j] = lam * v[3 * i + j];
    if (flags & (MD_BARO_ISO | MD_BARO_ANISO)) {  // set_cell(scale_atoms=True): fractional coordinates are kept
      double s[3];
      row_times(xi, cs + CS_LOLD_INV, s);
      row_times(s, cs + CS_L, xi);
#pragma unroll
      for (int j = 0; j < 3; ++j) x[3 * i + j] = xi[j];
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      vi[j] += 0.5 * dt * f[3 * i + j] * im;
      v[3 * i + j] = vi[j];
      p[j] = vi[j] / im;
    }
  }
  if (flags & MD_FIX_COM) {
    block_sum<3>(p, sh);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int j = 0; j < 3; ++j) mom_part[3 * blockIdx.x + j] = p[j];
    }
  }
}

__global__ void __launch_bounds__(256) md_com_drift_kernel(double* __restrict__ x, double* __restrict__ v,
                                                           const double* __restrict__ inv_mass, int n, double dt,
                                                           double* __restrict__ cs, const double* __restrict__ mom_part,
                                                           double* __restrict__ frac64, float* __restrict__ frac32,
                                                           const double* __restrict__ s_ref, int flags) {
  __shared__ double pbar[3];
  if (threadIdx.x < 32) {
    // every block reduces the same partials in the same order: the same mean momentum everywhere
    double p[3] = {0.0, 0.0, 0.0};
    if (flags & MD_FIX_COM) {
      for (int b = threadIdx.x; b < (int)gridDim.x; b += 32) {
#pragma unroll
        for (int j = 0; j < 3; ++j) p[j] += mom_part[3 * b + j];
      }
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) p[j] = sum32d(p[j]);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int j = 0; j < 3; ++j) pbar[j] = p[j] / n;
    }
  }
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double im = inv_mass[i];
  double xi[3], s[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const double vj = v[3 * i + j] - pbar[j] * im;
    v[3 * i + j] = vj;
    xi[j] = x[3 * i + j] + dt * vj;
    x[3 * i + j] = xi[j];
  }
  row_times(xi, cs + CS_LINV, s);
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    frac64[3 * i + j] = s[j];
    frac32[3 * i + j] = (float)s[j];
  }
  if (s_ref != nullptr) {
    double ds[3], d[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) ds[j] = s[j] - s_ref[3 * i + j];
    row_times(ds, cs + CS_LREF, d);
    atomic_max_nonneg(cs + CS_D2, d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
  }
}

__global__ void __launch_bounds__(256) md_kick_partials_kernel(double* __restrict__ v, const double* __restrict__ f,
                                                               const double* __restrict__ inv_mass, int n, double dt,
                                                               double* __restrict__ k_part) {
  __shared__ double sh[8][4];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double k[4] = {0.0, 0.0, 0.0, 0.0};
  if (i < n) {
    const double im = inv_mass[i];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      double vj = v[3 * i + j];
      if (f != nullptr) {
        vj += 0.5 * dt * f[3 * i + j] * im;
        v[3 * i + j] = vj;
      }
      k[j] = vj * vj / im;
    }
    k[3] = k[0] + k[1] + k[2];
  }
  block_sum<4>(k, sh);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int c = 0; c < 4; ++c) k_part[4 * blockIdx.x + c] = k[c];
  }
}

}  // namespace
}  // namespace chg

using namespace chg;

extern "C" int chg_md_kick_drift(double* x, double* v, const double* f, const double* inv_mass, int32_t n_atoms, double dt,
                                 const double* inv_lattice /* host, 9 */, double* frac64, float* frac32, const double* x_ref,
                                 double* max_disp2, void* stream) {
  CHG_CHECK_ARG(n_atoms >= 0, "negative size");
  if (n_atoms == 0) return CHG_OK;
  CHG_CHECK_ARG(x && v && f && inv_mass && inv_lattice && frac64 && frac32, "null pointer");
  Mat3 il;
  for (int i = 0; i < 9; ++i) il.m[i] = inv_lattice[i];
  md_kick_drift_kernel<<<blocks(n_atoms), 256, 0, as_stream(stream)>>>(x, v, f, inv_mass, n_atoms, dt, il, frac64, frac32, x_ref, max_disp2);
  CHG_LAUNCH_END();
}

extern "C" int chg_md_kick(double* v, const double* f, const double* inv_mass, int32_t n_atoms, double dt, double* e_kin,
                           void* stream) {
  CHG_CHECK_ARG(n_atoms >= 0, "negative size");
  if (n_atoms == 0) return CHG_OK;
  CHG_CHECK_ARG(v && f && inv_mass, "null pointer");
  md_kick_kernel<<<blocks(n_atoms), 256, 0, as_stream(stream)>>>(v, f, inv_mass, n_atoms, dt, e_kin);
  CHG_LAUNCH_END();
}

extern "C" int chg_fire_step(double* x, double* v, const double* f, int32_t n_atoms, double* state /* device, 12 doubles */,
                             const double* inv_lattice /* host, 9 */, double* frac64, float* frac32, double dt_max,
                             double max_step, void* stream) {
  CHG_CHECK_ARG(n_atoms >= 0, "negative size");
  if (n_atoms == 0) return CHG_OK;
  CHG_CHECK_ARG(x && v && f && state && inv_lattice && frac64 && frac32, "null pointer");
  Mat3 il;
  for (int i = 0; i < 9; ++i) il.m[i] = inv_lattice[i];
  cudaStream_t st = as_stream(stream);
  fire_reduce_kernel<<<blocks(n_atoms), 256, 0, st>>>(v, f, n_atoms, state);
  count_launch();
  fire_update_kernel<<<blocks(n_atoms), 256, 0, st>>>(x, v, f, n_atoms, state, il, frac64, frac32, dt_max, max_step);
  count_launch();
  fire_commit_kernel<<<1, 1, 0, st>>>(state);
  CHG_LAUNCH_END();
}

extern "C" int chg_md_partial_blocks(int32_t n_atoms) { return n_atoms > 0 ? (int)blocks(n_atoms) : 0; }

extern "C" int chg_md_cell_step(const double* params, double* cell_state, const double* k_part, int32_t n_atoms,
                                const double* virial, float* lattice32, int32_t flags, void* stream) {
  CHG_CHECK_ARG(n_atoms > 0, "need at least one atom");
  CHG_CHECK_ARG(params && cell_state && k_part && lattice32, "null pointer");
  CHG_CHECK_ARG(!(flags & (MD_BARO_ISO | MD_BARO_ANISO)) || virial, "a barostat needs the virial");
  CHG_CHECK_ARG((flags & (MD_BARO_ISO | MD_BARO_ANISO)) != (MD_BARO_ISO | MD_BARO_ANISO), "one barostat at a time");
  md_cell_kernel<<<1, 256, 0, as_stream(stream)>>>(params, cell_state, k_part, (int)blocks(n_atoms), virial, lattice32,
                                                   n_atoms, flags);
  CHG_LAUNCH_END();
}

extern "C" int chg_md_kick_drift_cell(double* x, double* v, const double* f, const double* inv_mass, int32_t n_atoms, double dt,
                                      double* cell_state, double* mom_part, double* frac64, float* frac32, const double* s_ref,
                                      int32_t flags, void* stream) {
  CHG_CHECK_ARG(n_atoms >= 0, "negative size");
  if (n_atoms == 0) return CHG_OK;
  CHG_CHECK_ARG(x && v && f && inv_mass && cell_state && frac64 && frac32, "null pointer");
  CHG_CHECK_ARG(!(flags & MD_FIX_COM) || mom_part, "fix_com needs the momentum partials");
  cudaStream_t st = as_stream(stream);
  md_scale_kick_kernel<<<blocks(n_atoms), 256, 0, st>>>(x, v, f, inv_mass, n_atoms, dt, cell_state, mom_part, flags);
  count_launch();
  md_com_drift_kernel<<<blocks(n_atoms), 256, 0, st>>>(x, v, inv_mass, n_atoms, dt, cell_state, mom_part, frac64, frac32,
                                                       s_ref, flags);
  CHG_LAUNCH_END();
}

extern "C" int chg_md_kick_partials(double* v, const double* f, const double* inv_mass, int32_t n_atoms, double dt,
                                    double* k_part, void* stream) {
  CHG_CHECK_ARG(n_atoms >= 0, "negative size");
  if (n_atoms == 0) return CHG_OK;
  CHG_CHECK_ARG(v && inv_mass && k_part, "null pointer");
  md_kick_partials_kernel<<<blocks(n_atoms), 256, 0, as_stream(stream)>>>(v, f, inv_mass, n_atoms, dt, k_part);
  CHG_LAUNCH_END();
}
