// Dense feature mixing  y[yr] = x[xr] @ wt (+ bias) (+ residual[yr])   — the "true GEMM" part of the
// path: the per-atom / per-bond halves of every GatedMLP first layer, mlp_out + residual
// (reference chgnet/model/layers.py:129-132, 256-260) and their transposes in the
// reverse pass.  x [m][k] row-major, wt [k][n_out] (k-major), k in {64,128,256}.
//
// FFMA version: 64-row x NT-col tile per CTA step, the whole [k][NT] weight panel
// resident in shared memory for the lifetime of a persistent CTA, x streamed in
// [64][64] chunks.  Thread tile 4 rows x (NT/16) cols.
#include <cstdlib>

#include "common.cuh"

namespace chg {
namespace {

constexpr int TM = 64;
constexpr int NTHR = 256;
constexpr int XS = 68;  // smem stride of the x chunk

template <int NT>
__global__ void __launch_bounds__(NTHR, 2)
linear_kernel(const float* __restrict__ x, const int32_t* __restrict__ x_rows, int m, int k,
              const float* __restrict__ wt, const float* __restrict__ bias, const float* residual,
              const int32_t* __restrict__ y_rows, int n_out, float* y) {
  extern __shared__ __align__(16) float smem[];
  float* s_w = smem;           // [k][NT]
  float* s_x = smem + k * NT;  // [64][XS]
  constexpr int CPT = NT / 16;  // columns per thread: 8 (two float4 halves) or 4
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int r0 = ty * 4, c0 = tx * 4;
  const int col_base = blockIdx.y * NT;

  // weight panel: rows of wt restricted to this CTA's NT columns
  for (int i = tid; i < k * (NT / 4); i += NTHR) {
    const int kr = i / (NT / 4), c4 = i % (NT / 4);
    sts4(s_w + kr * NT + c4 * 4, ldg4(wt + (size_t)kr * n_out + col_base + c4 * 4));
  }

  const int n_tiles = (m + TM - 1) / TM;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int base = tile * TM;
    float acc[4][CPT];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < CPT; ++j) acc[i][j] = 0.f;

    for (int kc = 0; kc < k; kc += 64) {
      __syncthreads();  // previous chunk consumed (first pass: weight panel visible)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int id = tid + q * NTHR;
        const int row = id >> 4, c4 = id & 15;
        int r = min(base + row, m - 1);
        if (x_rows != nullptr) r = __ldg(x_rows + r);  // fused row gather
        sts4(s_x + row * XS + c4 * 4, ldg4(x + (size_t)r * k + kc + c4 * 4));
      }
      __syncthreads();
#pragma unroll 2
      for (int k4 = 0; k4 < 16; ++k4) {
        float4 av[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) av[i] = lds4(s_x + (r0 + i) * XS + k4 * 4);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const float* wrow = s_w + (kc + k4 * 4 + kk) * NT;
          const float4 w0 = lds4(wrow + c0);
          float4 w1;
          if (CPT == 8) w1 = lds4(wrow + 64 + c0);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float a = f4at(av[i], kk);
            acc[i][0] = fmaf(a, w0.x, acc[i][0]);
            acc[i][1] = fmaf(a, w0.y, acc[i][1]);
            acc[i][2] = fmaf(a, w0.z, acc[i][2]);
            acc[i][3] = fmaf(a, w0.w, acc[i][3]);
            if (CPT == 8) {
              acc[i][4] = fmaf(a, w1.x, acc[i][4]);
              acc[i][5] = fmaf(a, w1.y, acc[i][5]);
              acc[i][6] = fmaf(a, w1.z, acc[i][6]);
              acc[i][7] = fmaf(a, w1.w, acc[i][7]);
            }
          }
        }
      }
    }

#pragma unroll
    for (int h = 0; h < CPT / 4; ++h) {
      const int col = col_base + h * 64 + c0;
      float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
      if (bias != nullptr) b = ldg4(bias + col);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int g = base + r0 + i;
        if (g < m) {
          if (y_rows != nullptr) g = __ldg(y_rows + g);  // fused row scatter (rows are unique)
          float4 v = make_float4(acc[i][h * 4 + 0], acc[i][h * 4 + 1], acc[i][h * 4 + 2], acc[i][h * 4 + 3]) + b;
          if (residual != nullptr) v = v + *reinterpret_cast<const float4*>(residual + (size_t)g * n_out + col);
          stg4(y + (size_t)g * n_out + col, v);
        }
      }
    }
  }
}

template <int NT>
int launch_linear(const float* x, const int32_t* x_rows, int m, int k, const float* wt, const float* bias,
                  const float* residual, const int32_t* y_rows, int n_out, float* y, cudaStream_t stream) {
  const int smem = (k * NT + TM * XS) * 4;
  static int max_smem_set = 0;
  if (smem > max_smem_set) {
    CHG_CUDA(cudaFuncSetAttribute(linear_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    max_smem_set = smem;
  }
  const int n_tiles = (m + TM - 1) / TM;
  const int col_tiles = n_out / NT;
  const int per_col = max(1, (2 * sm_count()) / col_tiles);
  dim3 grid(min(n_tiles, per_col), col_tiles);
  linear_kernel<NT><<<grid, NTHR, smem, stream>>>(x, x_rows, m, k, wt, bias, residual, y_rows, n_out, y);
  CHG_LAUNCH_END();
}

}  // namespace

int linear_tc(const float* x, const int32_t* x_rows, int m, int k, const float* wt, const float* bias,
              const float* residual, const int32_t* y_rows, int n_out, float* y, cudaStream_t stream);
int linear_ws(const float* x, int m, int k, const float* wt, const float* bias, const float* residual, int n_out,
              float* y, cudaStream_t stream);

}  // namespace chg

using namespace chg;

extern "C" int chg_linear(const float* x, const int32_t* x_rows, int32_t m, int32_t k, const float* wt,
                          const float* bias, const float* residual, const int32_t* y_rows, int32_t n_out, float* y,
                          void* stream) {
  CHG_CHECK_ARG(m >= 0, "negative size");
  CHG_CHECK_ARG(k == 64 || k == 128 || k == 256, "k must be 64, 128 or 256");
  CHG_CHECK_ARG(n_out > 0 && n_out % 64 == 0, "n_out must be a positive multiple of 64");
  if (m == 0) return CHG_OK;
  CHG_CHECK_ARG(x && wt && y, "null pointer");
  // below ~4k rows the tensor-core kernels' fixed cost (operand images, TMEM allocation) is not amortised: the FFMA
  // kernel is faster there
  if (m >= 4096) {
    if (x_rows == nullptr && y_rows == nullptr) {  // warp-specialised, fed by 2-D TMA tensor maps
      const int rc = linear_ws(x, m, k, wt, bias, residual, n_out, y, as_stream(stream));
      if (rc <= 0) return rc;  // rc == 1: not applicable (k = 256, or no tensor map for these operands)
    }
    return linear_tc(x, x_rows, m, k, wt, bias, residual, y_rows, n_out, y, as_stream(stream));
  }
  if (n_out % 128 == 0 && k <= 128)
    return launch_linear<128>(x, x_rows, m, k, wt, bias, residual, y_rows, n_out, y, as_stream(stream));
  return launch_linear<64>(x, x_rows, m, k, wt, bias, residual, y_rows, n_out, y, as_stream(stream));
}
