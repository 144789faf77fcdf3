// Segmented gather-reduce:  out[r] (+)= sum_{k in [ptr[r], ptr[r+1])} data[perm ? perm[k] : k]
//
// This is the atomics-free replacement of the reference's `aggregate`
// (chgnet/model/functions.py:25-37: zeros().index_add_(0, owners, data), an atomicAdd
// scatter on CUDA) for every scatter in the model: AtomConv messages -> atoms
// (layers.py:124-126; edges are center-sorted so perm == NULL and each segment is one
// contiguous HBM stream), BondConv updates -> bonds (layers.py:252-254), and the
// transposed gathers of the reverse pass (perm = the batch's neighbour / bond-j /
// atom groupings).  Deterministic: fixed summation order.
//
// A group of W/4 lanes (16 for 64-wide rows, 32 for 128-wide) carries one float4 column
// slice per lane; S in {1,2,4,8} such groups share one output row (chosen on the host from
// the mean segment length and the number of segments) and stream its input rows four at a
// time each, so long segments keep up to 32 independent 16-byte loads per row in flight.  HBM-bound: the
// algorithmic bytes are (4*W + 4 [+4 if perm]) per input row + 4*W per output row.
#include "common.cuh"

namespace chg {
namespace {

template <int W, int S>
__global__ void __launch_bounds__(256)
segment_sum_kernel(const float* __restrict__ data, const int32_t* __restrict__ perm,
                   const int32_t* __restrict__ ptr, int n_rows, int accumulate, float* out, int out_ld) {
  // LANES lanes carry one float4 column slice each; S such lane-groups share one output row and
  // take its input rows round-robin (more loads in flight for long segments), then combine their
  // partial sums through shared memory in a fixed order.
  constexpr int LANES = W / 4;
  constexpr int GROUPS = 256 / LANES;     // lane-groups per CTA
  constexpr int ROWS = GROUPS / S;        // output rows per CTA pass
  __shared__ float4 s_part[S > 1 ? 256 : 1];
  const int sub = threadIdx.x % LANES;
  const int grp = threadIdx.x / LANES;
  const int row_in_cta = grp / S, split = grp % S;
  const int n_pass = (n_rows + ROWS - 1) / ROWS;
  for (int pass = blockIdx.x; pass < n_pass; pass += gridDim.x) {
    const int r = pass * ROWS + row_in_cta;
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
    if (r < n_rows) {
      const int beg = ptr[r] + split, end = ptr[r + 1];
      const float* base = data + (size_t)sub * 4;
      int k = beg;
      if (perm == nullptr) {
        for (; k + 3 * S < end; k += 4 * S) {
          const float4 v0 = ldg4(base + (size_t)(k + 0 * S) * W);
          const float4 v1 = ldg4(base + (size_t)(k + 1 * S) * W);
          const float4 v2 = ldg4(base + (size_t)(k + 2 * S) * W);
          const float4 v3 = ldg4(base + (size_t)(k + 3 * S) * W);
          a0 = a0 + v0; a1 = a1 + v1; a2 = a2 + v2; a3 = a3 + v3;
        }
        for (; k < end; k += S) a0 = a0 + ldg4(base + (size_t)k * W);
      } else {
        for (; k + 3 * S < end; k += 4 * S) {
          const int i0 = perm[k], i1 = perm[k + S], i2 = perm[k + 2 * S], i3 = perm[k + 3 * S];
          const float4 v0 = ldg4(base + (size_t)i0 * W);
          const float4 v1 = ldg4(base + (size_t)i1 * W);
          const float4 v2 = ldg4(base + (size_t)i2 * W);
          const float4 v3 = ldg4(base + (size_t)i3 * W);
          a0 = a0 + v0; a1 = a1 + v1; a2 = a2 + v2; a3 = a3 + v3;
        }
        for (; k < end; k += S) a0 = a0 + ldg4(base + (size_t)perm[k] * W);
      }
    }
    // fixed combination order -> bitwise reproducible
    float4 s = (a0 + a1) + (a2 + a3);
    if (S > 1) {
      s_part[threadIdx.x] = s;
      __syncthreads();
      if (split == 0) {
#pragma unroll
        for (int j = 1; j < S; ++j) s = s + s_part[threadIdx.x + j * LANES];
      }
      __syncthreads();
    }
    if (split == 0 && r < n_rows) {
      float* dst = out + (size_t)r * out_ld + sub * 4;
      if (accumulate) s = s + *reinterpret_cast<const float4*>(dst);
      stg4(dst, s);
    }
  }
}

template <int W>
void launch_segsum(int S, const float* data, const int32_t* perm, const int32_t* ptr, int n_rows, int accumulate,
                   float* out, int out_ld, cudaStream_t stream) {
  const int rows = (256 / (W / 4)) / S;
  const int n_pass = (n_rows + rows - 1) / rows;
  const int blocks = max(1, min(n_pass, sm_count() * 8));
  const auto kernel = S == 1   ? segment_sum_kernel<W, 1>
                      : S == 2 ? segment_sum_kernel<W, 2>
                      : S == 4 ? segment_sum_kernel<W, 4>
                               : segment_sum_kernel<W, 8>;
  kernel<<<blocks, 256, 0, stream>>>(data, perm, ptr, n_rows, accumulate, out, out_ld);
}

// dst[i] = src[idx[i]] (gather) or dst[idx[i]] = src[i] (scatter); rows of `width` floats
template <bool SCATTER>
__global__ void move_rows_kernel(const float* __restrict__ src, const int32_t* __restrict__ idx, int n, int width,
                                 float* __restrict__ dst) {
  const int per_row = width / 4;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * per_row) return;
  const int i = (int)(t / per_row), c4 = (int)(t % per_row);
  const int j = idx[i];
  const size_t s_row = SCATTER ? (size_t)i : (size_t)j, d_row = SCATTER ? (size_t)j : (size_t)i;
  stg4(dst + d_row * width + c4 * 4, ldg4(src + s_row * width + c4 * 4));
}

}  // namespace
}  // namespace chg

using namespace chg;

extern "C" int chg_gather_rows(const float* src, const int32_t* idx, int32_t n, int32_t width, float* dst,
                               void* stream) {
  CHG_CHECK_ARG(n >= 0 && width > 0 && width % 4 == 0, "bad size");
  if (n == 0) return CHG_OK;
  CHG_CHECK_ARG(src && idx && dst, "null pointer");
  const long long total = (long long)n * (width / 4);
  move_rows_kernel<false><<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(src, idx, n, width, dst);
  CHG_LAUNCH_END();
}

extern "C" int chg_scatter_rows(const float* src, const int32_t* idx, int32_t n, int32_t width, float* dst,
                                void* stream) {
  CHG_CHECK_ARG(n >= 0 && width > 0 && width % 4 == 0, "bad size");
  if (n == 0) return CHG_OK;
  CHG_CHECK_ARG(src && idx && dst, "null pointer");
  const long long total = (long long)n * (width / 4);
  move_rows_kernel<true><<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(src, idx, n, width, dst);
  CHG_LAUNCH_END();
}

extern "C" int chg_segment_sum(const float* data, int32_t width, const int32_t* perm, const int32_t* ptr,
                               int32_t n_rows, int32_t n_items, int32_t accumulate, float* out, int32_t out_ld,
                               void* stream) {
  CHG_CHECK_ARG(n_rows >= 0 && n_items >= 0, "negative size");
  CHG_CHECK_ARG(width == 64 || width == 128, "width must be 64 or 128");
  CHG_CHECK_ARG(out_ld >= width && out_ld % 4 == 0, "out_ld must be >= width and a multiple of 4");
  if (n_rows == 0) return CHG_OK;
  CHG_CHECK_ARG(ptr && out, "null pointer");
  // lane-groups per output row: enough to keep >= ~8 rows per group for long segments and to
  // fill the machine when there are few segments (n_items is only a hint, any value is correct)
  const int avg = n_items / n_rows;
  const int groups = 256 / (width / 4);  // lane-groups per CTA
  const int resident = sm_count() * 8;   // CTAs of one wave
  int S = 1;
  // grow S while segments stay long enough AND all CTAs still fit in a single wave
  while (S < 8 && avg >= 16 * S && ((long long)n_rows * (2 * S) + groups - 1) / groups <= resident) S *= 2;
  // long segments with one lane-group each leave a latency-bound tail (the last, longest segments stream with 4 loads
  // in flight): two groups per row even when that takes more than one wave (c3: 67.5 -> 64.3 us, c4: 75.7 -> 71.8 us)
  if (S == 1 && avg >= 32) S = 2;
  if (width == 64)
    launch_segsum<64>(S, data, perm, ptr, n_rows, accumulate, out, out_ld, as_stream(stream));
  else
    launch_segsum<128>(S, data, perm, ptr, n_rows, accumulate, out, out_ld, as_stream(stream));
  CHG_LAUNCH_END();
}
