// AtomConv / BondConv message + aggregation as ONE warp-specialised tcgen05 kernel (sm_100a).
//
//   agg[s] = sum_{rows r of segment s} GatedMLP(pre_r) * w_r          (reference layers.py:113-126, 238-254)
//
// with pre_r = the gather-add of 3 (AtomConv) / 4 (BondConv) first-layer rows (DESIGN.md §3.1), the two
// 64x64 second-layer products on the tensor cores (3xTF32, accumulators in tensor memory), LayerNorm +
// SiLU x sigmoid in the epilogue, and the segmented reduction over the centre-sorted (bond-i-sorted) rows done
// inside the CTA: the [rows, 64] message never goes to HBM.
//
// One persistent CTA per SM, 17 warps (544 threads, <= 96 registers each), three roles connected by mbarriers:
//
//   warps 8-11  producer of the CORE half, warps 12-15 producer of the GATE half of every 128-row tile (two
//               independent groups, so one gathers while the other converts): 16 lanes x float4 per 64-float
//               half-row (coalesced) gather + add the first-layer rows, SiLU, store the [128 x 64] half-tile to
//               shared memory (16-byte chunks XOR-swizzled by row), group barrier, then thread t reads ITS row
//               (conflict-free), splits hi / lo and tcgen05.st's it into the group's A stage of tensor memory;
//               BondConv also writes save_pre
//   warp 16     MMA: one lane issues 8 k-steps x 3 split terms of tcgen05.mma.kind::tf32 (M=128, N=64) per
//               half into one of two D stages, tcgen05.commit -> mbarriers
//   warps 0-3   epilogue of the CORE half, warps 4-7 of the GATE half: thread t owns (half of) row t: two
//               tcgen05.ld sweeps (shifted one-pass mean / variance, then normalise: LayerNorm is in-thread, no
//               shuffles), SiLU (core) / sigmoid (gate) -> two [128 x 64] tiles in shared memory; then each of the
//               8 warps reduces a 16-row strip (core x gate x bond weights, the weights read coalesced) over runs
//               of equal segment id: complete segments are stored, strip-boundary partials go to `parts`
//
// A tiny second kernel (seg_stitch) adds the strip partials of every segment that spans strips, in strip
// order (deterministic, no atomics), and zeroes empty segments.
//
// TMEM: 2 x (64 hi + 64 lo) A + 2 x 128 D = 512 columns.  Shared memory: 4 weight images (64 KB) + 2 half-tiles
// (64 KB) + the core / gate output tiles (64 KB) + indices.
#include "gated_common.cuh"
#include "tc.cuh"

namespace chg {
namespace gated {
namespace {

constexpr int WS_THREADS = 544;  // 17 warps: 8 epilogue, 8 producer, 1 MMA
constexpr int TR = 128;          // rows per tile
constexpr int HALF_BYTES = TR * 64 * 4;
constexpr int IMG_BYTES = 64 * 64 * 4;
constexpr int STRIP = 16;        // rows per reduction strip (one half-warp)
constexpr int PB = 4;            // rows gathered per producer batch (x 3-4 loads each in flight)

struct WsSmem {
  static constexpr int IMG_OFF = 0;                          // Bc_hi, Bc_lo, Bg_hi, Bg_lo
  static constexpr int HS_OFF = 4 * IMG_BYTES;               // 2 x [128][64] fp32, swizzled (core | gate producer)
  static constexpr int O_OFF = HS_OFF + 2 * HALF_BYTES;      // 2 x [128][64] fp32, swizzled: silu(core), sigmoid(gate)
  static constexpr int GIDX_OFF = O_OFF + 2 * HALF_BYTES;    // 2 groups x 3 x 128 int
  static constexpr int EIDX_OFF = GIDX_OFF + 2 * 3 * TR * 4;  // 4 x 128 int: segment id, weight row, segment begin / end
  static constexpr int B2_OFF = EIDX_OFF + 4 * TR * 4;       // 128 floats
  static constexpr int LN_OFF = B2_OFF + 128 * 4;            // 256 floats
  static constexpr int TOTAL = LN_OFF + 256 * 4;
};

struct WsBars {
  uint64_t a_full[2], a_empty[2];
  uint64_t d_full[2], d_empty[2];
};

struct FusedArgs {
  const float* p_a;     // ATOM: pcn [N][256]        BOND: pij [Es][256]
  const float* p_b;     // ATOM: pe  [Eu][128]       BOND: px  [N][128]
  const float* p_c;     // BOND: pa [A][128], else null
  const float* wgt;     // ATOM: wag [Eu][64]        BOND: wbg_s [Es][64]
  const int32_t* idx0;  // row of p_a, first half = the SEGMENT id  (center | bond slot i)
  const int32_t* idx1;  // row of p_a, second half                  (nbr    | bond slot j)
  const int32_t* idx2;  // row of p_b                               (d2u    | atom)
  const int32_t* ptr;   // [n_seg + 1] CSR of idx0
  int32_t n_rows, n_seg;
  const float* w2t;     // [64][128]
  const float* b2;      // [128]
  const float* ln;      // [4][64] or null
  float* out;           // [n_seg][64]
  float* parts;         // [ceil(n_rows / 16)][2][64]
  float* save_pre;      // [rows][128] or null
  float* save_p;        // [rows][128] or null
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
// pull one 128-byte line towards L2 (no register, no dependency): issued one tile ahead of the gathers that read it
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// byte offset of 16-byte chunk c (0..15) of row r in a swizzled [128][64] fp32 tile
__device__ __forceinline__ int swz(int r, int c) { return r * 256 + ((c ^ (r & 7)) << 4); }

// image element (n, kk) = src[kk * ld + col0 + n]   (64 x 64, K-major, no swizzle), all threads of the CTA
__device__ __forceinline__ void build_image_ws(uint8_t* hi, uint8_t* lo, const float* __restrict__ src, int ld, int col0,
                                               int tid) {
  for (int i = tid; i < 4096; i += (int)blockDim.x) {
    const int kk = i >> 6, n = i & 63;
    uint32_t h, l;
    tc::split_tf32(__ldg(src + (size_t)kk * ld + col0 + n), h, l);
    const uint32_t off = tc::kmajor_offset(n, kk, 64);
    *reinterpret_cast<uint32_t*>(hi + off) = h;
    *reinterpret_cast<uint32_t*>(lo + off) = l;
  }
}

// ---- epilogue helper: one 64-wide half of row t out of tensor memory ----------------------------------------
// p = acc + b2; y = LN(p) (or p); CORE: out = silu(y);  GATE: out = sigmoid(y); out -> row t of the swizzled tile.
// LayerNorm statistics in one sweep, shifted by the row's first element (no cancellation for |mean| >> std).
template <bool GATE>
__device__ __forceinline__ void epilogue_half(uint32_t d_addr, const float* s_b2, const float* s_gamma, const float* s_beta,
                                              bool use_ln, uint8_t* s_tile, int t, float* save_row) {
  float mean = 0.f, rstd = 1.f;
  if (use_ln) {
    float s1 = 0.f, s2 = 0.f, s1b = 0.f, s2b = 0.f, x0 = 0.f;
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      uint32_t v[32];
      tc::tmem_ld32(d_addr + g * 32, v);
      tc::tmem_ld_wait();
      if (g == 0) x0 = __uint_as_float(v[0]) + s_b2[0];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 b = lds4(s_b2 + g * 32 + q * 4);  // broadcast
        const float d0 = __uint_as_float(v[q * 4]) + b.x - x0, d1 = __uint_as_float(v[q * 4 + 1]) + b.y - x0;
        const float d2 = __uint_as_float(v[q * 4 + 2]) + b.z - x0, d3 = __uint_as_float(v[q * 4 + 3]) + b.w - x0;
        s1 += d0 + d1;
        s1b += d2 + d3;
        s2 = fmaf(d0, d0, fmaf(d1, d1, s2));
        s2b = fmaf(d2, d2, fmaf(d3, d3, s2b));
      }
    }
    const float m1 = (s1 + s1b) * (1.f / 64.f);
    mean = x0 + m1;
    rstd = 1.f / sqrtf(fmaxf((s2 + s2b) * (1.f / 64.f) - m1 * m1, 0.f) + LN_EPS);
  }
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    uint32_t v[32];
    tc::tmem_ld32(d_addr + g * 32, v);
    tc::tmem_ld_wait();
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 b = lds4(s_b2 + g * 32 + q * 4);
      float4 p = make_float4(__uint_as_float(v[q * 4]) + b.x, __uint_as_float(v[q * 4 + 1]) + b.y,
                             __uint_as_float(v[q * 4 + 2]) + b.z, __uint_as_float(v[q * 4 + 3]) + b.w);
      if (save_row != nullptr) stg4(save_row + g * 32 + q * 4, p);
      if (use_ln) {
        const float4 ga = lds4(s_gamma + g * 32 + q * 4), be = lds4(s_beta + g * 32 + q * 4);
        p.x = fmaf((p.x - mean) * rstd, ga.x, be.x);
        p.y = fmaf((p.y - mean) * rstd, ga.y, be.y);
        p.z = fmaf((p.z - mean) * rstd, ga.z, be.z);
        p.w = fmaf((p.w - mean) * rstd, ga.w, be.w);
      }
      float4 o;
      if (GATE) {
        o = make_float4(sigmoid_f(p.x), sigmoid_f(p.y), sigmoid_f(p.z), sigmoid_f(p.w));
      } else {
        o = make_float4(silu_f(p.x), silu_f(p.y), silu_f(p.z), silu_f(p.w));
      }
      *reinterpret_cast<float4*>(s_tile + swz(t, g * 8 + q)) = o;
    }
  }
}

template <int MODE>
__global__ void __launch_bounds__(WS_THREADS, 1) gated_ws_fwd_kernel(const FusedArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* s_img = smem_raw + WsSmem::IMG_OFF;
  uint8_t* s_hs = smem_raw + WsSmem::HS_OFF;
  uint8_t* s_o = smem_raw + WsSmem::O_OFF;
  int* s_gidx = reinterpret_cast<int*>(smem_raw + WsSmem::GIDX_OFF);
  int* s_eidx = reinterpret_cast<int*>(smem_raw + WsSmem::EIDX_OFF);
  float* s_b2 = reinterpret_cast<float*>(smem_raw + WsSmem::B2_OFF);
  float* s_ln = reinterpret_cast<float*>(smem_raw + WsSmem::LN_OFF);
  __shared__ __align__(8) WsBars bars;
  __shared__ uint32_t s_tmem;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool use_ln = a.ln != nullptr;
  const int n_tiles = (a.n_rows + TR - 1) / TR;

  // ---- one-time setup: weight images, bias / LayerNorm rows, barriers, tensor memory ------------------------
  build_image_ws(s_img, s_img + IMG_BYTES, a.w2t, 128, 0, tid);                     // core: (n=c, kk=k) = w2t[k][c]
  build_image_ws(s_img + 2 * IMG_BYTES, s_img + 3 * IMG_BYTES, a.w2t, 128, 64, tid);  // gate
  if (tid < 128) s_b2[tid] = a.b2[tid];
  if (tid < 256) s_ln[tid] = use_ln ? a.ln[tid] : 0.f;
  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&bars.a_full[i], 128);
      tc::mbar_init(&bars.a_empty[i], 1);
      tc::mbar_init(&bars.d_full[i], 1);
      tc::mbar_init(&bars.d_empty[i], 256);
    }
    tc::mbar_fence_init();
  }
  if (warp == 16) tc::tmem_alloc(&s_tmem, 512);
  tc::fence_async_smem();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = s_tmem;
  // TMEM columns: A stage h (h = 0 core, 1 gate) at h*128 (hi) / h*128 + 64 (lo); D stage s at 256 + s*128
  // (core 0..63 | gate 64..127)

  if (warp >= 8 && warp < 16) {
    // ============================ producer groups (gather -> SiLU -> A operand) ============================
    const int half = (warp - 8) >> 2;            // 0: core columns, 1: gate columns
    const int gt = tid - 256 - half * 128;       // 0..127 inside the group; also this thread's tile row / TMEM lane
    const int tx = gt & 15, ty = gt >> 4;        // 16 lanes per row, 8 rows per pass
    const uint32_t lane_sel = (uint32_t)((warp & 3) * 32) << 16;
    int* gi = s_gidx + half * 3 * TR;
    uint8_t* stage = s_hs + half * HALF_BYTES;
    const int col = half * 64 + tx * 4;
    const uint32_t a_hi = tmem_base + half * 128 + lane_sel, a_lo = a_hi + 64;
    int tl = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
      const int base = tile * TR;
      {
        const int r = min(base + gt, a.n_rows - 1);
        gi[gt] = a.idx0[r];
        gi[TR + gt] = a.idx1[r];
        gi[2 * TR + gt] = a.idx2[r];
      }
      tc::wg_barrier(1 + half, 128);  // indices visible; every thread of the group is done with the previous half-tile
      {
        // the rows of the NEXT tile that stream from HBM (p_b: per-bond products for AtomConv; p_c: per-angle products for
        // BondConv): prefetch this group's half (2 lines of 128 B per row) towards L2 while this tile is gathered
        const int nt = tile + gridDim.x;
        if (nt < n_tiles) {
          const int r = min(nt * TR + gt, a.n_rows - 1);
          const float* row = MODE == BOND ? a.p_c + (size_t)r * 128 + half * 64 : a.p_b + (size_t)__ldg(a.idx2 + r) * 128 + half * 64;
          prefetch_l2(row);
          prefetch_l2(row + 32);
        }
      }
#pragma unroll 1
      for (int b = 0; b < 16 / PB; ++b) {
        float4 v[PB];
#pragma unroll
        for (int i = 0; i < PB; ++i) {
          const int row = ty + 8 * (b * PB + i);
          const float* s0 = a.p_a + (size_t)gi[row] * 256 + col;
          const float* s1 = a.p_a + (size_t)gi[TR + row] * 256 + 128 + col;
          const float* s2 = a.p_b + (size_t)gi[2 * TR + row] * 128 + col;
          v[i] = ldg4(s0) + ldg4(s1) + ldg4(s2);
          if (MODE == BOND) v[i] = v[i] + ldg4(a.p_c + (size_t)min(base + row, a.n_rows - 1) * 128 + col);
        }
#pragma unroll
        for (int i = 0; i < PB; ++i) {
          const int row = ty + 8 * (b * PB + i);
          if (a.save_pre != nullptr && base + row < a.n_rows) stg4(a.save_pre + (size_t)(base + row) * 128 + col, v[i]);
          *reinterpret_cast<float4*>(stage + swz(row, tx)) =
              make_float4(silu_f(v[i].x), silu_f(v[i].y), silu_f(v[i].z), silu_f(v[i].w));
        }
      }
      tc::wg_barrier(1 + half, 128);  // the half-tile is complete in shared memory
      tc::mbar_wait(&bars.a_empty[half], (tl & 1) ^ 1);  // the MMAs of the previous tile have read this A stage
      tc::fence_after_sync();
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 v = *reinterpret_cast<const float4*>(stage + swz(gt, g * 4 + q));
          tc::split_tf32(v.x, hi[q * 4 + 0], lo[q * 4 + 0]);
          tc::split_tf32(v.y, hi[q * 4 + 1], lo[q * 4 + 1]);
          tc::split_tf32(v.z, hi[q * 4 + 2], lo[q * 4 + 2]);
          tc::split_tf32(v.w, hi[q * 4 + 3], lo[q * 4 + 3]);
        }
        tc::tmem_st16(a_hi + g * 16, hi);
        tc::tmem_st16(a_lo + g * 16, lo);
      }
      tc::tmem_st_wait();
      tc::fence_before_sync();
      mbar_arrive(&bars.a_full[half]);
    }
  } else if (warp >= 16) {
    // ============================ MMA issuer (warp 16) ============================
    if (warp == 16 && lane == 0) {
      const uint32_t idesc = tc::idesc_tf32(128, 64);
      const uint32_t img = tc::smem_u32(s_img);
      int tl = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
        const int ds = tl & 1;
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          tc::mbar_wait(&bars.a_full[half], tl & 1);
          if (half == 0) tc::mbar_wait(&bars.d_empty[ds], ((tl >> 1) & 1) ^ 1);
          tc::fence_after_sync();
          const uint32_t d_acc = tmem_base + 256 + ds * 128 + half * 64;
          const uint32_t a_hi = tmem_base + half * 128, a_lo = a_hi + 64;
          const uint32_t bhi = img + half * 2 * IMG_BYTES, blo = bhi + IMG_BYTES;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint64_t bh = tc::smem_desc_kmajor(bhi + j * 256, 128, 2048);
            const uint64_t bl = tc::smem_desc_kmajor(blo + j * 256, 128, 2048);
            tc::mma_tf32_ts(d_acc, a_hi + j * 8, bh, idesc, j > 0 ? 1u : 0u);
            tc::mma_tf32_ts(d_acc, a_lo + j * 8, bh, idesc, 1u);
            tc::mma_tf32_ts(d_acc, a_hi + j * 8, bl, idesc, 1u);
          }
          tc::mma_commit(&bars.a_empty[half]);  // A stage reusable once these MMAs have read it
          if (half == 1) tc::mma_commit(&bars.d_full[ds]);
        }
      }
    }
  } else if (warp < 8) {
    // ============================ epilogue: warps 0-3 core half, warps 4-7 gate half ============================
    const int eh = warp >> 2;        // 0: core, 1: gate
    const int t = tid & 127;         // tile row == TMEM lane
    const uint32_t lane_sel = (uint32_t)((warp & 3) * 32) << 16;
    int* s_seg = s_eidx;             // segment id of every tile row
    int* s_wrow = s_eidx + TR;       // row of the bond weight (ATOM: d2u; BOND: slot j - slot i is the segment id)
    int* s_sa = s_eidx + 2 * TR;     // ptr[seg], ptr[seg + 1] of every tile row
    int* s_sb = s_eidx + 3 * TR;
    uint8_t* s_o1 = s_o;
    uint8_t* s_o2 = s_o + HALF_BYTES;
    int tl = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
      const int base = tile * TR;
      const int ds = tl & 1;
      {
        const int r = min(base + t, a.n_rows - 1);
        if (eh == 0) {
          const int seg = a.idx0[r];
          s_seg[t] = seg;
          s_sa[t] = __ldg(a.ptr + seg);
          s_sb[t] = __ldg(a.ptr + seg + 1);
        } else {
          const int wr = MODE == BOND ? a.idx1[r] : a.idx2[r];
          s_wrow[t] = wr;
          prefetch_l2(a.wgt + (size_t)wr * 64);  // the bond-weight row the strip reduction reads after the sweeps
          prefetch_l2(a.wgt + (size_t)wr * 64 + 32);
        }
      }
      tc::mbar_wait(&bars.d_full[ds], (tl >> 1) & 1);
      tc::fence_after_sync();
      const uint32_t d_acc = tmem_base + 256 + ds * 128 + eh * 64 + lane_sel;
      float* save_row = (a.save_p != nullptr && base + t < a.n_rows) ? a.save_p + (size_t)(base + t) * 128 + eh * 64 : nullptr;
      if (eh == 0) {
        epilogue_half<false>(d_acc, s_b2, s_ln, s_ln + 64, use_ln, s_o1, t, save_row);
      } else {
        epilogue_half<true>(d_acc, s_b2 + 64, s_ln + 128, s_ln + 192, use_ln, s_o2, t, save_row);
      }
      tc::fence_before_sync();
      mbar_arrive(&bars.d_empty[ds]);  // the accumulator stage can be overwritten
      tc::wg_barrier(3, 256);

      // ---- segmented reduction: warp w owns the 16-row strip w, lane l the columns 2l, 2l+1 ----------------
      const int strip_lo = base + warp * STRIP;
      const int strip_hi = min(strip_lo + STRIP, a.n_rows);
      if (strip_lo < a.n_rows) {
        float2 w[STRIP];
#pragma unroll
        for (int i = 0; i < STRIP; ++i) {
          const int rr = warp * STRIP + i;
          const float2 w0 = __ldg(reinterpret_cast<const float2*>(a.wgt + (size_t)s_wrow[rr] * 64) + lane);
          if (MODE == ATOM) {
            w[i] = w0;
          } else {
            const float2 wi = __ldg(reinterpret_cast<const float2*>(a.wgt + (size_t)s_seg[rr] * 64) + lane);
            w[i] = make_float2(wi.x * w0.x, wi.y * w0.y);  // (o * w_i) * w_j
          }
        }
        float2 acc = make_float2(0.f, 0.f);
        int cur_row = warp * STRIP;  // first row of the current run
        auto emit = [&](int row0, const float2& v) {
          const int seg = s_seg[row0], sa = s_sa[row0], sb = s_sb[row0];
          float* dst;
          if (sa >= strip_lo && sb <= strip_hi) {
            dst = a.out + (size_t)seg * 64;  // the whole segment lies in this strip
          } else {
            dst = a.parts + ((size_t)(strip_lo / STRIP) * 2 + (sa < strip_lo ? 0 : 1)) * 64;
          }
          *reinterpret_cast<float2*>(dst + lane * 2) = v;
        };
#pragma unroll
        for (int i = 0; i < STRIP; ++i) {
          const int rr = warp * STRIP + i;
          if (strip_lo + i < strip_hi) {
            if (s_seg[rr] != s_seg[cur_row]) {
              emit(cur_row, acc);
              cur_row = rr;
              acc = make_float2(0.f, 0.f);
            }
            const int off = swz(rr, lane >> 1) + (lane & 1) * 8;
            const float2 c = *reinterpret_cast<const float2*>(s_o1 + off);
            const float2 g = *reinterpret_cast<const float2*>(s_o2 + off);
            acc.x = fmaf(c.x * g.x, w[i].x, acc.x);
            acc.y = fmaf(c.y * g.y, w[i].y, acc.y);
          }
        }
        emit(cur_row, acc);
      }
      tc::wg_barrier(3, 256);  // the output tiles and the index rows are free for the next tile
    }
  }

  tc::fence_before_sync();
  __syncthreads();
  if (warp == 16) tc::tmem_dealloc(tmem_base, 512);
}

// out[s] for every segment that spans more than one strip (sum of its strip partials, in strip order) and for
// every empty segment (zeros); segments inside one strip were stored by the main kernel.
__global__ void seg_stitch_kernel(const int32_t* __restrict__ ptr, int n_seg, const float* __restrict__ parts,
                                  float* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int s = idx >> 4, l = idx & 15;
  if (s >= n_seg) return;
  const int a = ptr[s], b = ptr[s + 1];
  if (a >= b) {
    stg4(out + (size_t)s * 64 + l * 4, make_float4(0.f, 0.f, 0.f, 0.f));
    return;
  }
  const int k0 = a / STRIP, k1 = (b - 1) / STRIP;
  if (k0 == k1) return;
  float4 acc = ldg4(parts + ((size_t)k0 * 2 + 1) * 64 + l * 4);
  for (int k = k0 + 1; k <= k1; ++k) acc = acc + ldg4(parts + ((size_t)k * 2) * 64 + l * 4);
  stg4(out + (size_t)s * 64 + l * 4, acc);
}

template <int MODE>
int launch_fused(const FusedArgs& a, cudaStream_t stream) {
  if (a.n_seg == 0) return CHG_OK;
  if (a.n_rows > 0) {
    static bool attr_set = false;
    if (!attr_set) {
      CHG_CUDA(cudaFuncSetAttribute(gated_ws_fwd_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, WsSmem::TOTAL));
      attr_set = true;
    }
    const int n_tiles = (a.n_rows + TR - 1) / TR;
    gated_ws_fwd_kernel<MODE><<<min(n_tiles, sm_count()), WS_THREADS, WsSmem::TOTAL, stream>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      set_error("gated_ws_fwd_kernel: launch failed: %s", cudaGetErrorString(e));
      return CHG_ERR_CUDA;
    }
    count_launch();
  }
  seg_stitch_kernel<<<(a.n_seg * 16 + 255) / 256, 256, 0, stream>>>(a.ptr, a.n_seg, a.parts, a.out);
  CHG_LAUNCH_END();
}

}  // namespace

int atom_conv_fused_ws(const float* pcn, const float* pe, const float* wag, const int32_t* center, const int32_t* nbr,
                       const int32_t* d2u, const int32_t* ptr_c, int n_edges, int n_atoms, const float* w2t, const float* b2,
                       const float* ln, float* agg, float* save_p, float* parts, cudaStream_t stream) {
  FusedArgs a{pcn, pe, nullptr, wag, center, nbr, d2u, ptr_c, n_edges, n_atoms, w2t, b2, ln, agg, parts, nullptr, save_p};
  return launch_fused<ATOM>(a, stream);
}

int bond_conv_fused_ws(const float* pij, const float* px, const float* pa, const float* wbg, const int32_t* ang_atom,
                       const int32_t* ang_i, const int32_t* ang_j, const int32_t* ptr_i, int n_angles, int n_slots,
                       const float* w2t, const float* b2, const float* ln, float* agg, float* save_pre, float* save_p,
                       float* parts, cudaStream_t stream) {
  FusedArgs a{pij, px, pa, wbg, ang_i, ang_j, ang_atom, ptr_i, n_angles, n_slots, w2t, b2, ln, agg, parts, save_pre, save_p};
  return launch_fused<BOND>(a, stream);
}

}  // namespace gated
}  // namespace chg

using namespace chg;

// ---- C ABI: fused message + aggregation (include/chgnet_b200.h) -------------------------------------------------
extern "C" int64_t chg_gated_fused_workspace_floats(int32_t n_rows) {
  if (n_rows < 0) return -1;
  const int64_t msg = (int64_t)n_rows * 64, parts = ((int64_t)n_rows + 15) / 16 * 128;
  return (msg > parts ? msg : parts) + 64;
}

extern "C" int chg_atom_conv_fused(const float* pcn, const float* pe, const float* wag, const int32_t* center,
                                   const int32_t* nbr, const int32_t* d2u, const int32_t* ptr_c, int32_t n_edges,
                                   int32_t n_atoms, const float* w2t, const float* b2, const float* ln, float* agg,
                                   float* save_p, float* work, void* stream) {
  CHG_CHECK_ARG(n_edges >= 0 && n_atoms >= 0, "negative size");
  if (n_atoms == 0) return CHG_OK;
  CHG_CHECK_ARG(ptr_c && agg, "null pointer");
  CHG_CHECK_ARG(n_edges == 0 || (pcn && pe && wag && center && nbr && d2u && w2t && b2 && work), "null pointer");
  // tiny inputs (a few tiles) are launch-bound: the persistent tcgen05 kernel's fixed cost (weight images, TMEM) loses there
  if (n_edges >= ws_min_rows())
    return gated::atom_conv_fused_ws(pcn, pe, wag, center, nbr, d2u, ptr_c, n_edges, n_atoms, w2t, b2, ln, agg, save_p, work,
                                     as_stream(stream));
  // the unfused pair (FFMA message kernel -> segmented sum), the message in `work`
  const int rc = chg_atom_conv_fwd(pcn, pe, wag, center, nbr, d2u, n_edges, w2t, b2, ln, work, save_p, nullptr, stream);
  if (rc != CHG_OK) return rc;
  return chg_segment_sum(work, 64, nullptr, ptr_c, n_atoms, n_edges, 0, agg, 64, stream);
}

extern "C" int chg_bond_conv_fused(const float* pij, const float* px, const float* pa, const float* wbg,
                                   const int32_t* ang_atom, const int32_t* ang_i, const int32_t* ang_j,
                                   const int32_t* ptr_i, int32_t n_angles, int32_t n_slots, const float* w2t,
                                   const float* b2, const float* ln, float* agg, float* save_pre, float* save_p,
                                   float* work, void* stream) {
  CHG_CHECK_ARG(n_angles >= 0 && n_slots >= 0, "negative size");
  if (n_slots == 0) return CHG_OK;
  CHG_CHECK_ARG(ptr_i && agg, "null pointer");
  CHG_CHECK_ARG(n_angles == 0 || (pij && px && pa && wbg && ang_atom && ang_i && ang_j && w2t && b2 && work), "null pointer");
  if (n_angles >= ws_min_rows())
    return gated::bond_conv_fused_ws(pij, px, pa, wbg, ang_atom, ang_i, ang_j, ptr_i, n_angles, n_slots, w2t, b2, ln, agg,
                                     save_pre, save_p, work, as_stream(stream));
  const int rc = chg_bond_conv_fwd(pij, px, pa, wbg, ang_atom, ang_i, ang_j, n_angles, w2t, b2, ln, work, save_pre, save_p, stream);
  if (rc != CHG_OK) return rc;
  return chg_segment_sum(work, 64, nullptr, ptr_i, n_slots, n_angles, 0, agg, 64, stream);
}

// =====================================================================================================================
// Reverse of the AtomConv / BondConv message (same entry points and arithmetic as gated_bwd_kernel<MODE, false> in
// gated.cu; reference: autograd of layers.py:113-121, 238-249): warp-specialised tcgen05 version.
//
//   warps 0-7   P  16 lanes x float4 per 64-wide half-row: saved p -> LayerNorm statistics (shuffles) -> gates,
//                  bond-weight gradients (stored), LayerNorm reverse -> g_p tile in shared memory (two swizzled
//                  halves); group barrier; then thread t converts ITS half-row (t < 128: core, else gate) hi / lo into
//                  the A operand in tensor memory
//   warp 16     M  one lane: g_h = g_p . W2 per half (8 k-steps x 3 split terms of tcgen05.mma.kind::tf32 each)
//   warps 8-15  F  thread t reads its half-row of the accumulator (tcgen05.ld) into a shared-memory tile; group
//                  barrier; then 16 lanes x float4 per half-row: g_pre = g_h * silu'(pre), pre recomputed from the
//                  first-layer rows (AtomConv) or read from save_pre (BondConv), coalesced stores
// TMEM: A (64 hi + 64 lo) x 2 halves = 256 columns, D 2 stages x 128 = 256 columns.
// =====================================================================================================================
namespace chg {
namespace gated {
namespace {

struct WsBwdSmem {
  static constexpr int IMG_OFF = 0;                         // W2 images: core hi, lo, gate hi, lo
  static constexpr int T1_OFF = 4 * IMG_BYTES;              // g_p tile: 2 x [128][64] fp32 swizzled
  static constexpr int T2_OFF = T1_OFF + 2 * HALF_BYTES;    // g_h tile: 2 x [128][64] fp32 swizzled
  static constexpr int PIDX_OFF = T2_OFF + 2 * HALF_BYTES;  // 3 x 128 int (P group)
  static constexpr int FIDX_OFF = PIDX_OFF + 3 * TR * 4;    // 3 x 128 int (F group)
  static constexpr int LN_OFF = FIDX_OFF + 3 * TR * 4;      // 256 floats
  static constexpr int TOTAL = LN_OFF + 256 * 4;
};

struct WsBwdBars {
  uint64_t a_full, a_empty;
  uint64_t d_full[2], d_empty[2];
};

template <int MODE>
__global__ void __launch_bounds__(WS_THREADS, 1) gated_ws_bwd_kernel(const BwdArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* s_img = smem_raw + WsBwdSmem::IMG_OFF;
  uint8_t* s_t1 = smem_raw + WsBwdSmem::T1_OFF;
  uint8_t* s_t2 = smem_raw + WsBwdSmem::T2_OFF;
  int* s_pidx = reinterpret_cast<int*>(smem_raw + WsBwdSmem::PIDX_OFF);
  int* s_fidx = reinterpret_cast<int*>(smem_raw + WsBwdSmem::FIDX_OFF);
  float* s_ln = reinterpret_cast<float*>(smem_raw + WsBwdSmem::LN_OFF);
  __shared__ __align__(8) WsBwdBars bars;
  __shared__ uint32_t s_tmem;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool use_ln = a.ln != nullptr;
  const int n_tiles = (a.n_rows + TR - 1) / TR;

  // g_h[k] = sum_c g_p[c] W2[c][k]: image element (n = k, kk = c) = w2[c][k]
  build_image_ws(s_img, s_img + IMG_BYTES, a.w2, 64, 0, tid);
  build_image_ws(s_img + 2 * IMG_BYTES, s_img + 3 * IMG_BYTES, a.w2 + 64 * 64, 64, 0, tid);
  if (tid < 256) s_ln[tid] = use_ln ? a.ln[tid] : 0.f;
  if (tid == 0) {
    tc::mbar_init(&bars.a_full, 256);
    tc::mbar_init(&bars.a_empty, 1);
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&bars.d_full[i], 1);
      tc::mbar_init(&bars.d_empty[i], 256);
    }
    tc::mbar_fence_init();
  }
  if (warp == 16) tc::tmem_alloc(&s_tmem, 512);
  tc::fence_async_smem();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = s_tmem;
  // TMEM columns: A half h at h*128 (hi) / h*128 + 64 (lo); D stage s at 256 + s*128 (core 0..63 | gate 64..127)

  if (warp < 8) {
    // ============================ P: saved p -> g_p -> A operand ============================
    const int t = tid;                   // 0..255
    const int tx = t & 15, ty = t >> 4;  // 16 lanes per row, 16 rows per pass
    const int c0 = tx * 4;
    const int crow = t & 127, chalf = t >> 7;  // conversion: this thread's tile row and half
    const uint32_t lane_sel = (uint32_t)((warp & 3) * 32) << 16;
    int tl = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
      const int base = tile * TR;
      if (t < TR) {
        const int r = min(base + t, a.n_rows - 1);
        s_pidx[t] = a.idx0[r];
        s_pidx[TR + t] = a.idx1[r];
        if (MODE == ATOM) s_pidx[2 * TR + t] = a.idx2[r];
      }
      tc::wg_barrier(1, 256);  // indices visible; every thread has converted the previous tile
      {
        const int nt = tile + gridDim.x;  // next tile of this CTA: its saved p rows stream from HBM (4 lines of 128 B per row)
        if (nt < n_tiles) {
          const int r = min(nt * TR + (t & 127), a.n_rows - 1);
          const float* row = a.save_p + (size_t)r * 128 + (t >> 7) * 64;
          prefetch_l2(row);
          prefetch_l2(row + 32);
        }
      }
      float4 g1, g2, b1, b2v;
      if (use_ln) {
        g1 = lds4(s_ln + c0);
        b1 = lds4(s_ln + 64 + c0);
        g2 = lds4(s_ln + 128 + c0);
        b2v = lds4(s_ln + 192 + c0);
      }
#pragma unroll 2
      for (int pass = 0; pass < 8; ++pass) {
        const int row = pass * 16 + ty;
        const int g = base + row;
        const bool valid = g < a.n_rows;
        const int r = min(g, a.n_rows - 1);
        const float4 pc4 = ldg4(a.save_p + (size_t)r * 128 + c0);
        const float4 pg4 = ldg4(a.save_p + (size_t)r * 128 + 64 + c0);
        float4 gm, wv;
        if (MODE == ATOM) {
          gm = ldg4(a.g_in + (size_t)s_pidx[row] * 64 + c0);
          wv = ldg4(a.wgt + (size_t)s_pidx[2 * TR + row] * 64 + c0);
        } else {
          gm = ldg4(a.g_in + (size_t)s_pidx[row] * 64 + c0);
          wv = ldg4(a.wgt + (size_t)s_pidx[row] * 64 + c0);
        }
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
          if (valid) stg4(a.g_w0 + (size_t)g * 64 + c0, gm * o);
          go = gm * wv;
        } else {
          const float4 wj = ldg4(a.wgt + (size_t)s_pidx[TR + row] * 64 + c0);
          const float4 gmo = gm * o;
          if (valid) {
            stg4(a.g_w0 + (size_t)g * 64 + c0, gmo * wj);
            stg4(a.g_w1 + (size_t)g * 64 + c0, gmo * wv);
          }
          go = gm * wv * wj;
        }
        float gy1[4], gy2[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float gj = f4at(go, j);
          gy1[j] = gj * gate[j] * (s1[j] * fmaf(y1[j], 1.f - s1[j], 1.f));
          gy2[j] = gj * core[j] * gate[j] * (1.f - gate[j]);
        }
        if (use_ln) {
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
        *reinterpret_cast<float4*>(s_t1 + swz(row, tx)) = make_float4(gy1[0], gy1[1], gy1[2], gy1[3]);
        *reinterpret_cast<float4*>(s_t1 + HALF_BYTES + swz(row, tx)) = make_float4(gy2[0], gy2[1], gy2[2], gy2[3]);
      }
      tc::wg_barrier(1, 256);  // the g_p tile is complete
      tc::mbar_wait(&bars.a_empty, (tl & 1) ^ 1);  // the MMAs of the previous tile have read the A operand
      tc::fence_after_sync();
      const uint8_t* src = s_t1 + chalf * HALF_BYTES;
      const uint32_t a_hi = tmem_base + chalf * 128 + lane_sel, a_lo = a_hi + 64;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 v = *reinterpret_cast<const float4*>(src + swz(crow, g * 4 + q));
          tc::split_tf32(v.x, hi[q * 4 + 0], lo[q * 4 + 0]);
          tc::split_tf32(v.y, hi[q * 4 + 1], lo[q * 4 + 1]);
          tc::split_tf32(v.z, hi[q * 4 + 2], lo[q * 4 + 2]);
          tc::split_tf32(v.w, hi[q * 4 + 3], lo[q * 4 + 3]);
        }
        tc::tmem_st16(a_hi + g * 16, hi);
        tc::tmem_st16(a_lo + g * 16, lo);
      }
      tc::tmem_st_wait();
      tc::fence_before_sync();
      mbar_arrive(&bars.a_full);
    }
  } else if (warp == 16) {
    // ============================ M: g_h = g_p . W2 ============================
    if (lane == 0) {
      const uint32_t idesc = tc::idesc_tf32(128, 64);
      const uint32_t img = tc::smem_u32(s_img);
      int tl = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
        const int ds = tl & 1;
        tc::mbar_wait(&bars.a_full, tl & 1);
        tc::mbar_wait(&bars.d_empty[ds], ((tl >> 1) & 1) ^ 1);
        tc::fence_after_sync();
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          const uint32_t d_acc = tmem_base + 256 + ds * 128 + half * 64;
          const uint32_t a_hi = tmem_base + half * 128, a_lo = a_hi + 64;
          const uint32_t bhi = img + half * 2 * IMG_BYTES, blo = bhi + IMG_BYTES;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint64_t bh = tc::smem_desc_kmajor(bhi + j * 256, 128, 2048);
            const uint64_t bl = tc::smem_desc_kmajor(blo + j * 256, 128, 2048);
            tc::mma_tf32_ts(d_acc, a_hi + j * 8, bh, idesc, j > 0 ? 1u : 0u);
            tc::mma_tf32_ts(d_acc, a_lo + j * 8, bh, idesc, 1u);
            tc::mma_tf32_ts(d_acc, a_hi + j * 8, bl, idesc, 1u);
          }
        }
        tc::mma_commit(&bars.a_empty);
        tc::mma_commit(&bars.d_full[ds]);
      }
    }
  } else if (warp < 16) {
    // ============================ F: g_h -> g_pre = g_h * silu'(pre) ============================
    const int t = tid - 256;             // 0..255
    const int tx = t & 15, ty = t >> 4;
    const int c0 = tx * 4;
    const int crow = t & 127, chalf = t >> 7;
    const uint32_t lane_sel = (uint32_t)((warp & 3) * 32) << 16;
    int tl = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
      const int base = tile * TR;
      const int ds = tl & 1;
      if (MODE == ATOM && t < TR) {
        const int r = min(base + t, a.n_rows - 1);
        s_fidx[t] = a.idx0[r];
        s_fidx[TR + t] = a.idx1[r];
        s_fidx[2 * TR + t] = a.idx2[r];
      }
      {
        // the rows this tile's silu' needs that stream from HBM: per-bond products (AtomConv) / saved pre (BondConv)
        const int r = min(base + crow, a.n_rows - 1);
        const float* row = MODE == ATOM ? a.p_b + (size_t)__ldg(a.idx2 + r) * 128 + chalf * 64 : a.save_pre + (size_t)r * 128 + chalf * 64;
        prefetch_l2(row);
        prefetch_l2(row + 32);
      }
      tc::mbar_wait(&bars.d_full[ds], (tl >> 1) & 1);
      tc::fence_after_sync();
      {
        const uint32_t d_acc = tmem_base + 256 + ds * 128 + chalf * 64 + lane_sel;
        uint8_t* dst = s_t2 + chalf * HALF_BYTES;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          uint32_t v[32];
          tc::tmem_ld32(d_acc + g * 32, v);
          tc::tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(dst + swz(crow, g * 8 + q)) =
                make_float4(__uint_as_float(v[q * 4]), __uint_as_float(v[q * 4 + 1]), __uint_as_float(v[q * 4 + 2]),
                            __uint_as_float(v[q * 4 + 3]));
        }
      }
      tc::fence_before_sync();
      mbar_arrive(&bars.d_empty[ds]);
      tc::wg_barrier(2, 256);  // the g_h tile (and the index rows) are complete
#pragma unroll 2
      for (int pass = 0; pass < 8; ++pass) {
        const int row = pass * 16 + ty;
        const int g = base + row;
        float4 vc, vg;
        if (MODE == ATOM) {
          const float* s0 = a.p_a + (size_t)s_fidx[row] * 256 + c0;
          const float* s1 = a.p_a + (size_t)s_fidx[TR + row] * 256 + 128 + c0;
          const float* s2 = a.p_b + (size_t)s_fidx[2 * TR + row] * 128 + c0;
          vc = ldg4(s0) + ldg4(s1) + ldg4(s2);
          vg = ldg4(s0 + 64) + ldg4(s1 + 64) + ldg4(s2 + 64);
        } else {
          const int r = min(g, a.n_rows - 1);
          vc = ldg4(a.save_pre + (size_t)r * 128 + c0);
          vg = ldg4(a.save_pre + (size_t)r * 128 + 64 + c0);
        }
        const float4 hc = *reinterpret_cast<const float4*>(s_t2 + swz(row, tx));
        const float4 hg = *reinterpret_cast<const float4*>(s_t2 + HALF_BYTES + swz(row, tx));
        if (g < a.n_rows) {
          stg4(a.g_pre + (size_t)g * 128 + c0,
               make_float4(hc.x * dsilu_f(vc.x), hc.y * dsilu_f(vc.y), hc.z * dsilu_f(vc.z), hc.w * dsilu_f(vc.w)));
          stg4(a.g_pre + (size_t)g * 128 + 64 + c0,
               make_float4(hg.x * dsilu_f(vg.x), hg.y * dsilu_f(vg.y), hg.z * dsilu_f(vg.z), hg.w * dsilu_f(vg.w)));
        }
      }
      tc::wg_barrier(2, 256);  // the g_h tile can be overwritten
    }
  }

  tc::fence_before_sync();
  __syncthreads();
  if (warp == 16) tc::tmem_dealloc(tmem_base, 512);
}

template <int MODE>
int launch_ws_bwd(const BwdArgs& a, cudaStream_t stream) {
  if (a.n_rows == 0) return CHG_OK;
  static bool attr_set = false;
  if (!attr_set) {
    CHG_CUDA(cudaFuncSetAttribute(gated_ws_bwd_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, WsBwdSmem::TOTAL));
    attr_set = true;
  }
  const int n_tiles = (a.n_rows + TR - 1) / TR;
  gated_ws_bwd_kernel<MODE><<<min(n_tiles, sm_count()), WS_THREADS, WsBwdSmem::TOTAL, stream>>>(a);
  CHG_LAUNCH_END();
}

}  // namespace

int atom_conv_bwd_ws(const BwdArgs& a, cudaStream_t stream) { return launch_ws_bwd<ATOM>(a, stream); }
int bond_conv_bwd_ws(const BwdArgs& a, cudaStream_t stream) { return launch_ws_bwd<BOND>(a, stream); }

}  // namespace gated
}  // namespace chg
