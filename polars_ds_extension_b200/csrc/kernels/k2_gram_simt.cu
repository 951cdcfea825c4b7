// K2a — moments of column-major data:  M = [X|Y|1]^T diag(w) [X|Y|1]   (q1 x q1, f64, row-major)
//
// Replaces the reference's get_xtx_with_lambda + build_xty + column sums
// (/root/reference/src/linear/lr/lr_solvers.rs:183-211, 262-278, 483-484) and x^T w x
// (src/num_ext/linear_regression.rs:1026-1027) with ONE pass over the data.
//
// This file is the path for f64 data (the reference's default dtype), weighted fits, more than 4 targets, tiny inputs and
// every shape the tcgen05 kernel does not take (k2_gram_tcgen05.cu is the f32 headline path).  Three kernel families,
// chosen in moments_simt / moments_dmma below:
//   * gram_dmma_side_kernel / gram_dmma_wide_kernel — FP64 tensor cores (mma.sync.m8n8k4, SASS DMMA), up to 64 columns,
//     f64 and (widened on the fly) f32 columns, 16-byte loads through a register ring: the production kernels
//     (f64 with 32 features: 73 % of the HBM peak; 8 features: 93 %);
//   * gram_dmma_kernel — the same blocks with scalar loads, for columns that are not aligned for two-row loads;
//   * gram_simt_kernel — DFMA / FFMA register tiles, any width up to 260 columns and row-blocked frames (bstride != 0).
//
// gram_simt_kernel: X col-major [n x p] (ldx), Y col-major [n x t] (ldy).
// Each CTA walks row tiles of TILE_R rows: tile -> shared memory (row-major, row stride S), every thread owns
// up to MAXT 4x4 blocks of the upper triangle; per tile the block is accumulated in T (a short FMA chain)
// and then added to f64 accumulators, so f32 rounding never grows with n.  When there are fewer blocks than threads
// (q1 <= 88, the usual case) the 256 threads are dealt as (block, row slice): 256 / #blocks slices each take every
// nslices-th row of the tile, so all threads work (with one thread per block only 45 of 256 had work at q1 = 34).
// Per-(CTA, slice) partials are reduced in a fixed order by a second kernel -> bit-reproducible results.
#include "../common.h"
#include "kernels.h"
#include "glm_link.h"

namespace pdsb {

template <typename T>
struct Vec4 { T v[4]; };

template <typename T, int MAXT, bool WEIGHTED>
__global__ void __launch_bounds__(256)
gram_simt_kernel(const T* __restrict__ X, int64_t ldx, const T* __restrict__ Y, int64_t ldy,
                 const T* __restrict__ w, const T* __restrict__ mask, int64_t n, int p, int t,
                 int tile_r, int S, double* __restrict__ partials, int64_t bstride /* 0: column-major; else frame block stride */) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* Zs = reinterpret_cast<T*>(smem_raw);            // [tile_r][S]
  T* ws = Zs + (size_t)tile_r * S;                   // [tile_r]
  const int q1 = p + t + 1;
  const int nt = (q1 + 3) / 4;
  const int ntp = nt * (nt + 1) / 2;
  const int tid = threadIdx.x;

  // (block, row slice) decode for this thread; more than 256 blocks -> MAXT blocks per thread, one slice
  const int nslices = (MAXT == 1 && ntp <= 256) ? 256 / ntp : 1;
  const int slice = (MAXT == 1) ? tid / ntp : 0;
  int ti[MAXT], tj[MAXT];
  bool act[MAXT];
#pragma unroll
  for (int m = 0; m < MAXT; ++m) {
    int idx = (MAXT == 1) ? tid % ntp : tid + m * 256;
    act[m] = (MAXT == 1) ? (slice < nslices) : (idx < ntp);
    int a = 0, rem = act[m] ? idx : 0;
    // row a of the upper triangle has (nt - a) entries
    while (rem >= nt - a) { rem -= nt - a; ++a; }
    ti[m] = a; tj[m] = a + rem;
  }
  double acc[MAXT][16];
#pragma unroll
  for (int m = 0; m < MAXT; ++m)
#pragma unroll
    for (int k = 0; k < 16; ++k) acc[m][k] = 0.0;

  // zero the padding columns once
  for (int i = tid; i < tile_r * S; i += 256) Zs[i] = T(0);
  __syncthreads();

  const int64_t ntiles = (n + tile_r - 1) / tile_r;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t row0 = tile * tile_r;
    // ---- load tile (coalesced along rows).  LU independent loads are issued before the first shared-memory store:
    // with one load in flight per thread this phase was pure latency (~10 us per 128-row tile) ----
    constexpr int LU = 8;
    const int total = tile_r * q1;
    const int tshift = 31 - __clz(tile_r);          // tile_r is a power of two
    for (int base = tid; base < total; base += 256 * LU) {
      T v[LU];
#pragma unroll
      for (int u = 0; u < LU; ++u) {
        const int idx = base + u * 256;
        v[u] = T(0);
        if (idx < total) {
          const int c = idx >> tshift, r = idx & (tile_r - 1);
          const int64_t row = row0 + r;
          if (row < n) {
            if (bstride) {   // row-blocked frame: [block][column][FRAME_ROWS]
              const int64_t o = (row >> 7) * bstride + (row & 127);
              if (c < p) v[u] = X[o + ((int64_t)c << 7)];
              else if (c < p + t) v[u] = Y[o + ((int64_t)(c - p) << 7)];
              else v[u] = mask ? mask[row] : T(1);
            } else if (c < p) v[u] = X[(int64_t)c * ldx + row];
            else if (c < p + t) v[u] = Y[(int64_t)(c - p) * ldy + row];
            else v[u] = mask ? mask[row] : T(1);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < LU; ++u) {
        const int idx = base + u * 256;
        if (idx < total) Zs[(idx & (tile_r - 1)) * S + (idx >> tshift)] = v[u];
      }
    }
    if (WEIGHTED) {
      for (int r = tid; r < tile_r; r += 256) ws[r] = (row0 + r < n) ? w[row0 + r] : T(0);
    }
    __syncthreads();
    // ---- accumulate ----
#pragma unroll
    for (int m = 0; m < MAXT; ++m) {
      if (!act[m]) continue;
      T loc[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) loc[k] = T(0);
      const T* pa = Zs + 4 * ti[m];
      const T* pb = Zs + 4 * tj[m];
      for (int r = slice; r < tile_r; r += nslices) {
        Vec4<T> a = *reinterpret_cast<const Vec4<T>*>(pa + r * S);
        Vec4<T> b = *reinterpret_cast<const Vec4<T>*>(pb + r * S);
        if (WEIGHTED) {
          T wr = ws[r];
#pragma unroll
          for (int k = 0; k < 4; ++k) a.v[k] *= wr;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) loc[i * 4 + j] = fma(a.v[i], b.v[j], loc[i * 4 + j]);
      }
#pragma unroll
      for (int k = 0; k < 16; ++k) acc[m][k] += (double)loc[k];
    }
    __syncthreads();
  }
  // ---- write this CTA's partial (full symmetric) ----
  double* out = partials + ((size_t)blockIdx.x * nslices + slice) * q1 * q1;
#pragma unroll
  for (int m = 0; m < MAXT; ++m) {
    if (!act[m]) continue;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int gi = 4 * ti[m] + i, gj = 4 * tj[m] + j;
        if (gi < q1 && gj < q1) {
          double v = acc[m][i * 4 + j];
          if (ti[m] == tj[m]) {
            // diagonal block: both (i,j) and (j,i) were accumulated by this thread; with weights
            // a_i*w*b_j vs a_j*w*b_i round identically (commutative), so keep it symmetric anyway
            if (gi <= gj) { out[gi * q1 + gj] = v; out[gj * q1 + gi] = v; }
          } else {
            out[gi * q1 + gj] = v;
            out[gj * q1 + gi] = v;
          }
        }
      }
  }
}

// one CTA per moment entry: thread k sums parts k, k+128, ... in order, then a fixed-shape tree -> reproducible
__global__ void __launch_bounds__(128)
reduce_partials_kernel(const double* __restrict__ partials, int nparts, int len, double* __restrict__ out) {
  __shared__ double sh[128];
  const int i = blockIdx.x;
  double s = 0.0;
  for (int k = threadIdx.x; k < nparts; k += 128) s += partials[(size_t)k * len + i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int off = 64; off; off >>= 1) {
    if ((int)threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[i] = sh[0];
}

// ------------------------------------------------------------------------------------------------------------
// f64 data: the same moments on the FP64 tensor-core path (mma.sync m8n8k4, SASS DMMA).  Z~ = [X | Y | 1] is cut into
// NB blocks of 8 columns.  For a 4-row step, lane l holds ONE element per block: Z~[row k0 + l%4][col 8b + l/4] — which
// is at the same time the A fragment (8 x 4, "row") of block b and the B fragment (4 x 8, "col") of block b, so a step
// costs NB loads and NB(NB+1)/2 DMMAs per warp, no shared memory and 8x fewer issue slots than the DFMA kernel above.
// Weights scale the A side only.  Accumulation is f64 throughout; per-CTA partials are combined warp by warp in a
// fixed order, then across CTAs by reduce_partials_kernel: reproducible.
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

template <int NB>
__global__ void __launch_bounds__(256)
gram_dmma_kernel(const double* __restrict__ X, int64_t ldx, const double* __restrict__ Y, int64_t ldy,
                 const double* __restrict__ w, const double* __restrict__ mask, int64_t n, int p, int t,
                 double* __restrict__ partials /* [grid][q1*q1] */) {
  constexpr int NP = NB * (NB + 1) / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sm = reinterpret_cast<double*>(smem_raw);      // [NP][64] CTA-level sum of the warps' accumulators
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, k = lane & 3;
  const int q1 = p + t + 1;
  const double* colp[NB];
  int kind[NB];                                           // 0 data, 1 ones / mask, 2 zero padding
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    const int c = 8 * b + g;
    kind[b] = c < p + t ? 0 : (c == p + t ? 1 : 2);
    colp[b] = c < p ? X + (int64_t)c * ldx : (c < p + t ? Y + (int64_t)(c - p) * ldy : X);
  }
  double acc[NP][2];
#pragma unroll
  for (int i = 0; i < NP; ++i) { acc[i][0] = 0.0; acc[i][1] = 0.0; }

  const int64_t stride = (int64_t)gridDim.x * 8 * 4;
  auto load_step = [&](int64_t r0, double* z, double& wv) {
    const int64_t r = r0 + k;
    const bool in = r < n;
    wv = (in && w) ? w[r] : 1.0;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      double v = 0.0;
      if (in) {
        if (kind[b] == 0) v = colp[b][r];
        else if (kind[b] == 1) v = mask ? mask[r] : 1.0;
      }
      z[b] = v;
    }
  };
  int64_t r0 = ((int64_t)blockIdx.x * 8 + warp) * 4;
  double z[NB], zn[NB], wv = 1.0, wn = 1.0;
  if (r0 < n) load_step(r0, z, wv);
  for (; r0 < n; r0 += stride) {
    const bool more = r0 + stride < n;
    if (more) load_step(r0 + stride, zn, wn);             // next step's loads fly while this step's DMMAs issue
    int idx = 0;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      const double a = z[i] * wv;
#pragma unroll
      for (int j = i; j < NB; ++j) { dmma884(acc[idx][0], acc[idx][1], a, z[j]); ++idx; }
    }
    if (more) {
#pragma unroll
      for (int b = 0; b < NB; ++b) z[b] = zn[b];
      wv = wn;
    }
  }
  // ---- CTA reduction in a fixed order: warp 0 stores, warps 1..7 add one after the other ----
  for (int wturn = 0; wturn < 8; ++wturn) {
    if (warp == wturn) {
#pragma unroll
      for (int i = 0; i < NP; ++i) {
        double* d = sm + i * 64 + g * 8 + 2 * k;
        if (wturn == 0) { d[0] = acc[i][0]; d[1] = acc[i][1]; }
        else { d[0] += acc[i][0]; d[1] += acc[i][1]; }
      }
    }
    __syncthreads();
  }
  // ---- this CTA's partial, full symmetric q1 x q1 (upper entries of the diagonal blocks are mirrored) ----
  double* out = partials + (size_t)blockIdx.x * q1 * q1;
  for (int e = threadIdx.x; e < NP * 64; e += 256) {
    const int blk = e >> 6, rr = (e >> 3) & 7, cc = e & 7;
    int i = 0, rem = blk;
    while (rem >= NB - i) { rem -= NB - i; ++i; }
    const int j = i + rem;
    const int a = 8 * i + rr, b = 8 * j + cc;
    if (a < q1 && b < q1 && (i != j || a <= b)) {
      const double v = sm[e];
      out[(size_t)a * q1 + b] = v;
      out[(size_t)b * q1 + a] = v;
    }
  }
}

// two consecutive rows of a column as they sit in memory (the ring holds them RAW: a conversion right behind the load would
// make the warp wait for it) and as the DMMA wants them
template <typename T> struct Rows2;
template <> struct Rows2<double> { using V = double2; };
template <> struct Rows2<float> { using V = float2; };
__device__ __forceinline__ double2 rows2_f64(const double2& v) { return v; }
__device__ __forceinline__ double2 rows2_f64(const float2& v) { return make_double2((double)v.x, (double)v.y); }
template <typename V> __device__ __forceinline__ V rows2_fill(float a) { V v; v.x = a; v.y = a; return v; }

// ------------------------------------------------------------------------------------------------------------
// Wide variant: the direct kernel keeps 4 rows x (p + t) x 8 B in flight per warp and measured 33 % of the HBM peak with
// the DMMA pipe at 43 % of ITS measured peak (profiles/fp64_peak.cu: 37 TFLOP/s for every mma.sync f64 shape, 33 for
// DFMA) — it waits on memory latency, not on issue slots.  Here a lane loads TWO consecutive rows (16 bytes) per column
// block: lane (g, k) reads rows r0 + 2k, r0 + 2k + 1 of column 8b + g, an 8-row batch per warp.  The rows of a DMMA's
// k index can be any four rows, so the .x halves (rows r0 + {0, 2, 4, 6}) make one m8n8k4 step and the .y halves the
// next.  DEPTH batches live in a register ring (the loop is unrolled over the ring, so every index is static): DEPTH - 1
// batches = 8 (DEPTH - 1) rows per warp are in flight while one is multiplied.  The mask is just the "ones" column read
// from memory.  128-thread CTAs, as many per SM as the registers of the instantiation allow (occupancy query at launch).  Needs 16-byte aligned columns and even leading dimensions.
// T = float: the same kernel for f32 columns (8-byte loads, converted when multiplied): weighted / many-target f32 fits
// that the tcgen05 kernel does not take get exact f64 products and sums at the DMMA rate instead of the SIMT kernel's 15 %.
template <typename T, int NB, int DEPTH, int MINB, bool WEIGHTED>
__global__ void __launch_bounds__(128, MINB)
gram_dmma_wide_kernel(const T* __restrict__ X, int64_t ldx, const T* __restrict__ Y, int64_t ldy,
                      const T* __restrict__ w, const T* __restrict__ mask, int64_t n, int p, int t,
                      double* __restrict__ partials /* [grid][q1*q1] */) {
  using V = typename Rows2<T>::V;
  constexpr int NP = NB * (NB + 1) / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sm = reinterpret_cast<double*>(smem_raw);      // [NP][64]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, k = lane & 3;
  const int q1 = p + t + 1;
  const T* colp[NB];
  int kind[NB];                                           // 0 load, 1 ones, 2 zero padding
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    const int c = 8 * b + g;
    kind[b] = c < p + t ? 0 : (c == p + t ? (mask ? 0 : 1) : 2);
    colp[b] = c < p ? X + (int64_t)c * ldx : (c < p + t ? Y + (int64_t)(c - p) * ldy : (mask ? mask : X));
  }
  double acc[NP][2];
#pragma unroll
  for (int i = 0; i < NP; ++i) { acc[i][0] = 0.0; acc[i][1] = 0.0; }

  V buf[DEPTH][NB];
  V wb[DEPTH];
  const int64_t S = (int64_t)gridDim.x * 4 * 8;
  const int64_t r0 = ((int64_t)blockIdx.x * 4 + warp) * 8;
  int64_t rl = r0 + 2 * k;                                // this lane's first row of the NEXT batch to load
  const T* wp = WEIGHTED ? w + rl : nullptr;
#pragma unroll
  for (int b = 0; b < NB; ++b) colp[b] += rl;
  auto load_batch = [&](V* z, V& wv) {                    // n is a multiple of 8 here: a batch is all in or all out
    const bool in = rl < n;
    if constexpr (WEIGHTED) {
      wv = rows2_fill<V>(0.0f);
      if (in) wv = __ldcs(reinterpret_cast<const V*>(wp));
      wp += S;
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      V v = rows2_fill<V>(0.0f);
      if (in) {
        if (kind[b] == 0) v = __ldcs(reinterpret_cast<const V*>(colp[b]));
        else if (kind[b] == 1) v = rows2_fill<V>(1.0f);
      }
      z[b] = v;
      colp[b] += S;
    }
    rl += S;
  };
  auto multiply = [&](const V* zr, const V& wr) {
    double2 z[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) z[b] = rows2_f64(zr[b]);
    double2 wv = make_double2(1.0, 1.0);
    if constexpr (WEIGHTED) wv = rows2_f64(wr);
    // all block pairs for the even rows, then all for the odd rows: consecutive DMMAs never share an accumulator
    int idx = 0;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      const double a0 = WEIGHTED ? z[i].x * wv.x : z[i].x;
#pragma unroll
      for (int j = i; j < NB; ++j) { dmma884(acc[idx][0], acc[idx][1], a0, z[j].x); ++idx; }
    }
    idx = 0;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      const double a1 = WEIGHTED ? z[i].y * wv.y : z[i].y;
#pragma unroll
      for (int j = i; j < NB; ++j) { dmma884(acc[idx][0], acc[idx][1], a1, z[j].y); ++idx; }
    }
  };

#pragma unroll
  for (int d = 0; d < DEPTH - 1; ++d) load_batch(buf[d], wb[d]);
  for (int64_t rc = r0; rc < n; rc += DEPTH * S) {
#pragma unroll
    for (int d = 0; d < DEPTH; ++d) {
      load_batch(buf[(d + DEPTH - 1) % DEPTH], wb[(d + DEPTH - 1) % DEPTH]);
      multiply(buf[d], wb[d]);
    }
  }
  // ---- CTA reduction in a fixed order: warp 0 stores, warps 1..3 add one after the other ----
  for (int wturn = 0; wturn < 4; ++wturn) {
    if (warp == wturn) {
#pragma unroll
      for (int i = 0; i < NP; ++i) {
        double* d = sm + i * 64 + g * 8 + 2 * k;
        if (wturn == 0) { d[0] = acc[i][0]; d[1] = acc[i][1]; }
        else { d[0] += acc[i][0]; d[1] += acc[i][1]; }
      }
    }
    __syncthreads();
  }
  double* out = partials + (size_t)blockIdx.x * q1 * q1;
  for (int e = threadIdx.x; e < NP * 64; e += 128) {
    const int blk = e >> 6, rr = (e >> 3) & 7, cc = e & 7;
    int i = 0, rem = blk;
    while (rem >= NB - i) { rem -= NB - i; ++i; }
    const int j = i + rem;
    const int a = 8 * i + rr, b = 8 * j + cc;
    if (a < q1 && b < q1 && (i != j || a <= b)) {
      const double v = sm[e];
      out[(size_t)a * q1 + b] = v;
      out[(size_t)b * q1 + a] = v;
    }
  }
}

// Single-target variant of the wide kernel: only the FEATURE columns go through the tensor-core blocks (NB = ceil(p / 8));
// the products with y, the column sums and y'y / sum(y) / count are lane-local DFMAs on the same registers (a lane owns
// two rows of one column per block, and loads y / mask / weight for exactly those two rows — the 8 lanes that share k read
// the same 16 bytes).  p = 32 needs 10 block pairs instead of the 15 that [X | y | 1] = 34 -> 40 columns cost, p = 8 one
// instead of 3: the DMMA pipe (37 TFLOP/s measured) is the bound of this path, so the padding columns were the waste.
// AUX = weights and / or mask present (a missing one is loaded as ones).
// Rows = where the (y, weight) pair of a row comes from: LoadedRows reads both from memory; GlmRows<F> makes them one
// IRLS iteration of family F (K2a-GLM): y is the response, and per batch every lane forms its partial eta = x . beta
// over the feature blocks it holds (beta in NB registers), the 8 column lanes of a row pair add theirs up
// (shfl_xor 4 / 8 / 16), and the even column lanes evaluate the link for row .x, the odd ones for row .y; the weight
// w = 1 / (g'(mu)^2 V(mu)) and the working response z = eta + g'(mu) (y - mu) then take the places of (weight, y), so the
// kernel writes [X | z | 1]' diag(w) [X | z | 1] from ONE read of X and y.
struct LoadedRows { static constexpr bool kGlm = false; };
template <int F> struct GlmRows {
  static constexpr bool kGlm = true;
  static constexpr int family = F;
  const double* beta;   // p coefficients (+ the bias last when add_bias) of the current iterate; not read when `first`
  int add_bias;
  int first;            // first iteration: eta = g(mu_start(y)) instead of x . beta
  double mean_y;
};
template <typename T, int NB, int DEPTH, int MINB, bool AUX, typename Rows = LoadedRows>
__global__ void __launch_bounds__(128, MINB)
gram_dmma_side_kernel(const T* __restrict__ X, int64_t ldx, const T* __restrict__ y,
                      const T* __restrict__ w, const T* __restrict__ mask, int64_t n, int p,
                      double* __restrict__ partials /* [grid][(p+2)^2] */, Rows src) {
  constexpr bool WGT = AUX || Rows::kGlm;                 // products carry a per-row weight
  using V = typename Rows2<T>::V;
  constexpr int NP = NB * (NB + 1) / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sm = reinterpret_cast<double*>(smem_raw);      // [NP][64] blocks, then [NB * 8][2] (x.y, sum x), then 3 scalars
  double* sside = sm + NP * 64;
  double* sscal = sside + NB * 16;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, k = lane & 3;
  const int q1 = p + 2;
  const T* colp[NB];
  bool live[NB];
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    const int c = 8 * b + g;
    live[b] = c < p;
    colp[b] = X + (int64_t)(live[b] ? c : 0) * ldx;
  }
  double acc[NP][2];
#pragma unroll
  for (int i = 0; i < NP; ++i) { acc[i][0] = 0.0; acc[i][1] = 0.0; }
  double xy[NB], x1[NB], yy = 0.0, y1 = 0.0, c11 = 0.0;
#pragma unroll
  for (int b = 0; b < NB; ++b) { xy[b] = 0.0; x1[b] = 0.0; }
  double bet[NB], bias = 0.0;
  if constexpr (Rows::kGlm) {
#pragma unroll
    for (int b = 0; b < NB; ++b) bet[b] = (!src.first && live[b]) ? src.beta[8 * b + g] : 0.0;
    if (!src.first && src.add_bias) bias = src.beta[p];
  }

  struct Batch { V z[NB]; V y, w, m; };
  Batch ring[DEPTH];
  const int64_t S = (int64_t)gridDim.x * 4 * 8;
  const int64_t r0 = ((int64_t)blockIdx.x * 4 + warp) * 8;
  int64_t rl = r0 + 2 * k;
  const T* yp = y + rl;
  const T* wp = (AUX && w) ? w + rl : nullptr;
  const T* mp = (AUX && mask) ? mask + rl : nullptr;
#pragma unroll
  for (int b = 0; b < NB; ++b) colp[b] += rl;
  auto load_batch = [&](Batch& q) {                       // n is a multiple of 8 here: a batch is all in or all out
    const bool in = rl < n;
    const V zero = rows2_fill<V>(0.0f), one = rows2_fill<V>(1.0f);
    q.y = in ? __ldcs(reinterpret_cast<const V*>(yp)) : zero;
    yp += S;
    if constexpr (AUX) {
      q.w = in ? (wp ? __ldcs(reinterpret_cast<const V*>(wp)) : one) : zero;
      q.m = in ? (mp ? __ldcs(reinterpret_cast<const V*>(mp)) : one) : zero;
      if (wp) wp += S;
      if (mp) mp += S;
    } else {
      q.m = in ? one : zero;
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      q.z[b] = (in && live[b]) ? __ldcs(reinterpret_cast<const V*>(colp[b])) : zero;
      colp[b] += S;
    }
    rl += S;
  };
  auto multiply = [&](const Batch& q) {
    double2 z[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) z[b] = rows2_f64(q.z[b]);
    double2 yv = rows2_f64(q.y);
    const double2 mv = rows2_f64(q.m);
    double2 wv = make_double2(1.0, 1.0);
    if constexpr (AUX) wv = rows2_f64(q.w);
    if constexpr (Rows::kGlm) {
      constexpr int F = Rows::family;
      const bool odd = g & 1;                              // this lane evaluates row .y (odd g) or row .x (even g)
      const double yr = odd ? yv.y : yv.x;
      double eta, mu;
      if (src.first) {
        mu = glm::mu_start<F>(yr, src.mean_y);
        eta = glm::link<F>(mu);
      } else {
        double ex = 0.0, ey = 0.0;
#pragma unroll
        for (int b = 0; b < NB; ++b) { ex = fma(z[b].x, bet[b], ex); ey = fma(z[b].y, bet[b], ey); }
        // xor 4 pairs even and odd g: each keeps the sum of the row it evaluates, then the 4 lanes of its parity add up
        double e = (odd ? ey : ex) + __shfl_xor_sync(0xffffffffu, odd ? ex : ey, 4);
        e += __shfl_xor_sync(0xffffffffu, e, 8);
        e += __shfl_xor_sync(0xffffffffu, e, 16);
        eta = e + bias;
        mu = glm::inv<F>(eta);
      }
      double wr, zr;
      glm::irls_row<F>(eta, mu, yr, wr, zr);
      if (mv.x == 0.0) { wr = 0.0; zr = 0.0; }             // rows past n (a batch is all in or all out)
      const double wo = __shfl_xor_sync(0xffffffffu, wr, 4), zo = __shfl_xor_sync(0xffffffffu, zr, 4);
      wv = odd ? make_double2(wo, wr) : make_double2(wr, wo);
      yv = odd ? make_double2(zo, zr) : make_double2(zr, zo);
    }
    double2 wy, wm;                                        // w y, w m (the weight enters every product once)
    if constexpr (WGT) { wy = make_double2(wv.x * yv.x, wv.y * yv.y); wm = make_double2(wv.x * mv.x, wv.y * mv.y); }
    else { wy = yv; wm = mv; }
    yy = fma(wy.x, yv.x, fma(wy.y, yv.y, yy));
    y1 = fma(wy.x, mv.x, fma(wy.y, mv.y, y1));
    c11 = fma(wm.x, mv.x, fma(wm.y, mv.y, c11));
    // all block pairs for the even rows, then all for the odd rows: consecutive DMMAs never share an accumulator
    int idx = 0;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      xy[i] = fma(z[i].x, wy.x, xy[i]);
      x1[i] = fma(z[i].x, wm.x, x1[i]);
      const double a0 = WGT ? z[i].x * wv.x : z[i].x;
#pragma unroll
      for (int j = i; j < NB; ++j) { dmma884(acc[idx][0], acc[idx][1], a0, z[j].x); ++idx; }
    }
    idx = 0;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      xy[i] = fma(z[i].y, wy.y, xy[i]);
      x1[i] = fma(z[i].y, wm.y, x1[i]);
      const double a1 = WGT ? z[i].y * wv.y : z[i].y;
#pragma unroll
      for (int j = i; j < NB; ++j) { dmma884(acc[idx][0], acc[idx][1], a1, z[j].y); ++idx; }
    }
  };

#pragma unroll
  for (int d = 0; d < DEPTH - 1; ++d) load_batch(ring[d]);
  for (int64_t rc = r0; rc < n; rc += DEPTH * S) {
#pragma unroll
    for (int d = 0; d < DEPTH; ++d) {
      load_batch(ring[(d + DEPTH - 1) % DEPTH]);
      multiply(ring[d]);
    }
  }
  // lane-local sums -> warp sums over the 4 row slots (k); the y / count scalars are the same in all 8 column groups
#pragma unroll
  for (int off = 1; off <= 2; off <<= 1) {
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      xy[b] += __shfl_xor_sync(0xffffffffu, xy[b], off);
      x1[b] += __shfl_xor_sync(0xffffffffu, x1[b], off);
    }
    yy += __shfl_xor_sync(0xffffffffu, yy, off);
    y1 += __shfl_xor_sync(0xffffffffu, y1, off);
    c11 += __shfl_xor_sync(0xffffffffu, c11, off);
  }
  // ---- CTA reduction in a fixed order: warp 0 stores, warps 1..3 add one after the other ----
  for (int wturn = 0; wturn < 4; ++wturn) {
    if (warp == wturn) {
#pragma unroll
      for (int i = 0; i < NP; ++i) {
        double* d = sm + i * 64 + g * 8 + 2 * k;
        if (wturn == 0) { d[0] = acc[i][0]; d[1] = acc[i][1]; }
        else { d[0] += acc[i][0]; d[1] += acc[i][1]; }
      }
      if (k == 0) {
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          double* d = sside + (b * 8 + g) * 2;
          if (wturn == 0) { d[0] = xy[b]; d[1] = x1[b]; }
          else { d[0] += xy[b]; d[1] += x1[b]; }
        }
      }
      if (lane == 0) {
        if (wturn == 0) { sscal[0] = yy; sscal[1] = y1; sscal[2] = c11; }
        else { sscal[0] += yy; sscal[1] += y1; sscal[2] += c11; }
      }
    }
    __syncthreads();
  }
  double* out = partials + (size_t)blockIdx.x * q1 * q1;
  for (int e = threadIdx.x; e < NP * 64; e += 128) {
    const int blk = e >> 6, rr = (e >> 3) & 7, cc = e & 7;
    int i = 0, rem = blk;
    while (rem >= NB - i) { rem -= NB - i; ++i; }
    const int j = i + rem;
    const int a = 8 * i + rr, b = 8 * j + cc;
    if (a < p && b < p && (i != j || a <= b)) {
      const double v = sm[e];
      out[(size_t)a * q1 + b] = v;
      out[(size_t)b * q1 + a] = v;
    }
  }
  for (int c = threadIdx.x; c < p; c += 128) {
    const double vxy = sside[c * 2], vx1 = sside[c * 2 + 1];
    out[(size_t)c * q1 + p] = vxy;
    out[(size_t)p * q1 + c] = vxy;
    out[(size_t)c * q1 + p + 1] = vx1;
    out[(size_t)(p + 1) * q1 + c] = vx1;
  }
  if (threadIdx.x == 0) {
    out[(size_t)p * q1 + p] = sscal[0];
    out[(size_t)p * q1 + p + 1] = sscal[1];
    out[(size_t)(p + 1) * q1 + p] = sscal[1];
    out[(size_t)(p + 1) * q1 + p + 1] = sscal[2];
  }
}

// Ring depth per (kernel, AUX, NB): measured, not derived (profiles/r02/k2a_depth_sweep.txt, sweep build with every depth
// 2..9 instantiated under __launch_bounds__(128, 2), the number of resident CTAs following from the registers ptxas used).
// Two things decide: a spill inside the loop is expensive (p = 32: depth 4 with 234 registers and no spill 73 % of the
// HBM peak, depth 5 with a 16-byte spill 59 %), and for one or two blocks a shallow ring with more resident CTAs beats
// a deep one (p = 8: depth 2 93 %, depth 8 68 %).
constexpr int side_depth(int nb, bool aux) {
  constexpr int plain[8] = {2, 8, 6, 4, 3, 3, 2, 3}, auxd[8] = {2, 7, 5, 5, 2, 3, 2, 2};
  return aux ? auxd[nb - 1] : plain[nb - 1];
}
constexpr int wide_depth(int nb, bool aux) {
  constexpr int plain[8] = {2, 9, 2, 7, 4, 4, 3, 2}, auxd[8] = {7, 3, 9, 6, 5, 3, 3, 2};
  return aux ? auxd[nb - 1] : plain[nb - 1];
}

template <typename T, typename R = LoadedRows>
using SideFn = void (*)(const T*, int64_t, const T*, const T*, const T*, int64_t, int, double*, R);
template <typename T> using WideFn = void (*)(const T*, int64_t, const T*, int64_t, const T*, const T*, int64_t, int, int, double*);

#ifdef PDSB_K2A_SWEEP   // sweep build (profiles/_ab): every depth 2..9 is instantiated, PDSB_K2A_DEPTH picks one per call
static int k2a_sweep_depth() { const char* e = getenv("PDSB_K2A_DEPTH"); return e ? atoi(e) : 0; }
#define PDSB_DEPTH_CASES(KERNEL, NBV, AUXV)                                                                          \
  switch (k2a_sweep_depth()) {                                                                                       \
    case 2: return KERNEL<T, NBV, 2, 2, AUXV>; case 3: return KERNEL<T, NBV, 3, 2, AUXV>; case 4: return KERNEL<T, NBV, 4, 2, AUXV>; \
    case 5: return KERNEL<T, NBV, 5, 2, AUXV>; case 6: return KERNEL<T, NBV, 6, 2, AUXV>; case 7: return KERNEL<T, NBV, 7, 2, AUXV>; \
    case 8: return KERNEL<T, NBV, 8, 2, AUXV>; case 9: return KERNEL<T, NBV, 9, 2, AUXV>; default: break;                  \
  }
#else
#define PDSB_DEPTH_CASES(KERNEL, NBV, AUXV)
#endif

template <typename T, int NB, bool AUX> static SideFn<T> side_fn() {
  PDSB_DEPTH_CASES(gram_dmma_side_kernel, NB, AUX)
  return gram_dmma_side_kernel<T, NB, side_depth(NB, AUX), 2, AUX>;
}
template <typename T, int NB, bool AUX> static WideFn<T> wide_fn() {
  PDSB_DEPTH_CASES(gram_dmma_wide_kernel, NB, AUX)
  return gram_dmma_wide_kernel<T, NB, wide_depth(NB, AUX), 2, AUX>;
}
template <typename T> static SideFn<T> side_fn_rt(int nb, bool aux) {
  switch (nb) {
    case 1: return aux ? side_fn<T, 1, true>() : side_fn<T, 1, false>(); case 2: return aux ? side_fn<T, 2, true>() : side_fn<T, 2, false>();
    case 3: return aux ? side_fn<T, 3, true>() : side_fn<T, 3, false>(); case 4: return aux ? side_fn<T, 4, true>() : side_fn<T, 4, false>();
    case 5: return aux ? side_fn<T, 5, true>() : side_fn<T, 5, false>(); case 6: return aux ? side_fn<T, 6, true>() : side_fn<T, 6, false>();
    case 7: return aux ? side_fn<T, 7, true>() : side_fn<T, 7, false>(); default: return aux ? side_fn<T, 8, true>() : side_fn<T, 8, false>();
  }
}
template <typename T> static WideFn<T> wide_fn_rt(int nb, bool aux) {
  switch (nb) {
    case 1: return aux ? wide_fn<T, 1, true>() : wide_fn<T, 1, false>(); case 2: return aux ? wide_fn<T, 2, true>() : wide_fn<T, 2, false>();
    case 3: return aux ? wide_fn<T, 3, true>() : wide_fn<T, 3, false>(); case 4: return aux ? wide_fn<T, 4, true>() : wide_fn<T, 4, false>();
    case 5: return aux ? wide_fn<T, 5, true>() : wide_fn<T, 5, false>(); case 6: return aux ? wide_fn<T, 6, true>() : wide_fn<T, 6, false>();
    case 7: return aux ? wide_fn<T, 7, true>() : wide_fn<T, 7, false>(); default: return aux ? wide_fn<T, 8, true>() : wide_fn<T, 8, false>();
  }
}
#undef PDSB_DEPTH_CASES
// shared memory of the CTA-level reduction (both kernels): [NP][64] blocks + [NB * 8][2] side sums + scalars
static size_t ring_kernel_smem(int nb) { return (size_t)((nb * (nb + 1) / 2) * 64 + nb * 16 + 4) * sizeof(double); }

template <int NB>
static int launch_dmma(const double* X, int64_t ldx, const double* Y, int64_t ldy, const double* w, const double* mask,
                       int64_t n, int p, int t, int grid, double* partials, cudaStream_t s) {
  const size_t smem = (size_t)(NB * (NB + 1) / 2) * 64 * sizeof(double);
  gram_dmma_kernel<NB><<<grid, 256, smem, s>>>(X, ldx, Y, ldy, w, mask, n, p, t, partials);
  PDSB_LAUNCH_OK();
  count_launch();
  return 0;
}

// The last n % 8 rows of the wide / side kernels: one CTA, one thread per entry of the partial.
template <typename T>
__global__ void __launch_bounds__(128)
gram_rows_kernel(const T* __restrict__ X, int64_t ldx, const T* __restrict__ Y, int64_t ldy,
                 const T* __restrict__ w, const T* __restrict__ mask, int rows, int p, int t,
                 double* __restrict__ out /* [q1*q1] */) {
  const int q1 = p + t + 1;
  auto at = [&](int c, int r) -> double {
    if (c < p) return (double)X[(int64_t)c * ldx + r];
    if (c < p + t) return (double)Y[(int64_t)(c - p) * ldy + r];
    return mask ? (double)mask[r] : 1.0;
  };
  for (int e = threadIdx.x; e < q1 * q1; e += blockDim.x) {
    const int a = e / q1, b = e % q1;
    double v = 0.0;
    for (int r = 0; r < rows; ++r) v = fma(w ? (double)w[r] : 1.0, at(a, r) * at(b, r), v);   // a*b first: M stays symmetric bit for bit
    out[e] = v;
  }
}

#define PDSB_NB_SWITCH(NBEXPR, CALL)                                                                              \
  switch (NBEXPR) {                                                                                               \
    case 1: rc = CALL(1); break; case 2: rc = CALL(2); break; case 3: rc = CALL(3); break; case 4: rc = CALL(4); break; \
    case 5: rc = CALL(5); break; case 6: rc = CALL(6); break; case 7: rc = CALL(7); break; default: rc = CALL(8); break; \
  }

// 0 ok, 1 error, -1 not applicable (caller uses the DFMA kernel).  PDSB_K2A_DMMA=0 disables.
// Kernel choice (B200, profiles/r02/k2a_f64*.txt and k2a_depth_sweep.txt), % of the measured HBM peak for f64 frames with
// 8 / 16 / 24 / 32 / 48 / 62 features and one target:
//   direct (4-row steps, scalar loads)            30 / 26 /  - / 33 /  - / 24   <- unaligned columns only
//   wide   (8-row batches, 16-byte loads, ring)   several targets, or when side saves no block: 14 features 92, 30: 67, 62: 44
//   side   (wide + y, ones, weights on DFMAs)     93 / 79 / 78 / 73 / 52 /  -   <- one target and ceil(p / 8) < ceil((p + 2) / 8)
// (p = 63, 64: 21 %, the 8-block side kernel spills; the SIMT fallback measured 11 %.)
// Round-2 variants that lost and were removed: m16n8k8 blocks (26 % at 32 features), bulk-copy staged m8n8k4 (23 %), per-lane
// cp.async ring in shared memory (38 %).  ncu (profiles/r02/k2a_*_ncu_metrics.csv, before the depth sweep): DMMA pipe 54-63 %
// busy, DRAM 42-45 %, warps wait on the long scoreboard.
// PDSB_K2A_KERNEL=8 forces the direct kernel, =1 the wide one also for a single target.
template <typename T>
static int moments_dmma(const T* X, int64_t ldx, const T* Y, int64_t ldy, const T* w, const T* mask, int64_t n, int p,
                        int t, double* M, cudaStream_t s) {
  constexpr bool F64 = sizeof(T) == 8;
  static const bool enabled = [] { const char* e = getenv("PDSB_K2A_DMMA"); return !(e && e[0] == '0'); }();
  static const int kern = [] { const char* e = getenv("PDSB_K2A_KERNEL"); return e ? atoi(e) : 2; }();
  const int q1 = p + t + 1;
  const int nb = (q1 + 7) / 8, nbx = (p + 7) / 8;
  if (!enabled || n < 1) return -1;
  auto al2 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & (2 * sizeof(T) - 1)) == 0; };   // two rows per load
  const bool aligned = kern != 8 && n >= 8 && al2(X) && al2(Y) && (ldx % 2 == 0) && (ldy % 2 == 0) && (!w || al2(w)) &&
                       (!mask || al2(mask));
  const bool side = aligned && kern != 1 && t == 1 && nbx >= 1 && nbx <= 8 && nbx < nb;   // only when it saves a block
  const bool wide = aligned && !side && nb <= 8;
  if (!side && nb > 8) return -1;
  if (!F64 && !side && !wide) return -1;                 // f32 columns that are not 8-byte aligned: the SIMT kernel
  const int64_t n_main = (side || wide) ? n - n % 8 : 0;
  const int64_t n_tail = n - n_main;
  // resident CTAs of the chosen instantiation (128 threads): from the registers ptxas used for it
  SideFn<T> sfn = nullptr; WideFn<T> wfn = nullptr;
  int per_sm = 4;
  const size_t ring_smem = ring_kernel_smem(side ? nbx : nb);
  if (side) {
    sfn = side_fn_rt<T>(nbx, w || mask);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sfn, 128, ring_smem) != cudaSuccess || per_sm < 1) { (void)cudaGetLastError(); per_sm = 2; }
  } else if (wide) {
    wfn = wide_fn_rt<T>(nb, w != nullptr);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wfn, 128, ring_smem) != cudaSuccess || per_sm < 1) { (void)cudaGetLastError(); per_sm = 2; }
  }
  const int grid_main = n_main ? (int)std::min<int64_t>(ceil_div(n_main, 32), (int64_t)sm_count() * per_sm) : 0;
  int grid_tail = 0;
  if (n_tail > 0) grid_tail = n_main ? 1 : (int)std::min<int64_t>(ceil_div(n_tail, 32), (int64_t)sm_count() * 4);
  double* partials = nullptr;
  if (dev_alloc((void**)&partials, (size_t)(grid_main + grid_tail) * q1 * q1 * sizeof(double), s)) return 1;
  int rc = 0;
  if (side) {
    sfn<<<grid_main, 128, ring_smem, s>>>(X, ldx, Y, w, mask, n_main, p, partials, LoadedRows{});
    cudaError_t e = cudaGetLastError();
    count_launch();
    if (e != cudaSuccess) { set_error("gram_dmma_side launch failed: %s", cudaGetErrorString(e)); rc = 1; }
  } else if (wide) {
    wfn<<<grid_main, 128, ring_smem, s>>>(X, ldx, Y, ldy, w, mask, n_main, p, t, partials);
    cudaError_t e = cudaGetLastError();
    count_launch();
    if (e != cudaSuccess) { set_error("gram_dmma_wide launch failed: %s", cudaGetErrorString(e)); rc = 1; }
  }
  if (rc) { dev_free(partials, s); return rc; }
  if (grid_tail > 0) {
    const T* Xt = X + n_main; const T* Yt = Y + n_main;
    const T* wt = w ? w + n_main : nullptr; const T* mt = mask ? mask + n_main : nullptr;
    double* pt = partials + (size_t)grid_main * q1 * q1;
    if (n_main) {
      gram_rows_kernel<T><<<1, 128, 0, s>>>(Xt, ldx, Yt, ldy, wt, mt, (int)n_tail, p, t, pt);
      cudaError_t e = cudaGetLastError();
      count_launch();
      if (e != cudaSuccess) { set_error("gram_rows launch failed: %s", cudaGetErrorString(e)); rc = 1; }
    } else if constexpr (F64) {
#define PDSB_CALL(NBV) launch_dmma<NBV>(Xt, ldx, Yt, ldy, wt, mt, n_tail, p, t, grid_tail, pt, s)
      PDSB_NB_SWITCH(nb, PDSB_CALL)
#undef PDSB_CALL
    }
    if (rc) { dev_free(partials, s); return rc; }
  }
  const int len = q1 * q1;
  reduce_partials_kernel<<<len, 128, 0, s>>>(partials, grid_main + grid_tail, len, M);
  cudaError_t e = cudaGetLastError();
  count_launch();
  dev_free(partials, s);
  if (e != cudaSuccess) { set_error("reduce_partials launch failed: %s", cudaGetErrorString(e)); return 1; }
  return 0;
}
#undef PDSB_NB_SWITCH

template <typename T, int MAXT>
static int launch_gram(const T* X, int64_t ldx, const T* Y, int64_t ldy, const T* w, const T* mask,
                       int64_t n, int p, int t, int tile_r, int S, int grid, size_t smem, double* partials,
                       int64_t bstride, cudaStream_t s) {
  if (w) {
    auto k = gram_simt_kernel<T, MAXT, true>;
    PDSB_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, 256, smem, s>>>(X, ldx, Y, ldy, w, mask, n, p, t, tile_r, S, partials, bstride);
  } else {
    auto k = gram_simt_kernel<T, MAXT, false>;
    PDSB_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, 256, smem, s>>>(X, ldx, Y, ldy, w, mask, n, p, t, tile_r, S, partials, bstride);
  }
  PDSB_LAUNCH_OK();
  count_launch();
  return 0;
}

template <typename T>
int moments_simt(const T* X, int64_t ldx, const T* Y, int64_t ldy, const T* w, const T* mask, int64_t n,
                 int p, int t, double* M, cudaStream_t s, int64_t bstride) {
  const int q1 = p + t + 1;
  if (p < 0 || t < 0 || q1 > 260) { set_error("moments: p+t+1=%d out of range (max 260)", q1); return 1; }
  if (bstride == 0) {        // column-major: FP64 tensor-core path for up to 64 columns (f32 columns are widened on the fly)
    const int rc = moments_dmma<T>(X, ldx, Y, ldy, w, mask, n, p, t, M, s);
    if (rc >= 0) return rc;
  }
  const int nt = (q1 + 3) / 4, ntp = nt * (nt + 1) / 2;
  const int maxt = (ntp + 255) / 256;
  const int S = nt * 4;  // row stride, multiple of 4 elements
  // tile rows: keep the tile under ~64 KB
  int tile_r = 128;
  while (tile_r > 16 && (size_t)tile_r * (S + 1) * sizeof(T) > 64 * 1024) tile_r >>= 1;
  size_t smem = (size_t)tile_r * (S + 1) * sizeof(T);
  int64_t ntiles = ceil_div(n > 0 ? n : 1, tile_r);
  // persistent grid: as many CTAs per SM as registers / shared memory allow (load and FMA phases of different CTAs overlap)
  int per_sm = 2;
  {
    int occ = 0;
    cudaError_t oe = cudaSuccess;
    if (maxt == 1) {
      if (w) oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gram_simt_kernel<T, 1, true>, 256, smem);
      else oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gram_simt_kernel<T, 1, false>, 256, smem);
      if (oe == cudaSuccess && occ >= 1) per_sm = std::min(occ, 4);
      else (void)cudaGetLastError();
    }
  }
  int grid = (int)std::min<int64_t>(ntiles, (int64_t)sm_count() * per_sm);
  if (grid < 1) grid = 1;
  const int nslices = (maxt == 1) ? 256 / ntp : 1;      // must match the kernel's decode
  const int nparts = grid * nslices;
  double* partials = nullptr;
  if (dev_alloc((void**)&partials, (size_t)nparts * q1 * q1 * sizeof(double), s)) return 1;
  int rc;
  switch (maxt) {
    case 1: rc = launch_gram<T, 1>(X, ldx, Y, ldy, w, mask, n, p, t, tile_r, S, grid, smem, partials, bstride, s); break;
    case 2: rc = launch_gram<T, 2>(X, ldx, Y, ldy, w, mask, n, p, t, tile_r, S, grid, smem, partials, bstride, s); break;
    case 3: case 4: rc = launch_gram<T, 4>(X, ldx, Y, ldy, w, mask, n, p, t, tile_r, S, grid, smem, partials, bstride, s); break;
    default: rc = launch_gram<T, 9>(X, ldx, Y, ldy, w, mask, n, p, t, tile_r, S, grid, smem, partials, bstride, s); break;
  }
  if (rc) { dev_free(partials, s); return rc; }
  int len = q1 * q1;
  reduce_partials_kernel<<<len, 128, 0, s>>>(partials, nparts, len, M);
  cudaError_t e = cudaGetLastError();
  count_launch();
  dev_free(partials, s);
  if (e != cudaSuccess) { set_error("reduce_partials launch failed: %s", cudaGetErrorString(e)); return 1; }
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// K2a-GLM: the moments of one IRLS iteration, [X | z | 1]' diag(w) [X | z | 1] with (w, z) computed from (X, y, beta)
// on the fly — the side kernel with GlmRows<F> for the rows n - n % 8, glm_rows_kernel for the rest.  X: column-major,
// 16-byte aligned columns, even ldx; y 16-byte aligned (the caller checks).
//
// Ring depth per NB: the plain side kernel's depth where that compiles without a spill, shallower where beta's NB
// registers would push it into one (ptxas -v, sm_100a).
constexpr int glm_depth(int nb) {
  constexpr int d[8] = {2, 8, 6, 3, 2, 2, 2, 2};
  return d[nb - 1];
}
template <int F, int NB> static SideFn<double, GlmRows<F>> glm_fn() {
  return gram_dmma_side_kernel<double, NB, glm_depth(NB), 2, false, GlmRows<F>>;
}
template <int F> static SideFn<double, GlmRows<F>> glm_fn_rt(int nb) {
  switch (nb) {
    case 1: return glm_fn<F, 1>(); case 2: return glm_fn<F, 2>(); case 3: return glm_fn<F, 3>(); case 4: return glm_fn<F, 4>();
    case 5: return glm_fn<F, 5>(); case 6: return glm_fn<F, 6>(); case 7: return glm_fn<F, 7>(); default: return glm_fn<F, 8>();
  }
}

// The last n % 8 (< 8) rows: one CTA; (w, z) of each row first, then one thread per entry of the partial, in
// gram_rows_kernel's order.
template <int F>
__global__ void __launch_bounds__(128)
glm_rows_kernel(const double* __restrict__ X, int64_t ldx, const double* __restrict__ y, int rows, int p, GlmRows<F> src,
                double* __restrict__ out /* [(p+2)^2] */) {
  __shared__ double sw[8], sz[8];
  const int q1 = p + 2;
  if ((int)threadIdx.x < rows) {
    const int r = threadIdx.x;
    double eta, mu;
    if (src.first) {
      mu = glm::mu_start<F>(y[r], src.mean_y);
      eta = glm::link<F>(mu);
    } else {
      eta = 0.0;
      for (int c = 0; c < p; ++c) eta = fma(X[(int64_t)c * ldx + r], src.beta[c], eta);
      if (src.add_bias) eta += src.beta[p];
      mu = glm::inv<F>(eta);
    }
    glm::irls_row<F>(eta, mu, y[r], sw[r], sz[r]);
  }
  __syncthreads();
  auto at = [&](int c, int r) -> double { return c < p ? X[(int64_t)c * ldx + r] : (c == p ? sz[r] : 1.0); };
  for (int e = threadIdx.x; e < q1 * q1; e += blockDim.x) {
    const int a = e / q1, b = e % q1;
    double v = 0.0;
    for (int r = 0; r < rows; ++r) v = fma(sw[r], at(a, r) * at(b, r), v);
    out[e] = v;
  }
}

template <int F>
static int glm_moments_t(const double* X, int64_t ldx, const double* y, int64_t n, int p, int add_bias, const double* beta,
                         int first, double mean_y, double* M, cudaStream_t s) {
  const int q1 = p + 2;
  const GlmRows<F> src{beta, add_bias, first, mean_y};
  const int64_t n_main = n - n % 8, n_tail = n - n_main;
  SideFn<double, GlmRows<F>> fn = glm_fn_rt<F>((p + 7) / 8);
  const size_t ring_smem = ring_kernel_smem((p + 7) / 8);
  int per_sm = 2;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, 128, ring_smem) != cudaSuccess || per_sm < 1) {
    (void)cudaGetLastError();
    per_sm = 2;
  }
  const int grid_main = n_main ? (int)std::min<int64_t>(ceil_div(n_main, 32), (int64_t)sm_count() * per_sm) : 0;
  const int nparts = grid_main + (n_tail > 0 ? 1 : 0);
  double* partials = nullptr;
  if (dev_alloc((void**)&partials, (size_t)nparts * q1 * q1 * sizeof(double), s)) return 1;
  cudaError_t e = cudaSuccess;
  if (grid_main) {
    fn<<<grid_main, 128, ring_smem, s>>>(X, ldx, y, nullptr, nullptr, n_main, p, partials, src);
    e = cudaGetLastError();
    count_launch();
  }
  if (e == cudaSuccess && n_tail) {
    glm_rows_kernel<F><<<1, 128, 0, s>>>(X + n_main, ldx, y + n_main, (int)n_tail, p, src,
                                         partials + (size_t)grid_main * q1 * q1);
    e = cudaGetLastError();
    count_launch();
  }
  if (e == cudaSuccess) {
    reduce_partials_kernel<<<q1 * q1, 128, 0, s>>>(partials, nparts, q1 * q1, M);
    e = cudaGetLastError();
    count_launch();
  }
  dev_free(partials, s);
  if (e != cudaSuccess) { set_error("glm moments launch failed: %s", cudaGetErrorString(e)); return 1; }
  return 0;
}

int glm_moments(const double* X, int64_t ldx, const double* y, int64_t n, int p, int add_bias, int family,
                const double* beta, int first, double mean_y, double* M, cudaStream_t s) {
  if (p < 1 || p > 64) { set_error("glm: %d features are not supported (1..64)", p); return 1; }
  switch (family) {
    case glm::GAUSSIAN: return glm_moments_t<glm::GAUSSIAN>(X, ldx, y, n, p, add_bias, beta, first, mean_y, M, s);
    case glm::POISSON: return glm_moments_t<glm::POISSON>(X, ldx, y, n, p, add_bias, beta, first, mean_y, M, s);
    case glm::BINOMIAL: return glm_moments_t<glm::BINOMIAL>(X, ldx, y, n, p, add_bias, beta, first, mean_y, M, s);
    case glm::GAMMA: return glm_moments_t<glm::GAMMA>(X, ldx, y, n, p, add_bias, beta, first, mean_y, M, s);
    default: set_error("glm: unknown family %d", family); return 1;
  }
}

template int moments_simt<float>(const float*, int64_t, const float*, int64_t, const float*, const float*,
                                 int64_t, int, int, double*, cudaStream_t, int64_t);
template int moments_simt<double>(const double*, int64_t, const double*, int64_t, const double*, const double*,
                                  int64_t, int, int, double*, cudaStream_t, int64_t);

}  // namespace pdsb
