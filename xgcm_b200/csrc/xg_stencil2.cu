// xg_stencil2 — fused halo-pad + 2-point stencil + metric multiply/divide.
//
// Replaces, in ONE pass over HBM (read n, write n):
//   xgcm/padding.py:575-616   np.pad copy of the whole field
//   xgcm/gridops.py:23-24,76-77,123-126,172-175   the pairwise operator
//   xgcm/grid.py:806-808,830-832,1576-1578        metric multiply / divide
//
// Any C-contiguous field collapses to (outer, n, inner) around the operated
// axis.  Three kernels:
//   k_stencil_strided  inner > 1 (Y, Z, ...): a warp owns 32 x VEC contiguous
//       columns and marches J cells along the axis keeping the previous row in
//       registers, so each input element is read once; U independent 16-byte
//       loads are in flight per thread.
//   k_stencil_row_vec  inner == 1 (X), aligned rows, n_out == n: a warp owns a
//       512 B x U chunk of one row, the missing neighbour of each 16-byte
//       vector comes from a warp shuffle, and only the chunk edge does one
//       extra scalar load (or takes the boundary value).
//   k_stencil_row_scalar  inner == 1, any length / alignment / n_out != n.
//
// Roofline: HBM.  Algorithmic bytes = 2 * sizeof(T) per output cell
// (+ metric bytes), see DESIGN.md.
#include <stdlib.h>

#include "xg_common.cuh"
#include "xg_stencil_tile.cuh"
#include "xg_tma.cuh"

namespace {

template <typename T>
struct StencilArgs {
  const T* in;
  T* out;
  int64_t outer, n, inner, n_out;
  int64_t nx_last;     // extent of the innermost dim (inner is a multiple of it when inner > 1)
  int lo, hi, bc;
  T fill;
  int J;               // cells marched per warp-unit (strided kernel)
  int64_t nseg, nwc;   // segments along the axis, warp-columns (or row chunks)
  int64_t nunits;      // total warp-units
  bool small_units;    // nunits < 2^31: 32-bit unit decomposition
  XgFastDiv fd_nseg, fd_nwc;  // multiply-high forms of nseg / nwc (valid with small_units)
  bool seg_fast;       // unit order: segment index fastest (else warp-column fastest)
  XgOperand pre, post;
  int pre_axis_vec_ok, post_axis_vec_ok;  // row kernels: metric vector loads along x
  const T* halo_lo;
  const T* halo_hi;
};

constexpr int kThreads = 256;
constexpr int kWarpsPerBlock = kThreads / 32;

// ---------------------------------------------------------------------------
// strided-axis kernel
// ---------------------------------------------------------------------------
template <typename T, int VEC, int OP, bool MET, int U, int MINB = 4>
__global__ void __launch_bounds__(kThreads, MINB)  // MINB = 4: <= 64 registers, 4 CTAs (1024 threads) per SM
k_stencil_strided(const StencilArgs<T> a) {
  typedef XgPack<T, VEC> Pack;
  const int64_t unit =
      (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (unit >= a.nunits) return;
  const int lane = threadIdx.x & 31;
  int64_t wc, t, seg, o;
  if (a.seg_fast) {  // segments of one column group adjacent in launch order
    xg_divmod(unit, a.nseg, a.fd_nseg, a.small_units, t, seg);
    xg_divmod(t, a.nwc, a.fd_nwc, a.small_units, o, wc);
  } else {
    xg_divmod(unit, a.nwc, a.fd_nwc, a.small_units, t, wc);
    xg_divmod(t, a.nseg, a.fd_nseg, a.small_units, o, seg);
  }
  const int64_t i = (wc * 32 + lane) * VEC;
  if (i >= a.inner) return;

  const int64_t j0 = seg * a.J;
  const int64_t j1 = (j0 + a.J < a.n_out) ? (j0 + a.J) : a.n_out;

  const T* ibase = a.in + o * a.n * a.inner + i;
  T* obase = a.out + o * a.n_out * a.inner + i;
  const bool has_pre = MET && a.pre.ptr != nullptr;
  const bool has_post = MET && a.post.ptr != nullptr;
  XgOperandView<T, VEC> pre_v, post_v;
  if (MET) {
    // everything that depends only on (o, i) is hoisted out of the march
    if (has_pre) pre_v = xg_operand_view<T, VEC>(a.pre, xg_groups_offset(a.pre.outer, o), i);
    if (has_post) post_v = xg_operand_view<T, VEC>(a.post, xg_groups_offset(a.post.outer, o), i);
  }

  // A[s] = in[s] * pre[s], s in range
  auto loadA = [&](int64_t s) -> Pack {
    Pack v = xg_ld_stream<T, VEC>(ibase + s * a.inner);
    if (has_pre) {
      Pack m = xg_ld_view<T, VEC>(pre_v, s * a.pre.axis_stride);
#pragma unroll
      for (int k = 0; k < VEC; ++k) v.v[k] = v.v[k] * m.v[k];
    }
    return v;
  };
  auto emit = [&](int64_t j, const Pack& lo_v, const Pack& hi_v) {
    Pack r;
#pragma unroll
    for (int k = 0; k < VEC; ++k) r.v[k] = xg_apply_op<T, OP>(lo_v.v[k], hi_v.v[k]);
    if (has_post) {
      if (sizeof(T) == 4 && post_v.mode == XG_IM_BCAST) {
        // dz(Z) against a (Z, Y, X) field: one divisor for the whole vector, inverted once
        XgSharedDivisor<T> d;
        d.set(__ldg(post_v.p0 + j * a.post.axis_stride));
#pragma unroll
        for (int k = 0; k < VEC; ++k) r.v[k] = d.div(r.v[k]);
      } else {
        Pack m = xg_ld_view<T, VEC>(post_v, j * a.post.axis_stride);
#pragma unroll
        for (int k = 0; k < VEC; ++k) r.v[k] = r.v[k] / m.v[k];
      }
    }
    xg_st_stream<T, VEC>(obase + j * a.inner, r);
  };

  // P[k] with the boundary rule; only ever needed for the first row of the first segment
  // (s = -1) and the last row of the last segment (s = n)
  auto loadP = [&](int64_t k) -> Pack {
    int64_t s = k - a.lo;
    if (s >= 0 && s < a.n) return loadA(s);
    const bool low = s < 0;
    const T* halo = low ? a.halo_lo : a.halo_hi;
    Pack r;
    if (halo) return xg_ld_cached<T, VEC>(halo + o * a.inner + i);
    if (a.bc == XG_BC_FILL) {
#pragma unroll
      for (int k2 = 0; k2 < VEC; ++k2) r.v[k2] = a.fill;
      return r;
    }
    if (a.bc == XG_BC_PERIODIC) return loadA(low ? s + a.n : s - a.n);
    if (a.bc == XG_BC_EXTEND) return loadA(low ? 0 : a.n - 1);
    // extrapolate: 2*A[edge] - A[next]
    const int64_t e = low ? 0 : a.n - 1;
    const int64_t e2 = a.n > 1 ? (low ? 1 : a.n - 2) : e;
    Pack a0 = loadA(e), a1 = loadA(e2);
#pragma unroll
    for (int q = 0; q < VEC; ++q) r.v[q] = T(2) * a0.v[q] - a1.v[q];
    return r;
  };

  // Row j needs P[j] (carried in registers) and P[j+1] = A[j+1-lo].  Since lo <= 1 the source
  // index j+1-lo is never negative; it is in range while j < n+lo-1.  So the whole march is the
  // branch-free unrolled loop, plus one boundary-aware load at each end.
  Pack prev = loadP(j0);
  const int64_t jm = (j1 < a.n + a.lo - 1) ? j1 : (a.n + a.lo - 1);
  int64_t j = j0;
  for (; j + U <= jm; j += U) {
    Pack cur[U];
#pragma unroll
    for (int u = 0; u < U; ++u) cur[u] = loadA(j + u + 1 - a.lo);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      emit(j + u, prev, cur[u]);  // (hoisting the divisor loads here was measured slower: it costs
      prev = cur[u];              //  16 registers, i.e. one resident CTA per SM)
    }
  }
  for (; j < jm; ++j) {
    Pack cur = loadA(j + 1 - a.lo);
    emit(j, prev, cur);
    prev = cur;
  }
#pragma unroll 1
  for (; j < j1; ++j) {  // at most one row: the upper halo
    Pack cur = loadP(j + 1);
    emit(j, prev, cur);
    prev = cur;
  }
}

// ---------------------------------------------------------------------------
// row kernels (operated axis is the innermost one)
// ---------------------------------------------------------------------------

// scalar A[r, s] = in * pre and the boundary values of row r
template <typename T, bool MET>
struct RowAccess {
  const StencilArgs<T>& a;
  const T* row;
  int64_t r;
  int64_t pre_base;
  __device__ __forceinline__ RowAccess(const StencilArgs<T>& a_, int64_t r_)
      : a(a_), row(a_.in + r_ * a_.n), r(r_), pre_base(0) {
    if (MET && a.pre.ptr) pre_base = xg_groups_offset(a.pre.outer, r);
  }
  __device__ __forceinline__ T A(int64_t s) const {
    T v = __ldg(row + s);
    if (MET && a.pre.ptr)
      v = v * __ldg(reinterpret_cast<const T*>(a.pre.ptr) + pre_base +
                    s * a.pre.axis_stride);
    return v;
  }
  __device__ __forceinline__ T below() const {  // P at s = -1
    if (a.halo_lo) return __ldg(a.halo_lo + r);
    if (a.bc == XG_BC_FILL) return a.fill;
    if (a.bc == XG_BC_PERIODIC) return A(a.n - 1);
    if (a.bc == XG_BC_EXTEND) return A(0);
    return T(2) * A(0) - A(a.n > 1 ? 1 : 0);
  }
  __device__ __forceinline__ T above() const {  // P at s = n
    if (a.halo_hi) return __ldg(a.halo_hi + r);
    if (a.bc == XG_BC_FILL) return a.fill;
    if (a.bc == XG_BC_PERIODIC) return A(0);
    if (a.bc == XG_BC_EXTEND) return A(a.n - 1);
    return T(2) * A(a.n - 1) - A(a.n > 1 ? a.n - 2 : 0);
  }
  __device__ __forceinline__ T P(int64_t k) const {
    int64_t s = k - a.lo;
    if (s < 0) return below();
    if (s >= a.n) return above();
    return A(s);
  }
};

template <typename T, int OP, bool MET>
__global__ void __launch_bounds__(kThreads)
k_stencil_row_scalar(const StencilArgs<T> a) {
  const int64_t total = a.outer * a.n_out;
  for (int64_t g = (int64_t)blockIdx.x * kThreads + threadIdx.x; g < total;
       g += (int64_t)gridDim.x * kThreads) {
    const int64_t r = g / a.n_out;
    const int64_t xo = g - r * a.n_out;
    RowAccess<T, MET> ra(a, r);
    T lo_v = ra.P(xo);
    T hi_v = ra.P(xo + 1);
    T res = xg_apply_op<T, OP>(lo_v, hi_v);
    if (MET && a.post.ptr) {
      int64_t pb = xg_groups_offset(a.post.outer, r);
      res = res / __ldg(reinterpret_cast<const T*>(a.post.ptr) + pb +
                        xo * a.post.axis_stride);
    }
    a.out[g] = res;
  }
}

// metric values for the VEC elements starting at x0 of a row
template <typename T, int VEC>
__device__ __forceinline__ XgPack<T, VEC> row_metric(const XgOperand& m,
                                                    int64_t base, int64_t x0,
                                                    int vec_ok) {
  const T* p = reinterpret_cast<const T*>(m.ptr) + base;
  XgPack<T, VEC> r;
  if (m.axis_stride == 0) {
    T s = __ldg(p);
#pragma unroll
    for (int k = 0; k < VEC; ++k) r.v[k] = s;
  } else if (vec_ok) {
    r = xg_ld_cached<T, VEC>(p + x0);
  } else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) r.v[k] = __ldg(p + (x0 + k) * m.axis_stride);
  }
  return r;
}

template <typename T, int VEC, int OP, bool MET, int U>
__global__ void __launch_bounds__(kThreads)
k_stencil_row_vec(const StencilArgs<T> a) {
  typedef XgPack<T, VEC> Pack;
  const unsigned FULL = 0xffffffffu;
  const int64_t unit =
      (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (unit >= a.nunits) return;  // warp-uniform
  const int lane = threadIdx.x & 31;
  int64_t c, r;
  xg_divmod(unit, a.nwc, a.fd_nwc, a.small_units, r, c);
  const int64_t nv = a.n / VEC;
  RowAccess<T, MET> ra(a, r);
  T* orow = a.out + r * a.n;  // n_out == n
  int64_t post_base = 0;
  if (MET && a.post.ptr) post_base = xg_groups_offset(a.post.outer, r);

  Pack v[U], pm[U];
  bool act[U];
  int64_t x0[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int64_t q = (c * U + u) * 32 + lane;
    act[u] = q < nv;
    x0[u] = q * VEC;
    if (act[u]) {
      v[u] = xg_ld_stream<T, VEC>(ra.row + x0[u]);
      // the divisor is fetched together with the field so its latency overlaps the field's
      if (MET && a.post.ptr) pm[u] = row_metric<T, VEC>(a.post, post_base, x0[u], a.post_axis_vec_ok);
      if (MET && a.pre.ptr) {
        Pack m = row_metric<T, VEC>(a.pre, ra.pre_base, x0[u], a.pre_axis_vec_ok);
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[u].v[k] = v[u].v[k] * m.v[k];
      }
    } else {
#pragma unroll
      for (int k = 0; k < VEC; ++k) v[u].v[k] = T(0);
    }
  }

#pragma unroll
  for (int u = 0; u < U; ++u) {
    Pack res;
    if (a.lo == 1) {
      // out[x] = OP(A[x-1], A[x])
      T left = __shfl_up_sync(FULL, v[u].v[VEC - 1], 1);
      T wrap = (u > 0) ? __shfl_sync(FULL, v[u > 0 ? u - 1 : 0].v[VEC - 1], 31) : T(0);
      if (lane == 0 && act[u]) {
        if (x0[u] == 0) left = ra.below();
        else if (u > 0) left = wrap;
        else left = ra.A(x0[u] - 1);
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k)
        res.v[k] = xg_apply_op<T, OP>(k == 0 ? left : v[u].v[k > 0 ? k - 1 : 0], v[u].v[k]);
    } else {
      // out[x] = OP(A[x], A[x+1])
      T right = __shfl_down_sync(FULL, v[u].v[0], 1);
      T wrap = (u < U - 1) ? __shfl_sync(FULL, v[u < U - 1 ? u + 1 : u].v[0], 0) : T(0);
      if (act[u]) {
        if (x0[u] + VEC >= a.n) right = ra.above();
        else if (lane == 31) right = (u < U - 1) ? wrap : ra.A(x0[u] + VEC);
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k)
        res.v[k] = xg_apply_op<T, OP>(v[u].v[k], k == VEC - 1 ? right : v[u].v[k < VEC - 1 ? k + 1 : k]);
    }
    if (act[u]) {
      if (MET && a.post.ptr) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) res.v[k] = res.v[k] / pm[u].v[k];
      }
      xg_st_stream<T, VEC>(orow + x0[u], res);
    }
  }
}

// ---------------------------------------------------------------------------
// row kernel, divisor shared between levels ("z-batched")
// ---------------------------------------------------------------------------
// derivative('X') on a (Z, Y, X) field divides by dx(Y, X): the same divisor for every level.
// Here a warp owns one 512-byte chunk of a row at U consecutive LEVELS (rows r, r + P, ...,
// P = rows per level), so the divisor vector is loaded and inverted once and each of the U x VEC
// cells costs a multiply instead of an 11-instruction IEEE division (XgSharedDivisor keeps the
// quotient bit-identical).  Loads in flight per thread: U field vectors + one metric vector, as
// in k_stencil_row_vec; the unit decomposition is three multiply-high divisions.
template <typename T>
struct RowZbArgs {
  const T* in;
  T* out;
  int64_t n;       // row length (n_out == n)
  int64_t P, Zn;   // row r = z * P + p; the post metric depends on p only
  int lo, bc;      // hi == 1 - lo
  T fill;
  const T* halo_lo;
  const T* halo_hi;
  XgOperand pre, post;
  int pre_vec;     // pre: 16-byte loads along x are aligned
  int pre_shared;  // pre: also independent of z
  int64_t nwc, nunits;
  XgFastDiv fd_nwc, fd_P;
  bool small_units;
};

template <typename T, int VEC, int OP, int U>
__global__ void __launch_bounds__(kThreads) k_stencil_row_zb(const RowZbArgs<T> a) {
  typedef XgPack<T, VEC> Pack;
  const unsigned FULL = 0xffffffffu;
  const int64_t unit = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (unit >= a.nunits) return;  // warp-uniform
  const int lane = threadIdx.x & 31;
  int64_t c, t, p, zq;
  xg_divmod(unit, a.nwc, a.fd_nwc, a.small_units, t, c);
  xg_divmod(t, a.P, a.fd_P, a.small_units, zq, p);
  const int64_t z0 = zq * U;
  const int nz = (a.Zn - z0 < U) ? (int)(a.Zn - z0) : U;
  const int64_t nv = a.n / VEC;
  const int64_t q = c * 32 + lane;
  const bool act = q < nv;
  // spare lanes of the last chunk shadow the row's last vector: they stay in the shuffles and
  // hold valid addresses, but never store
  const int64_t x0 = (act ? q : nv - 1) * VEC;
  const int64_t row0 = z0 * a.P + p;
  const int64_t zstride = a.P * a.n;
  const T* ip = a.in + row0 * a.n;
  T* op = a.out + row0 * a.n + x0;
  const bool has_pre = a.pre.ptr != nullptr;
  const T* prep = reinterpret_cast<const T*>(a.pre.ptr);

  Pack v[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (u < nz) {
      v[u] = xg_ld_stream<T, VEC>(ip + u * zstride + x0);
    } else {
#pragma unroll
      for (int k = 0; k < VEC; ++k) v[u].v[k] = T(0);
    }
  }
  const Pack pm = xg_ld_cached<T, VEC>(reinterpret_cast<const T*>(a.post.ptr) +
                                       xg_groups_offset(a.post.outer, p) + x0);
  int64_t pre_off[U];
  if (has_pre) {
#pragma unroll
    for (int u = 0; u < U; ++u)
      pre_off[u] = (u == 0 || !a.pre_shared) ? xg_groups_offset(a.pre.outer, row0 + (u < nz ? u : 0) * a.P)
                                             : pre_off[0];
    Pack m;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (u < nz) {
        if (u == 0 || !a.pre_shared) {
          const T* pp = prep + pre_off[u];
          if (a.pre.axis_stride == 0) {
            const T sc = __ldg(pp);
#pragma unroll
            for (int k = 0; k < VEC; ++k) m.v[k] = sc;
          } else if (a.pre_vec) {
            m = xg_ld_cached<T, VEC>(pp + x0);
          } else {
#pragma unroll
            for (int k = 0; k < VEC; ++k) m.v[k] = __ldg(pp + (x0 + k) * a.pre.axis_stride);
          }
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[u].v[k] = v[u].v[k] * m.v[k];
      }
    }
  }
  // A[row u, s] = in * pre for the single elements the shuffles cannot provide
  auto A = [&](int u, int64_t s) -> T {
    T val = __ldg(ip + u * zstride + s);
    if (has_pre) val = val * __ldg(prep + pre_off[u] + s * a.pre.axis_stride);
    return val;
  };

  XgSharedDivisor<T> dv[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) dv[k].set(pm.v[k]);

#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (u >= nz) break;  // warp-uniform
    Pack res;
    if (a.lo == 1) {
      // out[x] = OP(A[x-1], A[x]); lane 0 has no lower lane to ask
      T nb = __shfl_up_sync(FULL, v[u].v[VEC - 1], 1);
      if (lane == 0) {
        if (c != 0) nb = A(u, x0 - 1);
        else if (a.halo_lo) nb = __ldg(a.halo_lo + row0 + u * a.P);
        else if (a.bc == XG_BC_FILL) nb = a.fill;
        else if (a.bc == XG_BC_PERIODIC) nb = A(u, a.n - 1);
        else if (a.bc == XG_BC_EXTEND) nb = v[u].v[0];
        else nb = T(2) * v[u].v[0] - v[u].v[1];
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k)
        res.v[k] = xg_apply_op<T, OP>(k == 0 ? nb : v[u].v[k > 0 ? k - 1 : 0], v[u].v[k]);
    } else {
      // out[x] = OP(A[x], A[x+1]); the row's last vector takes the upper boundary value
      T nb = __shfl_down_sync(FULL, v[u].v[0], 1);
      if (x0 + VEC >= a.n) {
        if (a.halo_hi) nb = __ldg(a.halo_hi + row0 + u * a.P);
        else if (a.bc == XG_BC_FILL) nb = a.fill;
        else if (a.bc == XG_BC_PERIODIC) nb = A(u, 0);
        else if (a.bc == XG_BC_EXTEND) nb = v[u].v[VEC - 1];
        else nb = T(2) * v[u].v[VEC - 1] - v[u].v[VEC - 2];
      } else if (lane == 31) {
        nb = A(u, x0 + VEC);
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k)
        res.v[k] = xg_apply_op<T, OP>(v[u].v[k], k == VEC - 1 ? nb : v[u].v[k < VEC - 1 ? k + 1 : k]);
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) res.v[k] = dv[k].div(res.v[k]);
    if (act) xg_st_stream<T, VEC>(op + u * zstride, res);
  }
}

// ---------------------------------------------------------------------------
// row kernel, divisor shared between levels, TMA-staged ("row_tma")
// ---------------------------------------------------------------------------
// Same decomposition as k_stencil_row_zb (U levels share one divisor row), but the operands arrive by
// bulk-async tensor loads: a tile is U levels x TY rows x TXE cells (+ one 16-byte halo vector), one
// cp.async.bulk.tensor box per operand, all boxes of a tile completing on one mbarrier.  A persistent
// CTA = 8 consumer warps + 1 producer warp around a ring of NST tiles (full / empty mbarriers, no
// block-wide barrier in the loop): shared memory, not registers, holds the bytes in flight.  Threads
// read 16-byte vectors from the tile, the neighbour element comes from a warp shuffle (the warp's
// edge lane reads it from the tile), results leave as streaming 16-byte stores.  TXE is a multiple of
// 128 bytes so stores of neighbouring tiles never share a sector.
// Tile order: row blocks of ~128 rows outermost, then the level batches, so the divisor rows of a
// block (~2 MB) are re-read from L2, not from DRAM, by each of the Zn / U level batches.
template <typename T>
struct RowTmaGeo;
template <>
struct RowTmaGeo<float> {
  static constexpr int VEC = 4, TXE = 224, TY = 4;  // 56 vectors per row, 64 thread slots
};
template <>
struct RowTmaGeo<double> {
  static constexpr int VEC = 2, TXE = 240, TY = 2;  // 120 vectors per row, 128 thread slots
};
enum { XG_PRE_NONE = 0, XG_PRE_FULL = 1, XG_PRE_SHARED = 2, XG_PRE_SCALAR = 3 };
constexpr int kTmaConsumers = kThreads;  // + one producer warp

template <typename T>
struct RowTmaArgs {
  const T* in;
  T* out;
  int64_t n, P, Zn;
  int bc;
  T fill;
  const T* halo_lo;
  const T* halo_hi;
  XgOperand pre;      // boundary elements and the per-row scalar mode
  int pre_mode;       // XG_PRE_*
  int pre_row_zero;   // shared pre without a row dim (dx(X)): always row 0 of its map
  int post_row_zero;
  int64_t npq;        // tile rows
  int64_t ntiles;     // virtual tiles: nrb * nzq * rbq * ntx (tile rows past npq are skipped)
  XgFastDiv fd_ntx, fd_rbq, fd_nzq;
  int nst;                    // tiles in flight
  int l2_hints;               // evict-first fields, evict-last metric tiles
  unsigned field_bytes, pre_bytes, post_bytes, stage_bytes;  // box sizes rounded up to 128
};

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// PRE: XG_PRE_NONE, XG_PRE_FULL, or XG_PRE_SHARED standing for both runtime modes shared / scalar
template <typename T, int OP, int PRE, bool LO, int U>
__global__ void __launch_bounds__(kTmaConsumers + 32, 3)
    k_stencil_row_tma(const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_pre,
                      const __grid_constant__ CUtensorMap map_post, const RowTmaArgs<T> a) {
  typedef RowTmaGeo<T> G;
  constexpr int VEC = G::VEC, TXE = G::TXE, TY = G::TY;
  constexpr int BOXW = TXE + VEC, LR = kTmaConsumers / TY, NVR = TXE / VEC, LS = TY * BOXW;
  constexpr int XS = LO ? VEC : 0;  // the box starts one vector left of the tile when the lower neighbour is needed
  constexpr int NBI = LO ? -1 : VEC;
  typedef XgPack<T, VEC> Pack;
  typedef typename XgVec<T, VEC>::type V;
  const unsigned FULL = 0xffffffffu;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x;
  const int NST = a.nst;
  const uint32_t full_u32 = smem_u32(smem_raw);  // full[NST], empty[NST]; the stages start at +128
  const uint32_t empty_u32 = full_u32 + 8u * NST;
  unsigned char* stage0 = smem_raw + 128;
  const int64_t nloc = (a.ntiles > blockIdx.x) ? (a.ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;

  // virtual tile -> (level batch, tile row, x tile); false for the padding rows of the last row block
  auto tile_geom = [&](int64_t i, int& z0, int& p0, int& x0) -> bool {
    const uint32_t g = (uint32_t)(i * gridDim.x + blockIdx.x);
    const uint32_t t = xg_fastdiv_q(g, a.fd_ntx);
    const uint32_t c = g - t * a.fd_ntx.d;
    const uint32_t t2 = xg_fastdiv_q(t, a.fd_rbq);
    const uint32_t pql = t - t2 * a.fd_rbq.d;
    const uint32_t rb = xg_fastdiv_q(t2, a.fd_nzq);
    const uint32_t zq = t2 - rb * a.fd_nzq.d;
    const uint32_t pq = rb * a.fd_rbq.d + pql;
    z0 = (int)(zq * U);
    p0 = (int)(pq * TY);
    x0 = (int)(c * TXE);
    return pq < (uint32_t)a.npq;
  };

  if (tid == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_in) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_post) : "memory");
    if (PRE != XG_PRE_NONE && a.pre_mode != XG_PRE_SCALAR)
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_pre) : "memory");
    for (int b = 0; b < NST; ++b) {
      mbar_init(full_u32 + 8u * b, 1);
      mbar_init(empty_u32 + 8u * b, kTmaConsumers / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (tid >= kTmaConsumers) {
    // ---- producer warp: one lane keeps the ring full
    if (tid == kTmaConsumers) {
      const unsigned fb = BOXW * TY * U * sizeof(T), mb = BOXW * TY * sizeof(T);
      const bool pre_box = PRE == XG_PRE_FULL || (PRE == XG_PRE_SHARED && a.pre_mode == XG_PRE_SHARED);
      const unsigned bytes = fb + mb + (PRE == XG_PRE_FULL ? fb : (pre_box ? mb : 0));
      const uint64_t once = l2_policy_evict_first(), keep = l2_policy_evict_last();
      int64_t k = 0;
      for (int64_t i = 0; i < nloc; ++i) {
        int z0, p0, x0;
        if (!tile_geom(i, z0, p0, x0)) continue;
        const int b = (int)(k % NST);
        if (k >= NST) mbar_wait(empty_u32 + 8u * b, (uint32_t)(((k / NST) - 1) & 1));
        const uint32_t bar = full_u32 + 8u * b;
        mbar_expect_tx(bar, bytes);
        const uint32_t dst = smem_u32(stage0 + (size_t)b * a.stage_bytes);
        const int cx = x0 - XS;
        if (a.l2_hints) {
          tensor_load_3d_hint(dst, &map_in, cx, p0, z0, bar, once);
          if (PRE == XG_PRE_FULL) tensor_load_3d_hint(dst + a.field_bytes, &map_pre, cx, p0, z0, bar, once);
          else if (pre_box) tensor_load_2d_hint(dst + a.field_bytes, &map_pre, cx, a.pre_row_zero ? 0 : p0, bar, keep);
          tensor_load_2d_hint(dst + a.field_bytes + a.pre_bytes, &map_post, cx, a.post_row_zero ? 0 : p0, bar, keep);
        } else {
          tensor_load_3d(dst, &map_in, cx, p0, z0, bar);
          if (PRE == XG_PRE_FULL) tensor_load_3d(dst + a.field_bytes, &map_pre, cx, p0, z0, bar);
          else if (pre_box) tensor_load_2d(dst + a.field_bytes, &map_pre, cx, a.pre_row_zero ? 0 : p0, bar);
          tensor_load_2d(dst + a.field_bytes + a.pre_bytes, &map_post, cx, a.post_row_zero ? 0 : p0, bar);
        }
        ++k;
      }
    }
    return;
  }

  // ---- consumers
  const int lane = tid & 31;
  const int ty = tid / LR, vx = tid - ty * LR;
  const int vxs = vx < NVR ? vx : NVR - 1;  // spare slots shadow the last vector: valid addresses, in the shuffles, no store
  const int sidx = ty * BOXW + vxs * VEC + XS;  // element 0 of this thread's vector inside a box level
  const int pidx = (PRE == XG_PRE_SHARED && a.pre_row_zero) ? sidx - ty * BOXW : sidx;  // a row-less pre sits in row 0
  const bool edge_lane = LO ? (lane == 0) : (lane == 31 || vx >= NVR - 1);  // no neighbouring lane holds the element
  const bool pre_scalar = PRE == XG_PRE_SHARED && a.pre_mode == XG_PRE_SCALAR;
  const T* prep = reinterpret_cast<const T*>(a.pre.ptr);
  const int64_t zstride = a.P * a.n;

  int64_t k = 0;
  for (int64_t i = 0; i < nloc; ++i) {
    int z0, p0, x0;
    if (!tile_geom(i, z0, p0, x0)) continue;
    const int b = (int)(k % NST);
    const int x = x0 + vxs * VEC, prow = p0 + ty;
    const bool act = vx < NVR && x < a.n && prow < a.P;
    const int nz = (a.Zn - z0 < U) ? (int)(a.Zn - z0) : U;
    const unsigned char* st = stage0 + (size_t)b * a.stage_bytes;
    const T* fs = reinterpret_cast<const T*>(st) + sidx;
    const T* ps = reinterpret_cast<const T*>(st + a.field_bytes) + pidx;
    const T* qs = reinterpret_cast<const T*>(st + a.field_bytes + a.pre_bytes) + sidx;
    mbar_wait(full_u32 + 8u * b, (uint32_t)((k / NST) & 1));
    Pack pm;
    *reinterpret_cast<V*>(pm.v) = *reinterpret_cast<const V*>(qs);
    XgSharedDivisor<T> dv[VEC];
#pragma unroll
    for (int kk = 0; kk < VEC; ++kk) dv[kk].set(pm.v[kk]);
    Pack pv;
    T pnb = T(1);
    if (PRE == XG_PRE_SHARED && !pre_scalar) {
      *reinterpret_cast<V*>(pv.v) = *reinterpret_cast<const V*>(ps);
      if (edge_lane) pnb = ps[NBI];
    }
    const int64_t row0 = (int64_t)z0 * a.P + prow;
    // the spare rows of the last tile row (prow >= P, nothing stored) load their global operands at the last row:
    // unclamped they would run past the field's, the halo's and the pre-metric's last level
    const int prc = prow < a.P ? prow : (int)a.P - 1;
    const bool at_edge = LO ? (x == 0) : (x + VEC >= a.n);
    T* op = a.out + row0 * a.n + x;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (u >= nz) break;  // block-uniform
      Pack v;
      *reinterpret_cast<V*>(v.v) = *reinterpret_cast<const V*>(fs + u * LS);
      T enb = T(0);
      if (edge_lane) enb = fs[u * LS + NBI];
      if (PRE != XG_PRE_NONE) {
        if (PRE == XG_PRE_FULL) {
          *reinterpret_cast<V*>(pv.v) = *reinterpret_cast<const V*>(ps + u * LS);
          if (edge_lane) pnb = ps[u * LS + NBI];
        } else if (pre_scalar) {
          pnb = __ldg(prep + xg_groups_offset(a.pre.outer, (int64_t)(z0 + u) * a.P + prc));
#pragma unroll
          for (int kk = 0; kk < VEC; ++kk) pv.v[kk] = pnb;
        }
#pragma unroll
        for (int kk = 0; kk < VEC; ++kk) v.v[kk] = v.v[kk] * pv.v[kk];
        enb = enb * pnb;
      }
      T nb = LO ? __shfl_up_sync(FULL, v.v[VEC - 1], 1) : __shfl_down_sync(FULL, v.v[0], 1);
      if (edge_lane) nb = enb;
      if (at_edge) {
        // A[row, s] = in * pre straight from global memory: the row's other end (periodic) only
        const int64_t row = (int64_t)(z0 + u) * a.P + prc;
        auto A = [&](int64_t s_) -> T {
          T val = __ldg(a.in + row * a.n + s_);
          if (PRE != XG_PRE_NONE) val = val * __ldg(prep + xg_groups_offset(a.pre.outer, row) + s_ * a.pre.axis_stride);
          return val;
        };
        const T* halo = LO ? a.halo_lo : a.halo_hi;
        if (halo) nb = __ldg(halo + row);
        else if (a.bc == XG_BC_FILL) nb = a.fill;
        else if (a.bc == XG_BC_PERIODIC) nb = A(LO ? a.n - 1 : 0);
        else if (a.bc == XG_BC_EXTEND) nb = LO ? v.v[0] : v.v[VEC - 1];
        else nb = LO ? T(2) * v.v[0] - v.v[1] : T(2) * v.v[VEC - 1] - v.v[VEC - 2];
      }
      Pack res;
#pragma unroll
      for (int kk = 0; kk < VEC; ++kk) {
        if (LO) res.v[kk] = xg_apply_op<T, OP>(kk == 0 ? nb : v.v[kk > 0 ? kk - 1 : 0], v.v[kk]);
        else res.v[kk] = xg_apply_op<T, OP>(v.v[kk], kk == VEC - 1 ? nb : v.v[kk < VEC - 1 ? kk + 1 : kk]);
      }
#pragma unroll
      for (int kk = 0; kk < VEC; ++kk) res.v[kk] = dv[kk].div(res.v[kk]);
      if (act) xg_st_stream<T, VEC>(op + u * zstride, res);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty_u32 + 8u * b);  // this warp is done with stage b
    ++k;
  }
}

// ---------------------------------------------------------------------------
// host dispatch
// ---------------------------------------------------------------------------
static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

template <typename T, int VEC, int OP, bool MET>
int launch_strided(StencilArgs<T>& a, cudaStream_t st) {
  const int64_t nvec = xg_ceil_div(a.inner, VEC);
  a.nwc = xg_ceil_div(nvec, 32);
  // march length: long enough that the re-read halo row is a few % of traffic,
  // short enough that there are plenty of warps for 148 SMs.
  static const int tune_j = env_int("XG_STRIDED_J", 0);  // tuning knobs (benchmarks only)
  static const int tune_u = env_int("XG_STRIDED_U", 0);
  // Tuning notes (profiles/r1b_tune_strided.txt): in a loop of identical launches short marches
  // (J = 4) look 8 % faster for Y, but per-launch ncu timings and the mixed sequence of bench.py
  // show no gain, and the fused-metric variants lose 20 % (per-segment operand setup is amortised
  // over fewer rows) — so 32 stays; a plane-strided axis marches as far as possible.
  int J;
  if (tune_j > 0) J = tune_j;
  else J = (a.n_out <= 96) ? (int)a.n_out : 32;
  if (J > a.n_out) J = (int)a.n_out;
  a.J = J;
  a.nseg = xg_ceil_div(a.n_out, J);
  a.nunits = a.outer * a.nseg * a.nwc;
  a.small_units = a.nunits < (1ll << 31);
  a.fd_nseg = xg_fastdiv_make(a.small_units ? a.nseg : 1);
  a.fd_nwc = xg_fastdiv_make(a.small_units ? a.nwc : 1);
  static const int tune_sf = env_int("XG_STRIDED_SEGFAST", 0);
  a.seg_fast = tune_sf != 0;
  const int64_t blocks = xg_ceil_div(a.nunits, kWarpsPerBlock);
  if (blocks > 0x7fffffffLL) return xg_fail(XG_EINVAL, "xg_stencil2: grid too large");
  static const int tune_met = env_int("XG_STRIDED_MET", 0);  // 1: U=2; 2: U=4 at 3 CTAs/SM (80 registers)
  if (!MET && tune_u == 8)
    k_stencil_strided<T, VEC, OP, MET, 8><<<(unsigned)blocks, kThreads, 0, st>>>(a);
  else if (!MET && tune_u == 2)
    k_stencil_strided<T, VEC, OP, MET, 2><<<(unsigned)blocks, kThreads, 0, st>>>(a);
  else if (MET && VEC > 1 && tune_met == 1)
    k_stencil_strided<T, VEC, OP, MET, 2><<<(unsigned)blocks, kThreads, 0, st>>>(a);
  else if (MET && VEC > 1 && tune_met == 2)
    k_stencil_strided<T, VEC, OP, MET, 4, 3><<<(unsigned)blocks, kThreads, 0, st>>>(a);
  else
    k_stencil_strided<T, VEC, OP, MET, 4><<<(unsigned)blocks, kThreads, 0, st>>>(a);
  return xg_check_launch("xg_stencil2(strided)");
}

template <typename T, int VEC, int OP, bool MET>
int launch_row_vec(StencilArgs<T>& a, cudaStream_t st) {
  constexpr int U = 4;
  const int64_t nv = a.n / VEC;
  a.nwc = xg_ceil_div(nv, 32 * U);
  a.nunits = a.outer * a.nwc;
  a.small_units = a.nunits < (1ll << 31);
  a.fd_nwc = xg_fastdiv_make(a.small_units ? a.nwc : 1);
  const int64_t blocks = xg_ceil_div(a.nunits, kWarpsPerBlock);
  if (blocks > 0x7fffffffLL) return xg_fail(XG_EINVAL, "xg_stencil2: grid too large");
  k_stencil_row_vec<T, VEC, OP, MET, U><<<(unsigned)blocks, kThreads, 0, st>>>(a);
  return xg_check_launch("xg_stencil2(row_vec)");
}

// The z-batched kernel applies when the divisor is x-contiguous, 16-byte aligned, and its
// outermost index group is a broadcast one (the level dim of a (Z, Y, X) field against dx(Y, X)).
template <typename T, int VEC, int OP>
int launch_row_zb(const StencilArgs<T>& s, cudaStream_t st, bool* launched) {
  constexpr int U = 4;
  *launched = false;
  static const int enabled = env_int("XG_ROW_ZB", 1);
  const XgOperand& m = s.post;
  if (!enabled || !m.ptr || m.axis_stride != 1 || !s.post_axis_vec_ok) return XG_OK;
  RowZbArgs<T> a;
  if (m.outer.n == 0) a.Zn = s.outer;  // dx(X): one divisor row for the whole field
  else if (m.outer.stride[0] == 0) a.Zn = m.outer.size[0];
  else return XG_OK;
  if (a.Zn < 2 || s.outer % a.Zn != 0) return XG_OK;
  a.P = s.outer / a.Zn;
  a.in = s.in;
  a.out = s.out;
  a.n = s.n;
  a.lo = s.lo;
  a.bc = s.bc;
  a.fill = s.fill;
  a.halo_lo = s.halo_lo;
  a.halo_hi = s.halo_hi;
  a.pre = s.pre;
  a.post = s.post;
  a.pre_vec = s.pre_axis_vec_ok;
  a.pre_shared = !s.pre.ptr || s.pre.outer.n == 0 ||
                 (s.pre.outer.stride[0] == 0 && s.pre.outer.size[0] % a.Zn == 0);
  // measured at C3 (profiles/r2_row_tma_sweep.txt, last line vs k_stencil_row_vec): ahead only when the
  // pre-metric is level-shared too (1.25 vs 1.54 ms); with no or a per-level pre-metric the four edge loads
  // per warp cost more than the shared divisor saves (1.18 vs 1.07, 2.02 vs 1.86 ms)
  if (!s.pre.ptr || !a.pre_shared) return XG_OK;
  a.nwc = xg_ceil_div(s.n / VEC, 32);
  a.nunits = xg_ceil_div(a.Zn, U) * a.P * a.nwc;
  a.small_units = a.nunits < (1ll << 31) && a.P < (1ll << 31);
  a.fd_nwc = xg_fastdiv_make(a.small_units ? a.nwc : 1);
  a.fd_P = xg_fastdiv_make(a.small_units ? a.P : 1);
  const int64_t blocks = xg_ceil_div(a.nunits, kWarpsPerBlock);
  if (blocks > 0x7fffffffLL) return XG_OK;
  k_stencil_row_zb<T, VEC, OP, U><<<(unsigned)blocks, kThreads, 0, st>>>(a);
  *launched = true;
  return xg_check_launch("xg_stencil2(row_zb)");
}

// Eligibility of the TMA-staged kernel: divisor x-contiguous with a broadcast level group (as for row_zb),
// rows long enough to fill tiles, diff / interp, and a pre-metric that is absent, laid out like the field,
// shared like the divisor, or one scalar per row.
template <typename T, int OP, int PRE, bool LO, int U>
int launch_row_tma_kernel(const CUtensorMap& map_in, const CUtensorMap& map_pre, const CUtensorMap& map_post,
                          const RowTmaArgs<T>& a, int64_t grid, size_t smem, cudaStream_t st) {
  auto kern = k_stencil_row_tma<T, OP, PRE, LO, U>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  kern<<<(unsigned)grid, kTmaConsumers + 32, smem, st>>>(map_in, map_pre, map_post, a);
  return 1;
}

template <typename T, int VEC, int OP>
int launch_row_tma(const StencilArgs<T>& s, cudaStream_t st, bool* launched) {
  typedef RowTmaGeo<T> G;
  static_assert(G::VEC == VEC, "vector width");
  constexpr int BOXW = G::TXE + VEC;
  *launched = false;
  if constexpr (OP != XG_OP_DIFF && OP != XG_OP_INTERP) {
    return XG_OK;
  } else {
    static const int enabled = env_int("XG_ROW_TMA", 1);
    constexpr int U = 4;  // 8 levels per tile measured no faster (profiles/r2_row_tma_sweep.txt)
    const XgOperand& m = s.post;
    if (!enabled || !m.ptr || m.axis_stride != 1 || !s.post_axis_vec_ok) return XG_OK;
    if (s.n < 2 * G::TXE || s.n >= (1ll << 30) || s.outer >= (1ll << 30)) return XG_OK;  // 32-bit tile coordinates
    RowTmaArgs<T> a;
    int64_t post_rs = 0;
    if (m.outer.n == 0) { a.Zn = s.outer; a.post_row_zero = 1; }
    else if (m.outer.n == 1 && m.outer.stride[0] == 0) { a.Zn = m.outer.size[0]; a.post_row_zero = 1; }
    else if (m.outer.n == 2 && m.outer.stride[0] == 0) { a.Zn = m.outer.size[0]; a.post_row_zero = 0; post_rs = m.outer.stride[1]; }
    else return XG_OK;
    if (a.Zn < 2 || s.outer % a.Zn != 0) return XG_OK;
    a.P = s.outer / a.Zn;
    if (a.post_row_zero && a.P != 1) return XG_OK;
    if (!a.post_row_zero && m.outer.size[1] != a.P) return XG_OK;
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return XG_OK;
    a.in = s.in;
    a.out = s.out;
    a.n = s.n;
    a.bc = s.bc;
    a.fill = s.fill;
    a.halo_lo = s.halo_lo;
    a.halo_hi = s.halo_hi;
    a.pre = s.pre;
    a.pre_row_zero = 0;
    int64_t pre_rs = 0;
    const XgOperand& q = s.pre;
    if (!q.ptr) a.pre_mode = XG_PRE_NONE;
    else if (q.axis_stride == 0) a.pre_mode = XG_PRE_SCALAR;
    else if (q.axis_stride != 1 || !s.pre_axis_vec_ok) return XG_OK;
    else if (q.outer.n == 1 && q.outer.stride[0] == s.n && q.outer.size[0] == s.outer) a.pre_mode = XG_PRE_FULL;
    else if (q.outer.n == 0 || (q.outer.n == 1 && q.outer.stride[0] == 0)) { a.pre_mode = XG_PRE_SHARED; a.pre_row_zero = 1; }
    else if (q.outer.n == 2 && q.outer.stride[0] == 0 && q.outer.size[0] == a.Zn && q.outer.size[1] == a.P) {
      a.pre_mode = XG_PRE_SHARED;
      pre_rs = q.outer.stride[1];
    } else return XG_OK;

    auto up128 = [](size_t v) { return (unsigned)((v + 127) / 128 * 128); };
    a.field_bytes = up128((size_t)BOXW * G::TY * U * sizeof(T));
    const unsigned metric_bytes = up128((size_t)BOXW * G::TY * sizeof(T));
    a.pre_bytes = a.pre_mode == XG_PRE_FULL ? a.field_bytes : (a.pre_mode == XG_PRE_SHARED ? metric_bytes : 0);
    a.post_bytes = metric_bytes;
    a.stage_bytes = a.field_bytes + a.pre_bytes + a.post_bytes;
    int dev = 0, sms = 148, smem_sm = 0, smem_max = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    // Tuning (profiles/r2_row_tma_sweep.txt): two tiles per CTA; three CTAs per SM while the tiles in flight
    // stay below ~135 KB per SM, else two (more bytes in flight measured slower, as did L2 eviction hints).
    static const int tune_nst = env_int("XG_ROW_TMA_NST", 0);
    static const int tune_ctas = env_int("XG_ROW_TMA_CTAS", 0);
    int ctas = (3 * 2 * (int)a.stage_bytes <= 135 * 1024) ? 3 : 2;
    if (tune_ctas >= 1 && tune_ctas <= 4) ctas = tune_ctas;
    int per_cta = smem_sm / ctas - 1024;  // the driver reserves 1 KB per resident CTA
    if (per_cta > smem_max) per_cta = smem_max;
    const int fit = (per_cta - 128) / (int)a.stage_bytes;
    int nst = fit < 2 ? fit : 2;
    if (tune_nst > 0) nst = tune_nst < fit ? tune_nst : fit;
    if (nst < 1) return XG_OK;
    a.nst = nst;
    static const int tune_hint = env_int("XG_ROW_TMA_HINT", 0);
    a.l2_hints = tune_hint;
    // row blocks: ~128 rows each, evened out
    const int64_t ntx = xg_ceil_div(s.n, G::TXE);
    a.npq = xg_ceil_div(a.P, G::TY);
    static const int tune_rb = env_int("XG_ROW_TMA_RB", 128);
    const int64_t rbq_target = xg_ceil_div(tune_rb > 0 ? tune_rb : 128, G::TY);
    const int64_t nrb = xg_ceil_div(a.npq, rbq_target);
    const int64_t rbq = xg_ceil_div(a.npq, nrb);
    const int64_t nzq = xg_ceil_div(a.Zn, U);
    a.ntiles = nrb * nzq * rbq * ntx;
    if (a.ntiles >= (1ll << 31)) return XG_OK;
    a.fd_ntx = xg_fastdiv_make(ntx);
    a.fd_rbq = xg_fastdiv_make(rbq);
    a.fd_nzq = xg_fastdiv_make(nzq);

    CUtensorMap map_in, map_pre, map_post;
    const cuuint64_t d3[3] = {(cuuint64_t)s.n, (cuuint64_t)a.P, (cuuint64_t)a.Zn};
    const cuuint64_t s3[2] = {(cuuint64_t)s.n * sizeof(T), (cuuint64_t)a.P * s.n * sizeof(T)};
    const cuuint32_t b3[3] = {(cuuint32_t)BOXW, (cuuint32_t)G::TY, (cuuint32_t)U};
    if (xg_encode_map<T>(enc, &map_in, s.in, 3, d3, s3, b3)) return XG_OK;
    auto encode_rows = [&](CUtensorMap* map, const void* ptr, bool row_zero, int64_t rs) -> int {
      // a row-less operand is a (n, 1) map read at row 0; its box still spans TY rows (the rest is zero fill)
      const cuuint64_t d2[2] = {(cuuint64_t)s.n, (cuuint64_t)(row_zero ? 1 : a.P)};
      const cuuint64_t s2[1] = {(cuuint64_t)(row_zero ? s.n : rs) * sizeof(T)};
      const cuuint32_t b2[2] = {(cuuint32_t)BOXW, (cuuint32_t)G::TY};
      return xg_encode_map<T>(enc, map, static_cast<const T*>(ptr), 2, d2, s2, b2);
    };
    if (encode_rows(&map_post, m.ptr, a.post_row_zero != 0, post_rs)) return XG_OK;
    map_pre = map_post;
    if (a.pre_mode == XG_PRE_FULL) {
      if (xg_encode_map<T>(enc, &map_pre, static_cast<const T*>(q.ptr), 3, d3, s3, b3)) return XG_OK;
    } else if (a.pre_mode == XG_PRE_SHARED) {
      if (encode_rows(&map_pre, q.ptr, a.pre_row_zero != 0, pre_rs)) return XG_OK;
    }
    const size_t smem = 128 + (size_t)nst * a.stage_bytes;
    int64_t grid = (int64_t)ctas * sms;
    if (grid > a.ntiles) grid = a.ntiles;
    const int pre_t = a.pre_mode == XG_PRE_NONE ? XG_PRE_NONE : (a.pre_mode == XG_PRE_FULL ? XG_PRE_FULL : XG_PRE_SHARED);
    int ok = 0;
#define XG_TMA_GO(PRE_, LO_, U_) ok = launch_row_tma_kernel<T, OP, PRE_, LO_, U_>(map_in, map_pre, map_post, a, grid, smem, st)
#define XG_TMA_LO(PRE_, U_) \
  if (s.lo) XG_TMA_GO(PRE_, true, U_); \
  else XG_TMA_GO(PRE_, false, U_)
#define XG_TMA_PRE(U_)                                   \
  if (pre_t == XG_PRE_NONE) { XG_TMA_LO(XG_PRE_NONE, U_); }  \
  else if (pre_t == XG_PRE_FULL) { XG_TMA_LO(XG_PRE_FULL, U_); } \
  else { XG_TMA_LO(XG_PRE_SHARED, U_); }
    XG_TMA_PRE(4)
#undef XG_TMA_PRE
#undef XG_TMA_LO
#undef XG_TMA_GO
    if (!ok) return XG_OK;
    *launched = true;
    return xg_check_launch("xg_stencil2(row_tma)");
  }
}

template <typename T, int OP, bool MET>
int launch_row_scalar(StencilArgs<T>& a, cudaStream_t st) {
  const int64_t total = a.outer * a.n_out;
  int64_t blocks = xg_ceil_div(total, kThreads);
  if (blocks > 148 * 64) blocks = 148 * 64;  // grid-stride beyond that
  k_stencil_row_scalar<T, OP, MET><<<(unsigned)blocks, kThreads, 0, st>>>(a);
  return xg_check_launch("xg_stencil2(row_scalar)");
}

template <typename T, int OP, bool MET>
int dispatch_layout(StencilArgs<T>& a, cudaStream_t st) {
  constexpr int VEC = XgVecWidth<T>::value;
  const bool ptr_ok = ((uintptr_t)a.in % 16 == 0) && ((uintptr_t)a.out % 16 == 0) &&
                      (!a.halo_lo || (uintptr_t)a.halo_lo % 16 == 0) &&
                      (!a.halo_hi || (uintptr_t)a.halo_hi % 16 == 0);
  if (a.inner > 1) {
    if constexpr (MET) {
      // the TMA-staged tile kernel, rows = the operated axis.  Either the dim right before x with the outer
      // index as levels (derivative('Y') on (Z, Y, X): dx(Y, X) is shared between levels), or — a single outer
      // index, e.g. any stencil along Z of a (Z, Y, X) field — the inner dims split as levels x x with per-row
      // scalar metrics (dz(Z)) shared by all of them.
      if (ptr_ok && a.inner % VEC == 0) {
        XgTileSpec<T> ts;
        ts.Pb = a.n;
        ts.Po = a.n_out;
        ts.a = nullptr;
        ts.op_a = ts.lo_a = ts.bc_a = 0;
        ts.fill_a = T(0);
        ts.b = a.in;
        ts.op_b = OP;
        ts.lo_b = a.lo;
        ts.hi_b = a.hi;
        ts.bc_b = a.bc;
        ts.fill_b = a.fill;
        ts.halo_lo = a.halo_lo;
        ts.halo_hi = a.halo_hi;
        ts.subtract = 0;
        ts.ma.ptr = nullptr;
        ts.ma.sz = ts.ma.sp = ts.ma.sx = 0;
        ts.out = a.out;
        bool ok = false;
        const int64_t nx = a.nx_last;
        if (a.outer == 1 && nx > 0 && nx < a.inner && a.inner % nx == 0) {
          ts.Zn = a.inner / nx;
          ts.n = nx;
          ts.f_sp = a.inner;
          ts.b_sz = ts.o_sz = nx;
          // metrics: broadcast over the inner dims (sx = sz = 0), or laid out like the field's inner dims
          auto inner_split = [&](const XgOperand& m, XgTileOperand<T>* o) -> bool {
            o->ptr = static_cast<const T*>(m.ptr);
            o->sz = o->sp = o->sx = 0;
            if (!m.ptr) return true;
            if (m.outer.n != 0) return false;
            o->sp = m.axis_stride;
            if (m.inner.n == 0 || (m.inner.n == 1 && m.inner.stride[0] == 0)) return true;
            if (m.inner.n == 1 && m.inner.size[0] == a.inner && m.inner.stride[0] == 1) {
              o->sx = 1;
              o->sz = nx;
              return true;
            }
            return false;
          };
          ok = inner_split(a.pre, &ts.mb) && inner_split(a.post, &ts.post);
        } else {
          ts.Zn = a.outer;
          ts.n = a.inner;
          ts.f_sp = a.inner;
          ts.b_sz = a.n * a.inner;
          ts.o_sz = a.n_out * a.inner;
          ok = xg_tile_operand_from<T>(a.pre, a.outer, a.inner, &ts.mb) &&
               xg_tile_operand_from<T>(a.post, a.outer, a.inner, &ts.post);
        }
        if (ok) {
          bool launched = false;
          const int rc = xg_tile_stencil<T>(ts, st, &launched, "xg_stencil2(tile_tma)");
          if (rc || launched) return rc;
        }
      }
    }
    if (ptr_ok && a.inner % VEC == 0) return launch_strided<T, VEC, OP, MET>(a, st);
    a.pre.vec_ok = 0;
    a.post.vec_ok = 0;
    return launch_strided<T, 1, OP, MET>(a, st);
  }
  if (ptr_ok && a.n_out == a.n && a.n % VEC == 0 && a.n / VEC >= 32) {
    if constexpr (MET) {
      bool launched = false;
      int rc = launch_row_tma<T, VEC, OP>(a, st, &launched);
      if (rc || launched) return rc;
      rc = launch_row_zb<T, VEC, OP>(a, st, &launched);
      if (rc || launched) return rc;
    }
    return launch_row_vec<T, VEC, OP, MET>(a, st);
  }
  return launch_row_scalar<T, OP, MET>(a, st);
}

template <typename T, int OP>
int dispatch_met(StencilArgs<T>& a, cudaStream_t st) {
  if (a.pre.ptr || a.post.ptr) return dispatch_layout<T, OP, true>(a, st);
  return dispatch_layout<T, OP, false>(a, st);
}

template <typename T>
int dispatch_op(int op, StencilArgs<T>& a, cudaStream_t st) {
  switch (op) {
    case XG_OP_DIFF: return dispatch_met<T, XG_OP_DIFF>(a, st);
    case XG_OP_INTERP: return dispatch_met<T, XG_OP_INTERP>(a, st);
    case XG_OP_MIN: return dispatch_met<T, XG_OP_MIN>(a, st);
    case XG_OP_MAX: return dispatch_met<T, XG_OP_MAX>(a, st);
  }
  return xg_fail(XG_EINVAL, "xg_stencil2: unknown op");
}

// vector loads of a metric along x in the row kernels
static int axis_vec_ok(const XgOperand& m, int vec, size_t es) {
  if (!m.ptr || m.axis_stride != 1) return 0;
  if ((uintptr_t)m.ptr % (vec * es) != 0) return 0;
  for (int k = 0; k < m.outer.n; ++k)
    if (m.outer.stride[k] % vec != 0) return 0;
  return 1;
}

template <typename T>
int stencil2_typed(int op, const void* in, void* out, int ndim, const int64_t* shape,
                   int axis, int lo, int hi, int bc, double fill_value,
                   const void* pre_metric, const int64_t* pre_strides,
                   const void* post_metric, const int64_t* post_strides,
                   const void* halo_lo, const void* halo_hi, cudaStream_t st) {
  constexpr int VEC = XgVecWidth<T>::value;
  XgView v;
  int rc = xg_collapse_view(ndim, shape, axis, &v);
  if (rc) return rc;
  StencilArgs<T> a;
  a.in = static_cast<const T*>(in);
  a.out = static_cast<T*>(out);
  a.outer = v.outer;
  a.n = v.n;
  a.inner = v.inner;
  a.n_out = v.n + lo + hi - 1;
  a.nx_last = ndim > 0 ? shape[ndim - 1] : 1;
  a.lo = lo;
  a.hi = hi;
  a.bc = bc;
  a.fill = static_cast<T>(fill_value);
  a.halo_lo = static_cast<const T*>(halo_lo);
  a.halo_hi = static_cast<const T*>(halo_hi);
  a.J = 0;
  a.nseg = a.nwc = a.nunits = 0;
  a.small_units = false;
  a.seg_fast = false;
  if (v.n == 0) return xg_fail(XG_EINVAL, "xg_stencil2: empty operated axis");
  if (v.outer == 0 || v.inner == 0 || a.n_out <= 0) return XG_OK;  // nothing to write

  int64_t out_shape[XG_MAX_NDIM];
  for (int d = 0; d < ndim; ++d) out_shape[d] = shape[d];
  out_shape[axis] = a.n_out;
  rc = xg_make_operand(pre_metric, pre_strides, ndim, shape, axis, VEC, sizeof(T), &a.pre,
                       "xg_stencil2(pre_metric)");
  if (rc) return rc;
  rc = xg_make_operand(post_metric, post_strides, ndim, out_shape, axis, VEC, sizeof(T),
                       &a.post, "xg_stencil2(post_metric)");
  if (rc) return rc;
  a.pre_axis_vec_ok = axis_vec_ok(a.pre, VEC, sizeof(T));
  a.post_axis_vec_ok = axis_vec_ok(a.post, VEC, sizeof(T));
  return dispatch_op<T>(op, a, st);
}

}  // namespace

extern "C" int xg_stencil2(int op, int dtype, const void* in, void* out, int ndim,
                           const int64_t* shape, int axis, int lo, int hi, int bc,
                           double fill_value, const void* pre_metric,
                           const int64_t* pre_strides, const void* post_metric,
                           const int64_t* post_strides, const void* halo_lo,
                           const void* halo_hi, void* stream) {
  if (!in || !out) return xg_fail(XG_EINVAL, "xg_stencil2: null field pointer");
  if (!shape) return xg_fail(XG_EINVAL, "xg_stencil2: null shape");
  if (lo < 0 || lo > 1 || hi < 0 || hi > 1)
    return xg_fail(XG_EINVAL, "xg_stencil2: halo widths must be 0 or 1");
  if (bc < XG_BC_NONE || bc > XG_BC_EXTRAPOLATE)
    return xg_fail(XG_EINVAL, "xg_stencil2: unknown boundary condition");
  if ((lo && !halo_lo && bc == XG_BC_NONE) || (hi && !halo_hi && bc == XG_BC_NONE))
    // padding.py:601-608
    return xg_fail(XG_EINVAL,
                   "xg_stencil2: no boundary condition was specified but the "
                   "operation needs to pad the axis");
  if (in == out) return xg_fail(XG_EINVAL, "xg_stencil2: in-place operation is not supported");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == XG_F32)
    return stencil2_typed<float>(op, in, out, ndim, shape, axis, lo, hi, bc, fill_value,
                                 pre_metric, pre_strides, post_metric, post_strides,
                                 halo_lo, halo_hi, st);
  if (dtype == XG_F64)
    return stencil2_typed<double>(op, in, out, ndim, shape, axis, lo, hi, bc, fill_value,
                                  pre_metric, pre_strides, post_metric, post_strides,
                                  halo_lo, halo_hi, st);
  return xg_fail(XG_EINVAL, "xg_stencil2: dtype must be XG_F32 or XG_F64");
}
