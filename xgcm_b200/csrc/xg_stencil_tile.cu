// xg_tile_stencil — the TMA-staged tile kernel behind the metric-fused stencils along the second-to-last
// dim (derivative('Y'), diff('Y') x hFac / dx ...) and the two-field composites of xg_stencil_pair
// (C-grid divergence / vorticity) when their metrics are shared between levels.
//
//     out = ( OPa(pad_a(A x ma)) along x   (+|-)   OPb(pad_b(B x mb)) along p ) / post        (z, p, x) view
//
// Replaces, per call, the chain xgcm/grid.py:796-832 (+ one xarray arithmetic pass per operator) exactly
// like k_stencil_strided / k_stencil_pair do; what changes is the data movement:
//   * a tile is U = 4 levels x TY output rows x TXE cells; every operand of the tile is ONE bulk tensor
//     load (cp.async.bulk.tensor, SASS UTMALDG): A with a 16-byte halo along x, B with one halo row
//     along p, the metrics as 2-D boxes (shared between levels: loaded once per tile, not per level) or as
//     3-D boxes like the fields (hFac(Z, Y, X));
//   * all boxes of a tile complete on one mbarrier; a persistent CTA = 8 consumer warps + 1 producer warp
//     around a ring of NST tiles (full / empty mbarriers), so the bytes in flight live in shared memory;
//   * tiles run row block by row block, level batches innermost: the (Y, X) metric rows of a block (~2 MB)
//     are re-read from L2, not from DRAM, by each level batch (explicit L2 eviction hints measured slower);
//   * the divisor of a cell is the same for the U levels: it is inverted once (XgSharedDivisor keeps the
//     quotient bit-identical to the IEEE division, xg_common.cuh) — 3 instructions per cell instead of 11.
// Boundary rows / cells (zero-filled by the TMA unit where the box leaves the array) are replaced per the
// boundary rule; the wrap-around partners of `periodic` and the second row of `extrapolate` come straight
// from global memory (one row in Pb).
#include <stdlib.h>

#include "xg_stencil_tile.cuh"
#include "xg_tma.cuh"

namespace {

constexpr int kConsumers = 256;
constexpr int kU = 4;

template <typename T>
struct TileGeo;
template <>
struct TileGeo<float> {
  static constexpr int VEC = 4, TXE = 224, TY = 4;  // 56 vectors per row, 64 thread slots
};
template <>
struct TileGeo<double> {
  static constexpr int VEC = 2, TXE = 240, TY = 2;  // 120 vectors per row, 128 thread slots
};

enum { M_NONE = 0, M_FULL = 1, M_SHARED = 2, M_SCALAR = 3 };

template <typename T>
struct TileArgs {
  XgTileSpec<T> s;
  int ma_mode, mb_mode, post_mode;
  int ma_row0, mb_row0, post_row0;  // shared metric without a row dim: row 0 of its map for every row
  int64_t npq, ntiles;
  XgFastDiv fd_ntx, fd_rbq, fd_nzq;
  int nst;
  int swap;      // levels are the faster dim in memory (stencil along Z as rows): boxes are (x, level, row)
  int l2_hints;  // evict-first fields / evict-last metric tiles (measured slower on the row kernel: off by default)
  unsigned off_b, off_ma, off_mb, off_post, stage_bytes, tx_bytes;
};

// tensor loads with an optional L2 eviction policy
__device__ __forceinline__ void load3(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar,
                                      bool hint, uint64_t policy, bool swap = false) {
  if (swap) {  // (x, level, row) maps
    const int t = c1;
    c1 = c2;
    c2 = t;
  }
  if (hint) tensor_load_3d_hint(dst, map, c0, c1, c2, bar, policy);
  else tensor_load_3d(dst, map, c0, c1, c2, bar);
}
__device__ __forceinline__ void load2(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar, bool hint,
                                      uint64_t policy) {
  if (hint) tensor_load_2d_hint(dst, map, c0, c1, bar, policy);
  else tensor_load_2d(dst, map, c0, c1, bar);
}

__device__ __forceinline__ void mbar_arrive_tile(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// OPA / OPB: the operators, compile-time (a runtime switch per cell doubled the instruction count)
// LEVELM: some metric changes per level (3-D boxes or per-level scalars); false compiles those paths out
template <typename T, bool HAS_A, int OPA, int OPB, bool LEVELM>
__global__ void __launch_bounds__(kConsumers + 32, HAS_A ? 2 : 3)  // the pair's stages only fit twice per SM anyway
    k_tile_stencil(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                   const __grid_constant__ CUtensorMap map_ma, const __grid_constant__ CUtensorMap map_mb,
                   const __grid_constant__ CUtensorMap map_post, const TileArgs<T> a) {
  typedef TileGeo<T> G;
  constexpr int VEC = G::VEC, TXE = G::TXE, TY = G::TY, U = kU;
  constexpr int BOXW = TXE + VEC, LR = kConsumers / TY, NVR = TXE / VEC;
  constexpr int LSA = TY * BOXW, LSB = (TY + 1) * TXE, LSQ = TY * TXE;
  typedef XgPack<T, VEC> Pack;
  typedef typename XgVec<T, VEC>::type V;
  const unsigned FULL = 0xffffffffu;
  const XgTileSpec<T>& s = a.s;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x;
  const int NST = a.nst;
  const uint32_t full_u32 = smem_u32(smem_raw);  // full[NST], empty[NST]; the stages start at +128
  const uint32_t empty_u32 = full_u32 + 8u * NST;
  unsigned char* stage0 = smem_raw + 128;
  const int64_t nloc = (a.ntiles > blockIdx.x) ? (a.ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
  const int xs = (HAS_A && s.lo_a) ? VEC : 0;  // A's box starts one vector left of the tile for a lower neighbour

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
    for (int b = 0; b < NST; ++b) {
      mbar_init(full_u32 + 8u * b, 1);
      mbar_init(empty_u32 + 8u * b, kConsumers / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (tid >= kConsumers) {
    if (tid == kConsumers) {  // ---- producer: one lane keeps the ring full
      const uint64_t once = l2_policy_evict_first(), keep = l2_policy_evict_last();
      int64_t k = 0;
      for (int64_t i = 0; i < nloc; ++i) {
        int z0, p0, x0;
        if (!tile_geom(i, z0, p0, x0)) continue;
        const int b = (int)(k % NST);
        if (k >= NST) mbar_wait(empty_u32 + 8u * b, (uint32_t)(((k / NST) - 1) & 1));
        const uint32_t bar = full_u32 + 8u * b;
        mbar_expect_tx(bar, a.tx_bytes);
        const uint32_t dst = smem_u32(stage0 + (size_t)b * a.stage_bytes);
        const int pb = p0 - s.lo_b;  // first source row of B the tile needs (may be -1: zero fill, replaced below)
        const bool h = a.l2_hints != 0;
        if (HAS_A) load3(dst, &map_a, x0 - xs, p0, z0, bar, h, once);
        const bool sw = a.swap != 0;
        load3(dst + a.off_b, &map_b, x0, pb, z0, bar, false, once, sw);  // B's halo row is re-read by the next tile row
        if (HAS_A) {
          if (a.ma_mode == M_FULL) load3(dst + a.off_ma, &map_ma, x0 - xs, p0, z0, bar, h, once);
          else if (a.ma_mode == M_SHARED) load2(dst + a.off_ma, &map_ma, x0 - xs, a.ma_row0 ? 0 : p0, bar, h, keep);
        }
        if (a.mb_mode == M_FULL) load3(dst + a.off_mb, &map_mb, x0, pb, z0, bar, false, once, sw);
        else if (a.mb_mode == M_SHARED) load2(dst + a.off_mb, &map_mb, x0, a.mb_row0 ? 0 : pb, bar, h, keep);
        if (a.post_mode == M_FULL) load3(dst + a.off_post, &map_post, x0, p0, z0, bar, h, once, sw);
        else if (a.post_mode == M_SHARED) load2(dst + a.off_post, &map_post, x0, a.post_row0 ? 0 : p0, bar, h, keep);
        ++k;
      }
    }
    return;
  }

  // ---- consumers
  const int lane = tid & 31;
  const int ty = tid / LR, vx = tid - ty * LR;
  const int vxs = vx < NVR ? vx : NVR - 1;  // spare slots shadow the last vector: valid addresses, in the shuffles, no store
  const int lo_a = HAS_A ? s.lo_a : 0, lo_b = s.lo_b, sub = s.subtract;
  const int ma_mode = HAS_A ? a.ma_mode : M_NONE, mb_mode = a.mb_mode, post_mode = a.post_mode;
  const int ia = ty * BOXW + vxs * VEC + xs;
  const int ima = (ma_mode == M_SHARED && a.ma_row0) ? vxs * VEC + xs : ia;
  // box layouts: (level, row, x) normally; (row, level, x) when the levels are the faster dim in memory
  const int b_ls = a.swap ? TXE : LSB, b_rs = a.swap ? U * TXE : TXE;
  const int q_ls = a.swap ? TXE : LSQ;
  const int ib = ty * b_rs + vxs * VEC;
  const int ishr = ty * TXE + vxs * VEC;  // 2-D (row, x) boxes of level-shared metrics
  const int imb = (mb_mode == M_SHARED && a.mb_row0) ? vxs * VEC : ishr;
  const int imb1 = (mb_mode == M_SHARED && a.mb_row0) ? imb : imb + TXE;
  const int iq = (post_mode == M_SHARED && a.post_row0) ? vxs * VEC : ishr;
  const int nbi = lo_a ? -1 : VEC;
  const bool edge_lane = lo_a ? (lane == 0) : (lane == 31 || vx >= NVR - 1);
  // metrics that change per level need work inside the level loop; everything else is set up once per tile and
  // an absent metric is a multiplication by one (exact, NaN / zero preserving) instead of a branch per cell
  // (a per-row scalar that does not depend on the level — dz(Z) with Z as the rows — is set up per tile like a shared one)
  const bool ma_rowsc = ma_mode == M_SCALAR && s.ma.sz == 0, mb_rowsc = mb_mode == M_SCALAR && s.mb.sz == 0;
  const bool post_rowsc = post_mode == M_SCALAR && s.post.sz == 0;
  const bool ma_level = LEVELM && (ma_mode == M_FULL || (ma_mode == M_SCALAR && !ma_rowsc));
  const bool mb_level = LEVELM && (mb_mode == M_FULL || (mb_mode == M_SCALAR && !mb_rowsc));
  const bool post_level = LEVELM && (post_mode == M_FULL || (post_mode == M_SCALAR && !post_rowsc));
  const int64_t Pb = s.Pb, Po = s.Po, n = s.n, fsp = s.f_sp, bsz = s.b_sz, ostride = s.o_sz;

  int64_t k = 0;
  for (int64_t i = 0; i < nloc; ++i) {
    int z0, p0, x0;
    if (!tile_geom(i, z0, p0, x0)) continue;
    const int b = (int)(k % NST);
    const int x = x0 + vxs * VEC, prow = p0 + ty;
    const int prc = prow < Po ? prow : (int)Po - 1;  // clamped row for the scalar metric loads of spare rows
    const bool act = vx < NVR && x < n && prow < Po;
    const int nz = (s.Zn - z0 < U) ? (int)(s.Zn - z0) : U;
    const unsigned char* st = stage0 + (size_t)b * a.stage_bytes;
    const T* As = reinterpret_cast<const T*>(st) + ia;
    const T* Bs = reinterpret_cast<const T*>(st + a.off_b) + ib;
    const T* MAs = reinterpret_cast<const T*>(st + a.off_ma);
    const T* MBs = reinterpret_cast<const T*>(st + a.off_mb);
    const T* Qs = reinterpret_cast<const T*>(st + a.off_post);
    const int s0 = prow - lo_b, s1 = s0 + 1;  // source rows of B for this output row
    const bool low_b = s0 < 0, high_b = s1 >= Pb;
    // clamped source rows for the scalar metric loads (boundary rows and the spare rows of the last tile)
    const int64_t s0c = s0 < 0 ? 0 : (s0 < Pb ? s0 : Pb - 1), s1c = s1 < Pb ? s1 : Pb - 1;
    const bool at_edge = HAS_A && (lo_a ? (x == 0) : (x + VEC >= n));
    mbar_wait(full_u32 + 8u * b, (uint32_t)((k / NST) & 1));

    XgSharedDivisor<T> dv[VEC];
    Pack ma_v, mb0, mb1;
    T ma_nb = T(1);
#pragma unroll
    for (int kk = 0; kk < VEC; ++kk) {
      dv[kk].set(T(1));
      ma_v.v[kk] = mb0.v[kk] = mb1.v[kk] = T(1);
    }
    if (post_mode == M_SHARED) {
      Pack pm;
      *reinterpret_cast<V*>(pm.v) = *reinterpret_cast<const V*>(Qs + iq);
#pragma unroll
      for (int kk = 0; kk < VEC; ++kk) dv[kk].set(pm.v[kk]);
    }
    if (ma_mode == M_SHARED) {
      *reinterpret_cast<V*>(ma_v.v) = *reinterpret_cast<const V*>(MAs + ima);
      if (edge_lane) ma_nb = MAs[ima + nbi];
    }
    if (mb_mode == M_SHARED) {
      *reinterpret_cast<V*>(mb0.v) = *reinterpret_cast<const V*>(MBs + imb);
      *reinterpret_cast<V*>(mb1.v) = *reinterpret_cast<const V*>(MBs + imb1);
    }
    if (post_rowsc) {
      const T d = __ldg(s.post.ptr + (int64_t)prc * s.post.sp);
#pragma unroll
      for (int kk = 0; kk < VEC; ++kk) dv[kk].set(d);
    }
    if (ma_rowsc) {
      ma_nb = __ldg(s.ma.ptr + (int64_t)prc * s.ma.sp);
#pragma unroll
      for (int kk = 0; kk < VEC; ++kk) ma_v.v[kk] = ma_nb;
    }
    if (mb_rowsc) {
      const T m0 = __ldg(s.mb.ptr + s0c * s.mb.sp);
      const T m1 = __ldg(s.mb.ptr + s1c * s.mb.sp);
#pragma unroll
      for (int kk = 0; kk < VEC; ++kk) {
        mb0.v[kk] = m0;
        mb1.v[kk] = m1;
      }
    }
    T* op = s.out + (int64_t)z0 * ostride + (int64_t)prow * fsp + x;

#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (u >= nz) break;  // block-uniform
      const int64_t z = z0 + u;
      // ---- row term: B x mb at source rows s0, s1
      Pack b0, b1;
      *reinterpret_cast<V*>(b0.v) = *reinterpret_cast<const V*>(Bs + u * b_ls);
      *reinterpret_cast<V*>(b1.v) = *reinterpret_cast<const V*>(Bs + u * b_ls + b_rs);
      if (mb_level) {
        if (mb_mode == M_FULL) {
          *reinterpret_cast<V*>(mb0.v) = *reinterpret_cast<const V*>(MBs + u * b_ls + ib);
          *reinterpret_cast<V*>(mb1.v) = *reinterpret_cast<const V*>(MBs + u * b_ls + ib + b_rs);
        } else {
          const T m0 = __ldg(s.mb.ptr + z * s.mb.sz + s0c * s.mb.sp);
          const T m1 = __ldg(s.mb.ptr + z * s.mb.sz + s1c * s.mb.sp);
#pragma unroll
          for (int kk = 0; kk < VEC; ++kk) {
            mb0.v[kk] = m0;
            mb1.v[kk] = m1;
          }
        }
      }
#pragma unroll
      for (int kk = 0; kk < VEC; ++kk) {
        b0.v[kk] = b0.v[kk] * mb0.v[kk];
        b1.v[kk] = b1.v[kk] * mb1.v[kk];
      }
      if (low_b || high_b) {
        // (B x mb)[z, row, x .. x + VEC) from global memory: wrap-around and extrapolation partners.  The spare
        // lanes of the last, partial x tile (x >= n, nothing stored) load at the row's last vector instead
        const int xl = x < n ? x : (int)n - VEC;
        auto Brow = [&](int64_t row) -> Pack {
          Pack r = xg_ld_cached<T, VEC>(s.b + z * bsz + row * fsp + xl);
          if (mb_mode != M_NONE) {
#pragma unroll
            for (int kk = 0; kk < VEC; ++kk)
              r.v[kk] = r.v[kk] * __ldg(s.mb.ptr + z * s.mb.sz + row * s.mb.sp + (int64_t)(xl + kk) * s.mb.sx);
          }
          return r;
        };
        if (low_b) {  // s0 == -1
          if (s.halo_lo) b0 = xg_ld_cached<T, VEC>(s.halo_lo + z * n + xl);
          else if (s.bc_b == XG_BC_FILL) {
#pragma unroll
            for (int kk = 0; kk < VEC; ++kk) b0.v[kk] = s.fill_b;
          } else if (s.bc_b == XG_BC_PERIODIC) b0 = Brow(Pb - 1);
          else if (s.bc_b == XG_BC_EXTEND) b0 = b1;
          else {
            const Pack nxt = Brow(Pb > 1 ? 1 : 0);
#pragma unroll
            for (int kk = 0; kk < VEC; ++kk) b0.v[kk] = T(2) * b1.v[kk] - nxt.v[kk];
          }
        }
        if (high_b) {  // s1 == Pb
          if (s.halo_hi) b1 = xg_ld_cached<T, VEC>(s.halo_hi + z * n + xl);
          else if (s.bc_b == XG_BC_FILL) {
#pragma unroll
            for (int kk = 0; kk < VEC; ++kk) b1.v[kk] = s.fill_b;
          } else if (s.bc_b == XG_BC_PERIODIC) b1 = Brow(0);
          else if (s.bc_b == XG_BC_EXTEND) b1 = b0;
          else {
            const Pack prv = Brow(Pb > 1 ? Pb - 2 : 0);
#pragma unroll
            for (int kk = 0; kk < VEC; ++kk) b1.v[kk] = T(2) * b0.v[kk] - prv.v[kk];
          }
        }
      }
      Pack res;
#pragma unroll
      for (int kk = 0; kk < VEC; ++kk) res.v[kk] = xg_apply_op<T, OPB>(b0.v[kk], b1.v[kk]);

      // ---- x term: A x ma, neighbour from the adjacent lane
      if (HAS_A) {
        Pack v;
        *reinterpret_cast<V*>(v.v) = *reinterpret_cast<const V*>(As + u * LSA);
        T enb = T(0);
        if (edge_lane) enb = As[u * LSA + nbi];
        if (ma_level) {
          if (ma_mode == M_FULL) {
            *reinterpret_cast<V*>(ma_v.v) = *reinterpret_cast<const V*>(MAs + u * LSA + ia);
            if (edge_lane) ma_nb = MAs[u * LSA + ia + nbi];
          } else {
            ma_nb = __ldg(s.ma.ptr + z * s.ma.sz + (int64_t)prc * s.ma.sp);
#pragma unroll
            for (int kk = 0; kk < VEC; ++kk) ma_v.v[kk] = ma_nb;
          }
        }
#pragma unroll
        for (int kk = 0; kk < VEC; ++kk) v.v[kk] = v.v[kk] * ma_v.v[kk];
        enb = enb * ma_nb;
        T nb = lo_a ? __shfl_up_sync(FULL, v.v[VEC - 1], 1) : __shfl_down_sync(FULL, v.v[0], 1);
        if (edge_lane) nb = enb;
        if (at_edge) {
          if (s.bc_a == XG_BC_FILL) nb = s.fill_a;
          else if (s.bc_a == XG_BC_PERIODIC) {
            const int64_t xx = lo_a ? n - 1 : 0;
            nb = __ldg(s.a + z * ostride + (int64_t)prc * fsp + xx);
            if (ma_mode != M_NONE) nb = nb * __ldg(s.ma.ptr + z * s.ma.sz + (int64_t)prc * s.ma.sp + xx * s.ma.sx);
          } else nb = lo_a ? v.v[0] : v.v[VEC - 1];  // extend
        }
#pragma unroll
        for (int kk = 0; kk < VEC; ++kk) {
          const T lo_v = kk == 0 ? nb : v.v[kk > 0 ? kk - 1 : 0];
          const T hi_v = kk == VEC - 1 ? nb : v.v[kk < VEC - 1 ? kk + 1 : kk];
          const T ta = lo_a ? xg_apply_op<T, OPA>(lo_v, v.v[kk]) : xg_apply_op<T, OPA>(v.v[kk], hi_v);
          const T tb = res.v[kk];
          res.v[kk] = sub == 0 ? ta + tb : (sub == 1 ? ta - tb : tb - ta);
        }
      }
      // ---- divide
      if (post_level) {
        if (post_mode == M_SCALAR) {
          XgSharedDivisor<T> d;
          d.set(__ldg(s.post.ptr + z * s.post.sz + (int64_t)prc * s.post.sp));
#pragma unroll
          for (int kk = 0; kk < VEC; ++kk) res.v[kk] = d.div(res.v[kk]);
        } else {
          Pack pm;
          *reinterpret_cast<V*>(pm.v) = *reinterpret_cast<const V*>(Qs + u * q_ls + ib);
#pragma unroll
          for (int kk = 0; kk < VEC; ++kk) res.v[kk] = res.v[kk] / pm.v[kk];
        }
      } else {
#pragma unroll
        for (int kk = 0; kk < VEC; ++kk) res.v[kk] = dv[kk].div(res.v[kk]);
      }
      if (act) xg_st_stream<T, VEC>(op + u * ostride, res);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive_tile(empty_u32 + 8u * b);  // this warp is done with stage b
    ++k;
  }
}

int tile_env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return (e && *e) ? atoi(e) : dflt;
}

// NONE / FULL / SHARED / SCALAR from the (z, p, x) strides; -1 when a tensor map cannot describe the operand
template <typename T>
int metric_mode(const XgTileOperand<T>& m, int vec, int64_t rows, int* row0) {
  *row0 = 0;
  if (!m.ptr) return M_NONE;
  if (m.sx == 0) return M_SCALAR;
  if (m.sx != 1) return -1;
  if ((uintptr_t)m.ptr % 16 != 0 || m.sp % vec != 0 || m.sz % vec != 0 || m.sp < 0 || m.sz < 0) return -1;
  if (m.sz == 0) {
    *row0 = m.sp == 0;
    return M_SHARED;
  }
  if (m.sp == 0 && rows > 1) return -1;  // hFac(Z, 1, X): no row stride for the map
  return M_FULL;
}

}  // namespace

template <typename T>
int xg_tile_stencil(const XgTileSpec<T>& s, cudaStream_t st, bool* launched, const char* label) {
  typedef TileGeo<T> G;
  constexpr int VEC = G::VEC, TXE = G::TXE, TY = G::TY, U = kU, BOXW = TXE + VEC;
  *launched = false;
  static const int enabled = tile_env_int("XG_TILE_TMA", 1);
  if (!enabled || !s.b || !s.out) return XG_OK;
  // (tile coordinates are 32-bit: extents below 2^30 leave room for the tile overhang)
  if (s.n < 2 * TXE || s.n % VEC != 0 || s.n >= (1ll << 30) || s.Zn < 2 || s.Zn >= (1ll << 30)) return XG_OK;
  if (s.Pb < 1 || s.Po < 1 || s.Pb >= (1ll << 30) || s.Po >= (1ll << 30)) return XG_OK;
  if (s.f_sp % VEC != 0 || s.b_sz % VEC != 0 || s.o_sz % VEC != 0 || s.f_sp <= 0 || s.b_sz <= 0 || s.o_sz <= 0) return XG_OK;
  if (((uintptr_t)s.b | (uintptr_t)s.out | (uintptr_t)s.a | (uintptr_t)s.halo_lo | (uintptr_t)s.halo_hi) % 16 != 0)
    return XG_OK;
  if (s.a && (s.Po != s.Pb || s.bc_a == XG_BC_EXTRAPOLATE || s.bc_a == XG_BC_NONE)) return XG_OK;
  if (s.a && (s.op_a > XG_OP_INTERP || s.op_b > XG_OP_INTERP)) return XG_OK;  // min / max pairs: k_stencil_pair
  TileArgs<T> a;
  a.s = s;
  a.swap = (s.b_sz < s.f_sp && s.Pb > 1) ? 1 : 0;
  if (a.swap && (s.a || s.o_sz >= s.f_sp)) return XG_OK;  // the x term's boxes are (level, row, x) only
  a.ma_mode = s.a ? metric_mode<T>(s.ma, VEC, s.Po, &a.ma_row0) : M_NONE;
  a.mb_mode = metric_mode<T>(s.mb, VEC, s.Pb, &a.mb_row0);
  a.post_mode = metric_mode<T>(s.post, VEC, s.Po, &a.post_row0);
  if (a.ma_mode < 0 || a.mb_mode < 0 || a.post_mode < 0) return XG_OK;
  // the point of the single-field kernel is the shared divisor / the shared metric tiles: without any, the
  // register-staged kernels do as well
  // (the two-field composite is faster here even without metrics: 1.37 vs 1.52 ms at C3, profiles/r2_pair_tma.txt)
  static const int always = tile_env_int("XG_TILE_ALWAYS", 0);  // benchmarking: take every call
  if (!always && !s.a && a.post_mode != M_SHARED && a.post_mode != M_SCALAR && a.mb_mode != M_SHARED) return XG_OK;
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return XG_OK;

  auto up128 = [](size_t v) { return (unsigned)((v + 127) / 128 * 128); };
  const unsigned a3 = BOXW * TY * U * sizeof(T), a2 = BOXW * TY * sizeof(T);
  const unsigned b3 = TXE * (TY + 1) * U * sizeof(T), b2 = TXE * (TY + 1) * sizeof(T);
  const unsigned q3 = TXE * TY * U * sizeof(T), q2 = TXE * TY * sizeof(T);
  unsigned off = 0, tx = 0;
  if (s.a) { off += up128(a3); tx += a3; }
  a.off_b = off; off += up128(b3); tx += b3;
  a.off_ma = off;
  if (a.ma_mode == M_FULL) { off += up128(a3); tx += a3; }
  else if (a.ma_mode == M_SHARED) { off += up128(a2); tx += a2; }
  a.off_mb = off;
  if (a.mb_mode == M_FULL) { off += up128(b3); tx += b3; }
  else if (a.mb_mode == M_SHARED) { off += up128(b2); tx += b2; }
  a.off_post = off;
  if (a.post_mode == M_FULL) { off += up128(q3); tx += q3; }
  else if (a.post_mode == M_SHARED) { off += up128(q2); tx += q2; }
  a.stage_bytes = off + 128;  // slack: spare thread slots of the last row read (never use) up to one vector past a box
  a.tx_bytes = tx;

  int dev = 0, sms = 148, smem_sm = 0, smem_max = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
  cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  static const int tune_nst = tile_env_int("XG_TILE_NST", 0);
  static const int tune_ctas = tile_env_int("XG_TILE_CTAS", 0);
  int ctas = (!s.a && 3 * 2 * (int)a.stage_bytes <= 135 * 1024) ? 3 : 2;  // as for k_stencil_row_tma
  if (tune_ctas >= 1 && tune_ctas <= (s.a ? 2 : 3)) ctas = tune_ctas;
  int nst = 0;
  for (; ctas >= 1; --ctas) {
    int per_cta = smem_sm / ctas - 1024;
    if (per_cta > smem_max) per_cta = smem_max;
    nst = (per_cta - 128) / (int)a.stage_bytes;
    if (nst >= 2 || (ctas == 1 && nst >= 1)) break;
  }
  if (ctas < 1 || nst < 1) return XG_OK;
  if (tune_nst > 0) nst = tune_nst < nst ? tune_nst : nst;
  else if (nst > 2) nst = 2;
  a.nst = nst;
  static const int tune_hint = tile_env_int("XG_TILE_HINT", 0);
  a.l2_hints = tune_hint;

  const int64_t ntx = xg_ceil_div(s.n, TXE);
  a.npq = xg_ceil_div(s.Po, TY);
  static const int tune_rb = tile_env_int("XG_TILE_RB", 128);
  const int64_t rbq_target = xg_ceil_div(tune_rb > 0 ? tune_rb : 128, TY);
  const int64_t nrb = xg_ceil_div(a.npq, rbq_target);
  const int64_t rbq = xg_ceil_div(a.npq, nrb);
  const int64_t nzq = xg_ceil_div(s.Zn, U);
  a.ntiles = nrb * nzq * rbq * ntx;
  if (a.ntiles >= (1ll << 31)) return XG_OK;
  a.fd_ntx = xg_fastdiv_make(ntx);
  a.fd_rbq = xg_fastdiv_make(rbq);
  a.fd_nzq = xg_fastdiv_make(nzq);

  // tensor maps: fields as (n, rows, Zn); shared metrics as (n, rows) (or (n, 1) when row-less)
  // the encoder wants ascending strides: (x, row, level) normally, (x, level, row) when the levels are the faster dim
  auto field_map = [&](CUtensorMap* map, const T* ptr, int64_t rows, int64_t sp, int64_t sz, int boxw, int boxr) -> int {
    if (sp == 0) sp = s.n;  // single row
    if ((sz < sp) != (a.swap != 0) && rows > 1) return 1;
    if (a.swap) {
      const cuuint64_t d3[3] = {(cuuint64_t)s.n, (cuuint64_t)s.Zn, (cuuint64_t)rows};
      const cuuint64_t s3[2] = {(cuuint64_t)sz * sizeof(T), (cuuint64_t)sp * sizeof(T)};
      const cuuint32_t bx[3] = {(cuuint32_t)boxw, (cuuint32_t)U, (cuuint32_t)boxr};
      return xg_encode_map<T>(enc, map, ptr, 3, d3, s3, bx);
    }
    const cuuint64_t d3[3] = {(cuuint64_t)s.n, (cuuint64_t)rows, (cuuint64_t)s.Zn};
    const cuuint64_t s3[2] = {(cuuint64_t)sp * sizeof(T), (cuuint64_t)sz * sizeof(T)};
    const cuuint32_t bx[3] = {(cuuint32_t)boxw, (cuuint32_t)boxr, (cuuint32_t)U};
    return xg_encode_map<T>(enc, map, ptr, 3, d3, s3, bx);
  };
  auto rows_map = [&](CUtensorMap* map, const XgTileOperand<T>& m, bool row0, int64_t rows, int boxw, int boxr) -> int {
    const cuuint64_t d2[2] = {(cuuint64_t)s.n, (cuuint64_t)(row0 ? 1 : rows)};
    const cuuint64_t s2[1] = {(cuuint64_t)(row0 ? s.n : m.sp) * sizeof(T)};
    const cuuint32_t bx[2] = {(cuuint32_t)boxw, (cuuint32_t)boxr};
    return xg_encode_map<T>(enc, map, m.ptr, 2, d2, s2, bx);
  };
  CUtensorMap map_a, map_b, map_ma, map_mb, map_post;
  if (field_map(&map_b, s.b, s.Pb, s.f_sp, s.b_sz, TXE, TY + 1)) return XG_OK;
  map_a = map_ma = map_mb = map_post = map_b;
  if (s.a && field_map(&map_a, s.a, s.Po, s.f_sp, s.o_sz, BOXW, TY)) return XG_OK;
  if (a.ma_mode == M_FULL && field_map(&map_ma, s.ma.ptr, s.Po, s.ma.sp, s.ma.sz, BOXW, TY)) return XG_OK;
  if (a.ma_mode == M_SHARED && rows_map(&map_ma, s.ma, a.ma_row0 != 0, s.Po, BOXW, TY)) return XG_OK;
  if (a.mb_mode == M_FULL && field_map(&map_mb, s.mb.ptr, s.Pb, s.mb.sp, s.mb.sz, TXE, TY + 1)) return XG_OK;
  if (a.mb_mode == M_SHARED && rows_map(&map_mb, s.mb, a.mb_row0 != 0, s.Pb, TXE, TY + 1)) return XG_OK;
  if (a.post_mode == M_FULL && field_map(&map_post, s.post.ptr, s.Po, s.post.sp, s.post.sz, TXE, TY)) return XG_OK;
  if (a.post_mode == M_SHARED && rows_map(&map_post, s.post, a.post_row0 != 0, s.Po, TXE, TY)) return XG_OK;

  const size_t smem = 128 + (size_t)nst * a.stage_bytes;
  int64_t grid = (int64_t)ctas * sms;
  if (grid > a.ntiles) grid = a.ntiles;
  auto go = [&](auto kern) -> int {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      cudaGetLastError();
      return 0;
    }
    kern<<<(unsigned)grid, kConsumers + 32, smem, st>>>(map_a, map_b, map_ma, map_mb, map_post, a);
    return 1;
  };
  auto per_level = [](int mode, const XgTileOperand<T>& m) { return mode == M_FULL || (mode == M_SCALAR && m.sz != 0); };
  const bool levelm = per_level(a.ma_mode, s.ma) || per_level(a.mb_mode, s.mb) || per_level(a.post_mode, s.post);
  int ok = 0;
#define XG_TILE_GO(HAS_A_, OPA_, OPB_) \
  ok = levelm ? go(k_tile_stencil<T, HAS_A_, OPA_, OPB_, true>) : go(k_tile_stencil<T, HAS_A_, OPA_, OPB_, false>)
  if (s.a) {
    switch (s.op_a * 4 + s.op_b) {
      case XG_OP_DIFF * 4 + XG_OP_DIFF: XG_TILE_GO(true, XG_OP_DIFF, XG_OP_DIFF); break;
      case XG_OP_DIFF * 4 + XG_OP_INTERP: XG_TILE_GO(true, XG_OP_DIFF, XG_OP_INTERP); break;
      case XG_OP_INTERP * 4 + XG_OP_DIFF: XG_TILE_GO(true, XG_OP_INTERP, XG_OP_DIFF); break;
      case XG_OP_INTERP * 4 + XG_OP_INTERP: XG_TILE_GO(true, XG_OP_INTERP, XG_OP_INTERP); break;
      default: break;
    }
  } else {
    switch (s.op_b) {
      case XG_OP_DIFF: XG_TILE_GO(false, XG_OP_DIFF, XG_OP_DIFF); break;
      case XG_OP_INTERP: XG_TILE_GO(false, XG_OP_DIFF, XG_OP_INTERP); break;
      case XG_OP_MIN: XG_TILE_GO(false, XG_OP_DIFF, XG_OP_MIN); break;
      case XG_OP_MAX: XG_TILE_GO(false, XG_OP_DIFF, XG_OP_MAX); break;
      default: break;
    }
  }
#undef XG_TILE_GO
  if (!ok) return XG_OK;
  *launched = true;
  return xg_check_launch(label);
}

template int xg_tile_stencil<float>(const XgTileSpec<float>&, cudaStream_t, bool*, const char*);
template int xg_tile_stencil<double>(const XgTileSpec<double>&, cudaStream_t, bool*, const char*);
