// xg_multi_tile — the TMA-staged form of xg_stencil_multi for the common chain order "innermost axis
// first": Grid.interp(da, ['X', 'Y']), ['X', 'Y', 'Z'], ['Y', 'Z'] (and diff / min / max) on a field seen
// as (levels, rows, x), every op length preserving (center <-> left / right).
//
//     out = OPz(pad_z( OPp(pad_p( OPx(pad_x(a)) )) ))        each intermediate rounded to the field dtype
//
// Same values as K consecutive xg_stencil2 calls (xgcm/grid.py:798-832), like k_stencil_multi; what
// changes is the data movement.  A tile is U = 4 levels x TY rows x TXE cells of the OUTPUT; its input is
// ONE bulk tensor load of (TXE + a 16-byte x halo) x (TY + 1 rows) x (U + 1 levels) (halo only along
// operated axes), completing on an mbarrier; a persistent CTA = 8 consumer warps + 1 producer warp around
// a ring of two tiles.  Each input cell is read from shared memory by the up to 2^K outputs that need it,
// the x neighbour comes from a warp shuffle, the level chain carries the previous level's (x, p) result
// in registers: per output vector 1 + 1 (+ 1) operator evaluations on top of the two x evaluations.
//
// Boundaries.  `periodic` and `extend` padding copy whole rows / planes / cells, so they commute with the
// operators along the OTHER axes: pad_p(OPx(a)) == OPx(pad_p(a)).  A tile that touches such a boundary
// therefore materialises the padded INPUT first (the out-of-array part of its box, zero-filled by the TMA
// unit, is overwritten with the wrapped / clamped cells from global memory: one cell, row or plane slab),
// then runs the same code as an interior tile.  `fill` does not commute (the padded intermediate is the
// constant, whatever the inner operators would have produced), so it is applied where it belongs: the
// operand of the op whose axis left the array is replaced by that op's fill value.
#include <stdlib.h>

#include <type_traits>

#include "xg_stencil_tile.cuh"
#include "xg_tma.cuh"

namespace {

constexpr int kConsumersM = 256;
constexpr int kUM = 4;

template <typename T>
struct MultiGeo;
template <>
struct MultiGeo<float> {
  static constexpr int VEC = 4, TXE = 224, TY = 4;
};
template <>
struct MultiGeo<double> {
  static constexpr int VEC = 2, TXE = 240, TY = 2;
};

template <typename T>
struct MultiTileArgs {
  XgMultiTileSpec<T> s;
  int hp, hz;          // halo rows / levels in the box (the axis is operated)
  int ox, op, oz;      // box origin relative to the tile origin: cells / rows / levels before it
  int64_t npq, ntiles;  // tile rows; virtual tiles = nrb * nzq * rbq * ntx (tile rows past npq are skipped)
  XgFastDiv fd_ntx, fd_rbq, fd_nzq;
  int nst;
  unsigned stage_bytes, tx_bytes;
};

__device__ __forceinline__ void mbar_arrive_multi(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// HX / HP / HZ: which of x, rows, levels are operated — compile-time, so box pitches are constants and the
// chain is straight-line code (the first version decided these at run time: 860 warp instructions per
// tile-warp, 17 % of them the operators; profiles/r2_ncu_multi_xyz_tma_v1_summary.json)
// LOX: the x op reads its lower (1) or upper (0) neighbour — compile-time too (a run-time choice cost a select per cell)
template <typename T, int OP, bool HX, bool HP, bool HZ, int LOX>
__global__ void __launch_bounds__(kConsumersM + 32, 3)
    k_tile_multi(const __grid_constant__ CUtensorMap map_in, const MultiTileArgs<T> a) {
  typedef MultiGeo<T> G;
  constexpr int VEC = G::VEC, TXE = G::TXE, TY = G::TY, U = kUM;
  constexpr int BOXW = TXE + VEC, LR = kConsumersM / TY, NVR = TXE / VEC;
  typedef XgPack<T, VEC> Pack;
  typedef typename XgVec<T, VEC>::type V;
  const unsigned FULL = 0xffffffffu;
  const XgMultiTileSpec<T>& s = a.s;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x;
  const int NST = a.nst;
  const uint32_t full_u32 = smem_u32(smem_raw);
  const uint32_t empty_u32 = full_u32 + 8u * NST;
  unsigned char* stage0 = smem_raw + 128;
  const int64_t nloc = (a.ntiles > blockIdx.x) ? (a.ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
  constexpr int rows_box = TY + (HP ? 1 : 0), lvl_pitch = rows_box * BOXW, HZI = HZ ? 1 : 0;

  // row blocks (~128 rows) outermost, then the level batches: the halo level of a batch is re-read from L2,
  // not DRAM, by the next batch.  false for the padding rows of the last row block.
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
      mbar_init(empty_u32 + 8u * b, kConsumersM / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (tid >= kConsumersM) {
    if (tid == kConsumersM) {  // ---- producer
      int64_t k = 0;
      for (int64_t i = 0; i < nloc; ++i) {
        int z0, p0, x0;
        if (!tile_geom(i, z0, p0, x0)) continue;
        const int b = (int)(k % NST);
        if (k >= NST) mbar_wait(empty_u32 + 8u * b, (uint32_t)(((k / NST) - 1) & 1));
        ++k;
        const uint32_t bar = full_u32 + 8u * b;
        mbar_expect_tx(bar, a.tx_bytes);
        tensor_load_3d(smem_u32(stage0 + (size_t)b * a.stage_bytes), &map_in, x0 - a.ox, p0 - a.op, z0 - a.oz, bar);
      }
    }
    return;
  }

  // ---- consumers
  const int lane = tid & 31;
  const int ty = tid / LR, vx = tid - ty * LR;
  const int vxs = vx < NVR ? vx : NVR - 1;
  constexpr bool has_x = HX, has_p = HP, has_z = HZ;
  constexpr int lo_x = LOX;
  const int lo_p = s.lo[1], lo_z = s.lo[2];
  const int nbi = lo_x ? -1 : VEC;
  const bool edge_lane = lo_x ? (lane == 0) : (lane == 31 || vx >= NVR - 1);
  const int64_t n = s.n, P = s.P, L = s.L;
  // axes whose padded input has to be materialised (periodic / extend); fill is applied in the chain
  const bool mat_x = has_x && s.bc[0] != XG_BC_FILL, mat_p = has_p && s.bc[1] != XG_BC_FILL;
  const bool mat_z = has_z && s.bc[2] != XG_BC_FILL;
  const bool fill_x = has_x && s.bc[0] == XG_BC_FILL, fill_p = has_p && s.bc[1] == XG_BC_FILL;
  const bool fill_z = has_z && s.bc[2] == XG_BC_FILL;

  int64_t k = 0;
  for (int64_t i = 0; i < nloc; ++i) {
    int z0, p0, x0;
    if (!tile_geom(i, z0, p0, x0)) continue;
    const int b = (int)(k % NST);
    const uint32_t full_parity = (uint32_t)((k / NST) & 1);
    ++k;
    T* tile = reinterpret_cast<T*>(stage0 + (size_t)b * a.stage_bytes);
    const int x = x0 + vxs * VEC, prow = p0 + ty;
    const bool act = vx < NVR && x < n && prow < P;
    const int nz = (L - z0 < U) ? (int)(L - z0) : U;
    mbar_wait(full_u32 + 8u * b, full_parity);

    // ---- materialise the padded input where the box left the array along a periodic / extend axis
    const int gx0 = x0 - a.ox, gp0 = p0 - a.op, gz0 = z0 - a.oz;  // global coordinates of the box origin
    const bool out_x = mat_x && (gx0 < 0 || gx0 + BOXW > n), out_p = mat_p && (gp0 < 0 || gp0 + rows_box > P);
    const bool out_z = mat_z && (gz0 < 0 || gz0 + nz + HZI > L);
    if (out_x || out_p || out_z) {  // block-uniform
      const int lvls = nz + HZI;
      // source coordinate of a box coordinate along one axis: in range -> itself (flag stays), outside ->
      // wrapped / clamped when the axis is materialised, else "irrelevant" (never read, or replaced by fill)
      auto src = [&](int g, int64_t len, bool mat, int bc, bool& need, bool& skip) -> int64_t {
        if (g >= 0 && g < len) return g;
        if (!mat) { skip = true; return 0; }
        need = true;
        if (bc == XG_BC_PERIODIC) return g < 0 ? g + len : g - len;
        return g < 0 ? 0 : len - 1;
      };
      auto fix = [&](int lz, int lp, int lx) {
        bool need = false, skip = false;
        const int64_t sz_ = src(gz0 + lz, L, mat_z, s.bc[2], need, skip);
        const int64_t sp_ = src(gp0 + lp, P, mat_p, s.bc[1], need, skip);
        const int64_t sx_ = src(gx0 + lx, n, mat_x, s.bc[0], need, skip);
        if (need && !skip) tile[lz * lvl_pitch + lp * BOXW + lx] = __ldg(s.in + (sz_ * P + sp_) * n + sx_);
      };
      if (out_x) {  // one cell per (level, row): the element the lower / upper neighbour reads
        const int lx = lo_x ? a.ox - 1 : (int)(n - x0);  // global -1 (first tile of a row) / global n (last tile)
        if (lo_x ? (x0 == 0) : (lx <= TXE))
          for (int c = tid; c < lvls * rows_box; c += kConsumersM) fix(c / rows_box, c % rows_box, lx);
      }
      if (out_p) {  // the box rows just outside the array
        if (gp0 < 0)
          for (int c = tid; c < lvls * BOXW; c += kConsumersM) fix(c / BOXW, 0, c % BOXW);
        const int lp = (int)(P - gp0);
        if (lp < rows_box)
          for (int c = tid; c < lvls * BOXW; c += kConsumersM) fix(c / BOXW, lp, c % BOXW);
      }
      if (out_z) {  // the box levels just outside the array
        if (gz0 < 0)
          for (int c = tid; c < rows_box * BOXW; c += kConsumersM) fix(0, c / BOXW, c % BOXW);
        const int lz = (int)(L - gz0);
        if (lz < lvls)
          for (int c = tid; c < rows_box * BOXW; c += kConsumersM) fix(lz, c / BOXW, c % BOXW);
      }
      // the cells above are generic-proxy writes into a stage the producer later refills through the async
      // proxy (cp.async.bulk.tensor): order them before this thread's share of the empty-barrier arrive
      fence_async_smem();
      asm volatile("bar.sync 1, %0;" ::"r"(kConsumersM) : "memory");
    }

    // ---- the chain.  A tile next to a `fill` boundary runs the copy with the operand overrides compiled in.
    const bool at_edge_x = lo_x ? (x == 0) : (x + VEC >= n);
    const int s0p = prow - lo_p, s1p = s0p + 1;  // source rows of the p op for this output row
    const bool fill_tile = (fill_x && (x0 == 0 || x0 + TXE >= n)) || (fill_p && (gp0 < 0 || gp0 + rows_box > P)) ||
                           (fill_z && (gz0 < 0 || gz0 + nz + HZI > L));
    const T* trow = tile + ty * BOXW + vxs * VEC + a.ox;  // this thread's vector in (level 0, row ty) of the box
    T* op_ = s.out + ((int64_t)z0 * P + prow) * n + x;
    const int64_t ostride = P * n;
    auto chain = [&](auto fill_tag) {
      constexpr bool FT = decltype(fill_tag)::value;
      // OPx on one box row (or the raw row when x is not operated)
      auto Xrow = [&](const T* rp) -> Pack {
        Pack v;
        *reinterpret_cast<V*>(v.v) = *reinterpret_cast<const V*>(rp);
        if constexpr (!has_x) {
          return v;
        } else {
          T nb = lo_x ? __shfl_up_sync(FULL, v.v[VEC - 1], 1) : __shfl_down_sync(FULL, v.v[0], 1);
          if (edge_lane) nb = rp[nbi];
          if (FT && fill_x && at_edge_x) nb = s.fill[0];
          Pack r;
#pragma unroll
          for (int kk = 0; kk < VEC; ++kk) {
            const T lo_v = kk == 0 ? nb : v.v[kk > 0 ? kk - 1 : 0];
            const T hi_v = kk == VEC - 1 ? nb : v.v[kk < VEC - 1 ? kk + 1 : kk];
            r.v[kk] = lo_x ? xg_apply_op<T, OP>(lo_v, v.v[kk]) : xg_apply_op<T, OP>(v.v[kk], hi_v);
          }
          return r;
        }
      };
      // OPp(OPx) at box level lz for this thread's output row
      auto XP = [&](int lz) -> Pack {
        Pack x0v = Xrow(trow + lz * lvl_pitch);
        if constexpr (!has_p) {
          return x0v;
        } else {
          Pack x1v = Xrow(trow + lz * lvl_pitch + BOXW);
          if (FT && fill_p) {
            if (s0p < 0) {
#pragma unroll
              for (int kk = 0; kk < VEC; ++kk) x0v.v[kk] = s.fill[1];
            }
            if (s1p >= P) {
#pragma unroll
              for (int kk = 0; kk < VEC; ++kk) x1v.v[kk] = s.fill[1];
            }
          }
          Pack r;
#pragma unroll
          for (int kk = 0; kk < VEC; ++kk) r.v[kk] = xg_apply_op<T, OP>(x0v.v[kk], x1v.v[kk]);
          return r;
        }
      };
      Pack prev;
      if constexpr (has_z) prev = XP(0);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (u >= nz) break;  // block-uniform
        Pack res;
        if constexpr (has_z) {
          const Pack cur = XP(u + 1);
          Pack a0 = prev, a1 = cur;
          if (FT && fill_z) {
            const int64_t zs0 = (int64_t)z0 + u - lo_z;
            if (zs0 < 0) {
#pragma unroll
              for (int kk = 0; kk < VEC; ++kk) a0.v[kk] = s.fill[2];
            }
            if (zs0 + 1 >= L) {
#pragma unroll
              for (int kk = 0; kk < VEC; ++kk) a1.v[kk] = s.fill[2];
            }
          }
#pragma unroll
          for (int kk = 0; kk < VEC; ++kk) res.v[kk] = xg_apply_op<T, OP>(a0.v[kk], a1.v[kk]);
          prev = cur;
        } else {
          res = XP(u);
        }
        if (act) xg_st_stream<T, VEC>(op_ + u * ostride, res);
      }
    };
    if (fill_tile) chain(std::true_type{});
    else chain(std::false_type{});
    __syncwarp();
    if (lane == 0) mbar_arrive_multi(empty_u32 + 8u * b);
  }
}

int multi_env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return (e && *e) ? atoi(e) : dflt;
}

}  // namespace

template <typename T>
int xg_multi_tile(const XgMultiTileSpec<T>& s, cudaStream_t st, bool* launched) {
  typedef MultiGeo<T> G;
  constexpr int VEC = G::VEC, TXE = G::TXE, TY = G::TY, U = kUM, BOXW = TXE + VEC;
  *launched = false;
  static const int enabled = multi_env_int("XG_MULTI_TMA", 1);
  if (!enabled || !s.in || !s.out) return XG_OK;
  if (s.n < 2 * TXE || s.n % VEC != 0 || s.n >= (1ll << 30) || s.P < 1 || s.P >= (1ll << 30) || s.L < 1 ||
      s.L >= (1ll << 30))  // 32-bit tile coordinates
    return XG_OK;
  if (((uintptr_t)s.in | (uintptr_t)s.out) % 16 != 0) return XG_OK;
  if (s.op < XG_OP_DIFF || s.op > XG_OP_MAX) return XG_OK;
  if (s.has[1] && s.P < 2) return XG_OK;
  if (s.has[2] && s.L < 2) return XG_OK;
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return XG_OK;
  MultiTileArgs<T> a;
  a.s = s;
  a.hp = s.has[1] ? 1 : 0;
  a.hz = s.has[2] ? 1 : 0;
  a.ox = (s.has[0] && s.lo[0]) ? VEC : 0;
  a.op = s.has[1] ? s.lo[1] : 0;
  a.oz = s.has[2] ? s.lo[2] : 0;
  const unsigned box_bytes = (unsigned)(BOXW * (TY + a.hp) * (U + a.hz) * sizeof(T));
  a.tx_bytes = box_bytes;
  a.stage_bytes = (box_bytes + 127) / 128 * 128;
  int dev = 0, sms = 148, smem_sm = 0, smem_max = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
  cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  static const int tune_nst = multi_env_int("XG_MULTI_NST", 0);
  static const int tune_ctas = multi_env_int("XG_MULTI_CTAS", 0);
  // measured (profiles/r2_multi_tma_sweep.txt): 3 CTAs x 2 tiles with an x op; without one (Y, Z) 4 CTAs x 1 tile
  int ctas = s.has[0] ? 3 : 4;
  if (tune_ctas >= 1 && tune_ctas <= 4) ctas = tune_ctas;
  int per_cta = smem_sm / ctas - 1024;
  if (per_cta > smem_max) per_cta = smem_max;
  const int fit = (per_cta - 128) / (int)a.stage_bytes;
  int nst = fit < 2 ? fit : 2;
  if (!s.has[0] && tune_ctas == 0) nst = 1;
  if (tune_nst > 0) nst = tune_nst < fit ? tune_nst : fit;
  if (nst < 1) return XG_OK;
  a.nst = nst;
  const int64_t ntx = xg_ceil_div(s.n, TXE);
  a.npq = xg_ceil_div(s.P, TY);
  static const int tune_rb = multi_env_int("XG_MULTI_RB", 128);
  const int64_t rbq_target = xg_ceil_div(tune_rb > 0 ? tune_rb : 128, TY);
  const int64_t nrb = xg_ceil_div(a.npq, rbq_target);
  const int64_t rbq = xg_ceil_div(a.npq, nrb);
  const int64_t nzq = xg_ceil_div(s.L, U);
  a.ntiles = nrb * nzq * rbq * ntx;
  if (a.ntiles >= (1ll << 31)) return XG_OK;
  a.fd_ntx = xg_fastdiv_make(ntx);
  a.fd_rbq = xg_fastdiv_make(rbq);
  a.fd_nzq = xg_fastdiv_make(nzq);
  CUtensorMap map_in;
  const cuuint64_t d3[3] = {(cuuint64_t)s.n, (cuuint64_t)s.P, (cuuint64_t)s.L};
  const cuuint64_t s3[2] = {(cuuint64_t)s.n * sizeof(T), (cuuint64_t)s.P * s.n * sizeof(T)};
  const cuuint32_t bx[3] = {(cuuint32_t)BOXW, (cuuint32_t)(TY + a.hp), (cuuint32_t)(U + a.hz)};
  if (xg_encode_map<T>(enc, &map_in, s.in, 3, d3, s3, bx)) return XG_OK;
  const size_t smem = 128 + (size_t)nst * a.stage_bytes;
  int64_t grid = (int64_t)ctas * sms;
  if (grid > a.ntiles) grid = a.ntiles;
  auto go = [&](auto kern) -> int {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      cudaGetLastError();
      return 0;
    }
    kern<<<(unsigned)grid, kConsumersM + 32, smem, st>>>(map_in, a);
    return 1;
  };
  int ok = 0;
  const int combo = (s.has[0] ? 1 : 0) | (s.has[1] ? 2 : 0) | (s.has[2] ? 4 : 0);
#define XG_MULTI_OPS(HX_, HP_, HZ_, LOX_)                                                 \
  switch (s.op) {                                                                         \
    case XG_OP_DIFF: ok = go(k_tile_multi<T, XG_OP_DIFF, HX_, HP_, HZ_, LOX_>); break;     \
    case XG_OP_INTERP: ok = go(k_tile_multi<T, XG_OP_INTERP, HX_, HP_, HZ_, LOX_>); break; \
    case XG_OP_MIN: ok = go(k_tile_multi<T, XG_OP_MIN, HX_, HP_, HZ_, LOX_>); break;       \
    default: ok = go(k_tile_multi<T, XG_OP_MAX, HX_, HP_, HZ_, LOX_>); break;              \
  }
#define XG_MULTI_LOX(HP_, HZ_)                      \
  if (s.lo[0]) { XG_MULTI_OPS(true, HP_, HZ_, 1) } \
  else { XG_MULTI_OPS(true, HP_, HZ_, 0) }
  switch (combo) {
    case 3: XG_MULTI_LOX(true, false) break;
    case 5: XG_MULTI_LOX(false, true) break;
    case 6: XG_MULTI_OPS(false, true, true, 0) break;
    case 7: XG_MULTI_LOX(true, true) break;
    default: break;
  }
#undef XG_MULTI_LOX
#undef XG_MULTI_OPS
  if (!ok) return XG_OK;
  *launched = true;
  return xg_check_launch("xg_stencil_multi(tile_tma)");
}

template int xg_multi_tile<float>(const XgMultiTileSpec<float>&, cudaStream_t, bool*);
template int xg_multi_tile<double>(const XgMultiTileSpec<double>&, cudaStream_t, bool*);
