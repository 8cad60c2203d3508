// kernels_planner.cu -- K2/K3/K5: the visibility-heuristic planner loop on the device.
//
// Replaces, per problem (map, start, end):
//   visibilityBasedSolver::solve            src/visibilityBasedSolver.cpp:76-160
//   visibilityBasedSolver::updateVisibility src/visibilityBasedSolver.cpp:379-565
//   resetQueue / heap_->top()               :65-71, :130
//   visibilityBasedSolver::reconstructPath  src/visibilityBasedSolver.cpp:1183-1213
//
// One persistent CTA per problem runs the whole data-dependent loop without any
// host round trip:
//   1. sweep from the current light source (the tile-wavefront K1 body of
//      sweep_tile_body.cuh, fp64 store) into the local visibility field `vis`
//      -- the DP part of updateVisibility;
//   2. fused per-cell epilogue over the grid (coalesced): global visibility
//      max-merge (:417-418), first-writer parent (:419-423), heuristic
//      h = scale*vg + (d(cell,end) + d(cell,parent)) (:424-430) and the arg-min
//      that stands for the heap: the reference pushes every visible cell and only
//      ever reads top(), which is the FIRST pushed element attaining the minimum h
//      (Node::operator< is strict).  The push order is quadrant Q1..Q4, i outer,
//      j inner, so the reduction key is (h, quadrant, i, j) with the first
//      quadrant that visits the cell;
//   3. next source = arg-min cell, ++nb_of_sources, max_iter check, end-visible
//      test (:127-140).
// Two exact shortcuts keep the loop cheap:
//   * h of a cell only depends on (vg, end, parent) and the parent never changes once
//     set (:419-423), so h is cached per cell (`hc`) and recomputed only where vg rose or
//     the parent was just assigned; the arg-min then reads 16 bytes per cell and the
//     push-order key is only evaluated for cells that tie or beat the running minimum.
//   * the reference has no closed set: once the arg-min cell IS the current source it is
//     picked again forever (same sweep -> same fields -> same h), until max_iter
//     (SURVEY A.2 item 7).  That fixed point is detected and the remaining identical
//     iterations are not executed: the light-source list is filled with the repeated
//     cell and the status is VHP_MAX_ITER, exactly as the reference ends.
// Afterwards thread 0 walks cameFrom_/lightSources_ from the end point
// (reconstructPath) and sums the segment lengths.
//
// Cells the reference never visits (column 0 / row 0 unless the source lies on
// them, loop bounds :434-438,:478-483,:522-527) get no epilogue.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstdint>

#include "planner_common.cuh"
#include "sweep_tile_body.cuh"

#ifndef VHP_FIRST_U
#define VHP_FIRST_U 4 // cells in flight per lane in the first sweep's epilogue
#endif
#ifndef VHP_EPI_U
#define VHP_EPI_U 4   // ... and in the later ones (four loads per cell)
#endif

namespace {

struct PlannerParams {
  TileArgs fp;
  const int32_t *se_xy, *prob_map;
  double thr;
  int max_iter, ls_cap;
  // working fields, fp64, [nprob][ny][nx]
  double *vis, *vg;
  double *hc;      // cached heuristic h per cell, +inf where the cell has no parent yet
  int32_t *came;
  // small outputs, [nprob]...
  int32_t *status, *nb, *ls, *path_n, *path;
  double *path_len;
  // optional fp32 exports of vg / vis (NULL: none)
  float *vg32, *vis32;
  // non-null: the first sweep and its epilogue were done batch-wide (planner_first_* kernels below);
  // resume[5q ..] = {done, next x, next y, status, nb_of_sources} of problem q after it
  const int *resume;
};

// NWK warps per CTA: 8 by default, capped at 128 registers so that two CTAs share an SM (the
// uncapped build takes 147 registers, one CTA per SM: 192k vs 239k solves/s on the 1024 x 256^2
// batch).  4- and 2-warp CTAs (more problems resident per SM) were measured slower even on
// batches of 256 x 256 maps -- the epilogue pass wants the threads -- and stay selectable with
// VHP_PLANNER_WARPS for experiments.  Also measured and dropped: 6 warps x 3 CTAs per SM and 10
// warps x 2 (both 96 registers: 182k / 180k), 12 warps x 1 (140 registers: 244k, no better).
template <int NWK, int MINB = 1>
__global__ void __launch_bounds__(NWK * 32, MINB) planner_kernel(const PlannerParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_ctl[5];              // {done, next x, next y, status, nb_of_sources}
  __shared__ Best s_best[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, NW = blockDim.x >> 5;
  const int64_t q = blockIdx.x;
  const int nx = p.fp.nx, ny = p.fp.ny;
  const size_t cells = (size_t)nx * ny;
  const int stx = p.se_xy[4 * q], sty = p.se_xy[4 * q + 1];
  const int ex = p.se_xy[4 * q + 2], ey = p.se_xy[4 * q + 3];
  const int map = p.prob_map ? p.prob_map[q] : 0;
  const uint32_t *rowbits = p.fp.pl.rowF + (size_t)map * p.fp.pl.row_plane;
  double *vis = p.vis + q * cells, *vg = p.vg + q * cells, *hc = p.hc + q * cells;
  int32_t *came = p.came + q * cells;
  int32_t *ls = p.ls + q * (size_t)p.ls_cap * 2;
  const double thr = p.thr;

  // reset() (:42-60) happens inside the first sweep's epilogue (epilogue_cell_first)
  if (tid == 0) {
    if (p.resume) { // the state after the batch-wide first sweep
      const int *r = p.resume + 5 * q;
      s_ctl[0] = r[0]; s_ctl[1] = r[1]; s_ctl[2] = r[2]; s_ctl[3] = r[3]; s_ctl[4] = r[4];
    } else {
      s_ctl[3] = planner_validate(rowbits, p.fp.pl.wx, nx, ny, stx, sty, ex, ey);
      s_ctl[1] = stx;
      s_ctl[2] = sty;
      s_ctl[0] = 0;
      s_ctl[4] = 0;
    }
  }
  __syncthreads();
  int status = s_ctl[3];
  int nb = s_ctl[4];
  if (status == VHP_OK) {
    if (tid == 0 && !p.resume) {
      ls[0] = stx; ls[1] = sty;                 // lightSources_[0] = start, :121
      // cameFrom_(start) = 0 (:122) is part of the first epilogue;
      // visibility_global_(end) = 0 (:123) holds after the reset; loop test :127
      s_ctl[0] = !(0.0 <= thr);
    }
    __syncthreads();
    const double scale =
        __dsqrt_rn((double)((unsigned long long)ny * ny + (unsigned long long)nx * nx)); // :49
    int sx = s_ctl[1], sy = s_ctl[2];
    bool done = s_ctl[0] != 0;
    while (!done) {
      // ---- 1. sweep (visibility_.reset() + the DP of updateVisibility)
      tile_sweep_cta<double, NWK>(p.fp, map, sx, sy, vis, smem_raw);
      // ---- 2. per-cell epilogue + arg-min: a warp per grid row, kEpiU cells per lane in flight
      // (one CTA has few threads for a whole map: with one cell in flight per thread the pass was
      // latency-bound at ~1 TB/s in total)
      Best best{~0ull, ~0ull};
      if (nb == 0) {
        // first sweep: the fields are still uninitialised workspace; nothing is loaded, everything
        // stored (reset() :42-60 and the first epilogue in one pass)
        constexpr int kFirstU = VHP_FIRST_U; // cells in flight per lane
        for (int Y = warp; Y < ny; Y += NW) {
          const size_t row = (size_t)Y * nx;
          for (int X0 = lane; X0 < nx; X0 += 32 * kFirstU) {
            double v[kFirstU];
#pragma unroll
            for (int u = 0; u < kFirstU; ++u)
              if (X0 + 32 * u < nx) v[u] = __ldcg(vis + row + X0 + 32 * u);
#pragma unroll
            for (int u = 0; u < kFirstU; ++u)
              if (X0 + 32 * u < nx)
                epilogue_cell_first(X0 + 32 * u, Y, row + X0 + 32 * u, v[u], sx, sy, ex, ey, thr, scale, ls, vg, hc,
                                    came, best);
          }
        }
      } else {
        constexpr int kEpiU = VHP_EPI_U;
        for (int Y = warp; Y < ny; Y += NW) {
          const size_t row = (size_t)Y * nx;
          for (int X0 = lane; X0 < nx; X0 += 32 * kEpiU) {
            double v[kEpiU], h[kEpiU], g0[kEpiU];
            int cf[kEpiU];
#pragma unroll
            for (int u = 0; u < kEpiU; ++u) {
              const int X = X0 + 32 * u;
              if (X < nx) {
                v[u] = __ldcg(vis + row + X);
                h[u] = __ldcg(hc + row + X);
                g0[u] = __ldcg(vg + row + X);
                cf[u] = __ldcg(came + row + X);
              }
            }
#pragma unroll
            for (int u = 0; u < kEpiU; ++u) {
              const int X = X0 + 32 * u;
              if (X < nx)
                epilogue_cell_loaded(X, Y, row + X, v[u], h[u], g0[u], cf[u], sx, sy, ex, ey, thr, scale, nb,
                                     ls, vg, hc, came, best);
            }
          }
        }
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        Best o;
        o.h = __shfl_xor_sync(0xffffffffu, best.h, off);
        o.key = __shfl_xor_sync(0xffffffffu, best.key, off);
        if (better(o, best)) best = o;
      }
      if (lane == 0) s_best[warp] = best;
      __syncthreads();
      if (warp == 0) {
        Best b = lane < NW ? s_best[lane] : Best{~0ull, ~0ull};
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          Best o;
          o.h = __shfl_xor_sync(0xffffffffu, b.h, off);
          o.key = __shfl_xor_sync(0xffffffffu, b.key, off);
          if (better(o, b)) b = o;
        }
        if (lane == 0) {
          // ---- 3. heap_->top() -> next light source, :130-139
          int tx, ty, d, st = s_ctl[3];
          const int nnb = planner_next_source(b, sx, sy, nb, p.max_iter, thr,
                                              __ldcg(vg + (size_t)ey * nx + ex), ls, tx, ty, d, st);
          s_ctl[1] = tx;
          s_ctl[2] = ty;
          s_ctl[3] = st;
          s_ctl[0] = d;
          s_ctl[4] = nnb;
        }
      }
      __syncthreads();
      nb = s_ctl[4];
      sx = s_ctl[1];
      sy = s_ctl[2];
      done = s_ctl[0] != 0;
      status = s_ctl[3];
      __syncthreads();
    }
  }

  if (nb == 0) { // no sweep ran: the fields keep the state of reset() (:42-60, :122)
    for (size_t c = tid; c < cells; c += blockDim.x) {
      vis[c] = 0.0;
      vg[c] = 0.0;
      came[c] = (status == VHP_OK && c == (size_t)sty * nx + stx) ? 0 : VHP_NO_PARENT;
    }
  }
  if (tid == 0) {
    p.status[q] = status;
    p.nb[q] = nb;
    int32_t *path = p.path + q * (size_t)p.ls_cap * 2;
    double total;
    const long n = planner_reconstruct(status, nb, ex, ey, nx, p.ls_cap, ls, came, path, total);
    p.path_n[q] = (int32_t)n;
    p.path_len[q] = total;
  }
  __syncthreads();
  if (p.vg32 || p.vis32) {
    for (size_t c = tid; c < cells; c += blockDim.x) {
      if (p.vg32) p.vg32[q * cells + c] = __double2float_rn(__ldcg(vg + c));
      if (p.vis32) p.vis32[q * cells + c] = __double2float_rn(__ldcg(vis + c));
    }
  }
}

// ---- large batches: the FIRST sweep of every problem batch-wide ---------------------------------
// A problem of bench.py's batch runs 1.8 sweeps on average, so more than half of all sweeps are
// first sweeps.  Inside the persistent kernel a sweep and its epilogue are bound by latency at
// 16 warps per SM; as one launch of the batched sweep kernel (K1: one single-warp CTA per problem,
// 24 per SM) followed by one launch of the epilogue over all problems at full occupancy they run
// near the instruction / HBM limits instead.  The persistent kernel then resumes every problem
// from its second sweep.  Same device functions, same results.
constexpr int kFirstSlabs = 8; // CTAs per problem in the batch-wide epilogue

__global__ void planner_first_begin_kernel(const VhpTilePlanes pl, int nx, int ny, const int32_t *se_xy,
                                           const int32_t *prob_map, double thr, int32_t *ls_all, int ls_cap,
                                           int32_t *src_xy, int *ctl, int64_t nprob) {
  const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q >= nprob) return;
  const int stx = se_xy[4 * q], sty = se_xy[4 * q + 1], ex = se_xy[4 * q + 2], ey = se_xy[4 * q + 3];
  const int map = prob_map ? prob_map[q] : 0;
  const int st = planner_validate(pl.rowF + (size_t)map * pl.row_plane, pl.wx, nx, ny, stx, sty, ex, ey);
  int done = 1;
  if (st == VHP_OK) {
    int32_t *ls = ls_all + q * (size_t)ls_cap * 2;
    ls[0] = stx; ls[1] = sty;   // lightSources_[0] = start, :121
    done = !(0.0 <= thr);       // loop test :127 with visibility_global_(end) = 0 (:123)
  }
  src_xy[2 * q] = done ? kSkipPair : stx;
  src_xy[2 * q + 1] = sty;
  int *c = ctl + 5 * q;
  c[0] = done; c[1] = stx; c[2] = sty; c[3] = st; c[4] = 0;
}

struct FirstEpilogueParams {
  int nx, ny, ls_cap;
  double thr, scale;
  const int32_t *se_xy, *ls;
  const int *ctl;
  const double *vis;
  double *vg, *hc;
  int32_t *came;
  Best *partial; // [problem][kFirstSlabs]
};

template <bool FIRST>
__global__ void __launch_bounds__(256) planner_first_epilogue_kernel(const FirstEpilogueParams p) {
  __shared__ Best s_best[8];
  const int64_t q = blockIdx.x / kFirstSlabs;
  const int slab = blockIdx.x % kFirstSlabs;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (p.ctl[5 * q]) return; // no sweep ran for this problem
  const size_t cells = (size_t)p.nx * p.ny;
  const int sx = p.ctl[5 * q + 1], sy = p.ctl[5 * q + 2], nb = p.ctl[5 * q + 4]; // the sweep's source
  const int ex = p.se_xy[4 * q + 2], ey = p.se_xy[4 * q + 3];
  const double *vis = p.vis + q * cells;
  double *vg = p.vg + q * cells, *hc = p.hc + q * cells;
  int32_t *came = p.came + q * cells;
  const int32_t *ls = p.ls + q * (size_t)p.ls_cap * 2;
  const int rows = (p.ny + kFirstSlabs - 1) / kFirstSlabs;
  const int y0 = slab * rows, y1 = min(p.ny, y0 + rows);
  Best best{~0ull, ~0ull};
  constexpr int kU = 4;
  for (int Y = y0 + warp; Y < y1; Y += 8) {
    const size_t row = (size_t)Y * p.nx;
    for (int X0 = lane; X0 < p.nx; X0 += 32 * kU) {
      double v[kU], h[kU], g0[kU];
      int cf[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u)
        if (X0 + 32 * u < p.nx) {
          const size_t c = row + X0 + 32 * u;
          v[u] = __ldcs(vis + c);
          if (!FIRST) { h[u] = __ldcg(hc + c); g0[u] = __ldcg(vg + c); cf[u] = __ldcg(came + c); }
        }
#pragma unroll
      for (int u = 0; u < kU; ++u)
        if (X0 + 32 * u < p.nx) {
          const int X = X0 + 32 * u;
          if (FIRST)
            epilogue_cell_first(X, Y, row + X, v[u], sx, sy, ex, ey, p.thr, p.scale, ls, vg, hc, came, best);
          else
            epilogue_cell_loaded(X, Y, row + X, v[u], h[u], g0[u], cf[u], sx, sy, ex, ey, p.thr, p.scale, nb, ls, vg,
                                 hc, came, best);
        }
    }
  }
  best = warp_best(best);
  if (lane == 0) s_best[warp] = best;
  __syncthreads();
  if (threadIdx.x < 32) {
    Best b = threadIdx.x < 8 ? s_best[threadIdx.x] : Best{~0ull, ~0ull};
    b = warp_best(b);
    if (threadIdx.x == 0) p.partial[q * kFirstSlabs + slab] = b;
  }
}

__global__ void planner_first_step_kernel(const Best *partial, int nx, const int32_t *se_xy, double thr,
                                          int max_iter, const double *vg_all, size_t cells, int32_t *ls_all,
                                          int ls_cap, int *ctl, int32_t *src_xy, int64_t nprob) {
  const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q >= nprob) return;
  int *c = ctl + 5 * q;
  if (c[0]) return;
  Best b{~0ull, ~0ull};
  for (int s = 0; s < kFirstSlabs; ++s)
    if (better(partial[q * kFirstSlabs + s], b)) b = partial[q * kFirstSlabs + s];
  const int ex = se_xy[4 * q + 2], ey = se_xy[4 * q + 3];
  int tx, ty, d, st = c[3];
  const int nnb = planner_next_source(b, c[1], c[2], c[4], max_iter, thr, __ldcg(vg_all + q * cells + (size_t)ey * nx + ex),
                                      ls_all + q * (size_t)ls_cap * 2, tx, ty, d, st);
  c[0] = d; c[1] = tx; c[2] = ty; c[3] = st; c[4] = nnb;
  src_xy[2 * q] = d ? kSkipPair : tx; // the next batch-wide sweep, if any, starts from the new source
  src_xy[2 * q + 1] = ty;
}

// ---- strip epilogue (giant-map path): the same per-cell epilogue over the rows
// [y0, y1) one rank owns, whole GPU, then a one-CTA reduction of the per-CTA minima.
struct StripEpilogueParams {
  int nx, y0, y1, sx, sy, ex, ey, nb;
  double thr, scale;
  const int32_t *ls;
  const double *vis;
  double *vg, *hc;
  int32_t *came;
  Best *partial; // [gridDim.x]
  const int *ctl; // non-null: {done, sx, sy, status, nb} on the device replace sx, sy, nb
};

__global__ void __launch_bounds__(256) strip_epilogue_kernel(const StripEpilogueParams p) {
  __shared__ Best s_best[8];
  const size_t cells = (size_t)(p.y1 - p.y0) * p.nx;
  int sx = p.sx, sy = p.sy, nb = p.nb, ex = p.ex, ey = p.ey;
  double thr = p.thr;
  if (p.ctl) { // loop state and query on the device (kernels_giant.cu)
    if (p.ctl[0]) return;
    sx = p.ctl[1]; sy = p.ctl[2]; nb = p.ctl[4];
    ex = p.ctl[6]; ey = p.ctl[7];
    thr = *reinterpret_cast<const double *>(p.ctl + 8);
  }
  Best best{~0ull, ~0ull};
  for (size_t c = blockIdx.x * (size_t)blockDim.x + threadIdx.x; c < cells;
       c += (size_t)gridDim.x * blockDim.x) {
    const int Yl = (int)(c / p.nx), X = (int)(c - (size_t)Yl * p.nx);
    epilogue_cell(X, p.y0 + Yl, c, sx, sy, ex, ey, thr, p.scale, nb, p.ls, p.vis, p.vg,
                  p.hc, p.came, best);
  }
  best = warp_best(best);
  if ((threadIdx.x & 31) == 0) s_best[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x < 32) {
    Best b = threadIdx.x < 8 ? s_best[threadIdx.x] : Best{~0ull, ~0ull};
    b = warp_best(b);
    if (threadIdx.x == 0) p.partial[blockIdx.x] = b;
  }
}

__global__ void __launch_bounds__(256) strip_best_kernel(const Best *partial, int n, Best *out,
                                                         const int *ctl) {
  __shared__ Best s_best[8];
  if (ctl && ctl[0]) return;
  Best best{~0ull, ~0ull};
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (better(partial[i], best)) best = partial[i];
  best = warp_best(best);
  if ((threadIdx.x & 31) == 0) s_best[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x < 32) {
    Best b = threadIdx.x < 8 ? s_best[threadIdx.x] : Best{~0ull, ~0ull};
    b = warp_best(b);
    if (threadIdx.x == 0) *out = b;
  }
}

// ---- one LARGE problem on the whole GPU: the loop runs in the strip engine (giant.cu,
// kernels_giant.cu: one strip = the whole map); ctl = {done, next x, next y, status,
// nb_of_sources, ...} stays on the device.
// tail of solve(): outputs of problem q; vis keeps the zeros of reset() if no sweep ran;
// optional fp32 exports
__global__ void grid_planner_finish_kernel(const int *ctl, int nx, int ny, int ex, int ey, int ls_cap,
                                           int32_t *ls, const int32_t *came, double *vis,
                                           const double *vg, int32_t *status, int32_t *nb_out,
                                           double *path_len, int32_t *path_n, int32_t *path,
                                           float *vg32, float *vis32) {
  const size_t cells = (size_t)nx * ny;
  const int st = ctl[3], nb = ctl[4];
  const size_t gtid = blockIdx.x * (size_t)blockDim.x + threadIdx.x, gn = (size_t)gridDim.x * blockDim.x;
  if (gtid == 0) {
    *status = st;
    *nb_out = nb;
    double total;
    const long n = planner_reconstruct(st, nb, ex, ey, nx, ls_cap, ls, came, path, total);
    *path_n = (int32_t)n;
    *path_len = total;
  }
  for (size_t c = gtid; c < cells; c += gn) {
    if (nb == 0) vis[c] = 0.0;
    if (vg32) vg32[c] = __double2float_rn(__ldcg(vg + c));
    if (vis32) vis32[c] = nb == 0 ? 0.0f : __double2float_rn(__ldcg(vis + c));
  }
}

} // namespace

cudaError_t vhp_launch_grid_planner_finish(const int *d_ctl, int nx, int ny, int ex, int ey,
                                           int ls_cap, int32_t *d_ls, const int32_t *d_came,
                                           double *d_vis, const double *d_vg, int32_t *d_status,
                                           int32_t *d_nb, double *d_path_len, int32_t *d_path_n,
                                           int32_t *d_path, float *d_vg32, float *d_vis32,
                                           cudaStream_t st, int64_t *launches) {
  grid_planner_finish_kernel<<<148 * 8, 256, 0, st>>>(d_ctl, nx, ny, ex, ey, ls_cap, d_ls, d_came,
                                                      d_vis, d_vg, d_status, d_nb, d_path_len,
                                                      d_path_n, d_path, d_vg32, d_vis32);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

int vhp_strip_epilogue_blocks(int sm_count) { return sm_count * 8; }

cudaError_t vhp_launch_strip_epilogue(int nx, int ny, int y0, int y1, int sx, int sy, int ex, int ey,
                                      double thr, int nb, const int32_t *d_ls, const double *d_vis,
                                      double *d_vg, double *d_hc, int32_t *d_came,
                                      unsigned long long *d_partial, int nblocks,
                                      unsigned long long *d_best, cudaStream_t st,
                                      int64_t *launches, const int *d_ctl) {
  StripEpilogueParams p;
  p.nx = nx; p.y0 = y0; p.y1 = y1; p.sx = sx; p.sy = sy; p.ex = ex; p.ey = ey; p.nb = nb;
  p.thr = thr;
  p.scale = std::sqrt((double)((unsigned long long)ny * ny + (unsigned long long)nx * nx)); // :49
  p.ls = d_ls; p.vis = d_vis; p.vg = d_vg; p.hc = d_hc; p.came = d_came;
  p.partial = reinterpret_cast<Best *>(d_partial);
  p.ctl = d_ctl;
  strip_epilogue_kernel<<<nblocks, 256, 0, st>>>(p);
  strip_best_kernel<<<1, 256, 0, st>>>(p.partial, nblocks, reinterpret_cast<Best *>(d_best), d_ctl);
  if (launches) *launches += 2;
  return cudaGetLastError();
}

bool vhp_planner_supported(int nx, int ny) { return vhp_sweep_tile_supported(nx, ny); }

size_t vhp_planner_first_ws_bytes(int64_t nprob) {
  return (((size_t)nprob * 8 + 255) & ~(size_t)255) + (((size_t)nprob * 20 + 255) & ~(size_t)255) +
         (size_t)nprob * kFirstSlabs * sizeof(Best) + 256;
}

cudaError_t vhp_launch_planner(const VhpTilePlanes &pl, int nx, int ny, const int32_t *d_se_xy,
                               const int32_t *d_prob_map, int64_t nprob, double threshold,
                               int32_t max_iter, int32_t ls_cap, const double *d_rcp2,
                               double *d_vis, double *d_vg, double *d_hc, int32_t *d_came,
                               int32_t *d_status,
                               int32_t *d_nb, int32_t *d_ls, double *d_path_len, int32_t *d_path_n,
                               int32_t *d_path, float *d_vg32, float *d_vis32, int *d_err,
                               cudaStream_t st, int64_t *launches, void *d_first_ws, int first_rounds) {
  if (!vhp_sweep_tile_supported(nx, ny)) return cudaErrorInvalidConfiguration;
  // large batches: every problem's first sweep and epilogue batch-wide (see planner_first_* above)
  const int *resume = nullptr;
  if (d_first_ws) {
    char *w = static_cast<char *>(d_first_ws);
    int32_t *src = reinterpret_cast<int32_t *>(w);
    int *ctl = reinterpret_cast<int *>(w + (((size_t)nprob * 8 + 255) & ~(size_t)255));
    Best *partial = reinterpret_cast<Best *>(reinterpret_cast<char *>(ctl) + (((size_t)nprob * 20 + 255) & ~(size_t)255));
    const unsigned nb1 = (unsigned)((nprob + 255) / 256);
    planner_first_begin_kernel<<<nb1, 256, 0, st>>>(pl, nx, ny, d_se_xy, d_prob_map, threshold, d_ls, ls_cap, src, ctl, nprob);
    FirstEpilogueParams f;
    f.nx = nx; f.ny = ny; f.ls_cap = ls_cap; f.thr = threshold;
    f.scale = std::sqrt((double)((unsigned long long)ny * ny + (unsigned long long)nx * nx)); // :49
    f.se_xy = d_se_xy; f.ls = d_ls; f.ctl = ctl; f.vis = d_vis; f.vg = d_vg; f.hc = d_hc; f.came = d_came;
    f.partial = partial;
    for (int round = 0; round < std::max(1, first_rounds); ++round) {
      cudaError_t e = vhp_launch_sweep_tile(pl, nx, ny, src, d_prob_map, nprob, VHP_F64, d_vis, d_rcp2, d_err, st, launches);
      if (e != cudaSuccess) return e;
      if (round == 0) planner_first_epilogue_kernel<true><<<(unsigned)(nprob * kFirstSlabs), 256, 0, st>>>(f);
      else planner_first_epilogue_kernel<false><<<(unsigned)(nprob * kFirstSlabs), 256, 0, st>>>(f);
      planner_first_step_kernel<<<nb1, 256, 0, st>>>(partial, nx, d_se_xy, threshold, max_iter, d_vg, (size_t)nx * ny,
                                                     d_ls, ls_cap, ctl, src, nprob);
      if (launches) *launches += 2;
    }
    if (launches) *launches += 1;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    resume = ctl;
  }
  PlannerParams p;
  p.fp.pl = pl;
  p.fp.nx = nx; p.fp.ny = ny;
  p.fp.src_xy = nullptr; p.fp.src_map = nullptr; p.fp.out = nullptr;
  p.fp.rtab = reinterpret_cast<const double2 *>(d_rcp2);
  p.fp.err = d_err;
  p.fp.vec = ((uintptr_t)d_vis % 16 == 0 && nx % 2 == 0) ? 1 : 0;
  p.fp.win_y0 = 0;
  p.fp.win_y1 = ny;
  p.se_xy = d_se_xy; p.prob_map = d_prob_map;
  p.thr = threshold; p.max_iter = max_iter; p.ls_cap = ls_cap;
  p.vis = d_vis; p.vg = d_vg; p.hc = d_hc; p.came = d_came;
  p.status = d_status; p.nb = d_nb; p.ls = d_ls;
  p.path_len = d_path_len; p.path_n = d_path_n; p.path = d_path;
  p.vg32 = d_vg32; p.vis32 = d_vis32;
  p.resume = resume;
  static const int forced = [] {
    const char *e = std::getenv("VHP_PLANNER_WARPS");
    return e ? std::atoi(e) : 0;
  }();
  int nw = 8; // measured on the 1024 x 256^2 batch: 8 warps 240k solves/s, 4 warps 206k, 2 warps slower still
  if (forced == 2 || forced == 4 || forced == 6 || forced == 8) nw = forced;
  auto go = [&](auto kern, int nwarps) -> cudaError_t {
    const size_t smem = tile_smem_bytes<double>(nx, ny, nwarps);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<(unsigned)nprob, nwarps * 32, smem, st>>>(p);
    if (launches) *launches += 1;
    return cudaGetLastError();
  };
  if (nw == 2) return go(planner_kernel<2>, 2);
  if (nw == 4) return go(planner_kernel<4>, 4);
  if (nw == 6) return go(planner_kernel<6, 3>, 6);     // 3 CTAs per SM: <= 112 registers
  return go(planner_kernel<8, 2>, 8);               // 2 CTAs per SM (<= 128 registers)
}
