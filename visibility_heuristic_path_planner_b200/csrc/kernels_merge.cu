// kernels_merge.cu -- merged visibility of groups of light sources (vhp_visibility_merge_batch): the per-pair
// table of the CSR group layout, the output fill and the fold of fp64 fields into the group outputs.
//
// The fold is the route every size and threshold can take (the sweeps themselves run through run_dev: tile
// kernel, grid mode or the naive kernel, into a chunk buffer); the direct route (kFmtMerge* of the tile kernel,
// thr > 0) folds inside the sweep.  Both compute, per cell of group g over its sources k = 0, 1, ...:
//   vmax  = max_k v_k                          (fp32: the fp64 maximum rounded once)
//   first = min { k : k writes the cell, v_k >= thr }, -1 if none
//   count = #{ k : k writes the cell, v_k >= thr }
// where source (sx, sy) writes every cell but column 0 (unless sx == 0) and row 0 (unless sy == 0).
// The range-limited form (vhp_visibility_merge_range_batch) counts v_k only where the cell is in k's range; its
// fallback folds fp64 windows (merge_window_fold_kernel) instead of whole fields, and so does the fallback of the view
// form (vhp_visibility_merge_view_batch), with only the cells in each source's view (MergeView).
#include <algorithm>
#include <cstdint>

#include "vhp_internal.h"
#include "sweep_common.cuh"

namespace {

constexpr int kErrGroups = 4; // d_err bit: inconsistent group layout / group map
constexpr int kErrView = 16;  // d_err bit: a bad view of vhp_visibility_merge_view_batch_dev

// Thread t < nsrc: pair t -> (group, index in group, map) by a binary search of group_ptr; thread t <= ngroups:
// group_ptr[0] == 0, non-decreasing, groups below 2^31 sources, group_ptr[ngroups] == nsrc.
__global__ void merge_table_kernel(const int64_t *__restrict__ gptr, const int32_t *__restrict__ gmap,
                                   int64_t ngroups, int64_t nsrc, int nmaps, int32_t *__restrict__ pg,
                                   int32_t *__restrict__ pk, int32_t *__restrict__ pmap, int *err) {
  const int64_t n = nsrc > ngroups + 1 ? nsrc : ngroups + 1;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    if (t <= ngroups) {
      const int64_t a = __ldg(gptr + t);
      bool ok = t == 0 ? a == 0 : true;
      if (t < ngroups) {
        const int64_t b = __ldg(gptr + t + 1);
        ok = ok && b >= a && b - a < ((int64_t)1 << 31);
      } else {
        ok = ok && a == nsrc;
      }
      if (!ok) atomicOr(err, kErrGroups);
    }
    if (t < nsrc) {
      int64_t lo = 0, hi = ngroups; // largest g < ngroups with gptr[g] <= t
      while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(gptr + mid) <= t) lo = mid;
        else hi = mid;
      }
      int32_t g = -1, k = 0, m = 0;
      if (ngroups > 0) {
        const int64_t a = __ldg(gptr + lo), b = __ldg(gptr + lo + 1);
        const int32_t mm = gmap ? __ldg(gmap + lo) : 0;
        if (a <= t && t < b && mm >= 0 && mm < nmaps) {
          g = (int32_t)lo;
          k = (int32_t)(t - a);
          m = mm;
        }
      }
      if (g < 0) atomicOr(err, kErrGroups);
      pg[t] = g;
      pk[t] = k;
      pmap[t] = m;
    }
  }
}

// One thread per cell of every group that has pairs in [p0, p0 + np): the thread of the group's first pair in
// the chunk folds that group's pairs in order (no atomics; groups that span chunks continue where the last
// chunk left them).
template <bool F32>
__global__ void merge_fold_kernel(const double *__restrict__ field, int64_t p0, int64_t np, int nx, size_t cells,
                                  const int32_t *__restrict__ xy, double thr, VhpMergeDev m) {
  const size_t total = (size_t)np * cells;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int64_t j = (int64_t)(idx / cells);
    const size_t c = idx - (size_t)j * cells;
    const int64_t p = p0 + j;
    const int32_t g = __ldg(m.pair_group + p);
    if (g < 0 || (j > 0 && __ldg(m.pair_group + p - 1) == g)) continue;
    const int x = (int)(c % nx), y = (int)(c / nx);
    const size_t o = (size_t)g * cells + c;
    double vm = 0.0;
    float vf = 0.0f;
    if (m.vmax) {
      if (F32) vf = reinterpret_cast<const float *>(m.vmax)[o];
      else vm = reinterpret_cast<const double *>(m.vmax)[o];
    }
    int32_t f = m.first ? m.first[o] : -1;
    uint32_t cnt = m.count ? m.count[o] : 0u;
    for (int64_t q = p; q < p0 + np && __ldg(m.pair_group + q) == g; ++q) {
      const double v = __ldg(field + (size_t)(q - p0) * cells + c);
      const int sx = __ldg(xy + 2 * q), sy = __ldg(xy + 2 * q + 1);
      if (F32) vf = fmaxf(vf, __double2float_rn(v));
      else vm = fmax(vm, v);
      const bool writes = !((x == 0 && sx != 0) || (y == 0 && sy != 0));
      if (writes && v >= thr) {
        if (f < 0) f = __ldg(m.pair_k + q);
        ++cnt;
      }
    }
    if (m.vmax) {
      if (F32) reinterpret_cast<float *>(m.vmax)[o] = vf;
      else reinterpret_cast<double *>(m.vmax)[o] = vm;
    }
    if (m.first) m.first[o] = f;
    if (m.count) m.count[o] = cnt;
  }
}

// One thread per window cell of pairs [p0, p0 + np): cells in the grid and in the pair's range fold into its
// group's outputs with the relaxed reductions of the direct route (kFmtMergeRange*), so the order of the pairs
// does not matter.  r2: a cell (dx, dy) of the window is in range iff dx^2 + dy^2 <= r2 (box: 2 R^2).  VIEW: only
// the cells in the pair's view views[q] fold instead; a bad view folds nothing and raises error value 16.
template <bool F32, bool VIEW>
__global__ void merge_window_fold_kernel(const double *__restrict__ win, int64_t p0, int64_t np, int nx, int ny,
                                         int R, int r2, const int32_t *__restrict__ xy, double thr, VhpMergeDev m,
                                         const int32_t *__restrict__ views, bool disk, int *err) {
  const int W = 2 * R + 1;
  const size_t ww = (size_t)W * W, total = (size_t)np * ww, cells = (size_t)nx * ny;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int64_t q = p0 + (int64_t)(idx / ww);
    const int rem = (int)(idx % ww), dy = rem / W - R, dx = rem % W - R;
    const int sx = __ldg(xy + 2 * q), sy = __ldg(xy + 2 * q + 1), x = sx + dx, y = sy + dy;
    if constexpr (VIEW) { // (a pair of an inconsistent group layout reads no view)
      MergeView w;
      if (__ldg(m.pair_group + q) < 0) continue;
      if (!merge_view_decode(views + 5 * q, R, disk, w)) {
        if (rem == 0) atomicOr(err, kErrView);
        continue;
      }
      if ((unsigned)x >= (unsigned)nx || (unsigned)y >= (unsigned)ny || !merge_view_has(w, dx, dy)) continue;
    } else {
      if ((unsigned)x >= (unsigned)nx || (unsigned)y >= (unsigned)ny || dx * dx + dy * dy > r2) continue;
    }
    const int32_t g = __ldg(m.pair_group + q);
    if (g < 0) continue;
    const double v = __ldg(win + idx);
    const size_t o = (size_t)g * cells + (size_t)y * nx + x;
    if (m.vmax && v > 0.0) {
      if (F32) red_max_u32(reinterpret_cast<uint32_t *>(m.vmax) + o, __float_as_uint(__double2float_rn(v)));
      else red_max_u64(reinterpret_cast<unsigned long long *>(m.vmax) + o, (unsigned long long)__double_as_longlong(v));
    }
    const bool writes = !((x == 0 && sx != 0) || (y == 0 && sy != 0));
    if (writes && v >= thr) {
      if (m.first) red_min_u32(reinterpret_cast<uint32_t *>(m.first) + o, (uint32_t)__ldg(m.pair_k + q));
      if (m.count) red_add_u32(m.count + o, 1u);
    }
  }
}

unsigned grid_for(size_t n, int bs, int sm_count) {
  return (unsigned)std::max<size_t>(1, std::min<size_t>((n + bs - 1) / bs, (size_t)sm_count * 32));
}

} // namespace

cudaError_t vhp_launch_merge_table(const int64_t *d_group_ptr, const int32_t *d_group_map, int64_t ngroups,
                                   int64_t nsrc, int nmaps, int32_t *d_pair_group, int32_t *d_pair_k,
                                   int32_t *d_pair_map, int *d_err, int sm_count, cudaStream_t st,
                                   int64_t *launches) {
  const int bs = 256;
  merge_table_kernel<<<grid_for((size_t)std::max(nsrc, ngroups + 1), bs, sm_count), bs, 0, st>>>(
      d_group_ptr, d_group_map, ngroups, nsrc, nmaps, d_pair_group, d_pair_k, d_pair_map, d_err);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t vhp_launch_merge_fill(const VhpMergeDev &m, size_t cells_total, cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  if (m.vmax) e = cudaMemsetAsync(m.vmax, 0, cells_total * (m.f32 ? 4 : 8), st);
  if (e == cudaSuccess && m.first) e = cudaMemsetAsync(m.first, 0xff, cells_total * 4, st); // VHP_NO_PARENT
  if (e == cudaSuccess && m.count) e = cudaMemsetAsync(m.count, 0, cells_total * 4, st);
  return e;
}

cudaError_t vhp_launch_merge_fold(const double *d_field, int64_t p0, int64_t np, int nx, int ny,
                                  const int32_t *d_src_xy, double thr, const VhpMergeDev &m, int sm_count,
                                  cudaStream_t st, int64_t *launches) {
  const size_t cells = (size_t)nx * ny;
  const int bs = 256;
  const unsigned grid = grid_for((size_t)np * cells, bs, sm_count);
  if (m.f32) merge_fold_kernel<true><<<grid, bs, 0, st>>>(d_field, p0, np, nx, cells, d_src_xy, thr, m);
  else merge_fold_kernel<false><<<grid, bs, 0, st>>>(d_field, p0, np, nx, cells, d_src_xy, thr, m);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t vhp_launch_merge_window_fold(const double *d_win, int64_t p0, int64_t np, int nx, int ny,
                                         const int32_t *d_src_xy, double thr, const VhpMergeRange &range,
                                         const VhpMergeDev &m, int *d_err, int sm_count, cudaStream_t st,
                                         int64_t *launches) {
  const int R = range.radius, r2 = range.shape == VHP_RANGE_DISK ? R * R : 2 * R * R;
  const size_t W = 2 * (size_t)R + 1;
  const int bs = 256;
  const unsigned grid = grid_for((size_t)np * W * W, bs, sm_count);
  const int32_t *v = range.views;
  const bool disk = range.shape == VHP_RANGE_DISK;
  if (v && m.f32)
    merge_window_fold_kernel<true, true><<<grid, bs, 0, st>>>(d_win, p0, np, nx, ny, R, r2, d_src_xy, thr, m, v, disk, d_err);
  else if (v)
    merge_window_fold_kernel<false, true><<<grid, bs, 0, st>>>(d_win, p0, np, nx, ny, R, r2, d_src_xy, thr, m, v, disk, d_err);
  else if (m.f32)
    merge_window_fold_kernel<true, false><<<grid, bs, 0, st>>>(d_win, p0, np, nx, ny, R, r2, d_src_xy, thr, m, v, disk, d_err);
  else
    merge_window_fold_kernel<false, false><<<grid, bs, 0, st>>>(d_win, p0, np, nx, ny, R, r2, d_src_xy, thr, m, v, disk, d_err);
  if (launches) *launches += 1;
  return cudaGetLastError();
}
