// kernels_sweep_tile.cu -- K1, batched visibility sweep as a tile wavefront (the
// default sweep kernel).
//
// Replaces visibilityBasedSolver::computeVisibility
// (reference src/visibilityBasedSolver.cpp:570-696) over a batch of (map, source)
// pairs: one CTA per pair, see sweep_tile_body.cuh for the decomposition.
#include <algorithm>
#include <cstdint>
#include <cstdlib>

#include "sweep_tile_body.cuh"

// Single-warp CTAs: 32 per SM would need 64 registers per thread, which the tile body only reaches with
// spills, and shared memory keeps fewer than 32 resident from about 64 x 64 maps on.  Compiled for 20
// per SM (80 registers, no spills): 256 x 256 maps (c4) 616 -> 647 Gcells/s (a bound of 24: 638; 16 and
// 12, 90 registers: 609), 101 x 101 and 64 x 64 maps +3 % (tools/small_batch_probe.py).
#ifndef VHP_NW1_MINB
#define VHP_NW1_MINB 20
#endif
#ifndef VHP_NW4_MINB
#define VHP_NW4_MINB 5 // 4-warp CTAs (mid-size batches of small maps): 96 registers, no spills; 2000 pairs of
#endif                 // 256 x 256: 370 (bound 8, 64 registers, spills) -> 436 (6) -> 444 Gcells/s (5)
#ifndef VHP_NW8_MINB
#define VHP_NW8_MINB 3 // resident 8-warp CTAs per SM the register allocation aims at
#endif

namespace {

// NW warps per CTA: 8 for large grids (a pair's boundary rows take tens of KB of shared
// memory, so few CTAs fit an SM and each must bring its own parallelism); small maps use 4,
// or 1 when the batch alone fills the machine (32 independent single-warp CTAs per SM: no
// flag polling, no imbalance between the warps of a pair).
template <typename OutT, int NW, int MINB, int FMT = kFmtValues>
__global__ void __launch_bounds__(NW * 32, MINB)
sweep_tile_kernel(const TileArgs p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int64_t pair = blockIdx.x;
  const int sx = __ldg(p.src_xy + 2 * pair), sy = __ldg(p.src_xy + 2 * pair + 1);
  if (sx == kSkipPair) return; // "no sweep for this item" (the planner's first batched sweep)
  if ((unsigned)sx >= (unsigned)p.nx || (unsigned)sy >= (unsigned)p.ny) { // uniform over the CTA
    if (threadIdx.x == 0) atomicOr(p.err, 1);
    return;
  }
  const int map = p.src_map ? __ldg(p.src_map + pair) : 0;
  if constexpr (fmt_merge(FMT)) { // fold into the outputs of the pair's group
    const int g = __ldg(p.m_pg + pair);
    if (g < 0) return; // a pair of an inconsistent group layout (the table kernel reported it)
    if constexpr (fmt_view(FMT)) { // the source's view into the tail; a bad one (error value 16) folds nothing
      MergeView w;
      if (!merge_view_decode(p.m_views + 5 * pair, p.w_r, p.m_disk != 0, w)) {
        if (threadIdx.x == 0) atomicOr(p.err, 16);
        return;
      }
      if (threadIdx.x == 0) {
        uint32_t dsmem;
        asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dsmem));
        *reinterpret_cast<int4 *>(smem_raw + dsmem - kViewTail) = make_int4(w.key | (sy * p.nx + sx), w.range, w.a, w.b);
      }
    }
    if (threadIdx.x == 0) *reinterpret_cast<int2 *>(smem_raw + kMergeHdr) = make_int2(g, __ldg(p.m_pk + pair));
    tile_sweep_cta<OutT, NW, kSweepCta, FMT>(p, map, sx, sy, reinterpret_cast<OutT *>(p.out), smem_raw);
    return;
  }
  if constexpr (FMT == kFmtWindow) { // the pair's window, addressed by absolute grid coordinates
    if ((unsigned)map >= (unsigned)p.w_nmaps) {
      if (threadIdx.x == 0) atomicOr(p.err, 1);
      return;
    }
    const int W = 2 * p.w_r + 1;
    OutT *out = reinterpret_cast<OutT *>(p.out) + (size_t)pair * W * W -
                ((ptrdiff_t)(sy - p.w_r) * W + (sx - p.w_r));
    tile_sweep_cta<OutT, NW, kSweepCta, FMT>(p, map, sx, sy, out, smem_raw);
    return;
  }
  if constexpr (FMT == kFmtCoverBits) { // the candidate's box bits (VhpCoverBox), addressed by absolute grid coordinates
    const VhpCoverBox b = vhp_cover_box(p.nx, p.ny, p.w_r, sx, sy);
    uint32_t *out = reinterpret_cast<uint32_t *>(p.out) + (size_t)pair * b.H * b.W - ((ptrdiff_t)b.y0 * b.W + b.w0);
    tile_sweep_cta<OutT, NW, kSweepCta, FMT>(p, map, sx, sy, reinterpret_cast<OutT *>(out), smem_raw);
    return;
  }
  // bit output: rows of (nx + 31) / 32 words
  const size_t per_pair = FMT == kFmtBits ? (size_t)((p.nx + 31) >> 5) * p.ny : (size_t)p.nx * p.ny;
  OutT *out = reinterpret_cast<OutT *>(p.out) + (size_t)pair * per_pair;
  tile_sweep_cta<OutT, NW, kSweepCta, FMT>(p, map, sx, sy, out, smem_raw);
}

// One sweep of map 0 restricted to the grid rows [win_y0, win_y1) (strip partition):
// p.out is the strip buffer, row win_y0 first.
template <typename OutT>
__global__ void __launch_bounds__(kTileWarps * 32, 1)
sweep_window_kernel(const TileArgs p, int sx, int sy) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  if (p.src_ctl) { // device-side loop control (see TileArgs::src_ctl)
    if (p.src_ctl[0]) return;
    sx = p.src_ctl[1];
    sy = p.src_ctl[2];
  }
  OutT *out = reinterpret_cast<OutT *>(p.out) - (ptrdiff_t)p.win_y0 * p.nx;
  tile_sweep_cta<OutT, kTileWarps>(p, 0, sx, sy, out, smem_raw);
}

// Grid mode of the same window sweep (giant maps): one sweep spread over many CTAs.  The init
// kernel (one CTA) leaves the staircase, the boundary rows, the row progress flags and the row
// counter in the global workspace; the work kernel, launched right after it on the same stream,
// writes the lit region and runs the tile rows (see tile_sweep_cta).
template <typename OutT, int MODE>
__global__ void __launch_bounds__(kTileWarps * 32, MODE == kSweepGridWork ? 2 : 1)
sweep_grid_kernel(const TileArgs p, int sx, int sy) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  if (p.src_ctl) {
    if (p.src_ctl[0]) return;
    sx = p.src_ctl[1];
    sy = p.src_ctl[2];
  }
  OutT *out = reinterpret_cast<OutT *>(p.out) - (ptrdiff_t)p.win_y0 * p.nx;
  tile_sweep_cta<OutT, kTileWarps, MODE>(p, 0, sx, sy, out, smem_raw);
}

// ---------------------------------------------------------------------------------
// Bit planes.  wx = ceil(nx/32) + 1 words per row line, wy likewise per column line
// (one zero word of padding so a 32-bit window may start in the last data word).
//   rowF[m][y][w] bit b = occ(32w + b, y)            rowR: x mirrored, p = 32*WX - 1 - x
//   colF[m][x][w] bit b = occ(x, 32w + b)            colR: y mirrored, p = 32*WY - 1 - y
// Bits outside the grid are 0 ("occupied").
// ---------------------------------------------------------------------------------
__global__ void pack_tile_rows_kernel(const uint8_t *__restrict__ occ, int nmaps, int nx, int ny,
                                      int wx, uint32_t *__restrict__ rowF,
                                      uint32_t *__restrict__ rowR) {
  const size_t total = (size_t)nmaps * ny * wx;
  const int W = 32 * (wx - 1);
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int w = (int)(idx % wx);
    const uint8_t *row = occ + (idx / wx) * nx;
    uint32_t f = 0, r = 0;
    for (int b = 0; b < 32; ++b) {
      const int xf = 32 * w + b, xr = W - 1 - xf;
      if (xf < nx && row[xf] != 0) f |= 1u << b;
      if (xr >= 0 && xr < nx && row[xr] != 0) r |= 1u << b;
    }
    rowF[idx] = f;
    rowR[idx] = r;
  }
}

__global__ void pack_tile_cols_kernel(const uint8_t *__restrict__ occ, int nmaps, int nx, int ny,
                                      int wy, uint32_t *__restrict__ colF,
                                      uint32_t *__restrict__ colR) {
  // x fastest across threads so the strided byte reads coalesce
  const size_t total = (size_t)nmaps * wy * nx;
  const int W = 32 * (wy - 1);
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(idx % nx);
    const size_t mw = idx / nx;
    const int w = (int)(mw % wy);
    const size_t m = mw / wy;
    const uint8_t *base = occ + m * (size_t)nx * ny + x;
    uint32_t f = 0, r = 0;
    for (int b = 0; b < 32; ++b) {
      const int yf = 32 * w + b, yr = W - 1 - yf;
      if (yf < ny && base[(size_t)yf * nx] != 0) f |= 1u << b;
      if (yr >= 0 && yr < ny && base[(size_t)yr * nx] != 0) r |= 1u << b;
    }
    const size_t o = (m * nx + x) * wy + w;
    colF[o] = f;
    colR[o] = r;
  }
}

// bsum[m][by][w] bit (bx & 31) of word bx >> 5 = every in-grid cell of the aligned block
// x in [32bx, 32bx+32), y in [32by, 32by+32) is free.  One warp per block (lane = row),
// from the forward row plane; bsum must be zeroed first.
__global__ void pack_tile_sum_kernel(const uint32_t *__restrict__ rowF, int nmaps, int nx, int ny,
                                     int wx, uint32_t *__restrict__ bsum) {
  const int nbx = (nx + 31) >> 5, nby = (ny + 31) >> 5, nbw = tile_sum_words(nx);
  const size_t total = (size_t)nmaps * nby * nbx;
  const int lane = threadIdx.x & 31;
  for (size_t blk = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5; blk < total;
       blk += ((size_t)gridDim.x * blockDim.x) >> 5) {
    const int bx = (int)(blk % nbx);
    const size_t mb = blk / nbx;
    const int by = (int)(mb % nby);
    const size_t m = mb / nby;
    const int y = 32 * by + lane;
    const int nv = nx - 32 * bx;
    const uint32_t valid = nv >= 32 ? ~0u : (1u << nv) - 1u;
    bool ok = true;
    if (y < ny) ok = (__ldg(rowF + (m * ny + y) * wx + bx) & valid) == valid;
    if (__all_sync(0xffffffffu, ok) && lane == 0)
      atomicOr(bsum + (m * nby + by) * nbw + (bx >> 5), 1u << (bx & 31));
  }
}

// rtab[k] = {rh, rl}: rh = RN(1/k), rl = RN((1 - rh*k) * rh)
__global__ void rcp2_table_kernel(double2 *table, int len) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < len) {
    double rh = 0.0, rl = 0.0;
    if (k > 0) {
      const double fk = (double)k;
      rh = __drcp_rn(fk);
      rl = __dmul_rn(__fma_rn(-rh, fk, 1.0), rh);
    }
    table[k] = make_double2(rh, rl);
  }
}

// diagnostic: count (d, k), 0 <= d < k <= kmax, where fma(d, rh, d*rl) != d/k
__global__ void ratio2_selftest_kernel(const double2 *__restrict__ tab, int kmax,
                                       unsigned long long *mismatches) {
  const int k = blockIdx.x + 1;
  if (k > kmax) return;
  const double fk = (double)k;
  const double2 rr = tab[k];
  unsigned long long bad = 0;
  for (int d = threadIdx.x; d < k; d += blockDim.x) {
    const double fd = (double)d;
    if (__fma_rn(fd, rr.x, __dmul_rn(fd, rr.y)) != __ddiv_rn(fd, fk)) ++bad;
  }
  if (bad) atomicAdd(mismatches, bad);
}

template <typename OutT, int NW, int MINB, int FMT = kFmtValues>
cudaError_t launch_tile_nw(const TileArgs &p, int64_t npairs, cudaStream_t st) {
  const size_t smem = fmt_clip(FMT) ? tile_smem_bytes_win<OutT>(p.nx, p.ny, p.w_r, NW) + (fmt_view(FMT) ? kViewTail : 0)
                                    : tile_smem_bytes<OutT>(p.nx, p.ny, NW);
  auto kern = sweep_tile_kernel<OutT, NW, MINB, FMT>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)npairs, NW * 32, smem, st>>>(p);
  return cudaGetLastError();
}

int tile_warps_for(int nx, int ny, int64_t npairs) {
  static const int forced = [] {
    const char *e = std::getenv("VHP_TILE_WARPS");
    return e ? std::atoi(e) : 0;
  }();
  if (forced == 1 || forced == 2 || forced == 4 || forced == 6 || forced == 8 || forced == 10 ||
      forced == 16)
    return forced;
  if (std::max(nx, ny) > 512) return 8;
  // a handful of small sweeps is a latency problem: 8 warps finish one 101 x 101 sweep in 20-25 us,
  // 4 warps in 29-33 us (tools/c1_probe.py); enough pairs fill the SMs with single-warp CTAs
  if (npairs <= 148 * 2) return 8;
  return npairs >= 148 * 16 ? 1 : 4;
}

template <typename OutT>
cudaError_t launch_tile(const TileArgs &p, int64_t npairs, cudaStream_t st) {
  int nw = tile_warps_for(p.nx, p.ny, npairs);
  // a forced 10 or 16 whose CTA does not fit shared memory runs 8 warps (vhp_sweep_tile_supported checked those)
  if (tile_smem_bytes<OutT>(p.nx, p.ny, nw) > 227u * 1024u) nw = 8;
  switch (nw) {
    case 1: return launch_tile_nw<OutT, 1, VHP_NW1_MINB>(p, npairs, st);
    case 2: return launch_tile_nw<OutT, 2, 12>(p, npairs, st);
    case 4: return launch_tile_nw<OutT, 4, VHP_NW4_MINB>(p, npairs, st);
    case 6: return launch_tile_nw<OutT, 6, 4>(p, npairs, st);
    case 10: return launch_tile_nw<OutT, 10, 3>(p, npairs, st);
    case 16: return launch_tile_nw<OutT, 16, 2>(p, npairs, st);
    default: return launch_tile_nw<OutT, 8, VHP_NW8_MINB>(p, npairs, st);
  }
}

// bit output (TileArgs::thr, kFmtBits): the warp counts the automatic choice makes
template <int FMT>
cudaError_t launch_tile_fmt(const TileArgs &p, int64_t npairs, cudaStream_t st) {
  switch (tile_warps_for(p.nx, p.ny, npairs)) {
    case 1: return launch_tile_nw<float, 1, VHP_NW1_MINB, FMT>(p, npairs, st);
    case 2: case 4: case 6: return launch_tile_nw<float, 4, VHP_NW4_MINB, FMT>(p, npairs, st);
    default: return launch_tile_nw<float, 8, VHP_NW8_MINB, FMT>(p, npairs, st);
  }
}

// merged output (kFmtMerge*): fp64 staging whatever the dtype of vmax, the warp counts of the bit output
template <int FMT>
cudaError_t launch_tile_merge(const TileArgs &p, int64_t npairs, cudaStream_t st) {
  switch (tile_warps_for(p.nx, p.ny, npairs)) {
    case 1: return launch_tile_nw<double, 1, VHP_NW1_MINB, FMT>(p, npairs, st);
    case 2: case 4: case 6: return launch_tile_nw<double, 4, VHP_NW4_MINB, FMT>(p, npairs, st);
    default: return launch_tile_nw<double, 8, VHP_NW8_MINB, FMT>(p, npairs, st);
  }
}

// windows (kFmtWindow): the warp count of a map of the window's size.  8-warp CTAs are bound for 2 per SM (at 3 the
// window code spills): they run windows wider than 512, whose shared memory admits about 2 anyway, or small batches.
template <typename OutT>
cudaError_t launch_tile_win(const TileArgs &p, int64_t npairs, cudaStream_t st) {
  switch (tile_warps_for(win_side(p.nx, p.w_r), win_side(p.ny, p.w_r), npairs)) {
    case 1: return launch_tile_nw<OutT, 1, VHP_NW1_MINB, kFmtWindow>(p, npairs, st);
    case 2: case 4: case 6: return launch_tile_nw<OutT, 4, VHP_NW4_MINB, kFmtWindow>(p, npairs, st);
    default: return launch_tile_nw<OutT, 8, 2, kFmtWindow>(p, npairs, st);
  }
}

// range-limited merged output (kFmtMergeRange*, kFmtMergeView*): fp64 staging, the warp counts and bounds of the windows
template <int FMT>
cudaError_t launch_tile_merge_range(const TileArgs &p, int64_t npairs, cudaStream_t st) {
  switch (tile_warps_for(win_side(p.nx, p.w_r), win_side(p.ny, p.w_r), npairs)) {
    case 1: return launch_tile_nw<double, 1, VHP_NW1_MINB, FMT>(p, npairs, st);
    case 2: case 4: case 6: return launch_tile_nw<double, 4, VHP_NW4_MINB, FMT>(p, npairs, st);
    default: return launch_tile_nw<double, 8, 2, FMT>(p, npairs, st);
  }
}

// candidate coverage bits (kFmtCoverBits): the warp counts and bounds of the windows
cudaError_t launch_tile_cover(const TileArgs &p, int64_t npairs, cudaStream_t st) {
  switch (tile_warps_for(win_side(p.nx, p.w_r), win_side(p.ny, p.w_r), npairs)) {
    case 1: return launch_tile_nw<float, 1, VHP_NW1_MINB, kFmtCoverBits>(p, npairs, st);
    case 2: case 4: case 6: return launch_tile_nw<float, 4, VHP_NW4_MINB, kFmtCoverBits>(p, npairs, st);
    default: return launch_tile_nw<float, 8, 2, kFmtCoverBits>(p, npairs, st);
  }
}

// fallback of the windows: window of pair p cut out of its full field, 0 outside the grid
template <typename T>
__global__ void window_crop_kernel(const T *__restrict__ field, int64_t np, int nx, int ny,
                                   const int32_t *__restrict__ src_xy, int R, T *__restrict__ out) {
  const int W = 2 * R + 1;
  const size_t total = (size_t)np * W * W;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const size_t pair = idx / ((size_t)W * W);
    const int rem = (int)(idx - pair * W * W), v = rem / W, u = rem - v * W;
    const int x = __ldg(src_xy + 2 * pair) - R + u, y = __ldg(src_xy + 2 * pair + 1) - R + v;
    out[idx] = ((unsigned)x < (unsigned)nx && (unsigned)y < (unsigned)ny)
                   ? field[(pair * ny + y) * nx + x] : T(0);
  }
}

// copy of the pairs with a map index out of range turned into a source outside the grid (which every sweep
// route reports), so that the fallback never reads beyond the maps
__global__ void window_pairs_kernel(const int32_t *__restrict__ src_xy, const int32_t *__restrict__ src_map,
                                    int64_t np, int nmaps, int32_t *__restrict__ xy_out,
                                    int32_t *__restrict__ map_out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < np; i += (int64_t)gridDim.x * blockDim.x) {
    const int m = src_map[i];
    const bool ok = (unsigned)m < (unsigned)nmaps;
    xy_out[2 * i] = ok ? src_xy[2 * i] : -1;
    xy_out[2 * i + 1] = ok ? src_xy[2 * i + 1] : -1;
    map_out[i] = ok ? m : 0;
  }
}

} // namespace

bool vhp_sweep_window_supported(int nx, int ny, int radius) {
  return nx >= 1 && ny >= 1 && std::max(nx, ny) <= 16384 && radius >= 0 &&
         tile_smem_bytes_win<double>(nx, ny, radius) <= 227u * 1024u;
}

bool vhp_sweep_merge_view_supported(int nx, int ny, int radius) {
  return vhp_sweep_window_supported(nx, ny, radius) &&
         tile_smem_bytes_win<double>(nx, ny, radius) + kViewTail <= 227u * 1024u;
}

cudaError_t vhp_launch_sweep_window_batch(const VhpTilePlanes &pl, int nmaps, int nx, int ny,
                                          const int32_t *d_src_xy, const int32_t *d_src_map, int64_t npairs,
                                          int radius, vhp_dtype dtype, void *d_out, const double *d_rcp2,
                                          int *d_err, cudaStream_t st, int64_t *launches) {
  TileArgs p;
  p.pl = pl;
  p.nx = nx;
  p.ny = ny;
  p.src_xy = d_src_xy;
  p.src_map = d_src_map;
  p.out = d_out;
  p.rtab = reinterpret_cast<const double2 *>(d_rcp2);
  p.err = d_err;
  p.vec = 0; // window rows are not 16-byte aligned
  p.win_y0 = 0;
  p.win_y1 = ny;
  p.w_r = radius;
  p.w_sw = win_sum_words(nx, radius);
  p.w_nmaps = nmaps;
  if (launches) *launches += 1;
  return dtype == VHP_F32 ? launch_tile_win<float>(p, npairs, st) : launch_tile_win<double>(p, npairs, st);
}

cudaError_t vhp_launch_window_crop(const void *d_fields, int64_t np, int nx, int ny, const int32_t *d_src_xy,
                                   int radius, vhp_dtype dtype, void *d_out, int sm_count, cudaStream_t st,
                                   int64_t *launches) {
  const size_t W = 2 * (size_t)radius + 1, total = (size_t)np * W * W;
  const unsigned grid = (unsigned)std::min<size_t>((total + 255) / 256, (size_t)sm_count * 16);
  if (dtype == VHP_F32)
    window_crop_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float *>(d_fields), np, nx, ny, d_src_xy,
                                                    radius, static_cast<float *>(d_out));
  else
    window_crop_kernel<double><<<grid, 256, 0, st>>>(static_cast<const double *>(d_fields), np, nx, ny, d_src_xy,
                                                     radius, static_cast<double *>(d_out));
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t vhp_launch_window_pairs(const int32_t *d_src_xy, const int32_t *d_src_map, int64_t np, int nmaps,
                                    int32_t *d_xy_out, int32_t *d_map_out, int sm_count, cudaStream_t st,
                                    int64_t *launches) {
  const unsigned grid = (unsigned)std::min<int64_t>((np + 255) / 256, (int64_t)sm_count * 4);
  window_pairs_kernel<<<grid, 256, 0, st>>>(d_src_xy, d_src_map, np, nmaps, d_xy_out, d_map_out);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t vhp_launch_sweep_merge(const VhpTilePlanes &pl, int nx, int ny, const int32_t *d_src_xy,
                                   const VhpMergeDev &m, int64_t npairs, double thr, const double *d_rcp2,
                                   int *d_err, cudaStream_t st, int64_t *launches, const VhpMergeRange *range) {
  if (!(thr > 0.0)) return cudaErrorInvalidValue; // cells of value 0 are never visited
  TileArgs p;
  p.pl = pl;
  p.nx = nx;
  p.ny = ny;
  p.src_xy = d_src_xy;
  p.src_map = m.pair_map;
  p.out = const_cast<int32_t *>(m.pair_group); // a base for cell indices only
  p.rtab = reinterpret_cast<const double2 *>(d_rcp2);
  p.err = d_err;
  p.vec = 0;
  p.win_y0 = 0;
  p.win_y1 = ny;
  p.thr = thr;
  p.m_vmax = m.vmax;
  p.m_first = m.first;
  p.m_count = m.count;
  p.m_cells = (size_t)nx * ny;
  p.m_pg = m.pair_group;
  p.m_pk = m.pair_k;
  if (launches) *launches += 1;
  if (range) {
    const int R = range->radius;
    p.w_r = R;
    p.w_sw = win_sum_words(nx, R);
    p.w_r2 = range->shape == VHP_RANGE_DISK ? R * R : 2 * R * R;
    if (range->views) {
      p.m_views = range->views;
      p.m_disk = range->shape == VHP_RANGE_DISK;
      return m.f32 ? launch_tile_merge_range<kFmtMergeView32>(p, npairs, st)
                   : launch_tile_merge_range<kFmtMergeView64>(p, npairs, st);
    }
    return m.f32 ? launch_tile_merge_range<kFmtMergeRange32>(p, npairs, st)
                 : launch_tile_merge_range<kFmtMergeRange64>(p, npairs, st);
  }
  return m.f32 ? launch_tile_merge<kFmtMerge32>(p, npairs, st) : launch_tile_merge<kFmtMerge64>(p, npairs, st);
}

cudaError_t vhp_launch_sweep_cover(const VhpTilePlanes &pl, int nx, int ny, const int32_t *d_src_xy,
                                   const int32_t *d_src_map, int64_t npairs, int radius, double thr, uint32_t *d_bits,
                                   const double *d_rcp2, int *d_err, cudaStream_t st, int64_t *launches) {
  if (!(thr > 0.0)) return cudaErrorInvalidValue; // cells below the threshold are never written
  const VhpCoverBox b = vhp_cover_box(nx, ny, radius, 0, 0);
  cudaError_t e = cudaMemsetAsync(d_bits, 0, (size_t)npairs * b.H * b.W * sizeof(uint32_t), st);
  if (e != cudaSuccess) return e;
  TileArgs p;
  p.pl = pl;
  p.nx = nx;
  p.ny = ny;
  p.src_xy = d_src_xy;
  p.src_map = d_src_map;
  p.out = d_bits;
  p.rtab = reinterpret_cast<const double2 *>(d_rcp2);
  p.err = d_err;
  p.vec = 0;
  p.win_y0 = 0;
  p.win_y1 = ny;
  p.thr = thr;
  p.w_r = radius;
  p.w_sw = win_sum_words(nx, radius);
  if (launches) *launches += 1;
  return launch_tile_cover(p, npairs, st);
}

bool vhp_sweep_tile_supported(int nx, int ny) {
  return nx >= 1 && ny >= 1 && std::max(nx, ny) <= 16384 &&
         tile_smem_bytes<double>(nx, ny) <= 227u * 1024u;
}

// grid mode keeps the boundary rows in global memory: wider maps than the one-CTA kernel
bool vhp_sweep_grid_supported(int nx, int ny) {
  return nx >= 1 && ny >= 1 && std::max(nx, ny) <= 16384 &&
         tile_smem_bytes_grid<double>(nx, ny) <= 227u * 1024u;
}

void vhp_tile_plane_geometry(int nx, int ny, int *wx, int *wy, int *sum_words_per_map) {
  *wx = ((nx + 31) >> 5) + 1;
  *wy = ((ny + 31) >> 5) + 1;
  *sum_words_per_map = tile_sum_words(nx) * ((ny + 31) >> 5);
}

cudaError_t vhp_launch_pack_tile(const uint8_t *d_occ, int nmaps, int nx, int ny, uint32_t *rowF,
                                 uint32_t *rowR, uint32_t *colF, uint32_t *colR, uint32_t *bsum,
                                 cudaStream_t st, int64_t *launches) {
  int wx, wy, nsum;
  vhp_tile_plane_geometry(nx, ny, &wx, &wy, &nsum);
  const size_t tr = (size_t)nmaps * ny * wx, tc = (size_t)nmaps * nx * wy;
  const int bs = 256;
  const unsigned gr = (unsigned)std::min<size_t>((tr + bs - 1) / bs, 148u * 32u);
  const unsigned gc = (unsigned)std::min<size_t>((tc + bs - 1) / bs, 148u * 32u);
  pack_tile_rows_kernel<<<gr, bs, 0, st>>>(d_occ, nmaps, nx, ny, wx, rowF, rowR);
  pack_tile_cols_kernel<<<gc, bs, 0, st>>>(d_occ, nmaps, nx, ny, wy, colF, colR);
  cudaError_t e = cudaMemsetAsync(bsum, 0, (size_t)nmaps * nsum * sizeof(uint32_t), st);
  if (e != cudaSuccess) return e;
  const size_t nblk = (size_t)nmaps * ((nx + 31) >> 5) * ((ny + 31) >> 5);
  const unsigned gs = (unsigned)std::min<size_t>((nblk * 32 + bs - 1) / bs, 148u * 32u);
  pack_tile_sum_kernel<<<gs, bs, 0, st>>>(rowF, nmaps, nx, ny, wx, bsum);
  if (launches) *launches += 3;
  return cudaGetLastError();
}

cudaError_t vhp_launch_rcp2_table(double *d_table, int len, cudaStream_t st, int64_t *launches) {
  rcp2_table_kernel<<<(len + 255) / 256, 256, 0, st>>>(reinterpret_cast<double2 *>(d_table), len);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t vhp_launch_ratio2_selftest(const double *d_rcp2, int kmax,
                                       unsigned long long *d_mismatches, cudaStream_t st,
                                       int64_t *launches) {
  ratio2_selftest_kernel<<<kmax, 128, 0, st>>>(reinterpret_cast<const double2 *>(d_rcp2), kmax,
                                               d_mismatches);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t vhp_launch_sweep_tile(const VhpTilePlanes &pl, int nx, int ny, const int32_t *d_src_xy,
                                  const int32_t *d_src_map, int64_t npairs, vhp_dtype dtype,
                                  void *d_out, const double *d_rcp2, int *d_err, cudaStream_t st,
                                  int64_t *launches, const double *thr, bool bits) {
  TileArgs p;
  p.pl = pl;
  p.nx = nx;
  p.ny = ny;
  p.src_xy = d_src_xy;
  p.src_map = d_src_map;
  p.out = d_out;
  p.rtab = reinterpret_cast<const double2 *>(d_rcp2);
  p.err = d_err;
  const size_t esz = dtype == VHP_F32 ? 4 : 8;
  p.vec = ((uintptr_t)d_out % 16 == 0 && ((size_t)nx * esz) % 16 == 0) ? 1 : 0;
  p.win_y0 = 0;
  p.win_y1 = ny;
  cudaError_t e;
  if (thr && bits) { // one bit per cell, (fp64 value >= thr), into a zeroed buffer
    if (!(*thr > 0.0)) return cudaErrorInvalidValue; // cells below the threshold are never written
    p.thr = *thr;
    e = cudaMemsetAsync(d_out, 0, (size_t)npairs * ny * ((nx + 31) / 32) * sizeof(uint32_t), st);
    if (e == cudaSuccess) e = launch_tile_fmt<kFmtBits>(p, npairs, st);
  } else if (thr || bits) {
    return cudaErrorInvalidValue;
  } else {
    e = dtype == VHP_F32 ? launch_tile<float>(p, npairs, st) : launch_tile<double>(p, npairs, st);
  }
  if (launches) *launches += 1;
  return e;
}

void vhp_window_halo_rows(int nx, int ny, int sx, int sy, int y0, int y1, int32_t rows[4]) {
  for (int q = 0; q < 4; ++q) {
    int jw0, jw1, Jlo, Jhi, hy;
    tile_window_of(q, nx, ny, sx, sy, y0, y1, &jw0, &jw1, &Jlo, &Jhi, &hy);
    rows[q] = hy;
  }
}

// offset and size of the progress flags inside a grid workspace (reset between sweeps when a peer
// raises them, see VhpSweepPeer)
void vhp_sweep_grid_ws_flags(int nx, int ny, size_t *offset, size_t *bytes) {
  *offset = sizeof(double) * (size_t)tile_edge_doubles(nx, kTileWarps) + sizeof(int) * 4 * (size_t)tile_lm_cap(ny);
  *bytes = sizeof(int) * 4 * (size_t)tile_lm_cap(ny);
}

size_t vhp_sweep_grid_ws_bytes(int nx, int ny) {
  return sizeof(double) * (size_t)tile_edge_doubles(nx, kTileWarps) +
         sizeof(int) * (8 * (size_t)tile_lm_cap(ny) + 4);
}

namespace {

template <typename OutT>
cudaError_t launch_window(TileArgs &p, int sx, int sy, void *d_grid_ws, int grid_ctas,
                          cudaStream_t st, int64_t *launches) {
  if (d_grid_ws && grid_ctas > 1) {
    const int lmcap = tile_lm_cap(p.ny);
    p.g_edges = static_cast<double *>(d_grid_ws);
    p.g_lm = reinterpret_cast<int *>(p.g_edges + tile_edge_doubles(p.nx, kTileWarps));
    p.g_prog = p.g_lm + 4 * lmcap;
    p.g_next_row = p.g_prog + 4 * lmcap;
    const size_t smem = tile_smem_bytes_grid<OutT>(p.nx, p.ny);
    auto init = sweep_grid_kernel<OutT, kSweepGridInit>;
    auto work = sweep_grid_kernel<OutT, kSweepGridWork>;
    cudaError_t e = cudaFuncSetAttribute(init, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(work, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    init<<<1, kTileWarps * 32, smem, st>>>(p, sx, sy);
    work<<<grid_ctas, kTileWarps * 32, smem, st>>>(p, sx, sy);
    if (launches) *launches += 2;
    return cudaGetLastError();
  }
  const size_t smem = tile_smem_bytes<OutT>(p.nx, p.ny);
  cudaError_t e = cudaFuncSetAttribute(sweep_window_kernel<OutT>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  sweep_window_kernel<OutT><<<1, kTileWarps * 32, smem, st>>>(p, sx, sy);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

} // namespace

// d_grid_ws: vhp_sweep_grid_ws_bytes(nx, ny) bytes of device scratch, or null; grid_ctas > 1
// spreads the sweep over that many CTAs (grid mode), else one CTA does it.
cudaError_t vhp_launch_sweep_window(const VhpTilePlanes &pl, int nx, int ny, int sx, int sy, int y0,
                                    int y1, const double *const d_halo[4], vhp_dtype dtype,
                                    void *d_out_strip, const double *d_rcp2, int *d_err,
                                    void *d_grid_ws, int grid_ctas, cudaStream_t st,
                                    int64_t *launches, int qmask, const int *d_src_ctl,
                                    const VhpSweepPeer *peer) {
  TileArgs p;
  p.pl = pl;
  p.nx = nx;
  p.ny = ny;
  p.src_xy = nullptr;
  p.src_map = nullptr;
  p.out = d_out_strip;
  p.rtab = reinterpret_cast<const double2 *>(d_rcp2);
  p.err = d_err;
  const size_t esz = dtype == VHP_F32 ? 4 : 8;
  p.vec = ((uintptr_t)d_out_strip % 16 == 0 && ((size_t)nx * esz) % 16 == 0) ? 1 : 0;
  p.win_y0 = y0;
  p.win_y1 = y1;
  for (int q = 0; q < 4; ++q) p.halo[q] = d_halo ? d_halo[q] : nullptr;
  p.qmask = qmask;
  p.src_ctl = d_src_ctl;
  if (peer && d_grid_ws && grid_ctas > 1) { // peer hand-over exists in grid mode only
    const int lmcap = tile_lm_cap(ny);
    if (peer->x_ws) {
      p.x_edges = static_cast<double *>(peer->x_ws);
      p.x_prog = reinterpret_cast<int *>(p.x_edges + tile_edge_doubles(nx, kTileWarps)) + 4 * lmcap;
      p.x_y0 = peer->x_y0;
      p.x_y1 = peer->x_y1;
    }
    p.remote_mask = peer->remote_mask;
  }
  return dtype == VHP_F32 ? launch_window<float>(p, sx, sy, d_grid_ws, grid_ctas, st, launches)
                          : launch_window<double>(p, sx, sy, d_grid_ws, grid_ctas, st, launches);
}
