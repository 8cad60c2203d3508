// capi.cu -- extern "C" entry points of include/vhp.h: context management and the
// batched sweep / ray-casting / planner calls.  Plain pointers in, status out.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "vhp_internal.h"

namespace {

thread_local std::string g_last_error;

vhp_status fail(vhp_context *ctx, vhp_status st, const std::string &msg) {
  g_last_error = msg;
  if (ctx) ctx->last_error = msg;
  return st;
}

vhp_status cuda_fail(vhp_context *ctx, cudaError_t e, const char *what) {
  // a refused call (e.g. cudaFuncSetAttribute) stays the thread's last error, which the next call's check after a good
  // launch would report as its own: clear it once it is reported here
  (void)cudaGetLastError();
  return fail(ctx, VHP_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define VHP_CUDA(ctx, call)                                   \
  do {                                                        \
    cudaError_t e_ = (call);                                  \
    if (e_ != cudaSuccess) return cuda_fail(ctx, e_, #call);  \
  } while (0)

// Entry points run on the context's device and leave the caller's current device as they found it
// (a torch process with several GPUs keeps its own notion of the current device).
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != device) err = cudaSetDevice(device);
    else prev = -1; // nothing to restore
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};
#define VHP_ON_DEVICE(ctx)                 \
  DeviceGuard device_guard_((ctx)->device); \
  if (device_guard_.err != cudaSuccess) return cuda_fail(ctx, device_guard_.err, "cudaSetDevice")

vhp_status ensure(vhp_context *ctx, VhpDevBuf &b, size_t bytes) {
  if (bytes <= b.cap) return VHP_OK;
  if (b.p) {
    VHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    VHP_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
    VHP_CUDA(ctx, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
  }
  VHP_CUDA(ctx, cudaMalloc(&b.p, bytes));
  b.cap = bytes;
  return VHP_OK;
}

vhp_status ensure_rcp2(vhp_context *ctx, int len) {
  if (len <= ctx->rcp2_len) return VHP_OK;
  len = std::max(len, 4096 + 8);
  if (ctx->rcp2_table) {
    VHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    VHP_CUDA(ctx, cudaFree(ctx->rcp2_table));
    ctx->rcp2_table = nullptr;
    ctx->rcp2_len = 0;
  }
  VHP_CUDA(ctx, cudaMalloc(&ctx->rcp2_table, (size_t)len * 2 * sizeof(double)));
  VHP_CUDA(ctx, vhp_launch_rcp2_table(ctx->rcp2_table, len, ctx->stream, &ctx->launches));
  ctx->rcp2_len = len;
  return VHP_OK;
}

// (re)build the bit planes of the tile kernel for d_occ unless they are cached for this pointer
vhp_status pack_tile(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                     bool force) {
  if (!force && ctx->planes_sticky && ctx->tile_src == d_occ && ctx->tile_nmaps == nmaps &&
      ctx->tile_nx == nx && ctx->tile_ny == ny)
    return VHP_OK;
  int wx, wy, nsum;
  vhp_tile_plane_geometry(nx, ny, &wx, &wy, &nsum);
  const size_t row_plane = (size_t)ny * wx, col_plane = (size_t)nx * wy;
  const size_t bytes = (size_t)nmaps * (2 * (row_plane + col_plane) + nsum) * sizeof(uint32_t);
  if (bytes > ctx->tile_bytes) {
    if (ctx->tile_buf) {
      VHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      VHP_CUDA(ctx, cudaFree(ctx->tile_buf));
      ctx->tile_buf = nullptr;
      ctx->tile_bytes = 0;
      ctx->tile_src = nullptr;
      ctx->planes_sticky = false;
    }
    VHP_CUDA(ctx, cudaMalloc(&ctx->tile_buf, bytes));
    ctx->tile_bytes = bytes;
  }
  uint32_t *rowF = ctx->tile_buf, *rowR = rowF + (size_t)nmaps * row_plane;
  uint32_t *colF = rowR + (size_t)nmaps * row_plane, *colR = colF + (size_t)nmaps * col_plane;
  uint32_t *bsum = colR + (size_t)nmaps * col_plane;
  VHP_CUDA(ctx, vhp_launch_pack_tile(d_occ, nmaps, nx, ny, rowF, rowR, colF, colR, bsum,
                                     ctx->stream, &ctx->launches));
  ctx->tile.rowF = rowF; ctx->tile.rowR = rowR;
  ctx->tile.colF = colF; ctx->tile.colR = colR;
  ctx->tile.bsum = bsum;
  ctx->tile.wx = wx; ctx->tile.wy = wy;
  ctx->tile.row_plane = row_plane; ctx->tile.col_plane = col_plane;
  ctx->tile_src = d_occ; ctx->tile_nmaps = nmaps; ctx->tile_nx = nx; ctx->tile_ny = ny;
  return VHP_OK;
}

vhp_status check_grid_dtype(vhp_context *ctx, int nx, int ny, int dtype) {
  if ((int64_t)nx * ny > (int64_t)1 << 30 || nx > 16384 || ny > 16384)
    return fail(ctx, VHP_ERR_UNSUPPORTED, "grid larger than 16384 x 16384 is not supported");
  if (dtype != VHP_F32 && dtype != VHP_F64) return fail(ctx, VHP_ERR_INVALID_ARG, "bad dtype");
  return VHP_OK;
}

vhp_status check_common(vhp_context *ctx, const void *occ, int nmaps, int nx, int ny,
                        const void *xy, int64_t n, int dtype, const void *out) {
  if (!ctx) return fail(nullptr, VHP_ERR_INVALID_ARG, "null context");
  if (!occ || !xy || !out) return fail(ctx, VHP_ERR_INVALID_ARG, "null buffer");
  if (nmaps < 1 || nx < 1 || ny < 1 || n < 0)
    return fail(ctx, VHP_ERR_INVALID_ARG, "bad sizes");
  return check_grid_dtype(ctx, nx, ny, dtype);
}

// host-side validation of (x, y[, map]) items
vhp_status check_points(vhp_context *ctx, const int32_t *xy, int per_item, const int32_t *maps,
                        int64_t n, int nmaps, int nx, int ny, const char *what) {
  for (int64_t i = 0; i < n; ++i) {
    if (maps && (maps[i] < 0 || maps[i] >= nmaps))
      return fail(ctx, VHP_ERR_INVALID_ARG, std::string(what) + ": map index out of range");
    if (per_item == 2) {
      const int x = xy[2 * i], y = xy[2 * i + 1];
      if (x < 0 || x >= nx || y < 0 || y >= ny)
        return fail(ctx, VHP_ERR_INVALID_ARG,
                    std::string(what) + ": source outside the grid at item " + std::to_string(i));
    }
  }
  return VHP_OK;
}

vhp_status check_device_error(vhp_context *ctx) {
  int flag = 0;
  VHP_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost,
                                ctx->stream));
  VHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (flag) {
    VHP_CUDA(ctx, cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
    if (flag & 4)
      return fail(ctx, VHP_ERR_INVALID_ARG, "inconsistent source groups (group_ptr / group_map)");
    if (flag & 8)
      return fail(ctx, VHP_ERR_INVALID_ARG,
                  "a candidate's view (r, ax, ay, bx, by) is invalid: r outside [0, radius], a or b (0, 0), or a "
                  "component outside [-32767, 32767]");
    if (flag & 16)
      return fail(ctx, VHP_ERR_INVALID_ARG,
                  "a source's view (r, ax, ay, bx, by) is invalid: r outside [0, radius], a or b (0, 0), or a "
                  "component outside [-32767, 32767]; that source contributed nothing");
    if (flag & 32)
      return fail(ctx, VHP_ERR_INVALID_ARG,
                  "vhp_visibility_cover_budget_batch_dev: a candidate's cost is 0; that candidate was never picked");
    return fail(ctx, VHP_ERR_INVALID_ARG, "a source / start / end point lies outside the grid");
  }
  return VHP_OK;
}

// Grid-mode strip sweep of rows [y0, y1) (see vhp_strip_sweep_dev): CTAs to spread one sweep over.
int grid_sweep_ctas(const vhp_context *ctx, int rows) {
  return std::max(2, std::min(2 * ctx->sm_count, (4 * (rows / 32 + 2) + 7) / 8));
}

// May a single sweep of this map be spread over many CTAs?  (Maps too wide for the one-CTA kernel need it.)
bool grid_mode_available(const vhp_context *ctx, int nx, int ny) {
  return ctx->grid_sweep != 0 && vhp_sweep_grid_supported(nx, ny);
}

// Do the batched sweeps of this map read the bit planes (the tile kernel or grid mode, not the naive kernel)?
bool sweeps_use_planes(const vhp_context *ctx, int nx, int ny) {
  return ctx->sweep_impl == 0 && (vhp_sweep_tile_supported(nx, ny) || vhp_sweep_grid_supported(nx, ny));
}

// Kernel of a batch of n whole-field sweeps.  A few sweeps of a large map run one at a time on the whole
// GPU (grid mode, see vhp_strip_sweep_dev) instead of one CTA per pair.  (1000^2: up to 4 pairs, 2048^2
// and up: 16; maps too wide for the one-CTA kernel's shared memory: up to 16 pairs whatever the size.)
// Every route that claims to equal run_dev's fields (bits, merged outputs) asks this function.
enum class SweepRoute { Tile, Grid, Naive };

SweepRoute sweep_route(const vhp_context *ctx, int nx, int ny, int64_t n) {
  if (ctx->sweep_impl != 0) return SweepRoute::Naive;
  const bool tile_ok = vhp_sweep_tile_supported(nx, ny);
  const int64_t grid_max = tile_ok ? std::min<int64_t>(16, (int64_t)((size_t)nx * ny / 250000)) : 16;
  if (vhp_sweep_grid_supported(nx, ny) && (ctx->grid_sweep == 2 || (ctx->grid_sweep == 1 && n <= grid_max)))
    return SweepRoute::Grid;
  return tile_ok ? SweepRoute::Tile : SweepRoute::Naive;
}

// Range-limited windows sweep only the window on one CTA whatever the batch size, so only a forced grid
// mode turns them away (their fallback goes through run_dev and sweep_route).
bool window_direct_route(const vhp_context *ctx, int nx, int ny, int radius) {
  return ctx->sweep_impl == 0 && ctx->grid_sweep != 2 && vhp_sweep_window_supported(nx, ny, radius);
}

// bit planes of map m of the packed batch (the grid kernels sweep "map 0")
VhpTilePlanes planes_of_map(const vhp_context *ctx, size_t m, int nx, int ny) {
  int wx, wy, nsum;
  vhp_tile_plane_geometry(nx, ny, &wx, &wy, &nsum);
  VhpTilePlanes pl = ctx->tile;
  pl.rowF += m * pl.row_plane; pl.rowR += m * pl.row_plane;
  pl.colF += m * pl.col_plane; pl.colR += m * pl.col_plane;
  pl.bsum += m * (size_t)nsum;
  return pl;
}

enum class Op { Sweep, Raycast, Window };

vhp_status run_dev(vhp_context *ctx, Op op, const uint8_t *d_occ, int nmaps, int nx, int ny,
                   const int32_t *d_xy, const int32_t *d_map, int64_t n, vhp_dtype dtype,
                   void *d_out) {
  if (n == 0) return VHP_OK;
  if (op == Op::Raycast) {
    VHP_CUDA(ctx, vhp_launch_raycast(d_occ, nx, ny, d_xy, d_map, n, dtype, d_out, ctx->d_err,
                                     ctx->stream, &ctx->launches));
    return VHP_OK;
  }
  const size_t esz = dtype == VHP_F32 ? 4 : 8;
  const size_t cells = (size_t)nx * ny;
  const SweepRoute route = sweep_route(ctx, nx, ny, n);
  vhp_status st;
  if (route == SweepRoute::Naive) {
    // chunk so that the scratch fronts stay small
    const int64_t chunk = 4096;
    if ((st = ensure(ctx, ctx->b_scratch, vhp_sweep_naive_scratch_bytes(nx, ny, std::min(n, chunk)))) != VHP_OK)
      return st;
    for (int64_t p0 = 0; p0 < n; p0 += chunk) {
      const int64_t np = std::min(chunk, n - p0);
      VHP_CUDA(ctx, vhp_launch_sweep_naive(d_occ, nx, ny, d_xy + 2 * p0, d_map ? d_map + p0 : nullptr,
                                           np, dtype, (char *)d_out + (size_t)p0 * nx * ny * esz,
                                           (double *)ctx->b_scratch.p, ctx->d_err, ctx->stream,
                                           &ctx->launches));
    }
    return VHP_OK;
  }
  if ((st = ensure_rcp2(ctx, std::max(nx, ny) + 64)) != VHP_OK) return st;
  if ((st = pack_tile(ctx, d_occ, nmaps, nx, ny, false)) != VHP_OK) return st;
  if (route == SweepRoute::Tile) {
    VHP_CUDA(ctx, vhp_launch_sweep_tile(ctx->tile, nx, ny, d_xy, d_map, n, dtype, d_out,
                                        ctx->rcp2_table, ctx->d_err, ctx->stream, &ctx->launches));
    return VHP_OK;
  }
  std::vector<int32_t> h_xy(2 * (size_t)n), h_map;
  VHP_CUDA(ctx, cudaMemcpyAsync(h_xy.data(), d_xy, h_xy.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (d_map) {
    h_map.resize((size_t)n);
    VHP_CUDA(ctx, cudaMemcpyAsync(h_map.data(), d_map, h_map.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  VHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if ((st = ensure(ctx, ctx->b_grid, vhp_sweep_grid_ws_bytes(nx, ny))) != VHP_OK) return st;
  const int ctas = grid_sweep_ctas(ctx, ny);
  for (int64_t k = 0; k < n; ++k) {
    const int sx = h_xy[2 * k], sy = h_xy[2 * k + 1];
    const int64_t m = d_map ? h_map[k] : 0;
    if (sx < 0 || sx >= nx || sy < 0 || sy >= ny || m < 0 || m >= nmaps)
      return fail(ctx, VHP_ERR_INVALID_ARG, "a source / start / end point lies outside the grid");
    VHP_CUDA(ctx, vhp_launch_sweep_window(planes_of_map(ctx, (size_t)m, nx, ny), nx, ny, sx, sy, 0, ny, nullptr,
                                          dtype, (char *)d_out + (size_t)k * cells * esz, ctx->rcp2_table,
                                          ctx->d_err, ctx->b_grid.p, ctas, ctx->stream, &ctx->launches));
  }
  return VHP_OK;
}

// pairs per chunk of fp64 fields (4 GB) where a route goes through whole fields (binary, merged and window outputs)
int64_t bin_chunk_pairs(size_t cells, int64_t n) {
  return std::min<int64_t>(n, std::max<int64_t>(1, (int64_t)(((size_t)4 << 30) / (cells * 8))));
}

// ---- range-limited windows (vhp_visibility_window_batch) ----------------------------------------
// Direct: the one-CTA tile kernel sweeps only each pair's window (kFmtWindow).  Otherwise (the naive kernel, grid
// mode forced, or a window whose state does not fit one CTA) chunks of full fields go through run_dev, which picks
// grid mode or the naive kernel as for vhp_visibility_batch, and window_crop_kernel cuts the windows out.
size_t window_pair_bytes(int radius, vhp_dtype dtype) {
  const size_t w = 2 * (size_t)radius + 1;
  return w * w * (dtype == VHP_F32 ? 4 : 8);
}

vhp_status run_window_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny, const int32_t *d_xy,
                          const int32_t *d_map, int64_t n, int radius, vhp_dtype dtype, void *d_out) {
  if (n == 0) return VHP_OK;
  vhp_status st;
  if (window_direct_route(ctx, nx, ny, radius)) {
    if ((st = ensure_rcp2(ctx, std::min(std::max(nx, ny), radius + 1) + 64)) != VHP_OK) return st;
    if ((st = pack_tile(ctx, d_occ, nmaps, nx, ny, false)) != VHP_OK) return st;
    VHP_CUDA(ctx, vhp_launch_sweep_window_batch(ctx->tile, nmaps, nx, ny, d_xy, d_map, n, radius, dtype, d_out,
                                                ctx->rcp2_table, ctx->d_err, ctx->stream, &ctx->launches));
    return VHP_OK;
  }
  const size_t cells = (size_t)nx * ny, esz = dtype == VHP_F32 ? 4 : 8;
  const int64_t chunk = bin_chunk_pairs(cells, n);
  if ((st = ensure(ctx, ctx->b_bin, (size_t)chunk * cells * esz)) != VHP_OK) return st;
  if (d_map && (st = ensure(ctx, ctx->b_misc, 12 * (size_t)chunk)) != VHP_OK) return st;
  for (int64_t p0 = 0; p0 < n; p0 += chunk) {
    const int64_t np = std::min(chunk, n - p0);
    const int32_t *xy = d_xy + 2 * p0, *mp = d_map ? d_map + p0 : nullptr;
    if (mp) { // the full sweeps must not read beyond the maps
      int32_t *sxy = (int32_t *)ctx->b_misc.p, *smp = sxy + 2 * chunk;
      VHP_CUDA(ctx, vhp_launch_window_pairs(xy, mp, np, nmaps, sxy, smp, ctx->sm_count, ctx->stream, &ctx->launches));
      xy = sxy;
      mp = smp;
    }
    if ((st = run_dev(ctx, Op::Sweep, d_occ, nmaps, nx, ny, xy, mp, np, dtype, ctx->b_bin.p)) != VHP_OK) return st;
    VHP_CUDA(ctx, vhp_launch_window_crop(ctx->b_bin.p, np, nx, ny, xy, radius, dtype,
                                         (char *)d_out + (size_t)p0 * window_pair_bytes(radius, dtype),
                                         ctx->sm_count, ctx->stream, &ctx->launches));
  }
  return VHP_OK;
}

// Upload of a host batch into b_occ / b_src / b_map: the maps, n items of item_bytes each and, when
// maps is not null, n map indices.  Bit planes of an older content of b_occ (sticky ones of
// vhp_prepare_maps_dev too) are dropped; pack: build them now, once for every chunk of the call.
// The caller holds a PlanesGuard, which drops them again when the call returns.
vhp_status stage_host_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny, const void *items,
                            size_t item_bytes, int64_t n, const int32_t *maps, bool pack) {
  const size_t occ_bytes = (size_t)nmaps * nx * ny;
  vhp_status st;
  if ((st = ensure(ctx, ctx->b_occ, occ_bytes)) != VHP_OK) return st;
  if ((st = ensure(ctx, ctx->b_src, item_bytes * (size_t)std::max<int64_t>(n, 1))) != VHP_OK) return st;
  if (maps && (st = ensure(ctx, ctx->b_map, (size_t)n * 4)) != VHP_OK) return st;
  VHP_CUDA(ctx, cudaMemcpyAsync(ctx->b_occ.p, occ, occ_bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (n > 0)
    VHP_CUDA(ctx, cudaMemcpyAsync(ctx->b_src.p, items, (size_t)n * item_bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (maps) VHP_CUDA(ctx, cudaMemcpyAsync(ctx->b_map.p, maps, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  ctx->planes_sticky = false;
  ctx->tile_src = nullptr;
  if (!pack) return VHP_OK;
  if ((st = pack_tile(ctx, (const uint8_t *)ctx->b_occ.p, nmaps, nx, ny, true)) != VHP_OK) return st;
  ctx->planes_sticky = true;
  return VHP_OK;
}

// The planes a host call packed point into b_occ, which the next call overwrites: drop them on every exit.
struct PlanesGuard {
  vhp_context *ctx;
  explicit PlanesGuard(vhp_context *c) : ctx(c) {}
  ~PlanesGuard() {
    ctx->planes_sticky = false;
    ctx->tile_src = nullptr;
  }
};

// Delivery of pairs [p_begin, n) to the host buffer `out` in chunks of `chunk` pairs of pair_bytes each:
// produce(p0, np, d_buf) computes a chunk into one of two device buffers on the stream, and the copy
// stream takes it to `out` under the work of the next chunk.  Both streams are synchronised on every exit.
template <class F>
vhp_status pipelined_d2h(vhp_context *ctx, int64_t p_begin, int64_t n, int64_t chunk, size_t pair_bytes, void *out,
                         F produce) {
  vhp_status result = ensure(ctx, ctx->b_out[0], (size_t)chunk * pair_bytes);
  if (result == VHP_OK && n - p_begin > chunk) result = ensure(ctx, ctx->b_out[1], (size_t)chunk * pair_bytes);
  int it = 0;
  for (int64_t p0 = p_begin; p0 < n && result == VHP_OK; p0 += chunk, ++it) {
    const int b = it & 1;
    const int64_t np = std::min(chunk, n - p0);
    cudaError_t e = cudaSuccess;
    if (it >= 2) e = cudaStreamWaitEvent(ctx->stream, ctx->ev_copied[b], 0); // the copy that last read buffer b is done
    if (e != cudaSuccess) { result = cuda_fail(ctx, e, "cudaStreamWaitEvent"); break; }
    if ((result = produce(p0, np, ctx->b_out[b].p)) != VHP_OK) break;
    e = cudaEventRecord(ctx->ev_done[b], ctx->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_done[b], 0);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync((char *)out + (size_t)p0 * pair_bytes, ctx->b_out[b].p, (size_t)np * pair_bytes,
                          cudaMemcpyDeviceToHost, ctx->copy_stream);
    if (e == cudaSuccess) e = cudaEventRecord(ctx->ev_copied[b], ctx->copy_stream);
    if (e != cudaSuccess) { result = cuda_fail(ctx, e, "D2H of a chunk: enqueue"); break; }
    ctx->last_d2h_bytes += (int64_t)((size_t)np * pair_bytes);
  }
  cudaError_t e1 = cudaStreamSynchronize(ctx->copy_stream);
  cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
  if (result != VHP_OK) return result;
  if (e1 != cudaSuccess) return cuda_fail(ctx, e1, "sync copy stream");
  if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "sync stream");
  return VHP_OK;
}

// Plain transport of the host-buffer entry points: run in chunks of pairs from p_begin on and
// overlap the D2H of chunk c with the kernel of chunk c+1 (pipelined_d2h).
// Op::Window delivers the windows of `radius`, every other op whole fields.
vhp_status run_host_plain(vhp_context *ctx, Op op, int nmaps, int nx, int ny, const int32_t *d_xy,
                          const int32_t *d_map, int64_t n, int64_t p_begin, vhp_dtype dtype,
                          void *out, int radius = 0) {
  const size_t pair_bytes =
      op == Op::Window ? window_pair_bytes(radius, dtype) : (size_t)nx * ny * (dtype == VHP_F32 ? 4 : 8);
  const int64_t chunk = std::min(std::max<int64_t>(1, (int64_t)(((size_t)1 << 30) / pair_bytes)), n - p_begin);
  // pin the caller's buffer for full-rate async copies (ignore "already pinned").  Page-locking
  // costs milliseconds: small results (a single 101 x 101 sweep is 80 KB) are copied as they are.
  const size_t out_bytes = (size_t)(n - p_begin) * pair_bytes;
  char *const out_first = (char *)out + (size_t)p_begin * pair_bytes;
  const bool registered = out_bytes >= ((size_t)32 << 20) &&
                          cudaHostRegister(out_first, out_bytes, cudaHostRegisterDefault) == cudaSuccess;
  (void)cudaGetLastError();
  const uint8_t *d_occ = (const uint8_t *)ctx->b_occ.p;
  auto produce = [&](int64_t p0, int64_t np, void *buf) {
    const int32_t *xy = d_xy + 2 * p0, *mp = d_map ? d_map + p0 : nullptr;
    return op == Op::Window ? run_window_dev(ctx, d_occ, nmaps, nx, ny, xy, mp, np, radius, dtype, buf)
                            : run_dev(ctx, op, d_occ, nmaps, nx, ny, xy, mp, np, dtype, buf);
  };
  const vhp_status result = pipelined_d2h(ctx, p_begin, n, chunk, pair_bytes, out, produce);
  if (registered) cudaHostUnregister(out_first);
  return result;
}

// Packed transport (result_transport.cu, host_expand.cpp): every chunk of results is packed on
// the device into uniform / literal 128-byte units; only the meta data and the literal units
// cross PCIe and a pool of host threads rebuilds the exact bytes in the caller's buffer.
// Three sets of buffers: while chunk c is computed and packed, the literals of chunk c-1 are
// copied and chunk c-2 is expanded.  When the caller's buffer is pinned, mapped and 16-byte
// aligned ("direct"), the pack kernel stores the literal units straight to their place in it
// and the host threads only write the uniform units.  In automatic mode the call gives up
// after the first chunks when they hardly compress; *resume_from is the first pair not
// delivered.
vhp_status run_host_packed(vhp_context *ctx, Op op, int nmaps, int nx, int ny, const int32_t *d_xy,
                           const int32_t *d_map, int64_t n, vhp_dtype dtype, void *out,
                           int64_t *resume_from) {
  constexpr int NS = vhp_context::kPackSets;
  const size_t cells = (size_t)nx * ny, esz = dtype == VHP_F32 ? 4 : 8;
  const size_t pair_bytes = cells * esz;
  int64_t chunk = std::max<int64_t>(1, (int64_t)(((size_t)256 << 20) / pair_bytes));
  chunk = std::min(chunk, n);
  const int64_t nchunks = (n + chunk - 1) / chunk;
  const int64_t units_max = (int64_t)(((size_t)chunk * pair_bytes + kVhpPackUnit - 1) / kVhpPackUnit);
  const size_t meta_max = vhp_pack_meta_bytes(units_max, (int)esz), lit_max = (size_t)units_max * kVhpPackUnit;
  vhp_status st;
  // direct mode: a device-accessible address of the caller's buffer, if it is pinned host memory
  char *out_dev = nullptr;
  {
    cudaPointerAttributes attr;
    void *dp = nullptr;
    if (ctx->result_direct && (((uintptr_t)out) & 15u) == 0 && pair_bytes % 16 == 0 &&
        cudaPointerGetAttributes(&attr, out) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
        cudaHostGetDevicePointer(&dp, out, 0) == cudaSuccess)
      out_dev = (char *)dp;
    (void)cudaGetLastError();
  }
  const bool direct = out_dev != nullptr;
  if (!ctx->expand_pool) {
    int t = 0;
    if (const char *e = std::getenv("VHP_HOST_THREADS")) t = std::atoi(e);
    if (t <= 0) t = (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
    try {
      ctx->expand_pool = new VhpExpandPool(t);
    } catch (...) { // no host threads to be had: deliver everything by plain copies
      ctx->expand_pool = nullptr;
      *resume_from = 0;
      return VHP_OK;
    }
  }
  ctx->last_transport_packed = direct ? 2 : 1;
  const int nsets = (int)std::min<int64_t>(NS, nchunks);
  for (int s = 0; s < nsets; ++s) {
    if ((st = ensure(ctx, ctx->b_pack_out[s], lit_max)) != VHP_OK) return st;
    if ((st = ensure(ctx, ctx->b_pack_meta[s], meta_max)) != VHP_OK) return st;
    if (!direct && (st = ensure(ctx, ctx->b_pack_lit[s], lit_max)) != VHP_OK) return st;
  }
  const size_t lit_need = direct ? 0 : lit_max;
  if (meta_max > ctx->h_pack_meta_cap || lit_need > ctx->h_pack_lit_cap) {
    for (int s = 0; s < NS; ++s) {
      if (ctx->h_pack_meta[s]) cudaFreeHost(ctx->h_pack_meta[s]);
      if (ctx->h_pack_lit[s]) cudaFreeHost(ctx->h_pack_lit[s]);
      ctx->h_pack_meta[s] = ctx->h_pack_lit[s] = nullptr;
    }
    ctx->h_pack_meta_cap = ctx->h_pack_lit_cap = 0;
    for (int s = 0; s < NS; ++s) {
      VHP_CUDA(ctx, cudaHostAlloc(&ctx->h_pack_meta[s], meta_max, cudaHostAllocDefault));
      if (lit_need) VHP_CUDA(ctx, cudaHostAlloc(&ctx->h_pack_lit[s], lit_need, cudaHostAllocDefault));
    }
    ctx->h_pack_meta_cap = meta_max;
    ctx->h_pack_lit_cap = lit_need;
  }
  VhpExpandPool &pool = *ctx->expand_pool;
  int64_t tickets[NS] = {0, 0, 0}, last_ticket = 0;
  int64_t lit_units_total = 0, units_total = 0;
  bool bail = false;
  vhp_status result = VHP_OK;

  // Direct mode: the device can also deliver a share of the mask words completely (uniform
  // units included).  Off by default: on the B200 boxes every byte that arrives over PCIe
  // while 16 host threads stream into the same memory costs about as much time as 3.5 bytes
  // written by the host threads (share 0 / 2 / 4 / 6 sixteenths: 96 / 125 / 155 / 184 ms for
  // 16.4 GB), so the fastest split moves as few bytes over PCIe as possible.
  double trace_pack_ms = 0.0, trace_wait_s = 0.0, trace_ticket_s = 0.0;
  const double trace_busy0 = pool.busy_seconds();
  const auto trace_t0 = std::chrono::steady_clock::now();
  int share_of[NS] = {0, 0, 0};
  auto gpu_share_now = [&]() -> int { return std::max(0, std::min(ctx->result_gpu_share, 16)); };
  auto chunk_units = [&](int64_t it) {
    const int64_t np = std::min(chunk, n - it * chunk);
    return (int64_t)(((size_t)np * pair_bytes + kVhpPackUnit - 1) / kVhpPackUnit);
  };
  auto launch = [&](int64_t it) -> vhp_status {
    const int s = (int)(it % NS);
    const int64_t p0 = it * chunk, np = std::min(chunk, n - p0);
    vhp_status r = run_dev(ctx, op, (const uint8_t *)ctx->b_occ.p, nmaps, nx, ny, d_xy + 2 * p0,
                           d_map ? d_map + p0 : nullptr, np, dtype, ctx->b_pack_out[s].p);
    if (r != VHP_OK) return r;
    // packing (PCIe-bound in direct mode) runs on the copy stream, so that the sweeps of the
    // next chunk overlap it
    VHP_CUDA(ctx, cudaEventRecord(ctx->ev_pack_lit[s], ctx->stream));
    VHP_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_pack_lit[s], 0));
    VHP_CUDA(ctx, cudaEventRecord(ctx->ev_pack_t0[s], ctx->copy_stream));
    const int64_t nu = chunk_units(it);
    const int tail_partial = ((size_t)np * pair_bytes) % kVhpPackUnit != 0;
    share_of[s] = direct ? gpu_share_now() : 0;
    VHP_CUDA(ctx, vhp_launch_pack_results(ctx->b_pack_out[s].p, nu, (int)esz, ctx->b_pack_meta[s].p,
                                          ctx->b_pack_lit[s].p,
                                          direct ? out_dev + (size_t)p0 * pair_bytes : nullptr,
                                          tail_partial, share_of[s], ctx->sm_count,
                                          ctx->copy_stream, &ctx->launches));
    VHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_pack_meta[s], ctx->b_pack_meta[s].p, vhp_pack_meta_bytes(nu, (int)esz),
                                  cudaMemcpyDeviceToHost, ctx->copy_stream));
    VHP_CUDA(ctx, cudaEventRecord(ctx->ev_pack_meta[s], ctx->copy_stream));
    return VHP_OK;
  };
  auto finish = [&](int64_t it) -> vhp_status {
    const int s = (int)(it % NS);
    const int64_t p0 = it * chunk, np = std::min(chunk, n - p0);
    const int64_t nu = chunk_units(it), nwords = (nu + 31) / 32;
    const auto tw0 = std::chrono::steady_clock::now();
    VHP_CUDA(ctx, cudaEventSynchronize(ctx->ev_pack_meta[s]));
    trace_wait_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - tw0).count();
    if (ctx->transport_trace) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ctx->ev_pack_t0[s], ctx->ev_pack_meta[s]) == cudaSuccess)
        trace_pack_ms += ms;
    }
    const char *meta = (const char *)ctx->h_pack_meta[s];
    const uint64_t nlit = *(const uint64_t *)meta;
    if (nlit && !direct) {
      VHP_CUDA(ctx, cudaMemcpyAsync(ctx->h_pack_lit[s], ctx->b_pack_lit[s].p,
                                    (size_t)nlit * kVhpPackUnit, cudaMemcpyDeviceToHost,
                                    ctx->copy_stream));
      VHP_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
    }
    // words the device delivered completely (their literal units are not in the cursor)
    const int64_t gpu_words = share_of[s] ? ((nwords - 1) / 16) * share_of[s] +
                                                std::min<int64_t>((nwords - 1) % 16, share_of[s])
                                          : 0;
    ctx->last_d2h_bytes += (int64_t)(vhp_pack_meta_bytes(nu, (int)esz) + (size_t)nlit * kVhpPackUnit +
                                     (size_t)gpu_words * 32 * kVhpPackUnit);
    lit_units_total += (int64_t)nlit;
    units_total += nu - gpu_words * 32; // the literal fraction is measured on the host's words
    VhpPackedChunk c;
    c.mask = (const uint32_t *)(meta + kVhpPackMetaHead);
    c.word_base = c.mask + nwords;
    c.vmask = c.word_base + nwords;
    c.elem_bytes = (int)esz;
    c.literals = direct ? nullptr : (const char *)ctx->h_pack_lit[s];
    c.tail = meta + 16;
    c.gpu_share = share_of[s];
    c.dst = (char *)out + (size_t)p0 * pair_bytes;
    c.nunits = nu;
    c.valid_bytes = (size_t)np * pair_bytes;
    tickets[s] = last_ticket = pool.submit(c);
    return VHP_OK;
  };

  int64_t launched = 0, finished = 0;
  for (int64_t it = 0; it < nchunks && result == VHP_OK && !bail; ++it) {
    const int s = (int)(it % NS);
    if (tickets[s]) { // staging set s is free again
      const auto tt0 = std::chrono::steady_clock::now();
      pool.wait(tickets[s]);
      trace_ticket_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - tt0).count();
    }
    if ((result = launch(it)) != VHP_OK) break;
    ++launched;
    if (it >= 1) {
      if ((result = finish(it - 1)) != VHP_OK) break;
      ++finished;
      // automatic mode: results that hardly compress are cheaper to copy directly
      if (ctx->result_transport == 1 && finished == 1 && lit_units_total * 10 > units_total * 6)
        bail = true;
    }
  }
  while (result == VHP_OK && finished < launched) {
    result = finish(finished);
    if (result == VHP_OK) ++finished;
  }
  if (last_ticket) pool.wait(last_ticket);
  cudaError_t e1 = cudaStreamSynchronize(ctx->copy_stream);
  cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
  if (e2 == cudaSuccess) e2 = e1;
  if (result != VHP_OK) return result;
  if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "sync stream");
  *resume_from = std::min(n, launched * chunk);
  if (ctx->transport_trace)
    std::fprintf(stderr,
                 "[vhp transport] %s, %lld chunks: wall %.1f ms | packing on the GPU %.1f ms | host "
                 "expansion %.1f ms (%d threads) | main thread waited %.1f ms for the GPU, %.1f ms "
                 "for the host threads | %.2f of %.2f GB over PCIe\n",
                 direct ? "direct" : "staged", (long long)launched,
                 1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - trace_t0).count(),
                 trace_pack_ms, 1e3 * (pool.busy_seconds() - trace_busy0), pool.threads(),
                 1e3 * trace_wait_s, 1e3 * trace_ticket_s, ctx->last_d2h_bytes / 1e9,
                 (double)(launched * chunk * pair_bytes) / 1e9);
  return VHP_OK;
}

// ---- packed handle: the lossless packed form of a batch of fields, kept on the host -------------
// vhp_visibility_batch_packed runs the same chunks as run_host_packed in staged form, but the meta
// blocks and literal streams stay in pinned memory owned by the handle instead of being expanded:
// the call moves 3-7 % of the field bytes over PCIe and writes nothing else to host memory.
// vhp_packed_expand rebuilds any range of pairs later (bit-identical to vhp_visibility_batch).
} // namespace

struct vhp_packed {
  struct Block { char *p; size_t cap, used; };
  struct Chunk { size_t meta_off, lit_off; int meta_blk, lit_blk; int64_t nunits, np; uint64_t nlit; };
  int device = 0;
  int nx = 0, ny = 0, elem = 4;
  int64_t npairs = 0, chunk_pairs = 0;
  size_t pair_bytes = 0;
  std::vector<Block> blocks; // pinned host memory, reused by the next call on this handle
  std::vector<Chunk> chunks;
  int64_t bytes_held = 0;

  // `bytes` of pinned memory, 256-byte aligned: from the first block with room, else a new block
  bool take(size_t bytes, int *blk, size_t *off) {
    bytes = (bytes + 255) & ~(size_t)255;
    for (size_t b = 0; b < blocks.size(); ++b)
      if (blocks[b].cap - blocks[b].used >= bytes) {
        *blk = (int)b; *off = blocks[b].used; blocks[b].used += bytes;
        return true;
      }
    Block nb{nullptr, std::max<size_t>(bytes, (size_t)128 << 20), 0};
    if (cudaHostAlloc((void **)&nb.p, nb.cap, cudaHostAllocDefault) != cudaSuccess) {
      (void)cudaGetLastError();
      return false;
    }
    nb.used = bytes;
    blocks.push_back(nb);
    *blk = (int)blocks.size() - 1; *off = 0;
    return true;
  }
  VhpPackedChunk view(const Chunk &c) const {
    const char *meta = blocks[c.meta_blk].p + c.meta_off;
    const int64_t nwords = (c.nunits + 31) / 32;
    VhpPackedChunk v;
    v.mask = (const uint32_t *)(meta + kVhpPackMetaHead);
    v.word_base = v.mask + nwords;
    v.vmask = v.word_base + nwords;
    v.elem_bytes = elem;
    v.literals = c.nlit ? blocks[c.lit_blk].p + c.lit_off : meta; // (never read when there are none)
    v.nunits = c.nunits;
    v.valid_bytes = (size_t)c.np * pair_bytes;
    return v;
  }
};

namespace {

vhp_status run_host_to_packed(vhp_context *ctx, int nmaps, int nx, int ny, const int32_t *d_xy,
                              const int32_t *d_map, int64_t n, vhp_dtype dtype, vhp_packed *h) {
  constexpr int NS = vhp_context::kPackSets;
  const size_t cells = (size_t)nx * ny, esz = dtype == VHP_F32 ? 4 : 8;
  const size_t pair_bytes = cells * esz;
  // chunks of 1 GB of fields (nothing is expanded here, so a chunk costs one event wait and two copies:
  // with 256 MB chunks those fixed costs were a third of the call)
  int64_t chunk = std::max<int64_t>(1, (int64_t)(((size_t)1 << 30) / pair_bytes));
  chunk = std::min(chunk, n);
  const int64_t nchunks = (n + chunk - 1) / chunk;
  const int64_t units_max = (int64_t)(((size_t)chunk * pair_bytes + kVhpPackUnit - 1) / kVhpPackUnit);
  const size_t meta_max = vhp_pack_meta_bytes(units_max, (int)esz), lit_max = (size_t)units_max * kVhpPackUnit;
  h->device = ctx->device; h->nx = nx; h->ny = ny; h->elem = (int)esz;
  h->npairs = n; h->chunk_pairs = chunk; h->pair_bytes = pair_bytes;
  h->chunks.assign((size_t)nchunks, vhp_packed::Chunk{});
  for (auto &b : h->blocks) b.used = 0;
  h->bytes_held = 0;
  vhp_status st;
  const int nsets = (int)std::min<int64_t>(NS, nchunks);
  for (int s = 0; s < nsets; ++s) {
    if ((st = ensure(ctx, ctx->b_pack_out[s], lit_max)) != VHP_OK) return st;
    if ((st = ensure(ctx, ctx->b_pack_meta[s], meta_max)) != VHP_OK) return st;
    if ((st = ensure(ctx, ctx->b_pack_lit[s], lit_max)) != VHP_OK) return st;
  }
  auto chunk_units = [&](int64_t it) {
    const int64_t np = std::min(chunk, n - it * chunk);
    return (int64_t)(((size_t)np * pair_bytes + kVhpPackUnit - 1) / kVhpPackUnit);
  };
  // chunk `it`: sweeps and packing on the compute stream, the copy of the meta block on the copy stream
  auto launch = [&](int64_t it) -> vhp_status {
    const int s = (int)(it % NS);
    const int64_t p0 = it * chunk, np = std::min(chunk, n - p0), nu = chunk_units(it);
    vhp_packed::Chunk &c = h->chunks[(size_t)it];
    c.nunits = nu; c.np = np;
    if (!h->take(vhp_pack_meta_bytes(nu, (int)esz), &c.meta_blk, &c.meta_off))
      return fail(ctx, VHP_ERR_CUDA, "vhp_visibility_batch_packed: out of pinned host memory");
    if (it >= NS) VHP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_pack_t0[s], 0)); // set s copied out
    vhp_status r = run_dev(ctx, Op::Sweep, (const uint8_t *)ctx->b_occ.p, nmaps, nx, ny, d_xy + 2 * p0,
                           d_map ? d_map + p0 : nullptr, np, dtype, ctx->b_pack_out[s].p);
    if (r != VHP_OK) return r;
    // (packing is an HBM-speed pass here -- nothing goes to host memory -- so it stays on the compute
    // stream and the copy stream carries copies only)
    VHP_CUDA(ctx, vhp_launch_pack_results(ctx->b_pack_out[s].p, nu, (int)esz, ctx->b_pack_meta[s].p,
                                          ctx->b_pack_lit[s].p, nullptr, 0, 0, ctx->sm_count, ctx->stream,
                                          &ctx->launches));
    VHP_CUDA(ctx, cudaEventRecord(ctx->ev_pack_lit[s], ctx->stream));
    VHP_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_pack_lit[s], 0));
    VHP_CUDA(ctx, cudaMemcpyAsync(h->blocks[c.meta_blk].p + c.meta_off, ctx->b_pack_meta[s].p,
                                  vhp_pack_meta_bytes(nu, (int)esz), cudaMemcpyDeviceToHost, ctx->copy_stream));
    VHP_CUDA(ctx, cudaEventRecord(ctx->ev_pack_meta[s], ctx->copy_stream));
    return VHP_OK;
  };
  // ... once its meta block has arrived the literal count is known: copy that many units
  auto finish = [&](int64_t it) -> vhp_status {
    const int s = (int)(it % NS);
    vhp_packed::Chunk &c = h->chunks[(size_t)it];
    VHP_CUDA(ctx, cudaEventSynchronize(ctx->ev_pack_meta[s]));
    c.nlit = *(const uint64_t *)(h->blocks[c.meta_blk].p + c.meta_off);
    const size_t meta_bytes = vhp_pack_meta_bytes(c.nunits, (int)esz), lit_bytes = (size_t)c.nlit * kVhpPackUnit;
    if (c.nlit) {
      if (!h->take(lit_bytes, &c.lit_blk, &c.lit_off))
        return fail(ctx, VHP_ERR_CUDA, "vhp_visibility_batch_packed: out of pinned host memory");
      VHP_CUDA(ctx, cudaMemcpyAsync(h->blocks[c.lit_blk].p + c.lit_off, ctx->b_pack_lit[s].p, lit_bytes,
                                    cudaMemcpyDeviceToHost, ctx->copy_stream));
    }
    VHP_CUDA(ctx, cudaEventRecord(ctx->ev_pack_t0[s], ctx->copy_stream)); // the set's device buffers are free
    ctx->last_d2h_bytes += (int64_t)(meta_bytes + lit_bytes);
    h->bytes_held += (int64_t)(meta_bytes + lit_bytes);
    return VHP_OK;
  };
  vhp_status result = VHP_OK;
  int64_t launched = 0, finished = 0;
  for (int64_t it = 0; it < nchunks && result == VHP_OK; ++it) {
    if ((result = launch(it)) != VHP_OK) break;
    ++launched;
    if (it >= 1) {
      if ((result = finish(it - 1)) != VHP_OK) break;
      ++finished;
    }
  }
  while (result == VHP_OK && finished < launched) {
    result = finish(finished);
    if (result == VHP_OK) ++finished;
  }
  cudaError_t e1 = cudaStreamSynchronize(ctx->copy_stream);
  cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
  if (e2 == cudaSuccess) e2 = e1;
  if (result != VHP_OK) return result;
  if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "sync stream");
  ctx->last_result_bytes = (int64_t)((size_t)n * pair_bytes);
  ctx->last_transport_packed = 1;
  return VHP_OK;
}

// host buffers: upload, run in chunks, deliver the results (packed or plain transport; windows: plain)
vhp_status run_host(vhp_context *ctx, Op op, const uint8_t *occ, int nmaps, int nx, int ny,
                    const int32_t *xy, const int32_t *maps, int64_t n, vhp_dtype dtype,
                    void *out, int radius = 0) {
  vhp_status st = check_common(ctx, occ, nmaps, nx, ny, xy, n, dtype, out);
  if (st != VHP_OK) return st;
  st = check_points(ctx, xy, 2, maps, n, nmaps, nx, ny,
                    op == Op::Sweep ? "vhp_visibility_batch"
                                    : (op == Op::Window ? "vhp_visibility_window_batch" : "vhp_raycast_batch"));
  if (st != VHP_OK) return st;
  ctx->last_d2h_bytes = ctx->last_result_bytes = 0;
  ctx->last_transport_packed = 0;
  if (n == 0) return VHP_OK;
  VHP_ON_DEVICE(ctx);
  PlanesGuard planes_guard(ctx);
  st = stage_host_batch(ctx, occ, nmaps, nx, ny, xy, 8, n, maps, op != Op::Raycast && sweeps_use_planes(ctx, nx, ny));
  if (st != VHP_OK) return st;
  const size_t cells = (size_t)nx * ny, esz = dtype == VHP_F32 ? 4 : 8;
  const int32_t *d_xy = (const int32_t *)ctx->b_src.p;
  const int32_t *d_map = maps ? (const int32_t *)ctx->b_map.p : nullptr;
  const size_t out_bytes = (size_t)n * (op == Op::Window ? window_pair_bytes(radius, dtype) : cells * esz);
  ctx->last_result_bytes = (int64_t)out_bytes;
  int64_t p_begin = 0;
  vhp_status result = VHP_OK;
  // small results are not worth the thread pool's wake-up
  if (op != Op::Window &&
      (ctx->result_transport == 2 || (ctx->result_transport == 1 && out_bytes >= ((size_t)64 << 20)))) {
    result = run_host_packed(ctx, op, nmaps, nx, ny, d_xy, d_map, n, dtype, out, &p_begin);
  }
  if (result == VHP_OK && p_begin < n)
    result = run_host_plain(ctx, op, nmaps, nx, ny, d_xy, d_map, n, p_begin, dtype, out, radius);
  if (result != VHP_OK) return result;
  return check_device_error(ctx);
}

// ---- thresholded binary visibility ------------------------------------------------------------
// Chunks of pairs: fp64 sweep into a device buffer, threshold_bits_kernel, and for host callers
// the D2H of chunk c (copy stream, two bit buffers) under the sweeps of chunk c + 1.

// Thresholded visibility of np pairs as bits (and, d_row_cnt != null, transition columns per row).
// Batches the one-CTA tile kernel takes are swept straight into bits (kFmtBits: the field itself is
// never stored); a non-positive threshold, a few pairs of a large map (grid mode) and the naive
// kernel go through the fp64 field in ctx->b_bin (at most bin_chunk_pairs pairs).
bool sweeps_into_bits(const vhp_context *ctx, int nx, int ny, int64_t np, double thr) {
  return ctx->bin_direct && thr > 0.0 && sweep_route(ctx, nx, ny, np) == SweepRoute::Tile;
}

vhp_status sweep_to_bits(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                         const int32_t *d_xy, const int32_t *d_map, int64_t np, double thr,
                         uint32_t *d_bits, uint16_t *d_row_cnt = nullptr) {
  if (sweeps_into_bits(ctx, nx, ny, np, thr)) {
    vhp_status st = ensure_rcp2(ctx, std::max(nx, ny) + 64);
    if (st != VHP_OK) return st;
    if ((st = pack_tile(ctx, d_occ, nmaps, nx, ny, false)) != VHP_OK) return st;
    VHP_CUDA(ctx, vhp_launch_sweep_tile(ctx->tile, nx, ny, d_xy, d_map, np, VHP_F32, d_bits, ctx->rcp2_table,
                                        ctx->d_err, ctx->stream, &ctx->launches, &thr, true));
    if (d_row_cnt)
      VHP_CUDA(ctx, vhp_launch_runs_row_count(d_bits, np * ny, nx, d_row_cnt, ctx->sm_count, ctx->stream,
                                              &ctx->launches));
    return VHP_OK;
  }
  vhp_status st = ensure(ctx, ctx->b_bin, (size_t)np * nx * ny * 8);
  if (st != VHP_OK) return st;
  if ((st = run_dev(ctx, Op::Sweep, d_occ, nmaps, nx, ny, d_xy, d_map, np, VHP_F64, ctx->b_bin.p)) != VHP_OK)
    return st;
  VHP_CUDA(ctx, vhp_launch_threshold_bits((const double *)ctx->b_bin.p, np * ny, nx, thr, d_bits,
                                          ctx->sm_count, ctx->stream, &ctx->launches, d_row_cnt));
  return VHP_OK;
}

vhp_status run_bin_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                       const int32_t *d_xy, const int32_t *d_map, int64_t n, double thr,
                       uint32_t *d_bits) {
  const size_t cells = (size_t)nx * ny, wpr = (size_t)(nx + 31) / 32;
  // no intermediate field when the sweep writes bits itself: one launch for the whole batch
  const int64_t chunk = sweeps_into_bits(ctx, nx, ny, n, thr) ? n : bin_chunk_pairs(cells, n);
  vhp_status st;
  for (int64_t p0 = 0; p0 < n; p0 += chunk) {
    const int64_t np = std::min(chunk, n - p0);
    st = sweep_to_bits(ctx, d_occ, nmaps, nx, ny, d_xy + 2 * p0, d_map ? d_map + p0 : nullptr, np, thr,
                       d_bits + (size_t)p0 * ny * wpr);
    if (st != VHP_OK) return st;
  }
  return VHP_OK;
}

vhp_status run_bin_host(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                        const int32_t *xy, const int32_t *maps, int64_t n, double thr,
                        uint32_t *out_bits) {
  vhp_status st = check_common(ctx, occ, nmaps, nx, ny, xy, n, VHP_F64, out_bits);
  if (st != VHP_OK) return st;
  if ((st = check_points(ctx, xy, 2, maps, n, nmaps, nx, ny, "vhp_visibility_batch_bin")) != VHP_OK) return st;
  ctx->last_d2h_bytes = ctx->last_result_bytes = 0;
  ctx->last_transport_packed = 0;
  if (n == 0) return VHP_OK;
  VHP_ON_DEVICE(ctx);
  PlanesGuard planes_guard(ctx);
  if ((st = stage_host_batch(ctx, occ, nmaps, nx, ny, xy, 8, n, maps, sweeps_use_planes(ctx, nx, ny))) != VHP_OK)
    return st;
  const size_t cells = (size_t)nx * ny, pair_bytes = (size_t)ny * ((nx + 31) / 32) * 4;
  const uint8_t *d_occ = (const uint8_t *)ctx->b_occ.p;
  const int32_t *d_xy = (const int32_t *)ctx->b_src.p;
  const int32_t *d_map = maps ? (const int32_t *)ctx->b_map.p : nullptr;
  // the sweep writes bits itself: four chunks (the D2H of one under the sweeps of the next), each
  // many waves of CTAs; else chunks bounded by the fp64 field
  const int64_t chunk = sweeps_into_bits(ctx, nx, ny, n, thr)
                            ? std::min<int64_t>(n, std::max<int64_t>((int64_t)ctx->sm_count * 6, (n + 3) / 4))
                            : bin_chunk_pairs(cells, n);
  auto produce = [&](int64_t p0, int64_t np, void *buf) {
    return sweep_to_bits(ctx, d_occ, nmaps, nx, ny, d_xy + 2 * p0, d_map ? d_map + p0 : nullptr, np, thr,
                         (uint32_t *)buf);
  };
  const vhp_status result = pipelined_d2h(ctx, 0, n, chunk, pair_bytes, out_bits, produce);
  ctx->last_result_bytes = (int64_t)((size_t)n * pair_bytes);
  if (result != VHP_OK) return result;
  return check_device_error(ctx);
}

// Row runs of the thresholded visibility (vhp_visibility_batch_runs): per chunk of pairs fp64 sweep,
// threshold bits, transitions per row / pair, exclusive scan, transition columns; the total of a
// chunk is read back (8 bytes) before its columns are written and copied.
vhp_status run_runs_host(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                         const int32_t *xy, const int32_t *maps, int64_t n, double thr,
                         uint16_t *row_count, uint64_t *pair_ptr, uint16_t *trans, int64_t trans_cap,
                         int64_t *trans_used) {
  vhp_status st = check_common(ctx, occ, nmaps, nx, ny, xy, n, VHP_F64, row_count);
  if (st != VHP_OK) return st;
  if (!pair_ptr || (!trans && trans_cap > 0) || trans_cap < 0)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_visibility_batch_runs: null buffer");
  if ((st = check_points(ctx, xy, 2, maps, n, nmaps, nx, ny, "vhp_visibility_batch_runs")) != VHP_OK) return st;
  ctx->last_d2h_bytes = ctx->last_result_bytes = 0;
  ctx->last_transport_packed = 0;
  if (trans_used) *trans_used = 0;
  pair_ptr[0] = 0;
  if (n == 0) return VHP_OK;
  VHP_ON_DEVICE(ctx);
  PlanesGuard planes_guard(ctx);
  if ((st = stage_host_batch(ctx, occ, nmaps, nx, ny, xy, 8, n, maps, sweeps_use_planes(ctx, nx, ny))) != VHP_OK)
    return st;
  const size_t cells = (size_t)nx * ny, wpr = (size_t)(nx + 31) / 32;
  const int32_t *d_xy = (const int32_t *)ctx->b_src.p;
  const int32_t *d_map = maps ? (const int32_t *)ctx->b_map.p : nullptr;
  // the sweep writes bits itself: a chunk is bounded by its bits (1 GB), not by an fp64 field
  const int64_t chunk = sweeps_into_bits(ctx, nx, ny, n, thr)
                            ? std::min<int64_t>(n, std::max<int64_t>(1, (int64_t)(((size_t)1 << 30) / ((size_t)ny * wpr * 4))))
                            : bin_chunk_pairs(cells, n);
  vhp_status result = ensure(ctx, ctx->b_out[0], (size_t)chunk * ny * wpr * 4);
  // small per-chunk arrays: row counts, row offsets, pair totals, pair offsets
  const size_t o_cnt = 0, o_off = ((size_t)chunk * ny * 2 + 255) & ~(size_t)255;
  const size_t o_tot = o_off + (((size_t)chunk * ny * 4 + 255) & ~(size_t)255);
  const size_t o_ptr = o_tot + (((size_t)chunk * 4 + 255) & ~(size_t)255);
  if (result == VHP_OK) result = ensure(ctx, ctx->b_misc, o_ptr + ((size_t)chunk + 1) * 8 + 256);
  unsigned long long total = 0;
  for (int64_t p0 = 0; p0 < n && result == VHP_OK; p0 += chunk) {
    const int64_t np = std::min(chunk, n - p0);
    char *misc = (char *)ctx->b_misc.p;
    uint16_t *d_cnt = (uint16_t *)(misc + o_cnt);
    uint32_t *d_off = (uint32_t *)(misc + o_off);
    uint32_t *d_tot = (uint32_t *)(misc + o_tot);
    result = sweep_to_bits(ctx, (const uint8_t *)ctx->b_occ.p, nmaps, nx, ny, d_xy + 2 * p0,
                           d_map ? d_map + p0 : nullptr, np, thr, (uint32_t *)ctx->b_out[0].p, d_cnt);
    if (result != VHP_OK) break;
    unsigned long long *d_ptr = (unsigned long long *)(misc + o_ptr);
    cudaError_t e = vhp_launch_runs_count(d_cnt, np, ny, d_off, d_tot, total, d_ptr, ctx->stream, &ctx->launches);
    unsigned long long new_total = 0;
    // the row counts and pair offsets are final here: they leave on the copy stream, under the write pass
    if (e == cudaSuccess) e = cudaEventRecord(ctx->ev_done[0], ctx->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_done[0], 0);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(row_count + (size_t)p0 * ny, d_cnt, (size_t)np * ny * 2, cudaMemcpyDeviceToHost, ctx->copy_stream);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(pair_ptr + p0, d_ptr, ((size_t)np + 1) * 8, cudaMemcpyDeviceToHost, ctx->copy_stream);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(&new_total, d_ptr + np, 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { result = cuda_fail(ctx, e, "row runs: count"); break; }
    if (trans_used) *trans_used = (int64_t)new_total;
    if ((int64_t)new_total > trans_cap) {
      result = fail(ctx, VHP_ERR_INVALID_ARG, "vhp_visibility_batch_runs: trans_cap too small (see *trans_used)");
      break;
    }
    const size_t chunk_elems = (size_t)(new_total - total);
    if ((result = ensure(ctx, ctx->b_out[1], std::max<size_t>(chunk_elems * 2, 256))) != VHP_OK) break;
    e = vhp_launch_runs_write((const uint32_t *)ctx->b_out[0].p, np, ny, nx, d_off, d_ptr, total,
                              (uint16_t *)ctx->b_out[1].p, ctx->sm_count, ctx->stream, &ctx->launches);
    if (e == cudaSuccess && chunk_elems)
      e = cudaMemcpyAsync(trans + total, ctx->b_out[1].p, chunk_elems * 2, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream); // the device buffers are reused by the next chunk
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->copy_stream);
    if (e != cudaSuccess) { result = cuda_fail(ctx, e, "row runs: write"); break; }
    ctx->last_d2h_bytes += (int64_t)(chunk_elems * 2 + (size_t)np * ny * 2 + ((size_t)np + 1) * 8 + 8);
    total = new_total;
  }
  (void)cudaStreamSynchronize(ctx->copy_stream); // (a failed chunk may have left its copies in flight)
  ctx->last_result_bytes = ctx->last_d2h_bytes;
  if (result != VHP_OK) return result;
  return check_device_error(ctx);
}

// ---- merged visibility of groups of sources (vhp_visibility_merge_batch) ----------------------------
// The outputs are filled on the stream, the per-pair table (group, index in the group, map) is built from the CSR
// layout, then either the sweeps fold straight into the outputs (kFmtMerge*: the one-CTA tile kernel takes the
// batch and thr > 0, so cells of value 0 never need a visit) or chunks of pairs are swept into the fp64 field in
// ctx->b_bin by any route of run_dev (grid mode, naive kernel, thr <= 0) and merge_fold_kernel folds them.
// With a range (vhp_visibility_merge_range_batch) the direct route sweeps only each source's box
// (kFmtMergeRange*, window_direct_route) and the fallback folds chunks of fp64 windows (run_window_dev, any of its
// routes) with merge_window_fold_kernel.  With views (vhp_visibility_merge_view_batch) both routes of the range form
// fold only each source's cells in its view (kFmtMergeView*, merge_window_fold_kernel<F32, true>).
const char *const kMergeViewName = "vhp_visibility_merge_view_batch";
const char *merge_name(const VhpMergeRange *range, bool view = false) {
  return view ? kMergeViewName : range ? "vhp_visibility_merge_range_batch" : "vhp_visibility_merge_batch";
}

vhp_status check_range(vhp_context *ctx, const std::string &what, const VhpMergeRange &range) {
  if (range.radius < 0 || range.radius > 16383)
    return fail(ctx, VHP_ERR_INVALID_ARG, what + ": radius outside [0, 16383]");
  if (range.shape != VHP_RANGE_BOX && range.shape != VHP_RANGE_DISK)
    return fail(ctx, VHP_ERR_INVALID_ARG, what + ": shape is neither VHP_RANGE_BOX nor VHP_RANGE_DISK");
  return VHP_OK;
}

vhp_status check_merge_args(vhp_context *ctx, const void *occ, int nmaps, int nx, int ny, const void *xy,
                            const void *group_ptr, int64_t ngroups, int64_t nsrc, double thr, int dtype,
                            const vhp_merge_out *out, const VhpMergeRange *range = nullptr, bool view = false) {
  const std::string what = merge_name(range, view);
  if (!ctx) return fail(nullptr, VHP_ERR_INVALID_ARG, "null context");
  if (!occ || !group_ptr || !out || (nsrc > 0 && !xy)) return fail(ctx, VHP_ERR_INVALID_ARG, "null buffer");
  if (nmaps < 1 || nx < 1 || ny < 1 || ngroups < 0 || nsrc < 0) return fail(ctx, VHP_ERR_INVALID_ARG, "bad sizes");
  if (ngroups > INT32_MAX) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": more than 2^31 - 1 groups");
  const vhp_status st = check_grid_dtype(ctx, nx, ny, dtype);
  if (st != VHP_OK) return st;
  if (thr != thr) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": threshold is NaN");
  if (!out->vmax && !out->first && !out->count)
    return fail(ctx, VHP_ERR_INVALID_ARG, what + ": no output requested");
  if (range) {
    const vhp_status sr = check_range(ctx, what, *range);
    if (sr != VHP_OK) return sr;
  }
  if (view && nsrc > 0 && !range->views) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": views is NULL");
  return VHP_OK;
}

// host-side validation of the views [n][5] = (r, ax, ay, bx, by), the rule of cover_view_kernel and MergeView; name / item: the
// call and what a view belongs to, for the message
vhp_status check_views_host(vhp_context *ctx, const int32_t *views, int64_t n, int radius, const char *name,
                            const char *item) {
  for (int64_t i = 0; i < n; ++i) {
    const int32_t *v = views + 5 * i;
    const char *bad = nullptr;
    if (v[0] < 0 || v[0] > radius) bad = "r outside [0, radius]";
    for (int j = 1; j < 5 && !bad; ++j)
      if (v[j] < -32767 || v[j] > 32767) bad = "a component outside [-32767, 32767]";
    if (!bad && ((v[1] == 0 && v[2] == 0) || (v[3] == 0 && v[4] == 0))) bad = "a or b is (0, 0)";
    if (bad)
      return fail(ctx, VHP_ERR_INVALID_ARG,
                  std::string(name) + ": view of " + item + " " + std::to_string(i) + ": " + bad);
  }
  return VHP_OK;
}

VhpMergeDev merge_dev_of(const vhp_merge_out &o, vhp_dtype dtype) {
  VhpMergeDev m;
  m.vmax = o.vmax;
  m.f32 = dtype == VHP_F32;
  m.first = o.first;
  m.count = o.count;
  return m;
}

vhp_status run_merge_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny, const int32_t *d_xy,
                         const int64_t *d_gptr, const int32_t *d_gmap, int64_t ngroups, int64_t nsrc, double thr,
                         VhpMergeDev m, const VhpMergeRange *range = nullptr) {
  const size_t cells = (size_t)nx * ny;
  VHP_CUDA(ctx, vhp_launch_merge_fill(m, (size_t)ngroups * cells, ctx->stream));
  if (ngroups == 0 && nsrc == 0) return VHP_OK;
  vhp_status st = ensure(ctx, ctx->b_merge, 12 * (size_t)std::max<int64_t>(nsrc, 1));
  if (st != VHP_OK) return st;
  int32_t *pg = (int32_t *)ctx->b_merge.p, *pk = pg + nsrc, *pm = pk + nsrc;
  VHP_CUDA(ctx, vhp_launch_merge_table(d_gptr, d_gmap, ngroups, nsrc, nmaps, pg, pk, pm, ctx->d_err, ctx->sm_count,
                                       ctx->stream, &ctx->launches));
  if (nsrc == 0) return VHP_OK;
  m.pair_group = pg;
  m.pair_k = pk;
  m.pair_map = pm;
  if (range) {
    const int R = range->radius;
    if (thr > 0.0 && window_direct_route(ctx, nx, ny, R) &&
        (!range->views || vhp_sweep_merge_view_supported(nx, ny, R))) {
      if ((st = ensure_rcp2(ctx, std::min(std::max(nx, ny), R + 1) + 64)) != VHP_OK) return st;
      if ((st = pack_tile(ctx, d_occ, nmaps, nx, ny, false)) != VHP_OK) return st;
      VHP_CUDA(ctx, vhp_launch_sweep_merge(ctx->tile, nx, ny, d_xy, m, nsrc, thr, ctx->rcp2_table, ctx->d_err,
                                           ctx->stream, &ctx->launches, range));
      return VHP_OK;
    }
    // fp64 windows of up to 1 GB of pairs at a time
    const size_t wbytes = window_pair_bytes(R, VHP_F64);
    const int64_t chunk = std::min<int64_t>(nsrc, std::max<int64_t>(1, (int64_t)(((size_t)1 << 30) / wbytes)));
    if ((st = ensure(ctx, ctx->b_mwin, (size_t)chunk * wbytes)) != VHP_OK) return st;
    for (int64_t p0 = 0; p0 < nsrc; p0 += chunk) {
      const int64_t np = std::min(chunk, nsrc - p0);
      if ((st = run_window_dev(ctx, d_occ, nmaps, nx, ny, d_xy + 2 * p0, pm + p0, np, R, VHP_F64, ctx->b_mwin.p)) !=
          VHP_OK)
        return st;
      VHP_CUDA(ctx, vhp_launch_merge_window_fold((const double *)ctx->b_mwin.p, p0, np, nx, ny, d_xy, thr, *range, m,
                                                 ctx->d_err, ctx->sm_count, ctx->stream, &ctx->launches));
    }
    return VHP_OK;
  }
  if (thr > 0.0 && sweep_route(ctx, nx, ny, nsrc) == SweepRoute::Tile) {
    if ((st = ensure_rcp2(ctx, std::max(nx, ny) + 64)) != VHP_OK) return st;
    if ((st = pack_tile(ctx, d_occ, nmaps, nx, ny, false)) != VHP_OK) return st;
    VHP_CUDA(ctx, vhp_launch_sweep_merge(ctx->tile, nx, ny, d_xy, m, nsrc, thr, ctx->rcp2_table, ctx->d_err,
                                         ctx->stream, &ctx->launches));
    return VHP_OK;
  }
  const int64_t chunk = bin_chunk_pairs(cells, nsrc);
  if ((st = ensure(ctx, ctx->b_bin, (size_t)chunk * cells * 8)) != VHP_OK) return st;
  for (int64_t p0 = 0; p0 < nsrc; p0 += chunk) {
    const int64_t np = std::min(chunk, nsrc - p0);
    if ((st = run_dev(ctx, Op::Sweep, d_occ, nmaps, nx, ny, d_xy + 2 * p0, pm + p0, np, VHP_F64, ctx->b_bin.p)) !=
        VHP_OK)
      return st;
    VHP_CUDA(ctx, vhp_launch_merge_fold((const double *)ctx->b_bin.p, p0, np, nx, ny, d_xy, thr, m, ctx->sm_count,
                                        ctx->stream, &ctx->launches));
  }
  return VHP_OK;
}

// host-side validation of a CSR group layout
vhp_status check_groups_host(vhp_context *ctx, const std::string &what, const int64_t *gptr, int64_t ngroups) {
  if (!ctx || !gptr || ngroups < 0) return VHP_OK; // (the argument checks report these)
  if (gptr[0] != 0) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": group_ptr[0] must be 0");
  for (int64_t g = 0; g < ngroups; ++g) {
    if (gptr[g + 1] < gptr[g])
      return fail(ctx, VHP_ERR_INVALID_ARG, what + ": group_ptr decreases at group " + std::to_string(g));
    if (gptr[g + 1] - gptr[g] >= ((int64_t)1 << 31))
      return fail(ctx, VHP_ERR_INVALID_ARG, what + ": group " + std::to_string(g) + " has 2^31 or more sources");
  }
  return VHP_OK;
}

// The host form of the group calls (merge and cover), after the call's argument checks: check the views (range->views,
// null but for the view calls), the sources and the group maps, upload maps, sources and views once, then runs of
// whole groups, as many as fit `budget` at per_src bytes per source plus per_group (at least one).  Each run's
// group_ptr, rebased, and its group maps go to b_misc / b_map, and run(g0, gc, d_xy, d_gptr, d_gmap, nsrc, range) runs
// the device form on groups [g0, g0 + gc) and copies their outputs (out_bytes per group) back with plain
// cudaMemcpyAsync, synchronised: h_ptr and the buffers are reused.  name / item: the call and what a source is called,
// for the messages.
template <class Run>
vhp_status run_groups_host(vhp_context *ctx, const char *name, const char *item, const uint8_t *occ, int nmaps,
                           int nx, int ny, const int32_t *xy, const int64_t *gptr, const int32_t *gmap,
                           int64_t ngroups, const VhpMergeRange *range, size_t per_src, size_t per_group,
                           size_t budget, size_t out_bytes, const char *upload_what, Run run) {
  const int64_t nsrc = gptr[ngroups];
  const int32_t *views = range ? range->views : nullptr;
  vhp_status st;
  if (views && (st = check_views_host(ctx, views, nsrc, range->radius, name, item)) != VHP_OK) return st;
  if ((st = check_points(ctx, xy, 2, nullptr, nsrc, nmaps, nx, ny, name)) != VHP_OK) return st;
  if (gmap && (st = check_points(ctx, nullptr, 0, gmap, ngroups, nmaps, nx, ny, name)) != VHP_OK) return st;
  ctx->last_d2h_bytes = ctx->last_result_bytes = 0;
  ctx->last_transport_packed = 0;
  if (ngroups == 0) return VHP_OK;
  VHP_ON_DEVICE(ctx);
  PlanesGuard planes_guard(ctx);
  // (the group maps are uploaded per run of groups below)
  if ((st = stage_host_batch(ctx, occ, nmaps, nx, ny, xy, 8, nsrc, nullptr, sweeps_use_planes(ctx, nx, ny))) != VHP_OK)
    return st;
  if (views && nsrc > 0) {
    if ((st = ensure(ctx, ctx->b_views, 20 * (size_t)nsrc)) != VHP_OK) return st;
    VHP_CUDA(ctx, cudaMemcpyAsync(ctx->b_views.p, views, 20 * (size_t)nsrc, cudaMemcpyHostToDevice, ctx->stream));
  }
  auto group_bytes = [&](int64_t g) { return (size_t)(gptr[g + 1] - gptr[g]) * per_src + per_group; };
  std::vector<int64_t> h_ptr;
  vhp_status result = VHP_OK;
  for (int64_t g0 = 0, gc = 0; g0 < ngroups && result == VHP_OK; g0 += gc) {
    size_t bytes = group_bytes(g0);
    for (gc = 1; g0 + gc < ngroups && bytes + group_bytes(g0 + gc) <= budget; ++gc) bytes += group_bytes(g0 + gc);
    const int64_t a = gptr[g0];
    h_ptr.resize((size_t)gc + 1);
    for (int64_t i = 0; i <= gc; ++i) h_ptr[(size_t)i] = gptr[g0 + i] - a;
    if ((result = ensure(ctx, ctx->b_misc, 8 * ((size_t)gc + 1))) != VHP_OK) break;
    if (gmap && (result = ensure(ctx, ctx->b_map, 4 * (size_t)gc)) != VHP_OK) break;
    cudaError_t e = cudaMemcpyAsync(ctx->b_misc.p, h_ptr.data(), 8 * ((size_t)gc + 1), cudaMemcpyHostToDevice,
                                    ctx->stream);
    if (e == cudaSuccess && gmap)
      e = cudaMemcpyAsync(ctx->b_map.p, gmap + g0, 4 * (size_t)gc, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) { result = cuda_fail(ctx, e, upload_what); break; }
    VhpMergeRange run_range;
    if (range) run_range = *range;
    if (views) run_range.views = (const int32_t *)ctx->b_views.p + 5 * a;
    result = run(g0, gc, (const int32_t *)ctx->b_src.p + 2 * a, (const int64_t *)ctx->b_misc.p,
                 gmap ? (const int32_t *)ctx->b_map.p : nullptr, gptr[g0 + gc] - a, range ? &run_range : nullptr);
    if (result == VHP_OK) ctx->last_d2h_bytes += (int64_t)((size_t)gc * out_bytes);
  }
  cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
  ctx->last_result_bytes = ctx->last_d2h_bytes;
  if (result != VHP_OK) return result;
  if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "sync stream");
  return check_device_error(ctx);
}

// host buffers: runs of whole groups whose outputs fit 1 GB of device memory (the merged result is already K times
// smaller than the fields it folds).  view: vhp_visibility_merge_view_batch, range->views [nsrc][5] on the host.
vhp_status run_merge_host(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny, const int32_t *xy,
                          const int64_t *gptr, const int32_t *gmap, int64_t ngroups, double thr, vhp_dtype dtype,
                          const vhp_merge_out *out, const VhpMergeRange *range = nullptr, bool view = false) {
  const char *what = merge_name(range, view);
  vhp_status st = check_groups_host(ctx, what, gptr, ngroups);
  if (st != VHP_OK) return st;
  const int64_t nsrc = (ctx && gptr && ngroups >= 0) ? gptr[ngroups] : 0;
  st = check_merge_args(ctx, occ, nmaps, nx, ny, xy, gptr, ngroups, nsrc, thr, dtype, out, range, view);
  if (st != VHP_OK) return st;
  const size_t cells = (size_t)nx * ny, esz = dtype == VHP_F32 ? 4 : 8;
  const size_t bv = out->vmax ? esz : 0, bf = out->first ? 4 : 0, bc = out->count ? 4 : 0;
  const size_t group_bytes = cells * (bv + bf + bc);
  auto run = [&](int64_t g0, int64_t gc, const int32_t *d_xy, const int64_t *d_gptr, const int32_t *d_gmap,
                 int64_t run_nsrc, const VhpMergeRange *run_range) {
    vhp_status r = ensure(ctx, ctx->b_out[0], (size_t)gc * group_bytes);
    if (r != VHP_OK) return r;
    char *base = (char *)ctx->b_out[0].p;
    VhpMergeDev m;
    m.f32 = dtype == VHP_F32;
    m.vmax = out->vmax ? base : nullptr;
    m.first = out->first ? (int32_t *)(base + (size_t)gc * cells * bv) : nullptr;
    m.count = out->count ? (uint32_t *)(base + (size_t)gc * cells * (bv + bf)) : nullptr;
    r = run_merge_dev(ctx, (const uint8_t *)ctx->b_occ.p, nmaps, nx, ny, d_xy, d_gptr, d_gmap, gc, run_nsrc, thr, m,
                      run_range);
    if (r != VHP_OK) return r;
    const size_t n = (size_t)gc * cells, off = (size_t)g0 * cells;
    cudaError_t e = cudaSuccess;
    if (out->vmax) e = cudaMemcpyAsync((char *)out->vmax + off * esz, m.vmax, n * esz, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out->first)
      e = cudaMemcpyAsync(out->first + off, m.first, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out->count)
      e = cudaMemcpyAsync(out->count + off, m.count, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    return e == cudaSuccess ? VHP_OK : cuda_fail(ctx, e, "merge: copy of the group outputs");
  };
  return run_groups_host(ctx, what, "source", occ, nmaps, nx, ny, xy, gptr, gmap, ngroups, range, 0, group_bytes,
                         (size_t)1 << 30, group_bytes, "merge: upload of the group layout", run);
}

// ---- greedy coverage placement (vhp_visibility_cover_greedy_batch) --------------------------------------
// Phase 1 stores every candidate's coverage bits over its box (VhpCoverBox): the direct route sweeps the boxes
// straight into bits (kFmtCoverBits: threshold > 0 and window_direct_route), the fallback folds chunks of fp64
// windows (run_window_dev, any of its routes) or, where a window would be larger than the map, of whole fields
// (run_dev) with cover_fold_kernel.  Phase 2 (kernels_cover.cu) runs min(k, nsrc) greedy rounds on the device.
// Every cover call is a CoverCall through check_cover_args and run_cover_dev (and run_cover_host): the weighted call
// (vhp_visibility_cover_greedy_weighted_batch) runs the same phase 1 and the weighted rounds, the m-fold call
// (vhp_visibility_cover_greedy_mfold_batch) the same phase 1 and the weighted rounds with counters, and the view call
// (vhp_visibility_cover_greedy_view_batch) the m-fold call with each candidate's bits masked by its view in between.
// The quota call (vhp_visibility_cover_quota_batch) is the view call, or the m-fold call without views, whose rounds
// loop on the device until each problem's gains reach its quota.  The budget call (vhp_visibility_cover_budget_batch)
// is the quota call with per-candidate costs and a budget per problem: its rounds pick by gain / cost among the
// candidates that still fit the budget, and the quota may be null.
const char *const kCoverName = "vhp_visibility_cover_greedy_batch";
const char *const kCoverWeightedName = "vhp_visibility_cover_greedy_weighted_batch";
const char *const kCoverMfoldName = "vhp_visibility_cover_greedy_mfold_batch";
const char *const kCoverViewName = "vhp_visibility_cover_greedy_view_batch";
const char *const kCoverQuotaName = "vhp_visibility_cover_quota_batch";
const char *const kCoverBudgetName = "vhp_visibility_cover_budget_batch";
// the weighted key keeps 28 bits for the index within the group (kernels_cover.cu)
constexpr int64_t kCoverWeightedMaxSrc = (int64_t)1 << 28;

// A cover call and its arguments.  weighted: uint64 gains and uint8 weights; mfold (with weighted): cells count until
// m picks cover them, `count` instead of `covered`; view (with mfold): range.views masks each candidate's bits; quota
// (with mfold, the quota call): a problem stops once the sum of its gains reaches its quota, k is kmax; budget (with
// mfold, the budget call): the picks go by gain / cost within each problem's budget, and quota may be null.
// extra: the target ([prob][ny][ceil(nx/32)] uint32) or the weights ([prob][ny][nx] uint8), may be null.
struct CoverCall {
  const char *name;
  bool weighted = false, mfold = false, view = false, budget = false;
  int32_t k, m = 1;
  VhpMergeRange range;
  double thr;
  const void *extra;
  const uint64_t *quota = nullptr;   // [prob]
  const uint32_t *cost = nullptr;    // [src], the budget call's
  const uint64_t *budgets = nullptr; // [prob], the budget call's
  CoverCall(const char *call, int32_t k_, int32_t radius, int32_t shape, double thr_, const void *extra_)
      : name(call), k(k_), range(radius, shape), thr(thr_), extra(extra_) {}
};

// a call's public outputs as VhpCoverOut; a null struct stays null (check_cover_args reports it).  Out: vhp_cover_out
// or vhp_cover_weighted_out
template <class Out>
const VhpCoverOut *cover_out(const Out *p, VhpCoverOut &o) {
  if (p) o = {p->pick, p->gain, p->npicked, p->covered, nullptr};
  return p ? &o : nullptr;
}
const VhpCoverOut *cover_out(const vhp_cover_mfold_out *p, VhpCoverOut &o) {
  if (p) o = {p->pick, p->gain, p->npicked, nullptr, p->count};
  return p ? &o : nullptr;
}
const VhpCoverOut *cover_out(const vhp_cover_quota_out *p, VhpCoverOut &o) {
  if (p) o = {p->pick, p->gain, p->npicked, nullptr, p->count, p->total};
  return p ? &o : nullptr;
}
const VhpCoverOut *cover_out(const vhp_cover_budget_out *p, VhpCoverOut &o) {
  if (p) o = {p->pick, p->gain, p->npicked, nullptr, p->count, p->total, p->spent, p->single, p->single_gain};
  return p ? &o : nullptr;
}

// The m-fold and view calls report these under the m-fold call's name, but for "views is NULL"; the quota and budget
// calls under their own names, with "kmax" for k.  The weighted key's
// limit on nsrc is checked before any candidate is read; the views' values by check_views_host, or by bit 3 of d_err
// on the device.
vhp_status check_cover_args(vhp_context *ctx, const CoverCall &c, const void *occ, int nmaps, int nx, int ny,
                            const void *xy, const void *group_ptr, int64_t nprob, int64_t nsrc,
                            const VhpCoverOut *out) {
  const bool quota = c.name == kCoverQuotaName || c.budget;
  const std::string what = c.mfold && !quota ? kCoverMfoldName : c.name;
  if (!ctx) return fail(nullptr, VHP_ERR_INVALID_ARG, "null context");
  if (!occ || !group_ptr || !out || (nsrc > 0 && !xy)) return fail(ctx, VHP_ERR_INVALID_ARG, "null buffer");
  if (nmaps < 1 || nx < 1 || ny < 1 || nprob < 0 || nsrc < 0) return fail(ctx, VHP_ERR_INVALID_ARG, "bad sizes");
  if (nprob > INT32_MAX) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": more than 2^31 - 1 problems");
  vhp_status st = check_grid_dtype(ctx, nx, ny, VHP_F64);
  if (st != VHP_OK) return st;
  if (c.thr != c.thr) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": threshold is NaN");
  if (c.k < 0) return fail(ctx, VHP_ERR_INVALID_ARG, what + (quota ? ": kmax < 0" : ": k < 0"));
  if (quota && !c.budget && nprob > 0 && !c.quota) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": quota is NULL");
  if (c.budget && nsrc > 0 && !c.cost) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": cost is NULL");
  if (c.budget && nprob > 0 && !c.budgets) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": budget is NULL");
  if (!out->pick && !out->gain && !out->npicked && !out->covered && !out->count && !out->total && !out->spent &&
      !out->single && !out->single_gain)
    return fail(ctx, VHP_ERR_INVALID_ARG, what + ": no output requested");
  if ((st = check_range(ctx, what, c.range)) != VHP_OK) return st;
  if (c.weighted && nsrc >= kCoverWeightedMaxSrc)
    return fail(ctx, VHP_ERR_INVALID_ARG, what + ": 2^28 or more candidates");
  if (c.mfold && (c.m < 1 || c.m > 255)) return fail(ctx, VHP_ERR_INVALID_ARG, what + ": m outside [1, 255]");
  if (c.view && nsrc > 0 && !c.range.views)
    return fail(ctx, VHP_ERR_INVALID_ARG, std::string(c.name) + ": views is NULL");
  return VHP_OK;
}

// a workspace buffer of the rounds; a failed allocation names its size
vhp_status ensure_cover(vhp_context *ctx, VhpDevBuf &b, size_t bytes, const char *what, const char *name) {
  if (ensure(ctx, b, bytes) == VHP_OK) return VHP_OK;
  (void)cudaGetLastError();
  return fail(ctx, VHP_ERR_CUDA, std::string(name) + ": " + what + " of " + std::to_string(bytes) +
                                     " bytes: " + ctx->last_error);
}

// what phase 1 leaves for the rounds
struct CoverBits {
  uint32_t *bits = nullptr;
  int32_t *pg = nullptr, *pk = nullptr; // candidate -> problem, index within it (vhp_launch_merge_table)
  int R = 0;                            // the geometry's radius
  int disk_r2 = -1;                     // >= 0: the direct route stored the whole box, the rounds apply the disk
};

// Phase 1 of the cover calls: the table, the workspace of the rounds (ws_bytes) and every candidate's coverage bits
vhp_status run_cover_phase1(vhp_context *ctx, const CoverCall &c, const uint8_t *d_occ, int nmaps, int nx, int ny,
                            const int32_t *d_xy, const int64_t *d_gptr, const int32_t *d_gmap, int64_t nprob,
                            int64_t nsrc, CoverBits &cb) {
  const int R = std::min(c.range.radius, std::max(nx, ny) - 1); // the geometry's radius: the same boxes
  const bool disk = c.range.shape == VHP_RANGE_DISK;
  const int r2 = c.range.radius * c.range.radius;
  const int64_t rounds = std::min<int64_t>(c.k, nsrc);
  cb.R = R;
  vhp_status st;
  if (nprob > 0 || nsrc > 0) {
    if ((st = ensure(ctx, ctx->b_merge, 12 * (size_t)std::max<int64_t>(nsrc, 1))) != VHP_OK) return st;
    cb.pg = (int32_t *)ctx->b_merge.p;
    cb.pk = cb.pg + nsrc;
    int32_t *pm = cb.pk + nsrc;
    VHP_CUDA(ctx, vhp_launch_merge_table(d_gptr, d_gmap, nprob, nsrc, nmaps, cb.pg, cb.pk, pm, ctx->d_err,
                                         ctx->sm_count, ctx->stream, &ctx->launches));
    if (rounds > 0 && nprob > 0) {
      const VhpCoverBox b = vhp_cover_box(nx, ny, R, 0, 0);
      if ((st = ensure_cover(ctx, ctx->b_cover, (size_t)nsrc * b.H * b.W * 4, "candidate coverage bits", c.name)) !=
          VHP_OK)
        return st;
      if ((st = ensure_cover(ctx, ctx->b_cover_ws,
                             vhp_cover_ws_bytes(nprob, nsrc, nx, ny, R, c.weighted, c.mfold, c.quota != nullptr,
                                                c.budget),
                             "workspace", c.name)) != VHP_OK)
        return st;
      uint32_t *bits = cb.bits = (uint32_t *)ctx->b_cover.p;
      if (c.thr > 0.0 && window_direct_route(ctx, nx, ny, R)) {
        if ((st = ensure_rcp2(ctx, std::min(std::max(nx, ny), R + 1) + 64)) != VHP_OK) return st;
        if ((st = pack_tile(ctx, d_occ, nmaps, nx, ny, false)) != VHP_OK) return st;
        VHP_CUDA(ctx, vhp_launch_sweep_cover(ctx->tile, nx, ny, d_xy, pm, nsrc, R, c.thr, bits, ctx->rcp2_table,
                                             ctx->d_err, ctx->stream, &ctx->launches));
        if (disk) cb.disk_r2 = r2;
      } else {
        // fp64 windows, or whole fields where a window would be larger than the map, up to 1 GB at a time
        const bool win = (2 * (size_t)R + 1) * (2 * (size_t)R + 1) <= (size_t)nx * ny;
        const size_t vbytes = win ? window_pair_bytes(R, VHP_F64) : (size_t)nx * ny * 8;
        const int64_t chunk = std::min<int64_t>(nsrc, std::max<int64_t>(1, (int64_t)(((size_t)1 << 30) / vbytes)));
        if ((st = ensure(ctx, ctx->b_mwin, (size_t)chunk * vbytes)) != VHP_OK) return st;
        for (int64_t p0 = 0; p0 < nsrc; p0 += chunk) {
          const int64_t np = std::min(chunk, nsrc - p0);
          st = win ? run_window_dev(ctx, d_occ, nmaps, nx, ny, d_xy + 2 * p0, pm + p0, np, R, VHP_F64, ctx->b_mwin.p)
                   : run_dev(ctx, Op::Sweep, d_occ, nmaps, nx, ny, d_xy + 2 * p0, pm + p0, np, VHP_F64, ctx->b_mwin.p);
          if (st != VHP_OK) return st;
          VHP_CUDA(ctx, vhp_launch_cover_fold((const double *)ctx->b_mwin.p, win ? R : -1, p0, np, nx, ny, R, disk, r2,
                                              d_xy, c.thr, bits, ctx->sm_count, ctx->stream, &ctx->launches));
        }
      }
    }
  }
  return VHP_OK;
}

// Phase 1, the view call's mask of the bits (range r_c in the call's shape, so the rounds apply no disk), then the
// rounds.  c.extra and c.range.views are on the device.
vhp_status run_cover_dev(vhp_context *ctx, const CoverCall &c, const uint8_t *d_occ, int nmaps, int nx, int ny,
                         const int32_t *d_xy, const int64_t *d_gptr, const int32_t *d_gmap, int64_t nprob,
                         int64_t nsrc, const VhpCoverOut &out) {
  CoverBits cb;
  const vhp_status st = run_cover_phase1(ctx, c, d_occ, nmaps, nx, ny, d_xy, d_gptr, d_gmap, nprob, nsrc, cb);
  if (st != VHP_OK) return st;
  if (c.view) {
    if (cb.bits)
      VHP_CUDA(ctx, vhp_launch_cover_view(cb.bits, nsrc, nx, ny, cb.R, c.range.radius, c.range.shape == VHP_RANGE_DISK,
                                          d_xy, c.range.views, ctx->d_err, ctx->sm_count, ctx->stream,
                                          &ctx->launches));
    cb.disk_r2 = -1;
  }
  const VhpCoverBudget bud{c.cost, c.budgets, ctx->d_err};
  VHP_CUDA(ctx, vhp_launch_cover_greedy(cb.bits, nsrc, nprob, nx, ny, cb.R, cb.disk_r2, d_xy, cb.pg, cb.pk, c.weighted,
                                        c.mfold, c.extra, c.k, c.m, c.quota, ctx->b_cover_ws.p, out, ctx->sm_count,
                                        ctx->stream, ctx->copy_stream, &ctx->launches, c.budget ? &bud : nullptr));
  return VHP_OK;
}

// the _dev entry point of every cover call
vhp_status cover_dev_entry(vhp_context *ctx, const CoverCall &c, const uint8_t *d_occ, int nmaps, int nx, int ny,
                           const int32_t *d_xy, const int64_t *d_gptr, const int32_t *d_gmap, int64_t nprob,
                           int64_t nsrc, const VhpCoverOut *out) {
  const vhp_status st = check_cover_args(ctx, c, d_occ, nmaps, nx, ny, d_xy, d_gptr, nprob, nsrc, out);
  if (st != VHP_OK) return st;
  VHP_ON_DEVICE(ctx);
  return run_cover_dev(ctx, c, d_occ, nmaps, nx, ny, d_xy, d_gptr, d_gmap, nprob, nsrc, *out);
}

// host buffers: runs of whole problems whose device memory (candidate bits, workspace, outputs) fits 4 GB, each with
// its slice of c.extra (and of c.quota, c.cost and c.budgets) uploaded.  c.range.views: the view call's [nsrc][5] on
// the host.  The budget call's costs are checked for zeros before any candidate is read.
vhp_status run_cover_host(vhp_context *ctx, const CoverCall &c, const uint8_t *occ, int nmaps, int nx, int ny,
                          const int32_t *xy, const int64_t *gptr, const int32_t *gmap, int64_t nprob,
                          const VhpCoverOut *out) {
  vhp_status st = check_groups_host(ctx, c.name, gptr, nprob);
  if (st != VHP_OK) return st;
  const int64_t nsrc = (ctx && gptr && nprob >= 0) ? gptr[nprob] : 0;
  if ((st = check_cover_args(ctx, c, occ, nmaps, nx, ny, xy, gptr, nprob, nsrc, out)) != VHP_OK) return st;
  for (int64_t i = 0; c.budget && i < nsrc; ++i)
    if (c.cost[i] == 0)
      return fail(ctx, VHP_ERR_INVALID_ARG, std::string(c.name) + ": the cost of candidate " + std::to_string(i) +
                                                " is 0");
  const size_t plane = (size_t)ny * ((nx + 31) / 32), gsz = c.weighted ? 8 : 4;
  const VhpCoverBox b = vhp_cover_box(nx, ny, std::min(c.range.radius, std::max(nx, ny) - 1), 0, 0);
  const size_t box = (size_t)b.H * b.W * 4;
  const size_t bp = out->pick ? 4 * (size_t)c.k : 0, bg = out->gain ? gsz * (size_t)c.k : 0;
  const size_t bn = out->npicked ? 4 : 0, bc = out->covered ? plane * 4 : out->count ? (size_t)ny * nx : 0;
  const size_t bt = c.extra ? (c.weighted ? (size_t)ny * nx : plane * 4) : 0;
  const size_t btot = out->total ? 8 : 0, bq = c.quota ? 8 : 0; // the quota call's total and quota
  // the budget call's spent, single_gain, budget and single outputs and inputs
  const size_t bsp = out->spent ? 8 : 0, bsg = out->single_gain ? 8 : 0, bb = c.budget ? 8 : 0,
               bs1 = out->single ? 4 : 0;
  // device bytes of problem q: its candidates' bits, table and gains, state, new, outputs, target or weights (and
  // the weighted rounds' 32-byte rows of weights, and the m-fold rounds' 32-byte rows of counters; views: 20 bytes;
  // the 64 bytes of per-problem scalars hold the quota rounds' total and quota copy too; the budget call's 4-byte
  // costs, and its ratio slot, remaining budget and spent cost, 32 bytes)
  const size_t per_src = box + 12 + gsz + (c.view ? 20 : 0) + (c.budget ? 4 : 0),
               per_prob = plane * 4 + box + bp + bg + bn + bc + bt + 64 + (c.weighted ? plane * 32 : 0) +
                          (c.mfold ? plane * 32 : 0) + btot + bq + bsp + bsg + bb + bs1 + (c.budget ? 32 : 0);
  void *const host_cells = out->covered ? (void *)out->covered : (void *)out->count;
  auto run = [&](int64_t q0, int64_t gc, const int32_t *d_xy, const int64_t *d_gptr, const int32_t *d_gmap,
                 int64_t run_nsrc, const VhpMergeRange *run_range) {
    vhp_status r;
    const size_t bytes = (size_t)gc * (bp + bg + btot + bq + bn + bc + bsp + bsg + bb + bs1) + 256;
    if ((r = ensure(ctx, ctx->b_out[0], bytes + (c.budget ? 4 * (size_t)run_nsrc : 0))) != VHP_OK) return r;
    if (c.extra && (r = ensure(ctx, ctx->b_out[1], (size_t)gc * bt)) != VHP_OK) return r;
    cudaError_t e = cudaSuccess;
    if (c.extra)
      e = cudaMemcpyAsync(ctx->b_out[1].p, (const char *)c.extra + (size_t)q0 * bt, (size_t)gc * bt,
                          cudaMemcpyHostToDevice, ctx->stream);
    char *base = (char *)ctx->b_out[0].p;
    const size_t o_gain = (gc * bp + gsz - 1) & ~(gsz - 1); // uint64 gains, totals and quotas: 8-byte aligned
    char *tot = base + o_gain + gc * bg, *spent = tot + gc * btot, *sgain = spent + gc * bsp;
    char *quota = sgain + gc * bsg, *budget = quota + gc * bq, *npk = budget + gc * bb, *single = npk + gc * bn;
    char *cells = single + gc * bs1;
    char *cost = base + ((size_t)(cells + gc * bc - base + 3) & ~(size_t)3); // 4-byte aligned, within the 256 spare
    if (e == cudaSuccess && c.quota)
      e = cudaMemcpyAsync(quota, c.quota + q0, gc * bq, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && c.budget)
      e = cudaMemcpyAsync(budget, c.budgets + q0, gc * bb, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && c.budget && run_nsrc > 0)
      e = cudaMemcpyAsync(cost, c.cost + gptr[q0], 4 * (size_t)run_nsrc, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "cover: upload of the problems");
    VhpCoverOut o;
    o.pick = out->pick ? (int32_t *)base : nullptr;
    o.gain = out->gain ? base + o_gain : nullptr;
    o.npicked = out->npicked ? (int32_t *)npk : nullptr;
    o.covered = out->covered ? (uint32_t *)cells : nullptr;
    o.count = out->count ? (uint8_t *)cells : nullptr;
    o.total = out->total ? (uint64_t *)tot : nullptr;
    o.spent = out->spent ? (uint64_t *)spent : nullptr;
    o.single = out->single ? (int32_t *)single : nullptr;
    o.single_gain = out->single_gain ? (uint64_t *)sgain : nullptr;
    CoverCall rc = c;
    rc.range = *run_range;
    rc.extra = c.extra ? ctx->b_out[1].p : nullptr;
    rc.quota = c.quota ? (const uint64_t *)quota : nullptr;
    rc.budgets = c.budget ? (const uint64_t *)budget : nullptr;
    rc.cost = c.budget ? (const uint32_t *)cost : nullptr;
    r = run_cover_dev(ctx, rc, (const uint8_t *)ctx->b_occ.p, nmaps, nx, ny, d_xy, d_gptr, d_gmap, gc, run_nsrc, o);
    if (r != VHP_OK) return r;
    if (out->pick) e = cudaMemcpyAsync(out->pick + q0 * c.k, o.pick, gc * bp, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out->gain)
      e = cudaMemcpyAsync((char *)out->gain + q0 * bg, o.gain, gc * bg, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out->npicked)
      e = cudaMemcpyAsync(out->npicked + q0, o.npicked, gc * bn, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && host_cells)
      e = cudaMemcpyAsync((char *)host_cells + q0 * bc, cells, gc * bc, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out->total)
      e = cudaMemcpyAsync(out->total + q0, o.total, gc * btot, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out->spent)
      e = cudaMemcpyAsync(out->spent + q0, o.spent, gc * bsp, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out->single)
      e = cudaMemcpyAsync(out->single + q0, o.single, gc * bs1, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out->single_gain)
      e = cudaMemcpyAsync(out->single_gain + q0, o.single_gain, gc * bsg, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    return e == cudaSuccess ? VHP_OK : cuda_fail(ctx, e, "cover: copy of the outputs");
  };
  return run_groups_host(ctx, c.name, "candidate", occ, nmaps, nx, ny, xy, gptr, gmap, nprob, &c.range, per_src,
                         per_prob, (size_t)4 << 30, bp + bg + bn + bc + btot + bsp + bs1 + bsg,
                         "cover: upload of the problems", run);
}

// ---- opt-in sweep variants ------------------------------------------------------------------------
vhp_status check_variant(vhp_context *ctx, const vhp_sweep_variant *v) {
  if (!v) return fail(ctx, VHP_ERR_INVALID_ARG, "sweep variant: null descriptor");
  if (v->model != VHP_VARIANT_MATLAB && v->model != VHP_VARIANT_QUEUE)
    return fail(ctx, VHP_ERR_INVALID_ARG, "sweep variant: model is VHP_VARIANT_MATLAB or VHP_VARIANT_QUEUE");
  if (v->model == VHP_VARIANT_MATLAB && !(v->fac > 0.0))
    return fail(ctx, VHP_ERR_INVALID_ARG, "sweep variant: fac must be positive");
  return VHP_OK;
}

vhp_status run_variant_dev(vhp_context *ctx, const uint8_t *d_occ, int nx, int ny, const int32_t *d_xy,
                           const int32_t *d_map, int64_t n, const vhp_sweep_variant &v, vhp_dtype dtype,
                           void *d_out) {
  const size_t cells = (size_t)nx * ny;
  const int64_t chunk = dtype == VHP_F64 ? n : bin_chunk_pairs(cells, n);
  vhp_status st;
  if (dtype == VHP_F32 && (st = ensure(ctx, ctx->b_bin, (size_t)chunk * cells * 8)) != VHP_OK) return st;
  for (int64_t p0 = 0; p0 < n; p0 += chunk) {
    const int64_t np = std::min(chunk, n - p0);
    double *buf = dtype == VHP_F64 ? (double *)d_out + (size_t)p0 * cells : (double *)ctx->b_bin.p;
    float *o32 = dtype == VHP_F32 ? (float *)d_out + (size_t)p0 * cells : nullptr;
    VHP_CUDA(ctx, vhp_launch_sweep_variant(d_occ, nx, ny, d_xy + 2 * p0, d_map ? d_map + p0 : nullptr, np,
                                           v.model, v.alpha, v.fac, v.light_strength, v.cutoff, buf, o32,
                                           ctx->d_err, ctx->stream, &ctx->launches));
  }
  return VHP_OK;
}

// ---- planner ------------------------------------------------------------------
// One LARGE problem on the whole GPU: solve() (src/visibilityBasedSolver.cpp:76-160) as the
// one-strip case of the strip engine (giant.cu).  Per iteration: grid-mode sweep of the whole
// map (many CTAs, the +y and -y quadrants as two concurrent launches), per-cell epilogue +
// arg-min, next-source selection -- all with the loop state on the device, captured as the
// body of a CUDA-graph WHILE node: no host round trip between the first sweep and the path.
// Same results as the persistent single-CTA planner kernel, which would leave all but one SM
// idle.
vhp_status planner_grid_one(vhp_context *ctx, const VhpTilePlanes &pl, int nx, int ny,
                            const int32_t se[4], double thr, int32_t max_iter, int32_t ls_cap,
                            double *vis, double *vg, double *hc, int32_t *came, int32_t *status,
                            int32_t *nb, int32_t *ls, double *plen, int32_t *pn, int32_t *path,
                            float *vg32, float *vis32) {
  vhp_status st = vhp_i_grid_planner_run(ctx, pl, nx, ny, se, thr, max_iter, ls_cap, vis, vg, hc, came, ls);
  if (st != VHP_OK) return st;
  VHP_CUDA(ctx, vhp_launch_grid_planner_finish(vhp_i_grid_planner_ctl(ctx), nx, ny, se[2], se[3], ls_cap,
                                               ls, came, vis, vg, status, nb, plen, pn, path, vg32,
                                               vis32, ctx->stream, &ctx->launches));
  return VHP_OK;
}

// device pointers in `o` (any may be null).  Fields the caller did not ask for in
// fp64 live in the context workspace, so large batches run in chunks.
vhp_status planner_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                       const int32_t *d_se, const int32_t *d_pmap, int64_t nprob, double thr,
                       int32_t max_iter, int32_t ls_cap, vhp_dtype dtype, const vhp_planner_out &o) {
  if (nprob == 0) return VHP_OK;
  // maps too wide for the persistent single-CTA kernel still run on the grid route
  const bool cta_ok = vhp_planner_supported(nx, ny);
  if (!cta_ok && !grid_mode_available(ctx, nx, ny))
    return fail(ctx, VHP_ERR_UNSUPPORTED, "planner: grid too large for the single-CTA kernel");
  if (ls_cap < max_iter + 2 || max_iter < 0)
    return fail(ctx, VHP_ERR_INVALID_ARG, "planner: ls_cap must be >= max_iter + 2");
  vhp_status st = ensure_rcp2(ctx, std::max(nx, ny) + 64);
  if (st != VHP_OK) return st;
  if ((st = pack_tile(ctx, d_occ, nmaps, nx, ny, false)) != VHP_OK) return st;
  const size_t cells = (size_t)nx * ny;
  const bool vis_user = dtype == VHP_F64 && o.vis, vg_user = dtype == VHP_F64 && o.vg;
  const size_t per_prob = (vis_user ? 0 : 8 * cells) + (vg_user ? 0 : 8 * cells) +
                          (o.came ? 0 : 4 * cells) + 8 * cells; // + the cached heuristic field
  const size_t small_pp = 4 + 4 + 8 + 4 + 2 * (size_t)ls_cap * 8 + 32;
  int64_t chunk = nprob;
  const size_t ws_limit = (size_t)32 << 30; // (of 180 GB: fewer chunks, fewer kernel tails)
  if (per_prob) chunk = std::max<int64_t>(1, std::min<int64_t>(nprob, (int64_t)(ws_limit / per_prob)));
  const size_t field_bytes = (size_t)chunk * per_prob;
  const size_t small_bytes = (size_t)nprob * small_pp;
  if ((st = ensure(ctx, ctx->b_planner, field_bytes + small_bytes + 256)) != VHP_OK) return st;
  char *w = (char *)ctx->b_planner.p;
  auto take = [&](size_t bytes) { char *r = w; w += (bytes + 15) & ~(size_t)15; return r; };
  double *ws_vis = vis_user ? nullptr : (double *)take(8 * cells * chunk);
  double *ws_vg = vg_user ? nullptr : (double *)take(8 * cells * chunk);
  double *ws_hc = (double *)take(8 * cells * chunk);
  int32_t *ws_came = o.came ? nullptr : (int32_t *)take(4 * cells * chunk);
  int32_t *status = o.status ? o.status : (int32_t *)take(4 * nprob);
  int32_t *nb = o.nb_sources ? o.nb_sources : (int32_t *)take(4 * nprob);
  int32_t *ls = o.light_sources ? o.light_sources : (int32_t *)take(8 * (size_t)ls_cap * nprob);
  double *plen = o.path_len ? o.path_len : (double *)take(8 * nprob);
  int32_t *pn = o.path_n ? o.path_n : (int32_t *)take(4 * nprob);
  int32_t *path = o.path ? o.path : (int32_t *)take(8 * (size_t)ls_cap * nprob);
  // A few problems on a large map: one problem at a time on the whole GPU (grid mode) instead
  // of one persistent CTA per problem.  grid_sweep 0: never, 1: by size, 2: always.
  // Measured on B200 (tools/planner_routes.py, ms per iteration): single CTA 0.6 @256^2, 3.3 @1000^2,
  // 48 @4096^2, 184 @8192^2; grid route 0.3, 0.7, 2.8, 7.5 -- but its problems run one after the
  // other, so it only wins for a handful of problems, more of them the larger the map.
  const int64_t grid_max_prob = std::max<int64_t>(1, std::min<int64_t>(24, (int64_t)(cells / 100000)));
  const bool grid_route = !cta_ok || ctx->grid_sweep == 2 ||
                          (ctx->grid_sweep == 1 && nprob <= grid_max_prob && vhp_sweep_grid_supported(nx, ny));
  std::vector<int32_t> h_se, h_pmap;
  if (grid_route) {
    h_se.resize(4 * (size_t)nprob);
    VHP_CUDA(ctx, cudaMemcpyAsync(h_se.data(), d_se, h_se.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (d_pmap) {
      h_pmap.resize((size_t)nprob);
      VHP_CUDA(ctx, cudaMemcpyAsync(h_pmap.data(), d_pmap, h_pmap.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    VHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int64_t k = 0; k < nprob; ++k)
      if (d_pmap && (h_pmap[k] < 0 || h_pmap[k] >= nmaps))
        return fail(ctx, VHP_ERR_INVALID_ARG, "planner: map index out of range");
  }
  for (int64_t q0 = 0; q0 < nprob; q0 += chunk) {
    const int64_t n = std::min(chunk, nprob - q0);
    double *vis = vis_user ? (double *)o.vis + q0 * cells : ws_vis;
    double *vg = vg_user ? (double *)o.vg + q0 * cells : ws_vg;
    int32_t *came = o.came ? o.came + q0 * cells : ws_came;
    float *vg32 = (dtype == VHP_F32 && o.vg) ? (float *)o.vg + q0 * cells : nullptr;
    float *vis32 = (dtype == VHP_F32 && o.vis) ? (float *)o.vis + q0 * cells : nullptr;
    if (grid_route) {
      for (int64_t k = 0; k < n; ++k) {
        const int64_t q = q0 + k;
        const VhpTilePlanes pl = planes_of_map(ctx, d_pmap ? (size_t)h_pmap[q] : 0, nx, ny);
        st = planner_grid_one(ctx, pl, nx, ny, &h_se[4 * q], thr, max_iter, ls_cap, vis + k * cells,
                              vg + k * cells, ws_hc + k * cells, came + k * cells, status + q, nb + q,
                              ls + 2 * (size_t)ls_cap * q, plen + q, pn + q,
                              path + 2 * (size_t)ls_cap * q, vg32 ? vg32 + k * cells : nullptr,
                              vis32 ? vis32 + k * cells : nullptr);
        if (st != VHP_OK) return st;
      }
      continue;
    }
    void *first_ws = nullptr;
    if (ctx->planner_first == 2 || (ctx->planner_first == 1 && n >= (int64_t)8 * ctx->sm_count)) {
      if ((st = ensure(ctx, ctx->b_misc, vhp_planner_first_ws_bytes(n))) != VHP_OK) return st;
      first_ws = ctx->b_misc.p;
    }
    VHP_CUDA(ctx, vhp_launch_planner(ctx->tile, nx, ny, d_se + 4 * q0, d_pmap ? d_pmap + q0 : nullptr,
                                     n, thr, max_iter, ls_cap, ctx->rcp2_table, vis, vg, ws_hc, came,
                                     status + q0, nb + q0, ls + 2 * (size_t)ls_cap * q0, plen + q0,
                                     pn + q0, path + 2 * (size_t)ls_cap * q0, vg32, vis32,
                                     ctx->d_err, ctx->stream, &ctx->launches, first_ws, ctx->planner_first_rounds));
  }
  return VHP_OK;
}

} // namespace

vhp_status vhp_i_fail(vhp_context *ctx, vhp_status st, const std::string &msg) { return fail(ctx, st, msg); }
vhp_status vhp_i_ensure_rcp2(vhp_context *ctx, int len) { return ensure_rcp2(ctx, len); }
int vhp_i_grid_ctas(const vhp_context *ctx, int nx, int ny, int rows) {
  if (!vhp_sweep_tile_supported(nx, ny) ||
      (grid_mode_available(ctx, nx, ny) && (int64_t)nx * rows >= (ctx->grid_sweep > 1 ? 0 : (1 << 20))))
    return grid_sweep_ctas(ctx, rows);
  return 1;
}

extern "C" {

int vhp_abi_version(void) { return VHP_ABI_VERSION; }

const char *vhp_version_string(void) {
  return "vhp_b200 0.1 (sm_100a; visibility sweep / planner / ray casting)";
}

int vhp_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return n;
}

const char *vhp_last_error(const vhp_context *ctx) {
  return ctx ? ctx->last_error.c_str() : g_last_error.c_str();
}

int64_t vhp_launch_count(const vhp_context *ctx) { return ctx ? ctx->launches : 0; }

vhp_status vhp_context_create(int device, void *cuda_stream, vhp_context **out) {
  if (!out) return fail(nullptr, VHP_ERR_INVALID_ARG, "null out pointer");
  *out = nullptr;
  const int n = vhp_device_count();
  if (n == 0) return fail(nullptr, VHP_ERR_NO_DEVICE, "no CUDA device available (no CPU fallback)");
  if (device < 0 || device >= n) return fail(nullptr, VHP_ERR_INVALID_ARG, "bad device index");
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return cuda_fail(nullptr, e, "cudaGetDeviceProperties");
  if (prop.major != 10)
    return fail(nullptr, VHP_ERR_NO_DEVICE,
                "device is not sm_100 (this library ships sm_100a code only)");
#define CTX_TRY(call)                                      \
  do {                                                     \
    cudaError_t e_ = (call);                               \
    if (e_ != cudaSuccess) {                               \
      vhp_context_destroy(ctx);                            \
      return cuda_fail(nullptr, e_, #call);                \
    }                                                      \
  } while (0)
  vhp_context *ctx = new vhp_context();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  DeviceGuard device_guard_(device);
  CTX_TRY(device_guard_.err);
  if (cuda_stream) {
    ctx->stream = (cudaStream_t)cuda_stream;
  } else {
    CTX_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->owns_stream = true;
  }
  CTX_TRY(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    CTX_TRY(cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming));
    CTX_TRY(cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming));
  }
  CTX_TRY(cudaMalloc(&ctx->d_err, sizeof(int)));
  CTX_TRY(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
  const char *impl = std::getenv("VHP_SWEEP_IMPL");
  ctx->sweep_impl = 0;
  if (impl && std::strcmp(impl, "naive") == 0) ctx->sweep_impl = 1;
  if (const char *e = std::getenv("VHP_GRID_SWEEP")) ctx->grid_sweep = std::atoi(e);
  if (const char *e = std::getenv("VHP_PLANNER_FIRST")) ctx->planner_first = std::atoi(e);
  if (const char *e = std::getenv("VHP_BIN_DIRECT")) ctx->bin_direct = std::atoi(e) != 0;
  if (const char *e = std::getenv("VHP_PLANNER_ROUNDS")) ctx->planner_first_rounds = std::max(1, std::atoi(e));
  for (int i = 0; i < vhp_context::kPackSets; ++i) {
    CTX_TRY(cudaEventCreate(&ctx->ev_pack_meta[i]));
    CTX_TRY(cudaEventCreate(&ctx->ev_pack_t0[i]));
    CTX_TRY(cudaEventCreateWithFlags(&ctx->ev_pack_lit[i], cudaEventDisableTiming));
  }
  if (const char *e = std::getenv("VHP_RESULT_TRANSPORT")) {
    if (std::strcmp(e, "plain") == 0) ctx->result_transport = 0;
    else if (std::strcmp(e, "packed") == 0) ctx->result_transport = 2;
  }
  if (const char *e = std::getenv("VHP_RESULT_DIRECT")) ctx->result_direct = std::atoi(e) != 0;
  if (const char *e = std::getenv("VHP_RESULT_GPU_SHARE")) ctx->result_gpu_share = std::atoi(e);
  ctx->transport_trace = std::getenv("VHP_TRANSPORT_TRACE") != nullptr;
#undef CTX_TRY
  *out = ctx;
  return VHP_OK;
}

void vhp_context_destroy(vhp_context *ctx) {
  if (!ctx) return;
  DeviceGuard device_guard_(ctx->device);
  vhp_i_grid_planner_release(ctx);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
  VhpDevBuf *bufs[] = {&ctx->b_occ, &ctx->b_src, &ctx->b_map, &ctx->b_out[0], &ctx->b_out[1],
                       &ctx->b_scratch, &ctx->b_planner, &ctx->b_misc, &ctx->b_grid, &ctx->b_bin,
                       &ctx->b_merge, &ctx->b_mwin, &ctx->b_cover, &ctx->b_cover_ws, &ctx->b_views};
  for (VhpDevBuf *b : bufs)
    if (b->p) cudaFree(b->p);
  delete ctx->expand_pool;
  for (int i = 0; i < vhp_context::kPackSets; ++i) {
    if (ctx->b_pack_out[i].p) cudaFree(ctx->b_pack_out[i].p);
    if (ctx->b_pack_meta[i].p) cudaFree(ctx->b_pack_meta[i].p);
    if (ctx->b_pack_lit[i].p) cudaFree(ctx->b_pack_lit[i].p);
    if (ctx->h_pack_meta[i]) cudaFreeHost(ctx->h_pack_meta[i]);
    if (ctx->h_pack_lit[i]) cudaFreeHost(ctx->h_pack_lit[i]);
    if (ctx->ev_pack_meta[i]) cudaEventDestroy(ctx->ev_pack_meta[i]);
    if (ctx->ev_pack_t0[i]) cudaEventDestroy(ctx->ev_pack_t0[i]);
    if (ctx->ev_pack_lit[i]) cudaEventDestroy(ctx->ev_pack_lit[i]);
  }
  if (ctx->tile_buf) cudaFree(ctx->tile_buf);
  if (ctx->rcp2_table) cudaFree(ctx->rcp2_table);
  if (ctx->d_err) cudaFree(ctx->d_err);
  for (int i = 0; i < 2; ++i) {
    if (ctx->ev_done[i]) cudaEventDestroy(ctx->ev_done[i]);
    if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
  }
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->owns_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  (void)cudaGetLastError();
  delete ctx;
}

vhp_status vhp_context_synchronize(vhp_context *ctx) {
  if (!ctx) return fail(nullptr, VHP_ERR_INVALID_ARG, "null context");
  VHP_ON_DEVICE(ctx);
  return check_device_error(ctx);
}

int vhp_context_device(const vhp_context *ctx) { return ctx ? ctx->device : -1; }

vhp_status vhp_prepare_maps_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                int ny) {
  if (!ctx || !d_occ || nmaps < 1 || nx < 1 || ny < 1)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_prepare_maps_dev: bad argument");
  VHP_ON_DEVICE(ctx);
  if (!vhp_sweep_tile_supported(nx, ny) && !vhp_sweep_grid_supported(nx, ny))
    return VHP_OK; // the naive kernel reads the byte maps
  const vhp_status st = pack_tile(ctx, d_occ, nmaps, nx, ny, true);
  if (st == VHP_OK) ctx->planes_sticky = true;
  return st;
}

vhp_status vhp_release_maps_dev(vhp_context *ctx) {
  if (!ctx) return fail(nullptr, VHP_ERR_INVALID_ARG, "null context");
  ctx->planes_sticky = false;
  ctx->tile_src = nullptr;
  return VHP_OK;
}

vhp_status vhp_visibility_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                    int ny, const int32_t *d_src_xy, const int32_t *d_src_map,
                                    int64_t npairs, vhp_dtype dtype, void *d_out) {
  vhp_status st = check_common(ctx, d_occ, nmaps, nx, ny, d_src_xy, npairs, dtype, d_out);
  if (st != VHP_OK) return st;
  VHP_ON_DEVICE(ctx);
  return run_dev(ctx, Op::Sweep, d_occ, nmaps, nx, ny, d_src_xy, d_src_map, npairs, dtype, d_out);
}

vhp_status vhp_visibility_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                const int32_t *src_xy, const int32_t *src_map, int64_t npairs,
                                vhp_dtype dtype, void *out) {
  return run_host(ctx, Op::Sweep, occ, nmaps, nx, ny, src_xy, src_map, npairs, dtype, out);
}

vhp_status vhp_visibility_window_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                       const int32_t *src_xy, const int32_t *src_map, int64_t npairs,
                                       int32_t radius, vhp_dtype dtype, void *out) {
  if (ctx && (radius < 0 || radius > 16383))
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_visibility_window_batch: radius outside [0, 16383]");
  return run_host(ctx, Op::Window, occ, nmaps, nx, ny, src_xy, src_map, npairs, dtype, out, radius);
}

vhp_status vhp_visibility_window_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                           const int32_t *d_src_xy, const int32_t *d_src_map, int64_t npairs,
                                           int32_t radius, vhp_dtype dtype, void *d_out) {
  vhp_status st = check_common(ctx, d_occ, nmaps, nx, ny, d_src_xy, npairs, dtype, d_out);
  if (st != VHP_OK) return st;
  if (radius < 0 || radius > 16383)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_visibility_window_batch_dev: radius outside [0, 16383]");
  VHP_ON_DEVICE(ctx);
  return run_window_dev(ctx, d_occ, nmaps, nx, ny, d_src_xy, d_src_map, npairs, radius, dtype, d_out);
}

vhp_status vhp_visibility_batch_packed(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                       const int32_t *src_xy, const int32_t *src_map, int64_t npairs,
                                       vhp_dtype dtype, vhp_packed **handle) {
  if (!handle) return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_visibility_batch_packed: null handle pointer");
  vhp_status st = check_common(ctx, occ, nmaps, nx, ny, src_xy, npairs, dtype, handle);
  if (st != VHP_OK) return st;
  if ((st = check_points(ctx, src_xy, 2, src_map, npairs, nmaps, nx, ny, "vhp_visibility_batch_packed")) != VHP_OK)
    return st;
  ctx->last_d2h_bytes = ctx->last_result_bytes = 0;
  ctx->last_transport_packed = 0;
  VHP_ON_DEVICE(ctx);
  vhp_packed *h = *handle;
  const bool fresh = h == nullptr;
  if (fresh) {
    h = new (std::nothrow) vhp_packed();
    if (!h) return fail(ctx, VHP_ERR_CUDA, "vhp_visibility_batch_packed: out of memory");
  } else if (h->device != ctx->device && !h->blocks.empty()) {
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_visibility_batch_packed: the handle belongs to another device");
  }
  h->device = ctx->device;
  h->npairs = 0;
  h->chunks.clear();
  auto run = [&]() -> vhp_status {
    if (npairs == 0) return VHP_OK;
    PlanesGuard planes_guard(ctx);
    vhp_status r = stage_host_batch(ctx, occ, nmaps, nx, ny, src_xy, 8, npairs, src_map, sweeps_use_planes(ctx, nx, ny));
    if (r != VHP_OK) return r;
    r = run_host_to_packed(ctx, nmaps, nx, ny, (const int32_t *)ctx->b_src.p,
                           src_map ? (const int32_t *)ctx->b_map.p : nullptr, npairs, dtype, h);
    if (r != VHP_OK) return r;
    return check_device_error(ctx);
  };
  st = run();
  if (st != VHP_OK) {
    h->npairs = 0;
    h->chunks.clear();
    if (fresh) vhp_packed_destroy(h);
    return st;
  }
  *handle = h;
  return VHP_OK;
}

int64_t vhp_packed_pairs(const vhp_packed *h) { return h ? h->npairs : 0; }
int64_t vhp_packed_bytes(const vhp_packed *h) { return h ? h->bytes_held : 0; }
int64_t vhp_packed_pair_bytes(const vhp_packed *h) { return h ? (int64_t)h->pair_bytes : 0; }

vhp_status vhp_packed_expand(const vhp_packed *h, int64_t first_pair, int64_t npairs, void *out, int nthreads) {
  if (!h || first_pair < 0 || npairs < 0 || first_pair + npairs > h->npairs || (npairs > 0 && !out))
    return vhp_i_fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_packed_expand: null handle / buffer or pairs out of range");
  if (npairs == 0) return VHP_OK;
  const size_t b_begin = (size_t)first_pair * h->pair_bytes, b_end = (size_t)(first_pair + npairs) * h->pair_bytes;
  const size_t chunk_bytes = (size_t)h->chunk_pairs * h->pair_bytes;
  // slices of about equal size, cut at 128-byte units of the batch's first chunk (any cut is valid)
  const size_t total = b_end - b_begin;
  int nt = nthreads > 0 ? nthreads : (int)std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()),
                                                           (total + ((size_t)64 << 20) - 1) / ((size_t)64 << 20));
  nt = std::max(1, std::min(nt, 64));
  auto work = [&](size_t lo, size_t hi) { // bytes [lo, hi) of the whole batch
    while (lo < hi) {
      const size_t ci = lo / chunk_bytes, c0 = ci * chunk_bytes;
      const size_t upto = std::min(hi, c0 + chunk_bytes);
      vhp_expand_bytes(h->view(h->chunks[ci]), lo - c0, upto - c0, (char *)out + (lo - b_begin));
      lo = upto;
    }
  };
  if (nt == 1) {
    work(b_begin, b_end);
    return VHP_OK;
  }
  const size_t per = ((total / nt) + 127) & ~(size_t)127;
  std::vector<std::thread> th;
  try {
    for (int t = 0; t < nt; ++t) {
      const size_t lo = b_begin + std::min(total, (size_t)t * per), hi = t == nt - 1 ? b_end : b_begin + std::min(total, (size_t)(t + 1) * per);
      if (lo < hi) th.emplace_back(work, lo, hi);
    }
  } catch (...) { // no more threads to be had: the caller's thread does the rest
    const size_t done = th.size();
    for (auto &t : th) t.join();
    work(b_begin + std::min(total, done * per), b_end);
    return VHP_OK;
  }
  for (auto &t : th) t.join();
  return VHP_OK;
}

void vhp_packed_destroy(vhp_packed *h) {
  if (!h) return;
  int cur = 0;
  const bool have = cudaGetDevice(&cur) == cudaSuccess;
  if (!h->blocks.empty()) cudaSetDevice(h->device);
  for (auto &b : h->blocks) cudaFreeHost(b.p);
  if (have) cudaSetDevice(cur);
  (void)cudaGetLastError();
  delete h;
}

vhp_status vhp_visibility_variant_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                            int ny, const int32_t *d_src_xy, const int32_t *d_src_map,
                                            int64_t npairs, const vhp_sweep_variant *variant,
                                            vhp_dtype dtype, void *d_out) {
  vhp_status st = check_common(ctx, d_occ, nmaps, nx, ny, d_src_xy, npairs, dtype, d_out);
  if (st != VHP_OK) return st;
  if ((st = check_variant(ctx, variant)) != VHP_OK) return st;
  VHP_ON_DEVICE(ctx);
  if (npairs == 0) return VHP_OK;
  return run_variant_dev(ctx, d_occ, nx, ny, d_src_xy, d_src_map, npairs, *variant, dtype, d_out);
}

vhp_status vhp_visibility_variant_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                        const int32_t *src_xy, const int32_t *src_map, int64_t npairs,
                                        const vhp_sweep_variant *variant, vhp_dtype dtype, void *out) {
  vhp_status st = check_common(ctx, occ, nmaps, nx, ny, src_xy, npairs, dtype, out);
  if (st != VHP_OK) return st;
  if ((st = check_variant(ctx, variant)) != VHP_OK) return st;
  if ((st = check_points(ctx, src_xy, 2, src_map, npairs, nmaps, nx, ny, "vhp_visibility_variant_batch")) != VHP_OK)
    return st;
  if (npairs == 0) return VHP_OK;
  VHP_ON_DEVICE(ctx);
  PlanesGuard planes_guard(ctx);
  if ((st = stage_host_batch(ctx, occ, nmaps, nx, ny, src_xy, 8, npairs, src_map, false)) != VHP_OK) return st;
  const size_t cells = (size_t)nx * ny, esz = dtype == VHP_F32 ? 4 : 8;
  // results leave in chunks of at most 1 GB through one device buffer
  const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(npairs, (int64_t)(((size_t)1 << 30) / (cells * esz))));
  if ((st = ensure(ctx, ctx->b_out[0], (size_t)chunk * cells * esz)) != VHP_OK) return st;
  for (int64_t p0 = 0; p0 < npairs; p0 += chunk) {
    const int64_t np = std::min(chunk, npairs - p0);
    st = run_variant_dev(ctx, (const uint8_t *)ctx->b_occ.p, nx, ny, (const int32_t *)ctx->b_src.p + 2 * p0,
                         src_map ? (const int32_t *)ctx->b_map.p + p0 : nullptr, np, *variant, dtype,
                         ctx->b_out[0].p);
    if (st != VHP_OK) return st;
    VHP_CUDA(ctx, cudaMemcpyAsync((char *)out + (size_t)p0 * cells * esz, ctx->b_out[0].p, (size_t)np * cells * esz,
                                  cudaMemcpyDeviceToHost, ctx->stream));
    VHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return check_device_error(ctx);
}

vhp_status vhp_visibility_batch_bin(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                    const int32_t *src_xy, const int32_t *src_map, int64_t npairs,
                                    double threshold, uint32_t *out_bits) {
  return run_bin_host(ctx, occ, nmaps, nx, ny, src_xy, src_map, npairs, threshold, out_bits);
}

vhp_status vhp_visibility_batch_runs(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                     const int32_t *src_xy, const int32_t *src_map, int64_t npairs,
                                     double threshold, uint16_t *row_count, uint64_t *pair_ptr,
                                     uint16_t *trans, int64_t trans_cap, int64_t *trans_used) {
  return run_runs_host(ctx, occ, nmaps, nx, ny, src_xy, src_map, npairs, threshold, row_count, pair_ptr, trans,
                       trans_cap, trans_used);
}

vhp_status vhp_runs_to_bits(const uint16_t *row_count, const uint64_t *pair_ptr, const uint16_t *trans,
                            int64_t npairs, int nx, int ny, uint32_t *out_bits) {
  if (!row_count || !pair_ptr || !out_bits || npairs < 0 || nx < 1 || ny < 1)
    return fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_runs_to_bits: bad argument");
  const size_t wpr = (size_t)(nx + 31) / 32;
  std::memset(out_bits, 0, (size_t)npairs * ny * wpr * 4);
  for (int64_t p = 0; p < npairs; ++p) {
    const uint16_t *t = trans + pair_ptr[p];
    for (int y = 0; y < ny; ++y) {
      const int c = row_count[(size_t)p * ny + y];
      uint32_t *row = out_bits + ((size_t)p * ny + y) * wpr;
      for (int k = 0; k + 1 < c; k += 2)
        for (int x = t[k]; x < t[k + 1] && x < nx; ++x) row[x >> 5] |= 1u << (x & 31);
      t += c;
    }
  }
  return VHP_OK;
}

vhp_status vhp_visibility_batch_bin_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                        int ny, const int32_t *d_src_xy, const int32_t *d_src_map,
                                        int64_t npairs, double threshold, uint32_t *d_out_bits) {
  vhp_status st = check_common(ctx, d_occ, nmaps, nx, ny, d_src_xy, npairs, VHP_F64, d_out_bits);
  if (st != VHP_OK) return st;
  VHP_ON_DEVICE(ctx);
  return run_bin_dev(ctx, d_occ, nmaps, nx, ny, d_src_xy, d_src_map, npairs, threshold, d_out_bits);
}

vhp_status vhp_visibility_merge_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                      const int32_t *src_xy, const int64_t *group_ptr, const int32_t *group_map,
                                      int64_t ngroups, double threshold, vhp_dtype dtype, const vhp_merge_out *out) {
  return run_merge_host(ctx, occ, nmaps, nx, ny, src_xy, group_ptr, group_map, ngroups, threshold, dtype, out);
}

vhp_status vhp_visibility_merge_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                          const int32_t *d_src_xy, const int64_t *d_group_ptr,
                                          const int32_t *d_group_map, int64_t ngroups, int64_t nsrc,
                                          double threshold, vhp_dtype dtype, const vhp_merge_out *d_out) {
  vhp_status st = check_merge_args(ctx, d_occ, nmaps, nx, ny, d_src_xy, d_group_ptr, ngroups, nsrc, threshold, dtype,
                                   d_out);
  if (st != VHP_OK) return st;
  VHP_ON_DEVICE(ctx);
  return run_merge_dev(ctx, d_occ, nmaps, nx, ny, d_src_xy, d_group_ptr, d_group_map, ngroups, nsrc, threshold,
                       merge_dev_of(*d_out, dtype));
}

vhp_status vhp_visibility_merge_range_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                            const int32_t *src_xy, const int64_t *group_ptr,
                                            const int32_t *group_map, int64_t ngroups, int32_t radius,
                                            int32_t shape, double threshold, vhp_dtype dtype,
                                            const vhp_merge_out *out) {
  const VhpMergeRange range(radius, shape);
  return run_merge_host(ctx, occ, nmaps, nx, ny, src_xy, group_ptr, group_map, ngroups, threshold, dtype, out,
                        &range);
}

vhp_status vhp_visibility_merge_range_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                                int ny, const int32_t *d_src_xy, const int64_t *d_group_ptr,
                                                const int32_t *d_group_map, int64_t ngroups, int64_t nsrc,
                                                int32_t radius, int32_t shape, double threshold,
                                                vhp_dtype dtype, const vhp_merge_out *d_out) {
  const VhpMergeRange range(radius, shape);
  vhp_status st = check_merge_args(ctx, d_occ, nmaps, nx, ny, d_src_xy, d_group_ptr, ngroups, nsrc, threshold, dtype,
                                   d_out, &range);
  if (st != VHP_OK) return st;
  VHP_ON_DEVICE(ctx);
  return run_merge_dev(ctx, d_occ, nmaps, nx, ny, d_src_xy, d_group_ptr, d_group_map, ngroups, nsrc, threshold,
                       merge_dev_of(*d_out, dtype), &range);
}

vhp_status vhp_visibility_merge_view_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                           const int32_t *src_xy, const int32_t *views, const int64_t *group_ptr,
                                           const int32_t *group_map, int64_t ngroups, int32_t radius, int32_t shape,
                                           double threshold, vhp_dtype dtype, const vhp_merge_out *out) {
  const VhpMergeRange range(radius, shape, views);
  return run_merge_host(ctx, occ, nmaps, nx, ny, src_xy, group_ptr, group_map, ngroups, threshold, dtype, out,
                        &range, true);
}

vhp_status vhp_visibility_merge_view_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                               const int32_t *d_src_xy, const int32_t *d_views,
                                               const int64_t *d_group_ptr, const int32_t *d_group_map,
                                               int64_t ngroups, int64_t nsrc, int32_t radius, int32_t shape,
                                               double threshold, vhp_dtype dtype, const vhp_merge_out *d_out) {
  const VhpMergeRange range(radius, shape, d_views);
  vhp_status st = check_merge_args(ctx, d_occ, nmaps, nx, ny, d_src_xy, d_group_ptr, ngroups, nsrc, threshold, dtype,
                                   d_out, &range, true);
  if (st != VHP_OK) return st;
  VHP_ON_DEVICE(ctx);
  return run_merge_dev(ctx, d_occ, nmaps, nx, ny, d_src_xy, d_group_ptr, d_group_map, ngroups, nsrc, threshold,
                       merge_dev_of(*d_out, dtype), &range);
}

vhp_status vhp_visibility_cover_greedy_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                             const int32_t *cand_xy, const int64_t *group_ptr,
                                             const int32_t *group_map, int64_t nprob, int32_t k, int32_t radius,
                                             int32_t shape, double threshold, const uint32_t *target,
                                             const vhp_cover_out *out) {
  const CoverCall c(kCoverName, k, radius, shape, threshold, target);
  VhpCoverOut o;
  return run_cover_host(ctx, c, occ, nmaps, nx, ny, cand_xy, group_ptr, group_map, nprob, cover_out(out, o));
}

vhp_status vhp_visibility_cover_greedy_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                                 const int32_t *d_cand_xy, const int64_t *d_group_ptr,
                                                 const int32_t *d_group_map, int64_t nprob, int64_t nsrc, int32_t k,
                                                 int32_t radius, int32_t shape, double threshold,
                                                 const uint32_t *d_target, const vhp_cover_out *d_out) {
  const CoverCall c(kCoverName, k, radius, shape, threshold, d_target);
  VhpCoverOut o;
  return cover_dev_entry(ctx, c, d_occ, nmaps, nx, ny, d_cand_xy, d_group_ptr, d_group_map, nprob, nsrc,
                         cover_out(d_out, o));
}

vhp_status vhp_visibility_cover_greedy_weighted_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                                      const int32_t *cand_xy, const int64_t *group_ptr,
                                                      const int32_t *group_map, int64_t nprob, int32_t k,
                                                      int32_t radius, int32_t shape, double threshold,
                                                      const uint8_t *weights, const vhp_cover_weighted_out *out) {
  CoverCall c(kCoverWeightedName, k, radius, shape, threshold, weights);
  c.weighted = true;
  VhpCoverOut o;
  return run_cover_host(ctx, c, occ, nmaps, nx, ny, cand_xy, group_ptr, group_map, nprob, cover_out(out, o));
}

vhp_status vhp_visibility_cover_greedy_weighted_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                                          int ny, const int32_t *d_cand_xy,
                                                          const int64_t *d_group_ptr, const int32_t *d_group_map,
                                                          int64_t nprob, int64_t nsrc, int32_t k, int32_t radius,
                                                          int32_t shape, double threshold, const uint8_t *d_weights,
                                                          const vhp_cover_weighted_out *d_out) {
  CoverCall c(kCoverWeightedName, k, radius, shape, threshold, d_weights);
  c.weighted = true;
  VhpCoverOut o;
  return cover_dev_entry(ctx, c, d_occ, nmaps, nx, ny, d_cand_xy, d_group_ptr, d_group_map, nprob, nsrc,
                         cover_out(d_out, o));
}

vhp_status vhp_visibility_cover_greedy_mfold_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                                   const int32_t *cand_xy, const int64_t *group_ptr,
                                                   const int32_t *group_map, int64_t nprob, int32_t k, int32_t radius,
                                                   int32_t shape, double threshold, const uint8_t *weights, int32_t m,
                                                   const vhp_cover_mfold_out *out) {
  CoverCall c(kCoverMfoldName, k, radius, shape, threshold, weights);
  c.weighted = c.mfold = true;
  c.m = m;
  VhpCoverOut o;
  return run_cover_host(ctx, c, occ, nmaps, nx, ny, cand_xy, group_ptr, group_map, nprob, cover_out(out, o));
}

vhp_status vhp_visibility_cover_greedy_mfold_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                                       int ny, const int32_t *d_cand_xy, const int64_t *d_group_ptr,
                                                       const int32_t *d_group_map, int64_t nprob, int64_t nsrc,
                                                       int32_t k, int32_t radius, int32_t shape, double threshold,
                                                       const uint8_t *d_weights, int32_t m,
                                                       const vhp_cover_mfold_out *d_out) {
  CoverCall c(kCoverMfoldName, k, radius, shape, threshold, d_weights);
  c.weighted = c.mfold = true;
  c.m = m;
  VhpCoverOut o;
  return cover_dev_entry(ctx, c, d_occ, nmaps, nx, ny, d_cand_xy, d_group_ptr, d_group_map, nprob, nsrc,
                         cover_out(d_out, o));
}

vhp_status vhp_visibility_cover_greedy_view_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                                  const int32_t *cand_xy, const int32_t *views,
                                                  const int64_t *group_ptr, const int32_t *group_map, int64_t nprob,
                                                  int32_t k, int32_t radius, int32_t shape, double threshold,
                                                  const uint8_t *weights, int32_t m, const vhp_cover_mfold_out *out) {
  CoverCall c(kCoverViewName, k, radius, shape, threshold, weights);
  c.weighted = c.mfold = c.view = true;
  c.m = m;
  c.range.views = views;
  VhpCoverOut o;
  return run_cover_host(ctx, c, occ, nmaps, nx, ny, cand_xy, group_ptr, group_map, nprob, cover_out(out, o));
}

vhp_status vhp_visibility_cover_greedy_view_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                                      int ny, const int32_t *d_cand_xy, const int32_t *d_views,
                                                      const int64_t *d_group_ptr, const int32_t *d_group_map,
                                                      int64_t nprob, int64_t nsrc, int32_t k, int32_t radius,
                                                      int32_t shape, double threshold, const uint8_t *d_weights,
                                                      int32_t m, const vhp_cover_mfold_out *d_out) {
  CoverCall c(kCoverViewName, k, radius, shape, threshold, d_weights);
  c.weighted = c.mfold = c.view = true;
  c.m = m;
  c.range.views = d_views;
  VhpCoverOut o;
  return cover_dev_entry(ctx, c, d_occ, nmaps, nx, ny, d_cand_xy, d_group_ptr, d_group_map, nprob, nsrc,
                         cover_out(d_out, o));
}

vhp_status vhp_visibility_cover_quota_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                            const int32_t *cand_xy, const int32_t *views, const int64_t *group_ptr,
                                            const int32_t *group_map, int64_t nprob, int32_t kmax, int32_t radius,
                                            int32_t shape, double threshold, const uint8_t *weights, int32_t m,
                                            const uint64_t *quota, const vhp_cover_quota_out *out) {
  CoverCall c(kCoverQuotaName, kmax, radius, shape, threshold, weights);
  c.weighted = c.mfold = true;
  c.view = views != nullptr;
  c.m = m;
  c.range.views = views;
  c.quota = quota;
  VhpCoverOut o;
  return run_cover_host(ctx, c, occ, nmaps, nx, ny, cand_xy, group_ptr, group_map, nprob, cover_out(out, o));
}

vhp_status vhp_visibility_cover_quota_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                                const int32_t *d_cand_xy, const int32_t *d_views,
                                                const int64_t *d_group_ptr, const int32_t *d_group_map, int64_t nprob,
                                                int64_t nsrc, int32_t kmax, int32_t radius, int32_t shape,
                                                double threshold, const uint8_t *d_weights, int32_t m,
                                                const uint64_t *d_quota, const vhp_cover_quota_out *d_out) {
  CoverCall c(kCoverQuotaName, kmax, radius, shape, threshold, d_weights);
  c.weighted = c.mfold = true;
  c.view = d_views != nullptr;
  c.m = m;
  c.range.views = d_views;
  c.quota = d_quota;
  VhpCoverOut o;
  return cover_dev_entry(ctx, c, d_occ, nmaps, nx, ny, d_cand_xy, d_group_ptr, d_group_map, nprob, nsrc,
                         cover_out(d_out, o));
}

vhp_status vhp_visibility_cover_budget_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                             const int32_t *cand_xy, const int32_t *views, const int64_t *group_ptr,
                                             const int32_t *group_map, int64_t nprob, int32_t kmax, int32_t radius,
                                             int32_t shape, double threshold, const uint8_t *weights, int32_t m,
                                             const uint64_t *quota, const uint32_t *cost, const uint64_t *budget,
                                             const vhp_cover_budget_out *out) {
  CoverCall c(kCoverBudgetName, kmax, radius, shape, threshold, weights);
  c.weighted = c.mfold = c.budget = true;
  c.view = views != nullptr;
  c.m = m;
  c.range.views = views;
  c.quota = quota;
  c.cost = cost;
  c.budgets = budget;
  VhpCoverOut o;
  return run_cover_host(ctx, c, occ, nmaps, nx, ny, cand_xy, group_ptr, group_map, nprob, cover_out(out, o));
}

vhp_status vhp_visibility_cover_budget_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                                 const int32_t *d_cand_xy, const int32_t *d_views,
                                                 const int64_t *d_group_ptr, const int32_t *d_group_map, int64_t nprob,
                                                 int64_t nsrc, int32_t kmax, int32_t radius, int32_t shape,
                                                 double threshold, const uint8_t *d_weights, int32_t m,
                                                 const uint64_t *d_quota, const uint32_t *d_cost,
                                                 const uint64_t *d_budget, const vhp_cover_budget_out *d_out) {
  CoverCall c(kCoverBudgetName, kmax, radius, shape, threshold, d_weights);
  c.weighted = c.mfold = c.budget = true;
  c.view = d_views != nullptr;
  c.m = m;
  c.range.views = d_views;
  c.quota = d_quota;
  c.cost = d_cost;
  c.budgets = d_budget;
  VhpCoverOut o;
  return cover_dev_entry(ctx, c, d_occ, nmaps, nx, ny, d_cand_xy, d_group_ptr, d_group_map, nprob, nsrc,
                         cover_out(d_out, o));
}

vhp_status vhp_raycast_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                 int ny, const int32_t *d_src_xy, const int32_t *d_src_map,
                                 int64_t npairs, vhp_dtype dtype, void *d_out) {
  vhp_status st = check_common(ctx, d_occ, nmaps, nx, ny, d_src_xy, npairs, dtype, d_out);
  if (st != VHP_OK) return st;
  VHP_ON_DEVICE(ctx);
  return run_dev(ctx, Op::Raycast, d_occ, nmaps, nx, ny, d_src_xy, d_src_map, npairs, dtype,
                 d_out);
}

vhp_status vhp_raycast_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                             const int32_t *src_xy, const int32_t *src_map, int64_t npairs,
                             vhp_dtype dtype, void *out) {
  return run_host(ctx, Op::Raycast, occ, nmaps, nx, ny, src_xy, src_map, npairs, dtype, out);
}

vhp_status vhp_selftest_ratio(vhp_context *ctx, int kmax, int64_t *mismatches) {
  if (!ctx || !mismatches || kmax < 1 || kmax > 16384)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_selftest_ratio: bad argument");
  VHP_ON_DEVICE(ctx);
  vhp_status st = ensure_rcp2(ctx, kmax + 8);
  if (st != VHP_OK) return st;
  if ((st = ensure(ctx, ctx->b_misc, 64)) != VHP_OK) return st;
  VHP_CUDA(ctx, cudaMemsetAsync(ctx->b_misc.p, 0, 8, ctx->stream));
  VHP_CUDA(ctx, vhp_launch_ratio2_selftest(ctx->rcp2_table, kmax,
                                           (unsigned long long *)ctx->b_misc.p, ctx->stream,
                                           &ctx->launches));
  unsigned long long bad = 0;
  VHP_CUDA(ctx, cudaMemcpyAsync(&bad, ctx->b_misc.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
  VHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *mismatches = (int64_t)bad;
  return VHP_OK;
}

uint32_t vhp_environment_draw(uint64_t seed, uint64_t map, uint64_t obstacle, uint32_t d) {
  return vhp_env_draw(seed, map, obstacle, d);
}

vhp_status vhp_environment_generate_batch_dev(vhp_context *ctx, const vhp_config *cfg,
                                              uint64_t seed, int64_t first_map, int nmaps,
                                              uint8_t *d_occ) {
  if (!ctx || !cfg || !d_occ || nmaps < 1 || first_map < 0)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_environment_generate_batch_dev: bad argument");
  if (cfg->ncols < 1 || cfg->nrows < 1 || cfg->ncols > 16384 || cfg->nrows > 16384 ||
      cfg->nb_of_obstacles < 0 || cfg->nb_of_obstacles > 0x7fffffff || cfg->min_width < 0 ||
      cfg->min_height < 0 || cfg->max_width < cfg->min_width || cfg->max_height < cfg->min_height)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_environment_generate_batch_dev: bad environment settings");
  VHP_ON_DEVICE(ctx);
  VHP_CUDA(ctx, vhp_launch_env_generate(d_occ, nmaps, (int)cfg->ncols, (int)cfg->nrows, first_map,
                                        seed, cfg->nb_of_obstacles, cfg->min_width, cfg->max_width,
                                        cfg->min_height, cfg->max_height, ctx->stream,
                                        &ctx->launches));
  if (ctx->tile_src == d_occ) { // bit planes of an older content of this buffer
    ctx->planes_sticky = false;
    ctx->tile_src = nullptr;
  }
  return VHP_OK;
}

vhp_status vhp_context_set_result_transport(vhp_context *ctx, int mode) {
  if (!ctx || mode < 0 || mode > 2)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_context_set_result_transport: mode is 0, 1 or 2");
  ctx->result_transport = mode;
  return VHP_OK;
}

vhp_status vhp_context_set_result_gpu_share(vhp_context *ctx, int sixteenths) {
  if (!ctx || sixteenths < 0 || sixteenths > 16)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_context_set_result_gpu_share: 0..16");
  ctx->result_gpu_share = sixteenths;
  return VHP_OK;
}

vhp_status vhp_context_last_transport(const vhp_context *ctx, int64_t *d2h_bytes,
                                      int64_t *result_bytes, int32_t *packed) {
  if (!ctx) return fail(nullptr, VHP_ERR_INVALID_ARG, "null context");
  if (d2h_bytes) *d2h_bytes = ctx->last_d2h_bytes;
  if (result_bytes) *result_bytes = ctx->last_result_bytes;
  if (packed) *packed = ctx->last_transport_packed;
  return VHP_OK;
}

vhp_status vhp_expand_packed_chunk(const uint32_t *mask, const uint32_t *word_base,
                                   const uint32_t *vmask, int elem_bytes, const void *literals,
                                   int64_t nunits, int64_t valid_bytes, void *dst, int threads) {
  if (elem_bytes != 4 && elem_bytes != 8)
    return fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_expand_packed_chunk: elem_bytes is 4 or 8");
  if (nunits < 0 || valid_bytes < 0 || valid_bytes > nunits * (int64_t)kVhpPackUnit ||
      valid_bytes <= (nunits - 1) * (int64_t)kVhpPackUnit)
    return fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_expand_packed_chunk: nunits does not match valid_bytes");
  if (nunits == 0) return VHP_OK;
  if (!mask || !word_base || !vmask || !dst)
    return fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_expand_packed_chunk: null argument");
  VhpPackedChunk c;
  c.mask = mask;
  c.word_base = word_base;
  c.vmask = vmask;
  c.elem_bytes = elem_bytes;
  c.literals = (const char *)literals;
  c.dst = (char *)dst;
  c.nunits = nunits;
  c.valid_bytes = (size_t)valid_bytes;
  VhpExpandPool pool(std::max(1, std::min(threads, 64)));
  pool.wait(pool.submit(c));
  return VHP_OK;
}

vhp_status vhp_expand_packed_range(const uint32_t *mask, const uint32_t *word_base,
                                   const uint32_t *vmask, int elem_bytes, const void *literals,
                                   int64_t nunits, int64_t valid_bytes, int64_t b0, int64_t b1, void *out) {
  if (elem_bytes != 4 && elem_bytes != 8)
    return fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_expand_packed_range: elem_bytes is 4 or 8");
  if (nunits < 0 || valid_bytes < 0 || valid_bytes > nunits * (int64_t)kVhpPackUnit ||
      valid_bytes <= (nunits - 1) * (int64_t)kVhpPackUnit)
    return fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_expand_packed_range: nunits does not match valid_bytes");
  if (b0 < 0 || b1 < b0 || b1 > valid_bytes || b0 % elem_bytes != 0)
    return fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_expand_packed_range: bad byte range");
  if (b0 == b1) return VHP_OK;
  if (!mask || !word_base || !vmask || !literals || !out)
    return fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_expand_packed_range: null argument");
  VhpPackedChunk c;
  c.mask = mask;
  c.word_base = word_base;
  c.vmask = vmask;
  c.elem_bytes = elem_bytes;
  c.literals = (const char *)literals;
  c.nunits = nunits;
  c.valid_bytes = (size_t)valid_bytes;
  vhp_expand_bytes(c, (size_t)b0, (size_t)b1, (char *)out);
  return VHP_OK;
}

vhp_status vhp_context_set_planner_loop(vhp_context *ctx, int mode) {
  if (!ctx || mode < 0 || mode > 3) return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_context_set_planner_loop: bad argument");
  ctx->grid_loop_mode = mode;
  return VHP_OK;
}

vhp_status vhp_context_set_grid_sweep(vhp_context *ctx, int mode) {
  if (!ctx || mode < 0 || mode > 2) return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_context_set_grid_sweep: bad argument");
  ctx->grid_sweep = mode;
  return VHP_OK;
}

void vhp_strip_halo_rows(int nx, int ny, int sx, int sy, int y0, int y1, int32_t rows[4]) {
  vhp_window_halo_rows(nx, ny, sx, sy, y0, y1, rows);
}

vhp_status vhp_strip_sweep_dev(vhp_context *ctx, const uint8_t *d_occ, int nx, int ny, int sx,
                               int sy, int y0, int y1, const double *const d_halo[4],
                               vhp_dtype dtype, void *d_vis_strip) {
  if (!ctx || !d_occ || !d_vis_strip || nx < 1 || ny < 1 || y0 < 0 || y1 > ny || y0 >= y1)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_strip_sweep_dev: bad argument");
  if (sx < 0 || sx >= nx || sy < 0 || sy >= ny)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_strip_sweep_dev: source outside the grid");
  if (dtype != VHP_F32 && dtype != VHP_F64) return fail(ctx, VHP_ERR_INVALID_ARG, "bad dtype");
  if (!vhp_sweep_tile_supported(nx, ny) && !grid_mode_available(ctx, nx, ny))
    return fail(ctx, VHP_ERR_UNSUPPORTED, "vhp_strip_sweep_dev: grid too wide for the tile kernel");
  int32_t rows[4];
  vhp_window_halo_rows(nx, ny, sx, sy, y0, y1, rows);
  for (int q = 0; q < 4; ++q)
    if (rows[q] >= 0 && (!d_halo || !d_halo[q]))
      return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_strip_sweep_dev: missing halo row");
  VHP_ON_DEVICE(ctx);
  vhp_status st = ensure_rcp2(ctx, std::max(nx, ny) + 64);
  if (st != VHP_OK) return st;
  if ((st = pack_tile(ctx, d_occ, 1, nx, ny, false)) != VHP_OK) return st;
  // Large windows are swept by many CTAs at once (grid mode): enough 8-warp CTAs for the tile
  // rows of the window, at most two per SM.
  const int grid_ctas = vhp_i_grid_ctas(ctx, nx, ny, y1 - y0);
  if (grid_ctas > 1 && (st = ensure(ctx, ctx->b_grid, vhp_sweep_grid_ws_bytes(nx, ny))) != VHP_OK) return st;
  VHP_CUDA(ctx, vhp_launch_sweep_window(ctx->tile, nx, ny, sx, sy, y0, y1, d_halo, dtype,
                                        d_vis_strip, ctx->rcp2_table, ctx->d_err,
                                        grid_ctas > 1 ? ctx->b_grid.p : nullptr, grid_ctas,
                                        ctx->stream, &ctx->launches));
  return VHP_OK;
}

vhp_status vhp_strip_epilogue_dev(vhp_context *ctx, int nx, int ny, int y0, int y1, int sx, int sy,
                                  int ex, int ey, double threshold, int32_t nb,
                                  const int32_t *d_light_sources, const double *d_vis_strip,
                                  double *d_vg_strip, double *d_h_strip, int32_t *d_came_strip,
                                  uint64_t *d_best) {
  if (!ctx || !d_light_sources || !d_vis_strip || !d_vg_strip || !d_h_strip || !d_came_strip ||
      !d_best || nx < 1 || ny < 1 || y0 < 0 || y1 > ny || y0 >= y1 || nb < 0)
    return fail(ctx, VHP_ERR_INVALID_ARG, "vhp_strip_epilogue_dev: bad argument");
  VHP_ON_DEVICE(ctx);
  const int nblocks = vhp_strip_epilogue_blocks(ctx->sm_count);
  vhp_status st = ensure(ctx, ctx->b_misc, (size_t)nblocks * 16 + 64);
  if (st != VHP_OK) return st;
  VHP_CUDA(ctx, vhp_launch_strip_epilogue(nx, ny, y0, y1, sx, sy, ex, ey, threshold, nb,
                                          d_light_sources, d_vis_strip, d_vg_strip, d_h_strip,
                                          d_came_strip, (unsigned long long *)ctx->b_misc.p,
                                          nblocks, (unsigned long long *)d_best, ctx->stream,
                                          &ctx->launches));
  return VHP_OK;
}

vhp_status vhp_planner_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                 int ny, const int32_t *d_se_xy, const int32_t *d_prob_map,
                                 int64_t nprob, double threshold, int32_t max_iter,
                                 int32_t ls_cap, vhp_dtype dtype, const vhp_planner_out *d_out) {
  static const vhp_planner_out none = {};
  vhp_status st = check_common(ctx, d_occ, nmaps, nx, ny, d_se_xy, nprob, dtype, ctx);
  if (st != VHP_OK) return st;
  VHP_ON_DEVICE(ctx);
  return planner_dev(ctx, d_occ, nmaps, nx, ny, d_se_xy, d_prob_map, nprob, threshold, max_iter,
                     ls_cap, dtype, d_out ? *d_out : none);
}

vhp_status vhp_planner_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                             const int32_t *se_xy, const int32_t *prob_map, int64_t nprob,
                             double threshold, int32_t max_iter, int32_t ls_cap, vhp_dtype dtype,
                             const vhp_planner_out *out) {
  static const vhp_planner_out none = {};
  const vhp_planner_out &h = out ? *out : none;
  vhp_status st = check_common(ctx, occ, nmaps, nx, ny, se_xy, nprob, dtype, ctx);
  if (st != VHP_OK) return st;
  if (prob_map)
    if ((st = check_points(ctx, nullptr, 0, prob_map, nprob, nmaps, nx, ny, "vhp_planner_batch")) != VHP_OK)
      return st;
  if (nprob == 0) return VHP_OK;
  VHP_ON_DEVICE(ctx);
  PlanesGuard planes_guard(ctx);
  // (the planner kernels always read the bit planes, whatever VHP_SWEEP_IMPL says)
  if ((st = stage_host_batch(ctx, occ, nmaps, nx, ny, se_xy, 16, nprob, prob_map, true)) != VHP_OK) return st;
  const size_t cells = (size_t)nx * ny, esz = dtype == VHP_F32 ? 4 : 8;
  // device staging for the requested outputs, a chunk of problems at a time
  const size_t per_prob = (h.vis ? esz * cells : 0) + (h.vg ? esz * cells : 0) + (h.came ? 4 * cells : 0) +
                          4 + 4 + 8 + 4 + 2 * (size_t)ls_cap * 8 + 64;
  const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(nprob, (int64_t)(((size_t)2 << 30) / per_prob)));
  vhp_status result = VHP_OK;
  if ((st = ensure(ctx, ctx->b_out[0], (size_t)chunk * per_prob + 256)) != VHP_OK) result = st;
  for (int64_t q0 = 0; q0 < nprob && result == VHP_OK; q0 += chunk) {
    const int64_t n = std::min(chunk, nprob - q0);
    char *w = (char *)ctx->b_out[0].p;
    auto take = [&](size_t bytes) { char *r = w; w += (bytes + 15) & ~(size_t)15; return r; };
    vhp_planner_out d = {};
    d.vis = h.vis ? take(esz * cells * n) : nullptr;
    d.vg = h.vg ? take(esz * cells * n) : nullptr;
    d.came = h.came ? (int32_t *)take(4 * cells * n) : nullptr;
    d.status = (int32_t *)take(4 * n);
    d.nb_sources = (int32_t *)take(4 * n);
    d.light_sources = (int32_t *)take(8 * (size_t)ls_cap * n);
    d.path_len = (double *)take(8 * n);
    d.path_n = (int32_t *)take(4 * n);
    d.path = (int32_t *)take(8 * (size_t)ls_cap * n);
    result = planner_dev(ctx, (const uint8_t *)ctx->b_occ.p, nmaps, nx, ny,
                         (const int32_t *)ctx->b_src.p + 4 * q0,
                         prob_map ? (const int32_t *)ctx->b_map.p + q0 : nullptr, n, threshold,
                         max_iter, ls_cap, dtype, d);
    if (result != VHP_OK) break;
    auto back = [&](void *dst, const void *src, size_t bytes) {
      if (dst && result == VHP_OK) {
        cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream);
        if (e != cudaSuccess) result = cuda_fail(ctx, e, "planner D2H");
      }
    };
    back(h.vis ? (char *)h.vis + q0 * cells * esz : nullptr, d.vis, esz * cells * n);
    back(h.vg ? (char *)h.vg + q0 * cells * esz : nullptr, d.vg, esz * cells * n);
    back(h.came ? h.came + q0 * cells : nullptr, d.came, 4 * cells * n);
    back(h.status ? h.status + q0 : nullptr, d.status, 4 * n);
    back(h.nb_sources ? h.nb_sources + q0 : nullptr, d.nb_sources, 4 * n);
    back(h.light_sources ? h.light_sources + 2 * (size_t)ls_cap * q0 : nullptr, d.light_sources, 8 * (size_t)ls_cap * n);
    back(h.path_len ? h.path_len + q0 : nullptr, d.path_len, 8 * n);
    back(h.path_n ? h.path_n + q0 : nullptr, d.path_n, 4 * n);
    back(h.path ? h.path + 2 * (size_t)ls_cap * q0 : nullptr, d.path, 8 * (size_t)ls_cap * n);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess && result == VHP_OK) result = cuda_fail(ctx, e, "planner sync");
  }
  if (result != VHP_OK) return result;
  return check_device_error(ctx);
}

void vhp_export_came_from_u64(const int32_t *came, int64_t n, uint64_t *out) {
  for (int64_t i = 0; i < n; ++i)
    out[i] = came[i] < 0 ? VHP_NO_PARENT_U64 : (uint64_t)came[i];
}

} // extern "C"
