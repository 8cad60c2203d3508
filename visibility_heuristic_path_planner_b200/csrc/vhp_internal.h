// vhp_internal.h -- shared declarations between the C-ABI layer and the kernels.
#ifndef VHP_INTERNAL_H
#define VHP_INTERNAL_H

#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "vhp.h"

// Bit planes of the tile sweep kernel (built by vhp_launch_pack_tile): row / column
// major, forward / mirrored, wx (wy) words per row (column) line including one zero
// word of padding (see kernels_sweep_tile.cu).
struct VhpTilePlanes {
  const uint32_t *rowF = nullptr, *rowR = nullptr, *colF = nullptr, *colR = nullptr;
  const uint32_t *bsum = nullptr;      // [map][block row][words]: 1 = aligned 32x32 block is free
  int wx = 0, wy = 0;
  size_t row_plane = 0, col_plane = 0; // words per map
};

// grow-only device buffer
struct VhpDevBuf {
  void *p = nullptr;
  size_t cap = 0;
};

// ---- packed result transport (result_transport.cu, host_expand.cpp) -------------
// A chunk of results (flat bytes) is cut into 128-byte units; 32 consecutive units make a
// mask word.  Unit u of word w is literal iff bit u of mask[w]; the literal units of a word
// are stored back to back from unit slot word_base[w] of the literal stream; a uniform unit is
// all 0.0 or, where bit u of vmask[w] is set, all 1.0 (elements of elem_bytes).
constexpr int kVhpPackUnit = 128;
constexpr int kVhpPackMetaHead = 16 + kVhpPackUnit; // cursor (padded) + the tail unit
struct VhpPackedChunk {
  const uint32_t *mask = nullptr;
  const uint32_t *word_base = nullptr;
  const uint32_t *vmask = nullptr; // bit u of word w: the uniform unit 32 w + u is 1.0 (else 0.0)
  int elem_bytes = 4;             // 4 or 8
  const char *literals = nullptr; // null: direct mode, the device stored the literal units in dst
  const char *tail = nullptr;     // direct mode: a partial, literal last unit
  int gpu_share = 0;              // direct mode: words w with w % 16 < gpu_share (not the last
                                  // one) were delivered completely by the device
  char *dst = nullptr;            // where the expanded chunk goes (caller's buffer)
  int64_t nunits = 0;
  size_t valid_bytes = 0;         // bytes of the chunk (the last unit may be partial)
};
// device-side meta block of one packed chunk: [cursor u64, pad to 16][tail unit][mask][word_base][vmask]
inline size_t vhp_pack_meta_bytes(int64_t nunits, int elem_bytes) {
  const int64_t nwords = (nunits + 31) / 32;
  (void)elem_bytes;
  return kVhpPackMetaHead + (size_t)nwords * 12;
}
// in: nunits * 128 readable bytes.  Writes the meta block and either the literal stream
// (host_dst null) or the literal units themselves to host_dst + 128 * unit (a device-accessible
// host address, 16-byte aligned; tail_partial: the last unit is partial and goes to the meta block).
cudaError_t vhp_launch_pack_results(const void *d_in, int64_t nunits, int elem_bytes, void *d_meta,
                                    void *d_literals, void *host_dst, int tail_partial,
                                    int gpu_share, int sm_count, cudaStream_t st,
                                    int64_t *launches);

// thresholded binary visibility: bits[row][ceil(nx/32)] from fp64 rows (result_transport.cu)
cudaError_t vhp_launch_threshold_bits(const double *d_vis, int64_t nrows, int nx, double thr,
                                      uint32_t *d_bits, int sm_count, cudaStream_t st, int64_t *launches,
                                      uint16_t *d_row_cnt = nullptr);
cudaError_t vhp_launch_runs_row_count(const uint32_t *d_bits, int64_t nrows, int nx, uint16_t *d_row_cnt,
                                      int sm_count, cudaStream_t st, int64_t *launches);
// row runs: d_row_cnt (uint16 per row) comes from the threshold pass or from runs_row_count; runs_count leaves row_off (uint32
// per row) and pair_ptr (npairs + 1) on the device, runs_write the transition columns
cudaError_t vhp_launch_runs_count(const uint16_t *d_row_cnt, int64_t npairs, int ny, uint32_t *d_row_off,
                                  uint32_t *d_pair_tot, unsigned long long base,
                                  unsigned long long *d_pair_ptr, cudaStream_t st, int64_t *launches);
cudaError_t vhp_launch_runs_write(const uint32_t *d_bits, int64_t npairs, int ny, int nx,
                                  const uint32_t *d_row_off, const unsigned long long *d_pair_ptr,
                                  unsigned long long chunk_base, uint16_t *d_trans, int sm_count,
                                  cudaStream_t st, int64_t *launches);

// bytes [b0, b1) of a packed chunk in staged form (literals != null) -> out (host_expand.cpp)
void vhp_expand_bytes(const VhpPackedChunk &c, size_t b0, size_t b1, char *out);

// host threads that expand packed chunks into the caller's buffer (FIFO, each job is spread
// over all threads)
class VhpExpandPool {
 public:
  explicit VhpExpandPool(int nthreads);
  ~VhpExpandPool();
  int threads() const;
  double busy_seconds() const;                 // time spent expanding so far (jobs are serial)
  int64_t submit(const VhpPackedChunk &chunk); // returns a ticket
  void wait(int64_t ticket);                   // returns when that job and all earlier ones are done
 private:
  struct Impl;
  Impl *impl_;
};

struct vhp_giant;

struct vhp_context {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr; // D2H of the host-buffer entry points
  bool owns_stream = false;
  int sm_count = 0;
  int64_t launches = 0;
  std::string last_error;
  // device-side error word (bit 0: a source / start / end outside the grid, bit 2: inconsistent source groups,
  // bit 3: a bad view of vhp_visibility_cover_greedy_view_batch_dev, bit 4: a bad view of
  // vhp_visibility_merge_view_batch_dev)
  int *d_err = nullptr;
  // workspace buffers (grown on demand, reused across calls)
  VhpDevBuf b_occ, b_src, b_map, b_out[2], b_scratch, b_planner, b_misc, b_grid, b_bin;
  VhpDevBuf b_merge; // vhp_visibility_merge_batch: per-pair table; host call: group layout too
  // vhp_visibility_merge_range_batch, fallback: the fp64 windows of a chunk of pairs (apart from b_bin and b_misc,
  // which the window routes use themselves)
  VhpDevBuf b_mwin;
  // vhp_visibility_cover_greedy_batch: the candidates' coverage bits, and the workspace of the greedy rounds
  VhpDevBuf b_cover, b_cover_ws;
  // vhp_visibility_cover_greedy_view_batch: the candidates' views, uploaded with the candidates
  VhpDevBuf b_views;
  cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
  // 1/k table {rh, rl} of the tile kernel (double-double reciprocal), device resident
  double *rcp2_table = nullptr;
  int rcp2_len = 0;
  // set by vhp_prepare_maps_dev: reuse the bit planes for the same d_occ pointer
  bool planes_sticky = false;
  // tile-kernel bit planes of the last packed batch of maps
  const uint8_t *tile_src = nullptr;
  int tile_nmaps = 0, tile_nx = 0, tile_ny = 0;
  uint32_t *tile_buf = nullptr;
  size_t tile_bytes = 0;
  VhpTilePlanes tile;
  // K1 implementation (env VHP_SWEEP_IMPL): 0 = tile wavefront kernel where its boundary
  // arrays fit shared memory, else the naive kernel; 1 = always the naive kernel
  int sweep_impl = 0;
  // strip sweeps over many CTAs: 0 never, 1 for windows of >= 2^20 cells, 2 always
  int grid_sweep = 1;
  // planner batches: first sweep of every problem batch-wide (0 never, 1 from 4 waves of problems on
  // (default), 2 always; env VHP_PLANNER_FIRST)
  int planner_first = 1;
  int bin_direct = 1; // binary outputs: the sweep writes bits itself (env VHP_BIN_DIRECT=0: fp64 field + threshold pass)
  int planner_first_rounds = 1; // sweeps per problem done batch-wide (env VHP_PLANNER_ROUNDS; measured: 1 is
                                // fastest -- later rounds have too few active problems for whole-batch launches)
  // packed result transport of the host-buffer entry points: 0 plain D2H, 1 automatic
  // (packed when the results compress), 2 always packed (env VHP_RESULT_TRANSPORT)
  int result_transport = 1;
  // packed transport into a pinned, mapped caller buffer: the device stores the literal units
  // straight into it (env VHP_RESULT_DIRECT=0 keeps the staged literal stream)
  bool result_direct = true;
  // direct mode: sixteenths of the mask words the device delivers completely (default 0: only
  // the literal units come over PCIe; env VHP_RESULT_GPU_SHARE)
  int result_gpu_share = 0;
  static constexpr int kPackSets = 3;
  VhpDevBuf b_pack_out[kPackSets], b_pack_meta[kPackSets], b_pack_lit[kPackSets];
  void *h_pack_meta[kPackSets] = {nullptr, nullptr, nullptr};
  void *h_pack_lit[kPackSets] = {nullptr, nullptr, nullptr};
  size_t h_pack_meta_cap = 0, h_pack_lit_cap = 0;
  cudaEvent_t ev_pack_meta[kPackSets] = {nullptr, nullptr, nullptr}; // packed + meta copied
  cudaEvent_t ev_pack_lit[kPackSets] = {nullptr, nullptr, nullptr};  // results of the set computed
  cudaEvent_t ev_pack_t0[kPackSets] = {nullptr, nullptr, nullptr};   // timing: packing starts
  bool transport_trace = false; // env VHP_TRANSPORT_TRACE: per-call timing summary on stderr
  VhpExpandPool *expand_pool = nullptr;
  // statistics of the last host-buffer call (vhp_context_last_transport)
  int64_t last_d2h_bytes = 0, last_result_bytes = 0;
  int last_transport_packed = 0; // 0 plain, 1 packed (staged literal stream), 2 packed (direct)
  // vhp_planner_batch, one large problem on the whole GPU: the strip engine of giant.cu with one
  // strip (cached with its captured graph); loop mode as vhp_giant_set_loop_mode
  vhp_giant *grid_engine = nullptr;
  int grid_loop_mode = 0;
};

// helpers of capi.cu used by giant.cu
vhp_status vhp_i_fail(vhp_context *ctx, vhp_status st, const std::string &msg);
vhp_status vhp_i_ensure_rcp2(vhp_context *ctx, int len);
// CTAs one strip sweep of `rows` rows is spread over (1: the single-CTA window kernel)
int vhp_i_grid_ctas(const vhp_context *ctx, int nx, int ny, int rows);
// giant.cu: solve() of one problem on buffers the caller owns (planner_dev's grid route)
vhp_status vhp_i_grid_planner_run(vhp_context *ctx, const VhpTilePlanes &pl, int nx, int ny,
                                  const int32_t se[4], double thr, int32_t max_iter, int32_t ls_cap,
                                  double *vis, double *vg, double *hc, int32_t *came, int32_t *ls);
const int *vhp_i_grid_planner_ctl(const vhp_context *ctx);
void vhp_i_grid_planner_release(vhp_context *ctx);

// ---- kernel launchers (all enqueue on `st`, return cudaGetLastError()) --------
// Each launcher returns the number of kernel launches it made through *launches.

// K1, straightforward L-front kernel (one CTA per (pair, quadrant), fronts in
// global memory).  Cross-check of the tile kernel and fallback for very large grids.
cudaError_t vhp_launch_sweep_naive(const uint8_t *d_occ, int nx, int ny,
                                   const int32_t *d_src_xy, const int32_t *d_src_map,
                                   int64_t npairs, vhp_dtype dtype, void *d_out,
                                   double *d_scratch, int *d_err, cudaStream_t st,
                                   int64_t *launches);
size_t vhp_sweep_naive_scratch_bytes(int nx, int ny, int64_t npairs);

// K1, tile wavefront (32 x 32 tiles, uniform tiles are plain fills): the default.
bool vhp_sweep_tile_supported(int nx, int ny);
bool vhp_sweep_grid_supported(int nx, int ny); // many-CTA grid mode (boundary rows in global memory)
void vhp_tile_plane_geometry(int nx, int ny, int *wx, int *wy, int *sum_words_per_map);
cudaError_t vhp_launch_pack_tile(const uint8_t *d_occ, int nmaps, int nx, int ny, uint32_t *rowF,
                                 uint32_t *rowR, uint32_t *colF, uint32_t *colR, uint32_t *bsum,
                                 cudaStream_t st, int64_t *launches);
cudaError_t vhp_launch_sweep_tile(const VhpTilePlanes &pl, int nx, int ny, const int32_t *d_src_xy,
                                  const int32_t *d_src_map, int64_t npairs, vhp_dtype dtype,
                                  void *d_out, const double *d_rcp2, int *d_err, cudaStream_t st,
                                  int64_t *launches, const double *thr = nullptr, bool bits = false);
// thr != null, bits: d_out = uint32 words, bit (x & 31) of word [pair][y][x >> 5] = (fp64 value >= thr);
// needs thr > 0 (zeroes d_out, then writes only the cells at or above the threshold).

// Range-limited windows (vhp_visibility_window_batch): the one-CTA tile kernel sweeps only the (2R+1)^2 window
// of each pair (kFmtWindow, shared memory sized by the window; supported: it fits one CTA), into d_out
// [pair][2R+1][2R+1]; a map index out of range raises bit 0 of d_err like a source outside the grid.
bool vhp_sweep_window_supported(int nx, int ny, int radius);
// ... and the direct route of vhp_visibility_merge_view_batch (kFmtMergeView*), whose CTAs keep their view in a
// shared-memory tail
bool vhp_sweep_merge_view_supported(int nx, int ny, int radius);
cudaError_t vhp_launch_sweep_window_batch(const VhpTilePlanes &pl, int nmaps, int nx, int ny,
                                          const int32_t *d_src_xy, const int32_t *d_src_map, int64_t npairs,
                                          int radius, vhp_dtype dtype, void *d_out, const double *d_rcp2,
                                          int *d_err, cudaStream_t st, int64_t *launches);
// fallback: the windows of np pairs cut out of their full fields d_fields[np][ny][nx] (0 outside the grid), and the
// copy of a batch's pairs whose out-of-range map indices become sources outside the grid
cudaError_t vhp_launch_window_crop(const void *d_fields, int64_t np, int nx, int ny, const int32_t *d_src_xy,
                                   int radius, vhp_dtype dtype, void *d_out, int sm_count, cudaStream_t st,
                                   int64_t *launches);
cudaError_t vhp_launch_window_pairs(const int32_t *d_src_xy, const int32_t *d_src_map, int64_t np, int nmaps,
                                    int32_t *d_xy_out, int32_t *d_map_out, int sm_count, cudaStream_t st,
                                    int64_t *launches);

// Merged visibility of groups of sources (vhp_visibility_merge_batch): the group outputs ([group][ny][nx], any may be
// null; vmax fp32 when f32) and the per-pair table merge_table_kernel builds from the CSR group layout.
struct VhpMergeDev {
  void *vmax = nullptr;
  int f32 = 0;
  int32_t *first = nullptr;
  uint32_t *count = nullptr;
  const int32_t *pair_group = nullptr; // group of the pair, -1: the layout is inconsistent there (skip it)
  const int32_t *pair_k = nullptr;     // index of the pair within its group
  const int32_t *pair_map = nullptr;   // map of the pair (its group's)
};
// range of vhp_visibility_merge_range_batch: 0 <= radius <= 16383, shape VHP_RANGE_BOX / VHP_RANGE_DISK.  views:
// vhp_visibility_merge_view_batch's [pair][5] = (r, ax, ay, bx, by) on the device, indexed like the pairs (null: the
// range merge)
struct VhpMergeRange {
  int radius = 0;
  int shape = VHP_RANGE_BOX;
  const int32_t *views = nullptr;
  VhpMergeRange() = default;
  VhpMergeRange(int r, int s, const int32_t *v = nullptr) : radius(r), shape(s), views(v) {}
};
// the sweeps fold straight into the group outputs (kFmtMerge*, one CTA per pair); needs thr > 0 and zero-filled
// vmax / count, -1-filled first.  range: sweep only each pair's box and fold only its cells in range
// (kFmtMergeRange*; supported where vhp_sweep_window_supported holds); range->views: fold only each pair's cells in
// its view (kFmtMergeView*, supported where vhp_sweep_merge_view_supported holds; a bad view raises bit 4 of d_err)
cudaError_t vhp_launch_sweep_merge(const VhpTilePlanes &pl, int nx, int ny, const int32_t *d_src_xy,
                                   const VhpMergeDev &m, int64_t npairs, double thr, const double *d_rcp2,
                                   int *d_err, cudaStream_t st, int64_t *launches,
                                   const VhpMergeRange *range = nullptr);
// kernels_merge.cu: the per-pair table (validates the layout: bit 4 of d_err), the output fill, and the fold of
// np fp64 fields of pairs [p0, p0 + np) (what the fallback sweeps into a chunk buffer) into the group outputs
cudaError_t vhp_launch_merge_table(const int64_t *d_group_ptr, const int32_t *d_group_map, int64_t ngroups,
                                   int64_t nsrc, int nmaps, int32_t *d_pair_group, int32_t *d_pair_k,
                                   int32_t *d_pair_map, int *d_err, int sm_count, cudaStream_t st,
                                   int64_t *launches);
cudaError_t vhp_launch_merge_fill(const VhpMergeDev &m, size_t cells_total, cudaStream_t st);
cudaError_t vhp_launch_merge_fold(const double *d_field, int64_t p0, int64_t np, int nx, int ny,
                                  const int32_t *d_src_xy, double thr, const VhpMergeDev &m, int sm_count,
                                  cudaStream_t st, int64_t *launches);
// the fold of np fp64 windows d_win[np][2R+1][2R+1] of pairs [p0, p0 + np) (vhp_visibility_window_batch's layout)
// into the group outputs, cells in range only (relaxed red atomics: any order gives the same result); with
// range.views the cells in each pair's view only (a bad view raises bit 4 of d_err and folds nothing)
cudaError_t vhp_launch_merge_window_fold(const double *d_win, int64_t p0, int64_t np, int nx, int ny,
                                         const int32_t *d_src_xy, double thr, const VhpMergeRange &range,
                                         const VhpMergeDev &m, int *d_err, int sm_count, cudaStream_t st,
                                         int64_t *launches);

// Greedy coverage placement (vhp_visibility_cover_greedy_batch).  The coverage bits of a candidate at (sx, sy) are
// stored over its box, clipped to the grid: H = min(2R+1, ny) rows from row y0 and W words (the span rule of
// win_sum_words) from word w0 of the map's 32-column words, so cell (x, y) is bit x & 31 of word
// (y - y0) * W + (x >> 5) - w0.  R is the radius clamped to max(nx, ny) - 1, which leaves the box unchanged.  Every
// box has the same H x W words; a candidate outside the grid gets the box of the nearest cell.
struct VhpCoverBox {
  int y0, w0, H, W;
};
__host__ __device__ inline int vhp_cover_words(int nx, int R) {
  const int nw = (nx + 31) >> 5, span = (2 * R + 31) / 32 + 1;
  return nw < span ? nw : span;
}
__host__ __device__ inline VhpCoverBox vhp_cover_box(int nx, int ny, int R, int sx, int sy) {
  sx = sx < 0 ? 0 : (sx >= nx ? nx - 1 : sx);
  sy = sy < 0 ? 0 : (sy >= ny ? ny - 1 : sy);
  VhpCoverBox b;
  b.H = ny < 2 * R + 1 ? ny : 2 * R + 1;
  b.W = vhp_cover_words(nx, R);
  const int y0 = sy - R < 0 ? 0 : sy - R, w0 = (sx - R < 0 ? 0 : sx - R) >> 5, nw = (nx + 31) >> 5;
  b.y0 = y0 < ny - b.H ? y0 : ny - b.H;
  b.w0 = w0 < nw - b.W ? w0 : nw - b.W;
  return b;
}
// Phase 1, direct route (thr > 0, vhp_sweep_window_supported): the one-CTA tile kernel sweeps each candidate's box
// straight into its bits (kFmtCoverBits; zeroes d_bits first, the box only, no disk).  Pair p's map is d_src_map[p].
cudaError_t vhp_launch_sweep_cover(const VhpTilePlanes &pl, int nx, int ny, const int32_t *d_src_xy,
                                   const int32_t *d_src_map, int64_t npairs, int radius, double thr, uint32_t *d_bits,
                                   const double *d_rcp2, int *d_err, cudaStream_t st, int64_t *launches);
// kernels_cover.cu.  Fallback of phase 1: the bits of pairs [p0, p0 + np) from their fp64 values, win_r >= 0: windows
// [np][2 win_r + 1]^2 centred on the candidate, win_r < 0: whole fields [np][ny][nx]; each bit is the cell's range
// test (box of radius R, disk dx^2 + dy^2 <= r2 if disk), "writes" test and v >= thr.
cudaError_t vhp_launch_cover_fold(const double *d_val, int win_r, int64_t p0, int64_t np, int nx, int ny, int R,
                                  bool disk, int r2, const int32_t *d_xy, double thr, uint32_t *d_bits, int sm_count,
                                  cudaStream_t st, int64_t *launches);
// Phase 2, the greedy rounds over the bits of nsrc candidates (table of vhp_launch_merge_table) of nprob problems.
// The outputs of every cover call (any may be null): gain is uint32 (cells) for the cover call, uint64 (summed
// weights) for the weighted ones; the m-fold rounds write count instead of covered.
struct VhpCoverOut {
  int32_t *pick = nullptr;     // [prob][k]
  void *gain = nullptr;        // [prob][k]
  int32_t *npicked = nullptr;  // [prob]
  uint32_t *covered = nullptr; // [prob][ny][ceil(nx/32)]
  uint8_t *count = nullptr;    // [prob][ny][nx], min(m, picks whose S covers the cell)
};
// cover_apply_kernel's parameter (kernels_cover.cu): the outputs but count, with the gain typed
template <class Gain>
struct VhpCoverDevT {
  int32_t *pick = nullptr;   // [prob][k]
  Gain *gain = nullptr;      // [prob][k]
  int32_t *npicked = nullptr; // [prob]
  uint32_t *covered = nullptr; // [prob][ny][ceil(nx/32)]
};
// workspace bytes of the rounds beyond the candidate bits (weighted: uint64 gains and the padded weight plane; m-fold:
// those of the weighted rounds and a counter plane of the padded plane's size)
size_t vhp_cover_ws_bytes(int64_t nprob, int64_t nsrc, int nx, int ny, int R, bool weighted, bool mfold = false);
// outputs are filled here; d_bits: the candidates' box bits; disk_r2 >= 0: apply the disk mask first (the direct
// route's sweep stores the whole box).  d_extra (may be null): [prob][ny][ceil(nx/32)] uint32 bits of the cells to
// cover, or for the weighted rounds [prob][ny][nx] uint8 weights (null: every cell weighs 1; nsrc < 2^28).  The
// m-fold rounds (with weighted) are the weighted rounds where a cell's weight counts until m in [1, 255] picks cover it.
cudaError_t vhp_launch_cover_greedy(uint32_t *d_bits, int64_t nsrc, int64_t nprob, int nx, int ny, int R, int disk_r2,
                                    const int32_t *d_xy, const int32_t *d_pair_group, const int32_t *d_pair_k,
                                    bool weighted, bool mfold, const void *d_extra, int32_t k, int m, void *d_ws,
                                    const VhpCoverOut &out, int sm_count, cudaStream_t st, int64_t *launches);
// the view call, between phase 1 and the m-fold rounds (which then run with disk_r2 = -1): every candidate's bits
// &= its view, d_views [nsrc][5] = (r, ax, ay, bx, by): range r in [0, radius] in the call's shape (disk or box), and
// the sector of a and b.  A bad view raises bit 3 of d_err and clears the candidate's bits.
cudaError_t vhp_launch_cover_view(uint32_t *d_bits, int64_t nsrc, int nx, int ny, int R, int radius, bool disk,
                                  const int32_t *d_xy, const int32_t *d_views, int *d_err, int sm_count,
                                  cudaStream_t st, int64_t *launches);

// opt-in sweep variants (kernels_sweep_variant.cu): model 1 getAccessibilityMap.m (alpha, fac),
// model 2 computeVisibilityUsingQueue as an order-free rule (cutoff)
cudaError_t vhp_launch_sweep_variant(const uint8_t *d_occ, int nx, int ny, const int32_t *d_src_xy,
                                     const int32_t *d_src_map, int64_t npairs, int model, double alpha,
                                     double fac, double light_strength, double cutoff, double *d_buf,
                                     float *d_out32, int *d_err, cudaStream_t st, int64_t *launches);

// giant-map path: one sweep of map 0 restricted to the rows [y0, y1) of a strip, and the
// planner epilogue + arg-min over a strip (whole GPU)
void vhp_window_halo_rows(int nx, int ny, int sx, int sy, int y0, int y1, int32_t rows[4]);
// d_grid_ws (vhp_sweep_grid_ws_bytes bytes) with grid_ctas > 1: the sweep is spread over that
// many CTAs (two launches), else a single CTA does it.
size_t vhp_sweep_grid_ws_bytes(int nx, int ny);
void vhp_sweep_grid_ws_flags(int nx, int ny, size_t *offset, size_t *bytes);
// Strip boundaries across GPUs, handed over tile by tile through peer memory (grid mode only; see
// TileArgs::x_edges in sweep_tile_body.cuh).  x_ws: the neighbour's grid workspace of this chain
// (peer-mapped, null: nothing to export), [x_y0, x_y1): its window; remote_mask: quadrants whose
// lower boundary this sweep receives that way.
struct VhpSweepPeer {
  void *x_ws = nullptr;
  int x_y0 = 0, x_y1 = 0;
  int remote_mask = 0;
};
cudaError_t vhp_launch_sweep_window(const VhpTilePlanes &pl, int nx, int ny, int sx, int sy, int y0,
                                    int y1, const double *const d_halo[4], vhp_dtype dtype,
                                    void *d_out_strip, const double *d_rcp2, int *d_err,
                                    void *d_grid_ws, int grid_ctas, cudaStream_t st,
                                    int64_t *launches, int qmask = 0xF,
                                    const int *d_src_ctl = nullptr, const VhpSweepPeer *peer = nullptr);
// one LARGE planner problem on the whole GPU (capi.cu: planner_grid_one -> giant.cu): outputs
// from the loop state d_ctl = {done, next x, next y, status, nb_of_sources, ...}
cudaError_t vhp_launch_grid_planner_finish(const int *d_ctl, int nx, int ny, int ex, int ey,
                                           int ls_cap, int32_t *d_ls, const int32_t *d_came,
                                           double *d_vis, const double *d_vg, int32_t *d_status,
                                           int32_t *d_nb, double *d_path_len, int32_t *d_path_n,
                                           int32_t *d_path, float *d_vg32, float *d_vis32,
                                           cudaStream_t st, int64_t *launches);
int vhp_strip_epilogue_blocks(int sm_count);
cudaError_t vhp_launch_strip_epilogue(int nx, int ny, int y0, int y1, int sx, int sy, int ex, int ey,
                                      double thr, int nb, const int32_t *d_ls, const double *d_vis,
                                      double *d_vg, double *d_hc, int32_t *d_came,
                                      unsigned long long *d_partial, int nblocks,
                                      unsigned long long *d_best, cudaStream_t st,
                                      int64_t *launches, const int *d_ctl = nullptr);

cudaError_t vhp_launch_rcp2_table(double *d_table, int len, cudaStream_t st, int64_t *launches);
cudaError_t vhp_launch_ratio2_selftest(const double *d_rcp2, int kmax,
                                       unsigned long long *d_mismatches, cudaStream_t st,
                                       int64_t *launches);

// random-rectangle environments on the device (kernels_env.cu); vhp_env_draw = its generator
uint32_t vhp_env_draw(uint64_t seed, uint64_t map, uint64_t obstacle, uint32_t d);
cudaError_t vhp_launch_env_generate(uint8_t *d_occ, int nmaps, int nx, int ny, int64_t first_map,
                                    uint64_t seed, int64_t nb_of_obstacles, int64_t min_w,
                                    int64_t max_w, int64_t min_h, int64_t max_h, cudaStream_t st,
                                    int64_t *launches);

// K4 ray casting
cudaError_t vhp_launch_raycast(const uint8_t *d_occ, int nx, int ny,
                               const int32_t *d_src_xy, const int32_t *d_src_map,
                               int64_t npairs, vhp_dtype dtype, void *d_out,
                               int *d_err, cudaStream_t st, int64_t *launches);

// K2/K3/K5 planner: one persistent CTA per problem (sweep + fused epilogue +
// arg-min + next-source selection + path reconstruction, no host round trip).
// Working fields are fp64; vg32/vis32 are optional fp32 exports.
bool vhp_planner_supported(int nx, int ny);
cudaError_t vhp_launch_planner(const VhpTilePlanes &pl, int nx, int ny, const int32_t *d_se_xy,
                               const int32_t *d_prob_map, int64_t nprob, double threshold,
                               int32_t max_iter, int32_t ls_cap, const double *d_rcp2,
                               double *d_vis, double *d_vg, double *d_hc, int32_t *d_came,
                               int32_t *d_status,
                               int32_t *d_nb, int32_t *d_ls, double *d_path_len, int32_t *d_path_n,
                               int32_t *d_path, float *d_vg32, float *d_vis32, int *d_err,
                               cudaStream_t st, int64_t *launches, void *d_first_ws = nullptr,
                               int first_rounds = 1);
// d_first_ws (vhp_planner_first_ws_bytes(nprob) bytes): run every problem's first sweep and epilogue
// batch-wide before the persistent kernel (worth it from a few waves of problems on)
size_t vhp_planner_first_ws_bytes(int64_t nprob);

#endif
