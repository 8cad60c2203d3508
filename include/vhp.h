/*
 * vhp.h -- C-ABI of libvhp_b200.so: the B200-native (sm_100a) replacement for the
 * hot path of IbrahimSquared/visibility-heuristic-path-planner:
 *
 *     visibilityBasedSolver::computeVisibility   src/visibilityBasedSolver.cpp:570-696
 *     visibilityBasedSolver::updateVisibility    src/visibilityBasedSolver.cpp:379-565
 *     visibilityBasedSolver::solve               src/visibilityBasedSolver.cpp:76-160
 *     visibilityBasedSolver::reconstructPath     src/visibilityBasedSolver.cpp:1183-1213
 *     visibilityBasedSolver::raycasting (+loops) src/visibilityBasedSolver.cpp:267-290,228-232
 *
 * The reference has no plugin / FFI layer: its surface is the C++ class
 * vbs::visibilityBasedSolver (include/solver/visibilityBasedSolver.h:23-175), the
 * config file (src/parser.cpp) and the .txt files it writes under ./output
 * (src/visibilityBasedSolver.cpp:1022-1178).  This header is what a binding for
 * that surface would call; include/vhp_solver.hpp is the C++ drop-in class built
 * on it and INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *  - plain pointers and sizes only; no C++/torch types.
 *  - 2-D fields use the reference's Field<T> layout: index = x + y*nx
 *    (include/environment/field.h:26-29).  Batches are [item][y][x].
 *  - occupancy ("occupancy complement" in the reference): uint8, 1 = free,
 *    0 = occupied (the reference stores 1.0 / 0.0 doubles, src/environment.cpp:198-209).
 *  - coordinates are (x, y) int32 pairs in the solver's internal frame (what
 *    ls_ / lightSources_ hold, i.e. after the mode-2 y flip of solve() :83-86).
 *  - all arithmetic is IEEE binary64 in the reference's operation order with one
 *    rounding per operation (no FMA contraction); VHP_F32 only rounds the final
 *    value once when it is stored.
 *  - functions ending in _dev take DEVICE pointers and enqueue on the context's
 *    stream without synchronising; the others take HOST pointers, copy in/out
 *    and return when the result is in the host buffers.
 *  - every entry point returns a vhp_status; negative = failure (message via
 *    vhp_last_error).  There is no CPU fallback: without a CUDA device every
 *    compute entry point fails with VHP_ERR_NO_DEVICE.
 */
#ifndef VHP_H
#define VHP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VHP_ABI_VERSION 1

typedef struct vhp_context vhp_context; /* one device + one stream + workspace */

typedef enum vhp_status {
  /* solve() outcomes, in the order the reference tests them (:89-116, :134-139) */
  VHP_OK = 0,
  VHP_START_OOB = 1,      /* "Start point is out of bounds." */
  VHP_END_OOB = 2,        /* "End point is out of bounds." */
  VHP_START_OCCUPIED = 3, /* "Start point is not valid (occupied)" */
  VHP_END_OCCUPIED = 4,   /* "End point is not valid (occupied)" */
  VHP_MAX_ITER = 5,       /* "Max iters hit. Solution could not be found. ..." */
  /* library failures */
  VHP_ERR_INVALID_ARG = -1,
  VHP_ERR_NO_DEVICE = -2,
  VHP_ERR_CUDA = -3,
  VHP_ERR_IO = -4,
  VHP_ERR_UNSUPPORTED = -5
} vhp_status;

typedef enum vhp_dtype {
  VHP_F32 = 0, /* fp64 on chip, rounded once to fp32 at the store */
  VHP_F64 = 1  /* bit-identical to the reference's Field<double> */
} vhp_dtype;

/* cameFrom_ "no parent" marker.  The reference keeps Field<size_t> filled with
 * 1e15 (:46); this library stores int32 parents with -1 and widens to the
 * reference's value only in vhp_export_came_from_u64 / cameFrom.txt. */
#define VHP_NO_PARENT (-1)
#define VHP_NO_PARENT_U64 1000000000000000ULL

/* ---- library / context ------------------------------------------------------ */
int vhp_abi_version(void);
const char *vhp_version_string(void);
int vhp_device_count(void);                  /* 0 when there is no usable GPU */

/* `cuda_stream` is a cudaStream_t (as void*) to enqueue on, or NULL to let the
 * context create its own non-blocking stream. */
vhp_status vhp_context_create(int device, void *cuda_stream, vhp_context **out);
void vhp_context_destroy(vhp_context *ctx);
vhp_status vhp_context_synchronize(vhp_context *ctx);
int vhp_context_device(const vhp_context *ctx); /* CUDA device index of the context (-1: NULL) */
const char *vhp_last_error(const vhp_context *ctx); /* ctx may be NULL: global */
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t vhp_launch_count(const vhp_context *ctx);

/* diagnostic: the sweep kernel computes c = i/k as fma(i, rh, i*rl) with (rh, rl) a
 * double-double 1/k instead of an IEEE divide; this counts the (i,k),
 * 0 <= i < k <= kmax, for which the two differ on this device (must be 0;
 * kmax <= 16384). */
vhp_status vhp_selftest_ratio(vhp_context *ctx, int kmax, int64_t *mismatches);

/* ---- a1: batched stand-alone visibility sweep (computeVisibility) ------------
 * npairs independent (map, source) pairs.  pair p uses map src_map[p] (NULL ->
 * map 0 for every pair) and source (src_xy[2p], src_xy[2p+1]).
 *   out[p][y][x] = visibility_ after computeVisibility() started from an all-zero
 *   field: cells the reference never writes (column 0 / row 0 when the source is
 *   not on them, SURVEY A.2 item 2) are 0.
 * A source outside the grid fails the call with VHP_ERR_INVALID_ARG; an occupied
 * source gives an all-zero field like the reference (v = 1*occ = 0). */
vhp_status vhp_visibility_batch(vhp_context *ctx, const uint8_t *occ, int nmaps,
                                int nx, int ny, const int32_t *src_xy,
                                const int32_t *src_map, int64_t npairs,
                                vhp_dtype dtype, void *out);
vhp_status vhp_visibility_batch_dev(vhp_context *ctx, const uint8_t *d_occ,
                                    int nmaps, int nx, int ny,
                                    const int32_t *d_src_xy,
                                    const int32_t *d_src_map, int64_t npairs,
                                    vhp_dtype dtype, void *d_out);
/* The same fields as a PACKED HANDLE: lossless, expanded lazily.  Visibility fields are mostly flat
 * (lit 1.0, shadow 0.0), so the device cuts the results into 128-byte units that are either uniform
 * (all 0.0 or all 1.0) or literal, and only two bits per unit plus the literal units cross PCIe --
 * 3.5 % of the bytes on the empty 1000 x 1000 batch.  vhp_visibility_batch expands that stream into the
 * caller's buffer inside the call (and is then bound by the host's memory bandwidth: 16 GB of stores per
 * 4096 sweeps); this entry point keeps it, in pinned host memory owned by the handle, and
 * vhp_packed_expand rebuilds any range of pairs on demand, bit-identical to what vhp_visibility_batch
 * writes.  *handle = NULL creates a handle; passing an existing one reuses its memory (the steady
 * state of a caller that processes batch after batch allocates nothing). */
typedef struct vhp_packed vhp_packed;
vhp_status vhp_visibility_batch_packed(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx,
                                       int ny, const int32_t *src_xy, const int32_t *src_map,
                                       int64_t npairs, vhp_dtype dtype, vhp_packed **handle);
int64_t vhp_packed_pairs(const vhp_packed *h);      /* pairs held */
int64_t vhp_packed_bytes(const vhp_packed *h);      /* bytes of packed data held (= moved over PCIe) */
int64_t vhp_packed_pair_bytes(const vhp_packed *h); /* bytes of one expanded pair: nx * ny * element size */
/* out[0 .. npairs * pair_bytes) = the fields of pairs [first_pair, first_pair + npairs); host threads
 * (nthreads <= 0: one per 64 MB, at most the hardware's) */
vhp_status vhp_packed_expand(const vhp_packed *h, int64_t first_pair, int64_t npairs, void *out,
                             int nthreads);
void vhp_packed_destroy(vhp_packed *h);
/* Thresholded binary visibility, bit-packed: the part of the result that decides (which cells a
 * light source sees), 32 x smaller than fp32 fields -- 125 KB instead of 4 MB per 1000 x 1000 sweep,
 * so the host-buffer call is no longer bound by the host's memory system and scales with the
 * GPUs' PCIe links.
 *   out_bits[p][y][w], w < ceil(nx / 32): bit b of word w = visibility_(32w + b, y) >= threshold
 * decided on the fp64 value, i.e. bit-exact against the reference's fp64 field compared with
 * `>= threshold` (the test the planner applies, :419); bits beyond nx are 0. */
vhp_status vhp_visibility_batch_bin(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx,
                                    int ny, const int32_t *src_xy, const int32_t *src_map,
                                    int64_t npairs, double threshold, uint32_t *out_bits);
vhp_status vhp_visibility_batch_bin_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps,
                                        int nx, int ny, const int32_t *d_src_xy,
                                        const int32_t *d_src_map, int64_t npairs,
                                        double threshold, uint32_t *d_out_bits);
/* The same thresholded visibility as ROW RUNS: the visible set of row y of pair p,
 * {x : visibility_(x, y) >= threshold}, as its sorted transition columns t0 < t1 < ... -- visible on
 * [t0, t1), [t2, t3), ...; a run that reaches the last cell ends at nx, so every row holds an even
 * number of columns.  A visibility polygon crosses a row a handful of times: 6 bytes per row on an
 * empty 1000 x 1000 map against 125 bytes of bits and 4000 bytes of fp32, which takes the host-buffer
 * call off the box's PCIe / host-memory path (bench.py: e2e.runs).  A caller can test a cell by a binary
 * search in its row, or rebuild the bit map with vhp_runs_to_bits.
 *   row_count[p * ny + y]  number of transition columns of the row (uint16)
 *   pair_ptr[p]            index into trans of the first column of pair p; pair_ptr[npairs] = total
 *   trans[...]             the columns, rows of a pair back to back (uint16; nx <= 16384)
 * trans_cap = capacity of trans in elements; the call fails with VHP_ERR_INVALID_ARG and *trans_used =
 * the elements needed (so far) when it is too small.  Decided on the fp64 value like the bit form. */
vhp_status vhp_visibility_batch_runs(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx,
                                     int ny, const int32_t *src_xy, const int32_t *src_map,
                                     int64_t npairs, double threshold, uint16_t *row_count,
                                     uint64_t *pair_ptr, uint16_t *trans, int64_t trans_cap,
                                     int64_t *trans_used);
/* host utility: row runs -> bit maps (the layout of vhp_visibility_batch_bin) */
vhp_status vhp_runs_to_bits(const uint16_t *row_count, const uint64_t *pair_ptr, const uint16_t *trans,
                            int64_t npairs, int nx, int ny, uint32_t *out_bits);

/* Merged visibility of SETS of light sources: ngroups groups, group g = sources
 * [group_ptr[g], group_ptr[g+1]) of src_xy (group_ptr[0] = 0, non-decreasing), all on map
 * group_map[g] (NULL -> map 0).  For every cell, over the group's sources k = 0, 1, ... (index
 * WITHIN the group; duplicates count as separate entries):
 *   vmax[g][y][x]   max_k of the field vhp_visibility_batch returns for source k (dtype; VHP_F32 =
 *                   the fp64 maximum rounded once)          -- visibility_global_ after those sweeps
 *   first[g][y][x]  smallest k whose sweep writes the cell with fp64 value >= threshold,
 *                   VHP_NO_PARENT if none                   -- cameFrom_ after those sweeps
 *   count[g][y][x]  number of k whose sweep writes the cell with fp64 value >= threshold
 * "writes": every cell except source k's never-written border (column 0 unless sx == 0, row 0
 * unless sy == 0).  Any output pointer may be NULL; at least one must be given.  The call writes
 * every cell of the outputs it is given (empty groups: 0 / VHP_NO_PARENT / 0).
 * Instead of K full fields per group, the sweeps fold straight into the group's outputs with
 * atomics where the batched tile kernel runs and threshold > 0 (a dark cell costs no store); any
 * other case (threshold <= 0, a few sweeps of a large map, the naive kernel) sweeps chunks of fields
 * and folds them, with the same result.  Errors (VHP_ERR_INVALID_ARG): a source outside the grid,
 * group_map out of range, group_ptr not starting at 0, decreasing, or a group of 2^31 sources or
 * more, a NaN threshold, no output.  In the _dev form nsrc = group_ptr[ngroups] sizes the launch;
 * a bad source or group layout is reported like an out-of-grid source of vhp_visibility_batch_dev
 * (by the next synchronising call). */
typedef struct vhp_merge_out {
  void *vmax;
  int32_t *first;
  uint32_t *count;
} vhp_merge_out;
vhp_status vhp_visibility_merge_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                      const int32_t *src_xy, const int64_t *group_ptr,
                                      const int32_t *group_map, int64_t ngroups, double threshold,
                                      vhp_dtype dtype, const vhp_merge_out *out);
vhp_status vhp_visibility_merge_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                          int ny, const int32_t *d_src_xy, const int64_t *d_group_ptr,
                                          const int32_t *d_group_map, int64_t ngroups, int64_t nsrc,
                                          double threshold, vhp_dtype dtype, const vhp_merge_out *d_out);

/* Range-limited merged visibility: what a set of sensors with sensing radius R covers together.  Inputs, group
 * layout, outputs, dtype rules and errors are those of vhp_visibility_merge_batch, except that source k only
 * contributes to the cells (x, y) in its range, dx = x - sx, dy = y - sy:
 *   VHP_RANGE_BOX   |dx| <= R and |dy| <= R        (the cells of its vhp_visibility_window_batch window)
 *   VHP_RANGE_DISK  dx*dx + dy*dy <= R*R           (integer arithmetic)
 *   vmax[g][y][x]   max_k of (source k's field where the cell is in k's range, else 0)
 *   first / count   the merge's "writes" rule narrowed to the range: the cell is in k's range, not on k's
 *                   never-written border, and has fp64 value >= threshold
 * Every in-range value equals the full field's (the box is closed under "upstream", the disk lies inside it), so
 * VHP_RANGE_BOX with R >= max(nx, ny) - 1 is bit-identical to vhp_visibility_merge_batch, and R = 0 covers the
 * source cells only.  Where threshold > 0 and the box fits one CTA of the batched tile kernel (maps up to
 * 16384 x 16384 with small R), the sweeps of the boxes fold straight into the group outputs and dark cells cost
 * nothing; otherwise chunks of fp64 windows (vhp_visibility_window_batch's routes) are folded, with the same
 * result.  Additional errors (VHP_ERR_INVALID_ARG): radius outside [0, 16383], a shape other than the two. */
typedef enum vhp_range_shape { VHP_RANGE_BOX = 0, VHP_RANGE_DISK = 1 } vhp_range_shape;
vhp_status vhp_visibility_merge_range_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                            const int32_t *src_xy, const int64_t *group_ptr,
                                            const int32_t *group_map, int64_t ngroups, int32_t radius,
                                            int32_t shape, double threshold, vhp_dtype dtype,
                                            const vhp_merge_out *out);
vhp_status vhp_visibility_merge_range_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                                int ny, const int32_t *d_src_xy, const int64_t *d_group_ptr,
                                                const int32_t *d_group_map, int64_t ngroups, int64_t nsrc,
                                                int32_t radius, int32_t shape, double threshold,
                                                vhp_dtype dtype, const vhp_merge_out *d_out);

/* Greedy sensor placement: which k of a set of candidate positions cover the most cells together.  nprob
 * independent problems in the CSR layout of vhp_visibility_merge_batch: problem q has the candidates
 * [group_ptr[q], group_ptr[q+1]) of cand_xy on map group_map[q] (NULL -> map 0); radius R, shape and threshold as in
 * vhp_visibility_merge_range_batch.
 *   S(c)  the cells where candidate c would add 1 to vhp_visibility_merge_range_batch's count: in range, not on c's
 *         never-written border, fp64 value of vhp_visibility_batch's field >= threshold
 *   T_q   the cells whose bit is set in target ([prob][ny][ceil(nx/32)] uint32, the layout of
 *         vhp_visibility_batch_bin; bits beyond nx are ignored); NULL: every cell.  "Add k sensors to those already
 *         placed" is the complement of their coverage as the target.
 * Greedy, U = {} and for r = 0 .. k-1: gain(c) = |S(c) & T_q \ U| for every candidate of the problem; p = argmax,
 * ties to the smallest index within the group; if gain(p) == 0 stop (npicked = r), else U |= S(p).  Duplicates are
 * separate entries.  Every decision is an integer comparison, so the result is exact.  Outputs (any may be NULL, at
 * least one must be given):
 *   pick[q][r]     index within the group of the r-th pick, -1 from npicked on            (int32 [prob][k])
 *   gain[q][r]     cells the r-th pick newly covers, 0 from npicked on; non-increasing    (uint32 [prob][k])
 *   npicked[q]                                                                            (int32 [prob])
 *   covered[q]     U after the last pick, every cell of the union (in the target or not), bits beyond nx 0
 *                  ([prob][ny][ceil(nx/32)] uint32) = count > 0 of vhp_visibility_merge_range_batch on the picks
 * so sum of gain = |U & T|.  Within (1 - 1/e) of the best k-subset.
 * Routes.  Phase 1 stores each candidate's S(c) as bits over its box clipped to the grid: min(2R+1, ny) rows and
 * min(ceil(nx/32), (2R+31)/32 + 1) words aligned to the map's 32-column words.  Where threshold > 0 and the box fits one
 * CTA of the batched tile kernel, the sweep of each box writes those bits itself; otherwise (threshold <= 0, the naive
 * kernel, grid mode 2, boxes too large) chunks of fp64 windows, or whole fields where a window would be larger than the
 * map, are thresholded into them.  Phase 2 runs min(k, nsrc) rounds of two kernels each on the device with no host
 * synchronisation: one takes every problem's pick, one updates exactly the gains of the candidates whose box meets it.
 * Workspace (device, grown on demand and kept by the context): 4 * nsrc * rows * words bytes of candidate bits, plus
 * 4 * ny * ceil(nx/32) + 4 * rows * words bytes per problem; the host form runs problems in batches that fit 4 GB
 * (at least one problem).  A failed allocation returns VHP_ERR_CUDA and names the bytes.
 * Errors (VHP_ERR_INVALID_ARG): those of vhp_visibility_merge_range_batch (radius outside [0, 16383], an unknown
 * shape, a NaN threshold, a candidate outside the grid, a bad group layout, group_map out of range), k < 0, no
 * output.  k == 0 is valid (npicked 0, covered all zero).  The _dev form takes nsrc = group_ptr[nprob] and reports a
 * bad candidate or group layout like vhp_visibility_merge_batch_dev, by the next synchronising call. */
typedef struct vhp_cover_out {
  int32_t *pick;
  uint32_t *gain;
  int32_t *npicked;
  uint32_t *covered;
} vhp_cover_out;
vhp_status vhp_visibility_cover_greedy_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                             const int32_t *cand_xy, const int64_t *group_ptr,
                                             const int32_t *group_map, int64_t nprob, int32_t k, int32_t radius,
                                             int32_t shape, double threshold, const uint32_t *target,
                                             const vhp_cover_out *out);
vhp_status vhp_visibility_cover_greedy_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                                 const int32_t *d_cand_xy, const int64_t *d_group_ptr,
                                                 const int32_t *d_group_map, int64_t nprob, int64_t nsrc, int32_t k,
                                                 int32_t radius, int32_t shape, double threshold,
                                                 const uint32_t *d_target, const vhp_cover_out *d_out);

/* Weighted greedy sensor placement: which k candidates cover the most summed importance together.  Problems,
 * candidates, group_map, radius, shape, threshold and S(c) are exactly those of vhp_visibility_cover_greedy_batch.
 *   W_q   weights ([prob][ny][nx] uint8, unpadded, no alignment needed): the importance W_q(x) in [0, 255] of cell x
 *         to problem q; NULL: every cell weighs 1.
 * Greedy, U = {} and for r = 0 .. k-1: gain(c) = sum of W_q(x) over x in S(c) \ U for every candidate of the problem;
 * p = argmax, ties to the smallest index within the group; if gain(p) == 0 stop (npicked = r), else U |= S(p).
 * Duplicates are separate entries.  Every gain is an exact integer sum and every decision an integer comparison, so
 * the result does not depend on the order of atomics or blocks.  Outputs (any may be NULL, at least one must be given):
 *   pick[q][r]     index within the group of the r-th pick, -1 from npicked on            (int32 [prob][k])
 *   gain[q][r]     summed weight the r-th pick newly covers, 0 from npicked on            (uint64 [prob][k])
 *   npicked[q]                                                                            (int32 [prob])
 *   covered[q]     U after the last pick, every cell of the union whatever its weight, bits beyond nx 0
 *                  ([prob][ny][ceil(nx/32)] uint32)
 * so sum of gain = sum of W over U, gains are non-increasing, and the result is within (1 - 1/e) of the best k-subset
 * (weighted coverage is monotone submodular).  There is no target: weights in {0, 1} are the target of
 * vhp_visibility_cover_greedy_batch (and give its result), and "add k sensors to those already placed" is weights
 * zeroed on their coverage.
 * Gains fit 36 bits (at most 2^28 cells of weight 255), which leaves 28 bits of the 64-bit argmax key for the index:
 * nsrc >= 2^28 is VHP_ERR_INVALID_ARG (the nsrc argument of the _dev form, group_ptr[nprob] of the host form),
 * checked before any candidate is read.
 * Routes and phase 1 are those of vhp_visibility_cover_greedy_batch; the rounds also read a copy of the weights in
 * 32-byte rows per 32-column word.  Workspace: that of vhp_visibility_cover_greedy_batch, plus 4 * nsrc bytes (uint64
 * gains) and 32 * ny * ceil(nx/32) bytes per problem; the host form's 4 GB batches also count each problem's ny * nx
 * weight bytes.  Errors (VHP_ERR_INVALID_ARG): those of vhp_visibility_cover_greedy_batch, and the 2^28 limit.
 * k == 0 is valid. */
typedef struct vhp_cover_weighted_out {
  int32_t *pick;
  uint64_t *gain;
  int32_t *npicked;
  uint32_t *covered;
} vhp_cover_weighted_out;
vhp_status vhp_visibility_cover_greedy_weighted_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                                      const int32_t *cand_xy, const int64_t *group_ptr,
                                                      const int32_t *group_map, int64_t nprob, int32_t k,
                                                      int32_t radius, int32_t shape, double threshold,
                                                      const uint8_t *weights, const vhp_cover_weighted_out *out);
vhp_status vhp_visibility_cover_greedy_weighted_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                                          int ny, const int32_t *d_cand_xy,
                                                          const int64_t *d_group_ptr, const int32_t *d_group_map,
                                                          int64_t nprob, int64_t nsrc, int32_t k, int32_t radius,
                                                          int32_t shape, double threshold, const uint8_t *d_weights,
                                                          const vhp_cover_weighted_out *d_out);

/* Redundant (m-fold) greedy sensor placement: which k candidates see the most summed importance, where a cell counts
 * until m of the picks cover it (coverage that survives a failed sensor, two or three views of a target, overlapping
 * camera views).  Problems, candidates, group_map, radius, shape, threshold, S(c) and the weights W_q (NULL: every
 * cell weighs 1) are exactly those of vhp_visibility_cover_greedy_weighted_batch.  m in [1, 255].
 *   f(A) = sum over x of W_q(x) * min(cnt_A(x), m), cnt_A(x) = the number of picks in A whose S covers x
 * Greedy, A = {} and every cnt 0, for r = 0 .. k-1: gain(c) = sum of W_q(x) over x in S(c) with cnt(x) < m for every
 * candidate of the problem not yet picked; p = argmax, ties to the smallest index within the group; if gain(p) == 0
 * stop (npicked = r), else cnt += 1 over S(p), saturating at m.  A candidate is picked at most once.  Duplicates are
 * separate entries, so with m >= 2 two identical candidates can both be picked.  Every gain is an exact integer sum and
 * every decision an integer comparison.  Outputs (any may be NULL, at least one must be given):
 *   pick[q][r]     index within the group of the r-th pick, -1 from npicked on            (int32 [prob][k])
 *   gain[q][r]     summed weight the r-th pick adds to f, 0 from npicked on               (uint64 [prob][k])
 *   npicked[q]                                                                            (int32 [prob])
 *   count[q]       min(m, number of picks whose S covers the cell), every cell whatever its weight
 *                  ([prob][ny][nx] uint8) = min(m, count) of vhp_visibility_merge_range_batch on the picks
 * so gains are non-increasing, sum of gain = sum over x of W_q(x) * count(x), and the result is within (1 - 1/e) of
 * the best k-subset (f is monotone submodular).  m = 1 gives exactly the pick, gain and npicked of
 * vhp_visibility_cover_greedy_weighted_batch, and count is its covered unpacked.  There is no target: weights in
 * {0, 1} are the target.
 * Routes, phase 1 and the 2^28 limit are those of vhp_visibility_cover_greedy_weighted_batch; the rounds also keep a
 * uint8 counter per cell in 32-byte rows per 32-column word.  Workspace: that of
 * vhp_visibility_cover_greedy_weighted_batch plus 32 * ny * ceil(nx/32) bytes per problem; the host form's 4 GB batches
 * also count each problem's ny * nx count bytes.  Errors (VHP_ERR_INVALID_ARG): those of
 * vhp_visibility_cover_greedy_weighted_batch (the 2^28 limit checked before any candidate is read), m outside
 * [1, 255], no output.  k == 0 is valid (npicked 0, count all zero). */
typedef struct vhp_cover_mfold_out {
  int32_t *pick;
  uint64_t *gain;
  int32_t *npicked;
  uint8_t *count;
} vhp_cover_mfold_out;
vhp_status vhp_visibility_cover_greedy_mfold_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                                   const int32_t *cand_xy, const int64_t *group_ptr,
                                                   const int32_t *group_map, int64_t nprob, int32_t k, int32_t radius,
                                                   int32_t shape, double threshold, const uint8_t *weights, int32_t m,
                                                   const vhp_cover_mfold_out *out);
vhp_status vhp_visibility_cover_greedy_mfold_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                                       int ny, const int32_t *d_cand_xy, const int64_t *d_group_ptr,
                                                       const int32_t *d_group_map, int64_t nprob, int64_t nsrc,
                                                       int32_t k, int32_t radius, int32_t shape, double threshold,
                                                       const uint8_t *d_weights, int32_t m,
                                                       const vhp_cover_mfold_out *d_out);

/* Directional greedy sensor placement: cameras with a field of view, and fleets that mix sensing ranges.  Everything
 * is vhp_visibility_cover_greedy_mfold_batch (problems, candidates, group_map, radius R, shape, threshold, weights,
 * m, the greedy, ties, outputs, the 2^28 limit, k == 0), with each candidate's S(c) narrowed to its view:
 *   S_view(c) = S(c) & view(c)
 * views ([nsrc][5] int32) holds (r, ax, ay, bx, by) for each candidate.  Directions are in the grid's (x, y), x the
 * column and y the row: a positive cross(a, b) turns from increasing column towards increasing row, which is clockwise
 * on an image drawn with row 0 at the top.  With dx = x - sx, dy = y - sy, d = (dx, dy) and cross(u, v) = u.x * v.y - u.y * v.x (64-bit), view(c)
 * is the cells with
 *   range      the call's shape with radius r: |dx|, |dy| <= r (VHP_RANGE_BOX) or dx^2 + dy^2 <= r^2 (VHP_RANGE_DISK);
 *              0 <= r <= R, the call's radius (R still sets the box of the candidate bits and the workspace)
 *   direction  c1 = cross(a, d) and c2 = cross(d, b):
 *              cross(a, b) > 0 (the sector from a towards b is under 180 degrees): c1 >= 0 and c2 >= 0;
 *              cross(a, b) < 0, or cross(a, b) == 0 and dot(a, b) < 0 (180 degrees or more): c1 >= 0 or c2 >= 0;
 *              cross(a, b) == 0 and dot(a, b) > 0 (a and b point the same way, a == b included): every direction;
 *              d = (0, 0), the sensor's own cell, is always in it.
 * The sectors are defined by integer vectors alone, so the result is exact and order-independent.  Every view
 * omnidirectional (a == b) with r = R gives exactly vhp_visibility_cover_greedy_mfold_batch's pick, gain, npicked
 * and count.
 * Routes and phase 1 are those of vhp_visibility_cover_greedy_mfold_batch; one more kernel then masks each candidate's
 * bits in place, once, before the rounds.  Workspace: that of vhp_visibility_cover_greedy_mfold_batch; the host form
 * uploads the views with the candidates and its 4 GB batches also count each candidate's 20 view bytes.
 * Errors (VHP_ERR_INVALID_ARG): those of vhp_visibility_cover_greedy_mfold_batch; views NULL with nsrc > 0; a view
 * with r outside [0, R], a or b equal to (0, 0), or a component outside [-32767, 32767].  The host form checks the
 * views before any candidate is read.  The _dev form reports a bad view like a bad candidate, by the next
 * synchronising call with its own message, and that candidate covers nothing; with k == 0 or no problem the views
 * are not read. */
vhp_status vhp_visibility_cover_greedy_view_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                                  const int32_t *cand_xy, const int32_t *views,
                                                  const int64_t *group_ptr, const int32_t *group_map, int64_t nprob,
                                                  int32_t k, int32_t radius, int32_t shape, double threshold,
                                                  const uint8_t *weights, int32_t m, const vhp_cover_mfold_out *out);
vhp_status vhp_visibility_cover_greedy_view_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx,
                                                      int ny, const int32_t *d_cand_xy, const int32_t *d_views,
                                                      const int64_t *d_group_ptr, const int32_t *d_group_map,
                                                      int64_t nprob, int64_t nsrc, int32_t k, int32_t radius,
                                                      int32_t shape, double threshold, const uint8_t *d_weights,
                                                      int32_t m, const vhp_cover_mfold_out *d_out);

/* Quota sensor placement: the fewest greedy picks that reach a coverage target ("how few cameras cover 95 % of this
 * floor", "how many sensors until every doorway is seen twice"), with the rounds looping on the device.  The inputs
 * are those of vhp_visibility_cover_greedy_view_batch (problems, candidates, views, group_map, radius R, shape,
 * threshold, weights, m, the 2^28 limit), except that views may be NULL (every candidate omnidirectional with r = R:
 * the call is then vhp_visibility_cover_greedy_mfold_batch), k is kmax, and quota ([prob] uint64, in the units of f)
 * is new.  With f(A) = sum over x of W_q(x) * min(cnt_A(x), m), problem q runs that call's greedy and stops at the
 * first of:
 *   reached    the picks so far have total = sum of gain >= quota[q] (quota 0: no pick);
 *   exhausted  the argmax gain is 0 (everything coverable is counted);
 *   capped     kmax picks.
 * So npicked[q] = min { j : sum_{i<j} gain_i >= quota[q] }, limited by the other two, and since the greedy sequence is
 * the same for any k the result is exactly a prefix: pick, gain and npicked are those of the view call (views given) or
 * the m-fold call (views NULL) with k = kmax, cut at npicked[q], and count is that call's count with k = npicked[q].
 * Every decision is an integer comparison, so the result is exact and order-independent.  quota = UINT64_MAX and
 * kmax >= the group's size is greedy set cover of the coverable weight.  Outputs (any may be NULL, at least one must be
 * given):
 *   pick[q][r]     index within the group of the r-th pick, -1 from npicked on             (int32 [prob][kmax])
 *   gain[q][r]     what the r-th pick adds to f, 0 from npicked on, non-increasing         (uint64 [prob][kmax])
 *   npicked[q]                                                                             (int32 [prob])
 *   count[q]       min(m, number of picks whose S covers the cell)                         (uint8 [prob][ny][nx])
 *   total[q]       f(picks) = sum of gain; the quota is reached exactly when total >= quota (uint64 [prob])
 * Routes, phase 1 and the view mask are those of vhp_visibility_cover_greedy_view_batch.  The rounds are the body of a
 * CUDA-graph WHILE node, built, launched and destroyed by each call (each run of problems of the host form), that runs
 * until no problem is active or min(kmax, nsrc) rounds have run; the launch count does not depend on the quotas or on
 * the rounds run, and the _dev form does not synchronise.  Workspace: that of vhp_visibility_cover_greedy_mfold_batch
 * plus 16 bytes per problem (total and a copy of the quota) and two counters; the host form's 4 GB batches also count
 * each problem's 8 quota and 8 total bytes.  A failure to build the graph is VHP_ERR_CUDA with the CUDA message.
 * Errors (VHP_ERR_INVALID_ARG): those of vhp_visibility_cover_greedy_view_batch (sizes, NaN threshold, radius and
 * shape, m outside [1, 255], the 2^28 limit, bad views when views are given), kmax < 0, quota NULL with nprob > 0, no
 * output.  The host form checks them all before any candidate is read; the _dev form reports a bad view as the view
 * call does.  kmax == 0 is valid (npicked 0, count and total zero). */
typedef struct vhp_cover_quota_out {
  int32_t *pick;     /* [prob][kmax], -1 from npicked on */
  uint64_t *gain;    /* [prob][kmax], 0 from npicked on, non-increasing */
  int32_t *npicked;  /* [prob] */
  uint8_t *count;    /* [prob][ny][nx], min(m, picks covering the cell) */
  uint64_t *total;   /* [prob], f(picks) = sum of gain; reached <=> total >= quota */
} vhp_cover_quota_out;
vhp_status vhp_visibility_cover_quota_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                            const int32_t *cand_xy, const int32_t *views, const int64_t *group_ptr,
                                            const int32_t *group_map, int64_t nprob, int32_t kmax, int32_t radius,
                                            int32_t shape, double threshold, const uint8_t *weights, int32_t m,
                                            const uint64_t *quota, const vhp_cover_quota_out *out);
vhp_status vhp_visibility_cover_quota_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                                const int32_t *d_cand_xy, const int32_t *d_views,
                                                const int64_t *d_group_ptr, const int32_t *d_group_map, int64_t nprob,
                                                int64_t nsrc, int32_t kmax, int32_t radius, int32_t shape,
                                                double threshold, const uint8_t *d_weights, int32_t m,
                                                const uint64_t *d_quota, const vhp_cover_quota_out *d_out);

/* Budgeted sensor placement: what to buy and where it goes when candidates cost different amounts ("10 000 EUR,
 * cameras cost 300, lidars 1 800"), greedy by coverage per unit cost.  The inputs are those of
 * vhp_visibility_cover_quota_batch (problems, candidates, views (NULL: omnidirectional with r = R), group_map, radius
 * R, shape, threshold, weights, m, kmax, the 2^28 limit), except that quota may be NULL (no quota), and two are new:
 * cost ([nsrc] uint32, each in [1, 2^32 - 1], the cost of choosing the candidate in any unit) and budget ([prob]
 * uint64, UINT64_MAX: no budget).  With f(A) = sum over x of W_q(x) * min(cnt_A(x), m) and gain(c) what c adds to f,
 * problem q starts with spent = 0 and repeats
 *   eligible(c) = c not picked, gain(c) > 0, cost(c) <= budget[q] - spent;
 *   stop when no candidate is eligible, kmax picks are made, or (quota given) total >= quota[q];
 *   otherwise pick p = argmax over eligible c of gain(c) / cost(c) (an exact rational comparison, ties to the smallest
 *   index in the group), spent += cost(p), total += gain(p), and count the pick as the m-fold call does.
 * This is the cost-effective greedy of Khuller, Moss and Naor.  A candidate that stops fitting never fits again, so
 * the rule equals "consider by ratio, skip what does not fit".  The call also returns the best affordable singleton:
 * single[q] = argmax over c with cost(c) <= budget[q] of f({c}) (ties to the smallest index; -1 when no such c has a
 * positive gain) and single_gain[q] = f({single}).  max(total, single_gain) >= (1 - 1/e) / 2 * OPT for the monotone
 * submodular f (Khuller et al. prove 1 - 1/sqrt(e) for m = 1); the call returns both and does not choose.  All costs
 * 1 and budget B with quota NULL is exactly the view call (views given) or the m-fold call (views NULL) with
 * k = min(B, kmax); all costs 1 and budget UINT64_MAX is exactly the quota call.  The ratio is compared through the
 * 128-bit key (floor(gain * 2^64 / cost) << 28) | (2^28 - 1 - index), which orders exactly by ratio and then by
 * index for gains < 2^36 and costs < 2^32, so the result is exact and order-independent.  Outputs (any may be NULL,
 * at least one must be given):
 *   pick[q][r]     index within the group of the r-th pick, -1 from npicked on             (int32 [prob][kmax])
 *   gain[q][r]     what the r-th pick adds to f, 0 from npicked on; not monotone in general (uint64 [prob][kmax])
 *   npicked[q]                                                                             (int32 [prob])
 *   count[q]       min(m, number of picks whose S covers the cell)                         (uint8 [prob][ny][nx])
 *   total[q]       f(picks) = sum of gain                                                  (uint64 [prob])
 *   spent[q]       sum of the picks' costs, <= budget[q]                                   (uint64 [prob])
 *   single[q]      the best affordable singleton, -1: none                                 (int32 [prob])
 *   single_gain[q] its gain, 0: none                                                       (uint64 [prob])
 * Routes, phase 1, the view mask and the device loop (a CUDA-graph WHILE node per call) are those of the quota call;
 * the launch count is that call's plus one and does not depend on costs, budgets, quotas or the rounds run, and the
 * _dev form does not synchronise.  Workspace: that of the quota call plus 32 bytes per problem (a 16-byte slot, the
 * remaining budget and the spent cost); the host form's 4 GB batches also count 4 cost bytes per candidate and each
 * problem's budget and the outputs above.  Errors (VHP_ERR_INVALID_ARG): those of vhp_visibility_cover_quota_batch
 * except that quota may be NULL, cost NULL with nsrc > 0, budget NULL with nprob > 0, a zero cost.  The host form
 * checks them all before any candidate is read; the _dev form reports a bad view as the view call does, and a zero
 * cost by the next synchronising call (that candidate is never picked nor the singleton).  kmax == 0 is valid
 * (npicked 0, count, total and spent zero, single -1). */
typedef struct vhp_cover_budget_out {
  int32_t *pick;         /* [prob][kmax], -1 from npicked on */
  uint64_t *gain;        /* [prob][kmax], 0 from npicked on */
  int32_t *npicked;      /* [prob] */
  uint8_t *count;        /* [prob][ny][nx], min(m, picks covering the cell) */
  uint64_t *total;       /* [prob], f(picks) = sum of gain */
  uint64_t *spent;       /* [prob], sum of the picks' costs */
  int32_t *single;       /* [prob], the best affordable singleton, -1: none */
  uint64_t *single_gain; /* [prob], its gain */
} vhp_cover_budget_out;
vhp_status vhp_visibility_cover_budget_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                             const int32_t *cand_xy, const int32_t *views, const int64_t *group_ptr,
                                             const int32_t *group_map, int64_t nprob, int32_t kmax, int32_t radius,
                                             int32_t shape, double threshold, const uint8_t *weights, int32_t m,
                                             const uint64_t *quota, const uint32_t *cost, const uint64_t *budget,
                                             const vhp_cover_budget_out *out);
vhp_status vhp_visibility_cover_budget_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                                 const int32_t *d_cand_xy, const int32_t *d_views,
                                                 const int64_t *d_group_ptr, const int32_t *d_group_map, int64_t nprob,
                                                 int64_t nsrc, int32_t kmax, int32_t radius, int32_t shape,
                                                 double threshold, const uint8_t *d_weights, int32_t m,
                                                 const uint64_t *d_quota, const uint32_t *d_cost,
                                                 const uint64_t *d_budget, const vhp_cover_budget_out *d_out);

/* Directional merged visibility: what a set of cameras with headings and fields of view covers together, the
 * evaluation counterpart of vhp_visibility_cover_greedy_view_batch.  Everything is vhp_visibility_merge_range_batch
 * (inputs, groups, group_map, radius R, shape, threshold, dtype, the outputs and the "writes" rule), with source k's
 * range narrowed to its view, views[k] = (r, ax, ay, bx, by) ([nsrc][5] int32), by exactly the rule of
 * vhp_visibility_cover_greedy_view_batch (range r <= R in the call's shape, the sector of a and b by integer cross
 * products, the sensor's own cell always in it):
 *   vmax[g][y][x]   max_k of (source k's field where the cell is in view(k), else 0)
 *   first / count   the range merge's rule further narrowed to view(k)
 * Every view omnidirectional (a == b) with r = R gives exactly vhp_visibility_merge_range_batch's outputs.  For a
 * singleton group {c}, count is 1 exactly on S_view(c) of the view cover call, and min(m, count) over its picks is
 * that call's count.  Routes and launches are those of vhp_visibility_merge_range_batch; the host form uploads the
 * views with the sources.
 * Errors (VHP_ERR_INVALID_ARG): those of vhp_visibility_merge_range_batch; views NULL with nsrc > 0; a view with r
 * outside [0, R], a or b equal to (0, 0), or a component outside [-32767, 32767].  The host form checks the views
 * before any source is read.  The _dev form reports a bad view by the next synchronising call with its own message,
 * and that source contributes nothing; with no groups the views are not read. */
vhp_status vhp_visibility_merge_view_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                           const int32_t *src_xy, const int32_t *views, const int64_t *group_ptr,
                                           const int32_t *group_map, int64_t ngroups, int32_t radius, int32_t shape,
                                           double threshold, vhp_dtype dtype, const vhp_merge_out *out);
vhp_status vhp_visibility_merge_view_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                               const int32_t *d_src_xy, const int32_t *d_views,
                                               const int64_t *d_group_ptr, const int32_t *d_group_map,
                                               int64_t ngroups, int64_t nsrc, int32_t radius, int32_t shape,
                                               double threshold, vhp_dtype dtype, const vhp_merge_out *d_out);

/* Range-limited visibility: for every (map, source) pair the (2R+1) x (2R+1) window centred on the source,
 *   out[p][v][u] = visibility_(sx - R + u, sy - R + v) of vhp_visibility_batch for pair p where that cell lies
 *                  inside the grid, 0 where it does not                           (u, v in [0, 2R])
 * i.e. bit-identical to the crop of the full field (the sweep's dependencies point towards the source, so
 * the window depends on nothing outside it), never-written border included.  dtype as vhp_visibility_batch
 * (VHP_F32 = the fp64 value rounded once).  0 <= radius <= 16383.  Work and traffic per pair scale with the
 * window, not with the map: the batched tile kernel sweeps only the window, with its per-pair state sized by
 * the window, so range-limited batches on maps up to 16384 x 16384 run on it.  The naive kernel, grid mode 2
 * and windows too large for one CTA sweep whole fields and crop them, with the same result.
 * Errors (VHP_ERR_INVALID_ARG): a radius out of range, a null out, a source outside the grid, a map index out
 * of range; the _dev form reports the last two like vhp_visibility_batch_dev (by the next synchronising
 * call) and reuses the bit planes of vhp_prepare_maps_dev. */
vhp_status vhp_visibility_window_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx, int ny,
                                       const int32_t *src_xy, const int32_t *src_map, int64_t npairs,
                                       int32_t radius, vhp_dtype dtype, void *out);
vhp_status vhp_visibility_window_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps, int nx, int ny,
                                           const int32_t *d_src_xy, const int32_t *d_src_map, int64_t npairs,
                                           int32_t radius, vhp_dtype dtype, void *d_out);

/* ---- opt-in variants of the sweep (SURVEY 8f): the paper's MATLAB algorithm and the reference's
 * early-terminating queue variant.  Same layouts as vhp_visibility_batch.
 *   VHP_VARIANT_MATLAB  getAccessibilityMap.m (MATLAB_code/visibility/getAccessibilityMap.m:1-118):
 *       every cell v = alpha * (a - c*(a - b)) * occ with c = (j*fac)/i for i > j*fac, i/(j*fac) for
 *       j*fac > i, v = alpha * q(i-1, j-1) * occ where i == j*fac; the source holds
 *       light_strength * occ; every cell of the grid is computed (no never-written border).
 *       alpha = fac = light_strength = 1 is the reference's sweep with the diagonal taken from
 *       (i-1, j-1) -- what MATLAB and computeVisibilityUsingQueue (:750-751) do -- instead of the
 *       C++ sweep's (i, j-1) (SURVEY A.2 item 1).
 *   VHP_VARIANT_QUEUE   computeVisibilityUsingQueue() (src/visibilityBasedSolver.cpp:701-893, the
 *       variant README.md:13 recommends for dense maps) as an order-free rule: a free cell is
 *       computed iff a cell that pushes it holds more than `cutoff` (0.001 in the reference) or it
 *       touches the source; all other cells are 0; diagonal from (i-1, j-1); the source holds 1
 *       whatever its occupancy.  The reference's function is a FIFO search whose result depends
 *       on the queue order where a cell is reached before one of its upstream neighbours; this
 *       entry computes what the search computes when every upstream cell is visited first and is
 *       bit-identical to the compiled reference wherever that holds (about three maps in four of
 *       the random test family, tests/test_oracle_golden.py).
 * alpha, fac and light_strength are ignored by VHP_VARIANT_QUEUE, cutoff by VHP_VARIANT_MATLAB. */
typedef enum vhp_variant_model { VHP_VARIANT_MATLAB = 1, VHP_VARIANT_QUEUE = 2 } vhp_variant_model;
typedef struct vhp_sweep_variant {
  int32_t model;
  double alpha, fac, light_strength, cutoff;
} vhp_sweep_variant;
vhp_status vhp_visibility_variant_batch(vhp_context *ctx, const uint8_t *occ, int nmaps, int nx,
                                        int ny, const int32_t *src_xy, const int32_t *src_map,
                                        int64_t npairs, const vhp_sweep_variant *variant,
                                        vhp_dtype dtype, void *out);
vhp_status vhp_visibility_variant_batch_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps,
                                            int nx, int ny, const int32_t *d_src_xy,
                                            const int32_t *d_src_map, int64_t npairs,
                                            const vhp_sweep_variant *variant, vhp_dtype dtype,
                                            void *d_out);
/* Optional, for repeated _dev calls on the same maps: packs the maps into the
 * bit-plane layout the sweep kernel reads (row- and column-major bit maps, forward
 * and mirrored, plus a free-block summary) once, so later vhp_visibility_batch_dev calls with the same d_occ pointer,
 * nmaps, nx, ny skip the packing pass.  Invalidate by calling it again. */
vhp_status vhp_prepare_maps_dev(vhp_context *ctx, const uint8_t *d_occ, int nmaps,
                                int nx, int ny);
/* Forget the prepared maps: call it before the buffer behind d_occ is freed or rewritten (a later
 * allocation may get the same address). */
vhp_status vhp_release_maps_dev(vhp_context *ctx);

/* Result transport of the host-buffer calls (vhp_visibility_batch, vhp_raycast_batch).
 * Their results are far larger than what PCIe moves in the time the kernels need (16.4 GB per
 * 4096 sweeps of a 1000 x 1000 grid), and visibility fields are mostly flat (lit 1.0, shadow
 * 0.0).  In the packed transport the device classifies every 128-byte unit of a chunk of
 * results as uniform (all 0.0 / all 1.0) or literal; only the literal units and two bits of meta
 * data per unit cross PCIe (into pinned, 16-byte aligned memory the GPU stores the literal
 * units straight to their place), and host threads (env VHP_HOST_THREADS, default: all cores, at most 32) rebuild
 * the exact bytes in `out`.  `out` is bit-identical either way.
 *   mode 0  plain: chunked device-to-host copies straight into `out`
 *   mode 1  automatic (default): packed for results of 64 MB and more, plain for the rest of
 *           a call whose first chunk is more than 60 % literal
 *   mode 2  always packed
 * env VHP_RESULT_TRANSPORT=plain|packed sets the mode at context creation.
 * vhp_context_last_transport reports the last host-buffer call: bytes moved device-to-host,
 * bytes of results delivered, transport used (0 plain, 1 packed with a staged literal stream,
 * 2 packed with literal units stored straight into the pinned caller buffer). */
vhp_status vhp_context_set_result_transport(vhp_context *ctx, int mode);
/* Packed transport into pinned memory: besides the literal units the GPU can deliver
 * `sixteenths`/16 of the result completely (uniform units included) while the host threads
 * write the rest.  Default 0 (measured fastest where the host has 16 threads: bytes arriving
 * over PCIe compete with the host threads for the same memory system); a host with few
 * threads per GPU may prefer a larger share.  env VHP_RESULT_GPU_SHARE. */
vhp_status vhp_context_set_result_gpu_share(vhp_context *ctx, int sixteenths);
vhp_status vhp_context_last_transport(const vhp_context *ctx, int64_t *d2h_bytes,
                                      int64_t *result_bytes, int32_t *packed);
/* The host half of the packed transport on its own (no GPU needed; tests): expand one packed
 * chunk into dst[0 .. valid_bytes) with `threads` host threads.  Unit u (128 bytes; the last
 * one may be partial) is literal iff bit u % 32 of mask[u / 32]; the literal units of mask
 * word w lie back to back from literals + 128 * word_base[w]; a uniform unit is all 0.0 or,
 * where bit u % 32 of vmask[u / 32] is set, all 1.0 (elements of elem_bytes = 4 or 8 bytes: fp32 /
 * fp64; units of equal elements of any other value are literal).  literals == NULL is the direct mode: the
 * literal units are taken to be in dst already (the device stored them there) and are left
 * untouched; only the uniform units are written. */
vhp_status vhp_expand_packed_chunk(const uint32_t *mask, const uint32_t *word_base,
                                   const uint32_t *vmask, int elem_bytes, const void *literals,
                                   int64_t nunits, int64_t valid_bytes, void *dst, int threads);

/* The lazy form of the same expansion (what vhp_packed_expand runs per chunk): bytes [b0, b1) of the
 * chunk -> out[0 .. b1 - b0), single-threaded; b0 a multiple of elem_bytes, literals not NULL. */
vhp_status vhp_expand_packed_range(const uint32_t *mask, const uint32_t *word_base,
                                   const uint32_t *vmask, int elem_bytes, const void *literals,
                                   int64_t nunits, int64_t valid_bytes, int64_t b0, int64_t b1,
                                   void *out);

/* ---- a5: batched ray casting (raycasting + the all-targets loop) -------------
 * out[p][y][x] = visibilityRayCasting_ after the loop of benchmark() :228-232 on
 * a field initialised to 1.0 (reset() :45). */
vhp_status vhp_raycast_batch(vhp_context *ctx, const uint8_t *occ, int nmaps,
                             int nx, int ny, const int32_t *src_xy,
                             const int32_t *src_map, int64_t npairs,
                             vhp_dtype dtype, void *out);
vhp_status vhp_raycast_batch_dev(vhp_context *ctx, const uint8_t *d_occ,
                                 int nmaps, int nx, int ny,
                                 const int32_t *d_src_xy,
                                 const int32_t *d_src_map, int64_t npairs,
                                 vhp_dtype dtype, void *d_out);

/* ---- a2-a4: batched planner (solve + reconstructPath) ------------------------
 * nprob independent problems; problem q uses map prob_map[q] (NULL -> map 0),
 * start (se_xy[4q], se_xy[4q+1]) and end (se_xy[4q+2], se_xy[4q+3]).
 * The whole loop of solve() (:127-140) runs on the device: sweep with fused
 * max-merge / first-writer parents / arg-min of h in heap push order, next
 * source selection, end-visible test and max_iter check, with no host round trip.
 * Outputs (any pointer may be NULL to skip it):
 *   status[q]        vhp_status of problem q (0..5)
 *   nb_sources[q]    nb_of_sources_ when solve() returned
 *   light_sources    [q][ls_cap][2] int32: lightSources_[0..nb] (entry nb = end on
 *                    VHP_OK, :141); ls_cap must be >= max_iter + 2
 *   path_len[q]      reconstructPath() length (0 unless VHP_OK)
 *   path_n[q], path  [q][ls_cap][2] int32 start->end points
 *   vg               [q][ny][x] global visibility (dtype), came [q][ny][nx] int32
 *                    parents (VHP_NO_PARENT where the reference holds 1e15),
 *   vis              [q][ny][nx] local visibility of the last sweep (dtype) */
typedef struct vhp_planner_out {
  int32_t *status;
  int32_t *nb_sources;
  int32_t *light_sources;
  double *path_len;
  int32_t *path_n;
  int32_t *path;
  void *vg;
  int32_t *came;
  void *vis;
} vhp_planner_out;

vhp_status vhp_planner_batch(vhp_context *ctx, const uint8_t *occ, int nmaps,
                             int nx, int ny, const int32_t *se_xy,
                             const int32_t *prob_map, int64_t nprob,
                             double threshold, int32_t max_iter, int32_t ls_cap,
                             vhp_dtype dtype, const vhp_planner_out *out);
vhp_status vhp_planner_batch_dev(vhp_context *ctx, const uint8_t *d_occ,
                                 int nmaps, int nx, int ny,
                                 const int32_t *d_se_xy,
                                 const int32_t *d_prob_map, int64_t nprob,
                                 double threshold, int32_t max_iter,
                                 int32_t ls_cap, vhp_dtype dtype,
                                 const vhp_planner_out *d_out);

/* ---- e: ONE giant map, row-strip partitioned over several GPUs (SURVEY 8e) -------
 * Every rank holds the whole occupancy map (its bit planes are small) and the rows
 * [y0, y1) of the fp64 working fields.  A sweep from (sx, sy) visits the strips in order of
 * distance from the strip that holds the source; a strip needs, per quadrant, ONE fp64
 * visibility row of its neighbour on the source side as lower boundary (the "halo" row; the
 * -x and +x quadrants cut their tile rows at different offsets, hence one row each):
 *   vhp_strip_halo_rows   grid row needed per quadrant Q1..Q4 (-1: none; the quadrant
 *                         starts at the source or has no rows in [y0, y1))
 *   vhp_strip_sweep_dev   computeVisibility restricted to rows [y0, y1): d_halo[q] points
 *                         at the fp64 row vhp_strip_halo_rows named (indexed by x), d_vis_strip
 *                         is the strip buffer [(y1 - y0)][nx] of `dtype` (fp64 for the planner)
 *   vhp_strip_epilogue_dev  the per-cell planner epilogue of updateVisibility (:417-430)
 *                         over the strip + the strip's arg-min: d_best[0] = IEEE bits of the
 *                         smallest h (all ones: no candidate), d_best[1] = push-order key
 *                         quadrant << 40 | i << 20 | j relative to (sx, sy).  The global next
 *                         source is the lexicographic minimum of (d_best[0], d_best[1]) over
 *                         the ranks (an all-gather of 16 bytes per rank).
 * d_h_strip caches the heuristic per cell: initialise it to +inf, d_vg_strip to 0 and
 * d_came_strip to VHP_NO_PARENT.  visibility_heuristic_path_planner_b200/giant.py drives
 * these calls with torch.distributed (NCCL send/recv of the halo rows, all_gather of keys).
 * A strip sweep is one launch of ONE sweep: large windows (>= 2^20 cells) are spread over many
 * CTAs ("grid mode": tile rows handed out from a global counter, boundary rows and progress
 * flags in global memory), small ones run on a single CTA.  vhp_context_set_grid_sweep:
 * 0 = never, 1 = by size (default; env VHP_GRID_SWEEP overrides at context creation),
 * 2 = always (tests). */
void vhp_strip_halo_rows(int nx, int ny, int sx, int sy, int y0, int y1, int32_t rows[4]);
vhp_status vhp_context_set_grid_sweep(vhp_context *ctx, int mode);
vhp_status vhp_strip_sweep_dev(vhp_context *ctx, const uint8_t *d_occ, int nx, int ny,
                               int sx, int sy, int y0, int y1,
                               const double *const d_halo[4], vhp_dtype dtype,
                               void *d_vis_strip);
vhp_status vhp_strip_epilogue_dev(vhp_context *ctx, int nx, int ny, int y0, int y1,
                                  int sx, int sy, int ex, int ey, double threshold,
                                  int32_t nb, const int32_t *d_light_sources,
                                  const double *d_vis_strip, double *d_vg_strip,
                                  double *d_h_strip, int32_t *d_came_strip,
                                  uint64_t *d_best);

/* ---- e: the planner on ONE giant map over several GPUs, as one call (SURVEY 8e, BASELINE
 * configs[4]).  One process per GPU; every rank creates a handle for the same map and calls
 * vhp_giant_solve with the same arguments (collective, like an MPI call).  The map's rows are cut
 * into world * strips_per_rank contiguous strips, rank r owns strips [r * spr, (r + 1) * spr).
 * Per planner iteration (updateVisibility :379-565 + the loop of solve() :127-140):
 *   - two chains of strip sweeps, the +y quadrants upwards and the -y quadrants downwards, on two
 *     streams.  With one strip per rank the ranks map each other's sweep workspaces (CUDA IPC) and
 *     a boundary is handed over tile by tile by peer stores over NVLink from inside the sweep
 *     kernel, so the strips of a chain run as one wavefront; otherwise (several strips per rank,
 *     no peer mapping, env VHP_GIANT_P2P=0) neighbours exchange 2 x nx doubles per chain with
 *     ncclSend / ncclRecv;
 *   - epilogue + arg-min per strip, ncclAllGather of 32 bytes per rank {h bits, push-order key,
 *     vg(end) bits}; every rank takes the lexicographic minimum = priority_queue::top()'s
 *     first-pushed tie-break and runs the loop control on the device.
 * The loop state lives in device memory and no launch argument depends on it: one process
 * captures the iteration as the body of a CUDA-graph WHILE node; several ranks enqueue
 * iterations in batches, reading a snapshot of the loop state one batch behind.  Either way the
 * GPU never waits for the host between the first sweep and reconstructPath.
 * Results are bit-identical to vhp_planner_batch on one GPU (tests/test_gpu_giant.py,
 * tests/test_gpu_giant_multirank.py).  NCCL is bound at run time (dlopen of libnccl.so.2, env
 * VHP_NCCL_LIB overrides); world == 1 needs none.
 *   vhp_giant_unique_id   rank 0: 128 bytes (an ncclUniqueId) to hand to every rank by any side
 *                         channel (a file, MPI, torch.distributed broadcast ...)
 *   vhp_giant_create      occ: host uint8 [ny][nx], the whole map on every rank; id: NULL if world == 1
 *   vhp_giant_solve       se_xy = {start x, start y, end x, end y}; `out` as in vhp_planner_batch
 *                         for ONE problem, host pointers, any may be NULL; the fields vg / came /
 *                         vis receive THIS rank's rows (vhp_giant_local_rows) as fp64 / int32
 *                         [rows][nx]; dtype must be VHP_F64 when vg or vis is requested
 *   vhp_giant_set_loop_mode  0 automatic (default), 1 CUDA-graph WHILE node (one process only),
 *                         2 batches of `batch` iterations (0: keep; default 4), 3 one read-back per
 *                         iteration (for comparisons).  env VHP_GIANT_LOOP / VHP_GIANT_BATCH. */
#define VHP_GIANT_ID_BYTES 128
typedef struct vhp_giant vhp_giant;
typedef struct vhp_giant_stats {
  int32_t iterations;       /* sweeps run (= nb_of_sources unless the fixed point was fast-forwarded) */
  int32_t loop_mode;        /* 1 graph, 2 batches, 3 read-back per iteration */
  double solve_ms;          /* host wall time of the call */
  double loop_ms;           /* device time of the loop (CUDA events on the main stream) */
  double nccl_ms;           /* device time between the events around this rank's NCCL calls of the
                             * loop, waiting for the neighbour included (batches mode) */
  int64_t nccl_ops, nccl_ops_timed;
  int64_t halo_bytes_sent;  /* bytes this rank sent to its neighbours in the iterations that ran */
  int64_t launches;         /* kernels launched by the call */
  int32_t peer_handover;    /* 1: strip boundaries travelled tile by tile through peer memory (NVLink
                             * stores inside the sweep kernels), 0: as finished rows by ncclSend/Recv */
  int32_t reserved;
} vhp_giant_stats;
vhp_status vhp_giant_unique_id(void *id);
vhp_status vhp_giant_create(vhp_context *ctx, const uint8_t *occ, int nx, int ny, int rank,
                            int world, const void *id, int strips_per_rank, vhp_giant **out);
void vhp_giant_destroy(vhp_giant *g);
vhp_status vhp_giant_strip_bounds(const vhp_giant *g, int strip, int *y0, int *y1);
vhp_status vhp_giant_local_rows(const vhp_giant *g, int *y0, int *y1);
vhp_status vhp_giant_set_loop_mode(vhp_giant *g, int mode, int batch);
vhp_status vhp_giant_solve(vhp_giant *g, const int32_t *se_xy, double threshold,
                           int32_t max_iter, int32_t ls_cap, vhp_dtype dtype,
                           const vhp_planner_out *out, vhp_giant_stats *stats);
/* How vhp_planner_batch drives a single large problem (the "grid route"): 0 automatic = CUDA-graph
 * WHILE node, 2 batches, 3 one read-back per iteration (round-1 behaviour).  env VHP_GIANT_LOOP. */
vhp_status vhp_context_set_planner_loop(vhp_context *ctx, int mode);

/* widen int32 parents to the reference's Field<size_t> content (host arrays) */
void vhp_export_came_from_u64(const int32_t *came, int64_t n, uint64_t *out);

/* ---- host-side boundary: config, environment, files ---------------------------
 * struct Config of include/parser/parser.h:11-37, same fields and defaults. */
typedef struct vhp_config {
  int32_t mode;             /* 1 random environment, 2 image */
  int64_t ncols, nrows;     /* nx, ny */
  int64_t nb_of_obstacles;
  int64_t min_width, max_width, min_height, max_height;
  int32_t random_seed;      /* bool */
  int32_t seed_value;
  char image_path[1024];
  int32_t start_x, start_y, end_x, end_y;
  int64_t max_iter;
  double visibility_threshold;
  float light_strength;     /* parsed, unused (reference: lightStrength_ = 1.0) */
  /* save_results: 0 no; 1 yes; 2 yes, but vhp_solver_create does not write visibilityField.txt
   * again (the drop-in class rebuilds its handle before every solve()) */
  int32_t timer, save_results, save_local_visibility, save_came_from,
      save_light_sources, save_global_visibility, save_visibility_field, silent;
  int32_t ball_radius;
} vhp_config;

void vhp_config_default(vhp_config *cfg);
/* ConfigParser::parse (src/parser.cpp:12-338): same keys, validation, messages
 * and stdout echo.  Returns VHP_OK or VHP_ERR_IO / VHP_ERR_INVALID_ARG where the
 * reference returns false. */
vhp_status vhp_config_parse(const char *filename, vhp_config *cfg);

/* environment::generateNewEnvironmentFromSettings (src/environment.cpp:40-88),
 * glibc srand/rand stream, into occ[ny][nx] (uint8).  Returns the seed used. */
vhp_status vhp_environment_generate(const vhp_config *cfg, uint8_t *occ,
                                    int64_t *seed_used);
/* The same rectangle rule (src/environment.cpp:57-79) for a BATCH of maps, generated on the
 * device: d_occ[nmaps][ny][nx] (uint8, device memory), map k of the call is environment
 * first_map + k of the family `seed`.  The reference's draws are one sequential glibc rand()
 * stream per map; a batch needs independent ones, so draw d (0..3: col_1, width, row_1,
 * height) of obstacle o of map m is vhp_environment_draw(seed, m, o, d): SplitMix64's finaliser
 * over seed + 0x9E3779B97F4A7C15 * (m * 0x100000001B3 + 4 * o + d + 1), top 31 bits.  Uses
 * cfg->ncols, nrows, nb_of_obstacles, min/max_width, min/max_height only.  Asynchronous. */
uint32_t vhp_environment_draw(uint64_t seed, uint64_t map, uint64_t obstacle, uint32_t d);
vhp_status vhp_environment_generate_batch_dev(vhp_context *ctx, const vhp_config *cfg,
                                              uint64_t seed, int64_t first_map, int nmaps,
                                              uint8_t *d_occ);
/* environment::loadImage (src/environment.cpp:183-214): red channel == 255 ->
 * free.  Reads PNG (8-bit gray/RGB/RGBA/palette, non-interlaced) and binary
 * PGM/PPM.  First call with occ == NULL to get nx, ny. */
vhp_status vhp_environment_load_image(const char *filename, uint8_t *occ,
                                      int *nx, int *ny);

/* Solver handle: the drop-in for one vbs::visibilityBasedSolver instance. */
typedef struct vhp_solver vhp_solver;
/* ctor (:13-37).  occ is copied (uint8 [ny][nx]). */
vhp_status vhp_solver_create(vhp_context *ctx, const vhp_config *cfg,
                             const uint8_t *occ, int nx, int ny,
                             vhp_solver **out);
void vhp_solver_destroy(vhp_solver *s);
/* solve() (:76-160): same stdout lines (unless silent), same ./output files. */
vhp_status vhp_solver_solve(vhp_solver *s);
/* standAloneVisibility() (:165-189) and benchmark() (:194-262), benchmarkSeries()
 * (:295-374; n_sizes <= 60 limits the series, 0 = all 60). */
vhp_status vhp_solver_stand_alone_visibility(vhp_solver *s);
vhp_status vhp_solver_benchmark(vhp_solver *s);
vhp_status vhp_solver_benchmark_series(vhp_solver *s, int n_sizes);
/* results of the last solve()/benchmark() (host copies, fp64 like the reference) */
typedef enum vhp_field {
  VHP_FIELD_VISIBILITY = 0,        /* visibility_           double[ny][nx] */
  VHP_FIELD_VISIBILITY_GLOBAL = 1, /* visibility_global_    double[ny][nx] */
  VHP_FIELD_CAME_FROM = 2,         /* cameFrom_             int32 [ny][nx] */
  VHP_FIELD_RAYCASTING = 3,        /* visibilityRayCasting_ double[ny][nx] */
  VHP_FIELD_OCCUPANCY = 4          /* occupancyComplement_  uint8 [ny][nx] */
} vhp_field;
vhp_status vhp_solver_get_field(const vhp_solver *s, vhp_field which, void *dst);
int64_t vhp_solver_nb_of_sources(const vhp_solver *s);
/* lightSources_[0..nb] and the reconstructed path; return the number of points */
int64_t vhp_solver_light_sources(const vhp_solver *s, int32_t *xy, int64_t cap);
int64_t vhp_solver_path(const vhp_solver *s, int32_t *xy, int64_t cap,
                        double *length);
/* saveResults() (:1022-1178) into `dir` ("./output" in the reference) */
vhp_status vhp_solver_save_results(const vhp_solver *s, const char *dir);

#ifdef __cplusplus
}
#endif
#endif /* VHP_H */
