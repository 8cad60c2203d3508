// sweep_tile_body.cuh -- K1 as a tile wavefront: the CTA-wide device function behind
// the batched sweep kernel (kernels_sweep_tile.cu).
//
// Math (SURVEY A.5, reference src/visibilityBasedSolver.cpp:570-696).  In the local
// frame of one quadrant, i = |x - sx|, j = |y - sy|, cell q(i, j) is
//     i >  j ("column octant"): (a - c*(a - b)) * occ,  a = q(i-1, j), b = q(i-1, j-1), c = j/i
//     j >  i ("row octant")   : (a - c*(a - b)) * occ,  a = q(i, j-1), b = q(i-1, j-1), c = i/j
//     i == j > 0              : q(i, j-1) * occ        (the reference has no i == j branch)
//     i == j == 0             : 1 * occ
// with every operation rounded once (no FMA contraction).  Axis cells (i == 0 or
// j == 0) are the c == 0 case of the same formula: a - 0*(a - b) == a for any finite
// b, so the virtual cells outside the quadrant can hold any finite value; they hold
// 1.0 here, which also makes the source cell q(0,0) = q(0,-1) * occ = 1 * occ.
//
// Every dependency of a cell lies in {i-1, i} x {j-1, j}.  The quadrant is cut into
// tiles (I, J) by the same break points 0, a, a+32, a+64, ... along i and j, so that the
// diagonal only crosses the tiles I == J; the first tile row / column is a <= 32 wide,
// with a chosen per quadrant so that every other tile column starts on an absolute x
// that is a multiple of 32 (row stores are then whole, aligned 128-byte segments).
// Tile (I, J) needs the top row of (I, J-1), the right column of (I-1, J) and one
// corner cell of (I-1, J-1).  Tile rows are pipelines: a warp owns tile row J of a
// quadrant and walks I = 0, 1, ... keeping the right column and the corner in
// registers; the top row of every finished tile goes to shared memory (fp64),
//     rowE[q][i] = q(i, j_last)    top row of the newest tile above local column i,
// followed by a release store of the row's progress counter.  The warp of row J + 1
// acquires that counter before it starts tile I, so rows run skewed by one tile with
// no block barrier at all (the first kernels of this repo had one barrier per ring).
// Rows are dealt to the 8 warps of the CTA in (J, quadrant) order, which keeps the
// four quadrants in flight together and cannot deadlock: a row only ever waits for a
// row earlier in that order.
//
// A tile whose inputs all equal one value v and whose cells are all free is v
// everywhere (a - c*(a - b) with a == b is exactly a): it is written with plain
// 128-bit row stores and no arithmetic.  Likewise all-zero inputs, or an all-occupied
// tile, give zeros.  Everything else runs the 32-step recurrence, one cell per lane:
//     column-octant tile: lanes along j, steps along i, values staged in shared
//                         memory and written as rows afterwards;
//     row-octant tile   : lanes along i, steps along j, each step is one coalesced row;
//     diagonal tile     : both fronts plus the diagonal cell, staged.
// c = d/k is fma(d, rh, d*rl) with (rh, rl) a double-double 1/k (correctly rounded for
// 0 <= d < k <= 16384, verified exhaustively by vhp_selftest_ratio).
//
// Lit staircase.  With the virtual boundary at 1.0, tile (I, J) is 1.0 everywhere iff
// every tile of the rectangle [0..I] x [0..J] is free, so the provably lit region of a
// quadrant is a staircase: Lm(J) = min over J' <= J of the number of leading free tiles
// of tile row J'.  Before the wavefront starts, the CTA writes that region as long
// contiguous row spans (the -x and +x quadrants of a grid row merge into one span) and
// the wavefront skips those tiles; on an empty map the whole sweep is this pass.
//
// Whether a tile is free is first asked of a per-map summary (one bit per aligned
// 32 x 32 block, copied to shared memory): a tile inside free blocks needs no global
// load at all.  Otherwise occupancy comes from four bit planes per map (row / column
// major, forward / mirrored) so that a 32-cell window of any quadrant is one funnel
// shift of two words.  The cells the reference never writes (x == 0 in the -x
// quadrants, y == 0 in the -y quadrants, SURVEY A.2 item 2) are treated as occupied
// and stored as 0.  Axis cells shared by two quadrants are stored by the + quadrant.
//
// Window mode (strip partition of one giant map over several GPUs, SURVEY 8e).  A call
// may be restricted to the grid rows [y0, y1): per quadrant only the tile rows that
// intersect the window run, stores are clipped to the window, and the boundary row below
// the first tile row is not the virtual 1.0 but the fp64 visibility row the neighbouring
// strip computed (the "halo" row, one per quadrant because the -x and +x quadrants cut
// their tile rows at different offsets).  Rows of a tile row that lie outside the window
// are recomputed (at most 31) and not stored.
#ifndef VHP_SWEEP_TILE_BODY_CUH
#define VHP_SWEEP_TILE_BODY_CUH

#include <cstdint>
#include <type_traits>

#include "vhp_internal.h"
#include "sweep_common.cuh"

// Unroll factors of the 32-step loops.  Single-warp CTAs (small-map batches: 25+ independent
// warps per SM, each somewhere else in the code) are instruction-fetch bound beyond the
// 32 KB L1.5 instruction cache, so they unroll less (ncu: stall_no_instruction was the top
// stall of the 256x256 batch with 4x unrolling); multi-warp CTAs prefer the longer bodies.
#ifndef VHP_STEP_UNROLL
#define VHP_STEP_UNROLL 4
#endif
#ifndef VHP_STEP_UNROLL_1W
#define VHP_STEP_UNROLL_1W 2
#endif
#ifndef VHP_POLL_BACKOFF
#define VHP_POLL_BACKOFF 1
#endif
#ifndef VHP_POLL_NS0 // first and longest sleep of a warp that waits for the row below (ns)
#define VHP_POLL_NS0 32
#endif
#ifndef VHP_POLL_NSMAX
#define VHP_POLL_NSMAX 256
#endif
#ifndef VHP_DIAG_UNROLL
#define VHP_DIAG_UNROLL 1
#endif
#ifndef VHP_FILL_UNROLL
#define VHP_FILL_UNROLL 4
#endif
// The select-free step loops only run on full 32 x 32 tiles: a literal trip count lets the
// compiler drop the exit test (and the convergence check in front of the shuffle) per step.
#ifndef VHP_FIXED32
#define VHP_FIXED32 1
#endif
// Runs of dark tiles of a tile row written in one go (see run_row).
#ifndef VHP_DARK_TAIL
#define VHP_DARK_TAIL 1
#endif

namespace {

constexpr int kSkipPair = -0x7fffffff - 1; // source x of a pair the batched kernel leaves alone
constexpr int kDiagUnroll = VHP_DIAG_UNROLL, kFillUnroll = VHP_FILL_UNROLL;
constexpr int kTileWarps = 8;          // warps per CTA (default; small maps use fewer)
constexpr int kTile = 32;              // tile side
constexpr int kTileHdr = 256;          // shared-memory header: quadrant geometry (4 x TQuad), the row counter
                                       // (+240) and the export tile rows of grid mode (4 x int16, +244)
constexpr int kStagePitch = 33;        // staging tile pitch (elements)
constexpr int kWarpScratch = 136;      // doubles per warp: bottom stream [34] (row-octant tiles: new left
                                       // column), left stream [34], 1/k table of the tile [33 x double2]
constexpr unsigned kAll = 0xffffffffu;

struct TileArgs {
  VhpTilePlanes pl;
  int nx, ny;
  const int32_t *src_xy, *src_map;
  void *out;
  const double2 *rtab; // {RN(1/k), RN((1 - k*rh)*rh)}
  int *err;
  int vec;             // rows are 16-byte aligned: 128-bit stores allowed
  // window mode: rows [win_y0, win_y1) only (whole grid: 0, ny); halo[q] = the fp64
  // visibility row (indexed by x) just below the first tile row of quadrant q, or null
  int win_y0, win_y1;
  const double *halo[4] = {nullptr, nullptr, nullptr, nullptr};
  // grid mode (one sweep spread over many CTAs): boundary rows, staircase, row progress and
  // the row counter live in global memory (null otherwise)
  double *g_edges = nullptr;
  int *g_lm = nullptr, *g_prog = nullptr, *g_next_row = nullptr;
  // quadrants to run, bit q = Q(q+1) (0xF: all).  The strip-partitioned planner sweeps the +y
  // quadrants (Q1, Q2) and the -y quadrants (Q3, Q4) of a strip as two launches: the two
  // directions travel along the strips independently of each other.
  int qmask = 0xF;
  // kFmtMergeView*: the call's shape is the disk (in the padding in front of src_ctl, so that no other member moves)
  int m_disk = 0;
  // window / grid kernels only: {done, sx, sy, ...} in device memory.  Non-null: the source comes
  // from there and the launch is a no-op once `done` is set, so a planner iteration can be
  // enqueued (or captured in a CUDA graph) before the host knows the next source.
  // kFmtMergeView* (the batched tile kernel, which never reads src_ctl): the views [pair][5] = (r, ax, ay, bx, by).
  union {
    const int *src_ctl = nullptr;
    const int32_t *m_views;
  };
  // grid mode across GPUs (strip-partitioned planner, one strip per rank): the boundary between
  // two strips is handed over tile by tile through peer memory instead of as a finished row.
  //   exporter: x_edges / x_prog = the boundary rows and progress flags of the NEIGHBOUR's
  //     workspace (a peer-mapped pointer, stores travel over NVLink); [x_y0, x_y1) = its window.
  //     The warp that owns the tile row just below the neighbour's first one copies every top row
  //     it finishes into the neighbour's boundary row and raises the neighbour's flag
  //     (system-scope fence + atomicMax), so the neighbour's first tile row runs one tile behind
  //     it, exactly like the next tile row on the same GPU, and the sweep's critical path does not
  //     grow with the number of strips;
  //   consumer: bit q of remote_mask = the boundary below quadrant q's first tile row arrives
  //     this way (its flag is raised with atomicMax by both sides, its boundary row is
  //     initialised only over the lit tiles, which nobody sends).
  double *x_edges = nullptr;
  int *x_prog = nullptr;
  int x_y0 = 0, x_y1 = 0;
  int remote_mask = 0;
  double thr = 0.0; // kFmtBits: bit = (fp64 value >= thr), thr > 0; kFmtMerge*: the count / first threshold
  // kFmtMerge*: the outputs of all groups ([group][ny][nx] each, any may be null) and the cells of one grid
  void *m_vmax = nullptr;
  int32_t *m_first = nullptr;
  uint32_t *m_count = nullptr;
  size_t m_cells = 0;
  const int32_t *m_pg = nullptr, *m_pk = nullptr; // per pair: group (-1: skip the pair) and index within it
  // kFmtWindow: radius R (windows of (2R+1)^2 per pair), block-summary words per window row (win_sum_words)
  // and the number of maps (a pair on another map is reported like a source outside the grid); kFmtMergeRange*:
  // R and w_sw, the sweep clipped to the box |dx|, |dy| <= R
  int w_r = 0, w_sw = 0, w_nmaps = 0;
  // kFmtMergeRange*: a cell of the box is in range iff dx^2 + dy^2 <= w_r2 (disk: R^2; box: 2 R^2, every cell)
  int w_r2 = 0;
};

// how tile_sweep_cta is used
constexpr int kSweepCta = 0;      // one CTA does the whole sweep (batches: one CTA per pair)
constexpr int kSweepGridInit = 1; // grid mode, first kernel (one CTA): staircase, boundary rows, flags
constexpr int kSweepGridWork = 2; // grid mode, second kernel (many CTAs): lit fill and tile rows

// geometry of one quadrant (shared memory, written once per sweep)
struct TQuad {
  int dirx, diry;   // +1 / -1
  int Ex, Ey;       // largest local i / j inside the grid
  int TX, TY;       // tile columns / rows (0: the quadrant does not exist)
  int rowOff;       // offset of rowE in the edge region (doubles)
  int psx, psy;     // plane coordinate of the source along x / y
  int a;            // width of the first tile row / column (1..32)
  int jw0, jw1;     // local rows j to store (window; whole quadrant: 0, Ey)
  int Jlo, Jhi;     // tile rows to run
};

__host__ __device__ inline int tile_row_of(const int a, const int j) {
  return j < a ? 0 : (j - a) / kTile + 1;
}

// Window geometry of quadrant q (Q1 (+,+), Q2 (-,+), Q3 (-,-), Q4 (+,-)) for a sweep from
// (sx, sy) restricted to rows [y0, y1): first tile row to run and the grid row whose fp64
// visibility is its lower boundary (-1: the quadrant has no rows in the window, or starts
// at the source).  Shared by the kernel and by the host-side exchange plan.
__host__ __device__ inline void tile_window_of(const int q, const int nx, const int ny, const int sx,
                                               const int sy, const int y0, const int y1, int *jw0,
                                               int *jw1, int *Jlo, int *Jhi, int *halo_y) {
  const int dirx = (q == 0 || q == 3) ? 1 : -1, diry = (q < 2) ? 1 : -1;
  const int Ey = diry > 0 ? ny - 1 - sy : sy;
  int a = dirx > 0 ? 32 - (sx & 31) : ((sx + 1) & 31);
  if (a == 0) a = 32;
  const bool exists = (dirx > 0 || sx > 0) && (diry > 0 || sy > 0);
  int lo = diry > 0 ? y0 - sy : sy - (y1 - 1), hi = diry > 0 ? y1 - 1 - sy : sy - y0;
  lo = lo < 0 ? 0 : lo;
  hi = hi > Ey ? Ey : hi;
  (void)nx;
  if (!exists || lo > hi) {
    *jw0 = 0; *jw1 = -1; *Jlo = 0; *Jhi = -1; *halo_y = -1;
    return;
  }
  *jw0 = lo; *jw1 = hi;
  *Jlo = tile_row_of(a, lo);
  *Jhi = tile_row_of(a, hi);
  *halo_y = *Jlo == 0 ? -1 : sy + diry * ((a + kTile * (*Jlo - 1)) - 1);
}

__host__ __device__ inline int tile_edge_doubles(int nx, int nwarps) {
  // per direction a quadrant has at most E/32 + 2 tile columns; two quadrants share each x
  // direction and the + and - extents add up to nx - 1.  A single-warp CTA sweeps one
  // quadrant after the other and reuses one boundary row.
  return nwarps == 1 ? kTile * ((nx - 1) / kTile + 2) : 2 * kTile * ((nx - 1) / kTile + 4);
}

// block summary: one bit per aligned 32 x 32 block, tile_sum_words(nx) words per block row
__host__ __device__ inline int tile_sum_words(int nx) { return (((nx + 31) >> 5) + 31) >> 5; }
__host__ __device__ inline int tile_sum_bytes(int nx, int ny) {
  return (4 * tile_sum_words(nx) * ((ny + 31) >> 5) + 15) & ~15;
}

// lit staircase Lm[q][J] and row progress prog[q][J]: tile_lm_cap(ny) entries per quadrant each
__host__ __device__ inline int tile_lm_cap(int ny) { return (ny - 1) / kTile + 4; }

// grid mode keeps the boundary rows in global memory
template <typename OutT>
__host__ __device__ inline size_t tile_smem_bytes_grid(int nx, int ny, int nwarps = kTileWarps) {
  return kTileHdr + tile_sum_bytes(nx, ny) + 32 * (size_t)tile_lm_cap(ny) +
         (size_t)nwarps * (kTile * kStagePitch * sizeof(OutT) + kWarpScratch * sizeof(double));
}

template <typename OutT>
__host__ __device__ inline size_t tile_smem_bytes(int nx, int ny, int nwarps = kTileWarps) {
  return kTileHdr + tile_sum_bytes(nx, ny) + 32 * (size_t)tile_lm_cap(ny) +
         sizeof(double) * (size_t)tile_edge_doubles(nx, nwarps) +
         (size_t)nwarps * (kTile * kStagePitch * sizeof(OutT) + kWarpScratch * sizeof(double));
}

// Range-limited sweeps (kFmtWindow): every dependency of a cell points towards the source, so the
// (2R+1)^2 window around it is swept on its own, in the map's absolute geometry (tile break points,
// bit planes, summary, never-written border), and the per-CTA state is sized by the window.
__host__ __device__ inline int win_side(int n, int R) { return n < 2 * R + 1 ? n : 2 * R + 1; }
// block-summary words per block row and block rows a window can touch
__host__ __device__ inline int win_sum_words(int nx, int R) {
  const int nbx = (nx + 31) >> 5, span = (2 * R + 31) / 32 + 1;
  const int b = nbx < span ? nbx : span, w = (b + 30) / 32 + 1;
  return tile_sum_words(nx) < w ? tile_sum_words(nx) : w;
}
__host__ __device__ inline int win_sum_rows(int ny, int R) {
  const int nby = (ny + 31) >> 5, span = (2 * R + 31) / 32 + 1;
  return nby < span ? nby : span;
}
__host__ __device__ inline int win_sum_bytes(int nx, int ny, int R) {
  return (4 * win_sum_words(nx, R) * win_sum_rows(ny, R) + 15) & ~15;
}
template <typename OutT>
__host__ __device__ inline size_t tile_smem_bytes_win(int nx, int ny, int R, int nwarps = kTileWarps) {
  return kTileHdr + win_sum_bytes(nx, ny, R) + 32 * (size_t)tile_lm_cap(win_side(ny, R)) +
         sizeof(double) * (size_t)tile_edge_doubles(win_side(nx, R), nwarps) +
         (size_t)nwarps * (kTile * kStagePitch * sizeof(OutT) + kWarpScratch * sizeof(double));
}

// 16-byte streaming store of one value replicated
__device__ __forceinline__ void stg16_fill(float *q, float v) {
  __stcs(reinterpret_cast<float4 *>(q), make_float4(v, v, v, v));
}
__device__ __forceinline__ void stg16_fill(double *q, double v) {
  __stcs(reinterpret_cast<double2 *>(q), make_double2(v, v));
}

// What a sweep stores.  kFmtValues: the field, one OutT per cell.  kFmtBits: one BIT per cell,
// bit (x & 31) of word [y][x >> 5] = (fp64 value >= TileArgs::thr), rows of (nx + 31) / 32 words,
// for thr > 0 and into a ZEROED buffer: cells below the threshold are not written at all, the
// words around the source column (shared by the -x and +x quadrants) are or-ed in atomically.
// kFmtMerge64 / kFmtMerge32: the sweep is folded into the outputs of its GROUP of sources (vhp_visibility_merge_batch):
// per cell with fp64 value v > 0, vmax = max(vmax, v) as an integer max on the bits (fp64, or fp32 of RN(v): non-negative
// IEEE values order like their bit patterns and rounding is monotone), and where v >= thr (> 0), first = min(first, k)
// and count += 1, k = the source's index within its group.  Cells of value 0 are not touched, which is why thr > 0.
// Other CTAs sweep sources of the same group at the same time, so every write is a relaxed atomic (red), never a
// plain store; count relies on the sweep storing each cell once (axis cells: the + quadrant only).  OutT is double
// (the staging tiles hold the fp64 values); `out` is only a base for cell indices.
// kFmtWindow: the field like kFmtValues, but only the (2R+1)^2 window around the source (TileArgs::w_r): each
// quadrant's extents are clipped to R, `out` is shifted so that cell (x, y) sits at out[y * (2R+1) + x], stores
// are scalar (window rows are not 16-byte aligned), and the window cells outside the grid are stored as 0.
// kFmtMergeRange64 / kFmtMergeRange32 (vhp_visibility_merge_range_batch): kFmtMerge* with the sweep clipped to the box
// |dx|, |dy| <= R like kFmtWindow (the box is closed under "upstream": its values are the full field's), cell indices
// in map pitch, and only the cells in range (TileArgs::w_r2) folded.
// kFmtCoverBits (vhp_visibility_cover_greedy_batch): kFmtBits's bit stores with kFmtMergeRange*'s clipped geometry, in
// the candidate's box layout (VhpCoverBox: rows of vhp_cover_words(nx, R) words, `out` shifted by the box origin, so
// the addressing is the whole-map bit layout's with another row pitch); only the box |dx|, |dy| <= R is stored, the
// disk is applied afterwards.
// kFmtMergeView64 / kFmtMergeView32 (vhp_visibility_merge_view_batch): kFmtMergeRange*, with only the cells of the box in
// the source's view (MergeView, TileArgs::m_views) folded.  The CTA's decoded view sits in kViewTail bytes after the
// layout of kFmtMergeRange* (the end of the dynamic shared memory), its key holding the source's cell index.
constexpr int kFmtValues = 0, kFmtBits = 2, kFmtMerge64 = 3, kFmtMerge32 = 4, kFmtWindow = 5, kFmtMergeRange64 = 6,
              kFmtMergeRange32 = 7, kFmtCoverBits = 8, kFmtMergeView64 = 9, kFmtMergeView32 = 10;
constexpr int kMergeHdr = 224; // shared-memory header: {group, k} of the CTA's source (int2)

constexpr int kViewTail = 16;  // kFmtMergeView*: shared-memory tail, the CTA's MergeView

// the sweep folds into group outputs (merge_cell), and it does so only within a range (and a view)
__host__ __device__ constexpr bool fmt_view(int f) { return f == kFmtMergeView64 || f == kFmtMergeView32; }
__host__ __device__ constexpr bool fmt_range(int f) {
  return f == kFmtMergeRange64 || f == kFmtMergeRange32 || fmt_view(f);
}
__host__ __device__ constexpr bool fmt_merge(int f) { return f == kFmtMerge64 || f == kFmtMerge32 || fmt_range(f); }
// clipped geometry: each quadrant's extents are clipped to R and the per-CTA state is sized by the box
// (tile_smem_bytes_win); the window output layout (pitch 2R+1, off-grid zeros) is kFmtWindow's alone
__host__ __device__ constexpr bool fmt_clip(int f) { return f == kFmtWindow || fmt_range(f) || f == kFmtCoverBits; }
// one bit per cell (v >= thr), into a zeroed buffer
__host__ __device__ constexpr bool fmt_bits(int f) { return f == kFmtBits || f == kFmtCoverBits; }

// fold value v of cell idx (y * nx + x) of this CTA's sweep into its group's outputs; (di, dj) = (|dx|, |dy|) of
// the cell from the source, for the range test of kFmtMergeRange*.  kFmtMergeView* recovers the signs from idx and
// the source's index s: with |dx| < nx, idx - s = dy * nx + dx is >= 0 exactly when dy >= 0 (dj > 0).
template <int FMT>
__device__ __forceinline__ void merge_cell(const TileArgs &p, const ptrdiff_t idx, const int di, const int dj,
                                           const double v) {
  if (!(v > 0.0)) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  if constexpr (fmt_view(FMT)) {
    uint32_t dsmem;
    asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dsmem));
    const int4 t = *reinterpret_cast<const int4 *>(smem_raw + dsmem - kViewTail);
    const int delta = (int)idx - (t.x & 0x7fffffff), dy = delta >= 0 ? dj : -dj;
    if (!merge_view_has(MergeView{t.x, t.y, t.z, t.w}, delta - dy * p.nx, dy)) return;
  } else if constexpr (fmt_range(FMT)) {
    if (di * di + dj * dj > p.w_r2) return;
  }
  const int2 gk = *reinterpret_cast<const int2 *>(smem_raw + kMergeHdr);
  const size_t o = (size_t)gk.x * p.m_cells + (size_t)idx;
  if (p.m_vmax) {
    if constexpr (FMT == kFmtMerge64 || FMT == kFmtMergeRange64 || FMT == kFmtMergeView64)
      red_max_u64(reinterpret_cast<unsigned long long *>(p.m_vmax) + o, (unsigned long long)__double_as_longlong(v));
    else
      red_max_u32(reinterpret_cast<uint32_t *>(p.m_vmax) + o, __float_as_uint(__double2float_rn(v)));
  }
  if (v >= p.thr) {
    if (p.m_first) red_min_u32(reinterpret_cast<uint32_t *>(p.m_first) + o, (uint32_t)gk.y);
    if (p.m_count) red_add_u32(p.m_count + o, 1u);
  }
}

// staging tile: element (row r, column c) of a 32 x 32 tile (odd pitch: column-wise writes
// and the row-wise read-out are both conflict-free)
__device__ __forceinline__ int stage_at(const int r, const int c) { return r * kStagePitch + c; }

// first local index and extent of tile column / row T
__device__ __forceinline__ int tile_start(const int a, const int T) {
  return T ? a + kTile * (T - 1) : 0;
}

// Last local column / row to compute: the extent without the never-written border (x == 0 in the
// -x quadrants, y == 0 in the -y quadrants).  A clipped sweep (CLIP) whose extent stops short of the
// grid's edge has no border cell.
template <bool CLIP = false>
__device__ __forceinline__ int ext_cx(const TQuad &g, const int sx) {
  return g.Ex - (g.dirx < 0 && (!CLIP || g.Ex == sx));
}
template <bool CLIP = false>
__device__ __forceinline__ int ext_cy(const TQuad &g, const int sy) {
  return g.Ey - (g.diry < 0 && (!CLIP || g.Ey == sy));
}

// Does the block summary prove every cell tile (I, J) has to compute is free?  (A tile
// with nothing to compute -- only border cells -- counts as free.)
template <bool CLIP = false>
__device__ __forceinline__ bool tile_sum_free(const TQuad &g, const uint32_t *bsum, const int nbw,
                                              const int sx, const int sy, const int I,
                                              const int J) {
  const int i0 = tile_start(g.a, I), j0 = tile_start(g.a, J);
  const int nvx = min(I ? kTile : g.a, ext_cx<CLIP>(g, sx) - i0 + 1);
  const int nvy = min(J ? kTile : g.a, ext_cy<CLIP>(g, sy) - j0 + 1);
  if (nvx <= 0 || nvy <= 0) return true;
  const int xa = sx + g.dirx * i0, xb = sx + g.dirx * (i0 + nvx - 1);
  const int ya = sy + g.diry * j0, yb = sy + g.diry * (j0 + nvy - 1);
  const int bx0 = min(xa, xb) >> 5, bx1 = max(xa, xb) >> 5;
  const int by0 = min(ya, yb) >> 5, by1 = max(ya, yb) >> 5;
  const uint32_t *s0 = bsum + by0 * nbw, *s1 = bsum + by1 * nbw;
  return ((s0[bx0 >> 5] >> (bx0 & 31)) & (s0[bx1 >> 5] >> (bx1 & 31)) &
          (s1[bx0 >> 5] >> (bx0 & 31)) & (s1[bx1 >> 5] >> (bx1 & 31)) & 1u) != 0u;
}

// row[xa..xb] = v by one warp (128-bit stores where the row is 16-byte aligned)
template <typename OutT>
__device__ __forceinline__ void fill_span(OutT *__restrict__ row, const int xa, const int xb,
                                          const OutT v, const int lane, const bool vec) {
  if (vec) {
    constexpr int EPL = 16 / (int)sizeof(OutT);
    for (int x = (xa & ~(EPL - 1)) + EPL * lane; x <= xb; x += 32 * EPL) {
      if (x >= xa && x + EPL - 1 <= xb) {
        stg16_fill(row + x, v);
      } else {
#pragma unroll
        for (int e = 0; e < EPL; ++e)
          if (x + e >= xa && x + e <= xb) __stcs(row + x + e, v);
      }
    }
  } else {
    for (int x = xa + lane; x <= xb; x += 32) __stcs(row + x, v);
  }
}

// q[0 .. n) = v by one warp, for any element-aligned q: scalar stores up to the first 16-byte boundary and
// after the last one, 128-bit stores in between (window rows, kFmtWindow, start anywhere)
template <typename OutT>
__device__ __forceinline__ void fill_run(OutT *__restrict__ q, const int n, const OutT v, const int lane) {
  constexpr int EPL = 16 / (int)sizeof(OutT);
  const int head = min(n, (int)((16 - ((uintptr_t)q & 15)) & 15) / (int)sizeof(OutT));
  if (lane < head) __stcs(q + lane, v);
  const int nv = (n - head) / EPL, t0 = head + nv * EPL;
  for (int k = lane; k < nv; k += 32) stg16_fill(q + head + k * EPL, v);
  if (t0 + lane < n) __stcs(q + t0 + lane, v);
}

// rows y0, y0 + dy, ... (nrows of them), columns [xa, xb] = v by one warp.  Short spans (a dark run
// of a few tiles) put several rows into one store instruction: per row a span costs its stores,
// not a loop set-up (fill_span row by row spent 16 % of the instructions of the dense-obstacle
// workload on the zeros of its dark runs).
template <typename OutT>
__device__ __forceinline__ void fill_block(OutT *__restrict__ out, const int nx, const int y0, const int dy,
                                           const int nrows, const int xa, const int xb, const OutT v,
                                           const int lane, const bool vec) {
  constexpr int EPL = 16 / (int)sizeof(OutT);
  const int xv = (xa + EPL - 1) & ~(EPL - 1);     // first aligned column
  const int nvec = vec ? max(0, (xb + 1 - xv) / EPL) : 0; // whole 16-byte pieces per row
  if (nvec > 0 && nvec <= 32) {
    const int lpr = nvec <= 8 ? 8 : (nvec <= 16 ? 16 : 32); // lanes per row (a power of two)
    const int rpp = 32 / lpr, rsub = lane / lpr, c = lane & (lpr - 1);
    if (c < nvec) {
      OutT *q = out + (ptrdiff_t)(y0 + dy * rsub) * nx + xv + c * EPL;
      const ptrdiff_t step = (ptrdiff_t)dy * rpp * nx;
      for (int r = rsub; r < nrows; r += rpp, q += step) stg16_fill(q, v);
    }
    // cells in front of the first and behind the last whole piece (the grid's edges only)
    const int xt = xv + nvec * EPL, nhead = xv - xa, nedge = nhead + (xb + 1 - xt);
    if (nedge > 0) {
      for (int idx = lane; idx < nrows * nedge; idx += 32) {
        const int r = idx / nedge, e = idx - r * nedge;
        const int x = e < nhead ? xa + e : xt + (e - nhead);
        __stcs(out + (ptrdiff_t)(y0 + dy * r) * nx + x, v);
      }
    }
  } else {
    for (int r = 0; r < nrows; ++r) fill_span<OutT>(out + (ptrdiff_t)(y0 + dy * r) * nx, xa, xb, v, lane, vec);
  }
}

__device__ __forceinline__ int ld_acquire_shared(const int *a) {
  int v;
  asm volatile("ld.acquire.cta.shared.s32 %0, [%1];"
               : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(a)) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_shared(int *a, int v) {
  asm volatile("st.release.cta.shared.s32 [%0], %1;"
               :: "r"((uint32_t)__cvta_generic_to_shared(a)), "r"(v) : "memory");
}

// What a tile needs from global memory, fetched while the previous tile of the row is still
// being computed (the loads are L2 hits of a few hundred cycles; issued at the head of the
// tile they were the first thing on its critical path): the block-summary verdict and,
// where the summary does not prove the tile free, the raw occupancy words of this lane's
// row (bit plane along x) and column (bit plane along y; diagonal and row-octant tiles).
struct TilePre {
  uint32_t r0, r1, c0, c1;
  int sumfree;
};

template <bool CLIP = false>
__device__ __forceinline__ TilePre tile_prefetch(const TileArgs &p, const TQuad &g,
                                                 const uint32_t *__restrict__ rowpl,
                                                 const uint32_t *__restrict__ colpl,
                                                 const uint32_t *__restrict__ bsum, const int sx,
                                                 const int sy, const int I, const int J,
                                                 const int lane) {
  TilePre t;
  t.r0 = t.r1 = t.c0 = t.c1 = 0u;
  t.sumfree = 0;
  const int wi = I ? kTile : g.a, wj = J ? kTile : g.a;
  const int i0 = tile_start(g.a, I), j0 = tile_start(g.a, J);
  const int nvx = min(wi, ext_cx<CLIP>(g, sx) - i0 + 1), nvy = min(wj, ext_cy<CLIP>(g, sy) - j0 + 1);
  if (nvx > 0 && nvy > 0) {
    t.sumfree = tile_sum_free<CLIP>(g, bsum, CLIP ? p.w_sw : tile_sum_words(p.nx), sx, sy, I, J);
    if (!t.sumfree) {
      if (lane < nvy) { // row j0 + lane, bit b <-> local column i0 + b
        const uint32_t *rp =
            rowpl + (size_t)(sy + g.diry * (j0 + lane)) * p.pl.wx + ((g.psx + i0) >> 5);
        t.r0 = __ldg(rp);
        t.r1 = __ldg(rp + 1);
      }
      if (J >= I && lane < nvx) { // column i0 + lane, bit b <-> local row j0 + b
        const uint32_t *cp =
            colpl + (size_t)(sx + g.dirx * (i0 + lane)) * p.pl.wy + ((g.psy + j0) >> 5);
        t.c0 = __ldg(cp);
        t.c1 = __ldg(cp + 1);
      }
    }
  }
  return t;
}

__device__ __forceinline__ int ld_acquire_gpu(const int *a) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(a) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int *a, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" :: "l"(a), "r"(v) : "memory");
}

__device__ __forceinline__ int ld_acquire_sys(const int *a) {
  int v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(a) : "memory");
  return v;
}

// One tile (I, J) of quadrant g by one warp.  Lv (lane r: q(i0-1, j0+r)) and cor
// (q(i0-1, j0-1)) are the left inputs; on return they hold the same for tile (I+1, J).
// GE: the boundary rows (edges) and the progress flag are in global memory and shared with
// warps of other CTAs (grid mode): boundary reads bypass L1, the flag is released at GPU scope.
template <typename OutT, int NW, bool GE, int FMT = kFmtValues>
__device__ __forceinline__ void process_tile(const TileArgs &p, const TQuad &g, const TilePre &pre,
                                             const int sx, const int sy, const int I, const int J,
                                             OutT *__restrict__ out, double *edges,
                                             OutT *stage, double *wscr, const int lane,
                                             double &Lv, double &cor, int *done_flag,
                                             int *xflag = nullptr) {
  // the row above may start its tile I as soon as rowE holds this tile's top row: publish
  // before the global stores
  constexpr int kStepUnroll = NW == 1 ? VHP_STEP_UNROLL_1W : VHP_STEP_UNROLL;
  constexpr bool BITS = fmt_bits(FMT);
  constexpr bool MERGE = fmt_merge(FMT);
  static_assert(!BITS || sizeof(OutT) == 4, "bit output: OutT is the 32-bit word");
  static_assert(!MERGE || (sizeof(OutT) == 8 && !GE), "merge output: fp64 staging, one-CTA sweeps");
  auto publish = [&]() {
    if (GE) __threadfence(); // this lane's boundary-row stores, before lane 0 raises the flag
    __syncwarp();
    if (lane == 0) {
      if (GE) st_release_gpu(done_flag, I + 1);
      else st_release_shared(done_flag, I + 1);
    }
    if (GE && xflag) {
      // hand this tile's top row to the strip on the next GPU (see TileArgs::x_edges); its boundary
      // row of the quadrant lies at the same offset as here (rowOff depends on the source alone)
      const int wi_ = I ? kTile : g.a;
      const int i0_ = tile_start(g.a, I);
      const double top = __ldcg(edges + g.rowOff + i0_ + lane);
      if (lane < wi_) p.x_edges[g.rowOff + i0_ + lane] = top;
      __threadfence_system();
      __syncwarp();
      if (lane == 0) atomicMax_system(xflag, I + 1);
    }
  };
  constexpr bool WIN = FMT == kFmtWindow, CLIP = fmt_clip(FMT);
  const int nx = WIN ? 2 * p.w_r + 1 : p.nx; // row pitch of `out` (kFmtMergeRange*: the map's)
  const int wi = I ? kTile : g.a, wj = J ? kTile : g.a;          // tile extent
  const int i0 = tile_start(g.a, I), j0 = tile_start(g.a, J);
  const int il = i0 + lane, jr = j0 + lane;
  // the never-written border column / row is "occupied": exclude it from the compute extent
  const int ExC = ext_cx<CLIP>(g, sx), EyC = ext_cy<CLIP>(g, sy);
  const int nvx = min(wi, ExC - i0 + 1), nvy = min(wj, EyC - j0 + 1); // columns / rows to compute
  const uint32_t cmask = nvx >= 32 ? ~0u : (nvx <= 0 ? 0u : (1u << nvx) - 1u);
  const uint32_t rmask = nvy >= 32 ? ~0u : (nvy <= 0 ? 0u : (1u << nvy) - 1u);
  const bool colc = (cmask >> lane) & 1u, rowc = (rmask >> lane) & 1u;
  double *rowE = edges + g.rowOff + i0;
  // 1/k of the 32 steps of this tile (k = i in column-octant and diagonal tiles, j in
  // row-octant tiles): one coalesced load here, parked in shared memory if the tile computes
  const double2 myr = __ldg(p.rtab + max(i0, j0) + lane);

  // ---- occupancy: block summary first, bit plane otherwise --------------------------
  bool allfree = false, allocc = true;
  const bool sumfree = pre.sumfree != 0;
  uint32_t wrow = 0;
  if (nvx > 0 && nvy > 0) {
    if (sumfree) {
      wrow = rowc ? cmask : 0u;
      allfree = true;
      allocc = false;
    } else {
      if (rowc) wrow = __funnelshift_r(pre.r0, pre.r1, (g.psx + i0) & 31) & cmask;
      allfree = __all_sync(kAll, wrow == (rowc ? cmask : 0u));
      allocc = __all_sync(kAll, wrow == 0u);
    }
  }
  const double Bv = GE ? __ldcg(rowE + lane) : rowE[lane];
  const bool inuni = __all_sync(kAll, (!colc || Bv == cor) && (!rowc || Lv == cor));
  const bool zero_in = inuni && cor == 0.0;

  // store geometry: lane <-> column il of rows j0 .. j0 + wj - 1
  const bool lane_st = lane < wi && il <= g.Ex && !(g.dirx < 0 && il == 0);
  const bool lane_st_all = nvx == 32 && (I > 0 || g.dirx > 0); // every lane stores
  OutT *const ptr = out + (ptrdiff_t)(sy + g.diry * j0) * nx + (sx + g.dirx * il);
  const ptrdiff_t rs = (ptrdiff_t)g.diry * nx;
  // rows to store: inside the grid and the window; the axis row belongs to the +y quadrant
  const int r0 = max((g.diry < 0 && j0 == 0) ? 1 : 0, g.jw0 - j0);
  const int rgrid = min(wj - 1, g.Ey - j0);          // last row inside the grid
  const int rlast = min(rgrid, g.jw1 - j0);
  // bit output: the tile's columns of one row are (part of) ONE word, since tile columns start on
  // multiples of 32 except the first one of a quadrant, which ends on one
  const int xw = g.dirx > 0 ? sx + i0 : sx - i0; // column of lane 0
  const int wpr = FMT == kFmtCoverBits ? vhp_cover_words(p.nx, p.w_r) : (nx + 31) >> 5; // words per row of `out`
  auto put_word = [&](const uint32_t m, const int rfirst, const int rend) { // m: bit l <-> column il
    const uint32_t w = g.dirx > 0 ? m << (xw & 31) : __brev(m) >> (31 - (xw & 31));
    if (lane >= rfirst && lane <= rend && w) { // lane <-> row j0 + lane
      uint32_t *q = reinterpret_cast<uint32_t *>(out) + (ptrdiff_t)(sy + g.diry * (j0 + lane)) * wpr + (xw >> 5);
      if (I == 0) atomicOr(q, w);
      else *q = w;
    }
  };
  uint32_t wb = 0; // BITS: the bits of row j0 + lane
  // value >= thr on the bit patterns: the values are never negative (or NaN) and thr > 0, where the
  // order of IEEE doubles is the order of their bits as integers -- two integer compares per cell
  // instead of one on the fp64 pipe, which the step loops already saturate
  const long long thrb = __double_as_longlong(p.thr);
  auto ge_thr = [&](const double v) -> bool { return __double_as_longlong(v) >= thrb; };

  if (allocc || zero_in || (inuni && allfree)) {
    // ---- uniform tile: no arithmetic -------------------------------------------------
    const bool zero = allocc || zero_in;
    if (allocc && !zero_in) { // live inputs end here
      if (lane < wi) rowE[lane] = 0.0;
      Lv = 0.0;
      cor = __shfl_sync(kAll, Bv, wi - 1);
    }
    publish();
    const int rc = min(min(wj - 1, EyC - j0), rlast); // last lit row; a border row (if any) follows
    if constexpr (BITS) {
      if (!zero && cor >= p.thr) put_word(__ballot_sync(kAll, lane_st && colc), r0, rc);
      return;
    }
    if constexpr (MERGE) { // the border row (if any) is 0: nothing to fold
      if (!zero && cor > 0.0 && lane_st && colc) {
        const ptrdiff_t i0c = ptr - out;
        for (int r = r0; r <= rc; ++r) merge_cell<FMT>(p, i0c + r * rs, il, j0 + r, cor);
      }
      return;
    }
    if (p.vec && nvx == 32 && (I > 0 || g.dirx > 0)) {
      // all 32 columns are stored and x0 is a multiple of 32: 128-bit stores
      constexpr int EPL = 16 / (int)sizeof(OutT), LPR = 32 / EPL; // elements per lane, lanes per row
      const int sub = lane / LPR;
      const int xlow = g.dirx > 0 ? sx + i0 : sx - i0 - 31;
      const OutT v = to_out<OutT>(zero ? 0.0 : cor);
      OutT *q = out + (ptrdiff_t)(sy + g.diry * (j0 + r0 + sub)) * nx + (xlow + (lane % LPR) * EPL);
#pragma unroll kFillUnroll
      for (int r = r0 + sub; r <= rc; r += EPL, q += EPL * rs) stg16_fill(q, v);
      if (rc < rlast && sub == 0)
        stg16_fill(out + (ptrdiff_t)(sy + g.diry * (j0 + rlast)) * nx + (xlow + (lane % LPR) * EPL),
                   to_out<OutT>(0.0));
    } else if (lane_st) {
      const OutT lv = to_out<OutT>((zero || !colc) ? 0.0 : cor);
      OutT *q = ptr + r0 * rs;
#pragma unroll kFillUnroll
      for (int r = r0; r <= rc; ++r, q += rs) __stcs(q, lv);
      if (rc < rlast) __stcs(ptr + rlast * rs, to_out<OutT>(0.0));
    }
    return;
  }

  const double fd = (double)(I > J ? jr : il); // offset along the front (i0 == j0 on the diagonal)
  double *lx = wscr + 34, *wnew = wscr; // wscr: bottom stream, lx: left stream; wnew (row-octant tiles
                                        // only, which never read wscr): the new left column
  double2 *const rts = reinterpret_cast<double2 *>(wscr + 68); // 1/k of step s (entry 32: never used)
  const double cor_next = __shfl_sync(kAll, Bv, wi - 1);
  __syncwarp();
  wscr[1 + lane] = Bv;
  lx[1 + lane] = Lv;
  rts[lane] = myr;
  if (lane == 0) {
    wscr[0] = cor;
    lx[0] = cor;
  }
  __syncwarp();

  if (I > J) {
    // ---- column-octant tile: lanes along j, steps along i (wi == 32) -------------------
    double F = Lv;
    const int ns = min(32, g.Ex - i0 + 1);
    // this tile's bottom inputs are in wscr by now: its top row goes straight into rowE
    if (ns < 32 && lane >= ns) rowE[lane] = 0.0; // columns beyond the grid
    auto steps = [&](auto masked) { // masked: the tile has occupied cells (or cells off the grid)
      double2 rn = rts[0]; // 1/i of the next step, read one step ahead
      const int nst = (VHP_FIXED32 && !decltype(masked)::value) ? kTile : ns;
#pragma unroll kStepUnroll
      for (int s = 0; s < nst; ++s) {
        const double2 rr = rn;
        rn = rts[s + 1];
        const double up = __shfl_up_sync(kAll, F, 1);
        const double b = lane ? up : wscr[s];
        const double c = __fma_rn(fd, rr.x, __dmul_rn(fd, rr.y));
        const double v = lerp_rn(F, b, c);
        F = (!decltype(masked)::value || ((wrow >> s) & 1u)) ? v : 0.0;
        // (storing this lane's row straight from registers, 16 bytes every few steps, was
        // measured slower than staging: 32 partial-sector requests per store instruction)
        if constexpr (BITS) wb |= (uint32_t)ge_thr(F) << s;
        else stage[stage_at(lane, s)] = to_out<OutT>(F);
        if (lane == wj - 1) rowE[s] = F;
      }
    };
    if (allfree && nvx == 32 && nvy == 32) steps(std::false_type{});
    else steps(std::true_type{});
    Lv = F;
    publish();
  } else {
    // occupancy of column il, bit b <-> local row j0 + b
    uint32_t wcol = 0;
    if (colc) {
      wcol = sumfree ? rmask : (__funnelshift_r(pre.c0, pre.c1, (g.psy + j0) & 31) & rmask);
    }
    if (J > I) {
      // ---- row-octant tile: lanes along i, steps along j (wj == 32) --------------------
      double F = Bv;
      const int ns = rgrid + 1;
      auto steps = [&](auto masked) {
        OutT *q = ptr;
        double2 rn = rts[0];
        const int nst = (VHP_FIXED32 && !decltype(masked)::value) ? kTile : ns;
#pragma unroll kStepUnroll
        for (int s = 0; s < nst; ++s, q += rs) {
          const double2 rr = rn;
          rn = rts[s + 1];
          const double up = __shfl_up_sync(kAll, F, 1);
          const double b = lane ? up : lx[s];
          const double c = __fma_rn(fd, rr.x, __dmul_rn(fd, rr.y));
          const double v = lerp_rn(F, b, c);
          F = (!decltype(masked)::value || ((wcol >> s) & 1u)) ? v : 0.0;
          if constexpr (BITS) {
            const uint32_t m = __ballot_sync(kAll, ge_thr(F));
            if (lane == s) wb = m;
          } else if constexpr (MERGE) {
            if (!decltype(masked)::value || (lane_st && s >= r0 && s <= rlast)) merge_cell<FMT>(p, q - out, il, j0 + s, F);
          } else if (!decltype(masked)::value || (lane_st && s >= r0 && s <= rlast)) {
            __stcs(q, to_out<OutT>(F));
          }
          if (lane == wi - 1) wnew[s] = F;
        }
      };
      if (allfree && nvx == 32 && nvy == 32 && lane_st_all && r0 == 0 && rlast == 31)
        steps(std::false_type{});
      else steps(std::true_type{});
      __syncwarp();
      if (lane < wi) rowE[lane] = F;
      Lv = wnew[lane];
      cor = cor_next;
      publish();
      if constexpr (BITS) put_word(wb & __ballot_sync(kAll, lane_st), r0, rlast);
      return;
    }
    // ---- diagonal tile: both fronts and the diagonal cell (wi == wj) ---------------------
    double C = 0.0, R = 0.0; // C[l] = q(k-1, j0+l), R[l] = q(i0+l, k-1); set when lane l joins
    const int ns = min(wi, max(g.Ex, g.Ey) - i0 + 1);
    double2 rn = rts[0];
#pragma unroll kDiagUnroll
    for (int k = 0; k < ns; ++k) {
      const double2 rr = rn;
      rn = rts[k + 1];
      const double c = __fma_rn(fd, rr.x, __dmul_rn(fd, rr.y));
      const double upC = __shfl_up_sync(kAll, C, 1);
      const double upR = __shfl_up_sync(kAll, R, 1);
      const double bC = lane ? upC : wscr[k];
      const double bR = lane ? upR : lx[k];
      const double vC = lerp_rn(C, bC, c), vR = lerp_rn(R, bR, c);
      if (lane < k) {
        C = ((wrow >> k) & 1u) ? vC : 0.0;
        R = ((wcol >> k) & 1u) ? vR : 0.0;
        if constexpr (BITS) {
          wb |= (uint32_t)ge_thr(C) << k; // row j0 + lane, column k
        } else {
          stage[stage_at(lane, k)] = to_out<OutT>(C);
          stage[stage_at(k, lane)] = to_out<OutT>(R);
        }
      }
      if constexpr (BITS) { // row j0 + k, columns below k
        const uint32_t m = __ballot_sync(kAll, lane < k && ge_thr(R));
        if (lane == k) wb |= m;
      }
      // diagonal cell q(k,k) = q(k,k-1) * occ: q(k,k-1) is lane k-1's new C (k == 0: B[0])
      const double dsrc = __shfl_up_sync(kAll, C, 1);
      if (lane == k) {
        const double dv = ((wrow >> k) & 1u) ? (k ? dsrc : Bv) : 0.0;
        C = dv;
        R = dv;
        if constexpr (BITS) wb |= (uint32_t)ge_thr(dv) << k;
        else stage[stage_at(k, k)] = to_out<OutT>(dv);
      }
    }
    __syncwarp();
    if (lane < wi) rowE[lane] = R;
    Lv = C;
    publish();
  }
  cor = cor_next;
  // ---- write the staged tile as rows ---------------------------------------------------
  __syncwarp();
  if constexpr (BITS) {
    put_word(wb & __ballot_sync(kAll, lane_st), r0, rlast);
  } else if constexpr (MERGE) {
    if (lane_st) {
      const ptrdiff_t i0c = ptr - out;
      for (int r = r0; r <= rlast; ++r) merge_cell<FMT>(p, i0c + r * rs, il, j0 + r, stage[stage_at(r, lane)]);
    }
  } else if (lane_st) {
    OutT *q = ptr + r0 * rs;
#pragma unroll kFillUnroll
    for (int r = r0; r <= rlast; ++r, q += rs) __stcs(q, stage[stage_at(r, lane)]);
  }
}

// One complete sweep from (sx, sy) by the whole CTA (NW warps, all threads must call).  Writes every cell of out[ny][nx] exactly once (cells on the never-
// written border get 0).  smem_raw: tile_smem_bytes<OutT>(nx, ny, NW) bytes, 16-aligned.
// Ends with a block barrier.
//
// kFmtWindow: every cell of the (2R+1)^2 window exactly once instead (out: see kFmtWindow),
// smem_raw: tile_smem_bytes_win<OutT>(nx, ny, R, NW) bytes.  kFmtMergeRange*: the cells of the box |dx|, |dy| <= R
// once each, in map pitch, smem_raw sized like kFmtWindow.  kFmtCoverBits: the bits of that box, `out` as kFmtBits's
// with the box's row pitch.
//
// Grid mode (MODE != kSweepCta; one sweep of a giant map by many CTAs): kSweepGridInit, run by
// one CTA, computes the staircase and writes it with the boundary rows, the progress flags and
// the row counter to global memory; kSweepGridWork, launched after it with any number of
// CTAs, writes the lit region (grid rows dealt over all warps of the grid) and then takes tile
// rows from the global counter.  A row only waits for a row handed out earlier, whose warp is
// therefore running: no co-residency of the CTAs is needed.
template <typename OutT, int NW, int MODE = kSweepCta, int FMT = kFmtValues>
__device__ __forceinline__ void tile_sweep_cta(const TileArgs &p, const int map, const int sx,
                                               const int sy, OutT *__restrict__ out,
                                               unsigned char *smem_raw) {
  constexpr bool GE = MODE != kSweepCta;
  constexpr bool BITS = fmt_bits(FMT);
  constexpr bool WIN = FMT == kFmtWindow, CLIP = fmt_clip(FMT);
  static_assert(!GE || NW > 1, "grid mode uses the multi-warp boundary layout");
  static_assert(!GE || !CLIP, "clipped sweeps are one-CTA sweeps");
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nx = p.nx, ny = p.ny;
  const int opitch = WIN ? 2 * p.w_r + 1 : nx; // row pitch of `out`
  TQuad *quads = reinterpret_cast<TQuad *>(smem_raw);
  // next tile row to hand out (NW > 1)
  int *next_row = GE ? p.g_next_row : reinterpret_cast<int *>(smem_raw + 240);
  static_assert(4 * sizeof(TQuad) <= kMergeHdr, "quadrant geometry overlaps the merge slot / row counter");
  uint32_t *bsum = reinterpret_cast<uint32_t *>(smem_raw + kTileHdr);
  const int nsum = tile_sum_words(nx) * ((ny + 31) >> 5);
  const int sum_bytes = CLIP ? win_sum_bytes(nx, ny, p.w_r) : tile_sum_bytes(nx, ny);
  const int lmcap = tile_lm_cap(CLIP ? win_side(ny, p.w_r) : ny);
  int *Lm = reinterpret_cast<int *>(smem_raw + kTileHdr + sum_bytes);
  int *prog = GE ? p.g_prog : Lm + 4 * lmcap; // tiles finished (or lit) at the head of tile row (q, J)
  double *const edges_s = reinterpret_cast<double *>(smem_raw + kTileHdr + sum_bytes + 32 * lmcap);
  double *edges = GE ? p.g_edges : edges_s;
  const int nedge = tile_edge_doubles(CLIP ? win_side(nx, p.w_r) : nx, NW);
  unsigned char *wbase = reinterpret_cast<unsigned char *>(GE ? edges_s : edges_s + nedge);
  double *wscr = reinterpret_cast<double *>(wbase) + warp * kWarpScratch;
  OutT *stage = reinterpret_cast<OutT *>(wbase + NW * kWarpScratch * sizeof(double)) +
                warp * (kTile * kStagePitch);

  if (tid == 0) {
    if (MODE != kSweepGridWork) *next_row = 0;
    const int WXb = 32 * ((nx + 31) >> 5), WYb = 32 * ((ny + 31) >> 5);
    int off = 0;
    for (int q = 0; q < 4; ++q) { // Q1 (+,+), Q2 (-,+), Q3 (-,-), Q4 (+,-): reference order
      TQuad g;
      g.dirx = (q == 0 || q == 3) ? 1 : -1;
      g.diry = (q < 2) ? 1 : -1;
      g.Ex = g.dirx > 0 ? nx - 1 - sx : sx;
      g.Ey = g.diry > 0 ? ny - 1 - sy : sy;
      if (CLIP) {
        g.Ex = min(g.Ex, p.w_r);
        g.Ey = min(g.Ey, p.w_r);
      }
      // first tile width: the next tile column starts (+x) / ends (-x) on a multiple of 32
      g.a = g.dirx > 0 ? 32 - (sx & 31) : ((sx + 1) & 31);
      if (g.a == 0) g.a = 32;
      const bool exists = (g.dirx > 0 || sx > 0) && (g.diry > 0 || sy > 0);
      g.TX = !exists ? 0 : (g.Ex < g.a ? 1 : (g.Ex - g.a) / kTile + 2);
      g.TY = !exists ? 0 : (g.Ey < g.a ? 1 : (g.Ey - g.a) / kTile + 2);
      g.rowOff = NW == 1 ? 0 : off;
      off += g.TX * kTile;
      g.psx = g.dirx > 0 ? sx : WXb - 1 - sx;
      g.psy = g.diry > 0 ? sy : WYb - 1 - sy;
      int halo_y;
      tile_window_of(q, nx, ny, sx, sy, p.win_y0, p.win_y1, &g.jw0, &g.jw1, &g.Jlo, &g.Jhi, &halo_y);
      if (g.Jhi < g.Jlo || !((p.qmask >> q) & 1)) g.TX = g.TY = 0; // nothing of this quadrant to do
      quads[q] = g;
    }
    if (GE) {
      // export plan: the tile row just below the neighbour's first one, per quadrant (from ITS window)
      short *xJ = reinterpret_cast<short *>(smem_raw + 244);
      for (int q = 0; q < 4; ++q) {
        const TQuad &g = quads[q];
        xJ[q] = -1;
        if (!p.x_edges) continue;
        int jw0, jw1, Jlo2, Jhi2, hy;
        tile_window_of(q, nx, ny, sx, sy, p.x_y0, p.x_y1, &jw0, &jw1, &Jlo2, &Jhi2, &hy);
        if (g.TX && Jhi2 >= Jlo2 && Jlo2 > 0 && Jlo2 - 1 >= g.Jlo && Jlo2 - 1 <= g.Jhi) xJ[q] = (short)(Jlo2 - 1);
      }
    }
  }
  // bsq: the summary addressed by absolute block row and word (a clipped sweep copies only the words its box
  // touches, rows of p.w_sw words)
  const uint32_t *bsq = bsum;
  if constexpr (CLIP) {
    const int R = p.w_r, nbw = tile_sum_words(nx), sw = p.w_sw;
    const int wlo = (max(sx - R, 0) >> 5) >> 5, whi = (min(sx + R, nx - 1) >> 5) >> 5;
    const int blo = max(sy - R, 0) >> 5, bhi = min(sy + R, ny - 1) >> 5;
    const int nw = whi - wlo + 1, nwin = nw * (bhi - blo + 1);
    const uint32_t *src = p.pl.bsum + (size_t)map * nsum + (size_t)blo * nbw + wlo;
    for (int i = tid; i < nwin; i += blockDim.x) {
      const int r = i / nw, c = i - r * nw;
      bsum[r * sw + c] = __ldg(src + (size_t)r * nbw + c);
    }
    bsq = bsum - (blo * sw + wlo);
    if constexpr (WIN) {
      // window cells outside the grid are 0: the rows above / below it, then the columns left / right of it
      const int W = 2 * R + 1, x0 = sx - R, y0 = sy - R;
      const int ul = max(0, -x0), uh = min(W - 1, nx - 1 - x0), vl = max(0, -y0), vh = min(W - 1, ny - 1 - y0);
      OutT *const wout = out + (ptrdiff_t)y0 * W + x0;
      const OutT z = to_out<OutT>(0.0);
      for (int v = warp; v < W; v += NW) {
        OutT *const row = wout + (ptrdiff_t)v * W;
        if (v < vl || v > vh) {
          fill_run<OutT>(row, W, z, lane);
        } else {
          if (ul > 0) fill_run<OutT>(row, ul, z, lane);
          if (uh < W - 1) fill_run<OutT>(row + uh + 1, W - 1 - uh, z, lane);
        }
      }
    }
  } else {
    for (int i = tid; i < nsum; i += blockDim.x) bsum[i] = __ldg(p.pl.bsum + (size_t)map * nsum + i);
  }
  if (MODE == kSweepCta)
    for (int i = tid; i < nedge; i += blockDim.x) edges[i] = 1.0; // virtual boundary
  __syncthreads();
  if (MODE == kSweepGridWork) { // the staircase was computed by the init kernel
    for (int i = tid; i < 4 * lmcap; i += blockDim.x) Lm[i] = __ldg(p.g_lm + i);
    __syncthreads();
  }

  // ---- lit staircase: leading free tiles per tile row, then the running minimum ---------
  const int nbw = CLIP ? p.w_sw : tile_sum_words(nx);
  if (MODE != kSweepGridWork) {
  for (int q = 0; q < 4; ++q) {
    const TQuad &g = quads[q];
    for (int J = warp; J < g.TY; J += NW) {
      int L = 0;
      for (int Ib = 0; Ib < g.TX; Ib += 32) {
        const bool fr = Ib + lane < g.TX && tile_sum_free<CLIP>(g, bsq, nbw, sx, sy, Ib + lane, J);
        const unsigned m = __ballot_sync(kAll, fr);
        const int run = __ffs(~m) - 1; // leading ones (-1: all 32)
        L += run < 0 ? 32 : run;
        if (run >= 0) break;
      }
      if (lane == 0) Lm[q * lmcap + J] = L;
    }
  }
  __syncthreads();
  if (tid < 4) {
    const TQuad &g = quads[tid];
    int m = g.TX;
    for (int J = 0; J < g.TY; ++J) {
      m = min(m, Lm[tid * lmcap + J]);
      Lm[tid * lmcap + J] = m;
      if (GE && ((p.remote_mask >> tid) & 1) && J == g.Jlo - 1)
        atomicMax_system(prog + tid * lmcap + J, m); // the row below arrives tile by tile from the neighbour
      else
        prog[tid * lmcap + J] = J < g.Jlo ? g.TX : m; // rows below the window count as finished
      if (GE) p.g_lm[tid * lmcap + J] = m;
    }
  }
  if (MODE == kSweepGridInit) {
    // virtual boundary -- except where the neighbouring strip writes the boundary row itself
    // (beyond the lit tiles of the row below this quadrant's first one)
    __syncthreads();
    for (int i = tid; i < nedge; i += blockDim.x) {
      bool mine = true;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const TQuad &g = quads[q];
        if (((p.remote_mask >> q) & 1) && g.TX && g.Jlo > 0) {
          const int lit = tile_start(g.a, Lm[q * lmcap + g.Jlo - 1]);
          if (i >= g.rowOff + lit && i < g.rowOff + g.TX * kTile) mine = false;
        }
      }
      if (mine) edges[i] = 1.0;
    }
    __syncthreads();
  }
  if (NW > 1) { // boundary row below the first tile row of the window = the neighbour's halo row
    for (int q = 0; q < 4; ++q) {
      const TQuad &g = quads[q];
      if (g.TX && g.Jlo > 0 && p.halo[q])
        for (int i = tid; i <= g.Ex; i += blockDim.x)
          edges[g.rowOff + i] = __ldg(p.halo[q] + (sx + g.dirx * i));
    }
  }
  }
  if (MODE == kSweepGridInit) return; // boundary rows, flags, staircase and counter are set
  __syncthreads();

  // ---- write the lit region: one warp per grid row, -x and +x runs merged -----------------
  {
    // per quadrant: first tile width, extent, existence (registers; q = 0..3)
    int qa[4], qex[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      qa[q] = quads[q].a;
      qex[q] = quads[q].TX ? quads[q].Ex : -1;
    }
    // lit cells i = 0 .. n-1 of quadrant q in local row j; the staircase is looked up once
    // per tile row (cj = cached tile row, cn = its run length)
    int cj[4] = {-1, -1, -1, -1}, cn[4] = {0, 0, 0, 0};
    auto lit_run = [&](const int q, const int j) -> int {
      if (qex[q] < 0) return 0;
      const int J = j < qa[q] ? 0 : ((j - qa[q]) >> 5) + 1;
      if (J != cj[q]) {
        cj[q] = J;
        cn[q] = min(tile_start(qa[q], Lm[q * lmcap + J]), qex[q] + 1);
      }
      return cn[q];
    };
    // Lm is non-increasing in J, so the lit rows of a quadrant are j < jl[q]
    int jl[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int Jz = 0;
      while (Jz < quads[q].TY && Lm[q * lmcap + Jz] > 0) ++Jz;
      jl[q] = qex[q] < 0 ? 0 : min(tile_start(qa[q], Jz), quads[q].Ey + 1);
    }
    // rows below the source are j = 1 .. jl - 1, rows from the source upwards j = 0 .. jl - 1
    const int ylo = sy - max(max(jl[2], jl[3]) - 1, 0), yhi = sy + max(jl[0], jl[1]) - 1;
    const int wfirst = GE ? (int)blockIdx.x * NW + warp : warp, wstride = GE ? (int)gridDim.x * NW : NW;
    if constexpr (BITS) {
      // Bit output: a lit row is one store of its words.  The runs (nL, nR) only change where a
      // quadrant's tile row changes, so the rows are cut into segments of constant runs (the union
      // of the -x and +x quadrants' tile-row boundaries), dealt over the warps; a segment computes its
      // word masks once and then stores them row after row.  (Row by row, with the staircase
      // looked up per row, the all-lit headline batch spent 135 instructions per row.)
      static_assert(!GE, "bit output is a one-CTA sweep");
      const int wprl = FMT == kFmtCoverBits ? vhp_cover_words(nx, p.w_r) : (nx + 31) >> 5;
      uint32_t *const wout = reinterpret_cast<uint32_t *>(out);
      int seg = 0;
      for (int half = 0; half < 2 && 1.0 >= p.thr; ++half) {
        const int qR = half ? 3 : 0, qL = half ? 2 : 1, dy = half ? -1 : 1;
        // rows j < jend; below the source they start at j = 1 and leave out y == 0 (never written)
        const int jend = half ? min(max(jl[2], jl[3]), sy) : max(jl[0], jl[1]);
        for (int j = half; j < jend;) {
          const int nbR = j < qa[qR] ? qa[qR] : qa[qR] + (((j - qa[qR]) >> 5) + 1) * 32;
          const int nbL = j < qa[qL] ? qa[qL] : qa[qL] + (((j - qa[qL]) >> 5) + 1) * 32;
          const int jn = min(jend, min(nbR, nbL));
          if (seg++ % NW == warp) {
            const int nR = lit_run(qR, j), nL = lit_run(qL, j);
            if (nR > 0 || nL > 1) {
              const int xfirst = nL > 1 ? max(sx - (nL - 1), 1) : sx, xend = nR > 0 ? sx + nR - 1 : sx - 1;
              for (int w = (xfirst >> 5) + lane; w <= (xend >> 5); w += 32) {
                uint32_t m = ~0u;
                if (w == (xfirst >> 5)) m &= ~0u << (xfirst & 31);
                if (w == (xend >> 5)) m &= ~0u >> (31 - (xend & 31));
                uint32_t *q = wout + (ptrdiff_t)(sy + dy * j) * wprl + w;
                const ptrdiff_t qs = (ptrdiff_t)dy * wprl;
                if (m == ~0u) { // a whole word inside the lit run has no other writer
                  for (int r = j; r < jn; ++r, q += qs) *q = m;
                } else {
                  for (int r = j; r < jn; ++r, q += qs) atomicOr(q, m);
                }
              }
            }
          }
          j = jn;
        }
      }
    } else if constexpr (fmt_merge(FMT)) {
      // merge output: the lit spans of the value loop below, folded cell by cell (value 1.0); the never-written
      // cells of those rows (x == 0 left of the source, row 0 below it) hold 0 and are left alone
      static_assert(!GE, "merge output is a one-CTA sweep");
      for (int y = ylo + warp; y <= yhi; y += NW) {
        const bool upper = y >= sy;
        if (!upper && y == 0) continue;
        const int j = upper ? y - sy : sy - y;
        const int nR = upper ? lit_run(0, j) : lit_run(3, j);
        const int nL = upper ? lit_run(1, j) : lit_run(2, j);
        if (nR == 0 && nL <= 1) continue;
        const int xl = nL > 1 ? max(sx - (nL - 1), 1) : sx; // first lit column
        const int xr = nR > 0 ? sx + nR - 1 : sx - 1;       // last lit column
        for (int x = xl + lane; x <= xr; x += 32) merge_cell<FMT>(p, (ptrdiff_t)y * nx + x, abs(x - sx), j, 1.0);
      }
    } else
    for (int y = max(ylo, p.win_y0) + wfirst; y <= min(yhi, p.win_y1 - 1); y += wstride) {
      const bool upper = y >= sy;
      const int j = upper ? y - sy : sy - y;
      const int nR = upper ? lit_run(0, j) : lit_run(3, j);
      const int nL = upper ? lit_run(1, j) : lit_run(2, j);
      if (nR == 0 && nL <= 1) continue;
      OutT *row = out + (size_t)y * opitch;
      const OutT v = to_out<OutT>((!upper && y == 0) ? 0.0 : 1.0); // y == 0 below the source: never written
      int xa = sx - (nL - 1), xb = sx + nR - 1;
      if (nL > 0 && xa == 0) { // x == 0 left of the source: never written
        if (lane == 0) __stcs(row, to_out<OutT>(0.0));
        xa = 1;
      }
      if (WIN) { // one run (the axis cell between the two quadrants' spans is lit whenever both are)
        if (nR > 0 && nL > 1) {
          fill_run<OutT>(row + xa, xb - xa + 1, v, lane);
        } else {
          if (nL > 1) fill_run<OutT>(row + xa, sx - xa, v, lane);
          if (nR > 0) fill_run<OutT>(row + sx, xb - sx + 1, v, lane);
        }
      } else if (nR > 0 && nL > 1) {
        fill_span<OutT>(row, xa, xb, v, lane, p.vec);
      } else {
        if (nL > 1) fill_span<OutT>(row, xa, sx - 1, v, lane, p.vec);
        if (nR > 0) fill_span<OutT>(row, sx, xb, v, lane, p.vec);
      }
    }
  }

  // ---- the rest: tile rows as pipelines ------------------------------------------------------
  auto run_row = [&](const int q, const int J, const int I0) {
    const TQuad &g = quads[q];
    const uint32_t *rowpl = (g.dirx > 0 ? p.pl.rowF : p.pl.rowR) + (size_t)map * p.pl.row_plane;
    const uint32_t *colpl = (g.diry > 0 ? p.pl.colF : p.pl.colR) + (size_t)map * p.pl.col_plane;
    double Lv = 1.0, cor = 1.0; // left of the first tile: lit tiles or the virtual boundary
    int *xflag = nullptr; // grid mode across GPUs: the neighbour's flag of this row, if it is the exported one
    if (GE && reinterpret_cast<const short *>(smem_raw + 244)[q] == J) xflag = p.x_prog + q * lmcap + J;
    TilePre pre = tile_prefetch<CLIP>(p, g, rowpl, colpl, bsq, sx, sy, I0, J, lane);
#if VHP_DARK_TAIL
    // rows of this tile row that hold cells to compute (lane <-> row j0 + lane), as in process_tile
    const int j0row = tile_start(g.a, J);
    const int nvyrow = min(J ? kTile : g.a, ext_cy<CLIP>(g, sy) - j0row + 1);
    const bool rowc_row = lane < nvyrow;
    int dark_seen = -1; // a boundary column >= the tile start known to be non-zero (finished row below)
#endif
#pragma unroll 1
    for (int I = I0; I < g.TX; ++I) {
#if VHP_DARK_TAIL
      // Dark run: the left inputs are zero and the top row of the row below is zero over the
      // next n finished tiles -> every cell of those n tiles is 0 (zero inputs give zero whatever
      // the occupancy; the boundary row stays zero and is not rewritten).  Hand them to the row
      // above at once and write the zeros as row spans, without per-tile set-up.  (Multi-warp
      // CTAs only: the single-warp kernels are bound by their code size.)
      if (NW > 1 && !GE && J > 0 && I > I0 && cor == 0.0 && tile_start(g.a, I) > dark_seen &&
          __all_sync(kAll, !rowc_row || Lv == 0.0)) {
        const int Iend = min(ld_acquire_shared(prog + q * lmcap + J - 1), g.TX); // finished below
        if (Iend > I) {
          const int i0 = tile_start(g.a, I);
          const int ilim = min(ext_cx<CLIP>(g, sx), tile_start(g.a, Iend) - 1);
          const double *rowB = edges + g.rowOff;
          int bad = -1;
          for (int ib = i0; ib <= ilim && bad < 0; ib += 32) {
            const unsigned nz = __ballot_sync(kAll, ib + lane <= ilim && rowB[ib + lane] != 0.0);
            if (nz) bad = ib + __ffs(nz) - 1;
          }
          int Istop = Iend; // first tile not known to be dark
          if (bad >= 0) {
            Istop = tile_row_of(g.a, bad);
            dark_seen = bad;
          }
          if (Istop > I) {
            __syncwarp();
            if (lane == 0) st_release_shared(prog + q * lmcap + J, Istop);
            const int r0 = max(0, g.jw0 - j0row);
            const int rlast = min(min((J ? kTile : g.a) - 1, g.Ey - j0row), g.jw1 - j0row);
            const int ie = min(g.Ex, tile_start(g.a, Istop) - 1); // last local column of the run
            const int xa = g.dirx > 0 ? sx + i0 : sx - ie, xb = g.dirx > 0 ? sx + ie : sx - i0;
            if constexpr (FMT == kFmtValues)
              fill_block<OutT>(out, nx, sy + g.diry * (j0row + r0), g.diry, rlast - r0 + 1, xa, xb,
                               to_out<OutT>(0.0), lane, p.vec != 0);
            if constexpr (WIN)
              for (int r = r0; r <= rlast; ++r)
                fill_run<OutT>(out + (ptrdiff_t)(sy + g.diry * (j0row + r)) * opitch + xa, xb - xa + 1,
                               to_out<OutT>(0.0), lane);
            if (Istop >= g.TX) return;
            pre = tile_prefetch<CLIP>(p, g, rowpl, colpl, bsq, sx, sy, Istop, J, lane);
            I = Istop - 1;
            continue;
          }
        }
      }
#endif
      const TilePre cur = pre;
      if (I + 1 < g.TX) pre = tile_prefetch<CLIP>(p, g, rowpl, colpl, bsq, sx, sy, I + 1, J, lane);
      if (GE && J > 0 && ((p.remote_mask >> q) & 1) && J == g.Jlo) {
        // the row below lives on the neighbouring GPU: its flag arrives over NVLink.  A watchdog
        // (a few seconds) turns a lost neighbour into an error instead of a hung GPU.
        const int *flag = prog + q * lmcap + J - 1;
        unsigned polls = 0;
        while (ld_acquire_sys(flag) <= I) {
          __nanosleep(200);
          if (++polls > (1u << 24)) {
            if (lane == 0) atomicOr(p.err, 2);
            break;
          }
        }
      } else if (NW > 1 && J > 0) { // tile (I, J-1) must be finished
        const int *flag = prog + q * lmcap + J - 1;
#if VHP_POLL_BACKOFF
        for (unsigned ns = VHP_POLL_NS0; (GE ? ld_acquire_gpu(flag) : ld_acquire_shared(flag)) <= I;
             ns = min(2 * ns, (unsigned)VHP_POLL_NSMAX))
          __nanosleep(ns);
#else
        while ((GE ? ld_acquire_gpu(flag) : ld_acquire_shared(flag)) <= I) __nanosleep(40);
#endif
      }
      process_tile<OutT, NW, GE, FMT>(p, g, cur, sx, sy, I, J, out, edges, stage, wscr, lane, Lv, cor,
                                  prog + q * lmcap + J, xflag);
      __syncwarp();
    }
  };
  if (NW == 1) {
    // one warp: quadrant after quadrant, rows in order (every dependency is program order);
    // the boundary row is shared, so reset it to the virtual boundary per quadrant
    for (int q = 0; q < 4; ++q) {
      const int TXq = quads[q].TX, TYq = quads[q].TY;
      if (TXq && (q > 0 || quads[q].Jlo > 0)) {
        const bool use_halo = quads[q].Jlo > 0 && p.halo[q];
        const int Exq = quads[q].Ex, dxq = quads[q].dirx;
        __syncwarp();
        for (int i = lane; i < TXq * kTile; i += 32)
          edges[i] = (use_halo && i <= Exq) ? __ldg(p.halo[q] + (sx + dxq * i)) : 1.0;
        __syncwarp();
      }
#pragma unroll 1
      for (int J = quads[q].Jlo; J <= quads[q].Jhi && J < TYq; ++J) {
        const int I0 = Lm[q * lmcap + J];
        if (I0 < TXq) run_row(q, J, I0);
      }
    }
  } else {
    // a warp that finishes a row takes the next one in (J, quadrant) order from a shared
    // counter: a row only waits for the row below it, which was taken earlier
    int maxTY = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) maxTY = max(maxTY, quads[q].TY);
#pragma unroll 1
    for (;;) {
      int c = 0;
      if (lane == 0) c = atomicAdd(next_row, 1);
      c = __shfl_sync(kAll, c, 0);
      if (c >= 4 * maxTY) break;
      const int J = c >> 2, q = c & 3;
      if (J >= quads[q].TY || J < quads[q].Jlo || J > quads[q].Jhi) continue;
      const int I0 = Lm[q * lmcap + J];
      if (I0 >= quads[q].TX) continue; // the whole row is lit
      run_row(q, J, I0);
    }
  }
  __syncthreads();
}

} // namespace
#endif
