// giant.cu -- the planner on ONE map whose rows are partitioned into strips (SURVEY 8e,
// BASELINE configs[4]): engine + C-ABI (vhp_giant_*).  Also the route of vhp_planner_batch for a
// few large problems (one strip = the whole map, one process).
//
// Replaces solve() / updateVisibility() / reconstructPath() of the reference
// (src/visibilityBasedSolver.cpp:76-160, :379-565, :1183-1213) for a map that is spread over the
// GPUs of a box, one process per GPU:
//
//   * every rank keeps the bit planes of the whole occupancy map (a few MB) and the rows
//     [y0, y1) of the fp64 working fields (visibility, global visibility, cached heuristic,
//     parents: 28 bytes per cell);
//   * one planner iteration = two chains of strip sweeps that run at the same time on two
//     streams.  The UP chain sweeps the +y quadrants (Q1, Q2), strips in ascending order; the
//     DOWN chain the -y quadrants (Q3, Q4) in descending order.  A strip hands its neighbour
//     the two fp64 visibility rows below that neighbour's first tile rows (2 x nx doubles,
//     ncclSend / ncclRecv over NVLink, a device copy between strips of one process).  The
//     communication pattern does not depend on where the source is -- strips the chain has not
//     reached the source in yet have nothing to compute and pass the (unused) rows on -- so an
//     iteration is a FIXED sequence of launches whose data-dependent inputs (source, loop
//     state, query) are read from device memory (kernels_giant.cu);
//   * then the per-cell epilogue + arg-min per strip, an ncclAllGather of 32 bytes per rank
//     {h bits, push-order key, vg(end) bits}, and the loop control of solve() on every rank.
//
// One strip per rank (the production layout): the ranks map each other's sweep workspaces
// (cudaIpc*) and a strip boundary is handed over TILE BY TILE through peer memory: the warp that
// finishes a tile of the row below the neighbour's first tile row stores its top row into the
// neighbour's boundary row over NVLink and raises the neighbour's progress flag, so all strips
// of a chain run as ONE wavefront, one tile apart, and the sweep's critical path is that of a
// single GPU (sweep_tile_body.cuh, TileArgs::x_edges).  ncclSend / ncclRecv of finished rows
// remains the fallback (several strips per rank, peer mapping unavailable, VHP_GIANT_P2P=0).
//
// No host round trip inside the loop.  One process: the iteration is captured once as the
// body of a CUDA-graph WHILE node whose condition the step kernel sets.  Several ranks (NCCL
// between the launches): the host enqueues iterations in batches and reads a 48-byte snapshot
// of the loop state one batch behind, so the GPU never waits for it; iterations enqueued
// after the loop ended return at once.  All ranks take the same decisions from the same
// snapshots, so their NCCL calls stay matched.
#include <algorithm>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "giant_internal.h"
#include "nccl_shim.h"

struct vhp_giant {
  vhp_context *ctx = nullptr;
  int nx = 0, ny = 0, rank = 0, world = 1, spr = 1, nstrips = 1, k0 = 0;
  std::vector<int> bounds; // row bounds of all strips, nstrips + 1 entries
  bool borrowed = false;   // planes / fields / outputs belong to the caller (vhp_planner_batch route)
  uint32_t *plane_buf = nullptr;
  VhpTilePlanes pl;
  char *field_buf = nullptr;
  GiantLocal loc;
  char *small_buf = nullptr; // everything below, one allocation
  double *halo = nullptr;    // [local strip][4][nx]
  double *send_up = nullptr, *send_dn = nullptr; // [2][nx]
  void *ws[2] = {nullptr, nullptr};              // grid-sweep workspaces of the two chains
  unsigned long long *bests = nullptr, *partial = nullptr, *key_send = nullptr, *key_all = nullptr;
  int nblocks = 0;
  int *ctl = nullptr;
  int32_t *ls = nullptr, *came_at = nullptr;
  int ls_cap = 0;
  int32_t *o_status = nullptr, *o_nb = nullptr, *o_pn = nullptr, *o_iters = nullptr, *o_path = nullptr;
  double *o_plen = nullptr;
  cudaStream_t s_dn = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_snap[2] = {nullptr, nullptr};
  cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
  std::vector<cudaEvent_t> ev_up; // "up sweep of local strip s done" (see enqueue_iteration)
  int *h_snap = nullptr;          // pinned, 2 x kGiantCtlInts
  char *h_out = nullptr;          // pinned staging of the small outputs
  size_t h_out_cap = 0;
  const VhpNccl *nccl = nullptr;
  vhpNcclComm comm_up = nullptr, comm_dn = nullptr;
  // peer hand-over of the strip boundaries (one strip per rank): both sweep workspaces in one
  // IPC-shareable allocation; the neighbours' copies mapped into this process
  bool p2p = false;
  char *p2p_buf = nullptr;
  size_t p2p_stride = 0;
  void *peer_next = nullptr, *peer_prev = nullptr; // p2p_buf of rank + 1 / rank - 1
  // loop: 0 automatic (graph for one process, batches otherwise), 1 graph, 2 batches,
  // 3 one host read-back per iteration (the round-1 behaviour; kept for A/B measurements)
  int loop_mode = 0;
  int batch = 4; // iterations enqueued per snapshot in mode 2
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  bool graph_failed = false;
  // what the capture baked into the sweep nodes: the context's ratio table (ensure_rcp2 frees it
  // when it grows) and its grid-sweep mode (vhp_i_grid_ctas fixes the CTA count)
  const double *graph_rcp2 = nullptr;
  int graph_grid_sweep = -1;
  // NCCL timing trace (env VHP_GIANT_TRACE or stats requested in mode 2)
  bool trace = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> trace_ev;
  size_t trace_used = 0;
  int64_t nccl_ops = 0;
};

namespace {

#define GCUDA(g, call)                                                           \
  do {                                                                           \
    cudaError_t e_ = (call);                                                     \
    if (e_ != cudaSuccess)                                                       \
      return vhp_i_fail((g)->ctx, VHP_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

#define GNCCL(g, call)                                                           \
  do {                                                                           \
    int r_ = (call);                                                             \
    if (r_ != 0)                                                                 \
      return vhp_i_fail((g)->ctx, VHP_ERR_CUDA,                                  \
                        std::string(#call) + ": NCCL error " + (g)->nccl->GetErrorString(r_)); \
  } while (0)

void strip_bounds(int ny, int nstrips, std::vector<int> &b) {
  b.resize(nstrips + 1);
  const int base = ny / nstrips, rem = ny % nstrips; // contiguous blocks, sizes differ by <= 1
  b[0] = 0;
  for (int k = 0; k < nstrips; ++k) b[k + 1] = b[k] + base + (k < rem ? 1 : 0);
}

double *halo_of(const vhp_giant *g, int s) { return g->halo + (size_t)s * 4 * g->nx; }

vhp_status sweep_strip(vhp_giant *g, int s, int qmask, cudaStream_t st, void *ws,
                       const VhpSweepPeer *peer = nullptr) {
  const GiantStripDev &sd = g->loc.s[s];
  const double *h[4];
  for (int q = 0; q < 4; ++q) // (a boundary that arrives through peer memory has no halo row)
    h[q] = (peer && ((peer->remote_mask >> q) & 1)) ? nullptr : halo_of(g, s) + (size_t)q * g->nx;
  int ctas = vhp_i_grid_ctas(g->ctx, g->nx, g->ny, sd.y1 - sd.y0);
  if (qmask == 0xF && ctas > 1) // all four quadrants in one launch: twice the warps of one chain's launch
    ctas = std::min(2 * g->ctx->sm_count, 2 * ctas);
  if (peer) // grid mode whatever the size, and at most one CTA per SM: the two chains' kernels must
            // be resident together (each may be waiting for the other GPU's other chain)
    ctas = std::max(2, std::min(g->ctx->sm_count, (4 * ((sd.y1 - sd.y0) / 32 + 2) + 7) / 8));
  GCUDA(g, vhp_launch_sweep_window(g->pl, g->nx, g->ny, 0, 0, sd.y0, sd.y1, h, VHP_F64, sd.vis,
                                   g->ctx->rcp2_table, g->ctx->d_err, ctas > 1 ? ws : nullptr, ctas, st,
                                   &g->ctx->launches, qmask, g->ctl, peer));
  return VHP_OK;
}

// NCCL op with optional timing events around it
template <typename F>
vhp_status traced(vhp_giant *g, cudaStream_t st, F &&op) {
  const bool tr = g->trace && g->trace_used < g->trace_ev.size();
  if (tr) GCUDA(g, cudaEventRecord(g->trace_ev[g->trace_used].first, st));
  GNCCL(g, op());
  if (tr) GCUDA(g, cudaEventRecord(g->trace_ev[g->trace_used++].second, st));
  ++g->nccl_ops;
  return VHP_OK;
}

// One planner iteration: a fixed sequence of launches (see the header of this file).
vhp_status enqueue_iteration(vhp_giant *g, unsigned long long cond, int use_cond) {
  cudaStream_t S = g->ctx->stream, D = g->s_dn;
  const int n = g->loc.n, nx = g->nx, ny = g->ny, last = g->nstrips - 1;
  const size_t row2 = 2 * (size_t)nx;
  vhp_status st;
  if (g->nstrips == 1) {
    // one strip: nothing to hand over, all four quadrants in one launch
    if ((st = sweep_strip(g, 0, 0xF, S, g->ws[0])) != VHP_OK) return st;
  } else if (g->p2p) {
    // one strip per rank, boundaries through peer memory: both chains start at once on every
    // rank and synchronise tile by tile inside the kernels
    const int k = g->k0;
    size_t foff, fbytes;
    vhp_sweep_grid_ws_flags(nx, ny, &foff, &fbytes);
    GCUDA(g, cudaEventRecord(g->ev_fork, S));
    GCUDA(g, cudaStreamWaitEvent(D, g->ev_fork, 0));
    VhpSweepPeer up, dn;
    if (k < last) { up.x_ws = (char *)g->peer_next; up.x_y0 = g->bounds[k + 1]; up.x_y1 = g->bounds[k + 2]; }
    up.remote_mask = k > 0 ? 0x3 : 0;
    if (k > 0) { dn.x_ws = (char *)g->peer_prev + g->p2p_stride; dn.x_y0 = g->bounds[k - 1]; dn.x_y1 = g->bounds[k]; }
    dn.remote_mask = k < last ? 0xC : 0;
    if ((st = sweep_strip(g, 0, 0x3, S, g->ws[0], &up)) != VHP_OK) return st;
    GCUDA(g, cudaMemsetAsync((char *)g->ws[0] + foff, 0, fbytes, S)); // flags the neighbour raised
    if ((st = sweep_strip(g, 0, 0xC, D, g->ws[1], &dn)) != VHP_OK) return st;
    GCUDA(g, cudaMemsetAsync((char *)g->ws[1] + foff, 0, fbytes, D));
    GCUDA(g, cudaEventRecord(g->ev_join, D));
    GCUDA(g, cudaStreamWaitEvent(S, g->ev_join, 0));
  } else {
  GCUDA(g, cudaEventRecord(g->ev_fork, S));
  GCUDA(g, cudaStreamWaitEvent(D, g->ev_fork, 0));
  // ---- UP chain: +y quadrants, ascending strips, stream S
  for (int s = 0; s < n; ++s) {
    const int k = g->k0 + s;
    if (k > 0) {
      if (s == 0) {
        if ((st = traced(g, S, [&] { return g->nccl->Recv(halo_of(g, 0), row2, kNcclFloat64, g->rank - 1, g->comm_up, S); })) != VHP_OK)
          return st;
      } else {
        GCUDA(g, vhp_launch_giant_halo_gather(g->ctl, nx, ny, g->loc.s[s - 1], g->loc.s[s].y0, g->loc.s[s].y1,
                                              0, halo_of(g, s), S, &g->ctx->launches));
      }
    }
    if ((st = sweep_strip(g, s, 0x3, S, g->ws[0])) != VHP_OK) return st;
    GCUDA(g, cudaEventRecord(g->ev_up[s], S));
    if (k < last && s == n - 1) {
      GCUDA(g, vhp_launch_giant_halo_gather(g->ctl, nx, ny, g->loc.s[s], g->bounds[k + 1], g->bounds[k + 2], 0,
                                            g->send_up, S, &g->ctx->launches));
      if ((st = traced(g, S, [&] { return g->nccl->Send(g->send_up, row2, kNcclFloat64, g->rank + 1, g->comm_up, S); })) != VHP_OK)
        return st;
    }
  }
  // ---- DOWN chain: -y quadrants, descending strips, stream D
  for (int s = n - 1; s >= 0; --s) {
    const int k = g->k0 + s;
    if (k < last) {
      if (s == n - 1) {
        if ((st = traced(g, D, [&] { return g->nccl->Recv(halo_of(g, s) + row2, row2, kNcclFloat64, g->rank + 1, g->comm_dn, D); })) != VHP_OK)
          return st;
      } else {
        GCUDA(g, vhp_launch_giant_halo_gather(g->ctl, nx, ny, g->loc.s[s + 1], g->loc.s[s].y0, g->loc.s[s].y1,
                                              2, halo_of(g, s) + row2, D, &g->ctx->launches));
      }
    }
    if ((st = sweep_strip(g, s, 0xC, D, g->ws[1])) != VHP_OK) return st;
    // The halo row of a -y quadrant can be the source's own row (first tile row one cell high),
    // which the +y quadrants store: the rows handed down must see the UP sweep of this strip.
    if (k > 0) GCUDA(g, cudaStreamWaitEvent(D, g->ev_up[s], 0));
    if (k > 0 && s == 0) {
      GCUDA(g, vhp_launch_giant_halo_gather(g->ctl, nx, ny, g->loc.s[0], g->bounds[k - 1], g->bounds[k], 2,
                                            g->send_dn, D, &g->ctx->launches));
      if ((st = traced(g, D, [&] { return g->nccl->Send(g->send_dn, row2, kNcclFloat64, g->rank - 1, g->comm_dn, D); })) != VHP_OK)
        return st;
    }
  }
  GCUDA(g, cudaEventRecord(g->ev_join, D));
  GCUDA(g, cudaStreamWaitEvent(S, g->ev_join, 0));
  }
  // ---- epilogue + arg-min per strip, exchange, loop control
  for (int s = 0; s < n; ++s) {
    const GiantStripDev &sd = g->loc.s[s];
    GCUDA(g, vhp_launch_strip_epilogue(nx, ny, sd.y0, sd.y1, 0, 0, 0, 0, 0.0, 0, g->ls, sd.vis, sd.vg, sd.hc,
                                       sd.came, g->partial, g->nblocks, g->bests + 2 * s, S,
                                       &g->ctx->launches, g->ctl));
  }
  GCUDA(g, vhp_launch_giant_pack_key(g->ctl, g->bests, g->loc, nx, g->key_send, S, &g->ctx->launches));
  const unsigned long long *all = g->key_send;
  if (g->world > 1) {
    if ((st = traced(g, S, [&] { return g->nccl->AllGather(g->key_send, g->key_all, 4, kNcclUint64, g->comm_up, S); })) != VHP_OK)
      return st;
    all = g->key_all;
  }
  GCUDA(g, vhp_launch_giant_step(all, g->world, g->ctl, g->ls, cond, use_cond, S, &g->ctx->launches));
  return VHP_OK;
}

// CUDA graph: one WHILE node whose body is one iteration; the step kernel sets the condition.
vhp_status build_graph(vhp_giant *g) {
  cudaStream_t S = g->ctx->stream;
  g->graph_rcp2 = g->ctx->rcp2_table;
  g->graph_grid_sweep = g->ctx->grid_sweep;
  GCUDA(g, cudaGraphCreate(&g->graph, 0));
  cudaGraphConditionalHandle handle;
  GCUDA(g, cudaGraphConditionalHandleCreate(&handle, g->graph, 1, cudaGraphCondAssignDefault));
  cudaGraphNodeParams np = {};
  np.type = cudaGraphNodeTypeConditional;
  np.conditional.handle = handle;
  np.conditional.type = cudaGraphCondTypeWhile;
  np.conditional.size = 1;
  cudaGraphNode_t node;
  GCUDA(g, cudaGraphAddNode(&node, g->graph, nullptr, 0, &np));
  cudaGraph_t body = np.conditional.phGraph_out[0];
  GCUDA(g, cudaStreamBeginCaptureToGraph(S, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
  const int64_t launches0 = g->ctx->launches; // capturing launches nothing
  vhp_status st = enqueue_iteration(g, (unsigned long long)handle, 1);
  g->ctx->launches = launches0;
  cudaGraph_t captured = nullptr;
  cudaError_t e = cudaStreamEndCapture(S, &captured);
  if (st != VHP_OK) return st;
  if (e != cudaSuccess) return vhp_i_fail(g->ctx, VHP_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
  GCUDA(g, cudaGraphInstantiate(&g->exec, g->graph, 0));
  return VHP_OK;
}

void drop_graph(vhp_giant *g) {
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->graph) cudaGraphDestroy(g->graph);
  g->exec = nullptr;
  g->graph = nullptr;
}

int launches_per_iteration(const vhp_giant *g) {
  int n = 0;
  for (int s = 0; s < g->loc.n; ++s) {
    const int ctas = vhp_i_grid_ctas(g->ctx, g->nx, g->ny, g->loc.s[s].y1 - g->loc.s[s].y0);
    n += (g->nstrips == 1 ? 1 : 2) * (ctas > 1 ? 2 : 1) + 2; // sweep(s), epilogue + its reduction
    if (g->k0 + s > 0) n += 1;                       // halo rows handed up / down (local copy
    if (g->k0 + s < g->nstrips - 1) n += 1;          // or the gather in front of a send)
  }
  return n + 2;                                      // key packing, loop control
}

// the loop of solve() (:127-140); the state is in g->ctl
vhp_status run_loop(vhp_giant *g, int max_iter, int *iters_out) {
  cudaStream_t S = g->ctx->stream;
  int mode = g->loop_mode;
  if (mode == 0) mode = g->world > 1 ? 2 : 1;
  if (mode == 1 && g->world > 1) mode = 2; // NCCL calls are not captured
  if ((g->exec || g->graph_failed) &&
      (g->graph_rcp2 != g->ctx->rcp2_table || g->graph_grid_sweep != g->ctx->grid_sweep)) {
    drop_graph(g); // its sweeps would read a freed table or run a stale CTA count: capture again
    g->graph_failed = false;
  }
  if (mode == 1 && !g->exec && !g->graph_failed) {
    const vhp_status st = build_graph(g);
    if (st != VHP_OK) { // e.g. a driver without conditional nodes: fall back to batches
      drop_graph(g);
      g->graph_failed = true;
      (void)cudaGetLastError();
    }
  }
  if (mode == 1 && g->exec) {
    GCUDA(g, cudaGraphLaunch(g->exec, S));
    // launches the graph performed: known after the loop, from the iteration counter
    GCUDA(g, cudaMemcpyAsync(g->h_snap, g->ctl, kGiantCtlInts * sizeof(int), cudaMemcpyDeviceToHost, S));
    GCUDA(g, cudaStreamSynchronize(S));
    const int it = std::max(1, g->h_snap[5]);
    g->ctx->launches += (int64_t)it * launches_per_iteration(g);
    *iters_out = g->h_snap[5];
    return VHP_OK;
  }
  vhp_status st;
  if (mode == 3) { // one read-back per iteration
    for (;;) {
      GCUDA(g, cudaMemcpyAsync(g->h_snap, g->ctl, kGiantCtlInts * sizeof(int), cudaMemcpyDeviceToHost, S));
      GCUDA(g, cudaStreamSynchronize(S));
      if (g->h_snap[0]) break;
      if ((st = enqueue_iteration(g, 0, 0)) != VHP_OK) return st;
    }
    *iters_out = g->h_snap[5];
    return VHP_OK;
  }
  // batches of K iterations; after batch j a snapshot of the loop state follows it down the
  // stream.  Before batch j + 1 goes out the host reads snapshot j - 1, i.e. it stays one whole
  // batch ahead of the GPU, which therefore never waits for the host.  Every rank sees the
  // same snapshots, takes the same decisions and issues the same NCCL calls.
  const int K = std::max(1, g->batch);
  const int max_batches = (max_iter + 2 + K - 1) / K + 1;
  int j = 0;
  while (j < max_batches) {
    for (int i = 0; i < K; ++i)
      if ((st = enqueue_iteration(g, 0, 0)) != VHP_OK) return st;
    ++j;
    GCUDA(g, cudaMemcpyAsync(g->h_snap + (j & 1) * kGiantCtlInts, g->ctl, kGiantCtlInts * sizeof(int),
                             cudaMemcpyDeviceToHost, S));
    GCUDA(g, cudaEventRecord(g->ev_snap[j & 1], S));
    if (j >= 2) {
      GCUDA(g, cudaEventSynchronize(g->ev_snap[(j - 1) & 1]));
      if (g->h_snap[((j - 1) & 1) * kGiantCtlInts]) break;
    }
  }
  GCUDA(g, cudaEventSynchronize(g->ev_snap[j & 1]));
  if (!g->h_snap[(j & 1) * kGiantCtlInts])
    return vhp_i_fail(g->ctx, VHP_ERR_CUDA, "strip planner: the loop did not end within max_iter + 2 iterations");
  *iters_out = g->h_snap[(j & 1) * kGiantCtlInts + 5];
  return VHP_OK;
}

vhp_status alloc_small(vhp_giant *g, int ls_cap) {
  // (re)allocate everything that depends on ls_cap; the graph holds these pointers
  if (g->small_buf && ls_cap <= g->ls_cap) return VHP_OK;
  drop_graph(g);
  g->graph_failed = false;
  if (g->small_buf) {
    GCUDA(g, cudaStreamSynchronize(g->ctx->stream));
    GCUDA(g, cudaFree(g->small_buf));
    g->small_buf = nullptr;
  }
  const int n = g->loc.n, nx = g->nx;
  g->nblocks = vhp_strip_epilogue_blocks(g->ctx->sm_count);
  const size_t ws_bytes = (vhp_sweep_grid_ws_bytes(nx, g->ny) + 255) & ~(size_t)255;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
  const size_t o_halo = take((size_t)n * 4 * nx * 8), o_su = take(2 * (size_t)nx * 8), o_sd = take(2 * (size_t)nx * 8);
  const size_t o_ws0 = take(ws_bytes), o_ws1 = take(ws_bytes);
  const size_t o_bests = take((size_t)n * 16), o_part = take((size_t)g->nblocks * 16);
  const size_t o_ks = take(32), o_ka = take((size_t)g->world * 32), o_ctl = take(kGiantCtlInts * 4);
  const size_t o_ls = take((size_t)ls_cap * 8), o_ca = take((size_t)ls_cap * 4);
  const size_t o_out = take(64), o_path = take((size_t)ls_cap * 8);
  GCUDA(g, cudaMalloc(&g->small_buf, off));
  GCUDA(g, cudaMemsetAsync(g->small_buf, 0, off, g->ctx->stream));
  char *b = g->small_buf;
  g->halo = (double *)(b + o_halo); g->send_up = (double *)(b + o_su); g->send_dn = (double *)(b + o_sd);
  if (!g->p2p) { g->ws[0] = b + o_ws0; g->ws[1] = b + o_ws1; }
  g->bests = (unsigned long long *)(b + o_bests); g->partial = (unsigned long long *)(b + o_part);
  g->key_send = (unsigned long long *)(b + o_ks); g->key_all = (unsigned long long *)(b + o_ka);
  g->ctl = (int *)(b + o_ctl);
  if (!g->borrowed) g->ls = (int32_t *)(b + o_ls);
  g->came_at = (int32_t *)(b + o_ca);
  g->o_plen = (double *)(b + o_out);
  g->o_status = (int32_t *)(b + o_out + 8); g->o_nb = g->o_status + 1; g->o_pn = g->o_status + 2; g->o_iters = g->o_status + 3;
  g->o_path = (int32_t *)(b + o_path);
  g->ls_cap = ls_cap;
  return VHP_OK;
}

vhp_status create_common(vhp_giant *g) {
  GCUDA(g, cudaStreamCreateWithFlags(&g->s_dn, cudaStreamNonBlocking));
  GCUDA(g, cudaEventCreateWithFlags(&g->ev_fork, cudaEventDisableTiming));
  GCUDA(g, cudaEventCreateWithFlags(&g->ev_join, cudaEventDisableTiming));
  for (int i = 0; i < 2; ++i) GCUDA(g, cudaEventCreateWithFlags(&g->ev_snap[i], cudaEventDisableTiming));
  GCUDA(g, cudaEventCreate(&g->ev_t0));
  GCUDA(g, cudaEventCreate(&g->ev_t1));
  g->ev_up.resize(g->loc.n);
  for (auto &e : g->ev_up) GCUDA(g, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  GCUDA(g, cudaHostAlloc(&g->h_snap, 2 * kGiantCtlInts * sizeof(int), cudaHostAllocDefault));
  if (const char *e = std::getenv("VHP_GIANT_LOOP")) g->loop_mode = std::atoi(e);
  if (const char *e = std::getenv("VHP_GIANT_BATCH")) g->batch = std::max(1, std::atoi(e));
  g->trace = std::getenv("VHP_GIANT_TRACE") != nullptr;
  return VHP_OK;
}

// Map the neighbours' sweep workspaces (one strip per rank).  Every rank must take the same
// decision, so the outcome is agreed with an all-reduce; on any failure all ranks keep the
// ncclSend / ncclRecv hand-over.
vhp_status setup_p2p(vhp_giant *g) {
  g->p2p = false;
  if (g->spr != 1) return VHP_OK;
  if (const char *e = std::getenv("VHP_GIANT_P2P"))
    if (std::atoi(e) == 0) return VHP_OK;
  cudaStream_t S = g->ctx->stream;
  const size_t stride = (vhp_sweep_grid_ws_bytes(g->nx, g->ny) + 4095) & ~(size_t)4095;
  int ok = 1;
  cudaIpcMemHandle_t mine;
  std::memset(&mine, 0, sizeof(mine));
  if (cudaMalloc(&g->p2p_buf, 2 * stride) != cudaSuccess || cudaMemset(g->p2p_buf, 0, 2 * stride) != cudaSuccess ||
      cudaIpcGetMemHandle(&mine, g->p2p_buf) != cudaSuccess)
    ok = 0;
  (void)cudaGetLastError();
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  // all-gather of the handles and of the verdicts through device memory
  char *d_x = nullptr;
  const size_t xb = 64 + 64 * (size_t)g->world + 16;
  GCUDA(g, cudaMalloc(&d_x, xb));
  std::vector<char> h_all(64 * (size_t)g->world);
  auto fin = [&](vhp_status r) { cudaFree(d_x); return r; };
  GCUDA(g, cudaMemcpyAsync(d_x, &mine, 64, cudaMemcpyHostToDevice, S));
  { const int r = g->nccl->AllGather(d_x, d_x + 64, 8, kNcclUint64, g->comm_up, S);
    if (r != 0) return fin(vhp_i_fail(g->ctx, VHP_ERR_CUDA, std::string("ncclAllGather: ") + g->nccl->GetErrorString(r))); }
  GCUDA(g, cudaMemcpyAsync(h_all.data(), d_x + 64, h_all.size(), cudaMemcpyDeviceToHost, S));
  GCUDA(g, cudaStreamSynchronize(S));
  auto open_peer = [&](int r, void **out) {
    if (!ok || r < 0 || r >= g->world) return;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, h_all.data() + 64 * (size_t)r, 64);
    if (cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      *out = nullptr;
      ok = 0;
      (void)cudaGetLastError();
    }
  };
  open_peer(g->rank + 1, &g->peer_next);
  open_peer(g->rank - 1, &g->peer_prev);
  // agree: min over the ranks of "everything worked here"
  int *d_ok = reinterpret_cast<int *>(d_x + 64 + 64 * (size_t)g->world);
  int neg = ok ? 0 : 1; // all-reduce (max) of the failure flags
  GCUDA(g, cudaMemcpyAsync(d_ok, &neg, sizeof(int), cudaMemcpyHostToDevice, S));
  { const int r = g->nccl->AllReduce(d_ok, d_ok, 1, kNcclInt32, kNcclMax, g->comm_up, S);
    if (r != 0) return fin(vhp_i_fail(g->ctx, VHP_ERR_CUDA, std::string("ncclAllReduce: ") + g->nccl->GetErrorString(r))); }
  GCUDA(g, cudaMemcpyAsync(&neg, d_ok, sizeof(int), cudaMemcpyDeviceToHost, S));
  GCUDA(g, cudaStreamSynchronize(S));
  if (neg == 0) {
    g->p2p = true;
    g->p2p_stride = stride;
    g->ws[0] = g->p2p_buf;
    g->ws[1] = g->p2p_buf + stride;
  }
  return fin(VHP_OK);
}

void destroy_giant(vhp_giant *g) {
  if (!g) return;
  cudaSetDevice(g->ctx->device);
  cudaStreamSynchronize(g->ctx->stream);
  if (g->s_dn) cudaStreamSynchronize(g->s_dn);
  drop_graph(g);
  if (g->peer_next) cudaIpcCloseMemHandle(g->peer_next);
  if (g->peer_prev) cudaIpcCloseMemHandle(g->peer_prev);
  if (g->p2p_buf) cudaFree(g->p2p_buf);
  if (g->nccl) {
    if (g->comm_dn) g->nccl->CommDestroy(g->comm_dn);
    if (g->comm_up) g->nccl->CommDestroy(g->comm_up);
  }
  for (auto &p : g->trace_ev) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
  for (auto &e : g->ev_up) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : {g->ev_fork, g->ev_join, g->ev_snap[0], g->ev_snap[1], g->ev_t0, g->ev_t1})
    if (e) cudaEventDestroy(e);
  if (g->s_dn) cudaStreamDestroy(g->s_dn);
  if (g->h_snap) cudaFreeHost(g->h_snap);
  if (g->h_out) cudaFreeHost(g->h_out);
  if (g->small_buf) cudaFree(g->small_buf);
  if (!g->borrowed) {
    if (g->field_buf) cudaFree(g->field_buf);
    if (g->plane_buf) cudaFree(g->plane_buf);
  }
  delete g;
}

} // namespace

// ---- route of vhp_planner_batch for one large problem (capi.cu: planner_dev) ------------------
// The caller owns planes, fields (one strip = the whole map), the light-source list and the
// outputs; the engine (and its captured graph) is cached in the context for as long as those
// pointers stay the same, which they do for repeated solves through one context.
vhp_status vhp_i_grid_planner_run(vhp_context *ctx, const VhpTilePlanes &pl, int nx, int ny,
                                  const int32_t se[4], double thr, int32_t max_iter, int32_t ls_cap,
                                  double *vis, double *vg, double *hc, int32_t *came, int32_t *ls) {
  vhp_giant *g = ctx->grid_engine;
  const bool same = g && g->nx == nx && g->ny == ny && g->pl.rowF == pl.rowF && g->pl.bsum == pl.bsum &&
                    g->loc.s[0].vis == vis && g->loc.s[0].vg == vg && g->loc.s[0].hc == hc &&
                    g->loc.s[0].came == came && g->ls == ls && g->ls_cap >= ls_cap &&
                    g->loop_mode == ctx->grid_loop_mode;
  if (!same) {
    if (g) destroy_giant(g);
    ctx->grid_engine = nullptr;
    g = new vhp_giant();
    g->ctx = ctx;
    g->nx = nx; g->ny = ny;
    g->borrowed = true;
    g->pl = pl;
    strip_bounds(ny, 1, g->bounds);
    g->loc.n = 1;
    g->loc.s[0] = GiantStripDev{0, ny, vis, vg, hc, came};
    g->ls = ls;
    vhp_status st = create_common(g);
    if (st == VHP_OK) st = alloc_small(g, ls_cap);
    if (st != VHP_OK) { destroy_giant(g); return st; }
    if (ctx->grid_loop_mode) g->loop_mode = ctx->grid_loop_mode;
    ctx->grid_engine = g;
  }
  cudaStream_t S = ctx->stream;
  GCUDA(g, vhp_launch_giant_reset(g->loc.s[0], nx, S, &ctx->launches));
  GCUDA(g, vhp_launch_giant_begin(g->pl, nx, ny, se, thr, max_iter, g->ls, g->loc, g->ctl, S, &ctx->launches));
  int iters = 0;
  return run_loop(g, max_iter, &iters);
}

const int *vhp_i_grid_planner_ctl(const vhp_context *ctx) { return ctx->grid_engine ? ctx->grid_engine->ctl : nullptr; }

void vhp_i_grid_planner_release(vhp_context *ctx) {
  if (ctx->grid_engine) destroy_giant(ctx->grid_engine);
  ctx->grid_engine = nullptr;
}

// ---- C-ABI ------------------------------------------------------------------------------------
extern "C" {

vhp_status vhp_giant_unique_id(void *id) {
  if (!id) return vhp_i_fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_giant_unique_id: null pointer");
  std::string why;
  const VhpNccl *n = vhp_nccl(&why);
  if (!n) return vhp_i_fail(nullptr, VHP_ERR_UNSUPPORTED, why);
  vhpNcclUniqueId uid;
  const int r = n->GetUniqueId(&uid);
  if (r != 0) return vhp_i_fail(nullptr, VHP_ERR_CUDA, std::string("ncclGetUniqueId: ") + n->GetErrorString(r));
  static_assert(sizeof(uid) == VHP_GIANT_ID_BYTES, "ncclUniqueId is 128 bytes");
  std::memcpy(id, &uid, sizeof(uid));
  return VHP_OK;
}

vhp_status vhp_giant_create(vhp_context *ctx, const uint8_t *occ, int nx, int ny, int rank, int world,
                            const void *id, int strips_per_rank, vhp_giant **out) {
  if (!out) return vhp_i_fail(ctx, VHP_ERR_INVALID_ARG, "vhp_giant_create: null out pointer");
  *out = nullptr;
  if (!ctx || !occ || nx < 1 || ny < 1 || world < 1 || rank < 0 || rank >= world ||
      strips_per_rank < 1 || strips_per_rank > kGiantMaxLocal || (world > 1 && !id))
    return vhp_i_fail(ctx, VHP_ERR_INVALID_ARG, "vhp_giant_create: bad argument");
  if (nx > 16384 || ny > 16384 || !vhp_sweep_grid_supported(nx, ny))
    return vhp_i_fail(ctx, VHP_ERR_UNSUPPORTED, "vhp_giant_create: grid larger than 16384 x 16384");
  const int nstrips = world * strips_per_rank;
  if (nstrips > 1 && ny / nstrips < 32)
    return vhp_i_fail(ctx, VHP_ERR_INVALID_ARG, "vhp_giant_create: strips must be at least 32 rows high (one tile row)");
  vhp_giant *g = new vhp_giant();
  g->ctx = ctx;
  auto bail = [&](vhp_status st) { destroy_giant(g); return st; };
#define GTRY(expr) do { vhp_status st_ = (expr); if (st_ != VHP_OK) return bail(st_); } while (0)
#define GTRYC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return bail(vhp_i_fail(ctx, VHP_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_))); } while (0)
  GTRYC(cudaSetDevice(ctx->device));
  g->nx = nx; g->ny = ny; g->rank = rank; g->world = world; g->spr = strips_per_rank; g->nstrips = nstrips;
  g->k0 = rank * strips_per_rank;
  strip_bounds(ny, nstrips, g->bounds);
  GTRY(vhp_i_ensure_rcp2(ctx, std::max(nx, ny) + 64));
  // bit planes of the whole map, private to this engine
  int wx, wy, nsum;
  vhp_tile_plane_geometry(nx, ny, &wx, &wy, &nsum);
  const size_t row_plane = (size_t)ny * wx, col_plane = (size_t)nx * wy;
  const size_t plane_bytes = (2 * (row_plane + col_plane) + nsum) * sizeof(uint32_t);
  const size_t cells = (size_t)nx * ny;
  uint8_t *d_occ = nullptr;
  GTRYC(cudaMalloc(&g->plane_buf, plane_bytes));
  GTRYC(cudaMalloc(&d_occ, cells));
  cudaStream_t S = ctx->stream;
  cudaError_t e = cudaMemcpyAsync(d_occ, occ, cells, cudaMemcpyHostToDevice, S);
  uint32_t *rowF = g->plane_buf, *rowR = rowF + row_plane, *colF = rowR + row_plane, *colR = colF + col_plane,
           *bsum = colR + col_plane;
  if (e == cudaSuccess) e = vhp_launch_pack_tile(d_occ, 1, nx, ny, rowF, rowR, colF, colR, bsum, S, &ctx->launches);
  if (e == cudaSuccess) e = cudaStreamSynchronize(S);
  cudaFree(d_occ);
  GTRYC(e);
  g->pl.rowF = rowF; g->pl.rowR = rowR; g->pl.colF = colF; g->pl.colR = colR; g->pl.bsum = bsum;
  g->pl.wx = wx; g->pl.wy = wy; g->pl.row_plane = row_plane; g->pl.col_plane = col_plane;
  // this rank's strips of the working fields
  g->loc.n = strips_per_rank;
  const size_t my_rows = (size_t)(g->bounds[g->k0 + g->loc.n] - g->bounds[g->k0]);
  GTRYC(cudaMalloc(&g->field_buf, my_rows * nx * 28 + (size_t)g->loc.n * 4 * 256));
  {
    char *p = g->field_buf;
    for (int s = 0; s < g->loc.n; ++s) {
      GiantStripDev &sd = g->loc.s[s];
      sd.y0 = g->bounds[g->k0 + s]; sd.y1 = g->bounds[g->k0 + s + 1];
      const size_t c = (size_t)(sd.y1 - sd.y0) * nx;
      auto adv = [&](size_t bytes) { char *r = p; p += (bytes + 255) & ~(size_t)255; return r; };
      sd.vis = (double *)adv(8 * c);
      sd.vg = (double *)adv(8 * c);
      sd.hc = (double *)adv(8 * c);
      sd.came = (int32_t *)adv(4 * c);
    }
  }
  GTRY(create_common(g));
  if (world > 1) {
    std::string why;
    g->nccl = vhp_nccl(&why);
    if (!g->nccl) return bail(vhp_i_fail(ctx, VHP_ERR_UNSUPPORTED, why));
    vhpNcclUniqueId uid;
    std::memcpy(&uid, id, sizeof(uid));
    int r = g->nccl->CommInitRank(&g->comm_up, world, uid, rank);
    if (r == 0) r = g->nccl->CommSplit(g->comm_up, 0, rank, &g->comm_dn, nullptr);
    if (r != 0) return bail(vhp_i_fail(ctx, VHP_ERR_CUDA, std::string("NCCL communicator: ") + g->nccl->GetErrorString(r)));
    GTRY(setup_p2p(g));
  }
#undef GTRY
#undef GTRYC
  *out = g;
  return VHP_OK;
}

void vhp_giant_destroy(vhp_giant *g) { destroy_giant(g); }

vhp_status vhp_giant_strip_bounds(const vhp_giant *g, int strip, int *y0, int *y1) {
  if (!g || strip < 0 || strip >= g->nstrips) return vhp_i_fail(g ? g->ctx : nullptr, VHP_ERR_INVALID_ARG, "vhp_giant_strip_bounds: bad argument");
  if (y0) *y0 = g->bounds[strip];
  if (y1) *y1 = g->bounds[strip + 1];
  return VHP_OK;
}

vhp_status vhp_giant_local_rows(const vhp_giant *g, int *y0, int *y1) {
  if (!g) return vhp_i_fail(nullptr, VHP_ERR_INVALID_ARG, "vhp_giant_local_rows: null handle");
  if (y0) *y0 = g->bounds[g->k0];
  if (y1) *y1 = g->bounds[g->k0 + g->loc.n];
  return VHP_OK;
}

vhp_status vhp_giant_set_loop_mode(vhp_giant *g, int mode, int batch) {
  if (!g || mode < 0 || mode > 3 || batch < 0) return vhp_i_fail(g ? g->ctx : nullptr, VHP_ERR_INVALID_ARG, "vhp_giant_set_loop_mode: bad argument");
  g->loop_mode = mode;
  if (batch > 0) g->batch = batch;
  return VHP_OK;
}

vhp_status vhp_giant_solve(vhp_giant *g, const int32_t *se_xy, double threshold, int32_t max_iter,
                           int32_t ls_cap, vhp_dtype dtype, const vhp_planner_out *out,
                           vhp_giant_stats *stats) {
  static const vhp_planner_out none = {};
  const vhp_planner_out &o = out ? *out : none;
  if (!g || !se_xy || max_iter < 0 || ls_cap < max_iter + 2)
    return vhp_i_fail(g ? g->ctx : nullptr, VHP_ERR_INVALID_ARG, "vhp_giant_solve: bad argument (ls_cap must be >= max_iter + 2)");
  if ((o.vg || o.vis) && dtype != VHP_F64)
    return vhp_i_fail(g->ctx, VHP_ERR_UNSUPPORTED, "vhp_giant_solve: strip fields are exported as fp64 only");
  vhp_context *ctx = g->ctx;
  int prev_dev = -1;
  cudaGetDevice(&prev_dev);
  GCUDA(g, cudaSetDevice(ctx->device));
  struct Restore { int d; ~Restore() { if (d >= 0) cudaSetDevice(d); } } restore_{prev_dev};
  const auto t_begin = std::chrono::steady_clock::now();
  vhp_status st = alloc_small(g, ls_cap);
  if (st != VHP_OK) return st;
  const size_t host_bytes = 64 + 16 * (size_t)g->ls_cap;
  if (host_bytes > g->h_out_cap) {
    if (g->h_out) cudaFreeHost(g->h_out);
    g->h_out = nullptr;
    g->h_out_cap = 0;
    GCUDA(g, cudaHostAlloc(&g->h_out, host_bytes, cudaHostAllocDefault));
    g->h_out_cap = host_bytes;
  }
  const bool want_trace = g->trace || (stats && g->world > 1);
  if (want_trace && g->trace_ev.empty()) {
    g->trace_ev.resize(4096);
    for (auto &p : g->trace_ev) { GCUDA(g, cudaEventCreate(&p.first)); GCUDA(g, cudaEventCreate(&p.second)); }
  }
  const bool trace_saved = g->trace;
  g->trace = want_trace;
  g->trace_used = 0;
  g->nccl_ops = 0;
  const int64_t launches0 = ctx->launches;
  cudaStream_t S = ctx->stream;
  const int nx = g->nx;
  for (int s = 0; s < g->loc.n; ++s) GCUDA(g, vhp_launch_giant_reset(g->loc.s[s], nx, S, &ctx->launches));
  GCUDA(g, vhp_launch_giant_begin(g->pl, nx, g->ny, se_xy, threshold, max_iter, g->ls, g->loc, g->ctl, S, &ctx->launches));
  GCUDA(g, cudaEventRecord(g->ev_t0, S));
  int iters = 0;
  st = run_loop(g, max_iter, &iters);
  g->trace = trace_saved;
  if (st != VHP_OK) return st;
  GCUDA(g, cudaEventRecord(g->ev_t1, S));
  // reconstructPath: parents at the light sources and at the end point, from the owning ranks
  GCUDA(g, vhp_launch_giant_came_at(g->ctl, g->ls, nx, g->loc, g->ls_cap, g->came_at, S, &ctx->launches));
  if (g->world > 1)
    GNCCL(g, g->nccl->AllReduce(g->came_at, g->came_at, (size_t)g->ls_cap, kNcclInt32, kNcclMax, g->comm_up, S));
  GCUDA(g, vhp_launch_giant_finish(g->ctl, g->came_at, g->ls_cap, g->ls, g->o_status, g->o_nb, g->o_plen,
                                   g->o_pn, g->o_path, g->o_iters, S, &ctx->launches));
  char *h = g->h_out;
  GCUDA(g, cudaMemcpyAsync(h, g->o_plen, 64, cudaMemcpyDeviceToHost, S));
  GCUDA(g, cudaMemcpyAsync(h + 64, g->ls, 8 * (size_t)ls_cap, cudaMemcpyDeviceToHost, S));
  GCUDA(g, cudaMemcpyAsync(h + 64 + 8 * (size_t)g->ls_cap, g->o_path, 8 * (size_t)ls_cap, cudaMemcpyDeviceToHost, S));
  // this rank's rows of the fields
  size_t done_cells = 0;
  for (int s = 0; s < g->loc.n; ++s) {
    const GiantStripDev &sd = g->loc.s[s];
    const size_t c = (size_t)(sd.y1 - sd.y0) * nx;
    if (o.vis) GCUDA(g, cudaMemcpyAsync((double *)o.vis + done_cells, sd.vis, 8 * c, cudaMemcpyDeviceToHost, S));
    if (o.vg) GCUDA(g, cudaMemcpyAsync((double *)o.vg + done_cells, sd.vg, 8 * c, cudaMemcpyDeviceToHost, S));
    if (o.came) GCUDA(g, cudaMemcpyAsync(o.came + done_cells, sd.came, 4 * c, cudaMemcpyDeviceToHost, S));
    done_cells += c;
  }
  GCUDA(g, cudaStreamSynchronize(S));
  const double plen = *(const double *)h;
  const int32_t *small = (const int32_t *)(h + 8);
  if (o.status) *o.status = small[0];
  if (o.nb_sources) *o.nb_sources = small[1];
  if (o.path_n) *o.path_n = small[2];
  if (o.path_len) *o.path_len = plen;
  if (o.light_sources) std::memcpy(o.light_sources, h + 64, 8 * (size_t)ls_cap);
  if (o.path) std::memcpy(o.path, h + 64 + 8 * (size_t)g->ls_cap, 8 * (size_t)ls_cap);
  if (stats) {
    std::memset(stats, 0, sizeof(*stats));
    stats->iterations = small[3];
    int mode = g->loop_mode ? g->loop_mode : (g->world > 1 ? 2 : 1);
    if (mode == 1 && (g->world > 1 || !g->exec)) mode = 2;
    stats->loop_mode = mode;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g->ev_t0, g->ev_t1) == cudaSuccess) stats->loop_ms = ms;
    double nccl_ms = 0.0;
    for (size_t i = 0; i < g->trace_used; ++i) {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, g->trace_ev[i].first, g->trace_ev[i].second) == cudaSuccess) nccl_ms += t;
    }
    (void)cudaGetLastError();
    stats->nccl_ms = nccl_ms;
    stats->nccl_ops = g->nccl_ops;
    stats->nccl_ops_timed = (int64_t)g->trace_used;
    // (iterations enqueued after the loop ended also exchange rows; count the real ones)
    {
      const int sends = (g->k0 + g->loc.n < g->nstrips ? 1 : 0) + (g->k0 > 0 ? 1 : 0);
      stats->halo_bytes_sent = (int64_t)small[3] * sends * 2 * nx * 8;
    }
    stats->launches = ctx->launches - launches0;
    stats->peer_handover = g->p2p ? 1 : 0;
    if (g->p2p) stats->halo_bytes_sent = 0; // rows travel as peer stores inside the sweep kernels, tile by tile
    stats->solve_ms = 1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count();
  }
  int flag = 0;
  GCUDA(g, cudaMemcpy(&flag, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost));
  if (flag) {
    cudaMemset(ctx->d_err, 0, sizeof(int));
    if (flag & 2)
      return vhp_i_fail(ctx, VHP_ERR_CUDA, "strip planner: a neighbouring rank did not deliver its boundary rows (peer hand-over timed out)");
    return vhp_i_fail(ctx, VHP_ERR_INVALID_ARG, "a source / start / end point lies outside the grid");
  }
  return VHP_OK;
}

} // extern "C"
