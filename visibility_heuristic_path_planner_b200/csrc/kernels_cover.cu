// kernels_cover.cu -- greedy coverage placement (vhp_visibility_cover_greedy_batch): the fallback that turns fp64
// values into candidate coverage bits, and the greedy rounds over those bits.
//
// A candidate's coverage set S(c) is stored as bits over its box (VhpCoverBox, vhp_internal.h).  Per problem q the
// rounds keep state_q = ~target_q | U (the cells that no longer count) and, per candidate, gain(c) = |S(c) \ state|.
// A round is two launches and no host synchronisation:
//   apply  (one CTA per problem): take the argmax of the problem's key slot, record the pick, write
//          new = S(p) \ state into a per-problem scratch over p's box, OR S(p) into state (and `covered`);
//   update (32 candidates per CTA): a candidate whose box meets the pick's takes gain -= |S(c) & new| over the
//          intersection (a warp per such candidate, lanes over rows), then every candidate puts its key into the slot.
// The key (gain << 32) | ~index makes atomicMax pick the largest gain and, among equal gains, the smallest index
// within the group.  Every quantity is an integer, so the result does not depend on the order of the atomics.
//
// The weighted rounds (vhp_visibility_cover_greedy_weighted_batch) are the same kernels instantiated with kW = true:
// state starts as {W == 0} (cover_weight_kernel, which also copies the weights into a plane of 32-byte rows per word),
// gains are uint64 sums of the weights of the set bits (weight_sum), and the key is (gain << 28) | (2^28 - 1 - index).
//
// The m-fold rounds (vhp_visibility_cover_greedy_mfold_batch) are the weighted rounds with the apply step instantiated
// with kM = true: a per-problem plane of uint8 counters cnt(x) = min(m, picks whose S covers x) in wpad's layout, and
// state |= new, new = the cells that reach m this round (so a cell's weight leaves the gains only then).  Init and
// update are the weighted instances as they are: a gain is still sum W over S(c) \ state, and it changes only by new.
//
// The view call (vhp_visibility_cover_greedy_view_batch) narrows every S(c) to its candidate's view once, in place,
// with cover_view_kernel between phase 1 and the m-fold rounds; the rounds cannot tell masked bits from swept ones.
#include <algorithm>
#include <cstdint>
#include <type_traits>

#include "vhp_internal.h"

namespace {

constexpr unsigned kAll = 0xffffffffu;
constexpr int kCand = 32;  // candidates per CTA of the init / update kernels (lane l of warp 0 <-> candidate l)
constexpr int kWarps = 8;  // warps per CTA of those kernels
constexpr int kApplyThreads = 512;

constexpr int kIdxBits = 28; // index bits of the weighted key: gains fit the other 36 (2^28 cells of weight <= 255)
constexpr unsigned long long kIdxMask = (1ull << kIdxBits) - 1;

// gain of a candidate: a cell count, or a sum of uint8 weights
template <bool kW>
using GainT = typename std::conditional<kW, uint64_t, uint32_t>::type;

struct CoverGeo {
  int nx, ny, R, nw; // R: the radius clamped for the geometry; nw = ceil(nx / 32)
};

// bits lo .. hi of a word (any lo, hi; empty if lo > hi after clamping to [0, 31])
__device__ __forceinline__ uint32_t span_mask(int lo, int hi) {
  lo = max(lo, 0);
  hi = min(hi, 31);
  return lo > hi ? 0u : ((~0u >> (31 - hi)) & (~0u << lo));
}

__device__ __forceinline__ int isqrt_floor(int v) {
  int h = (int)sqrt((double)v);
  while (h * h > v) --h;
  while ((h + 1) * (h + 1) <= v) ++h;
  return h;
}

__device__ __forceinline__ uint32_t warp_sum(uint32_t v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(kAll, v, o);
  return v;
}

__device__ __forceinline__ uint64_t warp_sum(uint64_t v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(kAll, v, o);
  return v;
}

// sum of the weights of the set bits of m; w: the word's 32 weights (32-byte aligned), bit b <-> byte b.  Each nibble
// of m becomes a {0, 1} byte selector for __dp4a.
__device__ __forceinline__ uint32_t weight_sum(uint32_t m, const uint8_t *w) {
  const uint4 a = __ldg(reinterpret_cast<const uint4 *>(w)), b = __ldg(reinterpret_cast<const uint4 *>(w) + 1);
  const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) s = __dp4a(v[j], (((m >> (4 * j)) & 0xfu) * 0x00204081u) & 0x01010101u, s);
  return s;
}

// slot[g] = max(slot[g], key) for the valid lanes of a warp: one atomic when they share a problem
__device__ __forceinline__ void put_keys(const bool valid, const int32_t g, const unsigned long long key,
                                         unsigned long long *slot) {
  const unsigned vm = __ballot_sync(kAll, valid);
  if (!vm) return;
  const int lead = __ffs(vm) - 1, lane = threadIdx.x & 31;
  const int32_t g0 = __shfl_sync(kAll, g, lead);
  if (__all_sync(kAll, !valid || g == g0)) {
    unsigned long long m = valid ? key : 0ull;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const unsigned long long t = __shfl_xor_sync(kAll, m, o);
      m = t > m ? t : m;
    }
    if (lane == lead) atomicMax(slot + g0, m);
  } else if (valid) {
    atomicMax(slot + g, key);
  }
}

__device__ __forceinline__ unsigned long long key_of(uint32_t gain, int32_t k) {
  return ((unsigned long long)gain << 32) | (uint32_t)~k;
}
__device__ __forceinline__ unsigned long long key_of(uint64_t gain, int32_t k) {
  return ((unsigned long long)gain << kIdxBits) | (kIdxMask - (uint32_t)k);
}

// Fallback of phase 1: one thread per box word of pairs [p0, p0 + np).
__global__ void cover_fold_kernel(const double *__restrict__ val, int win_r, int64_t p0, int64_t np, CoverGeo G,
                                  bool disk, int r2, const int32_t *__restrict__ xy, double thr,
                                  uint32_t *__restrict__ bits) {
  const VhpCoverBox b0 = vhp_cover_box(G.nx, G.ny, G.R, 0, 0);
  const size_t hw = (size_t)b0.H * b0.W, total = (size_t)np * hw;
  const int P = 2 * win_r + 1;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int64_t j = (int64_t)(idx / hw), q = p0 + j;
    const int i = (int)(idx - (size_t)j * hw), rr = i / b0.W, w = i - rr * b0.W;
    const int sx = __ldg(xy + 2 * q), sy = __ldg(xy + 2 * q + 1);
    uint32_t m = 0;
    if ((unsigned)sx < (unsigned)G.nx && (unsigned)sy < (unsigned)G.ny) {
      const VhpCoverBox b = vhp_cover_box(G.nx, G.ny, G.R, sx, sy);
      const int y = b.y0 + rr, dy = y - sy;
      if (abs(dy) <= G.R) {
        // row y of the value source: a window centred on the candidate, or the whole field
        const double *row = win_r >= 0 ? val + (size_t)j * P * P + (ptrdiff_t)(dy + win_r) * P - (sx - win_r)
                                       : val + (size_t)j * G.nx * G.ny + (size_t)y * G.nx;
        const bool row_writes = !(y == 0 && sy != 0);
        for (int bit = 0; bit < 32; ++bit) {
          const int x = 32 * (b.w0 + w) + bit, dx = x - sx;
          if (x >= G.nx || abs(dx) > G.R || (disk && dx * dx + dy * dy > r2)) continue;
          if (row_writes && !(x == 0 && sx != 0) && __ldg(row + x) >= thr) m |= 1u << bit;
        }
      }
    }
    bits[(size_t)q * hw + i] = m;
  }
}

__global__ void cover_state_kernel(const uint32_t *__restrict__ target, size_t n, uint32_t *__restrict__ state) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    state[i] = ~__ldg(target + i);
}

// Weighted rounds, before init: wpad[q][y][w][0..31] = W_q of the word's 32 columns (0 beyond nx; weights null: 1) and
// state = {W == 0}, bits beyond nx included.  A thread per 4 columns (8 lanes per word): 4-byte stores, and the word's
// zero-weight bits gathered over its 8 lanes with shuffles.
__global__ void cover_weight_kernel(const uint8_t *__restrict__ wts, int64_t nprob, CoverGeo G,
                                    uint8_t *__restrict__ wpad, uint32_t *__restrict__ state) {
  const int lane = threadIdx.x & 31;
  const size_t n4 = (size_t)nprob * G.ny * G.nw * 8, step = (size_t)gridDim.x * blockDim.x;
  // the loop is uniform over the warp (i0 is its first thread's index), so every lane takes part in the shuffles
  for (size_t i0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x - lane; i0 < n4; i0 += step) {
    const size_t i = i0 + lane; // 4-column group i & 7 of word i >> 3
    uint32_t z = 0;
    if (i < n4) {
      const size_t word = i >> 3, row = word / G.nw; // row = q * ny + y
      const int x = 32 * (int)(word - row * G.nw) + 4 * (int)(i & 7);
      uint32_t v = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        uint32_t c = 0;
        if (x + b < G.nx) c = wts ? __ldg(wts + row * G.nx + x + b) : 1u;
        v |= c << (8 * b);
        z |= (uint32_t)(c == 0) << b;
      }
      reinterpret_cast<uint32_t *>(wpad)[i] = v;
    }
    uint32_t m = z << (4 * (lane & 7));
    m |= __shfl_xor_sync(kAll, m, 1);
    m |= __shfl_xor_sync(kAll, m, 2);
    m |= __shfl_xor_sync(kAll, m, 4);
    if ((lane & 7) == 0 && i < n4) state[i >> 3] = m;
  }
}

// gain(c) = |S(c) \ state| of 32 candidates per CTA (a warp per candidate, lanes over rows); disk_r2 >= 0: the disk
// mask dx^2 + dy^2 <= disk_r2 is applied to the bits in place first.  Then the keys of round 0, and first[q] = the
// problem's candidate of index 0 (the rounds read no group_ptr: the host form's copy of it may be gone by then).
// kW: the gain sums the weights of wpad (cover_weight_kernel's plane) instead of counting cells.
template <bool kW>
__global__ void __launch_bounds__(kWarps * 32) cover_init_kernel(uint32_t *__restrict__ bits, int64_t nsrc, CoverGeo G,
                                                                 int disk_r2, const int32_t *__restrict__ xy,
                                                                 const int32_t *__restrict__ pg,
                                                                 const int32_t *__restrict__ pk,
                                                                 const uint32_t *__restrict__ state,
                                                                 GainT<kW> *__restrict__ gain,
                                                                 unsigned long long *slot, int64_t *first,
                                                                 const uint8_t *__restrict__ wpad) {
  __shared__ GainT<kW> sg[kCand];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t base = blockIdx.x * (int64_t)kCand;
  const VhpCoverBox b0 = vhp_cover_box(G.nx, G.ny, G.R, 0, 0);
  const size_t hw = (size_t)b0.H * b0.W;
  for (int j = warp; j < kCand; j += kWarps) {
    const int64_t c = base + j;
    GainT<kW> acc = 0;
    const int32_t g = c < nsrc ? __ldg(pg + c) : -1;
    if (g >= 0) {
      const int sx = __ldg(xy + 2 * c), sy = __ldg(xy + 2 * c + 1);
      const VhpCoverBox b = vhp_cover_box(G.nx, G.ny, G.R, sx, sy);
      uint32_t *bc = bits + (size_t)c * hw;
      const uint32_t *sq = state + (size_t)g * G.ny * G.nw;
      for (int r = lane; r < b.H; r += 32) {
        const int y = b.y0 + r;
        int xa = 0, xb = -1; // the disk's columns on row y
        if (disk_r2 >= 0) {
          const int v = disk_r2 - (y - sy) * (y - sy);
          if (v >= 0) {
            const int h = isqrt_floor(v);
            xa = sx - h;
            xb = sx + h;
          }
        }
        uint32_t *row = bc + (size_t)r * b.W;
        const uint32_t *srow = sq + (size_t)y * G.nw + b.w0;
        for (int w = 0; w < b.W; ++w) {
          uint32_t m = row[w];
          if (disk_r2 >= 0 && m) {
            const int x0 = 32 * (b.w0 + w);
            const uint32_t mm = m & span_mask(xa - x0, xb - x0);
            if (mm != m) row[w] = mm;
            m = mm;
          }
          if constexpr (kW) {
            const uint32_t v = m ? m & ~__ldg(srow + w) : 0u;
            if (v) acc += weight_sum(v, wpad + (((size_t)g * G.ny + y) * G.nw + b.w0 + w) * 32);
          } else {
            if (m) acc += __popc(m & ~__ldg(srow + w));
          }
        }
      }
      acc = warp_sum(acc);
    }
    if (lane == 0) sg[j] = acc;
  }
  __syncthreads();
  if (warp == 0) {
    const int64_t c = base + lane;
    const int32_t g = c < nsrc ? __ldg(pg + c) : -1;
    const GainT<kW> gn = sg[lane];
    const int32_t kc = g >= 0 ? __ldg(pk + c) : -1;
    if (c < nsrc) gain[c] = gn;
    if (kc == 0) first[g] = c;
    put_keys(g >= 0, g, key_of(gn, kc), slot);
  }
}

// Round r, one CTA per problem: take the slot's pick (gain 0 or a finished problem: done), record it, and update the
// problem's state over the pick's box.  kM (m-fold, with kW): cnt += 1 over S(p) saturating at mfold (cnt: the
// counter plane, wpad's layout), new = the cells that reach mfold now and are not in state, state |= new, and the
// pick's gain is zeroed (with mfold >= 2 it keeps gain on its own cells).  gain, cnt and mfold are unused otherwise.
template <bool kW, bool kM>
__global__ void __launch_bounds__(kApplyThreads) cover_apply_kernel(const uint32_t *__restrict__ bits,
                                                                    const int64_t *__restrict__ first, int64_t nsrc,
                                                                    CoverGeo G,
                                                                    const int32_t *__restrict__ xy, int32_t r,
                                                                    int32_t k, unsigned long long *slot, int64_t *cur,
                                                                    int *done, uint32_t *__restrict__ state,
                                                                    uint32_t *__restrict__ newb,
                                                                    VhpCoverDevT<GainT<kW>> out, GainT<kW> *gain,
                                                                    uint8_t *__restrict__ cnt, int mfold) {
  const int64_t q = blockIdx.x;
  if (done[q]) return;
  const unsigned long long key = slot[q];
  __syncthreads(); // every thread has read the slot before thread 0 resets it
  GainT<kW> gn;
  uint32_t idx;
  if constexpr (kW) {
    gn = key >> kIdxBits;
    idx = (uint32_t)(kIdxMask - (key & kIdxMask));
  } else {
    gn = (uint32_t)(key >> 32);
    idx = ~(uint32_t)key;
  }
  const int64_t c = first[q] + idx;
  if (gn == 0 || first[q] < 0 || c >= nsrc) { // (the last two: an inconsistent group layout, reported by the table)
    if (threadIdx.x == 0) done[q] = 1;
    return;
  }
  if (threadIdx.x == 0) {
    if (out.pick) out.pick[q * k + r] = (int32_t)idx;
    if (out.gain) out.gain[q * k + r] = gn;
    if (out.npicked) out.npicked[q] = r + 1;
    cur[q] = c;
    slot[q] = 0;
    if constexpr (kM) gain[c] = 0;
  }
  const VhpCoverBox b = vhp_cover_box(G.nx, G.ny, G.R, __ldg(xy + 2 * c), __ldg(xy + 2 * c + 1));
  const int hw = b.H * b.W;
  const uint32_t *bc = bits + (size_t)c * hw;
  const size_t plane = (size_t)G.ny * G.nw;
  uint32_t *sq = state + (size_t)q * plane, *nq = newb + (size_t)q * hw;
  uint32_t *cov = out.covered ? out.covered + (size_t)q * plane : nullptr;
  for (int i = threadIdx.x; i < hw; i += blockDim.x) {
    const int rr = i / b.W, w = i - rr * b.W;
    const size_t o = (size_t)(b.y0 + rr) * G.nw + b.w0 + w;
    const uint32_t m = __ldg(bc + i), s = sq[o];
    if constexpr (kM) {
      uint32_t nw = 0;
      if (m) {
        // the word's 32 counters, byte b <-> bit b; each nibble of m becomes a {0, 1} byte selector (weight_sum)
        uint4 *cw = reinterpret_cast<uint4 *>(cnt + ((size_t)q * plane + o) * 32);
        uint4 a = cw[0], b2 = cw[1];
        uint32_t v[8] = {a.x, a.y, a.z, a.w, b2.x, b2.y, b2.z, b2.w};
        const uint32_t top = (uint32_t)(mfold - 1) * 0x01010101u, lim = top + 0x01010101u;
        uint32_t eq = 0; // bits whose counter is mfold - 1 before this pick
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t sel = (((m >> (4 * j)) & 0xfu) * 0x00204081u) & 0x01010101u;
          eq |= ((((__vcmpeq4(v[j], top) & 0x01010101u) * 0x01020408u) >> 24) & 0xfu) << (4 * j);
          v[j] += sel & __vcmpltu4(v[j], lim); // counters < mfold <= 255: no carry between bytes
        }
        cw[0] = make_uint4(v[0], v[1], v[2], v[3]);
        cw[1] = make_uint4(v[4], v[5], v[6], v[7]);
        nw = m & ~s & eq;
        if (nw) sq[o] = s | nw;
      }
      nq[i] = nw;
    } else {
      nq[i] = m & ~s;
      if (m) {
        sq[o] = s | m;
        if (cov) cov[o] |= m;
      }
    }
  }
}

// m-fold output: count[row][x] = cnt[row][x] for rows (problem, y) of the padded counter plane (32 bytes per word).
// A thread per 16 columns: one aligned 16-byte load, and stores as wide as the destination's alignment allows (the
// caller's rows are nx bytes, so a row of count starts 16-byte aligned only where row * nx is a multiple of 16).
__global__ void cover_count_kernel(const uint8_t *__restrict__ cnt, size_t nrows, int nx, int nw,
                                   uint8_t *__restrict__ count) {
  const int nch = (nx + 15) >> 4;
  const size_t n = nrows * nch;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t row = i / nch;
    const int x = 16 * (int)(i - row * nch);
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(cnt + row * nw * 32 + x));
    uint8_t *dst = count + row * nx + x;
    const unsigned a = (unsigned)reinterpret_cast<uintptr_t>(dst) & 15u;
    if (x + 16 <= nx && a == 0) {
      *reinterpret_cast<uint4 *>(dst) = v;
    } else if (x + 16 <= nx && (a & 3u) == 0) {
      uint32_t *d = reinterpret_cast<uint32_t *>(dst);
      d[0] = v.x;
      d[1] = v.y;
      d[2] = v.z;
      d[3] = v.w;
    } else {
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int b = 0; b < 16; ++b)
        if (x + b < nx) dst[b] = (uint8_t)(w[b >> 2] >> (8 * (b & 3)));
    }
  }
}

// floor and ceiling of n / d, d != 0 (C division truncates toward zero)
__device__ __forceinline__ long long floor_div(long long n, long long d) {
  const long long q = n / d;
  return (n % d != 0 && ((n < 0) != (d < 0))) ? q - 1 : q;
}
__device__ __forceinline__ long long ceil_div(long long n, long long d) {
  const long long q = n / d;
  return (n % d != 0 && ((n < 0) == (d < 0))) ? q + 1 : q;
}

constexpr int kViewInf = 1 << 20; // beyond any dx of a box (|dx| <= 16383 + 31)

// the dx of a row with u * dx <= v, as [lo, hi] clamped to [-kViewInf, kViewInf] (empty: lo > hi)
__device__ __forceinline__ void half_plane(long long u, long long v, int &lo, int &hi) {
  lo = -kViewInf;
  hi = kViewInf;
  if (u > 0) {
    hi = (int)max(min(floor_div(v, u), (long long)kViewInf), (long long)-kViewInf);
  } else if (u < 0) {
    lo = (int)max(min(ceil_div(v, u), (long long)kViewInf), (long long)-kViewInf);
  } else if (v < 0) {
    lo = 1;
    hi = 0;
  }
}

// The view call, after phase 1: S(c) &= view(c) in place, a warp per candidate, lanes over its box's rows.  view(c) =
// range r (the call's shape) and the sector of a = (ax, ay), b = (bx, by): cross(a, d) >= 0 and cross(d, b) >= 0 under
// 180 degrees (cross(a, b) > 0), either one from 180 degrees on (cross(a, b) < 0, or 0 with dot(a, b) < 0), every d
// when a and b point the same way.  On a row each half-plane is one dx interval, so the row's view is at most two.  A
// bad view (r outside [0, radius], a or b zero or a component outside [-32767, 32767]) raises bit 3 of err and clears
// the candidate's bits.  Only words that change are stored.
__global__ void __launch_bounds__(kWarps * 32) cover_view_kernel(uint32_t *__restrict__ bits, int64_t nsrc, CoverGeo G,
                                                                 int radius, bool disk,
                                                                 const int32_t *__restrict__ xy,
                                                                 const int32_t *__restrict__ views, int *err) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const VhpCoverBox b0 = vhp_cover_box(G.nx, G.ny, G.R, 0, 0);
  const size_t hw = (size_t)b0.H * b0.W;
  for (int64_t c = blockIdx.x * (int64_t)kWarps + warp; c < nsrc; c += (int64_t)gridDim.x * kWarps) {
    const int sx = __ldg(xy + 2 * c), sy = __ldg(xy + 2 * c + 1);
    const int32_t *v = views + 5 * c;
    const int r = __ldg(v), ax = __ldg(v + 1), ay = __ldg(v + 2), bx = __ldg(v + 3), by = __ldg(v + 4);
    const auto comp_ok = [](int t) { return t >= -32767 && t <= 32767; };
    const bool ok = r >= 0 && r <= radius && comp_ok(ax) && comp_ok(ay) && comp_ok(bx) && comp_ok(by) &&
                    (ax | ay) != 0 && (bx | by) != 0;
    if (!ok && lane == 0) atomicOr(err, 8);
    const long long cab = (long long)ax * by - (long long)ay * bx, dab = (long long)ax * bx + (long long)ay * by;
    const int mode = cab > 0 ? 0 : (cab < 0 || dab < 0) ? 1 : 2; // intersection, union, every direction
    const VhpCoverBox b = vhp_cover_box(G.nx, G.ny, G.R, sx, sy);
    uint32_t *bc = bits + (size_t)c * hw;
    for (int rr = lane; rr < b.H; rr += 32) {
      const int dy = b.y0 + rr - sy;
      int lo1 = 1, hi1 = 0, lo2 = 1, hi2 = 0; // the row's view: [lo1, hi1] | [lo2, hi2] in dx
      if (ok && abs(dy) <= r) {
        const int h = disk ? isqrt_floor(r * r - dy * dy) : r;
        lo1 = -h;
        hi1 = h;
        if (mode != 2) {
          int la, ha, lb, hb;
          half_plane(ay, (long long)ax * dy, la, ha);   // cross(a, d) >= 0: ay * dx <= ax * dy
          half_plane(-by, -(long long)bx * dy, lb, hb); // cross(d, b) >= 0: by * dx >= bx * dy
          if (mode == 0) {
            lo1 = max(lo1, max(la, lb));
            hi1 = min(hi1, min(ha, hb));
          } else {
            lo2 = max(lo1, lb);
            hi2 = min(hi1, hb);
            lo1 = max(lo1, la);
            hi1 = min(hi1, ha);
          }
        }
      }
      uint32_t *row = bc + (size_t)rr * b.W;
      for (int w = 0; w < b.W; ++w) {
        const uint32_t m = row[w];
        if (!m) continue;
        const int o = sx - 32 * (b.w0 + w); // bit of dx = 0
        const uint32_t mm = m & (span_mask(o + lo1, o + hi1) | span_mask(o + lo2, o + hi2));
        if (mm != m) row[w] = mm;
      }
    }
  }
}

// After round r's apply: exact gain update of the candidates whose box meets their problem's pick, then the keys of
// round r + 1.  Candidates of finished problems do nothing; a candidate of gain 0 keeps it.  kW: the weights of
// wpad's words, loaded only for words where S(c) & new is not 0.
template <bool kW>
__global__ void __launch_bounds__(kWarps * 32) cover_update_kernel(const uint32_t *__restrict__ bits, int64_t nsrc,
                                                                   CoverGeo G, const int32_t *__restrict__ xy,
                                                                   const int32_t *__restrict__ pg,
                                                                   const int32_t *__restrict__ pk,
                                                                   const int64_t *__restrict__ cur,
                                                                   const int *__restrict__ done,
                                                                   const uint32_t *__restrict__ newb,
                                                                   GainT<kW> *__restrict__ gain,
                                                                   unsigned long long *slot,
                                                                   const uint8_t *__restrict__ wpad) {
  __shared__ GainT<kW> sdec[kCand];
  __shared__ unsigned sov;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t base = blockIdx.x * (int64_t)kCand;
  const VhpCoverBox b0 = vhp_cover_box(G.nx, G.ny, G.R, 0, 0);
  const size_t hw = (size_t)b0.H * b0.W;
  bool valid = false;
  int32_t g = -1;
  GainT<kW> gn = 0;
  if (warp == 0) {
    const int64_t c = base + lane;
    g = c < nsrc ? pg[c] : -1;
    valid = g >= 0 && !done[g];
    bool ov = false;
    if (valid) {
      gn = gain[c];
      const int64_t p = cur[g];
      if (gn > 0) {
        const VhpCoverBox cb = vhp_cover_box(G.nx, G.ny, G.R, xy[2 * c], xy[2 * c + 1]);
        const VhpCoverBox pb = vhp_cover_box(G.nx, G.ny, G.R, xy[2 * p], xy[2 * p + 1]);
        ov = abs(cb.y0 - pb.y0) < b0.H && abs(cb.w0 - pb.w0) < b0.W;
      }
    }
    sdec[lane] = 0;
    const unsigned m = __ballot_sync(kAll, ov);
    if (lane == 0) sov = m;
  }
  __syncthreads();
  const unsigned ovm = sov;
  int rank = 0;
  for (unsigned m = ovm; m; m &= m - 1, ++rank) {
    if (rank % kWarps != warp) continue;
    const int j = __ffs(m) - 1;
    const int64_t c = base + j;
    const int32_t q = pg[c];
    const int64_t p = cur[q];
    const VhpCoverBox cb = vhp_cover_box(G.nx, G.ny, G.R, xy[2 * c], xy[2 * c + 1]);
    const VhpCoverBox pb = vhp_cover_box(G.nx, G.ny, G.R, xy[2 * p], xy[2 * p + 1]);
    const int ra = max(cb.y0, pb.y0), rb = min(cb.y0, pb.y0) + b0.H;
    const int wa = max(cb.w0, pb.w0), wb = min(cb.w0, pb.w0) + b0.W;
    GainT<kW> acc = 0;
    for (int y = ra + lane; y < rb; y += 32) {
      const uint32_t *nr = newb + (size_t)q * hw + (size_t)(y - pb.y0) * b0.W - pb.w0;
      const uint32_t *br = bits + (size_t)c * hw + (size_t)(y - cb.y0) * b0.W - cb.w0;
      for (int w = wa; w < wb; ++w) {
        const uint32_t n = nr[w];
        if constexpr (kW) {
          const uint32_t m = n ? __ldg(br + w) & n : 0u;
          if (m) acc += weight_sum(m, wpad + (((size_t)q * G.ny + y) * G.nw + w) * 32);
        } else {
          if (n) acc += __popc(__ldg(br + w) & n);
        }
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) sdec[j] = acc;
  }
  __syncthreads();
  if (warp == 0) {
    const int64_t c = base + lane;
    if (valid && sdec[lane]) {
      gn -= sdec[lane];
      gain[c] = gn;
    }
    put_keys(valid, g, key_of(gn, valid ? pk[c] : 0), slot);
  }
}

unsigned grid_for(size_t n, int bs, int sm_count) {
  return (unsigned)std::max<size_t>(1, std::min<size_t>((n + bs - 1) / bs, (size_t)sm_count * 32));
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// workspace of the rounds: state [prob][ny][nw], new [prob][H][W], gain [src] (uint32, weighted uint64), slot [prob],
// cur [prob], first [prob], done [prob]; weighted: wpad [prob][ny][nw][32]; m-fold (weighted too): cnt, wpad's layout
struct CoverWs {
  uint32_t *state, *newb;
  void *gain;
  unsigned long long *slot;
  int64_t *cur, *first;
  int *done;
  uint8_t *wpad, *cnt;
  size_t bytes;
};
CoverWs cover_ws(void *base, int64_t nprob, int64_t nsrc, int nx, int ny, int R, bool weighted, bool mfold) {
  const VhpCoverBox b = vhp_cover_box(nx, ny, R, 0, 0);
  const size_t np = (size_t)nprob, plane = (size_t)ny * ((nx + 31) / 32);
  const size_t o_new = align256(np * plane * 4), o_gain = o_new + align256(np * b.H * b.W * 4);
  const size_t o_slot = o_gain + align256((size_t)nsrc * (weighted ? 8 : 4)), o_cur = o_slot + align256(np * 8);
  const size_t o_first = o_cur + align256(np * 8), o_done = o_first + align256(np * 8);
  const size_t o_wpad = o_done + align256(np * 4), o_cnt = o_wpad + (weighted ? align256(np * plane * 32) : 0);
  char *p = static_cast<char *>(base);
  CoverWs w{};
  w.bytes = o_cnt + (mfold ? align256(np * plane * 32) : 0);
  if (!p) return w;
  w.state = (uint32_t *)p;
  w.newb = (uint32_t *)(p + o_new);
  w.gain = p + o_gain;
  w.slot = (unsigned long long *)(p + o_slot);
  w.cur = (int64_t *)(p + o_cur);
  w.first = (int64_t *)(p + o_first);
  w.done = (int *)(p + o_done);
  w.wpad = weighted ? (uint8_t *)(p + o_wpad) : nullptr;
  w.cnt = mfold ? (uint8_t *)(p + o_cnt) : nullptr;
  return w;
}

// the rounds of the three calls: kW = false counts cells of d_target (null: all), kW = true sums d_weights (null:
// all 1), kM (with kW) counts each cell until mfold picks cover it and writes d_count (may be null) at the end
template <bool kW, bool kM = false>
cudaError_t launch_rounds(uint32_t *d_bits, int64_t nsrc, int64_t nprob, int nx, int ny, int R, int disk_r2,
                          const int32_t *d_xy, const int32_t *d_pair_group, const int32_t *d_pair_k,
                          const uint32_t *d_target, const uint8_t *d_weights, int32_t k, int mfold, void *d_ws,
                          const VhpCoverDevT<GainT<kW>> &out, uint8_t *d_count, int sm_count, cudaStream_t st,
                          int64_t *launches) {
  const CoverGeo G{nx, ny, R, (nx + 31) / 32};
  const size_t np = (size_t)nprob, plane = (size_t)ny * G.nw;
  cudaError_t e = cudaSuccess;
  if (out.pick) e = cudaMemsetAsync(out.pick, 0xff, np * k * 4, st); // -1 from npicked on
  if (e == cudaSuccess && out.gain) e = cudaMemsetAsync(out.gain, 0, np * k * sizeof(GainT<kW>), st);
  if (e == cudaSuccess && out.npicked) e = cudaMemsetAsync(out.npicked, 0, np * 4, st);
  if (e == cudaSuccess && out.covered) e = cudaMemsetAsync(out.covered, 0, np * plane * 4, st);
  const int64_t rounds = std::min<int64_t>(k, nsrc);
  if (e == cudaSuccess && d_count && rounds <= 0) e = cudaMemsetAsync(d_count, 0, np * ny * nx, st); // no pick
  if (e != cudaSuccess || rounds <= 0 || nprob == 0) return e;
  const CoverWs ws = cover_ws(d_ws, nprob, nsrc, nx, ny, R, kW, kM);
  GainT<kW> *gain = (GainT<kW> *)ws.gain;
  if (kW) {
    cover_weight_kernel<<<grid_for(np * plane * 8, 256, sm_count), 256, 0, st>>>(d_weights, nprob, G, ws.wpad,
                                                                                 ws.state);
    if (launches) *launches += 1;
  } else if (d_target) {
    cover_state_kernel<<<grid_for(np * plane, 256, sm_count), 256, 0, st>>>(d_target, np * plane, ws.state);
    if (launches) *launches += 1;
  } else {
    e = cudaMemsetAsync(ws.state, 0, np * plane * 4, st);
  }
  if (e == cudaSuccess) e = cudaMemsetAsync(ws.slot, 0, np * 8, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(ws.done, 0, np * 4, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(ws.first, 0xff, np * 8, st);
  if (e == cudaSuccess && kM) e = cudaMemsetAsync(ws.cnt, 0, np * plane * 32, st);
  if (e != cudaSuccess) return e;
  const unsigned cgrid = (unsigned)((nsrc + kCand - 1) / kCand);
  cover_init_kernel<kW><<<cgrid, kWarps * 32, 0, st>>>(d_bits, nsrc, G, disk_r2, d_xy, d_pair_group, d_pair_k, ws.state,
                                                      gain, ws.slot, ws.first, ws.wpad);
  for (int32_t r = 0; r < rounds; ++r) {
    cover_apply_kernel<kW, kM><<<(unsigned)nprob, kApplyThreads, 0, st>>>(d_bits, ws.first, nsrc, G, d_xy, r, k,
                                                                          ws.slot, ws.cur, ws.done, ws.state, ws.newb,
                                                                          out, gain, ws.cnt, mfold);
    if (r + 1 < rounds)
      cover_update_kernel<kW><<<cgrid, kWarps * 32, 0, st>>>(d_bits, nsrc, G, d_xy, d_pair_group, d_pair_k, ws.cur,
                                                            ws.done, ws.newb, gain, ws.slot, ws.wpad);
  }
  if (launches) *launches += 2 * rounds;
  if (kM && d_count) {
    const size_t nrows = np * ny;
    cover_count_kernel<<<grid_for(nrows * ((nx + 15) / 16), 256, sm_count), 256, 0, st>>>(ws.cnt, nrows, nx, G.nw,
                                                                                          d_count);
    if (launches) *launches += 1;
  }
  return cudaGetLastError();
}

} // namespace

cudaError_t vhp_launch_cover_fold(const double *d_val, int win_r, int64_t p0, int64_t np, int nx, int ny, int R,
                                  bool disk, int r2, const int32_t *d_xy, double thr, uint32_t *d_bits, int sm_count,
                                  cudaStream_t st, int64_t *launches) {
  const CoverGeo G{nx, ny, R, (nx + 31) / 32};
  const VhpCoverBox b = vhp_cover_box(nx, ny, R, 0, 0);
  const int bs = 256;
  cover_fold_kernel<<<grid_for((size_t)np * b.H * b.W, bs, sm_count), bs, 0, st>>>(d_val, win_r, p0, np, G, disk, r2,
                                                                                   d_xy, thr, d_bits);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t vhp_launch_cover_view(uint32_t *d_bits, int64_t nsrc, int nx, int ny, int R, int radius, bool disk,
                                  const int32_t *d_xy, const int32_t *d_views, int *d_err, int sm_count,
                                  cudaStream_t st, int64_t *launches) {
  if (nsrc <= 0) return cudaSuccess;
  const CoverGeo G{nx, ny, R, (nx + 31) / 32};
  cover_view_kernel<<<grid_for((size_t)nsrc * 32, kWarps * 32, sm_count), kWarps * 32, 0, st>>>(d_bits, nsrc, G, radius,
                                                                                             disk, d_xy, d_views,
                                                                                             d_err);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

size_t vhp_cover_ws_bytes(int64_t nprob, int64_t nsrc, int nx, int ny, int R, bool weighted, bool mfold) {
  return cover_ws(nullptr, nprob, nsrc, nx, ny, R, weighted || mfold, mfold).bytes;
}

cudaError_t vhp_launch_cover_greedy(uint32_t *d_bits, int64_t nsrc, int64_t nprob, int nx, int ny, int R, int disk_r2,
                                    const int32_t *d_xy, const int32_t *d_pair_group, const int32_t *d_pair_k,
                                    bool weighted, bool mfold, const void *d_extra, int32_t k, int m, void *d_ws,
                                    const VhpCoverOut &out, int sm_count, cudaStream_t st, int64_t *launches) {
  if (!weighted) {
    const VhpCoverDevT<uint32_t> o{out.pick, (uint32_t *)out.gain, out.npicked, out.covered};
    return launch_rounds<false>(d_bits, nsrc, nprob, nx, ny, R, disk_r2, d_xy, d_pair_group, d_pair_k,
                                (const uint32_t *)d_extra, nullptr, k, 1, d_ws, o, nullptr, sm_count, st, launches);
  }
  const VhpCoverDevT<uint64_t> o{out.pick, (uint64_t *)out.gain, out.npicked, out.covered};
  const uint8_t *d_weights = (const uint8_t *)d_extra;
  if (!mfold)
    return launch_rounds<true>(d_bits, nsrc, nprob, nx, ny, R, disk_r2, d_xy, d_pair_group, d_pair_k, nullptr,
                               d_weights, k, 1, d_ws, o, nullptr, sm_count, st, launches);
  return launch_rounds<true, true>(d_bits, nsrc, nprob, nx, ny, R, disk_r2, d_xy, d_pair_group, d_pair_k, nullptr,
                                   d_weights, k, m, d_ws, o, out.count, sm_count, st, launches);
}
