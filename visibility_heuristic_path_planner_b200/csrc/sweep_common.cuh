// sweep_common.cuh -- arithmetic shared by the sweep kernels (bit-parity contract).
#ifndef VHP_SWEEP_COMMON_CUH
#define VHP_SWEEP_COMMON_CUH

#include <cstdint>

namespace {

__device__ __forceinline__ double lerp_rn(double a, double b, double c) {
  return __dsub_rn(a, __dmul_rn(c, __dsub_rn(a, b)));
}

template <typename OutT> __device__ __forceinline__ OutT to_out(double v);
template <> __device__ __forceinline__ float to_out<float>(double v) { return __double2float_rn(v); }
template <> __device__ __forceinline__ double to_out<double>(double v) { return v; }

// relaxed reductions of the merged outputs (vhp_visibility_merge_batch and its range-limited form): max / min on
// the bits of non-negative values and indices, add for the counts; the result does not depend on their order
__device__ __forceinline__ void red_max_u64(unsigned long long *a, unsigned long long v) {
  asm volatile("red.relaxed.gpu.global.max.u64 [%0], %1;" :: "l"(a), "l"(v) : "memory");
}
__device__ __forceinline__ void red_max_u32(uint32_t *a, uint32_t v) {
  asm volatile("red.relaxed.gpu.global.max.u32 [%0], %1;" :: "l"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void red_min_u32(uint32_t *a, uint32_t v) {
  asm volatile("red.relaxed.gpu.global.min.u32 [%0], %1;" :: "l"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void red_add_u32(uint32_t *a, uint32_t v) {
  asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" :: "l"(a), "r"(v) : "memory");
}

// A view of vhp_visibility_merge_view_batch, (r, ax, ay, bx, by), decoded once per source by the rule of
// cover_view_kernel: range r in the call's shape, and the sector of a and b, cross(a, d) >= 0 and cross(d, b) >= 0
// under 180 degrees (cross(a, b) > 0), either one otherwise (from 180 degrees on; and every d when a and b point the
// same way, as cross(d, b) is then a negative multiple of cross(a, d)).  key: bit 31 set for "either one", bits 0-30
// free for the caller (the tile route keeps the source's cell index there); range: r^2 (disk) or ~r (box, negative);
// a, b: two int16 each.  |component| <= 32767 and |dx|, |dy| <= R <= 16383, so |cross| <= 2 * 32767 * 16383 < 2^31
// and the test runs in 32 bits.
struct MergeView {
  int key, range, a, b;
};
__device__ __forceinline__ bool merge_view_decode(const int32_t *__restrict__ v, int radius, bool disk, MergeView &w) {
  const int r = __ldg(v), ax = __ldg(v + 1), ay = __ldg(v + 2), bx = __ldg(v + 3), by = __ldg(v + 4);
  const auto comp_ok = [](int t) { return t >= -32767 && t <= 32767; };
  if (!(r >= 0 && r <= radius && comp_ok(ax) && comp_ok(ay) && comp_ok(bx) && comp_ok(by) && (ax | ay) != 0 &&
        (bx | by) != 0))
    return false;
  w.key = ax * by - ay * bx > 0 ? 0 : (int)0x80000000u;
  w.range = disk ? r * r : ~r;
  w.a = (ax & 0xffff) | (ay << 16);
  w.b = (bx & 0xffff) | (by << 16);
  return true;
}
// is the cell d = (dx, dy) from the source in the view
__device__ __forceinline__ bool merge_view_has(const MergeView &w, int dx, int dy) {
  const int adx = abs(dx), ady = abs(dy);
  if (w.range >= 0 ? adx * adx + ady * ady > w.range : max(adx, ady) > ~w.range) return false;
  const int ax = (short)w.a, ay = w.a >> 16, bx = (short)w.b, by = w.b >> 16;
  const bool c1 = ax * dy - ay * dx >= 0, c2 = dx * by - dy * bx >= 0;
  return w.key < 0 ? (c1 || c2) : (c1 && c2);
}

} // namespace
#endif
