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

} // namespace
#endif
