// common.cuh -- types, launch parameters, per-dtype numerics (Num<DT>) and PTX wrappers shared by the kernels.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdlib.h>

#include "sdnet_decode.h"

namespace {

typedef unsigned long long u64;
typedef unsigned int u32;

constexpr int kThreads = 256;          // peaks kernel CTA
constexpr int kWarps = kThreads / 32;
constexpr int kPanelW = 128;           // columns per warp (32 lanes x 4)
constexpr int kBins = 128;             // per-warp logit histogram used for pruning
constexpr float kBinLo = -16.0f;
constexpr float kBinScale = 4.0f;      // bins of 0.25 logit
constexpr int kFineBins = 512;         // shared (CTA-wide / plane-wide) histograms: bins of 1/16 logit
constexpr float kFineScale = 16.0f;    // (256 x 0.125: blobs 3 % slower; 1024 x 1/32: flushes 25 % slower)
constexpr int kFinePerLane = kFineBins / 32;
// Floor hint (peaks_tile.cuh): planes of a channel that must have finished before their lowest floor, less a margin, is
// applied to the channel's other planes.  Measured at 1024 cfg5 images, one B200 (1000 W), no plane through the exact
// select in 25 decodes with a margin of 1, 2 or 4 bins; 2 costs 3-10 % more candidates than 1, 4 another 5-20 %.
constexpr int kHintMinPlanes = 8;
constexpr int kHintMarginBins = 2;     // fine bins: 1/8 logit
constexpr float kSatX = 14.0f;         // |x| >= 14 is inside the clamp on both sides: S(x) == S(+-14)
constexpr float kPreScale = 8.0f;      // pre-activated maps: histogram runs on 8*value
constexpr float kClampLo = 1e-6f;
constexpr float kClampHi = (float)(1.0 - 1e-6);
constexpr float kFar = 1e6f;

constexpr int kSortN = 2048;           // tail sort buffer (>= SDNET_MAX_TOPK + boundary slack)

struct View4 {
  const void* data;      // element type given by the launch's dtype
  long long sb, sc, sh;  // strides in elements
};

struct PeaksParams {
  View4 anchor, part;
  int B, M, N, H, W, K, P;
  int strips, rows_per_strip, panels;
  int units;
  int cap;                 // records per plane list
  int pre_activated;
  u64* lists;              // [planes][cap]
  int* counts;             // [planes] records emitted (may exceed cap)
  u32* sched;              // [0] dynamic unit counter
  u32* ghist;              // [planes][kFineBins] plane-wide logit histogram of recorded candidates
  int* gfloor;             // [planes] highest fine bin b with >= K recorded candidates in bins >= b (0 = none)
  // tile kernel: the work is a line of columns (one panel of one plane, top to bottom), groups_per_col
  // groups of four rows each.  Units [0, tier1_units) are whole columns; unit tier1_units + j is the
  // j-th chunk of chunk_groups groups of the rest of the line and may run over a column's end into the
  // next column (plan_peaks in sdnet_decode.cu)
  int tier1_units, groups_per_col, chunk_groups;
  u32 total_groups;
  int odd_x;               // tile kernel, row-pair maps: tensor-map x coordinate of an odd row's column 0
};

// The tile kernel's floor hint (peaks_tile.cuh), an argument of its own so that PeaksParams -- which the suppress kernel
// takes too -- keeps its layout.  chint[c][0] = kFineBins - the lowest gfloor reported by a finished plane of channel c,
// chint[c][1] = planes that reported (zeroed = no hint); hint_used[plane] = highest hint bin applied to it (0 = none).
struct HintParams {
  u32* chint;
  int* hint_used;
};

// Numerics of the score function per input dtype DT (SDNET_DTYPE_*).
//
// fp32: S(x) = clamp(1/(1+expf(-x))), bit-identical to ATen's CUDA kernels (UnarySpecialOpsKernel.cu
// sigmoid: one / (one + std::exp(-a)); TensorCompare.cu clamp: min(max(v, lo), hi)).
// fp16 / bf16 (what the reference's `--amp` validation feeds the decoder): ATen evaluates both ops in
// fp32 and rounds each result to the tensor dtype, so S_T(x) = T(clamp(float(T(sigmoid(float(x)))))),
// returned here as the exactly representable float.  Every S_T is monotone non-decreasing in x.
//
// The margins say when two different logits x < h might share a score: only if x >= h - kNear with h in
// [kLo, kHi], or x >= h - kNear2 with h in (kHi, kHi2], or h > kHi2 and x > kHi2 - 1, or h < kLo.
// Outside that, S(x) < S(h) strictly; verified exhaustively on the device for every dtype
// (tests/test_gpu_parity.py, tests/test_gpu_halfprec.py).
template <int DT>
struct Num;

// For logits x < h: false only where S(x) < S(h) is certain (outside the zones above), so the exact
// scores need comparing only where it is true.  The first zone is tested for any h, a superset.
template <int DT>
__device__ __forceinline__ bool may_tie(float x, float h) {
  return (x >= h - Num<DT>::kNear) || (h > Num<DT>::kHi && x >= h - Num<DT>::kNear2) ||
         (h > Num<DT>::kHi2 && x > Num<DT>::kHi2 - 1.0f) || (h < Num<DT>::kLo);
}

template <>
struct Num<SDNET_DTYPE_F32> {
  typedef float In;
  static constexpr float kNear = 2e-3f, kHi = 8.0f, kLo = -13.0f;
  static constexpr float kNear2 = 2e-3f, kHi2 = 8.0f;  // no second zone
  static __device__ __forceinline__ float act(float x) {
    const float s = 1.0f / (1.0f + expf(-x));
    return fminf(fmaxf(s, kClampLo), kClampHi);
  }
  static __device__ __forceinline__ float to_float(float v) { return v; }
};

template <>
struct Num<SDNET_DTYPE_F16> {
  typedef __half In;
  static constexpr float kNear = 0.02f, kHi = 3.0f, kLo = -11.0f;
  static constexpr float kNear2 = 0.15f, kHi2 = 5.0f;  // 10-bit mantissa: ties reach 0.073 logit at h = 5
  static __device__ __forceinline__ float act(float x) {
    const float s = __half2float(__float2half_rn(1.0f / (1.0f + expf(-x))));
    return __half2float(__float2half_rn(fminf(fmaxf(s, kClampLo), kClampHi)));
  }
  static __device__ __forceinline__ float to_float(__half v) { return __half2float(v); }
};

template <>
struct Num<SDNET_DTYPE_BF16> {
  typedef __nv_bfloat16 In;
  static constexpr float kNear = 0.1f, kHi = 2.0f, kLo = -13.0f;
  static constexpr float kNear2 = 0.6f, kHi2 = 4.0f;   // 7-bit mantissa: ties reach 0.22 logit at h = 4
  static __device__ __forceinline__ float act(float x) {
    const float s = __bfloat162float(__float2bfloat16_rn(1.0f / (1.0f + expf(-x))));
    return __bfloat162float(__float2bfloat16_rn(fminf(fmaxf(s, kClampLo), kClampHi)));
  }
  static __device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
};

// element `idx` of a tensor whose dtype is DT, as float (exact)
template <int DT>
__device__ __forceinline__ float ld_in(const void* base, long long idx) {
  return Num<DT>::to_float(__ldg(static_cast<const typename Num<DT>::In*>(base) + idx));
}

__device__ __forceinline__ float max3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// Programmatic dependent launch: the next kernel of the decode may be scheduled while this one is
// still running (its CTAs take whatever SM resources free up and park at pdl_wait), which hides the
// launch latency between the three kernels.  pdl_wait returns once the previous kernel has fully
// completed and its memory is visible.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float comp(const float4& v, int j) {
  return j == 0 ? v.x : (j == 1 ? v.y : (j == 2 ? v.z : v.w));
}

__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }
// predicated cp.async: global -> shared, no register staging
__device__ __forceinline__ void cp_async4_if(u32 dst, const void* src, bool pred) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p cp.async.ca.shared.global [%0], [%1], 4;\n\t}"
               ::"r"(dst), "l"(src), "r"((int)pred));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ float4 lds128(u32 addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float2 lds64(u32 addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(u32 addr, float a) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};" ::"r"(addr), "f"(a) : "memory");
}
__device__ __forceinline__ void sts64(u32 addr, float a) {
  asm volatile("st.shared.v2.f32 [%0], {%1, %1};" ::"r"(addr), "f"(a) : "memory");
}

// ---- mbarrier + 1-D bulk copy (TMA unit; SASS: UBLKCP, SYNCS) ---------------------------------
__device__ __forceinline__ void mbar_init(u32 bar, u32 count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(u32 bar, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint: the warp sleeps until the phase completes instead of spinning.
// Measured: a spinning test_wait streams faster when nothing else runs (0.62 vs 0.94 ms with the
// slow path disabled) but steals issue slots from the working warps in the real kernel (0.724 vs 0.718 ms).
__device__ __forceinline__ void mbar_wait(u32 bar, u32 parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@!p bra WAIT_LOOP;\n\t}"
      ::"r"(bar), "r"(parity), "r"(1000u) : "memory");  // suspend-time hint, ns
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace
