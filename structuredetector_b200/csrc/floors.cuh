// floors.cuh -- pruning floors and the candidate flush shared by the peaks kernels: logit histograms (warp-local,
// exact; plane-wide, strict), the floors derived from them, and flush_candidates (exact scores of the buffered
// pixels, list append, histogram update).
#pragma once

namespace {

#ifndef SDNET_X_BUF
#define SDNET_X_BUF 64
#endif
constexpr int kBuf = SDNET_X_BUF;      // per-warp candidate buffer (records), a multiple of 32
#ifndef SDNET_X_GRATE
#define SDNET_X_GRATE 0
#endif
#ifndef SDNET_X_LRATE
#define SDNET_X_LRATE 0
#endif
// Floors are recomputed from the histograms only when that can change them: the plane-wide floor needs K
// recorded candidates in the plane, the warp-local one K in the unit; beyond that, every kGRate / kLRate
// new records (0 = at every flush).
constexpr int kGRate = SDNET_X_GRATE, kLRate = SDNET_X_LRATE;
constexpr int kGDiv = kGRate ? kGRate : 1, kLDiv = kLRate ? kLRate : 1;

__device__ __forceinline__ int logit_bin(float x) {
  int bin = __float2int_rd((x - kBinLo) * kBinScale);
  bin = max(0, min(kBins - 1, bin));
  // rounding guard: never count an element in a bin whose lower edge is above it
  if (bin > 0 && x < kBinLo + (float)bin * (1.0f / kBinScale)) --bin;
  return bin;
}

// order-preserving float <-> int (so atomicMin works on floats of either sign)
__device__ __forceinline__ int ord_of(float x) {
  const int b = __float_as_int(x);
  return b ^ ((b >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float ord_to_float(int o) { return __int_as_float(o ^ ((o >> 31) & 0x7fffffff)); }

// Highest bin b with (count in bins >= b) >= K given each lane's four bin counts; -1 if none.
__device__ __forceinline__ int floor_bin_of(const uint4 c, int lane, int K) {
  const u32 s = c.x + c.y + c.z + c.w;
  u32 suf = s;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    u32 t = __shfl_down_sync(0xffffffffu, suf, d);
    if (lane + d < 32) suf += t;
  }
  const u32 mask = __ballot_sync(0xffffffffu, suf >= (u32)K);
  if (mask == 0) return -1;
  const int L = 31 - __clz(mask);
  int b = 0;
  if (lane == L) {
    u32 above = suf - s;
    if (above + c.w >= (u32)K) b = 4 * L + 3;
    else if (above + c.w + c.z >= (u32)K) b = 4 * L + 2;
    else if (above + c.w + c.z + c.y >= (u32)K) b = 4 * L + 1;
    else b = 4 * L;
  }
  return __shfl_sync(0xffffffffu, b, L);
}

// Warp-local pruning floor.  Let b be the highest bin such that this warp-unit has already
// recorded >= K candidates in bins >= b.  Every one of those has a (saturation-clamped) logit
// >= minx[b] and a lower flat index than anything the unit will see later, so it beats any
// later pixel whose clamped logit is <= minx[b] under (score desc, index asc) -- equal scores
// included.  Returns minx[b], or -inf when fewer than K candidates were recorded.
__device__ __forceinline__ float local_floor(const u32* hist, const int* minx, int lane, int K) {
  const int b = floor_bin_of(*reinterpret_cast<const uint4*>(hist + 4 * lane), lane, K);
  if (b < 0) return -CUDART_INF_F;
  return ord_to_float(minx[b]);
}

__device__ __forceinline__ int fine_bin(float x) {
  // x * 16 is exact (a power of two), so floor(x * 16) - 16 * kBinLo is THE bin: an element is never
  // counted in a bin whose lower edge is above it.  Large |x| saturates in the conversion, then in the clamp.
  static_assert(kBinLo == -16.0f && kFineScale == 16.0f, "bin arithmetic below");
  return max(0, min(kFineBins - 1, __float2int_rd(fminf(fmaxf(x * kFineScale, -4096.0f), 4096.0f)) + 256));
}

// Highest fine bin b with (count in bins >= b) >= K; lane l owns bins 32l..32l+31.  -1 if none.
// kShared: the histogram lives in shared memory (volatile loads) instead of global (L2 loads).
template <bool kShared>
__device__ __forceinline__ uint4 load_bins(const u32* ptr) {
  uint4 v;
  if (kShared) {
    asm volatile("ld.volatile.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_u32(ptr)));
  } else {
    v = __ldcg(reinterpret_cast<const uint4*>(ptr));
  }
  return v;
}

template <bool kShared>
__device__ __forceinline__ int floor_bin_fine(const u32* hist, int lane, int K) {
  const u32* mine = hist + kFinePerLane * lane;
  uint4 v[kFinePerLane / 4];
#pragma unroll
  for (int q = 0; q < kFinePerLane / 4; ++q) v[q] = load_bins<kShared>(mine + 4 * q);
  u32 s = 0;
#pragma unroll
  for (int q = 0; q < kFinePerLane / 4; ++q) s += v[q].x + v[q].y + v[q].z + v[q].w;
  u32 suf = s;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    u32 t = __shfl_down_sync(0xffffffffu, suf, d);
    if (lane + d < 32) suf += t;
  }
  const u32 mask = __ballot_sync(0xffffffffu, suf >= (u32)K);
  if (mask == 0) return -1;
  const int L = 31 - __clz(mask);
  int b = kFinePerLane * L;
  if (lane == L) {
    u32 above = suf - s;
    bool found = false;
#pragma unroll
    for (int q = kFinePerLane / 4 - 1; q >= 0; --q) {
      const u32 c4[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
      for (int e = 3; e >= 0; --e) {
        if (!found) {
          if (above + c4[e] >= (u32)K) { b = kFinePerLane * L + 4 * q + e; found = true; }
          else above += c4[e];
        }
      }
    }
  }
  return __shfl_sync(0xffffffffu, b, L);
}

// Floor shared between warps working on the same plane (CTA-wide in shared memory, plane-wide in
// global memory).  Unlike the warp-local floor (which may drop equal scores because everything
// it counted has a lower index), a shared floor needs a strict score gap: a pixel is dropped
// only if its logit is below edge(b) - kNear with edge(b) in [kLo, kHi] (Num<DT>), where
// S(x - kNear) < S(x) is verified exhaustively (tests/test_gpu_parity.py).
// Pre-activated maps never go below a floor of 0: their zeros are the pixels NMS suppressed, which the tail's zero-fill
// supplies in torch.topk's order (class, then index).  Recording only some of them -- those a warp meets before its
// floor rises -- would put those ahead of the zero-filled ones.
template <int DT = SDNET_DTYPE_F32>
__device__ __forceinline__ float shared_floor(int fbin, float xscale) {
  const bool pre = xscale != 1.0f;
  if (fbin <= 0) return pre ? 0.0f : -CUDART_INF_F;
  const float edge = kBinLo + (float)fbin * (1.0f / kFineScale);
  if (pre) return fmaxf(edge / xscale, 0.0f);  // keys are strictly monotone in the value
  if (edge < Num<DT>::kLo || edge > Num<DT>::kHi2) return -CUDART_INF_F;
  return edge - (edge <= Num<DT>::kHi ? Num<DT>::kNear : Num<DT>::kNear2);
}

// Where a warp publishes / picks up shared floors.
struct SharedFloors {
  u32* ghist;      // global [kFineBins], or nullptr when the CTA covers the whole plane
  int* gfloor;     // global
};

// Flush the warp's candidate buffer: evaluate the exact score of up to 64 buffered pixels (all
// lanes busy), append (score, index) records to the plane's list with one atomic, feed the
// warp-local and plane-wide histograms and raise the pruning floor.
struct UnitState {
  float floorx;   // input units; a pixel can still matter only if x > floorx
  u32 emitted;    // records this unit has appended so far
  int nbuf;       // records waiting in the shared-memory buffer
};

template <int DT = SDNET_DTYPE_F32, bool kFlushCountsFine = true>
__device__ __forceinline__ void flush_candidates(UnitState& st, const u64* buf, u32* hist, int* minx,
                                                 const SharedFloors& sf, int* count_ptr, u64* __restrict__ list,
                                                 int cap, int K, int lane, bool pre, float xscale, float satx) {
  const int n = st.nbuf;  // warp-uniform, 1..kBuf
  int base = 0;
  if (lane == 0) base = atomicAdd(count_ptr, n);
  base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
  for (int half = 0; half < kBuf / 32; ++half) {
    const int i = half * 32 + lane;
    if (half * 32 < n) {  // warp-uniform
      const bool valid = i < n;
      const u64 rec = valid ? buf[i] : 0ull;
      const float x = __uint_as_float((u32)(rec >> 32));
      u32 key;
      if (pre) {
        const u32 bits = __float_as_uint(x);
        key = (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
      } else {
        key = __float_as_uint(Num<DT>::act(x));
      }
      if (valid) {
        if (base + i < cap) list[base + i] = ((u64)key << 32) | (u32)rec;
        // clamped logit: the score is a monotone function of it, saturation included
        const float xe = fminf(fmaxf(x * xscale, -satx), satx);
        const int bin = logit_bin(xe);
        atomicAdd(&hist[bin], 1u);
        atomicMin(&minx[bin], ord_of(xe));
        if (kFlushCountsFine && sf.ghist) atomicAdd(&sf.ghist[fine_bin(xe)], 1u);
      }
    }
  }
  const u32 before = st.emitted;
  st.emitted += n;
  st.nbuf = 0;
  __syncwarp();
  // xscale is a power of two, so the division is exact
  if (st.emitted >= (u32)K && (kLRate == 0 || before < (u32)K || before / kLDiv != st.emitted / kLDiv))
    st.floorx = fmaxf(st.floorx, local_floor(hist, minx, lane, K) / xscale);
  // publish / refresh the shared floors (`base` = records in the plane before this flush)
  if (sf.ghist && base + n >= K && (kGRate == 0 || base < K || base / kGDiv != (base + n) / kGDiv)) {
    const int gb = floor_bin_fine<false>(sf.ghist, lane, K);
    if (gb > 0) {
      if (lane == 0) atomicMax(sf.gfloor, gb);
      st.floorx = fmaxf(st.floorx, shared_floor<DT>(gb, xscale));
    }
  }
  // a floor at the saturation clamp means "nothing can beat what we have": every x >= satx has
  // the same score as the K recorded ones and a higher index
  if (st.floorx >= satx) st.floorx = CUDART_INF_F;
}


}  // namespace
