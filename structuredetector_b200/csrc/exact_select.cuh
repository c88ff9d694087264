// exact_select.cuh -- sdnet_exact_select_kernel: bounded-memory top-K straight from a heat-map plane.
#pragma once

namespace {

// ---------------------------------------------------------------------------------------------
// exact-select kernel: bounded-memory fallback for planes whose candidate list overflowed
// (or for every plane under SDNET_FLAG_EXACT_SELECT).  One CTA per plane: a 3-level radix
// select (11/11/10 bits) over the NMS'd scores recomputed straight from the heat map, then an
// index-ordered emission pass that keeps every score above the K-th and the lowest-index
// members of the K-th score's tie run.  Rewrites the plane's list with <= K records.
// ---------------------------------------------------------------------------------------------
// A THIN CTA on purpose: 128 threads x <= 80 registers is exactly the footprint of one peaks-kernel CTA, so the CTAs of
// the usual pass-through ("nothing overflowed": one look at the counts, exit) drop into whatever slot is free.  The
// 512-thread, 116-register CTA this kernel used to have needs a whole SM's register file: the block scheduler drained
// SM after SM of the next decode's peaks CTAs to place it, which cost 2.6 % of the step at 1024 images and 4-10 % at 128
// with several decodes in flight (measured by skipping the launch).  Six thin CTAs per SM hold more threads than one
// fat one, so a batch of saturated planes is not slower either; a single overflowed plane takes ~4x longer.
constexpr int kExactThreads = 128;
constexpr int kExactCtasPerSm = 6;

struct ExactParams {
  View4 anchor, part;
  int B, M, N, H, W, K, P;
  int radius, cap, force, pre_activated;
  u64* lists;
  int* counts;
  int* flags;
};

template <int DT>
__device__ __forceinline__ u32 exact_key(const void* plane, long long sh, int H, int W, int R, int y, int x, bool pre) {
  const float v = ld_in<DT>(plane, (long long)y * sh + x);
  if (pre) {  // zeros are suppressed pixels, left to the tail's zero-fill like in the peaks kernels (shared_floor)
    return v > 0.0f ? (__float_as_uint(v) | 0x80000000u) : 0u;
  }
  float h = v;
  for (int dy = -R; dy <= R; ++dy) {
    const int yy = y + dy;
    if (yy < 0 || yy >= H) continue;
    for (int dx = -R; dx <= R; ++dx) {
      const int xx = x + dx;
      if (xx >= 0 && xx < W) h = fmaxf(h, ld_in<DT>(plane, (long long)yy * sh + xx));
    }
  }
  const float sv = Num<DT>::act(v);
  const bool peak = (v == h) || (sv == Num<DT>::act(h));
  return peak ? __float_as_uint(sv) : 0u;
}

// key of a pixel already known to survive NMS
template <int DT>
__device__ __forceinline__ u32 survivor_key(const void* plane, long long idx, bool pre) {
  const float v = ld_in<DT>(plane, idx);
  if (pre) {
    const u32 bits = __float_as_uint(v);
    return (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
  }
  return __float_as_uint(Num<DT>::act(v));
}

// digit (from the top) at which the cumulative count reaches `need`; bins = 2048
__device__ void pick_digit(const u32* s_hist, int nbins, int need, int* s_out) {
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    const int per = nbins / 32;
    u32 s = 0;
    for (int q = 0; q < per; ++q) s += s_hist[lane * per + q];
    u32 suf = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      u32 t = __shfl_down_sync(0xffffffffu, suf, d);
      if (lane + d < 32) suf += t;
    }
    const u32 mask = __ballot_sync(0xffffffffu, suf >= (u32)need);
    if (mask == 0) {
      if (lane == 0) { s_out[0] = -1; s_out[1] = 0; }
    } else {
      const int L = 31 - __clz(mask);
      if (lane == L) {
        u32 above = suf - s;
        int dsel = L * per;
        for (int q = per - 1; q >= 0; --q) {
          const u32 cq = s_hist[L * per + q];
          if (above + cq >= (u32)need) { dsel = L * per + q; break; }
          above += cq;
        }
        s_out[0] = dsel;
        s_out[1] = (int)above;
      }
    }
  }
  __syncthreads();
}

template <int DT>
__global__ void __launch_bounds__(kExactThreads, kExactCtasPerSm) sdnet_exact_select_kernel(const __grid_constant__ ExactParams p) {
  __shared__ u32 s_hist[2048];
  __shared__ int s_out[2];
  __shared__ int s_warp[kExactThreads / 32][2];
  __shared__ int s_base[2];
  const int C = p.M + p.N;
  const int planes = p.B * C;
  pdl_launch_dependents();
  pdl_wait();  // the peaks kernel's lists and counts are complete and visible
  if (!p.force) {
    // common case: nothing overflowed.  One coalesced look at this CTA's planes, then leave.
    int mine = 0;
    for (int q = blockIdx.x + threadIdx.x * gridDim.x; q < planes; q += blockDim.x * gridDim.x)
      mine |= p.counts[q] > p.cap;
    if (!__syncthreads_or(mine)) return;
  }
  for (int plane_id = blockIdx.x; plane_id < planes; plane_id += gridDim.x) {
  const int emitted = p.counts[plane_id];
  if (!p.force && emitted <= p.cap) continue;  // block-uniform
  __syncthreads();
  const int b = plane_id / C, c = plane_id % C;
  const bool is_anchor = c < p.M;
  const View4& vw = is_anchor ? p.anchor : p.part;
  const void* plane = static_cast<const typename Num<DT>::In*>(vw.data) + (long long)b * vw.sb +
                      (long long)(is_anchor ? c : c - p.M) * vw.sc;
  const long long sh = vw.sh;
  const int K = is_anchor ? p.K : p.P;
  const int H = p.H, W = p.W, HW = H * W, R = p.radius;
  const bool pre = p.pre_activated != 0;
  const int tid = threadIdx.x;
  u64* list = p.lists + (size_t)plane_id * p.cap;
  // per-pixel key cache lives behind the K output records of this plane's list region
  // (cap*8 bytes >= K*8 + H*W/8*... see plan_workspace): 1 bit per pixel "survives NMS".
  u32* bitmap = reinterpret_cast<u32*>(list + K + 2);
  const int words = (HW + 31) / 32;

  // level 1 (top 11 bits) + NMS bitmap
  for (int i = tid; i < 2048; i += blockDim.x) s_hist[i] = 0;
  __syncthreads();
  for (int base = 0; base < words * 32; base += blockDim.x) {
    const int i = base + tid;
    u32 key = 0;
    if (i < HW) key = exact_key<DT>(plane, sh, H, W, R, i / W, i % W, pre);
    const u32 m = __ballot_sync(0xffffffffu, key != 0);
    if ((tid & 31) == 0 && (i >> 5) < words) bitmap[i >> 5] = m;
    if (key) atomicAdd(&s_hist[key >> 21], 1u);
  }
  __syncthreads();
  u32 prefix = 0;
  int need = K;
  bool all = false;
  pick_digit(s_hist, 2048, need, s_out);
  if (s_out[0] < 0) all = true;  // fewer than K survivors: keep them all
  u32 thresh = 0;
  if (!all) {
    need -= s_out[1];
    prefix = (u32)s_out[0];
    __syncthreads();
    // level 2 (next 11 bits)
    for (int i = tid; i < 2048; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    for (int i = tid; i < HW; i += blockDim.x) {
      if (!((bitmap[i >> 5] >> (i & 31)) & 1u)) continue;
      const u32 key = survivor_key<DT>(plane, (long long)(i / W) * sh + (i % W), pre);
      if ((key >> 21) == prefix) atomicAdd(&s_hist[(key >> 10) & 0x7ffu], 1u);
    }
    __syncthreads();
    pick_digit(s_hist, 2048, need, s_out);
    need -= s_out[1];
    prefix = (prefix << 11) | (u32)s_out[0];
    __syncthreads();
    // level 3 (last 10 bits)
    for (int i = tid; i < 1024; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    for (int i = tid; i < HW; i += blockDim.x) {
      if (!((bitmap[i >> 5] >> (i & 31)) & 1u)) continue;
      const u32 key = survivor_key<DT>(plane, (long long)(i / W) * sh + (i % W), pre);
      if ((key >> 10) == prefix) atomicAdd(&s_hist[key & 0x3ffu], 1u);
    }
    __syncthreads();
    pick_digit(s_hist, 1024, need, s_out);
    need -= s_out[1];  // members of the K-th score's tie run still to take, lowest index first
    thresh = (prefix << 10) | (u32)s_out[0];
    __syncthreads();
  }
  // ordered emission
  if (tid < 2) s_base[tid] = 0;  // [0] scores above the threshold so far, [1] tie-run members so far
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  for (int base = 0; base < HW; base += blockDim.x) {
    const int i = base + tid;
    u32 key = 0;
    if (i < HW && ((bitmap[i >> 5] >> (i & 31)) & 1u)) {
      key = survivor_key<DT>(plane, (long long)(i / W) * sh + (i % W), pre);
    }
    const bool gt = key != 0 && (all || key > thresh);
    const bool eq = key != 0 && !all && key == thresh;
    const u32 mg = __ballot_sync(0xffffffffu, gt), me = __ballot_sync(0xffffffffu, eq);
    if (lane == 0) { s_warp[warp][0] = __popc(mg); s_warp[warp][1] = __popc(me); }
    __syncthreads();
    int g_before = 0, e_before = 0;
    for (int w = 0; w < warp; ++w) { g_before += s_warp[w][0]; e_before += s_warp[w][1]; }
    const u32 lt = (1u << lane) - 1u;
    const int e_rank = s_base[1] + e_before + __popc(me & lt);  // tie-run members with a lower index
    const bool take_eq = eq && e_rank < need;
    const int pos = s_base[0] + g_before + __popc(mg & lt) + min(e_rank, need);
    if (gt || take_eq) list[pos] = ((u64)key << 32) | (u32)i;
    __syncthreads();
    if (tid == 0) {
      int g = 0, e = 0;
      for (int w = 0; w < kExactThreads / 32; ++w) { g += s_warp[w][0]; e += s_warp[w][1]; }
      s_base[0] += g;  // scores above the threshold so far
      s_base[1] += e;  // tie-run members so far
    }
    __syncthreads();
  }
  if (tid == 0) {
    p.counts[plane_id] = s_base[0] + min(s_base[1], need);
    p.flags[plane_id] = 1;
  }
  __syncthreads();
  }
}


}  // namespace
