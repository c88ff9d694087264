// peaks_warp.cuh -- sdnet_peaks_kernel: the any-shape, any-alignment form of the peaks kernel (per-lane cp.async
// for fp32, converting loads for fp16/bf16).
#pragma once

namespace {

// ---------------------------------------------------------------------------------------------
// peaks kernel, per-lane form (the fallback: any shape, stride and alignment)
//
// Work unit = (plane, row strip, 128-column panel), one warp per unit, units handed out by an
// atomic counter.  Each warp streams its panel top to bottom through a private shared-memory
// ring of kStages fp32 rows: fp32 maps are copied with per-lane cp.async (4 bytes each, no alignment
// needed), fp16/bf16 maps are loaded and widened by the lanes (RowFeedCvt):
//     row buffer (kPitch floats):  [pad pad hL hL | 128 panel columns | hR hR pad pad]
// Per row the common case is: issue the copy of the row kStages-1 ahead, wait for the row two
// below the centre, read the centre row (one LDS.128), and vote "does any pixel beat the
// pruning floor?".  Only then is the 5x5 window maximum formed (vertical max from the ring,
// neighbours' columns by shuffle, panel-edge columns from the halo slots) and the exact
// sigmoid evaluated for the pixels within a hair of their window maximum.
// ---------------------------------------------------------------------------------------------
constexpr int kStages = 8;             // ring depth (power of two); kStages - 1 - 2R rows stay in flight
constexpr int kPitch = 136;            // floats per ring row
constexpr int kPitchB = kPitch * 4;
// (the last kStages * 8 bytes are unused; dropping them changes the launch's shared memory and wants its own timing)
constexpr int kPeaksSmemPerWarp = kStages * kPitchB + kBins * 8 + kBuf * 8 + kStages * 8;
constexpr int kPeaksSmem = kWarps * kPeaksSmemPerWarp;

// Feeds one warp's ring in the fallback kernel: every lane copies its own four columns with
// 4-byte cp.async (any alignment).  Ring sequence number q of a unit <-> image row row0 + q.
struct RowFeed {
  u32 ring_s, base;
  const char* gown;
  const char* ghalo;
  long long pitch;
  u32 s_own, s_halo, own_ok, halo_ok;
  int row0, H, q_last;

  __device__ __forceinline__ void init(u32 ring, int lane) {
    ring_s = ring; base = 0;
    s_own = ring + (4 + 4 * lane) * 4;
    s_halo = ring + (lane == 31 ? 4 + kPanelW : 2) * 4;
  }
  __device__ __forceinline__ void begin_unit(const void* plane_v, long long sh, int r0, int H_, int W, int panel_col0,
                                             int q_last_, int lane) {
    const float* plane = static_cast<const float*>(plane_v);
    row0 = r0; H = H_; q_last = q_last_;
    const int col0 = panel_col0 + 4 * lane;
    const int halo_col = lane == 31 ? panel_col0 + kPanelW : panel_col0 - 2;
    pitch = sh * 4;
    gown = reinterpret_cast<const char*>(plane + (long long)r0 * sh + col0);
    ghalo = reinterpret_cast<const char*>(plane + (long long)r0 * sh + halo_col);
    own_ok = 0;
    for (int jj = 0; jj < 4; ++jj) own_ok |= (col0 + jj < W ? 1u : 0u) << jj;
    halo_ok = 0;
    if (lane == 0 || lane == 31)
      for (int jj = 0; jj < 2; ++jj) halo_ok |= ((halo_col + jj >= 0 && halo_col + jj < W) ? 1u : 0u) << jj;
    for (int i = lane; i < kStages * kPitch / 4; i += 32) sts128(ring_s + 16 * i, -CUDART_INF_F);
    __syncwarp();
  }
  __device__ __forceinline__ u32 slot_addr(int q) const { return ring_s + (q & (kStages - 1)) * kPitchB; }
  __device__ __forceinline__ void issue(int q, int lane) {
    if (q <= q_last) {
      const u32 so = s_own + (q & (kStages - 1)) * kPitchB, sh = s_halo + (q & (kStages - 1)) * kPitchB;
      if ((unsigned)(row0 + q) < (unsigned)H) {
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) cp_async4_if(so + 4 * jj, gown + 4 * jj, (own_ok >> jj) & 1u);
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) cp_async4_if(sh + 4 * jj, ghalo + 4 * jj, (halo_ok >> jj) & 1u);
      } else {
        sts128(so, -CUDART_INF_F);
        if (lane == 0 || lane == 31) sts64(sh, -CUDART_INF_F);
      }
    }
    gown += pitch;
    ghalo += pitch;
    cp_async_commit();
  }
  // cp.async groups complete in order: allowing kStages-1-2R groups in flight means the row
  // two below the centre has landed
  template <int R>
  __device__ __forceinline__ void wait_step() const { cp_async_wait<kStages - 1 - 2 * R>(); }
  __device__ __forceinline__ void end_unit() { cp_async_wait<0>(); }
};

// Feed for fp16 / bf16 maps: the ring stays fp32 (so everything downstream is shared with the
// fp32 path); each lane loads its own four columns (and lanes 0 / 31 the two halo columns) with
// plain 2-byte loads -- any alignment, any W -- converts, and stores to the ring three steps
// later, so kDepth rows per warp are in flight in registers.  Same call pattern as RowFeed:
// issue(q) makes row q - kDepth resident, which is exactly the row step q - 7 needs.
template <int DT>
struct RowFeedCvt {
  typedef typename Num<DT>::In In;
  static constexpr int kDepth = 3;
  u32 ring_s, s_own, s_halo, own_ok, halo_ok;
  bool vec_ok;  // every row of this lane's four columns is 8-byte aligned
  const In* gown;
  const In* ghalo;
  long long pitch;
  int row0, H, q_last;
  float4 own[kDepth];
  float2 halo[kDepth];

  __device__ __forceinline__ void init(u32 ring, int lane) {
    ring_s = ring;
    s_own = ring + (4 + 4 * lane) * 4;
    s_halo = ring + (lane == 31 ? 4 + kPanelW : 2) * 4;
  }
  __device__ __forceinline__ void begin_unit(const void* plane_v, long long sh, int r0, int H_, int W, int panel_col0,
                                             int q_last_, int lane) {
    const In* plane = static_cast<const In*>(plane_v);
    row0 = r0; H = H_; q_last = q_last_;
    const int col0 = panel_col0 + 4 * lane;
    const int halo_col = lane == 31 ? panel_col0 + kPanelW : panel_col0 - 2;
    pitch = sh;
    gown = plane + (long long)r0 * sh + col0;
    ghalo = plane + (long long)r0 * sh + halo_col;
    vec_ok = (reinterpret_cast<uintptr_t>(gown) % 8 == 0) && (sh % 4 == 0);
    own_ok = 0;
    for (int jj = 0; jj < 4; ++jj) own_ok |= (col0 + jj < W ? 1u : 0u) << jj;
    halo_ok = 0;
    if (lane == 0 || lane == 31)
      for (int jj = 0; jj < 2; ++jj) halo_ok |= ((halo_col + jj >= 0 && halo_col + jj < W) ? 1u : 0u) << jj;
    for (int i = lane; i < kStages * kPitch / 4; i += 32) sts128(ring_s + 16 * i, -CUDART_INF_F);
    __syncwarp();
  }
  __device__ __forceinline__ u32 slot_addr(int q) const { return ring_s + (q & (kStages - 1)) * kPitchB; }
  __device__ __forceinline__ void issue(int q, int lane) {
    const float ninf = -CUDART_INF_F;
    if (q >= kDepth && q - kDepth <= q_last) {  // retire the oldest register stage into the ring
      const u32 slot = (u32)(q - kDepth) & (kStages - 1);
      asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(s_own + slot * kPitchB), "f"(own[0].x), "f"(own[0].y),
                   "f"(own[0].z), "f"(own[0].w) : "memory");
      if (lane == 0 || lane == 31)
        asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(s_halo + slot * kPitchB), "f"(halo[0].x), "f"(halo[0].y) : "memory");
    }
#pragma unroll
    for (int d = 0; d + 1 < kDepth; ++d) { own[d] = own[d + 1]; halo[d] = halo[d + 1]; }
    float4 v = make_float4(ninf, ninf, ninf, ninf);
    float2 hv = make_float2(ninf, ninf);
    if (q <= q_last && (unsigned)(row0 + q) < (unsigned)H) {
      if (own_ok == 15u && vec_ok) {  // four columns in one 8-byte load
        const uint2 raw = __ldg(reinterpret_cast<const uint2*>(gown));
        In e[4];
        memcpy(e, &raw, 8);
        v = make_float4(Num<DT>::to_float(e[0]), Num<DT>::to_float(e[1]), Num<DT>::to_float(e[2]), Num<DT>::to_float(e[3]));
      } else {
        if (own_ok & 1u) v.x = Num<DT>::to_float(__ldg(gown + 0));
        if (own_ok & 2u) v.y = Num<DT>::to_float(__ldg(gown + 1));
        if (own_ok & 4u) v.z = Num<DT>::to_float(__ldg(gown + 2));
        if (own_ok & 8u) v.w = Num<DT>::to_float(__ldg(gown + 3));
      }
      if (halo_ok & 1u) hv.x = Num<DT>::to_float(__ldg(ghalo + 0));
      if (halo_ok & 2u) hv.y = Num<DT>::to_float(__ldg(ghalo + 1));
    }
    own[kDepth - 1] = v;
    halo[kDepth - 1] = hv;
    gown += pitch;
    ghalo += pitch;
  }
  template <int R>
  __device__ __forceinline__ void wait_step() const {}
  __device__ __forceinline__ void end_unit() {}
};

template <int DT>
struct FeedFor { typedef RowFeedCvt<DT> type; };
template <>
struct FeedFor<SDNET_DTYPE_F32> { typedef RowFeed type; };

// Which of a lane's four pixels survive NMS, given their window maxima h0..h3 (logit space).
//   x == h            -> certainly survives;
//   x <  h but so close that the two scores may round equal -> settled with the exact score.
// Columns outside the image hold -inf and never pass x > floorx.
template <int R, int DT = SDNET_DTYPE_F32>
__device__ __forceinline__ u32 classify_row(const float4 ctr, float h0, float h1, float h2, float h3, float floorx) {
  u32 cmask = 0, amb = 0;
#define SDNET_CLASSIFY(x, h, j)                                                                        \
  if ((x) > floorx) {                                                                                  \
    if ((x) == (h)) cmask |= 1u << j;                                                                  \
    else if (may_tie<DT>((x), (h))) amb |= 1u << j;                                                    \
  }
  SDNET_CLASSIFY(ctr.x, h0, 0)
  SDNET_CLASSIFY(ctr.y, h1, 1)
  SDNET_CLASSIFY(ctr.z, h2, 2)
  SDNET_CLASSIFY(ctr.w, h3, 3)
#undef SDNET_CLASSIFY
  // rare: resolve the ambiguous pixels with the exact score function, one per lane per round
  while (__any_sync(0xffffffffu, amb != 0)) {
    const bool has = amb != 0;
    const int jj = has ? __ffs(amb) - 1 : 0;
    const float x = jj == 0 ? ctr.x : (jj == 1 ? ctr.y : (jj == 2 ? ctr.z : ctr.w));
    const float h = jj == 0 ? h0 : (jj == 1 ? h1 : (jj == 2 ? h2 : h3));
    if (has && Num<DT>::act(x) == Num<DT>::act(h)) cmask |= 1u << jj;
    amb &= amb - 1;
  }
  return cmask;
}

// Append the selected pixels of one row as (logit, index) records to the warp's buffer.
// Common case (<= 32 records in the row): positions from three back-to-back ballots on the bits
// of each lane's record count, no branches.  Rows with more (plateaus) go column by column.
template <int DT = SDNET_DTYPE_F32>
__device__ __forceinline__ void append_row(UnitState& st, u32 cmask, const float4 ctr, u32 idx0, u64* buf, u32* hist,
                                           int* minx, const SharedFloors& sf, int* count_ptr,
                                           u64* __restrict__ list, int cap, int K, int lane, bool pre, float xscale,
                                           float satx) {
  const u32 cnt = __popc(cmask);
  const u32 b0 = __ballot_sync(0xffffffffu, cnt & 1u);
  const u32 b1 = __ballot_sync(0xffffffffu, cnt & 2u);
  const u32 b2 = __ballot_sync(0xffffffffu, cnt & 4u);
  const u32 total = __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
  if (total == 0) return;
  const u32 lt = (1u << lane) - 1u;
  if (total <= 32) {
    if (st.nbuf + (int)total > kBuf) {
      __syncwarp();
      flush_candidates<DT>(st, buf, hist, minx, sf, count_ptr, list, cap, K, lane, pre, xscale, satx);
    }
    int pos = st.nbuf + __popc(b0 & lt) + 2 * __popc(b1 & lt) + 4 * __popc(b2 & lt);
    if (cmask & 1u) buf[pos++] = ((u64)__float_as_uint(ctr.x) << 32) | (idx0 + 0);
    if (cmask & 2u) buf[pos++] = ((u64)__float_as_uint(ctr.y) << 32) | (idx0 + 1);
    if (cmask & 4u) buf[pos++] = ((u64)__float_as_uint(ctr.z) << 32) | (idx0 + 2);
    if (cmask & 8u) buf[pos++] = ((u64)__float_as_uint(ctr.w) << 32) | (idx0 + 3);
    st.nbuf += (int)total;
    return;
  }
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    const bool mine = (cmask >> jj) & 1u;
    const u32 m = __ballot_sync(0xffffffffu, mine);
    if (m) {  // warp-uniform
      if (st.nbuf > kBuf - 32) {
        __syncwarp();
        flush_candidates<DT>(st, buf, hist, minx, sf, count_ptr, list, cap, K, lane, pre, xscale, satx);
      }
      if (mine) buf[st.nbuf + __popc(m & lt)] = ((u64)__float_as_uint(comp(ctr, jj)) << 32) | (idx0 + jj);
      st.nbuf += __popc(m);
    }
  }
}

template <int R, int DT>
__global__ void __launch_bounds__(kThreads, DT == SDNET_DTYPE_F32 ? 4 : 3)
sdnet_peaks_kernel(const __grid_constant__ PeaksParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  unsigned char* wbase = smem_raw + (size_t)warp * kPeaksSmemPerWarp;
  const u32 ring_s = smem_u32(wbase);
  u32* hist = reinterpret_cast<u32*>(wbase + kStages * kPitchB);
  int* minx = reinterpret_cast<int*>(hist + kBins);
  u64* buf = reinterpret_cast<u64*>(minx + kBins);
  const bool pre = p.pre_activated != 0;
  const float xscale = pre ? kPreScale : 1.0f;
  const float satx = pre ? CUDART_INF_F : kSatX;
  const int C = p.M + p.N;
  const int H = p.H, W = p.W;
  const u32 own_off = (4 + 4 * lane) * 4;                      // this lane's four columns inside a ring row
  const u32 halo_off = (lane == 31 ? 4 + kPanelW : 2) * 4;     // the two columns beyond the panel edge
  typename FeedFor<DT>::type feed;
  feed.init(ring_s, lane);

  for (;;) {
    u32 unit = 0;
    if (lane == 0) unit = atomicAdd(p.sched, 1u);
    unit = __shfl_sync(0xffffffffu, unit, 0);
    if (unit >= (u32)p.units) break;
    const int panel = unit % p.panels;
    const int t1 = unit / p.panels;
    const int strip = t1 % p.strips;
    const int plane_id = t1 / p.strips;
    const int b = plane_id / C, c = plane_id % C;
    const bool is_anchor = c < p.M;
    const View4& vw = is_anchor ? p.anchor : p.part;
    const void* plane = static_cast<const typename Num<DT>::In*>(vw.data) + (long long)b * vw.sb +
                        (long long)(is_anchor ? c : c - p.M) * vw.sc;
    const int K = is_anchor ? p.K : p.P;
    const int panel_col0 = panel * kPanelW;
    const int col0 = panel_col0 + lane * 4;
    const int r_begin = strip * p.rows_per_strip;
    const int r_end = min(H, r_begin + p.rows_per_strip);
    const int nrows = r_end - r_begin;
    const int q_last = nrows - 1 + 2 * R;  // ring sequence number of the last row any centre row needs
    u64* __restrict__ list = p.lists + (size_t)plane_id * p.cap;
    int* count_ptr = p.counts + plane_id;
    int* gfloor_ptr = p.gfloor + plane_id;
    SharedFloors sf;
    sf.ghist = p.ghist + (size_t)plane_id * kFineBins;
    sf.gfloor = gfloor_ptr;

    UnitState st;
    st.floorx = shared_floor<DT>(__ldcg(gfloor_ptr), xscale);
    st.emitted = 0;
    st.nbuf = 0;

    __syncwarp();  // everyone is done with the previous unit's ring, histogram and buffer
    *reinterpret_cast<uint4*>(hist + 4 * lane) = make_uint4(0, 0, 0, 0);
    *reinterpret_cast<int4*>(minx + 4 * lane) = make_int4(0x7fffffff, 0x7fffffff, 0x7fffffff, 0x7fffffff);
    feed.begin_unit(plane, vw.sh, r_begin - R, H, W, panel_col0, q_last, lane);
#pragma unroll
    for (int q = 0; q < kStages - 1; ++q) feed.issue(q, lane);

    for (int t = 0; t < nrows; ++t) {
      // the slot of sequence number t-1 is free: every lane passed a warp-wide vote after reading it
      feed.issue(t + kStages - 1, lane);
      feed.template wait_step<R>();
      __syncwarp();
      const float4 ctr = lds128(feed.slot_addr(t + R) + own_off);
      const float m4 = fmaxf(fmaxf(ctr.x, ctr.y), fmaxf(ctr.z, ctr.w));
      if (__any_sync(0xffffffffu, m4 > st.floorx)) {
        const float floorx = st.floorx;
        u32 cmask = 0;  // bit j: pixel col0+j goes to the candidate buffer
        if (!pre) {
          // vertical (2R+1)-max of own columns and of this lane's halo pair (lanes 0 / 31 only)
          float4 v = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
          float2 hvv = make_float2(-CUDART_INF_F, -CUDART_INF_F);
#pragma unroll
          for (int d = 0; d <= 2 * R; ++d) {
            const u32 so = feed.slot_addr(t + d);
            const float4 o = lds128(so + own_off);
            const float2 ho = lds64(so + halo_off);
            v.x = fmaxf(v.x, o.x); v.y = fmaxf(v.y, o.y); v.z = fmaxf(v.z, o.z); v.w = fmaxf(v.w, o.w);
            hvv.x = fmaxf(hvv.x, ho.x); hvv.y = fmaxf(hvv.y, ho.y);
          }
          float L2 = __shfl_up_sync(0xffffffffu, v.z, 1);
          float L3 = __shfl_up_sync(0xffffffffu, v.w, 1);
          float R0 = __shfl_down_sync(0xffffffffu, v.x, 1);
          float R1 = __shfl_down_sync(0xffffffffu, v.y, 1);
          if (lane == 0) { L2 = hvv.x; L3 = hvv.y; }
          if (lane == 31) { R0 = hvv.x; R1 = hvv.y; }
          float h0, h1, h2, h3;
          if (R == 2) {
            const float m12 = fmaxf(v.y, v.z);
            h0 = max3(fmaxf(L2, L3), v.x, m12);
            h1 = max3(fmaxf(L3, v.x), m12, v.w);
            h2 = max3(fmaxf(v.x, R0), m12, v.w);
            h3 = max3(fmaxf(R0, R1), m12, v.w);
          } else {
            h0 = max3(L3, v.x, v.y);
            h1 = max3(v.x, v.y, v.z);
            h2 = max3(v.y, v.z, v.w);
            h3 = max3(v.z, v.w, R0);
          }
          cmask = classify_row<R, DT>(ctr, h0, h1, h2, h3, floorx);
        } else {
          // pre-activated maps (CoreMLDecoder): every pixel above the floor is a candidate
          if (ctr.x > floorx) cmask |= 1u;
          if (ctr.y > floorx) cmask |= 2u;
          if (ctr.z > floorx) cmask |= 4u;
          if (ctr.w > floorx) cmask |= 8u;
        }
        append_row<DT>(st, cmask, ctr, (u32)((r_begin + t) * W + col0), buf, hist, minx, sf, count_ptr, list,
                   p.cap, K, lane, pre, xscale, satx);
      }
      if ((t & 7) == 7) {
        // every 8 rows: pick up the plane-wide floor other warps may have raised
        st.floorx = fmaxf(st.floorx, shared_floor<DT>(__ldcg(gfloor_ptr), xscale));
      }
    }
    feed.end_unit();
    if (st.nbuf) {
      __syncwarp();
      flush_candidates<DT>(st, buf, hist, minx, sf, count_ptr, list, p.cap, K, lane, pre, xscale, satx);
    }
  }
}


}  // namespace
