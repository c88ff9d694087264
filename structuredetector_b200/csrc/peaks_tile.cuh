// peaks_tile.cuh -- sdnet_peaks_tile_kernel: the default peaks kernel (TMA tensor-map tiles, autonomous warps).
#pragma once

namespace {

// ---------------------------------------------------------------------------------------------
// peaks kernel, TMA-tile form (the default; needs a base and pitches TMA can describe, see
// tile_rows_per_tma_row in sdnet_decode.cu)
//
// Every warp is an autonomous pipeline over one (plane, row strip, panel) unit; a lane owns one
// 16-byte word per row (4 fp32 or 8 fp16/bf16 pixels), so a panel is 128 or 256 columns.  An elected
// lane pulls 4-row tiles (the panel plus one word either side) into the warp's private shared-memory
// ring with tensor-map bulk copies (TMA, SASS UTMALDG), completion on one mbarrier per ring slot.
// The tensor map is encoded with NaN out-of-bounds fill: fmaxf / max.f16x2 ignore a NaN operand and
// every ordered comparison with NaN is false, so out-of-image rows and columns behave exactly like
// max_pool2d's -inf padding with no edge code at all.  Per group of four output rows the warp waits
// on one barrier, reads its four centre rows (4 x LDS.128), takes the max of the 16 / 32 values and
// votes "does anything here beat the pruning floor?"; only then does it list the words that do and
// give every listed pixel a lane of its own (settle_entries).  No warp ever waits for another warp.
// ---------------------------------------------------------------------------------------------
constexpr int kGroupRows = 4;                                // output rows per TMA tile and per fast-path test
constexpr int kTileCols = kPanelW + 8;
constexpr int kTilePitchB = kTileCols * 4;                   // 544 B per ring row
constexpr int kTileBytes = kGroupRows * kTilePitchB;         // 2176 B per TMA tile (17 x 128 B)
constexpr int kTileWarps = 4;  // warps per CTA; they never talk to each other (no __syncthreads in the kernel)
constexpr int kTileMinCtas = 6;  // resident CTAs per SM the register allocation aims for (24 warps)
constexpr int kMinChunkGroups = 8;  // shortest tier-2 unit (32 rows)
constexpr int kTileNG = 3;   // ring slots (tiles) per warp: a group reads two of them, the others are in flight
constexpr int kWork = 128;   // per-warp work list: one byte per (row of the group, lane) whose 16-byte word holds a pixel above the floor
constexpr int kFlushAt = 16;  // buffered candidates that trigger a flush
// S = rows per TMA row (see the kernel).  Under S = 2 a tile arrives as two 2-row boxes and a TMA
// destination must be 128-byte aligned: the second box sits at +1152 and a slot takes 2304 bytes.
__host__ __device__ constexpr int tile_slot_bytes(int S) { return S == 1 ? kTileBytes : 2304; }
__host__ __device__ constexpr int tile_smem_per_warp(int S) {
  return ((kTileNG * tile_slot_bytes(S) + 32 + kBins * 8 + kBuf * 8 + kWork) + 127) / 128 * 128;
}
__host__ __device__ constexpr int tile_smem(int S) { return kTileWarps * tile_smem_per_warp(S); }
constexpr int kOddBoxOff = 1152;  // S = 2: offset of the odd rows' box inside a slot
constexpr int kOddShiftB = 8;     // S = 2: a box must start on a 16-byte boundary of global memory and odd rows start 8 bytes
                                  // off one, so their box starts 4 columns early and their pixels sit 8 bytes further right

// Element geometry of the tile kernel.  A lane owns one 16-byte word per row: 4 fp32 or 8 fp16/bf16
// pixels, so a warp's panel is 128 or 256 columns and a ring row is 544 bytes either way.
template <int DT>
struct TileGeom {
  static constexpr int kPx = DT == SDNET_DTYPE_F32 ? 4 : 8;  // pixels per lane per row = halo columns each side
  static constexpr int kEsz = 16 / kPx;                       // bytes per element
  static constexpr int kPanel = 32 * kPx;                     // columns per warp
  static constexpr int kCols = kPanel + 2 * kPx;              // columns per tile row
};
static_assert(TileGeom<SDNET_DTYPE_F32>::kCols * 4 == kTilePitchB && TileGeom<SDNET_DTYPE_F16>::kCols * 2 == kTilePitchB, "ring row pitch");

__device__ __forceinline__ void tma_tile_4d(u32 dst, const CUtensorMap* map, int x, int y, int c, int b, u32 bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(dst), "l"(map), "r"(x), "r"(y), "r"(c), "r"(b), "r"(bar) : "memory");
}
__device__ __forceinline__ uint4 lds64x2(u32 addr) {  // 16 bytes from an 8-byte-aligned address
  uint4 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.z), "=r"(v.w) : "r"(addr + 8));
  return v;
}
__device__ __forceinline__ uint4 lds128u(u32 addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// max of the 4 | 8 elements of one 16-byte word / of four words, as float; NaN elements (the TMA
// out-of-bounds fill) are ignored by fmaxf and by max.f16x2 / max.bf16x2 alike
template <int DT>
struct TileMax;
template <>
struct TileMax<SDNET_DTYPE_F32> {
  static __device__ __forceinline__ float word(const uint4& a) {
    return fmaxf(fmaxf(__uint_as_float(a.x), __uint_as_float(a.y)), fmaxf(__uint_as_float(a.z), __uint_as_float(a.w)));
  }
  static __device__ __forceinline__ float group(const uint4& a, const uint4& b, const uint4& c, const uint4& d) {
    return fmaxf(fmaxf(word(a), word(b)), fmaxf(word(c), word(d)));
  }
  static __device__ __forceinline__ float elem(u32 addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
  }
  // one element in its storage format (here: the float's bits), max in that format, back to float
  static __device__ __forceinline__ u32 raw(u32 addr) { return __float_as_uint(elem(addr)); }
  static __device__ __forceinline__ u32 rmax(u32 a, u32 b) { return __float_as_uint(fmaxf(__uint_as_float(a), __uint_as_float(b))); }
  static __device__ __forceinline__ float rfloat(u32 r) { return __uint_as_float(r); }
};
template <>
struct TileMax<SDNET_DTYPE_F16> {
  static __device__ __forceinline__ __half2 h2(u32 v) { return *reinterpret_cast<const __half2*>(&v); }
  static __device__ __forceinline__ __half2 word2(const uint4& a) { return __hmax2(__hmax2(h2(a.x), h2(a.y)), __hmax2(h2(a.z), h2(a.w))); }
  static __device__ __forceinline__ float fold(__half2 m) { return __half2float(__hmax(__low2half(m), __high2half(m))); }
  static __device__ __forceinline__ float word(const uint4& a) { return fold(word2(a)); }
  static __device__ __forceinline__ float group(const uint4& a, const uint4& b, const uint4& c, const uint4& d) {
    return fold(__hmax2(__hmax2(word2(a), word2(b)), __hmax2(word2(c), word2(d))));
  }
  static __device__ __forceinline__ float elem(u32 addr) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
    return __half2float(__ushort_as_half(v));
  }
  // storage format: the 16 bits in the low half of a register (high half +0); max.f16x2 ignores NaN
  static __device__ __forceinline__ u32 raw(u32 addr) {
    u32 v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
  }
  static __device__ __forceinline__ u32 rmax(u32 a, u32 b) {
    const __half2 m = __hmax2(h2(a), h2(b));
    return *reinterpret_cast<const u32*>(&m);
  }
  static __device__ __forceinline__ float rfloat(u32 r) { return __half2float(__ushort_as_half((unsigned short)r)); }
};
template <>
struct TileMax<SDNET_DTYPE_BF16> {
  static __device__ __forceinline__ __nv_bfloat162 h2(u32 v) { return *reinterpret_cast<const __nv_bfloat162*>(&v); }
  static __device__ __forceinline__ __nv_bfloat162 word2(const uint4& a) { return __hmax2(__hmax2(h2(a.x), h2(a.y)), __hmax2(h2(a.z), h2(a.w))); }
  static __device__ __forceinline__ float fold(__nv_bfloat162 m) { return __bfloat162float(__hmax(__low2bfloat16(m), __high2bfloat16(m))); }
  static __device__ __forceinline__ float word(const uint4& a) { return fold(word2(a)); }
  static __device__ __forceinline__ float group(const uint4& a, const uint4& b, const uint4& c, const uint4& d) {
    return fold(__hmax2(__hmax2(word2(a), word2(b)), __hmax2(word2(c), word2(d))));
  }
  static __device__ __forceinline__ float elem(u32 addr) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
    return __uint_as_float((u32)v << 16);
  }
  static __device__ __forceinline__ u32 raw(u32 addr) {
    u32 v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
  }
  static __device__ __forceinline__ u32 rmax(u32 a, u32 b) {
    const __nv_bfloat162 m = __hmax2(h2(a), h2(b));
    return *reinterpret_cast<const u32*>(&m);
  }
  static __device__ __forceinline__ float rfloat(u32 r) { return __uint_as_float(r << 16); }
};

// Byte offset of ring row rr (0..15) inside the ring.  S = 1: rows in order.  S = 2 (rows loaded as
// even/odd pairs, see the kernel): a slot holds rows 0, 2 at +0, +544 and rows 1, 3 at +1152, +1696,
// the odd rows shifted right by kOddShiftB bytes.
template <int S>
__device__ __forceinline__ u32 ring_row_off(u32 rr) {
  if (S == 1) return rr * kTilePitchB;
  return (rr >> 2) * tile_slot_bytes(2) + (rr & 1u) * (kOddBoxOff + kOddShiftB) + ((rr >> 1) & 1u) * kTilePitchB;
}

// Settle the work list of one 4-row group.  Entry e = (row in group << 5) | lane names one 16-byte
// word of centre pixels holding at least one pixel above the floor; kPx consecutive lanes take the
// pixels of an entry.  (Listing the two halves of a fp16 / bf16 word separately -- twice the ballots, half the
// passes -- measured 2-3 % slower: 0.656 / 0.775 ms against 0.639 / 0.757 ms.)  A lane whose pixel beats the
// floor reads the pixel's (2R+1)^2 window from the ring with scalar loads (columns and rows outside
// the image hold NaN or -inf and never win a max), classifies it like classify_row and appends a
// (logit, index) record to the warp's candidate buffer.
// `row0` = ring row of the window's first row for group row 0 (the centre is R rows further).
template <int R, int DT, int S>
__device__ __forceinline__ void settle_entries(UnitState& st, const unsigned char* work, int nent, u32 ring_s, u32 row0,
                                               u32 row_tab, float floorx, u32 idx0, int W, bool pre, u64* buf, u32* hist, int* minx,
                                               const SharedFloors& sf, int* count_ptr, u64* __restrict__ list, int cap,
                                               int K, int lane, float xscale, float satx) {
  constexpr u32 kRingRows = kTileNG * kGroupRows;
  constexpr int kPx = TileGeom<DT>::kPx, kEsz = TileGeom<DT>::kEsz;
  const int nslots = kPx * nent;
  for (int base = 0; base < nslots; base += 32) {  // warp-uniform
    const int slot = base + lane;
    const u32 e = slot < nslots ? work[slot / kPx] : 0u;
    const u32 i = e >> 5, colp = kPx * (e & 31u) + (u32)(slot % kPx);
    const u32 col_addr = ring_s + (kPx + colp - R) * kEsz;  // first column of the window
    // byte offsets of the window's rows.  Plain rows: a multiply.  Row pairs: the slot layout makes that
    // eight instructions per row, so lane k keeps the offset of ring row k (row_tab) and a shuffle looks it up
    u32 roff[2 * R + 1];
#pragma unroll
    for (int d = 0; d <= 2 * R; ++d) {
      u32 rr = row0 + i + d;  // < 2 * kRingRows
      if (rr >= kRingRows) rr -= kRingRows;
      roff[d] = S == 1 ? rr * kTilePitchB : __shfl_sync(0xffffffffu, row_tab, (int)rr);
    }
    const float x = TileMax<DT>::elem(col_addr + R * kEsz + roff[R]);
    bool keep = slot < nslots && x > floorx;
    if (!pre) {
      // Most pixels above the floor are not peaks but the flanks of one (a blob holds ~200 of them): four loads
      // settle those.  With m4 = the largest of the four direct neighbours (<= the window maximum h), x cannot
      // share h's score when x < m4 - kNear2, x <= kHi2 - 1 and x >= kLo (the four near-tie zones all need the
      // opposite); NaN neighbours (outside the image) are ignored by fmaxf.
      const u32 ctr = col_addr + R * kEsz;
      const float m4 = fmaxf(fmaxf(TileMax<DT>::elem(ctr + roff[R - 1]), TileMax<DT>::elem(ctr + roff[R + 1])),
                             fmaxf(TileMax<DT>::elem(ctr - kEsz + roff[R]), TileMax<DT>::elem(ctr + kEsz + roff[R])));
      if (x < m4 - Num<DT>::kNear2 && x <= Num<DT>::kHi2 - 1.0f && x >= Num<DT>::kLo) keep = false;
    }
    if (keep && !pre) {
      // window max in the storage format (no conversions for fp16/bf16), one accumulator per window row
      u32 hr[2 * R + 1];
#pragma unroll
      for (int d = 0; d <= 2 * R; ++d) {
        const u32 a = col_addr + roff[d];
        u32 v[2 * R + 1];
#pragma unroll
        for (int q = 0; q <= 2 * R; ++q) v[q] = TileMax<DT>::raw(a + kEsz * q);
        hr[d] = v[0];
#pragma unroll
        for (int q = 1; q <= 2 * R; ++q) hr[d] = TileMax<DT>::rmax(hr[d], v[q]);
      }
#pragma unroll
      for (int d = 1; d <= 2 * R; ++d) hr[0] = TileMax<DT>::rmax(hr[0], hr[d]);
      const float h = fmaxf(x, TileMax<DT>::rfloat(hr[0]));  // an all-NaN window cannot happen: the centre is in it
      if (x != h) keep = may_tie<DT>(x, h) && Num<DT>::act(x) == Num<DT>::act(h);  // rare
    }
    const u32 m = __ballot_sync(0xffffffffu, keep);
    if (m) {  // warp-uniform
      if (st.nbuf + __popc(m) > kBuf) {
        __syncwarp();
        flush_candidates<DT, false>(st, buf, hist, minx, sf, count_ptr, list, cap, K, lane, pre, xscale, satx);
      }
      if (keep) {
        buf[st.nbuf + __popc(m & ((1u << lane) - 1u))] = ((u64)__float_as_uint(x) << 32) | (idx0 + i * (u32)W + colp);
        // counted in the plane-wide histogram when found, not when flushed: the plane's other warps see it at once
        atomicAdd(&sf.ghist[fine_bin(fminf(fmaxf(x * xscale, -satx), satx))], 1u);
      }
      st.nbuf += __popc(m);
    }
  }
}

// Dense settle of one 4-row group (fp32, plain rows): when many blocks are hot -- the first groups of a unit, before
// the plane has a floor worth the name -- giving every pixel a lane of its own costs a pass of ~100 instructions per
// two blocks.  Here the whole (2R+1)^2 maximum filter of the group is formed once in registers instead: each lane
// loads its word of the 4 + 2R window rows (lanes 0 / 31 also the panel's halo words), takes the vertical maxima of
// its four columns for each of the four centre rows (one row at a time: few registers), fetches the two neighbouring columns either side from the
// adjacent lanes by shuffle, and classifies its 16 pixels exactly like the pixel-centric path.  ~300 instructions for
// the group, whatever the number of hot pixels.  Returns false (nothing recorded) when the group holds more
// survivors than the candidate buffer: the caller then takes the pixel-centric path, which flushes as it goes.
constexpr int kDenseLanes = 16;  // hot lanes from which the dense path is taken


// The dense maximum filter of one 4-row group (fp32, plain rows): bit 4 i + c of the result says that pixel
// (group row i, column c of this lane's word) is above `floorx` and survives the reference's NMS.
template <int R>
__device__ __forceinline__ u32 dense_keep_mask_f32(int rows_here, u32 ring_s, u32 ring_own, u32 row0, float floorx, bool pre, int lane) {
  constexpr int DT = SDNET_DTYPE_F32;
  constexpr u32 kRingRows = kTileNG * kGroupRows;
  // own word and, for the panel's edge lanes, the halo word next to it (the other lanes read word 0 for nothing)
  const u32 halo_a = ring_s + (lane == 31 ? 33u * 16u : 0u);
  u32 km = 0;  // bit 4 i + c: pixel (group row i, column c of this lane's word) is a candidate
#pragma unroll
  for (int i = 0; i < kGroupRows; ++i) {
    if (i < rows_here) {  // warp-uniform
      // vertical maxima over the window rows of centre row i, re-read from the ring row by row: shared-memory loads are
      // cheap, registers are what limits the kernel's occupancy (fmaxf ignores the NaN of out-of-image rows)
      float4 v, xc;
      float2 ev;
#pragma unroll
      for (int d = 0; d <= 2 * R; ++d) {
        u32 rr = row0 + i + d;
        if (rr >= kRingRows) rr -= kRingRows;
        const float4 a = lds128(ring_own + rr * kTilePitchB);
        const float4 w = lds128(halo_a + rr * kTilePitchB);
        const float2 e = lane == 31 ? make_float2(w.x, w.y) : make_float2(w.z, w.w);
        if (d == 0) {
          v = a;
          ev = e;
        } else {
          v.x = fmaxf(v.x, a.x); v.y = fmaxf(v.y, a.y); v.z = fmaxf(v.z, a.z); v.w = fmaxf(v.w, a.w);
          ev.x = fmaxf(ev.x, e.x); ev.y = fmaxf(ev.y, e.y);
        }
        if (d == R) xc = a;
      }
      // the two columns either side, from the neighbouring lanes (panel edges: from the halo words)
      float l2 = __shfl_up_sync(0xffffffffu, v.z, 1), l3 = __shfl_up_sync(0xffffffffu, v.w, 1);
      float r0 = __shfl_down_sync(0xffffffffu, v.x, 1), r1 = __shfl_down_sync(0xffffffffu, v.y, 1);
      if (lane == 0) { l2 = ev.x; l3 = ev.y; }
      if (lane == 31) { r0 = ev.x; r1 = ev.y; }
      float4 h;
      if (R == 2) {
        h.x = max3(max3(l2, l3, v.x), v.y, v.z);
        h.y = max3(max3(l3, v.x, v.y), v.z, v.w);
        h.z = max3(max3(v.x, v.y, v.z), v.w, r0);
        h.w = max3(max3(v.y, v.z, v.w), r0, r1);
      } else {
        h.x = max3(l3, v.x, v.y);
        h.y = max3(v.x, v.y, v.z);
        h.z = max3(v.y, v.z, v.w);
        h.w = max3(v.z, v.w, r0);
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float x = comp(xc, c), hh = comp(h, c);
        bool keep = x > floorx;
        if (keep && !pre && x != hh) keep = may_tie<DT>(x, hh) && Num<DT>::act(x) == Num<DT>::act(hh);  // rare
        km |= (keep ? 1u : 0u) << (4 * i + c);
      }
    }
  }
  return km;
}

template <int R>
__device__ __forceinline__ bool settle_dense_f32(UnitState& st, int rows_here, u32 ring_s, u32 ring_own, u32 row0, float floorx,
                                                 u32 idx0, int W, bool pre, u64* buf, u32* hist, int* minx, const SharedFloors& sf,
                                                 int* count_ptr, u64* __restrict__ list, int cap, int K, int lane, float xscale,
                                                 float satx) {
  constexpr int DT = SDNET_DTYPE_F32;
  constexpr u32 kRingRows = kTileNG * kGroupRows;
  u32 km = dense_keep_mask_f32<R>(rows_here, ring_s, ring_own, row0, floorx, pre, lane);
  // where this lane's records go: exclusive prefix of the per-lane counts
  const int cnt = __popc(km);
  int incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += t;
  }
  const int total = __shfl_sync(0xffffffffu, incl, 31);
  if (total == 0) return true;
  if (total > kBuf) return false;
  if (st.nbuf + total > kBuf) {
    __syncwarp();
    flush_candidates<DT, false>(st, buf, hist, minx, sf, count_ptr, list, cap, K, lane, pre, xscale, satx);
  }
  int pos = st.nbuf + incl - cnt;
  const u32 centre0 = row0 + R;
  while (km) {
    const int bit = __ffs(km) - 1;
    km &= km - 1;
    const u32 i = (u32)bit >> 2, c = (u32)bit & 3u;
    u32 rr = centre0 + i;
    if (rr >= kRingRows) rr -= kRingRows;
    const float x = TileMax<DT>::elem(ring_own + rr * kTilePitchB + 4 * c);
    buf[pos++] = ((u64)__float_as_uint(x) << 32) | (idx0 + i * (u32)W + 4u * (u32)lane + c);
    atomicAdd(&sf.ghist[fine_bin(fminf(fmaxf(x * xscale, -satx), satx))], 1u);
  }
  st.nbuf += total;
  return true;
}

// S = 2 only: a tile that touches the left or right image edge has read across a row boundary (see
// the kernel): overwrite what is not this row's data with -inf.  `slot_s` = the tile's ring slot.
template <int DT>
__device__ __forceinline__ void tile_fix_edges(u32 slot_s, int x0, int W, int lane) {
  constexpr int kPx = TileGeom<DT>::kPx;
  constexpr u32 kNinf2 = DT == SDNET_DTYPE_F16 ? 0xFC00FC00u : (DT == SDNET_DTYPE_BF16 ? 0xFF80FF80u : 0xFF800000u);
  if (x0 < 0) {  // odd rows (the second box): the 12 columns left of column 0 hold the end of the row above
    if (lane < 2) {
      const u32 a = slot_s + kOddBoxOff + lane * kTilePitchB;
      asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(a), "r"(kNinf2) : "memory");
      asm volatile("st.shared.v2.u32 [%0], {%1, %1};" ::"r"(a + 16), "r"(kNinf2) : "memory");
    }
  }
  if (x0 + TileGeom<DT>::kCols > W) {  // even rows (the first box): columns >= W hold the start of the row below
    // word w of a ring row covers columns x0 + kPx w ..; under S = 2 W is a multiple of kPx/2, not of kPx
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int w = k == 0 ? lane + 1 : 33;  // lane's own centre word; lane 31 also takes the right halo word
      if (k == 1 && lane != 31) break;
      const int first = x0 + kPx * w;
      const u32 a = slot_s + 16 * w;
      if (first >= W) {
        asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(a), "r"(kNinf2) : "memory");
        asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(a + kTilePitchB), "r"(kNinf2) : "memory");
      } else if (first + kPx / 2 >= W) {
        asm volatile("st.shared.v2.u32 [%0], {%1, %1};" ::"r"(a + 8), "r"(kNinf2) : "memory");
        asm volatile("st.shared.v2.u32 [%0], {%1, %1};" ::"r"(a + 8 + kTilePitchB), "r"(kNinf2) : "memory");
      }
    }
  }
}

// S = rows per TMA row: 1 when the row pitch is a multiple of 16 bytes.  S = 2 serves fp16/bf16 maps
// whose pitch is an odd multiple of 8 bytes (W = 612): the tensor map then describes PAIRS of image
// rows as one row of pitch + W elements, a tile is two 2-row boxes -- the even rows at x, the odd rows
// at pitch + x - 4 (a box has to start on a 16-byte boundary, measured: anything else is an illegal
// instruction) -- and lands in its slot as rows 0, 2 | 1, 3 with the odd rows 8 bytes further right.
// At the image edges such a box reads across the row boundary; tile_fix_edges repairs that after the wait.
// kHint: the launch has floor hints (HintParams; sdnet_decode.cu picks the instantiation).  Without, the hint code is
// compiled out: the flag it needs for the polling below costs a register, and a launch with no hints to give should not
// pay for it.
template <int R, int DT, int S, bool kHint>
__global__ void __launch_bounds__(kTileWarps * 32, kTileMinCtas)
sdnet_peaks_tile_kernel(const __grid_constant__ PeaksParams p, const __grid_constant__ CUtensorMap tm_anchor,
                        const __grid_constant__ CUtensorMap tm_part, const __grid_constant__ HintParams hp) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int NG = kTileNG;
  constexpr u32 kRingRows = NG * kGroupRows;
  constexpr int kPx = TileGeom<DT>::kPx, kPanel = TileGeom<DT>::kPanel;
  static_assert(NG >= 3 && kRingRows <= 32, "a group reads two slots; ring-row offsets are looked up by lane");
  static_assert(S == 1 || (R == 2 && DT != SDNET_DTYPE_F32), "row pairs: tiles must start on an even row");
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  constexpr u32 kSlotB = tile_slot_bytes(S);
  unsigned char* wbase = smem_raw + (size_t)warp * tile_smem_per_warp(S);
  const u32 ring_s = smem_u32(wbase);
  const u32 bars_s = ring_s + NG * kSlotB;
  u32* hist = reinterpret_cast<u32*>(wbase + NG * kSlotB + 32);
  int* minx = reinterpret_cast<int*>(hist + kBins);
  u64* buf = reinterpret_cast<u64*>(minx + kBins);
  unsigned char* work = reinterpret_cast<unsigned char*>(buf + kBuf);
  const u32 lt = (1u << lane) - 1u;
  const bool pre = p.pre_activated != 0;
  const float xscale = pre ? kPreScale : 1.0f;
  const float satx = pre ? CUDART_INF_F : kSatX;
  const int C = p.M + p.N;
  const int H = p.H, W = p.W;
  const u32 ring_own = ring_s + (u32)(16 + 16 * lane);  // this lane's word inside a ring row
  const u32 row_tab = ring_row_off<S>((u32)lane % kRingRows);  // lane k: byte offset of ring row k (see settle_entries)

  if (lane == 0) {
    for (int i = 0; i < NG; ++i) mbar_init(bars_s + 8 * i, 1);
    mbar_fence_init();
  }
  __syncwarp();

  // Tiles are numbered in one running sequence over all units this warp processes: tile number n
  // lives in ring slot n % NG (ring rows 4 (n % NG) ..) and is the (n / NG)-th use of that slot, so
  // the slot's mbarrier is waited with parity (n / NG) & 1.  Every issued tile is waited exactly once.
  // (slot, parity) of the current tile are carried in registers and stepped, so NG need not be a power of two.
  u32 cur_slot = 0, cur_par = 0;
  auto step_pos = [&](u32& slot, u32& par) {
    if (++slot == (u32)NG) { slot = 0; par ^= 1u; }
  };
  for (;;) {
    u32 unit = 0;
    if (lane == 0) unit = atomicAdd(p.sched, 1u);
    unit = __shfl_sync(0xffffffffu, unit, 0);
    if (unit >= (u32)p.units) break;
    // the unit's piece of the line of groups; it is walked one column segment at a time
    u32 pos, pos_end;
    if (unit < (u32)p.tier1_units) {
      pos = unit * (u32)p.groups_per_col;
      pos_end = pos + (u32)p.groups_per_col;
    } else {
      pos = (u32)p.tier1_units * (u32)p.groups_per_col + (unit - (u32)p.tier1_units) * (u32)p.chunk_groups;
      pos_end = min(p.total_groups, pos + (u32)p.chunk_groups);
    }
    while (pos < pos_end) {  // warp-uniform
    const u32 column = pos / (u32)p.groups_per_col;
    const int g_first = (int)(pos - column * (u32)p.groups_per_col);
    const int g_last = min(p.groups_per_col, g_first + (int)(pos_end - pos));
    pos += (u32)(g_last - g_first);
    const int panel = (int)(column % (u32)p.panels), plane_id = (int)(column / (u32)p.panels);
    const int r_begin = g_first * kGroupRows, r_end = min(H, g_last * kGroupRows);
    const int b = plane_id / C, c = plane_id % C;
    const bool is_anchor = c < p.M;
    const CUtensorMap* tmap = is_anchor ? &tm_anchor : &tm_part;
    const int csel = is_anchor ? c : c - p.M;
    const int K = is_anchor ? p.K : p.P;
    const int x0 = panel * kPanel - kPx;  // first column of the tile; tensor-map coordinates count 4-byte units
    const int xc = DT == SDNET_DTYPE_F32 ? x0 : x0 >> 1;
    const bool edge = S == 2 && (x0 < 0 || x0 + TileGeom<DT>::kCols > W);
    const int nrows = r_end - r_begin;
    const int groups = (nrows + 2 * R + kGroupRows - 1) / kGroupRows;  // tiles of the unit
    const int groups_out = (nrows + kGroupRows - 1) / kGroupRows;
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
    __syncwarp();

    // tile k of the unit = image rows r_begin - R + 4k ..
    auto issue = [&](u32 s, int y) {  // lane 0: pull the tile whose first image row is y into slot s
      mbar_arrive_expect_tx(bars_s + 8 * s, kTileBytes);
      if (S == 1) {
        tma_tile_4d(ring_s + s * kSlotB, tmap, xc, y, csel, b, bars_s + 8 * s);
      } else {  // y is even (r_begin even, R = 2): rows y, y+2 then rows y+1, y+3
        tma_tile_4d(ring_s + s * kSlotB, tmap, xc, y >> 1, csel, b, bars_s + 8 * s);
        tma_tile_4d(ring_s + s * kSlotB + kOddBoxOff, tmap, xc + p.odd_x - kOddShiftB / 4, y >> 1, csel, b, bars_s + 8 * s);
      }
    };
    auto wait_tile = [&](u32 slot, u32 par) {
      mbar_wait(bars_s + 8 * slot, par);
      if (edge) {  // warp-uniform
        tile_fix_edges<DT>(ring_s + slot * kSlotB, x0, W, lane);
        __syncwarp();
      }
    };
    int y_next = r_begin - R;  // first image row of the next tile to issue
    if (lane == 0) {
      const int first = min(NG, groups);
      u32 sl = cur_slot;
      for (int k = 0; k < first; ++k) {
        issue(sl, y_next + kGroupRows * k);
        if (++sl == (u32)NG) sl = 0;
      }
    }
    y_next += kGroupRows * NG;
    int gfloor_seen = 0;
    bool hinted = false;
    if (kHint) {
      // Start at the channel's floor hint: kHintMarginBins below the lowest floor that kHintMinPlanes or more finished
      // planes of this channel reached.  It is a guess for this plane, applied like a plane-wide floor; the exact-select
      // kernel checks it afterwards against the plane's histogram (hint_used) and redoes the plane when it pruned too much.
      const uint2 h = __ldcg(reinterpret_cast<const uint2*>(hp.chint) + c);
      if (h.y >= (u32)kHintMinPlanes && h.x != 0u) {
        const int hb = kFineBins - (int)h.x - kHintMarginBins;
        const float hf = shared_floor<DT>(hb, xscale);
        if (hf > st.floorx) {  // warp-uniform
          st.floorx = hf;
          gfloor_seen = hb;
          hinted = true;  // a floor to work with: poll the plane's own at the usual period, not every group
          if (lane == 0) atomicMax(hp.hint_used + plane_id, hb);
        }
      }
    }
    constexpr int poll_mask = 3;  // measured at 128-row strips: polling every group 0.179 ms, every 4th 0.136 ms, every 8th 0.146 ms
    u32 idx0 = (u32)(r_begin * W + panel * kPanel);  // flat index of the group's row 0, panel column 0
    wait_tile(cur_slot, cur_par);
    for (int g = 0; g < groups_out; ++g, idx0 += (u32)(kGroupRows * W)) {
      // cur_* = the tile holding the group's first window row, nxt_* = the one after it
      u32 nxt_slot = cur_slot, nxt_par = cur_par;
      step_pos(nxt_slot, nxt_par);
      if (R == 2 || g + 1 < groups) wait_tile(nxt_slot, nxt_par);
      if (gfloor_seen <= 0 && g > 0 && !hinted) {
        // The plane has no floor that this warp knows of: every pixel it looks at goes through the slow path, so a
        // fresh look at the published floor is worth its latency (one L2 round trip) -- every group, applied at once.
        gfloor_seen = __ldcg(gfloor_ptr);
        st.floorx = fmaxf(st.floorx, shared_floor<DT>(gfloor_seen, xscale));
      } else if ((g & poll_mask) == 0) {
        // every 16 rows: apply the plane-wide floor fetched one period ago
        // and start the next fetch.  The load writes straight into the register it will be read
        // from a period later, so its latency is never waited for.
        st.floorx = fmaxf(st.floorx, shared_floor<DT>(gfloor_seen, xscale));
        asm volatile("ld.global.cg.s32 %0, [%1];" : "=r"(gfloor_seen) : "l"(gfloor_ptr) : "memory");
      }
      // window rows of group row i are ring rows row0 + i .. row0 + i + 2R; its centre row is row0 + i + R
      const u32 row0 = cur_slot * kGroupRows;
      uint4 c0, c1, c2, c3;
      if (R == 2) {  // centres: rows 2, 3 of this tile's slot and rows 0, 1 of the next
        const u32 a01 = ring_own + cur_slot * kSlotB, a23 = ring_own + nxt_slot * kSlotB;
        if (S == 1) {
          c0 = lds128u(a01 + 2 * kTilePitchB); c1 = lds128u(a01 + 3 * kTilePitchB);
          c2 = lds128u(a23); c3 = lds128u(a23 + kTilePitchB);
        } else {  // a slot holds rows 0, 2 in its first box and rows 1, 3 in its second
          c0 = lds128u(a01 + kTilePitchB); c1 = lds64x2(a01 + kOddBoxOff + kOddShiftB + kTilePitchB);
          c2 = lds128u(a23); c3 = lds64x2(a23 + kOddBoxOff + kOddShiftB);
        }
      } else {  // S == 1
        const u32 a012 = ring_own + (row0 + 1) * kTilePitchB, a3 = ring_own + nxt_slot * kGroupRows * kTilePitchB;
        c0 = lds128u(a012); c1 = lds128u(a012 + kTilePitchB); c2 = lds128u(a012 + 2 * kTilePitchB); c3 = lds128u(a3);
      }
      const u32 hot = __ballot_sync(0xffffffffu, TileMax<DT>::group(c0, c1, c2, c3) > st.floorx);
      if (hot) {
        // Something in these four rows beats the floor (`hot` = the lanes whose 4 x kPx block holds such a pixel).  In
        // the last, partial group of a unit the rows past its end belong to the next unit: they may raise this alarm
        // for nothing but are never recorded.
        // Two ways to settle the group, by how many lanes are hot:
        //   many (the first groups of a unit, before the plane has a floor worth the name): the whole maximum filter
        //   of the group once, in registers (settle_dense_f32);
        //   otherwise: list the hot 16-byte words, one ballot per row, and give every pixel of a listed word a
        //   lane (settle_entries).
        // Measured and dropped (noise / blobs, 1024 images, against 0.69 / 0.74 ms): giving every pixel of a hot lane's
        // 4-row block a lane without building the list -- more, emptier passes: 0.72 / 0.78 ms; parking the hot pixels
        // of sparse groups and testing their windows 32 at a time from global memory (L2) -- the warp stalls on the
        // scattered loads longer than the saved passes cost: 0.91 / 1.01 ms.
        // Also measured and dropped (r02, same-run pairs): settling a hot lane's 4 x 4 block by the whole warp (one LDS.64
        // per lane of the 8 x 8 window region, separable 5-maxima by shuffles: ~35 instructions against ~160 for list +
        // pass) for groups with up to 1 / 3 / 6 hot lanes: 0.706 / 0.725 / 0.734 ms against 0.691 (noise), 0.767 / 0.768 /
        // 0.819 against 0.733 (blobs) -- nine dependent shuffles are a longer chain than the pass's independent loads,
        // and a warp's pace is set by dependent latency (10 cycles per issued instruction on average at 6 warps per
        // scheduler), not by issue slots; one out-of-line copy of the flush instead of four inlined ones (the kernel is
        // 4,872 SASS instructions = 78 KB, 3,512 with the call; no_instruction stalls 0.8 cycles per instruction): 0.707 /
        // 0.750 against 0.690 / 0.734 ms, fp16 0.709 against 0.640 -- the call's register shuffling costs more than the
        // instruction fetches it saves.
        // Also measured and dropped: loading the NEXT segment's first tiles into the ring slots a segment's last groups
        // free (unit fetched from the counter three groups early): 0.704 / 0.753 ms against 0.684 / 0.729 ms in the same
        // run -- with HBM the shared limit, one warp's cold ring is bandwidth the other warps use; and one warp per CTA
        // (24 CTAs per SM, so that a finished warp's slot is refilled at once): 0.707 / 0.765 against 0.699 / 0.774 ms.
        const int nhot = __popc(hot), rows_here = nrows - g * kGroupRows;
        const float floorx = st.floorx;
        bool settled = false;
        if (DT == SDNET_DTYPE_F32 && S == 1 && nhot >= kDenseLanes)
          settled = settle_dense_f32<R>(st, rows_here, ring_s, ring_own, row0, floorx, idx0, W, pre, buf, hist, minx, sf, count_ptr,
                                        list, p.cap, K, lane, xscale, satx);
        if (!settled) {
          int nent = 0;
#pragma unroll
          for (int i = 0; i < kGroupRows; ++i) {
            const uint4 ci = i == 0 ? c0 : (i == 1 ? c1 : (i == 2 ? c2 : c3));
            const bool mine = TileMax<DT>::word(ci) > floorx && i < rows_here;
            const u32 bm = __ballot_sync(0xffffffffu, mine);
            if (mine) work[nent + __popc(bm & lt)] = (unsigned char)((i << 5) | lane);
            nent += __popc(bm);
          }
          __syncwarp();
          settle_entries<R, DT, S>(st, work, nent, ring_s, row0, row_tab, floorx, idx0, W, pre, buf, hist, minx, sf, count_ptr, list,
                                   p.cap, K, lane, xscale, satx);
        }
        // flush in batches: candidates are counted in the plane-wide histogram when they are found, so a flush is
        // not what publishes them (flushing after every group while the plane has no floor only added its latency)
        if (st.nbuf >= kFlushAt) {
          __syncwarp();
          flush_candidates<DT, false>(st, buf, hist, minx, sf, count_ptr, list, p.cap, K, lane, pre, xscale, satx);
        }
      }
      // every lane's reads of the group's first tile are done (the votes above): refill its slot
      // with the tile NG ahead
      __syncwarp();
      if (lane == 0 && g + NG < groups) {
        if (edge) fence_proxy_async();  // the slot was patched with ordinary stores
        issue(cur_slot, y_next);
      }
      y_next += kGroupRows;
      cur_slot = nxt_slot;
      cur_par = nxt_par;
    }
    for (int k = groups_out; k < groups; ++k) step_pos(cur_slot, cur_par);  // the halo tile below the last group
    if (st.nbuf) {
      __syncwarp();
      flush_candidates<DT, false>(st, buf, hist, minx, sf, count_ptr, list, p.cap, K, lane, pre, xscale, satx);
    }
    if (kHint && lane == 0 && pos <= (u32)p.tier1_units * (u32)p.groups_per_col &&
        (pos / (u32)p.groups_per_col - 1u) % (u32)p.panels == 0) {
      // a tier-1 unit (a whole column) done: its plane's floor so far -- certified by >= K recorded survivors, so a lower
      // bound of the plane's final one -- joins the channel's hint.  One report per plane: its first panel's column.
      // A plane without a floor yet says nothing: a hinted plane records few candidates and may not have K of them
      // when this column ends.  (Everything here is recomputed from what the loop keeps anyway: registers are what
      // limits the occupancy.)
      const int gf = __ldcg(gfloor_ptr);
      if (gf > 0) {
        u32* hint = hp.chint + 2 * ((int)(gfloor_ptr - p.gfloor) % C);
        atomicMax(hint, (u32)(kFineBins - gf));
        __threadfence();  // the minimum before the count: a reader that sees the count sees a minimum
        atomicAdd(hint + 1, 1u);
      }
    }
    }  // segments of the unit
  }
}


}  // namespace
