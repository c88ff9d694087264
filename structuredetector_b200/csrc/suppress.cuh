// suppress.cuh -- sdnet_suppress_kernel: dense sigmoid + peak-NMS maps, the reference's RawDecoder
// (src/sdnet/cli/convert_coreml.py:12-19: nms(clamped_sigmoid(x)), src/sdnet/utils/utils.py:355-361,441-443),
// i.e. the pre-activated heat maps CoreMLDecoder consumes (src/sdnet/data/decoders.py:211,226).
#pragma once

namespace {

// out = S(x) where S(x) equals the maximum of S over the (2R+1)^2 window (-inf padding), else 0.
// S is monotone, so the window maximum is taken on raw logits and the exact score is evaluated only for
// survivors and for pixels within the near-tie margins of Num<DT> -- the same classification as the peaks
// kernels.  HBM-bound: one read of the logits, one write of the maps, nothing staged in shared memory:
// a warp walks a 128-column panel of one plane strip top to bottom, each lane holding four columns; the
// horizontal maxima come from the neighbours' registers by shuffle (panel-edge columns from two extra
// loads), the vertical ones from a register window of the last 2R+1 rows; rows are loaded two ahead.
// rows in flight per warp / CTAs per SM, measured on 256 cfg5 images (fp32): 2/3 0.596 ms, 3/3 0.615, 4/3 0.648,
// 2/4 0.582 (64 registers, spills), 4/2 0.774
constexpr int kSupWarps = 8, kSupStripRows = 64, kSupAhead = 2;

template <int DT>
__device__ __forceinline__ float4 sup_load4(const void* base, long long row_off, int x, int W, bool row_ok, bool vec_ok) {
  float4 v = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);  // max_pool2d pads with -inf
  if (!row_ok || x >= W) return v;
  if (DT == SDNET_DTYPE_F32 && vec_ok && x + 3 < W) return __ldg(reinterpret_cast<const float4*>(static_cast<const float*>(base) + row_off + x));
  v.x = ld_in<DT>(base, row_off + x);
  if (x + 1 < W) v.y = ld_in<DT>(base, row_off + x + 1);
  if (x + 2 < W) v.z = ld_in<DT>(base, row_off + x + 2);
  if (x + 3 < W) v.w = ld_in<DT>(base, row_off + x + 3);
  return v;
}

template <int DT>
__device__ __forceinline__ float sup_score(float x, float h) {
  if (x == h) return Num<DT>::act(x);
  if (may_tie<DT>(x, h)) {
    const float sx = Num<DT>::act(x);
    if (sx == Num<DT>::act(h)) return sx;
  }
  return 0.0f;
}

template <int R, int DT>
__global__ void __launch_bounds__(kSupWarps * 32, 3) sdnet_suppress_kernel(View4 in, int C, int H, int W, int panels, int strips,
                                                                         long long units, View4 outv) {
  constexpr int kWin = 2 * R + 1;
  const int lane = threadIdx.x & 31;
  const long long unit = (long long)blockIdx.x * kSupWarps + (threadIdx.x >> 5);
  if (unit >= units) return;
  const int panel = (int)(unit % panels);
  long long t = unit / panels;
  const int strip = (int)(t % strips);
  t /= strips;
  const int c = (int)(t % C);
  const long long b = t / C;
  const long long plane = b * in.sb + (long long)c * in.sc;
  const int x = panel * kPanelW + 4 * lane;
  const int r_begin = strip * kSupStripRows, r_end = min(H, r_begin + kSupStripRows);
  // fp32: a lane's four columns in one 16-byte load when base and pitches allow (an 8-byte load of four
  // fp16/bf16 elements measured slower than four 2-byte loads here: 0.89 vs 0.76 ms)
  const bool vec_ok = DT == SDNET_DTYPE_F32 && ((reinterpret_cast<uintptr_t>(in.data) | (uintptr_t)(in.sb * 4) | (uintptr_t)(in.sc * 4) |
                                                  (uintptr_t)(in.sh * 4)) & 15) == 0;
  float* out_plane = static_cast<float*>(const_cast<void*>(outv.data)) + b * outv.sb + (long long)c * outv.sc;
  const bool out_vec = (W & 3) == 0 && ((reinterpret_cast<uintptr_t>(outv.data) | (uintptr_t)(outv.sb * 4) | (uintptr_t)(outv.sc * 4) |
                                        (uintptr_t)(outv.sh * 4)) & 15) == 0;
  // halo columns of the panel: lane 0 fetches the R columns left of it, lane 31 the R columns right
  const int hx = lane == 0 ? x - R : x + 4;
  const bool halo_lane = lane == 0 || lane == 31;

  float4 hwin[kWin];  // horizontal maxima of the last 2R+1 rows, hwin[kWin-1] the newest
  float4 cwin[R + 1]; // centre values of the last R+1 rows, cwin[R] the newest
#pragma unroll
  for (int i = 0; i < kWin; ++i) hwin[i] = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
#pragma unroll
  for (int i = 0; i <= R; ++i) cwin[i] = hwin[0];

  auto fetch = [&](int y, float4& v, float& h0, float& h1) {
    const bool ok = y >= 0 && y < H;
    const long long off = plane + (long long)y * in.sh;
    v = sup_load4<DT>(in.data, off, x, W, ok, vec_ok);
    h0 = h1 = -CUDART_INF_F;
    if (halo_lane && ok) {
      if (hx >= 0 && hx < W) h0 = ld_in<DT>(in.data, off + hx);
      if (R == 2 && hx + 1 >= 0 && hx + 1 < W) h1 = ld_in<DT>(in.data, off + hx + 1);
    }
  };
  // kSupAhead rows in flight
  float4 pv[kSupAhead];
  float ph0[kSupAhead], ph1[kSupAhead];
#pragma unroll
  for (int k = 0; k < kSupAhead; ++k) fetch(r_begin - R + k, pv[k], ph0[k], ph1[k]);
  for (int y = r_begin - R; y < r_end + R; ++y) {
    const float4 v = pv[0];
    const float e_h0 = ph0[0], e_h1 = ph1[0];
#pragma unroll
    for (int k = 0; k + 1 < kSupAhead; ++k) { pv[k] = pv[k + 1]; ph0[k] = ph0[k + 1]; ph1[k] = ph1[k + 1]; }
    fetch(y + kSupAhead, pv[kSupAhead - 1], ph0[kSupAhead - 1], ph1[kSupAhead - 1]);
    // neighbours' columns: e = [l0 l1 | v.x v.y v.z v.w | r0 r1] (R = 2), [l1 | v | r0] (R = 1)
    float l0 = __shfl_up_sync(0xffffffffu, v.z, 1), l1 = __shfl_up_sync(0xffffffffu, v.w, 1);
    float r0 = __shfl_down_sync(0xffffffffu, v.x, 1), r1 = __shfl_down_sync(0xffffffffu, v.y, 1);
    if (lane == 0) { l0 = R == 2 ? e_h0 : -CUDART_INF_F; l1 = R == 2 ? e_h1 : e_h0; }
    if (lane == 31) { r0 = e_h0; r1 = R == 2 ? e_h1 : -CUDART_INF_F; }
    float4 hm;
    if (R == 2) {
      const float c12 = fmaxf(l1, v.x), c34 = fmaxf(v.y, v.z), c56 = fmaxf(v.w, r0);
      hm = make_float4(max3(l0, c12, c34), max3(c12, c34, v.w), max3(v.x, c34, c56), max3(c34, c56, r1));
    } else {
      hm = make_float4(max3(l1, v.x, v.y), max3(v.x, v.y, v.z), max3(v.y, v.z, v.w), max3(v.z, v.w, r0));
    }
#pragma unroll
    for (int i = 0; i + 1 < kWin; ++i) hwin[i] = hwin[i + 1];
    hwin[kWin - 1] = hm;
#pragma unroll
    for (int i = 0; i < R; ++i) cwin[i] = cwin[i + 1];
    cwin[R] = v;
    const int yo = y - R;  // the row whose window is now complete
    if (yo >= r_begin && x < W) {
      float4 h = hwin[0];
#pragma unroll
      for (int i = 1; i < kWin; ++i) {
        h.x = fmaxf(h.x, hwin[i].x); h.y = fmaxf(h.y, hwin[i].y); h.z = fmaxf(h.z, hwin[i].z); h.w = fmaxf(h.w, hwin[i].w);
      }
      const float4 ctr = cwin[0];
      const float4 s = make_float4(sup_score<DT>(ctr.x, h.x), sup_score<DT>(ctr.y, h.y), sup_score<DT>(ctr.z, h.z), sup_score<DT>(ctr.w, h.w));
      float* dst = out_plane + (long long)yo * outv.sh + x;
      if (out_vec) {
        *reinterpret_cast<float4*>(dst) = s;
      } else {
        dst[0] = s.x;
        if (x + 1 < W) dst[1] = s.y;
        if (x + 2 < W) dst[2] = s.z;
        if (x + 3 < W) dst[3] = s.w;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// TMA-tile form (fp32 maps whose base and pitches TMA can describe): the peaks kernel's feed -- autonomous warps,
// private ring of 4-row tiles pulled by tensor-map bulk copies, NaN out-of-bounds fill standing in for max_pool2d's
// -inf padding -- with the dense maximum filter of peaks_tile.cuh run on EVERY group.  Two to three tiles per warp
// are in flight (the register-window kernel above keeps two ROWS), which is what an HBM-bound pass needs.
// Output: each lane zero-fills its 16-byte word of the group's four rows with full-width vector stores, then
// overwrites the few pixels that survive with their score (same thread, same address: program order).
// Units are the peaks kernel's (whole columns, then balanced chunks), dealt round-robin: every group costs the same
// here, so no atomic counter -- and no workspace -- is needed.
// ---------------------------------------------------------------------------------------------
constexpr int kSupTileSmemPerWarp = (kTileNG * kTileBytes + 32 + 127) / 128 * 128;
constexpr int kSupTileSmem = kTileWarps * kSupTileSmemPerWarp;

template <int R>
__global__ void __launch_bounds__(kTileWarps * 32, 24 / kTileWarps)
sdnet_suppress_tile_kernel(const __grid_constant__ PeaksParams p, const __grid_constant__ CUtensorMap tm, const View4 outv) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int NG = kTileNG;
  constexpr u32 kRingRows = NG * kGroupRows;
  constexpr int DT = SDNET_DTYPE_F32;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  unsigned char* wbase = smem_raw + (size_t)warp * kSupTileSmemPerWarp;
  const u32 ring_s = smem_u32(wbase);
  const u32 bars_s = ring_s + NG * kTileBytes;
  const int C = p.M + p.N;
  const int H = p.H, W = p.W;
  const u32 ring_own = ring_s + (u32)(16 + 16 * lane);
  if (lane == 0) {
    for (int i = 0; i < NG; ++i) mbar_init(bars_s + 8 * i, 1);
    mbar_fence_init();
  }
  __syncwarp();
  u32 cur_slot = 0, cur_par = 0;
  auto step_pos = [&](u32& slot, u32& par) {
    if (++slot == (u32)NG) { slot = 0; par ^= 1u; }
  };
  for (u32 unit = blockIdx.x * kTileWarps + warp; unit < (u32)p.units; unit += gridDim.x * kTileWarps) {
    u32 pos, pos_end;
    if (unit < (u32)p.tier1_units) {
      pos = unit * (u32)p.groups_per_col;
      pos_end = pos + (u32)p.groups_per_col;
    } else {
      pos = (u32)p.tier1_units * (u32)p.groups_per_col + (unit - (u32)p.tier1_units) * (u32)p.chunk_groups;
      pos_end = min(p.total_groups, pos + (u32)p.chunk_groups);
    }
    while (pos < pos_end) {  // warp-uniform: one column segment at a time
      const u32 column = pos / (u32)p.groups_per_col;
      const int g_first = (int)(pos - column * (u32)p.groups_per_col);
      const int g_last = min(p.groups_per_col, g_first + (int)(pos_end - pos));
      pos += (u32)(g_last - g_first);
      const int panel = (int)(column % (u32)p.panels), plane_id = (int)(column / (u32)p.panels);
      const int r_begin = g_first * kGroupRows, r_end = min(H, g_last * kGroupRows);
      const int b = plane_id / C, c = plane_id % C;
      const int x0 = panel * kPanelW - 4;
      const int nrows = r_end - r_begin;
      const int groups = (nrows + 2 * R + kGroupRows - 1) / kGroupRows;
      const int groups_out = (nrows + kGroupRows - 1) / kGroupRows;
      const int col0 = panel * kPanelW + 4 * lane;
      const size_t orow = (size_t)outv.sh;  // output row pitch in elements (a multiple of 4: checked on the host)
      float* out_row = static_cast<float*>(const_cast<void*>(outv.data)) + (size_t)b * outv.sb + (size_t)c * outv.sc +
                       (size_t)r_begin * orow + col0;
      __syncwarp();  // everyone is done with the previous segment's ring
      auto issue = [&](u32 s, int y) {
        mbar_arrive_expect_tx(bars_s + 8 * s, kTileBytes);
        tma_tile_4d(ring_s + s * kTileBytes, &tm, x0, y, c, b, bars_s + 8 * s);
      };
      int y_next = r_begin - R;
      if (lane == 0) {
        const int first = min(NG, groups);
        u32 sl = cur_slot;
        for (int k = 0; k < first; ++k) {
          issue(sl, y_next + kGroupRows * k);
          if (++sl == (u32)NG) sl = 0;
        }
      }
      y_next += kGroupRows * NG;
      mbar_wait(bars_s + 8 * cur_slot, cur_par);
      for (int g = 0; g < groups_out; ++g, out_row += (size_t)kGroupRows * orow) {
        u32 nxt_slot = cur_slot, nxt_par = cur_par;
        step_pos(nxt_slot, nxt_par);
        if (R == 2 || g + 1 < groups) mbar_wait(bars_s + 8 * nxt_slot, nxt_par);
        const u32 row0 = cur_slot * kGroupRows;
        const int rows_here = nrows - g * kGroupRows;
        u32 km = dense_keep_mask_f32<R>(rows_here, ring_s, ring_own, row0, -CUDART_INF_F, false, lane);
        if (col0 < W) {  // W is a multiple of 4: the whole word is inside the image
#pragma unroll
          for (int i = 0; i < kGroupRows; ++i)
            if (i < rows_here) *reinterpret_cast<float4*>(out_row + (size_t)i * orow) = make_float4(0.f, 0.f, 0.f, 0.f);
          while (km) {
            const int bit = __ffs(km) - 1;
            km &= km - 1;
            const u32 i = (u32)bit >> 2, cc = (u32)bit & 3u;
            u32 rr = row0 + R + i;
            if (rr >= kRingRows) rr -= kRingRows;
            const float x = TileMax<DT>::elem(ring_own + rr * kTilePitchB + 4 * cc);
            out_row[(size_t)i * orow + cc] = Num<DT>::act(x);
          }
        }
        __syncwarp();
        if (lane == 0 && g + NG < groups) issue(cur_slot, y_next);
        y_next += kGroupRows;
        cur_slot = nxt_slot;
        cur_par = nxt_par;
      }
      for (int k = groups_out; k < groups; ++k) step_pos(cur_slot, cur_par);
    }
  }
}

}  // namespace
