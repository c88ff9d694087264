// tail.cuh -- sdnet_tail_kernel (per-image select, sort, gather, grouping, packed stores) and sdnet_activate_kernel.
#pragma once

namespace {

// ---------------------------------------------------------------------------------------------
// tail kernel: select + sort + gather + group, one CTA per image
// ---------------------------------------------------------------------------------------------
struct TailParams {
  View4 offsets, embeddings;
  int B, M, N, H, W, K, P;
  int cap;
  int pre_activated, no_grouping;
  float conf, dist_abs;
  const float* conf_class;  // [M + N] per-class thresholds (anchor classes, then part kinds), or nullptr: conf for all
  const u64* lists;
  const int* counts;
  float* anchor_out;
  float* part_out;
  long long* anchor_inds;
  long long* part_inds;
  float* part_emb;
  int* assign;
  int* out_counts;
  int* diag;
  const int* exact_flags;  // [planes] 1 if the exact select rewrote the list
  const u32* ghist;        // [planes][kFineBins] logit histogram of the recorded candidates (peaks kernels)
  int n_dest;              // fused gather: every output is stored n_dest times, at ptr + dest_delta[j]
  int dest_multicast;      // ... or once, with multimem.st, at the multicast address ptr + dest_delta[0]
  u32* done_flag;          // fused gather: completion flag of this rank (nullptr = none), stored like an output by the last CTA
  u32 done_value;
  u32* ticket;             // workspace counter (zeroed per launch): CTAs that have finished their stores
  // the workspace header, to be left zeroed for the next decode (SDNET_FLAG_WORKSPACE_CLEAN)
  int* ws_counts;
  int* ws_flags;
  int* ws_gfloor;
  u32* ws_ghist;
  int* ws_hint_used;
  u32* ws_chint;
  u32* ws_sched;
  long long dest_delta[SDNET_MAX_DEST];
};

// Store one output value locally (n_dest == 0) or into every destination copy of the output blob
// (fused detection gather: peer-mapped symmetric memory).  Two forms: plain st.global to each peer's
// address, n_dest stores per value; or -- dest_multicast -- ONE multimem.st to the NVSwitch multicast
// address of the blob (dest_delta[0] = multicast_base - local_base), which the switch replicates into
// every GPU's copy, the local one included: 1/n_dest of the store instructions and of the NVLink egress.
__device__ __forceinline__ void mc_store(void* a, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void mc_store(void* a, const float2& v) {
  asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1, %2};" ::"l"(a), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void mc_store(void* a, const long long& v) {
  asm volatile("multimem.st.relaxed.sys.global.b64 [%0], %1;" ::"l"(a), "l"(v) : "memory");
}
__device__ __forceinline__ void mc_store(void* a, const int& v) {
  asm volatile("multimem.st.relaxed.sys.global.b32 [%0], %1;" ::"l"(a), "r"(v) : "memory");
}
template <typename T>
__device__ __forceinline__ void store_out(const TailParams& p, T* ptr, const T& v) {
  if (p.n_dest == 0) {
    *ptr = v;
  } else if (p.dest_multicast) {
    mc_store(reinterpret_cast<char*>(ptr) + p.dest_delta[0], v);
  } else {
    for (int j = 0; j < p.n_dest; ++j) *reinterpret_cast<T*>(reinterpret_cast<char*>(ptr) + p.dest_delta[j]) = v;
  }
}

__device__ __forceinline__ u64 make_comp(u64 rec, int c_local) {
  // rec = key:32 | idx:32  ->  key:32 | (255-c):8 | (0xFFFFFF-idx):24 ; larger = earlier in the output
  const u32 key = (u32)(rec >> 32);
  const u32 idx = (u32)rec;
  return ((u64)key << 32) | ((u64)(255u - (u32)c_local) << 24) | (u64)(0xFFFFFFu - idx);
}

// The tail CTA is split into two teams of kTeamThreads threads that work concurrently: team 0
// selects the anchors, team 1 the parts; each has its own sort buffer and syncs on its own named
// barrier.  They meet once, before the grouping.
constexpr int kTeamThreads = 256;
constexpr float kNearField = 1e5f;   // see the grouping pass
constexpr int kRankPerThread = 4;     // composites a thread ranks at once
constexpr int kRankSortMax = kRankPerThread * kTeamThreads;  // up to this many collected composites are sorted by counting ranks
constexpr int kHistCollectSlack = 412;  // a histogram cut-off that collects more than want + this falls back to the radix refinement

struct Team {
  int tid;    // thread index inside the team
  int id;     // 0 = anchors, 1 = parts
  __device__ __forceinline__ void sync() const {
    asm volatile("bar.sync %0, %1;" ::"r"(id + 1), "r"(kTeamThreads) : "memory");
  }
};

__device__ void bitonic_sort_desc(const Team& tm, u64* s, int n /* power of two */) {
  if (n <= kTeamThreads) {
    // one element per thread, in a register: partners less than a warp apart are exchanged by shuffle, only
    // the j >= 32 steps (6 of the 36 at n = 256) go through shared memory and the team barrier
    const int i = tm.tid;
    u64 v = i < n ? s[i] : 0ull;
    for (int k = 2; k <= n; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        u64 o;
        if (j >= 32) {
          if (i < n) s[i] = v;
          tm.sync();
          o = s[(i ^ j) & (n - 1)];
          tm.sync();
        } else {
          o = __shfl_xor_sync(0xffffffffu, v, j);
        }
        const bool keep_max = ((i & k) == 0) == ((i & j) == 0);  // lower index of a descending pair, or upper of an ascending one
        v = keep_max ? (v > o ? v : o) : (v < o ? v : o);
      }
    }
    if (i < n) s[i] = v;
    tm.sync();
    return;
  }
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tm.tid; i < n; i += kTeamThreads) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const u64 a = s[i], b = s[ixj];
          const bool desc = (i & k) == 0;
          if (desc ? (a < b) : (a > b)) { s[i] = b; s[ixj] = a; }
        }
      }
      tm.sync();
    }
  }
}

// Composite key of the lowest score a candidate counted in fine bin `bin` (or a higher one) can have.
template <int DT>
__device__ __forceinline__ u32 bin_floor_key(int bin, bool pre) {
  if (bin <= 0) return 0u;  // bin 0 is open below
  const float edge = kBinLo + (float)bin * (1.0f / kFineScale);
  if (pre) {  // the histogram ran on kPreScale * value; keys are the order-preserving bits of the value
    const u32 bits = __float_as_uint(edge / kPreScale);
    return (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
  }
  return __float_as_uint(Num<DT>::act(edge));  // the score is monotone in the logit (saturation included)
}

// Select the `want` largest composites of planes [c0, c0+nc) of image b into s_sel (sorted
// descending).  Returns the number selected (< want only when fewer candidates exist).
//
// Cut-off: the peaks kernel left, per plane, a histogram of its recorded candidates over 1/16-logit bins.
// Summed over the group's planes it names the highest bin B with >= want candidates in bins >= B: everything
// whose score reaches the score of B's lower edge is collected (a superset of those bins, normally want plus
// a few dozen) and sorted.  When that cannot be used -- a plane went through the exact select, which rewrites
// its list, or the superset is too large (heavily tied scores) -- an 8-bit radix refinement over the
// composites finds the cut-off instead.
template <int DT>
__device__ int select_group(const Team& tm, const TailParams& p, int b, int c0, int nc, int want, u64* s_sel,
                            u32* s_hist, int* s_misc) {
  const int C = p.M + p.N;
  const int tid = tm.tid;
  const bool pre = p.pre_activated != 0;
  // total candidates
  if (tid == 0) {
    int tot = 0, rewritten = 0;
    for (int c = 0; c < nc; ++c) {
      tot += min(p.counts[(size_t)b * C + c0 + c], p.cap);
      rewritten |= p.exact_flags[(size_t)b * C + c0 + c];
    }
    s_misc[0] = tot;
    s_misc[1] = 0;  // collected
    s_misc[5] = rewritten;
  }
  tm.sync();
  const int total = s_misc[0];
  u64 prefix = 0;   // value of the top `bits` bits that boundary elements share
  int bits = 0;
  u32 floor_key = 0;  // histogram cut-off: collect every composite whose 32-bit key is >= floor_key
  // what is collected (everything certainly selected + the boundary bucket) should be a small sort: the bitonic
  // network costs O(n log^2 n)
  const int target = min(kSortN, max(want + 64, 128));
  bool by_hist = total > target && p.ghist != nullptr && s_misc[5] == 0;
  for (int attempt = 0; attempt < 2; ++attempt) {
    if (by_hist) {
      for (int bin = tid; bin < kFineBins; bin += kTeamThreads) {
        const u32* col = p.ghist + ((size_t)b * C + c0) * kFineBins + bin;
        u32 sum = 0;
        int c = 0;
        for (; c + 4 <= nc; c += 4) {  // four planes' loads in flight (20 planes at cfg4: one L2 round trip each otherwise)
          const u32 h0 = __ldcg(col + (size_t)c * kFineBins), h1 = __ldcg(col + (size_t)(c + 1) * kFineBins),
                    h2 = __ldcg(col + (size_t)(c + 2) * kFineBins), h3 = __ldcg(col + (size_t)(c + 3) * kFineBins);
          sum += (h0 + h1) + (h2 + h3);
        }
        for (; c < nc; ++c) sum += __ldcg(col + (size_t)c * kFineBins);
        s_hist[bin] = sum;
      }
      tm.sync();
      if (tid < 32) {
        const int fb = floor_bin_fine<true>(s_hist, tid, want);  // highest bin with >= want candidates at or above it; -1: none
        if (tid == 0) s_misc[2] = fb;
      }
      tm.sync();
      floor_key = s_misc[2] > 0 ? bin_floor_key<DT>(s_misc[2], pre) : 0u;
      tm.sync();
    } else if (total > target) {
      int need = want;      // how many still have to come from the boundary bucket
      int certain = 0;      // elements strictly above the boundary bucket
      for (int level = 0; level < 8; ++level) {
        const int shift = 56 - 8 * level;
        for (int i = tid; i < 256; i += kTeamThreads) s_hist[i] = 0;
        tm.sync();
        for (int c = 0; c < nc; ++c) {
          const int n = min(p.counts[(size_t)b * C + c0 + c], p.cap);
          const u64* list = p.lists + ((size_t)b * C + c0 + c) * p.cap;
          for (int i = tid; i < n; i += kTeamThreads) {
            const u64 v = make_comp(list[i], c);
            if (bits == 0 || (v >> (64 - bits)) == prefix) atomicAdd(&s_hist[(u32)(v >> shift) & 0xffu], 1u);
          }
        }
        tm.sync();
        if (tid < 32) {
          // lane l owns digits 8l..8l+7; suffix-scan from the top
          u32 loc[8], sum = 0;
#pragma unroll
          for (int q = 0; q < 8; ++q) { loc[q] = s_hist[8 * tid + q]; sum += loc[q]; }
          u32 suf = sum;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            u32 t = __shfl_down_sync(0xffffffffu, suf, d);
            if (tid + d < 32) suf += t;
          }
          const u32 mask = __ballot_sync(0xffffffffu, suf >= (u32)need);
          const int L = 31 - __clz(mask);  // mask != 0 because the bucket holds >= need elements
          if (tid == L) {
            u32 above = suf - sum;
            int dsel = 8 * L;
            for (int q = 7; q >= 0; --q) {
              if (above + loc[q] >= (u32)need) { dsel = 8 * L + q; break; }
              above += loc[q];
            }
            s_misc[2] = dsel;
            s_misc[3] = (int)above;                 // elements in this bucket with a larger digit
            s_misc[4] = (int)s_hist[dsel];          // size of the new boundary bucket
          }
        }
        tm.sync();
        const int dsel = s_misc[2], above = s_misc[3], binc = s_misc[4];
        certain += above;
        need -= above;
        prefix = (prefix << 8) | (u64)dsel;
        bits += 8;
        tm.sync();
        if (certain + binc <= target) break;  // everything at or above the boundary bucket is a small sort
      }
    }
    // collect: the composites at or above the cut-off
    for (int c = 0; c < nc; ++c) {
      const int n = min(p.counts[(size_t)b * C + c0 + c], p.cap);
      const u64* list = p.lists + ((size_t)b * C + c0 + c) * p.cap;
      for (int i0 = tid; i0 < n; i0 += 4 * kTeamThreads) {  // four records per thread in flight: the pass is L2-latency-bound
        u64 rec[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int i = i0 + e * kTeamThreads;
          rec[e] = i < n ? __ldcg(list + i) : 0ull;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const u64 v = make_comp(rec[e], c);
          if (i0 + e * kTeamThreads < n && (u32)(v >> 32) >= floor_key && (bits == 0 || (v >> (64 - bits)) >= prefix)) {
            const int slot = atomicAdd(&s_misc[1], 1);
            if (slot < kSortN) s_sel[slot] = v;
          }
        }
      }
    }
    tm.sync();
    if (!by_hist || s_misc[1] <= min(kSortN, want + kHistCollectSlack)) break;
    // the histogram's superset is too large to sort cheaply (heavily tied scores): refine by radix instead
    tm.sync();
    if (tid == 0) s_misc[1] = 0;
    by_hist = false;
    floor_key = 0;
    tm.sync();
  }
  const int got = min(s_misc[1], kSortN);
  if (got <= kRankSortMax) {
    // The usual case (want plus a few dozen; a few hundred more at K = 500): every thread ranks its own composites -- up
    // to four of them -- by counting the larger ones: got broadcast reads per thread, no barrier in the loop;
    // composites are pairwise distinct (they end in the pixel index and the class), so the ranks are a permutation.
    u64 mine[kRankPerThread];
    int rank[kRankPerThread];
#pragma unroll
    for (int e = 0; e < kRankPerThread; ++e) {
      const int i = tid + e * kTeamThreads;
      mine[e] = i < got ? s_sel[i] : 0ull;
      rank[e] = 0;
    }
    if (got <= kTeamThreads) {  // one composite per thread: the short loop
      if (tid < got)
        for (int j = 0; j < got; ++j) rank[0] += s_sel[j] > mine[0] ? 1 : 0;
    } else {
      for (int j = 0; j < got; ++j) {
        const u64 o = s_sel[j];
#pragma unroll
        for (int e = 0; e < kRankPerThread; ++e) rank[e] += o > mine[e] ? 1 : 0;
      }
    }
    tm.sync();
#pragma unroll
    for (int e = 0; e < kRankPerThread; ++e)
      if (tid + e * kTeamThreads < got) s_sel[rank[e]] = mine[e];
    tm.sync();
    return min(got, want);
  }
  int n2 = 32;
  while (n2 < got) n2 <<= 1;
  for (int i = got + tid; i < n2; i += kTeamThreads) s_sel[i] = 0;
  tm.sync();
  bitonic_sort_desc(tm, s_sel, n2);
  return min(got, want);
}

// Slots [have, want) of a group are the zero-valued entries torch.topk pads with: under
// (value desc, index asc) they are the lowest-index pixels of the group's first plane that
// did not survive NMS.  All of them lie below index `want`.
__device__ void zero_fill(const Team& tm, const TailParams& p, int b, int c0, int have, int want, u64* s_sel,
                          u32* s_bits) {
  const int C = p.M + p.N;
  const int tid = tm.tid;
  const int words = (want + 31) / 32;
  for (int i = tid; i < words; i += kTeamThreads) s_bits[i] = 0;
  tm.sync();
  const int n = min(p.counts[(size_t)b * C + c0], p.cap);
  const u64* list = p.lists + ((size_t)b * C + c0) * p.cap;
  for (int i = tid; i < n; i += kTeamThreads) {
    const u32 idx = (u32)list[i];
    if (idx < (u32)want) atomicOr(&s_bits[idx >> 5], 1u << (idx & 31));
  }
  tm.sync();
  for (int s = have + tid; s < want; s += kTeamThreads) {
    int rank = s - have;  // rank-th non-peak index
    int w = 0;
    for (; w < words; ++w) {
      const int z = 32 - __popc(s_bits[w]);
      if (rank < z) break;
      rank -= z;
    }
    const u32 free_mask = ~s_bits[w];
    const u32 bit = __fns(free_mask, 0, rank + 1);
    const u32 idx = (u32)(w * 32) + bit;
    // key 0 (score 0.0), class 0
    s_sel[s] = ((u64)255u << 24) | (u64)(0xFFFFFFu - idx);
  }
  tm.sync();
}

__device__ __forceinline__ float key_to_score(u32 key, bool pre) {
  if (!pre) return __uint_as_float(key);
  const u32 bits = (key == 0) ? 0u : ((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key);
  return __uint_as_float(bits);
}

// (A thin variant -- teams of 128 threads, sort buffers in dynamic shared memory sized by K and P: 256 threads x 40
// registers, 14 KB, the footprint of one peaks CTA -- measured the same with several decodes in flight (0.1094 against
// 0.1101 ms per 128-image step, 0.779 against 0.779 at 1024) and 30 % slower alone; launching the chain without
// programmatic dependent launch changes nothing either.)
template <int DT>
__global__ void __launch_bounds__(2 * kTeamThreads, 3) sdnet_tail_kernel(const __grid_constant__ TailParams p) {
  __shared__ u64 s_sel[2][kSortN];
  __shared__ __align__(16) u32 s_hist[2][kFineBins];
  __shared__ int s_misc[2][8];
  __shared__ float s_ax[SDNET_MAX_TOPK], s_ay[SDNET_MAX_TOPK];
  __shared__ int s_cnt[2];
  __shared__ int s_end[2];  // last valid anchor / part slot + 1
  __shared__ int s_far;  // a valid anchor or part origin lies outside +-kNearField: grouping must look at the masked slots too
  const int b = blockIdx.x;
  Team tm;
  tm.id = threadIdx.x / kTeamThreads;
  tm.tid = threadIdx.x % kTeamThreads;
  const int W = p.W;
  const bool pre = p.pre_activated != 0;
  if (threadIdx.x < 2) s_cnt[threadIdx.x] = s_end[threadIdx.x] = 0;
  if (threadIdx.x == 2) s_far = 0;
  pdl_wait();  // candidate lists (peaks kernel, possibly rewritten by the exact select) are final
  __syncthreads();
  typedef typename Num<DT>::In In;
  const In* offx = static_cast<const In*>(p.offsets.data) + (long long)b * p.offsets.sb;
  const In* offy = offx + p.offsets.sc;
  const long long osh = p.offsets.sh;
  u64* sel = s_sel[tm.id];

  if (tm.id == 0) {
    // ---- anchors
    const int have = select_group<DT>(tm, p, b, 0, p.M, p.K, sel, s_hist[0], s_misc[0]);
    if (have < p.K) zero_fill(tm, p, b, 0, have, p.K, sel, s_hist[0]);
    int n_valid = 0, end = 0;
    for (int s = tm.tid; s < p.K; s += kTeamThreads) {
      const u64 v = sel[s];
      const int cls = 255 - (int)((v >> 24) & 0xffu);
      const u32 idx = 0xFFFFFFu - (u32)(v & 0xFFFFFFu);
      const int yy = idx / W, xx = idx - yy * W;
      const float score = key_to_score((u32)(v >> 32), pre);
      const float x = __fadd_rn((float)xx, Num<DT>::to_float(__ldg(offx + (long long)yy * osh + xx)));
      const float y = __fadd_rn((float)yy, Num<DT>::to_float(__ldg(offy + (long long)yy * osh + xx)));
      store_out(p, reinterpret_cast<float4*>(p.anchor_out) + (size_t)b * p.K + s, make_float4(x, y, score, (float)cls));
      store_out(p, p.anchor_inds + (size_t)b * p.K + s, (long long)idx);
      const bool valid = score > (p.conf_class ? __ldg(p.conf_class + cls) : p.conf);
      // masked anchors sit at (+1e6, +1e6): decoders.py:85-86
      s_ax[s] = valid ? x : kFar;
      s_ay[s] = valid ? y : kFar;
      n_valid += valid ? 1 : 0;
      end = valid ? s + 1 : end;
      if (valid && !(fabsf(x) < kNearField && fabsf(y) < kNearField)) s_far = 1;
    }
    if (n_valid) {
      atomicAdd(&s_cnt[0], n_valid);
      atomicMax(&s_end[0], end);
    }
  } else {
    // ---- parts
    const int have = select_group<DT>(tm, p, b, p.M, p.N, p.P, sel, s_hist[1], s_misc[1]);
    if (have < p.P) zero_fill(tm, p, b, p.M, have, p.P, sel, s_hist[1]);
    const In* embx = p.embeddings.data ? static_cast<const In*>(p.embeddings.data) + (long long)b * p.embeddings.sb : nullptr;
    const In* emby = embx ? embx + p.embeddings.sc : nullptr;
    const long long esh = p.embeddings.sh;
    int n_valid = 0, end = 0;
    for (int s = tm.tid; s < p.P; s += kTeamThreads) {
      const u64 v = sel[s];
      const int cls = 255 - (int)((v >> 24) & 0xffu);
      const u32 idx = 0xFFFFFFu - (u32)(v & 0xFFFFFFu);
      const int yy = idx / W, xx = idx - yy * W;
      const float score = key_to_score((u32)(v >> 32), pre);
      const float x = __fadd_rn((float)xx, Num<DT>::to_float(__ldg(offx + (long long)yy * osh + xx)));
      const float y = __fadd_rn((float)yy, Num<DT>::to_float(__ldg(offy + (long long)yy * osh + xx)));
      float ex = 0.f, ey = 0.f;
      if (embx) {
        ex = Num<DT>::to_float(__ldg(embx + (long long)yy * esh + xx));
        ey = Num<DT>::to_float(__ldg(emby + (long long)yy * esh + xx));
      }
      const float ox = __fadd_rn(x, ex), oy = __fadd_rn(y, ey);
      float2* po = reinterpret_cast<float2*>(p.part_out + ((size_t)b * p.P + s) * 6);
      store_out(p, po + 0, make_float2(x, y));
      store_out(p, po + 1, make_float2(score, (float)cls));
      store_out(p, po + 2, make_float2(ox, oy));
      store_out(p, p.part_inds + (size_t)b * p.P + s, (long long)idx);
      if (p.part_emb) store_out(p, reinterpret_cast<float2*>(p.part_emb) + (size_t)b * p.P + s, make_float2(ex, ey));
      const bool valid = score > (p.conf_class ? __ldg(p.conf_class + p.M + cls) : p.conf);
      n_valid += valid ? 1 : 0;
      end = valid ? s + 1 : end;
      if (valid && !(fabsf(ox) < kNearField && fabsf(oy) < kNearField)) s_far = 1;
      // masked parts sit at (-1e6, -1e6): decoders.py:80-81.  The slot's composite is no longer
      // needed: keep the part's origin there for the grouping pass.
      reinterpret_cast<float2*>(sel)[s] = make_float2(valid ? ox : -kFar, valid ? oy : -kFar);
    }
    if (n_valid) {
      atomicAdd(&s_cnt[1], n_valid);
      atomicMax(&s_end[1], end);
    }
  }
  __syncthreads();

  // ---- grouping: every part to its nearest anchor (first minimum), gated by the distance threshold
  // (reference: hypot utils.py:422-437, min(dim=1) decoders.py:99).  A part is shared by g lanes of one
  // warp, lane `sub` taking anchors sub, sub + g, ...  The square root is monotone, so the smallest
  // distance is the root of the smallest squared distance m2 -- but two different squares can round to
  // the same root and the reference's min() then keeps the FIRST anchor.  Hence two sweeps without a
  // root in the loop: m2, then the first anchor whose square lies within 1e-6 of m2 (a root can only
  // tie if its square is within 2^-22 relative) AND whose root equals root(m2).
  // Masked slots sit 1e6 away (decoders.py:80-86); as long as every valid coordinate is within kNearField = 1e5 and the
  // gate is below 1e5, no pair with a masked member can pass the gate or tie with one that does, so only the slots up
  // to the last valid anchor / part are searched (13 x 36 instead of 100 x 100 on the realistic maps).  With one
  // threshold those are exactly the valid slots (slots are in score order); with per-class thresholds masked slots can
  // sit among them, at the 1e6 guard, where they cannot win.  Otherwise: the full P x K search.
  const float2* origin = reinterpret_cast<const float2*>(s_sel[1]);
  const bool full = s_far != 0 || !(p.dist_abs < kNearField);
  const int Ka = full ? p.K : s_end[0], Pp = full ? p.P : s_end[1];
  int g = 32;
  while (g > 1 && Pp * g > (int)blockDim.x) g >>= 1;
  const int sub = threadIdx.x & (g - 1), per_pass = blockDim.x / g;
  for (int s0 = 0; s0 < p.P; s0 += per_pass) {  // block-uniform
    const int s = s0 + (int)threadIdx.x / g;
    const bool live = s < p.P;
    int slot = -1;
    if (!p.no_grouping && s0 < Pp) {  // block-uniform
      const bool search = s < Pp;
      const float qx = search ? origin[s].x : 0.f, qy = search ? origin[s].y : 0.f;
      float m2 = CUDART_INF_F;
      for (int a = sub; a < Ka; a += g) {
        const float dx = __fsub_rn(qx, s_ax[a]), dy = __fsub_rn(qy, s_ay[a]);
        m2 = fminf(m2, __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
      }
      for (int w = g >> 1; w > 0; w >>= 1) m2 = fminf(m2, __shfl_xor_sync(0xffffffffu, m2, w));
      const float best = __fsqrt_rn(m2), near = m2 * 1.000001f;
      int arg = 0x7fffffff;
      for (int a = sub; a < Ka; a += g) {
        const float dx = __fsub_rn(qx, s_ax[a]), dy = __fsub_rn(qy, s_ay[a]);
        const float sq = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
        if (sq <= near && __fsqrt_rn(sq) == best) { arg = a; break; }
      }
      for (int w = g >> 1; w > 0; w >>= 1) arg = min(arg, __shfl_xor_sync(0xffffffffu, arg, w));
      slot = (search && best < p.dist_abs) ? arg : -1;
    }
    if (live && sub == 0) store_out(p, p.assign + (size_t)b * p.P + s, slot);
  }
  if (threadIdx.x < 2) store_out(p, p.out_counts + (size_t)b * 2 + threadIdx.x, s_cnt[threadIdx.x]);
  if (p.diag) {
    const int C = p.M + p.N;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      store_out(p, p.diag + ((size_t)b * C + c) * 2 + 0, p.counts[(size_t)b * C + c]);
      store_out(p, p.diag + ((size_t)b * C + c) * 2 + 1, p.exact_flags[(size_t)b * C + c]);
    }
  }
  // Leave the workspace header as a fresh memset would: this image's planes (counts, flags, floors, histograms, applied
  // hints -- all consumed above) and, once, the channels' floor hints and the unit counter (the peaks kernel is long
  // complete: pdl_wait).
  __syncthreads();
  {
    const int C = p.M + p.N;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      p.ws_counts[(size_t)b * C + c] = 0;
      p.ws_flags[(size_t)b * C + c] = 0;
      p.ws_gfloor[(size_t)b * C + c] = 0;
      p.ws_hint_used[(size_t)b * C + c] = 0;
    }
    if (b == 0)
      for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) p.ws_chint[i] = 0;
    uint4* gh = reinterpret_cast<uint4*>(p.ws_ghist + (size_t)b * C * kFineBins);
    for (int i = threadIdx.x; i < C * kFineBins / 4; i += blockDim.x) gh[i] = make_uint4(0, 0, 0, 0);
    if (b == 0 && threadIdx.x == 0) p.ws_sched[0] = 0;
  }
  if (p.n_dest) {
    if (p.done_flag == nullptr) {
      __threadfence_system();  // peer stores performed before the kernel retires (a barrier follows on the stream)
    } else {
      // Completion flag: every thread's stores are ordered before the CTA barrier, thread 0's system fence after it is
      // cumulative over them, then the CTA takes a ticket; the CTA that takes the last one knows every other CTA has
      // fenced, fences once more (acquire side of the ticket chain) and releases the flag into every copy.
      __syncthreads();
      if (threadIdx.x == 0) {
        __threadfence_system();
        if (atomicAdd(p.ticket, 1u) == gridDim.x - 1) {
          *p.ticket = 0;  // for the next decode
          __threadfence_system();
          if (p.dest_multicast) {
            asm volatile("multimem.st.release.sys.global.u32 [%0], %1;" ::"l"(reinterpret_cast<char*>(p.done_flag) + p.dest_delta[0]), "r"(p.done_value) : "memory");
          } else {
            for (int j = 0; j < p.n_dest; ++j)
              asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(reinterpret_cast<char*>(p.done_flag) + p.dest_delta[j]), "r"(p.done_value) : "memory");
          }
        }
      }
    }
  }
}

// The consumer side: wait until every rank's completion flag has reached `value`.
__global__ void sdnet_gather_wait_kernel(const u32* flags, int world, u32 value) {
  const int j = threadIdx.x;
  if (j < world) {
    u32 v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + j) : "memory");
    } while ((int)(v - value) < 0);  // wrap-safe "v < value"
  }
}

// ---------------------------------------------------------------------------------------------
// metadata: clamped-sigmoid maps
// ---------------------------------------------------------------------------------------------
template <int DT>
__global__ void sdnet_activate_kernel(View4 in, int C, int H, int W, size_t total, float* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(i % W);
    size_t t = i / W;
    const int y = (int)(t % H);
    t /= H;
    const int c = (int)(t % C);
    const long long b = (long long)(t / C);
    out[i] = Num<DT>::act(ld_in<DT>(in.data, b * in.sb + (long long)c * in.sc + (long long)y * in.sh + x));
  }
}


}  // namespace
