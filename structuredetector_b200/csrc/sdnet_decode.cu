// sdnet_decode.cu -- B200 (sm_100a) kernels + C ABI for the SDNet decoding path.
//
// Replaces the tensor half of the reference decoder
//   src/sdnet/data/decoders.py:44-100  (Decoder.__call__)
//   src/sdnet/utils/utils.py:355-361   clamped_sigmoid
//   src/sdnet/utils/utils.py:441-443   nms (5x5 max-pool equality)
//   src/sdnet/utils/utils.py:447-467   topk (per-channel, then cross-channel)
//   src/sdnet/utils/utils.py:347-351   transpose_and_gather
//   src/sdnet/utils/utils.py:422-437   hypot
// with three launches (kernels in the .cuh files next to this one, host side and C ABI below):
//   1. peaks kernel (peaks_tile.cuh; peaks_warp.cuh for shapes TMA cannot describe) -- the only pass over
//      the heat maps (HBM-bound).  One warp walks a panel of one plane top to bottom through a private
//      shared-memory ring, finds the pixels that survive the reference's NMS and appends (score, index)
//      records to a small per-plane candidate list, pruning everything that provably cannot reach the
//      plane's top-K (floors.cuh).
//   2. exact-select kernel (exact_select.cuh) -- only for planes whose candidate list overflowed (huge
//      exact plateaus): bounded-memory radix select straight from the heat map.
//   3. tail kernel (tail.cuh) -- one CTA per image: radix-select + sort of the candidates under the
//      total order (score desc, class asc, index asc), zero-fill, offset/embedding gather,
//      coordinate assembly, masking, nearest-anchor grouping.
// plus sdnet_activate_kernel (metadata maps), sdnet_match_kernel (match.cuh, the evaluator's matching) and
// sdnet_sweep_kernel (sweep.cuh, the evaluator at many confidence thresholds).
//
// Numerics contract (SURVEY.md appendix A):
//   * score  = min(max(1/(1+expf(-x)), 1e-6f), (float)(1-1e-6))   -- ATen's CUDA formula;
//   * a pixel survives NMS iff score == max score over its window.  With S monotone
//     non-decreasing in x (verified exhaustively on the device, tests/test_gpu_parity.py)
//     this is  S(x) == S(window-max of x), so the stencil runs on raw logits and the exact
//     sigmoid is evaluated only for the few pixels within a hair of their window maximum;
//   * ties: (score desc, class asc, flat index asc) -- what torch.topk does on CUDA for k > 32;
//   * grouping arithmetic uses explicitly rounded mul/add/sqrt (no FMA contraction) and the
//     first minimum wins.
#include <atomic>
#include <mutex>

#include "common.cuh"
#include "floors.cuh"
#include "peaks_warp.cuh"
#include "peaks_tile.cuh"
#include "exact_select.cuh"
#include "tail.cuh"
#include "match.cuh"
#include "sweep.cuh"
#include "suppress.cuh"

namespace {

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct Workspace {
  size_t off_counts, off_flags, off_sched, off_gfloor, off_hint_used, off_chint, off_ghist, off_lists, total;
  int cap;
};

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

Workspace plan_workspace(int B, int M, int N, int H, int W, int K, int P) {
  Workspace ws;
  const size_t planes = (size_t)B * (M + N);
  const int kmax = K > P ? K : P;
  // A tie-free plane of the benchmark configs records ~9-12 K candidates (K (1 + ln(maxima / K)) plus what the floors'
  // lag lets through); a plane that overflows `cap` (huge exact plateaus) goes through the exact select, which
  // keeps its 1-bit-per-pixel survivor bitmap behind the K output records of the same region.
  const size_t by_k = 8 * (size_t)kmax + 8192, by_map = (size_t)H * W / 8 + 2 * (size_t)kmax + 1024;
  const size_t exact_need = (size_t)kmax + 2 + ((size_t)H * W + 63) / 64 + 16;
  size_t cap = by_k < by_map ? by_k : by_map;
  if (cap < exact_need) cap = exact_need;
  ws.cap = (int)cap;
  size_t off = 0;
  ws.off_counts = off; off = align_up(off + planes * sizeof(int), 256);
  ws.off_flags = off;  off = align_up(off + planes * sizeof(int), 256);
  ws.off_sched = off;  off = align_up(off + 64, 256);
  ws.off_gfloor = off; off = align_up(off + planes * sizeof(int), 256);
  ws.off_hint_used = off; off = align_up(off + planes * sizeof(int), 256);
  ws.off_chint = off;  off = align_up(off + 2 * (size_t)(M + N) * sizeof(u32), 256);
  ws.off_ghist = off;  off = align_up(off + planes * kFineBins * sizeof(u32), 256);
  ws.off_lists = off;  off = align_up(off + planes * (size_t)ws.cap * sizeof(u64), 256);
  ws.total = off;
  return ws;
}

// SM count of the CURRENT device, cached per device ordinal (processes that drive several GPUs from
// different threads see their own device's count); relaxed atomics: the value is idempotent.
int device_sm_count() {
  constexpr int kMaxDev = 64;
  static std::atomic<int> cached[kMaxDev];
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev >= 0 && dev < kMaxDev) {
    sms = cached[dev].load(std::memory_order_relaxed);
    if (sms > 0) return sms;
  }
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) return 148;
  if (dev >= 0 && dev < kMaxDev) cached[dev].store(sms, std::memory_order_relaxed);
  return sms;
}

int validate(const SdnetDecodeParams* p) {
  if (!p) return SDNET_E_NULL;
  if (p->struct_size != sizeof(SdnetDecodeParams)) return SDNET_E_STRUCT;
  if (p->dtype != SDNET_DTYPE_F32 && p->dtype != SDNET_DTYPE_F16 && p->dtype != SDNET_DTYPE_BF16) return SDNET_E_DTYPE;
  if (p->B <= 0 || p->M <= 0 || p->N <= 0 || p->H <= 0 || p->W <= 0 || p->K <= 0 || p->P <= 0) return SDNET_E_SHAPE;
  const long long hw = (long long)p->H * p->W;
  if (hw >= (1ll << 24) || p->K > hw || p->P > hw) return SDNET_E_SHAPE;
  if (p->K > SDNET_MAX_TOPK || p->P > SDNET_MAX_TOPK || p->M + p->N > SDNET_MAX_CHANNELS) return SDNET_E_SHAPE;
  if (p->radius != 1 && p->radius != 2) return SDNET_E_RADIUS;
  if (p->n_dest < 0 || p->n_dest > SDNET_MAX_DEST) return SDNET_E_SHAPE;
  if (p->dest_mode != SDNET_DEST_PEER_STORES && p->dest_mode != SDNET_DEST_MULTICAST) return SDNET_E_SHAPE;
  if (p->dest_mode == SDNET_DEST_MULTICAST && p->n_dest != 1) return SDNET_E_SHAPE;
  const bool no_group = (p->flags & SDNET_FLAG_NO_GROUPING) != 0;
  if (!p->anchor_hm.data || !p->part_hm.data || !p->offsets.data || (!no_group && !p->embeddings.data)) return SDNET_E_NULL;
  if (!p->anchor_out || !p->part_out || !p->anchor_inds || !p->part_inds || !p->assign || !p->counts) return SDNET_E_NULL;
  if ((uintptr_t)p->conf_class_f32 % alignof(float)) return SDNET_E_TABLE;
  if (p->anchor_hm.stride_w != 1 || p->part_hm.stride_w != 1 || p->offsets.stride_w != 1 ||
      (p->embeddings.data && p->embeddings.stride_w != 1))
    return SDNET_E_STRIDE;
  const Workspace ws = plan_workspace(p->B, p->M, p->N, p->H, p->W, p->K, p->P);
  if (!p->workspace || ((uintptr_t)p->workspace & 255) || p->workspace_bytes < ws.total) return SDNET_E_WORKSPACE;
  return 0;
}

View4 to_view(const SdnetTensor4& t) {
  View4 v;
  v.data = t.data;
  v.sb = t.stride_b; v.sc = t.stride_c; v.sh = t.stride_h;
  return v;
}


constexpr int kPeaksCtasPerSm = 4;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      ptr = nullptr;
    return reinterpret_cast<EncodeTiledFn>(ptr);
  }();
  return fn;
}

// How the tile kernel can read a view: 0 = not at all (take the per-lane kernel), 1 = plain rows (pitch
// a multiple of 16 bytes), 2 = row pairs (fp16/bf16 with an 8-byte-multiple pitch, e.g. W = 612).
int tile_rows_per_tma_row(const SdnetTensor4& t, int dtype, int H, int W, int radius) {
  const int px = dtype == SDNET_DTYPE_F32 ? 4 : 8;  // elements per 16 bytes
  if ((uintptr_t)t.data % 16 != 0 || t.stride_b % px != 0 || t.stride_c % px != 0 || t.stride_h < W || W % 4 != 0) return 0;
  if (t.stride_h % px == 0) return 1;
  if (dtype != SDNET_DTYPE_F32 && t.stride_h % 8 == 4 && H % 2 == 0 && radius == 2) return 2;
  return 0;
}

// (W, H, channels, B) view -> tensor map with a (128|256 + halo) x 4 x 1 x 1 box and NaN out-of-bounds
// fill; rows_per_tma_row = 2: (pitch + W, H/2, channels, B) with a 2-row box (see the tile kernel)
bool make_tile_map(CUtensorMap* map, const SdnetTensor4& t, int dtype, int B, int Cn, int H, int W, int rows_per_tma_row) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  // A box side is limited to 256 elements and a fp16/bf16 tile row has 272, so those maps describe
  // PAIRS of elements as one 32-bit float.  Every stride and W are even there, coordinates are halved
  // in the kernel, and the out-of-bounds fill of a float32 map -- measured 0x7FF77FF7 on B200
  // (tools/probes/tma_fill.cu) -- reads as two NaNs in fp16 and in bf16 alike.
  const cuuint64_t esz = dtype == SDNET_DTYPE_F32 ? 4 : 2, per = 4 / esz;
  const int S = rows_per_tma_row;
  const cuuint64_t dims[4] = {(cuuint64_t)(S == 1 ? W : t.stride_h + W) / per, (cuuint64_t)(H / S), (cuuint64_t)Cn, (cuuint64_t)B};
  // strides of size-1 dimensions are arbitrary in torch: make them canonical
  const cuuint64_t sh = (cuuint64_t)t.stride_h * esz;
  const cuuint64_t sc = Cn > 1 ? (cuuint64_t)t.stride_c * esz : sh * (cuuint64_t)H;
  const cuuint64_t sb = B > 1 ? (cuuint64_t)t.stride_b * esz : sc * (cuuint64_t)Cn;
  const cuuint64_t strides[3] = {sh * S, sc, sb};
  const cuuint32_t box[4] = {(cuuint32_t)(kTilePitchB / 4), (cuuint32_t)(kGroupRows / S), 1, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(t.data), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NAN_REQUEST_ZERO_FMA) == CUDA_SUCCESS;
}

// the tile kernel instantiation for (radius, dtype, rows per TMA row)
typedef void (*TileKernel)(const PeaksParams, const CUtensorMap, const CUtensorMap, const HintParams);
template <bool H>
TileKernel tile_kernel_for(int radius, int dtype, int S) {
  if (dtype == SDNET_DTYPE_F32) return radius == 2 ? sdnet_peaks_tile_kernel<2, SDNET_DTYPE_F32, 1, H> : sdnet_peaks_tile_kernel<1, SDNET_DTYPE_F32, 1, H>;
  if (dtype == SDNET_DTYPE_F16) {
    if (S == 2) return sdnet_peaks_tile_kernel<2, SDNET_DTYPE_F16, 2, H>;
    return radius == 2 ? sdnet_peaks_tile_kernel<2, SDNET_DTYPE_F16, 1, H> : sdnet_peaks_tile_kernel<1, SDNET_DTYPE_F16, 1, H>;
  }
  if (S == 2) return sdnet_peaks_tile_kernel<2, SDNET_DTYPE_BF16, 2, H>;
  return radius == 2 ? sdnet_peaks_tile_kernel<2, SDNET_DTYPE_BF16, 1, H> : sdnet_peaks_tile_kernel<1, SDNET_DTYPE_BF16, 1, H>;
}

// Which peaks kernel a decode of these tensors runs (SDNET_PATH_*), encoding the tensor maps on the way.
int select_peaks_path(const SdnetDecodeParams* p, CUtensorMap* tm_anchor, CUtensorMap* tm_part, int* tile_s_out) {
  if (p->flags & SDNET_FLAG_WARP_KERNEL) return SDNET_PATH_WARP;
  int tile_s = tile_rows_per_tma_row(p->anchor_hm, p->dtype, p->H, p->W, p->radius);
  if (tile_s != tile_rows_per_tma_row(p->part_hm, p->dtype, p->H, p->W, p->radius) ||
      (tile_s == 2 && p->anchor_hm.stride_h != p->part_hm.stride_h))
    tile_s = 0;
  if (tile_s != 0 &&
      make_tile_map(tm_anchor, p->anchor_hm, p->dtype, p->B, p->M, p->H, p->W, tile_s) &&
      make_tile_map(tm_part, p->part_hm, p->dtype, p->B, p->N, p->H, p->W, tile_s)) {
    *tile_s_out = tile_s;
    return tile_s == 2 ? SDNET_PATH_TILE_ROW_PAIRS : SDNET_PATH_TILE;
  }
  return SDNET_PATH_WARP;
}

template <typename Kern>
cudaError_t launch_peaks(Kern kern, dim3 grid, dim3 block, cudaStream_t stream, const PeaksParams& pp) {
  // > 48 KB of dynamic shared memory needs the opt-in (idempotent, cheap)
  const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kPeaksSmem);
  if (e != cudaSuccess) return e;
  kern<<<grid, block, kPeaksSmem, stream>>>(pp);
  return cudaSuccess;
}

// Launch with programmatic stream serialization (PDL): see pdl_wait() in the kernels.
template <typename Kern, typename Params>
void launch_pdl(Kern kern, dim3 grid, dim3 block, cudaStream_t stream, const Params& prm) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kern, prm);
}

// Resident CTAs per SM of a tile-kernel instantiation, asked once per (device, instantiation); sets the
// kernel's shared-memory attributes on the way.  0 = the attributes could not be set (`*err` says why).
int tile_ctas_per_sm(TileKernel kern, int dtype, int tile_s, int radius, bool hint, int smem, cudaError_t* err) {
  constexpr int kMaxDev = 64;
  static std::mutex mu;
  static int cache[kMaxDev][3][3][3][2] = {};  // [device][dtype][rows per TMA row][radius][hints]; 0 = not asked yet
  int dev = 0;
  *err = cudaGetDevice(&dev);
  if (*err != cudaSuccess) return 0;
  if (dev < 0 || dev >= kMaxDev) dev = kMaxDev - 1;
  std::lock_guard<std::mutex> lock(mu);
  int& per_sm = cache[dev][dtype][tile_s][radius][hint ? 1 : 0];
  if (per_sm > 0) return per_sm;
  *err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (*err != cudaSuccess) return 0;
  *err = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (*err != cudaSuccess) return 0;
  int n = 0;
  *err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, kTileWarps * 32, smem);
  if (*err != cudaSuccess) return 0;
  per_sm = n < 1 ? 1 : n;
  return per_sm;
}

// Everything the peaks launch needs beyond the tensors: which kernel, how the planes are cut into
// units, how many CTAs.  Host-only (sdnet_decode_schedule reports it without launching).
struct PeaksPlan {
  int path, tile_s;
  TileKernel tile_kern;
  int smem, ctas, ctas_per_sm, sms;
  bool hint;  // the tile kernel runs with floor hints
  CUtensorMap tm_anchor, tm_part;
};

// Cut the line of columns x groups (pp.panels, pp.H set) into units for `resident` warps: see plan_peaks.
bool plan_tile_line(PeaksParams& pp, long long planes, long long resident, int* ctas, long long max_ctas) {
  const long long G = (pp.H + kGroupRows - 1) / kGroupRows;
  const long long columns = planes * pp.panels;
  if (columns * G >= (1ll << 31)) return false;
  const long long tier1 = (columns / resident) * resident;
  const long long rest = (columns - tier1) * G;
  long long chunk = (rest + resident - 1) / resident;
  if (chunk < kMinChunkGroups) chunk = kMinChunkGroups;
  if (chunk > G) chunk = G;
  pp.tier1_units = (int)tier1;
  pp.groups_per_col = (int)G;
  pp.chunk_groups = (int)chunk;
  pp.total_groups = (u32)(columns * G);
  pp.units = (int)(tier1 + (rest + chunk - 1) / chunk);
  long long n = ((long long)pp.units + kTileWarps - 1) / kTileWarps;
  if (n > max_ctas) n = max_ctas;
  *ctas = (int)n;
  return true;
}

cudaError_t plan_peaks(const SdnetDecodeParams* p, PeaksParams& pp, PeaksPlan& pl) {
  const int C = p->M + p->N;
  const long long planes = (long long)p->B * C;
  pl.sms = device_sm_count();
  pl.tile_s = 0;
  pl.hint = false;
  pl.path = select_peaks_path(p, &pl.tm_anchor, &pl.tm_part, &pl.tile_s);
  const bool use_tile = pl.path == SDNET_PATH_TILE || pl.path == SDNET_PATH_TILE_ROW_PAIRS;
  const bool is_f32 = p->dtype == SDNET_DTYPE_F32;
  pp.odd_x = (int)(p->anchor_hm.stride_h / (is_f32 ? 1 : 2));  // in tensor-map elements
  pp.tier1_units = 0;
  pp.groups_per_col = 0;
  pp.chunk_groups = 0;
  pp.total_groups = 0;
  pp.strips = 1;
  pp.rows_per_strip = p->H;
  if (use_tile) {
    pl.tile_kern = tile_kernel_for<false>(p->radius, p->dtype, pl.tile_s);
    const int panel_cols = is_f32 ? TileGeom<SDNET_DTYPE_F32>::kPanel : TileGeom<SDNET_DTYPE_F16>::kPanel;
    pl.smem = tile_smem(pl.tile_s);
    cudaError_t err = cudaSuccess;
    pl.ctas_per_sm = tile_ctas_per_sm(pl.tile_kern, p->dtype, pl.tile_s, p->radius, false, pl.smem, &err);
    if (pl.ctas_per_sm <= 0) return err != cudaSuccess ? err : cudaErrorUnknown;
    pp.panels = (p->W + panel_cols - 1) / panel_cols;
    // The work is a line of `columns` x G groups of four rows (a column = one panel of one plane, top to
    // bottom), cut into units handed out in order by an atomic counter.  Long units prune best (a unit
    // warms its pruning floor once; measured at 128 images: whole columns 0.169 ms, 7 strips 0.221 ms), so:
    //   tier 1: whole columns while they fill whole waves of the resident warps;
    //   tier 2: what is left of the line cut into equal chunks, one per resident warp (a chunk may run
    //           over the end of a column into the next one), so the last wave ends everywhere at once.
    // With fewer columns than resident warps (small shards) everything is tier 2: one balanced wave.
    pp.H = p->H;
    if (!plan_tile_line(pp, planes, (long long)pl.sms * pl.ctas_per_sm * kTileWarps, &pl.ctas, (long long)pl.sms * pl.ctas_per_sm))
      return cudaErrorInvalidValue;
    // Floor hints come from finished whole columns (tier-1 units): a launch without any, e.g. a shard that fits one
    // wave of the resident warps, has none to give and runs the instantiation without the hint code
    if (!(p->flags & SDNET_FLAG_NO_FLOOR_HINT) && pp.tier1_units > 0) {
      pl.hint = true;
      pl.tile_kern = tile_kernel_for<true>(p->radius, p->dtype, pl.tile_s);
      // sets its attributes; same registers and shared memory, so the same CTAs per SM
      if (tile_ctas_per_sm(pl.tile_kern, p->dtype, pl.tile_s, p->radius, true, pl.smem, &err) != pl.ctas_per_sm)
        return err != cudaSuccess ? err : cudaErrorUnknown;
    }
  } else {
    pl.tile_kern = nullptr;
    pl.smem = kPeaksSmem;
    pl.ctas_per_sm = kPeaksCtasPerSm;
    pp.panels = (p->W + kPanelW - 1) / kPanelW;
    const long long resident = (long long)pl.sms * kPeaksCtasPerSm * kWarps;
    const long long units1 = planes * pp.panels;
    int strips = (int)((4 * resident + units1 - 1) / units1);
    const int max_strips = (p->H + 31) / 32;  // strips of at least 32 rows
    if (strips > max_strips) strips = max_strips;
    if (strips < 1) strips = 1;
    pp.rows_per_strip = (p->H + strips - 1) / strips;
    pp.strips = (p->H + pp.rows_per_strip - 1) / pp.rows_per_strip;
    if (planes * pp.strips * pp.panels >= (1ll << 31)) return cudaErrorInvalidValue;
    pp.units = (int)(planes * pp.strips * pp.panels);
    long long ctas = ((long long)pp.units + kWarps - 1) / kWarps;
    if (ctas > (long long)pl.sms * kPeaksCtasPerSm) ctas = (long long)pl.sms * kPeaksCtasPerSm;
    pl.ctas = (int)ctas;
  }
  return cudaSuccess;
}

int launch_decode(const SdnetDecodeParams* p, cudaStream_t stream, cudaEvent_t* marks = nullptr) {
  const Workspace ws = plan_workspace(p->B, p->M, p->N, p->H, p->W, p->K, p->P);
  char* base = static_cast<char*>(p->workspace);
  const int C = p->M + p->N;
  const size_t planes = (size_t)p->B * C;
  const int sms = device_sm_count();

  PeaksParams pp;
  pp.anchor = to_view(p->anchor_hm);
  pp.part = to_view(p->part_hm);
  pp.B = p->B; pp.M = p->M; pp.N = p->N; pp.H = p->H; pp.W = p->W; pp.K = p->K; pp.P = p->P;
  pp.cap = ws.cap;
  pp.pre_activated = (p->flags & SDNET_FLAG_PRE_ACTIVATED) ? 1 : 0;
  pp.lists = reinterpret_cast<u64*>(base + ws.off_lists);
  pp.counts = reinterpret_cast<int*>(base + ws.off_counts);
  pp.sched = reinterpret_cast<u32*>(base + ws.off_sched);
  pp.ghist = reinterpret_cast<u32*>(base + ws.off_ghist);
  pp.gfloor = reinterpret_cast<int*>(base + ws.off_gfloor);
  PeaksPlan pl;
  cudaError_t err = plan_peaks(p, pp, pl);
  if (err != cudaSuccess) return (int)err;
  HintParams hp;
  hp.chint = reinterpret_cast<u32*>(base + ws.off_chint);
  hp.hint_used = reinterpret_cast<int*>(base + ws.off_hint_used);
  if (!(p->flags & SDNET_FLAG_WORKSPACE_CLEAN)) {  // else: the previous decode's tail kernel left the header zeroed
    err = cudaMemsetAsync(base, 0, ws.off_lists, stream);
    if (err != cudaSuccess) return (int)err;
  }
  if (marks) cudaEventRecord(marks[0], stream);

  if (pl.tile_kern) {
    pl.tile_kern<<<dim3((unsigned)pl.ctas), dim3(kTileWarps * 32), pl.smem, stream>>>(pp, pl.tm_anchor, pl.tm_part, hp);
  } else {
    dim3 grid((unsigned)pl.ctas), block(kThreads);
    const bool r2 = p->radius == 2;
    if (p->dtype == SDNET_DTYPE_F16) {
      err = r2 ? launch_peaks(sdnet_peaks_kernel<2, SDNET_DTYPE_F16>, grid, block, stream, pp)
               : launch_peaks(sdnet_peaks_kernel<1, SDNET_DTYPE_F16>, grid, block, stream, pp);
    } else if (p->dtype == SDNET_DTYPE_BF16) {
      err = r2 ? launch_peaks(sdnet_peaks_kernel<2, SDNET_DTYPE_BF16>, grid, block, stream, pp)
               : launch_peaks(sdnet_peaks_kernel<1, SDNET_DTYPE_BF16>, grid, block, stream, pp);
    } else {
      err = r2 ? launch_peaks(sdnet_peaks_kernel<2, SDNET_DTYPE_F32>, grid, block, stream, pp)
               : launch_peaks(sdnet_peaks_kernel<1, SDNET_DTYPE_F32>, grid, block, stream, pp);
    }
    if (err != cudaSuccess) return (int)err;
  }
  err = cudaGetLastError();
  if (err != cudaSuccess) return (int)err;
  if (marks) cudaEventRecord(marks[1], stream);

  {
    ExactParams ep;
    ep.anchor = pp.anchor; ep.part = pp.part;
    ep.B = p->B; ep.M = p->M; ep.N = p->N; ep.H = p->H; ep.W = p->W; ep.K = p->K; ep.P = p->P;
    ep.radius = p->radius; ep.cap = ws.cap;
    ep.force = (p->flags & SDNET_FLAG_EXACT_SELECT) ? 1 : 0;
    ep.pre_activated = pp.pre_activated;
    ep.lists = pp.lists; ep.counts = pp.counts;
    ep.flags = reinterpret_cast<int*>(base + ws.off_flags);
    ep.check_hints = pl.hint;
    ep.gfloor = pp.gfloor; ep.ghist = pp.ghist; ep.hint_used = hp.hint_used;
    // (with several decodes in flight this pass-through launch costs 0.5 % of the step at 1024 images and 1-4 % at 128
    // even with thin CTAs -- measured by skipping it; moving it behind the tail, with a fix-up tail launch after it, gets
    // back 1.5 % at 128 and was not worth a fourth launch)
    {
      const size_t exact_grid = planes < (size_t)sms * kExactCtasPerSm ? planes : (size_t)sms * kExactCtasPerSm;
      if (p->dtype == SDNET_DTYPE_F16) launch_pdl(sdnet_exact_select_kernel<SDNET_DTYPE_F16>, dim3((unsigned)exact_grid), dim3(kExactThreads), stream, ep);
      else if (p->dtype == SDNET_DTYPE_BF16) launch_pdl(sdnet_exact_select_kernel<SDNET_DTYPE_BF16>, dim3((unsigned)exact_grid), dim3(kExactThreads), stream, ep);
      else launch_pdl(sdnet_exact_select_kernel<SDNET_DTYPE_F32>, dim3((unsigned)exact_grid), dim3(kExactThreads), stream, ep);
    }
    err = cudaGetLastError();
    if (err != cudaSuccess) return (int)err;
    if (marks) cudaEventRecord(marks[2], stream);
  }

  TailParams tp;
  tp.offsets = to_view(p->offsets);
  tp.embeddings = to_view(p->embeddings);
  tp.B = p->B; tp.M = p->M; tp.N = p->N; tp.H = p->H; tp.W = p->W; tp.K = p->K; tp.P = p->P;
  tp.cap = ws.cap;
  tp.pre_activated = pp.pre_activated;
  tp.no_grouping = (p->flags & SDNET_FLAG_NO_GROUPING) ? 1 : 0;
  tp.conf = p->conf_f32;
  tp.conf_class = p->conf_class_f32;
  tp.dist_abs = p->dist_abs_f32;
  tp.lists = pp.lists;
  tp.counts = pp.counts;
  tp.anchor_out = p->anchor_out;
  tp.part_out = p->part_out;
  tp.anchor_inds = reinterpret_cast<long long*>(p->anchor_inds);
  tp.part_inds = reinterpret_cast<long long*>(p->part_inds);
  tp.part_emb = p->part_emb;
  tp.assign = p->assign;
  tp.out_counts = p->counts;
  tp.diag = p->diag;
  tp.exact_flags = reinterpret_cast<const int*>(base + ws.off_flags);
  tp.ghist = pp.ghist;
  tp.n_dest = p->n_dest;
  tp.dest_multicast = p->dest_mode == SDNET_DEST_MULTICAST ? 1 : 0;
  tp.done_flag = p->n_dest > 0 ? p->done_flag : nullptr;
  tp.done_value = p->done_value;
  tp.ticket = pp.sched + 1;  // second word of the scheduler block, zeroed with it
  tp.ws_counts = pp.counts;
  tp.ws_flags = reinterpret_cast<int*>(base + ws.off_flags);
  tp.ws_gfloor = pp.gfloor;
  tp.ws_ghist = pp.ghist;
  tp.ws_hint_used = hp.hint_used;
  tp.ws_chint = hp.chint;
  tp.ws_sched = pp.sched;
  for (int j = 0; j < SDNET_MAX_DEST; ++j) tp.dest_delta[j] = j < p->n_dest ? p->dest_delta[j] : 0;
  if (p->dtype == SDNET_DTYPE_F16) launch_pdl(sdnet_tail_kernel<SDNET_DTYPE_F16>, dim3((unsigned)p->B), dim3(2 * kTeamThreads), stream, tp);
  else if (p->dtype == SDNET_DTYPE_BF16) launch_pdl(sdnet_tail_kernel<SDNET_DTYPE_BF16>, dim3((unsigned)p->B), dim3(2 * kTeamThreads), stream, tp);
  else launch_pdl(sdnet_tail_kernel<SDNET_DTYPE_F32>, dim3((unsigned)p->B), dim3(2 * kTeamThreads), stream, tp);
  err = cudaGetLastError();
  if (marks) cudaEventRecord(marks[3], stream);
  return (int)err;
}

}  // namespace

extern "C" {

int sdnet_abi_version(void) { return SDNET_ABI_VERSION; }

const char* sdnet_error_string(int code) {
  switch (code) {
    case 0: return "ok";
    case SDNET_E_NULL: return "a required pointer is NULL";
    case SDNET_E_SHAPE: return "bad shape (non-positive dim, H*W >= 2^24, k out of range, or above SDNET_MAX_*)";
    case SDNET_E_STRIDE: return "innermost stride must be 1";
    case SDNET_E_DTYPE: return "unsupported dtype";
    case SDNET_E_WORKSPACE: return "workspace missing, misaligned or too small";
    case SDNET_E_RADIUS: return "unsupported NMS radius";
    case SDNET_E_STRUCT: return "SdnetDecodeParams.struct_size mismatch";
    case SDNET_E_TABLE: return "per-class threshold table not aligned to its element type";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
  }
}

int sdnet_decode_workspace_bytes(int B, int M, int N, int H, int W, int K, int P, int dtype, size_t* out_bytes) {
  if (!out_bytes) return SDNET_E_NULL;
  if (dtype != SDNET_DTYPE_F32 && dtype != SDNET_DTYPE_F16 && dtype != SDNET_DTYPE_BF16) return SDNET_E_DTYPE;
  if (B <= 0 || M <= 0 || N <= 0 || H <= 0 || W <= 0 || K <= 0 || P <= 0) return SDNET_E_SHAPE;
  if ((long long)H * W >= (1ll << 24)) return SDNET_E_SHAPE;
  *out_bytes = plan_workspace(B, M, N, H, W, K, P).total;
  return 0;
}

int sdnet_gather_wait_launch(const uint32_t* flags, int world, uint32_t value, void* stream) {
  if (!flags) return SDNET_E_NULL;
  if (world <= 0 || world > SDNET_MAX_DEST) return SDNET_E_SHAPE;
  sdnet_gather_wait_kernel<<<dim3(1), dim3(32), 0, static_cast<cudaStream_t>(stream)>>>(flags, world, value);
  return (int)cudaGetLastError();
}

int sdnet_match_launch(const SdnetMatchParams* p, void* stream) {
  if (!p) return SDNET_E_NULL;
  if (p->struct_size != sizeof(SdnetMatchParams)) return SDNET_E_STRUCT;
  if (!p->anchor_out || !p->part_out || !p->image_scale || !p->n_gt_anchors || !p->n_gt_parts || !p->anchor_stats ||
      !p->part_stats || !p->anchor_acc || !p->part_acc || (p->max_gt_anchors > 0 && !p->gt_anchors) ||
      (p->max_gt_parts > 0 && !p->gt_parts))
    return SDNET_E_NULL;
  if (p->B <= 0 || p->M <= 0 || p->N <= 0 || p->K <= 0 || p->P <= 0 || p->K > SDNET_MAX_TOPK || p->P > SDNET_MAX_TOPK ||
      p->M + p->N > SDNET_MAX_CHANNELS || p->max_gt_anchors < 0 || p->max_gt_parts < 0 || p->max_gt_anchors > SDNET_MAX_GT ||
      p->max_gt_parts > SDNET_MAX_GT)
    return SDNET_E_SHAPE;
  if ((uintptr_t)p->conf_class % alignof(double)) return SDNET_E_TABLE;
  sdnet_match_kernel<<<dim3((unsigned)p->B), dim3(kMatchThreads), 0, static_cast<cudaStream_t>(stream)>>>(*p);
  return (int)cudaGetLastError();
}

int sdnet_match_objects_launch(const SdnetObjectMatchParams* p, void* stream) {
  if (!p) return SDNET_E_NULL;
  if (p->struct_size != sizeof(SdnetObjectMatchParams)) return SDNET_E_STRUCT;
  if (!p->anchor_out || !p->part_out || !p->assign || !p->image_scale || !p->n_gt_objects || !p->n_gt_parts || !p->cls_group ||
      !p->csi_stats || !p->csi_acc || !p->classif_stats || !p->classif_acc || !p->pred_parts ||
      (p->max_gt_objects > 0 && !p->gt_objects) || (p->max_gt_parts > 0 && (!p->gt_parts || !p->gt_part_owner)))
    return SDNET_E_NULL;
  if (p->B <= 0 || p->M <= 0 || p->N <= 0 || p->K <= 0 || p->P <= 0 || p->K > SDNET_MAX_TOPK || p->P > SDNET_MAX_TOPK ||
      p->M + p->N > SDNET_MAX_CHANNELS || p->max_gt_objects < 0 || p->max_gt_parts < 0 || p->max_gt_objects > SDNET_MAX_GT ||
      p->max_gt_parts > SDNET_MAX_GT)
    return SDNET_E_SHAPE;
  if ((uintptr_t)p->conf_class % alignof(double)) return SDNET_E_TABLE;
  const size_t smem = match_objects_smem_bytes(p->max_gt_objects, p->max_gt_parts, p->K, p->P, p->M);
  cudaError_t err = cudaFuncSetAttribute(sdnet_match_objects_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return (int)err;
  sdnet_match_objects_kernel<<<dim3((unsigned)p->B), dim3(kMatchThreads), smem, static_cast<cudaStream_t>(stream)>>>(*p);
  return (int)cudaGetLastError();
}

int sdnet_sweep_launch(const SdnetSweepParams* p, void* stream) {
  if (!p) return SDNET_E_NULL;
  if (p->struct_size != sizeof(SdnetSweepParams)) return SDNET_E_STRUCT;
  const bool objects = (p->flags & SDNET_SWEEP_OBJECTS) != 0;
  if (!p->conf || !p->conf_group || !p->anchor_out || !p->part_out || !p->image_scale || !p->n_gt_objects ||
      !p->n_gt_parts || !p->anchor_stats || !p->part_stats || !p->anchor_acc || !p->part_acc ||
      (p->max_gt_objects > 0 && !p->gt_objects) || (p->max_gt_parts > 0 && !p->gt_parts) ||
      (p->G >= 1 && !p->dist_abs_grid))
    return SDNET_E_NULL;
  if (objects && (!p->cls_group || !p->csi_stats || !p->csi_acc || !p->classif_stats || !p->classif_acc ||
                  !p->pred_parts || (p->max_gt_parts > 0 && !p->gt_part_owner)))
    return SDNET_E_NULL;
  if (p->B <= 0 || p->M <= 0 || p->N <= 0 || p->K <= 0 || p->P <= 0 || p->K > SDNET_MAX_TOPK || p->P > SDNET_MAX_TOPK ||
      p->M + p->N > SDNET_MAX_CHANNELS || p->T < 1 || p->T > SDNET_MAX_THRESHOLDS || p->max_gt_objects < 0 ||
      p->max_gt_parts < 0 || p->max_gt_objects > SDNET_MAX_GT || p->max_gt_parts > SDNET_MAX_GT ||
      p->G < 0 || p->G > SDNET_MAX_GATES || (long long)p->B * p->T * (p->G > 1 ? p->G : 1) > 0x7fffffffll)
    return SDNET_E_SHAPE;
  const size_t smem = sweep_smem_bytes(*p);
  cudaError_t err = cudaFuncSetAttribute(sdnet_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return (int)err;
  sdnet_sweep_kernel<<<dim3((unsigned)(p->B * p->T)), dim3(kMatchThreads), smem, static_cast<cudaStream_t>(stream)>>>(*p);
  return (int)cudaGetLastError();
}

int sdnet_decode_peaks_path(const SdnetDecodeParams* params) {
  const int rc = validate(params);
  if (rc != 0) return rc;
  CUtensorMap a, b;
  int tile_s = 0;
  return select_peaks_path(params, &a, &b, &tile_s);
}

int sdnet_decode_schedule(const SdnetDecodeParams* params, SdnetSchedule* out) {
  const int rc = validate(params);
  if (rc != 0) return rc;
  if (!out) return SDNET_E_NULL;
  if (out->struct_size != sizeof(SdnetSchedule)) return SDNET_E_STRUCT;
  PeaksParams pp;
  PeaksPlan pl;
  const cudaError_t err = plan_peaks(params, pp, pl);
  if (err != cudaSuccess) return (int)err;
  out->path = pl.path;
  out->units = pp.units;
  out->tier1_units = pp.tier1_units;
  out->chunk_units = pl.tile_kern ? pp.units - pp.tier1_units : 0;
  out->chunk_groups = pp.chunk_groups;
  out->groups_per_column = pp.groups_per_col;
  out->panels = pp.panels;
  out->strips = pp.strips;
  out->rows_per_strip = pp.rows_per_strip;
  out->ctas = pl.ctas;
  out->warps_per_cta = pl.tile_kern ? kTileWarps : kWarps;
  out->ctas_per_sm = pl.ctas_per_sm;
  out->sms = pl.sms;
  out->list_capacity = plan_workspace(params->B, params->M, params->N, params->H, params->W, params->K, params->P).cap;
  return 0;
}

int sdnet_decode_launch(const SdnetDecodeParams* params, void* stream) {
  const int rc = validate(params);
  if (rc) return rc;
  return launch_decode(params, static_cast<cudaStream_t>(stream));
}

int sdnet_decode_launch_timed(const SdnetDecodeParams* params, void* stream_v, float* kernel_ms) {
  const int rc = validate(params);
  if (rc) return rc;
  if (!kernel_ms) return SDNET_E_NULL;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  cudaEvent_t marks[4];
  for (int i = 0; i < 4; ++i) {
    cudaError_t e = cudaEventCreate(&marks[i]);
    if (e != cudaSuccess) return (int)e;
  }
  int out = launch_decode(params, stream, marks);
  if (out == 0) {
    cudaError_t e = cudaEventSynchronize(marks[3]);
    if (e != cudaSuccess) out = (int)e;
    for (int i = 0; i < 3 && out == 0; ++i) {
      e = cudaEventElapsedTime(&kernel_ms[i], marks[i], marks[i + 1]);
      if (e != cudaSuccess) out = (int)e;
    }
  }
  for (int i = 0; i < 4; ++i) cudaEventDestroy(marks[i]);
  return out;
}

int sdnet_activate_launch(const SdnetTensor4* in, int dtype, int B, int C, int H, int W, float* out, void* stream) {
  if (!in || !in->data || !out) return SDNET_E_NULL;
  if (dtype != SDNET_DTYPE_F32 && dtype != SDNET_DTYPE_F16 && dtype != SDNET_DTYPE_BF16) return SDNET_E_DTYPE;
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return SDNET_E_SHAPE;
  if (in->stride_w != 1) return SDNET_E_STRIDE;
  const size_t total = (size_t)B * C * H * W;
  const int sms = device_sm_count();
  size_t blocks = (total + 255) / 256;
  if (blocks > (size_t)sms * 8) blocks = (size_t)sms * 8;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == SDNET_DTYPE_F16) sdnet_activate_kernel<SDNET_DTYPE_F16><<<dim3((unsigned)blocks), dim3(256), 0, st>>>(to_view(*in), C, H, W, total, out);
  else if (dtype == SDNET_DTYPE_BF16) sdnet_activate_kernel<SDNET_DTYPE_BF16><<<dim3((unsigned)blocks), dim3(256), 0, st>>>(to_view(*in), C, H, W, total, out);
  else sdnet_activate_kernel<SDNET_DTYPE_F32><<<dim3((unsigned)blocks), dim3(256), 0, st>>>(to_view(*in), C, H, W, total, out);
  return (int)cudaGetLastError();
}

int sdnet_suppress_into_launch(const SdnetTensor4* in, int dtype, int B, int C, int H, int W, int radius, const SdnetTensor4* out_t,
                               void* stream) {
  if (!in || !in->data || !out_t || !out_t->data) return SDNET_E_NULL;
  if (out_t->stride_w != 1 || out_t->stride_h < W) return SDNET_E_STRIDE;
  const View4 outv = to_view(*out_t);
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return SDNET_E_SHAPE;
  if (in->stride_w != 1) return SDNET_E_STRIDE;
  if (dtype != SDNET_DTYPE_F32 && dtype != SDNET_DTYPE_F16 && dtype != SDNET_DTYPE_BF16) return SDNET_E_DTYPE;
  if (radius != 1 && radius != 2) return SDNET_E_RADIUS;
  // fp32 maps that TMA can describe (and a 16-byte-aligned output): the tile kernel
  CUtensorMap tm;
  if (dtype == SDNET_DTYPE_F32 &&
      (((uintptr_t)out_t->data | (uintptr_t)(out_t->stride_b * 4) | (uintptr_t)(out_t->stride_c * 4) | (uintptr_t)(out_t->stride_h * 4)) & 15) == 0 && (long long)B * C * ((W + kPanelW - 1) / kPanelW) * ((H + 3) / 4) < (1ll << 31) &&
      tile_rows_per_tma_row(*in, dtype, H, W, radius) == 1 && make_tile_map(&tm, *in, dtype, B, C, H, W, 1)) {
    PeaksParams pp = {};
    pp.B = B; pp.M = C; pp.N = 0; pp.H = H; pp.W = W;
    pp.panels = (W + kPanelW - 1) / kPanelW;
    const auto kern = radius == 2 ? sdnet_suppress_tile_kernel<2> : sdnet_suppress_tile_kernel<1>;
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSupTileSmem);
    if (err != cudaSuccess) return (int)err;
    err = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (err != cudaSuccess) return (int)err;
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kTileWarps * 32, kSupTileSmem);
    if (err != cudaSuccess) return (int)err;
    if (per_sm < 1) per_sm = 1;
    const int sms = device_sm_count();
    int ctas = 0;
    plan_tile_line(pp, (long long)B * C, (long long)sms * per_sm * kTileWarps, &ctas, sms * per_sm);
    kern<<<dim3((unsigned)ctas), dim3(kTileWarps * 32), kSupTileSmem, static_cast<cudaStream_t>(stream)>>>(pp, tm, outv);
    return (int)cudaGetLastError();
  }
  const int panels = (W + kPanelW - 1) / kPanelW, strips = (H + kSupStripRows - 1) / kSupStripRows;
  const long long units = (long long)panels * strips * C * B;
  const long long blocks = (units + kSupWarps - 1) / kSupWarps;
  if (blocks > 0x7fffffffll) return SDNET_E_SHAPE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const dim3 grid((unsigned)blocks), block(kSupWarps * 32);
  const View4 v = to_view(*in);
#define SDNET_SUPPRESS(R, DT) sdnet_suppress_kernel<R, DT><<<grid, block, 0, st>>>(v, C, H, W, panels, strips, units, outv)
  if (dtype == SDNET_DTYPE_F16) { if (radius == 2) SDNET_SUPPRESS(2, SDNET_DTYPE_F16); else SDNET_SUPPRESS(1, SDNET_DTYPE_F16); }
  else if (dtype == SDNET_DTYPE_BF16) { if (radius == 2) SDNET_SUPPRESS(2, SDNET_DTYPE_BF16); else SDNET_SUPPRESS(1, SDNET_DTYPE_BF16); }
  else { if (radius == 2) SDNET_SUPPRESS(2, SDNET_DTYPE_F32); else SDNET_SUPPRESS(1, SDNET_DTYPE_F32); }
#undef SDNET_SUPPRESS
  return (int)cudaGetLastError();
}

int sdnet_suppress_launch(const SdnetTensor4* in, int dtype, int B, int C, int H, int W, int radius, float* out, void* stream) {
  if (!out) return SDNET_E_NULL;
  SdnetTensor4 dense;
  dense.data = out;
  dense.stride_w = 1;
  dense.stride_h = W;
  dense.stride_c = (int64_t)H * W;
  dense.stride_b = (int64_t)C * H * W;
  return sdnet_suppress_into_launch(in, dtype, B, C, H, W, radius, &dense, stream);
}

int sdnet_decode_host_launch(const SdnetDecodeParams* params, void* staging, size_t staging_bytes, void* stream_v) {
  const int rc = validate(params);
  if (rc) return rc;
  if (!staging) return SDNET_E_NULL;
  const SdnetDecodeParams& p = *params;
  const size_t esz = p.dtype == SDNET_DTYPE_F32 ? 4 : 2;
  const size_t plane_bytes = (size_t)p.H * p.W * esz;
  const size_t need = (size_t)p.B * (p.M + p.N) * plane_bytes;
  if (staging_bytes < need || ((uintptr_t)staging & 255)) return SDNET_E_WORKSPACE;
  // dense rows; dense channels (a single channel has no channel stride to speak of)
  if (p.anchor_hm.stride_h != p.W || p.part_hm.stride_h != p.W) return SDNET_E_STRIDE;
  if ((p.M > 1 && p.anchor_hm.stride_c != (long long)p.H * p.W) || (p.N > 1 && p.part_hm.stride_c != (long long)p.H * p.W))
    return SDNET_E_STRIDE;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  // heat planes: host (strided per image) -> dense device staging [B][M+N][H][W]
  char* dst = static_cast<char*>(staging);
  const size_t img_bytes = (size_t)(p.M + p.N) * plane_bytes;
  cudaError_t err = cudaMemcpy2DAsync(dst, img_bytes, p.anchor_hm.data, (size_t)p.anchor_hm.stride_b * esz,
                                      (size_t)p.M * plane_bytes, p.B, cudaMemcpyHostToDevice, stream);
  if (err != cudaSuccess) return (int)err;
  err = cudaMemcpy2DAsync(dst + (size_t)p.M * plane_bytes, img_bytes, p.part_hm.data, (size_t)p.part_hm.stride_b * esz,
                          (size_t)p.N * plane_bytes, p.B, cudaMemcpyHostToDevice, stream);
  if (err != cudaSuccess) return (int)err;
  SdnetDecodeParams q = p;
  q.anchor_hm.data = dst;
  q.anchor_hm.stride_b = (long long)(p.M + p.N) * p.H * p.W;
  q.anchor_hm.stride_c = (long long)p.H * p.W;
  q.part_hm.data = dst + (size_t)p.M * plane_bytes;
  q.part_hm.stride_b = q.anchor_hm.stride_b;
  q.part_hm.stride_c = q.anchor_hm.stride_c;
  // offsets / embeddings stay in pinned host memory: the tail kernel reads them through
  // the unified address space only at the K + 2P selected pixels per image.
  return launch_decode(&q, stream);
}

}  // extern "C"
