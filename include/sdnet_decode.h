/*
 * sdnet_decode.h -- C ABI of the B200-native SDNet decoding path.
 *
 * The reference (laclouis5/StructureDetector) is pure Python and has no FFI of its own;
 * these entry points are what a binding for its decoding path would call.  Each one
 * names the reference code it replaces (paths relative to the reference repo root).
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; no C++/torch types cross the boundary;
 *   - the caller owns every buffer (inputs, outputs, workspace); the library never
 *     allocates or frees device memory and keeps no per-call state;
 *   - stream-ordered and asynchronous: work is enqueued on `stream` (a cudaStream_t
 *     passed as void*), nothing synchronises;
 *   - re-entrant across host threads and streams given distinct workspaces;
 *   - return value: 0 = OK; negative = argument error detected on the host before any
 *     launch (SDNET_E_*); positive = a cudaError_t raised by a launch.
 *   - there is no CPU fallback: on a machine without a CUDA device every launch
 *     returns a positive cudaError_t.
 */
#ifndef SDNET_DECODE_H_
#define SDNET_DECODE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDNET_ABI_VERSION 10

/* element types of the four input tensors */
#define SDNET_DTYPE_F32 0
#define SDNET_DTYPE_F16 1  /* what the reference's --amp validation feeds the decoder (src/sdnet/model/trainer.py:40-42,142-157) */
#define SDNET_DTYPE_BF16 2

/* SdnetDecodeParams.flags */
#define SDNET_FLAG_PRE_ACTIVATED 1u /* heat maps already sigmoid+NMS'd: decoders.py:211,226 (CoreMLDecoder) */
#define SDNET_FLAG_NO_GROUPING 2u   /* skip part->anchor grouping: decoders.py:345-423 (KeypointDecoder) */
#define SDNET_FLAG_EXACT_SELECT 4u  /* route every plane through the bounded-memory exact select (testing) */
#define SDNET_FLAG_WARP_KERNEL 8u   /* use the any-alignment per-warp peaks kernel even when the TMA one applies (testing) */
#define SDNET_FLAG_WORKSPACE_CLEAN 16u /* the caller promises that the last thing that touched `workspace` was a completed
                                          decode of the same shape (every decode leaves the workspace header zeroed behind
                                          it), so the per-call cudaMemsetAsync of the header is skipped: one stream
                                          operation less per decode.  Never set it for a fresh or reused-elsewhere buffer. */

/* argument errors */
#define SDNET_E_NULL -1      /* a required pointer is NULL */
#define SDNET_E_SHAPE -2     /* non-positive dimension, H*W >= 2^24, K or P > H*W (torch.topk: "k out of range"),
                                K or P > SDNET_MAX_TOPK, M+N > SDNET_MAX_CHANNELS, T outside 1..SDNET_MAX_THRESHOLDS,
                                G outside 0..SDNET_MAX_GATES */
#define SDNET_E_STRIDE -3    /* innermost (w) stride is not 1 */
#define SDNET_E_DTYPE -4     /* unsupported dtype */
#define SDNET_E_WORKSPACE -5 /* workspace missing, misaligned (256 B) or smaller than sdnet_decode_workspace_bytes */
#define SDNET_E_RADIUS -6    /* NMS window radius other than 2 (5x5, utils.py:442) or 1 (3x3) */
#define SDNET_E_STRUCT -7    /* struct_size does not match this library's SdnetDecodeParams */

#define SDNET_MAX_TOPK 1024
#define SDNET_MAX_CHANNELS 255
#define SDNET_MAX_DEST 16
#define SDNET_DEST_PEER_STORES 0 /* SdnetDecodeParams.dest_mode: one st.global per destination */
#define SDNET_DEST_MULTICAST 1   /* one multimem.st to the multicast address of the destination blob */

/* A strided NCHW view.  Strides are in ELEMENTS.  The decoder consumes the channel-slice
 * views produced by the reference network (src/sdnet/model/network.py:79-84), which are
 * not contiguous in the batch dimension, so b/c/h strides are free; stride_w must be 1. */
typedef struct SdnetTensor4 {
  const void* data;
  int64_t stride_b, stride_c, stride_h, stride_w;
} SdnetTensor4;

typedef struct SdnetDecodeParams {
  uint32_t struct_size; /* sizeof(SdnetDecodeParams) */
  int32_t dtype;        /* SDNET_DTYPE_*: element type of all four input tensors */
  int32_t B, M, N, H, W; /* batch, anchor classes, part kinds, map rows, map cols */
  int32_t K, P;          /* max_objects, max_parts (decoders.py:25-26) */
  int32_t radius;        /* NMS window radius; 2 = the reference's 5x5 (utils.py:442) */
  uint32_t flags;        /* SDNET_FLAG_* */
  float conf_f32;        /* (float)conf_thresh: `scores > conf` is an fp32 compare (decoders.py:78,83) */
  float dist_abs_f32;    /* (float)(dist_thresh * min(W, H)) (decoders.py:100) */
  SdnetTensor4 anchor_hm;  /* (B, M, H, W) logits */
  SdnetTensor4 part_hm;    /* (B, N, H, W) logits */
  SdnetTensor4 offsets;    /* (B, 2, H, W) */
  SdnetTensor4 embeddings; /* (B, 2, H, W); may be NULL data with SDNET_FLAG_NO_GROUPING */
  /* outputs, all contiguous, all device memory */
  float* anchor_out;    /* (B, K, 4) x, y, score, class           decoders.py:55-57 */
  float* part_out;      /* (B, P, 6) x, y, score, kind, ox, oy    decoders.py:72-75 */
  int64_t* anchor_inds; /* (B, K) flat h*W+w index of each slot   utils.py:463 */
  int64_t* part_inds;   /* (B, P) */
  float* part_emb;      /* (B, P, 2) gathered embeddings, optional (NULL to skip)  decoders.py:66 */
  int32_t* assign;      /* (B, P) anchor slot of each part, -1 when not grouped  decoders.py:99-100,108-112 */
  int32_t* counts;      /* (B, 2) slots with score > conf: anchors, parts */
  int32_t* diag;        /* optional (B*(M+N), 2): candidates emitted per plane, 1 if the exact select ran */
  void* workspace;
  size_t workspace_bytes;
  /* Fused detection gather (multi-GPU): when n_dest > 0 every output above is written n_dest times, to
   * (char*)ptr + dest_delta[j].  With the outputs placed in a symmetric (peer-mapped) allocation,
   * dest_delta[j] = peer_base[j] - local_base makes the tail kernel store each rank's detections
   * straight into every peer's copy over NVLink; one cross-GPU barrier afterwards replaces the
   * all-gather.  Include 0 in dest_delta to also keep the local copy.  n_dest = 0: plain local stores.
   * dest_mode = SDNET_DEST_MULTICAST (with n_dest = 1): dest_delta[0] = multicast_base - local_base, where
   * multicast_base is the NVSwitch multicast mapping of the same symmetric allocation; every value is then
   * stored ONCE with multimem.st and the switch replicates it into every GPU's copy (the local one included). */
  int32_t n_dest;
  int32_t dest_mode; /* SDNET_DEST_* */
  int64_t dest_delta[SDNET_MAX_DEST];
  /* Completion flag of the fused gather (optional, n_dest > 0 only): when done_flag is not NULL, the last CTA of the
   * tail kernel to finish -- after every CTA's output stores and a system-scope fence -- stores done_value to
   * (char*)done_flag + dest_delta[j] in every destination copy (release, system scope; one multimem.st under
   * SDNET_DEST_MULTICAST).  With done_flag = &flags[rank] of a per-rank flag array inside the symmetric allocation and
   * done_value counting this rank's decodes, sdnet_gather_wait_launch on flags replaces the cross-GPU barrier. */
  uint32_t* done_flag;
  uint32_t done_value;
  uint32_t reserved1;
} SdnetDecodeParams;

/* Library / ABI identification. */
int sdnet_abi_version(void);
const char* sdnet_error_string(int code);

/* Scratch size for one in-flight decode of the given shape. */
int sdnet_decode_workspace_bytes(int B, int M, int N, int H, int W, int K, int P, int dtype, size_t* out_bytes);

/* The whole tensor half of Decoder.__call__ (src/sdnet/data/decoders.py:44-100 with
 * src/sdnet/utils/utils.py:355-361 clamped_sigmoid, 441-443 nms, 447-467 topk,
 * 347-351 transpose_and_gather, 422-437 hypot): heat maps -> packed detections. */
int sdnet_decode_launch(const SdnetDecodeParams* params, void* stream);

/* Which peaks kernel sdnet_decode_launch would run for these tensors (shape, strides, alignment, dtype,
 * flags): one of SDNET_PATH_*, or a negative SDNET_E_*.  Host-only; launches nothing.  The kernels give
 * identical results; tests use this to know which one they exercised. */
#define SDNET_PATH_WARP 0           /* per-lane cp.async / converting feed: any shape, stride and alignment */
#define SDNET_PATH_TILE 1           /* TMA tiles: base and strides multiples of 16 bytes, W % 4 == 0 */
#define SDNET_PATH_TILE_ROW_PAIRS 2 /* TMA tiles over row pairs: fp16/bf16 with an 8-byte-multiple row pitch (W = 612), H even */
int sdnet_decode_peaks_path(const SdnetDecodeParams* params);

/* How sdnet_decode_launch would cut these tensors into work for the peaks kernel on the current device
 * (host-only; launches nothing).  The TMA tile kernel walks a line of columns (one panel of one plane,
 * top to bottom; groups_per_column groups of four rows each): units [0, tier1_units) are whole columns,
 * the rest of the line is cut into chunks of chunk_groups groups, one unit each.  The per-lane kernel
 * cuts every plane into `strips` strips of rows_per_strip rows.  Parity tests use this to assert WHICH
 * schedule branch a case exercised (whole columns, chunks, or both). */
typedef struct SdnetSchedule {
  uint32_t struct_size;  /* sizeof(SdnetSchedule), set by the caller */
  int32_t path;          /* SDNET_PATH_* */
  int32_t units;         /* work units handed out by the kernel's atomic counter */
  int32_t tier1_units;   /* tile kernel: whole-column units */
  int32_t chunk_units;   /* tile kernel: units - tier1_units */
  int32_t chunk_groups;  /* tile kernel: groups of four rows per chunk unit */
  int32_t groups_per_column;
  int32_t panels;        /* panels per plane */
  int32_t strips, rows_per_strip; /* per-lane kernel */
  int32_t ctas, warps_per_cta, ctas_per_sm, sms;
  int32_t list_capacity; /* records per plane before the exact select takes over */
} SdnetSchedule;
int sdnet_decode_schedule(const SdnetDecodeParams* params, SdnetSchedule* out);

/* Profiling variant (bench.py's roofline leg): same work, but records CUDA events between the
 * three kernels on `stream`, WAITS for completion and returns the device time of each kernel in
 * milliseconds: kernel_ms[0] = peaks, [1] = exact-select, [2] = tail.  Synchronous by design. */
int sdnet_decode_launch_timed(const SdnetDecodeParams* params, void* stream, float* kernel_ms);

/* clamp(sigmoid(x), 1e-6, 1-1e-6) of a (B, C, H, W) view into a contiguous fp32 tensor:
 * the `anchor_hm_sig` / `part_hm_sig` metadata maps (decoders.py:44,60,163-164). */
int sdnet_activate_launch(const SdnetTensor4* in, int dtype, int B, int C, int H, int W, float* out, void* stream);

/* nms(clamped_sigmoid(x)) of a (B, C, H, W) view into a contiguous fp32 tensor: the score where it equals
 * the maximum score of its (2 radius + 1)^2 window, 0 elsewhere -- the reference's RawDecoder
 * (src/sdnet/cli/convert_coreml.py:12-19; utils.py:355-361,441-443), i.e. the heat maps CoreMLDecoder
 * expects (decoders.py:211,226; SDNET_FLAG_PRE_ACTIVATED). */
int sdnet_suppress_launch(const SdnetTensor4* in, int dtype, int B, int C, int H, int W, int radius, float* out, void* stream);

/* Same, written into a strided fp32 (B, C, H, W) view (`out->stride_w` == 1, `out->stride_h` >= W): the first
 * channels of a pre-allocated (B, C + 4, H, W) tensor, so that "network output with its heat maps baked" -- the
 * reference's RawDecoder / CoreMLModel (src/sdnet/cli/convert_coreml.py:12-29) -- needs no torch.cat pass. */
int sdnet_suppress_into_launch(const SdnetTensor4* in, int dtype, int B, int C, int H, int W, int radius, const SdnetTensor4* out,
                               void* stream);

/* The consumer side of the fused gather's completion flags: enqueue, on `stream`, a wait until flags[j] >= value for
 * every j < world (acquire loads, system scope; one tiny CTA that spins).  Everything enqueued on `stream` after it
 * sees every rank's detections of decode number `value`.  Replaces the all-gather's implicit synchronisation. */
int sdnet_gather_wait_launch(const uint32_t* flags, int world, uint32_t value, void* stream);

/* Same as sdnet_decode_launch but the four input tensors live in (pinned) HOST memory: the heat-map
 * planes are copied to `staging` (device, >= B*(M+N)*H*W*elem bytes, 256-byte aligned) with one strided
 * cudaMemcpy2DAsync per heat tensor on `stream`, then the three kernels run on `stream`;
 * offsets/embeddings stay on the host and are only touched, through the unified address space, at the
 * K + 2P selected peaks per image.  Outputs stay on the device.  Requirements: dense rows
 * (stride_h == W) and dense channels (stride_c == H*W, free when the tensor has one channel); any
 * batch stride.  Everything is enqueued on `stream`; no internal stream, no synchronisation.
 * To overlap the copy of batch i+1 with the kernels of batch i, call it for consecutive batches on two
 * streams with two staging buffers (what bench.py's e2e leg does). */
int sdnet_decode_host_launch(const SdnetDecodeParams* params, void* staging, size_t staging_bytes, void* stream);

/* ---- the step after the path: location matching of the reference evaluator, on the packed detections ----
 * Evaluator.eval_anchor (src/sdnet/model/evaluator.py:244-284) and Evaluator.eval_part (:286-334) for a
 * whole batch: per image and label, detections in score order each look for their nearest ground truth
 * of the same label (first minimum); a detection is a true positive if that distance is below the
 * image's threshold and no earlier detection claimed the same ground truth.  All arithmetic is the
 * reference's Python-float (double) arithmetic: x = (double)x_f32 * sx * rx, dist = hypot(dx, dy). */
#define SDNET_MAX_GT 1024
typedef struct SdnetMatchParams {
  uint32_t struct_size; /* sizeof(SdnetMatchParams) */
  int32_t B, M, N, K, P; /* images, anchor classes, part kinds, anchor slots, part slots */
  int32_t max_gt_anchors, max_gt_parts; /* row lengths of the ground-truth arrays, <= SDNET_MAX_GT */
  double conf;   /* objects: score > conf (decoders.py:116); raw parts: not score < conf (decoders.py:153) */
  double sx, sy; /* heat-map -> network-input scale, in/out (decoders.py:139) */
  const float* anchor_out;     /* (B, K, 4) as written by sdnet_decode_launch */
  const float* part_out;       /* (B, P, 6) */
  const double* image_scale;   /* (B, 4): img_w/args.width, img_h/args.height, min(img_size)*dist_threshold, min(img_size)
                                  (evaluator.py:245-250) */
  const double* gt_anchors;    /* (B, max_gt_anchors, 3): x, y, label index, network-input frame, annotation order */
  const int32_t* n_gt_anchors; /* (B) */
  const double* gt_parts;      /* (B, max_gt_parts, 3): every part of every ground-truth object, annotation order */
  const int32_t* n_gt_parts;   /* (B) */
  int32_t* anchor_stats;       /* (B, M, 3): ndet, npos, tp */
  int32_t* part_stats;         /* (B, N, 3) */
  double* anchor_acc;          /* (B, K): min_dist / min(img_size) of the true positives, NaN elsewhere (slot = score order) */
  double* part_acc;            /* (B, P) */
} SdnetMatchParams;

int sdnet_match_launch(const SdnetMatchParams* params, void* stream);

/* Object-level matching of the reference evaluator on the packed detections: Evaluator.eval_csi with
 * Evaluator.compute_csi (src/sdnet/model/evaluator.py:380-420, 539-581) and Evaluator.eval_classif (:429-474),
 * what `evaluate` accumulates with eval_csi=True, eval_classif=True (src/sdnet/cli/evaluate.py:43-45).
 * A predicted object is an anchor slot with score > conf plus the part slots `assign` groups onto it
 * (decoders.py:108-137); ground truth = the annotation's objects and, in object order, their parts. */
typedef struct SdnetObjectMatchParams {
  uint32_t struct_size; /* sizeof(SdnetObjectMatchParams) */
  int32_t B, M, N, K, P;
  int32_t max_gt_objects, max_gt_parts; /* row lengths of the ground-truth arrays, <= SDNET_MAX_GT */
  double conf;          /* objects: score > conf (decoders.py:116) */
  double sx, sy;        /* heat-map -> network-input scale, in/out (decoders.py:139) */
  double csi_threshold; /* args.csi_threshold (evaluator.py:414) */
  const float* anchor_out;     /* (B, K, 4) as written by sdnet_decode_launch */
  const float* part_out;       /* (B, P, 6) */
  const int32_t* assign;       /* (B, P) */
  const double* image_scale;   /* (B, 4): as in SdnetMatchParams */
  const double* gt_objects;    /* (B, max_gt_objects, 3): anchor x, y, class index; annotation order */
  const int32_t* n_gt_objects; /* (B) */
  const double* gt_parts;      /* (B, max_gt_parts, 3): x, y, kind index; grouped by object, object order */
  const int32_t* gt_part_owner;/* (B, max_gt_parts): index of the object each part belongs to (non-decreasing);
                                  at most 64 parts per object */
  const int32_t* n_gt_parts;   /* (B) */
  const int32_t* cls_group;    /* (M): 0 / 1 for the classes named "bean" / "maize" (the reference's hard-coded
                                  classification labels, evaluator.py:422-427), -1 for every other class */
  int32_t* csi_stats;          /* (B, M, 3): ndet, npos, tp per class */
  double* csi_acc;             /* (B, K): the CSI of the true positives, NaN elsewhere (slot = score order) */
  int32_t* classif_stats;      /* (B, 20, 3): ndet, npos, tp for "bean_0".."bean_9", "maize_0".."maize_9" */
  double* classif_acc;         /* (B, K): distance / min(img_size) of the true positives, NaN elsewhere */
  int32_t* pred_parts;         /* (B, K): number of parts of each emitted object, -1 for slots not emitted */
} SdnetObjectMatchParams;

int sdnet_match_objects_launch(const SdnetObjectMatchParams* params, void* stream);

/* Threshold sweep of the evaluator: for each of T confidence thresholds, and for each of G grouping distances
 * (gates), what sdnet_match_launch and (with SDNET_SWEEP_OBJECTS) sdnet_match_objects_launch compute on a decode at
 * that threshold and gate, from ONE decode.  anchor_out / part_out do not depend on the decoder's conf or gate; only
 * the grouping does, so it is redone per threshold: anchors with score > conf_group[t] keep (x, y), the others sit at
 * (+1e6, +1e6); parts with score > conf_group[t] keep their origin, the others sit at (-1e6, -1e6); every part goes to
 * the first anchor at the smallest fp32 distance sqrt(dx*dx + dy*dy) (each step rounded, no FMA), if that distance is
 * < the gate (decoders.py:80-100, the full P x K search).  The search is done once per threshold; only the final
 * compare is taken per gate.  The `assign` and `counts` the decode wrote are not read, so the decode's own conf and
 * gate do not matter; it must have grouped (part_out's origins are needed).
 * G = 0: one gate, dist_abs_f32, and every output is indexed [image][threshold] (as with ABI version 9).
 * G >= 1: the gates are dist_abs_grid[0 .. G-1].  The location outputs (anchor_*, part_*) do not depend on the gate
 * and stay indexed [image][threshold]; the object outputs (csi_*, classif_*, pred_parts) and assign_out are indexed
 * [image][threshold][gate], row (b*T + t)*G + g. */
#define SDNET_MAX_GATES 64
#define SDNET_MAX_THRESHOLDS 256
#define SDNET_SWEEP_OBJECTS 1u /* SdnetSweepParams.flags: also the object-level (CSI, classification) tables */
typedef struct SdnetSweepParams {
  uint32_t struct_size; /* sizeof(SdnetSweepParams) */
  int32_t B, M, N, K, P;
  int32_t T;            /* thresholds, 1 .. SDNET_MAX_THRESHOLDS */
  int32_t max_gt_objects, max_gt_parts; /* row lengths of the ground-truth arrays, <= SDNET_MAX_GT */
  uint32_t flags;       /* SDNET_SWEEP_* */
  float dist_abs_f32;   /* the decoder's gate: (float)(dist_thresh * min(W, H)) (decoders.py:100); read when G = 0 */
  double sx, sy;        /* heat-map -> network-input scale, in/out (decoders.py:139) */
  double csi_threshold; /* args.csi_threshold (evaluator.py:414); read with SDNET_SWEEP_OBJECTS */
  const double* conf;          /* (T): the evaluator's thresholds (objects: score > conf; raw parts: not score < conf) */
  const float* conf_group;     /* (T): the same thresholds rounded to the heat maps' dtype, for the grouping's score > conf */
  const float* anchor_out;     /* (B, K, 4) as written by sdnet_decode_launch */
  const float* part_out;       /* (B, P, 6) */
  const double* image_scale;   /* (B, 4): as in SdnetMatchParams */
  const double* gt_objects;    /* (B, max_gt_objects, 3): anchor x, y, class index; annotation order */
  const int32_t* n_gt_objects; /* (B) */
  const double* gt_parts;      /* (B, max_gt_parts, 3): x, y, kind index; grouped by object, object order */
  const int32_t* gt_part_owner;/* (B, max_gt_parts): as in SdnetObjectMatchParams; read with SDNET_SWEEP_OBJECTS */
  const int32_t* n_gt_parts;   /* (B) */
  const int32_t* cls_group;    /* (M): as in SdnetObjectMatchParams; read with SDNET_SWEEP_OBJECTS */
  int32_t* anchor_stats;       /* (B, T, M, 3): ndet, npos, tp */
  int32_t* part_stats;         /* (B, T, N, 3) */
  double* anchor_acc;          /* (B, T, K): as SdnetMatchParams.anchor_acc */
  double* part_acc;            /* (B, T, P) */
  int32_t* csi_stats;          /* (B, T, M, 3)   } SDNET_SWEEP_OBJECTS only: */
  double* csi_acc;             /* (B, T, K)      } as the fields of the same name */
  int32_t* classif_stats;      /* (B, T, 20, 3)  } in SdnetObjectMatchParams; */
  double* classif_acc;         /* (B, T, K)      } (B, T, G, ...) with G >= 1 */
  int32_t* pred_parts;         /* (B, T, K)      } */
  int32_t* assign_out;         /* optional (B, T, P), (B, T, G, P) with G >= 1: the regrouped assignment (NULL to skip) */
  int32_t G;                   /* gates, 0 .. SDNET_MAX_GATES; 0 = one gate, dist_abs_f32 */
  const float* dist_abs_grid;  /* (G): the gates, each (float)(dist_thresh * min(W, H)) as dist_abs_f32; read when G >= 1 */
} SdnetSweepParams;

int sdnet_sweep_launch(const SdnetSweepParams* params, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SDNET_DECODE_H_ */
