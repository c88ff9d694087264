// sweep.cuh -- sdnet_sweep_kernel: the evaluator at T confidence thresholds from one decode.
#pragma once

namespace {

// ---------------------------------------------------------------------------------------------
// One CTA per (image, threshold).  anchor_out / part_out do not depend on the decoder's conf (the tail kernel's
// `score > conf` only feeds its grouping and its counts), so a decode at any threshold holds every other
// threshold's detections; what changes is the grouping, redone here:
//   1. regroup at conf_group[t]: masked anchors at (+1e6, +1e6), masked part origins at (-1e6, -1e6)
//      (decoders.py:80-86), every part's first anchor at the smallest fp32 distance (decoders.py:88-99).  The plain
//      P x K search in slot order: no near-field restriction and no square-then-root shortcut as in tail.cuh, so it
//      holds for any coordinate and any gate.  The search does not depend on the gate: its slot and distance are
//      kept, and only the final `distance < gate` (decoders.py:100) is taken per gate in phase 3;
//   2. location matching at conf[t] (match_pass, as sdnet_match_kernel), which never reads the grouping: once per
//      (image, threshold), whatever the number of gates;
//   3. per gate g: the assignment at dist_abs_grid[g] (dist_abs_f32 when G = 0) and, with SDNET_SWEEP_OBJECTS, object
//      matching at conf[t] on it (match_objects, as sdnet_match_objects_kernel) into row (b*T + t)*G + g.
// The nearest slots, their distances and the gated assignment live at the front of the dynamic shared memory (12 B
// per part slot); the three phases share the rest.
// ---------------------------------------------------------------------------------------------
constexpr float kSweepFar = 1e6f;  // decoders.py:80-86 (kFar in tail.cuh)

// Dynamic shared memory of one sweep CTA: nearest slots, distances, assignment, then the largest of the three
// phases' scratch.
inline size_t sweep_smem_bytes(const SdnetSweepParams& p) {
  const size_t K = (size_t)p.K, P = (size_t)p.P;
  const size_t G = (size_t)(p.max_gt_objects > p.max_gt_parts ? p.max_gt_objects : p.max_gt_parts);
  const size_t S = K > P ? K : P;
  const size_t regroup = 8 * K;  // masked anchor positions
  // match_pass's arrays; its label counters take every class index a decode can emit (it does not check a slot's
  // class against the caller's M / N), like sdnet_match_kernel's static array
  const size_t location = 8 * (2 * G + S) + 4 * (2 * G + S + 3 * SDNET_MAX_CHANNELS);
  const size_t objects = (p.flags & SDNET_SWEEP_OBJECTS)
                             ? match_objects_smem_bytes(p.max_gt_objects, p.max_gt_parts, p.K, p.P, p.M) : 0;
  size_t scratch = regroup > location ? regroup : location;
  if (objects > scratch) scratch = objects;
  return (12 * P + 15) / 16 * 16 + scratch;
}

__global__ void __launch_bounds__(kMatchThreads) sdnet_sweep_kernel(const SdnetSweepParams p) {
  extern __shared__ __align__(16) unsigned char sweep_smem[];
  const int b = blockIdx.x / p.T, t = blockIdx.x - b * p.T;
  const size_t row = (size_t)b * p.T + t;
  const int K = p.K, P = p.P, tid = threadIdx.x, nt = blockDim.x;
  const int n_gates = p.G > 0 ? p.G : 1;
  int* s_arg = reinterpret_cast<int*>(sweep_smem);
  float* s_best = reinterpret_cast<float*>(s_arg + P);
  int* s_assign = reinterpret_cast<int*>(s_best + P);
  unsigned char* scratch = sweep_smem + ((size_t)12 * P + 15) / 16 * 16;
  const float* A = p.anchor_out + (size_t)b * K * 4;
  const float* Q = p.part_out + (size_t)b * P * 6;

  // ---- 1. nearest anchor of every part at conf_group[t]
  {
    const float cg = p.conf_group[t];
    float2* s_apos = reinterpret_cast<float2*>(scratch);
    for (int a = tid; a < K; a += nt) {
      const bool valid = A[4 * a + 2] > cg;
      s_apos[a] = valid ? make_float2(A[4 * a], A[4 * a + 1]) : make_float2(kSweepFar, kSweepFar);
    }
    __syncthreads();
    for (int q = tid; q < P; q += nt) {
      const bool valid = Q[6 * q + 2] > cg;
      const float ox = valid ? Q[6 * q + 4] : -kSweepFar, oy = valid ? Q[6 * q + 5] : -kSweepFar;
      float best = CUDART_INF_F;
      int arg = -1;
      for (int a = 0; a < K; ++a) {
        const float2 ap = s_apos[a];
        const float dx = __fsub_rn(ox, ap.x), dy = __fsub_rn(oy, ap.y);
        const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
        if (d < best) { best = d; arg = a; }
      }
      s_arg[q] = arg;
      s_best[q] = best;
    }
    __syncthreads();
  }

  // ---- 2. location matching at conf[t] (match_pass's arrays aliased into the scratch)
  const double conf = p.conf[t];
  const double* scale = p.image_scale + 4 * (size_t)b;
  {
    const int G = p.max_gt_objects > p.max_gt_parts ? p.max_gt_objects : p.max_gt_parts;
    const int S = K > P ? K : P;
    double* d = reinterpret_cast<double*>(scratch);
    double* s_gx = d; d += G;
    double* s_gy = d; d += G;
    double* s_dist = d; d += S;
    int* i = reinterpret_cast<int*>(d);
    int* s_glab = i; i += G;
    int* s_winner = i; i += G;
    int* s_jmin = i; i += S;
    int* s_stats = i;
    match_pass(A, 4, K, p.M, true, conf, p.sx, p.sy, scale, p.gt_objects + (size_t)b * p.max_gt_objects * 3,
               min(p.n_gt_objects[b], p.max_gt_objects), p.anchor_stats + row * p.M * 3, p.anchor_acc + row * K, s_gx,
               s_gy, s_glab, s_winner, s_jmin, s_dist, s_stats);
    match_pass(Q, 6, P, p.N, false, conf, p.sx, p.sy, scale, p.gt_parts + (size_t)b * p.max_gt_parts * 3,
               min(p.n_gt_parts[b], p.max_gt_parts), p.part_stats + row * p.N * 3, p.part_acc + row * P, s_gx, s_gy,
               s_glab, s_winner, s_jmin, s_dist, s_stats);
  }

  // ---- 3. per gate: the gated assignment, then object matching at conf[t] on it (match_pass ends with a barrier)
  const bool objects = (p.flags & SDNET_SWEEP_OBJECTS) != 0;
  SdnetObjectMatchParams op;
  if (objects) {
    op.K = K; op.P = P; op.M = p.M; op.N = p.N; op.B = p.B;
    op.max_gt_objects = p.max_gt_objects; op.max_gt_parts = p.max_gt_parts;
    op.conf = conf; op.sx = p.sx; op.sy = p.sy; op.csi_threshold = p.csi_threshold;
    op.anchor_out = p.anchor_out; op.part_out = p.part_out; op.assign = nullptr;
    op.image_scale = p.image_scale;
    op.gt_objects = p.gt_objects; op.n_gt_objects = p.n_gt_objects;
    op.gt_parts = p.gt_parts; op.gt_part_owner = p.gt_part_owner; op.n_gt_parts = p.n_gt_parts;
    op.cls_group = p.cls_group;
    op.csi_stats = p.csi_stats; op.csi_acc = p.csi_acc;
    op.classif_stats = p.classif_stats; op.classif_acc = p.classif_acc; op.pred_parts = p.pred_parts;
  }
  for (int g = 0; g < n_gates; ++g) {
    const float gate = p.G > 0 ? p.dist_abs_grid[g] : p.dist_abs_f32;
    const size_t grow = row * n_gates + g;
    for (int q = tid; q < P; q += nt) {
      const int arg = s_arg[q];
      const int slot = (arg >= 0 && s_best[q] < gate) ? arg : -1;
      s_assign[q] = slot;
      if (p.assign_out) p.assign_out[grow * P + q] = slot;
    }
    if (objects) {
      __syncthreads();
      match_objects(op, b, grow, s_assign, scratch);
      __syncthreads();  // the next gate overwrites the assignment match_objects reads
    }
  }
}

}  // namespace
