// match.cuh -- sdnet_match_kernel: the reference evaluator's nearest-ground-truth matching on the packed detections.
#pragma once

namespace {

// ---------------------------------------------------------------------------------------------
// evaluator matching (the step after the path): reference Evaluator.eval_anchor / eval_part,
// src/sdnet/model/evaluator.py:244-334, on the packed detections.  One CTA per image; the greedy
// "first detection in score order that claims a ground truth wins it" loop is order-free once every
// detection knows its nearest ground truth: the winner of ground truth j is the smallest slot index
// among the detections whose nearest is j and whose distance is under the threshold (atomicMin).
// Arithmetic is double throughout, like the reference's Python floats.
// ---------------------------------------------------------------------------------------------
constexpr int kMatchThreads = 256;

__device__ void match_pass(const float* __restrict__ out, int row_len, int slots, int n_classes, bool strict_gt,
                           double conf, double sx, double sy, const double* __restrict__ scale,
                           const double* __restrict__ gt, int n_gt, int* __restrict__ stats_out,
                           double* __restrict__ acc_out, double* s_gx, double* s_gy, int* s_glab, int* s_winner,
                           int* s_jmin, double* s_dist, int* s_stats) {
  const double rx = scale[0], ry = scale[1], thresh = scale[2], norm = scale[3];
  for (int j = threadIdx.x; j < n_gt; j += blockDim.x) {
    s_gx[j] = gt[3 * j + 0] * rx;  // annotation.resized(...): evaluator.py:247
    s_gy[j] = gt[3 * j + 1] * ry;
    s_glab[j] = (int)gt[3 * j + 2];
    s_winner[j] = 0x7fffffff;
  }
  for (int i = threadIdx.x; i < 3 * n_classes; i += blockDim.x) s_stats[i] = 0;
  __syncthreads();
  for (int j = threadIdx.x; j < n_gt; j += blockDim.x)
    if (s_glab[j] >= 0 && s_glab[j] < n_classes) atomicAdd(&s_stats[3 * s_glab[j] + 1], 1);  // npos
  for (int i = threadIdx.x; i < slots; i += blockDim.x) {
    const float* row = out + (size_t)i * row_len;
    const double score = (double)row[2];
    const bool det = strict_gt ? (score > conf) : !(score < conf);
    const int lab = (int)row[3];
    int jmin = -1;
    double best = 1.7976931348623157e308;  // sys.float_info.max
    if (det) {
      atomicAdd(&s_stats[3 * lab + 0], 1);  // ndet
      const double px = ((double)row[0] * sx) * rx, py = ((double)row[1] * sy) * ry;  // decoders.py:139 then evaluator.py:248
      for (int j = 0; j < n_gt; ++j) {
        if (s_glab[j] != lab) continue;
        const double d = hypot(px - s_gx[j], py - s_gy[j]);  // np.hypot, utils.py:31-32
        if (d < best) { best = d; jmin = j; }
      }
      if (jmin >= 0 && best < thresh) atomicMin(&s_winner[jmin], i);
    }
    s_jmin[i] = det ? jmin : -1;
    s_dist[i] = best;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < slots; i += blockDim.x) {
    const int jmin = s_jmin[i];
    const bool tp = jmin >= 0 && s_dist[i] < thresh && s_winner[jmin] == i;
    acc_out[i] = tp ? s_dist[i] / norm : __longlong_as_double(0x7ff8000000000000ll);
    if (tp) atomicAdd(&s_stats[3 * (int)out[(size_t)i * row_len + 3] + 2], 1);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * n_classes; i += blockDim.x) stats_out[i] = s_stats[i];
  __syncthreads();
}

__global__ void __launch_bounds__(kMatchThreads) sdnet_match_kernel(const SdnetMatchParams p) {
  __shared__ double s_gx[SDNET_MAX_GT], s_gy[SDNET_MAX_GT], s_dist[SDNET_MAX_TOPK];
  __shared__ int s_glab[SDNET_MAX_GT], s_winner[SDNET_MAX_GT], s_jmin[SDNET_MAX_TOPK], s_stats[3 * SDNET_MAX_CHANNELS];
  const int b = blockIdx.x;
  const double* scale = p.image_scale + 4 * (size_t)b;
  match_pass(p.anchor_out + (size_t)b * p.K * 4, 4, p.K, p.M, true, p.conf, p.sx, p.sy, scale,
             p.gt_anchors + (size_t)b * p.max_gt_anchors * 3, min(p.n_gt_anchors[b], p.max_gt_anchors),
             p.anchor_stats + (size_t)b * p.M * 3, p.anchor_acc + (size_t)b * p.K, s_gx, s_gy, s_glab, s_winner, s_jmin,
             s_dist, s_stats);
  match_pass(p.part_out + (size_t)b * p.P * 6, 6, p.P, p.N, false, p.conf, p.sx, p.sy, scale,
             p.gt_parts + (size_t)b * p.max_gt_parts * 3, min(p.n_gt_parts[b], p.max_gt_parts),
             p.part_stats + (size_t)b * p.N * 3, p.part_acc + (size_t)b * p.P, s_gx, s_gy, s_glab, s_winner, s_jmin, s_dist,
             s_stats);
}


// ---------------------------------------------------------------------------------------------
// object-level matching: reference Evaluator.eval_csi / compute_csi (evaluator.py:380-420, 539-581) and
// Evaluator.eval_classif (:429-474) on the packed detections.  A predicted object = an anchor slot with
// score > conf plus the part slots assigned to it (decoders.py:108-137); one CTA per image, one thread per
// predicted object.
//   classification: objects are keyed by (class, number of parts) -- the reference's hard-coded "bean_0" ..
//   "maize_9" labels, here cls_group[class] * 10 + parts -- and matched to the nearest ground truth of the same key
//   (first minimum, true positive if distance <= threshold and the ground truth is still free);
//   CSI: per class, every prediction takes the ground truth with the highest critical success index
//   tp / (npos + ndet - tp) of the (anchor + parts) pair (first maximum, strictly above 0), true positive if
//   that index reaches csi_threshold and the ground truth is still free.
// "Still free" is resolved like in match_pass: among the predictions that claim a ground truth, the one with
// the smallest slot (= highest score; the reference's sort is stable) wins.  Doubles throughout.
// ---------------------------------------------------------------------------------------------
struct ObjScratch {
  double *gx, *gy, *px, *py, *qx, *qy, *hx, *hy, *best;  // ground-truth anchors, predicted anchors, predicted parts, ground-truth parts
  int *glab, *gstart, *win, *npp, *pstart, *plist, *qkind, *hkind, *jbest, *stats;
};

__device__ __forceinline__ double csi_of_pair(const ObjScratch& s, int k, int j, double thresh) {
  // compute_csi (evaluator.py:539-581) for prediction slot k and ground truth j of the same class
  int tp = hypot(s.px[k] - s.gx[j], s.py[k] - s.gy[j]) < thresh ? 1 : 0;
  const int p0 = s.pstart[k], p1 = s.pstart[k + 1], h0 = s.gstart[j], h1 = s.gstart[j + 1];
  unsigned long long visited = 0ull;  // over the ground truth's parts (at most 64 per object, checked on the host)
  for (int a = p0; a < p1; ++a) {     // predicted parts in slot (= score) order
    const int q = s.plist[a];
    double best = 1.7976931348623157e308;
    int jmin = -1;
    for (int h = h0; h < h1; ++h) {
      if (s.hkind[h] != s.qkind[q]) continue;
      const double d = hypot(s.qx[q] - s.hx[h], s.qy[q] - s.hy[h]);
      if (d < best) { best = d; jmin = h; }
    }
    if (jmin >= 0 && best < thresh && !((visited >> (jmin - h0)) & 1ull)) {
      visited |= 1ull << (jmin - h0);
      ++tp;
    }
  }
  const int npos = 1 + (h1 - h0), ndet = 1 + (p1 - p0);
  return (double)tp / (double)(npos + ndet - tp);
}

// Dynamic shared memory match_objects needs (16-byte aligned base).
inline size_t match_objects_smem_bytes(int max_gt_objects, int max_gt_parts, int K, int P, int M) {
  const size_t Go = (size_t)max_gt_objects, Gp = (size_t)max_gt_parts, k = (size_t)K, q = (size_t)P;
  const size_t n_stats = 3 * (size_t)(M > 20 ? M : 20);
  return 8 * (2 * Go + 3 * k + 2 * q + 2 * Gp) + 4 * (3 * Go + 1 + 3 * k + 1 + 2 * q + Gp + n_stats) + 16;
}

// The object-level matching of image b with the part assignment `asg` (P entries; shared or global memory), its
// results stored in output row `row` of p's outputs.  `obj_smem` holds match_objects_smem_bytes.
__device__ __forceinline__ void match_objects(const SdnetObjectMatchParams& p, int b, size_t row, const int* asg,
                                              unsigned char* obj_smem) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const int K = p.K, P = p.P, Go = p.max_gt_objects, Gp = p.max_gt_parts;
  ObjScratch s;
  {
    double* d = reinterpret_cast<double*>(obj_smem);
    s.gx = d; d += Go; s.gy = d; d += Go; s.px = d; d += K; s.py = d; d += K; s.qx = d; d += P; s.qy = d; d += P;
    s.hx = d; d += Gp; s.hy = d; d += Gp; s.best = d; d += K;
    int* i = reinterpret_cast<int*>(d);
    s.glab = i; i += Go; s.gstart = i; i += Go + 1; s.win = i; i += Go; s.npp = i; i += K; s.pstart = i; i += K + 1;
    s.plist = i; i += P; s.qkind = i; i += P; s.hkind = i; i += Gp; s.jbest = i; i += K; s.stats = i;
  }
  const int n_stats = 3 * (p.M > 20 ? p.M : 20);
  const double* scale = p.image_scale + 4 * (size_t)b;
  const double rx = scale[0], ry = scale[1], thresh = scale[2], norm = scale[3];
  const float* A = p.anchor_out + (size_t)b * K * 4;
  const float* Q = p.part_out + (size_t)b * P * 6;
  const int n_go = min(p.n_gt_objects[b], Go), n_gp = min(p.n_gt_parts[b], Gp);
  const double* G = p.gt_objects + (size_t)b * Go * 3;
  const double* Hh = p.gt_parts + (size_t)b * Gp * 3;
  const int* owner = p.gt_part_owner + (size_t)b * Gp;

  // ---- stage everything in the evaluator's frame (annotation.resized / prediction.resized: evaluator.py:381-383)
  for (int j = tid; j < n_go; j += nt) {
    s.gx[j] = G[3 * j] * rx; s.gy[j] = G[3 * j + 1] * ry; s.glab[j] = (int)G[3 * j + 2];
  }
  for (int h = tid; h < n_gp; h += nt) {
    s.hx[h] = Hh[3 * h] * rx; s.hy[h] = Hh[3 * h + 1] * ry; s.hkind[h] = (int)Hh[3 * h + 2];
  }
  for (int k = tid; k < K; k += nt) {
    s.px[k] = ((double)A[4 * k] * p.sx) * rx; s.py[k] = ((double)A[4 * k + 1] * p.sy) * ry;
    s.npp[k] = 0;
  }
  for (int q = tid; q < P; q += nt) {
    s.qx[q] = ((double)Q[6 * q] * p.sx) * rx; s.qy[q] = ((double)Q[6 * q + 1] * p.sy) * ry; s.qkind[q] = (int)Q[6 * q + 3];
  }
  for (int j = tid; j <= n_go; j += nt) s.gstart[j] = 0;
  __syncthreads();
  // parts per ground-truth object (the parts array is ordered by object) and per emitted prediction
  for (int h = tid; h < n_gp; h += nt) atomicAdd(&s.gstart[owner[h] + 1], 1);
  for (int q = tid; q < P; q += nt) {
    const int k = asg[q];
    if (k >= 0 && k < K && (double)A[4 * k + 2] > p.conf) atomicAdd(&s.npp[k], 1);
  }
  __syncthreads();
  if (tid == 0) {  // prefix sums (at most ~1000 entries each)
    for (int j = 0; j < n_go; ++j) s.gstart[j + 1] += s.gstart[j];
    int acc = 0;
    for (int k = 0; k < K; ++k) { s.pstart[k] = acc; acc += s.npp[k]; }
    s.pstart[K] = acc;
    // part slots of every prediction, in slot order
    for (int k = 0; k < K; ++k) s.npp[k] = 0;
    for (int q = 0; q < P; ++q) {
      const int k = asg[q];
      if (k >= 0 && k < K && (double)A[4 * k + 2] > p.conf) s.plist[s.pstart[k] + s.npp[k]++] = q;
    }
  }
  __syncthreads();

  for (int pass = 0; pass < 2; ++pass) {  // 0: classification, 1: CSI
    const int n_lab = pass == 0 ? 20 : p.M;
    for (int i = tid; i < n_stats; i += nt) s.stats[i] = 0;
    for (int j = tid; j < n_go; j += nt) s.win[j] = 0x7fffffff;
    __syncthreads();
    auto key_of = [&](int cls, int nparts) -> int {  // label index of an object in this pass; -1 = counted nowhere
      if (pass == 1) return cls >= 0 && cls < p.M ? cls : -1;
      if (cls < 0 || cls >= p.M || nparts > 9) return -1;
      const int g = p.cls_group[cls];
      return g >= 0 && g < 2 ? g * 10 + nparts : -1;
    };
    for (int j = tid; j < n_go; j += nt) {
      const int key = key_of(s.glab[j], s.gstart[j + 1] - s.gstart[j]);
      if (key >= 0) atomicAdd(&s.stats[3 * key + 1], 1);  // npos
    }
    for (int k = tid; k < K; k += nt) {
      int jb = -1;
      double best = pass == 0 ? 1.7976931348623157e308 : 0.0;
      const bool det = (double)A[4 * k + 2] > p.conf;
      const int key = det ? key_of((int)A[4 * k + 3], s.npp[k]) : -1;
      if (key >= 0) {
        atomicAdd(&s.stats[3 * key + 0], 1);  // ndet
        for (int j = 0; j < n_go; ++j) {
          if (key_of(s.glab[j], s.gstart[j + 1] - s.gstart[j]) != key) continue;
          if (pass == 0) {
            const double d = hypot(s.px[k] - s.gx[j], s.py[k] - s.gy[j]);
            if (d < best) { best = d; jb = j; }
          } else {
            const double c = csi_of_pair(s, k, j, thresh);
            if (c > best) { best = c; jb = j; }
          }
        }
        const bool claim = jb >= 0 && (pass == 0 ? best <= thresh : best >= p.csi_threshold);
        if (claim) atomicMin(&s.win[jb], k);
        else jb = -1;
      }
      s.jbest[k] = jb;
      s.best[k] = best;
    }
    __syncthreads();
    double* acc_out = (pass == 0 ? p.classif_acc : p.csi_acc) + row * K;
    for (int k = tid; k < K; k += nt) {
      const int jb = s.jbest[k];
      const bool tp = jb >= 0 && s.win[jb] == k;
      acc_out[k] = tp ? (pass == 0 ? s.best[k] / norm : s.best[k]) : __longlong_as_double(0x7ff8000000000000ll);
      if (tp) atomicAdd(&s.stats[3 * key_of((int)A[4 * k + 3], s.npp[k]) + 2], 1);
    }
    __syncthreads();
    int* stats_out = pass == 0 ? p.classif_stats + row * 60 : p.csi_stats + row * p.M * 3;
    for (int i = tid; i < 3 * n_lab; i += nt) stats_out[i] = s.stats[i];
    if (pass == 0)
      for (int k = tid; k < K; k += nt) p.pred_parts[row * K + k] = (double)A[4 * k + 2] > p.conf ? s.npp[k] : -1;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kMatchThreads) sdnet_match_objects_kernel(const SdnetObjectMatchParams p) {
  extern __shared__ __align__(16) unsigned char obj_smem[];
  const int b = blockIdx.x;
  match_objects(p, b, (size_t)b, p.assign + (size_t)b * p.P, obj_smem);
}

}  // namespace
