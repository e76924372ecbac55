// Evaluation metrics on the device (SURVEY.md 8f N2), fed by the batched matching of match.cu:
//
//   confusion_kernel        one CTA per image: the confusion matrix of PredictionLabelMatch.convert_background_errors,
//                           read straight from the matched / missed / extra rows (shared histogram, one global atomic per
//                           bin); also checks every label class of the image
//   coco_match_kernel       one CTA per image: COCOeval.evaluateImg (bbox, no crowd, area "all") for every class: the
//                           detections ranked by score within their class, then one warp per (class, IoU threshold) walks
//                           the first 100 and takes ground truths greedily; one record per kept detection
//   coco_accumulate_kernel  one CTA per (class, IoU threshold, maxDet): COCOeval.accumulate over the score-sorted records
//   score_format_kernel     torchmetrics' format rule of one update: does any class value lie outside [0, 1]
//   score_rows_kernel       one CTA per image: the score rows of convert_background_errors (softmaxed or not) with their
//                           targets, NaN rows flagged, confidence / accuracy binned into per-CTA partials;
//                           score_bins_reduce_kernel sums the partials in image order
//   roc_keys_kernel,        compute(): class-major keys of every score; after a sort, one CTA per class walks its segment
//   roc_curve_kernel        (block scans of positives and of distinct-score boundaries) and writes the ROC curve and AUC
//
// tools/coco_eval_np.py and tools/roc_ece_np.py restate the same algorithms in numpy; the GPU tests compare against them
// bit for bit.
#include "common.cuh"

namespace yg {

constexpr int MET_MAX_CELLS = 16384;        // Sy*Sx limit, as the matching
constexpr int MET_MAX_CLASSES = 27;         // as format_preds
constexpr int COCO_MAX_DETS = 100;          // COCOeval maxDets[-1]
constexpr int CONF_THREADS = 256;
constexpr int COCO_MATCH_THREADS = 1024;
constexpr int COCO_ACC_THREADS = 512;

struct IouThrs { double t[YG_COCO_IOU_THRS]; };
struct RecThrs { double r[YG_COCO_REC_THRS]; };

// torch.argmax of the C class scores, with an appended 0 when with_zero (convert_background_errors adds a zero
// background column to every prediction row): first maximum, a NaN counts as the maximum
__device__ __forceinline__ int class_argmax(const float* __restrict__ v, int C, bool with_zero) {
  float best = v[0];
  int bi = 0;
  for (int k = 1; k < C; ++k) {
    const float x = v[k];
    if (x > best || (x != x && best == best)) { best = x; bi = k; }
  }
  if (with_zero && 0.f > best) bi = C;
  return bi;
}

// int(label[5]) when it lies in [0, C), else -1
__device__ __forceinline__ int label_class(float x, int C) { return (x > -1.f && x < (float)C) ? (int)x : -1; }

// fp32 score -> unsigned key whose ascending order is descending score
__device__ __forceinline__ unsigned score_desc_key(float s) {
  const unsigned u = __float_as_uint(s);
  return ~((u & 0x80000000u) ? ~u : (u | 0x80000000u));
}

// ---- confusion matrix ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CONF_THREADS) confusion_kernel(
    const float* __restrict__ out_preds, const float* __restrict__ out_labels, const float* __restrict__ missed,
    const float* __restrict__ extra, int C, int with_bg, const LsapDesc* __restrict__ desc, const long long* __restrict__ gather_off,
    const int* __restrict__ lsap_status, int* __restrict__ label_status, unsigned long long* __restrict__ confusion) {
  __shared__ int hist[(MET_MAX_CLASSES + 1) * (MET_MAX_CLASSES + 1)];
  __shared__ int bad;
  const int b = blockIdx.x, tid = threadIdx.x;
  if (lsap_status[b] != YG_LSAP_OK) {   // the gather wrote no rows for this image; the caller raises the solver's error
    if (tid == 0) label_status[b] = 0;
    return;
  }
  const int nb = C + (with_bg ? 1 : 0), D = 5 + C;
  for (int k = tid; k < nb * nb; k += CONF_THREADS) hist[k] = 0;
  if (tid == 0) bad = 0;
  __syncthreads();
  const LsapDesc d = desc[b];
  const int N = d.rows, M = d.cols, K = min(N, M);
  // matched pairs: (label class, argmax of the prediction row)
  for (int t = tid; t < K; t += CONF_THREADS) {
    const long long o = d.out_off + t;
    const int lc = label_class(out_labels[o * 6 + 5], C);
    if (lc < 0) { bad = 1; continue; }
    atomicAdd(&hist[lc * nb + class_argmax(out_preds + o * D + 5, C, with_bg)], 1);
  }
  // missed labels: (label class, background)
  for (int t = tid; t < N - K; t += CONF_THREADS) {
    const int lc = label_class(missed[(gather_off[2 * b] + t) * 6 + 5], C);
    if (lc < 0) { bad = 1; continue; }
    if (with_bg) atomicAdd(&hist[lc * nb + C], 1);
  }
  // extra predictions: (background, argmax of the prediction row)
  if (with_bg) {
    for (int t = tid; t < M - K; t += CONF_THREADS)
      atomicAdd(&hist[C * nb + class_argmax(extra + (gather_off[2 * b + 1] + t) * D + 5, C, true)], 1);
  }
  __syncthreads();
  for (int k = tid; k < nb * nb; k += CONF_THREADS)
    if (hist[k]) atomicAdd(&confusion[k], (unsigned long long)hist[k]);
  if (tid == 0) label_status[b] = bad;
}

// ---- COCO evaluateImg ------------------------------------------------------------------------------------------------
// dynamic shared memory: key[max_preds] (u64), gt_flags[(max_labels + 1) / 2] (u32: ground truth g owns bits
// 16 * (g & 1) + t), gt_cls[max_labels] (s8)
static size_t coco_match_smem(int max_labels, int max_preds) {
  return (size_t)max_preds * 8 + (size_t)((max_labels + 1) / 2) * 4 + (size_t)max_labels;
}

__global__ void __launch_bounds__(COCO_MATCH_THREADS) coco_match_kernel(
    const float* __restrict__ pred_rows, const float* __restrict__ label_rows, int cells, int C, const LsapDesc* __restrict__ desc,
    const long long* __restrict__ gather_off, long long image0, IouThrs thr, int* __restrict__ records, long long* __restrict__ keys,
    unsigned long long* __restrict__ gt_count) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ int det[MET_MAX_CLASSES * COCO_MAX_DETS];      // row index of the detection of rank r in class k
  __shared__ int det_pos[MET_MAX_CLASSES * COCO_MAX_DETS];  // its record position
  __shared__ unsigned det_mask[MET_MAX_CLASSES * COCO_MAX_DETS];
  __shared__ int n_det[MET_MAX_CLASSES], n_gt[MET_MAX_CLASSES];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const LsapDesc d = desc[b];
  const int N = d.rows, M = d.cols, D = 5 + C;
  const float* pb = pred_rows + (long long)b * cells * D;
  const float* lb = label_rows + (long long)b * cells * 6;
  unsigned long long* key = reinterpret_cast<unsigned long long*>(smem);
  unsigned* gt_flags = reinterpret_cast<unsigned*>(key + M);
  signed char* gt_cls = reinterpret_cast<signed char*>(gt_flags + (N + 1) / 2);
  // records of image b start at prefix(min(N, M)) + prefix(M - min(N, M)) = prefix(M): the kept rows of the batch
  const long long rec0 = d.out_off + gather_off[2 * b + 1];

  for (int k = tid; k < C; k += COCO_MATCH_THREADS) { n_det[k] = 0; n_gt[k] = 0; }
  for (int k = tid; k < C * COCO_MAX_DETS; k += COCO_MATCH_THREADS) det_mask[k] = 0;
  // rank key: class, then score descending, then row (NMS) index - np.argsort(-score, kind="mergesort") per class
  for (int j = tid; j < M; j += COCO_MATCH_THREADS) {
    const float* r = pb + (long long)j * D;
    const unsigned long long cls = (unsigned)class_argmax(r + 5, C, false);
    key[j] = (cls << 46) | ((unsigned long long)score_desc_key(r[4]) << 14) | (unsigned)j;
  }
  for (int g = tid; g < N; g += COCO_MATCH_THREADS) gt_cls[g] = (signed char)label_class(lb[(long long)g * 6 + 5], C);
  for (int w = tid; w < (N + 1) / 2; w += COCO_MATCH_THREADS) gt_flags[w] = 0;
  __syncthreads();
  for (int j = tid; j < M; j += COCO_MATCH_THREADS) {
    const unsigned long long kj = key[j], lo = kj & ~((1ull << 46) - 1);
    int before = 0, lower_class = 0;   // keys below kj, keys of lower classes
    for (int i = 0; i < M; ++i) {
      const unsigned long long ki = key[i];
      before += ki < kj;
      lower_class += ki < lo;
    }
    const int cls = (int)(kj >> 46), rank = before - lower_class;
    const float score = pb[(long long)j * D + 4];
    const long long o = rec0 + before;   // records of an image in (class, rank) order
    *reinterpret_cast<int4*>(records + o * 4) = make_int4(__float_as_int(score), cls, (int)(image0 + b), rank);
    keys[o] = ((long long)cls << 32) | score_desc_key(score);
    if (rank < COCO_MAX_DETS) {
      det[cls * COCO_MAX_DETS + rank] = j;
      det_pos[cls * COCO_MAX_DETS + rank] = (int)before;
      atomicAdd(&n_det[cls], 1);
    }
  }
  for (int g = tid; g < N; g += COCO_MATCH_THREADS)
    if (gt_cls[g] >= 0) atomicAdd(&n_gt[gt_cls[g]], 1);
  __syncthreads();
  for (int k = tid; k < C; k += COCO_MATCH_THREADS)
    if (n_gt[k]) atomicAdd(&gt_count[k], (unsigned long long)n_gt[k]);

  // greedy matching: one warp per (class, threshold); ground truths visited in grid order, the later of equal IoUs wins
  volatile unsigned* flags = gt_flags;
  for (int p = warp; p < C * YG_COCO_IOU_THRS; p += COCO_MATCH_THREADS / 32) {
    const int k = p / YG_COCO_IOU_THRS, t = p % YG_COCO_IOU_THRS;
    if (n_gt[k] == 0) continue;
    double tv = thr.t[0];   // select, not a dynamic index: that would copy the parameter to local memory
#pragma unroll
    for (int i = 1; i < YG_COCO_IOU_THRS; ++i) tv = i == t ? thr.t[i] : tv;
    const double best0 = fmin(tv, 1.0 - 1e-10);
    for (int r = 0; r < n_det[k]; ++r) {
      const float* dr = pb + (long long)det[k * COCO_MAX_DETS + r] * D;
      const float dx1 = dr[0], dy1 = dr[1], dx2 = dr[2], dy2 = dr[3], darea = box_area_f(dx1, dy1, dx2, dy2);
      float best = -INFINITY;
      int bg = -1;
      for (int g = lane; g < N; g += 32) {
        if (gt_cls[g] != k || ((flags[g >> 1] >> (16 * (g & 1) + t)) & 1u)) continue;
        const float* gr = lb + (long long)g * 6 + 1;
        const float iou = box_iou_f(gr[0], gr[1], gr[2], gr[3], box_area_f(gr[0], gr[1], gr[2], gr[3]), dx1, dy1, dx2, dy2, darea);
        if ((double)iou < best0) continue;
        if (iou > best || (iou == best && g > bg)) { best = iou; bg = g; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int og = __shfl_xor_sync(0xffffffffu, bg, o);
        if (ob > best || (ob == best && og > bg)) { best = ob; bg = og; }
      }
      if (bg >= 0 && lane == 0) {
        atomicOr(&gt_flags[bg >> 1], 1u << (16 * (bg & 1) + t));
        atomicOr(&det_mask[k * COCO_MAX_DETS + r], 1u << t);
      }
      __syncwarp();
    }
  }
  __syncthreads();
  for (int k = 0; k < C; ++k)
    for (int r = tid; r < n_det[k]; r += COCO_MATCH_THREADS)
      records[(rec0 + det_pos[k * COCO_MAX_DETS + r]) * 4 + 3] = r | (int)(det_mask[k * COCO_MAX_DETS + r] << 16);
}

// ---- COCO accumulate -------------------------------------------------------------------------------------------------
// q[r] = max(pr[i] for i with rc[i] >= recThrs[r]) equals COCOeval's pr[searchsorted(rc, recThrs[r], "left")] after the
// precision envelope (rc is non-decreasing), so every record adds pr[i] to the recall points up to rc[i] in any order:
// one atomicMax on the largest such point, then a suffix max.  pr >= 0, so its bits order like its values.
__global__ void __launch_bounds__(COCO_ACC_THREADS) coco_accumulate_kernel(
    const int* __restrict__ records, const long long* __restrict__ sorted_keys, const long long* __restrict__ perm, long long n_rec,
    const long long* __restrict__ gt_count, int C, RecThrs rec, double* __restrict__ precision, double* __restrict__ recall) {
  __shared__ unsigned long long q[YG_COCO_REC_THRS];
  __shared__ int warp_tot[32];
  __shared__ double rec_s[YG_COCO_REC_THRS];
  const int k = blockIdx.x, t = blockIdx.y, mi = blockIdx.z, tid = threadIdx.x;
  const int max_det = mi == 0 ? 1 : (mi == 1 ? 10 : 100);
  const long long npig = gt_count[k];
  double* prec_out = precision + ((long long)t * YG_COCO_REC_THRS * C + k) * 3 + mi;   // [t][r][k][m]
  if (npig == 0) {   // no ground truth of this class: -1, excluded from the summaries
    for (int r = tid; r < YG_COCO_REC_THRS; r += COCO_ACC_THREADS) prec_out[(long long)r * C * 3] = -1.0;
    if (tid == 0) recall[((long long)t * C + k) * 3 + mi] = -1.0;
    return;
  }
  for (int r = tid; r < YG_COCO_REC_THRS; r += COCO_ACC_THREADS) { q[r] = 0ull; rec_s[r] = rec.r[r]; }
  // this class's segment of the sorted records
  long long lo = 0, hi = n_rec;
  while (lo < hi) { const long long m = (lo + hi) >> 1; if (sorted_keys[m] < ((long long)k << 32)) lo = m + 1; else hi = m; }
  const long long s0 = lo;
  hi = n_rec;
  while (lo < hi) { const long long m = (lo + hi) >> 1; if (sorted_keys[m] < ((long long)(k + 1) << 32)) lo = m + 1; else hi = m; }
  const long long s1 = lo;
  __syncthreads();
  const double dnpig = (double)npig;
  long long nd = 0, ntp = 0;   // detections and true positives before this chunk
  for (long long c0 = s0; c0 < s1; c0 += COCO_ACC_THREADS) {
    const long long i = c0 + tid;
    bool in = false, tp = false;
    if (i < s1) {
      const int w = records[perm[i] * 4 + 3];
      in = (w & 0xffff) < max_det;
      tp = in && ((w >> (16 + t)) & 1);
    }
    int tot_in, tot_tp;
    const int r_in = block_rank<COCO_ACC_THREADS>(in, warp_tot, tot_in);
    const int r_tp = block_rank<COCO_ACC_THREADS>(tp, warp_tot, tot_tp);
    if (in) {
      const double tps = (double)(ntp + r_tp + (tp ? 1 : 0));
      const double fps = (double)(nd + r_in + 1) - tps;
      const double rc = __ddiv_rn(tps, dnpig);
      const double pr = __ddiv_rn(tps, __dadd_rn(__dadd_rn(fps, tps), 2.220446049250313e-16));   // np.spacing(1)
      // largest recall point <= rc
      int a = 0, z = YG_COCO_REC_THRS;
      while (a < z) { const int m = (a + z) >> 1; if (rec_s[m] <= rc) a = m + 1; else z = m; }
      if (a > 0) atomicMax(&q[a - 1], (unsigned long long)__double_as_longlong(pr));
    }
    nd += tot_in;
    ntp += tot_tp;
  }
  __syncthreads();
  if (tid == 0) {
    unsigned long long run = 0ull;
    for (int r = YG_COCO_REC_THRS - 1; r >= 0; --r) {
      run = q[r] > run ? q[r] : run;
      prec_out[(long long)r * C * 3] = __longlong_as_double((long long)run);
    }
    recall[((long long)t * C + k) * 3 + mi] = nd ? __ddiv_rn((double)ntp, dnpig) : 0.0;
  }
}

// ---- ROC and calibration: score rows ---------------------------------------------------------------------------------
// The rows are those of convert_background_errors(C + 1) (matched, missed, extra; without background the matched pairs
// alone), grouped by image: image b's start at out_off + gather_off[2b] + gather_off[2b + 1] (prefix of N + M - K).
constexpr int MET_MAX_BINS = 255;        // calibration bins; bins + 1 <= SCORE_THREADS, one accumulating thread per bin
constexpr int SCORE_THREADS = 256;
constexpr int ROC_THREADS = 512;
struct BinBounds { float b[MET_MAX_BINS + 1]; };

// torchmetrics' format rule: *flag = 1 when a class value of the matched (and, with background, extra) rows lies outside
// [0, 1] or is NaN; the caller zeroes *flag
__global__ void score_format_kernel(const float* __restrict__ out_preds, const float* __restrict__ extra, long long n_matched,
                                    long long n_extra, int C, int* __restrict__ flag) {
  const long long nm = n_matched * C, n = nm + n_extra * C;
  bool bad = false;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long j = i < nm ? i : i - nm;
    const float x = (i < nm ? out_preds : extra)[(j / C) * (5 + C) + 5 + j % C];
    bad |= !(x >= 0.f && x <= 1.f);
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

// column k of a score row before the format rule: the class columns and the appended 0 of a prediction row, or the
// one-hot background row of a missed label (src == nullptr)
__device__ __forceinline__ float raw_score(const float* __restrict__ src, int k, int C) {
  return src ? (k < C ? src[5 + k] : 0.f) : (k == C ? 1.f : 0.f);
}

// One CTA per image.  Each row: its nb scores (softmaxed in fp64 over all nb columns when *softmax_flag) into
// scores[row][.] and its target into targets[row] (when scores != nullptr); confidence = the row maximum of the stored
// scores, prediction = its first maximum, bin = bucketize(conf, bounds, right=True) - 1.  The per-bin sums go to
// partials[b] in a fixed order: rows in chunks of SCORE_THREADS, thread t sums bin t over a chunk in row order.
__global__ void __launch_bounds__(SCORE_THREADS) score_rows_kernel(
    const float* __restrict__ out_preds, const float* __restrict__ out_labels, const float* __restrict__ missed,
    const float* __restrict__ extra, int C, int with_bg, const LsapDesc* __restrict__ desc, const long long* __restrict__ gather_off,
    const int* __restrict__ lsap_status, const int* __restrict__ softmax_flag, const __grid_constant__ BinBounds bounds, int bins,
    float* __restrict__ scores, int* __restrict__ targets, int* __restrict__ nan_status, unsigned char* __restrict__ partials) {
  __shared__ float sb[MET_MAX_BINS + 1];
  __shared__ float chunk_conf[SCORE_THREADS];
  __shared__ int chunk_key[SCORE_THREADS];   // bin << 1 | correct, -1 for no row
  __shared__ int nan_row;
  const int b = blockIdx.x, tid = threadIdx.x, nb = C + (with_bg ? 1 : 0), nbin = bins + 1;
  double* p_conf = reinterpret_cast<double*>(partials) + (long long)b * nbin;
  int* p_count = reinterpret_cast<int*>(partials + (long long)gridDim.x * nbin * 8) + (long long)b * nbin * 2;
  for (int i = tid; i < nbin; i += SCORE_THREADS) sb[i] = bounds.b[i];
  if (tid == 0) nan_row = 0;
  const bool ok = lsap_status[b] == YG_LSAP_OK;   // else the gather wrote no rows; the caller raises the solver's error
  const LsapDesc d = desc[b];
  const int N = ok ? d.rows : 0, M = ok ? d.cols : 0, K = min(N, M);
  const int n_rows = with_bg ? N + M - K : K;
  const long long row0 = with_bg ? d.out_off + gather_off[2 * b] + gather_off[2 * b + 1] : d.out_off;
  const bool softmax = *softmax_flag != 0;
  __syncthreads();
  double acc_conf = 0.0;
  int acc_count = 0, acc_correct = 0;
  for (int c0 = 0; c0 < n_rows; c0 += SCORE_THREADS) {
    const int t = c0 + tid;
    int key = -1;
    float conf = 0.f;
    if (t < n_rows) {
      // target: int(label[5]) (-1 for a class outside [0, C): the confusion kernel's check raises), C for an extra row
      const float* src;
      int target;
      if (t < K) {
        src = out_preds + (d.out_off + t) * (5 + C);
        target = label_class(out_labels[(d.out_off + t) * 6 + 5], C);
      } else if (t < N) {
        src = nullptr;
        target = label_class(missed[(gather_off[2 * b] + t - K) * 6 + 5], C);
      } else {
        src = extra + (gather_off[2 * b + 1] + t - N) * (5 + C);
        target = C;
      }
      double m = -INFINITY;
      for (int k = 0; k < nb; ++k) m = fmax(m, (double)raw_score(src, k, C));
      double s = 0.0;
      if (softmax)
        for (int k = 0; k < nb; ++k) s += exp((double)raw_score(src, k, C) - m);
      float best = 0.f;
      int arg = 0;
      bool has_nan = false;   // a NaN class value, or an infinite one under the softmax
      for (int k = 0; k < nb; ++k) {
        const float x = raw_score(src, k, C);
        const float v = softmax ? (float)(exp((double)x - m) / s) : x;
        has_nan |= v != v;
        if (k == 0 || v > best) { best = v; arg = k; }
        if (scores) scores[(row0 + t) * nb + k] = v;
      }
      if (scores) targets[row0 + t] = target;
      if (has_nan) nan_row = 1;
      int lo = 0, hi = nbin;   // boundaries <= best
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (sb[mid] <= best) lo = mid + 1; else hi = mid; }
      key = ((lo > 0 ? lo - 1 : 0) << 1) | (arg == target ? 1 : 0);
      conf = best;
    }
    chunk_key[tid] = key;
    chunk_conf[tid] = conf;
    __syncthreads();
    if (tid < nbin) {
      const int lim = min(SCORE_THREADS, n_rows - c0);
      for (int i = 0; i < lim; ++i) {
        const int kk = chunk_key[i];
        if ((kk >> 1) == tid) { acc_conf += (double)chunk_conf[i]; ++acc_count; acc_correct += kk & 1; }
      }
    }
    __syncthreads();
  }
  if (tid < nbin) { p_conf[tid] = acc_conf; p_count[2 * tid] = acc_count; p_count[2 * tid + 1] = acc_correct; }
  if (tid == 0) nan_status[b] = nan_row;
}

// the fixed-order second step: bin i of every CTA partial, images in order
__global__ void score_bins_reduce_kernel(const unsigned char* __restrict__ partials, int B, int nbin, long long* __restrict__ count,
                                         long long* __restrict__ correct, double* __restrict__ conf) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nbin) return;
  const double* p_conf = reinterpret_cast<const double*>(partials);
  const int* p_count = reinterpret_cast<const int*>(partials + (long long)B * nbin * 8);
  double s = 0.0;
  long long n = 0, c = 0;
  for (int b = 0; b < B; ++b) {
    s += p_conf[(long long)b * nbin + i];
    n += p_count[((long long)b * nbin + i) * 2];
    c += p_count[((long long)b * nbin + i) * 2 + 1];
  }
  count[i] = n;
  correct[i] = c;
  conf[i] = s;
}

// ---- ROC curves ------------------------------------------------------------------------------------------------------
// key[k * R + r] = k << 32 | score_desc_key(score[r][k]); -0 is keyed as +0 so that equal scores form one group
__global__ void roc_keys_kernel(const float* __restrict__ scores, long long R, int nb, long long* __restrict__ keys) {
  const long long n = R * nb;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long k = i / R, r = i - k * R;
    const float s = scores[r * nb + k];
    keys[i] = (k << 32) | score_desc_key(s == 0.f ? 0.f : s);
  }
}

__device__ __forceinline__ float desc_key_score(unsigned key) {
  const unsigned u = ~key;
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// One CTA per class k over its sorted segment: _binary_clf_curve (one point at the last row of every distinct score,
// tps = positives so far, fps = rows so far - tps) after the prepended point (0, 0, threshold 1); fpr / tpr in fp64.
// AUC = sum over points of (fps_j - fps_j-1) * (tps_j + tps_j-1), an exact integer, over 2 * fps_last * tps_last.
__global__ void __launch_bounds__(ROC_THREADS) roc_curve_kernel(
    const long long* __restrict__ sorted_keys, const long long* __restrict__ perm, const int* __restrict__ targets, long long R,
    double* __restrict__ fpr, double* __restrict__ tpr, float* __restrict__ thresholds, long long* __restrict__ lengths,
    double* __restrict__ auc) {
  __shared__ int warp_tot[32];
  __shared__ long long pt_tps[ROC_THREADS], pt_row[ROC_THREADS];
  __shared__ unsigned long long area;
  __shared__ long long n_pos;
  const int k = blockIdx.x, tid = threadIdx.x;
  const long long seg = (long long)k * R, out0 = (long long)k * (R + 1);
  if (tid == 0) { area = 0ull; n_pos = 0; }
  __syncthreads();
  long long cnt = 0;
  for (long long r = tid; r < R; r += ROC_THREADS) cnt += targets[r] == k;
  atomicAdd(reinterpret_cast<unsigned long long*>(&n_pos), (unsigned long long)cnt);
  __syncthreads();
  const long long P = n_pos, F = R - P;
  const double dP = (double)P, dF = (double)F;
  if (tid == 0) { fpr[out0] = 0.0; tpr[out0] = 0.0; thresholds[out0] = 1.f; }
  long long tps_carry = 0, pts = 0, prev_tps = 0, prev_row = -1;   // prev_*: the last point so far (the prepended one)
  unsigned long long my_area = 0ull;
  for (long long c0 = 0; c0 < R; c0 += ROC_THREADS) {
    const long long i = c0 + tid;
    bool pos = false, last = false;
    unsigned key = 0u;
    if (i < R) {
      key = (unsigned)sorted_keys[seg + i];
      pos = targets[perm[seg + i] - seg] == k;
      last = i == R - 1 || (unsigned)sorted_keys[seg + i + 1] != key;
    }
    int tot_pos, tot_last;
    const int r_pos = block_rank<ROC_THREADS>(pos, warp_tot, tot_pos);
    const int r_last = block_rank<ROC_THREADS>(last, warp_tot, tot_last);
    const long long tps = tps_carry + r_pos + (pos ? 1 : 0);
    if (last) { pt_tps[r_last] = tps; pt_row[r_last] = i; }
    __syncthreads();
    if (last) {
      const long long fps = i + 1 - tps, o = out0 + pts + 1 + r_last;
      const long long ptp = r_last ? pt_tps[r_last - 1] : prev_tps, prw = r_last ? pt_row[r_last - 1] : prev_row;
      my_area += (unsigned long long)(fps - (prw + 1 - ptp)) * (unsigned long long)(tps + ptp);
      fpr[o] = F > 0 ? __ddiv_rn((double)fps, dF) : 0.0;
      tpr[o] = P > 0 ? __ddiv_rn((double)tps, dP) : 0.0;
      thresholds[o] = desc_key_score(key);
    }
    if (tot_last) { prev_tps = pt_tps[tot_last - 1]; prev_row = pt_row[tot_last - 1]; }
    tps_carry += tot_pos;
    pts += tot_last;
    __syncthreads();   // pt_* are rewritten by the next chunk
  }
  atomicAdd(&area, my_area);
  __syncthreads();
  if (tid == 0) {
    lengths[k] = pts + 1;
    auc[k] = (P > 0 && F > 0) ? __ddiv_rn((double)area, __dmul_rn(2.0 * dF, dP)) : -1.0;
  }
}

}  // namespace yg
using namespace yg;

extern "C" int yg_score_rows_batch(const float* out_preds, const float* out_labels, const float* missed, const float* extra,
                                   long long n_matched, long long n_extra, int B, int num_classes, int include_background,
                                   const void* desc, const long long* gather_off, const int* lsap_status, const float* bin_bounds,
                                   int bins, int* softmax_flag, float* scores, int* targets, int* nan_status, void* partials,
                                   long long* bin_count, long long* bin_correct, double* bin_conf, void* stream) {
  YG_CHECK_ARG(B >= 0 && num_classes >= 1 && num_classes <= MET_MAX_CLASSES && n_matched >= 0 && n_extra >= 0,
               "score_rows_batch: B = %d, num_classes = %d", B, num_classes);
  YG_CHECK_ARG(bins >= 1 && bins <= MET_MAX_BINS, "score_rows_batch: %d bins, between 1 and %d are supported", bins, MET_MAX_BINS);
  YG_CHECK_ARG(bin_bounds && softmax_flag && bin_count && bin_correct && bin_conf && (B == 0 || (desc && gather_off && lsap_status &&
               nan_status && partials)), "score_rows_batch: null pointer");
  YG_CHECK_ARG(!scores == !targets, "score_rows_batch: scores and targets go together");
  cudaStream_t st = (cudaStream_t)stream;
  YG_CUDA(cudaMemsetAsync(softmax_flag, 0, sizeof(int), st));
  const long long n_values = (n_matched + (include_background ? n_extra : 0)) * num_classes;
  if (n_values > 0) {
    score_format_kernel<<<(int)std::min<long long>(cdiv(n_values, 256), 1184), 256, 0, st>>>(
        out_preds, extra, n_matched, include_background ? n_extra : 0, num_classes, softmax_flag);
    YG_LAUNCH_CHECK("score_format");
  }
  BinBounds bb;
  for (int i = 0; i <= bins; ++i) bb.b[i] = bin_bounds[i];
  if (B > 0) {
    score_rows_kernel<<<B, SCORE_THREADS, 0, st>>>(out_preds, out_labels, missed, extra, num_classes, include_background ? 1 : 0,
                                                   (const LsapDesc*)desc, gather_off, lsap_status, softmax_flag, bb, bins, scores,
                                                   targets, nan_status, (unsigned char*)partials);
    YG_LAUNCH_CHECK("score_rows");
  }
  score_bins_reduce_kernel<<<cdiv(bins + 1, 256), 256, 0, st>>>((const unsigned char*)partials, B, bins + 1, bin_count, bin_correct,
                                                                bin_conf);
  YG_LAUNCH_CHECK("score_bins_reduce");
  return YG_OK;
}

extern "C" int yg_roc_keys(const float* scores, long long rows, int nb, long long* keys, void* stream) {
  YG_CHECK_ARG(rows >= 0 && rows < 0x7fffffffLL && nb >= 1 && nb <= MET_MAX_CLASSES + 1, "roc_keys: rows = %lld, nb = %d", rows, nb);
  if (rows == 0) return YG_OK;
  YG_CHECK_ARG(scores && keys, "roc_keys: null pointer");
  roc_keys_kernel<<<(int)std::min<long long>(cdiv(rows * nb, 256), 4736), 256, 0, (cudaStream_t)stream>>>(scores, rows, nb, keys);
  YG_LAUNCH_CHECK("roc_keys");
  return YG_OK;
}

extern "C" int yg_roc_curves(const long long* sorted_keys, const long long* perm, const int* targets, long long rows, int nb,
                             double* fpr, double* tpr, float* thresholds, long long* lengths, double* auc, void* stream) {
  YG_CHECK_ARG(rows >= 0 && rows < 0x7fffffffLL && nb >= 1 && nb <= MET_MAX_CLASSES + 1, "roc_curves: rows = %lld, nb = %d", rows, nb);
  YG_CHECK_ARG(fpr && tpr && thresholds && lengths && auc && (rows == 0 || (sorted_keys && perm && targets)), "roc_curves: null pointer");
  roc_curve_kernel<<<nb, ROC_THREADS, 0, (cudaStream_t)stream>>>(sorted_keys, perm, targets, rows, fpr, tpr, thresholds, lengths, auc);
  YG_LAUNCH_CHECK("roc_curves");
  return YG_OK;
}

extern "C" int yg_confusion_batch(const float* out_preds, const float* out_labels, const float* missed, const float* extra, int B,
                                  int num_classes, int include_background, const void* desc, const long long* gather_off,
                                  const int* lsap_status, int* label_status, long long* confusion, void* stream) {
  YG_CHECK_ARG(B >= 0 && num_classes >= 1 && num_classes <= MET_MAX_CLASSES, "confusion_batch: B = %d, num_classes = %d", B,
               num_classes);
  if (B == 0) return YG_OK;
  YG_CHECK_ARG(desc && gather_off && lsap_status && label_status && confusion, "confusion_batch: null pointer");
  confusion_kernel<<<B, CONF_THREADS, 0, (cudaStream_t)stream>>>(out_preds, out_labels, missed, extra, num_classes,
                                                                 include_background ? 1 : 0, (const LsapDesc*)desc, gather_off,
                                                                 lsap_status, label_status, (unsigned long long*)confusion);
  YG_LAUNCH_CHECK("confusion");
  return YG_OK;
}

extern "C" int yg_coco_match_batch(const float* pred_rows, const float* label_rows, int B, int cells, int num_classes,
                                   int max_labels, int max_preds, const void* desc, const long long* gather_off, long long image0,
                                   const double* iou_thrs, int* records, long long* keys, long long* gt_count, void* stream) {
  YG_CHECK_ARG(B >= 0 && num_classes >= 1 && num_classes <= MET_MAX_CLASSES, "coco_match_batch: B = %d, num_classes = %d", B,
               num_classes);
  YG_CHECK_ARG(cells >= 1 && cells <= MET_MAX_CELLS, "coco_match_batch: Sy*Sx = %d exceeds %d", cells, MET_MAX_CELLS);
  YG_CHECK_ARG(max_labels >= 0 && max_labels <= cells && max_preds >= 0 && max_preds <= cells && image0 >= 0 &&
               image0 + B <= 0x7fffffffLL, "coco_match_batch: bad sizes");
  if (B == 0) return YG_OK;
  YG_CHECK_ARG(pred_rows && label_rows && desc && gather_off && iou_thrs && gt_count, "coco_match_batch: null pointer");
  IouThrs thr;
  for (int t = 0; t < YG_COCO_IOU_THRS; ++t) thr.t[t] = iou_thrs[t];
  const size_t smem = coco_match_smem(max_labels, max_preds);
  YG_CUDA(cudaFuncSetAttribute(coco_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coco_match_smem(MET_MAX_CELLS, MET_MAX_CELLS)));
  coco_match_kernel<<<B, COCO_MATCH_THREADS, smem, (cudaStream_t)stream>>>(pred_rows, label_rows, cells, num_classes,
                                                                           (const LsapDesc*)desc, gather_off, image0, thr, records,
                                                                           keys, (unsigned long long*)gt_count);
  YG_LAUNCH_CHECK("coco_match");
  return YG_OK;
}

extern "C" int yg_coco_accumulate(const int* records, const long long* sorted_keys, const long long* perm, long long n_records,
                                  const long long* gt_count, int num_classes, const double* rec_thrs, double* precision,
                                  double* recall, void* stream) {
  YG_CHECK_ARG(n_records >= 0 && num_classes >= 1 && num_classes <= MET_MAX_CLASSES, "coco_accumulate: n = %lld, num_classes = %d",
               n_records, num_classes);
  YG_CHECK_ARG(gt_count && rec_thrs && precision && recall && (n_records == 0 || (records && sorted_keys && perm)),
               "coco_accumulate: null pointer");
  RecThrs rec;
  for (int r = 0; r < YG_COCO_REC_THRS; ++r) rec.r[r] = rec_thrs[r];
  coco_accumulate_kernel<<<dim3(num_classes, YG_COCO_IOU_THRS, 3), COCO_ACC_THREADS, 0, (cudaStream_t)stream>>>(
      records, sorted_keys, perm, n_records, gt_count, num_classes, rec, precision, recall);
  YG_LAUNCH_CHECK("coco_accumulate");
  return YG_OK;
}
