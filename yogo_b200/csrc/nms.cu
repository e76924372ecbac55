// Objectness threshold + box conversion + greedy NMS + class-confidence filter + per-class
// counts for a whole batch: five launches that keep every SM busy, no host synchronisation.
// Replaces the per-image Python loop over format_preds
// (/root/reference/yogo/utils/prediction_formatting.py:23-93: boolean-mask gather, box_convert,
// torchvision.ops.nms, fancy-index) and get_prediction_class_counts /
// count_cells_for_formatted_preds (/root/reference/yogo/infer.py:60-124).
//
//   1. nms_candidates_kernel  all cells of all images in parallel (the only pass over the 48 B/cell prediction
//                             tensor): obj > thr -> xyxy box, score key, compacted per image (block-aggregated atomics;
//                             the order inside an image does not matter, the sort key carries the cell index)
//   2. nms_sort_kernel        one CTA per image: bitonic sort of the candidates' 64-bit keys in shared memory
//   3. nms_mask_kernel        persistent CTAs over (image, 64x64 block of the upper triangle): suppression bit masks
//   4. nms_scan_kernel        one CTA per image: greedy resolve, 64 candidates per step, against the bit masks;
//                             then gather of the kept rows in output order, class-confidence filter, counts
//   (3, 4 run per group of images so that the masks of a group fit the workspace; skipped when iou_thresh == 0)
//
// Bit-exactness contract (SURVEY.md Appendix C): every floating-point operation that decides
// the result is a single IEEE fp32 operation issued through __f*_rn intrinsics, so nvcc can
// never contract them into FMAs; the score order is a stable descending sort (ties -> lower
// candidate index first); suppression is `iou > thr` (strict; NaN never suppresses) with the
// fp32 ratio compared against the threshold as a double, exactly as torchvision's CPU kernel.
#include "common.cuh"

namespace yg {

constexpr int NMS_THREADS = 1024;     // sort kernel
constexpr int NMS_MAX_CELLS = 16384;  // Sy*Sx limit (reference grid: 97*129 = 12513)
constexpr int NMS_CHUNK = 64;
constexpr int NMS_SCAN_THREADS = 256; // >= NMS_MAX_CELLS / 64 mask words per row
constexpr int NMS_SCAN_SMEM_WORDS = 20 * 1024;   // 160 KB: masks of images with up to ~1100 candidates
constexpr size_t NMS_MASK_CAP = 2ull << 30;   // bytes of suppression masks held at a time (images are processed in groups)

struct NmsWs {
  int* n_cand;                  // [B]          candidates per image
  unsigned long long* keys;     // [B][cells]   (~orderable(score) << 32) | cell, unsorted then unused
  float4* cell_box;             // [B][cells]   xyxy box of a candidate, indexed by grid cell
  int* sorted_cell;             // [B][cells]   grid cell of the i-th candidate in descending-score order
  float4* sorted_box;           // [B][cells]
  int* kept_ord;                // [B][cells]   sorted ordinal of each kept box, NMS order
  unsigned long long* mask;     // [G][cells][nw] bit j of word w of row i: candidate 64 w + j (> i) is suppressed by i
};

__device__ __forceinline__ bool iou_gt(const float4 a, const float area_a, const float4 b, const float area_b,
                                       const double thr) {
  // torchvision/csrc/ops/cpu/nms_kernel.cpp semantics
  const float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y);
  const float xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
  const float w = __fsub_rn(xx2, xx1);
  const float h = __fsub_rn(yy2, yy1);
  // disjoint boxes (or NaN coordinates): the clamped intersection is 0 and 0 / x > thr is false for the thr > 0 NMS runs
  // with (0 / 0 = NaN never suppresses either) - most pairs of a sparse image end here, before the IEEE division
  if (!(w > 0.f && h > 0.f)) return false;
  const float inter = __fmul_rn(w, h);
  const float ovr = __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_a, area_b), inter));
  return (double)ovr > thr;
}
// The same decision without the IEEE division for all but a sliver of pairs.  fl(inter / uni) > thr (fp32 quotient
// compared as a double) <=> fl(inter / uni) >= F, F = the smallest float above thr; with P = the largest float <= thr:
// inter / uni >= F certainly gives true, inter / uni < P certainly gives false.  t_hi = F (1 + 2^-20) and
// t_lo = P (1 - 2^-20) leave room for the rounding of one fp32 product; pairs in between take the exact path.
struct IouThr { double thr; float t_lo, t_hi; };
__device__ __forceinline__ bool iou_gt_fast(const float4 a, const float area_a, const float4 b, const float area_b, const IouThr t) {
  const float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y);
  const float xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
  const float w = __fsub_rn(xx2, xx1);
  const float h = __fsub_rn(yy2, yy1);
  if (!(w > 0.f && h > 0.f)) return false;
  const float inter = __fmul_rn(w, h);
  const float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
  if (uni > 0.f && inter < 3.0e38f && uni < 3.0e38f) {
    if (inter > __fmul_rn(t.t_hi, uni)) return true;
    if (inter < __fmul_rn(t.t_lo, uni)) return false;
  }
  return (double)__fdiv_rn(inter, uni) > t.thr;
}
__device__ __forceinline__ float box_area(const float4 b) {
  return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
}

// ---- 1. threshold + boxes + keys, every cell of the batch in parallel -------------------------------------------------
__global__ void __launch_bounds__(256) nms_candidates_kernel(const float* __restrict__ preds, int C, int cells, float obj_thresh,
                                                             int do_nms, NmsWs ws) {
  __shared__ int s_warp[8];
  __shared__ int s_base;
  const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int k = blockIdx.x * 256 + tid;
  const float* pb = preds + (long long)b * (5 + C) * cells;
  float obj = 0.f;
  bool flag = false;
  if (k < cells) { obj = __ldg(pb + 4LL * cells + k); flag = obj > obj_thresh; }
  const unsigned bal = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) s_warp[wid] = __popc(bal);
  __syncthreads();
  if (tid == 0) {
    int tot = 0;
    for (int w = 0; w < 8; ++w) { const int t = s_warp[w]; s_warp[w] = tot; tot += t; }
    s_base = tot ? atomicAdd(ws.n_cand + b, tot) : 0;
  }
  __syncthreads();
  if (!flag) return;
  const int pos = s_base + s_warp[wid] + __popc(bal & ((1u << lane) - 1u));
  const float cx = __ldg(pb + k), cy = __ldg(pb + (long long)cells + k), w = __ldg(pb + 2LL * cells + k), h = __ldg(pb + 3LL * cells + k);
  // torchvision _box_cxcywh_to_xyxy: x1 = cx - 0.5*w ...
  const float hw = __fmul_rn(0.5f, w), hh = __fmul_rn(0.5f, h);
  ws.cell_box[(long long)b * cells + k] = make_float4(__fsub_rn(cx, hw), __fsub_rn(cy, hh), __fadd_rn(cx, hw), __fadd_rn(cy, hh));
  unsigned hi = 0u;
  if (do_nms) {
    float mx = __ldg(pb + 5LL * cells + k);
    for (int c = 1; c < C; ++c) mx = fmaxf(mx, __ldg(pb + (long long)(5 + c) * cells + k));
    float score = __fmul_rn(mx, obj);
    if (score == 0.f) score = 0.f;  // -0 -> +0 (equal under torch's sort)
    unsigned u = __float_as_uint(score);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);  // ascending-orderable
    hi = ~u;                                          // descending score ...
  }
  // ... then ascending cell index = ascending candidate index (stable sort of the reference); with NMS disabled
  // (iou_thresh == 0, prediction_formatting.py:80) the key is the cell index alone: rows stay in grid order
  ws.keys[(long long)b * cells + pos] = ((unsigned long long)hi << 32) | (unsigned)k;
}

// ---- 2. per-image sort ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NMS_THREADS, 1) nms_sort_kernel(int cells, NmsWs ws) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = ws.n_cand[b];
  if (n == 0) return;
  int Pn = 1;
  while (Pn < n) Pn <<= 1;
  const unsigned long long* gk = ws.keys + (long long)b * cells;
  for (int i = tid; i < Pn; i += NMS_THREADS) keys[i] = i < n ? gk[i] : ~0ull;
  __syncthreads();
  for (int size = 2; size <= Pn; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < (Pn >> 1); t += NMS_THREADS) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const bool up = ((lo & size) == 0);
        const unsigned long long a = keys[lo], c = keys[hi];
        if ((a > c) == up) { keys[lo] = c; keys[hi] = a; }
      }
      __syncthreads();
    }
  }
  const float4* cb = ws.cell_box + (long long)b * cells;
  for (int i = tid; i < n; i += NMS_THREADS) {
    const int cell = (int)(keys[i] & 0xffffffffu);
    ws.sorted_cell[(long long)b * cells + i] = cell;
    ws.sorted_box[(long long)b * cells + i] = cb[cell];
  }
}

// ---- 3. suppression bit masks: persistent CTAs over (image, row block, column block >= row block) -------------------
__global__ void __launch_bounds__(NMS_CHUNK) nms_mask_kernel(int b0, int nb_img, int cells, int nw_stride, IouThr thr, NmsWs ws) {
  __shared__ long long s_prefix[257];   // work items before image g of the group (a group holds at most 256 images)
  __shared__ float4 s_cb[NMS_CHUNK];
  __shared__ float s_ca[NMS_CHUNK];
  const int tid = threadIdx.x;
  for (int g = tid; g < nb_img; g += NMS_CHUNK) {
    const long long nb = (ws.n_cand[b0 + g] + NMS_CHUNK - 1) / NMS_CHUNK;
    s_prefix[g + 1] = nb * (nb + 1) / 2;
  }
  __syncthreads();
  if (tid == 0) {
    long long acc = 0;
    s_prefix[0] = 0;
    for (int g = 1; g <= nb_img; ++g) { acc += s_prefix[g]; s_prefix[g] = acc; }
  }
  __syncthreads();
  const long long total = s_prefix[nb_img];
  int g = 0;
  for (long long item = blockIdx.x; item < total; item += gridDim.x) {
    while (s_prefix[g + 1] <= item) ++g;   // items are visited in increasing order
    const int b = b0 + g;
    const int n = ws.n_cand[b];
    const int nb = (n + NMS_CHUNK - 1) / NMS_CHUNK;
    // item t of the row-major upper triangle -> (rb, cb): rows before rb hold rb * nb - rb (rb - 1) / 2 items
    const long long t = item - s_prefix[g];
    int rb = (int)((2.0 * nb + 1.0 - sqrt((2.0 * nb + 1.0) * (2.0 * nb + 1.0) - 8.0 * (double)t)) * 0.5);
    rb = max(0, min(rb, nb - 1));
    while (rb > 0 && (long long)rb * nb - (long long)rb * (rb - 1) / 2 > t) --rb;
    while ((long long)(rb + 1) * nb - (long long)(rb + 1) * rb / 2 <= t) ++rb;
    const int cb = rb + (int)(t - ((long long)rb * nb - (long long)rb * (rb - 1) / 2));
    const float4* sb = ws.sorted_box + (long long)b * cells;
    __syncthreads();
    const int j = cb * NMS_CHUNK + tid;
    if (j < n) { const float4 bx = sb[j]; s_cb[tid] = bx; s_ca[tid] = box_area(bx); }
    __syncthreads();
    const int i = rb * NMS_CHUNK + tid;
    if (i < n) {
      const float4 bi = sb[i];
      const float ai = box_area(bi);
      const int m = min(NMS_CHUNK, n - cb * NMS_CHUNK);
      unsigned long long bits = 0ull;
      const int j0 = (rb == cb) ? tid + 1 : 0;
      for (int jj = j0; jj < m; ++jj)
        if (iou_gt_fast(bi, ai, s_cb[jj], s_ca[jj], thr)) bits |= (1ull << jj);
      ws.mask[((long long)g * cells + i) * nw_stride + cb] = bits;
    }
  }
}

// ---- 4. greedy resolve against the masks + output ------------------------------------------------------------------------
__global__ void __launch_bounds__(NMS_SCAN_THREADS) nms_scan_kernel(
    const float* __restrict__ preds, int C, int cells, int b0, int nw_stride, int do_nms, int xyxy, float min_cls,
    int* __restrict__ keep_count, float* __restrict__ rows, int* __restrict__ keep_index,
    unsigned long long* __restrict__ class_counts, NmsWs ws) {
  extern __shared__ __align__(16) unsigned long long s_m[];   // [NMS_SCAN_SMEM_WORDS]
  __shared__ unsigned long long s_keep;
  __shared__ int warp_tot[NMS_SCAN_THREADS / 32];
  __shared__ int s_hist[32];
  const int g = blockIdx.x, b = b0 + g, tid = threadIdx.x, lane = tid & 31;
  const int D = 5 + C;
  const float* pb = preds + (long long)b * D * cells;
  const int n = ws.n_cand[b];
  int* kept_ord = ws.kept_ord + (long long)b * cells;
  if (tid < 32) s_hist[tid] = 0;
  int kept = 0;
  if (!do_nms) {
    for (int i = tid; i < n; i += NMS_SCAN_THREADS) kept_ord[i] = i;
    kept = n;
  } else {
    const int nw = (n + NMS_CHUNK - 1) / NMS_CHUNK;
    const unsigned long long* mask = ws.mask + (long long)g * cells * nw_stride;
    // realistic images (a few hundred candidates): the whole mask goes to shared memory in one coalesced sweep, so the
    // windows below see shared-memory instead of L2 latency on their dependent loads (the resolve is a serial chain)
    if ((long long)n * nw <= NMS_SCAN_SMEM_WORDS) {
      for (int i = tid; i < n * nw; i += NMS_SCAN_THREADS) {
        const int r = i / nw, w = i - r * nw;
        s_m[i] = (w >= r / NMS_CHUNK) ? mask[(long long)r * nw_stride + w] : 0ull;
      }
      __syncthreads();
      mask = s_m;
      nw_stride = nw;
    }
    unsigned long long removed = 0ull;   // thread w owns word w of the "suppressed" bit vector (nw <= 256 threads)
    // diagonal-block words of the first window (lane l of warp 0: rows l and 32 + l), fetched one window ahead
    unsigned long long d0 = 0ull, d1 = 0ull;
    if (tid < 32 && nw > 0) {
      if (lane < n) d0 = mask[(long long)lane * nw_stride];
      if (32 + lane < n) d1 = mask[(long long)(32 + lane) * nw_stride];
    }
    for (int c = 0; c < nw; ++c) {
      const int m = min(NMS_CHUNK, n - c * NMS_CHUNK);
      if (tid < 32) {
        // warp 0 resolves the 64-candidate window serially from the diagonal block: every lane tracks the same
        // `alive` / `keep` words (uniform control flow), lane l supplies the mask words of rows l and 32 + l
        const unsigned long long rem_c = __shfl_sync(0xffffffffu, removed, c & 31);   // (c < 32: word c lives in warp 0 ...
        const unsigned long long c0 = d0, c1 = d1;
        if (c + 1 < nw) {
          const int r0 = (c + 1) * NMS_CHUNK + lane, r1 = r0 + 32;
          d0 = (r0 < n) ? mask[(long long)r0 * nw_stride + c + 1] : 0ull;
          d1 = (r1 < n) ? mask[(long long)r1 * nw_stride + c + 1] : 0ull;
        }
        unsigned long long alive = (m == 64 ? ~0ull : ((1ull << m) - 1ull));
        alive &= ~((c < 32) ? rem_c : s_keep);   // ... otherwise its owner published it through s_keep, see below)
        unsigned long long keep = 0ull;
#pragma unroll 8
        for (int i = 0; i < 32; ++i) {
          const unsigned long long w = __shfl_sync(0xffffffffu, c0, i);
          if ((alive >> i) & 1ull) { keep |= (1ull << i); alive &= ~w; }
        }
#pragma unroll 8
        for (int i = 0; i < 32; ++i) {
          const unsigned long long w = __shfl_sync(0xffffffffu, c1, i);
          if ((alive >> (32 + i)) & 1ull) { keep |= (1ull << (32 + i)); alive &= ~w; }
        }
        __syncwarp();
        if (lane == 0) s_keep = keep;
      }
      __syncthreads();
      const unsigned long long keep = s_keep;
      if (tid > c && tid < nw) {
        // candidates kept in this window suppress later candidates: OR their mask rows into this thread's word,
        // sixteen independent loads in flight
        const unsigned long long* mrow = mask + (long long)c * NMS_CHUNK * nw_stride + tid;
        unsigned long long acc = 0ull;
        unsigned long long kb = keep;
        while (kb) {
          int idx[16];
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            idx[u] = kb ? __ffsll((long long)kb) - 1 : -1;
            kb &= kb - 1ull;   // (0 stays 0)
          }
          unsigned long long v[16];
#pragma unroll
          for (int u = 0; u < 16; ++u) v[u] = idx[u] >= 0 ? mrow[(long long)idx[u] * nw_stride] : 0ull;
#pragma unroll
          for (int u = 0; u < 16; ++u) acc |= v[u];
        }
        removed |= acc;
      }
      if (tid < m && ((keep >> tid) & 1ull))
        kept_ord[kept + __popcll(keep & ((1ull << tid) - 1ull))] = c * NMS_CHUNK + tid;
      kept += __popcll(keep);
      __syncthreads();
      // the owner of the next window's word (beyond warp 0) hands it to warp 0 through shared memory
      if (c + 1 >= 32 && tid == c + 1) s_keep = removed;
      __syncthreads();
    }
  }
  __syncthreads();

  // ---- gather rows in output order, class-confidence filter, counts ----
  int out_n = 0;
  float* rb = rows + (long long)b * cells * D;
  int* kb = keep_index + (long long)b * cells;
  const int* sorted_cell = ws.sorted_cell + (long long)b * cells;
  for (int r0 = 0; r0 < kept; r0 += NMS_SCAN_THREADS) {
    const int r = r0 + tid;
    bool flag = false;
    int cell = 0, amax = 0;
    float mx = 0.f;
    if (r < kept) {
      cell = sorted_cell[kept_ord[r]];
      mx = pb[5LL * cells + cell];
      for (int c = 1; c < C; ++c) {
        const float v = pb[(long long)(5 + c) * cells + cell];
        if (v > mx) { mx = v; amax = c; }  // first max wins (torch.max / argmax)
      }
      flag = (min_cls > 0.f) ? (mx > min_cls) : true;
    }
    int tot;
    const int pos = out_n + block_rank<NMS_SCAN_THREADS>(flag, warp_tot, tot);
    if (flag) {
      float* o = rb + (long long)pos * D;
      if (xyxy) {
        const float4 bx = ws.cell_box[(long long)b * cells + cell];
        o[0] = bx.x; o[1] = bx.y; o[2] = bx.z; o[3] = bx.w;
      } else {
#pragma unroll
        for (int d = 0; d < 4; ++d) o[d] = pb[(long long)d * cells + cell];
      }
      for (int d = 4; d < D; ++d) o[d] = pb[(long long)d * cells + cell];
      kb[pos] = cell;
      // count_cells_for_formatted_preds: rows with max > 0 (default threshold) are counted
      if (mx > 0.f) atomicAdd(&s_hist[amax], 1);
    }
    out_n += tot;
  }
  __syncthreads();
  if (tid == 0) keep_count[b] = out_n;
  if (tid < C && s_hist[tid]) atomicAdd(&class_counts[tid], (unsigned long long)s_hist[tid]);
}

static int nms_group(int B, int cells) {
  const size_t per_img = (size_t)cells * cdiv(cells, NMS_CHUNK) * sizeof(unsigned long long);
  size_t g = NMS_MASK_CAP / per_img;
  if (g < 1) g = 1;
  if (g > 256) g = 256;
  return (int)(g < (size_t)B ? g : (size_t)B);
}
static size_t nms_ws_bytes(int B, int cells) {
  return (size_t)B * cells * (sizeof(int) * 2 + sizeof(float4) * 2 + sizeof(unsigned long long)) + (size_t)B * sizeof(int) +
         (size_t)nms_group(B, cells) * cells * cdiv(cells, NMS_CHUNK) * sizeof(unsigned long long) + 512;
}

}  // namespace yg
using namespace yg;

extern "C" size_t yg_format_preds_workspace(int B, int num_classes, int Sy, int Sx) {
  return nms_ws_bytes(B, Sy * Sx);
}

extern "C" int yg_format_preds_batch(const float* preds, int B, int num_classes, int Sy, int Sx,
                                     float obj_thresh, double iou_thresh, int xyxy, float min_class_conf,
                                     int* keep_count, float* rows, int* keep_index, long long* class_counts,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  YG_CHECK_ARG(preds && keep_count && rows && keep_index && class_counts, "format_preds: null pointer");
  const int cells = Sy * Sx;
  YG_CHECK_ARG(cells >= 1 && cells <= NMS_MAX_CELLS, "format_preds: Sy*Sx = %d exceeds %d", cells, NMS_MAX_CELLS);
  YG_CHECK_ARG(num_classes >= 1 && num_classes <= 27, "format_preds: num_classes %d", num_classes);
  cudaStream_t st = (cudaStream_t)stream;
  YG_CUDA(cudaMemsetAsync(class_counts, 0, sizeof(long long) * num_classes, st));
  if (B == 0) return YG_OK;
  const size_t need = nms_ws_bytes(B, cells);
  if (!workspace || workspace_bytes < need) {
    set_error("format_preds: workspace %zu < %zu", workspace_bytes, need);
    return YG_ERR_WORKSPACE;
  }
  // carve the workspace (16-byte aligned arrays first)
  unsigned char* p = (unsigned char*)workspace;
  p = (unsigned char*)(((uintptr_t)p + 255) & ~(uintptr_t)255);
  const int G = nms_group(B, cells), nw_stride = cdiv(cells, NMS_CHUNK);
  NmsWs ws;
  ws.cell_box = (float4*)p; p += (size_t)B * cells * sizeof(float4);
  ws.sorted_box = (float4*)p; p += (size_t)B * cells * sizeof(float4);
  ws.keys = (unsigned long long*)p; p += (size_t)B * cells * sizeof(unsigned long long);
  ws.mask = (unsigned long long*)p; p += (size_t)G * cells * nw_stride * sizeof(unsigned long long);
  ws.sorted_cell = (int*)p; p += (size_t)B * cells * sizeof(int);
  ws.kept_ord = (int*)p; p += (size_t)B * cells * sizeof(int);
  ws.n_cand = (int*)p;
  const int do_nms = iou_thresh > 0 ? 1 : 0;
  IouThr thr;
  thr.thr = iou_thresh;
  {
    float P = (float)iou_thresh;                       // nearest float; step down if it landed above the double threshold
    if ((double)P > iou_thresh) P = nextafterf(P, -INFINITY);
    const float F = nextafterf(P, INFINITY);           // smallest float > thr
    const double lo = (double)P * (1.0 - 1.0 / 1048576.0), hi = (double)F * (1.0 + 1.0 / 1048576.0);
    thr.t_lo = (float)lo; if ((double)thr.t_lo > lo) thr.t_lo = nextafterf(thr.t_lo, -INFINITY);
    thr.t_hi = (float)hi; if ((double)thr.t_hi < hi) thr.t_hi = nextafterf(thr.t_hi, INFINITY);
    if (!(thr.t_lo > 0.f) || !(thr.t_hi < 3.0e38f)) { thr.t_lo = 0.f; thr.t_hi = INFINITY; }   // degenerate thresholds: always the exact path
  }
  YG_CUDA(cudaMemsetAsync(ws.n_cand, 0, sizeof(int) * B, st));
  nms_candidates_kernel<<<dim3(cdiv(cells, 256), B), 256, 0, st>>>(preds, num_classes, cells, obj_thresh, do_nms, ws);
  YG_LAUNCH_CHECK("nms_candidates");
  int P = 1;
  while (P < cells) P <<= 1;
  const size_t smem = (size_t)P * sizeof(unsigned long long);
  static bool attr_set_dev[64] = {};   // the attribute is per device
  int dev_id = 0;
  cudaGetDevice(&dev_id);
  bool& attr_set = attr_set_dev[dev_id & 63];
  if (!attr_set) {
    YG_CUDA(cudaFuncSetAttribute(nms_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(NMS_MAX_CELLS * sizeof(unsigned long long))));
    YG_CUDA(cudaFuncSetAttribute(nms_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(NMS_SCAN_SMEM_WORDS * sizeof(unsigned long long))));
    attr_set = true;
  }
  nms_sort_kernel<<<B, NMS_THREADS, smem, st>>>(cells, ws);
  YG_LAUNCH_CHECK("nms_sort");
  int nsm = 148;
  for (int b0 = 0; b0 < B; b0 += G) {
    const int nb = (B - b0 < G) ? B - b0 : G;
    if (do_nms) {
      nms_mask_kernel<<<nsm * 16, NMS_CHUNK, 0, st>>>(b0, nb, cells, nw_stride, thr, ws);
      YG_LAUNCH_CHECK("nms_mask");
    }
    nms_scan_kernel<<<nb, NMS_SCAN_THREADS, NMS_SCAN_SMEM_WORDS * sizeof(unsigned long long), st>>>(preds, num_classes, cells, b0, nw_stride, do_nms, xyxy, min_class_conf,
                                                     keep_count, rows, keep_index, (unsigned long long*)class_counts, ws);
    YG_LAUNCH_CHECK("nms_scan");
  }
  return YG_OK;
}


// ------------------------------------------------------------------------------------------------
// Pairwise matching cost between labels and formatted predictions (SURVEY.md 8f N2):
// cost[i][j] = 1 - box_iou(label_i, pred_j), the matrix format_preds_and_labels_v2 hands to the Hungarian solver
// (/root/reference/yogo/utils/prediction_formatting.py:296-298; torchvision.ops.box_iou = _box_inter_union, boxes.py).
// Every operation is a single correctly rounded fp32 operation in torchvision's order (never contracted to FMA), so the
// matrix is bit-identical to the reference's and the assignment computed from it is the same.
// ------------------------------------------------------------------------------------------------
namespace yg {
__global__ void box_iou_cost_kernel(const float* __restrict__ a, int a_stride, int na, const float* __restrict__ b, int b_stride,
                                    int nb, float* __restrict__ cost) {
  box_iou_cost_tile(a, a_stride, na, b, b_stride, nb, cost, blockIdx.x * blockDim.x + threadIdx.x, blockIdx.y * 16);
}
}  // namespace yg

extern "C" int yg_box_iou_cost(const float* labels, int label_stride, int n_labels, const float* preds, int pred_stride,
                               int n_preds, float* cost, void* stream) {
  YG_CHECK_ARG(n_labels >= 0 && n_preds >= 0 && label_stride >= 4 && pred_stride >= 4, "box_iou_cost: bad sizes");
  if (n_labels == 0 || n_preds == 0) return YG_OK;
  YG_CHECK_ARG(labels && preds && cost, "box_iou_cost: null pointer");
  dim3 grid(cdiv(n_preds, 256), cdiv(n_labels, 16), 1);
  yg::box_iou_cost_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(labels, label_stride, n_labels, preds, pred_stride, n_preds, cost);
  YG_LAUNCH_CHECK("box_iou_cost");
  return YG_OK;
}
