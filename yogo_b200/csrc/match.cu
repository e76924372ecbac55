// Batched evaluation matching (SURVEY.md 8f N2): predictions of a whole batch matched to its labels with the assignment
// solved on the device.  Replaces the per-image loop over format_preds_and_labels_v2
// (/root/reference/yogo/utils/prediction_formatting.py:254-330: labelled-cell gather, 1 - box_iou cost,
// scipy.optimize.linear_sum_assignment on the host, matched / missed / extra gathers).
//
//   compact_labels_kernel  one CTA per image: the cells with label[0] != 0, in grid order (block scan, not atomics)
//   -- the host reads the per-image prediction / label counts once and sizes everything from them --
//   match_cost_kernel      every image's N x M cost matrix into one packed buffer (box_iou_cost_tile, as yg_box_iou_cost)
//   lsap_kernel            one warp per matrix: scipy's rectangular_lsap (shortest augmenting path, Crouse 2016),
//                          restated step for step so that row and column indices are identical to scipy's
//   match_gather_kernel    one CTA per image: matched pairs, missed labels, extra predictions in scipy's order
//
// The solver mirrors tools/lsap_np.py (linear_sum_assignment_np), which a CPU test pins to scipy.  Exactness: the costs
// are widened to double (exact), every reduced cost is ((minVal + c) - u) - v in three correctly rounded double
// operations (__dadd_rn / __dsub_rn, never contracted), and the column choice is the serial loop's argmin expressed as a total order, so a warp reduction in any
// order picks the same column: key (spc[j], assigned ? 1 : 0, assigned ? it : -it) with `it` the position in `remaining`.
#include "common.cuh"

namespace yg {

constexpr int MATCH_MAX_CELLS = 16384;   // Sy*Sx limit, as format_preds
constexpr int MATCH_THREADS = 256;       // gather kernel
constexpr int LABEL_THREADS = 1024;      // label compaction

// per-matrix workspace in 8-byte words: double u[nr], v[nc], spc[nc]; int path[nc], row4col[nc], remaining[nc],
// visited[nc], col4row[nr] (nr <= nc after the transpose)
__host__ __device__ inline long long lsap_words(int rows, int cols) {
  const long long nr = rows < cols ? rows : cols, nc = rows < cols ? cols : rows;
  return nr + 2 * nc + (4 * nc + nr + 1) / 2;
}

// ---- label compaction ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(LABEL_THREADS) compact_labels_kernel(const float* __restrict__ labels, int cells,
                                                                      float* __restrict__ rows, int* __restrict__ n_labels) {
  __shared__ int warp_tot[32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* lb = labels + (long long)b * 6 * cells;
  float* out = rows + (long long)b * cells * 6;
  int base = 0;
  for (int c0 = 0; c0 < cells; c0 += LABEL_THREADS) {
    const int c = c0 + tid;
    const bool flag = c < cells && lb[c] != 0.f;   // NaN counts as set, as for Tensor.bool()
    int tot;
    const int pos = base + block_rank<LABEL_THREADS>(flag, warp_tot, tot);
    if (flag) {
#pragma unroll
      for (int k = 0; k < 6; ++k) out[(long long)pos * 6 + k] = lb[(long long)k * cells + c];
    }
    base += tot;
  }
  if (tid == 0) n_labels[b] = base;
}

// ---- batched cost ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) match_cost_kernel(const float* __restrict__ label_rows, const float* __restrict__ pred_rows,
                                                        int cells, int D, const LsapDesc* __restrict__ desc, float* __restrict__ costs) {
  const int b = blockIdx.z;
  const LsapDesc d = desc[b];
  if ((int)blockIdx.x * 256 >= d.cols || (int)blockIdx.y * 16 >= d.rows) return;   // block-uniform
  box_iou_cost_tile(label_rows + (long long)b * cells * 6 + 1, 6, d.rows, pred_rows + (long long)b * cells * D, D, d.cols,
                    costs + d.cost_off, blockIdx.x * 256 + threadIdx.x, blockIdx.y * 16);
}

// ---- assignment: one warp per matrix -----------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) lsap_kernel(const float* __restrict__ costs, const LsapDesc* __restrict__ desc, int n_mat,
                                                 double* __restrict__ ws, long long* __restrict__ out_rows,
                                                 long long* __restrict__ out_cols, int* __restrict__ status) {
  const unsigned FULL = 0xffffffffu;
  const int m = blockIdx.x, lane = threadIdx.x;
  if (m >= n_mat) return;
  const LsapDesc d = desc[m];
  const int R = d.rows, Cc = d.cols;
  const bool tr = Cc < R;   // tall matrix: solve the transpose (its rows are the original columns)
  const int nr = tr ? Cc : R, nc = tr ? R : Cc;
  const float* c = costs + d.cost_off;
  const long long si = tr ? 1 : Cc, sj = tr ? Cc : 1;   // element (i, j) of the solved matrix is c[i * si + j * sj]
  if (nr == 0) {
    if (lane == 0) status[m] = YG_LSAP_OK;
    return;
  }
  bool bad = false;
  for (long long k = lane; k < (long long)R * Cc; k += 32) {
    const float x = c[k];
    bad |= (x != x) || (x == -INFINITY);
  }
  if (__any_sync(FULL, bad)) {
    if (lane == 0) status[m] = YG_LSAP_INVALID;
    return;
  }
  double* __restrict__ u = ws + d.ws_off;
  double* __restrict__ v = u + nr;
  double* __restrict__ spc = v + nc;
  int* __restrict__ path = reinterpret_cast<int*>(spc + nc);
  int* __restrict__ row4col = path + nc;
  int* __restrict__ remaining = row4col + nc;
  int* __restrict__ visited = remaining + nc;   // columns taken by the current augmentation, in order
  int* __restrict__ col4row = visited + nc;
  for (int k = lane; k < nr; k += 32) { u[k] = 0.0; col4row[k] = -1; }
  for (int k = lane; k < nc; k += 32) { v[k] = 0.0; row4col[k] = -1; path[k] = -1; }
  __syncwarp();

  int st = YG_LSAP_OK;
  for (int cur = 0; cur < nr; ++cur) {
    for (int k = lane; k < nc; k += 32) { remaining[k] = nc - 1 - k; spc[k] = INFINITY; }
    __syncwarp();
    double minVal = 0.0;
    int i = cur, sink = -1, nrem = nc, nvis = 0;
    while (sink < 0 && nrem > 0) {   // each step removes one column: at most nc steps
      const double ui = u[i];
      const float* ci = c + (long long)i * si;
      double best = INFINITY;
      int bt = 0x7fffffff, bj = -1, br = -1;
      for (int it = lane; it < nrem; it += 32) {
        const int j = remaining[it];
        const double r = __dsub_rn(__dsub_rn(__dadd_rn(minVal, (double)ci[(long long)j * sj]), ui), v[j]);
        double s = spc[j];
        if (r < s) { path[j] = i; spc[j] = r; s = r; }
        const int r4c = row4col[j];
        const int t = r4c < 0 ? nc - 1 - it : nc + it;   // the tie-break part of the key as one integer
        if (s < best || (s == best && t < bt)) { best = s; bt = t; bj = j; br = r4c; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(FULL, best, o);
        const int ot = __shfl_xor_sync(FULL, bt, o), oj = __shfl_xor_sync(FULL, bj, o), orr = __shfl_xor_sync(FULL, br, o);
        if (ob < best || (ob == best && ot < bt)) { best = ob; bt = ot; bj = oj; br = orr; }
      }
      minVal = best;
      if (best == INFINITY) { st = YG_LSAP_INFEASIBLE; break; }
      const int sel = bt < nc ? nc - 1 - bt : bt - nc;
      __syncwarp();   // every lane has read `remaining` and written its spc / path entries
      if (lane == 0) {
        visited[nvis] = bj;
        remaining[sel] = remaining[nrem - 1];
      }
      ++nvis;
      --nrem;
      if (br < 0) sink = bj; else i = br;
      __syncwarp();
    }
    if (st == YG_LSAP_OK && sink < 0) st = YG_LSAP_INFEASIBLE;   // (not reachable with nr <= nc)
    if (st != YG_LSAP_OK) break;
    // dual update over the rows and columns this augmentation visited: the rows other than cur are row4col[j] of the
    // visited columns other than the sink (before the augmentation rewires them)
    if (lane == 0) u[cur] = __dadd_rn(u[cur], minVal);
    for (int s = lane; s < nvis; s += 32) {
      const int j = visited[s];
      const double dl = __dsub_rn(minVal, spc[j]);
      if (j != sink) { const int k = row4col[j]; u[k] = __dadd_rn(u[k], dl); }
      v[j] = __dsub_rn(v[j], dl);
    }
    __syncwarp();
    if (lane == 0) {   // augment along the path back to cur: at most nr links
      int j = sink;
      for (int guard = 0; guard < nr; ++guard) {
        const int r = path[j];
        row4col[j] = r;
        const int t = col4row[r];
        col4row[r] = j;
        j = t;
        if (r == cur) break;
      }
    }
    __syncwarp();
  }
  if (st == YG_LSAP_OK) {
    // (row, column) pairs in ascending original row: scipy's order for both the plain and the transposed problem
    const int* match = tr ? row4col : col4row;   // original row -> original column, or -1
    const int k0 = min(R, Cc);
    int base = 0;
    for (int r0 = 0; r0 < R; r0 += 32) {
      const int r = r0 + lane;
      const int col = r < R ? match[r] : -1;
      const unsigned bal = __ballot_sync(FULL, col >= 0);
      if (col >= 0) {
        const int pos = base + __popc(bal & ((1u << lane) - 1u));
        if (pos < k0) { out_rows[d.out_off + pos] = r; out_cols[d.out_off + pos] = col; }
      }
      base += __popc(bal);
    }
  }
  if (lane == 0) status[m] = st;
}

// ---- matched / missed / extra rows ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(MATCH_THREADS) match_gather_kernel(
    const float* __restrict__ label_rows, const float* __restrict__ pred_rows, int cells, int D, const LsapDesc* __restrict__ desc,
    const long long* __restrict__ gather_off, const long long* __restrict__ pair_rows, const long long* __restrict__ pair_cols,
    const int* __restrict__ status, float* __restrict__ out_preds, float* __restrict__ out_labels, float* __restrict__ missed, float* __restrict__ extra) {
  __shared__ unsigned char used_l[MATCH_MAX_CELLS], used_p[MATCH_MAX_CELLS];
  __shared__ int warp_tot[32];
  const int b = blockIdx.x, tid = threadIdx.x;
  if (status[b] != YG_LSAP_OK) return;   // the solver wrote no pairs for this image; the caller raises
  const LsapDesc d = desc[b];
  const int N = d.rows, M = d.cols, K = min(N, M);
  const float* lb = label_rows + (long long)b * cells * 6;
  const float* pb = pred_rows + (long long)b * cells * D;
  for (int k = tid; k < N; k += MATCH_THREADS) used_l[k] = 0;
  for (int k = tid; k < M; k += MATCH_THREADS) used_p[k] = 0;
  __syncthreads();
  for (int t = tid; t < K; t += MATCH_THREADS) {
    const long long o = d.out_off + t;
    const int r = (int)pair_rows[o], cc = (int)pair_cols[o];
    used_l[r] = 1;
    used_p[cc] = 1;
#pragma unroll
    for (int k = 0; k < 6; ++k) out_labels[o * 6 + k] = lb[(long long)r * 6 + k];
    for (int k = 0; k < D; ++k) out_preds[o * D + k] = pb[(long long)cc * D + k];
  }
  __syncthreads();
  // missed labels in ascending label index, then extra predictions in ascending prediction (NMS) index
  int base = 0;
  for (int r0 = 0; r0 < N; r0 += MATCH_THREADS) {
    const int r = r0 + tid;
    const bool flag = r < N && !used_l[r];
    int tot;
    const int pos = base + block_rank<MATCH_THREADS>(flag, warp_tot, tot);
    if (flag) {
      const long long o = gather_off[2 * b] + pos;
#pragma unroll
      for (int k = 0; k < 6; ++k) missed[o * 6 + k] = lb[(long long)r * 6 + k];
    }
    base += tot;
  }
  base = 0;
  for (int c0 = 0; c0 < M; c0 += MATCH_THREADS) {
    const int cc = c0 + tid;
    const bool flag = cc < M && !used_p[cc];
    int tot;
    const int pos = base + block_rank<MATCH_THREADS>(flag, warp_tot, tot);
    if (flag) {
      const long long o = gather_off[2 * b + 1] + pos;
      for (int k = 0; k < D; ++k) extra[o * D + k] = pb[(long long)cc * D + k];
    }
    base += tot;
  }
}

static int lsap_launch(const float* costs, const LsapDesc* desc, int n, void* ws, long long* out_rows, long long* out_cols,
                       int* status, cudaStream_t st) {
  lsap_kernel<<<n, 32, 0, st>>>(costs, desc, n, (double*)ws, out_rows, out_cols, status);
  YG_LAUNCH_CHECK("lsap");
  return YG_OK;
}

}  // namespace yg
using namespace yg;

extern "C" int yg_compact_labels(const float* labels, int B, int Sy, int Sx, float* rows, int* n_labels, void* stream) {
  YG_CHECK_ARG(B >= 0 && Sy > 0 && Sx > 0, "compact_labels: bad sizes");
  if (B == 0) return YG_OK;
  YG_CHECK_ARG(labels && rows && n_labels, "compact_labels: null pointer");
  compact_labels_kernel<<<B, LABEL_THREADS, 0, (cudaStream_t)stream>>>(labels, Sy * Sx, rows, n_labels);
  YG_LAUNCH_CHECK("compact_labels");
  return YG_OK;
}

extern "C" long long yg_lsap_workspace_words(int rows, int cols) {
  if (rows < 0 || cols < 0) return -1;
  return lsap_words(rows, cols);
}

extern "C" int yg_lsap_batch(const float* costs, const void* desc, int n, void* workspace, long long* out_rows, long long* out_cols,
                             int* status, void* stream) {
  YG_CHECK_ARG(n >= 0, "lsap_batch: n = %d", n);
  if (n == 0) return YG_OK;
  YG_CHECK_ARG(desc && status, "lsap_batch: null pointer");
  return lsap_launch(costs, (const LsapDesc*)desc, n, workspace, out_rows, out_cols, status, (cudaStream_t)stream);
}

extern "C" int yg_match_batch(const float* label_rows, const float* pred_rows, int B, int cells, int num_classes, int max_labels,
                              int max_preds, const void* desc, const long long* gather_off, float* costs, void* workspace,
                              long long* pair_rows, long long* pair_cols, int* status, float* out_preds, float* out_labels,
                              float* missed, float* extra, void* stream) {
  YG_CHECK_ARG(B >= 0 && B <= 65535, "match_batch: B = %d", B);
  YG_CHECK_ARG(cells >= 1 && cells <= MATCH_MAX_CELLS, "match_batch: Sy*Sx = %d exceeds %d", cells, MATCH_MAX_CELLS);
  YG_CHECK_ARG(num_classes >= 1 && max_labels >= 0 && max_labels <= cells && max_preds >= 0 && max_preds <= cells,
               "match_batch: bad sizes");
  if (B == 0) return YG_OK;
  YG_CHECK_ARG(label_rows && pred_rows && desc && gather_off && status, "match_batch: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const LsapDesc* d = (const LsapDesc*)desc;
  const int D = 5 + num_classes;
  if (max_labels > 0 && max_preds > 0) {
    match_cost_kernel<<<dim3(cdiv(max_preds, 256), cdiv(max_labels, 16), B), 256, 0, st>>>(label_rows, pred_rows, cells, D, d, costs);
    YG_LAUNCH_CHECK("match_cost");
  }
  const int rc = lsap_launch(costs, d, B, workspace, pair_rows, pair_cols, status, st);
  if (rc != YG_OK) return rc;
  match_gather_kernel<<<B, MATCH_THREADS, 0, st>>>(label_rows, pred_rows, cells, D, d, gather_off, pair_rows, pair_cols, status, out_preds,
                                                   out_labels, missed, extra);
  YG_LAUNCH_CHECK("match_gather");
  return YG_OK;
}
