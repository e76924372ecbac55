/*
 * yogo_b200 - C ABI of the B200-native YOGO hot path (libyogo_b200.so).
 *
 * The reference (czbiohub-sf/yogo) has no native boundary of its own: its hot path calls
 * torch / torchvision library kernels from Python (SURVEY.md 2.2, 8b).  This header is
 * the boundary a maintainer binds instead; each entry point cites the reference call
 * site it replaces.  Conventions:
 *   - extern "C", plain pointers and sizes, no torch types.  All data pointers are DEVICE
 *     pointers unless the name ends in _host.  The library never owns tensor memory.
 *   - every function returns 0 on success or a negative yg_status; yg_last_error()
 *     returns a thread-local message.  No C++ exception crosses the ABI.
 *   - every launch is asynchronous on the caller's stream (last argument, a cudaStream_t
 *     passed as void*).
 *   - activations are NHWC; `dtype` selects their storage: YG_F32 or YG_BF16 (accumulation
 *     is always fp32).  Parameters and parameter gradients are fp32 in the reference's
 *     OIHW layout (state_dict compatible, model.py:94-147).
 */
#ifndef YOGO_B200_H
#define YOGO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  YG_OK = 0,
  YG_ERR_INVALID = -1,   /* bad argument / unsupported shape */
  YG_ERR_CUDA = -2,      /* CUDA runtime / driver error (message has the string) */
  YG_ERR_ARCH = -3,      /* device is not sm_100 */
  YG_ERR_WORKSPACE = -4  /* workspace too small */
} yg_status;

enum { YG_F32 = 0, YG_BF16 = 1, YG_U8 = 2 };
enum { YG_ACT_NONE = 0, YG_ACT_LRELU = 1, YG_ACT_SILU = 2 }; /* LeakyReLU(0.01) / SiLU */
enum { YG_IMPL_AUTO = 0, YG_IMPL_SIMT = 1, YG_IMPL_TCGEN05 = 2 };

int yg_version(void);
const char* yg_last_error(void);
/* 0 if the current device is compute capability 10.x, YG_ERR_ARCH otherwise. */
int yg_device_check(void);
/* Process-wide implementation switch for the 3x3 convolutions (AUTO = tcgen05 where the
 * shape qualifies, SIMT otherwise).  Used by the parity tests to cross-check both. */
int yg_set_conv_impl(int impl);
int yg_get_conv_impl(void);
/* option word of the convolution engines (default 0).  yg_set_tc_options returns YG_ERR_INVALID for any other bit.
 * bits 7-11 = profiling knobs of the tcgen05 engine read by tools/bench_conv.py: 7 = no global stores, 8 = no MMA issue,
 * 9 = the epilogue skips its TMEM loads and math, 10 = no TMA loads, 11 = cycle counters of the MMA and epilogue warps
 * (read with yg_tc_debug_read);
 * bit 21 = fp32 tensors as split-bf16 "x3" convolutions on the tensor cores (csrc/x3.cu; yogo_b200.set_fp32_tensor_cores;
 * off by default: the exact SIMT kernels are the fp32 parity path). */
int yg_set_tc_options(int options);
int yg_get_tc_options(void);
/* profiling hook: copies n (<= 2048) cycle counters written by the engine's MMA warps (8 per CTA) to host memory. */
int yg_tc_debug_read(unsigned long long* out, int n);
/* number of CUDA kernels this library has launched in this process (bench.py gpu_launches). */
unsigned long long yg_launch_count(void);

/* ---- epilogue descriptor shared by the convolution entry points -------------------- */
typedef struct {
  const float* scale;      /* [Cout] or NULL (=1): folded BatchNorm scale in eval mode   */
  const float* shift;      /* [Cout] or NULL (=0): conv bias, or folded BN shift         */
  int act;                 /* YG_ACT_*                                                   */
  const float* dropscale;  /* [N*Cout] or NULL: Dropout2d keep/(1-p) per (n, c)          */
  double* stats;           /* [2*Cout] or NULL: += sum(v), sum(v*v) of v = acc*scale+shift
                              (BatchNorm batch statistics, taken before act)             */
  void* preact;            /* NHWC, same dtype as y, or NULL: v before the activation    */
  void* actmask;           /* [N*Ho*Wo*Cout/8] bytes or NULL: bit e (NHWC element index, bit e%8 of byte
                              e/8) = (v > 0).  One bit instead of 16 to carry LeakyReLU's slope to
                              the backward pass; honoured by yg_conv_fwd, needs Cout % 32 == 0 */
} yg_fwd_epilogue;

typedef struct {
  const void* saved;       /* NHWC tensor of the layer that produced this input:
                              post-activation output (lrelu, no BN), pre-activation
                              (silu, no BN) or raw conv output (BN); NULL = no act bwd  */
  int act;                 /* YG_ACT_* of that layer                                     */
  const float* dropscale;  /* [N*Cin] or NULL                                            */
  const float* bn_scale;   /* [Cin] gamma*invstd, NULL if that layer has no BN           */
  const float* bn_shift;   /* [Cin] beta - mean*gamma*invstd                             */
  const float* bn_mean;    /* [Cin]                                                      */
  const float* bn_invstd;  /* [Cin]                                                      */
  double* bn_sums;         /* [2*Cin]: += sum(g), sum(g*xhat)                            */
  const void* actmask;     /* the producer's yg_fwd_epilogue.actmask or NULL.  Used instead of `saved`
                              by the tcgen05 path when act is LeakyReLU and that layer has no BN
                              (16x less data to read); other paths read `saved`, so pass both */
} yg_bwd_epilogue;

/* ---- first layer: direct stencil on the NCHW image (Cin = 1 or 3) -------------------
 * replaces nn.Conv2d(input_channels, C1, 3, stride=2, padding=1) (+BatchNorm2d+act),
 * /root/reference/yogo/model_defns.py:33-37.  x is (N,Cin,H,W) in x_dtype (YG_U8 or
 * YG_F32; YOGO.forward's `x.float()` of model.py:272-273 is folded in), w is OIHW fp32.
 * If ep->stats is set and y is NULL only the statistics are accumulated (pass 1 of
 * train-mode BN); otherwise y (NHWC, dtype) is written. */
int yg_conv_first_fwd(const void* x, int x_dtype, const float* w, void* y, int dtype,
                      int N, int H, int W, int Cin, int Cout, int stride,
                      const yg_fwd_epilogue* ep, void* stream);
/* backward of the first layer from da = grad wrt its (post-activation) output.
 * pass 1 (bn_sums != NULL in `be`, dw == NULL): accumulate BN backward sums.
 * pass 2 (dw != NULL): dW (OIHW fp32, overwritten) and, if dshift, d(bias or beta);
 *   bn_dy_mean/bn_dyx_mean = sums/M from pass 1 (NULL when no BN). */
int yg_conv_first_bwd(const void* x, int x_dtype, const float* w, const void* da, int dtype,
                      int N, int H, int W, int Cin, int Cout, int stride,
                      const yg_bwd_epilogue* be, const float* fwd_shift,
                      const float* bn_dy_mean, const float* bn_dyx_mean,
                      float* dw, float* dshift, float clip, void* workspace, size_t workspace_bytes,
                      void* stream);
size_t yg_conv_first_bwd_workspace(int Cin, int Cout);
/* Single-channel images (Cin == 1): the 9-tap Gram statistics of the image, gram[54] = S[9] then the upper
 * triangle of G[9][9] (fp64, overwritten).  With them the BatchNorm batch statistics of the first layer
 * (yg_conv_first_stats_from_gram: stats[2*Cout] += sum y, sum y^2) and the BN part of its backward
 * (yg_conv_first_bwd_finalize, from P = sum g*x_t and Sg = sum g as produced by yg_conv_first_bwd with
 * bn_dy_mean == NULL) follow in closed form instead of extra passes over the 16-channel activations. */
int yg_conv_first_gram(const void* x, int x_dtype, int N, int H, int W, int stride, double* gram, void* stream);
int yg_conv_first_stats_from_gram(const double* gram, const float* w, const float* bias, double count, int Cout,
                                  double* stats, void* stream);
int yg_conv_first_bwd_finalize(const float* P, const float* Sg, const double* gram, const float* w, const float* bias,
                               const float* gamma, const float* mean, const float* invstd, double count,
                               int batch_stats, float clip, int Cout, float* dw, float* dbias, float* dgamma,
                               float* dbeta, void* stream);
/* Gradient wrt the fp32 NCHW image x (N,Cin,H,W) of the first layer: dx (fp32 NCHW, overwritten, not clamped) =
 * conv_transpose(dz, w) with dz = d(loss)/d(conv output) recomputed from x and da = grad wrt the block's (post-activation,
 * post-Dropout2d) output (NHWC, dtype) exactly as yg_conv_first_bwd does: g' = da * dropscale * act'(pre), then
 * dz = bn_scale*(g' - bn_dy_mean - xhat*bn_dyx_mean) for train-mode BatchNorm (the means of g' and g'*xhat over the
 * N*Ho*Wo pixels), dz = bn_scale*g' when both means are NULL (running statistics), dz = g' when `be` has no BN.
 * `be` and fwd_shift as for yg_conv_first_bwd (be->saved and be->bn_sums are not used).
 * yg_conv_first_bn_means: those two means on the Gram path, from its raw P[Cout*9] / Sg[Cout] (yg_conv_first_bwd with
 * bn_dy_mean == NULL and clip 0): dy_mean = Sg/count, dyx_mean = invstd*(sum_t w_t P_t + (bias - mean)*Sg)/count. */
int yg_conv_first_dgrad(const float* x, const float* w, const void* da, int dtype, int N, int H, int W, int Cin, int Cout,
                        int stride, const yg_bwd_epilogue* be, const float* fwd_shift, const float* bn_dy_mean,
                        const float* bn_dyx_mean, float* dx, void* stream);
int yg_conv_first_bn_means(const float* P, const float* Sg, const float* w, const float* bias, const float* mean,
                           const float* invstd, double count, int Cout, float* dy_mean, float* dyx_mean, void* stream);

/* Alignment: activation tensors handed to the convolution entry points should be 32-byte aligned (torch allocations are
 * 256-byte aligned); tensors that are only 16-byte aligned run on the generic SIMT path. */
/* ---- generic convolution (3x3 pad 1 or 1x1 pad 0, stride 1 or 2), NHWC -------------
 * replaces nn.Conv2d fprop / dgrad / wgrad (cuDNN) at model_defns.py:34-67 and the
 * elementwise BatchNorm/LeakyReLU/SiLU/Dropout2d kernels that follow each conv. */
int yg_conv_fwd(const void* x, const float* w_oihw, void* y, int dtype,
                int N, int H, int W, int Cin, int Cout, int ksize, int stride,
                const yg_fwd_epilogue* ep, void* stream);
/* dx = conv_transpose(dz, w); the epilogue turns it into the gradient wrt the previous
 * layer's conv output (activation / dropout / BN-sum fusion), see yg_bwd_epilogue. */
int yg_conv_dgrad(const void* dz, const float* w_oihw, void* dx, int dtype,
                  int N, int H, int W, int Cin, int Cout, int ksize, int stride,
                  const yg_bwd_epilogue* be, void* stream);
/* dw (OIHW fp32) = sum over pixels dz * x ; dbias[Cout] = sum dz (NULL to skip).
 * Both are clamped to [-clip, clip] (YOGO's per-parameter grad hook, model.py:76-77);
 * clip <= 0 disables.  Deterministic split-K through `workspace`. */
size_t yg_conv_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int ksize, int stride);
int yg_conv_wgrad(const void* x, const void* dz, float* dw, float* dbias, int dtype,
                  int N, int H, int W, int Cin, int Cout, int ksize, int stride,
                  float clip, void* workspace, size_t workspace_bytes, void* stream);

/* ---- BatchNorm2d pieces (nn.BatchNorm2d, model_defns.py:35,55,60) ------------------ */
/* from stats (sum, sumsq over M = N*H*W values per channel): mean, invstd, fused
 * scale/shift, and the running-stat update (momentum 0.1, unbiased variance). */
int yg_bn_finalize(const double* stats, double count, const float* gamma, const float* beta,
                   float* running_mean, float* running_var, float momentum, float eps,
                   float* mean, float* invstd, float* scale, float* shift, int C, void* stream);
/* eval mode: scale = gamma/sqrt(rv+eps), shift = beta - rm*scale (+ conv_bias*scale). */
int yg_bn_fold_eval(const float* gamma, const float* beta, const float* running_mean,
                    const float* running_var, const float* conv_bias, float eps,
                    float* scale, float* shift, int C, void* stream);
/* a = act(y*scale[c] + shift[c]) * dropscale[n,c]   (elementwise, NHWC); actmask (or NULL): sign bits of the
 * activation input, same format as yg_fwd_epilogue.actmask (needs C % 8 == 0). */
int yg_bn_act_apply(const void* y, void* a, int dtype, int N, int HW, int C,
                    const float* scale, const float* shift, int act, const float* dropscale,
                    void* actmask, void* stream);
/* stats[0..C) += sum(y), stats[C..2C) += sum(y*y) over the N*HW pixels of an NHWC tensor (train-mode batch statistics
 * of a convolution output in one streaming pass; the alternative is yg_fwd_epilogue.stats).  C % 8 == 0. */
int yg_bn_stats(const void* y, int dtype, int N, int HW, int C, double* stats, void* stream);
/* sums[0..C) += sum(g), sums[C..2C) += sum(g * xhat), xhat = (y - mean) * invstd: the two reductions of BatchNorm
 * backward for a gradient g that already includes the activation backward (the alternative is yg_bwd_epilogue.bn_sums). */
int yg_bn_bwd_sums(const void* g, const void* y, int dtype, int N, int HW, int C, const float* mean,
                   const float* invstd, double* sums, void* stream);
/* dz = gamma*invstd*(g - sum_g/M - xhat*sum_gx/M) in place over g (batch_stats != 0), or
 * dz = gamma*invstd*g when the layer ran with running statistics (batch_stats == 0, BN in
 * eval mode inside a training graph: YOGO(tuning=True), model.py:69-70).  Also writes
 * dgamma = clamp(sum_gx), dbeta = clamp(sum_g). y = raw conv output (for xhat). */
int yg_bn_bwd_apply(void* g, const void* y, int dtype, int N, int HW, int C,
                    const double* sums, const float* gamma, const float* mean, const float* invstd,
                    float* dgamma, float* dbeta, float clip, int batch_stats, void* stream);

/* ---- head: 1x1 conv to 5+C channels fused with YOGO.forward's transform -------------
 * replaces model_defns.py:67 + model.py:277-313.  x NHWC (N,Sy,Sx,Cin) -> out (N,5+C,Sy,Sx)
 * fp32 NCHW; t_raw (N,Sy,Sx,5+C) fp32 keeps the raw logits for the backward (or NULL).
 * cxs/cys: the module's _Cxs/_Cys buffers (Sy*Sx fp32, model.py:48-59) or NULL to recompute. */
int yg_head_fwd(const void* x, int dtype, const float* w, const float* bias, float* out, float* t_raw,
                int N, int Sy, int Sx, int Cin, int num_classes,
                float anchor_w, float anchor_h, float width_mult, float height_mult,
                int inference, const float* cxs, const float* cys, void* stream);
/* dpred (N,5+C,Sy,Sx) fp32 + t_raw -> dx NHWC (with the previous block's bwd epilogue),
 * dw (OIHW [5+C,Cin,1,1]) and dbias, clamped.  dw == NULL skips both parameter gradients (dbias is ignored): the
 * backward of a frozen model.  dpred is the gradient wrt the raw class logits: for a head run with inference != 0 pass
 * it through yg_head_softmax_bwd first. */
size_t yg_head_bwd_workspace(int N, int Sy, int Sx, int Cin, int num_classes);
int yg_head_bwd(const float* dpred, const float* t_raw, const void* x, const float* w, void* dx, int dtype,
                float* dw, float* dbias, int N, int Sy, int Sx, int Cin, int num_classes,
                float anchor_w, float anchor_h, float width_mult, float height_mult,
                const yg_bwd_epilogue* be, float clip, void* workspace, size_t workspace_bytes,
                void* stream);
/* Softmax backward of the inference head (yg_head_fwd with inference != 0): out (N,5+C,Sy,Sx) fp32 = dpred with its class
 * planes replaced by p * (dp - sum_j p_j dp_j), p = softmax of the raw class logits in t_raw computed as yg_head_fwd
 * computes it; planes 0-4 are copied.  out must not overlap dpred. */
int yg_head_softmax_bwd(const float* dpred, const float* t_raw, float* out, int N, int Sy, int Sx, int num_classes,
                        void* stream);

/* ---- YOGOLoss forward + backward in one pass -----------------------------------------
 * replaces yogo_loss.py:38-129 (+ torchvision box_convert / complete_box_iou_loss).
 * pred (N,5+C,Sy,Sx) fp32, label (N,6,Sy,Sx) fp32.  out4 (device, 4 floats) =
 * [loss, iou_loss, objectness_loss, classification_loss]; dpred may be NULL. */
size_t yg_yogo_loss_workspace(int N, int Sy, int Sx);
int yg_yogo_loss_fwd_bwd(const float* pred, const float* label, float* out4, float* dpred,
                         int N, int num_classes, int Sy, int Sx,
                         float no_obj_weight, float iou_weight, float classify_weight,
                         float label_smoothing, void* workspace, size_t workspace_bytes, void* stream);

/* ---- threshold + NMS + per-class counts, whole batch ----------------------------------
 * replaces format_preds (utils/prediction_formatting.py:23-93, torchvision.ops.nms) and
 * get_prediction_class_counts (infer.py:60-124).  preds (B,5+C,Sy,Sx) fp32.
 * Outputs: keep_count[B] (int32), rows (B, Sy*Sx, 5+C) fp32 - image b's kept rows packed
 * at rows[b][0..keep_count[b]) in the reference's output order - keep_index (B, Sy*Sx)
 * int32 grid-cell index of each kept row, class_counts[C] (int64, summed over the batch,
 * overwritten).  xyxy != 0 returns converted boxes (box_format="xyxy"). */
size_t yg_format_preds_workspace(int B, int num_classes, int Sy, int Sx);
int yg_format_preds_batch(const float* preds, int B, int num_classes, int Sy, int Sx,
                          float obj_thresh, double iou_thresh, int xyxy, float min_class_conf,
                          int* keep_count, float* rows, int* keep_index, long long* class_counts,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- evaluation matching (SURVEY.md 8f N2) ------------------------------------------------
 * cost[i][j] = 1 - IoU(label box i, prediction box j), the matrix format_preds_and_labels_v2 gives to the Hungarian
 * solver (utils/prediction_formatting.py:296-298, torchvision.ops.box_iou); bit-identical to the reference's.
 * labels / preds: rows of label_stride / pred_stride floats whose first four are xyxy (pass labels + 1 for
 * [mask, x1, y1, x2, y2, class] rows); cost (n_labels, n_preds) fp32, row-major. */
int yg_box_iou_cost(const float* labels, int label_stride, int n_labels, const float* preds, int pred_stride,
                    int n_preds, float* cost, void* stream);

/* Batched matching (format_preds_and_labels_v2 for a whole batch, the assignment solved on the device).
 * yg_compact_labels: labels (B,6,Sy,Sx) fp32 -> rows (B, Sy*Sx, 6), image b's labelled cells (label[0] != 0, NaN
 * included) packed at rows[b][0..n_labels[b]) in grid order.
 * yg_lsap_batch: scipy.optimize.linear_sum_assignment of n fp32 matrices in one launch, identical indices.  desc (device,
 * n x 4 int64) per matrix = [cost_off (floats into costs, row-major), ws_off (8-byte words into workspace, each matrix
 * needs yg_lsap_workspace_words(rows, cols), a host function), out_off, rows | cols << 32]; out_rows / out_cols (int64)
 * get the min(rows, cols) assigned pairs at out_off in ascending row; status[n] (int32) is always written with a
 * yg_lsap_status, and outputs of a matrix whose status is not YG_LSAP_OK are undefined.
 * yg_match_batch: after yg_format_preds_batch (xyxy rows) and yg_compact_labels, with desc[b] = (rows = labels of image b,
 * cols = its kept predictions) and gather_off (device, B x 2 int64) = offsets of image b's missed / extra rows: one
 * launch each for the cost matrices (into costs, same expression as yg_box_iou_cost), the assignment and the gather of
 * out_preds (K, 5+C) / out_labels (K, 6) matched pairs in ascending label, missed (., 6) labels in ascending label and
 * extra (., 5+C) predictions in ascending prediction index.  max_labels / max_preds bound the per-image counts. */
enum { YG_LSAP_OK = 0, YG_LSAP_INVALID = 1 /* NaN or -inf entry */, YG_LSAP_INFEASIBLE = 2 /* a row cannot be assigned */ };
int yg_compact_labels(const float* labels, int B, int Sy, int Sx, float* rows, int* n_labels, void* stream);
long long yg_lsap_workspace_words(int rows, int cols);
int yg_lsap_batch(const float* costs, const void* desc, int n, void* workspace, long long* out_rows, long long* out_cols,
                  int* status, void* stream);
int yg_match_batch(const float* label_rows, const float* pred_rows, int B, int cells, int num_classes, int max_labels,
                   int max_preds, const void* desc, const long long* gather_off, float* costs, void* workspace,
                   long long* pair_rows, long long* pair_cols, int* status, float* out_preds, float* out_labels,
                   float* missed, float* extra, void* stream);

/* Evaluation metrics (yogo_b200.metrics.Metrics), after yg_match_batch with the same rows, desc and gather_off.
 * yg_confusion_batch: adds to confusion (int64, row-major nb x nb, nb = num_classes + 1 with include_background, else
 * num_classes; rows = true class, columns = predicted class) the confusion matrix of
 * PredictionLabelMatch.convert_background_errors(num_classes + 1): matched pairs (int(label[5]), argmax of the class
 * columns and an appended 0), missed labels (int(label[5]), num_classes), extra predictions (num_classes, argmax of the
 * class columns and an appended 0); without background only matched pairs, argmax over the class columns alone.
 * out_preds / out_labels / missed / extra are yg_match_batch's outputs; lsap_status[B] its status (images whose status is
 * not YG_LSAP_OK are skipped).  label_status[B] (int32) is written 1 for an image with a label class outside
 * [0, num_classes) (such labels are not counted), else 0.
 * yg_coco_match_batch: COCOeval.evaluateImg (bbox, no crowd, area "all", maxDet 100) of every image and class.  Detections
 * are the kept xyxy rows of yg_format_preds_batch (pred_rows (B, cells, 5+C)), class = argmax of the class columns,
 * score = objectness; ground truths are yg_compact_labels' rows (class int(label[5]), box label[1:5]).  iou_thrs (HOST,
 * YG_COCO_IOU_THRS doubles) are COCO's np.linspace(.5, .95, 10).  Writes one record per kept detection, image b's at
 * [prefix of the kept counts of images < b, + its kept count), in (class, rank) order: records (int32 n x 4) = [score
 * (fp32 bits), class, image0 + b, rank | matched mask << 16] with rank the position within (image, class) by score
 * descending then row index, and bit t of the mask set when the detection matched a ground truth at iou_thrs[t] (only
 * ranks < 100 are matched); keys (int64 n) = class << 32 | a 32-bit key ascending in descending score, for a stable sort.
 * Adds the per-class ground-truth counts to gt_count (int64 [num_classes]).  max_labels / max_preds bound the per-image
 * counts (they size the shared memory).
 * yg_coco_accumulate: COCOeval.accumulate over n_records records in the order perm (int64) that stably sorts keys
 * (sorted_keys = keys[perm]), for every class, IoU threshold and maxDet in (1, 10, 100); rec_thrs (HOST,
 * YG_COCO_REC_THRS doubles) = np.linspace(0, 1, 101).  precision (double [T][R][num_classes][3]) and recall
 * (double [T][num_classes][3]) are overwritten, COCOeval's eval["precision"] / eval["recall"] without the area axis: -1
 * for a class with gt_count 0. */
enum { YG_COCO_IOU_THRS = 10, YG_COCO_REC_THRS = 101 };
int yg_confusion_batch(const float* out_preds, const float* out_labels, const float* missed, const float* extra, int B,
                       int num_classes, int include_background, const void* desc, const long long* gather_off,
                       const int* lsap_status, int* label_status, long long* confusion, void* stream);
int yg_coco_match_batch(const float* pred_rows, const float* label_rows, int B, int cells, int num_classes, int max_labels,
                        int max_preds, const void* desc, const long long* gather_off, long long image0, const double* iou_thrs,
                        int* records, long long* keys, long long* gt_count, void* stream);
int yg_coco_accumulate(const int* records, const long long* sorted_keys, const long long* perm, long long n_records,
                       const long long* gt_count, int num_classes, const double* rec_thrs, double* precision, double* recall,
                       void* stream);

/* ROC and calibration error (torchmetrics MulticlassROC(thresholds=None) / MulticlassCalibrationError(norm="l1")) over the
 * rows of convert_background_errors(num_classes + 1): matched pairs (score = class columns and an appended 0, target
 * int(label[5])), missed labels (one-hot background, target int(label[5])), extra predictions (class columns and a 0,
 * target num_classes); without background the matched pairs alone over the num_classes columns.  nb = the columns.
 * yg_score_rows_batch: after yg_match_batch with the same outputs, desc, gather_off and lsap_status (n_matched / n_extra =
 * the row counts of out_preds / extra).  *softmax_flag (device int, overwritten) = 1 when a class value of the matched or
 * (with background) extra rows lies outside [0, 1] or is NaN; then every score row is softmaxed (fp64, rounded to fp32).
 * With scores (float R x nb) and targets (int32 R) non-null, image b's rows are written at [out_off + gather_off[2b] +
 * gather_off[2b+1], + N + M - K) (with background; else [out_off, + K)) in matched / missed / extra order.  nan_status[B]
 * (int32) is written 1 for an image with a NaN score.  Calibration: confidence = row maximum, prediction = its first
 * maximum, bin = bucketize(confidence, bin_bounds, right=True) - 1 with bin_bounds (HOST, bins + 1 floats, bins <= 255)
 * torch.linspace(0, 1, bins + 1); partials (device, B * (bins + 1) * 16 bytes) hold the per-image sums, and bin_count,
 * bin_correct (int64 [bins + 1]) and bin_conf (double [bins + 1], the confidence sums) are overwritten with their sums over
 * the images in order.  Images whose lsap_status is not YG_LSAP_OK contribute nothing.
 * yg_roc_keys: keys[k * rows + r] = k << 32 | a 32-bit key ascending in descending scores[r][k] (-0 keyed as +0).
 * yg_roc_curves: after sorting those keys (sorted_keys = keys[perm], int64), per class k the curve of _binary_clf_curve
 * with the point (0, 0, threshold 1) prepended: fpr / tpr (double) and thresholds (float) of class k at [k * (rows + 1),
 * + lengths[k]) (int64 [nb]); fpr = fps / fps_last (all 0 without negatives), tpr = tps / tps_last (all 0 without
 * positives), the thresholds are the scores.  auc (double [nb]) = the trapezoidal area, -1 for a class without positive or
 * negative rows. */
int yg_score_rows_batch(const float* out_preds, const float* out_labels, const float* missed, const float* extra,
                        long long n_matched, long long n_extra, int B, int num_classes, int include_background, const void* desc,
                        const long long* gather_off, const int* lsap_status, const float* bin_bounds, int bins, int* softmax_flag,
                        float* scores, int* targets, int* nan_status, void* partials, long long* bin_count,
                        long long* bin_correct, double* bin_conf, void* stream);
int yg_roc_keys(const float* scores, long long rows, int nb, long long* keys, void* stream);
int yg_roc_curves(const long long* sorted_keys, const long long* perm, const int* targets, long long rows, int nb, double* fpr,
                  double* tpr, float* thresholds, long long* lengths, double* auc, void* stream);

/* ---- input side (SURVEY.md 8f N3) --------------------------------------------------------
 * RandomHorizontal/VerticalFlipWithBBs (data/data_transforms.py:51-98) of a whole batch, out of place:
 * images (N,C,H,W) uint8 (YG_U8) or fp32, labels (N,6,Sy,Sx) = [mask,x1,y1,x2,y2,class] with x1' = 1 - x2, x2' = 1 - x1
 * (hflip) / y1' = 1 - y2, y2' = 1 - y1 (vflip) on every cell and the cells mirrored; both flips may be combined. */
int yg_flip_images(const void* in, void* out, int dtype, int N, int C, int H, int W, int hflip, int vflip, void* stream);
int yg_flip_labels(const float* in, float* out, int N, int Sy, int Sx, int hflip, int vflip, void* stream);
/* format_labels_tensor (data/yogo_dataset.py:24-46) for a batch of ragged label lists: labels (total,5) =
 * [class,x1,y1,x2,y2] rows of all images back to back, offsets[B+1] (int32) the row range of each image, max_labels the
 * largest per-image count; out (B,6,Sy,Sx) fp32 overwritten; owner (B*Sy*Sx int32) is scratch; *err (device int) is set
 * to 1 when a label centre falls outside the grid (the reference raises IndexError). */
int yg_format_labels_batch(const float* labels, const int* offsets, int B, int max_labels, int Sy, int Sx,
                           int* owner, float* out, int* err, void* stream);
/* Device-resident dataset (data/device_dataset.py), one batch of an epoch per call of each, all graph-capturable:
 * yg_dd_draw: state (3 x uint64) = [seed, call counter, batch cursor]; writes flags (int32) = [hflip, vflip, batch]
 * (hflip = u < p_hflip, vflip = u' < p_vflip with u, u' uniform in [0, 1) from Philox keyed by seed, stream_id and the
 * counter; batch = cursor mod nbatches) and advances counter and cursor.  The table holds nbatches * stride entries.  yg_dd_gather_images: out[n] = the flags' flips of store[table[batch * stride
 * + n]], n < N <= stride, (N, C, H, W) uint8 / fp32, C in {1, 3}.  yg_dd_build_labels: out (N, 6, Sy, Sx) fp32 = what
 * yg_flip_labels gives for the stacked dense labels of the same images; records: 8 int32 per labelled cell {cell, the six
 * channel values' bits, 0}, sorted by cell within a stored image, rec_off (int64) the record range of each stored image. */
int yg_dd_draw(void* state, int* flags, float p_hflip, float p_vflip, int stream_id, int nbatches, void* stream);
int yg_dd_gather_images(const void* store, void* out, int dtype, const int* table, const int* flags, int stride,
                        int N, int C, int H, int W, void* stream);
int yg_dd_build_labels(const int* table, const int* flags, int stride, const void* records, const long long* rec_off,
                       int N, int Sy, int Sx, float* out, void* stream);
/* Sharded store (a dataset larger than one GPU, spread over the ranks of one host; data/device_dataset.py):
 * yg_dd_gather_images_peers writes what yg_dd_gather_images writes, bit for bit, but stored slot s is image
 * s % shard_items of shards[s / shard_items]; shards is a DEVICE array of W base pointers (this rank's own shard and the
 * peers' shards opened with yg_dd_shard_open), each the start of an allocation.
 * Shard memory: yg_dd_shard_alloc is a plain cudaMalloc on the current device (its own allocation, so that its IPC
 * handle maps exactly the buffer); yg_dd_shard_export writes its YG_IPC_HANDLE_BYTES-byte handle to `handle` (host
 * memory); yg_dd_shard_open maps a handle exported by ANOTHER process of this host on the current device (peer access
 * enabled lazily); yg_dd_shard_close unmaps it; yg_dd_shard_free frees an own shard.  Teardown is a protocol across
 * processes: every importer synchronises and closes its handles, all processes meet in a barrier, and only then does each
 * owner free (freeing memory another process still has open is undefined in CUDA). */
#define YG_IPC_HANDLE_BYTES 64
int yg_dd_gather_images_peers(const void* const* shards, long long shard_items, void* out, int dtype, const int* table,
                              const int* flags, int stride, int N, int C, int H, int W, void* stream);
int yg_dd_shard_alloc(size_t bytes, void** ptr);
int yg_dd_shard_export(const void* ptr, void* handle);
int yg_dd_shard_open(const void* handle, void** ptr);
int yg_dd_shard_close(void* ptr);
int yg_dd_shard_free(void* ptr);

/* ---- PNG decoding: 8-bit grayscale, non-interlaced files (yogo_b200.data.decode_png_batch) ----------------------
 * One call decodes n files of the same H x W.  `files` (device, files_bytes) holds what the host uploaded; the host has
 * walked each file's chunks and lists every IDAT as a yg_png_chunk and each image as a yg_png_image:
 *   chunk.src     offset in `files` of the chunk's type field (the CRC covers type + payload);
 *   chunk.dst     offset of its payload in the workspace's stream region (the image's zlib stream, chunks back to back);
 *   chunk.length  payload bytes; chunk.crc the stored CRC-32;
 *   image.stream  offset of the image's zlib stream in the stream region (a multiple of 16), image.length its bytes;
 *   image.chunk_begin / chunk_end  its range of `chunks`.
 * yg_png_gray8_workspace(n, H, W, stream_bytes) is the workspace for a stream region of stream_bytes (the end of the
 * last stream, rounded up to 16); it must be 16-byte aligned (the inflate reads it in 16-byte loads), chunks and images
 * 8-byte aligned.  out is (n, 1, H, W) uint8.  status[n] (int32) is always written with a
 * yg_png_status; the output of an image whose status is not YG_PNG_OK is undefined.  Kernels: IDAT gather + CRC,
 * inflate (one warp per image), unfilter + Adler-32 (one warp per image), all on `stream`. */
enum {
  YG_PNG_OK = 0,
  YG_PNG_BAD_CRC = 1,            /* an IDAT CRC-32 does not match */
  YG_PNG_BAD_ZLIB_HEADER = 2,    /* CM != 8, CINFO > 7, FCHECK, or a preset dictionary */
  YG_PNG_BAD_BLOCK_TYPE = 3,     /* BTYPE 3 */
  YG_PNG_BAD_STORED_LENGTH = 4,  /* stored block LEN != ~NLEN */
  YG_PNG_BAD_CODE_LENGTHS = 5,   /* over-subscribed or incomplete code, bad repeat, too many symbols, no end-of-block */
  YG_PNG_BAD_SYMBOL = 6,         /* length symbol 286/287, distance symbol 30/31 or an unused distance code */
  YG_PNG_BAD_DISTANCE = 7,       /* distance beyond the bytes produced or the window */
  YG_PNG_OUTPUT_OVERFLOW = 8,    /* more than H * (1 + W) bytes */
  YG_PNG_TRUNCATED = 9,          /* the stream ends early, or its image data is short */
  YG_PNG_TRAILING_DATA = 10,     /* bytes after the Adler-32 */
  YG_PNG_BAD_ADLER = 11,         /* Adler-32 mismatch */
  YG_PNG_BAD_FILTER = 12,        /* scanline filter byte > 4 */
  YG_PNG_BAD_LAYOUT = 13         /* a chunk or stream outside the buffers it was described in */
};
typedef struct {
  long long src, dst;
  int length;
  unsigned int crc;
} yg_png_chunk;
typedef struct {
  long long stream, length;
  int chunk_begin, chunk_end;
} yg_png_image;
size_t yg_png_gray8_workspace(int n, int H, int W, long long stream_bytes);
int yg_png_decode_gray8(const void* files, long long files_bytes, const yg_png_chunk* chunks, const yg_png_image* images,
                        int n, int H, int W, unsigned char* out, int* status, void* workspace, size_t ws_bytes,
                        void* stream);

/* ---- optimizer (SURVEY.md 8f N1): fused AdamW over one flat fp32 buffer ---------------
 * replaces torch.optim.AdamW.step (train.py:213-217, 324). grads are pre-scaled by
 * grad_scale (1/world_size after an all-reduce SUM). */
int yg_adamw_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                  float lr, float beta1, float beta2, float eps, float weight_decay,
                  long long step, float grad_scale, void* stream);
/* graph-replayable variant: hyper_dev (device, 8 floats) = [lr, beta1, beta2, eps, weight_decay,
 * 1-beta1^t, sqrt(1-beta2^t), grad_scale] */
int yg_adamw_flat_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                      const float* hyper_dev, void* stream);

/* ---- Dropout2d keep-scales of every block of a step + BatchNorm step counters, one launch -------------------------
 * replaces nn.Dropout2d's mask draw (model_defns.py:44-57) and `num_batches_tracked += 1`.  out: `total` floats, the
 * blocks' (N, C) scale matrices back to back; table (device): nblocks x int4 (offset, count, p as float bits, 0);
 * state (device, 3 x uint64): [seed, call counter, 0] - the kernel advances the counter, so CUDA-graph replays draw
 * fresh masks; counters (device): ncounters pointers to int64 `num_batches_tracked` buffers, each incremented by one. */
int yg_dropout_scales(float* out, const void* table, int nblocks, int total, void* state, const void* counters,
                      int ncounters, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* YOGO_B200_H */
