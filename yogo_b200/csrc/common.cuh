// Shared helpers for the yogo_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/yogo_b200.h"

namespace yg {

void set_error(const char* fmt, ...);
extern unsigned long long g_launches;  // kernels launched by this library (yg_launch_count)

#define YG_CHECK_ARG(cond, ...)                 \
  do {                                          \
    if (!(cond)) {                              \
      yg::set_error(__VA_ARGS__);               \
      return YG_ERR_INVALID;                    \
    }                                           \
  } while (0)

#define YG_CUDA(expr)                                                             \
  do {                                                                            \
    cudaError_t _e = (expr);                                                      \
    if (_e != cudaSuccess) {                                                      \
      yg::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),       \
                    __FILE__, __LINE__);                                          \
      return YG_ERR_CUDA;                                                         \
    }                                                                             \
  } while (0)

#define YG_LAUNCH_CHECK(name)                                                     \
  do {                                                                            \
    cudaError_t _e = cudaGetLastError();                                          \
    if (_e != cudaSuccess) {                                                      \
      yg::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));     \
      return YG_ERR_CUDA;                                                         \
    }                                                                             \
    ++yg::g_launches;                                                             \
  } while (0)

typedef __nv_bfloat16 bf16;

template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<bf16>(bf16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f<uint8_t>(uint8_t v) { return (float)v; }

template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__device__ __forceinline__ float act_fwd(float v, int act) {
  if (act == YG_ACT_LRELU) return v > 0.f ? v : 0.01f * v;
  if (act == YG_ACT_SILU) return v * sigmoidf_(v);
  return v;
}
// derivative of the activation at pre-activation `pre`
__device__ __forceinline__ float act_grad(float pre, int act) {
  if (act == YG_ACT_LRELU) return pre > 0.f ? 1.f : 0.01f;
  if (act == YG_ACT_SILU) {
    float s = sigmoidf_(pre);
    return s * (1.f + pre * (1.f - s));
  }
  return 1.f;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// torch.clamp(grad, -c, c) of the reference's parameter hook (model.py:76-77) propagates NaN; fminf / fmaxf would
// return the finite operand and turn a NaN gradient into a silent -c
__device__ __forceinline__ float clampf(float v, float c) {
  return (c > 0.f && v == v) ? fminf(fmaxf(v, -c), c) : v;
}

// The shared backward epilogue (yg_bwd_epilogue semantics): g = d(loss)/d(layer output)
// -> gradient wrt the layer's conv output (or wrt BN output when the layer has BN).
// Returns the transformed gradient; xhat is set when the layer has BN.
struct BwdEpi {
  const void* saved;
  int act;
  const float* dropscale;
  const float* bn_scale;
  const float* bn_shift;
  const float* bn_mean;
  const float* bn_invstd;
  double* bn_sums;
  const void* actmask;
  int io_f32;   // internal: `saved` is read and the output written as fp32 (x3.cu)
};
inline BwdEpi make_bwd_epi(const yg_bwd_epilogue* be) {
  BwdEpi e{};
  if (be) {
    e.saved = be->saved; e.act = be->act; e.dropscale = be->dropscale;
    e.bn_scale = be->bn_scale; e.bn_shift = be->bn_shift; e.bn_mean = be->bn_mean;
    e.bn_invstd = be->bn_invstd; e.bn_sums = be->bn_sums; e.actmask = be->actmask;
  }
  return e;
}
template <typename T>
__device__ __forceinline__ float bwd_epi_apply(const BwdEpi& e, float g, long long idx, int n, int c, int C,
                                               float& xhat) {
  xhat = 0.f;
  if (e.dropscale) g *= e.dropscale[(long long)n * C + c];
  if (e.saved) {
    float sv = to_f<T>(((const T*)e.saved)[idx]);
    float pre = sv;
    if (e.bn_scale) {
      pre = sv * e.bn_scale[c] + e.bn_shift[c];
      xhat = (sv - e.bn_mean[c]) * e.bn_invstd[c];
    }
    g *= act_grad(pre, e.act);
  }
  return g;
}

struct FwdEpi {
  const float* scale;
  const float* shift;
  int act;
  const float* dropscale;
  double* stats;
  void* preact;
  void* actmask;
  int io_f32;   // internal: the output / pre-activation copy are written as fp32 (x3.cu)
};
inline FwdEpi make_fwd_epi(const yg_fwd_epilogue* ep) {
  FwdEpi e{};
  if (ep) {
    e.scale = ep->scale; e.shift = ep->shift; e.act = ep->act; e.dropscale = ep->dropscale;
    e.stats = ep->stats; e.preact = ep->preact; e.actmask = ep->actmask;
  }
  return e;
}

inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// exclusive scan of one flag per thread over the block; returns rank, total via reference
template <int THREADS>
__device__ __forceinline__ int block_rank(bool flag, int* warp_tot /*[32]*/, int& total) {
  const unsigned b = __ballot_sync(0xffffffffu, flag);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int r = __popc(b & ((1u << lane) - 1u));
  __syncthreads();  // protect warp_tot reuse
  if (lane == 0) warp_tot[wid] = __popc(b);
  __syncthreads();
  int base = 0, tot = 0;
  for (int w = 0; w < THREADS / 32; ++w) {
    const int t = warp_tot[w];
    if (w < wid) base += t;
    tot += t;
  }
  total = tot;
  return base + r;
}

// box_iou(a, b) of torchvision.ops (_box_inter_union) for two xyxy boxes with their areas (x2 - x1) * (y2 - y1)
// precomputed the same way.  Every operation is a single correctly rounded fp32 operation in torchvision's order (never
// contracted to FMA).  The one copy of the IoU expression: the matching cost tile below and the COCO matching
// (metrics.cu) both use it.
__device__ __forceinline__ float box_iou_f(float ax1, float ay1, float ax2, float ay2, float aarea, float bx1, float by1,
                                           float bx2, float by2, float barea) {
  const float ltx = ax1 > bx1 ? ax1 : bx1, lty = ay1 > by1 ? ay1 : by1;
  const float rbx = ax2 < bx2 ? ax2 : bx2, rby = ay2 < by2 ? ay2 : by2;
  float w = __fsub_rn(rbx, ltx), h = __fsub_rn(rby, lty);
  w = w < 0.f ? 0.f : w;   // clamp(min=0) keeps NaN
  h = h < 0.f ? 0.f : h;
  const float inter = __fmul_rn(w, h);
  const float uni = __fsub_rn(__fadd_rn(aarea, barea), inter);
  return __fdiv_rn(inter, uni);
}
__device__ __forceinline__ float box_area_f(float x1, float y1, float x2, float y2) {
  return __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
}

// One tile of the matching cost cost[i][j] = 1 - box_iou(a_i, b_j): column j (this thread's prediction box) of label
// rows i0 .. i0 + 15, bit-identical to the reference's matrix.  Shared by yg_box_iou_cost (nms.cu) and the batched
// matching (match.cu); call with a block-uniform i0.
__device__ __forceinline__ void box_iou_cost_tile(const float* __restrict__ a, int a_stride, int na, const float* __restrict__ b,
                                                  int b_stride, int nb, float* __restrict__ cost, int j, int i0) {
  __shared__ float sb[16][5];
  // this thread's prediction box
  float bx1 = 0.f, by1 = 0.f, bx2 = 0.f, by2 = 0.f, barea = 0.f;
  if (j < nb) {
    const float* r = b + (long long)j * b_stride;
    bx1 = r[0]; by1 = r[1]; bx2 = r[2]; by2 = r[3];
    barea = box_area_f(bx1, by1, bx2, by2);
  }
  // 16 label boxes of this block row through shared memory
  if (threadIdx.x < 16 && i0 + threadIdx.x < na) {
    const float* r = a + (long long)(i0 + threadIdx.x) * a_stride;
    sb[threadIdx.x][0] = r[0]; sb[threadIdx.x][1] = r[1]; sb[threadIdx.x][2] = r[2]; sb[threadIdx.x][3] = r[3];
    sb[threadIdx.x][4] = box_area_f(r[0], r[1], r[2], r[3]);
  }
  __syncthreads();
  if (j >= nb) return;
  for (int k = 0; k < 16 && i0 + k < na; ++k) {
    const float iou = box_iou_f(sb[k][0], sb[k][1], sb[k][2], sb[k][3], sb[k][4], bx1, by1, bx2, by2, barea);
    cost[(long long)(i0 + k) * nb + j] = __fsub_rn(1.f, iou);
  }
}

// one cost matrix of the batched matching: host-built, uploaded as int64 [4] = cost_off, ws_off (8-byte words), out_off,
// rows | cols << 32 (rows = labels, cols = kept predictions of one image).  Read by match.cu and metrics.cu.
struct LsapDesc {
  long long cost_off;
  long long ws_off;
  long long out_off;
  int rows, cols;
};

}  // namespace yg
