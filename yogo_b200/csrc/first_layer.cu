// First convolution block as a direct stencil on the NCHW image (Cin = 1 or 3, K = 9*Cin):
// HBM-bound, not GEMM-shaped, so it is a SIMT kernel (SURVEY.md Appendix A, layer 1).
// Train-mode BatchNorm is handled by recomputation: pass 1 accumulates the batch statistics
// without writing anything, pass 2 recomputes the 9-tap stencil and writes the normalised,
// activated output once.  Replaces nn.Conv2d(1,16,3,stride=2,padding=1,bias=False) +
// BatchNorm2d + LeakyReLU/SiLU at /root/reference/yogo/model_defns.py:33-37 (and x.float(),
// model.py:272-273).
#include "common.cuh"

namespace yg {

constexpr int FL_CO = 16, FL_THREADS = 128;

template <typename TX, int CO>
__device__ __forceinline__ void first_conv_pixel(const TX* __restrict__ x, const float* ws, int n, int ho, int wo,
                                                 int H, int W, int Cin, int stride, float (&acc)[CO]) {
#pragma unroll
  for (int c = 0; c < CO; ++c) acc[c] = 0.f;
  for (int ci = 0; ci < Cin; ++ci) {
    const TX* xp = x + ((long long)n * Cin + ci) * H * W;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int ih = ho * stride - 1 + r;
      if (ih < 0 || ih >= H) continue;
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const int iw = wo * stride - 1 + s;
        if (iw < 0 || iw >= W) continue;
        const float xv = to_f<TX>(xp[(long long)ih * W + iw]);
        const float* wr = ws + (ci * 9 + r * 3 + s) * CO;
#pragma unroll
        for (int c = 0; c < CO; ++c) acc[c] += xv * wr[c];
      }
    }
  }
}

template <int CO>
__device__ __forceinline__ void load_first_weights(float* ws, const float* __restrict__ w, int Cin, int Cout, int co0) {
  for (int i = threadIdx.x; i < Cin * 9 * CO; i += blockDim.x) {
    int c = i % CO, t = i / CO;  // t = ci*9 + tap
    int co = co0 + c;
    ws[i] = co < Cout ? w[(long long)co * Cin * 9 + t] : 0.f;
  }
}

template <typename TX, typename T>
__global__ void __launch_bounds__(FL_THREADS) conv_first_fwd_kernel(
    const TX* __restrict__ x, const float* __restrict__ w, T* __restrict__ y,
    int N, int H, int W, int Cin, int Ho, int Wo, int Cout, int stride, FwdEpi ep) {
  __shared__ float ws[3 * 9 * FL_CO];
  __shared__ float ssum[FL_CO], ssq[FL_CO];
  const int co0 = blockIdx.y * FL_CO;
  load_first_weights<FL_CO>(ws, w, Cin, Cout, co0);
  if (threadIdx.x < FL_CO) { ssum[threadIdx.x] = 0.f; ssq[threadIdx.x] = 0.f; }
  __syncthreads();
  float sc[FL_CO], sh[FL_CO];
#pragma unroll
  for (int c = 0; c < FL_CO; ++c) {
    const int co = co0 + c;
    sc[c] = (ep.scale && co < Cout) ? ep.scale[co] : 1.f;
    sh[c] = (ep.shift && co < Cout) ? ep.shift[co] : 0.f;
  }
  float s1[FL_CO], s2[FL_CO];
#pragma unroll
  for (int c = 0; c < FL_CO; ++c) { s1[c] = 0.f; s2[c] = 0.f; }
  const long long total = (long long)N * Ho * Wo;
  // grid-stride loop: statistics accumulate in registers, one reduction per thread at the end
  for (long long q = (long long)blockIdx.x * FL_THREADS + threadIdx.x; q < total;
       q += (long long)gridDim.x * FL_THREADS) {
    const int n = (int)(q / ((long long)Ho * Wo));
    const int p = (int)(q % ((long long)Ho * Wo));
    float acc[FL_CO];
    first_conv_pixel<TX, FL_CO>(x, ws, n, p / Wo, p % Wo, H, W, Cin, stride, acc);
    float v[FL_CO];
#pragma unroll
    for (int c = 0; c < FL_CO; ++c) {
      v[c] = acc[c] * sc[c] + sh[c];
      s1[c] += v[c];
      s2[c] += v[c] * v[c];
    }
    if (y) {
      const long long o = q * Cout + co0;
      if (sizeof(T) == 2 && co0 + FL_CO <= Cout && (Cout & 7) == 0 && !ep.preact) {
        __align__(16) T ob[FL_CO];
#pragma unroll
        for (int c = 0; c < FL_CO; ++c) {
          const float ds = ep.dropscale ? ep.dropscale[(long long)n * Cout + co0 + c] : 1.f;
          ob[c] = from_f<T>(act_fwd(v[c], ep.act) * ds);
        }
        uint4* dst = reinterpret_cast<uint4*>(y + o);
        dst[0] = reinterpret_cast<uint4*>(ob)[0];
        dst[1] = reinterpret_cast<uint4*>(ob)[1];
      } else {
#pragma unroll
        for (int c = 0; c < FL_CO; ++c) {
          const int co = co0 + c;
          if (co < Cout) {
            const float ds = ep.dropscale ? ep.dropscale[(long long)n * Cout + co] : 1.f;
            if (ep.preact) ((T*)ep.preact)[o + c] = from_f<T>(v[c]);
            y[o + c] = from_f<T>(act_fwd(v[c], ep.act) * ds);
          }
        }
      }
    }
  }
  if (ep.stats) {
#pragma unroll
    for (int c = 0; c < FL_CO; ++c) {
      const float a = warp_sum(s1[c]), b = warp_sum(s2[c]);
      if ((threadIdx.x & 31) == 0) { atomicAdd(&ssum[c], a); atomicAdd(&ssq[c], b); }
    }
    __syncthreads();
    if (threadIdx.x < FL_CO && co0 + threadIdx.x < Cout) {
      atomicAdd(&ep.stats[co0 + threadIdx.x], (double)ssum[threadIdx.x]);
      atomicAdd(&ep.stats[Cout + co0 + threadIdx.x], (double)ssq[threadIdx.x]);
    }
  }
}

constexpr int FLB_CO = 8;  // couts per backward block (keeps 9x8 accumulators + state under 128 registers)

// Backward.  mode 0: accumulate BN sums (sum g, sum g*xhat).  mode 1: weight gradient partials.
// One block = (co chunk, ci) pair looping over pixels with a grid stride.
template <typename TX, typename T, int MODE>
__global__ void __launch_bounds__(FL_THREADS, 4) conv_first_bwd_kernel(
    const TX* __restrict__ x, const float* __restrict__ w, const T* __restrict__ da,
    int N, int H, int W, int Cin, int Ho, int Wo, int Cout, int stride, BwdEpi be,
    const float* __restrict__ fwd_shift, const float* __restrict__ dy_mean, const float* __restrict__ dyx_mean,
    float* __restrict__ partial, int nchunks) {
  __shared__ float ws[3 * 9 * FLB_CO];
  __shared__ float red[9 * FLB_CO + FLB_CO];
  const int chunk = blockIdx.y % nchunks, ci_sel = blockIdx.y / nchunks;
  const int co0 = chunk * FLB_CO;
  load_first_weights<FLB_CO>(ws, w, Cin, Cout, co0);
  for (int i = threadIdx.x; i < 9 * FLB_CO + FLB_CO; i += blockDim.x) red[i] = 0.f;
  __syncthreads();

  float wacc[MODE == 1 ? 9 : 1][FLB_CO];
  float s1[FLB_CO], s2[FLB_CO];
#pragma unroll
  for (int c = 0; c < FLB_CO; ++c) {
    s1[c] = 0.f; s2[c] = 0.f;
#pragma unroll
    for (int t = 0; t < (MODE == 1 ? 9 : 1); ++t) wacc[t][c] = 0.f;
  }
  float scl[FLB_CO], sft[FLB_CO], mean[FLB_CO], istd[FLB_CO], m1[FLB_CO], m2[FLB_CO], fsh[FLB_CO];
#pragma unroll
  for (int c = 0; c < FLB_CO; ++c) {
    const int co = co0 + c;
    const bool ok = co < Cout;
    scl[c] = (be.bn_scale && ok) ? be.bn_scale[co] : 1.f;
    sft[c] = (be.bn_shift && ok) ? be.bn_shift[co] : 0.f;
    mean[c] = (be.bn_mean && ok) ? be.bn_mean[co] : 0.f;
    istd[c] = (be.bn_invstd && ok) ? be.bn_invstd[co] : 1.f;
    m1[c] = (dy_mean && ok) ? dy_mean[co] : 0.f;
    m2[c] = (dyx_mean && ok) ? dyx_mean[co] : 0.f;
    fsh[c] = (fwd_shift && ok) ? fwd_shift[co] : 0.f;
  }
  const long long total = (long long)N * Ho * Wo;
  for (long long q = (long long)blockIdx.x * FL_THREADS + threadIdx.x; q < total;
       q += (long long)gridDim.x * FL_THREADS) {
    const int n = (int)(q / ((long long)Ho * Wo));
    const int p = (int)(q % ((long long)Ho * Wo));
    const int ho = p / Wo, wo = p % Wo;
    float acc[FLB_CO];
    first_conv_pixel<TX, FLB_CO>(x, ws, n, ho, wo, H, W, Cin, stride, acc);
    float dzv[FLB_CO];
    const long long o = q * Cout + co0;
#pragma unroll
    for (int c = 0; c < FLB_CO; ++c) {
      const int co = co0 + c;
      float g = 0.f, xhat = 0.f;
      if (co < Cout) {
        g = to_f<T>(da[o + c]);
        if (be.dropscale) g *= be.dropscale[(long long)n * Cout + co];
        const float yv = acc[c] + fsh[c];           // conv output (+bias when no BN)
        float pre = yv;
        if (be.bn_scale) { pre = yv * scl[c] + sft[c]; xhat = (yv - mean[c]) * istd[c]; }
        g *= act_grad(pre, be.act);
      }
      if (MODE == 0) { s1[c] += g; s2[c] += g * xhat; }
      else {
        // BN backward: dz = gamma*invstd*(g - mean(g) - xhat*mean(g*xhat)); scl = gamma*invstd
        dzv[c] = (be.bn_scale && dy_mean) ? scl[c] * (g - m1[c] - xhat * m2[c]) : g;
        s1[c] += dzv[c];
      }
    }
    if (MODE == 1) {
      const TX* xp = x + ((long long)n * Cin + ci_sel) * H * W;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const int ih = ho * stride - 1 + r;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          const int iw = wo * stride - 1 + s;
          float xv = 0.f;
          if (ih >= 0 && ih < H && iw >= 0 && iw < W) xv = to_f<TX>(xp[(long long)ih * W + iw]);
#pragma unroll
          for (int c = 0; c < FLB_CO; ++c) wacc[r * 3 + s][c] += dzv[c] * xv;
        }
      }
    }
  }
  // block reduction -> partials
#pragma unroll
  for (int c = 0; c < FLB_CO; ++c) {
    float a = warp_sum(s1[c]);
    float b = MODE == 0 ? warp_sum(s2[c]) : 0.f;
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(&red[9 * FLB_CO + c], a);
      if (MODE == 0) atomicAdd(&red[c], b);
    }
    if (MODE == 1) {
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        float v = warp_sum(wacc[t][c]);
        if ((threadIdx.x & 31) == 0) atomicAdd(&red[t * FLB_CO + c], v);
      }
    }
  }
  __syncthreads();
  if (MODE == 0) {
    if (threadIdx.x < FLB_CO && co0 + threadIdx.x < Cout && ci_sel == 0) {
      atomicAdd(&be.bn_sums[co0 + threadIdx.x], (double)red[9 * FLB_CO + threadIdx.x]);
      atomicAdd(&be.bn_sums[Cout + co0 + threadIdx.x], (double)red[threadIdx.x]);
    }
  } else {
    // partial layout per slice (= blockIdx.x): [Cout][Cin][9] then [Cout]
    float* base = partial + (long long)blockIdx.x * ((long long)Cout * Cin * 9 + Cout);
    for (int i = threadIdx.x; i < 9 * FLB_CO; i += blockDim.x) {
      const int c = i % FLB_CO, t = i / FLB_CO;
      if (co0 + c < Cout) base[((long long)(co0 + c) * Cin + ci_sel) * 9 + t] = red[i];
    }
    if (threadIdx.x < FLB_CO && co0 + threadIdx.x < Cout && ci_sel == 0)
      base[(long long)Cout * Cin * 9 + co0 + threadIdx.x] = red[9 * FLB_CO + threadIdx.x];
  }
}

__global__ void wgrad_reduce_kernel2(const float* __restrict__ partial, float* __restrict__ dw,
                                     float* __restrict__ dbias, long long nw, int Cout, int slices, float clip) {
  // one warp per element (the first layer has 160 of them and ~600 slices): lanes stride over the slices
  const long long stride_slice = nw + Cout;
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= nw + Cout) return;
  float s = 0.f;
  for (int k = lane; k < slices; k += 32) s += partial[k * stride_slice + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane != 0) return;
  s = clampf(s, clip);
  if (i < nw) dw[i] = s;
  else if (dbias) dbias[i - nw] = s;
}


// ------------------------------------------------------------------------------------------------
// Fast path for the configuration every YOGO model uses: one input channel, 16 output channels, bf16
// activations.  Same arithmetic as the generic kernels above, restructured so that the instruction stream
// is dominated by the 9x16 FMAs instead of index arithmetic (the generic kernels spend ~950 instructions
// per pixel and 8-channel chunk, mostly 64-bit div/mod, bounds checks and reloading the 9 taps):
//   * work = (image, contiguous pixel chunk) tasks, (ho, wo) advanced incrementally - no per-pixel division
//   * one thread owns all 16 channels of a pixel; the 9 taps are loaded once and shared by the stencil
//     recomputation and the weight-gradient accumulation
//   * weights / per-channel constants are read as 128-bit shared-memory broadcasts
// ------------------------------------------------------------------------------------------------
constexpr int FF_CO = 16;

struct PixCursor {
  int p, ho, wo;
  __device__ __forceinline__ void init(int p0, int Wo) { p = p0; ho = p0 / Wo; wo = p0 - ho * Wo; }
  __device__ __forceinline__ void advance(int step, int Wo) {
    p += step; wo += step;
    while (wo >= Wo) { wo -= Wo; ++ho; }
  }
};

template <typename TX>
__device__ __forceinline__ void load_taps1(const TX* __restrict__ xim, int H, int W, int stride, int ho, int wo,
                                           float (&v)[9]) {
  const int ih0 = ho * stride - 1, iw0 = wo * stride - 1;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const int ih = ih0 + r;
    const bool rok = (unsigned)ih < (unsigned)H;
    const TX* row = xim + ih * W;
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      const int iw = iw0 + s;
      v[r * 3 + s] = (rok && (unsigned)iw < (unsigned)W) ? to_f<TX>(__ldg(row + iw)) : 0.f;
    }
  }
}

// acc[c] = sum_t v[t] * ws[t][c], ws in shared memory as [9][16]
__device__ __forceinline__ void stencil16(const float* ws, const float (&v)[9], float (&acc)[FF_CO]) {
#pragma unroll
  for (int c = 0; c < FF_CO; ++c) acc[c] = 0.f;
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const float4* w4 = reinterpret_cast<const float4*>(ws + t * FF_CO);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 q = w4[i];
      acc[4 * i] += v[t] * q.x; acc[4 * i + 1] += v[t] * q.y; acc[4 * i + 2] += v[t] * q.z; acc[4 * i + 3] += v[t] * q.w;
    }
  }
}

__device__ __forceinline__ void lds16(const float* s, float (&o)[FF_CO]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 q = reinterpret_cast<const float4*>(s)[i];
    o[4 * i] = q.x; o[4 * i + 1] = q.y; o[4 * i + 2] = q.z; o[4 * i + 3] = q.w;
  }
}

template <typename TX, bool STATS>
__global__ void __launch_bounds__(FL_THREADS, 3) first_fwd16_kernel(
    const TX* __restrict__ x, const float* __restrict__ w, bf16* __restrict__ y, int H, int W, int Ho, int Wo,
    int stride, FwdEpi ep, int chunk, int cpi, int ntasks) {
  __shared__ __align__(16) float ws[9 * FF_CO];
  __shared__ __align__(16) float s_ds[FF_CO];
  __shared__ float ssum[2 * FF_CO];
  for (int i = threadIdx.x; i < 9 * FF_CO; i += FL_THREADS) ws[i] = w[(i % FF_CO) * 9 + i / FF_CO];
  if (threadIdx.x < 2 * FF_CO) ssum[threadIdx.x] = 0.f;
  if (threadIdx.x < FF_CO) s_ds[threadIdx.x] = 1.f;
  float sc[FF_CO], sh[FF_CO];
#pragma unroll
  for (int c = 0; c < FF_CO; ++c) { sc[c] = ep.scale ? ep.scale[c] : 1.f; sh[c] = ep.shift ? ep.shift[c] : 0.f; }
  float s1[STATS ? FF_CO : 1], s2[STATS ? FF_CO : 1];
#pragma unroll
  for (int c = 0; c < (STATS ? FF_CO : 1); ++c) { s1[c] = 0.f; s2[c] = 0.f; }
  __syncthreads();
  const int npix = Ho * Wo, act = ep.act;
  for (int task = blockIdx.x; task < ntasks; task += gridDim.x) {
    const int n = task / cpi, p0 = (task - n * cpi) * chunk;
    const int p1 = min(p0 + chunk, npix);
    if (ep.dropscale) {
      __syncthreads();
      if (threadIdx.x < FF_CO) s_ds[threadIdx.x] = ep.dropscale[(long long)n * FF_CO + threadIdx.x];
      __syncthreads();
    }
    const TX* xim = x + (long long)n * H * W;
    bf16* yim = y ? y + (long long)n * npix * FF_CO : nullptr;
    PixCursor cur;
    cur.init(p0 + (int)threadIdx.x, Wo);
    for (; cur.p < p1; cur.advance(FL_THREADS, Wo)) {
      float v[9], acc[FF_CO];
      load_taps1<TX>(xim, H, W, stride, cur.ho, cur.wo, v);
      stencil16(ws, v, acc);
#pragma unroll
      for (int c = 0; c < FF_CO; ++c) {
        acc[c] = acc[c] * sc[c] + sh[c];
        if (STATS) { s1[c] += acc[c]; s2[c] += acc[c] * acc[c]; }
      }
      if (yim) {
        if (act == YG_ACT_LRELU) {
#pragma unroll
          for (int c = 0; c < FF_CO; ++c) acc[c] = fmaxf(acc[c], 0.01f * acc[c]);
        } else if (act == YG_ACT_SILU) {
#pragma unroll
          for (int c = 0; c < FF_CO; ++c) acc[c] = acc[c] * sigmoidf_(acc[c]);
        }
        if (ep.dropscale) {
          float ds[FF_CO];
          lds16(s_ds, ds);
#pragma unroll
          for (int c = 0; c < FF_CO; ++c) acc[c] *= ds[c];
        }
        __align__(16) __nv_bfloat162 ob[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) ob[i] = __floats2bfloat162_rn(acc[2 * i], acc[2 * i + 1]);
        uint4* dst = reinterpret_cast<uint4*>(yim + (long long)cur.p * FF_CO);
        dst[0] = reinterpret_cast<uint4*>(ob)[0];
        dst[1] = reinterpret_cast<uint4*>(ob)[1];
      }
    }
  }
  if (STATS) {
#pragma unroll
    for (int c = 0; c < (STATS ? FF_CO : 1); ++c) {
      const float a = warp_sum(s1[c]), b = warp_sum(s2[c]);
      if ((threadIdx.x & 31) == 0) { atomicAdd(&ssum[c], a); atomicAdd(&ssum[FF_CO + c], b); }
    }
    __syncthreads();
    if (threadIdx.x < FF_CO) {
      atomicAdd(&ep.stats[threadIdx.x], (double)ssum[threadIdx.x]);
      atomicAdd(&ep.stats[FF_CO + threadIdx.x], (double)ssum[FF_CO + threadIdx.x]);
    }
  }
}

// weight-gradient pass (mode 1 of conv_first_bwd_kernel): CO of the 16 channels per thread, blockIdx.y selects the
// channel group (CO = 8: 72 + 72 FMAs per pixel at ~128 registers, four blocks per SM)
template <int CO>
__device__ __forceinline__ void ldsN(const float* s, float (&o)[CO]) {
#pragma unroll
  for (int i = 0; i < CO / 4; ++i) {
    const float4 q = reinterpret_cast<const float4*>(s)[i];
    o[4 * i] = q.x; o[4 * i + 1] = q.y; o[4 * i + 2] = q.z; o[4 * i + 3] = q.w;
  }
}

template <typename TX, int CO>
__global__ void __launch_bounds__(FL_THREADS, CO == 8 ? 3 : 2) first_bwd16_kernel(
    const TX* __restrict__ x, const float* __restrict__ w, const bf16* __restrict__ da, int H, int W, int Ho, int Wo,
    int stride, BwdEpi be, const float* __restrict__ fwd_shift, const float* __restrict__ dy_mean,
    const float* __restrict__ dyx_mean, float* __restrict__ partial, int chunk, int cpi, int ntasks) {
  __shared__ __align__(16) float ws[9 * CO];
  __shared__ __align__(16) float cst[8 * CO];   // scl, sft, mean, istd, m1, m2, fsh, ds
  __shared__ float red[10 * CO];
  const int co0 = blockIdx.y * CO;
  for (int i = threadIdx.x; i < 9 * CO; i += FL_THREADS) ws[i] = w[(co0 + i % CO) * 9 + i / CO];
  for (int i = threadIdx.x; i < 10 * CO; i += FL_THREADS) red[i] = 0.f;
  if (threadIdx.x < CO) {
    const int c = threadIdx.x, co = co0 + c;
    cst[c] = be.bn_scale ? be.bn_scale[co] : 1.f;
    cst[CO + c] = be.bn_shift ? be.bn_shift[co] : 0.f;
    cst[2 * CO + c] = be.bn_mean ? be.bn_mean[co] : 0.f;
    cst[3 * CO + c] = be.bn_invstd ? be.bn_invstd[co] : 1.f;
    cst[4 * CO + c] = dy_mean ? dy_mean[co] : 0.f;
    cst[5 * CO + c] = dyx_mean ? dyx_mean[co] : 0.f;
    cst[6 * CO + c] = fwd_shift ? fwd_shift[co] : 0.f;
    cst[7 * CO + c] = 1.f;
  }
  float wacc[9][CO], s1[CO];
#pragma unroll
  for (int c = 0; c < CO; ++c) {
    s1[c] = 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) wacc[t][c] = 0.f;
  }
  __syncthreads();
  const int npix = Ho * Wo, act = be.act;
  const bool bn = be.bn_scale != nullptr, bn_full = bn && dy_mean != nullptr;
  for (int task = blockIdx.x; task < ntasks; task += gridDim.x) {
    const int n = task / cpi, p0 = (task - n * cpi) * chunk;
    const int p1 = min(p0 + chunk, npix);
    if (be.dropscale) {
      __syncthreads();
      if (threadIdx.x < CO) cst[7 * CO + threadIdx.x] = be.dropscale[(long long)n * FF_CO + co0 + threadIdx.x];
      __syncthreads();
    }
    const TX* xim = x + (long long)n * H * W;
    const bf16* dim = da + (long long)n * npix * FF_CO + co0;
    PixCursor cur;
    cur.init(p0 + (int)threadIdx.x, Wo);
    for (; cur.p < p1; cur.advance(FL_THREADS, Wo)) {
      float v[9], acc[CO], g[CO];
      const uint4* gp = reinterpret_cast<const uint4*>(dim + (long long)cur.p * FF_CO);
      uint4 gv[CO / 8];
#pragma unroll
      for (int i = 0; i < CO / 8; ++i) gv[i] = __ldg(gp + i);
      load_taps1<TX>(xim, H, W, stride, cur.ho, cur.wo, v);
#pragma unroll
      for (int c = 0; c < CO; ++c) acc[c] = 0.f;
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        float wr[CO];
        ldsN<CO>(ws + t * CO, wr);
#pragma unroll
        for (int c = 0; c < CO; ++c) acc[c] += v[t] * wr[c];
      }
#pragma unroll
      for (int i = 0; i < CO / 8; ++i) {
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&gv[i]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 a = __bfloat1622float2(h[j]);
          g[8 * i + 2 * j] = a.x; g[8 * i + 2 * j + 1] = a.y;
        }
      }
      float k0[CO], k1[CO];
      ldsN<CO>(cst + 6 * CO, k0);   // forward shift (conv bias when there is no BN)
#pragma unroll
      for (int c = 0; c < CO; ++c) acc[c] += k0[c];          // yv
      if (be.dropscale) {
        ldsN<CO>(cst + 7 * CO, k0);
#pragma unroll
        for (int c = 0; c < CO; ++c) g[c] *= k0[c];
      }
      if (bn) {
        ldsN<CO>(cst, k0); ldsN<CO>(cst + CO, k1);
#pragma unroll
        for (int c = 0; c < CO; ++c) g[c] *= act_grad(acc[c] * k0[c] + k1[c], act);
      } else {
#pragma unroll
        for (int c = 0; c < CO; ++c) g[c] *= act_grad(acc[c], act);
      }
      if (bn_full) {
        // BN backward: dz = gamma*invstd*(g - mean(g) - xhat*mean(g*xhat))
        ldsN<CO>(cst + 2 * CO, k0); ldsN<CO>(cst + 3 * CO, k1);
#pragma unroll
        for (int c = 0; c < CO; ++c) acc[c] = (acc[c] - k0[c]) * k1[c];   // xhat
        ldsN<CO>(cst + 4 * CO, k0); ldsN<CO>(cst + 5 * CO, k1);
#pragma unroll
        for (int c = 0; c < CO; ++c) g[c] = g[c] - k0[c] - acc[c] * k1[c];
        ldsN<CO>(cst, k0);
#pragma unroll
        for (int c = 0; c < CO; ++c) g[c] *= k0[c];
      }
#pragma unroll
      for (int c = 0; c < CO; ++c) {
        s1[c] += g[c];
#pragma unroll
        for (int t = 0; t < 9; ++t) wacc[t][c] += g[c] * v[t];
      }
    }
  }
#pragma unroll
  for (int c = 0; c < CO; ++c) {
    const float a = warp_sum(s1[c]);
    if ((threadIdx.x & 31) == 0) atomicAdd(&red[9 * CO + c], a);
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const float b = warp_sum(wacc[t][c]);
      if ((threadIdx.x & 31) == 0) atomicAdd(&red[c * 9 + t], b);
    }
  }
  __syncthreads();
  // partial layout per slice (= blockIdx.x): [16][1][9] then [16] (what wgrad_reduce_kernel2 sums)
  float* base = partial + (long long)blockIdx.x * (10 * FF_CO);
  for (int i = threadIdx.x; i < 9 * CO; i += FL_THREADS) base[co0 * 9 + i] = red[i];
  if (threadIdx.x < CO) base[9 * FF_CO + co0 + threadIdx.x] = red[9 * CO + threadIdx.x];
}


// ------------------------------------------------------------------------------------------------
// Weight-gradient pass of the first layer on the (legacy, warp-level) tensor cores - uint8 image, 1 -> 16 channels, the
// "raw P / Sg" mode of the Gram-matrix backward (dy_mean == NULL).  Per warp and 32 pixels (thread = pixel for the loads):
//   X[px][16]  = the 9 taps of the pixel as bf16 (exact for uint8), a column of ones, zero padding        -> shared memory
//   DA[px][16] = d(activation), bf16                                                                        -> shared memory
//   acc^T[ch][px] = (W_hi + W_lo) . X^T        two mma.m16n8k16 per 8 pixels: the stencil recomputed with split-bf16
//                                              weights (|error| ~ 2^-17 relative, the sign of the pre-activation is safe)
//   g[ch][px]  = DA * act'(BN(acc)) * dropscale                      in the accumulator fragment layout ...
//   P[ch][tap] += g . X                        ... which is exactly the A fragment layout of the second mma (k = pixels);
//                                              the ones column makes P[:, 9] = sum(g)
// ~6 warp instructions per pixel instead of ~17 of the SIMT kernel; 8 accumulator registers instead of 9 x 16.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void hmma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}

constexpr int FM_WARPS = 4;

// Row segments: a warp works on 32 consecutive output pixels of ONE output row (lane = pixel), so the input row
// pointers and the row-validity tests are warp-uniform, and with stride 2 and an even image width each lane fetches its
// centre / right tap of a row as one aligned 16-bit load (a fully coalesced 64-byte warp request) and takes the left tap
// from its neighbour's register: 3 loads + 3 shuffles per pixel instead of 9 predicated byte loads with per-lane
// address arithmetic (ncu: the byte-load version issued 175-270 instructions per 32 pixels and was issue-bound).
struct SegCursor {
  int ho, sg;   // output row, segment inside the row
  __device__ __forceinline__ void init(int s, int spr) { ho = s / spr; sg = s - ho * spr; }
  __device__ __forceinline__ void advance(int step, int spr) {
    sg += step;
    while (sg >= spr) { sg -= spr; ++ho; }
  }
};

// Raw taps of one pixel as they come from memory: requested one iteration ahead (fetch), turned into the nine floats
// only when the pixel is processed (unpack) - the shuffles of the fast path would otherwise wait for the loads at once.
template <bool FAST> struct TapRaw;
template <> struct TapRaw<true> { unsigned cr[3], lf[3]; };   // per input row: centre | right << 8; left tap of lane 0
template <> struct TapRaw<false> { float v[9]; };

__device__ __forceinline__ void fetch_taps(TapRaw<true>& t, const uint8_t* __restrict__ xim, int H, int W, int stride, int ho,
                                           int wo, bool pv, int lane) {
  (void)stride;
  // one address per pixel (row 2 ho - 1, column 2 wo), the other two rows are W and 2 W bytes further; the row tests are
  // warp-uniform, the left tap of lane 0 sits one byte before its centre tap
  const int ih0 = 2 * ho - 1;
  const uint8_t* p = xim + ((long long)ih0 * W + 2 * wo);
  const bool lf = lane == 0 && wo > 0;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const bool ok = pv && (unsigned)(ih0 + r) < (unsigned)H;
    t.cr[r] = 0u;                                          // (W even: column 2 wo + 1 exists whenever wo < Wo)
    t.lf[r] = 0u;
    if (ok) t.cr[r] = __ldg(reinterpret_cast<const unsigned short*>(p));
    if (ok && lf) t.lf[r] = __ldg(p - 1);
    p += W;
  }
}
__device__ __forceinline__ void fetch_taps(TapRaw<false>& t, const uint8_t* __restrict__ xim, int H, int W, int stride, int ho,
                                           int wo, bool pv, int lane) {
  (void)lane;
  if (pv) load_taps1<uint8_t>(xim, H, W, stride, ho, wo, t.v);
  else {
#pragma unroll
    for (int i = 0; i < 9; ++i) t.v[i] = 0.f;
  }
}
__device__ __forceinline__ void unpack_taps(const TapRaw<true>& t, bool pv, int lane, float (&v)[9]) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    unsigned left = __shfl_up_sync(0xffffffffu, t.cr[r] >> 8, 1);
    if (lane == 0) left = t.lf[r];
    v[3 * r] = pv ? (float)left : 0.f;   // (an invalid lane next to a valid one would inherit its neighbour's byte)
    v[3 * r + 1] = (float)(t.cr[r] & 0xFFu);
    v[3 * r + 2] = (float)(t.cr[r] >> 8);
  }
}
__device__ __forceinline__ void unpack_taps(const TapRaw<false>& t, bool pv, int lane, float (&v)[9]) {
  (void)pv; (void)lane;
#pragma unroll
  for (int i = 0; i < 9; ++i) v[i] = t.v[i];
}

// NM = number of 16-channel M tiles (Cout = 16 NM): the X tile and its two B fragments are shared by all of them
template <int NM, bool FAST>
__global__ void __launch_bounds__(FM_WARPS * 32, NM == 1 ? 5 : (NM == 2 ? 4 : 3)) first_bwd_mma_kernel(
    const uint8_t* __restrict__ x, const float* __restrict__ w, const bf16* __restrict__ da, int H, int W, int Ho, int Wo,
    int stride, BwdEpi be, const float* __restrict__ fwd_shift, float* __restrict__ partial, int chunk, int cpi, int ntasks) {
  constexpr int CO = 16 * NM;
  __shared__ __align__(128) unsigned char tiles[FM_WARPS][1 + NM][32 * 32];   // per warp: X tile, NM DA tiles (32 B per pixel row)
  __shared__ float red[10 * CO];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, j = lane & 3;
  for (int i = threadIdx.x; i < 10 * CO; i += FM_WARPS * 32) red[i] = 0.f;
  // A fragments of the weights, split into two bf16 terms: A[m = ch][k = tap] (taps >= 9 are zero)
  uint32_t whi[NM][4], wlo[NM][4];
#pragma unroll
  for (int m = 0; m < NM; ++m) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int ch = 16 * m + g + (q & 1) * 8, t0 = 2 * j + (q >> 1) * 8;
      float hi[2], lo[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float v = (t0 + e < 9) ? w[ch * 9 + t0 + e] : 0.f;
        hi[e] = __bfloat162float(__float2bfloat16_rn(v));
        lo[e] = v - hi[e];
      }
      whi[m][q] = pack_bf16(hi[0], hi[1]);
      wlo[m][q] = pack_bf16(lo[0], lo[1]);
    }
  }
  // per-channel constants of this thread's channels (16 m + g, 16 m + g + 8)
  float c_fsh[NM][2], c_scl[NM][2], c_sft[NM][2], c_ds[NM][2];
#pragma unroll
  for (int m = 0; m < NM; ++m) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int ch = 16 * m + g + e * 8;
      c_fsh[m][e] = fwd_shift ? fwd_shift[ch] : 0.f;
      c_scl[m][e] = be.bn_scale ? be.bn_scale[ch] : 1.f;
      c_sft[m][e] = be.bn_shift ? be.bn_shift[ch] : 0.f;
      c_ds[m][e] = 1.f;
    }
  }
  const int act = be.act;
  float P0[NM][4], P1[NM][4];
#pragma unroll
  for (int m = 0; m < NM; ++m) {
#pragma unroll
    for (int e = 0; e < 4; ++e) { P0[m][e] = 0.f; P1[m][e] = 0.f; }
  }
  unsigned char* xt = tiles[warp][0];
  const uint32_t xt_s = (uint32_t)__cvta_generic_to_shared(xt);
  // this lane's row addresses for the three ldmatrix.x4 patterns (see the header comment); rows 4..7 of every group of 8
  // keep their two 16-byte halves swapped so that 8 consecutive rows hit 8 different bank groups
  const int lm = lane >> 3, lr = lane & 7;
  auto row_addr = [](uint32_t base, int px, int half) { return base + (uint32_t)(px * 32 + ((half ^ ((px >> 2) & 1)) << 4)); };
  __syncthreads();
  const int npix = Ho * Wo;
  const int spr = (Wo + 31) >> 5, nseg = Ho * spr;   // 32-pixel segments per output row / per image
  for (int task = blockIdx.x; task < ntasks; task += gridDim.x) {
    const int n = task / cpi, s0 = (task - n * cpi) * chunk;
    const int s1 = min(s0 + chunk, nseg);
    if (be.dropscale) {
#pragma unroll
      for (int m = 0; m < NM; ++m) {
        c_ds[m][0] = be.dropscale[(long long)n * CO + 16 * m + g];
        c_ds[m][1] = be.dropscale[(long long)n * CO + 16 * m + g + 8];
      }
    }
    const uint8_t* xim = x + (long long)n * H * W;
    const bf16* dim = da + (long long)n * npix * CO;
    SegCursor cur;
    cur.init(s0 + warp, spr);
    // software pipeline: the taps and the gradient row of the NEXT 32 pixels are requested before this iteration's tile is
    // staged and multiplied, so their HBM latency overlaps the ldmatrix / mma chain instead of heading it
    TapRaw<FAST> tn;
    bool pvn = false;
    uint4 dn[2 * NM];
    auto fetch = [&](const SegCursor& c) {
      const int wo = c.sg * 32 + lane;
      const bool pv = wo < Wo;
      pvn = pv;
      fetch_taps(tn, xim, H, W, stride, c.ho, wo, pv, lane);
#pragma unroll
      for (int i = 0; i < 2 * NM; ++i) dn[i] = make_uint4(0, 0, 0, 0);
      if (pv) {
        const uint4* gp = reinterpret_cast<const uint4*>(dim + ((long long)c.ho * Wo + wo) * CO);
#pragma unroll
        for (int m = 0; m < NM; ++m)
          asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                       : "=r"(dn[2 * m].x), "=r"(dn[2 * m].y), "=r"(dn[2 * m].z), "=r"(dn[2 * m].w), "=r"(dn[2 * m + 1].x),
                         "=r"(dn[2 * m + 1].y), "=r"(dn[2 * m + 1].z), "=r"(dn[2 * m + 1].w) : "l"(gp + 2 * m));
      }
    };
    if (s0 + warp < s1) fetch(cur);
    for (int sb = s0 + warp; sb < s1; sb += FM_WARPS) {
      // ---- stage the 32 pixels of this warp: thread = pixel
      {
        float v[9];
        uint4 d[2 * NM];
        const TapRaw<FAST> tc = tn;
        const bool pvc = pvn;
#pragma unroll
        for (int i = 0; i < 2 * NM; ++i) d[i] = dn[i];
        cur.advance(FM_WARPS, spr);
        if (sb + FM_WARPS < s1) fetch(cur);
        unpack_taps(tc, pvc, lane, v);
        const uint4 x0 = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
        const uint4 x1 = make_uint4(pack_bf16(v[8], 1.f), 0u, 0u, 0u);   // tap 8, the ones column, zero padding
        const int sw = (lane >> 2) & 1;
        __syncwarp();   // the previous iteration's ldmatrix reads are done
        *reinterpret_cast<uint4*>(xt + lane * 32 + ((0 ^ sw) << 4)) = x0;
        *reinterpret_cast<uint4*>(xt + lane * 32 + ((1 ^ sw) << 4)) = x1;
#pragma unroll
        for (int m = 0; m < NM; ++m) {
          unsigned char* dt = tiles[warp][1 + m];
          *reinterpret_cast<uint4*>(dt + lane * 32 + ((0 ^ sw) << 4)) = d[2 * m];
          *reinterpret_cast<uint4*>(dt + lane * 32 + ((1 ^ sw) << 4)) = d[2 * m + 1];
        }
        __syncwarp();
      }
#pragma unroll
      for (int kb = 0; kb < 2; ++kb) {   // two blocks of 16 pixels
        uint32_t b1[4], b2[4];
        ldsm_x4(b1, row_addr(xt_s, kb * 16 + (lm >> 1) * 8 + lr, lm & 1));      // MMA1 B: (k = taps, n = pixels), tiles 0 / 1
        ldsm_x4_t(b2, row_addr(xt_s, kb * 16 + (lm & 1) * 8 + lr, lm >> 1));    // MMA2 B: (k = pixels, n = taps 0-7 / 8-15)
#pragma unroll
        for (int m = 0; m < NM; ++m) {
          uint32_t dd[4];
          const uint32_t dt_s = xt_s + (uint32_t)((1 + m) * 32 * 32);
          ldsm_x4_t(dd, row_addr(dt_s, kb * 16 + (lm >> 1) * 8 + lr, lm & 1));    // DA in the accumulator layout, tiles 0 / 1
          uint32_t a2[4];
#pragma unroll
          for (int t = 0; t < 2; ++t) {    // two tiles of 8 pixels
            float c[4] = {0.f, 0.f, 0.f, 0.f};
            hmma16816(c, whi[m], b1[2 * t], b1[2 * t + 1]);
            hmma16816(c, wlo[m], b1[2 * t], b1[2 * t + 1]);
            float gv[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int hc = e >> 1;                       // channel g (0) or g + 8 (1); pixel 2j + (e & 1) of the tile
              const float yv = c[e] + c_fsh[m][hc];
              const float pre = be.bn_scale ? yv * c_scl[m][hc] + c_sft[m][hc] : yv;
              const uint32_t dword = dd[2 * t + hc];
              const float dav = __uint_as_float((e & 1) ? (dword & 0xFFFF0000u) : (dword << 16));
              gv[e] = dav * act_grad(pre, act) * c_ds[m][hc];
            }
            a2[2 * t] = pack_bf16(gv[0], gv[1]);
            a2[2 * t + 1] = pack_bf16(gv[2], gv[3]);
          }
          hmma16816(P0[m], a2, b2[0], b2[1]);
          hmma16816(P1[m], a2, b2[2], b2[3]);
        }
      }
    }
  }
  // P fragment: (ch g, taps 2j, 2j+1), (ch g+8, same); second tile: taps 8 + 2j .. -> tap 8 and the sum(g) column
#pragma unroll
  for (int m = 0; m < NM; ++m) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int ch = 16 * m + g + (e >> 1) * 8, t = 2 * j + (e & 1);
      atomicAdd(&red[ch * 9 + t], P0[m][e]);
      if (j == 0) {
        if ((e & 1) == 0) atomicAdd(&red[ch * 9 + 8], P1[m][e]);
        else atomicAdd(&red[9 * CO + ch], P1[m][e]);
      }
    }
  }
  __syncthreads();
  float* base = partial + (long long)blockIdx.x * (10 * CO);
  for (int i = threadIdx.x; i < 10 * CO; i += FM_WARPS * 32) base[i] = red[i];
}


// ------------------------------------------------------------------------------------------------
// Forward and Gram-matrix passes of the first layer on the warp-level tensor cores (uint8 image, 1 -> 16 channels),
// same staging as first_bwd_mma_kernel: per warp and 32 pixels the taps go to shared memory as an exact bf16 tile X[px][16]
// (9 taps, a ones column, zeros).
//   forward: acc^T[ch][px] = (W_hi + W_lo) . X^T, scale/shift/activation/Dropout2d in the accumulator layout, stmatrix.trans
//            turns it back into pixel-major rows, each thread stores the 32 bytes of its pixel.
//   Gram:    G = X^T . X (one mma per 16 pixels and 8 columns); the ones column makes G[:, 9] = S.  uint8 products are
//            integers: the fp32 accumulators are flushed to fp64 before they can exceed 2^24, so G and S are EXACT.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void stsm_x4_t(uint32_t addr, const uint32_t (&r)[4]) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};"
               ::"r"(addr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}

__device__ __forceinline__ void stage_taps_tile(unsigned char* xt, int lane, const float (&v)[9]) {
  const uint4 x0 = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
  const uint4 x1 = make_uint4(pack_bf16(v[8], 1.f), 0u, 0u, 0u);   // tap 8, the ones column, zero padding
  const int sw = (lane >> 2) & 1;
  *reinterpret_cast<uint4*>(xt + lane * 32 + ((0 ^ sw) << 4)) = x0;
  *reinterpret_cast<uint4*>(xt + lane * 32 + ((1 ^ sw) << 4)) = x1;
}

template <int NM, bool FAST>
__global__ void __launch_bounds__(FM_WARPS * 32, NM == 1 ? 8 : 6) first_fwd_mma_kernel(
    const uint8_t* __restrict__ x, const float* __restrict__ w, bf16* __restrict__ y, int H, int W, int Ho, int Wo,
    int stride, FwdEpi ep, int chunk, int cpi, int ntasks) {
  constexpr int CO = 16 * NM;
  __shared__ __align__(128) unsigned char tiles[FM_WARPS][1 + NM][32 * 32];   // per warp: X tile, NM output tiles of 16 channels
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, j = lane & 3;
  uint32_t whi[NM][4], wlo[NM][4];
  float c_sc[NM][2], c_sh[NM][2], c_ds[NM][2];
#pragma unroll
  for (int m = 0; m < NM; ++m) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int ch = 16 * m + g + (q & 1) * 8, t0 = 2 * j + (q >> 1) * 8;
      float hi[2], lo[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float v = (t0 + e < 9) ? w[ch * 9 + t0 + e] : 0.f;
        hi[e] = __bfloat162float(__float2bfloat16_rn(v));
        lo[e] = v - hi[e];
      }
      whi[m][q] = pack_bf16(hi[0], hi[1]);
      wlo[m][q] = pack_bf16(lo[0], lo[1]);
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int ch = 16 * m + g + e * 8;
      c_sc[m][e] = ep.scale ? ep.scale[ch] : 1.f;
      c_sh[m][e] = ep.shift ? ep.shift[ch] : 0.f;
      c_ds[m][e] = 1.f;
    }
  }
  const int act = ep.act;
  unsigned char* xt = tiles[warp][0];
  const uint32_t xt_s = (uint32_t)__cvta_generic_to_shared(xt);
  const int lm = lane >> 3, lr = lane & 7;
  auto row_addr = [](uint32_t base, int px, int half) { return base + (uint32_t)(px * 32 + ((half ^ ((px >> 2) & 1)) << 4)); };
  const int npix = Ho * Wo;
  const int spr = (Wo + 31) >> 5, nseg = Ho * spr;
  for (int task = blockIdx.x; task < ntasks; task += gridDim.x) {
    const int n = task / cpi, s0 = (task - n * cpi) * chunk;
    const int s1 = min(s0 + chunk, nseg);
    if (ep.dropscale) {
#pragma unroll
      for (int m = 0; m < NM; ++m) {
        c_ds[m][0] = ep.dropscale[(long long)n * CO + 16 * m + g];
        c_ds[m][1] = ep.dropscale[(long long)n * CO + 16 * m + g + 8];
      }
    }
    const uint8_t* xim = x + (long long)n * H * W;
    bf16* yim = y + (long long)n * npix * CO;
    SegCursor cur, nxt;
    cur.init(s0 + warp, spr);
    nxt = cur;
    TapRaw<FAST> tn;
    if (s0 + warp < s1) fetch_taps(tn, xim, H, W, stride, cur.ho, cur.sg * 32 + lane, cur.sg * 32 + lane < Wo, lane);
    for (int sb = s0 + warp; sb < s1; sb += FM_WARPS, cur = nxt) {
      const int wo = cur.sg * 32 + lane;
      const bool pv = wo < Wo;
      const TapRaw<FAST> tc = tn;
      nxt.advance(FM_WARPS, spr);
      if (sb + FM_WARPS < s1)   // the next segment's taps are in flight while this one is multiplied and stored
        fetch_taps(tn, xim, H, W, stride, nxt.ho, nxt.sg * 32 + lane, nxt.sg * 32 + lane < Wo, lane);
      float v[9];
      unpack_taps(tc, pv, lane, v);
      __syncwarp();
      stage_taps_tile(xt, lane, v);
      __syncwarp();
#pragma unroll
      for (int kb = 0; kb < 2; ++kb) {
        uint32_t b1[4];
        ldsm_x4(b1, row_addr(xt_s, kb * 16 + (lm >> 1) * 8 + lr, lm & 1));
#pragma unroll
        for (int m = 0; m < NM; ++m) {
          uint32_t o[4];
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            float c[4] = {0.f, 0.f, 0.f, 0.f};
            hmma16816(c, whi[m], b1[2 * t], b1[2 * t + 1]);
            hmma16816(c, wlo[m], b1[2 * t], b1[2 * t + 1]);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int hc = e >> 1;
              c[e] = act_fwd(c[e] * c_sc[m][hc] + c_sh[m][hc], act) * c_ds[m][hc];
            }
            o[2 * t] = pack_bf16(c[0], c[1]);       // (ch 16 m + g;     pixels 2j, 2j+1 of tile t)
            o[2 * t + 1] = pack_bf16(c[2], c[3]);   // (ch 16 m + g + 8; same pixels)
          }
          stsm_x4_t(row_addr(xt_s + (uint32_t)((1 + m) * 32 * 32), kb * 16 + (lm >> 1) * 8 + lr, lm & 1), o);
        }
      }
      __syncwarp();
      if (pv) {
        const int sw = (lane >> 2) & 1;
        uint4* dst = reinterpret_cast<uint4*>(yim + ((long long)cur.ho * Wo + wo) * CO);
#pragma unroll
        for (int m = 0; m < NM; ++m) {
          const unsigned char* yt = tiles[warp][1 + m];
          const uint4 lo = *reinterpret_cast<const uint4*>(yt + lane * 32 + ((0 ^ sw) << 4));
          const uint4 hi = *reinterpret_cast<const uint4*>(yt + lane * 32 + ((1 ^ sw) << 4));
          // the 16 channels of this M tile leave as one 32-byte store (a full sector) instead of two halves
          asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + 2 * m), "r"(lo.x), "r"(lo.y),
                       "r"(lo.z), "r"(lo.w), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w) : "memory");
        }
      }
    }
  }
}

template <bool FAST>
__global__ void __launch_bounds__(FM_WARPS * 32, 8) first_gram_mma_kernel(const uint8_t* __restrict__ x, int H, int W, int Ho,
                                                                          int Wo, int stride, double* __restrict__ gram,
                                                                          int chunk, int cpi, int ntasks) {
  __shared__ __align__(128) unsigned char tiles[FM_WARPS][32 * 32];
  __shared__ double red[54];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, j = lane & 3;
  if (threadIdx.x < 54) red[threadIdx.x] = 0.0;
  __syncthreads();
  unsigned char* xt = tiles[warp];
  const uint32_t xt_s = (uint32_t)__cvta_generic_to_shared(xt);
  const int lm = lane >> 3, lr = lane & 7;
  auto row_addr = [](uint32_t base, int px, int half) { return base + (uint32_t)(px * 32 + ((half ^ ((px >> 2) & 1)) << 4)); };
  float D0[4] = {0.f, 0.f, 0.f, 0.f}, D1[4] = {0.f, 0.f, 0.f, 0.f};
  // D0: (a = g | g+8, b = 2j, 2j+1);  D1: (a, b = 8 + 2j, 9 + 2j): b = 8 and the ones column b = 9 (= S[a]) for j == 0
  // The fp32 fragments hold exact integers < 2^24; every 7 iterations they move into 64-bit integer registers (8 conversions
  // and adds per lane instead of shared-memory fp64 atomics), which are reduced once
  // at the end.
  unsigned long long I0[4] = {0ull, 0ull, 0ull, 0ull}, I1[4] = {0ull, 0ull, 0ull, 0ull};
  auto flush = [&]() {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      I0[e] += (unsigned long long)__float2uint_rn(D0[e]);
      I1[e] += (unsigned long long)__float2uint_rn(D1[e]);
      D0[e] = 0.f; D1[e] = 0.f;
    }
  };
  auto reduce = [&]() {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int a = g + (e >> 1) * 8, b = 2 * j + (e & 1);
      if (a <= 8 && a <= b) atomicAdd(&red[9 + a * 9 - a * (a - 1) / 2 + (b - a)], (double)I0[e]);
      if (a <= 8 && j == 0) {
        if ((e & 1) == 0) atomicAdd(&red[9 + a * 9 - a * (a - 1) / 2 + (8 - a)], (double)I1[e]);   // G[a][8]
        else atomicAdd(&red[a], (double)I1[e]);                                                         // S[a]
      }
    }
  };
  const int spr = (Wo + 31) >> 5, nseg = Ho * spr;
  int since_flush = 0;
  for (int task = blockIdx.x; task < ntasks; task += gridDim.x) {
    const int n = task / cpi, s0 = (task - n * cpi) * chunk;
    const int s1 = min(s0 + chunk, nseg);
    const uint8_t* xim = x + (long long)n * H * W;
    SegCursor cur, nxt;
    cur.init(s0 + warp, spr);
    nxt = cur;
    TapRaw<FAST> tn;
    if (s0 + warp < s1) fetch_taps(tn, xim, H, W, stride, cur.ho, cur.sg * 32 + lane, cur.sg * 32 + lane < Wo, lane);
    for (int sb = s0 + warp; sb < s1; sb += FM_WARPS, cur = nxt) {
      const int wo = cur.sg * 32 + lane;
      const bool pv = wo < Wo;
      const TapRaw<FAST> tc = tn;
      nxt.advance(FM_WARPS, spr);
      if (sb + FM_WARPS < s1)
        fetch_taps(tn, xim, H, W, stride, nxt.ho, nxt.sg * 32 + lane, nxt.sg * 32 + lane < Wo, lane);
      float v[9];
      unpack_taps(tc, pv, lane, v);
      __syncwarp();
      stage_taps_tile(xt, lane, v);
      if (!pv) *reinterpret_cast<uint4*>(xt + lane * 32 + ((1 ^ ((lane >> 2) & 1)) << 4)) = make_uint4(0, 0, 0, 0);   // no ones
      __syncwarp();
#pragma unroll
      for (int kb = 0; kb < 2; ++kb) {
        uint32_t a[4], b[4];
        ldsm_x4_t(a, row_addr(xt_s, kb * 16 + (lm >> 1) * 8 + lr, lm & 1));   // A[m = tap][k = pixel]
        ldsm_x4_t(b, row_addr(xt_s, kb * 16 + (lm & 1) * 8 + lr, lm >> 1));   // B[k = pixel][n = tap]
        hmma16816(D0, a, b[0], b[1]);
        hmma16816(D1, a, b[2], b[3]);
      }
      // 32 pixels add at most 32 * 255^2 < 2^21 to an accumulator: flushing every 7 iterations keeps it below 2^24 (exact)
      if (++since_flush == 7) { flush(); since_flush = 0; }
    }
  }
  flush();
  reduce();   // (per-lane totals stay below 2^53 for any image this kernel accepts: exact in fp64)
  __syncthreads();
  if (threadIdx.x < 54) atomicAdd(&gram[threadIdx.x], red[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------
// Input gradient of the first layer: dx = conv_transpose(dz, W) onto the fp32 NCHW image, with dz = d(loss)/d(conv output)
// recomputed from (image, da) the way conv_first_bwd_kernel / first_bwd16_kernel do it (same stencil order, same
// pre-activation expression, so a pre-activation on the LeakyReLU kink takes the same slope as in the weight gradient).
// One CTA = FD_OH x FD_OW output pixels = (FD_OH*stride) x (FD_OW*stride) input pixels, per 16-channel chunk:
//   phase 1: dz of the tile's output pixels plus the one-pixel halo its input pixels read, into shared memory
//   phase 2: each thread gathers the taps of its input pixels from shared memory (no atomics).  At stride 2 a warp holds
//            32 input pixels of one row and one column parity, so every lane of it takes the same taps (1 or 2 per axis).
// ------------------------------------------------------------------------------------------------
constexpr int FD_OH = 8, FD_OW = 32, FD_CO = 16, FD_THREADS = 128;
constexpr int FD_DZS = FD_CO + 4;   // shared-memory pitch of one dz pixel: float4 reads of 8 consecutive pixels hit 32 banks
constexpr int FD_DZ_PIX = (FD_OH + 2) * (FD_OW + 2);   // stride 1: one halo pixel on each side (stride 2: one at the end)

// input pixel p of a tile -> (row, column) inside the tile; at stride 2 a run of 32 is one row and one column parity
template <int STRIDE>
__device__ __forceinline__ void fd_pixel(int p, int& ihl, int& iwl) {
  if (STRIDE == 2) { ihl = p / 64; const int rem = p % 64; iwl = 2 * (rem % 32) + rem / 32; }
  else { ihl = p / FD_OW; iwl = p % FD_OW; }
}

template <typename T, int STRIDE>
__global__ void __launch_bounds__(FD_THREADS, 3) first_dgrad_kernel(
    const float* __restrict__ x, const float* __restrict__ w, const T* __restrict__ da, float* __restrict__ dx,
    int H, int W, int Cin, int Ho, int Wo, int Cout, BwdEpi be, const float* __restrict__ fwd_shift,
    const float* __restrict__ dy_mean, const float* __restrict__ dyx_mean, int tiles_h, int tiles_w) {
  __shared__ __align__(16) float ws[3 * 9 * FD_CO];        // [ci * 9 + tap][co]
  __shared__ float cst[8 * FD_CO];                          // scl, sft, mean, istd, m1, m2, fsh, dropscale
  __shared__ __align__(16) float dz[FD_DZ_PIX * FD_DZS];
  const int tile = blockIdx.x;
  const int n = tile / (tiles_h * tiles_w), tr = tile - n * tiles_h * tiles_w;
  const int oh0 = (tr / tiles_w) * FD_OH, ow0 = (tr % tiles_w) * FD_OW;
  constexpr int stride = STRIDE, NPT = STRIDE * STRIDE * FD_OH * FD_OW / FD_THREADS;   // input pixels per thread
  const int ih0 = oh0 * stride, iw0 = ow0 * stride;
  const int tih = FD_OH * stride, tiw = FD_OW * stride;
  // output pixels the tile's input pixels receive from: ho * stride - 1 + r = ih, r = 0..2
  const int ho_lo = max(0, (ih0 - 1 + stride - 1) / stride), ho_hi = min(Ho - 1, (ih0 + tih) / stride);
  const int wo_lo = max(0, (iw0 - 1 + stride - 1) / stride), wo_hi = min(Wo - 1, (iw0 + tiw) / stride);
  const int nrow = ho_hi - ho_lo + 1, ncol = wo_hi - wo_lo + 1;
  const bool bn = be.bn_scale != nullptr, bn_batch = bn && dy_mean != nullptr;
  float acc[NPT][3];
#pragma unroll
  for (int k = 0; k < NPT; ++k)
#pragma unroll
    for (int ci = 0; ci < 3; ++ci) acc[k][ci] = 0.f;

  for (int co0 = 0; co0 < Cout; co0 += FD_CO) {
    __syncthreads();   // the previous chunk's dz / weights are no longer read
    load_first_weights<FD_CO>(ws, w, Cin, Cout, co0);
    if (threadIdx.x < FD_CO) {
      const int c = threadIdx.x, co = co0 + c;
      const bool ok = co < Cout;
      cst[c] = (bn && ok) ? be.bn_scale[co] : 1.f;
      cst[FD_CO + c] = (bn && ok) ? be.bn_shift[co] : 0.f;
      cst[2 * FD_CO + c] = (bn && ok) ? be.bn_mean[co] : 0.f;
      cst[3 * FD_CO + c] = (bn && ok) ? be.bn_invstd[co] : 1.f;
      cst[4 * FD_CO + c] = (bn_batch && ok) ? dy_mean[co] : 0.f;
      cst[5 * FD_CO + c] = (bn_batch && ok) ? dyx_mean[co] : 0.f;
      cst[6 * FD_CO + c] = (fwd_shift && ok) ? fwd_shift[co] : 0.f;
      cst[7 * FD_CO + c] = (be.dropscale && ok) ? be.dropscale[(long long)n * Cout + co] : 1.f;
    }
    __syncthreads();
    // ---- phase 1: dz of the (halo) output pixels
    for (int q = threadIdx.x; q < nrow * ncol; q += FD_THREADS) {
      const int ho = ho_lo + q / ncol, wo = wo_lo + q % ncol;
      float a[FD_CO];
      first_conv_pixel<float, FD_CO>(x, ws, n, ho, wo, H, W, Cin, stride, a);
      const T* dp = da + (((long long)n * Ho + ho) * Wo + wo) * Cout + co0;
      float* out = dz + q * FD_DZS;
#pragma unroll
      for (int c = 0; c < FD_CO; ++c) {
        float d = 0.f;
        if (co0 + c < Cout) {
          float g = to_f<T>(dp[c]) * cst[7 * FD_CO + c];
          const float yv = a[c] + cst[6 * FD_CO + c];   // conv output (+bias when no BN)
          float pre = yv;
          if (bn) pre = yv * cst[c] + cst[FD_CO + c];
          g *= act_grad(pre, be.act);
          if (bn_batch) {
            const float xhat = (yv - cst[2 * FD_CO + c]) * cst[3 * FD_CO + c];
            d = cst[c] * (g - cst[4 * FD_CO + c] - xhat * cst[5 * FD_CO + c]);
          } else {
            d = bn ? cst[c] * g : g;
          }
        }
        out[c] = d;
      }
    }
    __syncthreads();
    // ---- phase 2: transposed 3x3 convolution, gathered per input pixel
#pragma unroll
    for (int k = 0; k < NPT; ++k) {
      int ihl, iwl;
      fd_pixel<STRIDE>(threadIdx.x + k * FD_THREADS, ihl, iwl);
      const int ih = ih0 + ihl, iw = iw0 + iwl;
      if (ih >= H || iw >= W) continue;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const int th = ih + 1 - r;
        if (th < 0 || (stride == 2 && (th & 1))) continue;
        const int ho = th / stride;
        if (ho >= Ho) continue;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          const int tw = iw + 1 - s;
          if (tw < 0 || (stride == 2 && (tw & 1))) continue;
          const int wo = tw / stride;
          if (wo >= Wo) continue;
          const float* d = dz + ((ho - ho_lo) * ncol + (wo - wo_lo)) * FD_DZS;
#pragma unroll
          for (int c4 = 0; c4 < FD_CO / 4; ++c4) {
            const float4 dv = reinterpret_cast<const float4*>(d)[c4];
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) {
              if (ci < Cin) {
                const float4 wv = reinterpret_cast<const float4*>(ws + (ci * 9 + r * 3 + s) * FD_CO)[c4];
                acc[k][ci] += dv.x * wv.x + dv.y * wv.y + dv.z * wv.z + dv.w * wv.w;
              }
            }
          }
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < NPT; ++k) {
    int ihl, iwl;
    fd_pixel<STRIDE>(threadIdx.x + k * FD_THREADS, ihl, iwl);
    const int ih = ih0 + ihl, iw = iw0 + iwl;
    if (ih >= H || iw >= W) continue;
#pragma unroll
    for (int ci = 0; ci < 3; ++ci)
      if (ci < Cin) dx[(((long long)n * Cin + ci) * H + ih) * W + iw] = acc[k][ci];
  }
}

// m1 = sum(g') / M and m2 = sum(g' xhat) / M of the Gram path from its raw P / Sg (the clamped dgamma / dbeta cannot be used)
__global__ void first_bn_means_kernel(const float* __restrict__ P, const float* __restrict__ Sg, const float* __restrict__ w,
                                      const float* __restrict__ bias, const float* __restrict__ mean,
                                      const float* __restrict__ invstd, double count, int Cout, float* __restrict__ m1,
                                      float* __restrict__ m2) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Cout) return;
  const double bi = bias ? (double)bias[c] : 0.0;
  double wp = 0.0;
  for (int t = 0; t < 9; ++t) wp += (double)w[c * 9 + t] * (double)P[c * 9 + t];
  const double sg = Sg[c];
  m1[c] = (float)(sg / count);
  m2[c] = (float)((double)invstd[c] * (wp + (bi - (double)mean[c]) * sg) / count);
}

constexpr int FL_BWD_BLOCKS = 592;

// aligned 16-bit tap loads: stride 2, even width (every row starts on an even offset) and an even base address
static bool first_fast_taps(const void* x, int W, int stride) {
  return stride == 2 && (W & 1) == 0 && (reinterpret_cast<uintptr_t>(x) & 1u) == 0;
}

}  // namespace yg

using namespace yg;

extern "C" int yg_conv_first_fwd(const void* x, int x_dtype, const float* w, void* y, int dtype,
                                 int N, int H, int W, int Cin, int Cout, int stride,
                                 const yg_fwd_epilogue* epp, void* stream) {
  YG_CHECK_ARG(x && w, "conv_first_fwd: null pointer");
  YG_CHECK_ARG(Cin >= 1 && Cin <= 3, "conv_first_fwd: Cin must be 1..3, got %d", Cin);
  YG_CHECK_ARG(stride == 1 || stride == 2, "conv_first_fwd: stride %d", stride);
  YG_CHECK_ARG(x_dtype == YG_U8 || x_dtype == YG_F32, "conv_first_fwd: x_dtype %d", x_dtype);
  YG_CHECK_ARG(dtype == YG_F32 || dtype == YG_BF16, "conv_first_fwd: dtype %d", dtype);
  if (N == 0) return YG_OK;
  FwdEpi ep = make_fwd_epi(epp);
  const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (Cin == 1 && (Cout == 16 || Cout == 32 || Cout == 48) && dtype == YG_BF16 && !ep.preact && (long long)Ho * Wo < (1LL << 30) &&
      (long long)H * W < (1LL << 31) && x_dtype == YG_U8 && !ep.stats && y && (reinterpret_cast<uintptr_t>(y) & 31u) == 0 &&
      yg_get_conv_impl() != YG_IMPL_SIMT) {
    // warp-level tensor cores, one M tile per 16 output channels (base 16, double_filters 32, triple_filters 48)
    // tasks of 16 row segments (32 pixels of one output row) per warp
    const int chunkm = 16 * FM_WARPS, cpim = cdiv((long long)Ho * cdiv(Wo, 32), chunkm), ntasksm = N * cpim;
    const int per_sm = Cout == 16 ? 8 : 6;
    const int gridm = ntasksm < 148 * per_sm ? ntasksm : 148 * per_sm;
    const bool fast = first_fast_taps(x, W, stride);
#define LAUNCHM(NM) do { if (fast) first_fwd_mma_kernel<NM, true><<<gridm, FM_WARPS * 32, 0, st>>>((const uint8_t*)x, w, (bf16*)y, H, W, Ho, Wo, stride, ep, chunkm, cpim, ntasksm); \
                         else first_fwd_mma_kernel<NM, false><<<gridm, FM_WARPS * 32, 0, st>>>((const uint8_t*)x, w, (bf16*)y, H, W, Ho, Wo, stride, ep, chunkm, cpim, ntasksm); } while (0)
    if (Cout == 16) LAUNCHM(1); else if (Cout == 32) LAUNCHM(2); else LAUNCHM(3);
#undef LAUNCHM
    YG_LAUNCH_CHECK("conv_first_fwd_mma");
    return YG_OK;
  }
  if (Cin == 1 && Cout == FF_CO && dtype == YG_BF16 && !ep.preact && (long long)Ho * Wo < (1LL << 30) &&
      (long long)H * W < (1LL << 31)) {
    const int chunk = 16 * FL_THREADS, cpi = cdiv((long long)Ho * Wo, chunk), ntasks = N * cpi;
    const int grid1 = ntasks < 148 * 3 ? ntasks : 148 * 3;
#define LAUNCHF(TX, ST) first_fwd16_kernel<TX, ST><<<grid1, FL_THREADS, 0, st>>>((const TX*)x, w, (bf16*)y, H, W, Ho, Wo, stride, ep, chunk, cpi, ntasks)
    if (x_dtype == YG_U8) { if (ep.stats) LAUNCHF(uint8_t, true); else LAUNCHF(uint8_t, false); }
    else { if (ep.stats) LAUNCHF(float, true); else LAUNCHF(float, false); }
#undef LAUNCHF
    YG_LAUNCH_CHECK("conv_first_fwd16");
    return YG_OK;
  }
  long long nblk = ((long long)N * Ho * Wo + FL_THREADS - 1) / FL_THREADS;
  if (nblk > 148 * 16) nblk = 148 * 16;
  dim3 grid((unsigned)nblk, cdiv(Cout, FL_CO), 1);
#define LAUNCH(TX, T) conv_first_fwd_kernel<TX, T><<<grid, FL_THREADS, 0, st>>>((const TX*)x, w, (T*)y, N, H, W, Cin, Ho, Wo, Cout, stride, ep)
  if (x_dtype == YG_U8) { if (dtype == YG_BF16) LAUNCH(uint8_t, bf16); else LAUNCH(uint8_t, float); }
  else { if (dtype == YG_BF16) LAUNCH(float, bf16); else LAUNCH(float, float); }
#undef LAUNCH
  YG_LAUNCH_CHECK("conv_first_fwd");
  return YG_OK;
}

extern "C" int yg_conv_first_bwd(const void* x, int x_dtype, const float* w, const void* da, int dtype,
                                 int N, int H, int W, int Cin, int Cout, int stride,
                                 const yg_bwd_epilogue* bep, const float* fwd_shift,
                                 const float* bn_dy_mean, const float* bn_dyx_mean,
                                 float* dw, float* dshift, float clip, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  YG_CHECK_ARG(x && w && da, "conv_first_bwd: null pointer");
  YG_CHECK_ARG(Cin >= 1 && Cin <= 3, "conv_first_bwd: Cin must be 1..3, got %d", Cin);
  YG_CHECK_ARG(x_dtype == YG_U8 || x_dtype == YG_F32, "conv_first_bwd: x_dtype %d", x_dtype);
  if (N == 0) return YG_OK;
  BwdEpi be = make_bwd_epi(bep);
  const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
  const int nchunks = cdiv(Cout, FLB_CO);
  cudaStream_t st = (cudaStream_t)stream;
  const int mode = dw ? 1 : 0;
  YG_CHECK_ARG(mode == 1 || be.bn_sums, "conv_first_bwd: pass 1 needs bn_sums");
  long long total = (long long)N * Ho * Wo;
  int blocks = (int)((total + FL_THREADS - 1) / FL_THREADS);
  if (blocks > FL_BWD_BLOCKS) blocks = FL_BWD_BLOCKS;
  const long long nw = (long long)Cout * Cin * 9;
  if (mode == 1) {
    size_t need = (size_t)blocks * (nw + Cout) * sizeof(float);
    if (!workspace || workspace_bytes < need) {
      set_error("conv_first_bwd: workspace %zu < %zu", workspace_bytes, need);
      return YG_ERR_WORKSPACE;
    }
  }
  if (mode == 1 && Cin == 1 && (Cout == 16 || Cout == 32 || Cout == 48) && dtype == YG_BF16 && x_dtype == YG_U8 && !bn_dy_mean &&
      Wo >= 32 && (long long)Ho * Wo < (1LL << 30) && (long long)H * W < (1LL << 31) && (reinterpret_cast<uintptr_t>(da) & 31u) == 0 &&
      yg_get_conv_impl() != YG_IMPL_SIMT) {
    // raw P / Sg pass on the tensor cores (first_bwd_mma_kernel), one M tile per 16 output channels
    const int chunk = 64 * FM_WARPS, cpi = cdiv((long long)Ho * cdiv(Wo, 32), chunk), ntasks = N * cpi;
    const int grid1 = ntasks < FL_BWD_BLOCKS ? ntasks : FL_BWD_BLOCKS;
    const bool fast = first_fast_taps(x, W, stride);
#define LAUNCHM(NM) do { if (fast) first_bwd_mma_kernel<NM, true><<<grid1, FM_WARPS * 32, 0, st>>>((const uint8_t*)x, w, (const bf16*)da, H, W, Ho, Wo, stride, be, fwd_shift, (float*)workspace, chunk, cpi, ntasks); \
                         else first_bwd_mma_kernel<NM, false><<<grid1, FM_WARPS * 32, 0, st>>>((const uint8_t*)x, w, (const bf16*)da, H, W, Ho, Wo, stride, be, fwd_shift, (float*)workspace, chunk, cpi, ntasks); } while (0)
    if (Cout == 16) LAUNCHM(1); else if (Cout == 32) LAUNCHM(2); else LAUNCHM(3);
#undef LAUNCHM
    YG_LAUNCH_CHECK("conv_first_bwd_mma");
    wgrad_reduce_kernel2<<<cdiv((nw + Cout) * 32, 256), 256, 0, st>>>((const float*)workspace, dw, dshift, nw, Cout, grid1, clip);
    YG_LAUNCH_CHECK("conv_first_bwd reduce");
    return YG_OK;
  }
  if (mode == 1 && Cin == 1 && Cout == FF_CO && dtype == YG_BF16 && (long long)Ho * Wo < (1LL << 30) &&
      (long long)H * W < (1LL << 31)) {
    const int chunk = 32 * FL_THREADS, cpi = cdiv((long long)Ho * Wo, chunk), ntasks = N * cpi;
    const int grid1 = ntasks < 222 ? ntasks : 222;   // x 2 channel groups = one wave of 3 blocks per SM; <= FL_BWD_BLOCKS slices
    const dim3 gridf(grid1, 2, 1);
    if (x_dtype == YG_U8)
      first_bwd16_kernel<uint8_t, 8><<<gridf, FL_THREADS, 0, st>>>((const uint8_t*)x, w, (const bf16*)da, H, W, Ho, Wo, stride, be,
                                                                   fwd_shift, bn_dy_mean, bn_dyx_mean, (float*)workspace, chunk, cpi, ntasks);
    else
      first_bwd16_kernel<float, 8><<<gridf, FL_THREADS, 0, st>>>((const float*)x, w, (const bf16*)da, H, W, Ho, Wo, stride, be,
                                                                 fwd_shift, bn_dy_mean, bn_dyx_mean, (float*)workspace, chunk, cpi, ntasks);
    YG_LAUNCH_CHECK("conv_first_bwd16");
    wgrad_reduce_kernel2<<<cdiv((nw + Cout) * 32, 256), 256, 0, st>>>((const float*)workspace, dw, dshift, nw, Cout, grid1, clip);
    YG_LAUNCH_CHECK("conv_first_bwd reduce");
    return YG_OK;
  }
  dim3 grid(blocks, nchunks * (mode == 1 ? Cin : 1), 1);
#define LAUNCH(TX, T, M) conv_first_bwd_kernel<TX, T, M><<<grid, FL_THREADS, 0, st>>>((const TX*)x, w, (const T*)da, N, H, W, Cin, Ho, Wo, Cout, stride, be, fwd_shift, bn_dy_mean, bn_dyx_mean, (float*)workspace, nchunks)
#define LAUNCH_M(TX, T) do { if (mode == 1) LAUNCH(TX, T, 1); else LAUNCH(TX, T, 0); } while (0)
  if (x_dtype == YG_U8) { if (dtype == YG_BF16) LAUNCH_M(uint8_t, bf16); else LAUNCH_M(uint8_t, float); }
  else { if (dtype == YG_BF16) LAUNCH_M(float, bf16); else LAUNCH_M(float, float); }
#undef LAUNCH_M
#undef LAUNCH
  YG_LAUNCH_CHECK("conv_first_bwd");
  if (mode == 1) {
    wgrad_reduce_kernel2<<<cdiv((nw + Cout) * 32, 256), 256, 0, st>>>((const float*)workspace, dw, dshift, nw, Cout, blocks, clip);
    YG_LAUNCH_CHECK("conv_first_bwd reduce");
  }
  return YG_OK;
}

extern "C" size_t yg_conv_first_bwd_workspace(int Cin, int Cout) {
  return (size_t)FL_BWD_BLOCKS * ((size_t)Cout * Cin * 9 + Cout) * sizeof(float);
}

// ------------------------------------------------------------------------------------------------
// Single-channel images: BatchNorm statistics and the BN part of the backward are obtained
// algebraically from the 9-tap Gram matrix of the image instead of extra passes over the activations.
//   y_c(px) = sum_t w[c][t] x_t(px) (+ bias)            x_t = the 9 shifted / strided views of the image
//   sum y_c   = w_c . S + bias*M,   sum y_c^2 = w_c^T G w_c + 2 bias (w_c . S) + bias^2 M
//   S_t = sum_px x_t,  G[t][t'] = sum_px x_t x_t'        (channel independent, 9 + 45 numbers)
// Backward: P[c][t] = sum g x_t and Sg[c] = sum g come from ONE pass over (da, image); sum g*xhat,
// dgamma, dbeta and dW follow in closed form from P, Sg, S, G (yg_conv_first_bwd_finalize).
// ------------------------------------------------------------------------------------------------
namespace yg {

constexpr int GR_THREADS = 256;

template <typename TX>
__global__ void __launch_bounds__(GR_THREADS) first_gram_kernel(const TX* __restrict__ x, int N, int H, int W,
                                                                int Ho, int Wo, int stride, double* __restrict__ gram,
                                                                int chunk, int cpi, int ntasks) {
  float S[9], G[45];
#pragma unroll
  for (int i = 0; i < 9; ++i) S[i] = 0.f;
#pragma unroll
  for (int i = 0; i < 45; ++i) G[i] = 0.f;
  const int npix = Ho * Wo;
  // (image, pixel chunk) tasks with an incrementally advanced (ho, wo): no per-pixel division
  for (int task = blockIdx.x; task < ntasks; task += gridDim.x) {
    const int n = task / cpi, p0 = (task - n * cpi) * chunk;
    const int p1 = min(p0 + chunk, npix);
    const TX* xim = x + (long long)n * H * W;
    PixCursor cur;
    cur.init(p0 + (int)threadIdx.x, Wo);
    for (; cur.p < p1; cur.advance(GR_THREADS, Wo)) {
      float v[9];
      load_taps1<TX>(xim, H, W, stride, cur.ho, cur.wo, v);
      int k = 0;
#pragma unroll
      for (int a = 0; a < 9; ++a) {
        S[a] += v[a];
#pragma unroll
        for (int b = a; b < 9; ++b) G[k++] += v[a] * v[b];
      }
    }
  }
  __shared__ double red[54];
  if (threadIdx.x < 54) red[threadIdx.x] = 0.0;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const float s = warp_sum(S[i]);
    if ((threadIdx.x & 31) == 0) atomicAdd(&red[i], (double)s);
  }
#pragma unroll
  for (int i = 0; i < 45; ++i) {
    const float s = warp_sum(G[i]);
    if ((threadIdx.x & 31) == 0) atomicAdd(&red[9 + i], (double)s);
  }
  __syncthreads();
  if (threadIdx.x < 54) atomicAdd(&gram[threadIdx.x], red[threadIdx.x]);
}

__device__ __forceinline__ double gram_at(const double* gram, int a, int b) {
  if (a > b) { const int t = a; a = b; b = t; }
  // upper triangle, row-major: offset(a) = sum_{i<a} (9 - i) = a*9 - a*(a-1)/2
  return gram[9 + a * 9 - a * (a - 1) / 2 + (b - a)];
}

__global__ void first_stats_from_gram_kernel(const double* __restrict__ gram, const float* __restrict__ w,
                                             const float* __restrict__ bias, double count, int Cout,
                                             double* __restrict__ stats) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Cout) return;
  double ws = 0.0, q = 0.0;
  for (int a = 0; a < 9; ++a) {
    const double wa = w[c * 9 + a];
    ws += wa * gram[a];
    for (int b = 0; b < 9; ++b) q += wa * (double)w[c * 9 + b] * gram_at(gram, a, b);
  }
  const double bi = bias ? (double)bias[c] : 0.0;
  stats[c] += ws + bi * count;
  stats[Cout + c] += q + 2.0 * bi * ws + bi * bi * count;
}

__global__ void first_bwd_finalize_kernel(const float* __restrict__ P, const float* __restrict__ Sg,
                                          const double* __restrict__ gram, const float* __restrict__ w,
                                          const float* __restrict__ bias, const float* __restrict__ gamma,
                                          const float* __restrict__ mean, const float* __restrict__ invstd,
                                          double count, int batch_stats, float clip, int Cout,
                                          float* __restrict__ dw, float* __restrict__ dbias,
                                          float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Cout) return;
  const double bi = bias ? (double)bias[c] : 0.0;
  const double mu = mean[c], is = invstd[c], ga = gamma ? (double)gamma[c] : 1.0;
  const double sg = Sg[c];
  double wp = 0.0;
  for (int t = 0; t < 9; ++t) wp += (double)w[c * 9 + t] * (double)P[c * 9 + t];
  const double sgx = is * (wp + (bi - mu) * sg);  // sum g * xhat
  if (dgamma) dgamma[c] = clampf((float)sgx, clip);
  if (dbeta) dbeta[c] = clampf((float)sg, clip);
  const double m1 = batch_stats ? sg / count : 0.0, m2 = batch_stats ? sgx / count : 0.0;
  const double scl = ga * is;
  double sum_x = 0.0;  // sum over pixels of xhat (for d bias)
  for (int t = 0; t < 9; ++t) {
    double wg = 0.0;
    for (int u = 0; u < 9; ++u) wg += (double)w[c * 9 + u] * gram_at(gram, u, t);
    const double X = is * (wg + (bi - mu) * gram[t]);  // sum xhat * x_t
    dw[c * 9 + t] = clampf((float)(scl * ((double)P[c * 9 + t] - m1 * gram[t] - m2 * X)), clip);
  }
  if (dbias) {
    double ws = 0.0;
    for (int t = 0; t < 9; ++t) ws += (double)w[c * 9 + t] * gram[t];
    sum_x = is * (ws + (bi - mu) * count);
    dbias[c] = clampf((float)(scl * (sg - m1 * count - m2 * sum_x)), clip);
  }
}

}  // namespace yg

extern "C" int yg_conv_first_gram(const void* x, int x_dtype, int N, int H, int W, int stride, double* gram,
                                  void* stream) {
  YG_CHECK_ARG(x && gram, "conv_first_gram: null pointer");
  YG_CHECK_ARG(x_dtype == YG_U8 || x_dtype == YG_F32, "conv_first_gram: x_dtype %d", x_dtype);
  YG_CHECK_ARG(stride == 1 || stride == 2, "conv_first_gram: stride %d", stride);
  cudaStream_t st = (cudaStream_t)stream;
  YG_CUDA(cudaMemsetAsync(gram, 0, 54 * sizeof(double), st));
  if (N == 0) return YG_OK;
  const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
  YG_CHECK_ARG((long long)Ho * Wo < (1LL << 30) && (long long)H * W < (1LL << 31), "conv_first_gram: image too large");
  if (x_dtype == YG_U8 && yg_get_conv_impl() != YG_IMPL_SIMT) {
    const int chunkm = 32 * FM_WARPS, cpim = cdiv((long long)Ho * cdiv(Wo, 32), chunkm), ntasksm = N * cpim;
    const int gridm = ntasksm < 148 * 8 ? ntasksm : 148 * 8;
    if (first_fast_taps(x, W, stride))
      first_gram_mma_kernel<true><<<gridm, FM_WARPS * 32, 0, st>>>((const uint8_t*)x, H, W, Ho, Wo, stride, gram, chunkm, cpim, ntasksm);
    else
      first_gram_mma_kernel<false><<<gridm, FM_WARPS * 32, 0, st>>>((const uint8_t*)x, H, W, Ho, Wo, stride, gram, chunkm, cpim, ntasksm);
    YG_LAUNCH_CHECK("first_gram_mma");
    return YG_OK;
  }
  const int chunk = 32 * GR_THREADS, cpi = cdiv((long long)Ho * Wo, chunk), ntasks = N * cpi;
  const int nblk = ntasks < 148 * 4 ? ntasks : 148 * 4;
  if (x_dtype == YG_U8)
    first_gram_kernel<uint8_t><<<nblk, GR_THREADS, 0, st>>>((const uint8_t*)x, N, H, W, Ho, Wo, stride, gram, chunk, cpi, ntasks);
  else
    first_gram_kernel<float><<<nblk, GR_THREADS, 0, st>>>((const float*)x, N, H, W, Ho, Wo, stride, gram, chunk, cpi, ntasks);
  YG_LAUNCH_CHECK("first_gram");
  return YG_OK;
}

extern "C" int yg_conv_first_stats_from_gram(const double* gram, const float* w, const float* bias, double count,
                                             int Cout, double* stats, void* stream) {
  YG_CHECK_ARG(gram && w && stats && Cout > 0, "conv_first_stats_from_gram: bad arguments");
  first_stats_from_gram_kernel<<<cdiv(Cout, 64), 64, 0, (cudaStream_t)stream>>>(gram, w, bias, count, Cout, stats);
  YG_LAUNCH_CHECK("first_stats_from_gram");
  return YG_OK;
}

extern "C" int yg_conv_first_bwd_finalize(const float* P, const float* Sg, const double* gram, const float* w,
                                          const float* bias, const float* gamma, const float* mean,
                                          const float* invstd, double count, int batch_stats, float clip, int Cout,
                                          float* dw, float* dbias, float* dgamma, float* dbeta, void* stream) {
  YG_CHECK_ARG(P && Sg && gram && w && mean && invstd && dw && Cout > 0, "conv_first_bwd_finalize: bad arguments");
  first_bwd_finalize_kernel<<<cdiv(Cout, 64), 64, 0, (cudaStream_t)stream>>>(P, Sg, gram, w, bias, gamma, mean, invstd,
                                                                             count, batch_stats, clip, Cout, dw, dbias,
                                                                             dgamma, dbeta);
  YG_LAUNCH_CHECK("first_bwd_finalize");
  return YG_OK;
}

extern "C" int yg_conv_first_dgrad(const float* x, const float* w, const void* da, int dtype, int N, int H, int W, int Cin,
                                   int Cout, int stride, const yg_bwd_epilogue* bep, const float* fwd_shift,
                                   const float* bn_dy_mean, const float* bn_dyx_mean, float* dx, void* stream) {
  YG_CHECK_ARG(x && w && da && dx, "conv_first_dgrad: null pointer");
  YG_CHECK_ARG(Cin >= 1 && Cin <= 3, "conv_first_dgrad: Cin must be 1..3, got %d", Cin);
  YG_CHECK_ARG(Cout >= 1, "conv_first_dgrad: Cout %d", Cout);
  YG_CHECK_ARG(stride == 1 || stride == 2, "conv_first_dgrad: stride %d", stride);
  YG_CHECK_ARG(dtype == YG_F32 || dtype == YG_BF16, "conv_first_dgrad: dtype %d", dtype);
  YG_CHECK_ARG((bn_dy_mean == nullptr) == (bn_dyx_mean == nullptr), "conv_first_dgrad: pass both BN means or neither");
  BwdEpi be = make_bwd_epi(bep);
  YG_CHECK_ARG(!be.bn_scale || (be.bn_shift && be.bn_mean && be.bn_invstd), "conv_first_dgrad: incomplete BN epilogue");
  YG_CHECK_ARG(be.bn_scale || !bn_dy_mean, "conv_first_dgrad: BN means without BN");
  if (N == 0 || H == 0 || W == 0) return YG_OK;
  const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
  const int tiles_h = cdiv(Ho, FD_OH), tiles_w = cdiv(Wo, FD_OW);
  const long long nblk = (long long)N * tiles_h * tiles_w;
  YG_CHECK_ARG(nblk < (1LL << 31), "conv_first_dgrad: image too large");
  cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(T, S) first_dgrad_kernel<T, S><<<(unsigned)nblk, FD_THREADS, 0, st>>>(x, w, (const T*)da, dx, H, W, Cin, Ho, Wo, \
                                                   Cout, be, fwd_shift, bn_dy_mean, bn_dyx_mean, tiles_h, tiles_w)
  if (dtype == YG_BF16) { if (stride == 2) LAUNCH(bf16, 2); else LAUNCH(bf16, 1); }
  else { if (stride == 2) LAUNCH(float, 2); else LAUNCH(float, 1); }
#undef LAUNCH
  YG_LAUNCH_CHECK("conv_first_dgrad");
  return YG_OK;
}

extern "C" int yg_conv_first_bn_means(const float* P, const float* Sg, const float* w, const float* bias, const float* mean,
                                      const float* invstd, double count, int Cout, float* dy_mean, float* dyx_mean,
                                      void* stream) {
  YG_CHECK_ARG(P && Sg && w && mean && invstd && dy_mean && dyx_mean && Cout > 0 && count > 0,
               "conv_first_bn_means: bad arguments");
  first_bn_means_kernel<<<cdiv(Cout, 64), 64, 0, (cudaStream_t)stream>>>(P, Sg, w, bias, mean, invstd, count, Cout, dy_mean,
                                                                        dyx_mean);
  YG_LAUNCH_CHECK("first_bn_means");
  return YG_OK;
}
