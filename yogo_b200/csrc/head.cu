// The 1x1 prediction head fused with YOGO.forward's output transform, and its backward.
// Replaces nn.Conv2d(C4, 5+num_classes, 1) (/root/reference/yogo/model_defns.py:67) and the
// ~12 elementwise kernels + torch.cat of /root/reference/yogo/model.py:277-313.
// HBM-bound (K = Cin, N = 5+C = 12): reads the NHWC feature map once, writes the fp32 NCHW
// prediction tensor once.
#include "common.cuh"

namespace yg {

constexpr int HD_PX = 128;   // pixels per block
constexpr int HD_KC = 32;    // input channels per smem chunk

template <typename T, int DMAX>
__global__ void __launch_bounds__(HD_PX) head_fwd_kernel(
    const T* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
    float* __restrict__ out, float* __restrict__ t_raw, long long npix, int Sy, int Sx, int Cin, int D,
    float anchor_w, float anchor_h, float wmul, float hmul, int inference,
    const float* __restrict__ cxs, const float* __restrict__ cys) {
  extern __shared__ float smem[];
  float* wsm = smem;                       // [D][Cin]
  float* xs = smem + (size_t)D * Cin;      // [HD_KC][HD_PX + 1]
  for (int i = threadIdx.x; i < D * Cin; i += HD_PX) wsm[i] = w[i];
  const long long p0 = (long long)blockIdx.x * HD_PX;
  const long long p = p0 + threadIdx.x;
  float acc[DMAX];
#pragma unroll
  for (int d = 0; d < DMAX; ++d) acc[d] = (d < D && bias) ? bias[d] : 0.f;
  for (int c0 = 0; c0 < Cin; c0 += HD_KC) {
    __syncthreads();
    for (int i = threadIdx.x; i < HD_PX * HD_KC; i += HD_PX) {
      const int c = i % HD_KC, pp = i / HD_KC;
      const long long q = p0 + pp;
      float v = 0.f;
      if (q < npix && c0 + c < Cin) v = to_f<T>(x[q * Cin + c0 + c]);
      xs[c * (HD_PX + 1) + pp] = v;
    }
    __syncthreads();
    const int kc = min(HD_KC, Cin - c0);
    for (int c = 0; c < kc; ++c) {
      const float xv = xs[c * (HD_PX + 1) + threadIdx.x];
#pragma unroll
      for (int d = 0; d < DMAX; ++d)
        if (d < D) acc[d] += xv * wsm[d * Cin + c0 + c];
    }
  }
  if (p >= npix) return;
  const int SS = Sy * Sx;
  const int n = (int)(p / SS), cell = (int)(p % SS);
  const int j = cell / Sx, i = cell % Sx;
  if (t_raw) {
#pragma unroll
    for (int d = 0; d < DMAX; ++d)
      if (d < D) t_raw[p * D + d] = acc[d];
  }
  float* o = out + (long long)n * D * SS + cell;
  // model.py:295-313.  _Cxs[j,i] = linspace(0, 1-1/Sx, Sx)[i] (model.py:48)
  // the _Cxs/_Cys buffers of the module are used when given (they are part of the state_dict)
  const float cx = cxs ? cxs[cell] : (Sx > 1 ? (float)i * ((1.f - 1.f / (float)Sx) / (float)(Sx - 1)) : 0.f);
  const float cy = cys ? cys[cell] : (Sy > 1 ? (float)j * ((1.f - 1.f / (float)Sy) / (float)(Sy - 1)) : 0.f);
  o[0] = (1.f / (float)Sx) * sigmoidf_(acc[0]) + cx;
  o[(long long)SS] = (1.f / (float)Sy) * sigmoidf_(acc[1]) + cy;
  o[2LL * SS] = anchor_w * expf(fminf(acc[2], 80.f)) * wmul;
  o[3LL * SS] = anchor_h * expf(fminf(acc[3], 80.f)) * hmul;
  o[4LL * SS] = sigmoidf_(acc[4]);
  if (inference) {
    float mx = -INFINITY;
#pragma unroll
    for (int d = 5; d < DMAX; ++d)
      if (d < D) mx = fmaxf(mx, acc[d]);
    float se = 0.f;
#pragma unroll
    for (int d = 5; d < DMAX; ++d)
      if (d < D) { acc[d] = expf(acc[d] - mx); se += acc[d]; }
    const float inv = 1.f / se;
#pragma unroll
    for (int d = 5; d < DMAX; ++d)
      if (d < D) o[(long long)d * SS] = acc[d] * inv;
  } else {
#pragma unroll
    for (int d = 5; d < DMAX; ++d)
      if (d < D) o[(long long)d * SS] = acc[d];
  }
}

// Backward.  Persistent blocks loop over 128-pixel tiles:
//   dt[p][d] from dpred and the raw logits (model.py:287-313 differentiated);
//   dx[p][ci] = sum_d dt[p][d] w[d][ci]  (+ the previous block's backward epilogue);
//   dw[d][ci] += sum_p dt[p][d] x[p][ci], dbias[d] += sum_p dt[p][d]  (per-block partials).
template <typename T, int DMAX>
__global__ void __launch_bounds__(HD_PX) head_bwd_kernel(
    const float* __restrict__ dpred, const float* __restrict__ t_raw, const T* __restrict__ x,
    const float* __restrict__ w, T* __restrict__ dx, float* __restrict__ partial,
    long long npix, int Sy, int Sx, int Cin, int D, float anchor_w, float anchor_h, float wmul, float hmul,
    BwdEpi be) {
  extern __shared__ float smem[];
  float* wsm = smem;                               // [D][Cin]
  float* dts = wsm + (size_t)D * Cin;              // [HD_PX][DMAX]
  float* xs = dts + (size_t)HD_PX * DMAX;          // [HD_PX][HD_KC + 1]
  float* dwacc = xs + (size_t)HD_PX * (HD_KC + 1); // [D][Cin] + [D]
  __shared__ float ssum[HD_KC], ssq[HD_KC];
  for (int i = threadIdx.x; i < D * Cin; i += HD_PX) { wsm[i] = w[i]; dwacc[i] = 0.f; }
  if (threadIdx.x < D) dwacc[D * Cin + threadIdx.x] = 0.f;
  const int SS = Sy * Sx;
  const long long ntiles = (npix + HD_PX - 1) / HD_PX;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long p0 = tile * HD_PX;
    const long long p = p0 + threadIdx.x;
    __syncthreads();
    {
      float dt[DMAX];
#pragma unroll
      for (int d = 0; d < DMAX; ++d) dt[d] = 0.f;
      if (p < npix) {
        const int n = (int)(p / SS), cell = (int)(p % SS);
        const float* g = dpred + (long long)n * D * SS + cell;
        const float* t = t_raw + p * D;
        const float s0 = sigmoidf_(t[0]), s1 = sigmoidf_(t[1]), s4 = sigmoidf_(t[4]);
        dt[0] = g[0] * (1.f / (float)Sx) * s0 * (1.f - s0);
        dt[1] = g[(long long)SS] * (1.f / (float)Sy) * s1 * (1.f - s1);
        // clamp(max=80) passes gradient where t <= 80
        dt[2] = t[2] <= 80.f ? g[2LL * SS] * anchor_w * expf(t[2]) * wmul : 0.f;
        dt[3] = t[3] <= 80.f ? g[3LL * SS] * anchor_h * expf(t[3]) * hmul : 0.f;
        dt[4] = g[4LL * SS] * s4 * (1.f - s4);
#pragma unroll
        for (int d = 5; d < DMAX; ++d)
          if (d < D) dt[d] = g[(long long)d * SS];
      }
#pragma unroll
      for (int d = 0; d < DMAX; ++d) dts[threadIdx.x * DMAX + d] = dt[d];
    }
    __syncthreads();
    if (threadIdx.x < D) {  // bias gradient
      float s = 0.f;
      for (int pp = 0; pp < HD_PX; ++pp) s += dts[pp * DMAX + threadIdx.x];
      dwacc[D * Cin + threadIdx.x] += s;
    }
    for (int c0 = 0; c0 < Cin; c0 += HD_KC) {
      const int kc = min(HD_KC, Cin - c0);
      if (be.bn_sums && threadIdx.x < HD_KC) { ssum[threadIdx.x] = 0.f; ssq[threadIdx.x] = 0.f; }
      __syncthreads();
      // stage x tile and produce dx for this channel chunk (coalesced over channels)
      for (int i = threadIdx.x; i < HD_PX * HD_KC; i += HD_PX) {
        const int c = i % HD_KC, pp = i / HD_KC;
        const long long q = p0 + pp;
        float xv = 0.f;
        if (q < npix && c < kc) {
          const int ci = c0 + c;
          xv = to_f<T>(x[q * Cin + ci]);
          float g = 0.f;
#pragma unroll
          for (int d = 0; d < DMAX; ++d)
            if (d < D) g += dts[pp * DMAX + d] * wsm[d * Cin + ci];
          if (dx) {
            const int n = (int)(q / SS);
            float xhat;
            g = bwd_epi_apply<T>(be, g, q * Cin + ci, n, ci, Cin, xhat);
            if (be.bn_sums) {
              g = to_f<T>(from_f<T>(g));
              atomicAdd(&ssum[c], g);
              atomicAdd(&ssq[c], g * xhat);
            }
            dx[q * Cin + ci] = from_f<T>(g);
          }
        }
        xs[pp * (HD_KC + 1) + c] = xv;
      }
      __syncthreads();
      if (be.bn_sums && threadIdx.x < kc) {
        atomicAdd(&be.bn_sums[c0 + threadIdx.x], (double)ssum[threadIdx.x]);
        atomicAdd(&be.bn_sums[Cin + c0 + threadIdx.x], (double)ssq[threadIdx.x]);
      }
      // dw[d][c0 + c]: D*kc outputs over 128 threads
      for (int o = threadIdx.x; o < D * kc; o += HD_PX) {
        const int c = o % kc, d = o / kc;
        float s = 0.f;
#pragma unroll 8
        for (int pp = 0; pp < HD_PX; ++pp) s += dts[pp * DMAX + d] * xs[pp * (HD_KC + 1) + c];
        dwacc[d * Cin + c0 + c] += s;
      }
    }
  }
  __syncthreads();
  float* base = partial + (long long)blockIdx.x * ((long long)D * Cin + D);
  for (int i = threadIdx.x; i < D * Cin + D; i += HD_PX) base[i] = dwacc[i];
}


// Faster backward for the common case (Cin = 32*CPL, D <= 16): one warp per run of 32 pixels.
//   phase A (lane = pixel): dt[d] from dpred planes (coalesced) and the raw logits -> warp-private smem
//   phase B (lane = CPL consecutive channels, loop over the 32 pixels): dx = dt.W with the fused backward
//            epilogue, dw / BN sums accumulate in registers for the whole kernel (one block reduction at
//            the end), 8-byte (CPL = 4) coalesced loads and stores.
template <typename T, int CPL>
__global__ void __launch_bounds__(256) head_bwd_warp_kernel(
    const float* __restrict__ dpred, const float* __restrict__ t_raw, const T* __restrict__ x,
    const float* __restrict__ w, T* __restrict__ dx, float* __restrict__ partial,
    long long npix, int Sy, int Sx, int Cin, int D, float anchor_w, float anchor_h, float wmul, float hmul,
    BwdEpi be) {
  constexpr int DM = 16;
  extern __shared__ float smem[];
  float* wsm = smem;                         // [D][Cin]
  float* dwacc = wsm + (size_t)D * Cin;      // [D][Cin] + [D]
  float* dts_all = dwacc + (size_t)D * Cin + DM;  // [8 warps][32][DM]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* dts = dts_all + (size_t)warp * 32 * DM;
  for (int i = threadIdx.x; i < D * Cin; i += 256) { wsm[i] = w[i]; dwacc[i] = 0.f; }
  if (threadIdx.x < DM) dwacc[D * Cin + threadIdx.x] = 0.f;
  __syncthreads();
  const int SS = Sy * Sx;
  const int c0 = lane * CPL;
  float acc[DM][CPL];
#pragma unroll
  for (int d = 0; d < DM; ++d)
#pragma unroll
    for (int k = 0; k < CPL; ++k) acc[d][k] = 0.f;
  float db[DM];
#pragma unroll
  for (int d = 0; d < DM; ++d) db[d] = 0.f;
  float bsum[CPL], bsx[CPL], k_scale[CPL], k_shift[CPL], k_mean[CPL], k_istd[CPL];
#pragma unroll
  for (int k = 0; k < CPL; ++k) {
    bsum[k] = 0.f; bsx[k] = 0.f;
    k_scale[k] = be.bn_scale ? be.bn_scale[c0 + k] : 1.f;
    k_shift[k] = be.bn_scale ? be.bn_shift[c0 + k] : 0.f;
    k_mean[k] = be.bn_scale ? be.bn_mean[c0 + k] : 0.f;
    k_istd[k] = be.bn_scale ? be.bn_invstd[c0 + k] : 0.f;
  }
  const long long nruns = (npix + 31) / 32;
  const long long gw = (long long)blockIdx.x * 8 + warp, nw = (long long)gridDim.x * 8;
  for (long long run = gw; run < nruns; run += nw) {
    const long long p0 = run * 32;
    {  // phase A
      const long long p = p0 + lane;
      float dt[DM];
#pragma unroll
      for (int d = 0; d < DM; ++d) dt[d] = 0.f;
      if (p < npix) {
        const int n = (int)(p / SS), cell = (int)(p % SS);
        const float* g = dpred + (long long)n * D * SS + cell;
        const float* t = t_raw + p * D;
        const float t0 = t[0], t1 = t[1], t2 = t[2], t3 = t[3], t4 = t[4];
        const float s0 = sigmoidf_(t0), s1 = sigmoidf_(t1), s4 = sigmoidf_(t4);
        dt[0] = g[0] * (1.f / (float)Sx) * s0 * (1.f - s0);
        dt[1] = g[(long long)SS] * (1.f / (float)Sy) * s1 * (1.f - s1);
        dt[2] = t2 <= 80.f ? g[2LL * SS] * anchor_w * expf(t2) * wmul : 0.f;
        dt[3] = t3 <= 80.f ? g[3LL * SS] * anchor_h * expf(t3) * hmul : 0.f;
        dt[4] = g[4LL * SS] * s4 * (1.f - s4);
#pragma unroll
        for (int d = 5; d < DM; ++d)
          if (d < D) dt[d] = g[(long long)d * SS];
      }
#pragma unroll
      for (int d = 0; d < DM; ++d) { dts[lane * DM + d] = dt[d]; db[d] += dt[d]; }
    }
    __syncwarp();
    const int npx = (int)min((long long)32, npix - p0);
    for (int pp = 0; pp < npx; ++pp) {
      const long long q = p0 + pp;
      const int n = (int)(q / SS);
      float xv[CPL], g[CPL], sv[CPL];
      {
        __align__(16) T tmp[CPL];
        if (CPL * sizeof(T) == 8) *reinterpret_cast<uint2*>(tmp) = *reinterpret_cast<const uint2*>(x + q * Cin + c0);
        else if (CPL * sizeof(T) == 16) *reinterpret_cast<uint4*>(tmp) = *reinterpret_cast<const uint4*>(x + q * Cin + c0);
        else {
#pragma unroll
          for (int k = 0; k < CPL; ++k) tmp[k] = x[q * Cin + c0 + k];
        }
#pragma unroll
        for (int k = 0; k < CPL; ++k) { xv[k] = to_f<T>(tmp[k]); g[k] = 0.f; sv[k] = 0.f; }
        if (be.saved) {
          const T* sp = (const T*)be.saved + q * Cin + c0;
          if (CPL * sizeof(T) == 8) *reinterpret_cast<uint2*>(tmp) = *reinterpret_cast<const uint2*>(sp);
          else if (CPL * sizeof(T) == 16) *reinterpret_cast<uint4*>(tmp) = *reinterpret_cast<const uint4*>(sp);
          else {
#pragma unroll
            for (int k = 0; k < CPL; ++k) tmp[k] = sp[k];
          }
#pragma unroll
          for (int k = 0; k < CPL; ++k) sv[k] = to_f<T>(tmp[k]);
        }
      }
#pragma unroll
      for (int d = 0; d < DM; ++d) {
        if (d < D) {
          const float dtd = dts[pp * DM + d];
#pragma unroll
          for (int k = 0; k < CPL; ++k) {
            g[k] += dtd * wsm[d * Cin + c0 + k];
            acc[d][k] += dtd * xv[k];
          }
        }
      }
      if (dx) {
        __align__(16) T ob[CPL];
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          float gg = g[k];
          if (be.dropscale) gg *= be.dropscale[(long long)n * Cin + c0 + k];
          float xhat = 0.f;
          if (be.saved) {
            float pre = sv[k];
            if (be.bn_scale) { pre = sv[k] * k_scale[k] + k_shift[k]; xhat = (sv[k] - k_mean[k]) * k_istd[k]; }
            gg *= act_grad(pre, be.act);
          }
          if (be.bn_sums) gg = to_f<T>(from_f<T>(gg));
          bsum[k] += gg; bsx[k] += gg * xhat;
          ob[k] = from_f<T>(gg);
        }
        if (CPL * sizeof(T) == 8) *reinterpret_cast<uint2*>(dx + q * Cin + c0) = *reinterpret_cast<uint2*>(ob);
        else if (CPL * sizeof(T) == 16) *reinterpret_cast<uint4*>(dx + q * Cin + c0) = *reinterpret_cast<uint4*>(ob);
        else {
#pragma unroll
          for (int k = 0; k < CPL; ++k) dx[q * Cin + c0 + k] = ob[k];
        }
      }
    }
    __syncwarp();
  }
  // block reduction: lanes own distinct channels, the 8 warps share them
#pragma unroll
  for (int d = 0; d < DM; ++d) {
    if (d < D) {
#pragma unroll
      for (int k = 0; k < CPL; ++k) atomicAdd(&dwacc[d * Cin + c0 + k], acc[d][k]);
      const float s = warp_sum(db[d]);
      if (lane == 0) atomicAdd(&dwacc[D * Cin + d], s);
    }
  }
  float* bn_s = dts_all + 8 * 32 * DM;  // [2][Cin], zeroed below before use
  __syncthreads();
  if (be.bn_sums) {
    for (int i = threadIdx.x; i < 2 * Cin; i += 256) bn_s[i] = 0.f;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      atomicAdd(&bn_s[c0 + k], bsum[k]);
      atomicAdd(&bn_s[Cin + c0 + k], bsx[k]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * Cin; i += 256) atomicAdd(&be.bn_sums[i], (double)bn_s[i]);
  }
  float* base = partial + (long long)blockIdx.x * ((long long)D * Cin + D);
  for (int i = threadIdx.x; i < D * Cin + D; i += 256) base[i] = dwacc[i];
}

__global__ void head_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw,
                                   float* __restrict__ dbias, long long nw, int D, int slices, float clip) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nw + D) return;
  float s = 0.f;
  for (int k = 0; k < slices; ++k) s += partial[k * (nw + D) + i];
  s = clampf(s, clip);
  if (i < nw) dw[i] = s;
  else if (dbias) dbias[i - nw] = s;
}

// sum over the per-block partials [slices][D] of one element per warp (lanes stride over the slices)
__global__ void head_bias_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dbias, int D, int slices, float clip) {
  const int d = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (d >= D) return;
  float s = 0.f;
  for (int k = lane; k < slices; k += 32) s += partial[(long long)k * D + d];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) dbias[d] = clampf(s, clip);
}

constexpr int HD_BWD_BLOCKS = 296;
constexpr int HD_DP = 32;          // channels of the padded bf16 logit-gradient tensor fed to the tensor cores
constexpr int HD_DT_BLOCKS = 592;

// conv_tc.cu
bool head_bwd_tc_supported(int Cin, int D);
bool head_fwd_tc_supported(int Cin, int D);
int head_fwd_tc(const void* x, const float* w, const float* bias, float* out, float* t_raw, int N, int Sy, int Sx, int Cin,
                int D, float aw, float ah, float wm, float hm, int inference, const float* cxs, const float* cys,
                cudaStream_t st);
size_t head_bwd_tc_workspace(int Cin);
int head_bwd_tc(const void* dt, const void* x, const float* w, void* dx, float* dw, int N, int Sy, int Sx, int Cin, int D,
                const BwdEpi& be, float clip, void* ws, size_t ws_bytes, cudaStream_t st);

// dt[p][0..32) (bf16, zero padded) = d(loss)/d(raw logits) from dpred and the raw logits; per-block bias partials
__global__ void __launch_bounds__(256) head_dt_kernel(const float* __restrict__ dpred, const float* __restrict__ t_raw,
                                                      bf16* __restrict__ dt, float* __restrict__ db_partial,
                                                      long long npix, int Sy, int Sx, int D, float anchor_w,
                                                      float anchor_h, float wmul, float hmul) {
  __shared__ float sdb[HD_DP];
  if (threadIdx.x < HD_DP) sdb[threadIdx.x] = 0.f;
  __syncthreads();
  const int SS = Sy * Sx;
  float db[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) db[d] = 0.f;
  float db_hi[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) db_hi[d] = 0.f;
  for (long long p = (long long)blockIdx.x * 256 + threadIdx.x; p < npix; p += (long long)gridDim.x * 256) {
    const int n = (int)(p / SS), cell = (int)(p % SS);
    const float* g = dpred + (long long)n * D * SS + cell;
    const float* t = t_raw + p * D;
    float v[HD_DP];
#pragma unroll
    for (int d = 0; d < HD_DP; ++d) v[d] = 0.f;
    const float t0 = t[0], t1 = t[1], t2 = t[2], t3 = t[3], t4 = t[4];
    const float s0 = sigmoidf_(t0), s1 = sigmoidf_(t1), s4 = sigmoidf_(t4);
    v[0] = g[0] * (1.f / (float)Sx) * s0 * (1.f - s0);
    v[1] = g[(long long)SS] * (1.f / (float)Sy) * s1 * (1.f - s1);
    v[2] = t2 <= 80.f ? g[2LL * SS] * anchor_w * expf(t2) * wmul : 0.f;
    v[3] = t3 <= 80.f ? g[3LL * SS] * anchor_h * expf(t3) * hmul : 0.f;
    v[4] = g[4LL * SS] * s4 * (1.f - s4);
#pragma unroll
    for (int d = 5; d < HD_DP; ++d)
      if (d < D) v[d] = g[(long long)d * SS];
    __align__(16) bf16 ob[HD_DP];
#pragma unroll
    for (int d = 0; d < HD_DP; ++d) ob[d] = __float2bfloat16_rn(v[d]);
    // the 64-byte row of this pixel as two 32-byte stores (full sectors)
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const uint4 lo = reinterpret_cast<uint4*>(ob)[2 * i], hi = reinterpret_cast<uint4*>(ob)[2 * i + 1];
      asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dt + p * HD_DP + 16 * i), "r"(lo.x), "r"(lo.y),
                   "r"(lo.z), "r"(lo.w), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w) : "memory");
    }
#pragma unroll
    for (int d = 0; d < 16; ++d) { db[d] += v[d]; db_hi[d] += v[16 + d]; }
  }
#pragma unroll
  for (int d = 0; d < 16; ++d) {
    const float a = warp_sum(db[d]);
    const float b = (D > 16) ? warp_sum(db_hi[d]) : 0.f;
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sdb[d], a); if (D > 16) atomicAdd(&sdb[16 + d], b); }
  }
  __syncthreads();
  if (threadIdx.x < D) db_partial[(long long)blockIdx.x * D + threadIdx.x] = sdb[threadIdx.x];
}

// Softmax backward of the inference head: the class planes of dpred (d loss / d softmax output) become d loss / d logits,
// p * (dp - sum_j p_j dp_j), with p recomputed from the raw logits exactly as head_fwd_kernel computes it; planes 0-4 are
// copied.  One thread per grid cell.
template <int DMAX>
__global__ void __launch_bounds__(256) head_softmax_bwd_kernel(const float* __restrict__ dpred, const float* __restrict__ t_raw,
                                                               float* __restrict__ out, long long npix, int SS, int D) {
  const long long p = (long long)blockIdx.x * 256 + threadIdx.x;
  if (p >= npix) return;
  const int n = (int)(p / SS), cell = (int)(p % SS);
  const float* g = dpred + (long long)n * D * SS + cell;
  float* o = out + (long long)n * D * SS + cell;
  const float* t = t_raw + p * D;
#pragma unroll
  for (int d = 0; d < 5; ++d) o[(long long)d * SS] = g[(long long)d * SS];
  float e[DMAX];
  float mx = -INFINITY;
#pragma unroll
  for (int d = 5; d < DMAX; ++d)
    if (d < D) { e[d] = t[d]; mx = fmaxf(mx, e[d]); }
  float se = 0.f;
#pragma unroll
  for (int d = 5; d < DMAX; ++d)
    if (d < D) { e[d] = expf(e[d] - mx); se += e[d]; }
  const float inv = 1.f / se;
  float dot = 0.f;
#pragma unroll
  for (int d = 5; d < DMAX; ++d)
    if (d < D) { e[d] *= inv; dot += e[d] * g[(long long)d * SS]; }
#pragma unroll
  for (int d = 5; d < DMAX; ++d)
    if (d < D) o[(long long)d * SS] = e[d] * (g[(long long)d * SS] - dot);
}

}  // namespace yg
using namespace yg;

extern "C" int yg_head_fwd(const void* x, int dtype, const float* w, const float* bias, float* out, float* t_raw,
                           int N, int Sy, int Sx, int Cin, int num_classes,
                           float anchor_w, float anchor_h, float width_mult, float height_mult,
                           int inference, const float* cxs, const float* cys, void* stream) {
  const int D = 5 + num_classes;
  YG_CHECK_ARG(x && w && out, "head_fwd: null pointer");
  YG_CHECK_ARG(num_classes >= 1 && D <= 32, "head_fwd: 5+num_classes must be <= 32, got %d", D);
  YG_CHECK_ARG(dtype == YG_F32 || dtype == YG_BF16, "head_fwd: dtype %d", dtype);
  const long long npix = (long long)N * Sy * Sx;
  if (npix == 0) return YG_OK;
  if (dtype == YG_BF16 && yg_get_conv_impl() != YG_IMPL_SIMT && head_fwd_tc_supported(Cin, D))
    return head_fwd_tc(x, w, bias, out, t_raw, N, Sy, Sx, Cin, D, anchor_w, anchor_h, width_mult, height_mult, inference,
                       cxs, cys, (cudaStream_t)stream);
  const size_t smem = ((size_t)D * Cin + (size_t)HD_KC * (HD_PX + 1)) * sizeof(float);
  YG_CHECK_ARG(smem <= 200 * 1024, "head_fwd: Cin %d too large", Cin);
  const int blocks = cdiv(npix, HD_PX);
  cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(T, DM)                                                                                        \
  do {                                                                                                       \
    YG_CUDA(cudaFuncSetAttribute(head_fwd_kernel<T, DM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    head_fwd_kernel<T, DM><<<blocks, HD_PX, smem, st>>>((const T*)x, w, bias, out, t_raw, npix, Sy, Sx, Cin, D, \
                                                         anchor_w, anchor_h, width_mult, height_mult, inference, cxs, cys); \
  } while (0)
  if (dtype == YG_BF16) { if (D <= 16) LAUNCH(bf16, 16); else LAUNCH(bf16, 32); }
  else { if (D <= 16) LAUNCH(float, 16); else LAUNCH(float, 32); }
#undef LAUNCH
  YG_LAUNCH_CHECK("head_fwd");
  return YG_OK;
}

static size_t head_tc_offsets(int N, int Sy, int Sx, int Cin, int D, size_t* off_db, size_t* off_wg) {
  const size_t npix = (size_t)N * Sy * Sx;
  size_t o = npix * HD_DP * sizeof(bf16);
  o = (o + 255) & ~(size_t)255;
  *off_db = o;
  o += (size_t)HD_DT_BLOCKS * D * sizeof(float);
  o = (o + 255) & ~(size_t)255;
  *off_wg = o;
  return o + head_bwd_tc_workspace(Cin);
}

extern "C" size_t yg_head_bwd_workspace(int N, int Sy, int Sx, int Cin, int num_classes) {
  const int D = 5 + num_classes;
  size_t a = (size_t)HD_BWD_BLOCKS * ((size_t)D * Cin + D) * sizeof(float);
  if (head_bwd_tc_supported(Cin, D)) {
    size_t o1, o2;
    const size_t b = head_tc_offsets(N, Sy, Sx, Cin, D, &o1, &o2);
    if (b > a) a = b;
  }
  return a;
}

extern "C" int yg_head_bwd(const float* dpred, const float* t_raw, const void* x, const float* w, void* dx, int dtype,
                           float* dw, float* dbias, int N, int Sy, int Sx, int Cin, int num_classes,
                           float anchor_w, float anchor_h, float width_mult, float height_mult,
                           const yg_bwd_epilogue* bep, float clip, void* workspace, size_t workspace_bytes,
                           void* stream) {
  const int D = 5 + num_classes;
  YG_CHECK_ARG(dpred && t_raw && x && w, "head_bwd: null pointer");
  YG_CHECK_ARG(num_classes >= 1 && D <= 32, "head_bwd: 5+num_classes must be <= 32, got %d", D);
  const long long npix = (long long)N * Sy * Sx;
  const size_t need = yg_head_bwd_workspace(N, Sy, Sx, Cin, num_classes);
  if (!workspace || workspace_bytes < need) {
    set_error("head_bwd: workspace %zu < %zu", workspace_bytes, need);
    return YG_ERR_WORKSPACE;
  }
  BwdEpi be = make_bwd_epi(bep);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == YG_BF16 && dx && npix > 0 && yg_get_conv_impl() != YG_IMPL_SIMT && head_bwd_tc_supported(Cin, D)) {
    // tensor-core path: dt (bf16, padded) -> dgrad engine (1 tap) + wgrad engine (1 column); bias from the dt pass
    size_t off_db, off_wg;
    head_tc_offsets(N, Sy, Sx, Cin, D, &off_db, &off_wg);
    bf16* dt = (bf16*)workspace;
    float* dbp = (float*)((char*)workspace + off_db);
    int nb = (int)((npix + 255) / 256);
    if (nb > HD_DT_BLOCKS) nb = HD_DT_BLOCKS;
    head_dt_kernel<<<nb, 256, 0, st>>>(dpred, t_raw, dt, dbp, npix, Sy, Sx, D, anchor_w, anchor_h, width_mult, height_mult);
    YG_LAUNCH_CHECK("head_dt");
    if (dw && dbias) {
      head_bias_reduce_kernel<<<cdiv(D * 32, 256), 256, 0, st>>>(dbp, dbias, D, nb, clip);
      YG_LAUNCH_CHECK("head_bias_reduce");
    }
    return head_bwd_tc(dt, x, w, dx, dw, N, Sy, Sx, Cin, D, be, clip, (char*)workspace + off_wg,
                       workspace_bytes - off_wg, st);
  }
  int blocks = cdiv(npix, HD_PX);
  if (blocks > HD_BWD_BLOCKS) blocks = HD_BWD_BLOCKS;
  if (blocks < 1) blocks = 1;
  const int cpl = (Cin % 32 == 0) ? Cin / 32 : 0;
  if (D <= 16 && (cpl == 1 || cpl == 2 || cpl == 4 || cpl == 8) && npix > 0) {
    blocks = (int)((npix + 255) / 256);
    if (blocks > HD_BWD_BLOCKS) blocks = HD_BWD_BLOCKS;
    const size_t smemw = ((size_t)D * Cin * 2 + 16 + 8 * 32 * 16 + 2 * (size_t)Cin) * sizeof(float);
#define LAUNCHW(T, CPLV)                                                                                          \
  do {                                                                                                            \
    YG_CUDA(cudaFuncSetAttribute(head_bwd_warp_kernel<T, CPLV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemw)); \
    head_bwd_warp_kernel<T, CPLV><<<blocks, 256, smemw, st>>>(dpred, t_raw, (const T*)x, w, (T*)dx, (float*)workspace,     \
                                                              npix, Sy, Sx, Cin, D, anchor_w, anchor_h, width_mult,        \
                                                              height_mult, be);                                            \
  } while (0)
#define LAUNCHW_T(CPLV) do { if (dtype == YG_BF16) LAUNCHW(bf16, CPLV); else LAUNCHW(float, CPLV); } while (0)
    if (cpl == 1) LAUNCHW_T(1); else if (cpl == 2) LAUNCHW_T(2); else if (cpl == 4) LAUNCHW_T(4); else LAUNCHW_T(8);
#undef LAUNCHW_T
#undef LAUNCHW
    YG_LAUNCH_CHECK("head_bwd_warp");
    if (!dw) return YG_OK;
    const long long nw2 = (long long)D * Cin;
    head_reduce_kernel<<<cdiv(nw2 + D, 256), 256, 0, st>>>((const float*)workspace, dw, dbias, nw2, D, blocks, clip);
    YG_LAUNCH_CHECK("head_reduce");
    return YG_OK;
  }
  const int DM = D <= 16 ? 16 : 32;
  const size_t smem = ((size_t)D * Cin * 2 + D + (size_t)HD_PX * DM + (size_t)HD_PX * (HD_KC + 1)) * sizeof(float);
  YG_CHECK_ARG(smem <= 200 * 1024, "head_bwd: Cin %d too large", Cin);
#define LAUNCH(T, DMX)                                                                                        \
  do {                                                                                                        \
    YG_CUDA(cudaFuncSetAttribute(head_bwd_kernel<T, DMX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    head_bwd_kernel<T, DMX><<<blocks, HD_PX, smem, st>>>(dpred, t_raw, (const T*)x, w, (T*)dx, (float*)workspace, \
                                                          npix, Sy, Sx, Cin, D, anchor_w, anchor_h, width_mult,  \
                                                          height_mult, be);                                      \
  } while (0)
  if (dtype == YG_BF16) { if (DM == 16) LAUNCH(bf16, 16); else LAUNCH(bf16, 32); }
  else { if (DM == 16) LAUNCH(float, 16); else LAUNCH(float, 32); }
#undef LAUNCH
  YG_LAUNCH_CHECK("head_bwd");
  if (!dw) return YG_OK;
  const long long nw = (long long)D * Cin;
  head_reduce_kernel<<<cdiv(nw + D, 256), 256, 0, st>>>((const float*)workspace, dw, dbias, nw, D, blocks, clip);
  YG_LAUNCH_CHECK("head_reduce");
  return YG_OK;
}

extern "C" int yg_head_softmax_bwd(const float* dpred, const float* t_raw, float* out, int N, int Sy, int Sx, int num_classes,
                                   void* stream) {
  const int D = 5 + num_classes;
  YG_CHECK_ARG(dpred && t_raw && out, "head_softmax_bwd: null pointer");
  YG_CHECK_ARG(num_classes >= 1 && D <= 32, "head_softmax_bwd: 5+num_classes must be <= 32, got %d", D);
  const long long npix = (long long)N * Sy * Sx;
  if (npix == 0) return YG_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (D <= 16) head_softmax_bwd_kernel<16><<<cdiv(npix, 256), 256, 0, st>>>(dpred, t_raw, out, npix, Sy * Sx, D);
  else head_softmax_bwd_kernel<32><<<cdiv(npix, 256), 256, 0, st>>>(dpred, t_raw, out, npix, Sy * Sx, D);
  YG_LAUNCH_CHECK("head_softmax_bwd");
  return YG_OK;
}
