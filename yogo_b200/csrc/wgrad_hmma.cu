// Weight gradient of the 16 -> 32 channel stride-1 3x3 convolution on the warp-level tensor cores.  Replaces cuDNN wgrad
// for base_model layer 2 (/root/reference/yogo/model_defns.py:39-47).  (The 32 -> 64 stride-2 layer 3 is faster on the
// tcgen05 wgrad: this kernel is bound there by the mma.sync rate, 0.55 vs 0.47 ms.)
//
// The tcgen05 wgrad needs M = 128: with 32 or 64 output channels it runs W-folded (4x / 2x structurally-zero MACs) and its
// three filter-column units re-read every tile, which makes it L2-bandwidth bound (0.5 ms for 1.2 GB of tensors).  Here:
//   dW[co][ci][r][s] = sum_px dz[px][co] * x[px*stride + (r-1, s-1)][ci]       D[M = co][N = (tap, ci)] += A[co][px] B[px][(tap,ci)]
//   * one TMA box of dz (TH x 32 pixels) and one halo box of x per tile and stage (OOB zero fill = padding and ragged edges),
//     hardware swizzle matching the row size so that ldmatrix is conflict free;
//   * ldmatrix.trans turns the pixel-major rows straight into mma.m16n8k16 fragments; the im2col of B is nothing but the row
//     ADDRESS each lane hands to ldmatrix (pixel + tap offset, pixel stride 2 for stride-2 convolutions);
//   * a warp = (block of 32 output channels, filter row r): 3 taps x CI/8 column tiles x 2 row tiles of accumulators stay in
//     registers for the whole kernel; per-block partials are summed by a second kernel in a fixed order (deterministic);
//   * d(bias) = row sums of the A fragments (filter-row-1 warps).
// HBM-bound by construction: every tensor element is read once from DRAM, ~4-13 warp instructions per pixel.
#include "common.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <mutex>

namespace yg {

namespace {

PFN_cuTensorMapEncodeTiled_v12000 h_encode = nullptr;
std::once_flag h_encode_once;
int* h_error_flag = nullptr;

bool h_get_encode() {
  std::call_once(h_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      h_encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
  });
  return h_encode != nullptr;
}

int h_make_map(CUtensorMap* m, const void* base, int C, int W, int H, int N, int boxw, int boxh) {
  uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)N};
  uint64_t str[3] = {(uint64_t)C * 2, (uint64_t)W * C * 2, (uint64_t)H * W * C * 2};
  uint32_t box[4] = {(uint32_t)C, (uint32_t)boxw, (uint32_t)boxh, 1};
  uint32_t estr[4] = {1, 1, 1, 1};
  const CUtensorMapSwizzle sw = C == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (C == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  CUresult r = h_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, str, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("wgrad_hmma: cuTensorMapEncodeTiled failed with %d", (int)r); return YG_ERR_CUDA; }
  return YG_OK;
}

__device__ __forceinline__ uint32_t sm32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void hb_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sm32(bar)), "r"(count));
}
__device__ __forceinline__ void hb_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sm32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void hb_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(sm32(bar)) : "memory");
}
__device__ __forceinline__ void hb_wait(uint64_t* bar, uint32_t parity, int* error_flag, int code) {
  uint32_t spins = 0;
  for (;;) {
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(sm32(bar)), "r"(parity) : "memory");
    if (ok) return;
    if (++spins > (1u << 24)) {   // bounded: trap instead of hanging the GPU
      if (error_flag) atomicExch(error_flag, code);
      __trap();
    }
  }
}
__device__ __forceinline__ void h_tma_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(sm32(dst)), "l"(map), "r"(sm32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void h_ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void h_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

struct HwMaps { CUtensorMap dz, x; };
struct HwParams {
  int N, tiles_h, tiles_w, total_tiles;
  int nstages, stage_bytes, dz_bytes, x_bytes;
  float* partial;      // [grid][CO*CI*9 + CO]
  int* error_flag;
};

constexpr int HW_TW = 32;   // output pixels per tile row (two 16-pixel strips)

// byte offset of (pixel row p, 16-byte chunk c) inside a TMA-written tile whose rows are ROWB bytes (hardware swizzle modes)
template <int ROWB>
__device__ __forceinline__ uint32_t sw_off(int p, int c) {
  if (ROWB == 32) return (uint32_t)(p * 32 + ((c ^ ((p >> 2) & 1)) << 4));
  if (ROWB == 64) return (uint32_t)(p * 64 + ((c ^ ((p >> 1) & 3)) << 4));
  return (uint32_t)(p * 128 + ((c ^ (p & 7)) << 4));
}

template <int CI, int CO, int STRIDE>
__global__ void __launch_bounds__(((CO / 32) * 3 + 1) * 32, CO == 32 ? 4 : 2) wgrad_hmma_kernel(const __grid_constant__ HwMaps maps,
                                                                              const __grid_constant__ HwParams p) {
  constexpr int TH = STRIDE == 1 ? 8 : 4;                         // output rows per tile
  constexpr int XW = (HW_TW - 1) * STRIDE + 3, XH = (TH - 1) * STRIDE + 3;
  constexpr int ROLES = (CO / 32) * 3;
  constexpr int NT = CI / 8;                                      // 8-column tiles of B per tap
  extern __shared__ __align__(1024) unsigned char hsm_raw[];
  unsigned char* smem = hsm_raw + ((1024u - (sm32(hsm_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.nstages * p.stage_bytes);
  uint64_t* empty_bar = full_bar + 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < p.nstages; ++i) { hb_init(&full_bar[i], 1); hb_init(&empty_bar[i], ROLES); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  if (warp == ROLES) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        int t = tile;
        const int tw = t % p.tiles_w; t /= p.tiles_w;
        const int th = t % p.tiles_h;
        const int n = t / p.tiles_h;
        hb_wait(&empty_bar[stage], phase ^ 1u, p.error_flag, 21);
        unsigned char* sd = smem + (size_t)stage * p.stage_bytes;
        hb_expect_tx(&full_bar[stage], (uint32_t)(TH * HW_TW * CO * 2 + XH * XW * CI * 2));
        h_tma_4d(sd, &maps.dz, &full_bar[stage], 0, tw * HW_TW, th * TH, n);
        h_tma_4d(sd + p.dz_bytes, &maps.x, &full_bar[stage], 0, tw * HW_TW * STRIDE - 1, th * TH * STRIDE - 1, n);
        if (++stage == p.nstages) { stage = 0; phase ^= 1u; }
      }
    }
    return;
  }
  // -------------------------------------------------------------------- MMA warps: (32-channel block mb, filter row r)
  const int mb = warp / 3, r = warp % 3;
  const int g = lane >> 2, j = lane & 3;
  const int lm = lane >> 3, lr = lane & 7;
  float acc[2][3][NT][4];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int s = 0; s < 3; ++s)
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[a][s][nt][e] = 0.f;
  float bsum[2][2] = {{0.f, 0.f}, {0.f, 0.f}};   // [m tile][row g / g+8]: d(bias) partials (r == 1 warps)
  int stage = 0;
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    hb_wait(&full_bar[stage], phase, p.error_flag, 22);
    const uint32_t dzs = sm32(smem + (size_t)stage * p.stage_bytes);
    const uint32_t xs = dzs + (uint32_t)p.dz_bytes;
#pragma unroll 1
    for (int strip = 0; strip < TH * 2; ++strip) {
      const int row = strip >> 1, col0 = (strip & 1) * 16;
      // A[m = co][k = px] from dz[px][co]: matrices (k 0-7, m 0-7), (k 0-7, m 8-15), (k 8-15, m 0-7), (k 8-15, m 8-15)
      uint32_t af[2][4];
      const int apx = row * HW_TW + col0 + (lm >> 1) * 8 + lr;
#pragma unroll
      for (int a = 0; a < 2; ++a)
        h_ldsm_x4_t(af[a], dzs + sw_off<CO * 2>(apx, (mb * 32 + a * 16) / 8 + (lm & 1)));
      if (r == 1) {
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&af[a][q]));
            bsum[a][q & 1] += f.x + f.y;
          }
      }
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        // B[k = px][n = ci] from x[px*stride + tap][ci]: matrices (k 0-7, n 0-7), (k 8-15, n 0-7), (k 0-7, n 8-15), (k 8-15, n 8-15)
        const int kpx = col0 + (lm & 1) * 8 + lr;
        const int xp = (row * STRIDE + r) * XW + kpx * STRIDE + s;
#pragma unroll
        for (int h = 0; h < NT / 2; ++h) {
          uint32_t bf[4];
          h_ldsm_x4_t(bf, xs + sw_off<CI * 2>(xp, 2 * h + (lm >> 1)));
#pragma unroll
          for (int a = 0; a < 2; ++a) {
            h_mma(acc[a][s][2 * h], af[a], bf[0], bf[1]);
            h_mma(acc[a][s][2 * h + 1], af[a], bf[2], bf[3]);
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) hb_arrive(&empty_bar[stage]);
    if (++stage == p.nstages) { stage = 0; phase ^= 1u; }
  }
  // -------------------------------------------------------------------- partials: [co][ci][r][s] then [co]
  float* base = p.partial + (size_t)blockIdx.x * (CO * CI * 9 + CO);
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int s = 0; s < 3; ++s)
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int co = mb * 32 + a * 16 + g + (e >> 1) * 8, ci = nt * 8 + 2 * j + (e & 1);
          base[((size_t)co * CI + ci) * 9 + r * 3 + s] = acc[a][s][nt][e];
        }
  if (r == 1) {
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        float v = bsum[a][e];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        if (j == 0) base[(size_t)CO * CI * 9 + mb * 32 + a * 16 + g + e * 8] = v;
      }
  }
}

__global__ void __launch_bounds__(256) wgrad_hmma_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw,
                                                                float* __restrict__ dbias, int nw, int CO, int slices, float clip) {
  // block = 32 consecutive elements x 8 warps; warp w sums slices w, w + 8, ... (coalesced 128-byte rows, four independent chains),
  // the eight partial sums are added in a fixed order.  (One thread per element walked all ~590 slices alone: 19 blocks, 46 us.)
  __shared__ float red[8][32];
  const int lane = threadIdx.x & 31, sub = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  const size_t stride = (size_t)nw + CO;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (i < nw + CO) {
    int k = sub;
    for (; k + 24 < slices; k += 32) {
      s0 += partial[(size_t)k * stride + i];
      s1 += partial[(size_t)(k + 8) * stride + i];
      s2 += partial[(size_t)(k + 16) * stride + i];
      s3 += partial[(size_t)(k + 24) * stride + i];
    }
    for (; k < slices; k += 8) s0 += partial[(size_t)k * stride + i];
  }
  red[sub][lane] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (sub == 0 && i < nw + CO) {
    float v = red[0][lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) v += red[w][lane];
    v = clampf(v, clip);
    if (i < nw) dw[i] = v;
    else if (dbias) dbias[i - nw] = v;
  }
}

constexpr int HW_GRID = 148 * 4;   // upper bound on the grid (partial buffer sizing)

template <int CI, int CO, int STRIDE>
int launch_hmma(const void* x, const void* dz, float* dw, float* dbias, int N, int H, int W, float clip, void* ws,
                cudaStream_t st) {
  constexpr int TH = STRIDE == 1 ? 8 : 4;
  constexpr int XW = (HW_TW - 1) * STRIDE + 3, XH = (TH - 1) * STRIDE + 3;
  const int Ho = (H + 2 - 3) / STRIDE + 1, Wo = (W + 2 - 3) / STRIDE + 1;
  HwMaps maps;
  HwParams p;
  memset(&maps, 0, sizeof(maps));
  memset(&p, 0, sizeof(p));
  int rc = h_make_map(&maps.dz, dz, CO, Wo, Ho, N, HW_TW, TH);
  if (rc) return rc;
  rc = h_make_map(&maps.x, x, CI, W, H, N, XW, XH);
  if (rc) return rc;
  p.N = N;
  p.tiles_h = cdiv(Ho, TH); p.tiles_w = cdiv(Wo, HW_TW);
  p.total_tiles = N * p.tiles_h * p.tiles_w;
  p.dz_bytes = (TH * HW_TW * CO * 2 + 1023) & ~1023;
  p.x_bytes = (XH * XW * CI * 2 + 1023) & ~1023;
  p.stage_bytes = p.dz_bytes + p.x_bytes;
  p.nstages = 2;
  p.partial = (float*)ws;
  if (!h_error_flag) {
    YG_CUDA(cudaMalloc(&h_error_flag, sizeof(int)));
    YG_CUDA(cudaMemset(h_error_flag, 0, sizeof(int)));
  }
  p.error_flag = h_error_flag;
  const int gmax = 148 * (CO == 32 ? 4 : 2);   // resident blocks: 4 x 55 KB or 2 x 106 KB of shared memory per SM
  const int grid = p.total_tiles < gmax ? p.total_tiles : gmax;
  const size_t smem = (size_t)p.nstages * p.stage_bytes + 1024 + 256;
  constexpr int THREADS = ((CO / 32) * 3 + 1) * 32;
  YG_CUDA(cudaFuncSetAttribute(wgrad_hmma_kernel<CI, CO, STRIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  wgrad_hmma_kernel<CI, CO, STRIDE><<<grid, THREADS, smem, st>>>(maps, p);
  YG_LAUNCH_CHECK("wgrad_hmma_kernel");
  const int nw = CO * CI * 9;
  wgrad_hmma_reduce_kernel<<<cdiv(nw + CO, 32), 256, 0, st>>>((const float*)ws, dw, dbias, nw, CO, grid, clip);
  YG_LAUNCH_CHECK("wgrad_hmma_reduce");
  return YG_OK;
}

}  // namespace

bool wgrad_hmma_supported(int dtype, int W, int Cin, int Cout, int ks, int stride) {
  if (dtype != YG_BF16 || ks != 3) return false;
  const int Wo = (W + 2 - 3) / stride + 1;
  if (Wo < 1) return false;
  return Cin == 16 && Cout == 32 && stride == 1;
}

size_t wgrad_hmma_workspace(int Cin, int Cout) { return (size_t)HW_GRID * ((size_t)Cout * Cin * 9 + Cout) * sizeof(float) + 256; }

int conv_wgrad_hmma(const void* x, const void* dz, float* dw, float* dbias, int N, int H, int W, int Cin, int Cout, int ks,
                    int stride, float clip, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (!h_get_encode()) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return YG_ERR_CUDA; }
  const size_t need = wgrad_hmma_workspace(Cin, Cout);
  if (!ws || ws_bytes < need) { set_error("conv_wgrad_hmma: workspace %zu < %zu", ws_bytes, need); return YG_ERR_WORKSPACE; }
  (void)ks;
  if (Cin == 16 && Cout == 32 && stride == 1) return launch_hmma<16, 32, 1>(x, dz, dw, dbias, N, H, W, clip, ws, st);
  set_error("conv_wgrad_hmma: unsupported shape");
  return YG_ERR_INVALID;
}

}  // namespace yg
