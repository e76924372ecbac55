// Input side of the training step (SURVEY.md 8f N3): the bounding-box aware flips applied to every batch
// (/root/reference/yogo/data/data_transforms.py:51-98) and the rasterisation of ragged label lists into the
// (6, Sy, Sx) label tensor (/root/reference/yogo/data/yogo_dataset.py:24-46), whole batch per launch.
// HBM-bound byte/element shuffles: 8- or 16-byte accesses on both sides, nothing is re-read.
#include "common.cuh"
#include <string.h>
#include <algorithm>
#include <type_traits>

namespace yg {

// one block = FLIP_ROWS consecutive output rows, one thread = one V-element vector at a time;
// out[y][x] = in[vflip ? H-1-y : y][hflip ? W-1-x : x].  32-bit index arithmetic; the only 64-bit division is one per block.
// `Src` says where output plane p (= n * C + c) comes from and which flips apply: FlipArgs (the batch flip, plane p of the
// input, flips from the arguments) or GatherSrc (the device-resident dataset: plane of a stored image, flips from memory).
constexpr int FLIP_ROWS = 16;
struct FlipArgs {
  int hflip, vflip;
  __device__ __forceinline__ void load() {}
  __device__ __forceinline__ long long plane(long long p) const { return p; }
};
// batch `flags[2]` of an epoch's index table (row stride `stride`): output image n is stored image table[batch * stride + n]
struct GatherSrc {
  const int* table;
  const int* flags;   // [hflip, vflip, batch] written by dd_draw_kernel
  int stride, C;
  int hflip, vflip;
  long long base;
  __device__ __forceinline__ void load() {
    hflip = flags[0];
    vflip = flags[1];
    base = (long long)flags[2] * stride;
  }
  __device__ __forceinline__ long long plane(long long p) const {
    const int pi = (int)p, n = pi / C;
    return (long long)__ldg(table + base + n) * C + (pi - n * C);
  }
};
template <typename T, int V, typename Src>
__global__ void __launch_bounds__(256) flip_images_kernel(const T* __restrict__ in, T* __restrict__ out, long long rows, int H,
                                                          int W, Src src) {
  src.load();
  const int hflip = src.hflip, vflip = src.vflip;
  const int vpr = W / V;   // vectors per row
  struct alignas(sizeof(T) * V) Vec { T e[V]; };
  const long long row0 = (long long)blockIdx.x * FLIP_ROWS;
  const long long plane0 = row0 / H;
  const int y0 = (int)(row0 - plane0 * H);
  const int nrows = (int)(rows - row0 < FLIP_ROWS ? rows - row0 : FLIP_ROWS);
  for (int idx = threadIdx.x; idx < nrows * vpr; idx += blockDim.x) {
    const int r = idx / vpr, vx = idx - r * vpr;
    int y = y0 + r;
    long long plane = plane0;
    while (y >= H) { y -= H; ++plane; }
    const int sy = vflip ? H - 1 - y : y;
    const int sv = hflip ? vpr - 1 - vx : vx;
    const Vec v = *reinterpret_cast<const Vec*>(in + (src.plane(plane) * H + sy) * (long long)W + sv * V);
    Vec o;
    if (hflip) {
#pragma unroll
      for (int k = 0; k < V; ++k) o.e[k] = v.e[V - 1 - k];
    } else {
      o = v;
    }
    *reinterpret_cast<Vec*>(out + (row0 + r) * (long long)W + vx * V) = o;
  }
}

// labels (N, 6, Sy, Sx) = [mask, x1, y1, x2, y2, class]: cells mirrored, x1' = 1 - x2, x2' = 1 - x1 (hflip) and
// y1' = 1 - y2, y2' = 1 - y1 (vflip) on EVERY cell, labelled or not, exactly as the reference's tensor expression does
__global__ void __launch_bounds__(256) flip_labels_kernel(const float* __restrict__ in, float* __restrict__ out, int N, int Sy,
                                                          int Sx, int hflip, int vflip) {
  // blockIdx.y = n * 6 + c (one channel plane), blockIdx.x * 256 + threadIdx.x = cell of the plane: 32-bit arithmetic only
  const int cell = blockIdx.x * 256 + threadIdx.x;
  if (cell >= Sy * Sx) return;
  const int plane = blockIdx.y;
  const int n = plane / 6, c = plane - n * 6;
  const int y = cell / Sx, x = cell - y * Sx;
  const int sx = hflip ? Sx - 1 - x : x, sy = vflip ? Sy - 1 - y : y;
  int sc = c;
  bool comp = false;
  if (hflip && (c == 1 || c == 3)) { sc = 4 - c; comp = true; }
  if (vflip && (c == 2 || c == 4)) { sc = 6 - c; comp = true; }
  const float v = in[((long long)(n * 6 + sc) * Sy + sy) * Sx + sx];
  out[(long long)plane * Sy * Sx + cell] = comp ? __fsub_rn(1.f, v) : v;
}

// pass 1: owner[b][cell] = the LAST label of image b whose centre falls into the cell (the reference's Python loop
// overwrites in order); cell indices as torch computes them: ((x1 + x2) * Sx) // 2 in fp32, truncated to int, negative
// indices wrap like Python indexing, anything else out of range raises IndexError in the reference -> error flag
__global__ void label_owner_kernel(const float* __restrict__ labels, const int* __restrict__ offsets, int B, int Sy, int Sx,
                                   int* __restrict__ owner, int* __restrict__ err) {
  const int b = blockIdx.y;
  const int lo = offsets[b], hi = offsets[b + 1];
  for (int l = lo + blockIdx.x * blockDim.x + threadIdx.x; l < hi; l += gridDim.x * blockDim.x) {
    const float* r = labels + (long long)l * 5;
    const float fi = floorf(__fmul_rn(__fadd_rn(r[1], r[3]), (float)Sx) / 2.f);
    const float fj = floorf(__fmul_rn(__fadd_rn(r[2], r[4]), (float)Sy) / 2.f);
    int i = (int)fi, j = (int)fj;
    if (i < 0) i += Sx;
    if (j < 0) j += Sy;
    if (!(fi == fi) || !(fj == fj) || i < 0 || i >= Sx || j < 0 || j >= Sy) { atomicExch(err, 1); continue; }
    atomicMax(&owner[((long long)b * Sy + j) * Sx + i], l - lo);
  }
}

// pass 2: (B, 6, Sy, Sx) = [1, x1, y1, x2, y2, class] of the owning label, zeros elsewhere
__global__ void label_fill_kernel(const float* __restrict__ labels, const int* __restrict__ offsets, int B, int Sy, int Sx,
                                  const int* __restrict__ owner, float* __restrict__ out) {
  const long long cells = (long long)B * Sy * Sx;
  const long long plane = (long long)Sy * Sx;
  for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < cells; c += (long long)gridDim.x * blockDim.x) {
    const long long b = c / plane, cell = c - b * plane;
    const int o = owner[c];
    float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (o >= 0) {
      const float* r = labels + ((long long)offsets[b] + o) * 5;
      v[0] = 1.f; v[1] = r[1]; v[2] = r[2]; v[3] = r[3]; v[4] = r[4]; v[5] = r[0];
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) out[(b * 6 + k) * plane + cell] = v[k];
  }
}

}  // namespace yg
using namespace yg;

static unsigned flip_grid(long long rows) { return (unsigned)((rows + FLIP_ROWS - 1) / FLIP_ROWS); }
static int grid_for(long long work_items) {
  long long b = (work_items + 255) / 256;
  return (int)(b < 1 ? 1 : (b > 148 * 16 ? 148 * 16 : b));
}

extern "C" int yg_flip_images(const void* in, void* out, int dtype, int N, int C, int H, int W, int hflip, int vflip,
                              void* stream) {
  YG_CHECK_ARG(dtype == YG_U8 || dtype == YG_F32, "flip_images: dtype %d", dtype);
  const long long rows = (long long)N * C * H;
  if (rows == 0 || W == 0) return YG_OK;
  YG_CHECK_ARG(in && out && in != out, "flip_images: null or aliased pointers (the flip is out of place)");
  YG_CHECK_ARG(rows / FLIP_ROWS < (1LL << 31), "flip_images: too many rows");
  cudaStream_t st = (cudaStream_t)stream;
  const bool al = (((uintptr_t)in | (uintptr_t)out) & 15) == 0;
  if (dtype == YG_U8) {
    if (al && W % 16 == 0) flip_images_kernel<uint8_t, 16><<<flip_grid(rows), 256, 0, st>>>((const uint8_t*)in, (uint8_t*)out, rows, H, W, FlipArgs{hflip, vflip});
    else if (al && W % 8 == 0) flip_images_kernel<uint8_t, 8><<<flip_grid(rows), 256, 0, st>>>((const uint8_t*)in, (uint8_t*)out, rows, H, W, FlipArgs{hflip, vflip});
    else flip_images_kernel<uint8_t, 1><<<flip_grid(rows), 256, 0, st>>>((const uint8_t*)in, (uint8_t*)out, rows, H, W, FlipArgs{hflip, vflip});
  } else {
    if (al && W % 4 == 0) flip_images_kernel<float, 4><<<flip_grid(rows), 256, 0, st>>>((const float*)in, (float*)out, rows, H, W, FlipArgs{hflip, vflip});
    else flip_images_kernel<float, 1><<<flip_grid(rows), 256, 0, st>>>((const float*)in, (float*)out, rows, H, W, FlipArgs{hflip, vflip});
  }
  YG_LAUNCH_CHECK("flip_images");
  return YG_OK;
}

extern "C" int yg_flip_labels(const float* in, float* out, int N, int Sy, int Sx, int hflip, int vflip, void* stream) {
  const long long total = (long long)N * 6 * Sy * Sx;
  if (total == 0) return YG_OK;
  YG_CHECK_ARG(in && out && in != out, "flip_labels: null or aliased pointers (the flip is out of place)");
  YG_CHECK_ARG((long long)N * 6 <= 65535, "flip_labels: batch %d too large for one launch", N);
  dim3 grid(cdiv((long long)Sy * Sx, 256), N * 6, 1);
  flip_labels_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in, out, N, Sy, Sx, hflip, vflip);
  YG_LAUNCH_CHECK("flip_labels");
  return YG_OK;
}

extern "C" int yg_format_labels_batch(const float* labels, const int* offsets, int B, int max_labels, int Sy, int Sx,
                                      int* owner, float* out, int* err, void* stream) {
  if (B == 0) return YG_OK;
  YG_CHECK_ARG(offsets && owner && out && err && Sy > 0 && Sx > 0, "format_labels_batch: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const long long cells = (long long)B * Sy * Sx;
  cudaMemsetAsync(owner, 0xFF, cells * sizeof(int), st);   // -1 = no label
  cudaMemsetAsync(err, 0, sizeof(int), st);
  if (max_labels > 0) {
    YG_CHECK_ARG(labels != nullptr, "format_labels_batch: labels is null");
    dim3 grid(cdiv(max_labels, 256), B, 1);
    label_owner_kernel<<<grid, 256, 0, st>>>(labels, offsets, B, Sy, Sx, owner, err);
    YG_LAUNCH_CHECK("format_labels owner");
  }
  label_fill_kernel<<<grid_for(cells), 256, 0, st>>>(labels, offsets, B, Sy, Sx, owner, out);
  YG_LAUNCH_CHECK("format_labels fill");
  return YG_OK;
}


// ------------------------------------------------------------------------------------------------
// Dropout2d keep-scales of ALL blocks of a step in one launch (nn.Dropout2d(p), model_defns.py:44-57: whole (n, c)
// planes are zeroed with probability p, the rest scaled by 1 / (1 - p)), plus the `num_batches_tracked += 1` of the
// BatchNorm layers.  Replaces ~5 torch elementwise launches per block (rand, >=, float, div, contiguous) and one per counter.
// Philox4x32-10 keyed by (seed, call counter, element): the counter lives in device memory and is advanced by the kernel
// itself, so that a CUDA-graph replay draws fresh masks.  state = [seed, counter, ticket].
// ------------------------------------------------------------------------------------------------
namespace yg {
__device__ __forceinline__ uint32_t mulhilo32(uint32_t a, uint32_t b, uint32_t* hi) {
  const unsigned long long p = (unsigned long long)a * b;
  *hi = (uint32_t)(p >> 32);
  return (uint32_t)p;
}
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, hi1;
    const uint32_t lo0 = mulhilo32(0xD2511F53u, ctr.x, &hi0), lo1 = mulhilo32(0xCD9E8D57u, ctr.z, &hi1);
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u; key.y += 0xBB67AE85u;
  }
  return ctr;
}

// table: per block (offset, count, p as float bits, unused), nblk <= 16
__global__ void dropout_scales_kernel(float* __restrict__ out, const int4* __restrict__ table, int nblk, int total,
                                      unsigned long long* __restrict__ state, long long* const* __restrict__ counters, int ncounters) {
  const unsigned long long seed = state[0], call = state[1];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) {
    float p = 0.f;
    for (int b = 0; b < nblk; ++b) {
      const int4 t = table[b];
      if (i >= t.x && i < t.x + t.y) p = __int_as_float(t.z);
    }
    const uint4 r = philox4x32_10(make_uint4((uint32_t)i, 0u, (uint32_t)call, (uint32_t)(call >> 32)),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float u = (float)(r.x >> 8) * (1.0f / 16777216.0f);     // uniform in [0, 1)
    out[i] = (u >= p) ? 1.f / (1.f - p) : 0.f;
  }
  // the last block to finish advances the call counter and the BatchNorm counters (every block has read `call` by then)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned long long done = atomicAdd(&state[2], 1ull);
    if (done == gridDim.x - 1) {
      state[2] = 0ull;
      state[1] = call + 1ull;
      for (int c = 0; c < ncounters; ++c) *counters[c] += 1;
    }
  }
}
}  // namespace yg

extern "C" int yg_dropout_scales(float* out, const void* table, int nblocks, int total, void* state, const void* counters,
                                 int ncounters, void* stream) {
  YG_CHECK_ARG(state && nblocks >= 0 && nblocks <= 16 && total >= 0 && ncounters >= 0, "dropout_scales: bad arguments");
  YG_CHECK_ARG(total == 0 || (out && table), "dropout_scales: null pointer");
  const int grid = total > 0 ? yg::cdiv(total, 256) : 1;
  yg::dropout_scales_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out, (const int4*)table, nblocks, total,
                                                                    (unsigned long long*)state, (long long* const*)counters, ncounters);
  YG_LAUNCH_CHECK("dropout_scales");
  return YG_OK;
}


// ------------------------------------------------------------------------------------------------
// Device-resident dataset (data/device_dataset.py): every batch of an epoch is built on the device from the decoded store,
// so that a CUDA-graph replay of the training step draws, gathers and rasterises its own batch.
//   draw:   one (hflip, vflip) pair per batch (the reference flips whole batches in the collate function,
//           data_transforms.py:51-98) from Philox keyed by (seed, call counter); state = [seed, counter, batch cursor] in
//           device memory, advanced by the kernel itself like dropout_scales; flags = [hflip, vflip, batch] of the batch
//           just drawn, read by the two kernels below and by callers.
//   images: flip_images_kernel with GatherSrc (one HBM pass, vector accesses).
//   labels: the (B, 6, Sy, Sx) tensor flip_batch(stack(labels), h, v) produces, from per-image compact cell records.
// ------------------------------------------------------------------------------------------------
namespace yg {
__global__ void dd_draw_kernel(unsigned long long* __restrict__ state, int* __restrict__ flags, float ph, float pv,
                               uint32_t stream_id, int nbatches) {
  const unsigned long long seed = state[0], call = state[1], cursor = state[2];
  const uint4 r = philox4x32_10(make_uint4(stream_id, 0x464C4950u, (uint32_t)call, (uint32_t)(call >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const float uh = (float)(r.x >> 8) * (1.0f / 16777216.0f), uv = (float)(r.y >> 8) * (1.0f / 16777216.0f);  // [0, 1)
  flags[0] = uh < ph;   // p = 0: never, p = 1: always
  flags[1] = uv < pv;
  flags[2] = (int)(cursor % (unsigned long long)nbatches);   // a draw past the epoch's end starts it again
  state[1] = call + 1ull;
  state[2] = cursor + 1ull;
}

// records: two int4 per labelled cell {cell, 6 channel values as float bits, 0}, sorted by cell within each stored image;
// rec_off[i], rec_off[i + 1]: record range of stored image i.  One block = `rpb` output rows of one image: it writes the
// mirrored default of its rows (channels that the flip complements are 1 - 0 = 1, the rest 0, as flip_labels_kernel gives
// for an unlabelled cell), then its labelled cells, whose sources are one contiguous record range (rows map to rows).
__global__ void __launch_bounds__(256) dd_labels_kernel(const int* __restrict__ table, const int* __restrict__ flags, int stride,
                                                        const int4* __restrict__ rec, const long long* __restrict__ rec_off,
                                                        int Sy, int Sx, int rpb, float* __restrict__ out) {
  const int hflip = flags[0], vflip = flags[1];
  const int b = blockIdx.y;
  const int img = table[(long long)flags[2] * stride + b];
  const int r0 = blockIdx.x * rpb, r1 = min(Sy, r0 + rpb);
  const int plane = Sy * Sx;
  float* o = out + (long long)b * 6 * plane;
  const float one = __fsub_rn(1.f, 0.f);
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const float d = (hflip && (k == 1 || k == 3)) || (vflip && (k == 2 || k == 4)) ? one : 0.f;
    for (int c = r0 * Sx + threadIdx.x; c < r1 * Sx; c += blockDim.x) o[k * plane + c] = d;
  }
  __syncthreads();   // the labelled cells below overwrite defaults written by other threads of this block
  const int s0 = vflip ? Sy - r1 : r0, s1 = vflip ? Sy - r0 : r1;   // source rows of output rows [r0, r1)
  const long long lo = rec_off[img], hi = rec_off[img + 1];
  long long a = lo, e = hi;
  while (a < e) { const long long m = (a + e) >> 1; if (rec[2 * m].x < s0 * Sx) a = m + 1; else e = m; }
  const long long first = a;
  e = hi;
  while (a < e) { const long long m = (a + e) >> 1; if (rec[2 * m].x < s1 * Sx) a = m + 1; else e = m; }
  for (long long i = first + threadIdx.x; i < a; i += blockDim.x) {
    const int4 h0 = rec[2 * i], h1 = rec[2 * i + 1];
    const int sy = h0.x / Sx, sx = h0.x - sy * Sx;
    const int oc = (vflip ? Sy - 1 - sy : sy) * Sx + (hflip ? Sx - 1 - sx : sx);
    float v[6] = {__int_as_float(h0.y), __int_as_float(h0.z), __int_as_float(h0.w),
                  __int_as_float(h1.x), __int_as_float(h1.y), __int_as_float(h1.z)};
    if (hflip) { const float t = v[1]; v[1] = __fsub_rn(1.f, v[3]); v[3] = __fsub_rn(1.f, t); }
    if (vflip) { const float t = v[2]; v[2] = __fsub_rn(1.f, v[4]); v[4] = __fsub_rn(1.f, t); }
#pragma unroll
    for (int k = 0; k < 6; ++k) o[k * plane + oc] = v[k];
  }
}

// Sharded store (each rank of one host keeps a contiguous 1/W of the slots, peers' shards mapped over NVLink): stored
// slot s is image s % shard_items of shards[s / shard_items].  One block = `rpb` consecutive rows of one output plane, so
// the source plane is resolved once per block; every thread issues PG_UNROLL independent vector loads before its first
// store, which keeps enough bytes in flight to cover a remote round trip.  Same output as flip_images_kernel<GatherSrc>.
constexpr int PG_THREADS = 256, PG_UNROLL = 8;
template <typename T, int V>
__global__ void __launch_bounds__(PG_THREADS) dd_gather_peers_kernel(const T* const* __restrict__ shards, long long shard_items,
                                                                     T* __restrict__ out, const int* __restrict__ table,
                                                                     const int* __restrict__ flags, int stride, int C, int H,
                                                                     int W, int rpb, int blocks_per_plane) {
  struct alignas(sizeof(T) * V) Vec { T e[V]; };
  const int hflip = flags[0], vflip = flags[1];
  const int plane = blockIdx.x / blocks_per_plane;   // n * C + c
  const int y0 = (blockIdx.x - plane * blocks_per_plane) * rpb;
  const int n = plane / C, c = plane - n * C;
  const long long s = table[(long long)flags[2] * stride + n];
  const long long shard = s / shard_items, item = s - shard * shard_items;
  const long long plane_elems = (long long)H * W;
  const T* src = shards[shard] + (item * C + c) * plane_elems;
  T* dst = out + (long long)plane * plane_elems + (long long)y0 * W;
  const int vpr = W / V;
  const int total = min(rpb, H - y0) * vpr;
  for (int i0 = threadIdx.x; i0 < total; i0 += PG_THREADS * PG_UNROLL) {
    Vec v[PG_UNROLL];
#pragma unroll
    for (int u = 0; u < PG_UNROLL; ++u) {
      const int idx = i0 + u * PG_THREADS;
      if (idx < total) {
        const int r = idx / vpr, vx = idx - r * vpr;
        const int sy = vflip ? H - 1 - (y0 + r) : y0 + r;
        const int sv = hflip ? vpr - 1 - vx : vx;
        v[u] = *reinterpret_cast<const Vec*>(src + (long long)sy * W + sv * V);
      }
    }
#pragma unroll
    for (int u = 0; u < PG_UNROLL; ++u) {
      const int idx = i0 + u * PG_THREADS;
      if (idx < total) {
        const int r = idx / vpr, vx = idx - r * vpr;
        Vec o = v[u];
        if (hflip) {
          if constexpr (sizeof(T) == 1 && V >= 4) {   // byte reversal as word swaps + byte permutes
            uint32_t* ow = reinterpret_cast<uint32_t*>(o.e);
            const uint32_t* iw = reinterpret_cast<const uint32_t*>(v[u].e);
#pragma unroll
            for (int k = 0; k < V / 4; ++k) ow[k] = __byte_perm(iw[V / 4 - 1 - k], 0, 0x0123);
          } else {
#pragma unroll
            for (int k = 0; k < V; ++k) o.e[k] = v[u].e[V - 1 - k];
          }
        }
        *reinterpret_cast<Vec*>(dst + (long long)r * W + vx * V) = o;
      }
    }
  }
}
}  // namespace yg

extern "C" int yg_dd_draw(void* state, int* flags, float p_hflip, float p_vflip, int stream_id, int nbatches, void* stream) {
  YG_CHECK_ARG(state && flags && nbatches > 0, "dd_draw: bad arguments");
  YG_CHECK_ARG(p_hflip >= 0.f && p_hflip <= 1.f && p_vflip >= 0.f && p_vflip <= 1.f, "dd_draw: p outside [0, 1]");
  yg::dd_draw_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((unsigned long long*)state, flags, p_hflip, p_vflip,
                                                         (uint32_t)stream_id, nbatches);
  YG_LAUNCH_CHECK("dd_draw");
  return YG_OK;
}

extern "C" int yg_dd_gather_images(const void* store, void* out, int dtype, const int* table, const int* flags, int stride,
                                   int N, int C, int H, int W, void* stream) {
  YG_CHECK_ARG(dtype == YG_U8 || dtype == YG_F32, "dd_gather_images: dtype %d", dtype);
  YG_CHECK_ARG(C == 1 || C == 3, "dd_gather_images: C = %d (1 or 3)", C);
  const long long rows = (long long)N * C * H;
  if (rows == 0 || W == 0) return YG_OK;
  YG_CHECK_ARG(store && out && table && flags && store != out && N <= stride, "dd_gather_images: bad arguments");
  YG_CHECK_ARG(rows / FLIP_ROWS < (1LL << 31), "dd_gather_images: too many rows");
  cudaStream_t st = (cudaStream_t)stream;
  const bool al = (((uintptr_t)store | (uintptr_t)out) & 15) == 0;
  const GatherSrc g{table, flags, stride, C, 0, 0, 0};
  if (dtype == YG_U8) {
    if (al && W % 16 == 0) flip_images_kernel<uint8_t, 16><<<flip_grid(rows), 256, 0, st>>>((const uint8_t*)store, (uint8_t*)out, rows, H, W, g);
    else if (al && W % 8 == 0) flip_images_kernel<uint8_t, 8><<<flip_grid(rows), 256, 0, st>>>((const uint8_t*)store, (uint8_t*)out, rows, H, W, g);
    else flip_images_kernel<uint8_t, 1><<<flip_grid(rows), 256, 0, st>>>((const uint8_t*)store, (uint8_t*)out, rows, H, W, g);
  } else {
    if (al && W % 4 == 0) flip_images_kernel<float, 4><<<flip_grid(rows), 256, 0, st>>>((const float*)store, (float*)out, rows, H, W, g);
    else flip_images_kernel<float, 1><<<flip_grid(rows), 256, 0, st>>>((const float*)store, (float*)out, rows, H, W, g);
  }
  YG_LAUNCH_CHECK("dd_gather_images");
  return YG_OK;
}

extern "C" int yg_dd_gather_images_peers(const void* const* shards, long long shard_items, void* out, int dtype,
                                         const int* table, const int* flags, int stride, int N, int C, int H, int W,
                                         void* stream) {
  YG_CHECK_ARG(dtype == YG_U8 || dtype == YG_F32, "dd_gather_images_peers: dtype %d", dtype);
  YG_CHECK_ARG(C == 1 || C == 3, "dd_gather_images_peers: C = %d (1 or 3)", C);
  const long long rows = (long long)N * C * H;
  if (rows == 0 || W == 0) return YG_OK;
  YG_CHECK_ARG(shards && out && table && flags && shard_items > 0 && N <= stride && H > 0 && W > 0,
               "dd_gather_images_peers: bad arguments");
  YG_CHECK_ARG(rows / FLIP_ROWS < (1LL << 31), "dd_gather_images_peers: too many rows");
  cudaStream_t st = (cudaStream_t)stream;
  const bool al = ((uintptr_t)out & 15) == 0;   // shard bases are allocation starts (256-byte aligned)
  auto launch = [&](auto* tp, auto vw) -> int {
    using T = std::remove_pointer_t<decltype(tp)>;
    constexpr int V = decltype(vw)::value;
    const int vpr = W / V;
    const int rpb = std::max(1, std::min(H, PG_THREADS * PG_UNROLL / vpr));
    const int bpp = (H + rpb - 1) / rpb;
    const long long blocks = (long long)N * C * bpp;
    YG_CHECK_ARG(blocks < (1LL << 31), "dd_gather_images_peers: too many rows");
    dd_gather_peers_kernel<T, V><<<(unsigned)blocks, PG_THREADS, 0, st>>>((const T* const*)shards, shard_items, (T*)out, table,
                                                                          flags, stride, C, H, W, rpb, bpp);
    return YG_OK;
  };
  using std::integral_constant;
  int rc;
  if (dtype == YG_U8) {
    if (al && W % 16 == 0) rc = launch((uint8_t*)nullptr, integral_constant<int, 16>{});
    else if (al && W % 8 == 0) rc = launch((uint8_t*)nullptr, integral_constant<int, 8>{});
    else rc = launch((uint8_t*)nullptr, integral_constant<int, 1>{});
  } else {
    if (al && W % 4 == 0) rc = launch((float*)nullptr, integral_constant<int, 4>{});
    else rc = launch((float*)nullptr, integral_constant<int, 1>{});
  }
  if (rc != YG_OK) return rc;
  YG_LAUNCH_CHECK("dd_gather_images_peers");
  return YG_OK;
}

// Shard memory of a sharded store: plain cudaMalloc (an allocation of its own, so its IPC handle maps exactly this
// buffer), exported to and opened by the other processes of the host.  Teardown order is the caller's protocol
// (DeviceResidentDataset.close): every importer closes its handle before the owner frees.
static_assert(sizeof(cudaIpcMemHandle_t) == YG_IPC_HANDLE_BYTES, "IPC handle size");

extern "C" int yg_dd_shard_alloc(size_t bytes, void** ptr) {
  YG_CHECK_ARG(ptr && bytes > 0, "dd_shard_alloc: bad arguments");
  *ptr = nullptr;
  YG_CUDA(cudaMalloc(ptr, bytes));
  return YG_OK;
}

extern "C" int yg_dd_shard_export(const void* ptr, void* handle) {
  YG_CHECK_ARG(ptr && handle, "dd_shard_export: bad arguments");
  cudaIpcMemHandle_t h;
  YG_CUDA(cudaIpcGetMemHandle(&h, const_cast<void*>(ptr)));
  memcpy(handle, &h, sizeof(h));
  return YG_OK;
}

extern "C" int yg_dd_shard_open(const void* handle, void** ptr) {
  YG_CHECK_ARG(handle && ptr, "dd_shard_open: bad arguments");
  *ptr = nullptr;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  YG_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return YG_OK;
}

extern "C" int yg_dd_shard_close(void* ptr) {
  YG_CHECK_ARG(ptr, "dd_shard_close: null pointer");
  YG_CUDA(cudaIpcCloseMemHandle(ptr));
  return YG_OK;
}

extern "C" int yg_dd_shard_free(void* ptr) {
  YG_CHECK_ARG(ptr, "dd_shard_free: null pointer");
  YG_CUDA(cudaFree(ptr));
  return YG_OK;
}

extern "C" int yg_dd_build_labels(const int* table, const int* flags, int stride, const void* records, const long long* rec_off,
                                  int N, int Sy, int Sx, float* out, void* stream) {
  if (N == 0 || Sy == 0 || Sx == 0) return YG_OK;
  YG_CHECK_ARG(table && flags && records && rec_off && out && N <= stride, "dd_build_labels: bad arguments");
  YG_CHECK_ARG(N <= 65535 && (long long)Sy * Sx * 6 < (1LL << 31), "dd_build_labels: batch %d or grid too large", N);
  const int rpb = Sx >= 2048 ? 1 : 2048 / Sx;
  dim3 grid(cdiv(Sy, rpb), N, 1);
  dd_labels_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(table, flags, stride, (const int4*)records, rec_off, Sy, Sx, rpb, out);
  YG_LAUNCH_CHECK("dd_build_labels");
  return YG_OK;
}
