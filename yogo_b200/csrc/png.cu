// PNG decoding of 8-bit grayscale, non-interlaced files on the device (yg_png_decode_gray8).  The host walks each
// file's chunks (yogo_b200/data/png.py) and hands over an IDAT table; three kernels do the rest:
//
//   png_gather_crc_kernel  one CTA per image, one warp per IDAT chunk: CRC-32 of type + payload, lane k over the k-th
//                          32nd of the chunk, the 32 partial CRCs combined with zlib's crc32_combine algebra; the
//                          payload copied to the image's contiguous zlib stream
//   png_inflate_kernel     one warp per image: lane 0 decodes up to INF_QUEUE symbols into a shared-memory queue
//                          (Huffman tables in shared memory, the compressed input staged in a shared window), then the
//                          warp writes the queued literals 32 at a time and runs each LZ77 copy across its lanes
//   png_unfilter_kernel    one warp per image, a row wavefront: lane k owns row r0 + k and runs one column behind lane
//                          k - 1, so the up / upper-left bytes arrive by __shfl_up; 32 rows x UNF_STRIP columns are
//                          staged in shared memory so that global reads and writes stay coalesced.  Adler-32 of the
//                          filtered bytes is summed on the way.
//
// The per-stream logic (bit reader, table build, symbol decode, unfilter) is png_core.cuh, shared with host builds.
// Any malformed input ends in a nonzero per-image status (the caller then decodes that file with libpng), never in an
// access outside the image's buffers: every stream read is bounds-checked, every queued entry is checked against the
// output capacity, and table indices are < 1 << bits by construction.
#include "common.cuh"
#include "png_core.cuh"

namespace yg {

using namespace png;

constexpr int GATHER_WARPS = 8;
constexpr int INF_WARPS = 4;
constexpr int INF_QUEUE = 128;    // symbols decoded by lane 0 per round
constexpr int INF_WINDOW = 2048;  // staged compressed bytes; refreshed when fewer than INF_AHEAD remain ahead
constexpr int INF_AHEAD = 1024;   // > INF_QUEUE * 6 bytes (the most one round can consume) + 4 bytes of look-ahead
constexpr int UNF_WARPS = 4;
constexpr int UNF_STRIP = 128;    // columns per wavefront tile
constexpr int UNF_PITCH = UNF_STRIP + 4;

__constant__ CrcTables c_crc = make_crc_tables();

struct PngLayout {
  long long scratch, aux, streams, total;
};
// workspace: filtered scanlines (n x H x (1 + W)), the stored Adler-32 of each image, then the zlib streams
inline PngLayout png_layout(int n, int H, int W, long long stream_bytes) {
  auto up = [](long long v) { return (v + 255) & ~255ll; };
  PngLayout l;
  l.scratch = 0;
  l.aux = up((long long)n * H * (W + 1));
  l.streams = l.aux + up(4ll * n);
  l.total = l.streams + up(stream_bytes);
  return l;
}

__device__ __forceinline__ void set_status(int* status, int img, int code) { atomicCAS(status + img, YG_PNG_OK, code); }

// ---- IDAT gather + CRC ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * GATHER_WARPS) png_gather_crc_kernel(
    const uint8_t* __restrict__ files, long long files_bytes, const yg_png_chunk* __restrict__ chunks,
    const yg_png_image* __restrict__ images, uint8_t* __restrict__ streams, long long stream_bytes, int* status) {
  __shared__ CrcTables t;
  for (int i = threadIdx.x; i < 256 + 32; i += blockDim.x) (i < 256 ? t.byte[i] : t.x2n[i - 256]) = (i < 256 ? c_crc.byte[i] : c_crc.x2n[i - 256]);
  __syncthreads();
  const int img = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const yg_png_image im = images[img];
  if (im.stream < 0 || (im.stream & 15) || im.length < 0 || im.stream + ((im.length + 15) & ~15ll) > stream_bytes) {
    if (threadIdx.x == 0) set_status(status, img, YG_PNG_BAD_LAYOUT);
    return;
  }
  for (int c = im.chunk_begin + warp; c < im.chunk_end; c += GATHER_WARPS) {
    const yg_png_chunk ch = chunks[c];
    const long long n = (long long)ch.length + 4;   // type + payload
    if (ch.src < 0 || ch.length < 0 || ch.src + n > files_bytes || ch.dst < im.stream ||
        ch.dst + ch.length > im.stream + im.length) {
      if (lane == 0) set_status(status, img, YG_PNG_BAD_LAYOUT);
      continue;
    }
    const uint8_t* p = files + ch.src;
    const long long seg = (n + 31) >> 5, b0 = min(n, lane * seg), b1 = min(n, b0 + seg);
    uint32_t crc = 0xffffffffu;
    for (long long i = b0; i < b1; ++i) crc = t.byte[(crc ^ p[i]) & 0xff] ^ (crc >> 8);
    uint32_t v = b1 > b0 ? multmodp(x2nmodp(t, (unsigned long long)(n - b1), 3), ~crc) : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v ^= __shfl_xor_sync(0xffffffffu, v, o);
    if (v != ch.crc && lane == 0) set_status(status, img, YG_PNG_BAD_CRC);
    uint8_t* d = streams + ch.dst;
    for (long long i = lane; i < ch.length; i += 32) d[i] = p[4 + i];
  }
}

// ---- inflate -------------------------------------------------------------------------------------------------------
struct InflateSmem {
  InflateTables t;
  uint32_t q[INF_QUEUE];
  alignas(16) uint8_t win[INF_WINDOW];
};

__global__ void __launch_bounds__(32 * INF_WARPS) png_inflate_kernel(
    const uint8_t* __restrict__ streams, const yg_png_image* __restrict__ images, int n, long long cap,
    uint8_t* __restrict__ scratch, uint32_t* __restrict__ adler, int* status) {
  __shared__ InflateSmem smem[INF_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, img = blockIdx.x * INF_WARPS + warp;
  if (img >= n || status[img] != YG_PNG_OK) return;   // warp-uniform
  InflateSmem& s = smem[warp];
  const yg_png_image im = images[img];                // layout checked by the gather kernel
  const uint8_t* src = streams + im.stream;
  const long long padded = (im.length + 15) & ~15ll;
  uint8_t* out = scratch + (long long)img * cap;
  BitReader br{src, im.length, s.win, 0, 0, 0, 0, 0};   // meaningful in lane 0 only
  long long out_pos = 0;                                // lane 0
  int window = 0, err = YG_PNG_OK;

  // keep INF_AHEAD bytes past lane 0's read position in the shared window (warp-collective)
  auto refresh = [&]() {
    const long long pos = __shfl_sync(0xffffffffu, br.pos, 0);
    if (br.wlen == 0 || pos + INF_AHEAD > br.wbase + INF_WINDOW) {
      __syncwarp();
      const long long base = pos & ~15ll;
      for (int k = lane; k < INF_WINDOW / 16; k += 32) {
        const long long off = base + 16ll * k;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (off + 16 <= padded) v = *reinterpret_cast<const uint4*>(src + off);
        *reinterpret_cast<uint4*>(s.win + 16 * k) = v;
      }
      br.wbase = base;
      br.wlen = INF_WINDOW;
      __syncwarp();
    }
  };

  refresh();
  if (lane == 0) err = zlib_header(br, window);
  err = __shfl_sync(0xffffffffu, err, 0);
  bool last = false;
  while (!err && !last) {
    refresh();
    int btype = 0, final_block = 0, slen = 0;
    long long sfrom = 0, opos = 0;
    if (lane == 0) {
      final_block = (int)br.bits(1);
      btype = (int)br.bits(2);
      if (btype == 0) {
        br.align();
        const long long p = br.byte_pos();
        const uint32_t len = br.byte(p) | br.byte(p + 1) << 8, nlen = br.byte(p + 2) | br.byte(p + 3) << 8;
        if (len != (~nlen & 0xffffu)) {
          err = YG_PNG_BAD_STORED_LENGTH;
        } else if (p + 4 + len > im.length) {
          err = YG_PNG_TRUNCATED;
        } else if (len > cap - out_pos) {
          err = YG_PNG_OUTPUT_OVERFLOW;
        } else {
          sfrom = p + 4;
          slen = (int)len;
          opos = out_pos;
          out_pos += len;
          br.seek(p + 4 + len);
        }
      } else if (btype == 3) {
        err = YG_PNG_BAD_BLOCK_TYPE;
      } else if (btype == 1) {
        fixed_lengths(s.t);
      } else {
        err = dynamic_lengths(br, s.t);
      }
    }
    err = __shfl_sync(0xffffffffu, err, 0);
    btype = __shfl_sync(0xffffffffu, btype, 0);
    last = __shfl_sync(0xffffffffu, final_block, 0) != 0;
    if (err) break;
    if (btype == 0) {
      sfrom = __shfl_sync(0xffffffffu, sfrom, 0);
      opos = __shfl_sync(0xffffffffu, opos, 0);
      slen = __shfl_sync(0xffffffffu, slen, 0);
      for (int i = lane; i < slen; i += 32) out[opos + i] = src[sfrom + i];
      __syncwarp();
      continue;
    }
    // primary tables of this block, filled by the whole warp
    __syncwarp();
    for (int i = lane; i < (1 << LIT_BITS); i += 32) s.t.lit[i] = 0;
    for (int i = lane; i < (1 << DIST_BITS); i += 32) s.t.dist[i] = 0;
    __syncwarp();
    huff_fill(s.t.hl, s.t.lens, s.t.lit, LIT_BITS, lane, 32);
    huff_fill(s.t.hd, s.t.lens + MAX_LIT, s.t.dist, DIST_BITS, lane, 32);
    __syncwarp();
    bool eob = false;
    while (!eob) {
      refresh();
      int nq = 0;
      long long base = out_pos;
      if (lane == 0) {
        err = decode_symbols(br, s.t, s.q, INF_QUEUE, out_pos, cap, window, nq, eob);
        if (!err && br.consumed_bits() > im.length * 8) err = YG_PNG_TRUNCATED;
      }
      err = __shfl_sync(0xffffffffu, err, 0);
      if (err) break;
      nq = __shfl_sync(0xffffffffu, nq, 0);
      eob = __shfl_sync(0xffffffffu, (int)eob, 0) != 0;
      base = __shfl_sync(0xffffffffu, base, 0);
      __syncwarp();
      for (int g = 0; g < nq; g += 32) {
        const int k = g + lane;
        const uint32_t e = k < nq ? s.q[k] : 0u;
        const int len = k < nq ? q_len(e) : 0;
        int incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += v;
        }
        const long long p = base + incl - len;
        const bool match = k < nq && (e & Q_MATCH);
        if (k < nq && !match) out[p] = (uint8_t)e;
        unsigned mm = __ballot_sync(0xffffffffu, match);
        __syncwarp();
        while (mm) {
          const int j = __ffs(mm) - 1;
          mm &= mm - 1;
          const uint32_t ej = __shfl_sync(0xffffffffu, e, j);
          const long long pj = __shfl_sync(0xffffffffu, p, j);
          const int L = q_len(ej), D = q_dist(ej);
          // out[pj + i] = out[pj - D + i mod D]: every source byte precedes pj, so all lanes copy at once
          for (int i = lane; i < L; i += 32) out[pj + i] = out[pj - D + (D >= L ? i : i % D)];
          __syncwarp();
        }
        base += __shfl_sync(0xffffffffu, incl, 31);
      }
    }
  }
  if (lane == 0) {
    if (!err) {
      br.align();
      uint32_t a = br.bits(8) << 24;
      a |= br.bits(8) << 16;
      a |= br.bits(8) << 8;
      a |= br.bits(8);
      if (br.consumed_bits() > im.length * 8 || out_pos != cap) err = YG_PNG_TRUNCATED;
      else if (br.byte_pos() != im.length) err = YG_PNG_TRAILING_DATA;
      else adler[img] = a;
    } else if (br.consumed_bits() > im.length * 8) {
      err = YG_PNG_TRUNCATED;   // whatever failed was read past the end of the stream
    }
    if (err) set_status(status, img, err);
  }
}

// ---- unfilter + Adler-32 -------------------------------------------------------------------------------------------
struct UnfilterSmem {
  uint8_t fin[32][UNF_PITCH];    // filtered bytes of the tile
  uint8_t fout[32][UNF_PITCH];   // reconstructed bytes of the tile
  uint8_t prev[UNF_PITCH];       // row r0 - 1, columns c0 - 1 .. c0 + UNF_STRIP - 1
};

__global__ void __launch_bounds__(32 * UNF_WARPS) png_unfilter_kernel(
    const uint8_t* __restrict__ scratch, int n, int H, int W, const uint32_t* __restrict__ adler,
    uint8_t* __restrict__ out, int* status) {
  __shared__ UnfilterSmem smem[UNF_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, img = blockIdx.x * UNF_WARPS + warp;
  if (img >= n || status[img] != YG_PNG_OK) return;   // warp-uniform
  UnfilterSmem& s = smem[warp];
  const long long pitch = (long long)W + 1, cap = (long long)H * pitch;
  const uint8_t* f = scratch + (long long)img * cap;
  uint8_t* o = out + (long long)img * H * W;
  unsigned long long sa = 0, sb = 0;   // Adler-32 partial sums: sum b_i and sum (cap - i) b_i
  for (int r0 = 0; r0 < H; r0 += 32) {
    const int nrows = min(32, H - r0);
    const bool row_ok = lane < nrows;
    const long long rbase = (long long)(r0 + lane) * pitch;
    const int ft = row_ok ? f[rbase] : 0;
    if (__any_sync(0xffffffffu, ft > 4)) {
      if (lane == 0) set_status(status, img, YG_PNG_BAD_FILTER);
      return;
    }
    if (row_ok) {
      sa += ft;
      sb += (unsigned long long)(cap - rbase) * ft;
    }
    uint32_t left = 0;
    for (int c0 = 0; c0 < W; c0 += UNF_STRIP) {
      const int sw = min(UNF_STRIP, W - c0);
      for (int k = 0; k < nrows; ++k) {
        const long long rb = (long long)(r0 + k) * pitch + 1 + c0;
        for (int j = lane; j < sw; j += 32) {
          const uint32_t v = f[rb + j];
          s.fin[k][j] = (uint8_t)v;
          sa += v;
          sb += (unsigned long long)(cap - rb - j) * v;
        }
      }
      for (int j = lane; j <= sw; j += 32)
        s.prev[j] = (r0 > 0 && c0 + j >= 1) ? o[(long long)(r0 - 1) * W + c0 - 1 + j] : 0;
      __syncwarp();
      uint32_t last = left, upprev = 0;
      for (int t = 0; t < sw + nrows - 1; ++t) {
        const uint32_t up = __shfl_up_sync(0xffffffffu, last, 1);
        const int j = t - lane;
        if (row_ok && j >= 0 && j < sw) {
          const uint32_t b = lane == 0 ? s.prev[j + 1] : up, c = lane == 0 ? s.prev[j] : upprev;
          const uint32_t x = unfilter_byte(ft, s.fin[lane][j], left, b, c);
          s.fout[lane][j] = (uint8_t)x;
          left = last = x;
        }
        upprev = up;
      }
      __syncwarp();
      for (int k = 0; k < nrows; ++k) {
        uint8_t* ro = o + (long long)(r0 + k) * W + c0;
        for (int j = lane; j < sw; j += 32) ro[j] = s.fout[k][j];
      }
      __syncwarp();
      sa %= ADLER_MOD;
      sb %= ADLER_MOD;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    sa += __shfl_xor_sync(0xffffffffu, sa, off);
    sb += __shfl_xor_sync(0xffffffffu, sb, off);
  }
  const uint32_t A = (uint32_t)((1 + sa) % ADLER_MOD), B = (uint32_t)(((unsigned long long)cap % ADLER_MOD + sb) % ADLER_MOD);
  if (lane == 0 && ((B << 16) | A) != adler[img]) set_status(status, img, YG_PNG_BAD_ADLER);
}

}  // namespace yg
using namespace yg;

extern "C" size_t yg_png_gray8_workspace(int n, int H, int W, long long stream_bytes) {
  if (n < 0 || H < 1 || W < 1 || stream_bytes < 0) return 0;
  return (size_t)png_layout(n, H, W, stream_bytes).total;
}

extern "C" int yg_png_decode_gray8(const void* files, long long files_bytes, const yg_png_chunk* chunks,
                                   const yg_png_image* images, int n, int H, int W, unsigned char* out, int* status,
                                   void* workspace, size_t ws_bytes, void* stream) {
  YG_CHECK_ARG(n >= 0 && H >= 1 && W >= 1 && files_bytes >= 0, "png_decode_gray8: bad sizes n=%d H=%d W=%d", n, H, W);
  if (n == 0) return YG_OK;
  YG_CHECK_ARG(files && chunks && images && out && status && workspace, "png_decode_gray8: null pointer");
  YG_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 15) == 0 && (reinterpret_cast<uintptr_t>(chunks) & 7) == 0 &&
                   (reinterpret_cast<uintptr_t>(images) & 7) == 0 && (reinterpret_cast<uintptr_t>(status) & 3) == 0,
               "png_decode_gray8: workspace must be 16-byte aligned, chunks / images 8-byte, status 4-byte");
  const PngLayout l = png_layout(n, H, W, 0);
  YG_CHECK_ARG((long long)ws_bytes >= l.total, "png_decode_gray8: workspace of %zu bytes is smaller than %lld", ws_bytes,
               l.total);
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  const long long cap = (long long)H * (W + 1), stream_bytes = (long long)ws_bytes - l.streams;
  YG_CUDA(cudaMemsetAsync(status, 0, sizeof(int) * n, st));
  png_gather_crc_kernel<<<n, 32 * GATHER_WARPS, 0, st>>>((const uint8_t*)files, files_bytes, chunks, images,
                                                         ws + l.streams, stream_bytes, status);
  YG_LAUNCH_CHECK("png_gather_crc");
  png_inflate_kernel<<<cdiv(n, INF_WARPS), 32 * INF_WARPS, 0, st>>>(ws + l.streams, images, n, cap, ws + l.scratch,
                                                                    (uint32_t*)(ws + l.aux), status);
  YG_LAUNCH_CHECK("png_inflate");
  png_unfilter_kernel<<<cdiv(n, UNF_WARPS), 32 * UNF_WARPS, 0, st>>>(ws + l.scratch, n, H, W,
                                                                     (const uint32_t*)(ws + l.aux), out, status);
  YG_LAUNCH_CHECK("png_unfilter");
  return YG_OK;
}
