// tcgen05 implicit-GEMM convolution engine for sm_100a (bf16 NHWC activations, fp32 accumulate).
//
// One persistent, warp-specialised kernel serves fprop and dgrad of the 3x3 convolutions and the 1x1 head
// (replacing cuDNN fprop/dgrad dispatched by nn.Conv2d, /root/reference/yogo/model_defns.py:34-64):
//   GEMM view   D[128 pixels x BN channels] += A[128 pixels x KC] * B[BN x KC]^T  per (tap, K chunk)
//   A operand   4-D tiled TMA maps over the NHWC tensor, OOB zero fill = the conv padding.  Two box schemes:
//               * 2-D halo boxes (weights resident): the tile is 16 x 8 pixels, ONE (16+2) x (8+2) box per K chunk; a tap
//                 (r, s) is a descriptor start offset of r * box_cols + s pixel rows (the swizzle is a function of the
//                 absolute shared-memory address), SBO = the box row pitch;
//               * per-filter-column boxes (streamed weights): the tile is 8 x 16 pixels, one (8+2) x 16 box per filter
//                 column, the three filter rows reuse it with row offsets of 16 pixels.
//               Stride-2 fprop reads four parity sub-grids of the input (one tensor map each); stride-2 dgrad runs as four
//               (or, with folded column pairs, two) output-parity classes; small-channel stride-1 layers are W-folded.
//   B operand   packed bf16 weights [tap][N][K] through a 3-D tensor map; resident in shared memory whenever they fit.
//   MMA         tcgen05.mma.kind::f16, M = 128, N = BN <= 256, up to four accumulators in TMEM so the epilogue of tile i
//               overlaps the MMAs of tiles i+1..; the producer and MMA warps issue warp-uniformly (elect.sync predicate
//               inside the asm).  128 -> 128 layers run as CTA pairs: cta_group::2, M = 256, half of B per CTA.
//   epilogue    tcgen05.ld 32x32b -> registers -> bias / folded BN / activation / Dropout2d scale / sign mask (fwd),
//               activation backward from the sign mask or the saved tensor, optional BN sums (dgrad), 16-byte bf16
//               stores; straight-line 32-column fast paths for the common flavours; the YOGO head transform.
// Warp roles (352 threads): warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2-9 epilogue, warp 10 idle (see
// conv_tc_kernel).  The weight-gradient kernel (wgrad_tc_kernel, below) has its own header.
#include "common.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <map>
#include <mutex>

namespace yg {

constexpr int TC_TH = 8, TC_TW = 16;          // output tile (pixels), M = 128
// conv_tc_kernel: 1 producer warp + 1 MMA warp + 8 epilogue warps + 1 idle warp
constexpr int TC_MAX_GROUPS = 9, TC_MAX_TAPS = 9, TW_MAX_TAPS = 3;
// MMA issue list bounds: W-folded layers have a folded K <= 256 (see fold_factor), i.e. at most 16 K steps of 16 per tap:
// 9 taps x 16 = 144 MMAs per tile in at most 16 per-chunk lists; every other layer has one list of at most 9 taps x 4 K steps
constexpr int TC_MAX_LISTS = 16, TC_MAX_MMAS = 144;
constexpr int TC_SMEM_BUDGET = 227 * 1024 - 14 * 1024;
constexpr uint32_t TC_SPIN_LIMIT = 1u << 24;   // bounded mbarrier spin: trap instead of hanging the GPU

struct TcMaps {
  CUtensorMap a[4];
  CUtensorMap b;
};

struct TcGroup {
  int map, dh, dw, rows, ntaps;
  int cols;               // box width in pixels (0 = TC_TW: legacy per-filter-column boxes)
  int ro[TC_MAX_TAPS];    // A row offset (in tile rows) of each tap inside the halo box
  int co[TC_MAX_TAPS];    // A column offset (pixels) of each tap inside the halo box (2-D halo boxes)
  int widx[TC_MAX_TAPS];  // weight slice index
  unsigned kmask[TC_MAX_TAPS];  // bit kk: global 16-wide K step kk of this tap has non-zero weights (W-folded convs)
};

struct TcClass {   // one output-parity class of a stride-2 dgrad (or the whole problem when ncls == 1)
  int g0, ng, gpi;          // its groups: p.g[g0 .. g0+ng), merged gpi at a time into one pipeline item
  int TSH, TSW, oh0, ow0;   // tile-space extent and output offset
};

struct TcParams {
  int N, tiles_h, tiles_w, n_ntiles, total_tiles;
  int TH, TW, tw_shift;             // output tile in pixels (8 x 16 legacy, 16 x 8 with 2-D halo boxes), log2(TW)
  int bt_stride;                    // weight-tile slots per group in a streamed-weight stage
  int cta2;                         // CTA pairs (cta_group::2): M = 256 per MMA, each CTA holds BN/2 rows of every weight tile
  int ncls, cls_rot;                // classes and the rotation period max(1, grid / ncls) (see tile_class)
  unsigned long long fd_ncls, fd_rot, fd_nnt, fd_tw, fd_th, fd_ocr;   // ceil(2^32 / d): division by multiply-high (decode_tile)
  TcClass cls[4];
  int b_resident, resb_bytes;     // all weight tiles live in smem for the whole kernel
  int OH, OW, OC, osh, osw;       // output tensor (NHWC) and tile-space -> output strides (rows, columns)
  int OCr;                        // real channel count (OC / W-fold factor): per-channel arrays are indexed modulo OCr
  int BN, kchunks, nstages, nacc;
  int a_box_bytes, b_stage_bytes;   // bytes reserved per A box / per stage for streamed weight tiles
  int ntaps_total;                  // weight slices in the packed weight tensor (9 for 3x3, 1 for 1x1)
  int a_stage_bytes, b_tap_bytes, tmem_cols;
  TcGroup g[TC_MAX_GROUPS];
  void* out;
  // forward epilogue
  const float* scale; const float* shift; int act; const float* dropscale; double* stats; void* preact;
  // prediction head (1x1 conv + YOGO output transform fused into the forward epilogue, see head_fwd_tc)
  float* head_out; float* head_traw; const float* head_cxs; const float* head_cys;
  float head_aw, head_ah, head_wm, head_hm; int head_D, head_inf;
  void* actmask_out;        // forward: sign bits of the pre-activation (see yg_fwd_epilogue.actmask)
  const void* actmask_in;   // backward: the producer's sign bits, replaces `saved` for LeakyReLU without BN
  // backward epilogue
  const void* saved; const float* bn_scale; const float* bn_shift; const float* bn_mean; const float* bn_invstd;
  double* bn_sums;
  int* error_flag;
  // MMA issue list (host-built, read through the constant bank = uniform loads): one word per MMA, A offset | B offset << 16
  // inside a stage in 16-byte descriptor units, K steps with structurally zero weights of W-folded layers left out, so the
  // issue loop is load - add - issue.  flat_rng[L][g] = first MMA of group g in list L; W-folded layers have one list per
  // K chunk (L = kc), everything else one list for all chunks.  a_hi[g]: high descriptor word of group g's A operand
  // (SBO = box row pitch: the parity boxes of one stride-2 pipeline item differ in width).
  int flat_perkc;
  int flat_rng[TC_MAX_LISTS][TC_MAX_GROUPS + 1];
  uint32_t flat_ab[TC_MAX_MMAS];
  uint32_t a_hi[TC_MAX_GROUPS];
  int io_f32;  // the epilogue reads `saved` and writes `out` / `preact` as fp32 (split-bf16 "x3" convolutions of fp32 tensors, see x3.cu)
  int debug;   // profiling knobs (tools/bench_conv.py): 1 = no global stores, 2 = no MMA issue, 4 = epilogue skips TMEM loads and math, 8 = no TMA loads, 16 = MMA-warp cycle counters -> g_tc_dbg
};

// cycle counters of the MMA warp, one row of 8 per CTA (debug bit 16): wait tempty, wait full, issue, commit, rest
__device__ unsigned long long g_tc_dbg[256 * 16];   // per CTA: 0-5 MMA warp, 8-13 first epilogue warp

// Output-parity class of a tile.  Sibling classes of one spatial tile are neighbours in the tile order (they
// share dz and saved-activation lines in L2); the class of slot c rotates with the spatial index so that a
// persistent CTA, whose stride gridDim.x is normally a multiple of ncls, cycles through all classes instead
// of being stuck with the cheapest (1 tap) or the most expensive (4 taps) one.
__device__ __forceinline__ int fdiv(int n, unsigned long long m) {   // n / d for n * d < 2^32, m = ceil(2^32 / d)
  return (int)(((unsigned long long)(unsigned)n * m) >> 32);
}
__device__ __forceinline__ int tile_class(const TcParams& p, int tile) {
  if (p.ncls == 1) return 0;
  const int sp = fdiv(tile, p.fd_ncls), c = tile - sp * p.ncls;
  const int x = c + fdiv(sp, p.fd_rot);
  return x - fdiv(x, p.fd_ncls) * p.ncls;
}
// tile index -> (class, N tile, tile column, tile row, image); the class is the fastest index.  Division by multiply-high:
// every role decodes every tile, and four runtime integer divisions cost several hundred cycles of a single warp.
// The padding tile of a CTA pair decodes to n >= N: all its loads are out of bounds (zero fill) and the epilogue stores
// nothing.
__device__ __forceinline__ void decode_tile(const TcParams& p, int tile, int& cls, int& nt, int& tw, int& th, int& n) {
  cls = tile_class(p, tile);
  int t = fdiv(tile, p.fd_ncls);
  int q = fdiv(t, p.fd_nnt); nt = t - q * p.n_ntiles; t = q;
  q = fdiv(t, p.fd_tw); tw = t - q * p.tiles_w; t = q;
  q = fdiv(t, p.fd_th); th = t - q * p.tiles_h; n = q;
}

// ------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n.reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int* error_flag, int code) {
  uint32_t spins = 0;
  while (!mbar_try(bar, parity)) {
    if (++spins > TC_SPIN_LIMIT) {
      if (error_flag) atomicExch(error_flag, code);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// same, descriptors given as (low word, shared high word): the issuing thread only ever adds to the low words
__device__ __forceinline__ void umma_bf16_lh(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc,
                                             uint32_t accum) {
  asm volatile(
      "{\n.reg .pred p;\n.reg .b64 da, db;\nsetp.ne.b32 p, %5, 0;\n"
      "mov.b64 da, {%1, %4};\nmov.b64 db, {%2, %4};\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n}\n"
      ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(hi), "r"(accum)
      : "memory");
}
// same with separate high words (the MN-major wgrad operands have different strides / swizzles)
__device__ __forceinline__ void umma_bf16_lh2(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                              uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n.reg .pred p;\n.reg .b64 da, db;\nsetp.ne.b32 p, %6, 0;\n"
      "mov.b64 da, {%1, %2};\nmov.b64 db, {%3, %4};\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n}\n"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accum)
      : "memory");
}
// ---- "one elected lane issues" variants: executed by the whole (converged) warp with the election result as a
// predicate inside the asm.  With warp-uniform operands ptxas emits the bare uniform-datapath instruction; issuing
// from an `if (lane == 0)` branch instead costs an ELECT / BRA.U.ANY waterfall loop around every instruction
// (~90 cycles per tcgen05.mma measured, more than the 64 cycles a 128x128x16 MMA takes to execute).
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}" : "=r"(pred));
  return pred;
}
__device__ __forceinline__ void umma_bf16_lh_p(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc,
                                               uint32_t accum, uint32_t leader) {
  asm volatile(
      "{\n.reg .pred p, q;\n.reg .b64 da, db;\nsetp.ne.b32 p, %5, 0;\nsetp.ne.b32 q, %6, 0;\n"
      "mov.b64 da, {%1, %4};\nmov.b64 db, {%2, %4};\n"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n}\n"
      ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(hi), "r"(accum), "r"(leader)
      : "memory");
}
// v * 0.01 where `bit` of `word` is clear (LeakyReLU backward from the producer's sign bits), v otherwise
__device__ __forceinline__ float mul_slope_if_clear(float v, uint32_t word, uint32_t bit) {
  asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.eq.u32 p, t, 0;\n\t@p mul.f32 %0, %0, 0f3C23D70A;\n\t}"
      : "+f"(v) : "r"(word), "r"(bit));
  return v;
}

__device__ __forceinline__ void umma_bf16_lh2_p(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                uint32_t idesc, uint32_t accum, uint32_t leader) {
  asm volatile(
      "{\n.reg .pred p, q;\n.reg .b64 da, db;\nsetp.ne.b32 p, %6, 0;\nsetp.ne.b32 q, %7, 0;\n"
      "mov.b64 da, {%1, %2};\nmov.b64 db, {%3, %4};\n"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n}\n"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accum), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void umma_commit_p(uint64_t* bar, uint32_t leader) {
  asm volatile(
      "{\n.reg .pred q;\nsetp.ne.b32 q, %1, 0;\n"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n}\n"
      ::"r"(smem_u32(bar)), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_p(uint64_t* bar, uint32_t bytes, uint32_t leader) {
  asm volatile("{\n.reg .pred q;\nsetp.ne.b32 q, %2, 0;\n@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n}\n"
               ::"r"(smem_u32(bar)), "r"(bytes), "r"(leader) : "memory");
}
__device__ __forceinline__ void mbar_arrive_p(uint64_t* bar, uint32_t leader) {
  asm volatile("{\n.reg .pred q;\nsetp.ne.b32 q, %1, 0;\n@q mbarrier.arrive.shared::cta.b64 _, [%0];\n}\n"
               ::"r"(smem_u32(bar)), "r"(leader) : "memory");
}
__device__ __forceinline__ void tma_load_4d_p(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                              int c3, uint32_t leader) {
  asm volatile(
      "{\n.reg .pred q;\nsetp.ne.b32 q, %7, 0;\n"
      "@q cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n}\n"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_p(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                              uint32_t leader) {
  asm volatile(
      "{\n.reg .pred q;\nsetp.ne.b32 q, %6, 0;\n"
      "@q cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n}\n"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// wait for the TMEM loads AND tie the destination registers to the wait, so that no use of them can be scheduled
// above it (the loads complete asynchronously; plain register reads have no other dependency on the wait)
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :: "memory");
}
// 32-byte global store (sm_100: STG.256): a pixel row's 64 bytes of an epilogue iteration leave as two full sectors
// instead of four 16-byte pieces of them
__device__ __forceinline__ void st_global_256(void* p, const uint32_t* v) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void ld_global_nc_256(const void* p, uint4& lo, uint4& hi) {
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w) : "l"(p));
}
// 1 / (1 + 2^(-x log2 e)) on the SFU: one ex2.approx and one rcp.approx (x -> -inf gives 1 / inf = 0, x -> +inf gives 1)
__device__ __forceinline__ float fast_sigmoid(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.f + e));
  return r;
}
__device__ __forceinline__ void tmem_ld_wait32(uint32_t (&a)[16], uint32_t (&b)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                 "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                 "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]),
                 "+r"(b[8]), "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15])
               :: "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- CTA pairs (cta_group::2): two CTAs of a cluster execute one M = 256 MMA; each holds its own 128 A rows and HALF of B.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {   // shared::cluster address of saddr in CTA `rank`
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// TMA loads of a CTA pair: data lands in the issuing CTA, the transaction bytes are signalled on the LEADER's barrier
__device__ __forceinline__ void tma2_load_4d_p(void* dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1,
                                               int c2, int c3, uint32_t leader) {
  asm volatile(
      "{\n.reg .pred q;\nsetp.ne.b32 q, %7, 0;\n"
      "@q cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n}\n"
      ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tma2_load_3d(void* dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16_lh2_p(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                 uint32_t idesc, uint32_t accum, uint32_t leader) {
  asm volatile(
      "{\n.reg .pred p, q;\n.reg .b64 da, db;\nsetp.ne.b32 p, %6, 0;\nsetp.ne.b32 q, %7, 0;\n"
      "mov.b64 da, {%1, %2};\nmov.b64 db, {%3, %4};\n"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n}\n"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accum), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void umma2_commit_p(uint64_t* bar, uint32_t leader) {   // arrives on `bar` of BOTH CTAs
  asm volatile(
      "{\n.reg .pred q;\n.reg .b16 m;\nsetp.ne.b32 q, %1, 0;\nmov.b16 m, 3;\n"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n}\n"
      ::"r"(smem_u32(bar)), "r"(leader)
      : "memory");
}

// K-major, swizzled shared-memory matrix descriptor (sm_100 UMMA).  bits: start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout [61,64) (2 = SWIZZLE_128B, 4 = 64B, 6 = 32B).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}

// sum over the 32 lanes (= 32 pixels) of 16 per-lane values; afterwards lane l holds the total of
// value index (l & 15) in v[0].  31 shuffles instead of 80.
__device__ __forceinline__ float lane_transpose_reduce16(float (&v)[16], int lane) {
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], 16);
#pragma unroll
  for (int step = 8, n = 16; step >= 1; step >>= 1, n >>= 1) {
    const bool upper = (lane & step) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float send = upper ? v[i] : v[i + n / 2];
      const float keep = upper ? v[i + n / 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, step);
    }
  }
  return v[0];
}

__device__ __forceinline__ float round_bf16(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// ------------------------------------------------------------------------------------------ kernel
// 352 threads, of which warp 10 has no role: with a 320-thread bound ptxas allocates the 168 registers differently and the
// dgrad instantiations spill more (52 instead of 40 bytes, 60 instead of 56 for CTA pairs; nvcc 12.9 -Xptxas -v).
template <int KC, int MODE, int CTA2 = 0>
__global__ void __launch_bounds__(352, 1)
conv_tc_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcParams p) {
  constexpr int NTHREADS = 352;
  constexpr uint32_t ROW_BYTES = KC * 2;
  constexpr uint32_t SBO = 8 * ROW_BYTES;
  constexpr uint32_t LAYOUT = KC == 64 ? 2u : (KC == 32 ? 4u : 6u);

  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // SWIZZLE_128B operands need 1024-byte aligned stage bases: align by hand, do not trust the attribute
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int stage_bytes = p.a_stage_bytes + (p.b_resident ? 0 : p.b_stage_bytes);
  unsigned char* resb = smem + (size_t)p.nstages * stage_bytes;
  unsigned char* tail = resb + p.resb_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + 16;
  uint64_t* tfull_bar = empty_bar + 16;
  uint64_t* tempty_bar = tfull_bar + 4;
  uint64_t* resb_bar = tempty_bar + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(resb_bar + 2);
  float* s_stat = reinterpret_cast<float*>(tmem_slot + 4);  // [2][256]
  float* s_const = s_stat + 2 * 256;                        // [4][512] per-channel epilogue constants
  float* s_ds = s_const + 4 * 512;                          // [2][256] Dropout2d scales of the image each epilogue group works on

  // warp index through a shuffle: the compiler then knows that role dispatch and everything derived from kernel
  // parameters inside a role is warp-uniform (uniform registers feed UTCHMMA / UTMALDG directly)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int BN = p.BN;
  const long long t_kernel0 = (p.debug & 16) ? clock64() : 0;

  // CTA pair: rank 0 (leader) issues the MMAs for both; every barrier the MMA warp waits on lives in the leader
  const uint32_t cta_rank = CTA2 ? cluster_ctarank() : 0u;
  const int total_tiles = CTA2 ? ((p.total_tiles + 1) & ~1) : p.total_tiles;   // both CTAs of a pair run the same iterations
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) prefetch_tmap(&maps.a[i]);
    prefetch_tmap(&maps.b);
    for (int i = 0; i < p.nstages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    // the two epilogue warp groups alternate tiles (4 arrivals per accumulator and CTA); only with several N tiles per CTA and
    // fused statistics do all eight warps share every tile (they then flush the statistics together)
    const bool alt0 = !(p.n_ntiles > 1 && ((MODE == 0 ? p.stats : p.bn_sums) != nullptr));
    for (int i = 0; i < p.nacc; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], (alt0 ? 4 : 8) * (CTA2 ? 2 : 1)); }
    mbar_init(&resb_bar[0], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (p.b_resident && !CTA2) {
      // every (tap, K chunk) weight tile is fetched once and stays in shared memory
      mbar_expect_tx(&resb_bar[0], (uint32_t)(p.ntaps_total * p.kchunks * p.b_tap_bytes));
      for (int tap = 0; tap < p.ntaps_total; ++tap)
        for (int kc = 0; kc < p.kchunks; ++kc)
          tma_load_3d(resb + (size_t)(tap * p.kchunks + kc) * p.b_tap_bytes, &maps.b, &resb_bar[0], kc * KC, 0, tap);
    }
  }
  if (warp == 1) { if (CTA2) tmem_alloc2(tmem_slot, (uint32_t)p.tmem_cols); else tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols); }
  // epilogue constants and statistics accumulators (the N tile is fixed per CTA only when n_ntiles == 1,
  // so constants are indexed by absolute channel and reloaded per tile below when needed)
  for (int i = threadIdx.x; i < 2 * 256; i += NTHREADS) s_stat[i] = 0.f;
  for (int i = threadIdx.x; i < p.OC; i += NTHREADS) {
    const int ir = i % p.OCr;
    if (MODE == 0) {
      s_const[i] = p.scale ? p.scale[ir] : 1.f;
      s_const[512 + i] = (p.shift && (p.head_D == 0 || i < p.head_D)) ? p.shift[ir] : 0.f;
    } else if (p.bn_scale) {
      s_const[i] = p.bn_scale[ir];
      s_const[512 + i] = p.bn_shift[ir];
      s_const[1024 + i] = p.bn_mean[ir];
      s_const[1536 + i] = p.bn_invstd[ir];
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (CTA2) {
    cluster_sync_all();   // the peer's barriers exist before anything is signalled on them
    if (warp == 0 && lane == 0) {
      // resident weights of a pair: each CTA keeps BN/2 rows of every tile; all bytes are counted on the leader's barrier
      const uint32_t lbar = map_to_cta(smem_u32(&resb_bar[0]), 0u);
      if (cta_rank == 0) mbar_expect_tx(&resb_bar[0], 2u * (uint32_t)(p.ntaps_total * p.kchunks * p.b_tap_bytes));
      for (int tap = 0; tap < p.ntaps_total; ++tap)
        for (int kc = 0; kc < p.kchunks; ++kc)
          tma2_load_3d(resb + (size_t)(tap * p.kchunks + kc) * p.b_tap_bytes, &maps.b, lbar, kc * KC,
                       (int)cta_rank * (BN / 2), tap);
    }
  }


  if (warp == 0) {
    // ===================================================================== TMA producer
    // the whole warp runs the loop (uniform control flow), one elected lane issues
    const uint32_t leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    const int nstages = p.nstages, kchunks = p.kchunks, b_resident = p.b_resident;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      int ci, nt, tw, th, n;
      decode_tile(p, tile, ci, nt, tw, th, n);
      const TcClass& C = p.cls[ci];
      const int cg0 = C.g0, cg1 = C.g0 + C.ng, gpi = C.gpi;
      for (int kc = 0; kc < kchunks; ++kc) {
        for (int g0 = cg0; g0 < cg1; g0 += gpi) {
          mbar_wait(&empty_bar[stage], phase ^ 1u, p.error_flag, 1);
          unsigned char* sa = smem + (size_t)stage * stage_bytes;
          unsigned char* sb = sa + p.a_stage_bytes;
          if (p.debug & 8) {
            mbar_arrive_p(&full_bar[stage], leader);
            if (++stage == nstages) { stage = 0; phase ^= 1u; }
            continue;
          }
          uint32_t bytes = 0;
          for (int gi = g0; gi < g0 + gpi; ++gi)
            bytes += (uint32_t)(p.g[gi].rows * p.g[gi].cols * (int)ROW_BYTES + (b_resident ? 0 : p.g[gi].ntaps * p.b_tap_bytes));
          if (CTA2) {
            // both CTAs load their own A boxes; the bytes of both are expected on the leader's barrier
            if (cta_rank == 0) mbar_expect_tx_p(&full_bar[stage], 2u * bytes, leader);
            const uint32_t lbar = map_to_cta(smem_u32(&full_bar[stage]), 0u);
            for (int gi = g0; gi < g0 + gpi; ++gi) {
              const TcGroup& g = p.g[gi];
              tma2_load_4d_p(sa + (size_t)(gi - g0) * p.a_box_bytes, &maps.a[g.map], lbar, kc * KC,
                             tw * p.TW + g.dw, th * p.TH + g.dh, n, leader);
            }
            if (++stage == nstages) { stage = 0; phase ^= 1u; }
            continue;
          }
          mbar_expect_tx_p(&full_bar[stage], bytes, leader);
          for (int gi = g0; gi < g0 + gpi; ++gi) {
            const TcGroup& g = p.g[gi];
            tma_load_4d_p(sa + (size_t)(gi - g0) * p.a_box_bytes, &maps.a[g.map], &full_bar[stage], kc * KC,
                          tw * p.TW + g.dw, th * p.TH + g.dh, n, leader);
            if (!b_resident)
              for (int tp = 0; tp < g.ntaps; ++tp)
                tma_load_3d_p(sb + (size_t)((gi - g0) * p.bt_stride + tp) * p.b_tap_bytes, &maps.b, &full_bar[stage],
                              kc * KC, nt * BN, g.widx[tp], leader);
          }
          if (++stage == nstages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    // instruction descriptor: D=f32 [4,6)=1, A=bf16 [7,10)=1, B=bf16 [10,13)=1, K-major A/B, N>>3 [17,23), M>>4 [24,29)
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | (((CTA2 ? 256u : 128u) >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    if (p.b_resident && cta_rank == 0) mbar_wait(&resb_bar[0], 0, p.error_flag, 5);
    // descriptors differ only in their 14-bit start-address field (16-byte units): build one and add offsets
    const uint64_t desc0 = umma_desc(smem_u32(smem), SBO, LAYOUT);
    const uint32_t desc_hi = (uint32_t)(desc0 >> 32), desc0_lo = (uint32_t)desc0;
    const uint32_t bres0_lo = (uint32_t)umma_desc(smem_u32(resb), SBO, LAYOUT);
    const uint32_t stage_units = (uint32_t)stage_bytes >> 4, a_units = (uint32_t)p.a_stage_bytes >> 4;
    const uint32_t tap_units = (uint32_t)p.b_tap_bytes >> 4;
    const int b_resident = p.b_resident, kchunks = p.kchunks, nstages = p.nstages, nacc = p.nacc;
    const bool prof = (p.debug & 16) != 0;
    const uint32_t leader = elect_one();
    long long c_tempty = 0, c_full = 0, c_issue = 0, c_commit = 0, c_rest = 0, c_items = 0, tprev = clock64();
    const long long t_loop0 = tprev;
    for (int tile = blockIdx.x; tile < total_tiles && cta_rank == 0; tile += gridDim.x) {   // pair: the leader issues
      long long ta = 0;
      if (prof) ta = clock64();
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1u, p.error_flag, 2);
      if (prof) { const long long tb = clock64(); c_tempty += tb - ta; c_rest += ta - tprev; tprev = tb; }
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
      const TcClass& C = p.cls[tile_class(p, tile)];
      const int cg0 = C.g0, cg1 = C.g0 + C.ng, gpi = C.gpi;
      uint32_t started = 0;   // 0 until the first MMA of this tile has been issued (overwrite vs accumulate)
      for (int kc = 0; kc < kchunks; ++kc) {
        for (int g0 = cg0; g0 < cg1; g0 += gpi) {
          long long t0 = 0, t1 = 0, t2 = 0;
          if (prof) t0 = clock64();
          mbar_wait(&full_bar[stage], phase, p.error_flag, 3);
          tc_fence_after();
          if (prof) t1 = clock64();
          // whole warp, uniform control flow; the elected lane issues (predicate inside the asm)
          const uint32_t ast = desc0_lo + (uint32_t)stage * stage_units;
          const uint32_t bst = b_resident ? bres0_lo + (uint32_t)kc * tap_units : ast + a_units;
          const int L = p.flat_perkc ? kc : 0;
          for (int gi = g0; gi < g0 + gpi; ++gi) {
            const uint32_t a_hi = p.a_hi[gi];
            const int i0 = p.flat_rng[L][gi], i1 = (p.debug & 2) ? i0 : p.flat_rng[L][gi + 1];
#pragma unroll 4
            for (int i = i0; i < i1; ++i) {
              const uint32_t ab = p.flat_ab[i];
              if (CTA2) umma2_bf16_lh2_p(d_tmem, ast + (ab & 0xFFFFu), a_hi, bst + (ab >> 16), desc_hi, idesc, started, leader);
              else umma_bf16_lh2_p(d_tmem, ast + (ab & 0xFFFFu), a_hi, bst + (ab >> 16), desc_hi, idesc, started, leader);
              started = 1u;
            }
          }
          if (prof) t2 = clock64();
          if (CTA2) {
            umma2_commit_p(&empty_bar[stage], leader);                                 // both CTAs' slots and accumulators
            if (kc == kchunks - 1 && g0 + gpi >= cg1) umma2_commit_p(&tfull_bar[acc], leader);
          } else {
            umma_commit_p(&empty_bar[stage], leader);                                  // frees the smem slot when the MMAs retire
            if (kc == kchunks - 1 && g0 + gpi >= cg1) umma_commit_p(&tfull_bar[acc], leader);  // accumulator complete
          }
          if (prof) {
            const long long t3 = clock64();
            c_rest += t0 - tprev; c_full += t1 - t0; c_issue += t2 - t1; c_commit += t3 - t2; tprev = t3; ++c_items;
          }
          if (++stage == nstages) { stage = 0; phase ^= 1u; }
        }
      }
      if (++acc == nacc) { acc = 0; acc_phase ^= 1u; }
    }
    if (prof && lane == 0 && blockIdx.x < 256) {
      unsigned long long* d = g_tc_dbg + blockIdx.x * 16;
      d[0] = c_tempty; d[1] = c_full; d[2] = c_issue; d[3] = c_commit; d[4] = c_rest; d[5] = c_items;
      d[6] = (unsigned long long)(t_loop0 - t_kernel0); d[7] = (unsigned long long)(clock64() - t_kernel0);   // loop entry, loop exit
    }
  } else if (warp < 10) {
    // ===================================================================== epilogue (8 warps)
    // warp w may only touch TMEM lanes [32*(w&3), +32).  The eight warps form two groups of four (one warp per lane
    // quarter); the groups ALTERNATE TILES, so the fixed per-tile work (decode, barrier waits, hand-back) is paid by four warps
    // instead of eight - the epilogue, not the tensor pipe, bounds most layers.
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int m = q * 32 + lane;       // row of the tile = pixel
    const int hl = m >> p.tw_shift, wl = m & (p.TW - 1);
    int acc_it = 0;
    uint32_t acc_phase_it = 0;
    int it = 0, ds_n = -1;
    bf16* out = reinterpret_cast<bf16*>(p.out);
    const float* s_k0 = s_const;             // fwd: scale      bwd: bn_scale
    const float* s_k1 = s_const + 512;       // fwd: shift      bwd: bn_shift
    const float* s_k2 = s_const + 1024;      //                 bwd: bn_mean
    const float* s_k3 = s_const + 1536;      //                 bwd: bn_invstd
    const bool has_bn = p.bn_scale != nullptr;
    // parameters used per chunk live in registers: the parameter block is larger than the fastest constant cache
    // level and every LDC in the chunk loop is a potential miss on the critical path of the accumulator hand-back
    const float* const e_dropscale = p.dropscale;
    const void* const e_saved = p.saved;
    double* const e_stats = p.stats;
    double* const e_bn_sums = p.bn_sums;
    void* const e_preact = p.preact;
    void* const e_mask_out = p.actmask_out;
    float* const e_head_out = p.head_out;
    const bool e_has_scale = p.scale != nullptr;
    const int e_act = p.act, e_OC = p.OC, e_OH = p.OH, e_OW = p.OW, e_dbg = p.debug, e_nnt = p.n_ntiles, e_OCr = p.OCr;
    const int e_TH = p.TH, e_TW = p.TW, e_osh = p.osh, e_osw = p.osw, e_total = p.total_tiles, e_nacc = p.nacc;
    const bool alt = !(e_nnt > 1 && ((MODE == 0 ? (const void*)e_stats : (const void*)e_bn_sums) != nullptr));
    const bool ds_smem = e_dropscale != nullptr && alt && e_OC <= 256;   // else the scales are read through L1 per chunk
    const bool eprof = (p.debug & 16) != 0 && warp == 2;
    long long ec_tfull = 0, ec_ld = 0, ec_pre = 0, ec_math = 0, ec_store = 0, ec_rest = 0, ec_tiles = 0, eprev = clock64();
    const bool io_f32 = p.io_f32 != 0;
    const bool use_mask = MODE == 1 && p.actmask_in && e_act == YG_ACT_LRELU && !has_bn && (BN % 32) == 0 && (e_OC % 32) == 0 && !io_f32;
    // (dgrad fast path: the multiplication order differs from the generic path only by commuting g*ds*slope)
    const bool fast_fwd = MODE == 0 && !io_f32 && !e_head_out && !e_has_scale && !e_stats && !e_preact && (BN % 64) == 0 &&
                          (e_act == YG_ACT_LRELU || e_act == YG_ACT_NONE) && !(p.debug & 4) && out != nullptr;
    const bool fast_bwd = MODE == 1 && use_mask && !e_bn_sums && (BN % 64) == 0 && !(p.debug & 4);
    // SiLU flavours (silu_model): forward = bias + SiLU (+ Dropout2d) with the bf16 pre-activation saved for backward,
    // backward = SiLU'(saved pre-activation, or saved raw output through the BatchNorm affine) without the BN sums
    const bool fast_fwd_silu = MODE == 0 && !io_f32 && !e_head_out && !e_has_scale && !e_stats && e_preact && e_act == YG_ACT_SILU &&
                               alt && (BN % 32) == 0 && !(p.debug & 4) && out != nullptr && !e_mask_out;
    const bool fast_bwd_silu = MODE == 1 && !io_f32 && !use_mask && e_saved && e_act == YG_ACT_SILU && !e_bn_sums && alt &&
                               (BN % 32) == 0 && !(p.debug & 4);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int acc = acc_it;
      const uint32_t acc_phase = acc_phase_it;
      if (++acc_it == e_nacc) { acc_it = 0; acc_phase_it ^= 1u; }
      if (alt && (it & 1) != half) continue;   // the other warp group's tile
      int ci, nt, tw, th, n;
      decode_tile(p, tile, ci, nt, tw, th, n);
      const TcClass& C = p.cls[ci];
      const int a = th * e_TH + hl, b = tw * e_TW + wl;
      const int oh = a * e_osh + C.oh0, ow = b * e_osw + C.ow0;
      const bool valid = a < C.TSH && b < C.TSW && oh < e_OH && ow < e_OW && n < p.N;   // (n >= N: padding tile)
      const long long pix = ((long long)n * e_OH + oh) * e_OW + ow;
      // Dropout2d scales of this image: read through L1 per chunk (16 consecutive channels; folded layers index modulo
      // the real channel count)
      const float* dsrow = e_dropscale ? e_dropscale + (long long)(n < p.N ? n : p.N - 1) * e_OCr : nullptr;
      if (ds_smem && n != ds_n) {
        // stage the row of this image in this group's half of the shared buffer, already expanded to folded channels
        const int tg = (int)threadIdx.x - 64 - half * 128;
        if (half == 0) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory");
        for (int i = tg; i < e_OC; i += 128) s_ds[half * 256 + i] = dsrow[i - fdiv(i, p.fd_ocr) * e_OCr];
        if (half == 0) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory");
        ds_n = n;
      }
      if (MODE == 1 && e_saved && (alt || half == 0) && !use_mask) {
        // pull the saved-activation rows of the tile after next into L2 now: by the time its epilogue runs,
        // the 32-byte operand loads hit L2 instead of paying an HBM round trip per 16-column chunk
        const int tile2 = tile + 2 * (int)gridDim.x;
        if (tile2 < e_total) {
          int ci2, nt2, tw2, th2, n2;
          decode_tile(p, tile2, ci2, nt2, tw2, th2, n2);
          const TcClass& C2 = p.cls[ci2];
          const int a2 = th2 * e_TH + hl, b2 = tw2 * e_TW + wl;
          const int oh2 = a2 * e_osh + C2.oh0, ow2 = b2 * e_osw + C2.ow0;
          if (a2 < C2.TSH && b2 < C2.TSW && oh2 < e_OH && ow2 < e_OW) {
            const int esz = io_f32 ? 2 : 1;   // in units of bf16 elements
            const bf16* row = reinterpret_cast<const bf16*>(e_saved) +
                              ((((long long)n2 * e_OH + oh2) * e_OW + ow2) * e_OC + nt2 * BN) * esz;
            for (int c = 0; c < BN * esz; c += 64)
              asm volatile("prefetch.global.L2 [%0];" ::"l"(row + c));
          }
        }
      }
      // LeakyReLU backward from the producer's sign bits: the BN / 8 bytes of this pixel are requested before the
      // accumulator wait, so their latency hides behind the MMAs (the 16x larger `saved` row never does)
      uint32_t mk[8];
      if (MODE == 1 && use_mask) {
        const uint32_t* mp = reinterpret_cast<const uint32_t*>(p.actmask_in) + ((pix * e_OC + nt * BN) >> 5);
#pragma unroll
        for (int w = 0; w < 8; ++w) mk[w] = (valid && w * 32 < BN) ? __ldg(mp + w) : 0u;
      }
      long long et0 = 0, et1 = 0;
      if (eprof) et0 = clock64();
      mbar_wait(&tfull_bar[acc], acc_phase, p.error_flag, 4);
      tc_fence_after();
      if (eprof) { et1 = clock64(); ec_tfull += et1 - et0; ec_rest += et0 - eprev; eprev = et1; }
      const uint32_t taddr0 = tmem_base + (uint32_t)(acc * BN) + ((uint32_t)(q * 32) << 16);
      // the two warps of a TMEM lane quarter split the 16-column chunks into a lower and an upper contiguous half
      const int nchunks = (e_dbg & 4) ? 0 : BN / 16, nper = (nchunks + 1) >> 1;
      const int jb = alt ? 0 : half * nper;
      const int j_end = alt ? nchunks : min(nchunks, (half + 1) * nper);
      unsigned long long mbits0 = 0ull, mbits1 = 0ull, mbits2 = 0ull, mbits3 = 0ull;   // forward: sign bits of this thread's chunks
      // ---- straight-line fast paths for the common epilogue flavours: 32 columns per iteration, no branches inside,
      // so the compiler can interleave 32 independent element chains (the generic loop below issues at IPC ~0.25)
      if (MODE == 0 && fast_fwd && ((j_end - jb) & 3) == 0) {
        // 64 columns per iteration of the runtime loop, as two unrolled 32-column halves: the sign-mask word of the group
        // leaves as one 8-byte store, no per-chunk bookkeeping (ncu: the previous form spent ~100 of its 350 instructions
        // per 32 columns on loop / select overhead, and the epilogue's issue slots are what bounds the forward layers)
        bf16* orow = out + pix * e_OC + nt * BN;
        unsigned long long* mrow = e_mask_out ? reinterpret_cast<unsigned long long*>(
            reinterpret_cast<unsigned char*>(e_mask_out) + ((pix * e_OC + nt * BN) >> 3)) : nullptr;
        const float slope1 = e_act == YG_ACT_LRELU ? 0.01f : 1.f;
        const float2 slope2 = make_float2(slope1, slope1);
        for (int j = jb; j < j_end; j += 4) {
          unsigned long long mb64 = 0ull;
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const int jq = j + 2 * hh;
            uint32_t ra[16], rb[16];
            tmem_ld16(taddr0 + (uint32_t)(jq * 16), ra);
            tmem_ld16(taddr0 + (uint32_t)(jq * 16 + 16), rb);
            const int c0 = nt * BN + jq * 16;
            // packed fp32 arithmetic (FADD2 / FMUL2: two IEEE operations per issue slot, same results as the scalar
            // forms): the epilogue warps are bound by their issue slots, not by the fp32 pipe
            float2 v[16], k[16];
            {
              const float4* k4 = reinterpret_cast<const float4*>(s_k1 + c0);
#pragma unroll
              for (int i = 0; i < 8; ++i) { const float4 t4 = k4[i]; k[2*i] = make_float2(t4.x, t4.y); k[2*i+1] = make_float2(t4.z, t4.w); }
            }
            tmem_ld_wait32(ra, rb);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              v[i] = __fadd2_rn(make_float2(__uint_as_float(ra[2*i]), __uint_as_float(ra[2*i+1])), k[i]);
              v[8 + i] = __fadd2_rn(make_float2(__uint_as_float(rb[2*i]), __uint_as_float(rb[2*i+1])), k[8 + i]);
            }
            {
              // no activation = slope 1 (max(v, 1 * v) is v): no branch, so no register shuffling where the two flavours would meet
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float2 t = __fmul2_rn(v[i], slope2);
                v[i].x = fmaxf(v[i].x, t.x); v[i].y = fmaxf(v[i].y, t.y);
              }
            }
            if (ds_smem) {   // (two copies: a pointer that may be shared or global costs generic loads and their address setup)
              const float4* k4 = reinterpret_cast<const float4*>(s_ds + half * 256 + c0);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float4 t4 = k4[i];
                v[2*i] = __fmul2_rn(v[2*i], make_float2(t4.x, t4.y)); v[2*i+1] = __fmul2_rn(v[2*i+1], make_float2(t4.z, t4.w));
              }
            } else if (e_dropscale) {
              const float4* k4 = reinterpret_cast<const float4*>(dsrow + (e_OC == e_OCr ? c0 : c0 - fdiv(c0, p.fd_ocr) * e_OCr));
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float4 t4 = __ldg(k4 + i);
                v[2*i] = __fmul2_rn(v[2*i], make_float2(t4.x, t4.y)); v[2*i+1] = __fmul2_rn(v[2*i+1], make_float2(t4.z, t4.w));
              }
            }
            __align__(16) uint32_t ob32[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const __nv_bfloat162 pk = __floats2bfloat162_rn(v[i].x, v[i].y);
              ob32[i] = *reinterpret_cast<const uint32_t*>(&pk);
            }
            if (e_mask_out) {
              // sign bits from the packed outputs: bf16 > 0 <=> its bit pattern, read as int16, is > 0; sign(y) = sign(v)
              // wherever the Dropout2d scale is non-zero (and a dropped channel's gradient is zero whatever the bit says)
              // word i holds elements 2i (low half) and 2i+1 (high half): select bit 2i of the low and bit 2i+1 of the high
              // compare mask and OR everything together - one compare and one three-input logic op per word
              // (one packed bf16x2 compare per word - HSET2 - instead of the four-instruction integer emulation of
              // __vcmpgts2; bf16 > 0 is false for -0 / +0 exactly like the signed integer compare)
              uint32_t acc0 = 0, acc1 = 0;
              const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const uint32_t sel = (1u << (2 * i)) | (1u << (2 * i + 17));
                acc0 |= __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&ob32[i]), zero2) & sel;
                acc1 |= __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&ob32[8 + i]), zero2) & sel;
              }
              const unsigned long long bits =
                  (unsigned long long)(((acc0 & 0xFFFFu) | (acc0 >> 16)) | ((((acc1 & 0xFFFFu) | (acc1 >> 16))) << 16));
              mb64 |= bits << (32 * hh);
            }
            if (valid && !(e_dbg & 1)) {
              st_global_256(orow + jq * 16, ob32);
              st_global_256(orow + jq * 16 + 16, ob32 + 8);
            }
          }
          if (mrow && valid) mrow[j >> 2] = mb64;
        }
      } else if (MODE == 1 && fast_bwd) {
        bf16* orow = out + pix * e_OC + nt * BN;
        for (int j = jb; j < j_end; j += 2) {
          uint32_t ra[16], rb[16];
          tmem_ld16(taddr0 + (uint32_t)(j * 16), ra);
          tmem_ld16(taddr0 + (uint32_t)(j * 16 + 16), rb);
          const int c0 = nt * BN + j * 16;
          const int wi = j >> 1;   // j is even: one 32-bit mask word covers both chunks
          uint32_t word = mk[0];
#pragma unroll
          for (int w = 1; w < 8; ++w) word = (wi == w) ? mk[w] : word;
          float2 v[16];
          tmem_ld_wait32(ra, rb);
          // slope where the sign bit is clear: a predicated multiply (x * 1 is x, so skipping it changes nothing), then the
          // Dropout2d scales as packed multiplies - 2.5 issue slots per element instead of 4 (bit test, select, two multiplies)
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            v[i] = make_float2(mul_slope_if_clear(__uint_as_float(ra[2*i]), word, 1u << (2*i)),
                               mul_slope_if_clear(__uint_as_float(ra[2*i+1]), word, 1u << (2*i+1)));
            v[8 + i] = make_float2(mul_slope_if_clear(__uint_as_float(rb[2*i]), word, 1u << (16 + 2*i)),
                                   mul_slope_if_clear(__uint_as_float(rb[2*i+1]), word, 1u << (16 + 2*i+1)));
          }
          if (ds_smem) {   // (two copies: a pointer that may be shared or global costs generic loads and their address setup)
            const float4* k4 = reinterpret_cast<const float4*>(s_ds + half * 256 + c0);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 t4 = k4[i];
              v[2*i] = __fmul2_rn(v[2*i], make_float2(t4.x, t4.y)); v[2*i+1] = __fmul2_rn(v[2*i+1], make_float2(t4.z, t4.w));
            }
          } else if (e_dropscale) {
            const float4* k4 = reinterpret_cast<const float4*>(dsrow + (e_OC == e_OCr ? c0 : c0 - fdiv(c0, p.fd_ocr) * e_OCr));
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 t4 = __ldg(k4 + i);
              v[2*i] = __fmul2_rn(v[2*i], make_float2(t4.x, t4.y)); v[2*i+1] = __fmul2_rn(v[2*i+1], make_float2(t4.z, t4.w));
            }
          }
          __align__(16) uint32_t ob32[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const __nv_bfloat162 pk = __floats2bfloat162_rn(v[i].x, v[i].y);
            ob32[i] = *reinterpret_cast<const uint32_t*>(&pk);
          }
          if (valid && !(e_dbg & 1)) {
            st_global_256(orow + j * 16, ob32);
            st_global_256(orow + j * 16 + 16, ob32 + 8);
          }
        }
      } else if (MODE == 0 && fast_fwd_silu) {
        bf16* orow = out + pix * e_OC + nt * BN;
        bf16* prow = reinterpret_cast<bf16*>(e_preact) + pix * e_OC + nt * BN;
        for (int j = jb; j < j_end; j += 2) {
          uint32_t ra[16], rb[16];
          tmem_ld16(taddr0 + (uint32_t)(j * 16), ra);
          tmem_ld16(taddr0 + (uint32_t)(j * 16 + 16), rb);
          const int c0 = nt * BN + j * 16;
          float v[32];
          {
            const float4* k4 = reinterpret_cast<const float4*>(s_k1 + c0);
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float4 t4 = k4[i]; v[4*i] = t4.x; v[4*i+1] = t4.y; v[4*i+2] = t4.z; v[4*i+3] = t4.w; }
          }
          tmem_ld_wait32(ra, rb);
#pragma unroll
          for (int i = 0; i < 16; ++i) { v[i] += __uint_as_float(ra[i]); v[16 + i] += __uint_as_float(rb[i]); }
          // the saved pre-activation is bf16; the activation is taken from the rounded value (what backward will see)
          __align__(16) uint32_t pb32[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const __nv_bfloat162 pk = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
            pb32[i] = *reinterpret_cast<const uint32_t*>(&pk);
            const float2 f2 = __bfloat1622float2(pk);
            v[2 * i] = f2.x; v[2 * i + 1] = f2.y;
          }
          if (valid && !(e_dbg & 1)) {
            st_global_256(prow + j * 16, pb32);
            st_global_256(prow + j * 16 + 16, pb32 + 8);
          }
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] *= fast_sigmoid(v[i]);
          if (e_dropscale) {
            const float4* k4 = reinterpret_cast<const float4*>(ds_smem ? s_ds + half * 256 + c0 : dsrow + (e_OC == e_OCr ? c0 : c0 - fdiv(c0, p.fd_ocr) * e_OCr));
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float4 t4 = k4[i]; v[4*i] *= t4.x; v[4*i+1] *= t4.y; v[4*i+2] *= t4.z; v[4*i+3] *= t4.w; }
          }
          __align__(16) uint32_t ob32[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const __nv_bfloat162 pk = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
            ob32[i] = *reinterpret_cast<const uint32_t*>(&pk);
          }
          if (valid && !(e_dbg & 1)) {
            st_global_256(orow + j * 16, ob32);
            st_global_256(orow + j * 16 + 16, ob32 + 8);
          }
        }
      } else if (MODE == 1 && fast_bwd_silu) {
        bf16* orow = out + pix * e_OC + nt * BN;
        const bf16* srow = reinterpret_cast<const bf16*>(e_saved) + pix * e_OC + nt * BN;
        // the saved row of the next chunk pair is requested one iteration ahead (it sits in L2: prefetched two tiles ago)
        uint4 nx[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) nx[i] = make_uint4(0, 0, 0, 0);
        if (valid && jb < j_end) { ld_global_nc_256(srow + jb * 16, nx[0], nx[1]); ld_global_nc_256(srow + jb * 16 + 16, nx[2], nx[3]); }
        for (int j = jb; j < j_end; j += 2) {
          uint32_t ra[16], rb[16];
          tmem_ld16(taddr0 + (uint32_t)(j * 16), ra);
          tmem_ld16(taddr0 + (uint32_t)(j * 16 + 16), rb);
          const int c0 = nt * BN + j * 16;
          uint4 cu[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) cu[i] = nx[i];
          if (j + 2 < j_end && valid) { ld_global_nc_256(srow + (j + 2) * 16, nx[0], nx[1]); ld_global_nc_256(srow + (j + 2) * 16 + 16, nx[2], nx[3]); }
          float pre[32];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float2 f2 = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(cu)[i]);
            pre[2 * i] = f2.x; pre[2 * i + 1] = f2.y;
          }
          if (has_bn) {
            const float4* k0 = reinterpret_cast<const float4*>(s_k0 + c0);
            const float4* k1 = reinterpret_cast<const float4*>(s_k1 + c0);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 a4 = k0[i], b4 = k1[i];
              pre[4*i] = pre[4*i] * a4.x + b4.x; pre[4*i+1] = pre[4*i+1] * a4.y + b4.y;
              pre[4*i+2] = pre[4*i+2] * a4.z + b4.z; pre[4*i+3] = pre[4*i+3] * a4.w + b4.w;
            }
          }
          // d(SiLU)/d(pre) = s (1 + pre (1 - s)), times the Dropout2d scale of the channel
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float sg = fast_sigmoid(pre[i]);
            pre[i] = sg * (1.f + pre[i] * (1.f - sg));
          }
          if (e_dropscale) {
            const float4* k4 = reinterpret_cast<const float4*>(ds_smem ? s_ds + half * 256 + c0 : dsrow + (e_OC == e_OCr ? c0 : c0 - fdiv(c0, p.fd_ocr) * e_OCr));
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float4 t4 = k4[i]; pre[4*i] *= t4.x; pre[4*i+1] *= t4.y; pre[4*i+2] *= t4.z; pre[4*i+3] *= t4.w; }
          }
          tmem_ld_wait32(ra, rb);
          __align__(16) uint32_t ob32[16];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const __nv_bfloat162 pa = __floats2bfloat162_rn(__uint_as_float(ra[2 * i]) * pre[2 * i], __uint_as_float(ra[2 * i + 1]) * pre[2 * i + 1]);
            const __nv_bfloat162 pb = __floats2bfloat162_rn(__uint_as_float(rb[2 * i]) * pre[16 + 2 * i], __uint_as_float(rb[2 * i + 1]) * pre[16 + 2 * i + 1]);
            ob32[i] = *reinterpret_cast<const uint32_t*>(&pa);
            ob32[8 + i] = *reinterpret_cast<const uint32_t*>(&pb);
          }
          if (valid && !(e_dbg & 1)) {
            st_global_256(orow + j * 16, ob32);
            st_global_256(orow + j * 16 + 16, ob32 + 8);
          }
        }
      } else {
      // software pipeline over the chunks: the TMEM load of chunk j+1 is in flight while chunk j is processed
      uint32_t rn[16];
      if (jb < j_end) tmem_ld16(taddr0 + (uint32_t)(jb * 16), rn);
      for (int j = jb; j < j_end; ++j) {
        uint32_t r[16];
        const int cl = j * 16;          // channel inside the N tile
        const int c0 = nt * BN + cl;    // absolute output channel
        // global operands of this chunk are fetched while the TMEM load is in flight
        float ds[16];
        if (e_dropscale) {
          const float4* dp = reinterpret_cast<const float4*>(ds_smem ? s_ds + half * 256 + c0 : dsrow + (e_OC == e_OCr ? c0 : c0 - fdiv(c0, p.fd_ocr) * e_OCr));
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 v4 = dp[i];
            ds[4 * i] = v4.x; ds[4 * i + 1] = v4.y; ds[4 * i + 2] = v4.z; ds[4 * i + 3] = v4.w;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) ds[i] = 1.f;
        }
        __align__(16) bf16 sv[16];
        __align__(16) float svf[16];
        if (MODE == 1) {
          if (e_saved && valid && !use_mask && io_f32) {
            const float* sp = reinterpret_cast<const float*>(e_saved) + pix * e_OC + c0;
            ld_global_nc_256(sp, reinterpret_cast<uint4*>(svf)[0], reinterpret_cast<uint4*>(svf)[1]);
            ld_global_nc_256(sp + 8, reinterpret_cast<uint4*>(svf)[2], reinterpret_cast<uint4*>(svf)[3]);
          } else if (e_saved && valid && !use_mask) {
            ld_global_nc_256(reinterpret_cast<const bf16*>(e_saved) + pix * e_OC + c0, reinterpret_cast<uint4*>(sv)[0],
                             reinterpret_cast<uint4*>(sv)[1]);
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) { sv[i] = __float2bfloat16_rn(0.f); svf[i] = 0.f; }
          }
        }
        long long ec0 = 0;
        if (eprof) ec0 = clock64();
        tmem_ld_wait16(rn);
        if (eprof) { const long long t = clock64(); ec_ld += t - ec0; ec_pre += ec0 - eprev; eprev = t; }
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = rn[i];
        if (j + 1 < j_end) tmem_ld16(taddr0 + (uint32_t)((j + 1) * 16), rn);
        __align__(16) bf16 ob[16];
        float s1[16], s2[16];
        if (MODE == 0 && e_head_out) {
          // prediction head: the 16 accumulators of this pixel are the raw logits (5 + classes, zero padded);
          // /root/reference/yogo/model.py:295-313 applied in registers, written straight to the NCHW fp32 tensor
          if (valid) {
            const int D = p.head_D;
            float t[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) t[i] = __uint_as_float(r[i]) + s_k1[i];
            if (p.head_traw) {
              float* tr = p.head_traw + pix * D;
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (i < D) tr[i] = t[i];
            }
            const int SS = e_OH * e_OW, cell = oh * e_OW + ow;
            float* o = e_head_out + (long long)n * D * SS + cell;
            const float cx = p.head_cxs ? p.head_cxs[cell]
                                        : (e_OW > 1 ? (float)ow * ((1.f - 1.f / (float)e_OW) / (float)(e_OW - 1)) : 0.f);
            const float cy = p.head_cys ? p.head_cys[cell]
                                        : (e_OH > 1 ? (float)oh * ((1.f - 1.f / (float)e_OH) / (float)(e_OH - 1)) : 0.f);
            o[0] = (1.f / (float)e_OW) * sigmoidf_(t[0]) + cx;
            o[(long long)SS] = (1.f / (float)e_OH) * sigmoidf_(t[1]) + cy;
            o[2LL * SS] = p.head_aw * expf(fminf(t[2], 80.f)) * p.head_wm;
            o[3LL * SS] = p.head_ah * expf(fminf(t[3], 80.f)) * p.head_hm;
            o[4LL * SS] = sigmoidf_(t[4]);
            if (p.head_inf) {
              float mx = -INFINITY;
#pragma unroll
              for (int i = 5; i < 16; ++i)
                if (i < D) mx = fmaxf(mx, t[i]);
              float se = 0.f;
#pragma unroll
              for (int i = 5; i < 16; ++i)
                if (i < D) { t[i] = expf(t[i] - mx); se += t[i]; }
              const float inv = 1.f / se;
#pragma unroll
              for (int i = 5; i < 16; ++i)
                if (i < D) o[(long long)i * SS] = t[i] * inv;
            } else {
#pragma unroll
              for (int i = 5; i < 16; ++i)
                if (i < D) o[(long long)i * SS] = t[i];
            }
          }
        } else if (MODE == 0) {
          __align__(16) bf16 pb[16];
          const bool rnd = (e_stats || e_preact) && !io_f32;
          {
            // per-channel constants: 128-bit broadcast loads from smem
            const float4* sh4 = reinterpret_cast<const float4*>(s_k1 + c0);
            float shf[16];
#pragma unroll
            for (int i = 0; i < 4; ++i) { const float4 t4 = sh4[i]; shf[4*i] = t4.x; shf[4*i+1] = t4.y; shf[4*i+2] = t4.z; shf[4*i+3] = t4.w; }
            if (e_has_scale) {
              const float4* sc4 = reinterpret_cast<const float4*>(s_k0 + c0);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float4 t4 = sc4[i];
                r[4*i]   = __float_as_uint(__uint_as_float(r[4*i])   * t4.x + shf[4*i]);
                r[4*i+1] = __float_as_uint(__uint_as_float(r[4*i+1]) * t4.y + shf[4*i+1]);
                r[4*i+2] = __float_as_uint(__uint_as_float(r[4*i+2]) * t4.z + shf[4*i+2]);
                r[4*i+3] = __float_as_uint(__uint_as_float(r[4*i+3]) * t4.w + shf[4*i+3]);
              }
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) + shf[i]);
            }
          }
          if (rnd) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const __nv_bfloat162 pk = __floats2bfloat162_rn(__uint_as_float(r[2*i]), __uint_as_float(r[2*i+1]));
              reinterpret_cast<__nv_bfloat162*>(pb)[i] = pk;
              const float2 f2 = __bfloat1622float2(pk);
              r[2*i] = __float_as_uint(f2.x); r[2*i+1] = __float_as_uint(f2.y);
            }
          }
          if (rnd || (io_f32 && e_stats)) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float x = __uint_as_float(r[i]);
              s1[i] = valid ? x : 0.f;
              s2[i] = valid ? x * x : 0.f;
            }
          }
          if (io_f32 && e_preact && valid && !(e_dbg & 1)) {   // fp32 pre-activation copy (before the activation below)
            float* pp = reinterpret_cast<float*>(e_preact) + pix * e_OC + c0;
            st_global_256(pp, r);
            st_global_256(pp + 8, r + 8);
          }
          if (e_mask_out && valid) {
            uint32_t bits = 0;
#pragma unroll
            for (int i = 0; i < 16; ++i) bits |= (__uint_as_float(r[i]) > 0.f ? 1u : 0u) << i;
            const int jj = j - jb, mb = jj >> 2, sh = 16 * (jj & 3);
            if (mb == 0) mbits0 |= (unsigned long long)bits << sh;
            else if (mb == 1) mbits1 |= (unsigned long long)bits << sh;
            else if (mb == 2) mbits2 |= (unsigned long long)bits << sh;
            else mbits3 |= (unsigned long long)bits << sh;
          }
          if (e_act == YG_ACT_LRELU) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float x = __uint_as_float(r[i]);
              r[i] = __float_as_uint(fmaxf(x, 0.01f * x));
            }
          } else if (e_act == YG_ACT_SILU) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float x = __uint_as_float(r[i]);
              r[i] = __float_as_uint(x * __frcp_rn(1.f + __expf(-x)));
            }
          }
          if (e_dropscale) {
#pragma unroll
            for (int i = 0; i < 16; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * ds[i]);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i)
            reinterpret_cast<__nv_bfloat162*>(ob)[i] = __floats2bfloat162_rn(__uint_as_float(r[2*i]), __uint_as_float(r[2*i+1]));
          if (eprof) { const long long t = clock64(); ec_math += t - eprev; eprev = t; }
          if (valid && !(e_dbg & 1)) {
            if (out && io_f32) {
              float* op = reinterpret_cast<float*>(p.out) + pix * e_OC + c0;
              st_global_256(op, r);
              st_global_256(op + 8, r + 8);
            } else if (out) {
              st_global_256(out + pix * e_OC + c0, reinterpret_cast<const uint32_t*>(ob));
            }
            if (e_preact && !io_f32) {
              st_global_256(reinterpret_cast<bf16*>(e_preact) + pix * e_OC + c0, reinterpret_cast<const uint32_t*>(pb));
            }
          }
          if (eprof) { const long long t = clock64(); ec_store += t - eprev; eprev = t; }
          if (e_stats) {
            const float t1 = lane_transpose_reduce16(s1, lane);
            const float t2 = lane_transpose_reduce16(s2, lane);
            if (lane < 16) {
              atomicAdd(&s_stat[cl + lane], t1);
              atomicAdd(&s_stat[256 + cl + lane], t2);
            }
          }
        } else {
          float pre[16];
          // saved activations: packed bf16x2 -> float2
          if (io_f32) {
#pragma unroll
            for (int i = 0; i < 16; ++i) pre[i] = svf[i];
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float2 f2 = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(sv)[i]);
              pre[2*i] = f2.x; pre[2*i+1] = f2.y;
            }
          }
          if (has_bn) {
            const float4* k0 = reinterpret_cast<const float4*>(s_k0 + c0);
            const float4* k1 = reinterpret_cast<const float4*>(s_k1 + c0);
            const float4* k2 = reinterpret_cast<const float4*>(s_k2 + c0);
            const float4* k3 = reinterpret_cast<const float4*>(s_k3 + c0);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 a4 = k0[i], b4 = k1[i], m4 = k2[i], i4 = k3[i];
              const float sc_[4] = {a4.x, a4.y, a4.z, a4.w}, sh_[4] = {b4.x, b4.y, b4.z, b4.w};
              const float mn_[4] = {m4.x, m4.y, m4.z, m4.w}, is_[4] = {i4.x, i4.y, i4.z, i4.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float sval = pre[4*i+k];
                s2[4*i+k] = (sval - mn_[k]) * is_[k];     // xhat
                pre[4*i+k] = sval * sc_[k] + sh_[k];
              }
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) s2[i] = 0.f;
          }
          if (e_dropscale) {
#pragma unroll
            for (int i = 0; i < 16; ++i) s1[i] = __uint_as_float(r[i]) * ds[i];
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) s1[i] = __uint_as_float(r[i]);
          }
          if (use_mask) {
            const int wi = j >> 1;   // 32-channel word of this chunk; chunks j = half, half+2, .. -> words 0, 1, ..
            uint32_t word = mk[0];
#pragma unroll
            for (int w = 1; w < 8; ++w) word = (wi == w) ? mk[w] : word;
            const uint32_t bits = word >> ((j & 1) * 16);
#pragma unroll
            for (int i = 0; i < 16; ++i) s1[i] *= ((bits >> i) & 1u) ? 1.f : 0.01f;
          } else if (e_saved) {
            if (e_act == YG_ACT_LRELU) {
#pragma unroll
              for (int i = 0; i < 16; ++i) s1[i] *= pre[i] > 0.f ? 1.f : 0.01f;
            } else if (e_act == YG_ACT_SILU) {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float sg = __frcp_rn(1.f + __expf(-pre[i]));
                s1[i] *= sg * (1.f + pre[i] * (1.f - sg));
              }
            }
          }
          if (io_f32) {
            if (valid && !(e_dbg & 1)) {
              float* op = reinterpret_cast<float*>(p.out) + pix * e_OC + c0;
              uint32_t sb[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) sb[i] = __float_as_uint(s1[i]);
              st_global_256(op, sb);
              st_global_256(op + 8, sb + 8);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const __nv_bfloat162 pk = __floats2bfloat162_rn(s1[2*i], s1[2*i+1]);
              reinterpret_cast<__nv_bfloat162*>(ob)[i] = pk;
              if (e_bn_sums) {
                const float2 f2 = __bfloat1622float2(pk);
                s1[2*i] = f2.x; s1[2*i+1] = f2.y;
              }
            }
          }
          if (e_bn_sums) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float g = valid ? s1[i] : 0.f;
              s1[i] = g;
              s2[i] = g * s2[i];
            }
          }
          const bool second_sum = has_bn;   // sum(g * xhat) only exists for BatchNorm layers; sum(g) alone = d(bias)
          if (valid && !(e_dbg & 1) && !io_f32) {
            st_global_256(out + pix * e_OC + c0, reinterpret_cast<const uint32_t*>(ob));
          }
          if (e_bn_sums) {
            const float t1 = lane_transpose_reduce16(s1, lane);
            if (lane < 16) atomicAdd(&s_stat[cl + lane], t1);
            if (second_sum) {
              const float t2 = lane_transpose_reduce16(s2, lane);
              if (lane < 16) atomicAdd(&s_stat[256 + cl + lane], t2);
            }
          }
        }
      }
      }   // generic chunk loop
      if (MODE == 0 && e_mask_out && valid && j_end > jb && !(fast_fwd && ((j_end - jb) & 3) == 0)) {
        // one store per thread and tile: 2 bytes per chunk, contiguous because the chunks are
        unsigned char* mp = reinterpret_cast<unsigned char*>(e_mask_out) + ((pix * e_OC + nt * BN) >> 3) + jb * 2;
        const int nmine = j_end - jb;
        const bool al8 = (e_OC & 63) == 0 && (BN & 63) == 0;   // 8-byte aligned rows
        if (nmine == 4 && al8) *reinterpret_cast<unsigned long long*>(mp) = mbits0;
        else if (nmine == 8 && al8) {
          reinterpret_cast<unsigned long long*>(mp)[0] = mbits0;
          reinterpret_cast<unsigned long long*>(mp)[1] = mbits1;
        } else if (nmine == 16 && al8) {
          reinterpret_cast<unsigned long long*>(mp)[0] = mbits0;
          reinterpret_cast<unsigned long long*>(mp)[1] = mbits1;
          reinterpret_cast<unsigned long long*>(mp)[2] = mbits2;
          reinterpret_cast<unsigned long long*>(mp)[3] = mbits3;
        } else if (nmine == 2) *reinterpret_cast<unsigned int*>(mp) = (unsigned int)mbits0;
        else {
          for (int c = 0; c < nmine; ++c) {
            const unsigned long long wv = (c >> 2) == 0 ? mbits0 : ((c >> 2) == 1 ? mbits1 : ((c >> 2) == 2 ? mbits2 : mbits3));
            reinterpret_cast<unsigned short*>(mp)[c] = (unsigned short)((wv >> (16 * (c & 3))) & 0xFFFFull);
          }
        }
      }
      // accumulator drained: hand the TMEM buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CTA2) mbar_arrive_cluster(map_to_cta(smem_u32(&tempty_bar[acc]), 0u));   // the leader's MMA warp waits for both
        else mbar_arrive(&tempty_bar[acc]);
      }
      // with several N tiles per CTA the statistics must be flushed per tile (channels change)
      if (e_nnt > 1 && (e_stats || e_bn_sums)) {
        asm volatile("bar.sync 1, 256;" ::: "memory");
        double* dst = MODE == 0 ? e_stats : e_bn_sums;
        for (int i = threadIdx.x - 64; i < BN; i += 256) {
          const float a1 = s_stat[i], a2 = s_stat[256 + i];
          if (a1 != 0.f || a2 != 0.f) {
            atomicAdd(dst + (nt * BN + i) % e_OCr, (double)a1);
            atomicAdd(dst + e_OCr + (nt * BN + i) % e_OCr, (double)a2);
          }
          s_stat[i] = 0.f; s_stat[256 + i] = 0.f;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      ++ec_tiles;
    }
    if (eprof && lane == 0 && blockIdx.x < 256) {
      unsigned long long* d = g_tc_dbg + blockIdx.x * 16 + 8;
      d[0] = ec_tfull; d[1] = ec_ld; d[2] = ec_pre; d[3] = ec_math; d[4] = ec_store; d[5] = ec_rest; d[6] = ec_tiles;
    }

  }

  // ------------------------------------------------------------------------- teardown
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (p.n_ntiles == 1) {
    double* dst = MODE == 0 ? p.stats : p.bn_sums;
    if (dst) {
      for (int i = threadIdx.x; i < BN; i += NTHREADS) {
        atomicAdd(dst + i % p.OCr, (double)s_stat[i]);
        atomicAdd(dst + p.OCr + i % p.OCr, (double)s_stat[256 + i]);
      }
    }
  }
  if (CTA2) cluster_sync_all();   // neither CTA leaves (or frees TMEM) while its peer may still signal it
  if (warp == 1) { if (CTA2) tmem_dealloc2(tmem_base, (uint32_t)p.tmem_cols); else tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols); }
}

// ------------------------------------------------------------------------------------------ weights
// OIHW fp32 -> bf16 [tap][Cout][Cin] (transpose == 0, fprop) or [tap][Cin][Cout] (transpose == 1, dgrad).
// W-fold factor g > 1: the NHWC tensors are viewed as (N, H, W/g, g*C) - g adjacent pixels become one
// "super pixel" - and the 3x3 convolution becomes a 3x3 convolution over super pixels with structured weights
//   W'[tap=(r,s')][(q,co)][(pi,ci)] = W[co][ci][r][s],  s = g*(s'-1) + pi - q + 1  (zero if s is not in 0..2).
// Same bytes, g x fewer and g x longer TMA rows, K and N large enough for efficient UMMA tiles.
__global__ void pack_weights_kernel(const float* __restrict__ w, bf16* __restrict__ out, int Cout, int Cin, int taps,
                                    int transpose, int g) {
  const int Cof = Cout * g, Cif = Cin * g;
  const long long total = (long long)Cof * Cif * taps;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int inner, outer, tap;
  if (!transpose) { inner = (int)(i % Cif); outer = (int)((i / Cif) % Cof); tap = (int)(i / ((long long)Cif * Cof)); }
  else { inner = (int)(i % Cof); outer = (int)((i / Cof) % Cif); tap = (int)(i / ((long long)Cif * Cof)); }
  const int cof = transpose ? inner : outer, cif = transpose ? outer : inner;
  const int q = cof / Cout, co = cof % Cout, pi = cif / Cin, ci = cif % Cin;
  const int r = tap / 3, sp = tap % 3;
  const int sreal = g * (sp - 1) + pi - q + 1;
  float v = 0.f;
  if (sreal >= 0 && sreal <= 2) v = w[((long long)co * Cin + ci) * taps + r * 3 + sreal];
  out[i] = __float2bfloat16_rn(v);
}

// Stride-2 dgrad with column pairs folded (see conv_dgrad_tc): [slice = r*2 + dxo][(q,ci)][co], where the
// output column is x = 2x'+q and the tap reads dz column x'+dxo:  (q=0,dxo=0) -> s=1, (q=1,dxo=0) -> s=2,
// (q=1,dxo=1) -> s=0, (q=0,dxo=1) -> structurally zero.
__global__ void pack_weights_s2fold_kernel(const float* __restrict__ w, bf16* __restrict__ out, int Cout, int Cin) {
  const long long total = 6LL * 2 * Cin * Cout;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int co = (int)(i % Cout);
  const int cif = (int)((i / Cout) % (2 * Cin));
  const int sl = (int)(i / ((long long)2 * Cin * Cout));
  const int q = cif / Cin, ci = cif % Cin, r = sl >> 1, dxo = sl & 1;
  const int s = q == 0 ? (dxo == 0 ? 1 : -1) : (dxo == 0 ? 2 : 0);
  float v = 0.f;
  if (s >= 0) v = w[((long long)co * Cin + ci) * 9 + r * 3 + s];
  out[i] = __float2bfloat16_rn(v);
}

// ------------------------------------------------------------------------------------------ host
// yg_set_tc_options (include/yogo_b200.h): bits 7-11 = profiling knobs of the engine (TcParams::debug), bit 21 = fp32 tensors as
// split-bf16 convolutions (api.cu)
constexpr int TC_OPTION_BITS = (31 << 7) | (1 << 21);
static int g_tc_options = 0;
// W-fold factor for stride-1 convolutions with few channels (see pack_weights_kernel): fold while the folded
// input channel count stays <= 64 and everything remains a legal UMMA shape.
static int fold_factor(int Cin, int Cout, int W, int stride) {
  if (stride != 1) return 1;
  for (int g = 4; g >= 2; g >>= 1)
    if (W % g == 0 && g * Cin <= 64 && g * Cout <= 256 && (g * Cin) % 16 == 0 && (g * Cout) % 16 == 0) return g;
  return 1;
}
// Stride-2 dgrad with few input channels: fold output column pairs (2 classes x N = 2*Cin instead of 4 x N = Cin).
static bool s2fold_dgrad(int Cin, int W, int stride) {
  return stride == 2 && W % 2 == 0 && 2 * Cin <= 64 && (2 * Cin) % 16 == 0;
}
// bit kk set <=> K step kk (16 folded channels) of folded tap column sp touches a sub-pixel with non-zero weights.
// kdim_is_input: K runs over (pi, ci) [fprop / wgrad-B], otherwise over (q, co) [dgrad].
static unsigned fold_kmask(int g, int Cr, int sp, bool kdim_is_input) {
  if (g == 1) return 0xFFFFFFFFu;
  unsigned valid = 0;  // valid sub-pixel indices of the K dimension
  for (int a = 0; a < g; ++a)
    for (int b = 0; b < g; ++b) {
      const int pi = kdim_is_input ? a : b, q = kdim_is_input ? b : a;
      const int sreal = g * (sp - 1) + pi - q + 1;
      if (sreal >= 0 && sreal <= 2) valid |= 1u << a;
    }
  unsigned m = 0;
  const int ksteps = g * Cr / 16;
  for (int kk = 0; kk < ksteps && kk < 32; ++kk) {
    const int lo = (kk * 16) / Cr, hi = (kk * 16 + 15) / Cr;
    for (int a = lo; a <= hi && a < g; ++a)
      if ((valid >> a) & 1u) m |= 1u << kk;
  }
  return m;
}

static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
static std::once_flag g_encode_once;
static int* g_error_flag = nullptr;  // device int, reports which barrier wait timed out

static bool get_encode() {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      g_encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
  });
  return g_encode != nullptr;
}

static int make_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, int kc) {
  uint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUtensorMapSwizzle sw = kc == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                                         : (kc == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims,
                        strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with %d (rank %d dims %llu %llu %llu box %u %u %u)", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)dims[2], box[0], box[1],
              box[2]);
    return YG_ERR_CUDA;
  }
  return YG_OK;
}

static int pick_kc(int K) { return (K % 64 == 0) ? 64 : ((K % 32 == 0) ? 32 : ((K % 16 == 0) ? 16 : 0)); }
static int pick_bn(int Nc) {
  if (Nc % 16) return 0;
  if (Nc <= 256) return Nc;
  for (int bn = 256; bn >= 16; bn -= 16)
    if (Nc % bn == 0) return bn;
  return 0;
}

bool tc_fwd_supported(int dtype, int W, int Cin, int Cout, int ks, int stride) {
  if (dtype != YG_BF16 || ks != 3 || (stride != 1 && stride != 2)) return false;
  const int g = fold_factor(Cin, Cout, W, stride);
  return pick_kc(Cin * g) && pick_bn(Cout * g) && Cout * g <= 512;
}
bool tc_dgrad_supported(int dtype, int W, int Cin, int Cout, int ks, int stride) {
  if (dtype != YG_BF16 || ks != 3 || (stride != 1 && stride != 2)) return false;
  const int g = s2fold_dgrad(Cin, W, stride) ? 2 : fold_factor(Cin, Cout, W, stride);
  return pick_kc(Cout * (stride == 1 ? g : 1)) && pick_bn(Cin * g) && Cin * g <= 512;
}


// ==========================================================================================
// wgrad: dW[co][ci][r][s] = sum over pixels dz[p][co] * x[p + tap][ci]
//   GEMM view  D[M = 128 couts][N = BNW cins] += A^T[K = 16 pixels x M] * B[K = 16 pixels x N], both operands
//              MN-major straight out of the NHWC tensors (pixel rows, channels contiguous): the TMA boxes of
//              the fprop engine are reused unchanged, only the UMMA descriptors say "MN-major".
//   K loop     over ALL pixels a CTA owns: accumulators stay in TMEM for the whole kernel (3 taps x BNW
//              columns), one epilogue at the end writes fp32 partials; a deterministic second kernel sums
//              the per-CTA partials, clamps and writes OIHW fp32.
//   work split unit = (filter column s, M tile, N tile); CTA c works on unit c % nunits and on every
//              nslices-th pixel tile.
// ==========================================================================================
struct TwGroup {
  int map, dh, dw, rows, ntaps;
  int ro[TW_MAX_TAPS];
  int slot[TW_MAX_TAPS];  // accumulator slot (= filter row r)
};
struct TwMaps {
  CUtensorMap a;     // dz
  CUtensorMap b[4];  // x (parity sub-grids for stride 2)
};
struct TwParams {
  int N, tiles_h, tiles_w, total_tiles;
  int Cin, Cout, BNW, n_ntiles, n_mtiles, nunits, nslices;
  int kb, nbblocks, a_block_bytes, b_block_bytes, stage_bytes, nstages, tmem_cols;
  int ngroups;                 // groups per filter column
  int ncols;                   // filter columns = work-unit columns (3 for 3x3, 1 for 1x1)
  TwGroup g[3][2];
  float* partial;
  int share_a;          // stride 2 (two parity groups per tile): ONE stage per tile holds the dz tile once and both x boxes
                        // (the dz tile used to be fetched from L2 once per group - the kernel is L2-bandwidth bound)
  int merge2;           // stride 2, one B block per tap: the two row taps of the odd-parity group (filter rows 0 and 2, adjacent
                        // rows of the same box) run as ONE N = 2 BNW MMA; they own the adjacent accumulator slots 0 and 1
  int row_slot[3];      // accumulator slot of filter row r (identity unless merge2)
  int merge3;           // stride 1, one 64-channel B block per tap: the three filter rows of a column run as ONE N = 3 BNW MMA
                        // (the B descriptor's leading-dimension stride = one tile row of the halo box = the next row tap)
  int do_bias;          // also accumulate d(bias)[co] = sum over pixels of dz: one extra N = 16 MMA per K step against
  float* bias_partial;  // a block of ones (units with s == 0, nt == 0); partials [slice][mtile][128]
  int* error_flag;
};

__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}

template <int KB, int KA>
__global__ void __launch_bounds__(192, 1)
wgrad_tc_kernel(const __grid_constant__ TwMaps maps, const __grid_constant__ TwParams p) {
  constexpr int NTHREADS = 192;                           // warp 0 producer, warp 1 MMA, warps 2-5 epilogue
  constexpr uint32_t ROWB = KB * 2;                       // bytes per pixel row of a B block
  constexpr uint32_t LAYOUT_B = KB == 64 ? 2u : (KB == 32 ? 4u : 6u);
  constexpr uint32_t ROWA = KA * 2;                       // A blocks are KA couts wide (64: SWIZZLE_128B, 32: 64B)
  constexpr uint32_t LAYOUT_A = KA == 64 ? 2u : 4u;
  constexpr int MBLOCKS = 128 / KA;                       // blocks that make up the M = 128 operand
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* tail = smem + (size_t)p.nstages * p.stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + 8;
  uint64_t* done_bar = empty_bar + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 2);
  unsigned char* ones = tail + 1024;   // 16 pixel rows x ROWB bytes of bf16 1.0 (B operand of the bias column)

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // provably uniform
  const int unit = blockIdx.x % p.nunits, slice = blockIdx.x / p.nunits;
  const int sg = unit % p.ncols, mt = (unit / p.ncols) % p.n_mtiles, nt = unit / (p.ncols * p.n_mtiles);
  const int a_blocks = min(MBLOCKS, (p.Cout - mt * 128) / KA);
  const int BNW = p.BNW;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&maps.a);
    for (int i = 0; i < 4; ++i) prefetch_tmap(&maps.b[i]);
    for (int i = 0; i < p.nstages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(&done_bar[0], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (a_blocks < MBLOCKS) {
    // short Cout tile: the missing rows of the M = 128 operand are blocks of zeros that TMA never touches
    for (int st = 0; st < p.nstages; ++st) {
      uint4* z = reinterpret_cast<uint4*>(smem + (size_t)st * p.stage_bytes + (size_t)a_blocks * p.a_block_bytes);
      const int n16 = (MBLOCKS - a_blocks) * p.a_block_bytes / 16;
      for (int i = threadIdx.x; i < n16; i += NTHREADS) z[i] = make_uint4(0, 0, 0, 0);
    }
  }
  if (p.do_bias)
    for (int i = threadIdx.x; i < 512; i += NTHREADS) reinterpret_cast<uint32_t*>(ones)[i] = 0x3F803F80u;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // the bias column of a pixel tile is taken by one of the units that share this M tile, round robin over the tiles
  const bool do_bias = p.do_bias != 0;
  const int bias_period = p.ncols * p.n_ntiles, bias_phase = sg + p.ncols * nt;

  if (warp == 0) {
    // whole warp, uniform control flow; the elected lane issues (see elect_one)
    const uint32_t leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    const int nstages = p.nstages, ngroups = p.ngroups, nbblocks = p.nbblocks;
    for (int tile = slice; tile < p.total_tiles; tile += p.nslices) {
      int t = tile;
      const int tw = t % p.tiles_w; t /= p.tiles_w;
      const int th = t % p.tiles_h;
      const int n = t / p.tiles_h;
      const bool share = p.share_a != 0;
      for (int gi = 0; gi < ngroups; ++gi) {
        const TwGroup& g = p.g[sg][gi];
        unsigned char* sa = smem + (size_t)stage * p.stage_bytes;
        unsigned char* sb = sa + MBLOCKS * p.a_block_bytes + (share ? (size_t)gi * nbblocks * p.b_block_bytes : 0);
        if (!share || gi == 0) {
          mbar_wait(&empty_bar[stage], phase ^ 1u, p.error_flag, 11);
          int brows = g.rows;
          if (share) for (int g2 = 1; g2 < ngroups; ++g2) brows += p.g[sg][g2].rows;
          const uint32_t bytes = (uint32_t)(a_blocks * p.a_block_bytes + nbblocks * brows * TC_TW * (int)ROWB);
          mbar_expect_tx_p(&full_bar[stage], bytes, leader);
          for (int ab = 0; ab < a_blocks; ++ab)
            tma_load_4d_p(sa + (size_t)ab * p.a_block_bytes, &maps.a, &full_bar[stage], mt * 128 + ab * KA, tw * TC_TW,
                          th * TC_TH, n, leader);
        }
        for (int bb = 0; bb < nbblocks; ++bb)
          tma_load_4d_p(sb + (size_t)bb * p.b_block_bytes, &maps.b[g.map], &full_bar[stage], nt * BNW + bb * KB,
                        tw * TC_TW + g.dw, th * TC_TH + g.dh, n, leader);
        if (!share || gi == ngroups - 1) {
          if (++stage == nstages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // D=f32, A=B=bf16, both MN-major (bits 15,16), N = BNW, M = 128
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                           ((uint32_t)(BNW >> 3) << 17) | ((128u >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    uint32_t started = 0;  // bit r set once accumulator slot r holds data
    // descriptors of stage 0; everything else is an addition to the low words (16-byte units)
    const uint64_t ad_base = umma_desc_mn(smem_u32(smem), (uint32_t)p.a_block_bytes, 8 * ROWA, LAYOUT_A);
    const uint64_t bd_base = umma_desc_mn(smem_u32(smem) + (uint32_t)MBLOCKS * (uint32_t)p.a_block_bytes,
                                          (uint32_t)p.b_block_bytes, 8 * ROWB, LAYOUT_B);
    const uint32_t a_lo0 = (uint32_t)ad_base, a_hi = (uint32_t)(ad_base >> 32);
    const uint32_t b_lo0 = (uint32_t)bd_base, b_hi = (uint32_t)(bd_base >> 32);
    const uint32_t stage_units = (uint32_t)p.stage_bytes >> 4;
    const int nstages = p.nstages, ngroups = p.ngroups;
    const uint32_t ones_lo = (uint32_t)umma_desc_mn(smem_u32(ones), (uint32_t)p.b_block_bytes, 8 * ROWB, LAYOUT_B);
    const uint32_t idesc_bias = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((16u >> 3) << 17) | ((128u >> 4) << 24);
    uint32_t bias_started = 0;
    const uint32_t leader = elect_one();   // whole warp runs the loop, the elected lane issues
    int bias_it = 0;
    const bool merge2 = p.merge2 != 0;
    const uint32_t idesc2 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                            ((uint32_t)((2 * BNW) >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t b2_lo0 = (uint32_t)umma_desc_mn(smem_u32(smem) + (uint32_t)MBLOCKS * (uint32_t)p.a_block_bytes,
                                                   (uint32_t)TC_TW * ROWB, 8 * ROWB, LAYOUT_B);
    const bool share_a = p.share_a != 0;
    const uint32_t group_units = (uint32_t)(p.nbblocks * p.b_block_bytes) >> 4;
    // merged row taps: N = 3 BNW, block n of the N dimension = the same 64 channels one tile row (TC_TW pixels) further down
    const bool merge3 = p.merge3 != 0;
    const uint32_t idesc3 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                            ((uint32_t)((3 * BNW) >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t b3_lo0 = (uint32_t)umma_desc_mn(smem_u32(smem) + (uint32_t)MBLOCKS * (uint32_t)p.a_block_bytes,
                                                   (uint32_t)TC_TW * ROWB, 8 * ROWB, LAYOUT_B);
    for (int tile = slice; tile < p.total_tiles; tile += p.nslices) {
      const bool bias_tile = do_bias && bias_it == bias_phase;
      if (++bias_it == bias_period) bias_it = 0;
      for (int gi = 0; gi < ngroups; ++gi) {
        const TwGroup& g = p.g[sg][gi];
        if (!share_a || gi == 0) {
          mbar_wait(&full_bar[stage], phase, p.error_flag, 13);
          tc_fence_after();
        }
        const uint32_t a_lo = a_lo0 + (uint32_t)stage * stage_units;
        const uint32_t b_lo_s = b_lo0 + (uint32_t)stage * stage_units + (share_a ? (uint32_t)gi * group_units : 0u);
        const int ntaps = g.ntaps;
        if (bias_tile && gi == 0) {
          // d(bias) column: dz^T . ones, once per pixel tile
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_bf16_lh2_p(tmem_base + (uint32_t)(3 * BNW), a_lo + (uint32_t)k * ROWA, a_hi, ones_lo, b_hi, idesc_bias,
                            (k > 0 ? 1u : bias_started), leader);
          bias_started = 1u;
        }
        if (merge3) {
          // slots 0..2 are adjacent TMEM column ranges and rows 0..2 of the halo box are adjacent tile rows
          const uint32_t b_lo = b3_lo0 + (uint32_t)stage * stage_units;
          const uint32_t acc0 = started & 1u;
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_bf16_lh2_p(tmem_base, a_lo + (uint32_t)k * ROWA, a_hi, b_lo + (uint32_t)k * ROWB, b_hi, idesc3,
                            (k > 0 ? 1u : acc0), leader);
          started |= 7u;
        } else if (merge2 && ntaps == 2) {
          const int slot = g.slot[0];   // slots slot, slot + 1 <-> box rows ro[0], ro[0] + 1
          const uint32_t b_lo = b2_lo0 + (uint32_t)stage * stage_units + (share_a ? (uint32_t)gi * group_units : 0u) +
                                (((uint32_t)(g.ro[0] * TC_TW) * ROWB) >> 4);
          const uint32_t acc0 = (started >> slot) & 1u;
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_bf16_lh2_p(tmem_base + (uint32_t)(slot * BNW), a_lo + (uint32_t)k * ROWA, a_hi, b_lo + (uint32_t)k * ROWB, b_hi,
                            idesc2, (k > 0 ? 1u : acc0), leader);
          started |= 3u << slot;
        } else
        for (int tp = 0; tp < ntaps; ++tp) {
          const int slot = g.slot[tp];
          const uint32_t d_tmem = tmem_base + (uint32_t)(slot * BNW);
          const uint32_t b_lo = b_lo_s + (((uint32_t)(g.ro[tp] * TC_TW) * ROWB) >> 4);
          const uint32_t acc0 = (started >> slot) & 1u;
          umma_bf16_lh2_p(d_tmem, a_lo, a_hi, b_lo, b_hi, idesc, acc0, leader);
#pragma unroll
          for (int k = 1; k < 8; ++k)  // 8 x 16 pixels = one 8x16 tile; 16 pixel rows = ROW bytes = ROW/16 x 16 units
            umma_bf16_lh2_p(d_tmem, a_lo + (uint32_t)k * ROWA, a_hi, b_lo + (uint32_t)k * ROWB, b_hi, idesc, 1u, leader);
          started |= 1u << slot;
        }
        if (!share_a || gi == ngroups - 1) {
          umma_commit_p(&empty_bar[stage], leader);
          if (++stage == nstages) { stage = 0; phase ^= 1u; }
        }
      }
    }
    umma_commit_p(&done_bar[0], leader);
    __syncwarp();
  } else {
    // epilogue: once, after the last MMA retired
    const int q = warp & 3;
    const int row = q * 32 + lane;  // cout inside the M tile
    mbar_wait(&done_bar[0], 0, p.error_flag, 14);
    tc_fence_after();
    const bool any_tile = slice < p.total_tiles;
    float* dst = p.partial + ((size_t)blockIdx.x * 3) * 128 * BNW;
    if (do_bias) {
      uint32_t v[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = 0u;
      // this unit took tiles slice + (bias_phase + k * bias_period) * nslices: at least one exists iff the first does
      if (slice + (long long)bias_phase * p.nslices < p.total_tiles) {
        tmem_ld16(tmem_base + (uint32_t)(3 * BNW) + ((uint32_t)(q * 32) << 16), v);
        tmem_ld_wait();
      }
      p.bias_partial[(size_t)blockIdx.x * 128 + row] = __uint_as_float(v[0]);
    }
    for (int r = 0; r < 3; ++r) {
      for (int j = 0; j < BNW / 16; ++j) {
        uint32_t v[16];
        if (any_tile) {
          tmem_ld16(tmem_base + (uint32_t)(p.row_slot[r] * BNW + j * 16) + ((uint32_t)(q * 32) << 16), v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = 0u;
        }
        float4* o = reinterpret_cast<float4*>(dst + ((size_t)r * 128 + row) * BNW + j * 16);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          o[i] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]), __uint_as_float(v[4 * i + 2]),
                             __uint_as_float(v[4 * i + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// Sums the per-CTA partials in a fixed order.  The kernel ran on (possibly W-folded) dimensions Coutf = g*Cout,
// Cinf = g*Cin; a real weight (co, ci, r, s) collects every folded position (q, pi, s') with
// s = g*(s'-1) + pi - q + 1 (g = 1: the identity).
// The blocks from nb_w on sum d(bias) (same launch: one kernel less per layer):
// d(bias)[co] = sum over the CTAs that share the M tile and over the W-fold sub-pixels q of the bias-column
// partials [cta][128]  (cta = unit + nunits * slice, unit = s + ncols * (mtile + n_mtiles * ntile))
__global__ void wgrad_tc_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, int Cout, int Cin,
                                       int g, int BNW, int n_mtiles, int nunits, int nslices, float clip, int nb_w,
                                       const float* __restrict__ bias_part, float* __restrict__ dbias, int ncols, int grid_ctas) {
  if ((int)blockIdx.x >= nb_w) {
    // one warp per output channel: the lanes stride over the CTAs (independent loads in flight), then a shuffle reduction
    const int co = (((int)blockIdx.x - nb_w) * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (co >= Cout) return;
    float acc = 0.f;
    for (int b = lane; b < grid_ctas; b += 32) {
      const int mt = ((b % nunits) / ncols) % n_mtiles;
      for (int q = 0; q < g; ++q) {
        const int cof = q * Cout + co;
        if (cof / 128 == mt) acc += bias_part[(size_t)b * 128 + cof % 128];
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) dbias[co] = clampf(acc, clip);
    return;
  }
  // thread order [co][r][s][ci] (ci fastest): a warp reads consecutive floats of a partial row; the OIHW store is strided but tiny.
  // The per-element summation order (fold position, then slice) is fixed, so the result does not depend on this mapping.
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= (long long)Cout * Cin * 9) return;
  const int ci = (int)(j % Cin), s = (int)((j / Cin) % 3), r = (int)((j / (3LL * Cin)) % 3);
  const int co = (int)(j / (9LL * Cin));
  const long long i = (((long long)co * Cin + ci) * 3 + r) * 3 + s;
  float acc = 0.f;
  for (int sp = 0; sp < 3; ++sp)
    for (int q = 0; q < g; ++q) {
      const int pi = s - 1 + q - g * (sp - 1);
      if (pi < 0 || pi >= g) continue;
      const int cof = q * Cout + co, cif = pi * Cin + ci;
      const int mt = cof / 128, nt = cif / BNW;
      const int unit = sp + 3 * (mt + n_mtiles * nt);
#pragma unroll 8
      for (int sl = 0; sl < nslices; ++sl) {   // independent loads, adds in slice order
        const size_t cta = (size_t)unit + (size_t)nunits * sl;
        acc += __ldg(&partial[((cta * 3 + r) * 128 + (cof % 128)) * BNW + (cif % BNW)]);
      }
    }
  dw[i] = clampf(acc, clip);
}

// per-channel sum over pixels (conv bias gradient), deterministic two-stage
template <typename T>
__global__ void colsum_partial_kernel(const T* __restrict__ g, float* __restrict__ partial, long long npix, int C) {
  const int c = blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const long long per = (npix + gridDim.x - 1) / gridDim.x;
  const long long p0 = blockIdx.x * per;
  long long p1 = p0 + per;
  if (p1 > npix) p1 = npix;
  float s = 0.f;
  for (long long q = p0; q < p1; ++q) s += to_f<T>(g[q * C + c]);
  partial[(long long)blockIdx.x * C + c] = s;
}
__global__ void colsum_final_kernel(const float* __restrict__ partial, float* __restrict__ out, int C, int nblk, float clip) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  for (int b = 0; b < nblk; ++b) s += partial[(long long)b * C + c];
  out[c] = clampf(s, clip);
}
constexpr int COLSUM_BLOCKS = 592;

static int wgrad_bnw(int Cin, int kb) {
  if (Cin <= 128) return Cin;
  for (int bn = 128; bn >= kb; bn -= kb)
    if (Cin % bn == 0) return bn;
  return 0;
}

bool tc_wgrad_supported(int dtype, int W, int Cin, int Cout, int ks, int stride) {
  if (dtype != YG_BF16 || ks != 3 || (stride != 1 && stride != 2)) return false;
  const int g = fold_factor(Cin, Cout, W, stride);
  Cin *= g; Cout *= g;
  if (Cout % 32 != 0) return false;
  const int kb = pick_kc(Cin);
  return kb != 0 && wgrad_bnw(Cin, kb) != 0;
}

static void wgrad_grid(int Cin, int Cout, int* nunits, int* nslices, int* grid, int* bnw, int* n_mtiles, int* n_ntiles,
                       int ncols = 3) {
  const int kb = pick_kc(Cin);
  *bnw = wgrad_bnw(Cin, kb);
  *n_mtiles = (Cout + 127) / 128;
  *n_ntiles = Cin / *bnw;
  *nunits = ncols * *n_mtiles * *n_ntiles;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int sl = sms / *nunits;
  if (sl < 1) sl = 1;
  *nslices = sl;
  *grid = *nunits * sl;
}

size_t tc_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int ks, int stride) {
  if (!tc_wgrad_supported(YG_BF16, W, Cin, Cout, ks, stride)) return 0;
  const int g = fold_factor(Cin, Cout, W, stride);
  Cin *= g; Cout *= g;
  int nunits, nslices, grid, bnw, nm, nn;
  wgrad_grid(Cin, Cout, &nunits, &nslices, &grid, &bnw, &nm, &nn);
  return (size_t)grid * 3 * 128 * bnw * sizeof(float) + (size_t)COLSUM_BLOCKS * Cout * sizeof(float) + 256;
}

int conv_wgrad_tc(const void* x, const void* dz, float* dw, float* dbias, int N, int H, int W, int Cin, int Cout, int ks,
                  int stride, float clip, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (!get_encode()) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return YG_ERR_CUDA; }
  const size_t need = tc_wgrad_workspace(N, H, W, Cin, Cout, ks, stride);
  if (!ws || ws_bytes < need) { set_error("conv_wgrad_tc: workspace %zu < %zu", ws_bytes, need); return YG_ERR_WORKSPACE; }
  // W-folded view (see pack_weights_kernel): from here on W, Cin, Cout are the folded dimensions
  const int fg = fold_factor(Cin, Cout, W, stride);
  const int Cin_r = Cin, Cout_r = Cout, Wo_r = (W + 2 - 3) / stride + 1;
  W /= fg; Cin *= fg; Cout *= fg;
  const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
  TwMaps maps;
  memset(&maps, 0, sizeof(maps));
  TwParams p;
  memset(&p, 0, sizeof(p));
  int grid;
  wgrad_grid(Cin, Cout, &p.nunits, &p.nslices, &grid, &p.BNW, &p.n_mtiles, &p.n_ntiles);
  const int kb = pick_kc(Cin);
  p.kb = kb; p.nbblocks = p.BNW / kb;
  p.ncols = 3;
  for (int r = 0; r < 3; ++r) p.row_slot[r] = r;
  // stride 2 with one B block per tap: filter rows 0 and 2 take the adjacent slots 0 and 1 so that one MMA covers both
  if (stride == 2 && p.BNW == kb) { p.merge2 = 1; p.row_slot[0] = 0; p.row_slot[2] = 1; p.row_slot[1] = 2; }
  // base L4 wgrad 0.50 -> 0.38 ms (1235 TFLOP/s): three N = 64 MMAs (48 cycles each, bound by the shared-memory operand fetch)
  // become one N = 192 MMA (96 cycles of math, 80 of fetch); results are bit-identical.
  p.merge3 = (stride == 1 && kb == 64 && p.BNW == 64) ? 1 : 0;
  p.N = N; p.Cin = Cin; p.Cout = Cout;
  p.tiles_h = cdiv(Ho, TC_TH); p.tiles_w = cdiv(Wo, TC_TW);
  p.total_tiles = N * p.tiles_h * p.tiles_w;
  const int max_rows = stride == 1 ? TC_TH + 2 : TC_TH + 1;
  const int ka = (Cout % 64 == 0) ? 64 : 32;
  p.a_block_bytes = TC_TH * TC_TW * ka * 2;
  p.b_block_bytes = (max_rows * TC_TW * kb * 2 + 1023) & ~1023;
  p.stage_bytes = (128 / ka) * p.a_block_bytes + p.nbblocks * p.b_block_bytes;
  // stride 2: both parity groups of a tile in one stage, sharing the dz tile
  {
    const int shared_stage = (128 / ka) * p.a_block_bytes + 2 * p.nbblocks * p.b_block_bytes;
    if (stride == 2 && TC_SMEM_BUDGET / shared_stage >= 2) {
      p.share_a = 1;
      p.stage_bytes = shared_stage;
    }
  }
  int nst = TC_SMEM_BUDGET / p.stage_bytes;
  if (nst > 6) nst = 6;
  if (nst < 2) { set_error("conv_wgrad_tc: stage of %d bytes does not fit twice", p.stage_bytes); return YG_ERR_INVALID; }
  p.nstages = nst;
  // the bias column needs 16 more TMEM columns; without room for them the column sums come from a separate pass
  const bool bias_col = dbias != nullptr && 3 * p.BNW + 16 <= 512;
  int cols = 32;
  while (cols < 3 * p.BNW + (bias_col ? 16 : 0)) cols <<= 1;
  p.tmem_cols = cols;
  p.do_bias = bias_col ? 1 : 0;
  p.bias_partial = (float*)((char*)ws + (size_t)grid * 3 * 128 * p.BNW * sizeof(float));
  int rc;
  {
    uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)Cout * 2, (uint64_t)Wo * Cout * 2, (uint64_t)Ho * Wo * Cout * 2};
    uint32_t box[4] = {(uint32_t)ka, TC_TW, TC_TH, 1};
    rc = make_map(&maps.a, dz, 4, dims, str, box, ka);
    if (rc) return rc;
  }
  const bf16* xb = (const bf16*)x;
  if (stride == 1) {
    uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
    uint32_t box[4] = {(uint32_t)kb, TC_TW, TC_TH + 2, 1};
    rc = make_map(&maps.b[0], xb, 4, dims, str, box, kb);
    if (rc) return rc;
    for (int i = 1; i < 4; ++i) maps.b[i] = maps.b[0];
    p.ngroups = 1;
    for (int s = 0; s < 3; ++s) {
      TwGroup& g = p.g[s][0];
      g.map = 0; g.dh = -1; g.dw = s - 1; g.rows = TC_TH + 2; g.ntaps = 3;
      for (int r = 0; r < 3; ++r) { g.ro[r] = r; g.slot[r] = r; }
    }
  } else {
    for (int ph = 0; ph < 2; ++ph)
      for (int pw = 0; pw < 2; ++pw) {
        const int H2 = (H - ph + 1) / 2, W2 = (W - pw + 1) / 2;
        if (H2 < 1 || W2 < 1) { set_error("conv_wgrad_tc: image too small for stride 2"); return YG_ERR_INVALID; }
        uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W2, (uint64_t)H2, (uint64_t)N};
        uint64_t str[3] = {(uint64_t)2 * Cin * 2, (uint64_t)2 * W * Cin * 2, (uint64_t)H * W * Cin * 2};
        uint32_t box[4] = {(uint32_t)kb, TC_TW, (uint32_t)(ph ? TC_TH + 1 : TC_TH), 1};
        rc = make_map(&maps.b[ph * 2 + pw], xb + ((long long)ph * W + pw) * Cin, 4, dims, str, box, kb);
        if (rc) return rc;
      }
    p.ngroups = 2;
    for (int s = 0; s < 3; ++s) {
      const int pw = (s == 1) ? 0 : 1, dw_ = (s == 0) ? -1 : 0;
      TwGroup& g1 = p.g[s][0];
      g1.map = 2 + pw; g1.dh = -1; g1.dw = dw_; g1.rows = TC_TH + 1; g1.ntaps = 2;
      g1.ro[0] = 0; g1.slot[0] = p.row_slot[0];
      g1.ro[1] = 1; g1.slot[1] = p.row_slot[2];
      TwGroup& g0 = p.g[s][1];
      g0.map = pw; g0.dh = 0; g0.dw = dw_; g0.rows = TC_TH; g0.ntaps = 1;
      g0.ro[0] = 0; g0.slot[0] = p.row_slot[1];
    }
  }
  p.partial = (float*)ws;
  if (!g_error_flag) {
    YG_CUDA(cudaMalloc(&g_error_flag, sizeof(int)));
    YG_CUDA(cudaMemset(g_error_flag, 0, sizeof(int)));
  }
  p.error_flag = g_error_flag;
  const size_t smem = (size_t)nst * p.stage_bytes + 1024 + 1024 + 2048;   // align slack, barriers, ones block
#define TW_LAUNCH(KBV, KAV)                                                                                            \
  do {                                                                                                                   \
    YG_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel<KBV, KAV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   \
    wgrad_tc_kernel<KBV, KAV><<<grid, 192, smem, st>>>(maps, p);                                                         \
  } while (0)
  if (ka == 64) {
    if (kb == 64) TW_LAUNCH(64, 64); else if (kb == 32) TW_LAUNCH(32, 64); else TW_LAUNCH(16, 64);
  } else {
    if (kb == 64) TW_LAUNCH(64, 32); else if (kb == 32) TW_LAUNCH(32, 32); else TW_LAUNCH(16, 32);
  }
#undef TW_LAUNCH
  YG_LAUNCH_CHECK("wgrad_tc_kernel");
  const long long nw = (long long)Cout_r * Cin_r * 9;
  const int nb_w = (int)cdiv(nw, 256), nb_b = bias_col ? (int)cdiv(Cout_r * 32, 256) : 0;
  wgrad_tc_reduce_kernel<<<nb_w + nb_b, 256, 0, st>>>((const float*)ws, dw, Cout_r, Cin_r, fg, p.BNW, p.n_mtiles, p.nunits, p.nslices,
                                                      clip, nb_w, p.bias_partial, dbias, p.ncols, grid);
  YG_LAUNCH_CHECK("wgrad_tc_reduce");
  if (!bias_col && dbias) {
    float* part = (float*)((char*)ws + (size_t)grid * 3 * 128 * p.BNW * sizeof(float));
    const long long npix = (long long)N * Ho * Wo_r;   // the bias gradient is taken on the real (unfolded) view
    const int nblk = (int)(npix < COLSUM_BLOCKS ? npix : COLSUM_BLOCKS);
    dim3 g2(nblk, cdiv(Cout_r, 128));
    colsum_partial_kernel<bf16><<<g2, 128, 0, st>>>((const bf16*)dz, part, npix, Cout_r);
    YG_LAUNCH_CHECK("colsum_partial");
    colsum_final_kernel<<<cdiv(Cout_r, 128), 128, 0, st>>>(part, dbias, Cout_r, nblk, clip);
    YG_LAUNCH_CHECK("colsum_final");
  }
  return YG_OK;
}

// Launch the engine on an already described problem.
static int launch_engine(TcMaps& maps, TcParams& p, int KCc, int mode, int max_rows, cudaStream_t st) {
  (void)max_rows;
  const bool two_d = p.TH != 0;   // 2-D halo boxes: the builder set the tile shape
  if (!two_d) { p.TH = TC_TH; p.TW = TC_TW; }
  p.tw_shift = p.TW == 16 ? 4 : 3;
  // box sizes from the groups (legacy groups leave cols = 0: TC_TW wide per-filter-column boxes)
  int max_box = 0, max_taps = 1, ngroups_all = 0;
  for (int c = 0; c < p.ncls; ++c) ngroups_all = std::max(ngroups_all, p.cls[c].g0 + p.cls[c].ng);
  for (int gi = 0; gi < ngroups_all; ++gi) {
    if (p.g[gi].cols == 0) p.g[gi].cols = TC_TW;
    max_box = std::max(max_box, p.g[gi].rows * p.g[gi].cols * KCc * 2);
    max_taps = std::max(max_taps, p.g[gi].ntaps);
  }
  p.a_box_bytes = (max_box + 1023) & ~1023;
  p.bt_stride = max_taps;
  // small-K layers: merge all tap groups of a K chunk into one pipeline item, so that the fixed per-item
  // cost (mbarrier round trips, MMA issue, commit) is paid once per tile instead of 3-6 times
  p.b_tap_bytes = (p.cta2 ? p.BN / 2 : p.BN) * KCc * 2;
  if (p.ntaps_total == 0) p.ntaps_total = 9;
  const int resb = (p.ntaps_total * p.kchunks * p.b_tap_bytes + 1023) & ~1023;
  const int merge_limit = two_d ? 48 * 1024 : 32 * 1024;
  for (int merge = 1; merge >= 0; --merge) {
    int max_gpi = 1;
    for (int c = 0; c < p.ncls; ++c) {
      p.cls[c].gpi = (merge && p.cls[c].ng * p.a_box_bytes <= merge_limit) ? p.cls[c].ng : 1;
      if (p.cls[c].gpi > max_gpi) max_gpi = p.cls[c].gpi;
    }
    p.a_stage_bytes = max_gpi * p.a_box_bytes;
    p.b_stage_bytes = max_gpi * p.bt_stride * p.b_tap_bytes;
    // resident weights: all 9 x kchunks tiles stay in smem if at least 3 A stages still fit
    p.b_resident = 0;
    p.resb_bytes = 0;
    if (p.n_ntiles == 1 && (TC_SMEM_BUDGET - resb) / p.a_stage_bytes >= 3) {
      p.b_resident = 1;
      p.resb_bytes = resb;
    }
    // merged items with streamed weights can outgrow shared memory: fall back to one group per item
    if (p.b_resident || TC_SMEM_BUDGET / (p.a_stage_bytes + p.b_stage_bytes) >= 3) break;
  }
  if (two_d && !p.b_resident) { set_error("tcgen05 conv: 2-D halo boxes need resident weights"); return YG_ERR_INVALID; }
  const int stage_bytes = p.a_stage_bytes + (p.b_resident ? 0 : p.b_stage_bytes);
  int nst = (TC_SMEM_BUDGET - p.resb_bytes) / stage_bytes;
  // Four stages at most: deeper A pipelines are not faster anywhere and measurably slower where the producer can run far ahead
  // (same box, ms: L3 dgrad 0.350 with every stage that fits, 0.331 / 0.325 / 0.323 with 6 / 4 / 3; CTA-pair L4 dgrad 0.439 /
  // 0.439 / 0.428 / 0.429).
  if (nst > 4) nst = 4;
  if (nst < 2) {
    set_error("tcgen05 conv: stage of %d bytes does not fit twice in shared memory", stage_bytes);
    return YG_ERR_INVALID;
  }
  p.nstages = nst;
  // as many TMEM accumulators as fit in the 512 columns (up to 4): decouples MMA bursts from the epilogue
  p.nacc = 512 / p.BN;
  if (p.nacc > 4) p.nacc = 4;
  int cols = 32;
  while (cols < p.nacc * p.BN) cols <<= 1;
  p.tmem_cols = cols;
  if (!g_error_flag) {
    YG_CUDA(cudaMalloc(&g_error_flag, sizeof(int)));
    YG_CUDA(cudaMemset(g_error_flag, 0, sizeof(int)));
  }
  // MMA issue list (see TcParams::flat_ab) in issue order: group, tap, 16-wide K step.  The structurally zero K steps of
  // W-folded layers differ per K chunk, so those layers get one list per chunk.
  {
    const int ksteps = KCc / 16;
    const uint32_t layout = KCc == 64 ? 2u : (KCc == 32 ? 4u : 6u);
    bool masked = false;
    for (int gi = 0; gi < ngroups_all; ++gi)
      for (int tp = 0; tp < p.g[gi].ntaps; ++tp) masked = masked || p.g[gi].kmask[tp] != 0xFFFFFFFFu;
    const int nlists = masked ? p.kchunks : 1;
    if (nlists > TC_MAX_LISTS || (masked && nlists * ksteps > 32)) {
      set_error("tcgen05 conv: %d K chunks of %d channels exceed the MMA issue lists", nlists, KCc);
      return YG_ERR_INVALID;
    }
    int n = 0;
    for (int L = 0; L < nlists; ++L) {
      for (int c = 0; c < p.ncls; ++c) {
        const TcClass& C = p.cls[c];
        for (int gi = C.g0; gi < C.g0 + C.ng; ++gi) {
          const TcGroup& g = p.g[gi];
          const int pos = (gi - C.g0) % C.gpi;   // position of the group inside its pipeline item
          // A descriptor high word: the 8-pixel row groups of the M = 128 operand are SBO apart.  Legacy 16-wide
          // boxes: consecutive groups are contiguous (8 pixel rows); 2-D boxes (8-wide tiles): one box row apart.
          const uint32_t sbo = (uint32_t)((two_d ? g.cols : 8) * KCc * 2);
          p.a_hi[gi] = ((sbo >> 4) & 0x3FFFu) | (1u << 14) | (layout << 29);
          p.flat_rng[L][gi] = n;
          for (int tp = 0; tp < g.ntaps; ++tp) {
            const uint32_t a_off = (uint32_t)(pos * p.a_box_bytes + (g.ro[tp] * g.cols + g.co[tp]) * KCc * 2);
            const uint32_t b_off = p.b_resident ? (uint32_t)(g.widx[tp] * p.kchunks * p.b_tap_bytes)
                                                : (uint32_t)((pos * p.bt_stride + tp) * p.b_tap_bytes);
            const unsigned km = g.kmask[tp] == 0xFFFFFFFFu ? (1u << ksteps) - 1u : (g.kmask[tp] >> (L * ksteps)) & ((1u << ksteps) - 1u);
            for (int k = 0; k < ksteps; ++k) {
              if (!((km >> k) & 1u)) continue;
              const uint32_t a = (a_off >> 4) + 2u * k, b = (b_off >> 4) + 2u * k;   // 32 bytes per K step
              if (n >= TC_MAX_MMAS || a > 0xFFFFu || b > 0xFFFFu) {
                set_error("tcgen05 conv: MMA issue list overflow (entry %d, A offset %u, B offset %u units)", n, a, b);
                return YG_ERR_INVALID;
              }
              p.flat_ab[n++] = a | (b << 16);
            }
          }
        }
      }
      p.flat_rng[L][ngroups_all] = n;
    }
    p.flat_perkc = masked ? 1 : 0;
  }
  p.error_flag = g_error_flag;
  p.debug = (g_tc_options >> 7) & 31;
  const size_t smem = (size_t)nst * stage_bytes + p.resb_bytes + 1024 /*align*/ + 512 /*barriers*/ +
                      (2 * 256 + 5 * 512 + 16) * sizeof(float) + 64;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int grid = p.total_tiles < sms ? p.total_tiles : sms;
  if (p.cta2) {
    const int padded = (p.total_tiles + 1) & ~1;
    grid = (padded < sms ? padded : sms) & ~1;
    if (KCc != 64 || mode > 1 || grid < 2 || !p.b_resident || p.n_ntiles != 1 || p.ncls != 1) {
      set_error("tcgen05 conv: CTA-pair configuration not supported");
      return YG_ERR_INVALID;
    }
  }
  p.cls_rot = grid / p.ncls > 0 ? grid / p.ncls : 1;
  {
    auto magic = [](int d) { return ((1ull << 32) + (unsigned long long)d - 1) / (unsigned long long)d; };
    p.fd_ncls = magic(p.ncls); p.fd_rot = magic(p.cls_rot); p.fd_nnt = magic(p.n_ntiles);
    p.fd_tw = magic(p.tiles_w); p.fd_th = magic(p.tiles_h); p.fd_ocr = magic(p.OCr > 0 ? p.OCr : 1);
    const long long dmax = std::max(std::max(p.ncls, p.n_ntiles), std::max(std::max(p.tiles_w, p.tiles_h), p.cls_rot));
    if ((long long)p.total_tiles * dmax >= (1ll << 32)) { set_error("tcgen05 conv: %d tiles exceed the fast-division range", p.total_tiles); return YG_ERR_INVALID; }
  }
#define TC_LAUNCH(KCV, MODEV)                                                                                           \
  do {                                                                                                                  \
    YG_CUDA(cudaFuncSetAttribute(conv_tc_kernel<KCV, MODEV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  \
    conv_tc_kernel<KCV, MODEV><<<grid, 352, smem, st>>>(maps, p);                                                       \
  } while (0)
  if (p.cta2) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(352, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (mode == 0) {
      YG_CUDA(cudaFuncSetAttribute(conv_tc_kernel<64, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      YG_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<64, 0, 1>, maps, p));
    } else {
      YG_CUDA(cudaFuncSetAttribute(conv_tc_kernel<64, 1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      YG_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<64, 1, 1>, maps, p));
    }
  } else if (mode == 0) {
    if (KCc == 64) TC_LAUNCH(64, 0); else if (KCc == 32) TC_LAUNCH(32, 0); else TC_LAUNCH(16, 0);
  } else {
    if (KCc == 64) TC_LAUNCH(64, 1); else if (KCc == 32) TC_LAUNCH(32, 1); else TC_LAUNCH(16, 1);
  }
#undef TC_LAUNCH
  YG_LAUNCH_CHECK("conv_tc_kernel");
  return YG_OK;
}

int set_tc_options(int v) {
  if (v & ~TC_OPTION_BITS) {
    set_error("yg_set_tc_options: unknown option bits 0x%x (only bits 7-11 and 21 exist)", (unsigned)(v & ~TC_OPTION_BITS));
    return YG_ERR_INVALID;
  }
  g_tc_options = v;
  return YG_OK;
}
int get_tc_options() { return g_tc_options; }
int tc_debug_read(unsigned long long* out, int n) {
  if (n > 256 * 16) n = 256 * 16;
  YG_CUDA(cudaDeviceSynchronize());
  YG_CUDA(cudaMemcpyFromSymbol(out, g_tc_dbg, (size_t)n * sizeof(unsigned long long)));
  return YG_OK;
}

// choose KC so that at least 2 stages fit
static int fit_kc(int K, int BN, int max_rows) {
  int kc = pick_kc(K);
  while (kc >= 16) {
    const int stage = ((max_rows * TC_TW * kc * 2 + 1023) & ~1023) + 3 * BN * kc * 2;
    if (K % kc == 0 && TC_SMEM_BUDGET / stage >= 2) return kc;
    kc >>= 1;
  }
  return 0;
}

// 2-D halo boxes: ONE TMA box per (tile, K chunk) - (TH+2) x (TW+2) pixels for a stride-1 3x3 - instead
// of one column-shifted box per filter column.  The tile is 16 rows x 8 pixels, so every 8-pixel row group of the
// M = 128 operand lies inside one box row and the groups are a constant SBO = box row pitch apart; a tap (r, s) is
// just a start-address offset of (r * box_cols + s) pixel rows (the 128B / 64B / 32B swizzle is a function of the
// absolute shared-memory address, so offsets that are not multiples of the 8-row atom are fine - measured bit-exact).
// 3x fewer bytes through TMA, 3x fewer pipeline items (a whole 9-tap tile is one uninterrupted MMA burst).
// Needs all weights resident in shared memory (a streamed 9-tap stage would not fit).
constexpr int T2_TH = 16, T2_TW = 8;
static bool two_d_fits(int K, int BN, int n_ntiles, int ntaps_total, int box_px, int ngroups, int* kc_out) {
  // (BN = weight rows kept per CTA: the whole N tile, or half of it for a CTA pair)
  if (n_ntiles != 1) return false;
  const int kc = pick_kc(K);
  if (!kc) return false;
  const int a_box = (box_px * kc * 2 + 1023) & ~1023;
  const int a_stage = (ngroups * a_box <= 48 * 1024) ? ngroups * a_box : a_box;
  const int resb = (ntaps_total * (K / kc) * BN * kc * 2 + 1023) & ~1023;
  if (resb + 3 * a_stage > TC_SMEM_BUDGET) return false;
  *kc_out = kc;
  return true;
}

// Packed-weight scratch: one persistent device buffer per (weight pointer, layout), allocated on first
// use and re-packed on every call (weights change every optimizer step; the pack is a ~1 us kernel).
// Persistent buffers avoid per-call cudaMallocAsync/FreeAsync traffic on the driver's memory pool.
// Calls for the same weight tensor must be issued on one stream (the library's single-stream contract).
struct PackKey {
  const void* w; int transpose; int dev;
  bool operator<(const PackKey& o) const {
    if (w != o.w) return w < o.w;
    if (transpose != o.transpose) return transpose < o.transpose;
    return dev < o.dev;
  }
};
static std::map<PackKey, std::pair<void*, size_t>> g_pack_cache;
static std::mutex g_pack_mutex;
// Keys are raw weight pointers: models that come and go (or temporaries handed in as weights) would otherwise leave their
// packed copies behind for ever.  Beyond 256 entries everything is released (after a device synchronisation - kernels in
// flight may still read the buffers) and rebuilt on demand; a training run of one model never gets there.
static void pack_cache_trim_locked() {
  if (g_pack_cache.size() < 256) return;
  cudaDeviceSynchronize();
  for (auto& kv : g_pack_cache) cudaFree(kv.second.first);
  g_pack_cache.clear();
}

static int pack_weights(const float* w, bf16** out, int Cout, int Cin, int transpose, int g, cudaStream_t st) {
  // transpose == 2: stride-2 dgrad with folded column pairs (6 slices of [2 Cin][Cout])
  const long long total = transpose == 2 ? 12LL * Cout * Cin : (long long)Cout * Cin * 9 * g * g;
  {
    std::lock_guard<std::mutex> lock(g_pack_mutex);
    int dev = 0;
    cudaGetDevice(&dev);
    PackKey key{w, transpose, dev};
    if (g_pack_cache.find(key) == g_pack_cache.end()) pack_cache_trim_locked();
    auto it = g_pack_cache.find(key);
    if (it == g_pack_cache.end() || it->second.second < (size_t)total * sizeof(bf16)) {
      void* buf = nullptr;
      YG_CUDA(cudaMalloc(&buf, total * sizeof(bf16)));
      if (it != g_pack_cache.end()) { cudaFree(it->second.first); it->second = {buf, (size_t)total * sizeof(bf16)}; }
      else g_pack_cache[key] = {buf, (size_t)total * sizeof(bf16)};
      *out = (bf16*)buf;
    } else {
      *out = (bf16*)it->second.first;
    }
  }
  if (transpose == 2) pack_weights_s2fold_kernel<<<cdiv(total, 256), 256, 0, st>>>(w, *out, Cout, Cin);
  else pack_weights_kernel<<<cdiv(total, 256), 256, 0, st>>>(w, *out, Cout, Cin, 9, transpose, g);
  YG_LAUNCH_CHECK("pack_weights");
  return YG_OK;
}

int conv_fwd_tc(const void* x, const float* w, void* y, int N, int H, int W, int Cin, int Cout, int ks, int stride,
                const FwdEpi& ep, cudaStream_t st) {
  if (!get_encode()) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return YG_ERR_CUDA; }
  // W-folded view for small-channel stride-1 layers: from here on W, Cin, Cout are the folded dimensions
  const int fg = fold_factor(Cin, Cout, W, stride);
  const int Cin_r = Cin, Cout_r = Cout;
  W /= fg; Cin *= fg; Cout *= fg;
  const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  TcParams p;
  memset(&p, 0, sizeof(p));
  const int BN = pick_bn(Cout);
  const int max_rows = stride == 1 ? TC_TH + 2 : TC_TH + 1;
  int kc2 = 0;
  const bool two_d1 = two_d_fits(Cin, BN, Cout / BN, 9, stride == 1 ? (T2_TH + 2) * (T2_TW + 2) : (T2_TH + 1) * (T2_TW + 1),
                                 stride == 1 ? 1 : 4, &kc2);
  bool two_d = two_d1;
  // weights too large to stay resident in one CTA: a CTA pair keeps half of every weight tile each (cta_group::2)
  bool cta2 = false;
  if (!two_d && Cout == BN && BN % 32 == 0 && pick_kc(Cin) == 64 &&
      two_d_fits(Cin, BN / 2, 1, 9, stride == 1 ? (T2_TH + 2) * (T2_TW + 2) : (T2_TH + 1) * (T2_TW + 1), stride == 1 ? 1 : 4, &kc2))
    two_d = cta2 = true;
  const int KCc = two_d ? kc2 : fit_kc(Cin, BN, max_rows);
  if (!KCc) { set_error("conv_fwd_tc: no K chunk fits (Cin %d Cout %d)", Cin, Cout); return YG_ERR_INVALID; }
  bf16* wp = nullptr;
  int rc = pack_weights(w, &wp, Cout_r, Cin_r, 0, fg, st);
  if (rc) return rc;
  // B map: [tap][Cout][Cin]
  {
    uint64_t dims[3] = {(uint64_t)Cin, (uint64_t)Cout, 9};
    uint64_t str[2] = {(uint64_t)Cin * 2, (uint64_t)Cin * Cout * 2};
    uint32_t box[3] = {(uint32_t)KCc, (uint32_t)(cta2 ? BN / 2 : BN), 1};
    rc = make_map(&maps.b, wp, 3, dims, str, box, KCc);
    if (rc) return rc;
  }
  p.cta2 = cta2 ? 1 : 0;
  const bf16* xb = (const bf16*)x;
  int ngroups = 0;
  if (two_d && stride == 1) {
    uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
    uint32_t box[4] = {(uint32_t)KCc, T2_TW + 2, T2_TH + 2, 1};
    rc = make_map(&maps.a[0], xb, 4, dims, str, box, KCc);
    if (rc) return rc;
    for (int i = 1; i < 4; ++i) maps.a[i] = maps.a[0];
    ngroups = 1;
    TcGroup& g = p.g[0];
    g.map = 0; g.dh = -1; g.dw = -1; g.rows = T2_TH + 2; g.cols = T2_TW + 2; g.ntaps = 9;
    for (int r = 0; r < 3; ++r)
      for (int sx = 0; sx < 3; ++sx) {
        const int t = r * 3 + sx;
        g.ro[t] = r; g.co[t] = sx; g.widx[t] = t; g.kmask[t] = fold_kmask(fg, Cin_r, sx, true);
      }
    p.TH = T2_TH; p.TW = T2_TW;
  } else if (two_d) {
    // stride 2: one box per parity sub-grid (ph, pw); input row 2*ho + r - 1: r=1 -> (ph=0, h2=ho), r=0 -> (ph=1, ho-1),
    // r=2 -> (ph=1, ho); same for columns
    for (int ph = 0; ph < 2; ++ph)
      for (int pw = 0; pw < 2; ++pw) {
        const int H2 = (H - ph + 1) / 2, W2 = (W - pw + 1) / 2;
        if (H2 < 1 || W2 < 1) { set_error("conv_fwd_tc: image too small for stride 2"); return YG_ERR_INVALID; }
        uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W2, (uint64_t)H2, (uint64_t)N};
        uint64_t str[3] = {(uint64_t)2 * Cin * 2, (uint64_t)2 * W * Cin * 2, (uint64_t)H * W * Cin * 2};
        uint32_t box[4] = {(uint32_t)KCc, (uint32_t)(T2_TW + pw), (uint32_t)(T2_TH + ph), 1};
        rc = make_map(&maps.a[ph * 2 + pw], xb + ((long long)ph * W + pw) * Cin, 4, dims, str, box, KCc);
        if (rc) return rc;
        TcGroup& g = p.g[ngroups++];
        g.map = ph * 2 + pw; g.dh = ph ? -1 : 0; g.dw = pw ? -1 : 0; g.rows = T2_TH + ph; g.cols = T2_TW + pw;
        g.ntaps = 0;
        for (int ri = 0; ri < (ph ? 2 : 1); ++ri)
          for (int si = 0; si < (pw ? 2 : 1); ++si) {
            const int r = ph ? (ri == 0 ? 0 : 2) : 1, sx = pw ? (si == 0 ? 0 : 2) : 1;
            const int t = g.ntaps++;
            g.ro[t] = ri; g.co[t] = si; g.widx[t] = r * 3 + sx; g.kmask[t] = 0xFFFFFFFFu;
          }
      }
    p.TH = T2_TH; p.TW = T2_TW;
  } else if (stride == 1) {
    uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
    uint32_t box[4] = {(uint32_t)KCc, TC_TW, TC_TH + 2, 1};
    rc = make_map(&maps.a[0], xb, 4, dims, str, box, KCc);
    if (rc) return rc;
    for (int i = 1; i < 4; ++i) maps.a[i] = maps.a[0];
    ngroups = 3;
    for (int s = 0; s < 3; ++s) {
      TcGroup& g = p.g[s];
      g.map = 0; g.dh = -1; g.dw = s - 1; g.rows = TC_TH + 2; g.ntaps = 3;
      for (int r = 0; r < 3; ++r) { g.ro[r] = r; g.widx[r] = r * 3 + s; g.kmask[r] = fold_kmask(fg, Cin_r, s, true); }
    }
  } else {
    // parity sub-grids: element (h2, w2) of map (ph, pw) is x[2*h2+ph][2*w2+pw]
    for (int ph = 0; ph < 2; ++ph)
      for (int pw = 0; pw < 2; ++pw) {
        const int H2 = (H - ph + 1) / 2, W2 = (W - pw + 1) / 2;
        if (H2 < 1 || W2 < 1) { set_error("conv_fwd_tc: image too small for stride 2"); return YG_ERR_INVALID; }
        uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W2, (uint64_t)H2, (uint64_t)N};
        uint64_t str[3] = {(uint64_t)2 * Cin * 2, (uint64_t)2 * W * Cin * 2, (uint64_t)H * W * Cin * 2};
        uint32_t box[4] = {(uint32_t)KCc, TC_TW, (uint32_t)(ph ? TC_TH + 1 : TC_TH), 1};
        rc = make_map(&maps.a[ph * 2 + pw], xb + ((long long)ph * W + pw) * Cin, 4, dims, str, box, KCc);
        if (rc) return rc;
      }
    // input row 2*ho + r - 1: r=0 -> (ph=1, h2=ho-1), r=1 -> (ph=0, h2=ho), r=2 -> (ph=1, h2=ho)
    ngroups = 6;
    int gi = 0;
    for (int s = 0; s < 3; ++s) {
      const int pw = (s == 1) ? 0 : 1, dw = (s == 0) ? -1 : 0;
      TcGroup& g1 = p.g[gi++];
      g1.map = 2 + pw; g1.dh = -1; g1.dw = dw; g1.rows = TC_TH + 1; g1.ntaps = 2;
      g1.ro[0] = 0; g1.widx[0] = 0 * 3 + s;
      g1.ro[1] = 1; g1.widx[1] = 2 * 3 + s;
      g1.kmask[0] = g1.kmask[1] = 0xFFFFFFFFu;
      TcGroup& g0 = p.g[gi++];
      g0.map = pw; g0.dh = 0; g0.dw = dw; g0.rows = TC_TH; g0.ntaps = 1;
      g0.ro[0] = 0; g0.widx[0] = 1 * 3 + s;
      g0.kmask[0] = 0xFFFFFFFFu;
    }
  }
  p.N = N;
  p.ncls = 1;
  p.cls[0] = TcClass{0, ngroups, 1, Ho, Wo, 0, 0};
  p.tiles_h = cdiv(Ho, two_d ? T2_TH : TC_TH); p.tiles_w = cdiv(Wo, two_d ? T2_TW : TC_TW);
  p.n_ntiles = Cout / BN;
  p.total_tiles = N * p.tiles_h * p.tiles_w * p.n_ntiles;
  p.OH = Ho; p.OW = Wo; p.OC = Cout; p.OCr = Cout_r; p.osh = p.osw = 1;
  p.BN = BN; p.kchunks = Cin / KCc;
  p.out = y;
  p.scale = ep.scale; p.shift = ep.shift; p.act = ep.act; p.dropscale = ep.dropscale; p.stats = ep.stats;
  p.preact = ep.preact;
  p.io_f32 = ep.io_f32;
  p.actmask_out = ep.actmask;
  rc = launch_engine(maps, p, KCc, 0, max_rows, st);
  return rc;
}

int conv_dgrad_tc(const void* dz, const float* w, void* dx, int N, int H, int W, int Cin, int Cout, int ks, int stride,
                  const BwdEpi& be, cudaStream_t st) {
  if (!get_encode()) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return YG_ERR_CUDA; }
  const bool s2f = s2fold_dgrad(Cin, W, stride);
  const int fg = fold_factor(Cin, Cout, W, stride);
  const int Cin_r = Cin, Cout_r = Cout;
  const int Ho = (H + 2 - 3) / stride + 1;
  int Wo;
  if (s2f) { Wo = (W + 2 - 3) / 2 + 1; W /= 2; Cin *= 2; }   // dx viewed as (N, H, W/2, 2 Cin); dz unchanged
  else { W /= fg; Cin *= fg; Cout *= fg; Wo = (W + 2 - 3) / stride + 1; }
  const int BN = pick_bn(Cin);
  const int max_rows = stride == 1 ? TC_TH + 2 : TC_TH + 1;
  int kc2 = 0;
  const bool two_d1 = two_d_fits(Cout, BN, Cin / BN, s2f ? 6 : 9,
                                 stride == 1 ? (T2_TH + 2) * (T2_TW + 2) : (T2_TH + 1) * (T2_TW + 1), 1, &kc2);
  bool two_d = two_d1, cta2 = false;
  // (no pairs for stride-2 dgrad: as four parity classes in a class-per-round tile order they measured slower, 0.64 vs 0.47 ms
  //  on base L5; its tiles carry 8-32 MMAs each and the pair's barrier round trips dominate)
  // pairs also where the weights WOULD fit one CTA when N = 64 (unfolded): an M = 128, N = 64 MMA is bound by its
  // shared-memory operand fetch (4 KB of A + 2 KB of B for 32 cycles of math); in a pair each CTA fetches half of B.
  // base L4 dgrad 0.49 -> 0.44 ms; the W-folded 16-channel layer does not gain (0.42 -> 0.43).
  const bool force_pair = two_d && stride == 1 && BN == 64 && fg == 1;
  if ((!two_d || force_pair) && stride == 1 && Cin == BN && BN % 32 == 0 &&
      pick_kc(Cout) == 64 &&
      two_d_fits(Cout, BN / 2, 1, 9, stride == 1 ? (T2_TH + 2) * (T2_TW + 2) : (T2_TH + 1) * (T2_TW + 1), 1, &kc2))
    two_d = cta2 = true;   // CTA pair, see conv_fwd_tc
  const int KCc = two_d ? kc2 : fit_kc(Cout, BN, max_rows);
  if (!KCc) { set_error("conv_dgrad_tc: no K chunk fits (Cin %d Cout %d)", Cin, Cout); return YG_ERR_INVALID; }
  bf16* wp = nullptr;
  int rc = pack_weights(w, &wp, Cout_r, Cin_r, s2f ? 2 : 1, fg, st);
  if (rc) return rc;
  const bf16* gb = (const bf16*)dz;
  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  TcParams p;
  memset(&p, 0, sizeof(p));
  {
    uint64_t dims[3] = {(uint64_t)Cout, (uint64_t)Cin, (uint64_t)(s2f ? 6 : 9)};
    uint64_t str[2] = {(uint64_t)Cout * 2, (uint64_t)Cin * Cout * 2};
    uint32_t box[3] = {(uint32_t)KCc, (uint32_t)(cta2 ? BN / 2 : BN), 1};
    rc = make_map(&maps.b, wp, 3, dims, str, box, KCc);
    if (rc) return rc;
  }
  p.cta2 = cta2 ? 1 : 0;
  // A maps over dz: map 0 has the tallest box of the problem, map 1 (stride 2 only) the 8-row box
  for (int mi = 0; mi < 2 && !two_d; ++mi) {
    const int rows = stride == 1 ? TC_TH + 2 : (mi == 0 ? TC_TH + 1 : TC_TH);
    uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)Cout * 2, (uint64_t)Wo * Cout * 2, (uint64_t)Ho * Wo * Cout * 2};
    uint32_t box[4] = {(uint32_t)KCc, TC_TW, (uint32_t)rows, 1};
    rc = make_map(&maps.a[mi], gb, 4, dims, str, box, KCc);
    if (rc) return rc;
  }
  maps.a[2] = maps.a[0]; maps.a[3] = maps.a[0];
  // 2-D halo boxes over dz (see two_d_fits): map index = box shape (rows = T2_TH + a, cols = T2_TW + b)
  auto dz_map = [&](int mi, int rows, int cols) -> int {
    uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)Cout * 2, (uint64_t)Wo * Cout * 2, (uint64_t)Ho * Wo * Cout * 2};
    uint32_t box[4] = {(uint32_t)KCc, (uint32_t)cols, (uint32_t)rows, 1};
    return make_map(&maps.a[mi], gb, 4, dims, str, box, KCc);
  };
  if (two_d && stride == 1) {
    // dx(h,w) = sum_{r,s} dz(h+1-r, w+1-s) W[r][s]^T: box origin (h-1, w-1), tap (r,s) at box offset (2-r, 2-s)
    rc = dz_map(0, T2_TH + 2, T2_TW + 2);
    if (rc) return rc;
    for (int i = 1; i < 4; ++i) maps.a[i] = maps.a[0];
    TcGroup& g = p.g[0];
    g.map = 0; g.dh = -1; g.dw = -1; g.rows = T2_TH + 2; g.cols = T2_TW + 2; g.ntaps = 9;
    for (int r = 0; r < 3; ++r)
      for (int sx = 0; sx < 3; ++sx) {
        const int t = r * 3 + sx;
        g.ro[t] = 2 - r; g.co[t] = 2 - sx; g.widx[t] = t; g.kmask[t] = fold_kmask(fg, Cout_r, sx, false);
      }
    p.ncls = 1;
    p.cls[0] = TcClass{0, 1, 1, H, W, 0, 0};
    p.osh = p.osw = 1;
    p.TH = T2_TH; p.TW = T2_TW;
    p.tiles_h = cdiv(H, T2_TH); p.tiles_w = cdiv(W, T2_TW);
  } else if (two_d && s2f) {
    // two row-parity classes over the column-pair-folded dx; taps (r, dxo) read dz (a + [r==0], x' + dxo)
    for (int qh = 0; qh < 2; ++qh) {
      rc = dz_map(qh, T2_TH + qh, T2_TW + 1);
      if (rc) return rc;
      TcClass& C = p.cls[qh];
      C.g0 = qh; C.ng = 1; C.TSH = (H - qh + 1) / 2; C.TSW = W; C.oh0 = qh; C.ow0 = 0; C.gpi = 1;
      TcGroup& g = p.g[qh];
      g.map = qh; g.dh = 0; g.dw = 0; g.rows = T2_TH + qh; g.cols = T2_TW + 1; g.ntaps = 0;
      for (int ri = 0; ri < (qh ? 2 : 1); ++ri)
        for (int dxo = 0; dxo < 2; ++dxo) {
          const int r = qh ? (ri == 0 ? 0 : 2) : 1;
          const int t = g.ntaps++;
          g.ro[t] = qh ? (r == 0 ? 1 : 0) : 0; g.co[t] = dxo; g.widx[t] = r * 2 + dxo; g.kmask[t] = 0xFFFFFFFFu;
        }
    }
    maps.a[2] = maps.a[0]; maps.a[3] = maps.a[0];
    p.ncls = 2;
    p.osh = 2; p.osw = 1;
    p.ntaps_total = 6;
    p.TH = T2_TH; p.TW = T2_TW;
    p.tiles_h = cdiv((H + 1) / 2, T2_TH); p.tiles_w = cdiv(W, T2_TW);
  } else if (two_d) {
    // four output-parity classes (qh, qw), one box each: rows a .. a+qh, columns b .. b+qw of dz
    for (int cls = 0; cls < 4; ++cls) {
      const int qh = cls >> 1, qw = cls & 1;
      rc = dz_map(cls, T2_TH + qh, T2_TW + qw);
      if (rc) return rc;
      TcClass& C = p.cls[cls];
      C.g0 = cls; C.ng = 1; C.TSH = (H - qh + 1) / 2; C.TSW = (W - qw + 1) / 2; C.oh0 = qh; C.ow0 = qw; C.gpi = 1;
      TcGroup& g = p.g[cls];
      g.map = cls; g.dh = 0; g.dw = 0; g.rows = T2_TH + qh; g.cols = T2_TW + qw; g.ntaps = 0;
      for (int ri = 0; ri < (qh ? 2 : 1); ++ri)
        for (int si = 0; si < (qw ? 2 : 1); ++si) {
          const int r = qh ? (ri == 0 ? 0 : 2) : 1, sx = qw ? (si == 0 ? 0 : 2) : 1;
          const int t = g.ntaps++;
          g.ro[t] = qh ? (r == 0 ? 1 : 0) : 0; g.co[t] = qw ? (sx == 0 ? 1 : 0) : 0;
          g.widx[t] = r * 3 + sx; g.kmask[t] = 0xFFFFFFFFu;
        }
    }
    p.ncls = 4;
    p.osh = p.osw = 2;
    p.TH = T2_TH; p.TW = T2_TW;
    p.tiles_h = cdiv((H + 1) / 2, T2_TH); p.tiles_w = cdiv((W + 1) / 2, T2_TW);
  } else if (stride == 1) {
    // dx(h,w) = sum_{r,s} dz(h+1-r, w+1-s) W[r][s]^T
    for (int s = 0; s < 3; ++s) {
      TcGroup& g = p.g[s];
      g.map = 0; g.dh = -1; g.dw = 1 - s; g.rows = TC_TH + 2; g.ntaps = 3;
      for (int r = 0; r < 3; ++r) { g.ro[r] = 2 - r; g.widx[r] = r * 3 + s; g.kmask[r] = fold_kmask(fg, Cout_r, s, false); }
    }
    p.ncls = 1;
    p.cls[0] = TcClass{0, 3, 1, H, W, 0, 0};
    p.osh = p.osw = 1;
    p.tiles_h = cdiv(H, TC_TH); p.tiles_w = cdiv(W, TC_TW);
  } else if (s2f) {
    // Few input channels: output column pairs (x = 2x'+q) are folded into the channel dimension, which leaves two
    // row-parity classes with N = 2 Cin and taps over dz columns x', x'+1: half the tiles, twice as wide MMAs,
    // and every output pixel pair is written as one contiguous run instead of two strided halves.
    int gi = 0;
    for (int qh = 0; qh < 2; ++qh) {
      TcClass& C = p.cls[qh];
      C.g0 = gi; C.TSH = (H - qh + 1) / 2; C.TSW = W; C.oh0 = qh; C.ow0 = 0; C.gpi = 1;
      for (int dxo = 0; dxo < 2; ++dxo) {
        TcGroup& g = p.g[gi++];
        g.map = qh ? 0 : 1; g.dh = 0; g.dw = dxo; g.rows = TC_TH + qh;
        if (qh) { g.ntaps = 2; g.ro[0] = 1; g.widx[0] = 0 * 2 + dxo; g.ro[1] = 0; g.widx[1] = 2 * 2 + dxo; }
        else { g.ntaps = 1; g.ro[0] = 0; g.widx[0] = 1 * 2 + dxo; }
        g.kmask[0] = g.kmask[1] = 0xFFFFFFFFu;
      }
      C.ng = 2;
    }
    p.ncls = 2;
    p.osh = 2; p.osw = 1;
    p.ntaps_total = 6;
    p.tiles_h = cdiv((H + 1) / 2, TC_TH); p.tiles_w = cdiv(W, TC_TW);
  } else {
    // Four output-parity classes (qh, qw): h = 2a+qh, w = 2b+qw.  qh=0: r=1 (dz row a).  qh=1: r=0 (row a+1), r=2
    // (row a); same for columns.  All four run in ONE launch with the class as the fastest tile index, so the dz
    // tile and the saved-activation lines shared by sibling classes are fetched from HBM once and hit L2 after.
    int gi = 0, nc = 0;
    for (int cls = 0; cls < 4; ++cls) {
      const int qh = cls >> 1, qw = cls & 1;
      const int TSH = (H - qh + 1) / 2, TSW = (W - qw + 1) / 2;
      TcClass& C = p.cls[nc++];
      C.g0 = gi; C.TSH = TSH; C.TSW = TSW; C.oh0 = qh; C.ow0 = qw; C.gpi = 1;
      const int ns = qw ? 2 : 1;
      for (int si = 0; si < ns; ++si) {
        const int s = qw ? (si == 0 ? 0 : 2) : 1;
        const int dw = qw ? (si == 0 ? 1 : 0) : 0;
        TcGroup& g = p.g[gi++];
        g.map = qh ? 0 : 1; g.dh = 0; g.dw = dw; g.rows = TC_TH + qh;
        if (qh) { g.ntaps = 2; g.ro[0] = 1; g.widx[0] = 0 * 3 + s; g.ro[1] = 0; g.widx[1] = 2 * 3 + s; }
        else { g.ntaps = 1; g.ro[0] = 0; g.widx[0] = 1 * 3 + s; }
        g.kmask[0] = g.kmask[1] = 0xFFFFFFFFu;
      }
      C.ng = gi - C.g0;
    }
    p.ncls = 4;
    p.osh = p.osw = 2;
    // tile space of the largest class (qh = qw = 0); smaller classes mask their last row / column
    p.tiles_h = cdiv((H + 1) / 2, TC_TH); p.tiles_w = cdiv((W + 1) / 2, TC_TW);
  }
  p.N = N;
  p.n_ntiles = Cin / BN;
  p.total_tiles = N * p.tiles_h * p.tiles_w * p.n_ntiles * p.ncls;
  p.OH = H; p.OW = W; p.OC = Cin; p.OCr = Cin_r;
  p.BN = BN; p.kchunks = Cout / KCc;
  p.out = dx;
  p.saved = be.saved; p.act = be.act; p.dropscale = be.dropscale; p.bn_scale = be.bn_scale; p.bn_shift = be.bn_shift;
  p.io_f32 = be.io_f32;
  p.bn_mean = be.bn_mean; p.bn_invstd = be.bn_invstd; p.bn_sums = be.bn_sums;
  p.actmask_in = be.actmask;
  return launch_engine(maps, p, KCc, 1, max_rows, st);
}

// ------------------------------------------------------------------------------------------------
// 1x1 prediction head backward on the tensor cores (called from head.cu):
//   dt   (N,Sy,Sx,32) bf16: gradient wrt the raw head logits, zero padded from D = 5+C to 32 channels
//   dx = dt . W    -> the dgrad engine with a single tap, K = 32, N = Cin, MODE 1 epilogue (activation / BN
//                     backward of the last conv block fused, exactly as for the 3x3 layers)
//   dW = dt^T . x  -> the wgrad engine with one column / one accumulator slot
// ------------------------------------------------------------------------------------------------
__global__ void pack_head_weights_kernel(const float* __restrict__ w, bf16* __restrict__ out, int D, int Cin, int DP) {
  // packed [1 tap][N = Cin][K = DP]: out[ci][d] = w[d][ci] (zero for d >= D)
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Cin * DP) return;
  const int d = i % DP, ci = i / DP;
  out[i] = __float2bfloat16_rn(d < D ? w[(long long)d * Cin + ci] : 0.f);
}

__global__ void head_wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, int D, int Cin,
                                         int BNW, int n_mtiles, int nunits, int nslices, float clip) {
  // one warp per [d][ci] element: the lanes stride over the ~148 slices (independent loads in flight instead of one serial
  // chain per thread), then a fixed shuffle tree - the order of the summation does not depend on the launch
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= D * Cin) return;
  const int ci = i % Cin, d = i / Cin;
  const int nt = ci / BNW;
  const int unit = 0 + 1 * (0 + n_mtiles * nt);
  float acc = 0.f;
  for (int sl = lane; sl < nslices; sl += 32) {
    const size_t cta = (size_t)unit + (size_t)nunits * sl;
    acc += partial[((cta * 3 + 0) * 128 + d) * BNW + (ci % BNW)];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) dw[i] = clampf(acc, clip);
}

bool head_bwd_tc_supported(int Cin, int D) {
  if (D > 32 || Cin % 16 != 0 || Cin > 512) return false;
  const int kb = pick_kc(Cin);
  return pick_bn(Cin) != 0 && kb != 0 && wgrad_bnw(Cin, kb) != 0;
}

size_t head_bwd_tc_workspace(int Cin) {
  int nunits, nslices, grid, bnw, nm, nn;
  wgrad_grid(Cin, 32, &nunits, &nslices, &grid, &bnw, &nm, &nn, 1);
  return (size_t)grid * 3 * 128 * bnw * sizeof(float) + 256;
}

__global__ void pack_head_weights_fwd_kernel(const float* __restrict__ w, bf16* __restrict__ out, int D, int Cin) {
  // packed [1 tap][N = 16][K = Cin]: rows d >= D are zero
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 16 * Cin) return;
  const int ci = i % Cin, d = i / Cin;
  out[i] = __float2bfloat16_rn(d < D ? w[(long long)d * Cin + ci] : 0.f);
}

bool head_fwd_tc_supported(int Cin, int D) { return D <= 16 && Cin % 16 == 0 && Cin >= 16 && Cin <= 512 && pick_kc(Cin) != 0; }

// 1x1 prediction head forward on the tensor cores: one tap, N = 16 (5 + classes zero padded), K = Cin; the YOGO
// output transform runs in the epilogue (replaces head_fwd_kernel, which is shared-memory-bandwidth bound).
int head_fwd_tc(const void* x, const float* w, const float* bias, float* out, float* t_raw, int N, int Sy, int Sx, int Cin,
                int D, float aw, float ah, float wm, float hm, int inference, const float* cxs, const float* cys,
                cudaStream_t st) {
  if (!get_encode()) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return YG_ERR_CUDA; }
  bf16* wp = nullptr;
  {
    std::lock_guard<std::mutex> lock(g_pack_mutex);
    int dev = 0;
    cudaGetDevice(&dev);
    PackKey key{w, 4, dev};
    auto it = g_pack_cache.find(key);
    const size_t need = (size_t)Cin * 16 * sizeof(bf16);
    if (it == g_pack_cache.end() || it->second.second < need) {
      void* buf = nullptr;
      YG_CUDA(cudaMalloc(&buf, need));
      if (it != g_pack_cache.end()) { cudaFree(it->second.first); it->second = {buf, need}; }
      else g_pack_cache[key] = {buf, need};
      wp = (bf16*)buf;
    } else wp = (bf16*)it->second.first;
  }
  pack_head_weights_fwd_kernel<<<cdiv(16LL * Cin, 256), 256, 0, st>>>(w, wp, D, Cin);
  YG_LAUNCH_CHECK("pack_head_weights_fwd");
  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  TcParams p;
  memset(&p, 0, sizeof(p));
  const int BN = 16, KCc = pick_kc(Cin);
  const bf16* xb = (const bf16*)x;
  int rc;
  {
    uint64_t dims[3] = {(uint64_t)Cin, 16, 1};
    uint64_t str[2] = {(uint64_t)Cin * 2, (uint64_t)Cin * 16 * 2};
    uint32_t box[3] = {(uint32_t)KCc, (uint32_t)BN, 1};
    rc = make_map(&maps.b, wp, 3, dims, str, box, KCc);
    if (rc) return rc;
  }
  {
    uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)Sx, (uint64_t)Sy, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)Cin * 2, (uint64_t)Sx * Cin * 2, (uint64_t)Sy * Sx * Cin * 2};
    uint32_t box[4] = {(uint32_t)KCc, TC_TW, TC_TH, 1};
    rc = make_map(&maps.a[0], xb, 4, dims, str, box, KCc);
    if (rc) return rc;
    for (int i = 1; i < 4; ++i) maps.a[i] = maps.a[0];
  }
  TcGroup& g = p.g[0];
  g.map = 0; g.dh = 0; g.dw = 0; g.rows = TC_TH; g.ntaps = 1; g.ro[0] = 0; g.widx[0] = 0; g.kmask[0] = 0xFFFFFFFFu;
  p.ncls = 1;
  p.cls[0] = TcClass{0, 1, 1, Sy, Sx, 0, 0};
  p.osh = p.osw = 1;
  p.N = N;
  p.tiles_h = cdiv(Sy, TC_TH); p.tiles_w = cdiv(Sx, TC_TW);
  p.n_ntiles = 1;
  p.total_tiles = N * p.tiles_h * p.tiles_w;
  p.OH = Sy; p.OW = Sx; p.OC = 16; p.OCr = 16;
  p.BN = BN; p.kchunks = Cin / KCc; p.ntaps_total = 1;
  p.shift = bias;
  p.head_out = out; p.head_traw = t_raw; p.head_cxs = cxs; p.head_cys = cys;
  p.head_aw = aw; p.head_ah = ah; p.head_wm = wm; p.head_hm = hm; p.head_D = D; p.head_inf = inference;
  return launch_engine(maps, p, KCc, 0, TC_TH, st);
}

int head_bwd_tc(const void* dt, const void* x, const float* w, void* dx, float* dw, int N, int Sy, int Sx, int Cin, int D,
                const BwdEpi& be, float clip, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (!get_encode()) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return YG_ERR_CUDA; }
  constexpr int DP = 32;
  const bf16* dtb = (const bf16*)dt;
  int rc;
  // ---------------- dx = dt . W (+ fused backward epilogue of the last block)
  {
    bf16* wp = nullptr;
    {
      std::lock_guard<std::mutex> lock(g_pack_mutex);
      int dev = 0;
      cudaGetDevice(&dev);
      PackKey key{w, 2, dev};
      auto it = g_pack_cache.find(key);
      const size_t need = (size_t)Cin * DP * sizeof(bf16);
      if (it == g_pack_cache.end() || it->second.second < need) {
        void* buf = nullptr;
        YG_CUDA(cudaMalloc(&buf, need));
        if (it != g_pack_cache.end()) { cudaFree(it->second.first); it->second = {buf, need}; }
        else g_pack_cache[key] = {buf, need};
        wp = (bf16*)buf;
      } else wp = (bf16*)it->second.first;
    }
    pack_head_weights_kernel<<<cdiv((long long)Cin * DP, 256), 256, 0, st>>>(w, wp, D, Cin, DP);
    YG_LAUNCH_CHECK("pack_head_weights");
    TcMaps maps;
    memset(&maps, 0, sizeof(maps));
    TcParams p;
    memset(&p, 0, sizeof(p));
    const int BN = pick_bn(Cin), KCc = 32;
    {
      uint64_t dims[3] = {(uint64_t)DP, (uint64_t)Cin, 1};
      uint64_t str[2] = {(uint64_t)DP * 2, (uint64_t)Cin * DP * 2};
      uint32_t box[3] = {(uint32_t)KCc, (uint32_t)BN, 1};
      rc = make_map(&maps.b, wp, 3, dims, str, box, KCc);
      if (rc) return rc;
    }
    {
      uint64_t dims[4] = {(uint64_t)DP, (uint64_t)Sx, (uint64_t)Sy, (uint64_t)N};
      uint64_t str[3] = {(uint64_t)DP * 2, (uint64_t)Sx * DP * 2, (uint64_t)Sy * Sx * DP * 2};
      uint32_t box[4] = {(uint32_t)KCc, TC_TW, TC_TH, 1};
      rc = make_map(&maps.a[0], dtb, 4, dims, str, box, KCc);
      if (rc) return rc;
      for (int i = 1; i < 4; ++i) maps.a[i] = maps.a[0];
    }
    TcGroup& g = p.g[0];
    g.map = 0; g.dh = 0; g.dw = 0; g.rows = TC_TH; g.ntaps = 1; g.ro[0] = 0; g.widx[0] = 0;
    g.kmask[0] = D <= 16 ? 1u : 3u;   // the second 16-wide K step is all padding when D <= 16
    p.ncls = 1;
    p.cls[0] = TcClass{0, 1, 1, Sy, Sx, 0, 0};
    p.osh = p.osw = 1;
    p.tiles_h = cdiv(Sy, TC_TH); p.tiles_w = cdiv(Sx, TC_TW);
    p.N = N; p.n_ntiles = Cin / BN;
    p.total_tiles = N * p.tiles_h * p.tiles_w * p.n_ntiles;
    p.OH = Sy; p.OW = Sx; p.OC = Cin; p.OCr = Cin;
    p.BN = BN; p.kchunks = 1; p.ntaps_total = 1;
    p.out = dx;
    p.saved = be.saved; p.act = be.act; p.dropscale = be.dropscale; p.bn_scale = be.bn_scale; p.bn_shift = be.bn_shift;
    p.bn_mean = be.bn_mean; p.bn_invstd = be.bn_invstd; p.bn_sums = be.bn_sums;
    p.actmask_in = be.actmask;
    rc = launch_engine(maps, p, KCc, 1, TC_TH, st);
    if (rc) return rc;
  }
  // ---------------- dW = dt^T . x (skipped when the caller needs no parameter gradients)
  if (dw) {
    const size_t need = head_bwd_tc_workspace(Cin);
    if (!ws || ws_bytes < need) { set_error("head_bwd_tc: workspace %zu < %zu", ws_bytes, need); return YG_ERR_WORKSPACE; }
    TwMaps maps;
    memset(&maps, 0, sizeof(maps));
    TwParams p;
    memset(&p, 0, sizeof(p));
    int grid;
    wgrad_grid(Cin, DP, &p.nunits, &p.nslices, &grid, &p.BNW, &p.n_mtiles, &p.n_ntiles, 1);
    const int kb = pick_kc(Cin), ka = 32;
    p.kb = kb; p.nbblocks = p.BNW / kb; p.ncols = 1;
    for (int r = 0; r < 3; ++r) p.row_slot[r] = r;
    p.N = N; p.Cin = Cin; p.Cout = DP;
    p.tiles_h = cdiv(Sy, TC_TH); p.tiles_w = cdiv(Sx, TC_TW);
    p.total_tiles = N * p.tiles_h * p.tiles_w;
    p.a_block_bytes = TC_TH * TC_TW * ka * 2;
    p.b_block_bytes = (TC_TH * TC_TW * kb * 2 + 1023) & ~1023;
    p.stage_bytes = (128 / ka) * p.a_block_bytes + p.nbblocks * p.b_block_bytes;
    int nst = TC_SMEM_BUDGET / p.stage_bytes;
    if (nst > 6) nst = 6;
    if (nst < 2) { set_error("head_bwd_tc: stage does not fit"); return YG_ERR_INVALID; }
    p.nstages = nst;
    int cols = 32;
    while (cols < 3 * p.BNW) cols <<= 1;
    p.tmem_cols = cols;
    {
      uint64_t dims[4] = {(uint64_t)DP, (uint64_t)Sx, (uint64_t)Sy, (uint64_t)N};
      uint64_t str[3] = {(uint64_t)DP * 2, (uint64_t)Sx * DP * 2, (uint64_t)Sy * Sx * DP * 2};
      uint32_t box[4] = {(uint32_t)ka, TC_TW, TC_TH, 1};
      rc = make_map(&maps.a, dtb, 4, dims, str, box, ka);
      if (rc) return rc;
    }
    {
      const bf16* xb = (const bf16*)x;
      uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)Sx, (uint64_t)Sy, (uint64_t)N};
      uint64_t str[3] = {(uint64_t)Cin * 2, (uint64_t)Sx * Cin * 2, (uint64_t)Sy * Sx * Cin * 2};
      uint32_t box[4] = {(uint32_t)kb, TC_TW, TC_TH, 1};
      rc = make_map(&maps.b[0], xb, 4, dims, str, box, kb);
      if (rc) return rc;
      for (int i = 1; i < 4; ++i) maps.b[i] = maps.b[0];
    }
    p.ngroups = 1;
    TwGroup& g = p.g[0][0];
    g.map = 0; g.dh = 0; g.dw = 0; g.rows = TC_TH; g.ntaps = 1; g.ro[0] = 0; g.slot[0] = 0;
    p.partial = (float*)ws;
    p.error_flag = g_error_flag;
    const size_t smem = (size_t)nst * p.stage_bytes + 1024 + 1024 + 2048;
#define HW_LAUNCH(KBV)                                                                                                 \
  do {                                                                                                                 \
    YG_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel<KBV, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    wgrad_tc_kernel<KBV, 32><<<grid, 192, smem, st>>>(maps, p);                                                     \
  } while (0)
    if (kb == 64) HW_LAUNCH(64); else if (kb == 32) HW_LAUNCH(32); else HW_LAUNCH(16);
#undef HW_LAUNCH
    YG_LAUNCH_CHECK("wgrad_tc_kernel(head)");
    head_wgrad_reduce_kernel<<<cdiv((long long)D * Cin * 32, 256), 256, 0, st>>>((const float*)ws, dw, D, Cin, p.BNW,
                                                                            p.n_mtiles, p.nunits, p.nslices, clip);
    YG_LAUNCH_CHECK("head_wgrad_reduce");
  }
  return YG_OK;
}



}  // namespace yg
