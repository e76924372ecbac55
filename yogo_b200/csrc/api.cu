// C-ABI glue: error reporting, device check, implementation dispatch for the convolutions.
#include "common.cuh"
#include <stdarg.h>
#include <string.h>

namespace yg {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
static int g_conv_impl = YG_IMPL_AUTO;
unsigned long long g_launches = 0;

// conv_simt.cu
int conv_fwd_simt(const void*, const float*, void*, int, int, int, int, int, int, int, int, const FwdEpi&, cudaStream_t);
int conv_dgrad_simt(const void*, const float*, void*, int, int, int, int, int, int, int, int, const BwdEpi&, cudaStream_t);
int conv_wgrad_simt(const void*, const void*, float*, float*, int, int, int, int, int, int, int, int, float, void*, size_t, cudaStream_t);
size_t simt_wgrad_workspace(int, int, int, int, int, int, int);
// conv_tc.cu
bool tc_fwd_supported(int dtype, int W, int Cin, int Cout, int ks, int stride);
bool tc_dgrad_supported(int dtype, int W, int Cin, int Cout, int ks, int stride);
bool tc_wgrad_supported(int dtype, int W, int Cin, int Cout, int ks, int stride);
int conv_fwd_tc(const void*, const float*, void*, int, int, int, int, int, int, int, const FwdEpi&, cudaStream_t);
int conv_dgrad_tc(const void*, const float*, void*, int, int, int, int, int, int, int, const BwdEpi&, cudaStream_t);
int conv_wgrad_tc(const void*, const void*, float*, float*, int, int, int, int, int, int, int, float, void*, size_t, cudaStream_t);
size_t tc_wgrad_workspace(int, int, int, int, int, int, int);
// fp32 tensors on the bf16 tensor cores (x3.cu)
bool x3_fwd_supported(int W, int Cin, int Cout, int ks, int stride);
bool x3_dgrad_supported(int W, int Cin, int Cout, int ks, int stride);
bool x3_wgrad_supported(int W, int Cin, int Cout, int ks, int stride);
size_t x3_wgrad_workspace(int, int, int, int, int, int, int);
int conv_fwd_x3(const float*, const float*, float*, int, int, int, int, int, int, int, FwdEpi, cudaStream_t);
int conv_dgrad_x3(const float*, const float*, float*, int, int, int, int, int, int, int, BwdEpi, cudaStream_t);
int conv_wgrad_x3(const float*, const float*, float*, float*, int, int, int, int, int, int, int, float, void*, size_t, cudaStream_t);
bool wgrad_hmma_supported(int dtype, int W, int Cin, int Cout, int ks, int stride);
size_t wgrad_hmma_workspace(int Cin, int Cout);
int conv_wgrad_hmma(const void*, const void*, float*, float*, int, int, int, int, int, int, int, float, void*, size_t, cudaStream_t);
int set_tc_options(int);
int get_tc_options();
int tc_debug_read(unsigned long long*, int);

static int check_conv_args(const char* who, int dtype, int N, int H, int W, int Cin, int Cout, int ks, int stride) {
  YG_CHECK_ARG(dtype == YG_F32 || dtype == YG_BF16, "%s: dtype %d", who, dtype);
  YG_CHECK_ARG(ks == 1 || ks == 3, "%s: ksize %d (1 or 3)", who, ks);
  YG_CHECK_ARG(stride == 1 || stride == 2, "%s: stride %d (1 or 2)", who, stride);
  YG_CHECK_ARG(N >= 0 && H >= 1 && W >= 1 && Cin >= 1 && Cout >= 1, "%s: bad shape", who);
  return YG_OK;
}

}  // namespace yg
using namespace yg;

extern "C" int yg_version(void) { return 100; }
extern "C" unsigned long long yg_launch_count(void) { return g_launches; }
extern "C" const char* yg_last_error(void) { return g_err; }

extern "C" int yg_device_check(void) {
  int dev = 0;
  YG_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  YG_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) {
    set_error("yogo_b200 needs an sm_100 device, found sm_%d%d (%s)", prop.major, prop.minor, prop.name);
    return YG_ERR_ARCH;
  }
  return YG_OK;
}

extern "C" int yg_set_conv_impl(int impl) {
  YG_CHECK_ARG(impl >= YG_IMPL_AUTO && impl <= YG_IMPL_TCGEN05, "set_conv_impl: %d", impl);
  g_conv_impl = impl;
  return YG_OK;
}
extern "C" int yg_get_conv_impl(void) { return g_conv_impl; }
static int yg_get_tc_options_raw() { return get_tc_options(); }
extern "C" int yg_set_tc_options(int v) { return set_tc_options(v); }
extern "C" int yg_get_tc_options(void) { return get_tc_options(); }
extern "C" int yg_tc_debug_read(unsigned long long* out, int n) { return tc_debug_read(out, n); }

static inline bool aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }

template <typename T>
__global__ void actmask_from_output_kernel(const T* __restrict__ y, uint32_t* __restrict__ mask, long long nwords) {
  const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nwords) return;
  uint32_t bits = 0;
  for (int i = 0; i < 32; ++i) bits |= (to_f<T>(y[w * 32 + i]) > 0.f ? 1u : 0u) << i;
  mask[w] = bits;
}

extern "C" int yg_conv_fwd(const void* x, const float* w, void* y, int dtype, int N, int H, int W, int Cin, int Cout,
                           int ks, int stride, const yg_fwd_epilogue* epp, void* stream) {
  int rc = check_conv_args("conv_fwd", dtype, N, H, W, Cin, Cout, ks, stride);
  if (rc) return rc;
  YG_CHECK_ARG(x && w, "conv_fwd: null pointer");
  if (N == 0) return YG_OK;
  FwdEpi ep = make_fwd_epi(epp);
  // the tensor-core epilogues move pixel rows with 32-byte accesses: tensors that are not 32-byte aligned (never the case for
  // torch allocations) take the generic path
  const bool tc_ok = tc_fwd_supported(dtype, W, Cin, Cout, ks, stride) && aligned32(x) && aligned32(y) && aligned32(ep.preact);
  if (g_conv_impl == YG_IMPL_TCGEN05 && !tc_ok) {
    set_error("conv_fwd: tcgen05 path forced but shape or alignment unsupported (dtype %d Cin %d Cout %d k %d s %d)", dtype, Cin, Cout, ks, stride);
    return YG_ERR_INVALID;
  }
  if (ep.actmask) YG_CHECK_ARG(Cout % 32 == 0 && y, "conv_fwd: actmask needs Cout % 32 == 0 and an output tensor");
  if (tc_ok && g_conv_impl != YG_IMPL_SIMT)
    return conv_fwd_tc(x, w, y, N, H, W, Cin, Cout, ks, stride, ep, (cudaStream_t)stream);
  // fp32 tensors: split-bf16 convolution on the tensor cores (opt-in, option bit 21: yogo_b200.set_fp32_tensor_cores)
  if (dtype == YG_F32 && g_conv_impl != YG_IMPL_SIMT && (yg_get_tc_options_raw() & 2097152) && y && !ep.actmask &&
      x3_fwd_supported(W, Cin, Cout, ks, stride) && aligned32(x) && aligned32(y) && aligned32(ep.preact))
    return conv_fwd_x3((const float*)x, w, (float*)y, N, H, W, Cin, Cout, ks, stride, ep, (cudaStream_t)stream);
  rc = conv_fwd_simt(x, w, y, dtype, N, H, W, Cin, Cout, ks, stride, ep, (cudaStream_t)stream);
  if (rc == YG_OK && ep.actmask) {
    // generic path: derive the sign bits from the stored output (sign(y) == sign(v) wherever dropscale != 0)
    const int Ho = (H + 2 * (ks / 2) - ks) / stride + 1, Wo = (W + 2 * (ks / 2) - ks) / stride + 1;
    const long long nwords = (long long)N * Ho * Wo * Cout / 32;
    if (dtype == YG_BF16)
      actmask_from_output_kernel<bf16><<<cdiv(nwords, 256), 256, 0, (cudaStream_t)stream>>>((const bf16*)y, (uint32_t*)ep.actmask, nwords);
    else
      actmask_from_output_kernel<float><<<cdiv(nwords, 256), 256, 0, (cudaStream_t)stream>>>((const float*)y, (uint32_t*)ep.actmask, nwords);
    YG_LAUNCH_CHECK("actmask_from_output");
  }
  return rc;
}

extern "C" int yg_conv_dgrad(const void* dz, const float* w, void* dx, int dtype, int N, int H, int W, int Cin,
                             int Cout, int ks, int stride, const yg_bwd_epilogue* bep, void* stream) {
  int rc = check_conv_args("conv_dgrad", dtype, N, H, W, Cin, Cout, ks, stride);
  if (rc) return rc;
  YG_CHECK_ARG(dz && w && dx, "conv_dgrad: null pointer");
  if (N == 0) return YG_OK;
  BwdEpi be = make_bwd_epi(bep);
  const bool tc_ok = tc_dgrad_supported(dtype, W, Cin, Cout, ks, stride) && aligned32(dz) && aligned32(dx) && aligned32(be.saved);
  if (g_conv_impl == YG_IMPL_TCGEN05 && !tc_ok) {
    set_error("conv_dgrad: tcgen05 path forced but shape or alignment unsupported");
    return YG_ERR_INVALID;
  }
  if (tc_ok && g_conv_impl != YG_IMPL_SIMT)
    return conv_dgrad_tc(dz, w, dx, N, H, W, Cin, Cout, ks, stride, be, (cudaStream_t)stream);
  if (dtype == YG_F32 && g_conv_impl != YG_IMPL_SIMT && (yg_get_tc_options_raw() & 2097152) && !be.actmask &&
      x3_dgrad_supported(W, Cin, Cout, ks, stride) && aligned32(dz) && aligned32(dx) && aligned32(be.saved))
    return conv_dgrad_x3((const float*)dz, w, (float*)dx, N, H, W, Cin, Cout, ks, stride, be, (cudaStream_t)stream);
  return conv_dgrad_simt(dz, w, dx, dtype, N, H, W, Cin, Cout, ks, stride, be, (cudaStream_t)stream);
}

extern "C" size_t yg_conv_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int ks, int stride) {
  size_t a = simt_wgrad_workspace(N, H, W, Cin, Cout, ks, stride);
  size_t b = tc_wgrad_workspace(N, H, W, Cin, Cout, ks, stride);
  { const size_t c = x3_wgrad_workspace(N, H, W, Cin, Cout, ks, stride); if (c > b) b = c; }
  if (wgrad_hmma_supported(YG_BF16, W, Cin, Cout, ks, stride)) { const size_t c = wgrad_hmma_workspace(Cin, Cout); if (c > b) b = c; }
  return a > b ? a : b;
}

extern "C" int yg_conv_wgrad(const void* x, const void* dz, float* dw, float* dbias, int dtype, int N, int H, int W,
                             int Cin, int Cout, int ks, int stride, float clip, void* workspace,
                             size_t workspace_bytes, void* stream) {
  int rc = check_conv_args("conv_wgrad", dtype, N, H, W, Cin, Cout, ks, stride);
  if (rc) return rc;
  YG_CHECK_ARG(x && dz && dw, "conv_wgrad: null pointer");
  YG_CHECK_ARG(N >= 1, "conv_wgrad: empty batch");
  const bool tc_ok = tc_wgrad_supported(dtype, W, Cin, Cout, ks, stride);
  if (g_conv_impl == YG_IMPL_TCGEN05 && !tc_ok) {
    set_error("conv_wgrad: tcgen05 path forced but shape unsupported");
    return YG_ERR_INVALID;
  }
  // 16 -> 32 channels: warp-level tensor cores without W-fold waste (wgrad_hmma.cu: 0.54 -> 0.38 ms on base L2)
  if (g_conv_impl != YG_IMPL_SIMT && wgrad_hmma_supported(dtype, W, Cin, Cout, ks, stride))
    return conv_wgrad_hmma(x, dz, dw, dbias, N, H, W, Cin, Cout, ks, stride, clip, workspace, workspace_bytes, (cudaStream_t)stream);
  if (tc_ok && g_conv_impl != YG_IMPL_SIMT)
    return conv_wgrad_tc(x, dz, dw, dbias, N, H, W, Cin, Cout, ks, stride, clip, workspace, workspace_bytes, (cudaStream_t)stream);
  if (dtype == YG_F32 && g_conv_impl != YG_IMPL_SIMT && (yg_get_tc_options_raw() & 2097152) &&
      x3_wgrad_supported(W, Cin, Cout, ks, stride) && aligned32(x) && aligned32(dz) &&
      workspace_bytes >= x3_wgrad_workspace(N, H, W, Cin, Cout, ks, stride))
    return conv_wgrad_x3((const float*)x, (const float*)dz, dw, dbias, N, H, W, Cin, Cout, ks, stride, clip, workspace, workspace_bytes,
                         (cudaStream_t)stream);
  return conv_wgrad_simt(x, dz, dw, dbias, dtype, N, H, W, Cin, Cout, ks, stride, clip, workspace, workspace_bytes, (cudaStream_t)stream);
}
