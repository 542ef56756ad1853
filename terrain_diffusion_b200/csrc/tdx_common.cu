// Error reporting, device probe and TMA tensor-map construction for libtdx.
#include "tdx_common.h"

#include <cudaTypedefs.h>
#include <stdlib.h>
#include <string.h>

namespace tdx {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  // per CURRENT device (the Python host makes a tensor's device current around every call, _lib.call)
  static int n[16] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 16) dev = 0;
  if (n[dev] == 0) {
    cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev);
    if (n[dev] <= 0) n[dev] = 148;
  }
  return n[dev];
}

// True the first time it is called for the CURRENT device with this flag set (cudaFuncSetAttribute is per device: a
// process that drives two GPUs must opt each kernel in to its dynamic shared memory on both).
bool first_use_on_device(bool (&seen)[16]) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 16) dev = 0;
  if (seen[dev]) return false;
  seen[dev] = true;
  return true;
}

static bool use_pdl() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("TDX_PDL");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

void fill_launch_config(cudaLaunchConfig_t* cfg, cudaLaunchAttribute* attr, dim3 grid, dim3 block, size_t smem,
                        cudaStream_t stream) {
  memset(cfg, 0, sizeof(*cfg));
  cfg->gridDim = grid;
  cfg->blockDim = block;
  cfg->dynamicSmemBytes = smem;
  cfg->stream = stream;
  if (use_pdl()) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg->attrs = attr;
    cfg->numAttrs = 1;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

int make_act_tensor_map(CUtensorMap* out, const void* base, int n_img, int channels, int height, int width) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point not available (driver too old or no device)");
    return TDX_E_CUDA;
  }
  TDX_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0, "activation pointer %p is not 16-byte aligned", base);
  const cuuint64_t dims[4] = {(cuuint64_t)width * 8, (cuuint64_t)height, (cuuint64_t)channels / 8, (cuuint64_t)n_img};
  const cuuint64_t strides[3] = {(cuuint64_t)width * 16, (cuuint64_t)width * height * 16,
                                 (cuuint64_t)width * height * 16 * (channels / 8)};
  const cuuint32_t box[4] = {80, 18, 8, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for n=%d c=%d h=%d w=%d", (int)r, n_img, channels, height, width);
    return TDX_E_CUDA;
  }
  return TDX_OK;
}

}  // namespace tdx

extern "C" const char* tdx_last_error(void) { return tdx::g_err; }

extern "C" int tdx_device_info(int* sm_count_out, int* cc_major, int* cc_minor) {
  int dev = 0;
  TDX_CHECK_CUDA(cudaGetDevice(&dev));
  int major = 0, minor = 0, sms = 0;
  TDX_CHECK_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  TDX_CHECK_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  TDX_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (sm_count_out) *sm_count_out = sms;
  if (cc_major) *cc_major = major;
  if (cc_minor) *cc_minor = minor;
  if (major != 10) {
    tdx::set_error("libtdx is built for sm_100a only; device reports compute capability %d.%d", major, minor);
    return TDX_E_UNSUPPORTED;
  }
  return TDX_OK;
}

// ABI self-check for language bindings: sizeof of the public POD structs.
extern "C" int tdx_abi_sizeof(int which) {
  switch (which) {
    case 0: return (int)sizeof(TdxOutSpec);
    case 1: return (int)sizeof(TdxIgemmDesc);
    case 2: return (int)sizeof(TdxConvInDesc);
    case 3: return (int)sizeof(TdxConvOutDesc);
    case 4: return (int)sizeof(TdxEmbedBlock);
    case 5: return (int)sizeof(TdxEmbedDesc);
    case 6: return (int)sizeof(TdxAttnDesc);
    case 7: return (int)sizeof(TdxIm2colDesc);
    case 8: return (int)sizeof(TdxConvOutGuidedDesc);
    default: return -1;
  }
}
