#include "common.h"

#include <cudaTypedefs.h>

#include <cstring>
#include <mutex>

namespace cstp {

static thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  });
  return fn;
}

int encode_tmap_bf16(CUtensorMap* map, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                     const uint32_t* box, int swizzle_bytes, bool oob_nan) {
  auto fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled driver entry point unavailable (no CUDA driver?)");
    return CSTP_ECUDA;
  }
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bdim[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = 1;
    if (i > 0) gstr[i - 1] = strides_bytes[i - 1];
  }
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, static_cast<cuuint32_t>(rank), const_cast<void*>(ptr), gdim,
                  gstr, bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                      : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B),
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  oob_nan ? CU_TENSOR_MAP_FLOAT_OOB_FILL_NAN_REQUEST_ZERO_FMA : CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d dims %llu %llu %llu %llu %llu box %u %u %u %u %u)",
              static_cast<int>(r), rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
              (unsigned long long)(rank > 4 ? dims[4] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0,
              rank > 3 ? box[3] : 0, rank > 4 ? box[4] : 0);
    return CSTP_ECUDA;
  }
  return CSTP_OK;
}

int num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}

}  // namespace cstp

extern "C" {
const char* cstp_last_error(void) { return cstp::g_err; }
int cstp_version(void) { return 100; }
long long cstp_launch_count(void) { return cstp::g_launches.load(); }
}
