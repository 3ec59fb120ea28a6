// Host-side helpers shared by every translation unit of libcstp_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>

#include "../../include/cstp_b200.h"

namespace cstp {

void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

inline int fail_inval(const char* what) {
  set_error("invalid argument: %s", what);
  return CSTP_EINVAL;
}

#define CSTP_REQUIRE(cond)                                   \
  do {                                                       \
    if (!(cond)) return ::cstp::fail_inval(#cond);           \
  } while (0)

#define CSTP_CUDA(expr)                                                                          \
  do {                                                                                           \
    cudaError_t e__ = (expr);                                                                    \
    if (e__ != cudaSuccess) {                                                                    \
      ::cstp::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return CSTP_ECUDA;                                                                         \
    }                                                                                            \
  } while (0)

// Call after every kernel launch: counts it and surfaces launch-configuration errors.
#define CSTP_LAUNCHED()                                 \
  do {                                                  \
    ::cstp::g_launches.fetch_add(1);                    \
    CSTP_CUDA(cudaGetLastError());                      \
  } while (0)

// Encodes a tiled bf16 tensor map (128B swizzle, zero OOB fill) through the driver entry point obtained from
// the runtime, so the library never links libcuda directly (it must dlopen on a box without a driver).
// swizzle_bytes: 128 (default), 64 or 32 -- the shared-memory row pitch of the box (its inner extent in bytes).
// oob_nan: out-of-range elements are filled with NaN instead of zero (operands that pass through the BatchNorm + ReLU
// prologue of ptx.cuh, where fmaxf(NaN, 0) restores the exact zero of the convolution padding).
int encode_tmap_bf16(CUtensorMap* map, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                     const uint32_t* box, int swizzle_bytes = 128, bool oob_nan = false);

int num_sms();

// Shared-memory budget (bytes) of the one-CTA-per-SM tensor-core kernels and the CTAs-per-SM share of the streaming
// kernels: together they decide whether an HBM-bound kernel on one stream can be co-resident with a tensor-bound
// kernel on the other (every resident CTA also costs 1 KB of reserved shared memory; the co-residency sweep of
// profiles/r01_overlap_sweep.txt kept these values).  ops.py SMEM_LIMIT is the same budget.
constexpr int kSmemBudget = 227 * 1024;
constexpr int kStreamCtasPerSm = 8;

inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }

}  // namespace cstp
