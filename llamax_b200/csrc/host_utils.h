// Host-side helpers shared by the C-ABI entry points: error reporting and TMA descriptor encoding.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace lx {

int set_error(int code, const char* msg);
int set_cuda_error(cudaError_t e, const char* where);
int sm_count();

// rank-2 tensor map: dims {inner, outer}, row pitch ld (elements), box {box_inner, box_outer}, 128B swizzle
// (swizzle128 = false: the box lands in shared memory as plain rows of box_inner elements).
int make_tmap_2d(CUtensorMap* map, CUtensorMapDataType dt, int esz, const void* ptr, int64_t inner, int64_t outer,
                 int64_t ld, int box_inner, int box_outer, bool swizzle128 = true);

// rank-4 tensor map over a [d3, d2, d1, d0] view (d0 contiguous) with element strides s1, s2, s3.
int make_tmap_4d(CUtensorMap* map, CUtensorMapDataType dt, int esz, const void* ptr, const int64_t dims[4],
                 const int64_t strides[3], const int box[4]);

// One-time cudaFuncSetAttribute(MaxDynamicSharedMemorySize) per (device, kernel): the attribute is per device, so the
// "already configured" memo is keyed by the current device ordinal (a per-thread flag alone left the first launch on a
// second GPU of the same thread with the 48 KB default).
int ensure_dyn_smem(const void* kernel, int bytes, const char* who);

// out[d] (fp32) = sum_p partial[p, d] in part order (elementwise.cu; the deterministic lora_wgrad's split reduction)
int launch_reduce_partials_f32(const float* partial, float* out, int nparts, int64_t D, cudaStream_t stream);

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace lx

#define LX_CHECK_LAUNCH(where)                                  \
  do {                                                          \
    cudaError_t e__ = cudaGetLastError();                       \
    if (e__ != cudaSuccess) return lx::set_cuda_error(e__, where); \
  } while (0)
