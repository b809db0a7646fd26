// HBM-bound passes of the decoder block: RMSNorm (+ fused row quantisation), row-wise int8 quantisation,
// SwiGLU (+ fused row quantisation), RoPE, weight de-quantisation, and their backward passes.
// All of them are one read + one write of each tensor with 16-byte vector accesses, fp32 math in registers
// and warp-shuffle reductions; a row is held in registers between the reduction and the write so that no
// element is read twice.
#include "common.cuh"
#include "host_utils.h"
#include <algorithm>

#include <cstdlib>
#include <type_traits>

#include "llamax_b200.h"

namespace lx {

struct RowCfg {
  int threads;
  int nvec;
  int V;  // 16-byte vectors (8 bf16) held per thread: 1, 2, 4 or 8
};

static inline bool row_cfg(int64_t D, RowCfg& c, bool one_vec_per_thread = false) {
  if (D <= 0 || D % 8) return false;
  const int nvec = (int)(D / 8);
  // two 16-byte vectors per thread when the row allows it (measured on B200: 256 threads x 2 vectors beats
  // 512 x 1 for D = 4096 rows by ~25 %), at most 512 threads per row
  static const int vec_target = getenv("LLAMAX_ROW_VECS") ? std::max(1, atoi(getenv("LLAMAX_ROW_VECS"))) : 2;  // A/B only
  int threads = std::min(512, (((nvec + vec_target - 1) / vec_target + 31) / 32) * 32);
  if (one_vec_per_thread) threads = std::min(512, ((nvec + 31) / 32) * 32);  // persistent kernels: more warps per CTA
  int v = (nvec + threads - 1) / threads;
  if (v > 8) return false;
  c.V = v <= 1 ? 1 : v <= 2 ? 2 : v <= 4 ? 4 : 8;
  c.threads = threads;
  c.nvec = nvec;
  return true;
}

#define LX_DISPATCH_V(V_, ...)                    \
  switch (V_) {                                   \
    case 1: { constexpr int kV = 1; __VA_ARGS__; } break; \
    case 2: { constexpr int kV = 2; __VA_ARGS__; } break; \
    case 4: { constexpr int kV = 4; __VA_ARGS__; } break; \
    default: { constexpr int kV = 8; __VA_ARGS__; } break; \
  }

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  f[0] = bf16_lo(u.x); f[1] = bf16_hi(u.x);
  f[2] = bf16_lo(u.y); f[3] = bf16_hi(u.y);
  f[4] = bf16_lo(u.z); f[5] = bf16_hi(u.z);
  f[6] = bf16_lo(u.w); f[7] = bf16_hi(u.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 u;
  u.x = pack_bf16(f[0], f[1]);
  u.y = pack_bf16(f[2], f[3]);
  u.z = pack_bf16(f[4], f[5]);
  u.w = pack_bf16(f[6], f[7]);
  return u;
}

template <bool kMax>
__device__ __forceinline__ float block_reduce(float v, float* sm) {
  v = kMax ? warp_max(v) : warp_sum(v);
  const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();  // protect sm reuse between consecutive reductions
  if (lane_id() == 0) sm[w] = v;
  __syncthreads();
  float r = kMax ? 0.f : 0.f;
  if (kMax) {
    r = sm[0];
    for (int i = 1; i < nw; ++i) r = fmaxf(r, sm[i]);
  } else {
    for (int i = 0; i < nw; ++i) r += sm[i];
  }
  return r;
}

// Row quantisation, bit-identical to the reference's IEEE division + round-half-even (subclasses/int8.py:10-16) at two
// FMAs and one logic op per element: with inv = fl(1/sc), the exact quotient x/sc lies between x*inv_lo and x*inv_hi,
// inv_lo/hi = inv * (1 -/+ 2^-21) (fl(1/sc) and the two products' roundings are each within 2^-24). Rounding to
// integer is monotonic, so when both ends round to the same integer that integer is rint(fl(x/sc)) too; when they
// differ (the quotient is within ~2^-20 relative of a half-integer: ~1e-4 of all elements) the whole 8-element vector
// is redone with the reference's exact divisions (one rare branch per vector).
// Rounding without the conversion pipe: fma(x, inv, 1.5*2^23) rounds x*inv ONCE, to the nearest-even integer held in
// the float's low mantissa bits (|x*inv| < 2^22); the low byte of that word is the two's-complement int8 code.
// FRND / F2I (XU pipe, 16 lanes/clk) are not used.
constexpr float kRoundMagic = 12582912.0f;  // 1.5 * 2^23
__device__ __forceinline__ uint32_t pack4_low_bytes(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  return __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
}

// The rare vector (a quotient within ~2^-20 of a half-integer), redone with the reference's exact divisions. Out of line on
// purpose: inlined, the eight IEEE divisions are ~250 instructions per call site, and the warp-per-row kernels (16 call
// sites per row) grew to 70 KB of code whose hot path kept missing the instruction cache (ncu: `no_instruction` the top
// stall, 2.9 warps per issue slot).
__device__ __noinline__ uint2 quant_vec_exact(float f0, float f1, float f2, float f3, float f4, float f5, float f6,
                                              float f7, float sc) {
  const float f[8] = {f0, f1, f2, f3, f4, f5, f6, f7};
  uint32_t c[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) c[e] = __float_as_uint(__fadd_rn(f[e] / sc, kRoundMagic));
  return make_uint2(pack4_low_bytes(c[0], c[1], c[2], c[3]), pack4_low_bytes(c[4], c[5], c[6], c[7]));
}

// Eight int8 codes of one 16-byte vector (see the comment above kRoundMagic)
__device__ __forceinline__ uint2 quant_vec(const float (&f)[8], float sc, float inv_lo, float inv_hi) {
  uint32_t c[8];
  uint32_t differ = 0;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    c[e] = __float_as_uint(__fmaf_rn(f[e], inv_lo, kRoundMagic));
    differ |= c[e] ^ __float_as_uint(__fmaf_rn(f[e], inv_hi, kRoundMagic));
  }
  if (differ) return quant_vec_exact(f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7], sc);
  return make_uint2(pack4_low_bytes(c[0], c[1], c[2], c[3]), pack4_low_bytes(c[4], c[5], c[6], c[7]));
}

template <int kMaxV>
__device__ __forceinline__ void quant_row_store(const float (&v)[kMaxV][8], int nvec, float amax, int8_t* qrow,
                                                __nv_bfloat16* scale_out) {
  const float s = amax / 127.0f;
  const float sc = fmaxf(s, 1e-12f);
  const float inv = 1.0f / sc;
  const float inv_lo = inv * (1.0f - 0x1p-21f), inv_hi = inv * (1.0f + 0x1p-21f);
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int idx = threadIdx.x + j * blockDim.x;
    if (idx < nvec) *reinterpret_cast<uint2*>(qrow + (int64_t)idx * 8) = quant_vec(v[j], sc, inv_lo, inv_hi);
  }
  if (threadIdx.x == 0) *scale_out = __float2bfloat16_rn(s);
}

// ------------------------------------------------------------------------------------------------
// RMSNorm forward (+ optional fused row quantisation)
// ------------------------------------------------------------------------------------------------
template <int kMaxV>
__global__ void rmsnorm_fwd_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w,
                                   __nv_bfloat16* __restrict__ y, float* __restrict__ rstd_out,
                                   int8_t* __restrict__ q8, __nv_bfloat16* __restrict__ qscale, int D, int nvec,
                                   float eps) {
  __shared__ float sm[32];
  const int64_t row = blockIdx.x;
  const __nv_bfloat16* xr = x + row * D;
  float v[kMaxV][8];
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int idx = threadIdx.x + j * blockDim.x;
    if (idx < nvec) {
      unpack8(ldg_nc_v4(xr + (int64_t)idx * 8), v[j]);
#pragma unroll
      for (int e = 0; e < 8; ++e) ss = fmaf(v[j][e], v[j][e], ss);
    }
  }
  ss = block_reduce<false>(ss, sm);
  const float rstd = 1.0f / sqrtf(ss / (float)D + eps);
  if (threadIdx.x == 0 && rstd_out != nullptr) rstd_out[row] = rstd;
  float amax = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int idx = threadIdx.x + j * blockDim.x;
    if (idx < nvec) {
      float wf[8];
      unpack8(*reinterpret_cast<const uint4*>(w + (int64_t)idx * 8), wf);
      // round once with the packing conversion (needed for the y store anyway) and take the quantiser's input from
      // the packed words: integer round_bf16 (4 ALU-pipe instructions per element) made this pass ALU-pipe bound
#pragma unroll
      for (int e = 0; e < 8; ++e) v[j][e] = (v[j][e] * rstd) * wf[e];
      const uint4 yp = pack8(v[j]);
      unpack8(yp, v[j]);
#pragma unroll
      for (int e = 0; e < 8; ++e) amax = fmaxf(amax, fabsf(v[j][e]));
      if (y != nullptr) *reinterpret_cast<uint4*>(y + row * D + (int64_t)idx * 8) = yp;
    }
  }
  if (q8 != nullptr) {
    amax = block_reduce<true>(amax, sm);
    quant_row_store(v, nvec, amax, q8 + row * D, qscale + row);
  }
}

// ------------------------------------------------------------------------------------------------
// row-wise int8 quantisation alone
// ------------------------------------------------------------------------------------------------
// kColScale: quantise x[m, c] * col_scale[c] (fp32 product) instead of x — the opt-in INT8 grad_input path quantises
// grad_output * weight_scale (subclasses/int8.py:127) row-wise in one pass.
template <int kMaxV, bool kColScale = false>
__global__ void rowquant_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, int8_t* __restrict__ q8,
                                __nv_bfloat16* __restrict__ qscale, int K, int nvec,
                                const __nv_bfloat16* __restrict__ col_scale = nullptr) {
  __shared__ float sm[32];
  const int64_t row = blockIdx.x;
  const __nv_bfloat16* xr = x + row * ldx;
  float v[kMaxV][8];
  float amax = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int idx = threadIdx.x + j * blockDim.x;
    if (idx < nvec) {
      unpack8(ldg_nc_v4(xr + (int64_t)idx * 8), v[j]);
      if (kColScale) {
        float cs[8];
        unpack8(*reinterpret_cast<const uint4*>(col_scale + (int64_t)idx * 8), cs);
#pragma unroll
        for (int e = 0; e < 8; ++e) v[j][e] *= cs[e];
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) amax = fmaxf(amax, fabsf(v[j][e]));
    }
  }
  amax = block_reduce<true>(amax, sm);
  quant_row_store(v, nvec, amax, q8 + row * K, qscale + row);
}

// ------------------------------------------------------------------------------------------------
// Persistent "ring" variants of the row kernels.  One CTA per row exposes each row's global-load latency once per CTA
// lifetime (load -> reduce -> scale -> reduce -> quantise -> store). Here a CTA walks rows r, r + grid, ... and keeps
// the next kRingStages - 1 rows of its walk in flight as cp.async copies into a shared-memory ring. Every thread copies
// exactly the 16-byte slots it later reads itself, so cp.async.wait_group is the only synchronisation the ring needs.
// ------------------------------------------------------------------------------------------------
constexpr int kRingStages = 3;

__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Issue the copies of one row into ring stage `stage` (an empty group past the last row keeps the group count uniform)
template <int kMaxV>
__device__ __forceinline__ void ring_issue(uint4* ring, int slots, int stage, const __nv_bfloat16* xrow, bool valid,
                                           int nvec) {
  if (valid) {
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) cp_async_16(ring + stage * slots + idx, xrow + (int64_t)idx * 8);
    }
  }
  cp_async_commit();
}

template <int kMaxV>
__global__ void rmsnorm_fwd_ring_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w,
                                        __nv_bfloat16* __restrict__ y, float* __restrict__ rstd_out,
                                        int8_t* __restrict__ q8, __nv_bfloat16* __restrict__ qscale, int64_t M, int D,
                                        int nvec, float eps) {
  extern __shared__ uint4 ring[];
  __shared__ float sm[32];
  const int slots = blockDim.x * kMaxV;
  uint4 wp[kMaxV];  // the norm weight, packed, for the CTA lifetime
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int idx = threadIdx.x + j * blockDim.x;
    if (idx < nvec) wp[j] = *reinterpret_cast<const uint4*>(w + (int64_t)idx * 8);
  }
#pragma unroll
  for (int s = 0; s < kRingStages; ++s) {
    const int64_t r = blockIdx.x + (int64_t)s * gridDim.x;
    ring_issue<kMaxV>(ring, slots, s, x + r * D, r < M, nvec);
  }
  int stage = 0;
  for (int64_t row = blockIdx.x; row < M; row += gridDim.x) {
    cp_async_wait<kRingStages - 1>();
    float v[kMaxV][8];
    float ss = 0.f;
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        unpack8(ring[stage * slots + idx], v[j]);
#pragma unroll
        for (int e = 0; e < 8; ++e) ss = fmaf(v[j][e], v[j][e], ss);
      }
    }
    const int64_t rnext = row + (int64_t)kRingStages * gridDim.x;   // refill the stage just consumed
    ring_issue<kMaxV>(ring, slots, stage, x + rnext * D, rnext < M, nvec);
    stage = stage + 1 == kRingStages ? 0 : stage + 1;
    ss = block_reduce<false>(ss, sm);
    const float rstd = 1.0f / sqrtf(ss / (float)D + eps);
    if (threadIdx.x == 0 && rstd_out != nullptr) rstd_out[row] = rstd;
    float amax = 0.f;
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        float wf[8];
        unpack8(wp[j], wf);
#pragma unroll
        for (int e = 0; e < 8; ++e) v[j][e] = (v[j][e] * rstd) * wf[e];
        const uint4 yp = pack8(v[j]);
        unpack8(yp, v[j]);
#pragma unroll
        for (int e = 0; e < 8; ++e) amax = fmaxf(amax, fabsf(v[j][e]));
        if (y != nullptr) *reinterpret_cast<uint4*>(y + row * D + (int64_t)idx * 8) = yp;
      }
    }
    if (q8 != nullptr) {
      amax = block_reduce<true>(amax, sm);
      quant_row_store(v, nvec, amax, q8 + row * D, qscale + row);
    }
  }
  cp_async_wait<0>();
}

template <int kMaxV>
__global__ void rowquant_ring_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, int8_t* __restrict__ q8,
                                     __nv_bfloat16* __restrict__ qscale, int64_t M, int K, int nvec) {
  extern __shared__ uint4 ring[];
  __shared__ float sm[32];
  const int slots = blockDim.x * kMaxV;
#pragma unroll
  for (int s = 0; s < kRingStages; ++s) {
    const int64_t r = blockIdx.x + (int64_t)s * gridDim.x;
    ring_issue<kMaxV>(ring, slots, s, x + r * ldx, r < M, nvec);
  }
  int stage = 0;
  for (int64_t row = blockIdx.x; row < M; row += gridDim.x) {
    cp_async_wait<kRingStages - 1>();
    float v[kMaxV][8];
    float amax = 0.f;
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        unpack8(ring[stage * slots + idx], v[j]);
#pragma unroll
        for (int e = 0; e < 8; ++e) amax = fmaxf(amax, fabsf(v[j][e]));
      }
    }
    const int64_t rnext = row + (int64_t)kRingStages * gridDim.x;
    ring_issue<kMaxV>(ring, slots, stage, x + rnext * ldx, rnext < M, nvec);
    stage = stage + 1 == kRingStages ? 0 : stage + 1;
    amax = block_reduce<true>(amax, sm);
    quant_row_store(v, nvec, amax, q8 + row * K, qscale + row);
  }
  cp_async_wait<0>();
}

// ------------------------------------------------------------------------------------------------
// Warp-per-row RMSNorm forward (+ quantisation) and row quantiser, for rows of <= 4096 elements (the model width): the
// default for those rows. Measured at the clocks of a power-capped step (tools/ew_sustained.py: each pass right after a long
// GEMM, SM ~1.2 GHz) a device copy keeps 5.3 TB/s while the block-per-row ring kernels above reach 2.3-2.5: they issue
// ~32 instructions per element, two thirds of them per-ROW cost (two block reductions with four barriers, the scale
// arithmetic with its IEEE divisions, loop and address arithmetic) that 256 threads each pay for only 16 elements.
// Here a warp owns a row, lane l the 16-byte vectors l, l + 32, ...: the per-row cost is paid once per 128 elements per
// lane, both reductions are five shuffles, there is no barrier. The first version of this kernel loaded the row straight
// into registers and was SLOWER than the ring kernels (92 vs 79 us): nothing overlapped a warp's load with its arithmetic
// and the warps of an SM fell into step. Now every warp keeps the NEXT row of its walk in flight as cp.async copies into a
// warp-private shared-memory row buffer (each lane copies exactly the slots it reads: cp.async.wait_group is the only
// synchronisation): the row is pulled into registers (packed) when it has arrived and its slots are refilled at once, so one
// row per warp is in flight for the whole time the current one is worked on. The row maximum is taken on the packed bf16 pairs (one logic op +
// one HMNMX2 per two elements). Arithmetic and rounding order per element are those of the kernels above; only the
// summation order of the mean square differs.
// kNorm = false: row quantiser alone (w, y, rstd unused).
// ------------------------------------------------------------------------------------------------
constexpr int kWprWarps = 4;

__device__ __forceinline__ uint32_t absmax_bf16x2(uint32_t acc, uint32_t v) {
  uint32_t a = v & 0x7fff7fffu, r;
  asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(acc), "r"(a));
  return r;
}

// kFull: the row has exactly 32 * kVec vectors (the model width with kVec = 16): no per-vector bounds branch, so the
// passes are straight-line code the compiler can schedule across vectors (and ~30 % less of it)
template <int kVec, bool kNorm, bool kFull>
__global__ void __launch_bounds__(32 * kWprWarps, kNorm ? 3 : 4)   // the norm variant spills below 168 registers
row_wpr_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, const __nv_bfloat16* __restrict__ w,
               __nv_bfloat16* __restrict__ y, float* __restrict__ rstd_out, int8_t* __restrict__ q8,
               __nv_bfloat16* __restrict__ qscale, int64_t M, int D, int nvec, float eps) {
  extern __shared__ uint4 ring[];   // [warp][32 * kVec] (one row in flight per warp), then (kNorm) the norm weight [32 * kVec]
  const int lane = lane_id(), wib = threadIdx.x >> 5;
  constexpr int kSlots = 32 * kVec;
  uint4* my = ring + wib * kSlots;
  const uint4* wsm = ring + kWprWarps * kSlots;
  if constexpr (kNorm) {
    for (int i = threadIdx.x; i < nvec; i += blockDim.x)
      ring[kWprWarps * kSlots + i] = *reinterpret_cast<const uint4*>(w + (int64_t)i * 8);
    __syncthreads();
  }
  const int64_t warps = (int64_t)gridDim.x * kWprWarps;
  auto issue = [&](int64_t row) {
    if (row < M) {
      const __nv_bfloat16* xr = x + row * ldx;
#pragma unroll
      for (int j = 0; j < kVec; ++j) {
        const int idx = lane + 32 * j;
        if (kFull || idx < nvec) cp_async_16(my + idx, xr + (int64_t)idx * 8);
      }
    }
    cp_async_commit();
  };
  int64_t row = (int64_t)blockIdx.x * kWprWarps + wib;
  issue(row);
  for (; row < M; row += warps) {
    // the row arrives in registers (packed), and its slots are refilled at once with the warp's next row: one row per warp
    // in flight for the whole time the current one is worked on, at half the shared memory of a two-stage ring (16 instead
    // of 12 warps per SM for the quantiser alone)
    cp_async_wait<0>();
    uint4 pk[kVec];
#pragma unroll
    for (int j = 0; j < kVec; ++j) pk[j] = (kFull || lane + 32 * j < nvec) ? my[lane + 32 * j] : make_uint4(0, 0, 0, 0);
    issue(row + warps);
    if constexpr (kNorm) {
      float ss4[4] = {0.f, 0.f, 0.f, 0.f};   // four independent chains: few warps per scheduler do not hide a 128-deep one
#pragma unroll
      for (int j = 0; j < kVec; ++j) {
        float f[8];
        unpack8(pk[j], f);
#pragma unroll
        for (int e = 0; e < 8; ++e) ss4[e & 3] = fmaf(f[e], f[e], ss4[e & 3]);
      }
      const float ss = warp_sum((ss4[0] + ss4[1]) + (ss4[2] + ss4[3]));
      const float rstd = 1.0f / sqrtf(ss / (float)D + eps);
      if (lane == 0 && rstd_out != nullptr) rstd_out[row] = rstd;
#pragma unroll
      for (int j = 0; j < kVec; ++j) {
        const int idx = lane + 32 * j;
        if (kFull || idx < nvec) {
          float f[8], wf[8];
          unpack8(pk[j], f);
          unpack8(wsm[idx], wf);
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = (f[e] * rstd) * wf[e];
          pk[j] = pack8(f);   // y, rounded once; the quantiser below reads these bf16 values
          if (y != nullptr) *reinterpret_cast<uint4*>(y + row * D + (int64_t)idx * 8) = pk[j];
        }
      }
    }
    if (q8 == nullptr) continue;
    uint32_t m4[4] = {0, 0, 0, 0};   // running maxima of |.| on packed bf16 pairs (exact: a maximum rounds nothing)
#pragma unroll
    for (int j = 0; j < kVec; ++j) {
      m4[0] = absmax_bf16x2(m4[0], pk[j].x);
      m4[1] = absmax_bf16x2(m4[1], pk[j].y);
      m4[2] = absmax_bf16x2(m4[2], pk[j].z);
      m4[3] = absmax_bf16x2(m4[3], pk[j].w);
    }
    const uint32_t m2 = absmax_bf16x2(absmax_bf16x2(m4[0], m4[1]), absmax_bf16x2(m4[2], m4[3]));
    const float amax = warp_max(fmaxf(bf16_lo(m2), bf16_hi(m2)));
    const float s = amax / 127.0f;
    const float sc = fmaxf(s, 1e-12f);
    const float inv = 1.0f / sc;
    const float inv_lo = inv * (1.0f - 0x1p-21f), inv_hi = inv * (1.0f + 0x1p-21f);
    int8_t* qrow = q8 + row * D;
#pragma unroll
    for (int j = 0; j < kVec; ++j) {
      const int idx = lane + 32 * j;
      if (kFull || idx < nvec) {
        float f[8];
        unpack8(pk[j], f);
        *reinterpret_cast<uint2*>(qrow + (int64_t)idx * 8) = quant_vec(f, sc, inv_lo, inv_hi);
      }
    }
    if (lane == 0) qscale[row] = __float2bfloat16_rn(s);
  }
  cp_async_wait<0>();
}

// rows of up to 32 * 16 vectors, 16-byte aligned, enough of them to fill the machine. LLAMAX_ROW_WPR=0 falls back to the
// block-per-row ring kernels (A/B).
static bool wpr_cfg(int nvec, int64_t M, bool aligned, int& kvec, int& grid, int& smem, bool norm) {
  static const bool enabled = getenv("LLAMAX_ROW_WPR") == nullptr || atoi(getenv("LLAMAX_ROW_WPR")) != 0;
  static const int per_sm_env = getenv("LLAMAX_ROW_WPR_CTAS") ? std::max(1, atoi(getenv("LLAMAX_ROW_WPR_CTAS"))) : 0;
  const int per_sm = per_sm_env > 0 ? per_sm_env : (norm ? 3 : 4);   // = the kernels' launch bounds (registers)
  if (!enabled || !aligned || nvec > 512 || M < 1024) return false;
  const int v = (nvec + 31) / 32;
  kvec = v <= 1 ? 1 : v <= 2 ? 2 : v <= 4 ? 4 : v <= 8 ? 8 : 16;
  smem = (kWprWarps + (norm ? 1 : 0)) * 32 * kvec * 16;
  grid = (int)std::min<int64_t>((M + kWprWarps - 1) / kWprWarps, (int64_t)sm_count() * per_sm);
  return true;
}
#define LX_DISPATCH_WPR(V_, ...)                            \
  switch (V_) {                                             \
    case 1: { constexpr int kV = 1; __VA_ARGS__; } break;   \
    case 2: { constexpr int kV = 2; __VA_ARGS__; } break;   \
    case 4: { constexpr int kV = 4; __VA_ARGS__; } break;   \
    case 8: { constexpr int kV = 8; __VA_ARGS__; } break;   \
    default: { constexpr int kV = 16; __VA_ARGS__; } break; \
  }

// ------------------------------------------------------------------------------------------------
// SwiGLU forward: g = bf16( bf16(silu(a)) * b ), optional fused row quantisation
// ------------------------------------------------------------------------------------------------
// silu in fp32; the result is rounded to bf16 right away, so the fast exp / divide (~2 ulp fp32) are invisible
__device__ __forceinline__ float silu_f(float a) { return __fdividef(a, 1.0f + exp_neg_f(a)); }

template <int kMaxV>
__global__ void swiglu_fwd_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ b,
                                  int64_t ld, __nv_bfloat16* __restrict__ g, int8_t* __restrict__ q8,
                                  __nv_bfloat16* __restrict__ qscale, int F, int nvec) {
  __shared__ float sm[32];
  const int64_t row = blockIdx.x;
  float v[kMaxV][8];
  float amax = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int idx = threadIdx.x + j * blockDim.x;
    if (idx < nvec) {
      const uint4 ua = ldg_nc_v4(a + row * ld + (int64_t)idx * 8), ub = ldg_nc_v4(b + row * ld + (int64_t)idx * 8);
      const uint32_t wa[4] = {ua.x, ua.y, ua.z, ua.w}, wb[4] = {ub.x, ub.y, ub.z, ub.w};
      uint32_t wg[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        // bf16(silu(a)) for two elements, then the bf16 product with b (exact product, one rounding)
        wg[e] = mul_bf16x2(pack_bf16(silu_f(bf16_lo(wa[e])), silu_f(bf16_hi(wa[e]))), wb[e]);
        v[j][2 * e] = bf16_lo(wg[e]);
        v[j][2 * e + 1] = bf16_hi(wg[e]);
        amax = fmaxf(amax, fmaxf(fabsf(v[j][2 * e]), fabsf(v[j][2 * e + 1])));
      }
      if (g != nullptr) *reinterpret_cast<uint4*>(g + row * F + (int64_t)idx * 8) = make_uint4(wg[0], wg[1], wg[2], wg[3]);
    }
  }
  if (q8 != nullptr) {
    amax = block_reduce<true>(amax, sm);
    quant_row_store(v, nvec, amax, q8 + row * F, qscale + row);
  }
}

// Ring variant of the forward (default when it fits): persistent CTAs, the a and b rows of the next kRingStages - 1 rows of
// the CTA's walk in flight as cp.async copies (168 KB for F = 14336: one 512-thread CTA per SM), g kept PACKED in registers
// between the activation and the quantiser (row maximum on bf16 pairs), one barrier per row. The one-CTA-per-row kernel
// above exposes load -> activation -> reduction -> quantiser -> store once per CTA with two CTAs per SM to overlap them:
// 3.6 TB/s at the clocks of a power-capped step (tools/ew_sustained.py) where a device copy keeps 5.8.
template <int kMaxV>
__global__ void __launch_bounds__(512, 1)
swiglu_fwd_ring_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ b, int64_t ld,
                       __nv_bfloat16* __restrict__ g, int8_t* __restrict__ q8, __nv_bfloat16* __restrict__ qscale,
                       int64_t M, int F, int nvec) {
  extern __shared__ uint4 ring[];   // [stage][a | b][slots]
  __shared__ float sm[2][32];
  const int slots = blockDim.x * kMaxV;
  const int nw = blockDim.x >> 5;
  const uint32_t ring_s = smem_u32(ring) + threadIdx.x * 16;   // this thread's first slot of stage 0, stream a
  // byte offset from a row of a to the same row of b (same pitch; normally two column blocks of one buffer)
  const int64_t b_off = reinterpret_cast<const char*>(b) - reinterpret_cast<const char*>(a);
  auto issue = [&](int stage, int64_t row) {
    if (row < M) {
      // row base computed once; per vector one 64-bit add and one 32-bit add
      const char* src = reinterpret_cast<const char*>(a + row * ld) + threadIdx.x * 16;
      const uint32_t dst = ring_s + stage * 2 * slots * 16;
#pragma unroll
      for (int j = 0; j < kMaxV; ++j) {
        const int idx = threadIdx.x + j * blockDim.x;
        if (idx < nvec) {
          const char* sj = src + (int64_t)(j * blockDim.x) * 16;
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + j * blockDim.x * 16), "l"(sj) : "memory");
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (slots + j * blockDim.x) * 16),
                       "l"(sj + b_off) : "memory");
        }
      }
    }
    cp_async_commit();
  };
#pragma unroll
  for (int s = 0; s < kRingStages; ++s) issue(s, blockIdx.x + (int64_t)s * gridDim.x);
  int stage = 0, par = 0;
  for (int64_t row = blockIdx.x; row < M; row += gridDim.x) {
    cp_async_wait<kRingStages - 1>();
    const uint4* st = ring + (int64_t)stage * 2 * slots;
    uint32_t wg[kMaxV][4];
    uint32_t m2 = 0;
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
#pragma unroll
      for (int e = 0; e < 4; ++e) wg[j][e] = 0;
      if (idx < nvec) {
        const uint4 ua = st[idx], ub = st[slots + idx];
        const uint32_t wa[4] = {ua.x, ua.y, ua.z, ua.w}, wb[4] = {ub.x, ub.y, ub.z, ub.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          // bf16(silu(a)) for two elements, then the bf16 product with b (exact product, one rounding)
          wg[j][e] = mul_bf16x2(pack_bf16(silu_f(bf16_lo(wa[e])), silu_f(bf16_hi(wa[e]))), wb[e]);
          m2 = absmax_bf16x2(m2, wg[j][e]);
        }
        if (g != nullptr)
          *reinterpret_cast<uint4*>(g + row * F + (int64_t)idx * 8) = make_uint4(wg[j][0], wg[j][1], wg[j][2], wg[j][3]);
      }
    }
    issue(stage, row + (int64_t)kRingStages * gridDim.x);   // refill the stage just consumed
    stage = stage + 1 == kRingStages ? 0 : stage + 1;
    if (q8 == nullptr) continue;
    float amax = warp_max(fmaxf(bf16_lo(m2), bf16_hi(m2)));
    if (lane_id() == 0) sm[par][threadIdx.x >> 5] = amax;
    __syncthreads();   // one barrier per row: sm[par] is rewritten two rows later, after every thread passed the next one
    amax = sm[par][0];
    for (int i = 1; i < nw; ++i) amax = fmaxf(amax, sm[par][i]);
    par ^= 1;
    const float s = amax / 127.0f;
    const float sc = fmaxf(s, 1e-12f);
    const float inv = 1.0f / sc;
    const float inv_lo = inv * (1.0f - 0x1p-21f), inv_hi = inv * (1.0f + 0x1p-21f);
    int8_t* qrow = q8 + row * F;
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        float f[8];
        unpack8(make_uint4(wg[j][0], wg[j][1], wg[j][2], wg[j][3]), f);
        *reinterpret_cast<uint2*>(qrow + (int64_t)idx * 8) = quant_vec(f, sc, inv_lo, inv_hi);
      }
    }
    if (threadIdx.x == 0) qscale[row] = __float2bfloat16_rn(s);
  }
  cp_async_wait<0>();
}

// SwiGLU backward (grid-stride over 16-byte vectors)
__global__ void swiglu_bwd_kernel(const __nv_bfloat16* __restrict__ dg, const __nv_bfloat16* __restrict__ a,
                                  const __nv_bfloat16* __restrict__ b, int64_t ld, __nv_bfloat16* __restrict__ da,
                                  __nv_bfloat16* __restrict__ db, int64_t ldd, __nv_bfloat16* __restrict__ g,
                                  int64_t M, int nvec) {
  const int64_t total = M * nvec;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / nvec;
    const int c = (int)(i - row * nvec) * 8;
    const uint4 ua = ldg_nc_v4(a + row * ld + c), ub = ldg_nc_v4(b + row * ld + c);
    const uint4 ud = ldg_nc_v4(dg + row * (int64_t)nvec * 8 + c);
    uint4 oa, ob, og;
    swiglu_bwd_pair(ud.x, ua.x, ub.x, oa.x, ob.x, og.x);
    swiglu_bwd_pair(ud.y, ua.y, ub.y, oa.y, ob.y, og.y);
    swiglu_bwd_pair(ud.z, ua.z, ub.z, oa.z, ob.z, og.z);
    swiglu_bwd_pair(ud.w, ua.w, ub.w, oa.w, ob.w, og.w);
    *reinterpret_cast<uint4*>(da + row * ldd + c) = oa;
    *reinterpret_cast<uint4*>(db + row * ldd + c) = ob;
    if (g != nullptr) *reinterpret_cast<uint4*>(g + row * (int64_t)nvec * 8 + c) = og;
  }
}

// ------------------------------------------------------------------------------------------------
// RMSNorm backward.  Persistent over rows: CTA p handles rows p, p+nparts, ...; dw partial sums stay in
// registers and are written once per CTA.
// ------------------------------------------------------------------------------------------------
template <int kMaxV>
__global__ void __launch_bounds__(512, kMaxV == 1 ? 2 : 1)
rmsnorm_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
                   const __nv_bfloat16* __restrict__ w, const float* __restrict__ rstd,
                   const __nv_bfloat16* __restrict__ dres, __nv_bfloat16* __restrict__ dx,
                   float* __restrict__ dw_partial, int64_t M, int D, int nvec) {
  __shared__ float sm[32];
  float wf[kMaxV][8], dwacc[kMaxV][8];
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int idx = threadIdx.x + j * blockDim.x;
#pragma unroll
    for (int e = 0; e < 8; ++e) dwacc[j][e] = 0.f;
    if (idx < nvec) unpack8(*reinterpret_cast<const uint4*>(w + (int64_t)idx * 8), wf[j]);
  }
  // Software pipeline over this CTA's rows: the three streams of the NEXT row (x, dy, residual gradient) are in
  // flight, still packed, while the current row is reduced and written. Without it a CTA exposes two dependent
  // global-load latencies per row (x|dy, then the residual after the block reduction): 2.7 TB/s on B200.
  uint4 nx[kMaxV], ndy[kMaxV], nres[kMaxV];
  float nrs = 0.f;
  auto prefetch = [&](int64_t row) {
    if (row >= M) return;
    nrs = rstd[row];
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        nx[j] = ldg_nc_v4(x + row * D + (int64_t)idx * 8);
        ndy[j] = ldg_nc_v4(dy + row * D + (int64_t)idx * 8);
        if (dres != nullptr) nres[j] = ldg_nc_v4(dres + row * D + (int64_t)idx * 8);
      }
    }
  };
  prefetch(blockIdx.x);
  for (int64_t row = blockIdx.x; row < M; row += gridDim.x) {
    const float rs = nrs;
    uint4 cx[kMaxV], cdy[kMaxV], cres[kMaxV];
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      cx[j] = nx[j];
      cdy[j] = ndy[j];
      cres[j] = nres[j];
    }
    prefetch(row + gridDim.x);
    float xh[kMaxV][8], gy[kMaxV][8];
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        float dyf[8];
        unpack8(cx[j], xh[j]);
        unpack8(cdy[j], dyf);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          xh[j][e] *= rs;
          dwacc[j][e] = fmaf(dyf[e], xh[j][e], dwacc[j][e]);
          gy[j][e] = dyf[e] * wf[j][e];
          dot = fmaf(gy[j][e], xh[j][e], dot);
        }
      }
    }
    dot = block_reduce<false>(dot, sm) / (float)D;
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        float o[8];
        if (dres != nullptr) unpack8(cres[j], o);
        else {
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = 0.f;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] += rs * (gy[j][e] - xh[j][e] * dot);
        *reinterpret_cast<uint4*>(dx + row * D + (int64_t)idx * 8) = pack8(o);
      }
    }
  }
  if (dw_partial != nullptr) {
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        float* dst = dw_partial + (int64_t)blockIdx.x * D + (int64_t)idx * 8;
        *reinterpret_cast<float4*>(dst) = make_float4(dwacc[j][0], dwacc[j][1], dwacc[j][2], dwacc[j][3]);
        *reinterpret_cast<float4*>(dst + 4) = make_float4(dwacc[j][4], dwacc[j][5], dwacc[j][6], dwacc[j][7]);
      }
    }
  }
}

// Ring variant (default when it fits): two 16-byte vectors per thread instead of one (per-row fixed cost — reduction,
// loop and address arithmetic — amortised over 16 elements, not 8: the kernel above issues 32 instructions per element and
// runs at 2.9 TB/s at the clocks of a power-capped step where a device copy keeps 5.3), the three input streams of the next
// kRingStages - 1 rows of the CTA's walk in flight as cp.async copies into shared memory (no registers held by the
// prefetch; every thread copies exactly the slots it reads itself, so cp.async.wait_group is the only synchronisation of
// the ring), and ONE barrier per row: the per-warp partial sums go to one of two alternating shared-memory rows.
template <int kMaxV>
__global__ void __launch_bounds__(256, 2)
rmsnorm_bwd_ring_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
                        const __nv_bfloat16* __restrict__ w, const float* __restrict__ rstd,
                        const __nv_bfloat16* __restrict__ dres, __nv_bfloat16* __restrict__ dx,
                        float* __restrict__ dw_partial, int64_t M, int D, int nvec) {
  extern __shared__ uint4 ring[];   // [stage][stream: x, dy, dres][slots]
  __shared__ float sm[2][32];
  const int slots = blockDim.x * kMaxV;
  const int nstream = dres != nullptr ? 3 : 2;
  const int nw = blockDim.x >> 5;
  float wf[kMaxV][8], dwacc[kMaxV][8];
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int idx = threadIdx.x + j * blockDim.x;
#pragma unroll
    for (int e = 0; e < 8; ++e) dwacc[j][e] = 0.f;
    if (idx < nvec) unpack8(*reinterpret_cast<const uint4*>(w + (int64_t)idx * 8), wf[j]);
  }
  const uint32_t ring_s = smem_u32(ring) + threadIdx.x * 16;
  auto issue = [&](int stage, int64_t row) {
    if (row < M) {
      const int64_t off = (row * D + threadIdx.x * 8) * 2;   // byte offset of this thread's first vector in every stream
      const uint32_t dst = ring_s + stage * 3 * slots * 16;
#pragma unroll
      for (int j = 0; j < kMaxV; ++j) {
        const int idx = threadIdx.x + j * blockDim.x;
        if (idx < nvec) {
          const int64_t oj = off + (int64_t)(j * blockDim.x) * 16;
          const uint32_t dj = dst + j * blockDim.x * 16;
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dj), "l"(reinterpret_cast<const char*>(x) + oj) : "memory");
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dj + slots * 16),
                       "l"(reinterpret_cast<const char*>(dy) + oj) : "memory");
          if (nstream == 3)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dj + 2 * slots * 16),
                         "l"(reinterpret_cast<const char*>(dres) + oj) : "memory");
        }
      }
    }
    cp_async_commit();
  };
#pragma unroll
  for (int s = 0; s < kRingStages; ++s) issue(s, blockIdx.x + (int64_t)s * gridDim.x);
  int stage = 0, par = 0;
  float rs_next = blockIdx.x < M ? rstd[blockIdx.x] : 0.f;   // one row ahead: its L2 latency is never on the critical path
  for (int64_t row = blockIdx.x; row < M; row += gridDim.x) {
    const float rs = rs_next;
    if (row + gridDim.x < M) rs_next = rstd[row + gridDim.x];
    cp_async_wait<kRingStages - 1>();
    const uint4* st = ring + (int64_t)stage * 3 * slots;
    float xh[kMaxV][8], gy[kMaxV][8];
    uint4 cres[kMaxV];
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        float dyf[8];
        unpack8(st[idx], xh[j]);
        unpack8(st[slots + idx], dyf);
        if (nstream == 3) cres[j] = st[2 * slots + idx];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          xh[j][e] *= rs;
          dwacc[j][e] = fmaf(dyf[e], xh[j][e], dwacc[j][e]);
          gy[j][e] = dyf[e] * wf[j][e];
          dot = fmaf(gy[j][e], xh[j][e], dot);
        }
      }
    }
    issue(stage, row + (int64_t)kRingStages * gridDim.x);   // refill the stage just consumed (all reads are in registers)
    stage = stage + 1 == kRingStages ? 0 : stage + 1;
    dot = warp_sum(dot);
    if (lane_id() == 0) sm[par][threadIdx.x >> 5] = dot;
    __syncthreads();
    // the row after next writes sm[par] again: every thread has passed the next row's barrier by then, i.e. has read it
    if (nw == 8) {
      const float4 a = *reinterpret_cast<const float4*>(&sm[par][0]), b = *reinterpret_cast<const float4*>(&sm[par][4]);
      dot = ((a.x + a.y) + (a.z + a.w)) + ((b.x + b.y) + (b.z + b.w));
    } else {
      dot = 0.f;
      for (int i = 0; i < nw; ++i) dot += sm[par][i];
    }
    par ^= 1;
    dot = dot / (float)D;
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        float o[8];
        if (nstream == 3) unpack8(cres[j], o);
        else {
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = 0.f;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] += rs * (gy[j][e] - xh[j][e] * dot);
        *reinterpret_cast<uint4*>(dx + row * D + (int64_t)idx * 8) = pack8(o);
      }
    }
  }
  cp_async_wait<0>();
  if (dw_partial != nullptr) {
#pragma unroll
    for (int j = 0; j < kMaxV; ++j) {
      const int idx = threadIdx.x + j * blockDim.x;
      if (idx < nvec) {
        float* dst = dw_partial + (int64_t)blockIdx.x * D + (int64_t)idx * 8;
        *reinterpret_cast<float4*>(dst) = make_float4(dwacc[j][0], dwacc[j][1], dwacc[j][2], dwacc[j][3]);
        *reinterpret_cast<float4*>(dst + 4) = make_float4(dwacc[j][4], dwacc[j][5], dwacc[j][6], dwacc[j][7]);
      }
    }
  }
}

// out[d] = sum_p partial[p, d], summed in part order: bf16 out (RMSNorm dw), fp32 out (deterministic lora_wgrad)
template <typename T = __nv_bfloat16>
__global__ void reduce_partials_kernel(const float* __restrict__ partial, T* __restrict__ out, int nparts, int64_t D) {
  const int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  float s = 0.f;
  for (int p = 0; p < nparts; ++p) s += partial[(int64_t)p * D + d];
  if constexpr (std::is_same_v<T, float>) out[d] = s;
  else out[d] = __float2bfloat16_rn(s);
}

int launch_reduce_partials_f32(const float* partial, float* out, int nparts, int64_t D, cudaStream_t stream) {
  reduce_partials_kernel<float><<<(unsigned)((D + 255) / 256), 256, 0, stream>>>(partial, out, nparts, D);
  LX_CHECK_LAUNCH("reduce_partials");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// RoPE in place, interleaved pairs (modelling/llama.py:63-73).  One thread = 8 bf16 = 4 pairs.
// ------------------------------------------------------------------------------------------------
// grid = (row pairs, column chunks of 256 vectors): the row (and its position s = row % S) is uniform per CTA and the column
// comes from the thread index — no 64-bit division per thread. The first version (one grid-stride loop over
// rows * vectors with `i / vec_per_row`, `row % S`) spent ~19 instructions per element, most of them in those two
// divisions, and was issue-bound at the clocks of a power-capped step (3.2 TB/s where a device copy keeps 5.3).
constexpr int kRopeRows = 2;   // rows per thread: both rows' loads are in flight before the first is rotated
__global__ void __launch_bounds__(256) rope_kernel(__nv_bfloat16* __restrict__ x, int64_t ld,
                                                   const float* __restrict__ rope, int64_t rows, int S,
                                                   int vec_per_row, int D, int inverse) {
  const int v = blockIdx.y * 256 + threadIdx.x;
  if (v >= vec_per_row) return;
  const int c = v * 8;                               // column within the row
  const int d = (D & (D - 1)) == 0 ? (c & (D - 1)) : c % D;   // offset inside the head, multiple of 8
  uint4 in[kRopeRows];
  float4 cs0[kRopeRows], cs1[kRopeRows];
#pragma unroll
  for (int r = 0; r < kRopeRows; ++r) {
    const int64_t row = (int64_t)blockIdx.x * kRopeRows + r;
    if (row < rows) {
      const int s = (int)((unsigned)row % (unsigned)S);   // uniform per CTA; rows < 2^31 (checked by the launcher)
      in[r] = ldg_nc_v4(x + row * ld + c);
      const float4* cs = reinterpret_cast<const float4*>(rope + ((int64_t)s * (D / 2) + d / 2) * 2);
      cs0[r] = __ldg(cs);                            // (c0,s0,c1,s1)
      cs1[r] = __ldg(cs + 1);                        // (c2,s2,c3,s3)
    }
  }
#pragma unroll
  for (int r = 0; r < kRopeRows; ++r) {
    const int64_t row = (int64_t)blockIdx.x * kRopeRows + r;
    if (row >= rows) break;
    float f[8], o[8];
    unpack8(in[r], f);
    const float cc[4] = {cs0[r].x, cs0[r].z, cs1[r].x, cs1[r].z};
    float sn[4] = {cs0[r].y, cs0[r].w, cs1[r].y, cs1[r].w};
    if (inverse) {
#pragma unroll
      for (int e = 0; e < 4; ++e) sn[e] = -sn[e];
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      // out0 = x0*c - x1*s ; out1 = x1*c + x0*s   (each product rounded as in the fp32 reference)
      o[2 * e] = __fsub_rn(__fmul_rn(f[2 * e], cc[e]), __fmul_rn(f[2 * e + 1], sn[e]));
      o[2 * e + 1] = __fadd_rn(__fmul_rn(f[2 * e + 1], cc[e]), __fmul_rn(f[2 * e], sn[e]));
    }
    *reinterpret_cast<uint4*>(x + row * ld + c) = pack8(o);
  }
}

// ------------------------------------------------------------------------------------------------
// weight de-quantisation into a bf16 GEMM operand
// ------------------------------------------------------------------------------------------------
__global__ void dequant_plain_kernel(const int8_t* __restrict__ w8, const __nv_bfloat16* __restrict__ scale,
                                     __nv_bfloat16* __restrict__ out, int64_t ldo, int64_t N, int64_t K,
                                     int apply_scale) {
  const int64_t nvec = N * K / 16;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = i * 16;
    const int64_t n = e0 / K, kk = e0 - n * K;
    const float s = apply_scale ? __bfloat162float(scale[n]) : 1.0f;
    const uint4 u = ldg_nc_v4(w8 + e0);
    const uint32_t words[4] = {u.x, u.y, u.z, u.w};
    float f[16];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int e = 0; e < 4; ++e) f[q * 4 + e] = s8_to_float(words[q] >> (8 * e)) * s;
    float lo[8], hi[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { lo[e] = f[e]; hi[e] = f[8 + e]; }
    *reinterpret_cast<uint4*>(out + n * ldo + kk) = pack8(lo);
    *reinterpret_cast<uint4*>(out + n * ldo + kk + 8) = pack8(hi);
  }
}

// out[k, n] = bf16(w8[n, k] * scale[n]); 64 x 64 tiles through shared memory
__global__ void __launch_bounds__(256)
dequant_transpose_kernel(const int8_t* __restrict__ w8, const __nv_bfloat16* __restrict__ scale,
                         __nv_bfloat16* __restrict__ out, int64_t ldo, int N, int K, int apply_scale) {
  __shared__ __align__(16) __nv_bfloat16 tile[64][72];
  const int n0 = blockIdx.y * 64, k0 = blockIdx.x * 64;
  {
    const int n = threadIdx.x >> 2, kc = (threadIdx.x & 3) * 16;
    if (n0 + n < N && k0 + kc < K) {
      const float s = apply_scale ? __bfloat162float(scale[n0 + n]) : 1.0f;
      const uint4 u = ldg_nc_v4(w8 + (int64_t)(n0 + n) * K + k0 + kc);
      const uint32_t words[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int e = 0; e < 4; ++e)
          tile[kc + q * 4 + e][n] = __float2bfloat16_rn(s8_to_float(words[q] >> (8 * e)) * s);
    } else {
#pragma unroll
      for (int e = 0; e < 16; ++e) tile[kc + e][n] = __float2bfloat16_rn(0.f);
    }
  }
  __syncthreads();
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int t = threadIdx.x + it * 256;
    const int k = t >> 3, nc = (t & 7) * 8;
    if (k0 + k < K && n0 + nc < N)
      *reinterpret_cast<uint4*>(out + (int64_t)(k0 + k) * ldo + n0 + nc) = *reinterpret_cast<const uint4*>(&tile[k][nc]);
  }
}

// ------------------------------------------------------------------------------------------------
// Cross-entropy over bf16 logits, forward + backward in place (F.cross_entropy(logits.float(), labels),
// modelling/llama.py:216-218): per row lse = logsumexp(f32(logits)); loss_sum += lse - logit[label];
// logits <- (softmax - onehot(label)) * inv_n   (0 for ignored rows, label == -100).
// One CTA per row: one HBM read (online max/sum), one L2 re-read + one write. No fp32 [M, vocab] tensor.
// ------------------------------------------------------------------------------------------------
// kRowLoss (deterministic mode): loss_sum is an fp32 [M] buffer that receives each row's loss (0 for ignored rows),
// summed in a fixed order by the caller, instead of one scalar accumulated with fp32 atomics in CTA completion order.
template <bool kRowLoss = false>
__global__ void __launch_bounds__(512)
cross_entropy_kernel(__nv_bfloat16* __restrict__ logits, int64_t ld, const int64_t* __restrict__ labels,
                     float* __restrict__ loss_sum, const float* __restrict__ inv_n, int V, int write_grad) {
  __shared__ float sm_m[16], sm_s[16];
  const int64_t row = blockIdx.x;
  __nv_bfloat16* lr = logits + row * ld;
  const int64_t label = labels[row];
  const int nvec = V / 8;
  if (label < 0) {  // ignore_index
    if constexpr (kRowLoss) {
      if (threadIdx.x == 0) loss_sum[row] = 0.f;
    }
    if (write_grad)
      for (int i = threadIdx.x; i < nvec; i += blockDim.x) *reinterpret_cast<uint4*>(lr + (int64_t)i * 8) = make_uint4(0, 0, 0, 0);
    return;
  }
  float m = -INFINITY, ssum = 0.f;
  for (int i = threadIdx.x; i < nvec; i += blockDim.x) {
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(lr + (int64_t)i * 8), f);
    float vm = f[0];
#pragma unroll
    for (int e = 1; e < 8; ++e) vm = fmaxf(vm, f[e]);
    const float mn = fmaxf(m, vm);
    float part = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) part += __expf(f[e] - mn);
    ssum = ssum * (m == -INFINITY ? 0.f : __expf(m - mn)) + part;
    m = mn;
  }
  // block reduce of (m, s); threads / warps without elements carry (m = -inf, s = 0)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, ssum, o);
    const float mn = fmaxf(m, m2);
    ssum = (m == -INFINITY ? 0.f : ssum * __expf(m - mn)) + (m2 == -INFINITY ? 0.f : s2 * __expf(m2 - mn));
    m = mn;
  }
  const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if (lane_id() == 0) { sm_m[w] = m; sm_s[w] = ssum; }
  __syncthreads();
  float M_ = sm_m[0];
  for (int i = 1; i < nw; ++i) M_ = fmaxf(M_, sm_m[i]);
  float S_ = 0.f;
  for (int i = 0; i < nw; ++i) S_ += (sm_m[i] == -INFINITY) ? 0.f : sm_s[i] * __expf(sm_m[i] - M_);
  const float lse = M_ + logf(S_);
  if constexpr (kRowLoss) {
    if (threadIdx.x == 0) loss_sum[row] = lse - __bfloat162float(lr[label]);
  } else {
    if (threadIdx.x == 0) atomicAdd(loss_sum, lse - __bfloat162float(lr[label]));
  }
  if (!write_grad) return;
  const float scale = *inv_n;
  __syncthreads();  // every thread has read lr[label]-independent data; row is rewritten below
  for (int i = threadIdx.x; i < nvec; i += blockDim.x) {
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(lr + (int64_t)i * 8), f);
    const int64_t c0 = (int64_t)i * 8;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float pr = __expf(f[e] - lse);
      if (c0 + e == label) pr -= 1.f;
      f[e] = pr * scale;
    }
    *reinterpret_cast<uint4*>(lr + c0) = pack8(f);
  }
}

// ------------------------------------------------------------------------------------------------
// Audio stem (modelling/audio.py:26-31): bias + exact (erf) GELU around the conv-as-GEMM outputs, and the
// overlap-add of the stride-2 k=3 convolution's input gradient. Rows are channels-last [batch * period, C];
// rows whose index inside a batch slab (row % period) is not in [lo, hi) are padding and are written as zeros.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_erf(float z) { return 0.5f * z * (1.0f + erff(z * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_erf_grad(float z) {
  const float cdf = 0.5f * (1.0f + erff(z * 0.70710678118654752f));
  const float pdf = 0.3989422804014327f * __expf(-0.5f * z * z);
  return cdf + z * pdf;
}

// z (in place) = bf16(z + bias[col]);  y = bf16(gelu(z))
__global__ void gelu_bias_fwd_kernel(__nv_bfloat16* __restrict__ z, const __nv_bfloat16* __restrict__ bias,
                                     __nv_bfloat16* __restrict__ y, int64_t rows, int nvec, int period, int lo, int hi) {
  const int64_t total = rows * nvec;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / nvec;
    const int c = (int)(i - row * nvec) * 8;
    const int rr = (int)(row % period);
    float zf[8], bf[8], yf[8];
    if (rr >= lo && rr < hi) {
      unpack8(*reinterpret_cast<const uint4*>(z + row * (int64_t)nvec * 8 + c), zf);
      unpack8(*reinterpret_cast<const uint4*>(bias + c), bf);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        zf[e] = round_bf16(zf[e] + bf[e]);
        yf[e] = gelu_erf(zf[e]);
      }
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) zf[e] = yf[e] = 0.f;
    }
    *reinterpret_cast<uint4*>(z + row * (int64_t)nvec * 8 + c) = pack8(zf);
    *reinterpret_cast<uint4*>(y + row * (int64_t)nvec * 8 + c) = pack8(yf);
  }
}

// dz = bf16(dy * gelu'(z)) on valid rows, 0 on padding rows (dz may alias dy)
__global__ void gelu_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ z,
                                __nv_bfloat16* __restrict__ dz, int64_t rows, int nvec, int period, int lo, int hi) {
  const int64_t total = rows * nvec;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / nvec;
    const int c = (int)(i - row * nvec) * 8;
    const int rr = (int)(row % period);
    float o[8];
    if (rr >= lo && rr < hi) {
      float g[8], zf[8];
      unpack8(*reinterpret_cast<const uint4*>(dy + row * (int64_t)nvec * 8 + c), g);
      unpack8(*reinterpret_cast<const uint4*>(z + row * (int64_t)nvec * 8 + c), zf);
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = g[e] * gelu_erf_grad(zf[e]);
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = 0.f;
    }
    *reinterpret_cast<uint4*>(dz + row * (int64_t)nvec * 8 + c) = pack8(o);
  }
}

// Input gradient of Conv1d(k = 3, stride 2, pad 1) from the column gradient dcol [B, Tp/2, 3, C] (slab row t holds the
// gradients of padded input rows 2t, 2t+1, 2t+2):  dxp[b, i] = sum over (t, j) with 2t + j = i.  dxp [B, Tp, C].
__global__ void conv_s2k3_col2im_kernel(const __nv_bfloat16* __restrict__ dcol, __nv_bfloat16* __restrict__ dxp,
                                        int64_t B, int Tp, int nvec) {
  const int half = Tp / 2;                       // column-matrix rows per batch slab (the last one is padding)
  const int64_t total = B * Tp * (int64_t)nvec;
  const int64_t C = (int64_t)nvec * 8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % nvec) * 8;
    const int64_t r = i / nvec;
    const int ip = (int)(r % Tp);
    const int64_t b = r / Tp;
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int tt = ip - j;
      if (tt >= 0 && (tt & 1) == 0 && (tt >> 1) < half - 1) {   // valid output rows: t < Tp/2 - 1
        float v[8];
        unpack8(*reinterpret_cast<const uint4*>(dcol + ((b * half + (tt >> 1)) * 3 + j) * C + c), v);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] += v[e];
      }
    }
    *reinterpret_cast<uint4*>(dxp + r * C + c) = pack8(acc);
  }
}

// ------------------------------------------------------------------------------------------------
// Batched small copies (LoRA bookkeeping): job = blockIdx.y, 32 x 32 tiles through shared memory
// ------------------------------------------------------------------------------------------------
struct CopyJobs {
  llamax_copy_job_t j[LLAMAX_MAX_COPY_JOBS];
};

__global__ void __launch_bounds__(256) batched_copy_kernel(const __grid_constant__ CopyJobs jobs) {
  __shared__ float tile[32][33];
  const llamax_copy_job_t& jb = jobs.j[blockIdx.y];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  const int tiles_c = (jb.cols + 31) / 32, tiles_r = (jb.rows + 31) / 32;
  const bool f32 = jb.flags & 1, tr = jb.flags & 2;
  for (int t = blockIdx.x; t < tiles_r * tiles_c; t += gridDim.x) {
    const int r0 = (t / tiles_c) * 32, c0 = (t % tiles_c) * 32;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int r = r0 + ty + k * 8, c = c0 + tx;
      float v = 0.f;
      if (r < jb.rows && c < jb.cols) {
        const int64_t off = (int64_t)r * jb.src_ld + c;
        v = f32 ? static_cast<const float*>(jb.src)[off] : __bfloat162float(static_cast<const __nv_bfloat16*>(jb.src)[off]);
      }
      tile[ty + k * 8][tx] = v * jb.scale;
    }
    __syncthreads();
    __nv_bfloat16* dst = static_cast<__nv_bfloat16*>(jb.dst);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (tr) {
        const int c = c0 + ty + k * 8, r = r0 + tx;      // dst[c, r]
        if (r < jb.rows && c < jb.cols) dst[(int64_t)c * jb.dst_ld + r] = __float2bfloat16_rn(tile[tx][ty + k * 8]);
      } else {
        const int r = r0 + ty + k * 8, c = c0 + tx;
        if (r < jb.rows && c < jb.cols) dst[(int64_t)r * jb.dst_ld + c] = __float2bfloat16_rn(tile[ty + k * 8][tx]);
      }
    }
    __syncthreads();
  }
}

}  // namespace lx

using namespace lx;
typedef __nv_bfloat16 bf16;

// Ring (persistent, cp.async-prefetched) row kernels: used when the ring fits next to enough resident CTAs and there
// are enough rows for the prefetch depth to matter. LLAMAX_ROW_RING=0 keeps the one-CTA-per-row kernels (A/B).
static bool ring_cfg(const RowCfg& c, int64_t M, bool aligned, int& grid, int& smem) {
  static const bool enabled = getenv("LLAMAX_ROW_RING") == nullptr || atoi(getenv("LLAMAX_ROW_RING")) != 0;
  static const int per_sm_env = getenv("LLAMAX_ROW_RING_CTAS") ? atoi(getenv("LLAMAX_ROW_RING_CTAS")) : 0;
  smem = kRingStages * c.threads * c.V * 16;
  if (!enabled || !aligned || smem > 96 * 1024) return false;
  const int by_smem = (200 * 1024) / (smem + 1024), by_threads = 2048 / c.threads;
  int per_sm = std::max(1, std::min(by_smem, by_threads));
  if (per_sm_env > 0) per_sm = std::min(per_sm, per_sm_env);
  grid = sm_count() * per_sm;
  if (M < (int64_t)grid * 2) return false;
  return true;
}
#define LX_RING_SMEM(kern, smem, what)                                                                      \
  do {                                                                                                      \
    int rc_ = ensure_dyn_smem(reinterpret_cast<const void*>(kern), (smem), what ": cudaFuncSetAttribute");  \
    if (rc_) return rc_;                                                                                    \
  } while (0)

extern "C" {

int llamax_rmsnorm_fwd(const void* x, const void* w, void* y, void* rstd, void* q8, void* qscale, int64_t M,
                       int64_t D, float eps, void* stream) {
  RowCfg c;
  if (!x || !w) return set_error(LLAMAX_ERR_ARG, "rmsnorm_fwd: null input");
  if ((q8 == nullptr) != (qscale == nullptr)) return set_error(LLAMAX_ERR_ARG, "rmsnorm_fwd: q8 and qscale go together");
  if (!row_cfg(D, c)) return set_error(LLAMAX_ERR_ARG, "rmsnorm_fwd: D must be a multiple of 8 and <= 65536");
  if (M == 0) return 0;
  int ring_grid, ring_smem, wv, wgrid, wsmem;
  if (wpr_cfg(c.nvec, M, ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w)) % 16) == 0, wv, wgrid, wsmem,
              true)) {
    LX_DISPATCH_WPR(wv, {
      if (c.nvec == 32 * kV) {
        LX_RING_SMEM((row_wpr_kernel<kV, true, true>), wsmem, "rmsnorm_fwd");
        row_wpr_kernel<kV, true, true><<<wgrid, 32 * kWprWarps, wsmem, (cudaStream_t)stream>>>(
            (const bf16*)x, D, (const bf16*)w, (bf16*)y, (float*)rstd, (int8_t*)q8, (bf16*)qscale, M, (int)D, c.nvec, eps);
      } else {
        LX_RING_SMEM((row_wpr_kernel<kV, true, false>), wsmem, "rmsnorm_fwd");
        row_wpr_kernel<kV, true, false><<<wgrid, 32 * kWprWarps, wsmem, (cudaStream_t)stream>>>(
            (const bf16*)x, D, (const bf16*)w, (bf16*)y, (float*)rstd, (int8_t*)q8, (bf16*)qscale, M, (int)D, c.nvec, eps);
      }
    });
  } else if (ring_cfg(c, M, (reinterpret_cast<uintptr_t>(x) % 16) == 0, ring_grid, ring_smem)) {
    LX_DISPATCH_V(c.V, {
      LX_RING_SMEM(rmsnorm_fwd_ring_kernel<kV>, ring_smem, "rmsnorm_fwd");
      rmsnorm_fwd_ring_kernel<kV><<<ring_grid, c.threads, ring_smem, (cudaStream_t)stream>>>(
          (const bf16*)x, (const bf16*)w, (bf16*)y, (float*)rstd, (int8_t*)q8, (bf16*)qscale, M, (int)D, c.nvec, eps);
    });
  } else {
    LX_DISPATCH_V(c.V, rmsnorm_fwd_kernel<kV><<<(unsigned)M, c.threads, 0, (cudaStream_t)stream>>>(
        (const bf16*)x, (const bf16*)w, (bf16*)y, (float*)rstd, (int8_t*)q8, (bf16*)qscale, (int)D, c.nvec, eps));
  }
  LX_CHECK_LAUNCH("rmsnorm_fwd");
  return 0;
}

int llamax_rowquant_int8(const void* x, int64_t ldx, void* q8, void* scale_out, int64_t M, int64_t K,
                         void* stream) {
  RowCfg c;
  if (!x || !q8 || !scale_out) return set_error(LLAMAX_ERR_ARG, "rowquant_int8: null pointer");
  if (!row_cfg(K, c) || ldx % 8) return set_error(LLAMAX_ERR_ARG, "rowquant_int8: K and ldx must be multiples of 8");
  if (M == 0) return 0;
  int ring_grid, ring_smem, wv, wgrid, wsmem;
  if (wpr_cfg(c.nvec, M, (reinterpret_cast<uintptr_t>(x) % 16) == 0, wv, wgrid, wsmem, false)) {
    LX_DISPATCH_WPR(wv, {
      if (c.nvec == 32 * kV) {
        LX_RING_SMEM((row_wpr_kernel<kV, false, true>), wsmem, "rowquant_int8");
        row_wpr_kernel<kV, false, true><<<wgrid, 32 * kWprWarps, wsmem, (cudaStream_t)stream>>>(
            (const bf16*)x, ldx, nullptr, nullptr, nullptr, (int8_t*)q8, (bf16*)scale_out, M, (int)K, c.nvec, 0.f);
      } else {
        LX_RING_SMEM((row_wpr_kernel<kV, false, false>), wsmem, "rowquant_int8");
        row_wpr_kernel<kV, false, false><<<wgrid, 32 * kWprWarps, wsmem, (cudaStream_t)stream>>>(
            (const bf16*)x, ldx, nullptr, nullptr, nullptr, (int8_t*)q8, (bf16*)scale_out, M, (int)K, c.nvec, 0.f);
      }
    });
  } else if (ring_cfg(c, M, (reinterpret_cast<uintptr_t>(x) % 16) == 0, ring_grid, ring_smem)) {
    LX_DISPATCH_V(c.V, {
      LX_RING_SMEM(rowquant_ring_kernel<kV>, ring_smem, "rowquant_int8");
      rowquant_ring_kernel<kV><<<ring_grid, c.threads, ring_smem, (cudaStream_t)stream>>>(
          (const bf16*)x, ldx, (int8_t*)q8, (bf16*)scale_out, M, (int)K, c.nvec);
    });
  } else {
    LX_DISPATCH_V(c.V, rowquant_kernel<kV><<<(unsigned)M, c.threads, 0, (cudaStream_t)stream>>>(
        (const bf16*)x, ldx, (int8_t*)q8, (bf16*)scale_out, (int)K, c.nvec));
  }
  LX_CHECK_LAUNCH("rowquant_int8");
  return 0;
}

int llamax_swiglu_fwd(const void* a, const void* b, int64_t ld, void* g, void* q8, void* qscale, int64_t M,
                      int64_t F, void* stream) {
  RowCfg c;
  if (!a || !b) return set_error(LLAMAX_ERR_ARG, "swiglu_fwd: null input");
  if ((q8 == nullptr) != (qscale == nullptr)) return set_error(LLAMAX_ERR_ARG, "swiglu_fwd: q8 and qscale go together");
  if (!row_cfg(F, c) || ld % 8) return set_error(LLAMAX_ERR_ARG, "swiglu_fwd: F and ld must be multiples of 8");
  if (M == 0) return 0;
  static const bool ring_on = getenv("LLAMAX_SWIGLU_RING") == nullptr || atoi(getenv("LLAMAX_SWIGLU_RING")) != 0;
  const bool aligned = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) % 16) == 0;
  const int smem = kRingStages * 2 * c.threads * c.V * 16;
  if (ring_on && aligned && c.V <= 4 && smem <= 200 * 1024) {
    const int per_sm = std::max(1, std::min((216 * 1024) / (smem + 1280), 2048 / c.threads));
    const int grid = sm_count() * per_sm;
    if (M >= (int64_t)grid * 2) {
      LX_DISPATCH_V(c.V, {
        if constexpr (kV <= 4) {
          LX_RING_SMEM(swiglu_fwd_ring_kernel<kV>, smem, "swiglu_fwd");
          swiglu_fwd_ring_kernel<kV><<<grid, c.threads, smem, (cudaStream_t)stream>>>(
              (const bf16*)a, (const bf16*)b, ld, (bf16*)g, (int8_t*)q8, (bf16*)qscale, M, (int)F, c.nvec);
        }
      });
      LX_CHECK_LAUNCH("swiglu_fwd");
      return 0;
    }
  }
  LX_DISPATCH_V(c.V, swiglu_fwd_kernel<kV><<<(unsigned)M, c.threads, 0, (cudaStream_t)stream>>>(
      (const bf16*)a, (const bf16*)b, ld, (bf16*)g, (int8_t*)q8, (bf16*)qscale, (int)F, c.nvec));
  LX_CHECK_LAUNCH("swiglu_fwd");
  return 0;
}

int llamax_swiglu_bwd(const void* dg, const void* a, const void* b, int64_t ld, void* da, void* db, int64_t ldd,
                      void* g, int64_t M, int64_t F, void* stream) {
  if (!dg || !a || !b || !da || !db) return set_error(LLAMAX_ERR_ARG, "swiglu_bwd: null pointer");
  if (F % 8 || ld % 8 || ldd % 8) return set_error(LLAMAX_ERR_ARG, "swiglu_bwd: F, ld and ldd must be multiples of 8");
  if (M == 0) return 0;
  const int64_t total = M * (F / 8);
  const int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 16);
  swiglu_bwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const bf16*)dg, (const bf16*)a, (const bf16*)b, ld,
                                                              (bf16*)da, (bf16*)db, ldd, (bf16*)g, M, (int)(F / 8));
  LX_CHECK_LAUNCH("swiglu_bwd");
  return 0;
}

int llamax_rmsnorm_bwd(const void* dy, const void* x, const void* w, const void* rstd, const void* dres, void* dx,
                       void* dw_partial, int32_t nparts, int64_t M, int64_t D, void* stream) {
  RowCfg c;
  if (!dy || !x || !w || !rstd || !dx) return set_error(LLAMAX_ERR_ARG, "rmsnorm_bwd: null pointer");
  if (!row_cfg(D, c, true)) return set_error(LLAMAX_ERR_ARG, "rmsnorm_bwd: D must be a multiple of 8 and <= 65536");
  if (nparts <= 0 || nparts > 4096) return set_error(LLAMAX_ERR_ARG, "rmsnorm_bwd: nparts out of range");
  // ring kernel: rows of up to 256 threads x 2 vectors (the model width), 16-byte aligned streams, a few rows per CTA
  static const bool ring_on = getenv("LLAMAX_RMSNORM_BWD_RING") == nullptr || atoi(getenv("LLAMAX_RMSNORM_BWD_RING")) != 0;
  RowCfg cr;
  const bool aligned = ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) |
                         reinterpret_cast<uintptr_t>(dres)) % 16) == 0;
  if (ring_on && aligned && row_cfg(D, cr) && cr.threads <= 256 && cr.V <= 2 && M >= (int64_t)nparts * 2) {
    const int smem = kRingStages * 3 * cr.threads * cr.V * 16;
    LX_DISPATCH_V(cr.V, {
      LX_RING_SMEM(rmsnorm_bwd_ring_kernel<kV>, smem, "rmsnorm_bwd");
      rmsnorm_bwd_ring_kernel<kV><<<nparts, cr.threads, smem, (cudaStream_t)stream>>>(
          (const bf16*)dy, (const bf16*)x, (const bf16*)w, (const float*)rstd, (const bf16*)dres, (bf16*)dx,
          (float*)dw_partial, M, (int)D, cr.nvec);
    });
    LX_CHECK_LAUNCH("rmsnorm_bwd");
    return 0;
  }
  LX_DISPATCH_V(c.V, rmsnorm_bwd_kernel<kV><<<nparts, c.threads, 0, (cudaStream_t)stream>>>(
      (const bf16*)dy, (const bf16*)x, (const bf16*)w, (const float*)rstd, (const bf16*)dres, (bf16*)dx,
      (float*)dw_partial, M, (int)D, c.nvec));
  LX_CHECK_LAUNCH("rmsnorm_bwd");
  return 0;
}

int llamax_reduce_partials(const void* partial, void* out, int32_t nparts, int64_t D, void* stream) {
  if (!partial || !out) return set_error(LLAMAX_ERR_ARG, "reduce_partials: null pointer");
  reduce_partials_kernel<<<(unsigned)((D + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const float*)partial,
                                                                                        (bf16*)out, nparts, D);
  LX_CHECK_LAUNCH("reduce_partials");
  return 0;
}

int llamax_rope_inplace(void* x, int64_t ld, const void* rope, int64_t B, int64_t S, int32_t nheads, int32_t D,
                        int inverse, void* stream) {
  if (!x || !rope) return set_error(LLAMAX_ERR_ARG, "rope: null pointer");
  if (D % 8 || ld % 8) return set_error(LLAMAX_ERR_ARG, "rope: D and ld must be multiples of 8");
  const int64_t rows = B * S;
  const int vec_per_row = nheads * D / 8;
  if (rows == 0 || vec_per_row == 0) return 0;
  if (rows > 0x7fffffffLL) return set_error(LLAMAX_ERR_ARG, "rope: more than 2^31 - 1 rows");
  if (reinterpret_cast<uintptr_t>(x) % 16) return set_error(LLAMAX_ERR_ARG, "rope: x must be 16-byte aligned");
  dim3 grid((unsigned)((rows + kRopeRows - 1) / kRopeRows), (unsigned)((vec_per_row + 255) / 256));
  rope_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((bf16*)x, ld, (const float*)rope, rows, (int)S, vec_per_row, D,
                                                      inverse);
  LX_CHECK_LAUNCH("rope");
  return 0;
}

int llamax_dequant_weight(const void* w8, const void* scale, void* out, int64_t ldo, int64_t N, int64_t K,
                          int transpose, int apply_scale, void* stream) {
  if (!w8 || !out || (apply_scale && !scale)) return set_error(LLAMAX_ERR_ARG, "dequant_weight: null pointer");
  if (K % 16 || N % 8 || ldo % 8 || (reinterpret_cast<uintptr_t>(out) % 16))
    return set_error(LLAMAX_ERR_ARG, "dequant_weight: K % 16, N % 8, ldo % 8 and 16-byte aligned out required");
  if (!transpose) {
    const int64_t nvec = N * K / 16;
    const int blocks = (int)std::min<int64_t>((nvec + 255) / 256, (int64_t)sm_count() * 16);
    dequant_plain_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const int8_t*)w8, (const bf16*)scale, (bf16*)out,
                                                                   ldo, N, K, apply_scale);
  } else {
    dim3 grid((unsigned)((K + 63) / 64), (unsigned)((N + 63) / 64));
    dequant_transpose_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const int8_t*)w8, (const bf16*)scale,
                                                                     (bf16*)out, ldo, (int)N, (int)K, apply_scale);
  }
  LX_CHECK_LAUNCH("dequant_weight");
  return 0;
}

int llamax_cross_entropy(void* logits, int64_t ld, const void* labels, void* loss_sum, const void* inv_n, int64_t M,
                         int64_t V, int write_grad, void* stream) {
  if (!logits || !labels || !loss_sum || (write_grad && !inv_n)) return set_error(LLAMAX_ERR_ARG, "cross_entropy: null pointer");
  if (V % 8 || ld % 8) return set_error(LLAMAX_ERR_ARG, "cross_entropy: V and ld must be multiples of 8");
  if (M == 0) return 0;
  cross_entropy_kernel<<<(unsigned)M, 512, 0, (cudaStream_t)stream>>>((bf16*)logits, ld, (const int64_t*)labels,
                                                                      (float*)loss_sum, (const float*)inv_n, (int)V,
                                                                      write_grad);
  LX_CHECK_LAUNCH("cross_entropy");
  return 0;
}

int llamax_cross_entropy_rows(void* logits, int64_t ld, const void* labels, void* loss_rows, const void* inv_n,
                              int64_t M, int64_t V, int write_grad, void* stream) {
  if (!logits || !labels || !loss_rows || (write_grad && !inv_n)) return set_error(LLAMAX_ERR_ARG, "cross_entropy: null pointer");
  if (V % 8 || ld % 8) return set_error(LLAMAX_ERR_ARG, "cross_entropy: V and ld must be multiples of 8");
  if (M == 0) return 0;
  cross_entropy_kernel<true><<<(unsigned)M, 512, 0, (cudaStream_t)stream>>>((bf16*)logits, ld, (const int64_t*)labels,
                                                                            (float*)loss_rows, (const float*)inv_n,
                                                                            (int)V, write_grad);
  LX_CHECK_LAUNCH("cross_entropy");
  return 0;
}

int llamax_batched_copy(const llamax_copy_job_t* jobs, int32_t n_jobs, void* stream) {
  if (n_jobs == 0) return 0;
  if (!jobs || n_jobs < 0 || n_jobs > LLAMAX_MAX_COPY_JOBS) return set_error(LLAMAX_ERR_ARG, "batched_copy: bad job list");
  CopyJobs cj;
  int max_tiles = 1;
  for (int i = 0; i < n_jobs; ++i) {
    const llamax_copy_job_t& j = jobs[i];
    if (!j.src || !j.dst || j.rows <= 0 || j.cols <= 0) return set_error(LLAMAX_ERR_ARG, "batched_copy: bad job");
    cj.j[i] = j;
    max_tiles = std::max(max_tiles, ((j.rows + 31) / 32) * ((j.cols + 31) / 32));
  }
  dim3 grid((unsigned)std::min(max_tiles, 512), (unsigned)n_jobs);   // tiny tiles: one per CTA where possible
  batched_copy_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(cj);
  LX_CHECK_LAUNCH("batched_copy");
  return 0;
}

int llamax_gelu_bias_fwd(void* z, const void* bias, void* y, int64_t rows, int64_t C, int32_t period, int32_t lo,
                         int32_t hi, void* stream) {
  if (!z || !bias || !y) return set_error(LLAMAX_ERR_ARG, "gelu_bias_fwd: null pointer");
  if (C % 8 || period <= 0 || lo < 0 || hi > period) return set_error(LLAMAX_ERR_ARG, "gelu_bias_fwd: bad shape");
  if (rows == 0) return 0;
  const int64_t total = rows * (C / 8);
  const int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 16);
  gelu_bias_fwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((bf16*)z, (const bf16*)bias, (bf16*)y, rows, (int)(C / 8),
                                                                 period, lo, hi);
  LX_CHECK_LAUNCH("gelu_bias_fwd");
  return 0;
}

int llamax_gelu_bwd(const void* dy, const void* z, void* dz, int64_t rows, int64_t C, int32_t period, int32_t lo,
                    int32_t hi, void* stream) {
  if (!dy || !z || !dz) return set_error(LLAMAX_ERR_ARG, "gelu_bwd: null pointer");
  if (C % 8 || period <= 0 || lo < 0 || hi > period) return set_error(LLAMAX_ERR_ARG, "gelu_bwd: bad shape");
  if (rows == 0) return 0;
  const int64_t total = rows * (C / 8);
  const int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 16);
  gelu_bwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const bf16*)dy, (const bf16*)z, (bf16*)dz, rows, (int)(C / 8),
                                                            period, lo, hi);
  LX_CHECK_LAUNCH("gelu_bwd");
  return 0;
}

int llamax_conv_s2k3_col2im(const void* dcol, void* dxp, int64_t B, int64_t Tp, int64_t C, void* stream) {
  if (!dcol || !dxp) return set_error(LLAMAX_ERR_ARG, "conv_s2k3_col2im: null pointer");
  if (C % 8 || Tp % 2 || Tp < 4 || B <= 0) return set_error(LLAMAX_ERR_ARG, "conv_s2k3_col2im: bad shape");
  const int64_t total = B * Tp * (C / 8);
  const int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 16);
  conv_s2k3_col2im_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const bf16*)dcol, (bf16*)dxp, B, (int)Tp, (int)(C / 8));
  LX_CHECK_LAUNCH("conv_s2k3_col2im");
  return 0;
}

int llamax_rowquant_int8_colscale(const void* x, int64_t ldx, const void* col_scale, void* q8, void* scale_out,
                                  int64_t M, int64_t K, void* stream) {
  RowCfg c;
  if (!x || !col_scale || !q8 || !scale_out) return set_error(LLAMAX_ERR_ARG, "rowquant_int8_colscale: null pointer");
  if (!row_cfg(K, c) || ldx % 8) return set_error(LLAMAX_ERR_ARG, "rowquant_int8_colscale: K and ldx must be multiples of 8");
  if (M == 0) return 0;
  LX_DISPATCH_V(c.V, rowquant_kernel<kV, true><<<(unsigned)M, c.threads, 0, (cudaStream_t)stream>>>(
      (const bf16*)x, ldx, (int8_t*)q8, (bf16*)scale_out, (int)K, c.nvec, (const bf16*)col_scale));
  LX_CHECK_LAUNCH("rowquant_int8_colscale");
  return 0;
}

}  // extern "C"
