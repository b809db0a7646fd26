// Shared device-side helpers for the llamax_b200 kernels (sm_100a only).
// Thin inline-PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace lx {

// ----------------------------------------------------------------------------------------------
// generic
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Warpgroup register re-allocation (every warp of the warpgroup executes it; counts are multiples of 8).
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// bf16 helpers -----------------------------------------------------------------------------------
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 r = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&r);
}
// fp32 -> nearest-even bf16 -> fp32, in integer arithmetic (ALU pipe). The cvt.rn.bf16.f32 instruction runs on the
// 16-lane/clk conversion (XU) pipe, which made the fused norm / SwiGLU passes XU-bound instead of HBM-bound.
__device__ __forceinline__ float round_bf16(float v) {
  uint32_t u = __float_as_uint(v);
  u += 0x7FFFu + ((u >> 16) & 1u);
  return __uint_as_float(u & 0xFFFF0000u);
}
// exact float of a signed byte held in the low 8 bits of w (any upper bits), without I2F (XU pipe):
// 0x4B400000 | (b ^ 0x80) is the float 12582912 + (b ^ 0x80), and (b ^ 0x80) = b + 128 for b read as int8.
__device__ __forceinline__ float s8_to_float(uint32_t w) {
  return __uint_as_float(0x4B400000u | ((w & 0xFFu) ^ 0x80u)) - 12583040.0f;
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Arrive on the barrier at the same smem offset in CTA `cta` of the cluster.
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
// Same, with the default (CTA-scope release) semantics. The explicit .release.cluster form above costs the arriving
// thread ~1500 cycles (measured with tools/mixed_gemm_trace.py: it drains the thread's outstanding shared-memory stores
// to cluster scope first) — fine once per tile, ruinous once per k-block. Use this one when the data the arrive
// publishes is consumed by the async proxy of the arriving thread's OWN CTA (tensor-core reads of this CTA's shared
// memory, ordered by fence.proxy.async) and only the barrier lives in the peer.
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Blocking wait. Built with -DLX_WATCHDOG (LLAMAX_NVCC_FLAGS=-DLX_WATCHDOG python -m llamax_b200.build --force) the
// wait traps after 2^26 failed polls, so a protocol bug surfaces as a launch failure instead of a hung GPU; it is off
// by default because even a poll counter in this loop costs ~5 % in the attention kernels (measured, same box).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
#ifdef LX_WATCHDOG
  uint32_t polls = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++polls == (1u << 26)) __trap();
  }
#else
  while (!mbar_try_wait(bar, parity)) {
  }
#endif
}

// Same wait with cluster-scope acquire: the arrivals come from threads of the peer CTA that published shared-memory
// writes (release.cluster) this CTA's tensor-core instruction is about to consume.
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
#ifdef LX_WATCHDOG
  uint32_t polls = 0;
#endif
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
#ifdef LX_WATCHDOG
    if (!ok && ++polls == (1u << 26)) __trap();
#endif
  } while (!ok);
}

// ----------------------------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// 2-CTA variant: data lands in this CTA's smem, completion bytes are signalled on the barrier of the
// CTA that owns the (cluster-mapped) barrier address `bar_cluster_addr`.
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr,
                                                int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
// smem -> global bulk reduction (fp32 add performed at L2): dst[i] += src[i] for `bytes` bytes (multiple of 16)
__device__ __forceinline__ void bulk_reduce_add_f32(float* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(gdst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ----------------------------------------------------------------------------------------------
// cluster
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta));
  return r;
}

// ----------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------------------------
template <int CG = 1>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  if constexpr (CG == 1)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
                 "r"(ncols)
                 : "memory");
  else
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
                 "r"(ncols)
                 : "memory");
}
template <int CG = 1>
__device__ __forceinline__ void tmem_relinquish() {
  if constexpr (CG == 1)
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  else
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int CG = 1>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (CG == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// Wait for outstanding tcgen05.ld and pin the destination registers behind the wait (zero-cost compiler fence:
// keeps uses of r[] from being scheduled above the wait).
template <int N>
__device__ __forceinline__ void tmem_wait_ld_regs(uint32_t (&r)[N]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < N; ++i) asm volatile("" : "+r"(r[i])::"memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// MMA completion -> mbarrier (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 2-CTA: arrive on the barrier at this smem offset in every CTA of `cta_mask`.
__device__ __forceinline__ void umma_commit_cg2(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// Shared-memory matrix descriptor (sm_100 "version 1"), 128-byte swizzle.
//   K-major  operand: rows of 128 B along K, 8-row atoms of 1024 B; SBO = bytes between 8-row groups.
//   MN-major operand: rows of 128 B along MN (64 x 16-bit), 8 K-rows per 1024 B atom;
//                     LBO = bytes between 64-element MN atoms, SBO = bytes between 8-row K groups.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= 1ull << 46;  // descriptor version (Blackwell)
  d |= 2ull << 61;  // SWIZZLE_128B
  return d;
}

// Split form for hot issue loops: hi word is constant per operand kind, lo word = (addr >> 4) | (lbo >> 4) << 16,
// so stepping an operand costs one 32-bit add (byte offset >> 4).
__device__ __forceinline__ uint32_t desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
  return ((smem_addr & 0x3FFFFu) >> 4) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__host__ __device__ constexpr uint32_t desc_hi(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | (2u << 29);
}
__device__ __forceinline__ uint64_t desc_join(uint32_t lo, uint32_t hi) {
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

// Instruction descriptor (upper 32 bits of idescE), dense, no negate, no saturate.
//   c_fmt: 1 = F32, 2 = S32; ab_fmt: kind::f16 -> 0 F16 / 1 BF16, kind::i8 -> 0 U8 / 1 S8
//   a_mn / b_mn: 1 = operand is MN-major in smem
__host__ __device__ constexpr uint32_t make_idesc(uint32_t c_fmt, uint32_t ab_fmt, uint32_t M, uint32_t N,
                                                  uint32_t a_mn = 0, uint32_t b_mn = 0) {
  return (c_fmt << 4) | (ab_fmt << 7) | (ab_fmt << 10) | (a_mn << 15) | (b_mn << 16) | ((N >> 3) << 17) |
         ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]
template <bool kInt8, int CG = 1>
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
  if constexpr (kInt8) {
    if constexpr (CG == 1) {
      asm volatile(
          "{\n\t"
          ".reg .pred p;\n\t"
          "setp.ne.b32 p, %4, 0;\n\t"
          "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
          "}\n" ::"r"(d_tmem),
          "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
          : "memory");
    } else {
      asm volatile(
          "{\n\t"
          ".reg .pred p;\n\t"
          "setp.ne.b32 p, %4, 0;\n\t"
          "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t"
          "}\n" ::"r"(d_tmem),
          "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
          : "memory");
    }
  } else {
    if constexpr (CG == 1) {
      asm volatile(
          "{\n\t"
          ".reg .pred p;\n\t"
          "setp.ne.b32 p, %4, 0;\n\t"
          "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
          "}\n" ::"r"(d_tmem),
          "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
          : "memory");
    } else {
      asm volatile(
          "{\n\t"
          ".reg .pred p;\n\t"
          "setp.ne.b32 p, %4, 0;\n\t"
          "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
          "}\n" ::"r"(d_tmem),
          "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
          : "memory");
    }
  }
}

// D[tmem] (+)= A[tmem] * B[smem]   (bf16, cta_group::1)
__device__ __forceinline__ void umma_ts_f16(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// TMEM -> registers: 32 lanes x 32 consecutive 32-bit columns; thread i of the warp gets lane (base+i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// registers -> TMEM, same shape.
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
// registers -> TMEM: 32 lanes x 16 consecutive 32-bit columns.
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// 16-lane fragment shapes (layouts verified with tools/tmem_layout_probe.cu; `taddr` lane field = first of the 16 lanes,
// which must lie in the warp's own quarter, i.e. 32 * (warp % 4) or that + 16):
//   16x256b.x4 (32 fp32 columns): register 4g + {0, 1} = row lane / 4,     columns 8g + 2 (lane % 4) + {0, 1}
//                                 register 4g + {2, 3} = row lane / 4 + 8, same columns               (g = 0..3)
//   16x128b.x4 (16 32-bit columns): register 2g = row lane / 4, column 4g + lane % 4; register 2g + 1 = row lane / 4 + 8
// so two adjacent fp32 columns of the first shape, packed to a bf16 pair, are exactly one word of the second.
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_16x256b_x4(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.16x256b.x4.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_16x128b_x4(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.16x128b.x4.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}

__device__ __forceinline__ void red_add_f32(float* p, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// four consecutive fp32 adds as ONE L2 reduction (16-byte aligned address)
__device__ __forceinline__ void red_add_v4_f32(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// 16-byte global access helpers
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_v4(void* p, const uint4& v) {
  asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

// 32-byte global accesses (one full sector per thread; sm_100 LDG/STG.256). `wide` = the address is 32-byte aligned,
// otherwise two 16-byte accesses.
__device__ __forceinline__ void ldg_nc_32B(const void* p, uint32_t (&r)[8], bool wide) {
  if (wide) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
  } else {
    const uint4 lo = ldg_nc_v4(p), hi = ldg_nc_v4(static_cast<const uint8_t*>(p) + 16);
    r[0] = lo.x; r[1] = lo.y; r[2] = lo.z; r[3] = lo.w; r[4] = hi.x; r[5] = hi.y; r[6] = hi.z; r[7] = hi.w;
  }
}
__device__ __forceinline__ void stg_32B(void* p, const uint32_t (&r)[8], bool wide) {
  if (wide) {
    asm volatile("st.global.v8.u32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]),
                 "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
  } else {
    stg_v4(p, make_uint4(r[0], r[1], r[2], r[3]));
    stg_v4(static_cast<uint8_t*>(p) + 16, make_uint4(r[4], r[5], r[6], r[7]));
  }
}


// bf16x2 * bf16x2 -> bf16x2, round-to-nearest-even of the exact products (HMUL2.BF16). The fp32 product of two bf16
// values is exact, so this equals bf16(float(x) * float(y)) — the reference's bf16 multiply — in one instruction per
// two elements instead of two unpacks, two FMULs and a rounding each.
__device__ __forceinline__ uint32_t mul_bf16x2(uint32_t x, uint32_t y) {
  uint32_t d;
  asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(x), "r"(y));
  return d;
}

// sigmoid in fp32 (fast exp / divide, ~2 ulp; every use is rounded to bf16 right after)
// exp(-a) through ex2.approx.ftz: the non-ftz form __expf compiles to spends a compare and two predicated multiplies per
// element on denormal RESULTS (ex2(x/2)^2 below 2^-126); here the result only ever feeds 1 + exp(-a), where anything below
// 2^-126 rounds away — same value bit for bit, three instructions less.
__device__ __forceinline__ float exp_neg_f(float a) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a * -1.4426950216293334961f));
  return r;
}
__device__ __forceinline__ float sigmoid_f(float a) { return __fdividef(1.0f, 1.0f + exp_neg_f(a)); }

// SwiGLU backward for TWO adjacent elements held as packed bf16 pairs (modelling/llama.py:143-152 differentiated,
// with the reference's bf16 roundings: sl = bf16(silu(a)), dsl = bf16(dg * b), outputs bf16):
//   db = bf16(dg * sl)    da = bf16(dsl * silu'(a))    g = bf16(sl * b)
// Products of two bf16 values use mul_bf16x2 (exact product, one rounding). Shared by swiglu_bwd_kernel and the fused
// epilogue of the w2 grad_input GEMM, so both give identical results.
__device__ __forceinline__ void swiglu_bwd_pair(uint32_t dg2, uint32_t a2, uint32_t b2, uint32_t& da2, uint32_t& db2,
                                                uint32_t& g2) {
  const float a0 = bf16_lo(a2), a1 = bf16_hi(a2);
  const float sig0 = sigmoid_f(a0), sig1 = sigmoid_f(a1);
  const uint32_t sl2 = pack_bf16(a0 * sig0, a1 * sig1);
  const uint32_t dsl2 = mul_bf16x2(dg2, b2);
  db2 = mul_bf16x2(dg2, sl2);
  g2 = mul_bf16x2(sl2, b2);
  da2 = pack_bf16(bf16_lo(dsl2) * (sig0 * (1.0f + a0 * (1.0f - sig0))),
                  bf16_hi(dsl2) * (sig1 * (1.0f + a1 * (1.0f - sig1))));
}

}  // namespace lx
