// tcgen05 GEMM for the frozen-base projections of the Llama decoder block.
//
//   C[M,N] = epilogue( A[M,K] * B[N,K]^T )       A, B both contraction-contiguous ("K-major")
//
// Two instantiations of one warp-specialised persistent kernel:
//   kInt8 = true  : int8 x int8 -> int32 (tcgen05.mma.kind::i8), epilogue (f32(acc) * a_scale[m]) * b_scale[n]
//                   replaces the Triton kernel of the reference (subclasses/int8_mm.py:50-118)
//   kInt8 = false : bf16 x bf16 -> fp32 (tcgen05.mma.kind::f16); weight-only forward (subclasses/int8.py:118)
//                   and grad_input (subclasses/int8.py:127) run on it with a de-quantised weight operand.
// Fused epilogue options: LoRA up-projection (modelling/lora.py:43), residual add (modelling/llama.py:172-173), and
// (kSwi) the SwiGLU backward behind the w2 grad_input GEMM (modelling/llama.py:152 differentiated).
// kMN: both operands stored [K, M] / [K, N] (weight-gradient form dW = dY^T X), consumed as MN-major UMMA operands.
// kRes: residual (or, in row-dot mode, the attention output for delta = rowsum(dO * O)) read through a prefetch pipeline.
// kMix: mixed-input variants (SURVEY K4 / K5): B arrives as the frozen INT8 weight and is expanded to bf16 by converter
//       warps between the TMA ring and the tensor core (640 threads, three rings; see the comment above gemm_kernel).
// gemm_wide_kernel: 512 x 256 outputs per CTA-pair visit for long contractions without an epilogue (further down).
//
// Structure (per CTA, 384 threads): warp0 = TMA producer, warp1 = MMA issuer, warp2 = TMEM allocator, warp3 idle,
// warps4-11 = epilogue (TMEM -> registers -> global; two warps per TMEM lane quarter, one per column half of the
// tile). smem ring of kStages {A,B} tiles with 128B swizzle, two TMEM accumulator stages (2 x 256 columns) so the
// epilogue of tile i overlaps the main loop of tile i+1.
// CG = 2 runs CTA pairs (cta_group::2, UMMA 256 x 256): each CTA loads its 128 rows of A and half of B.
#include "common.cuh"
#include "host_utils.h"
#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdlib>
#include <mutex>

#include "llamax_b200.h"

namespace lx {

#ifdef LX_MIX_TRACE
// tools-only build: SM-clock timestamps of the mixed-input pipeline's roles (cluster 0, leader CTA), read back through
// llamax_debug_mix_trace. Row layout: [role 0 = MMA issuer, 1 = converter warp 12][64 k-blocks][8 marks].
__device__ long long g_mix_trace[2 * 64 * 8];
#define MIX_MARK(role, idx, m)                                                                       \
  do {                                                                                               \
    if (blockIdx.x == 0 && (idx) < 64) g_mix_trace[((role) * 64 + (idx)) * 8 + (m)] = clock64();     \
  } while (0)
#else
#define MIX_MARK(role, idx, m) do {} while (0)
#endif

constexpr int kBM = 128;          // rows of A per CTA
constexpr int kBN = 256;          // accumulator columns per tile
constexpr int kBKBytes = 128;     // one 128B swizzle row of K per stage
constexpr int kMaxLoraRank = 16;
constexpr int kGemmThreads = 384;      // warps 0-3: TMA / MMA / TMEM alloc / idle; warps 4-11: epilogue
constexpr int kEpiThreads = 256;
constexpr int kGroupM = 8;        // tiles of the shorter dimension per scheduling group (L2 reuse of the operand panels)

struct GemmParams {
  int M, N, K;
  void* C;
  int64_t ldc;
  const __nv_bfloat16* row_scale;
  const __nv_bfloat16* col_scale;
  const __nv_bfloat16* lora_h;
  int64_t ldh;
  const __nv_bfloat16* lora_b;
  int lora_rank;
  float lora_scale;
  const __nv_bfloat16* resid;
  int64_t ldr;
  int seg_n0, seg_n1;  // LoRA column segments (0 = none): see llamax_epilogue_t
  // row-dot mode (flags & 4, kRes kernels): `resid` is not added; dot_out[(m / dot_S) * (N / 128) + g][m % dot_S] =
  // sum over the 128 columns of group g of bf16(C[m, c]) * resid[m, c]  (the attention backward's delta)
  float* dot_out;
  int dot_S;
  int* wave_sync;   // wave alignment counters (one per sync point) or null; sync_every: visits between two sync points
  int sync_every;
  int flags;  // 1: dump raw accumulator (int32 / fp32) to C; 2: round to bf16 before the column scale; 4: row-dot mode
  // kSwi epilogue (SwiGLU backward fused behind the w2 grad_input GEMM): C is not written
  const __nv_bfloat16* swi_ab;  // [M, 2N] pitch ld_ab: a = w1 x in columns [0, N), b = w3 x in [N, 2N)
  int64_t ld_ab;
  __nv_bfloat16* swi_dab;       // da -> columns [0, N), db -> [N, 2N), pitch ld_dab
  int64_t ld_dab;
  __nv_bfloat16* swi_g;         // optional g = bf16(silu(a)) * b, [M, N] contiguous
  int group;                    // tile-order group (set by the launcher, see tile_coords)
  // mixed-input variants (kMix): B arrives as int8 and is expanded to bf16 in shared memory
  // kRope epilogue (INT8 q | k | v projection): RoPE applied to the bf16-rounded outputs of columns [0, rope_cols) before
  // the store; rope fp32 [rope_S, 64, 2] (cos, sin), head_dim 128, position = row % rope_S
  const float* rope;
  int rope_S, rope_cols;
  const __nv_bfloat16* k_scale; // kMix == 2: per-contraction-index scale folded into the operand, bf16 [K1]
  int K1;                       // kMix == 2: contraction indices [0, K1) come from the int8 tensor (K1 % 64 == 0),
                                // [K1, K) from the bf16 tail tensor (LoRA A rows)
};

// kMix != 0 (mixed-input bf16 x int8, CG = 2 only): three rings instead of one. A: kStages x 16 KB (TMA -> MMA);
// raw: kRawStages x 8 KB int8 boxes of the B half-tile (TMA -> converter warps); B: kBStages x 16 KB bf16 (converter
// warps -> MMA). The raw ring is what hides the global-memory latency of B (small stages: it can be deep); the B ring
// only has to cover the local conversion latency. With one ring of {A, B, raw} stages only 5 fit and every stage's
// round trip contained TMA latency + conversion + MMA: 740-830 TFLOP/s against 1300 for the plain bf16 kernel.
template <int CG, int kMix = 0>
struct GemmSmem {
  static constexpr int kABytes = kBM * kBKBytes;               // 16 KB
  static constexpr int kBBytes = (kBN / CG) * kBKBytes;        // 32 KB / 16 KB
  static constexpr int kRawBytes = kMix ? (kBN / CG) * 64 : 0; // 8 KB of int8
  static constexpr int kStages = CG == 1 ? 4 : 6;
  static constexpr int kBStages = kMix ? 4 : kStages;          // kMix == 0: B lives in the A ring's stages
  static constexpr int kRawStages = kMix ? 6 : 1;              // (1: keeps the dead kMix code of plain variants well-formed)
  static constexpr int kStageBytes = kMix ? kABytes : kABytes + kBBytes;
  static constexpr int kOffB = kStages * kStageBytes;          // kMix: B ring
  static constexpr int kOffRaw = kOffB + (kMix ? kBStages * kBBytes : 0);
  static constexpr int kOffAux = kOffRaw + kRawStages * kRawBytes;
  static constexpr int kAuxBytes = kBN * 4 + kBN * kMaxLoraRank * 4;  // col scale + lora_b (fp32)
  static constexpr int kNumBars = 2 * kStages + 4 + 1 + 2 * kRawStages + (kMix ? 2 * kBStages : 0);
  static constexpr int kBarBytes = kNumBars * 8 + 16;
  static constexpr int kTotal = kOffAux + kAuxBytes + kBarBytes + 1024;  // + align slack
  static_assert(kTotal <= 232448, "GEMM shared memory budget");
};

constexpr int kMixThreads = 640;        // + warps 12-19: int8 -> bf16 converters of the mixed-input variants
constexpr int kMixPairs = 4;            // converter warp pairs, round-robin over the k-blocks
// setmaxnreg budgets. The pool is what the CTA was launched with — 640 threads x 96 registers (launch bound) = 61440,
// not the whole register file (a first version that summed to 65536 dead-locked in setmaxnreg.inc):
// 128 x 40 (control) + 256 x 152 (epilogue) + 256 x 64 (converters) = 60416
constexpr int kMixRegsCtrl = 40, kMixRegsEpi = 152, kMixRegsConv = 64;
static_assert(128 * kMixRegsCtrl + 256 * kMixRegsEpi + 256 * kMixRegsConv <= kMixThreads * 96, "setmaxnreg pool");

// Exact bf16 pairs of four signed bytes (one raw word): 0x43xx is the bf16 128 + (xx & 0x7f) when bit 7 of xx is
// clear and the exponent's last bit when it is set, so with t = [0x43, b] per 16-bit lane,
//   (t & 0x437f) - (t & 0x4380) = (128 + (b & 127)) - (128 | 256) = b as a signed byte, exactly — one byte permute,
// two logic ops and one packed subtract per two elements, nothing on the conversion (XU) pipe.
__device__ __forceinline__ uint32_t sub_bf16x2(uint32_t x, uint32_t y) {
  uint32_t d;
  asm("sub.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(x), "r"(y));
  return d;
}
__device__ __forceinline__ void s8x4_to_bf16x4(uint32_t w, uint32_t& lo, uint32_t& hi) {
  const uint32_t t0 = __byte_perm(w, 0x43434343u, 0x4140), t1 = __byte_perm(w, 0x43434343u, 0x4342);
  lo = sub_bf16x2(t0 & 0x437F437Fu, t0 & 0x43804380u);
  hi = sub_bf16x2(t1 & 0x437F437Fu, t1 & 0x43804380u);
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Tile order. One wave = `clusters` consecutive tiles (74 CTA pairs), and the operand panels a wave touches should stay
// as few as possible: a group takes kGroupM tiles of one dimension and sweeps the other dimension completely, fastest
// index inside the group, so a wave covers ~8 x 9.25 tiles = 17.25 live panels — except where it straddles two groups.
// Groups therefore run along the LONGER dimension (fewer, longer groups): with 64 x 16 tiles (M = 16384, N = 4096),
// groups of 8 m-tiles x 16 n-tiles (128 tiles, 1.7 waves) keep 21.7 panels live on average, groups of 8 n-tiles x 64
// m-tiles (512 tiles, 6.9 waves) 18.3. group > 0: m-groups sweeping n; group < 0: n-groups sweeping m.
__device__ __forceinline__ void tile_coords(int tile, int num_m, int num_n, int group, int& tm, int& tn) {
  if (group > 0) {
    const int per_group = group * num_n;
    const int g = tile / per_group;
    const int first_m = g * group;
    const int gsize = min(num_m - first_m, group);
    const int r = tile - g * per_group;
    tm = first_m + r % gsize;
    tn = r / gsize;
  } else {
    const int gn = -group;
    const int per_group = gn * num_m;
    const int g = tile / per_group;
    const int first_n = g * gn;
    const int gsize = min(num_n - first_n, gn);
    const int r = tile - g * per_group;
    tn = first_n + r % gsize;
    tm = r / gsize;
  }
}

__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds_f1(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}

// kRank: compile-time LoRA rank of the epilogue (0 = none, 8, 16); runtime ranks are zero-padded up to it.
// kMN: both operands are stored "transposed", A_t [K, M] and B_t [K, N] with the M / N index contiguous (the
// weight-gradient form dW[out, in] = sum_tokens dY[token, out] * X[token, in] with tokens = K): the tiles are loaded as
// [64 k] x [64 mn] boxes and fed to the UMMA as MN-major operands — no transposed copy of either tensor.
// kSwi: the accumulator (+ LoRA term) is d(loss)/d(g) of the SwiGLU (llama.py:152); the epilogue rounds it to bf16 as
// the stand-alone GEMM would, then applies the SwiGLU backward to the thread's a / b columns and writes da | db (| g)
// instead of dg: one [M, F] bf16 write + read and one launch less per block than GEMM -> swiglu_bwd_kernel.
// kRes: the residual term is read through the same one-group-ahead pipeline as kSwi's a / b (a 16-byte load per 8
// columns issued right before its use exposed one global-load latency per 8 columns: +37..64 % kernel time on the
// K = 4096 shapes, whose main loop is only ~16k cycles per tile). Requires resid != C.
// kMix (mixed-input, bf16 activations x frozen int8 weight, SURVEY K4 / K5; CG = 2, 512 threads): tmB maps the INT8
// weight as stored; the producer lands its raw [128 x 64]-byte box next to the stage, warps 12-15 expand it to bf16
// into the B slot of the stage (same 128B-swizzled layout a TMA load of a bf16 operand would have produced) and signal
// the leader CTA's conv barrier; the MMA issuer waits for both the A bytes and the converted B halves of the pair.
//   kMix == 1: B8 [N, K] (K contiguous), K-major operand — weight-only forward (subclasses/int8.py:118): exact
//              bf16(int8) values, the weight scale is applied to the bf16-rounded accumulator by the epilogue.
//   kMix == 2: B8 [K1, N] (N contiguous) = the weight AS STORED seen from grad_input (subclasses/int8.py:127),
//              MN-major operand, bf16(f32(w) * f32(k_scale[k])) — bit-identical to llamax_dequant_weight(transpose,
//              apply_scale) — followed by an optional bf16 tail tmT [K - K1, N] (the LoRA A rows) loaded by TMA
//              straight into the B slot. Neither a transposed nor a de-quantised copy of the weight exists.
template <bool kInt8, int CG, int kRank, bool kMN = false, bool kSwi = false, bool kRes = false, int kMix = 0,
          bool kRope = false>
__global__ void __launch_bounds__(kMix ? kMixThreads : kGemmThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmT, const GemmParams p) {
  static_assert(kMix == 0 || (!kInt8 && CG == 2 && !kMN), "mixed-input variants: bf16 accumulate, CTA pairs");
  static_assert(!kRope || (kRes && kInt8 && !kSwi && kMix == 0), "RoPE epilogue: a mode of the INT8 side-input (kRes) variant");
  using S = GemmSmem<CG, kMix>;
  constexpr int kStages = S::kStages;
  constexpr int kElemPerRow = kInt8 ? 128 : 64;  // K elements per 128 B
  constexpr int kTileM = kBM * CG;               // rows per cluster tile
  constexpr bool kBmn = kMN || kMix == 2;        // B operand is MN-major in shared memory

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  float* s_colscale = reinterpret_cast<float*>(smem + S::kOffAux);
  float* s_lorab = s_colscale + kBN;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_lorab + kBN * kMaxLoraRank);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kStages;
  uint64_t* tfull_bar = bars + 2 * kStages;
  uint64_t* tempty_bar = bars + 2 * kStages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);
  // kMix rings: raw int8 boxes (this CTA's barriers) and converted B halves (full: the leader's barrier, arrived on by
  // the converters of both CTAs; empty: MMA commit, multicast to both CTAs)
  constexpr int kRawStages = S::kRawStages, kBStages = S::kBStages;
  uint64_t* raw_full = bars + 2 * kStages + 5;
  uint64_t* raw_empty = raw_full + kRawStages;
  uint64_t* conv_bar = raw_empty + kRawStages;
  uint64_t* bempty_bar = conv_bar + kBStages;
  uint8_t* b_ring = smem + S::kOffB;
  uint8_t* raw_ring = smem + S::kOffRaw;

  const int warp = threadIdx.x >> 5;
  const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0;
  const bool is_leader = cta_rank == 0;

  const int num_m = (p.M + kTileM - 1) / kTileM;
  const int num_n = (p.N + kBN - 1) / kBN;
  const int num_tiles = num_m * num_n;
  const int num_kb = (p.K + kElemPerRow - 1) / kElemPerRow;
  const int cluster_id = blockIdx.x / CG;
  const int num_clusters = gridDim.x / CG;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && elect_one()) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 8 * CG);  // one arrive per epilogue warp of every CTA in the group
    }
    if constexpr (kMix != 0) {
      for (int i = 0; i < kRawStages; ++i) {
        mbar_init(&raw_full[i], 1);
        mbar_init(&raw_empty[i], 2);       // the two warps of the converting pair
      }
      for (int i = 0; i < kBStages; ++i) {
        mbar_init(&conv_bar[i], 2 * CG);   // one arrive per warp of the converting pair, both CTAs
        mbar_init(&bempty_bar[i], 1);
      }
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<CG>(tmem_slot, 512);
    tmem_relinquish<CG>();
  }
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int kb1 = kMix == 2 ? p.K1 / 64 : num_kb;   // k-blocks fed from the int8 tensor

  // kMix register budget (512 threads start with 128 each; the epilogue variants need up to 168): every role branch
  // below starts with its warpgroup's setmaxnreg
  if (kMix != 0 && warp < 4) setmaxnreg_dec<kMixRegsCtrl>();

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t full_addr = CG == 2 ? mapa_u32(smem_u32(&full_bar[0]), 0) : smem_u32(&full_bar[0]);
      int visit_p = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++visit_p) {
        int tm, tn;
        tile_coords(tile, num_m, num_n, p.group, tm, tn);
        const int row_a = tm * kTileM + cta_rank * kBM;
        const int row_b = tn * kBN + cta_rank * (kBN / CG);
        if (p.wave_sync != nullptr && visit_p > 0 && visit_p % p.sync_every == 0) {   // see gemm_wide_kernel
          const int expected = CG * min(num_clusters, num_tiles - visit_p * num_clusters);
          int* ctr = p.wave_sync + visit_p / p.sync_every;
          atomicAdd(ctr, 1);
          int seen;
          uint32_t polls = 0;
          do {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(ctr) : "memory");
          } while (seen < expected && ++polls < (1u << 14));
        }
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = stage_base + stage * S::kStageBytes;
          uint8_t* sb = sa + S::kABytes;
          if constexpr (kMix != 0) {   // A only: the raw B boxes have their own producer (warp 3) and ring
            if (is_leader) mbar_expect_tx(&full_bar[stage], S::kABytes * 2);
            tma_load_2d_cg2(sa, &tmA, full_addr + stage * 8, kb * 64, row_a);
          } else if constexpr (kMN) {
            // boxes of [64 k rows] x [64 mn elements = 128 B]: inner coordinate = mn index, outer = k
            constexpr int kBoxBytes = 64 * 128;
            if constexpr (CG == 1) {
              mbar_expect_tx(&full_bar[stage], S::kStageBytes);
#pragma unroll
              for (int i = 0; i < kBM / 64; ++i)
                tma_load_2d(sa + i * kBoxBytes, &tmA, &full_bar[stage], row_a + i * 64, kb * 64);
#pragma unroll
              for (int i = 0; i < kBN / 64; ++i)
                tma_load_2d(sb + i * kBoxBytes, &tmB, &full_bar[stage], row_b + i * 64, kb * 64);
            } else {
              if (is_leader) mbar_expect_tx(&full_bar[stage], S::kStageBytes * 2);
              const uint32_t bar_addr = full_addr + stage * 8;
#pragma unroll
              for (int i = 0; i < kBM / 64; ++i)
                tma_load_2d_cg2(sa + i * kBoxBytes, &tmA, bar_addr, row_a + i * 64, kb * 64);
#pragma unroll
              for (int i = 0; i < kBN / CG / 64; ++i)
                tma_load_2d_cg2(sb + i * kBoxBytes, &tmB, bar_addr, row_b + i * 64, kb * 64);
            }
          } else if constexpr (CG == 1) {
            mbar_expect_tx(&full_bar[stage], S::kStageBytes);
            tma_load_2d(sa, &tmA, &full_bar[stage], kb * kElemPerRow, row_a);
            tma_load_2d(sb, &tmB, &full_bar[stage], kb * kElemPerRow, row_b);
          } else {
            if (is_leader) mbar_expect_tx(&full_bar[stage], S::kStageBytes * 2);
            const uint32_t bar_addr = full_addr + stage * 8;
            tma_load_2d_cg2(sa, &tmA, bar_addr, kb * kElemPerRow, row_a);
            tma_load_2d_cg2(sb, &tmB, bar_addr, kb * kElemPerRow, row_b);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (is_leader && elect_one()) {
      constexpr uint32_t idesc = kInt8 ? make_idesc(2, 1, kTileM, kBN)
                                       : make_idesc(1, 1, kTileM, kBN, kMN ? 1 : 0, kBmn ? 1 : 0);
      int stage = 0;
      uint32_t phase = 0;
      int bstage = 0;
      uint32_t bphase = 0;
      int local_tile = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++local_tile) {
        const int as = local_tile & 1;
        const uint32_t aphase = (local_tile >> 1) & 1;
        mbar_wait(&tempty_bar[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * kBN;
        for (int kb = 0; kb < num_kb; ++kb) {
          if constexpr (kMix != 0) MIX_MARK(0, kb + local_tile * num_kb, 0);
          mbar_wait(&full_bar[stage], phase);
          if constexpr (kMix != 0) MIX_MARK(0, kb + local_tile * num_kb, 1);
          if constexpr (kMix != 0) mbar_wait_cluster(&conv_bar[bstage], bphase);
          if constexpr (kMix != 0) MIX_MARK(0, kb + local_tile * num_kb, 2);
          tc_fence_after();
          const uint32_t sa = smem_u32(stage_base + stage * S::kStageBytes);
          const uint32_t sb = kMix != 0 ? smem_u32(b_ring + bstage * S::kBBytes) : sa + S::kABytes;
          // K-major: 8-row atoms 1024 B apart, +32 B per k-step inside the swizzle atom (+2 in the addr >> 4 field);
          // MN-major: 64-element mn atoms one 8 KB box apart (LBO), 8-k-row groups 1024 B apart, +16 k rows = 2048 B
          const uint64_t adesc = make_smem_desc_sw128(sa, kMN ? 8192 : 16, 1024);
          const uint64_t bdesc = make_smem_desc_sw128(sb, kBmn ? 8192 : 16, 1024);
          constexpr int kStepA = kMN ? 128 : 2, kStepB = kBmn ? 128 : 2;
#pragma unroll
          for (int k = 0; k < kBKBytes / 32; ++k)
            umma_ss<kInt8, CG>(d_tmem, adesc + kStepA * k, bdesc + kStepB * k, idesc, (kb | k) != 0);
          if constexpr (CG == 1) umma_commit(&empty_bar[stage]); else umma_commit_cg2(&empty_bar[stage], 3);
          if constexpr (kMix != 0) {
            umma_commit_cg2(&bempty_bar[bstage], 3);
            if (++bstage == kBStages) { bstage = 0; bphase ^= 1; }
            MIX_MARK(0, kb + local_tile * num_kb, 3);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        if constexpr (CG == 1) umma_commit(&tfull_bar[as]); else umma_commit_cg2(&tfull_bar[as], 3);
      }
    }
    __syncwarp();
  } else if (kMix != 0 && warp == 3) {
    // ================================ raw int8 producer (kMix) ================================
    if (elect_one()) {
      int rs = 0;
      uint32_t rphase = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        int tm, tn;
        tile_coords(tile, num_m, num_n, p.group, tm, tn);
        const int row_b = tn * kBN + cta_rank * (kBN / CG);
        for (int kb = 0; kb < kb1; ++kb) {
          mbar_wait(&raw_empty[rs], rphase ^ 1);
          mbar_expect_tx(&raw_full[rs], S::kRawBytes);
          if constexpr (kMix == 1) tma_load_2d(raw_ring + rs * S::kRawBytes, &tmB, &raw_full[rs], kb * 64, row_b);
          else tma_load_2d(raw_ring + rs * S::kRawBytes, &tmB, &raw_full[rs], row_b, kb * 64);
          if (++rs == kRawStages) { rs = 0; rphase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (kMix != 0 && warp >= 12) {
    // ================================ int8 -> bf16 converters (kMix) ================================
    // Four pairs of warps take the k-blocks round-robin: a pair expands one raw box (512 sixteen-byte chunks, 8 per
    // thread) into a slot of the B ring. Measured with tools/mixed_gemm_trace.py, one k-block costs a pair ~700-800
    // cycles of conversion (ALU-pipe bound: byte permutes and logic ops issue at half rate) plus ~600-900 cycles of
    // serial overhead (two barrier waits, proxy fence, arrives, loop): two warps per scheduler overlap one pair's
    // overhead with another pair's arithmetic. Lane mappings keep every quarter-warp on 128 contiguous raw bytes and on
    // eight distinct 16-byte bank groups per store.
    setmaxnreg_dec<kMixRegsConv>();
    const int cw = warp - 12, cl = lane_id();
    const int pair = cw >> 1;
    const int t2 = (cw & 1) * 32 + cl;       // 0..63 within the pair
    const uint32_t conv_addr = mapa_u32(smem_u32(&conv_bar[0]), 0);   // the leader's conv barriers
    int it = 0;                               // k-block counter over all tiles of this CTA (B ring position)
    int rit = 0;                              // ... counting only the k-blocks that come from the int8 tensor (raw ring)
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
      int tm, tn;
      tile_coords(tile, num_m, num_n, p.group, tm, tn);
      const int row_b = tn * kBN + cta_rank * (kBN / CG);
      for (int kb = 0; kb < num_kb; ++kb, ++it) {
        const bool from_raw = kb < kb1;
        const int my_rit = rit;
        rit += from_raw ? 1 : 0;
        if ((it & (kMixPairs - 1)) != pair) continue;
        const int bs = it % kBStages;
        const uint32_t bphase = (it / kBStages) & 1;
        const uint32_t sb = smem_u32(b_ring + bs * S::kBBytes);
        if (from_raw) {
          const int rs = my_rit % kRawStages;
          const uint32_t rphase = (my_rit / kRawStages) & 1;
          uint32_t sc[8];
          if constexpr (kMix == 2) {   // this thread's eight k rows of the box: their scales, in flight during the waits
#pragma unroll
            for (int j = 0; j < 8; ++j)
              sc[j] = *reinterpret_cast<const uint16_t*>(p.k_scale + kb * 64 + j * 8 + (t2 >> 3));
          }
          if (cw == 0 && cl == 0) MIX_MARK(1, it >> 2, 0);
          mbar_wait(&raw_full[rs], rphase);
          if (cw == 0 && cl == 0) MIX_MARK(1, it >> 2, 1);
          mbar_wait(&bempty_bar[bs], bphase ^ 1);
          if (cw == 0 && cl == 0) MIX_MARK(1, it >> 2, 2);
          const uint32_t sraw = smem_u32(raw_ring + rs * S::kRawBytes);
#pragma unroll
          for (int half = 0; half < 4; ++half) {
            uint4 w[2];
            if constexpr (kMix == 1) {
              // raw rows of 64 B (n index), chunk c = 16 k values; bf16 tile rows of 128 B, chunk c -> chunks 2c, 2c+1
              const int c = t2 & 3;
#pragma unroll
              for (int j = 0; j < 2; ++j) w[j] = lds_v4(sraw + ((half * 2 + j) * 16 + (t2 >> 2)) * 64 + c * 16);
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const int r = (half * 2 + j) * 16 + (t2 >> 2);
                uint4 lo, hi;
                s8x4_to_bf16x4(w[j].x, lo.x, lo.y); s8x4_to_bf16x4(w[j].y, lo.z, lo.w);
                s8x4_to_bf16x4(w[j].z, hi.x, hi.y); s8x4_to_bf16x4(w[j].w, hi.z, hi.w);
                const uint32_t row = sb + r * 128;
                sts_v4(row + (((2 * c) ^ (r & 7)) << 4), lo);
                sts_v4(row + (((2 * c + 1) ^ (r & 7)) << 4), hi);
              }
            } else {
              // raw rows of 128 B (k index), chunk c = 16 n values -> box c / 4, bf16 chunks 2 (c % 4), + 1 of row kr.
              // Lanes c >= 4 store their upper half first: within a quarter-warp the stores of box 0 and box 1 then
              // fall on different bank groups.
              const int c = t2 & 7;
              const bool swp = (c & 4) != 0;
              const int c2 = 2 * (c & 3) + (swp ? 1 : 0);
#pragma unroll
              for (int j = 0; j < 2; ++j) w[j] = lds_v4(sraw + ((half * 2 + j) * 8 + (t2 >> 3)) * 128 + c * 16);
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const int kr = (half * 2 + j) * 8 + (t2 >> 3);
                uint4 v = w[j];
                if (swp) { const uint32_t a0 = v.x, a1 = v.y; v.x = v.z; v.y = v.w; v.z = a0; v.w = a1; }
                uint4 lo, hi;
                s8x4_to_bf16x4(v.x, lo.x, lo.y); s8x4_to_bf16x4(v.y, lo.z, lo.w);
                s8x4_to_bf16x4(v.z, hi.x, hi.y); s8x4_to_bf16x4(v.w, hi.z, hi.w);
                const uint32_t s16 = sc[half * 2 + j];
                const uint32_t s2 = s16 | (s16 << 16);
                lo.x = mul_bf16x2(lo.x, s2); lo.y = mul_bf16x2(lo.y, s2); lo.z = mul_bf16x2(lo.z, s2); lo.w = mul_bf16x2(lo.w, s2);
                hi.x = mul_bf16x2(hi.x, s2); hi.y = mul_bf16x2(hi.y, s2); hi.z = mul_bf16x2(hi.z, s2); hi.w = mul_bf16x2(hi.w, s2);
                const uint32_t row = sb + (c >> 2) * 8192 + kr * 128;
                sts_v4(row + ((c2 ^ (kr & 7)) << 4), lo);
                sts_v4(row + (((c2 ^ 1) ^ (kr & 7)) << 4), hi);
              }
            }
          }
          if (cw == 0 && cl == 0) MIX_MARK(1, it >> 2, 3);
          fence_proxy_async_smem();   // generic-proxy stores -> visible to the tensor core's async-proxy reads
          if (cw == 0 && cl == 0) MIX_MARK(1, it >> 2, 4);
          __syncwarp();
          if (cl == 0) {
            mbar_arrive(&raw_empty[rs]);                      // the raw box has been read (loads completed above)
            mbar_arrive_remote(&conv_bar[bs], 0);
          }
          if (cw == 0 && cl == 0) MIX_MARK(1, it >> 2, 5);
        } else {
          // tail k-block (kMix == 2): the bf16 LoRA-A rows go by TMA straight into this CTA's B slot, [64 k] x [64 n]
          // boxes = the MN-major operand layout. The pair's first warp posts the transaction bytes on the leader's conv
          // barrier together with its arrive; the second warp just arrives.
          mbar_wait(&bempty_bar[bs], bphase ^ 1);
          if (cl == 0) {
            const uint32_t bar = conv_addr + bs * 8;
            if ((cw & 1) == 0) {
              asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(bar),
                           "r"((uint32_t)S::kBBytes) : "memory");
#pragma unroll
              for (int i = 0; i < kBN / CG / 64; ++i)
                tma_load_2d_cg2(b_ring + bs * S::kBBytes + i * 8192, &tmT, bar, row_b + i * 64, (kb - kb1) * 64);
            } else {
              mbar_arrive_remote(&conv_bar[bs], 0);
            }
          }
          __syncwarp();
        }
      }
    }
  } else if (warp >= 4) {
    // ================================ epilogue ================================
    if constexpr (kMix != 0) setmaxnreg_inc<kMixRegsEpi>();
    const int ew = warp & 3;                 // TMEM lanes [32*ew, 32*ew+32) (hardware: warp % 4)
    const int ch = (warp - 4) >> 2;          // column half of the tile handled by this warp: chunks 4*ch .. 4*ch+3
    const int et = threadIdx.x - 128;        // 0..255
    const int R = p.lora_rank;
    constexpr int kRS = kRank > 0 ? kRank : 4;  // floats per staged lora_b row
    const uint32_t s_cs = smem_u32(s_colscale);
    const uint32_t s_lb = smem_u32(s_lorab);
    const bool dump = (p.flags & 1) != 0;
    const bool has_cs = p.col_scale != nullptr;
    const bool pre_round = (p.flags & 2) != 0;
    // 32-byte accesses when every row start of ab / dab / g is 32-byte aligned (N % 16 == 0 is required by the host)
    const bool res_wide = kRes && reinterpret_cast<uintptr_t>(p.resid) % 32 == 0 && p.ldr % 16 == 0;
    const bool swi_wide = kSwi && ((reinterpret_cast<uintptr_t>(p.swi_ab) | reinterpret_cast<uintptr_t>(p.swi_dab) |
                                    reinterpret_cast<uintptr_t>(p.swi_g)) % 32 == 0) &&
                          p.ld_ab % 16 == 0 && p.ld_dab % 16 == 0;
    // INT8 forward GEMMs: the per-tile operands of the epilogue (column scale and LoRA-B row of the thread's column,
    // row scale and LoRA-h row of the thread's row) are fetched one tile ahead into registers. Fetched at the top of
    // the tile, their global-load latency sat on the epilogue's critical path before every tile — which IS the kernel's
    // critical path at K = 4096 (~16k cycles of main loop per tile): the "+LoRA" cost of those shapes.
    static_assert(kBN == kEpiThreads, "one staged column per epilogue thread");
    constexpr bool kPipeStage = kInt8 || kSwi;
    constexpr int kRV = kRank > 0 ? kRank / 8 : 1;
    // h_vec: every h row starts on a 16-byte boundary (segment offsets are multiples of kRank, hence of 8 elements),
    // so h may be read with 16-byte loads. The header allows any h pitch and base: otherwise h is read element-wise.
    const bool h_vec = R == kRank && reinterpret_cast<uintptr_t>(p.lora_h) % 16 == 0 && p.ldh % 8 == 0;
    const bool fast_stage = kPipeStage && !dump &&
                            (kRank == 0 || (h_vec && reinterpret_cast<uintptr_t>(p.lora_b) % 16 == 0));
    uint32_t ncs = 0;
    float nrs = 1.f;
    uint4 nlb[kRV], nh[kRV];
    auto stage_fetch = [&](int t) {
      if (t >= num_tiles) return;
      int fm, fn;
      tile_coords(t, num_m, num_n, p.group, fm, fn);
      const int n = fn * kBN + et;
      const int frow = fm * kTileM + cta_rank * kBM + ew * 32 + lane_id();
      const int hoff = p.seg_n0 > 0 ? (fn * kBN >= p.seg_n1 ? 2 * kRank : fn * kBN >= p.seg_n0 ? kRank : 0) : 0;
      ncs = (has_cs && n < p.N) ? (uint32_t) * reinterpret_cast<const uint16_t*>(p.col_scale + n) : 0u;
      nrs = (p.row_scale != nullptr && frow < p.M) ? __bfloat162float(p.row_scale[frow]) : 1.f;
      if constexpr (kRank > 0) {
#pragma unroll
        for (int r8 = 0; r8 < kRV; ++r8) {
          nlb[r8] = n < p.N ? ldg_nc_v4(p.lora_b + (int64_t)n * kRank + r8 * 8) : make_uint4(0, 0, 0, 0);
          nh[r8] = frow < p.M ? ldg_nc_v4(p.lora_h + (int64_t)frow * p.ldh + hoff + r8 * 8) : make_uint4(0, 0, 0, 0);
        }
      }
    };
    if (fast_stage) stage_fetch(cluster_id);
    int local_tile = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++local_tile) {
      int tm, tn;
      tile_coords(tile, num_m, num_n, p.group, tm, tn);
      const int as = local_tile & 1;
      const uint32_t aphase = (local_tile >> 1) & 1;
      const int row = tm * kTileM + cta_rank * kBM + ew * 32 + lane_id();
      const int col0 = tn * kBN;
      const bool row_ok = row < p.M;

      // stage per-column data for this tile (previous tile's readers are done: barrier below)
      named_bar_sync(1, kEpiThreads);
      if (fast_stage) {
        if (has_cs) s_colscale[et] = bf16_lo(ncs);
        if constexpr (kRank > 0) {
#pragma unroll
          for (int r8 = 0; r8 < kRV; ++r8) {
            float* d = s_lorab + et * kRank + r8 * 8;
            const uint4 u = nlb[r8];
            d[0] = bf16_lo(u.x) * p.lora_scale; d[1] = bf16_hi(u.x) * p.lora_scale;
            d[2] = bf16_lo(u.y) * p.lora_scale; d[3] = bf16_hi(u.y) * p.lora_scale;
            d[4] = bf16_lo(u.z) * p.lora_scale; d[5] = bf16_hi(u.z) * p.lora_scale;
            d[6] = bf16_lo(u.w) * p.lora_scale; d[7] = bf16_hi(u.w) * p.lora_scale;
          }
        }
      } else {
        if (has_cs) {
          for (int i = et; i < kBN; i += kEpiThreads)
            s_colscale[i] = (col0 + i < p.N) ? __bfloat162float(p.col_scale[col0 + i]) : 0.f;
        }
        if constexpr (kRank > 0) {
          for (int i = et; i < kBN * kRank; i += kEpiThreads) {
            const int n = i / kRank, r = i % kRank;
            s_lorab[i] = (col0 + n < p.N && r < R)
                             ? __bfloat162float(p.lora_b[(int64_t)(col0 + n) * R + r]) * p.lora_scale : 0.f;
          }
        }
      }
      named_bar_sync(1, kEpiThreads);

      float rs = 1.f;
      float h[kRS];
#pragma unroll
      for (int r = 0; r < kRS; ++r) h[r] = 0.f;
      if (fast_stage) {
        rs = nrs;
        if constexpr (kRank > 0) {
#pragma unroll
          for (int r8 = 0; r8 < kRV; ++r8) {
            const uint4 u = nh[r8];
            const int r = r8 * 8;
            h[r + 0] = bf16_lo(u.x); h[r + 1] = bf16_hi(u.x); h[r + 2] = bf16_lo(u.y); h[r + 3] = bf16_hi(u.y);
            h[r + 4] = bf16_lo(u.z); h[r + 5] = bf16_hi(u.z); h[r + 6] = bf16_lo(u.w); h[r + 7] = bf16_hi(u.w);
          }
        }
        stage_fetch(tile + num_clusters);   // in flight during this tile's epilogue
      } else if (p.row_scale != nullptr && row_ok) {
        rs = __bfloat162float(p.row_scale[row]);
      }
      if constexpr (kRank > 0) {
        if (row_ok && !fast_stage) {
          const __nv_bfloat16* hp = p.lora_h + (int64_t)row * p.ldh +
                                    (p.seg_n0 > 0 ? (col0 >= p.seg_n1 ? 2 * R : col0 >= p.seg_n0 ? R : 0) : 0);
          if (h_vec) {
#pragma unroll
            for (int r = 0; r < kRank; r += 8) {
              const uint4 u = *reinterpret_cast<const uint4*>(hp + r);
              h[r + 0] = bf16_lo(u.x); h[r + 1] = bf16_hi(u.x); h[r + 2] = bf16_lo(u.y); h[r + 3] = bf16_hi(u.y);
              h[r + 4] = bf16_lo(u.z); h[r + 5] = bf16_hi(u.z); h[r + 6] = bf16_lo(u.w); h[r + 7] = bf16_hi(u.w);
            }
          } else {
#pragma unroll
            for (int r = 0; r < kRank; ++r)
              if (r < R) h[r] = __bfloat162float(hp[r]);
          }
        }
      }

      const int n_chunks = min(ch * 4 + 4, min(kBN / 32, (p.N - col0 + 31) / 32));
      // kSwi: this row's a / b values, 16 columns (32 B) per buffer, loaded one 16-column group ahead of their use
      // (two epilogue warps per scheduler cannot hide a global-load latency by themselves); oda / odb / odg collect
      // the packed results of a group for one 32 B store each.
      uint32_t pa[2][8], pb[2][8], oda[8], odb[8], odg[8];
      const unsigned rope_pos = kRope ? (unsigned)row % (unsigned)p.rope_S : 0u;
      auto swi_load = [&](int c16, uint32_t(&da)[8], uint32_t(&db)[8]) {   // c16: first of 16 columns
        if constexpr (kSwi) {
          if (row_ok && c16 < p.N) {
            const __nv_bfloat16* ap = p.swi_ab + (int64_t)row * p.ld_ab + c16;
            ldg_nc_32B(ap, da, swi_wide);
            ldg_nc_32B(ap + p.N, db, swi_wide);
          }
        } else if constexpr (kRope) {   // (cos, sin) of this row's position for the 8 pairs of 16 columns: 2 x 32 B
          if (row_ok && c16 < p.rope_cols) {
            const float* tp = p.rope + ((int64_t)rope_pos * 64 + ((c16 & 127) >> 1)) * 2;
            ldg_nc_32B(tp, da, true);
            ldg_nc_32B(tp + 8, db, true);
          }
        } else if constexpr (kRes) {   // residual row segment (N % 8 == 0: the last group may be half a group)
          if (row_ok && c16 < p.N) {
            const __nv_bfloat16* rp = p.resid + (int64_t)row * p.ldr + c16;
            if (c16 + 16 <= p.N) {
              ldg_nc_32B(rp, da, res_wide);
            } else {
              const uint4 lo = ldg_nc_v4(rp);
              da[0] = lo.x; da[1] = lo.y; da[2] = lo.z; da[3] = lo.w;
            }
          }
        }
      };
      if constexpr (kSwi || kRes) {
        if (ch * 4 < n_chunks) swi_load(col0 + ch * 4 * 32, pa[0], pb[0]);
      }
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t(ew * 32) << 16) + as * kBN;

      // accumulator chunks: double-buffered (next chunk's tcgen05.ld in flight) except with the kSwi epilogue, whose
      // per-chunk arithmetic dwarfs the TMEM latency and which needs the 32 registers for the a / b pipeline
      constexpr bool kSide = kSwi || kRes || (kPipeStage && kRank > 0);   // pipelined side inputs need the registers
      constexpr int kVBufs = kSide ? 1 : 2;
      uint32_t v[kVBufs][32];
      const bool rowdot = kRes && !kRope && (p.flags & 4) != 0;
      float dacc = 0.f;
      if constexpr (!kSide) {
        if (ch * 4 < n_chunks) tmem_ld_32x32(taddr + ch * 4 * 32, v[0]);
      }
#pragma unroll 1
      for (int c = ch * 4; c < n_chunks; c += 2) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int cc = c + half;
          if (cc >= n_chunks) break;
          uint32_t(&vv)[32] = v[kSide ? 0 : half];
          const int col = col0 + cc * 32;
          if constexpr (kSide) tmem_ld_32x32(taddr + cc * 32, vv);
          tmem_wait_ld_regs(vv);
          if constexpr (!kSide) {
            if (cc + 1 < n_chunks) tmem_ld_32x32(taddr + (cc + 1) * 32, v[half ^ 1]);  // prefetch next chunk
          }
          if (dump) {
            if (row_ok) {
              uint32_t* dst = reinterpret_cast<uint32_t*>(p.C) + (int64_t)row * p.ldc + col;
#pragma unroll
              for (int j = 0; j < 32; j += 4)
                if (col + j < p.N) stg_v4(dst + j, make_uint4(vv[j], vv[j + 1], vv[j + 2], vv[j + 3]));
            }
            continue;
          }
          const __nv_bfloat16* rsd = (p.resid && row_ok) ? p.resid + (int64_t)row * p.ldr + col : nullptr;
          __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.C) + (int64_t)row * p.ldc + col;
#pragma unroll
          for (int j8 = 0; j8 < 32; j8 += 8) {
            float f[8];
            float cs[8];
            if (kInt8 || has_cs) {
              const float4 c0 = lds_f4(s_cs + (cc * 32 + j8) * 4), c1 = lds_f4(s_cs + (cc * 32 + j8 + 4) * 4);
              cs[0] = c0.x; cs[1] = c0.y; cs[2] = c0.z; cs[3] = c0.w; cs[4] = c1.x; cs[5] = c1.y; cs[6] = c1.z; cs[7] = c1.w;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float a = kInt8 ? static_cast<float>(static_cast<int32_t>(vv[j8 + j])) : __uint_as_float(vv[j8 + j]);
              if constexpr (kInt8) {
                a = (a * rs) * cs[j];              // reference order: int8_mm.py:114
              } else if (has_cs) {
                if (pre_round) a = round_bf16(a);  // reference: bf16(x @ W^T) * s  (int8.py:118)
                a = a * cs[j];
              }
              if constexpr (kRank > 0) {
                const uint32_t lb = s_lb + (cc * 32 + j8 + j) * (kRank * 4);
                float acc = 0.f;
#pragma unroll
                for (int q = 0; q < kRank; q += 4) {
                  const float4 b4 = lds_f4(lb + q * 4);
                  acc = fmaf(h[q + 0], b4.x, acc);
                  acc = fmaf(h[q + 1], b4.y, acc);
                  acc = fmaf(h[q + 2], b4.z, acc);
                  acc = fmaf(h[q + 3], b4.w, acc);
                }
                a += acc;
              }
              f[j] = a;
            }
            if constexpr (kSwi) {
              // columns j8 .. j8+7 of the chunk: buffer (j8 >> 4) holds their a / b values; the other buffer is refilled
              // with the next 16-column group (second half of this chunk, or first half of the next one) meanwhile
              if (j8 == 0) swi_load(col + 16, pa[1], pb[1]);
              if (j8 == 16 && cc + 1 < n_chunks) swi_load(col + 32, pa[0], pb[0]);
#pragma unroll
              for (int j = 0; j < 8; j += 2) {
                const int w = ((j8 & 8) + j) >> 1;   // dg pair rounded to bf16 exactly as the stand-alone GEMM stores it
                swiglu_bwd_pair(pack_bf16(f[j], f[j + 1]), pa[j8 >> 4][w], pb[j8 >> 4][w], oda[w], odb[w], odg[w]);
              }
              if ((j8 & 8) && row_ok && col + (j8 & 16) < p.N) {
                const int64_t c16 = col + (j8 & 16);
                __nv_bfloat16* dp = p.swi_dab + (int64_t)row * p.ld_dab + c16;
                stg_32B(dp, oda, swi_wide);
                stg_32B(dp + p.N, odb, swi_wide);
                if (p.swi_g != nullptr) stg_32B(p.swi_g + (int64_t)row * p.N + c16, odg, swi_wide);
              }
            } else if constexpr (kRope) {
              if (j8 == 0) swi_load(col + 16, pa[1], pb[1]);
              if (j8 == 16 && cc + 1 < n_chunks) swi_load(col + 32, pa[0], pb[0]);
              if (row_ok && col + j8 < p.N) {
                uint32_t o[4] = {pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7])};
                if (col + j8 < p.rope_cols) {
                  // the linear's bf16 output, rotated pair by pair exactly like rope_kernel (separate products and
                  // sum, each rounded: modelling/llama.py:63-73), rounded to bf16 again
                  const uint32_t* t = (j8 & 8) ? pb[j8 >> 4] : pa[j8 >> 4];
#pragma unroll
                  for (int w = 0; w < 4; ++w) {
                    const float x0 = bf16_lo(o[w]), x1 = bf16_hi(o[w]);
                    const float cw = __uint_as_float(t[2 * w]), sw = __uint_as_float(t[2 * w + 1]);
                    o[w] = pack_bf16(__fsub_rn(__fmul_rn(x0, cw), __fmul_rn(x1, sw)),
                                     __fadd_rn(__fmul_rn(x1, cw), __fmul_rn(x0, sw)));
                  }
                }
                stg_v4(dst + j8, make_uint4(o[0], o[1], o[2], o[3]));
              }
            } else if constexpr (kRes) {
              if (j8 == 0) swi_load(col + 16, pa[1], pb[1]);
              if (j8 == 16 && cc + 1 < n_chunks) swi_load(col + 32, pa[0], pb[0]);
              if (row_ok && col + j8 < p.N) {
                const uint32_t* r4 = &pa[j8 >> 4][(j8 & 8) >> 1];
                uint4 o;
                if (rowdot) {   // C is stored as is; the side operand is multiplied with the ROUNDED outputs and summed
                  o.x = pack_bf16(f[0], f[1]);
                  o.y = pack_bf16(f[2], f[3]);
                  o.z = pack_bf16(f[4], f[5]);
                  o.w = pack_bf16(f[6], f[7]);
                  dacc += bf16_lo(o.x) * bf16_lo(r4[0]) + bf16_hi(o.x) * bf16_hi(r4[0]) + bf16_lo(o.y) * bf16_lo(r4[1]) +
                          bf16_hi(o.y) * bf16_hi(r4[1]) + bf16_lo(o.z) * bf16_lo(r4[2]) + bf16_hi(o.z) * bf16_hi(r4[2]) +
                          bf16_lo(o.w) * bf16_lo(r4[3]) + bf16_hi(o.w) * bf16_hi(r4[3]);
                } else {
                  o.x = pack_bf16(f[0] + bf16_lo(r4[0]), f[1] + bf16_hi(r4[0]));
                  o.y = pack_bf16(f[2] + bf16_lo(r4[1]), f[3] + bf16_hi(r4[1]));
                  o.z = pack_bf16(f[4] + bf16_lo(r4[2]), f[5] + bf16_hi(r4[2]));
                  o.w = pack_bf16(f[6] + bf16_lo(r4[3]), f[7] + bf16_hi(r4[3]));
                }
                stg_v4(dst + j8, o);
              }
            } else if (row_ok && col + j8 < p.N) {
              if (rsd != nullptr) {
                const uint4 r4 = *reinterpret_cast<const uint4*>(rsd + j8);
                f[0] += bf16_lo(r4.x); f[1] += bf16_hi(r4.x);
                f[2] += bf16_lo(r4.y); f[3] += bf16_hi(r4.y);
                f[4] += bf16_lo(r4.z); f[5] += bf16_hi(r4.z);
                f[6] += bf16_lo(r4.w); f[7] += bf16_hi(r4.w);
              }
              uint4 o;
              o.x = pack_bf16(f[0], f[1]);
              o.y = pack_bf16(f[2], f[3]);
              o.z = pack_bf16(f[4], f[5]);
              o.w = pack_bf16(f[6], f[7]);
              stg_v4(dst + j8, o);
            }
          }
        }
      }
      if constexpr (kRes) {
        // this thread's 128 columns (chunks 4 ch .. 4 ch + 3 of the tile) are one group: [batch][group][position]
        if (rowdot && row_ok && col0 + ch * 128 < p.N) {
          const int bb = row / p.dot_S;
          p.dot_out[((int64_t)bb * (p.N / 128) + (col0 / 128 + ch)) * p.dot_S + (row - bb * p.dot_S)] = dacc;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) {
        if constexpr (CG == 1) mbar_arrive(&tempty_bar[as]); else mbar_arrive_cluster(&tempty_bar[as], 0);
      }
    }
  }

  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) tmem_dealloc<CG>(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// Wave-alignment counters (see the producer of gemm_wide_kernel): one int per sync point, a slot of kSyncInts per launch
// out of a per-device ring (concurrent launches from other streams / threads get different slots), zeroed in stream
// order before the launch. Returns null when the launch has too many sync points or allocation fails.
static int* acquire_wave_sync(int points, cudaStream_t stream) {
  constexpr int kSyncInts = 128, kSyncSlots = 64, kMaxDev = 16;
  if (points > kSyncInts) return nullptr;
  static std::mutex mu;
  static int* ring[kMaxDev] = {nullptr};
  static std::atomic<unsigned> next_slot{0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= kMaxDev) return nullptr;
  {
    std::lock_guard<std::mutex> lk(mu);
    if (ring[dev] == nullptr && cudaMalloc(&ring[dev], (size_t)kSyncSlots * kSyncInts * sizeof(int)) != cudaSuccess) {
      ring[dev] = nullptr;
      (void)cudaGetLastError();
    }
  }
  if (ring[dev] == nullptr) return nullptr;
  int* slot = ring[dev] + (size_t)(next_slot.fetch_add(1) % kSyncSlots) * kSyncInts;
  if (cudaMemsetAsync(slot, 0, kSyncInts * sizeof(int), stream) != cudaSuccess) return nullptr;
  return slot;
}

template <bool kInt8, int CG, int kRank, bool kMN = false, bool kSwi = false, bool kRes = false, bool kRope = false>
static int launch_gemm_r(const void* A, int64_t lda, const void* B, int64_t ldb, const GemmParams& p,
                       cudaStream_t stream) {
  using S = GemmSmem<CG>;
  const int esz = kInt8 ? 1 : 2;
  const int elem_per_row = kBKBytes / esz;
  if (p.M <= 0 || p.N <= 0 || p.K <= 0) return set_error(LLAMAX_ERR_ARG, "gemm: empty problem");
  if ((lda * esz) % 16 || (ldb * esz) % 16 || (reinterpret_cast<uintptr_t>(A) % 16) ||
      (reinterpret_cast<uintptr_t>(B) % 16))
    return set_error(LLAMAX_ERR_ARG, "gemm: operand base / leading dimension must be 16-byte aligned");
  if (p.N % 8 || p.ldc % 8 || (reinterpret_cast<uintptr_t>(p.C) % 16))
    return set_error(LLAMAX_ERR_ARG, "gemm: N and ldc must be multiples of 8, C 16-byte aligned");
  if (p.resid && (p.ldr % 8 || reinterpret_cast<uintptr_t>(p.resid) % 16))
    return set_error(LLAMAX_ERR_ARG, "gemm: residual must be 16-byte aligned with ldr % 8 == 0");
  if (p.lora_rank < 0 || p.lora_rank > kMaxLoraRank || (p.lora_rank % 4))
    return set_error(LLAMAX_ERR_ARG, "gemm: lora rank must be a multiple of 4 in [0, 16]");
  if (p.seg_n0 != 0 && (p.seg_n0 % kBN || p.seg_n1 % kBN || p.seg_n0 <= 0 || p.seg_n1 <= p.seg_n0))
    return set_error(LLAMAX_ERR_ARG, "gemm: LoRA column segments must be increasing multiples of 256");

  CUtensorMap tmA, tmB;
  const CUtensorMapDataType dt = kInt8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  int rc;
  if constexpr (kMN) {   // A_t [K, M], B_t [K, N]: inner dimension = M / N, boxes [64 mn] x [64 k]
    static_assert(!kInt8, "MN-major operands: bf16 only");
    rc = make_tmap_2d(&tmA, dt, esz, A, p.M, p.K, lda, 64, 64);
    if (rc) return rc;
    rc = make_tmap_2d(&tmB, dt, esz, B, p.N, p.K, ldb, 64, 64);
    if (rc) return rc;
  } else {
    rc = make_tmap_2d(&tmA, dt, esz, A, p.K, p.M, lda, elem_per_row, kBM);
    if (rc) return rc;
    rc = make_tmap_2d(&tmB, dt, esz, B, p.K, p.N, ldb, elem_per_row, kBN / CG);
    if (rc) return rc;
  }

  auto kern = gemm_kernel<kInt8, CG, kRank, kMN, kSwi, kRes, 0, kRope>;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), S::kTotal, "gemm: cudaFuncSetAttribute"))) return rc;
  const int num_sms = sm_count();
  const int num_tiles = ((p.M + kBM * CG - 1) / (kBM * CG)) * ((p.N + kBN - 1) / kBN);
  int clusters = num_sms / CG;
  if (clusters > num_tiles) clusters = num_tiles;

  GemmParams pp = p;
  {
    const int num_m = (p.M + kBM * CG - 1) / (kBM * CG), num_n = (p.N + kBN - 1) / kBN;
    pp.group = num_m >= num_n ? -kGroupM : kGroupM;
    // Wave alignment every `sync_every` visits (see gemm_wide_kernel). Measured per kernel form, sustained, same box:
    // the w2 grad_input GEMM with the SwiGLU-backward epilogue — the form that moves the most
    // DRAM bytes per flop (5.8 GB per launch) — gains 2.5 % at any period 1..8 (1016-1026 -> 1044-1050 TFLOP/s); the
    // INT8 forward GEMM (2429-2437 -> 2291-2414 TOP/s) and the short-K bf16 GEMMs (1292-1295 -> 1270-1291) lose: their
    // operand panels fit the L2 whatever the drift, and the barrier only adds a wait. So: that one form, period 2.
    constexpr int kSyncEvery = 2;
    const int visits = (num_tiles + clusters - 1) / clusters;
    if (kSwi && visits > kSyncEvery) {
      pp.wave_sync = acquire_wave_sync(visits / kSyncEvery + 1, stream);
      pp.sync_every = kSyncEvery;
    }
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(clusters * CG);
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = S::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmA, pp);
  if (e != cudaSuccess) return set_cuda_error(e, "gemm: launch");
  return 0;
}

// Mixed-input launch (always CTA pairs). kMix == 1: B8 int8 [N, K] pitch ldb8. kMix == 2: B8 int8 [K1, N] pitch ldb8,
// tail bf16 [K - K1, N] pitch ldt (or null when K == K1).
template <int kMix, int kRank, bool kSwi = false>
static int launch_gemm_mix(const void* A, int64_t lda, const void* B8, int64_t ldb8, const void* tail, int64_t ldt,
                           const GemmParams& p, cudaStream_t stream) {
  using S = GemmSmem<2, kMix>;
  if (p.M <= 0 || p.N <= 0 || p.K <= 0) return set_error(LLAMAX_ERR_ARG, "gemm: empty problem");
  if ((lda * 2) % 16 || ldb8 % 16 || (reinterpret_cast<uintptr_t>(A) % 16) || (reinterpret_cast<uintptr_t>(B8) % 16))
    return set_error(LLAMAX_ERR_ARG, "mixed gemm: operand base / leading dimension must be 16-byte aligned");
  if (!kSwi && (p.N % 8 || p.ldc % 8 || (reinterpret_cast<uintptr_t>(p.C) % 16)))
    return set_error(LLAMAX_ERR_ARG, "gemm: N and ldc must be multiples of 8, C 16-byte aligned");
  if (p.resid && (p.ldr % 8 || reinterpret_cast<uintptr_t>(p.resid) % 16))
    return set_error(LLAMAX_ERR_ARG, "gemm: residual must be 16-byte aligned with ldr % 8 == 0");
  if (p.lora_rank < 0 || p.lora_rank > kMaxLoraRank || (p.lora_rank % 4))
    return set_error(LLAMAX_ERR_ARG, "gemm: lora rank must be a multiple of 4 in [0, 16]");
  if constexpr (kMix == 2) {   // argument checks before any driver call
    if (p.K1 <= 0 || p.K1 % 64 || p.K1 > p.K || p.K - p.K1 > 64 || !p.k_scale)
      return set_error(LLAMAX_ERR_ARG, "mixed gemm: K1 must be a positive multiple of 64, the tail at most 64 rows");
    if ((p.K > p.K1) != (tail != nullptr))
      return set_error(LLAMAX_ERR_ARG, "mixed gemm: tail tensor and K - K1 disagree");
    if (tail != nullptr && ((ldt * 2) % 16 || reinterpret_cast<uintptr_t>(tail) % 16))
      return set_error(LLAMAX_ERR_ARG, "mixed gemm: tail must be 16-byte aligned with a pitch multiple of 8");
  }
  CUtensorMap tmA, tmB, tmT;
  int rc = make_tmap_2d(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, A, p.K, p.M, lda, 64, kBM);
  if (rc) return rc;
  if constexpr (kMix == 1) {
    rc = make_tmap_2d(&tmB, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, B8, p.K, p.N, ldb8, 64, kBN / 2, false);
    if (rc) return rc;
    tmT = tmA;
  } else {
    rc = make_tmap_2d(&tmB, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, B8, p.N, p.K1, ldb8, kBN / 2, 64, false);
    if (rc) return rc;
    if (tail != nullptr) {
      rc = make_tmap_2d(&tmT, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, tail, p.N, p.K - p.K1, ldt, 64, 64);
      if (rc) return rc;
    } else {
      tmT = tmA;
    }
  }
  auto kern = gemm_kernel<false, 2, kRank, false, kSwi, false, kMix>;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), S::kTotal, "mixed gemm: cudaFuncSetAttribute"))) return rc;
  const int num_m = (p.M + 2 * kBM - 1) / (2 * kBM), num_n = (p.N + kBN - 1) / kBN;
  const int clusters = std::min(sm_count() / 2, num_m * num_n);
  GemmParams pp = p;
  pp.group = num_m >= num_n ? -kGroupM : kGroupM;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(clusters * 2);
  cfg.blockDim = dim3(kMixThreads);
  cfg.dynamicSmemBytes = S::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmT, pp);
  if (e != cudaSuccess) return set_cuda_error(e, "mixed gemm: launch");
  return 0;
}

template <bool kInt8, int CG>
static int launch_gemm(const void* A, int64_t lda, const void* B, int64_t ldb, const GemmParams& p,
                       cudaStream_t stream) {
  if constexpr (kInt8 && CG == 2) {
    // q | k | v projection with RoPE in the epilogue (opt-in): the side-input pipeline of the residual variant reads the
    // (cos, sin) table instead; no residual in this form
    if (p.rope != nullptr) {
      if (p.resid != nullptr || (p.flags & 1) || p.rope_S <= 0 || p.rope_cols <= 0 || p.rope_cols % kBN ||
          p.rope_cols > p.N || reinterpret_cast<uintptr_t>(p.rope) % 32)
        return set_error(LLAMAX_ERR_ARG, "gemm: RoPE epilogue needs no residual, rope_S > 0, rope_cols a multiple of 256 "
                                         "within N and a 32-byte aligned table");
      if (p.lora_rank <= 0) return launch_gemm_r<kInt8, CG, 0, false, false, true, true>(A, lda, B, ldb, p, stream);
      if (p.lora_rank <= 8) return launch_gemm_r<kInt8, CG, 8, false, false, true, true>(A, lda, B, ldb, p, stream);
      return set_error(LLAMAX_ERR_ARG, "gemm: RoPE epilogue supports LoRA rank 0 or 8");
    }
  }
  if (p.rope != nullptr) return set_error(LLAMAX_ERR_ARG, "gemm: RoPE epilogue exists for the INT8 GEMM with CTA pairs only");
  if constexpr (kInt8) {
    // forward projections with the residual connection (wo, w2): pipelined residual reads; needs resid != C and a
    // 16-byte aligned residual (rows start on 16-byte boundaries when ldr % 8 == 0)
    if (p.resid != nullptr && (p.flags & 1) == 0 && static_cast<const void*>(p.resid) != p.C &&
        reinterpret_cast<uintptr_t>(p.resid) % 16 == 0 && p.ldr % 8 == 0) {
      if (p.lora_rank <= 0) return launch_gemm_r<kInt8, CG, 0, false, false, true>(A, lda, B, ldb, p, stream);
      if (p.lora_rank <= 8) return launch_gemm_r<kInt8, CG, 8, false, false, true>(A, lda, B, ldb, p, stream);
      return launch_gemm_r<kInt8, CG, 16, false, false, true>(A, lda, B, ldb, p, stream);
    }
  }
  if (p.lora_rank <= 0) return launch_gemm_r<kInt8, CG, 0>(A, lda, B, ldb, p, stream);
  if (p.lora_rank <= 8) return launch_gemm_r<kInt8, CG, 8>(A, lda, B, ldb, p, stream);
  return launch_gemm_r<kInt8, CG, 16>(A, lda, B, ldb, p, stream);
}

// ------------------------------------------------------------------------------------------------
// Wide bf16 GEMM for long contractions: C[M,N] = A[M,K] * B[N,K]^T, plain bf16 store, CTA pairs, 512 x 256 output per
// visit (two 256 x 256 cta_group::2 accumulators that share the B tile).
//
// Why a second tile shape. The w1|w3 grad_input GEMM [16384, 4096, K = 28688] is the largest kernel of the step. Measured
// against cuBLAS on the same box (tools/gemm_vs_cublas.py, profiles/r2_gemm_vs_cublas.txt; `ncu --set full`): the 256 x 256
// kernel above keeps the tensor pipe as busy per cycle as cuBLAS' nvjet 256x256 2-CTA kernel (96 % vs 95 %), but at the
// 1 kW cap it runs at 1.22 GHz against 1.40 GHz — it spends its power budget on data movement: 7.8 GB of DRAM reads per
// launch against 3.4 GB (1.3 GB algorithmic) and 30.1 GB against 22.6 GB from L2 into the SMs. Both follow from the tile:
// a CTA pair that owns 512 x 256 outputs per visit loads 48 KB per CTA and k-block for twice the MMA work of 32 KB, and a
// wave of 74 pairs touches ~17 x 512-row / 256-column operand panels instead of ~17 x 256 / 256.
// Price: both TMEM accumulator buffers belong to one visit, so the epilogue of a visit is only half hidden (the first
// k-block's MMAs into accumulator 0 run while accumulator 1 is still being drained). Used only where the main loop of a
// visit is >= 128 k-blocks (K >= 8192): there the exposed part is < 2 %.
// ------------------------------------------------------------------------------------------------
namespace wd {
constexpr int kStages = 4;
constexpr int kABytes = 256 * 128;   // [256 rows] x [64 bf16]: rows 0..127 feed accumulator 0, rows 128..255 accumulator 1
constexpr int kBBytes = 128 * 128;   // this CTA's half of the [256 x 64] B tile
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kSmem = kStages * kStageBytes + (2 * kStages + 4) * 8 + 16 + 1024;
}  // namespace wd

__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_wide_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 __nv_bfloat16* __restrict__ C, int64_t ldc, int M, int N, int K, int group, int* wave_sync) {
  using namespace wd;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kStages;
  uint64_t* tfull_bar = bars + 2 * kStages;
  uint64_t* tempty_bar = bars + 2 * kStages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const uint32_t cta_rank = cluster_ctarank();
  const bool is_leader = cta_rank == 0;
  const int num_m = (M + 511) / 512;
  const int num_n = (N + kBN - 1) / kBN;
  const int num_tiles = num_m * num_n;
  const int num_kb = (K + 63) / 64;
  const int cluster_id = blockIdx.x / 2;
  const int num_clusters = gridDim.x / 2;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && elect_one()) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 16);  // one arrive per epilogue warp of both CTAs
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<2>(tmem_slot, 512);
    tmem_relinquish<2>();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t full_addr = mapa_u32(smem_u32(&full_bar[0]), 0);
      int visit_p = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++visit_p) {
        int tm, tn;
        tile_coords(tile, num_m, num_n, group, tm, tn);
        const int row_a = tm * 512 + cta_rank * 256;
        const int row_b = tn * kBN + cta_rank * 128;
        if (wave_sync != nullptr && visit_p > 0) {
          // Wave alignment. The CTA pairs of a wave share operand panels (one 512-row A panel is read by ~8 pairs, one B
          // panel by ~9) and with K = 28688 a wave's live panels are 2-3 x the L2, so the sharing only works while the pairs
          // walk K in step — and nothing re-aligned them between visits: after the first visit they drift apart and
          // every pair fetches its panels from DRAM on its own (ncu: 7.1 GB per launch, L2 hit 61 %). Every producer
          // checks in at the start of a visit and waits for the other producers of that visit: 3.0 GB, L2 hit 77 %,
          // 2.62 -> 2.41 ms under ncu, 1327-1341 -> 1377-1379 TFLOP/s sustained at the 1 kW cap (less DRAM traffic =
          // higher clocks), same box. All pairs are co-resident (persistent grid, one CTA per SM); the wait is bounded
          // all the same, so that a device shared with another stream's kernel can only lose the alignment, not hang.
          const int expected = 2 * min(num_clusters, num_tiles - visit_p * num_clusters);
          atomicAdd(&wave_sync[visit_p], 1);
          int seen;
          uint32_t polls = 0;
          do {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(wave_sync + visit_p) : "memory");
          } while (seen < expected && ++polls < (1u << 14));
        }
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * kStageBytes;
          if (is_leader) mbar_expect_tx(&full_bar[stage], kStageBytes * 2);
          const uint32_t bar_addr = full_addr + stage * 8;
          tma_load_2d_cg2(sa, &tmA, bar_addr, kb * 64, row_a);
          tma_load_2d_cg2(sa + kABytes, &tmB, bar_addr, kb * 64, row_b);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (is_leader && elect_one()) {
      constexpr uint32_t idesc = make_idesc(1, 1, 256, kBN);
      constexpr uint32_t kHi = desc_hi(1024);
      int stage = 0;
      uint32_t phase = 0;
      int visit = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++visit) {
        const uint32_t aphase = visit & 1;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          if (kb == 0) mbar_wait(&tempty_bar[0], aphase ^ 1);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * kStageBytes);
          const uint32_t la0 = desc_lo(sa, 16), la1 = desc_lo(sa + 128 * 128, 16), lb = desc_lo(sa + kABytes, 16);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_ss<false, 2>(tmem_base, desc_join(la0 + 2 * k, kHi), desc_join(lb + 2 * k, kHi), idesc, (kb | k) != 0);
          if (kb == 0) {   // accumulator 1 may still be draining: its first MMAs go behind accumulator 0's
            mbar_wait(&tempty_bar[1], aphase ^ 1);
            tc_fence_after();
          }
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_ss<false, 2>(tmem_base + kBN, desc_join(la1 + 2 * k, kHi), desc_join(lb + 2 * k, kHi), idesc, (kb | k) != 0);
          umma_commit_cg2(&empty_bar[stage], 3);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_cg2(&tfull_bar[0], 3);
        umma_commit_cg2(&tfull_bar[1], 3);
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ================================ epilogue ================================
    const int ew = warp & 3;                 // TMEM lanes [32*ew, 32*ew+32)
    const int ch = (warp - 4) >> 2;          // column half of the accumulator handled by this warp
    int visit = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++visit) {
      int tm, tn;
      tile_coords(tile, num_m, num_n, group, tm, tn);
      const int col0 = tn * kBN;
      const int n_chunks = min(ch * 4 + 4, min(kBN / 32, (N - col0 + 31) / 32));
#pragma unroll 1
      for (int a = 0; a < 2; ++a) {
        const int row = tm * 512 + cta_rank * 256 + a * 128 + ew * 32 + lane_id();
        const bool row_ok = row < M;
        mbar_wait(&tfull_bar[a], visit & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t(ew * 32) << 16) + a * kBN;
        uint32_t v[2][32];
        if (ch * 4 < n_chunks) tmem_ld_32x32(taddr + ch * 4 * 32, v[0]);
#pragma unroll 1
        for (int c = ch * 4; c < n_chunks; c += 2) {
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int cc = c + half;
            if (cc >= n_chunks) break;
            uint32_t(&vv)[32] = v[half];
            tmem_wait_ld_regs(vv);
            if (cc + 1 < n_chunks) tmem_ld_32x32(taddr + (cc + 1) * 32, v[half ^ 1]);
            const int col = col0 + cc * 32;
            if (row_ok) {
              __nv_bfloat16* dst = C + (int64_t)row * ldc + col;
#pragma unroll
              for (int j8 = 0; j8 < 32; j8 += 8) {
                if (col + j8 < N) {
                  uint4 o;
                  o.x = pack_bf16(__uint_as_float(vv[j8 + 0]), __uint_as_float(vv[j8 + 1]));
                  o.y = pack_bf16(__uint_as_float(vv[j8 + 2]), __uint_as_float(vv[j8 + 3]));
                  o.z = pack_bf16(__uint_as_float(vv[j8 + 4]), __uint_as_float(vv[j8 + 5]));
                  o.w = pack_bf16(__uint_as_float(vv[j8 + 6]), __uint_as_float(vv[j8 + 7]));
                  stg_v4(dst + j8, o);
                }
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane_id() == 0) mbar_arrive_cluster(&tempty_bar[a], 0);
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc<2>(tmem_base, 512);
}

static int launch_gemm_wide(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int M, int N,
                            int K, cudaStream_t stream) {
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, A, K, M, lda, 64, 256);
  if (rc) return rc;
  rc = make_tmap_2d(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, B, K, N, ldb, 64, 128);
  if (rc) return rc;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(gemm_wide_kernel), wd::kSmem, "wide gemm: cudaFuncSetAttribute")))
    return rc;
  const int num_m = (M + 511) / 512, num_n = (N + kBN - 1) / kBN;
  int clusters = std::min(sm_count() / 2, num_m * num_n);
  const int group = num_m >= num_n ? -kGroupM : kGroupM;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(clusters * 2);
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = wd::kSmem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const int visits = (num_m * num_n + clusters - 1) / clusters;
  int* wave_sync = visits > 1 ? acquire_wave_sync(visits, stream) : nullptr;
  cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_wide_kernel, tmA, tmB, (__nv_bfloat16*)C, ldc, M, N, K, group, wave_sync);
  if (e != cudaSuccess) return set_cuda_error(e, "wide gemm: launch");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// LoRA weight gradient on tensor cores:  out[p, r] += alpha * sum_m X[m, p] * H[m, r]
//   = GEMM with M' = P (128 per CTA), N' = 32 (rank zero-padded), K' = tokens.
// A' = X^T is read straight from X [tokens, P] as an MN-major operand (64-column boxes, like V in attention),
// B' = H^T [R, tokens] K-major.  grid = (P / 128, splits over tokens); fp32 red.add of the few outputs.
// ------------------------------------------------------------------------------------------------
namespace wg {
constexpr int kStages = 8;
constexpr int kABytes = 128 * 64 * 2;  // [64 tokens] x [128 P-columns] bf16 = two boxes of [64 x 128 B]
constexpr int kBBytes = 32 * 64 * 2;   // [32 rank rows] x [64 tokens]
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kSmem = kStages * kStageBytes + (2 * kStages + 1) * 8 + 16 + 1024;
}  // namespace wg

// kPartials (deterministic mode): split s stores its partial with plain stores into out[s, P, R]; the splits are then
// summed in split order by reduce_partials_kernel instead of with order-dependent fp32 atomics.
template <bool kPartials = false>
__global__ void __launch_bounds__(192, 1)
lora_wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmHt,
                     float* __restrict__ out, int P, int R, int M, int k_per_split, float alpha) {
  using namespace wg;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* done_bar = empty_bar + kStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);
  const int warp = threadIdx.x >> 5;
  const int p0 = blockIdx.x * 128;
  const int k_begin = blockIdx.y * k_per_split;
  const int k_end = min(M, k_begin + k_per_split);
  const int num_kb = (k_end - k_begin + 63) / 64;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmHt);
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(done_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, 32);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * kStageBytes;
        mbar_expect_tx(&full_bar[stage], kStageBytes);
        const int k0 = k_begin + kb * 64;
        tma_load_2d(sa, &tmX, &full_bar[stage], p0, k0);
        tma_load_2d(sa + kABytes / 2, &tmX, &full_bar[stage], p0 + 64, k0);
        tma_load_2d(sa + kABytes, &tmHt, &full_bar[stage], k0, 0);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc(1, 1, 128, 32, 1, 0);  // A MN-major, B K-major
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + stage * kStageBytes);
        const uint32_t sb = sa + kABytes;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const uint64_t ad = make_smem_desc_sw128(sa + ks * 16 * 128, 8192, 1024);
          const uint64_t bd = make_smem_desc_sw128(sb + ks * 32, 16, 1024);
          umma_ss<false, 1>(tmem_base, ad, bd, idesc, (kb | ks) != 0);
        }
        umma_commit(&empty_bar[stage]);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      umma_commit(done_bar);
    }
    __syncwarp();
  } else {
    // epilogue warps 2..5: TMEM lanes 32*(warp % 4)
    const int lq = warp & 3;
    const int row = p0 + lq * 32 + lane_id();
    if constexpr (kPartials) {
      uint32_t v[32] = {};
      if (num_kb > 0) {
        mbar_wait(done_bar, 0);
        tc_fence_after();
        tmem_ld_32x32(tmem_base + (uint32_t(lq * 32) << 16), v);
        tmem_wait_ld_regs(v);
      }
      if (row < P) {
        float* dst = out + ((int64_t)blockIdx.y * P + row) * R;
#pragma unroll
        for (int r = 0; r < 32; ++r)
          if (r < R) dst[r] = alpha * __uint_as_float(v[r]);
      }
    } else if (num_kb > 0) {
      mbar_wait(done_bar, 0);
      tc_fence_after();
      uint32_t v[32];
      tmem_ld_32x32(tmem_base + (uint32_t(lq * 32) << 16), v);
      tmem_wait_ld_regs(v);
      if (row < P) {
#pragma unroll
        for (int r = 0; r < 32; ++r)
          if (r < R) atomicAdd(out + (int64_t)row * R + r, alpha * __uint_as_float(v[r]));
      }
    }
    tc_fence_before();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<1>(tmem_base, 32);
}

// ------------------------------------------------------------------------------------------------
// Skinny GEMM for the LoRA projections: C[M, N<=32] = A[M,K] * B[N,K]^T (bf16, fp32 accumulate).
// HBM-bound on A: one CTA per 128 rows streams its rows once through an 8-stage TMA ring; UMMA 128 x 32 x 16
// (the persistent 256-wide kernel would spend 8x the tensor time on zero columns).
// ------------------------------------------------------------------------------------------------
namespace sk {
constexpr int kStages = 8;
constexpr int kABytes = 128 * 128;     // [128 rows] x [64 bf16]
constexpr int kBBytes = 32 * 128;      // [32 rows]  x [64 bf16]
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kSmem = kStages * kStageBytes + (2 * kStages + 1) * 8 + 16 + 1024;
}  // namespace sk

__global__ void __launch_bounds__(192, 1)
skinny_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   __nv_bfloat16* __restrict__ C, int64_t ldc, int M, int N, int K) {
  using namespace sk;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* done_bar = empty_bar + kStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);
  const int warp = threadIdx.x >> 5;
  const int m0 = blockIdx.x * 128;
  const int num_kb = (K + 63) / 64;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(done_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, 32);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * kStageBytes;
        mbar_expect_tx(&full_bar[stage], kStageBytes);
        tma_load_2d(sa, &tmA, &full_bar[stage], kb * 64, m0);
        tma_load_2d(sa + kABytes, &tmB, &full_bar[stage], kb * 64, 0);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc(1, 1, 128, 32, 0, 0);
      constexpr uint32_t kHi = desc_hi(1024);
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t la = desc_lo(smem_u32(smem + stage * kStageBytes), 16);
        const uint32_t lb = desc_lo(smem_u32(smem + stage * kStageBytes + kABytes), 16);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          umma_ss<false, 1>(tmem_base, desc_join(la + ks * 2, kHi), desc_join(lb + ks * 2, kHi), idesc, (kb | ks) != 0);
        umma_commit(&empty_bar[stage]);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      umma_commit(done_bar);
    }
    __syncwarp();
  } else {
    const int lq = warp & 3;  // warps 2..5 cover the four TMEM lane quarters
    const int row = m0 + lq * 32 + lane_id();
    mbar_wait(done_bar, 0);
    tc_fence_after();
    uint32_t v[32];
    tmem_ld_32x32(tmem_base + (uint32_t(lq * 32) << 16), v);
    tmem_wait_ld_regs(v);
    if (row < M) {
      __nv_bfloat16* dst = C + (int64_t)row * ldc;
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        if (j < N) {
          uint4 o;
          o.x = pack_bf16(__uint_as_float(v[j + 0]), __uint_as_float(v[j + 1]));
          o.y = pack_bf16(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
          o.z = pack_bf16(__uint_as_float(v[j + 4]), __uint_as_float(v[j + 5]));
          o.w = pack_bf16(__uint_as_float(v[j + 6]), __uint_as_float(v[j + 7]));
          stg_v4(dst + j, o);
        }
      }
    }
    tc_fence_before();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<1>(tmem_base, 32);
}

static int launch_skinny(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int M, int N,
                         int K, cudaStream_t stream) {
  if ((lda * 2) % 16 || (ldb * 2) % 16 || (reinterpret_cast<uintptr_t>(A) % 16) || (reinterpret_cast<uintptr_t>(B) % 16))
    return set_error(LLAMAX_ERR_ARG, "gemm: operand base / leading dimension must be 16-byte aligned");
  if (N % 8 || ldc % 8 || (reinterpret_cast<uintptr_t>(C) % 16))
    return set_error(LLAMAX_ERR_ARG, "gemm: N and ldc must be multiples of 8, C 16-byte aligned");
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, A, K, M, lda, 64, 128);
  if (rc) return rc;
  rc = make_tmap_2d(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, B, K, N, ldb, 64, 32);
  if (rc) return rc;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(skinny_gemm_kernel), sk::kSmem, "skinny gemm: cudaFuncSetAttribute")))
    return rc;
  skinny_gemm_kernel<<<(M + 127) / 128, 192, sk::kSmem, stream>>>(tmA, tmB, (__nv_bfloat16*)C, ldc, M, N, K);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error(e, "skinny gemm: launch");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Fused LoRA backward pair for one linear: ONE pass over dY [tokens, N] yields both
//   dh [tokens, R] = dY . Bt^T          (Bt = scale * B^T, [R, N];  contraction over N)
//   dB [N, R]     += alpha * dY^T . h   (Ht = h^T, [R, tokens];     contraction over tokens)
// dY is the big operand (0.94 GB for the w1|w3 group at 16 k tokens); read separately by the skinny dh GEMM and by
// lora_wgrad it was streamed from HBM twice. Here a CTA owns 128 tokens x a range of N and streams [128 x 128] tiles:
// the tile is the K-major A operand of the dh MMA and, viewed MN-major, the A operand of the dB MMA (M = 128 columns
// of N, K = the 128 tokens). dh accumulates in TMEM over the whole range; each tile's dB block [128 x R] is drained
// from a double-buffered TMEM accumulator and reduced into dB with fp32 red.add. grid = (token blocks, N splits).
// ------------------------------------------------------------------------------------------------
namespace lp {
constexpr int kStages = 5;
constexpr int kABytes = 128 * 128 * 2;   // [128 tokens] x [128 columns] bf16 = two boxes of [128 x 128 B]
constexpr int kBBytes = 32 * 128 * 2;    // [32 rank rows] x [128 columns]   = two boxes of [32 x 128 B]
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kHtBytes = 32 * 128 * 2;   // [32 rank rows] x [128 tokens]
constexpr int kOffHt = kStages * kStageBytes;
constexpr int kOffBar = kOffHt + kHtBytes;
constexpr int kNumBars = 2 * kStages + 1 + 4 + 1;   // full/empty ring, ht_full, d2 full/empty[2], d1_done
constexpr int kSmem = kOffBar + kNumBars * 8 + 16 + 1024;
}  // namespace lp

__global__ void __launch_bounds__(192, 1)
lora_bwd_pair_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmBt,
                     const __grid_constant__ CUtensorMap tmHt, __nv_bfloat16* __restrict__ dh, int64_t lddh,
                     __nv_bfloat16* __restrict__ dht, int64_t lddht, float* __restrict__ dh_accum,
                     float* __restrict__ dB, int M, int N, int R, int chunks_per_split, float alpha) {
  using namespace lp;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* ht_full = empty_bar + kStages;
  uint64_t* d2_full = ht_full + 1;
  uint64_t* d2_empty = d2_full + 2;
  uint64_t* d1_done = d2_empty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d1_done + 1);
  const int warp = threadIdx.x >> 5;
  const int m0 = blockIdx.x * 128;
  const int total_chunks = (N + 127) / 128;
  const int c_begin = blockIdx.y * chunks_per_split;
  const int num_c = min(chunks_per_split, total_chunks - c_begin);

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmY);
    tma_prefetch_desc(&tmBt);
    tma_prefetch_desc(&tmHt);
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(ht_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&d2_full[i], 1);
      mbar_init(&d2_empty[i], 4);
    }
    mbar_init(d1_done, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, 128);   // dh: columns 0..31; dB blocks: 32..63 and 64..95
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(ht_full, kHtBytes);
      tma_load_2d(smem + kOffHt, &tmHt, ht_full, m0, 0);
      tma_load_2d(smem + kOffHt + kHtBytes / 2, &tmHt, ht_full, m0 + 64, 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int c = 0; c < num_c; ++c) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * kStageBytes;
        mbar_expect_tx(&full_bar[stage], kStageBytes);
        const int n0 = (c_begin + c) * 128;
        tma_load_2d(sa, &tmY, &full_bar[stage], n0, m0);
        tma_load_2d(sa + kABytes / 2, &tmY, &full_bar[stage], n0 + 64, m0);
        tma_load_2d(sa + kABytes, &tmBt, &full_bar[stage], n0, 0);
        tma_load_2d(sa + kABytes + kBBytes / 2, &tmBt, &full_bar[stage], n0 + 64, 0);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_dh = make_idesc(1, 1, 128, 32, 0, 0);  // [tokens x n] . [r x n]^T
      constexpr uint32_t idesc_db = make_idesc(1, 1, 128, 32, 1, 0);  // [tokens x n]^T (MN-major) . [r x tokens]^T
      constexpr uint32_t kHi = desc_hi(1024);
      const uint32_t loHt = desc_lo(smem_u32(smem + kOffHt), 16);
      mbar_wait(ht_full, 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int c = 0; c < num_c; ++c) {
        const int b = c & 1;
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + stage * kStageBytes);
        const uint32_t la = desc_lo(sa, 16), lamn = desc_lo(sa, 16384), lb = desc_lo(sa + kABytes, 16);
#pragma unroll
        for (int bx = 0; bx < 2; ++bx)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_ss<false, 1>(tmem_base, desc_join(la + (bx * 16384 + ks * 32) / 16, kHi),
                              desc_join(lb + (bx * 4096 + ks * 32) / 16, kHi), idesc_dh, (c | bx | ks) != 0);
        mbar_wait(&d2_empty[b], ((c >> 1) & 1) ^ 1);
        tc_fence_after();
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)   // 16 tokens per step
          umma_ss<false, 1>(tmem_base + 32 + b * 32, desc_join(lamn + ks * 128, kHi),
                            desc_join(loHt + ((ks >> 2) * 4096 + (ks & 3) * 32) / 16, kHi), idesc_db, ks != 0);
        umma_commit(&d2_full[b]);
        umma_commit(&empty_bar[stage]);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      umma_commit(d1_done);
    }
    __syncwarp();
  } else {
    // epilogue warps 2..5: TMEM lanes 32 * (warp % 4)
    const int lq = warp & 3;
    const int lrow = lq * 32 + lane_id();
    const uint32_t lane_off = uint32_t(lq * 32) << 16;
    for (int c = 0; c < num_c; ++c) {
      const int b = c & 1;
      mbar_wait(&d2_full[b], (c >> 1) & 1);
      tc_fence_after();
      uint32_t v[32];
      tmem_ld_32x32(tmem_base + 32 + b * 32 + lane_off, v);
      tmem_wait_ld_regs(v);
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(&d2_empty[b]);
      const int n = (c_begin + c) * 128 + lrow;
      if (n < N) {
        float* dst = dB + (int64_t)n * R;   // R is a multiple of 8: rows are 32-byte aligned
#pragma unroll
        for (int r = 0; r < 32; r += 4)
          if (r < R)
            red_add_v4_f32(dst + r, alpha * __uint_as_float(v[r]), alpha * __uint_as_float(v[r + 1]),
                           alpha * __uint_as_float(v[r + 2]), alpha * __uint_as_float(v[r + 3]));
      }
    }
    if (num_c > 0) {
      mbar_wait(d1_done, 0);
      tc_fence_after();
      uint32_t v[32];
      tmem_ld_32x32(tmem_base + lane_off, v);
      tmem_wait_ld_regs(v);
      const int row = m0 + lrow;
      if (row < M) {
        if (dh_accum != nullptr) {   // N is split across CTAs: fp32 partial sums, converted by lora_dh_convert_kernel
#pragma unroll
          for (int r = 0; r < 32; r += 4)
            if (r < R)
              red_add_v4_f32(dh_accum + (int64_t)row * R + r, __uint_as_float(v[r]), __uint_as_float(v[r + 1]),
                             __uint_as_float(v[r + 2]), __uint_as_float(v[r + 3]));
        } else {
          __nv_bfloat16* dst = dh + (int64_t)row * lddh;
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            if (j < R) {
              uint4 o;
              o.x = pack_bf16(__uint_as_float(v[j + 0]), __uint_as_float(v[j + 1]));
              o.y = pack_bf16(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
              o.z = pack_bf16(__uint_as_float(v[j + 4]), __uint_as_float(v[j + 5]));
              o.w = pack_bf16(__uint_as_float(v[j + 6]), __uint_as_float(v[j + 7]));
              stg_v4(dst + j, o);
            }
          }
          if (dht != nullptr) {   // dh^T [R, M]: the operand of the dA weight gradient; 64 contiguous bytes per warp and r
#pragma unroll
            for (int r = 0; r < 32; ++r)
              if (r < R) dht[(int64_t)r * lddht + row] = __float2bfloat16_rn(__uint_as_float(v[r]));
          }
        }
      }
    }
    tc_fence_before();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<1>(tmem_base, 128);
}

// fp32 [M, R] partial sums -> bf16 dh rows (pitch lddh) and, optionally, dh^T [R, M]; one thread per 8 values
__global__ void lora_dh_convert_kernel(const float* __restrict__ acc, __nv_bfloat16* __restrict__ dh, int64_t lddh,
                                       __nv_bfloat16* __restrict__ dht, int64_t lddht, int64_t M, int R) {
  const int per_row = R / 8;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * per_row) return;
  const int64_t row = i / per_row;
  const int j = (int)(i - row * per_row) * 8;
  const float4 a = *reinterpret_cast<const float4*>(acc + row * R + j);
  const float4 b = *reinterpret_cast<const float4*>(acc + row * R + j + 4);
  uint4 o;
  o.x = pack_bf16(a.x, a.y);
  o.y = pack_bf16(a.z, a.w);
  o.z = pack_bf16(b.x, b.y);
  o.w = pack_bf16(b.z, b.w);
  stg_v4(dh + row * lddh + j, o);
  if (dht != nullptr) {
    const float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) dht[(int64_t)(j + k) * lddht + row] = __float2bfloat16_rn(f[k]);
  }
}

static std::atomic<int> g_gemm_cg{2};  // CTA-group size used by the GEMMs (1 or 2); see llamax_set_gemm_cta_group

}  // namespace lx

using namespace lx;

extern "C" {

#ifdef LX_MIX_TRACE
int llamax_debug_mix_trace(long long* host_out) {
  return cudaMemcpyFromSymbol(host_out, g_mix_trace, sizeof(long long) * 2 * 64 * 8) == cudaSuccess ? 0 : -2;
}
#endif

int llamax_set_gemm_cta_group(int cg) {
  if (cg != 1 && cg != 2) return set_error(LLAMAX_ERR_ARG, "cta group must be 1 or 2");
  g_gemm_cg = cg;
  return 0;
}

static void fill_epilogue(GemmParams& p, const llamax_epilogue_t* epi) {
  if (epi == nullptr) return;
  p.lora_h = static_cast<const __nv_bfloat16*>(epi->lora_h);
  p.ldh = epi->ldh;
  p.lora_b = static_cast<const __nv_bfloat16*>(epi->lora_b);
  p.lora_rank = epi->lora_h ? epi->lora_rank : 0;
  p.lora_scale = epi->lora_scale;
  p.resid = static_cast<const __nv_bfloat16*>(epi->resid);
  p.ldr = epi->ldr;
  p.seg_n0 = epi->lora_h ? epi->seg_n0 : 0;
  p.seg_n1 = epi->lora_h ? epi->seg_n1 : 0;
  p.rope = static_cast<const float*>(epi->rope);
  p.rope_S = epi->rope_S;
  p.rope_cols = epi->rope_cols;
}

int llamax_int8_gemm_dequant(const void* A, int64_t lda, const void* B, int64_t ldb, const void* a_scale,
                             const void* b_scale, void* C, int64_t ldc, int64_t M, int64_t N, int64_t K,
                             const llamax_epilogue_t* epi, void* stream) {
  if (!A || !B || !C || !a_scale || !b_scale) return set_error(LLAMAX_ERR_ARG, "int8_gemm_dequant: null pointer");
  GemmParams p{};
  p.M = (int)M; p.N = (int)N; p.K = (int)K;
  p.C = C; p.ldc = ldc;
  p.row_scale = static_cast<const __nv_bfloat16*>(a_scale);
  p.col_scale = static_cast<const __nv_bfloat16*>(b_scale);
  fill_epilogue(p, epi);
  return g_gemm_cg == 2 ? launch_gemm<true, 2>(A, lda, B, ldb, p, (cudaStream_t)stream)
                        : launch_gemm<true, 1>(A, lda, B, ldb, p, (cudaStream_t)stream);
}

int llamax_int8_gemm_s32(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t M,
                         int64_t N, int64_t K, void* stream) {
  if (!A || !B || !C) return set_error(LLAMAX_ERR_ARG, "int8_gemm_s32: null pointer");
  GemmParams p{};
  p.M = (int)M; p.N = (int)N; p.K = (int)K;
  p.C = C; p.ldc = ldc;
  p.flags = 1;
  return g_gemm_cg == 2 ? launch_gemm<true, 2>(A, lda, B, ldb, p, (cudaStream_t)stream)
                        : launch_gemm<true, 1>(A, lda, B, ldb, p, (cudaStream_t)stream);
}

int llamax_bf16_gemm(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t M,
                     int64_t N, int64_t K, const void* col_scale, int round_before_scale,
                     const llamax_epilogue_t* epi, void* stream) {
  if (!A || !B || !C) return set_error(LLAMAX_ERR_ARG, "bf16_gemm: null pointer");
  if (M <= 0 || N <= 0 || K <= 0) return set_error(LLAMAX_ERR_ARG, "gemm: empty problem");
  const bool plain = col_scale == nullptr && (epi == nullptr || (epi->lora_h == nullptr && epi->resid == nullptr));
  if (plain && N <= 32)  // LoRA down / dh projections: HBM-bound skinny kernel
    return launch_skinny(A, lda, B, ldb, C, ldc, (int)M, (int)N, (int)K, (cudaStream_t)stream);
  // long contractions without an epilogue (w1|w3 grad_input, LM-head grad_input): 512 x 256 outputs per CTA-pair visit;
  // LLAMAX_GEMM_WIDE=0 keeps them on the 256 x 256 kernel
  static const bool no_wide = getenv("LLAMAX_GEMM_WIDE") != nullptr && getenv("LLAMAX_GEMM_WIDE")[0] == '0';
  // Very wide outputs with a short contraction (the LM-head logits GEMM [8192, 128256, 4096]) stay on the 256 x 256 kernel:
  // back to back at the power cap the wide tile looked better there (1106-1113 -> 1230-1236 TFLOP/s),
  // but INSIDE the step, where the LM head runs at the clocks the lighter passes before it leave, it is slower — 7.1 ms
  // (1203-1222 TFLOP/s) against 5.5-5.7 ms (1509-1573) in the bench line's per-shape table, same code otherwise.
  if (plain && !no_wide && g_gemm_cg == 2 && K >= 8192 && M >= 1024 &&
      N >= 256 && N % 8 == 0 && ldc % 8 == 0 &&
      lda % 8 == 0 && ldb % 8 == 0 && reinterpret_cast<uintptr_t>(A) % 16 == 0 && reinterpret_cast<uintptr_t>(B) % 16 == 0 &&
      reinterpret_cast<uintptr_t>(C) % 16 == 0)
    return launch_gemm_wide(A, lda, B, ldb, C, ldc, (int)M, (int)N, (int)K, (cudaStream_t)stream);
  GemmParams p{};
  p.M = (int)M; p.N = (int)N; p.K = (int)K;
  p.C = C; p.ldc = ldc;
  p.col_scale = static_cast<const __nv_bfloat16*>(col_scale);
  p.flags = round_before_scale ? 2 : 0;
  fill_epilogue(p, epi);
  return g_gemm_cg == 2 ? launch_gemm<false, 2>(A, lda, B, ldb, p, (cudaStream_t)stream)
                        : launch_gemm<false, 1>(A, lda, B, ldb, p, (cudaStream_t)stream);
}

}  // extern "C"

// Token splits of lora_wgrad: one CTA per SM is resident (147 KB ring), so the kernel lasts waves x (tokens per split + a
// fixed fill/drain cost of ~5 stages). Pick the split count that minimises that: "just enough CTAs to cover the SMs" left
// a nearly empty second wave (P = 4096: 32 tiles x 5 splits = 160 CTAs on 148 SMs; 9 splits = 288 CTAs, two full waves
// of half the length). At most LLAMAX_LORA_WGRAD_MAX_SPLITS splits.
static void lora_wgrad_splits(int64_t M, int p_tiles, int& splits, int& k_per_split) {
  splits = std::max(1, std::min(LLAMAX_LORA_WGRAD_MAX_SPLITS, (sm_count() + p_tiles - 1) / p_tiles));
  k_per_split = (int)((M + splits - 1) / splits);
  k_per_split = ((k_per_split + 63) / 64) * 64;
  splits = (int)((M + k_per_split - 1) / k_per_split);
  if (p_tiles * 2 <= sm_count()) {   // wide outputs (P = 14336) stream at HBM rate either way: 79 vs 81 us
    int64_t best_cost = INT64_MAX;
    for (int s = 1; s <= LLAMAX_LORA_WGRAD_MAX_SPLITS; ++s) {
      int kp = (int)((M + s - 1) / s);
      kp = ((kp + 63) / 64) * 64;
      const int s_eff = (int)((M + kp - 1) / kp);
      if (s_eff != s) continue;
      const int64_t waves = ((int64_t)p_tiles * s + sm_count() - 1) / sm_count();
      const int64_t cost = waves * (kp + 320);
      if (cost < best_cost) { best_cost = cost; splits = s; k_per_split = kp; }
    }
  }
}

// workspace == NULL: splits are reduced into `out` with fp32 atomics; else the deterministic form (partials + ordered sum)
static int lora_wgrad_run(const void* X, int64_t ldx, const void* Ht, int64_t ldht, void* out, void* workspace, int64_t M,
                          int64_t P, int32_t R, float alpha, void* stream) {
  if (!X || !Ht || !out) return set_error(LLAMAX_ERR_ARG, "lora_wgrad: null pointer");
  if (R < 1 || R > 32) return set_error(LLAMAX_ERR_ARG, "lora_wgrad: rank must be in [1, 32]");
  if (M <= 0 || P <= 0) return set_error(LLAMAX_ERR_ARG, "lora_wgrad: empty problem");
  if (ldx % 8 || ldht % 8 || (reinterpret_cast<uintptr_t>(X) % 16) || (reinterpret_cast<uintptr_t>(Ht) % 16))
    return set_error(LLAMAX_ERR_ARG, "lora_wgrad: X / H^T must be 16-byte aligned with pitches multiple of 8");
  cudaStream_t st = (cudaStream_t)stream;
  if (workspace == nullptr) {
    cudaError_t e = cudaMemsetAsync(out, 0, (size_t)P * R * sizeof(float), st);
    if (e != cudaSuccess) return set_cuda_error(e, "lora_wgrad: memset");
  }
  CUtensorMap tmX, tmHt;
  int rc = make_tmap_2d(&tmX, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, X, P, M, ldx, 64, 64);
  if (rc) return rc;
  rc = make_tmap_2d(&tmHt, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, Ht, M, R, ldht, 64, 32);
  if (rc) return rc;
  auto kern = workspace ? lora_wgrad_tc_kernel<true> : lora_wgrad_tc_kernel<false>;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), wg::kSmem, "lora_wgrad: cudaFuncSetAttribute")))
    return rc;
  const int p_tiles = (int)((P + 127) / 128);
  int splits, k_per_split;
  lora_wgrad_splits(M, p_tiles, splits, k_per_split);
  dim3 grid(p_tiles, splits);
  kern<<<grid, 192, wg::kSmem, st>>>(tmX, tmHt, (float*)(workspace ? workspace : out), (int)P, R, (int)M, k_per_split,
                                     alpha);
  LX_CHECK_LAUNCH("lora_wgrad");
  if (workspace) return launch_reduce_partials_f32((const float*)workspace, (float*)out, splits, P * R, st);
  return 0;
}

extern "C" {

int llamax_lora_wgrad(const void* X, int64_t ldx, const void* Ht, int64_t ldht, void* out, int64_t M, int64_t P,
                      int32_t R, float alpha, void* stream) {
  return lora_wgrad_run(X, ldx, Ht, ldht, out, nullptr, M, P, R, alpha, stream);
}

int llamax_lora_wgrad_deterministic(const void* X, int64_t ldx, const void* Ht, int64_t ldht, void* out,
                                    void* workspace, int64_t M, int64_t P, int32_t R, float alpha, void* stream) {
  if (!workspace) return set_error(LLAMAX_ERR_ARG, "lora_wgrad: null pointer");
  return lora_wgrad_run(X, ldx, Ht, ldht, out, workspace, M, P, R, alpha, stream);
}

int llamax_lora_bwd_pair(const void* dY, int64_t lddy, const void* Bt, int64_t ldbt, const void* Ht, int64_t ldht,
                         void* dh, int64_t lddh, void* dht, int64_t lddht, void* dh_accum, void* dB, int64_t M,
                         int64_t N, int32_t R, float alpha, void* stream) {
  if (!dY || !Bt || !Ht || !dh || !dh_accum || !dB) return set_error(LLAMAX_ERR_ARG, "lora_bwd_pair: null pointer");
  if (R < 8 || R > 32 || R % 8) return set_error(LLAMAX_ERR_ARG, "lora_bwd_pair: rank must be 8, 16, 24 or 32");
  if (M <= 0 || N <= 0) return set_error(LLAMAX_ERR_ARG, "lora_bwd_pair: empty problem");
  if (lddy % 8 || ldbt % 8 || ldht % 8 || lddh % 8 || (reinterpret_cast<uintptr_t>(dY) % 16) ||
      (reinterpret_cast<uintptr_t>(Bt) % 16) || (reinterpret_cast<uintptr_t>(Ht) % 16) ||
      (reinterpret_cast<uintptr_t>(dh) % 16))
    return set_error(LLAMAX_ERR_ARG, "lora_bwd_pair: operands must be 16-byte aligned with pitches multiple of 8");
  cudaStream_t st = (cudaStream_t)stream;
  const int m_blocks = (int)((M + 127) / 128);
  const int total_chunks = (int)((N + 127) / 128);
  // Enough token blocks to cover most of the SMs (16 k tokens: 128 of 148): no split — one wave, every CTA streams its
  // whole row of tiles through one pipeline fill, dh is final in the CTA (no fp32 partial buffer, its memset and the
  // convert launch). Measured at the clocks of a power-capped step (tools/ew_sustained.py): dY [M, 4096] 66.6 -> 57.2 us,
  // [M, 14336] 134.9 -> 126.8 us against the 3-way split. Fewer token blocks: enough CTAs for ~2.5 waves, a split streams
  // at least 8 tiles.
  int splits = m_blocks * 4 >= sm_count() * 3
                   ? 1
                   : std::max(1, std::min(total_chunks / 8, (5 * sm_count() / 2 + m_blocks - 1) / m_blocks));
  int chunks_per_split = (total_chunks + splits - 1) / splits;
  splits = (total_chunks + chunks_per_split - 1) / chunks_per_split;
  cudaError_t e = cudaMemsetAsync(dB, 0, (size_t)N * R * sizeof(float), st);
  if (e != cudaSuccess) return set_cuda_error(e, "lora_bwd_pair: memset");
  if (splits > 1) {
    e = cudaMemsetAsync(dh_accum, 0, (size_t)M * R * sizeof(float), st);
    if (e != cudaSuccess) return set_cuda_error(e, "lora_bwd_pair: memset");
  }
  CUtensorMap tmY, tmBt, tmHt;
  int rc = make_tmap_2d(&tmY, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dY, N, M, lddy, 64, 128);
  if (rc) return rc;
  rc = make_tmap_2d(&tmBt, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, Bt, N, R, ldbt, 64, 32);
  if (rc) return rc;
  rc = make_tmap_2d(&tmHt, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, Ht, M, R, ldht, 64, 32);
  if (rc) return rc;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(lora_bwd_pair_kernel), lp::kSmem, "lora_bwd_pair: cudaFuncSetAttribute")))
    return rc;
  dim3 grid(m_blocks, splits);
  lora_bwd_pair_kernel<<<grid, 192, lp::kSmem, st>>>(tmY, tmBt, tmHt, (__nv_bfloat16*)dh, lddh,
                                                     splits > 1 ? nullptr : (__nv_bfloat16*)dht, lddht,
                                                     splits > 1 ? (float*)dh_accum : nullptr, (float*)dB, (int)M, (int)N,
                                                     R, chunks_per_split, alpha);
  LX_CHECK_LAUNCH("lora_bwd_pair");
  if (splits > 1) {
    const int64_t n = M * (R / 8);
    lora_dh_convert_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const float*)dh_accum, (__nv_bfloat16*)dh, lddh,
                                                                        (__nv_bfloat16*)dht, lddht, M, R);
    LX_CHECK_LAUNCH("lora_bwd_pair: convert");
  }
  return 0;
}

int llamax_bf16_gemm_swiglu_bwd(const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int64_t N, int64_t K,
                                const llamax_epilogue_t* epi, const void* ab, int64_t ld_ab, void* dab, int64_t ld_dab,
                                void* g, void* stream) {
  if (!A || !B || !ab || !dab) return set_error(LLAMAX_ERR_ARG, "bf16_gemm_swiglu_bwd: null pointer");
  if (M <= 0 || N <= 0 || K <= 0) return set_error(LLAMAX_ERR_ARG, "gemm: empty problem");
  if (N % 16 || ld_ab % 8 || ld_dab % 8 || ld_ab < 2 * N || ld_dab < 2 * N)
    return set_error(LLAMAX_ERR_ARG, "bf16_gemm_swiglu_bwd: N % 16 == 0 and pitches % 8 == 0, >= 2N required");
  if ((reinterpret_cast<uintptr_t>(ab) | reinterpret_cast<uintptr_t>(dab) | reinterpret_cast<uintptr_t>(g)) % 16)
    return set_error(LLAMAX_ERR_ARG, "bf16_gemm_swiglu_bwd: ab / dab / g must be 16-byte aligned");
  if (epi != nullptr && epi->resid != nullptr)
    return set_error(LLAMAX_ERR_ARG, "bf16_gemm_swiglu_bwd: no residual term in this epilogue");
  GemmParams p{};
  p.M = (int)M; p.N = (int)N; p.K = (int)K;
  fill_epilogue(p, epi);
  p.swi_ab = static_cast<const __nv_bfloat16*>(ab); p.ld_ab = ld_ab;
  p.swi_dab = static_cast<__nv_bfloat16*>(dab); p.ld_dab = ld_dab;
  p.swi_g = static_cast<__nv_bfloat16*>(g);
  cudaStream_t st = (cudaStream_t)stream;
  const int r = p.lora_rank <= 0 ? 0 : p.lora_rank <= 8 ? 8 : 16;
  if (g_gemm_cg == 2) {
    if (r == 0) return launch_gemm_r<false, 2, 0, false, true>(A, lda, B, ldb, p, st);
    if (r == 8) return launch_gemm_r<false, 2, 8, false, true>(A, lda, B, ldb, p, st);
    return launch_gemm_r<false, 2, 16, false, true>(A, lda, B, ldb, p, st);
  }
  if (r == 0) return launch_gemm_r<false, 1, 0, false, true>(A, lda, B, ldb, p, st);
  if (r == 8) return launch_gemm_r<false, 1, 8, false, true>(A, lda, B, ldb, p, st);
  return launch_gemm_r<false, 1, 16, false, true>(A, lda, B, ldb, p, st);
}

int llamax_bf16_gemm_rowdot(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t M,
                            int64_t N, int64_t K, const llamax_epilogue_t* epi, const void* other, int64_t ld_other,
                            void* dot_out, int64_t S, void* stream) {
  if (!A || !B || !C || !other || !dot_out) return set_error(LLAMAX_ERR_ARG, "bf16_gemm_rowdot: null pointer");
  if (M <= 0 || N <= 0 || K <= 0 || S <= 0 || M % S) return set_error(LLAMAX_ERR_ARG, "bf16_gemm_rowdot: M must be a multiple of S");
  if (N % 256) return set_error(LLAMAX_ERR_ARG, "bf16_gemm_rowdot: N must be a multiple of 256 (groups of 128 columns, two per tile)");
  if (other == C) return set_error(LLAMAX_ERR_ARG, "bf16_gemm_rowdot: `other` must not alias C");
  if (epi != nullptr && epi->resid != nullptr) return set_error(LLAMAX_ERR_ARG, "bf16_gemm_rowdot: no residual term in this form");
  if (g_gemm_cg != 2) return set_error(LLAMAX_ERR_ARG, "bf16_gemm_rowdot: needs the CTA-pair configuration");
  GemmParams p{};
  p.M = (int)M; p.N = (int)N; p.K = (int)K;
  p.C = C; p.ldc = ldc;
  fill_epilogue(p, epi);
  p.resid = static_cast<const __nv_bfloat16*>(other);
  p.ldr = ld_other;
  p.dot_out = static_cast<float*>(dot_out);
  p.dot_S = (int)S;
  p.flags = 4;
  cudaStream_t st = (cudaStream_t)stream;
  const int r = p.lora_rank <= 0 ? 0 : p.lora_rank <= 8 ? 8 : 16;
  if (r == 0) return launch_gemm_r<false, 2, 0, false, false, true>(A, lda, B, ldb, p, st);
  if (r == 8) return launch_gemm_r<false, 2, 8, false, false, true>(A, lda, B, ldb, p, st);
  return launch_gemm_r<false, 2, 16, false, false, true>(A, lda, B, ldb, p, st);
}

int llamax_bf16_int8_gemm(const void* A, int64_t lda, const void* B8, int64_t ldb8, const void* b_scale, int b_layout,
                          const void* tail, int64_t ldt, void* C, int64_t ldc, int64_t M, int64_t N, int64_t K,
                          int64_t K1, const llamax_epilogue_t* epi, void* stream) {
  if (!A || !B8 || !C || !b_scale) return set_error(LLAMAX_ERR_ARG, "bf16_int8_gemm: null pointer");
  GemmParams p{};
  p.M = (int)M; p.N = (int)N; p.K = (int)K;
  p.C = C; p.ldc = ldc;
  fill_epilogue(p, epi);
  cudaStream_t st = (cudaStream_t)stream;
  const int r = p.lora_rank <= 0 ? 0 : p.lora_rank <= 8 ? 8 : 16;
  if (b_layout == 0) {   // weight-only forward: bf16(acc) * scale[n]
    if (tail != nullptr || K1 != K) return set_error(LLAMAX_ERR_ARG, "bf16_int8_gemm: layout 0 has no tail (K1 == K)");
    p.col_scale = static_cast<const __nv_bfloat16*>(b_scale);
    p.flags = 2;
    if (r == 0) return launch_gemm_mix<1, 0>(A, lda, B8, ldb8, nullptr, 0, p, st);
    if (r == 8) return launch_gemm_mix<1, 8>(A, lda, B8, ldb8, nullptr, 0, p, st);
    return launch_gemm_mix<1, 16>(A, lda, B8, ldb8, nullptr, 0, p, st);
  }
  if (b_layout != 1) return set_error(LLAMAX_ERR_ARG, "bf16_int8_gemm: b_layout must be 0 or 1");
  p.k_scale = static_cast<const __nv_bfloat16*>(b_scale);
  p.K1 = (int)K1;
  if (r == 0) return launch_gemm_mix<2, 0>(A, lda, B8, ldb8, tail, ldt, p, st);
  if (r == 8) return launch_gemm_mix<2, 8>(A, lda, B8, ldb8, tail, ldt, p, st);
  return launch_gemm_mix<2, 16>(A, lda, B8, ldb8, tail, ldt, p, st);
}

int llamax_bf16_int8_gemm_swiglu_bwd(const void* A, int64_t lda, const void* B8, int64_t ldb8, const void* k_scale,
                                     int64_t M, int64_t N, int64_t K, const llamax_epilogue_t* epi, const void* ab,
                                     int64_t ld_ab, void* dab, int64_t ld_dab, void* g, void* stream) {
  if (!A || !B8 || !k_scale || !ab || !dab) return set_error(LLAMAX_ERR_ARG, "bf16_int8_gemm_swiglu_bwd: null pointer");
  if (M <= 0 || N <= 0 || K <= 0) return set_error(LLAMAX_ERR_ARG, "gemm: empty problem");
  if (N % 16 || ld_ab % 8 || ld_dab % 8 || ld_ab < 2 * N || ld_dab < 2 * N)
    return set_error(LLAMAX_ERR_ARG, "bf16_int8_gemm_swiglu_bwd: N % 16 == 0 and pitches % 8 == 0, >= 2N required");
  if ((reinterpret_cast<uintptr_t>(ab) | reinterpret_cast<uintptr_t>(dab) | reinterpret_cast<uintptr_t>(g)) % 16)
    return set_error(LLAMAX_ERR_ARG, "bf16_int8_gemm_swiglu_bwd: ab / dab / g must be 16-byte aligned");
  if (epi != nullptr && epi->resid != nullptr)
    return set_error(LLAMAX_ERR_ARG, "bf16_int8_gemm_swiglu_bwd: no residual term in this epilogue");
  GemmParams p{};
  p.M = (int)M; p.N = (int)N; p.K = (int)K;
  fill_epilogue(p, epi);
  p.swi_ab = static_cast<const __nv_bfloat16*>(ab); p.ld_ab = ld_ab;
  p.swi_dab = static_cast<__nv_bfloat16*>(dab); p.ld_dab = ld_dab;
  p.swi_g = static_cast<__nv_bfloat16*>(g);
  p.k_scale = static_cast<const __nv_bfloat16*>(k_scale);
  p.K1 = (int)K;
  cudaStream_t st = (cudaStream_t)stream;
  const int r = p.lora_rank <= 0 ? 0 : p.lora_rank <= 8 ? 8 : 16;
  if (r == 0) return launch_gemm_mix<2, 0, true>(A, lda, B8, ldb8, nullptr, 0, p, st);
  if (r == 8) return launch_gemm_mix<2, 8, true>(A, lda, B8, ldb8, nullptr, 0, p, st);
  return launch_gemm_mix<2, 16, true>(A, lda, B8, ldb8, nullptr, 0, p, st);
}

int llamax_bf16_gemm_tn(const void* At, int64_t ldat, const void* Bt, int64_t ldbt, void* C, int64_t ldc, int64_t M,
                        int64_t N, int64_t K, void* stream) {
  if (!At || !Bt || !C) return set_error(LLAMAX_ERR_ARG, "bf16_gemm_tn: null pointer");
  if (M <= 0 || N <= 0 || K <= 0) return set_error(LLAMAX_ERR_ARG, "gemm: empty problem");
  if (M % 8) return set_error(LLAMAX_ERR_ARG, "bf16_gemm_tn: M must be a multiple of 8");
  GemmParams p{};
  p.M = (int)M; p.N = (int)N; p.K = (int)K;
  p.C = C; p.ldc = ldc;
  return g_gemm_cg == 2 ? launch_gemm_r<false, 2, 0, true>(At, ldat, Bt, ldbt, p, (cudaStream_t)stream)
                        : launch_gemm_r<false, 1, 0, true>(At, ldat, Bt, ldbt, p, (cudaStream_t)stream);
}

}  // extern "C"
