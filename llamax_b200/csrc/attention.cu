// Prefix-LM flash attention for the Llama decoder block (modelling/llama.py:129-137), forward and backward,
// on tcgen05 tensor cores with TMEM accumulators and TMA-fed 128B-swizzled shared-memory tiles.
//
//   mask(q, kv) = (kv < P) | (q >= kv)      P = prefix_len (bidirectional prefix, causal suffix; P = 0: causal)
//
// GQA native: the 4 (Hq/Hkv) query heads of a group read the same K/V tiles straight from the [B,S,Hkv,D]
// projection output (no repeat_interleave, no transposes: TMA walks the strided layout). The mask is applied at
// tile granularity: tiles that are fully masked are never visited, fully visible tiles skip the element test.
//
// Optional packed-sequence document mask: additionally kv >= doc_start[q] (tiles outside a row's document skipped).
//
// Forward  : default = attn_fwd5_kernel, persistent: one CTA per SM walks a length-balanced list of items (pair of
//            128-row query tiles, query head, sequence); warp0 TMA, warps1-2 MMA issue (one per tile), two softmax
//            warpgroups (thread = row). Per tile S = Q K^T in TMEM is read once into registers, P (bf16 pairs) is written
//            back over the score columns in four chunks and consumed by the PV MMA straight from TMEM, O accumulates
//            in TMEM with lazy rescaling; exp2-domain online softmax, LSE saved in natural log. Older forms kept behind
//            LLAMAX_ATTN_FWD (1: one tile per CTA, 2: two tiles / one issuer — also the packed-document path, 3: two
//            threads per row, 4: v5 without the persistent loop).
// Backward : CTA = (128 kv rows, 1 kv head), loops over the group's query heads x 128-row query tiles; every MMA is
//            128 x 128 x 16. S^T = K Q^T and dP^T = V dO^T in TMEM (thread = kv row); P^T goes back to TMEM as bf16 pairs
//            (A operand of dV += P^T dO straight from TMEM), dS^T through smem (dK += dS^T Q, dQ^T = K^T dS^T); dV, dK
//            accumulate in TMEM for the CTA lifetime; dQ^T is drained to registers and reduced into an fp32 buffer with
//            coalesced red.global.add; RoPE's backward is applied to dK in the epilogue and to dQ in the fp32 -> bf16
//            convert. See the comment block above attn_bwd_kernel for the TMEM aliasing and the MMA issue order.
// head_dim 128 natively; head_dim 64 runs on the same 128-wide tiles (TMA zero-fills the missing half).
#include <type_traits>

#include "common.cuh"
#include "host_utils.h"
#include "llamax_b200.h"

namespace lx {

constexpr int kHD = 128;                    // head dim
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

#ifdef LX_ATTN_TRACE
// Debug build only (tools/attn_trace.py): SM-clock timestamps of one CTA's pipeline phases, 16 slots per step.
__device__ long long* g_attn_trace = nullptr;
#define LX_TR(on, s, slot)                                                        \
  do {                                                                            \
    if ((on) && g_attn_trace && (s) < 128) g_attn_trace[(s) * 32 + (slot)] = clock64(); \
  } while (0)
#else
#define LX_TR(on, s, slot) \
  do {                     \
  } while (0)
#endif

__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// ================================================================================================
// forward
// ================================================================================================
struct AttnFwdParams {
  __nv_bfloat16* o;
  int64_t ldo;
  float* lse;
  int B, S, Hq, Hkv, P;
  int D;             // real head dim (64 or 128); tiles are always 128 wide, TMA zero-fills columns >= D
  float scale_log2;  // softmax scale * log2(e)
  const int32_t* doc_start;  // [B, S] first position of the document containing each position, or null
  const int32_t* prefix_b;   // null, or [B]: per-sequence prefix length (overrides P)
};

namespace fwd {
constexpr int kTile = 128;
constexpr int kTileBytes = kTile * kHD * 2;       // 32 KB: two 16 KB boxes of [128 rows x 128 B]
constexpr int kOffQ = 0;
constexpr int kOffK = kOffQ + kTileBytes;         // kNB stages of K, then kNB stages of V
constexpr int kNumBars = 1 + 4 + 4 + 4 + 2;       // q_full, k full/empty[2], v full/empty[2], s full/empty[2], p_full, pv_done
constexpr int smem_bytes(int nb) { return kTileBytes * (1 + 2 * nb) + kNumBars * 8 + 16 + 1024; }
constexpr int kNB = 2;                             // smem stages of K and V, TMEM score buffers
constexpr int kThreads = 256;                     // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warps 4-7 softmax
}  // namespace fwd

// Tile classification of a 128-row query tile starting at q0 (attn_fwd_kernel, attn_bwd_dq_kernel): the kv tiles it
// visits are [j_begin, j_begin + n_kv) — up to max(P, q0 + 128), and, with packed documents, from the start of the first
// row's document on; a visited tile needs no element test when every (q, kv) pair of it is visible and in range.
template <bool kDocs>
__device__ __forceinline__ void q_tile_kv_range(int S, int Pb, const int32_t* doc_start, int b, int q0, int& j_begin,
                                                int& n_kv) {
  const int kv_end = min(S, max(Pb, q0 + 128));
  j_begin = kDocs ? doc_start[(int64_t)b * S + q0] / 128 : 0;
  n_kv = (kv_end + 127) / 128 - j_begin;
}
// ds_tile: document start of the tile's last row (0 without documents)
__device__ __forceinline__ bool q_tile_full(int S, int Pb, int ds_tile, int q0, int kv0) {
  return (kv0 + 128 <= S) && ((kv0 + 128 <= Pb) || (kv0 + 127 <= q0)) && (kv0 >= ds_tile);
}

// kDocs: packed-document mask compiled in; kD: real head dim (64 runs on zero-padded 128-wide tiles).
// (A variant with two softmax warpgroups per query tile — column halves, row maxima exchanged through smem — was
// measured 10 % slower than this single-warpgroup version on B200: the extra 256-thread barrier per tile and the
// doubled TMEM read contention cost more than the halved per-thread work saves.)
// K/V are double-buffered in smem and S in TMEM (kNB = 2), one CTA per SM (160 KB smem, 512 TMEM columns).
// P is handed to the PV MMA through TMEM: bf16 pairs written over the score columns just read, consumed by
// tcgen05.mma with the A operand in TMEM (+9 % over staging P in 128B-swizzled smem).
// Rejected after measurement: single buffers with two CTAs per SM and setmaxnreg register rebalancing (-12 %), and two
// softmax warpgroups per query tile (-10 %).
template <bool kDocs, int kD>
__global__ void __launch_bounds__(fwd::kThreads, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, const AttnFwdParams p) {
  using namespace fwd;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int kOffV = kOffK + kNB * kTileBytes;
  constexpr int kOffBar = kOffV + kNB * kTileBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;
  uint64_t* k_empty = bars + 3;
  uint64_t* v_full = bars + 5;
  uint64_t* v_empty = bars + 7;
  uint64_t* s_full = bars + 9;
  uint64_t* s_empty = bars + 11;
  uint64_t* p_full = bars + 13;
  uint64_t* pv_done = bars + 14;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);

  const int warp = threadIdx.x >> 5;
#ifdef LX_ATTN_TRACE
  const bool tr_cta = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 && (threadIdx.x & 31) == 0 && (warp == 1 || warp == 4);
#endif
  // grid = (query heads, batch, query tiles): the tile index is the slowest one and runs backwards, so CTAs are
  // dispatched longest-first (the last query tile visits every kv tile); the 4 heads of a GQA group run together
  const int qt = gridDim.z - 1 - blockIdx.z;
  const int h = blockIdx.x, b = blockIdx.y;
  const int Pb = p.prefix_b ? min(max(p.prefix_b[b], 0), p.S) : p.P;   // prefix length of this sequence
  const int hk = h / (p.Hq / p.Hkv);
  const int q0 = qt * kTile;
  int j_begin, n_kv;   // visited kv tiles
  q_tile_kv_range<kDocs>(p.S, Pb, p.doc_start, b, q0, j_begin, n_kv);

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
  }
  if (warp == 1 && elect_one()) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&s_empty[i], 4);
    }
    mbar_init(p_full, 4);
    mbar_init(pv_done, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<1>(tmem_slot, 256 * kNB);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base;              // kNB x 128 columns
  const uint32_t tmem_O = tmem_base + kNB * 128;  // 128 columns

  if (warp == 0) {
    // ------------------------------------ TMA producer ------------------------------------
    if (elect_one()) {
      mbar_expect_tx(q_full, kTileBytes);
      tma_load_4d(smem + kOffQ, &tmQ, q_full, 0, h, q0, b);
      tma_load_4d(smem + kOffQ + kTileBytes / 2, &tmQ, q_full, 64, h, q0, b);
      for (int j = 0; j < n_kv; ++j) {
        const int st = kNB == 2 ? (j & 1) : 0;
        const uint32_t ph = (kNB == 2 ? (j >> 1) : j) & 1;
        mbar_wait(&k_empty[st], ph ^ 1);
        mbar_expect_tx(&k_full[st], kTileBytes);
        uint8_t* sk = smem + kOffK + st * kTileBytes;
        tma_load_4d(sk, &tmK, &k_full[st], 0, hk, (j_begin + j) * kTile, b);
        tma_load_4d(sk + kTileBytes / 2, &tmK, &k_full[st], 64, hk, (j_begin + j) * kTile, b);
        mbar_wait(&v_empty[st], ph ^ 1);
        mbar_expect_tx(&v_full[st], kTileBytes);
        uint8_t* sv = smem + kOffV + st * kTileBytes;
        tma_load_4d(sv, &tmV, &v_full[st], 0, hk, (j_begin + j) * kTile, b);
        tma_load_4d(sv + kTileBytes / 2, &tmV, &v_full[st], 64, hk, (j_begin + j) * kTile, b);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------ MMA issuer ------------------------------------
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc(1, 1, 128, 128, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc(1, 1, 128, 128, 0, 1);  // B = V is MN-major
      constexpr uint32_t kHi = desc_hi(1024);
      const uint32_t loQ = desc_lo(smem_u32(smem + kOffQ), 16);
      const uint32_t loK0 = desc_lo(smem_u32(smem + kOffK), 16), loV0 = desc_lo(smem_u32(smem + kOffV), 16384);
      auto issue_s = [&](int j) {
        const int st = kNB == 2 ? (j & 1) : 0;
        const uint32_t ph = (kNB == 2 ? (j >> 1) : j) & 1;
        mbar_wait(&k_full[st], ph);
        mbar_wait(&s_empty[st], ph ^ 1);
        tc_fence_after();
        const uint32_t loK = loK0 + st * (kTileBytes / 16);
#pragma unroll
        for (int dh = 0; dh < 2; ++dh)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_ss<false, 1>(tmem_S + st * 128, desc_join(loQ + dh * 1024 + ks * 2, kHi),
                              desc_join(loK + dh * 1024 + ks * 2, kHi), idesc_s, (dh | ks) != 0);
        umma_commit(&s_full[st]);
        umma_commit(&k_empty[st]);
      };
      mbar_wait(q_full, 0);
      issue_s(0);
      for (int j = 0; j < n_kv; ++j) {
        if (kNB == 2 && j + 1 < n_kv) issue_s(j + 1);  // next scores into the other TMEM buffer
        const int st = kNB == 2 ? (j & 1) : 0;
        LX_TR(tr_cta, j, 0);
        mbar_wait(&v_full[st], (kNB == 2 ? (j >> 1) : j) & 1);
        mbar_wait(p_full, j & 1);
        tc_fence_after();
        LX_TR(tr_cta, j, 1);
        const uint32_t loV = loV0 + st * (kTileBytes / 16);
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t bd = desc_join(loV + (kb * 64 + ks * 16) * 8, kHi);
            // A = P read from TMEM: bf16 pairs, 8 columns per 16-wide k-step, aliasing the score buffer
            umma_ts_f16(tmem_O, tmem_S + st * 128 + (kb * 4 + ks) * 8, bd, idesc_pv, (j | kb | ks) != 0);
          }
        umma_commit(pv_done);
        umma_commit(&v_empty[st]);
        if (kNB == 1 && j + 1 < n_kv) issue_s(j + 1);  // single score buffer: free once PV_j (in order) consumed P_j
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ------------------------------------ softmax / correction / epilogue ------------------------------------
    const int r = threadIdx.x - 128;  // row in tile == TMEM lane
    const int ew = warp - 4;
    const uint32_t lane_off = uint32_t(ew * 32) << 16;
    const int q = q0 + r;
    float m_used = -INFINITY, l = 0.f;
    const int ds_row = kDocs ? p.doc_start[(int64_t)b * p.S + min(q, p.S - 1)] : 0;
    const int ds_tile = kDocs ? p.doc_start[(int64_t)b * p.S + min(q0 + kTile - 1, p.S - 1)] : 0;
    for (int j = 0; j < n_kv; ++j) {
      const int st = kNB == 2 ? (j & 1) : 0;
      const int kv0 = (j_begin + j) * kTile;
      const bool full_tile = q_tile_full(p.S, Pb, ds_tile, q0, kv0);
      LX_TR(tr_cta, j, 4);
      mbar_wait(&s_full[st], (kNB == 2 ? (j >> 1) : j) & 1);
      tc_fence_after();
      LX_TR(tr_cta, j, 5);
      const uint32_t tS = tmem_S + st * 128 + lane_off;
      // single pass over TMEM: the whole score row (128 fp32) lives in registers
      uint32_t sv[4][32];
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld_32x32(tS + c * 32, sv[c]);
      tmem_wait_ld_regs(sv[0]);
      tmem_wait_ld_regs(sv[1]);
      tmem_wait_ld_regs(sv[2]);
      tmem_wait_ld_regs(sv[3]);
      LX_TR(tr_cta, j, 6);
      // S is in registers: release the TMEM buffer for the next QK^T right away
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(&s_empty[st]);
      if (!full_tile) {
        // the visible keys of a row are ONE interval of the tile's columns, [lo, lo + width): the prefix-LM mask keeps
        // kv < max(P, q + 1) (and kv < S), packed documents additionally cut the head (kv >= ds_row) — one unsigned
        // compare against a per-row constant and a select per element instead of three compares
        const int lo = kDocs ? ds_row - kv0 : 0;
        const uint32_t width = (uint32_t)max(min(p.S, max(Pb, q + 1)) - kv0 - lo, 0);
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if ((uint32_t)(c * 32 + i - lo) >= width) sv[c][i] = 0xff800000u;  // -inf
      }
      // four independent max chains (one per 32-column chunk): a single chain of 64 dependent FMNMX3 is ~300 cycles of
      // pure latency for the one softmax warp a scheduler has
      float mx4[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        mx4[c] = __uint_as_float(sv[c][0]);
#pragma unroll
        for (int i = 1; i < 32; ++i) mx4[c] = fmaxf(mx4[c], __uint_as_float(sv[c][i]));
      }
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      const float m_tile = mx * p.scale_log2;
      float alpha = 1.f;
      if (m_tile > m_used + 8.f) {  // lazy rescale: only when the running max grows by more than 2^8
        alpha = ex2(m_used - m_tile);
        m_used = m_tile;
      }
      uint32_t preg[64];
      float rowsum = 0.f;
      // a row may see nothing in a visited tile (packed documents): keep the exponent finite so that exp2(-inf) = 0
      const float m_exp = (m_used == -INFINITY) ? 0.f : m_used;
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const float p0 = ex2(fmaf(__uint_as_float(sv[c][i]), p.scale_log2, -m_exp));      // -inf -> 0
          const float p1 = ex2(fmaf(__uint_as_float(sv[c][i + 1]), p.scale_log2, -m_exp));
          rowsum += p0 + p1;
          preg[c * 16 + i / 2] = pack_bf16(p0, p1);
        }

      l = l * alpha + rowsum;
      LX_TR(tr_cta, j, 7);

      if (j > 0) {
        mbar_wait(pv_done, (j - 1) & 1);  // O stable, P buffer free
        tc_fence_after();
        LX_TR(tr_cta, j, 8);
        if (__any_sync(0xffffffffu, alpha != 1.f)) {
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(tmem_O + lane_off + c * 32, v);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * alpha);
            tmem_st_32x32(tmem_O + lane_off + c * 32, v);
          }
          tmem_wait_st();
        }
      }
      {
        // P (bf16 pairs) -> TMEM, over the first 64 columns of the score buffer this row was just read from
        uint32_t(&p0)[32] = *reinterpret_cast<uint32_t(*)[32]>(&preg[0]);
        uint32_t(&p1)[32] = *reinterpret_cast<uint32_t(*)[32]>(&preg[32]);
        tmem_st_32x32(tS, p0);
        tmem_st_32x32(tS + 32, p1);
        tmem_wait_st();
      }
      LX_TR(tr_cta, j, 9);
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(p_full);
    }
    // epilogue
    mbar_wait(pv_done, (n_kv - 1) & 1);
    tc_fence_after();
    const float inv_l = 1.f / l;
    const bool row_ok = q < p.S;
    __nv_bfloat16* orow = p.o + ((int64_t)b * p.S + q) * p.ldo + (int64_t)h * kD;
#pragma unroll 1
    for (int c = 0; c < kD / 32; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(tmem_O + lane_off + c * 32, v);
      tmem_wait_ld();
      if (row_ok) {
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          uint4 o4;
          o4.x = pack_bf16(__uint_as_float(v[i]) * inv_l, __uint_as_float(v[i + 1]) * inv_l);
          o4.y = pack_bf16(__uint_as_float(v[i + 2]) * inv_l, __uint_as_float(v[i + 3]) * inv_l);
          o4.z = pack_bf16(__uint_as_float(v[i + 4]) * inv_l, __uint_as_float(v[i + 5]) * inv_l);
          o4.w = pack_bf16(__uint_as_float(v[i + 6]) * inv_l, __uint_as_float(v[i + 7]) * inv_l);
          stg_v4(orow + c * 32 + i, o4);
        }
      }
    }
    if (row_ok) p.lse[((int64_t)b * p.Hq + h) * p.S + q] = (m_used + log2f(l)) * kLn2;
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<1>(tmem_base, 256 * kNB);
}

// ------------------------------------------------------------------------------------------------
// Forward, two query tiles per CTA ("ping-pong"). tools/attn_trace.py on the one-tile kernel above: the softmax
// warpgroup needs ~2400 cycles per 128x128 tile (128 ex2 per thread on the 16-lane XU pipe = 1024, the max, TMEM
// round-trips, barriers — one warp per scheduler, nothing to overlap with) against 1364 cycles of MMA work, and the
// chain softmax(j) -> PV(j) is serial. Here a CTA owns TWO 128-row query tiles with one softmax warpgroup each: while
// one group is in its exp phase the other waits for its MMAs, so XU pipe and tensor pipe are both kept busy and each
// K/V tile is loaded once for 256 query rows.
//   TMEM (512 columns): S0 | S1 (P written over the score columns read, A operand of PV from TMEM) | O0 | O1
//   MMA issue order   : S0(j0), S1(j0);  then per kv tile j:  PV0(j), S0(j+1) | PV1(j), S1(j+1)
// ------------------------------------------------------------------------------------------------
namespace fwd2 {
constexpr int kTile = 128;
constexpr int kTileBytes = kTile * kHD * 2;        // 32 KB
constexpr int kOffQ = 0;                           // 2 query tiles
constexpr int kOffK = kOffQ + 2 * kTileBytes;      // 2 stages
constexpr int kOffV = kOffK + 2 * kTileBytes;      // 2 stages
constexpr int kOffBar = kOffV + 2 * kTileBytes;
// q_full, k full/empty[2], v full/empty[2], s_full[2 tiles], p_full[2 tiles], pv_done[2 tiles]
constexpr int kNumBars = 1 + 4 + 4 + 2 + 2 + 2;
constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16 + 1024;
constexpr int kThreads = 384;                      // warpgroup 0: TMA / MMA / TMEM alloc; warpgroups 1, 2: softmax of tile 0, 1
constexpr int kRegsCtrl = 56, kRegsSoftmax = 224;  // 56 + 2 * 224 = 504 <= 512
}  // namespace fwd2

template <bool kDocs, int kD>
__global__ void __launch_bounds__(fwd2::kThreads, 1)
attn_fwd2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                 const __grid_constant__ CUtensorMap tmV, const AttnFwdParams p) {
  using namespace fwd2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;
  uint64_t* k_empty = bars + 3;
  uint64_t* v_full = bars + 5;
  uint64_t* v_empty = bars + 7;
  uint64_t* s_full = bars + 9;     // [tile]
  uint64_t* p_full = bars + 11;    // [tile]
  uint64_t* pv_done = bars + 13;   // [tile]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);

  const int warp = threadIdx.x >> 5;
#ifdef LX_ATTN_TRACE
  const bool tr_cta = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 && (threadIdx.x & 31) == 0 && (warp == 1 || warp == 4);
#endif
  // grid = (query heads, batch, pairs of query tiles): pairs run backwards so CTAs are dispatched longest-first
  const int pr = gridDim.z - 1 - blockIdx.z;
  const int h = blockIdx.x, b = blockIdx.y;
  const int Pb = p.prefix_b ? min(max(p.prefix_b[b], 0), p.S) : p.P;   // prefix length of this sequence
  const int hk = h / (p.Hq / p.Hkv);
  // per-tile kv tile ranges [jb_x, je_x); a tile past the end of the sequence has an empty range
  int jb_[2], je_[2];
#pragma unroll
  for (int x = 0; x < 2; ++x) {
    const int q0 = (2 * pr + x) * kTile;
    if (q0 < p.S) {
      const int kv_end = min(p.S, max(Pb, q0 + kTile));
      je_[x] = (kv_end + kTile - 1) / kTile;
      jb_[x] = kDocs ? p.doc_start[(int64_t)b * p.S + q0] / kTile : 0;
    } else {
      jb_[x] = je_[x] = 0;
    }
  }
  const bool act1 = je_[1] > jb_[1];
  const int jb = act1 ? min(jb_[0], jb_[1]) : jb_[0];
  const int je = max(je_[0], je_[1]);

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
  }
  if (warp == 1 && elect_one()) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);
      mbar_init(&pv_done[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<1>(tmem_slot, 512);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    setmaxnreg_dec<kRegsCtrl>();
    if (warp == 0) {
      // ------------------------------------ TMA producer ------------------------------------
      if (elect_one()) {
        mbar_expect_tx(q_full, 2 * kTileBytes);
#pragma unroll
        for (int x = 0; x < 2; ++x) {   // rows past the end of the sequence are zero-filled
          tma_load_4d(smem + kOffQ + x * kTileBytes, &tmQ, q_full, 0, h, (2 * pr + x) * kTile, b);
          tma_load_4d(smem + kOffQ + x * kTileBytes + kTileBytes / 2, &tmQ, q_full, 64, h, (2 * pr + x) * kTile, b);
        }
        for (int j = jb; j < je; ++j) {
          const int st = (j - jb) & 1;
          const uint32_t ph = ((j - jb) >> 1) & 1;
          mbar_wait(&k_empty[st], ph ^ 1);
          mbar_expect_tx(&k_full[st], kTileBytes);
          uint8_t* sk = smem + kOffK + st * kTileBytes;
          tma_load_4d(sk, &tmK, &k_full[st], 0, hk, j * kTile, b);
          tma_load_4d(sk + kTileBytes / 2, &tmK, &k_full[st], 64, hk, j * kTile, b);
          mbar_wait(&v_empty[st], ph ^ 1);
          mbar_expect_tx(&v_full[st], kTileBytes);
          uint8_t* sv = smem + kOffV + st * kTileBytes;
          tma_load_4d(sv, &tmV, &v_full[st], 0, hk, j * kTile, b);
          tma_load_4d(sv + kTileBytes / 2, &tmV, &v_full[st], 64, hk, j * kTile, b);
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ------------------------------------ MMA issuer ------------------------------------
      if (elect_one()) {
        constexpr uint32_t idesc_s = make_idesc(1, 1, 128, 128, 0, 0);
        constexpr uint32_t idesc_pv = make_idesc(1, 1, 128, 128, 0, 1);  // B = V is MN-major
        constexpr uint32_t kHi = desc_hi(1024);
        const uint32_t loQ0 = desc_lo(smem_u32(smem + kOffQ), 16);
        const uint32_t loK0 = desc_lo(smem_u32(smem + kOffK), 16), loV0 = desc_lo(smem_u32(smem + kOffV), 16384);
        auto active = [&](int x, int j) { return j >= jb_[x] && j < je_[x]; };
        // S_x(j) = Q_x K(j)^T; releases K(j) if x is the last tile that reads it
        auto issue_s = [&](int x, int j) {
          const int st = (j - jb) & 1;
          mbar_wait(&k_full[st], ((j - jb) >> 1) & 1);
          tc_fence_after();
          const uint32_t loQ = loQ0 + x * (kTileBytes / 16), loK = loK0 + st * (kTileBytes / 16);
#pragma unroll
          for (int dh = 0; dh < 2; ++dh)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma_ss<false, 1>(tmem_base + x * 128, desc_join(loQ + dh * 1024 + ks * 2, kHi),
                                desc_join(loK + dh * 1024 + ks * 2, kHi), idesc_s, (dh | ks) != 0);
          umma_commit(&s_full[x]);
          if (x == 1 || !active(1, j)) umma_commit(&k_empty[st]);
        };
        mbar_wait(q_full, 0);
        int it[2] = {0, 0};   // iterations done per tile
#pragma unroll
        for (int x = 0; x < 2; ++x)
          if (active(x, jb)) issue_s(x, jb);
        for (int j = jb; j < je; ++j) {
          const int st = (j - jb) & 1;
#pragma unroll
          for (int x = 0; x < 2; ++x) {
            if (!active(x, j)) continue;
            if (j == jb_[x] && j != jb) issue_s(x, j);   // a tile whose document starts later than its partner's
            if (x == 0) LX_TR(tr_cta, j, 0);
            mbar_wait(&v_full[st], ((j - jb) >> 1) & 1);
            mbar_wait(&p_full[x], it[x] & 1);
            tc_fence_after();
            if (x == 0) LX_TR(tr_cta, j, 1);
            const uint32_t loV = loV0 + st * (kTileBytes / 16);
#pragma unroll
            for (int kb = 0; kb < 2; ++kb)
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                umma_ts_f16(tmem_base + 256 + x * 128, tmem_base + x * 128 + (kb * 4 + ks) * 8,
                            desc_join(loV + (kb * 64 + ks * 16) * 8, kHi), idesc_pv, (it[x] | kb | ks) != 0);
            umma_commit(&pv_done[x]);
            if (x == 1 || !active(1, j)) umma_commit(&v_empty[st]);
            ++it[x];
            if (active(x, j + 1)) issue_s(x, j + 1);     // in order behind PV_x(j), which reads P from the same columns
          }
        }
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------ softmax / correction / epilogue: one warpgroup per query tile ------------
    setmaxnreg_inc<kRegsSoftmax>();
    const int x = (warp - 4) >> 2;
    const int ew = warp & 3;
    const int r = ew * 32 + lane_id();  // row in tile == TMEM lane
    const uint32_t lane_off = uint32_t(ew * 32) << 16;
    const int q0 = (2 * pr + x) * kTile;
    const int q = q0 + r;
    const int jb_x = x ? jb_[1] : jb_[0], je_x = x ? je_[1] : je_[0];
    const int n_kv = je_x - jb_x;
    const uint32_t tS = tmem_base + x * 128 + lane_off;
    const uint32_t tO = tmem_base + 256 + x * 128 + lane_off;
    float m_used = -INFINITY, l = 0.f;
    const int ds_row = kDocs ? p.doc_start[(int64_t)b * p.S + min(q, p.S - 1)] : 0;
    const int ds_tile = kDocs ? p.doc_start[(int64_t)b * p.S + min(q0 + kTile - 1, p.S - 1)] : 0;
    for (int i = 0; i < n_kv; ++i) {
      const int kv0 = (jb_x + i) * kTile;
      // tile needs the element test unless every (q, kv) pair is visible and in range
      const bool full_tile = (kv0 + kTile <= p.S) && ((kv0 + kTile <= Pb) || (kv0 + kTile - 1 <= q0)) && (kv0 >= ds_tile);
      if (x == 0) LX_TR(tr_cta, jb_x + i, 4);
      mbar_wait(&s_full[x], i & 1);
      tc_fence_after();
      if (x == 0) LX_TR(tr_cta, jb_x + i, 5);
      // single pass over TMEM: the whole score row (128 fp32) lives in registers
      uint32_t sv[4][32];
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld_32x32(tS + c * 32, sv[c]);
      tmem_wait_ld_regs(sv[0]);
      tmem_wait_ld_regs(sv[1]);
      tmem_wait_ld_regs(sv[2]);
      tmem_wait_ld_regs(sv[3]);
      if (x == 0) LX_TR(tr_cta, jb_x + i, 6);
      if (!full_tile) {
        // the visible keys of a row are ONE interval of the tile's columns, [lo, lo + width): the prefix-LM mask keeps
        // kv < max(P, q + 1) (and kv < S), packed documents additionally cut the head (kv >= ds_row) — one unsigned
        // compare against a per-row constant and a select per element instead of three compares
        const int lo = kDocs ? ds_row - kv0 : 0;
        const uint32_t width = (uint32_t)max(min(p.S, max(Pb, q + 1)) - kv0 - lo, 0);
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if ((uint32_t)(c * 32 + e - lo) >= width) sv[c][e] = 0xff800000u;  // -inf
      }
      float mx4[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        mx4[c] = __uint_as_float(sv[c][0]);
#pragma unroll
        for (int e = 1; e < 32; ++e) mx4[c] = fmaxf(mx4[c], __uint_as_float(sv[c][e]));
      }
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      const float m_tile = mx * p.scale_log2;
      float alpha = 1.f;
      if (m_tile > m_used + 8.f) {  // lazy rescale: only when the running max grows by more than 2^8
        alpha = ex2(m_used - m_tile);
        m_used = m_tile;
      }
      uint32_t preg[64];
      float rowsum = 0.f;
      // a row may see nothing in a visited tile (packed documents): keep the exponent finite so that exp2(-inf) = 0
      const float m_exp = (m_used == -INFINITY) ? 0.f : m_used;
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int e = 0; e < 32; e += 2) {
          const float p0 = ex2(fmaf(__uint_as_float(sv[c][e]), p.scale_log2, -m_exp));      // -inf -> 0
          const float p1 = ex2(fmaf(__uint_as_float(sv[c][e + 1]), p.scale_log2, -m_exp));
          rowsum += p0 + p1;
          preg[c * 16 + e / 2] = pack_bf16(p0, p1);
        }
      l = l * alpha + rowsum;
      if (x == 0) LX_TR(tr_cta, jb_x + i, 7);
      if (i > 0) {
        mbar_wait(&pv_done[x], (i - 1) & 1);  // O stable
        tc_fence_after();
        if (x == 0) LX_TR(tr_cta, jb_x + i, 8);
        if (__any_sync(0xffffffffu, alpha != 1.f)) {
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(tO + c * 32, v);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * alpha);
            tmem_st_32x32(tO + c * 32, v);
          }
          tmem_wait_st();
        }
      }
      {
        // P (bf16 pairs) -> TMEM, over the first 64 columns of the score tile this row was just read from
        uint32_t(&p0)[32] = *reinterpret_cast<uint32_t(*)[32]>(&preg[0]);
        uint32_t(&p1)[32] = *reinterpret_cast<uint32_t(*)[32]>(&preg[32]);
        tmem_st_32x32(tS, p0);
        tmem_st_32x32(tS + 32, p1);
        tmem_wait_st();
      }
      if (x == 0) LX_TR(tr_cta, jb_x + i, 9);
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(&p_full[x]);
    }
    // epilogue
    if (n_kv > 0) {
      mbar_wait(&pv_done[x], (n_kv - 1) & 1);
      tc_fence_after();
      const float inv_l = 1.f / l;
      const bool row_ok = q < p.S;
      __nv_bfloat16* orow = p.o + ((int64_t)b * p.S + q) * p.ldo + (int64_t)h * kD;
#pragma unroll 1
      for (int c = 0; c < kD / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(tO + c * 32, v);
        tmem_wait_ld();
        if (row_ok) {
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            uint4 o4;
            o4.x = pack_bf16(__uint_as_float(v[e]) * inv_l, __uint_as_float(v[e + 1]) * inv_l);
            o4.y = pack_bf16(__uint_as_float(v[e + 2]) * inv_l, __uint_as_float(v[e + 3]) * inv_l);
            o4.z = pack_bf16(__uint_as_float(v[e + 4]) * inv_l, __uint_as_float(v[e + 5]) * inv_l);
            o4.w = pack_bf16(__uint_as_float(v[e + 6]) * inv_l, __uint_as_float(v[e + 7]) * inv_l);
            stg_v4(orow + c * 32 + e, o4);
          }
        }
      }
      if (row_ok) p.lse[((int64_t)b * p.Hq + h) * p.S + q] = (m_used + log2f(l)) * kLn2;
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<1>(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// Forward v3: two query tiles per CTA as above, but every score row is shared by TWO threads (column halves), i.e. four
// softmax warpgroups per CTA. Measured (tools/xu_bench.cu, profiles/r2_xu_bench.txt): one warp issues a MUFU.EX2 at most
// every 8 cycles, while two warps on the same scheduler together reach one per ~5.5 cycles — a thread-per-row softmax is
// bound by its own 128 dependent-free ex2 (>= 1024 cycles per tile) no matter how idle the XU pipe is, and that softmax
// sits on the serial chain S(j) -> softmax(j) -> PV(j) -> S(j+1) of its tile (P aliases S in TMEM, so the chain cannot
// be broken), which is what paces the kernel: 4250 cycles per pair of tiles against 2728 cycles of MMA work.
// With 64 columns per thread the per-warp ex2 floor halves, four warps per scheduler fill the XU pipe, the O rescale and
// the epilogue split by head-dim halves, and PV starts on the first 64 kv columns while the second half is still in exp.
//   row maxima / row sums of the two halves are exchanged through shared memory (double-buffered slots, one 64-thread
//   named barrier per lane quarter and tile); both halves take identical rescale decisions (same inputs).
//   TMEM (512 columns): S0 | S1 | O0 | O1; P half h (bf16 pairs, 32 columns) is written over the first 32 columns of
//   the 64 score columns its own warpgroup has just read.
// ------------------------------------------------------------------------------------------------
namespace fwd3 {
constexpr int kTile = 128;
constexpr int kTileBytes = kTile * kHD * 2;        // 32 KB
constexpr int kOffQ = 0;                           // 2 query tiles
constexpr int kOffK = kOffQ + 2 * kTileBytes;      // 2 stages
constexpr int kOffV = kOffK + 2 * kTileBytes;      // 2 stages
constexpr int kOffStat = kOffV + 2 * kTileBytes;   // exchange slots: [2 buffers][2 tiles][2 halves][128 rows] fp32
constexpr int kStatBytes = 2 * 2 * 2 * kTile * 4;
constexpr int kOffBar = kOffStat + kStatBytes;
// q_full, k full/empty[2], v full/empty[2], s_full[2 tiles], p_full[2 tiles][2 halves], pv_done[2 tiles]
constexpr int kNumBars = 1 + 4 + 4 + 2 + 4 + 2;
constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16 + 1024;
// warps 0-15: four softmax warpgroups (tile 0 halves 0, 1; tile 1 halves 0, 1); warp 16: TMA producer + TMEM allocator;
// warp 17: MMA issuer. 18 warps get 112 registers each straight from the launch (65536 / 576 = 113): no setmaxnreg —
// it can only trade registers inside the CTA's launch allocation, and 640 threads would start at 96 registers with
// nothing to take the 16 extra per softmax thread from but a 32-register control warpgroup (measured: spills around
// every MMA group of the issuer).
constexpr int kThreads = 576;
static_assert(kSmemBytes <= 232448, "attention forward shared memory budget");
}  // namespace fwd3

template <bool kDocs, int kD>
__global__ void __launch_bounds__(fwd3::kThreads, 1)
attn_fwd3_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                 const __grid_constant__ CUtensorMap tmV, const AttnFwdParams p) {
  using namespace fwd3;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* s_stat = reinterpret_cast<float*>(smem + kOffStat);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;
  uint64_t* k_empty = bars + 3;
  uint64_t* v_full = bars + 5;
  uint64_t* v_empty = bars + 7;
  uint64_t* s_full = bars + 9;     // [tile]
  uint64_t* p_full = bars + 11;    // [tile * 2 + half]
  uint64_t* pv_done = bars + 15;   // [tile]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);

  const int warp = threadIdx.x >> 5;
  // grid = (query heads, batch, pairs of query tiles): pairs run backwards so CTAs are dispatched longest-first
  const int pr = gridDim.z - 1 - blockIdx.z;
  const int h = blockIdx.x, b = blockIdx.y;
  const int Pb = p.prefix_b ? min(max(p.prefix_b[b], 0), p.S) : p.P;   // prefix length of this sequence
  const int hk = h / (p.Hq / p.Hkv);
  // per-tile kv tile ranges [jb_x, je_x); a tile past the end of the sequence has an empty range
  int jb_[2], je_[2];
#pragma unroll
  for (int x = 0; x < 2; ++x) {
    const int q0 = (2 * pr + x) * kTile;
    if (q0 < p.S) {
      const int kv_end = min(p.S, max(Pb, q0 + kTile));
      je_[x] = (kv_end + kTile - 1) / kTile;
      jb_[x] = kDocs ? p.doc_start[(int64_t)b * p.S + q0] / kTile : 0;
    } else {
      jb_[x] = je_[x] = 0;
    }
  }
  const bool act1 = je_[1] > jb_[1];
  const int jb = act1 ? min(jb_[0], jb_[1]) : jb_[0];
  const int je = max(je_[0], je_[1]);

  if (warp == 16 && elect_one()) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
  }
  if (warp == 17 && elect_one()) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&pv_done[i], 1);
    }
    for (int i = 0; i < 4; ++i) mbar_init(&p_full[i], 4);
    fence_mbar_init();
  }
  if (warp == 16) {
    tmem_alloc<1>(tmem_slot, 512);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= 16) {
    if (warp == 16) {
      // ------------------------------------ TMA producer ------------------------------------
      if (elect_one()) {
        mbar_expect_tx(q_full, 2 * kTileBytes);
#pragma unroll
        for (int x = 0; x < 2; ++x) {   // rows past the end of the sequence are zero-filled
          tma_load_4d(smem + kOffQ + x * kTileBytes, &tmQ, q_full, 0, h, (2 * pr + x) * kTile, b);
          tma_load_4d(smem + kOffQ + x * kTileBytes + kTileBytes / 2, &tmQ, q_full, 64, h, (2 * pr + x) * kTile, b);
        }
        for (int j = jb; j < je; ++j) {
          const int st = (j - jb) & 1;
          const uint32_t ph = ((j - jb) >> 1) & 1;
          mbar_wait(&k_empty[st], ph ^ 1);
          mbar_expect_tx(&k_full[st], kTileBytes);
          uint8_t* sk = smem + kOffK + st * kTileBytes;
          tma_load_4d(sk, &tmK, &k_full[st], 0, hk, j * kTile, b);
          tma_load_4d(sk + kTileBytes / 2, &tmK, &k_full[st], 64, hk, j * kTile, b);
          mbar_wait(&v_empty[st], ph ^ 1);
          mbar_expect_tx(&v_full[st], kTileBytes);
          uint8_t* sv = smem + kOffV + st * kTileBytes;
          tma_load_4d(sv, &tmV, &v_full[st], 0, hk, j * kTile, b);
          tma_load_4d(sv + kTileBytes / 2, &tmV, &v_full[st], 64, hk, j * kTile, b);
        }
      }
      __syncwarp();
    } else {
      // ------------------------------------ MMA issuer ------------------------------------
      if (elect_one()) {
        constexpr uint32_t idesc_s = make_idesc(1, 1, 128, 128, 0, 0);
        constexpr uint32_t idesc_pv = make_idesc(1, 1, 128, 128, 0, 1);  // B = V is MN-major
        constexpr uint32_t kHi = desc_hi(1024);
        const uint32_t loQ0 = desc_lo(smem_u32(smem + kOffQ), 16);
        const uint32_t loK0 = desc_lo(smem_u32(smem + kOffK), 16), loV0 = desc_lo(smem_u32(smem + kOffV), 16384);
        auto active = [&](int x, int j) { return j >= jb_[x] && j < je_[x]; };
        // S_x(j) = Q_x K(j)^T; releases K(j) if x is the last tile that reads it
        auto issue_s = [&](int x, int j) {
          const int st = (j - jb) & 1;
          mbar_wait(&k_full[st], ((j - jb) >> 1) & 1);
          tc_fence_after();
          const uint32_t loQ = loQ0 + x * (kTileBytes / 16), loK = loK0 + st * (kTileBytes / 16);
#pragma unroll
          for (int dh = 0; dh < 2; ++dh)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma_ss<false, 1>(tmem_base + x * 128, desc_join(loQ + dh * 1024 + ks * 2, kHi),
                                desc_join(loK + dh * 1024 + ks * 2, kHi), idesc_s, (dh | ks) != 0);
          umma_commit(&s_full[x]);
          if (x == 1 || !active(1, j)) umma_commit(&k_empty[st]);
        };
        mbar_wait(q_full, 0);
        int it[2] = {0, 0};   // iterations done per tile
#pragma unroll
        for (int x = 0; x < 2; ++x)
          if (active(x, jb)) issue_s(x, jb);
        for (int j = jb; j < je; ++j) {
          const int st = (j - jb) & 1;
#pragma unroll
          for (int x = 0; x < 2; ++x) {
            if (!active(x, j)) continue;
            if (j == jb_[x] && j != jb) issue_s(x, j);   // a tile whose document starts later than its partner's
            mbar_wait(&v_full[st], ((j - jb) >> 1) & 1);
            const uint32_t loV = loV0 + st * (kTileBytes / 16);
            // O_x += P_x V in two halves of the kv range: half hh of P comes from warpgroup hh of the tile and lives in
            // the first 32 columns of that warpgroup's 64 score columns
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              mbar_wait(&p_full[x * 2 + hh], it[x] & 1);
              tc_fence_after();
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                umma_ts_f16(tmem_base + 256 + x * 128, tmem_base + x * 128 + hh * 64 + ks * 8,
                            desc_join(loV + (hh * 64 + ks * 16) * 8, kHi), idesc_pv, (it[x] | hh | ks) != 0);
            }
            umma_commit(&pv_done[x]);
            if (x == 1 || !active(1, j)) umma_commit(&v_empty[st]);
            ++it[x];
            if (active(x, j + 1)) issue_s(x, j + 1);     // in order behind PV_x(j), which reads P from the same columns
          }
        }
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------ softmax / correction / epilogue: two warpgroups per query tile ------------
    const int wg = warp >> 2;           // 0..3
    const int x = wg >> 1;              // query tile
    const int hf = wg & 1;              // column half (scores: kv columns; O / epilogue: head-dim columns)
    const int ew = warp & 3;            // TMEM lane quarter (hardware: warp % 4)
    const int r = ew * 32 + lane_id();  // row in tile == TMEM lane
    const uint32_t lane_off = uint32_t(ew * 32) << 16;
    const int q0 = (2 * pr + x) * kTile;
    const int q = q0 + r;
    const int jb_x = x ? jb_[1] : jb_[0], je_x = x ? je_[1] : je_[0];
    const int n_kv = je_x - jb_x;
    const uint32_t tS = tmem_base + x * 128 + hf * 64 + lane_off;         // my 64 score columns (P over the first 32)
    const uint32_t tO = tmem_base + 256 + x * 128 + hf * 64 + lane_off;   // my 64 O columns
    const uint32_t bar_id = 1 + x * 4 + ew;                               // the 64 threads that share my 32 rows
    float* my_slot = s_stat + (x * 2 + hf) * kTile + r;                   // + buffer * 4 * kTile
    float* peer_slot = s_stat + (x * 2 + (hf ^ 1)) * kTile + r;
    float m_used = -INFINITY, l = 0.f;
    const int ds_row = kDocs ? p.doc_start[(int64_t)b * p.S + min(q, p.S - 1)] : 0;
    const int ds_tile = kDocs ? p.doc_start[(int64_t)b * p.S + min(q0 + kTile - 1, p.S - 1)] : 0;
    for (int i = 0; i < n_kv; ++i) {
      const int kv0 = (jb_x + i) * kTile;
      // tile needs the element test unless every (q, kv) pair is visible and in range
      const bool full_tile = (kv0 + kTile <= p.S) && ((kv0 + kTile <= Pb) || (kv0 + kTile - 1 <= q0)) && (kv0 >= ds_tile);
      mbar_wait(&s_full[x], i & 1);
      tc_fence_after();
      uint32_t sv[2][32];
      tmem_ld_32x32(tS, sv[0]);
      tmem_ld_32x32(tS + 32, sv[1]);
      tmem_wait_ld_regs(sv[0]);
      tmem_wait_ld_regs(sv[1]);
      if (!full_tile) {
        // the visible keys of a row are ONE interval of the tile's columns, [lo, lo + width): the prefix-LM mask keeps
        // kv < max(P, q + 1) (and kv < S), packed documents additionally cut the head (kv >= ds_row) — one unsigned
        // compare against a per-row constant and a select per element instead of three compares
        const int lo = kDocs ? ds_row - kv0 : 0;
        const uint32_t width = (uint32_t)max(min(p.S, max(Pb, q + 1)) - kv0 - lo, 0);
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if ((uint32_t)(hf * 64 + c * 32 + e - lo) >= width) sv[c][e] = 0xff800000u;  // -inf
      }
      float mx4[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        mx4[c] = __uint_as_float(sv[c >> 1][(c & 1) * 16]);
#pragma unroll
        for (int e = 1; e < 16; ++e) mx4[c] = fmaxf(mx4[c], __uint_as_float(sv[c >> 1][(c & 1) * 16 + e]));
      }
      float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      // row maximum over both column halves (double-buffered slot: the peer reads slot i & 1 after barrier i, my next
      // write to it is after barrier i + 1)
      my_slot[(i & 1) * 4 * kTile] = mx;
      named_bar_sync(bar_id, 64);
      mx = fmaxf(mx, peer_slot[(i & 1) * 4 * kTile]);
      const float m_tile = mx * p.scale_log2;
      float alpha = 1.f;
      if (m_tile > m_used + 8.f) {  // lazy rescale: only when the running max grows by more than 2^8
        alpha = ex2(m_used - m_tile);
        m_used = m_tile;
      }
      uint32_t preg[32];
      float rs0 = 0.f, rs1 = 0.f;
      // a row may see nothing in a visited tile (packed documents): keep the exponent finite so that exp2(-inf) = 0
      const float m_exp = (m_used == -INFINITY) ? 0.f : m_used;
#pragma unroll
      for (int c = 0; c < 2; ++c)
#pragma unroll
        for (int e = 0; e < 32; e += 2) {
          const float p0 = ex2(fmaf(__uint_as_float(sv[c][e]), p.scale_log2, -m_exp));      // -inf -> 0
          const float p1 = ex2(fmaf(__uint_as_float(sv[c][e + 1]), p.scale_log2, -m_exp));
          rs0 += p0;
          rs1 += p1;
          preg[c * 16 + e / 2] = pack_bf16(p0, p1);
        }
      l = l * alpha + (rs0 + rs1);
      if (i > 0) {
        mbar_wait(&pv_done[x], (i - 1) & 1);  // O stable
        tc_fence_after();
        if (__any_sync(0xffffffffu, alpha != 1.f)) {   // the peer warp sees the same maxima: same decision
#pragma unroll 1
          for (int c = 0; c < 2; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(tO + c * 32, v);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * alpha);
            tmem_st_32x32(tO + c * 32, v);
          }
          tmem_wait_st();
        }
      }
      tmem_st_32x32(tS, preg);   // P half (bf16 pairs) over the first 32 of my 64 score columns
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(&p_full[x * 2 + hf]);
    }
    // epilogue: row sum over both halves, then my 64 head-dim columns of O
    if (n_kv > 0) {
      float* eslot = s_stat + (n_kv & 1) * 4 * kTile;   // the buffer the last iteration did NOT use
      eslot[(x * 2 + hf) * kTile + r] = l;
      named_bar_sync(bar_id, 64);
      l += eslot[(x * 2 + (hf ^ 1)) * kTile + r];
      mbar_wait(&pv_done[x], (n_kv - 1) & 1);
      tc_fence_after();
      const float inv_l = 1.f / l;
      const bool row_ok = q < p.S;
      __nv_bfloat16* orow = p.o + ((int64_t)b * p.S + q) * p.ldo + (int64_t)h * kD + hf * 64;
      if (hf * 64 < kD) {
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(tO + c * 32, v);
          tmem_wait_ld();
          if (row_ok) {
#pragma unroll
            for (int e = 0; e < 32; e += 8) {
              uint4 o4;
              o4.x = pack_bf16(__uint_as_float(v[e]) * inv_l, __uint_as_float(v[e + 1]) * inv_l);
              o4.y = pack_bf16(__uint_as_float(v[e + 2]) * inv_l, __uint_as_float(v[e + 3]) * inv_l);
              o4.z = pack_bf16(__uint_as_float(v[e + 4]) * inv_l, __uint_as_float(v[e + 5]) * inv_l);
              o4.w = pack_bf16(__uint_as_float(v[e + 6]) * inv_l, __uint_as_float(v[e + 7]) * inv_l);
              stg_v4(orow + c * 32 + e, o4);
            }
          }
        }
      }
      if (row_ok && hf == 0) p.lse[((int64_t)b * p.Hq + h) * p.S + q] = (m_used + log2f(l)) * kLn2;
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 16) tmem_dealloc<1>(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// Forward v4: the v2 structure (two query tiles per CTA, one softmax warpgroup per tile, thread = row) with the serial
// chain of a tile cut where it can be:  S(j) -> softmax(j) -> PV(j) -> S(j+1)  cannot be broken (P aliases S in TMEM, 512
// columns are S0 | S1 | O0 | O1), and that chain — not a pipe — paces v2: 1364 cycles of the tile's own MMAs + ~2500 of
// softmax latency + hand-offs = the measured ~4250 cycles per pair of tiles, with the tensor pipe busy 64 % of the time.
//   * P is handed over in FOUR 32-column chunks, each with its own mbarrier: the two PV MMAs of a chunk run while the
//     softmax warpgroup is in the exponentials of the next chunks, so of PV only the last chunk's MMAs stay on the chain;
//   * one MMA-issuing warp PER TILE: with chunked hand-offs a single issuer thread would sit in tile 0's chunk waits
//     while tile 1's chunks are ready (head-of-line blocking); the K / V stages are released by BOTH issuers (count 2);
//   * the per-step wait on pv_done is gone: S(j) is issued behind PV(j-1) by the same thread, so s_full(j) implies it.
// ------------------------------------------------------------------------------------------------
namespace fwd4 {
constexpr int kTile = 128;
constexpr int kTileBytes = kTile * kHD * 2;        // 32 KB
constexpr int kOffQ = 0;                           // 2 query tiles
constexpr int kOffK = kOffQ + 2 * kTileBytes;      // 2 stages
constexpr int kOffV = kOffK + 2 * kTileBytes;      // 2 stages
constexpr int kOffBar = kOffV + 2 * kTileBytes;
// q_full, k full/empty[2], v full/empty[2], s_full[2 tiles], p_chunk[2 tiles][4], pv_done[2 tiles], xu_tok[2 tiles]
constexpr int kNumBars = 1 + 4 + 4 + 2 + 8 + 2 + 2;
constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16 + 1024;
constexpr int kThreads = 384;                      // warp 0 TMA, warps 1-2 MMA issue (tile 0, 1), warp 3 TMEM alloc; warpgroups 1, 2: softmax
constexpr int kRegsCtrl = 56, kRegsSoftmax = 224;  // 128 * 56 + 256 * 224 = 384 * 168
}  // namespace fwd4

template <bool kDocs, int kD, bool kAluPack, bool kStagger>
__global__ void __launch_bounds__(fwd4::kThreads, 1)
attn_fwd4_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                 const __grid_constant__ CUtensorMap tmV, const AttnFwdParams p) {
  using namespace fwd4;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;
  uint64_t* k_empty = bars + 3;
  uint64_t* v_full = bars + 5;
  uint64_t* v_empty = bars + 7;
  uint64_t* s_full = bars + 9;     // [tile]
  uint64_t* p_chunk = bars + 11;   // [tile * 4 + chunk]
  uint64_t* pv_done = bars + 19;   // [tile]
  uint64_t* xu_tok = bars + 21;    // [tile]: "tile x may run its next exp phase" (arrived on by the OTHER tile's 4 warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);

  const int warp = threadIdx.x >> 5;
#ifdef LX_ATTN_TRACE
  const bool tr_cta = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 && (threadIdx.x & 31) == 0 &&
                      (warp == 1 || warp == 2 || warp == 4 || warp == 8);
#endif
  // grid = (query heads, batch, pairs of query tiles): pairs run backwards so CTAs are dispatched longest-first
  const int pr = gridDim.z - 1 - blockIdx.z;
  const int h = blockIdx.x, b = blockIdx.y;
  const int Pb = p.prefix_b ? min(max(p.prefix_b[b], 0), p.S) : p.P;   // prefix length of this sequence
  const int hk = h / (p.Hq / p.Hkv);
  // per-tile kv tile ranges [jb_x, je_x); a tile past the end of the sequence has an empty range
  int jb_[2], je_[2];
#pragma unroll
  for (int x = 0; x < 2; ++x) {
    const int q0 = (2 * pr + x) * kTile;
    if (q0 < p.S) {
      const int kv_end = min(p.S, max(Pb, q0 + kTile));
      je_[x] = (kv_end + kTile - 1) / kTile;
      jb_[x] = kDocs ? p.doc_start[(int64_t)b * p.S + q0] / kTile : 0;
    } else {
      jb_[x] = je_[x] = 0;
    }
  }
  const bool act1 = je_[1] > jb_[1];
  const int jb = act1 ? min(jb_[0], jb_[1]) : jb_[0];
  const int je = max(je_[0], je_[1]);

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
  }
  if (warp == 1 && elect_one()) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 2);   // one commit from each tile's issuer
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 2);
      mbar_init(&s_full[i], 1);
      mbar_init(&pv_done[i], 1);
    }
    for (int i = 0; i < 8; ++i) mbar_init(&p_chunk[i], 4);
    for (int i = 0; i < 2; ++i) mbar_init(&xu_tok[i], 4);
    fence_mbar_init();
  }
  if (warp == 3) {
    tmem_alloc<1>(tmem_slot, 512);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    setmaxnreg_dec<kRegsCtrl>();
    if (warp == 0) {
      // ------------------------------------ TMA producer ------------------------------------
      if (elect_one()) {
        mbar_expect_tx(q_full, 2 * kTileBytes);
#pragma unroll
        for (int x = 0; x < 2; ++x) {   // rows past the end of the sequence are zero-filled
          tma_load_4d(smem + kOffQ + x * kTileBytes, &tmQ, q_full, 0, h, (2 * pr + x) * kTile, b);
          tma_load_4d(smem + kOffQ + x * kTileBytes + kTileBytes / 2, &tmQ, q_full, 64, h, (2 * pr + x) * kTile, b);
        }
        for (int j = jb; j < je; ++j) {
          const int st = (j - jb) & 1;
          const uint32_t ph = ((j - jb) >> 1) & 1;
          mbar_wait(&k_empty[st], ph ^ 1);
          mbar_expect_tx(&k_full[st], kTileBytes);
          uint8_t* sk = smem + kOffK + st * kTileBytes;
          tma_load_4d(sk, &tmK, &k_full[st], 0, hk, j * kTile, b);
          tma_load_4d(sk + kTileBytes / 2, &tmK, &k_full[st], 64, hk, j * kTile, b);
          mbar_wait(&v_empty[st], ph ^ 1);
          mbar_expect_tx(&v_full[st], kTileBytes);
          uint8_t* sv = smem + kOffV + st * kTileBytes;
          tma_load_4d(sv, &tmV, &v_full[st], 0, hk, j * kTile, b);
          tma_load_4d(sv + kTileBytes / 2, &tmV, &v_full[st], 64, hk, j * kTile, b);
        }
      }
      __syncwarp();
    } else if (warp <= 2) {
      // ------------------------------------ MMA issuer of tile x ------------------------------------
      // Walks EVERY kv tile of the CTA's range, also those its own query tile does not visit (causal: the first tile of a
      // pair skips the last kv tile; packed documents: later start): there it only waits for the stage and releases it,
      // so the K / V barriers always see two arrivals and neither issuer can run a stage ahead of the other.
      const int x = warp - 1;
      if (elect_one()) {
        constexpr uint32_t idesc_s = make_idesc(1, 1, 128, 128, 0, 0);
        constexpr uint32_t idesc_pv = make_idesc(1, 1, 128, 128, 0, 1);  // B = V is MN-major
        constexpr uint32_t kHi = desc_hi(1024);
        const uint32_t loQ = desc_lo(smem_u32(smem + kOffQ), 16) + x * (kTileBytes / 16);
        const uint32_t loK0 = desc_lo(smem_u32(smem + kOffK), 16), loV0 = desc_lo(smem_u32(smem + kOffV), 16384);
        const int jb_x = x ? jb_[1] : jb_[0], je_x = x ? je_[1] : je_[0];
        const uint32_t tSx = tmem_base + x * 128, tOx = tmem_base + 256 + x * 128;
        auto issue_s = [&](int j) {
          const int st = (j - jb) & 1;
          mbar_wait(&k_full[st], ((j - jb) >> 1) & 1);
          if (j >= jb_x && j < je_x) {
            tc_fence_after();
            const uint32_t loK = loK0 + st * (kTileBytes / 16);
#pragma unroll
            for (int dh = 0; dh < 2; ++dh)
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                umma_ss<false, 1>(tSx, desc_join(loQ + dh * 1024 + ks * 2, kHi), desc_join(loK + dh * 1024 + ks * 2, kHi),
                                  idesc_s, (dh | ks) != 0);
            umma_commit(&s_full[x]);
          }
          umma_commit(&k_empty[st]);
        };
        mbar_wait(q_full, 0);
        int it = 0;   // PV steps done
        issue_s(jb);
        for (int j = jb; j < je; ++j) {
          const int st = (j - jb) & 1;
          mbar_wait(&v_full[st], ((j - jb) >> 1) & 1);
          if (j >= jb_x && j < je_x) {
            const uint32_t loV = loV0 + st * (kTileBytes / 16);
            LX_TR(tr_cta, j, x * 16 + 0);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              mbar_wait(&p_chunk[x * 4 + c], it & 1);
              tc_fence_after();
              if (c == 0) LX_TR(tr_cta, j, x * 16 + 1);
#pragma unroll
              for (int k2 = 0; k2 < 2; ++k2) {
                const int ks = c * 2 + k2;   // 16 kv rows per MMA: P columns 8 ks .. 8 ks + 7, V rows 16 ks .. 16 ks + 15
                umma_ts_f16(tOx, tSx + ks * 8, desc_join(loV + ((ks >> 2) * 64 + (ks & 3) * 16) * 8, kHi), idesc_pv,
                            (it | ks) != 0);
              }
            }
            umma_commit(&pv_done[x]);
            LX_TR(tr_cta, j, x * 16 + 2);
            ++it;
          }
          umma_commit(&v_empty[st]);
          if (j + 1 < je) issue_s(j + 1);   // in order behind PV_x(j), which reads P from the same columns
        }
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------ softmax / correction / epilogue: one warpgroup per query tile ------------
    setmaxnreg_inc<kRegsSoftmax>();
    const int x = (warp - 4) >> 2;
    const int ew = warp & 3;
    const int r = ew * 32 + lane_id();  // row in tile == TMEM lane
    const uint32_t lane_off = uint32_t(ew * 32) << 16;
    const int q0 = (2 * pr + x) * kTile;
    const int q = q0 + r;
    const int jb_x = x ? jb_[1] : jb_[0], je_x = x ? je_[1] : je_[0];
    const int n_kv = je_x - jb_x;
    const uint32_t tS = tmem_base + x * 128 + lane_off;
    const uint32_t tO = tmem_base + 256 + x * 128 + lane_off;
    float m_used = -INFINITY, l = 0.f;
    const int ds_row = kDocs ? p.doc_start[(int64_t)b * p.S + min(q, p.S - 1)] : 0;
    const int ds_tile = kDocs ? p.doc_start[(int64_t)b * p.S + min(q0 + kTile - 1, p.S - 1)] : 0;
    for (int i = 0; i < n_kv; ++i) {
      const int kv0 = (jb_x + i) * kTile;
      // tile needs the element test unless every (q, kv) pair is visible and in range
      const bool full_tile = (kv0 + kTile <= p.S) && ((kv0 + kTile <= Pb) || (kv0 + kTile - 1 <= q0)) && (kv0 >= ds_tile);
      LX_TR(tr_cta, jb_x + i, x * 16 + 4);
      mbar_wait(&s_full[x], i & 1);   // also: PV(i-1) has completed (same issuing thread, in order): O is stable
      tc_fence_after();
      LX_TR(tr_cta, jb_x + i, x * 16 + 5);
      // single pass over TMEM: the whole score row (128 fp32) lives in registers
      uint32_t sv[4][32];
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld_32x32(tS + c * 32, sv[c]);
      tmem_wait_ld_regs(sv[0]);
      tmem_wait_ld_regs(sv[1]);
      tmem_wait_ld_regs(sv[2]);
      tmem_wait_ld_regs(sv[3]);
      LX_TR(tr_cta, jb_x + i, x * 16 + 6);
      if (!full_tile) {
        // the visible keys of a row are ONE interval of the tile's columns, [lo, lo + width): the prefix-LM mask keeps
        // kv < max(P, q + 1) (and kv < S), packed documents additionally cut the head (kv >= ds_row) — one unsigned
        // compare against a per-row constant and a select per element instead of three compares
        const int lo = kDocs ? ds_row - kv0 : 0;
        const uint32_t width = (uint32_t)max(min(p.S, max(Pb, q + 1)) - kv0 - lo, 0);
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if ((uint32_t)(c * 32 + e - lo) >= width) sv[c][e] = 0xff800000u;  // -inf
      }
      float mx4[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        mx4[c] = __uint_as_float(sv[c][0]);
#pragma unroll
        for (int e = 1; e < 32; ++e) mx4[c] = fmaxf(mx4[c], __uint_as_float(sv[c][e]));
      }
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      const float m_tile = mx * p.scale_log2;
      float alpha = 1.f;
      if (m_tile > m_used + 8.f) {  // lazy rescale: only when the running max grows by more than 2^8
        alpha = ex2(m_used - m_tile);
        m_used = m_tile;
      }
      if (i > 0 && __any_sync(0xffffffffu, alpha != 1.f)) {
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(tO + c * 32, v);
          tmem_wait_ld();
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * alpha);
          tmem_st_32x32(tO + c * 32, v);
        }
        tmem_wait_st();
      }
      LX_TR(tr_cta, jb_x + i, x * 16 + 7);
      // The exponentials of the two tiles share the XU pipe (16 ex2 / clk / SM = 8 cycles per warp instruction per
      // scheduler). tools/attn_trace.py: left alone, the two tiles drift INTO phase within two steps, whatever their initial
      // offset — both sit in their exp phase together (~2200 cycles each instead of ~1100 alone) and then both sit in
      // their XU-idle part together (wait for S, TMEM load, row max: ~1700 cycles): ~3900 cycles per step. A token makes
      // the exp phases mutually exclusive and strictly alternating, t0(0) t1(0) t0(1) t1(1) ..., so that one tile's
      // XU-idle part hides under the other's exponentials. Without packed documents both tiles start at kv tile 0 and
      // tile 1 has at least as many steps as tile 0, so the chain of waits is acyclic; with packed documents a tile may
      // start several kv tiles after its partner and the token could wait on a K / V stage that waits on the token: off.
      if (kStagger && !kDocs) {
        // tile 1's exp i follows tile 0's exp i (if tile 0 has one); tile 0's exp i follows tile 1's exp i - 1 (if any)
        if (x == 1 ? (i < je_[0] - jb_[0]) : (i > 0 && i - 1 < je_[1] - jb_[1])) mbar_wait(&xu_tok[x], (x == 1 ? i : i - 1) & 1);
      }
      float m_exp = (m_used == -INFINITY) ? 0.f : m_used;
      asm volatile("" : "+f"(m_exp));   // pins the exponentials behind the wait (they are pure: ptxas hoists them otherwise)
      // (a row may see nothing in a visited tile (packed documents): m_exp keeps the exponent finite, exp2(-inf) = 0)
      float rowsum = 0.f;   // same summation order as v2 (packed-document masks run on v2): bit-identical outputs
      // chunk c: exponentials of kv columns 32 c .. 32 c + 31 -> 16 bf16 pairs -> P columns 16 c .. 16 c + 15 (over score
      // columns this thread holds in registers). The store of chunk c completes under the exponentials of chunk c + 1.
      uint32_t pc[2][16];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
#pragma unroll
        for (int e = 0; e < 32; e += 2) {
#ifdef LX_FAKE_EXP   // what-if build (tools only): no MUFU in the loop, results are meaningless
          const float p0 = fmaf(__uint_as_float(sv[c][e]), p.scale_log2, -m_exp);
          const float p1 = fmaf(__uint_as_float(sv[c][e + 1]), p.scale_log2, -m_exp);
#else
          const float p0 = ex2(fmaf(__uint_as_float(sv[c][e]), p.scale_log2, -m_exp));      // -inf -> 0
          const float p1 = ex2(fmaf(__uint_as_float(sv[c][e + 1]), p.scale_log2, -m_exp));
#endif
          rowsum += p0 + p1;
          pc[c & 1][e / 2] = kAluPack ? pack_bf16_alu(p0, p1) : pack_bf16(p0, p1);
        }
        if (c > 0) {   // chunk c - 1 is in TMEM: hand it to the issuer
          tmem_wait_st();
          tc_fence_before();
          __syncwarp();
          if (lane_id() == 0) mbar_arrive(&p_chunk[x * 4 + c - 1]);
          if (c == 1) LX_TR(tr_cta, jb_x + i, x * 16 + 8);
        }
        tmem_st_32x16(tS + c * 16, pc[c & 1]);
      }
      if (kStagger && !kDocs) {   // exponentials done: the other tile may start its own
        __syncwarp();
        if (lane_id() == 0) mbar_arrive(&xu_tok[x ^ 1]);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(&p_chunk[x * 4 + 3]);
      LX_TR(tr_cta, jb_x + i, x * 16 + 9);
      l = l * alpha + rowsum;
    }
    // epilogue
    if (n_kv > 0) {
      mbar_wait(&pv_done[x], (n_kv - 1) & 1);
      tc_fence_after();
      const float inv_l = 1.f / l;
      const bool row_ok = q < p.S;
      __nv_bfloat16* orow = p.o + ((int64_t)b * p.S + q) * p.ldo + (int64_t)h * kD;
#pragma unroll 1
      for (int c = 0; c < kD / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(tO + c * 32, v);
        tmem_wait_ld();
        if (row_ok) {
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            uint4 o4;
            o4.x = pack_bf16(__uint_as_float(v[e]) * inv_l, __uint_as_float(v[e + 1]) * inv_l);
            o4.y = pack_bf16(__uint_as_float(v[e + 2]) * inv_l, __uint_as_float(v[e + 3]) * inv_l);
            o4.z = pack_bf16(__uint_as_float(v[e + 4]) * inv_l, __uint_as_float(v[e + 5]) * inv_l);
            o4.w = pack_bf16(__uint_as_float(v[e + 6]) * inv_l, __uint_as_float(v[e + 7]) * inv_l);
            stg_v4(orow + c * 32 + e, o4);
          }
        }
      }
      if (row_ok) p.lse[((int64_t)b * p.Hq + h) * p.S + q] = (m_used + log2f(l)) * kLn2;
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 3) tmem_dealloc<1>(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// Forward v5 = v4 made PERSISTENT. One CTA per SM walks a static, length-balanced list of work items (pair of query
// tiles, head, sequence) and every ring — K / V stages, the S / P / O hand-offs, the XU token — keeps running across
// items, so that of an item's fixed cost only the O drain stays exposed:
//   * v4 pays per item (= per CTA): launch, barrier init, TMEM allocation, then Q and the first K from global memory and
//     the first S MMA before any softmax can start (~2400 cycles, tools/attn_trace.py), and at the end one tile alone in
//     its last step, the O drain and the tear-down — ~8-12k cycles on items that average ~9 steps of ~3550 cycles at
//     S = 2048 causal (13.8 items per SM): a quarter of the kernel;
//   * here the producer loads the next item's Q as soon as both issuers have committed the item's last S MMA (q_empty),
//     its K / V follow through the ring, and each issuer puts S(0) of the next item right behind its last PV: the next
//     item's first scores are in TMEM while the softmax warpgroup still normalises and stores O. The first PV of the next
//     item (accumulate = 0) needs that warpgroup's first P chunk, which it only produces after its O reads: no extra
//     hand-shake for O.
// Items are ordered longest first (pairs from the end of the sequence, heads of one kv head adjacent) and dealt to the
// CTAs in boustrophedon order (round r forwards, round r + 1 backwards), which levels the per-CTA sums of a monotone
// length list to within one step without a work counter. XU-token arrivals are made conditional so that every arrival
// has exactly one wait (v4 leaves unmatched arrivals behind at the end of a CTA; here the barrier lives on).
// Packed-document masks stay on v2 (the token's wait chain is only acyclic when both tiles start at kv tile 0).
// ------------------------------------------------------------------------------------------------
namespace fwd5 {
using namespace fwd4;   // same shared-memory layout, thread roles and register split
constexpr int kNumBars5 = fwd4::kNumBars + 1 + 2;   // + q_empty, + a second pair of XU-token barriers
constexpr int kSmemBytes5 = fwd4::kOffBar + kNumBars5 * 8 + 16 + 1024;
}  // namespace fwd5

template <int kD>
__global__ void __launch_bounds__(fwd4::kThreads, 1)
attn_fwd5_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                 const __grid_constant__ CUtensorMap tmV, const AttnFwdParams p, int n_pairs) {
  using namespace fwd5;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;
  uint64_t* k_empty = bars + 3;
  uint64_t* v_full = bars + 5;
  uint64_t* v_empty = bars + 7;
  uint64_t* s_full = bars + 9;     // [tile]
  uint64_t* p_chunk = bars + 11;   // [tile * 4 + chunk]
  uint64_t* pv_done = bars + 19;   // [tile]
  // XU token [item parity][tile]: consecutive items use different barriers. Within an item a tile is never more than one
  // arrival ahead of the other tile's waits, but tile 0 finishes an item one step before tile 1 and its first arrival of
  // the next item could otherwise land on a barrier whose previous phase tile 1 has not waited for yet (parity alias).
  // A tile cannot start item n + 2 before the other has finished item n (q_empty), so two sets are enough.
  uint64_t* xu_tok = bars + 21;
  uint64_t* q_empty = bars + 25;   // both issuers have committed the item's last S MMA: the Q tiles may be overwritten
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars5);

  const int warp = threadIdx.x >> 5;
  const int heads_per_kv = p.Hq / p.Hkv;
  const int per_pair = p.B * p.Hq;            // items per pair index
  const int n_items = n_pairs * per_pair;
  const int G = gridDim.x;

  // item of round r for this CTA; -1 past the end. Rounds alternate direction (see above).
  auto item_of = [&](int r) {
    const int k = r * G + ((r & 1) ? (G - 1 - (int)blockIdx.x) : (int)blockIdx.x);
    return k < n_items ? k : -1;
  };
  // kv tile ranges of an item's two query tiles: [0, je_x); a tile past the end of the sequence has je_x = 0
  struct Item { int pr, b, h, je0, je1, je, Pb; };
  auto decode = [&](int k) {
    Item it;
    it.pr = n_pairs - 1 - k / per_pair;
    const int rem = k % per_pair;
    it.b = rem / p.Hq;
    it.h = rem % p.Hq;
    it.Pb = p.prefix_b ? min(max(p.prefix_b[it.b], 0), p.S) : p.P;
    int je[2];
#pragma unroll
    for (int x = 0; x < 2; ++x) {
      const int q0 = (2 * it.pr + x) * kTile;
      je[x] = q0 < p.S ? (min(p.S, max(it.Pb, q0 + kTile)) + kTile - 1) / kTile : 0;
    }
    it.je0 = je[0]; it.je1 = je[1]; it.je = max(je[0], je[1]);
    return it;
  };

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
  }
  if (warp == 1 && elect_one()) {
    mbar_init(q_full, 1);
    mbar_init(q_empty, 2);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 2);   // one commit from each tile's issuer
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 2);
      mbar_init(&s_full[i], 1);
      mbar_init(&pv_done[i], 1);
    }
    for (int i = 0; i < 8; ++i) mbar_init(&p_chunk[i], 4);
    for (int i = 0; i < 4; ++i) mbar_init(&xu_tok[i], 4);
    fence_mbar_init();
  }
  if (warp == 3) {
    tmem_alloc<1>(tmem_slot, 512);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    setmaxnreg_dec<kRegsCtrl>();
    if (warp == 0) {
      // ------------------------------------ TMA producer ------------------------------------
      if (elect_one()) {
        uint32_t kvc = 0;   // K / V stages filled so far (ring position across items)
        for (int r = 0;; ++r) {
          const int k = item_of(r);
          if (k < 0) break;
          const Item it = decode(k);
          const int hk = it.h / heads_per_kv;
          mbar_wait(q_empty, (r & 1) ^ 1);   // the previous item's last S MMAs have read Q (first item: passes)
          mbar_expect_tx(q_full, 2 * kTileBytes);
#pragma unroll
          for (int x = 0; x < 2; ++x) {   // rows past the end of the sequence are zero-filled
            tma_load_4d(smem + kOffQ + x * kTileBytes, &tmQ, q_full, 0, it.h, (2 * it.pr + x) * kTile, it.b);
            tma_load_4d(smem + kOffQ + x * kTileBytes + kTileBytes / 2, &tmQ, q_full, 64, it.h, (2 * it.pr + x) * kTile, it.b);
          }
          for (int j = 0; j < it.je; ++j, ++kvc) {
            const int st = kvc & 1;
            const uint32_t ph = (kvc >> 1) & 1;
            mbar_wait(&k_empty[st], ph ^ 1);
            mbar_expect_tx(&k_full[st], kTileBytes);
            uint8_t* sk = smem + kOffK + st * kTileBytes;
            tma_load_4d(sk, &tmK, &k_full[st], 0, hk, j * kTile, it.b);
            tma_load_4d(sk + kTileBytes / 2, &tmK, &k_full[st], 64, hk, j * kTile, it.b);
            mbar_wait(&v_empty[st], ph ^ 1);
            mbar_expect_tx(&v_full[st], kTileBytes);
            uint8_t* sv = smem + kOffV + st * kTileBytes;
            tma_load_4d(sv, &tmV, &v_full[st], 0, hk, j * kTile, it.b);
            tma_load_4d(sv + kTileBytes / 2, &tmV, &v_full[st], 64, hk, j * kTile, it.b);
          }
        }
      }
      __syncwarp();
    } else if (warp <= 2) {
      // ------------------------------------ MMA issuer of tile x ------------------------------------
      // Walks EVERY kv tile of the item, also the one its own query tile does not visit (causal: the first tile of a pair
      // skips the last kv tile): there it only waits for the stage and releases it, so the K / V barriers always see two
      // arrivals and neither issuer can run a stage ahead of the other.
      const int x = warp - 1;
      if (elect_one()) {
        constexpr uint32_t idesc_s = make_idesc(1, 1, 128, 128, 0, 0);
        constexpr uint32_t idesc_pv = make_idesc(1, 1, 128, 128, 0, 1);  // B = V is MN-major
        constexpr uint32_t kHi = desc_hi(1024);
        const uint32_t loQ = desc_lo(smem_u32(smem + kOffQ), 16) + x * (kTileBytes / 16);
        const uint32_t loK0 = desc_lo(smem_u32(smem + kOffK), 16), loV0 = desc_lo(smem_u32(smem + kOffV), 16384);
        const uint32_t tSx = tmem_base + x * 128, tOx = tmem_base + 256 + x * 128;
        uint32_t kc = 0, vc = 0;   // K / V stages consumed so far
        uint32_t pvc = 0;          // PV steps issued so far (phase of the P-chunk barriers)
        for (int r = 0;; ++r) {
          const int k = item_of(r);
          if (k < 0) break;
          const Item it = decode(k);
          const int je_x = x ? it.je1 : it.je0;
          auto issue_s = [&](int j) {
            const int st = kc & 1;
            mbar_wait(&k_full[st], (kc >> 1) & 1);
            ++kc;
            if (j < je_x) {
              tc_fence_after();
              const uint32_t loK = loK0 + st * (kTileBytes / 16);
#pragma unroll
              for (int dh = 0; dh < 2; ++dh)
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                  umma_ss<false, 1>(tSx, desc_join(loQ + dh * 1024 + ks * 2, kHi), desc_join(loK + dh * 1024 + ks * 2, kHi),
                                    idesc_s, (dh | ks) != 0);
              umma_commit(&s_full[x]);
            }
            umma_commit(&k_empty[st]);
            // the item's last K tile: once these MMAs (and, in order, all earlier ones) are done Q is no longer needed
            if (j == it.je - 1) umma_commit(q_empty);
          };
          mbar_wait(q_full, r & 1);
          issue_s(0);
          for (int j = 0; j < it.je; ++j) {
            const int st = vc & 1;
            mbar_wait(&v_full[st], (vc >> 1) & 1);
            ++vc;
            if (j < je_x) {
              const uint32_t loV = loV0 + st * (kTileBytes / 16);
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                mbar_wait(&p_chunk[x * 4 + c], pvc & 1);
                tc_fence_after();
#pragma unroll
                for (int k2 = 0; k2 < 2; ++k2) {
                  const int ks = c * 2 + k2;   // 16 kv rows per MMA: P columns 8 ks .. 8 ks + 7, V rows 16 ks .. 16 ks + 15
                  umma_ts_f16(tOx, tSx + ks * 8, desc_join(loV + ((ks >> 2) * 64 + (ks & 3) * 16) * 8, kHi), idesc_pv,
                              (j | ks) != 0);
                }
              }
              umma_commit(&pv_done[x]);
              ++pvc;
            }
            umma_commit(&v_empty[st]);
            if (j + 1 < it.je) issue_s(j + 1);   // in order behind PV_x(j), which reads P from the same columns
          }
        }
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------ softmax / correction / epilogue: one warpgroup per query tile ------------
    setmaxnreg_inc<kRegsSoftmax>();
    const int x = (warp - 4) >> 2;
    const int ew = warp & 3;
    const int rr = ew * 32 + lane_id();  // row in tile == TMEM lane
    const uint32_t lane_off = uint32_t(ew * 32) << 16;
    const uint32_t tS = tmem_base + x * 128 + lane_off;
    const uint32_t tO = tmem_base + 256 + x * 128 + lane_off;
    uint32_t sc = 0;             // s_full waits done (= steps of this tile so far, over all items)
    uint32_t tokw[2] = {0, 0};   // XU-token waits done, per barrier set
    for (int r = 0;; ++r) {
      const int k = item_of(r);
      if (k < 0) break;
      const Item it = decode(k);
      const int n0 = it.je0, n1 = it.je1;
      const int n_kv = x ? n1 : n0;
      const int q0 = (2 * it.pr + x) * kTile;
      const int q = q0 + rr;
      const int Pb = it.Pb;
      float m_used = -INFINITY, l = 0.f;
      for (int i = 0; i < n_kv; ++i) {
        const int kv0 = i * kTile;
        // tile needs the element test unless every (q, kv) pair is visible and in range
        const bool full_tile = (kv0 + kTile <= p.S) && ((kv0 + kTile <= Pb) || (kv0 + kTile - 1 <= q0));
        mbar_wait(&s_full[x], sc & 1);   // also: PV(i-1) has completed (same issuing thread, in order): O is stable
        ++sc;
        tc_fence_after();
        uint32_t sv[4][32];
#pragma unroll
        for (int c = 0; c < 4; ++c) tmem_ld_32x32(tS + c * 32, sv[c]);
        tmem_wait_ld_regs(sv[0]);
        tmem_wait_ld_regs(sv[1]);
        tmem_wait_ld_regs(sv[2]);
        tmem_wait_ld_regs(sv[3]);
        if (!full_tile) {
          // the visible keys of a row are the first `width` columns of the tile: kv < max(P, q + 1) and kv < S
          const uint32_t width = (uint32_t)max(min(p.S, max(Pb, q + 1)) - kv0, 0);
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if ((uint32_t)(c * 32 + e) >= width) sv[c][e] = 0xff800000u;  // -inf
        }
        float mx4[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          mx4[c] = __uint_as_float(sv[c][0]);
#pragma unroll
          for (int e = 1; e < 32; ++e) mx4[c] = fmaxf(mx4[c], __uint_as_float(sv[c][e]));
        }
        const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
        const float m_tile = mx * p.scale_log2;
        float alpha = 1.f;
        if (m_tile > m_used + 8.f) {  // lazy rescale: only when the running max grows by more than 2^8
          alpha = ex2(m_used - m_tile);
          m_used = m_tile;
        }
        if (i > 0 && __any_sync(0xffffffffu, alpha != 1.f)) {
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(tO + c * 32, v);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * alpha);
            tmem_st_32x32(tO + c * 32, v);
          }
          tmem_wait_st();
        }
        // XU token (see v4): within an item the exp phases alternate t0(0) t1(0) t0(1) t1(1) ...; tile 1's exp i follows
        // tile 0's exp i (if tile 0 has one), tile 0's exp i follows tile 1's exp i - 1. Every arrival below has exactly
        // one wait here, so the barrier phases can be counted across items.
        if (x == 1 ? (i < n0) : (i > 0 && i - 1 < n1)) {
          mbar_wait(&xu_tok[(r & 1) * 2 + x], tokw[r & 1] & 1);
          ++tokw[r & 1];
        }
        float m_exp = (m_used == -INFINITY) ? 0.f : m_used;
        asm volatile("" : "+f"(m_exp));   // pins the exponentials behind the wait (they are pure: ptxas hoists them otherwise)
        float rowsum = 0.f;
        uint32_t pc[2][16];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const float p0 = ex2(fmaf(__uint_as_float(sv[c][e]), p.scale_log2, -m_exp));      // -inf -> 0
            const float p1 = ex2(fmaf(__uint_as_float(sv[c][e + 1]), p.scale_log2, -m_exp));
            rowsum += p0 + p1;
            pc[c & 1][e / 2] = pack_bf16(p0, p1);
          }
          if (c > 0) {   // chunk c - 1 is in TMEM: hand it to the issuer
            tmem_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane_id() == 0) mbar_arrive(&p_chunk[x * 4 + c - 1]);
          }
          tmem_st_32x16(tS + c * 16, pc[c & 1]);
        }
        // exponentials done: the other tile may start the exp phase that waits for this one (if it has such a step)
        if (x == 0 ? (i < n1) : (i + 1 < n0)) {
          __syncwarp();
          if (lane_id() == 0) mbar_arrive(&xu_tok[(r & 1) * 2 + (x ^ 1)]);
        }
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane_id() == 0) mbar_arrive(&p_chunk[x * 4 + 3]);
        l = l * alpha + rowsum;
      }
      // epilogue of the item: the issuer is already past S(0) of the next one
      if (n_kv > 0) {
        mbar_wait(&pv_done[x], (sc - 1) & 1);   // PV steps == S steps of this tile
        tc_fence_after();
        const float inv_l = 1.f / l;
        const bool row_ok = q < p.S;
        __nv_bfloat16* orow = p.o + ((int64_t)it.b * p.S + q) * p.ldo + (int64_t)it.h * kD;
#pragma unroll 1
        for (int c = 0; c < kD / 32; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(tO + c * 32, v);
          tmem_wait_ld();
          if (row_ok) {
#pragma unroll
            for (int e = 0; e < 32; e += 8) {
              uint4 o4;
              o4.x = pack_bf16(__uint_as_float(v[e]) * inv_l, __uint_as_float(v[e + 1]) * inv_l);
              o4.y = pack_bf16(__uint_as_float(v[e + 2]) * inv_l, __uint_as_float(v[e + 3]) * inv_l);
              o4.z = pack_bf16(__uint_as_float(v[e + 4]) * inv_l, __uint_as_float(v[e + 5]) * inv_l);
              o4.w = pack_bf16(__uint_as_float(v[e + 6]) * inv_l, __uint_as_float(v[e + 7]) * inv_l);
              stg_v4(orow + c * 32 + e, o4);
            }
          }
        }
        if (row_ok) p.lse[((int64_t)it.b * p.Hq + it.h) * p.S + q] = (m_used + log2f(l)) * kLn2;
        tc_fence_before();
      }
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 3) tmem_dealloc<1>(tmem_base, 512);
}

// ================================================================================================
// backward
// ================================================================================================
struct AttnBwdParams {
  const float* lse;    // [B, Hq, S]
  const float* delta;  // [B, Hq, S]
  float* dq_accum;     // [B, Hq, S, D] fp32 (tile-contiguous for the bulk reduce)
  __nv_bfloat16* dk;
  int64_t lddk;
  __nv_bfloat16* dv;
  int64_t lddv;
  int B, S, Hq, Hkv, P;
  int D;  // real head dim (64 or 128)
  float scale, scale_log2;
  const int32_t* doc_start;  // [B, S] or null (packed-sequence document-causal mask)
  const int32_t* doc_end;    // [B, S] last position of the document containing each position
  const float* rope;         // null, or [>= S, D/2, 2] (cos, sin): dk (here) and dq (convert kernel) get the RoPE backward
  const int32_t* prefix_b;   // null, or [B]: per-sequence prefix length (overrides P)
};

namespace bwd {
constexpr int kKV = 128;                          // kv rows per CTA
constexpr int kQ = 128;                           // query rows per step
// warpgroup 0: control (warp 0 TMA, warp 1 MMA issue, warp 2 TMEM alloc); warpgroups 1-2: softmax-grad workers;
// warpgroup 3: dQ drain (TMEM -> fp32 smem tile -> bulk reduce-add)
constexpr int kThreads = 512;
constexpr int kThreadsNoDQ = 384;                 // attn_bwd_kernel<.., kNoDQ = true>: no drain warpgroup
constexpr int kWorkers = 256;
constexpr int kRegsCtrl = 64, kRegsWork = 144, kRegsDrain = 160;   // setmaxnreg: 64 + 2 * 144 + 160 = 4 * 128
constexpr int kTileBytes = 128 * kHD * 2;         // 32 KB: two 16 KB boxes of [128 rows x 128 B]
constexpr int kOffK = 0;
constexpr int kOffV = kOffK + kTileBytes;
constexpr int kOffQ = kOffV + kTileBytes;         // 2 stages (Q(s) lives from S^T(s) to dK(s), across S^T(s+1))
constexpr int kOffdO = kOffQ + 2 * kTileBytes;    // 1 stage  (dO(s): dP^T(s) and dV(s) are adjacent in the MMA order)
constexpr int kOffdS = kOffdO + kTileBytes;       // dS^T [128 kv][128 q] bf16: two boxes (q halves) of [128 x 128 B]
constexpr int kOffdQ = kOffdS + kTileBytes;       // fp32 [32 q][128 d] staging for the bulk reduce-add
constexpr int kStageRows = 32;
constexpr int kdQBytes = kStageRows * kHD * 4;    // 16 KB
constexpr int kOffStat = kOffdQ + kdQBytes;       // lse2 / delta*scale / doc_start: 2 buffers x 3 x 128 words
constexpr int kOffBar = kOffStat + 2 * 3 * kQ * 4;
// kv_full, q full/empty[2], do full/empty, s_full, p_full, dp_full, ds_full, dq full/empty, acc_done
constexpr int kNumBars = 1 + 4 + 2 + 4 + 2 + 1;
constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16 + 1024;
static_assert(kSmemBytes <= 232448, "attention backward shared memory budget");
// TMEM columns: dV, dK accumulators; X = S^T, then P^T as bf16 pairs over the columns each warp read;
// Y = dP^T, then dQ^T
constexpr int kColdV = 0, kColdK = 128, kColX = 256, kColY = 384;
}  // namespace bwd

// Backward v5. Every tcgen05.mma of this kernel is 128 x 128 x 16: measured with tools/attn_trace.py, an SS-mode MMA with
// M = 128 occupies the tensor pipe for >= 64 cycles whatever N is (the A-operand smem read), so the 64-query-row steps of
// the previous version (N = 64 for S^T, dP^T, dQ^T) ran the pipe at half rate and were MMA-issue bound at ~2950 cycles
// per 64 rows. With 128-row steps the five GEMMs need all 512 TMEM columns twice over, hence the aliasing:
//   X: S^T(s) -> workers -> P^T(s) bf16 (A operand of dV, read straight from TMEM) -> S^T(s+1) once dV(s) has run
//   Y: dP^T(s) -> workers -> dQ^T(s) -> drain warps -> dP^T(s+1)
// MMA issue order per step:  dV(s), S^T(s+1) | dQ^T(s), dK(s) | dP^T(s+1)
//   workers compute dS(s) under dV(s)/S^T(s+1), P(s+1) under dQ^T(s)/dK(s)/dP^T(s+1); the drain pulls dQ^T(s) into
//   registers under dK(s), so the pipe only waits on semaphores that have normally fired already.
// kNoDQ (deterministic mode): dQ^T(s) is neither computed nor drained — attn_bwd_dq_kernel produces dQ without atomics —
// and dP^T(s+1) waits only for dS^T(s); dV and dK accumulate in the same MMA order, so they are bitwise those of the
// default instantiation. Without the drain warpgroup the CTA has 384 threads and no setmaxnreg rebalancing (the 168
// registers a thread gets need no spills).
template <bool kDocs, int kD, bool kNoDQ = false>
__global__ void __launch_bounds__(kNoDQ ? bwd::kThreadsNoDQ : bwd::kThreads, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdO,
                const AttnBwdParams p) {
  using namespace bwd;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* s_stat = reinterpret_cast<float*>(smem + kOffStat);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* kv_full = bars;
  uint64_t* q_full = bars + 1;     // [2]
  uint64_t* q_empty = bars + 3;    // [2]
  uint64_t* do_full = bars + 5;
  uint64_t* do_empty = bars + 6;
  uint64_t* s_full = bars + 7;
  uint64_t* p_full = bars + 8;
  uint64_t* dp_full = bars + 9;
  uint64_t* ds_full = bars + 10;
  uint64_t* dq_full = bars + 11;
  uint64_t* dq_empty = bars + 12;
  uint64_t* acc_done = bars + 13;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);

  const int warp = threadIdx.x >> 5;
  // grid = (kv heads, kv tiles, batch): within a batch element CTAs are dispatched longest-first (tile 0 is visited by
  // every query tile, the last tile only by the last one); batch elements follow one another so that the fp32 dQ
  // accumulator being reduced into stays L2-resident (one element = 33 MB at 8B shape, S = 2048)
  const int hk = blockIdx.x, jt = blockIdx.y, b = blockIdx.z;
  const int Pb = p.prefix_b ? min(max(p.prefix_b[b], 0), p.S) : p.P;   // prefix length of this sequence
#ifdef LX_ATTN_TRACE
  const bool tr_cta = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 && (threadIdx.x & 31) == 0 &&
                      (warp == 1 || warp == 4 || warp == 12);
#endif
  const int kv0 = jt * kKV;
  const int G = p.Hq / p.Hkv;
  const int nq_tiles = (p.S + kQ - 1) / kQ;
  const int i_start = (kv0 < Pb) ? 0 : kv0 / kQ;  // first query tile that sees this kv tile
  // packed documents: queries after the end of the last kv row's document never see this tile
  const int i_end = kDocs ? min(nq_tiles, p.doc_end[(int64_t)b * p.S + min(kv0 + kKV - 1, p.S - 1)] / kQ + 1) : nq_tiles;
  const int steps_per_head = i_end - i_start;
  const int n_steps = G * steps_per_head;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmdO);
  }
  if (warp == 1 && elect_one()) {
    mbar_init(kv_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
    }
    mbar_init(do_full, 1);
    mbar_init(do_empty, 1);
    mbar_init(s_full, 1);
    mbar_init(p_full, 8);
    mbar_init(dp_full, 1);
    mbar_init(ds_full, 8);
    mbar_init(dq_full, 1);
    mbar_init(dq_empty, 4);
    mbar_init(acc_done, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<1>(tmem_slot, 512);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    if constexpr (!kNoDQ) setmaxnreg_dec<kRegsCtrl>();
    if (warp == 0) {
      // ------------------------------------ TMA producer ------------------------------------
      if (elect_one()) {
        mbar_expect_tx(kv_full, 2 * kTileBytes);
        tma_load_4d(smem + kOffK, &tmK, kv_full, 0, hk, kv0, b);
        tma_load_4d(smem + kOffK + kTileBytes / 2, &tmK, kv_full, 64, hk, kv0, b);
        tma_load_4d(smem + kOffV, &tmV, kv_full, 0, hk, kv0, b);
        tma_load_4d(smem + kOffV + kTileBytes / 2, &tmV, kv_full, 64, hk, kv0, b);
        for (int s = 0; s < n_steps; ++s) {
          const int st = s & 1;
          const int hq = hk * G + s / steps_per_head;
          const int q0 = (i_start + s % steps_per_head) * kQ;
          mbar_wait(&q_empty[st], ((s >> 1) & 1) ^ 1);     // dK(s-2) has read Q[st]
          mbar_expect_tx(&q_full[st], kTileBytes);
          uint8_t* sq = smem + kOffQ + st * kTileBytes;
          tma_load_4d(sq, &tmQ, &q_full[st], 0, hq, q0, b);
          tma_load_4d(sq + kTileBytes / 2, &tmQ, &q_full[st], 64, hq, q0, b);
          mbar_wait(do_empty, (s & 1) ^ 1);                // dV(s-1) has read dO
          mbar_expect_tx(do_full, kTileBytes);
          uint8_t* sdo = smem + kOffdO;
          tma_load_4d(sdo, &tmdO, do_full, 0, hq, q0, b);
          tma_load_4d(sdo + kTileBytes / 2, &tmdO, do_full, 64, hq, q0, b);
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ------------------------------------ MMA issuer ------------------------------------
      if (elect_one()) {
        constexpr uint32_t idesc_st = make_idesc(1, 1, 128, 128, 0, 0);   // S^T, dP^T : [kv x d] . [q x d]^T
        constexpr uint32_t idesc_acc = make_idesc(1, 1, 128, 128, 0, 1);  // dV, dK    : [kv x q] . [q x d]   (B MN-major)
        constexpr uint32_t idesc_dq = make_idesc(1, 1, 128, 128, 1, 1);   // dQ^T      : [kv x d]^T . [kv x q] (A, B MN-major)
        constexpr uint32_t kHi = desc_hi(1024);
        // descriptor low words (address >> 4 | LBO): K-major operands carry LBO 16 (unused), MN-major ones the stride
        // between the two 64-element atoms of a 128-wide tile (= one 16 KB box)
        const uint32_t loK = desc_lo(smem_u32(smem + kOffK), 16), loV = desc_lo(smem_u32(smem + kOffV), 16);
        const uint32_t loKmn = desc_lo(smem_u32(smem + kOffK), 16384);
        const uint32_t loQ0 = desc_lo(smem_u32(smem + kOffQ), 16), loQmn0 = desc_lo(smem_u32(smem + kOffQ), 16384);
        const uint32_t lodO = desc_lo(smem_u32(smem + kOffdO), 16), lodOmn = desc_lo(smem_u32(smem + kOffdO), 16384);
        const uint32_t lodS = desc_lo(smem_u32(smem + kOffdS), 16), lodSmn = desc_lo(smem_u32(smem + kOffdS), 16384);
        const uint32_t tX = tmem_base + kColX, tY = tmem_base + kColY;
        // [128 x 128] += A[128 x 128 (K-major, two 64-wide boxes)] . B[128 x 128 (K-major)]^T
        auto mma_kk = [&](uint32_t d, uint32_t a_lo, uint32_t b_lo) {
#pragma unroll
          for (int dh = 0; dh < 2; ++dh)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma_ss<false, 1>(d, desc_join(a_lo + (dh * 16384 + ks * 32) / 16, kHi),
                                desc_join(b_lo + (dh * 16384 + ks * 32) / 16, kHi), idesc_st, (dh | ks) != 0);
        };
        mbar_wait(kv_full, 0);
        mbar_wait(&q_full[0], 0);
        tc_fence_after();
        mma_kk(tX, loK, loQ0);                       // S^T(0)
        umma_commit(s_full);
        mbar_wait(do_full, 0);
        tc_fence_after();
        mma_kk(tY, loV, lodO);                       // dP^T(0)
        umma_commit(dp_full);
        for (int s = 0; s < n_steps; ++s) {
          const int st = s & 1;
          const uint32_t qmn_lo = loQmn0 + st * (kTileBytes / 16);
          LX_TR(tr_cta, s, 0);
          mbar_wait(p_full, s & 1);                  // P^T(s) is in X
          tc_fence_after();
          LX_TR(tr_cta, s, 1);
          // dV += P^T dO   (A = P^T from TMEM: k-step ks covers queries 16 ks .. 16 ks + 15, written by worker group ks / 4)
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)
            umma_ts_f16(tmem_base + kColdV, tX + (ks >> 2) * 64 + (ks & 3) * 8, desc_join(lodOmn + ks * 128, kHi),
                        idesc_acc, (s | ks) != 0);
          umma_commit(do_empty);
          if (s + 1 < n_steps) {
            mbar_wait(&q_full[st ^ 1], ((s + 1) >> 1) & 1);
            tc_fence_after();
            mma_kk(tX, loK, loQ0 + (st ^ 1) * (kTileBytes / 16));   // S^T(s+1), in order behind dV(s)
            umma_commit(s_full);
          }
          LX_TR(tr_cta, s, 2);
          mbar_wait(ds_full, s & 1);                 // dS^T(s) is in smem, dP^T(s) has been read
          tc_fence_after();
          LX_TR(tr_cta, s, 3);
          if constexpr (!kNoDQ) {
            // dQ^T = K^T dS^T   (M = d, N = q, K dim = kv)
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
              umma_ss<false, 1>(tY, desc_join(loKmn + ks * 128, kHi), desc_join(lodSmn + ks * 128, kHi), idesc_dq, ks != 0);
            umma_commit(dq_full);
          }
          // dK += dS^T Q      (K dim = q: boxes of 64 queries)
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)
            umma_ss<false, 1>(tmem_base + kColdK, desc_join(lodS + ((ks >> 2) * 16384 + (ks & 3) * 32) / 16, kHi),
                              desc_join(qmn_lo + ks * 128, kHi), idesc_acc, (s | ks) != 0);
          umma_commit(&q_empty[st]);
          LX_TR(tr_cta, s, 4);
          if (s + 1 < n_steps) {
            if constexpr (!kNoDQ) mbar_wait(dq_empty, s & 1);   // the drain warps hold dQ^T(s) in registers
            mbar_wait(do_full, (s + 1) & 1);
            tc_fence_after();
            mma_kk(tY, loV, lodO);                   // dP^T(s+1)
            umma_commit(dp_full);
          }
          LX_TR(tr_cta, s, 5);
        }
        umma_commit(acc_done);
      }
      __syncwarp();
    }
  } else if (warp < 12) {
    // ------------------------------------ workers: thread = kv row, 64 query columns ------------------------------------
    if constexpr (!kNoDQ) setmaxnreg_inc<kRegsWork>();
    const int wt = threadIdx.x - 128;           // 0..255
    const int grp = (warp - 4) >> 2;            // query-column half handled by this warp
    const int lq = warp & 3;                    // TMEM lane quarter (hardware: warp % 4)
    const int t = lq * 32 + lane_id();          // kv row
    const uint32_t lane_off = uint32_t(lq * 32) << 16;
    const int kv = kv0 + t;
    const uint32_t s_stat_u = smem_u32(s_stat);
    const uint32_t tXw = tmem_base + kColX + grp * 64 + lane_off;
    const uint32_t tYw = tmem_base + kColY + grp * 64 + lane_off;
    const uint32_t sdS = smem_u32(smem + kOffdS) + grp * (kTileBytes / 2) + t * 128;

    // stats of one step: lse (wt < 128; stored in log2 units), delta (wt >= 128; stored times the softmax scale) and,
    // for packed documents, the document start of each query (loaded by wt < 128 as a second value).
    // Raw global loads only: nothing may depend on the value before it is stored a step later.
    auto load_stat = [&](int s, float& a, int& d) {
      a = 0.f; d = 0;
      if (s >= n_steps) return;
      const int hq = hk * G + s / steps_per_head;
      const int qq = (i_start + s % steps_per_head) * kQ + (wt & 127);
      const int64_t idx = ((int64_t)b * p.Hq + hq) * p.S + qq;
      if (wt < 128) {
        a = (qq < p.S) ? p.lse[idx] : INFINITY;
        if (kDocs) d = (qq < p.S) ? p.doc_start[(int64_t)b * p.S + qq] : 0;
      } else {
        a = (qq < p.S) ? p.delta[idx] : 0.f;
      }
    };
    auto store_stat = [&](int buf, float a, int d) {
      float* base = s_stat + buf * 3 * kQ;
      if (wt < 128) {
        base[wt] = a * kLog2e;
        if (kDocs) base[2 * kQ + wt] = __int_as_float(d);
      } else {
        base[wt] = a * p.scale;                   // [kQ + (wt - 128)]
      }
    };

    float nxt_a; int nxt_d;
    load_stat(0, nxt_a, nxt_d);
    store_stat(0, nxt_a, nxt_d);
    for (int s = 0; s < n_steps; ++s) {
      const int st = s & 1;
      const int q0 = (i_start + s % steps_per_head) * kQ;
      LX_TR(tr_cta, s, 6);
      named_bar_sync(1, kWorkers);               // stats of step s visible; all workers finished step s-1
      load_stat(s + 1, nxt_a, nxt_d);            // prefetch next step's stats (global)
      const uint32_t stat_u = s_stat_u + st * (3 * kQ * 4) + grp * 64 * 4;
      const int ds_tile = kDocs ? p.doc_start[(int64_t)b * p.S + min(q0 + kQ - 1, p.S - 1)] : 0;
      const bool full_tile = (kv0 + kKV <= p.S) && (q0 + kQ <= p.S) && ((kv0 + kKV <= Pb) || (kv0 + kKV - 1 <= q0)) &&
                             (kv0 >= ds_tile);
      mbar_wait(s_full, s & 1);
      tc_fence_after();
      LX_TR(tr_cta, s, 7);
      uint32_t pr[32];                           // P^T of this row: 64 queries as bf16 pairs
      {
        uint32_t sv[2][32];
        tmem_ld_32x32(tXw, sv[0]);
        tmem_ld_32x32(tXw + 32, sv[1]);
        tmem_wait_ld_regs(sv[0]);
        tmem_wait_ld_regs(sv[1]);
        LX_TR(tr_cta, s, 8);
        // prefix-LM without documents: a kv row inside the sequence is seen by every query if it lies in the prefix, else
        // by the queries q >= kv: a suffix of this thread's 64 query columns, starting at first_q (one compare per element)
        const int first_q = (kv >= p.S) ? (1 << 30) : (kv < Pb ? -(1 << 30) : kv - q0 - grp * 64);
        auto block = [&](auto masked_tag) {
          constexpr bool kMasked = decltype(masked_tag)::value;
#pragma unroll
          for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 l4 = lds_f4(stat_u + (c * 32 + i) * 4);                 // lse2 of 4 query columns
              const float ls[4] = {l4.x, l4.y, l4.z, l4.w};
              int dst4[4] = {0, 0, 0, 0};
              if (kDocs && kMasked) {
                const float4 s4 = lds_f4(stat_u + 2 * kQ * 4 + (c * 32 + i) * 4);  // document start of each query column
                dst4[0] = __float_as_int(s4.x); dst4[1] = __float_as_int(s4.y);
                dst4[2] = __float_as_int(s4.z); dst4[3] = __float_as_int(s4.w);
              }
              float pv[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                float pe = ex2(fmaf(__uint_as_float(sv[c][i + e]), p.scale_log2, -ls[e]));
                if (kMasked) {
                  if (kDocs) {
                    const int qa = q0 + grp * 64 + c * 32 + i + e;
                    if (!((kv < p.S) && ((kv < Pb) || (kv <= qa)) && kv >= dst4[e])) pe = 0.f;
                  } else if (c * 32 + i + e < first_q) {   // this kv row is visible to the queries from first_q on
                    pe = 0.f;
                  }
                }
                pv[e] = pe;
              }
              pr[c * 16 + i / 2] = pack_bf16(pv[0], pv[1]);
              pr[c * 16 + i / 2 + 1] = pack_bf16(pv[2], pv[3]);
            }
        };
        if (full_tile) block(std::false_type{});
        else block(std::true_type{});
      }
      // P^T -> the first 32 of the 64 X columns this warp has just read (no other warp touches them)
      tmem_st_32x32(tXw, pr);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(p_full);
      LX_TR(tr_cta, s, 9);

      mbar_wait(dp_full, s & 1);                 // also: dQ^T(s-1), dK(s-1) have finished reading the dS^T tile
      tc_fence_after();
      LX_TR(tr_cta, s, 10);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t dv[32], dsr[16];
        tmem_ld_32x32(tYw + c * 32, dv);
        tmem_wait_ld_regs(dv);
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 d4 = lds_f4(stat_u + kQ * 4 + (c * 32 + i) * 4);          // delta * scale
          const uint32_t p01 = pr[c * 16 + i / 2], p23 = pr[c * 16 + i / 2 + 1];
          const float ds0 = bf16_lo(p01) * fmaf(__uint_as_float(dv[i]), p.scale, -d4.x);
          const float ds1 = bf16_hi(p01) * fmaf(__uint_as_float(dv[i + 1]), p.scale, -d4.y);
          const float ds2 = bf16_lo(p23) * fmaf(__uint_as_float(dv[i + 2]), p.scale, -d4.z);
          const float ds3 = bf16_hi(p23) * fmaf(__uint_as_float(dv[i + 3]), p.scale, -d4.w);
          dsr[i / 2] = pack_bf16(ds0, ds1);
          dsr[i / 2 + 1] = pack_bf16(ds2, ds3);
        }
        // box `grp` of the dS^T tile: row t = 128 B = 8 chunks of 16 B (8 queries), swizzled by (row & 7)
#pragma unroll
        for (int cc = 0; cc < 4; ++cc)
          sts_v4(sdS + (((c * 4 + cc) ^ (t & 7)) << 4), dsr[cc * 4], dsr[cc * 4 + 1], dsr[cc * 4 + 2], dsr[cc * 4 + 3]);
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(ds_full);
      LX_TR(tr_cta, s, 11);
      store_stat(st ^ 1, nxt_a, nxt_d);          // stats of step s+1 (buffer last read in step s-1)
    }
    // write dV (group 0) / dK (group 1); thread = kv row
    mbar_wait(acc_done, 0);
    tc_fence_after();
    const bool row_ok = kv < p.S;
    __nv_bfloat16* drow = grp == 0 ? p.dv + ((int64_t)b * p.S + kv) * p.lddv + (int64_t)hk * kD
                                   : p.dk + ((int64_t)b * p.S + kv) * p.lddk + (int64_t)hk * kD;
#pragma unroll 1
    for (int c = 0; c < kD / 32; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(tmem_base + (grp == 0 ? kColdV : kColdK) + lane_off + c * 32, v);
      tmem_wait_ld_regs(v);
      if (row_ok && grp == 1 && p.rope != nullptr) {
        // dK through the RoPE backward: (g0, g1) -> (g0 c + g1 s, g1 c - g0 s) per adjacent pair, position = kv row
        const float4* cs = reinterpret_cast<const float4*>(p.rope + ((int64_t)kv * (kD / 2) + c * 16) * 2);
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 t4 = cs[i / 4];   // (c0, s0, c1, s1)
          const float g0 = __uint_as_float(v[i]), g1 = __uint_as_float(v[i + 1]);
          const float g2 = __uint_as_float(v[i + 2]), g3 = __uint_as_float(v[i + 3]);
          v[i] = __float_as_uint(g0 * t4.x + g1 * t4.y);
          v[i + 1] = __float_as_uint(g1 * t4.x - g0 * t4.y);
          v[i + 2] = __float_as_uint(g2 * t4.z + g3 * t4.w);
          v[i + 3] = __float_as_uint(g3 * t4.z - g2 * t4.w);
        }
      }
      if (row_ok) {
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          uint4 o4;
          o4.x = pack_bf16(__uint_as_float(v[i]), __uint_as_float(v[i + 1]));
          o4.y = pack_bf16(__uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
          o4.z = pack_bf16(__uint_as_float(v[i + 4]), __uint_as_float(v[i + 5]));
          o4.w = pack_bf16(__uint_as_float(v[i + 6]), __uint_as_float(v[i + 7]));
          stg_v4(drow + c * 32 + i, o4);
        }
      }
    }
    tc_fence_before();
  } else if constexpr (!kNoDQ) {
    // ------------------------------------ dQ drain (thread = head-dim element) ------------------------------------
    // TMEM dQ^T [d][128 q] -> registers (Y is released at once) -> red.global.add into dq_accum[b, hq, q0 : q0 + 128, :]
    setmaxnreg_inc<kRegsDrain>();
    const int lq = warp & 3;
    const int t = lq * 32 + lane_id();          // head-dim element == TMEM lane
    const uint32_t lane_off = uint32_t(lq * 32) << 16;
    for (int s = 0; s < n_steps; ++s) {
      const int hq = hk * G + s / steps_per_head;
      const int q0 = (i_start + s % steps_per_head) * kQ;
      LX_TR(tr_cta, s, 12);
      mbar_wait(dq_full, s & 1);
      tc_fence_after();
      LX_TR(tr_cta, s, 13);
      uint32_t v[4][32];
#pragma unroll
      for (int r = 0; r < 4; ++r) tmem_ld_32x32(tmem_base + kColY + r * 32 + lane_off, v[r]);
#pragma unroll
      for (int r = 0; r < 4; ++r) tmem_wait_ld_regs(v[r]);
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(dq_empty);
      LX_TR(tr_cta, s, 14);
      // fp32 adds performed at L2, straight from registers: a warp covers 32 consecutive head-dim elements of one
      // query row per instruction (one 128-byte request). The kernel is shared-memory-bandwidth bound (MMA operand
      // fetches, see tools/mma_bench.cu), so the former smem staging + cp.reduce.async.bulk cost 128 KB of smem
      // traffic per step that this path does not.
      if (t < kD) {
        float* dst = p.dq_accum + (((int64_t)b * p.Hq + hq) * p.S + q0) * kD + t;
        const int rows = min(kQ, p.S - q0);
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (r * 32 + i < rows) red_add_f32(dst + (r * 32 + i) * kD, __uint_as_float(v[r][i]));
      }
      LX_TR(tr_cta, s, 15);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<1>(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// Deterministic dQ (torch.use_deterministic_algorithms): CTA = (128 query rows, 1 query head), the forward's structure.
// The CTA walks the visible kv tiles of its rows in ascending order (attn_fwd_kernel's tile range and full-tile test)
// and accumulates dQ in TMEM, so the summation order is fixed by construction: no fp32 atomics, no dq_accum.
// Per kv tile j (every MMA 128 x 128 x 16):
//   S = Q K^T, dP = dO V^T          (TMEM, thread = query row)
//   P = exp2(S * scale_log2 - lse2) from the saved LSE (no online max), dS = P o (dP - delta) * scale, written as bf16
//   pairs over the score columns just read
//   dQ += dS K                      (A = dS from TMEM, B = K as the MN-major operand, like V in the forward's PV)
//   TMEM (512 columns): S0 | S1 | dP | dQ.   MMA issue order: S(j+1) | dQ(j), dP(j+1)
// The epilogue applies the RoPE backward to the fp32 accumulator with attn_dq_convert_kernel's arithmetic and rounds
// once to bf16. The S and dP products are recomputed here (attn_bwd_kernel<.., kNoDQ> computes them for dK / dV).
// ------------------------------------------------------------------------------------------------
namespace bwdq {
constexpr int kTile = 128;
constexpr int kTileBytes = kTile * kHD * 2;        // 32 KB
constexpr int kOffQ = 0;
constexpr int kOffdO = kOffQ + kTileBytes;
constexpr int kOffK = kOffdO + kTileBytes;         // 2 stages
constexpr int kOffV = kOffK + 2 * kTileBytes;      // 2 stages
constexpr int kOffBar = kOffV + 2 * kTileBytes;
// qdo_full, k full/empty[2], v full/empty[2], s full/empty[2], dp_full, ds_full, dq_done
constexpr int kNumBars = 1 + 4 + 4 + 4 + 3;
constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16 + 1024;
static_assert(kSmemBytes <= 232448, "deterministic dQ shared memory budget");
constexpr int kThreads = 256;                      // warp 0 TMA, warp 1 MMA, warp 2 TMEM alloc, warps 4-7: thread = query row
constexpr int kColS = 0, kColdP = 256, kColdQ = 384;
}  // namespace bwdq

template <bool kDocs, int kD>
__global__ void __launch_bounds__(bwdq::kThreads, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdO,
                   const AttnBwdParams p, __nv_bfloat16* __restrict__ dq, int64_t lddq) {
  using namespace bwdq;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* qdo_full = bars;
  uint64_t* k_full = bars + 1;     // [2]
  uint64_t* k_empty = bars + 3;    // [2]
  uint64_t* v_full = bars + 5;     // [2]
  uint64_t* v_empty = bars + 7;    // [2]
  uint64_t* s_full = bars + 9;     // [2]
  uint64_t* s_empty = bars + 11;   // [2]: dQ(j) has consumed dS(j), written over S buffer j & 1
  uint64_t* dp_full = bars + 13;
  uint64_t* ds_full = bars + 14;   // dS(j) is in TMEM and dP(j) has been read
  uint64_t* dq_done = bars + 15;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);

  const int warp = threadIdx.x >> 5;
  // grid = (query heads, batch, query tiles), longest tiles first (as attn_fwd_kernel)
  const int qt = gridDim.z - 1 - blockIdx.z;
  const int h = blockIdx.x, b = blockIdx.y;
  const int Pb = p.prefix_b ? min(max(p.prefix_b[b], 0), p.S) : p.P;
  const int hk = h / (p.Hq / p.Hkv);
  const int q0 = qt * kTile;
  int j_begin, n_kv;
  q_tile_kv_range<kDocs>(p.S, Pb, p.doc_start, b, q0, j_begin, n_kv);

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmdO);
  }
  if (warp == 1 && elect_one()) {
    mbar_init(qdo_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&s_empty[i], 1);
    }
    mbar_init(dp_full, 1);
    mbar_init(ds_full, 4);
    mbar_init(dq_done, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<1>(tmem_slot, 512);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base + kColS, tmem_dP = tmem_base + kColdP, tmem_dQ = tmem_base + kColdQ;

  if (warp == 0) {
    // ------------------------------------ TMA producer ------------------------------------
    if (elect_one()) {
      mbar_expect_tx(qdo_full, 2 * kTileBytes);
      tma_load_4d(smem + kOffQ, &tmQ, qdo_full, 0, h, q0, b);
      tma_load_4d(smem + kOffQ + kTileBytes / 2, &tmQ, qdo_full, 64, h, q0, b);
      tma_load_4d(smem + kOffdO, &tmdO, qdo_full, 0, h, q0, b);
      tma_load_4d(smem + kOffdO + kTileBytes / 2, &tmdO, qdo_full, 64, h, q0, b);
      for (int j = 0; j < n_kv; ++j) {
        const int st = j & 1;
        const uint32_t ph = (j >> 1) & 1;
        const int kv0 = (j_begin + j) * kTile;
        mbar_wait(&k_empty[st], ph ^ 1);
        mbar_expect_tx(&k_full[st], kTileBytes);
        uint8_t* sk = smem + kOffK + st * kTileBytes;
        tma_load_4d(sk, &tmK, &k_full[st], 0, hk, kv0, b);
        tma_load_4d(sk + kTileBytes / 2, &tmK, &k_full[st], 64, hk, kv0, b);
        mbar_wait(&v_empty[st], ph ^ 1);
        mbar_expect_tx(&v_full[st], kTileBytes);
        uint8_t* sv = smem + kOffV + st * kTileBytes;
        tma_load_4d(sv, &tmV, &v_full[st], 0, hk, kv0, b);
        tma_load_4d(sv + kTileBytes / 2, &tmV, &v_full[st], 64, hk, kv0, b);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------ MMA issuer ------------------------------------
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc(1, 1, 128, 128, 0, 0);   // S, dP: [q x d] . [kv x d]^T
      constexpr uint32_t idesc_dq = make_idesc(1, 1, 128, 128, 0, 1);  // dQ: [q x kv] . [kv x d]  (B = K MN-major)
      constexpr uint32_t kHi = desc_hi(1024);
      const uint32_t loQ = desc_lo(smem_u32(smem + kOffQ), 16), lodO = desc_lo(smem_u32(smem + kOffdO), 16);
      const uint32_t loK0 = desc_lo(smem_u32(smem + kOffK), 16), loKmn0 = desc_lo(smem_u32(smem + kOffK), 16384);
      const uint32_t loV0 = desc_lo(smem_u32(smem + kOffV), 16);
      auto mma_kk = [&](uint32_t d, uint32_t a_lo, uint32_t b_lo) {
#pragma unroll
        for (int dh = 0; dh < 2; ++dh)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_ss<false, 1>(d, desc_join(a_lo + dh * 1024 + ks * 2, kHi), desc_join(b_lo + dh * 1024 + ks * 2, kHi),
                              idesc_s, (dh | ks) != 0);
      };
      auto issue_s = [&](int j) {
        const int st = j & 1;
        const uint32_t ph = (j >> 1) & 1;
        mbar_wait(&k_full[st], ph);
        mbar_wait(&s_empty[st], ph ^ 1);
        tc_fence_after();
        mma_kk(tmem_S + st * 128, loQ, loK0 + st * (kTileBytes / 16));
        umma_commit(&s_full[st]);
      };
      auto issue_dp = [&](int j) {   // dP buffer: free once the workers have read dP(j - 1) (ds_full waited before)
        const int st = j & 1;
        mbar_wait(&v_full[st], (j >> 1) & 1);
        tc_fence_after();
        mma_kk(tmem_dP, lodO, loV0 + st * (kTileBytes / 16));
        umma_commit(dp_full);
        umma_commit(&v_empty[st]);
      };
      mbar_wait(qdo_full, 0);
      issue_s(0);
      issue_dp(0);
      for (int j = 0; j < n_kv; ++j) {
        const int st = j & 1;
        if (j + 1 < n_kv) issue_s(j + 1);
        mbar_wait(ds_full, j & 1);
        tc_fence_after();
        const uint32_t loKmn = loKmn0 + st * (kTileBytes / 16);
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            // A = dS from TMEM: bf16 pairs, 8 columns per 16-wide k-step (16 kv rows of K)
            umma_ts_f16(tmem_dQ, tmem_S + st * 128 + (kb * 4 + ks) * 8, desc_join(loKmn + (kb * 64 + ks * 16) * 8, kHi),
                        idesc_dq, (j | kb | ks) != 0);
        umma_commit(&s_empty[st]);
        umma_commit(&k_empty[st]);
        if (j + 1 < n_kv) issue_dp(j + 1);
      }
      umma_commit(dq_done);
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ------------------------------------ dS workers: thread = query row ------------------------------------
    const int r = threadIdx.x - 128;
    const uint32_t lane_off = uint32_t((warp - 4) * 32) << 16;
    const int q = q0 + r;
    const bool row_ok = q < p.S;
    const int64_t sidx = ((int64_t)b * p.Hq + h) * p.S + q;
    const float lse2 = row_ok ? p.lse[sidx] * kLog2e : INFINITY;   // rows past the end: P = 0
    const float dlt = row_ok ? p.delta[sidx] * p.scale : 0.f;
    const int ds_row = kDocs ? p.doc_start[(int64_t)b * p.S + min(q, p.S - 1)] : 0;
    const int ds_tile = kDocs ? p.doc_start[(int64_t)b * p.S + min(q0 + kTile - 1, p.S - 1)] : 0;
    for (int j = 0; j < n_kv; ++j) {
      const int st = j & 1;
      const int kv0 = (j_begin + j) * kTile;
      const bool full_tile = q_tile_full(p.S, Pb, ds_tile, q0, kv0);
      mbar_wait(&s_full[st], (j >> 1) & 1);
      tc_fence_after();
      const uint32_t tS = tmem_S + st * 128 + lane_off;
      uint32_t pr[64];   // P of this row: 128 kv columns as bf16 pairs
      {
        uint32_t sv[4][32];
#pragma unroll
        for (int c = 0; c < 4; ++c) tmem_ld_32x32(tS + c * 32, sv[c]);
        tmem_wait_ld_regs(sv[0]);
        tmem_wait_ld_regs(sv[1]);
        tmem_wait_ld_regs(sv[2]);
        tmem_wait_ld_regs(sv[3]);
        if (!full_tile) {   // the visible keys of a row are one interval of the tile's columns (see attn_fwd_kernel)
          const int lo = kDocs ? ds_row - kv0 : 0;
          const uint32_t width = (uint32_t)max(min(p.S, max(Pb, q + 1)) - kv0 - lo, 0);
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if ((uint32_t)(c * 32 + i - lo) >= width) sv[c][i] = 0xff800000u;  // -inf
        }
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int i = 0; i < 32; i += 2)
            pr[c * 16 + i / 2] = pack_bf16(ex2(fmaf(__uint_as_float(sv[c][i]), p.scale_log2, -lse2)),
                                           ex2(fmaf(__uint_as_float(sv[c][i + 1]), p.scale_log2, -lse2)));
      }
      mbar_wait(dp_full, j & 1);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t dv[32], dsr[16];
        tmem_ld_32x32(tmem_dP + lane_off + c * 32, dv);
        tmem_wait_ld_regs(dv);
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const uint32_t p01 = pr[c * 16 + i / 2];
          dsr[i / 2] = pack_bf16(bf16_lo(p01) * fmaf(__uint_as_float(dv[i]), p.scale, -dlt),
                                 bf16_hi(p01) * fmaf(__uint_as_float(dv[i + 1]), p.scale, -dlt));
        }
        // dS (bf16 pairs) over the score columns of this row: A operand of dQ(j), read straight from TMEM
        tmem_st_32x16(tS + c * 16, dsr);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(ds_full);
    }
    // epilogue: dQ row (fp32, TMEM) -> RoPE backward -> bf16
    mbar_wait(dq_done, 0);
    tc_fence_after();
    __nv_bfloat16* drow = dq + ((int64_t)b * p.S + q) * lddq + (int64_t)h * kD;
#pragma unroll 1
    for (int c = 0; c < kD / 32; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(tmem_dQ + lane_off + c * 32, v);
      tmem_wait_ld_regs(v);
      if (row_ok && p.rope != nullptr) {
        const float4* cs = reinterpret_cast<const float4*>(p.rope + ((int64_t)q * (kD / 2) + c * 16) * 2);
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 t4 = cs[i / 4];   // (c0, s0, c1, s1)
          const float g0 = __uint_as_float(v[i]), g1 = __uint_as_float(v[i + 1]);
          const float g2 = __uint_as_float(v[i + 2]), g3 = __uint_as_float(v[i + 3]);
          v[i] = __float_as_uint(g0 * t4.x + g1 * t4.y);
          v[i + 1] = __float_as_uint(g1 * t4.x - g0 * t4.y);
          v[i + 2] = __float_as_uint(g2 * t4.z + g3 * t4.w);
          v[i + 3] = __float_as_uint(g3 * t4.z - g2 * t4.w);
        }
      }
      if (row_ok) {
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          uint4 o4;
          o4.x = pack_bf16(__uint_as_float(v[i]), __uint_as_float(v[i + 1]));
          o4.y = pack_bf16(__uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
          o4.z = pack_bf16(__uint_as_float(v[i + 4]), __uint_as_float(v[i + 5]));
          o4.w = pack_bf16(__uint_as_float(v[i + 6]), __uint_as_float(v[i + 7]));
          stg_v4(drow + c * 32 + i, o4);
        }
      }
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<1>(tmem_base, 512);
}

// delta[b,h,s] = sum_d dO * O. 16-byte loads: D / 8 lanes per (row, head), so a warp covers 2 (D = 128) or 4 (D = 64)
// heads of one row; the 8-byte-per-lane version ran at half the HBM rate.
template <int D>
__global__ void __launch_bounds__(256) attn_delta_kernel(const __nv_bfloat16* __restrict__ o, int64_t ldo,
                                                         const __nv_bfloat16* __restrict__ dout, int64_t lddo,
                                                         float* __restrict__ delta, int S, int Hq) {
  // grid = (rows, groups of 8 warps): the row is uniform per CTA and the head comes from the warp index — the first version
  // derived both from one flat warp index with two 64-bit divisions per thread, more instructions than the dot product
  constexpr int kLanes = D / 8;                 // lanes per head: 16 or 8
  constexpr int kHeadsPerWarp = 32 / kLanes;
  const int lane = threadIdx.x & 31;
  const int grp = blockIdx.y * 8 + (threadIdx.x >> 5);
  const int h = grp * kHeadsPerWarp + lane / kLanes;
  if (grp * kHeadsPerWarp >= Hq) return;        // whole warp
  const int64_t row = blockIdx.x;
  float s = 0.f;
  if (h < Hq) {
    const int c = h * D + (lane % kLanes) * 8;
    const uint4 a = ldg_nc_v4(o + row * ldo + c);
    const uint4 g = ldg_nc_v4(dout + row * lddo + c);
    s = bf16_lo(a.x) * bf16_lo(g.x) + bf16_hi(a.x) * bf16_hi(g.x) + bf16_lo(a.y) * bf16_lo(g.y) +
        bf16_hi(a.y) * bf16_hi(g.y) + bf16_lo(a.z) * bf16_lo(g.z) + bf16_hi(a.z) * bf16_hi(g.z) +
        bf16_lo(a.w) * bf16_lo(g.w) + bf16_hi(a.w) * bf16_hi(g.w);
  }
#pragma unroll
  for (int off = kLanes / 2; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  if (h < Hq && (lane % kLanes) == 0) {
    const unsigned bb = blockIdx.x / (unsigned)S, ss = blockIdx.x - bb * (unsigned)S;   // rows < 2^31 (launcher)
    delta[((int64_t)bb * Hq + h) * S + ss] = s;
  }
}

// dq_accum fp32 [B, Hq, S, D] -> dq bf16 [B*S, Hq*D] (row pitch lddq); one thread = 2 x 8 head-dim elements.
// grid = (B * Hq, chunks of 512 vectors of one head's [S, D] slab): batch and head are uniform per CTA, position and column
// come from the thread index by a shift and a mask (the first version: four 64-bit divisions per thread and vector)
template <int D>
__global__ void __launch_bounds__(256) attn_dq_convert_kernel(const float* __restrict__ acc,
                                                              __nv_bfloat16* __restrict__ dq, int64_t lddq, int S,
                                                              int Hq, const float* __restrict__ rope) {
  constexpr int kVecs = D / 8;
  const unsigned bh = blockIdx.x, b = bh / (unsigned)Hq, h = bh - b * (unsigned)Hq;
  const float* slab = acc + (int64_t)bh * S * D;
  const int nvec = S * kVecs;
  float4 lo[2], hi[2], t0[2], t1[2];
  int t[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    t[k] = blockIdx.y * 512 + k * 256 + threadIdx.x;
    if (t[k] < nvec) {
      const float* src = slab + (int64_t)t[k] * 8;
      lo[k] = __ldcs(reinterpret_cast<const float4*>(src));       // read once: streaming
      hi[k] = __ldcs(reinterpret_cast<const float4*>(src + 4));
      if (rope != nullptr) {
        const int s_ = t[k] / kVecs, c = (t[k] % kVecs) * 8;
        const float4* cs = reinterpret_cast<const float4*>(rope + ((int64_t)s_ * (D / 2) + c / 2) * 2);
        t0[k] = __ldg(cs);
        t1[k] = __ldg(cs + 1);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    if (t[k] >= nvec) continue;
    const int s_ = t[k] / kVecs, c = (t[k] % kVecs) * 8;
    float4 a = lo[k], b4 = hi[k];
    if (rope != nullptr) {  // RoPE backward on the fp32 sums (one rounding fewer than rotating the bf16 result)
      const float4 u0 = t0[k], u1 = t1[k];
      a = make_float4(a.x * u0.x + a.y * u0.y, a.y * u0.x - a.x * u0.y, a.z * u0.z + a.w * u0.w, a.w * u0.z - a.z * u0.w);
      b4 = make_float4(b4.x * u1.x + b4.y * u1.y, b4.y * u1.x - b4.x * u1.y, b4.z * u1.z + b4.w * u1.w,
                       b4.w * u1.z - b4.z * u1.w);
    }
    uint4 o4;
    o4.x = pack_bf16(a.x, a.y);
    o4.y = pack_bf16(a.z, a.w);
    o4.z = pack_bf16(b4.x, b4.y);
    o4.w = pack_bf16(b4.z, b4.w);
    *reinterpret_cast<uint4*>(dq + ((int64_t)b * S + s_) * lddq + (int64_t)h * D + c) = o4;
  }
}

// [B, S, H, D] view with row pitch ld; 64-column boxes. For D = 64 the second box of a 128-wide tile starts at
// column 64 = out of bounds and is zero-filled by TMA, so the 128-wide kernels run unchanged on zero-padded heads.
static int make_head_tmap(CUtensorMap* m, const void* ptr, int64_t ld, int64_t B, int64_t S, int H, int D,
                          int box_rows) {
  const int64_t dims[4] = {D, H, S, B};
  const int64_t strides[3] = {D, ld, S * ld};
  const int box[4] = {64, 1, box_rows, 1};
  return make_tmap_4d(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ptr, dims, strides, box);
}

static int check_attn_args(int64_t B, int64_t S, int Hq, int Hkv, int D, int64_t P, const char* who) {
  if (D != 128 && D != 64) return set_error(LLAMAX_ERR_ARG, "attention: head_dim must be 64 or 128");
  if (B <= 0 || S <= 0 || Hq <= 0 || Hkv <= 0 || Hq % Hkv) return set_error(LLAMAX_ERR_ARG, "attention: bad B/S/H");
  if (P < 0) return set_error(LLAMAX_ERR_ARG, "attention: prefix_len < 0");
  // grids are indexed by rows and by (batch, head) pairs, 32-bit position arithmetic inside the side kernels
  if (B * S > 0x7fffffffLL || B * Hq > 0x7fffffffLL || S * 16 > 0x7fffffffLL)
    return set_error(LLAMAX_ERR_ARG, "attention: B * S, B * Hq and 16 * S must be below 2^31");
  (void)who;
  return 0;
}

}  // namespace lx

using namespace lx;

extern "C" {

#ifdef LX_ATTN_TRACE
int llamax_debug_attn_trace(void* buf) {
  long long* b = (long long*)buf;
  cudaError_t e = cudaMemcpyToSymbol(g_attn_trace, &b, sizeof(b));
  return e == cudaSuccess ? 0 : set_cuda_error(e, "debug_attn_trace");
}
#endif

int llamax_attn_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o,
                    int64_t ldo, void* lse, int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D,
                    int64_t prefix_len, const void* prefix_len_b, const void* doc_start, float scale, void* stream) {
  if (!q || !k || !v || !o || !lse) return set_error(LLAMAX_ERR_ARG, "attn_fwd: null pointer");
  int rc = check_attn_args(B, S, Hq, Hkv, D, prefix_len, "attn_fwd");
  if (rc) return rc;
  if (ldq % 8 || ldk % 8 || ldv % 8 || ldo % 8) return set_error(LLAMAX_ERR_ARG, "attn_fwd: pitches must be multiples of 8");
  CUtensorMap tq, tk, tv;
  if ((rc = make_head_tmap(&tq, q, ldq, B, S, Hq, D, fwd::kTile))) return rc;
  if ((rc = make_head_tmap(&tk, k, ldk, B, S, Hkv, D, fwd::kTile))) return rc;
  if ((rc = make_head_tmap(&tv, v, ldv, B, S, Hkv, D, fwd::kTile))) return rc;
  // A/B switch: LLAMAX_ATTN_FWD = 1 (one query tile per CTA), 2 (two tiles, thread per row, one issuer), 3 (two tiles,
  // two threads per row), 4 (two tiles, thread per row, chunked P hand-off, one issuer per tile), 5 (default: v4 made
  // persistent, one CTA per SM over a static item list)
  static const int version = [] {
    const char* e = getenv("LLAMAX_ATTN_FWD");
    if (getenv("LLAMAX_ATTN_FWD_ONE_TILE") && getenv("LLAMAX_ATTN_FWD_ONE_TILE")[0] == '1') return 1;
    return (e != nullptr && e[0] >= '1' && e[0] <= '5') ? e[0] - '0' : 5;
  }();
  // packed documents: the XU token of v4 / v5 is off there (see the kernels) and without it they lose to v2 -> v2
  const int version_eff = (version >= 4 && doc_start != nullptr) ? 2 : version;
  if (version_eff == 5) {   // persistent: one CTA per SM over a static item list
    auto kern5 = D == 128 ? attn_fwd5_kernel<128> : attn_fwd5_kernel<64>;
    if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern5), fwd5::kSmemBytes5, "attn_fwd: cudaFuncSetAttribute"))) return rc;
    AttnFwdParams p5;
    p5.o = (__nv_bfloat16*)o;
    p5.ldo = ldo;
    p5.lse = (float*)lse;
    p5.B = (int)B; p5.S = (int)S; p5.Hq = Hq; p5.Hkv = Hkv;
    p5.P = (int)std::min<int64_t>(prefix_len, S);
    p5.D = D;
    p5.scale_log2 = scale * kLog2e;
    p5.doc_start = nullptr;
    p5.prefix_b = (const int32_t*)prefix_len_b;
    const int n_pairs = (int)((ceil_div(S, fwd::kTile) + 1) / 2);
    const int64_t n_items = (int64_t)n_pairs * B * Hq;
    const int grid5 = (int)std::min<int64_t>(n_items, sm_count());
    kern5<<<grid5, fwd4::kThreads, fwd5::kSmemBytes5, (cudaStream_t)stream>>>(tq, tk, tv, p5, n_pairs);
    LX_CHECK_LAUNCH("attn_fwd");
    return 0;
  }
  const bool one_tile = version_eff == 1;
  auto kern1 = doc_start ? (D == 128 ? attn_fwd_kernel<true, 128> : attn_fwd_kernel<true, 64>)
                         : (D == 128 ? attn_fwd_kernel<false, 128> : attn_fwd_kernel<false, 64>);
  auto kern2 = doc_start ? (D == 128 ? attn_fwd2_kernel<true, 128> : attn_fwd2_kernel<true, 64>)
                         : (D == 128 ? attn_fwd2_kernel<false, 128> : attn_fwd2_kernel<false, 64>);
  auto kern3 = doc_start ? (D == 128 ? attn_fwd3_kernel<true, 128> : attn_fwd3_kernel<true, 64>)
                         : (D == 128 ? attn_fwd3_kernel<false, 128> : attn_fwd3_kernel<false, 64>);
  static const bool alu_pack = getenv("LLAMAX_ATTN_ALU_PACK") && getenv("LLAMAX_ATTN_ALU_PACK")[0] == '1';
  static const bool stagger = !(getenv("LLAMAX_ATTN_STAGGER") && getenv("LLAMAX_ATTN_STAGGER")[0] == '0');
  auto pick4 = [&](auto docs_tag, auto d_tag) {
    constexpr bool kDc = decltype(docs_tag)::value;
    constexpr int kDd = decltype(d_tag)::value;
    return alu_pack ? (stagger ? attn_fwd4_kernel<kDc, kDd, true, true> : attn_fwd4_kernel<kDc, kDd, true, false>)
                    : (stagger ? attn_fwd4_kernel<kDc, kDd, false, true> : attn_fwd4_kernel<kDc, kDd, false, false>);
  };
  auto kern4 = doc_start ? (D == 128 ? pick4(std::true_type{}, std::integral_constant<int, 128>{})
                                     : pick4(std::true_type{}, std::integral_constant<int, 64>{}))
                         : (D == 128 ? pick4(std::false_type{}, std::integral_constant<int, 128>{})
                                     : pick4(std::false_type{}, std::integral_constant<int, 64>{}));
  auto kern = version_eff == 1 ? kern1 : version_eff == 2 ? kern2 : version_eff == 3 ? kern3 : kern4;
  const int smem_bytes = version_eff == 1 ? fwd::smem_bytes(fwd::kNB) : version_eff == 2 ? fwd2::kSmemBytes
                         : version_eff == 3 ? fwd3::kSmemBytes : fwd4::kSmemBytes;
  const int threads = version_eff == 1 ? fwd::kThreads : version_eff == 2 ? fwd2::kThreads
                      : version_eff == 3 ? fwd3::kThreads : fwd4::kThreads;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), smem_bytes, "attn_fwd: cudaFuncSetAttribute"))) return rc;
  AttnFwdParams p;
  p.o = (__nv_bfloat16*)o;
  p.ldo = ldo;
  p.lse = (float*)lse;
  p.B = (int)B; p.S = (int)S; p.Hq = Hq; p.Hkv = Hkv;
  p.P = (int)std::min<int64_t>(prefix_len, S);
  p.D = D;
  p.scale_log2 = scale * kLog2e;
  p.doc_start = (const int32_t*)doc_start;
  p.prefix_b = (const int32_t*)prefix_len_b;
  const unsigned q_tiles = (unsigned)ceil_div(S, fwd::kTile);
  dim3 grid(Hq, (unsigned)B, one_tile ? q_tiles : (q_tiles + 1) / 2);
  kern<<<grid, threads, smem_bytes, (cudaStream_t)stream>>>(tq, tk, tv, p);
  LX_CHECK_LAUNCH("attn_fwd");
  return 0;
}

}  // extern "C"

// dq_accum == NULL: deterministic mode (attn_bwd_dq_kernel writes dq, attn_bwd_kernel<.., kNoDQ> dk / dv)
static int attn_bwd_run(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                        const void* o, int64_t ldo, const void* lse, const void* dout, int64_t lddo, void* dq,
                        int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, void* dq_accum, void* delta,
                        int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D, int64_t prefix_len,
                        const void* prefix_len_b, const void* doc_start, const void* doc_end, float scale,
                        const void* rope_inverse, void* stream) {
  const bool det = dq_accum == nullptr;
  if ((doc_start == nullptr) != (doc_end == nullptr))
    return set_error(LLAMAX_ERR_ARG, "attn_bwd: doc_start and doc_end go together");
  if (!q || !k || !v || !lse || !dout || !dq || !dk || !dv || !delta)   // o may be NULL: delta is given
    return set_error(LLAMAX_ERR_ARG, "attn_bwd: null pointer");
  int rc = check_attn_args(B, S, Hq, Hkv, D, prefix_len, "attn_bwd");
  if (rc) return rc;
  if (ldq % 8 || ldk % 8 || ldv % 8 || (o != nullptr && ldo % 8) || lddo % 8 || lddq % 8 || lddk % 8 || lddv % 8)
    return set_error(LLAMAX_ERR_ARG, "attn_bwd: pitches must be multiples of 8");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows = B * S;
  if (!det) {
    cudaError_t e = cudaMemsetAsync(dq_accum, 0, (size_t)rows * Hq * D * sizeof(float), st);
    if (e != cudaSuccess) return set_cuda_error(e, "attn_bwd: memset");
  }
  if (o != nullptr) {
    const int groups = (int)ceil_div(Hq, 32 / (D / 8));   // warps per row
    dim3 dgrid((unsigned)rows, (unsigned)ceil_div(groups, 8));
    if (D == 128)
      attn_delta_kernel<128><<<dgrid, 256, 0, st>>>((const __nv_bfloat16*)o, ldo, (const __nv_bfloat16*)dout, lddo,
                                                    (float*)delta, (int)S, Hq);
    else
      attn_delta_kernel<64><<<dgrid, 256, 0, st>>>((const __nv_bfloat16*)o, ldo, (const __nv_bfloat16*)dout, lddo,
                                                   (float*)delta, (int)S, Hq);
    LX_CHECK_LAUNCH("attn_bwd: delta");
  }
  CUtensorMap tq, tk, tv, tdo;
  if ((rc = make_head_tmap(&tq, q, ldq, B, S, Hq, D, bwd::kQ))) return rc;
  if ((rc = make_head_tmap(&tdo, dout, lddo, B, S, Hq, D, bwd::kQ))) return rc;
  if ((rc = make_head_tmap(&tk, k, ldk, B, S, Hkv, D, bwd::kKV))) return rc;
  if ((rc = make_head_tmap(&tv, v, ldv, B, S, Hkv, D, bwd::kKV))) return rc;
  auto kern = det ? (doc_start ? (D == 128 ? attn_bwd_kernel<true, 128, true> : attn_bwd_kernel<true, 64, true>)
                               : (D == 128 ? attn_bwd_kernel<false, 128, true> : attn_bwd_kernel<false, 64, true>))
                  : (doc_start ? (D == 128 ? attn_bwd_kernel<true, 128> : attn_bwd_kernel<true, 64>)
                               : (D == 128 ? attn_bwd_kernel<false, 128> : attn_bwd_kernel<false, 64>));
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), bwd::kSmemBytes, "attn_bwd: cudaFuncSetAttribute"))) return rc;
  AttnBwdParams p;
  p.lse = (const float*)lse;
  p.delta = (const float*)delta;
  p.dq_accum = (float*)dq_accum;
  p.dk = (__nv_bfloat16*)dk; p.lddk = lddk;
  p.dv = (__nv_bfloat16*)dv; p.lddv = lddv;
  p.B = (int)B; p.S = (int)S; p.Hq = Hq; p.Hkv = Hkv;
  p.P = (int)std::min<int64_t>(prefix_len, S);
  p.D = D;
  p.scale = scale;
  p.scale_log2 = scale * kLog2e;
  p.doc_start = (const int32_t*)doc_start;
  p.doc_end = (const int32_t*)doc_end;
  p.rope = (const float*)rope_inverse;
  p.prefix_b = (const int32_t*)prefix_len_b;
  dim3 grid(Hkv, (unsigned)ceil_div(S, bwd::kKV), (unsigned)B);
  kern<<<grid, det ? bwd::kThreadsNoDQ : bwd::kThreads, bwd::kSmemBytes, st>>>(tq, tk, tv, tdo, p);
  LX_CHECK_LAUNCH("attn_bwd");
  if (det) {
    auto kdq = doc_start ? (D == 128 ? attn_bwd_dq_kernel<true, 128> : attn_bwd_dq_kernel<true, 64>)
                         : (D == 128 ? attn_bwd_dq_kernel<false, 128> : attn_bwd_dq_kernel<false, 64>);
    if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kdq), bwdq::kSmemBytes, "attn_bwd: cudaFuncSetAttribute")))
      return rc;
    dim3 qgrid(Hq, (unsigned)B, (unsigned)ceil_div(S, bwdq::kTile));
    kdq<<<qgrid, bwdq::kThreads, bwdq::kSmemBytes, st>>>(tq, tk, tv, tdo, p, (__nv_bfloat16*)dq, lddq);
    LX_CHECK_LAUNCH("attn_bwd: dq");
    return 0;
  }
  {
    dim3 cgrid((unsigned)(B * Hq), (unsigned)ceil_div(S * (D / 8), 512));
    if (D == 128)
      attn_dq_convert_kernel<128><<<cgrid, 256, 0, st>>>((const float*)dq_accum, (__nv_bfloat16*)dq, lddq, (int)S, Hq,
                                                          (const float*)rope_inverse);
    else
      attn_dq_convert_kernel<64><<<cgrid, 256, 0, st>>>((const float*)dq_accum, (__nv_bfloat16*)dq, lddq, (int)S, Hq,
                                                         (const float*)rope_inverse);
    LX_CHECK_LAUNCH("attn_bwd: dq convert");
  }
  return 0;
}

extern "C" {

int llamax_attn_bwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                    const void* o, int64_t ldo, const void* lse, const void* dout, int64_t lddo, void* dq,
                    int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, void* dq_accum, void* delta,
                    int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D, int64_t prefix_len,
                    const void* prefix_len_b, const void* doc_start, const void* doc_end, float scale,
                    const void* rope_inverse, void* stream) {
  if (!dq_accum) return set_error(LLAMAX_ERR_ARG, "attn_bwd: null pointer");
  return attn_bwd_run(q, ldq, k, ldk, v, ldv, o, ldo, lse, dout, lddo, dq, lddq, dk, lddk, dv, lddv, dq_accum, delta,
                      B, S, Hq, Hkv, D, prefix_len, prefix_len_b, doc_start, doc_end, scale, rope_inverse, stream);
}

int llamax_attn_bwd_deterministic(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                                  const void* o, int64_t ldo, const void* lse, const void* dout, int64_t lddo, void* dq,
                                  int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, void* delta, int64_t B,
                                  int64_t S, int32_t Hq, int32_t Hkv, int32_t D, int64_t prefix_len,
                                  const void* prefix_len_b, const void* doc_start, const void* doc_end, float scale,
                                  const void* rope_inverse, void* stream) {
  return attn_bwd_run(q, ldq, k, ldk, v, ldv, o, ldo, lse, dout, lddo, dq, lddq, dk, lddk, dv, lddv, nullptr, delta,
                      B, S, Hq, Hkv, D, prefix_len, prefix_len_b, doc_start, doc_end, scale, rope_inverse, stream);
}

}  // extern "C"
