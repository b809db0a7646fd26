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
// Forward  : two 128-row query tiles per CTA, two softmax warpgroups (thread = row). Per tile S = Q K^T in TMEM is read
//            once into registers, P (bf16 pairs) is written back over the score columns and consumed by the PV MMA
//            straight from TMEM, O accumulates in TMEM with lazy rescaling; exp2-domain online softmax, LSE saved in
//            natural log. attn_fwd5_kernel is persistent: one CTA per SM walks a length-balanced list of items (pair of
//            query tiles, query head, sequence); warp0 TMA, warps1-2 MMA issue (one per tile), P handed over in four
//            chunks. With packed documents attn_fwd2_kernel runs instead: one CTA per pair of query tiles, one MMA
//            issuer, each tile starting at its own document's first kv tile.
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

// ------------------------------------------------------------------------------------------------
// Attention dropout (the semantics of F.scaled_dot_product_attention(dropout_p = p)). The keep mask Z of (batch b,
// query head hq, query q, key kv) comes from Philox4x32-10 (Random123 / curand), key = the 64-bit seed, counter =
// (kv / 16, q, b * Hq + hq, call): one call decides 16 consecutive keys of one query row, key kv is kept when byte
// kv % 16 of the four output words (little-endian) is >= t = round(p * 256), and kept values are scaled by
// 256 / (256 - t), so the expectation is exact and the drop rate is t / 256. The forward, both backward kernels and
// tests/attention_dropout_ref.py build the same Z, regenerated, never stored. The LSE is that of the undropped softmax.
// ------------------------------------------------------------------------------------------------
struct AttnDrop {
  uint32_t key0, key1;   // seed: low / high word
  uint32_t call;         // counter word 3 (generator offset / 4)
  uint32_t t4;           // t in each of the four bytes (t = 256: 0xffffffff, with scale 0)
  float scale;           // 256 / (256 - t); 0 when t = 256 (everything dropped)
};

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                               uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    const uint32_t lo0 = 0xD2511F53u * c0, hi0 = __umulhi(0xD2511F53u, c0);
    const uint32_t lo1 = 0xCD9E8D57u * c2, hi1 = __umulhi(0xCD9E8D57u, c2);
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
  }
  return make_uint4(c0, c1, c2, c3);
}

// keep mask of the 16 keys [16 g, 16 g + 16) of query row q: 0xff in each kept byte, 0x00 in each dropped one
__device__ __forceinline__ void drop_keep16(const AttnDrop& d, uint32_t g, uint32_t q, uint32_t bh, uint32_t (&z)[4]) {
  const uint4 r = philox4x32_10(g, q, bh, d.call, d.key0, d.key1);
  z[0] = __vcmpgeu4(r.x, d.t4);
  z[1] = __vcmpgeu4(r.y, d.t4);
  z[2] = __vcmpgeu4(r.z, d.t4);
  z[3] = __vcmpgeu4(r.w, d.t4);
}

// bf16-pair mask of bytes b, b + 1 (b even) of a keep word: AND it into a packed pair of P values
__device__ __forceinline__ uint32_t drop_pair_mask(uint32_t z, int b) { return __byte_perm(z, 0, b ? 0x3322 : 0x1100); }
// all-ones / all-zeros word from byte b of a keep word: AND it into an fp32 value
__device__ __forceinline__ uint32_t drop_elem_mask(uint32_t z, int b) { return __byte_perm(z, 0, b * 0x1111); }

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

// Layout and thread roles of both forward kernels: a CTA holds two 128-row query tiles, each with its own softmax
// warpgroup, and double-buffered K / V tiles; warpgroup 0 does TMA, MMA issue and TMEM allocation.
namespace fwd {
constexpr int kTile = 128;
constexpr int kTileBytes = kTile * kHD * 2;        // 32 KB: two 16 KB boxes of [128 rows x 128 B]
constexpr int kOffQ = 0;                           // 2 query tiles
constexpr int kOffK = kOffQ + 2 * kTileBytes;      // 2 stages
constexpr int kOffV = kOffK + 2 * kTileBytes;      // 2 stages
constexpr int kOffBar = kOffV + 2 * kTileBytes;    // mbarriers, then the TMEM address slot
// attn_fwd2_kernel: q_full, k full/empty[2], v full/empty[2], s_full[2 tiles], p_full[2 tiles], pv_done[2 tiles]
constexpr int kNumBars2 = 1 + 4 + 4 + 2 + 2 + 2;
// attn_fwd5_kernel: q_full, k full/empty[2], v full/empty[2], s_full[2 tiles], p_chunk[2 tiles][4], pv_done[2 tiles],
// xu_tok[2 item parities][2 tiles], q_empty
constexpr int kNumBars5 = 1 + 4 + 4 + 2 + 8 + 2 + 4 + 1;
constexpr int kSmemBytes2 = kOffBar + kNumBars2 * 8 + 16 + 1024;   // + 1 KB alignment slack
constexpr int kSmemBytes5 = kOffBar + kNumBars5 * 8 + 16 + 1024;
constexpr int kThreads = 384;                      // warpgroup 0: control; warpgroups 1, 2: softmax of tile 0, 1
constexpr int kRegsCtrl = 56, kRegsSoftmax = 224;  // 128 * 56 + 256 * 224 = 384 * 168
}  // namespace fwd

// ------------------------------------------------------------------------------------------------
// Packed-document forward: two query tiles per CTA ("ping-pong"), one MMA-issuing thread. Traced with one query tile per
// CTA (round 1, tools/attn_trace.py), the softmax warpgroup needs ~2400 cycles per 128x128 tile (128 ex2 per thread on
// the 16-lane XU pipe = 1024, the max, TMEM round-trips, barriers — one warp per scheduler, nothing to overlap with)
// against 1364 cycles of MMA work, and the chain softmax(j) -> PV(j) is serial. Here a CTA owns TWO 128-row query tiles
// with one softmax warpgroup each: while one group is in its exp phase the other waits for its MMAs, so XU pipe and
// tensor pipe are both kept busy and each K/V tile is loaded once for 256 query rows. Each tile starts at the kv tile of
// its first row's document, so the two tiles may start at different kv tiles, which attn_fwd5_kernel cannot handle.
//   TMEM (512 columns): S0 | S1 (P written over the score columns read, A operand of PV from TMEM) | O0 | O1
//   MMA issue order   : S0(j0), S1(j0);  then per kv tile j:  PV0(j), S0(j+1) | PV1(j), S1(j+1)
// ------------------------------------------------------------------------------------------------
template <int kD, bool kDrop = false>
__global__ void __launch_bounds__(fwd::kThreads, 1)
attn_fwd2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                 const __grid_constant__ CUtensorMap tmV, const AttnFwdParams p, const AttnDrop drop) {
  using namespace fwd;
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
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars2);

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
      jb_[x] = p.doc_start[(int64_t)b * p.S + q0] / kTile;
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
            mbar_wait(&v_full[st], ((j - jb) >> 1) & 1);
            mbar_wait(&p_full[x], it[x] & 1);
            tc_fence_after();
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
    const int ds_row = p.doc_start[(int64_t)b * p.S + min(q, p.S - 1)];
    const int ds_tile = p.doc_start[(int64_t)b * p.S + min(q0 + kTile - 1, p.S - 1)];
    for (int i = 0; i < n_kv; ++i) {
      const int kv0 = (jb_x + i) * kTile;
      // tile needs the element test unless every (q, kv) pair is visible and in range
      const bool full_tile = (kv0 + kTile <= p.S) && ((kv0 + kTile <= Pb) || (kv0 + kTile - 1 <= q0)) && (kv0 >= ds_tile);
      mbar_wait(&s_full[x], i & 1);
      tc_fence_after();
      // single pass over TMEM: the whole score row (128 fp32) lives in registers
      uint32_t sv[4][32];
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld_32x32(tS + c * 32, sv[c]);
      tmem_wait_ld_regs(sv[0]);
      tmem_wait_ld_regs(sv[1]);
      tmem_wait_ld_regs(sv[2]);
      tmem_wait_ld_regs(sv[3]);
      if (!full_tile) {
        // the visible keys of a row are ONE interval of the tile's columns, [lo, lo + width): the prefix-LM mask keeps
        // kv < max(P, q + 1) (and kv < S), packed documents additionally cut the head (kv >= ds_row) — one unsigned
        // compare against a per-row constant and a select per element instead of three compares
        const int lo = ds_row - kv0;
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
      for (int c = 0; c < 4; ++c) {
        uint32_t z[8];   // dropout: keep bytes of the chunk's 32 keys (the sum l stays that of the undropped P)
        if constexpr (kDrop) {
          drop_keep16(drop, (kv0 + c * 32) >> 4, q, b * p.Hq + h, *reinterpret_cast<uint32_t(*)[4]>(&z[0]));
          drop_keep16(drop, (kv0 + c * 32 + 16) >> 4, q, b * p.Hq + h, *reinterpret_cast<uint32_t(*)[4]>(&z[4]));
        }
#pragma unroll
        for (int e = 0; e < 32; e += 2) {
          const float p0 = ex2(fmaf(__uint_as_float(sv[c][e]), p.scale_log2, -m_exp));      // -inf -> 0
          const float p1 = ex2(fmaf(__uint_as_float(sv[c][e + 1]), p.scale_log2, -m_exp));
          rowsum += p0 + p1;
          preg[c * 16 + e / 2] = pack_bf16(p0, p1);
          if constexpr (kDrop) preg[c * 16 + e / 2] &= drop_pair_mask(z[e / 4], e & 2);
        }
      }
      l = l * alpha + rowsum;
      if (i > 0) {
        mbar_wait(&pv_done[x], (i - 1) & 1);  // O stable
        tc_fence_after();
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
      tc_fence_before();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(&p_full[x]);
    }
    // epilogue
    if (n_kv > 0) {
      mbar_wait(&pv_done[x], (n_kv - 1) & 1);
      tc_fence_after();
      const float inv_l = kDrop ? drop.scale / l : 1.f / l;
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
// Persistent forward, used without packed documents. It keeps attn_fwd2_kernel's structure (two query tiles per CTA,
// one softmax warpgroup per tile, thread = row) and cuts the serial chain of a tile where it can be cut. The chain
// S(j) -> softmax(j) -> PV(j) -> S(j+1) cannot be broken (P aliases S in TMEM, 512 columns are S0 | S1 | O0 | O1), and
// it, not a pipe, paces attn_fwd2_kernel: 1364 cycles of the tile's own MMAs + ~2500 of softmax latency + hand-offs =
// the measured ~4250 cycles per pair of tiles, with the tensor pipe busy 64 % of the time.
//   * P is handed over in FOUR 32-column chunks, each with its own mbarrier: the two PV MMAs of a chunk run while the
//     softmax warpgroup is in the exponentials of the next chunks, so of PV only the last chunk's MMAs stay on the chain;
//   * one MMA-issuing warp PER TILE: with chunked hand-offs a single issuer thread would sit in tile 0's chunk waits
//     while tile 1's chunks are ready (head-of-line blocking); the K / V stages are released by BOTH issuers (count 2);
//   * no per-step wait on pv_done: S(j) is issued behind PV(j-1) by the same thread, so s_full(j) implies it;
//   * an XU token makes the exp phases of the two tiles strictly alternate (see the softmax loop).
// The kernel is PERSISTENT: one CTA per SM walks a static, length-balanced list of work items (pair of query tiles, head,
// sequence) and every ring — K / V stages, the S / P / O hand-offs, the XU token — keeps running across items, so that
// of an item's fixed cost only the O drain stays exposed:
//   * with one CTA per item, every item pays launch, barrier init, TMEM allocation, then Q and the first K from global
//     memory and the first S MMA before any softmax can start (~2400 cycles, traced), and at the end one tile alone in
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
// has exactly one wait: the barriers live on across items, so no arrival may be left unmatched.
// Packed-document masks run on attn_fwd2_kernel (the token's wait chain is only acyclic when both tiles start at kv
// tile 0).
// ------------------------------------------------------------------------------------------------
template <int kD, bool kDrop = false>
__global__ void __launch_bounds__(fwd::kThreads, 1)
attn_fwd5_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                 const __grid_constant__ CUtensorMap tmV, const AttnFwdParams p, int n_pairs, const AttnDrop drop) {
  using namespace fwd;
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
        // XU token. The exponentials of the two tiles share the XU pipe (16 ex2 / clk / SM = 8 cycles per warp instruction
        // per scheduler). Traced, the two tiles left alone drift INTO phase within two steps, whatever their initial offset:
        // both sit in their exp phase together (~2200 cycles each instead of ~1100 alone) and then both sit in their
        // XU-idle part together (wait for S, TMEM load, row max: ~1700 cycles), ~3900 cycles per step. The token makes the
        // exp phases mutually exclusive and strictly alternating, so that one tile's XU-idle part hides under the other's
        // exponentials. Within an item the exp phases run t0(0) t1(0) t0(1) t1(1) ...; tile 1's exp i follows tile 0's
        // exp i (if tile 0 has one), tile 0's exp i follows tile 1's exp i - 1. Both tiles start at kv tile 0 and tile 1
        // has at least as many steps as tile 0, so the chain of waits is acyclic. Every arrival below has exactly one wait
        // here, so the barrier phases can be counted across items.
        if (x == 1 ? (i < n0) : (i > 0 && i - 1 < n1)) {
          mbar_wait(&xu_tok[(r & 1) * 2 + x], tokw[r & 1] & 1);
          ++tokw[r & 1];
        }
        float m_exp = (m_used == -INFINITY) ? 0.f : m_used;
        asm volatile("" : "+f"(m_exp));   // pins the exponentials behind the wait (they are pure: ptxas hoists them otherwise)
        float rowsum = 0.f;   // same summation order as attn_fwd2_kernel: bit-identical outputs
        uint32_t pc[2][16];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t z[8];   // dropout: keep bytes of the chunk's 32 keys (the sum l stays that of the undropped P)
          if constexpr (kDrop) {
            const uint32_t bh = it.b * p.Hq + it.h;
            drop_keep16(drop, (kv0 + c * 32) >> 4, q, bh, *reinterpret_cast<uint32_t(*)[4]>(&z[0]));
            drop_keep16(drop, (kv0 + c * 32 + 16) >> 4, q, bh, *reinterpret_cast<uint32_t(*)[4]>(&z[4]));
          }
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const float p0 = ex2(fmaf(__uint_as_float(sv[c][e]), p.scale_log2, -m_exp));      // -inf -> 0
            const float p1 = ex2(fmaf(__uint_as_float(sv[c][e + 1]), p.scale_log2, -m_exp));
            rowsum += p0 + p1;
            pc[c & 1][e / 2] = pack_bf16(p0, p1);
            if constexpr (kDrop) pc[c & 1][e / 2] &= drop_pair_mask(z[e / 4], e & 2);
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
        const float inv_l = kDrop ? drop.scale / l : 1.f / l;
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
constexpr int kOffdQ = kOffdS + kTileBytes;       // 16 KB: with dropout, each worker warp's 2 KB keep-byte exchange
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
template <bool kDocs, int kD, bool kNoDQ = false, bool kDrop = false>
__global__ void __launch_bounds__(kNoDQ ? bwd::kThreadsNoDQ : bwd::kThreads, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdO,
                const AttnBwdParams p, const AttnDrop drop) {
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
      // dropout: a thread (kv row x 64 query columns) holds the transpose of the Philox layout (one call = 16 keys of
      // one query). The 16 lanes that share kv / 16 make the 64 calls of their query columns, 4 each, and swap the keep
      // bytes through the warp's 2 KB of shared memory (a 128 B line per kv row, 16 B slots XOR-swizzled by the row:
      // the stores and the v4 loads are free of bank conflicts). zr[w] byte j: query column 4 w + j. Made before the
      // wait for S^T, under the MMAs.
      uint32_t zr[16];
      if constexpr (kDrop) {
        const int hh = lane_id() >> 4, L = lane_id() & 15;
        const uint32_t bh = b * p.Hq + hk * G + s / steps_per_head;
        const uint32_t blk = smem_u32(smem + kOffdQ) + (warp - 4) * 2048;
        uint32_t zk[4][4];   // [call j: query column 4 L + j][word w: kv rows 4 w .. 4 w + 3 of the 16]
#pragma unroll
        for (int j = 0; j < 4; ++j) drop_keep16(drop, kv >> 4, q0 + grp * 64 + 4 * L + j, bh, zk[j]);
#pragma unroll
        for (int w = 0; w < 4; ++w) {   // 4 x 4 byte transpose: word bb -> kv row 4 w + bb, byte j = call j
          const uint32_t a01l = __byte_perm(zk[0][w], zk[1][w], 0x5140), a01h = __byte_perm(zk[0][w], zk[1][w], 0x7362);
          const uint32_t a23l = __byte_perm(zk[2][w], zk[3][w], 0x5140), a23h = __byte_perm(zk[2][w], zk[3][w], 0x7362);
          const uint32_t tw[4] = {__byte_perm(a01l, a23l, 0x5410), __byte_perm(a01l, a23l, 0x7632),
                                  __byte_perm(a01h, a23h, 0x5410), __byte_perm(a01h, a23h, 0x7632)};
#pragma unroll
          for (int bb = 0; bb < 4; ++bb) {
            const int m = 4 * w + bb;
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(blk + m * 128 + (((hh * 4 + (L >> 2)) ^ (m & 7)) << 4) + (L & 3) * 4),
                         "r"(tw[bb]) : "memory");
          }
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 4; ++k)
          asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                       : "=r"(zr[4 * k]), "=r"(zr[4 * k + 1]), "=r"(zr[4 * k + 2]), "=r"(zr[4 * k + 3])
                       : "r"(blk + L * 128 + (((hh * 4 + k) ^ (L & 7)) << 4)) : "memory");
      }
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
      // P^T -> the first 32 of the 64 X columns this warp has just read (no other warp touches them); with dropout
      // (P o Z)^T, the A operand of dV (pr itself stays undropped for dS)
      if constexpr (kDrop) {
        uint32_t pz[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) pz[k] = pr[k] & drop_pair_mask(zr[k / 2], (k & 1) * 2);
        tmem_st_32x32(tXw, pz);
      } else {
        tmem_st_32x32(tXw, pr);
      }
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
          if constexpr (kDrop) {   // dS = P o (Z / (1 - p) o dP - delta)
            const uint32_t zw = zr[c * 8 + i / 4];
#pragma unroll
            for (int e = 0; e < 4; ++e) dv[i + e] &= drop_elem_mask(zw, e);
          }
          const float dsc = kDrop ? p.scale * drop.scale : p.scale;
          const float ds0 = bf16_lo(p01) * fmaf(__uint_as_float(dv[i]), dsc, -d4.x);
          const float ds1 = bf16_hi(p01) * fmaf(__uint_as_float(dv[i + 1]), dsc, -d4.y);
          const float ds2 = bf16_lo(p23) * fmaf(__uint_as_float(dv[i + 2]), dsc, -d4.z);
          const float ds3 = bf16_hi(p23) * fmaf(__uint_as_float(dv[i + 3]), dsc, -d4.w);
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
      if (kDrop && grp == 0) {   // dV = (P o Z)^T dO / (1 - p)
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * drop.scale);
      }
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

// Tile classification of a 128-row query tile starting at q0 (attn_bwd_dq_kernel): the kv tiles it visits are
// [j_begin, j_begin + n_kv) — up to max(P, q0 + 128), and, with packed documents, from the start of the first row's
// document on; a visited tile needs no element test when every (q, kv) pair of it is visible and in range.
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

// ------------------------------------------------------------------------------------------------
// Deterministic dQ (torch.use_deterministic_algorithms): CTA = (128 query rows, 1 query head), the forward's structure.
// The CTA walks the visible kv tiles of its rows in ascending order (q_tile_kv_range, q_tile_full)
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

template <bool kDocs, int kD, bool kDrop = false>
__global__ void __launch_bounds__(bwdq::kThreads, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdO,
                   const AttnBwdParams p, __nv_bfloat16* __restrict__ dq, int64_t lddq, const AttnDrop drop) {
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
  // grid = (query heads, batch, query tiles): the tile index runs backwards, so the longest tiles are dispatched first
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
        if (!full_tile) {   // the visible keys of a row are one interval of the tile's columns (see attn_fwd2_kernel)
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
        if constexpr (kDrop) {   // dS = P o (Z / (1 - p) o dP - delta): Z of keys kv0 + 32 c .. kv0 + 32 c + 31
          uint32_t z[8];
          drop_keep16(drop, (kv0 + c * 32) >> 4, q, b * p.Hq + h, *reinterpret_cast<uint32_t(*)[4]>(&z[0]));
          drop_keep16(drop, (kv0 + c * 32 + 16) >> 4, q, b * p.Hq + h, *reinterpret_cast<uint32_t(*)[4]>(&z[4]));
          tmem_ld_32x32(tmem_dP + lane_off + c * 32, dv);
          tmem_wait_ld_regs(dv);
#pragma unroll
          for (int i = 0; i < 32; ++i) dv[i] &= drop_elem_mask(z[i / 4], i & 3);
        } else {
          tmem_ld_32x32(tmem_dP + lane_off + c * 32, dv);
          tmem_wait_ld_regs(dv);
        }
        const float dsc = kDrop ? p.scale * drop.scale : p.scale;
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const uint32_t p01 = pr[c * 16 + i / 2];
          dsr[i / 2] = pack_bf16(bf16_lo(p01) * fmaf(__uint_as_float(dv[i]), dsc, -dlt),
                                 bf16_hi(p01) * fmaf(__uint_as_float(dv[i + 1]), dsc, -dlt));
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

// dropout_p -> the kernels' dropout descriptor; *on = false when t = round(256 p) is 0 (the plain kernels run)
static int make_attn_drop(float dropout_p, uint64_t seed, uint64_t offset, AttnDrop* d, bool* on) {
  if (!(dropout_p >= 0.f && dropout_p < 1.f)) return set_error(LLAMAX_ERR_ARG, "attention: dropout_p must be in [0, 1)");
  const int t = (int)lrintf(dropout_p * 256.f);
  d->key0 = (uint32_t)seed;
  d->key1 = (uint32_t)(seed >> 32);
  d->call = (uint32_t)(offset / 4);
  d->t4 = t >= 256 ? 0xffffffffu : (uint32_t)t * 0x01010101u;
  d->scale = t >= 256 ? 0.f : 256.f / (float)(256 - t);
  *on = t > 0;
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

}  // extern "C"

template <bool kDrop>
static int attn_fwd_launch(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const AttnFwdParams& p,
                           int64_t B, int64_t S, int32_t Hq, int32_t D, const AttnDrop& drop, cudaStream_t stream) {
  int rc;
  const int n_pairs = (int)((ceil_div(S, fwd::kTile) + 1) / 2);
  if (p.doc_start) {   // packed documents: one CTA per pair of query tiles
    auto kern = D == 128 ? attn_fwd2_kernel<128, kDrop> : attn_fwd2_kernel<64, kDrop>;
    if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), fwd::kSmemBytes2, "attn_fwd: cudaFuncSetAttribute"))) return rc;
    dim3 grid(Hq, (unsigned)B, (unsigned)n_pairs);
    kern<<<grid, fwd::kThreads, fwd::kSmemBytes2, stream>>>(tq, tk, tv, p, drop);
  } else {   // persistent: one CTA per SM over a static item list
    auto kern = D == 128 ? attn_fwd5_kernel<128, kDrop> : attn_fwd5_kernel<64, kDrop>;
    if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), fwd::kSmemBytes5, "attn_fwd: cudaFuncSetAttribute"))) return rc;
    const int64_t n_items = (int64_t)n_pairs * B * Hq;
    const int grid = (int)std::min<int64_t>(n_items, sm_count());
    kern<<<grid, fwd::kThreads, fwd::kSmemBytes5, stream>>>(tq, tk, tv, p, n_pairs, drop);
  }
  LX_CHECK_LAUNCH("attn_fwd");
  return 0;
}

static int attn_fwd_run(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o,
                        int64_t ldo, void* lse, int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D,
                        int64_t prefix_len, const void* prefix_len_b, const void* doc_start, float scale,
                        const AttnDrop& drop, bool drop_on, void* stream) {
  if (!q || !k || !v || !o || !lse) return set_error(LLAMAX_ERR_ARG, "attn_fwd: null pointer");
  int rc = check_attn_args(B, S, Hq, Hkv, D, prefix_len, "attn_fwd");
  if (rc) return rc;
  if (ldq % 8 || ldk % 8 || ldv % 8 || ldo % 8) return set_error(LLAMAX_ERR_ARG, "attn_fwd: pitches must be multiples of 8");
  CUtensorMap tq, tk, tv;
  if ((rc = make_head_tmap(&tq, q, ldq, B, S, Hq, D, fwd::kTile))) return rc;
  if ((rc = make_head_tmap(&tk, k, ldk, B, S, Hkv, D, fwd::kTile))) return rc;
  if ((rc = make_head_tmap(&tv, v, ldv, B, S, Hkv, D, fwd::kTile))) return rc;
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
  return drop_on ? attn_fwd_launch<true>(tq, tk, tv, p, B, S, Hq, D, drop, (cudaStream_t)stream)
                 : attn_fwd_launch<false>(tq, tk, tv, p, B, S, Hq, D, drop, (cudaStream_t)stream);
}

extern "C" {

int llamax_attn_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o,
                    int64_t ldo, void* lse, int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D,
                    int64_t prefix_len, const void* prefix_len_b, const void* doc_start, float scale, void* stream) {
  return attn_fwd_run(q, ldq, k, ldk, v, ldv, o, ldo, lse, B, S, Hq, Hkv, D, prefix_len, prefix_len_b, doc_start, scale,
                      AttnDrop{}, false, stream);
}

int llamax_attn_fwd_dropout(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o,
                            int64_t ldo, void* lse, int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D,
                            int64_t prefix_len, const void* prefix_len_b, const void* doc_start, float scale,
                            float dropout_p, uint64_t seed, uint64_t offset, void* stream) {
  AttnDrop drop;
  bool on;
  const int rc = make_attn_drop(dropout_p, seed, offset, &drop, &on);
  if (rc) return rc;
  return attn_fwd_run(q, ldq, k, ldk, v, ldv, o, ldo, lse, B, S, Hq, Hkv, D, prefix_len, prefix_len_b, doc_start, scale,
                      drop, on, stream);
}

}  // extern "C"

template <bool kDrop>
static auto bwd_kernel_for(bool det, bool docs, int D) {
  return det ? (docs ? (D == 128 ? attn_bwd_kernel<true, 128, true, kDrop> : attn_bwd_kernel<true, 64, true, kDrop>)
                     : (D == 128 ? attn_bwd_kernel<false, 128, true, kDrop> : attn_bwd_kernel<false, 64, true, kDrop>))
             : (docs ? (D == 128 ? attn_bwd_kernel<true, 128, false, kDrop> : attn_bwd_kernel<true, 64, false, kDrop>)
                     : (D == 128 ? attn_bwd_kernel<false, 128, false, kDrop> : attn_bwd_kernel<false, 64, false, kDrop>));
}

template <bool kDrop>
static auto bwd_dq_kernel_for(bool docs, int D) {
  return docs ? (D == 128 ? attn_bwd_dq_kernel<true, 128, kDrop> : attn_bwd_dq_kernel<true, 64, kDrop>)
              : (D == 128 ? attn_bwd_dq_kernel<false, 128, kDrop> : attn_bwd_dq_kernel<false, 64, kDrop>);
}

// dq_accum == NULL: deterministic mode (attn_bwd_dq_kernel writes dq, attn_bwd_kernel<.., kNoDQ> dk / dv)
static int attn_bwd_run(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                        const void* o, int64_t ldo, const void* lse, const void* dout, int64_t lddo, void* dq,
                        int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, void* dq_accum, void* delta,
                        int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D, int64_t prefix_len,
                        const void* prefix_len_b, const void* doc_start, const void* doc_end, float scale,
                        const void* rope_inverse, const AttnDrop& drop, bool drop_on, void* stream) {
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
  auto kern = drop_on ? bwd_kernel_for<true>(det, doc_start != nullptr, D) : bwd_kernel_for<false>(det, doc_start != nullptr, D);
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
  kern<<<grid, det ? bwd::kThreadsNoDQ : bwd::kThreads, bwd::kSmemBytes, st>>>(tq, tk, tv, tdo, p, drop);
  LX_CHECK_LAUNCH("attn_bwd");
  if (det) {
    auto kdq = drop_on ? bwd_dq_kernel_for<true>(doc_start != nullptr, D) : bwd_dq_kernel_for<false>(doc_start != nullptr, D);
    if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kdq), bwdq::kSmemBytes, "attn_bwd: cudaFuncSetAttribute")))
      return rc;
    dim3 qgrid(Hq, (unsigned)B, (unsigned)ceil_div(S, bwdq::kTile));
    kdq<<<qgrid, bwdq::kThreads, bwdq::kSmemBytes, st>>>(tq, tk, tv, tdo, p, (__nv_bfloat16*)dq, lddq, drop);
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
                      B, S, Hq, Hkv, D, prefix_len, prefix_len_b, doc_start, doc_end, scale, rope_inverse, AttnDrop{},
                      false, stream);
}

int llamax_attn_bwd_dropout(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                            const void* o, int64_t ldo, const void* lse, const void* dout, int64_t lddo, void* dq,
                            int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, void* dq_accum, void* delta,
                            int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D, int64_t prefix_len,
                            const void* prefix_len_b, const void* doc_start, const void* doc_end, float scale,
                            const void* rope_inverse, float dropout_p, uint64_t seed, uint64_t offset, void* stream) {
  AttnDrop drop;
  bool on;
  int rc = make_attn_drop(dropout_p, seed, offset, &drop, &on);
  if (rc) return rc;
  if (!dq_accum) return set_error(LLAMAX_ERR_ARG, "attn_bwd: null pointer");
  return attn_bwd_run(q, ldq, k, ldk, v, ldv, o, ldo, lse, dout, lddo, dq, lddq, dk, lddk, dv, lddv, dq_accum, delta,
                      B, S, Hq, Hkv, D, prefix_len, prefix_len_b, doc_start, doc_end, scale, rope_inverse, drop, on,
                      stream);
}

int llamax_attn_bwd_deterministic(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                                  const void* o, int64_t ldo, const void* lse, const void* dout, int64_t lddo, void* dq,
                                  int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, void* delta, int64_t B,
                                  int64_t S, int32_t Hq, int32_t Hkv, int32_t D, int64_t prefix_len,
                                  const void* prefix_len_b, const void* doc_start, const void* doc_end, float scale,
                                  const void* rope_inverse, void* stream) {
  return attn_bwd_run(q, ldq, k, ldk, v, ldv, o, ldo, lse, dout, lddo, dq, lddq, dk, lddk, dv, lddv, nullptr, delta,
                      B, S, Hq, Hkv, D, prefix_len, prefix_len_b, doc_start, doc_end, scale, rope_inverse, AttnDrop{},
                      false, stream);
}

int llamax_attn_bwd_deterministic_dropout(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v,
                                          int64_t ldv, const void* o, int64_t ldo, const void* lse, const void* dout,
                                          int64_t lddo, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv,
                                          int64_t lddv, void* delta, int64_t B, int64_t S, int32_t Hq, int32_t Hkv,
                                          int32_t D, int64_t prefix_len, const void* prefix_len_b,
                                          const void* doc_start, const void* doc_end, float scale,
                                          const void* rope_inverse, float dropout_p, uint64_t seed, uint64_t offset,
                                          void* stream) {
  AttnDrop drop;
  bool on;
  const int rc = make_attn_drop(dropout_p, seed, offset, &drop, &on);
  if (rc) return rc;
  return attn_bwd_run(q, ldq, k, ldk, v, ldv, o, ldo, lse, dout, lddo, dq, lddq, dk, lddk, dv, lddv, nullptr, delta,
                      B, S, Hq, Hkv, D, prefix_len, prefix_len_b, doc_start, doc_end, scale, rope_inverse, drop, on,
                      stream);
}

}  // extern "C"
