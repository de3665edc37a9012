// vdb200 — flash-style scaled-dot-product attention on tcgen05/TMEM (sm_100a).
//
// Replaces the reference's materialised  sim = q k^T * d^-1/2 ; softmax ; attn v  of
// CrossAttention.forward (lib/model_zoo/attention.py:178-192) — self-attention N = M in
// {4096,1024,256,64}, d_head in {40,80,160}; cross-attention M = 77 (text) / 257 (image) /
// n*257 (multi-image) — and the CLIP encoder attention (d_head 64, optional causal mask).
//
// One CTA = one (q-tile of 128 rows, head, batch).  192 threads:
//   warp 0    : TMA producer (Q once; K and V^T tiles through two independent 2-stage rings)
//   warp 1    : MMA issuer   (S_j = Q K_j^T into double-buffered TMEM; O += P_j V_j into TMEM)
//   warps 2-5 : online softmax in fp32 registers (one query row per thread), P_j -> bf16 ->
//               128B-swizzled shared memory (double buffered), lazy O rescale in TMEM, final
//               normalise + store.
// Operand layouts (all K-major, 128B swizzle, written by the projection GEMMs):
// Batch b occupies rows [b*q_bs, b*q_bs+Nq) of Q/O, rows [b*kv_bs, +Nk) of K, columns [b*kv_bs, +Nk) of Vt.
//   Q  [B*Nq, ldq]  head h at columns q_col0 + h*DK .. (+DK, zero padded beyond d_head)
//   K  [B*Nk, ldk]  head h at columns k_col0 + h*DK ..
//   Vt [H*DVP, >=B*Nk]  row h*DVP + c = channel c of head h (zero rows beyond d_head), column b*Nk + j
//   O  [B*Nq, ldo]  head h at columns h*dv .. (+dv)   (dense, feeds to_out)
#include "common.cuh"
#include "host_util.h"
#include <cstdlib>
#include <type_traits>

namespace vdb {


constexpr int kBQ = 128;   // query rows per CTA
constexpr int kMaxKvStages = 4;
constexpr float kRescaleThreshold = 8.0f;  // in log2 units (P stays <= 2^8)

struct alignas(64) AttnParams {
  CUtensorMap tmQ;   // 2D (cols, rows) box (64, 128)
  CUtensorMap tmK;   // 2D (cols, rows) box (64, 128)
  CUtensorMap tmV;   // 2D (kv, H*DVP) box (64, DVP)
  int Nq, Nk;        // per-batch query / key counts
  int q_bs, kv_bs;   // per-batch row stride of Q/out, row (K) / column (Vt) stride of the keys (kv_bs % 8 == 0)
  int q_col0, k_col0;
  int dv;            // valid head channels (<= DVP)
  int causal;
  float scale_log2;  // d^-1/2 * log2(e)
  __nv_bfloat16* out;
  long long ldo;
  unsigned long long* timeline;   // debug (-DVDB_TIMELINE): per-tile role timestamps of CTA (0,0,0); null = off
  const int* kv_len;              // per-batch key counts [B] of the KL = 1 kernels, clamped to [1, Nk]
};

// Debug build only (tools/attention_timeline.py): globaltimer stamps of one softmax warp (warp 2: lane quarter 2, first
// half of the columns) and of the MMA issuer, 16 slots per kv tile, first 16 tiles of CTA (0,0,0).
//   softmax: 0 wants S_j, 1 S_j ready, 2 scores in registers + own max, 3 max exchanged, 4 exp2 + P stored,
//            5 O settled / rescaled, 6 arrived on p_full          MMA: 8 wants P_j, 9 P_j ready, 10 next S issued, 11 PV_j issued
#ifdef VDB_TIMELINE
#define VDB_ATL(slot, j, who) do { if (p.timeline && (who) && (blockIdx.x | blockIdx.y | blockIdx.z) == 0 && (j) < 16) p.timeline[(j) * 16 + (slot)] = gtime(); } while (0)
#else
#define VDB_ATL(slot, j, who) do { } while (0)
#endif

// SB = S accumulator buffers in TMEM (1 or 2), PB = P buffers in smem (1 or 2). SB = PB = 1 keeps the CTA at
// <= 110 KB smem / 256 TMEM columns so TWO CTAs share an SM: one CTA's softmax (MUFU-bound) overlaps the other's MMAs.
// SW = softmax warps per TMEM lane quarter (1 or 2).  With SW = 2 the two warps of a quarter split every BKV-column
// S tile (BKV/2 columns each) and the O columns; they exchange the row max once per tile through shared memory.  One
// softmax warp per SM sub-partition was measured to be instruction-latency bound (the exp pipe was ~30 % busy).
// BKV = kv columns per tile (64 or 128).  BKV = 64 halves the S / P buffers, so S and P can BOTH be double buffered
// inside 256 TMEM columns / < 113 KB shared memory and two CTAs still share an SM: with a single S buffer the softmax
// warps of a CTA sat in mbar_wait(s_full) for 29 % of all warp samples (profiles/r01_ncu_hot_lines_v7.txt) because
// S_{j+1} can only be issued once every warp is done with S_j.
template <int DK, int DVP, int BKV>
constexpr size_t attention_smem_bytes(int kv_stages, int pb) {
  return (DK / 64) * kBQ * 128 + kv_stages * ((DK / 64) * BKV * 128 + (BKV / 64) * DVP * 128) + pb * ((BKV / 64) * kBQ * 128) +
         24 * 8 + (512 + 256) * 4 + 1024;
}
template <int DK, int DVP, int BKV, int KV_STAGES, int SB, int PB>
constexpr int attention_ctas_per_sm() {   // by TMEM columns (512 per SM) and shared memory (227 KB + 1 KB reserved per CTA)
  constexpr int cols = SB * BKV + (DVP <= 64 ? 64 : (DVP <= 128 ? 128 : 256));
  constexpr size_t smem = attention_smem_bytes<DK, DVP, BKV>(KV_STAGES, PB);
  return (cols <= 128 && smem <= 75 * 1024) ? 3 : ((cols <= 256 && smem <= 113 * 1024) ? 2 : 1);
}

// KL = 1: per-batch key counts p.kv_len (vdb_attention_keylen_bf16); KL = 0 compiles to the kernel without them.
template <int DK, int DVP, int BKV, int KV_STAGES, int SB, int PB, int SW, int KL>
__global__ void __launch_bounds__(64 + 128 * SW, attention_ctas_per_sm<DK, DVP, BKV, KV_STAGES, SB, PB>())
attention_kernel(const __grid_constant__ AttnParams p) {
  constexpr int kBKV = BKV;
  constexpr int KA = DK / 64;                      // 64-wide K atoms of the QK^T reduction
  constexpr int KVA = BKV / 64;                    // 64-kv atoms per tile (K dimension of the PV product)
  constexpr uint32_t kQBytes = KA * kBQ * 128;     // Q tile
  constexpr uint32_t kKBytes = KA * kBKV * 128;    // one K stage
  constexpr uint32_t kVAtom = DVP * 128;           // one 64-kv atom of V^T
  constexpr uint32_t kVBytes = KVA * kVAtom;       // one V stage (BKV kv)
  constexpr uint32_t kPBytes = KVA * kBQ * 128;    // one P buffer (128 x BKV bf16)
  constexpr uint32_t kOCols = DVP <= 64 ? 64 : (DVP <= 128 ? 128 : 256);
  constexpr uint32_t kTmemCols = (SB * BKV + kOCols <= 128) ? 128 : ((SB * BKV + kOCols <= 256) ? 256 : 512);
  static_assert(BKV == 64 || BKV == 128, "kv tile");
  static_assert(KV_STAGES >= 1 && KV_STAGES <= kMaxKvStages, "kv stages");
  static_assert(SB * BKV + DVP <= 512, "TMEM budget");
  static_assert(kVAtom % 1024 == 0, "V atom must keep 1024B alignment");
  static_assert(DVP % 16 == 0 && DVP <= 256, "invalid UMMA N for PV");

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + kQBytes;
  uint8_t* sV = sK + KV_STAGES * kKBytes;
  uint8_t* sP = sV + KV_STAGES * kVBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + PB * kPBytes);
  uint64_t* q_full = bars;            // 1
  uint64_t* k_full = bars + 1;        // [kMaxKvStages]
  uint64_t* k_empty = bars + 5;       // [kMaxKvStages]
  uint64_t* v_full = bars + 9;        // [kMaxKvStages]
  uint64_t* v_empty = bars + 13;      // [kMaxKvStages]
  uint64_t* s_full = bars + 17;       // [2]
  uint64_t* p_full = bars + 19;       // [PF] (count 4 * SW: one arrive per softmax warp)
  uint64_t* pv_done = bars + 21;      // 1
  // BKV == 64 skips the pv_done wait on tiles without a rescale, so a fast softmax warp may arrive for tile j+1 before
  // a slow one arrived for tile j (never further ahead: S_{j+2} is issued after p_full(j) completes): two barriers.
  constexpr int PF = (BKV == 64) ? 2 : 1;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 22);
  float* sxm = reinterpret_cast<float*>(bars + 24);   // [2 parity][2 halves][128 rows] partial row max (SW == 2)
  float* sxl = sxm + 512;                              // [2 halves][128 rows] partial row sums (SW == 2)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * kBQ;
  const int head = blockIdx.y;
  const int b = blockIdx.z;

  int nk = 0;        // keys of this batch item (KL = 1; the KL = 0 kernels read p.Nk, a constant-bank operand)
  int ntiles = (p.Nk + kBKV - 1) / kBKV;
  if (p.causal) ntiles = min(ntiles, (q0 + kBQ + kBKV - 1) / kBKV);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmQ);
    tma_prefetch_desc(&p.tmK);
    tma_prefetch_desc(&p.tmV);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < KV_STAGES; ++s) {
      mbar_init(&k_full[s], 1); mbar_init(&k_empty[s], 1);
      mbar_init(&v_full[s], 1); mbar_init(&v_empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) mbar_init(&s_full[s], 1);
    for (int s = 0; s < PF; ++s) mbar_init(&p_full[s], 4 * SW);
    mbar_init(pv_done, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<kTmemCols>(tmem_holder);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  pdl_launch_dependents();
  pdl_wait();
  if constexpr (KL) {
    // the batch item's own key count (read after the wait: an earlier kernel may have written it): the tiles past it are
    // never loaded and the last tile masks the columns past it, exactly like the columns past Nk
    nk = min(max(__ldg(p.kv_len + b), 1), p.Nk);
    ntiles = (nk + kBKV - 1) / kBKV;
    if (p.causal) ntiles = min(ntiles, (q0 + kBQ + kBKV - 1) / kBKV);
  }
  const uint32_t tmem_S = tmem_base;             // SB x BKV columns
  const uint32_t tmem_O = tmem_base + SB * BKV;  // DVP columns

  if (warp == 0) {
    if (lane == 0) {
      // Q tile
      mbar_arrive_expect_tx(q_full, kQBytes);
      for (int a = 0; a < KA; ++a)
        tma_load_2d(sQ + a * kBQ * 128, &p.tmQ, q_full, p.q_col0 + head * DK + a * 64, b * p.q_bs + q0);
      // K / V rings
      for (int j = 0; j < ntiles; ++j) {
        const int st = j % KV_STAGES;
        const uint32_t ph = (j / KV_STAGES) & 1;
        mbar_wait(&k_empty[st], ph ^ 1);
        mbar_arrive_expect_tx(&k_full[st], kKBytes);
        for (int a = 0; a < KA; ++a)
          tma_load_2d(sK + st * kKBytes + a * kBKV * 128, &p.tmK, &k_full[st], p.k_col0 + head * DK + a * 64,
                      b * p.kv_bs + j * kBKV);
        mbar_wait(&v_empty[st], ph ^ 1);
        mbar_arrive_expect_tx(&v_full[st], kVBytes);
        for (int a = 0; a < KVA; ++a)
          tma_load_2d(sV + st * kVBytes + a * kVAtom, &p.tmV, &v_full[st], b * p.kv_bs + j * kBKV + a * 64, head * DVP);
      }
    }
  } else if (warp == 1) {
    {   // whole warp, one elected lane per tcgen05 instruction (see umma_bf16_ss_w)
      constexpr uint32_t idesc_s = make_idesc_bf16(kBQ, kBKV);
      constexpr uint32_t idesc_o = make_idesc_bf16(kBQ, DVP);
      const int ksteps = (p.dv + 15) / 16;   // K16 steps of QK^T that can hold non-zero channels
      auto issue_S = [&](int j) {
        const int st = j % KV_STAGES;
        mbar_wait(&k_full[st], (j / KV_STAGES) & 1);
        tc_fence_after();
        const uint32_t d = tmem_S + (j % SB) * BKV;
#pragma unroll
        for (int a = 0; a < KA; ++a) {
          const uint64_t qd = make_desc_sw128(smem_u32(sQ + a * kBQ * 128));
          const uint64_t kd = make_desc_sw128(smem_u32(sK + st * kKBytes + a * kBKV * 128));
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (a * 4 + k < ksteps)      // the K16 steps past d_head multiply zero padding (d 80 in DK 128: 5 of 8 steps, d 40: 3 of 4)
              umma_bf16_ss_w(d, qd + 2 * k, kd + 2 * k, idesc_s, (a > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit_w(&k_empty[st]);
        umma_commit_w(&s_full[j % SB]);
      };
      mbar_wait(q_full, 0);
      issue_S(0);
      if (SB == 2 && ntiles > 1) issue_S(1);
      for (int j = 0; j < ntiles; ++j) {
        const int st = j % KV_STAGES;
        VDB_ATL(8, j, lane == 0);
        mbar_wait(&p_full[j % PF], (j / PF) & 1);   // P_j written, O rescaled, S_j consumed
        VDB_ATL(9, j, lane == 0);
        if (SB == 1 && j + 1 < ntiles) issue_S(j + 1);   // single S buffer: free now; queue it ahead of PV_j
        VDB_ATL(10, j, lane == 0);
        mbar_wait(&v_full[st], (j / KV_STAGES) & 1);
        tc_fence_after();
        const uint8_t* pb = sP + (j % PB) * kPBytes;
#pragma unroll
        for (int a = 0; a < KVA; ++a) {
          const uint64_t pd = make_desc_sw128(smem_u32(pb + a * kBQ * 128));
          const uint64_t vd = make_desc_sw128(smem_u32(sV + st * kVBytes + a * kVAtom));
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ss_w(tmem_O, pd + 2 * k, vd + 2 * k, idesc_o, (j > 0 || a > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit_w(&v_empty[st]);
        umma_commit_w(pv_done);
        VDB_ATL(11, j, lane == 0);
        if (SB == 2 && j + 2 < ntiles) issue_S(j + 2);
      }
    }
  } else {
    // ------------------------------ softmax / correction / epilogue ------------------------------
    const int quarter = warp & 3;
    const int hw = (warp - 2) >> 2;              // which softmax warp of the quarter (0 when SW == 1)
    const int r = quarter * 32 + lane;           // query row inside the tile == TMEM lane
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    const int q_idx = q0 + r;
    constexpr int CPW = (BKV / 32) / SW;         // 32-column S chunks per warp and tile
    constexpr int WC = BKV / SW;                 // S columns per warp and tile
    constexpr int OCH = DVP / 16;                // 16-column O chunks
    const int oc_begin = (SW == 1) ? 0 : (hw == 0 ? 0 : (OCH + 1) / 2);
    const int oc_end = (SW == 1) ? OCH : (hw == 0 ? (OCH + 1) / 2 : OCH);
    auto pair_sync = [&] { asm volatile("bar.sync %0, 64;" ::"r"(1 + quarter) : "memory"); };   // the quarter's two warps
    float m_ref = -INFINITY;  // reference max (raw score units)
    float l_sum = 0.f;        // this thread's share of the row sum
    const bool tl_warp = (warp == 2) && (lane == 0);   // (debug timeline)
    (void)tl_warp;
    // One kv tile.  MASKED = this tile needs the validity test (columns past Nk, or the causal mask): the per-element compare /
    // select pairs of the mask were if-converted into EVERY tile's instruction stream (329 of 895 SASS instructions per tile in the
    // d_head 80 kernel) until the masked tile became its own instantiation of the body.
    auto tile_body = [&](const int j, auto masked_tag) {
      constexpr bool need_mask = decltype(masked_tag)::value;
      VDB_ATL(0, j, tl_warp);
      mbar_wait(&s_full[j % SB], (j / SB) & 1);
      tc_fence_after();
      VDB_ATL(1, j, tl_warp);
      const uint32_t ts = tmem_S + (j % SB) * BKV + lane_off;
      const int kv0 = j * kBKV;
      const int nk_b = KL ? nk : p.Nk;
      const int kv_lim = p.causal ? min(nk_b, q_idx + 1) : nk_b;  // valid kv indices are < kv_lim
      // pass 1: row max over this warp's columns.  With SW == 2 a thread owns only 64 columns, so the scores stay in
      // registers for pass 2 and S is read from TMEM once per tile instead of twice.
      float mx = -INFINITY;
      uint32_t keep[SW == 2 ? WC : 1];
      if constexpr (SW == 2) {
        if constexpr (WC == 64) {
          uint32_t v0[32], v1[32];
          tmem_ld32(ts + hw * WC, v0);
          tmem_ld32(ts + hw * WC + 32, v1);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) { keep[i] = v0[i]; keep[32 + i] = v1[i]; }
        } else {
          uint32_t v0[32];
          tmem_ld32(ts + hw * WC, v0);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) keep[i] = v0[i];
        }
        if (need_mask) {
#pragma unroll
          for (int i = 0; i < WC; ++i)
            if (kv0 + hw * WC + i < kv_lim) mx = fmaxf(mx, __uint_as_float(keep[i]));
        } else {
#pragma unroll
          for (int i = 0; i < WC; ++i) mx = fmaxf(mx, __uint_as_float(keep[i]));
        }
      } else {
#pragma unroll 1
        for (int cc = 0; cc < CPW; ++cc) {
          const int c = hw * CPW + cc;
          uint32_t v[32];
          tmem_ld32(ts + c * 32, v);
          tmem_wait_ld();
          if (need_mask) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (kv0 + c * 32 + i < kv_lim) mx = fmaxf(mx, __uint_as_float(v[i]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) mx = fmaxf(mx, __uint_as_float(v[i]));
          }
        }
      }
      VDB_ATL(2, j, tl_warp);
      if (SW == 2) {   // combine with the partner warp's half of the row
        sxm[((j & 1) * 2 + hw) * 128 + r] = mx;
        pair_sync();
        mx = fmaxf(mx, sxm[((j & 1) * 2 + (hw ^ 1)) * 128 + r]);
      }
      VDB_ATL(3, j, tl_warp);
      // lazy rescale decision (warp-uniform because tcgen05.ld/st are warp collectives; identical in both warps
      // of a quarter because they see the same 32 rows)
      const float m_new = fmaxf(m_ref, mx);
      bool rescale = false;
      float factor = 1.f;
      if (j == 0) {
        m_ref = m_new;
      } else {
        const bool want = (m_new - m_ref) * p.scale_log2 > kRescaleThreshold;
        rescale = __any_sync(0xffffffffu, want);
        if (rescale) {
          factor = ex2_mufu((m_ref - m_new) * p.scale_log2);  // m_ref finite for j > 0
          m_ref = m_new;
          l_sum *= factor;
        }
      }
      const float m_scaled = (m_ref == -INFINITY) ? 0.f : m_ref * p.scale_log2;
      // pass 2: P = exp2(s*scale - m), row sum, bf16 -> swizzled smem
      // single P buffer: PV_{j-1} must have finished reading it (and O must be settled) before pass 2
      if (PB == 1 && j > 0) {
        mbar_wait(pv_done, (j - 1) & 1);
        tc_fence_after();
      }
      uint8_t* prow = sP + (j % PB) * kPBytes + r * 128;
      if constexpr (SW == 2) {
        // this warp's columns [hw*WC, +WC): one whole 64-wide K atom of P (WC == 64) or half of the only atom (WC == 32)
        uint8_t* patom = prow + ((hw * WC) / 64) * (kBQ * 128);
        const int chunk0 = ((hw * WC) % 64) / 8;    // first 16-byte chunk inside the 128-byte row
        // the scale / subtract and the row sum run as packed fp32 pairs (FFMA2 / FADD2): the softmax warps are
        // issue-limited next to the MUFU pipe, and the pairs halve those two instruction streams
        const unsigned long long sc2 = pack_f2(p.scale_log2, p.scale_log2), nm2 = pack_f2(-m_scaled, -m_scaled);
        unsigned long long l2 = pack_f2(0.f, 0.f);
#pragma unroll
        for (int q = 0; q < WC / 8; ++q) {          // 8 scores -> one 16-byte chunk
          float e[8];
#pragma unroll
          for (int i = 0; i < 8; i += 2) {
            float xa, xb;
            unpack_f2(fma_f2(pack_f2(__uint_as_float(keep[q * 8 + i]), __uint_as_float(keep[q * 8 + i + 1])), sc2, nm2), xa, xb);
            e[i] = ex2_mufu(xa);
            e[i + 1] = ex2_mufu(xb);
            if (need_mask && !(kv0 + hw * WC + q * 8 + i < kv_lim)) e[i] = 0.f;
            if (need_mask && !(kv0 + hw * WC + q * 8 + i + 1 < kv_lim)) e[i + 1] = 0.f;
            l2 = add_f2(l2, pack_f2(e[i], e[i + 1]));
          }
          const uint4 pk = make_uint4(pack_bf16x2(e[0], e[1]), pack_bf16x2(e[2], e[3]), pack_bf16x2(e[4], e[5]), pack_bf16x2(e[6], e[7]));
          *reinterpret_cast<uint4*>(patom + (((chunk0 + q) ^ (r & 7)) << 4)) = pk;
        }
        {
          float la, lb;
          unpack_f2(l2, la, lb);
          l_sum += la + lb;
        }
      } else {
#pragma unroll 1
        for (int cc = 0; cc < CPW; ++cc) {
          const int c = hw * CPW + cc;
          uint32_t v[32];
          tmem_ld32(ts + c * 32, v);
          tmem_wait_ld();
          float pf[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            float e = ex2_mufu(fmaf(__uint_as_float(v[i]), p.scale_log2, -m_scaled));
            if (need_mask && !(kv0 + c * 32 + i < kv_lim)) e = 0.f;
            pf[i] = e;
            l_sum += e;
          }
          uint8_t* patom = prow + (c >> 1) * (kBQ * 128);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int chunk = (c & 1) * 4 + q;  // 16-byte chunk inside the 128-byte row
            const uint4 pk = make_uint4(pack_bf16x2(pf[q * 8], pf[q * 8 + 1]), pack_bf16x2(pf[q * 8 + 2], pf[q * 8 + 3]),
                                        pack_bf16x2(pf[q * 8 + 4], pf[q * 8 + 5]), pack_bf16x2(pf[q * 8 + 6], pf[q * 8 + 7]));
            *reinterpret_cast<uint4*>(patom + ((chunk ^ (r & 7)) << 4)) = pk;
          }
        }
      }
      VDB_ATL(4, j, tl_warp);
      // O must be settled (PV_{j-1} retired) before it is rescaled / accumulated into again
      // (BKV == 64 variant: the wait is only needed when O is actually rescaled.  The P buffer this tile wrote was last
      //  read by PV_{j-2}, which retired before S_j — MMAs of a CTA complete in issue order and s_full(j) tracks every
      //  MMA issued before it — so a tile without a rescale never has to see PV_{j-1} finish.)
      if (j > 0) {
        if (PB == 2 && (BKV != 64 || rescale || j == ntiles - 1)) {   // (last tile: keeps the epilogue's parity wait sound)
          mbar_wait(pv_done, (j - 1) & 1);
          tc_fence_after();
        }
        if (rescale) {
#pragma unroll 1
          for (int c = oc_begin; c < oc_end; ++c) {   // each warp of the quarter rescales its share of the O columns
            uint32_t o[16];
            tmem_ld16(tmem_O + lane_off + c * 16, o);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * factor);
            tmem_st16(tmem_O + lane_off + c * 16, o);
          }
          tmem_wait_st();
        }
      }
      VDB_ATL(5, j, tl_warp);
      fence_proxy_async_smem();  // P (generic-proxy stores) -> visible to the MMA's async-proxy reads
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[j % PF]);
      VDB_ATL(6, j, tl_warp);
    };
#pragma unroll 1
    for (int j = 0; j < ntiles; ++j) {
      if ((j * kBKV + kBKV > (KL ? nk : p.Nk)) || p.causal) tile_body(j, std::true_type{});
      else tile_body(j, std::false_type{});
    }
    // epilogue: O / l -> bf16
    if (SW == 2) {
      sxl[hw * 128 + r] = l_sum;
      pair_sync();
      l_sum += sxl[(hw ^ 1) * 128 + r];
    }
    mbar_wait(pv_done, (ntiles - 1) & 1);
    tc_fence_after();
    const float inv_l = 1.f / l_sum;
    const bool row_ok = q_idx < p.Nq;
    __nv_bfloat16* orow = p.out + (static_cast<long long>(b) * p.q_bs + q_idx) * p.ldo + head * p.dv;
#pragma unroll 1
    for (int c = oc_begin; c < oc_end; ++c) {
      uint32_t o[16];
      tmem_ld16(tmem_O + lane_off + c * 16, o);
      tmem_wait_ld();
      if (row_ok) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int col = c * 16 + q * 8;
          if (col + 8 <= p.dv) {
            const uint4 pk = make_uint4(
                pack_bf16x2(__uint_as_float(o[q * 8]) * inv_l, __uint_as_float(o[q * 8 + 1]) * inv_l),
                pack_bf16x2(__uint_as_float(o[q * 8 + 2]) * inv_l, __uint_as_float(o[q * 8 + 3]) * inv_l),
                pack_bf16x2(__uint_as_float(o[q * 8 + 4]) * inv_l, __uint_as_float(o[q * 8 + 5]) * inv_l),
                pack_bf16x2(__uint_as_float(o[q * 8 + 6]) * inv_l, __uint_as_float(o[q * 8 + 7]) * inv_l));
            *reinterpret_cast<uint4*>(orow + col) = pk;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<kTmemCols>(tmem_base);
}

// (Round 1 left a "ping-pong" variant here — 2-3 query tiles per CTA taking turns on the MUFU pipe through named barriers, with
// the single S buffer released only after P was written.  First GPU run, round 2: 566 us (G = 2) / 596 us (G = 3) against
// 459 us for the kernel above on the B = 8, N = 4096, d = 40 launch (profiles/r02_visit_a_pending_variants.log): the S round
// trip through the MMA warp stayed on every group's critical path.  Removed; the two-tile kernels below release S early.)

#ifdef VDB_TIMELINE   // two-tile kernel: 24 slots per kv tile (tools/attention_fa_timeline.py)
#define VDB_FTL(slot, j, who) do { if (p.timeline && (who) && (blockIdx.x | blockIdx.y | blockIdx.z) == 0 && (j) < 16) p.timeline[(j) * 24 + (slot)] = gtime(); } while (0)
#else
#define VDB_FTL(slot, j, who) do { } while (0)
#endif

// ---------------------------------------------------------------------------------------------------------------------
// Two-tile kernel for long, unmasked-or-tail-masked contexts at d_head <= 64 (round 2; default for self-attention at
// the 64x64 / 32x32 ... levels where d_head = 40).  Built from the round-1 role timeline: the column-split kernel above
// spends 0.9 us of every 2.05 us tile outside its exp2 phase (S round trip through the MMA warp, TMEM load, row-max
// exchange), and the two CTAs of an SM run those phases in lock step, so the MUFU pipe idles ~45 % of the time.
//   * ONE CTA per SM owns TWO 128-row query tiles (softmax warpgroups 0 / 1, 4 warps each = one warp per TMEM lane quarter).
//   * a thread owns one query ROW and reads its whole 128-column S tile from TMEM into registers ONCE; the S buffer is
//     released to the MMA warp right after that load (s_free), so S_{j+1} = Q K_{j+1}^T is computed underneath the exp2
//     phase of S_j — no row-max exchange, no S round trip on the critical path, single S buffer per warpgroup.
//   * the two warpgroups take strict turns on the MUFU pipe (named-barrier token): while one runs exp2, the other waits
//     for its S, loads it, reduces the row max and (rarely) rescales O.
//   * POLY of every 8 column pairs are exponentiated on the FMA pipe (packed fp32x2 Cody-Waite + cubic, rel. error
//     7.7e-5 << bf16's 2e-3): at d_head 40 the MUFU pipe, not the tensor pipe, is the floor (1.07 G exp2 per launch).
//   * QK^T skips the k-steps whose 16 channels are zero padding (d_head 40: 3 of the 4 K16 steps of the 64-wide atom).
//   * K / V^T tiles are staged once per CTA and used by both warpgroups (half the L2 -> shared-memory traffic per FLOP).
//   TMEM: S0 [0,128) S1 [128,256) O0 [256,320) O1 [320,384).   warps: 0 TMA, 1 MMA, (2, 3 idle), 4-7 warpgroup 0, 8-11 warpgroup 1;
//   the control warpgroup gives its registers away (setmaxnreg.dec 40) and the softmax warpgroups take 232 each: a row's
//   128 scores live in registers across the whole tile.
//   MMA issue order (steady state): PV_0(j), S_0(j+2), PV_1(j), S_1(j+2), ...
// ---------------------------------------------------------------------------------------------------------------------
template <int DVP, int KV_STAGES, int PT = 1>
constexpr size_t attention_fa_smem_bytes() {
  return 2 * kBQ * 128 + KV_STAGES * (128 * 128 + 2 * DVP * 128) + (PT ? 0 : 2 * (2 * kBQ * 128)) + 32 * 8 + 1024;
}

// 2^x for a packed pair on the FMA / ALU pipes (x <= 0 expected; clamped at -126)
VDB_DEVINL void ex2_poly2(float xa, float xb, float& ea, float& eb) {
  xa = fmaxf(xa, -126.0f);
  xb = fmaxf(xb, -126.0f);
  const unsigned long long x2 = pack_f2(xa, xb);
  const unsigned long long magic = pack_f2(12582912.0f, 12582912.0f), nmagic = pack_f2(-12582912.0f, -12582912.0f);
  const unsigned long long one2 = pack_f2(1.0f, 1.0f), mone2 = pack_f2(-1.0f, -1.0f);
  const unsigned long long r2 = add_f2(x2, magic);              // low mantissa bits hold rint(x)
  const unsigned long long t2 = add_f2(r2, nmagic);             // rint(x) as a float
  const unsigned long long f2 = fma_f2(t2, mone2, x2);          // f = x - rint(x) in [-0.5, 0.5]
  unsigned long long p2 = fma_f2(pack_f2(0.0550886838f, 0.0550886838f), f2, pack_f2(0.242604051f, 0.242604051f));
  p2 = fma_f2(p2, f2, pack_f2(0.693276242f, 0.693276242f));
  p2 = fma_f2(p2, f2, pack_f2(0.99992894f, 0.99992894f));
  (void)one2;
  float pa, pb, ra, rb;
  unpack_f2(p2, pa, pb);
  unpack_f2(r2, ra, rb);
  ea = __int_as_float(__float_as_int(pa) + (__float_as_int(ra) << 23));
  eb = __int_as_float(__float_as_int(pb) + (__float_as_int(rb) << 23));
}

//   * ONES (d_head < DVP, i.e. the V^T tile has a zero-padding row): the row sums come out of the tensor core.  The TMA box
//     of a V^T tile covers only the d_head real rows; row d_head of every stage is written ONCE with bf16 ones (the rest of
//     the padding with zeros), so column d_head of O accumulates sum_j P (of the bf16-rounded probabilities the PV product
//     actually uses, rescaled with O for free) and the softmax threads drop their 64 packed adds per tile (~12 % of the loop).
template <int DVP, int KV_STAGES, int POLY, int TOKEN, int ONES>
__global__ void __launch_bounds__(384, 1) attention_fa_kernel(const __grid_constant__ AttnParams p) {
  constexpr int PT = 1;   // P in tensor memory (TS product).  PT = 0 (P through shared memory, SS product) measured the same: 350 vs 347 us
  constexpr int BKV = 128;
  constexpr uint32_t kQBytes = kBQ * 128;          // one warpgroup's Q tile (DK = 64: one K atom)
  constexpr uint32_t kKBytes = BKV * 128;          // one K stage (128 keys x 64 channels)
  constexpr uint32_t kVAtom = DVP * 128;           // one 64-kv atom of V^T
  constexpr uint32_t kVBytes = 2 * kVAtom;         // one V stage
  constexpr uint32_t kPBytes = 2 * kBQ * 128;      // one warpgroup's P buffer (128 x 128 bf16, two 64-kv atoms)
  static_assert(DVP % 16 == 0 && DVP <= 64, "O must fit 64 TMEM columns per warpgroup");
  static_assert(KV_STAGES >= 2 && KV_STAGES <= kMaxKvStages, "kv stages");
  static_assert(kVAtom % 1024 == 0, "V atom must keep 1024B alignment");
  static_assert(POLY >= 0 && POLY <= 4, "poly pairs per 8 pairs");

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                               // [2][16 KB]
  uint8_t* sK = sQ + 2 * kQBytes;                   // [KV_STAGES][16 KB]
  uint8_t* sV = sK + KV_STAGES * kKBytes;           // [KV_STAGES][kVBytes]
  uint8_t* sP = sV + KV_STAGES * kVBytes;           // [2][32 KB]  (PT = 0 only; PT = 1 keeps P in tensor memory)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + (PT ? 0 : 2 * kPBytes));
  uint64_t* q_full = bars;            // 1
  uint64_t* k_full = bars + 1;        // [kMaxKvStages]
  uint64_t* k_empty = bars + 5;       // [kMaxKvStages]
  uint64_t* v_full = bars + 9;        // [kMaxKvStages]
  uint64_t* v_empty = bars + 13;      // [kMaxKvStages]
  uint64_t* s_full = bars + 17;       // [2]
  uint64_t* s_free = bars + 19;       // [2]  (count 4: one arrive per warp of the group once S is in registers)
  uint64_t* p_full = bars + 21;       // [2]  (count 4)
  uint64_t* pv_done = bars + 23;      // [2]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 26);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * (2 * kBQ);
  const int head = blockIdx.y;
  const int b = blockIdx.z;
  const int ntiles = (p.Nk + BKV - 1) / BKV;
  constexpr int KS = (DVP + 15) / 16;              // K16 steps of QK^T that can hold non-zero channels (d_head <= DVP)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmQ);
    tma_prefetch_desc(&p.tmK);
    tma_prefetch_desc(&p.tmV);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < KV_STAGES; ++s) {
      mbar_init(&k_full[s], 1); mbar_init(&k_empty[s], 1);
      mbar_init(&v_full[s], 1); mbar_init(&v_empty[s], 1);
    }
    for (int g = 0; g < 2; ++g) {
      mbar_init(&s_full[g], 1);
      mbar_init(&s_free[g], 4);
      mbar_init(&p_full[g], 4);
      mbar_init(&pv_done[g], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_holder);
  const int vrows = ONES ? p.dv : DVP;              // rows of a V^T atom the TMA box fills
  if (ONES && warp == 3) {
    // static padding rows [d_head, DVP) of every V^T atom: row d_head = ones, the others zero (128-byte rows; the 16-byte-chunk
    // swizzle permutes equal chunks, so the row can be written linearly)
    const int prow = DVP - p.dv;                    // a multiple of 8 rows, starting on an 8-row swizzle group
    for (int i = lane; i < KV_STAGES * 2 * prow * 8; i += 32) {
      const int chunk = i & 7, row = (i >> 3) % prow, atom = (i >> 3) / prow;
      const uint32_t v = (row == 0) ? 0x3F803F80u : 0u;
      *reinterpret_cast<uint4*>(sV + atom * kVAtom + (p.dv + row) * 128 + chunk * 16) = make_uint4(v, v, v, v);
    }
    fence_proxy_async_smem();                       // generic-proxy stores -> visible to the tensor core's async-proxy reads
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  pdl_launch_dependents();
  pdl_wait();

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");
  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(q_full, 2 * kQBytes);
      for (int g = 0; g < 2; ++g)
        tma_load_2d(sQ + g * kQBytes, &p.tmQ, q_full, p.q_col0 + head * 64, b * p.q_bs + q0 + g * kBQ);
      for (int j = 0; j < ntiles; ++j) {
        const int st = j % KV_STAGES;
        const uint32_t ph = (j / KV_STAGES) & 1;
        mbar_wait(&k_empty[st], ph ^ 1);
        mbar_arrive_expect_tx(&k_full[st], kKBytes);
        tma_load_2d(sK + st * kKBytes, &p.tmK, &k_full[st], p.k_col0 + head * 64, b * p.kv_bs + j * BKV);
        mbar_wait(&v_empty[st], ph ^ 1);
        mbar_arrive_expect_tx(&v_full[st], static_cast<uint32_t>(2 * vrows * 128));
        for (int a = 0; a < 2; ++a)
          tma_load_2d(sV + st * kVBytes + a * kVAtom, &p.tmV, &v_full[st], b * p.kv_bs + j * BKV + a * 64, head * DVP);
      }
    }
  } else if (warp == 1) {
    {   // the whole warp runs the issue loop (convergent control flow); one elected lane issues each tcgen05 instruction
      constexpr uint32_t idesc_s = make_idesc_bf16(kBQ, BKV);
      constexpr uint32_t idesc_o = make_idesc_bf16(kBQ, DVP);
      // S_g(j) = Q_g K_j^T; the K stage is released after warpgroup 1's product of that tile
      auto issue_S = [&](int g, int j) {
        const int st = j % KV_STAGES;
        mbar_wait(&k_full[st], (j / KV_STAGES) & 1);   // (already complete for g = 1: returns at once)
        tc_fence_after();
        const uint64_t qd = make_desc_sw128(smem_u32(sQ + g * kQBytes));
        const uint64_t kd = make_desc_sw128(smem_u32(sK + st * kKBytes));
#pragma unroll
        for (int k = 0; k < KS; ++k) umma_bf16_ss_w(tmem_base + g * 128, qd + 2 * k, kd + 2 * k, idesc_s, k > 0 ? 1u : 0u);
        if (g == 1) umma_commit_w(&k_empty[st]);
        umma_commit_w(&s_full[g]);
      };
      // Issue order (steady state): PV_0(j), S_1(j+1), PV_1(j), S_0(j+2), ...  Every S product is queued half a cycle
      // after the s_free arrival it depends on (the group loaded its previous scores long ago), so the only wait of this
      // thread that can block is p_full.  (First version: PV_g(j) was followed by a wait for s_free_g(j+1), i.e. for the
      // group to fetch its NEXT scores, ~0.25 us during which the other group's finished P tile sat unserved; ncu showed the
      // softmax warps spending 37 % of their time waiting for pv_done: profiles/r02_ncu_attention_fa_v1.txt.)
      auto issue_PV = [&](int g, int j) {
        const int st = j % KV_STAGES;
        mbar_wait(&p_full[g], j & 1);                  // P_g(j) written, O_g rescaled
        VDB_FTL(16 + 3 * g, j, lane == 0);
        mbar_wait(&v_full[st], (j / KV_STAGES) & 1);
        tc_fence_after();
#pragma unroll
        for (int a = 0; a < 2; ++a) {
          const uint64_t vd = make_desc_sw128(smem_u32(sV + st * kVBytes + a * kVAtom));
          if constexpr (PT) {
            // P_g(j) in tensor memory: 128 lanes x 64 packed columns at [384 + 64 g, ..); a K16 step reads 8 columns
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_ts_w(tmem_base + 256 + g * 64, tmem_base + 384 + g * 64 + a * 32 + k * 8, vd + 2 * k, idesc_o,
                           (j > 0 || a > 0 || k > 0) ? 1u : 0u);
          } else {
            const uint64_t pd = make_desc_sw128(smem_u32(sP + g * kPBytes + a * kBQ * 128));
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_ss_w(tmem_base + 256 + g * 64, pd + 2 * k, vd + 2 * k, idesc_o, (j > 0 || a > 0 || k > 0) ? 1u : 0u);
          }
        }
        if (g == 1) umma_commit_w(&v_empty[st]);
        umma_commit_w(&pv_done[g]);
        VDB_FTL(17 + 3 * g, j, lane == 0);
      };
      auto next_S = [&](int g, int j) {                // S_g(j) once the group holds S_g(j-1) in registers
        mbar_wait(&s_free[g], (j - 1) & 1);
        tc_fence_after();
        issue_S(g, j);
        VDB_FTL(18 + 3 * g, j - 1, lane == 0);              // (slot of the tile during which it was issued)
      };
      mbar_wait(q_full, 0);
      issue_S(0, 0);
      issue_S(1, 0);
      if (ntiles > 1) next_S(0, 1);
      for (int j = 0; j < ntiles; ++j) {
        issue_PV(0, j);
        if (j + 1 < ntiles) next_S(1, j + 1);
        issue_PV(1, j);
        if (j + 2 < ntiles) next_S(0, j + 2);
      }
    }
  }
  } else {
    // ------------------------------ softmax warpgroup g: one query row per thread ------------------------------
    asm volatile("setmaxnreg.inc.sync.aligned.u32 208;");
    const int g = (warp - 4) >> 2;
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int r = quarter * 32 + lane;            // query row inside the group's tile == TMEM lane
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    const int q_idx = q0 + g * kBQ + r;
    const uint32_t tmem_S = tmem_base + g * 128 + lane_off;
    const uint32_t tmem_O = tmem_base + 256 + g * 64 + lane_off;
    const uint32_t tmem_P = tmem_base + 384 + g * 64 + lane_off;   // PT = 1: this row's 64 packed bf16x2 columns
    (void)tmem_P;
    constexpr int OCH = DVP / 16;                 // 16-column O chunks
    // exp2 token: group g owns the MUFU pipe between token_wait() and token_pass() (128 waiting + 128 arriving threads)
    auto token_wait = [&] { if (TOKEN) asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory"); };
    auto token_pass = [&] { if (TOKEN) asm volatile("bar.arrive %0, 256;" ::"r"(1 + (g ^ 1)) : "memory"); };
    if (g == 1) token_pass();                     // prime the ring: group 0 goes first
    float m_ref = -INFINITY;
    float l_sum = 0.f;
    const uint32_t prow = smem_u32(sP + g * kPBytes + r * 128);   // 32-bit shared address: STS, no generic address math
    const bool tlw = (quarter == 0) && (lane == 0);   // (debug timeline: first warp of each group)
    (void)tlw;
    // One kv tile of this row.  MASKED = the tile holds columns past Nk (only ever the LAST tile): the 128 compare / select
    // pairs of the tail mask were if-converted into EVERY tile's instruction stream (384 of 1026 SASS instructions per tile,
    // profiles/r02_sass_attention_loop.txt) until the masked tile became its own instantiation of the body.
    auto tile_body = [&](const int j, auto masked_tag) {
      constexpr bool MASKED = decltype(masked_tag)::value;
      VDB_FTL(8 * g + 7, j, tlw);
      mbar_wait(&s_full[g], j & 1);
      tc_fence_after();
      VDB_FTL(8 * g + 0, j, tlw);
      uint32_t keep[BKV];
      {
        uint32_t v0[32], v1[32], v2[32], v3[32];
        tmem_ld32(tmem_S, v0);
        tmem_ld32(tmem_S + 32, v1);
        tmem_ld32(tmem_S + 64, v2);
        tmem_ld32(tmem_S + 96, v3);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; ++i) { keep[i] = v0[i]; keep[32 + i] = v1[i]; keep[64 + i] = v2[i]; keep[96 + i] = v3[i]; }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_free[g]);     // the MMA warp may overwrite S with the next tile's scores
      VDB_FTL(8 * g + 1, j, tlw);
      const int kv0 = j * BKV;
      float mx;
      {
        float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
        if constexpr (MASKED) {
#pragma unroll
          for (int i = 0; i < BKV; ++i)
            if (kv0 + i >= p.Nk) keep[i] = 0xff800000u;   // -inf: contributes exp2 = 0 and never wins the max
        }
#pragma unroll
        for (int i = 0; i < BKV; i += 8) {
          m0 = fmaxf(m0, fmaxf(__uint_as_float(keep[i]), __uint_as_float(keep[i + 1])));
          m1 = fmaxf(m1, fmaxf(__uint_as_float(keep[i + 2]), __uint_as_float(keep[i + 3])));
          m2 = fmaxf(m2, fmaxf(__uint_as_float(keep[i + 4]), __uint_as_float(keep[i + 5])));
          m3 = fmaxf(m3, fmaxf(__uint_as_float(keep[i + 6]), __uint_as_float(keep[i + 7])));
        }
        mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
      }
      const float m_new = fmaxf(m_ref, mx);
      bool rescale = false;
      float factor = 1.f;
      if (j == 0) {
        m_ref = m_new;
      } else {
        const bool want = (m_new - m_ref) * p.scale_log2 > kRescaleThreshold;
        rescale = __any_sync(0xffffffffu, want);
        if (rescale) {
          factor = ex2_mufu((m_ref - m_new) * p.scale_log2);
          m_ref = m_new;
          l_sum *= factor;
        }
      }
      const float m_scaled = (m_ref == -INFINITY) ? 0.f : m_ref * p.scale_log2;
      // PV_g(j-1) must have retired: it reads the group's only P buffer and accumulates into O
      VDB_FTL(8 * g + 2, j, tlw);
      if (j > 0) {
        mbar_wait(&pv_done[g], (j - 1) & 1);
        tc_fence_after();
        VDB_FTL(8 * g + 3, j, tlw);
        if (rescale) {
#pragma unroll 1
          for (int c = 0; c < OCH; ++c) {
            uint32_t o[16];
            tmem_ld16(tmem_O + c * 16, o);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * factor);
            tmem_st16(tmem_O + c * 16, o);
          }
          tmem_wait_st();
        }
      }
      {
        token_wait();
        VDB_FTL(8 * g + 4, j, tlw);
        {
          const unsigned long long sc2 = pack_f2(p.scale_log2, p.scale_log2), nm2 = pack_f2(-m_scaled, -m_scaled);
          unsigned long long l2 = pack_f2(0.f, 0.f), l2b = pack_f2(0.f, 0.f);
          uint32_t pk[PT ? 32 : 4];
          (void)pk;
  #pragma unroll
          for (int q = 0; q < BKV / 8; ++q) {          // 8 scores -> one 16-byte chunk of the P row
            float e[8];
  #pragma unroll
            for (int i = 0; i < 8; i += 2) {
              float xa, xb;
              unpack_f2(fma_f2(pack_f2(__uint_as_float(keep[q * 8 + i]), __uint_as_float(keep[q * 8 + i + 1])), sc2, nm2), xa, xb);
              // pair index inside a group of 8 pairs (two chunks): the LAST `POLY` pairs go to the FMA pipe
              const int pair8 = (q & 1) * 4 + (i >> 1);
              if (pair8 >= 8 - POLY) {
                ex2_poly2(xa, xb, e[i], e[i + 1]);
              } else {
                e[i] = ex2_mufu(xa);
                e[i + 1] = ex2_mufu(xb);
              }
              if constexpr (!ONES) {
                if (i & 2) l2b = add_f2(l2b, pack_f2(e[i], e[i + 1])); else l2 = add_f2(l2, pack_f2(e[i], e[i + 1]));
              }
            }
            if constexpr (PT) {
              // packed bf16 pairs -> 32-bit tensor-memory columns [4 q, 4 q + 4) of this lane's P row; stored 32 columns at a time
  #pragma unroll
              for (int i = 0; i < 4; ++i) pk[(q & 7) * 4 + i] = pack_bf16x2(e[2 * i], e[2 * i + 1]);
              if ((q & 7) == 7) tmem_st32(tmem_P + (q >> 3) * 32, pk);
            } else {
              const uint4 v4 = make_uint4(pack_bf16x2(e[0], e[1]), pack_bf16x2(e[2], e[3]), pack_bf16x2(e[4], e[5]), pack_bf16x2(e[6], e[7]));
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(prow + (q >> 3) * (kBQ * 128) + (((q & 7) ^ (r & 7)) << 4)),
                           "r"(v4.x), "r"(v4.y), "r"(v4.z), "r"(v4.w) : "memory");
            }
          }
          if constexpr (!ONES) {
            float la, lb;
            unpack_f2(add_f2(l2, l2b), la, lb);
            l_sum += la + lb;
          }
        }
        VDB_FTL(8 * g + 5, j, tlw);
        if (!(j == ntiles - 1 && g == 1)) token_pass();   // (the ring is primed once: skip the one surplus hand-over)
      }
      if constexpr (PT) tmem_wait_st(); else fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[g]);
      VDB_FTL(8 * g + 6, j, tlw);
    };
    {
      const bool tail = (p.Nk % BKV) != 0;
      const int nfull = tail ? ntiles - 1 : ntiles;
#pragma unroll 1
      for (int j = 0; j < nfull; ++j) tile_body(j, std::false_type{});
      if (tail) tile_body(ntiles - 1, std::true_type{});
    }
    mbar_wait(&pv_done[g], (ntiles - 1) & 1);
    tc_fence_after();
    if constexpr (ONES) {                         // column d_head of O = sum_j P (the ones row of V^T)
      uint32_t o[16];                             // (16 columns from d_head on: element 0 is the sum; the rest is ignored)
      tmem_ld16(tmem_O + p.dv, o);
      tmem_wait_ld();
      l_sum = __uint_as_float(o[0]);
    }
    const float inv_l = 1.f / l_sum;
    const bool row_ok = q_idx < p.Nq;
    __nv_bfloat16* orow = p.out + (static_cast<long long>(b) * p.q_bs + q_idx) * p.ldo + head * p.dv;
#pragma unroll 1
    for (int c = 0; c < OCH; ++c) {
      uint32_t o[16];
      tmem_ld16(tmem_O + c * 16, o);
      tmem_wait_ld();
      if (row_ok) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int col = c * 16 + q * 8;
          if (col + 8 <= p.dv) {
            const uint4 pk = make_uint4(
                pack_bf16x2(__uint_as_float(o[q * 8]) * inv_l, __uint_as_float(o[q * 8 + 1]) * inv_l),
                pack_bf16x2(__uint_as_float(o[q * 8 + 2]) * inv_l, __uint_as_float(o[q * 8 + 3]) * inv_l),
                pack_bf16x2(__uint_as_float(o[q * 8 + 4]) * inv_l, __uint_as_float(o[q * 8 + 5]) * inv_l),
                pack_bf16x2(__uint_as_float(o[q * 8 + 6]) * inv_l, __uint_as_float(o[q * 8 + 7]) * inv_l));
            *reinterpret_cast<uint4*>(orow + col) = pk;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

// (A column-split variant of the kernel above — sixteen softmax warps, the two warps of a TMEM lane quarter sharing a row's 128
// columns as in attention_kernel — was measured at 346-376 us against 329-335 us on the B = 8, N = 4096, d = 40 launch: 43 % more
// instructions per tile (row-max exchange, twice the per-tile bookkeeping) at 60 % issue utilisation and 54 % MUFU utilisation
// (profiles/r02_ncu_attention_fa2.txt).  Its first version also hung: setmaxnreg.inc can only hand out registers of the CTA's
// own launch allocation (20 warps x 96), never of the rest of the SM.  Removed.)

struct AttnArgs {   // what the C ABI received; the tensor maps depend on the kernel variant's kv tile
  const void *Q, *K, *Vt;
  long long ldq, ldk, ldv;
  int B, H, q_bstride, kv_bstride;
};

// debug aid: which kernel family the last attention call on this thread launched (vdb_debug_attention_last)
enum { kAttNone = 0, kAttTwoTile = 1, kAttCols64Dbuf = 2, kAttCols64ThreeCta = 3, kAttCols128 = 4, kAttD80 = 5, kAttD160 = 6,
       kAttKeylen64 = 7, kAttKeylen128 = 8 };
static thread_local int g_att_last = kAttNone;

template <int DK, int DVP, int BKV, int KV_STAGES, int SB, int PB, int SW, int KL = 0>
static int launch_attention(AttnParams& p, const AttnArgs& a, cudaStream_t stream) {
  constexpr size_t smem = attention_smem_bytes<DK, DVP, BKV>(KV_STAGES, PB);
  static_assert(smem <= 227 * 1024, "attention smem budget");
  auto kernel = attention_kernel<DK, DVP, BKV, KV_STAGES, SB, PB, SW, KL>;
  static bool configured = false;
  if (!configured) {
    VDB_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    prefer_max_smem(kernel);
    configured = true;
  }
  int rc = make_tmap_2d(&p.tmQ, a.Q, static_cast<uint64_t>(a.ldq), static_cast<uint64_t>(a.B) * a.q_bstride, a.ldq * 2, 64, kBQ);
  if (rc) return rc;
  rc = make_tmap_2d(&p.tmK, a.K, static_cast<uint64_t>(a.ldk), static_cast<uint64_t>(a.B) * a.kv_bstride, a.ldk * 2, 64, BKV);
  if (rc) return rc;
  rc = make_tmap_2d(&p.tmV, a.Vt, static_cast<uint64_t>(a.B) * a.kv_bstride, static_cast<uint64_t>(a.H) * DVP, a.ldv * 2, 64, DVP);
  if (rc) return rc;
  dim3 grid((p.Nq + kBQ - 1) / kBQ, a.H, a.B);
  g_att_last = KL ? (BKV == 64 ? kAttKeylen64 : kAttKeylen128)
                  : (DK == 192 ? kAttD160 : (DK == 128 ? kAttD80 : (BKV == 128 ? kAttCols128 : (SB == 2 ? kAttCols64Dbuf : kAttCols64ThreeCta))));
  VDB_CUDA_CHECK(launch_pdl(kernel, grid, dim3(64 + 128 * SW), smem, stream, p));
  count_launch();
  return VDB_OK;
}

template <int DVP, int KV_STAGES, int POLY, int TOKEN, int ONES>
static int launch_attention_fa(AttnParams& p, const AttnArgs& a, cudaStream_t stream) {
  constexpr size_t smem = attention_fa_smem_bytes<DVP, KV_STAGES>();
  static_assert(smem <= 227 * 1024, "attention (two-tile) smem budget");
  auto kernel = attention_fa_kernel<DVP, KV_STAGES, POLY, TOKEN, ONES>;
  static bool configured = false;
  if (!configured) {
    VDB_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    prefer_max_smem(kernel);
    configured = true;
  }
  int rc = make_tmap_2d(&p.tmQ, a.Q, static_cast<uint64_t>(a.ldq), static_cast<uint64_t>(a.B) * a.q_bstride, a.ldq * 2, 64, kBQ);
  if (rc) return rc;
  rc = make_tmap_2d(&p.tmK, a.K, static_cast<uint64_t>(a.ldk), static_cast<uint64_t>(a.B) * a.kv_bstride, a.ldk * 2, 64, 128);
  if (rc) return rc;
  rc = make_tmap_2d(&p.tmV, a.Vt, static_cast<uint64_t>(a.B) * a.kv_bstride, static_cast<uint64_t>(a.H) * DVP, a.ldv * 2, 64,
                    ONES ? p.dv : DVP);          // ONES: the box leaves the static padding rows of the stage alone
  if (rc) return rc;
  dim3 grid((p.Nq + 2 * kBQ - 1) / (2 * kBQ), a.H, a.B);
  g_att_last = kAttTwoTile;
  VDB_CUDA_CHECK(launch_pdl(kernel, grid, dim3(384), smem, stream, p));
  count_launch();
  return VDB_OK;
}

template <int DVP, int TOKEN>
static int dispatch_attention_fa2(int poly, AttnParams& p, const AttnArgs& a, cudaStream_t st) {
  // row sums through the ones row of V^T whenever the head has a padding row (VDB_ATT_ONES=0: summed by the softmax threads)
  static const int ones_on = [] { const char* e = getenv("VDB_ATT_ONES"); return (e && e[0] == '0') ? 0 : 1; }();
  // (measured with the ones row, B = 8, N = 4096, d = 40: no MUFU token 316.5 us, four K / V^T stages 316.5 us, default 316.0 us —
  // the tile time is the softmax warpgroup's own instruction stream; profiles/r02_visit_u_attention_token_stages.log)
  if (ones_on && TOKEN == 1 && p.dv < DVP) {
    switch (poly) {
      case 2: return launch_attention_fa<DVP, 3, 2, 1, 1>(p, a, st);
      case 3: return launch_attention_fa<DVP, 3, 3, 1, 1>(p, a, st);
      case 4: return launch_attention_fa<DVP, 3, 4, 1, 1>(p, a, st);
      case 1: return launch_attention_fa<DVP, 3, 1, 1, 1>(p, a, st);
      default: break;
    }
  }
  switch (poly) {
    case 0: return launch_attention_fa<DVP, 3, 0, TOKEN, 0>(p, a, st);
    case 2: return launch_attention_fa<DVP, 3, 2, TOKEN, 0>(p, a, st);
    case 3: return launch_attention_fa<DVP, 3, 3, TOKEN, 0>(p, a, st);
    default: return launch_attention_fa<DVP, 3, 1, TOKEN, 0>(p, a, st);
  }
}
template <int DVP>
static int dispatch_attention_fa(int mode, AttnParams& p, const AttnArgs& a, cudaStream_t st) {
  // mode digits "PT": P = exp2 pairs of every 8 on the FMA pipe (0..3), T = 1 MUFU token between the two groups / 0 free-running
  const int poly = (mode / 10) % 10, token = mode % 10 ? 1 : 0;
  return token ? dispatch_attention_fa2<DVP, 1>(poly, p, a, st) : dispatch_attention_fa2<DVP, 0>(poly, p, a, st);
}

}  // namespace vdb

using namespace vdb;

static unsigned long long* g_att_timeline = nullptr;

extern "C" {

// debug aid (not part of the product ABI; stamps exist only in a -DVDB_TIMELINE build): 16 x 16 u64 device buffer
void vdb_debug_attention_timeline(void* buf) { g_att_timeline = reinterpret_cast<unsigned long long*>(buf); }
// debug aid (host side, not part of the product ABI): kernel family of the last attention launch on this thread —
// 1 two-tile, 2 64-column double-buffered, 3 64-column three-CTA, 4 128-column, 5 d_head 65..80, 6 d_head 81..160,
// 7 key-length 64-column, 8 key-length 128-column; 0 before the first launch
int vdb_debug_attention_last(void) { return g_att_last; }

// Padded head sizes the projection GEMMs must produce for a given d_head (see include/vdb200.h): one (DK, DVP) pair per
// instantiated kernel, (64, 48 | 64), (128, 80) and (192, 160); d_head 81..160 all run on the last one.
int vdb_attention_dk_pad(int d_head) { return d_head <= 64 ? 64 : (d_head <= 80 ? 128 : (d_head <= 160 ? 192 : -1)); }
int vdb_attention_dv_pad(int d_head) {
  if (d_head <= 48) return 48;
  if (d_head <= 64) return 64;
  if (d_head <= 80) return 80;
  if (d_head <= 160) return 160;
  return -1;
}

static int attention_entry(const void* Q, long long ldq, int q_col0, const void* K, long long ldk, int k_col0,
                           const void* Vt, long long ldv, void* out, long long ldo, int B, int H, int Nq, int Nk,
                           int q_bstride, int kv_bstride, int d_head, float scale, int causal, const int* kv_len,
                           void* stream) {
  if (!Q || !K || !Vt || !out || B <= 0 || H <= 0 || Nq <= 0 || Nk <= 0)
    return set_error(VDB_ERR_INVALID, "attention: null/empty argument");
  const int DK = vdb_attention_dk_pad(d_head), DVP = vdb_attention_dv_pad(d_head);
  if (DK < 0 || DVP < 0) return set_error(VDB_ERR_UNSUPPORTED, "attention: d_head %d not supported (<= 160)", d_head);
  if ((d_head % 8) || (ldo % 8) || (ldq % 8) || (ldk % 8) || (ldv % 8))
    return set_error(VDB_ERR_INVALID, "attention: d_head and leading dims must be multiples of 8");
  if (q_bstride <= 0) q_bstride = Nq;
  if (kv_bstride <= 0) kv_bstride = Nk;
  // TMA needs the innermost box coordinate (the kv column of V^T) on a 16-byte boundary
  if (q_bstride < Nq || kv_bstride < Nk || (kv_bstride % 8))
    return set_error(VDB_ERR_INVALID, "attention: need q_bstride >= Nq, kv_bstride >= Nk and kv_bstride %% 8 == 0 (got %d, %d)",
                     q_bstride, kv_bstride);
  AttnParams p;
  memset(&p, 0, sizeof(p));
  const AttnArgs a{Q, K, Vt, ldq, ldk, ldv, B, H, q_bstride, kv_bstride};
  p.Nq = Nq; p.Nk = Nk; p.q_bs = q_bstride; p.kv_bs = kv_bstride; p.q_col0 = q_col0; p.k_col0 = k_col0; p.dv = d_head; p.causal = causal;
  p.kv_len = kv_len;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.out = reinterpret_cast<__nv_bfloat16*>(out);
  p.ldo = ldo;
  p.timeline = g_att_timeline;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  static const int sw = [] { const char* e = getenv("VDB_ATT_SW"); return (e && e[0] == '1') ? 1 : 2; }();
  // 64-column kv tiles for d_head <= 64 (profiles/r01_variants_v8.txt, r01_ncu_attention_variants_v8.txt):
  //   VDB_ATT_BKV=64   double-buffered S and P, two CTAs per SM            (self-attention N = 4096: 470 us vs 458 us default)
  //   VDB_ATT_BKV=643  single S / P buffers in 128 TMEM columns and < 75 KB shared memory: THREE CTAs (24 softmax warps)
  //                    per SM (N = 4096: 491 us; but 31.3 vs 36.8 us on the 77-key text context, whose second 64 keys
  //                    of a 128-column tile are masked padding)
  //   VDB_ATT_BKV=128  the 128-column kernel everywhere
  // default: the three-CTA kernel for short contexts (65..512 keys), the 128-column kernel otherwise
  // VDB_ATT_FA: the two-tile kernel (attention_fa_kernel).  0 = off; otherwise digits "PT": P = exp2 pairs of every 8 on the FMA
  // pipe (0..4), T = 1 MUFU token / 0 free-running.  Without the ones row 11 was best (329 us on the B = 8, N = 4096, d = 40 launch;
  // 1 -> 358, 21 -> 334, 31 -> 334, 10 -> 340: profiles/r02_visit_f_summary.log).
  static const int fa = [] { const char* e = getenv("VDB_ATT_FA"); return e ? atoi(e) : -1; }();
  // (per-batch key counts only exist in the kernel below: the two-tile kernel masks the last tile of Nk)
  if (fa != 0 && !kv_len && DK == 64 && !causal && Nk >= 512 && Nq >= 256 && (Nq % 256) == 0) {
    // default: 3 of 8 pairs on the FMA pipe when the row sums come out of the tensor core (ONES: 315 us; 2 -> 318, 1 -> 340),
    // 1 of 8 otherwise (328 us; profiles/r02_visit_o_attention_ones.log)
    static const int ones_on = [] { const char* e = getenv("VDB_ATT_ONES"); return (e && e[0] == '0') ? 0 : 1; }();
    const int mode = fa < 0 ? ((ones_on && d_head < DVP) ? 31 : 11) : fa;
    if (DVP == 48) return dispatch_attention_fa<48>(mode, p, a, st);
    if (DVP == 64) return dispatch_attention_fa<64>(mode, p, a, st);
  }
  static const int bkv = [] { const char* e = getenv("VDB_ATT_BKV"); const int v = e ? atoi(e) : 0; return (v == 64 || v == 643 || v == 128) ? v : 0; }();
  if (kv_len) {   // the default tile choice below for BERT's d_head 64, with per-batch key counts
    if (DK != 64 || DVP != 64) return set_error(VDB_ERR_UNSUPPORTED, "attention_keylen: d_head %d (needs 49..64)", d_head);
    if (Nk > 64 && Nk <= 512) return launch_attention<64, 64, 64, 2, 1, 1, 2, 1>(p, a, st);
    return launch_attention<64, 64, 128, 2, 1, 1, 2, 1>(p, a, st);
  }
  if (sw == 2) {
    if (bkv == 64 && Nk > 64) {
      if (DK == 64 && DVP == 48) return launch_attention<64, 48, 64, 4, 2, 2, 2>(p, a, st);
      if (DK == 64 && DVP == 64) return launch_attention<64, 64, 64, 3, 2, 2, 2>(p, a, st);
    }
    if ((bkv == 643 && Nk > 64) || (bkv == 0 && Nk > 64 && Nk <= 512)) {
      if (DK == 64 && DVP == 48) return launch_attention<64, 48, 64, 2, 1, 1, 2>(p, a, st);
      if (DK == 64 && DVP == 64) return launch_attention<64, 64, 64, 2, 1, 1, 2>(p, a, st);
    }
    if (DK == 64 && DVP == 48) return launch_attention<64, 48, 128, 2, 1, 1, 2>(p, a, st);   // 2 CTAs / SM, 16 softmax warps / SM
    if (DK == 64 && DVP == 64) return launch_attention<64, 64, 128, 2, 1, 1, 2>(p, a, st);
    if (DK == 128 && DVP == 80) return launch_attention<128, 80, 128, 2, 2, 2, 2>(p, a, st);
    if (DK == 192 && DVP == 160) return launch_attention<192, 160, 128, 1, 2, 2, 2>(p, a, st);
  } else {
    if (DK == 64 && DVP == 48) return launch_attention<64, 48, 128, 2, 1, 1, 1>(p, a, st);
    if (DK == 64 && DVP == 64) return launch_attention<64, 64, 128, 2, 1, 1, 1>(p, a, st);
    if (DK == 128 && DVP == 80) return launch_attention<128, 80, 128, 2, 2, 2, 1>(p, a, st);
    if (DK == 192 && DVP == 160) return launch_attention<192, 160, 128, 1, 2, 2, 1>(p, a, st);
  }
  return set_error(VDB_ERR_UNSUPPORTED, "attention: no kernel for d_head %d", d_head);
}

int vdb_attention_bf16(const void* Q, long long ldq, int q_col0, const void* K, long long ldk, int k_col0,
                       const void* Vt, long long ldv, void* out, long long ldo, int B, int H, int Nq, int Nk,
                       int q_bstride, int kv_bstride, int d_head, float scale, int causal, void* stream) {
  return attention_entry(Q, ldq, q_col0, K, ldk, k_col0, Vt, ldv, out, ldo, B, H, Nq, Nk, q_bstride, kv_bstride, d_head,
                         scale, causal, nullptr, stream);
}

int vdb_attention_keylen_bf16(const void* Q, long long ldq, int q_col0, const void* K, long long ldk, int k_col0,
                              const void* Vt, long long ldv, void* out, long long ldo, int B, int H, int Nq, int Nk,
                              int q_bstride, int kv_bstride, int d_head, float scale, int causal, const int* kv_len,
                              void* stream) {
  if (!kv_len) return set_error(VDB_ERR_INVALID, "attention_keylen: kv_len is null");
  return attention_entry(Q, ldq, q_col0, K, ldk, k_col0, Vt, ldv, out, ldo, B, H, Nq, Nk, q_bstride, kv_bstride, d_head,
                         scale, causal, kv_len, stream);
}

}  // extern "C"
