// vdb200 — persistent tcgen05 implicit-GEMM mainloop (sm_100a).
//
// One kernel family serves every GEMM-shaped stage of the Versatile-Diffusion sampling path:
//   * Linear layers and 1x1 convs on NHWC activations (CrossAttention.to_q/k/v/to_out,
//     FeedForward/GEGLU, SpatialTransformer.proj_in/out — reference lib/model_zoo/attention.py:37-64,
//     152-193, 221-266; AutoencoderKL AttnBlock q/k/v/proj_out — autokl_modules.py:150-202),
//   * 3x3 convolutions as implicit GEMM over 9 filter taps (ResBlock in_layers[2]/out_layers[3],
//     Downsample.op, Upsample.conv — openaimodel.py:89-274; VAE ResnetBlock/Downsample/Upsample —
//     autokl_modules.py:42-141), with the 1x1 skip_connection of a channel-changing ResBlock folded
//     in as extra K segments of the same accumulator.
//
// Structure: grid = #SMs (persistent, static round-robin over output tiles), 320 threads:
//   warp 0   : TMA producer  (cp.async.bulk.tensor 4D box loads of A, 2D box loads of W)
//   warp 1   : MMA issuer    (tcgen05.mma cta_group::1 kind::f16, 128 x BN x 16, fp32 accum in TMEM)
//   warps 2-9: epilogue      (tcgen05.ld -> smem transpose -> bias/act/residual -> coalesced bf16 stores)
// smem ring of STAGES x (A 128x64 bf16 | W BNx64 bf16), both 128B-swizzled K-major; TMEM holds two
// accumulator stages (2 x 256 columns) so the epilogue of tile i overlaps the MMAs of tile i+1.
#include "common.cuh"
#include "host_util.h"

namespace vdb {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // bf16 elements = 128 B = one swizzle row
constexpr int kMaxA = 6;     // A tensor maps per launch
constexpr int kMaxSeg = 12;  // K segments per launch
// threads = 64 + 32 * EW: warp 0 TMA, warp 1 MMA, EW epilogue warps (8, or 16 for the short-K GEMMs whose tiles
// are bound by the epilogue's instruction latency rather than by the mainloop)
constexpr uint32_t kABytes = kBlockM * kBlockK * 2;

struct ASeg {
  int16_t tmap;  // which A tensor map
  int16_t dw;    // W-coordinate shift of this segment (filter tap / parity lattice)
  int16_t dh;    // H-coordinate shift
  int16_t nkb;   // number of 64-channel k-blocks
  int32_t c0;    // first channel coordinate
};

struct alignas(64) IgemmParams {
  CUtensorMap tmA[kMaxA];  // 4D (C, W, H, B) bf16, box (64, TW, TH, TB), SWIZZLE_128B
  CUtensorMap tmB;         // 2D (Ktot, N) bf16, box (64, BN), SWIZZLE_128B (CTA-pair launches: box (64, BN/2))
  CUtensorMap tmO;         // TMA-store epilogues: 4D (N, Wo, Ho, Bo) bf16 output, box (32, bw, bh, bb) = one warp's 32 x 32 chunk, SWIZZLE_64B
  ASeg seg[kMaxSeg];
  int nseg;
  int kb_total;      // total k-blocks over all segments
  int ksplit;        // split-K factor (>=1); >1 => fp32 partial output
  int kb_per_split;  // ceil(kb_total / ksplit)
  int TW, TH, TB;    // M tile = TW*TH*TB = 128 output pixels
  int Wo, Ho, Bo;    // output pixel grid (GEMM view: Wo = M, Ho = Bo = 1)
  int tilesW, tilesH, tilesB, tilesN;
  int N;             // valid output columns (GEGLU: packed columns, output has N/2)
  // epilogue
  const float* bias;          // [bias_rows, N] fp32 or null
  long long bias_bstride;     // 0: shared bias row; else stride between per-batch rows
  int rows_per_batch;         // output pixels per batch element (for bias_bstride != 0)
  const __nv_bfloat16* resid; // [M, ldr] bf16 or null (added after activation)
  long long ldr;
  void* out;                  // bf16 or fp32 [M, ldo]
  long long ldo;
  int out_f32;                // 1: fp32 output
  int act;                    // 0 none, 1 silu, 2 gelu(erf), 3 quick_gelu, 4 geglu (packed halves), 5 gelu(tanh), 6 tanh
  float alpha;                // out = act(alpha * (acc + bias)) + resid
  float* partial;             // split-K: [ksplit, M, N] fp32
  // LayerNorm folded into the GEMM (modes 5 / 6 consume, mode 7 produces; see the epilogue):
  const float* ln_stats;      // [ln_parts][ln_mstat][2] fp32: partial (sum, sum of squares) over column ranges of the normalised rows
  long long ln_mstat;         // rows of the statistics table
  int ln_parts;               // partials per row (what the producer launch reported)
  int ln_on_cols;             // 0: the statistics belong to the OUTPUT ROWS (x is the A operand); 1: to the output COLUMNS (x is B)
  float ln_inv_dim, ln_eps;   // 1 / normalised width, epsilon
  const float* ln_colsum;     // on_cols 0: [N] sum_k W'[n, k];  on_cols 1: [M] (per output row)
  const float* ln_rowbias;    // on_cols 1: [M] beta-term of the output row (null = 0); on_cols 0 the beta term lives in `bias`
  float* stats_out;           // mode 7: [2 * tilesN][M][2] fp32: (sum, sum of squares) of the columns each of the two epilogue
                              // warps of a TMEM lane quarter handled in each N tile, for every OUTPUT row
  int epi_alt;                // 1: the two warps of a TMEM quarter swap chunk parity every tile (odd chunk counts)
  int nfast;                  // 1: N is the fast tile index (tile t -> n = t % tilesN, m = t / tilesN); needs ksplit == 1
  unsigned long long* timeline; // debug: per-tile role timestamps of CTA 0 (null = off)
  unsigned smem_bytes;        // dynamic shared memory of the launch (LN modes check their carve-up against it)
  int chunked;                // 1: every CTA walks a contiguous range of tiles instead of a grid-strided one
};

enum { ACT_NONE = 0, ACT_SILU = 1, ACT_GELU = 2, ACT_QGELU = 3, ACT_GEGLU = 4, ACT_GELU_TANH = 5, ACT_TANH = 6 };

#ifdef VDB_TIMELINE   // debug build only (tools/gemm_timeline.py): per-tile role timestamps of CTA 0
#define VDB_TL(slot, it) do { if (p.timeline && blockIdx.x == 0 && (it) < 8) p.timeline[(it) * 16 + (slot)] = gtime(); } while (0)
#define VDB_TLE(slot, it) do { if (warp == 2 && lane == 0) VDB_TL(slot, it); } while (0)
#else
#define VDB_TL(slot, it) do { } while (0)
#define VDB_TLE(slot, it) do { } while (0)
#endif

// mbarrier wait with a watchdog (CTA-pair kernels): a protocol error between the two CTAs traps after ~2 s instead
// of hanging the device
VDB_DEVINL void mbar_wait_wd(uint64_t* bar, uint32_t parity, int who) {
  uint32_t n = 0;
  unsigned long long t0 = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++n == 4096) {
      t0 = gtime();
    } else if (n > 4096 && (n & 1023) == 0 && gtime() - t0 > 2000000000ull) {
      printf("igemm pair watchdog: block %d thread %d wait %d parity %u\n", blockIdx.x, threadIdx.x, who, parity);
      __trap();
    }
  }
}

VDB_DEVINL float apply_act(float v, int act) {
  switch (act) {
    case ACT_SILU: return silu_f(v);
    case ACT_GELU: return gelu_erf_f(v);
    case ACT_QGELU: return quick_gelu_f(v);
    case ACT_GELU_TANH: return gelu_tanh_f(v);
    case ACT_TANH: return tanhf(v);
    default: return v;
  }
}

// CTAS == 2: the kernel runs as CTA pairs (2-cluster, cta_group::2).  A pair owns a 256 x BN output tile: CTA r stages
// its own 128 rows of A and rows [r*BN/2, (r+1)*BN/2) of the B tile, so the L2 -> shared-memory traffic per FLOP
// drops by ~28 % (BN 160) / 33 % (BN 256) against two independent CTAs and the smaller stage buys two more pipeline
// stages.  MEASURED SLOWER than single CTAs on every UNet shape (conv 64x64 320->320: 73.9 vs 60.2 us in-graph,
// GEMM 32768x320x320: 22.7 vs 16.7 us; profiles/r01_variants_v8.txt), so it stays opt-in (VDB_PAIR=1).  Rank 0 issues the MMAs; every
// TMA of the pair completes on rank 0's full barrier; commits multicast to both CTAs; each CTA drains its own 128
// accumulator lanes with the same epilogue.
// MODE selects the epilogue that is compiled in: 0 = every path (split-K partials, GEGLU, fp32 / ragged / per-row-bias
// tiles), 1 = only the bf16 fast path (act none, alpha 1, N % 32 == 0, one bias row per tile) with the residual of the
// NEXT chunk prefetched, 2 = only GEGLU.  The generic kernel is ~6300 SASS instructions; ncu's source view of the
// K = 320 GEMMs showed 9 % instruction-fetch stalls and 10 % branch-resolve stalls in the epilogue warps, and the
// residual's first use exposed its full load latency (hot lines of the current build: profiles/r01_ncu_hot_lines_v7.txt).
// Modes 3 / 4 are modes 1 / 2 with the tile leaving through shared memory + TMA stores.  Modes 5 / 6 are modes 3 / 4 for a GEMM whose
// input is a LayerNorm: the operand is the RAW activation x and the weights carry gamma (W' = W * gamma), so with the row's mean mu
// and rstd r       LN(x) W^T + b  =  r * (x W'^T  -  mu * s) + c,     s[n] = sum_k W'[n,k],  c[n] = sum_k beta_k W[n,k] + b[n]
// is a rank-1 correction in the epilogue (2 FMAs per element) — the normalised tensor is never written or read.  mu and r come
// from per-32-channel partial sums that the PRODUCER of x wrote from its own epilogue (mode 7 = mode 3 + those sums).  When x is
// the B operand (the transposed V^T projection) the statistics belong to the output columns instead (ln_on_cols).
template <int BN, int STAGES, int CTAS, int EW, int MODE>
__global__ void __launch_bounds__(64 + 32 * EW, 1) igemm_kernel(const __grid_constant__ IgemmParams p) {
  constexpr bool kTmaEpi = MODE >= 3;                 // TMA-store epilogues
  constexpr bool kGegluEpi = MODE == 4 || MODE == 6;
  constexpr bool kLnIn = MODE == 5 || MODE == 6;
  constexpr bool kStatsOut = MODE == 7;
  constexpr int kNumEpiWarps = EW;
  constexpr int kNumEpiThreads = EW * 32;
  constexpr int kWPQ = EW / 4;           // epilogue warps per TMEM lane quarter
  static_assert(EW == 8 || EW == 12 || EW == 16, "");   // 12 / 16 were measured: no gain (DESIGN.md)
  constexpr uint32_t kBBytes = (BN / CTAS) * kBlockK * 2;    // this CTA's share of the B tile
  constexpr uint32_t kStageBytes = kABytes + kBBytes;
  static_assert(kBBytes % 1024 == 0, "B stage must keep 1024B alignment");
  static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "invalid UMMA N");
  static_assert(CTAS == 1 || CTAS == 2, "");
  const uint32_t cta_rank = (CTAS == 2) ? cluster_ctarank() : 0u;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smemA = smem;
  uint8_t* smemB = smem + STAGES * kABytes;
  float* sstage = reinterpret_cast<float*>(smem + STAGES * kStageBytes);   // kNumEpiWarps x 4 KB, 1024-byte aligned: [32][32] fp32
                                                                           // transposition tiles, or 2 x 2 KB bf16 TMA-store tiles
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * kStageBytes + EW * 4096);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;       // [2]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* sbias = reinterpret_cast<float*>(tmem_holder + 4);   // [BN] bias of the current output tile
  float* slnx = sbias + BN;                                   // [BN] LN modes: colsum s (on_cols 0) / column mean (on_cols 1)
  const uint32_t sbias_s = smem_u32(sbias), slnx_s = smem_u32(slnx);   // (shared-space addresses: LDS, not generic LD)
  (void)slnx_s;
  if constexpr (kLnIn) {
    // (BN 256 leaves 912 instead of 1024 bytes of alignment slack; the dynamic window starts 1024-aligned in practice)
    if (reinterpret_cast<uint8_t*>(slnx + BN) > smem_raw + p.smem_bytes) __trap();
  }
  auto epi_bar_sync = [] { asm volatile("bar.sync 1, %0;" ::"n"(EW * 32) : "memory"); };   // the epilogue warps only

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < kMaxA; ++i) tma_prefetch_desc(&p.tmA[i]);
    tma_prefetch_desc(&p.tmB);
    if constexpr (MODE >= 3) tma_prefetch_desc(&p.tmO);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], kNumEpiWarps * CTAS);   // pair: the peer's epilogue warps arrive remotely
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (CTAS == 2) tmem_alloc_pair<512>(tmem_holder); else tmem_alloc<512>(tmem_holder);
  }
  tc_fence_before();
  if constexpr (CTAS == 2) cluster_sync_all(); else __syncthreads();   // pair: the peer's barriers are initialised too
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  pdl_launch_dependents();
  pdl_wait();   // everything above overlapped the previous kernel's tail; global inputs are valid from here

  // scheduling unit = CTAS consecutive M tiles x one N tile; CTA r of a pair takes M tile 2*unit + r (host: tilesM even)
  const int tilesM = p.tilesW * p.tilesH * p.tilesB;
  const int unitsM = tilesM / CTAS;
  const int num_tiles = unitsM * p.tilesN * p.ksplit;
  // Tile walk of this CTA (all three roles use the same bounds): strided (tile c, c + grid, ...) or, p.chunked, a contiguous range.
  // With M as the fast tile index a strided walk changes its N tile every unitsM / grid tiles — every 1.7 tiles on the 64x64-level
  // GEMMs with many N tiles (GEGLU: 10) — and every change reloads the bias / LayerNorm tables behind two barriers; a contiguous
  // range changes it once or twice per launch.
  const int n_ctas = gridDim.x / CTAS, cta_id = blockIdx.x / CTAS;
  const int per_cta = (num_tiles + n_ctas - 1) / n_ctas;
  const int t_first = p.chunked ? cta_id * per_cta : cta_id, t_step = p.chunked ? 1 : n_ctas;
  const int t_end = p.chunked ? min(num_tiles, t_first + per_cta) : num_tiles;

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      const bool flat = (p.tilesH == 1) && (p.tilesB == 1);
      const int step_m = t_step % unitsM, step_r = t_step / unitsM;
      int unit_m = t_first % unitsM, rest = t_first / unitsM;
      // N-fast order (opt-in): the N tiles of one M tile run on neighbouring CTAs at the same time, so an A operand larger
      // than L2 is fetched from DRAM once instead of once per N tile
      const int nf_step_n = p.nfast ? t_step % p.tilesN : 0, nf_step_m = p.nfast ? t_step / p.tilesN : 0;
      int nf_n = p.nfast ? t_first % p.tilesN : 0, nf_m = p.nfast ? t_first / p.tilesN : 0;
      for (int t = t_first; t < t_end; t += t_step) {
        const int m_idx = (p.nfast ? nf_m : unit_m) * CTAS + static_cast<int>(cta_rank);
        int n_idx = p.nfast ? nf_n : rest, ks = 0;
        if (p.ksplit > 1) { n_idx = rest % p.tilesN; ks = rest / p.tilesN; }
        nf_n += nf_step_n; nf_m += nf_step_m;
        if (p.nfast && nf_n >= p.tilesN) { nf_n -= p.tilesN; ++nf_m; }
        int wt = m_idx, ht = 0, bt = 0;
        if (!flat) {
          wt = m_idx % p.tilesW;
          const int q = m_idx / p.tilesW;
          ht = q % p.tilesH;
          bt = q / p.tilesH;
        }
        unit_m += step_m; rest += step_r;
        if (unit_m >= unitsM) { unit_m -= unitsM; ++rest; }
        const int w0 = wt * p.TW, h0 = ht * p.TH, b0 = bt * p.TB;
        const int n0 = n_idx * BN + static_cast<int>(cta_rank) * (BN / CTAS);
        const int kb_begin = ks * p.kb_per_split;
        const int kb_end = min(p.kb_total, kb_begin + p.kb_per_split);
        int kb = 0;
        VDB_TL(0, (t - t_first) / t_step);   // producer: starts issuing this tile
        for (int s = 0; s < p.nseg; ++s) {
          const ASeg sg = p.seg[s];
          if (kb + sg.nkb <= kb_begin) { kb += sg.nkb; continue; }
          for (int j = 0; j < sg.nkb; ++j, ++kb) {
            if (kb < kb_begin) continue;
            if (kb >= kb_end) break;
            if constexpr (CTAS == 2) mbar_wait_wd(&empty_bar[stage], phase ^ 1, 0); else mbar_wait(&empty_bar[stage], phase ^ 1);
            if constexpr (CTAS == 2) {
              // rank 0 arms its barrier for the bytes of BOTH CTAs (the peer's may land first: the transaction
              // count is signed and the phase cannot complete before this arrival)
              if (cta_rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * kStageBytes);
              const uint32_t leader_full = mapa_u32(smem_u32(&full_bar[stage]), 0);   // rank 0's barrier
              tma_load_4d_pair(smemA + stage * kABytes, &p.tmA[sg.tmap], leader_full,
                               sg.c0 + j * kBlockK, w0 + sg.dw, h0 + sg.dh, b0);
              tma_load_2d_pair(smemB + stage * kBBytes, &p.tmB, leader_full, kb * kBlockK, n0);
            } else {
              mbar_arrive_expect_tx(&full_bar[stage], kStageBytes);
              tma_load_4d(smemA + stage * kABytes, &p.tmA[sg.tmap], &full_bar[stage],
                          sg.c0 + j * kBlockK, w0 + sg.dw, h0 + sg.dh, b0);
              tma_load_2d(smemB + stage * kBBytes, &p.tmB, &full_bar[stage], kb * kBlockK, n0);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          if (kb >= kb_end) break;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer ------------------------------
    // single CTAs: the WHOLE warp runs the issue loop and one elected lane issues each tcgen05 instruction (convergent control
    // flow keeps the descriptors in uniform registers; under `if (lane == 0)` every MMA sat in an ELECT / R2UR / BRA.U.ANY
    // loop of ~90 cycles, more than the 32-80 tensor cycles of a BN <= 160 MMA).  CTA pairs: the same, in rank 0's warp.
    if ((CTAS == 1) || (cta_rank == 0)) {
      constexpr uint32_t idesc = make_idesc_bf16(kBlockM * CTAS, BN);
      uint32_t stage = 0, phase = 0;
      int it = 0;
      for (int t = t_first; t < t_end; t += t_step, ++it) {
        const int ks = (p.ksplit > 1) ? (t / unitsM) / p.tilesN : 0;
        const int kb_begin = ks * p.kb_per_split;
        const int kb_end = min(p.kb_total, kb_begin + p.kb_per_split);
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        VDB_TL(1, it);                             // MMA: wants the accumulator stage
        if constexpr (CTAS == 2) mbar_wait_wd(&tmem_empty[as], aphase ^ 1, 1); else mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        VDB_TL(2, it);                             // MMA: got it
        const uint32_t tmem_d = tmem_base + as * 256;
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          if constexpr (CTAS == 2) mbar_wait_wd(&full_bar[stage], phase, 2); else mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t adesc = make_desc_sw128(smem_u32(smemA + stage * kABytes));
          const uint64_t bdesc = make_desc_sw128(smem_u32(smemB + stage * kBBytes));
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            // advance 16 bf16 = 32 B along K inside the swizzle atom: +2 in (addr >> 4) units
            if constexpr (CTAS == 2) umma_bf16_ss_pair_w(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > kb_begin || k > 0) ? 1u : 0u);
            else umma_bf16_ss_w(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > kb_begin || k > 0) ? 1u : 0u);
          }
          if constexpr (CTAS == 2) umma_commit_pair_w(&empty_bar[stage]); else umma_commit_w(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if constexpr (CTAS == 2) umma_commit_pair_w(&tmem_full[as]); else umma_commit_w(&tmem_full[as]);
        VDB_TL(3, it);                             // MMA: all MMAs of the tile issued
      }
    }
  } else {
    // ------------------------------ epilogue ------------------------------
    // Eight warps: warps w and w+4 own the same TMEM lane quarter (w & 3) and alternate 32-column chunks, so each
    // SM sub-partition interleaves two epilogue warps (a single warp per sub-partition was measured to be
    // instruction-latency bound: ~770 ns per chunk).  tcgen05.ld hands each thread one ROW of 32 columns; the
    // warp writes the raw fp32 block to a private XOR-swizzled 4 KB shared-memory tile and reads it back
    // transposed, so every global access is 8 rows x 64 contiguous bytes per instruction (4 lanes per row), and
    // bias / activation / residual / bf16 conversion run on 8 fixed columns per lane (bias lives in registers).
    const int quarter = warp & 3;          // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;      // which of the kWPQ warps of the quarter
    const int r = quarter * 32 + lane;
    const int tr_row = lane >> 2, tr_q = lane & 3;   // transposed role: rows tr_row + 8k, columns tr_q*8 .. +7
    float* stage = sstage + (warp - 2) * 1024;       // [32 rows][32 fp32], 16-byte chunk j of row i at (j ^ (i & 7))
    auto stage_write = [&](const uint32_t (&v)[32]) {
      float* srow = stage + lane * 32;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<uint4*>(srow + ((j ^ (lane & 7)) << 2)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    };
    auto stage_read = [&](int k, float (&o)[8]) {   // row tr_row + 8k, columns tr_q*8 .. +7
      const int row = k * 8 + tr_row;
      const float* srow = stage + row * 32;
      const float4 x0 = *reinterpret_cast<const float4*>(srow + (((2 * tr_q) ^ (row & 7)) << 2));
      const float4 x1 = *reinterpret_cast<const float4*>(srow + (((2 * tr_q + 1) ^ (row & 7)) << 2));
      o[0] = x0.x; o[1] = x0.y; o[2] = x0.z; o[3] = x0.w; o[4] = x1.x; o[5] = x1.y; o[6] = x1.z; o[7] = x1.w;
    };
    int it = 0;
    int st_buf = 0;                     // TMA-store epilogues: which of this warp's two staging tiles is written next
    (void)st_buf;
    const float* sbias_src = nullptr;   // which bias row/offset currently sits in sbias
    const uint32_t leader_tmem_empty[2] = {(CTAS == 2) ? mapa_u32(smem_u32(&tmem_empty[0]), 0) : 0u,
                                           (CTAS == 2) ? mapa_u32(smem_u32(&tmem_empty[1]), 0) : 0u};
    // The per-tile bookkeeping sits on the critical path of epilogue-bound GEMMs (it was ~0.75 us of every ~3.6 us
    // tile): the tile index advances incrementally (no divisions in the GEMM view), row indices are 32-bit, and
    // everything that depends only on the thread is hoisted.
    const int tw = r % p.TW;
    const int th = (r / p.TW) % p.TH;
    const int tb = r / (p.TW * p.TH);
    const bool flat = (p.tilesH == 1) && (p.tilesB == 1);   // GEMM view: M tiles along W only
    const int step_m = t_step % unitsM, step_r = t_step / unitsM;
    int unit_m = t_first % unitsM, rest = t_first / unitsM;
    const int nf_step_n = p.nfast ? t_step % p.tilesN : 0, nf_step_m = p.nfast ? t_step / p.tilesN : 0;   // (see the producer)
    int nf_n = p.nfast ? t_first % p.tilesN : 0, nf_m = p.nfast ? t_first / p.tilesN : 0;
    // folded LayerNorm, row statistics: partial sums of the row this thread owns in the NEXT tile, requested a tile ahead
    constexpr int kLnPre = 16;
    float2 ln_pre[kLnIn ? kLnPre : 1];
    auto ln_prefetch = [&](int row) {
      if constexpr (kLnIn) {
        const bool ok = row < p.Wo;
#pragma unroll
        for (int i = 0; i < kLnPre; ++i)
          ln_pre[i] = (ok && i < p.ln_parts) ? __ldg(reinterpret_cast<const float2*>(p.ln_stats) + static_cast<long long>(i) * p.ln_mstat + row)
                                              : make_float2(0.f, 0.f);
      }
    };
    if constexpr (kLnIn) {
      if (!p.ln_on_cols && p.ln_parts <= kLnPre && t_first < t_end) ln_prefetch((t_first % unitsM) * kBlockM + r);
    }
    for (int t = t_first; t < t_end; t += t_step, ++it) {
      const int m_idx = (p.nfast ? nf_m : unit_m) * CTAS + static_cast<int>(cta_rank);
      int n_idx = p.nfast ? nf_n : rest, ks = 0;
      if (p.ksplit > 1) { n_idx = rest % p.tilesN; ks = rest / p.tilesN; }
      nf_n += nf_step_n; nf_m += nf_step_m;
      if (p.nfast && nf_n >= p.tilesN) { nf_n -= p.tilesN; ++nf_m; }
      int wt = m_idx, ht = 0, bt = 0;
      if (!flat) {
        wt = m_idx % p.tilesW;
        const int q = m_idx / p.tilesW;
        ht = q % p.tilesH;
        bt = q / p.tilesH;
      }
      unit_m += step_m; rest += step_r;
      if (unit_m >= unitsM) { unit_m -= unitsM; ++rest; }
      const int w = wt * p.TW + tw, h = ht * p.TH + th, b = bt * p.TB + tb;
      const bool row_ok = (w < p.Wo) && (h < p.Ho) && (b < p.Bo);
      const int gp = (b * p.Ho + h) * p.Wo + w;     // output pixel (row of the GEMM); host guarantees M < 2^31
      const int gp_first = ((bt * p.TB) * p.Ho + ht * p.TH) * p.Wo + wt * p.TW;
      const int n0 = n_idx * BN;
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;

      // per-tile row bookkeeping for the transposed role (independent of the accumulator: done before the wait)
      int gp_k[4];
      bool ok_k[4];
      {
        const unsigned okmask = __ballot_sync(0xffffffffu, row_ok);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int src = k * 8 + tr_row;
          gp_k[k] = __shfl_sync(0xffffffffu, gp, src);
          ok_k[k] = (okmask >> src) & 1u;
        }
      }
      // bias tile -> shared memory (one global read per tile); one row serves the tile unless the bias is per-batch
      // and the tile's first / last rows belong to different batch items
      const int gp_last = ((bt * p.TB + p.TB - 1) * p.Ho + ht * p.TH + p.TH - 1) * p.Wo + wt * p.TW + p.TW - 1;
      const bool bias_uniform = (MODE != 0) ? (p.bias != nullptr)    // host: a tile never straddles two bias rows
                                            : (p.bias && p.ksplit == 1 &&
                                               (p.bias_bstride == 0 || gp_first / p.rows_per_batch == gp_last / p.rows_per_batch));
      if constexpr (kLnIn) {
        // folded-LayerNorm tiles: sbias = c[n] (beta term + bias), slnx = s[n]; or, when the statistics belong to the
        // columns, sbias = rstd[n], slnx = mean[n] computed here from the producer's partial sums (one column per thread)
        const float* key = reinterpret_cast<const float*>(static_cast<uintptr_t>(n0) + 1);
        if (key != sbias_src) {
          epi_bar_sync();
          for (int i = threadIdx.x - 64; i < BN; i += kNumEpiThreads) {
            const int n = n0 + i;
            float a = 0.f, b = 0.f;
            if (n < p.N) {
              if (p.ln_on_cols) {
                float su = 0.f, sq = 0.f;
#pragma unroll 8
                for (int ch = 0; ch < p.ln_parts; ++ch) {
                  const float2 v = __ldg(reinterpret_cast<const float2*>(p.ln_stats) + static_cast<long long>(ch) * p.ln_mstat + n);
                  su += v.x; sq += v.y;
                }
                const float mu = su * p.ln_inv_dim;
                a = mu;
                b = rsqrtf(fmaxf(sq * p.ln_inv_dim - mu * mu, 0.f) + p.ln_eps);
              } else {
                a = __ldg(p.ln_colsum + n);
                b = p.bias ? __ldg(p.bias + n) : 0.f;
              }
            }
            slnx[i] = a;
            sbias[i] = b;
          }
          epi_bar_sync();
          sbias_src = key;
        }
      } else if (bias_uniform) {
        // consecutive tiles of a CTA usually share the N tile (M is the fast tile index): reload only on change,
        // otherwise the ~0.7 us global-load latency + two barriers sit between every two tiles
        const float* brow = p.bias + (p.bias_bstride ? static_cast<long long>(gp_first / p.rows_per_batch) * p.bias_bstride : 0) + n0;
        if (brow != sbias_src) {              // uniform across the epilogue threads
          epi_bar_sync();                     // previous tile's readers are done with sbias
          for (int i = threadIdx.x - 64; i < BN; i += kNumEpiThreads) sbias[i] = (n0 + i < p.N) ? __ldg(brow + i) : 0.f;
          epi_bar_sync();
          sbias_src = brow;
        }
      }
      const float* bias_g = (p.bias && !bias_uniform)
                                ? p.bias + (p.bias_bstride ? static_cast<long long>(gp / p.rows_per_batch) * p.bias_bstride : 0) : nullptr;

      // MODE 1: this warp's chunk range and the residual rows of its first chunk, requested BEFORE the accumulator wait
      const int f_nchunks = min(BN / 32, (p.N - n0) / 32);
      const bool has_resid = p.resid != nullptr;
      const int f_first = (((BN / 32) % kWPQ) != 0) ? ((half + it) % kWPQ) : half;
      auto load_resid_fast = [&](int c, uint4 (&rr)[4]) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (ok_k[k]) rr[k] = __ldg(reinterpret_cast<const uint4*>(p.resid + static_cast<long long>(gp_k[k]) * p.ldr + n0 + c * 32 + tr_q * 8));
      };
      uint4 rr_first[4];
      if constexpr (MODE == 1) {
        if (has_resid && f_first < f_nchunks) load_resid_fast(f_first, rr_first);
      }

      // folded LayerNorm: this thread's row scalars (requested before the accumulator wait)
      float ln_a0 = 0.f, ln_a1 = 1.f;     // on_cols 0: (mean, rstd) of the row;  on_cols 1: (s[m], c[m]) of the output row
      if constexpr (kLnIn) {
        if (row_ok) {
          if (p.ln_on_cols) {
            ln_a0 = __ldg(p.ln_colsum + gp);
            ln_a1 = p.ln_rowbias ? __ldg(p.ln_rowbias + gp) : 0.f;
          } else {
            float su = 0.f, sq = 0.f;
            if (p.ln_parts <= kLnPre) {
              // the partials of THIS tile's row were requested one tile ago (ln_pre): a tile's own request would sit on the
              // critical path of every epilogue-bound tile (first version: +75 % on the K = 320 GEMMs)
#pragma unroll
              for (int i = 0; i < kLnPre; ++i) { su += ln_pre[i].x; sq += ln_pre[i].y; }
            } else {
#pragma unroll 8
              for (int ch = 0; ch < p.ln_parts; ++ch) {
                const float2 v = __ldg(reinterpret_cast<const float2*>(p.ln_stats) + static_cast<long long>(ch) * p.ln_mstat + gp);
                su += v.x; sq += v.y;
              }
            }
            ln_a0 = su * p.ln_inv_dim;
            ln_a1 = rsqrtf(fmaxf(sq * p.ln_inv_dim - ln_a0 * ln_a0, 0.f) + p.ln_eps);
          }
        }
        // request the next tile's row partials (GEMM view, M-fast order: unit_m already points at the next tile)
        if (!p.ln_on_cols && p.ln_parts <= kLnPre && t + t_step < t_end) ln_prefetch(unit_m * kBlockM + r);
      }
      VDB_TLE(4, it);   // epilogue: waiting for the accumulator
      if constexpr (CTAS == 2) mbar_wait_wd(&tmem_full[as], aphase, 3); else mbar_wait(&tmem_full[as], aphase);
      tc_fence_after();
      VDB_TLE(5, it);   // epilogue: accumulator complete
      const uint32_t trow = tmem_base + as * 256 + (static_cast<uint32_t>(quarter * 32) << 16);

      auto geglu_tile = [&] {
        // packed tile: columns [0,BN/2) = value rows, [BN/2,BN) = gate rows of the same outputs
        constexpr int HALF = BN / 2;
        const int nout0 = n_idx * HALF;
        const int Nout = p.N / 2;
#pragma unroll 1
        for (int c = (((HALF / 32) % kWPQ) != 0) ? ((half + it) % kWPQ) : half; c < HALF / 32; c += kWPQ) {
          uint32_t v[32];
          float a[4][8];
          tmem_ld32(trow + c * 32, v);
          tmem_wait_ld();
          stage_write(v);
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 4; ++k) stage_read(k, a[k]);
          __syncwarp();
          tmem_ld32(trow + HALF + c * 32, v);
          tmem_wait_ld();
          stage_write(v);
          __syncwarp();
          float bv[8], bg[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            bv[i] = p.bias ? sbias[c * 32 + tr_q * 8 + i] : 0.f;
            bg[i] = p.bias ? sbias[HALF + c * 32 + tr_q * 8 + i] : 0.f;
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float g[8];
            stage_read(k, g);
            if (ok_k[k] && nout0 + c * 32 + tr_q * 8 + 7 < Nout) {
              float o[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) o[i] = (a[k][i] + bv[i]) * gelu_fast_f(g[i] + bg[i]);
              *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + static_cast<long long>(gp_k[k]) * p.ldo + nout0 + c * 32 + tr_q * 8) =
                  make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
            }
          }
          __syncwarp();
        }
      };
      if constexpr (kTmaEpi) {
        // ---- TMA-store epilogues (round 2).  Everything stays in the tcgen05.ld layout (one ROW of 32 columns per thread):
        // bias from shared memory (broadcast reads), residual as this row's own 64 contiguous bytes, bf16 pack, four 16-byte
        // shared-memory stores into this warp's 32 x 32 staging tile (64-byte rows, SWIZZLE_64B pattern: conflict-free),
        // then ONE thread hands the tile to the TMA unit (cp.async.bulk.tensor store; out-of-range rows / columns are clipped by
        // the tensor map).  Against the fp32 transposition above this halves the shared-memory traffic of the epilogue
        // (2 x 64 B instead of 2 x 128 B per row and chunk) and removes the 8 global-store instructions per thread and chunk —
        // the K <= 640 GEMMs were bound by exactly that (profiles/r01_ncu_hot_lines_v7.txt).  Two staging tiles per warp:
        // the store of chunk i is read out while chunk i+1 is built.
        uint8_t* stg = reinterpret_cast<uint8_t*>(sstage) + (warp - 2) * 4096;
        const int qrow = quarter * 32;                                   // first tile row of this warp's TMEM lane quarter
        const int ow = wt * p.TW + (qrow % p.TW), oh = ht * p.TH + ((qrow / p.TW) % p.TH), ob = bt * p.TB + qrow / (p.TW * p.TH);
        constexpr int OUTC = kGegluEpi ? BN / 2 : BN;                    // output columns per tile
        const int ochunks = kGegluEpi ? OUTC / 32 : f_nchunks;
        const int ocol0 = n_idx * OUTC;
        const int o_first = (((OUTC / 32) % kWPQ) != 0) ? ((half + it) % kWPQ) : half;
        auto load_resid_row = [&](int c, uint4 (&rr)[4]) {
          const uint4* src = reinterpret_cast<const uint4*>(p.resid + static_cast<long long>(gp) * p.ldr + ocol0 + c * 32);
#pragma unroll
          for (int k = 0; k < 4; ++k) rr[k] = __ldg(src + k);
        };
        uint4 rr[4];
        float st_su = 0.f, st_sq = 0.f;                                  // mode 7: partial LayerNorm sums of this thread's columns
        (void)st_su; (void)st_sq;
        const bool do_resid = (MODE == 3 || MODE == 7) && has_resid && row_ok;
        if (do_resid && o_first < ochunks) load_resid_row(o_first, rr);
#pragma unroll 1
        for (int c = o_first; c < ochunks; c += kWPQ) {
          float o[32];
          if constexpr (MODE == 6) {
            // GEGLU over a folded LayerNorm (row statistics only): value and gate both get the rank-1 correction
            uint32_t va[32], vg[32];
            tmem_ld32(trow + c * 32, va);
            tmem_ld32(trow + OUTC + c * 32, vg);
            tmem_wait_ld();
            // r * (acc - mu * s) + c  ==  fma(r, acc, fma(-r mu, s, c)); the tables are read as 16-byte broadcasts
            const float nrm = -ln_a1 * ln_a0;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 sa = lds_f4(slnx_s + 4 * (c * 32 + j)), ca = lds_f4(sbias_s + 4 * (c * 32 + j));
              const float4 sg = lds_f4(slnx_s + 4 * (OUTC + c * 32 + j)), cg = lds_f4(sbias_s + 4 * (OUTC + c * 32 + j));
              o[j] = fmaf(ln_a1, __uint_as_float(va[j]), fmaf(nrm, sa.x, ca.x)) * gelu_fast_f(fmaf(ln_a1, __uint_as_float(vg[j]), fmaf(nrm, sg.x, cg.x)));
              o[j + 1] = fmaf(ln_a1, __uint_as_float(va[j + 1]), fmaf(nrm, sa.y, ca.y)) * gelu_fast_f(fmaf(ln_a1, __uint_as_float(vg[j + 1]), fmaf(nrm, sg.y, cg.y)));
              o[j + 2] = fmaf(ln_a1, __uint_as_float(va[j + 2]), fmaf(nrm, sa.z, ca.z)) * gelu_fast_f(fmaf(ln_a1, __uint_as_float(vg[j + 2]), fmaf(nrm, sg.z, cg.z)));
              o[j + 3] = fmaf(ln_a1, __uint_as_float(va[j + 3]), fmaf(nrm, sa.w, ca.w)) * gelu_fast_f(fmaf(ln_a1, __uint_as_float(vg[j + 3]), fmaf(nrm, sg.w, cg.w)));
            }
          } else if constexpr (MODE == 5) {
            uint32_t v[32];
            tmem_ld32(trow + c * 32, v);
            tmem_wait_ld();
            if (p.ln_on_cols) {          // out = rstd[n] * (acc - mean[n] * s[m]) + c[m]
              const float ns = -ln_a0;
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const float4 mu = lds_f4(slnx_s + 4 * (c * 32 + j)), rs = lds_f4(sbias_s + 4 * (c * 32 + j));
                o[j] = fmaf(rs.x, fmaf(mu.x, ns, __uint_as_float(v[j])), ln_a1);
                o[j + 1] = fmaf(rs.y, fmaf(mu.y, ns, __uint_as_float(v[j + 1])), ln_a1);
                o[j + 2] = fmaf(rs.z, fmaf(mu.z, ns, __uint_as_float(v[j + 2])), ln_a1);
                o[j + 3] = fmaf(rs.w, fmaf(mu.w, ns, __uint_as_float(v[j + 3])), ln_a1);
              }
            } else {                     // out = rstd[m] * (acc - mean[m] * s[n]) + c[n] == fma(r, acc, fma(-r mu, s, c))
              const float nrm = -ln_a1 * ln_a0;
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const float4 sx = lds_f4(slnx_s + 4 * (c * 32 + j)), cx = lds_f4(sbias_s + 4 * (c * 32 + j));
                o[j] = fmaf(ln_a1, __uint_as_float(v[j]), fmaf(nrm, sx.x, cx.x));
                o[j + 1] = fmaf(ln_a1, __uint_as_float(v[j + 1]), fmaf(nrm, sx.y, cx.y));
                o[j + 2] = fmaf(ln_a1, __uint_as_float(v[j + 2]), fmaf(nrm, sx.z, cx.z));
                o[j + 3] = fmaf(ln_a1, __uint_as_float(v[j + 3]), fmaf(nrm, sx.w, cx.w));
              }
            }
          } else if constexpr (MODE == 4) {
            uint32_t va[32], vg[32];
            tmem_ld32(trow + c * 32, va);
            tmem_ld32(trow + OUTC + c * 32, vg);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 ba = p.bias ? lds_f4(sbias_s + 4 * (c * 32 + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
              const float4 bg = p.bias ? lds_f4(sbias_s + 4 * (OUTC + c * 32 + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
              o[j] = (__uint_as_float(va[j]) + ba.x) * gelu_fast_f(__uint_as_float(vg[j]) + bg.x);
              o[j + 1] = (__uint_as_float(va[j + 1]) + ba.y) * gelu_fast_f(__uint_as_float(vg[j + 1]) + bg.y);
              o[j + 2] = (__uint_as_float(va[j + 2]) + ba.z) * gelu_fast_f(__uint_as_float(vg[j + 2]) + bg.z);
              o[j + 3] = (__uint_as_float(va[j + 3]) + ba.w) * gelu_fast_f(__uint_as_float(vg[j + 3]) + bg.w);
            }
          } else {
            uint32_t v[32];
            tmem_ld32(trow + c * 32, v);
            uint4 rn[4];
            const bool more = c + kWPQ < ochunks;
            if (do_resid && more) load_resid_row(c + kWPQ, rn);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 bb = p.bias ? lds_f4(sbias_s + 4 * (c * 32 + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
              o[j] = __uint_as_float(v[j]) + bb.x; o[j + 1] = __uint_as_float(v[j + 1]) + bb.y;
              o[j + 2] = __uint_as_float(v[j + 2]) + bb.z; o[j + 3] = __uint_as_float(v[j + 3]) + bb.w;
            }
            if (do_resid) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t w4[4] = {rr[k].x, rr[k].y, rr[k].z, rr[k].w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const float2 x = unpack_bf16x2(w4[q]);
                  o[k * 8 + 2 * q] += x.x;
                  o[k * 8 + 2 * q + 1] += x.y;
                }
              }
              if (more) {
#pragma unroll
                for (int k = 0; k < 4; ++k) rr[k] = rn[k];
              }
            }
          }
          if constexpr (kStatsOut) {
            // LayerNorm statistics of the rows this GEMM produces: this thread's columns of the tile (fp32, before the rounding)
            float su = 0.f, sq = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) { su += o[j]; sq = fmaf(o[j], o[j], sq); }
            st_su += su; st_sq += sq;
          }
          // the staging tile about to be rewritten was handed to the TMA unit two chunks ago: wait until it has been read
          if (lane == 0) bulk_wait_read<1>();
          __syncwarp();
          uint8_t* tile = stg + st_buf * 2048;
          const uint32_t trow_s = smem_u32(tile) + lane * 64;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(trow_s + ((q ^ ((lane >> 1) & 3)) << 4)),
                         "r"(pack_bf16x2(o[q * 8], o[q * 8 + 1])), "r"(pack_bf16x2(o[q * 8 + 2], o[q * 8 + 3])),
                         "r"(pack_bf16x2(o[q * 8 + 4], o[q * 8 + 5])), "r"(pack_bf16x2(o[q * 8 + 6], o[q * 8 + 7]))
                         : "memory");
          }
          fence_proxy_async_smem();      // every writer: generic-proxy stores -> visible to the TMA (async proxy) read
          __syncwarp();
          if (lane == 0) {
            tma_store_4d(&p.tmO, tile, ocol0 + c * 32, ow, oh, ob);
            bulk_commit();
          }
          st_buf ^= 1;
        }
        if constexpr (kStatsOut) {
          // one partial per (N tile, warp of the lane quarter): the two warps own disjoint chunk sets (o_first = 0 / 1)
          if (row_ok)
            reinterpret_cast<float2*>(p.stats_out)[static_cast<long long>(n_idx * kWPQ + o_first) * (static_cast<long long>(p.Bo) * p.Ho * p.Wo) + gp] =
                make_float2(st_su, st_sq);
        }
      } else if constexpr (MODE == 1) {
        // lean fast path: every chunk is a full 32-column bf16 chunk with one bias row; the residual rows of the
        // next chunk are requested before this chunk is processed (their first use otherwise exposes ~1 us)
        uint4 rr[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) rr[k] = rr_first[k];
#pragma unroll 1
        for (int c = f_first; c < f_nchunks; c += kWPQ) {
          uint32_t v[32];
          tmem_ld32(trow + c * 32, v);
          uint4 rn[4];
          if (has_resid && c + kWPQ < f_nchunks) load_resid_fast(c + kWPQ, rn);
          tmem_wait_ld();
          stage_write(v);
          __syncwarp();
          float bb[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) bb[i] = p.bias ? sbias[c * 32 + tr_q * 8 + i] : 0.f;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float o[8];
            stage_read(k, o);
            if (ok_k[k]) {
#pragma unroll
              for (int i = 0; i < 8; ++i) o[i] += bb[i];
              if (has_resid) {
                const uint32_t w4[4] = {rr[k].x, rr[k].y, rr[k].z, rr[k].w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const float2 x = unpack_bf16x2(w4[q]);
                  o[2 * q] += x.x;
                  o[2 * q + 1] += x.y;
                }
              }
              *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + static_cast<long long>(gp_k[k]) * p.ldo + n0 + c * 32 + tr_q * 8) =
                  make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
            }
          }
          __syncwarp();   // the staging tile is rewritten by this warp's next chunk
#pragma unroll
          for (int k = 0; k < 4; ++k) rr[k] = rn[k];
        }
      } else if constexpr (MODE == 2) {
        geglu_tile();
      } else if (p.ksplit > 1) {
        // fp32 partials, reduced (+bias/act/residual) by splitk_reduce_kernel
        const long long Mtot = static_cast<long long>(p.Bo) * p.Ho * p.Wo;
        float* dst = p.partial + (static_cast<long long>(ks) * Mtot + gp) * p.N + n0;
#pragma unroll 1
        for (int c = half; c < BN / 32; c += kWPQ) {
          if (n0 + c * 32 >= p.N) break;
          uint32_t v[32];
          tmem_ld32(trow + c * 32, v);
          tmem_wait_ld();
          if (row_ok) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const int n = n0 + c * 32 + j;
              if (n + 3 < p.N) {
                *reinterpret_cast<float4*>(dst + c * 32 + j) =
                    make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
              } else {
                for (int q = 0; q < 4; ++q)
                  if (n + q < p.N) dst[c * 32 + j + q] = __uint_as_float(v[j + q]);
              }
            }
          }
        }
      } else if (p.act == ACT_GEGLU) {
        geglu_tile();
      } else {
        const int nchunks = min(BN / 32, (p.N - n0 + 31) / 32);
        auto chunk = [&](int c, const uint32_t (&v)[32], const uint4 (&rr)[4], bool fast) {
          const int nb = n0 + c * 32;
          if (fast) {
            stage_write(v);
            __syncwarp();
            if (c == half) VDB_TLE(8, it);
            float bb[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) bb[i] = p.bias ? sbias[c * 32 + tr_q * 8 + i] : 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              float o[8];
              stage_read(k, o);
              if (ok_k[k]) {
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] += bb[i];
                if (p.alpha != 1.f) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) o[i] *= p.alpha;
                }
                if (p.act != ACT_NONE) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) o[i] = apply_act(o[i], p.act);
                }
                if (p.resid) {
                  const uint32_t w4[4] = {rr[k].x, rr[k].y, rr[k].z, rr[k].w};
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    const float2 x = unpack_bf16x2(w4[q]);
                    o[2 * q] += x.x;
                    o[2 * q + 1] += x.y;
                  }
                }
                *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + static_cast<long long>(gp_k[k]) * p.ldo + nb + tr_q * 8) =
                    make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
              }
              if (c == half && k == 0) VDB_TLE(9, it);
            }
            __syncwarp();   // the tile is rewritten by this warp's next chunk
            if (c == half) VDB_TLE(10, it);
          } else if (row_ok) {
            // slow path (fp32 output, partial last chunk, per-row bias): one row per thread
            float f[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
            if (p.bias) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (nb + j < p.N) f[j] += bias_uniform ? sbias[c * 32 + j] : __ldg(bias_g + nb + j);
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = apply_act(f[j] * p.alpha, p.act);
            if (p.resid) {
              const __nv_bfloat16* rs = p.resid + static_cast<long long>(gp) * p.ldr + nb;
#pragma unroll
              for (int j = 0; j < 32; ++j) if (nb + j < p.N) f[j] += __bfloat162float(rs[j]);
            }
            if (p.out_f32) {
              float* dst = reinterpret_cast<float*>(p.out) + static_cast<long long>(gp) * p.ldo + nb;
#pragma unroll
              for (int j = 0; j < 32; ++j) if (nb + j < p.N) dst[j] = f[j];
            } else {
              __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + static_cast<long long>(gp) * p.ldo + nb;
#pragma unroll
              for (int j = 0; j < 32; ++j) if (nb + j < p.N) dst[j] = __float2bfloat16(f[j]);
            }
          }
        };
        auto is_fast = [&](int c) { return (n0 + c * 32 + 32 <= p.N) && !p.out_f32 && (bias_uniform || !p.bias); };
        auto load_resid = [&](int c, uint4 (&rr)[4]) {
          if (p.resid && is_fast(c)) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (ok_k[k]) rr[k] = __ldg(reinterpret_cast<const uint4*>(p.resid + static_cast<long long>(gp_k[k]) * p.ldr + n0 + c * 32 + tr_q * 8));
          }
        };
        // this warp's chunks: half, half+2, ... (kept un-pipelined: double-buffering the 32-register TMEM chunk
        // pushed the kernel into spills and was measured slower)
        // chunk count not a multiple of the warps per quarter (BN = 160: five): rotate who takes the extra chunk
        const int first = (p.epi_alt && ((BN / 32) % kWPQ) != 0) ? ((half + it) % kWPQ) : half;
#pragma unroll 1
        for (int c = first; c < nchunks; c += kWPQ) {
          uint4 rr[4];
          load_resid(c, rr);          // residual loads are in flight while the accumulator chunk is fetched
          uint32_t v[32];
          tmem_ld32(trow + c * 32, v);
          tmem_wait_ld();
          if (c == first) VDB_TLE(7, it);
          chunk(c, v, rr, is_fast(c));
        }
      }
      tc_fence_before();
      __syncwarp();
      VDB_TLE(6, it);   // epilogue: tile stored (this warp)
      if (lane == 0) {
        if constexpr (CTAS == 2) mbar_arrive_cluster(leader_tmem_empty[as]);   // the MMA issuer lives in rank 0
        else mbar_arrive(&tmem_empty[as]);
      }
    }
    if constexpr (MODE >= 3) {
      if (lane == 0) bulk_wait<0>();     // every TMA store of this thread has completed before the CTA may exit
    }
  }

  tc_fence_before();
  if constexpr (CTAS == 2) {
    __syncwarp();
    cluster_sync_all();   // the peer may still be reading this CTA's operands / signalling its barriers
    if (warp == 2) tmem_dealloc_pair<512>(tmem_base);
  } else {
    __syncthreads();
    if (warp == 2) tmem_dealloc<512>(tmem_base);
  }
}

// split-K reduction + epilogue: out[m, n] = act(alpha * (sum_s partial[s, m, n] + bias)) + resid
__global__ void splitk_reduce_kernel(const float* __restrict__ partial, int ksplit, long long M, int N,
                                     const float* __restrict__ bias, long long bias_bstride, int rows_per_batch,
                                     const __nv_bfloat16* __restrict__ resid, long long ldr, void* out,
                                     long long ldo, int out_f32, int act, float alpha) {
  pdl_launch_dependents();
  pdl_wait();
  const long long total = M * (N / 4);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = i / (N / 4);
    const int n = static_cast<int>(i % (N / 4)) * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    // (one partial per iteration on purpose: with all ksplit loads of a thread in flight at once — addresses M*N*4 bytes apart —
    // the 8x8-level convs got 4.4 us SLOWER per launch, 26.3 -> 30.7 us; profiles/r02_visit_final_splitk_reduce_unrolled.log)
    for (int s = 0; s < ksplit; ++s) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(partial + (static_cast<long long>(s) * M + m) * N + n));
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    float f[4] = {acc.x, acc.y, acc.z, acc.w};
    if (bias) {
      const float* bp = bias + (bias_bstride ? (m / rows_per_batch) * bias_bstride : 0) + n;
      for (int q = 0; q < 4; ++q) f[q] += __ldg(bp + q);
    }
    for (int q = 0; q < 4; ++q) f[q] *= alpha;
    for (int q = 0; q < 4; ++q) f[q] = apply_act(f[q], act);
    if (resid) {
      for (int q = 0; q < 4; ++q) f[q] += __bfloat162float(resid[m * ldr + n + q]);
    }
    if (out_f32) {
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + m * ldo + n) = make_float4(f[0], f[1], f[2], f[3]);
    } else {
      uint2 o = make_uint2(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]));
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out) + m * ldo + n) = o;
    }
  }
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
template <int BN, int STAGES, int CTAS, int EW, int MODE>
static int launch_igemm(const IgemmParams& p0, int num_units, cudaStream_t stream) {
  constexpr bool kLn = MODE == 5 || MODE == 6;       // one more [BN] fp32 table (colsum / column mean)
  constexpr size_t need = STAGES * (kABytes + (BN / CTAS) * kBlockK * 2) + (2 * STAGES + 4) * 8 + 16 + BN * 4 +
                          (kLn ? BN * 4 : 0) + EW * 4096;
  // + up to 1024 bytes of slack for the 1024-byte alignment of the operand ring (the LN modes at BN 256 get 912: the dynamic
  // window starts 1024-aligned on every driver seen so far, and the kernel traps if its carve-up would not fit)
  constexpr size_t smem = (need + 1024 <= 227 * 1024) ? need + 1024 : 227 * 1024;
  static_assert(need + 896 <= 227 * 1024, "igemm shared-memory budget");
  constexpr int threads = 64 + 32 * EW;
  IgemmParams p = p0;
  p.smem_bytes = static_cast<unsigned>(smem);
  static bool configured = false;
  if (!configured) {
    VDB_CUDA_CHECK(cudaFuncSetAttribute(igemm_kernel<BN, STAGES, CTAS, EW, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem)));
    prefer_max_smem(igemm_kernel<BN, STAGES, CTAS, EW, MODE>);
    configured = true;
  }
  if (CTAS == 2) {
    // persistent CTA pairs: one 2-cluster per TPC
    const int grid = 2 * std::min(num_units, num_sms() / 2);
    VDB_CUDA_CHECK(launch_cluster2(igemm_kernel<BN, STAGES, CTAS, EW, MODE>, dim3(grid), dim3(threads), smem, stream, p));
  } else {
    const int grid = std::min(num_units, num_sms());
    VDB_CUDA_CHECK(launch_pdl(igemm_kernel<BN, STAGES, CTAS, EW, MODE>, dim3(grid), dim3(threads), smem, stream, p));
  }
  count_launch();
  return VDB_OK;
}

static int pick_bn(int N, int act, int forced) {
  if (forced) return forced;
  if (act == ACT_GEGLU) return 256;
  if (N <= 64) return 64;
  if (N % 256 == 0) return 256;
  if (N % 160 == 0) return 160;
  if (N % 128 == 0) return 128;
  if (N <= 128) return 128;
  if (N <= 160) return 160;
  return 256;
}

static unsigned long long* g_timeline = nullptr;
static long long g_pair_launches = 0;
// debug aid: {epilogue mode, BN, ksplit, CTA pair} of the last launch on this thread (vdb_debug_igemm_last)
static thread_local int g_igemm_last[4] = {-1, 0, 0, 0};

struct IgemmEpilogue {
  const float* bias = nullptr;
  long long bias_bstride = 0;
  int rows_per_batch = 1;
  const void* resid = nullptr;
  long long ldr = 0;
  void* out = nullptr;
  long long ldo = 0;
  int out_f32 = 0;
  int act = 0;
  float alpha = 1.f;
  // folded LayerNorm (see igemm_kernel): consumer side ...
  const float* ln_stats = nullptr;
  long long ln_mstat = 0;
  int ln_parts = 0;
  int ln_dim = 0;
  float ln_eps = 0.f;
  const float* ln_colsum = nullptr;
  int ln_on_cols = 0;
  const float* ln_rowbias = nullptr;
  // ... and producer side
  float* stats_out = nullptr;
  int* stats_parts = nullptr;     // host out: partials per row the launch wrote (2 * N tiles)
  // folded upsample writing straight into the interleaved [B, 2Ho, 2Wo, N] tensor: output parity (py * 2 + px), -1 = compact output
  int out_parity = -1;
};

// Finish IgemmParams (tiling, split-K, B map) and launch.
static int run_igemm(IgemmParams& p, const void* Wt, long long N, long long Ktot, long long ldw,
                     const IgemmEpilogue& e, int bn_forced, int ksplit_forced, void* workspace,
                     size_t ws_bytes, cudaStream_t stream) {
  const bool ln_in = e.ln_stats != nullptr, st_out = e.stats_out != nullptr;
  if (ln_in || st_out) ksplit_forced = 1;               // the statistics ride on the single-pass TMA-store epilogues
  int BN = pick_bn(static_cast<int>(N), e.act, bn_forced);
  // Tile-width model (round 2; VDB_BN_MODEL=0 restores the divisibility rule above): the persistent grid runs
  // waves = ceil(tiles / #SMs) rounds of one tile per CTA, a tile costs kb * c(BN) cycles of mainloop (operand fill at ~90 B/clk
  // per SM or the MMA itself, whichever is longer) plus ~1500 cycles of pipeline fill / epilogue tail.  The divisibility rule sent
  // e.g. M 2048 x N 1280 x K 1280 (15 launches per step) to BN 256 = 80 tiles on 148 SMs; BN 160 gives 128 shorter tiles.
  static const int bn_model = [] { const char* ev = getenv("VDB_BN_MODEL"); return (ev && ev[0] == '0') ? 0 : 1; }();
  if (bn_model && !bn_forced && e.act != ACT_GEGLU && p.kb_total >= 8) {
    const long long tm = static_cast<long long>(p.tilesW) * p.tilesH * p.tilesB;
    const int cand[4] = {256, 160, 128, 64};
    double best = 1e30;
    for (int c : cand) {
      const long long tiles = tm * ((N + c - 1) / c);      // (a partial last N tile is computed in full)
      // split-K exactly as decided below: small MN grids with a deep K run kb / ks blocks per unit plus a reduction pass
      long long ks = 1;
      if (ksplit_forced > 0) ks = ksplit_forced;
      else if (tiles * 2 <= num_sms() && p.kb_total >= 16 && (N % 4) == 0 && workspace)
        ks = std::max<long long>(1, std::min<long long>(std::min<long long>(num_sms() / tiles, p.kb_total / 8), 16));
      const long long waves = (tiles * ks + num_sms() - 1) / num_sms();
      const double per_kb = std::max(2.0 * c, (16384.0 + 128.0 * c) / 90.0);
      const double kb_unit = static_cast<double>((p.kb_total + ks - 1) / ks);
      const double cost = static_cast<double>(waves) * (kb_unit * per_kb + 1500.0) + (ks > 1 ? 12000.0 : 0.0);
      if (cost < best * 0.97) { best = cost; BN = c; }     // (prefer the wider tile unless the gain is clear)
    }
  }
  if (!bn_forced && !bn_model && e.act != ACT_GEGLU && p.kb_total < 32) {
    // short K and a small MN grid (the 8x8 level): narrower tiles fill more SMs and need no split-K reduction pass
    // (M 512, N 1280, K 1280: 10.7 us with BN 64 vs 18.1 us with BN 256 + split-K 2, tools/bn_sweep.py)
    const int tm = p.tilesW * p.tilesH * p.tilesB;
    auto tiles = [&](int bn) { return tm * static_cast<int>((N + bn - 1) / bn); };
    while (BN > 64 && tiles(BN) * 2 <= num_sms()) BN = (BN == 256) ? 160 : (BN == 160 ? 128 : 64);
  }
  if (BN != 64 && BN != 128 && BN != 160 && BN != 256) return set_error(VDB_ERR_INVALID, "igemm: bad BN");
  if (e.act == ACT_GEGLU && (N % BN) != 0) return set_error(VDB_ERR_INVALID, "igemm: GEGLU needs N % 256 == 0");
  p.N = static_cast<int>(N);
  p.tilesN = static_cast<int>((N + BN - 1) / BN);
  p.bias = e.bias; p.bias_bstride = e.bias_bstride; p.rows_per_batch = e.rows_per_batch > 0 ? e.rows_per_batch : 1;
  p.resid = reinterpret_cast<const __nv_bfloat16*>(e.resid); p.ldr = e.ldr;
  p.out = e.out; p.ldo = e.ldo; p.out_f32 = e.out_f32; p.act = e.act; p.alpha = e.alpha;
  if (!e.out_f32 && (e.ldo % 8)) return set_error(VDB_ERR_INVALID, "igemm: ldo must be a multiple of 8 for bf16 out");
  if (e.resid && (e.ldr % 8)) return set_error(VDB_ERR_INVALID, "igemm: ldr must be a multiple of 8");
  const long long M = static_cast<long long>(p.Bo) * p.Ho * p.Wo;
  if (M >= (1LL << 30)) return set_error(VDB_ERR_UNSUPPORTED, "igemm: more than 2^30 output rows");
  const int tilesM = p.tilesW * p.tilesH * p.tilesB;
  const int mn_tiles = tilesM * p.tilesN;
  // split-K heuristic: fill the machine when the MN grid is small and K is deep
  int ksplit = 1;
  if (ksplit_forced > 0) {
    ksplit = ksplit_forced;
  } else if (e.act != ACT_GEGLU && mn_tiles * 2 <= num_sms() && p.kb_total >= 16 && (N % 4) == 0) {
    ksplit = std::min(std::min(num_sms() / mn_tiles, p.kb_total / 8), 16);
    if (ksplit < 1) ksplit = 1;
  }
  if (ksplit > 1) {
    const size_t need = static_cast<size_t>(ksplit) * M * N * sizeof(float);
    if (workspace == nullptr || ws_bytes < need || e.act == ACT_GEGLU || (N % 4)) ksplit = 1;
  }
  p.ksplit = ksplit;
  p.kb_per_split = (p.kb_total + ksplit - 1) / ksplit;
  // drop empty trailing splits
  p.ksplit = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  p.partial = reinterpret_cast<float*>(workspace);
  p.ln_stats = e.ln_stats; p.ln_mstat = e.ln_mstat; p.ln_parts = e.ln_parts; p.ln_on_cols = e.ln_on_cols;
  if (e.stats_parts) *e.stats_parts = 2 * p.tilesN;
  p.ln_inv_dim = e.ln_dim > 0 ? 1.f / static_cast<float>(e.ln_dim) : 0.f; p.ln_eps = e.ln_eps;
  p.ln_colsum = e.ln_colsum; p.ln_rowbias = e.ln_rowbias; p.stats_out = e.stats_out;
  p.timeline = g_timeline;
  static const int epi_alt = [] { const char* ev = getenv("VDB_EPI_ALT"); return (ev && ev[0] == '0') ? 0 : 1; }();
  p.epi_alt = epi_alt;
  // CTA pairs (cta_group::2) whenever the M tiles pair up and there is no split-K pass
  static const int pair_mode = [] { const char* ev = getenv("VDB_PAIR"); return ev ? atoi(ev) : 0; }();
  const bool pair = pair_mode != 0 && p.ksplit == 1 && (tilesM % 2) == 0 && BN >= 128 && !ln_in && !st_out && e.act != ACT_GEGLU;
  // N-fast tile order (VDB_NFAST=1, opt-in until measured): only when every CTA keeps its N tile from one of its tiles to
  // the next (grid % tilesN == 0: the bias tile cached in shared memory stays valid) and A is too big to survive in L2
  // between two M sweeps (FF-out at the 64x64 level re-reads its 84 MB A operand: 170.7 MB of DRAM traffic against
  // 127 MB algorithmic, profiles/r01_ncu_full_v8.txt)
  static const int nfast_mode = [] { const char* ev = getenv("VDB_NFAST"); return ev ? atoi(ev) : 0; }();
  {
    const int grid = std::min(mn_tiles * p.ksplit, num_sms());
    const double a_bytes = static_cast<double>(M) * static_cast<double>(Ktot) * 2.0;
    p.nfast = (nfast_mode != 0 && !pair && p.ksplit == 1 && p.tilesN > 1 && (grid % p.tilesN) == 0 &&
               (nfast_mode == 2 || a_bytes > 48e6) && !ln_in) ? 1 : 0;   // (the LN modes prefetch along the M-fast order)
  }
  // contiguous tile ranges (VDB_CHUNKED=1; default off) where the strided walk would change its N tile within a CTA's sequence
  // more than a contiguous one does: several N tiles and a few tiles per CTA.  Measured neutral on every UNet shape (GEGLU 64x64:
  // 50.4 vs 50.3 us, bench 481.96 vs 481.62 ms; profiles/r02_visit_ch_chunked_tile_walk.log): the table reloads it saves were not
  // on the critical path.
  {
    static const int chunked_mode = [] { const char* ev = getenv("VDB_CHUNKED"); return ev ? atoi(ev) : 0; }();
    const long long units = static_cast<long long>(tilesM / (pair ? 2 : 1)) * p.tilesN * p.ksplit;
    const int grid = static_cast<int>(std::min<long long>(units, pair ? num_sms() / 2 : num_sms()));
    p.chunked = (chunked_mode != 0 && !p.nfast && p.ksplit == 1 && p.tilesN > 1 && units >= 3LL * grid) ? 1 : 0;
  }
  int rc = make_tmap_2d(&p.tmB, Wt, static_cast<uint64_t>(Ktot), static_cast<uint64_t>(N),
                        static_cast<uint64_t>(ldw) * 2, kBlockK, pair ? BN / 2 : BN);
  if (rc) return rc;
  const int num_tiles = mn_tiles * p.ksplit;
  // epilogue specialisation (see igemm_kernel): 1 = plain bf16 fast path, 2 = GEGLU, 0 = everything else
  static const int spec = [] { const char* ev = getenv("VDB_IGEMM_SPEC"); return (ev && ev[0] == '0') ? 0 : 1; }();
  int mode = 0;
  // one bias row per tile: shared bias, or per-image rows with tiles that never straddle two images
  const bool one_bias_row = e.bias == nullptr || e.bias_bstride == 0 ||
                            (p.TB == 1 && (static_cast<long long>(p.Ho) * p.Wo == p.rows_per_batch ||
                                           (p.Ho == 1 && p.Bo == 1 && p.rows_per_batch % kBlockM == 0)));
  if (spec && p.ksplit == 1 && !e.out_f32 && one_bias_row) {
    if (e.act == ACT_GEGLU && BN == 256) mode = 2;
    else if (e.act == ACT_NONE && e.alpha == 1.f && (N % 32) == 0) mode = 1;
  }
  // TMA-store epilogues (modes 3 / 4 = modes 1 / 2 with the output tile leaving through shared memory + cp.async.bulk.tensor;
  // VDB_EPI_TMA=0 keeps the transposing epilogues): the warp's 32 rows x 32 columns must be one box of the output tensor map
  static const int epi_tma = [] { const char* ev = getenv("VDB_EPI_TMA"); return (ev && ev[0] == '0') ? 0 : 1; }();
  if (epi_tma && (mode == 1 || mode == 2) && (reinterpret_cast<uintptr_t>(e.out) & 15) == 0 &&
      (!e.resid || (reinterpret_cast<uintptr_t>(e.resid) & 15) == 0)) {
    const int bw = std::min(p.TW, 32), bh = std::min(p.TH, 32 / bw), bb = 32 / (bw * bh);
    const long long ncols = (mode == 2) ? N / 2 : N;
    // out_parity >= 0: the same tile, written into every second pixel of every second row of the [B, 2Ho, 2Wo, N] tensor —
    // only the strides and the base of the output tensor map change, the kernel does not know
    const int py = e.out_parity >= 0 ? (e.out_parity >> 1) : 0, px = e.out_parity >= 0 ? (e.out_parity & 1) : 0;
    const uint64_t il = e.out_parity >= 0 ? 2 : 1;
    const void* obase = reinterpret_cast<const __nv_bfloat16*>(e.out) + (static_cast<long long>(py) * (il * p.Wo) + px) * e.ldo;
    if (bb <= p.TB &&
        make_tmap_4d_sw64(&p.tmO, obase, static_cast<uint64_t>(ncols), static_cast<uint64_t>(p.Wo), static_cast<uint64_t>(p.Ho),
                          static_cast<uint64_t>(p.Bo), il * static_cast<uint64_t>(e.ldo) * 2,
                          il * il * static_cast<uint64_t>(p.Wo) * e.ldo * 2,
                          il * il * static_cast<uint64_t>(p.Ho) * p.Wo * e.ldo * 2, 32, bw, bh, bb) == 0)
      mode += 2;
  }
  if (e.out_parity >= 0 && mode != 3)
    return set_error(VDB_ERR_UNSUPPORTED, "igemm: the interleaved-output upsample modes need the TMA-store epilogue (bf16 out, no "
                                          "activation, N %% 32 == 0, aligned out, VDB_EPI_TMA != 0)");
  if (ln_in || st_out) {
    // folded LayerNorm: only on the TMA-store epilogues (bf16 out, act none / GEGLU, alpha 1, N % 32 == 0, aligned pointers)
    if (ln_in && st_out) return set_error(VDB_ERR_UNSUPPORTED, "igemm: a launch either consumes or produces LayerNorm statistics");
    if (mode != 3 && !(mode == 4 && ln_in))
      return set_error(VDB_ERR_UNSUPPORTED, "igemm: LayerNorm statistics need the TMA-store epilogue (bf16 out, no activation or "
                                            "GEGLU, alpha 1, N %% 32 == 0, 16-byte aligned out / resid, VDB_EPI_TMA != 0)");
    if (ln_in && e.resid) return set_error(VDB_ERR_UNSUPPORTED, "igemm: a folded-LayerNorm GEMM takes no residual");
    if (ln_in && mode == 4 && e.ln_on_cols) return set_error(VDB_ERR_UNSUPPORTED, "igemm: GEGLU with column statistics");
    mode = st_out ? 7 : mode + 2;
  }
  g_igemm_last[0] = mode; g_igemm_last[1] = BN; g_igemm_last[2] = p.ksplit; g_igemm_last[3] = pair ? 1 : 0;
  if (pair && mode == 3) {
    ++g_pair_launches;                 // CTA pairs with the TMA-store epilogue (each CTA stores its own 128 rows)
    switch (BN) {
      case 128: rc = launch_igemm<128, 7, 2, 8, 3>(p, num_tiles / 2, stream); break;
      case 160: rc = launch_igemm<160, 7, 2, 8, 3>(p, num_tiles / 2, stream); break;
      default: rc = launch_igemm<256, 6, 2, 8, 3>(p, num_tiles / 2, stream); break;
    }
  } else if (pair) {
    ++g_pair_launches;
    switch (BN) {
      case 128: rc = launch_igemm<128, 7, 2, 8, 0>(p, num_tiles / 2, stream); break;
      case 160: rc = launch_igemm<160, 7, 2, 8, 0>(p, num_tiles / 2, stream); break;
      default: rc = launch_igemm<256, 6, 2, 8, 0>(p, num_tiles / 2, stream); break;
    }
  } else if (mode == 7) {
    switch (BN) {
      case 64: rc = launch_igemm<64, 8, 1, 8, 7>(p, num_tiles, stream); break;
      case 128: rc = launch_igemm<128, 6, 1, 8, 7>(p, num_tiles, stream); break;
      case 160: rc = launch_igemm<160, 5, 1, 8, 7>(p, num_tiles, stream); break;
      default: rc = launch_igemm<256, 4, 1, 8, 7>(p, num_tiles, stream); break;
    }
  } else if (mode == 6) {
    rc = launch_igemm<256, 4, 1, 8, 6>(p, num_tiles, stream);
  } else if (mode == 5) {
    switch (BN) {
      case 64: rc = launch_igemm<64, 8, 1, 8, 5>(p, num_tiles, stream); break;
      case 128: rc = launch_igemm<128, 6, 1, 8, 5>(p, num_tiles, stream); break;
      case 160: rc = launch_igemm<160, 5, 1, 8, 5>(p, num_tiles, stream); break;
      default: rc = launch_igemm<256, 4, 1, 8, 5>(p, num_tiles, stream); break;
    }
  } else if (mode == 4) {
    rc = launch_igemm<256, 4, 1, 8, 4>(p, num_tiles, stream);
  } else if (mode == 3) {
    switch (BN) {
      case 64: rc = launch_igemm<64, 8, 1, 8, 3>(p, num_tiles, stream); break;
      case 128: rc = launch_igemm<128, 6, 1, 8, 3>(p, num_tiles, stream); break;
      case 160: rc = launch_igemm<160, 5, 1, 8, 3>(p, num_tiles, stream); break;
      default: rc = launch_igemm<256, 4, 1, 8, 3>(p, num_tiles, stream); break;
    }
  } else if (mode == 2) {
    rc = launch_igemm<256, 4, 1, 8, 2>(p, num_tiles, stream);
  } else if (mode == 1) {
    switch (BN) {
      case 64: rc = launch_igemm<64, 8, 1, 8, 1>(p, num_tiles, stream); break;
      case 128: rc = launch_igemm<128, 6, 1, 8, 1>(p, num_tiles, stream); break;
      case 160: rc = launch_igemm<160, 5, 1, 8, 1>(p, num_tiles, stream); break;
      default: rc = launch_igemm<256, 4, 1, 8, 1>(p, num_tiles, stream); break;
    }
  } else {
    switch (BN) {
      case 64: rc = launch_igemm<64, 8, 1, 8, 0>(p, num_tiles, stream); break;
      case 128: rc = launch_igemm<128, 6, 1, 8, 0>(p, num_tiles, stream); break;
      case 160: rc = launch_igemm<160, 5, 1, 8, 0>(p, num_tiles, stream); break;
      default: rc = launch_igemm<256, 4, 1, 8, 0>(p, num_tiles, stream); break;
    }
  }
  if (rc) return rc;
  if (p.ksplit > 1) {
    const long long total = M * (N / 4);
    const int threads = 256;
    const int blocks = static_cast<int>(std::min<long long>((total + threads - 1) / threads, num_sms() * 8LL));
    VDB_PREFER_MAX_SMEM(splitk_reduce_kernel);
    VDB_CUDA_CHECK(launch_pdl(splitk_reduce_kernel, dim3(blocks), dim3(threads), 0, stream, (const float*)p.partial,
                              p.ksplit, M, static_cast<int>(N), p.bias, p.bias_bstride, p.rows_per_batch, p.resid,
                              p.ldr, p.out, p.ldo, p.out_f32, p.act, p.alpha));
    count_launch();
  }
  return VDB_OK;
}

static int pow2_ceil(int v) { int t = 1; while (t < v) t <<= 1; return t; }

// M tile = 128 output pixels as a (TW, TH, TB) box of the (W, H, B) pixel grid; box extents are
// powers of two so that TW*TH*TB == 128 (rows past the grid are zero-filled by TMA and masked on store).
static void set_tile_shape(IgemmParams& p, int Wo, int Ho, int Bo) {
  p.Wo = Wo; p.Ho = Ho; p.Bo = Bo;
  const int TW = std::min(pow2_ceil(Wo), 128);
  const int TH = std::min(pow2_ceil(Ho), 128 / TW);
  const int TB = 128 / (TW * TH);
  p.TW = TW; p.TH = TH; p.TB = TB;
  p.tilesW = (Wo + TW - 1) / TW;
  p.tilesH = (Ho + TH - 1) / TH;
  p.tilesB = (Bo + TB - 1) / TB;
}

}  // namespace vdb

using namespace vdb;

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

// debug aid (not part of the product ABI): device buffer of 16*8 u64 receiving CTA 0's per-tile role timestamps
void vdb_debug_igemm_timeline(void* buf) { g_timeline = reinterpret_cast<unsigned long long*>(buf); }
// debug aid: how many igemm launches ran as CTA pairs (cta_group::2)
long long vdb_debug_pair_launches(void) { return g_pair_launches; }
// debug aid (host side): out4 = {epilogue mode after the TMA-store / LayerNorm promotion (0..7), BN, ksplit, CTA pair 0/1} of the
// last vdb_gemm_bf16 / vdb_gemm_ln_bf16 / vdb_conv3x3_bf16 launch on the calling thread ({-1, 0, 0, 0} before the first one)
void vdb_debug_igemm_last(int* out4) { for (int i = 0; i < 4; ++i) out4[i] = g_igemm_last[i]; }

// out[M,N] = act(alpha * ([A | A2] @ W^T + bias)) + resid     (see include/vdb200.h)
int vdb_gemm_bf16(const void* A, long long M, long long K, long long lda, const void* A2, long long K2,
                  long long lda2, const void* W, long long N, long long ldw, const float* bias,
                  long long bias_bstride, long long rows_per_batch, const void* resid, long long ldr, void* out,
                  long long ldo, int out_f32, int act, float alpha, int bn, int ksplit, void* workspace,
                  size_t ws_bytes, void* stream) {
  if (!A || !W || !out || M <= 0 || N <= 0 || K <= 0) return set_error(VDB_ERR_INVALID, "gemm: null/empty argument");
  if ((K % 8) || (lda % 8) || (ldw % 8)) return set_error(VDB_ERR_INVALID, "gemm: K, lda, ldw must be multiples of 8");
  if (A2 && ((K % kBlockK) || (K2 % 8) || (lda2 % 8)))
    return set_error(VDB_ERR_INVALID, "gemm: two-source A needs K % 64 == 0 and K2, lda2 % 8 == 0");
  if (M > 0x7fffffffLL || N > 0x7fffffffLL) return set_error(VDB_ERR_INVALID, "gemm: dimension too large");
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  // GEMM view of the pixel grid: one row of M "pixels"; the box is always 128 rows (TMA zero-fills past M)
  p.Wo = static_cast<int>(M); p.Ho = 1; p.Bo = 1;
  p.TW = kBlockM; p.TH = 1; p.TB = 1;
  p.tilesW = static_cast<int>((M + kBlockM - 1) / kBlockM); p.tilesH = 1; p.tilesB = 1;
  int rc = make_tmap_4d(&p.tmA[0], A, K, M, 1, 1, lda * 2, lda * 2 * M, lda * 2 * M, kBlockK, p.TW, 1, 1);
  if (rc) return rc;
  p.seg[0] = ASeg{0, 0, 0, static_cast<int16_t>((K + kBlockK - 1) / kBlockK), 0};
  p.nseg = 1;
  p.kb_total = p.seg[0].nkb;
  if (A2) {
    rc = make_tmap_4d(&p.tmA[1], A2, K2, M, 1, 1, lda2 * 2, lda2 * 2 * M, lda2 * 2 * M, kBlockK, p.TW, 1, 1);
    if (rc) return rc;
    p.seg[1] = ASeg{1, 0, 0, static_cast<int16_t>((K2 + kBlockK - 1) / kBlockK), 0};
    p.nseg = 2;
    p.kb_total += p.seg[1].nkb;
  }
  for (int i = p.nseg; i < kMaxA; ++i) p.tmA[i] = p.tmA[0];
  IgemmEpilogue e;
  e.bias = bias; e.bias_bstride = bias_bstride; e.rows_per_batch = static_cast<int>(rows_per_batch);
  e.resid = resid; e.ldr = ldr; e.out = out; e.ldo = ldo; e.out_f32 = out_f32; e.act = act; e.alpha = alpha;
  return run_igemm(p, W, N, K + (A2 ? K2 : 0), ldw, e, bn, ksplit, workspace, ws_bytes,
                   reinterpret_cast<cudaStream_t>(stream));
}

// GEMM with a LayerNorm folded in (consumer) or LayerNorm statistics written out (producer); see include/vdb200.h
int vdb_gemm_ln_bf16(const void* A, long long M, long long K, long long lda, const void* W, long long N, long long ldw,
                     const float* bias, const void* resid, long long ldr, void* out, long long ldo, int act,
                     const float* ln_stats, long long ln_rows, int ln_parts, int ln_dim, float ln_eps, const float* ln_colsum,
                     int ln_on_cols, const float* ln_rowbias, float* stats_out, int* stats_parts, int bn, void* stream) {
  if (!A || !W || !out || M <= 0 || N <= 0 || K <= 0) return set_error(VDB_ERR_INVALID, "gemm_ln: null/empty argument");
  if ((K % 8) || (lda % 8) || (ldw % 8)) return set_error(VDB_ERR_INVALID, "gemm_ln: K, lda, ldw must be multiples of 8");
  if (M > 0x7fffffffLL || N > 0x7fffffffLL) return set_error(VDB_ERR_INVALID, "gemm_ln: dimension too large");
  if (!ln_stats && !stats_out) return set_error(VDB_ERR_INVALID, "gemm_ln: neither ln_stats nor stats_out given (use vdb_gemm_bf16)");
  if (ln_stats) {
    if (!ln_colsum || ln_dim <= 0 || ln_dim != K || ln_parts <= 0)
      return set_error(VDB_ERR_INVALID, "gemm_ln: need ln_colsum, ln_parts > 0 and ln_dim == K");
    if (ln_rows < (ln_on_cols ? N : M)) return set_error(VDB_ERR_INVALID, "gemm_ln: statistics table has too few rows");
  }
  if (stats_out && ((N % 32) || !stats_parts)) return set_error(VDB_ERR_INVALID, "gemm_ln: stats_out needs N %% 32 == 0 and stats_parts");
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  p.Wo = static_cast<int>(M); p.Ho = 1; p.Bo = 1;
  p.TW = kBlockM; p.TH = 1; p.TB = 1;
  p.tilesW = static_cast<int>((M + kBlockM - 1) / kBlockM); p.tilesH = 1; p.tilesB = 1;
  int rc = make_tmap_4d(&p.tmA[0], A, K, M, 1, 1, lda * 2, lda * 2 * M, lda * 2 * M, kBlockK, p.TW, 1, 1);
  if (rc) return rc;
  p.seg[0] = ASeg{0, 0, 0, static_cast<int16_t>((K + kBlockK - 1) / kBlockK), 0};
  p.nseg = 1;
  p.kb_total = p.seg[0].nkb;
  for (int i = p.nseg; i < kMaxA; ++i) p.tmA[i] = p.tmA[0];
  IgemmEpilogue e;
  e.bias = bias; e.resid = resid; e.ldr = ldr; e.out = out; e.ldo = ldo; e.act = act;
  e.ln_stats = ln_stats; e.ln_mstat = ln_rows; e.ln_parts = ln_parts; e.ln_dim = ln_dim; e.ln_eps = ln_eps; e.ln_colsum = ln_colsum;
  e.ln_on_cols = ln_on_cols; e.ln_rowbias = ln_rowbias; e.stats_out = stats_out; e.stats_parts = stats_parts;
  return run_igemm(p, W, N, K, ldw, e, bn, 1, nullptr, 0, reinterpret_cast<cudaStream_t>(stream));
}

// 3x3 convolution on NHWC bf16 as implicit GEMM.
//   mode 0: stride 1, pad 1                       (out H x W)
//   mode 1: stride 2, pad 1                       (out H/2 x W/2)      openaimodel.py:150-152
//   mode 2: stride 2, pad (0,1,0,1) then pad 0    (out H/2 x W/2)      autokl_modules.py:72-76
//   mode 3 + 2*py + px: one parity sub-lattice of "nearest 2x upsample, then 3x3 conv pad 1" (openaimodel.py:107-117,
//           autokl_modules.py:54-58) computed on the SOURCE image: output pixel (2y+py, 2x+px) of the upsampled conv only
//           sees the 2x2 source pixels (y + ty - 1 + py, x + tx - 1 + px), ty, tx in {0,1}, so the 9 taps fold into 4 with
//           pre-summed weights (host: fold_upsample_conv3x3).  X = source [B,H,W,C], out = [B,H,W,N] (that parity, dense),
//           Wt = [N, 4*C] with K ordered (ty, tx, c).  2.25x fewer FLOPs than upsampling first; no skip inputs.
// Wt is [N, 9*C + Cs1 + Cs2] bf16 with K ordered (ky, kx, c) then the 1x1-skip columns.
// skip1/skip2: optional raw NHWC tensors at OUTPUT resolution whose 1x1 conv is accumulated too.
int vdb_conv3x3_bf16(const void* X, int B, int H, int Wd, int C, int mode, const void* Wt, int N, long long ldw,
                     const void* skip1, int Cs1, const void* skip2, int Cs2, const float* bias,
                     long long bias_bstride, const void* resid, long long ldr, void* out, long long ldo,
                     int out_f32, int act, int bn, int ksplit, void* workspace, size_t ws_bytes, void* stream) {
  if (!X || !Wt || !out || B <= 0 || H <= 0 || Wd <= 0 || C <= 0 || N <= 0)
    return set_error(VDB_ERR_INVALID, "conv3x3: null/empty argument");
  if ((C % kBlockK) || (ldw % 8)) return set_error(VDB_ERR_INVALID, "conv3x3: C must be a multiple of 64, ldw of 8");
  if ((skip1 && (Cs1 % kBlockK)) || (skip2 && (Cs2 % kBlockK)))
    return set_error(VDB_ERR_INVALID, "conv3x3: skip channels must be multiples of 64");
  if (mode < 0 || mode > 10) return set_error(VDB_ERR_INVALID, "conv3x3: bad mode");
  const int out_parity = mode >= 7 ? mode - 7 : -1;     // modes 7..10 = modes 3..6 writing into the interleaved [B, 2H, 2W, N] tensor
  if (mode >= 7) mode -= 4;
  if (out_parity >= 0 && (resid || out_f32 || ksplit > 1)) return set_error(VDB_ERR_INVALID, "conv3x3: modes 7..10 take no residual, bf16 out, no split-K");
  if (out_parity >= 0) ksplit = 1;
  const bool strided = (mode == 1 || mode == 2), folded = mode >= 3;
  if (strided && ((H & 1) || (Wd & 1))) return set_error(VDB_ERR_UNSUPPORTED, "conv3x3: stride 2 needs even H, W");
  if (folded && (skip1 || skip2)) return set_error(VDB_ERR_INVALID, "conv3x3: the folded-upsample modes take no skip inputs");
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  const int Ho = strided ? H / 2 : H, Wo = strided ? Wd / 2 : Wd;
  set_tile_shape(p, Wo, Ho, B);
  const uint64_t eb = 2;
  const int nkb = C / kBlockK;
  int rc;
  int nmaps = 0;
  int ntaps = 9;
  if (mode == 0 || folded) {
    rc = make_tmap_4d(&p.tmA[0], X, C, Wd, H, B, C * eb, (uint64_t)Wd * C * eb, (uint64_t)H * Wd * C * eb, kBlockK,
                      p.TW, p.TH, p.TB);
    if (rc) return rc;
    nmaps = 1;
    if (mode == 0) {
      for (int t = 0; t < 9; ++t)
        p.seg[t] = ASeg{0, static_cast<int16_t>(t % 3 - 1), static_cast<int16_t>(t / 3 - 1), static_cast<int16_t>(nkb), 0};
    } else {
      const int py = (mode - 3) >> 1, px = (mode - 3) & 1;
      ntaps = 4;
      for (int t = 0; t < 4; ++t)      // t = ty * 2 + tx; source pixel (y + ty - 1 + py, x + tx - 1 + px)
        p.seg[t] = ASeg{0, static_cast<int16_t>((t & 1) - 1 + px), static_cast<int16_t>((t >> 1) - 1 + py), static_cast<int16_t>(nkb), 0};
    }
  } else {
    // four parity sub-lattices of the input: X[b, 2*yo+py, 2*xo+px, c]
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        const uint8_t* base = reinterpret_cast<const uint8_t*>(X) + (static_cast<uint64_t>(py) * Wd + px) * C * eb;
        rc = make_tmap_4d(&p.tmA[py * 2 + px], base, C, Wo, Ho, B, 2ull * C * eb, 2ull * Wd * C * eb,
                          (uint64_t)H * Wd * C * eb, kBlockK, p.TW, p.TH, p.TB);
        if (rc) return rc;
      }
    nmaps = 4;
    for (int t = 0; t < 9; ++t) {
      const int ky = t / 3, kx = t % 3;
      int py, dy, px, dx;
      if (mode == 1) {  // input row = 2*yo + ky - 1
        py = (ky == 1) ? 0 : 1; dy = (ky == 0) ? -1 : 0;
        px = (kx == 1) ? 0 : 1; dx = (kx == 0) ? -1 : 0;
      } else {          // input row = 2*yo + ky (zero pad on bottom/right only)
        py = (ky == 1) ? 1 : 0; dy = (ky == 2) ? 1 : 0;
        px = (kx == 1) ? 1 : 0; dx = (kx == 2) ? 1 : 0;
      }
      p.seg[t] = ASeg{static_cast<int16_t>(py * 2 + px), static_cast<int16_t>(dx), static_cast<int16_t>(dy),
                      static_cast<int16_t>(nkb), 0};
    }
  }
  p.nseg = ntaps;
  p.kb_total = ntaps * nkb;
  const void* sk[2] = {skip1, skip2};
  const int sc[2] = {Cs1, Cs2};
  for (int i = 0; i < 2; ++i) {
    if (!sk[i]) continue;
    rc = make_tmap_4d(&p.tmA[nmaps], sk[i], sc[i], Wo, Ho, B, sc[i] * eb, (uint64_t)Wo * sc[i] * eb,
                      (uint64_t)Ho * Wo * sc[i] * eb, kBlockK, p.TW, p.TH, p.TB);
    if (rc) return rc;
    p.seg[p.nseg] = ASeg{static_cast<int16_t>(nmaps), 0, 0, static_cast<int16_t>(sc[i] / kBlockK), 0};
    p.kb_total += sc[i] / kBlockK;
    ++p.nseg;
    ++nmaps;
  }
  for (int i = nmaps; i < kMaxA; ++i) p.tmA[i] = p.tmA[0];
  IgemmEpilogue e;
  e.bias = bias; e.bias_bstride = bias_bstride; e.rows_per_batch = Ho * Wo;
  e.resid = resid; e.ldr = ldr; e.out = out; e.ldo = ldo; e.out_f32 = out_f32; e.act = act; e.alpha = 1.f;
  e.out_parity = out_parity;
  return run_igemm(p, Wt, N, static_cast<long long>(p.kb_total) * kBlockK, ldw, e, bn, ksplit, workspace, ws_bytes,
                   reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
