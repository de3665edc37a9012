// Common sm_100a device helpers for the vdb200 kernels: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (UMMA / TMEM) wrappers and small math utils.
// Everything here is inline PTX; no CUTLASS/CuTe dependency.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace vdb {

#define VDB_DEVINL __device__ __forceinline__

// ----------------------------------------------------------------------------
// status codes of the C ABI (include/vdb200.h mirrors these)
// ----------------------------------------------------------------------------
enum : int {
  VDB_OK = 0,
  VDB_ERR_INVALID = 1,     // bad argument (shape/alignment/null)
  VDB_ERR_CUDA = 2,        // CUDA runtime / driver error (see vdb_last_error)
  VDB_ERR_UNSUPPORTED = 3, // shape outside what the kernels implement
};

// 16-byte shared-memory load through a 32-bit shared address (a pointer derived from the aligned dynamic window has lost its
// address space: the compiler emits generic LD.E instead of LDS)
VDB_DEVINL float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

VDB_DEVINL uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

VDB_DEVINL uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}

VDB_DEVINL bool elect_one() {
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

// ----------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------
VDB_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
VDB_DEVINL void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
VDB_DEVINL void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
VDB_DEVINL void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
VDB_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
VDB_DEVINL bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
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
VDB_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ----------------------------------------------------------------------------
// TMA tiled loads (global -> shared), completion on an mbarrier
// ----------------------------------------------------------------------------
VDB_DEVINL void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
VDB_DEVINL void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
VDB_DEVINL void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// TMA tiled store (shared -> global), bulk-group completion.  The issuing thread must have ordered the generic-proxy
// shared-memory writes of the tile before it (fence.proxy.async by every writer, then a barrier).
VDB_DEVINL void tma_store_4d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
          reinterpret_cast<uint64_t>(m)),
      "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
VDB_DEVINL void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
VDB_DEVINL void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
VDB_DEVINL void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

// ----------------------------------------------------------------------------
// tcgen05: TMEM allocation, MMA, commit, loads/stores, fences
// ----------------------------------------------------------------------------
template <uint32_t kCols>
VDB_DEVINL void tmem_alloc(uint32_t* smem_holder) {  // whole warp must call
  static_assert(kCols == 32 || kCols == 64 || kCols == 128 || kCols == 256 || kCols == 512, "");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_holder)),
               "n"(kCols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
template <uint32_t kCols>
VDB_DEVINL void tmem_dealloc(uint32_t taddr) {  // whole warp must call
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols));
}
VDB_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
VDB_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, issued by ONE thread.
VDB_DEVINL void umma_bf16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Warp-uniform issue forms (suffix _w): EVERY lane of the warp executes the call with identical operands and ONE elected lane
// issues the instruction.  Keeping the surrounding control flow convergent lets ptxas hold descriptors in uniform registers:
// under `if (lane == 0)` every tcgen05.mma was wrapped in an ELECT / R2UR / BRA.U.ANY loop (~90 cycles per MMA in the
// attention kernel, whose MMAs only run 24-64 tensor cycles each: profiles/r02_attention_fa_timeline_v1.txt).
VDB_DEVINL void umma_bf16_ss_w(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
VDB_DEVINL void umma_bf16_ts_w(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
VDB_DEVINL void umma_commit_w(uint64_t* bar) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}\n" ::"r"(smem_u32(bar))
      : "memory");
}
// Arrive (count 1) on an mbarrier once all previously issued MMAs of this thread retire.
VDB_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}

// ----------------------------------------------------------------------------
// CTA pair (cta_group::2): two CTAs of a 2-cluster (one TPC) execute ONE 256-row MMA.  Each CTA stages its own
// 128 rows of A and HALF of the B tile; the leader (cluster rank 0) issues the MMA, which reads both shared
// memories and writes 128 accumulator lanes into each CTA's TMEM.  TMA completions of both CTAs land on the
// leader's mbarrier; tcgen05.commit multicasts its arrival to the same barrier offset in both CTAs.
// ----------------------------------------------------------------------------
VDB_DEVINL uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
VDB_DEVINL void cluster_sync_all() {   // every thread of both CTAs
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
VDB_DEVINL uint32_t mapa_u32(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
VDB_DEVINL void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
VDB_DEVINL void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
VDB_DEVINL void tma_load_4d_pair(void* smem_dst, const CUtensorMap* m, uint32_t leader_bar, int c0, int c1,
                                 int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
template <uint32_t kCols>
VDB_DEVINL void tmem_alloc_pair(uint32_t* smem_holder) {  // the same warp of BOTH CTAs must call, same holder offset
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_holder)),
               "n"(kCols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
}
template <uint32_t kCols>
VDB_DEVINL void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols));
}
VDB_DEVINL void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrival (count 1) on the barrier at this shared-memory offset in BOTH CTAs once the issued MMAs retire
VDB_DEVINL void umma_commit_pair(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// warp-uniform forms (see umma_bf16_ss_w): every lane of the issuing warp runs the loop, one elected lane issues
VDB_DEVINL void umma_bf16_ss_pair_w(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
VDB_DEVINL void umma_commit_pair_w(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "h"(mask)
      : "memory");
}

// K-major, 128-byte-swizzled shared-memory operand descriptor.
// Tile = rows of 128 B (64 bf16 along K), 8-row groups 1024 B apart (SBO), base 1024-B aligned.
// Bits: [0,14) addr>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) layout=2.
VDB_DEVINL uint64_t make_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;            // LBO (unused for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;    // SBO
  d |= static_cast<uint64_t>(1) << 46;            // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;            // SWIZZLE_128B
  return d;
}

// Instruction descriptor, kind::f16: bf16 x bf16 -> f32, both operands K-major, dense.
VDB_DEVINL constexpr uint32_t make_idesc_bf16(uint32_t m, uint32_t n) {
  return (1u << 4)            // c_format = F32
         | (1u << 7)          // a_format = BF16
         | (1u << 10)         // b_format = BF16
         | ((n >> 3) << 17)   // N >> 3
         | ((m >> 4) << 24);  // M >> 4
}

// TMEM -> registers, 32 lanes x 32 bit, 32 consecutive columns (thread i <- lane base+i).
VDB_DEVINL void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
VDB_DEVINL void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
VDB_DEVINL void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
VDB_DEVINL void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
      "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
      "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T: A (M x 16 bf16 per step = 128 lanes x 8 packed 32-bit columns, K-major) read from
// tensor memory, B from shared memory.  Used for O += P V with P written by the softmax warps (tcgen05.st): the 128 x 128
// bf16 P tile never crosses shared memory (an SS product at N = 48 re-reads 4 KB of A per 24 tensor cycles and made the
// attention kernel shared-memory-bandwidth bound).
VDB_DEVINL void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
VDB_DEVINL void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
VDB_DEVINL void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// nanosecond wall clock shared by all SMs (debug timelines, watchdogs)
VDB_DEVINL unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ----------------------------------------------------------------------------
// programmatic dependent launch: a kernel launched with the PDL attribute may start while its predecessor
// drains; it must not touch dependent global memory before pdl_wait(). No-ops for ordinary launches.
// ----------------------------------------------------------------------------
VDB_DEVINL void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
VDB_DEVINL void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ----------------------------------------------------------------------------
// small math / packing helpers
// ----------------------------------------------------------------------------
VDB_DEVINL uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
VDB_DEVINL float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}
// Packed fp32 pairs (sm_100 FFMA2 / FADD2: two IEEE fp32 operations per issue slot, same rounding as the scalar forms)
VDB_DEVINL unsigned long long pack_f2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
VDB_DEVINL void unpack_f2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
VDB_DEVINL unsigned long long fma_f2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
VDB_DEVINL unsigned long long add_f2(unsigned long long a, unsigned long long b) {
  unsigned long long d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// 2^x on the MUFU pipe (one SFU op)
VDB_DEVINL float ex2_mufu(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 2^x on the FMA/ALU pipes: round-to-nearest split x = n + f, cubic minimax of 2^f on [-0.5, 0.5]
// (max rel. error 7.7e-5, far below bf16's 4e-3), exponent add through the integer pipe.
VDB_DEVINL float ex2_poly(float x) {
  x = fmaxf(x, -126.0f);
  const float r = x + 12582912.0f;          // 1.5 * 2^23: low mantissa bits now hold rint(x)
  const float f = x - (r - 12582912.0f);
  float p = fmaf(0.0550886838f, f, 0.242604051f);
  p = fmaf(p, f, 0.693276242f);
  p = fmaf(p, f, 0.99992894f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(r) << 23));
}
VDB_DEVINL float silu_f(float x) { return __fdividef(x, 1.0f + __expf(-x)); }
// SiLU for bf16 outputs: x * sigmoid(x) = 0.5x * (1 + tanh(x/2)) with ONE MUFU op (tanh.approx, rel. error < 5e-4,
// below bf16 rounding); the exp+rcp form needs two and made GroupNorm-apply MUFU-bound.
VDB_DEVINL float silu_bf16_f(float x) {
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(0.5f * x));
  const float hx = 0.5f * x;
  return fmaf(hx, th, hx);
}
VDB_DEVINL float gelu_erf_f(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
// exact-erf GELU through Abramowitz-Stegun 7.1.26 (|erf error| <= 1.5e-7): 2 MUFU + ~10 FMA instead of erff()
VDB_DEVINL float gelu_as_f(float x) {
  const float z = fabsf(x) * 0.70710678118654752f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, z, 1.0f));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float erf_abs = 1.0f - poly * t * __expf(-z * z);
  return 0.5f * x * (1.0f + copysignf(erf_abs, x));
}
// GELU for bf16 outputs (GEGLU epilogue): x * Phi(x) with Phi through one tanh.approx MUFU op.  The tanh form
// differs from the erf form by < 3e-4 absolute in Phi and tanh.approx adds < 5e-4 relative — both below the
// 2^-9 relative rounding of the bf16 value this feeds, so results match the exact-erf GELU to within one bf16 ulp.
VDB_DEVINL float gelu_fast_f(float x) {
  const float u = x * fmaf(0.0356774081f, x * x, 0.7978845608f);
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(u));
  const float hx = 0.5f * x;
  return fmaf(hx, th, hx);
}
VDB_DEVINL float quick_gelu_f(float x) { return __fdividef(x, 1.0f + __expf(-1.702f * x)); }
// GPT-2's tanh-form GELU, 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3))) (optimus_gpt2.py:99-100), with the accurate tanhf
VDB_DEVINL float gelu_tanh_f(float x) {
  return 0.5f * x * (1.0f + tanhf(0.7978845608028654f * (x + 0.044715f * x * x * x)));
}

}  // namespace vdb
