// tc.cuh -- hand-written sm_100a building blocks: mbarrier, bulk (TMA) copies, tcgen05 MMA /
// TMEM access, and the 128-byte-swizzled operand "panel" format shared by all MLP kernels.
//
// Panel format (the one data layout every tensor-core operand in this repo uses):
//   a panel holds R rows x 64 16-bit elements (128 bytes per row), rows grouped by 8 into
//   1024-byte swizzle atoms.  Element (r, c) lives at byte
//       (r / 8) * 1024 + (r % 8) * 128 + (((c / 8) ^ (r % 8)) * 16) + (c % 8) * 2
//   which is exactly the canonical UMMA SWIZZLE_128B layout: K-major when the 64 columns are
//   the reduction dimension (SBO = 1024), and -- read transposed -- MN-major when the rows
//   are the reduction dimension (LBO = panel stride, SBO = 1024).  Because the image is the
//   same in shared and global memory, operands move with plain 1-D bulk copies
//   (cp.async.bulk, the TMA engine) and need no tensor maps.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

namespace nerf {
namespace tc {

constexpr uint32_t kPanelCols = 64;         // 16-bit elements per panel row
constexpr uint32_t kPanelRowBytes = 128;
constexpr uint32_t kAtomBytes = 1024;       // 8 rows x 128 B

__host__ __device__ __forceinline__ uint32_t panel_offset(uint32_t row, uint32_t col) {
  return (row >> 3) * kAtomBytes + (row & 7) * kPanelRowBytes + ((((col >> 3) ^ (row & 7)) & 7) << 4) + ((col & 7) << 1);
}
// byte offset of 16-byte chunk `chunk` (0..7) of row `row`
__host__ __device__ __forceinline__ uint32_t panel_chunk_offset(uint32_t row, uint32_t chunk) {
  return (row >> 3) * kAtomBytes + (row & 7) * kPanelRowBytes + (((chunk ^ (row & 7)) & 7) << 4);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---- mbarrier ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---- proxy fences -----------------------------------------------------------------------
// generic-proxy shared-memory writes -> visible to the async proxy (UMMA operand reads, bulk stores)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- bulk copies (TMA engine, 1-D) --------------------------------------------------------
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_smem), "r"(bytes) : "memory");
}
// L2 eviction-priority policies: streamed stash traffic must not evict the (L2-resident, re-read) weight images
__device__ __forceinline__ uint64_t l2_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void bulk_g2s_hint(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(bar), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void bulk_s2g_hint(void* dst, uint32_t src_smem, uint32_t bytes, uint64_t policy) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst), "r"(src_smem), "r"(bytes),
               "l"(policy)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all but the newest N bulk stores have finished READING shared memory
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---- TMEM ------------------------------------------------------------------------------
// one full warp; writes the TMEM base address to *dst_smem
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (taddr.lane + t)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
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

// wait for outstanding tcgen05.ld AND pin the destination registers behind the wait: the "+r" operands stop the
// compiler from hoisting arithmetic on r[] above the wait (the load itself only names them as outputs)
__device__ __forceinline__ void tmem_ld_wait32(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                 "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                 "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// 32 lanes x 16 consecutive fp32 columns (the split epilogues double-buffer at this granularity)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// register reallocation between warp roles (whole warpgroups): producer / MMA warps give registers to the epilogues
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// ---- UMMA descriptors ---------------------------------------------------------------------
// shared-memory matrix descriptor, SWIZZLE_128B (layout type 2), sm_100 version field = 1
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;  // SWIZZLE_128B
  return d;
}
// K-major panel operand: rows = M or N index, 64 columns = one K block; one MMA consumes 16
// columns (32 bytes), so K step j of a panel starts at +32*j bytes.
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t panel_smem, uint32_t kstep) {
  return make_smem_desc(panel_smem + kstep * 32u, 16u, kAtomBytes);
}
// MN-major operand: rows = K (reduction) index, columns = M or N index; successive 64-wide
// column groups are `panel_stride` bytes apart; one MMA consumes 16 rows = 2 atoms.
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t panel_smem, uint32_t kstep, uint32_t panel_stride) {
  return make_smem_desc(panel_smem + kstep * 2u * kAtomBytes, panel_stride, kAtomBytes);
}

enum : uint32_t { kF16 = 0, kBF16 = 1 };
// instruction descriptor for kind::f16, fp32 accumulate
__host__ __device__ constexpr uint32_t make_idesc(uint32_t m, uint32_t n, uint32_t a_fmt, uint32_t b_fmt, uint32_t a_mn_major,
                                                  uint32_t b_mn_major) {
  return (1u << 4) | (a_fmt << 7) | (b_fmt << 10) | (a_mn_major << 15) | (b_mn_major << 16) | ((n >> 3) << 17) |
         ((m >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all MMAs issued so far by this thread arrive on `bar` when they complete (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// ---- CTA pairs (cta_group::2): two CTAs of one cluster share every MMA ------------------------------
// The leader (cluster rank 0) issues M = 256 instructions: rows 0..127 come from its own A operand / TMEM, rows
// 128..255 from the peer's, and each CTA supplies HALF of the B operand (N/2 rows at the same shared-memory
// offset), so per 128 samples only half of every weight panel crosses L2 -> SM and is read from shared memory.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `smem_addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
// Arrive on a barrier of another CTA of the cluster.  Default semantics (release at CTA scope), exactly what the
// CUTLASS cluster barriers use: the data handed over lives in the ARRIVING CTA's shared memory, is made visible to
// the async proxy by fence.proxy.async, and is only ever read through that proxy (tcgen05.mma of the pair).  The
// .release.cluster / .acquire.cluster forms compile to MEMBAR.ALL.GPU before every arrive and CCTL.IVALL (an L1
// flush) after every wait -- measured: the pair kernels ran SLOWER than single-CTA ones with them.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// wait on a LOCAL barrier that threads / TMA / tensor cores of either CTA arrive on
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) { mbar_wait(bar, parity); }
__device__ __forceinline__ void tmem_alloc2(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all MMAs issued so far arrive (once) on the barrier at offset `bar` in EVERY CTA of `cta_mask`
__device__ __forceinline__ void umma_commit2(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(cta_mask)
               : "memory");
}

// ---- misc ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_bf162(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
// 0xFFFF in each 16-bit half whose fp16 value is > 0 (one HSET2.BM)
__device__ __forceinline__ uint32_t half2_gt0_mask(uint32_t w) {
  const __half2 z = __floats2half2_rn(0.f, 0.f);
  return __hgt2_mask(*reinterpret_cast<__half2*>(&w), z);
}
// max(x, 0) on both halves (one HMNMX2): ReLU after the fp16 rounding equals the rounding of the fp32 ReLU
__device__ __forceinline__ uint32_t half2_relu(uint32_t w) {
  const __half2 r = __hmax2(*reinterpret_cast<__half2*>(&w), __floats2half2_rn(0.f, 0.f));
  return *reinterpret_cast<const uint32_t*>(&r);
}
// ReLU mask bit layout used by the forward stash and the dgrad chain: within a 32-column chunk, column j is bit
// (j >> 1) + 16 * (j & 1), i.e. the packed half2 word q = j >> 1 contributes bits q (low half) and 16 + q (high half).
__host__ __device__ __forceinline__ uint32_t relu_mask_bit(uint32_t j) { return (j >> 1) + ((j & 1u) << 4); }

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

}  // namespace tc
}  // namespace nerf
