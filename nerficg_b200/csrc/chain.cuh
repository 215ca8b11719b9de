// chain.cuh -- the skeleton shared by the two MLP chain kernels, mlp_fwd_kernel (K3, mlp_fwd.cu) and mlp_dgrad_kernel
// (K4a, mlp_bwd.cu): barrier map, set-up / teardown, persistent schedule, the three weight-ring roles and the epilogue
// helpers.  Each kernel supplies its stage table, its weight panels, the A operand of each MMA and its epilogue.
//
// Two CTAs on the two SMs of a TPC form a cluster and work as a cta_group::2 PAIR: each CTA owns 128 samples of a
// 256-sample "group" per slot, and walks two groups ("slots" 0/1) through the whole chain of stages without touching HBM
// in between:
//   warp 0      weight producer (producer()): streams THIS CTA's HALF of every fp16 weight panel (pre-swizzled UMMA
//               images, 128 of the 256 rows) from L2 into a shared-memory ring with 1-D bulk copies + mbarriers
//   warp 1      leader CTA: MMA issuer (issuer()) -- the warp runs the loop uniformly and ONE elected lane issues
//               tcgen05.mma.cta_group::2 (M=256, K=16): rows 0..127 from its own A operand panels and TMEM, rows
//               128..255 from the peer's, B = the two CTAs' ring stages (one half each), so a weight byte is fetched
//               once per 256 samples; completion is multicast to both CTAs' barriers.
//               peer CTA: relay (relay()) -- forwards "my half of ring stage s has landed" to the leader's barrier.
//               accumulators live in TMEM (2 slots x 256 fp32 columns = all 512 columns, in each CTA)
//   warp 2      TMEM allocator
//   warps 4-11  epilogue of slot 0 \  tcgen05.ld accumulator -> the kernel's arithmetic -> fp16 -> swizzled A operand
//   warps 12-19 epilogue of slot 1 /  panels of the next stage (in place); the two slots ping-pong so one slot's
//               epilogue overlaps the other slot's MMAs.  Each slot has EIGHT warps: warp w owns TMEM lane quarter
//               w % 4 (hardware rule) and column half (w / 4) % 2, so two warps per scheduler work on one accumulator.
//               Measured with four warps per slot: the serial loop MMA (2 K cycles) -> epilogue (4 K cycles, one
//               latency-bound warp per scheduler) -> MMA left the tensor pipe idle half of the time.
//
// Measured lessons baked into the structure (DESIGN.md "K3"):
//   * one CTA per tile pair was weight-starved: 128 KB of weights per 128 samples and layer is 64 B/cycle/SM at tensor
//     peak (18 TB/s chip-wide) and the MMA issuer spent 24-40 % of its time waiting for ring stages; the CTA pair halves
//     both the L2 -> SM stream and the shared-memory reads of B;
//   * the issuing warp must stay warp-uniform with elect.sync around the tcgen05 instructions: issued under
//     `if (lane == 0)` every MMA was wrapped in a compiler-generated ELECT/BRA.U.ANY waterfall and cost ~190 cycles of
//     issue for 64 cycles of tensor work.
//
// A kernel describes its chain with a stage policy C:
//   C::kStages        chain stages per tile
//   C::kRingStages    depth of the weight ring (16 KB stages)
//   C::kProfBase      first of the kernel's ten stall-counter slots
//   C::panels(st)     K panels of stage st, one ring stage each
//   C::shared(st)     slot 1 re-uses the ring stages slot 0 loaded for stage st.  The two slots of a CTA walk the chain
//                     one stage apart, so the weight panels of stage st are needed by slot 0 and, one accumulator later,
//                     by slot 1: they are loaded ONCE and slot 1's MMAs release the ring stages (half the L2 -> SM weight
//                     stream).  Only a stage whose panels all fit in the ring can be shared (slot 0 holds them until
//                     slot 1 is done).
//
// Stall counters (common.cuh NERF_TIMED, tools/kernel_timing.py): the roles add to the timing buffer `prof` from the
// kernel's counter base C::kProfBase on (forward 0, dgrad 10): issuer +0 A-ready wait, +1 W-full wait, +2 total, +9 CTA
// count; producer +3 W-empty wait, +4 total; epilogue (one thread of slot 0) +5 ACC-ready wait, +6 total, +7 image-store
// drain, +8 prologue.
#pragma once
#include "common.cuh"
#include "mlp_layout.cuh"
#include "tc.cuh"

namespace nerf {
namespace chain {
using namespace tc;

constexpr int kEpiThreadsPerSlot = 256;  // 8 warps: 4 TMEM lane quarters x 2 column halves
constexpr int kThreads = 128 + 2 * kEpiThreadsPerSlot;
constexpr int kRegsEpilogue = 112, kRegsOther = 32;
// setmaxnreg moves registers inside the CTA's OWN allocation (launch: 640 threads x 96): what the 128 producer / MMA threads
// release (96 - 32 each = 8192) must cover what the 512 epilogue threads request (112 - 96 each = 8192), or the
// increase blocks forever
constexpr uint32_t kRingStageBytes = kPanelBytes128;  // one K panel (64 inputs) x this CTA's 128 of the panel's 256 rows

// barrier map at `base` (8 bytes per barrier), followed by the TMEM base address
struct Bars {
  int ring_stages;
  bool with_bias;
  uint32_t w_full;     // [ring_stages] this CTA's half of the ring stage has landed
  uint32_t w_empty;    // [ring_stages] the MMAs reading the ring stage have completed (multicast commit)
  uint32_t w_peer;     // [ring_stages] leader only: the peer's half of the ring stage has landed
  uint32_t a_ready;    // [2] leader only: operands of BOTH CTAs written + accumulators drained
  uint32_t acc_ready;  // [2] accumulator complete (multicast commit)
  uint32_t bias;       // [2] with_bias (forward): the slot's bias vector of the next stage has landed
  uint32_t tmem_slot;  // uint32: TMEM base address
  __device__ Bars(uint32_t base, int ring_stages_, bool with_bias_)
      : ring_stages(ring_stages_), with_bias(with_bias_), w_full(base), w_empty(base + 8 * ring_stages_),
        w_peer(base + 16 * ring_stages_), a_ready(base + 24 * ring_stages_), acc_ready(a_ready + 16), bias(acc_ready + 16),
        tmem_slot(bias + (with_bias_ ? 16 : 0)) {}
};

// Every thread: barrier init, TMEM allocation (all 512 columns, cta_group::2) and the cluster sync that orders both before
// any remote arrive / multicast commit.  Returns the TMEM base address.
__device__ __forceinline__ uint32_t setup(const Bars& b, int warp) {
  if (threadIdx.x == 0) {
    for (int i = 0; i < b.ring_stages; ++i) {
      mbar_init(b.w_full + 8 * i, 1);
      mbar_init(b.w_empty + 8 * i, 1);
      mbar_init(b.w_peer + 8 * i, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(b.a_ready + 8 * s, 16);  // one arrival per epilogue warp of either CTA
      mbar_init(b.acc_ready + 8 * s, 1);
      if (b.with_bias) mbar_init(b.bias + 8 * s, 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc2(b.tmem_slot, 512);
    tmem_relinquish2();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(b.tmem_slot));
  return tmem_base;
}

__device__ __forceinline__ void teardown(uint32_t tmem_base, int warp) {
  tc_fence_before();
  cluster_sync_all();  // the peer may still be reading this CTA's shared memory / arriving on its barriers
  if (warp == 2) tmem_dealloc2(tmem_base, 512);
}

// Persistent schedule: group = 256 samples = one tile per CTA of the pair; a cluster handles two groups (slots) per
// iteration.  Identical in both CTAs.
struct Schedule {
  int n_clusters, cluster_id, n_groups, n_iters;
  __device__ explicit Schedule(int n_tiles)
      : n_clusters((int)gridDim.x / 2), cluster_id((int)blockIdx.x / 2), n_groups((n_tiles + 1) / 2),
        n_iters(((n_groups + 1) / 2 + n_clusters - 1) / n_clusters) {}
  __device__ int group_of(int it, int slot) const { return (it * n_clusters + cluster_id) * 2 + slot; }
  __device__ bool active(int it, int slot) const { return group_of(it, slot) < n_groups; }
  // this CTA's tile; the last group may have none for the peer (tile >= n_tiles): it still takes part in the MMAs
  __device__ int tile(int it, int slot, uint32_t rank) const { return group_of(it, slot) * 2 + (int)rank; }
};

// host: clusters for `n_tiles` tiles, at most one per TPC (one cluster iteration = 2 slots x 2 tiles)
inline int grid(int n_tiles) {
  const int group_pairs = ((n_tiles + 1) / 2 + 1) / 2;
  return 2 * (group_pairs < kNumSMs / 2 ? group_pairs : kNumSMs / 2);
}

// position in the weight ring; the parity flips each time the ring wraps
template <int kDepth>
struct RingCursor {
  uint32_t stage = 0, phase = 0;
  __device__ void next() {
    if (++stage == kDepth) {
      stage = 0;
      phase ^= 1;
    }
  }
};

// THIS CTA's half of one weight panel: global source and byte count
struct Panel {
  const void* src;
  uint32_t bytes;
};

// `ring` is the shared::cta address of ring stage 0.  Both kernels compute it in the argument list: computed once above
// the role branch, it made ptxas move dgrad's schedule out of uniform registers and spill 24 more bytes.
//
// warp 0: one ring stage per K panel.  panel(st, pp) gives this CTA's half of panel pp of stage st (the cta_group::2 MMA
// takes the other half from the peer's ring).
template <class C, class PanelFn>
__device__ __forceinline__ void producer(const Schedule& sch, const Bars& b, uint32_t ring, bool prof_on, unsigned long long* prof,
                                         PanelFn panel) {
  RingCursor<C::kRingStages> r;
  const uint64_t keep = l2_evict_last();
  long long t_wait = 0;
  const long long t_begin = prof_on ? clock64() : 0;
  for (int it = 0; it < sch.n_iters; ++it) {
    for (int st = 0; st < C::kStages; ++st) {
      for (int slot = 0; slot < 2; ++slot) {
        if (!sch.active(it, slot)) continue;
        if (slot == 1 && C::shared(st)) continue;  // slot 1 re-uses the panels loaded for slot 0
        const int np = C::panels(st);
#pragma unroll 1  // unrolled, the loop added ~280 instructions to every forward instantiation for no gain in a 32-register warp
        for (int pp = 0; pp < np; ++pp) {
          NERF_TIMED(prof_on, t_wait, mbar_wait(b.w_empty + 8 * r.stage, r.phase ^ 1));
          if (elect_one()) {
            const Panel w = panel(st, pp);
            mbar_arrive_expect_tx(b.w_full + 8 * r.stage, w.bytes);
            bulk_g2s_hint(ring + r.stage * kRingStageBytes, w.src, w.bytes, b.w_full + 8 * r.stage, keep);
          }
          __syncwarp();
          r.next();
        }
      }
    }
  }
  if (prof_on && (threadIdx.x & 31) == 0) {
    atomicAdd(prof + C::kProfBase + 3, (unsigned long long)t_wait);
    atomicAdd(prof + C::kProfBase + 4, (unsigned long long)(clock64() - t_begin));
  }
}

// warp 1 of the leader CTA.  mma(st, slot, pp, d_tmem, db) issues the MMAs of panel pp (one elected lane): A operand,
// instruction descriptor and K steps; db is the descriptor of the ring stage that holds the panel.
template <class C, class MmaFn>
__device__ __forceinline__ void issuer(const Schedule& sch, const Bars& b, uint32_t ring, uint32_t tmem_base, bool prof_on,
                                       unsigned long long* prof, MmaFn mma) {
  RingCursor<C::kRingStages> r;
  uint32_t a_phase[2] = {0, 0};
  long long t_a = 0, t_w = 0;
  const long long t_begin = prof_on ? clock64() : 0;
  for (int it = 0; it < sch.n_iters; ++it) {
    for (int st = 0; st < C::kStages; ++st) {
      const bool sh = C::shared(st);
      const bool both = sch.active(it, 1);
      const RingCursor<C::kRingStages> r0 = r;
      for (int slot = 0; slot < 2; ++slot) {
        if (!sch.active(it, slot)) continue;
        if (sh && slot == 1) r = r0;  // replay the ring stages slot 0 has just used (their barriers are still in the same phase)
        const bool release = !sh || slot == 1 || !both;
        const uint32_t d_tmem = tmem_base + slot * 256;
        NERF_TIMED(prof_on, t_a, mbar_wait_cluster(b.a_ready + 8 * slot, a_phase[slot]));
        a_phase[slot] ^= 1;
        tc_fence_after();
        const int np = C::panels(st);
        for (int pp = 0; pp < np; ++pp) {
          NERF_TIMED(prof_on, t_w, mbar_wait(b.w_full + 8 * r.stage, r.phase));
          NERF_TIMED(prof_on, t_w, mbar_wait_cluster(b.w_peer + 8 * r.stage, r.phase));
          tc_fence_after();
          if (elect_one()) {
            mma(st, slot, pp, d_tmem, make_smem_desc(ring + r.stage * kRingStageBytes, 16u, kAtomBytes));
            if (release) umma_commit2(b.w_empty + 8 * r.stage, 3);
            if (pp == np - 1) umma_commit2(b.acc_ready + 8 * slot, 3);
          }
          __syncwarp();
          r.next();
        }
      }
    }
  }
  if (prof_on && (threadIdx.x & 31) == 0) {
    atomicAdd(prof + C::kProfBase + 0, (unsigned long long)t_a);
    atomicAdd(prof + C::kProfBase + 1, (unsigned long long)t_w);
    atomicAdd(prof + C::kProfBase + 2, (unsigned long long)(clock64() - t_begin));
    atomicAdd(prof + C::kProfBase + 9, 1ull);
  }
}

// warp 1 of the peer CTA: tells the leader's issuer that this CTA's half of ring stage s has landed (bulk copies can only
// signal a barrier of their own CTA, and mbarriers cannot be waited on remotely)
template <class C>
__device__ __forceinline__ void relay(const Schedule& sch, const Bars& b) {
  RingCursor<C::kRingStages> r;
  for (int it = 0; it < sch.n_iters; ++it)
    for (int st = 0; st < C::kStages; ++st)
      for (int slot = 0; slot < 2; ++slot) {
        if (!sch.active(it, slot)) continue;
        if (slot == 1 && C::shared(st)) continue;
        const int np = C::panels(st);
        for (int pp = 0; pp < np; ++pp) {
          mbar_wait(b.w_full + 8 * r.stage, r.phase);
          if (elect_one()) mbar_arrive_cluster(mapa(b.w_peer + 8 * r.stage, 0));
          __syncwarp();
          r.next();
        }
      }
}

// Geometry of an epilogue thread (warps 4..19) and the steps every epilogue repeats.
struct Epilogue {
  int lane, slot;
  int half;                 // column half of the accumulator owned by this warp
  int row;                  // row of the tile; the thread of the other half has the same row
  int tg;                   // 0..255 within the slot
  uint32_t act;             // the slot's A operand panels
  uint32_t t_slot;          // TMEM: the slot's accumulator, this warp's lane quarter
  uint32_t row_off;         // this row in a panel
  uint32_t xr;              // swizzle term of this row: 16-byte chunk ch lives at ((ch << 4) ^ xr)
  uint32_t act_h;           // this row in the first of this half's two act panels
  uint32_t bar_id;          // named barrier of this slot's eight warps
  uint32_t a_ready_leader;  // both CTAs announce their operands to the leader
  __device__ Epilogue(int warp, int lane_, uint32_t smem_base, uint32_t slot_bytes, uint32_t tmem_base, const Bars& b) {
    const int ew = warp - 4;  // 0..15
    const int wq = warp & 3;  // TMEM lane quarter of this warp (hardware: warp id % 4)
    lane = lane_;
    slot = ew >> 3;
    half = (ew >> 2) & 1;
    row = wq * 32 + lane;
    tg = threadIdx.x - 128 - slot * kEpiThreadsPerSlot;
    act = smem_base + slot * slot_bytes;
    t_slot = tmem_base + slot * 256 + (static_cast<uint32_t>(wq * 32) << 16);
    bar_id = 1 + slot;
    row_off = (uint32_t)(row >> 3) * kAtomBytes + (uint32_t)(row & 7) * kPanelRowBytes;
    xr = (uint32_t)(row & 7) << 4;
    // opaque to the optimiser: otherwise ptxas re-derives these from %cluster_ctaid / %tid inside every chunk
    // (S2UR + 10 dependent integer ops on the critical path of the operand stores)
    asm volatile("" : "+r"(act), "+r"(t_slot), "+r"(row_off), "+r"(xr));
    act_h = act + 2 * half * kPanelBytes128 + row_off;
    a_ready_leader = mapa(b.a_ready + 8 * slot, 0);
  }

  __device__ __forceinline__ void sync() const { named_bar_sync(bar_id, kEpiThreadsPerSlot); }

  // hands this warp's operands to the MMA issuer: one (possibly remote) arrival per warp, because per-thread remote
  // arrivals serialise on the leader's barrier
  __device__ __forceinline__ void hand_off() const {
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive_cluster(a_ready_leader);
  }

  // one thread bulk-stores an image from shared memory to dst() (evaluated by that thread only); call after the slot's
  // warps fenced their writes and met
  template <class DstFn>
  __device__ __forceinline__ void image_issue(DstFn dst, uint32_t src, uint32_t bytes, bool tile_ok) const {
    if (tg == 0 && tile_ok) {
      bulk_s2g_hint(dst(), src, bytes, l2_evict_first());
      bulk_commit();
    }
  }
  template <class DstFn>
  __device__ __forceinline__ void image_store(DstFn dst, uint32_t src, uint32_t bytes, bool tile_ok) const {
    fence_proxy_async_smem();
    sync();
    image_issue(dst, src, bytes, tile_ok);
  }
  // before overwriting a buffer that may still be read by an in-flight image store
  __device__ __forceinline__ void image_drain(bool prof, long long& t_drain) const {
    const long long t0 = prof ? clock64() : 0;
    if (tg == 0) bulk_wait_read<0>();
    sync();
    if (prof) t_drain += clock64() - t0;
  }
};

// the epilogue's counters (+5..+8, see the top of this file)
template <class C>
__device__ __forceinline__ void epilogue_counters(unsigned long long* prof, long long t_accw, long long t_begin, long long t_drain,
                                                  long long t_pro) {
  atomicAdd(prof + C::kProfBase + 5, (unsigned long long)t_accw);
  atomicAdd(prof + C::kProfBase + 6, (unsigned long long)(clock64() - t_begin));
  atomicAdd(prof + C::kProfBase + 7, (unsigned long long)t_drain);
  atomicAdd(prof + C::kProfBase + 8, (unsigned long long)t_pro);
}

template <bool kV>
struct BoolTag {
  static constexpr bool value = kV;
};

}  // namespace chain
}  // namespace nerf
