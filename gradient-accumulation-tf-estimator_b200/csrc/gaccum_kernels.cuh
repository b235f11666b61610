// gaccum_kernels.cuh -- sm_100a kernels of the gradient-accumulation train_op.
//
// All kernels walk a static tile table (<= 2048 elements of one tensor per tile), so the work split --
// and therefore every reduction -- is deterministic.
//
//   accumulate_kernel    a += G                                  optimization.py:81,93    (12 B/elem)
//                        one tile per CTA (hardware block scheduler)
//   apply_kernel         the apply branch WITHOUT clipping (plain Adam of the example scripts, or
//                        clip_norm <= 0): a' = a + G; n = a'/N; Adam; a = 0 in a single pass (36 B/elem).
//   apply_clip_kernel    the apply branch WITH tf.clip_by_global_norm (36 B/elem), optimization.py:80-88,
//                        128-177: see the block comment above its definition.
// Arithmetic uses round-to-nearest intrinsics (__fmul_rn, __fadd_rn, __fdiv_rn, __fsqrt_rn) so nvcc
// cannot contract mul+add into FMA: the reference graph is un-fused, one rounding per TF op, and we
// reproduce it bit for bit (the kernels are HBM-bound, the extra flops are free).
// Measurements and the experiments behind each choice: profiles/r01_tune_sweep.md, profiles/r02_*.md.
#pragma once

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace gaccum {
namespace cg = cooperative_groups;

constexpr int kThreads = 256;                    // 8 warps per CTA / per consumer group
constexpr int kUnroll = 2;                       // 128-bit vectors per thread per stream per tile
constexpr int kTile = kThreads * 4 * kUnroll;    // 2048 elements = 8 KB per stream
constexpr int kSlabAlign = 32;                   // tensors start at multiples of 32 elements (128 B)

// One unit of work: <= kTile consecutive elements of ONE tensor (so pointers and the decay flag
// are tile-uniform).  16 bytes, read with a single LDG.128.
struct __align__(16) TileDesc {
  uint32_t tensor_flags;   // bits 0..30 tensor index, bit 31 = apply weight decay (optimization.py:166)
  uint32_t len;            // elements in this tile (1..kTile)
  uint32_t toff;           // element offset inside the tensor (multiple of kTile)
  uint32_t soff32;         // element offset inside the slabs, in units of 32 elements
};

// Scattered inputs arrive as a pointer table that lives in the kernel-parameter (constant)
// space: no device-side table to keep in sync, launches stay re-entrant and graph-capturable.
// CAP = 0 is the packed layout (grads/params are slabs with the same offsets as accum).
template <int CAP>
struct PtrTable {
  const float* g[CAP];
  float* p[CAP];
};
template <>
struct PtrTable<0> {
  const float* g;
  float* p;
};

struct Scalars {
  float nf;      // fp32(N)                                   optimization.py:83
  float inv_nf;  // 1/N when N is a power of two (exact), else 0 -> the kernels divide
  float lr;      // learning rate of this micro-step          optimization.py:29-54
  float b1, b2;  // fp32(beta)                                optimization.py:151,153
  float omb1;    // A: fp32(1.0 - beta1) from double (:152);  B: 1.0f - fp32(beta1)
  float omb2;
  float eps;     //                                           optimization.py:157
  float wd;      //                                           optimization.py:167
  float clip;    //                                           optimization.py:84
  float alpha;   // B only: lr*sqrt(1-b2^t)/(1-b1^t)          TF1 ApplyAdam
};

template <int CAP>
struct KernelParams {
  const TileDesc* tiles;
  int32_t num_tiles;
  float* accum;
  float* m;
  float* v;
  float* stats;       // gaccum_stats
  unsigned long long* barrier;  // apply_clip_kernel: monotonic arrival counter of the consumers' grid barrier
  struct LaunchCounters* counters;  // apply_clip_kernel: two sets of per-launch counters (tickets, pool length, norm accumulator)
  Scalars sc;
  PtrTable<CAP> tab;
};

// ---------------------------------------------------------------------------------------------
// memory helpers: G is read exactly once -> streaming (evict-first) loads; zeroing the
// accumulator is a streaming store.  a' must survive in L2 from pass 1 to pass 2, so it is
// tagged evict_last while everything that is touched once is tagged evict-first.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ld_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ld_policy(const float4* p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol) : "memory");
  return v;
}
__device__ __forceinline__ void st_policy(float4* p, const float4 v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}

template <int CAP>
__device__ __forceinline__ const float* grad_ptr(const PtrTable<CAP>& tab, const TileDesc& d) {
  if constexpr (CAP == 0) {
    return tab.g ? tab.g + (size_t)d.soff32 * kSlabAlign : nullptr;
  } else {
    const float* b = tab.g[d.tensor_flags & 0x7fffffffu];
    return b ? b + d.toff : nullptr;
  }
}
template <int CAP>
__device__ __forceinline__ float* param_ptr(const PtrTable<CAP>& tab, const TileDesc& d) {
  if constexpr (CAP == 0) {
    return tab.p + (size_t)d.soff32 * kSlabAlign;
  } else {
    return tab.p[d.tensor_flags & 0x7fffffffu] + d.toff;
  }
}
__device__ __forceinline__ bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

// ---------------------------------------------------------------------------------------------
// per-element math, one rounding per reference op
// ---------------------------------------------------------------------------------------------
// optimization.py:83  (1.0*a)/N  -- the multiply by 1.0 is exact.  When N is a power of two, 1/N is
// exact and a * (1/N) is the same correctly rounded real number as a / N (bit-identical, subnormals
// included), which saves a ~12-instruction IEEE division per element; otherwise divide.
__device__ __forceinline__ float normalize(float a, float nf, float inv_nf) {
  return inv_nf != 0.f ? __fmul_rn(a, inv_nf) : __fdiv_rn(a, nf);
}

template <int VARIANT>
__device__ __forceinline__ void adam_elem(float c, float& p, float& m, float& v, bool decay,
                                          const Scalars& sc) {
  if constexpr (VARIANT == 0) {
    // optimization.py:151-171
    const float m2 = __fadd_rn(__fmul_rn(sc.b1, m), __fmul_rn(sc.omb1, c));
    const float v2 = __fadd_rn(__fmul_rn(sc.b2, v), __fmul_rn(sc.omb2, __fmul_rn(c, c)));
    float u = __fdiv_rn(m2, __fadd_rn(__fsqrt_rn(v2), sc.eps));
    if (decay) u = __fadd_rn(u, __fmul_rn(sc.wd, p));
    p = __fsub_rn(p, __fmul_rn(sc.lr, u));
    m = m2;
    v = v2;
  } else {
    // TF1 ApplyAdam: m += (g-m)(1-b1); v += (g*g-v)(1-b2); var -= (m*alpha)/(sqrt(v)+eps)
    const float m2 = __fadd_rn(m, __fmul_rn(__fsub_rn(c, m), sc.omb1));
    const float v2 = __fadd_rn(v, __fmul_rn(__fsub_rn(__fmul_rn(c, c), v), sc.omb2));
    p = __fsub_rn(p, __fdiv_rn(__fmul_rn(m2, sc.alpha), __fadd_rn(__fsqrt_rn(v2), sc.eps)));
    m = m2;
    v = v2;
  }
}

// tf.clip_by_global_norm (TF 1.15): scale = clip * min(1/gn, 1/clip) + (gn - gn)
__device__ __forceinline__ float clip_scale(float gn, float clip) {
  const float inv = __fdiv_rn(1.0f, gn);
  const float invc = __fdiv_rn(1.0f, clip);
  float mn = inv < invc ? inv : invc;
  if (inv != inv) mn = inv;
  return __fadd_rn(__fmul_rn(clip, mn), __fsub_rn(gn, gn));
}

// ---------------------------------------------------------------------------------------------
// accumulate: a += G                                                   optimization.py:81,93
// ---------------------------------------------------------------------------------------------
template <int CAP>
__device__ __forceinline__ void accumulate_tile(const TileDesc d, const KernelParams<CAP>& prm) {
  const float* __restrict__ g = grad_ptr(prm.tab, d);
  if (g == nullptr) return;   // optimization.py:132 -- tensors without a gradient are skipped
  float* __restrict__ a = prm.accum + (size_t)d.soff32 * kSlabAlign;
  const uint32_t len = d.len, tid = threadIdx.x;
  if (aligned16(g)) {
    const uint32_t nvec = len >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* a4 = reinterpret_cast<float4*>(a);
    float4 vg[kUnroll], va[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) { vg[u] = ld_stream(g4 + i); va[u] = a4[i]; }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) {
        va[u].x = __fadd_rn(va[u].x, vg[u].x); va[u].y = __fadd_rn(va[u].y, vg[u].y);
        va[u].z = __fadd_rn(va[u].z, vg[u].z); va[u].w = __fadd_rn(va[u].w, vg[u].w);
        a4[i] = va[u];
      }
    }
    const uint32_t i = (nvec << 2) + tid;      // < 4 trailing elements
    if (i < len) a[i] = __fadd_rn(a[i], ld_stream(g + i));
  } else {
    for (uint32_t i = tid; i < len; i += kThreads) a[i] = __fadd_rn(a[i], ld_stream(g + i));
  }
}

template <int CAP>
__global__ void __launch_bounds__(kThreads)
accumulate_kernel(const __grid_constant__ KernelParams<CAP> prm) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    prm.stats[0] = 0.f; prm.stats[1] = prm.sc.lr; prm.stats[2] = 0.f; prm.stats[3] = 1.f;
  }
  if ((int)blockIdx.x < prm.num_tiles) accumulate_tile(prm.tiles[blockIdx.x], prm);
}

// ---------------------------------------------------------------------------------------------
// apply without clipping: one pass.  HAS_G = false applies the accumulators as they are.
// ---------------------------------------------------------------------------------------------
template <int VARIANT, bool LOAD_G, int CAP>
__device__ __forceinline__ void update_tile(const TileDesc d, const KernelParams<CAP>& prm) {
  const float* __restrict__ g = nullptr;
  if constexpr (LOAD_G) g = grad_ptr(prm.tab, d);
  const size_t soff = (size_t)d.soff32 * kSlabAlign;
  float* __restrict__ a = prm.accum + soff;
  float* __restrict__ m = prm.m + soff;
  float* __restrict__ v = prm.v + soff;
  float* __restrict__ p = param_ptr(prm.tab, d);
  const bool decay = (d.tensor_flags >> 31) != 0;
  const uint32_t len = d.len, tid = threadIdx.x;
  const Scalars& sc = prm.sc;

  // no gradient for this tile: a + 0 would turn -0 into +0 only; the add is skipped entirely
  auto elem = [&](float ax, float gx, bool has_g, float& px, float& mx, float& vx) {
    if (has_g) ax = __fadd_rn(ax, gx);                            // optimization.py:81
    const float c = normalize(ax, sc.nf, sc.inv_nf);              // :83
    adam_elem<VARIANT>(c, px, mx, vx, decay, sc);                 // :85
  };

  if (aligned16(p) && (g == nullptr || aligned16(g))) {
    const uint32_t nvec = len >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* a4 = reinterpret_cast<float4*>(a);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    float4* p4 = reinterpret_cast<float4*>(p);
    float4 va[kUnroll], vg[kUnroll], vp[kUnroll], vm[kUnroll], vv[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) {
        va[u] = __ldcs(a4 + i); vp[u] = __ldcs(p4 + i); vm[u] = __ldcs(m4 + i); vv[u] = __ldcs(v4 + i);
        if (LOAD_G && g) vg[u] = ld_stream(g4 + i);
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) {
        const bool hg = LOAD_G && g;
        elem(va[u].x, vg[u].x, hg, vp[u].x, vm[u].x, vv[u].x); elem(va[u].y, vg[u].y, hg, vp[u].y, vm[u].y, vv[u].y);
        elem(va[u].z, vg[u].z, hg, vp[u].z, vm[u].z, vv[u].z); elem(va[u].w, vg[u].w, hg, vp[u].w, vm[u].w, vv[u].w);
        __stcs(p4 + i, vp[u]); __stcs(m4 + i, vm[u]); __stcs(v4 + i, vv[u]);
        __stcs(a4 + i, make_float4(0.f, 0.f, 0.f, 0.f));   // optimization.py:86-87
      }
    }
    const uint32_t i = (nvec << 2) + tid;
    if (i < len) {
      float px = p[i], mx = m[i], vx = v[i];
      const bool hg = LOAD_G && g;
      elem(a[i], hg ? ld_stream(g + i) : 0.f, hg, px, mx, vx);
      p[i] = px; m[i] = mx; v[i] = vx; a[i] = 0.f;
    }
  } else {
    for (uint32_t i = tid; i < len; i += kThreads) {
      float px = p[i], mx = m[i], vx = v[i];
      const bool hg = LOAD_G && g;
      elem(a[i], hg ? ld_stream(g + i) : 0.f, hg, px, mx, vx);
      p[i] = px; m[i] = mx; v[i] = vx; a[i] = 0.f;
    }
  }
}

template <int VARIANT, bool HAS_G, int CAP>
__global__ void __launch_bounds__(kThreads)
apply_kernel(const __grid_constant__ KernelParams<CAP> prm) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    prm.stats[0] = 1.f; prm.stats[1] = prm.sc.lr; prm.stats[2] = 0.f; prm.stats[3] = 1.f;
  }
  if ((int)blockIdx.x < prm.num_tiles) update_tile<VARIANT, HAS_G>(prm.tiles[blockIdx.x], prm);
}

// =============================================================================================
// apply with clipping: ONE cooperative launch, one CTA per SM =
//     3 consumer groups x 256 threads  +  3 producer warps (one per group)          (864 threads)
//
// NO consumer ever issues a bulk load: every input stream of both passes is moved by TMA
// (cp.async.bulk shared <- global, completing on an mbarrier by byte count) into a per-group ring in
// shared memory, fed by the group's producer warp.  Why (measured, profiles/r02_tune_sweep.md):
//   * an LDG-fed pass can keep only as many bytes in flight as it has registers AND L1 lines to land them
//     in; L1 and shared memory split 256 KB, so every KB of on-chip stash was paid for with bytes in
//     flight (round 1: pass 1 at 4.6 TB/s with 192 KB of stash and 60 KB of L1);
//   * TMA loads need neither registers nor L1: bytes in flight = ring size, descriptors and addresses are
//     computed by the producers ahead of the consumers, whose loop is wait -> LDS -> math -> store.
// NO tile is bound to an SM before it is fetched: with the memory system saturated some SMs get a larger share
// of it than others (with static tiles the first SM finished pass 2 forty microseconds before the last), so the
// producers draw tiles from global atomic ticket counters -- every SM stays busy until the pass is over.
//
// pass 1   tickets over ALL tiles.  ring slot = [G tile | a tile] (16 KB, kP1Slots per group).  a' = a + G;
//          sum((a'/N)^2): thread fp32 per tile -> warp shuffle in fp64 (fixed order) -> EXACT accumulation of the
//          per-warp, per-tile sums in a 2176-bit fixed-point accumulator (integer atomics: associative, so the
//          total does not depend on which SM reduced which tile -- the norm is bit-identical from run to run
//          and across replicas although the schedule is dynamic).  a' of the first kTmemTiles tiles a group
//          processes is parked in Tensor Memory (tcgen05.st: 256 KB per SM that a kernel without MMA leaves
//          idle) and the tile is remembered in shared memory; every other a' goes back in place tagged
//          L2::evict_last.  One flag per tile (plain store) says which of the two happened.
// barrier  only the CONSUMERS rendezvous (named barrier + one atomic per CTA).  The producers do not: p, m, v do
//          not depend on the clip scale, so they start streaming the group's own Tensor-Memory tiles into the
//          ring as soon as pass 1 is drained -- HBM stays busy while the CTAs wait for each other.
// pass 2   ring slot = [p | m | v | a'] (32 KB).  First the group's own Tensor-Memory tiles, then tickets over
//          all tiles, youngest first (a' still in L2), skipping the parked ones: clip, AdamWeightDecay/Adam,
//          STG p, m, v, a = 0.
// Tiles that bulk copies cannot move (gradient / parameter pointer not 16-byte aligned, or shorter than one
// float4) go through the same full/empty protocol with nothing copied and are loaded by the consumers with
// scalar LDGs; producer and consumers evaluate the same predicates (bulk_vecs / bulk_vecs2).
// Per-launch counters (tickets, pool length, accumulator) exist twice; launch k uses set k & 1 and clears the
// other one, k being read off the monotonic barrier counter -- no host-side state, so launches replay in CUDA graphs.
// =============================================================================================
constexpr int kGroups = 3;                        // consumer groups per CTA
constexpr int kConsumerThreads = kThreads * kGroups;        // 768
constexpr int kClipThreads = kConsumerThreads + 32 * kGroups;   // + one producer warp per group = 864
constexpr int kTmemCols = 512;                    // one CTA per SM: take all columns
constexpr int kTmemColsPerWarp = 80;              // 6 warps share a lane quadrant: 6 x 80 = 480 <= 512
constexpr int kTmemTiles = kTmemColsPerWarp / 8;  // 10 tiles per group
constexpr uint32_t kNoTmem = 0xffffffffu;
constexpr int kP1Slots = 2;                       // pass-1 ring slots per group, 16 KB each
constexpr int kP1SlotVecs = 2 * (kTile / 4);      // float4 per pass-1 slot: G | a
constexpr int kP2SlotVecs = 4 * (kTile / 4);      // float4 per pass-2 slot: p | m | v | a'
constexpr int kRingVecs = kP1Slots * kP1SlotVecs; // per group
constexpr int kP2Slots = kRingVecs / kP2SlotVecs; // 2 x 16 KB = 32 KB -> 1 x 32 KB (deeper rings measured slower: r02_tune_sweep.md)
constexpr int kRingBytes = kGroups * kRingVecs * 16;   // dynamic shared memory of the kernel (96 KB)
static_assert(kP2Slots >= 1, "ring must hold at least one [p|m|v|a'] slot");
constexpr int kTicketBatch = 4;                   // pass-1 tickets a producer draws at once while plenty of tiles are left
// what the producer tells the consumers about the tile it put into a slot
struct __align__(16) SlotMeta {
  TileDesc d;          // len == 0: end of the pass
  uint32_t tile;       // index into the tile table
  uint32_t tmem_slot;  // pass 2: a' is parked in this Tensor-Memory slot of the group (kNoTmem: it is in the slot's 4th quarter / in global memory)
  uint32_t pad[2];
};
// exact accumulation of non-negative doubles: 68 bins of 32 payload bits in 64-bit containers cover the whole
// binary64 range (2^-1074 .. 2^1024); a container overflows only after 2^31 additions
constexpr int kAccBins = 68;
struct LaunchCounters {
  unsigned long long p1_ticket, p2_ticket;
  unsigned int nonfinite, pad;                  // nonfinite: bit 0 = +inf seen, bit 1 = NaN seen
  unsigned long long bins[kAccBins];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
// TMA bulk copy global -> shared, completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// ---------------------------------------------------------------------------------------------
// Tensor Memory as a scratchpad.  TMEM (256 KB per SM, 512 columns x 128 lanes x 32 bit) normally
// holds tcgen05.mma accumulators; this kernel has no MMA, so it is idle silicon -- 37 MB across the
// chip.  The CTA allocates all 512 columns (one CTA per SM by construction); every consumer warp parks
// a' values in the 32 lanes it may address (lane quadrant = warp % 4; the 6 warps sharing a quadrant
// take 80 columns each): tcgen05.st 32x32b.x8 writes the thread's 8 words of a tile to 8 consecutive
// columns of its own lane, tcgen05.ld reads them back in pass 2.  A thread only ever reads what it
// wrote itself.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"((uint32_t)kTmemCols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"((uint32_t)kTmemCols) : "memory");
}
__device__ __forceinline__ void tmem_store8(uint32_t taddr, const float4& a, const float4& b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), "r"(__float_as_uint(a.x)), "r"(__float_as_uint(a.y)), "r"(__float_as_uint(a.z)),
                 "r"(__float_as_uint(a.w)), "r"(__float_as_uint(b.x)), "r"(__float_as_uint(b.y)),
                 "r"(__float_as_uint(b.z)), "r"(__float_as_uint(b.w)) : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_load8(uint32_t taddr, float4& a, float4& b) {
  uint32_t r0, r1, r2, r3, r4, r5, r6, r7;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5), "=r"(r6), "=r"(r7) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  a = make_float4(__uint_as_float(r0), __uint_as_float(r1), __uint_as_float(r2), __uint_as_float(r3));
  b = make_float4(__uint_as_float(r4), __uint_as_float(r5), __uint_as_float(r6), __uint_as_float(r7));
}
// TMEM address of this warp's slot for stashed tile `slot` (0..kTmemTiles-1): lane quadrant = warp % 4,
// column block = warp / 4 (0..5 across the three groups)
__device__ __forceinline__ uint32_t tmem_slot_addr(uint32_t base, int slot) {
  const uint32_t warp = threadIdx.x >> 5;
  return base + (((warp & 3u) * 32u) << 16) + (warp >> 2) * kTmemColsPerWarp + (uint32_t)slot * 8u;
}

// Number of float4 vectors of this tile that pass 1 moves by bulk copy (0: scalar fallback).  The producer and
// the consumers MUST agree on this.
__device__ __forceinline__ uint32_t bulk_vecs(const TileDesc& d, const float* g) {
  return (g == nullptr || aligned16(g)) ? (d.len >> 2) : 0u;
}
// ... and that pass 2 moves by bulk copy
__device__ __forceinline__ uint32_t bulk_vecs2(const TileDesc& d, const float* p) {
  return aligned16(p) ? (d.len >> 2) : 0u;
}

// a' of a tile may be parked in Tensor Memory only if BOTH passes take the vector path for it and it is a full tile
template <bool HAS_G, int CAP>
__device__ __forceinline__ bool tmem_ok(const TileDesc& d, const KernelParams<CAP>& prm) {
  bool ok = d.len == (uint32_t)kTile && aligned16(param_ptr(prm.tab, d));
  if constexpr (HAS_G) { const float* g = grad_ptr(prm.tab, d); ok = ok && (g == nullptr || aligned16(g)); }
  return ok;
}

// one thread's view of a ring: slot index + how often the ring has wrapped
struct RingPos {
  int slot = 0;
  uint32_t use = 0;
  __device__ __forceinline__ void advance(int nslots) { if (++slot == nslots) { slot = 0; ++use; } }
};

// ---- exact accumulator ---------------------------------------------------------------------------------------
// add the non-negative double w to `bins` exactly; non-finite values only raise a flag.  `bins` is PRIVATE to the
// calling thread (one accumulator per warp, lane 0 owns it): plain read-modify-write, no atomics, no contention
__device__ __forceinline__ void acc_add(unsigned long long* bins, unsigned int& nonfinite, const double w) {
  const unsigned long long bits = (unsigned long long)__double_as_longlong(w);
  const unsigned int e = (unsigned int)(bits >> 52) & 0x7ffu;
  if (e == 0x7ffu) { nonfinite |= (bits & 0x000fffffffffffffull) ? 2u : 1u; return; }
  unsigned long long mant = bits & 0x000fffffffffffffull;
  if (e != 0) mant |= 1ull << 52;
  if (mant == 0) return;
  const unsigned int pos = e ? e - 1u : 0u;           // bit position of mant's LSB: value = mant * 2^(pos - 1074)
  const unsigned int q = pos >> 5, r = pos & 31u;
  const unsigned long long lo = mant << r;            // r <= 31, mant < 2^53: the 85-bit product is split by hand
  const unsigned long long hi = r ? (mant >> (64u - r)) : 0ull;
  bins[q] += lo & 0xffffffffull;
  bins[q + 1] += lo >> 32;
  bins[q + 2] += hi;
}
// the accumulated value as a double (deterministic: carries are propagated low to high, the three leading 32-bit
// digits are combined in a fixed order; relative error <= 2^-52); executed by one thread
__device__ __forceinline__ double acc_value(const unsigned long long* bins /* kAccBins */, const unsigned int nonfinite) {
  if (nonfinite & 2u) return __longlong_as_double(0x7ff8000000000000ll);
  if (nonfinite & 1u) return __longlong_as_double(0x7ff0000000000000ll);
  unsigned long long carry = 0;
  int top = -1;
  for (int i = 0; i < kAccBins; ++i) {
    const unsigned long long t = bins[i] + carry;
    carry = t >> 32;
    if (t & 0xffffffffull) top = i;
  }
  if (top < 0) return 0.0;
  carry = 0;
  unsigned int g0 = 0, g1 = 0, g2 = 0;                 // digits top-2, top-1, top
  for (int i = 0; i <= top; ++i) {
    const unsigned long long t = bins[i] + carry;
    const unsigned int digit = (unsigned int)(t & 0xffffffffull);
    carry = t >> 32;
    if (i == top - 2) g0 = digit;
    if (i == top - 1) g1 = digit;
    if (i == top) g2 = digit;
  }
  const double m = ((double)g2 * 4294967296.0 + (double)g1) * 4294967296.0 + (double)g0;
  return scalbn(m, 32 * (top - 2) - 1074);
}

// ---- pass 1, consumer side: one tile out of slot [G | a]; returns this THREAD's partial of sum((a'/N)^2) ----
template <bool HAS_G, int CAP>
__device__ __forceinline__ float norm_tile(const TileDesc& d, const KernelParams<CAP>& prm, const float4* slot, uint64_t* empty,
                                           const uint32_t tmem, const uint64_t pol) {
  const float* __restrict__ g = nullptr;
  if constexpr (HAS_G) g = grad_ptr(prm.tab, d);
  float* __restrict__ a = prm.accum + (size_t)d.soff32 * kSlabAlign;
  const uint32_t len = d.len, tid = threadIdx.x & (kThreads - 1);
  const float nf = prm.sc.nf, inv_nf = prm.sc.inv_nf;
  const uint32_t nvec = bulk_vecs(d, g);
  float acc = 0.f;
  if (nvec > 0) {
    float4* a4 = reinterpret_cast<float4*>(a);
    float4 x[kUnroll], gg[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) { x[u] = slot[kTile / 4 + i]; if (g) gg[u] = slot[i]; }
    }
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(empty);        // this warp is done with the slot
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) {
        if (g) {
          x[u].x = __fadd_rn(x[u].x, gg[u].x); x[u].y = __fadd_rn(x[u].y, gg[u].y);
          x[u].z = __fadd_rn(x[u].z, gg[u].z); x[u].w = __fadd_rn(x[u].w, gg[u].w);
          if (tmem == kNoTmem) st_policy(a4 + i, x[u], pol);
        }
        const float nx = normalize(x[u].x, nf, inv_nf), ny = normalize(x[u].y, nf, inv_nf),
                    nz = normalize(x[u].z, nf, inv_nf), nw = normalize(x[u].w, nf, inv_nf);
        acc = fmaf(nx, nx, acc); acc = fmaf(ny, ny, acc); acc = fmaf(nz, nz, acc); acc = fmaf(nw, nw, acc);
      }
    }
    if (tmem != kNoTmem) tmem_store8(tmem, x[0], x[1]);   // full tile: every lane of every warp carries data
    const uint32_t i = (nvec << 2) + tid;      // < 4 tail elements always travel through global memory
    if (i < len) {
      float xs = a[i];
      if (g) { xs = __fadd_rn(xs, ld_stream(g + i)); a[i] = xs; }
      const float n = normalize(xs, nf, inv_nf);
      acc = fmaf(n, n, acc);
    }
  } else {
    // unaligned gradient view, or a tile shorter than one float4: nothing was copied
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(empty);
    for (uint32_t i = tid; i < len; i += kThreads) {
      float xs = a[i];
      if (g) { xs = __fadd_rn(xs, ld_stream(g + i)); a[i] = xs; }
      const float n = normalize(xs, nf, inv_nf);
      acc = fmaf(n, n, acc);
    }
  }
  return acc;
}

// ---- pass 2, consumer side: one tile out of slot [p | m | v | a']; a' from the slot or from Tensor Memory ----
// The caller has waited on the slot's `full` barrier (it had to, to learn which tile this is).
template <int VARIANT, int CAP>
__device__ __forceinline__ void update_tile2(const TileDesc& d, const KernelParams<CAP>& prm, const float s, const float4* slot,
                                             uint64_t* empty, const uint32_t tmem) {
  const size_t soff = (size_t)d.soff32 * kSlabAlign;
  float* __restrict__ a = prm.accum + soff;
  float* __restrict__ m = prm.m + soff;
  float* __restrict__ v = prm.v + soff;
  float* __restrict__ p = param_ptr(prm.tab, d);
  const bool decay = (d.tensor_flags >> 31) != 0;
  const uint32_t len = d.len, tid = threadIdx.x & (kThreads - 1);
  const Scalars& sc = prm.sc;
  auto elem = [&](float ax, float& px, float& mx, float& vx) {
    const float c = __fmul_rn(normalize(ax, sc.nf, sc.inv_nf), s);     // optimization.py:83-84
    adam_elem<VARIANT>(c, px, mx, vx, decay, sc);           // :85
  };
  const uint32_t nvec = bulk_vecs2(d, p);
  if (nvec > 0) {
    float4* a4 = reinterpret_cast<float4*>(a);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    float4* p4 = reinterpret_cast<float4*>(p);
    float4 va[kUnroll], vp[kUnroll], vm[kUnroll], vv[kUnroll];
    if (tmem != kNoTmem) tmem_load8(tmem, va[0], va[1]);
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) {
        vp[u] = slot[i]; vm[u] = slot[kTile / 4 + i]; vv[u] = slot[2 * (kTile / 4) + i];
        if (tmem == kNoTmem) va[u] = slot[3 * (kTile / 4) + i];
      }
    }
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(empty);
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) {
        elem(va[u].x, vp[u].x, vm[u].x, vv[u].x); elem(va[u].y, vp[u].y, vm[u].y, vv[u].y);
        elem(va[u].z, vp[u].z, vm[u].z, vv[u].z); elem(va[u].w, vp[u].w, vm[u].w, vv[u].w);
        __stcs(p4 + i, vp[u]); __stcs(m4 + i, vm[u]); __stcs(v4 + i, vv[u]);
        __stcs(a4 + i, make_float4(0.f, 0.f, 0.f, 0.f));   // optimization.py:86-87
      }
    }
    const uint32_t i = (nvec << 2) + tid;
    if (i < len) {
      float px = p[i], mx = m[i], vx = v[i];
      elem(a[i], px, mx, vx);
      p[i] = px; m[i] = mx; v[i] = vx; a[i] = 0.f;
    }
  } else {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(empty);
    for (uint32_t i = tid; i < len; i += kThreads) {
      float px = p[i], mx = m[i], vx = v[i];
      elem(a[i], px, mx, vx);
      p[i] = px; m[i] = mx; v[i] = vx; a[i] = 0.f;
    }
  }
}

// Dynamic shared memory of apply_clip_kernel: 3 groups x kRingVecs float4 (96 KB).
template <int VARIANT, bool HAS_G, int CAP>
__global__ void __launch_bounds__(kClipThreads, 1)
apply_clip_kernel(const __grid_constant__ KernelParams<CAP> prm) {
  extern __shared__ __align__(128) unsigned char smem_dyn[];
  __shared__ unsigned long long s_bins[kConsumerThreads / 32][kAccBins];   // one exact accumulator per consumer warp (13 KB)
  __shared__ unsigned int s_nonfinite;
  __shared__ float s_bcast[2];
  __shared__ uint32_t s_tmem_base, s_set;
  __shared__ __align__(8) uint64_t s_full1[kGroups][kP1Slots], s_empty1[kGroups][kP1Slots];
  __shared__ __align__(8) uint64_t s_full2[kGroups][kP2Slots], s_empty2[kGroups][kP2Slots];
  __shared__ __align__(8) uint64_t s_go[kGroups];
  __shared__ SlotMeta s_meta1[kGroups][kP1Slots], s_meta2[kGroups][kP2Slots];

  const int warp = (int)threadIdx.x >> 5;
  const bool is_producer = warp >= kConsumerThreads / 32;
  const int grp = is_producer ? warp - kConsumerThreads / 32 : (int)threadIdx.x / kThreads;   // group served / group id
  const int nt = prm.num_tiles, G = (int)gridDim.x * kGroups;
  const int b = (int)blockIdx.x * kGroups + grp;                   // virtual block id
  const int C = b < nt ? (nt - 1 - b) / G + 1 : 0;                 // tiles b, b + G, ... of this group's static share
  const int n_tm = min(kTmemTiles, C);                             // own tiles: a' parked in Tensor Memory
  const int pool_lo = min(nt, kTmemTiles * G);                     // tiles [pool_lo, nt): a' goes back to global memory
  float4* const ring = reinterpret_cast<float4*>(smem_dyn) + (size_t)grp * kRingVecs;
  const uint64_t pol_last = policy_evict_last();

  // ---- set-up: which counter set this launch uses, mbarriers, accumulator, Tensor Memory ---------------------
  if (threadIdx.x == 0) {
    // every CTA that has not yet arrived at this launch's barrier reads a value in [k*grid, (k+1)*grid)
    const unsigned long long k = ld_acquire_gpu_u64(prm.barrier) / gridDim.x;
    s_set = (uint32_t)(k & 1ull);
    s_nonfinite = 0;
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
      for (int sl = 0; sl < kP1Slots; ++sl) { mbar_init(&s_full1[g][sl], 1); mbar_init(&s_empty1[g][sl], kThreads / 32); }
      for (int sl = 0; sl < kP2Slots; ++sl) { mbar_init(&s_full2[g][sl], 1); mbar_init(&s_empty2[g][sl], kThreads / 32); }
      mbar_init(&s_go[g], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  for (int i = threadIdx.x; i < (kConsumerThreads / 32) * kAccBins; i += kClipThreads) (&s_bins[0][0])[i] = 0ull;
  if (warp == 1) tmem_alloc(&s_tmem_base);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = s_tmem_base;
  LaunchCounters* const ctr = prm.counters + s_set;
  if (blockIdx.x == 0 && threadIdx.x >= 64 && threadIdx.x < 64 + (int)(sizeof(LaunchCounters) / 8)) {
    // the other set was used by the previous launch on this plan, which is complete: clear it for the next one
    reinterpret_cast<unsigned long long*>(prm.counters + (s_set ^ 1u))[threadIdx.x - 64] = 0ull;
  }

  if (is_producer) {
    // =========================== producer warp of group `grp` ===========================
    const int lane = (int)threadIdx.x & 31;
    const uint64_t pol_first = policy_evict_first();
    // ---- pass 1.  First the group's OWN tiles b + j*G, j < n_tm: their a' is parked in this SM's Tensor Memory, so
    //      they are bound to it in both passes.  Then the rest of the model, tiles [pool_lo, nt), in whatever order the
    //      global ticket counter hands them out -- kTicketBatch tickets at a time while plenty are left (one atomic per
    //      lane, the descriptor loads of a batch overlap), single tickets near the end so that no SM is left holding a
    //      batch ----
    {
      RingPos rp;
      auto issue = [&](const TileDesc& dl, const uint32_t tile) {          // lane 0 only
        const float* g = nullptr;
        if constexpr (HAS_G) g = grad_ptr(prm.tab, dl);
        const uint32_t nvec = bulk_vecs(dl, g);
        uint64_t* full = &s_full1[grp][rp.slot];
        mbar_wait(&s_empty1[grp][rp.slot], rp.use & 1u);             // the consumers have released the slot
        SlotMeta* meta = &s_meta1[grp][rp.slot];
        meta->d = dl;
        meta->tile = tile;
        if (nvec > 0) {
          float4* dst = ring + (size_t)rp.slot * kP1SlotVecs;
          mbar_arrive_expect_tx(full, nvec * 16u * (g ? 2u : 1u));
          if (g) bulk_g2s(dst, g, nvec * 16u, full, pol_first);
          bulk_g2s(dst + kTile / 4, prm.accum + (size_t)dl.soff32 * kSlabAlign, nvec * 16u, full, pol_first);
        } else {
          mbar_arrive(full);                                                 // nothing to copy: complete the phase
        }
      };
      auto shuffled = [&](const TileDesc& d, int l) {
        TileDesc dl;
        dl.tensor_flags = __shfl_sync(0xffffffffu, d.tensor_flags, l);
        dl.len = __shfl_sync(0xffffffffu, d.len, l);
        dl.toff = __shfl_sync(0xffffffffu, d.toff, l);
        dl.soff32 = __shfl_sync(0xffffffffu, d.soff32, l);
        return dl;
      };
      {
        static_assert(kTmemTiles <= 32, "one descriptor per lane");
        TileDesc d{};
        if (lane < n_tm) d = prm.tiles[b + lane * G];
        for (int l = 0; l < n_tm; ++l) {
          const TileDesc dl = shuffled(d, l);
          if (lane == 0) issue(dl, (uint32_t)(b + l * G));
          rp.advance(kP1Slots);
        }
      }
      bool done = false;
      long long last = pool_lo;
      while (!done) {
        const long long left = (long long)nt - last;
        const int batch = left > 8ll * G ? kTicketBatch : (left > 2ll * G ? 2 : 1);
        long long tile = nt;
        TileDesc d{};
        if (lane < batch) {
          tile = (long long)pool_lo + (long long)atomicAdd(&ctr->p1_ticket, 1ull);
          if (tile < nt) d = prm.tiles[tile];
        }
        for (int l = 0; l < batch; ++l) {
          const long long tl = __shfl_sync(0xffffffffu, tile, l);
          if (tl >= nt) { done = true; continue; }       // lanes get their tickets in no particular order: a valid one may follow
          last = tl;
          const TileDesc dl = shuffled(d, l);
          if (lane == 0) issue(dl, (uint32_t)tl);
          rp.advance(kP1Slots);
        }
      }
      if (lane == 0) {
        // end marker, then drain: pass 2's slots overlay pass 1's, so every slot must have been released for the last time
        mbar_wait(&s_empty1[grp][rp.slot], rp.use & 1u);
        s_meta1[grp][rp.slot].d.len = 0;
        mbar_arrive(&s_full1[grp][rp.slot]);
        for (int sl = 0; sl < kP1Slots; ++sl) {
          if (sl == rp.slot) continue;
          const uint32_t n = rp.use + (sl < rp.slot ? 1u : 0u);              // times slot sl was armed
          if (n > 0) mbar_wait(&s_empty1[grp][sl], n & 1u);
        }
      }
      __syncwarp();
    }
    // ---- pass 2.  First the group's own Tensor-Memory tiles (their a' cannot move; their p, m, v do not depend on
    //      the clip scale, so these copies start BEFORE the grid barrier and HBM stays busy while the CTAs wait for
    //      each other).  Then tickets over the pool of L2-resident tiles, youngest first.  Pool tiles carry their a'
    //      in the slot's 4th quarter; they may only be fetched once every CTA has passed the barrier. ----
    if (lane == 0) {
      RingPos rp;
      int jb = 0;
      bool past_barrier = false;
      const unsigned long long pool_n = (unsigned long long)max(0, nt - pool_lo);
      while (true) {
        int tile;
        uint32_t tmem_slot = kNoTmem;
        if (jb < n_tm) {
          tile = b + jb * G;
          tmem_slot = (uint32_t)jb;
          ++jb;
        } else {
          if (!past_barrier) {
            mbar_wait(&s_go[grp], 0);                                           // the consumers are through the grid barrier
            asm volatile("fence.proxy.async;" ::: "memory");                    // generic-proxy a' stores -> our bulk reads
            past_barrier = true;
          }
          const unsigned long long tk = atomicAdd(&ctr->p2_ticket, 1ull);
          if (tk >= pool_n) break;
          tile = nt - 1 - (int)tk;                                              // youngest a' lines first
        }
        const TileDesc d = prm.tiles[tile];
        const float* p = param_ptr(prm.tab, d);
        const uint32_t nvec = bulk_vecs2(d, p);
        const bool in_tmem = tmem_slot != kNoTmem && tmem_ok<HAS_G>(d, prm);
        if (!in_tmem && !past_barrier) {                                        // an own tile whose a' had to go to global memory
          mbar_wait(&s_go[grp], 0);
          asm volatile("fence.proxy.async;" ::: "memory");
          past_barrier = true;
        }
        uint64_t* full = &s_full2[grp][rp.slot];
        mbar_wait(&s_empty2[grp][rp.slot], rp.use & 1u);
        SlotMeta* meta = &s_meta2[grp][rp.slot];
        meta->d = d;
        meta->tmem_slot = in_tmem ? tmem_slot : kNoTmem;
        if (nvec > 0) {
          const size_t soff = (size_t)d.soff32 * kSlabAlign;
          float4* dst = ring + (size_t)rp.slot * kP2SlotVecs;
          mbar_arrive_expect_tx(full, nvec * 16u * (in_tmem ? 3u : 4u));
          bulk_g2s(dst, p, nvec * 16u, full, pol_first);
          bulk_g2s(dst + kTile / 4, prm.m + soff, nvec * 16u, full, pol_first);
          bulk_g2s(dst + 2 * (kTile / 4), prm.v + soff, nvec * 16u, full, pol_first);
          if (!in_tmem) bulk_g2s(dst + 3 * (kTile / 4), prm.accum + soff, nvec * 16u, full, pol_first);
        } else {
          mbar_arrive(full);
        }
        rp.advance(kP2Slots);
      }
      mbar_wait(&s_empty2[grp][rp.slot], rp.use & 1u);                   // end marker
      s_meta2[grp][rp.slot].d.len = 0;
      mbar_arrive(&s_full2[grp][rp.slot]);
    }
    __syncwarp();
  } else {
    // =========================== consumer group ===========================
    const bool leader = (threadIdx.x & (kThreads - 1)) == 0;
    // every slot starts out empty: the consumers say so (phase 0 of each `empty` barrier), so that the producer's very
    // first wait is an ordinary wait on a phase that completes -- use u of a slot waits for phase u
    if ((threadIdx.x & 31) == 0) {
      for (int sl = 0; sl < kP1Slots; ++sl) mbar_arrive(&s_empty1[grp][sl]);
      for (int sl = 0; sl < kP2Slots; ++sl) mbar_arrive(&s_empty2[grp][sl]);
    }
    // ---- pass 1: whatever tiles the producer hands over, until its end marker ----
    unsigned int my_nonfinite = 0;
    {
      RingPos rp;
      int n_seen = 0;
      while (true) {
        mbar_wait(&s_full1[grp][rp.slot], rp.use & 1u);
        const SlotMeta meta = s_meta1[grp][rp.slot];
        if (meta.d.len == 0) break;
        // Tensor Memory takes the group's own tiles j < n_tm (the first ones it is handed) when they are FULL,
        // vector-path tiles (tcgen05.st/ld are warp-collective)
        const bool own = n_seen < n_tm;
        const bool park = own && tmem_ok<HAS_G>(meta.d, prm);
        const uint32_t tm = park ? tmem_slot_addr(tmem_base, n_seen) : kNoTmem;
        const float part = norm_tile<HAS_G>(meta.d, prm, ring + (size_t)rp.slot * kP1SlotVecs, &s_empty1[grp][rp.slot], tm, pol_last);
        // warp total in fp64, fixed butterfly order; lane 0 adds it EXACTLY into its warp's accumulator
        double w = (double)part;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
        if ((threadIdx.x & 31) == 0) acc_add(s_bins[warp], my_nonfinite, w);
        ++n_seen;
        rp.advance(kP1Slots);
      }
    }
    named_bar_sync(1, kConsumerThreads);                     // every consumer thread of this CTA is through pass 1
    // flush this CTA's accumulators into the launch's global one (integer adds: order does not matter)
    if (my_nonfinite) atomicOr(&s_nonfinite, my_nonfinite);
    if (threadIdx.x < kAccBins) {
      unsigned long long v = 0;
      for (int w = 0; w < kConsumerThreads / 32; ++w) v += s_bins[w][threadIdx.x];
      if (v) atomicAdd(&ctr->bins[threadIdx.x], v);
    }
    named_bar_sync(1, kConsumerThreads);
    if (threadIdx.x == 0 && s_nonfinite) atomicOr(&ctr->nonfinite, s_nonfinite);
    // ---- grid barrier of the consumers: one atomic per CTA on a monotonic counter (every launch of this plan
    //      uses the same grid, so the counter advances by gridDim.x per launch); cooperative launch guarantees
    //      that all CTAs are co-resident ----
    if (threadIdx.x == 0) {
      __threadfence();
      const unsigned long long old = atomicAdd(prm.barrier, 1ull);
      const unsigned long long target = (old / gridDim.x + 1ull) * gridDim.x;
      while (ld_acquire_gpu_u64(prm.barrier) < target) { __nanosleep(20); }
    }
    named_bar_sync(1, kConsumerThreads);
    if (leader) mbar_arrive(&s_go[grp]);                     // this group's producer may now fetch pool tiles
    // ---- every CTA evaluates the same exact sum the same way: bit-identical gn and clip scale everywhere ----
    if (threadIdx.x < kAccBins) s_bins[0][threadIdx.x] = __ldcg(&ctr->bins[threadIdx.x]);
    named_bar_sync(1, kConsumerThreads);
    if (threadIdx.x == 0) {
      const double tot = acc_value(s_bins[0], __ldcg(&ctr->nonfinite));
      const float g_norm = __fsqrt_rn((float)tot);          // tf.linalg.global_norm
      s_bcast[0] = clip_scale(g_norm, prm.sc.clip);
      s_bcast[1] = g_norm;
    }
    named_bar_sync(1, kConsumerThreads);
    const float s = s_bcast[0];
    // ---- pass 2: whatever tiles the producer hands over, until its end marker ----
    {
      RingPos rp;
      while (true) {
        mbar_wait(&s_full2[grp][rp.slot], rp.use & 1u);
        const SlotMeta meta = s_meta2[grp][rp.slot];
        if (meta.d.len == 0) break;
        const uint32_t tm = meta.tmem_slot != kNoTmem ? tmem_slot_addr(tmem_base, (int)meta.tmem_slot) : kNoTmem;
        update_tile2<VARIANT>(meta.d, prm, s, ring + (size_t)rp.slot * kP2SlotVecs, &s_empty2[grp][rp.slot], tm);
        rp.advance(kP2Slots);
      }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      prm.stats[0] = 1.f; prm.stats[1] = prm.sc.lr; prm.stats[2] = s_bcast[1]; prm.stats[3] = s;
    }
  }
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base);
}

}  // namespace gaccum
