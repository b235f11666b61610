// gaccum_dp.cuh -- the data-parallel apply step as ONE kernel over NVLink peer memory.
//
// Replaces what reference distributedExample/04 does with MultiWorkerMirroredStrategy:
// per-variable all-reduces on EVERY micro-step (04:55,58,70) followed by a replicated
// apply (04:59-66).  Here every rank accumulates locally for the whole window and the exchange
// happens once, inside the apply kernel.  Rank r OWNS the contiguous tile range
// [bounds[r], bounds[r+1]) (equal element counts); m and v are only ever touched by their owner
// (ZeRO-1 style).  The kernel is PUSH based -- remote STORES are fire-and-forget, remote loads would
// have to cover ~2-3 us of NVLink latency with registers:
//
//   phase A   every tile of the model: x = a + G (the window's last local accumulate, folded in:
//             optimization.py:81).  Owned tile: a <- x.  Foreign tile: x is STORED INTO THE OWNER'S
//             STAGING AREA over NVLink (slot = source rank) and the local accumulator is zeroed
//             (optimization.py:86-87).  Each rank starts its sweep at its right-hand neighbour's shard, so
//             at any moment every owner receives from about one source.        == reduce-scatter, push
//   flag 0    "all my pushes have landed" (block-completion counter -> system-scope release flags)
//   (tiles of every phase are handed to the blocks by atomic tickets: the blocks finish together)
//   phase B   owned tiles: a' = sum over ranks 0..W-1 of their contribution (own: a, others: staging),
//             FIXED rank order => deterministic; a <- a'; partial sum((a'/N)^2)
//   flag 1    per-rank partial norms travel with the flag; every rank adds the W partials in rank
//             order => bit-identical gn and clip scale everywhere
//   phase C   clip + AdamWeightDecay/Adam on the owned tiles, a <- 0, and the new parameters are STORED
//             INTO EVERY RANK'S PARAMETER SLAB over NVLink                       == all-gather, push
//   flag 2    all peers' parameter stores into my slab have landed before this kernel completes
//   (a flag wait longer than 60 s means a dead peer: the kernel traps instead of hanging the GPU)
//
// NVLink bytes per rank and direction: 2 * (W-1)/W * 4P (the all-reduce lower bound); the update's HBM
// bytes shrink to 1/W.  There is no grid-wide barrier: a phase ends when the last block of a rank bumps a
// completion counter and raises that rank's flag in every control block; every block polls its own rank's
// control block (local memory).  All blocks must be co-resident (cooperative launch guarantees it).
// Parameters must live in one packed, peer-mapped slab (plan offsets); the host side (PyTorch symmetric
// memory, NVSHMEM, cuMem IPC, ...) only supplies the W base pointers of the parameter slabs, staging areas
// and control blocks.
#pragma once

#include "gaccum_kernels.cuh"

namespace gaccum {

constexpr int kMaxRanks = 8;
// control block layout (uint32 words), one block per rank, zero-initialised once:
//   [phase * kMaxRanks + src]  epoch flags, phase 0..2
//   byte 128: double norm_partial[kMaxRanks]
constexpr int kCtrlFlagWords = 3 * kMaxRanks;
constexpr int kCtrlNormByteOffset = 128;
constexpr int kCtrlBytes = 256;
constexpr unsigned long long kDpTimeoutNs = 60ull * 1000 * 1000 * 1000;   // a flag wait longer than 60 s is a dead peer

template <int CAP>
struct GradTable {
  const float* g[CAP];
};

template <int CAP>
struct DpParams {
  const TileDesc* tiles;
  int32_t num_tiles;
  int32_t bounds[kMaxRanks + 1];        // tile range of every rank's shard
  uint32_t shard_base32[kMaxRanks + 1]; // slab offset (units of 32 elements) at which every shard starts
  int64_t stage_span;                   // elements per source region of a staging area (multiple of 32)
  float* accum;                         // local accumulator slab
  float* m;
  float* v;
  double* partials;
  float* stats;
  uint32_t* sync;                       // [0..2] block-completion counters, [3], [5] tile tickets of phases A and C; zero between launches
  Scalars sc;
  int32_t rank, world;
  uint32_t epoch;
  float* param[kMaxRanks];
  float* stage[kMaxRanks];
  uint32_t* ctrl[kMaxRanks];
  GradTable<CAP> tab;
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// End of a phase on this rank: the block's (local and remote) stores are ordered at system scope, the block
// bumps the phase's completion counter, and the LAST block to arrive raises this rank's flag in every
// rank's control block (its own included).  `extra` (run by ALL threads of that last block, before the flags go
// up) lets it publish the norm first.
template <int CAP, typename F>
__device__ __forceinline__ void dp_phase_done(const DpParams<CAP>& prm, int phase, F&& extra) {
  __shared__ int s_last;
  // bar.sync orders every thread's stores before thread 0's fence, and a system-scope fence is cumulative: ONE
  // MEMBAR.SYS per block publishes the whole block's local and remote stores (one per thread -- 150 000 of them,
  // all at the end of a phase -- cost 30 us per phase)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    s_last = atomicAdd(prm.sync + phase, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last) {                                // block-uniform
    if (threadIdx.x == 0) {
      __threadfence_system();                  // acquire side of the counter chain
      prm.sync[phase] = 0;                     // re-arm for the next launch (nobody touches it again in this one)
      if (phase == 2) { prm.sync[3] = 0; prm.sync[4] = 0; prm.sync[5] = 0; }   // every block has left its last ticket loop
    }
    extra();
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence_system();
      for (int w = 0; w < prm.world; ++w) st_release_sys(prm.ctrl[w] + phase * kMaxRanks + prm.rank, prm.epoch);
    }
  }
}
// Tiles of a phase are handed to the blocks by an atomic ticket counter (SMs see different shares of HBM and NVLink
// bandwidth: with a static split the first block finished phase A 40 us before the last).  The block works on ticket i
// while every thread already holds ticket i+1 (so the caller can load that tile's descriptor) and thread 0 draws
// ticket i+2: neither the atomic's round trip nor the descriptor load is on the critical path.
struct TicketLoop {
  uint32_t* ctr;
  int* slot;      // 3 ints of shared memory
  int it;
  int cur, nxt;
  __device__ __forceinline__ void begin(uint32_t* counter, int* s_slot) {
    ctr = counter; slot = s_slot; it = 0;
    if (threadIdx.x == 0) { slot[0] = (int)atomicAdd(ctr, 1u); slot[1] = (int)atomicAdd(ctr, 1u); }
    __syncthreads();
    cur = slot[0]; nxt = slot[1];
  }
  // top of an iteration: thread 0 draws the ticket after next
  __device__ __forceinline__ void prefetch() {
    if (threadIdx.x == 0) slot[(it + 2) % 3] = (int)atomicAdd(ctr, 1u);
  }
  // bottom of an iteration
  __device__ __forceinline__ void advance() {
    __syncthreads();
    ++it;
    cur = nxt;
    nxt = slot[(it + 1) % 3];
  }
};
// Every block: wait until all W ranks have raised `phase` for this epoch (polling this rank's own control block)
template <int CAP>
__device__ __forceinline__ void dp_wait(const DpParams<CAP>& prm, int phase) {
  const int t = threadIdx.x;
  if (t < prm.world) {
    const uint32_t* mine = prm.ctrl[prm.rank] + phase * kMaxRanks + t;
    // poll with relaxed loads (no fence per probe), acquire once when the flag has flipped
    uint32_t seen;
    unsigned long long t_start = 0;
    uint32_t spins = 0;
    do {
      asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(mine) : "memory");
      // A peer that never arrives (crashed rank, mismatched epoch) must not hang the GPU for ever:
      // after kDpTimeoutNs the kernel traps, which surfaces as a sticky CUDA error on the host.
      if (seen != prm.epoch && (++spins & 0x3fffu) == 0) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t_start == 0) t_start = now;
        else if (now - t_start > kDpTimeoutNs) __trap();
      }
    } while (seen != prm.epoch);
    asm volatile("fence.acq_rel.sys;" ::: "memory");
  }
  __syncthreads();
}

template <int CAP>
__device__ __forceinline__ int dp_owner(const DpParams<CAP>& prm, int t) {
  int o = 0;
#pragma unroll
  for (int w = 1; w < kMaxRanks; ++w) o += (w < prm.world && t >= prm.bounds[w]) ? 1 : 0;
  return o;
}

// ---- phase A: one tile.  x = a + G; owned -> a = x (kept for phase B), foreign -> owner's staging, a = 0 ----
template <int CAP>
__device__ __forceinline__ void dp_push_tile(const TileDesc d, const int t, const DpParams<CAP>& prm, const uint64_t pol) {
  const float* __restrict__ g = prm.tab.g[d.tensor_flags & 0x7fffffffu];
  if (g) g += d.toff;
  const size_t soff = (size_t)d.soff32 * kSlabAlign;
  float* __restrict__ a = prm.accum + soff;
  const int owner = dp_owner(prm, t);
  const bool mine = owner == prm.rank;
  float* __restrict__ dst = nullptr;
  if (!mine) {
    const int slot = prm.rank < owner ? prm.rank : prm.rank - 1;
    dst = prm.stage[owner] + (size_t)slot * prm.stage_span + (soff - (size_t)prm.shard_base32[owner] * kSlabAlign);
  }
  const uint32_t len = d.len, tid = threadIdx.x;
  if (mine && g == nullptr) return;                       // nothing to add, nothing to send
  if (g == nullptr || aligned16(g)) {
    const uint32_t nvec = len >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* a4 = reinterpret_cast<float4*>(a);
    float4* d4 = reinterpret_cast<float4*>(dst);
    float4 va[kUnroll], vg[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) { va[u] = __ldcs(a4 + i); if (g) vg[u] = ld_stream(g4 + i); }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t i = u * kThreads + tid;
      if (i < nvec) {
        if (g) {
          va[u].x = __fadd_rn(va[u].x, vg[u].x); va[u].y = __fadd_rn(va[u].y, vg[u].y);
          va[u].z = __fadd_rn(va[u].z, vg[u].z); va[u].w = __fadd_rn(va[u].w, vg[u].w);
        }
        if (mine) st_policy(a4 + i, va[u], pol);
        else { d4[i] = va[u]; __stcs(a4 + i, make_float4(0.f, 0.f, 0.f, 0.f)); }
      }
    }
    const uint32_t i = (nvec << 2) + tid;
    if (i < len) {
      float x = a[i];
      if (g) x = __fadd_rn(x, ld_stream(g + i));
      if (mine) a[i] = x; else { dst[i] = x; a[i] = 0.f; }
    }
  } else {
    for (uint32_t i = tid; i < len; i += kThreads) {
      const float x = __fadd_rn(a[i], ld_stream(g + i));
      if (mine) a[i] = x; else { dst[i] = x; a[i] = 0.f; }
    }
  }
}

// ---- phase B: one owned tile.  a' = sum_w contribution_w in rank order; returns sum((a'/N)^2) ----
template <int CAP>
__device__ __forceinline__ float dp_reduce_tile(const TileDesc d, const DpParams<CAP>& prm, const uint64_t pol) {
  const size_t soff = (size_t)d.soff32 * kSlabAlign;
  const size_t rel = soff - (size_t)prm.shard_base32[prm.rank] * kSlabAlign;
  float* __restrict__ a = prm.accum + soff;
  const float* __restrict__ stg = prm.stage[prm.rank] + rel;
  const int64_t span = prm.stage_span;
  const uint32_t len = d.len, tid = threadIdx.x, nvec = len >> 2;
  const float nf = prm.sc.nf, inv_nf = prm.sc.inv_nf;
  const int W = prm.world, R = prm.rank;
  float acc = 0.f;
  float4* a4 = reinterpret_cast<float4*>(a);
#pragma unroll
  for (int u = 0; u < kUnroll; ++u) {
    const uint32_t i = u * kThreads + tid;
    if (i < nvec) {
      float4 part[kMaxRanks];
#pragma unroll
      for (int w = 0; w < kMaxRanks; ++w) {
        if (w < W) {
          // contributions arrived from other SMs / other GPUs during this kernel: read them at L2
          const float4* src = (w == R) ? (a4 + i) : reinterpret_cast<const float4*>(stg + (size_t)(w < R ? w : w - 1) * span) + i;
          part[w] = __ldcg(src);
        }
      }
      float4 s = part[0];
#pragma unroll
      for (int w = 1; w < kMaxRanks; ++w) {
        if (w < W) {
          s.x = __fadd_rn(s.x, part[w].x); s.y = __fadd_rn(s.y, part[w].y);
          s.z = __fadd_rn(s.z, part[w].z); s.w = __fadd_rn(s.w, part[w].w);
        }
      }
      st_policy(a4 + i, s, pol);
      const float nx = normalize(s.x, nf, inv_nf), ny = normalize(s.y, nf, inv_nf), nz = normalize(s.z, nf, inv_nf), nw = normalize(s.w, nf, inv_nf);
      acc = fmaf(nx, nx, acc); acc = fmaf(ny, ny, acc); acc = fmaf(nz, nz, acc); acc = fmaf(nw, nw, acc);
    }
  }
  const uint32_t i = (nvec << 2) + tid;
  if (i < len) {
    float s = 0.f;
    for (int w = 0; w < W; ++w) {
      const float x = __ldcg((w == R) ? (a + i) : (stg + (size_t)(w < R ? w : w - 1) * span + i));
      s = (w == 0) ? x : __fadd_rn(s, x);
    }
    a[i] = s;
    const float n = normalize(s, nf, inv_nf);
    acc = fmaf(n, n, acc);
  }
  return acc;
}

// ---- phase C: one owned tile.  update from the reduced a', broadcast p' to every rank ----
template <int VARIANT, int CAP>
__device__ __forceinline__ void dp_update_tile(const TileDesc d, const DpParams<CAP>& prm, const float s) {
  const size_t soff = (size_t)d.soff32 * kSlabAlign;
  float* __restrict__ a = prm.accum + soff;
  float* __restrict__ m = prm.m + soff;
  float* __restrict__ v = prm.v + soff;
  const float* __restrict__ p = prm.param[prm.rank] + soff;
  const bool decay = (d.tensor_flags >> 31) != 0;
  const uint32_t len = d.len, tid = threadIdx.x, nvec = len >> 2;
  const Scalars& sc = prm.sc;
  const int W = prm.world;
  auto elem = [&](float ax, float& px, float& mx, float& vx) {
    const float c = sc.clip > 0.f ? __fmul_rn(normalize(ax, sc.nf, sc.inv_nf), s) : normalize(ax, sc.nf, sc.inv_nf);
    adam_elem<VARIANT>(c, px, mx, vx, decay, sc);
  };
  float4* a4 = reinterpret_cast<float4*>(a);
  float4* m4 = reinterpret_cast<float4*>(m);
  float4* v4 = reinterpret_cast<float4*>(v);
  const float4* p4 = reinterpret_cast<const float4*>(p);
  float4 va[kUnroll], vp[kUnroll], vm[kUnroll], vv[kUnroll];
#pragma unroll
  for (int u = 0; u < kUnroll; ++u) {
    const uint32_t i = u * kThreads + tid;
    if (i < nvec) { va[u] = __ldcg(a4 + i); vp[u] = __ldcs(p4 + i); vm[u] = __ldcs(m4 + i); vv[u] = __ldcs(v4 + i); }
  }
#pragma unroll
  for (int u = 0; u < kUnroll; ++u) {
    const uint32_t i = u * kThreads + tid;
    if (i < nvec) {
      elem(va[u].x, vp[u].x, vm[u].x, vv[u].x); elem(va[u].y, vp[u].y, vm[u].y, vv[u].y);
      elem(va[u].z, vp[u].z, vm[u].z, vv[u].z); elem(va[u].w, vp[u].w, vm[u].w, vv[u].w);
      __stcs(m4 + i, vm[u]); __stcs(v4 + i, vv[u]);
      __stcs(a4 + i, make_float4(0.f, 0.f, 0.f, 0.f));
#pragma unroll
      for (int w = 0; w < kMaxRanks; ++w)      // all-gather: peer stores over NVLink (and the local copy)
        if (w < W) *(reinterpret_cast<float4*>(prm.param[w] + soff) + i) = vp[u];
    }
  }
  const uint32_t i = (nvec << 2) + tid;
  if (i < len) {
    float px = p[i], mx = m[i], vx = v[i];
    elem(__ldcg(a + i), px, mx, vx);
    m[i] = mx; v[i] = vx; a[i] = 0.f;
    for (int w = 0; w < W; ++w) prm.param[w][soff + i] = px;
  }
}

// Deterministic CTA reduction of one double per thread -> total in thread 0.  Threads add each
// tile's 8-element fp32 partial into an fp64 running sum, so the norm of a 335 M-element model is
// good to ~1e-7 relative even for adversarial (constant) data.
__device__ __forceinline__ double block_reduce_to_double(double x, double* smem /* blockDim.x/32 */) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) smem[warp] = x;
  __syncthreads();
  double tot = 0.0;
  if (threadIdx.x == 0) {
    const int nw = ((int)blockDim.x + 31) >> 5;
    for (int w = 0; w < nw; ++w) tot += smem[w];
  }
  return tot;
}

template <int VARIANT, int CAP>
__global__ void __launch_bounds__(kThreads, 4)
dp_apply_kernel(const __grid_constant__ DpParams<CAP> prm) {
  __shared__ double red[kThreads / 32];
  __shared__ float s_bcast[2];
  const uint64_t pol = policy_evict_last();
  const int W = prm.world, R = prm.rank, nt = prm.num_tiles;
  const int lo = prm.bounds[R], hi = prm.bounds[R + 1];

  __shared__ int s_ticket[3];
  TicketLoop tl;
  // ---- phase A: local accumulate + reduce-scatter by pushes.  Ticket q -> tile i = q / W of shard (R + 1 + q % W) % W:
  //      consecutive tickets go to W different owners (the last one is this rank itself), so pushes to every peer are
  //      spread evenly over the whole phase instead of arriving in one burst that NVLink then needs 30 us to drain, and
  //      at any moment every owner receives from every source at the same rate ----
  {
    int max_shard = 0;
    for (int w = 0; w < W; ++w) max_shard = max(max_shard, prm.bounds[w + 1] - prm.bounds[w]);
    const int nq = max_shard * W;
    auto tile_of = [&](int q) -> int {
      if (q >= nq) return -1;
      int o = R + 1 + q % W;
      if (o >= W) o -= W;
      const int t = prm.bounds[o] + q / W;
      return t < prm.bounds[o + 1] ? t : -1;
    };
    tl.begin(prm.sync + 3, s_ticket);
    int t = tile_of(tl.cur);
    TileDesc d{};
    if (t >= 0) d = prm.tiles[t];
    while (tl.cur < nq) {
      tl.prefetch();
      const int tn = tile_of(tl.nxt);
      TileDesc dn{};
      if (tn >= 0) dn = prm.tiles[tn];                      // next descriptor: in flight while this tile is processed
      if (t >= 0) dp_push_tile(d, t, prm, pol);
      tl.advance();
      t = tn; d = dn;
    }
  }
  dp_phase_done(prm, 0, [] {});
  dp_wait(prm, 0);

  // ---- phase B: reduction of the owned shard in fixed rank order + norm partial.  Local traffic only and short: a static
  //      split (block b takes owned tiles b, b + G, ...) beats tickets here (31 vs 48 us at W=2: per-tile barriers
  //      cost more than the imbalance), and keeps the reduction order fixed: thread fp64 running sums -> block tree ->
  //      one partial per block -> the last block adds the partials in block order ---------------------------------
  {
    double acc = 0.0;
    const int G = (int)gridDim.x;
    int t = lo + (int)blockIdx.x;
    TileDesc d{};
    if (t < hi) d = prm.tiles[t];
    while (t < hi) {
      TileDesc dn{};
      if (t + G < hi) dn = prm.tiles[t + G];
      acc += (double)dp_reduce_tile(d, prm, pol);
      t += G; d = dn;
    }
    const double part = block_reduce_to_double(acc, red);
    if (threadIdx.x == 0) prm.partials[blockIdx.x] = part;
  }
  dp_phase_done(prm, 1, [&] {
    // last block of this rank: per-block partials, fixed tree -> this rank's partial norm -> every rank
    double tot = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += kThreads) tot += __ldcg(prm.partials + i);
    tot = block_reduce_to_double(tot, red);
    if (threadIdx.x == 0) {
      for (int w = 0; w < W; ++w) {
        double* slot = reinterpret_cast<double*>(reinterpret_cast<char*>(prm.ctrl[w]) + kCtrlNormByteOffset) + R;
        asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(slot), "d"(tot) : "memory");
      }
    }
  });
  dp_wait(prm, 1);
  if (threadIdx.x == 0) {
    const double* slots = reinterpret_cast<const double*>(reinterpret_cast<const char*>(prm.ctrl[R]) + kCtrlNormByteOffset);
    double tot = 0.0;
    for (int w = 0; w < W; ++w) {
      double x;
      asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(x) : "l"(slots + w) : "memory");
      tot += x;
    }
    const float g_norm = prm.sc.clip > 0.f ? __fsqrt_rn((float)tot) : 0.f;
    s_bcast[0] = prm.sc.clip > 0.f ? clip_scale(g_norm, prm.sc.clip) : 1.f;
    s_bcast[1] = g_norm;
    if (blockIdx.x == 0) {
      prm.stats[0] = 1.f; prm.stats[1] = prm.sc.lr; prm.stats[2] = g_norm; prm.stats[3] = s_bcast[0];
    }
  }
  __syncthreads();
  const float s = s_bcast[0];

  // ---- phase C: sharded update + all-gather by pushes ----------------------------------------------------
  {
    tl.begin(prm.sync + 5, s_ticket);
    TileDesc d{};
    if (lo + tl.cur < hi) d = prm.tiles[lo + tl.cur];
    while (lo + tl.cur < hi) {
      tl.prefetch();
      TileDesc dn{};
      if (lo + tl.nxt < hi) dn = prm.tiles[lo + tl.nxt];
      dp_update_tile<VARIANT>(d, prm, s);
      tl.advance();
      d = dn;
    }
  }
  dp_phase_done(prm, 2, [] {});
  // every peer's parameter stores into my slab are complete before the kernel ends
  if (blockIdx.x == 0) dp_wait(prm, 2);
}

}  // namespace gaccum
