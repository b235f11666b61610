// gaccum_abi.cu -- host side of libgaccum.so: plan (slab layout + static tile table), the
// scalar host logic of the reference graph, and the C ABI declared in include/gaccum.h.
// No CPU compute path exists here on purpose: without a device every step call fails.
#include <regex.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/gaccum.h"
#include "gaccum_kernels.cuh"
#include "gaccum_dp.cuh"

using namespace gaccum;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CUDA_TRY(expr)                                                                        \
  do {                                                                                        \
    cudaError_t e_ = (expr);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(GACCUM_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// ------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------
constexpr int kCapSmall = 256;    // 4 KB pointer table   (MNIST, BERT-Small 73, BERT-Base 201)
constexpr int kCapLarge = 1920;   // 30 KB pointer table  (BERT-Large 393, ...; CUDA >= 12.1 32 KB params)

struct gaccum_plan {
  int32_t T = 0;
  int32_t device = -1;
  gaccum_hparams hp{};
  std::vector<int64_t> numel, offset;
  std::vector<uint8_t> decay;
  std::vector<TileDesc> tiles;
  int64_t P = 0, padded = 0;
  // device side
  TileDesc* d_tiles = nullptr;
  double* d_partials = nullptr;           // data-parallel kernel: one norm partial per block
  float* d_stats = nullptr;
  uint32_t* d_dp_sync = nullptr;           // data-parallel kernel: block-completion counters and tile tickets (zero between launches)
  unsigned long long* d_barrier = nullptr; // clip-apply kernel: monotonic arrival counter of the consumers' grid barrier
  LaunchCounters* d_counters = nullptr;    // ... two sets of per-launch counters (tickets, pool length, norm accumulator)
  int num_sms = 0;
  int max_grid = 0;
  std::mutex mu;
  std::map<const void*, int> grid_cache;   // kernel -> co-resident grid size
};

static int build_layout(gaccum_plan* pl) {
  pl->offset.resize(pl->T);
  int64_t off = 0, P = 0;
  pl->tiles.clear();
  for (int32_t t = 0; t < pl->T; ++t) {
    const int64_t n = pl->numel[t];
    if (n < 0) return fail(GACCUM_EINVAL, "numels[%d] = %lld is negative", t, (long long)n);
    if (n >= (int64_t)1 << 32) return fail(GACCUM_EINVAL, "tensor %d has %lld elements; limit is 2^32-1", t, (long long)n);
    pl->offset[t] = off;
    for (int64_t to = 0; to < n; to += kTile) {
      TileDesc d;
      d.tensor_flags = (uint32_t)t | (pl->decay[t] ? 0x80000000u : 0u);
      d.len = (uint32_t)std::min<int64_t>(kTile, n - to);
      d.toff = (uint32_t)to;
      const int64_t s32 = (off + to) / kSlabAlign;
      if (s32 >= (int64_t)1 << 32) return fail(GACCUM_EINVAL, "slab too large (> 2^37 elements)");
      d.soff32 = (uint32_t)s32;
      pl->tiles.push_back(d);
    }
    P += n;
    off += (n + kSlabAlign - 1) / kSlabAlign * kSlabAlign;
  }
  if (pl->tiles.size() >= (size_t)1 << 31) return fail(GACCUM_EINVAL, "too many tiles");
  pl->P = P;
  pl->padded = off;
  return GACCUM_OK;
}

// ------------------------------------------------------------------------------------------
// scalars of one apply step
// ------------------------------------------------------------------------------------------
static Scalars make_scalars(const gaccum_hparams& hp, const gaccum_step_args* a) {
  Scalars s{};
  s.nf = a ? (float)a->accum_n : 1.0f;
  {
    const int32_t n = a ? a->accum_n : 1;
    s.inv_nf = (n > 0 && (n & (n - 1)) == 0 && n <= (1 << 24)) ? 1.0f / (float)n : 0.0f;
  }
  s.lr = a ? a->lr : 0.0f;
  s.b1 = (float)hp.beta1;
  s.b2 = (float)hp.beta2;
  s.eps = (float)hp.epsilon;
  s.wd = (float)hp.weight_decay_rate;
  s.clip = (float)hp.clip_norm;
  if (hp.variant == GACCUM_ADAM_WEIGHT_DECAY) {
    s.omb1 = (float)(1.0 - hp.beta1);   // optimization.py:152 -- Python double, then fp32
    s.omb2 = (float)(1.0 - hp.beta2);   // optimization.py:154
  } else {
    volatile float o1 = 1.0f - s.b1, o2 = 1.0f - s.b2;   // ApplyAdam: T(1) - beta1()
    s.omb1 = o1;
    s.omb2 = o2;
    if (a) {
      volatile float t1 = 1.0f - a->beta2_power;
      volatile float t2 = sqrtf(t1);
      volatile float t3 = a->lr * t2;
      volatile float t4 = 1.0f - a->beta1_power;
      volatile float t5 = t3 / t4;
      s.alpha = t5;
    }
  }
  return s;
}

// ------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------
static int grid_for(gaccum_plan* pl, const void* fn, int* out) {
  std::lock_guard<std::mutex> lk(pl->mu);
  auto it = pl->grid_cache.find(fn);
  if (it != pl->grid_cache.end()) { *out = it->second; return GACCUM_OK; }
  int per_sm = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kThreads, 0));
  if (per_sm < 1) return fail(GACCUM_ECUDA, "kernel does not fit on an SM");
  int g = std::min(per_sm * pl->num_sms, pl->max_grid);
  pl->grid_cache[fn] = g;
  *out = g;
  return GACCUM_OK;
}

template <int CAP>
static int launch_accumulate(KernelParams<CAP>& prm, cudaStream_t st) {
  // one tile per CTA: the hardware block scheduler balances better than a persistent loop (r01_tune_sweep.md)
  const int grid = std::max(1, prm.num_tiles);
  accumulate_kernel<CAP><<<grid, kThreads, 0, st>>>(prm);
  CUDA_TRY(cudaGetLastError());
  return GACCUM_OK;
}

template <int VARIANT, bool HAS_G, int CAP>
static int launch_apply_noclip(KernelParams<CAP>& prm, cudaStream_t st) {
  const int grid = std::max(1, prm.num_tiles);
  apply_kernel<VARIANT, HAS_G, CAP><<<grid, kThreads, 0, st>>>(prm);
  CUDA_TRY(cudaGetLastError());
  return GACCUM_OK;
}

// clip-apply: one cooperative launch, ONE 864-thread CTA per SM (it allocates all of Tensor Memory, so a second
// CTA could never be co-resident -- the grid is clamped to the SM count, not derived from the occupancy API)
template <int VARIANT, bool HAS_G, int CAP>
static int launch_apply_clip(gaccum_plan* pl, KernelParams<CAP>& prm, cudaStream_t st) {
  const void* fn = (const void*)&apply_clip_kernel<VARIANT, HAS_G, CAP>;
  {
    std::lock_guard<std::mutex> lk(pl->mu);
    if (pl->grid_cache.find(fn) == pl->grid_cache.end()) {
      CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kRingBytes));
      int per_sm = 0;
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kClipThreads, (size_t)kRingBytes));
      if (per_sm < 1) return fail(GACCUM_ECUDA, "apply_clip_kernel does not fit on an SM (%d B dynamic shared memory)", kRingBytes);
      pl->grid_cache[fn] = pl->num_sms;
    }
  }
  // the grid must be the same for every launch on this plan: the consumers' barrier counter advances by gridDim.x
  const int grid = std::max(1, std::min(pl->num_sms, ((int)pl->tiles.size() + kGroups - 1) / kGroups));
  prm.barrier = pl->d_barrier;
  prm.counters = pl->d_counters;
  void* args[] = {(void*)&prm};
  CUDA_TRY(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kClipThreads), args, (size_t)kRingBytes, st));
  return GACCUM_OK;
}

template <int CAP>
static int launch_apply(gaccum_plan* pl, KernelParams<CAP>& prm, bool has_g, cudaStream_t st) {
  const bool clip = pl->hp.clip_norm > 0.0;
  const int key = (pl->hp.variant == GACCUM_ADAM ? 4 : 0) | (clip ? 2 : 0) | (has_g ? 1 : 0);
  switch (key) {
    case 0: return launch_apply_noclip<0, false>(prm, st);
    case 1: return launch_apply_noclip<0, true>(prm, st);
    case 2: return launch_apply_clip<0, false>(pl, prm, st);
    case 3: return launch_apply_clip<0, true>(pl, prm, st);
    case 4: return launch_apply_noclip<1, false>(prm, st);
    case 5: return launch_apply_noclip<1, true>(prm, st);
    case 6: return launch_apply_clip<1, false>(pl, prm, st);
    default: return launch_apply_clip<1, true>(pl, prm, st);
  }
}

static inline bool aligned16_host(const void* p) { return ((uintptr_t)p & 15u) == 0; }

static int check_compute(gaccum_plan* pl, const float* accum, const float* m, const float* v, bool need_mv) {
  if (!pl) return fail(GACCUM_EINVAL, "plan is NULL");
  if (pl->device < 0)
    return fail(GACCUM_ENODEVICE, "layout-only plan (device=-1): libgaccum has no CPU fallback, a CUDA device is required");
  if (!accum || !aligned16_host(accum)) return fail(GACCUM_EINVAL, "accum must be a 16-byte aligned device pointer");
  if (need_mv && (!m || !v || !aligned16_host(m) || !aligned16_host(v)))
    return fail(GACCUM_EINVAL, "m and v must be 16-byte aligned device pointers");
  return GACCUM_OK;
}

template <int CAP>
static void fill_common(gaccum_plan* pl, KernelParams<CAP>& prm, float* accum, float* m, float* v,
                        const Scalars& sc) {
  prm.tiles = pl->d_tiles;
  prm.num_tiles = (int32_t)pl->tiles.size();
  prm.accum = accum;
  prm.m = m;
  prm.v = v;
  prm.stats = pl->d_stats;
  prm.sc = sc;
}

template <int CAP>
static int fill_table(gaccum_plan* pl, PtrTable<CAP>& tab, const float* const* grads, float* const* params) {
  for (int32_t t = 0; t < pl->T; ++t) {
    tab.g[t] = grads ? grads[t] : nullptr;
    if (params) {
      if (!params[t] && pl->numel[t] > 0) return fail(GACCUM_EINVAL, "params[%d] is NULL", t);
      tab.p[t] = params[t];
    }
  }
  return GACCUM_OK;
}

struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
    else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0 && ok) cudaSetDevice(prev); }
};

template <int CAP>
static int do_accumulate_tab(gaccum_plan* pl, const float* const* grads, float* accum,
                             const gaccum_step_args* a, cudaStream_t st) {
  KernelParams<CAP>* prm = new (std::nothrow) KernelParams<CAP>();
  if (!prm) return fail(GACCUM_ENOMEM, "out of host memory");
  fill_common(pl, *prm, accum, nullptr, nullptr, make_scalars(pl->hp, a));
  int rc = fill_table(pl, prm->tab, grads, nullptr);
  if (rc == GACCUM_OK) rc = launch_accumulate(*prm, st);
  delete prm;
  return rc;
}

template <int CAP>
static int do_apply_tab(gaccum_plan* pl, const float* const* grads, float* const* params, float* accum,
                        float* m, float* v, const gaccum_step_args* a, cudaStream_t st) {
  KernelParams<CAP>* prm = new (std::nothrow) KernelParams<CAP>();
  if (!prm) return fail(GACCUM_ENOMEM, "out of host memory");
  fill_common(pl, *prm, accum, m, v, make_scalars(pl->hp, a));
  int rc = fill_table(pl, prm->tab, grads, params);
  if (rc == GACCUM_OK) rc = launch_apply(pl, *prm, grads != nullptr, st);
  delete prm;
  return rc;
}

static int check_args(const gaccum_step_args* a) {
  if (!a) return fail(GACCUM_EINVAL, "args is NULL");
  if (a->accum_n <= 0) return fail(GACCUM_EINVAL, "accum_n must be > 0 (got %d)", a->accum_n);
  if (a->reserved != 0 || a->reserved2 != 0.0f) return fail(GACCUM_EINVAL, "reserved fields must be 0");
  return GACCUM_OK;
}

static void free_plan_device(gaccum_plan* pl) {
  cudaFree(pl->d_tiles); cudaFree(pl->d_partials); cudaFree(pl->d_stats); cudaFree(pl->d_dp_sync); cudaFree(pl->d_barrier); cudaFree(pl->d_counters);
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

int gaccum_version(void) { return GACCUM_VERSION; }
const char* gaccum_last_error(void) { return g_err.c_str(); }

int gaccum_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// optimization.py:29-54, fp32 op order (volatile: one rounding per TF op, no double promotion)
float gaccum_learning_rate(double init_lr, int64_t num_train_steps, int64_t num_warmup_steps,
                           int64_t global_step) {
  volatile float lr0 = (float)init_lr;
  volatile float gs = (float)global_step;
  volatile float ds = (float)num_train_steps;
  if (gs > ds) gs = ds;
  volatile float p = gs / ds;
  volatile float omp = 1.0f - p;
  volatile float lr = lr0 * omp;
  if (num_warmup_steps) {
    const int32_t gi = (int32_t)global_step, wi = (int32_t)num_warmup_steps;
    volatile float pct = (float)gi / (float)wi;
    volatile float wlr = (float)init_lr * pct;
    volatile float isw = gi < wi ? 1.0f : 0.0f;
    volatile float x = (1.0f - isw) * lr;
    volatile float y = isw * wlr;
    lr = x + y;
  }
  return lr;
}

int gaccum_is_apply_step(int64_t global_step, int32_t accum_n) {
  if (accum_n <= 0) return 0;
  return ((int32_t)global_step % accum_n) == 0;   // optimization.py:77,91
}

int gaccum_decay_mask(int32_t T, const char* const* names, double weight_decay_rate,
                      const char* const* exclude, int32_t num_exclude, uint8_t* out) {
  if (T < 0 || (T > 0 && (!names || !out))) return fail(GACCUM_EINVAL, "bad arguments to gaccum_decay_mask");
  std::vector<regex_t> res((size_t)std::max(0, num_exclude));
  int compiled = 0;
  int rc = GACCUM_OK;
  for (; compiled < num_exclude; ++compiled) {
    if (!exclude || !exclude[compiled] || regcomp(&res[compiled], exclude[compiled], REG_EXTENDED | REG_NOSUB) != 0) {
      rc = fail(GACCUM_EINVAL, "exclude[%d] is not a valid regular expression", compiled);
      break;
    }
  }
  if (rc == GACCUM_OK) {
    for (int32_t t = 0; t < T; ++t) {
      std::string nm = names[t] ? names[t] : "";
      // optimization.py:189-194 -- strip ":<digits>"
      size_t c = nm.rfind(':');
      if (c != std::string::npos && c + 1 < nm.size() &&
          std::all_of(nm.begin() + c + 1, nm.end(), [](char ch) { return ch >= '0' && ch <= '9'; }))
        nm.resize(c);
      uint8_t use = weight_decay_rate != 0.0;      // optimization.py:181 `if not self.weight_decay_rate`
      for (int i = 0; use && i < num_exclude; ++i)
        if (regexec(&res[i], nm.c_str(), 0, nullptr, 0) == 0) use = 0;   // :183-186 re.search
      out[t] = use;
    }
  }
  for (int i = 0; i < compiled; ++i) regfree(&res[i]);
  return rc;
}

int gaccum_plan_create(gaccum_plan** out, int32_t T, const int64_t* numels, const uint8_t* decay,
                       const gaccum_hparams* hp, int32_t device) {
  if (!out) return fail(GACCUM_EINVAL, "out is NULL");
  *out = nullptr;
  if (T < 0 || (T > 0 && !numels)) return fail(GACCUM_EINVAL, "bad tensor list");
  if (!hp) return fail(GACCUM_EINVAL, "hp is NULL");
  if (hp->variant != GACCUM_ADAM_WEIGHT_DECAY && hp->variant != GACCUM_ADAM)
    return fail(GACCUM_EINVAL, "unknown optimizer variant %d", hp->variant);
  if (hp->reserved != 0) return fail(GACCUM_EINVAL, "reserved fields must be 0");
  if (T > kCapLarge)
    return fail(GACCUM_EINVAL, "%d tensors exceed the %d-entry pointer table; use the packed entry point with one slab", T, kCapLarge);
  gaccum_plan* pl = new (std::nothrow) gaccum_plan();
  if (!pl) return fail(GACCUM_ENOMEM, "out of host memory");
  pl->T = T;
  pl->hp = *hp;
  pl->numel.assign(numels, numels + T);
  pl->decay.assign((size_t)T, 0);
  if (hp->variant == GACCUM_ADAM_WEIGHT_DECAY && decay) pl->decay.assign(decay, decay + T);
  if (int rc = build_layout(pl)) { delete pl; return rc; }
  pl->device = -1;
  if (device >= 0) {
    int n = gaccum_device_count();
    if (device >= n) { delete pl; return fail(GACCUM_ENODEVICE, "CUDA device %d requested but %d device(s) visible; libgaccum has no CPU fallback", device, n); }
    DeviceGuard guard(device);
    cudaDeviceProp prop{};
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e == cudaSuccess && !prop.cooperativeLaunch) e = cudaErrorNotSupported;
    const size_t tb = std::max<size_t>(1, pl->tiles.size()) * sizeof(TileDesc);
    pl->num_sms = prop.multiProcessorCount;
    pl->max_grid = pl->num_sms * 16;
    if (e == cudaSuccess) e = cudaMalloc(&pl->d_tiles, tb);
    if (e == cudaSuccess && !pl->tiles.empty())
      e = cudaMemcpy(pl->d_tiles, pl->tiles.data(), pl->tiles.size() * sizeof(TileDesc), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&pl->d_partials, sizeof(double) * (size_t)pl->max_grid);
    if (e == cudaSuccess) e = cudaMalloc(&pl->d_dp_sync, sizeof(uint32_t) * 8);
    if (e == cudaSuccess) e = cudaMemset(pl->d_dp_sync, 0, sizeof(uint32_t) * 8);
    if (e == cudaSuccess) e = cudaMalloc(&pl->d_barrier, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(pl->d_barrier, 0, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&pl->d_counters, 2 * sizeof(LaunchCounters));
    if (e == cudaSuccess) e = cudaMemset(pl->d_counters, 0, 2 * sizeof(LaunchCounters));
    if (e == cudaSuccess) e = cudaMalloc(&pl->d_stats, sizeof(gaccum_stats));
    if (e == cudaSuccess) e = cudaMemset(pl->d_stats, 0, sizeof(gaccum_stats));
    if (e != cudaSuccess) {
      free_plan_device(pl);
      delete pl;
      return fail(GACCUM_ECUDA, "plan device setup failed: %s", cudaGetErrorString(e));
    }
    pl->device = device;
  }
  *out = pl;
  return GACCUM_OK;
}

int gaccum_plan_destroy(gaccum_plan* pl) {
  if (!pl) return GACCUM_OK;
  if (pl->device >= 0) {
    DeviceGuard guard(pl->device);
    free_plan_device(pl);
  }
  delete pl;
  return GACCUM_OK;
}

int64_t gaccum_padded_size(const gaccum_plan* pl) { return pl ? pl->padded : fail(GACCUM_EINVAL, "plan is NULL"); }
int32_t gaccum_num_tensors(const gaccum_plan* pl) { return pl ? pl->T : fail(GACCUM_EINVAL, "plan is NULL"); }
int64_t gaccum_num_elements(const gaccum_plan* pl) { return pl ? pl->P : fail(GACCUM_EINVAL, "plan is NULL"); }
int32_t gaccum_num_tiles(const gaccum_plan* pl) { return pl ? (int32_t)pl->tiles.size() : fail(GACCUM_EINVAL, "plan is NULL"); }

int gaccum_offsets(const gaccum_plan* pl, int64_t* out) {
  if (!pl || (!out && pl->T > 0)) return fail(GACCUM_EINVAL, "bad arguments to gaccum_offsets");
  std::copy(pl->offset.begin(), pl->offset.end(), out);
  return GACCUM_OK;
}

int64_t gaccum_algorithmic_bytes(const gaccum_plan* pl, int32_t is_apply) {
  if (!pl) return fail(GACCUM_EINVAL, "plan is NULL");
  // accumulate: read G, read a, write a.  apply: read G,a,p,m,v + write p,m,v,a  (SURVEY.md 8(d))
  return pl->P * (is_apply ? 36 : 12);
}

static int accumulate_impl(gaccum_plan* pl, const float* const* grads, float* accum,
                           const gaccum_step_args* a, gaccum_stream_t stream) {
  if (int rc = check_compute(pl, accum, nullptr, nullptr, false)) return rc;
  if (!grads) return fail(GACCUM_EINVAL, "grads is NULL");
  DeviceGuard guard(pl->device);
  cudaStream_t st = (cudaStream_t)stream;
  return pl->T <= kCapSmall ? do_accumulate_tab<kCapSmall>(pl, grads, accum, a, st)
                            : do_accumulate_tab<kCapLarge>(pl, grads, accum, a, st);
}

int gaccum_accumulate(gaccum_plan* pl, const float* const* grads, float* accum, gaccum_stream_t stream) {
  return accumulate_impl(pl, grads, accum, nullptr, stream);
}

int gaccum_apply(gaccum_plan* pl, const float* const* grads, float* const* params, float* accum,
                 float* m, float* v, const gaccum_step_args* a, gaccum_stream_t stream) {
  if (int rc = check_compute(pl, accum, m, v, true)) return rc;
  if (int rc = check_args(a)) return rc;
  if (!params) return fail(GACCUM_EINVAL, "params is NULL");
  DeviceGuard guard(pl->device);
  cudaStream_t st = (cudaStream_t)stream;
  return pl->T <= kCapSmall ? do_apply_tab<kCapSmall>(pl, grads, params, accum, m, v, a, st)
                            : do_apply_tab<kCapLarge>(pl, grads, params, accum, m, v, a, st);
}

int gaccum_step(gaccum_plan* pl, const float* const* grads, float* const* params, float* accum,
                float* m, float* v, const gaccum_step_args* a, gaccum_stream_t stream) {
  if (int rc = check_args(a)) return rc;
  if (!grads) return fail(GACCUM_EINVAL, "grads is NULL");
  if (gaccum_is_apply_step(a->global_step, a->accum_n)) return gaccum_apply(pl, grads, params, accum, m, v, a, stream);
  return accumulate_impl(pl, grads, accum, a, stream);
}

int gaccum_step_packed(gaccum_plan* pl, const float* grad_slab, float* param_slab, float* accum,
                       float* m, float* v, const gaccum_step_args* a, int32_t force_branch,
                       gaccum_stream_t stream) {
  if (int rc = check_args(a)) return rc;
  const bool apply = force_branch < 0 ? gaccum_is_apply_step(a->global_step, a->accum_n) != 0 : force_branch != 0;
  if (int rc = check_compute(pl, accum, m, v, apply)) return rc;
  if (grad_slab && !aligned16_host(grad_slab)) return fail(GACCUM_EINVAL, "grad_slab must be 16-byte aligned");
  DeviceGuard guard(pl->device);
  cudaStream_t st = (cudaStream_t)stream;
  KernelParams<0> prm{};
  fill_common(pl, prm, accum, m, v, make_scalars(pl->hp, a));
  prm.tab.g = grad_slab;
  prm.tab.p = param_slab;
  if (!apply) {
    if (!grad_slab) return fail(GACCUM_EINVAL, "grad_slab is NULL on an accumulate step");
    return launch_accumulate(prm, st);
  }
  if (!param_slab || !aligned16_host(param_slab)) return fail(GACCUM_EINVAL, "param_slab must be a 16-byte aligned device pointer");
  return launch_apply(pl, prm, grad_slab != nullptr, st);
}

// contiguous tile ranges with (nearly) equal element counts: boundary r = first tile whose cumulative
// element count reaches r * P / world
static void shard_bounds(const gaccum_plan* pl, int world, int* bounds /* world + 1 */) {
  const int nt = (int)pl->tiles.size();
  int64_t cum = 0;
  int r = 1;
  bounds[0] = 0;
  for (int t = 0; t < nt && r < world; ++t) {
    cum += pl->tiles[t].len;
    while (r < world && cum >= (pl->P * r + world - 1) / world) bounds[r++] = t + 1;
  }
  while (r <= world) bounds[r++] = nt;
}
// slab offset (in units of 32 elements) at which tile t starts; t == num_tiles -> end of the slab
static uint32_t tile_soff32(const gaccum_plan* pl, int t) {
  return t < (int)pl->tiles.size() ? pl->tiles[t].soff32 : (uint32_t)(pl->padded / kSlabAlign);
}
// elements of one source region of a staging area = the widest shard's slab span
static int64_t stage_span(const gaccum_plan* pl, int world) {
  int bounds[GACCUM_MAX_RANKS + 1];
  shard_bounds(pl, world, bounds);
  int64_t span = 0;
  for (int r = 0; r < world; ++r)
    span = std::max<int64_t>(span, ((int64_t)tile_soff32(pl, bounds[r + 1]) - (int64_t)tile_soff32(pl, bounds[r])) * kSlabAlign);
  return std::max<int64_t>(span, kSlabAlign);
}

int gaccum_dp_shard_range(const gaccum_plan* pl, int32_t world, int32_t rank, int32_t* tile_lo,
                          int32_t* tile_hi, int64_t* num_elements) {
  if (!pl || !tile_lo || !tile_hi) return fail(GACCUM_EINVAL, "bad arguments to gaccum_dp_shard_range");
  if (world < 1 || world > GACCUM_MAX_RANKS || rank < 0 || rank >= world)
    return fail(GACCUM_EINVAL, "world must be 1..%d and 0 <= rank < world (got world=%d rank=%d)", GACCUM_MAX_RANKS, world, rank);
  int bounds[GACCUM_MAX_RANKS + 1];
  shard_bounds(pl, world, bounds);
  *tile_lo = bounds[rank];
  *tile_hi = bounds[rank + 1];
  if (num_elements) {
    int64_t e = 0;
    for (int t = bounds[rank]; t < bounds[rank + 1]; ++t) e += pl->tiles[t].len;
    *num_elements = e;
  }
  return GACCUM_OK;
}

int64_t gaccum_dp_stage_elements(const gaccum_plan* pl, int32_t world) {
  if (!pl) return fail(GACCUM_EINVAL, "plan is NULL");
  if (world < 2 || world > GACCUM_MAX_RANKS) return fail(GACCUM_EINVAL, "world must be 2..%d", GACCUM_MAX_RANKS);
  return stage_span(pl, world) * (world - 1);
}

extern "C++" {
template <int CAP>
static int do_apply_dp(gaccum_plan* pl, const gaccum_dp_comm* comm, const float* const* grads, float* m, float* v,
                       const gaccum_step_args* a, uint32_t epoch, cudaStream_t st) {
  DpParams<CAP>* prm = new (std::nothrow) DpParams<CAP>();
  if (!prm) return fail(GACCUM_ENOMEM, "out of host memory");
  const int W = comm->world;
  for (int w = 0; w < W; ++w) {
    prm->param[w] = comm->param_peers[w];
    prm->stage[w] = comm->stage_peers[w];
    prm->ctrl[w] = comm->ctrl_peers[w];
  }
  prm->tiles = pl->d_tiles;
  prm->num_tiles = (int32_t)pl->tiles.size();
  int bounds[GACCUM_MAX_RANKS + 1];
  shard_bounds(pl, W, bounds);
  for (int r = 0; r <= W; ++r) { prm->bounds[r] = bounds[r]; prm->shard_base32[r] = tile_soff32(pl, bounds[r]); }
  prm->stage_span = stage_span(pl, W);
  prm->accum = comm->accum;
  prm->m = m;
  prm->v = v;
  prm->partials = pl->d_partials;
  prm->stats = pl->d_stats;
  prm->sync = pl->d_dp_sync;
  prm->sc = make_scalars(pl->hp, a);
  prm->rank = comm->rank;
  prm->world = W;
  prm->epoch = epoch;
  for (int32_t t = 0; t < pl->T; ++t) prm->tab.g[t] = grads ? grads[t] : nullptr;
  const void* fn = pl->hp.variant == GACCUM_ADAM ? (const void*)&dp_apply_kernel<1, CAP> : (const void*)&dp_apply_kernel<0, CAP>;
  int grid = 0;
  int rc = grid_for(pl, fn, &grid);
  if (rc == GACCUM_OK) {
    grid = std::max(1, std::min(grid, prm->num_tiles));
    void* args[] = {(void*)prm};
    cudaError_t e = cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kThreads), args, 0, st);
    if (e != cudaSuccess) rc = fail(GACCUM_ECUDA, "cudaLaunchCooperativeKernel(dp_apply_kernel) failed: %s", cudaGetErrorString(e));
  }
  delete prm;
  return rc;
}
}  // extern "C++"

int gaccum_apply_dp(gaccum_plan* pl, const gaccum_dp_comm* comm, const float* const* grads, float* m, float* v,
                    const gaccum_step_args* a, uint32_t epoch, gaccum_stream_t stream) {
  if (!comm) return fail(GACCUM_EINVAL, "comm is NULL");
  if (comm->world < 2 || comm->world > GACCUM_MAX_RANKS || comm->rank < 0 || comm->rank >= comm->world)
    return fail(GACCUM_EINVAL, "world must be 2..%d and 0 <= rank < world", GACCUM_MAX_RANKS);
  if (epoch == 0) return fail(GACCUM_EINVAL, "epoch must be non-zero");
  if (int rc = check_args(a)) return rc;
  if (int rc = check_compute(pl, comm->accum, m, v, true)) return rc;
  static_assert(kMaxRanks == GACCUM_MAX_RANKS && kCtrlBytes == GACCUM_DP_CTRL_BYTES, "header and kernel disagree");
  if (comm->stage_elements < stage_span(pl, comm->world) * (comm->world - 1))
    return fail(GACCUM_EINVAL, "staging areas hold %lld elements, gaccum_dp_stage_elements() asks for %lld",
                (long long)comm->stage_elements, (long long)(stage_span(pl, comm->world) * (comm->world - 1)));
  for (int w = 0; w < comm->world; ++w)
    if (!comm->param_peers[w] || !comm->stage_peers[w] || !comm->ctrl_peers[w] ||
        !aligned16_host(comm->param_peers[w]) || !aligned16_host(comm->stage_peers[w]))
      return fail(GACCUM_EINVAL, "peer pointers of rank %d must be non-NULL and 16-byte aligned", w);
  DeviceGuard guard(pl->device);
  cudaStream_t st = (cudaStream_t)stream;
  return pl->T <= kCapSmall ? do_apply_dp<kCapSmall>(pl, comm, grads, m, v, a, epoch, st)
                            : do_apply_dp<kCapLarge>(pl, comm, grads, m, v, a, epoch, st);
}

int gaccum_step_dp(gaccum_plan* pl, const gaccum_dp_comm* comm, const float* const* grads, float* m, float* v,
                   const gaccum_step_args* a, uint32_t epoch, gaccum_stream_t stream) {
  if (!comm) return fail(GACCUM_EINVAL, "comm is NULL");
  if (int rc = check_args(a)) return rc;
  if (!grads) return fail(GACCUM_EINVAL, "grads is NULL");
  if (gaccum_is_apply_step(a->global_step, a->accum_n)) return gaccum_apply_dp(pl, comm, grads, m, v, a, epoch, stream);
  return accumulate_impl(pl, grads, comm->accum, a, stream);      // rank-local: no bytes cross NVLink
}

// ------------------------------------------------------------------------------------------
// host-buffer session
// ------------------------------------------------------------------------------------------
struct gaccum_host_session {
  gaccum_plan* plan = nullptr;
  float *d_params = nullptr, *d_accum = nullptr, *d_m = nullptr, *d_v = nullptr;
  float* d_stage[2] = {nullptr, nullptr};                    // H2D staging of the gradients, double-buffered
  std::vector<const float*> stage_ptrs[2];                   // per-tensor views of the staging slabs (pointer table of the DP kernel)
  cudaStream_t compute = nullptr, h2d = nullptr, d2h = nullptr;
  cudaEvent_t buf_free[2] = {nullptr, nullptr}, h2d_done[2] = {nullptr, nullptr}, k_done = nullptr, d2h_done = nullptr;
  uint64_t calls = 0;
  // data parallel (gaccum_host_session_dp_export / _connect)
  int dp_rank = 0, dp_world = 1;
  float* d_dp_stage = nullptr;                               // this rank's reduce-scatter staging area (peer-written)
  uint32_t* d_dp_ctrl = nullptr;
  int64_t dp_stage_elements = 0;
  gaccum_dp_comm comm{};
  std::vector<void*> ipc_opened;
  uint32_t dp_epoch = 0;
};

// One cudaMemcpyAsync per RUN of tensors whose host addresses are laid out like the device slab (same distance
// between consecutive tensors on both sides, padding included): a caller that keeps its gradients / parameters
// in one pinned arena with the plan's offsets gets a single copy per direction instead of one per tensor
// (each costs ~6 us of copy-engine gap: 73 copies held the link at 44 GB/s, one copy reaches ~55).
extern "C++" {
template <typename HostPtr, typename F>
static int for_each_run(const gaccum_plan* pl, HostPtr const* host, F&& copy /* (t0, host_ptr, dev_offset, elements) -> cudaError_t */) {
  int32_t t = 0;
  while (t < pl->T) {
    if (pl->numel[t] == 0 || !host[t]) { ++t; continue; }
    const int32_t t0 = t;
    int64_t span = pl->numel[t];
    while (t + 1 < pl->T && host[t + 1] && pl->numel[t + 1] > 0 &&
           (const float*)host[t + 1] - (const float*)host[t0] == pl->offset[t + 1] - pl->offset[t0]) {
      ++t;
      span = pl->offset[t] - pl->offset[t0] + pl->numel[t];
    }
    cudaError_t e = copy(t0, host[t0], pl->offset[t0], span);
    if (e != cudaSuccess) return fail(GACCUM_ECUDA, "host<->device copy failed: %s", cudaGetErrorString(e));
    ++t;
  }
  return GACCUM_OK;
}
}  // extern "C++"

int gaccum_host_session_destroy(gaccum_host_session* s) {
  if (!s) return GACCUM_OK;
  if (s->plan && s->plan->device >= 0) {
    DeviceGuard guard(s->plan->device);
    if (s->compute) cudaStreamSynchronize(s->compute);
    if (s->h2d) cudaStreamSynchronize(s->h2d);
    if (s->d2h) cudaStreamSynchronize(s->d2h);
    for (void* p : s->ipc_opened) cudaIpcCloseMemHandle(p);
    cudaFree(s->d_params); cudaFree(s->d_accum); cudaFree(s->d_m); cudaFree(s->d_v);
    cudaFree(s->d_stage[0]); cudaFree(s->d_stage[1]); cudaFree(s->d_dp_stage); cudaFree(s->d_dp_ctrl);
    for (int i = 0; i < 2; ++i) { if (s->buf_free[i]) cudaEventDestroy(s->buf_free[i]); if (s->h2d_done[i]) cudaEventDestroy(s->h2d_done[i]); }
    if (s->k_done) cudaEventDestroy(s->k_done);
    if (s->d2h_done) cudaEventDestroy(s->d2h_done);
    if (s->compute) cudaStreamDestroy(s->compute);
    if (s->h2d) cudaStreamDestroy(s->h2d);
    if (s->d2h) cudaStreamDestroy(s->d2h);
  }
  delete s;
  return GACCUM_OK;
}

int gaccum_host_session_create(gaccum_host_session** out, gaccum_plan* pl) {
  if (!out) return fail(GACCUM_EINVAL, "out is NULL");
  *out = nullptr;
  if (!pl) return fail(GACCUM_EINVAL, "plan is NULL");
  if (pl->device < 0) return fail(GACCUM_ENODEVICE, "layout-only plan (device=-1): libgaccum has no CPU fallback, a CUDA device is required");
  DeviceGuard guard(pl->device);
  gaccum_host_session* s = new (std::nothrow) gaccum_host_session();
  if (!s) return fail(GACCUM_ENOMEM, "out of host memory");
  s->plan = pl;
  const size_t bytes = (size_t)std::max<int64_t>(pl->padded, kSlabAlign) * sizeof(float);
  cudaError_t e = cudaSuccess;
  float** bufs[] = {&s->d_params, &s->d_accum, &s->d_m, &s->d_v, &s->d_stage[0], &s->d_stage[1]};
  for (float** b : bufs) {
    if (e == cudaSuccess) e = cudaMalloc(b, bytes);
    if (e == cudaSuccess) e = cudaMemset(*b, 0, bytes);
  }
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->compute, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->h2d, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->d2h, cudaStreamNonBlocking);
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
    e = cudaEventCreateWithFlags(&s->buf_free[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->h2d_done[i], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->k_done, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->d2h_done, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    gaccum_host_session_destroy(s);
    return fail(GACCUM_ECUDA, "host session setup failed: %s", cudaGetErrorString(e));
  }
  for (int b = 0; b < 2; ++b) {
    s->stage_ptrs[b].resize((size_t)pl->T);
    for (int32_t t = 0; t < pl->T; ++t) s->stage_ptrs[b][t] = s->d_stage[b] + pl->offset[t];
  }
  *out = s;
  return GACCUM_OK;
}

int gaccum_host_session_set_params(gaccum_host_session* s, const float* const* host_params) {
  if (!s || !host_params) return fail(GACCUM_EINVAL, "bad arguments to gaccum_host_session_set_params");
  gaccum_plan* pl = s->plan;
  DeviceGuard guard(pl->device);
  for (int32_t t = 0; t < pl->T; ++t)
    if (pl->numel[t] && !host_params[t]) return fail(GACCUM_EINVAL, "host_params[%d] is NULL", t);
  if (int rc = for_each_run(pl, host_params, [&](int32_t, const float* h, int64_t off, int64_t n) {
        return cudaMemcpyAsync(s->d_params + off, h, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, s->compute);
      })) return rc;
  CUDA_TRY(cudaStreamSynchronize(s->compute));
  return GACCUM_OK;
}

// ---- data parallel over host buffers: every rank's session exports IPC handles of its parameter slab, staging
//      area and control block; the caller exchanges the (plain-byte) records between the ranks with whatever
//      transport it has (MPI, torch.distributed, TF collectives) and hands all of them back ----
int gaccum_host_session_dp_export(gaccum_host_session* s, int32_t world, gaccum_dp_ipc* out) {
  if (!s || !out) return fail(GACCUM_EINVAL, "bad arguments to gaccum_host_session_dp_export");
  if (world < 2 || world > GACCUM_MAX_RANKS) return fail(GACCUM_EINVAL, "world must be 2..%d", GACCUM_MAX_RANKS);
  static_assert(sizeof(cudaIpcMemHandle_t) == GACCUM_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t is 64 bytes");
  gaccum_plan* pl = s->plan;
  DeviceGuard guard(pl->device);
  if (!s->d_dp_stage) {
    s->dp_stage_elements = stage_span(pl, world) * (world - 1);
    CUDA_TRY(cudaMalloc(&s->d_dp_stage, (size_t)s->dp_stage_elements * sizeof(float)));
    CUDA_TRY(cudaMalloc(&s->d_dp_ctrl, GACCUM_DP_CTRL_BYTES));
    CUDA_TRY(cudaMemset(s->d_dp_ctrl, 0, GACCUM_DP_CTRL_BYTES));
    CUDA_TRY(cudaDeviceSynchronize());
  }
  std::memset(out, 0, sizeof *out);
  cudaIpcMemHandle_t h;
  CUDA_TRY(cudaIpcGetMemHandle(&h, s->d_params)); std::memcpy(out->param, &h, sizeof h);
  CUDA_TRY(cudaIpcGetMemHandle(&h, s->d_dp_stage)); std::memcpy(out->stage, &h, sizeof h);
  CUDA_TRY(cudaIpcGetMemHandle(&h, s->d_dp_ctrl)); std::memcpy(out->ctrl, &h, sizeof h);
  out->stage_elements = s->dp_stage_elements;
  out->padded_size = pl->padded;
  return GACCUM_OK;
}

int gaccum_host_session_dp_connect(gaccum_host_session* s, int32_t rank, int32_t world, const gaccum_dp_ipc* all) {
  if (!s || !all) return fail(GACCUM_EINVAL, "bad arguments to gaccum_host_session_dp_connect");
  if (world < 2 || world > GACCUM_MAX_RANKS || rank < 0 || rank >= world) return fail(GACCUM_EINVAL, "world must be 2..%d and 0 <= rank < world", GACCUM_MAX_RANKS);
  if (!s->d_dp_stage) return fail(GACCUM_EINVAL, "call gaccum_host_session_dp_export first");
  gaccum_plan* pl = s->plan;
  DeviceGuard guard(pl->device);
  gaccum_dp_comm c{};
  c.rank = rank; c.world = world; c.accum = s->d_accum; c.stage_elements = s->dp_stage_elements;
  for (int w = 0; w < world; ++w) {
    if (all[w].padded_size != pl->padded || all[w].stage_elements != s->dp_stage_elements)
      return fail(GACCUM_EINVAL, "rank %d exported a different layout (padded %lld vs %lld): all ranks must use the same plan",
                  w, (long long)all[w].padded_size, (long long)pl->padded);
    if (w == rank) { c.param_peers[w] = s->d_params; c.stage_peers[w] = s->d_dp_stage; c.ctrl_peers[w] = s->d_dp_ctrl; continue; }
    void* ptr[3] = {nullptr, nullptr, nullptr};
    const unsigned char* src[3] = {all[w].param, all[w].stage, all[w].ctrl};
    for (int k = 0; k < 3; ++k) {
      cudaIpcMemHandle_t h;
      std::memcpy(&h, src[k], sizeof h);
      cudaError_t e = cudaIpcOpenMemHandle(&ptr[k], h, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) return fail(GACCUM_ECUDA, "cudaIpcOpenMemHandle(rank %d, buffer %d) failed: %s (ranks must be GPUs of one NVLink/PCIe peer domain)", w, k, cudaGetErrorString(e));
      s->ipc_opened.push_back(ptr[k]);
    }
    c.param_peers[w] = (float*)ptr[0]; c.stage_peers[w] = (float*)ptr[1]; c.ctrl_peers[w] = (uint32_t*)ptr[2];
  }
  s->comm = c;
  s->dp_rank = rank; s->dp_world = world;
  return GACCUM_OK;
}

int gaccum_step_host(gaccum_host_session* s, const float* const* host_grads, float* const* host_params_out,
                     const gaccum_step_args* a, gaccum_stats* stats_out) {
  if (!s || !host_grads) return fail(GACCUM_EINVAL, "bad arguments to gaccum_step_host");
  if (int rc = check_args(a)) return rc;
  gaccum_plan* pl = s->plan;
  DeviceGuard guard(pl->device);
  const int b = (int)(s->calls & 1);
  ++s->calls;
  // H2D of this step's gradients into staging buffer b, once the kernel that last read it is done
  CUDA_TRY(cudaStreamWaitEvent(s->h2d, s->buf_free[b], 0));
  if (int rc = for_each_run(pl, host_grads, [&](int32_t, const float* h, int64_t off, int64_t n) {
        return cudaMemcpyAsync(s->d_stage[b] + off, h, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, s->h2d);
      })) return rc;
  for (int32_t t = 0; t < pl->T; ++t)     // tensors without a gradient contribute nothing (optimization.py:132): stage zeros
    if (pl->numel[t] && !host_grads[t])
      CUDA_TRY(cudaMemsetAsync(s->d_stage[b] + pl->offset[t], 0, (size_t)pl->numel[t] * sizeof(float), s->h2d));
  CUDA_TRY(cudaEventRecord(s->h2d_done[b], s->h2d));
  CUDA_TRY(cudaStreamWaitEvent(s->compute, s->h2d_done[b], 0));
  const bool apply = gaccum_is_apply_step(a->global_step, a->accum_n) != 0;
  if (s->dp_world > 1 && apply) {
    // 04:55-62 through host buffers: the fused exchange + apply kernel reads this rank's staged gradients
    if (++s->dp_epoch == 0) s->dp_epoch = 1;
    if (int rc = gaccum_apply_dp(pl, &s->comm, s->stage_ptrs[b].data(), s->d_m, s->d_v, a, s->dp_epoch, s->compute)) return rc;
  } else {
    if (int rc = gaccum_step_packed(pl, s->d_stage[b], s->d_params, s->d_accum, s->d_m, s->d_v, a, -1, s->compute)) return rc;
  }
  CUDA_TRY(cudaEventRecord(s->buf_free[b], s->compute));
  if (stats_out)
    CUDA_TRY(cudaMemcpyAsync(stats_out, pl->d_stats, sizeof(gaccum_stats), cudaMemcpyDeviceToHost, s->compute));
  if (apply && host_params_out) {
    CUDA_TRY(cudaEventRecord(s->k_done, s->compute));
    CUDA_TRY(cudaStreamWaitEvent(s->d2h, s->k_done, 0));
    if (int rc = for_each_run(pl, host_params_out, [&](int32_t, float* h, int64_t off, int64_t n) {
          return cudaMemcpyAsync(h, s->d_params + off, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, s->d2h);
        })) return rc;
    CUDA_TRY(cudaEventRecord(s->d2h_done, s->d2h));
    CUDA_TRY(cudaStreamWaitEvent(s->compute, s->d2h_done, 0));   // the next apply must not overwrite params mid-copy
  }
  return GACCUM_OK;
}

int gaccum_host_session_sync(gaccum_host_session* s) {
  if (!s) return fail(GACCUM_EINVAL, "session is NULL");
  DeviceGuard guard(s->plan->device);
  CUDA_TRY(cudaStreamSynchronize(s->h2d));
  CUDA_TRY(cudaStreamSynchronize(s->compute));
  CUDA_TRY(cudaStreamSynchronize(s->d2h));
  return GACCUM_OK;
}

int gaccum_host_session_slabs(gaccum_host_session* s, float** out) {
  if (!s || !out) return fail(GACCUM_EINVAL, "bad arguments to gaccum_host_session_slabs");
  out[0] = s->d_params; out[1] = s->d_accum; out[2] = s->d_m; out[3] = s->d_v;
  return GACCUM_OK;
}

int gaccum_read_stats(gaccum_plan* pl, gaccum_stats* host_out, gaccum_stream_t stream) {
  if (!pl || !host_out) return fail(GACCUM_EINVAL, "bad arguments to gaccum_read_stats");
  if (pl->device < 0) return fail(GACCUM_ENODEVICE, "layout-only plan has no stats");
  DeviceGuard guard(pl->device);
  CUDA_TRY(cudaMemcpyAsync(host_out, pl->d_stats, sizeof(gaccum_stats), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return GACCUM_OK;
}

}  // extern "C"
