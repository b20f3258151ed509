// te_api.cu - host side of libtraffic_b200.so (C ABI declared in include/traffic_b200.h).
//
// Builds the GridRoad topology tables (reference: gym_traffic/envs/roadgraph.py:26-64),
// owns the device state of num_envs env instances, and launches the kernels in
// te_kernels.cuh.  There is no CPU implementation of the simulation in this library:
// every entry point either runs on the CUDA device or fails.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstddef>
#include <cstring>
#include <atomic>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "../../include/traffic_b200.h"
#include "te_kernels.cuh"

using namespace te;

static thread_local std::string g_err;

static int fail(const char *fmt, ...) __attribute__((format(printf, 1, 2)));
static int fail(const char *fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return -1;
}

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// Owners of CUDA resources (handle members, test hooks): each frees its resource when it goes.
struct DeviceMem {
  static cudaError_t alloc(void **p, size_t bytes) { return cudaMalloc(p, bytes); }
  void operator()(void *p) const { cudaFree(p); }
};
struct PinnedMem {
  static cudaError_t alloc(void **p, size_t bytes) { return cudaHostAlloc(p, bytes, cudaHostAllocDefault); }
  void operator()(void *p) const { cudaFreeHost(p); }
};
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
template <typename T> using dev_buf = std::unique_ptr<T[], DeviceMem>;       // device memory
template <typename T> using pinned_buf = std::unique_ptr<T[], PinnedMem>;    // page-locked host memory
using stream_ptr = std::unique_ptr<CUstream_st, StreamDestroy>;
using event_ptr = std::unique_ptr<CUevent_st, EventDestroy>;

// (Re)allocation of n elements (16 bytes at least); the old buffer is freed first.
template <typename T, typename Mem> static cudaError_t alloc(std::unique_ptr<T[], Mem> &b, size_t n) {
  b.reset();
  void *p = nullptr;
  const cudaError_t e = Mem::alloc(&p, n * sizeof(T) > 0 ? n * sizeof(T) : 16);
  b.reset(e == cudaSuccess ? static_cast<T *>(p) : nullptr);
  return e;
}
static cudaError_t create(stream_ptr &s) {
  cudaStream_t raw = nullptr;
  const cudaError_t e = cudaStreamCreateWithFlags(&raw, cudaStreamNonBlocking);
  s.reset(e == cudaSuccess ? raw : nullptr);
  return e;
}
static cudaError_t create(event_ptr &ev, unsigned flags = cudaEventDisableTiming) {
  cudaEvent_t raw = nullptr;
  const cudaError_t e = cudaEventCreateWithFlags(&raw, flags);
  ev.reset(e == cudaSuccess ? raw : nullptr);
  return e;
}

// A staging buffer replaced by one of n elements (zeroed when asked) once the device is idle: steps queued on other
// streams may still use the old one.
template <typename Buf> static int grow(Buf &b, size_t n, bool zero = false) {
  CU(cudaDeviceSynchronize());
  CU(alloc(b, n));
  if (zero) CU(cudaMemset(b.get(), 0, n * sizeof(*b.get())));
  return 0;
}

// ---- host side of the wire format (te_kernels.cuh: wire_layout): expand compact env records into the caller's
// float observation / reward / done arrays (te_host.cpp).  The work is memory-bound and overlapped with the simulation
// of the following slices (ExpandPool).
void te_expand_records_host(const unsigned char *recs, const te_wire_layout_t &wl, int r, int I, long long n, float *obs,
                            float *reward, uint8_t *done);   // te_host.cpp

// A few helper threads per handle that wait for a slice's device-to-host copy (CUDA event) and expand it while the
// GPU simulates the next slices.  Slices are dealt round-robin; the calling thread takes its share too.
struct ExpandJob {
  const unsigned char *recs; float *obs, *reward; uint8_t *done;
  const uint8_t *mask;           // nullable (host pointer): only envs with a non-zero byte were stepped
  te_wire_layout_t wl;
  int r, I, nslice, per, E, nsteps;
  const event_ptr *copied;
};
struct ExpandPool {
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv_go, cv_done;
  ExpandJob job;
  unsigned long long generation = 0;
  int pending = 0, device = 0, nthreads = 1;
  bool stop = false;
  std::atomic<int> failed{0};

  void run_share(const ExpandJob &j, int tid) {
    for (int k = tid; k < j.nslice; k += nthreads) {
      if (cudaEventSynchronize(j.copied[k].get()) != cudaSuccess) { failed.store(1); continue; }
      const int e0 = k * j.per, ne = std::min(j.per, j.E - e0);
      if (ne <= 0) continue;
      const int ol = 2 * j.r + j.I;
      for (int st = 0; st < j.nsteps; st++) {
        const size_t eo = (size_t)st * j.E + e0;       // [nsteps][E] env slots
        if (!j.mask) {
          te_expand_records_host(j.recs + eo * j.wl.stride, j.wl, j.r, j.I, ne, j.obs + eo * ol, j.reward + eo * j.I, j.done + eo);
        } else {
          for (int e = 0; e < ne; e++)
            if (j.mask[e0 + e])
              te_expand_records_host(j.recs + (eo + e) * j.wl.stride, j.wl, j.r, j.I, 1, j.obs + (eo + e) * ol, j.reward + (eo + e) * j.I, j.done + eo + e);
        }
      }
    }
  }
  void start(int dev, int n) {
    device = dev; nthreads = n < 1 ? 1 : n;
    for (int t = 1; t < nthreads; t++)
      workers.emplace_back([this, t]() {
        cudaSetDevice(device);
        unsigned long long seen = 0;
        for (;;) {
          ExpandJob j;
          {
            std::unique_lock<std::mutex> lk(mu);
            cv_go.wait(lk, [&] { return stop || generation != seen; });
            if (stop) return;
            seen = generation; j = job;
          }
          run_share(j, t);
          { std::lock_guard<std::mutex> lk(mu); if (--pending == 0) cv_done.notify_all(); }
        }
      });
  }
  // called by the stepping thread once every slice's kernel and copy have been queued
  bool run(const ExpandJob &j) {
    failed.store(0);
    { std::lock_guard<std::mutex> lk(mu); job = j; pending = nthreads - 1; generation++; }
    cv_go.notify_all();
    run_share(j, 0);
    { std::unique_lock<std::mutex> lk(mu); cv_done.wait(lk, [&] { return pending == 0; }); }
    return failed.load() == 0;
  }
  ~ExpandPool() {
    { std::lock_guard<std::mutex> lk(mu); stop = true; }
    cv_go.notify_all();
    for (std::thread &t : workers) t.join();
  }
};

struct StepVariant;

// Members go in reverse order of declaration: the helper threads stop before the page-locked records they read are
// freed, and every event and buffer goes before the streams.
struct te_handle {
  te_config cfg = {};
  int V = 0, r = 0, R = 0, Rp = 0, I = 0, n_entry = 0;
  int device = 0;
  stream_ptr stream, stream2, stream_copy;
  event_ptr ev0, ev1, ev_fork, ev_join, ev_copied, ev_slice[64], ev_copy[64];
  bool timed = false;
  StepParams base = {};  // everything except per-call pointers
  std::vector<int> dest, nexts, phases, entry;
  // device buffers
  dev_buf<float> x, v;
  dev_buf<int> elapsed;
  dev_buf<uint8_t> phase, passed_dst;
  dev_buf<EnvScalars> env;
  dev_buf<DeviceStats> stats;
  dev_buf<short> d_nexts, d_up;
  dev_buf<signed char> d_entry_idx;
  dev_buf<long long> d_sched_off;
  dev_buf<short> d_sched_roads;
  dev_buf<uint32_t> d_gap_cdf;
  // staging for TE_HOST calls
  dev_buf<uint8_t> d_actions, d_done, d_mask, d_init_phase;
  dev_buf<float> d_reward;
  dev_buf<int> d_obs_i, d_cars;   // d_obs_i: raw observations, or (read as float) fused ones: never live together
  dev_buf<float> w; dev_buf<TripRecord> d_trips; dev_buf<unsigned long long> d_trip_count; long long trip_cap = 0;
  int warps = 0;
  int G = 1, threads = 0;        // env instances per CTA, threads per CTA (G * R rounded up to whole warps)
  const StepVariant *sv = nullptr;   // the step kernel the handle runs now (select_layout)
  te_step_variant_t plan = {};       // the same, as te_get_step_variant reports it
  int smem_optin = 0;
  // wire path of the host API
  dev_buf<unsigned char> d_wire; pinned_buf<unsigned char> h_wire;   // [steps][E][wire_stride] device / page-locked host
  int wire_stride = 0, host_slices = 1;
  int wire_steps = 1, float_steps = 1;   // actor steps the wire records / float staging have room for
  // masked steps on the float route: page-locked [nsteps][E] obs | reward | done, of which only the stepped envs' rows
  // are copied to the caller (launch_sliced)
  pinned_buf<unsigned char> h_float; int h_float_steps = 0;
  bool tame = false;     // every car the device has seen is tame (te_math.cuh: idm_update<TAME = true> may run)
  float v_cap = 0.f;     // speed bound of the tame domain for this archetype (tame_archetype)
  int ctrl_spacing = 0;  // TE_CTRL_GREEDY: a new decision every so many actor steps inside a te_step_multi launch (0: one per launch)
  int actions_cap = 1;   // decisions d_actions has room for
  bool float_dma = false;  // te_step(TE_HOST) with float outputs: let the copy engine write the float arrays (no host expansion)
  // snapshot records (te_save_envs / te_load_envs, and te_get_state / te_set_state through them): device staging of host
  // records, and the check pass's status word
  dev_buf<unsigned char> d_snap; size_t snap_cap = 0;
  dev_buf<SnapStatus> d_snap_status;
  std::unique_ptr<ExpandPool> pool;
  ~te_handle() { cudaSetDevice(device); }
};

// One thread per (padded) road.  A kernel variant is compiled per row capacity MAXT >= Rp (its shared-memory layout
// is a compile-time function of MAXT); the register cap follows from the CTA size and the number of CTAs an SM
// should hold: 1024 resident threads per SM at 64 registers wherever shared memory allows it (10x10 grid: 512 threads
// x 2 CTAs, 101.7 KB each; 3x3 grid: 64 threads x 16 CTAs).
typedef void (*step_kernel_t)(const StepParams);
// te_step_kernel<MAXT, MINB, VALIDATE, TAME, GROUPED>: MAXT rows, MINB CTAs per SM for the register cap; TAME = the car
// loop compiled in the tame form (runs_tame_form); GROUPED = several env instances per CTA (small grids with the
// reference's archetype, plan_layout).
struct StepVariant { step_kernel_t fn; int maxt, minb; bool validate, tame, grouped; };
#define TE_STEP_VARIANT(MAXT, MINB, VALIDATE, TAME, GROUPED) \
  {te_step_kernel<MAXT, MINB, VALIDATE, TAME, GROUPED>, MAXT, MINB, VALIDATE, TAME, GROUPED}
// The 19 instantiations of the step kernel (te_step_variants), in increasing MAXT within each kind: the set is kept
// small for the sake of build time.
static const StepVariant STEP_VARIANTS[] = {
    // validate: + the birth-tick plane in shared memory, one CTA fewer per SM
    TE_STEP_VARIANT(256, 2, true, false, false), TE_STEP_VARIANT(512, 1, true, false, false),
    TE_STEP_VARIANT(768, 1, true, false, false),
    // grouped (only built in the tame form: plan_layout keeps G = 1 otherwise).  Default 3x3 grid: two envs (2 x 48 roads)
    // on three warps, 20 envs per SM at 64 registers (72 registers and 9 CTAs per SM measured 2.4 % slower).  No grid
    // yields 97..128 threads at G > 1, so those would run the 160 variant.
    TE_STEP_VARIANT(64, 16, false, true, true), TE_STEP_VARIANT(96, 10, false, true, true),
    TE_STEP_VARIANT(160, 6, false, true, true), TE_STEP_VARIANT(256, 4, false, true, true),
    // tame, one env per CTA
    TE_STEP_VARIANT(64, 16, false, true, false), TE_STEP_VARIANT(128, 8, false, true, false),
    TE_STEP_VARIANT(256, 4, false, true, false), TE_STEP_VARIANT(512, 2, false, true, false),
    TE_STEP_VARIANT(768, 1, false, true, false), TE_STEP_VARIANT(1024, 1, false, true, false),
    // checked: per-car validity predicate and generic fallback
    TE_STEP_VARIANT(64, 16, false, false, false), TE_STEP_VARIANT(128, 8, false, false, false),
    TE_STEP_VARIANT(256, 4, false, false, false), TE_STEP_VARIANT(512, 2, false, false, false),
    TE_STEP_VARIANT(768, 1, false, false, false), TE_STEP_VARIANT(1024, 1, false, false, false),
};
#undef TE_STEP_VARIANT
static constexpr int NUM_STEP_VARIANTS = (int)(sizeof(STEP_VARIANTS) / sizeof(STEP_VARIANTS[0]));
// The smallest variant of the kind with room for `threads` rows, else the largest of the kind (the caller compares
// `threads` with its maxt).  Validate variants are neither tame nor grouped; grouped ones are tame.
static const StepVariant &step_variant_for(int threads, bool validate, bool tame, bool grouped) {
  if (validate) tame = grouped = false;
  if (grouped) tame = true;
  const StepVariant *last = nullptr;
  for (const StepVariant &v : STEP_VARIANTS) {
    if (v.validate != validate || v.tame != tame || v.grouped != grouped) continue;
    if (threads <= v.maxt) return v;
    last = &v;
  }
  return *last;
}
// The double literals of the IDM update live in constant memory (te_math.cuh: g_mc); one upload per device.
static cudaError_t upload_math_consts() {
  const MathConsts m = math_consts_host();
  return cudaMemcpyToSymbol(g_mc, &m, sizeof(m));
}

// IdmConst from the archetype and the tick length (one place: te_create and the test hooks)
static bool is_pow2_f(float f) {
  int e = 0;
  return f > 0.f && std::isfinite(f) && frexpf(f, &e) == 0.5f && e >= -19 && e <= 21;   // 2^-20 .. 2^20
}
static void fill_idm(IdmConst &c, const float *a, float rate) {
  c.rate = rate; c.x_new = a[0]; c.v_new = a[1]; c.len = a[2]; c.a = a[3]; c.delta = a[4]; c.v0 = a[5]; c.T = a[7]; c.s0 = a[8];
  { volatile float ab = a[3] * a[6]; c.two_sqrt_ab = (double)sqrtf(ab) * 2.0; }  // traffic_env.py:54
  c.rcp_two_sqrt_ab = 1.0 / c.two_sqrt_ab;
  c.v0_d = (double)a[5]; c.rcp_v0 = 1.0 / (double)a[5];
  c.s0_d = (double)a[8]; c.a_d = (double)a[3]; c.rate_d = (double)rate; c.delta_d = (double)a[4];
  c.delta_is_four = (a[4] == 4.0f) && !getenv("TE_NO_POWF4_SHORTCUT");
  c.half_rate_d = 0.5 * (double)rate; c.s0_z = (float)(0.0 + (double)a[8]);
  c.T_d = (double)a[7];
  c.pow2 = is_pow2_f(a[7]) && is_pow2_f(rate) && !getenv("TE_NO_POW2_SHORTCUT");
}

// The one rule for which form of the IDM update runs (te_math.cuh: idm_update<TAME>).  The tame kernels are compiled for
// the reference's archetype AND without the per-car validity predicate: they may only run while the handle (or, for the
// test hooks, the archetype) is tame.
static bool runs_tame_form(const IdmConst &c, bool tame) { return c.pow2 && c.delta_is_four && tame; }

// Archetype ranges under which tame car state stays tame and every fast sequence of idm_update is exact (te_math.cuh).
// *v_cap = the speed bound of the tame domain for this archetype: twice the fastest speed the dynamics can produce
// (v' <= max(v, v0 + a rate)), and at least the speed cars arrive with.  Closure needs the float dv = a (1 - p - q^2) to stay
// finite (an infinite dv makes x NaN in the reference's arithmetic, and NaN state is not tame): q = s_star / (s + 1e-8)
// is largest when the float gap s is -RN_f32(1e-8), where |s + 1e-8| = 6.08e-17, and s_star <= s0 + v T + v^2 / (2 sqrt(a b)).
static bool tame_archetype(const te_config *cfg, float *v_cap) {
  const float *a = cfg->archetype;
  auto in = [](double v, double lo, double hi) { return std::isfinite(v) && v >= lo && v <= hi; };
  const double tiny = ldexp(1.0, -10), big = ldexp(1.0, 19);
  *v_cap = 0.f;
  // (x_new = -0: cars would enter at a position tame_car (te_kernels.cuh) rejects)
  if (!(in(a[0], -ldexp(1.0, 30), ldexp(1.0, 30)) && !(a[0] == 0.f && std::signbit(a[0])) &&
        (a[1] == 0.f || in(a[1], tiny, big)) && in(a[2], 0.0, big) && in(a[3], tiny, big) && in(a[4], tiny, 64.0) && in(a[5], tiny, big) && in(a[6], tiny, big) && in(a[7], tiny, big) &&
        in(a[8], tiny, big) && in(cfg->rate, tiny, 1024.0) && in(cfg->length, tiny, ldexp(1.0, 30))))
    return false;
  const double cap = 2.0 * std::max((double)a[1], (double)a[5] + (double)a[3] * cfg->rate);
  if (!(cap < big)) return false;
  const double den_min = fabs((double)(float)1e-8 - 1e-8);
  const double s_star_max = 1.01 * ((double)a[8] + cap * a[7] + cap * cap / (2.0 * sqrt((double)a[3] * a[6])));
  const double q_max = s_star_max / den_min;
  if (!((double)a[3] * (q_max * q_max + pow(cap / a[5], (double)a[4]) + 1.0) < ldexp(1.0, 126))) return false;
  *v_cap = (float)cap;
  return true;
}
static int select_layout(te_handle *h);

extern "C" const char *te_last_error(void) { return g_err.c_str(); }

extern "C" int te_device_count(int32_t *count) {
  if (!count) return fail("te_device_count: null argument");
  int n = 0;
  const cudaError_t e = cudaGetDeviceCount(&n);
  *count = (e == cudaSuccess) ? n : 0;
  if (e != cudaSuccess) { (void)cudaGetLastError(); return fail("te_device_count: %s", cudaGetErrorString(e)); }
  return 0;
}

extern "C" void te_default_config(te_config *c) {
  memset(c, 0, sizeof(*c));
  c->struct_size = (int32_t)sizeof(te_config);
  c->m = 3; c->n = 3; c->length = 250.f; c->rate = 0.5f;   // traffic_test.py:80, traffic_env.py:12
  c->num_envs = 1; c->env_id_base = 0; c->device = 0;
  c->flags = TE_REMI;                                     // traffic_test.py:17 (--remi True)
  c->entry_spec = 0;                                      // FLAGS.entry == 'all', traffic_env.py:392
  c->arrival_mode = TE_ARRIVALS_PHILOX;
  c->cars_per_tick = 0.12 * 3 * 4 * 0.5;                  // local_cars_per_sec * m * inv_popcount(0) * rate
  c->seed = 0; c->episode_len = 0; c->gamma = 0.8f;       // alg_flags.py:13
  const float arch[TE_PARAMS] = {0.f, 11.11f, 4.f, 3.f, 4.f, 13.89f, 6.f, 2.f, 1.f, 0.f};  // traffic_env.py:35-43
  memcpy(c->archetype, arch, sizeof(arch));
}

// roadgraph.py:54-64
static int grid_next(int i, int m, int n) {
  const int v = m * n;
  if (i >= 4 * v) return -1;
  const int col = i % n, row = (i % v) / n;
  if (i < v) return col < n - 1 ? i + 1 : 4 * v + n + row;
  if (i < 2 * v) return col > 0 ? i - 1 : 4 * v + 2 * n + m + row;
  if (i < 3 * v) return row < m - 1 ? i + n : 4 * v + n + m + col;
  return row > 0 ? i - n : 4 * v + col;
}

// Thresholds T[k] = floor(2^32 * P(round(Exp(scale)) <= k)), scale = 1 / cars_per_tick ticks.
// round() is Python's round-half-even; ties have measure zero, so P(gap <= k) = 1 - exp(-(k + 0.5) / scale).
// Built on the host in double and shared verbatim with the CPU oracle (traffic_env_b200/arrivals.py builds
// the same table for tests), so no transcendental is evaluated on the device.
static std::vector<uint32_t> build_gap_cdf(double cars_per_tick) {
  std::vector<uint32_t> t;
  if (!(cars_per_tick > 0)) return t;
  for (int k = 0; k < 8192; k++) {
    const double cdf = -expm1(-(k + 0.5) * cars_per_tick);
    const double scaled = floor(cdf * 4294967296.0);
    if (scaled >= 4294967295.0) break;
    t.push_back((uint32_t)scaled);
  }
  return t;
}

extern "C" int te_destroy(te_handle *h) { delete h; return 0; }

// Rows of one env in HBM and in a one-env CTA: R roads padded to whole warps, or to whole groups of four warps when that
// costs at most 20 % more rows.  Whole groups of four warps keep the SM's four schedulers evenly loaded (a 14-warp CTA
// puts 4, 4, 3, 3 warps on them; two such CTAs 8, 8, 6, 6).  10x10 grid: 440 roads -> 512 threads, 16 warps, 64
// registers: +1.7 % (measured A/B, 3 runs each).
static int padded_rows(int R) {
  const int rp32 = (R + GROUP_ROADS - 1) / GROUP_ROADS * GROUP_ROADS, rp128 = (R + 127) / 128 * 128;
  return rp128 * 5 <= R * 6 ? rp128 : rp32;
}

// The configurations te_create accepts, apart from the device: physically sensible ones only (bit-parity with the
// reference is established for these): finite positive tick length, road length, desired speed, acceleration and
// braking; and a road longer than twice the farthest a car can travel in one tick, so that a car handed to the next road
// cannot leave that road in the same tick (the reference's sequential road loop could pop it again; the parallel
// transfer phase does not).
static int check_config(const te_config *cfg, const char *who) {
  if (cfg->struct_size != (int32_t)sizeof(te_config)) return fail("%s: te_config size mismatch (%d vs %zu)", who, cfg->struct_size, sizeof(te_config));
  if (cfg->m < 1 || cfg->n < 1 || cfg->num_envs < 1) return fail("%s: bad dimensions", who);
  const float *a = cfg->archetype;
  auto pos = [](float f) { return std::isfinite(f) && f > 0.f; };
  if (!pos(cfg->rate) || !pos(cfg->length)) return fail("%s: rate and length must be finite and positive", who);
  if (!pos(a[5]) || !pos(a[3]) || !pos(a[6]) || !pos(a[4]) || !pos(a[7]))
    return fail("%s: archetype v0, a, b, delta and T must be finite and positive", who);
  for (int i = 0; i < TE_PARAMS; i++) if (!std::isfinite(a[i])) return fail("%s: archetype[%d] is not finite", who, i);
  if (a[1] < 0.f || a[2] < 0.f || a[8] < 0.f) return fail("%s: archetype v, l and s0 must be non-negative", who);
  const double vmax = std::max((double)a[5] + (double)a[3] * cfg->rate, (double)a[1]);
  const double max_disp = cfg->rate * vmax + 0.5 * (double)a[3] * cfg->rate * cfg->rate;
  if ((double)cfg->length <= 2.0 * max_disp)
    return fail("%s: road length %.3f is not above twice the maximum displacement per tick (%.3f)", who, cfg->length, max_disp);
  return 0;
}

// The one place that decides the CTA layout and the step kernel of a configuration (select_layout, te_plan_step_variant).
// tame: every car the handle has seen is tame (tame_archetype, and no wild car loaded).  Touches no device.
// One thread per road.  Small grids put G env instances on one CTA (its rows are the G * R roads of those envs) so that no
// lane is a padding lane and a warp's car list is long: G in 1..4 with at most 256 rows, chosen for the fewest padding
// lanes (ties: the smaller G).  Default 3x3 grid: R = 48 -> G = 2, 96 threads, three warps.  Large grids: G = 1, the CTA
// padded like the HBM rows (padded_rows).
static int plan_layout(const te_config *cfg, bool tame, const char *who, te_step_variant_t *out, const StepVariant **sv_out) {
  if (cfg->m > 1024 || cfg->n > 1024) return fail("%s: a %d x %d grid exceeds one CTA (max 1024 roads)", who, cfg->m, cfg->n);
  const int R = 4 * cfg->m * cfg->n + 2 * cfg->n + 2 * cfg->m, Rp = padded_rows(R);
  if (Rp > 1024) return fail("%s: %d roads exceed one CTA (max 1024)", who, Rp);
  IdmConst c = {};
  fill_idm(c, cfg->archetype, cfg->rate);
  const bool validate = (cfg->flags & TE_VALIDATE) != 0, tame_form = runs_tame_form(c, tame);
  int G = 1, threads = Rp;
  if (!validate && R < 128 && tame_form) {
    double best = (double)(Rp - R) / Rp;
    for (int g = 2; g <= 4 && g * R <= 256; g++) {
      const int th = (g * R + 31) / 32 * 32;
      const double waste = (double)(th - g * R) / th;
      if (waste < best - 1e-9) { best = waste; G = g; threads = th; }
    }
  }
  const StepVariant &sv = step_variant_for(threads, validate, tame_form, G > 1);
  if (threads > sv.maxt)
    return fail("%s: %d roads exceed the largest%s kernel variant (te_step_kernel<%d, %d, %s>)", who, threads,
                validate ? " validate-mode" : "", sv.maxt, sv.minb, validate ? "validate" : sv.tame ? "tame" : "checked");
  *out = {sv.maxt, sv.minb, sv.validate, sv.tame, sv.grouped, R, Rp, G, threads};
  if (sv_out) *sv_out = &sv;
  return 0;
}

// Threads per CTA, env instances per CTA and the kernel variant of a handle; called by te_create and again when a
// handle stops being tame (a wild car in loaded records, load_records: the checked, one-env-per-CTA kernels take over).
static int select_layout(te_handle *h) {
  const StepVariant *sv = nullptr;
  if (int rc = plan_layout(&h->cfg, h->tame, "te_create", &h->plan, &sv)) return rc;
  h->sv = sv; h->G = h->plan.envs_per_cta; h->threads = h->plan.threads;
  h->warps = h->threads / GROUP_ROADS;
  h->base.G = h->G;
  CU(cudaDeviceGetAttribute(&h->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
  const int smem_max = smem_bytes(sv->maxt, sv->validate, MAX_K, h->n_entry, h->G);
  if (smem_max > h->smem_optin) { return fail("te_create: env needs %d B of shared memory, device allows %d", smem_max, h->smem_optin); }
  CU(cudaFuncSetAttribute(sv->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
  return 0;
}

extern "C" int te_step_variants(te_step_variant_t *out, int32_t cap, int32_t *count) {
  if (!count || cap < 0 || (cap > 0 && !out)) return fail("te_step_variants: bad argument");
  for (int i = 0; i < NUM_STEP_VARIANTS && i < cap; i++) {
    const StepVariant &v = STEP_VARIANTS[i];
    out[i] = {v.maxt, v.minb, v.validate, v.tame, v.grouped, 0, 0, 0, 0};
  }
  *count = NUM_STEP_VARIANTS;
  return 0;
}

extern "C" int te_plan_step_variant(const te_config *cfg, int32_t wild, te_step_variant_t *out) {
  if (!cfg || !out) return fail("te_plan_step_variant: null argument");
  if (int rc = check_config(cfg, "te_plan_step_variant")) return rc;
  float v_cap = 0.f;
  const bool tame = tame_archetype(cfg, &v_cap) && !wild;
  return plan_layout(cfg, tame, "te_plan_step_variant", out, nullptr);
}

extern "C" int te_get_step_variant(const te_handle *h, te_step_variant_t *out) {
  if (!h || !out) return fail("te_get_step_variant: null argument");
  *out = h->plan;
  return 0;
}

extern "C" int te_create(const te_config *cfg, te_handle **out) {
  if (!cfg || !out) return fail("te_create: null argument");
  if (int rc = check_config(cfg, "te_create")) return rc;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail("te_create: no CUDA device (%s); this library has no CPU path", cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail("te_create: device %d out of range", cfg->device);
  std::unique_ptr<te_handle> owner(new te_handle());   // frees whatever was set up when te_create fails
  te_handle *h = owner.get();
  h->cfg = *cfg; h->device = cfg->device;
  CU(cudaSetDevice(h->device));
  CU(upload_math_consts());
  const int m = cfg->m, n = cfg->n;
  h->V = m * n; h->I = h->V; h->r = 4 * h->V; h->R = h->r + 2 * n + 2 * m;
  h->Rp = padded_rows(h->R);
  // topology (roadgraph.py:35-39, 42-51)
  h->dest.resize(h->R); h->nexts.resize(h->R); h->phases.resize(h->R);
  std::vector<short> nx(h->Rp, -1), up(h->Rp, -1);
  std::vector<signed char> eidx(h->Rp, -1);
  for (int i = 0; i < h->R; i++) {
    h->phases[i] = (i / h->V) < 2;
    h->dest[i] = i < 4 * h->V ? i % h->V : -1;
    h->nexts[i] = grid_next(i, m, n);
    nx[i] = (short)h->nexts[i];
  }
  for (int i = 0; i < h->R; i++) if (h->nexts[i] >= 0) {
    if (up[h->nexts[i]] != -1) return fail("te_create: successor table is not injective");
    up[h->nexts[i]] = (short)i;
  }
  const uint32_t spec = cfg->entry_spec;
  const int v = h->V;
  if ((spec & 1) == 0) for (int i = 0; i < m; i++) h->entry.push_back(n * i);
  if (((spec >> 1) & 1) == 0) for (int i = 1; i <= m; i++) h->entry.push_back(v + n * i - 1);
  if (((spec >> 2) & 1) == 0) for (int i = 0; i < n; i++) h->entry.push_back(2 * v + i);
  if (((spec >> 3) & 1) == 0) for (int i = 0; i < n; i++) h->entry.push_back(3 * v + n * (m - 1) + i);
  h->n_entry = (int)h->entry.size();
  if (h->n_entry > 127) return fail("te_create: more than 127 entry roads");
  for (int k = 0; k < h->n_entry; k++) eidx[h->entry[k]] = (signed char)k;

  const size_t E = (size_t)cfg->num_envs;
  CU(create(h->stream)); CU(create(h->stream2)); CU(create(h->stream_copy));
  CU(create(h->ev_copied));
  for (event_ptr &e : h->ev_slice) CU(create(e));
  for (event_ptr &e : h->ev_copy) CU(create(e));
  CU(create(h->ev0, cudaEventDefault)); CU(create(h->ev1, cudaEventDefault));
  CU(create(h->ev_fork)); CU(create(h->ev_join));
  CU(alloc(h->x, E * h->Rp * CAP)); CU(alloc(h->v, E * h->Rp * CAP));
  if (cfg->flags & TE_VALIDATE) {
    CU(alloc(h->w, E * h->Rp * CAP));
    CU(cudaMemset(h->w.get(), 0, E * h->Rp * CAP * sizeof(float)));
    h->trip_cap = std::max<long long>(1ll << 20, 64ll * (long long)E);
    CU(alloc(h->d_trips, (size_t)h->trip_cap)); CU(alloc(h->d_trip_count, 1));
    CU(cudaMemset(h->d_trip_count.get(), 0, sizeof(unsigned long long)));
  }
  CU(alloc(h->elapsed, E * h->I)); CU(alloc(h->phase, E * h->I)); CU(alloc(h->passed_dst, E * h->I));
  CU(alloc(h->env, E)); CU(alloc(h->stats, 1));
  CU(alloc(h->d_nexts, (size_t)h->Rp)); CU(alloc(h->d_up, (size_t)h->Rp));
  CU(alloc(h->d_entry_idx, (size_t)h->Rp));
  CU(alloc(h->d_actions, E * h->I)); CU(alloc(h->d_done, E)); CU(alloc(h->d_mask, E));
  CU(alloc(h->d_init_phase, E * h->I));
  CU(alloc(h->d_obs_i, E * (2 * h->r + 2 * h->I)));
  CU(alloc(h->d_reward, E * h->I));
  h->wire_stride = wire_layout(h->r, h->I).stride;
  CU(alloc(h->d_wire, E * (size_t)h->wire_stride));
  CU(alloc(h->h_wire, E * (size_t)h->wire_stride));
  {
    // Host path: the batch is launched in slices (te_step, TE_HOST) and a few helper threads expand the compact
    // records of finished slices into the caller's float arrays meanwhile.  TE_HOST_SLICES / TE_HOST_THREADS tune it.
    int nslice = cfg->num_envs / 512;              // measured on the 16384-env workload: 4 / 8 / 16 / 32 / 64 slices
    nslice = nslice < 1 ? 1 : (nslice > 32 ? 32 : nslice);  //   -> 1.10 / 1.16 / 1.20 / 1.22 / 1.17e11 vehicle-updates/s end to end
    if (const char *ev = getenv("TE_HOST_SLICES")) { const int v = atoi(ev); if (v >= 1 && v <= 64) nslice = v; }
    h->host_slices = nslice;
    int nthr = 4;
    const unsigned hw = std::thread::hardware_concurrency();
    if (hw && hw < 8) nthr = 2;
    if ((size_t)cfg->num_envs * (size_t)(2 * h->r) < (1u << 20)) nthr = 1;   // small batches: not worth waking anybody
    if (const char *ev = getenv("TE_HOST_THREADS")) { const int v = atoi(ev); if (v >= 1 && v <= 64) nthr = v; }
    if (nthr > nslice) nthr = nslice;
    h->pool.reset(new ExpandPool());
    h->pool->start(h->device, nthr);
    // Float outputs in host memory can travel two ways: as wire records expanded by the helper threads (fewer PCIe
    // bytes; needs ~4 spare cores per GPU: measured 0.91 of the device rate on a 16-core / 1-GPU box, 0.51 with 8 ranks
    // on 32 cores) or as float arrays written by the copy engine (r1 scheme: no host work, 2.5 x the PCIe bytes: 0.90 /
    // 0.73).  Default: expansion when the host has at least 8 hardware threads per visible GPU.  TE_HOST_FLOAT_DMA = 0 / 1
    // overrides.  (te_step_wire never expands: 0.97 with 8 ranks.)
    h->float_dma = hw && ndev > 0 && hw / (unsigned)ndev < 8;
    if (const char *ev = getenv("TE_HOST_FLOAT_DMA")) h->float_dma = atoi(ev) != 0;
  }
  CU(cudaMemcpy(h->d_nexts.get(), nx.data(), nx.size() * sizeof(short), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_up.get(), up.data(), up.size() * sizeof(short), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_entry_idx.get(), eidx.data(), eidx.size(), cudaMemcpyHostToDevice));
  CU(cudaMemset(h->stats.get(), 0, sizeof(DeviceStats)));
  CU(cudaMemset(h->x.get(), 0, E * h->Rp * CAP * sizeof(float)));
  CU(cudaMemset(h->v.get(), 0, E * h->Rp * CAP * sizeof(float)));
  CU(cudaMemset(h->elapsed.get(), 0, E * h->I * sizeof(int)));
  CU(cudaMemset(h->phase.get(), 0, E * h->I)); CU(cudaMemset(h->passed_dst.get(), 0, E * h->I));
  CU(cudaMemset(h->d_done.get(), 0, E));

  std::vector<uint32_t> cdf = build_gap_cdf(cfg->cars_per_tick);
  if (cfg->arrival_mode == TE_ARRIVALS_PHILOX && (cdf.empty() || h->n_entry == 0)) {
    return fail("te_create: Philox arrivals need cars_per_tick > 0 and at least one entry road");
  }
  if (cfg->arrival_mode == TE_ARRIVALS_PHILOX && cfg->cars_per_tick > 16.0 * h->n_entry) {
    // per-tick per-road arrival counts are 8-bit; a ring holds 18 cars anyway
    return fail("te_create: cars_per_tick %.1f is beyond what %d entry roads can take", cfg->cars_per_tick, h->n_entry);
  }
  CU(alloc(h->d_gap_cdf, cdf.size()));
  if (!cdf.empty()) CU(cudaMemcpy(h->d_gap_cdf.get(), cdf.data(), cdf.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));

  // per-env scalars; the Philox stream draws its first gap at seeding time, like poisson() does on first next()
  std::vector<EnvScalars> es(E);
  for (size_t i = 0; i < E; i++) {
    memset(&es[i], 0, sizeof(EnvScalars));
    es[i].ep_mult = 1.0;
  }
  CU(cudaMemcpy(h->env.get(), es.data(), E * sizeof(EnvScalars), cudaMemcpyHostToDevice));

  StepParams &p = h->base;
  p.V = h->V; p.r = h->r; p.R = h->R; p.Rp = h->Rp; p.I = h->I; p.n_entry = h->n_entry;
  p.num_envs = cfg->num_envs; p.length = cfg->length;
  {
    const double det_thr = (double)cfg->length - 10.0;
    float f = (float)det_thr;                         // round to nearest, then step down if that went above
    if ((double)f > det_thr) f = nextafterf(f, -INFINITY);
    p.det_thr_f = f;
  }
  p.flags = cfg->flags; p.arrival_mode = cfg->arrival_mode; p.K = 1; p.raw = 0; p.episode_len = cfg->episode_len;
  p.gamma = cfg->gamma;
  fill_idm(p.idm, cfg->archetype, cfg->rate);
  h->tame = tame_archetype(cfg, &h->v_cap);
  p.x = h->x.get(); p.v = h->v.get(); p.w = h->w.get(); p.trips = h->d_trips.get(); p.trip_count = h->d_trip_count.get(); p.trip_cap = h->trip_cap;
  p.elapsed = h->elapsed.get(); p.phase = h->phase.get(); p.passed_dst = h->passed_dst.get();
  p.env = h->env.get(); p.stats = h->stats.get(); p.nexts = h->d_nexts.get(); p.up = h->d_up.get(); p.entry_idx = h->d_entry_idx.get();
  p.gap_cdf = h->d_gap_cdf.get(); p.n_gap = (int)cdf.size();
  p.seed = (uint32_t)(cfg->seed ^ (cfg->seed >> 32)); p.env_id_base = cfg->env_id_base;
  p.sched_off = nullptr; p.sched_roads = nullptr; p.horizon = 0; p.sched_first = 0;
  p.nsteps = 1; p.controller = CTRL_GIVEN; p.actions_out = nullptr; p.env_mask = nullptr; p.decide_every = 0;

  if (int rc = select_layout(h)) return rc;

  // as-if-reset initial state with all-zero phases (the reference leaves state undefined before reset())
  cudaStream_t st = h->stream.get();
  te_reset_kernel<<<(cfg->num_envs + RESET_ENVS_PER_CTA - 1) / RESET_ENVS_PER_CTA, 128, 0, st>>>(p, nullptr, nullptr, 0);
  CU(cudaGetLastError());
  CU(cudaMemsetAsync(h->phase.get(), 0, E * h->I, st));
  // seed the arrival stream (draw 0 is the initial gap)
  if (cfg->arrival_mode == TE_ARRIVALS_PHILOX) {
    // done on the host: one Philox block per env, identical integer arithmetic
    for (size_t i = 0; i < E; i++) {
      uint32_t c[4] = {0, 0, 0, 0}, k[2] = {p.seed, (uint32_t)(cfg->env_id_base + (int64_t)i)};
      for (int rd = 0; rd < 10; rd++) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k[0], n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k[1], n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k[0] += 0x9E3779B9u; k[1] += 0xBB67AE85u;
      }
      size_t lo = 0, hi = cdf.size();
      while (lo < hi) { const size_t mid = (lo + hi) / 2; if (cdf[mid] <= c[0]) lo = mid + 1; else hi = mid; }
      es[i].ph_skip = (uint32_t)lo; es[i].ph_draw = 1; es[i].reset_count = 1;
    }
    CU(cudaStreamSynchronize(st));
    CU(cudaMemcpy(h->env.get(), es.data(), E * sizeof(EnvScalars), cudaMemcpyHostToDevice));
  }
  CU(cudaStreamSynchronize(st));
  CU(cudaDeviceSynchronize());   // the blocking table / scalar uploads above are complete before any stream steps
  *out = owner.release();
  return 0;
}

extern "C" int te_get_dims(const te_handle *h, te_dims *d) {
  if (!h || !d) return fail("te_get_dims: null argument");
  d->m = h->cfg.m; d->n = h->cfg.n; d->intersections = h->I; d->train_roads = h->r; d->roads = h->R;
  d->roads_padded = h->Rp; d->num_envs = h->cfg.num_envs; d->num_entry = h->n_entry;
  d->obs_raw = 2 * h->r + 2 * h->I; d->obs_actor = 2 * h->r + h->I;
  return 0;
}

extern "C" int te_get_topology(const te_handle *h, int32_t *dest, int32_t *nexts, int32_t *phases, int32_t *entry) {
  if (!h) return fail("te_get_topology: null handle");
  if (dest) memcpy(dest, h->dest.data(), h->R * sizeof(int));
  if (nexts) memcpy(nexts, h->nexts.data(), h->R * sizeof(int));
  if (phases) memcpy(phases, h->phases.data(), h->R * sizeof(int));
  if (entry) memcpy(entry, h->entry.data(), h->n_entry * sizeof(int));
  return 0;
}

static cudaStream_t pick_stream(te_handle *h, void *stream) { return stream ? (cudaStream_t)stream : h->stream.get(); }

extern "C" int te_reset(te_handle *h, const uint8_t *env_mask, const uint8_t *init_phase, int memspace, void *stream) {
  if (!h) return fail("te_reset: null handle");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = pick_stream(h, stream);
  const size_t E = (size_t)h->cfg.num_envs;
  const uint8_t *dm = env_mask, *dp = init_phase;
  if (memspace == TE_HOST) {
    if (env_mask) { CU(cudaMemcpyAsync(h->d_mask.get(), env_mask, E, cudaMemcpyHostToDevice, st)); dm = h->d_mask.get(); }
    if (init_phase) { CU(cudaMemcpyAsync(h->d_init_phase.get(), init_phase, E * h->I, cudaMemcpyHostToDevice, st)); dp = h->d_init_phase.get(); }
  }
  te_reset_kernel<<<(h->cfg.num_envs + RESET_ENVS_PER_CTA - 1) / RESET_ENVS_PER_CTA, 128, 0, st>>>(h->base, dm, dp, 0);
  CU(cudaGetLastError());
  if (memspace == TE_HOST) CU(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int te_set_arrivals(te_handle *h, const int64_t *offsets, const int16_t *roads, int64_t num_roads,
                               int64_t first_tick, int32_t horizon) {
  if (!h || !offsets || horizon < 0 || first_tick < 0 || num_roads < 0) return fail("te_set_arrivals: bad argument");
  if (num_roads > 0 && !roads) return fail("te_set_arrivals: roads is NULL but num_roads = %lld", (long long)num_roads);
  CU(cudaSetDevice(h->device));
  const size_t E = (size_t)h->cfg.num_envs, no = E * ((size_t)horizon + 1);
  // every range [off[e][t], off[e][t+1]) must lie inside roads[0 .. num_roads): the kernel indexes roads with them
  for (size_t e = 0; e < E; e++) {
    const int64_t *row = offsets + e * ((size_t)horizon + 1);
    if (row[0] < 0 || row[0] > num_roads) return fail("te_set_arrivals: env %zu: offset %lld outside [0, %lld]", e, (long long)row[0], (long long)num_roads);
    for (int t = 0; t < horizon; t++) {
      const int64_t a0 = row[t], a1 = row[t + 1];
      if (a0 > a1) return fail("te_set_arrivals: env %zu tick %d: offsets not monotone", e, t);
      if (a1 > num_roads) return fail("te_set_arrivals: env %zu tick %d: offset %lld beyond num_roads %lld", e, t, (long long)a1, (long long)num_roads);
      if (a1 - a0 > 255) return fail("te_set_arrivals: more than 255 arrivals in one tick of one env");
    }
  }
  std::vector<signed char> is_entry(h->R, 0);
  for (int rd : h->entry) is_entry[rd] = 1;
  for (int64_t k = 0; k < num_roads; k++)
    if (roads[k] < 0 || roads[k] >= h->R || !is_entry[roads[k]]) return fail("te_set_arrivals: road %d is not an entry road", (int)roads[k]);
  // steps may still be queued on caller-provided streams (TE_DEVICE) and read the old schedule
  CU(cudaDeviceSynchronize());
  h->base.sched_off = nullptr; h->base.sched_roads = nullptr; h->base.horizon = 0;
  CU(alloc(h->d_sched_off, no)); CU(alloc(h->d_sched_roads, (size_t)(num_roads > 0 ? num_roads : 1)));
  static_assert(sizeof(long long) == sizeof(int64_t), "int64");
  cudaStream_t st = h->stream.get();
  CU(cudaMemcpyAsync(h->d_sched_off.get(), offsets, no * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  if (num_roads > 0) CU(cudaMemcpyAsync(h->d_sched_roads.get(), roads, (size_t)num_roads * sizeof(int16_t), cudaMemcpyHostToDevice, st));
  CU(cudaStreamSynchronize(st));
  CU(cudaDeviceSynchronize());   // order the upload against every stream a later step may be launched on
  h->base.sched_off = h->d_sched_off.get(); h->base.sched_roads = h->d_sched_roads.get(); h->base.horizon = horizon;
  h->base.sched_first = first_tick;
  return 0;
}

// One request to the step kernel.  wire_only: the caller wants the compact records themselves (te_step_wire): `obs` is the
// record buffer.  nsteps > 1 / controller / env_mask: te_step_multi / te_step_masked.
struct StepReq {
  const uint8_t *actions = nullptr;   // CTRL_GIVEN: input [E][I]; CTRL_GREEDY: output (nullable)
  int K = 1, raw = 0, nsteps = 1, controller = CTRL_GIVEN;
  void *obs = nullptr; float *reward = nullptr; uint8_t *done = nullptr;
  const uint8_t *env_mask = nullptr;
  int memspace = TE_HOST; void *stream = nullptr;
  bool wire_only = false;
  const char *who = "te_step";
};

// Where a step's results go.  DEVICE: the caller's device buffers (te_step_wire: records).  WIRE: compact records
// copied to host memory (te_step_wire's buffer, or the handle's, which its helper threads expand into the caller's
// float arrays).  FLOATS: float (te_step_raw: int) arrays staged on the device and copied into the caller's arrays.
enum class Route { DEVICE, WIRE, FLOATS };

// Host float outputs travel as wire records unless the handle lets the copy engine write them (float_dma); a masked
// step takes records whenever they fit, so that only the stepped envs are expanded.  Raw ticks and steps of more than
// WIRE_MAX_K ticks do not fit a record.  The kernel writes no staging row of an env it does not step, so a masked step on
// the float route goes through the handle's page-locked staging and only the stepped rows reach the caller
// (launch_sliced).
static Route pick_route(const te_handle *h, const StepReq &q) {
  if (q.memspace != TE_HOST) return Route::DEVICE;
  const bool wire = !q.raw && q.K <= WIRE_MAX_K && (q.wire_only || !h->float_dma || q.env_mask);
  return wire ? Route::WIRE : Route::FLOATS;
}

// controller decisions of a launch
static int decisions(const StepParams &p) { return p.decide_every > 0 ? (p.nsteps + p.decide_every - 1) / p.decide_every : 1; }

// The kernel parameters of a request on its route.  The host routes stage the inputs (actions, env mask) on `st` and
// first grow the handle's staging buffers to the launch; a buffer's capacity reads 0 while it is being replaced.
static int step_params(te_handle *h, const StepReq &q, Route route, cudaStream_t st, StepParams &p) {
  const bool greedy = q.controller == CTRL_GREEDY;
  p = h->base;
  p.K = q.K; p.raw = q.raw; p.nsteps = q.nsteps; p.controller = q.controller;
  p.decide_every = greedy ? h->ctrl_spacing : 0;
  if (route == Route::DEVICE) {
    p.actions = q.actions; p.actions_out = greedy ? const_cast<uint8_t *>(q.actions) : nullptr; p.env_mask = q.env_mask;
    p.obs_f = (float *)q.obs; p.obs_i = (int *)q.obs; p.reward = q.reward; p.done = q.done;
    if (q.wire_only) { p.wire = (unsigned char *)q.obs; p.wire_stride = h->wire_stride; }
    return 0;
  }
  const size_t E = (size_t)h->cfg.num_envs;
  const int ndec = decisions(p);
  if (ndec > h->actions_cap) {
    h->actions_cap = 0;
    if (int rc = grow(h->d_actions, (size_t)ndec * E * h->I)) return rc;
    h->actions_cap = ndec;
  }
  if (!greedy) CU(cudaMemcpyAsync(h->d_actions.get(), q.actions, E * h->I, cudaMemcpyHostToDevice, st));
  if (q.env_mask) CU(cudaMemcpyAsync(h->d_mask.get(), q.env_mask, E, cudaMemcpyHostToDevice, st));
  if (route == Route::WIRE && q.nsteps > h->wire_steps) {
    const size_t n = (size_t)q.nsteps * E * h->wire_stride;
    h->wire_steps = 0;
    if (int rc = grow(h->d_wire, n)) return rc;
    if (int rc = grow(h->h_wire, n)) return rc;
    h->wire_steps = q.nsteps;
  }
  if (route == Route::FLOATS && q.nsteps > h->float_steps) {
    const size_t n = (size_t)q.nsteps * E;
    h->float_steps = 0;
    if (int rc = grow(h->d_obs_i, n * (2 * h->r + 2 * h->I))) return rc;
    if (int rc = grow(h->d_reward, n * h->I)) return rc;
    if (int rc = grow(h->d_done, n, true)) return rc;
    h->float_steps = q.nsteps;
  }
  if (route == Route::FLOATS && q.env_mask && q.nsteps > h->h_float_steps) {
    h->h_float_steps = 0;
    if (int rc = grow(h->h_float, (size_t)q.nsteps * E * (4 * (2 * h->r + 2 * h->I) + 4 * h->I + 1))) return rc;
    h->h_float_steps = q.nsteps;
  }
  p.actions = h->d_actions.get(); p.actions_out = greedy ? h->d_actions.get() : nullptr;
  p.env_mask = q.env_mask ? h->d_mask.get() : nullptr;
  p.obs_f = reinterpret_cast<float *>(h->d_obs_i.get()); p.obs_i = h->d_obs_i.get();
  p.reward = h->d_reward.get(); p.done = h->d_done.get();
  if (route == Route::WIRE) { p.wire = h->d_wire.get(); p.wire_stride = h->wire_stride; }
  return 0;
}

// The record layout of a handle (te_kernels.cuh: wire_layout) and the host path te_create chose for it.
static te_wire_layout_t wire_layout_of(const te_handle *h) {
  const WireLayout w = wire_layout(h->r, h->I);
  return {w.stride, w.passed, w.detected, w.light, w.reward, w.done, WIRE_MAX_K, h->float_dma ? 1 : 0};
}

// Host buffers: the batch is launched in slices on two alternating streams (the tail of one slice overlaps the
// head of the next), and a third stream copies each finished slice's results to the host while the following slices
// are simulated (envs are independent: any slicing gives the same results).  Fused steps of up to WIRE_MAX_K ticks
// travel as compact wire records (one copy per slice and actor step, 2.5 x fewer bytes than the float observation)
// that the handle's helper threads expand into the caller's arrays while the GPU works on the next slices.
static int launch_sliced(te_handle *h, const StepReq &q, Route route, StepParams &p, const StepVariant &sv, int smem,
                         cudaStream_t st) {
  const int nsteps = q.nsteps, G = h->G;
  const size_t E = (size_t)h->cfg.num_envs;
  const size_t obs_len = q.raw ? (size_t)(2 * h->r + 2 * h->I) : (size_t)(2 * h->r + h->I);
  const int E_i = h->cfg.num_envs;
  const int nslice = h->host_slices;
  const int per = ((E_i + nslice - 1) / nslice + G - 1) / G * G;   // whole CTAs (G envs each) per slice
  CU(cudaEventRecord(h->ev_fork.get(), st));         // actions (and the auto-reset) are complete on `st`
  CU(cudaStreamWaitEvent(h->stream2.get(), h->ev_fork.get(), 0));
  cudaStream_t lanes[2] = {st, h->stream2.get()}, cs_copy = h->stream_copy.get();
  const char *src_obs = (const char *)h->d_obs_i.get();   // int (raw) or float observations
  // float route: the caller's arrays, or for a masked step the handle's page-locked staging (same [nsteps][E] layout)
  const bool staged = route == Route::FLOATS && q.env_mask;
  unsigned char *const stage = h->h_float.get();
  char *dst_obs = staged ? (char *)stage : (char *)q.obs;
  float *dst_reward = staged ? (float *)(stage + (size_t)nsteps * E * obs_len * 4) : q.reward;
  uint8_t *dst_done = staged ? stage + (size_t)nsteps * E * (obs_len + h->I) * 4 : q.done;
  unsigned char *host_wire = q.wire_only ? (unsigned char *)q.obs : h->h_wire.get();
  const unsigned char *dev_wire = h->d_wire.get();
  const size_t wstep = E * (size_t)h->wire_stride;   // records of one actor step
  int nk = 0;
  for (int k = 0, e0 = 0; e0 < E_i; k++, e0 += per) {
    const int ne = (E_i - e0) < per ? (E_i - e0) : per;
    cudaStream_t cs = lanes[k & 1];
    p.env0 = e0; p.env_end = e0 + ne;
    sv.fn<<<(ne + G - 1) / G, h->threads, smem, cs>>>(p);
    CU(cudaGetLastError());
    CU(cudaEventRecord(h->ev_slice[k].get(), cs));
    CU(cudaStreamWaitEvent(cs_copy, h->ev_slice[k].get(), 0));
    if (route == Route::WIRE) {
      for (int j = 0; j < nsteps; j++)
        CU(cudaMemcpyAsync(host_wire + j * wstep + (size_t)e0 * h->wire_stride, dev_wire + j * wstep + (size_t)e0 * h->wire_stride,
                           (size_t)ne * h->wire_stride, cudaMemcpyDeviceToHost, cs_copy));
      CU(cudaEventRecord(h->ev_copy[k].get(), cs_copy));
    } else {
      for (int j = 0; j < nsteps; j++) {      // float arrays written by the copy engine, [nsteps][E][...]
        const size_t eo = (size_t)j * E + e0;
        CU(cudaMemcpyAsync(dst_obs + eo * obs_len * 4, src_obs + eo * obs_len * 4, (size_t)ne * obs_len * 4,
                           cudaMemcpyDeviceToHost, cs_copy));
        CU(cudaMemcpyAsync(dst_reward + eo * h->I, h->d_reward.get() + eo * h->I, (size_t)ne * h->I * sizeof(float),
                           cudaMemcpyDeviceToHost, cs_copy));
        CU(cudaMemcpyAsync(dst_done + eo, h->d_done.get() + eo, (size_t)ne, cudaMemcpyDeviceToHost, cs_copy));
      }
    }
    nk = k + 1;
  }
  if (q.controller == CTRL_GREEDY && q.actions)   // the controller's choices, for the caller
    CU(cudaMemcpyAsync(const_cast<uint8_t *>(q.actions), h->d_actions.get(), (size_t)decisions(p) * E * h->I,
                       cudaMemcpyDeviceToHost, cs_copy));
  CU(cudaEventRecord(h->ev_join.get(), h->stream2.get()));
  CU(cudaEventRecord(h->ev_copied.get(), cs_copy));
  CU(cudaStreamWaitEvent(st, h->ev_join.get(), 0));
  CU(cudaStreamWaitEvent(st, h->ev_copied.get(), 0));
  CU(cudaEventRecord(h->ev1.get(), st));
  h->timed = true;
  if (route == Route::WIRE && !q.wire_only) {
    const ExpandJob j = {h->h_wire.get(), (float *)q.obs, q.reward, q.done, q.env_mask, wire_layout_of(h), h->r, h->I, nk,
                         per, E_i, nsteps, h->ev_copy};
    const bool ok = h->pool->run(j);
    CU(cudaStreamSynchronize(st));
    if (!ok) return fail("%s: a device-to-host copy failed: %s", q.who, cudaGetErrorString(cudaGetLastError()));
    return 0;
  }
  CU(cudaStreamSynchronize(st));
  if (staged)
    for (size_t eo = 0; eo < (size_t)nsteps * E; eo++)
      if (q.env_mask[eo % E]) {
        memcpy((char *)q.obs + eo * obs_len * 4, dst_obs + eo * obs_len * 4, obs_len * 4);
        memcpy(q.reward + eo * h->I, dst_reward + eo * h->I, (size_t)h->I * sizeof(float));
        q.done[eo] = dst_done[eo];
      }
  return 0;
}

static int launch_step(te_handle *h, const StepReq &q) {
  const int K = q.K, nsteps = q.nsteps;
  const bool greedy = q.controller == CTRL_GREEDY;
  if (!h || !q.obs || (!greedy && !q.actions) || (!q.wire_only && (!q.reward || !q.done))) return fail("%s: null argument", q.who);
  if (K < 1 || K > MAX_K) return fail("%s: k_ticks must be in [1, %d]", q.who, MAX_K);
  if (nsteps < 1 || nsteps * K > MAX_K) return fail("%s: n_steps * k_ticks must be in [1, %d]", q.who, MAX_K);
  if (q.wire_only && K > WIRE_MAX_K) return fail("te_step_wire: k_ticks must be <= %d (passed counts travel as bytes)", WIRE_MAX_K);
  if (nsteps > 1 && (h->cfg.flags & TE_AUTO_RESET)) return fail("%s: a TE_AUTO_RESET handle resets between te_step calls; multi-step launches need a handle without it", q.who);
  if (h->cfg.arrival_mode == TE_ARRIVALS_INJECTED && !h->base.sched_off) return fail("%s: no arrival schedule set", q.who);
  CU(cudaSetDevice(h->device));
  cudaStream_t st = pick_stream(h, q.stream);
  const Route route = pick_route(h, q);
  StepParams p;
  if (int rc = step_params(h, q, route, st, p)) return rc;
  if (!q.raw && (h->cfg.flags & TE_AUTO_RESET)) {
    te_reset_kernel<<<(h->cfg.num_envs + RESET_ENVS_PER_CTA - 1) / RESET_ENVS_PER_CTA, 128, 0, st>>>(p, p.env_mask, nullptr, 1);
    CU(cudaGetLastError());
  }
  const StepVariant &sv = *h->sv;
  const int smem = smem_bytes(sv.maxt, sv.validate, K * nsteps, h->n_entry, h->G);
  CU(cudaEventRecord(h->ev0.get(), st));
  if (route != Route::DEVICE) return launch_sliced(h, q, route, p, sv, smem, st);
  p.env0 = 0; p.env_end = h->cfg.num_envs;
  sv.fn<<<(h->cfg.num_envs + h->G - 1) / h->G, h->threads, smem, st>>>(p);
  CU(cudaGetLastError());
  CU(cudaEventRecord(h->ev1.get(), st));
  h->timed = true;
  return 0;
}

extern "C" int te_step(te_handle *h, const uint8_t *actions, int32_t k_ticks, float *obs, float *reward, uint8_t *done,
                       int memspace, void *stream) {
  StepReq q; q.actions = actions; q.K = k_ticks; q.obs = obs; q.reward = reward; q.done = done; q.memspace = memspace; q.stream = stream;
  return launch_step(h, q);
}

extern "C" int te_step_masked(te_handle *h, const uint8_t *actions, const uint8_t *env_mask, int32_t k_ticks, float *obs,
                              float *reward, uint8_t *done, int memspace, void *stream) {
  if (!env_mask) return fail("te_step_masked: null mask");
  StepReq q; q.actions = actions; q.K = k_ticks; q.obs = obs; q.reward = reward; q.done = done; q.memspace = memspace; q.stream = stream;
  q.env_mask = env_mask; q.who = "te_step_masked";
  return launch_step(h, q);
}

extern "C" int te_step_multi(te_handle *h, int32_t n_steps, int32_t controller, uint8_t *actions, int32_t k_ticks, float *obs,
                             float *reward, uint8_t *done, int memspace, void *stream) {
  if (controller != TE_CTRL_GIVEN && controller != TE_CTRL_GREEDY) return fail("te_step_multi: unknown controller %d", controller);
  StepReq q; q.actions = actions; q.K = k_ticks; q.nsteps = n_steps; q.controller = controller == TE_CTRL_GREEDY ? CTRL_GREEDY : CTRL_GIVEN;
  q.obs = obs; q.reward = reward; q.done = done; q.memspace = memspace; q.stream = stream; q.who = "te_step_multi";
  return launch_step(h, q);
}

extern "C" int te_set_controller_spacing(te_handle *h, int32_t spacing) {
  if (!h) return fail("te_set_controller_spacing: null handle");
  if (spacing < 0 || spacing > MAX_K) return fail("te_set_controller_spacing: spacing must be in [0, %d]", MAX_K);
  h->ctrl_spacing = spacing;
  return 0;
}

extern "C" int te_step_multi_wire(te_handle *h, int32_t n_steps, int32_t controller, uint8_t *actions, int32_t k_ticks,
                                  void *records, int memspace, void *stream) {
  if (controller != TE_CTRL_GIVEN && controller != TE_CTRL_GREEDY) return fail("te_step_multi_wire: unknown controller %d", controller);
  StepReq q; q.actions = actions; q.K = k_ticks; q.nsteps = n_steps; q.controller = controller == TE_CTRL_GREEDY ? CTRL_GREEDY : CTRL_GIVEN;
  q.obs = records; q.memspace = memspace; q.stream = stream; q.wire_only = true; q.who = "te_step_multi_wire";
  return launch_step(h, q);
}

extern "C" int te_step_wire(te_handle *h, const uint8_t *actions, int32_t k_ticks, void *records, int memspace, void *stream) {
  StepReq q; q.actions = actions; q.K = k_ticks; q.obs = records; q.memspace = memspace; q.stream = stream; q.wire_only = true;
  q.who = "te_step_wire";
  return launch_step(h, q);
}

extern "C" int te_wire_layout(const te_handle *h, te_wire_layout_t *out) {
  if (!h || !out) return fail("te_wire_layout: null argument");
  *out = wire_layout_of(h);
  return 0;
}

extern "C" int te_expand_wire(const te_handle *h, const void *records, int32_t count, float *obs, float *reward, uint8_t *done) {
  if (!h || !records || !obs || !reward || !done || count < 0) return fail("te_expand_wire: bad argument");
  te_expand_records_host((const unsigned char *)records, wire_layout_of(h), h->r, h->I, count, obs, reward, done);
  return 0;
}

extern "C" int te_step_raw(te_handle *h, const uint8_t *actions, int32_t *obs, float *reward, uint8_t *done,
                           int memspace, void *stream) {
  StepReq q; q.actions = actions; q.K = 1; q.raw = 1; q.obs = obs; q.reward = reward; q.done = done; q.memspace = memspace;
  q.stream = stream; q.who = "te_step_raw";
  return launch_step(h, q);
}

extern "C" int te_remi_reward(te_handle *h, float *reward, int memspace, void *stream) {
  if (!h || !reward) return fail("te_remi_reward: null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = pick_stream(h, stream);
  float *dr = memspace == TE_HOST ? h->d_reward.get() : reward;
  te_remi_kernel<<<h->cfg.num_envs, 128, 0, st>>>(h->base, dr);
  CU(cudaGetLastError());
  if (memspace == TE_HOST) {
    CU(cudaMemcpyAsync(reward, dr, (size_t)h->cfg.num_envs * h->I * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  return 0;
}

extern "C" int te_cars_on_roads(te_handle *h, int32_t *out, int memspace, void *stream) {
  if (!h || !out) return fail("te_cars_on_roads: null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = pick_stream(h, stream);
  const size_t n = (size_t)h->cfg.num_envs * h->R;
  int *d = out;
  if (memspace == TE_HOST) {
    if (!h->d_cars) CU(alloc(h->d_cars, n));
    d = h->d_cars.get();
  }
  te_cars_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->base, d);
  CU(cudaGetLastError());
  if (memspace == TE_HOST) {
    CU(cudaMemcpyAsync(out, d, n * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  return 0;
}

extern "C" int te_greedy_actions(te_handle *h, uint8_t *actions, int memspace, void *stream) {
  if (!h || !actions) return fail("te_greedy_actions: null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = pick_stream(h, stream);
  const size_t n = (size_t)h->cfg.num_envs * h->I;
  uint8_t *d = memspace == TE_HOST ? h->d_actions.get() : actions;
  te_greedy_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->base, d);
  CU(cudaGetLastError());
  if (memspace == TE_HOST) {
    CU(cudaMemcpyAsync(actions, d, n, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  return 0;
}

// ---- snapshot records (te_kernels.cuh: snap_layout)
static SnapLayout snap_layout_of(const te_handle *h) { return snap_layout(h->R, h->I, (h->cfg.flags & TE_VALIDATE) != 0); }

extern "C" int te_snapshot_layout(const te_handle *h, te_snapshot_layout_t *out) {
  if (!h || !out) return fail("te_snapshot_layout: null argument");
  const SnapLayout L = snap_layout_of(h);
  *out = {L.stride, L.x, L.v, L.w, L.phase, L.elapsed, L.passed_dst, L.scalars};
  return 0;
}

// Shared argument checks of te_save_envs / te_load_envs: ids in range (and, for a load, each at most once).
static int snap_check_args(const te_handle *h, const char *who, const int32_t *env_ids, int32_t count, const void *records,
                           int memspace, bool unique) {
  if (!h) return fail("%s: null handle", who);
  if (count < 0) return fail("%s: count %d is negative", who, count);
  if (count > 0 && !records) return fail("%s: null records", who);
  if (memspace != TE_HOST && memspace != TE_DEVICE) return fail("%s: unknown memspace %d", who, memspace);
  if (memspace == TE_DEVICE && ((uintptr_t)records & 15)) return fail("%s: device records must be 16-byte aligned", who);
  const int E = h->cfg.num_envs;
  if (!env_ids) {
    if (count > E) return fail("%s: count %d exceeds the %d envs of the handle", who, count, E);
    return 0;
  }
  std::vector<uint8_t> seen(unique ? E : 0, 0);
  for (int32_t j = 0; j < count; j++) {
    const int e = env_ids[j];
    if (e < 0 || e >= E) return fail("%s: env_ids[%d] = %d is outside [0, %d)", who, j, e, E);
    if (unique && seen[e]++) return fail("%s: env %d is listed twice (env_ids[%d])", who, e, j);
  }
  return 0;
}

// The kernel arguments of `count` records, and the grid that covers them.
static SnapArgs snap_args(const te_handle *h, int32_t count, unsigned *blocks) {
  SnapArgs a = {};
  a.L = snap_layout_of(h);
  const int units = (a.L.w >= 0 ? 3 : 2) * h->R * CAP / 4;
  a.per_cta = std::max(1, std::min(16, SNAP_UNITS_PER_CTA / units));
  a.count = count; a.m = h->cfg.m; a.n = h->cfg.n;
  a.check_tame = h->tame ? 1 : 0; a.v_cap = h->v_cap;
  *blocks = (unsigned)((count + a.per_cta - 1) / a.per_cta);
  return a;
}

// A device copy of a host id list.  A synchronous call passes `staged`, room in the handle's staging; an asynchronous
// save gets a copy allocated (and later freed) in the order of `st`, so that it keeps its own ids while the caller goes
// on.  (The synchronous calls do not allocate: the default pool returns freed memory at every synchronisation, and mapping
// it again costs each call ~0.4 ms, at times tens of ms.)
static int upload_ids(const int32_t *env_ids, int32_t count, cudaStream_t st, int *staged, int **out) {
  *out = nullptr;
  if (!env_ids) return 0;
  *out = staged;
  if (!staged) CU(cudaMallocAsync((void **)out, (size_t)count * sizeof(int), st));
  CU(cudaMemcpyAsync(*out, env_ids, (size_t)count * sizeof(int), cudaMemcpyHostToDevice, st));
  return 0;
}

// Device staging for records in host memory and for the ids of synchronous calls (the device is idle when this is
// called).
static int snap_staging(te_handle *h, size_t bytes) {
  if (bytes > h->snap_cap) {
    h->snap_cap = 0;
    if (int rc = grow(h->d_snap, bytes)) return rc;
    h->snap_cap = bytes;
  }
  return 0;
}

// te_save_envs, and te_get_state / te_set_state, which read and patch host records; `who` names the caller's entry
// point in every error message.
static int save_records(te_handle *h, const char *who, const int32_t *env_ids, int32_t count, void *records, int memspace,
                        void *stream) {
  if (int rc = snap_check_args(h, who, env_ids, count, records, memspace, false)) return rc;
  if (count == 0) return 0;
  CU(cudaSetDevice(h->device));
  unsigned blocks = 0;
  const SnapArgs a = snap_args(h, count, &blocks);
  const size_t bytes = (size_t)count * a.L.stride;
  cudaStream_t st = pick_stream(h, stream);
  unsigned char *dst = (unsigned char *)records;
  int *staged_ids = nullptr;
  if (memspace == TE_HOST) {   // steps may be queued on caller-provided streams
    CU(cudaDeviceSynchronize());
    st = h->stream.get();
    if (int rc = snap_staging(h, bytes + (env_ids ? (size_t)count * sizeof(int) : 0))) return rc;   // records | ids
    dst = h->d_snap.get();
    staged_ids = reinterpret_cast<int *>(dst + bytes);
  }
  int *d_ids = nullptr;
  if (int rc = upload_ids(env_ids, count, st, staged_ids, &d_ids)) return rc;
  te_snap_save_kernel<<<blocks, SNAP_THREADS, 0, st>>>(h->base, a, d_ids, dst);
  CU(cudaGetLastError());
  if (d_ids && !staged_ids) CU(cudaFreeAsync(d_ids, st));
  if (memspace == TE_HOST) {
    CU(cudaMemcpyAsync(records, dst, bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  return 0;
}

// te_load_envs and te_set_state: synchronous, the records are checked before anything is written.
static int load_records(te_handle *h, const char *who, const int32_t *env_ids, int32_t count, const void *records,
                        int memspace) {
  if (int rc = snap_check_args(h, who, env_ids, count, records, memspace, true)) return rc;
  if (count == 0) return 0;
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());   // steps queued on caller-provided streams have finished with the state
  unsigned blocks = 0;
  const SnapArgs a = snap_args(h, count, &blocks);
  const size_t bytes = (size_t)count * a.L.stride;
  cudaStream_t st = h->stream.get();
  const unsigned char *src = (const unsigned char *)records;
  const size_t ids_at = memspace == TE_HOST ? bytes : 0;   // staging: host records, then ids
  if (int rc = snap_staging(h, ids_at + (env_ids ? (size_t)count * sizeof(int) : 0))) return rc;
  if (memspace == TE_HOST) {
    CU(cudaMemcpyAsync(h->d_snap.get(), records, bytes, cudaMemcpyHostToDevice, st));
    src = h->d_snap.get();
  }
  if (!h->d_snap_status) CU(alloc(h->d_snap_status, 1));
  SnapStatus status = {~0ull, 0u, 0u};
  CU(cudaMemcpyAsync(h->d_snap_status.get(), &status, sizeof(status), cudaMemcpyHostToDevice, st));
  te_snap_check_kernel<<<blocks, SNAP_THREADS, 0, st>>>(h->base, a, src, h->d_snap_status.get());
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(&status, h->d_snap_status.get(), sizeof(status), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (status.first_bad != ~0ull) {
    static const char *const what[] = {"magic", "format version", "dimensions (m, n)", "validate bit", "leading",
                                       "lastcar", "row header (top byte)", "phase", "passed_dst"};
    const long long j = (long long)(status.first_bad >> 4);
    const unsigned field = (unsigned)(status.first_bad & 15);
    return fail("%s: record %lld (for env %d): bad %s; no env was changed", who, j, env_ids ? env_ids[j] : (int)j,
                field < sizeof(what) / sizeof(what[0]) ? what[field] : "field");
  }
  int *d_ids = nullptr;
  if (int rc = upload_ids(env_ids, count, st, reinterpret_cast<int *>(h->d_snap.get() + ids_at), &d_ids)) return rc;
  te_snap_load_kernel<<<blocks, SNAP_THREADS, 0, st>>>(h->base, a, d_ids, src);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(st));
  if (status.wild && h->tame) {   // from now on: the kernels with the per-car validity predicate, one env per CTA
    h->tame = false;
    if (int rc = select_layout(h)) return rc;
  }
  return 0;
}

extern "C" int te_save_envs(te_handle *h, const int32_t *env_ids, int32_t count, void *records, int memspace, void *stream) {
  return save_records(h, "te_save_envs", env_ids, count, records, memspace, stream);
}

extern "C" int te_load_envs(te_handle *h, const int32_t *env_ids, int32_t count, const void *records, int memspace,
                            void *stream) {
  (void)stream;
  return load_records(h, "te_load_envs", env_ids, count, records, memspace);
}

// te_get_state / te_set_state: the reference's view of envs [env_begin, env_begin + count), decoded from and encoded
// into their snapshot records on the host.
extern "C" int te_get_state(te_handle *h, int32_t env_begin, int32_t count, int32_t *leading, int32_t *lastcar, float *x,
                            float *v, int32_t *obs, int32_t *waiting, uint8_t *passed_dst, float *steps) {
  if (!h) return fail("te_get_state: null handle");
  if (env_begin < 0 || count < 0 || env_begin + count > h->cfg.num_envs) return fail("te_get_state: env range out of bounds");
  const SnapLayout L = snap_layout_of(h);
  std::vector<int32_t> ids(count);
  std::iota(ids.begin(), ids.end(), env_begin);
  std::vector<unsigned char> recs((size_t)count * L.stride);
  if (int rc = save_records(h, "te_get_state", ids.data(), count, recs.data(), TE_HOST, nullptr)) return rc;
  const int R = h->R, r = h->r, I = h->I, ol = 2 * r + 2 * I;
  for (int e = 0; e < count; e++) {
    const unsigned char *rec = recs.data() + (size_t)e * L.stride;
    for (int rd = 0; rd < R; rd++) {
      const unsigned char *xr = rec + L.x + rd * CAP * 4, *vr = rec + L.v + rd * CAP * 4;
      const size_t er = (size_t)e * R + rd;
      uint32_t w0; memcpy(&w0, xr, 4);
      int wt; memcpy(&wt, vr, 4);
      const RowHeader m = unpack_meta(w0);
      if (leading) leading[er] = m.leading;
      if (lastcar) lastcar[er] = m.lastcar;
      if (obs && rd < r) { obs[(size_t)e * ol + rd] = 0; obs[(size_t)e * ol + r + rd] = m.detected; }
      if (waiting && rd < r) waiting[(size_t)e * r + rd] = wt;
      if (x) { memcpy(&x[er * CAP], xr, CAP * 4); x[er * CAP] = NAN; }
      if (v) { memcpy(&v[er * CAP], vr, CAP * 4); v[er * CAP] = NAN; }
    }
    for (int i = 0; i < I; i++) {
      int el; memcpy(&el, rec + L.elapsed + 4 * i, 4);
      if (obs) { obs[(size_t)e * ol + 2 * r + i] = rec[L.phase + i]; obs[(size_t)e * ol + 2 * r + I + i] = el; }
      if (passed_dst) passed_dst[(size_t)e * I + i] = rec[L.passed_dst + i];
    }
    if (steps) memcpy(&steps[e], rec + L.scalars + offsetof(EnvScalars, steps), 4);
  }
  return 0;
}

// Saves the range, overwrites what the caller gives and loads the records back: the rest of each env (birth ticks,
// arrival-stream position, clocks, return statistics) is kept, and the load's check pass decides whether a car is wild.
extern "C" int te_set_state(te_handle *h, int32_t env_begin, int32_t count, const int32_t *leading, const int32_t *lastcar,
                            const float *x, const float *v, const int32_t *obs, const int32_t *waiting,
                            const uint8_t *passed_dst, const float *steps) {
  if (!h) return fail("te_set_state: null handle");
  if (env_begin < 0 || count < 0 || env_begin + count > h->cfg.num_envs) return fail("te_set_state: env range out of bounds");
  if (!leading || !lastcar || !x || !v || !obs || !waiting || !passed_dst) return fail("te_set_state: all state arrays are required");
  const int R = h->R, r = h->r, I = h->I, ol = 2 * r + 2 * I;
  for (int e = 0; e < count; e++)   // every check before anything is written
    for (int rd = 0; rd < R; rd++) {
      const int ld = leading[(size_t)e * R + rd], lc = lastcar[(size_t)e * R + rd];
      if (ld < 1 || ld >= CAP || lc < 1 || lc >= CAP)
        return fail("te_set_state: ring index out of range (env %d, road %d)", env_begin + e, rd);
      const int det = rd < r ? obs[(size_t)e * ol + r + rd] : 0;
      if (det < 0 || det > 255)   // a byte of the row header word
        return fail("te_set_state: env %d road %d: detected = %d is outside [0, 255]", env_begin + e, rd, det);
    }
  const SnapLayout L = snap_layout_of(h);
  std::vector<int32_t> ids(count);
  std::iota(ids.begin(), ids.end(), env_begin);
  std::vector<unsigned char> recs((size_t)count * L.stride);
  if (int rc = save_records(h, "te_set_state", ids.data(), count, recs.data(), TE_HOST, nullptr)) return rc;
  for (int e = 0; e < count; e++) {
    unsigned char *rec = recs.data() + (size_t)e * L.stride;
    for (int rd = 0; rd < R; rd++) {
      unsigned char *xr = rec + L.x + rd * CAP * 4, *vr = rec + L.v + rd * CAP * 4;
      const size_t er = (size_t)e * R + rd;
      const uint32_t w0 = pack_meta(leading[er], lastcar[er], rd < r ? obs[(size_t)e * ol + r + rd] : 0);
      const int wt = rd < r ? waiting[(size_t)e * r + rd] : 0;
      memcpy(xr, &w0, 4); memcpy(xr + 4, &x[er * CAP + 1], (CAP - 1) * 4);
      memcpy(vr, &wt, 4); memcpy(vr + 4, &v[er * CAP + 1], (CAP - 1) * 4);
    }
    for (int i = 0; i < I; i++) {
      rec[L.phase + i] = obs[(size_t)e * ol + 2 * r + i] != 0;
      memcpy(rec + L.elapsed + 4 * i, &obs[(size_t)e * ol + 2 * r + I + i], 4);
      rec[L.passed_dst + i] = passed_dst[(size_t)e * I + i] != 0;
    }
    if (steps) memcpy(rec + L.scalars + offsetof(EnvScalars, steps), &steps[e], 4);
  }
  return load_records(h, "te_set_state", ids.data(), count, recs.data(), TE_HOST);
}

extern "C" int te_tame_speed_cap(const float *archetype, float rate, float length, float *v_cap) {
  if (!archetype || !v_cap) return fail("te_tame_speed_cap: null argument");
  te_config cfg; te_default_config(&cfg);
  memcpy(cfg.archetype, archetype, sizeof(cfg.archetype)); cfg.rate = rate; cfg.length = length;
  tame_archetype(&cfg, v_cap);
  return 0;
}

extern "C" int te_is_tame(const te_handle *h, int32_t *tame, float *v_cap) {
  if (!h || !tame) return fail("te_is_tame: null argument");
  *tame = h->tame ? 1 : 0;
  if (v_cap) *v_cap = h->v_cap;
  return 0;
}

extern "C" int te_get_stats(te_handle *h, te_stats *out) {
  if (!h || !out) return fail("te_get_stats: null argument");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());  // steps may have been queued on caller-provided streams
  DeviceStats s;
  CU(cudaMemcpy(&s, h->stats.get(), sizeof(s), cudaMemcpyDeviceToHost));
  out->ticks = s.ticks; out->actor_steps = s.actor_steps; out->vehicle_updates = s.vehicle_updates;
  out->overflows = s.overflows; out->cars_generated = s.cars_generated; out->episodes = s.episodes;
  out->return_sum = s.return_sum; out->disc_return_sum = s.disc_return_sum; out->seq_fallback_ticks = s.seq_fallback_ticks; out->cars_exited = s.cars_exited;
  out->arrival_saturations = s.arrival_saturations;
  return 0;
}

extern "C" int te_get_trip_times(te_handle *h, int32_t *env_out, float *trip_out, int64_t cap, int64_t *count, int clear) {
  if (!h || !count) return fail("te_get_trip_times: null argument");
  if (!(h->cfg.flags & TE_VALIDATE)) return fail("te_get_trip_times: handle was not created with TE_VALIDATE");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  unsigned long long n = 0;
  CU(cudaMemcpy(&n, h->d_trip_count.get(), sizeof(n), cudaMemcpyDeviceToHost));
  // The device counts every trip but records only the first trip_cap of them: on overflow the recorded ones are still
  // returned (and cleared when asked), and the call reports the truncation with return code 1.
  const bool truncated = (long long)n > h->trip_cap;
  const unsigned long long have = truncated ? (unsigned long long)h->trip_cap : n;
  *count = (int64_t)have;
  if (have && (env_out || trip_out)) {
    std::vector<TripRecord> recs(have);
    CU(cudaMemcpy(recs.data(), h->d_trips.get(), have * sizeof(TripRecord), cudaMemcpyDeviceToHost));
    // the reference appends in (env-local) tick order, road-index order, pop order
    std::sort(recs.begin(), recs.end(), [](const TripRecord &a, const TripRecord &b) {
      return a.env != b.env ? a.env < b.env : a.order < b.order; });
    const int64_t m = (int64_t)have < cap ? (int64_t)have : cap;
    for (int64_t i = 0; i < m; i++) { if (env_out) env_out[i] = recs[i].env; if (trip_out) trip_out[i] = recs[i].trip; }
  }
  if (clear) CU(cudaMemset(h->d_trip_count.get(), 0, sizeof(unsigned long long)));
  if (truncated) {
    g_err = "te_get_trip_times: " + std::to_string(n) + " trips since the last clear but the buffer holds " +
            std::to_string(h->trip_cap) + "; the first ones were returned, read more often";
    return 1;
  }
  return 0;
}

extern "C" int te_synchronize(te_handle *h) {
  if (!h) return fail("te_synchronize: null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream.get()));
  return 0;
}

extern "C" int te_stage_bandwidth(te_handle *h, int32_t repeats, double *gbytes_per_sec) {
  if (!h || !gbytes_per_sec || repeats < 1) return fail("te_stage_bandwidth: bad argument");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  const bool validate = (h->cfg.flags & TE_VALIDATE) != 0;
  // same dynamic shared-memory footprint as the step kernel, so the same number of CTAs (copies in flight) per SM
  const int stage_smem = smem_bytes(step_variant_for(h->Rp, validate, false, false).maxt, validate, 10, h->n_entry, 1);
  CU(cudaFuncSetAttribute(te_stage_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, stage_smem));
  StepParams p = h->base;
  p.K = 10;
  cudaStream_t st = h->stream.get();
  te_stage_kernel<<<h->cfg.num_envs, h->Rp, stage_smem, st>>>(p);  // warm-up (state is rewritten unchanged)
  CU(cudaEventRecord(h->ev0.get(), st));
  for (int i = 0; i < repeats; i++) te_stage_kernel<<<h->cfg.num_envs, h->Rp, stage_smem, st>>>(p);
  CU(cudaEventRecord(h->ev1.get(), st));
  CU(cudaEventSynchronize(h->ev1.get()));
  CU(cudaGetLastError());
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, h->ev0.get(), h->ev1.get()));
  const double bytes = 2.0 /* planes */ * 2.0 /* in + out */ * (double)h->cfg.num_envs * h->R * CAP * 4.0 * repeats;
  *gbytes_per_sec = bytes / (ms * 1e-3) / 1e9;
  return 0;
}

extern "C" int te_host_alloc(uint64_t bytes, void **out) {
  if (!out) return fail("te_host_alloc: null argument");
  CU(cudaHostAlloc(out, bytes ? bytes : 16, cudaHostAllocDefault));
  return 0;
}

extern "C" int te_host_free(void *ptr) {
  if (ptr) CU(cudaFreeHost(ptr));
  return 0;
}

extern "C" int te_last_kernel_ms(te_handle *h, float *ms) {
  if (!h || !ms) return fail("te_last_kernel_ms: null argument");
  if (!h->timed) return fail("te_last_kernel_ms: no step has been launched");
  CU(cudaEventSynchronize(h->ev1.get()));
  CU(cudaEventElapsedTime(ms, h->ev0.get(), h->ev1.get()));
  return 0;
}

// ------------------------------------------------------------------ test hooks
extern "C" int te_test_powf(int device, const float *x, float y, float *out, int64_t n) {
  CU(cudaSetDevice(device));
  dev_buf<float> dx, dout;
  CU(alloc(dx, n)); CU(alloc(dout, n));
  CU(cudaMemcpy(dx.get(), x, n * 4, cudaMemcpyHostToDevice));
  te_test_powf_kernel<<<(unsigned)((n + 255) / 256), 256>>>(dx.get(), y, dout.get(), n);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, dout.get(), n * 4, cudaMemcpyDeviceToHost));
  return 0;
}

// tame_archetype for the hooks below, which have no handle: the default config's road length.
static bool archetype_is_tame(const float *a, float rate) {
  te_config cfg; te_default_config(&cfg);
  memcpy(cfg.archetype, a, sizeof(cfg.archetype)); cfg.rate = rate;
  float cap;
  return tame_archetype(&cfg, &cap);
}

static int test_idm(int device, float rate, const float *a, const float *xl, const float *vl, const float *ll,
                    const float *x, const float *v, float *x_out, float *v_out, int64_t n, bool tame);
extern "C" int te_test_idm(int device, float rate, const float *a, const float *xl, const float *vl, const float *ll,
                           const float *x, const float *v, float *x_out, float *v_out, int64_t n) {
  return test_idm(device, rate, a, xl, vl, ll, x, v, x_out, v_out, n, false);
}
extern "C" int te_test_idm_tame(int device, float rate, const float *a, const float *xl, const float *vl, const float *ll,
                                const float *x, const float *v, float *x_out, float *v_out, int64_t n) {
  return test_idm(device, rate, a, xl, vl, ll, x, v, x_out, v_out, n, true);
}
static int test_idm(int device, float rate, const float *a, const float *xl, const float *vl, const float *ll,
                    const float *x, const float *v, float *x_out, float *v_out, int64_t n, bool tame) {
  IdmConst c;
  fill_idm(c, a, rate);
  if (tame && !runs_tame_form(c, archetype_is_tame(a, rate)))
    return fail("te_test_idm_tame: the tame form needs T and rate powers of two, delta = 4 and an archetype inside the "
                "tame ranges");
  CU(cudaSetDevice(device));
  CU(upload_math_consts());
  dev_buf<float> d[7];
  const float *src[5] = {xl, vl, ll, x, v};
  for (int i = 0; i < 7; i++) CU(alloc(d[i], n));
  for (int i = 0; i < 5; i++) CU(cudaMemcpy(d[i].get(), src[i], n * 4, cudaMemcpyHostToDevice));
  te_test_idm_kernel<<<(unsigned)((n + 255) / 256), 256>>>(c, d[0].get(), d[1].get(), d[2].get(), d[3].get(),
                                                           d[4].get(), d[5].get(), d[6].get(), n, tame);
  CU(cudaGetLastError());
  CU(cudaMemcpy(x_out, d[5].get(), n * 4, cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(v_out, d[6].get(), n * 4, cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int te_idm_peak_form(int device, const float *a, float rate, int32_t iters, int32_t form, int32_t warps_per_sm,
                                double *updates_per_sec) {
  if (!a || !updates_per_sec || iters < 1 || warps_per_sm < 0 || warps_per_sm > 32)
    return fail("te_idm_peak_form: bad argument");
  if (form != -1 && form != 0 && form != 5)
    return fail("te_idm_peak_form: unknown form %d (accepted: -1 = the form the step kernels run for this archetype, "
                "0 = general, 5 = tame)", form);
  IdmConst c;
  fill_idm(c, a, rate);
  if (form == 5 && !runs_tame_form(c, true)) return fail("te_idm_peak_form: form 5 needs the power-of-two, delta = 4 archetype");
  const bool tame = form == 5 || (form == -1 && runs_tame_form(c, archetype_is_tame(a, rate)));
  CU(cudaSetDevice(device));
  CU(upload_math_consts());
  int sms = 0;
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  int threads = 256, blocks = sms * 8;  // warps_per_sm == 0: 2048 resident threads per SM
  if (warps_per_sm) { threads = 32 * warps_per_sm; blocks = sms; }   // one CTA of w warps per SM
  dev_buf<float> sink;
  CU(alloc(sink, (size_t)threads * blocks));
  event_ptr e0, e1;
  CU(create(e0, cudaEventDefault)); CU(create(e1, cudaEventDefault));
  void (*kernel)(IdmConst, int, float *) = tame ? te_idm_peak_kernel<true> : te_idm_peak_kernel<false>;
  kernel<<<blocks, threads>>>(c, iters / 4 + 1, sink.get());  // warm-up
  CU(cudaEventRecord(e0.get()));
  kernel<<<blocks, threads>>>(c, iters, sink.get());
  CU(cudaEventRecord(e1.get()));
  CU(cudaEventSynchronize(e1.get()));
  CU(cudaGetLastError());
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, e0.get(), e1.get()));
  *updates_per_sec = (double)threads * blocks * iters / (ms * 1e-3);
  return 0;
}

extern "C" int te_test_powf4_exhaustive(int device, uint64_t tau, uint64_t out[4]) {
  if (!out) return fail("te_test_powf4_exhaustive: null argument");
  CU(cudaSetDevice(device));
  dev_buf<unsigned long long> d;
  CU(alloc(d, 4));
  CU(cudaMemset(d.get(), 0, 4 * sizeof(unsigned long long)));
  te_powf4_exhaustive_kernel<<<148 * 16, 256>>>((unsigned long long)tau, d.get());
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, d.get(), 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int te_test_philox(int device, const uint32_t *ctr, const uint32_t *key, uint32_t *out) {
  CU(cudaSetDevice(device));
  dev_buf<uint32_t> d;
  CU(alloc(d, 10));
  CU(cudaMemcpy(d.get(), ctr, 16, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(d.get() + 4, key, 8, cudaMemcpyHostToDevice));
  te_test_philox_kernel<<<1, 1>>>(d.get(), d.get() + 4, d.get() + 6);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, d.get() + 6, 16, cudaMemcpyDeviceToHost));
  return 0;
}
