// te_kernels.cuh - sm_100a kernels of the traffic-env simulation step.
//
// One CTA advances one env instance by K physics ticks (one actor step of the reference's
// Repeater wrapper, traffic_test.py:37-56).  The env's per-road ring buffers
// (traffic_env.py:364-366: state[R,10,20], leading[R], lastcar[R]) are staged in shared memory
// as two float planes x[Rp][20], v[Rp][20] - every car has the same archetype
// (traffic_env.py:35-43), so x and v are the only dynamic fields - and flushed once.
//
// Roads map to warps: every lane owns one road for the whole launch; the road's ring indices and counters
// live in that lane's registers.  The assignment is rebuilt per launch from the car counts (counting sort +
// snake deal) so the warps carry even loads between the two CTA barriers of a tick.
//
// Per tick (order of traffic_env.py:224-248, see DESIGN.md "tick phases"):
//   phase A  (warp-local, no CTA barrier inside)
//     - lane = road: entry arrivals -> add_car                 (traffic_env.py:274-283, 97-114)
//     - lane = road: virtual leader x from the light state     (update_lights, :81-94)
//     - car loop: the warp's live cars, road after road in ring order, form one list (warp prefix sum over
//       the per-road counts); every lane simulates a contiguous run of it, keeping the pre-update (x, v, l)
//       of the car ahead in registers from its previous iteration, so the in-place update is the Jacobi
//       update of sim (:50-62) / move_cars (:187-212); a per-warp road table holds the shared-memory
//       addresses a run walks; waiting/detected counts go back to the road lanes with shared-memory adds
//     - lane = road: pops - leading advances past cars with x > length (advance_finished_cars, :117-135)
//   barrier
//   phase C  (lane = destination road)
//     - popped cars of the unique upstream road are inserted with add_car semantics;
//       whether the insert sees the destination's pre- or post-pop `leading` follows the
//       reference's road-index order (upstream < dest: pre-pop)
//     - tail x of the road for the next tick's lights
//   barrier
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "te_math.cuh"

namespace te {

constexpr int CAP = 20;            // CAPACITY, traffic_env.py:24
constexpr int RING = CAP - 1;      // live ring positions 1..19
constexpr int YELLOW_TICKS = 6;    // traffic_env.py:21
constexpr int GROUP_ROADS = 32;    // one road per lane of the owning warp
constexpr int WARP_AREA = 720;     // per-warp tables of the car loop: 33 x 16 B road entry, 32 x (4 B counters + 2 B list start)
constexpr int MAX_K = 64;

enum : int { F_LEARN_SWITCH = 1, F_REMI = 2, F_AUTO_RESET = 4, F_VALIDATE = 8, F_ORDERED = 16 };
enum : int { ARR_NONE = 0, ARR_INJECTED = 1, ARR_PHILOX = 2 };
enum : int { CTRL_GIVEN = 0, CTRL_GREEDY = 1 };

struct EnvScalars {
  float steps;            // np.float32 tick counter of the current episode (traffic_env.py:260,247)
  uint32_t ph_draw;       // next Philox draw index
  uint32_t ph_skip;       // empty ticks left before the next car
  uint32_t reset_count;
  long long sched_cursor; // ticks consumed from the arrival process since creation (never reset)
  int ep_step;            // actor steps in the current episode
  int done;               // last te_step overflowed
  double ep_ret, ep_disc, ep_mult;
};

// The episode clock after n ticks: the reference adds 1 to its np.float32 clock once per tick (traffic_env.py:247,
// float32 under NumPy 2's promotion rules), so the clock stops at 2^24 (and at -2^24 from below), and a clock with a
// fractional part rounds when it reaches 2^23.  One add of n rounds differently in both cases.
__host__ __device__ __forceinline__ float clock_after(float c, int n) {
#pragma unroll 1
  for (int i = 0; i < n; i++) {
#ifdef __CUDA_ARCH__
    c = __fadd_rn(c, 1.f);
#else
    c = c + 1.f;
#endif
  }
  return c;
}

struct DeviceStats {
  unsigned long long ticks, actor_steps, vehicle_updates, overflows, cars_generated, episodes, seq_fallback_ticks,
      cars_exited, arrival_saturations;
  double return_sum, disc_return_sum;
};

// One car that left the map in validate mode (advance_hack, traffic_env.py:153-154).  `order` restores the
// reference's list order (tick, then road index, then pop order) after a host-side sort.
struct TripRecord {
  int env;
  float trip;             // (tick - w) / 2, seconds
  unsigned long long order;
};

struct StepParams {
  int V, r, R, Rp, I, n_entry;
  int num_envs;
  int env0;               // first env of this launch (te_step with host buffers launches the batch in slices)
  int env_end;            // one past the last env of this launch
  int G;                  // env instances per CTA (small grids share a CTA: te_api.cu envs_per_cta)
  float length;
  float det_thr_f;        // largest float <= (double)length - 10.0 (traffic_env.py:201: float32 - int64 types as float64):
                          // for every float x, (double)x > (double)length - 10.0  <=>  x > det_thr_f
  int flags, arrival_mode, K, raw, episode_len;
  float gamma;
  IdmConst idm;
  long long env_id_base;        // Philox key of env e: (seed, env_id_base + e).  (Here rather than next to `seed`: at the
                                // end of the struct, ptxas gives the 768-thread validate kernel two more registers.)
  // state (HBM)
  float *x, *v;           // [E][Rp][20]; slot 0 of a row carries packed ring indices (see pack_meta)
  float *w;               // [E][Rp][20] birth tick of each car (validate mode only, traffic_env.py:34,279)
  TripRecord *trips;      // validate mode: append buffer of finished trips
  unsigned long long *trip_count;
  long long trip_cap;
  int *elapsed;           // [E][I]
  uint8_t *phase, *passed_dst;  // [E][I]
  EnvScalars *env;
  DeviceStats *stats;
  // topology (HBM, read-only)
  const short *nexts, *up;      // [Rp], -1 = none
  const signed char *entry_idx; // [Rp], index into the entry list or -1
  // per-call I/O (device pointers)
  const uint8_t *actions;       // [E][I]
  float *obs_f;                 // [E][2r+I]   (fused actor step)
  int *obs_i;                   // [E][2r+2I]  (raw tick)
  float *reward;                // [E][I]
  uint8_t *done;                // [E]
  // compact wire record per env (te_step with host buffers / te_step_wire) instead of obs_f / reward / done:
  //   u8 passed[r] | u8 detected[r] | f32 light[I] | f32 reward[I] | u8 done | pad   (wire_stride bytes, see wire_layout)
  unsigned char *wire;
  int wire_stride;
  // multi-step launches (te_step_multi): nsteps actor steps of K ticks each (one controller decision, or one every
  // decide_every steps); the outputs
  // of actor step j go to obs / reward / done / wire + j * (their size for num_envs envs)
  int nsteps;
  int controller;               // CTRL_GIVEN: `actions` is read; CTRL_GREEDY: computed in the kernel from the ring counts
  uint8_t *actions_out;         // CTRL_GREEDY: the actions chosen, [decisions][E][I] (nullable)
  int decide_every;             // CTRL_GREEDY: a new decision every so many actor steps of the launch (0: one per launch)
  const uint8_t *env_mask;      // nullable; [E], zero = this env is not stepped (te_step_masked)
  // arrivals
  const long long *sched_off;   // [E*(horizon+1)]
  const short *sched_roads;
  int horizon;
  long long sched_first;        // arrival-process tick of schedule column 0
  const uint32_t *gap_cdf;
  int n_gap;
  uint32_t seed;
};

// Wire record of one env actor step: everything te_step returns, in 1/2.5 of the bytes of the float observation
// (passed <= 19 K and detected <= 18 fit a byte for K <= 13 ticks).  Byte offsets of the fields of a record and the
// stride between records: u8 passed[r] | u8 detected[r] | f32 light[I] (4-byte aligned: r = 4 V) | f32 reward[I] |
// u8 done, rounded up to 16 bytes.  The kernel epilogue, te_wire_layout and the host expansion read it from here.
struct WireLayout { int passed, detected, light, reward, done, stride; };
__host__ __device__ constexpr WireLayout wire_layout(int r, int I) {
  return {0, r, 2 * r, 2 * r + 4 * I, 2 * r + 8 * I, (2 * r + 8 * I + 1 + 15) / 16 * 16};
}
constexpr int WIRE_MAX_K = 13;     // 13 * 19 = 247 <= 255

// HBM row header: x[road][0] bits = leading | lastcar << 8 | detected << 16, v[road][0] bits = waiting.
struct RowHeader { int leading, lastcar, detected; };
__host__ __device__ inline uint32_t pack_meta(int leading, int lastcar, int detected) {
  return (uint32_t)leading | ((uint32_t)lastcar << 8) | ((uint32_t)detected << 16);
}
__host__ __device__ inline RowHeader unpack_meta(uint32_t w) {
  return {(int)(w & 0xff), (int)((w >> 8) & 0xff), (int)((w >> 16) & 0xff)};
}

// Shared-memory layout of one CTA.  A CTA simulates G env instances (G = 1 for large grids; small grids share a CTA so
// that no lane is a padding lane and a warp's car list is long): its rows are the G * R roads of those envs
// ("super-roads": row g * R + road), per-intersection arrays are indexed g * I + intersection.  Every offset is a
// compile-time function of the kernel variant's row capacity MAXT (>= G * R rounded up to whole warps) so that the tick
// loop addresses shared memory with immediates; only the tail has a run-time size: per env the arrival-count table
// (K * n_entry bytes) and the Philox (draw, skip) snapshots before each tick.
enum : int { ENVM_OVF = 0,    // first overflowing tick of the current actor step (NO_OVERFLOW: none yet)
             ENVM_ORD = 1,    // last tick of the launch (CTA-wide count) that needs ordered transfers
             ENVM_TB = 2,     // ticks this env ran in the earlier actor steps of this launch
             ENVM_SKIP = 3,   // env not stepped (env_mask)
             ENVM_SEG = 4,    // tick of the launch (for this env) at which the current controller decision was applied
             ENVM_WORDS = 5 };
// CTA-level counters (Smem::misc)
enum : int { CTA_RUNNING = 0,         // envs still running (an env stops after its first overflowing tick)
             CTA_ORD_TICK = 1,        // last tick of the launch in which some env needed ordered transfers (-1: none)
             CTA_VEH_UPDATES = 2,     // vehicle updates
             CTA_OVERFLOWS = 3,       // cars dropped on full rings
             CTA_GENERATED = 4,       // cars generated
             CTA_ORD_ENV_TICKS = 5,   // env-ticks that ran ordered transfers
             CTA_EXITED = 6 };        // cars that left the map
constexpr int MAX_G = 8;           // most env instances one CTA can hold (te_api.cu: select_layout)

struct SmemLayout {
  int sink, xs, vs, ws, tabs, mbar, tailx, meta, wait, elapsed, ovf, rew, misc, envm, warp, phase, act, pdst, cnt;
};

__host__ __device__ constexpr int align_up(int a, int b) { return (a + b - 1) / b * b; }

__host__ __device__ constexpr SmemLayout make_layout(int maxt, bool validate) {
  SmemLayout L = {};
  const int icap = align_up(maxt / 4, 4);               // 4 I = r < R <= Rp <= maxt
  int o = 0;
  // The car loop's sink slot: x at L.sink, below every row, and v at the same distance from it as the v plane from the
  // x plane, in the 16 bytes between the two planes.
  L.sink = o; o += 16;
  L.xs = o; o += maxt * CAP * 4;
  o += 16;
  L.vs = o; o += maxt * CAP * 4;
  L.ws = o; o += validate ? maxt * CAP * 4 : 0;
  L.tabs = o;                                           // (the powf tables stay in global memory: only the rare full-powf path reads them)
  L.mbar = o; o += 8;
  L.tailx = o; o += maxt * 4;
  L.meta = o; o += maxt * 4;
  L.wait = o; o += maxt * 4;
  L.elapsed = o; o += icap * 4;
  L.ovf = o; o += icap * 4;
  L.rew = o; o += icap * 4;
  L.misc = o; o += 32;
  L.envm = o; o += MAX_G * ENVM_WORDS * 4;                // per-env words (ENVM_*): a fixed place, so the tick loop reaches them with immediates
  o = align_up(o, 16);
  L.warp = o; o += (maxt / GROUP_ROADS) * WARP_AREA;
  L.phase = o; o += icap;
  L.act = o; o += icap;
  L.pdst = o; o += icap;
  L.cnt = align_up(o, 16);
  return L;
}

static_assert(make_layout(64, false).warp % 16 == 0 && make_layout(512, false).warp % 16 == 0 && make_layout(256, true).warp % 16 == 0 &&
              make_layout(1024, false).warp % 16 == 0 && make_layout(96, false).warp % 16 == 0 && make_layout(160, false).warp % 16 == 0 &&
              WARP_AREA % 16 == 0 && make_layout(512, false).mbar % 8 == 0 &&
              make_layout(96, false).mbar % 8 == 0 && make_layout(160, false).mbar % 8 == 0 &&
              make_layout(512, false).vs % 16 == 0 && make_layout(512, true).ws % 16 == 0 && make_layout(64, false).cnt % 16 == 0,
              "shared-memory layout alignment");
// run-time tail, KT = ticks of the whole launch (nsteps * K):
//   [G][cnt_stride] arrival counts | [G][KT + 1][2] Philox snapshots
__host__ __device__ constexpr int cnt_stride_bytes(int KT, int n_entry) { return align_up(KT * (n_entry > 0 ? n_entry : 1), 4); }
__host__ __device__ constexpr int tail_snap_offset(int KT, int n_entry, int G) { return align_up(G * cnt_stride_bytes(KT, n_entry), 8); }
__host__ __device__ constexpr int smem_bytes(int maxt, bool validate, int KT, int n_entry, int G) {
  return make_layout(maxt, validate).cnt + align_up(tail_snap_offset(KT, n_entry, G) + G * (KT + 1) * 8, 16);
}

// ---- 1-D bulk TMA (cp.async.bulk, SASS UBLKCP) + mbarrier: the env's ring planes are contiguous in HBM, so
// one elected thread moves each plane with a single instruction while the other threads set up the tick loop.
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gmem_src, uint32_t bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
  asm volatile("{\n"
               ".reg .pred p;\n"
               "TE_WAIT_%=:\n"
               "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
               "@!p bra TE_WAIT_%=;\n"
               "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_store(void *gmem_dst, const void *smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
// Commit the bulk stores and wait until the copy engine has READ their shared-memory source (the CTA may then retire
// and free its shared memory; the writes themselves complete before the grid does).
__device__ __forceinline__ void bulk_commit_wait() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// Explicit shared-window accesses for the car loop: 32-bit shared addresses kept in registers (no generic-pointer
// arithmetic inside the loop), plane offsets as immediates.
__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
  return v;
}
template <int OFF>
__device__ __forceinline__ float lds_f32_off(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(a), "n"(OFF) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
template <int OFF>
__device__ __forceinline__ void sts_f32_off(uint32_t a, float v) {
  asm volatile("st.shared.f32 [%0+%1], %2;" ::"r"(a), "n"(OFF), "f"(v) : "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
  return v;
}
template <int OFF>
__device__ __forceinline__ void sts_u32_off(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u32 [%0+%1], %2;" ::"r"(a), "n"(OFF), "r"(v) : "memory");
}
template <int OFF>
__device__ __forceinline__ uint32_t lds_u32_off(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF) : "memory");
  return v;
}
template <int OFF>
__device__ __forceinline__ void sts_u16_off(uint32_t a, unsigned short v) {
  asm volatile("st.shared.u16 [%0+%1], %2;" ::"r"(a), "n"(OFF), "h"(v) : "memory");
}
template <int OFF>
__device__ __forceinline__ int lds_u16_off(uint32_t a) {
  unsigned short v;
  asm volatile("ld.shared.u16 %0, [%1+%2];" : "=h"(v) : "r"(a), "n"(OFF) : "memory");
  return (int)v;
}
__device__ __forceinline__ void sts_v4(uint32_t a, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void red_add_shared(uint32_t a, uint32_t v) {
  asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
// Predicated load: every lane issues it, the lanes where `pred` holds execute it (no branch); elsewhere v keeps its value.
__device__ __forceinline__ void lds_v4_if(bool pred, uint32_t a, uint4 &v) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %4, 0;\n\t@p ld.shared.v4.u32 {%0, %1, %2, %3}, [%5];\n\t}"
               : "+r"(v.x), "+r"(v.y), "+r"(v.z), "+r"(v.w) : "r"((uint32_t)pred), "r"(a) : "memory");
}

__device__ __forceinline__ int ring_wrap(int a) { return a >= CAP ? 1 : a; }
__device__ __forceinline__ int ring_count(int ld, int lc) { return lc - ld + (ld > lc ? RING : 0); }
// cars on a road from its row header (or from any word with the header's leading and lastcar bytes)
__device__ __forceinline__ int ring_count(uint32_t header) {
  const RowHeader m = unpack_meta(header);
  return ring_count(m.leading, m.lastcar);
}

// greedy controller (algorithms/greedy.py:14-16): cars_on_roads()[row, col, :] . [1, 1, -1, -1] < 0, where
// cars(dd) is the number of cars on approach dd (road dd * V + intersection) of the intersection
template <class Cars>
__device__ __forceinline__ int greedy_action(Cars cars) {
  int bal = 0;
  for (int dd = 0; dd < 4; dd++) {
    const int n = cars(dd);
    bal += dd < 2 ? n : -n;
  }
  return bal < 0;
}

// phase / elapsed after the first tick of action `act` (traffic_env.py:225-232)
__device__ __forceinline__ void apply_action(int &ph, int &el, int act, bool learn_switch) {
  int change;
  if (learn_switch) { change = act; ph ^= act; } else { change = ph ^ act; ph = act; }
  el = (el + 1) * (change ? 0 : 1);
}

// phase / elapsed n ticks later while the action stays the same: learn_switch with a set action (ls_act) toggles the
// phase every tick, which keeps elapsed at 0; otherwise the phase is constant and elapsed grows by one per tick
__device__ __forceinline__ void light_after(int &ph, int &el, bool ls_act, int n) {
  if (ls_act) { ph ^= n & 1; el = 0; } else el += n;
}

// remi (traffic_env.py:64-78) of one intersection in phase ph, over its 4 approaches in road order; waiting(dd): cars
// wait on approach dd
template <class Waiting>
__device__ __forceinline__ float remi_reward(int ph, bool passed_dst, Waiting waiting) {
  float rew = 0.f;
  for (int dd = 0; dd < 4; dd++) {
    const bool green = ((dd < 2) ? 1 : 0) != ph;
    const bool w = waiting(dd);
    if (w && !green && !passed_dst) rew = __fsub_rn(rew, 0.5f);
    else if (passed_dst && green && !w) rew = __fadd_rn(rew, 0.5f);
  }
  return rew;
}

// add_car (traffic_env.py:97-114) for one identical-archetype car at (xin, vin); `chk` is the value
// of leading[road] the reference would see at that moment.  Returns false when the ring is full.
__device__ __forceinline__ bool ring_push(float *xr, float *vr, float *wr, int chk, int &lc, float xin, float vin,
                                          float win, const IdmConst &c) {
  const int pos = ring_wrap(lc + 1);
  float start = __int_as_float(0x7f800000);
  if (lc != chk) start = __fsub_rn(__fsub_rn(xr[lc], c.len), c.s0);
  if (pos == chk) return false;
  xr[pos] = (start < xin) ? start : xin;
  vr[pos] = vin;
  if (wr) wr[pos] = win;  // validate mode only
  lc = pos;
  return true;
}

struct Smem {
  float *xs, *vs, *ws, *tailx;
  uint32_t *meta;        // published after phase A: leading | lastcar << 8 | pre-pop leading << 16 | npop << 24
  int *wait, *elapsed, *ovf;
  float *rew;            // reward of the finished actor step per intersection (for the return statistic)
  unsigned long long *mbar;
  int *envm;             // per env of the CTA: ENVM_WORDS words (tick stamps, ticks run, skip flag)
  int *misc;             // CTA level: the CTA_* counters
  uint8_t *warp, *phase, *act, *pdst, *cnt;
  const PowfTables *tabs;  // glibc powf tables (global memory, L1-resident: read by ~0.4 % of the cars)
  // word w (ENVM_*) of env g of the CTA
  __device__ __forceinline__ int &env_word(int g, int w) const { return envm[g * ENVM_WORDS + w]; }
};

__device__ __forceinline__ Smem carve(unsigned char *base, const SmemLayout &L) {
  Smem s;
  s.xs = (float *)(base + L.xs); s.vs = (float *)(base + L.vs); s.ws = (float *)(base + L.ws);
  s.tailx = (float *)(base + L.tailx); s.mbar = (unsigned long long *)(base + L.mbar);
  s.meta = (uint32_t *)(base + L.meta); s.wait = (int *)(base + L.wait);
  s.elapsed = (int *)(base + L.elapsed); s.ovf = (int *)(base + L.ovf); s.rew = (float *)(base + L.rew);
  s.misc = (int *)(base + L.misc); s.envm = (int *)(base + L.envm); s.warp = base + L.warp; s.phase = base + L.phase; s.act = base + L.act;
  s.pdst = base + L.pdst; s.cnt = base + L.cnt; s.tabs = &g_powf_tables;
  return s;
}

// Move the popped cars of (super-)road u to the tail of (super-)road d (advance_finished_cars -> add_car,
// traffic_env.py:126-132).  `chk` is the value of leading[d] the reference sees at that moment:
// the pre-pop value when u < d (the reference inserts before d's own pops of this tick).
// Returns the number of cars dropped on a full ring.
__device__ __forceinline__ int transfer(const StepParams &p, const Smem &s, int u, int d, int chk, int &dlc,
                                        bool validate) {
  const uint32_t mu = s.meta[u];
  const int np = mu >> 24;
  int slot = (mu >> 16) & 0xff, dropped = 0;
  float *xd = s.xs + d * CAP, *vd = s.vs + d * CAP, *wd = validate ? s.ws + d * CAP : nullptr;
  for (int k = 0; k < np; k++) {
    slot = ring_wrap(slot + 1);
    const float xin = __fsub_rn(s.xs[u * CAP + slot], p.length);
    const float vin = s.vs[u * CAP + slot];
    const float win = validate ? s.ws[u * CAP + slot] : 0.f;
    if (!ring_push(xd, vd, wd, chk, dlc, xin, vin, win, p.idm)) dropped++;
  }
  return dropped;
}

constexpr int NO_OVERFLOW = 0x7fffffff;

// `dropped` cars of env g were lost on full rings in tick t; the env's first overflow stops it after this tick
__device__ __forceinline__ void note_overflow(const Smem &s, int g, int t, int dropped) {
  atomicAdd(&s.misc[CTA_OVERFLOWS], dropped);
  if (atomicMin(&s.env_word(g, ENVM_OVF), t) == NO_OVERFLOW) atomicSub(&s.misc[CTA_RUNNING], 1);
}

// update_lights (traffic_env.py:81-94) in closed form: while an action holds, the approach of train road `road` of
// intersection i is blocked (red or yellow) at tick tt of the launch  <=>  tt < light_ylim(...).  learn_switch with a set
// action toggles every tick, which keeps elapsed at 0 (always yellow); otherwise phase is constant and elapsed grows by
// one per tick from the state s.phase / s.elapsed that the action's first tick, tick `origin` of the launch, left.
// (A new actor step with the same action changes nothing: its first tick finds phase == action.)
__device__ __forceinline__ int light_ylim(const Smem &s, int i, int road, int V, bool learn_switch, int origin) {
  const bool ls_act = learn_switch && s.act[i];
  const int road_phase = (road / V) < 2;
  return (ls_act || road_phase == (int)s.phase[i]) ? 0x7fffffff : origin + YELLOW_TICKS - s.elapsed[i];
}

// GROUPED = false: one env per CTA (p.G == 1), everything about env groups folds away at compile time.
template <int MAXT, int MINB, bool VALIDATE, bool TAME, bool GROUPED>
__global__ void __launch_bounds__(MAXT, MINB) te_step_kernel(const StepParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr SmemLayout L = make_layout(MAXT, VALIDATE);
  const Smem s = carve(smem_raw, L);
  const int G = GROUPED ? p.G : 1;
  const int env_first = p.env0 + blockIdx.x * G;             // this CTA simulates envs [env_first, env_first + ng)
  const int ng = GROUPED ? min(G, p.env_end - env_first) : 1;  // (the last CTA of a launch may hold fewer than G)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nwarps = blockDim.x >> 5;                        // blockDim.x == G * R rounded up to whole warps
  const unsigned FULL = 0xffffffffu;
  const float INF = __int_as_float(0x7f800000);
  const bool learn_switch = (p.flags & F_LEARN_SWITCH) != 0;
  const int KT = p.K * p.nsteps;                             // ticks of the whole launch
  // te_step_masked: envs whose mask byte is zero are not stepped; a CTA with nothing to do retires at once
  int nactive = ng;
  if (p.env_mask) {
    nactive = 0;
    for (int g = 0; g < ng; g++) nactive += p.env_mask[env_first + g] != 0;
    if (nactive == 0) return;
  }
  // run-time tail of the shared-memory layout (per env: arrival counts, Philox snapshots)
  const int cnt_stride = cnt_stride_bytes(KT, p.n_entry);
  uint32_t *const snap_base = reinterpret_cast<uint32_t *>(s.cnt + tail_snap_offset(KT, p.n_entry, G));
  const int nrows = ng * p.R;                                // live rows (super-roads) of this CTA
  const int nI = ng * p.I;
  const size_t ibase = (size_t)env_first * p.I;              // the per-intersection arrays of consecutive envs are contiguous

  // ------------------------------------------------------------ prologue: stage the envs
  // only the R real roads of an env travel (its padding rows in HBM do not); rows nrows .. blockDim.x-1 are set up below
  const uint32_t plane_bytes = (uint32_t)p.R * CAP * 4;   // multiple of 16: rows of 80 B
  if (tid == 0) {
    mbar_init(s.mbar, 1);
    fence_proxy_async();
    mbar_expect_tx(s.mbar, plane_bytes * (VALIDATE ? 3u : 2u) * (uint32_t)ng);
    for (int g = 0; g < ng; g++) {
      const size_t off = (size_t)(env_first + g) * p.Rp * CAP;
      bulk_load(s.xs + g * p.R * CAP, p.x + off, plane_bytes, s.mbar);
      bulk_load(s.vs + g * p.R * CAP, p.v + off, plane_bytes, s.mbar);
      if (VALIDATE) bulk_load(s.ws + g * p.R * CAP, p.w + off, plane_bytes, s.mbar);
    }
  }
  if (tid == 0) {
    s.misc[CTA_RUNNING] = nactive; s.misc[CTA_ORD_TICK] = -1; s.misc[CTA_VEH_UPDATES] = 0; s.misc[CTA_OVERFLOWS] = 0;
    s.misc[CTA_GENERATED] = 0; s.misc[CTA_ORD_ENV_TICKS] = 0; s.misc[CTA_EXITED] = 0;
    // the sink car (see the car loop): x = NaN, v = +0
    reinterpret_cast<float *>(smem_raw + L.sink)[0] = __int_as_float(0x7fffffff);
    reinterpret_cast<float *>(smem_raw + L.sink + (L.vs - L.xs))[0] = 0.f;
  }
  if (tid < G) {
    s.env_word(tid, ENVM_OVF) = NO_OVERFLOW; s.env_word(tid, ENVM_ORD) = -1; s.env_word(tid, ENVM_TB) = 0;
    s.env_word(tid, ENVM_SEG) = 0;
    s.env_word(tid, ENVM_SKIP) = (tid >= ng) || (p.env_mask && p.env_mask[env_first + tid] == 0);
  }
  for (int g = warp; g < ng; g += nwarps) {
    // arrivals of the KT ticks of env g as per-tick, per-entry-road counts (cars are identical, so the
    // order of arrivals within a tick only matters per road, where it is preserved); one warp per env
    const int env = env_first + g;
    uint8_t *const cntg = s.cnt + g * cnt_stride;
    uint32_t *const snapg = snap_base + g * 2 * (KT + 1);
    const EnvScalars *esg = p.env + env;
    for (int i = lane; i < cnt_stride; i += 32) cntg[i] = 0;
    __syncwarp();
    if (p.arrival_mode == ARR_INJECTED) {
      const long long cur = esg->sched_cursor;
      for (int t = lane; t < KT; t += 32) {
        const long long tick = cur + t - p.sched_first;
        if (tick >= 0 && tick < p.horizon) {
          const long long *off = p.sched_off + (size_t)env * (p.horizon + 1) + tick;
          for (long long k = off[0]; k < off[1]; k++) {
            const int idx = p.entry_idx[p.sched_roads[k]];
            if (idx >= 0 && cntg[t * p.n_entry + idx] < 255) cntg[t * p.n_entry + idx]++;
          }
        }
      }
    } else if (p.arrival_mode == ARR_PHILOX) {
      // The gap process is sequential (k empty ticks, a car, a new gap ...) but its draws are counter-based:
      // draw d arrives at tick skip0 + sum of the gaps of the draws before it.  32 draws per round, one per
      // lane, exclusive prefix sum of the gaps, until a draw lands past the KT ticks of this launch.
      // snap[T] = (draw, skip) state after T ticks, written by the lane whose car is the next one due.
      uint32_t draw0 = esg->ph_draw;
      long long tbase = esg->ph_skip;         // arrival tick of draw `draw0`
      long long prev = 0;                     // arrival tick of the draw before draw0 (ticks <= prev are settled)
      const uint32_t k0 = p.seed, k1 = (uint32_t)(p.env_id_base + env);
      if (lane == 0) { snapg[0] = draw0; snapg[1] = (uint32_t)tbase; }
      for (;;) {
        uint32_t o[4];
        philox4x32_10(draw0 + lane, 0, 0, 0, k0, k1, o);
        const int gap = (int)gap_from_u32(p.gap_cdf, p.n_gap, o[0]);
        int incl = gap;
#pragma unroll
        for (int sh = 1; sh < 32; sh <<= 1) { const int y = __shfl_up_sync(FULL, incl, sh); if (lane >= sh) incl += y; }
        const long long tick = tbase + incl - gap;              // arrival tick of my draw
        long long before = __shfl_up_sync(FULL, tick, 1);
        if (lane == 0) before = prev;
        if (tick < KT) {
          // 8-bit count per (tick, entry road), four to a word; bumped with a CAS so that a 256th arrival saturates
          // (and is reported through te_stats.arrival_saturations) instead of carrying into the neighbouring count
          const int idx = (int)__umulhi(o[1], (uint32_t)p.n_entry) + (int)tick * p.n_entry;
          unsigned int *wp = reinterpret_cast<unsigned int *>(cntg) + (idx >> 2);
          const int sh = (idx & 3) * 8;
          unsigned int seen = *wp;
          for (;;) {
            if (((seen >> sh) & 0xffu) == 0xffu) { atomicAdd(&p.stats->arrival_saturations, 1ull); break; }
            const unsigned int prevw = atomicCAS(wp, seen, seen + (1u << sh));
            if (prevw == seen) break;
            seen = prevw;
          }
        }
        // after T ticks, for before < T <= tick (and T <= KT), my draw is the next car: skip = tick - T
        for (long long T = (before + 1 > 1 ? before + 1 : 1); T <= tick && T <= KT; T++) {
          snapg[2 * T] = draw0 + lane; snapg[2 * T + 1] = (uint32_t)(tick - T);
        }
        const long long last = __shfl_sync(FULL, tick, 31);
        const long long next_base = __shfl_sync(FULL, tbase + incl, 31);
        if (last >= KT) break;
        draw0 += 32; tbase = next_base; prev = last;
      }
    }
  }
  // phase / elapsed update of the first tick (traffic_env.py:225-232); later ticks of the launch repeat the same
  // action and are derived in closed form below.  A CTA has fewer intersections than threads: thread i < nI handles
  // intersection i.  Its global loads are issued before the wait on the bulk copy, so the two latencies overlap.
  int li_ph = 0, li_el = 0, li_act = 0, li_pd = 0;
  if (tid < nI) {
    li_ph = p.phase[ibase + tid] != 0;
    li_el = p.elapsed[ibase + tid];
    li_pd = p.passed_dst[ibase + tid];
    if (p.controller != CTRL_GREEDY) li_act = p.actions[ibase + tid] != 0;
  }
  __syncthreads();       // (the mbarrier is initialised for everybody)
  mbar_wait(s.mbar, 0);  // the ring planes have landed
  if (tid < nI) {
    const int i = tid;
    if (p.controller == CTRL_GREEDY) {   // from the row headers as staged
      const int g = i / p.I, ii = i - g * p.I;
      li_act = greedy_action([&](int dd) { return ring_count(__float_as_uint(s.xs[(g * p.R + dd * p.V + ii) * CAP])); });
      if (p.actions_out) p.actions_out[ibase + i] = (uint8_t)li_act;
    }
    apply_action(li_ph, li_el, li_act, learn_switch);
    s.phase[i] = (uint8_t)li_ph; s.act[i] = (uint8_t)li_act; s.elapsed[i] = li_el;
    s.pdst[i] = (uint8_t)li_pd; s.ovf[i] = 0;
  }
  if (tid >= nrows) {    // a padding row: an empty ring behind a free road, like te_reset leaves one
    s.xs[tid * CAP] = __uint_as_float(pack_meta(1, 1, 0)); s.vs[tid * CAP] = __int_as_float(0);
    s.xs[tid * CAP + 1] = INF; s.vs[tid * CAP + 1] = 0.f;
  }
  {
    // Every road-table entry starts with addresses above the sink slot (here: the table's own), so that every entry the
    // car loop can load - the one past the last listed road included - has them: a lane on the sink never crosses and
    // its waiting test reads x.  The tick loop only writes row addresses, above the sink too; entry 32 (the one past 32
    // listed roads) keeps this one.
    const uint32_t t_a = smem_u32(s.warp + warp * WARP_AREA);
    sts_v4(t_a + 16u * lane, make_uint4(t_a, t_a, t_a, 0u));
    if (lane == 0) sts_v4(t_a + 16u * 32, make_uint4(t_a, t_a, t_a, 0u));
  }

  // ---- row -> (warp, lane) assignment for this launch, balanced by car count: counting sort of the rows by
  // their current number of cars (0..18), then dealt to the warps in snake order, so every warp simulates
  // nearly the same number of cars per tick and the two CTA barriers of a tick wait on even warps.
  // Any bijection gives the same results (the update is per car); only the waiting changes.
  int my_sr;
  {
    int *hist = s.wait;                                      // [0..19] counts, [20..39] tickets (idle until the epilogue)
    short *owner = reinterpret_cast<short *>(s.meta);        // idle until the tick loop
    for (int i = tid; i < 40; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const int n0 = ring_count(__float_as_uint(s.xs[tid * CAP]));
    atomicAdd(&hist[n0], 1);
    __syncthreads();
    int base = 0;
    for (int c2 = RING - 1; c2 > n0; --c2) base += hist[c2];  // rows with more cars come first
    const int rank = base + atomicAdd(&hist[20 + n0], 1);
    const int row = rank / nwarps, pos = rank - row * nwarps;
    const int w = (row & 1) ? nwarps - 1 - pos : pos;
    owner[w * 32 + row] = (short)tid;
    __syncthreads();
    my_sr = owner[tid];
    __syncthreads();                                         // the scratch regions are reused below
  }
  // ---- lane = road: ring indices, counters and topology of my road live in registers
  const bool is_road = my_sr < nrows;
  const int my_g = (GROUPED && is_road) ? my_sr / p.R : 0;   // env of my road within the CTA
  const int my_road = GROUPED ? (is_road ? my_sr - my_g * p.R : p.R) : my_sr;   // road index inside its env (padding rows: >= R)
  const bool is_train = my_road < p.r;
  float *xr = s.xs + my_sr * CAP, *vr = s.vs + my_sr * CAP;
  float *wr = VALIDATE ? s.ws + my_sr * CAP : nullptr;
  // validate mode: the episode clock of the current tick (birth stamps, trip times), one clock_after step per tick my env
  // runs.  (Validate kernels run one env per CTA: every lane's env is the CTA's, and every lane runs every tick.)
  float clk = VALIDATE ? p.env[env_first].steps : 0.f;
  int ld, lc, wait, det, passed = 0;
  float leadx;
  {
    const RowHeader m = unpack_meta(__float_as_uint(xr[0]));
    ld = m.leading; lc = m.lastcar; det = m.detected;
    wait = __float_as_int(vr[0]);
    leadx = xr[ld];
    s.tailx[my_sr] = (lc != ld) ? xr[lc] : INF;
  }
  // topology in row (super-road) indices; -1 = none
  int nxt = -1, upr = -1, ei = -1;
  if (!GROUPED || is_road) {   // (one env per CTA: the topology tables are padded like the CTA, -1 in padding rows)
    nxt = p.nexts[my_road]; upr = p.up[my_road]; ei = p.entry_idx[my_road];
    if (GROUPED) {
      if (nxt >= 0) nxt += my_g * p.R;
      if (upr >= 0) upr += my_g * p.R;
      if (ei >= 0) ei += my_g * cnt_stride;                  // index of my entry road's tick-0 arrival count inside s.cnt
    }
  }
  const int dst = is_train ? my_g * p.I + my_road % p.V : 0;
  int ylim = is_train ? light_ylim(s, dst, my_road, p.V, learn_switch, 0) : 0;   // the approach is blocked while tt < ylim
  // per-warp tables of the car loop (rebuilt every tick)
  // (all three are reached from ONE 32-bit shared address, rt_a, with immediates: no generic pointers kept per table)
  const uint32_t rt_a = smem_u32(s.warp + warp * WARP_AREA);             // rt: non-empty roads of the warp, in lane order:
                                                                         // shared addresses of x[leading], x[lastcar], x[19]; leader x
                                                                         // (entry 32: only ever the prologue's, see there)
  constexpr int WCNT_OFF = 33 * 16;                                      // wcnt: waiting | detected << 16 per listed road
  constexpr int WST_OFF = WCNT_OFF + 32 * 4;                             // wst: first list position of each listed road (u16)
  const uint32_t wcnt_a = rt_a + WCNT_OFF;
  const uint32_t xrow_a = smem_u32(xr);                                  // shared address of x[my row][0]
  constexpr int VOFF = L.vs - L.xs;                                      // v plane relative to the x plane
  const uint32_t sink_a = smem_u32(smem_raw + L.sink);                   // x of the sink car (v at + VOFF)
  const unsigned lt_mask = (1u << lane) - 1u;
  __syncthreads();

  const IdmConst c = p.idm;
  const int obs_f_len = 2 * p.r + p.I, obs_i_len = 2 * p.r + 2 * p.I;
  const bool clear_remi = !p.raw && (p.flags & F_REMI);
  const bool use_wire = !p.raw && p.wire;
  // a row that never takes part: padding, or a road of an env that is not stepped (env_mask)
  const bool out_of_play = GROUPED ? (!is_road || s.env_word(my_g, ENVM_SKIP) != 0) : false;
  int veh_local = 0, gen_local = 0, exit_local = 0;
  int tb = 0;            // ticks my env ran in the earlier actor steps of this launch (te_step_multi)

  for (int step = 0;; step++) {
  // A lane takes part in a tick while its env is still running: an env whose ring overflowed in tick t stops after t
  // (Repeater: `if done: break`, traffic_test.py:55) while the other envs of the CTA carry on; padding rows never run.
  // (One env per CTA: never frozen - padding rows are empty rings with no topology, and the loop simply ends.)
  if (p.controller == CTRL_GREEDY && p.decide_every > 0 && step > 0 && step % p.decide_every == 0) {   // (CTA-uniform)
    // A new controller decision inside the launch (greedy.py:13-17 decides every `--spacing` actor steps): what the
    // prologue does from the staged state, on the live state.  Road lanes publish their ring indices; thread i < nI
    // takes intersection i's light state after the last tick its env ran, evaluates the controller, applies the
    // first-tick rule of the new action (traffic_env.py:225-232); road lanes re-derive their closed-form light limit
    // with the env's tick count so far (tb) as the origin.
    s.meta[my_sr] = (uint32_t)ld | ((uint32_t)lc << 8);
    __syncthreads();
    if (tid < nI) {
      const int i = tid, g = i / p.I, ii = i - g * p.I;
      if (!(GROUPED && s.env_word(g, ENVM_SKIP))) {
        int ph = s.phase[i], el = s.elapsed[i];
        light_after(ph, el, learn_switch && s.act[i],   // to the last tick run, from the segment origin
                    s.env_word(g, ENVM_TB) - 1 - s.env_word(g, ENVM_SEG));
        const int act = greedy_action([&](int dd) { return ring_count(s.meta[g * p.R + dd * p.V + ii]); });
        if (p.actions_out) p.actions_out[(size_t)(step / p.decide_every) * p.num_envs * p.I + ibase + i] = (uint8_t)act;
        apply_action(ph, el, act, learn_switch);
        s.phase[i] = (uint8_t)ph; s.act[i] = (uint8_t)act; s.elapsed[i] = el;
      }
    }
    __syncthreads();
    if (tid < ng) s.env_word(tid, ENVM_SEG) = s.env_word(tid, ENVM_TB);
    if (is_train) ylim = light_ylim(s, dst, my_road, p.V, learn_switch, tb);
  }
  bool frozen = out_of_play;
  for (int t = 0; t < p.K; t++) {
    const int tt = tb + t;     // tick of the launch for my env: arrival-process tick, light clock, birth stamp
    const int gt = step * p.K + t;   // CTA-wide tick counter of the launch: stamps the ordered-transfer requests, which are
                                     // raised before the first barrier of a tick and therefore never reset
    // ---------------------------------------------------------------- phase A
    int dropped = 0;
    if (ei >= 0 && !frozen) {  // entry arrivals, traffic_env.py:274-283
      const int na = s.cnt[ei + tt * p.n_entry];
      for (int k = 0; k < na; k++) {
        gen_local++;
        if (!ring_push(xr, vr, wr, ld, lc, c.x_new, c.v_new, clk, c)) dropped++;  // car[wi] = tick, :279
      }
    }
    if (is_train && !frozen) {  // update_lights
      if (tt < ylim) leadx = p.length;
      else leadx = nxt >= 0 ? __fadd_rn(s.tailx[nxt], p.length) : INF;
    }
    const int n = frozen ? 0 : ring_count(ld, lc);
    // The warp's live cars, road after road in ring order, form one list of `total` cars; lane l simulates the
    // q = ceil(total / 32) consecutive cars [l q, l q + q).  A car's leader is the list entry before it (or the
    // road's virtual leader), so a lane keeps the leader's PRE-update (x, v) in registers from its previous
    // iteration - the Jacobi update of sim (:50-62) / move_cars (:187-212) - and only the first car of a run reads
    // its leader from shared memory, before any lane has written (the __syncwarp below).
    int incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += y; }
    const int start = incl - n;
    const int total = __shfl_sync(FULL, incl, 31);
    const unsigned mne = __ballot_sync(FULL, n > 0);
    const int nroads = __popc(mne);
    const int cidx = n > 0 ? __popc(mne & lt_mask) : nroads + __popc(~mne & lt_mask);
    sts_u16_off<WST_OFF>(rt_a + 2u * cidx, n > 0 ? (unsigned short)start : (unsigned short)0xffff);
    if (n > 0) {
      sts_v4(rt_a + 16u * cidx, make_uint4(xrow_a + 4u * ld, xrow_a + 4u * lc, xrow_a + 4u * RING, __float_as_uint(leadx)));
      sts_u32_off<WCNT_OFF>(rt_a + 4u * cidx, 0u);
    }
    __syncwarp();
    if (total > 0) {
      const int q = (total + 31) >> 5;
      const int target = lane * q;
      const int cnt = min(q, total - target);                  // cars of my run (<= 0: none)
      // run state: address of my car's x slot; x[leading], x[lastcar], x[19] of its road; table cursors;
      // (px, pv, pl) = pre-update x, v and length of the car ahead (virtual leader: v = 0, l = 0, SURVEY 8a quirks).
      // A lane without a run starts on the sink (below), with the table's own address as its road addresses.
      uint32_t addr = sink_a, ldaddr = rt_a, lcaddr = rt_a, endaddr = rt_a, jaddr = rt_a, caddr = wcnt_a;
      float px = 0.f, pv = 0.f, pl = 0.f;
      if (cnt > 0) {
        int lo = 0;
#pragma unroll
        for (int st = 16; st > 0; st >>= 1) if (lds_u16_off<WST_OFF>(rt_a + 2u * (lo + st)) <= target) lo += st;
        const int k = target - lds_u16_off<WST_OFF>(rt_a + 2u * lo);   // my first car is the k-th from the front of road `lo`
        jaddr = rt_a + 16u * lo; caddr = wcnt_a + 4u * lo;
        const uint4 e = lds_v4(rt_a + 16u * lo);
        ldaddr = e.x; lcaddr = e.y; endaddr = e.z; px = __uint_as_float(e.w);
        addr = ldaddr + 4u * (k + 1);
        if (addr > endaddr) addr -= 4u * RING;                 // ring position ((leading + k) mod 19) + 1
        if (k != 0) {
          const uint32_t pa = (addr == endaddr - 4u * (RING - 1)) ? endaddr : addr - 4u;  // slot 1 follows slot 19
          px = lds_f32(pa); pv = lds_f32_off<VOFF>(pa); pl = c.len;
        }
      }
      __syncwarp();  // every run has read the leader of its first car before any lane overwrites a slot
      // a uniform trip count: a per-lane one (the lanes of the shorter runs leaving early) measured 4.5 % / 8 % slower
      // (10x10 / 3x3): lanes drifting apart cost more than the re-convergence.
      // A lane whose run is over, or empty, does not branch around the body: it updates the sink car, one slot shared
      // by every such lane of the CTA (x = NaN, v = +0, set up in the prologue).  Whatever its leader, its update writes
      // back x = NaN and v = +0 (te_math.cuh: idm_update), and v = +0 keeps it on the powf shortcut.  Its slot lies below
      // every row (addr < ldaddr), so its waiting test reads x: NaN < 0.2f and NaN > det_thr_f are false, and its red.add
      // adds 0.  It never crosses: lcaddr is always a row or table address, above the sink.
      for (int i = 0; i < q; i++) {
        float xn = lds_f32(addr), vn = lds_f32_off<VOFF>(addr);
        const float xl = px, vl = pv, ll = pl;
        px = xn; pv = vn; pl = c.len;
        // the tame kernels run the unchecked arithmetic; te_api.cu only launches them on tame handles
        idm_update<TAME>(c, s.tabs, xl, vl, ll, xn, vn, i < cnt);
        sts_f32(addr, xn); sts_f32_off<VOFF>(addr, vn);
        // wrapped ring, low segment (slot < leading): the reference tests x, not v (traffic_env.py:210).
        // THRESH = 0.2 is compared in double by the reference; 0.2f is the smallest float above 0.2, so for every
        // float w: (double)w < 0.2  <=>  w < 0.2f.  Same for the detector threshold with det_thr_f (see StepParams).
        // My car's counts go straight to its road's counters, so moving on to the next road hands nothing over.
        uint32_t cw = (((addr < ldaddr) ? xn : vn) < 0.2f) ? 1u : 0u;
        if (xn > p.det_thr_f) cw += 0x10000u;
        red_add_shared(caddr, cw);
        // Past the road's last car: move on to the next listed road.  Some lane of the warp does so in nearly every
        // iteration, so the cursors and the run state are updated by predicated instructions, not in a branch.
        const bool cross = addr == lcaddr;
        if (cross) { jaddr += 16u; caddr += 4u; }
        uint4 e = make_uint4(ldaddr, lcaddr, endaddr, __float_as_uint(px));
        lds_v4_if(cross, jaddr, e);  // (past the last listed road: an entry from an earlier tick or the prologue's; the sink follows)
        ldaddr = e.x; lcaddr = e.y; endaddr = e.z; px = __uint_as_float(e.w);
        pv = cross ? 0.f : pv; pl = cross ? 0.f : pl;
        const uint32_t from = cross ? ldaddr : addr;  // the slot before my next car
        addr = (from == endaddr) ? from - 4u * (RING - 1) : from + 4u;
        addr = (i + 1 < cnt) ? addr : sink_a;
      }
      __syncwarp();
    }
    int npop = 0;
    const int ld_pre = ld;
    if (n > 0) {
      veh_local += n;
      if (is_train) {
        const unsigned int cw = lds_u32_off<WCNT_OFF>(rt_a + 4u * cidx);
        wait += (int)(cw & 0xffffu); det = (int)(cw >> 16);  // detected is only rewritten for non-empty roads (:194)
      }
      // advance_finished_cars, traffic_env.py:123: pop while the front car is past the end of the road
      int f = ld;
      while (npop < n) {
        const int f2 = ring_wrap(f + 1);
        if (!(xr[f2] > p.length)) break;
        f = f2; npop++;
      }
      if (npop > 0) {
        if (VALIDATE && nxt < 0) {
          // advance_hack, traffic_env.py:153-154: trip time of every car that leaves the map
          const unsigned long long base = atomicAdd(p.trip_count, (unsigned long long)npop);
          int fs = ld;
          for (int k = 0; k < npop; k++) {
            fs = ring_wrap(fs + 1);
            if ((long long)(base + k) < p.trip_cap) {
              TripRecord rec;
              rec.env = env_first + my_g;
              rec.trip = __fsub_rn(clk, wr[fs]) / 2.0f;
              rec.order = (((unsigned long long)(p.env[env_first + my_g].sched_cursor + tt)) << 24) | ((unsigned long long)my_road << 8) | (unsigned)k;
              p.trips[base + k] = rec;
            }
          }
        }
        ld = f;
        if (nxt < 0) exit_local += npop;                // cars leaving the map
        if (nxt >= 0) {
          passed += npop;                               // traffic_env.py:127
          s.pdst[dst] = 1;                              // :128
          // Two or more pops while the upstream road has a higher index: its insert (which in the
          // reference runs after these pops were consumed) could reuse the slots the popped cars
          // still occupy.  Run this tick's transfers of this env in strict road order instead.
          if (npop >= 2 && upr > my_sr) { s.env_word(my_g, ENVM_ORD) = gt; s.misc[CTA_ORD_TICK] = gt; }
        }
      }
    }
    s.meta[my_sr] = (uint32_t)ld | ((uint32_t)lc << 8) | ((uint32_t)ld_pre << 16) | ((uint32_t)npop << 24);
    __syncthreads();
    // ---------------------------------------------------------------- phase C
    const bool want_parallel = !frozen && upr >= 0 && (s.meta[upr] >> 24) != 0;
    // (CTA-uniform) some env of the CTA needs ordered transfers in this tick
    const bool ordered_tick = s.misc[CTA_ORD_TICK] == gt || (p.flags & F_ORDERED);
    const bool ord_env = ordered_tick && !frozen && (GROUPED ? is_road : true) &&
                         (s.env_word(my_g, ENVM_ORD) == gt || (p.flags & F_ORDERED));
    if (ord_env) {
      if (my_road == 0) {                                // one lane per env walks its roads in the reference's order
        const int row0 = my_g * p.R;
        int dr_total = 0;
        for (int e = 0; e < p.R; e++) {
          const int d = p.nexts[e];
          if (d < 0 || (s.meta[row0 + e] >> 24) == 0) continue;
          const uint32_t md = s.meta[row0 + d];
          int dlc = (md >> 8) & 0xff;
          const int chk = (e < d) ? (md >> 16) & 0xff : md & 0xff;
          const int dr = transfer(p, s, row0 + e, row0 + d, chk, dlc, VALIDATE);
          s.meta[row0 + d] = (md & 0xffff00ffu) | ((uint32_t)dlc << 8);
          if (dr) { if (d < p.r) atomicAdd(&s.ovf[my_g * p.I + d % p.V], dr); dr_total += dr; }
        }
        if (dr_total) note_overflow(s, my_g, t, dr_total);
        atomicAdd(&s.misc[CTA_ORD_ENV_TICKS], 1);
      }
    } else if (want_parallel) {
      dropped += transfer(p, s, upr, my_sr, (upr < my_sr) ? ld_pre : ld, lc, VALIDATE);
    }
    if (ordered_tick) {
      __syncthreads();
      if (ord_env) lc = (s.meta[my_sr] >> 8) & 0xff;
    }
    if (dropped) {  // OVERFLOW_PENALTY on the road's intersection, traffic_env.py:109-111; done
      if (is_train) atomicAdd(&s.ovf[dst], dropped);
      note_overflow(s, my_g, t, dropped);
    }
    s.tailx[my_sr] = (lc != ld) ? xr[lc] : INF;
    __syncthreads();
    if (VALIDATE) clk = clock_after(clk, 1);   // (the tick ran, also when it stops the env below)
    // tick-stamped (a fast warp that has already flagged tick t + 1 cannot be mistaken for tick t)
    if (GROUPED) {
      frozen = frozen || s.env_word(my_g, ENVM_OVF) <= t;
      if (s.misc[CTA_RUNNING] <= 0) break;  // every env of the CTA has stopped
    } else if (s.env_word(0, ENVM_OVF) <= t) break;
  }

  // ------------------------------------------------------------ end of the actor step: observation, reward, done
  const bool last_step = step + 1 >= p.nsteps;
  s.wait[my_sr] = wait;
  __syncthreads();
  {
    const int ov = s.env_word(my_g, ENVM_OVF);
    tb += (ov != NO_OVERFLOW) ? ov + 1 : p.K;     // ticks my env has run so far in this launch
  }
  const size_t step_env0 = (size_t)step * p.num_envs;      // outputs of actor step j: j * num_envs env slots further on
  // final light state after the ticks each env ran, reward
  for (int i = tid; i < nI; i += blockDim.x) {
    const int g = i / p.I, ii = i - g * p.I;
    if (GROUPED && s.env_word(g, ENVM_SKIP)) continue;
    const int env = env_first + g;
    const int ov = s.env_word(g, ENVM_OVF);
    // the last tick of the launch env g ran, counted from the tick its current controller decision was applied at
    const int last = s.env_word(g, ENVM_TB) + ((ov != NO_OVERFLOW) ? ov : p.K - 1) - s.env_word(g, ENVM_SEG);
    unsigned char *wire_rec = use_wire ? p.wire + (step_env0 + env) * p.wire_stride : nullptr;
    int ph_f = s.phase[i], el_f = s.elapsed[i];
    light_after(ph_f, el_f, learn_switch && s.act[i], last);
    if (last_step) {
      p.phase[ibase + i] = (uint8_t)ph_f;
      p.elapsed[ibase + i] = el_f;
    }
    float rew = (float)(-10 * s.ovf[i]);  // OVERFLOW_PENALTY summed over the ticks: small integers, exact, +0 when none
    if (clear_remi) {
      rew = remi_reward(ph_f, s.pdst[i] != 0, [&](int dd) { return s.wait[g * p.R + dd * p.V + ii] > 0; });
      s.pdst[i] = 0;
    }
    if (last_step) p.passed_dst[ibase + i] = s.pdst[i];
    if (p.raw) {
      p.reward[ibase + i] = rew;
      p.obs_i[(size_t)env * obs_i_len + 2 * p.r + ii] = ph_f;
      p.obs_i[(size_t)env * obs_i_len + 2 * p.r + p.I + ii] = el_f;
    } else {
      // Repeater: obs[-I:] / 100 * (2 * phase - 1): int32 / int -> float64, cast to float32 on store
      const float light = __double2float_rn(__dmul_rn(__ddiv_rn((double)el_f, 100.0), (double)(2 * ph_f - 1)));
      if (wire_rec) {
        reinterpret_cast<float *>(wire_rec + wire_layout(p.r, p.I).light)[ii] = light;
        reinterpret_cast<float *>(wire_rec + wire_layout(p.r, p.I).reward)[ii] = rew;
      } else {
        p.reward[step_env0 * p.I + ibase + i] = rew;
        p.obs_f[(step_env0 + env) * obs_f_len + 2 * p.r + ii] = light;
      }
    }
    s.rew[i] = rew;     // for the return statistic below
    s.ovf[i] = 0;       // penalties of the next actor step start from zero
  }
  if (is_train && !out_of_play) {
    const int env = env_first + my_g;
    if (p.raw) {
      p.obs_i[(size_t)env * obs_i_len + my_road] = passed;
      p.obs_i[(size_t)env * obs_i_len + p.r + my_road] = det;
    } else if (use_wire) {
      unsigned char *wire_rec = p.wire + (step_env0 + env) * p.wire_stride;
      wire_rec[wire_layout(p.r, p.I).passed + my_road] = (unsigned char)passed;
      wire_rec[wire_layout(p.r, p.I).detected + my_road] = (unsigned char)det;
    } else {
      p.obs_f[(step_env0 + env) * obs_f_len + my_road] = (float)passed;
      p.obs_f[(step_env0 + env) * obs_f_len + p.r + my_road] = (float)det;
    }
    passed = 0;                     // Repeater starts the next actor step from zero (traffic_test.py:40)
    if (clear_remi) wait = 0;       // remi clears `waiting` (traffic_env.py:77)
  }
  if (last_step) {
    for (int o = 16; o > 0; o >>= 1) {
      veh_local += __shfl_xor_sync(FULL, veh_local, o);
      gen_local += __shfl_xor_sync(FULL, gen_local, o);
      exit_local += __shfl_xor_sync(FULL, exit_local, o);
    }
    if (lane == 0) {
      atomicAdd(&s.misc[CTA_VEH_UPDATES], veh_local); atomicAdd(&s.misc[CTA_GENERATED], gen_local);
      atomicAdd(&s.misc[CTA_EXITED], exit_local);
    }
  }
  if (last_step && !out_of_play) {
    // pack ring indices back into the row headers, restore the virtual leader's x (then: flush)
    xr[ld] = leadx;
    xr[0] = __uint_as_float(pack_meta(ld, lc, det));
    vr[0] = __int_as_float(is_train ? wait : 0);
    fence_proxy_async();  // my generic-proxy writes to the planes become visible to the bulk-copy engine
  }
  __syncthreads();
  if (tid < ng && !s.env_word(tid, ENVM_SKIP)) {          // thread g: the scalars of env g for this actor step
    const int g = tid, env = env_first + g;
    const int ov = s.env_word(g, ENVM_OVF);
    const bool overflowed = ov != NO_OVERFLOW;
    const int ticks_run = overflowed ? ov + 1 : p.K;   // >= 1
    const int ticks_total = s.env_word(g, ENVM_TB) + ticks_run;   // ticks env g has run in this launch
    EnvScalars *esg = p.env + env;
    // (wire_layout(p.r, p.I).done, spelled out: through the function the compiler schedules this kernel differently)
    if (use_wire) p.wire[(step_env0 + env) * p.wire_stride + 2 * p.r + 8 * p.I] = overflowed ? 1 : 0;
    else p.done[step_env0 + env] = overflowed ? 1 : 0;
    if (!p.raw) {
      double mean = 0.0;
      for (int i = 0; i < p.I; i++) mean += (double)s.rew[g * p.I + i];
      mean /= (double)p.I;
      const double mult = esg->ep_mult;
      esg->ep_ret += mean; esg->ep_disc += mult * mean; esg->ep_mult = mult * (double)p.gamma;
    }
    if (last_step) {
      esg->steps = clock_after(esg->steps, ticks_total);
      esg->sched_cursor += ticks_total;
      if (p.arrival_mode == ARR_PHILOX) {
        const uint32_t *snapg = snap_base + g * 2 * (KT + 1);
        esg->ph_draw = snapg[2 * ticks_total]; esg->ph_skip = snapg[2 * ticks_total + 1];
      }
      if (!p.raw) {
        esg->ep_step += p.nsteps;
        esg->done = overflowed ? 1 : 0;
        atomicAdd(&p.stats->actor_steps, (unsigned long long)p.nsteps);
      }
      atomicAdd(&p.stats->ticks, (unsigned long long)ticks_total);
    } else {   // re-arm the stamps of env g for the next actor step
      s.env_word(g, ENVM_TB) = ticks_total;
      s.env_word(g, ENVM_OVF) = NO_OVERFLOW;   // (raised only after the first barrier of a tick: safe to reset here)
    }
  }
  if (last_step) break;
  if (tid == 0) s.misc[CTA_RUNNING] = nactive;   // (decremented only after the first barrier of a tick: safe to reset here)
  }

  // ------------------------------------------------------------ flush
  if (tid == 0) {
    for (int g = 0; g < ng; g++) {
      const size_t off = (size_t)(env_first + g) * p.Rp * CAP;
      bulk_store(p.x + off, s.xs + g * p.R * CAP, plane_bytes);
      bulk_store(p.v + off, s.vs + g * p.R * CAP, plane_bytes);
      if (VALIDATE) bulk_store(p.w + off, s.ws + g * p.R * CAP, plane_bytes);
    }
    atomicAdd(&p.stats->vehicle_updates, (unsigned long long)s.misc[CTA_VEH_UPDATES]);
    if (s.misc[CTA_OVERFLOWS]) atomicAdd(&p.stats->overflows, (unsigned long long)s.misc[CTA_OVERFLOWS]);
    atomicAdd(&p.stats->cars_generated, (unsigned long long)s.misc[CTA_GENERATED]);
    if (s.misc[CTA_ORD_ENV_TICKS]) atomicAdd(&p.stats->seq_fallback_ticks, (unsigned long long)s.misc[CTA_ORD_ENV_TICKS]);
    if (s.misc[CTA_EXITED]) atomicAdd(&p.stats->cars_exited, (unsigned long long)s.misc[CTA_EXITED]);
    bulk_commit_wait();  // the flush has left shared memory before the CTA retires
  }
}

// Staging only: the step kernel's bulk-TMA stage-in and flush of one env's ring planes with no ticks in
// between (same CTA shape and shared-memory footprint, so the same number of copies is in flight per SM).
// Measures the HBM bandwidth the load/flush phases of te_step_kernel run at.
__global__ void te_stage_kernel(const StepParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int env = blockIdx.x;
  const uint32_t plane_bytes = (uint32_t)p.R * CAP * 4;   // the real roads, like the step kernel
  float *xs = reinterpret_cast<float *>(smem_raw), *vs = reinterpret_cast<float *>(smem_raw + plane_bytes);
  unsigned long long *mbar = reinterpret_cast<unsigned long long *>(smem_raw + 2 * plane_bytes);
  if (threadIdx.x == 0) {
    mbar_init(mbar, 1);
    fence_proxy_async();
    mbar_expect_tx(mbar, plane_bytes * 2u);
    bulk_load(xs, p.x + (size_t)env * p.Rp * CAP, plane_bytes, mbar);
    bulk_load(vs, p.v + (size_t)env * p.Rp * CAP, plane_bytes, mbar);
  }
  __syncthreads();
  mbar_wait(mbar, 0);
  __syncthreads();
  if (threadIdx.x == 0) {
    bulk_store(p.x + (size_t)env * p.Rp * CAP, xs, plane_bytes);
    bulk_store(p.v + (size_t)env * p.Rp * CAP, vs, plane_bytes);
    bulk_commit_wait();
  }
}

// TrafficEnv._reset (traffic_env.py:259-272) on the HBM state.  mask == nullptr: every env;
// use_done != 0: of those, the envs whose last actor step ended the episode (TE_AUTO_RESET).
// A CTA looks after RESET_ENVS_PER_CTA consecutive envs: the auto-reset pass runs before every actor step and usually
// finds nothing to do, so it should not cost a CTA per env.
constexpr int RESET_ENVS_PER_CTA = 16;
__global__ void te_reset_kernel(StepParams p, const uint8_t *mask, const uint8_t *init_phase, int use_done) {
  const int tid = threadIdx.x;
  const int env_end = min(p.num_envs, (int)(blockIdx.x + 1) * RESET_ENVS_PER_CTA);
  for (int env = blockIdx.x * RESET_ENVS_PER_CTA; env < env_end; env++) {
    EnvScalars *es = p.env + env;
    bool doit = mask ? mask[env] != 0 : true;     // (CTA-uniform)
    if (use_done) doit = doit && (es->done || (p.episode_len > 0 && es->ep_step >= p.episode_len));
    if (!doit) continue;
    float *x = p.x + (size_t)env * p.Rp * CAP, *v = p.v + (size_t)env * p.Rp * CAP;
    for (int road = tid; road < p.Rp; road += blockDim.x) {
      const int det = unpack_meta(__float_as_uint(x[road * CAP])).detected;  // `detected` survives a reset
      x[road * CAP] = __uint_as_float(pack_meta(1, 1, det));
      v[road * CAP] = __int_as_float(0);
      x[road * CAP + 1] = __int_as_float(0x7f800000);
      v[road * CAP + 1] = 0.f;
    }
    const uint32_t reset_count = es->reset_count;
    for (int i = tid; i < p.I; i += blockDim.x) {
      int ph;
      if (init_phase) ph = init_phase[(size_t)env * p.I + i] != 0;
      else {
        uint32_t o[4];
        philox4x32_10(reset_count, (uint32_t)(i >> 7), 1u, 0x5e5e7u, p.seed, (uint32_t)(p.env_id_base + env), o);
        ph = (o[(i >> 5) & 3] >> (i & 31)) & 1;
      }
      p.phase[(size_t)env * p.I + i] = (uint8_t)ph;
      p.elapsed[(size_t)env * p.I + i] = 0;
      p.passed_dst[(size_t)env * p.I + i] = 0;
    }
    __syncthreads();   // every thread has read reset_count / done before thread 0 rewrites the scalars
    if (tid == 0) {
      if (es->ep_step > 0) {
        atomicAdd(&p.stats->episodes, 1ull);
        atomicAdd(&p.stats->return_sum, es->ep_ret);
        atomicAdd(&p.stats->disc_return_sum, es->ep_disc);
      }
      es->steps = 0.f; es->ep_step = 0; es->done = 0;
      es->ep_ret = 0.0; es->ep_disc = 0.0; es->ep_mult = 1.0;
      es->reset_count = reset_count + 1;
    }
  }
}

// remi_reward as a stand-alone call (traffic_env.py:384-387) for the single-tick API.
__global__ void te_remi_kernel(StepParams p, float *reward) {
  const int env = blockIdx.x;
  float *v = p.v + (size_t)env * p.Rp * CAP;
  for (int i = threadIdx.x; i < p.I; i += blockDim.x) {
    reward[(size_t)env * p.I + i] = remi_reward(p.phase[(size_t)env * p.I + i], p.passed_dst[(size_t)env * p.I + i] != 0,
                                                [&](int dd) { return __float_as_int(v[(dd * p.V + i) * CAP]) > 0; });
  }
  __syncthreads();
  for (int i = threadIdx.x; i < p.I; i += blockDim.x) p.passed_dst[(size_t)env * p.I + i] = 0;
  for (int e = threadIdx.x; e < p.r; e += blockDim.x) v[e * CAP] = __int_as_float(0);
}

// cars_on_roads (traffic_env.py:214-218): out[E][R]
__global__ void te_cars_kernel(StepParams p, int *out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)p.num_envs * p.R) return;
  const int env = (int)(i / p.R), road = (int)(i % p.R);
  out[i] = ring_count(__float_as_uint(p.x[((size_t)env * p.Rp + road) * CAP]));
}

// the greedy controller's actions from the row headers in HBM
__global__ void te_greedy_kernel(StepParams p, uint8_t *actions) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)p.num_envs * p.I) return;
  const int env = (int)(i / p.I), it = (int)(i % p.I);
  actions[i] = (uint8_t)greedy_action([&](int dd) { return ring_count(__float_as_uint(p.x[((size_t)env * p.Rp + dd * p.V + it) * CAP])); });
}

// ---- snapshot records (te_save_envs / te_load_envs): the complete state of one env in one fixed-size blob.
//   header u32[8]: magic | version | m | n | flags (bit 0: validate) | R | I | 0
//   x[R][20], v[R][20] (and w[R][20] on validate handles) exactly as HBM holds the real rows, slot-0 header words included
//   u8 phase[I], u8 passed_dst[I], i32 elapsed[I], EnvScalars - each region padded with zeros to 16 bytes
// Every offset is a multiple of 16, so the planes move as 16-byte vectors; padding rows (R..Rp) are not carried: the step
// kernel rebuilds them in shared memory.
constexpr uint32_t SNAP_MAGIC = 0x4e534554u;   // "TESN"
constexpr uint32_t SNAP_VERSION = 1;
constexpr int SNAP_HEADER_BYTES = 32;
constexpr int SNAP_THREADS = 256;
constexpr int SNAP_UNITS_PER_CTA = 4096;        // 16-byte plane vectors a CTA moves (several envs per CTA on small grids)
struct SnapLayout { int stride, x, v, w, phase, elapsed, passed_dst, scalars; };   // bytes; w = -1 without validate
__host__ __device__ constexpr SnapLayout snap_layout(int R, int I, bool validate) {
  const int plane = R * CAP * 4;
  const int x = SNAP_HEADER_BYTES, v = x + plane, w = validate ? v + plane : -1;
  const int phase = v + plane + (validate ? plane : 0);
  const int passed_dst = phase + align_up(I, 16);
  const int elapsed = passed_dst + align_up(I, 16);
  const int scalars = elapsed + align_up(4 * I, 16);
  return {scalars + align_up((int)sizeof(EnvScalars), 16), x, v, w, phase, elapsed, passed_dst, scalars};
}
static_assert(sizeof(EnvScalars) % 4 == 0 && (CAP * 4) % 16 == 0, "snapshot record alignment");

// First failed check of te_load_envs: (record << 4) | field, the lowest one wins (atomicMin).
enum : int { SNAP_BAD_MAGIC = 0, SNAP_BAD_VERSION, SNAP_BAD_DIMS, SNAP_BAD_VALIDATE, SNAP_BAD_LEADING, SNAP_BAD_LASTCAR,
             SNAP_BAD_HEADER, SNAP_BAD_PHASE, SNAP_BAD_PASSED_DST };
struct SnapStatus {
  unsigned long long first_bad;   // ~0: every record passed
  unsigned int wild;              // some live car or leading slot is outside the tame domain (tame_car / tame_leader)
  unsigned int pad;
};
struct SnapArgs {
  SnapLayout L;
  int count, per_cta, m, n;
  int check_tame;                 // the handle is tame: look for wild cars
  float v_cap;
};

// Record j of a launch: the env it comes from / goes to.
__device__ __forceinline__ int snap_env(const int *ids, int j) { return ids ? ids[j] : j; }

// The bulk of a record: its 2 (3) planes of R * 20 floats, 16 bytes per unit.  Units of the CTA's records are dealt to
// the threads round-robin, four in flight per thread.  SAVE: state -> record, else record -> state.
template <bool SAVE>
__device__ __forceinline__ void snap_planes(const StepParams &p, const SnapArgs &a, const int *ids, unsigned char *recs,
                                            int j0, int nj) {
  const int planes = a.L.w >= 0 ? 3 : 2;
  const int n16 = p.R * CAP / 4;
  const int per_rec = planes * n16, total = nj * per_rec;
  for (int i0 = threadIdx.x; i0 < total; i0 += 4 * SNAP_THREADS) {
    uint4 val[4];
    uint4 *dst[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int i = i0 + u * SNAP_THREADS;
      dst[u] = nullptr;
      if (i < total) {
        const int jj = i / per_rec, rem = i - jj * per_rec, pl = rem / n16, k = rem - pl * n16;
        const int j = j0 + jj;
        float *plane = pl == 0 ? p.x : (pl == 1 ? p.v : p.w);
        uint4 *st = reinterpret_cast<uint4 *>(plane + (size_t)snap_env(ids, j) * p.Rp * CAP) + k;
        uint4 *rc = reinterpret_cast<uint4 *>(recs + (size_t)j * a.L.stride + (pl == 0 ? a.L.x : (pl == 1 ? a.L.v : a.L.w))) + k;
        val[u] = SAVE ? *st : *rc;
        dst[u] = SAVE ? rc : st;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; u++)
      if (dst[u]) *dst[u] = val[u];
  }
}

// te_save_envs: gather the listed envs into records (records [count][stride], 16-byte aligned).
__global__ void __launch_bounds__(SNAP_THREADS) te_snap_save_kernel(const StepParams p, const SnapArgs a, const int *ids,
                                                                    unsigned char *recs) {
  const int j0 = blockIdx.x * a.per_cta, nj = min(a.per_cta, a.count - j0);
  snap_planes<true>(p, a, ids, recs, j0, nj);
  // header and the small per-intersection / per-env regions, one 32-bit word per thread, padding written as zeros
  const int hw = SNAP_HEADER_BYTES / 4, sw = (a.L.stride - a.L.phase) / 4, per = hw + sw;
  for (int i = threadIdx.x; i < nj * per; i += SNAP_THREADS) {
    const int jj = i / per, k = i - jj * per, j = j0 + jj, env = snap_env(ids, j);
    uint32_t *rec = reinterpret_cast<uint32_t *>(recs + (size_t)j * a.L.stride);
    if (k < hw) {
      const uint32_t h[8] = {SNAP_MAGIC, SNAP_VERSION, (uint32_t)a.m, (uint32_t)a.n, p.w ? 1u : 0u, (uint32_t)p.R,
                             (uint32_t)p.I, 0u};
      rec[k] = h[k];
      continue;
    }
    const int o = a.L.phase + 4 * (k - hw);   // byte offset inside the record
    uint32_t word = 0;
    if (o < a.L.elapsed) {                    // phase / passed_dst bytes
      const bool ph = o < a.L.passed_dst;
      const int b = o - (ph ? a.L.phase : a.L.passed_dst);
      const uint8_t *src = (ph ? p.phase : p.passed_dst) + (size_t)env * p.I;
      for (int t = 0; t < 4; t++)
        if (b + t < p.I) word |= (uint32_t)src[b + t] << (8 * t);
    } else if (o < a.L.scalars) {
      const int idx = (o - a.L.elapsed) / 4;
      if (idx < p.I) word = (uint32_t)p.elapsed[(size_t)env * p.I + idx];
    } else {
      const int idx = (o - a.L.scalars) / 4;
      if (idx < (int)(sizeof(EnvScalars) / 4)) word = reinterpret_cast<const uint32_t *>(p.env + env)[idx];
    }
    rec[a.L.phase / 4 + (k - hw)] = word;
  }
}

// The tame-car rule (te_math.cuh, idm_update), its one definition: the check pass of every load (te_load_envs,
// te_set_state) applies it.  x = -0 is not tame: the tame kernels move a car with dx <= 0 by keeping x, where the
// reference adds +-0.
__device__ __forceinline__ bool tame_car(float x, float v, float v_cap) {
  return isfinite(x) && fabsf(x) < 0x1p40f && __float_as_uint(x) != 0x80000000u && isfinite(v) && (v == 0.f ? !signbit(v) : (v >= 0x1p-100f && v <= v_cap));
}
__device__ __forceinline__ bool tame_leader(float x) {
  return x == __int_as_float(0x7f800000) || (isfinite(x) && fabsf(x) < 0x1p40f);
}

// te_load_envs, first pass: check every record (nothing is written to the state).  One item per 16-byte quad of the x
// plane (ring indices from the row's header word; live cars and the leading slot of that quad against the tame predicate
// when the handle is tame), per intersection (phase, passed_dst) and per record (header).
__global__ void __launch_bounds__(SNAP_THREADS) te_snap_check_kernel(const StepParams p, const SnapArgs a,
                                                                     const unsigned char *recs, SnapStatus *status) {
  const int j0 = blockIdx.x * a.per_cta, nj = min(a.per_cta, a.count - j0);
  const int nq = p.R * CAP / 4, items = nq + p.I + 1;
  bool wild = false;
  for (int i = threadIdx.x; i < nj * items; i += SNAP_THREADS) {
    const int jj = i / items, it = i - jj * items, j = j0 + jj;
    const unsigned char *rec = recs + (size_t)j * a.L.stride;
    int bad = -1;
    if (it < nq) {
      const int rd = it / (CAP / 4), q = it - rd * (CAP / 4);
      const uint32_t hw = *reinterpret_cast<const uint32_t *>(rec + a.L.x + rd * CAP * 4);
      const int ld = (int)(hw & 0xff), lc = (int)((hw >> 8) & 0xff);
      const bool ld_ok = ld >= 1 && ld < CAP, lc_ok = lc >= 1 && lc < CAP, top_ok = (hw >> 24) == 0;
      if (q == 0) bad = !ld_ok ? SNAP_BAD_LEADING : (!lc_ok ? SNAP_BAD_LASTCAR : (!top_ok ? SNAP_BAD_HEADER : -1));
      if (a.check_tame && ld_ok && lc_ok) {
        const float4 xq = *reinterpret_cast<const float4 *>(rec + a.L.x + rd * CAP * 4 + q * 16);
        const float4 vq = *reinterpret_cast<const float4 *>(rec + a.L.v + rd * CAP * 4 + q * 16);
        const float xs[4] = {xq.x, xq.y, xq.z, xq.w}, vs[4] = {vq.x, vq.y, vq.z, vq.w};
        const int cnt = ring_count(ld, lc);
#pragma unroll
        for (int t = 0; t < 4; t++) {
          const int s = 4 * q + t;
          if (s == 0) continue;                  // the header word
          int d = s - ld;
          if (d < 0) d += RING;                  // ring distance behind the leading slot: 0 = leading, 1..cnt = live cars
          if (d == 0) wild |= !tame_leader(xs[t]);
          else if (d <= cnt) wild |= !tame_car(xs[t], vs[t], a.v_cap);
        }
      }
    } else if (it < nq + p.I) {
      const int b = it - nq;
      if (rec[a.L.phase + b] > 1) bad = SNAP_BAD_PHASE;
      else if (rec[a.L.passed_dst + b] > 1) bad = SNAP_BAD_PASSED_DST;
    } else {
      const uint32_t *h = reinterpret_cast<const uint32_t *>(rec);
      if (h[0] != SNAP_MAGIC) bad = SNAP_BAD_MAGIC;
      else if (h[1] != SNAP_VERSION) bad = SNAP_BAD_VERSION;
      else if (h[2] != (uint32_t)a.m || h[3] != (uint32_t)a.n || h[5] != (uint32_t)p.R || h[6] != (uint32_t)p.I) bad = SNAP_BAD_DIMS;
      else if (h[4] != (p.w ? 1u : 0u)) bad = SNAP_BAD_VALIDATE;
    }
    if (bad >= 0) atomicMin(&status->first_bad, ((unsigned long long)j << 4) | (unsigned)bad);
  }
  if (__syncthreads_or(wild) && threadIdx.x == 0) status->wild = 1;
}

// te_load_envs, second pass (every record checked): scatter record j into env ids[j].  The header is not stored.
__global__ void __launch_bounds__(SNAP_THREADS) te_snap_load_kernel(const StepParams p, const SnapArgs a, const int *ids,
                                                                    const unsigned char *recs) {
  const int j0 = blockIdx.x * a.per_cta, nj = min(a.per_cta, a.count - j0);
  snap_planes<false>(p, a, ids, const_cast<unsigned char *>(recs), j0, nj);
  const int ns = (int)(sizeof(EnvScalars) / 4), per = 3 * p.I + ns;
  for (int i = threadIdx.x; i < nj * per; i += SNAP_THREADS) {
    const int jj = i / per, k = i - jj * per, j = j0 + jj, env = snap_env(ids, j);
    const unsigned char *rec = recs + (size_t)j * a.L.stride;
    if (k < p.I) p.phase[(size_t)env * p.I + k] = rec[a.L.phase + k];
    else if (k < 2 * p.I) p.passed_dst[(size_t)env * p.I + k - p.I] = rec[a.L.passed_dst + k - p.I];
    else if (k < 3 * p.I) p.elapsed[(size_t)env * p.I + k - 2 * p.I] = reinterpret_cast<const int *>(rec + a.L.elapsed)[k - 2 * p.I];
    else reinterpret_cast<uint32_t *>(p.env + env)[k - 3 * p.I] = reinterpret_cast<const uint32_t *>(rec + a.L.scalars)[k - 3 * p.I];
  }
}

// ---- test hooks
__global__ void te_test_powf_kernel(const float *x, float y, float *out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = powf_glibc(x[i], y, &g_powf_tables);
}
__global__ void te_test_idm_kernel(IdmConst c, const float *xl, const float *vl, const float *ll, const float *x,
                                   const float *v, float *xo, float *vo, long long n, int tame) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    float xx = x[i], vv = v[i];
    if (tame) idm_update<true>(c, &g_powf_tables, xl[i], vl[i], ll[i], xx, vv);   // tame operands only
    else idm_update<false>(c, &g_powf_tables, xl[i], vl[i], ll[i], xx, vv);
    xo[i] = xx; vo[i] = vv;
  }
}
// Arithmetic-only ceiling: every lane runs `iters` dependent IDM updates of one car behind a leader that drives at
// constant speed (registers only), in the form a step kernel with the same TAME runs.  One instantiation per form, so
// that each timed loop is compiled on its own.  __maxnreg__(40) keeps the register budget the rates in DESIGN.md
// section 4 were measured with: 48 warps per SM at warps_per_sm = 0 (six 256-thread CTAs) and the same loop schedule.
// Left to itself ptxas gives the tame form 30 registers and a schedule that runs 5 % slower at 32 warps per SM.
template <bool TAME>
__global__ void __maxnreg__(40) te_idm_peak_kernel(IdmConst c, int iters, float *sink) {
  __shared__ PowfTables tabs;
  for (int i = threadIdx.x; i < (int)(sizeof(PowfTables) / 8); i += blockDim.x)
    reinterpret_cast<unsigned long long *>(&tabs)[i] = reinterpret_cast<const unsigned long long *>(&g_powf_tables)[i];
  __syncthreads();
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  float x = 0.f, v = 5.f + 0.001f * (float)(gid & 1023);
  float xl = 30.f + 0.01f * (float)(gid & 255);
  const float vl = 9.f, step = __fmul_rn(vl, c.rate);
  for (int i = 0; i < iters; i++) {
    idm_update<TAME>(c, &tabs, xl, vl, c.len, x, v);
    xl = __fadd_rn(xl, step);
  }
  sink[gid] = x + v;
}

// Exhaustive study of powf(r, 4) over EVERY non-negative finite float r: compares glibc's algorithm with
// RN_f32((r*r)*(r*r)) (double products) and records, for the inputs where they differ, how far the double
// r^4 sits from the float rounding boundary (in units of 2^-52 of the significand).  out[0] = #inputs where the
// two differ, out[1] = max boundary distance among them, out[2] = #inputs the filter (distance <= tau or result
// outside the normal float range) sends to the full algorithm, out[3] = #inputs where the filter accepts but the
// results differ (must be 0).
__global__ void te_powf4_exhaustive_kernel(unsigned long long tau, unsigned long long *out) {
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  unsigned long long diff = 0, maxd = 0, slow = 0, bad = 0;
  for (unsigned long long ix = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; ix < 0x7f800000ull; ix += stride) {
    const float r = __uint_as_float((uint32_t)ix);
    const float ref = powf_glibc(r, 4.0f, &g_powf_tables);
    float fast;
    unsigned dist;
    const bool acc = powf4_try(r, (unsigned)tau, fast, dist);
    const bool same = __float_as_uint(fast) == __float_as_uint(ref);
    if (!same) { diff++; if (acc) bad++; if (dist > maxd && dist != 0xffffffffu) maxd = dist; }
    if (!acc) slow++;
    // the step kernel's form of the filter (powf4_fast) must never accept an input whose shortcut differs
    double pd2;
    if (powf4_fast_d((double)r, pd2) && !(pd2 == (double)ref && __float_as_uint(__double2float_rn(pd2)) == __float_as_uint(ref))) bad++;
  }
  atomicAdd(&out[0], diff); atomicMax(&out[1], maxd); atomicAdd(&out[2], slow); atomicAdd(&out[3], bad);
}

__global__ void te_test_philox_kernel(const uint32_t *ctr, const uint32_t *key, uint32_t *out) {
  uint32_t o[4];
  philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1], o);
  for (int i = 0; i < 4; i++) out[i] = o[i];
}

}  // namespace te
