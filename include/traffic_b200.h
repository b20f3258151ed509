/*
 * traffic_b200.h - C ABI of libtraffic_b200.so, the B200 (sm_100a) implementation of
 * the traffic-env simulation step.
 *
 * The reference (samanklesaria/traffic-env) has no FFI of its own: its boundary is
 * the Python class gym_traffic.envs.traffic_env.TrafficEnv (traffic_env.py:221-394)
 * plus the Repeater/Remi wrappers that sit on the tick loop (traffic_test.py:27-64).
 * Each entry point below names the reference interface it replaces.  A maintainer
 * binds these with ctypes from inside TrafficEnv (see INTEGRATION.md).
 *
 * Conventions
 *  - plain C, no torch/CUDA types in signatures; `stream` is a cudaStream_t passed as
 *    void* (NULL = the handle's own stream);
 *  - every function returns 0 on success, <0 on error (te_last_error() has the text);
 *    simulation overflow is DATA (done[e] = 1), never an error (traffic_env.py:109-113,
 *    246-248);
 *  - `memspace` says where caller buffers live: TE_HOST (pageable or pinned host memory;
 *    the call is synchronous) or TE_DEVICE (device memory on the handle's device; the
 *    call is asynchronous on `stream`);
 *  - E = num_envs, I = m*n intersections, r = 4*I train roads, R = r + 2m + 2n roads
 *    (roadgraph.py:30-33), CAP = 20 ring slots (traffic_env.py:24);
 *  - one handle = one device = one contiguous block of env instances; a handle may be
 *    used from one thread at a time, different handles from different threads freely
 *    (a3c.py:69-72 steps envs from several Python threads).
 */
#ifndef TRAFFIC_B200_H
#define TRAFFIC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TE_CAP 20
#define TE_PARAMS 10

enum te_memspace { TE_HOST = 0, TE_DEVICE = 1 };

enum te_flags {
  TE_LEARN_SWITCH = 1 << 0, /* FLAGS.learn_switch, traffic_env.py:225-230 */
  TE_REMI = 1 << 1,         /* te_step returns remi_reward() (traffic_test.py:59-64) instead of the summed env reward */
  TE_AUTO_RESET = 1 << 2,   /* an env that finished (overflow or episode_len) is _reset at the start of its next te_step */
  TE_VALIDATE = 1 << 3,     /* FLAGS.mode == 'validate': record trip times (traffic_env.py:139-157) */
  TE_ORDERED_TRANSFERS = 1 << 4 /* verification aid: run every tick's road-to-road transfers in strict road-index order
                                   (the reference's loop order) instead of in parallel; results are identical */
};

enum te_arrival_mode {
  TE_ARRIVALS_NONE = 0,
  TE_ARRIVALS_INJECTED = 1, /* replay a schedule given with te_set_arrivals (equivalence runs) */
  TE_ARRIVALS_PHILOX = 2    /* counter-based Philox4x32-10 stream, same process as poisson() (traffic_env.py:160-164) */
};

typedef struct te_config {
  int32_t struct_size;   /* = sizeof(te_config) */
  int32_t m, n;          /* GridRoad(m, n, length), roadgraph.py:26 */
  float length;          /* road length in metres */
  float rate;            /* FLAGS.rate: seconds per tick, traffic_env.py:12 */
  int32_t num_envs;      /* env instances on this device */
  int64_t env_id_base;   /* global id of local env 0 (keys the Philox stream; makes results independent of sharding) */
  int32_t device;        /* CUDA device ordinal */
  int32_t flags;         /* te_flags */
  uint32_t entry_spec;   /* generate_entrypoints(spec), roadgraph.py:42-51: bit k set = side k closed */
  int32_t arrival_mode;  /* te_arrival_mode */
  double cars_per_tick;  /* FLAGS.cars_per_sec * FLAGS.rate (traffic_env.py:161, 394); Philox mode */
  uint64_t seed;         /* Philox key (with the global env id) */
  int32_t episode_len;   /* actor steps per episode for TE_AUTO_RESET (0 = only overflow ends an episode) */
  float gamma;           /* FLAGS.gamma for the discounted return statistic (util.py:68-94) */
  float archetype[TE_PARAMS]; /* x,v,l,a,delta,v0,b,T,s0,w of a new car, traffic_env.py:33-43 */
} te_config;

typedef struct te_dims {
  int32_t m, n, intersections, train_roads, roads, roads_padded, num_envs, num_entry;
  int32_t obs_raw;   /* 2r + 2I ints: TrafficEnv.obs, traffic_env.py:370-376 */
  int32_t obs_actor; /* 2r + I floats: Repeater observation, traffic_test.py:33 */
} te_dims;

typedef struct te_stats {
  uint64_t ticks;            /* env-ticks executed */
  uint64_t actor_steps;      /* env actor steps executed by te_step */
  uint64_t vehicle_updates;  /* real cars advanced by one tick (one element of one sim() call) */
  uint64_t overflows;        /* cars dropped on a full ring */
  uint64_t cars_generated;
  uint64_t episodes;         /* episodes closed by TE_AUTO_RESET / te_reset */
  double return_sum;         /* sum over closed episodes of sum_t mean_i reward (util.py:75) */
  double disc_return_sum;    /* same with gamma^t weighting */
  uint64_t seq_fallback_ticks; /* env-ticks whose transfer phase ran in strict road order (see DESIGN.md) */
  uint64_t cars_exited;      /* cars that drove off an exit road (generated = live + exited + dropped) */
  uint64_t arrival_saturations; /* Philox arrivals dropped because one entry road already had 255 arrivals in that tick
                                   (must stay 0: te_create bounds the arrival rate far below; non-zero = misuse) */
} te_stats;

typedef struct te_handle te_handle;

/* Fills cfg with the reference defaults (traffic_env.py:11-25,33-43; traffic_test.py:80): 3x3 grid,
   length 250, rate 0.5, one env, Philox arrivals at 0.12 cars/s per side-lane. */
void te_default_config(te_config *cfg);

/* TrafficEnv.set_graph + seed_generator + reset_entrypoints (traffic_env.py:361-382, 250-253, 389-394)
   for num_envs instances; uploads the topology tables of GridRoad (roadgraph.py:26-64).  Rejects configurations
   outside what parity is established for: non-finite or non-positive rate / length / v0 / a / b / delta / T, and
   roads not longer than twice the farthest a car can travel in one tick. */
int te_create(const te_config *cfg, te_handle **out);
int te_destroy(te_handle *h);
int te_get_dims(const te_handle *h, te_dims *out);
const char *te_last_error(void);
/* Number of CUDA devices the library can see (0 and an error when the driver is missing): lets callers and the
   test-suite detect a GPU box without importing torch. */
int te_device_count(int32_t *count);

/* Topology tables as the device holds them (for tests): dest/nexts/phases int32[R], entry int32[num_entry]. */
int te_get_topology(const te_handle *h, int32_t *dest, int32_t *nexts, int32_t *phases, int32_t *entry);

/* TrafficEnv._reset (traffic_env.py:259-272) for the envs whose mask byte is non-zero (NULL = all).
   init_phase uint8[E, I] replaces action_space.sample(); NULL draws from the Philox stream. */
int te_reset(te_handle *h, const uint8_t *env_mask, const uint8_t *init_phase, int memspace, void *stream);

/* Injected arrival schedule (TE_ARRIVALS_INJECTED).  CSR over (env, tick): the entry roads of
   env e at arrival-process tick first_tick + t are roads[offsets[e*(horizon+1)+t] ..
   offsets[e*(horizon+1)+t+1]) in arrival order; offsets are absolute into roads.  Replaces the
   rand_car/rand pair that add_new_cars pulls from (traffic_env.py:274-283).  The arrival-process
   tick of an env counts the ticks it has executed since te_create and is NOT rewound by reset (the
   reference never re-seeds its generator, SURVEY 3.3).  Ticks outside [first_tick, first_tick +
   horizon) have no arrivals; call again with a later window to stream a long schedule.
   num_roads = length of roads[]; every offset must lie in [0, num_roads], each row non-decreasing, at most 255
   arrivals per env tick, every road an entry road - otherwise the call fails and the old schedule stays.
   Buffers are copied; always host pointers. */
int te_set_arrivals(te_handle *h, const int64_t *offsets, const int16_t *roads, int64_t num_roads, int64_t first_tick,
                    int32_t horizon);

/* One actor step = Repeater(k_ticks)._step (+ Remi when TE_REMI) for every env (traffic_test.py:37-64).
   actions uint8[E, I] (non-zero = 1); obs float[E, 2r+I]; reward float[E, I]; done uint8[E].  The tick loop
   of an env stops after the tick that overflowed.  TE_DEVICE: one kernel launch on `stream`, asynchronous.
   TE_HOST: synchronous; the batch is launched in slices; each finished slice's results travel to the host as compact
   wire records (see te_step_wire) while the next slices run, and helper threads of the handle expand them into the
   caller's arrays (TE_HOST_SLICES / TE_HOST_THREADS environment variables tune slices and threads). */
int te_step(te_handle *h, const uint8_t *actions, int32_t k_ticks, float *obs, float *reward, uint8_t *done,
            int memspace, void *stream);

/* te_step for a SUBSET of the envs: envs whose env_mask byte is zero are not stepped - their state, arrival stream and
   rows of obs / reward / done stay untouched.  For learners that step their env slots at different times (A3C worker
   threads, a3c.py:66-72: traffic_env_b200.pool.EnvPool steps whichever slots have an action ready). */
int te_step_masked(te_handle *h, const uint8_t *actions, const uint8_t *env_mask, int32_t k_ticks, float *obs, float *reward,
                   uint8_t *done, int memspace, void *stream);

/* n_steps actor steps in ONE launch under one controller decision: the env state stays in shared memory for
   n_steps * k_ticks ticks (<= 64); obs float[n_steps, E, 2r+I], reward float[n_steps, E, I], done uint8[n_steps, E] hold
   every actor step's results exactly as n_steps calls of te_step with the same action would produce them.
   controller TE_CTRL_GIVEN: `actions` uint8[E, I] is the input.  TE_CTRL_GREEDY: the kernel evaluates the reference's
   greedy controller (algorithms/greedy.py:14-16, its decision holds for `--spacing` = n_steps actor steps) on the ring
   counts at launch and writes the chosen actions to `actions` (nullable).  Not for TE_AUTO_RESET handles. */
enum te_controller { TE_CTRL_GIVEN = 0, TE_CTRL_GREEDY = 1 };
int te_step_multi(te_handle *h, int32_t n_steps, int32_t controller, uint8_t *actions, int32_t k_ticks, float *obs,
                  float *reward, uint8_t *done, int memspace, void *stream);
/* TE_CTRL_GREEDY launches of this handle take a new decision every `spacing` actor steps (greedy.py's --spacing: steps
   0, spacing, 2 spacing ... of the launch), so one launch can hold several decisions: a whole device-resident rollout
   segment of n_steps * k_ticks <= 64 ticks without the state leaving shared memory.  `actions` then receives
   uint8[ceil(n_steps / spacing)][E, I], one block per decision.  Results are those of ceil(n_steps / spacing) launches
   of `spacing` steps each.  0 (the default): one decision per launch. */
int te_set_controller_spacing(te_handle *h, int32_t spacing);

/* Env-slot pool for learner threads (a3c.py:66-72: FLAGS.threads workers, each stepping its own env): te_pool_step
   queues slot `slot`'s action (uint8[I]) and blocks until that slot has been advanced by one actor step of k_ticks ticks;
   whichever caller finds no launch in flight becomes the leader and advances every slot queued so far with one
   te_step_masked launch - no lock-step round, a slow learner only delays itself (a would-be leader waits once, at most
   linger_us, when fewer slots are queued than the previous launch served).  Thread-safe; one pool per handle, and the
   handle must not be stepped directly while a pool uses it.  te_pool_reset: TrafficEnv._reset of one slot with the
   given initial phases (uint8[I]); te_pool_cars: cars_on_roads of one slot (int32[R]). */
typedef struct te_pool te_pool;
int te_pool_create(te_handle *h, int32_t k_ticks, int32_t linger_us, te_pool **out);
int te_pool_destroy(te_pool *p);
int te_pool_step(te_pool *p, int32_t slot, const uint8_t *action, float *obs, float *reward, uint8_t *done);
int te_pool_reset(te_pool *p, int32_t slot, const uint8_t *init_phase);
int te_pool_cars(te_pool *p, int32_t slot, int32_t *out);
int te_pool_counters(te_pool *p, uint64_t *launches, uint64_t *stepped);
const char *te_pool_last_error(te_pool *p);

/* The same actor step with its results as compact WIRE RECORDS, one per env (what te_step(TE_HOST) moves over PCIe
   internally): u8 passed[r] | u8 detected[r] | f32 light[I] | f32 reward[I] | u8 done, `stride` bytes apart
   (te_wire_layout) - 2.5 x fewer bytes than the float observation; the integer-valued observation entries
   (passed <= 19 k_ticks, detected <= 18) travel as bytes, so k_ticks <= 13.  A consumer that feeds a policy can read the
   records directly; te_expand_wire turns `count` records into te_step's float obs[count, 2r+I] / reward / done arrays
   (host memory).  records: E * stride bytes, device memory (TE_DEVICE, asynchronous) or host memory (TE_HOST). */
typedef struct te_wire_layout_t {
  int32_t stride, passed, detected, light, reward, done; /* byte offsets inside one record */
  int32_t max_k_ticks;
  int32_t host_float_dma; /* 1: te_step(TE_HOST) has the copy engine write the float arrays instead of expanding
                             wire records on the host (few host cores per GPU, or TE_HOST_FLOAT_DMA=1 at te_create) */
} te_wire_layout_t;
int te_wire_layout(const te_handle *h, te_wire_layout_t *out);
int te_step_wire(te_handle *h, const uint8_t *actions, int32_t k_ticks, void *records, int memspace, void *stream);
int te_expand_wire(const te_handle *h, const void *records, int32_t count, float *obs, float *reward, uint8_t *done);
/* te_step_multi with wire records: records[n_steps][E][stride]. */
int te_step_multi_wire(te_handle *h, int32_t n_steps, int32_t controller, uint8_t *actions, int32_t k_ticks, void *records,
                       int memspace, void *stream);

/* One physics tick = bare TrafficEnv._step (traffic_env.py:224-248): obs int32[E, 2r+2I]
   (passed | detected | current_phase | elapsed), reward float[E, I], done uint8[E]. */
int te_step_raw(te_handle *h, const uint8_t *actions, int32_t *obs, float *reward, uint8_t *done, int memspace,
                void *stream);

/* TrafficEnv.remi_reward (traffic_env.py:384-387, 64-78): reward float[E, I]; clears waiting and passed_dst. */
int te_remi_reward(te_handle *h, float *reward, int memspace, void *stream);

/* cars_on_roads (traffic_env.py:214-218): out int32[E, R]. */
int te_cars_on_roads(te_handle *h, int32_t *out, int memspace, void *stream);

/* Device-resident greedy controller (algorithms/greedy.py:14-16): actions[e, i] =
   (cars(E-bound) + cars(W-bound) - cars(S-bound) - cars(N-bound)) < 0 at intersection i. */
int te_greedy_actions(te_handle *h, uint8_t *actions, int memspace, void *stream);

/* Full state of envs [env_begin, env_begin+count) in the reference's layout, host pointers, any may be
   NULL: leading/lastcar int32[count,R]; x, v float[count,R,20] (only live slots and the leading slot are
   meaningful, as in the reference); obs int32[count,2r+2I]; waiting int32[count,r];
   passed_dst uint8[count,I]; steps float[count]. */
int te_get_state(te_handle *h, int32_t env_begin, int32_t count, int32_t *leading, int32_t *lastcar, float *x,
                 float *v, int32_t *obs, int32_t *waiting, uint8_t *passed_dst, float *steps);
int te_set_state(te_handle *h, int32_t env_begin, int32_t count, const int32_t *leading, const int32_t *lastcar,
                 const float *x, const float *v, const int32_t *obs, const int32_t *waiting,
                 const uint8_t *passed_dst, const float *steps);

/* Snapshot records: the complete state of one env in one fixed-size, 16-byte-aligned blob, for bit-exact rewind,
   checkpoint / resume and cloning of envs.  A record holds a header (magic, format version, m, n, validate bit), the R
   real rows of the x and v ring planes exactly as the device holds them (slot 0 of a row is the packed header word:
   leading | lastcar << 8 | detected << 16 in the x plane, waiting in the v plane), the birth-tick plane w (TE_VALIDATE
   handles only), phase / passed_dst (u8) and elapsed (i32) of the I intersections, and the env's private scalars (episode
   tick counter, position in the Philox arrival stream, injected-schedule clock, reset counter, episode step / done flag /
   return statistics).  About 71 KB per 10x10 env, 7.8 KB per 3x3 env.  A record carries no env id.
   Continuation: arrivals and reset phases are keyed by (seed, env_id_base + slot) and a record restores only the
   position in that stream, so a loaded env continues exactly as the saved env would have when it sits in the same slot
   of a handle with the same configuration, seed and env_id_base; loaded into another slot it has the same state and
   continues that slot's own stream from the saved draw index (independent noise, what branching rollouts want).
   Not part of a record: the handle's te_stats counters, the trip-time buffer, the injected schedule itself and the
   controller spacing. */
typedef struct te_snapshot_layout_t {
  int32_t stride;                              /* bytes per record */
  int32_t x, v, w, phase, elapsed, passed_dst; /* byte offsets inside a record; w = -1 without TE_VALIDATE */
  int32_t scalars;                             /* library-private bytes from here on */
} te_snapshot_layout_t;
int te_snapshot_layout(const te_handle *h, te_snapshot_layout_t *out);
/* env_ids is always a host array; NULL = envs [0, count).  records: count * stride bytes in `memspace` (16-byte aligned
   in device memory).  te_save_envs gathers the listed envs into records (duplicates allowed).  TE_DEVICE: asynchronous,
   ordered on `stream` after earlier work on it (explicit env_ids are copied from the caller's pageable array, which may
   make the call wait for that stream); TE_HOST: synchronous. */
int te_save_envs(te_handle *h, const int32_t *env_ids, int32_t count, void *records, int memspace, void *stream);
/* te_load_envs scatters record j into env env_ids[j] (each id at most once); synchronous in both memspaces (`stream` is
   not used), like te_set_state.  Every record is checked on the device before anything is written - magic, version,
   m / n, the validate bit, every row's leading and lastcar in [1, 20) with the header word's top byte zero, phase and
   passed_dst in {0, 1} - and on a failure the call returns an error naming the first bad record and field and leaves
   every env untouched.  On a tame handle the same pass applies te_set_state's tame predicate to every live car and
   leading slot: one wild car moves the handle to the checked kernels for good, exactly as te_set_state does. */
int te_load_envs(te_handle *h, const int32_t *env_ids, int32_t count, const void *records, int memspace, void *stream);

/* *tame = 1 while the handle runs the unchecked arithmetic: its archetype is inside the supported ranges and every car ever
   handed to te_set_state was tame - x finite with |x| < 2^40, v zero or in [2^-100, *v_cap], *v_cap = twice the fastest
   speed the archetype's dynamics can produce.  Tame state stays tame under the step, and no operand of the IDM update can
   then leave the domain on which its fast sequences are exact, so the per-car validity predicate and the generic
   fallback are not compiled into the kernels that run (DESIGN.md section 4).  One wild car in te_set_state switches the
   handle to the checked kernels for good.  v_cap may be NULL. */
int te_is_tame(const te_handle *h, int32_t *tame, float *v_cap);
/* The speed cap of the tame domain for an archetype / tick length / road length, 0 when the archetype is outside the
   supported ranges (host arithmetic only: needs no device). */
int te_tame_speed_cap(const float *archetype, float rate, float length, float *v_cap);

/* Counters since te_create (device -> host; synchronises the device). */
int te_get_stats(te_handle *h, te_stats *out);

/* Trip times recorded in validate mode (advance_hack, traffic_env.py:139-157): seconds between a car's
   arrival and its leaving the map, one (env, trip) pair per car, sorted by env and, within an env, in the
   order the reference appends them (tick, road index, pop order).  *count receives the number available;
   up to cap pairs are copied (either output may be NULL).  `clear` empties the device buffer afterwards. */
int te_get_trip_times(te_handle *h, int32_t *env_out, float *trip_out, int64_t cap, int64_t *count, int clear);
/* (returns 1, not an error, when more trips happened since the last clear than the device buffer - max(2^20, 64 E)
   records - holds: the recorded ones are returned and `clear` is honoured; te_last_error() has the counts) */

int te_synchronize(te_handle *h);

/* Page-locked host memory for the TE_HOST entry points (so their copies run at full PCIe rate and
   asynchronously to the launch); plain cudaHostAlloc / cudaFreeHost behind a C signature. */
int te_host_alloc(uint64_t bytes, void **out);
int te_host_free(void *ptr);

/* Kernel time of the last te_step/te_step_raw launch in milliseconds (CUDA events on the launch stream). */
int te_last_kernel_ms(te_handle *h, float *ms);

/* HBM bandwidth (GB/s, read + written bytes) of the step kernel's stage-in + flush alone: the same bulk-TMA
   copies with the same CTA shape and shared-memory footprint, no ticks in between.  The state is rewritten
   unchanged.  Used by bench.py to report what the flush achieves against the HBM peak. */
int te_stage_bandwidth(te_handle *h, int32_t repeats, double *gbytes_per_sec);

/* Arithmetic-only ceiling of the path: vehicle-updates/s of a micro-kernel in which every lane does nothing but
   dependent IDM updates (traffic_env.py:50-62) in registers.  Used by bench.py as the compute roofline of the step
   kernel.  form: -1 = the form the step kernels run for this archetype on a tame handle (5 or 0), 0 = the general form
   (checked: archetype flags tested, validity predicate and generic fallback), 5 = the tame form (the reference's
   archetype flags known at compile time, no predicate; needs T and rate powers of two and delta = 4); any other form is
   an error.  warps_per_sm: 0 = 2048 resident threads per SM, else one CTA of that many warps per SM (1..32). */
int te_idm_peak_form(int device, const float *archetype, float rate, int32_t iters, int32_t form, int32_t warps_per_sm,
                     double *updates_per_sec);

/* ---- test hooks (host pointers): device arithmetic exposed for bit-exactness tests */
/* out[i] = device restatement of glibc powf(x[i], y) (numba lowers float32 ** to libm powf). */
int te_test_powf(int device, const float *x, float y, float *out, int64_t n);
/* One IDM update per element (traffic_env.py:50-62): follower (x,v) behind leader (xl,vl,ll). */
int te_test_idm(int device, float rate, const float *archetype, const float *xl, const float *vl, const float *ll,
                const float *x, const float *v, float *x_out, float *v_out, int64_t n);
/* The same through the tame form (valid for tame operands only).  An error when the archetype and tick length would not
   run it (T and rate powers of two, delta = 4, archetype inside the tame ranges). */
int te_test_idm_tame(int device, float rate, const float *archetype, const float *xl, const float *vl, const float *ll,
                     const float *x, const float *v, float *x_out, float *v_out, int64_t n);
/* powf(r, 4) over every non-negative finite float r: out[0] = #r where RN_f32((r*r)*(r*r)) differs from the
   glibc algorithm, out[1] = largest distance (2^-52 units of the significand) of such a product from the float
   rounding boundary, out[2] = #r the shortcut filter with threshold tau declines, out[3] = #r it accepts although
   the results differ (the proof obligation: must be 0). */
int te_test_powf4_exhaustive(int device, uint64_t tau, uint64_t out[4]);
/* Philox4x32-10 block: out[4] for counter ctr[4], key[2]. */
int te_test_philox(int device, const uint32_t *ctr, const uint32_t *key, uint32_t *out);

#ifdef __cplusplus
}
#endif
#endif /* TRAFFIC_B200_H */
