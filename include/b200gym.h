/*
 * b200gym.h -- C ABI of the B200-native vectorised Gym environment engine.
 *
 * openai/gym 0.26.2 is pure Python: it has no FFI of its own.  The seam this
 * library sits behind is gym's Python plugin API -- a `gym.vector.VectorEnv`
 * subclass (reference gym/vector/vector_env.py:12-275) registered through
 * `gym.envs.registration.register` (gym/envs/registration.py:434-499).  The
 * entry points below are what such a subclass binds through ctypes (the stub
 * is shown in INTEGRATION.md and shipped as gym_b200/_lib.py); every one names
 * the reference behaviour it replaces.
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in signatures.  `stream` is a
 *     cudaStream_t passed as void* (NULL = legacy default stream).
 *   - "dev" pointers are device pointers owned by the caller (e.g. the
 *     data_ptr() of a torch.cuda tensor); "host" pointers are host memory.
 *   - every call returns 0 on success, non-zero on failure;
 *     b200gym_last_error() then describes the failure.
 *   - calls are asynchronous on `stream` unless stated otherwise; a handle is
 *     bound to one device and is not thread-safe.
 *   - there is NO CPU fallback: without a CUDA device create() fails.
 */
#ifndef B200GYM_H
#define B200GYM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200GYM_VERSION 2

/* Environment kinds: the dynamics classes on the hot path. */
enum b200gym_kind {
    B200GYM_CARTPOLE = 0,         /* gym/envs/classic_control/cartpole.py:130-207 */
    B200GYM_MOUNTAINCAR = 1,      /* gym/envs/classic_control/mountain_car.py:127-164 */
    B200GYM_MOUNTAINCAR_CONT = 2, /* gym/envs/classic_control/continuous_mountain_car.py:142-186 */
    B200GYM_PENDULUM = 3,         /* gym/envs/classic_control/pendulum.py:119-163 */
    B200GYM_ACROBOT = 4,          /* gym/envs/classic_control/acrobot.py:181-277,418-465 */
    B200GYM_LUNARLANDER = 5,      /* gym/envs/box2d/lunar_lander.py:308-600 (discrete, no wind); the Box2D
                                     arithmetic it delegates to is re-derived in csrc/lunar.cuh */
    B200GYM_BIPEDALWALKER = 6,    /* gym/envs/box2d/bipedal_walker.py:277-606 (non-hardcore); Box2D arithmetic
                                     re-derived in csrc/b2lite.cuh */
    B200GYM_LUNARLANDER_CONT = 7, /* LunarLanderContinuous-v2 = LunarLander(continuous=True), gym/envs/__init__.py:71-77,
                                     lunar_lander.py:152-160,479-481,496-533: Box(2) float32 actions */
    B200GYM_BIPEDALWALKER_HARDCORE = 8, /* BipedalWalkerHardcore-v3 = BipedalWalker(hardcore=True), gym/envs/__init__.py:79-85,
                                     bipedal_walker.py:300-373: stumps, stairs and pits as static polygons */
    B200GYM_NUM_KINDS = 9
};

/* b200gym_config.flags */
#define B200GYM_LUNAR_ENABLE_WIND 1 /* LunarLander(enable_wind=True), lunar_lander.py:449-477 */

/* dtype codes for the `actions` argument of b200gym_step */
enum b200gym_action_dtype {
    B200GYM_ACT_I64 = 0, /* Discrete: int64 (numpy default, MultiDiscrete dtype; gym/vector/utils/spaces.py:53-60) */
    B200GYM_ACT_I32 = 1,
    B200GYM_ACT_U8 = 2,
    B200GYM_ACT_F32 = 3  /* Box: float32 [n][act_dim] */
};

/*
 * Construction arguments: what `gym.make(id, **kwargs)` resolves from the
 * registry (gym/envs/__init__.py:11-60, gym/envs/registration.py:502-691).
 */
typedef struct b200gym_config {
    int32_t kind;              /* enum b200gym_kind */
    int32_t max_episode_steps; /* TimeLimit (gym/wrappers/time_limit.py:39-68); <= 0: no limit */
    int32_t autoreset;         /* 1: SyncVectorEnv same-step autoreset (gym/vector/sync_vector_env.py:152-156);
                                  0: plain Env semantics (state keeps evolving after termination) */
    int32_t flags;             /* B200GYM_LUNAR_ENABLE_WIND, else 0 */
    double param[4];           /* param[0]: Pendulum `g` (pendulum.py:95), MountainCar* `goal_velocity`
                                  (mountain_car.py:103, continuous_mountain_car.py:108), LunarLander* `gravity`
                                  (lunar_lander.py:195,210-213; must lie in (-12, 0) like the reference asserts -- the
                                  reference's default is -10.0; 0.0 is rejected, not defaulted);
                                  param[1], param[2]: LunarLander* `wind_power`, `turbulence_power`
                                  (lunar_lander.py:197-198), read only with B200GYM_LUNAR_ENABLE_WIND */
} b200gym_config;

typedef struct b200gym b200gym_t;

/* static shape queries (host only, no device needed) */
int b200gym_obs_dim(int kind);     /* observation_space.shape[0] */
int b200gym_act_dim(int kind);     /* 0: Discrete; k: Box(k,) float32 */
int b200gym_num_actions(int kind); /* Discrete n (0 for Box) */
int b200gym_state_dim(int kind);   /* float64 words of integrator state per env */
int b200gym_version(void);

/* Message for the last failing call on `h` (h == NULL: last create failure). */
const char *b200gym_last_error(const b200gym_t *h);

/*
 * Replaces: SyncVectorEnv.__init__ building num_envs Python env objects
 * (gym/vector/sync_vector_env.py:45-76).  Allocates the persistent SoA state
 * for `num_envs` environments in the HBM of CUDA device `device`:
 * float64 state[state_dim][n], int32 elapsed[n], PCG64 rng[n] (32 B records).
 */
int b200gym_create(const b200gym_config *cfg, int64_t num_envs, int device, b200gym_t **out);
/* Replaces: VectorEnv.close (gym/vector/vector_env.py:182-206). */
void b200gym_destroy(b200gym_t *h);

int64_t b200gym_num_envs(const b200gym_t *h);
int b200gym_device(const b200gym_t *h);

/*
 * Replaces: the `seed + i` fan-out of SyncVectorEnv.reset_wait
 * (gym/vector/sync_vector_env.py:106-107) followed, per env, by
 * Env.reset(seed=) -> seeding.np_random -> Generator(PCG64(SeedSequence(seed)))
 * (gym/core.py:149-151, gym/utils/seeding.py:9-27), done on the device.
 * Env i is seeded with the integer  base + first_index + i,  base given as four
 * little-endian uint32 words (base < 2^128).  `first_index` is the global index
 * of this handle's env 0 when a batch is sharded over GPUs.
 */
int b200gym_seed_range(b200gym_t *h, const uint32_t base_words[4], int64_t first_index, void *stream);
/*
 * Per-env seeds (reset(seed=[s0, s1, ...])).  ent_host: [n][4] little-endian
 * uint32 words; mask_host: [n] bytes, 0 = leave that env's stream untouched
 * (a None entry), may be NULL.  Synchronous (copies from pageable host memory).
 */
int b200gym_seed_each(b200gym_t *h, const uint32_t *ent_host, const uint8_t *mask_host, void *stream);

/*
 * Replaces: SyncVectorEnv.reset_wait's loop of env.reset() calls
 * (gym/vector/sync_vector_env.py:90-129; per env e.g. cartpole.py:190-207).
 * Every env whose mask byte is non-zero (mask_dev == NULL: all) draws a new
 * initial state from its own PCG64 stream, zeroes its TimeLimit counter and
 * writes its float32 observation row obs_dev[i][0..obs_dim).
 * bounds_host: NULL for the defaults, else two doubles: {low, high} of
 * options={"low","high"} (classic_control/utils.py:17-46) or {x_init, y_init}
 * for Pendulum (pendulum.py:147-152).  Validation of the bounds (low <= high,
 * castable) is the caller's job, as in the reference it happens in Python.
 */
int b200gym_reset(b200gym_t *h, const uint8_t *mask_dev, const double *bounds_host,
                  float *obs_dev, void *stream);

/*
 * Replaces: SyncVectorEnv.step_wait (gym/vector/sync_vector_env.py:135-169) =
 * for every env: TimeLimit.step (time_limit.py:39-56) around Env.step (e.g.
 * cartpole.py:130-188) and, when the episode ended and cfg.autoreset, the
 * unseeded env.reset() of the same call (:152-156).  Classic-control kinds: ONE kernel launch.  Box2D
 * kinds: three launches -- the step kernel, the continuous-collision (TOI) kernel over the envs whose step
 * may contain a TOI event, and (with cfg.autoreset) the compacted resets of the envs whose episode ended.
 *   actions_dev   [n] integers of `action_dtype`, or [n][act_dim] float32
 *   obs_dev       [n][obs_dim] float32   post-autoreset observation
 *   reward_dev    [n] float64            (SyncVectorEnv._rewards dtype, :69)
 *   terminated_dev, truncated_dev [n] uint8 (0/1)
 *   final_obs_dev [n][obs_dim] float32 or NULL: rows written only where
 *                 terminated|truncated (info["final_observation"], :155)
 * Out-of-range Discrete actions (the reference raises AssertionError,
 * cartpole.py:132) leave that env untouched, set reward NaN and bump a sticky
 * device counter read by b200gym_invalid_actions().
 */
int b200gym_step(b200gym_t *h, const void *actions_dev, int action_dtype, float *obs_dev,
                 double *reward_dev, uint8_t *terminated_dev, uint8_t *truncated_dev,
                 float *final_obs_dev, void *stream);

/* Number of invalid Discrete actions seen since the last call (synchronises `stream`). */
int b200gym_invalid_actions(b200gym_t *h, void *stream, int64_t *count_out);

/* 1 when some kernel launched on this handle has met an invalid Discrete action since the last
 * b200gym_invalid_actions() / b200gym_step_host(), 0 otherwise, -1 on a null handle.  Never synchronises: the
 * kernels raise a flag in page-locked host memory, so a caller that must not stall its stream (the torch backend)
 * can poll this before every step and raise the reference's error (cartpole.py:132, mountain_car.py:128-130,
 * acrobot.py:199, lunar_lander.py:482-484: `assert self.action_space.contains(action)`) one call late instead of
 * never. */
int b200gym_invalid_seen(const b200gym_t *h);

/*
 * Host-buffer step: the same call for a caller that lives on the CPU (what a
 * numpy agent does with SyncVectorEnv.step: numpy actions in, numpy results
 * out).  Copies the actions host->device and runs the step kernel with the
 * library's page-locked, device-mapped staging buffers as its output arrays:
 * the kernel's own stores (bulk shared->global copies of 256-env tiles) are the
 * device->host transfer.  Pipelined over up to 4 chunks of the env range on two
 * streams so that both PCIe directions overlap; returns when all results have
 * landed in host memory.
 *   actions_host  [n] integers of `action_dtype` / [n][act_dim] float32, or
 *                 NULL = the library's page-locked staging buffer (see below)
 *   obs_host, reward_host, terminated_host, truncated_host
 *                 NULL = results stay in the staging buffers (the fast path); otherwise they are
 *                 additionally copied there on the host
 *   final_obs_host destination (only the rows of envs that finished are written), or NULL = final
 *                 observations are not transferred
 * Page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory) buffers
 * copy at full PCIe speed; pageable memory works but is staged by the driver.
 * b200gym_host_buffers() exposes the library's own page-locked staging buffers
 * so a caller can fill actions / read results in place.
 */
typedef struct b200gym_host_io {
    void *actions;       /* [n] int64  or [n][act_dim] float32 */
    float *obs;          /* [n][obs_dim] */
    double *reward;      /* [n] */
    uint8_t *terminated; /* [n] */
    uint8_t *truncated;  /* [n] */
    float *final_obs;    /* [n][obs_dim] */
} b200gym_host_io;
int b200gym_host_buffers(b200gym_t *h, b200gym_host_io *out);
int b200gym_step_host(b200gym_t *h, const void *actions_host, int action_dtype, float *obs_host,
                      double *reward_host, uint8_t *terminated_host, uint8_t *truncated_host,
                      float *final_obs_host, int64_t *invalid_out /* out-of-range Discrete actions seen (and
                      cleared) by this call; may be NULL */);
/* reset() with the observations delivered to host memory (obs_host NULL = staging). */
int b200gym_reset_host(b200gym_t *h, const uint8_t *mask_host, const double *bounds_host, float *obs_host);

/*
 * State access (parity harness, checkpointing; the reference exposes
 * `env.state` / `env.unwrapped.state` as a Python attribute).
 * state_dev: float64 [n][state_dim] (AoS on the wire; the library converts
 * from/to its SoA layout), elapsed_dev: int32 [n], rng_dev: uint64 [n][4] =
 * {state_hi, state_lo, inc_hi, inc_lo} of numpy's PCG64.  Any pointer may be NULL.
 */
int b200gym_get_state(b200gym_t *h, double *state_dev, int32_t *elapsed_dev, uint64_t *rng_dev, void *stream);
int b200gym_set_state(b200gym_t *h, const double *state_dev, const int32_t *elapsed_dev,
                      const uint64_t *rng_dev, void *stream);

/*
 * LunarLander only (state_dim is 0 for it; get/set_state handle the TimeLimit counters and RNG):
 * the three rigid bodies {lander, leg(-1), leg(+1)} of every env as float32 [n][18] =
 * 3 x {c.x, c.y, angle, v.x, v.y, omega} and int32 [n][6] = {game_over, leg0 contact, leg1 contact,
 * awake, elapsed, #touching contacts} -- what `env.lander.position` etc. expose in the reference.
 */
int b200gym_lunar_get_bodies(b200gym_t *h, float *bodies_dev, int32_t *flags_dev, void *stream);
/*
 * LunarLander with B200GYM_LUNAR_ENABLE_WIND: the per-env wind phase counters.  Replaces
 * `self.wind_idx = np.random.randint(-9999, 9999)` / `self.torque_idx = ...` of LunarLander.__init__
 * (lunar_lander.py:234-235; drawn from numpy's GLOBAL generator, once per env object, advanced by one per windy
 * step and never reset): the caller draws them and hands them over.  set != 0: copy the two host arrays [n] into
 * the env state; set == 0: read them back.  Synchronous.
 */
int b200gym_lunar_wind_idx(b200gym_t *h, int32_t *wind_idx_host, int32_t *torque_idx_host, int set);
/* BipedalWalker: float32 [n][30] = 5 x {c.x, c.y, angle, v.x, v.y, omega} (hull, leg(-1), lower(-1), leg(+1),
 * lower(+1)) and int32 [n][4] = {game_over, legs[1] contact, legs[3] contact, #touching contacts}. */
int b200gym_walker_get_bodies(b200gym_t *h, float *bodies_dev, int32_t *flags_dev, void *stream);
/* BipedalWalker*: what `env.terrain_y` (bipedal_walker.py:377) and the `fd_polygon` static bodies of the hardcore
 * terrain (:309-316,336,365) hold: float32 terrain_dev[n][200]; polys_dev[n][40][4] = {x0, y_low, x1, y_high} of each
 * obstacle box in creation order (unused rows 0) and int32 npoly_dev[n] (both may be NULL). */
int b200gym_walker_get_terrain(b200gym_t *h, float *terrain_dev, float *polys_dev, int32_t *npoly_dev, void *stream);

/*
 * Multi-GPU: fused step + all-gather over NVLink peer memory.
 *
 * Replaces (no reference counterpart in gym; nearest analogue: AsyncVectorEnv gathering worker
 * results through shared memory, gym/vector/async_vector_env.py:319-328,
 * gym/vector/utils/shared_memory.py:164-170).  One process per GPU; rank r of `world` owns the
 * global envs [r*n, (r+1)*n).  Every rank allocates one "gather allocation" holding two sets
 * (double buffering by step parity) of the GLOBAL result arrays
 *     obs float32 [world*n][obs_dim], reward float64 [world*n], terminated/truncated uint8 [world*n]
 * plus a flag word per rank, exports it as a CUDA IPC handle (b200gym_p2p_create), maps the
 * peers' allocations (b200gym_p2p_connect, after the caller has all-gathered the 64-byte
 * handles, e.g. with torch.distributed), and from then on b200gym_step_p2p() runs the fused step
 * kernel in its gather form: each 256-env tile of results is assembled in shared memory and pushed
 * to this rank's rows of the local set AND, through the mapped peer pointers, of every peer's set
 * with bulk shared->global copies (cp.async.bulk over NVLink 5 / NVSwitch) -- the all-gather is the
 * kernel's own store stream, tile by tile, overlapped with the arithmetic of the other tiles, with
 * no separate collective and no extra pass over the data.  (Shards whose rows are not 16-byte
 * aligned, ragged tails and the Box2D tasks use per-thread peer stores instead.)  The step ends
 * with ONE 1-warp kernel on `stream`: each rank publishes "my rows of step k are complete" to all
 * peers (system-scope fence + flag store) and waits on its own flag words for theirs, for at most
 * B200GYM_P2P_TIMEOUT_S seconds (default 30): a lost peer is recorded, not waited for for ever
 * (b200gym_p2p_status).
 */
#define B200GYM_MAX_PEERS 7
typedef struct b200gym_p2p_layout {
    void *base;            /* device pointer of this rank's gather allocation */
    uint64_t set_bytes;    /* set s (0/1) starts at base + s*set_bytes */
    uint64_t off_obs, off_reward, off_terminated, off_truncated; /* byte offsets inside a set */
    int64_t rows;          /* world * n */
} b200gym_p2p_layout;
int b200gym_p2p_create(b200gym_t *h, int world, int rank, void *ipc_handle_out /* 64 bytes */,
                       b200gym_p2p_layout *layout_out);
int b200gym_p2p_connect(b200gym_t *h, const void *all_ipc_handles /* world x 64 bytes, rank order */);
/* *set_out = which set (0/1) holds this step's global results once `stream` reaches this point */
int b200gym_step_p2p(b200gym_t *h, const void *actions_dev, int action_dtype, float *final_obs_dev,
                     void *stream, int *set_out);
/* Synchronises `stream`; *timed_out_peer = -1 when every step barrier so far completed, else the rank
 * whose rows did not arrive in time (the call then fails). */
int b200gym_p2p_status(b200gym_t *h, void *stream, int *timed_out_peer);

/*
 * Vector-aware wrappers of the reference, on the device (SURVEY.md 8f).  All state lives in caller-owned
 * device buffers; the stateless utilities report errors through b200gym_last_error(NULL) and run on the
 * device their buffers live on.
 *
 * RecordEpisodeStatistics (gym/wrappers/record_episode_statistics.py:79-151), fused INTO the step kernels:
 * after b200gym_set_episode_stats() every step launch also keeps the float32 return / int32 length
 * accumulators (`episode_returns += rewards` on a float32 array: add in float64, round to float32),
 * writes infos["episode"]["r"/"l"] for the envs whose episode ended in that step (the `_episode` mask is
 * terminated | truncated) and appends them to a ring of `ring_size` recent episodes (return_queue /
 * length_queue); *counter_dev counts finished episodes.  ring_dev[k] = (uint64)length << 32 | float32 bits
 * of the return, one store per episode into slot (episode number mod ring_size); episodes that finish in
 * the same step are numbered in no particular order (the reference appends them in env order), and when
 * more than ring_size finish at once the ring keeps an arbitrary ring_size of them.  The pointers may be
 * changed between steps (double buffering of the r / l rows); return_acc_dev == NULL switches it off.
 * No extra launch, no extra pass over reward / flags.
 */
int b200gym_set_episode_stats(b200gym_t *h, float *return_acc_dev, int32_t *length_acc_dev, float *episode_r_dev,
                              int32_t *episode_l_dev, uint64_t *ring_dev, uint64_t *counter_dev, int ring_size);
/* The same bookkeeping as ONE stand-alone launch over arbitrary (reward, terminated, truncated) device arrays --
 * e.g. the gathered global tensors of a sharded env; also writes the `_episode` mask. */
int b200gym_episode_stats(const double *reward_dev, const uint8_t *terminated_dev, const uint8_t *truncated_dev,
                          float *return_acc_dev, int32_t *length_acc_dev, float *episode_r_dev, int32_t *episode_l_dev,
                          uint8_t *episode_mask_dev, uint64_t *ring_dev, uint64_t *counter_dev,
                          int ring_size, int64_t n, void *stream);
/*
 * NormalizeObservation / NormalizeReward (gym/wrappers/normalize.py:8-144): RunningMeanStd over the batch axis in
 * two launches per step and ONE pass over the batch for the moments.
 *   stats   float64 [2][2*dim + 1] = {mean[dim], var[dim], count}, double-buffered: a step reads set `cur` and
 *           writes set `cur ^ 1` (initialise set 0 to mean 0, var 1, count 1e-4: normalize.py:11-15)
 *   scratch float64 [2][2*dim]     = per-column sums of (x - mean) and (x - mean)^2 of THIS step's batch,
 *           accumulated into set `cur` (zero on first use; the apply launch clears the other set)
 * b200gym_rms_moments      one coalesced pass over x [n][dim] (float32, or float64 with is_f64): sums into scratch
 * b200gym_return_moments   NormalizeReward.step's `returns = returns * gamma + reward` (normalize.py:130) fused
 *                          with the same pass over `returns`
 * (a sharded env all-reduces scratch[cur] over the GPUs here and passes the GLOBAL row count as batch_count)
 * b200gym_rms_apply_obs    Chan update (normalize.py:32-46) of stats[cur] with the batch moments into stats[cur^1]
 *                          when `update`, then out = (obs - mean) / sqrt(var + epsilon) with the NEW statistics
 * b200gym_rms_apply_reward same update, out = reward / sqrt(var + epsilon) (normalize.py:143),
 *                          returns[terminated | truncated] = 0 (:135-136)
 * dim must be one of 1, 2, 3, 4, 6, 8, 24 (the observation sizes of the in-scope envs).
 */
int b200gym_rms_moments(const void *x_dev, int is_f64, int64_t n, int dim, const double *stats_dev, double *scratch_dev,
                        void *stream);
int b200gym_return_moments(double *returns_dev, const double *reward_dev, double gamma, int64_t n, const double *stats_dev,
                           double *scratch_dev, void *stream);
int b200gym_rms_apply_obs(const float *obs_dev, float *out_dev, int64_t n, int dim, const double *stats_dev,
                          double *stats_next_dev, const double *scratch_dev, double *scratch_next_dev, double batch_count,
                          double epsilon, int update, void *stream);
int b200gym_rms_apply_reward(const double *reward_dev, double *out_dev, double *returns_dev, const uint8_t *terminated_dev,
                             const uint8_t *truncated_dev, int64_t n, const double *stats_dev, double *stats_next_dev,
                             const double *scratch_dev, double *scratch_next_dev, double batch_count, double epsilon,
                             void *stream);

/*
 * Box2D tasks: number of envs in which a touching (body, ground fixture) pair was ever dropped because the scene's
 * manifold table was full (8 pairs for LunarLander*, 10 for BipedalWalker*; real Box2D has no such limit).  The
 * dropped pair is treated as not touching -- the CPU oracle applies the identical rule -- so this counts
 * "physics differs from Box2D here"; it is 0 in every workload measured so far (max 7 simultaneous pairs).
 * Synchronises `stream`.
 */
int b200gym_box2d_overflows(b200gym_t *h, void *stream, int64_t *count_out);

/*
 * Device self-test of the kernels' constant-divisor division (csrc/envs.cuh:div_by_const)
 * against IEEE `/`: `samples` pseudo-random doubles (both signs, 64 binades) x 4 divisors.
 * Synchronous; *mismatches_out must come back 0.
 */
int b200gym_selftest(int device, int64_t samples, uint64_t seed, int64_t *mismatches_out);
/*
 * Device self-test of the float64 sin / cos / x**2 the dynamics use (csrc/glibc_trig.cuh: glibc's results, bit for
 * bit): evaluates them on x_dev[n]; the caller compares with its own libm (math.sin, math.cos, math.pow(x, 2.0)).
 * sq_dev may be NULL.  Asynchronous.
 */
int b200gym_selftest_trig(const double *x_dev, int64_t n, double *sin_dev, double *cos_dev, double *sq_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* B200GYM_H */
