// b200gym.cu -- kernels + C ABI of the B200-native vectorised Gym engine.
//
// Hot path (reference: SyncVectorEnv.step_wait, gym/vector/sync_vector_env.py:135-169):
//   ONE kernel launch per vector step; one thread per environment instance;
//   Env.step + TimeLimit + same-step autoreset (with the env's own PCG64
//   stream) + observation/reward/flag emission fused.
//
// HBM layout (persistent, owned by the handle)
//   state   float64 [S][n]   SoA: lane i of a warp reads word k of env i -> 256 B
//                            contiguous per warp per word, fully coalesced
//   elapsed int32   [n]      TimeLimit._elapsed_steps
//   flags   uint8   [n]      bit0: "already terminated" (plain-Env mode only)
//   rng     uint64  [n][4]   numpy PCG64 {state_hi, state_lo, inc_hi, inc_lo}; AoS,
//                            touched only by lanes that reset
// I/O buffers are caller-owned (torch.cuda tensors): actions in; obs [n][D]
// float32, reward float64 [n], terminated/truncated uint8 [n], final_obs [n][D].
//
// Built for sm_100a only, with -fmad=false (see envs.cuh).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <type_traits>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>

#include "../../include/b200gym.h"
#include "envs.cuh"
#include "lunar.cuh"
#include "walker.cuh"
#include "box2d_consts.h"
#include "rng.cuh"

using namespace bgym;

// ---------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------
struct b200gym {
    b200gym_config cfg;
    int64_t n = 0;
    int device = 0;
    int S = 0, D = 0, A = 0, NACT = 0;
    double *state = nullptr;
    int32_t *elapsed = nullptr;
    uint8_t *flags = nullptr;
    uint64_t *rng = nullptr;
    uint32_t *lunar_rec = nullptr;          // LunarLander / BipedalWalker: solver record, kWords 32-bit words per env, SoA
    bool is_lunar = false, is_walker = false;
    lunar::Opts lunar_opts{};
    unsigned long long *invalid = nullptr;  // sticky device counter
    unsigned long long *invalid_seen = nullptr;      // page-locked, device-mapped word: set to 1 by any kernel that meets an
    unsigned long long *invalid_seen_dev = nullptr;  // invalid action (host-visible WITHOUT a synchronisation); device alias
    struct {                                // caller-owned buffers of the fused RecordEpisodeStatistics (all null = off)
        float *acc = nullptr; int32_t *len = nullptr; float *r = nullptr; int32_t *l = nullptr;
        unsigned long long *ring = nullptr, *counter = nullptr; int ring_size = 0;
    } ep;
    int sm_count = 148;
    int occ[B200GYM_NUM_KINDS][3][2] = {};  // cached CTAs/SM of step_kernel_persistent per (kind, action width, lean)
    int kernel_choice = 2;                  // 0: kernel A (one tile per CTA), 1: kernel P (resident grid, asynchronous
                                            // prefetch, deferred resets), 2: P's lean instantiation where it applies
                                            // (else P); B200GYM_KERNEL=a|p|l overrides
    // Box2D tasks (see launch_box2d_step)
    int32_t *toi_list = nullptr;            // [n] env offsets parked for the TOI kernel, per launch range
    int32_t *toi_count = nullptr;           // [kResetSlots]
    uint32_t *toi_mid = nullptr;            // [kToiMidWords][n] SoA side buffer of the parked envs
    int32_t *reset_list = nullptr;          // [n] env offsets to reset, filled per launch range
    int32_t *reset_count = nullptr;         // [kResetSlots] one counter per concurrently running launch range
    // fused all-gather over peer memory (b200gym_p2p_*)
    struct {
        int world = 0, rank = 0;
        unsigned char *base = nullptr;               // this rank's gather allocation (2 sets + flags)
        unsigned char *peer[B200GYM_MAX_PEERS + 1] = {};  // peer[r]: rank r's allocation mapped here (own = base)
        size_t set_bytes = 0, off_obs = 0, off_reward = 0, off_term = 0, off_trunc = 0, off_flags = 0, bytes = 0;
        unsigned long long step = 0;
        unsigned long long timeout_ns = 30ull * 1000000000ull;   // B200GYM_P2P_TIMEOUT_S overrides
        bool connected = false;
    } p2p;
    // host-I/O path (lazily created)
    b200gym_host_io hio{};
    b200gym_host_io dio{};  // device side: .actions in HBM; the result pointers are device aliases of hio's mapped buffers
    uint8_t *d_mask = nullptr;
    unsigned long long *h_invalid = nullptr;   // page-locked landing word of the invalid-action counter
    cudaEvent_t hevent = nullptr;
    unsigned long long **d_peer_flags = nullptr;
    cudaStream_t hstream[2] = {nullptr, nullptr};
    bool host_ready = false;
    mutable std::string err;
};

static thread_local std::string g_create_err;

static int fail(const b200gym *h, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    else g_create_err = buf;
    return 1;
}

#define CK(h, call)                                                                       \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(h, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

static const int k_obs_dim[B200GYM_NUM_KINDS] = {4, 2, 2, 3, 6, 8, 24, 8, 24};
static const int k_act_dim[B200GYM_NUM_KINDS] = {0, 0, 1, 1, 0, 0, 4, 2, 4};
static const int k_nact[B200GYM_NUM_KINDS] = {2, 3, 0, 0, 3, 4, 0, 0, 0};
static const int k_state_dim[B200GYM_NUM_KINDS] = {4, 2, 2, 2, 4, 0, 0, 0, 0};

static bool kind_ok(int k) { return k >= 0 && k < B200GYM_NUM_KINDS; }

extern "C" int b200gym_obs_dim(int kind) { return kind_ok(kind) ? k_obs_dim[kind] : -1; }
extern "C" int b200gym_act_dim(int kind) { return kind_ok(kind) ? k_act_dim[kind] : -1; }
extern "C" int b200gym_num_actions(int kind) { return kind_ok(kind) ? k_nact[kind] : -1; }
extern "C" int b200gym_state_dim(int kind) { return kind_ok(kind) ? k_state_dim[kind] : -1; }
extern "C" int b200gym_version(void) { return B200GYM_VERSION; }
extern "C" const char *b200gym_last_error(const b200gym_t *h) {
    return h ? h->err.c_str() : g_create_err.c_str();
}
extern "C" int64_t b200gym_num_envs(const b200gym_t *h) { return h ? h->n : -1; }
extern "C" int b200gym_device(const b200gym_t *h) { return h ? h->device : -1; }

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
constexpr int kThreads = 256;

struct StepArgs {
    double *state;
    int32_t *elapsed;
    uint8_t *flags;
    uint64_t *rng;
    unsigned long long *invalid;
    unsigned long long *invalid_seen;   // device-mapped host word, see b200gym_invalid_seen
    uint32_t *lunar_rec;
    const void *actions;
    float *obs;
    double *reward;
    uint8_t *terminated;
    uint8_t *truncated;
    float *final_obs;
    int64_t n;        // envs in the handle (SoA stride)
    int64_t first;    // sub-range processed by this launch
    int64_t count;
    int32_t max_steps;
    int32_t autoreset;
    double param0;
    lunar::Opts lunar_opts;   // LunarLander constructor variants (uniform over the batch)
    // Box2D tasks: envs whose episode ended in this launch are appended here (offset from `first`) and reset by
    // box2d_reset_list_kernel, which follows on the stream
    int32_t *reset_list;
    int32_t *reset_count;
    // Box2D tasks: envs whose step may contain a continuous-collision event (b2l::toi_needed) are parked after the
    // discrete solve -- world record + the sweep starts / env intermediates in toi_mid -- and finished by
    // box2d_toi_kernel, which follows on the stream, in warps full of such envs
    int32_t *toi_list;
    int32_t *toi_count;
    uint32_t *toi_mid;
    // RecordEpisodeStatistics fused into the step (b200gym_set_episode_stats; nullptr = off): float32 return and
    // int32 length accumulators, infos["episode"]["r"/"l"] rows of finishing envs, ring of recent episodes
    float *ep_acc;
    int32_t *ep_len;
    float *ep_r;
    int32_t *ep_l;
    unsigned long long *ep_ring, *ep_counter;
    int32_t ep_ring_size;
    int32_t bulk_sink;   // 1: use kernel G's staged bulk stores even without peers (host path: the output arrays are
                         // mapped host memory, where many small stores are what hurts)
    // fused all-gather (multi-GPU): every result is ALSO stored into the same rows of the peers'
    // gather buffers over NVLink (peer-mapped pointers, slice offset already applied)
    int32_t npeer;
    float *peer_obs[B200GYM_MAX_PEERS];
    double *peer_reward[B200GYM_MAX_PEERS];
    uint8_t *peer_term[B200GYM_MAX_PEERS];
    uint8_t *peer_trunc[B200GYM_MAX_PEERS];
};

template <int D, typename I>
__device__ __forceinline__ void store_row(float *base, I i, const float (&v)[D]) {
    if constexpr (D == 4) {
        reinterpret_cast<float4 *>(base)[i] = make_float4(v[0], v[1], v[2], v[3]);
    } else if constexpr (D == 2) {
        reinterpret_cast<float2 *>(base)[i] = make_float2(v[0], v[1]);
    } else if constexpr (D == 8 || D == 24) {
        float4 *p = reinterpret_cast<float4 *>(base) + (D / 4) * i;
#pragma unroll
        for (int k = 0; k < D / 4; k++) p[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
    } else if constexpr (D == 6) {
        float2 *p = reinterpret_cast<float2 *>(base) + 3 * i;
        p[0] = make_float2(v[0], v[1]);
        p[1] = make_float2(v[2], v[3]);
        p[2] = make_float2(v[4], v[5]);
    } else {
#pragma unroll
        for (int k = 0; k < D; k++) base[i * D + k] = v[k];
    }
}

template <int D, typename I>
__device__ __forceinline__ void store_obs_all(const StepArgs &a, I i, const float (&v)[D]) {
    store_row<D>(a.obs, i, v);
    for (int p = 0; p < a.npeer; p++) store_row<D>(a.peer_obs[p], i, v);
}

template <typename I>
__device__ __forceinline__ void store_scalars_all(const StepArgs &a, I i, double reward, uint8_t term,
                                                  uint8_t trunc) {
    a.reward[i] = reward;
    a.terminated[i] = term;
    a.truncated[i] = trunc;
    for (int p = 0; p < a.npeer; p++) {
        a.peer_reward[p][i] = reward;
        a.peer_term[p][i] = term;
        a.peer_trunc[p][i] = trunc;
    }
}

// RecordEpisodeStatistics.step (gym/wrappers/record_episode_statistics.py:103-151) for env i, fused into the step
// kernels: `episode_returns += rewards` on a float32 array with float64 rewards (add in float64, round to float32),
// `episode_lengths += 1`; on terminated | truncated emit both, append to the ring (return_queue / length_queue),
// start over from zero.
template <typename I>
__device__ __forceinline__ void episode_account(const StepArgs &a, I i, double reward, bool done) {
    if (!a.ep_acc) return;
    const float ret = (float)((double)a.ep_acc[i] + reward);
    const int32_t len = a.ep_len[i] + 1;
    if (done) {
        a.ep_r[i] = ret;
        a.ep_l[i] = len;
        const unsigned long long slot = atomicAdd(a.ep_counter, 1ULL);
        if (a.ep_ring_size > 0)   // one 64-bit store per episode {length : return bits}: a slot never mixes two episodes
            a.ep_ring[slot % (unsigned long long)a.ep_ring_size] =
                ((unsigned long long)(uint32_t)len << 32) | (unsigned long long)__float_as_uint(ret);
        a.ep_acc[i] = 0.0f;
        a.ep_len[i] = 0;
    } else {
        a.ep_acc[i] = ret;
        a.ep_len[i] = len;
    }
}

// Where the results of env i go.  DirectSink: straight to the caller's arrays (and, when peers are mapped,
// to theirs) with per-thread stores.  StagedSink: into the CTA's shared-memory tile, which leaves the SM as a few
// bulk copies per destination (step_kernel_gather).
// PEERS = false: the caller knows there are no peer-mapped destinations (single-GPU step), so the per-destination
// loops and their constant-bank traffic disappear from the hot loop.
template <bool PEERS>
struct DirectSinkT {
    const StepArgs &a;
    template <int D, typename I>
    __device__ __forceinline__ void obs(I i, const float (&v)[D]) const {
        if constexpr (PEERS) store_obs_all<D>(a, i, v);
        else store_row<D>(a.obs, i, v);
    }
    template <typename I>
    __device__ __forceinline__ void scalars(I i, double reward, uint8_t term, uint8_t trunc) const {
        if constexpr (PEERS) store_scalars_all(a, i, reward, term, trunc);
        else { a.reward[i] = reward; a.terminated[i] = term; a.truncated[i] = trunc; }
    }
};
using DirectSink = DirectSinkT<true>;

struct StagedSink {
    float *s_obs;
    double *s_reward;
    uint8_t *s_term, *s_trunc;
    int64_t base;   // env index of row 0 of the tile
    template <int D, typename I>
    __device__ __forceinline__ void obs(I i, const float (&v)[D]) const { store_row<D>(s_obs, (int)(i - base), v); }
    template <typename I>
    __device__ __forceinline__ void scalars(I i, double reward, uint8_t term, uint8_t trunc) const {
        const int r = (int)(i - base);
        s_reward[r] = reward; s_term[r] = term; s_trunc[r] = trunc;
    }
};

// Tuning knobs (overridable at build time for A/B measurements).
// The per-env work is one long dependent float64 chain and the SMs are latency-bound, but occupancy is not the
// lever: at 32 registers (8 CTAs x 256 threads = 64 warps/SM) the hot loop spills the state across the division
// slow-path calls, and those local-memory round trips cost more than the extra warps hide.  Measured on B200
// (CartPole, 2^20 envs, cold L2, median of 400 launches, profiles/r2b_register_budget_ab.txt):
//   32 registers / 8 CTAs: kernel A 26.7 us, P 28.7, lean P 30.7;  40 / 6: A 26.7, P 26.5, lean P 24.6;
//   48 / 5: A 26.7, P 24.6, lean P 24.6.   -> 6 CTAs/SM (40 registers, no spills in the lean loop).
#ifndef B200_MIN_CTAS
#define B200_MIN_CTAS 6
#endif
template <int KIND>
struct Tuning {
    // Acrobot (RK4, ~70 live doubles) would spill heavily below 64 registers.  (The MountainCar kinds fit 32 registers
    // without a spill, which makes BASELINE's 2^18 envs one round of tiles instead of two -- measured: 10.1 vs 10.2 us,
    // no gain, so they keep the common budget.)
    static constexpr int kMinCtas = (KIND == B200GYM_ACROBOT) ? 3 : B200_MIN_CTAS;
};

// Phase 1, by the thread that owns env i (its inputs are in registers): Env.step, TimeLimit,
// stores of reward / flags / final_obs, and -- unless the episode ended -- of the new state and
// observation.  Returns true when the env must be reset by phase 2.
template <int KIND, bool EP = true, typename Sink, typename I>
__device__ __forceinline__ bool advance_env(const StepArgs &a, const Sink &sink, I i, double (&s)[Env<KIND>::S],
                                            int32_t elapsed, long long action_int, float a0) {
    using E = Env<KIND>;
    int act = 0;
    if constexpr (E::A == 0) {
        if (action_int < 0 || action_int >= E::NACT) {
            // the reference raises (cartpole.py:132 / mountain_car.py:128-130 / acrobot.py:199): leave the env
            // untouched, count it (sticky), return a NaN reward and the env's CURRENT observation, so that the
            // double-buffered output row does not show the observation of two steps ago
            atomicAdd(a.invalid, 1ULL);
            *reinterpret_cast<volatile unsigned long long *>(a.invalid_seen) = 1ULL;
            float cur[E::D];
            E::observe(s, cur);
            sink.scalars(i, __longlong_as_double(0x7ff8000000000000LL), 0, 0);
            sink.template obs<E::D>(i, cur);
            return false;
        }
        act = (int)action_int;
    }

    float obs[E::D];
    double reward;
    bool terminated;
    E::step(s, elapsed == 0, act, a0, a.param0, obs, reward, terminated);

    if (!a.autoreset) {
        if constexpr (KIND == B200GYM_CARTPOLE) {
            // cartpole.py:169-184: reward 0.0 once the pole has already fallen
            const uint8_t f = a.flags[i];
            if (terminated) {
                if (f & 1) reward = 0.0;
                else a.flags[i] = f | 1;
            }
        }
    }

    elapsed += 1;                                                        // time_limit.py:51
    const bool truncated = (a.max_steps > 0) && (elapsed >= a.max_steps);  // :53-54
    const bool needs_reset = (terminated || truncated) && a.autoreset;   // sync_vector_env.py:152-156

    sink.scalars(i, reward, terminated ? 1 : 0, truncated ? 1 : 0);
    if constexpr (EP) episode_account(a, i, reward, terminated || truncated);
    if (needs_reset) {
        if (a.final_obs) store_row<E::D>(a.final_obs, i, obs);           // info["final_observation"]
    } else {
#pragma unroll
        for (int k = 0; k < E::S; k++) a.state[k * a.n + i] = s[k];
        a.elapsed[i] = elapsed;
        sink.template obs<E::D>(i, obs);
    }
    return needs_reset;
}

// Phase 2: the unseeded env.reset() of the autoreset (sync_vector_env.py:154) for env i, by
// whichever thread picked it off the CTA's compacted list.
template <int KIND, typename Sink, typename I>
__device__ __forceinline__ void reset_env(const StepArgs &a, const Sink &sink, I i) {
    using E = Env<KIND>;
    double s[E::S];
    float obs[E::D];
    Pcg64 g = pcg64_load(a.rng + 4 * (size_t)i);
    double lo, hi;
    E::default_bounds(lo, hi);
    E::reset(s, g, lo, hi, obs);
    pcg64_store(a.rng + 4 * (size_t)i, g);
#pragma unroll
    for (int k = 0; k < E::S; k++) a.state[k * a.n + i] = s[k];
    a.elapsed[i] = 0;                                                    // time_limit.py:67
    sink.template obs<E::D>(i, obs);
}

// Why two phases: only ~1 env in 22 finishes per CartPole step, but then 77 % of the warps
// contain at least one finishing lane and would all walk the ~170-instruction PCG64 path
// (4 x 128-bit LCG steps) with 1-2 active lanes.  Instead finishing lanes push their env index
// onto a shared-memory list and, after one barrier, the first `count` threads of the CTA do
// the resets with full lanes: ~11 resets per 256-env tile = half a warp instead of 6 warps.

// --- kernel A: one thread per environment, inputs loaded straight from HBM -------------
// Used for small / ragged / unaligned batches and for the tail of kernel B.
template <int KIND, typename ActT>
__global__ void __launch_bounds__(kThreads, Tuning<KIND>::kMinCtas) step_kernel(const StepArgs a) {
    using E = Env<KIND>;
    __shared__ int reset_list[kThreads];
    __shared__ int reset_count;
    if (threadIdx.x == 0) reset_count = 0;
    __syncthreads();
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < a.count) {
        const int64_t i = a.first + j;
        double s[E::S];
#pragma unroll
        for (int k = 0; k < E::S; k++) s[k] = a.state[k * a.n + i];
        const int32_t elapsed = a.elapsed[i];
        long long action_int = 0;
        float a0 = 0.0f;
        const ActT av = __ldg(reinterpret_cast<const ActT *>(a.actions) + i);
        if constexpr (E::A == 0) action_int = (long long)av;
        else a0 = (float)av;
        if (advance_env<KIND>(a, DirectSink{a}, i, s, elapsed, action_int, a0)) reset_list[atomicAdd(&reset_count, 1)] = threadIdx.x;
    }
    __syncthreads();
    const int cnt = reset_count;
    if ((int)threadIdx.x < cnt)
        reset_env<KIND>(a, DirectSink{a}, a.first + (int64_t)blockIdx.x * blockDim.x + reset_list[threadIdx.x]);
}

// --- asynchronous-copy helpers (sm_100a PTX) --------------------------------------------------------
namespace acp {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// per-thread LDGSTS: global -> shared without a register in between (SASS LDGSTS)
template <int BYTES>
__device__ __forceinline__ void ld_async(void *smem_dst, const void *gmem_src) {
    static_assert(BYTES == 4 || BYTES == 8 || BYTES == 16, "cp.async moves 4, 8 or 16 bytes");
    if constexpr (BYTES == 16)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void ld_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void ld_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// bulk (TMA, SASS UBLKCP) shared -> global store of a contiguous block; works on peer-mapped addresses
__device__ __forceinline__ void st_bulk(void *gmem_dst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void st_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void st_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// generic-proxy writes to shared memory -> visible to the async proxy that executes the bulk copy
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace acp

__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// --- kernel P: persistent CTAs, per-thread asynchronous prefetch, CTA-deferred resets ---------------
// Kernel A is latency-bound: every warp issues its six loads, waits a cold HBM round trip, runs a ~330
// instruction float64 chain, stores and leaves; while it computes it has no load in flight, so the SM never
// holds the ~70 KB of outstanding reads that 6.5 TB/s x ~1.5 us ask for.  Here a resident grid (SMs x occupancy)
// walks the tiles; each THREAD copies the inputs of its env in the next tile (S state words, TimeLimit counter,
// action) into its own shared-memory slots with cp.async (LDGSTS: no registers, no barrier -- a thread only ever
// reads back what it wrote itself) while it advances the current tile, so loads stay in flight through the whole
// kernel.  Warps never meet at a barrier inside the loop: finishing envs go onto one CTA-wide list that is
// drained ONCE, with full lanes, after the loop (a warp where many lanes finish at once -- synchronised
// TimeLimit truncation -- resets inline instead, which is then equally dense).
constexpr int kResetCap = 1024;   // entries of the CTA's deferred-reset list; overflow resets inline

template <int KIND, typename ActT>
struct PrefetchLayout {
    using E = Env<KIND>;
    static constexpr int kActPerEnv = E::A == 0 ? 1 : E::A;
    static constexpr int kActBytes = kActPerEnv * (int)sizeof(ActT);
    static constexpr bool kActAsync = kActBytes == 4 || kActBytes == 8 || kActBytes == 16;
    static constexpr int kStateOff = 0;                                   // [S][256] float64
    static constexpr int kActOff = E::S * kThreads * 8;                   // [256] action (if async)
    static constexpr int kElapsedOff = kActOff + (kActAsync ? kThreads * kActBytes : 0);   // [256] int32
    static constexpr int kBytes = kElapsedOff + kThreads * 4;
};

// LEAN (the single-GPU step without the fused RecordEpisodeStatistics, fewer than 2^31 envs): 32-bit env indices
// (one IMAD.WIDE per address instead of a 64-bit add chain), no per-peer store loops, no episode accounting --
// same arithmetic, same stores, fewer issue slots.
template <int KIND, typename ActT, bool LEAN>
__global__ void __launch_bounds__(kThreads, Tuning<KIND>::kMinCtas) step_kernel_persistent(const StepArgs a, const int num_tiles) {
    using E = Env<KIND>;
    using L = PrefetchLayout<KIND, ActT>;
    using Idx = typename std::conditional<LEAN, uint32_t, int64_t>::type;
    // one stage of per-thread input slots holds the next tile in flight: a thread moves its slot into registers
    // before it refills it
    __shared__ __align__(16) unsigned char in_mem[L::kBytes];
    __shared__ int reset_list[kResetCap];
    __shared__ int reset_count;
    const int tid = threadIdx.x;
    if (tid == 0) reset_count = 0;
    __syncthreads();

    const ActT *actions = reinterpret_cast<const ActT *>(a.actions);
    const DirectSinkT<!LEAN> sink{a};
    const Idx first = (Idx)a.first, count = (Idx)a.count;

    auto prefetch = [&](int tile) {
        unsigned char *base = in_mem;
        double *s_state = reinterpret_cast<double *>(base + L::kStateOff);
        int32_t *s_elapsed = reinterpret_cast<int32_t *>(base + L::kElapsedOff);
        const Idx j = (Idx)tile * kThreads + tid;
        if (tile < num_tiles && j < count) {
            const Idx i = first + j;
#pragma unroll
            for (int k = 0; k < E::S; k++) acp::ld_async<8>(s_state + k * kThreads + tid, a.state + k * a.n + i);
            acp::ld_async<4>(s_elapsed + tid, a.elapsed + i);
            if constexpr (L::kActAsync)
                acp::ld_async<L::kActBytes>(base + L::kActOff + tid * L::kActBytes, actions + (size_t)i * L::kActPerEnv);
        }
        acp::ld_commit();   // always one group per call: the wait below counts groups
    };

    int tile = blockIdx.x;
    prefetch(tile);
    for (; tile < num_tiles; tile += gridDim.x) {
        const Idx j = (Idx)tile * kThreads + tid;
        const bool in_range = j < count;
        const Idx i = first + j;
        ActT av{};
        if constexpr (!L::kActAsync) { if (in_range) av = __ldg(actions + (size_t)i * L::kActPerEnv); }
        acp::ld_wait_all();
        unsigned char *base = in_mem;
        const double *s_state = reinterpret_cast<const double *>(base + L::kStateOff);
        double s[E::S];
#pragma unroll
        for (int k = 0; k < E::S; k++) s[k] = s_state[k * kThreads + tid];
        const int32_t elapsed = reinterpret_cast<const int32_t *>(base + L::kElapsedOff)[tid];
        if constexpr (L::kActAsync) av = *reinterpret_cast<const ActT *>(base + L::kActOff + tid * L::kActBytes);
        // this thread's slots are in registers now: refill them with its env in the next tile
        prefetch(tile + (int)gridDim.x);
        long long action_int = 0;
        float a0 = 0.0f;
        if constexpr (E::A == 0) action_int = (long long)av;
        else a0 = (float)av;
        bool need = false;
        if (in_range) need = advance_env<KIND, !LEAN>(a, sink, i, s, elapsed, action_int, a0);
        const unsigned m = __ballot_sync(0xffffffffu, need);
        if (m != 0u) {
            bool inline_reset = __popc(m) >= 12;          // dense enough: reset right here
            if (need && !inline_reset) {
                const int slot = atomicAdd(&reset_count, 1);
                if (slot < kResetCap) {
                    reset_list[slot] = (int)j;
                    // the drain after the loop starts with this env's 32-byte PCG64 record: have it in L2 by then
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(a.rng + 4 * (size_t)i));
                } else inline_reset = true;               // list full (whole batch truncating at once)
            }
            if (need && inline_reset) reset_env<KIND>(a, sink, i);
        }
    }
    __syncthreads();
    const int cnt = min(reset_count, kResetCap);
    for (int q = tid; q < cnt; q += kThreads) reset_env<KIND>(a, sink, (Idx)(first + (Idx)reset_list[q]));
}

// --- kernel G: one tile per CTA, results staged in shared memory and pushed with bulk stores ---------
// The multi-GPU step (b200gym_step_p2p): every result must land in this rank's rows of EVERY rank's gather
// buffers.  Per-thread peer stores put 16-, 8- and 1-byte writes on NVLink; here the 256-env tile of
// (obs, reward, terminated, truncated) is assembled in shared memory (reset observations included) and warp w
// pushes it to destination w -- peer w, or this rank's own buffers -- as four bulk copies (cp.async.bulk
// shared -> global, SASS UBLKCP), so NVLink carries full-size write packets and the LSU carries none of it.
// Needs 16-byte aligned destination rows; ragged tails and unaligned shards use kernel A's per-thread stores.
template <int KIND, typename ActT>
__global__ void __launch_bounds__(kThreads, Tuning<KIND>::kMinCtas) step_kernel_gather(const StepArgs a) {
    using E = Env<KIND>;
    __shared__ __align__(128) float s_obs[kThreads * E::D];
    __shared__ __align__(16) double s_reward[kThreads];
    __shared__ __align__(16) uint8_t s_term[kThreads];
    __shared__ __align__(16) uint8_t s_trunc[kThreads];
    __shared__ int reset_list[kThreads];
    __shared__ int reset_count;
    if (threadIdx.x == 0) reset_count = 0;
    __syncthreads();
    const int64_t j0 = (int64_t)blockIdx.x * kThreads;      // full tiles only: no bound check
    const int64_t i0 = a.first + j0;
    const StagedSink sink{s_obs, s_reward, s_term, s_trunc, i0};
    {
        const int64_t i = i0 + threadIdx.x;
        double s[E::S];
#pragma unroll
        for (int k = 0; k < E::S; k++) s[k] = a.state[k * a.n + i];
        const int32_t elapsed = a.elapsed[i];
        long long action_int = 0;
        float a0 = 0.0f;
        const ActT av = __ldg(reinterpret_cast<const ActT *>(a.actions) + i);
        if constexpr (E::A == 0) action_int = (long long)av;
        else a0 = (float)av;
        if (advance_env<KIND>(a, sink, i, s, elapsed, action_int, a0)) reset_list[atomicAdd(&reset_count, 1)] = threadIdx.x;
    }
    __syncthreads();
    if ((int)threadIdx.x < reset_count) reset_env<KIND>(a, sink, i0 + reset_list[threadIdx.x]);
    acp::fence_async_smem();
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0 && warp <= a.npeer) {
        float *obs = warp < a.npeer ? a.peer_obs[warp] : a.obs;
        double *reward = warp < a.npeer ? a.peer_reward[warp] : a.reward;
        uint8_t *term = warp < a.npeer ? a.peer_term[warp] : a.terminated;
        uint8_t *trunc = warp < a.npeer ? a.peer_trunc[warp] : a.truncated;
        acp::st_bulk(obs + i0 * E::D, s_obs, kThreads * E::D * 4);
        acp::st_bulk(reward + i0, s_reward, kThreads * 8);
        acp::st_bulk(term + i0, s_term, kThreads);
        acp::st_bulk(trunc + i0, s_trunc, kThreads);
        acp::st_bulk_commit();
        acp::st_bulk_wait_read();   // the tile must stay in shared memory until the copy engine has read it
    }
}

template <int KIND>
__global__ void __launch_bounds__(kThreads) reset_kernel(double *state, int32_t *elapsed, uint8_t *flags,
                                                         uint64_t *rng, const uint8_t *mask, float *obs,
                                                         int64_t n, double lo, double hi) {
    using E = Env<KIND>;
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    if (mask && !mask[i]) return;
    double s[E::S];
    float o[E::D];
    Pcg64 g = pcg64_load(rng + 4 * i);
    E::reset(s, g, lo, hi, o);
    pcg64_store(rng + 4 * i, g);
#pragma unroll
    for (int k = 0; k < E::S; k++) state[k * n + i] = s[k];
    elapsed[i] = 0;
    flags[i] = 0;
    if (obs) store_row<E::D>(obs, i, o);
}

// SeedSequence(base + first + i) -> PCG64, one thread per env
__global__ void __launch_bounds__(kThreads) seed_range_kernel(uint64_t *rng, int64_t n, uint32_t b0, uint32_t b1,
                                                              uint32_t b2, uint32_t b3, uint64_t first) {
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const u128 base = ((u128)b3 << 96) | ((u128)b2 << 64) | ((u128)b1 << 32) | (u128)b0;
    const u128 seed = base + (u128)(first + (uint64_t)i);
    const uint32_t ent[4] = {(uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)(seed >> 64), (uint32_t)(seed >> 96)};
    Pcg64 g;
    pcg64_from_entropy(g, ent);
    pcg64_store_full(rng + 4 * i, g);
}

__global__ void __launch_bounds__(kThreads) seed_each_kernel(uint64_t *rng, int64_t n, const uint32_t *ent,
                                                             const uint8_t *mask) {
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    if (mask && !mask[i]) return;
    const uint32_t e[4] = {ent[4 * i], ent[4 * i + 1], ent[4 * i + 2], ent[4 * i + 3]};
    Pcg64 g;
    pcg64_from_entropy(g, e);
    pcg64_store_full(rng + 4 * i, g);
}

// [n][S] AoS wire format <-> [S][n] SoA
__global__ void __launch_bounds__(kThreads) state_get_kernel(const double *soa, double *aos, int64_t n, int S) {
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    for (int k = 0; k < S; k++) aos[i * S + k] = soa[k * n + i];
}
__global__ void __launch_bounds__(kThreads) state_set_kernel(double *soa, const double *aos, int64_t n, int S) {
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    for (int k = 0; k < S; k++) soa[k * n + i] = aos[i * S + k];
}

// ---- the Box2D tasks (lunar.cuh, walker.cuh): one thread per env, the whole b2World::Step in registers/local ----
// A step is three launches on the stream:
//   box2d_step_kernel        validates the action and runs env_pre without SolveTOI; an env whose step may contain a
//                            continuous-collision event is parked (record + toi_mid) for the TOI kernel, every other
//                            env finishes here
//   box2d_toi_kernel         b2l::solve_toi of the parked envs, in warps full of them, then finish
//   box2d_reset_list_kernel  the autoresets of the step, compacted
// Finish (box2d_finish) is env_post, TimeLimit, the outputs and the episode statistics; an env whose episode ended
// goes onto the reset list.  What differs between the tasks -- record, what crosses the park, env_pre / env_post, the
// per-env reset, register budgets -- is in the task types below (LunarTask, LunarStep, WalkerTask).
constexpr int kBox2dThreads = 128;
constexpr int kResetSlots = 64;   // launch ranges of one handle that may be in flight at once (host path: <= 64 chunks)

// The TOI kernel runs one warp per CTA and gives each warp as FEW parked envs as the resident grid allows: the lanes
// of a warp diverge completely in this code (different contact lists, GJK / root-finder trip counts, event counts),
// so a warp takes the SUM of its lanes' paths, and with a few thousand parked envs on 148 SMs there are more warp
// slots than envs.  Measured (LunarLander, 2^16 envs, ~3 300 parked per step, ncu): 32 envs per warp 1.19 ms for
// the launch, 2 per warp 1.06 ms, 1 per warp 0.87 ms -- the floor is ONE env's serial chain (up to 5 sub-steps and
// ~30 b2TimeOfImpact evaluations of dependent, local-memory-heavy code at ~13 cycles per instruction).
__device__ __forceinline__ int toi_lanes_per_warp(int cnt, int nwarps) {
    const int L = (cnt + nwarps - 1) / nwarps;
    return L < 1 ? 1 : (L > 32 ? 32 : L);
}
// One-warp CTAs per SM of the TOI kernel; the kernel strides over the list.  12 warps of up to 168 registers per thread
// fit in an SM's 65 536 registers at once (12 x 32 x 168 = 64 512), which covers every TOI instantiation.  Larger grids
// (fewer envs per warp) were measured: LunarLander 1.74 / 1.82 / 1.85 ms at 12 / 64 / 256 CTAs per SM, BipedalWalker
// (nearly every env parked) 7.4 / 12.2 / 17.1 ms
constexpr int kToiCtasPerSm = 12;

// side buffer of a parked env ([kToiMidWords][n] SoA): the sweep starts of the bodies + env_pre's intermediates
constexpr int kToiMidWords = 20;   // LunarLander uses 13, BipedalWalker 15

__device__ __forceinline__ void store_sweep_starts(const StepArgs &a, int64_t i, const b2l::Body *b, int nb) {
    uint32_t *m = a.toi_mid + i;
    for (int k = 0; k < nb; k++) {
        m[(int64_t)(3 * k + 0) * a.n] = __float_as_uint(b[k].c0.x);
        m[(int64_t)(3 * k + 1) * a.n] = __float_as_uint(b[k].c0.y);
        m[(int64_t)(3 * k + 2) * a.n] = __float_as_uint(b[k].a0);
    }
}
__device__ __forceinline__ void load_sweep_starts(const StepArgs &a, int64_t i, b2l::Body *b, int nb) {
    const uint32_t *m = a.toi_mid + i;
    for (int k = 0; k < nb; k++) {
        b[k].c0.x = __uint_as_float(m[(int64_t)(3 * k + 0) * a.n]);
        b[k].c0.y = __uint_as_float(m[(int64_t)(3 * k + 1) * a.n]);
        b[k].a0 = __uint_as_float(m[(int64_t)(3 * k + 2) * a.n]);
    }
}

// LunarLander.  The phases after the step kernel do not read the action, so all four step instantiations (LunarStep)
// share this type's TOI and reset-list kernels.
struct LunarTask {
    using World = lunar::World;
    using Scene = lunar::Scene;
    struct Carry { Pcg64 g; lunar::Mid mid; };   // the env's PCG64 stream, env_pre's intermediates
    static constexpr int kObs = 8;
    static constexpr int kResetMinBlocks = 0;    // __launch_bounds__ of the reset-list kernel: no minimum
    static __device__ __forceinline__ void load(const StepArgs &a, int64_t i, World &W, Carry &c) {
        lunar::load_world(W, a.lunar_rec, a.n, i, a.lunar_opts.wind != 0);
        c.g = pcg64_load(a.rng + 4 * i);
    }
    static __device__ __forceinline__ void store(const StepArgs &a, int64_t i, const World &W, const Carry &c) {
        lunar::store_world(W, a.lunar_rec, a.n, i, a.lunar_opts.wind != 0);
        pcg64_store(a.rng + 4 * i, c.g);
    }
    static __device__ __forceinline__ void store_mid(const StepArgs &a, int64_t i, const World &W, const Carry &c) {
        store_sweep_starts(a, i, W.b, lunar::NB);
        uint32_t *m = a.toi_mid + i;
        const unsigned long long mc = (unsigned long long)__double_as_longlong(c.mid.main_cost);
        const unsigned long long sc = (unsigned long long)__double_as_longlong(c.mid.side_cost);
        m[(int64_t)9 * a.n] = (uint32_t)mc; m[(int64_t)10 * a.n] = (uint32_t)(mc >> 32);
        m[(int64_t)11 * a.n] = (uint32_t)sc; m[(int64_t)12 * a.n] = (uint32_t)(sc >> 32);
    }
    static __device__ __forceinline__ void load_mid(const StepArgs &a, int64_t i, World &W, Carry &c) {
        load_sweep_starts(a, i, W.b, lunar::NB);
        const uint32_t *m = a.toi_mid + i;
        c.mid.main_cost = __longlong_as_double((long long)(((unsigned long long)m[(int64_t)10 * a.n] << 32) | m[(int64_t)9 * a.n]));
        c.mid.side_cost = __longlong_as_double((long long)(((unsigned long long)m[(int64_t)12 * a.n] << 32) | m[(int64_t)11 * a.n]));
        c.mid.awake = true;   // only awake islands are parked
    }
    static __device__ __forceinline__ void post(World &W, const Carry &c, float (&obs)[kObs], double &reward, bool &terminated) {
        lunar::env_post(W, c.mid, obs, reward, terminated);
    }
    static __device__ __forceinline__ void reset(uint32_t *rec, const int64_t &n, int64_t i, uint64_t *rng, const lunar::Opts &O,
                                                 float (&obs)[kObs]) {
        lunar::reset_from_record(rec, n, i, rng, O, obs);
    }
};

// the LunarLander step kernel's part: the action encoding (Discrete(4) as ActT, or Box(2) float32 with CONT)
template <typename ActT, bool CONT>
struct LunarStep : LunarTask {
    using Task = LunarTask;
    // __launch_bounds__(256, 2) although it launches 128-thread CTAs: the register budget of DESIGN §4.4
    static constexpr int kStepMaxThreads = 256, kStepMinBlocks = 2;
    struct Action { long long act; float ca0, ca1; };
    static __device__ __forceinline__ bool read_action(const StepArgs &a, int64_t i, Action &v) {
        v.act = 0; v.ca0 = 0.0f; v.ca1 = 0.0f;
        if constexpr (CONT) {
            const float2 c = __ldg(reinterpret_cast<const float2 *>(a.actions) + i);   // Box(2) float32, lunar_lander.py:285-287
            v.ca0 = c.x; v.ca1 = c.y;
            return true;
        } else {
            v.act = (long long)__ldg(reinterpret_cast<const ActT *>(a.actions) + i);
            return !(v.act < 0 || v.act > 3);   // lunar_lander.py:482-484
        }
    }
    // env_pre without SolveTOI; true: the env needs the TOI phase
    static __device__ __forceinline__ bool pre(const StepArgs &a, World &W, Carry &c, const Action &v) {
        lunar::env_pre(W, c.g, a.lunar_opts, (int)v.act, v.ca0, v.ca1, lunar::V(0.0f, 0.0f), c.mid, 0u, /*run_toi=*/false);
        return c.mid.awake && b2l::toi_needed<Scene>(W);
    }
};

// BipedalWalker (HC: hardcore).  Step kernel and later phases alike.
template <bool HC>
struct WalkerTask {
    using Task = WalkerTask;
    using World = walker::World;
    using Scene = walker::SceneT<HC>;
    // numpy's 32-bit cache (the record holds it; the PCG64 stream is only drawn by reset()), the action, which
    // env_post charges for
    struct Carry { walker::Rng rng; float action[4]; };
    struct Action { float v[4]; };
    static constexpr int kObs = 24;
    static constexpr int kStepMaxThreads = kBox2dThreads, kStepMinBlocks = 4, kResetMinBlocks = 4;
    static __device__ __forceinline__ void load(const StepArgs &a, int64_t i, World &W, Carry &c) {
        walker::load_world(W, a.lunar_rec, a.n, i, c.rng, HC);
    }
    static __device__ __forceinline__ void store(const StepArgs &a, int64_t i, const World &W, const Carry &c) {
        walker::store_world(W, a.lunar_rec, a.n, i, c.rng, HC);
    }
    static __device__ __forceinline__ void store_mid(const StepArgs &a, int64_t i, const World &W, const Carry &) {
        store_sweep_starts(a, i, W.b, walker::NB);
    }
    // the sweep starts, the action (read again), and the window of obstacle boxes env_pre computed around the hull's
    // position before the step
    static __device__ __forceinline__ void load_mid(const StepArgs &a, int64_t i, World &W, Carry &c) {
        const float4 av = __ldg(reinterpret_cast<const float4 *>(a.actions) + i);
        c.action[0] = av.x; c.action[1] = av.y; c.action[2] = av.z; c.action[3] = av.w;
        load_sweep_starts(a, i, W.b, walker::NB);
        if constexpr (HC) walker::poly_window(W, W.b[0].c0.x - 4.0f, W.b[0].c0.x + 4.0f, W.p_lo, W.p_hi);
    }
    static __device__ __forceinline__ bool read_action(const StepArgs &a, int64_t i, Action &v) {
        const float4 av = __ldg(reinterpret_cast<const float4 *>(a.actions) + i);
        v.v[0] = av.x; v.v[1] = av.y; v.v[2] = av.z; v.v[3] = av.w;
        return true;
    }
    static __device__ __forceinline__ bool pre(const StepArgs &, World &W, Carry &c, const Action &v) {
        for (int k = 0; k < 4; k++) c.action[k] = v.v[k];
        bool awake;
        walker::env_pre<HC>(W, c.action, walker::V(0.0f, 0.0f), awake, 0u, /*run_toi=*/false);
        return awake && b2l::toi_needed<Scene>(W);
    }
    static __device__ __forceinline__ void post(World &W, const Carry &c, float (&obs)[kObs], double &reward, bool &terminated) {
        walker::env_post<HC>(W, c.action, false, obs, reward, terminated);
    }
    static __device__ __forceinline__ void reset(uint32_t *rec, const int64_t &n, int64_t i, uint64_t *rng, const lunar::Opts &,
                                                 float (&obs)[kObs]) {
        walker::reset_from_record<HC>(rec, n, i, rng, obs);
    }
};

// everything after world.Step of the task's step(), then TimeLimit, outputs and the same-step autoreset's bookkeeping:
// the new episode is drawn by box2d_reset_list_kernel, in warps full of resetting envs
template <typename Task>
__device__ __noinline__ void box2d_finish(const StepArgs &a, int64_t i, int64_t j, typename Task::World &W,
                                          const typename Task::Carry &c, int32_t elapsed) {
    float obs[Task::kObs];
    double reward;
    bool terminated;
    Task::post(W, c, obs, reward, terminated);
    elapsed += 1;                                                        // time_limit.py:51
    const bool truncated = (a.max_steps > 0) && (elapsed >= a.max_steps);
    store_scalars_all(a, i, reward, terminated ? 1 : 0, truncated ? 1 : 0);
    episode_account(a, i, reward, terminated || truncated);
    const bool reset = (terminated || truncated) && a.autoreset;        // sync_vector_env.py:152-156
    if (reset) {
        if (a.final_obs) store_row<Task::kObs>(a.final_obs, i, obs);
        a.reset_list[a.first + atomicAdd(a.reset_count, 1)] = (int32_t)j;
    }
    Task::store(a, i, W, c);
    a.elapsed[i] = elapsed;
    if (!reset) store_obs_all<Task::kObs>(a, i, obs);
}

template <typename Step>
__global__ void __launch_bounds__(Step::kStepMaxThreads, Step::kStepMinBlocks) box2d_step_kernel(const StepArgs a) {
    using Task = typename Step::Task;
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.count) return;
    const int64_t i = a.first + j;
    typename Step::Action act;
    if (!Step::read_action(a, i, act)) {
        atomicAdd(a.invalid, 1ULL);
        *reinterpret_cast<volatile unsigned long long *>(a.invalid_seen) = 1ULL;
        store_scalars_all(a, i, __longlong_as_double(0x7ff8000000000000LL), 0, 0);
        return;
    }
    typename Task::World W;
    typename Task::Carry c;
    Task::load(a, i, W, c);
    const int32_t elapsed = a.elapsed[i];
    if (Step::pre(a, W, c, act)) {   // park the env for box2d_toi_kernel
        Task::store(a, i, W, c);
        Task::store_mid(a, i, W, c);
        a.toi_list[a.first + atomicAdd(a.toi_count, 1)] = (int32_t)j;
        return;
    }
    box2d_finish<Task>(a, i, j, W, c, elapsed);
}

// The continuous-collision phase of the envs that box2d_step_kernel parked, one warp of parked envs per CTA: the
// TOI code (GJK, root finder, the sub-step solver) is large and runs for a few percent of the envs, so it gets
// its own launch -- dense warps and a warm instruction cache instead of one or two lanes per warp walking it at the
// end of every warp's critical path -- and the warp-synchronous event rounds of b2l::solve_toi.
template <typename Task>
__global__ void __launch_bounds__(32) box2d_toi_kernel(const StepArgs a) {
    const int cnt = *a.toi_count;
    const int L = toi_lanes_per_warp(cnt, (int)gridDim.x);
    for (int base = blockIdx.x * L; base < cnt; base += gridDim.x * L) {
        const int idx = base + (int)threadIdx.x;
        const bool on = (int)threadIdx.x < L && idx < cnt;
        const unsigned live = __ballot_sync(0xffffffffu, on);
        if (on) {
            const int64_t j = a.toi_list[a.first + idx];
            const int64_t i = a.first + j;
            typename Task::World W;
            typename Task::Carry c;
            Task::load(a, i, W, c);
            Task::load_mid(a, i, W, c);
            const int32_t elapsed = a.elapsed[i];
            b2l::solve_toi<typename Task::Scene>(W, (float)(1.0 / 50), true, live);
            box2d_finish<Task>(a, i, j, W, c, elapsed);
        }
    }
}

// The autoresets of one step, compacted: a lone finishing env would otherwise keep its whole warp waiting through
// a full reset() (terrain draw + the embedded world step) with one active lane.
template <typename Task>
__global__ void __launch_bounds__(kBox2dThreads, Task::kResetMinBlocks) box2d_reset_list_kernel(const StepArgs a) {
    const int cnt = *a.reset_count;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < cnt; idx += gridDim.x * blockDim.x) {
        const int64_t i = a.first + a.reset_list[a.first + idx];
        float obs[Task::kObs];
        Task::reset(a.lunar_rec, a.n, i, a.rng, a.lunar_opts, obs);
        a.elapsed[i] = 0;
        store_obs_all<Task::kObs>(a, i, obs);
    }
}

// reset() of the (masked) envs
template <typename Task>
__global__ void __launch_bounds__(kBox2dThreads) box2d_reset_kernel(uint32_t *rec, int32_t *elapsed, uint64_t *rng,
                                                                    const uint8_t *mask, float *obs, int64_t n,
                                                                    const lunar::Opts O) {
    const int64_t i = (int64_t)blockIdx.x * kBox2dThreads + threadIdx.x;
    if (i >= n) return;
    if (mask && !mask[i]) return;
    float o[Task::kObs];
    Task::reset(rec, n, i, rng, O, o);
    elapsed[i] = 0;
    if (obs) store_row<Task::kObs>(obs, i, o);
}

// ---- LunarLander-v2 only ------------------------------------------------------------------------------------
// wind_idx / torque_idx of every env (lunar_lander.py:234-235): two int32 SoA rows of the record
__global__ void lunar_wind_idx_kernel(uint32_t *rec, int32_t *wind, int32_t *torque, int64_t n, int set) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (set) { rec[(int64_t)lunar::W_WIND * n + i] = (uint32_t)wind[i]; rec[(int64_t)(lunar::W_WIND + 1) * n + i] = (uint32_t)torque[i]; }
    else { wind[i] = (int32_t)rec[(int64_t)lunar::W_WIND * n + i]; torque[i] = (int32_t)rec[(int64_t)(lunar::W_WIND + 1) * n + i]; }
}

// bodies of every env as [n][18] floats {c.x, c.y, a, v.x, v.y, w} x 3 + [n][6] int32 flags (parity harness)
__global__ void lunar_bodies_kernel(const uint32_t *rec, const int32_t *elapsed, float *out, int32_t *flags, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int b = 0; b < 3; b++)
        for (int k = 0; k < 6; k++) out[i * 18 + 6 * b + k] = __uint_as_float(rec[(int64_t)(lunar::W_BODY + 7 * b + k) * n + i]);
    const uint32_t f = rec[(int64_t)lunar::W_FLAGS * n + i];
    int touching = 0;
    for (int sl = 0; sl < lunar::kSlots; sl++) touching += (rec[(int64_t)(lunar::W_SLOT + 7 * sl) * n + i] >> 16) != 0;
    flags[i * 6 + 0] = f & 1u; flags[i * 6 + 1] = (f >> 1) & 1u; flags[i * 6 + 2] = (f >> 2) & 1u;
    flags[i * 6 + 3] = 1; flags[i * 6 + 4] = elapsed[i]; flags[i * 6 + 5] = touching;
}

// envs whose manifold table ever overflowed (b2l::kFlagOverflow in the record's flag word)
__global__ void box2d_overflow_kernel(const uint32_t *flags_row, int64_t n, unsigned long long *count) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && (flags_row[i] & b2l::kFlagOverflow)) atomicAdd(count, 1ULL);
}

static int lunar_upload_consts(b200gym *h) {
    lunar::Consts c;
    b2l_host::lunar_consts(c);
    CK(h, cudaMemcpyToSymbol(lunar::kC, &c, sizeof c));
    return 0;
}

// ---- BipedalWalker-v3 only ------------------------------------------------------------------------------------
// a fresh Generator has an empty 32-bit cache: clear {has_uint32, uinteger} of the (re)seeded envs
__global__ void walker_clear_rng32_kernel(uint32_t *rec, const uint8_t *mask, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || (mask && !mask[i])) return;
    rec[(int64_t)walker::W_RNG32 * n + i] = 0u;
    rec[(int64_t)(walker::W_RNG32 + 1) * n + i] = 0u;
}

// terrain heights [n][200] and (hardcore) obstacle boxes [n][40][4] = {x0, ylo, x1, yhi} + their number [n]
__global__ void walker_terrain_kernel(const uint32_t *rec, float *terrain, float *polys, int32_t *npoly, int64_t n, int hardcore) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int k = 0; k < walker::kTerrain; k++) terrain[i * walker::kTerrain + k] = __uint_as_float(rec[(int64_t)(walker::W_TERRAIN + k) * n + i]);
    if (!polys || !npoly) return;
    const int np = hardcore ? (int)rec[(int64_t)walker::W_NPOLY * n + i] : 0;
    npoly[i] = np;
    for (int k = 0; k < 4 * walker::NP; k++)
        polys[i * 4 * walker::NP + k] = k < 4 * np ? __uint_as_float(rec[(int64_t)(walker::W_POLY + k) * n + i]) : 0.0f;
}

__global__ void walker_bodies_kernel(const uint32_t *rec, float *out, int32_t *flags, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int b = 0; b < walker::NB; b++)
        for (int k = 0; k < 6; k++) out[i * 30 + 6 * b + k] = __uint_as_float(rec[(int64_t)(walker::W_BODY + 7 * b + k) * n + i]);
    const uint32_t f = rec[(int64_t)walker::W_FLAGS * n + i];
    int touching = 0;
    for (int sl = 0; sl < walker::kSlots; sl++) touching += (rec[(int64_t)(walker::W_SLOT + 7 * sl) * n + i] >> 16) != 0;
    flags[i * 4 + 0] = f & 1u; flags[i * 4 + 1] = (f >> 1) & 1u; flags[i * 4 + 2] = (f >> 2) & 1u; flags[i * 4 + 3] = touching;
}

static int walker_upload_consts(b200gym *h) {
    walker::Consts c;
    b2l_host::walker_consts(c);
    CK(h, cudaMemcpyToSymbol(walker::kC, &c, sizeof c));
    return 0;
}

// ---- SURVEY.md 8(f): vector-aware wrappers fused on the device ---------------------------------------
// RecordEpisodeStatistics (gym/wrappers/record_episode_statistics.py:103-151): the reference walks the
// batch in a Python loop; here one launch updates the float32 return / int32 length accumulators,
// emits infos["episode"]["r"/"l"] + the `_episode` mask, and appends finished episodes to a small ring
// (the return_queue / length_queue deques).
__global__ void __launch_bounds__(kThreads) episode_stats_kernel(const double *reward, const uint8_t *term,
                                                                const uint8_t *trunc, float *ret_acc, int32_t *len_acc,
                                                                float *ep_r, int32_t *ep_l, uint8_t *ep_mask,
                                                                unsigned long long *ring,
                                                                unsigned long long *counter, int ring_size, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    // `self.episode_returns += rewards` on a float32 array with float64 rewards: add in float64, round to float32
    const float ret = (float)((double)ret_acc[i] + reward[i]);
    const int32_t len = len_acc[i] + 1;
    const bool done = term[i] | trunc[i];
    ep_mask[i] = done ? 1 : 0;
    if (done) {
        ep_r[i] = ret;
        ep_l[i] = len;
        if (ring_size > 0) {
            // one 64-bit store per episode {length : return bits}: when more than ring_size episodes finish in one
            // step several of them land on the same slot, and a slot must never mix two episodes
            const unsigned long long slot = atomicAdd(counter, 1ULL);
            ring[slot % (unsigned long long)ring_size] =
                ((unsigned long long)(uint32_t)len << 32) | (unsigned long long)__float_as_uint(ret);
        } else atomicAdd(counter, 1ULL);
        ret_acc[i] = 0.0f;
        len_acc[i] = 0;
    } else {
        ret_acc[i] = ret;
        len_acc[i] = len;
    }
}

// NormalizeObservation / NormalizeReward (gym/wrappers/normalize.py:8-144): RunningMeanStd over the batch axis,
// two launches per step and ONE pass over the batch for the moments.
//   launch 1 (moments): the batch is read as a flat [n*D] stream; the CTA size is a multiple of D, so every
//     thread stays on one column and the loads are perfectly coalesced whatever D is.  Per column: sum and sum of
//     squares of the deviations from a pivot (the current running mean: numerically tame), float64, reduced through
//     shared-memory atomics to one global atomic per CTA and column.
//   (between the launches a sharded env all-reduces the 2*D sums across GPUs: torch.distributed, 8 * 2 * D bytes)
//   launch 2 (apply): every CTA folds the batch moments into the running ones (Chan et al., normalize.py:32-46) on
//     its own -- D <= 24 columns, a few dozen flops -- normalises its share of the batch with the NEW statistics
//     (normalize.py:83-95) and CTA 0 publishes them.  Statistics and scratch are double-buffered by step parity, so
//     no CTA can read a half-updated value.
// stats layout (float64, caller-owned): [2][2*D + 1] = {mean[D], var[D], count}; scratch: [2][2*D] = {sum[D], sumsq[D]}.
constexpr int kMaxNormDim = 24;

__device__ __forceinline__ int norm_block(int D) { return (D == 3 || D == 6 || D == 24) ? 192 : 256; }

template <typename T, bool RETURNS>
__global__ void rms_moments_kernel(const T *x, double *returns, const double *reward, double gamma, int64_t total, int D,
                                   const double *stats, double *scratch) {
    __shared__ double sh[2][kMaxNormDim];
    const int tid = threadIdx.x;
    if (tid < D) { sh[0][tid] = 0.0; sh[1][tid] = 0.0; }
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;      // a multiple of D: the column of a thread is fixed
    const int64_t start = (int64_t)blockIdx.x * blockDim.x + tid;
    const int col = (int)(start % D);
    const double pivot = stats[col];
    double s = 0.0, q = 0.0;
    for (int64_t k = start; k < total; k += stride) {
        double v;
        if constexpr (RETURNS) {   // NormalizeReward.step (normalize.py:130): returns = returns * gamma + reward
            v = returns[k] * gamma + reward[k];
            returns[k] = v;
        } else {
            v = (double)x[k];
        }
        v -= pivot;
        s += v;
        q += v * v;
    }
    atomicAdd(&sh[0][col], s);
    atomicAdd(&sh[1][col], q);
    __syncthreads();
    if (tid < D) {
        atomicAdd(&scratch[tid], sh[0][tid]);
        atomicAdd(&scratch[D + tid], sh[1][tid]);
    }
}

// update_mean_var_count_from_moments (normalize.py:32-46) for column d, from the pivoted batch sums
__device__ __forceinline__ void chan_update(const double *stats, const double *scratch, int D, int d, double bn, double &mean,
                                            double &var, double &count) {
    const double dm = scratch[d] / bn;                 // batch_mean - pivot (pivot = old mean) = delta
    const double batch_var = scratch[D + d] / bn - dm * dm;
    const double cnt = stats[2 * D];
    const double tot = cnt + bn;
    mean = stats[d] + dm * bn / tot;
    const double m2 = stats[D + d] * cnt + batch_var * bn + dm * dm * cnt * bn / tot;
    var = m2 / tot;
    count = tot;
}

template <bool REWARD>
__global__ void rms_apply_kernel(const float *x, float *out, const double *reward, double *out_r, double *returns,
                                 const uint8_t *term, const uint8_t *trunc, int64_t total, int D, const double *stats,
                                 double *stats_next, const double *scratch, double *scratch_next, double batch_count,
                                 double eps, int update) {
    __shared__ double sh_mean[kMaxNormDim], sh_inv[kMaxNormDim];
    const int tid = threadIdx.x;
    if (tid < D) {
        double mean = stats[tid], var = stats[D + tid], count = stats[2 * D];
        if (update) chan_update(stats, scratch, D, tid, batch_count, mean, var, count);
        sh_mean[tid] = mean;
        sh_inv[tid] = sqrt(var + eps);
        if (blockIdx.x == 0 && update) {
            stats_next[tid] = mean;
            stats_next[D + tid] = var;
            if (tid == 0) stats_next[2 * D] = count;
            scratch_next[tid] = 0.0;                   // next step accumulates into the other scratch buffer
            scratch_next[D + tid] = 0.0;
        }
    }
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t start = (int64_t)blockIdx.x * blockDim.x + tid;
    const int col = (int)(start % D);
    const double mean = sh_mean[col], sd = sh_inv[col];
    for (int64_t k = start; k < total; k += stride) {
        if constexpr (REWARD) {
            out_r[k] = reward[k] / sd;                                 // normalize.py:143 (no mean subtraction)
            if (term[k] | trunc[k]) returns[k] = 0.0;                  // :135-136
        } else {
            out[k] = (float)(((double)x[k] - mean) / sd);              // normalize.py:95
        }
    }
}

// ---- cross-GPU step barrier for the fused all-gather ---------------------------------------
// flags[r] (uint64, in every rank's gather allocation) = number of steps whose results rank r has fully written
// into THIS rank's buffers.  One launch per step, after the step kernel on the same stream: lane p publishes
// "my rows of step k are in your buffers" to peer p (the kernel boundary has drained the step kernel's stores,
// bulk ones included; the system-scope fence orders them before the flag) and then waits for peer p's flag.
// A peer that died does not hang the stream for ever: after `timeout_ns` the lane records the peer in
// `*timed_out` (sticky, read by b200gym_p2p_status) and gives up.
__global__ void p2p_sync_kernel(unsigned long long *const *peer_flags, const unsigned long long *my_flags, int world,
                                int rank, unsigned long long step, unsigned long long timeout_ns, int *timed_out) {
    const int p = threadIdx.x;
    if (p < world && p != rank) {
        __threadfence_system();
        volatile unsigned long long *f = peer_flags[p] + rank;
        *f = step;
        const volatile unsigned long long *w = my_flags + p;
        const unsigned long long t0 = global_ns();
        while (*w < step) {
            if (global_ns() - t0 > timeout_ns) {
                atomicExch(timed_out, p + 1);
                break;
            }
        }
        __threadfence_system();
    }
}

// device self-test: div_by_const(x, c, RN(1/c)) must equal x / c bit for bit
__global__ void __launch_bounds__(kThreads) selftest_div_kernel(int64_t samples, uint64_t seed,
                                                                unsigned long long *mismatches) {
    const double cs[4] = {1.1, 0.1 + 1.0, 3.0, 9.8};
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= samples) return;
    // splitmix64 bits -> doubles spread over many binades, both signs
    uint64_t z = seed + 0x9E3779B97F4A7C15ULL * (uint64_t)(i + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    z ^= z >> 31;
    const double mant = 1.0 + (double)(z >> 12) * (1.0 / 4503599627370496.0);
    const int e = (int)((z >> 3) & 0x3F) - 32;
    double x = ldexp(mant, e);
    if (z & 1) x = -x;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const double c = cs[k];
        const double rc = 1.0 / c;
        const double fast = div_by_const(x, c, rc);
        const double ref = x / c;
        if (__double_as_longlong(fast) != __double_as_longlong(ref)) atomicAdd(mismatches, 1ULL);
    }
}

// device self-test: csrc/glibc_trig.cuh evaluated on caller-supplied arguments (the host compares with its libm)
__global__ void __launch_bounds__(kThreads) selftest_trig_kernel(const double *x, int64_t n, double *sn, double *cs, double *sq) {
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    sn[i] = gt::sin(x[i]);
    cs[i] = gt::cos(x[i]);
    if (sq) sq[i] = gt::sq(x[i]);
}

static inline unsigned blocks_for(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

// ---------------------------------------------------------------------------
// dispatch
// ---------------------------------------------------------------------------
template <int KIND, typename ActT>
static int launch_step_typed(b200gym *h, const StepArgs &a, cudaStream_t st) {
    int64_t done = 0;
    const int64_t tiles = a.count / kThreads;
    if ((a.npeer > 0 || a.bulk_sink) && tiles > 0) {
        // kernel G (bulk pushes): every destination row block must be 16-byte aligned
        auto ok = [&](const float *o, const double *r, const uint8_t *te, const uint8_t *tr) {
            return (uintptr_t)(o + a.first * Env<KIND>::D) % 16 == 0 && (uintptr_t)(r + a.first) % 16 == 0 &&
                   (uintptr_t)(te + a.first) % 16 == 0 && (uintptr_t)(tr + a.first) % 16 == 0;
        };
        bool aligned = ok(a.obs, a.reward, a.terminated, a.truncated);
        for (int p = 0; p < a.npeer; p++) aligned = aligned && ok(a.peer_obs[p], a.peer_reward[p], a.peer_term[p], a.peer_trunc[p]);
        if (aligned) {
            step_kernel_gather<KIND, ActT><<<(unsigned)tiles, kThreads, 0, st>>>(a);
            CK(h, cudaGetLastError());
            done = tiles * kThreads;
        }
    }
    if (done == 0 && h->kernel_choice >= 1 && a.npeer == 0 && a.count >= (int64_t)h->sm_count * kThreads) {
        // kernel P: resident grid; needs naturally aligned input words for cp.async (always true for the
        // handle's own arrays; the caller's action pointer is checked)
        using L = PrefetchLayout<KIND, ActT>;
        const bool aligned = !L::kActAsync || ((uintptr_t)a.actions % L::kActBytes == 0);
        if (aligned) {
            // the lean instantiation: no fused episode statistics, every index fits 32 bits
            const bool lean = h->kernel_choice == 2 && !a.ep_acc && h->n < (int64_t)1 << 30;
            int &occ = h->occ[KIND][sizeof(ActT) == 8 ? 0 : sizeof(ActT) == 4 ? 1 : 2][lean ? 1 : 0];
            if (occ == 0) {
                if (lean) CK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, step_kernel_persistent<KIND, ActT, true>, kThreads, 0));
                else CK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, step_kernel_persistent<KIND, ActT, false>, kThreads, 0));
                if (occ < 1) occ = 1;
            }
            const int64_t all_tiles = (a.count + kThreads - 1) / kThreads;
            int64_t grid = (int64_t)h->sm_count * occ;
            if (grid > all_tiles) grid = all_tiles;
            if (lean) step_kernel_persistent<KIND, ActT, true><<<(unsigned)grid, kThreads, 0, st>>>(a, (int)all_tiles);
            else step_kernel_persistent<KIND, ActT, false><<<(unsigned)grid, kThreads, 0, st>>>(a, (int)all_tiles);
            CK(h, cudaGetLastError());
            done = a.count;
        }
    }
    if (done < a.count) {
        StepArgs t = a;
        t.first = a.first + done;
        t.count = a.count - done;
        step_kernel<KIND, ActT><<<blocks_for(t.count), kThreads, 0, st>>>(t);
        CK(h, cudaGetLastError());
    }
    return 0;
}

template <int KIND>
static int launch_step_kind(b200gym *h, const StepArgs &a, int action_dtype, cudaStream_t st) {
    using E = Env<KIND>;
    if constexpr (E::A == 0) {
        switch (action_dtype) {
        case B200GYM_ACT_I64: return launch_step_typed<KIND, long long>(h, a, st);
        case B200GYM_ACT_I32: return launch_step_typed<KIND, int>(h, a, st);
        case B200GYM_ACT_U8: return launch_step_typed<KIND, unsigned char>(h, a, st);
        default: return fail(h, "Discrete env needs an integer action dtype (got code %d)", action_dtype);
        }
    } else {
        if (action_dtype != B200GYM_ACT_F32)
            return fail(h, "Box env needs float32 actions (got dtype code %d)", action_dtype);
        return launch_step_typed<KIND, float>(h, a, st);
    }
}

// The Box2D step: box2d_step_kernel -> box2d_toi_kernel -> box2d_reset_list_kernel on the stream.  The caller may
// have picked the counters' slot (one per concurrently running launch range).
template <typename Step>
static int launch_box2d_step(b200gym *h, const StepArgs &a, cudaStream_t st) {
    using Task = typename Step::Task;
    if (a.autoreset) CK(h, cudaMemsetAsync(a.reset_count, 0, sizeof(int32_t), st));
    CK(h, cudaMemsetAsync(a.toi_count, 0, sizeof(int32_t), st));
    box2d_step_kernel<Step><<<(unsigned)((a.count + kBox2dThreads - 1) / kBox2dThreads), kBox2dThreads, 0, st>>>(a);
    CK(h, cudaGetLastError());
    box2d_toi_kernel<Task><<<(unsigned)std::min<int64_t>(a.count, (int64_t)kToiCtasPerSm * h->sm_count), 32, 0, st>>>(a);
    CK(h, cudaGetLastError());
    if (a.autoreset) {
        // at most this many CTAs (the kernel strides over the list)
        const int64_t grid = std::min<int64_t>((a.count + kBox2dThreads - 1) / kBox2dThreads, 2 * h->sm_count);
        box2d_reset_list_kernel<Task><<<(unsigned)grid, kBox2dThreads, 0, st>>>(a);
        CK(h, cudaGetLastError());
    }
    return 0;
}

static int launch_step(b200gym *h, const StepArgs &a, int action_dtype, cudaStream_t st) {
    switch (h->cfg.kind) {
    case B200GYM_CARTPOLE: return launch_step_kind<B200GYM_CARTPOLE>(h, a, action_dtype, st);
    case B200GYM_MOUNTAINCAR: return launch_step_kind<B200GYM_MOUNTAINCAR>(h, a, action_dtype, st);
    case B200GYM_MOUNTAINCAR_CONT: return launch_step_kind<B200GYM_MOUNTAINCAR_CONT>(h, a, action_dtype, st);
    case B200GYM_PENDULUM: return launch_step_kind<B200GYM_PENDULUM>(h, a, action_dtype, st);
    case B200GYM_ACROBOT: return launch_step_kind<B200GYM_ACROBOT>(h, a, action_dtype, st);
    case B200GYM_LUNARLANDER:
        switch (action_dtype) {
        case B200GYM_ACT_I64: return launch_box2d_step<LunarStep<long long, false>>(h, a, st);
        case B200GYM_ACT_I32: return launch_box2d_step<LunarStep<int, false>>(h, a, st);
        case B200GYM_ACT_U8: return launch_box2d_step<LunarStep<unsigned char, false>>(h, a, st);
        default: return fail(h, "Discrete env needs an integer action dtype (got code %d)", action_dtype);
        }
    case B200GYM_LUNARLANDER_CONT:
        if (action_dtype != B200GYM_ACT_F32) return fail(h, "Box env needs float32 actions (got dtype code %d)", action_dtype);
        if ((uintptr_t)a.actions % 8 != 0) return fail(h, "LunarLanderContinuous actions must be 8-byte aligned");
        return launch_box2d_step<LunarStep<float, true>>(h, a, st);
    case B200GYM_BIPEDALWALKER:
    case B200GYM_BIPEDALWALKER_HARDCORE:
        if (action_dtype != B200GYM_ACT_F32) return fail(h, "Box env needs float32 actions (got dtype code %d)", action_dtype);
        if ((uintptr_t)a.actions % 16 != 0) return fail(h, "BipedalWalker actions must be 16-byte aligned");
        if (h->cfg.kind == B200GYM_BIPEDALWALKER_HARDCORE) return launch_box2d_step<WalkerTask<true>>(h, a, st);
        return launch_box2d_step<WalkerTask<false>>(h, a, st);
    }
    return fail(h, "bad kind %d", h->cfg.kind);
}

template <int KIND>
static void launch_reset_kind(b200gym *h, const uint8_t *mask, const double *bounds, float *obs, cudaStream_t st) {
    double lo, hi;
    Env<KIND>::default_bounds(lo, hi);
    if (bounds) { lo = bounds[0]; hi = bounds[1]; }
    reset_kernel<KIND><<<blocks_for(h->n), kThreads, 0, st>>>(h->state, h->elapsed, h->flags, h->rng, mask, obs,
                                                              h->n, lo, hi);
}

template <typename Task>
static void launch_box2d_reset(b200gym *h, const uint8_t *mask, float *obs, cudaStream_t st) {
    box2d_reset_kernel<Task><<<(unsigned)((h->n + kBox2dThreads - 1) / kBox2dThreads), kBox2dThreads, 0, st>>>(
        h->lunar_rec, h->elapsed, h->rng, mask, obs, h->n, h->lunar_opts);
}

static int launch_reset(b200gym *h, const uint8_t *mask, const double *bounds, float *obs, cudaStream_t st) {
    switch (h->cfg.kind) {
    case B200GYM_CARTPOLE: launch_reset_kind<B200GYM_CARTPOLE>(h, mask, bounds, obs, st); break;
    case B200GYM_MOUNTAINCAR: launch_reset_kind<B200GYM_MOUNTAINCAR>(h, mask, bounds, obs, st); break;
    case B200GYM_MOUNTAINCAR_CONT: launch_reset_kind<B200GYM_MOUNTAINCAR_CONT>(h, mask, bounds, obs, st); break;
    case B200GYM_PENDULUM: launch_reset_kind<B200GYM_PENDULUM>(h, mask, bounds, obs, st); break;
    case B200GYM_ACROBOT: launch_reset_kind<B200GYM_ACROBOT>(h, mask, bounds, obs, st); break;
    case B200GYM_LUNARLANDER:
    case B200GYM_LUNARLANDER_CONT: launch_box2d_reset<LunarTask>(h, mask, obs, st); break;
    case B200GYM_BIPEDALWALKER: launch_box2d_reset<WalkerTask<false>>(h, mask, obs, st); break;
    case B200GYM_BIPEDALWALKER_HARDCORE: launch_box2d_reset<WalkerTask<true>>(h, mask, obs, st); break;
    default: return fail(h, "bad kind %d", h->cfg.kind);
    }
    CK(h, cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// the device a caller-owned buffer lives on (these utilities take no handle)
static int device_of(const void *ptr) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
        cudaGetLastError();
        return -1;
    }
    return at.device;
}

extern "C" int b200gym_create(const b200gym_config *cfg, int64_t num_envs, int device, b200gym_t **out) {
    if (!cfg || !out) return fail(nullptr, "b200gym_create: null argument");
    *out = nullptr;
    if (!kind_ok(cfg->kind)) return fail(nullptr, "b200gym_create: unknown env kind %d", cfg->kind);
    if ((cfg->kind == B200GYM_LUNARLANDER || cfg->kind == B200GYM_LUNARLANDER_CONT) &&
        !(-12.0 < cfg->param[0] && cfg->param[0] < 0.0))  // the assert of lunar_lander.py:210-212 (0.0 included: no
                                                          // silent default -- callers pass the reference's -10.0)
        return fail(nullptr, "b200gym_create: gravity (current value: %g) must be between -12 and 0", cfg->param[0]);
    if (num_envs <= 0) return fail(nullptr, "b200gym_create: num_envs must be positive (got %lld)", (long long)num_envs);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, "b200gym_create: no CUDA device available (%s); this engine has no CPU fallback",
                    cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(nullptr, "b200gym_create: bad device %d (have %d)", device, ndev);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess && prop.major != 10)
        return fail(nullptr, "b200gym_create: device %d is sm_%d%d; this library contains sm_100a code only",
                    device, prop.major, prop.minor);
    b200gym *h = new (std::nothrow) b200gym();
    if (!h) return fail(nullptr, "b200gym_create: out of host memory");
    h->cfg = *cfg;
    h->n = num_envs;
    h->device = device;
    h->S = k_state_dim[cfg->kind];
    h->D = k_obs_dim[cfg->kind];
    h->A = k_act_dim[cfg->kind];
    h->NACT = k_nact[cfg->kind];
    h->sm_count = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
    if (const char *kc = getenv("B200GYM_KERNEL"))
        if (kc[0] == 'a' || kc[0] == 'p' || kc[0] == 'l') h->kernel_choice = kc[0] == 'a' ? 0 : kc[0] == 'p' ? 1 : 2;
    DeviceGuard guard(device);
    const size_t n = (size_t)num_envs;
    cudaError_t es[5] = {
        cudaMalloc(&h->state, sizeof(double) * n * (h->S > 0 ? h->S : 1)), cudaMalloc(&h->elapsed, sizeof(int32_t) * n),
        cudaMalloc(&h->flags, n), cudaMalloc(&h->rng, 32 * n), cudaMalloc(&h->invalid, sizeof(unsigned long long))};
    for (cudaError_t ei : es)
        if (ei != cudaSuccess) {
            fail(nullptr, "b200gym_create: cudaMalloc failed: %s", cudaGetErrorString(ei));
            b200gym_destroy(h);
            return 1;
        }
    if (cudaHostAlloc((void **)&h->invalid_seen, sizeof(unsigned long long), cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer((void **)&h->invalid_seen_dev, h->invalid_seen, 0) != cudaSuccess) {
        fail(nullptr, "b200gym_create: cannot allocate the mapped invalid-action flag: %s", cudaGetErrorString(cudaGetLastError()));
        b200gym_destroy(h);
        return 1;
    }
    *h->invalid_seen = 0ULL;
    h->is_lunar = cfg->kind == B200GYM_LUNARLANDER || cfg->kind == B200GYM_LUNARLANDER_CONT;
    h->is_walker = cfg->kind == B200GYM_BIPEDALWALKER || cfg->kind == B200GYM_BIPEDALWALKER_HARDCORE;
    if (h->is_lunar) {  // LunarLander.__init__ arguments (lunar_lander.py:194-233)
        h->lunar_opts.continuous = cfg->kind == B200GYM_LUNARLANDER_CONT;
        h->lunar_opts.wind = (cfg->flags & B200GYM_LUNAR_ENABLE_WIND) != 0;
        h->lunar_opts.gravity = (float)cfg->param[0];
        h->lunar_opts.wind_power = cfg->param[1];
        h->lunar_opts.turbulence_power = cfg->param[2];
    }
    if (h->is_lunar || h->is_walker) {
        const bool lun = h->is_lunar;
        const size_t words = lun ? lunar::kWords
                                 : (cfg->kind == B200GYM_BIPEDALWALKER_HARDCORE ? walker::kWordsHC : walker::kWords);
        if (cudaMalloc(&h->lunar_rec, sizeof(uint32_t) * words * n) != cudaSuccess ||
            cudaMemset(h->lunar_rec, 0, sizeof(uint32_t) * words * n) != cudaSuccess ||
            cudaMalloc((void **)&h->reset_list, sizeof(int32_t) * n) != cudaSuccess ||
            cudaMalloc((void **)&h->toi_list, sizeof(int32_t) * n) != cudaSuccess ||
            cudaMalloc((void **)&h->toi_count, sizeof(int32_t) * kResetSlots) != cudaSuccess ||
            cudaMemset(h->toi_count, 0, sizeof(int32_t) * kResetSlots) != cudaSuccess ||
            cudaMalloc((void **)&h->toi_mid, sizeof(uint32_t) * kToiMidWords * n) != cudaSuccess ||
            cudaMalloc((void **)&h->reset_count, sizeof(int32_t) * kResetSlots) != cudaSuccess ||
            cudaMemset(h->reset_count, 0, sizeof(int32_t) * kResetSlots) != cudaSuccess ||
            (lun ? lunar_upload_consts(h) : walker_upload_consts(h))) {
            fail(nullptr, "b200gym_create: Box2D-task state allocation failed");
            b200gym_destroy(h);
            return 1;
        }
    }
    const cudaError_t ms[5] = {cudaMemset(h->state, 0, sizeof(double) * n * (h->S > 0 ? h->S : 1)),
                               cudaMemset(h->elapsed, 0, sizeof(int32_t) * n), cudaMemset(h->flags, 0, n),
                               cudaMemset(h->rng, 0, 32 * n), cudaMemset(h->invalid, 0, sizeof(unsigned long long))};
    bool ms_ok = true;
    for (cudaError_t mi : ms) ms_ok = ms_ok && mi == cudaSuccess;
    if (!ms_ok || cudaDeviceSynchronize() != cudaSuccess) {
        fail(nullptr, "b200gym_create: device initialisation failed: %s", cudaGetErrorString(cudaGetLastError()));
        b200gym_destroy(h);
        return 1;
    }
    *out = h;
    return 0;
}

static void free_host_io(b200gym *h) {
    if (!h->host_ready) return;
    cudaFreeHost(h->hio.actions); cudaFreeHost(h->hio.obs); cudaFreeHost(h->hio.reward);
    cudaFreeHost(h->hio.terminated); cudaFreeHost(h->hio.truncated); cudaFreeHost(h->hio.final_obs);
    cudaFreeHost(h->h_invalid);
    cudaFree(h->dio.actions);
    cudaFree(h->d_mask);
    if (h->hevent) cudaEventDestroy(h->hevent);
    for (cudaStream_t st : h->hstream)
        if (st) cudaStreamDestroy(st);
    h->host_ready = false;
}

extern "C" void b200gym_destroy(b200gym_t *h) {
    if (!h) return;
    DeviceGuard guard(h->device);
    free_host_io(h);
    cudaFree(h->state);
    cudaFree(h->elapsed);
    cudaFree(h->flags);
    cudaFree(h->rng);
    cudaFree(h->invalid);
    if (h->invalid_seen) cudaFreeHost(h->invalid_seen);
    cudaFree(h->lunar_rec);
    cudaFree(h->reset_list);
    cudaFree(h->reset_count);
    cudaFree(h->toi_list);
    cudaFree(h->toi_count);
    cudaFree(h->toi_mid);
    if (h->p2p.base) {
        for (int r = 0; r < h->p2p.world; r++)
            if (r != h->p2p.rank && h->p2p.peer[r]) cudaIpcCloseMemHandle(h->p2p.peer[r]);
        cudaFree(h->p2p.base);
        cudaFree(h->d_peer_flags);
    }
    delete h;
}

extern "C" int b200gym_seed_range(b200gym_t *h, const uint32_t base_words[4], int64_t first_index, void *stream) {
    if (!h || !base_words) return fail(h, "b200gym_seed_range: null argument");
    if (first_index < 0) return fail(h, "b200gym_seed_range: negative first_index");
    DeviceGuard guard(h->device);
    seed_range_kernel<<<blocks_for(h->n), kThreads, 0, (cudaStream_t)stream>>>(
        h->rng, h->n, base_words[0], base_words[1], base_words[2], base_words[3], (uint64_t)first_index);
    CK(h, cudaGetLastError());
    if (h->is_walker) {
        walker_clear_rng32_kernel<<<blocks_for(h->n), kThreads, 0, (cudaStream_t)stream>>>(h->lunar_rec, nullptr, h->n);
        CK(h, cudaGetLastError());
    }
    return 0;
}

extern "C" int b200gym_seed_each(b200gym_t *h, const uint32_t *ent_host, const uint8_t *mask_host, void *stream) {
    if (!h || !ent_host) return fail(h, "b200gym_seed_each: null argument");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t *d_ent = nullptr;
    uint8_t *d_mask = nullptr;
    CK(h, cudaMalloc(&d_ent, 16 * (size_t)h->n));
    cudaError_t e = cudaMemcpyAsync(d_ent, ent_host, 16 * (size_t)h->n, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && mask_host) {
        e = cudaMalloc(&d_mask, (size_t)h->n);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_mask, mask_host, (size_t)h->n, cudaMemcpyHostToDevice, st);
    }
    if (e == cudaSuccess) {
        seed_each_kernel<<<blocks_for(h->n), kThreads, 0, st>>>(h->rng, h->n, d_ent, d_mask);
        if (h->is_walker)
            walker_clear_rng32_kernel<<<blocks_for(h->n), kThreads, 0, st>>>(h->lunar_rec, d_mask, h->n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_ent);
    cudaFree(d_mask);
    if (e != cudaSuccess) return fail(h, "b200gym_seed_each: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int b200gym_reset(b200gym_t *h, const uint8_t *mask_dev, const double *bounds_host, float *obs_dev,
                             void *stream) {
    if (!h) return fail(h, "b200gym_reset: null handle");
    DeviceGuard guard(h->device);
    return launch_reset(h, mask_dev, bounds_host, obs_dev, (cudaStream_t)stream);
}

static StepArgs make_args(b200gym *h, const void *actions, float *obs, double *reward, uint8_t *term,
                          uint8_t *trunc, float *final_obs) {
    StepArgs a;
    a.state = h->state; a.elapsed = h->elapsed; a.flags = h->flags; a.rng = h->rng; a.invalid = h->invalid;
    a.invalid_seen = h->invalid_seen_dev;
    a.lunar_rec = h->lunar_rec;
    a.actions = actions; a.obs = obs; a.reward = reward; a.terminated = term; a.truncated = trunc;
    a.final_obs = final_obs;
    a.n = h->n; a.first = 0; a.count = h->n;
    a.max_steps = h->cfg.max_episode_steps; a.autoreset = h->cfg.autoreset; a.param0 = h->cfg.param[0];
    a.lunar_opts = h->lunar_opts;
    a.reset_list = h->reset_list; a.reset_count = h->reset_count;   // Box2D tasks (null otherwise); counter slot 0
    a.toi_list = h->toi_list; a.toi_count = h->toi_count; a.toi_mid = h->toi_mid;
    a.npeer = 0;
    a.bulk_sink = 0;
    a.ep_acc = h->ep.acc; a.ep_len = h->ep.len; a.ep_r = h->ep.r; a.ep_l = h->ep.l;
    a.ep_ring = h->ep.ring; a.ep_counter = h->ep.counter; a.ep_ring_size = h->ep.ring_size;
    return a;
}

extern "C" int b200gym_step(b200gym_t *h, const void *actions_dev, int action_dtype, float *obs_dev,
                            double *reward_dev, uint8_t *terminated_dev, uint8_t *truncated_dev,
                            float *final_obs_dev, void *stream) {
    if (!h) return fail(h, "b200gym_step: null handle");
    if (!actions_dev || !obs_dev || !reward_dev || !terminated_dev || !truncated_dev)
        return fail(h, "b200gym_step: null buffer");
    DeviceGuard guard(h->device);
    const StepArgs a = make_args(h, actions_dev, obs_dev, reward_dev, terminated_dev, truncated_dev, final_obs_dev);
    return launch_step(h, a, action_dtype, (cudaStream_t)stream);
}

extern "C" int b200gym_invalid_actions(b200gym_t *h, void *stream, int64_t *count_out) {
    if (!h || !count_out) return fail(h, "b200gym_invalid_actions: null argument");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long v = 0;
    CK(h, cudaMemcpyAsync(&v, h->invalid, sizeof v, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemsetAsync(h->invalid, 0, sizeof v, st));
    CK(h, cudaStreamSynchronize(st));
    *h->invalid_seen = 0ULL;
    *count_out = (int64_t)v;
    return 0;
}

extern "C" int b200gym_invalid_seen(const b200gym_t *h) {
    if (!h || !h->invalid_seen) return -1;
    return *reinterpret_cast<volatile unsigned long long *>(h->invalid_seen) != 0ULL ? 1 : 0;
}

extern "C" int b200gym_selftest_trig(const double *x_dev, int64_t n, double *sin_dev, double *cos_dev, double *sq_dev,
                                     void *stream) {
    if (!x_dev || !sin_dev || !cos_dev || n <= 0) return fail(nullptr, "b200gym_selftest_trig: bad argument");
    const int dev = device_of(x_dev);
    if (dev < 0) return fail(nullptr, "b200gym_selftest_trig: x is not a device pointer");
    DeviceGuard guard(dev);
    selftest_trig_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(x_dev, n, sin_dev, cos_dev, sq_dev);
    CK(nullptr, cudaGetLastError());
    return 0;
}

extern "C" int b200gym_box2d_overflows(b200gym_t *h, void *stream, int64_t *count_out) {
    if (!h || !count_out) return fail(h, "b200gym_box2d_overflows: null argument");
    if (!h->is_lunar && !h->is_walker) return fail(h, "b200gym_box2d_overflows: not a Box2D-task handle");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long *d = nullptr, v = 0;
    CK(h, cudaMalloc((void **)&d, sizeof *d));
    cudaError_t e = cudaMemsetAsync(d, 0, sizeof *d, st);
    if (e == cudaSuccess) {
        const int64_t row = h->is_lunar ? lunar::W_FLAGS : walker::W_FLAGS;
        box2d_overflow_kernel<<<blocks_for(h->n), kThreads, 0, st>>>(h->lunar_rec + row * h->n, h->n, d);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&v, d, sizeof v, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d);
    if (e != cudaSuccess) return fail(h, "b200gym_box2d_overflows: %s", cudaGetErrorString(e));
    *count_out = (int64_t)v;
    return 0;
}

extern "C" int b200gym_selftest(int device, int64_t samples, uint64_t seed, int64_t *mismatches_out) {
    if (!mismatches_out || samples <= 0) return fail(nullptr, "b200gym_selftest: bad argument");
    DeviceGuard guard(device);
    unsigned long long *d = nullptr;
    if (cudaMalloc(&d, sizeof *d) != cudaSuccess) return fail(nullptr, "b200gym_selftest: cudaMalloc failed");
    cudaMemset(d, 0, sizeof *d);
    selftest_div_kernel<<<blocks_for(samples), kThreads>>>(samples, seed, d);
    unsigned long long v = 0;
    cudaError_t e = cudaMemcpy(&v, d, sizeof v, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(nullptr, "b200gym_selftest: %s", cudaGetErrorString(e));
    *mismatches_out = (int64_t)v;
    return 0;
}

// ---- fused all-gather over NVLink peer memory ----------------------------------------------
static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

extern "C" int b200gym_p2p_create(b200gym_t *h, int world, int rank, void *ipc_handle_out /*64 B*/,
                                  b200gym_p2p_layout *layout_out) {
    if (!h || !ipc_handle_out || !layout_out) return fail(h, "b200gym_p2p_create: null argument");
    if (world < 1 || world > B200GYM_MAX_PEERS + 1 || rank < 0 || rank >= world)
        return fail(h, "b200gym_p2p_create: bad world/rank %d/%d (at most %d ranks)", world, rank, B200GYM_MAX_PEERS + 1);
    if (h->p2p.base) return fail(h, "b200gym_p2p_create: already created");
    DeviceGuard guard(h->device);
    auto &P = h->p2p;
    const size_t rows = (size_t)world * (size_t)h->n;
    P.world = world;
    P.rank = rank;
    P.off_obs = 0;
    P.off_reward = align_up(P.off_obs + rows * h->D * sizeof(float), 256);
    P.off_term = align_up(P.off_reward + rows * sizeof(double), 256);
    P.off_trunc = align_up(P.off_term + rows, 256);
    P.set_bytes = align_up(P.off_trunc + rows, 256);
    P.off_flags = 2 * P.set_bytes;          // [0,64): one uint64 step counter per rank; [128,132): sticky time-out word
    P.bytes = P.off_flags + 256;
    if (const char *ts = getenv("B200GYM_P2P_TIMEOUT_S")) {
        const double v = atof(ts);
        if (v > 0.0) P.timeout_ns = (unsigned long long)(v * 1e9);
    }
    CK(h, cudaMalloc((void **)&P.base, P.bytes));
    CK(h, cudaMemset(P.base, 0, P.bytes));
    CK(h, cudaDeviceSynchronize());
    cudaIpcMemHandle_t ipc;
    CK(h, cudaIpcGetMemHandle(&ipc, P.base));
    static_assert(sizeof(ipc) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(ipc_handle_out, &ipc, sizeof ipc);
    layout_out->base = P.base;
    layout_out->set_bytes = P.set_bytes;
    layout_out->off_obs = P.off_obs;
    layout_out->off_reward = P.off_reward;
    layout_out->off_terminated = P.off_term;
    layout_out->off_truncated = P.off_trunc;
    layout_out->rows = (int64_t)rows;
    return 0;
}

extern "C" int b200gym_p2p_connect(b200gym_t *h, const void *all_ipc_handles /*world x 64 B*/) {
    if (!h || !all_ipc_handles) return fail(h, "b200gym_p2p_connect: null argument");
    auto &P = h->p2p;
    if (!P.base) return fail(h, "b200gym_p2p_connect: call b200gym_p2p_create first");
    if (P.connected) return 0;
    DeviceGuard guard(h->device);
    for (int r = 0; r < P.world; r++) {
        if (r == P.rank) {
            P.peer[r] = P.base;
            continue;
        }
        cudaIpcMemHandle_t ipc;
        memcpy(&ipc, (const char *)all_ipc_handles + 64 * r, sizeof ipc);
        void *ptr = nullptr;
        CK(h, cudaIpcOpenMemHandle(&ptr, ipc, cudaIpcMemLazyEnablePeerAccess));
        P.peer[r] = (unsigned char *)ptr;
    }
    P.connected = true;
    return 0;
}

extern "C" int b200gym_step_p2p(b200gym_t *h, const void *actions_dev, int action_dtype, float *final_obs_dev,
                                void *stream, int *set_out) {
    if (!h || !actions_dev) return fail(h, "b200gym_step_p2p: null argument");
    auto &P = h->p2p;
    if (!P.connected) return fail(h, "b200gym_step_p2p: peers are not connected");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    P.step += 1;
    const int set = (int)(P.step & 1);
    const size_t row0 = (size_t)P.rank * (size_t)h->n;
    auto obs_of = [&](unsigned char *b) { return (float *)(b + set * P.set_bytes + P.off_obs) + row0 * h->D; };
    auto rew_of = [&](unsigned char *b) { return (double *)(b + set * P.set_bytes + P.off_reward) + row0; };
    auto term_of = [&](unsigned char *b) { return (uint8_t *)(b + set * P.set_bytes + P.off_term) + row0; };
    auto trunc_of = [&](unsigned char *b) { return (uint8_t *)(b + set * P.set_bytes + P.off_trunc) + row0; };
    StepArgs a = make_args(h, actions_dev, obs_of(P.base), rew_of(P.base), term_of(P.base), trunc_of(P.base),
                           final_obs_dev);
    int np = 0;
    for (int r = 0; r < P.world; r++) {
        if (r == P.rank) continue;
        a.peer_obs[np] = obs_of(P.peer[r]);
        a.peer_reward[np] = rew_of(P.peer[r]);
        a.peer_term[np] = term_of(P.peer[r]);
        a.peer_trunc[np] = trunc_of(P.peer[r]);
        np++;
    }
    a.npeer = np;
    if (P.world > 1 && !h->d_peer_flags) {
        unsigned long long *pf[B200GYM_MAX_PEERS + 1];
        for (int r = 0; r < P.world; r++) pf[r] = (unsigned long long *)(P.peer[r] + P.off_flags);
        CK(h, cudaMalloc((void **)&h->d_peer_flags, sizeof pf));
        CK(h, cudaMemcpy(h->d_peer_flags, pf, sizeof pf, cudaMemcpyHostToDevice));
    }
    if (launch_step(h, a, action_dtype, st)) return 1;
    if (P.world > 1) {
        // tell every peer that my rows of step `P.step` are in its buffers, then wait for theirs
        p2p_sync_kernel<<<1, 32, 0, st>>>(h->d_peer_flags, (const unsigned long long *)(P.base + P.off_flags), P.world,
                                          P.rank, P.step, P.timeout_ns, (int *)(P.base + P.off_flags + 128));
        CK(h, cudaGetLastError());
    }
    if (set_out) *set_out = set;
    return 0;
}

extern "C" int b200gym_p2p_status(b200gym_t *h, void *stream, int *timed_out_peer) {
    if (!h || !timed_out_peer) return fail(h, "b200gym_p2p_status: null argument");
    auto &P = h->p2p;
    if (!P.base) return fail(h, "b200gym_p2p_status: no gather allocation");
    DeviceGuard guard(h->device);
    int v = 0;
    CK(h, cudaMemcpyAsync(&v, P.base + P.off_flags + 128, sizeof v, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK(h, cudaStreamSynchronize((cudaStream_t)stream));
    *timed_out_peer = v - 1;   // -1: every step barrier completed
    if (v) return fail(h, "b200gym_step_p2p: rank %d did not deliver its rows within %.0f s (peer lost?)", v - 1,
                       (double)P.timeout_ns * 1e-9);
    return 0;
}

// ---- stateless device utilities for the vector-aware wrappers (SURVEY.md 8f) -----------------------
extern "C" int b200gym_set_episode_stats(b200gym_t *h, float *return_acc_dev, int32_t *length_acc_dev, float *episode_r_dev,
                                         int32_t *episode_l_dev, uint64_t *ring_dev, uint64_t *counter_dev, int ring_size) {
    if (!h) return fail(h, "b200gym_set_episode_stats: null handle");
    if (!return_acc_dev) {   // off
        h->ep = {};
        return 0;
    }
    if (!length_acc_dev || !episode_r_dev || !episode_l_dev || !counter_dev || ring_size < 0 || (ring_size > 0 && !ring_dev))
        return fail(h, "b200gym_set_episode_stats: bad argument");
    h->ep.acc = return_acc_dev; h->ep.len = length_acc_dev; h->ep.r = episode_r_dev; h->ep.l = episode_l_dev;
    h->ep.ring = (unsigned long long *)ring_dev; h->ep.counter = (unsigned long long *)counter_dev; h->ep.ring_size = ring_size;
    return 0;
}

extern "C" int b200gym_episode_stats(const double *reward_dev, const uint8_t *terminated_dev, const uint8_t *truncated_dev,
                                     float *return_acc_dev, int32_t *length_acc_dev, float *episode_r_dev,
                                     int32_t *episode_l_dev, uint8_t *episode_mask_dev, uint64_t *ring_dev,
                                     uint64_t *counter_dev, int ring_size, int64_t n, void *stream) {
    if (!reward_dev || !terminated_dev || !truncated_dev || !return_acc_dev || !length_acc_dev || !episode_r_dev ||
        !episode_l_dev || !episode_mask_dev || !counter_dev || n <= 0 || (ring_size > 0 && !ring_dev))
        return fail(nullptr, "b200gym_episode_stats: bad argument");
    const int dev = device_of(reward_dev);
    if (dev < 0) return fail(nullptr, "b200gym_episode_stats: reward is not a device pointer");
    DeviceGuard guard(dev);
    episode_stats_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(
        reward_dev, terminated_dev, truncated_dev, return_acc_dev, length_acc_dev, episode_r_dev, episode_l_dev,
        episode_mask_dev, (unsigned long long *)ring_dev, (unsigned long long *)counter_dev, ring_size, n);
    CK(nullptr, cudaGetLastError());
    return 0;
}

static int norm_dims_ok(int dim) { return dim == 1 || dim == 2 || dim == 3 || dim == 4 || dim == 6 || dim == 8 || dim == 24; }

static unsigned norm_grid(int64_t total, int block) {
    int64_t g = (total + block - 1) / block;
    if (g > 1184) g = 1184;       // 148 SMs x 8: one resident wave, grid-stride beyond
    return (unsigned)(g < 1 ? 1 : g);
}

extern "C" int b200gym_rms_moments(const void *x_dev, int is_f64, int64_t n, int dim, const double *stats_dev,
                                   double *scratch_dev, void *stream) {
    if (!x_dev || !stats_dev || !scratch_dev || n <= 0 || !norm_dims_ok(dim))
        return fail(nullptr, "b200gym_rms_moments: bad argument (dim must be one of 1, 2, 3, 4, 6, 8, 24)");
    const int dev = device_of(x_dev);
    if (dev < 0) return fail(nullptr, "b200gym_rms_moments: x is not a device pointer");
    DeviceGuard guard(dev);
    const int block = (dim == 3 || dim == 6 || dim == 24) ? 192 : 256;
    const int64_t total = n * dim;
    cudaStream_t st = (cudaStream_t)stream;
    if (is_f64)
        rms_moments_kernel<double, false><<<norm_grid(total, block), block, 0, st>>>((const double *)x_dev, nullptr, nullptr,
                                                                                   0.0, total, dim, stats_dev, scratch_dev);
    else
        rms_moments_kernel<float, false><<<norm_grid(total, block), block, 0, st>>>((const float *)x_dev, nullptr, nullptr,
                                                                                  0.0, total, dim, stats_dev, scratch_dev);
    CK(nullptr, cudaGetLastError());
    return 0;
}

extern "C" int b200gym_return_moments(double *returns_dev, const double *reward_dev, double gamma, int64_t n,
                                      const double *stats_dev, double *scratch_dev, void *stream) {
    if (!returns_dev || !reward_dev || !stats_dev || !scratch_dev || n <= 0)
        return fail(nullptr, "b200gym_return_moments: bad argument");
    const int dev = device_of(returns_dev);
    if (dev < 0) return fail(nullptr, "b200gym_return_moments: returns is not a device pointer");
    DeviceGuard guard(dev);
    rms_moments_kernel<double, true><<<norm_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(nullptr, returns_dev, reward_dev, gamma,
                                                                                         n, 1, stats_dev, scratch_dev);
    CK(nullptr, cudaGetLastError());
    return 0;
}

extern "C" int b200gym_rms_apply_obs(const float *obs_dev, float *out_dev, int64_t n, int dim, const double *stats_dev,
                                     double *stats_next_dev, const double *scratch_dev, double *scratch_next_dev,
                                     double batch_count, double epsilon, int update, void *stream) {
    if (!obs_dev || !out_dev || !stats_dev || !stats_next_dev || !scratch_dev || !scratch_next_dev || n <= 0 ||
        !norm_dims_ok(dim))
        return fail(nullptr, "b200gym_rms_apply_obs: bad argument");
    const int dev = device_of(obs_dev);
    if (dev < 0) return fail(nullptr, "b200gym_rms_apply_obs: obs is not a device pointer");
    DeviceGuard guard(dev);
    const int block = (dim == 3 || dim == 6 || dim == 24) ? 192 : 256;
    rms_apply_kernel<false><<<norm_grid(n * dim, block), block, 0, (cudaStream_t)stream>>>(
        obs_dev, out_dev, nullptr, nullptr, nullptr, nullptr, nullptr, n * dim, dim, stats_dev, stats_next_dev, scratch_dev,
        scratch_next_dev, batch_count, epsilon, update);
    CK(nullptr, cudaGetLastError());
    return 0;
}

extern "C" int b200gym_rms_apply_reward(const double *reward_dev, double *out_dev, double *returns_dev,
                                        const uint8_t *terminated_dev, const uint8_t *truncated_dev, int64_t n,
                                        const double *stats_dev, double *stats_next_dev, const double *scratch_dev,
                                        double *scratch_next_dev, double batch_count, double epsilon, void *stream) {
    if (!reward_dev || !out_dev || !returns_dev || !terminated_dev || !truncated_dev || !stats_dev || !stats_next_dev ||
        !scratch_dev || !scratch_next_dev || n <= 0)
        return fail(nullptr, "b200gym_rms_apply_reward: bad argument");
    const int dev = device_of(reward_dev);
    if (dev < 0) return fail(nullptr, "b200gym_rms_apply_reward: reward is not a device pointer");
    DeviceGuard guard(dev);
    rms_apply_kernel<true><<<norm_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(
        nullptr, nullptr, reward_dev, out_dev, returns_dev, terminated_dev, truncated_dev, n, 1, stats_dev, stats_next_dev,
        scratch_dev, scratch_next_dev, batch_count, epsilon, 1);
    CK(nullptr, cudaGetLastError());
    return 0;
}

// ---- host-buffer path -------------------------------------------------------
// The staging buffers are page-locked AND mapped into the device's address space: the step kernel writes its
// results straight into host memory (for the classic-control kinds as bulk shared->global copies of 256-env
// tiles, kernel G with the host as its only destination), so the device->host transfer IS the kernel's store
// stream -- no result mirrors in HBM, no separate D2H copies, no compaction pass for the final observations.
static int ensure_host_io(b200gym *h) {
    if (h->host_ready) return 0;
    const size_t n = (size_t)h->n;
    const size_t act_bytes = h->A == 0 ? n * sizeof(int64_t) : n * h->A * sizeof(float);
    const size_t obs_bytes = n * h->D * sizeof(float);
    const unsigned fl = cudaHostAllocMapped;
    for (int k = 0; k < 2; k++) CK(h, cudaStreamCreateWithFlags(&h->hstream[k], cudaStreamNonBlocking));
    CK(h, cudaHostAlloc(&h->hio.actions, act_bytes, fl));
    CK(h, cudaHostAlloc((void **)&h->hio.obs, obs_bytes, fl));
    CK(h, cudaHostAlloc((void **)&h->hio.reward, n * sizeof(double), fl));
    CK(h, cudaHostAlloc((void **)&h->hio.terminated, n, fl));
    CK(h, cudaHostAlloc((void **)&h->hio.truncated, n, fl));
    CK(h, cudaHostAlloc((void **)&h->hio.final_obs, obs_bytes, fl));
    CK(h, cudaHostAlloc((void **)&h->h_invalid, sizeof(unsigned long long), fl));
    memset(h->hio.actions, 0, act_bytes);
    memset(h->hio.final_obs, 0, obs_bytes);
    // device aliases of the mapped host buffers (identical to the host pointers under unified addressing)
    CK(h, cudaHostGetDevicePointer((void **)&h->dio.obs, h->hio.obs, 0));
    CK(h, cudaHostGetDevicePointer((void **)&h->dio.reward, h->hio.reward, 0));
    CK(h, cudaHostGetDevicePointer((void **)&h->dio.terminated, h->hio.terminated, 0));
    CK(h, cudaHostGetDevicePointer((void **)&h->dio.truncated, h->hio.truncated, 0));
    CK(h, cudaHostGetDevicePointer((void **)&h->dio.final_obs, h->hio.final_obs, 0));
    CK(h, cudaMalloc(&h->dio.actions, act_bytes));   // the actions do live in HBM: every env reads its own once
    CK(h, cudaMalloc((void **)&h->d_mask, n));
    CK(h, cudaEventCreateWithFlags(&h->hevent, cudaEventDisableTiming));
    h->host_ready = true;
    return 0;
}

extern "C" int b200gym_host_buffers(b200gym_t *h, b200gym_host_io *out) {
    if (!h || !out) return fail(h, "b200gym_host_buffers: null argument");
    DeviceGuard guard(h->device);
    if (ensure_host_io(h)) return 1;
    *out = h->hio;
    return 0;
}

static size_t action_size(int action_dtype) {
    switch (action_dtype) {
    case B200GYM_ACT_I64: return 8;
    case B200GYM_ACT_I32: return 4;
    case B200GYM_ACT_U8: return 1;
    default: return 4;
    }
}

// enqueue the chunked pipeline; any failure is reported after both streams have drained
static int step_host_enqueue(b200gym *h, const void *actions_host, int action_dtype, bool want_final) {
    const size_t asz = action_size(action_dtype) * (h->A == 0 ? 1 : h->A);
    const int64_t n = h->n;
    int64_t chunks = n >> 18;                       // 2^20 envs -> 4 chunks: H2D of chunk c+1 under the kernel of c
    chunks = chunks < 1 ? 1 : (chunks > 4 ? 4 : chunks);
    if (const char *hc = getenv("B200GYM_HOST_CHUNKS")) {  // tuning runs
        const int v = atoi(hc);
        if (v >= 1 && v <= 64) chunks = v;
    }
    const int64_t per = ((n + chunks - 1) / chunks + kThreads - 1) / kThreads * kThreads;
    StepArgs a = make_args(h, h->dio.actions, h->dio.obs, h->dio.reward, h->dio.terminated, h->dio.truncated,
                           want_final ? h->dio.final_obs : nullptr);
    a.bulk_sink = 1;
    int c = 0;
    for (int64_t lo = 0; lo < n; lo += per, c++) {
        const int64_t cnt = (lo + per < n) ? per : n - lo;
        cudaStream_t st = h->hstream[c & 1];
        CK(h, cudaMemcpyAsync((char *)h->dio.actions + lo * asz, (const char *)actions_host + lo * asz, cnt * asz,
                              cudaMemcpyHostToDevice, st));
        a.first = lo;
        a.count = cnt;
        a.reset_count = h->reset_count ? h->reset_count + (c % kResetSlots) : nullptr;
        a.toi_count = h->toi_count ? h->toi_count + (c % kResetSlots) : nullptr;
        if (launch_step(h, a, action_dtype, st)) return 1;
    }
    if (c > 1) {  // stream 0 also waits for the chunks of stream 1
        CK(h, cudaEventRecord(h->hevent, h->hstream[1]));
        CK(h, cudaStreamWaitEvent(h->hstream[0], h->hevent, 0));
    }
    // the sticky invalid-action counter rides along (no separate round trip afterwards)
    CK(h, cudaMemcpyAsync(h->h_invalid, h->invalid, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->hstream[0]));
    CK(h, cudaMemsetAsync(h->invalid, 0, sizeof(unsigned long long), h->hstream[0]));
    return 0;
}

extern "C" int b200gym_step_host(b200gym_t *h, const void *actions_host, int action_dtype, float *obs_host,
                                 double *reward_host, uint8_t *terminated_host, uint8_t *truncated_host,
                                 float *final_obs_host, int64_t *invalid_out) {
    if (!h) return fail(h, "b200gym_step_host: null handle");
    DeviceGuard guard(h->device);
    if (ensure_host_io(h)) return 1;
    if (h->A == 0 ? (action_dtype == B200GYM_ACT_F32) : (action_dtype != B200GYM_ACT_F32))
        return fail(h, "b200gym_step_host: action dtype code %d does not fit this env's action space", action_dtype);
    if (!actions_host) {
        actions_host = h->hio.actions;
        action_dtype = h->A == 0 ? B200GYM_ACT_I64 : B200GYM_ACT_F32;
    }
    const bool want_final = final_obs_host != nullptr && h->cfg.autoreset;
    const int rc = step_host_enqueue(h, actions_host, action_dtype, want_final);
    // drain both streams whatever happened: nothing may still be writing into host memory when we return
    const cudaError_t e1 = cudaStreamSynchronize(h->hstream[1]), e0 = cudaStreamSynchronize(h->hstream[0]);
    if (rc) return 1;
    if (e0 != cudaSuccess || e1 != cudaSuccess)
        return fail(h, "b200gym_step_host: %s", cudaGetErrorString(e0 != cudaSuccess ? e0 : e1));
    if (invalid_out) *invalid_out = (int64_t)*h->h_invalid;
    *h->invalid_seen = 0ULL;   // reported (and the device counter cleared) with this call
    // results are in the mapped staging buffers; callers that brought their own arrays get a host copy
    const size_t n = (size_t)h->n, osz = sizeof(float) * h->D;
    if (obs_host && obs_host != h->hio.obs) memcpy(obs_host, h->hio.obs, n * osz);
    if (reward_host && reward_host != h->hio.reward) memcpy(reward_host, h->hio.reward, n * sizeof(double));
    if (terminated_host && terminated_host != h->hio.terminated) memcpy(terminated_host, h->hio.terminated, n);
    if (truncated_host && truncated_host != h->hio.truncated) memcpy(truncated_host, h->hio.truncated, n);
    if (want_final && final_obs_host != h->hio.final_obs)   // rows of the envs that finished in this step only
        for (size_t i = 0; i < n; i++)
            if (h->hio.terminated[i] | h->hio.truncated[i])
                memcpy((char *)final_obs_host + i * osz, (const char *)h->hio.final_obs + i * osz, osz);
    return 0;
}

extern "C" int b200gym_reset_host(b200gym_t *h, const uint8_t *mask_host, const double *bounds_host,
                                  float *obs_host) {
    if (!h) return fail(h, "b200gym_reset_host: null handle");
    DeviceGuard guard(h->device);
    if (ensure_host_io(h)) return 1;
    const size_t n = (size_t)h->n;
    cudaStream_t st = h->hstream[0];
    // the reset kernel writes the rows of the (masked) envs straight into the mapped staging buffer; rows of
    // envs that are not reset keep their content
    if (obs_host && obs_host != h->hio.obs && mask_host) memcpy(h->hio.obs, obs_host, n * h->D * sizeof(float));
    if (mask_host) CK(h, cudaMemcpyAsync(h->d_mask, mask_host, n, cudaMemcpyHostToDevice, st));
    const int rc = launch_reset(h, mask_host ? h->d_mask : nullptr, bounds_host, h->dio.obs, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (rc) return 1;
    if (e != cudaSuccess) return fail(h, "b200gym_reset_host: %s", cudaGetErrorString(e));
    if (obs_host && obs_host != h->hio.obs) memcpy(obs_host, h->hio.obs, n * h->D * sizeof(float));
    return 0;
}

// ---- state access -----------------------------------------------------------
extern "C" int b200gym_get_state(b200gym_t *h, double *state_dev, int32_t *elapsed_dev, uint64_t *rng_dev,
                                 void *stream) {
    if (!h) return fail(h, "b200gym_get_state: null handle");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (state_dev) {
        state_get_kernel<<<blocks_for(h->n), kThreads, 0, st>>>(h->state, state_dev, h->n, h->S);
        CK(h, cudaGetLastError());
    }
    if (elapsed_dev)
        CK(h, cudaMemcpyAsync(elapsed_dev, h->elapsed, sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToDevice, st));
    if (rng_dev) CK(h, cudaMemcpyAsync(rng_dev, h->rng, 32 * (size_t)h->n, cudaMemcpyDeviceToDevice, st));
    return 0;
}

extern "C" int b200gym_lunar_get_bodies(b200gym_t *h, float *bodies_dev, int32_t *flags_dev, void *stream) {
    if (!h || !bodies_dev || !flags_dev) return fail(h, "b200gym_lunar_get_bodies: null argument");
    if (!h->is_lunar) return fail(h, "b200gym_lunar_get_bodies: not a LunarLander handle");
    DeviceGuard guard(h->device);
    lunar_bodies_kernel<<<blocks_for(h->n), kThreads, 0, (cudaStream_t)stream>>>(h->lunar_rec, h->elapsed, bodies_dev,
                                                                                 flags_dev, h->n);
    CK(h, cudaGetLastError());
    return 0;
}

extern "C" int b200gym_lunar_wind_idx(b200gym_t *h, int32_t *wind_idx_host, int32_t *torque_idx_host, int set) {
    if (!h || !wind_idx_host || !torque_idx_host) return fail(h, "b200gym_lunar_wind_idx: null argument");
    if (!h->is_lunar) return fail(h, "b200gym_lunar_wind_idx: not a LunarLander handle");
    DeviceGuard guard(h->device);
    int32_t *d = nullptr;
    const size_t bytes = sizeof(int32_t) * (size_t)h->n;
    CK(h, cudaMalloc((void **)&d, 2 * bytes));
    cudaError_t e = cudaSuccess;
    if (set) {
        e = cudaMemcpy(d, wind_idx_host, bytes, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(d + h->n, torque_idx_host, bytes, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) {
        lunar_wind_idx_kernel<<<blocks_for(h->n), kThreads>>>(h->lunar_rec, d, d + h->n, h->n, set);
        e = cudaDeviceSynchronize();
    }
    if (e == cudaSuccess && !set) {
        e = cudaMemcpy(wind_idx_host, d, bytes, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(torque_idx_host, d + h->n, bytes, cudaMemcpyDeviceToHost);
    }
    cudaFree(d);
    if (e != cudaSuccess) return fail(h, "b200gym_lunar_wind_idx: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int b200gym_walker_get_bodies(b200gym_t *h, float *bodies_dev, int32_t *flags_dev, void *stream) {
    if (!h || !bodies_dev || !flags_dev) return fail(h, "b200gym_walker_get_bodies: null argument");
    if (!h->is_walker) return fail(h, "b200gym_walker_get_bodies: not a BipedalWalker handle");
    DeviceGuard guard(h->device);
    walker_bodies_kernel<<<blocks_for(h->n), kThreads, 0, (cudaStream_t)stream>>>(h->lunar_rec, bodies_dev, flags_dev, h->n);
    CK(h, cudaGetLastError());
    return 0;
}

extern "C" int b200gym_walker_get_terrain(b200gym_t *h, float *terrain_dev, float *polys_dev, int32_t *npoly_dev, void *stream) {
    if (!h || !terrain_dev) return fail(h, "b200gym_walker_get_terrain: null argument");
    if (!h->is_walker) return fail(h, "b200gym_walker_get_terrain: not a BipedalWalker handle");
    DeviceGuard guard(h->device);
    walker_terrain_kernel<<<blocks_for(h->n), kThreads, 0, (cudaStream_t)stream>>>(
        h->lunar_rec, terrain_dev, polys_dev, npoly_dev, h->n, h->cfg.kind == B200GYM_BIPEDALWALKER_HARDCORE);
    CK(h, cudaGetLastError());
    return 0;
}

extern "C" int b200gym_set_state(b200gym_t *h, const double *state_dev, const int32_t *elapsed_dev,
                                 const uint64_t *rng_dev, void *stream) {
    if (!h) return fail(h, "b200gym_set_state: null handle");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (state_dev) {
        state_set_kernel<<<blocks_for(h->n), kThreads, 0, st>>>(h->state, state_dev, h->n, h->S);
        CK(h, cudaGetLastError());
    }
    if (elapsed_dev)
        CK(h, cudaMemcpyAsync(h->elapsed, elapsed_dev, sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToDevice, st));
    if (rng_dev) CK(h, cudaMemcpyAsync(h->rng, rng_dev, 32 * (size_t)h->n, cudaMemcpyDeviceToDevice, st));
    return 0;
}
