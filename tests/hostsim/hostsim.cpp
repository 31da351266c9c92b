// hostsim.cpp -- the device solver source of the Box2D tasks, compiled for the CPU.
//
// TEST INFRASTRUCTURE (never shipped, never imported by gym_b200/): includes gym_b200/csrc/{rng,envs,b2lite,lunar,
// walker}.cuh and box2d_consts.h through tests/hostsim/cuda_shim.h.  tests/test_hostsim_cpu.py compares it bit for bit
// with the C oracle, so the `-m "not gpu"` suite exercises the code the kernels run: solver, scenes, record packing,
// host-computed constants, numpy-compatible RNG.
//   hs_reset calls the per-env reset body the reset kernels of gym_b200/csrc/b200gym.cu call
//   (lunar::reset_from_record, walker::reset_from_record).
//   hs_step drives env_step with a plain loop on the record layout of box2d_step_kernel, with SolveTOI and the
//   autoreset inline, as the oracle does (load -> env_step -> TimeLimit -> autoreset -> store).  Its autoreset resets
//   the in-flight World by hand: the device's autoreset (box2d_reset_list_kernel, which resets from the record) is
//   covered in this suite only through hs_reset, not through the step.
#include "cuda_shim.h"

#include <cstdlib>
#include <vector>

#include "../../gym_b200/csrc/rng.cuh"
#include "../../gym_b200/csrc/envs.cuh"
#include "../../gym_b200/csrc/box2d_consts.h"

using bgym::Pcg64;

namespace {

struct Sim {
    int kind = 0;            // enum b200gym_kind: 5 lunar, 7 lunar continuous, 6 walker, 8 walker hardcore
    int64_t n = 0;
    int max_steps = 0;
    lunar::Opts opts{};
    std::vector<uint32_t> rec;       // [words][n]
    std::vector<uint64_t> rng;       // [n][4]
    std::vector<int32_t> elapsed;
    bool lunar() const { return kind == 5 || kind == 7; }
    bool hardcore() const { return kind == 8; }
};

bool g_consts_ready = false;
void ensure_consts() {
    if (g_consts_ready) return;
    b2l_host::lunar_consts(lunar::kC);
    b2l_host::walker_consts(walker::kC);
    g_consts_ready = true;
}

template <bool HC>
void walker_step_env(Sim &S, int64_t i, const float *act, float *obs_out, double *reward, uint8_t *term, uint8_t *trunc,
                     float *final_obs) {                  // box2d_step_kernel<WalkerTask<HC>>
    const float action[4] = {act[4 * i], act[4 * i + 1], act[4 * i + 2], act[4 * i + 3]};
    walker::World W;
    walker::Rng rng;
    walker::load_world(W, S.rec.data(), S.n, i, rng, HC);
    int32_t elapsed = S.elapsed[i];
    float obs[24];
    double r;
    bool terminated;
    walker::env_step<HC>(W, action, false, walker::V(0.0f, 0.0f), obs, r, terminated);
    elapsed += 1;
    const bool truncated = (S.max_steps > 0) && (elapsed >= S.max_steps);
    reward[i] = r; term[i] = terminated ? 1 : 0; trunc[i] = truncated ? 1 : 0;
    if (terminated || truncated) {
        if (final_obs) std::memcpy(final_obs + 24 * i, obs, sizeof obs);
        rng.g = bgym::pcg64_load(&S.rng[4 * i]);
        walker::env_reset<HC>(W, rng, obs);
        bgym::pcg64_store(&S.rng[4 * i], rng.g);
        elapsed = 0;
    }
    walker::store_world(W, S.rec.data(), S.n, i, rng, HC);
    S.elapsed[i] = elapsed;
    std::memcpy(obs_out + 24 * i, obs, sizeof obs);
}

}  // namespace

extern "C" {

void *hs_create(int kind, int64_t n, int max_steps, int wind, double gravity, double wind_power, double turbulence_power) {
    if (n <= 0 || kind < 5 || kind > 8) return nullptr;
    ensure_consts();
    Sim *S = new Sim();
    S->kind = kind; S->n = n; S->max_steps = max_steps;
    S->opts.continuous = kind == 7; S->opts.wind = wind != 0; S->opts.gravity = (float)gravity;
    S->opts.wind_power = wind_power; S->opts.turbulence_power = turbulence_power;
    const size_t words = S->lunar() ? lunar::kWords : (S->hardcore() ? walker::kWordsHC : walker::kWords);
    S->rec.assign(words * (size_t)n, 0u);
    S->rng.assign(4 * (size_t)n, 0ull);
    S->elapsed.assign((size_t)n, 0);
    return S;
}
void hs_destroy(void *h) { delete (Sim *)h; }

void hs_seed_range(void *h, const uint32_t base[4], int64_t first) {   // seed_range_kernel (+ walker_clear_rng32_kernel)
    Sim &S = *(Sim *)h;
    using bgym::u128;
    const u128 b = ((u128)base[3] << 96) | ((u128)base[2] << 64) | ((u128)base[1] << 32) | (u128)base[0];
    for (int64_t i = 0; i < S.n; i++) {
        const u128 seed = b + (u128)(uint64_t)(first + i);
        const uint32_t ent[4] = {(uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)(seed >> 64), (uint32_t)(seed >> 96)};
        Pcg64 g;
        bgym::pcg64_from_entropy(g, ent);
        bgym::pcg64_store_full(&S.rng[4 * i], g);
        if (!S.lunar()) { S.rec[(int64_t)walker::W_RNG32 * S.n + i] = 0u; S.rec[(int64_t)(walker::W_RNG32 + 1) * S.n + i] = 0u; }
    }
}

void hs_set_wind_idx(void *h, const int32_t *wind, const int32_t *torque) {
    Sim &S = *(Sim *)h;
    for (int64_t i = 0; i < S.n; i++) {
        S.rec[(int64_t)lunar::W_WIND * S.n + i] = (uint32_t)wind[i];
        S.rec[(int64_t)(lunar::W_WIND + 1) * S.n + i] = (uint32_t)torque[i];
    }
}
void hs_get_wind_idx(void *h, int32_t *wind, int32_t *torque) {
    Sim &S = *(Sim *)h;
    for (int64_t i = 0; i < S.n; i++) {
        wind[i] = (int32_t)S.rec[(int64_t)lunar::W_WIND * S.n + i];
        torque[i] = (int32_t)S.rec[(int64_t)(lunar::W_WIND + 1) * S.n + i];
    }
}

void hs_reset(void *h, float *obs) {
    Sim &S = *(Sim *)h;
    for (int64_t i = 0; i < S.n; i++) {   // box2d_reset_kernel
        if (S.lunar()) {
            float o[8];
            lunar::reset_from_record(S.rec.data(), S.n, i, S.rng.data(), S.opts, o);
            if (obs) std::memcpy(obs + 8 * i, o, sizeof o);
        } else {
            float o[24];
            if (S.hardcore()) walker::reset_from_record<true>(S.rec.data(), S.n, i, S.rng.data(), o);
            else walker::reset_from_record<false>(S.rec.data(), S.n, i, S.rng.data(), o);
            if (obs) std::memcpy(obs + 24 * i, o, sizeof o);
        }
        S.elapsed[i] = 0;
    }
}

// actions: int64 [n] (kind 5) or float32 [n][2] (kind 7) or float32 [n][4] (kinds 6, 8); returns #invalid actions
int64_t hs_step(void *h, const void *actions, float *obs_out, double *reward, uint8_t *term, uint8_t *trunc, float *final_obs) {
    Sim &S = *(Sim *)h;
    int64_t invalid = 0;
    for (int64_t i = 0; i < S.n; i++) {
        if (!S.lunar()) {
            if (S.hardcore()) walker_step_env<true>(S, i, (const float *)actions, obs_out, reward, term, trunc, final_obs);
            else walker_step_env<false>(S, i, (const float *)actions, obs_out, reward, term, trunc, final_obs);
            continue;
        }
        // box2d_step_kernel<LunarStep<ActT, CONT>>
        long long act = 0;
        float ca0 = 0.0f, ca1 = 0.0f;
        if (S.kind == 7) { ca0 = ((const float *)actions)[2 * i]; ca1 = ((const float *)actions)[2 * i + 1]; }
        else {
            act = ((const int64_t *)actions)[i];
            if (act < 0 || act > 3) { invalid++; continue; }
        }
        lunar::World W;
        lunar::load_world(W, S.rec.data(), S.n, i, S.opts.wind != 0);
        Pcg64 g = bgym::pcg64_load(&S.rng[4 * i]);
        int32_t elapsed = S.elapsed[i];
        float obs[8];
        double r;
        bool terminated;
        lunar::env_step(W, g, S.opts, (int)act, ca0, ca1, lunar::V(0.0f, 0.0f), obs, r, terminated);
        elapsed += 1;
        const bool truncated = (S.max_steps > 0) && (elapsed >= S.max_steps);
        reward[i] = r; term[i] = terminated ? 1 : 0; trunc[i] = truncated ? 1 : 0;
        if (terminated || truncated) {
            if (final_obs) std::memcpy(final_obs + 8 * i, obs, sizeof obs);
            lunar::env_reset(W, g, S.opts, obs);
            elapsed = 0;
        }
        lunar::store_world(W, S.rec.data(), S.n, i, S.opts.wind != 0);
        bgym::pcg64_store(&S.rng[4 * i], g);
        S.elapsed[i] = elapsed;
        std::memcpy(obs_out + 8 * i, obs, sizeof obs);
    }
    return invalid;
}

// the 200 terrain heights and the hardcore boxes of env i (walker kinds); returns the number of boxes
int hs_walker_terrain(void *h, int64_t i, float *terrain200, float *boxes /* [40][4] */) {
    Sim &S = *(Sim *)h;
    for (int k = 0; k < walker::kTerrain; k++) terrain200[k] = __uint_as_float(S.rec[(int64_t)(walker::W_TERRAIN + k) * S.n + i]);
    const int np = S.hardcore() ? (int)S.rec[(int64_t)walker::W_NPOLY * S.n + i] : 0;
    for (int k = 0; k < 4 * np; k++) boxes[k] = __uint_as_float(S.rec[(int64_t)(walker::W_POLY + k) * S.n + i]);
    return np;
}


// envs whose manifold table ever overflowed (b200gym_box2d_overflows on the device)
int64_t hs_overflows(void *h) {
    Sim &S = *(Sim *)h;
    const int64_t row = S.lunar() ? lunar::W_FLAGS : walker::W_FLAGS;
    int64_t c = 0;
    for (int64_t i = 0; i < S.n; i++) c += (S.rec[row * S.n + i] & b2l::kFlagOverflow) != 0;
    return c;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// classic control: Env<KIND>::step / reset of gym_b200/csrc/envs.cuh driven like advance_env / reset_env of b200gym.cu
// (autoreset mode: TimeLimit counter, same-step reset with the env's own PCG64 stream, final_obs rows)
// ---------------------------------------------------------------------------------------------------------------
namespace {

struct Classic {
    int kind = 0;
    int64_t n = 0;
    int max_steps = 0;
    double param0 = 0.0;
    std::vector<double> state;     // [S][n]
    std::vector<uint64_t> rng;     // [n][4]
    std::vector<int32_t> elapsed;
};

template <int KIND>
void classic_reset(Classic &C, const double *bounds, float *obs) {
    using E = bgym::Env<KIND>;
    double lo, hi;
    E::default_bounds(lo, hi);
    if (bounds) { lo = bounds[0]; hi = bounds[1]; }
    for (int64_t i = 0; i < C.n; i++) {
        double s[E::S];
        float o[E::D];
        Pcg64 g = bgym::pcg64_load(&C.rng[4 * i]);
        E::reset(s, g, lo, hi, o);
        bgym::pcg64_store(&C.rng[4 * i], g);
        for (int k = 0; k < E::S; k++) C.state[(int64_t)k * C.n + i] = s[k];
        C.elapsed[i] = 0;
        std::memcpy(obs + (int64_t)E::D * i, o, sizeof o);
    }
}

template <int KIND>
int64_t classic_step(Classic &C, const void *actions, float *obs_out, double *reward, uint8_t *term, uint8_t *trunc,
                     float *final_obs) {
    using E = bgym::Env<KIND>;
    int64_t invalid = 0;
    for (int64_t i = 0; i < C.n; i++) {
        double s[E::S];
        for (int k = 0; k < E::S; k++) s[k] = C.state[(int64_t)k * C.n + i];
        int32_t elapsed = C.elapsed[i];
        int act = 0;
        float a0 = 0.0f;
        if (E::A == 0) {
            const long long v = ((const int64_t *)actions)[i];
            if (v < 0 || v >= E::NACT) { invalid++; continue; }
            act = (int)v;
        } else {
            a0 = ((const float *)actions)[i];
        }
        float obs[E::D];
        double r;
        bool terminated;
        E::step(s, elapsed == 0, act, a0, C.param0, obs, r, terminated);
        elapsed += 1;
        const bool truncated = (C.max_steps > 0) && (elapsed >= C.max_steps);
        reward[i] = r; term[i] = terminated ? 1 : 0; trunc[i] = truncated ? 1 : 0;
        if (terminated || truncated) {
            if (final_obs) std::memcpy(final_obs + (int64_t)E::D * i, obs, sizeof obs);
            Pcg64 g = bgym::pcg64_load(&C.rng[4 * i]);
            double lo, hi;
            E::default_bounds(lo, hi);
            E::reset(s, g, lo, hi, obs);
            bgym::pcg64_store(&C.rng[4 * i], g);
            elapsed = 0;
        }
        for (int k = 0; k < E::S; k++) C.state[(int64_t)k * C.n + i] = s[k];
        C.elapsed[i] = elapsed;
        std::memcpy(obs_out + (int64_t)E::D * i, obs, sizeof obs);
    }
    return invalid;
}

}  // namespace

extern "C" {

void *hs_classic_create(int kind, int64_t n, int max_steps, double param0) {
    if (n <= 0 || kind < 0 || kind > 4) return nullptr;
    Classic *C = new Classic();
    C->kind = kind; C->n = n; C->max_steps = max_steps; C->param0 = param0;
    C->state.assign(4 * (size_t)n, 0.0);
    C->rng.assign(4 * (size_t)n, 0ull);
    C->elapsed.assign((size_t)n, 0);
    return C;
}
void hs_classic_destroy(void *h) { delete (Classic *)h; }

void hs_classic_seed_range(void *h, const uint32_t base[4], int64_t first) {
    Classic &C = *(Classic *)h;
    using bgym::u128;
    const u128 b = ((u128)base[3] << 96) | ((u128)base[2] << 64) | ((u128)base[1] << 32) | (u128)base[0];
    for (int64_t i = 0; i < C.n; i++) {
        const u128 seed = b + (u128)(uint64_t)(first + i);
        const uint32_t ent[4] = {(uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)(seed >> 64), (uint32_t)(seed >> 96)};
        Pcg64 g;
        bgym::pcg64_from_entropy(g, ent);
        bgym::pcg64_store_full(&C.rng[4 * i], g);
    }
}

void hs_classic_reset(void *h, const double *bounds, float *obs) {
    Classic &C = *(Classic *)h;
    switch (C.kind) {
    case 0: classic_reset<B200GYM_CARTPOLE>(C, bounds, obs); break;
    case 1: classic_reset<B200GYM_MOUNTAINCAR>(C, bounds, obs); break;
    case 2: classic_reset<B200GYM_MOUNTAINCAR_CONT>(C, bounds, obs); break;
    case 3: classic_reset<B200GYM_PENDULUM>(C, bounds, obs); break;
    default: classic_reset<B200GYM_ACROBOT>(C, bounds, obs); break;
    }
}

int64_t hs_classic_step(void *h, const void *actions, float *obs, double *reward, uint8_t *term, uint8_t *trunc,
                        float *final_obs) {
    Classic &C = *(Classic *)h;
    switch (C.kind) {
    case 0: return classic_step<B200GYM_CARTPOLE>(C, actions, obs, reward, term, trunc, final_obs);
    case 1: return classic_step<B200GYM_MOUNTAINCAR>(C, actions, obs, reward, term, trunc, final_obs);
    case 2: return classic_step<B200GYM_MOUNTAINCAR_CONT>(C, actions, obs, reward, term, trunc, final_obs);
    case 3: return classic_step<B200GYM_PENDULUM>(C, actions, obs, reward, term, trunc, final_obs);
    default: return classic_step<B200GYM_ACROBOT>(C, actions, obs, reward, term, trunc, final_obs);
    }
}

void hs_classic_get_state(void *h, double *state_aos /* [n][S] */, int S) {
    Classic &C = *(Classic *)h;
    for (int64_t i = 0; i < C.n; i++)
        for (int k = 0; k < S; k++) state_aos[i * S + k] = C.state[(int64_t)k * C.n + i];
}

// CartPole's small-angle sin/cos kernel alone (csrc/envs.cuh: sincos_small)
void hs_sincos_small(const double *x, int64_t n, double *sn, double *cs) {
    for (int64_t i = 0; i < n; i++) bgym::sincos_small(x[i], sn[i], cs[i]);
}


// glibc_trig.cuh: the restated glibc sin / cos, evaluated by the host build of the device header
void hs_glibc_trig(const double *x, int64_t n, double *sn, double *cs) {
    for (int64_t i = 0; i < n; i++) { sn[i] = bgym::gt::sin(x[i]); cs[i] = bgym::gt::cos(x[i]); }
}
// arguments in [lo, hi) (splitmix64 stream) where gt::sq(x) differs bitwise from libm pow(x, 2.0); *neq_out counts
// those where pow(x, 2.0) itself differs from x * x (why the restatement exists)
int64_t hs_glibc_sq_mismatches(uint64_t seed, int64_t n, double lo, double hi, int64_t *neq_out) {
    int64_t bad = 0, neq = 0;
    uint64_t st = seed;
    volatile double two = 2.0;   // keep the compiler from folding pow(x, 2.0) into x * x
    for (int64_t i = 0; i < n; i++) {
        uint64_t z = (st += 0x9E3779B97F4A7C15ULL);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
        z ^= z >> 31;
        const double x = lo + (hi - lo) * ((double)(z >> 11) * (1.0 / 9007199254740992.0));
        const double a = std::pow(x, two), b = bgym::gt::sq(x), c = x * x;
        bad += std::memcmp(&a, &b, 8) != 0;
        neq += std::memcmp(&a, &c, 8) != 0;
    }
    if (neq_out) *neq_out = neq;
    return bad;
}

// number of arguments in [lo, hi) (splitmix64 stream) where sin or cos differs bitwise from this process's libm
int64_t hs_glibc_trig_mismatches(uint64_t seed, int64_t n, double lo, double hi) {
    int64_t bad = 0;
    uint64_t st = seed;
    for (int64_t i = 0; i < n; i++) {
        uint64_t z = (st += 0x9E3779B97F4A7C15ULL);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
        z ^= z >> 31;
        const double x = lo + (hi - lo) * ((double)(z >> 11) * (1.0 / 9007199254740992.0));
        const double a = std::sin(x), b = bgym::gt::sin(x), c = std::cos(x), d = bgym::gt::cos(x);
        bad += (std::memcmp(&a, &b, 8) != 0) + (std::memcmp(&c, &d, 8) != 0);
    }
    return bad;
}


// The device's b2TimeOfImpact and the conservative shortcut in front of it (b2lite_toi.cuh), for one sweep of a
// task polygon (shape 0 = lander, 1 = lander leg, 2 = walker hull, 3 = walker upper leg, 4 = walker lower leg)
// against the static edge v1-v2 or, with `box` set, the axis-aligned box {x0, ylo, x1, yhi}.
// Returns the b2TOIOutput state (3 = touching), *t_out, and *cannot_touch = what toi_cannot_touch says.
int hs_toi_probe(int shape, const float *c0, float a0, const float *c1, float a1, const float *v1, const float *v2,
                 const float *box, float *t_out, int *cannot_touch) {
    ensure_consts();
    const b2l::ShapeConst &sh = shape < 2 ? lunar::kC.shape[shape] : walker::kC.shape[shape - 2];
    b2l::DProxy pA, pB;
    if (box) {
        pA.count = 4;
        pA.v[0] = b2l::V(box[2], box[1]); pA.v[1] = b2l::V(box[2], box[3]); pA.v[2] = b2l::V(box[0], box[3]); pA.v[3] = b2l::V(box[0], box[1]);
    } else {
        pA.count = 2;
        pA.v[0] = b2l::V(v1[0], v1[1]); pA.v[1] = b2l::V(v2[0], v2[1]);
    }
    pB.count = sh.count;
    for (int i = 0; i < sh.count; i++) pB.v[i] = sh.verts[i];
    b2l::Sweep sA, sB;
    sA.localCenter = b2l::V(0.0f, 0.0f); sA.c0 = b2l::V(0.0f, 0.0f); sA.c = b2l::V(0.0f, 0.0f); sA.a0 = 0.0f; sA.a = 0.0f; sA.alpha0 = 0.0f;
    sB.localCenter = sh.localCenter; sB.c0 = b2l::V(c0[0], c0[1]); sB.c = b2l::V(c1[0], c1[1]); sB.a0 = a0; sB.a = a1; sB.alpha0 = 0.0f;
    b2l::xform xf1;
    xf1.q = b2l::rot_of(a1);
    xf1.p = b2l::sub(sB.c, b2l::rmul(xf1.q, sh.localCenter));
    *cannot_touch = b2l::toi_cannot_touch(sh, xf1, sB, pA) ? 1 : 0;
    return b2l::time_of_impact(*t_out, pA, sA, pB, sB, 1.0f);
}

// The task polygon `shape` as the device constants hold it: vertices (x, y pairs) into out, local centre into lc;
// returns the vertex count.
int hs_shape_verts(int shape, float *out, float *lc) {
    ensure_consts();
    const b2l::ShapeConst &sh = shape < 2 ? lunar::kC.shape[shape] : walker::kC.shape[shape - 2];
    for (int i = 0; i < sh.count; i++) { out[2 * i] = sh.verts[i].x; out[2 * i + 1] = sh.verts[i].y; }
    lc[0] = sh.localCenter.x; lc[1] = sh.localCenter.y;
    return sh.count;
}

}  // extern "C"
