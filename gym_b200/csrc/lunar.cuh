// lunar.cuh -- LunarLander-v2 / LunarLanderContinuous-v2 on the device (scene + environment logic on top of
// b2lite.cuh), with the constructor variants of the reference: continuous actions, gravity, wind.
//
// Reference: gym/envs/box2d/lunar_lander.py (reset :308-420, step :444-600, ContactDetector
// :54-72).  Scene: lander (6-gon, density 5) + two legs (boxes, density 1) tied by two revolute
// joints (limits + motor, maxMotorTorque 40), eleven static edges (base + 10 terrain chunks).
// Cosmetic particles are not simulated: they collide only with the ground (categoryBits 0x0100
// vs the lander/leg maskBits 0x001) and draw no random numbers.
#pragma once
#include <cstdint>

#include "b2lite.cuh"
#include "glibc_trig.cuh"
#include "rng.cuh"

namespace lunar {

using namespace b2l;
using bgym::Pcg64;
namespace gt = bgym::gt;   // math.sin / math.cos as glibc evaluates them

#define LD __device__ __forceinline__

constexpr int NB = 3;    // dynamic bodies: 0 lander, 1 leg (i=-1), 2 leg (i=+1)
constexpr int NJ = 2;
constexpr int NE = 11;   // ground edges: 0 base, 1..10 terrain
#ifndef B2L_LUNAR_MAX_VC
#define B2L_LUNAR_MAX_VC 8   // manifold-table capacity (touching pairs per env; tests build a smaller one)
#endif
constexpr int kSlots = 8;

struct Consts {
    ShapeConst shape[2];  // 0 lander, 1 leg
    JointDef jd[NJ];      // lander -> leg (i=-1), lander -> leg (i=+1)
    float motorSpeed[NJ];
    float chunk_x[NE];    // terrain vertex abscissae (float32 of W/(CHUNKS-1)*i)
    float world_w;        // W as float32
    float lander_x0, leg_x0[2], y0, leg_a0[2];
};
__constant__ Consts kC;

// ---- HBM record: kWords 32-bit words per env, SoA ([word][n]) ----------------------------------
constexpr int W_BODY = 0;     // 3 x {cx, cy, a, vx, vy, w, sleepTime}
constexpr int W_JOINT = 21;   // 2 x {impulse x, y, z, motorImpulse, limitState}
constexpr int W_TERRAIN = 31; // smooth_y[11]
constexpr int W_FLAGS = 42;   // bit0 game_over, bit1/2 leg contact, bit3 has_prev_shaping, bit4 world has stepped
constexpr int W_SHAPING = 43; // prev_shaping (double, 2 words)
constexpr int W_SLOT = 45;    // kSlots x {key, id0, nI0, tI0, id1, nI1, tI1}
constexpr int W_WIND = W_SLOT + 7 * kSlots;  // wind_idx, torque_idx (int32; touched only when wind is enabled)
constexpr int kWords = W_WIND + 2;           // 103

// constructor arguments of LunarLander (lunar_lander.py:194-199), uniform over the batch
struct Opts {
    float gravity;           // b2World(gravity=(0, gravity)), :240
    uint32_t continuous;     // :247
    uint32_t wind;           // enable_wind, :233
    double wind_power, turbulence_power;
};

struct World : WorldBase<NB, NJ, kSlots> {
    float terrain[NE];
    double prev_shaping;
    int32_t wind_idx, torque_idx;   // :234-235, drawn once per env object, never reset
};

struct Scene {
    static constexpr int NB = lunar::NB, NJ = lunar::NJ, NE = lunar::NE, kSlots = lunar::kSlots, kMaxVC = B2L_LUNAR_MAX_VC;
    static constexpr int NP = 0;   // no static polygons in this scene
    static constexpr bool kOneStaticBody = true;   // every edge is a fixture of the one static body `moon`
    using World = lunar::World;
    LD static const ShapeConst &shape(int b) { return kC.shape[b == 0 ? 0 : 1]; }
    LD static const JointDef &jdef(int k) { return kC.jd[k]; }
    // b2World::Solve's depth-first island walk starts at the newest body: leg(+1), lander, leg(-1)
    __host__ __device__ static constexpr int body_order(int k) { return k == 0 ? 2 : (k == 1 ? 0 : 1); }
    __host__ __device__ static constexpr int joint_order(int k) { return 1 - k; }
    // joint k ties the lander (body 0) to leg k (body k + 1); the runtime JointDef holds the same indices
    __host__ __device__ static constexpr int joint_body_a(int) { return 0; }
    __host__ __device__ static constexpr int joint_body_b(int k) { return k + 1; }
    LD static void edge(const World &W, int e, v2 &v1, v2 &v2_, float &friction) {
        if (e == 0) { v1 = V(0.0f, 0.0f); v2_ = V(kC.world_w, 0.0f); friction = 0.2f; }
        else { v1 = V(kC.chunk_x[e - 1], W.terrain[e - 1]); v2_ = V(kC.chunk_x[e], W.terrain[e]); friction = 0.1f; }
    }
    LD static void edge_range(const World &, float, float, int &lo, int &hi) { lo = 0; hi = NE - 1; }
    // ContactDetector (lunar_lander.py:59-72)
    LD static void on_event(World &W, int b, bool begin) {
        if (begin) { if (b == 0) W.flags |= 1u; else W.flags |= (2u << (b - 1)); }
        else if (b > 0) W.flags &= ~(2u << (b - 1));
    }
};

// ---- the environment ---------------------------------------------------------------------------
// lunar_lander.py:444-600.  `action` is the Discrete(4) action, `ca` the Box(2) float32 action of the
// continuous variant.  In the continuous branch m_power / s_power / direction are numpy float32 scalars:
// under NEP 50 every Python float they meet is rounded to float32 first, which is what the casts restate.
// what env_pre hands to env_post across world.Step (and, for envs whose continuous-collision phase is deferred to
// the TOI kernel, across kernels: b200gym.cu keeps it in a side buffer)
struct Mid { double main_cost, side_cost; bool awake; };

// lunar_lander.py:444-556: wind, engines, world.Step.  run_toi = false leaves b2World::SolveTOI to the caller.
LD void env_pre(World &W, Pcg64 &rng, const Opts &O, int action, float ca0, float ca1, v2 lander_force, Mid &mid,
                unsigned live, bool run_toi) {
    const double SCALE = 30.0;
    Body &L = W.b[0];
    const ShapeConst &sh = kC.shape[0];
    float torque = 0.0f;
    if (O.wind && !(W.flags & 6u)) {                                             // :449-477
        const double kPi = 3.141592653589793;
        const double wind_mag = tanh(gt::sin(0.02 * W.wind_idx) + gt::sin(kPi * 0.01 * W.wind_idx)) * O.wind_power;
        W.wind_idx += 1;
        lander_force = add(lander_force, V((float)wind_mag, 0.0f));              // ApplyForceToCenter
        const double torque_mag = tanh(gt::sin(0.02 * W.torque_idx) + gt::sin(kPi * 0.01 * W.torque_idx)) * O.turbulence_power;
        W.torque_idx += 1;
        torque += (float)torque_mag;                                             // ApplyTorque
    }
    const double ang = (double)L.a;
    const double tip0 = gt::sin(ang), tip1 = gt::cos(ang);                       // :487 math.sin / math.cos
    const double side0 = -tip1, side1 = tip0;
    const double disp0 = bgym::pcg64_uniform(rng, -1.0, +1.0) / SCALE;          // :489
    const double disp1 = bgym::pcg64_uniform(rng, -1.0, +1.0) / SCALE;
    float a0 = 0.0f, a1 = 0.0f;
    if (O.continuous) {                                                          // :480
        a0 = ca0 < -1.0f ? -1.0f : (ca0 > 1.0f ? 1.0f : ca0);
        a1 = ca1 < -1.0f ? -1.0f : (ca1 > 1.0f ? 1.0f : ca1);
    }
    double main_cost = 0.0, side_cost = 0.0;
    if (O.continuous ? (a0 > 0.0f) : (action == 2)) {                           // :491-520
        const double ox = tip0 * (4 / SCALE + 2 * disp0) + side0 * disp1;
        const double oy = -tip1 * (4 / SCALE + 2 * disp0) - side1 * disp1;
        const v2 pt = V((float)((double)L.xf.p.x + ox), (float)((double)L.xf.p.y + oy));
        v2 imp;
        if (O.continuous) {
            const float c = a0 < 0.0f ? 0.0f : (a0 > 1.0f ? 1.0f : a0);
            const float m_power = (c + 1.0f) * 0.5f;                             // :497
            imp = V((float)(-ox * 13.0) * m_power, (float)(-oy * 13.0) * m_power);
            main_cost = (double)(m_power * 0.30f);
        } else {
            imp = V((float)(-ox * 13.0 * 1.0), (float)(-oy * 13.0 * 1.0));
            main_cost = 1.0 * 0.30;
        }
        L.v = add(L.v, scl(sh.invMass, imp));                                   // b2Body::ApplyLinearImpulse
        L.w += sh.invI * crs(sub(pt, L.c), imp);
    }
    if (O.continuous ? (fabsf(a1) > 0.5f) : (action == 1 || action == 3)) {      // :522-554
        v2 imp, pt;
        if (O.continuous) {
            const float direction = a1 > 0.0f ? 1.0f : -1.0f;                    // np.sign with |a1| > 0.5
            const float ab = fabsf(a1);
            const float s_power = ab < 0.5f ? 0.5f : (ab > 1.0f ? 1.0f : ab);
            const float t = direction * 12.0f / 30.0f;
            const float u = (float)(3 * disp1) + t;
            const float ox = (float)(tip0 * disp0) + (float)side0 * u;
            const float oy = (float)(-tip1 * disp0) - (float)side1 * u;
            pt = V((L.xf.p.x + ox) - (float)(tip0 * 17 / SCALE), (L.xf.p.y + oy) + (float)(tip1 * 14.0 / SCALE));
            imp = V((-ox * 0.6f) * s_power, (-oy * 0.6f) * s_power);
            side_cost = (double)(s_power * 0.03f);
        } else {
            const double direction = action - 2;
            const double ox = tip0 * disp0 + side0 * (3 * disp1 + direction * 12.0 / SCALE);
            const double oy = -tip1 * disp0 - side1 * (3 * disp1 + direction * 12.0 / SCALE);
            pt = V((float)((double)L.xf.p.x + ox - tip0 * 17 / SCALE), (float)((double)L.xf.p.y + oy + tip1 * 14.0 / SCALE));
            imp = V((float)(-ox * 0.6 * 1.0), (float)(-oy * 0.6 * 1.0));
            side_cost = 1.0 * 0.03;
        }
        L.v = add(L.v, scl(sh.invMass, imp));
        L.w += sh.invI * crs(sub(pt, L.c), imp);
    }
    bool awake;
    world_step<Scene>(W, lander_force, torque, O.gravity, awake, live, run_toi);                           // :556
    mid.main_cost = main_cost; mid.side_cost = side_cost; mid.awake = awake;
}

// lunar_lander.py:558-600: observation, shaping reward, termination
LD void env_post(World &W, const Mid &mid, float (&obs)[8], double &reward, bool &terminated) {
    const double SCALE = 30.0, FPS = 50;
    const double VW = 600 / SCALE, VH = 400 / SCALE;
    const Body &L = W.b[0];
    const double main_cost = mid.main_cost, side_cost = mid.side_cost;
    const bool awake = mid.awake;
    double st[8];
    const double helipad_y = VH / 4;
    st[0] = ((double)L.xf.p.x - VW / 2) / (VW / 2);                              // :560-569
    st[1] = ((double)L.xf.p.y - (helipad_y + 18 / SCALE)) / (VH / 2);
    st[2] = (double)L.v.x * (VW / 2) / FPS;
    st[3] = (double)L.v.y * (VH / 2) / FPS;
    st[4] = (double)L.a;
    st[5] = 20.0 * (double)L.w / FPS;
    st[6] = (W.flags & 2u) ? 1.0 : 0.0;
    st[7] = (W.flags & 4u) ? 1.0 : 0.0;
    double r = 0;
    const double shaping = -100 * sqrt(st[0] * st[0] + st[1] * st[1]) - 100 * sqrt(st[2] * st[2] + st[3] * st[3])
                           - 100 * fabs(st[4]) + 10 * st[6] + 10 * st[7];        // :572-578
    if (W.flags & 8u) r = shaping - W.prev_shaping;                              // :581-583
    W.prev_shaping = shaping;
    W.flags |= 8u;
    r -= main_cost;                                                              // :585-588
    r -= side_cost;
    bool term = false;
    if ((W.flags & 1u) || fabs(st[0]) >= 1.0) { term = true; r = -100; }         // :590-593
    if (!awake) { term = true; r = +100; }                                       // :594-596
#pragma unroll
    for (int k = 0; k < 8; k++) obs[k] = (float)st[k];                           // :600
    reward = r;
    terminated = term;
}

LD void env_step(World &W, Pcg64 &rng, const Opts &O, int action, float ca0, float ca1, v2 lander_force,
                 float (&obs)[8], double &reward, bool &terminated, unsigned live = 0u) {
    Mid mid;
    env_pre(W, rng, O, action, ca0, ca1, lander_force, mid, live, true);
    env_post(W, mid, obs, reward, terminated);
}

// lunar_lander.py:308-420 (the b2World object survives reset(): bit4 of flags is kept)
LD void env_reset(World &W, Pcg64 &rng, const Opts &O, float (&obs)[8]) {
    const double SCALE = 30.0;
    const double Wd = 600 / SCALE, Hd = 400 / SCALE;
    const uint32_t stepped = W.flags & kFlagsKept;
    double height[12];
    for (int i = 0; i < 12; i++) height[i] = bgym::pcg64_uniform(rng, 0, Hd / 2);   // :326
    const double helipad_y = Hd / 4;
    for (int k = -2; k <= 2; k++) height[11 / 2 + k] = helipad_y;                // :331-335
    for (int i = 0; i < NE; i++)                                                 // :336-339
        W.terrain[i] = (float)(0.33 * (height[(i + 11) % 12] + height[i] + height[i + 1]));
    (void)Wd;
    for (int b = 0; b < NB; b++) {
        Body &B = W.b[b];
        const ShapeConst &sh = Scene::shape(b);
        const v2 pos = b == 0 ? V(kC.lander_x0, kC.y0) : V(kC.leg_x0[b - 1], kC.y0);
        const float angle = b == 0 ? 0.0f : kC.leg_a0[b - 1];
        B.xf.p = pos;
        B.xf.q = rot_of(angle);
        B.c = xmul(B.xf, sh.localCenter);
        B.a = angle;
        B.v = V(0.0f, 0.0f);
        B.w = 0.0f;
        B.sleepTime = 0.0f;
    }
    for (int j = 0; j < NJ; j++) {
        W.j[j].imp[0] = W.j[j].imp[1] = W.j[j].imp[2] = 0.0f; W.j[j].motorImpulse = 0.0f; W.j[j].limitState = 0;
        W.j[j].motorSpeed = kC.motorSpeed[j]; W.j[j].maxMotorTorque = 40.0f;   // LEG_SPRING_TORQUE
    }
    W.flags = stepped;
    W.prev_shaping = 0.0;
    for (int s = 0; s < kSlots; s++) W.slot_key[s] = 0u;
    const double fx = bgym::pcg64_uniform(rng, -1000.0, 1000.0);                 // :371-377
    const double fy = bgym::pcg64_uniform(rng, -1000.0, 1000.0);
    double r;
    bool t;
    env_step(W, rng, O, 0, 0.0f, 0.0f, V((float)fx, (float)fy), obs, r, t);      // :420
}

// ---- HBM <-> registers/local ---------------------------------------------------------------------
LD void load_world(World &W, const uint32_t *rec, int64_t n, int64_t i, bool wind) {
    auto ld = [&](int k) { return rec[(int64_t)k * n + i]; };
    for (int b = 0; b < NB; b++) {
        Body &B = W.b[b];
        B.c.x = __uint_as_float(ld(W_BODY + 7 * b + 0)); B.c.y = __uint_as_float(ld(W_BODY + 7 * b + 1));
        B.a = __uint_as_float(ld(W_BODY + 7 * b + 2));
        B.v.x = __uint_as_float(ld(W_BODY + 7 * b + 3)); B.v.y = __uint_as_float(ld(W_BODY + 7 * b + 4));
        B.w = __uint_as_float(ld(W_BODY + 7 * b + 5)); B.sleepTime = __uint_as_float(ld(W_BODY + 7 * b + 6));
        sync_xf(B, Scene::shape(b));
    }
    for (int j = 0; j < 2; j++) {
        for (int k = 0; k < 3; k++) W.j[j].imp[k] = __uint_as_float(ld(W_JOINT + 5 * j + k));
        W.j[j].motorImpulse = __uint_as_float(ld(W_JOINT + 5 * j + 3));
        W.j[j].limitState = (int)ld(W_JOINT + 5 * j + 4);
        W.j[j].motorSpeed = kC.motorSpeed[j];
        W.j[j].maxMotorTorque = 40.0f;   // LEG_SPRING_TORQUE
    }
    for (int e = 0; e < NE; e++) W.terrain[e] = __uint_as_float(ld(W_TERRAIN + e));
    W.flags = ld(W_FLAGS);
    W.wind_idx = wind ? (int32_t)ld(W_WIND) : 0;
    W.torque_idx = wind ? (int32_t)ld(W_WIND + 1) : 0;
    W.prev_shaping = __longlong_as_double((long long)(((unsigned long long)ld(W_SHAPING + 1) << 32) | ld(W_SHAPING)));
    for (int s = 0; s < kSlots; s++) {
        W.slot_key[s] = ld(W_SLOT + 7 * s);
        for (int p = 0; p < 2; p++) {
            W.slot_id[s][p] = ld(W_SLOT + 7 * s + 1 + 3 * p);
            W.slot_nI[s][p] = __uint_as_float(ld(W_SLOT + 7 * s + 2 + 3 * p));
            W.slot_tI[s][p] = __uint_as_float(ld(W_SLOT + 7 * s + 3 + 3 * p));
        }
    }
}

LD void store_world(const World &W, uint32_t *rec, int64_t n, int64_t i, bool wind) {
    auto st = [&](int k, uint32_t v) { rec[(int64_t)k * n + i] = v; };
    for (int b = 0; b < NB; b++) {
        const Body &B = W.b[b];
        st(W_BODY + 7 * b + 0, __float_as_uint(B.c.x)); st(W_BODY + 7 * b + 1, __float_as_uint(B.c.y));
        st(W_BODY + 7 * b + 2, __float_as_uint(B.a));
        st(W_BODY + 7 * b + 3, __float_as_uint(B.v.x)); st(W_BODY + 7 * b + 4, __float_as_uint(B.v.y));
        st(W_BODY + 7 * b + 5, __float_as_uint(B.w)); st(W_BODY + 7 * b + 6, __float_as_uint(B.sleepTime));
    }
    for (int j = 0; j < 2; j++) {
        for (int k = 0; k < 3; k++) st(W_JOINT + 5 * j + k, __float_as_uint(W.j[j].imp[k]));
        st(W_JOINT + 5 * j + 3, __float_as_uint(W.j[j].motorImpulse));
        st(W_JOINT + 5 * j + 4, (uint32_t)W.j[j].limitState);
    }
    for (int e = 0; e < NE; e++) st(W_TERRAIN + e, __float_as_uint(W.terrain[e]));
    st(W_FLAGS, W.flags);
    if (wind) { st(W_WIND, (uint32_t)W.wind_idx); st(W_WIND + 1, (uint32_t)W.torque_idx); }
    const unsigned long long ps = (unsigned long long)__double_as_longlong(W.prev_shaping);
    st(W_SHAPING, (uint32_t)ps); st(W_SHAPING + 1, (uint32_t)(ps >> 32));
    for (int s = 0; s < kSlots; s++) {
        st(W_SLOT + 7 * s, W.slot_key[s]);
        for (int p = 0; p < 2; p++) {
            st(W_SLOT + 7 * s + 1 + 3 * p, W.slot_id[s][p]);
            st(W_SLOT + 7 * s + 2 + 3 * p, __float_as_uint(W.slot_nI[s][p]));
            st(W_SLOT + 7 * s + 3 + 3 * p, __float_as_uint(W.slot_tI[s][p]));
        }
    }
}

// reset() of env i in the SoA record `rec` and the [n][4] PCG64 records `rng`.  The b2World object survives reset():
// so do the kept flag bits and wind_idx / torque_idx.  `n` is taken by reference: a kernel that passes a field of its
// parameter block then reads it where the record is addressed, and the compiler keeps one multiply per record row out
// of the reset-list kernel's loop instead of re-deriving rows from each other and spilling (8 / 24 / 44 bytes)
LD void reset_from_record(uint32_t *rec, const int64_t &n, int64_t i, uint64_t *rng, const Opts &O, float (&obs)[8]) {
    World W;
    W.flags = rec[(int64_t)W_FLAGS * n + i] & kFlagsKept;
    W.wind_idx = O.wind ? (int32_t)rec[(int64_t)W_WIND * n + i] : 0;
    W.torque_idx = O.wind ? (int32_t)rec[(int64_t)(W_WIND + 1) * n + i] : 0;
    Pcg64 g = bgym::pcg64_load(rng + 4 * i);
    env_reset(W, g, O, obs);
    store_world(W, rec, n, i, O.wind != 0);
    bgym::pcg64_store(rng + 4 * i, g);
}

#undef LD
}  // namespace lunar
