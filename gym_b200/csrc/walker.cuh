// walker.cuh -- BipedalWalker-v3 / BipedalWalkerHardcore-v3 on the device (scene + environment logic on top of
// b2lite.cuh).
//
// Reference: gym/envs/box2d/bipedal_walker.py (reset :425-515, _generate_terrain :277-402,
// _generate_clouds :404-423, step :517-606, ContactDetector :80-98, LidarCallback :504-510).
// Scene: hull (5-gon, density 5) + two upper and two lower leg boxes (density 1), four revolute
// joints (hips, knees; limits + motors whose speed/torque the action sets every step), 199
// static terrain edges (friction 2.5), 10 lidar rays; hardcore=True (template parameter HC) adds up to 39 static
// boxes -- stumps, stair steps, pit walls (:300-373) -- that collide (b2CollidePolygons) and stop the lidar.
#pragma once
#include <cstdint>

#include "b2lite.cuh"
#include "rng.cuh"

namespace walker {

using namespace b2l;
using bgym::Pcg64;

#define LD __device__ __forceinline__

constexpr int NB = 5;     // 0 hull, 1 leg(-1), 2 lower(-1), 3 leg(+1), 4 lower(+1)
constexpr int NJ = 4;     // 0 hip(-1), 1 knee(-1), 2 hip(+1), 3 knee(+1)   (self.joints order)
constexpr int NE = 199;   // terrain edges i -> i+1
#ifndef B2L_WALKER_MAX_VC
#define B2L_WALKER_MAX_VC 10   // manifold-table capacity (touching pairs per env; tests build a smaller one)
#endif
constexpr int kSlots = 10;
constexpr int kTerrain = 200;

struct Consts {
    ShapeConst shape[3];  // 0 hull, 1 upper leg, 2 lower leg
    JointDef jd[NJ];
    float init_x, init_y, leg_y, lower_y, leg_a0[2];
};
__constant__ Consts kC;

// ---- HBM record: kWords 32-bit words per env, SoA ([word][n]) ----------------------------------
constexpr int W_BODY = 0;       // 5 x {cx, cy, a, vx, vy, w, sleepTime}
constexpr int W_JOINT = 35;     // 4 x {impulse x, y, z, motorImpulse, limitState}
constexpr int W_FLAGS = 55;     // bit0 game_over, bit1 legs[1] contact, bit2 legs[3] contact, bit3 has_prev_shaping, bit4 stepped
constexpr int W_SHAPING = 56;   // prev_shaping (double, 2 words)
constexpr int W_RNG32 = 58;     // numpy's buffered next_uint32: {has_uint32, uinteger}
constexpr int W_SLOT = 60;      // kSlots x {key, id0, nI0, tI0, id1, nI1, tI1}
constexpr int W_TERRAIN = W_SLOT + 7 * kSlots;  // terrain_y[200] (read on demand, written by reset)
constexpr int kWords = W_TERRAIN + kTerrain;    // 330
// hardcore only: the obstacle boxes, in creation (ascending x) order
constexpr int NP = 40;                          // at most 39 can be generated on 200 segments (DESIGN.md)
constexpr int W_NPOLY = kWords;                 // number of boxes
constexpr int W_POLY = W_NPOLY + 1;             // NP x {x0, ylo, x1, yhi}
constexpr int kWordsHC = W_POLY + 4 * NP;       // 491

struct World : WorldBase<NB, NJ, kSlots> {
    double prev_shaping;
    uint32_t *terrain;        // &rec[W_TERRAIN * n + i]; element k lives at terrain[k * n]
    int64_t n;
    int np, p_lo, p_hi;       // hardcore: boxes in use; the window of boxes near the walker this step
};

LD float terrain_x(int k) { return (float)((double)k * (14 / 30.0)); }          // i * TERRAIN_STEP
// plain (coherent) load: an autoreset in the same kernel rewrites the terrain this thread then reads
LD float terrain_y(const World &W, int k) { return __uint_as_float(W.terrain[(int64_t)k * W.n]); }
LD float poly_word(const World &W, int p, int k) {
    return __uint_as_float(W.terrain[(int64_t)(W_POLY - W_TERRAIN + 4 * p + k) * W.n]);
}
// boxes whose x-extent meets [lo_x, hi_x]: they are sorted by x and disjoint in x
LD void poly_window(const World &W, float lo_x, float hi_x, int &lo, int &hi) {
    lo = 0; hi = -1;
    bool any = false;
    for (int p = 0; p < W.np; p++) {
        const float x0 = poly_word(W, p, 0), x1 = poly_word(W, p, 2);
        if (x1 >= lo_x && x0 <= hi_x) { if (!any) { lo = p; any = true; } hi = p; }
    }
}

template <bool HC>
struct SceneT {
    static constexpr int NB = walker::NB, NJ = walker::NJ, NE = walker::NE, kSlots = walker::kSlots, kMaxVC = B2L_WALKER_MAX_VC;
    static constexpr int NP = HC ? walker::NP : 0;
    static constexpr bool kOneStaticBody = false;  // one static body per terrain edge / box (bipedal_walker.py:375-396)
    using World = walker::World;
    // fd_polygon: friction 2.5 (bipedal_walker.py:180-184)
    LD static void poly(const World &W, int p, float &x0, float &ylo, float &x1, float &yhi, float &friction) {
        x0 = poly_word(W, p, 0); ylo = poly_word(W, p, 1); x1 = poly_word(W, p, 2); yhi = poly_word(W, p, 3);
        friction = 2.5f;
    }
    // the window computed once per step around the whole walker (every body lies inside it)
    LD static void poly_range(const World &W, float, float, int &lo, int &hi) { lo = W.p_lo; hi = W.p_hi; }
    LD static const ShapeConst &shape(int b) { return kC.shape[b == 0 ? 0 : ((b & 1) ? 1 : 2)]; }
    LD static const JointDef &jdef(int k) { return kC.jd[k]; }
    // b2World::Solve's depth-first island walk from the newest body: lower(+1), leg(+1), hull, leg(-1), lower(-1);
    // joints in discovery order: knee(+1), hip(+1), hip(-1), knee(-1)
    __host__ __device__ static constexpr int body_order(int k) { return k == 0 ? 4 : (k == 1 ? 3 : (k == 2 ? 0 : (k == 3 ? 1 : 2))); }
    __host__ __device__ static constexpr int joint_order(int k) { return k == 0 ? 3 : (k == 1 ? 2 : (k == 2 ? 0 : 1)); }
    // hips (0, 2) tie the hull to the upper legs (1, 3); knees (1, 3) tie the upper to the lower legs (2, 4)
    __host__ __device__ static constexpr int joint_body_a(int k) { return k == 0 ? 0 : (k == 1 ? 1 : (k == 2 ? 0 : 3)); }
    __host__ __device__ static constexpr int joint_body_b(int k) { return k + 1; }
    LD static void edge(const World &W, int e, v2 &v1, v2 &v2_, float &friction) {
        v1 = V(terrain_x(e), terrain_y(W, e));
        v2_ = V(terrain_x(e + 1), terrain_y(W, e + 1));
        friction = 2.5f;
    }
    // every edge whose fat AABB can overlap [lo_x, hi_x] (both already widened once), plus one on each side
    LD static void edge_range(const World &, float lo_x, float hi_x, int &lo, int &hi) {
        const float step = (float)(14 / 30.0);
        lo = (int)floorf((lo_x - 0.2f) / step) - 1;
        hi = (int)floorf((hi_x + 0.2f) / step) + 1;
        lo = lo < 0 ? 0 : lo;
        hi = hi > NE - 1 ? NE - 1 : hi;
    }
    // ContactDetector (bipedal_walker.py:85-98)
    LD static void on_event(World &W, int b, bool begin) {
        if (begin) {
            if (b == 0) W.flags |= 1u;
            if (b == 2) W.flags |= 2u;
            if (b == 4) W.flags |= 4u;
        } else {
            if (b == 2) W.flags &= ~2u;
            if (b == 4) W.flags &= ~4u;
        }
    }
};
using Scene = SceneT<false>;

// numpy Generator with the 32-bit cache that Generator.integers() uses
struct Rng { Pcg64 g; uint32_t has32, val32; };
LD uint32_t next32(Rng &r) {  // pcg64_next32
    if (r.has32) { r.has32 = 0; return r.val32; }
    const uint64_t next = bgym::pcg64_next64(r.g);
    r.has32 = 1;
    r.val32 = (uint32_t)(next >> 32);
    return (uint32_t)(next & 0xffffffffu);
}
LD long long integers(Rng &r, long long low, long long high) {  // Lemire, ranges below 2^32
    const uint32_t rng = (uint32_t)(high - low - 1);
    if (rng == 0) return low;
    const uint32_t rng_excl = rng + 1u;
    unsigned long long m = (unsigned long long)next32(r) * rng_excl;
    uint32_t leftover = (uint32_t)m;
    if (leftover < rng_excl) {
        const uint32_t threshold = (0xFFFFFFFFu - rng) % rng_excl;
        while (leftover < threshold) { m = (unsigned long long)next32(r) * rng_excl; leftover = (uint32_t)m; }
    }
    return low + (long long)(m >> 32);
}

// b2EdgeShape::RayCast against terrain edge e
LD bool edge_raycast(v2 v1, v2 v2_, v2 p1, v2 p2, float maxFraction, float &t_out) {
    const v2 d = sub(p2, p1);
    const v2 ed = sub(v2_, v1);
    v2 normal = V(ed.y, -ed.x);
    const float len = sqrtf(normal.x * normal.x + normal.y * normal.y);
    if (len >= 1.1920929e-07f) { const float inv = 1.0f / len; normal.x *= inv; normal.y *= inv; }
    const float numerator = dot(normal, sub(v1, p1));
    const float denominator = dot(normal, d);
    if (denominator == 0.0f) return false;
    const float t = numerator / denominator;
    if (t < 0.0f || maxFraction < t) return false;
    const v2 q = add(p1, scl(t, d));
    const v2 r = sub(v2_, v1);
    const float rr = dot(r, r);
    if (rr == 0.0f) return false;
    const float s = dot(sub(q, v1), r) / rr;
    if (s < 0.0f || 1.0f < s) return false;
    t_out = t;
    return true;
}

LD float sgnf(float a) { return a > 0.0f ? 1.0f : (a < 0.0f ? -1.0f : 0.0f); }
LD float clip01_abs(float a) { float x = fabsf(a); x = x < 0.0f ? 0.0f : x; return x > 1.0f ? 1.0f : x; }

// bipedal_walker.py:517-606
// bipedal_walker.py:517-545: motor commands, world.Step.  run_toi = false leaves b2World::SolveTOI to the caller.
template <bool HC>
LD void env_pre(World &W, const float (&action)[4], v2 hull_force, bool &awake, unsigned live, bool run_toi) {
    const float speed[NJ] = {4.0f, 6.0f, 4.0f, 6.0f};                            // SPEED_HIP, SPEED_KNEE
    for (int k = 0; k < NJ; k++) {                                               // :528-543
        W.j[k].motorSpeed = speed[k] * sgnf(action[k]);
        W.j[k].maxMotorTorque = 80.0f * clip01_abs(action[k]);
    }
    if constexpr (HC) {
        // every body stays within two leg lengths (2 x 34/30 m) of the hull: one window of boxes for all of them
        poly_window(W, W.b[0].c.x - 4.0f, W.b[0].c.x + 4.0f, W.p_lo, W.p_hi);
    }
    world_step<SceneT<HC>>(W, hull_force, 0.0f, -10.0f, awake, live, run_toi);   // :545
}

// bipedal_walker.py:547-606: lidar, observation, shaping reward, termination
template <bool HC>
__device__ __noinline__ void env_post(World &W, const float (&action)[4], bool from_reset, float (&obs)[24], double &reward,
                                      bool &terminated) {
    const double SCALE = 30.0, FPS = 50;
    const Body &H = W.b[0];
    const double posx = (double)H.xf.p.x, posy = (double)H.xf.p.y;
    double st[24];
    const float step = (float)(14 / 30.0);
    int lp_lo = 0, lp_hi = -1;
    if constexpr (HC) poly_window(W, (float)posx - 0.5f, (float)posx + 6.0f, lp_lo, lp_hi);   // LIDAR_RANGE = 160/30
    for (int i = 0; i < 10; i++) {                                               // :550-557
        // math.sin / math.cos(1.5 * i / 10.0): compile-time constants, spelled out so that the device uses
        // the host libm's values
        const double kSin[10] = {0.0, 0.14943813247359922, 0.29552020666133955, 0.43496553411123023, 0.5646424733950354,
                                 0.6816387600233341, 0.7833269096274834, 0.867423225594017, 0.9320390859672263,
                                 0.9757233578266591};
        const double kCos[10] = {1.0, 0.9887710779360422, 0.955336489125606, 0.9004471023526769, 0.8253356149096783,
                                 0.7316888688738209, 0.6216099682706644, 0.49757104789172696, 0.3623577544766736,
                                 0.2190066870930415};
        const double sn = kSin[i], cs = kCos[i];
        const double p2x = posx + sn * (160 / SCALE), p2y = posy - cs * (160 / SCALE);
        const v2 p1 = V((float)posx, (float)posy), p2 = V((float)p2x, (float)p2y);
        float frac = 1.0f, maxFraction = 1.0f;
        int lo = (int)floorf(p1.x / step) - 1, hi = (int)floorf(p2.x / step) + 1;
        lo = lo < 0 ? 0 : lo;
        hi = hi > NE - 1 ? NE - 1 : hi;
        for (int e = lo; e <= hi; e++) {
            float t;
            if (edge_raycast(V(terrain_x(e), terrain_y(W, e)), V(terrain_x(e + 1), terrain_y(W, e + 1)), p1, p2,
                             maxFraction, t)) { frac = t; maxFraction = t; }
        }
        if constexpr (HC) {   // LidarCallback accepts every fixture with categoryBits & 1: the boxes too (:504-510)
            for (int q = lp_lo; q <= lp_hi; q++) {
                StaticBox sb;
                static_box(sb, poly_word(W, q, 0), poly_word(W, q, 1), poly_word(W, q, 2), poly_word(W, q, 3));
                float t;
                if (static_box_raycast(sb, p1, p2, maxFraction, t)) { frac = t; maxFraction = t; }
            }
        }
        st[14 + i] = (double)frac;
    }
    st[0] = (double)H.a;                                                         // :559-577
    st[1] = 2.0 * (double)H.w / FPS;
    st[2] = 0.3 * (double)H.v.x * (600 / SCALE) / FPS;
    st[3] = 0.3 * (double)H.v.y * (400 / SCALE) / FPS;
    for (int li = 0; li < 2; li++) {
        const JointDef &hip = kC.jd[2 * li], &knee = kC.jd[2 * li + 1];
        const float hip_angle = W.b[hip.bodyB].a - W.b[hip.bodyA].a - 0.0f;      // GetJointAngle
        const float hip_speed = W.b[hip.bodyB].w - W.b[hip.bodyA].w;             // GetJointSpeed
        const float knee_angle = W.b[knee.bodyB].a - W.b[knee.bodyA].a - 0.0f;
        const float knee_speed = W.b[knee.bodyB].w - W.b[knee.bodyA].w;
        st[4 + 5 * li] = (double)hip_angle;
        st[5 + 5 * li] = (double)hip_speed / 4;
        st[6 + 5 * li] = (double)knee_angle + 1.0;
        st[7 + 5 * li] = (double)knee_speed / 6;
        st[8 + 5 * li] = (W.flags & (2u << li)) ? 1.0 : 0.0;
    }
    double shaping = 130 * posx / SCALE;                                         // :582-587
    shaping -= 5.0 * fabs(st[0]);
    double r = 0;
    if (W.flags & 8u) r = shaping - W.prev_shaping;                              // :589-592
    W.prev_shaping = shaping;
    W.flags |= 8u;
    // :594-596 -- `python_float - np.float32` is float32 under numpy >= 2: torque costs in float32
    double rew = r;
    if (!from_reset) {
        float r32 = (float)r;
        for (int k = 0; k < NJ; k++) r32 = r32 - (float)(0.00035 * 80) * clip01_abs(action[k]);
        rew = (double)r32;
    }
    bool term = false;
    if ((W.flags & 1u) || posx < 0) { rew = -100; term = true; }                 // :598-601
    if (posx > (200 - 10) * (14 / SCALE)) term = true;                           // :602-603
    for (int k = 0; k < 24; k++) obs[k] = (float)st[k];                          // :606
    reward = rew;
    terminated = term;
}

template <bool HC>
__device__ __noinline__ void env_step(World &W, const float (&action)[4], bool from_reset, v2 hull_force, float (&obs)[24],
                                      double &reward, bool &terminated, unsigned live = 0u) {
    bool awake;
    env_pre<HC>(W, action, hull_force, awake, live, true);
    env_post<HC>(W, action, from_reset, obs, reward, terminated);
}

// bipedal_walker.py:425-515 (W.terrain / W.n must be bound to this env's record)
template <bool HC>
__device__ __noinline__ void env_reset(World &W, Rng &rng, float (&obs)[24]) {
    uint32_t *terrain_out = W.terrain;
    const double SCALE = 30.0;
    const double TERRAIN_HEIGHT = 400 / SCALE / 4, TERRAIN_STEP = 14 / SCALE;
    const uint32_t stepped = W.flags & kFlagsKept;
    {   // _generate_terrain(hardcore) :277-402
        enum { GRASS = 0, STUMP, STAIRS, PIT, STATES };
        int state = GRASS;
        double velocity = 0.0, y = TERRAIN_HEIGHT, original_y = 0;
        long long counter = 20, stair_steps = 0, stair_width = 0, stair_height = 0;
        bool oneshot = false;
        int np = 0;
        auto box = [&](double x0, double ylo, double x1, double yhi) {   // CreateStaticBody(fixtures=fd_polygon)
            const int64_t base = (int64_t)(W_POLY - W_TERRAIN + 4 * np) * W.n;
            terrain_out[base] = __float_as_uint((float)x0);
            terrain_out[base + W.n] = __float_as_uint((float)ylo);
            terrain_out[base + 2 * W.n] = __float_as_uint((float)x1);
            terrain_out[base + 3 * W.n] = __float_as_uint((float)yhi);
            np++;
        };
        for (int i = 0; i < kTerrain; i++) {
            const double x = i * TERRAIN_STEP;
            if (state == GRASS && !oneshot) {
                const double d = TERRAIN_HEIGHT - y;
                const double sgn = d > 0 ? 1.0 : (d < 0 ? -1.0 : 0.0);
                velocity = 0.8 * velocity + 0.01 * sgn;                          // :296
                if (i > 20) velocity += bgym::pcg64_uniform(rng.g, -1, 1) / SCALE;  // :297-298
                y += velocity;
            } else if (HC && state == PIT && oneshot) {                          // :301-323
                counter = integers(rng, 3, 5);
                box(x, y - 4 * TERRAIN_STEP, x + TERRAIN_STEP, y);
                box(x + TERRAIN_STEP * counter, y - 4 * TERRAIN_STEP, x + TERRAIN_STEP + TERRAIN_STEP * counter, y);
                counter += 2;
                original_y = y;
            } else if (HC && state == PIT && !oneshot) {                         // :325-328
                y = original_y;
                if (counter > 1) y -= 4 * TERRAIN_STEP;
            } else if (HC && state == STUMP && oneshot) {                        // :330-341
                counter = integers(rng, 1, 3);
                box(x, y, x + counter * TERRAIN_STEP, y + counter * TERRAIN_STEP);
            } else if (HC && state == STAIRS && oneshot) {                       // :343-371
                stair_height = bgym::pcg64_next_double(rng.g) > 0.5 ? +1 : -1;
                stair_width = integers(rng, 4, 5);
                stair_steps = integers(rng, 3, 5);
                original_y = y;
                for (long long st = 0; st < stair_steps; st++)
                    box(x + (st * stair_width) * TERRAIN_STEP, y + (-1 + st * stair_height) * TERRAIN_STEP,
                        x + ((1 + st) * stair_width) * TERRAIN_STEP, y + (st * stair_height) * TERRAIN_STEP);
                counter = stair_steps * stair_width;
            } else if (HC && state == STAIRS && !oneshot) {                      // :373-376
                const long long sq = stair_steps * stair_width - counter - stair_height;
                const double nn = (double)sq / (double)stair_width;
                y = original_y + (nn * stair_height) * TERRAIN_STEP;
            }
            oneshot = false;
            terrain_out[(int64_t)i * W.n] = __float_as_uint((float)y);
            counter -= 1;
            if (counter == 0) {
                counter = integers(rng, 10 / 2, 10);                             // :379
                if (HC && state == GRASS) state = (int)integers(rng, 1, STATES); // :380-382
                else state = GRASS;                                              // :383-385
                oneshot = true;
            }
        }
        W.np = np;
    }
    for (int i = 0; i < kTerrain / 20; i++) {   // _generate_clouds :404-423 (cosmetic, consumes the stream)
        (void)bgym::pcg64_next64(rng.g);
        for (int a = 0; a < 10; a++) (void)bgym::pcg64_next64(rng.g);
    }
    for (int b = 0; b < NB; b++) {                                               // :444-500
        Body &B = W.b[b];
        const ShapeConst &sh = Scene::shape(b);
        const float y = b == 0 ? kC.init_y : ((b & 1) ? kC.leg_y : kC.lower_y);
        const float angle = b == 0 ? 0.0f : kC.leg_a0[(b - 1) >> 1];
        B.xf.p = V(kC.init_x, y);
        B.xf.q = rot_of(angle);
        B.c = xmul(B.xf, sh.localCenter);
        B.a = angle;
        B.v = V(0.0f, 0.0f);
        B.w = 0.0f;
        B.sleepTime = 0.0f;
    }
    for (int j = 0; j < NJ; j++) {
        W.j[j].imp[0] = W.j[j].imp[1] = W.j[j].imp[2] = 0.0f; W.j[j].motorImpulse = 0.0f; W.j[j].limitState = 0;
    }
    W.flags = stepped;
    W.prev_shaping = 0.0;
    for (int s = 0; s < kSlots; s++) W.slot_key[s] = 0u;
    const double fx = bgym::pcg64_uniform(rng.g, -5, 5);                         // :450-452 INITIAL_RANDOM
    const float zero[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    double r;
    bool t;
    env_step<HC>(W, zero, true, V((float)fx, 0.0f), obs, r, t);                  // :515
}

// ---- HBM <-> registers/local ---------------------------------------------------------------------
LD void bind_world(World &W, uint32_t *rec, int64_t n, int64_t i) {
    W.terrain = rec + (int64_t)W_TERRAIN * n + i;
    W.n = n;
}

LD void load_world(World &W, uint32_t *rec, int64_t n, int64_t i, Rng &rng, bool hardcore = false) {
    auto ld = [&](int k) { return rec[(int64_t)k * n + i]; };
    for (int b = 0; b < NB; b++) {
        Body &B = W.b[b];
        B.c.x = __uint_as_float(ld(W_BODY + 7 * b + 0)); B.c.y = __uint_as_float(ld(W_BODY + 7 * b + 1));
        B.a = __uint_as_float(ld(W_BODY + 7 * b + 2));
        B.v.x = __uint_as_float(ld(W_BODY + 7 * b + 3)); B.v.y = __uint_as_float(ld(W_BODY + 7 * b + 4));
        B.w = __uint_as_float(ld(W_BODY + 7 * b + 5)); B.sleepTime = __uint_as_float(ld(W_BODY + 7 * b + 6));
        sync_xf(B, Scene::shape(b));
    }
    for (int j = 0; j < NJ; j++) {
        for (int k = 0; k < 3; k++) W.j[j].imp[k] = __uint_as_float(ld(W_JOINT + 5 * j + k));
        W.j[j].motorImpulse = __uint_as_float(ld(W_JOINT + 5 * j + 3));
        W.j[j].limitState = (int)ld(W_JOINT + 5 * j + 4);
        W.j[j].motorSpeed = 0.0f;
        W.j[j].maxMotorTorque = 0.0f;
    }
    W.flags = ld(W_FLAGS);
    W.prev_shaping = __longlong_as_double((long long)(((unsigned long long)ld(W_SHAPING + 1) << 32) | ld(W_SHAPING)));
    rng.has32 = ld(W_RNG32);
    rng.val32 = ld(W_RNG32 + 1);
    for (int s = 0; s < kSlots; s++) {
        W.slot_key[s] = ld(W_SLOT + 7 * s);
        for (int p = 0; p < 2; p++) {
            W.slot_id[s][p] = ld(W_SLOT + 7 * s + 1 + 3 * p);
            W.slot_nI[s][p] = __uint_as_float(ld(W_SLOT + 7 * s + 2 + 3 * p));
            W.slot_tI[s][p] = __uint_as_float(ld(W_SLOT + 7 * s + 3 + 3 * p));
        }
    }
    bind_world(W, rec, n, i);
    W.np = hardcore ? (int)ld(W_NPOLY) : 0;
    W.p_lo = 0; W.p_hi = -1;
}

LD void store_world(const World &W, uint32_t *rec, int64_t n, int64_t i, const Rng &rng, bool hardcore = false) {
    auto st = [&](int k, uint32_t v) { rec[(int64_t)k * n + i] = v; };
    for (int b = 0; b < NB; b++) {
        const Body &B = W.b[b];
        st(W_BODY + 7 * b + 0, __float_as_uint(B.c.x)); st(W_BODY + 7 * b + 1, __float_as_uint(B.c.y));
        st(W_BODY + 7 * b + 2, __float_as_uint(B.a));
        st(W_BODY + 7 * b + 3, __float_as_uint(B.v.x)); st(W_BODY + 7 * b + 4, __float_as_uint(B.v.y));
        st(W_BODY + 7 * b + 5, __float_as_uint(B.w)); st(W_BODY + 7 * b + 6, __float_as_uint(B.sleepTime));
    }
    for (int j = 0; j < NJ; j++) {
        for (int k = 0; k < 3; k++) st(W_JOINT + 5 * j + k, __float_as_uint(W.j[j].imp[k]));
        st(W_JOINT + 5 * j + 3, __float_as_uint(W.j[j].motorImpulse));
        st(W_JOINT + 5 * j + 4, (uint32_t)W.j[j].limitState);
    }
    st(W_FLAGS, W.flags);
    const unsigned long long ps = (unsigned long long)__double_as_longlong(W.prev_shaping);
    st(W_SHAPING, (uint32_t)ps); st(W_SHAPING + 1, (uint32_t)(ps >> 32));
    st(W_RNG32, rng.has32); st(W_RNG32 + 1, rng.val32);
    if (hardcore) st(W_NPOLY, (uint32_t)W.np);
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
// so do the kept flag bits and numpy's 32-bit cache.  `n` by reference: see lunar::reset_from_record
template <bool HC>
LD void reset_from_record(uint32_t *rec, const int64_t &n, int64_t i, uint64_t *rng, float (&obs)[24]) {
    World W;
    Rng r;
    bind_world(W, rec, n, i);
    W.flags = rec[(int64_t)W_FLAGS * n + i] & kFlagsKept;
    r.has32 = rec[(int64_t)W_RNG32 * n + i];
    r.val32 = rec[(int64_t)(W_RNG32 + 1) * n + i];
    r.g = bgym::pcg64_load(rng + 4 * i);
    W.np = 0; W.p_lo = 0; W.p_hi = -1;
    env_reset<HC>(W, r, obs);
    store_world(W, rec, n, i, r, HC);
    bgym::pcg64_store(rng + 4 * i, r.g);
}

#undef LD
}  // namespace walker
