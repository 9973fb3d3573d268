// drone_core.cuh -- the per-environment arithmetic of one DroneGame.step(), written once as
// __host__ __device__ code and instantiated for float (throughput) and double (exact parity).
//
// This is a from-scratch statement of the reference's semantics, not a translation of its
// object structure.  Reference anchors (/root/reference/delivery_drone/game/):
//   drone.py:44-76     apply_thrust (sequential fuel gating)
//   drone.py:78-103    update (gravity, drag, integrate, rotate, wrap)
//   physics.py:6-23    rotate_point      physics.py:26-39 normalize_angle
//   game_engine.py:179-279  reward priority: landing, ground, fuel, out of bounds, shaping
//   game_engine.py:140-177  observation normalisation
#pragma once
#include <stdint.h>
#include <string.h>
#include <math.h>
#include <cmath>
#include "../../include/drone_b200.h"

#if defined(__CUDACC__)
#define DD_HD __host__ __device__ __forceinline__
#else
#define DD_HD inline
#endif

namespace dd {

// Constants derived on the host from DDParams, in the kernel's arithmetic type.
template <typename R>
struct Consts {
    R gravity, drag, ang_drag;
    R main_thrust, side_thrust, fuel_main, fuel_side, max_fuel;
    R half_h;                       // drone_height / 2       drone.py:136
    R plat_half_w, plat_half_h;     // platform.py:57-60
    R land_speed, land_angle;
    R ground_y;                     // height - ground_margin game_engine.py:254
    R x_lo, x_hi, y_lo, y_hi;       // game_engine.py:275-279
    R r_step, r_land, r_crash, r_fuel, r_oob;
    R shape_offset, shape_div, inv_shape_div;
    R width, height, vel_norm, angle_norm, angvel_norm;
    R inv_width, inv_height, inv_vel, inv_angle, inv_angvel, inv_fuel;
    R start_x, start_y, plat_x, plat_y;
    R spawn_x_min, spawn_y_min, plat_x_min, plat_y_min;
    uint32_t spawn_x_count, spawn_y_count, plat_x_count, plat_y_count;
    // reach of the bottom-centre point from the body centre, for the cheap landing pre-test
    R reach_x, reach_y;
    // speed > land_speed  <=>  vx^2 + vy^2 > speed2_max   (sqrt is correctly rounded and monotonic;
    // speed2_max = the largest R whose square root rounds to <= land_speed)
    R speed2_max;
    // r_step + terminal reward, rounded once in R exactly like the reference's `reward += ...`
    R rs_land, rs_crash, rs_fuel, rs_oob;
};

// Everything that is plain arithmetic on DDParams: usable at compile time for the default
// parameters (the kernels then see immediates instead of constant-bank loads).
template <typename R>
constexpr Consts<R> make_consts_base(const DDParams& p) {
    Consts<R> k{};
    k.gravity = (R)p.gravity; k.drag = (R)p.drag; k.ang_drag = (R)p.angular_drag;
    k.main_thrust = (R)p.main_thrust; k.side_thrust = (R)p.side_thrust;
    k.fuel_main = (R)p.fuel_main; k.fuel_side = (R)p.fuel_side; k.max_fuel = (R)p.max_fuel;
    k.half_h = (R)(p.drone_height / 2);
    k.plat_half_w = (R)(p.platform_w / 2); k.plat_half_h = (R)(p.platform_h / 2);
    k.land_speed = (R)p.land_speed; k.land_angle = (R)p.land_angle;
    k.ground_y = (R)(p.height - p.ground_margin);
    k.x_lo = (R)(-p.oob_margin); k.x_hi = (R)(p.width + p.oob_margin);
    k.y_lo = (R)(-p.oob_margin); k.y_hi = (R)(p.height + p.oob_margin);
    k.r_step = (R)p.r_step; k.r_land = (R)p.r_land; k.r_crash = (R)p.r_crash;
    k.r_fuel = (R)p.r_fuel; k.r_oob = (R)p.r_oob;
    k.shape_offset = (R)p.shape_offset; k.shape_div = (R)p.shape_div; k.inv_shape_div = (R)(1.0 / p.shape_div);
    k.width = (R)p.width; k.height = (R)p.height;
    k.vel_norm = (R)p.vel_norm; k.angle_norm = (R)p.angle_norm; k.angvel_norm = (R)p.angvel_norm;
    k.inv_width = (R)(1.0 / p.width); k.inv_height = (R)(1.0 / p.height);
    k.inv_vel = (R)(1.0 / p.vel_norm); k.inv_angle = (R)(1.0 / p.angle_norm);
    k.inv_angvel = (R)(1.0 / p.angvel_norm); k.inv_fuel = (R)(1.0 / p.max_fuel);
    k.start_x = (R)p.start_x; k.start_y = (R)p.start_y;
    k.plat_x = (R)p.plat_default_x; k.plat_y = (R)p.plat_default_y;
    k.spawn_x_min = (R)p.spawn_x_min; k.spawn_y_min = (R)p.spawn_y_min;
    k.plat_x_min = (R)p.plat_x_min; k.plat_y_min = (R)p.plat_y_min;
    k.spawn_x_count = (uint32_t)p.spawn_x_count; k.spawn_y_count = (uint32_t)p.spawn_y_count;
    k.plat_x_count = (uint32_t)p.plat_x_count; k.plat_y_count = (uint32_t)p.plat_y_count;
    // + 1: slack so that no rounding of (px - x) can reject a state the exact box test accepts
    k.reach_x = (R)(p.platform_w / 2 + p.drone_height / 2 + 1);
    k.reach_y = (R)(p.platform_h / 2 + p.drone_height / 2 + 1);
    k.speed2_max = (R)((R)p.land_speed * (R)p.land_speed);     // refined by make_consts()
    k.rs_land = (R)((R)p.r_step + (R)p.r_land); k.rs_crash = (R)((R)p.r_step + (R)p.r_crash);
    k.rs_fuel = (R)((R)p.r_step + (R)p.r_fuel); k.rs_oob = (R)((R)p.r_step + (R)p.r_oob);
    return k;
}

constexpr DDParams kDefaultParams = {
    800, 600, 0.3, 0.99, 0.95, 20, 0.6, 0.3, 1000.0, 2.0, 1.0, 100, 20, 3.0, 20.0, 50, 50,
    100.0, -100.0, -50.0, -50.0, -0.1, 500, 5000, 400, 100, 400, 500,
    100, 601, 50, 201, 100, 600, 100, 450, 10.0, 180.0, 10.0,
};

// Largest s with fl(sqrt(s)) <= limit, found by walking neighbours of limit^2 (host only).
template <typename R>
inline R speed2_threshold(R limit) {
    R s = limit * limit;
    const R inf = (R)INFINITY;
    for (int i = 0; i < 64 && std::sqrt(std::nextafter(s, inf)) <= limit; ++i) s = std::nextafter(s, inf);
    for (int i = 0; i < 64 && std::sqrt(s) > limit; ++i) s = std::nextafter(s, -inf);
    return s;
}

// Decision margin of step_core's PRE_SC landing shortcut (px): the shortcut and the exact evaluation can round the
// bottom centre to neighbouring floats -- one ulp of the largest coordinate the world allows apart -- and differ by the
// polynomial's error (< 1e-6 of half_h) besides.  8 ulps + 1e-5 half_h covers both; 1e-3 is the floor, which is the
// value for config.py's world (8 ulps of 850 = 4.9e-4 px), so the default-parameter kernels keep it as an immediate.
inline float pre_sc_margin(const DDParams& p) {
    const double far = std::fmax(p.width + p.oob_margin, p.height + p.oob_margin);
    int ex = 0;
    std::frexp(far, &ex);                                  // far in [2^(ex-1), 2^ex): one float ulp there is 2^(ex-24)
    const double m = 8.0 * std::ldexp(1.0, ex - 24) + 1e-5 * std::fabs(p.drone_height / 2);
    return m > 1e-3 ? (float)m : 1e-3f;
}

template <typename R>
inline Consts<R> make_consts(const DDParams& p) {
    Consts<R> k = make_consts_base<R>(p);
    k.speed2_max = speed2_threshold<R>((R)p.land_speed);
    return k;
}

// ---------------------------------------------------------------------------------------
// Arithmetic policy.  double: every product and sum rounded separately (no FMA contraction)
// and true division, so results track the float64 reference to the last sin/cos ulp.
// float: FMAs welcome, divisions by constants become reciprocal multiplies (<= 1.5 ulp).
// ---------------------------------------------------------------------------------------
template <typename R> struct Arith;

template <> struct Arith<double> {
    static DD_HD double mul(double a, double b) {
#if defined(__CUDA_ARCH__)
        return __dmul_rn(a, b);
#else
        return a * b;           // host build uses -ffp-contract=off
#endif
    }
    static DD_HD double add(double a, double b) {
#if defined(__CUDA_ARCH__)
        return __dadd_rn(a, b);
#else
        return a + b;
#endif
    }
    static DD_HD double fma_(double a, double b, double c) { return add(mul(a, b), c); }   // never fused
    static DD_HD double div(double a, double d, double /*inv_d*/) { return a / d; }
    static DD_HD double sqrt_(double a) { return sqrt(a); }
    static DD_HD double exp_(double a) { return exp(a); }
    static DD_HD double abs_(double a) { return fabs(a); }
    // sin / cos of an angle in degrees: np.radians(a) == a * (pi / 180)   physics.py:16-18
    static DD_HD void sincos_deg(double deg, double& s, double& c) {
        const double rad = mul(deg, 3.14159265358979323846 / 180.0);
#if defined(__CUDA_ARCH__)
        sincos(rad, &s, &c);
#else
        s = sin(rad); c = cos(rad);
#endif
    }
};

template <> struct Arith<float> {
    // Explicit roundings: the compiler may not contract or re-associate, so every kernel that
    // inlines step_core (one step per launch, T steps per launch, fused policy) is bit-identical.
#if defined(__CUDA_ARCH__)
    static DD_HD float mul(float a, float b) { return __fmul_rn(a, b); }
    static DD_HD float add(float a, float b) { return __fadd_rn(a, b); }
    static DD_HD float fma_(float a, float b, float c) { return __fmaf_rn(a, b, c); }
#else
    static DD_HD float mul(float a, float b) { return a * b; }
    static DD_HD float add(float a, float b) { return a + b; }
    static DD_HD float fma_(float a, float b, float c) { return fmaf(a, b, c); }
#endif
    static DD_HD float div(float a, float /*d*/, float inv_d) { return mul(a, inv_d); }
    static DD_HD float sqrt_(float a) { return sqrtf(a); }
    static DD_HD float exp_(float a) { return expf(a); }
    static DD_HD float abs_(float a) { return fabsf(a); }
    static DD_HD void sincos_deg(float deg, float& s, float& c) {
#if defined(__CUDA_ARCH__)
        // sin(pi * deg/180): exact range reduction, no radians rounding, <= 1 ulp each
        sincospif(deg * (1.0f / 180.0f), &s, &c);
#else
        // host twin: the same argument rounding as the device (deg / 180 in float), then sin / cos of pi * that in
        // float64 rounded once -- within 1 ulp of sincospif's result
        const double a = (double)(deg * (1.0f / 180.0f)) * 3.14159265358979323846;
        s = (float)sin(a); c = (float)cos(a);
#endif
    }
};

template <typename R>
struct Env {
    R x, y, vx, vy;             // pos_vel
    R angle, angvel, fuel, ret; // att_fuel
    R px, py;                   // platform
    int32_t steps;
};

// One DroneGame.step() for a live (not done) environment.  Returns the DD_* flags of this
// step (0 = still flying) and the engine reward.  `dist` (and `speed` when WANT_SPEED) come back
// because the observation wants them too (game_engine.py:166,171).
//
// Written for issue-slot economy (the kernels around it are HBM-bound only if this stays near
// ~100 instructions): the terminal priority chain is evaluated as selects, not branches; the
// landing test pays for sin/cos only when the cheap necessary conditions hold (rare); the speed
// limit is tested on vx^2+vy^2 against a pre-rounded threshold, so the step-only path has a
// single square root.  Every decision is the reference's, bit for bit, in R arithmetic.
//
// PRE_SC: the caller already holds (s_pre, c_pre) = sincos_deg(e.angle) of the PRE-update angle -- it does not
// depend on the action, so the fused policy kernel evaluates it while the network runs.  Same function of
// the same input: results are bit-identical to the PRE_SC = false instantiation, provided `pre_margin` is
// pre_sc_margin() of the parameters (1e-3 for config.py's).
template <typename R, bool WANT_SPEED, bool PRE_SC = false>
DD_HD uint32_t step_core(Env<R>& e, uint32_t act, const Consts<R>& k, R& reward, R& speed, R& dist,
                         R s_pre = (R)0, R c_pre = (R)0, R pre_margin = (R)1e-3)
{
    using A = Arith<R>;
    R vx = e.vx, vy = e.vy, w = e.angvel, fuel = e.fuel;

    // --- apply_thrust, drone.py:58-76: fuel re-tested before every thruster ------------
    if ((act & DD_ACT_MAIN) && fuel > (R)0) {
        R s = s_pre, c = c_pre;
        if (!PRE_SC) A::sincos_deg(e.angle, s, c);         // pre-update angle
        vx = A::fma_(k.main_thrust, s, vx);                // 0*c - (-0.6)*s    physics.py:20
        vy = A::fma_(-k.main_thrust, c, vy);               // 0*s + (-0.6)*c    physics.py:21
        fuel -= k.fuel_main;
    }
    if ((act & DD_ACT_LEFT) && fuel > (R)0) { w -= k.side_thrust; fuel -= k.fuel_side; }
    if ((act & DD_ACT_RIGHT) && fuel > (R)0) { w += k.side_thrust; fuel -= k.fuel_side; }
    fuel = fuel < (R)0 ? (R)0 : fuel;

    // --- update, drone.py:88-103 (dt == 1) -------------------------------------------------
    vy = A::add(vy, k.gravity);
    vx = A::mul(vx, k.drag);
    vy = A::mul(vy, k.drag);
    const R x = A::add(e.x, vx);
    const R y = A::add(e.y, vy);
    const R w_add = w;                                     // the angular velocity the angle advances by this step
    R ang = A::add(e.angle, w);
    w = A::mul(w, k.ang_drag);
    if (A::abs_(ang) > (R)180) {                           // physics.py:35-39 (rarely taken)
        while (ang > (R)180) ang -= (R)360;
        while (ang < (R)-180) ang += (R)360;
    }
    e.x = x; e.y = y; e.vx = vx; e.vy = vy; e.angle = ang; e.angvel = w; e.fuel = fuel;

    // --- terminal tests, game_engine.py:185-216 ----------------------------------------------
    const R speed2 = A::fma_(vx, vx, A::mul(vy, vy));                  // drone.py:145 (before sqrt)
    if (WANT_SPEED) speed = A::sqrt_(speed2);
    const R ddx = e.px - x, ddy = e.py - y;
    dist = A::sqrt_(A::fma_(ddx, ddx, A::mul(ddy, ddy)));              // physics.py:44

    // Priority (game_engine.py:187-214): landing, ground, fuel, out of bounds, else shaping.
    // Build it from the lowest priority up with selects.
    const bool oob = (x < k.x_lo) | (x > k.x_hi) | (y < k.y_lo) | (y > k.y_hi);   // :275-279
    const bool fuel_out = fuel <= (R)0;                                             // :200-204
    const bool ground = y > k.ground_y;                                             // :254-265
    R r = A::add(k.r_step, A::div(k.shape_offset - dist, k.shape_div, k.inv_shape_div));   // :213-214
    uint32_t f = 0;
    if (oob) { f = DD_DONE | DD_CRASHED | DD_CAUSE_OOB; r = k.rs_oob; }
    if (fuel_out) { f = DD_DONE | DD_CRASHED | DD_CAUSE_FUEL; r = k.rs_fuel; }
    if (ground) { f = DD_DONE | DD_CRASHED | DD_CAUSE_GROUND; r = k.rs_crash; }
    // Landing needs all of: bottom centre in the closed platform box, speed <= 3, |angle| <= 20
    // (game_engine.py:224-242).  The bottom centre is at most half_h from the body centre, so
    // the box test can only pass when |dx| <= w/2 + half_h and |dy| <= h/2 + half_h (+1 slack):
    // test that and the two cheap conditions before paying for sin/cos of the post-update angle.
    if (!(speed2 > k.speed2_max) && A::abs_(ang) <= k.land_angle &&
        A::abs_(ddx) <= k.reach_x && A::abs_(ddy) <= k.reach_y) {
        bool decided = false, inside = false;
        if constexpr (PRE_SC && sizeof(R) == 4) {
            // The caller holds sin / cos of the PRE-update angle (computed off the critical path).  The post-update
            // angle is that plus w_add (|w_add| is a few degrees), so sin / cos of it follow from the angle-addition
            // formulas and two short polynomials -- no range reduction, no MUFU -- to ~2e-7.  That is only used to
            // DECIDE: if the bottom-centre point so obtained is farther than pre_margin from every edge of the platform
            // box, inside / outside is certain and equals the exact decision bit for bit; otherwise the exact path runs.
            // The exact evaluation below can differ from the shortcut by one float ulp of the coordinates plus the
            // polynomial's error: < 1e-4 px while |x|, |y| < 2048 (config.py's world: pre_margin = 1e-3, the exact path
            // runs with probability ~1e-5 per test), but 1.95e-3 px at |x| >= 16384 -- pre_sc_margin() scales the
            // margin with the world.  The landing test sits on the serial chain of the fused policy kernel, where
            // sincospif's latency is paid by the whole tile.
            if (A::abs_(w_add) <= (R)8) {
                const R th = w_add * (R)0.017453292519943295, t2 = th * th;
                const R sn = th * ((R)1 + t2 * ((R)-0.16666666666666666 + t2 * (R)0.008333333333333333));
                const R cs = (R)1 + t2 * ((R)-0.5 + t2 * ((R)0.041666666666666664 + t2 * (R)-0.001388888888888889));
                const R sa = s_pre * cs + c_pre * sn, ca = c_pre * cs - s_pre * sn;
                const R bxa = x - k.half_h * sa, bya = y + k.half_h * ca;
                const R x0 = e.px - k.plat_half_w, x1 = e.px + k.plat_half_w, y0 = e.py - k.plat_half_h, y1 = e.py + k.plat_half_h;
                const R mx = fminf(A::abs_(bxa - x0), A::abs_(bxa - x1)), my = fminf(A::abs_(bya - y0), A::abs_(bya - y1));
                if (fminf(mx, my) > pre_margin) {
                    decided = true;
                    inside = (x0 <= bxa) && (bxa <= x1) && (y0 <= bya) && (bya <= y1);
                }
            }
        }
        if (!decided) {
            R s, c;
            A::sincos_deg(ang, s, c);
            const R bx = A::fma_(-k.half_h, s, x);         // x + (0*c - 10*s)  drone.py:136-137
            const R by = A::fma_(k.half_h, c, y);          // y + (0*s + 10*c)
            inside = (e.px - k.plat_half_w <= bx) && (bx <= e.px + k.plat_half_w) &&
                     (e.py - k.plat_half_h <= by) && (by <= e.py + k.plat_half_h);      // platform.py:74
        }
        if (inside) { f = DD_DONE | DD_LANDED; r = k.rs_land; }
    }
    reward = r;
    e.ret = A::add(e.ret, r);                              // game_engine.py:131
    e.steps += 1;                                          // game_engine.py:132
    return f;
}

// get_state(), game_engine.py:146-177, in the policy's key order (Actor_Critic_PPO.ipynb c10).
// `put(j, v)` stores element j.
template <typename R, typename Put>
DD_HD void write_obs(const Env<R>& e, uint32_t flags, R speed, R dist, const Consts<R>& k, Put put)
{
    using A = Arith<R>;
    put(0, A::div(e.x, k.width, k.inv_width));
    put(1, A::div(e.y, k.height, k.inv_height));
    put(2, A::div(e.vx, k.vel_norm, k.inv_vel));
    put(3, A::div(e.vy, k.vel_norm, k.inv_vel));
    put(4, A::div(e.angle, k.angle_norm, k.inv_angle));
    put(5, A::div(e.angvel, k.angvel_norm, k.inv_angvel));
    put(6, A::div(e.fuel, k.max_fuel, k.inv_fuel));
    put(7, A::div(e.px, k.width, k.inv_width));
    put(8, A::div(e.py, k.height, k.inv_height));
    put(9, A::div(dist, k.width, k.inv_width));            // distance normalised by WIDTH (:166)
    put(10, A::div(e.px - e.x, k.width, k.inv_width));
    put(11, A::div(e.py - e.y, k.height, k.inv_height));
    put(12, A::div(speed, k.vel_norm, k.inv_vel));
    put(13, (flags & DD_LANDED) ? (R)1 : (R)0);
    put(14, (flags & DD_CRASHED) ? (R)1 : (R)0);
}

// ---------------------------------------------------------------------------------------
// 16-bit observation formats (DDEnvConfig.obs_format): float -> binary16 / bfloat16 bits, round to nearest even --
// the bits torch's .to(torch.float16) / .to(torch.bfloat16) give.  The kernels convert a pair per instruction
// (cvt.rn.f16x2.f32 / cvt.rn.bf16x2.f32, SASS F2FP); the host twin uses the portable routines below, which give the
// same bits for every input but NaN (a quiet NaN either way).
// ---------------------------------------------------------------------------------------
inline uint16_t f16_bits_rn_portable(float f)
{
    uint32_t x;
    memcpy(&x, &f, 4);
    const uint32_t sign = (x >> 16) & 0x8000u, ax = x & 0x7fffffffu;
    if (ax >= 0x7f800000u) return (uint16_t)(sign | (ax > 0x7f800000u ? 0x7e00u : 0x7c00u));   // NaN / inf
    if (ax >= 0x477ff000u) return (uint16_t)(sign | 0x7c00u);          // >= 65520 (the 65504 / 65536 tie) -> inf
    if (ax < 0x38800000u) {                                            // |f| < 2^-14: subnormal or zero, units of 2^-24
        if (ax <= 0x33000000u) return (uint16_t)sign;                  // <= 2^-25 (the tie goes to the even 0)
        const uint32_t e = ax >> 23, m = (ax & 0x7fffffu) | 0x800000u, sh = 126u - e;   // sh in [14, 24]
        uint32_t r = m >> sh;
        const uint32_t rem = m & ((1u << sh) - 1u), half = 1u << (sh - 1u);
        if (rem > half || (rem == half && (r & 1u))) ++r;
        return (uint16_t)(sign | r);
    }
    const uint32_t y = ax - 0x38000000u;                               // re-bias the exponent: 127 -> 15
    uint32_t r = y >> 13;
    const uint32_t rem = y & 0x1fffu;
    if (rem > 0x1000u || (rem == 0x1000u && (r & 1u))) ++r;            // a carry into the exponent is correct
    return (uint16_t)(sign | r);
}

inline uint16_t bf16_bits_rn_portable(float f)
{
    uint32_t x;
    memcpy(&x, &f, 4);
    if ((x & 0x7fffffffu) > 0x7f800000u) return (uint16_t)0x7fc0u;    // NaN
    return (uint16_t)((x + 0x7fffu + ((x >> 16) & 1u)) >> 16);
}

// Bits 0-15: lo, bits 16-31: hi, in format FMT (DD_OBS_F16 / DD_OBS_BF16).
template <int FMT>
DD_HD uint32_t obs16_pack2(float lo, float hi)
{
    static_assert(FMT == DD_OBS_F16 || FMT == DD_OBS_BF16, "16-bit observation format");
#if defined(__CUDA_ARCH__)
    uint32_t r;
    if (FMT == DD_OBS_F16) asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
#else
    if (FMT == DD_OBS_F16) return (uint32_t)f16_bits_rn_portable(lo) | ((uint32_t)f16_bits_rn_portable(hi) << 16);
    return (uint32_t)bf16_bits_rn_portable(lo) | ((uint32_t)bf16_bits_rn_portable(hi) << 16);
#endif
}

// One observation row in a 16-bit format: write_obs's 15 values (+ `steps_col`: column 15 = `steps`) converted in pairs.
// `put16(j, bits)` stores element j.
template <int FMT, typename Put16>
DD_HD void write_obs16(const Env<float>& e, uint32_t flags, float speed, float dist, const Consts<float>& k,
                       bool steps_col, float steps, Put16 put16)
{
    float v[16];
    write_obs(e, flags, speed, dist, k, [&](int j, float x) { v[j] = x; });
    v[15] = steps;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < 14; j += 2) {
        const uint32_t w = obs16_pack2<FMT>(v[j], v[j + 1]);
        put16(j, (uint16_t)w); put16(j + 1, (uint16_t)(w >> 16));
    }
    const uint32_t w = obs16_pack2<FMT>(v[14], v[15]);
    put16(14, (uint16_t)w);
    if (steps_col) put16(DD_OBS_DIM, (uint16_t)(w >> 16));
}

template <typename R>
DD_HD void speed_dist(const Env<R>& e, R& speed, R& dist)
{
    using A = Arith<R>;
    speed = A::sqrt_(A::fma_(e.vx, e.vx, A::mul(e.vy, e.vy)));
    const R ddx = e.px - e.x, ddy = e.py - e.y;
    dist = A::sqrt_(A::fma_(ddx, ddx, A::mul(ddy, ddy)));
}

// ---------------------------------------------------------------------------------------
// N2: the PPO notebook's client-side training reward, fused as an epilogue of the step.
// calc_reward(state, prev_state) of Actor_Critic_PPO.ipynb c7:L2-101 + the time-out rule of
// c16:L89-93, in the notebook's statement order (restated in oracle/shaping_port.py, pinned by
// executing the notebook's cells).  Inputs are the normalised observation fields of the
// POST-step state (before any auto-reset); `prev_dist` is prev_state.distance_to_platform, i.e. the
// normalised distance of the state observed before the PREVIOUS step (c16:L71-72,101-102), NaN when
// there is none (first step of an episode).
// ---------------------------------------------------------------------------------------
template <typename R>
DD_HD R shaped_reward_ppo(const Env<R>& e, uint32_t flags, R speed, R dist, R prev_dist, bool timed_out,
                          const Consts<R>& k)
{
    using A = Arith<R>;
    const R nd = A::div(dist, k.width, k.inv_width);                   // distance_to_platform
    const R ns = A::div(speed, k.vel_norm, k.inv_vel);                 // speed
    const R nvx = A::div(e.vx, k.vel_norm, k.inv_vel), nvy = A::div(e.vy, k.vel_norm, k.inv_vel);
    const R ndx = A::div(e.px - e.x, k.width, k.inv_width), ndy = A::div(e.py - e.y, k.height, k.inv_height);
    const R nang = A::div(e.angle, k.angle_norm, k.inv_angle);
    const R nfuel = A::div(e.fuel, k.max_fuel, k.inv_fuel);

    R total = (R)-0.5;                                                  // 0 + (-0.5)
    R r_distance = (R)0, r_hover = (R)0;
    if (prev_dist == prev_dist) {                                       // prev_state is not None
        const R delta = prev_dist - nd;
        const R toward = nd > (R)1e-6 ? A::add(A::mul(nvx, ndx), A::mul(nvy, ndy)) / nd : (R)0;
        if (ns >= (R)0.15 && toward > (R)0.1 && nd > (R)0.065) {
            R v = A::mul(A::mul(delta, (R)1000), A::add((R)1.0, A::mul(ns, (R)2.0)));
            v = v < (R)-2 ? (R)-2 : v; v = v > (R)5 ? (R)5 : v;         // np.clip(., -2, 5)
            r_distance = v;
        } else if (delta < (R)-0.001) {
            r_distance = A::mul(A::mul((R)-2.0, A::abs_(delta)), (R)1000);
        } else if (ns < (R)0.05) {
            r_hover = (R)-1.0;
        } else if (ns < (R)0.15) {
            r_hover = (R)-0.3;
        }
    }
    total = A::add(total, r_distance);
    total = A::add(total, r_hover);
    const R excess = A::abs_(nang) - A::add(A::mul((R)(0.20 - 0.111), nd), (R)0.111);
    total = A::add(total, excess > (R)0 ? -excess : (R)0);
    const R over = nd < (R)1 ? A::mul((R)-2, (ns - (R)0.1 > (R)0 ? ns - (R)0.1 : (R)0))
                             : A::mul((R)-1, (ns - (R)0.6 > (R)0 ? ns - (R)0.6 : (R)0));
    total = A::add(total, over);
    total = A::add(total, ndy > (R)0 ? (R)0 : A::mul(ndy, (R)4.0));
    R terminal = (R)0;
    if (flags & DD_LANDED) terminal = A::add((R)800.0, A::mul(nfuel, (R)100.0));
    else if (flags & DD_CRASHED) terminal = nd > (R)0.3 ? (R)-300.0 : (R)-200.0;
    total = A::add(total, terminal);
    if (timed_out && !(flags & DD_LANDED)) total -= (R)500;             // c16:L89-93
    return total;
}

// calc_reward(state) of Policy_Gradients.ipynb (code cell 6; calc_velocity_alignment of code cell 5,
// inverse_quadratic / scaled_shifted_negative_sigmoid of rl_helpers/scalers.py:14-15,20-21) + the same -500
// time-out (collect_episodes of that notebook), in the notebook's statement order; restated in
// oracle/shaping_port.py (shaped_reward_pg), pinned by executing the notebook's cells.  Stateless.
template <typename R>
DD_HD R shaped_reward_pg(const Env<R>& e, uint32_t flags, R speed, R dist, bool timed_out, const Consts<R>& k)
{
    using A = Arith<R>;
    const R nd = A::div(dist, k.width, k.inv_width);                   // distance_to_platform
    const R ns = A::div(speed, k.vel_norm, k.inv_vel);                 // speed
    const R nvx = A::div(e.vx, k.vel_norm, k.inv_vel), nvy = A::div(e.vy, k.vel_norm, k.inv_vel);
    const R ndx = A::div(e.px - e.x, k.width, k.inv_width), ndy = A::div(e.py - e.y, k.height, k.inv_height);
    const R nang = A::div(e.angle, k.angle_norm, k.inv_angle);
    const R nfuel = A::div(e.fuel, k.max_fuel, k.inv_fuel);

    // time penalty: -inverse_quadratic(dist, decay=50, scaler=1-0.3) - 0.3
    R total = -A::mul((R)(1 - 0.3), (R)1 / A::add((R)1, A::mul((R)50, A::mul(nd, nd)))) - (R)0.3;
    // velocity alignment; note the notebook's sign: optimal_dx = -state.dx_to_platform
    R va;
    R odx = -ndx, ody = -ndy;
    const R onorm = A::sqrt_(A::add(A::mul(odx, odx), A::mul(ody, ody)));
    if (onorm < (R)1e-6) {
        va = (R)1;
    } else {
        odx = odx / onorm; ody = ody / onorm;
        va = ns < (R)1e-6 ? (R)0 : A::add(A::mul(nvx / ns, odx), A::mul(nvy / ns, ody));
    }
    R r_distance = (R)0, r_align = (R)0;
    if (nd > (R)0.065 && ndy > (R)0) {
        const R sig = A::mul((R)4.5, (R)1 / A::add((R)1, A::exp_(A::mul((R)10, nd - (R)0.5))));
        r_distance = A::mul(A::mul(va > (R)0 ? (R)1 : (R)0, ns), sig);
        if (va > (R)0) r_align = (R)0.5;
    }
    total = A::add(total, r_distance);
    total = A::add(total, r_align);
    const R excess = A::abs_(nang) - A::add(A::mul((R)(0.20 - 0.111), nd), (R)0.111);
    total = A::add(total, excess > (R)0 ? -excess : (R)0);
    const R over = nd < (R)1 ? A::mul((R)-2, (ns - (R)0.1 > (R)0 ? ns - (R)0.1 : (R)0))
                             : A::mul((R)-1, (ns - (R)0.4 > (R)0 ? ns - (R)0.4 : (R)0));
    total = A::add(total, over);
    total = A::add(total, ndy > (R)0 ? (R)0 : A::mul(ndy, (R)4.0));
    R terminal = (R)0;
    if (flags & DD_LANDED) terminal = A::add((R)500.0, A::mul(nfuel, (R)100.0));
    else if (flags & DD_CRASHED) terminal = nd > (R)0.3 ? (R)-300.0 : (R)-200.0;
    total = A::add(total, terminal);
    if (timed_out && !(flags & DD_LANDED)) total -= (R)500;
    return total;
}

// one switch for the kernels: `mode` is DDEnvConfig.shaping
template <typename R>
DD_HD R shaped_reward(int mode, const Env<R>& e, uint32_t flags, R speed, R dist, R prev_dist, bool timed_out,
                      const Consts<R>& k)
{
    return mode == DD_SHAPING_PG ? shaped_reward_pg(e, flags, speed, dist, timed_out, k)
                                 : shaped_reward_ppo(e, flags, speed, dist, prev_dist, timed_out, k);
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon, Moraes, Dror, Shaw, SC'11).  Counter-based: the spawn of episode k of
// global env g under seed s is a pure function of (s, g, k), whatever the grid or GPU count.
// ---------------------------------------------------------------------------------------
struct U4 { uint32_t a, b, c, d; };

DD_HD uint32_t mulhi_u32(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

DD_HD U4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1)
{
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = mulhi_u32(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = mulhi_u32(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return U4{c0, c1, c2, c3};
}

// DroneGame.reset(), game_engine.py:59-93 + drone.py:221-238 + platform.py:104-114.
// `episode` is the number of resets this env has had so far (the Philox counter).
// The four spawn coordinates of episode `episode` of env `env_id` (the random part of reset()).
template <typename R>
DD_HD void spawn_draw(const Consts<R>& k, uint64_t seed, uint64_t env_id, uint32_t episode, bool rand_drone, bool rand_platform,
                      R& x, R& y, R& px, R& py)
{
    Env<R> e;
    e.x = k.start_x; e.y = k.start_y; e.px = k.plat_x; e.py = k.plat_y;
    if (rand_drone || rand_platform) {
        const U4 r = philox4x32_10((uint32_t)env_id, (uint32_t)(env_id >> 32), episode, 0u,
                                   (uint32_t)seed, (uint32_t)(seed >> 32));
        if (rand_drone) {                                  // np.random.randint(lo, hi + 1)
            e.x = k.spawn_x_min + (R)mulhi_u32(r.a, k.spawn_x_count);
            e.y = k.spawn_y_min + (R)mulhi_u32(r.b, k.spawn_y_count);
        }
        if (rand_platform) {                               // np.random.randint(lo, hi)
            e.px = k.plat_x_min + (R)mulhi_u32(r.c, k.plat_x_count);
            e.py = k.plat_y_min + (R)mulhi_u32(r.d, k.plat_y_count);
        }
    }
    x = e.x; y = e.y; px = e.px; py = e.py;
}

// reset() given the spawn coordinates: everything else of a fresh episode
template <typename R>
DD_HD void spawn_apply(Env<R>& e, const Consts<R>& k, R x, R y, R px, R py)
{
    e.x = x; e.y = y; e.px = px; e.py = py;
    e.vx = (R)0; e.vy = (R)0; e.angle = (R)0; e.angvel = (R)0;
    e.fuel = k.max_fuel; e.ret = (R)0; e.steps = 0;
}

template <typename R>
DD_HD void spawn(Env<R>& e, const Consts<R>& k, uint64_t seed, uint64_t env_id, uint32_t episode,
                 bool rand_drone, bool rand_platform)
{
    e.x = k.start_x; e.y = k.start_y; e.px = k.plat_x; e.py = k.plat_y;
    if (rand_drone || rand_platform) {
        const U4 r = philox4x32_10((uint32_t)env_id, (uint32_t)(env_id >> 32), episode, 0u,
                                   (uint32_t)seed, (uint32_t)(seed >> 32));
        if (rand_drone) {                                  // np.random.randint(lo, hi + 1)
            e.x = k.spawn_x_min + (R)mulhi_u32(r.a, k.spawn_x_count);
            e.y = k.spawn_y_min + (R)mulhi_u32(r.b, k.spawn_y_count);
        }
        if (rand_platform) {                               // np.random.randint(lo, hi)
            e.px = k.plat_x_min + (R)mulhi_u32(r.c, k.plat_x_count);
            e.py = k.plat_y_min + (R)mulhi_u32(r.d, k.plat_y_count);
        }
    }
    e.vx = (R)0; e.vy = (R)0; e.angle = (R)0; e.angvel = (R)0;
    e.fuel = k.max_fuel; e.ret = (R)0; e.steps = 0;
}

// ---------------------------------------------------------------------------------------
// Per-env parameter sets (DDParamSets, include/drone_b200.h).  The table is Consts<R> of up to DD_MAX_PARAM_SETS sets
// laid out [word][set]: word j of set s (words of sizeof(R) bytes; the four uint32 counts pack into whole words) sits
// at j * DD_MAX_PARAM_SETS + s.  A warp's load of one field touches at most 64 * sizeof(R) contiguous bytes -- two
// 128-byte lines for float -- whatever mix of sets its lanes hold.  param_sets_build is the table's only writer and
// param_set its only reader, on the device and in the host twin alike.
// ---------------------------------------------------------------------------------------
template <typename R> struct ParamWord { using type = unsigned int; };
template <> struct ParamWord<double> { using type = unsigned long long; };
template <typename R> constexpr int kParamWords = (int)(sizeof(Consts<R>) / sizeof(R));
static_assert(sizeof(Consts<float>) == kParamWords<float> * 4 && sizeof(Consts<double>) == kParamWords<double> * 8,
              "Consts<R> must be whole words of R");
static_assert(sizeof(Consts<double>) * DD_MAX_PARAM_SETS <= DD_PARAM_TABLE_BYTES, "DD_PARAM_TABLE_BYTES too small");

// The constants of set `s` (already clamped to count - 1).  Fields the caller does not use are never loaded.
template <typename R>
DD_HD Consts<R> param_set(const void* table, uint32_t s)
{
    using W = typename ParamWord<R>::type;
    const W* t = static_cast<const W*>(table) + s;
    W w[kParamWords<R>];
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int j = 0; j < kParamWords<R>; ++j) w[j] = __ldg(t + j * DD_MAX_PARAM_SETS);
#else
    for (int j = 0; j < kParamWords<R>; ++j) w[j] = t[j * DD_MAX_PARAM_SETS];
#endif
    Consts<R> k;
    memcpy(&k, w, sizeof k);
    return k;
}

DD_HD uint32_t param_set_clamp(uint32_t index, uint32_t count) { return index < count ? index : count - 1u; }

// Host only: make_consts of sets[0 .. count) into the DD_PARAM_TABLE_BYTES at `out` (unused slots zero).
template <typename R>
inline void param_sets_build(const DDParams* sets, int count, void* out)
{
    using W = typename ParamWord<R>::type;
    memset(out, 0, DD_PARAM_TABLE_BYTES);
    for (int s = 0; s < count; ++s) {
        const Consts<R> k = make_consts<R>(sets[s]);
        W w[kParamWords<R>];
        memcpy(w, &k, sizeof k);
        for (int j = 0; j < kParamWords<R>; ++j) static_cast<W*>(out)[j * DD_MAX_PARAM_SETS + s] = w[j];
    }
}

// dd_param_sets_build (both libraries)
inline int param_sets_build_checked(const DDParams* sets, int32_t count, int32_t dtype, void* out)
{
    if (!sets || !out) return DD_E_NULL;
    if (count < 1 || count > DD_MAX_PARAM_SETS) return DD_E_RANGE;
    if (dtype == DD_F32) { param_sets_build<float>(sets, count, out); return 0; }
    if (dtype == DD_F64) { param_sets_build<double>(sets, count, out); return 0; }
    return DD_E_DTYPE;
}

// The set an env resampling at its reset number `episode` draws (DD_PARAM_SETS_RESAMPLE): Philox stream 3.
DD_HD uint32_t param_set_draw(uint64_t seed, uint64_t env_id, uint32_t episode, uint32_t count)
{
    const U4 r = philox4x32_10((uint32_t)env_id, (uint32_t)(env_id >> 32), episode, 3u,
                               (uint32_t)seed, (uint32_t)(seed >> 32));
    return mulhi_u32(r.a, count);
}

// 3-bit synthetic random action of step t (p = 0.5 per thruster).  One Philox call serves 32
// consecutive steps: action j = t % 32 is bits [3j, 3j+3) of the 96-bit string a | b<<32 | c<<64.
DD_HD U4 action_block(uint64_t seed, uint64_t env_id, uint32_t t)
{
    return philox4x32_10((uint32_t)env_id, (uint32_t)(env_id >> 32), t >> 5, 1u,
                         (uint32_t)seed, (uint32_t)(seed >> 32));
}
DD_HD uint32_t action_from_block(const U4& r, uint32_t t)
{
    const uint32_t bit = 3u * (t & 31u), w = bit >> 5, sh = bit & 31u;
    const uint32_t lo = w == 0 ? r.a : (w == 1 ? r.b : r.c);
    const uint32_t hi = w == 0 ? r.b : (w == 1 ? r.c : r.d);
    const uint64_t two = (uint64_t)lo | ((uint64_t)hi << 32);
    return (uint32_t)(two >> sh) & 7u;
}

}  // namespace dd
