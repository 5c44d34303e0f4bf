// hlynr_device.cuh -- device code of the batched Hlynr Intercept simulator (sm_100a).
//
// One environment per thread.  State lives in HBM as planes of 16-byte (fp32 build) or 32-byte
// (fp64 build) vectors, one plane per group of four words, so every load/store of a warp is one fully
// coalesced 512-byte (or 1 KiB) transaction.  The sensor-delay FIFOs of the reference
// (rl_system/core.py:147 SensorDelayBuffer) are ring planes indexed by the GLOBAL tick, so all envs
// read and write the same ring row in a step: one slot read + one slot write per env, coalesced.
//
// The arithmetic restates the reference step (rl_system/environment.py:605-859 and callees).
//   R = float : "fp32 build".  The integration sums, the distance and the reward -- the quantities whose
//               rounding the parity contract can see (reward = f(prev_distance - distance)) -- use the
//               never-contracted IEEE operations in the reference's order, so positions, velocities,
//               distances and rewards stay bit-identical to the native NumPy-2 reference almost always.
//               Everything that enters those sums far below one ulp (ISA, drag, wind) or only reaches an
//               observation channel uses cheap forms (MUFU reciprocal / rsqrt / lg2 / ex2, FMA chains).
//   R = double: "fp64 build" (matches the up-cast float64 reference, SURVEY Appendix B.5): integrator, ISA,
//               drag, distance, reward in exact double operations; observation geometry in float as the
//               reference forces it.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/hlynr.h"
#include "../../include/hlynr_rng.h"

namespace hlynr {

#define HD __device__ __forceinline__

// ------------------------------------------------------------------------------------------------
// never-contracted IEEE arithmetic (parity-critical sums)
// ------------------------------------------------------------------------------------------------
HD float mul(float a, float b) { return __fmul_rn(a, b); }
HD float add(float a, float b) { return __fadd_rn(a, b); }
HD float sub(float a, float b) { return __fsub_rn(a, b); }
HD float dvd(float a, float b) { return __fdiv_rn(a, b); }
HD float sqr(float a) { return __fsqrt_rn(a); }
HD double mul(double a, double b) { return __dmul_rn(a, b); }
HD double add(double a, double b) { return __dadd_rn(a, b); }
HD double sub(double a, double b) { return __dsub_rn(a, b); }
// fp64 build: a / b as a * (1 / b) with the reciprocal from rcp.approx.ftz.f64 (20 bits) + two Newton steps (80 bits -> full
// double): ~8 instructions and no slow-path call instead of the ~30 of the correctly rounded IEEE division.  The build's contract
// is rtol 1e-5 against the float64 reference, not bit-exactness, and the reciprocal and the quotient are within 1 ulp over the
// normal range (worst measured on a B200, tests/test_device_math.py); the profile that
// motivated it (profiles/r02_b_fp64_*) shows 3729 instructions per env-step of 165 KB straight-line code with `no_instruction`
// (instruction-cache misses) as the top stall reason.  Every divisor on the path is positive and finite (guards are at the call
// sites, as in the reference).  Outside the normal range the ftz reciprocal is not IEEE: drcp(+-0), drcp(subnormal) and
// drcp(+-inf) are NaN, drcp(b) is +-0 for |b| > 2^1022.  -DHLYNR_F64_EXACT_DIV restores __ddiv_rn.
// The final product is __dmul_rn like every operation of this section: a plain `*` may be contracted with an addition that follows
// it into an FMA, and whether the compiler does so depends on the code around the call: with a plain `*` the FT_V2OFF and the
// generic step kernels of this build left the missile state of cfg2 different in the last bits (tests/test_kernel_variants.py).
HD double drcp(double b) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));
    double e = fma(-b, r, 1.0);
    r = fma(r, e, r);
    e = fma(-b, r, 1.0);
    return fma(r, e, r);
}
#ifdef HLYNR_F64_EXACT_DIV
HD double dvd(double a, double b) { return __ddiv_rn(a, b); }
#else
HD double dvd(double a, double b) { return __dmul_rn(a, drcp(b)); }
#endif
#if defined(HLYNR_F64_EXACT_DIV) || defined(HLYNR_F64_EXACT_SQRT)
HD double sqr(double a) { return __dsqrt_rn(a); }
#else
// sqrt(a) = a * rsqrt(a): rsqrt.approx.ftz.f64 + two Newton steps, within 3 ulp on [2.3e-308, DBL_MAX] (worst measured on a B200).
// Below 2.3e-308 (zero, subnormals, the smallest normals), for negative a and for NaN it returns +0; sqr(+inf) is NaN.  The
// arguments on the path are finite sums of squares (the state stays finite: spawns are finite and accelerations bounded or guarded).
HD double sqr(double a) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    const double h = 0.5 * a;
    y = y * fma(-h * y, y, 1.5);
    y = y * fma(-h * y, y, 1.5);
    return a > 2.3e-308 ? a * y : 0.0;
}
#endif

// np.dot / np.linalg.norm on float32 vectors: float products, double accumulator, one final rounding
// (OpenBLAS sdot as used by the reference's NumPy; see oracle/hlynr_oracle.c dotn).
HD float dot3(float ax, float ay, float az, float bx, float by, float bz) {
    double s = (double)__fmul_rn(ax, bx) + (double)__fmul_rn(ay, by);
    s += (double)__fmul_rn(az, bz);
    return (float)s;
}
HD double dot3(double ax, double ay, double az, double bx, double by, double bz) {
    return add(add(mul(ax, bx), mul(ay, by)), mul(az, bz));
}
template <typename T> HD T norm3(T x, T y, T z) { return sqr(dot3(x, y, z, x, y, z)); }
HD float dot2(float ax, float ay, float bx, float by) { return (float)((double)__fmul_rn(ax, bx) + (double)__fmul_rn(ay, by)); }
HD double dot2(double ax, double ay, double bx, double by) { return add(mul(ax, bx), mul(ay, by)); }

HD double clip(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }
HD float clip(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

// ------------------------------------------------------------------------------------------------
// "near" operations: used where an error of a few float ulps is far below what the parity contract can see.
// float: MUFU approximations / FMA chains; double (fp64 build): the exact operation.
// ------------------------------------------------------------------------------------------------
HD float nrcp(float a) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r; }
#ifdef HLYNR_F64_EXACT_DIV
HD double nrcp(double a) { return __ddiv_rn(1.0, a); }
#else
HD double nrcp(double a) {   // defined below: rcp.approx.ftz.f64 + two Newton steps
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
    double e = fma(-a, r, 1.0);
    r = fma(r, e, r);
    e = fma(-a, r, 1.0);
    return fma(r, e, r);
}
#endif
HD float ndiv(float a, float b) { return a * nrcp(b); }
HD double ndiv(double a, double b) { return dvd(a, b); }
HD float nsqrt(float a) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r; }
HD double nsqrt(double a) { return sqr(a); }
HD float ndot3(float ax, float ay, float az, float bx, float by, float bz) { return fmaf(az, bz, fmaf(ay, by, ax * bx)); }
HD double ndot3(double ax, double ay, double az, double bx, double by, double bz) { return dot3(ax, ay, az, bx, by, bz); }
template <typename T> HD T nnorm3(T x, T y, T z) { return nsqrt(ndot3(x, y, z, x, y, z)); }
HD float npow(float x, float y) { return exp2f(y * __log2f(x)); }
HD double npow(double x, double y) { return exp(y * log(x)); }   // x > 0 on this path (temperature ratio, altitude / 10 m): isa_props within 11 ulp (B200) at a third of pow()'s code
HD float nexp(float x) { return __expf(x); }
HD double nexp(double x) { return exp(x); }
// x / c for a constant c with rc = RN(1/c): Markstein's correction in 3 instructions instead of the ~13 of an IEEE division.
// It is not correctly rounded for every c; it is, float and double, for the constants the kernel passes (500, 100 and dt = 0.01,
// the dt of every shipped configuration), checked on a B200 for every normal quotient (tests/test_device_math.py).  A subnormal
// quotient may be 1 ulp off, and the quotient of -0 is +0.
HD float cdiv(float x, float c, float rc) {
    float q = __fmul_rn(x, rc);
    float r = __fmaf_rn(-q, c, x);
    return __fmaf_rn(r, rc, q);
}
#ifdef HLYNR_F64_EXACT_DIV
HD double cdiv(double x, double c, double) { return __ddiv_rn(x, c); }
#else
HD double cdiv(double x, double c, double rc) {   // division by a constant: Markstein's correction with rc = RN(1 / c)
    const double q = x * rc;
    return fma(fma(-q, c, x), rc, q);
}
#endif

// atan2 / asin for the euler-angle channels obs[9:12] (core.py:1103-1121): degree-7 minimax polynomial of atan(a)/a in
// a^2 on [0,1] (1.9e-7 rad from the polynomial), one MUFU reciprocal, quadrant fix-up: ~20 instructions instead of the ~57
// of atan2f.  Worst error measured on a B200 over all octants: 3.4e-7 rad for fast_atan2 (the final pi/2 - r, pi - r
// roundings add to the polynomial's), 2.4e-7 rad for fast_asin.  Domain: 2^-126 <= max(|x|, |y|) < 2^126 or x = y = 0;
// from 2^126 on the ftz reciprocal is 0 and the angle collapses (fast_atan2(1e38, 2e38) = 0), and x = -0 counts as positive.
// The kernel's arguments have magnitude <= 2.  The channels are observations only (they never feed the dynamics).
HD float fast_atan2(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const float a = mx > 0.f ? mn * nrcp(mx) : 0.f;
    const float s = a * a;
    float p = -0.004780525807291269f;
    p = fmaf(p, s, 0.024557389318943024f);
    p = fmaf(p, s, -0.05990511178970337f);
    p = fmaf(p, s, 0.09942789375782013f);
    p = fmaf(p, s, -0.14029431343078613f);
    p = fmaf(p, s, 0.1997137814760208f);
    p = fmaf(p, s, -0.3333209455013275f);
    p = fmaf(p, s, 0.9999999403953552f);
    float r = p * a;
    if (ay > ax) r = 1.57079632679489662f - r;
    if (x < 0.f) r = 3.14159265358979324f - r;
    return copysignf(r, y);
}
HD float fast_asin(float x) { return fast_atan2(x, nsqrt((1.f - x) * (1.f + x))); }  // x already clipped to [-1, 1]

template <typename T> struct alignas(sizeof(T) * 4) Vec4 { T x, y, z, w; };

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 + the draw contract of include/hlynr_rng.h
// ------------------------------------------------------------------------------------------------
// The key schedule k_r = k + r*W depends only on the seed: the 10 round keys are computed on the host and
// read from the kernel-parameter bank; each round is two 32x32->64 multiplies (IMAD.WIDE) and two LOP3.
struct RoundKeys { uint32_t k[20]; };
struct RngKey { const RoundKeys* rk; uint32_t c0, c3hi; };  // c0 = env id low word, c3hi = (env id >> 32) << 16

HD uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const RoundKeys& rk) {
#pragma unroll   // (unrolled by 2 instead, for code size: cfg4 98.5 -> 111.6 us, fp64 build 218.9 -> 228.9 us: indexed round keys)
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)HLYNR_PHILOX_M0 * c0, p1 = (uint64_t)HLYNR_PHILOX_M1 * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ rk.k[2 * r], n2 = (uint32_t)(p0 >> 32) ^ c3 ^ rk.k[2 * r + 1];
        c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
    }
    return make_uint4(c0, c1, c2, c3);
}
HD uint4 draw_raw(const RngKey& k, uint32_t episode, uint32_t step, uint32_t blk) {
    return philox4x32_10(k.c0, episode, step, blk | k.c3hi, *k.rk);
}
HD float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-8f; }
HD float u01_open(uint32_t x) { return (float)((x >> 8) + 1u) * 5.9604644775390625e-8f; }
// accurate Box-Muller (reset path: domain-randomization draws, gust direction): within 1.8e-7 r of float64 (B200)
HD void box_muller(uint32_t xa, uint32_t xb, float* z0, float* z1) {
    float r = sqrtf(-2.0f * logf(u01_open(xa)));
    float s, c;
    sincospif(2.0f * u01(xb), &s, &c);
    *z0 = r * c; *z1 = r * s;
}
// per-tick draws: the same Box-Muller pairs evaluated with MUFU lg2/sqrt/sin/cos (absolute error ~1e-6 on a
// standard normal, i.e. ~1e-5 m on the noisiest channel: far below every parity tolerance).  Near u = 1 the absolute error
// of __log2f (CUDA documents up to 2^-22) dominates the small radius.  Worst measured on a B200 over every radius word and
// every angle word: |z - z_exact| <= 2.1e-6 for radii >= 0.1, and |z - z_exact| * r <= 7.5e-8 below (2.2e-4 at the smallest
// nonzero radius, 3.5e-4).  __log2f could in principle make the square root's argument negative there; over all 2^24 radius
// words it never does on a B200 (tests/test_device_math.py).
HD void fast_pair(uint32_t xa, uint32_t xb, float* z0, float* z1) {
    float r = nsqrt(-1.3862943611198906f * __log2f(u01_open(xa)));  // sqrt(-2 ln u)
    float t = 2.0f * u01(xb);
    t = (t < 1.0f ? t : t - 2.0f) * 3.14159265358979f;             // pi*t folded into [-pi, pi)
    *z0 = r * __cosf(t); *z1 = r * __sinf(t);
}
HD void draw_normal3(const RngKey& k, uint32_t episode, uint32_t step, uint32_t blk, float* z0, float* z1, float* z2) {
    uint4 r = draw_raw(k, episode, step, blk);
    float z3;
    fast_pair(r.x, r.y, z0, z1);
    fast_pair(r.z, r.w, z2, &z3);
}

// ------------------------------------------------------------------------------------------------
// resolved parameters, pre-rounded on the host to the dtype they meet in the reference
// ------------------------------------------------------------------------------------------------
template <typename R> struct KParams {
    // ---- S context (integrator dtype) ----
    R dt, rc_dt, tau, dt_over_tau, isa_expo, gas_R, gamma_R, sub_mach, sup_mach, sup_minus_sub;
    R peak_minus1, cd_sup, cd_base, missile_ratio, rho_weak, cs_weak, half_rho_weak, nhcr_weak;
    R blh, rc_blh, pf_top, ti_low, ti_high, turb, lp, wind_var;
    R kill_radius, target_x, target_y;
    R base_wind[3];
    double sup_mult_d;  // DR: base_cd * sup_mult in float64
    double dt_d;        // dt as the Python float it is in the reference
    double radar_quality_d, gust_scale_d;
    // ---- float context (observation geometry) ----
    float radar_range, rc_radar_range, radar_quality, rc_max_velocity_f, rc_max_range_f, max_velocity_f, max_range_f;
    float gpos[3], g_max_range, rc_g_max_range, g_sin_min_el, g_sin_max_el, g_base_q, max_link, rc_max_link, pkt_loss;
    float dtf, q_pp, q_pv, q_vv;  // Kalman F/Q entries (float32 matrices, core.py:33-56)
    float fus_035q;
    // ---- island context (W = R) ----
    R sigma_r, sigma_v, rc_max_range_w, rc_max_velocity_w;
    // ---- spawn / DR (double, reset path only) ----
    double m_pos_lo[3], m_pos_hi[3], m_speed_lo, m_speed_hi, m_radius_lo, m_radius_hi, m_az_lo, m_az_hi, m_el_lo, m_el_hi;
    double i_pos_lo[3], i_pos_hi[3], i_vel_lo[3], i_vel_hi[3], i_speed_lo, i_speed_hi, target_d[3];
    double dr_var[HLYNR_N_DR];
    // ---- switches ----
    int32_t max_steps, isa, mach, enh_wind, thrust_dyn, dr, validate, evasion, onboard_delay, ground, ground_delay;
    int32_t spherical, toward_missile, obs_mode, precision_mode, fuze, onb_ring_len, gnd_ring_len;
    int32_t volley_k;  // 0 = volley_mode off, else missiles per env (environment.py:42-43)
};

// ------------------------------------------------------------------------------------------------
// Feature sets: F < 0 = generic (every switch read from the parameters at run time); F >= 0 = the switches are
// compile-time constants, so the uniform flag tests and the dead branches disappear.  The host launches a
// specialised instantiation when the resolved configuration matches one, else the generic kernel.
// ------------------------------------------------------------------------------------------------
enum { FT_ISA = 1, FT_MACH = 2, FT_ENHW = 4, FT_THRUST = 8, FT_ONBD = 16, FT_GROUND = 32, FT_GDELAY = 64, FT_EVADE = 128, FT_DR = 256 };
#define FT_GENERIC (-1)        /* every switch at run time, world_frame observations */
#define FT_GENERIC_MODES (-2)  /* the same + observation_mode body_frame / los_frame (and the LOS action transform) + volley mode */
#define FT_V2ON (FT_ISA | FT_MACH | FT_ENHW | FT_THRUST | FT_ONBD | FT_GROUND | FT_GDELAY | FT_EVADE)  /* cfg4: medium, v2.0 on */
#define FT_V2OFF (FT_GROUND | FT_GDELAY | FT_EVADE)                                                   /* cfg2: medium, v2.0 off */
#define FT_V2ON_DR (FT_V2ON | FT_DR)                                                                   /* cfg3: hard, v2.0 on + domain randomization */
template <int F> struct Feat {
    static constexpr bool generic = F < 0;
    template <typename P> static HD bool isa(const P& p) { if constexpr (F < 0) return p.isa != 0; else return (F & FT_ISA) != 0; }
    template <typename P> static HD bool mach(const P& p) { if constexpr (F < 0) return p.mach != 0; else return (F & FT_MACH) != 0; }
    template <typename P> static HD bool enh_wind(const P& p) { if constexpr (F < 0) return p.enh_wind != 0; else return (F & FT_ENHW) != 0; }
    template <typename P> static HD bool thrust_dyn(const P& p) { if constexpr (F < 0) return p.thrust_dyn != 0; else return (F & FT_THRUST) != 0; }
    template <typename P> static HD bool onboard_delay(const P& p) { if constexpr (F < 0) return p.onboard_delay > 0; else return (F & FT_ONBD) != 0; }
    template <typename P> static HD bool ground(const P& p) { if constexpr (F < 0) return p.ground != 0; else return (F & FT_GROUND) != 0; }
    template <typename P> static HD bool ground_delay(const P& p) { if constexpr (F < 0) return p.ground_delay > 0; else return (F & FT_GDELAY) != 0; }
    template <typename P> static HD bool evasion(const P& p) { if constexpr (F < 0) return p.evasion != 0; else return (F & FT_EVADE) != 0; }
    template <typename P> static HD bool dr(const P& p) { if constexpr (F < 0) return p.dr != 0; else return (F & FT_DR) != 0; }
    // never part of a specialised set: the non-standard modes
    template <typename P> static HD bool precision_mode(const P& p) { if constexpr (F < 0) return p.precision_mode != 0; else return false; }
    template <typename P> static HD bool fuze(const P& p) { if constexpr (F < 0) return p.fuze != 0; else return false; }
    template <typename P> static HD int volley(const P& p) { if constexpr (F == FT_GENERIC_MODES) return p.volley_k; else return 0; }
    template <typename P> static HD int obs_mode(const P& p) { if constexpr (F == FT_GENERIC_MODES) return p.obs_mode; else return HLYNR_OBS_WORLD; }
};

template <typename R> struct KCurriculum {
    R intercept_radius;   // S context
    float cos_half_beam;  // beam gate acos(c) > radians(width/2)  <=>  c < cos(radians(width/2))
    float onboard_rel, ground_rel;
};

template <typename R> struct StatePlanes {
    Vec4<R>* r[7];   // r0 ipos+fuel, r1 ivel+fuel_used, r2 mpos+prev_d, r3 mvel+last_d, r4 kf_xp+min_d,
                     // r5 kf_xv+ep_return, r6 thrust+T0
    float4* f[4];    // f0 quat, f1 wind+base_cd, f2 Ppv,Pvp,Pvv,Ppp, f3 peak (DR only)
    int4* i0;        // steps, worsen, flags (bit0 crossed, bit1 kf_init, bits 8.. onboard delay), episode
    Vec4<R>* vm;     // volley mode: [volley_k][2][stride]: {pos.xyz, min_distance}, {vel.xyz, active}
    Vec4<R>* gring;  // [gnd_ring_len][2][stride]: {rel.xyz, quality}, {vel.xyz, -}
    float4* oring;   // [onb_ring_len][stride]: {rel.xyz, detected}
};

struct StepIO {
    const float* actions;   // [N,6] (or [k,N,6] for the fused rollout; NULL = in-kernel random policy)
    float* obs;             // [N,26]
    float* reward;          // [N]
    uint8_t* terminated;    // [N]
    uint8_t* truncated;     // [N]
    uint8_t* done;          // [N] or NULL: terminated | truncated (the host path's SB3 `dones`, saves a host pass over both)
    float* terminal_obs;    // [N,26] or NULL
    HlynrInfoSoA info;      // optional arrays
    const uint8_t* reset_mask;  // reset kernel only
    float* reward_sum;      // rollout
    int32_t* done_count;    // rollout
    double* stats;          // [STAT_SLOTS][HLYNR_STATS_WORDS]
    HlynrDoneRecord* done_records;  // optional compact list of the episodes that finished in this call
    int32_t* done_counter;          // records appended so far (atomic); may exceed done_cap (then the tail is dropped)
    int32_t done_cap;
};
#define HLYNR_STAT_SLOTS 64

template <typename R> struct KernelArgs {
    KParams<R> P;
    KCurriculum<R> C;
    StatePlanes<R> st;
    // Delayed ring rows this tick READS (API-mode launches; set with the tick on the host, next to the plane pointers so the
    // prologue gets them with the same constant-bank lines): the row written `onboard_delay` ticks ago, the two planes of the oldest
    // ground row.  NULL = no such ring (or a per-env delay: domain randomization).
    const float4* pf_o;
    const Vec4<R>* pf_g;
    StepIO io;
    RoundKeys rk;
    int64_t n;
    int64_t first, lim;   // env range [first, lim) of this launch (host-pipelined chunks; whole shard = [0, n))
    int64_t ring_stride;  // row pitch of the ring planes (n rounded up to 32 envs)
    int64_t env_offset;
    uint32_t tick;        // global tick of this launch (rollout: tick of the first fused step)
    int32_t g_row, o_row; // ring rows written at `tick` (tick % ring_len, computed on the host)
    int32_t auto_reset;
    int32_t k_steps;
    int32_t has_info;
    int32_t prefetch_ahead;  // envs per resident wave of CTAs (0 = no L2 prefetch of the next wave's planes)
    int32_t obs_dim;         // row pitch of io.obs / io.terminal_obs: HLYNR_OBS_DIM, or 17 = the leading "17-D radar" channels only
    int32_t compact;         // compact plane layout (see load_env): the counters ride in r6.w / f1.w, the i0 plane is unused
    // NULL = the curriculum is C.  Else the device slot curriculum_tick_kernel (hlynr_capi.cu) filled before this launch from the
    // attached schedule's training-step counter, and the host launches the kCur instantiation, which reads it (cur_*() below).
    const KCurriculum<R>* cur_dev;
};

// Curriculum scalars of a launch.  kCur = false: the by-value C, exactly the code of a build without schedules.  kCur = true (a
// separate instantiation, launched while a schedule is attached): the slot at cur_dev, which the kernel launched right before this
// one wrote, read at each use site and only after griddepcontrol.wait (nothing calls these earlier).  `ldu` is PTX's load of a
// warp-uniform read-only address; volatile so that the compiler neither hoists it above the wait nor keeps the value in a register
// across the tick (the step kernel holds 112 registers with no spills).
HD float ldu_slot(const float* p) { float v; asm volatile("ldu.global.f32 %0, [%1];" : "=f"(v) : "l"(p)); return v; }
HD double ldu_slot(const double* p) { double v; asm volatile("ldu.global.f64 %0, [%1];" : "=d"(v) : "l"(p)); return v; }
template <bool kCur, typename R> HD R cur_radius(const KernelArgs<R>& A) {
    if constexpr (kCur) return ldu_slot(&A.cur_dev->intercept_radius); else return A.C.intercept_radius;
}
template <bool kCur, typename R> HD float cur_cos_half_beam(const KernelArgs<R>& A) {
    if constexpr (kCur) return ldu_slot(&A.cur_dev->cos_half_beam); else return A.C.cos_half_beam;
}
template <bool kCur, typename R> HD float cur_onboard_rel(const KernelArgs<R>& A) {
    if constexpr (kCur) return ldu_slot(&A.cur_dev->onboard_rel); else return A.C.onboard_rel;
}
template <bool kCur, typename R> HD float cur_ground_rel(const KernelArgs<R>& A) {
    if constexpr (kCur) return ldu_slot(&A.cur_dev->ground_rel); else return A.C.ground_rel;
}

// ------------------------------------------------------------------------------------------------
// per-env register state
// ------------------------------------------------------------------------------------------------
template <typename R> struct Env {
    R ipx, ipy, ipz, fuel;
    R ivx, ivy, ivz, fuel_used;
    R mpx, mpy, mpz, prev_d;
    R mvx, mvy, mvz, last_d;
    R kpx, kpy, kpz, min_d;
    R kvx, kvy, kvz, ep_ret;
    R thx, thy, thz, T0;
    float qw, qx, qy, qz;
    float wx, wy, wz, Ppp;
    float Ppv, Pvp, Pvv, base_cd;
    float peak;
    int steps, worsen, flags, episode;
};
#define FLAG_CROSSED 1
#define FLAG_KF_INIT 2
#define FLAG_KF_F64 4   /* fp64 build: the reference's Kalman state array has become float64 (core.py:108) */
// flags word: bit 0 crossed, bit 1 kf_init, bit 2 kf state is float64 (fp64 build), bits 8-11 onboard delay (samples), bits 12-14 index of the priority missile
// (volley: which list entry self.missile_state aliases), bits 16-19 missiles intercepted so far (volley)
#define FLAG_ODELAY(f) (((f) >> 8) & 0xf)
#define FLAG_VCUR(f) (((f) >> 12) & 0x7)
#define FLAG_VCOUNT(f) (((f) >> 16) & 0xf)

// Compact layout (KernelArgs::compact; fp32 build, the cfg4 feature set FT_V2ON without domain randomization, max_steps < 65536):
// the two words that are constants there -- T0 in r6.w and the base Cd in f1.w -- carry the counters instead, so the i0 plane is
// never touched: 10 planes (160 B read + 160 B written per env-step) instead of 11.
//   r6.w = bits(steps | worsen << 16)          f1.w = bits(episode (25 bits, signed) | flags7 << 25)
//   flags7 = crossed | kf_init << 1 | kf_f64 << 2 | onboard delay << 3   (the volley fields of the flag word do not exist here)
// Limits that follow: steps and the worsening counter stay below 65536 (hlynr_create checks max_steps), the episode counter of an
// env wraps after 2^25 episodes (~3e10 ticks of one env; it only keys the Philox streams), and hlynr_import_state cannot set T0 /
// base Cd to anything but the constants the configuration implies (they are not state here).
HD int word_bits(float x) { return __float_as_int(x); }
HD int word_bits(double) { return 0; }
HD float bits_word(int x, float) { return __int_as_float(x); }
HD double bits_word(int, double) { return 0.0; }
// F = the kernel's feature set: only FT_V2ON (and the generic kernels, which serve every handle) can meet a compact handle, so the
// other specialised instantiations carry no trace of it
template <typename R, int F = FT_GENERIC> HD bool compact_layout(const KernelArgs<R>& A) {
    if constexpr (!std::is_same<R, float>::value || F == FT_V2OFF || F == FT_V2ON_DR) return false;
    else return A.compact == 1;
}
// Second compact layout (KernelArgs::compact == 2; fp32 build, cfg3's feature set FT_V2ON_DR, max_steps < 65536): with domain
// randomization T0 and the base Cd are real state, but the f3 plane holds ONE float (the transonic drag peak).  steps and the worsening
// counter share a word of i0, the peak takes the freed one, and the f3 plane is never touched: 11 planes instead of 12.
//   i0 = { steps | worsen << 16, bits(peak), flags, episode }
template <typename R, int F = FT_GENERIC> HD bool dr_compact_layout(const KernelArgs<R>& A) {
    if constexpr (!std::is_same<R, float>::value || F == FT_V2OFF || F == FT_V2ON) return false;
    else return A.compact == 2;
}

template <typename R, int F = FT_GENERIC> HD void load_env(const KernelArgs<R>& A, int64_t i, Env<R>& e) {
    typedef Feat<F> FT;
    const StatePlanes<R>& s = A.st;
    const bool compact = compact_layout<R, F>(A), drc = dr_compact_layout<R, F>(A);
    Vec4<R> v;
    float4 f;
    // Issue order = order of first use.  The planes that carry the counters go first: steps / episode key every Philox draw of the
    // tick, which is the first work a tick can do while the other planes are still in flight (cfg4 102.2 -> 100.6 us, cfg2 94.3 ->
    // 90.6 us against the former r0 ... r6, f0 ... f2, i0 order: profiles/r02_l_draws_early_ab.log); then the interceptor's planes,
    // the missile's, and the track filter's, which only observe() reads.
    int4 q = make_int4(0, 0, 0, 0);
    if (!compact) q = s.i0[i];
    if (compact || FT::thrust_dyn(A.P) || FT::dr(A.P)) { v = s.r[6][i]; e.thx = v.x; e.thy = v.y; e.thz = v.z; e.T0 = v.w; }
    else { e.thx = e.thy = e.thz = R(0); e.T0 = R(288.15); }
    f = s.f[1][i]; e.wx = f.x; e.wy = f.y; e.wz = f.z; e.base_cd = f.w;
    v = s.r[0][i]; e.ipx = v.x; e.ipy = v.y; e.ipz = v.z; e.fuel = v.w;
    v = s.r[1][i]; e.ivx = v.x; e.ivy = v.y; e.ivz = v.z; e.fuel_used = v.w;
    v = s.r[2][i]; e.mpx = v.x; e.mpy = v.y; e.mpz = v.z; e.prev_d = v.w;
    v = s.r[3][i]; e.mvx = v.x; e.mvy = v.y; e.mvz = v.z; e.last_d = v.w;
    v = s.r[4][i]; e.kpx = v.x; e.kpy = v.y; e.kpz = v.z; e.min_d = v.w;
    v = s.r[5][i]; e.kvx = v.x; e.kvy = v.y; e.kvz = v.z; e.ep_ret = v.w;
    f = s.f[0][i]; e.qw = f.x; e.qx = f.y; e.qy = f.z; e.qz = f.w;
    f = s.f[2][i]; e.Ppv = f.x; e.Pvp = f.y; e.Pvv = f.z; e.Ppp = f.w;
    if (FT::dr(A.P) && !drc) { f = s.f[3][i]; e.peak = f.x; } else e.peak = 0.f;
    if (compact) {
        const int sw = word_bits(e.T0), ef = word_bits(e.base_cd);
        e.T0 = R(288.15); e.base_cd = 0.3f;
        e.steps = sw & 0xffff; e.worsen = (int)((unsigned)sw >> 16);
        e.episode = (ef << 7) >> 7;
        const int p = (int)((unsigned)ef >> 25);
        e.flags = (p & 7) | (((p >> 3) & 0xf) << 8);
    } else if (drc) {
        e.steps = q.x & 0xffff; e.worsen = (int)((unsigned)q.x >> 16); e.peak = __int_as_float(q.y); e.flags = q.z; e.episode = q.w;
    } else {
        e.steps = q.x; e.worsen = q.y; e.flags = q.z; e.episode = q.w;
    }
}
template <typename R, int F = FT_GENERIC> HD void store_env(const KernelArgs<R>& A, int64_t i, const Env<R>& e) {
    typedef Feat<F> FT;
    const StatePlanes<R>& s = A.st;
    const bool compact = compact_layout<R, F>(A), drc = dr_compact_layout<R, F>(A);
    R r6w = e.T0;
    float f1w = e.base_cd;
    if (compact) {
        r6w = bits_word((e.steps & 0xffff) | (e.worsen << 16), R(0));
        f1w = __int_as_float((e.episode & 0x1ffffff) | (((e.flags & 7) | (((e.flags >> 8) & 0xf) << 3)) << 25));
    }
    s.r[0][i] = Vec4<R>{e.ipx, e.ipy, e.ipz, e.fuel};
    s.r[1][i] = Vec4<R>{e.ivx, e.ivy, e.ivz, e.fuel_used};
    s.r[2][i] = Vec4<R>{e.mpx, e.mpy, e.mpz, e.prev_d};
    s.r[3][i] = Vec4<R>{e.mvx, e.mvy, e.mvz, e.last_d};
    s.r[4][i] = Vec4<R>{e.kpx, e.kpy, e.kpz, e.min_d};
    s.r[5][i] = Vec4<R>{e.kvx, e.kvy, e.kvz, e.ep_ret};
    if (compact || FT::thrust_dyn(A.P) || FT::dr(A.P)) s.r[6][i] = Vec4<R>{e.thx, e.thy, e.thz, r6w};
    s.f[0][i] = make_float4(e.qw, e.qx, e.qy, e.qz);
    s.f[1][i] = make_float4(e.wx, e.wy, e.wz, f1w);
    s.f[2][i] = make_float4(e.Ppv, e.Pvp, e.Pvv, e.Ppp);
    if (FT::dr(A.P) && !drc) s.f[3][i] = make_float4(e.peak, 0.f, 0.f, 0.f);
    if (drc) s.i0[i] = make_int4((e.steps & 0xffff) | (e.worsen << 16), __float_as_int(e.peak), e.flags, e.episode);
    else if (!compact) s.i0[i] = make_int4(e.steps, e.worsen, e.flags, e.episode);
}

// ------------------------------------------------------------------------------------------------
// physics_models.py
// ------------------------------------------------------------------------------------------------
// AtmosphericModel.get_atmospheric_properties (physics_models.py:154-177)
// Hot / cold layout.  ptxas lays basic blocks out in source order, so a rarely taken `if` body in the middle of the tick is
// a taken branch over it on EVERY tick, and the instruction fetch after a taken branch is what the `no_instructions` stall
// samples of profiles/r01_e sit on (12 % of all samples in the steady state, almost all on reconvergence points).  The
// rare bodies below are therefore separate __noinline__ functions that return by value (no addresses taken), and short
// two-way choices are written branch-free where that is bit-identical.
template <typename R> struct Pair { R a, b; };
template <typename R> __device__ __noinline__ Pair<R> isa_above_11km(R alt) {  // physics_models.py:163-171
    Pair<R> o;
    if (alt <= R(20000.0)) {
        o.a = R(216.65);
        o.b = mul(R(22632.0), nexp(ndiv(mul(R(-9.80665), sub(alt, R(11000.0))), R(287.05 * 216.65))));
    } else {
        R ex = sub(alt, R(20000.0));
        o.a = mul(R(216.65), nexp(ndiv(-ex, R(10000.0))));
        o.b = mul(R(5474.790039909648), nexp(ndiv(-ex, R(6000.0))));  // get_pressure(20000.0) in python floats: 22632 exp(-g 9000 / (R 216.65))
    }
    return o;
}
// rho and cs within 1.3e-6 relative (fp32 build) / 11 ulp (fp64 build) of the float64 formula, worst measured on a B200
template <typename R> HD void isa_props(const KParams<R>& P, R T0, R alt, R* rho, R* cs) {
    R T, Pr;
    if (alt <= R(11000.0)) {
        T = sub(T0, mul(R(0.0065), alt));
        Pr = mul(R(101325.0), npow(ndiv(T, T0), P.isa_expo));
    } else {
        const Pair<R> hi = isa_above_11km<R>(alt);
        T = hi.a; Pr = hi.b;
    }
    *rho = ndiv(Pr, mul(P.gas_R, T));
    *cs = nsqrt(mul(P.gamma_R, T));
}

// Drag acceleration: MachDragModel.get_drag_force (physics_models.py:236-264) / mass, or the constant-Cd
// fallback (environment.py:920-921, :1099-1100).  F = -(v/|v|) * (0.5 rho |v|^2 Cd A) * post_scale.
// With domain randomization base_cd/peak are np.float64 scalars and the product is a float64 island
// (physics_randomizer.py:273,278); the fp32 build evaluates it in float.
template <typename R, int F>
HD void drag_accel(const KParams<R>& P, const Env<R>& e, R vx, R vy, R vz, R alt, R area, R post_scale, R rc_mass, R mass,
                   R* ax, R* ay, R* az) {
    typedef Feat<F> FT;
    R rho = P.rho_weak, cs = P.cs_weak;
    bool weak = true;
    if (FT::isa(P)) { isa_props(P, e.T0, alt, &rho, &cs); weak = false; }
    R vmag = nnorm3(vx, vy, vz);
    if (FT::mach(P) && vmag > R(1e-6)) {
        R mach = ndiv(vmag, cs);
        R cd;
        if (FT::dr(P)) {
            double bc = (double)e.base_cd, pk = (double)e.peak, c;
            // two selects in the reference's test order (exact for any parameters, also subsonic_mach > supersonic_mach)
            const R ramp = ndiv(sub(mach, P.sub_mach), P.sup_minus_sub);
            c = mach < P.sup_mach ? bc * (1.0 + (pk - 1.0) * (double)ramp) : bc * P.sup_mult_d;
            c = mach < P.sub_mach ? bc : c;
            cd = (R)c;
        } else {
            // branch-free: two selects in the reference's test order (exact for any parameters, also subsonic_mach > supersonic_mach)
            const R ramp = ndiv(sub(mach, P.sub_mach), P.sup_minus_sub);
            const R mid = mul(P.cd_base, add(R(1.0), mul(P.peak_minus1, ramp)));
            cd = mach < P.sup_mach ? mid : P.cd_sup;
            cd = mach < P.sub_mach ? P.cd_base : cd;
        }
        if constexpr (std::is_same<R, float>::value) {
            float k = -((weak ? P.half_rho_weak : 0.5f * rho) * vmag * cd * area * post_scale * rc_mass);
            *ax = k * vx; *ay = k * vy; *az = k * vz;
        } else {
            R t = weak ? P.half_rho_weak : mul(R(0.5), rho);
            t = mul(mul(mul(t, mul(vmag, vmag)), cd), area);
            R fx = mul(dvd(-vx, vmag), t), fy = mul(dvd(-vy, vmag), t), fz = mul(dvd(-vz, vmag), t);
            if (post_scale != R(1.0)) { fx = mul(fx, post_scale); fy = mul(fy, post_scale); fz = mul(fz, post_scale); }
            *ax = dvd(fx, mass); *ay = dvd(fy, mass); *az = dvd(fz, mass);
        }
    } else {
        R c = mul(weak ? P.nhcr_weak : mul(R(-0.5 * 0.3), rho), vmag);
        if constexpr (std::is_same<R, float>::value) { c *= rc_mass; *ax = c * vx; *ay = c * vy; *az = c * vz; }
        else { *ax = dvd(mul(c, vx), mass); *ay = dvd(mul(c, vy), mass); *az = dvd(mul(c, vz), mass); }
    }
}

// true iff any of the three is NaN or +-inf: 0 * x is NaN exactly for those (float); exponent test on the high words (double)
HD bool any_nonfinite(float a, float b, float c) { const float t = fmaf(a, 0.f, fmaf(b, 0.f, c * 0.f)); return t != t; }
HD bool any_nonfinite(double a, double b, double c) {
    const int e = max(max(__double2hiint(a) & 0x7ff00000, __double2hiint(b) & 0x7ff00000), __double2hiint(c) & 0x7ff00000);
    return e == 0x7ff00000;
}
template <typename R> HD R nan_guard(R a, R lim) {  // np.nan_to_num(nan=0, posinf=lim, neginf=-lim)
    if (a != a) return R(0);
    if (isinf(a)) return a > R(0) ? lim : -lim;
    return a;
}

template <typename R> struct Tri { R x, y, z; };
template <typename R> __device__ __noinline__ Tri<R> nan_guard3(R a, R b, R c, R lim) {
    return Tri<R>{nan_guard(a, lim), nan_guard(b, lim), nan_guard(c, lim)};
}
// SafetyClamp scaling (core.py:1085-1097): only reached when the squared norm exceeds the limit (never for actions in [-1, 1])
template <typename R> __device__ __noinline__ Vec4<R> clamp_norm_slow(R a, R b, R c, R lim) {
    const R m = norm3(a, b, c);
    if (m > lim) { const R f = dvd(lim, m); return Vec4<R>{mul(a, f), mul(b, f), mul(c, f), R(1)}; }
    return Vec4<R>{a, b, c, R(0)};
}
// full-range sine / cosine of the quaternion half-angle: actions outside [-1, 1] only
__device__ __noinline__ Pair<float> sincos_full(float h) { return Pair<float>{sinf(h), cosf(h)}; }
__device__ __noinline__ Pair<double> sincos_full_d(double h) { double s, c; sincos(h, &s, &c); return Pair<double>{s, c}; }

// The LOS basis shared by the observation (core.py:803-845, :929-945) and the action transform
// (environment.py:965-1020): lu = rel/|rel|, lh = normalize(lu x world_up) = (lu.y, -lu.x, 0)/n, lv = lu x lh.
template <typename T> struct LosBasis { T ux, uy, uz, hx, hy, vx, vy, vz; };  // lh.z == 0
template <typename T> HD LosBasis<T> los_basis_near(T px, T py, T pz, T rr) {
    LosBasis<T> b;
    if (rr > T(1e-6)) { const T ir = nrcp(rr); b.ux = px * ir; b.uy = py * ir; b.uz = pz * ir; }
    else { b.ux = T(1); b.uy = T(0); b.uz = T(0); }
    const T n = nsqrt(b.ux * b.ux + b.uy * b.uy);
    if (n > T(1e-6)) { const T in = nrcp(n); b.hx = b.uy * in; b.hy = -b.ux * in; }
    else { b.hx = T(1); b.hy = T(0); }
    b.vx = -(b.uz * b.hy); b.vy = b.uz * b.hx; b.vz = b.ux * b.hy - b.uy * b.hx;
    return b;
}

// Observation sink: channel k of this lane's row goes straight into the warp's shared-memory tile (row pitch 26
// words), so the 26 channels never occupy registers at the same time.  emit == false (non-final fused ticks)
// drops the stores and lets the compiler remove the channel arithmetic.
struct ObsOut {
    float* row;  // tile + lane * 26
    bool emit;
    bool onboard_det, ground_det;
    HD void put(int k, float v) const { if (emit) row[k] = v; }
};

// ------------------------------------------------------------------------------------------------
// Radar26DObservation.compute_radar_detection + compute (core.py:511-1032), world_frame.
// `tick` indexes the ring planes; `e.steps` is the call index since reset (0 = the reset call).
// Geometry is float32 in both builds (the reference casts the state to float32 on entry, core.py:522-529);
// W = R is the dtype of the reference's float64 islands (ground measurement, Kalman state).
// ------------------------------------------------------------------------------------------------
// fp64 build, float32 phase of the Kalman state (FLAG_KF_F64 clear): the reference evaluates the track-derived channels
// (core.py:779-918: filtered relative position / velocity, range, closing speed, LOS rates, time to intercept, off-axis cosine) in
// float32 because every operand is a float32 array.  Positions of ~1e4 m carry 5e-4 m of float32 rounding, which the LOS-rate and
// direction-cosine channels amplify by |v| / range to ~3e-5 -- above this build's 1e-5 tolerance -- so the phase is followed with
// the same correctly rounded float32 operations in the same order (oracle/hlynr_oracle.c observe(), pk == F32) instead of in double.
struct TrackF32 { float ux, uy, uz, hx, hy, hz, vx, vy, vz; bool have_los; };
template <typename R>
__device__ __noinline__ TrackF32 track_obs_f32_phase(const KParams<R>& P, int mode, bool o_det, float Ppp, float kpx, float kpy, float kpz,
                                                     float kvx, float kvy, float kvz, float ipx, float ipy, float ipz, float ivx, float ivy,
                                                     float ivz, float fx, float fy, float fz, float rx_, float ry_, float rz_, float ux_,
                                                     float uy_, float uz_, const ObsOut out) {
    TrackF32 lb{1.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 0.f, 0.f, false};
    const float mr = P.max_range_f, mv = P.max_velocity_f;   // weak Python scalars rounded to float32
    const float px = sub(kpx, ipx), py = sub(kpy, ipy), pz = sub(kpz, ipz);
    const float vx = sub(kvx, ivx), vy = sub(kvy, ivy), vz = sub(kvz, ivz);
    const float rr = norm3(px, py, pz);
    const float cl = dvd(-dot3(px, py, pz, vx, vy, vz), add(rr, 1e-6f));
    if (mode == HLYNR_OBS_LOS) {
        lb.have_los = true;
        out.put(0, clip(dvd(rr, mr), 0.f, 1.f));
        out.put(1, clip(dvd(cl, mv), -1.f, 1.f));
        if (rr > 1e-6f) { lb.ux = dvd(px, rr); lb.uy = dvd(py, rr); lb.uz = dvd(pz, rr); }
        {   // lh = normalize(lu x world_up), lv = lu x lh (oracle los_basis / cross3)
            const float cx = sub(mul(lb.uy, 1.f), mul(lb.uz, 0.f)), cy = sub(mul(lb.uz, 0.f), mul(lb.ux, 1.f)), cz = sub(mul(lb.ux, 0.f), mul(lb.uy, 0.f));
            const float n = norm3(cx, cy, cz);
            if (n > 1e-6f) { lb.hx = dvd(cx, n); lb.hy = dvd(cy, n); lb.hz = dvd(cz, n); }
            lb.vx = sub(mul(lb.uy, lb.hz), mul(lb.uz, lb.hy));
            lb.vy = sub(mul(lb.uz, lb.hx), mul(lb.ux, lb.hz));
            lb.vz = sub(mul(lb.ux, lb.hy), mul(lb.uy, lb.hx));
        }
        const float rden = add(rr, 1e-6f);
        const float tx = dvd(sub(vx, mul(cl, lb.ux)), rden), ty = dvd(sub(vy, mul(cl, lb.uy)), rden), tz = dvd(sub(vz, mul(cl, lb.uz)), rden);
        out.put(2, clip(dvd(dot3(tx, ty, tz, lb.hx, lb.hy, lb.hz), 0.5f), -1.f, 1.f));
        out.put(3, clip(dvd(dot3(tx, ty, tz, lb.vx, lb.vy, lb.vz), 0.5f), -1.f, 1.f));
        const float ivm = norm3(ivx, ivy, ivz);
        out.put(4, ivm > 1e-6f ? dot3(dvd(ivx, ivm), dvd(ivy, ivm), dvd(ivz, ivm), lb.ux, lb.uy, lb.uz) : 0.f);
        const float ax = add(vx, ivx), ay = add(vy, ivy), az = add(vz, ivz);
        const float am = norm3(ax, ay, az);
        out.put(5, am > 1e-6f ? dot3(dvd(ax, am), dvd(ay, am), dvd(az, am), -lb.ux, -lb.uy, -lb.uz) : 0.f);
    } else if (mode == HLYNR_OBS_BODY) {
        out.put(0, clip(dvd(dot3(px, py, pz, fx, fy, fz), mr), -1.f, 1.f));
        out.put(1, clip(dvd(dot3(px, py, pz, rx_, ry_, rz_), mr), -1.f, 1.f));
        out.put(2, clip(dvd(dot3(px, py, pz, ux_, uy_, uz_), mr), -1.f, 1.f));
        out.put(3, clip(dvd(dot3(vx, vy, vz, fx, fy, fz), mv), -1.f, 1.f));
        out.put(4, clip(dvd(dot3(vx, vy, vz, rx_, ry_, rz_), mv), -1.f, 1.f));
        out.put(5, clip(dvd(dot3(vx, vy, vz, ux_, uy_, uz_), mv), -1.f, 1.f));
    } else {
        out.put(0, clip(dvd(px, mr), -1.f, 1.f)); out.put(1, clip(dvd(py, mr), -1.f, 1.f)); out.put(2, clip(dvd(pz, mr), -1.f, 1.f));
        out.put(3, clip(dvd(vx, mv), -1.f, 1.f)); out.put(4, clip(dvd(vy, mv), -1.f, 1.f)); out.put(5, clip(dvd(vz, mv), -1.f, 1.f));
    }
    out.put(13, cl > 0.f ? clip(sub(1.f, dvd(dvd(rr, cl), 100.f)), -1.f, 1.f) : -1.f);
    {   // np.trace(P[0:3,0:3]) in float32, then python-float arithmetic (core.py:899-905)
        const float tr = add(add(Ppp, Ppp), Ppp);
        double tq = clip(1.0 - (double)tr / 10000.0, 0.0, 1.0);
        if (o_det) tq *= P.radar_quality_d;
        out.put(14, (float)tq);
    }
    out.put(15, clip(dvd(cl, mv), -1.f, 1.f));
    out.put(16, rr > 1e-6f ? dot3(fx, fy, fz, dvd(px, rr), dvd(py, rr), dvd(pz, rr)) : 1.f);
    return lb;
}

// Pieces of the observation that depend on the interceptor state only.
// forward vector, core.py:1143-1152
HD void forward_vec(float w, float x, float y, float z, float* fx, float* fy, float* fz) {
    float a = 2.f * fmaf(x, z, w * y), b = 2.f * fmaf(y, z, -(w * x)), c = 1.f - 2.f * fmaf(x, x, y * y);
    float inv = nrcp(nnorm3(a, b, c) + 1e-6f);
    *fx = a * inv; *fy = b * inv; *fz = c * inv;
}
// datalink quality, core.py:440-474 (urw = the tick's packet-loss draw)
template <typename R>
HD float datalink_quality(const KParams<R>& P, float ipx, float ipy, float ipz, float ivx, float ivy, float ivz, uint32_t urw) {
    float link = 0.f;
    float lr = nnorm3(ipx - P.gpos[0], ipy - P.gpos[1], ipz - P.gpos[2]);
    if (!(lr > P.max_link)) {
        float r1 = lr * P.rc_max_link;
        float dop = 1.f - fminf(nnorm3(ivx, ivy, ivz) * 1e-3f, 0.3f);
        if (u01(urw) < P.pkt_loss) link = 0.f;
        else link = clip((1.f - r1 * r1) * dop * 0.95f, 0.f, 1.f);
    }
    return link;
}
// quaternion_to_euler / pi, core.py:1103-1121 (float32): observation channels 9-11 of the world frame
HD void euler_over_pi(float w, float x, float y, float z, float* roll, float* pitch, float* yaw) {
    const float sinr = 2.f * fmaf(w, x, y * z), cosr = 1.f - 2.f * fmaf(x, x, y * y);
    const float sinp = 2.f * fmaf(w, y, -(z * x));
    const float siny = 2.f * fmaf(w, z, x * y), cosy = 1.f - 2.f * fmaf(y, y, z * z);
    const float ipi = 0.318309886183790672f;
    *roll = fast_atan2(sinr, cosr) * ipi;
    *pitch = fast_asin(clip(sinp, -1.f, 1.f)) * ipi;
    *yaw = fast_atan2(siny, cosy) * ipi;
}
template <typename R, int F, bool kCur = false>
HD void observe(const KernelArgs<R>& A, Env<R>& e, const RngKey& key, const uint4 ur, int64_t i, int g_row, int o_row, ObsOut& out) {
    typedef R W;
    typedef Feat<F> FT;
    const KParams<R>& P = A.P;
    const int64_t n = A.ring_stride;
    const float ipx = (float)e.ipx, ipy = (float)e.ipy, ipz = (float)e.ipz;
    const float ivx = (float)e.ivx, ivy = (float)e.ivy, ivz = (float)e.ivz;
    const float mpx = (float)e.mpx, mpy = (float)e.mpy, mpz = (float)e.mpz;
    // ur = the tick's BLK_UNI block (x gust, y onboard dropout, z ground dropout, w packet loss)

    // === onboard radar, core.py:531-593 ===
    const float rx = sub(mpx, ipx), ry = sub(mpy, ipy), rz = sub(mpz, ipz);
    const float range = nnorm3(rx, ry, rz);
    float fx, fy, fz;
    forward_vec(e.qw, e.qx, e.qy, e.qz, &fx, &fy, &fz);
    bool onb = !(range > P.radar_range);
    if (onb) {
        float cb = ndot3(fx, fy, fz, rx, ry, rz) * nrcp(range + 1e-6f);
        if (cb < cur_cos_half_beam<kCur>(A)) onb = false;  // acos(clip(cb)) > radians(beam/2), core.py:547-553
    }
    if (onb) {
        float q = P.radar_quality * (1.f - range * P.rc_radar_range * 0.5f) * cur_onboard_rel<kCur>(A);
        if (u01(ur.y) > q) onb = false;
    }
    float orx, ory, orz;
    bool o_det;
    if (FT::onboard_delay(P)) {
        const int L = P.onb_ring_len;
        const int odelay = FLAG_ODELAY(e.flags);
        A.st.oring[(int64_t)o_row * n + i] = make_float4(rx, ry, rz, onb ? 1.f : 0.f);
        if (e.steps >= odelay) {
            int rrow = o_row - odelay;  // sample written `odelay` ticks ago
            if (rrow < 0) rrow += L;
            const float4 s = A.st.oring[(int64_t)rrow * n + i];
            orx = s.x; ory = s.y; orz = s.z; o_det = s.w != 0.f;
        } else { orx = ory = orz = 0.f; o_det = false; }
    } else { orx = rx; ory = ry; orz = rz; o_det = onb; }

    // === ground radar, core.py:368-438 ===
    bool gdet = false;
    W grx = W(0), gry = W(0), grz = W(0), gvx = W(0), gvy = W(0), gvz = W(0);
    float gq = 0.f;
    if (FT::ground(P)) {
        float gx = mpx - P.gpos[0], gy = mpy - P.gpos[1], gz = mpz - P.gpos[2];
        float gr = nnorm3(gx, gy, gz);
        bool ok = !(gr > P.g_max_range);
        if (ok && gr > 1e-6f) {  // elevation gates: asin(s) < min  <=>  s < sin(min)
            float se = gz * nrcp(gr);
            if (se < P.g_sin_min_el || se > P.g_sin_max_el) ok = false;
        }
        if (ok && mpz < 50.f) ok = false;
        if (ok) {
            float prob = P.g_base_q * (1.f - gr * P.rc_g_max_range * 0.4f) * cur_ground_rel<kCur>(A);
            if (u01(ur.z) > prob) ok = false;
            else {
                float z0, z1, z2, y0, y1, y2;
                draw_normal3(key, (uint32_t)e.episode, (uint32_t)e.steps, HLYNR_BLK_GPOS, &z0, &z1, &z2);
                draw_normal3(key, (uint32_t)e.episode, (uint32_t)e.steps, HLYNR_BLK_GVEL, &y0, &y1, &y2);
                const float mvx = (float)e.mvx, mvy = (float)e.mvy, mvz = (float)e.mvz;
                grx = (W)rx + P.sigma_r * (W)z0; gry = (W)ry + P.sigma_r * (W)z1; grz = (W)rz + P.sigma_r * (W)z2;
                gvx = (W)sub(mvx, ivx) + P.sigma_v * (W)y0;
                gvy = (W)sub(mvy, ivy) + P.sigma_v * (W)y1;
                gvz = (W)sub(mvz, ivz) + P.sigma_v * (W)y2;
                gq = prob; gdet = true;
            }
        }
    }
    W dgx, dgy, dgz, dvx, dvy, dvz;
    float dgq;
    bool dg_det;
    bool dg_f64 = gdet;  // the measurement arrays are float64 iff they hold a detected sample (float32 geometry + float64 noise)
    if (FT::ground(P) && FT::ground_delay(P)) {  // delayed values, CURRENT flag (core.py:626, quirk Q3)
        const int L = P.gnd_ring_len;
        Vec4<W>* wr = A.st.gring + (int64_t)g_row * 2 * n;
        wr[i] = Vec4<W>{grx, gry, grz, (W)gq};
        wr[n + i] = Vec4<W>{gvx, gvy, gvz, gdet ? W(1) : W(0)};   // .w: the sample is a detection (dtype of the reference's arrays)
        if (e.steps >= P.ground_delay) {
            const int rrow = g_row + 1 == L ? 0 : g_row + 1;  // oldest slot = written ground_delay ticks ago
            const Vec4<W>* rr = A.st.gring + (int64_t)rrow * 2 * n;
            const Vec4<W> a = rr[i], b = rr[n + i];
            dgx = a.x; dgy = a.y; dgz = a.z; dgq = (float)a.w; dvx = b.x; dvy = b.y; dvz = b.z;
            dg_det = gdet; dg_f64 = b.w != W(0);
        } else { dgx = dgy = dgz = dvx = dvy = dvz = W(0); dgq = 0.f; dg_det = false; }
    } else { dgx = grx; dgy = gry; dgz = grz; dvx = gvx; dvy = gvy; dvz = gvz; dgq = gq; dg_det = gdet; }

    // === datalink, core.py:440-474 ===
    float link = 0.f;
    if (FT::ground(P)) link = datalink_quality(P, ipx, ipy, ipz, ivx, ivy, ivz, ur.w);

    // fp32 build, world frame: the channels that depend on the interceptor alone (own velocity, euler angles, fuel) are emitted
    // HERE, between the issue of the delayed ring loads and the first use of their samples (fusion, Kalman filter): ~100 independent
    // instructions behind which part of that latency hides (-0.9 ... -1.2 us per launch on cfg2 / cfg3 / cfg4; the fp64 build, bound by
    // instruction fetch, loses 3.7 us with the same move and keeps them at the end; profiles/r02_l_own_channels_ab.log)
    constexpr bool kOwnEarly = std::is_same<R, float>::value;
    if (kOwnEarly && FT::obs_mode(P) == HLYNR_OBS_WORLD) {
        out.put(6, clip(ivx * P.rc_max_velocity_f, -1.f, 1.f));
        out.put(7, clip(ivy * P.rc_max_velocity_f, -1.f, 1.f));
        out.put(8, clip(ivz * P.rc_max_velocity_f, -1.f, 1.f));
        if (out.emit) {
            float roll, pitch, yaw;
            euler_over_pi(e.qw, e.qx, e.qy, e.qz, &roll, &pitch, &yaw);
            out.put(9, roll); out.put(10, pitch); out.put(11, yaw);
        }
        out.put(12, clip((float)e.fuel * 0.01f, 0.f, 1.f));
    }
    // === fusion confidence, core.py:476-509 ===
    float fus;
    if (!o_det && !dg_det) fus = 0.f;
    else if (o_det && !dg_det) fus = (float)(P.radar_quality_d * 0.5);
    else if (!o_det) fus = dgq * 0.6f;
    else {
        W perr = nnorm3((W)orx - dgx, (W)ory - dgy, (W)orz - dgz);
        W r = perr * W(0.005);
        W agr = W(1.0) - (r < W(1.0) ? r : W(1.0));
        fus = (float)clip((W)(P.fus_035q + 0.5f * dgq) + W(0.15) * agr, W(0.0), W(1.0));
    }
    out.onboard_det = o_det;
    out.ground_det = dg_det;

    // === Kalman filter (core.py:12-133) reduced to x[6] + one shared 2x2 covariance block ===
    // dtype of self.state in the reference: float32 from reset() / initialize() until the first update() with a float64
    // measurement (any measurement that contains a DETECTED ground sample: float32 geometry + float64 noise, core.py:424-428),
    // float64 from then on (`self.state = self.state + K @ y` rebinds the array).  P, K, F, Q stay float32 throughout.
    // The fp64 build reproduces the switch (FLAG_KF_F64); the fp32 build keeps the state in float (documented deviation,
    // below its rtol 1e-3: the reference's float64 phase is then followed in float32).
    bool kf_init = (e.flags & FLAG_KF_INIT) != 0;
    if constexpr (std::is_same<R, double>::value) {
        bool x64 = (e.flags & FLAG_KF_F64) != 0;
        if (o_det || dg_det) {
            const bool z64 = dg_det && dg_f64;
            double zx, zy, zz;
            const float ow = P.radar_quality;
            if (o_det && dg_det) {  // quality-weighted fusion, core.py:734-739; total_weight is float32
                const float tw = add(ow, dgq);
                if (z64) {
                    zx = add((double)ipx, dvd(add((double)mul(orx, ow), mul(dgx, (double)dgq)), (double)tw));
                    zy = add((double)ipy, dvd(add((double)mul(ory, ow), mul(dgy, (double)dgq)), (double)tw));
                    zz = add((double)ipz, dvd(add((double)mul(orz, ow), mul(dgz, (double)dgq)), (double)tw));
                } else {            // the delayed ground sample is the float32 zero placeholder of a non-detection
                    zx = (double)add(ipx, dvd(add(mul(orx, ow), mul((float)dgx, dgq)), tw));
                    zy = (double)add(ipy, dvd(add(mul(ory, ow), mul((float)dgy, dgq)), tw));
                    zz = (double)add(ipz, dvd(add(mul(orz, ow), mul((float)dgz, dgq)), tw));
                }
            } else if (o_det) {
                zx = (double)add(ipx, orx); zy = (double)add(ipy, ory); zz = (double)add(ipz, orz);
            } else if (z64) {
                zx = add((double)ipx, dgx); zy = add((double)ipy, dgy); zz = add((double)ipz, dgz);
            } else {
                zx = (double)add(ipx, (float)dgx); zy = (double)add(ipy, (float)dgy); zz = (double)add(ipz, (float)dgz);
            }
            if (!kf_init) {  // first measurement only initialises (core.py:93-96): assignment into the float32 state array
                e.kpx = (double)(float)zx; e.kpy = (double)(float)zy; e.kpz = (double)(float)zz;
                e.kvx = e.kvy = e.kvz = 0.0;
                kf_init = true;
            } else {
                const float Si = dvd(1.f, add(e.Ppp, 400.f));   // inv(S): exact reciprocal of the diagonal innovation block
                const float Kp = mul(e.Ppp, Si), Kv = mul(e.Pvp, Si);
                if (x64 || z64) {   // state = state + K @ y in float64
                    const double yx = sub(zx, e.kpx), yy = sub(zy, e.kpy), yz = sub(zz, e.kpz);
                    e.kpx = add(e.kpx, mul((double)Kp, yx)); e.kpy = add(e.kpy, mul((double)Kp, yy)); e.kpz = add(e.kpz, mul((double)Kp, yz));
                    e.kvx = add(e.kvx, mul((double)Kv, yx)); e.kvy = add(e.kvy, mul((double)Kv, yy)); e.kvz = add(e.kvz, mul((double)Kv, yz));
                    x64 = true;
                } else {            // ... in float32
                    const float yx = sub((float)zx, (float)e.kpx), yy = sub((float)zy, (float)e.kpy), yz = sub((float)zz, (float)e.kpz);
                    e.kpx = (double)add((float)e.kpx, mul(Kp, yx)); e.kpy = (double)add((float)e.kpy, mul(Kp, yy));
                    e.kpz = (double)add((float)e.kpz, mul(Kp, yz));
                    e.kvx = (double)add((float)e.kvx, mul(Kv, yx)); e.kvy = (double)add((float)e.kvy, mul(Kv, yy));
                    e.kvz = (double)add((float)e.kvz, mul(Kv, yz));
                }
                // P = (I - K H) @ P, float32, sgemm accumulation order (FMA chain over k, oracle matmul66)
                const float a = sub(1.f, Kp);
                const float npp = mul(a, e.Ppp), npv = mul(a, e.Ppv);
                const float nvp = add(mul(-Kv, e.Ppp), e.Pvp), nvv = add(mul(-Kv, e.Ppv), e.Pvv);
                e.Ppp = npp; e.Ppv = npv; e.Pvp = nvp; e.Pvv = nvv;
            }
        } else if (kf_init) {  // predict only when no measurement (quirk Q4)
            if (x64) {
                const double d = (double)P.dtf;
                e.kpx = add(e.kpx, mul(d, e.kvx)); e.kpy = add(e.kpy, mul(d, e.kvy)); e.kpz = add(e.kpz, mul(d, e.kvz));
            } else {
                e.kpx = (double)add((float)e.kpx, mul(P.dtf, (float)e.kvx)); e.kpy = (double)add((float)e.kpy, mul(P.dtf, (float)e.kvy));
                e.kpz = (double)add((float)e.kpz, mul(P.dtf, (float)e.kvz));
            }
            const float fpp = __fmaf_rn(P.dtf, e.Pvp, e.Ppp), fpv = __fmaf_rn(P.dtf, e.Pvv, e.Ppv);  // F @ P
            const float cpp = __fmaf_rn(fpv, P.dtf, fpp), cvp = __fmaf_rn(e.Pvv, P.dtf, e.Pvp);      // (F P) @ F^T
            e.Ppp = add(cpp, P.q_pp); e.Ppv = add(fpv, P.q_pv); e.Pvp = add(cvp, P.q_pv); e.Pvv = add(e.Pvv, P.q_vv);
        }
        e.flags = (e.flags & ~(FLAG_KF_INIT | FLAG_KF_F64)) | (kf_init ? FLAG_KF_INIT : 0) | (x64 ? FLAG_KF_F64 : 0);
    } else {
    if (o_det || dg_det) {
        W zx, zy, zz;
        if (o_det && dg_det) {  // quality-weighted fusion, core.py:734-739
            const float ow = P.radar_quality;
            const W itw = nrcp((W)(ow + dgq));
            zx = (W)ipx + ((W)(orx * ow) + dgx * (W)dgq) * itw;
            zy = (W)ipy + ((W)(ory * ow) + dgy * (W)dgq) * itw;
            zz = (W)ipz + ((W)(orz * ow) + dgz * (W)dgq) * itw;
        } else if (o_det) {
            zx = (W)add(ipx, orx); zy = (W)add(ipy, ory); zz = (W)add(ipz, orz);
        } else {
            zx = (W)ipx + dgx; zy = (W)ipy + dgy; zz = (W)ipz + dgz;
        }
        if (!kf_init) {  // first measurement only initialises (core.py:93-96), state array is float32
            e.kpx = (W)(float)zx; e.kpy = (W)(float)zy; e.kpz = (W)(float)zz;
            e.kvx = e.kvy = e.kvz = W(0);
            kf_init = true;
        } else {
            const float Si = nrcp(e.Ppp + 400.f);
            const float Kp = e.Ppp * Si, Kv = e.Pvp * Si;
            const W yx = zx - e.kpx, yy = zy - e.kpy, yz = zz - e.kpz;
            e.kpx += (W)Kp * yx; e.kpy += (W)Kp * yy; e.kpz += (W)Kp * yz;
            e.kvx += (W)Kv * yx; e.kvy += (W)Kv * yy; e.kvz += (W)Kv * yz;
            const float a = 1.f - Kp;  // P = (I - K H) P
            const float npp = a * e.Ppp, npv = a * e.Ppv;
            const float nvp = fmaf(-Kv, e.Ppp, e.Pvp), nvv = fmaf(-Kv, e.Ppv, e.Pvv);
            e.Ppp = npp; e.Ppv = npv; e.Pvp = nvp; e.Pvv = nvv;
        }
    } else if (kf_init) {  // predict only when no measurement (quirk Q4)
        const W d = (W)P.dtf;
        e.kpx += d * e.kvx; e.kpy += d * e.kvy; e.kpz += d * e.kvz;
        const float fpp = fmaf(P.dtf, e.Pvp, e.Ppp), fpv = fmaf(P.dtf, e.Pvv, e.Ppv);  // F @ P
        const float cpp = fmaf(fpv, P.dtf, fpp), cvp = fmaf(e.Pvv, P.dtf, e.Pvp);      // (F P) @ F^T
        e.Ppp = cpp + P.q_pp; e.Ppv = fpv + P.q_pv; e.Pvp = cvp + P.q_pv; e.Pvv = e.Pvv + P.q_vv;
    }
    e.flags = (e.flags & ~FLAG_KF_INIT) | (kf_init ? FLAG_KF_INIT : 0);
    }

    const int mode = FT::obs_mode(P);
    LosBasis<W> lb;
    bool have_los = false;
    struct { float rx, ry, rz, ux, uy, uz; } bx = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // body right / up axes (core.py:1155-1176), body_frame only
    if (mode == HLYNR_OBS_BODY) {
        const float w = e.qw, x = e.qx, y = e.qy, z = e.qz;
        float a = 1.f - 2.f * fmaf(y, y, z * z), b = 2.f * fmaf(x, y, w * z), c = 2.f * fmaf(x, z, -(w * y));
        float inv = nrcp(nnorm3(a, b, c) + 1e-6f);
        bx.rx = a * inv; bx.ry = b * inv; bx.rz = c * inv;
        a = 2.f * fmaf(x, y, -(w * z)); b = 1.f - 2.f * fmaf(x, x, z * z); c = 2.f * fmaf(y, z, w * x);
        inv = nrcp(nnorm3(a, b, c) + 1e-6f);
        bx.ux = a * inv; bx.uy = b * inv; bx.uz = c * inv;
    }
    bool f32_phase = false;
    if constexpr (std::is_same<R, double>::value) f32_phase = kf_init && !(e.flags & FLAG_KF_F64);
    if (f32_phase) {
        if constexpr (std::is_same<R, double>::value) {
            const TrackF32 t = track_obs_f32_phase<R>(P, mode, o_det, e.Ppp, (float)e.kpx, (float)e.kpy, (float)e.kpz, (float)e.kvx,
                                                      (float)e.kvy, (float)e.kvz, ipx, ipy, ipz, ivx, ivy, ivz, fx, fy, fz, bx.rx, bx.ry, bx.rz,
                                                      bx.ux, bx.uy, bx.uz, out);
            have_los = t.have_los;   // channels 7 / 8 of the los_frame (core.py:929-945) project the interceptor velocity on this basis
            lb.ux = t.ux; lb.uy = t.uy; lb.uz = t.uz; lb.hx = t.hx; lb.hy = t.hy; lb.vx = t.vx; lb.vy = t.vy; lb.vz = t.vz;
        }
    } else if (kf_init) {
        const W px = e.kpx - (W)ipx, py = e.kpy - (W)ipy, pz = e.kpz - (W)ipz;
        const W vx = e.kvx - (W)ivx, vy = e.kvy - (W)ivy, vz = e.kvz - (W)ivz;
        const W rr = nnorm3(px, py, pz);
        const W cl = -ndot3(px, py, pz, vx, vy, vz) * nrcp(rr + W(1e-6));
        if (mode == HLYNR_OBS_LOS) {  // core.py:791-872
            lb = los_basis_near<W>(px, py, pz, rr);
            have_los = true;
            out.put(0, (float)clip(rr * P.rc_max_range_w, W(0), W(1)));
            out.put(1, (float)clip(cl * P.rc_max_velocity_w, W(-1), W(1)));
            const W ird = nrcp(rr + W(1e-6));
            const W tx = (vx - cl * lb.ux) * ird, ty = (vy - cl * lb.uy) * ird, tz = (vz - cl * lb.uz) * ird;  // LOS rate vector
            out.put(2, (float)clip((tx * lb.hx + ty * lb.hy) * W(2), W(-1), W(1)));                 // / max_los_rate 0.5
            out.put(3, (float)clip(ndot3(tx, ty, tz, lb.vx, lb.vy, lb.vz) * W(2), W(-1), W(1)));
            const float ivm = nnorm3(ivx, ivy, ivz);
            out.put(4, ivm > 1e-6f ? (float)(ndot3((W)ivx, (W)ivy, (W)ivz, lb.ux, lb.uy, lb.uz) * (W)nrcp(ivm)) : 0.f);
            const W ax = vx + (W)ivx, ay = vy + (W)ivy, az = vz + (W)ivz;  // approximate target velocity
            const W am = nnorm3(ax, ay, az);
            out.put(5, am > W(1e-6) ? (float)(-ndot3(ax, ay, az, lb.ux, lb.uy, lb.uz) * nrcp(am)) : 0.f);
        } else if (mode == HLYNR_OBS_BODY) {  // core.py:874-880: np.dot against the float32 body axes, float32 result
            const float b0 = (float)ndot3(px, py, pz, (W)fx, (W)fy, (W)fz), b1 = (float)ndot3(px, py, pz, (W)bx.rx, (W)bx.ry, (W)bx.rz);
            const float b2 = (float)ndot3(px, py, pz, (W)bx.ux, (W)bx.uy, (W)bx.uz);
            const float c0 = (float)ndot3(vx, vy, vz, (W)fx, (W)fy, (W)fz), c1 = (float)ndot3(vx, vy, vz, (W)bx.rx, (W)bx.ry, (W)bx.rz);
            const float c2 = (float)ndot3(vx, vy, vz, (W)bx.ux, (W)bx.uy, (W)bx.uz);
            out.put(0, clip(b0 * P.rc_max_range_f, -1.f, 1.f)); out.put(1, clip(b1 * P.rc_max_range_f, -1.f, 1.f));
            out.put(2, clip(b2 * P.rc_max_range_f, -1.f, 1.f));
            out.put(3, clip(c0 * P.rc_max_velocity_f, -1.f, 1.f)); out.put(4, clip(c1 * P.rc_max_velocity_f, -1.f, 1.f));
            out.put(5, clip(c2 * P.rc_max_velocity_f, -1.f, 1.f));
        } else {
        out.put(0, (float)clip(px * P.rc_max_range_w, W(-1), W(1)));
        out.put(1, (float)clip(py * P.rc_max_range_w, W(-1), W(1)));
        out.put(2, (float)clip(pz * P.rc_max_range_w, W(-1), W(1)));
        out.put(3, (float)clip(vx * P.rc_max_velocity_w, W(-1), W(1)));
        out.put(4, (float)clip(vy * P.rc_max_velocity_w, W(-1), W(1)));
        out.put(5, (float)clip(vz * P.rc_max_velocity_w, W(-1), W(1)));
        }
        out.put(13, cl > W(0) ? (float)clip(W(1) - rr * nrcp(cl) * W(0.01), W(-1), W(1)) : -1.f);
        float tq = clip(fmaf(e.Ppp * 3.f, -1e-4f, 1.f), 0.f, 1.f);   // explicit fma: the contraction must not depend on the surrounding code
        if (o_det) tq *= P.radar_quality;
        out.put(14, tq);
        out.put(15, (float)clip(cl * P.rc_max_velocity_w, W(-1), W(1)));
        out.put(16, rr > W(1e-6) ? (float)(ndot3((W)fx, (W)fy, (W)fz, px, py, pz) * nrcp(rr)) : 1.f);
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) out.put(k, -2.f);
        out.put(13, -1.f); out.put(14, 0.f); out.put(15, 0.f); out.put(16, 0.f);
    }
    if (mode == HLYNR_OBS_LOS) {  // core.py:920-958
        out.put(6, clip(nnorm3(ivx, ivy, ivz) * P.rc_max_velocity_f, 0.f, 1.f));
        if (have_los) {
            out.put(7, (float)clip(((W)ivx * lb.hx + (W)ivy * lb.hy) * P.rc_max_velocity_w, W(-1), W(1)));
            out.put(8, (float)clip(ndot3((W)ivx, (W)ivy, (W)ivz, lb.vx, lb.vy, lb.vz) * P.rc_max_velocity_w, W(-1), W(1)));
        } else { out.put(7, 0.f); out.put(8, 0.f); }
    } else if (mode == HLYNR_OBS_BODY) {  // :959-962
        out.put(6, clip(ndot3(ivx, ivy, ivz, fx, fy, fz) * P.rc_max_velocity_f, -1.f, 1.f));
        out.put(7, clip(ndot3(ivx, ivy, ivz, bx.rx, bx.ry, bx.rz) * P.rc_max_velocity_f, -1.f, 1.f));
        out.put(8, clip(ndot3(ivx, ivy, ivz, bx.ux, bx.uy, bx.uz) * P.rc_max_velocity_f, -1.f, 1.f));
    } else if (!kOwnEarly) {
    out.put(6, clip(ivx * P.rc_max_velocity_f, -1.f, 1.f));
    out.put(7, clip(ivy * P.rc_max_velocity_f, -1.f, 1.f));
    out.put(8, clip(ivz * P.rc_max_velocity_f, -1.f, 1.f));
    }
    if (mode != HLYNR_OBS_WORLD) { out.put(9, 0.f); out.put(10, 0.f); out.put(11, 0.f); }  // core.py:966-970
    else if (!kOwnEarly && out.emit) {
        float roll, pitch, yaw;
        euler_over_pi(e.qw, e.qx, e.qy, e.qz, &roll, &pitch, &yaw);
        out.put(9, roll); out.put(10, pitch); out.put(11, yaw);
    }
    if (!kOwnEarly || mode != HLYNR_OBS_WORLD) out.put(12, clip((float)e.fuel * 0.01f, 0.f, 1.f));
    if (dg_det && link > 0.1f && mode == HLYNR_OBS_LOS) {  // core.py:985-1006: redundant range / rate measurements
        const W gr = nnorm3(dgx, dgy, dgz);
        const W gc = -ndot3(dgx, dgy, dgz, dvx, dvy, dvz) * nrcp(gr + W(1e-6));
        out.put(17, (float)clip(gr * P.rc_max_range_w, W(0), W(1)));
        out.put(18, (float)clip(gc * P.rc_max_velocity_w, W(-1), W(1)));
        if (gr > W(1e-6)) {
            const W ig = nrcp(gr);
            const W k = gc * ig;
            out.put(19, (float)clip(nnorm3(dvx - k * dgx, dvy - k * dgy, dvz - k * dgz) * ig * W(2), W(0), W(1)));
        } else out.put(19, 0.f);
        out.put(20, 0.f); out.put(21, 0.f); out.put(22, 0.f);
        out.put(23, dgq);
    } else if (dg_det && link > 0.1f && mode == HLYNR_OBS_BODY) {  // :1008-1012
        out.put(17, clip((float)ndot3(dgx, dgy, dgz, (W)fx, (W)fy, (W)fz) * P.rc_max_range_f, -1.f, 1.f));
        out.put(18, clip((float)ndot3(dgx, dgy, dgz, (W)bx.rx, (W)bx.ry, (W)bx.rz) * P.rc_max_range_f, -1.f, 1.f));
        out.put(19, clip((float)ndot3(dgx, dgy, dgz, (W)bx.ux, (W)bx.uy, (W)bx.uz) * P.rc_max_range_f, -1.f, 1.f));
        out.put(20, clip((float)ndot3(dvx, dvy, dvz, (W)fx, (W)fy, (W)fz) * P.rc_max_velocity_f, -1.f, 1.f));
        out.put(21, clip((float)ndot3(dvx, dvy, dvz, (W)bx.rx, (W)bx.ry, (W)bx.rz) * P.rc_max_velocity_f, -1.f, 1.f));
        out.put(22, clip((float)ndot3(dvx, dvy, dvz, (W)bx.ux, (W)bx.uy, (W)bx.uz) * P.rc_max_velocity_f, -1.f, 1.f));
        out.put(23, dgq);
    } else if (dg_det && link > 0.1f) {
        out.put(17, (float)clip(dgx * P.rc_max_range_w, W(-1), W(1)));
        out.put(18, (float)clip(dgy * P.rc_max_range_w, W(-1), W(1)));
        out.put(19, (float)clip(dgz * P.rc_max_range_w, W(-1), W(1)));
        out.put(20, (float)clip(dvx * P.rc_max_velocity_w, W(-1), W(1)));
        out.put(21, (float)clip(dvy * P.rc_max_velocity_w, W(-1), W(1)));
        out.put(22, (float)clip(dvz * P.rc_max_velocity_w, W(-1), W(1)));
        out.put(23, dgq);
    } else {
#pragma unroll
        for (int k = 17; k < 23; ++k) out.put(k, -2.f);
        out.put(23, 0.f);
    }
    out.put(24, link);
    out.put(25, fus);
}

// ------------------------------------------------------------------------------------------------
// reset (environment.py:353-603).  Rare path: double arithmetic where the reference has float64.
// ------------------------------------------------------------------------------------------------
// The draws and the float64 geometry live in an out-of-line function that RETURNS its results by value, so the
// (rare) reset path is the only code that touches the stack and the env state never has its address taken.
struct SpawnOut {
    float mx, my, mz, mvx, mvy, mvz, ix, iy, iz, vx, vy, vz, qw, qx, qy, qz, d0;
    float base_cd, peak;
    double dT0;
    int odelay;
    uint4 ur;  // BLK_UNI of step 0 of the new episode (the observation of the reset), drawn here to keep the call site short
};

// one missile's spawn (environment.py:389-427) from its uniform block
template <typename R>
HD void spawn_missile(const KParams<R>& P, const uint4 r, float* mx, float* my, float* mz, float* vx, float* vy, float* vz) {
    const double u0 = u01(r.x), u1 = u01(r.y), u2 = u01(r.z), u3 = u01(r.w);
    if (P.spherical) {  // :390-406
        double radius = P.m_radius_lo + (P.m_radius_hi - P.m_radius_lo) * u0;
        double az = (P.m_az_lo + (P.m_az_hi - P.m_az_lo) * u1) * CUDART_PI / 180.0;
        double el = (P.m_el_lo + (P.m_el_hi - P.m_el_lo) * u2) * CUDART_PI / 180.0;
        *mx = (float)(P.target_d[0] + radius * cos(el) * cos(az));
        *my = (float)(P.target_d[1] + radius * cos(el) * sin(az));
        *mz = (float)(P.target_d[2] + radius * sin(el));
    } else {            // :409
        *mx = (float)(P.m_pos_lo[0] + (P.m_pos_hi[0] - P.m_pos_lo[0]) * u0);
        *my = (float)(P.m_pos_lo[1] + (P.m_pos_hi[1] - P.m_pos_lo[1]) * u1);
        *mz = (float)(P.m_pos_lo[2] + (P.m_pos_hi[2] - P.m_pos_lo[2]) * u2);
    }
    const float speed = (float)(P.m_speed_lo + (P.m_speed_hi - P.m_speed_lo) * u3);
    const float tx = sub((float)P.target_d[0], *mx), ty = sub((float)P.target_d[1], *my), tz = sub((float)P.target_d[2], *mz);
    const float td = norm3(tx, ty, tz);
    *vx = mul(dvd(tx, td), speed); *vy = mul(dvd(ty, td), speed); *vz = mul(dvd(tz, td), speed);
}

template <typename R>
__device__ __noinline__ SpawnOut spawn_values(const KernelArgs<R>& A, uint32_t c0, uint32_t c3hi, uint32_t ep, int64_t plane_i) {
    const KParams<R>& P = A.P;
    RngKey key;
    key.rk = &A.rk; key.c0 = c0; key.c3hi = c3hi;
    SpawnOut o;
    uint4 r0 = draw_raw(key, ep, 0u, HLYNR_BLK_SPAWN0);
    uint4 r1 = draw_raw(key, ep, 0u, HLYNR_BLK_SPAWN1);
    uint4 r2 = draw_raw(key, ep, 0u, HLYNR_BLK_SPAWN2);
    double u00 = u01(r0.x), u01_ = u01(r0.y), u02 = u01(r0.z), u03 = u01(r0.w);
    double u10 = u01(r1.x), u11 = u01(r1.y), u12 = u01(r1.z), u13 = u01(r1.w);
    double u20 = u01(r2.x), u21 = u01(r2.y);
    float mx, my, mz;
    spawn_missile(P, r0, &mx, &my, &mz, &o.mvx, &o.mvy, &o.mvz);
    (void)u00; (void)u01_; (void)u02; (void)u03;
    float ix = (float)(P.i_pos_lo[0] + (P.i_pos_hi[0] - P.i_pos_lo[0]) * u10);
    float iy = (float)(P.i_pos_lo[1] + (P.i_pos_hi[1] - P.i_pos_lo[1]) * u11);
    float iz = (float)(P.i_pos_lo[2] + (P.i_pos_hi[2] - P.i_pos_lo[2]) * u12);
    float lx = sub(mx, ix), ly = sub(my, iy), lz = sub(mz, iz);
    float ld = norm3(lx, ly, lz);
    o.d0 = ld;  // |missile_states[0] - interceptor| on the float32 state (environment.py:579-581)
    float ox = lx, oy = ly, oz = lz, od = ld;  // the launch orientation points at the CLOSEST missile of a volley (:476-486)
    if (P.volley_k > 0) {  // fill the missile planes: {pos, min_distance}, {vel, active}
        const int64_t n = A.ring_stride;
        A.st.vm[plane_i] = Vec4<R>{(R)mx, (R)my, (R)mz, (R)ld};
        A.st.vm[n + plane_i] = Vec4<R>{(R)o.mvx, (R)o.mvy, (R)o.mvz, R(1)};
        for (int m = 1; m < P.volley_k; ++m) {
            float px, py, pz, vx, vy, vz;
            spawn_missile(P, draw_raw(key, ep, 0u, HLYNR_BLK_VSPAWN(m)), &px, &py, &pz, &vx, &vy, &vz);
            const float dx = sub(px, ix), dy = sub(py, iy), dz = sub(pz, iz);
            const float d = norm3(dx, dy, dz);
            A.st.vm[(int64_t)(2 * m) * n + plane_i] = Vec4<R>{(R)px, (R)py, (R)pz, (R)d};
            A.st.vm[(int64_t)(2 * m + 1) * n + plane_i] = Vec4<R>{(R)vx, (R)vy, (R)vz, R(1)};
            if (d < od) { od = d; ox = dx; oy = dy; oz = dz; }
        }
    }
    if (P.toward_missile) {
        float sp = (float)(P.i_speed_lo + (P.i_speed_hi - P.i_speed_lo) * u13);
        o.vx = mul(dvd(lx, ld), sp); o.vy = mul(dvd(ly, ld), sp); o.vz = mul(dvd(lz, ld), sp);
    } else {
        o.vx = (float)(P.i_vel_lo[0] + (P.i_vel_hi[0] - P.i_vel_lo[0]) * u13);
        o.vy = (float)(P.i_vel_lo[1] + (P.i_vel_hi[1] - P.i_vel_lo[1]) * u20);
        o.vz = (float)(P.i_vel_lo[2] + (P.i_vel_hi[2] - P.i_vel_lo[2]) * u21);
    }
    // orientation: rotate +Z onto the line of sight (environment.py:492-530); float64 on float32 inputs
    o.qw = 1.f; o.qx = 0.f; o.qy = 0.f; o.qz = 0.f;
    if (od > 1e-6f) {
        double fx = dvd(ox, od), fy = dvd(oy, od), fz = dvd(oz, od);
        double ax = -fy, ay = fx;
        double al = sqrt(ax * ax + ay * ay + 0.0);
        if (al > 1e-6) {
            // h = acos(fz) / 2 without the transcendentals: cos h = sqrt((1 + fz) / 2), sin h = sqrt((1 - fz) / 2), and the
            // cancelling one of the two comes from sin(2h) = al instead (al = |f x z| = sin(acos fz) for the unit vector f).
            // (f is a float32 vector divided by its float32 norm, so |f|^2 = 1 + eps with |eps| ~ 1e-7, and the two forms differ
            // by up to about eps / (2 al): ~1e-7 in general, 2e-4 within 1e-3 rad of +-Z, where the reference's acos of a
            // float32 fz next to +-1 is itself quantised in steps of ~3.5e-4 rad.  Below the fp32 build's tolerance, visible at
            // the fp64 build's, which therefore keeps acos / sin / cos.)
            ax /= al; ay /= al;
            const double cz = clip(fz, -1.0, 1.0);
            double sh, ch;
            if constexpr (std::is_same<R, float>::value) {
                if (cz >= 0.0) { ch = sqrt((1.0 + cz) * 0.5); sh = al / (2.0 * ch); }
                else { sh = sqrt((1.0 - cz) * 0.5); ch = al / (2.0 * sh); }
            } else {
                const double h = acos(cz) / 2.0;
                sh = sin(h); ch = cos(h);
            }
            o.qw = (float)ch; o.qx = (float)(ax * sh); o.qy = (float)(ay * sh); o.qz = 0.f;
        } else if (!(fz > 0)) { o.qw = 0.f; o.qx = 1.f; }  // anti-aligned (quirk Q9: aligned -> identity)
    }
    o.mx = mx; o.my = my; o.mz = mz; o.ix = ix; o.iy = iy; o.iz = iz;
    o.ur = draw_raw(key, ep, 0u, HLYNR_BLK_UNI);
    o.dT0 = 0.0; o.base_cd = 0.3f; o.peak = (float)(P.peak_minus1 + R(1.0)); o.odelay = P.onboard_delay;
    if (P.dr) {  // physics_randomizer.py:166-214, 243-297
        float z0, z1, z2, z3, z4, zd;
        uint4 a = draw_raw(key, ep, 0u, HLYNR_BLK_DR0), b = draw_raw(key, ep, 0u, HLYNR_BLK_DR1);
        box_muller(a.x, a.y, &z0, &z1);
        box_muller(a.z, a.w, &z2, &z3);
        box_muller(b.x, b.y, &z4, &zd);
        (void)z0;
        o.dT0 = 0.0 + P.dr_var[1] * (double)z1;
        o.base_cd = (float)(0.3 * clip(1.0 + P.dr_var[2] * (double)z2, 0.1, 3.0));
        o.peak = (float)(3.0 * clip(1.0 + P.dr_var[3] * (double)z3, 0.1, 3.0));
        int nd = (int)(3.0 * clip(1.0 + P.dr_var[4] * (double)z4, 0.1, 3.0));
        o.odelay = nd < 1 ? 1 : (nd > 10 ? 10 : nd);
    }
    return o;
}

template <typename R> HD uint4 spawn(const KernelArgs<R>& A, Env<R>& e, const RngKey& key, int64_t plane_i) {
    const KParams<R>& P = A.P;
    const SpawnOut o = spawn_values(A, key.c0, key.c3hi, (uint32_t)e.episode, plane_i);
    e.mpx = o.mx; e.mpy = o.my; e.mpz = o.mz; e.mvx = o.mvx; e.mvy = o.mvy; e.mvz = o.mvz;
    e.ipx = o.ix; e.ipy = o.iy; e.ipz = o.iz; e.ivx = o.vx; e.ivy = o.vy; e.ivz = o.vz;
    e.qw = o.qw; e.qx = o.qx; e.qy = o.qy; e.qz = o.qz;
    e.fuel = R(100.0); e.fuel_used = R(0);
    e.wx = (float)P.base_wind[0]; e.wy = (float)P.base_wind[1]; e.wz = (float)P.base_wind[2];
    e.thx = e.thy = e.thz = R(0);
    int odelay = P.onboard_delay;
    if (P.dr) {
        if (P.isa) e.T0 = (R)((double)e.T0 + o.dT0);  // compounding random walk (quirk Q7)
        if (P.mach) { e.base_cd = o.base_cd; e.peak = o.peak; }
        if (P.onboard_delay > 0) odelay = o.odelay;
    }
    e.steps = 0; e.worsen = 0;
    e.flags = odelay << 8;  // crossed = false, kalman not initialised
    e.kpx = e.kpy = e.kpz = e.kvx = e.kvy = e.kvz = R(0);
    e.Ppp = 1000.f; e.Ppv = 0.f; e.Pvp = 0.f; e.Pvv = 1000.f;
    e.prev_d = e.last_d = e.min_d = (R)o.d0;
    e.ep_ret = R(0);
    return o.ur;
}

// EnhancedWindModel gust (physics_models.py:381-385): 0.1 % of the ticks, out of line
template <typename R>
__device__ __noinline__ Tri<R> wind_gust(const KernelArgs<R>& A, uint32_t c0, uint32_t c3hi, uint32_t ep, uint32_t st, R wvx, R wvy, R wvz) {
    RngKey key;
    key.rk = &A.rk; key.c0 = c0; key.c3hi = c3hi;
    float g0, g1, g2, g3;
    uint4 gd = draw_raw(key, ep, st, HLYNR_BLK_GUST_DIR);
    box_muller(gd.x, gd.y, &g0, &g1);
    box_muller(gd.z, gd.w, &g2, &g3);
    uint4 gm = draw_raw(key, ep, st, HLYNR_BLK_GUST_MAG);
    double nn = sqrt((double)g0 * g0 + (double)g1 * g1 + (double)g2 * g2) + 1e-6;
    double mag = A.P.gust_scale_d * (double)(-logf(u01_open(gm.x)));
    return Tri<R>{(R)((double)wvx + ((double)g0 / nn) * mag), (R)((double)wvy + ((double)g1 / nn) * mag),
                  (R)((double)wvz + ((double)g2 / nn) * mag)};
}

// ------------------------------------------------------------------------------------------------
// one tick (environment.py:605-859)
// ------------------------------------------------------------------------------------------------
struct TickOut {
    uint4 ur;  // the tick's BLK_UNI block, drawn once (gust / onboard dropout / ground dropout / packet loss)
    float reward;
    float distance;
    bool terminated, truncated, intercepted, hit, clamped, fuze;
};

// quaternion integration (environment.py:937-956): q <- normalize(dq(w dt) (x) q), product rounded to float32
HD void quat_step(Env<float>& e, float wx, float wy, float wz, float dt) {
    float w2 = fmaf(wz, wz, fmaf(wy, wy, wx * wx));
    float wn = nsqrt(w2);
    if (wn * dt > 1e-6f) {
        float h = 0.5f * wn * dt, h2 = h * h;  // h <= 0.18 rad for |a| <= 1: Taylor to float accuracy (step within 1.8e-7 of float64, B200)
        float sh = h * fmaf(h2, fmaf(h2, fmaf(h2, -1.98412698e-4f, 8.33333333e-3f), -1.66666667e-1f), 1.f);
        float ch = fmaf(h2, fmaf(h2, fmaf(h2, fmaf(h2, 2.48015873e-5f, -1.38888889e-3f), 4.16666667e-2f), -0.5f), 1.f);
        if (h > 0.5f) { const Pair<float> sc = sincos_full(h); sh = sc.a; ch = sc.b; }  // actions outside [-1,1]
        float k = sh * nrcp(wn);
        float w1 = ch, x1 = wx * k, y1 = wy * k, z1 = wz * k;
        float w2q = e.qw, x2 = e.qx, y2 = e.qy, z2 = e.qz;
        float nw = fmaf(-z1, z2, fmaf(-y1, y2, fmaf(-x1, x2, w1 * w2q)));
        float nx = fmaf(-z1, y2, fmaf(y1, z2, fmaf(x1, w2q, w1 * x2)));
        float ny = fmaf(z1, x2, fmaf(y1, w2q, fmaf(-x1, z2, w1 * y2)));
        float nz = fmaf(z1, w2q, fmaf(-y1, x2, fmaf(x1, y2, w1 * z2)));
        float inv = rsqrtf(fmaf(nz, nz, fmaf(ny, ny, fmaf(nx, nx, nw * nw))));
        e.qw = nw * inv; e.qx = nx * inv; e.qy = ny * inv; e.qz = nz * inv;
    }
}
HD void quat_step(Env<double>& e, double wx, double wy, double wz, double dt) {
    double wn = norm3(wx, wy, wz);
    double ang = mul(wn, dt);
    if (ang > 1e-6) {
        double sh, ch;
        const double h = mul(ang, 0.5), h2 = h * h;
        if (h <= 0.5) {   // |a| <= 1 gives h <= 0.18 rad: Taylor series to 1e-19 instead of the full-range sincos (Payne-Hanek slow path)
            sh = h * fma(h2, fma(h2, fma(h2, fma(h2, fma(h2, fma(h2, fma(h2, -7.6471637318198164e-13, 1.6059043836821613e-10), -2.5052108385441720e-08),
                                                                       2.7557319223985893e-06), -1.9841269841269841e-04), 8.3333333333333332e-03),
                                 -1.6666666666666666e-01), 1.0);
            ch = fma(h2, fma(h2, fma(h2, fma(h2, fma(h2, fma(h2, fma(h2, fma(h2, 4.7794773323873853e-14, -1.1470745597729725e-11), 2.0876756987868100e-09),
                                                                     -2.7557319223985888e-07), 2.4801587301587302e-05), -1.3888888888888889e-03),
                                             4.1666666666666664e-02), -0.5), 1.0);
        } else {
            const Pair<double> sc = sincos_full_d(h);
            sh = sc.a; ch = sc.b;
        }
        double w1 = ch, x1 = mul(dvd(wx, wn), sh), y1 = mul(dvd(wy, wn), sh), z1 = mul(dvd(wz, wn), sh);
        double w2 = (double)e.qw, x2 = (double)e.qx, y2 = (double)e.qy, z2 = (double)e.qz;
        float nw = (float)sub(sub(sub(mul(w1, w2), mul(x1, x2)), mul(y1, y2)), mul(z1, z2));
        float nx = (float)sub(add(add(mul(w1, x2), mul(x1, w2)), mul(y1, z2)), mul(z1, y2));
        float ny = (float)add(add(sub(mul(w1, y2), mul(x1, z2)), mul(y1, w2)), mul(z1, x2));
        float nz = (float)add(sub(add(mul(w1, z2), mul(x1, y2)), mul(y1, x2)), mul(z1, w2));
        double s2 = (double)__fmul_rn(nw, nw) + (double)__fmul_rn(nx, nx);
        s2 += (double)__fmul_rn(ny, ny);
        s2 += (double)__fmul_rn(nz, nz);
        float nn = __fsqrt_rn((float)s2);
        e.qw = dvd(nw, nn); e.qx = dvd(nx, nn); e.qy = dvd(ny, nn); e.qz = dvd(nz, nn);
    }
}

// _update_missile_state (environment.py:1069-1117) for one missile; every missile of a volley sees the same current_wind
template <typename R, int F>
HD void missile_update(const KParams<R>& P, const Env<R>& e, const RngKey& key, uint32_t ep, uint32_t st, uint32_t evade_blk,
                       R& mpx, R& mpy, R& mpz, R& mvx, R& mvy, R& mvz, const float* pre_z = nullptr) {
    typedef Feat<F> FT;
    const R dt = P.dt;
    R alt = mpz > R(0) ? mpz : R(0);
    R vax = sub(mvx, (R)e.wx), vay = sub(mvy, (R)e.wy), vaz = sub(mvz, (R)e.wz);
    R dax, day, daz;
    drag_accel<R, F>(P, e, vax, vay, vaz, alt, R(2.0), P.missile_ratio, R(1.0 / 1000.0), R(1000.0), &dax, &day, &daz);
    double ex = 0.0, ey = 0.0, ez = 0.0;
    if (FT::evasion(P)) {
        float z0, z1, z2;
        if (pre_z) { z0 = pre_z[0]; z1 = pre_z[1]; z2 = pre_z[2]; }
        else draw_normal3(key, ep, st, evade_blk, &z0, &z1, &z2);
        ex = (double)(z0 * 2.0f); ey = (double)(z1 * 2.0f); ez = (double)(z2 * 2.0f);
    }
    // total_accel = drag + gravity + evasion is float64 in the reference even without evasion
    // (evasion = np.zeros(3)), and velocity += total_accel * dt is evaluated in float64: kept as is.
    double ax = (double)dax + ex, ay = (double)day + ey, az = (double)add(daz, (R)(-9.81f)) + ez;
    if (P.validate && any_nonfinite(ax, ay, az)) {
        const Tri<double> g = nan_guard3<double>(ax, ay, az, 20.0);
        ax = g.x; ay = g.y; az = g.z;
    }
    mvx = (R)add((double)mvx, mul(ax, P.dt_d));
    mvy = (R)add((double)mvy, mul(ay, P.dt_d));
    mvz = (R)add((double)mvz, mul(az, P.dt_d));
    mpx = add(mpx, mul(mvx, dt)); mpy = add(mpy, mul(mvy, dt)); mpz = add(mpz, mul(mvz, dt));
}

// Volley mode (environment.py:236-267, 631-692, 724-748): advance every active missile, pick the priority missile
// (closest ACTIVE one after the update, strict <, first wins; missile 0 if none is active), intercept checks with
// per-missile minimum distances, distance = closest still-active missile (0.0 if none), ground hits.  One pass over the
// K missile planes; the priority missile's state becomes e.mp* / e.mv* (self.missile_state aliases that list entry).
struct VolleyOut { bool intercepted, hit, all_inactive; };
template <typename R, int F>
HD VolleyOut volley_step(const KernelArgs<R>& A, Env<R>& e, const RngKey& key, uint32_t ep, uint32_t st, int64_t i, R radius, R* distance) {
    const KParams<R>& P = A.P;
    const int K = P.volley_k;
    const int64_t n = A.ring_stride;
    VolleyOut o{false, false, true};
    int pri = -1, count = FLAG_VCOUNT(e.flags);
    R pbest = R(0), dist = R(0);
    bool any_active = false;
    R ppx = R(0), ppy = R(0), ppz = R(0), pvx = R(0), pvy = R(0), pvz = R(0);
#pragma unroll 1
    for (int m = 0; m < K; ++m) {
        Vec4<R> a = A.st.vm[(int64_t)(2 * m) * n + i], b = A.st.vm[(int64_t)(2 * m + 1) * n + i];
        bool act = b.w != R(0);
        if (act) {
            missile_update<R, F>(P, e, key, ep, st, m == 0 ? HLYNR_BLK_EVADE : HLYNR_BLK_VEVADE(m), a.x, a.y, a.z, b.x, b.y, b.z);
            const R d = norm3(sub(a.x, e.ipx), sub(a.y, e.ipy), sub(a.z, e.ipz));
            if (pri < 0 || d < pbest) { pri = m; pbest = d; ppx = a.x; ppy = a.y; ppz = a.z; pvx = b.x; pvy = b.y; pvz = b.z; }
            if (d < a.w) a.w = d;
            if (d < radius) { o.intercepted = true; count += 1; act = false; }
            else if (!any_active || d < dist) { dist = d; any_active = true; }
        }
        if (a.z <= R(0)) {  // every missile at or below the ground, also one that got there in an earlier tick
            act = false;
            const R gx = sub(a.x, P.target_x), gy = sub(a.y, P.target_y);
            if (sqr(dot2(gx, gy, gx, gy)) < R(500.0)) o.hit = true;
        }
        if (act) o.all_inactive = false;
        b.w = act ? R(1) : R(0);
        A.st.vm[(int64_t)(2 * m) * n + i] = a;
        A.st.vm[(int64_t)(2 * m + 1) * n + i] = b;
    }
    if (pri < 0) {  // nothing was active: self.missile_state = missile_states[0]
        const Vec4<R> a = A.st.vm[i], b = A.st.vm[n + i];
        pri = 0; ppx = a.x; ppy = a.y; ppz = a.z; pvx = b.x; pvy = b.y; pvz = b.z;
    }
    e.mpx = ppx; e.mpy = ppy; e.mpz = ppz; e.mvx = pvx; e.mvy = pvy; e.mvz = pvz;
    e.flags = (e.flags & ~((0x7 << 12) | (0xf << 16))) | (pri << 12) | (count << 16);
    *distance = dist;
    return o;
}

// The tick in four sections (the order of environment.py:605-859): interceptor, missile(s), wind, outcome.
template <typename R, int F>
HD void tick_interceptor(const KernelArgs<R>& A, Env<R>& e, const float act[6], bool* clamped_out) {
    typedef Feat<F> FT;
    const KParams<R>& P = A.P;
    R a0 = (R)act[0], a1 = (R)act[1], a2 = (R)act[2], a3 = (R)act[3], a4 = (R)act[4], a5 = (R)act[5];
    if (FT::obs_mode(P) == HLYNR_OBS_LOS) {
        // _update_los_frame + _transform_los_action_to_world (environment.py:965-1061): the basis is built in float32
        // from the TRUE positions before the physics update; thrust = a0 * lu + a1 * lh + a2 * lv
        const float rx = sub((float)e.mpx, (float)e.ipx), ry = sub((float)e.mpy, (float)e.ipy), rz = sub((float)e.mpz, (float)e.ipz);
        const float rr = norm3(rx, ry, rz);
        float ux = 1.f, uy = 0.f, uz = 0.f, hx = 1.f, hy = 0.f;
        if (rr > 1e-6f) { ux = dvd(rx, rr); uy = dvd(ry, rr); uz = dvd(rz, rr); }
        const float hn = norm3(uy, -ux, 0.f);
        if (hn > 1e-6f) { hx = dvd(uy, hn); hy = dvd(-ux, hn); }
        const float vx = -mul(uz, hy), vy = mul(uz, hx), vz = sub(mul(ux, hy), mul(uy, hx));
        const R t0 = add(add(mul(a0, (R)ux), mul(a1, (R)hx)), mul(a2, (R)vx));
        const R t1 = add(add(mul(a0, (R)uy), mul(a1, (R)hy)), mul(a2, (R)vy));
        const R t2 = add(mul(a0, (R)uz), mul(a2, (R)vz));  // lh.z == 0
        a0 = t0; a1 = t1; a2 = t2;
    }
    // SafetyClamp.apply (core.py:1069-1100); limits are in action units (quirk Q8)
    bool clamped = false;
    if (e.fuel <= R(0)) { a0 = a1 = a2 = R(0); clamped = true; }
    if (a0 * a0 + a1 * a1 + a2 * a2 > R(2499.0)) {
        const Vec4<R> c = clamp_norm_slow<R>(a0, a1, a2, R(50.0));
        a0 = c.x; a1 = c.y; a2 = c.z; clamped = clamped || c.w != R(0);
    }
    if (a3 * a3 + a4 * a4 + a5 * a5 > R(24.9)) {
        const Vec4<R> c = clamp_norm_slow<R>(a3, a4, a5, R(5.0));
        a3 = c.x; a4 = c.y; a5 = c.z; clamped = clamped || c.w != R(0);
    }
    *clamped_out = clamped;
    const R dt = P.dt;
    // ---- _update_interceptor (environment.py:861-963) ----
    {
        R Tx = mul(a0, R(10000.0)), Ty = mul(a1, R(10000.0)), Tz = mul(a2, R(10000.0));
        if (FT::thrust_dyn(P)) {  // first-order lag, :874-880
            if constexpr (std::is_same<R, float>::value) {
                e.thx = fmaf(Tx - e.thx, P.dt_over_tau, e.thx);
                e.thy = fmaf(Ty - e.thy, P.dt_over_tau, e.thy);
                e.thz = fmaf(Tz - e.thz, P.dt_over_tau, e.thz);
            } else {
                e.thx = add(e.thx, dvd(mul(sub(Tx, e.thx), dt), P.tau));
                e.thy = add(e.thy, dvd(mul(sub(Ty, e.thy), dt), P.tau));
                e.thz = add(e.thz, dvd(mul(sub(Tz, e.thz), dt), P.tau));
            }
            Tx = e.thx; Ty = e.thy; Tz = e.thz;
        }
        R tm = nnorm3(Tx, Ty, Tz);
        R burn = mul(mul(cdiv(tm, R(500.0), R(1.0 / 500.0)), R(0.1)), dt);
        e.fuel = sub(e.fuel, burn);
        e.fuel_used = add(e.fuel_used, burn);
        if (e.fuel <= R(0)) { e.fuel = R(0); Tx = Ty = Tz = R(0); e.thx = e.thy = e.thz = R(0); }
        R tax = cdiv(Tx, R(500.0), R(1.0 / 500.0)), tay = cdiv(Ty, R(500.0), R(1.0 / 500.0)), taz = cdiv(Tz, R(500.0), R(1.0 / 500.0));
        R alt = e.ipz > R(0) ? e.ipz : R(0);
        R vax = sub(e.ivx, (R)e.wx), vay = sub(e.ivy, (R)e.wy), vaz = sub(e.ivz, (R)e.wz);
        R dax, day, daz;
        drag_accel<R, F>(P, e, vax, vay, vaz, alt, R(1.0), R(1.0), R(1.0 / 500.0), R(500.0), &dax, &day, &daz);
        R ax = add(tax, dax), ay = add(tay, day), az = add(add(taz, daz), (R)(-9.81f));
        if (P.validate && any_nonfinite(ax, ay, az)) {
            const Tri<R> g = nan_guard3<R>(ax, ay, az, R(50));
            ax = g.x; ay = g.y; az = g.z;
        }
        // semi-implicit Euler, :933-934 (exact float ops, reference order)
        e.ivx = add(e.ivx, mul(ax, dt)); e.ivy = add(e.ivy, mul(ay, dt)); e.ivz = add(e.ivz, mul(az, dt));
        e.ipx = add(e.ipx, mul(e.ivx, dt)); e.ipy = add(e.ipy, mul(e.ivy, dt)); e.ipz = add(e.ipz, mul(e.ivz, dt));
        quat_step(e, mul(a3, R(20.0)), mul(a4, R(20.0)), mul(a5, R(20.0)), dt);
    }
}

// ---- _update_wind (environment.py:1119-1129): the wind used by the NEXT tick; ur = the tick's BLK_UNI block ----
template <typename R, int F>
HD void tick_wind(const KernelArgs<R>& A, Env<R>& e, const RngKey& key, uint32_t ep, uint32_t st, const uint4 ur, const float* pre_z = nullptr) {
    typedef Feat<F> FT;
    const KParams<R>& P = A.P;
    if (FT::enh_wind(P)) {  // EnhancedWindModel.get_wind_vector, physics_models.py:351-387
        R alt = e.ipz > R(0) ? e.ipz : R(0);
        R pf, ti;
        if (alt <= R(10.0)) { pf = R(1.0); ti = P.ti_low; }
        else if (alt <= P.blh) { pf = npow(alt * R(0.1), R(0.143)); ti = P.turb * (R(1.0) - alt * P.rc_blh * R(0.7)); }
        else { pf = P.pf_top; ti = P.ti_high; }
        R wvx = P.base_wind[0] * pf, wvy = P.base_wind[1] * pf, wvz = P.base_wind[2] * pf;
        if (ti > R(0)) {
            R scale = ti * nnorm3(wvx, wvy, wvz) * P.lp;
            float z0, z1, z2;
            if (pre_z) { z0 = pre_z[0]; z1 = pre_z[1]; z2 = pre_z[2]; }
            else draw_normal3(key, ep, st, HLYNR_BLK_WIND, &z0, &z1, &z2);
            wvx += scale * (R)z0; wvy += scale * (R)z1; wvz += scale * (R)z2;
        }
        if (u01(ur.x) < 0.001f) {  // gust, :381-385 (0.1 % of ticks)
            const Tri<R> g = wind_gust<R>(A, key.c0, key.c3hi, ep, st, wvx, wvy, wvz);
            wvx = g.x; wvy = g.y; wvz = g.z;
        }
        e.wx = (float)wvx; e.wy = (float)wvy; e.wz = (float)wvz;
    } else if (P.wind_var > R(0)) {  // AR(1) wind, environment.py:1127-1129 (float64 in the reference)
        float z0, z1, z2;
        draw_normal3(key, ep, st, HLYNR_BLK_WIND, &z0, &z1, &z2);
        e.wx = (float)(R(0.95) * (R)e.wx + R(0.05) * (P.base_wind[0] + (R)z0 * P.wind_var));
        e.wy = (float)(R(0.95) * (R)e.wy + R(0.05) * (P.base_wind[1] + (R)z1 * P.wind_var));
        e.wz = (float)(R(0.95) * (R)e.wz + R(0.05) * (P.base_wind[2] + (R)z2 * P.wind_var));
    }
}

// ---- distance / intercept / termination (environment.py:657-814) and _calculate_reward (:1131-1320).  Reads the interceptor's
// position, velocity and fuel AFTER its update; `dist` / `vo` come from volley_step() in volley mode ----
template <typename R, int F, bool kCur = false>
HD void tick_outcome(const KernelArgs<R>& A, Env<R>& e, const float act0, R dist, const VolleyOut vo, TickOut& t) {
    typedef Feat<F> FT;
    const KParams<R>& P = A.P;
    const R dt = P.dt;
    const R radius = FT::fuze(P) ? P.kill_radius : cur_radius<kCur>(A);
    bool intercepted, term = false, hit = false;
    if (FT::volley(P)) {
        intercepted = vo.intercepted; hit = vo.hit;
    } else {
        dist = norm3(sub(e.mpx, e.ipx), sub(e.mpy, e.ipy), sub(e.mpz, e.ipz));  // exact: feeds the reward
        intercepted = dist < radius;
    }
    if (dist < e.min_d) e.min_d = dist;
    if (intercepted) e.flags |= FLAG_CROSSED;
    bool fuze = false;
    if (FT::fuze(P) && e.min_d < P.kill_radius) { fuze = true; intercepted = true; }
    if (FT::volley(P)) {
        term = vo.all_inactive || fuze;
    } else {
        const bool missile_down = e.mpz <= R(0);
        {   // ground-impact distance to the target < 500 m (environment.py:769-776), branch-free: sqrt.rn(x) < 500 <=> x < 250000
            // (the largest x below 250000 has a root more than half an ulp below 500, in float and in double)
            const R gx = sub(e.mpx, P.target_x), gy = sub(e.mpy, P.target_y);
            hit = (FT::precision_mode(P) ? missile_down : (!intercepted && missile_down)) && dot2(gx, gy, gx, gy) < R(250000.0);
        }
        if (FT::precision_mode(P)) term = missile_down;
        else term = intercepted || missile_down;
    }
    if (e.ipz < R(0)) term = true;
    else if (e.fuel <= R(0)) term = true;
    else if (e.steps > 1000) {  // smart early termination, :795-811 (last_d only refreshed here, quirk Q11)
        if (dist > e.last_d) e.worsen += 1;
        else e.worsen = e.worsen - 5 > 0 ? e.worsen - 5 : 0;
        e.last_d = dist;
        if (e.worsen > 500 && dist > R(2500.0)) term = true;
    }
    t.truncated = e.steps >= P.max_steps;
    t.terminated = term; t.intercepted = intercepted; t.hit = hit; t.fuze = fuze;
    t.distance = (float)dist;
    // ---- _calculate_reward (environment.py:1131-1320), exact ops in the reference order ----
    R r;
    const bool crashed = e.ipz < R(0), dry = e.fuel <= R(0);
    if (FT::precision_mode(P)) {
        if (term) {
            R md = e.min_d;
            if (e.flags & FLAG_CROSSED) {
                R cr = cur_radius<kCur>(A);
                r = R(3000.0);
                if (md < cr) r = add(r, mul(dvd(sub(cr, md), cr), R(1000.0)));
                r = add(r, mul(nexp(dvd(-md, R(25.0))), R(500.0)));
                r = add(r, mul(nexp(dvd(-md, R(10.0))), R(1000.0)));
                r = add(r, mul(nexp(dvd(-md, R(3.0))), R(500.0)));
                r = add(r, (R)((double)(P.max_steps - e.steps) * 0.3));
            } else {
                r = mul(-md, R(0.5));
                if (r < R(-2000.0)) r = R(-2000.0);
                if (hit) r = sub(r, R(1000.0));
                else if (crashed) r = sub(r, R(500.0));
                else if (dry) r = sub(r, R(300.0));
            }
        } else {
            R dl = sub(e.prev_d, dist);
            r = mul(clip(cdiv(cdiv(dl, dt, P.rc_dt), R(100.0), R(0.01)), R(-0.5), R(2.0)), R(0.5));
            if (dist < R(50.0)) { r = add(r, mul(dl, R(5.0))); r = add(r, nexp(dvd(-dist, R(10.0)))); }
            else if (dist < R(150.0)) r = add(r, mul(dl, R(3.0)));
            else if (dist < R(500.0)) r = add(r, mul(dl, R(1.5)));
            else r = add(r, mul(dl, R(0.8)));
            R sp = norm3(e.ivx, e.ivy, e.ivz);
            if (sp > R(1.0) && dist > R(10.0)) {
                R al = dot3(dvd(e.ivx, sp), dvd(e.ivy, sp), dvd(e.ivz, sp), dvd(sub(e.mpx, e.ipx), dist),
                            dvd(sub(e.mpy, e.ipy), dist), dvd(sub(e.mpz, e.ipz), dist));
                r = add(r, mul(al, R(0.3)));
            }
            if (FT::obs_mode(P) == HLYNR_OBS_LOS) r = add(r, mul((R)act0, R(0.4)));  // forward-thrust shaping, :1252-1264
            r = sub(r, R(0.2));
            e.prev_d = dist;
        }
    } else if (intercepted) {
        r = (R)(5000.0 + (double)(P.max_steps - e.steps) * 0.5);
    } else if (term) {
        r = mul(-dist, R(0.5));
        if (r < R(-2000.0)) r = R(-2000.0);
        if (hit) r = sub(r, R(1000.0));
        else if (crashed) r = sub(r, R(500.0));
        else if (dry) r = sub(r, R(300.0));
    } else {
        R dl = sub(e.prev_d, dist);
        r = mul(clip(cdiv(cdiv(dl, dt, P.rc_dt), R(100.0), R(0.01)), R(-0.5), R(2.0)), R(0.3));
        r = add(r, mul(dl, dist < R(200.0) ? R(2.0) : (dist < R(500.0) ? R(1.0) : R(0.5))));
        r = sub(r, R(0.5));
        e.prev_d = dist;
    }
    e.ep_ret = e.ep_ret + r;
    t.reward = (float)r;
}

template <typename R, int F, bool kCur = false>
HD void tick_physics(const KernelArgs<R>& A, Env<R>& e, const RngKey& key, const float act[6], int64_t ring_i, TickOut& t) {
    typedef Feat<F> FT;
    const KParams<R>& P = A.P;
    e.steps += 1;
    const uint32_t ep = (uint32_t)e.episode, st = (uint32_t)e.steps;
    t.ur = draw_raw(key, ep, st, HLYNR_BLK_UNI);
    // The evasion and wind draws only need the counters, which arrive with the first planes (load_env): drawn HERE they run while the
    // other planes are still in flight -- the second first-use stall of the prologue was 3.6 % of the samples -- instead of inside
    // missile_update() / tick_wind() (cfg4 100.5 -> 98.9 us, fp64 build 222.0 -> 219.0 us; profiles/r02_l_load_order_ab.log).
    float ze[3], zw[3];
    const bool pre = !FT::generic && !FT::volley(P);
    if (pre && FT::evasion(P)) draw_normal3(key, ep, st, HLYNR_BLK_EVADE, &ze[0], &ze[1], &ze[2]);
    if (pre && FT::enh_wind(P)) draw_normal3(key, ep, st, HLYNR_BLK_WIND, &zw[0], &zw[1], &zw[2]);
    tick_interceptor<R, F>(A, e, act, &t.clamped);
    // ---- missiles (environment.py:631-638), advanced with the wind of THIS tick (before _update_wind); a volley's
    // missiles, their priority selection and intercept checks are one pass over the missile planes ----
    R dist = R(0);
    VolleyOut vo{false, false, false};
    const R radius = FT::fuze(P) ? P.kill_radius : cur_radius<kCur>(A);
    if (FT::volley(P)) vo = volley_step<R, F>(A, e, key, ep, st, ring_i, radius, &dist);
    else missile_update<R, F>(P, e, key, ep, st, HLYNR_BLK_EVADE, e.mpx, e.mpy, e.mpz, e.mvx, e.mvy, e.mvz, (pre && FT::evasion(P)) ? ze : nullptr);
    tick_wind<R, F>(A, e, key, ep, st, t.ur, (pre && FT::enh_wind(P)) ? zw : nullptr);
    tick_outcome<R, F, kCur>(A, e, act[0], dist, vo, t);
}

// ------------------------------------------------------------------------------------------------
// episode statistics: warp-level reduction, one atomic per warp per finished-episode event
// ------------------------------------------------------------------------------------------------
HD double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// kDirect = false is the pure warp reduction.  ptxas negotiates registers across __noinline__ calls: under a 96-register cap
// (5 CTAs per SM, as the v2.0-off kernel once ran) the register needs of the direct-atomics path cost the CALLER 60 B of
// hot-path spills (86 -> 100 us per launch); every step kernel now runs at 4 CTAs per SM, where there is room.
template <bool kDirect>
__device__ __noinline__ void account_episodes_slow(double* stats, bool d, float ep_ret, int steps, float min_d, float dist,
                                                   int cause, bool intercepted, bool terminated) {
    double* slot = stats + (size_t)(blockIdx.x % HLYNR_STAT_SLOTS) * HLYNR_STATS_WORDS;
    if (kDirect && __popc(__ballot_sync(0xffffffffu, d)) <= 4) {   // the usual case is ONE finished env in the warp: its lane adds its own
        if (d) {                                        // terms (fire-and-forget reductions) instead of 12 warp-wide double sums
            atomicAdd(slot + 0, 1.0);
            if (intercepted) atomicAdd(slot + 1, 1.0);
            atomicAdd(slot + 2, (double)ep_ret); atomicAdd(slot + 3, (double)steps);
            atomicAdd(slot + 4, (double)min_d); atomicAdd(slot + 5, (double)dist);
            if (cause >= 0) atomicAdd(slot + 6 + cause, 1.0);
            if (!terminated) atomicAdd(slot + 11, 1.0);
        }
        return;
    }
    double v[12];   // many envs of the warp finished together (e.g. a time-out of envs that are still in phase): one atomic per warp
    v[0] = d ? 1.0 : 0.0;
    v[1] = (d && intercepted) ? 1.0 : 0.0;
    v[2] = d ? (double)ep_ret : 0.0;
    v[3] = d ? (double)steps : 0.0;
    v[4] = d ? (double)min_d : 0.0;
    v[5] = d ? (double)dist : 0.0;
#pragma unroll
    for (int c = 0; c < 5; ++c) v[6 + c] = (d && cause == c) ? 1.0 : 0.0;
    v[11] = (d && !terminated) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 0; k < 12; ++k) {
        double s = warp_sum(v[k]);
        if ((threadIdx.x & 31) == 0 && s != 0.0) atomicAdd(slot + k, s);
    }
}

template <typename R, bool kDirect = true>
HD void account_episodes(const KernelArgs<R>& A, bool active, bool done, const Env<R>& e, const TickOut& t) {
    // called by all lanes of the warp; finished episodes are rare (~1 per 1000 ticks per env)
    if (__ballot_sync(0xffffffffu, active && done) == 0u) return;
    const bool d = active && done;
    int cause = -1;  // first matching termination cause, in the reference's reward order
    if (d && t.terminated && !t.intercepted) {
        if (t.hit) cause = 0;
        else if (e.ipz < R(0)) cause = 1;
        else if (e.fuel <= R(0)) cause = 2;
        else if (e.mpz <= R(0)) cause = 3;
        else cause = 4;
    }
    account_episodes_slow<kDirect>(A.io.stats, d, (float)e.ep_ret, e.steps, (float)e.min_d, t.distance, cause, t.intercepted,
                          t.terminated);
}

// ------------------------------------------------------------------------------------------------
// coalesced [N,26] store through shared memory (one warp-private tile per warp)
// ------------------------------------------------------------------------------------------------
// The observation channels are written by observe() straight into the warp's tile (row pitch 26 words); here the
// warp streams the 32*26 floats out linearly as float4 (the tile offset of a linear index is the index itself).
#define OBS_TILE (32 * HLYNR_OBS_DIM)
__device__ __noinline__ void flush_obs_ragged(const float* tile, float* base, int valid, unsigned lane) {  // last warp of a ragged shard
    for (int idx = (int)lane; idx < valid; idx += 32) base[idx] = tile[idx];
}
HD void flush_obs_tile(const float* tile, float* dst, int64_t warp_first_env, int64_t n, unsigned lane) {
    __syncwarp();
    const int64_t rows = n - warp_first_env;
    float* base = dst + warp_first_env * HLYNR_OBS_DIM;  // 32 * 104 B per warp: 16-byte aligned
    if (rows >= 32) {
        const float4* t4 = reinterpret_cast<const float4*>(tile);
        float4* b4 = reinterpret_cast<float4*>(base);
#pragma unroll
        for (int k = 0; k < 7; ++k) {
            const int idx = k * 32 + (int)lane;
            if (k < 6 || idx < OBS_TILE / 4) b4[idx] = t4[idx];
        }
    } else if (rows > 0) {
        flush_obs_ragged(tile, base, (int)rows * HLYNR_OBS_DIM, lane);
    }
    __syncwarp();
}
// narrow observation rows (obs_dim < 26: the 17-D radar layout obs[0:17], rl_system/hrl/observation_schema.py:13-46): the warp
// streams rows * dim floats out linearly (coalesced 128-byte stores), gathering them from the 26-word tile rows
__device__ __noinline__ void flush_obs_narrow(const float* tile, float* base, int rows, int dim, unsigned lane) {
    const int total = rows * dim;
    for (int idx = (int)lane; idx < total; idx += 32) {
        const int r = idx / dim;
        base[idx] = tile[r * HLYNR_OBS_DIM + (idx - r * dim)];
    }
}
__device__ __noinline__ void copy_obs_row_n(const float* row, float* dst_row, int dim) {
    for (int k = 0; k < dim; ++k) dst_row[k] = row[k];
}
// this lane's row of the tile -> one row of a [N,26] array (terminal observation of a finished episode: rare)
__device__ __noinline__ void copy_obs_row(const float* row, float* dst_row) {
#pragma unroll
    for (int k = 0; k < HLYNR_OBS_DIM; ++k) dst_row[k] = row[k];
}

HD uint32_t info_flags(int eflags, bool intercepted, bool hit, bool clamped, bool onboard_det, bool ground_det, bool fuze) {
    return (uint32_t)((intercepted ? 1 : 0) | (hit ? 2 : 0) | (clamped ? 4 : 0) | (onboard_det ? 8 : 0) | (ground_det ? 16 : 0) |
                      ((eflags & FLAG_CROSSED) ? 32 : 0) | (fuze ? 64 : 0) | ((eflags & FLAG_KF_INIT) ? 128 : 0));
}

// info['missiles_intercepted'], ['missiles_remaining'], ['missile_min_distances'] (environment.py:846-848), written straight
// to their destinations; out of line (rare: info requests and finished episodes) so the hot body carries no extra registers
template <typename R>
__device__ __noinline__ void volley_info(const KernelArgs<R>& A, int64_t i, int eflags, float distance, bool intercepted,
                                         int32_t* intercepted_n, int32_t* remaining_n, float* md) {
#pragma unroll
    for (int m = 0; m < HLYNR_MAX_VOLLEY; ++m) md[m] = 0.f;
    if (A.P.volley_k > 0) {
        int left = 0;
        for (int m = 0; m < A.P.volley_k; ++m) {
            md[m] = (float)A.st.vm[(int64_t)(2 * m) * A.ring_stride + i].w;
            left += A.st.vm[(int64_t)(2 * m + 1) * A.ring_stride + i].w != R(0) ? 1 : 0;
        }
        *intercepted_n = FLAG_VCOUNT(eflags); *remaining_n = left;
    } else {
        md[0] = distance; *intercepted_n = intercepted ? 1 : 0; *remaining_n = intercepted ? 0 : 1;
    }
}

// Optional per-env info arrays (HlynrInfoSoA).  Out of line and fed by value: the eager-info path is not the hot one and
// must not cost the step kernel registers.
template <typename R>
__device__ __noinline__ void write_info_slow(const KernelArgs<R>& A, int64_t i, float distance, float min_d, float fuel, float fuel_used,
                                             int steps, int eflags, uint32_t flags8, bool intercepted, float ix, float iy, float iz,
                                             float mx, float my, float mz, float ep_ret) {
    const HlynrInfoSoA& f = A.io.info;
    if (f.distance) f.distance[i] = distance;
    if (f.min_distance) f.min_distance[i] = min_d;
    if (f.fuel_remaining) f.fuel_remaining[i] = fuel;
    if (f.fuel_used) f.fuel_used[i] = fuel_used;
    if (f.steps) f.steps[i] = steps;
    if (f.flags) f.flags[i] = (uint8_t)flags8;
    if (f.interceptor_pos) { f.interceptor_pos[3 * i] = ix; f.interceptor_pos[3 * i + 1] = iy; f.interceptor_pos[3 * i + 2] = iz; }
    if (f.missile_pos) { f.missile_pos[3 * i] = mx; f.missile_pos[3 * i + 1] = my; f.missile_pos[3 * i + 2] = mz; }
    if (f.episode_return) f.episode_return[i] = ep_ret;
    if (f.episode_length) f.episode_length[i] = steps;
    if (f.radar_quality)   // 0.0 while the onboard delay buffer fills (core.py:579-584), else the configured quality
        f.radar_quality[i] = (A.P.onboard_delay > 0 && steps < FLAG_ODELAY(eflags)) ? 0.f : A.P.radar_quality;
    if (f.missiles_intercepted && f.missiles_remaining && f.missile_min_distances)  // environment.py:844-848 (all three or none)
        volley_info(A, i, eflags, distance, intercepted, f.missiles_intercepted + i, f.missiles_remaining + i,
                    f.missile_min_distances + (int64_t)HLYNR_MAX_VOLLEY * i);
}
template <typename R> HD void write_info(const KernelArgs<R>& A, int64_t i, const Env<R>& e, const TickOut& t, const ObsOut& ob) {
    write_info_slow(A, i, t.distance, (float)e.min_d, (float)e.fuel, (float)e.fuel_used, e.steps, e.flags,
                    info_flags(e.flags, t.intercepted, t.hit, t.clamped, ob.onboard_det, ob.ground_det, t.fuze), t.intercepted,
                    (float)e.ipx, (float)e.ipy, (float)e.ipz, (float)e.mpx, (float)e.mpy, (float)e.mpz, (float)e.ep_ret);
}

// Appends the finished episode of env i to the compact done list (rare: ~1 per 1000 ticks per env).  Out of line
// and fed by value so the env state never has its address taken.
__device__ __noinline__ int32_t append_done_record(HlynrDoneRecord* recs, int32_t* counter, int32_t cap, int32_t env, int32_t steps,
                                                uint32_t flags, float distance, float min_d, float fuel, float fuel_used,
                                                float ep_ret, float ix, float iy, float iz, float mx, float my, float mz,
                                                const float* obs_row) {
    const int32_t slot = atomicAdd(counter, 1);
    if (slot >= cap) return -1;
    HlynrDoneRecord* r = recs + slot;
    r->env = env; r->steps = steps; r->flags = flags;
    r->distance = distance; r->min_distance = min_d; r->fuel_remaining = fuel; r->fuel_used = fuel_used; r->episode_return = ep_ret;
    r->interceptor_pos[0] = ix; r->interceptor_pos[1] = iy; r->interceptor_pos[2] = iz;
    r->missile_pos[0] = mx; r->missile_pos[1] = my; r->missile_pos[2] = mz;
#pragma unroll
    for (int k = 0; k < HLYNR_OBS_DIM; ++k) r->terminal_obs[k] = obs_row[k];
    return slot;
}
// One out-of-line call per finished episode: flag word, record, volley fields (the call site only marshals scalars).
template <typename R>
__device__ __noinline__ void record_done(const KernelArgs<R>& A, int64_t i, int steps, int eflags, bool terminated, bool truncated,
                                         bool intercepted, bool hit, bool clamped, bool onboard_det, bool ground_det, bool fuze,
                                         float distance, float min_d, float fuel, float fuel_used, float ep_ret, float ix, float iy,
                                         float iz, float mx, float my, float mz, const float* obs_row) {
    const uint32_t flags = info_flags(eflags, intercepted, hit, clamped, onboard_det, ground_det, fuze) |
                           (terminated ? HLYNR_DONE_TERMINATED : 0u) | (truncated ? HLYNR_DONE_TRUNCATED : 0u) |
                           ((A.P.onboard_delay > 0 && steps < FLAG_ODELAY(eflags)) ? HLYNR_DONE_ONBOARD_FILL : 0u);
    const int32_t slot = append_done_record(A.io.done_records, A.io.done_counter, A.io.done_cap, (int32_t)i, steps, flags, distance,
                                            min_d, fuel, fuel_used, ep_ret, ix, iy, iz, mx, my, mz, obs_row);
    if (slot >= 0) {
        HlynrDoneRecord* r = A.io.done_records + slot;
        volley_info(A, i, eflags, distance, intercepted, &r->missiles_intercepted, &r->missiles_remaining, r->missile_min_distances);
    }
}
template <typename R> HD RngKey make_key(const KernelArgs<R>& A, int64_t global_env) {
    RngKey k;
    k.rk = &A.rk;
    k.c0 = (uint32_t)((uint64_t)global_env & 0xffffffffu);
    k.c3hi = (uint32_t)((uint64_t)global_env >> 32) << 16;
    return k;
}

#define HLYNR_BLOCK 128
// CTA size of the direct step kernel (a multiple of 32 that divides HLYNR_BLOCK).  Nothing in that kernel is CTA-wide (warp-private
// observation tiles, no barrier), so the CTA is only the unit in which SM slots are handed back.
#ifndef HLYNR_STEP_BLOCK
#define HLYNR_STEP_BLOCK 64   /* 128 / 64 / 32 threads with the final kernel of round 2: cfg4 99.0 / 98.0 / 98.0 us at 2^20 envs, cfg3 at 262144 envs 35.0 / 34.6 / 34.4 us, cfg2 at 4096 envs 8.16 / 8.01 / 8.01 us per tick in a graph (profiles/r02_o_cta_size_ab.log): SM slots are handed back at a finer grain */
#endif

// The delay-ring samples a tick reads (one onboard slot, two ground planes) are needed only deep inside observe(),
// ~1000 instructions after the kernel starts; without help their DRAM latency is fully exposed there (9 % + 3 % of all
// stall samples in profiles/r01_c).  Their addresses depend only on the tick, so the lines are pulled into L1 up front,
// at no register cost.  (With domain randomization the onboard delay is per-env state: that row is not prefetched.)
HD void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
HD void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// State planes + actions of the CTA `prefetch_ahead` envs further on are touched with prefetch.global.L2 right after this
// CTA's own loads are issued.  The up-front plane loads are the one latency nothing else in a warp can hide (16 % of the
// stall samples in profiles/r01_c sit on their first use); measured on B200 at 2^20 envs (cfg4, 2000-tick bench):
// look-ahead 0 / 1 / 2 / 3 / 4 CTAs per SM -> 122.9 / 116.0 / 118.4 / 119.7 / 124 us per launch.  DRAM traffic is unchanged.
template <typename R, int F> HD void prefetch_next_wave(const KernelArgs<R>& A, int64_t j) {
    typedef Feat<F> FT;
    const StatePlanes<R>& s = A.st;
#pragma unroll
    for (int k = 0; k < 6; ++k) prefetch_l2(s.r[k] + j);
    if (FT::thrust_dyn(A.P) || FT::dr(A.P)) prefetch_l2(s.r[6] + j);
#pragma unroll
    for (int k = 0; k < 3; ++k) prefetch_l2(s.f[k] + j);
    if (FT::dr(A.P) && !dr_compact_layout<R, F>(A)) prefetch_l2(s.f[3] + j);
    if (!compact_layout<R, F>(A)) prefetch_l2(s.i0 + j);
    if (A.io.actions) prefetch_l2(A.io.actions + j * HLYNR_ACT_DIM);
}
#ifndef HLYNR_RING_PF
#define HLYNR_RING_PF 1   /* 0 = no prefetch of the delayed ring rows, 1 = prefetch.global.L1, 2 = prefetch.global.L2 */
#endif
HD void prefetch_ring(const void* p) {
    if (HLYNR_RING_PF == 1) prefetch_l1(p);
    else if (HLYNR_RING_PF == 2) prefetch_l2(p);
}
// API-mode prologue: the row addresses come ready-made from the host.  Computing them here (o_row - P.onboard_delay, ring lengths)
// put two more constant-bank lines on the path in front of the demand loads: with the loads-first order of the prologue the stall
// of profiles/r02_k_* simply moved to the uniform subtraction that waited for them (6.5 % of the samples; worth 0.3 us per launch).
template <typename R, int F> HD void prefetch_ring_reads_api(const KernelArgs<R>& A, int64_t i) {
    typedef Feat<F> FT;
    if (FT::onboard_delay(A.P) && !FT::dr(A.P)) prefetch_ring(A.pf_o + i);
    if (FT::ground(A.P) && FT::ground_delay(A.P)) { prefetch_ring(A.pf_g + i); prefetch_ring(A.pf_g + A.ring_stride + i); }
}
template <typename R, int F> HD void prefetch_ring_reads(const KernelArgs<R>& A, int64_t i, int g_row, int o_row) {
    typedef Feat<F> FT;
    const KParams<R>& P = A.P;
    const int64_t n = A.ring_stride;
    if (FT::onboard_delay(P) && !FT::dr(P)) {
        int rrow = o_row - P.onboard_delay;
        if (rrow < 0) rrow += P.onb_ring_len;
        prefetch_ring(A.st.oring + (int64_t)rrow * n + i);
    }
    if (FT::ground(P) && FT::ground_delay(P)) {
        const int rrow = g_row + 1 == P.gnd_ring_len ? 0 : g_row + 1;
        const Vec4<R>* rr = A.st.gring + (int64_t)rrow * 2 * n;
        prefetch_ring(rr + i);
        prefetch_ring(rr + n + i);
    }
}

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
// step(): one tick of every env + SB3 auto-reset.  kRollout: k fused ticks, state stays in registers.
// CTAs per SM: 4 for the fp32 build (<= 128 registers, no spills).  The fp64 build holds ~60 doubles of env state (120
// registers) before any temporaries: at 4 CTAs per SM it spills (cfg4 steady state 308 us at 2^20 envs), at 2 (<= 255 registers)
// too few warps are resident (355 us); 3 CTAs per SM (<= 168 registers, no spills) is the measured optimum (300 us).
#ifndef HLYNR_F64_MIN_BLOCKS
#define HLYNR_F64_MIN_BLOCKS 3
#endif
template <typename R> struct StepOcc { static constexpr int ctas = std::is_same<R, double>::value ? HLYNR_F64_MIN_BLOCKS : 4; };
// kCur: the curriculum comes from the attached schedule's device slot (KernelArgs::cur_dev), API-mode ticks only.
template <typename R, bool kRollout, int F, bool kCur = false>
__global__ void __launch_bounds__(HLYNR_STEP_BLOCK, StepOcc<R>::ctas * (HLYNR_BLOCK / HLYNR_STEP_BLOCK))
step_kernel(const __grid_constant__ KernelArgs<R> A) {
    __shared__ __align__(16) float tiles[HLYNR_STEP_BLOCK / 32][OBS_TILE];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const int64_t i = A.first + (int64_t)blockIdx.x * HLYNR_STEP_BLOCK + threadIdx.x;
    const int64_t warp_first = i - lane;
    const bool active = i < A.lim;
    const int64_t ii = active ? i : A.lim - 1;  // inactive lanes shadow the last env and never store
    // Programmatic dependent launch (option "pdl"): this grid may have been scheduled while the previous kernel of the stream was
    // still running.  Tell the scheduler the NEXT launch may do the same, then wait until the previous kernel has completed and
    // its writes are visible -- nothing above touches global memory.  Both are no-ops in an ordinary launch.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    Env<R> e;
    load_env<R, F>(A, ii, e);
    // Issue order of the prologue: every demand load (planes, actions) first, THEN the prefetches.  A prefetch (CCTL.E.PF1 / PF2) keeps
    // its address registers on the scoreboard until it completes; with the ring prefetches ahead of the loads, the third action load
    // reused such a register and waited a full memory latency (6 % of all stall samples in profiles/r02_i_step_kernel_*), holding back
    // the eight plane loads queued behind it.  Loads first: -0.9 us per launch on every configuration (profiles/r02_j_*).
    float2 a0 = make_float2(0.f, 0.f), a1 = a0, a2 = a0;
    if (!kRollout) {
        const float2* ap = reinterpret_cast<const float2*>(A.io.actions + ii * HLYNR_ACT_DIM);
        a0 = __ldg(ap); a1 = __ldg(ap + 1); a2 = __ldg(ap + 2);
    }
    if (kRollout) prefetch_ring_reads<R, F>(A, i, A.g_row, A.o_row);
    else prefetch_ring_reads_api<R, F>(A, i);
    if (!kRollout && A.prefetch_ahead > 0 && i + A.prefetch_ahead < A.lim) prefetch_next_wave<R, F>(A, i + A.prefetch_ahead);
    const RngKey key = make_key(A, A.env_offset + ii);
    if (!kRollout && Feat<F>::onboard_delay(A.P) && Feat<F>::dr(A.P)) {
        // domain randomization: the onboard delay is per-env state, so the delayed row is only known once the counter plane has
        // arrived; prefetched here (the tick's first instructions need that plane anyway) instead of read cold deep in observe()
        int rrow = A.o_row - FLAG_ODELAY(e.flags);
        if (rrow < 0) rrow += A.P.onb_ring_len;
        prefetch_l1(A.st.oring + (int64_t)rrow * A.ring_stride + i);
    }
    const int steps = kRollout ? A.k_steps : 1;
    float rsum = 0.f;
    int dcount = 0, locks = 0;
    ObsOut ob;
    ob.row = tiles[warp] + lane * HLYNR_OBS_DIM;
    int g_row = A.g_row, o_row = A.o_row;
#pragma unroll 1
    for (int s = 0; s < steps; ++s) {
        float act[6];
        if (kRollout && A.io.actions == nullptr) {  // synthetic random policy, a = 2u-1
            uint4 r0 = draw_raw(key, (uint32_t)e.episode, (uint32_t)e.steps + 1u, HLYNR_BLK_ACT0);
            uint4 r1 = draw_raw(key, (uint32_t)e.episode, (uint32_t)e.steps + 1u, HLYNR_BLK_ACT1);
            act[0] = 2.f * u01(r0.x) - 1.f; act[1] = 2.f * u01(r0.y) - 1.f; act[2] = 2.f * u01(r0.z) - 1.f;
            act[3] = 2.f * u01(r0.w) - 1.f; act[4] = 2.f * u01(r1.x) - 1.f; act[5] = 2.f * u01(r1.y) - 1.f;
        } else {
            float2 p0 = a0, p1 = a1, p2 = a2;   // API mode: loaded in the prologue
            if (kRollout) {
                const float2* ap = reinterpret_cast<const float2*>(A.io.actions + ((int64_t)s * A.n + ii) * HLYNR_ACT_DIM);
                p0 = __ldg(ap); p1 = __ldg(ap + 1); p2 = __ldg(ap + 2);
            }
            act[0] = p0.x; act[1] = p0.y; act[2] = p1.x; act[3] = p1.y; act[4] = p2.x; act[5] = p2.y;
        }
        TickOut t;
        tick_physics<R, F, kCur>(A, e, key, act, i, t);
        ob.emit = !kRollout || (s == steps - 1 && A.io.obs != nullptr);
        uint4 ur = t.ur;
        bool need_reset = false;
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {  // pass 1 = in-kernel auto-reset of finished envs (one copy of observe)
            if (pass == 1) {
                if (!need_reset) break;
                e.episode += 1;
                ur = spawn(A, e, key, i);
            }
            // ring planes are indexed by the lane's OWN (padded) slot: a shadow lane of another warp may run ticks
            // ahead in a fused rollout and must never touch the rows of the env it shadows
            observe<R, F, kCur>(A, e, key, ur, i, g_row, o_row, ob);
            if (pass == 0) {
                const bool done = t.terminated || t.truncated;
                if (ob.onboard_det) locks += 1;
                if (!kRollout && active) {
                    A.io.reward[i] = t.reward;
                    A.io.terminated[i] = t.terminated ? 1 : 0;
                    if (A.io.done) A.io.done[i] = (t.terminated || t.truncated) ? 1 : 0;
                    A.io.truncated[i] = t.truncated ? 1 : 0;
                    if (A.has_info) write_info(A, i, e, t, ob);
                }
                rsum += t.reward;
                account_episodes<R>(A, active, done, e, t);
                if (!kRollout && done && active && A.io.done_records) {
                    record_done<R>(A, i, e.steps, e.flags, t.terminated, t.truncated, t.intercepted, t.hit, t.clamped, ob.onboard_det,
                                   ob.ground_det, t.fuze, t.distance, (float)e.min_d, (float)e.fuel, (float)e.fuel_used, (float)e.ep_ret,
                                   (float)e.ipx, (float)e.ipy, (float)e.ipz, (float)e.mpx, (float)e.mpy, (float)e.mpz, ob.row);
                }
                need_reset = done && A.auto_reset;
                if (need_reset) {
                    dcount += 1;
                    if (!kRollout && active && A.io.terminal_obs) {
                        if (A.obs_dim == HLYNR_OBS_DIM) copy_obs_row(ob.row, A.io.terminal_obs + i * HLYNR_OBS_DIM);
                        else copy_obs_row_n(ob.row, A.io.terminal_obs + i * A.obs_dim, A.obs_dim);
                    }
                }
            }
        }
        if (kRollout) {  // next tick's ring rows
            g_row = g_row + 1 >= A.P.gnd_ring_len ? 0 : g_row + 1;
            o_row = o_row + 1 >= A.P.onb_ring_len ? 0 : o_row + 1;
            if (s + 1 < steps) prefetch_ring_reads<R, F>(A, i, g_row, o_row);
        }
    }
    {   // onboard-lock ticks: one atomic per warp that saw a lock, spread over the stat slots.  Ahead of the output stores: placed
        // after them, the thread-index re-read it needs landed in a register the in-flight observation stores still held as their
        // address, and waited for them (3.4 % of the fp64 build's stall samples, profiles/r02_k_*)
        const int wl = __reduce_add_sync(0xffffffffu, active ? locks : 0);
        if (lane == 0 && wl) atomicAdd(A.io.stats + (size_t)(blockIdx.x % HLYNR_STAT_SLOTS) * HLYNR_STATS_WORDS + 13, (double)wl);
    }
    if (A.io.obs) {
        if (A.obs_dim == HLYNR_OBS_DIM) flush_obs_tile(tiles[warp], A.io.obs, warp_first, A.lim, lane);
        else {
            __syncwarp();
            const int64_t rows = A.lim - warp_first;
            if (rows > 0) flush_obs_narrow(tiles[warp], A.io.obs + warp_first * A.obs_dim, rows >= 32 ? 32 : (int)rows, A.obs_dim, lane);
            __syncwarp();
        }
    }
    if (kRollout && active) {
        if (A.io.reward_sum) A.io.reward_sum[i] = rsum;
        if (A.io.done_count) A.io.done_count[i] = dcount;
    }
    if (active) store_env<R, F>(A, i, e);
}

// reset(): environment.py:353.  mask == NULL resets every env.
template <typename R, bool kCur = false> __global__ void __launch_bounds__(HLYNR_BLOCK) reset_kernel(const __grid_constant__ KernelArgs<R> A) {
    __shared__ __align__(16) float tiles[HLYNR_BLOCK / 32][OBS_TILE];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * HLYNR_BLOCK + threadIdx.x;
    if (i >= A.n) return;
    if (A.io.reset_mask != nullptr && A.io.reset_mask[i] == 0) return;
    Env<R> e;
    load_env(A, i, e);
    const RngKey key = make_key(A, A.env_offset + i);
    ObsOut ob;
    ob.row = tiles[warp] + lane * HLYNR_OBS_DIM;
    ob.emit = true;
    e.episode += 1;
    const uint4 ur = spawn(A, e, key, i);
    observe<R, FT_GENERIC_MODES, kCur>(A, e, key, ur, i, A.g_row, A.o_row, ob);
    store_env(A, i, e);
    if (A.io.obs) copy_obs_row_n(ob.row, A.io.obs + i * A.obs_dim, A.obs_dim);
}

}  // namespace hlynr
