// step_kernel.cu — K1: fused controller cascade + mixer + motor lag + RK4 rigid body + post-step,
// for K consecutive makeStep(dt) calls per launch.  One thread per UAV, FP64, state in registers.
//
// What it computes, per UAV and per substep, is exactly UavSystem::makeStep (US:304-380):
//   cascade  Position -> Velocity -> Acceleration -> Attitude/Tilt -> Rate -> Mixer   (CTL/*.hpp)
//   MultirotorModel::setInput (MM:392-410), MultirotorModel::step (MM:220-286) with the
//   derivative MM:301-366 and odeint's classic RK4 (ODE/stepper/runge_kutta4.hpp:42-95).
// How it computes it is new (this is not a transcription):
//   * the re-orthonormalisation R*chol(R^T R)^-1 (MM:314-316, 249-253) uses the closed-form
//     inverse of the lower-triangular factor and three rsqrt, not a general 3x3 cofactor inverse
//     (17 divisions + 7 sqrt per derivative in the reference -> 4 rsqrt here);
//   * thrust/torque from the motor speeds and F_ext/m are hoisted out of the four RK stages
//     (the reference recomputes them from the frozen members every stage, MM:332-335, 346);
//   * drag c*pi*l^2*|v|^2 * v/|v| / m collapses to (c*pi*l^2/m)*|v| * v;
//   * the oblique projection of the heading vector (CTL/acceleration_controller.hpp:60-80,
//     seven dynamic matrices and a 2x2 LU) is its closed form (cos h, sin h, -(nx cos h+ny sin h)/nz);
//   * the SO(3) error needs only the six off-diagonal dot products of Rd^T R;
//   * RK4 keeps a running weighted sum instead of four stored slopes, and skips the zero-
//     coefficient terms odeint multiplies through (generic_rk_operations.hpp:30-68);
//   * reciprocals, reciprocal square roots and square roots are the hardware approximation
//     (MUFU.RCP64H / MUFU.RSQ64H, 2^-23) followed by ONE third-order Newton step in FP64 (error
//     ~2^-66 before the final rounding): branch-free, no slow-path calls; a division is a
//     multiplication by such a reciprocal (<= 2 ulp instead of correctly rounded);
//   * the NaN -> 0 scrub of the slopes (MM:361-365) and the NaN -> restore check (MM:228-233) first
//     screen the exponent fields with integer max (any Inf/NaN?) and only then do the exact test;
//   * exp(-dt/tau) of the motor lag (MM:244) comes from the parameter table (evaluated once per set and dt by
//     prep_params_kernel), 1/dt from the host; the integral of a rate PID whose ki is zero (the default) is dead state
//     and is neither loaded nor stored; the K > 1 staged kernels park the PID state in shared memory between substeps;
//   * every fused multiply-add is written out (`fma`) and the file is compiled with -fmad=false, so
//     that all instantiations of the kernel (direct / staged, K = 1 / K > 1, any register budget)
//     produce the same bits: K fused substeps equal K launches, a sharded swarm equals the unsharded one.
// All of these change results only at rounding level (<= a few ulp per operation); parity with the
// CPU oracle is asserted within the tolerances of DESIGN.md §5 by tests/test_step_parity.py.
//
// Roofline (DESIGN.md §4): ~0.4-0.8 kB of state traffic and ~2.6 kFLOP (as-written census) per
// UAV-step; FP64-pipe bound on B200 once K >= 2, close to balanced at K = 1.
#include <cstdlib>
#include <type_traits>

#pragma once
#include "internal.h"

namespace {

#define DEV __device__ __forceinline__

// 1/sqrt(x) for normal positive x: MUFU.RSQ64H seed (rel. error 2^-22.9) + one third-order step.
// x = 0 / negative / Inf / NaN give NaN or Inf garbage, as does the reference's Cholesky there.
DEV double rsqrt_fast(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double t = x * y;
  const double e = fma(-t, y, 1.0);
  const double p = fma(0.375, e, 0.5);
  return fma(y * e, p, y);
}
// 1/b for normal b: MUFU.RCP64H seed (2^-23) + one third-order step
DEV double rcp_fast(double b) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));
  const double e = fma(-b, r, 1.0);
  const double p = fma(e, e, e);
  return fma(r, p, r);
}
// sqrt(x); exact IEEE path only for the rare tiny / zero / negative / non-finite arguments
DEV double sqrt_fast(double x) {
  if (x > 1e-290 && x < 1e300) return x * rsqrt_fast(x);
  return sqrt(x);
}
DEV unsigned expo(double v) { return unsigned(__double2hiint(v)) & 0x7ff00000u; }

struct Vec3 {
  double x, y, z;
};
DEV Vec3 mk(double x, double y, double z) {
  Vec3 r;
  r.x = x;
  r.y = y;
  r.z = z;
  return r;
}
DEV Vec3   operator+(Vec3 a, Vec3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
DEV Vec3   operator-(Vec3 a, Vec3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
DEV Vec3   operator*(Vec3 a, double s) { return mk(a.x * s, a.y * s, a.z * s); }
DEV double dot(Vec3 a, Vec3 b) { return fma(a.x, b.x, fma(a.y, b.y, a.z * b.z)); }
DEV Vec3   cross(Vec3 a, Vec3 b) { return mk(fma(a.y, b.z, -(a.z * b.y)), fma(a.z, b.x, -(a.x * b.z)), fma(a.x, b.y, -(a.y * b.x))); }
DEV Vec3   fma3(Vec3 a, double s, Vec3 b) { return mk(fma(a.x, s, b.x), fma(a.y, s, b.y), fma(a.z, s, b.z)); }  // a*s + b
// Eigen normalized(): divide by the norm only if the squared norm is positive
DEV Vec3 normalized(Vec3 a) {
  const double z = dot(a, a);
  if (z > 1e-290 && z < 1e300) return a * rsqrt_fast(z);
  if (z > 0.0) return a * (1.0 / sqrt(z));
  return a;
}
DEV unsigned expo3(Vec3 a) { return max(expo(a.x), max(expo(a.y), expo(a.z))); }
DEV bool isnan3(Vec3 a) { return (a.x != a.x) | (a.y != a.y) | (a.z != a.z); }
DEV Vec3 nan0(Vec3 a) { return mk(a.x != a.x ? 0.0 : a.x, a.y != a.y ? 0.0 : a.y, a.z != a.z ? 0.0 : a.z); }

struct Rot {
  Vec3 c0, c1, c2;  // columns
};

// R * chol(R^T R)^-1  with chol = lower Cholesky factor L (MM:314-316 / MM:249-253); L^-1 is the
// closed form for a lower-triangular 3x3.  MRSB_CHOL_PARALLEL=1 is an experiment that derives the
// three pivots from the leading minors of G so that the reciprocal square roots are independent;
// measured on B200 it is not faster than the textbook recurrence (profiles/README.md), which
// stays the default.
#ifndef MRSB_CHOL_PARALLEL
#define MRSB_CHOL_PARALLEL 0
#endif
DEV Rot reortho(const Rot& R) {
  const double g00 = dot(R.c0, R.c0), g10 = dot(R.c1, R.c0), g20 = dot(R.c2, R.c0);
  const double g11 = dot(R.c1, R.c1), g21 = dot(R.c2, R.c1), g22 = dot(R.c2, R.c2);
#if !MRSB_CHOL_PARALLEL
  const double i00 = rsqrt_fast(g00);
  const double l10 = g10 * i00, l20 = g20 * i00;
  const double d1  = fma(-l10, l10, g11);
  const double i11 = rsqrt_fast(d1);
  const double l11 = d1 * i11;
  const double l21 = fma(-l20, l10, g21) * i11;
  const double d2  = fma(-l21, l21, fma(-l20, l20, g22));
  const double i22 = rsqrt_fast(d2);
#else
  const double m1  = fma(g00, g11, -(g10 * g10));
  const double c0  = fma(g11, g22, -(g21 * g21));
  const double c1  = fma(g10, g22, -(g21 * g20));
  const double c2  = fma(g10, g21, -(g11 * g20));
  const double det = fma(g00, c0, fma(-g10, c1, g20 * c2));
  const double i00 = rsqrt_fast(g00);
  const double r1  = rsqrt_fast(m1);
  const double rd  = rsqrt_fast(det);
  const double s00 = g00 * i00;  // sqrt(g00)  = L00
  const double s1  = m1 * r1;    // sqrt(m1)
  const double i11 = s00 * r1;   // 1 / L11
  const double l11 = s1 * i00;   // L11
  const double i22 = s1 * rd;    // 1 / L22
  const double l10 = g10 * i00, l20 = g20 * i00;
  const double l21 = fma(-l20, l10, g21) * i11;
#endif
  const double a10 = -(l10 * i00) * i11;
  const double a21 = -(l21 * i11) * i22;
  const double a20 = fma(l10, l21, -(l20 * l11)) * ((i00 * i11) * i22);
  Rot          N;
  N.c0 = fma3(R.c2, a20, fma3(R.c1, a10, R.c0 * i00));
  N.c1 = fma3(R.c2, a21, R.c1 * i11);
  N.c2 = R.c2 * i22;
  return N;
}

// quantities frozen over the four RK stages of one step (MM:332-350: members, not ODE state)
struct Frozen {
  double g;
  double thrust_m;  // thrust / mass
  double air_m;     // c*pi*l^2 / mass
  Vec3   f_m;       // F_ext / mass
  Vec3   tau;       // allocation torque + external moment
};

struct Slope {
  Vec3 dv, dw;
  Rot  dR;
};

// MultirotorModel::operator() (MM:301-366) without the x_dot = v rows (handled by the caller).
// NaN slopes are scrubbed to zero element by element (MM:361-365): always when EXACT, otherwise only
// after an integer screen of the exponent fields found something Inf/NaN.
// (Tried and dropped, profiles/r2/history.md: skipping the re-orthonormalisation in the first RK stage, whose input left the
// previous step's closing reortho — no measurable time at K = 1, and in open-loop tumbling flight the missing projection lets
// the trajectories drift from the reference's by 1e-3 m after 10 s instead of 1e-11 m.)
template <bool EXACT>
DEV Slope derivative(Vec3 v, const Rot& Rraw, Vec3 w, const Frozen& f, const DevParams* __restrict__ P, bool jdiag, Vec3 Jd, Vec3 Jdi, unsigned& screen) {
  Slope        k;
  const Rot    R     = reortho(Rraw);
  const double vv    = dot(v, v);
  const double sp    = vv * rsqrt_fast(vv);
  const double speed = vv > 1e-290 ? sp : 0.0;  // |v| < 1e-145 m/s: the drag term is zero to 1e-290
  const double kd    = f.air_m * speed;
  k.dv = mk(fma(-kd, v.x, fma(R.c2.x, f.thrust_m, f.f_m.x)), fma(-kd, v.y, fma(R.c2.y, f.thrust_m, f.f_m.y)),
            fma(-kd, v.z, fma(R.c2.z, f.thrust_m, f.f_m.z) - f.g));
  // R * [w]x
  k.dR.c0 = fma3(R.c1, w.z, R.c2 * -w.y);
  k.dR.c1 = fma3(R.c2, w.x, R.c0 * -w.z);
  k.dR.c2 = fma3(R.c0, w.y, R.c1 * -w.x);
  if (jdiag) {
    const Vec3 Jw = mk(Jd.x * w.x, Jd.y * w.y, Jd.z * w.z);
    const Vec3 r  = f.tau - cross(w, Jw);
    k.dw          = mk(r.x * Jdi.x, r.y * Jdi.y, r.z * Jdi.z);
  } else {
    const double* J  = P->J;
    const double* Ji = P->Jinv;
    const Vec3    Jw = mk(dot(mk(J[0], J[1], J[2]), w), dot(mk(J[3], J[4], J[5]), w), dot(mk(J[6], J[7], J[8]), w));
    const Vec3    r  = f.tau - cross(w, Jw);
    k.dw = mk(dot(mk(Ji[0], Ji[1], Ji[2]), r), dot(mk(Ji[3], Ji[4], Ji[5]), r), dot(mk(Ji[6], Ji[7], Ji[8]), r));
  }
  if (EXACT) {
    k.dv    = nan0(k.dv);
    k.dw    = nan0(k.dw);
    k.dR.c0 = nan0(k.dR.c0);
    k.dR.c1 = nan0(k.dR.c1);
    k.dR.c2 = nan0(k.dR.c2);
  } else {
    // screen: is any exponent field all ones, i.e. is anything Inf or NaN at all?  (rarely taken)
    screen = max(max(expo3(k.dv), expo3(k.dw)), max(expo3(k.dR.c0), max(expo3(k.dR.c1), expo3(k.dR.c2))));
    if (screen == 0x7ff00000u) {
      k.dv    = nan0(k.dv);
      k.dw    = nan0(k.dw);
      k.dR.c0 = nan0(k.dR.c0);
      k.dR.c1 = nan0(k.dR.c1);
      k.dR.c2 = nan0(k.dR.c2);
    }
  }
  return k;
}

struct Rigid {
  Vec3 x, v, w;
  Rot  R;
};

// odeint's classic RK4 (ODE/stepper/runge_kutta4.hpp:42-95) as a running weighted sum.
// Returns the non-finite screen of the four slope evaluations (always 0 when EXACT).
template <bool EXACT>
DEV unsigned rk4(const Rigid& a, Rigid& out, double dt, const Frozen& fz, const DevParams* __restrict__ P, bool jdiag, Vec3 Jd, Vec3 Jdi) {
  unsigned     screen = 0;
  const double h      = 0.5 * dt;
  Slope        k      = derivative<EXACT>(a.v, a.R, a.w, fz, P, jdiag, Jd, Jdi, screen);
  Vec3         sx = a.v, sv = k.dv, sw = k.dw;
  Rot          sR = k.dR;
  Vec3         vt = fma3(k.dv, h, a.v), wt = fma3(k.dw, h, a.w);
  Rot          Rt;
  Rt.c0 = fma3(k.dR.c0, h, a.R.c0);
  Rt.c1 = fma3(k.dR.c1, h, a.R.c1);
  Rt.c2 = fma3(k.dR.c2, h, a.R.c2);
#pragma unroll
  for (int stage = 0; stage < 2; stage++) {
    const double c = stage == 0 ? h : dt;
    k              = derivative<EXACT>(vt, Rt, wt, fz, P, jdiag, Jd, Jdi, screen);
    sx             = fma3(vt, 2.0, sx);
    sv             = fma3(k.dv, 2.0, sv);
    sw             = fma3(k.dw, 2.0, sw);
    sR.c0          = fma3(k.dR.c0, 2.0, sR.c0);
    sR.c1          = fma3(k.dR.c1, 2.0, sR.c1);
    sR.c2          = fma3(k.dR.c2, 2.0, sR.c2);
    vt             = fma3(k.dv, c, a.v);
    wt             = fma3(k.dw, c, a.w);
    Rt.c0          = fma3(k.dR.c0, c, a.R.c0);
    Rt.c1          = fma3(k.dR.c1, c, a.R.c1);
    Rt.c2          = fma3(k.dR.c2, c, a.R.c2);
  }
  k  = derivative<EXACT>(vt, Rt, wt, fz, P, jdiag, Jd, Jdi, screen);
  sx = sx + vt;
  sv = sv + k.dv;
  sw = sw + k.dw;
  sR.c0 = sR.c0 + k.dR.c0;
  sR.c1 = sR.c1 + k.dR.c1;
  sR.c2 = sR.c2 + k.dR.c2;
  const double h6 = dt * (1.0 / 6.0);
  out.x    = fma3(sx, h6, a.x);
  out.v    = fma3(sv, h6, a.v);
  out.w    = fma3(sw, h6, a.w);
  out.R.c0 = fma3(sR.c0, h6, a.R.c0);
  out.R.c1 = fma3(sR.c1, h6, a.R.c1);
  out.R.c2 = fma3(sR.c2, h6, a.R.c2);
  return screen;
}

// PIDController::update (CTL/pid.hpp:67-96)
DEV double pid(double e, double dt, double inv_dt, double kp, double kd, double ki, double sat, double aw, double& last, double& integ) {
  const double diff = (e - last) * inv_dt;
  last              = e;
  double u          = fma(ki, integ, fma(kd, diff, kp * e));
  if (sat > 0.0) {
    if (u >= sat) {
      u = sat;
    } else if (u <= -sat) {
      u = -sat;
    }
  }
  if (aw > 0.0 && fabs(u) < aw) integ = fma(e, dt, integ);
  return u;
}

DEV int signum(double v) { return (0.0 < v) - (v < 0.0); }

// attitude error vee( 1/2 (Rd^T R - R^T Rd) ) / 2  (CTL/attitude_controller.hpp:82-89)
DEV Vec3 attitude_error(const Rot& Rd, const Rot& R) {
  const double a12 = dot(Rd.c1, R.c2), a21 = dot(Rd.c2, R.c1);
  const double a20 = dot(Rd.c2, R.c0), a02 = dot(Rd.c0, R.c2);
  const double a01 = dot(Rd.c0, R.c1), a10 = dot(Rd.c1, R.c0);
  return mk((a12 - a21) * 0.5, (a20 - a02) * 0.5, (a01 - a10) * 0.5);
}

#ifndef MRSB_STEP_THREADS
#define MRSB_STEP_THREADS 128
#endif
// CTAs per SM the register allocator aims for.  Measured on B200 (profiles/r1_history.md): the K = 1
// kernels gain from 3 CTAs (168 registers, 12 warps per SM) except PositionCmd, whose extra PID
// state then spills; the K > 1 kernels keep PID state, command and motor speeds live across the
// substep loop and are faster with 2 CTAs (<= 255 registers, no spills).
#ifndef MRSB_STEP_MINB_K1
#define MRSB_STEP_MINB_K1 3
#endif
#ifndef MRSB_STEP_MINB
#define MRSB_STEP_MINB(ONE, MODE_T) (((ONE) && (MODE_T) != MRSB_POSITION_CMD) ? MRSB_STEP_MINB_K1 : 2)
#endif

// ---- TMA / mbarrier plumbing for the staged kernel ---------------------------------------------
DEV uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }
DEV void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
DEV void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
DEV void mbar_wait(uint64_t* bar, uint32_t phase) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MRSB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MRSB_DONE;\n"
      "bra MRSB_WAIT;\n"
      "MRSB_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(phase)
      : "memory");
}
// 1-D bulk copy global -> shared through the TMA unit, completion counted on `bar`
DEV void tma_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)), "l"(gmem_src),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// order-preserving code of a float (for integer min / max); fdec() in collide.cu is its inverse
DEV uint32_t fenc(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b >> 31) ? ~b : (b | 0x80000000u);
}
// Bounding box of the 32 UAVs of this warp, rounded outwards to float: six warp reductions (REDUX), one 24-byte row per warp.
// Lanes past the end of the shard contribute nothing; a NaN coordinate yields a NaN bound, which every reader treats as
// "cannot be excluded".
DEV void store_group_box(uint32_t* row, bool inside, Vec3 x) {
  const uint32_t full = 0xffffffffu;
  uint32_t lo0 = inside ? fenc(__double2float_rd(x.x)) : 0xFFFFFFFFu, lo1 = inside ? fenc(__double2float_rd(x.y)) : 0xFFFFFFFFu,
           lo2 = inside ? fenc(__double2float_rd(x.z)) : 0xFFFFFFFFu;
  uint32_t hi0 = inside ? fenc(__double2float_ru(x.x)) : 0u, hi1 = inside ? fenc(__double2float_ru(x.y)) : 0u, hi2 = inside ? fenc(__double2float_ru(x.z)) : 0u;
  lo0 = __reduce_min_sync(full, lo0);
  lo1 = __reduce_min_sync(full, lo1);
  lo2 = __reduce_min_sync(full, lo2);
  hi0 = __reduce_max_sync(full, hi0);
  hi1 = __reduce_max_sync(full, hi1);
  hi2 = __reduce_max_sync(full, hi2);
  if ((threadIdx.x & 31) == 0) {
    reinterpret_cast<uint2*>(row)[0] = make_uint2(lo0, lo1);
    reinterpret_cast<uint2*>(row)[1] = make_uint2(lo2, hi0);
    reinterpret_cast<uint2*>(row)[2] = make_uint2(hi1, hi2);
  }
}

// where one thread reads its UAV's inputs: tile base + lane, rows 128 doubles apart — either the
// tile in HBM (direct kernel) or its copy in shared memory (staged kernel)
struct TileIn {
  const double *st, *rpm, *pid, *cmd, *fext;
};

// NM_T: motors per UAV if uniform over the batch (4/6/8), 0 = read per UAV.  MODE_T: INPUT_MODE if
// uniform, -1 = read per UAV.  ONE: k_sub == 1 (no substep loop: PID state, commands and motor
// speeds are dead after their single use, which is worth ~60 registers).  `after_loads` runs once
// per thread after the last read through `in` (the staged kernel re-arms its TMA there).
template <int NM_T, int MODE_T, bool ONE, class Hook>
DEV void step_uav(const DevState& s, const TileIn& in, const int64_t tile, const uint32_t flags0, const DevParams* batch_params, const int32_t pset,
                  const double dt, const double inv_dt, const int k_sub_arg, const int any_moment, uint32_t& disp_bits, Hook after_loads,
                  double* park = nullptr) {
  // batch_params: the whole batch's single parameter set in the constant bank (staged kernel), or
  // nullptr -> this UAV's entry of the table in HBM (read-only path)
  const DevParams* __restrict__ P = batch_params ? batch_params : s.params + pset;
  const int k_sub = ONE ? 1 : k_sub_arg;
  static_assert(MRSB_STEP_THREADS == MRSB_TILE, "one CTA per 128-UAV tile");
  const int64_t i_raw  = tile * MRSB_TILE + threadIdx.x;
  const bool    inside = i_raw < s.n;  // lanes past the end of the last tile compute on padding and store nothing
  // ROSW:265: with iterate_without_input off, a UAV that never received a command is not stepped at all: nothing of it is stored
  const bool    valid  = inside && !((s.opts & STEP_OPT_NEED_INPUT) && !(flags0 & FLAG_HAD_INPUT));
  const int64_t i      = inside ? i_raw : s.n - 1;
  // tile base pointers: every access below is [pointer + compile-time offset]
  const double* const t_st   = in.st;
  const double* const t_rpm  = in.rpm;
  const double* const t_pid  = in.pid;
  const double* const t_cmd  = in.cmd;
  const double* const t_fext = in.fext;
  double* const o_st    = s.st + (tile * ST_ROWS) * MRSB_TILE + threadIdx.x;
  double* const o_rpm   = s.rpm + (tile * MRSB_NM) * MRSB_TILE + threadIdx.x;
  double* const o_pid   = s.pid + (tile * PID_ROWS) * MRSB_TILE + threadIdx.x;
  double* const o_imu   = s.imu + (tile * F3_ROWS) * MRSB_TILE + threadIdx.x;
  const double* const t_ff    = s.ff + (tile * FF_ROWS) * MRSB_TILE + threadIdx.x;
  const double* const t_mext  = s.mext + (tile * F3_ROWS) * MRSB_TILE + threadIdx.x;
  const double* const t_vprev = s.vprev + (tile * VPREV_ROWS) * MRSB_TILE + threadIdx.x;

  const int nm                    = NM_T > 0 ? NM_T : P->n_motors;
  const int mode0                 = MODE_T >= 0 ? MODE_T : int(s.mode[i]);
  uint32_t flags                  = flags0;

#define LD(tp, row) (tp)[(row) * MRSB_TILE]
#define ST(tp, row, val)                         \
  do {                                           \
    if (valid) (tp)[(row) * MRSB_TILE] = (val);  \
  } while (0)

  // ---- load state -------------------------------------------------------------------------
  Vec3 x = mk(LD(t_st, 0), LD(t_st, 1), LD(t_st, 2));
  const Vec3 x_start = x;  // for the displacement bound of the collision pass' neighbour lists
  Vec3 v = mk(LD(t_st, 3), LD(t_st, 4), LD(t_st, 5));
  Rot  R;
  R.c0   = mk(LD(t_st, 6), LD(t_st, 7), LD(t_st, 8));
  R.c1   = mk(LD(t_st, 9), LD(t_st, 10), LD(t_st, 11));
  R.c2   = mk(LD(t_st, 12), LD(t_st, 13), LD(t_st, 14));
  Vec3 w = mk(LD(t_st, 15), LD(t_st, 16), LD(t_st, 17));
  double rpm[MRSB_NM];
#pragma unroll
  for (int m = 0; m < MRSB_NM; m++) rpm[m] = (m < nm) ? LD(t_rpm, m) : 0.0;
  Vec3 vprev = v;
  if (flags & FLAG_VPREV) vprev = mk(LD(t_vprev, 0), LD(t_vprev, 1), LD(t_vprev, 2));
  const Vec3 fext = mk(LD(t_fext, 0), LD(t_fext, 1), LD(t_fext, 2));
  Vec3       mext = mk(0, 0, 0);
  if (any_moment) mext = mk(LD(t_mext, 0), LD(t_mext, 1), LD(t_mext, 2));

  const bool live = !(flags & FLAG_CRASHED) && mode0 != MRSB_INPUT_UNKNOWN;  // US:308
  // which controllers are on this UAV's path (decides which PID rows are touched)
  const bool on_pos  = live && mode0 == MRSB_POSITION_CMD;
  const bool on_vel  = live && mode0 >= MRSB_VELOCITY_HDG_RATE_CMD;
  const bool on_att  = live && mode0 >= MRSB_ATTITUDE_CMD;
  const bool on_rate = live && mode0 >= MRSB_ATTITUDE_RATE_CMD;

  // PID state of PID k (0-2 position, 3-5 velocity, 6-8 attitude, 9-11 rate): last error in row k, integral in row 12 + k.
  // A rate PID whose ki is zero (the default, CTL/rate_controller.hpp:62-64: gains (4, .04, 0) * J_ii) never reads its integral, and
  // every way of changing ki (setParams, setRateControllerParams) resets it: the three rows are dead and neither loaded nor stored.
#define RATE_INT (P->rate_ki[0] != 0.0 || P->rate_ki[1] != 0.0 || P->rate_ki[2] != 0.0)
  double pe[12], pi[12];
#pragma unroll
  for (int k = 0; k < 12; k++) {
    const bool on = k < 3 ? on_pos : (k < 6 ? on_vel : (k < 9 ? on_att : on_rate));
    pe[k]         = on ? LD(t_pid, k) : 0.0;
    pi[k]         = (on && (k < 9 || RATE_INT)) ? LD(t_pid, 12 + k) : 0.0;
  }

  // command payload
  double c[CMD_ROWS];
#pragma unroll
  for (int r = 0; r < CMD_ROWS; r++) c[r] = 0.0;
  if (live) {
    if (mode0 == MRSB_ACTUATOR_CMD) {
#pragma unroll
      for (int m = 0; m < MRSB_NM; m++)
        if (m < nm) c[m] = LD(t_cmd, m);
    } else if (mode0 == MRSB_ATTITUDE_CMD) {
#pragma unroll
      for (int r = 0; r < 10; r++) c[r] = LD(t_cmd, r);
    } else {
#pragma unroll
      for (int r = 0; r < 4; r++) c[r] = LD(t_cmd, r);
      if (mode0 == MRSB_TILT_HDG_RATE_CMD) c[4] = LD(t_cmd, 4);
      if (mode0 == MRSB_POSITION_CMD || mode0 == MRSB_VELOCITY_HDG_CMD || mode0 == MRSB_ACCELERATION_HDG_CMD) {
        c[CMD_COS] = LD(t_cmd, CMD_COS);
        c[CMD_SIN] = LD(t_cmd, CMD_SIN);
      }
    }
  }
  // sticky feed-forwards (US:318-346)
  Vec3   ff_vel = mk(0, 0, 0), ff_acc = mk(0, 0, 0);
  double ff_hdg_rate = 0.0;
  if (on_pos) {
    if (flags & FLAG_FF_VEL_HDG) {
      ff_vel = mk(LD(t_ff, FF_VEL_HDG + 0), LD(t_ff, FF_VEL_HDG + 1), LD(t_ff, FF_VEL_HDG + 2));
    } else if (flags & FLAG_FF_VEL_HDG_RATE) {
      ff_vel = mk(LD(t_ff, FF_VEL_HDG_RATE + 0), LD(t_ff, FF_VEL_HDG_RATE + 1), LD(t_ff, FF_VEL_HDG_RATE + 2));
    }
  }
  if (on_vel) {
    const bool hdg_branch = mode0 != MRSB_VELOCITY_HDG_RATE_CMD;  // POSITION and VELOCITY_HDG go through ACCELERATION_HDG
    const bool has_a      = flags & FLAG_FF_ACC_HDG;
    const bool has_ar     = flags & FLAG_FF_ACC_HDG_RATE;
    // hdg branch: acc_hdg first, else acc_hdg_rate (US:330-334); rate branch: acc_hdg_rate first (+heading_rate), else acc_hdg (US:341-346)
    const bool use_ar = hdg_branch ? (!has_a && has_ar) : has_ar;
    const bool use_a  = hdg_branch ? has_a : (!has_ar && has_a);
    if (use_a) ff_acc = mk(LD(t_ff, FF_ACC_HDG + 0), LD(t_ff, FF_ACC_HDG + 1), LD(t_ff, FF_ACC_HDG + 2));
    if (use_ar) {
      ff_acc = mk(LD(t_ff, FF_ACC_HDG_RATE + 0), LD(t_ff, FF_ACC_HDG_RATE + 1), LD(t_ff, FF_ACC_HDG_RATE + 2));
      if (!hdg_branch) ff_hdg_rate = LD(t_ff, FF_ACC_HDG_RATE + 3);
    }
  }
  const double initz = (flags & FLAG_TAKEOFF) ? s.initz[i] : 0.0;

  after_loads();  // nothing below reads through `in`

  // ---- per-launch constants ---------------------------------------------------------------
  const double filt     = P->filt;  // exp(-dt / tau), MM:244 (prep_params_kernel)
  const double inv_mass = P->inv_mass;
  const double g        = P->g;
  const bool   jdiag    = P->j_diagonal != 0;
  const Vec3   Jd       = mk(P->J[0], P->J[4], P->J[8]);
  const Vec3   Jdi      = mk(P->Jinv[0], P->Jinv[4], P->Jinv[8]);
  const double min_rpm = P->min_rpm, rpm_range = P->rpm_range;
  const double inv_nm  = 1.0 / double(nm);

  Vec3 imu = mk(0, 0, 0);

  // K > 1 staged kernels: the PID state (up to 24 doubles) would stay live across the whole substep loop on top of the RK4's live
  // set — more than 255 registers hold.  It waits in a private column of shared memory between the cascades instead
  // (`park`: 24 rows of 128 doubles).
  volatile double* const pk = (!ONE && park) ? park + threadIdx.x : nullptr;
  // first PID that can be on this kernel's path (12: none, e.g. ActuatorCmd): the others are never touched
  constexpr int kPidLo = MODE_T < 0 ? 0 : MODE_T == MRSB_POSITION_CMD ? 0 : MODE_T >= MRSB_VELOCITY_HDG_RATE_CMD ? 3 : MODE_T >= MRSB_ATTITUDE_CMD ? 6 : MODE_T >= MRSB_ATTITUDE_RATE_CMD ? 9 : 12;
  if (!ONE && pk) {
#pragma unroll
    for (int k = kPidLo; k < 12; k++) {
      pk[k * MRSB_TILE]        = pe[k];
      pk[(12 + k) * MRSB_TILE] = pi[k];
    }
  }

  for (int sub = 0; sub < k_sub; sub++) {
    if (!ONE && pk) {
#pragma unroll
      for (int k = kPidLo; k < 12; k++) {
        pe[k] = pk[k * MRSB_TILE];
        pi[k] = pk[(12 + k) * MRSB_TILE];
      }
    }
    // ======================= controller cascade (US:304-374) =================================
    double u[MRSB_NM];
#pragma unroll
    for (int m = 0; m < MRSB_NM; m++) u[m] = 0.0;

    if (live) {
      int    mode = mode0;
      Vec3   vec  = mk(c[0], c[1], c[2]);  // position / velocity / acceleration / tilt / rates / roll-pitch-yaw
      double sc   = c[3];                  // heading | heading_rate | throttle
      double throttle = 0.0;
      Rot    Rd;
      Rd.c0 = Rd.c1 = Rd.c2 = mk(0, 0, 0);

      if (mode == MRSB_POSITION_CMD) {  // CTL/position_controller.hpp:73-86
        const Vec3   e   = vec - x;
        const double sat = P->pos_sat;
        vec.x = pid(e.x, dt, inv_dt, P->pos_kp, P->pos_kd, P->pos_ki, sat, 1.0, pe[0], pi[0]);
        vec.y = pid(e.y, dt, inv_dt, P->pos_kp, P->pos_kd, P->pos_ki, sat, 1.0, pe[1], pi[1]);
        vec.z = pid(e.z, dt, inv_dt, P->pos_kp, P->pos_kd, P->pos_ki, sat, 1.0, pe[2], pi[2]);
        vec   = vec + ff_vel;
        mode  = MRSB_VELOCITY_HDG_CMD;
      }
      if (mode == MRSB_VELOCITY_HDG_CMD || mode == MRSB_VELOCITY_HDG_RATE_CMD) {  // CTL/velocity_controller.hpp:68-102
        const Vec3   e   = vec - v;
        const double sat = P->vel_sat;
        vec.x = pid(e.x, dt, inv_dt, P->vel_kp, P->vel_kd, P->vel_ki, sat, 1.0, pe[3], pi[3]);
        vec.y = pid(e.y, dt, inv_dt, P->vel_kp, P->vel_kd, P->vel_ki, sat, 1.0, pe[4], pi[4]);
        vec.z = pid(e.z, dt, inv_dt, P->vel_kp, P->vel_kd, P->vel_ki, sat, 1.0, pe[5], pi[5]);
        vec   = vec + ff_acc;
        sc += ff_hdg_rate;
        mode = (mode == MRSB_VELOCITY_HDG_CMD) ? MRSB_ACCELERATION_HDG_CMD : MRSB_ACCELERATION_HDG_RATE_CMD;
      }
      if (mode == MRSB_ACCELERATION_HDG_CMD || mode == MRSB_ACCELERATION_HDG_RATE_CMD) {  // CTL/acceleration_controller.hpp:44-122
        const double mass = P->mass;
        const Vec3   fd   = mk(vec.x * mass, vec.y * mass, (vec.z + g) * mass);
        const Vec3   n    = normalized(fd);
        const double tf   = dot(fd, R.c2);
        throttle          = (sqrt_fast(tf * P->inv_kf_n) - min_rpm) * P->inv_rpm_range;
        if (mode == MRSB_ACCELERATION_HDG_CMD) {
          const double ch = c[CMD_COS], sh = c[CMD_SIN];
          const double num = fma(n.x, ch, n.y * sh);
          const double z3  = (num == 0.0) ? 0.0 : -num * rcp_fast(n.z);
          Rd.c2            = n;
          Rd.c0            = normalized(mk(ch, sh, z3));
          Rd.c1            = normalized(cross(Rd.c2, Rd.c0));
          mode             = MRSB_ATTITUDE_CMD;
        } else {
          vec  = n;  // tilt vector; sc stays the heading rate
          mode = MRSB_TILT_HDG_RATE_CMD;
        }
      } else if (mode == MRSB_ATTITUDE_CMD) {
        Rd.c0    = mk(c[0], c[1], c[2]);
        Rd.c1    = mk(c[3], c[4], c[5]);
        Rd.c2    = mk(c[6], c[7], c[8]);
        throttle = c[9];
      } else if (mode == MRSB_TILT_HDG_RATE_CMD) {
        throttle = c[4];
      } else {
        throttle = c[3];  // ATTITUDE_RATE / CONTROL_GROUP
      }

      if (mode == MRSB_ATTITUDE_CMD || mode == MRSB_TILT_HDG_RATE_CMD) {  // CTL/attitude_controller.hpp:79-145
        const bool tilt = (mode == MRSB_TILT_HDG_RATE_CMD);
        if (tilt) {
          Rd.c2 = normalized(vec);
          Rd.c1 = normalized(cross(Rd.c2, R.c0));
          Rd.c0 = normalized(cross(Rd.c1, Rd.c2));
        }
        const Vec3 e = attitude_error(Rd, R);
        double rx = pid(e.x, dt, inv_dt, P->att_kp, P->att_kd, P->att_ki, P->att_sat_rp, 0.1, pe[6], pi[6]);
        double ry = pid(e.y, dt, inv_dt, P->att_kp, P->att_kd, P->att_ki, P->att_sat_rp, 0.1, pe[7], pi[7]);
        double rz = pid(e.z, dt, inv_dt, P->att_kp, P->att_kd, P->att_ki, P->att_sat_yaw, 0.1, pe[8], pi[8]);
        if (tilt) {
          // intrinsicBodyRateToHeadingRate (:177-206): d/dt atan2(R10, R00) under body rates (rx,ry,rz)
          const double rd00 = fma(R.c1.x, rz, -(R.c2.x * ry));  // (R*[w]x)(0,0)
          const double rd10 = fma(R.c1.y, rz, -(R.c2.y * ry));  // (R*[w]x)(1,0)
          const double hx = R.c0.x, hy = R.c0.y;
          const double den = fma(hx, hx, hy * hy);
          double       parasitic = 0.0;
          if (!(fabs(den) <= 1e-5)) {
            const double iden = rcp_fast(den);
            parasitic         = fma(-hy * iden, rd00, (hx * iden) * rd10);
          }
          // getYawRateIntrinsic (:212-251)
          const double hr  = sc - parasitic;
          double       yaw = 0.0;
          if (!(fabs(hr) < 1e-3)) {
            const Vec3   orb  = mk(-hr * hy, hr * hx, 0.0);
            const Vec3   b    = normalized(mk(-hy, hx, 0.0));
            const double bp   = dot(b, R.c1);
            const Vec3   proj = b * bp;
            const double on = sqrt_fast(dot(orb, orb)), pn = sqrt_fast(dot(proj, proj));
            if (!(fabs(pn) < 1e-5)) {
              const double o = double(signum(dot(orb, proj))) * (on * rcp_fast(pn));
              yaw            = isfinite(o) ? o : 0.0;
            }
          }
          rz += yaw;
        }
        vec  = mk(rx, ry, rz);
        mode = MRSB_ATTITUDE_RATE_CMD;
      }
      if (mode == MRSB_ATTITUDE_RATE_CMD) {  // CTL/rate_controller.hpp:67-81
        const Vec3 e = vec - w;
        vec.x = pid(e.x, dt, inv_dt, P->rate_kp[0], P->rate_kd[0], P->rate_ki[0], -1.0, 1.0, pe[9], pi[9]);
        vec.y = pid(e.y, dt, inv_dt, P->rate_kp[1], P->rate_kd[1], P->rate_ki[1], -1.0, 1.0, pe[10], pi[10]);
        vec.z = pid(e.z, dt, inv_dt, P->rate_kp[2], P->rate_kd[2], P->rate_ki[2], -1.0, 1.0, pe[11], pi[11]);
        mode  = MRSB_CONTROL_GROUP_CMD;
      }
      if (mode == MRSB_CONTROL_GROUP_CMD) {  // CTL/mixer.hpp:107-144
        double mn = 1e300, mx = -1e300, sum = 0.0;
#pragma unroll
        for (int m = 0; m < MRSB_NM; m++) {
          if (m < nm) {
            u[m] = fma(P->mix[m][0], vec.x, P->mix[m][1] * vec.y) + fma(P->mix[m][2], vec.z, P->mix[m][3] * throttle);
            mn   = fmin(mn, u[m]);
          }
        }
        if (P->mixer_desaturation) {
          // fmin/fmax drop NaN operands; Eigen's minCoeff/maxCoeff comparisons also never select a NaN after a number
          if (mn < 0.0) {
            const double sh = fabs(mn);
#pragma unroll
            for (int m = 0; m < MRSB_NM; m++)
              if (m < nm) u[m] += sh;
          }
#pragma unroll
          for (int m = 0; m < MRSB_NM; m++)
            if (m < nm) {
              mx = fmax(mx, u[m]);
              sum += u[m];
            }
          if (mx > 1.0) {
            if (throttle > 1e-2) {
              const double isc = throttle * rcp_fast(sum * inv_nm);  // 1 / (mean(m) / throttle)
              const double r0 = vec.x * isc, r1 = vec.y * isc, r2 = vec.z * isc;
#pragma unroll
              for (int m = 0; m < MRSB_NM; m++)
                if (m < nm) u[m] = fma(P->mix[m][0], r0, P->mix[m][1] * r1) + fma(P->mix[m][2], r2, P->mix[m][3] * throttle);
            } else {
              const double imx = rcp_fast(mx);
#pragma unroll
              for (int m = 0; m < MRSB_NM; m++)
                if (m < nm) u[m] *= imx;
            }
          }
        }
      } else {  // ACTUATOR_CMD
#pragma unroll
        for (int m = 0; m < MRSB_NM; m++) u[m] = c[m];
      }
    }

    const bool last = ONE || (sub == k_sub - 1);
    if (!ONE && pk && !last) {
#pragma unroll
      for (int k = kPidLo; k < 12; k++) {
        pk[k * MRSB_TILE]        = pe[k];
        pk[(12 + k) * MRSB_TILE] = pi[k];
      }
    }
    if (last) {  // controller state is final for this launch: store it now, not after the RK4 (register pressure)
#pragma unroll
      for (int k = 0; k < 12; k++) {
        const bool on = k < 3 ? on_pos : (k < 6 ? on_vel : (k < 9 ? on_att : on_rate));
        if (on) {
          ST(o_pid, k, pe[k]);
          if (k < 9 || RATE_INT) ST(o_pid, 12 + k, pi[k]);
        }
      }
    }

    // ======================= MultirotorModel::setInput (MM:392-410) ==========================
    // ... and the parts of MultirotorModel::step that only need the motor speeds: allocation
    // (MM:332-335, frozen over the RK stages) and the first-order lag (MM:244-246), which does not
    // depend on the integration result and is therefore done (and stored) before it.
    Frozen fz;
    double usum = 0.0;
    {
      double t0 = 0, t1 = 0, t2 = 0, t3 = 0;
#pragma unroll
      for (int m = 0; m < MRSB_NM; m++) {
        if (m < nm) {
          double val = u[m];
          if (!isfinite(val)) val = 0.0;
          val = val < 0.0 ? 0.0 : (val > 1.0 ? 1.0 : val);
          const double target = fma(rpm_range, val, min_rpm);
          usum += target;
          const double sq = rpm[m] * rpm[m];
          t0 = fma(P->alloc[0][m], sq, t0);
          t1 = fma(P->alloc[1][m], sq, t1);
          t2 = fma(P->alloc[2][m], sq, t2);
          t3 = fma(P->alloc[3][m], sq, t3);
          rpm[m] = fma(filt, rpm[m], (1.0 - filt) * target);
          if (last) ST(o_rpm, m, rpm[m]);
        }
      }
      fz.g        = g;
      fz.thrust_m = t3 * inv_mass;
      fz.air_m    = P->air_k * inv_mass;
      fz.f_m      = fext * inv_mass;
      fz.tau      = mk(t0, t1, t2) + mext;
    }

    // classic RK4
    Rigid cur, nxt;
    cur.x = x;
    cur.v = v;
    cur.w = w;
    cur.R = R;
    rk4<false>(cur, nxt, dt, fz, P, jdiag, Jd, Jdi);

    // MM:228-233: any NaN -> keep the pre-step state
    bool bad = false;
    if (max(max(expo3(nxt.x), expo3(nxt.v)), max(max(expo3(nxt.w), expo3(nxt.R.c0)), max(expo3(nxt.R.c1), expo3(nxt.R.c2)))) == 0x7ff00000u)
      bad = isnan3(nxt.x) | isnan3(nxt.v) | isnan3(nxt.w) | isnan3(nxt.R.c0) | isnan3(nxt.R.c1) | isnan3(nxt.R.c2);
    if (!bad) {
      x = nxt.x;
      v = nxt.v;
      w = nxt.w;
      R = nxt.R;
    }

    R = reortho(R);  // MM:249-253

    if (P->ground_enabled) {  // MM:256-262
      if (x.z < P->ground_z && v.z < 0.0) {
        x.z = P->ground_z;
        v   = mk(0, 0, 0);
        w   = mk(0, 0, 0);
      }
    }
    if (flags & FLAG_TAKEOFF) {  // MM:264-277
      if (usum * inv_nm <= P->takeoff_rpm) {
        if (x.z < initz && v.z < 0.0) {
          x.z = initz;
          v   = mk(0, 0, 0);
          w   = mk(0, 0, 0);
        }
      } else {
        flags &= ~FLAG_TAKEOFF;
      }
    }

    // MM:280-281 fabricated accelerometer
    const Vec3 lin = mk((v.x - vprev.x) * inv_dt, (v.y - vprev.y) * inv_dt, fma(v.z - vprev.z, inv_dt, g));
    imu            = mk(dot(R.c0, lin), dot(R.c1, lin), dot(R.c2, lin));
    vprev          = v;
  }

  // ---- store ------------------------------------------------------------------------------
  ST(o_st, 0, x.x);
  ST(o_st, 1, x.y);
  ST(o_st, 2, x.z);
  ST(o_st, 3, v.x);
  ST(o_st, 4, v.y);
  ST(o_st, 5, v.z);
  ST(o_st, 6, R.c0.x);
  ST(o_st, 7, R.c0.y);
  ST(o_st, 8, R.c0.z);
  ST(o_st, 9, R.c1.x);
  ST(o_st, 10, R.c1.y);
  ST(o_st, 11, R.c1.z);
  ST(o_st, 12, R.c2.x);
  ST(o_st, 13, R.c2.y);
  ST(o_st, 14, R.c2.z);
  ST(o_st, 15, w.x);
  ST(o_st, 16, w.y);
  ST(o_st, 17, w.z);
  if (s.opts & STEP_OPT_IMU) {
    ST(o_imu, 0, imu.x);
    ST(o_imu, 1, imu.y);
    ST(o_imu, 2, imu.z);
  }
  const uint32_t new_flags = flags & ~FLAG_VPREV;
  if (!valid) x = x_start;  // frozen: its position is published unchanged
  if (valid) {
    // squared displacement of this launch as float bits, rounded up (NaN keeps the largest pattern)
    const double ddx = x.x - x_start.x, ddy = x.y - x_start.y, ddz = x.z - x_start.z;
    disp_bits = max(disp_bits, __float_as_uint(fabsf(__double2float_ru(fma(ddx, ddx, fma(ddy, ddy, ddz * ddz))))));
    if (new_flags != flags0) s.flags[i] = new_flags;
  }
  if (inside && (s.opts & STEP_OPT_GPOS)) {
    // packed position for the collision pass / position download / the peers that pull it over NVLink (external index order)
    double* gp = s.gpos + 3 * (s.shard_begin + (s.inv ? int64_t(s.inv[i]) : i));
    gp[0]      = x.x;
    gp[1]      = x.y;
    gp[2]      = x.z;
  }
  if (s.gbox) store_group_box(s.gbox + 6 * (tile * (MRSB_TILE / 32) + (threadIdx.x >> 5)), inside, x);
#undef LD
#undef ST
#undef RATE_INT
}

// Largest squared displacement of the launch (float bits) -> DevState::disp_max: one atomic per warp
// at most, and none once the word already holds a value at least as large.
DEV void report_displacement(const DevState& s, uint32_t disp_bits) {
  if (!s.disp_max) return;
  disp_bits = __reduce_max_sync(0xffffffffu, disp_bits);
  if ((threadIdx.x & 31) == 0 && disp_bits > *reinterpret_cast<volatile uint32_t*>(s.disp_max)) atomicMax(s.disp_max, disp_bits);
}

// ---- direct kernel: one CTA per tile, inputs read straight from HBM ----------------------------
template <int NM_T, int MODE_T, bool ONE>
__global__ void __launch_bounds__(MRSB_STEP_THREADS, MRSB_STEP_MINB(ONE, MODE_T))
    uav_step_kernel(DevState s, double dt, double inv_dt, int k_sub, int any_moment) {
  const int64_t tile = blockIdx.x;
  TileIn        in;
  in.st   = s.st + (tile * ST_ROWS) * MRSB_TILE + threadIdx.x;
  in.rpm  = s.rpm + (tile * MRSB_NM) * MRSB_TILE + threadIdx.x;
  in.pid  = s.pid + (tile * PID_ROWS) * MRSB_TILE + threadIdx.x;
  in.cmd  = s.cmd + (tile * CMD_ROWS) * MRSB_TILE + threadIdx.x;
  in.fext = s.fext + (tile * F3_ROWS) * MRSB_TILE + threadIdx.x;
  const int64_t i = min(tile * MRSB_TILE + threadIdx.x, s.n - 1);
  uint32_t disp_bits = 0u;
  step_uav<NM_T, MODE_T, ONE>(s, in, tile, s.flags[i], nullptr, s.pset[s.shard_begin + (s.inv ? int64_t(s.inv[i]) : i)], dt, inv_dt, k_sub, any_moment, disp_bits,
                              [] {});
  report_displacement(s, disp_bits);
}

// ---- staged kernel: persistent CTAs, the NEXT tile's inputs are fetched by the TMA unit into
// shared memory while the current tile is being integrated out of registers ----------------------
// shared-memory tile image (rows of 128 doubles): st 18 | rpm n | pid rows on the mode's path | command rows of the mode | fext 3
// Image layout of one instantiation: only the rows the mode touches take space (44-50 KiB for the velocity modes of a quad
// instead of 65), so that more CTAs fit per SM.  PID rows keep their spacing (last error of PID k in image row k - pid_lo of the
// PID block, integral in row 12 + k - pid_lo: one pointer serves both), which leaves pid_lo unused rows between the two groups.
template <int NM_T, int MODE_T>
struct Img {
  static constexpr int  pid_lo   = MODE_T == MRSB_POSITION_CMD ? 0 : MODE_T >= MRSB_VELOCITY_HDG_RATE_CMD ? 3 : MODE_T >= MRSB_ATTITUDE_CMD ? 6 : MODE_T >= MRSB_ATTITUDE_RATE_CMD ? 9 : 12;
  static constexpr int  cmd_rows = MODE_T == MRSB_ACTUATOR_CMD ? NM_T : MODE_T == MRSB_ATTITUDE_CMD ? 10 : MODE_T == MRSB_TILT_HDG_RATE_CMD ? 5 : 4;
  static constexpr bool hdg      = MODE_T == MRSB_POSITION_CMD || MODE_T == MRSB_VELOCITY_HDG_CMD || MODE_T == MRSB_ACCELERATION_HDG_CMD;
  static constexpr int  ST       = 0;
  static constexpr int  RPM      = ST + ST_ROWS;
  static constexpr int  PID      = RPM + NM_T;                         // image row of PID row `pid_lo`
  static constexpr int  CMD      = PID + (pid_lo < 12 ? PID_ROWS - pid_lo : 0);
  static constexpr int  FEXT     = CMD + (hdg ? CMD_ROWS : cmd_rows);  // the cached cos / sin sit in command rows 10, 11
  static constexpr int  ROWS     = FEXT + F3_ROWS;
};

template <int NM_T, int MODE_T>
DEV void stage_tile(const DevState& s, const DevParams& P, double* sm, uint64_t* bar, int64_t tile) {
  static_assert(MODE_T >= 0 && NM_T > 0, "the staged kernel is for batches with a uniform input mode and motor count");
  using I = Img<NM_T, MODE_T>;
  const bool     rate_int = P.rate_ki[0] != 0.0 || P.rate_ki[1] != 0.0 || P.rate_ki[2] != 0.0;  // same test as step_uav
  constexpr int  kRow     = MRSB_TILE * int(sizeof(double));
  constexpr int  pid_lo   = I::pid_lo;
  // integrals: rows 12 + pid_lo .. 23, without the three dead rate integrals when their ki is zero
  const int      int_rows = pid_lo < 12 ? (rate_int ? 12 - pid_lo : 9 - pid_lo) : 0;
  const uint32_t bytes    = uint32_t(kRow) * uint32_t(ST_ROWS + NM_T + (12 - pid_lo) + int_rows + I::cmd_rows + (I::hdg ? 2 : 0) + F3_ROWS);
  mbar_expect_tx(bar, bytes);
  tma_load(sm + I::ST * MRSB_TILE, s.st + (tile * ST_ROWS) * MRSB_TILE, kRow * ST_ROWS, bar);
  tma_load(sm + I::RPM * MRSB_TILE, s.rpm + (tile * MRSB_NM) * MRSB_TILE, kRow * NM_T, bar);
  if (pid_lo < 12) tma_load(sm + I::PID * MRSB_TILE, s.pid + (tile * PID_ROWS + pid_lo) * MRSB_TILE, kRow * (12 - pid_lo), bar);
  if (int_rows > 0) tma_load(sm + (I::PID + 12) * MRSB_TILE, s.pid + (tile * PID_ROWS + 12 + pid_lo) * MRSB_TILE, uint32_t(kRow) * uint32_t(int_rows), bar);
  tma_load(sm + I::CMD * MRSB_TILE, s.cmd + (tile * CMD_ROWS) * MRSB_TILE, kRow * I::cmd_rows, bar);
  if (I::hdg) tma_load(sm + (I::CMD + CMD_COS) * MRSB_TILE, s.cmd + (tile * CMD_ROWS + CMD_COS) * MRSB_TILE, kRow * 2, bar);
  tma_load(sm + I::FEXT * MRSB_TILE, s.fext + (tile * F3_ROWS) * MRSB_TILE, kRow * F3_ROWS, bar);
}

template <int NM_T, int MODE_T, bool ONE>
__global__ void __launch_bounds__(MRSB_STEP_THREADS, MRSB_STEP_MINB(ONE, MODE_T))
    uav_step_staged_kernel(DevState s, const __grid_constant__ DevParams params, double dt, double inv_dt, int k_sub, int any_moment, int64_t n_tiles,
                           uint32_t* sweep) {
  // `params`: the one parameter set of the whole batch, passed BY VALUE: it lives in the constant
  // bank, so airframe constants and gains are instruction operands instead of ~80 loads per UAV
  using I = Img<NM_T, MODE_T>;
  extern __shared__ __align__(128) double sm[];  // I::ROWS x 128 doubles (tile image) [+ PID_ROWS x 128: PID parking, K > 1]
  __shared__ uint64_t bar;
  __shared__ uint32_t ticket;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    // `sweep` (nullptr: always forward): every other launch walks the tiles from the end, so that it starts on those the previous
    // launch wrote last, while their lines are still in L2.  The word lives on the device because a captured tick graph replays the
    // same launch.  Each launch adds exactly 2^16 to it (CTA 0 adds 2^16 - (gridDim.x - 1), every other CTA 1), so whatever value
    // a CTA's add returns, its bit 16 is the parity of the launch — one atomic per CTA, nothing to wait for at the end.
    ticket = sweep ? atomicAdd(sweep, blockIdx.x == 0 ? 65536u - (gridDim.x - 1u) : 1u) : 0u;
  }
  __syncthreads();
  // a CTA's k-th tile is blockIdx.x + k * gridDim.x, counted from the end on a backward sweep; tiles outside [0, n_tiles) end the
  // sweep.  The step is re-read from shared memory where it is needed rather than kept in a register across step_uav, whose live
  // set is what limits the register budget.
  const auto stride   = [&] { return ((*reinterpret_cast<volatile uint32_t*>(&ticket) >> 16) & 1u) ? -int64_t(gridDim.x) : int64_t(gridDim.x); };
  const auto in_range = [&](int64_t t) { return uint64_t(t) < uint64_t(n_tiles); };
  int64_t    tile     = ((ticket >> 16) & 1u) ? n_tiles - 1 - blockIdx.x : int64_t(blockIdx.x);
  if (threadIdx.x == 0 && in_range(tile)) stage_tile<NM_T, MODE_T>(s, params, sm, &bar, tile);
  TileIn in;
  in.st   = sm + I::ST * MRSB_TILE + threadIdx.x;
  in.rpm  = sm + I::RPM * MRSB_TILE + threadIdx.x;
  in.pid  = sm + (I::PID - I::pid_lo) * MRSB_TILE + threadIdx.x;  // addressed by PID row number; rows below pid_lo are never read
  in.cmd  = sm + I::CMD * MRSB_TILE + threadIdx.x;
  in.fext = sm + I::FEXT * MRSB_TILE + threadIdx.x;
  uint32_t phase = 0;
  // the per-UAV word that is not part of the tile image is prefetched one tile ahead
  int64_t  i0        = min(tile * MRSB_TILE + threadIdx.x, s.n - 1);
  uint32_t flags_cur = in_range(tile) ? s.flags[i0] : 0u;
  uint32_t disp_bits = 0u;
  for (; in_range(tile); tile += stride()) {
    const int64_t next       = tile + stride();
    uint32_t      flags_next = 0u;
    if (in_range(next)) flags_next = s.flags[min(next * MRSB_TILE + threadIdx.x, s.n - 1)];
    mbar_wait(&bar, phase);
    phase ^= 1u;
    step_uav<NM_T, MODE_T, ONE>(
        s, in, tile, flags_cur, &params, 0, dt, inv_dt, k_sub, any_moment, disp_bits,
        [&] {
          __syncthreads();  // every lane has its inputs in registers: the image may be overwritten
          if (threadIdx.x == 0 && in_range(next)) stage_tile<NM_T, MODE_T>(s, params, sm, &bar, next);
        },
        ONE ? nullptr : sm + I::ROWS * MRSB_TILE);
    flags_cur = flags_next;
  }
  report_displacement(s, disp_bits);
}

// CTAs of the staged kernel that fit on the device (persistent grid), cached per instantiation
template <int NM_T, int MODE_T, bool ONE>
int staged_grid(size_t smem) {
  static int cached = -1;
  if (cached < 0) {
    auto* k = uav_step_staged_kernel<NM_T, MODE_T, ONE>;
    if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)) != cudaSuccess) {
      cudaGetLastError();
      cached = 0;
      return cached;
    }
    int dev = 0, sms = 0, per_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, MRSB_STEP_THREADS, smem);
    cached = sms * per_sm;
  }
  return cached;
}

// L2 size of the current device, cached
inline int64_t l2_bytes() {
  static int64_t cached = -1;
  if (cached < 0) {
    int dev = 0, bytes = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&bytes, cudaDevAttrL2CacheSize, dev);
    cached = bytes;
  }
  return cached;
}

template <int NM_T, int MODE_T>
void launch_one(const DevState& s, const DevParams* uniform_params, uint32_t* sweep, double dt, int k, int any_moment, cudaStream_t st, int* info) {
  const int     threads = MRSB_STEP_THREADS;
  const int64_t n_tiles = (s.n + threads - 1) / threads;
  const double  inv_dt  = 1.0 / dt;
  info[2] = NM_T;
  info[3] = MODE_T;
  if constexpr (NM_T > 0 && MODE_T >= 0) if (uniform_params && !getenv("MRSB_NO_STAGING")) {
    // enough tiles to fill the machine more than once: persistent CTAs + TMA staging hide the HBM
    // latency behind the integration of the previous tile
    auto launch = [&](auto one) -> bool {
      constexpr bool kOne = decltype(one)::value;
      const size_t   smem = size_t(Img<NM_T, MODE_T>::ROWS + (kOne ? 0 : PID_ROWS)) * MRSB_TILE * sizeof(double);  // tile image (+ PID parking rows, K > 1)
      const int      grid = staged_grid<NM_T, MODE_T, kOne>(smem);
      if (grid <= 0 || n_tiles <= grid) return false;
      // alternating the direction pays only when the launch streams more than L2 holds: a smaller state stays resident either way
      const int64_t streamed = n_tiles * int64_t(Img<NM_T, MODE_T>::ROWS) * MRSB_TILE * int64_t(sizeof(double));
      uint32_t*     dir      = streamed > l2_bytes() ? sweep : nullptr;
      uav_step_staged_kernel<NM_T, MODE_T, kOne><<<grid, threads, smem, st>>>(s, *uniform_params, dt, inv_dt, k, any_moment, n_tiles, dir);
      info[0] = 2;
      info[1] = grid;
      return true;
    };
    if ((k == 1) ? launch(std::true_type{}) : launch(std::false_type{})) return;
  }
  info[0] = 1;
  info[1] = int(n_tiles);
  if (k == 1) {
    uav_step_kernel<NM_T, MODE_T, true><<<unsigned(n_tiles), threads, 0, st>>>(s, dt, inv_dt, k, any_moment);
  } else {
    uav_step_kernel<NM_T, MODE_T, false><<<unsigned(n_tiles), threads, 0, st>>>(s, dt, inv_dt, k, any_moment);
  }
}

template <int NM_T>
void launch_nm(const DevState& s, const DevParams* up, uint32_t* sweep, double dt, int k, int mode, int any_moment, cudaStream_t st, int* info) {
  switch (mode) {
    case MRSB_ACTUATOR_CMD:
      launch_one<NM_T, MRSB_ACTUATOR_CMD>(s, up, sweep, dt, k, any_moment, st, info);
      break;
    case MRSB_VELOCITY_HDG_RATE_CMD:
      launch_one<NM_T, MRSB_VELOCITY_HDG_RATE_CMD>(s, up, sweep, dt, k, any_moment, st, info);
      break;
    case MRSB_VELOCITY_HDG_CMD:
      launch_one<NM_T, MRSB_VELOCITY_HDG_CMD>(s, up, sweep, dt, k, any_moment, st, info);
      break;
    case MRSB_POSITION_CMD:
      launch_one<NM_T, MRSB_POSITION_CMD>(s, up, sweep, dt, k, any_moment, st, info);
      break;
    default:
      launch_one<NM_T, -1>(s, up, sweep, dt, k, any_moment, st, info);
      break;
  }
}

}  // namespace

// one translation unit per motor count (step_kernel_nm{0,4,6,8}.cu) instantiates this, so that the
// ~40 kernel instantiations compile in parallel
template <int NM_T>
void launch_step_nm(const DevState& s, const DevParams* uniform_params, uint32_t* sweep, double dt, int k_substeps, int uniform_mode, bool any_moment,
                    cudaStream_t stream, int* info) {
  launch_nm<NM_T>(s, uniform_params, sweep, dt, k_substeps, uniform_mode, any_moment, stream, info);
}
