// tb_device.cuh - device-side dynamics of the tennisbot env step, templated on the arithmetic type.
//
// One thread owns one env and keeps its whole state in registers across every physics substep of an env step
// (up to 776 inside SwingRacket's 26th step) and across the K env steps of a fused rollout.  The scene
// (parameters + the two convex-prism edge tables) arrives as a __grid_constant__ kernel argument, so every
// table lookup is a uniform constant-bank load and contexts with different parameters can share a device.
//
// What is restated here (paths relative to the reference checkout; Bullet semantics per SURVEY.md Appendix A):
//   physics_step        <- pybullet.stepSimulation() as called at swingracket_env.py:82,107, tennisbot_env.py:121
//   contact bits        <- pybullet.getContactPoints at swingracket_env.py:99,111,119, tennisbot_env.py:170
//   swing/hit env logic <- swingracket_env.py:75-145, tennisbot_env.py:104-207
//   episode placement   <- swingracket_env.py:151-186, tennisbot_env.py:217-261
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tennisbot_b200.h"
#include "tb_scene_data.h"

namespace tb {

// rare-path hint: lets the compiler lay the cold block out of the substep loop's straight line (I-cache)
#define TB_UNLIKELY(x) __builtin_expect(!!(x), 0)

// ------------------------------------------------------------------------------------------------ math shims
template <typename T> struct M;
template <> struct M<float> {
  static __device__ __forceinline__ float sqrt(float x) { return sqrtf(x); }
  // 1-ulp hardware square root for the speed norms that only feed the damping factor k (1 + |v|)
  static __device__ __forceinline__ float sqrt_fast(float x) {
    float y;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
  }
  static __device__ __forceinline__ float norm_damp(float x2) { return sqrt_fast(x2); }
  static __device__ __forceinline__ float rsqrt(float x) { return 1.0f / sqrtf(x); }
  static __device__ __forceinline__ float abs(float x) { return fabsf(x); }
  static __device__ __forceinline__ void sincos(float x, float *s, float *c) { sincosf(x, s, c); }
  static __device__ __forceinline__ float inf() { return __int_as_float(0x7f800000); }
};
template <> struct M<double> {
  static __device__ __forceinline__ double sqrt(double x) { return ::sqrt(x); }
  // Speed norms that only feed the damping factor k (1 + |v|) need ~1e-10, not the last bit: float rsqrt estimate
  // (2^-22) + one Newton step in double = 1e-13 relative, half the instructions of the IEEE square root.
  static __device__ __forceinline__ double sqrt_fast(double x) {
    double y = (double)rsqrtf((float)x);
    y = y * (1.5 - 0.5 * x * y * y);
    return x > 1e-30 ? x * y : 0.0;
  }
  // the same without the zero test: the float estimate is taken of max(x, 1e-37), so x = 0 gives 0 and |v| below
  // 3e-19 is off by at most its own size (it enters only as 1 + |v|)
  static __device__ __forceinline__ double norm_damp(double x2) {
    float e;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(fmaxf((float)x2, 1e-37f)));
    double y = (double)e;
    y = y * (1.5 - 0.5 * x2 * y * y);
    return x2 * y;
  }
  static __device__ __forceinline__ double rsqrt(double x) { return 1.0 / ::sqrt(x); }
  static __device__ __forceinline__ double abs(double x) { return fabs(x); }
  static __device__ __forceinline__ void sincos(double x, double *s, double *c) { ::sincos(x, s, c); }
  static __device__ __forceinline__ double inf() { return __longlong_as_double(0x7ff0000000000000LL); }
};

__device__ __forceinline__ float clampv(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }
__device__ __forceinline__ double clampv(double x, double lo, double hi) { return fmin(fmax(x, lo), hi); }
// |x| >= vmax, decided on the exponent/high mantissa word alone (an integer compare; double min/max are multi-
// instruction sequences on sm_100).  `thr` is the high word of vmax; for double the test may fire a little below
// vmax, which only sends the caller into the exact clamp for nothing.
__device__ __forceinline__ bool near_limit(float x, unsigned thr) { return (__float_as_uint(x) & 0x7fffffffu) >= thr; }
__device__ __forceinline__ bool near_limit(double x, unsigned thr) { return ((unsigned)__double2hiint(x) & 0x7fffffffu) >= thr; }
// Bullet clamps every velocity coordinate to +-max_coord_vel whenever it writes one (btMultiBody::applyDeltaVee).
// The bound is never reached in these envs, so test all twelve coordinates with integer compares and clamp out of line.
template <typename T> __device__ __forceinline__ void clamp_velocities(T *bv, T *bw, T *rv, T *rw, T vmax, unsigned thr) {
  bool over = false;
#pragma unroll
  for (int i = 0; i < 3; ++i) over = over | near_limit(bv[i], thr) | near_limit(bw[i], thr) | near_limit(rv[i], thr) | near_limit(rw[i], thr);
  if (TB_UNLIKELY(over)) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      bv[i] = clampv(bv[i], -vmax, vmax); bw[i] = clampv(bw[i], -vmax, vmax);
      rv[i] = clampv(rv[i], -vmax, vmax); rw[i] = clampv(rw[i], -vmax, vmax);
    }
  }
}
__device__ __forceinline__ void opaque(double &x) { asm volatile("" : "+d"(x)); }
__device__ __forceinline__ void opaque(float &x) { asm volatile("" : "+f"(x)); }
template <typename T> __device__ __forceinline__ T dot3(const T *a, const T *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
template <typename T> __device__ __forceinline__ void cross3(const T *a, const T *b, T *o) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
template <typename T> __device__ __forceinline__ T norm3(const T *a) { return M<T>::sqrt(dot3(a, a)); }
template <typename T> __device__ __forceinline__ T norm3_fast(const T *a) { return M<T>::sqrt_fast(dot3(a, a)); }

// ------------------------------------------------------------------------------------------------ scene
// unroll depth of the loops over the edge tables: the entries are constant-bank loads with a lane-dependent index (long
// latency), and a lone lane of a server warp has nothing else to overlap them with
constexpr int kEdgeUnroll = 6;
constexpr int kBallVzEntries = 32;  // Scene::ball_vz (SwingRacket's control phase is 26 substeps long)
constexpr int kRacketEdges = TB_RACKET_OUTLINE_N;
constexpr int kGoalEdges = TB_GOAL_SIDES;

constexpr int kCoarseEdges = 18, kCoarseUnroll = 6;
template <typename T> struct Edge {
  T ax, ay, ex, ey, inv_len2, nx, ny;
};
template <typename T, int NE> struct Prism {
  Edge<T> e[NE];
  T half_thick, bound_radius;
  // Two regions that lie inside the outline for certain (prism_inside_fast): an ellipse centred on the v axis, shrunk on
  // the host until it clears every edge line, and the quadrilateral between two outline edges and two lines of constant v
  // (the racket's throat; tz_lo > tz_hi: none).  A ball that rests or rolls on the racket face, or lands on the goal
  // disc, is inside one of them, and the loops over the edge table are skipped.
  T in_c, in_inv_a, in_inv_b, tz_lo, tz_hi;
  T t_ax[2], t_ay[2], t_nx[2], t_ny[2];
  // ... and the converse (prism_outside_fast): out_a, out_b = semi-axes of an ellipse about the same centre that contains
  // every outline vertex at or above out_v (all of them when there is no quadrilateral); below out_v the outline lies
  // between the quadrilateral's two edge lines and above v = out_lo.
  T out_a, out_b, out_v, out_lo;
  T out_inv_a, out_inv_b;  // reciprocal semi-axes of the ellipse that contains the rim-neighbourhood of E(out_a, out_b), rim = ffp_rim
  // A coarse outline for what the two quick tests leave undecided: a subset of the edge lines (the long edges, and one of
  // every few along the arcs: a convex polygon that CONTAINS the outline and overshoots it by a millimetre or two), as
  // point + outward unit normal; unused entries repeat the first.  (ff_kernel's flight loop: a lane in the band between
  // the quick tests keeps 31 others waiting while it walks the edge table.)
  T c_ax[kCoarseEdges], c_ay[kCoarseEdges], c_nx[kCoarseEdges], c_ny[kCoarseEdges];
};
// true: (u, v) is strictly inside the outline (false says nothing)
template <typename T, int NE> __device__ __forceinline__ bool prism_inside_fast(const Prism<T, NE> &pr, T u, T v) {
  T du = u * pr.in_inv_a, dv = (v - pr.in_c) * pr.in_inv_b;
  bool ell = du * du + dv * dv < 1;
  bool quad = (v > pr.tz_lo) & (v < pr.tz_hi) & ((u - pr.t_ax[0]) * pr.t_nx[0] + (v - pr.t_ay[0]) * pr.t_ny[0] < 0) &
              ((u - pr.t_ax[1]) * pr.t_nx[1] + (v - pr.t_ay[1]) * pr.t_ny[1] < 0);
  return ell | quad;
}

template <typename T> struct Scene {
  T dt, gravity_z, lin_damping, ang_damping, max_coord_vel;
  T rest_racket, rest_court, rest_goal, mu_racket, mu_court, mu_goal;
  T erp, slop, rest_vel_threshold, solver_residual, contact_threshold, hull_margin, box_margin, gyro;
  int iters, shoot_start, shoot_frames;  // Tennisbot-v0: env steps on which the ball's shoot force acts (tennisbot_env.py:21,118)
  T ball_vz[kBallVzEntries];             // vz of a ball after k free-fall substeps from rest (kStPristine), filled on the device
  int racket_court;                      // 1: racket vs the court's floor box is modelled (parameter racket_court_contact), on the
                                         // generic path only: a state with TB_EV_RACKET_LOW never takes a straight-line substep then
  T rest_racket_court, mu_racket_court;
  unsigned vmax_hi;  // high 32 bits of max_coord_vel in T's format (clamp_velocities)
  T pid_kp, pid_ki, pid_kd, pid_lim, pid_bias_z, pid_hit_z;  // TB_CONTROL_PID (racket.py:47-64,103-122)
  T ball_r, ball_inv_m, ball_inv_i, racket_inv_m;
  T racket_i[3], racket_inv_i[3];
  T com_z;
  T swing_q[4], swing_off[3]; // spawn quaternion for rpy (0,0.5,0) and R*(0,0,com_z), built on the host in double
  T floor_h[3], net_h[3], goal_r, goal_hz;
  T racket_box[3];  // outline bounding box in the COM frame: max |y|, min z, max z (grown by 1e-6: reject only)
  T racket_obb[3];  // the same box, exact: TB_EV_RACKET_LOW
  T racket_obb_radius;  // distance of its farthest corner from the COM (pre-check of the same test)
  // derived constants of the fast-forward substep (ff_substep), formed on the host in double
  T ff_hack[3];    // dt / m_racket * (-50, -2, -2): the force law of swingracket_env.py:135-141 as velocity per metre
  T ff_gyro[3];    // dt * gyro * (I_k - I_j) / I_i: Euler's equations in the principal (= body) frame
  T ff_dtg;        // dt * gravity_z
  T ff_kl, ff_ka;  // dt * lin_damping, dt * ang_damping
  T ff_qx2;        // dt^2 / 4
  T ff_slab;       // |face-normal coordinate| of the ball beyond which the racket is out of reach (grown: reject only)
  T ff_low_z;      // racket COM height above which TB_EV_RACKET_LOW cannot fire
  T ff_ball_z;     // ball height above which floor, net and goal are all out of reach
  unsigned vmax2_hi;  // high word of max_coord_vel^2 in T's format (limit test on |omega|^2)
  // ff_fast's "this substep needs the full treatment" predicates (all grown: they may only park a lane for nothing)
  T ffp_racket_r2;             // (hull bounding radius + reach)^2
  T ffp_floor[3], ffp_net[3];  // half extents + reach
  T ffp_goal_z, ffp_goal_r2;   // goal half height + reach, (goal radius + reach)^2
  T ffp_a2;                    // |omega|^2 above which the short half-angle series or the velocity limit is in doubt
  T ffp_v2;                    // squared speed above which a coordinate could reach the velocity limit within a substep
  T ffp_face[3];               // the floor's top face without its margin rim: x, y half extents and the core's top
  T ffp_low, ffp_court[2];     // TB_EV_RACKET_LOW: floor top + contact threshold; court half extents + 1
  T ffp_box[3];                // racket outline bounding box + reach (max |y|, min z, max z), grown
  T ffp_rim;                   // reach beyond the racket outline, grown
  T ffl_inv_dt, ffl_erp_dt, ffl_m, ffl_jinv_t;  // landing hook: 1/dt, erp/dt, ball mass, 1/(1/m + r^2/I)
  Prism<T, kRacketEdges> racket;
  Prism<T, kGoalEdges> goal;
};

// ------------------------------------------------------------------------------------------------ state
template <typename T> struct St {
  T rp[3], rq[4], rv[3], rw[3], bp[3], bv[3], bw[3], aux[3], goal[2], d0, ret;
  int step, flags;
  uint32_t episode;
};

// ------------------------------------------------------------------------------------------------ RNG
// Philox4x32-10, counter = (global env id lo, hi, episode, stream word), key = seed.
__device__ __forceinline__ void philox4x32(uint64_t seed, uint64_t env_id, uint32_t episode, uint32_t w3, uint32_t out[4]) {
  uint32_t c0 = (uint32_t)env_id, c1 = (uint32_t)(env_id >> 32), c2 = episode, c3 = w3;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    c0 = h1 ^ c1 ^ k0;
    c1 = l1;
    c2 = h0 ^ c3 ^ k1;
    c3 = l0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
template <typename T> __device__ __forceinline__ T u01(uint32_t x) { return (T)(x >> 8) * (T)(1.0 / 16777216.0); }
constexpr uint32_t kStreamReset = 0u, kStreamAction = 1u;
__device__ __forceinline__ uint32_t stream_word(uint32_t stream, uint32_t step, uint32_t block) {
  return (stream << 28) | ((step & 0xFFFFFu) << 4) | (block & 0xFu);
}

// ------------------------------------------------------------------------------------------------ geometry
template <typename T> __device__ __forceinline__ void quat_to_mat(const T *q, T *R) {
  T x = q[0], y = q[1], z = q[2], w = q[3];
  R[0] = 1 - 2 * (y * y + z * z); R[1] = 2 * (x * y - z * w);     R[2] = 2 * (x * z + y * w);
  R[3] = 2 * (x * y + z * w);     R[4] = 1 - 2 * (x * x + z * z); R[5] = 2 * (y * z - x * w);
  R[6] = 2 * (x * z - y * w);     R[7] = 2 * (y * z + x * w);     R[8] = 1 - 2 * (x * x + y * y);
}
template <typename T> __device__ __forceinline__ void mat_vec(const T *R, const T *v, T *o) {
  o[0] = R[0] * v[0] + R[1] * v[1] + R[2] * v[2];
  o[1] = R[3] * v[0] + R[4] * v[1] + R[5] * v[2];
  o[2] = R[6] * v[0] + R[7] * v[1] + R[8] * v[2];
}
template <typename T> __device__ __forceinline__ void matT_vec(const T *R, const T *v, T *o) {
  o[0] = R[0] * v[0] + R[3] * v[1] + R[6] * v[2];
  o[1] = R[1] * v[0] + R[4] * v[1] + R[7] * v[2];
  o[2] = R[2] * v[0] + R[5] * v[1] + R[8] * v[2];
}

// Distance from (t; u,v) to a convex prism core: polygon in (u,v), extruded +-half_thick along t.
// n = unit normal core -> point as (nt,nu,nv); q = closest core point.  Inside the core the minimum
// translation axis (face vs outline) stands in for Bullet's EPA.
// Two passes over the outline: which side of every edge line the point is on (cheap; the signed distance to any
// edge line is a lower bound of the distance to the polygon, so beyond `far` the pass's maximum is returned as is,
// n and q unset), and - only for a point outside the outline but within `far` - the closest point on its edges.
template <typename T, int NE>
__device__ __noinline__ T prism_distance(const Prism<T, NE> &pr, T t, T u, T v, T far, T *n, T *q) {
  if (M<T>::abs(t) - pr.half_thick > 0 && prism_inside_fast(pr, u, v)) {  // over a face, inside the outline: the loops below
    T st = t < 0 ? (T)-1 : (T)1;                                          // would end in exactly this case
    n[0] = st; n[1] = 0; n[2] = 0;
    q[0] = st * pr.half_thick; q[1] = u; q[2] = v;
    return M<T>::abs(t) - pr.half_thick;
  }
  T max_side = -M<T>::inf();
  int max_edge = 0;
#pragma unroll kEdgeUnroll
  for (int i = 0; i < NE; ++i) {
    const Edge<T> &e = pr.e[i];
    T side = (u - e.ax) * e.nx + (v - e.ay) * e.ny;
    if (side > max_side) { max_side = side; max_edge = i; }
  }
  if (max_side > far) return max_side;
  T et = M<T>::abs(t) - pr.half_thick;
  T st = t < 0 ? (T)-1 : (T)1;
  if (max_side > 0) {
    T best_d2 = M<T>::inf(), bq0 = 0, bq1 = 0;
#pragma unroll 1
    for (int i = 0; i < NE; ++i) {
      const Edge<T> &e = pr.e[i];
      T ru = u - e.ax, rv = v - e.ay;
      T s = (ru * e.ex + rv * e.ey) * e.inv_len2;
      s = s < 0 ? (T)0 : (s > 1 ? (T)1 : s);
      T q0 = e.ax + s * e.ex, q1 = e.ay + s * e.ey;
      T d0 = u - q0, d1 = v - q1;
      T d2 = d0 * d0 + d1 * d1;
      if (d2 < best_d2) { best_d2 = d2; bq0 = q0; bq1 = q1; }
    }
    T du = u - bq0, dv = v - bq1;
    if (et > 0) {
      T dist = M<T>::sqrt(et * et + best_d2);
      n[0] = st * et / dist; n[1] = du / dist; n[2] = dv / dist;
      q[0] = st * pr.half_thick; q[1] = bq0; q[2] = bq1;
      return dist;
    }
    T dist = M<T>::sqrt(best_d2);
    n[0] = 0; n[1] = du / dist; n[2] = dv / dist;
    q[0] = t; q[1] = bq0; q[2] = bq1;
    return dist;
  }
  if (et > 0) {
    n[0] = st; n[1] = 0; n[2] = 0;
    q[0] = st * pr.half_thick; q[1] = u; q[2] = v;
    return et;
  }
  T pen_face = -et, pen_poly = -max_side;
  if (pen_face <= pen_poly) {
    n[0] = st; n[1] = 0; n[2] = 0;
    q[0] = st * pr.half_thick; q[1] = u; q[2] = v;
    return -pen_face;
  }
  const Edge<T> &e = pr.e[max_edge];
  n[0] = 0; n[1] = e.nx; n[2] = e.ny;
  q[0] = t; q[1] = u + pen_poly * e.nx; q[2] = v + pen_poly * e.ny;
  return -pen_poly;
}

// sphere centre vs box core (half extents shrunk by the embedded margin)
template <typename T> __device__ __forceinline__ T box_distance(const T *h, T margin, const T *p, T *n) {
  T d[3], q[3], d2 = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    T c = h[i] - margin;
    q[i] = p[i] < -c ? -c : (p[i] > c ? c : p[i]);
    d[i] = p[i] - q[i];
    d2 += d[i] * d[i];
  }
  if (d2 > 0) {
    T dist = M<T>::sqrt(d2);
#pragma unroll
    for (int i = 0; i < 3; ++i) n[i] = d[i] / dist;
    return dist;
  }
  int ax = 0;
  T pen = M<T>::inf();
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    T pi = (h[i] - margin) - M<T>::abs(p[i]);
    if (pi < pen) { pen = pi; ax = i; }
  }
  n[0] = n[1] = n[2] = 0;
  T sg = p[ax] < 0 ? (T)-1 : (T)1;
  if (ax == 0) n[0] = sg; else if (ax == 1) n[1] = sg; else n[2] = sg;
  return -pen;
}

// Bullet's btPlaneSpace1
template <typename T> __device__ __forceinline__ void plane_space(const T *n, T *p, T *q) {
  if (M<T>::abs(n[2]) > (T)0.70710678118654752440) {
    T a = n[1] * n[1] + n[2] * n[2], k = M<T>::rsqrt(a);
    p[0] = 0; p[1] = -n[2] * k; p[2] = n[1] * k;
    q[0] = a * k; q[1] = -n[0] * p[2]; q[2] = n[0] * p[1];
  } else {
    T a = n[0] * n[0] + n[1] * n[1], k = M<T>::rsqrt(a);
    p[0] = -n[1] * k; p[1] = n[0] * k; p[2] = 0;
    q[0] = -n[2] * p[1]; q[1] = n[2] * p[0]; q[2] = a * k;
  }
}

// true: (u, v) is farther than `rim` from the outline for certain (false says nothing).  Far from the part at or above out_v:
// outside an ellipse that contains everything within rim of the containing ellipse (out_inv_a, out_inv_b: the semi-axes
// grown by rim AND scaled up on the host until they do - growing alone falls short between the axes).  Far from the part
// below out_v, which lies between two edge lines: beyond one of those lines,
// below out_lo or above out_v, each by more than rim.
template <typename T, int NE> __device__ __forceinline__ bool prism_outside_fast(const Prism<T, NE> &pr, T u, T v, T rim) {
  T du = u * pr.out_inv_a, dv = (v - pr.in_c) * pr.out_inv_b;  // (rim == the rim the reciprocals were formed with)
  bool far_head = du * du + dv * dv > 1;
  bool far_quad = (pr.tz_lo > pr.tz_hi) | (v > pr.out_v + rim) | (v < pr.out_lo - rim) |
                  ((u - pr.t_ax[0]) * pr.t_nx[0] + (v - pr.t_ay[0]) * pr.t_ny[0] > rim) |
                  ((u - pr.t_ax[1]) * pr.t_nx[1] + (v - pr.t_ay[1]) * pr.t_ny[1] > rim);
  return far_head & far_quad;
}

// ------------------------------------------------------------------------------------------------ ray casting (tb_render)
// float32, coordinates relative to the eye: the ray is s -> s d with |d| = 1, and a shape counts where it is entered at s > 0.
// A convex body is the intersection of planes n.p <= h; with c = n.(eye) - h and den = n.d the ray crosses a plane at
// s = -c / den, entering where den < 0 and leaving where den > 0 (a parallel ray outside a plane misses the body): the
// Cyrus-Beck clip.  f0 is the entry plane.
__device__ __forceinline__ void clip_plane(float c, float den, int face, float &s0, float &s1, int &f0) {
  if (den < 0.f) {
    const float s = -c / den;
    if (s > s0) { s0 = s; f0 = face; }
  } else if (den > 0.f) {
    s1 = fminf(s1, -c / den);
  } else if (c > 0.f) {
    s1 = -M<float>::inf();
  }
}
__device__ __forceinline__ float clip_entry(float s0, float s1) { return s0 > 0.f && s0 < s1 ? s0 : M<float>::inf(); }
// Box |p_k| <= h_k about the origin; cb[2k] = eye_k - h_k, cb[2k + 1] = -eye_k - h_k.  face 2k: +axis k, 2k + 1: -axis k.
__device__ __forceinline__ float ray_box(const float *cb, const float *d, int &face) {
  float s0 = -M<float>::inf(), s1 = M<float>::inf();
  face = 0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    clip_plane(cb[2 * k], d[k], 2 * k, s0, s1, face);
    clip_plane(cb[2 * k + 1], -d[k], 2 * k + 1, s0, s1, face);
  }
  return clip_entry(s0, s1);
}
// Prism of the narrow phase in its own frame (t; u, v): |t| <= half_thick, inside every outline edge.  o_t = the eye's t,
// ce[i] = the eye's c of edge i (formed per frame), dl = the direction in that frame.  face 0: +t, 1: -t, 2 + i: edge i.
template <typename T, int NE>
__device__ __forceinline__ float ray_prism(const Prism<T, NE> &pr, const float *ce, float o_t, const float *dl, int &face) {
  const float ht = (float)pr.half_thick;
  float s0 = -M<float>::inf(), s1 = M<float>::inf();
  face = 0;
  clip_plane(o_t - ht, dl[0], 0, s0, s1, face);
  clip_plane(-o_t - ht, -dl[0], 1, s0, s1, face);
#pragma unroll 2
  for (int i = 0; i < NE; ++i) clip_plane(ce[i], (float)pr.e[i].nx * dl[1] + (float)pr.e[i].ny * dl[2], 2 + i, s0, s1, face);
  return clip_entry(s0, s1);
}
// Sphere of radius r about c (relative to the eye), through the perpendicular from c to the ray (no cancellation of |c|^2
// against (c.d)^2 for a small sphere far away).
__device__ __forceinline__ float ray_sphere(const float *c, float r, const float *d) {
  const float b = c[0] * d[0] + c[1] * d[1] + c[2] * d[2];
  const float q0 = c[0] - b * d[0], q1 = c[1] - b * d[1], q2 = c[2] - b * d[2];
  const float h = r * r - (q0 * q0 + q1 * q1 + q2 * q2);
  if (h < 0.f) return M<float>::inf();
  return clip_entry(b - sqrtf(h), M<float>::inf());
}
// true: the ray passes the bounding sphere (c, r) for certain, or reaches it only beyond `best` (reject only: grown)
__device__ __forceinline__ bool ray_skips(const float *c, float r, const float *d, float best) {
  const float b = c[0] * d[0] + c[1] * d[1] + c[2] * d[2];
  const float q0 = c[0] - b * d[0], q1 = c[1] - b * d[1], q2 = c[2] - b * d[2];
  const float rr = r * 1.001f + 1e-4f;
  return q0 * q0 + q1 * q1 + q2 * q2 > rr * rr || b + rr < 0.f || b - rr > best;
}

// ------------------------------------------------------------------------------------------------ contacts
constexpr int kMaxContacts = 8;  // the ball's (racket, floor, net, goal) + up to four racket-floor points
template <typename T> struct Contact {
  int dyn;   // the racket takes part (as the body the normal points away from)
  int ball;  // the ball is the second body; 0: racket against a static body - the static body takes the ball's place in every
             // row with zero inverse mass and zero velocity, and n points racket -> static body
  T n[3], d, ra[3], rest, mu;
};
template <typename T> struct Row {
  T u[3], rbxu[3], raxu[3], ia[3], jinv, denom, rhs, lam;  // denom = 1 / jinv
};
// The rare-path functions below are out of line and exchange data through these records ONLY: no address of a
// register-resident variable of the substep loop (state, control block) may escape into a call, or the compiler
// would have to keep that variable in local memory for the whole loop.
template <typename T> struct ContactSet {
  Contact<T> c[kMaxContacts];
};
template <typename T> struct NarrowIn {
  T rp[3], rq[4], bp[3], goal[2];
};
template <typename T> struct SolveIO {
  T rq[4], bv[3], bw[3], rv[3], rw[3];  // in: pose + velocities after force integration
  T dvb[3], dwb[3], dva[3], dwa[3];     // out: velocity changes
};
constexpr int kNeedRacket = 1, kNeedFloor = 2, kNeedNet = 4, kNeedGoal = 8, kNeedRacketFloor = 16;

// Projected Gauss-Seidel over the ball's contacts: per contact one normal row and a friction pair with an
// implicit cone clamp, early exit on the squared-residual threshold (A.6).  Rare path (about one physics step
// per episode), kept out of line so the substep loop stays small.  The rows are ALWAYS solved in double, also
// by the float32 kernel: the residual early exit makes the impulse sensitive to the sweep count, and a float
// solve that stops one sweep apart from the double oracle moves the ball's exit velocity by ~1e-2 m/s.
template <typename T>
__device__ __noinline__ void solve_contacts(const Scene<T> &sc, const ContactSet<T> *cs, int nc, SolveIO<T> *io) {
  typedef double S;
  const Contact<T> *ct = cs->c;
  const S rb = sc.ball_r, inv_mb = sc.ball_inv_m, inv_ib = sc.ball_inv_i, inv_mr = sc.racket_inv_m, dt = sc.dt;
  S R[9], bv[3], bw[3], rv[3], rw[3];
  {
    S q[4] = {(S)io->rq[0], (S)io->rq[1], (S)io->rq[2], (S)io->rq[3]};
    if (sizeof(T) == sizeof(S)) {
      quat_to_mat(q, R);
    } else {  // the float kernel forms R in float everywhere else; keep the same matrix here
      T qt[4] = {io->rq[0], io->rq[1], io->rq[2], io->rq[3]}, Rt[9];
      quat_to_mat(qt, Rt);
#pragma unroll
      for (int i = 0; i < 9; ++i) R[i] = Rt[i];
    }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) { bv[i] = io->bv[i]; bw[i] = io->bw[i]; rv[i] = io->rv[i]; rw[i] = io->rw[i]; }
  S dvb[3] = {0, 0, 0}, dwb[3] = {0, 0, 0}, dva[3] = {0, 0, 0}, dwa[3] = {0, 0, 0};
  Row<S> rows[kMaxContacts][3];
#pragma unroll 1
  for (int k = 0; k < nc; ++k) {
    const Contact<T> &c = ct[k];
    S dirs[3][3];
    dirs[0][0] = c.n[0]; dirs[0][1] = c.n[1]; dirs[0][2] = c.n[2];
    plane_space<S>(dirs[0], dirs[1], dirs[2]);
    S rbv[3] = {-rb * dirs[0][0], -rb * dirs[0][1], -rb * dirs[0][2]};
    S ra[3] = {(S)c.ra[0], (S)c.ra[1], (S)c.ra[2]};
#pragma unroll 1
    for (int r = 0; r < 3; ++r) {
      Row<S> &w = rows[k][r];
      w.u[0] = dirs[r][0]; w.u[1] = dirs[r][1]; w.u[2] = dirs[r][2];
      S denom = 0, rel = 0;
      if (c.ball) {
        cross3(rbv, w.u, w.rbxu);
        denom = inv_mb + dot3(w.rbxu, w.rbxu) * inv_ib;
        rel = dot3(w.u, bv) + dot3(w.rbxu, bw);
      } else {
        w.rbxu[0] = w.rbxu[1] = w.rbxu[2] = 0;
      }
      if (c.dyn) {
        cross3(ra, w.u, w.raxu);
        S l[3], li[3];
        matT_vec(R, w.raxu, l);
        li[0] = l[0] * (S)sc.racket_inv_i[0]; li[1] = l[1] * (S)sc.racket_inv_i[1]; li[2] = l[2] * (S)sc.racket_inv_i[2];
        mat_vec(R, li, w.ia);
        denom += inv_mr + dot3(w.raxu, w.ia);
        rel -= dot3(w.u, rv) + dot3(w.raxu, rw);
      } else {
        w.raxu[0] = w.raxu[1] = w.raxu[2] = 0;
        w.ia[0] = w.ia[1] = w.ia[2] = 0;
      }
      w.jinv = 1 / denom;
      w.denom = denom;
      w.lam = 0;
      if (r == 0) {
        S e = fabs(rel) < (S)sc.rest_vel_threshold ? (S)0 : -(S)c.rest * rel;
        if (e < 0) e = 0;
        S pen = (S)c.d + (S)sc.slop, vel_err = e - rel, pos_err = 0;
        if (pen > 0) vel_err -= pen / dt;
        else pos_err = -pen * (S)sc.erp / dt;
        w.rhs = (pos_err + vel_err) * w.jinv;
      } else {
        w.rhs = -rel * w.jinv;
      }
    }
  }
#pragma unroll 1
  for (int it = 0; it < sc.iters; ++it) {
    S resid = 0;
#pragma unroll 1
    for (int k = 0; k < nc; ++k) {
      Row<S> &w = rows[k][0];
      S jd = dot3(w.u, dvb) + dot3(w.rbxu, dwb) - dot3(w.u, dva) - dot3(w.raxu, dwa);
      S dl = w.rhs - jd * w.jinv;
      S sum = w.lam + dl;
      if (sum < 0) { dl = -w.lam; sum = 0; }
      w.lam = sum;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        if (ct[k].ball) { dvb[i] += w.u[i] * dl * inv_mb; dwb[i] += w.rbxu[i] * dl * inv_ib; }
        if (ct[k].dyn) { dva[i] -= w.u[i] * dl * inv_mr; dwa[i] -= w.ia[i] * dl; }
      }
      S rr = dl * w.denom;  // (= dl / jinv to an ulp; feeds the early-exit test only: no division on the servers' critical path)
      if (rr * rr > resid) resid = rr * rr;
    }
#pragma unroll 1
    for (int k = 0; k < nc; ++k) {
      S lam_n = rows[k][0].lam;
      if (!(lam_n > 0)) continue;
      S lim = (S)ct[k].mu * lam_n;
      S sum[2];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        Row<S> &w = rows[k][1 + r];
        S jd = dot3(w.u, dvb) + dot3(w.rbxu, dwb) - dot3(w.u, dva) - dot3(w.raxu, dwa);
        sum[r] = w.lam + (w.rhs - jd * w.jinv);
      }
      S m2 = sum[0] * sum[0] + sum[1] * sum[1];
      if (m2 > lim * lim) {
        S sf = lim / ::sqrt(m2);
        sum[0] *= sf; sum[1] *= sf;
      }
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        Row<S> &w = rows[k][1 + r];
        S d = sum[r] - w.lam;
        w.lam = sum[r];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          if (ct[k].ball) { dvb[i] += w.u[i] * d * inv_mb; dwb[i] += w.rbxu[i] * d * inv_ib; }
          if (ct[k].dyn) { dva[i] -= w.u[i] * d * inv_mr; dwa[i] -= w.ia[i] * d; }
        }
        S rr = d * w.denom;
        if (rr * rr > resid) resid = rr * rr;
      }
    }
    if (resid <= (S)sc.solver_residual) break;
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) { io->dvb[i] = (T)dvb[i]; io->dwb[i] = (T)dwb[i]; io->dva[i] = (T)dva[i]; io->dwa[i] = (T)dwa[i]; }
}

// Narrow phase of every pair whose broad-phase test passed, one out-of-line call.  Appends to cs->c[] in the
// fixed order racket, floor, net, goal; returns event bits | (number of contacts << 8).
template <typename T, bool WITH_GOAL>
__device__ __noinline__ int narrow_phase(const Scene<T> &sc, int need, const NarrowIn<T> *in, ContactSet<T> *cs) {
  int nc = 0, bits = 0;
  const T thr = sc.contact_threshold;
  T R[9];
  if (need & (kNeedRacket | kNeedRacketFloor)) quat_to_mat(in->rq, R);
  if (need & kNeedRacket) {
    T rel[3] = {in->bp[0] - in->rp[0], in->bp[1] - in->rp[1], in->bp[2] - in->rp[2]}, pl[3];
    matT_vec(R, rel, pl);
    // second-level reject in the racket frame (plate slab and outline bounding box, both grown by the reach):
    // conservative, so the oracle, which runs the narrow phase whenever the bounding sphere is entered, agrees
    T reach = sc.ball_r + sc.hull_margin + thr;
    if (!(M<T>::abs(pl[0]) - sc.racket.half_thick > reach || M<T>::abs(pl[1]) - sc.racket_box[0] > reach ||
          pl[2] - sc.racket_box[2] > reach || sc.racket_box[1] - pl[2] > reach)) {
      T nl[3], ql[3];
      T dc = prism_distance<T, kRacketEdges>(sc.racket, pl[0], pl[1], pl[2], reach * (T)1.0001, nl, ql);
      T d = dc - (sc.ball_r + sc.hull_margin);
      if (d <= thr) {
        Contact<T> &k = cs->c[nc++];
        k.dyn = 1; k.ball = 1;
        mat_vec(R, nl, k.n);
        T qs[3] = {ql[0] + sc.hull_margin * nl[0], ql[1] + sc.hull_margin * nl[1], ql[2] + sc.hull_margin * nl[2]};
        mat_vec(R, qs, k.ra);
        k.d = d; k.rest = sc.rest_racket; k.mu = sc.mu_racket;
        bits |= TB_EV_RACKET_BALL;
      }
    }
  }
#pragma unroll 1
  for (int b = 0; b < 2; ++b) {
    if (!(need & (b ? kNeedNet : kNeedFloor))) continue;
    const T *h = b ? sc.net_h : sc.floor_h;
    T n[3];
    T dc = box_distance(h, sc.box_margin, in->bp, n);
    T d = dc - (sc.ball_r + sc.box_margin);
    if (d <= thr) {
      Contact<T> &k = cs->c[nc++];
      k.dyn = 0; k.ball = 1;
      k.n[0] = n[0]; k.n[1] = n[1]; k.n[2] = n[2];
      k.ra[0] = k.ra[1] = k.ra[2] = 0;
      k.d = d; k.rest = sc.rest_court; k.mu = sc.mu_court;
      bits |= TB_EV_COURT_BALL | (b ? TB_EV_NET_BALL : 0);
    }
  }
  if (WITH_GOAL && (need & kNeedGoal)) {
    T nl[3], ql[3];
    T dc = prism_distance<T, kGoalEdges>(sc.goal, in->bp[2], in->bp[0] - in->goal[0], in->bp[1] - in->goal[1],
                                         (sc.ball_r + sc.hull_margin + thr) * (T)1.0001, nl, ql);
    T d = dc - (sc.ball_r + sc.hull_margin);
    if (d <= thr) {
      Contact<T> &k = cs->c[nc++];
      k.dyn = 0; k.ball = 1;
      k.n[0] = nl[1]; k.n[1] = nl[2]; k.n[2] = nl[0];
      k.ra[0] = k.ra[1] = k.ra[2] = 0;
      k.d = d; k.rest = sc.rest_goal; k.mu = sc.mu_goal;
      bits |= TB_EV_GOAL_BALL;
    }
  }
  if (need & kNeedRacketFloor) {
    // Racket vs the floor box's top face (court.urdf:19-24): the corners of the hull's oriented bounding box (outline box x
    // plate thickness, inflated by the hull margin) that are within the contact threshold of the face and over it, the four
    // deepest if there are more (a manifold holds four points), in corner order.  Normal: racket -> floor = -z.
    T dz[8], cr[8][3];
    int m = 0;
#pragma unroll 1
    for (int q = 0; q < 8; ++q) {
      const T l[3] = {(q & 1) ? sc.racket.half_thick : -sc.racket.half_thick, (q & 2) ? sc.racket_obb[0] : -sc.racket_obb[0],
                      (q & 4) ? sc.racket_obb[2] : sc.racket_obb[1]};
      T w[3];
      mat_vec(R, l, w);
      const T px = in->rp[0] + w[0], py = in->rp[1] + w[1], pz = in->rp[2] + w[2];
      const T d = pz - sc.hull_margin - sc.floor_h[2];
      if (d <= thr && M<T>::abs(px) <= sc.floor_h[0] && M<T>::abs(py) <= sc.floor_h[1]) {
        dz[m] = d; cr[m][0] = w[0]; cr[m][1] = w[1]; cr[m][2] = w[2] - sc.hull_margin; ++m;
      }
    }
    while (m > 4) {  // drop the shallowest (first of equals)
      int worst = 0;
      for (int q = 1; q < m; ++q) if (dz[q] > dz[worst]) worst = q;
      for (int q = worst; q + 1 < m; ++q) { dz[q] = dz[q + 1]; cr[q][0] = cr[q + 1][0]; cr[q][1] = cr[q + 1][1]; cr[q][2] = cr[q + 1][2]; }
      --m;
    }
    for (int q = 0; q < m; ++q) {
      Contact<T> &k = cs->c[nc++];
      k.dyn = 1; k.ball = 0;
      k.n[0] = 0; k.n[1] = 0; k.n[2] = -1;
      k.ra[0] = cr[q][0]; k.ra[1] = cr[q][1]; k.ra[2] = cr[q][2];
      k.d = dz[q]; k.rest = sc.rest_racket_court; k.mu = sc.mu_racket_court;
    }
  }
  return bits | (nc << 8);
}

// TB_EV_RACKET_LOW: the lowest corner of the hull's oriented bounding box (outline box x plate thickness, margin included) is
// at or below the floor's contact threshold while the COM is over the court (same expression wherever it is evaluated)
template <typename T> __device__ __forceinline__ bool racket_low(const Scene<T> &sc, const T *rp, const T *rq) {
  const T x = rq[0], y = rq[1], z = rq[2], w = rq[3];
  T r6 = 2 * (x * z - y * w), r7 = 2 * (y * z + x * w), r8 = 1 - 2 * (x * x + y * y);
  T zlo = r8 * sc.racket_obb[1], zhi = r8 * sc.racket_obb[2];
  T low = rp[2] - M<T>::abs(r6) * sc.racket.half_thick - M<T>::abs(r7) * sc.racket_obb[0] + (zlo < zhi ? zlo : zhi) - sc.hull_margin;
  return (low <= sc.ffp_low) & (M<T>::abs(rp[0]) <= sc.ffp_court[0]) & (M<T>::abs(rp[1]) <= sc.ffp_court[1]);
}

// Half-angle factors of one substep's rotation, as even functions of |omega|: with x = |omega| dt / 2,
//   sinc(x) = sin(x)/x and cos(x) are power series in x^2 = a2 dt^2 / 4, so neither |omega|, its reciprocal nor a
// small-angle special case (Bullet switches to a Taylor form below 0.001 rad/s) is ever needed.  |x| <= 0.37
// because every velocity coordinate is clamped to +-100; the short series covers |omega| < 24 rad/s (x^2 < 2.5e-3)
// to the last bit, the long one the rest.  The oracle calls libm sin/cos; the difference is below 1 ulp.
__device__ __forceinline__ void sinc_cos_x2(float x2, float *sinc, float *c) {
  *sinc = 1.0f + x2 * (-1.0f / 6 + x2 * (1.0f / 120 + x2 * (-1.0f / 5040 + x2 * (1.0f / 362880))));
  *c = 1.0f + x2 * (-0.5f + x2 * (1.0f / 24 + x2 * (-1.0f / 720 + x2 * (1.0f / 40320 + x2 * (-1.0f / 3628800)))));
}
__device__ __forceinline__ void sinc_cos_x2(double x2, double *sinc, double *c) {
  if (x2 < 2.5e-3) {
    *sinc = 1.0 + x2 * (-1.0 / 6 + x2 * (1.0 / 120 + x2 * (-1.0 / 5040 + x2 * (1.0 / 362880 + x2 * (-1.0 / 39916800)))));
    *c = 1.0 + x2 * (-0.5 + x2 * (1.0 / 24 + x2 * (-1.0 / 720 + x2 * (1.0 / 40320 + x2 * (-1.0 / 3628800 +
         x2 * (1.0 / 479001600.0))))));
  } else {
    *sinc = 1.0 + x2 * (-1.0 / 6 + x2 * (1.0 / 120 + x2 * (-1.0 / 5040 + x2 * (1.0 / 362880 + x2 * (-1.0 / 39916800 +
            x2 * (1.0 / 6227020800.0 + x2 * (-1.0 / 1307674368000.0 + x2 * (1.0 / 355687428096000.0))))))));
    *c = 1.0 + x2 * (-0.5 + x2 * (1.0 / 24 + x2 * (-1.0 / 720 + x2 * (1.0 / 40320 + x2 * (-1.0 / 3628800 +
         x2 * (1.0 / 479001600.0 + x2 * (-1.0 / 87178291200.0 + x2 * (1.0 / 20922789888000.0 +
         x2 * (-1.0 / 6402373705728000.0)))))))));
  }
}
// the short branch alone (x^2 < 2.5e-3, i.e. |omega| < 24 rad/s)
__device__ __forceinline__ void sinc_cos_short(float x2, float *sinc, float *c) { sinc_cos_x2(x2, sinc, c); }
__device__ __forceinline__ void sinc_cos_short(double x2, double *sinc, double *c) {
  // first dropped terms at x2 = 2.5e-3: 2.4e-21 and 2.0e-25
  *sinc = 1.0 + x2 * (-1.0 / 6 + x2 * (1.0 / 120 + x2 * (-1.0 / 5040 + x2 * (1.0 / 362880))));
  *c = 1.0 + x2 * (-0.5 + x2 * (1.0 / 24 + x2 * (-1.0 / 720 + x2 * (1.0 / 40320 + x2 * (-1.0 / 3628800)))));
}
__device__ __forceinline__ float fast_rsqrt(float x) {
  float y = rsqrtf(x);
  return y * (1.5f - 0.5f * x * y * y);  // one Newton step on the 2-ulp hardware estimate
}
__device__ __forceinline__ double fast_rsqrt(double x) { return ::rsqrt(x); }

// q <- exp(omega dt) q by the exponential map, then normalise (btMultiBody::stepPositionsMultiDof [R]).
template <typename T> __device__ __forceinline__ void integrate_quat(const Scene<T> &sc, St<T> &s) {
  const T dt = sc.dt;
  if (s.rw[0] != 0 || s.rw[1] != 0 || s.rw[2] != 0) {
    T a2 = dot3(s.rw, s.rw), sinc, cw;
    sinc_cos_x2((T)0.25 * dt * dt * a2, &sinc, &cw);
    T k = (T)0.5 * dt * sinc;  // sin(|omega| dt / 2) / |omega|
    T ax = s.rw[0] * k, ay = s.rw[1] * k, az = s.rw[2] * k;
    const T *q = s.rq;
    T x = cw * q[0] + ax * q[3] + ay * q[2] - az * q[1];
    T y = cw * q[1] - ax * q[2] + ay * q[3] + az * q[0];
    T z = cw * q[2] + ax * q[1] - ay * q[0] + az * q[3];
    T w = cw * q[3] - ax * q[0] - ay * q[1] - az * q[2];
    // the product of two unit quaternions is unit up to rounding: 1/sqrt(1 + e) = 1 - e/2 to ~e^2, so one
    // multiply-add renormalises; a quaternion that is off by more (injected through tb_set_state) takes the exact path
    T n2 = x * x + y * y + z * z + w * w;
    T inv = (T)1.5 - (T)0.5 * n2;
    if (TB_UNLIKELY(M<T>::abs(n2 - 1) > (T)1e-4)) inv = fast_rsqrt(n2);
    s.rq[0] = x * inv; s.rq[1] = y * inv; s.rq[2] = z * inv; s.rq[3] = w * inv;
  }
}

// One stepSimulation(): detect at the start-of-step poses, integrate velocities with Bullet's multibody
// damping, solve contacts, integrate poses.  Returns the TB_EV_* contact bits getContactPoints would report.
template <typename T, bool WITH_GOAL>
__device__ __forceinline__ int physics_step(const Scene<T> &sc, St<T> &s, const T *f_racket, const T *t_racket,
                                            const T *f_ball) {
  const T dt = sc.dt, thr = sc.contact_threshold, rb = sc.ball_r;
  ContactSet<T> cs;  // lives in local memory; touched on the rare path only
  int nc = 0, bits = 0;

  // ---- (1) detection: conservative broad-phase rejects in line and branch-free, every narrow phase in one rare call
  T R[9];
  quat_to_mat(s.rq, R);
  {
    int need = 0;
    {
      // racket: inside the hull's bounding sphere AND, in the racket frame, inside the plate's slab and the outline's
      // bounding box (each grown by ball radius + margin + threshold).  A ball that merely lingers near a racket
      // it missed - the common case, both are in free fall side by side - never leaves the straight line.
      T rel[3] = {s.bp[0] - s.rp[0], s.bp[1] - s.rp[1], s.bp[2] - s.rp[2]}, pl[3];
      matT_vec(R, rel, pl);
      const T reach = rb + sc.hull_margin + thr, rs = sc.racket.bound_radius + reach;
      bool near_racket = dot3(rel, rel) <= rs * rs && !(M<T>::abs(pl[0]) - sc.racket.half_thick > reach) &&
                         !(M<T>::abs(pl[1]) - sc.racket_box[0] > reach) && !(pl[2] - sc.racket_box[2] > reach) &&
                         !(sc.racket_box[1] - pl[2] > reach);
      need |= near_racket ? kNeedRacket : 0;
    }
    const T reach_b = rb + sc.box_margin + thr;
    need |= !(M<T>::abs(s.bp[2]) - sc.floor_h[2] > reach_b || M<T>::abs(s.bp[0]) - sc.floor_h[0] > reach_b ||
              M<T>::abs(s.bp[1]) - sc.floor_h[1] > reach_b) ? kNeedFloor : 0;
    need |= !(M<T>::abs(s.bp[0]) - sc.net_h[0] > reach_b || M<T>::abs(s.bp[2]) - sc.net_h[2] > reach_b ||
              M<T>::abs(s.bp[1]) - sc.net_h[1] > reach_b) ? kNeedNet : 0;
    if (WITH_GOAL) {
      const T reach_g = rb + sc.hull_margin + thr, rxy = sc.goal_r + reach_g;
      T gx = s.bp[0] - s.goal[0], gy = s.bp[1] - s.goal[1];
      need |= (M<T>::abs(s.bp[2]) - sc.goal_hz <= reach_g && gx * gx + gy * gy <= rxy * rxy) ? kNeedGoal : 0;
    }
    // Racket vs floor is not modelled (the racket falls through the court once the episode's control phase is
    // over); TB_EV_RACKET_LOW marks the steps from which its pose is outside the parity horizon: the lowest
    // corner of the hull's oriented bounding box (outline box x plate thickness, margin included) is at or below
    // the floor's contact threshold while the COM is over the court.
    {
      T zlo = R[8] * sc.racket_obb[1], zhi = R[8] * sc.racket_obb[2];
      T low = s.rp[2] - M<T>::abs(R[6]) * sc.racket.half_thick - M<T>::abs(R[7]) * sc.racket_obb[0] + (zlo < zhi ? zlo : zhi) -
              sc.hull_margin;
      bits |= (low <= sc.floor_h[2] + thr && M<T>::abs(s.rp[0]) <= sc.floor_h[0] + 1 && M<T>::abs(s.rp[1]) <= sc.floor_h[1] + 1)
                  ? TB_EV_RACKET_LOW : 0;
    }
    if (sc.racket_court && (bits & TB_EV_RACKET_LOW)) need |= kNeedRacketFloor;
    if (TB_UNLIKELY(need)) {
      NarrowIn<T> in;
#pragma unroll
      for (int i = 0; i < 3; ++i) { in.rp[i] = s.rp[i]; in.bp[i] = s.bp[i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i) in.rq[i] = s.rq[i];
      in.goal[0] = s.goal[0]; in.goal[1] = s.goal[1];
      int r = narrow_phase<T, WITH_GOAL>(sc, need, &in, &cs);
      bits |= r & 0xff;
      nc = r >> 8;
    }
  }

  // ---- (2) velocities: v += dt (F/m + g - v (k + k|v|)); omega likewise in the body frame with the gyro term
  const T vmax = sc.max_coord_vel;
  {
    T kv = sc.lin_damping * (1 + norm3_fast(s.bv));
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      T g = i == 2 ? sc.gravity_z : (T)0;
      s.bv[i] = s.bv[i] + dt * (f_ball[i] * sc.ball_inv_m + g - s.bv[i] * kv);
    }
    if (s.bw[0] != 0 || s.bw[1] != 0 || s.bw[2] != 0) {  // the ball spins only after a frictional contact
      T kw = sc.ang_damping * (1 + norm3_fast(s.bw));
#pragma unroll
      for (int i = 0; i < 3; ++i) s.bw[i] = s.bw[i] + dt * (-s.bw[i] * kw);
    }
  }
  const bool rotating = s.rw[0] != 0 || s.rw[1] != 0 || s.rw[2] != 0 || t_racket[0] != 0 || t_racket[1] != 0 ||
                        t_racket[2] != 0;
  {
    T kv = sc.lin_damping * (1 + norm3_fast(s.rv));
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      T g = i == 2 ? sc.gravity_z : (T)0;
      s.rv[i] = s.rv[i] + dt * (f_racket[i] * sc.racket_inv_m + g - s.rv[i] * kv);
    }
    if (rotating) {  // the hit env's racket never rotates: no torque is ever applied to it
      T wl[3], tl[3], iw[3], gy[3], al[3], aw[3];
      matT_vec(R, s.rw, wl);
      matT_vec(R, t_racket, tl);
#pragma unroll
      for (int i = 0; i < 3; ++i) iw[i] = sc.racket_i[i] * wl[i];
      cross3(wl, iw, gy);
      T kw = sc.ang_damping * (1 + norm3_fast(wl));
#pragma unroll
      for (int i = 0; i < 3; ++i) al[i] = (tl[i] - sc.gyro * gy[i]) * sc.racket_inv_i[i] - wl[i] * kw;
      mat_vec(R, al, aw);
#pragma unroll
      for (int i = 0; i < 3; ++i) s.rw[i] = s.rw[i] + dt * aw[i];
    }
  }
  clamp_velocities(s.bv, s.bw, s.rv, s.rw, vmax, sc.vmax_hi);

  // ---- (3) contact solve
  if (TB_UNLIKELY(nc > 0)) {
    SolveIO<T> io;
#pragma unroll
    for (int i = 0; i < 3; ++i) { io.bv[i] = s.bv[i]; io.bw[i] = s.bw[i]; io.rv[i] = s.rv[i]; io.rw[i] = s.rw[i]; }
#pragma unroll
    for (int i = 0; i < 4; ++i) io.rq[i] = s.rq[i];
    solve_contacts(sc, &cs, nc, &io);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      s.bv[i] += io.dvb[i]; s.bw[i] += io.dwb[i]; s.rv[i] += io.dva[i]; s.rw[i] += io.dwa[i];
    }
    clamp_velocities(s.bv, s.bw, s.rv, s.rw, vmax, sc.vmax_hi);
  }

  // ---- (4) poses: x += dt v ; q <- exp(omega dt) q
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    s.bp[i] += dt * s.bv[i];
    s.rp[i] += dt * s.rv[i];
  }
  integrate_quat(sc, s);
  return bits;
}

// ------------------------------------------------------------------------------------------------ episodes
template <typename T, int KIND> __device__ __forceinline__ void place(const Scene<T> &sc, St<T> &s, const T *in) {
#pragma unroll
  for (int i = 0; i < 3; ++i) { s.rv[i] = 0; s.rw[i] = 0; s.bv[i] = 0; s.bw[i] = 0; }
  if (KIND == TB_ENV_SWING) {
    // swingracket_env.py:161-175
    s.rq[0] = sc.swing_q[0]; s.rq[1] = sc.swing_q[1]; s.rq[2] = sc.swing_q[2]; s.rq[3] = sc.swing_q[3];
    s.rp[0] = in[0] + sc.swing_off[0]; s.rp[1] = in[1] + sc.swing_off[1]; s.rp[2] = in[2] + sc.swing_off[2];
    s.bp[0] = in[0] - (T)0.1; s.bp[1] = in[1]; s.bp[2] = in[2] + (T)0.8;
    s.aux[0] = in[0]; s.aux[1] = in[1]; s.aux[2] = in[2];
    s.goal[0] = in[3]; s.goal[1] = in[4];
    T dx = s.bp[0] - in[3], dy = s.bp[1] - in[4];
    s.d0 = M<T>::sqrt(dx * dx + dy * dy);
  } else {
    // tennisbot_env.py:227-246
    s.rq[0] = 0; s.rq[1] = 0; s.rq[2] = 0; s.rq[3] = 1;
    s.rp[0] = in[0]; s.rp[1] = in[1]; s.rp[2] = in[2] + sc.com_z;
    s.aux[0] = in[3]; s.aux[1] = in[4]; s.aux[2] = (T)(25.0 * 0.8);
    s.bp[0] = in[5]; s.bp[1] = in[6]; s.bp[2] = in[7];
    s.goal[0] = 0; s.goal[1] = 0; s.d0 = 0;
  }
}
template <typename T, int KIND>
__device__ __forceinline__ void draw_init(uint64_t seed, uint64_t gid, uint32_t episode, T *in) {
  uint32_t r[4];
  philox4x32(seed, gid, episode, stream_word(kStreamReset, 0, 0), r);
  if (KIND == TB_ENV_SWING) {
    in[0] = (T)5.5 + (T)5.5 * u01<T>(r[0]);
    in[1] = (T)-4.0 + (T)8.0 * u01<T>(r[1]);
    in[2] = (T)0.6;
    in[3] = (T)-3.0 - (T)9.0 * u01<T>(r[2]);
    in[4] = (T)-5.0 + (T)10.0 * u01<T>(r[3]);
    in[5] = in[6] = in[7] = 0;
  } else {
    uint32_t r2[4];
    philox4x32(seed, gid, episode, stream_word(kStreamReset, 0, 1), r2);
    in[0] = (T)7.5 + (T)5.0 * u01<T>(r[0]);
    in[1] = (T)-5.0 + (T)10.0 * u01<T>(r[1]);
    in[2] = (T)0.2 + (T)0.01 * u01<T>(r[2]);
    in[3] = (T)25.0 + (T)12.5 * u01<T>(r[3]);
    in[4] = (T)-10.0 + (T)20.0 * u01<T>(r2[0]);
    in[5] = (T)-12.0 + (T)6.0 * u01<T>(r2[1]);
    in[6] = (T)-1.0 + (T)2.0 * u01<T>(r2[2]);
    in[7] = (T)1.0 + (T)0.5 * u01<T>(r2[3]);
  }
}
// Bits of the flags word that tell step_kernel which packs it need not load (the packs in HBM are always complete):
//   kStDerived  the episode constants equal place(draw_init(seed, global env id, episode)): goal / d0 / spawn (swing) can be
//               re-derived from the counter-based RNG instead of loaded; set by every RNG-placed episode start, not by
//               explicit placements (tb_reset_from) or injected states (tb_set_state).  Tennisbot-v0: pack 6 holds only the
//               constant z shoot force, so there the bit is set by every episode start
//   kStSpin     the ball's spin has a y or z component (it has none until a frictional contact): pack 5 must be loaded
//   kStPristine (SwingRacket) the ball has only fallen freely from rest since the episode began: its velocity is (0, 0, vz[k])
//               after k substeps whatever the placement (Scene::ball_vz, tabulated by the kernels' own arithmetic) and it does
//               not spin, so pack 4 (ball velocity | spin x) is neither loaded nor written while the bit is set; HBM holds a
//               stale pack 4 meanwhile.  The bit lives through step_kernel's straight-line control substep only: every other
//               path materialises the pack on load and clears the bit
constexpr int kStDerived = 1 << 24, kStSpin = 1 << 25, kStPristine = 1 << 26;
template <typename T, int KIND>
__device__ __forceinline__ void start_episode(const Scene<T> &sc, St<T> &s, const T *in, uint32_t episode, bool from_rng) {
  place<T, KIND>(sc, s, in);
  s.ret = 0; s.step = 0; s.episode = episode;
  s.flags = ((from_rng || KIND == TB_ENV_HIT) ? kStDerived : 0) | (KIND == TB_ENV_SWING ? kStPristine : 0);
}
template <typename T, int KIND> __device__ __forceinline__ void pack_obs(const St<T> &s, float *o) {
  if (KIND == TB_ENV_SWING) {
    o[0] = (float)s.rp[0]; o[1] = (float)s.rp[1]; o[2] = (float)s.bp[0]; o[3] = (float)s.bp[1];
    o[4] = (float)s.goal[0]; o[5] = (float)s.goal[1];
  } else {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      o[i] = (float)s.rp[i]; o[3 + i] = (float)s.rv[i]; o[6 + i] = (float)s.bp[i]; o[9 + i] = (float)s.bv[i];
    }
  }
}

template <typename T> __device__ __forceinline__ T moved_dist(T bx, T by, T gx, T gy, T d0) {
  T dx = bx - gx, dy = by - gy;
  return (d0 - M<T>::sqrt(dx * dx + dy * dy)) / d0 * (T)20;
}
template <typename T> __device__ __forceinline__ T moved_dist_to_goal(const St<T> &s) {
  return moved_dist(s.bp[0], s.bp[1], s.goal[0], s.goal[1], s.d0);
}
template <typename T> __device__ __forceinline__ T dist_to_reward(T d) {
  return d < (T)0.5 ? (T)20 : d < 1 ? (T)15 : d < 2 ? (T)10 : d < 3 ? (T)5 : d < 4 ? (T)1 : (T)0;
}

// TB_CONTROL_PID: three simple_pid.PID controllers on the racket COM position, evaluated with dt = 1/240
// (racket.py:47-64,103-122).  e = sp - x; I = clamp(I + ki e dt); D = -kd (x - x_last)/dt, 0 on the first call;
// out = clamp(kp e + I + D); force = (0, 0, bias) + out.  pid = {I xyz, x_last xyz, has_last, -}.
template <typename T> __device__ __forceinline__ void pid_force(const Scene<T> &sc, T *pid, const T *pos, const T *sp, T *F) {
  const T lim = sc.pid_lim, dt = sc.dt;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    T e = sp[i] - pos[i];
    T integ = clampv(pid[i] + sc.pid_ki * e * dt, -lim, lim);
    T d_in = pid[6] != 0 ? pos[i] - pid[3 + i] : (T)0;
    F[i] = clampv(sc.pid_kp * e + integ - sc.pid_kd * d_in / dt, -lim, lim);
    pid[i] = integ;
    pid[3 + i] = pos[i];
  }
  pid[6] = 1;
  F[2] += sc.pid_bias_z;
}

// Per-lane progress of one agent-visible step().  SwingRacket's 26th step re-enters the substep many times:
//   phase 0: the substep driven by the action (swingracket_env.py:76-83)
//   phase 1: first fast-forward substep, no external force (the step above cleared them) (:105-107)
//   phase 2: later fast-forward substeps, driven by the "hack" force queued after the previous one (:135-141)
template <typename T> __device__ __forceinline__ int hit_physics(const Scene<T> &sc, St<T> &s, const T *F, const T *Fb);  // below

struct StepCtl {
  int phase, events, hit;
  float reward;
  bool done;
  int last;  // contact bits of the most recent substep alone (ff_substep)
};

// One physics substep of the env step in flight plus the env logic that follows it.  Returns true when the
// env step is complete (reward / done / events are final).
// pid: this env's controller memory when the context runs TB_CONTROL_PID, else nullptr.
// bits_out: receives the contact bits physics_step / hit_physics returned for this substep alone (trace_kernel), or nullptr.
template <typename T, int KIND>
__device__ __forceinline__ bool env_substep(const Scene<T> &sc, St<T> &s, const float *a, StepCtl &c, T *pid = nullptr,
                                            int *bits_out = nullptr) {
  T zero[3] = {0, 0, 0};
  if (KIND == TB_ENV_SWING) {
    T F[3], Tq[3] = {0, 0, 0};
    if (c.phase == 0) {
      F[0] = (T)a[0] * 400; F[1] = (T)a[1] * 400; F[2] = (T)a[2] * 400 + (T)(4 * 9.81);
      Tq[0] = (T)a[3] * 5; Tq[1] = (T)a[4] * 5; Tq[2] = (T)a[5] * 5;
      if (pid) {
        T sp[3] = {(T)a[0], (T)a[1], (T)a[2]};
        pid_force(sc, pid, s.rp, sp, F);
        Tq[0] = Tq[1] = Tq[2] = 0;
      }
    } else if (c.phase == 1) {
      F[0] = F[1] = F[2] = 0;
    } else {  // the force the reference queued from the post-step pose of the previous substep = this one's pre-step pose
      F[0] = -50 * (s.rp[0] - s.aux[0]);
      F[1] = -2 * (s.rp[1] - s.aux[1]);
      F[2] = -2 * (s.rp[2] - s.aux[2] - 4);
    }
    int bits = physics_step<T, true>(sc, s, F, Tq, zero);
    if (bits_out) *bits_out = bits;
    int k = ++s.step;
    c.events |= bits;
    if (c.phase == 0) {
      if (k < 25 && (bits & TB_EV_RACKET_BALL)) { c.reward += 2.0f; c.hit = 1; }
      c.phase = 1;
      return !(k > 25) || c.done;
    }
    c.phase = 2;
    T reward = 0;
    if (bits & TB_EV_COURT_BALL) { c.done = true; reward += moved_dist_to_goal(s); }
    if (bits & TB_EV_GOAL_BALL) { reward += moved_dist_to_goal(s); reward += 50; c.done = true; }
    if (k > 800) { c.done = true; c.events |= TB_EV_TIMEOUT; }
    if (c.done) c.reward = (float)reward;
    return c.done;
  } else {
    T F[3] = {(T)a[0] * 10, (T)a[1] * 10, (T)(4 * 9.81)};
    if (pid) {
      T sp[3] = {(T)a[0], (T)a[1], sc.pid_hit_z};
      pid_force(sc, pid, s.rp, sp, F);
    }
    T Fb[3] = {0, 0, 0};
    if (s.step >= sc.shoot_start && s.step < sc.shoot_start + sc.shoot_frames) { Fb[0] = s.aux[0]; Fb[1] = s.aux[1]; Fb[2] = s.aux[2]; }
    int bits = hit_physics<T>(sc, s, F, Fb);
    if (bits_out) *bits_out = bits;
    int k = ++s.step;
    c.events = bits;
    if (k < sc.shoot_frames) { c.done = false; return true; }  // returns False regardless of self.done (tennisbot_env.py:138-139)
    T dz = s.bp[2] - s.rp[2], dy = s.bp[1] - s.rp[1];
    T delta = M<T>::sqrt(dz * dz + dy * dy);
    T reward = 0;
    if (bits & TB_EV_RACKET_BALL) { reward += 25; reward += dist_to_reward(delta); c.hit = 1; }
    T xbr = s.bp[0] - s.rp[0];
    if (!(xbr < (T)0.5)) { c.done = true; reward += dist_to_reward(delta); c.events |= TB_EV_BALL_PASSED; }
    if (k > 1000) { c.done = true; c.events |= TB_EV_TIMEOUT; }
    c.reward = (float)reward;
    return true;
  }
}

// ------------------------------------------------------------------------------------------------ fast-forward
// SwingRacket's 26th step (swingracket_env.py:105-141) repeats the same torque-free substep up to 775 times, so it
// has its own restatement of physics_step + the env logic, equal to env_substep's phases 1 and 2 in exact arithmetic
// and to ~1e-16 per substep in floating point, at half the double-precision work:
//   * the racket's angular velocity is carried in the BODY frame (s.rw holds R^T omega between ff_enter and ff_leave).
//     With no torque, omega_body <- omega_body + dt * alpha_body(omega_body) is closed: the pose update rotates
//     about omega itself, which leaves R^T omega unchanged; and exp(omega dt) q = q exp(omega_body dt).  No rotation
//     matrix is needed for the dynamics at all.  The principal axes are the body axes, so the gyroscopic term is
//     three products with host-side constants;
//   * damping enters as one factor per body, v <- v (1 - dt k (1 + |v|)) + dt g, the force law as a velocity
//     increment per metre;
//   * detection evaluates one coordinate each first: the ball's face-normal coordinate in the racket frame (one
//     column of R), its height against floor / net / goal, the racket's COM height against TB_EV_RACKET_LOW.  All
//     three rejects are conservative; whatever passes runs the same exact tests as physics_step.
template <typename T> struct FfRare {
  T rq[4], bv[3], bw[3], rv[3], wl[3];  // in/out: pose + velocities after force integration (omega in the body frame)
};
__device__ __forceinline__ bool nonzero3(const float *a) {
  return ((__float_as_uint(a[0]) | __float_as_uint(a[1]) | __float_as_uint(a[2])) & 0x7fffffffu) != 0;
}
__device__ __forceinline__ bool nonzero3(const double *a) {
  unsigned hi = (unsigned)(__double2hiint(a[0]) | __double2hiint(a[1]) | __double2hiint(a[2])) & 0x7fffffffu;
  unsigned lo = (unsigned)(__double2loint(a[0]) | __double2loint(a[1]) | __double2loint(a[2]));
  return (hi | lo) != 0;
}
// Rare continuation of a substep: contact solve and / or the exact +-max_coord_vel clamp, both of which act on the
// world-frame angular velocity.  Out of line; data crosses through FfRare only.
template <typename T>
__device__ __noinline__ void ff_rare(const Scene<T> &sc, const ContactSet<T> *cs, int nc, FfRare<T> *io) {
  T R[9], w[3];
  quat_to_mat(io->rq, R);
  mat_vec(R, io->wl, w);
  const T vmax = sc.max_coord_vel;
  T bv[3] = {io->bv[0], io->bv[1], io->bv[2]}, bw[3] = {io->bw[0], io->bw[1], io->bw[2]};
  T rv[3] = {io->rv[0], io->rv[1], io->rv[2]};
  clamp_velocities(bv, bw, rv, w, vmax, sc.vmax_hi);
  if (nc > 0) {
    SolveIO<T> so;
#pragma unroll
    for (int i = 0; i < 3; ++i) { so.bv[i] = bv[i]; so.bw[i] = bw[i]; so.rv[i] = rv[i]; so.rw[i] = w[i]; }
#pragma unroll
    for (int i = 0; i < 4; ++i) so.rq[i] = io->rq[i];
    solve_contacts(sc, cs, nc, &so);
#pragma unroll
    for (int i = 0; i < 3; ++i) { bv[i] += so.dvb[i]; bw[i] += so.dwb[i]; rv[i] += so.dva[i]; w[i] += so.dwa[i]; }
    clamp_velocities(bv, bw, rv, w, vmax, sc.vmax_hi);
  }
  T wl[3];
  matT_vec(R, w, wl);
#pragma unroll
  for (int i = 0; i < 3; ++i) { io->bv[i] = bv[i]; io->bw[i] = bw[i]; io->rv[i] = rv[i]; io->wl[i] = wl[i]; }
}

// world <-> body frame of the racket's angular velocity, once per env on either side of the fast-forward
template <typename T> __device__ __forceinline__ void ff_enter(St<T> &s) {
  T R[9], wl[3];
  quat_to_mat(s.rq, R);
  matT_vec(R, s.rw, wl);
  s.rw[0] = wl[0]; s.rw[1] = wl[1]; s.rw[2] = wl[2];
}
template <typename T> __device__ __forceinline__ void ff_leave(St<T> &s) {
  T R[9], w[3];
  quat_to_mat(s.rq, R);
  mat_vec(R, s.rw, w);
  s.rw[0] = w[0]; s.rw[1] = w[1]; s.rw[2] = w[2];
}

// One fast-forward substep + the env logic that follows it (swingracket_env.py:105-141).  c.phase is 1 on the first
// substep (no external force: the control step cleared it) and 2 afterwards.  Returns true when the env step is over.
template <typename T> __device__ __forceinline__ bool ff_substep(const Scene<T> &sc, St<T> &s, StepCtl &c) {
  const T dt = sc.dt, thr = sc.contact_threshold, rb = sc.ball_r;
  ContactSet<T> cs;  // local memory; rare path only
  int nc = 0, bits = 0;

  // ---- (1) detection at the start-of-step poses
  {
    int need = 0;
    const T x = s.rq[0], y = s.rq[1], z = s.rq[2], w = s.rq[3];
    const T r6 = 2 * (x * z - y * w);
    T rel[3] = {s.bp[0] - s.rp[0], s.bp[1] - s.rp[1], s.bp[2] - s.rp[2]};
    T pl0 = (1 - 2 * (y * y + z * z)) * rel[0] + 2 * (x * y + z * w) * rel[1] + r6 * rel[2];
    if (TB_UNLIKELY(!(M<T>::abs(pl0) > sc.ff_slab))) {  // inside the plate's slab: the remaining racket rejects
      T R[9], pl[3];
      quat_to_mat(s.rq, R);
      matT_vec(R, rel, pl);
      const T reach = rb + sc.hull_margin + thr, rs = sc.racket.bound_radius + reach;
      bool near_racket = dot3(rel, rel) <= rs * rs && !(M<T>::abs(pl[0]) - sc.racket.half_thick > reach) &&
                         !(M<T>::abs(pl[1]) - sc.racket_box[0] > reach) && !(pl[2] - sc.racket_box[2] > reach) &&
                         !(sc.racket_box[1] - pl[2] > reach);
      need |= near_racket ? kNeedRacket : 0;
    }
    if (TB_UNLIKELY(!(s.bp[2] > sc.ff_ball_z))) {  // low enough to reach the floor, the net's top or the goal's
      const T reach_b = rb + sc.box_margin + thr;
      need |= !(M<T>::abs(s.bp[2]) - sc.floor_h[2] > reach_b || M<T>::abs(s.bp[0]) - sc.floor_h[0] > reach_b ||
                M<T>::abs(s.bp[1]) - sc.floor_h[1] > reach_b) ? kNeedFloor : 0;
      need |= !(M<T>::abs(s.bp[0]) - sc.net_h[0] > reach_b || M<T>::abs(s.bp[2]) - sc.net_h[2] > reach_b ||
                M<T>::abs(s.bp[1]) - sc.net_h[1] > reach_b) ? kNeedNet : 0;
      const T reach_g = rb + sc.hull_margin + thr, rxy = sc.goal_r + reach_g;
      T gx = s.bp[0] - s.goal[0], gy = s.bp[1] - s.goal[1];
      need |= (M<T>::abs(s.bp[2]) - sc.goal_hz <= reach_g && gx * gx + gy * gy <= rxy * rxy) ? kNeedGoal : 0;
    }
    if (!(s.rp[2] > sc.ff_low_z)) {  // TB_EV_RACKET_LOW, exact test as in physics_step
      T r7 = 2 * (y * z + x * w), r8 = 1 - 2 * (x * x + y * y);
      T zlo = r8 * sc.racket_obb[1], zhi = r8 * sc.racket_obb[2];
      T low = s.rp[2] - M<T>::abs(r6) * sc.racket.half_thick - M<T>::abs(r7) * sc.racket_obb[0] + (zlo < zhi ? zlo : zhi) -
              sc.hull_margin;
      bits |= (low <= sc.floor_h[2] + thr && M<T>::abs(s.rp[0]) <= sc.floor_h[0] + 1 && M<T>::abs(s.rp[1]) <= sc.floor_h[1] + 1)
                  ? TB_EV_RACKET_LOW : 0;
    }
    if (sc.racket_court && (bits & TB_EV_RACKET_LOW)) need |= kNeedRacketFloor;
    if (TB_UNLIKELY(need)) {
      NarrowIn<T> in;
#pragma unroll
      for (int i = 0; i < 3; ++i) { in.rp[i] = s.rp[i]; in.bp[i] = s.bp[i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i) in.rq[i] = s.rq[i];
      in.goal[0] = s.goal[0]; in.goal[1] = s.goal[1];
      int r = narrow_phase<T, true>(sc, need, &in, &cs);
      bits |= r & 0xff;
      nc = r >> 8;
    }
  }

  // ---- (2) velocities
  {
    T fb = 1 - sc.ff_kl * (1 + M<T>::norm_damp(dot3(s.bv, s.bv)));
    s.bv[0] *= fb; s.bv[1] *= fb; s.bv[2] = s.bv[2] * fb + sc.ff_dtg;
    if (nonzero3(s.bw)) {  // the ball spins only after a frictional contact
      T fs = 1 - sc.ff_ka * (1 + M<T>::norm_damp(dot3(s.bw, s.bw)));
      s.bw[0] *= fs; s.bw[1] *= fs; s.bw[2] *= fs;
    }
    T fr = 1 - sc.ff_kl * (1 + M<T>::norm_damp(dot3(s.rv, s.rv)));
    T h0 = 0, h1 = 0, h2 = sc.ff_dtg;
    if (c.phase == 2) {  // the force the reference queued from the pose the previous substep ended with (:135-141)
      h0 = sc.ff_hack[0] * (s.rp[0] - s.aux[0]);  // s.aux = spawn + (0, 0, 4) here, see ff_full
      h1 = sc.ff_hack[1] * (s.rp[1] - s.aux[1]);
      h2 = sc.ff_hack[2] * (s.rp[2] - s.aux[2]) + sc.ff_dtg;
    }
    s.rv[0] = s.rv[0] * fr + h0; s.rv[1] = s.rv[1] * fr + h1; s.rv[2] = s.rv[2] * fr + h2;
    T fw = 1 - sc.ff_ka * (1 + M<T>::norm_damp(dot3(s.rw, s.rw)));
    T p12 = s.rw[1] * s.rw[2], p20 = s.rw[2] * s.rw[0], p01 = s.rw[0] * s.rw[1];
    s.rw[0] = s.rw[0] * fw - sc.ff_gyro[0] * p12;
    s.rw[1] = s.rw[1] * fw - sc.ff_gyro[1] * p20;
    s.rw[2] = s.rw[2] * fw - sc.ff_gyro[2] * p01;
  }
  T a2 = dot3(s.rw, s.rw);
  {
    bool over = near_limit(a2, sc.vmax2_hi);  // some world coordinate of omega may have reached the limit
#pragma unroll
    for (int i = 0; i < 3; ++i) over = over | near_limit(s.bv[i], sc.vmax_hi) | near_limit(s.bw[i], sc.vmax_hi) | near_limit(s.rv[i], sc.vmax_hi);
    // ---- (3) contact solve, exact clamps
    if (TB_UNLIKELY(over || nc > 0)) {
      FfRare<T> io;
#pragma unroll
      for (int i = 0; i < 3; ++i) { io.bv[i] = s.bv[i]; io.bw[i] = s.bw[i]; io.rv[i] = s.rv[i]; io.wl[i] = s.rw[i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i) io.rq[i] = s.rq[i];
      ff_rare(sc, &cs, nc, &io);
#pragma unroll
      for (int i = 0; i < 3; ++i) { s.bv[i] = io.bv[i]; s.bw[i] = io.bw[i]; s.rv[i] = io.rv[i]; s.rw[i] = io.wl[i]; }
      a2 = dot3(s.rw, s.rw);
    }
  }

  // ---- (4) poses: x += dt v ; q <- q exp(omega_body dt), renormalised to first order (see integrate_quat)
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    s.bp[i] += dt * s.bv[i];
    s.rp[i] += dt * s.rv[i];
  }
  {
    T sinc, cw;
    sinc_cos_x2(sc.ff_qx2 * a2, &sinc, &cw);
    T k = (T)0.5 * dt * sinc;
    T ax = s.rw[0] * k, ay = s.rw[1] * k, az = s.rw[2] * k;
    const T q0 = s.rq[0], q1 = s.rq[1], q2 = s.rq[2], q3 = s.rq[3];
    T x = cw * q0 + ax * q3 + az * q1 - ay * q2;
    T y = cw * q1 + ay * q3 + ax * q2 - az * q0;
    T z = cw * q2 + az * q3 + ay * q0 - ax * q1;
    T w = cw * q3 - ax * q0 - ay * q1 - az * q2;
    T n2 = x * x + y * y + z * z + w * w;
    T inv = (T)1.5 - (T)0.5 * n2;
    if (TB_UNLIKELY(M<T>::abs(n2 - 1) > (T)1e-4)) inv = fast_rsqrt(n2);
    s.rq[0] = x * inv; s.rq[1] = y * inv; s.rq[2] = z * inv; s.rq[3] = w * inv;
  }

  // ---- env logic (swingracket_env.py:109-133)
  int k = ++s.step;
  c.events |= bits;
  c.last = bits;
  c.phase = 2;
  T reward = 0;
  if (bits & TB_EV_COURT_BALL) { c.done = true; reward += moved_dist_to_goal(s); }
  if (bits & TB_EV_GOAL_BALL) { reward += moved_dist_to_goal(s); reward += 50; c.done = true; }
  if (k > 800) { c.done = true; c.events |= TB_EV_TIMEOUT; }
  if (c.done) c.reward = (float)reward;
  return c.done;
}

// ------------------------------------------------------------------------------------------------ fast lane
// What a lane of ff_kernel keeps in registers between substeps: omega in the body frame, tgt = spawn + (0,0,4), the
// squared speeds nb, nr, nw of ball, racket and omega - the classification of a state needs them and the next
// substep's damping factors reuse them - and the ball's spin rate sb = |bw|, which free flight only scales
// (bw <- bw f, so |bw| <- |bw| f: no square root per substep).  rq is NOT renormalised per substep here: the product
// of unit quaternions drifts from unit length by rounding only (~1e-16 per substep, < 1e-14 over the longest flight);
// ff_kernel renormalises when the lane's state goes back to HBM.
template <typename T> struct FfLane {
  T rp[3], rq[4], rv[3], wl[3], bp[3], bv[3], bw[3], tgt[3], goal[2], nb, nr, nw, sb;
  int step, events;
};
// How the substep that starts from a state has to be taken:
constexpr int kFfFree = 0;  // ff_fast, no contact possible
constexpr int kFfLand = 1;  // ff_fast with the floor-face contact hook: the ball is within reach of the court's top face only
constexpr int kFfFull = 2;  // ff_full: racket slab, net, goal or a floor edge within reach, the 800-step time-out, a speed
                            // near the +-max_coord_vel clamp or |omega| beyond the short half-angle series
constexpr int kFfDone = 3;  // (returned by the step functions) the env step is over
// Conservative (a lane may be sent to ff_full for nothing, never the other way), and decided by the env's own state
// only, so which path integrates a given substep never depends on the other lanes of the warp.
// nb, nr, nw: squared speeds of ball, racket and racket spin.
// QUICK: the outline test with its quick accept / reject first (ff_kernel's loops); else the plain loop (step_kernel).
// Around the rim: is the ball within `rim` of the hull?  pl0: its face-normal coordinate, max_side: the largest signed
// distance to an edge line of the outline (a lower bound of the in-plane distance to it).  Beyond the plate's thickness
// AND beyond the outline the two offsets are orthogonal, so the distance is at least their root sum of squares; taking
// each bound alone (a mitred corner around the rim's edge) kept a ball that falls alongside the racket "within reach"
// for tens of substeps in which the narrow phase found nothing.  Used by step_kernel's classification (fewer control
// substeps deferred to the generic path); ff_kernel's flight loop keeps the cheaper bound, see there.
template <typename T> __device__ __forceinline__ bool ff_rim_within(const Scene<T> &sc, T pl0, T max_side) {
  T et = M<T>::abs(pl0) - sc.racket.half_thick;
  et = et > 0 ? et : (T)0;
  const T ms = max_side > 0 ? max_side : (T)0;
  return !(et * et + ms * ms > sc.ffp_rim * sc.ffp_rim);
}
template <typename T, bool WITH_GOAL = true, bool QUICK = false>
__device__ __forceinline__ int ff_classify_core(const Scene<T> &sc, const T *rp, const T *rq, const T *bp, const T *goal, T nb, T nr,
                                                T nw, int step) {
  const T x = rq[0], y = rq[1], z = rq[2], w = rq[3];
  T rel[3] = {bp[0] - rp[0], bp[1] - rp[1], bp[2] - rp[2]};
  T pl0 = (1 - 2 * (y * y + z * z)) * rel[0] + 2 * (x * y + z * w) * rel[1] + 2 * (x * z - y * w) * rel[2];
  // bitwise on purpose: one straight line of compares, no short-circuit branches
  bool racket = !(M<T>::abs(pl0) > sc.ff_slab) & !(dot3(rel, rel) > sc.ffp_racket_r2);
  if (TB_UNLIKELY(racket)) {  // inside the plate's slab and the hull's bounding sphere: the outline's bounding box decides
    T pl1 = 2 * (x * y - z * w) * rel[0] + (1 - 2 * (x * x + z * z)) * rel[1] + 2 * (y * z + x * w) * rel[2];
    T pl2 = 2 * (x * z + y * w) * rel[0] + 2 * (y * z - x * w) * rel[1] + (1 - 2 * (x * x + y * y)) * rel[2];
    racket = !(M<T>::abs(pl1) > sc.ffp_box[0]) & !(pl2 > sc.ffp_box[2]) & !(pl2 < sc.ffp_box[1]);
    if (QUICK && racket) {
      // ... and the outline itself.  Two quick tests settle all but a thin band around it (a flight lane whose ball falls
      // alongside the racket comes here every substep); there the signed distance to every edge line decides (a lower
      // bound of the distance to the hull).  The opaque copies pin all of this into the cold block: hoisted into the
      // straight line of the substep it would cost every lane ~20 FP64 instructions, and as an out-of-line call it split
      // the substep loop's schedule (measured on B200: +7 % on the whole fast-forward launch).
      T q1 = pl1, q2 = pl2;
      opaque(q1); opaque(q2);
      if (prism_inside_fast(sc.racket, q1, q2)) racket = true;
      else if (prism_outside_fast(sc.racket, q1, q2, sc.ffp_rim)) racket = false;
      else {  // the coarse outline decides (it contains the outline: the signed distance to its edge lines is a lower bound too)
        T max_side = -M<T>::inf();
#pragma unroll kCoarseUnroll
        for (int i = 0; i < kCoarseEdges; ++i) {
          T side = (q1 - sc.racket.c_ax[i]) * sc.racket.c_nx[i] + (q2 - sc.racket.c_ay[i]) * sc.racket.c_ny[i];
          max_side = side > max_side ? side : max_side;
        }
        // (the in-plane bound alone: ff_rim_within here keeps a ball in the corner band in this lane, where it takes the edge
        // loop above every substep with the other 31 lanes waiting - measured +0.06 ms per launch, more than the servers save)
        racket = !(max_side > sc.ffp_rim);
      }
    } else if (!QUICK && racket) {
      // ... and the outline itself: the signed distance to any edge line is a lower bound of the distance to the hull.
      T max_side = -M<T>::inf();
#pragma unroll kEdgeUnroll
      for (int i = 0; i < kRacketEdges; ++i) {
        const Edge<T> &e = sc.racket.e[i];
        T side = (pl1 - e.ax) * e.nx + (pl2 - e.ay) * e.ny;
        max_side = side > max_side ? side : max_side;
      }
      racket = ff_rim_within(sc, pl0, max_side);
    }
  }
  const T ax = M<T>::abs(bp[0]), ay = M<T>::abs(bp[1]), az = M<T>::abs(bp[2]);
  bool full = racket | (!(ax > sc.ffp_net[0]) & !(az > sc.ffp_net[2]) & !(ay > sc.ffp_net[1])) |
              !(nb < sc.ffp_v2) | !(nr < sc.ffp_v2) | !(nw < sc.ffp_a2);
  if (TB_UNLIKELY(sc.racket_court != 0)) full |= racket_low(sc, rp, rq);  // racket-court contact lives on the generic path
  if (WITH_GOAL) {  // SwingRacket: the goal disc and the 800-step time-out (Tennisbot-v0 has neither in its scene)
    T gx = bp[0] - goal[0], gy = bp[1] - goal[1];
    full |= (!(az > sc.ffp_goal_z) & !(gx * gx + gy * gy > sc.ffp_goal_r2)) | (step >= 800);
  }
  bool floor = !(az > sc.ffp_floor[2]) & !(ax > sc.ffp_floor[0]) & !(ay > sc.ffp_floor[1]);
  bool face = (bp[2] > sc.ffp_face[2]) & (ax < sc.ffp_face[0]) & (ay < sc.ffp_face[1]);
  return (full | (floor & !face)) ? kFfFull : (floor ? kFfLand : kFfFree);
}
template <typename T> __device__ __forceinline__ int ff_classify(const Scene<T> &sc, FfLane<T> &L) {
  L.nb = dot3(L.bv, L.bv); L.nr = dot3(L.rv, L.rv); L.nw = dot3(L.wl, L.wl);
  return ff_classify_core<T, true, true>(sc, L.rp, L.rq, L.bp, L.goal, L.nb, L.nr, L.nw, L.step);
}
// the same for a state record (omega in the world frame: same norm)
template <typename T> __device__ __forceinline__ int ff_classify_state(const Scene<T> &sc, const St<T> &s) {
  return ff_classify_core(sc, s.rp, s.rq, s.bp, s.goal, dot3(s.bv, s.bv), dot3(s.rv, s.rv), dot3(s.rw, s.rw), s.step);
}

// The control-phase substep of SwingRacket-v0 (swingracket_env.py:76-83) for an env that ff_classify_state() puts in
// kFfFree: the substep cannot touch anything, so it is physics_step without detection, contact solve and clamps, as
// one straight line: force and torque of the action at the COM (racket.py:92-100), damping as one factor per body,
// Euler's equations in the body (= principal) frame, q <- q exp(omega_body dt) with the short half-angle series (the
// classification bounds |omega| and every speed with room for one substep of the largest action).  Equal to
// physics_step in exact arithmetic, to ~1e-16 per substep in floating point.  Returns the event bits of the substep
// (TB_EV_RACKET_LOW at most).  step_kernel defers every other env to the generic path (ff_kernel's prologue).
// the ball's part of a contact-free substep: damping as one factor, gravity (shared with the kernel that tabulates ball_vz)
template <typename T> __device__ __forceinline__ void ball_free_velocities(const Scene<T> &sc, T *bv, T *bw) {
  T fb = 1 - sc.ff_kl * (1 + M<T>::norm_damp(dot3(bv, bv)));
  bv[0] *= fb; bv[1] *= fb; bv[2] = bv[2] * fb + sc.ff_dtg;
  T fs = 1 - sc.ff_ka * (1 + M<T>::norm_damp(dot3(bw, bw)));
  bw[0] *= fs; bw[1] *= fs; bw[2] *= fs;
}
// a state whose pack 4 was not loaded / is stale in HBM (kStPristine): the ball's velocity from the table, no spin
template <typename T> __device__ __forceinline__ void materialise_ball(const Scene<T> &sc, St<T> &s) {
  if (s.flags & kStPristine) {
    s.bv[0] = 0; s.bv[1] = 0; s.bv[2] = sc.ball_vz[s.step < kBallVzEntries ? s.step : kBallVzEntries - 1];
    s.bw[0] = 0;
  }
}
template <typename T> __device__ __forceinline__ int ctl_fast(const Scene<T> &sc, St<T> &s, const float *a) {
  const T dt = sc.dt;
  T R[9];
  quat_to_mat(s.rq, R);
  int bits;
  {  // TB_EV_RACKET_LOW at the start-of-step pose, exact test as in physics_step
    T zlo = R[8] * sc.racket_obb[1], zhi = R[8] * sc.racket_obb[2];
    T low = s.rp[2] - M<T>::abs(R[6]) * sc.racket.half_thick - M<T>::abs(R[7]) * sc.racket_obb[0] + (zlo < zhi ? zlo : zhi) - sc.hull_margin;
    bool is_low = (low <= sc.ffp_low) & (M<T>::abs(s.rp[0]) <= sc.ffp_court[0]) & (M<T>::abs(s.rp[1]) <= sc.ffp_court[1]);
    bits = is_low ? TB_EV_RACKET_LOW : 0;
  }
  const T F[3] = {(T)a[0] * 400, (T)a[1] * 400, (T)a[2] * 400 + (T)(4 * 9.81)};
  const T Tq[3] = {(T)a[3] * 5, (T)a[4] * 5, (T)a[5] * 5};
  ball_free_velocities(sc, s.bv, s.bw);
  T fr = 1 - sc.ff_kl * (1 + M<T>::norm_damp(dot3(s.rv, s.rv)));
  const T dtm = dt * sc.racket_inv_m;
  s.rv[0] = s.rv[0] * fr + dtm * F[0]; s.rv[1] = s.rv[1] * fr + dtm * F[1]; s.rv[2] = s.rv[2] * fr + (dtm * F[2] + sc.ff_dtg);
  T fw = 1 - sc.ff_ka * (1 + M<T>::norm_damp(dot3(s.rw, s.rw)));  // |omega| is the same in both frames
  T wl[3], tl[3];
  matT_vec(R, s.rw, wl);
  matT_vec(R, Tq, tl);
  T p12 = wl[1] * wl[2], p20 = wl[2] * wl[0], p01 = wl[0] * wl[1];
  wl[0] = wl[0] * fw - sc.ff_gyro[0] * p12 + dt * sc.racket_inv_i[0] * tl[0];
  wl[1] = wl[1] * fw - sc.ff_gyro[1] * p20 + dt * sc.racket_inv_i[1] * tl[1];
  wl[2] = wl[2] * fw - sc.ff_gyro[2] * p01 + dt * sc.racket_inv_i[2] * tl[2];
  mat_vec(R, wl, s.rw);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    s.bp[i] += dt * s.bv[i];
    s.rp[i] += dt * s.rv[i];
  }
  {
    T sinc, cw;
    sinc_cos_short(sc.ff_qx2 * dot3(wl, wl), &sinc, &cw);
    T k = (T)0.5 * dt * sinc;
    T ax = wl[0] * k, ay = wl[1] * k, az = wl[2] * k;
    const T q0 = s.rq[0], q1 = s.rq[1], q2 = s.rq[2], q3 = s.rq[3];
    T x = cw * q0 + ax * q3 + az * q1 - ay * q2;
    T y = cw * q1 + ay * q3 + ax * q2 - az * q0;
    T z = cw * q2 + az * q3 + ay * q0 - ax * q1;
    T w = cw * q3 - ax * q0 - ay * q1 - az * q2;
    T n2 = x * x + y * y + z * z + w * w;
    T inv = (T)1.5 - (T)0.5 * n2;  // first-order renormalisation, see integrate_quat
    if (TB_UNLIKELY(M<T>::abs(n2 - 1) > (T)1e-4)) inv = fast_rsqrt(n2);
    s.rq[0] = x * inv; s.rq[1] = y * inv; s.rq[2] = z * inv; s.rq[3] = w * inv;
  }
  return bits;
}

// Tennisbot-v0's substep (tennisbot_env.py:112-121) for a state ff_classify_core<T, false> does not send to the generic
// path: physics_step<T, false> without detection, solve and clamps, as one straight line - planar force on the racket
// at the COM (racket.py:92-100), the shoot force on the ball during the first frames (objects.py:67-72), damping as one
// factor per body, and the one contact that is routine in this env, the ball's bounce on the court's top face
// (kind == kFfLand), in closed form exactly as in ff_fast below.  The racket only rotates after a ball has hit it
// (no torque is ever applied): that case runs Euler's equations in the body frame like ctl_fast.  Equal to
// physics_step in exact arithmetic, to ~1e-16 per substep in floating point.  Returns the event bits of the substep
// (TB_EV_RACKET_LOW, TB_EV_COURT_BALL).
template <typename T> __device__ __forceinline__ int hit_fast(const Scene<T> &sc, St<T> &s, const T *F, const T *Fb, int kind) {
  const T dt = sc.dt;
  int bits;
  {  // TB_EV_RACKET_LOW at the start-of-step pose, exact test as in physics_step
    const T x = s.rq[0], y = s.rq[1], z = s.rq[2], w = s.rq[3];
    T r6 = 2 * (x * z - y * w), r7 = 2 * (y * z + x * w), r8 = 1 - 2 * (x * x + y * y);
    T zlo = r8 * sc.racket_obb[1], zhi = r8 * sc.racket_obb[2];
    T low = s.rp[2] - M<T>::abs(r6) * sc.racket.half_thick - M<T>::abs(r7) * sc.racket_obb[0] + (zlo < zhi ? zlo : zhi) - sc.hull_margin;
    bool is_low = (low <= sc.ffp_low) & (M<T>::abs(s.rp[0]) <= sc.ffp_court[0]) & (M<T>::abs(s.rp[1]) <= sc.ffp_court[1]);
    bits = is_low ? TB_EV_RACKET_LOW : 0;
  }
  // signed distance of the ball to the court's top face at the start-of-step pose (box_distance's face case)
  const T d_floor = (s.bp[2] - (sc.floor_h[2] - sc.box_margin)) - (sc.ball_r + sc.box_margin);
  const T dtb = dt * sc.ball_inv_m, dtm = dt * sc.racket_inv_m;
  T fb = 1 - sc.ff_kl * (1 + M<T>::norm_damp(dot3(s.bv, s.bv)));
  s.bv[0] = s.bv[0] * fb + dtb * Fb[0]; s.bv[1] = s.bv[1] * fb + dtb * Fb[1]; s.bv[2] = s.bv[2] * fb + (dtb * Fb[2] + sc.ff_dtg);
  T fs = 1 - sc.ff_ka * (1 + M<T>::norm_damp(dot3(s.bw, s.bw)));
  s.bw[0] *= fs; s.bw[1] *= fs; s.bw[2] *= fs;
  T fr = 1 - sc.ff_kl * (1 + M<T>::norm_damp(dot3(s.rv, s.rv)));
  s.rv[0] = s.rv[0] * fr + dtm * F[0]; s.rv[1] = s.rv[1] * fr + dtm * F[1]; s.rv[2] = s.rv[2] * fr + (dtm * F[2] + sc.ff_dtg);
  const bool rotating = (s.rw[0] != 0) | (s.rw[1] != 0) | (s.rw[2] != 0);
  T wl[3] = {0, 0, 0};
  if (TB_UNLIKELY(rotating)) {
    T R[9];
    quat_to_mat(s.rq, R);
    T fw = 1 - sc.ff_ka * (1 + M<T>::norm_damp(dot3(s.rw, s.rw)));  // |omega| is the same in both frames
    matT_vec(R, s.rw, wl);
    T p12 = wl[1] * wl[2], p20 = wl[2] * wl[0], p01 = wl[0] * wl[1];
    wl[0] = wl[0] * fw - sc.ff_gyro[0] * p12;
    wl[1] = wl[1] * fw - sc.ff_gyro[1] * p20;
    wl[2] = wl[2] * fw - sc.ff_gyro[2] * p01;
    mat_vec(R, wl, s.rw);
  }
  if (TB_UNLIKELY(kind == kFfLand && d_floor <= sc.contact_threshold)) {  // the bounce: see ff_fast
    bits |= TB_EV_COURT_BALL;
    const T rb = sc.ball_r, inv_m = sc.ball_inv_m, inv_i = sc.ball_inv_i;
    T rel = s.bv[2];
    T e = M<T>::abs(rel) < sc.rest_vel_threshold ? (T)0 : -sc.rest_court * rel;
    if (e < 0) e = 0;
    T pen = d_floor + sc.slop, vel_err = e - rel, pos_err = 0;
    if (pen > 0) vel_err -= pen * sc.ffl_inv_dt;
    else pos_err = -pen * sc.ffl_erp_dt;
    T lam_n = (pos_err + vel_err) * sc.ffl_m;
    if (lam_n > 0) {
      s.bv[2] += lam_n * inv_m;
      T s1 = (s.bv[1] + rb * s.bw[0]) * sc.ffl_jinv_t, s2 = -(s.bv[0] - rb * s.bw[1]) * sc.ffl_jinv_t;
      T lim = sc.mu_court * lam_n, m2 = s1 * s1 + s2 * s2;
      if (m2 > lim * lim) {
        T y = (T)rsqrtf((float)m2);  // float estimate + two Newton steps: ~1e-15 relative
        y = y * ((T)1.5 - (T)0.5 * m2 * y * y);
        y = y * ((T)1.5 - (T)0.5 * m2 * y * y);
        T sf = lim * y;
        s1 *= sf; s2 *= sf;
      }
      s.bv[1] -= s1 * inv_m; s.bw[0] -= rb * s1 * inv_i;
      s.bv[0] += s2 * inv_m; s.bw[1] -= rb * s2 * inv_i;
      const T vmax = sc.max_coord_vel;  // the clamp physics_step applies after a solve
#pragma unroll
      for (int i = 0; i < 3; ++i) { s.bv[i] = clampv(s.bv[i], -vmax, vmax); s.bw[i] = clampv(s.bw[i], -vmax, vmax); }
    }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    s.bp[i] += dt * s.bv[i];
    s.rp[i] += dt * s.rv[i];
  }
  if (TB_UNLIKELY(rotating)) {
    T sinc, cw;
    sinc_cos_short(sc.ff_qx2 * dot3(wl, wl), &sinc, &cw);
    T k = (T)0.5 * dt * sinc;
    T ax = wl[0] * k, ay = wl[1] * k, az = wl[2] * k;
    const T q0 = s.rq[0], q1 = s.rq[1], q2 = s.rq[2], q3 = s.rq[3];
    T x = cw * q0 + ax * q3 + az * q1 - ay * q2;
    T y = cw * q1 + ay * q3 + ax * q2 - az * q0;
    T z = cw * q2 + az * q3 + ay * q0 - ax * q1;
    T w = cw * q3 - ax * q0 - ay * q1 - az * q2;
    T n2 = x * x + y * y + z * z + w * w;
    T inv = (T)1.5 - (T)0.5 * n2;  // first-order renormalisation, see integrate_quat
    if (TB_UNLIKELY(M<T>::abs(n2 - 1) > (T)1e-4)) inv = fast_rsqrt(n2);
    s.rq[0] = x * inv; s.rq[1] = y * inv; s.rq[2] = z * inv; s.rq[3] = w * inv;
  }
  return bits;
}
// The generic substep of Tennisbot-v0, out of line (ball within reach of the racket, the net or an edge of the floor; a
// speed near the clamp): data crosses through *r only, so the caller's state stays in registers around the call.
template <typename T> struct HitRec {
  T rp[3], rq[4], rv[3], rw[3], bp[3], bv[3], bw[3], F[3], Fb[3];
};
template <typename T> __device__ __noinline__ int hit_generic(const Scene<T> &sc, HitRec<T> *r) {
  St<T> s;
  T zero[3] = {0, 0, 0}, F[3], Fb[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    s.rp[i] = r->rp[i]; s.rv[i] = r->rv[i]; s.rw[i] = r->rw[i]; s.bp[i] = r->bp[i]; s.bv[i] = r->bv[i]; s.bw[i] = r->bw[i];
    F[i] = r->F[i]; Fb[i] = r->Fb[i];
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) s.rq[i] = r->rq[i];
  int bits = physics_step<T, false>(sc, s, F, zero, Fb);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    r->rp[i] = s.rp[i]; r->rv[i] = s.rv[i]; r->rw[i] = s.rw[i]; r->bp[i] = s.bp[i]; r->bv[i] = s.bv[i]; r->bw[i] = s.bw[i];
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) r->rq[i] = s.rq[i];
  return bits;
}

// One stepSimulation() of Tennisbot-v0 with racket force F and ball force Fb: contact-free substeps and bounces on the
// court's top face take the straight line, everything else the generic step out of line (a few substeps per episode:
// ball within reach of the racket, the net or a floor edge).  Returns the event bits.
template <typename T> __device__ __forceinline__ int hit_physics(const Scene<T> &sc, St<T> &s, const T *F, const T *Fb) {
  int bits;
  const int kind = ff_classify_core<T, false>(sc, s.rp, s.rq, s.bp, s.goal, dot3(s.bv, s.bv), dot3(s.rv, s.rv), dot3(s.rw, s.rw), 0);
  if (kind != kFfFull) {
    bits = hit_fast<T>(sc, s, F, Fb, kind);
  } else {
    HitRec<T> r;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      r.rp[i] = s.rp[i]; r.rv[i] = s.rv[i]; r.rw[i] = s.rw[i]; r.bp[i] = s.bp[i]; r.bv[i] = s.bv[i]; r.bw[i] = s.bw[i];
      r.F[i] = F[i]; r.Fb[i] = Fb[i];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) r.rq[i] = s.rq[i];
    bits = hit_generic<T>(sc, &r);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      s.rp[i] = r.rp[i]; s.rv[i] = r.rv[i]; s.rw[i] = r.rw[i]; s.bp[i] = r.bp[i]; s.bv[i] = r.bv[i]; s.bw[i] = r.bw[i];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) s.rq[i] = r.rq[i];
  }
  return bits;
}

// The substep without a narrow phase: ff_substep with phase 2, no clamp, the short series and at most the one contact
// a free-falling ball ends almost every flight with - the court's top face (kind == kFfLand).  There the contact
// normal is +z, the tangents btPlaneSpace1 gives are -y and +x, and the three rows of a single sphere contact
// against a static body are orthogonal in the mass metric (r x n = 0), so projected Gauss-Seidel converges in its
// first sweep: normal impulse = max(0, rhs), friction pair = rhs scaled into the cone.  solve_contacts' second
// sweep would change that by rounding only.  Only valid from a state ff_classify() did not send to ff_full.
// Returns ff_classify() of the state it leaves, or kFfDone after a landing (TB_EV_COURT_BALL set in L.events).
template <typename T> __device__ __forceinline__ int ff_fast(const Scene<T> &sc, FfLane<T> &L, int kind) {
  const T dt = sc.dt;
  {  // TB_EV_RACKET_LOW at the start-of-step pose, exact test as in physics_step
    const T x = L.rq[0], y = L.rq[1], z = L.rq[2], w = L.rq[3];
    T r6 = 2 * (x * z - y * w), r7 = 2 * (y * z + x * w), r8 = 1 - 2 * (x * x + y * y);
    T zlo = r8 * sc.racket_obb[1], zhi = r8 * sc.racket_obb[2];
    T low = L.rp[2] - M<T>::abs(r6) * sc.racket.half_thick - M<T>::abs(r7) * sc.racket_obb[0] + (zlo < zhi ? zlo : zhi) - sc.hull_margin;
    bool is_low = (low <= sc.ffp_low) & (M<T>::abs(L.rp[0]) <= sc.ffp_court[0]) & (M<T>::abs(L.rp[1]) <= sc.ffp_court[1]);
    L.events |= is_low ? TB_EV_RACKET_LOW : 0;
  }
  // signed distance of the ball to the court's top face at the start-of-step pose (box_distance's face case)
  const T d_floor = (L.bp[2] - (sc.floor_h[2] - sc.box_margin)) - (sc.ball_r + sc.box_margin);
  T fb = 1 - sc.ff_kl * (1 + M<T>::norm_damp(L.nb));
  L.bv[0] *= fb; L.bv[1] *= fb; L.bv[2] = L.bv[2] * fb + sc.ff_dtg;
  {  // unconditional: a warp almost always holds a ball that spins, and 0 * f stays 0 for the others
    T fs = 1 - sc.ff_ka * (1 + L.sb);
    L.bw[0] *= fs; L.bw[1] *= fs; L.bw[2] *= fs; L.sb *= fs;
  }
  T fr = 1 - sc.ff_kl * (1 + M<T>::norm_damp(L.nr));
  L.rv[0] = L.rv[0] * fr + sc.ff_hack[0] * (L.rp[0] - L.tgt[0]);
  L.rv[1] = L.rv[1] * fr + sc.ff_hack[1] * (L.rp[1] - L.tgt[1]);
  L.rv[2] = L.rv[2] * fr + (sc.ff_hack[2] * (L.rp[2] - L.tgt[2]) + sc.ff_dtg);
  T fw = 1 - sc.ff_ka * (1 + M<T>::norm_damp(L.nw));
  T p12 = L.wl[1] * L.wl[2], p20 = L.wl[2] * L.wl[0], p01 = L.wl[0] * L.wl[1];
  L.wl[0] = L.wl[0] * fw - sc.ff_gyro[0] * p12;
  L.wl[1] = L.wl[1] * fw - sc.ff_gyro[1] * p20;
  L.wl[2] = L.wl[2] * fw - sc.ff_gyro[2] * p01;
  bool landed = false;
  if (TB_UNLIKELY(kind == kFfLand && d_floor <= sc.contact_threshold)) {
    landed = true;
    L.events |= TB_EV_COURT_BALL;
    const T rb = sc.ball_r, inv_m = sc.ball_inv_m, inv_i = sc.ball_inv_i;
    // normal row: u = (0,0,1), r x u = 0.  Divisions by constants are products with host-side reciprocals (the
    // block sits in the substep loop's instruction footprint).
    T rel = L.bv[2];
    T e = M<T>::abs(rel) < sc.rest_vel_threshold ? (T)0 : -sc.rest_court * rel;
    if (e < 0) e = 0;
    T pen = d_floor + sc.slop, vel_err = e - rel, pos_err = 0;
    if (pen > 0) vel_err -= pen * sc.ffl_inv_dt;
    else pos_err = -pen * sc.ffl_erp_dt;
    T lam_n = (pos_err + vel_err) * sc.ffl_m;
    if (lam_n > 0) {
      L.bv[2] += lam_n * inv_m;
      // friction pair: u1 = (0,-1,0), r x u1 = (-rb,0,0); u2 = (1,0,0), r x u2 = (0,-rb,0)
      T s1 = (L.bv[1] + rb * L.bw[0]) * sc.ffl_jinv_t, s2 = -(L.bv[0] - rb * L.bw[1]) * sc.ffl_jinv_t;
      T lim = sc.mu_court * lam_n, m2 = s1 * s1 + s2 * s2;
      if (m2 > lim * lim) {
        T y = (T)rsqrtf((float)m2);  // float estimate + two Newton steps: ~1e-15 relative
        y = y * ((T)1.5 - (T)0.5 * m2 * y * y);
        y = y * ((T)1.5 - (T)0.5 * m2 * y * y);
        T sf = lim * y;
        s1 *= sf; s2 *= sf;
      }
      L.bv[1] -= s1 * inv_m; L.bw[0] -= rb * s1 * inv_i;
      L.bv[0] += s2 * inv_m; L.bw[1] -= rb * s2 * inv_i;
      const T vmax = sc.max_coord_vel;  // the clamp physics_step applies after a solve
#pragma unroll
      for (int i = 0; i < 3; ++i) { L.bv[i] = clampv(L.bv[i], -vmax, vmax); L.bw[i] = clampv(L.bw[i], -vmax, vmax); }
    }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    L.bp[i] += dt * L.bv[i];
    L.rp[i] += dt * L.rv[i];
  }
  {
    T sinc, cw;
    sinc_cos_short(sc.ff_qx2 * dot3(L.wl, L.wl), &sinc, &cw);
    T k = (T)0.5 * dt * sinc;
    T ax = L.wl[0] * k, ay = L.wl[1] * k, az = L.wl[2] * k;
    const T q0 = L.rq[0], q1 = L.rq[1], q2 = L.rq[2], q3 = L.rq[3];
    T x = cw * q0 + ax * q3 + az * q1 - ay * q2;
    T y = cw * q1 + ay * q3 + ax * q2 - az * q0;
    T z = cw * q2 + az * q3 + ay * q0 - ax * q1;
    T w = cw * q3 - ax * q0 - ay * q1 - az * q2;
    L.rq[0] = x; L.rq[1] = y; L.rq[2] = z; L.rq[3] = w;
  }
  ++L.step;
  int next = ff_classify(sc, L);
  return landed ? kFfDone : next;
}

// The full substep (first substep of a flight that starts in contact, racket / net / goal / floor-edge contact,
// time-out, ...): ff_substep on a copy of the lane.  Out of line, data crosses through *Lp only.  Returns what comes
// next (kFfFree .. kFfDone); the env step's accumulated event bits are left in Lp->events, the contact bits of this
// substep alone in *last (the reward of the env step depends on those only, swingracket_env.py:111-126).
template <typename T>
__device__ __noinline__ int ff_full(const Scene<T> &sc, FfLane<T> *Lp, int phase, int *last) {
  St<T> s;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    s.rp[i] = Lp->rp[i]; s.rv[i] = Lp->rv[i]; s.rw[i] = Lp->wl[i]; s.bp[i] = Lp->bp[i]; s.bv[i] = Lp->bv[i];
    s.bw[i] = Lp->bw[i]; s.aux[i] = Lp->tgt[i];
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) s.rq[i] = Lp->rq[i];
  s.goal[0] = Lp->goal[0]; s.goal[1] = Lp->goal[1];
  s.d0 = 1; s.ret = 0; s.step = Lp->step; s.flags = 0; s.episode = 0;  // the reward is formed by ff_reward later
  StepCtl c = {phase, Lp->events, 0, 0.0f, false, 0};
  bool fin = ff_substep<T>(sc, s, c);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    Lp->rp[i] = s.rp[i]; Lp->rv[i] = s.rv[i]; Lp->wl[i] = s.rw[i]; Lp->bp[i] = s.bp[i]; Lp->bv[i] = s.bv[i];
    Lp->bw[i] = s.bw[i];
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) Lp->rq[i] = s.rq[i];
  Lp->step = s.step; Lp->events = c.events;
  Lp->sb = norm3(s.bw);
  *last = c.last;
  int next = ff_classify(sc, *Lp);
  return fin ? kFfDone : next;
}

// The server warps' short cut for the substep that fills most of their time: the ball is high above the court and meets -
// or just misses - the racket (over a face - projection inside the outline for certain, prism_inside_fast - the narrow
// phase is one coordinate; near the rim it is prism_distance's loops).  Same substep as
// ff_substep in exact arithmetic, to rounding otherwise, with a fraction of the instructions (a lone lane's generic substep
// is bound by instruction fetch: ~3000 instructions of cold code):
//   * the single contact's three rows are solved in IMPULSE space: A = J M^-1 J^T (3 x 3) once, then projected Gauss-Seidel
//     on lambda alone - sweep for sweep what solve_contacts does on the velocities (jd_i = sum_j A_ij lambda_j), the same
//     clamps and the same residual test, so it stops after the same sweep;
//   * everything that involves the racket's rotation stays in its body frame: J's angular part is q x (R^T u), the effective
//     inertia is diagonal there, and omega_body takes the impulse directly - no world-frame angular velocity, no R I^-1 R^T.
// Returns what comes next like ff_full (the env step cannot end here), or -1 without touching *Lp when the state is outside
// what this covers (ball low enough for the court, the net or the goal; a speed near the clamp; the time-out step): ff_full
// takes it then.
template <typename T>
__device__ __noinline__ int ff_contact_lean(const Scene<T> &sc, FfLane<T> *Lp, int phase, int *last) {
  if (sizeof(T) != 8) return -1;  // (the float32 kernel keeps the generic path: its rows are solved in double there)
  const T dt = sc.dt, thr = sc.contact_threshold, rb = sc.ball_r;
  if (!(Lp->nb < sc.ffp_v2) | !(Lp->nr < sc.ffp_v2) | !(Lp->nw < sc.ffp_a2) | (Lp->step >= 799)) return -1;
  if (!(Lp->bp[2] > sc.ff_ball_z)) {  // low ball: only if the court, the net and the goal are all out of reach (ff_substep's tests)
    const T b0 = Lp->bp[0], b1 = Lp->bp[1], b2 = Lp->bp[2];
    const T reach_b = rb + sc.box_margin + thr, reach_g = rb + sc.hull_margin + thr, rxy = sc.goal_r + reach_g;
    const T gx = b0 - Lp->goal[0], gy = b1 - Lp->goal[1];
    const bool floor = !(M<T>::abs(b2) - sc.floor_h[2] > reach_b || M<T>::abs(b0) - sc.floor_h[0] > reach_b || M<T>::abs(b1) - sc.floor_h[1] > reach_b);
    const bool net = !(M<T>::abs(b0) - sc.net_h[0] > reach_b || M<T>::abs(b2) - sc.net_h[2] > reach_b || M<T>::abs(b1) - sc.net_h[1] > reach_b);
    const bool goal = M<T>::abs(b2) - sc.goal_hz <= reach_g && gx * gx + gy * gy <= rxy * rxy;
    if (floor | net | goal) return -1;
  }
  T R[9], rq[4] = {Lp->rq[0], Lp->rq[1], Lp->rq[2], Lp->rq[3]};
  quat_to_mat(rq, R);
  const T rp[3] = {Lp->rp[0], Lp->rp[1], Lp->rp[2]}, bp[3] = {Lp->bp[0], Lp->bp[1], Lp->bp[2]};
  T rel[3] = {bp[0] - rp[0], bp[1] - rp[1], bp[2] - rp[2]}, pl[3];
  matT_vec(R, rel, pl);
  // ---- (1) detection at the start-of-step poses
  int bits = 0;
  bool contact = false;
  T d = 0, nl[3] = {1, 0, 0}, ql[3] = {0, 0, 0};  // normal and closest point of the hull core in the racket frame
  {
    const T reach = rb + sc.hull_margin + thr, rs = sc.racket.bound_radius + reach;
    const bool near_racket = dot3(rel, rel) <= rs * rs && !(M<T>::abs(pl[0]) - sc.racket.half_thick > reach) &&
                             !(M<T>::abs(pl[1]) - sc.racket_box[0] > reach) && !(pl[2] - sc.racket_box[2] > reach) &&
                             !(sc.racket_box[1] - pl[2] > reach);
    if (near_racket) {
      const T et = M<T>::abs(pl[0]) - sc.racket.half_thick;
      T dc;
      if (et > 0 && prism_inside_fast(sc.racket, pl[1], pl[2])) {  // over a face
        const T st = pl[0] < 0 ? (T)-1 : (T)1;
        dc = et;
        nl[0] = st;
        ql[0] = st * sc.racket.half_thick; ql[1] = pl[1]; ql[2] = pl[2];
      } else {  // near the rim, or inside the plate: the loops over the outline
        dc = prism_distance<T, kRacketEdges>(sc.racket, pl[0], pl[1], pl[2], reach * (T)1.0001, nl, ql);
      }
      d = dc - (rb + sc.hull_margin);
      contact = d <= thr;
    }
    T zlo = R[8] * sc.racket_obb[1], zhi = R[8] * sc.racket_obb[2];
    T low = rp[2] - M<T>::abs(R[6]) * sc.racket.half_thick - M<T>::abs(R[7]) * sc.racket_obb[0] + (zlo < zhi ? zlo : zhi) - sc.hull_margin;
    bits |= (low <= sc.floor_h[2] + thr && M<T>::abs(rp[0]) <= sc.floor_h[0] + 1 && M<T>::abs(rp[1]) <= sc.floor_h[1] + 1) ? TB_EV_RACKET_LOW : 0;
    if (sc.racket_court && bits) return -1;  // racket on the court: its contact points join the solve (generic path)
  }
  // ---- (2) velocities, as in ff_substep
  T bv[3] = {Lp->bv[0], Lp->bv[1], Lp->bv[2]}, bw[3] = {Lp->bw[0], Lp->bw[1], Lp->bw[2]};
  T rv[3] = {Lp->rv[0], Lp->rv[1], Lp->rv[2]}, wl[3] = {Lp->wl[0], Lp->wl[1], Lp->wl[2]};
  {
    T fb = 1 - sc.ff_kl * (1 + M<T>::norm_damp(Lp->nb));
    bv[0] *= fb; bv[1] *= fb; bv[2] = bv[2] * fb + sc.ff_dtg;
    if (nonzero3(bw)) {
      T fs = 1 - sc.ff_ka * (1 + M<T>::norm_damp(dot3(bw, bw)));
      bw[0] *= fs; bw[1] *= fs; bw[2] *= fs;
    }
    T fr = 1 - sc.ff_kl * (1 + M<T>::norm_damp(Lp->nr));
    T h0 = 0, h1 = 0, h2 = sc.ff_dtg;
    if (phase == 2) {
      h0 = sc.ff_hack[0] * (rp[0] - Lp->tgt[0]);
      h1 = sc.ff_hack[1] * (rp[1] - Lp->tgt[1]);
      h2 = sc.ff_hack[2] * (rp[2] - Lp->tgt[2]) + sc.ff_dtg;
    }
    rv[0] = rv[0] * fr + h0; rv[1] = rv[1] * fr + h1; rv[2] = rv[2] * fr + h2;
    T fw = 1 - sc.ff_ka * (1 + M<T>::norm_damp(Lp->nw));
    T p12 = wl[1] * wl[2], p20 = wl[2] * wl[0], p01 = wl[0] * wl[1];
    wl[0] = wl[0] * fw - sc.ff_gyro[0] * p12;
    wl[1] = wl[1] * fw - sc.ff_gyro[1] * p20;
    wl[2] = wl[2] * fw - sc.ff_gyro[2] * p01;
  }
  // ---- (3) the contact
  if (contact) {
    bits |= TB_EV_RACKET_BALL;
    const T inv_mb = sc.ball_inv_m, inv_ib = sc.ball_inv_i, inv_mr = sc.racket_inv_m;
    // world frame: normal u0 = R nl and Bullet's two tangents; body frame: ub_j = R^T u_j, contact point qs on the hull
    T u[3][3], ub[3][3], l[3][3], li[3][3], rbxu[3][3];
    mat_vec(R, nl, u[0]);
    plane_space<T>(u[0], u[1], u[2]);
    ub[0][0] = nl[0]; ub[0][1] = nl[1]; ub[0][2] = nl[2];
    matT_vec(R, u[1], ub[1]);
    matT_vec(R, u[2], ub[2]);
    const T qs[3] = {ql[0] + sc.hull_margin * nl[0], ql[1] + sc.hull_margin * nl[1], ql[2] + sc.hull_margin * nl[2]};
    const T rbv[3] = {-rb * u[0][0], -rb * u[0][1], -rb * u[0][2]};
    T A[3][3], jinv[3], rhs[3], lam[3] = {0, 0, 0};
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      cross3(qs, ub[j], l[j]);
      cross3(rbv, u[j], rbxu[j]);
#pragma unroll
      for (int i = 0; i < 3; ++i) li[j][i] = l[j][i] * sc.racket_inv_i[i];
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      T relv = dot3(u[j], bv) + dot3(rbxu[j], bw) - (dot3(u[j], rv) + dot3(l[j], wl));
      A[j][j] = inv_mb + dot3(rbxu[j], rbxu[j]) * inv_ib + (inv_mr + dot3(l[j], li[j]));
      jinv[j] = 1 / A[j][j];
      if (j == 0) {
        T e = M<T>::abs(relv) < sc.rest_vel_threshold ? (T)0 : -sc.rest_racket * relv;
        if (e < 0) e = 0;
        T pen = d + sc.slop, vel_err = e - relv, pos_err = 0;
        if (pen > 0) vel_err -= pen / dt;
        else pos_err = -pen * sc.erp / dt;
        rhs[0] = (pos_err + vel_err) * jinv[0];
      } else {
        rhs[j] = -relv * jinv[j];
      }
    }
    A[0][1] = A[1][0] = dot3(l[0], li[1]); A[0][2] = A[2][0] = dot3(l[0], li[2]); A[1][2] = A[2][1] = dot3(l[1], li[2]);
#pragma unroll 1
    for (int it = 0; it < sc.iters; ++it) {
      T resid = 0;
      {
        T jd = A[0][0] * lam[0] + A[0][1] * lam[1] + A[0][2] * lam[2];
        T dl = rhs[0] - jd * jinv[0], sum = lam[0] + dl;
        if (sum < 0) { dl = -lam[0]; sum = 0; }
        lam[0] = sum;
        T rr = dl * A[0][0];
        resid = rr * rr;
      }
      if (lam[0] > 0) {
        const T lim = sc.mu_racket * lam[0];
        T jd1 = A[1][0] * lam[0] + A[1][1] * lam[1] + A[1][2] * lam[2], jd2 = A[2][0] * lam[0] + A[2][1] * lam[1] + A[2][2] * lam[2];
        T s1 = lam[1] + (rhs[1] - jd1 * jinv[1]), s2 = lam[2] + (rhs[2] - jd2 * jinv[2]);
        T m2 = s1 * s1 + s2 * s2;
        if (m2 > lim * lim) {
          T sf = lim / M<T>::sqrt(m2);
          s1 *= sf; s2 *= sf;
        }
        T r1 = (s1 - lam[1]) * A[1][1], r2 = (s2 - lam[2]) * A[2][2];
        lam[1] = s1; lam[2] = s2;
        if (r1 * r1 > resid) resid = r1 * r1;
        if (r2 * r2 > resid) resid = r2 * r2;
      }
      if (resid <= sc.solver_residual) break;
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      T ju = u[0][i] * lam[0] + u[1][i] * lam[1] + u[2][i] * lam[2];
      bv[i] += ju * inv_mb;
      rv[i] -= ju * inv_mr;
      bw[i] += (rbxu[0][i] * lam[0] + rbxu[1][i] * lam[1] + rbxu[2][i] * lam[2]) * inv_ib;
      wl[i] -= li[0][i] * lam[0] + li[1][i] * lam[1] + li[2][i] * lam[2];
    }
    // Bullet's +-max_coord_vel clamp after the solve (world coordinates of omega): far away in practice, exact when not
    bool over = near_limit(dot3(wl, wl), sc.vmax2_hi);
#pragma unroll
    for (int i = 0; i < 3; ++i) over = over | near_limit(bv[i], sc.vmax_hi) | near_limit(bw[i], sc.vmax_hi) | near_limit(rv[i], sc.vmax_hi);
    if (TB_UNLIKELY(over)) {
      T w[3];
      mat_vec(R, wl, w);
      clamp_velocities(bv, bw, rv, w, sc.max_coord_vel, sc.vmax_hi);
      matT_vec(R, w, wl);
    }
  }
  // ---- (4) poses, as in ff_substep
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    Lp->bp[i] = bp[i] + dt * bv[i];
    Lp->rp[i] = rp[i] + dt * rv[i];
    Lp->bv[i] = bv[i]; Lp->bw[i] = bw[i]; Lp->rv[i] = rv[i]; Lp->wl[i] = wl[i];
  }
  {
    T sinc, cw;
    sinc_cos_x2(sc.ff_qx2 * dot3(wl, wl), &sinc, &cw);
    T k = (T)0.5 * dt * sinc;
    T ax = wl[0] * k, ay = wl[1] * k, az = wl[2] * k;
    T x = cw * rq[0] + ax * rq[3] + az * rq[1] - ay * rq[2];
    T y = cw * rq[1] + ay * rq[3] + ax * rq[2] - az * rq[0];
    T z = cw * rq[2] + az * rq[3] + ay * rq[0] - ax * rq[1];
    T w = cw * rq[3] - ax * rq[0] - ay * rq[1] - az * rq[2];
    T n2 = x * x + y * y + z * z + w * w;
    T inv = (T)1.5 - (T)0.5 * n2;
    if (TB_UNLIKELY(M<T>::abs(n2 - 1) > (T)1e-4)) inv = fast_rsqrt(n2);
    Lp->rq[0] = x * inv; Lp->rq[1] = y * inv; Lp->rq[2] = z * inv; Lp->rq[3] = w * inv;
  }
  // ---- env logic (swingracket_env.py:109-133): no court or goal contact and no time-out is possible here
  Lp->step += 1;
  Lp->events |= bits;
  Lp->sb = norm3(bw);
  *last = bits;
  return ff_classify(sc, *Lp);
}

// Reward of the env step a fast-forward ended with, from the contact bits of its last substep (swingracket_env.py:111-126;
// same order of operations as ff_substep).
template <typename T> __device__ __forceinline__ float ff_reward(const St<T> &s, int last) {
  T reward = 0;
  if (last & TB_EV_COURT_BALL) reward += moved_dist_to_goal(s);
  if (last & TB_EV_GOAL_BALL) { reward += moved_dist_to_goal(s); reward += 50; }
  return (float)reward;
}

}  // namespace tb
