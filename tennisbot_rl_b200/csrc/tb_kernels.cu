// tb_kernels.cu - kernels and the C ABI of libtennisbot_b200.so (include/tennisbot_b200.h).
//
// HBM layout: the state of N envs is 8 "packs" of 4 scalars, pack-major: element (pack p, env i) sits at
// ((p * N + i) * 4) scalars.  A warp therefore reads/writes 32 consecutive 16-byte (f32) or 32-byte (f64)
// records per pack: fully coalesced 128-bit accesses, 128 B (f32) / 256 B (f64) of state per env each way.
//   pack0 racket pos xyz | ball pos x      pack4 ball vel xyz  | ball angvel x
//   pack1 racket quat xyzw                 pack5 ball angvel yz | aux x, aux y
//   pack2 racket vel xyz | ball pos y      pack6 aux z | goal x, goal y | d0
//   pack3 racket angvel xyz | ball pos z   pack7 return | step | flags | episode   (integers bit-cast)
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <type_traits>
#include <utility>
#include <vector>

#include "tb_device.cuh"

namespace tb {

constexpr int kPacks = 8;
constexpr int kBlock = 128;     // threads per CTA of the step kernel
// CTAs per SM ff_kernel's register budget is held to: 5 x 128 threads -> 96 regs/thread (f32), 4 -> 128 (f64); measured best on B200
template <typename T> struct MinBlocks { static constexpr int v = 5; };
template <> struct MinBlocks<double> { static constexpr int v = 4; };

// ------------------------------------------------------------------------------------------------ pack I/O
template <typename T> struct Pack { T x, y, z, w; };

__device__ __forceinline__ Pack<float> ld_pack(const float *base, int64_t n, int p, int64_t i) {
  float4 v = *reinterpret_cast<const float4 *>(base + ((int64_t)p * n + i) * 4);
  return {v.x, v.y, v.z, v.w};
}
__device__ __forceinline__ void st_pack(float *base, int64_t n, int p, int64_t i, Pack<float> v) {
  *reinterpret_cast<float4 *>(base + ((int64_t)p * n + i) * 4) = make_float4(v.x, v.y, v.z, v.w);
}
__device__ __forceinline__ Pack<double> ld_pack(const double *base, int64_t n, int p, int64_t i) {
  const double2 *q = reinterpret_cast<const double2 *>(base + ((int64_t)p * n + i) * 4);
  double2 a = q[0], b = q[1];
  return {a.x, a.y, b.x, b.y};
}
__device__ __forceinline__ void st_pack(double *base, int64_t n, int p, int64_t i, Pack<double> v) {
  double2 *q = reinterpret_cast<double2 *>(base + ((int64_t)p * n + i) * 4);
  q[0] = make_double2(v.x, v.y);
  q[1] = make_double2(v.z, v.w);
}
__device__ __forceinline__ float int_as(float, int64_t v) { return __int_as_float((int)v); }
__device__ __forceinline__ double int_as(double, int64_t v) { return __longlong_as_double((long long)v); }
__device__ __forceinline__ int64_t as_int(float v) { return (int64_t)__float_as_int(v); }
__device__ __forceinline__ int64_t as_int(double v) { return (int64_t)__double_as_longlong(v); }

template <typename T> __device__ __forceinline__ void load_state(const T *base, int64_t n, int64_t i, St<T> &s) {
  Pack<T> p0 = ld_pack(base, n, 0, i), p1 = ld_pack(base, n, 1, i), p2 = ld_pack(base, n, 2, i),
          p3 = ld_pack(base, n, 3, i), p4 = ld_pack(base, n, 4, i), p5 = ld_pack(base, n, 5, i),
          p6 = ld_pack(base, n, 6, i), p7 = ld_pack(base, n, 7, i);
  s.rp[0] = p0.x; s.rp[1] = p0.y; s.rp[2] = p0.z; s.bp[0] = p0.w;
  s.rq[0] = p1.x; s.rq[1] = p1.y; s.rq[2] = p1.z; s.rq[3] = p1.w;
  s.rv[0] = p2.x; s.rv[1] = p2.y; s.rv[2] = p2.z; s.bp[1] = p2.w;
  s.rw[0] = p3.x; s.rw[1] = p3.y; s.rw[2] = p3.z; s.bp[2] = p3.w;
  s.bv[0] = p4.x; s.bv[1] = p4.y; s.bv[2] = p4.z; s.bw[0] = p4.w;
  s.bw[1] = p5.x; s.bw[2] = p5.y; s.aux[0] = p5.z; s.aux[1] = p5.w;
  s.aux[2] = p6.x; s.goal[0] = p6.y; s.goal[1] = p6.z; s.d0 = p6.w;
  s.ret = p7.x; s.step = (int)as_int(p7.y); s.flags = (int)as_int(p7.z); s.episode = (uint32_t)as_int(p7.w);
}
// Packs 5 and 6 hold episode constants (spawn / shoot force, goal, d0) next to the y, z spin of the ball, which is zero
// until a frictional contact: step_kernel writes them back only when they changed (p5: spin or reset, p6: reset).
template <typename T> __device__ __forceinline__ int flags_with_spin(const St<T> &s) {
  return (s.flags & ~kStSpin) | ((s.bw[1] != 0 || s.bw[2] != 0) ? kStSpin : 0);
}
template <typename T> __device__ __forceinline__ void store_state_changed(T *base, int64_t n, int64_t i, const St<T> &s, bool p5, bool p6, bool have_aux = true) {
  st_pack(base, n, 0, i, Pack<T>{s.rp[0], s.rp[1], s.rp[2], s.bp[0]});
  st_pack(base, n, 1, i, Pack<T>{s.rq[0], s.rq[1], s.rq[2], s.rq[3]});
  st_pack(base, n, 2, i, Pack<T>{s.rv[0], s.rv[1], s.rv[2], s.bp[1]});
  st_pack(base, n, 3, i, Pack<T>{s.rw[0], s.rw[1], s.rw[2], s.bp[2]});
  if (!(s.flags & kStPristine) || p6) st_pack(base, n, 4, i, Pack<T>{s.bv[0], s.bv[1], s.bv[2], s.bw[0]});  // (p6: episode restarted)
  if (p5 && have_aux) st_pack(base, n, 5, i, Pack<T>{s.bw[1], s.bw[2], s.aux[0], s.aux[1]});
  if (p5 && !have_aux) {  // (pack 5 was not loaded: its aux half stays as it is in HBM)
    T *q = base + ((int64_t)5 * n + i) * 4;
    q[0] = s.bw[1]; q[1] = s.bw[2];
  }
  if (p6) st_pack(base, n, 6, i, Pack<T>{s.aux[2], s.goal[0], s.goal[1], s.d0});
  st_pack(base, n, 7, i, Pack<T>{s.ret, int_as(T(), s.step), int_as(T(), flags_with_spin(s)), int_as(T(), (int64_t)s.episode)});
}
template <typename T> __device__ __forceinline__ void store_state(T *base, int64_t n, int64_t i, const St<T> &s) {
  st_pack(base, n, 0, i, Pack<T>{s.rp[0], s.rp[1], s.rp[2], s.bp[0]});
  st_pack(base, n, 1, i, Pack<T>{s.rq[0], s.rq[1], s.rq[2], s.rq[3]});
  st_pack(base, n, 2, i, Pack<T>{s.rv[0], s.rv[1], s.rv[2], s.bp[1]});
  st_pack(base, n, 3, i, Pack<T>{s.rw[0], s.rw[1], s.rw[2], s.bp[2]});
  st_pack(base, n, 4, i, Pack<T>{s.bv[0], s.bv[1], s.bv[2], s.bw[0]});
  st_pack(base, n, 5, i, Pack<T>{s.bw[1], s.bw[2], s.aux[0], s.aux[1]});
  st_pack(base, n, 6, i, Pack<T>{s.aux[2], s.goal[0], s.goal[1], s.d0});
  st_pack(base, n, 7, i, Pack<T>{s.ret, int_as(T(), s.step), int_as(T(), flags_with_spin(s)), int_as(T(), (int64_t)s.episode)});
}

// step_kernel's load: the packs a control step needs.  Packs 5 and 6 (ball spin y, z | episode constants) are loaded only
// when the flags word says they carry something that cannot be had otherwise (kStSpin, kStDerived); the goal of an RNG-placed
// SwingRacket episode is re-derived from the counter-based generator - the kernel is HBM-bound with issue slots to spare.
// aux and d0 stay undefined then: a control step never reads them, and pack 5 / 6 are only written back by a lane that
// loaded them (spin changed) or restarted the episode (all fields fresh).
// Returns whether pack 5 was loaded (if not, its aux half is unknown and a lane whose spin changes writes the spin half only).
template <typename T, int KIND>
__device__ __forceinline__ bool load_state_ctl(const Scene<T> &sc, const T *base, int64_t n, int64_t i, uint64_t seed, uint64_t gid, St<T> &s) {
  Pack<T> p0 = ld_pack(base, n, 0, i), p1 = ld_pack(base, n, 1, i), p2 = ld_pack(base, n, 2, i),
          p3 = ld_pack(base, n, 3, i), p7 = ld_pack(base, n, 7, i);
  s.rp[0] = p0.x; s.rp[1] = p0.y; s.rp[2] = p0.z; s.bp[0] = p0.w;
  s.rq[0] = p1.x; s.rq[1] = p1.y; s.rq[2] = p1.z; s.rq[3] = p1.w;
  s.rv[0] = p2.x; s.rv[1] = p2.y; s.rv[2] = p2.z; s.bp[1] = p2.w;
  s.rw[0] = p3.x; s.rw[1] = p3.y; s.rw[2] = p3.z; s.bp[2] = p3.w;
  s.ret = p7.x; s.step = (int)as_int(p7.y); s.flags = (int)as_int(p7.z); s.episode = (uint32_t)as_int(p7.w);
  if (KIND == TB_ENV_SWING && (s.flags & kStPristine)) {  // ball in free fall from rest: pack 4 is a table entry
    materialise_ball(sc, s);
  } else {
    Pack<T> p4 = ld_pack(base, n, 4, i);
    s.bv[0] = p4.x; s.bv[1] = p4.y; s.bv[2] = p4.z; s.bw[0] = p4.w;
  }
  const bool derived = (s.flags & kStDerived) != 0;
  // Tennisbot-v0 reads the shoot force (aux x, y in pack 5) during the first frames of every episode
  const bool need5 = (s.flags & kStSpin) != 0 || (KIND == TB_ENV_HIT && s.step < sc.shoot_start + sc.shoot_frames) || (KIND == TB_ENV_SWING && !derived);
  s.bw[1] = 0; s.bw[2] = 0; s.aux[0] = 0; s.aux[1] = 0; s.aux[2] = 0; s.goal[0] = 0; s.goal[1] = 0; s.d0 = 0;
  if (need5) {
    Pack<T> p5 = ld_pack(base, n, 5, i);
    s.bw[1] = p5.x; s.bw[2] = p5.y; s.aux[0] = p5.z; s.aux[1] = p5.w;
  }
  if (!derived) {
    Pack<T> p6 = ld_pack(base, n, 6, i);
    s.aux[2] = p6.x; s.goal[0] = p6.y; s.goal[1] = p6.z; s.d0 = p6.w;
  } else if (KIND == TB_ENV_SWING) {
    T in[TB_INIT_WORDS];
    draw_init<T, KIND>(seed, gid, s.episode, in);
    s.goal[0] = in[3]; s.goal[1] = in[4];
  } else {
    s.aux[2] = (T)(25.0 * 0.8);  // tennisbot_env.py:237: the z shoot force is a constant (place())
  }
  return need5;
}

// controller memory of TB_CONTROL_PID: two more packs per env in a separate array (allocated when the mode is set)
template <typename T> __device__ __forceinline__ void load_pid(const T *pb, int64_t n, int64_t i, T *pid) {
  Pack<T> a = ld_pack(pb, n, 0, i), b = ld_pack(pb, n, 1, i);
  pid[0] = a.x; pid[1] = a.y; pid[2] = a.z; pid[3] = a.w; pid[4] = b.x; pid[5] = b.y; pid[6] = b.z; pid[7] = b.w;
}
template <typename T> __device__ __forceinline__ void store_pid(T *pb, int64_t n, int64_t i, const T *pid) {
  st_pack(pb, n, 0, i, Pack<T>{pid[0], pid[1], pid[2], pid[3]});
  st_pack(pb, n, 1, i, Pack<T>{pid[4], pid[5], pid[6], pid[7]});
}

// ------------------------------------------------------------------------------------------------ kernels
struct StepIO {
  void *state;
  int64_t n, id_offset;
  uint64_t seed;
  int auto_reset, k_steps, action_mode;
  const float *actions;
  float *obs, *reward, *term_obs, *reward_sum;
  uint8_t *done, *events;
  int32_t *done_count;
  unsigned long long *stats;
  int *queue;                        // env indices waiting for ff_kernel: long flights from the front, short from the back
  int *queue_full;                   // envs whose FIRST fast-forward substep needs the full treatment (step_kernel fills it)
  int *queue_ctl;                    // SwingRacket envs whose control-phase substep needs the generic path (deferred by
                                     // step_kernel, taken by ff_kernel's prologue)
  unsigned long long *dq_full, *dq_late;  // ff_kernel's dynamic queues (slots tagged with `epoch`): envs parked for a full
                                     // substep; envs whose flight goes on after one.  dq_cap slots each
  long long dq_cap;
  unsigned *epoch;                   // three device words: [0] steps completed (read by step_kernel, advanced by ff_kernel),
                                     // [1] = [0] + 1 written by step_kernel = the tag of this step's queue slots,
                                     // [2] Tennisbot-v0 steps completed (advanced by step_kernel; no ff_kernel advances [0]
                                     // there): the noise counter of the policy rollout
  int prefetch_ahead;                // step_kernel: CTAs resident at a time (the L2 prefetch distance), 0 = none
  unsigned long long *fault;         // sticky: non-zero once a wait inside ff_kernel has timed out (every later call on the
                                     // context fails); fault_host: the same word in mapped host memory, read by the host
                                     // without synchronising
  volatile unsigned long long *fault_host;
  long long spin_limit;              // clock cycles any wait inside ff_kernel may take before the launch gives up
  int server_sm_stride;              // ff_kernel: > 0 = every warp on an SM whose id is a multiple of this is a server warp and
                                     // all others are flight warps (full persistent grids); 0 = one server warp per
                                     // kServerStride CTAs
  unsigned long long *queue_ctrs;    // two sets of kCtrWords counters (kC* below) used by alternate steps: [0] front,
                                     // [1] back entries appended by the step's step_kernel, the rest ff_kernel's.  Which set
                                     // a step uses is decided on the device (ctr_sets), so captured CUDA graphs of any
                                     // number of steps can be replayed
  void *pid;                         // TB_CONTROL_PID: 2 packs x N of controller memory, else nullptr
};

template <int KIND> struct Dims {
  static constexpr int obs = KIND == TB_ENV_SWING ? 6 : 12;
  static constexpr int act = KIND == TB_ENV_SWING ? 6 : 2;
};

template <int KIND> __device__ __forceinline__ void load_action(const float *actions, int64_t i, float *a) {
  if (KIND == TB_ENV_SWING) {
    const float2 *p = reinterpret_cast<const float2 *>(actions + i * 6);
    float2 a0 = p[0], a1 = p[1], a2 = p[2];
    a[0] = a0.x; a[1] = a0.y; a[2] = a1.x; a[3] = a1.y; a[4] = a2.x; a[5] = a2.y;
  } else {
    float2 v = *reinterpret_cast<const float2 *>(actions + i * 2);
    a[0] = v.x; a[1] = v.y;
  }
}
template <int KIND> __device__ __forceinline__ void store_obs(float *obs, int64_t i, const float *o) {
  if (KIND == TB_ENV_SWING) {
    float2 *p = reinterpret_cast<float2 *>(obs + i * 6);
    p[0] = make_float2(o[0], o[1]); p[1] = make_float2(o[2], o[3]); p[2] = make_float2(o[4], o[5]);
  } else {
    float4 *p = reinterpret_cast<float4 *>(obs + i * 12);
    p[0] = make_float4(o[0], o[1], o[2], o[3]); p[1] = make_float4(o[4], o[5], o[6], o[7]);
    p[2] = make_float4(o[8], o[9], o[10], o[11]);
  }
}
template <int KIND> __device__ __forceinline__ void random_action(uint64_t seed, uint64_t gid, uint32_t episode, int step, float *a) {
  uint32_t r[4];
#pragma unroll
  for (int b = 0; b * 4 < Dims<KIND>::act; ++b) {
    philox4x32(seed, gid, episode, stream_word(kStreamAction, (uint32_t)step, b), r);
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (b * 4 + q < 8) a[b * 4 + q] = 2.0f * u01<float>(r[q]) - 1.0f;
  }
}

// ------------------------------------------------------------------------------------------------ step kernels
// An env step is one physics substep for every env, except SwingRacket's 26th step, which goes on for up to
// 775 more.  The step is therefore issued as two launches on the same stream:
//
//   step_kernel  one thread per env, plain grid: loads state + action (128-bit coalesced), runs the substep the
//                action drives and the env logic; envs whose step is complete write obs / reward / done,
//                auto-reset and store their state.  HBM-bound.  SwingRacket: only the straight-line substep
//                (ctl_fast) lives here; an env within reach of anything is appended to a list instead.  Envs that
//                enter the fast-forward store their state with the in-flight mark and append their index to one of
//                three work lists (one atomic per CTA and list).  Tennisbot-v0: the straight-line substep hit_fast
//                (floor bounce in closed form) in line, the generic step out of line for the few states within reach
//                of the racket, the net or a floor edge.
//   ff_kernel    (SwingRacket) persistent; prologue: the deferred control substeps through the generic path, in dense
//                warps.  Then flight warps (every LANE a small state machine that claims an env, keeps its flight state
//                in registers, one straight-line substep per loop iteration) and server warps (generic substeps for
//                flights that come within reach of something), linked by ticketed queues; finally the completion pass
//                for every env that landed.  FP64-pipe / latency-bound; launched on every step, exits at once when
//                nothing is queued.
//
// Episode statistics are warp-uniform popc()/redux sums kept in shared memory, one atomic per counter per warp.
constexpr int kFlagDone = 1, kFlagInFlight = 2, kFlagEventShift = 8;
// marks ff_kernel's phases hand an env on with (all cleared again before the env step completes):
constexpr int kFlagLanded = 4;      // the env step is over; outputs / statistics / auto-reset pending
constexpr int kFlagFirst = 8;       // the flight's first substep (no external force) has not been taken yet
constexpr int kFlagLastShift = 16;  // contact bits of the flight's last substep
constexpr int kFlagVisitShift = 4;  // 2 bits: visits to the full path during this flight
// counter words of one step's set
constexpr int kCtrWords = 512;  // words that are polled never share a 128-byte line with words that are claimed from
constexpr int kCFront = 0, kCBack = 1, kCSafe = 2, kCError = 3;
constexpr int kDRounds = 48, kDFullEnvs = 49, kDPhase = 50, kDFinish = 62;  // tb_ff_diagnostics
constexpr int kCFull0 = 4;        // entries of queue_full (appended by step_kernel)
constexpr int kCClaim0 = 5;       // claimed entries of queue (ff_kernel's flight lanes)
constexpr int kCFullClaim0 = 6;   // claimed entries of queue_full (ff_kernel's servers)
constexpr int kCFullTail = 16, kCFullHead = 17;  // dq_full: reserved by producers / claimed by servers
constexpr int kCLateTail = 32, kCLateHead = 33;  // dq_late: reserved by servers / claimed by flight lanes
constexpr int kCCtl = 13;         // entries of queue_ctl
constexpr int kCCtlClaim = 14;    // claimed entries of queue_ctl (ff_kernel's prologue, 32 per warp)
constexpr int kCLanded = 64;      // envs whose env step is over (own line, with the two words below: idle warps poll them)
constexpr int kCCtlDone = 65;     // entries of queue_ctl that have been stepped (their flights, if any, are published)
constexpr int kCDynTotal = 66;    // flights that were queued by the prologue (on top of step_kernel's three lists)
constexpr int kCFinDone = 67;     // finishing pass 1: tiles of 32 envs that have been looked at
constexpr int kCRetryTail = 68;   // ... envs that were still in flight then (listed in queue_ctl, finished in pass 2)
constexpr int kCStarted = 9;      // ff_kernel CTAs that have taken their role; kCServers: those that are servers (role by SM)
constexpr int kCServers = 10;
constexpr int kCFinClaim = 7;     // finishing pass 1: claimed tiles
constexpr int kCRetryClaim = 8;   // finishing pass 2: claimed entries of the retry list

struct WarpStats {
  unsigned long long *acc;  // this warp's row of the CTA's shared accumulators
  int lane;
  __device__ __forceinline__ void init(unsigned long long *row, int l) {
    acc = row; lane = l;
    if (lane < TB_NUM_STATS) acc[lane] = 0;
    __syncwarp();
  }
  __device__ __forceinline__ void flush(unsigned long long *global) {
    __syncwarp();
    if (lane < TB_NUM_STATS) {
      unsigned long long v = acc[lane];
      if (v) atomicAdd(global + lane, v);
    }
  }
};

// Bookkeeping of completed env steps, called by all 32 lanes (fin = this lane's env step completed now).
template <typename T>
__device__ __forceinline__ void account(WarpStats &ws, bool fin, bool done, int hit, int events, int step, T ret) {
  const unsigned full = 0xffffffffu;
  unsigned fin_mask = __ballot_sync(full, fin);
  if (!TB_UNLIKELY(fin_mask)) return;
  bool dn = fin && done;
  unsigned done_mask = __ballot_sync(full, dn), hit_mask = __ballot_sync(full, fin && hit);
  if (done_mask) {
    unsigned goal_m = __ballot_sync(full, dn && (events & TB_EV_GOAL_BALL));
    unsigned court_m = __ballot_sync(full, dn && (events & TB_EV_COURT_BALL));
    unsigned to_m = __ballot_sync(full, dn && (events & TB_EV_TIMEOUT) &&
                                            !(events & (TB_EV_GOAL_BALL | TB_EV_COURT_BALL | TB_EV_BALL_PASSED)));
    int len = __reduce_add_sync(full, dn ? step : 0);
    double r = dn ? (double)ret : 0.0;
    long long r1 = __double2ll_rn(r * 1048576.0), r2 = __double2ll_rn(r * r * 1024.0);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      r1 += __shfl_down_sync(full, r1, o);
      r2 += __shfl_down_sync(full, r2, o);
    }
    if (ws.lane == 0) {
      ws.acc[TB_STAT_EPISODES] += __popc(done_mask);
      ws.acc[TB_STAT_SUM_LENGTH] += len;
      ws.acc[TB_STAT_GOALS] += __popc(goal_m);
      ws.acc[TB_STAT_COURT] += __popc(court_m);
      ws.acc[TB_STAT_TIMEOUTS] += __popc(to_m);
      ws.acc[TB_STAT_SUM_RETURN_Q20] += (unsigned long long)r1;
      ws.acc[TB_STAT_SUM_RETURN2_Q10] += (unsigned long long)r2;
    }
  }
  if (ws.lane == 0) {
    ws.acc[TB_STAT_ENV_STEPS] += __popc(fin_mask);
    ws.acc[TB_STAT_RACKET_HITS] += __popc(hit_mask);
  }
}

// Completion of an env step for one lane: terminal observation, auto-reset, outputs.  The caller stores the state.
// ob_out != nullptr: hand the observation row back instead of storing it (step_kernel stores whole tiles coalesced).
template <typename T, int KIND>
__device__ __forceinline__ void finish_api(const Scene<T> &sc, const StepIO &io, int64_t me, St<T> &s, float reward,
                                           bool done, int events, float *ob_out = nullptr) {
  float ob[12];
  pack_obs<T, KIND>(s, ob);
  if (done) {
    if (io.term_obs) store_obs<KIND>(io.term_obs, me, ob);
    if (io.auto_reset) {
      uint32_t ep = s.episode + 1;
      T in[TB_INIT_WORDS];
      draw_init<T, KIND>(io.seed, (uint64_t)(io.id_offset + me), ep, in);
      start_episode<T, KIND>(sc, s, in, ep, true);
      pack_obs<T, KIND>(s, ob);
    } else {
      s.flags |= kFlagDone;
    }
  }
  if (ob_out) {
#pragma unroll
    for (int j = 0; j < Dims<KIND>::obs; ++j) ob_out[j] = ob[j];
  } else {
    store_obs<KIND>(io.obs, me, ob);
  }
  io.reward[me] = reward;
  io.done[me] = (uint8_t)done;
  if (io.events) io.events[me] = (uint8_t)events;
}

// CTAs per SM the register budget of step_kernel is held to.  SwingRacket's instantiation holds the straight-line control
// substep only (everything else is deferred to ff_kernel), Tennisbot's hit_fast plus the generic physics_step out of line.
template <typename T, int KIND> struct StepMinBlocks { static constexpr int v = KIND == TB_ENV_SWING ? 5 : 3; };
template <int KIND> struct StepMinBlocks<double, KIND> { static constexpr int v = KIND == TB_ENV_SWING ? 4 : 3; };

// The counter set of the step with index e (= epoch[0] when its step_kernel starts): sets alternate, and every step_kernel
// zeroes the set of the step after it.  Indices run 0 .. kEpochLast - 1 and wrap (an even period, so the sets keep
// alternating); tags are index + 1, so no tag is 0, the value of a slot that was never written.
constexpr unsigned kEpochLast = 0xfffffffeu;
__device__ __forceinline__ unsigned long long *ctr_set(const StepIO &io, unsigned e) { return io.queue_ctrs + (size_t)(e & 1u) * kCtrWords; }

// Programmatic dependent launch (sm_90+): a kernel launched with the stream-serialisation attribute may be staged on the
// device while its predecessor drains; it must not touch the predecessor's results before pdl_wait(), which returns once
// that grid has completed and flushed.  Without the attribute both are no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Everything an env step does once the state and the action of the warp's 32 envs sit in registers: the substep the
// action drives, env logic, statistics, outputs, auto-reset, queueing for ff_kernel, state back to HBM.
// DEFER (step_kernel, SwingRacket): envs that ff_classify_state() puts in kFfFree take the straight-line ctl_fast; every
// other env is left untouched and appended to queue_ctl, for ff_kernel's prologue to run this same function on it
// with DEFER off - gathered into dense warps there, and with the generic path's registers and rare code kept out of
// step_kernel.  me: the lane's env (tile0 + lane in step_kernel; tile0 is only used by the STAGE row tiles).
template <typename T, int KIND, bool STAGE, bool DEFER>
__device__ __forceinline__ void step_tile(const Scene<T> &sc, const StepIO &io, unsigned long long *qctr, int64_t tile0, int64_t me, int rows,
                                          bool valid, St<T> &s, const float *a, WarpStats &ws, int *s_cnt, unsigned long long *s_base,
                                          float *s_tile, bool have5) {
  constexpr int OD = Dims<KIND>::obs;
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  T *base = static_cast<T *>(io.state);
  StepCtl c = {0, 0, 0, 0.0f, false};
  bool fin = false;
  const T spin1 = s.bw[1], spin2 = s.bw[2];
  const uint32_t episode0 = s.episode;
  if (DEFER) {
    bool defer = false;
    if (valid) {
      defer = io.pid != nullptr || (s.flags & kFlagDone) || ff_classify_state(sc, s) != kFfFree;
      if (!defer) {
        c.events = ctl_fast<T>(sc, s, a);
        fin = !(++s.step > 25);  // swingracket_env.py:85-86; no contact, hence no reward in this substep
      }
    }
    unsigned dm = __ballot_sync(full, defer);
    if (TB_UNLIKELY(dm)) {
      unsigned long long at = 0;
      if (lane == 0) at = atomicAdd(qctr + kCCtl, (unsigned long long)__popc(dm));
      at = __shfl_sync(full, at, 0);
      if (defer) io.queue_ctl[at + __popc(dm & ((1u << lane) - 1u))] = (int)me;
    }
    valid = valid && !defer;
  } else if (valid) {
    c.done = s.flags & kFlagDone;
    if (TB_UNLIKELY(io.pid != nullptr)) {
      T pid[8];
      load_pid(static_cast<const T *>(io.pid), io.n, me, pid);
      fin = env_substep<T, KIND>(sc, s, a, c, pid);
      if (fin && c.done && io.auto_reset) {  // reset() builds a new Racket, hence fresh controllers
#pragma unroll
        for (int j = 0; j < 8; ++j) pid[j] = 0;
      }
      store_pid(static_cast<T *>(io.pid), io.n, me, pid);
    } else {
      fin = env_substep<T, KIND>(sc, s, a, c);
    }
    if (fin) s.ret += (T)c.reward;
  }
  unsigned act_mask = __ballot_sync(full, valid);
  if (lane == 0) ws.acc[TB_STAT_PHYSICS_STEPS] += __popc(act_mask);
  account<T>(ws, fin, c.done, c.hit, c.events, s.step, s.ret);
  // every env of the warp's tile completed its step (always, except in a launch that feeds the fast-forward): the
  // rows go out through the tile; otherwise finished envs store their own row and ff_kernel writes the others later
  const bool whole_tile = STAGE && __all_sync(full, fin || !valid);
  if (valid && fin) finish_api<T, KIND>(sc, io, me, s, c.reward, c.done, c.events, whole_tile ? s_tile + lane * OD : nullptr);
  if (whole_tile) {
    __syncwarp();
    float *dst = io.obs + tile0 * OD;
    const int nf = rows * OD, nv = nf >> 2;
    for (int i = lane; i < nv; i += 32) reinterpret_cast<float4 *>(dst)[i] = reinterpret_cast<const float4 *>(s_tile)[i];
    for (int i = (nv << 2) + lane; i < nf; i += 32) dst[i] = s_tile[i];
  }

  // envs entering the fast-forward: queue them for ff_kernel (only SwingRacket ever does).  Longest-job-first:
  // a ball the racket has hit flies for up to 775 more substeps and is queued from the FRONT, a ball still in free
  // fall lands after ~100 and is queued from the BACK, so the long flights start first and the short ones fill
  // the tail of ff_kernel.  LAST come the free-falling balls that are moving away from the racket's plane at 0.5 m/s
  // or more: they do not meet the racket on the way down (2 in 60 000 do, against 3 % of the other free-falling ones,
  // and a visit to the servers shortly before the landing is what the launch would end up waiting for).  An env whose
  // first fast-forward substep needs the full treatment (ball within reach of the racket, mostly: a hit in progress)
  // goes to the full queue, which ff_kernel serves before anything else.
  constexpr int kNone = 4;
  bool queued = valid && !fin;
  int cls = kNone;
  if (KIND == TB_ENV_SWING && queued) {
    // front of the queue as well: a ball that is closing in on the racket's plane and would cross it within ~0.6 s.
    // If the racket is there when it does, the flight that follows is a long one, and it should not start last.
    const T x = s.rq[0], y = s.rq[1], z = s.rq[2], w = s.rq[3];
    const T nx = 1 - 2 * (y * y + z * z), ny = 2 * (x * y + z * w), nz = 2 * (x * z - y * w);
    const T d = nx * (s.bp[0] - s.rp[0]) + ny * (s.bp[1] - s.rp[1]) + nz * (s.bp[2] - s.rp[2]);
    const T vn = nx * (s.bv[0] - s.rv[0]) + ny * (s.bv[1] - s.rv[1]) + nz * (s.bv[2] - s.rv[2]);
    const bool closing = d * vn < 0 && M<T>::abs(d) < (T)0.6 * M<T>::abs(vn);
    cls = ff_classify_state(sc, s) == kFfFull ? 2 : ((dot3(s.bv, s.bv) > (T)9 || closing) ? 0 : (d * vn > 0 && M<T>::abs(vn) >= (T)0.5) ? 3 : 1);
    s.flags = (s.flags & ~((0xff << kFlagEventShift) | kStPristine)) | kFlagInFlight | kFlagFirst | (c.events << kFlagEventShift);
  }
  // the state goes back first: the bookkeeping below synchronises the CTA, and on 25 steps out of 26 it has nothing to do
  if (valid) {
    const bool restarted = s.episode != episode0;
    store_state_changed(base, io.n, me, s, restarted || s.bw[1] != spin1 || s.bw[2] != spin2, restarted, have5 || restarted);
  }
  if (KIND == TB_ENV_SWING) {
    constexpr int W = kBlock / 32;
    if (!__syncthreads_or(cls != kNone)) return;  // (every thread of the CTA gets here: DEFER lanes and tail lanes included)
    unsigned m0 = __ballot_sync(full, cls == 0), m1 = __ballot_sync(full, cls == 1), m2 = __ballot_sync(full, cls == 2),
             m3 = __ballot_sync(full, cls == 3);
    if (lane == 0) { s_cnt[wib] = __popc(m0); s_cnt[W + wib] = __popc(m1); s_cnt[2 * W + wib] = __popc(m2); s_cnt[3 * W + wib] = __popc(m3); }
    __syncthreads();
    if (threadIdx.x < 4) {
      int k = threadIdx.x, tot = 0;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        int a = s_cnt[k * W + w];
        s_cnt[k * W + w] = tot;
        tot += a;
      }
      unsigned long long *ctr = qctr + (k == 0 ? kCFront : k == 1 ? kCBack : k == 2 ? kCFull0 : kCSafe);
      s_base[k] = tot ? atomicAdd(ctr, (unsigned long long)tot) : 0ULL;
    }
    __syncthreads();
    if (queued) {
      // queue: front entries from [0] up, back entries from [n - 1] down; queue_full: full entries from [0] up, the
      // last-to-start entries from [n - 1] down (an env is in one list only, so neither pair can meet)
      const unsigned lt = (1u << lane) - 1u;
      if (cls == 0) io.queue[s_base[0] + s_cnt[wib] + __popc(m0 & lt)] = (int)me;
      else if (cls == 1) io.queue[io.n - 1 - (int64_t)(s_base[1] + s_cnt[W + wib] + __popc(m1 & lt))] = (int)me;
      else if (cls == 2) io.queue_full[s_base[2] + s_cnt[2 * W + wib] + __popc(m2 & lt)] = (int)me;
      else io.queue_full[io.n - 1 - (int64_t)(s_base[3] + s_cnt[3 * W + wib] + __popc(m3 & lt))] = (int)me;
    }
  }
}


// STAGE: move the action / observation rows through warp-private shared-memory tiles (see below); chosen by the host
// when the caller's buffers are pinned host memory, off for buffers in HBM where it only costs registers.
// MINB: CTAs per SM the registers are capped for, 0 = StepMinBlocks (the fastest build for grids of many waves).  The host
// picks MINB = 4 (128 registers, some spills) for Tennisbot-v0 grids that fit the SMs in ONE wave at 4 CTAs per SM but
// not at the default 3 - 65 536 envs = 512 CTAs on 148 SMs is such a size: no second, nearly empty wave.
template <typename T, int KIND, bool STAGE, int MINB = 0>
__global__ void __launch_bounds__(kBlock, MINB ? MINB : StepMinBlocks<T, KIND>::v) step_kernel(const __grid_constant__ Scene<T> sc, const __grid_constant__ StepIO io) {
  __shared__ unsigned long long sacc[kBlock / 32][TB_NUM_STATS];
  __shared__ int s_cnt[4 * (kBlock / 32)];
  __shared__ unsigned long long s_base[4];
  // Each warp's 32 action rows come in and its 32 observation rows go out as one contiguous tile through shared
  // memory (warp-private, __syncwarp only): [N, act] / [N, obs] float32 rows are 24 / 8 / 48 bytes, which per-thread
  // accesses would turn into strided partial sectors - harmless in HBM behind L2, costly when the caller's buffers
  // are pinned host memory and every sector is a PCIe transaction (tb_step_host's zero-copy path).
  constexpr int AD = Dims<KIND>::act, OD = Dims<KIND>::obs;
  __shared__ __align__(16) float s_tiles[STAGE ? kBlock / 32 : 1][STAGE ? 32 * OD : 4];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  float *s_tile = s_tiles[STAGE ? wib : 0];
  pdl_wait();  // (programmatic dependent launch: this grid may be staged while the previous kernel of the stream drains)
  WarpStats ws;
  ws.init(sacc[wib], lane);
  const unsigned e = io.epoch[0];  // index of this step; constant while this grid runs (ff_kernel advances it)
  unsigned long long *qctr = ctr_set(io, e);
  if (blockIdx.x == 0) {
    unsigned long long *next = ctr_set(io, e + 1u);
    for (int i = threadIdx.x; i < kCtrWords; i += kBlock) next[i] = 0;
    if (threadIdx.x == 0) io.epoch[1] = e + 1u;  // the tag of this step's queue slots, never 0
    // (policy_kernel reads [2] after its pdl_wait, i.e. after this grid has finished; nothing in this grid reads it)
    if (KIND == TB_ENV_HIT && threadIdx.x == 0) io.epoch[2] += 1u;
  }

  const int64_t tile0 = (int64_t)blockIdx.x * kBlock + wib * 32, me = tile0 + lane;
  const bool valid = me < io.n;
  const int rows = io.n - tile0 >= 32 ? 32 : (io.n > tile0 ? (int)(io.n - tile0) : 0);
  St<T> s;
  float a[8];
  if (STAGE) {
    const float *src = io.actions + tile0 * AD;
    const int nf = rows * AD, nv = nf >> 2;
    for (int i = lane; i < nv; i += 32) reinterpret_cast<float4 *>(s_tile)[i] = reinterpret_cast<const float4 *>(src)[i];
    for (int i = (nv << 2) + lane; i < nf; i += 32) s_tile[i] = src[i];
    __syncwarp();
#pragma unroll
    for (int j = 0; j < AD; ++j) a[j] = valid ? s_tile[lane * AD + j] : 0.0f;
    __syncwarp();
  }
  // One thread pulls the tile that the CTA one wave ahead will work on into L2 (bulk prefetches: eight pack chunks of
  // 128 envs + their action rows), so that CTA's loads are L2 hits.  With 168-register threads only 12 warps fit an SM
  // and every CTA loads once at the start of its life; the prefetch keeps HBM requests in flight during the
  // arithmetic.  (A persistent variant that staged whole tiles in shared memory through cp.async.bulk + mbarrier was
  // 15 % faster in float32 but slower in float64: two 35 KB stages x 3 CTAs leave almost no L1 for the rare paths'
  // local-memory records.  Measured on B200, see DESIGN.md.)
  if (!STAGE && threadIdx.x == 0 && io.prefetch_ahead > 0) {
    const int64_t e0 = ((int64_t)blockIdx.x + io.prefetch_ahead) * kBlock;
    if (e0 + kBlock <= io.n) {
      const T *b0 = static_cast<const T *>(io.state);
#pragma unroll
      for (int p = 0; p < kPacks; ++p)
        if (p != 5 && p != 6)  // (the two packs load_state_ctl usually skips)
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(b0 + ((int64_t)p * io.n + e0) * 4), "r"((uint32_t)(kBlock * 4 * sizeof(T))) : "memory");
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(io.actions + e0 * AD), "r"((uint32_t)(kBlock * AD * 4)) : "memory");
    }
  }
  bool have5 = true;
  if (valid) {
    have5 = load_state_ctl<T, KIND>(sc, static_cast<const T *>(io.state), io.n, me, io.seed, (uint64_t)(io.id_offset + me), s);
    if (!STAGE) load_action<KIND>(io.actions, me, a);
  }
  step_tile<T, KIND, STAGE, KIND == TB_ENV_SWING>(sc, io, qctr, tile0, me, rows, valid, s, a, ws, s_cnt, s_base, s_tile, have5);
  ws.flush(io.stats);
  pdl_trigger();
}

// Fast-forward continuation (SwingRacket only): one persistent launch (a CTA per resident slot) whose warps have roles.
// Nothing in it waits for a particular other CTA: all work is claimed from counters and queues, so any subset of the CTAs
// completes the launch (another stream may hold SMs).
//
//   prologue      the control substeps step_kernel deferred (ball within reach of something), 32 list entries per warp.
//   flight warps  every LANE is a small state machine: claim an env, keep its flight state in registers and take ff_fast
//                 substeps (a straight line, the court landing included) until the flight ends or a substep needs the full
//                 treatment; then hand the env on through HBM (landed mark, or the dynamic full queue) and claim the next
//                 one - from step_kernel's lists (balls the racket has hit or is about to first, plain free fall next, the
//                 free-falling balls that move away from the racket last) and from the late queue (flights that go on after a
//                 visit to the servers).  Leaving / claiming is done for several lanes of a warp at once.  A lane in an
//                 800-substep flight delays nobody, and no rare code ever enters these warps' instruction stream.
//   server warps  (all warps of every io.server_sm_stride-th SM; one warp in kServerStride CTAs when the grid does not fill the
//                 device) poll the full queues: ff_contact_lean / ff_full (narrow phase, contact solve, time-out) for one env
//                 per lane until ff_fast applies again; the env then goes to the late queue, or is marked landed.  Contact
//                 chains (a ball rolling on the racket face takes dozens of full substeps) therefore run concurrently with
//                 the bulk of the flights, and the long flight that follows a late hit starts at once.
//   finishing     reward, statistics, outputs, auto-reset for every env that has landed, coalesced like step_kernel: done by
//                 whichever flight warps have nothing to integrate, tile by tile, overlapping the tail of the flights.
//
// History (measured on B200, 1 Mi envs, f64): everything in one loop per lane 6.8 ms (every landing / claim /
// contact stalled 31 other lanes and streamed ~40 KB of rare code through the instruction caches of the substep
// loop); the same work in barrier-separated phases 4.6 - 5.0 ms (every round of "contact, then fly on" paid the latency
// of its longest chain and longest flight); roles: see profiles/.
constexpr int kServeMin = 6, kServeWait = 12, kServerStride = 2;
constexpr int kIdle = 4, kWait = 5, kRetired = 6;  // lane states 0..3 = kFfFree, kFfLand (running), kFfFull, kFfDone (leaving);
                                                   // no env; no env, holds a late-queue ticket; no env, never will
constexpr int kFfMaxVisits = 3;  // an env that comes to the servers this often finishes its flight there
__device__ __forceinline__ unsigned long long ld_ctr(const unsigned long long *p) { return *reinterpret_cast<const volatile unsigned long long *>(p); }
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// Has every flight of this launch landed?  total0 = entries of step_kernel's three lists; the prologue adds the flights
// of the deferred envs it steps (kCDynTotal) and counts the entries it is through with (kCCtlDone) after publishing them,
// so once kCCtlDone has reached nctl the sum is final.
__device__ __forceinline__ bool ff_all_landed(const unsigned long long *ctr, long long nctl, long long total0) {
  if (ld_ctr(ctr + kCCtlDone) < (unsigned long long)nctl) return false;
  if (ld_ctr(ctr + kCLanded) < (unsigned long long)total0 + ld_ctr(ctr + kCDynTotal)) return false;
  __threadfence();  // (kCDynTotal is final once kCCtlDone has reached nctl: read it again behind the fence)
  return ld_ctr(ctr + kCLanded) >= (unsigned long long)total0 + ld_ctr(ctr + kCDynTotal);
}
// a wait gave up: mark the launch (every role leaves when it sees the mark) and the context
__device__ __forceinline__ void ff_give_up(const StepIO &io, unsigned long long *ctr, unsigned long long code) {
  atomicExch(ctr + kCError, code);
  atomicExch(io.fault, code);
  *io.fault_host = code;
  __threadfence_system();
}

// warp-aggregated reservation of slots in a dynamic queue + tagged publication of `me` (for lanes with pred).  The
// env's state must have been stored before the call.
__device__ __forceinline__ void dq_push(unsigned long long *q, long long cap, unsigned long long *tail, unsigned epoch, bool pred,
                                        int me, int lane, unsigned long long *err) {
  const unsigned full = 0xffffffffu;
  unsigned m = __ballot_sync(full, pred);
  if (!m) return;
  int leader = __ffs(m) - 1;
  unsigned long long at = 0;
  if (lane == leader) at = atomicAdd(tail, (unsigned long long)__popc(m));
  at = __shfl_sync(full, at, leader);
  if (pred) {
    unsigned long long idx = at + __popc(m & ((1u << lane) - 1u));
    if ((long long)idx < cap) {
      __threadfence();  // state before publication
      *reinterpret_cast<volatile unsigned long long *>(q + idx) = ((unsigned long long)epoch << 32) | (unsigned)me;
    } else {
      atomicExch(err, 2ULL);  // cannot happen: every env is pushed at most kFfMaxVisits times
    }
  }
}
// Consumers take TICKETS: one atomicAdd per warp reserves the next slots of a queue, filled or not, and every lane then
// polls its own slot (its own address: no contention) until a producer's tagged store lands there - entries and
// waiting lanes are matched first come, first served.  (Claiming only what is already there needs a compare-and-swap
// loop on the head, which collapses when a thousand warps go for the same late entries: measured 3 entries / us.)
__device__ __forceinline__ long long dq_reserve(unsigned long long *head, unsigned idle_mask, int lane) {
  long long at = 0;
  if (lane == 0) at = (long long)atomicAdd(head, (unsigned long long)__popc(idle_mask));
  at = __shfl_sync(0xffffffffu, at, 0);
  return at + __popc(idle_mask & ((1u << lane) - 1u));
}
// the env index in slot `ticket` if its producer has published it (state visible to the caller afterwards), else -1
__device__ __forceinline__ int dq_poll(const unsigned long long *q, long long ticket, unsigned epoch) {
  unsigned long long v = *reinterpret_cast<const volatile unsigned long long *>(q + ticket);
  if ((unsigned)(v >> 32) != epoch) return -1;
  __threadfence();
  return (int)(unsigned)v;
}

// state loads that bypass L1: another SM may have rewritten the env since this SM last saw it (same launch)
__device__ __forceinline__ Pack<float> ldcg_pack(const float *base, int64_t n, int p, int64_t i) {
  float4 v = __ldcg(reinterpret_cast<const float4 *>(base + ((int64_t)p * n + i) * 4));
  return {v.x, v.y, v.z, v.w};
}
__device__ __forceinline__ Pack<double> ldcg_pack(const double *base, int64_t n, int p, int64_t i) {
  const double2 *q = reinterpret_cast<const double2 *>(base + ((int64_t)p * n + i) * 4);
  double2 a = __ldcg(q), b = __ldcg(q + 1);
  return {a.x, a.y, b.x, b.y};
}
// an env's flight state HBM -> lane (omega to the body frame); returns the flags word
template <typename T> __device__ __forceinline__ int ff_load(const T *base, int64_t n, int64_t me, FfLane<T> &L) {
  Pack<T> p0 = ldcg_pack(base, n, 0, me), p1 = ldcg_pack(base, n, 1, me), p2 = ldcg_pack(base, n, 2, me), p3 = ldcg_pack(base, n, 3, me),
          p4 = ldcg_pack(base, n, 4, me), p5 = ldcg_pack(base, n, 5, me), p6 = ldcg_pack(base, n, 6, me), p7 = ldcg_pack(base, n, 7, me);
  St<T> s;
  s.rq[0] = p1.x; s.rq[1] = p1.y; s.rq[2] = p1.z; s.rq[3] = p1.w;
  s.rw[0] = p3.x; s.rw[1] = p3.y; s.rw[2] = p3.z;
  ff_enter(s);
  L.rp[0] = p0.x; L.rp[1] = p0.y; L.rp[2] = p0.z; L.bp[0] = p0.w;
  L.rq[0] = p1.x; L.rq[1] = p1.y; L.rq[2] = p1.z; L.rq[3] = p1.w;
  L.rv[0] = p2.x; L.rv[1] = p2.y; L.rv[2] = p2.z; L.bp[1] = p2.w;
  L.wl[0] = s.rw[0]; L.wl[1] = s.rw[1]; L.wl[2] = s.rw[2]; L.bp[2] = p3.w;
  L.bv[0] = p4.x; L.bv[1] = p4.y; L.bv[2] = p4.z; L.bw[0] = p4.w;
  L.bw[1] = p5.x; L.bw[2] = p5.y;
  L.sb = norm3(L.bw);
  L.tgt[0] = p5.z; L.tgt[1] = p5.w; L.tgt[2] = p6.x + 4;  // swingracket_env.py:135-141
  L.goal[0] = p6.y; L.goal[1] = p6.z;
  L.step = (int)as_int(p7.y);
  int flags = (int)as_int(p7.z);
  L.events = (flags >> kFlagEventShift) & 0xff;
  return flags;
}
// lane -> HBM: the packs a flight changes (0..4, the spin half of 5) and step / flags of pack 7
template <typename T> __device__ __forceinline__ void ff_store(T *base, int64_t n, int64_t me, const FfLane<T> &L, int flags) {
  St<T> s;
  {  // ff_fast does not renormalise the quaternion per substep
    T inv = M<T>::rsqrt(L.rq[0] * L.rq[0] + L.rq[1] * L.rq[1] + L.rq[2] * L.rq[2] + L.rq[3] * L.rq[3]);
#pragma unroll
    for (int i = 0; i < 4; ++i) s.rq[i] = L.rq[i] * inv;
  }
  s.rw[0] = L.wl[0]; s.rw[1] = L.wl[1]; s.rw[2] = L.wl[2];
  ff_leave(s);
  st_pack(base, n, 0, me, Pack<T>{L.rp[0], L.rp[1], L.rp[2], L.bp[0]});
  st_pack(base, n, 1, me, Pack<T>{s.rq[0], s.rq[1], s.rq[2], s.rq[3]});
  st_pack(base, n, 2, me, Pack<T>{L.rv[0], L.rv[1], L.rv[2], L.bp[1]});
  st_pack(base, n, 3, me, Pack<T>{s.rw[0], s.rw[1], s.rw[2], L.bp[2]});
  st_pack(base, n, 4, me, Pack<T>{L.bv[0], L.bv[1], L.bv[2], L.bw[0]});
  T *p5 = base + ((int64_t)5 * n + me) * 4, *p7 = base + ((int64_t)7 * n + me) * 4;
  p5[0] = L.bw[1]; p5[1] = L.bw[2];
  p7[1] = int_as(T(), L.step); p7[2] = int_as(T(), flags);
}
// The landed mark of an env whose state ff_store has written, after a fence: the finishing pass may look at the env at any time
// and takes the mark as "the state is complete".
template <typename T> __device__ __forceinline__ void ff_mark_landed(T *base, int64_t n, int64_t me, int flags) {
  base[((int64_t)7 * n + me) * 4 + 2] = int_as(T(), flags | kFlagLanded);
}

// The finishing pass for 32 envs (a tile of consecutive envs in pass 1, entries of the retry list in pass 2): complete the
// env step of those whose flight has landed - reward (swingracket_env.py:111-126, from the contact bits of the final
// substep), statistics, terminal observation, outputs, auto-reset - coalesced like step_kernel.  Warps run it whenever
// they have no flight to integrate, so it overlaps the tail of the launch instead of following it.  Pass 1 visits every
// tile once and lists the envs that were still in flight (collect); pass 2, after the last landing, visits exactly those.
template <typename T>
__device__ __noinline__ void ff_finish_dense(const Scene<T> &sc, const StepIO &io, unsigned long long *ctr, int64_t me, bool valid, bool collect,
                                             WarpStats *wsp) {
  constexpr int KIND = TB_ENV_SWING;
  const unsigned full = 0xffffffffu;
  T *base = static_cast<T *>(io.state);
  bool fin = false, retry = false;
  St<T> s;
  s.step = 0; s.ret = 0;
  int events = 0;
  float reward = 0.0f;
  if (valid) {
    Pack<T> p7 = ldcg_pack(base, io.n, 7, me);
    int flags = (int)as_int(p7.z);
    // pass 2 runs once every landing has been counted; a mark may still be on its way (it is written next to the count)
    for (int spin = 0; !collect && !(flags & kFlagLanded) && spin < (1 << 20); ++spin) {
      p7 = ldcg_pack(base, io.n, 7, me);
      flags = (int)as_int(p7.z);
    }
    if (flags & kFlagLanded) {
      fin = true;
      __threadfence();  // the mark was written after the state (ff_store)
      Pack<T> p0 = ldcg_pack(base, io.n, 0, me), p1 = ldcg_pack(base, io.n, 1, me), p2 = ldcg_pack(base, io.n, 2, me),
              p3 = ldcg_pack(base, io.n, 3, me), p4 = ldcg_pack(base, io.n, 4, me), p5 = ldcg_pack(base, io.n, 5, me),
              p6 = ldcg_pack(base, io.n, 6, me);
      s.rp[0] = p0.x; s.rp[1] = p0.y; s.rp[2] = p0.z; s.bp[0] = p0.w;
      s.rq[0] = p1.x; s.rq[1] = p1.y; s.rq[2] = p1.z; s.rq[3] = p1.w;
      s.rv[0] = p2.x; s.rv[1] = p2.y; s.rv[2] = p2.z; s.bp[1] = p2.w;
      s.rw[0] = p3.x; s.rw[1] = p3.y; s.rw[2] = p3.z; s.bp[2] = p3.w;
      s.bv[0] = p4.x; s.bv[1] = p4.y; s.bv[2] = p4.z; s.bw[0] = p4.w;
      s.bw[1] = p5.x; s.bw[2] = p5.y; s.aux[0] = p5.z; s.aux[1] = p5.w;
      s.aux[2] = p6.x; s.goal[0] = p6.y; s.goal[1] = p6.z; s.d0 = p6.w;
      s.step = (int)as_int(p7.y);
      s.episode = (uint32_t)as_int(p7.w);
      events = (flags >> kFlagEventShift) & 0xff;
      reward = ff_reward(s, (flags >> kFlagLastShift) & 0xff);
      s.ret = p7.x + (T)reward;
      s.flags = flags & kFlagDone;  // drop every in-flight mark
    } else {
      retry = (flags & kFlagInFlight) != 0;
    }
  }
  account<T>(*wsp, fin, true, 0, events, s.step, s.ret);
  if (fin) {
    finish_api<T, KIND>(sc, io, me, s, reward, true, events);
    store_state(base, io.n, me, s);
    if (io.pid && io.auto_reset) {
      T z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      store_pid(static_cast<T *>(io.pid), io.n, me, z);
    }
  }
  if (collect) {
    const unsigned rm = __ballot_sync(full, retry);
    if (rm) {
      unsigned long long at = 0;
      if (wsp->lane == 0) at = atomicAdd(ctr + kCRetryTail, (unsigned long long)__popc(rm));
      at = __shfl_sync(full, at, 0);
      if (retry) io.queue_ctl[at + __popc(rm & ((1u << wsp->lane) - 1u))] = (int)me;
    }
  }
}

// What a warp does when it has no flight to integrate: a piece of the finishing pass.  Returns 0 = nothing to do right
// now (the caller backs off), 1 = did some, 2 = the launch is complete (every env finished): leave.
template <typename T>
__device__ __forceinline__ int ff_finishing_duty(const Scene<T> &sc, const StepIO &io, unsigned long long *ctr, long long nctl, long long total0,
                                                 WarpStats &ws, bool &pass1_over) {
  const unsigned full = 0xffffffffu;
  const int lane = ws.lane;
  const long long ntiles = (io.n + 31) >> 5;
  if (!pass1_over) {
    // (the retry list lives in queue_ctl: not before the prologue has read all of it)
    if (ld_ctr(ctr + kCCtlDone) < (unsigned long long)nctl) return 0;
    // a launch that only had deferred control substeps to take (no flight was queued): nothing to finish
    if (total0 == 0 && ld_ctr(ctr + kCDynTotal) == 0) return 2;
    long long t = 0;
    if (lane == 0) t = (long long)atomicAdd(ctr + kCFinClaim, 1ULL);
    t = __shfl_sync(full, t, 0);
    if (t < ntiles) {
      const int64_t me = (t << 5) + lane;
      ff_finish_dense<T>(sc, io, ctr, me, me < io.n, true, &ws);
      __threadfence();  // retry entries before the count
      __syncwarp();
      if (lane == 0) atomicAdd(ctr + kCFinDone, 1ULL);
      return 1;
    }
    pass1_over = true;
  }
  if (!ff_all_landed(ctr, nctl, total0) || ld_ctr(ctr + kCFinDone) < (unsigned long long)ntiles) return 0;
  __threadfence();
  const long long nretry = (long long)ld_ctr(ctr + kCRetryTail);
  for (;;) {
    long long at = 0;
    if (lane == 0) at = (long long)atomicAdd(ctr + kCRetryClaim, 32ULL);
    at = __shfl_sync(full, at, 0);
    if (at >= nretry) break;
    const bool valid = at + lane < nretry;
    const int64_t me = valid ? (int64_t)__ldcg(io.queue_ctl + at + lane) : 0;
    ff_finish_dense<T>(sc, io, ctr, me, valid, false, &ws);
  }
  return 2;
}

// A flight warp.  n0 / qfront / qmid: step_kernel's lists in the order they are claimed (front: [0, qfront), back: [qfront, qmid),
// last-to-start: [qmid, n0)); nctl, total0: see ff_all_landed.
template <typename T>
__device__ __forceinline__ void ff_flight_warp(const Scene<T> &sc, const StepIO &io, unsigned epoch, long long n0, long long qfront, long long qmid,
                                               long long nctl, long long total0, WarpStats &ws, int &nsub) {
  const unsigned full = 0xffffffffu;
  const int lane = ws.lane;
  T *base = static_cast<T *>(io.state);
  unsigned long long *ctr = ctr_set(io, epoch - 1u);
  FfLane<T> L;
  {  // defined values for lanes that never get an env (ff_fast is never run on them)
    T *z = reinterpret_cast<T *>(&L);
#pragma unroll
    for (int i = 0; i < (int)(offsetof(FfLane<T>, step) / sizeof(T)); ++i) z[i] = 0;
    L.step = 0; L.events = 0;
  }
  int me = 0, st = kIdle, waited = 0, step0 = 0, visits = 0;
  long long ticket = 0;
  unsigned serves = 0;
  bool exhausted0 = n0 == 0, first = false, first_pending = false, pass1_over = false;
  long long idle_since = 0;
  unsigned nap = 0;  // idle back-off: thousands of warps polling one cache line would starve the servers' atomics on it
  for (;;) {
    // ---- substeps until enough lanes want to leave / claim (no call, no rare code in this loop)
    unsigned run_m, leave_m;
#pragma unroll 1
    for (;;) {
      if (st <= kFfLand) st = ff_fast<T>(sc, L, st);
      if (TB_UNLIKELY(first_pending)) {  // warp-uniform: some lanes just took a flight's first substep, see below
        if (first) {
          const T *p5 = base + ((int64_t)5 * io.n + me) * 4, *p6 = base + ((int64_t)6 * io.n + me) * 4;
          L.tgt[0] = __ldcg(p5 + 2); L.tgt[1] = __ldcg(p5 + 3); L.tgt[2] = __ldcg(p6) + 4;
          first = false;
        }
        first_pending = false;
      }
      run_m = __ballot_sync(full, st <= kFfLand);
      leave_m = __ballot_sync(full, st == kFfFull || st == kFfDone);
      // lanes that wait: the leaving ones, and the idle ones while step_kernel's queue still has entries; idle lanes
      // look at the late queue every kServeWait iterations
      unsigned wait_m = exhausted0 ? leave_m : ~run_m;
      waited = (wait_m | ~run_m) ? waited + 1 : 0;
      if (!run_m || __popc(wait_m) >= kServeMin || waited >= kServeWait) break;
    }
    waited = 0;
    // ---- lanes whose flight left ff_fast: state back to HBM; landed mark (ff_fast ends on the court's top face only), or
    //      the servers' queue
    if (leave_m) {
      const bool to_full = st == kFfFull, landed = st == kFfDone;
      int flags = 0;
      if (to_full || landed) {
        nsub += L.step - step0;
        flags = kFlagInFlight | (L.events << kFlagEventShift) | (visits << kFlagVisitShift);
        if (landed) flags |= TB_EV_COURT_BALL << kFlagLastShift;
        ff_store(base, io.n, (int64_t)me, L, flags);
      }
      dq_push(io.dq_full, io.dq_cap, ctr + kCFullTail, epoch, to_full, me, lane, ctr + kCError);
      unsigned done_m = __ballot_sync(full, landed);
      if (done_m) {
        __threadfence();  // landed states before the marks and the count
        if (landed) ff_mark_landed(base, io.n, (int64_t)me, flags);
        if (lane == 0) atomicAdd(ctr + kCLanded, (unsigned long long)__popc(done_m));
      }
      if (to_full || landed) st = kIdle;
    }
    // ---- lanes without an env: the next entries of step_kernel's queue (one atomic per warp); once that is empty, a
    //      ticket each for the late queue, polled here every time round
    bool got = false;
    if (st == kWait) {
      int e = dq_poll(io.dq_late, ticket, epoch);
      if (e >= 0) { me = e; got = true; }
    }
    unsigned idle = __ballot_sync(full, st == kIdle);
    if (idle) {
      const int rank = __popc(idle & ((1u << lane) - 1u));
      // late entries first (a flight that goes on after a racket contact is likely a long one): as many tickets as
      // entries wait right now, looked up every fourth time while step_kernel's queue lasts; everything after that
      int nlate = 32;
      if (!exhausted0) {
        nlate = 0;
        if ((serves++ & 3u) == 0) {
          if (lane == 0) {
            long long avail = (long long)(ld_ctr(ctr + kCLateTail) - ld_ctr(ctr + kCLateHead));
            nlate = avail < 0 ? 0 : avail > 32 ? 32 : (int)avail;
          }
          nlate = __shfl_sync(full, nlate, 0);
        }
      }
      const bool pick_late = st == kIdle && rank < nlate;
      const unsigned late_m = __ballot_sync(full, pick_late), init_m = idle & ~late_m;
      if (late_m) {
        long long t = dq_reserve(ctr + kCLateHead, late_m, lane);
        if (pick_late) {
          ticket = t;
          st = t < io.dq_cap ? kWait : kRetired;  // (more tickets than slots: only possible long after the last entry)
        }
      }
      if (init_m && !exhausted0) {
        const int want = __popc(init_m);
        long long at = 0;
        if (lane == 0) at = (long long)atomicAdd(ctr + kCClaim0, (unsigned long long)want);
        at = __shfl_sync(full, at, 0);
        if (at + want >= n0) exhausted0 = true;
        long long idx = at + __popc(init_m & ((1u << lane) - 1u));
        if (st == kIdle && idx < n0) {
          me = __ldcg(idx < qfront ? io.queue + idx : idx < qmid ? io.queue + (io.n - 1 - (idx - qfront)) : io.queue_full + (io.n - 1 - (idx - qmid)));
          got = true;
        }
      }
    }
    bool to_full = false;
    if (got) {
      int flags = ff_load(base, io.n, (int64_t)me, L);
      visits = (flags >> kFlagVisitShift) & 3;
      step0 = L.step;
      st = ff_classify(sc, L);
      if (st == kFfFull) {  // within reach of something (rounding apart, only after set_state): untouched, to the servers
        to_full = true;
      } else if (flags & kFlagFirst) {
        // the flight's first substep carries no force (swingracket_env.py:105-107): with the target on the racket
        // itself the force law gives exactly zero; the real target comes back after that substep (first_pending)
        L.tgt[0] = L.rp[0]; L.tgt[1] = L.rp[1]; L.tgt[2] = L.rp[2];
        first = true;
      }
    }
    dq_push(io.dq_full, io.dq_cap, ctr + kCFullTail, epoch, to_full, me, lane, ctr + kCError);
    if (to_full) st = kIdle;
    first_pending = __any_sync(full, first);
    const int got_any = __any_sync(full, got);
    // ---- nothing to run and nothing to claim: a piece of the finishing pass; when there is none, wait for the servers
    if (!run_m && !got_any) {
      if (ld_ctr(ctr + kCError) != 0) break;
      const int duty = ff_finishing_duty<T>(sc, io, ctr, nctl, total0, ws, pass1_over);
      if (duty == 2) break;
      if (duty == 1) {
        idle_since = 0;
        nap = 0;
      } else {
        long long now = clock64();
        if (!idle_since) idle_since = now;
        if (now - idle_since > io.spin_limit) { ff_give_up(io, ctr, 4ULL); break; }
        nap = nap ? min(nap * 2, 32000u) : 1000u;
        __nanosleep(nap);
      }
    } else {
      idle_since = 0;
      nap = 0;
    }
  }
}

// A server warp: every lane holds one parked env at a time and takes generic substeps with it until ff_fast applies again
// (or, for an env that keeps coming back, until its env step is over); then it hands the env on, or completes its env
// step (ff_finish), and claims the next one.  Chains differ wildly in length (one contact step ... a ball rolling on the
// racket face for the rest of its flight), so lanes are refilled one by one, not batch by batch.
template <typename T>
__device__ __noinline__ void ff_server_warp(const Scene<T> &sc, const StepIO &io, unsigned epoch, long long nfull0, long long nctl,
                                            long long total0, WarpStats *wsp, int *nsub) {
  const unsigned full = 0xffffffffu;
  const int lane = wsp->lane;
  T *base = static_cast<T *>(io.state);
  unsigned long long *ctr = ctr_set(io, epoch - 1u);
  bool exhausted0 = nfull0 == 0, busy = false, to_end = false, waiting = false;
  long long idle_since = 0, ticket = 0;
  unsigned nap = 0;
  FfLane<T> L;
  {
    T *z = reinterpret_cast<T *>(&L);
#pragma unroll
    for (int i = 0; i < (int)(offsetof(FfLane<T>, step) / sizeof(T)); ++i) z[i] = 0;
    L.step = 0; L.events = 0;
  }
  int me = 0, r = kFfDone, phase = 2, last = 0, visits = 0, step0 = 0;
  for (;;) {
    // ---- lanes without an env: step_kernel's list (envs whose first fast-forward substep is a full one), then a ticket
    //      each for the full queue.
    bool got = false;
    if (waiting) {
      int e = dq_poll(io.dq_full, ticket, epoch);
      if (e >= 0) { me = e; got = true; waiting = false; }
    }
    const unsigned held = __ballot_sync(full, busy || waiting || got);
    if (held != full) {
      const unsigned cand = ~held;
      if (!exhausted0) {
        const int want = __popc(cand);
        long long at = 0;
        if (lane == 0) at = (long long)atomicAdd(ctr + kCFullClaim0, (unsigned long long)want);
        at = __shfl_sync(full, at, 0);
        if (at + want >= nfull0) exhausted0 = true;
        long long idx = at + __popc(cand & ((1u << lane) - 1u));
        if (((cand >> lane) & 1u) && idx < nfull0) { me = __ldcg(io.queue_full + idx); got = true; }
      } else {
        long long t = dq_reserve(ctr + kCFullHead, cand, lane);
        if (((cand >> lane) & 1u) && t < io.dq_cap) { ticket = t; waiting = true; }
      }
    }
    if (got) {
      int flags = ff_load(base, io.n, (int64_t)me, L);
      phase = (flags & kFlagFirst) ? 1 : 2;
      visits = min(((flags >> kFlagVisitShift) & 3) + 1, 3);
      to_end = visits >= kFfMaxVisits;
      step0 = L.step;
      last = 0;
      // no classification here: the lane that parked the env found it within reach of something, and the substep functions
      // cope with a state that is just outside after the trip through HBM (3 % of a server iteration)
      L.nb = dot3(L.bv, L.bv); L.nr = dot3(L.rv, L.rv); L.nw = dot3(L.wl, L.wl);
      r = kFfFull;
      busy = true;
    }
    if (!__any_sync(full, busy)) {  // nothing to do: done when every flight has landed
      if (ff_all_landed(ctr, nctl, total0) || ld_ctr(ctr + kCError) != 0) break;
      long long now = clock64();
      if (!idle_since) idle_since = now;
      if (now - idle_since > io.spin_limit) { ff_give_up(io, ctr, 5ULL); break; }
      nap = nap ? min(nap * 2, 4000u) : 500u;
      __nanosleep(nap);
      continue;
    }
    idle_since = 0;
    nap = 0;
    // ---- one substep per busy lane
    bool leave = false;
    int lflags = 0;
    if (busy) {
      if (r == kFfFull) {
        int rl = ff_contact_lean<T>(sc, &L, phase, &last);  // ball against a racket face, high above the court: the short cut
        if (rl < 0) rl = ff_full<T>(sc, &L, phase, &last);
        r = rl;
      } else {  // (to_end, or a rounding-level disagreement with the classification that queued the env)
        if (phase == 1) {  // the force-free first substep (see ff_flight_warp)
          const T t0 = L.tgt[0], t1 = L.tgt[1], t2 = L.tgt[2];
          L.tgt[0] = L.rp[0]; L.tgt[1] = L.rp[1]; L.tgt[2] = L.rp[2];
          r = ff_fast<T>(sc, L, r);
          L.tgt[0] = t0; L.tgt[1] = t1; L.tgt[2] = t2;
        } else {
          // an env that is finished here (to_end) takes its contact-free substeps in one go: a server iteration lasts as
          // long as the slowest generic substep among the warp's lanes
          do r = ff_fast<T>(sc, L, r); while (to_end && r <= kFfLand);
        }
        last = TB_EV_COURT_BALL;  // if this was the last one: ff_fast ends on the court's top face only
      }
      phase = 2;
      leave = r == kFfDone || (r != kFfFull && !to_end);
      if (leave) {
        *nsub += L.step - step0;
        lflags = kFlagInFlight | (L.events << kFlagEventShift) | (visits << kFlagVisitShift);
        if (r == kFfDone) lflags |= last << kFlagLastShift;
        ff_store(base, io.n, (int64_t)me, L, lflags);
        busy = false;
      }
    }
    const bool landed = leave && r == kFfDone;
    dq_push(io.dq_late, io.dq_cap, ctr + kCLateTail, epoch, leave && r != kFfDone, me, lane, ctr + kCError);
    unsigned done_m = __ballot_sync(full, landed);
    if (done_m) {
      __threadfence();  // landed states before the marks and the count
      if (landed) ff_mark_landed(base, io.n, (int64_t)me, lflags);
      if (lane == 0) atomicAdd(ctr + kCLanded, (unsigned long long)__popc(done_m));
    }
  }
}

// ff_kernel's prologue: the control-phase substeps step_kernel deferred (ball within reach of something, PID mode, ...)
// through the generic path, 32 entries of queue_ctl per warp at a time (claimed, so a CTA that becomes resident late
// finds nothing left and no CTA waits for another).  An env whose 26th step this was joins the flights through the
// dynamic queues.  Out of line: the generic step's registers and spills stay out of the flight loop.
template <typename T>
__device__ __noinline__ void ff_prologue(const Scene<T> &sc, const StepIO &io, unsigned epoch, unsigned long long *ctr, long long nctl, WarpStats *wsp) {
  constexpr int KIND = TB_ENV_SWING;
  const unsigned full = 0xffffffffu;
  const int lane = wsp->lane;
  T *base = static_cast<T *>(io.state);
  for (;;) {
    long long at = 0;
    if (lane == 0) at = (long long)atomicAdd(ctr + kCCtlClaim, 32ULL);
    at = __shfl_sync(full, at, 0);
    if (at >= nctl) break;
    const bool valid = at + lane < nctl;
    const int me = valid ? __ldcg(io.queue_ctl + at + lane) : 0;
    St<T> s;
    s.step = 0; s.ret = 0;
    StepCtl c = {0, 0, 0, 0.0f, false, 0};
    bool fin = false;
    T spin1 = 0, spin2 = 0;
    uint32_t episode0 = 0;
    if (valid) {
      float a[8];
      load_state(static_cast<const T *>(io.state), io.n, (int64_t)me, s);
      materialise_ball(sc, s);
      s.flags &= ~kStPristine;  // (the generic step may touch the ball: pack 4 goes back to HBM from here on)
      load_action<KIND>(io.actions, (int64_t)me, a);
      spin1 = s.bw[1]; spin2 = s.bw[2]; episode0 = s.episode;
      c.done = s.flags & kFlagDone;
      if (TB_UNLIKELY(io.pid != nullptr)) {
        T pid[8];
        load_pid(static_cast<const T *>(io.pid), io.n, (int64_t)me, pid);
        fin = env_substep<T, KIND>(sc, s, a, c, pid);
        if (fin && c.done && io.auto_reset) {  // reset() builds a new Racket, hence fresh controllers
#pragma unroll
          for (int j = 0; j < 8; ++j) pid[j] = 0;
        }
        store_pid(static_cast<T *>(io.pid), io.n, (int64_t)me, pid);
      } else {
        fin = env_substep<T, KIND>(sc, s, a, c);
      }
      if (fin) s.ret += (T)c.reward;
    }
    const unsigned valid_m = __ballot_sync(full, valid);
    if (lane == 0) wsp->acc[TB_STAT_PHYSICS_STEPS] += __popc(valid_m);
    account<T>(*wsp, fin, c.done, c.hit, c.events, s.step, s.ret);
    if (valid && fin) finish_api<T, KIND>(sc, io, (int64_t)me, s, c.reward, c.done, c.events);
    // an env that enters the fast-forward here: to the servers if its first substep is a full one, else to the flights
    const bool queued = valid && !fin;
    bool to_full = false;
    if (queued) {
      to_full = ff_classify_state(sc, s) == kFfFull;
      s.flags = (s.flags & ~((0xff << kFlagEventShift) | kStPristine)) | kFlagInFlight | kFlagFirst | (c.events << kFlagEventShift);
    }
    if (valid) {
      const bool restarted = s.episode != episode0;
      store_state_changed(base, io.n, (int64_t)me, s, restarted || s.bw[1] != spin1 || s.bw[2] != spin2, restarted);
    }
    dq_push(io.dq_full, io.dq_cap, ctr + kCFullTail, epoch, to_full, me, lane, ctr + kCError);
    dq_push(io.dq_late, io.dq_cap, ctr + kCLateTail, epoch, queued && !to_full, me, lane, ctr + kCError);
    const unsigned queued_m = __ballot_sync(full, queued);
    __threadfence();  // results and queue entries before the counts
    if (lane == 0) {
      if (queued_m) atomicAdd(ctr + kCDynTotal, (unsigned long long)__popc(queued_m));
      __threadfence();
      atomicAdd(ctr + kCCtlDone, (unsigned long long)__popc(valid_m));
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(kBlock, MinBlocks<T>::v) ff_kernel(const __grid_constant__ Scene<T> sc, const __grid_constant__ StepIO io) {
  __shared__ unsigned long long sacc[kBlock / 32][TB_NUM_STATS];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  pdl_wait();
  const unsigned epoch = io.epoch[1];  // this step's tag, written by its step_kernel; the step's index is epoch - 1
  if (blockIdx.x == 0 && threadIdx.x == 0) io.epoch[0] = epoch == kEpochLast ? 0u : epoch;  // (read by the next step_kernel only)
  unsigned long long *ctr = ctr_set(io, epoch - 1u);
  // (all four written by step_kernel, same stream)
  const long long nctl = (long long)ctr[kCCtl], qfront = (long long)ctr[kCFront], qmid = qfront + (long long)ctr[kCBack],
                  qn0 = qmid + (long long)ctr[kCSafe], nfull0 = (long long)ctr[kCFull0];
  const long long total0 = qn0 + nfull0;
  if (nctl == 0 && total0 == 0) return;
  WarpStats ws;
  ws.init(sacc[wib], lane);
  // No CTA ever waits for a particular other CTA: all work - deferred control substeps, flights, parked envs - is claimed
  // from counters and queues, so the launch completes whichever CTAs are resident when (another stream may hold SMs).
  if (nctl) ff_prologue<T>(sc, io, epoch, ctr, nctl, &ws);
  int nsub = 0;  // substeps this lane integrated
  const bool diag = blockIdx.x == 0 && threadIdx.x == 0;  // times as this CTA's first warp sees them
  unsigned long long t_mark = diag ? global_ns() : 0;
  // Roles.  The generic substep is ~3000 instructions of code and constants that no flight warp needs, and a chain of
  // dependent FP64 operations that crawls when it shares a scheduler with three flight warps that keep the FP64 pipe full.
  // A full persistent grid therefore gives whole SMs to the servers (every warp of every CTA that runs there), chosen by
  // %smid; a grid that does not fill the device keeps one server warp per kServerStride CTAs.
  bool server = wib == kBlock / 32 - 1 && blockIdx.x % kServerStride == 0;
  if (io.server_sm_stride > 0) {
    __shared__ int s_server;
    if (threadIdx.x == 0) {
      unsigned smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      int srv = smid % (unsigned)io.server_sm_stride == 0;
      // Liveness does not depend on where the CTAs land: every CTA registers, and if the last one to start finds that no CTA
      // is a server (other work kept the server SMs away from this grid), it becomes one.  As with per-CTA roles, the launch
      // completes once all of its CTAs have run, whatever the order.
      if (srv) atomicAdd(ctr + kCServers, 1ULL);
      __threadfence();
      const unsigned long long started = atomicAdd(ctr + kCStarted, 1ULL) + 1ULL;
      if (!srv && started == (unsigned long long)gridDim.x && ld_ctr(ctr + kCServers) == 0) srv = 1;
      s_server = srv;
    }
    __syncthreads();
    server = s_server != 0;
  }
  if (server) ff_server_warp<T>(sc, io, epoch, nfull0, nctl, total0, &ws, &nsub);
  else ff_flight_warp<T>(sc, io, epoch, qn0, qfront, qmid, nctl, total0, ws, nsub);
  if (diag) {
    ctr[kDPhase] = global_ns() - t_mark;
    ctr[kDRounds] = 1;
    ctr[kDFullEnvs] = ld_ctr(ctr + kCFullTail) + (unsigned long long)nfull0;
    ctr[kDFinish] = 0;
  }
  nsub = __reduce_add_sync(0xffffffffu, nsub);
  if (lane == 0) ws.acc[TB_STAT_PHYSICS_STEPS] += nsub;
  ws.flush(io.stats);
}

// In-kernel action sources of the fused rollout.  TB_ACT_RANDOM: U(-1,1) = action_space.sample().  TB_ACT_TRACK (Tennisbot-v0):
// a scripted ball tracker - a small random drive along x and a PD law on ball y - racket y, formed in float32 on the
// observation's own float32 entries - so that racket-ball contacts actually occur (SURVEY 8(d), BASELINE config 3).
template <typename T, int KIND>
__device__ __forceinline__ void rollout_action(const StepIO &io, int64_t me, const St<T> &s, float *a) {
  random_action<KIND>(io.seed, (uint64_t)(io.id_offset + me), s.episode, s.step, a);
  if (KIND == TB_ENV_HIT && io.action_mode == TB_ACT_TRACK) {
    const float ry = (float)s.rp[1], vy = (float)s.rv[1], by = (float)s.bp[1];
    const float u = 4.0f * (by - ry) - 1.5f * vy;
    a[0] = 0.2f * a[0];
    a[1] = u < -1.0f ? -1.0f : (u > 1.0f ? 1.0f : u);
  }
}

// Fused rollout: K env steps per env in one launch with in-kernel Philox actions; one thread per env, the state
// stays in registers for the whole rollout (the fast-forward runs in line).
template <typename T, int KIND>
__global__ void __launch_bounds__(kBlock) rollout_kernel(const __grid_constant__ Scene<T> sc, const __grid_constant__ StepIO io) {
  __shared__ unsigned long long sacc[kBlock / 32][TB_NUM_STATS];
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  WarpStats ws;
  ws.init(sacc[wib], lane);
  const int64_t me = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  T *base = static_cast<T *>(io.state);
  St<T> s;
  StepCtl c = {0, 0, 0, 0.0f, false};
  float a[8], ob[12] = {0}, rsum = 0;
  int left = 0, dcount = 0;
  bool active = me < io.n && io.k_steps > 0;
  if (me < io.n) {
    load_state(base, io.n, me, s);
    materialise_ball(sc, s);
    s.flags &= ~kStPristine;
  }
  if (active) {
    left = io.k_steps;
    rollout_action<T, KIND>(io, me, s, a);
    c.done = s.flags & kFlagDone;
  }
#pragma unroll 1
  while (true) {
    unsigned act_mask = __ballot_sync(full, active);
    if (!act_mask) break;
    bool fin = false;
    if (active) fin = env_substep<T, KIND>(sc, s, a, c);
    if (lane == 0) ws.acc[TB_STAT_PHYSICS_STEPS] += __popc(act_mask);
    if (fin) s.ret += (T)c.reward;
    account<T>(ws, fin, c.done, c.hit, c.events, s.step, s.ret);
    if (fin) {
      pack_obs<T, KIND>(s, ob);
      if (c.done) {
        if (io.auto_reset) {
          uint32_t ep = s.episode + 1;
          T in[TB_INIT_WORDS];
          draw_init<T, KIND>(io.seed, (uint64_t)(io.id_offset + me), ep, in);
          start_episode<T, KIND>(sc, s, in, ep, true);
          pack_obs<T, KIND>(s, ob);
        } else {
          s.flags |= kFlagDone;
        }
      }
      rsum += c.reward;
      dcount += c.done ? 1 : 0;
      if (--left > 0) {
        rollout_action<T, KIND>(io, me, s, a);
        c.phase = 0; c.events = 0; c.hit = 0; c.reward = 0.0f; c.done = s.flags & kFlagDone;
      } else {
        active = false;
      }
    }
  }
  if (me < io.n) {
    if (io.k_steps > 0) {
      if (io.obs) store_obs<KIND>(io.obs, me, ob);
      if (io.reward_sum) io.reward_sum[me] = rsum;
      if (io.done_count) io.done_count[me] = dcount;
      if (s.step > 0) s.flags &= ~kStPristine;  // (stepped through the generic path since its last episode start)
    }
    store_state(base, io.n, me, s);
  }
  ws.flush(io.stats);
}

// ------------------------------------------------------------------------------------------------ policy rollout
// SURVEY 8(f)-1: the policy of train_swing.py:80-91 (SB3 MlpPolicy, net_arch pi = vf = [32, 64, 32], tanh, Gaussian head with
// a state-independent log_std) evaluated on the device, so that a rollout is K x (policy_kernel, step_kernel, ff_kernel) on
// one stream: observations, actions and the per-step records PPO needs never leave HBM and no host code runs between steps.
// One thread per env; the parameters (layout TB_POLICY_* in the header) sit in shared memory and are read as broadcast
// float4; activations stay in registers (every loop is unrolled).  float32 throughout, like the torch policy.
// policy_kernel<OBS, ACT> is instantiated for SwingRacket-v0 (6 -> 6) and Tennisbot-v0 (12 -> 2); both use the same towers.
__host__ __device__ constexpr int pad4(int x) { return (x + 3) & ~3; }
template <int OBS, int ACT> struct PolLayout {  // float offsets; every tensor row-major [out][in], padded to 4 floats
  static constexpr int W1 = 0, B1 = 32 * OBS, W2 = B1 + 32, B2 = W2 + 64 * 32, W3 = B2 + 64, B3 = W3 + 32 * 64, Head = B3 + 32;
  static constexpr int PiTower = Head + ACT * 32 + pad4(ACT);  // + action_net W [ACT x 32], b
  static constexpr int VfTower = Head + 32 + 4;                // + value_net W [1 x 32], b
  static constexpr int LogStd = PiTower + VfTower, Floats = LogStd + pad4(ACT);
};
static_assert(PolLayout<6, 6>::Head == 4416 && PolLayout<6, 6>::PiTower == 4616 && PolLayout<6, 6>::VfTower == 4452 &&
              PolLayout<6, 6>::Floats == TB_POLICY_FLOATS, "policy layout / header mismatch (SwingRacket-v0)");
static_assert(PolLayout<12, 2>::PiTower == 4676 && PolLayout<12, 2>::VfTower == 4644 && PolLayout<12, 2>::Floats == TB_POLICY_FLOATS_HIT,
              "policy layout / header mismatch (Tennisbot-v0)");

// tanh(x) = 1 - 2 / (exp(2x) + 1) on the fast exponential: ~1e-6 absolute, a quarter of tanhf's instructions (a thread takes
// 256 of them per step)
__device__ __forceinline__ float tanh_fast(float x) {
  const float e = __expf(2.0f * fminf(fmaxf(x, -15.0f), 15.0f));
  return 1.0f - __fdividef(2.0f, e + 1.0f);
}
// y = tanh(W x + b): four outputs at a time, i.e. four independent accumulation chains per thread (at 16 384 envs there is
// one warp per scheduler: a single chain would run at the FMA latency)
template <int IN, int OUT>
__device__ __forceinline__ void dense_tanh(const float *__restrict__ W, const float *__restrict__ b, const float *x, float *y) {
  static_assert(OUT % 4 == 0, "outputs are taken four at a time");
#pragma unroll
  for (int o = 0; o < OUT; o += 4) {
    float acc[4] = {b[o], b[o + 1], b[o + 2], b[o + 3]};
    if (IN % 4 == 0) {
#pragma unroll
      for (int i = 0; i < IN / 4; ++i) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 w = reinterpret_cast<const float4 *>(W + (o + k) * IN)[i];
          acc[k] = fmaf(w.x, x[4 * i], acc[k]); acc[k] = fmaf(w.y, x[4 * i + 1], acc[k]);
          acc[k] = fmaf(w.z, x[4 * i + 2], acc[k]); acc[k] = fmaf(w.w, x[4 * i + 3], acc[k]);
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < IN; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[k] = fmaf(W[(o + k) * IN + i], x[i], acc[k]);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) y[o + k] = tanh_fast(acc[k]);
  }
}
// the three tanh layers of one tower: OBS -> 32 -> 64 -> 32
template <int OBS, int ACT>
__device__ __forceinline__ void tower(const float *P, const float *x, float *h3) {
  using L = PolLayout<OBS, ACT>;
  float h1[32], h2[64];
  dense_tanh<OBS, 32>(P + L::W1, P + L::B1, x, h1);
  dense_tanh<32, 64>(P + L::W2, P + L::B2, h1, h2);
  dense_tanh<64, 32>(P + L::W3, P + L::B3, h2, h3);
}
constexpr uint32_t kStreamPolicy = 2u;
struct PolicyIO {
  const float *params;     // PolLayout<OBS, ACT>::Floats floats in HBM
  const float *obs;        // [N, OBS] observation the action is computed from
  float *act_raw;          // [N, ACT] mean + std * eps, NOT clipped (what PPO's ratio is formed with), may be nullptr
  float *act_env;          // [N, ACT] clipped to the Box (what env.step gets: SB3 clips before stepping), may be nullptr
  float *logp, *value;     // [N] log-density of act_raw; value estimate (either may be nullptr)
  int64_t n, id_offset;
  uint64_t seed;           // noise streams are keyed (seed, global env id, tick): independent of the env's own streams
  const unsigned *tick;    // device word that advances with every env step (StepIO::epoch[0] for SwingRacket-v0, epoch[2]
                           // for Tennisbot-v0): a rollout captured in a CUDA graph draws fresh noise on every replay
  int deterministic;       // 1: act_raw = mean (validate_swing.py's predict(deterministic=True) counterpart)
  // NORM instances only (VecNormalize, header tb_set_vecnorm): obs holds RAW rows, which both towers normalise in registers
  const double *vn_stats;  // the running record, TB_VECNORM_WORDS(OBS) doubles
  float *vn_obs;           // [N, OBS] receives the normalised row (policy tower), may be nullptr
  float *vn_reward;        // [N] the previous step's raw reward, replaced by its normalised value (policy tower), may be nullptr
  double vn_clip_obs, vn_clip_reward, vn_eps;
  int vn_norm_obs, vn_norm_reward;
  // POP instances only (tb_set_policies): params holds one PolLayout row per agent; env i acts with agent i / envs_per_agent
  int64_t envs_per_agent;
};
// VecNormalize's two formulas in float64 with each operation rounded (no contraction), so that numpy reproduces them bit for
// bit: clip((o - mean) / sqrt(var + eps), -clip, clip), and the same for a reward with mean 0
__device__ __forceinline__ float vn_apply(float v, double mean, double var, double eps, double clip) {
  const double d = __ddiv_rn(__dsub_rn((double)v, mean), __dsqrt_rn(__dadd_rn(var, eps)));
  return __double2float_rn(fmin(fmax(d, -clip), clip));
}
// grid (ceil(N / 128), 2): blockIdx.y = 0 the policy tower (action, log-density), 1 the value tower.  NORM: the normalising
// instance of tb_policy_rollout with a normaliser attached; the policy tower also writes vn_obs and vn_reward.
// POP: the population instance (tb_set_policies, agents > 1).  A CTA stages the tower of each agent its 128 envs belong to in
// turn, and only that agent's threads compute with it: one pass when envs_per_agent is a multiple of 128, up to 128 passes
// (one env per agent) when agents straddle the CTA.  NORM && POP (tb_set_vecnorms): each agent pass normalises with that
// agent's record, vn_stats + agent TB_VECNORM_WORDS(OBS).
template <int OBS, int ACT, bool NORM, bool POP>
__global__ void __launch_bounds__(kBlock) policy_kernel(const __grid_constant__ PolicyIO io) {
  using L = PolLayout<OBS, ACT>;
  static_assert(OBS % 2 == 0 && ACT % 2 == 0, "observation rows are read as float2 / float4, actions written as float2");
  __shared__ __align__(16) float P[L::PiTower + pad4(ACT)];
  const bool vf = blockIdx.y != 0;
  pdl_wait();
  if (vf ? io.value == nullptr : (!io.act_raw && !io.act_env && !io.logp) && !(NORM && (io.vn_obs || io.vn_reward))) return;
  int64_t agent = 0, last_agent = 0;  // POP: the agents of this CTA's first and last env
  if (POP) {
    const int64_t first = (int64_t)blockIdx.x * kBlock;
    agent = first / io.envs_per_agent;
    last_agent = (min(first + kBlock, io.n) - 1) / io.envs_per_agent;
  }
  for (;; ++agent) {
    {
      const float *par = POP ? io.params + agent * L::Floats : io.params;
      const float4 *src = reinterpret_cast<const float4 *>(par + (vf ? L::PiTower : 0));
      const int nv = (vf ? L::VfTower : L::PiTower) / 4;
      for (int i = threadIdx.x; i < nv; i += kBlock) reinterpret_cast<float4 *>(P)[i] = src[i];
      if (!vf && threadIdx.x < pad4(ACT) / 4) reinterpret_cast<float4 *>(P + L::PiTower)[threadIdx.x] = reinterpret_cast<const float4 *>(par + L::LogStd)[threadIdx.x];
    }
    __syncthreads();
    const int64_t me = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (me < io.n && (!POP || (me >= agent * io.envs_per_agent && me < (agent + 1) * io.envs_per_agent))) {
      float x[OBS];
      if (OBS % 4 == 0) {  // 48 B rows (Tennisbot-v0): three float4
#pragma unroll
        for (int j = 0; j < OBS / 4; ++j) {
          const float4 a = reinterpret_cast<const float4 *>(io.obs + me * OBS)[j];
          x[4 * j] = a.x; x[4 * j + 1] = a.y; x[4 * j + 2] = a.z; x[4 * j + 3] = a.w;
        }
      } else {  // 24 B rows (SwingRacket-v0): three float2
#pragma unroll
        for (int j = 0; j < OBS / 2; ++j) {
          const float2 a = reinterpret_cast<const float2 *>(io.obs + me * OBS)[j];
          x[2 * j] = a.x; x[2 * j + 1] = a.y;
        }
      }
      if (NORM) {
        const double *st = POP ? io.vn_stats + agent * (2 * OBS + 4) : io.vn_stats;
        if (io.vn_norm_obs) {
#pragma unroll
          for (int c = 0; c < OBS; ++c) x[c] = vn_apply(x[c], st[c], st[OBS + c], io.vn_eps, io.vn_clip_obs);
        }
        if (!vf && io.vn_obs) {
          float2 *q = reinterpret_cast<float2 *>(io.vn_obs + me * OBS);
#pragma unroll
          for (int j = 0; j < OBS / 2; ++j) q[j] = make_float2(x[2 * j], x[2 * j + 1]);
        }
        if (!vf && io.vn_reward && io.vn_norm_reward)
          io.vn_reward[me] = vn_apply(io.vn_reward[me], 0.0, st[2 * OBS + 2], io.vn_eps, io.vn_clip_reward);
        if (!vf && !io.act_raw && !io.act_env && !io.logp) {  // the last launch: normalised reward only
          if (POP) goto next_agent;  // (the CTA's other agents' threads still meet the __syncthreads below)
          return;
        }
      }
      float h[32];
      tower<OBS, ACT>(P, x, h);
      if (!vf) {
        const float *Wa = P + L::Head, *ba = P + L::Head + ACT * 32, *ls = P + L::PiTower;
        // one Box-Muller pair (two uniforms) per two components: one Philox call per four components
        constexpr int NR = (ACT + 3) / 4;
        uint32_t rr[4 * NR];
        const uint32_t tick = *io.tick;
#pragma unroll
        for (int j = 0; j < NR; ++j) philox4x32(io.seed, (uint64_t)(io.id_offset + me), tick, stream_word(kStreamPolicy, 0, j), rr + 4 * j);
        float raw[ACT], lp = 0.0f;
#pragma unroll
        for (int o = 0; o < ACT; ++o) {
          float mu = ba[o];
#pragma unroll
          for (int i = 0; i < 32; ++i) mu = fmaf(Wa[o * 32 + i], h[i], mu);
          // Box-Muller on a pair of uniforms: component o takes the cosine (o even) or sine (o odd) branch of pair o / 2
          const float u1 = ((float)(rr[2 * (o / 2)] >> 8) + 0.5f) * (1.0f / 16777216.0f), u2 = (float)(rr[2 * (o / 2) + 1] >> 8) * (1.0f / 16777216.0f);
          const float rad = sqrtf(-2.0f * logf(u1));
          float sc;
          if (OBS == 6 && ACT == 6) {  // SwingRacket-v0 keeps sinf / cosf, so its rollouts stay what they were (their
            const float ang = 6.283185307179586f * u2;  // large-argument range reduction costs a 32-byte stack frame)
            sc = (o & 1) ? sinf(ang) : cosf(ang);
          } else {  // sin / cos of pi * 2 u2, 2 u2 in [0, 2): exact range reduction, nothing in local memory
            sc = (o & 1) ? sinpif(2.0f * u2) : cospif(2.0f * u2);
          }
          const float eps = io.deterministic ? 0.0f : rad * sc;
          raw[o] = fmaf(expf(ls[o]), eps, mu);
          lp += -0.5f * eps * eps - ls[o] - 0.9189385332046727f;
        }
        if (io.act_raw) {
          float2 *q = reinterpret_cast<float2 *>(io.act_raw + me * ACT);
#pragma unroll
          for (int j = 0; j < ACT / 2; ++j) q[j] = make_float2(raw[2 * j], raw[2 * j + 1]);
        }
        if (io.act_env) {
          float2 *q = reinterpret_cast<float2 *>(io.act_env + me * ACT);
#pragma unroll
          for (int o = 0; o < ACT; ++o) raw[o] = fminf(fmaxf(raw[o], -1.0f), 1.0f);
#pragma unroll
          for (int j = 0; j < ACT / 2; ++j) q[j] = make_float2(raw[2 * j], raw[2 * j + 1]);
        }
        if (io.logp) io.logp[me] = lp;
      } else {
        const float *Wv = P + L::Head;
        float v = Wv[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) v = fmaf(Wv[i], h[i], v);
        io.value[me] = v;
      }
    }
  next_agent:
    if (!POP || agent == last_agent) break;
    __syncthreads();  // every thread is done with this agent's tower before the next agent's is staged over it
  }
  pdl_trigger();
}

// ------------------------------------------------------------------------------------------------ ES fitness rollout
// SURVEY 8(f)-2: fitness_static (fitness_functions.py:18-158) for a whole population on the device.  Env i evaluates
// individual i / repeats with the reference's GatedCNN (policies.py:59-128) on an 8-step history of observations normalised by
// the env's own running normaliser (evolution_strategy_static.py:25-44, float64).  A rollout is K x (es_kernel, step_kernel,
// ff_kernel) on one stream plus one fold-only es_kernel: nothing between two env steps runs on the host.
// Parameters in parameters_to_vector order (es_eval.gated_cnn_sizes), each conv weight [out][in][2]:
//   conv_0 W[8 x C x 2] b[8], conv_gate_0 (same), conv_1 W[12 x 8 x 2] b[12] (dilation 2), conv_gate_1 (same),
//   conv_2 W[A x 12 x 2] b[A] (dilation 4)
template <int C, int A> struct EsLayout {
  static constexpr int W0 = 0, B0 = W0 + 16 * C, G0 = B0 + 8, GB0 = G0 + 16 * C, W1 = GB0 + 8, B1 = W1 + 192, G1 = B1 + 12,
                       GB1 = G1 + 192, W2 = GB1 + 12, B2 = W2 + 24 * A, Floats = B2 + A;
};
static_assert(EsLayout<6, 6>::Floats == TB_ES_FLOATS && EsLayout<12, 2>::Floats == TB_ES_FLOATS_HIT, "GatedCNN layout / header mismatch");
static_assert(TB_ES_HISTORY == 8, "the history ring is indexed with & 7");

struct EsIO {
  const float *w;               // [Floats][individuals]: the population parameter-major (tb_es_begin transposes the caller's rows),
                                // so lanes of one individual read one address and neighbouring individuals neighbouring ones
  int64_t n, individuals;
  int repeats;                  // env i evaluates individual i / repeats
  double *norm;                 // [2 OBS][N] normaliser: mean rows, then mean_diff rows
  double *n0;                   // [OBS] the master normaliser's count; every env has observed the same number of values since
  float *hist;                  // [8 OBS][N] ring of normalised observations; slot (tick - base) % 8 holds the newest
  double *ret;                  // [N] return summed while alive
  uint8_t *alive;               // [N] no done yet
  unsigned *stop;               // [N] tick - base when alive flipped: the observations the env's normaliser took (valid once dead)
  const unsigned *tick;         // the env-step counter (StepIO::epoch[0] / [2]): constant while an es_kernel runs
  unsigned *base;               // its value at tb_es_begin, so tick - base = env steps since then
  const float *obs, *term, *reward;  // the previous env step's outputs (the context's buffers)
  const uint8_t *done;
  int fold;                     // 1: fold the previous step into return, alive, normaliser and history
  float *act;                   // [N, A] clipped action for step_kernel; nullptr: fold only (the launch ending a rollout)
  float *obs_trace, *act_trace, *rew_trace;  // optional: step obs consumed [N, C], action [N, A], reward [N]
  uint8_t *done_trace;          // optional: done [N]
  double *ret_out;              // optional: return and alive copied out (the launch ending a rollout)
  uint8_t *alive_out;
};

// tanh(a) * sigmoid(g), on the accurate tanhf: tanh_fast's ~1e-6 per activation, carried through two layers of 16 and 24
// weighted terms, can reach ~1e-5 in the action
__device__ __forceinline__ float es_gate(float a, float g) { return tanhf(a) * fmaf(0.5f, tanhf(0.5f * g), 0.5f); }

// Observe x (float64, no contraction: the same roundings as BatchedNormalizer.observe), return the normalised value.
__device__ __forceinline__ float es_observe(double x, double nn, double &mean, double &md) {
  const double last = mean;
  mean = __dadd_rn(mean, (x - mean) / nn);
  md = __dadd_rn(md, __dmul_rn(x - last, x - mean));
  const double var = fmax(md / nn, 1e-2);
  return (float)((x - mean) / sqrt(var));
}

// One thread per env.  Only the network's last output position is needed, so conv_0 is evaluated at positions 0, 2, 4, 6
// and conv_1 at 0 and 4.  After an env's first done nothing it computes matters: it skips the fold and the network and
// hands a zero action to the env step.
template <int OBS, int ACT>
__global__ void __launch_bounds__(kBlock, 4) es_kernel(const __grid_constant__ EsIO io) {
  using L = EsLayout<OBS, ACT>;
  static_assert(OBS % 2 == 0 && ACT % 2 == 0, "observation and action rows are accessed as float2");
  pdl_wait();
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x, n = io.n;
  if (i < n) {
    const unsigned s = *io.tick - *io.base;
    const bool trace = io.obs_trace != nullptr;
    bool live = io.alive[i] != 0;
    const bool fold = io.fold && live;
    const uint8_t d = (trace || fold) ? io.done[i] : 0;
    if (io.fold) {
      if (io.rew_trace) io.rew_trace[i] = io.reward[i];
      if (io.done_trace) io.done_trace[i] = io.done[i];
    }
    double ret = 0.0;
    if (fold) {
      ret = io.ret[i] + (double)io.reward[i];
      io.ret[i] = ret;
      if (d) { live = false; io.alive[i] = 0; io.stop[i] = s; }
    } else if (io.ret_out) {
      ret = io.ret[i];
    }
    if (trace || (fold && live)) {
      float x[OBS];
      const float2 *src = reinterpret_cast<const float2 *>((d ? io.term : io.obs) + i * OBS);
#pragma unroll
      for (int j = 0; j < OBS / 2; ++j) { const float2 v = src[j]; x[2 * j] = v.x; x[2 * j + 1] = v.y; }
      if (trace) {
        float2 *q = reinterpret_cast<float2 *>(io.obs_trace + i * OBS);
#pragma unroll
        for (int j = 0; j < OBS / 2; ++j) q[j] = make_float2(x[2 * j], x[2 * j + 1]);
      }
      if (fold && live) {
        const int slot = (int)(s & 7u);
#pragma unroll
        for (int c = 0; c < OBS; ++c) {
          double mean = io.norm[c * n + i], md = io.norm[(OBS + c) * n + i];
          io.hist[(slot * OBS + c) * n + i] = es_observe((double)x[c], io.n0[c] + (double)(s + 1u), mean, md);
          io.norm[c * n + i] = mean; io.norm[(OBS + c) * n + i] = md;
        }
      }
    }
    if (io.act) {
      float a[ACT];
#pragma unroll
      for (int o = 0; o < ACT; ++o) a[o] = 0.0f;
      if (live) {
        const float *wp = io.w + i / io.repeats;
        const unsigned ld = (unsigned)io.individuals;  // (tb_es_begin keeps individuals x floats below 2^32)
        auto W = [&](int f) { return __ldg(wp + (unsigned)f * ld); };
        // conv_0 / conv_gate_0 (dilation 1) at positions 0, 2, 4, 6: position p reads history columns p and p + 1
        float h0[8][4], g0[8][4];
#pragma unroll
        for (int o = 0; o < 8; ++o) {
          const float b = W(L::B0 + o), bg = W(L::GB0 + o);
#pragma unroll
          for (int j = 0; j < 4; ++j) { h0[o][j] = b; g0[o][j] = bg; }
        }
        // The loops over conv_0's input channels and conv_1's outputs stay rolled: unrolled, ptxas hoists hundreds of
        // independent weight loads and spills.
        const int oldest = (int)((s + 1u) & 7u);
#pragma unroll 1
        for (int c = 0; c < OBS; ++c) {
          float x[8];  // channel c, oldest first
#pragma unroll
          for (int t = 0; t < 8; ++t) x[t] = io.hist[(((oldest + t) & 7) * OBS + c) * n + i];
#pragma unroll
          for (int o = 0; o < 8; ++o)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const float wa = W(L::W0 + (o * OBS + c) * 2 + k), wg = W(L::G0 + (o * OBS + c) * 2 + k);
#pragma unroll
              for (int j = 0; j < 4; ++j) { h0[o][j] = fmaf(wa, x[2 * j + k], h0[o][j]); g0[o][j] = fmaf(wg, x[2 * j + k], g0[o][j]); }
            }
        }
#pragma unroll
        for (int o = 0; o < 8; ++o)
#pragma unroll
          for (int j = 0; j < 4; ++j) h0[o][j] = es_gate(h0[o][j], g0[o][j]);
        // conv_1 / conv_gate_1 (dilation 2) at positions 0 and 4 (position 4 m reads conv_0 positions 4 m and 4 m + 2), each
        // output channel folded straight into conv_2 (dilation 4), whose one output position reads conv_1 positions 0 and 4
#pragma unroll
        for (int o = 0; o < ACT; ++o) a[o] = W(L::B2 + o);
#pragma unroll 1
        for (int o = 0; o < 12; ++o) {
          float acc[2], gac[2];
          acc[0] = acc[1] = W(L::B1 + o);
          gac[0] = gac[1] = W(L::GB1 + o);
#pragma unroll
          for (int c = 0; c < 8; ++c)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const float wa = W(L::W1 + (o * 8 + c) * 2 + k), wg = W(L::G1 + (o * 8 + c) * 2 + k);
#pragma unroll
              for (int m = 0; m < 2; ++m) { acc[m] = fmaf(wa, h0[c][2 * m + k], acc[m]); gac[m] = fmaf(wg, h0[c][2 * m + k], gac[m]); }
            }
          const float h1[2] = {es_gate(acc[0], gac[0]), es_gate(acc[1], gac[1])};
#pragma unroll
          for (int q = 0; q < ACT; ++q)
#pragma unroll
            for (int k = 0; k < 2; ++k) a[q] = fmaf(W(L::W2 + (q * 12 + o) * 2 + k), h1[k], a[q]);
        }
#pragma unroll
        for (int o = 0; o < ACT; ++o) a[o] = fminf(fmaxf(a[o], -1.0f), 1.0f);
      }
      float2 *q = reinterpret_cast<float2 *>(io.act + i * ACT);
#pragma unroll
      for (int j = 0; j < ACT / 2; ++j) q[j] = make_float2(a[2 * j], a[2 * j + 1]);
      if (io.act_trace) {
        q = reinterpret_cast<float2 *>(io.act_trace + i * ACT);
#pragma unroll
        for (int j = 0; j < ACT / 2; ++j) q[j] = make_float2(a[2 * j], a[2 * j + 1]);
      }
    }
    if (io.ret_out) { io.ret_out[i] = ret; io.alive_out[i] = live ? 1 : 0; }
  }
  pdl_trigger();
}

// After the reset of tb_es_begin: seed every env's normaliser from the master state (or zeros), observe the reset observation
// (io.obs), fill the history with its normalised value, zero the return, mark the env alive.
template <int OBS>
__global__ void __launch_bounds__(kBlock) es_begin_kernel(const __grid_constant__ EsIO io, const double *master) {
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x, n = io.n;
  if (blockIdx.x == 0 && threadIdx.x == 0) *io.base = *io.tick;
  if (blockIdx.x == 0 && threadIdx.x < OBS) io.n0[threadIdx.x] = master ? master[threadIdx.x] : 0.0;
  if (i >= n) return;
#pragma unroll
  for (int c = 0; c < OBS; ++c) {
    double mean = master ? master[OBS + c] : 0.0, md = master ? master[2 * OBS + c] : 0.0;
    const float z = es_observe((double)io.obs[i * OBS + c], (master ? master[c] : 0.0) + 1.0, mean, md);
    io.norm[c * n + i] = mean; io.norm[(OBS + c) * n + i] = md;
#pragma unroll
    for (int t = 0; t < 8; ++t) io.hist[(t * OBS + c) * n + i] = z;
  }
  io.ret[i] = 0.0;
  io.alive[i] = 1;
}

// [rows][cols] -> [cols][rows] through 32 x 32 shared tiles (block 32 x 8); rows on grid x, cols on grid y
__global__ void es_transpose_kernel(const float *in, int64_t rows, int cols, float *out) {
  __shared__ float tile[32][33];
  const int64_t r0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (r0 + j < rows && c0 + (int)threadIdx.x < cols) tile[j][threadIdx.x] = in[(r0 + j) * cols + c0 + threadIdx.x];
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += 8)
    if (c0 + j < cols && r0 + (int)threadIdx.x < rows) out[(int64_t)(c0 + j) * rows + r0 + threadIdx.x] = tile[threadIdx.x][j];
}

// ------------------------------------------------------------------------------------------------ ES population and update
// ARS V2-t (Mania, Guy and Recht 2018) with the perturbations keyed by seed, as OpenAI-ES does: nothing of size
// [individuals x floats] exists outside es_w, and every shard regenerates any direction it needs.
// Noise of direction j (a global index), parameter f, generation g, noise seed s: one Philox call per four parameters,
//   r = philox4x32(seed = s, id = j, episode = g, word = stream_word(kStreamEsNoise, f / 4, 0)),
// and Box-Muller in float64 on the pairs (r[0], r[1]) -> parameters 4q, 4q + 1 and (r[2], r[3]) -> 4q + 2, 4q + 3 (q = f / 4):
//   u1 = (r[2k] + 0.5) / 2^32,  u2 = r[2k + 1] / 2^32,  rho = sqrt(-2 ln u1),
//   eps[4q + 2k] = float32(rho cos(2 pi u2)),  eps[4q + 2k + 1] = float32(rho sin(2 pi u2))   (one rounding, to nearest)
// The stream id sits beside kStreamReset (0), kStreamAction (1) and kStreamPolicy (2); the env and policy streams are keyed by
// env ids, this one by direction ids, so they never share a counter.
constexpr uint32_t kStreamEsNoise = 3u;
__device__ __forceinline__ void es_noise4(uint64_t seed, int64_t j, uint32_t gen, int q, float eps[4]) {
  uint32_t r[4];
  philox4x32(seed, (uint64_t)j, gen, stream_word(kStreamEsNoise, (uint32_t)q, 0), r);
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const double u1 = ((double)r[2 * k] + 0.5) * 0x1p-32, u2 = (double)r[2 * k + 1] * 0x1p-32;
    const double rho = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    eps[2 * k] = __double2float_rn(rho * cs);
    eps[2 * k + 1] = __double2float_rn(rho * sn);
  }
}

// The population of tb_es_begin_noise straight into es_w [floats][2 pairs]: local individual p is global individual
// g = g0 + p (g0 even), of direction j = g >> 1, with w = theta + d for even g and theta - d for odd g, d = sigma * eps_j
// (each rounded on its own: no contraction).  Thread t makes the pair (2t, 2t + 1) of direction j0 + t and stores it as one
// float2, so stores are coalesced along individuals; grid y runs over the quads of parameters.
__global__ void __launch_bounds__(kBlock) es_perturb_kernel(const float *theta, int64_t pairs, int floats, float sigma,
                                                            uint64_t seed, uint32_t gen, int64_t j0, float *w) {
  const int64_t t = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  const int q = blockIdx.y;
  if (t >= pairs) return;
  float eps[4];
  es_noise4(seed, j0 + t, gen, q, eps);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int f = 4 * q + k;
    if (f < floats) {
      const float th = __ldg(theta + f), d = __fmul_rn(sigma, eps[k]);
      reinterpret_cast<float2 *>(w + (int64_t)f * 2 * pairs)[t] = make_float2(__fadd_rn(th, d), __fsub_rn(th, d));
    }
  }
}

// out[f] = sum_k coef[k] * eps_{dirs[k]}[f], accumulated in float64 in the order k = 0, 1, ... and rounded to float32 once, so
// the result depends on the inputs only.  One CTA per quad of parameters: its threads regenerate the terms of kBlock
// directions at a time (each product of two float32 values is exact in float64), threads 0..3 add them in order.
__global__ void __launch_bounds__(kBlock) es_combine_kernel(const int64_t *dirs, const float *coef, int64_t count, uint64_t seed,
                                                            uint32_t gen, int floats, float *out) {
  __shared__ double term[4][kBlock];
  const int q = blockIdx.x;
  double acc = 0.0;
  for (int64_t k0 = 0; k0 < count; k0 += kBlock) {
    const int64_t k = k0 + threadIdx.x;
    if (k < count) {
      float eps[4];
      es_noise4(seed, dirs[k], gen, q, eps);
      const double c = (double)coef[k];
#pragma unroll
      for (int m = 0; m < 4; ++m) term[m][threadIdx.x] = c * (double)eps[m];
    }
    __syncthreads();
    if (threadIdx.x < 4) {
      const int m = count - k0 < kBlock ? (int)(count - k0) : kBlock;
      for (int i = 0; i < m; ++i) acc += term[threadIdx.x][i];
    }
    __syncthreads();
  }
  const int f = 4 * q + (int)threadIdx.x;
  if (threadIdx.x < 4 && f < floats) out[f] = __double2float_rn(acc);
}

// Count, mean and M2 of a set of observations, the mean kept as its offset from the master's mean (small, well-conditioned).
struct EsMoments { double n, d, m2; };
// Chan, Golub and LeVeque's pairwise merge
__device__ __forceinline__ EsMoments es_merge(EsMoments a, EsMoments b) {
  if (b.n == 0.0) return a;
  if (a.n == 0.0) return b;
  const double n = a.n + b.n, delta = b.d - a.d;
  return {n, a.d + delta * (b.n / n), a.m2 + b.m2 + delta * delta * (a.n * (b.n / n))};
}
constexpr int kEsStatsPer = 8;  // envs per thread of es_norm_partial_kernel

// CTA-wide merge of one EsMoments per thread in a fixed tree; thread 0 gets the result
__device__ __forceinline__ EsMoments es_merge_cta(EsMoments v) {
  __shared__ double sh[3][kBlock];
  __syncthreads();
  sh[0][threadIdx.x] = v.n; sh[1][threadIdx.x] = v.d; sh[2][threadIdx.x] = v.m2;
  for (int h = kBlock / 2; h > 0; h >>= 1) {
    __syncthreads();
    if ((int)threadIdx.x < h) {
      const EsMoments r = es_merge({sh[0][threadIdx.x], sh[1][threadIdx.x], sh[2][threadIdx.x]},
                                   {sh[0][threadIdx.x + h], sh[1][threadIdx.x + h], sh[2][threadIdx.x + h]});
      sh[0][threadIdx.x] = r.n; sh[1][threadIdx.x] = r.d; sh[2][threadIdx.x] = r.m2;
    }
  }
  __syncthreads();
  return {sh[0][0], sh[1][0], sh[2][0]};
}

// Pass 1 of tb_es_normalizer_stats: each env's own share of its normaliser, the observations since tb_es_begin*, split off
// the master's (n0, mu0, M0).  Env e took m_e observations (tick - base + 1 while alive: the reset observation and one per
// step; io.stop once dead) and holds N = n0 + m_e, mean mu_e and mean_diff D_e, so its own observations have
//   mean - mu0 = (mu_e - mu0) N / m_e,   M2 = (D_e - M0) - (mean - mu0)^2 n0 m_e / N.
// Each thread merges kEsStatsPer envs in order, the CTA merges its threads in a fixed tree: part[blockIdx.x][3][OBS].
template <int OBS>
__global__ void __launch_bounds__(kBlock) es_norm_partial_kernel(const __grid_constant__ EsIO io, const double *m0, double *part) {
  const int64_t n = io.n, e0 = (int64_t)blockIdx.x * kBlock * kEsStatsPer + threadIdx.x;
  const unsigned s = *io.tick - *io.base;
  for (int c = 0; c < OBS; ++c) {
    const double n0 = m0[c], mu0 = m0[OBS + c], M0 = m0[2 * OBS + c];
    EsMoments v = {0.0, 0.0, 0.0};
    for (int r = 0; r < kEsStatsPer; ++r) {
      const int64_t e = e0 + (int64_t)r * kBlock;
      if (e >= n) break;
      const double m = io.alive[e] ? (double)(s + 1u) : (double)io.stop[e], nn = n0 + m;
      const double d = (io.norm[c * n + e] - mu0) * (nn / m);
      v = es_merge(v, {m, d, (io.norm[(OBS + c) * n + e] - M0) - d * d * (n0 * (m / nn))});
    }
    v = es_merge_cta(v);
    if (threadIdx.x == 0) {
      double *p = part + (int64_t)blockIdx.x * 3 * OBS;
      p[c] = v.n; p[OBS + c] = v.d; p[2 * OBS + c] = v.m2;
    }
  }
}

// Pass 2: one CTA per observation channel merges the `blocks` partials (each thread a strided subset in order, then the
// fixed tree) and writes out [3][OBS] = (count, mean, M2).
__global__ void __launch_bounds__(kBlock) es_norm_final_kernel(const double *part, int64_t blocks, int obs, const double *m0,
                                                               double *out) {
  const int c = blockIdx.x;
  EsMoments v = {0.0, 0.0, 0.0};
  for (int64_t b = threadIdx.x; b < blocks; b += kBlock) {
    const double *p = part + b * 3 * obs;
    v = es_merge(v, {p[c], p[obs + c], p[2 * obs + c]});
  }
  v = es_merge_cta(v);
  if (threadIdx.x == 0) { out[c] = v.n; out[obs + c] = m0[obs + c] + v.d; out[2 * obs + c] = v.m2; }
}

// ------------------------------------------------------------------------------------------------ VecNormalize (policy rollout)
// SB3 VecNormalize's running statistics (header tb_set_vecnorm), folded on the device after every env step of
// tb_policy_rollout in two launches: vecnorm_partial_kernel forms per-CTA moments of the N envs' observations (one channel
// each) and of their discounted returns, in the fixed order of es_norm_partial_kernel (kEsStatsPer envs per thread in order,
// then es_merge_cta); vecnorm_final_kernel merges the partials in one CTA and updates the record in place.  The moments are
// kept as offsets from the record's current mean, so the batch's delta of Chan's update is the merged offset itself.
// SEG (tb_set_vecnorms, A > 1 records): the segmented pass over A agents of io.n envs each, env i belonging to record i / io.n.
// The partial kernel runs es_norm_blocks(io.n) CTAs per agent, CTA k covering block k % blocks of agent k / blocks's slice
// (one flat grid: blockIdx.y would cap A at 65 535), with the geometry block b of a context of io.n envs has; the final kernel
// runs one CTA per agent.  So record p comes out bit-identical to the record of a context of io.n envs at env_id_offset p io.n.
struct VecNormIO {
  double *stats;           // the running record, TB_VECNORM_WORDS(OBS) doubles
  double *ret;             // [N] discounted returns
  const float *obs;        // [N, OBS] raw observations to fold
  float *copy;             // entry pass: obs is copied here (the library's raw buffer); else nullptr
  const float *reward;     // [N] the step's raw reward; nullptr = entry pass (obs only, and only while *armed)
  const uint8_t *done;     // [N] the step's done flags (step pass)
  double *part;            // [blocks][OBS + 1][3] per-CTA (count, mean offset, M2)
  uint8_t *armed;          // 1 until the entry pass after tb_set_vecnorm / a full reset has folded its observation
  int64_t n;
  double gamma;
  int fold_obs;            // training && norm_obs
};
template <int OBS, bool SEG = false>
__global__ void __launch_bounds__(kBlock) vecnorm_partial_kernel(const __grid_constant__ VecNormIO io) {
  // SEG: this CTA's agent, its block b within the agent, and the agent's first env
  const int64_t blocks = SEG ? (io.n + kBlock * kEsStatsPer - 1) / (kBlock * kEsStatsPer) : 1;
  const int64_t agent = SEG ? blockIdx.x / blocks : 0, b = SEG ? blockIdx.x - agent * blocks : blockIdx.x, first = agent * io.n;
  const double *st = SEG ? io.stats + agent * (2 * OBS + 4) : io.stats;
  const int64_t n = io.n, e0 = b * kBlock * kEsStatsPer + threadIdx.x;
  const bool fold_obs = io.fold_obs && (io.reward || *io.armed), fold_ret = io.reward != nullptr;
  double m0[OBS + 1];
  EsMoments v[OBS + 1];
#pragma unroll
  for (int c = 0; c <= OBS; ++c) { m0[c] = st[c < OBS ? c : 2 * OBS + 1]; v[c] = {0.0, 0.0, 0.0}; }
  for (int r = 0; r < kEsStatsPer; ++r) {
    const int64_t e = e0 + (int64_t)r * kBlock, g = SEG ? first + e : e;
    if (e >= n) break;
    float x[OBS];
#pragma unroll
    for (int j = 0; j < OBS / 2; ++j) {
      const float2 a = reinterpret_cast<const float2 *>(io.obs + g * OBS)[j];
      x[2 * j] = a.x; x[2 * j + 1] = a.y;
      if (io.copy) reinterpret_cast<float2 *>(io.copy + g * OBS)[j] = a;
    }
    if (fold_obs) {
#pragma unroll
      for (int c = 0; c < OBS; ++c) v[c] = es_merge(v[c], {1.0, __dsub_rn((double)x[c], m0[c]), 0.0});
    }
    if (fold_ret) {  // returns = returns * gamma + reward, folded; then returns[done] = 0
      const double R = __dadd_rn(__dmul_rn(io.ret[g], io.gamma), (double)io.reward[g]);
      v[OBS] = es_merge(v[OBS], {1.0, __dsub_rn(R, m0[OBS]), 0.0});
      io.ret[g] = io.done[g] ? 0.0 : R;
    }
  }
  double *p = io.part + (int64_t)blockIdx.x * (OBS + 1) * 3;
#pragma unroll
  for (int c = 0; c <= OBS; ++c) {
    if (c < OBS ? !fold_obs : !fold_ret) {  // (uniform over the CTA)
      // SEG: an empty partial tells the final kernel not to fold (it cannot read *io.armed: its CTA 0 clears it)
      if (SEG && c < OBS && io.fold_obs && threadIdx.x == 0) { p[3 * c] = 0.0; p[3 * c + 1] = 0.0; p[3 * c + 2] = 0.0; }
      continue;
    }
    const EsMoments s = es_merge_cta(v[c]);
    if (threadIdx.x == 0) { p[3 * c] = s.n; p[3 * c + 1] = s.d; p[3 * c + 2] = s.m2; }
  }
}
// One CTA: merge the `blocks` partials of each channel (each thread a strided subset in order, then the fixed tree) and apply
// RunningMeanStd.update_from_moments with batch mean = mean + d, batch variance M2 / N, batch count N:
//   tot = count + N, mean += d N / tot, var = (var count + M2 / N N + d^2 count N / tot) / tot, count = tot.
// SEG: CTA p merges agent p's `blocks` partials into record p; an obs channel whose partials are empty is not folded.
template <int OBS, bool SEG = false>
__global__ void __launch_bounds__(kBlock) vecnorm_final_kernel(const __grid_constant__ VecNormIO io, int64_t blocks) {
  const bool fold_obs = io.fold_obs && (SEG || io.reward || *io.armed), fold_ret = io.reward != nullptr;
  double *st = SEG ? io.stats + (int64_t)blockIdx.x * (2 * OBS + 4) : io.stats;
  double cnt[2] = {st[2 * OBS], st[2 * OBS + 3]}, tot[2] = {cnt[0], cnt[1]};
#pragma unroll
  for (int c = 0; c <= OBS; ++c) {
    if (c < OBS ? !fold_obs : !fold_ret) continue;
    EsMoments v = {0.0, 0.0, 0.0};
    for (int64_t b = threadIdx.x; b < blocks; b += kBlock) {
      const double *p = io.part + ((SEG ? (int64_t)blockIdx.x * blocks + b : b) * (OBS + 1) + c) * 3;
      v = es_merge(v, {p[0], p[1], p[2]});
    }
    v = es_merge_cta(v);
    if (threadIdx.x == 0 && (!SEG || v.n != 0.0)) {
      const int k = c < OBS ? 0 : 1;
      double *mean = c < OBS ? st + c : st + 2 * OBS + 1, *var = c < OBS ? st + OBS + c : st + 2 * OBS + 2;
      const double N = v.n, t = __dadd_rn(cnt[k], N), d = v.d;
      const double m2 = __dadd_rn(__dadd_rn(__dmul_rn(*var, cnt[k]), __dmul_rn(__ddiv_rn(v.m2, N), N)),
                                  __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(d, d), cnt[k]), N), t));
      *mean = __dadd_rn(*mean, __ddiv_rn(__dmul_rn(d, N), t));
      *var = __ddiv_rn(m2, t);
      tot[k] = t;
    }
  }
  if (threadIdx.x == 0) {
    st[2 * OBS] = tot[0]; st[2 * OBS + 3] = tot[1];
    if (!fold_ret && (!SEG || blockIdx.x == 0)) *io.armed = 0;
  }
}
// tb_set_vecnorm: the record from `src` (nullptr: fresh, RunningMeanStd(epsilon=1e-4)), returns zeroed, the fold armed
template <int OBS>
__global__ void __launch_bounds__(kBlock) vecnorm_init_kernel(const __grid_constant__ VecNormIO io, const double *src) {
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i < io.n) io.ret[i] = 0.0;
  if (i < 2 * OBS + 4) io.stats[i] = src ? src[i] : (i < OBS || i == 2 * OBS + 1) ? 0.0 : (i == 2 * OBS || i == 2 * OBS + 3) ? 1e-4 : 1.0;
  if (i == 0) *io.armed = 1;
}
// tb_set_vecnorms with A > 1: `records` records from `src` ([records][TB_VECNORM_WORDS(OBS)], nullptr: all fresh), returns
// zeroed, the fold armed
template <int OBS>
__global__ void __launch_bounds__(kBlock) vecnorm_init_records_kernel(const __grid_constant__ VecNormIO io, const double *src,
                                                                      int64_t records) {
  constexpr int W = 2 * OBS + 4;
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  const int w = (int)(i % W);
  if (i < io.n) io.ret[i] = 0.0;
  if (i < records * W) io.stats[i] = src ? src[i] : (w < OBS || w == 2 * OBS + 1) ? 0.0 : (w == 2 * OBS || w == 2 * OBS + 3) ? 1e-4 : 1.0;
  if (i == 0) *io.armed = 1;
}
// tb_reset / tb_reset_from with a normaliser in training: returns of the reset envs zeroed; a full reset arms the fold
__global__ void __launch_bounds__(kBlock) vecnorm_reset_kernel(const __grid_constant__ VecNormIO io, const uint8_t *mask) {
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i < io.n && (!mask || mask[i])) io.ret[i] = 0.0;
  if (i == 0 && !mask) *io.armed = 1;
}
// tb_sac_rollout with TB_SAC_VECNORM and a training normaliser, first launch: while the reset of tb_sac_begin is pending
// (io.armed = the SAC flag, cleared by the entry pass that follows and folds the reset observation), every return starts at 0
__global__ void __launch_bounds__(kBlock) vecnorm_sac_entry_kernel(const __grid_constant__ VecNormIO io) {
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i < io.n && *io.armed) io.ret[i] = 0.0;
}
// tb_vecnorm_apply: out = vn_apply of `in` with the record as it is when the kernel runs; reward rows use mean 0 and the
// return variance.  norm = 0 copies.  Element-wise, so in == out is allowed.
template <int OBS>
__global__ void __launch_bounds__(kBlock) vecnorm_apply_kernel(const double *stats, const float *in, float *out, int64_t count,
                                                               int reward, int norm, double clip, double eps) {
  const int64_t e = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (e >= count) return;
  const float v = in[e];
  if (!norm) { out[e] = v; return; }
  const int c = reward ? 0 : (int)(e % OBS);
  out[e] = reward ? vn_apply(v, 0.0, stats[2 * OBS + 2], eps, clip) : vn_apply(v, stats[c], stats[OBS + c], eps, clip);
}

// ------------------------------------------------------------------------------------------------ SAC actor and replay ring
// SURVEY 8(f)-5: the actor of SB3 SAC's MlpPolicy (latent_pi = Linear(obs, 256), ReLU, Linear(256, 256), ReLU; mu and log_std
// heads Linear(256, act); log_std clamped to [-20, 2]; action tanh(mu + exp(log_std) eps)) evaluated on the device, and every
// transition folded into a caller-owned replay ring.  A rollout is K x (sac_kernel, step_kernel, ff_kernel) + one fold-only
// sac_kernel, as the ES rollout.  Layer 2 (256 x 256) is the one dense contraction of the library: it runs on the tensor cores
// (tcgen05.mma, BF16 operands, FP32 accumulate in tensor memory); layer 1 and the heads stay float32 on the CUDA cores.
template <int OBS, int ACT> struct SacLayout {  // the caller's vector (header TB_SAC_*): float offsets, row-major [out][in]
  static constexpr int H = 256;
  static constexpr int W1 = 0, B1 = H * OBS, W2 = B1 + H, B2 = W2 + H * H, MuW = B2 + H, MuB = MuW + ACT * H,
                       LsW = MuB + pad4(ACT), LsB = LsW + ACT * H, Floats = LsB + pad4(ACT);
  // the image tb_set_sac_actor builds: W2 as BF16 in the canonical layout below (128 KB), then every other tensor in float32
  // in the same order and padding ("small" offsets = the vector's offsets with W2 taken out)
  static constexpr int SW1 = W1, SB1 = B1, SB2 = W2, SMuW = SB2 + H, SMuB = SMuW + ACT * H, SLsW = SMuB + pad4(ACT),
                       SLsB = SLsW + ACT * H, Small = SLsB + pad4(ACT);
  static constexpr int W2Bytes = H * H * 2, ABytes = 128 * H * 2;
  static constexpr int Smem = W2Bytes + ABytes + Small * 4 + 16;  // + mbarrier, TMEM address
};
static_assert(SacLayout<6, 6>::Floats == TB_SAC_FLOATS && SacLayout<12, 2>::Floats == TB_SAC_FLOATS_HIT, "SAC layout / header mismatch");
static_assert(SacLayout<6, 6>::Smem <= 227 * 1024 && SacLayout<12, 2>::Smem <= 227 * 1024, "SAC shared memory above 227 KB");

// UMMA canonical K-major layout without swizzle: 8 x 16-byte "core matrices" (8 rows x 8 BF16 along K, 128 contiguous bytes).
// Core matrix (row group g, K group kc) of an operand with R rows sits at byte (kc * R / 8 + g) * 128: one K = 16 step of the
// MMA reads K groups 2s and 2s + 1, i.e. leading byte offset (K direction) R * 16, stride byte offset (rows) 128.
__host__ __device__ constexpr uint32_t umma_offset(int row, int k, int rows) {
  return (uint32_t)(((k >> 3) * (rows >> 3) + (row >> 3)) * 128 + (row & 7) * 16 + (k & 7) * 2);
}
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
         (1ull << 46);  // bits 46-48 = 0b001 (sm_100 descriptor), base offset 0, swizzle none (bits 61-63 = 0)
}
// kind::f16 instruction descriptor: D FP32 (bits 4-5 = 1), A and B BF16 (bits 7-9, 10-12 = 1), both K-major, N >> 3 at bit 17,
// M >> 4 at bit 24
constexpr uint32_t kSacIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((256u >> 3) << 17) | ((128u >> 4) << 24);
__device__ __forceinline__ uint32_t bf16x2(float lo, float hi) {  // round to nearest even, lo in the low half
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

constexpr uint32_t kStreamSac = 4u;  // beside kStreamReset (0), kStreamAction (1), kStreamPolicy (2), kStreamEsNoise (3)
struct SacIO {
  const uint4 *w2;              // [8192] W2 image (BF16, canonical layout)
  const float *small;           // SacLayout::Small floats
  int64_t n, id_offset;
  uint64_t seed;
  const unsigned *tick;         // the env-step counter (StepIO::epoch[0] / [2]): constant while a sac_kernel runs
  const unsigned *base;         // its value at tb_sac_begin: step j since then writes ring slot j mod slots
  int mode;                     // TB_SAC_*
  int fold;                     // 1: fold the previous step into the ring and `cur`
  float *act;                   // [N, A] action for step_kernel; nullptr: fold only (the launch ending a rollout)
  const float *act_prev;        // the same buffer: the action the previous step took
  float *cur;                   // [N, C] the observation the next action is computed from
  const float *obs, *term, *reward;  // the previous env step's outputs (the context's buffers)
  const uint8_t *done;
  int64_t slots;                // ring (all nullptr: nothing stored)
  float *r_obs, *r_act, *r_reward, *r_next;
  uint8_t *r_done;
  float *last_obs;              // optional: `cur` after the fold (the launch ending a rollout)
  // NORM instances only (TB_SAC_VECNORM): the network acts on vn_apply of the raw observation; ring and `cur` stay raw
  const double *vn_stats;       // the running record, TB_VECNORM_WORDS(OBS) doubles
  double vn_clip_obs, vn_eps;
  int vn_norm_obs;
  // POP instances only (tb_set_sac_actors): w2 and small hold one image per agent, image_w2 uint4 and image_small floats
  // apart; env i acts with agent i / per_agent, a multiple of 128 so that every tile belongs to one agent
  int64_t image_w2, image_small, per_agent;
};

// Fold step j = tick - base - 1 of env i into the ring and `cur`; x receives the observation the next action is computed from.
template <int OBS, int ACT>
__device__ __forceinline__ void sac_fold(const SacIO &io, int64_t i, float *x) {
  const float2 *src = reinterpret_cast<const float2 *>((io.fold ? io.obs : io.cur) + i * OBS);
#pragma unroll
  for (int j = 0; j < OBS / 2; ++j) { const float2 v = src[j]; x[2 * j] = v.x; x[2 * j + 1] = v.y; }
  if (!io.fold) return;
  const int64_t n = io.n;
  if (io.r_obs) {
    const int64_t row = (int64_t)((uint64_t)(*io.tick - *io.base - 1u) % (uint64_t)io.slots) * n + i;
    const uint8_t d = io.done[i];
    const float2 *prev = reinterpret_cast<const float2 *>(io.cur + i * OBS);
    const float2 *nxt = reinterpret_cast<const float2 *>((d ? io.term : io.obs) + i * OBS);
    float2 *ro = reinterpret_cast<float2 *>(io.r_obs + row * OBS), *rn = reinterpret_cast<float2 *>(io.r_next + row * OBS);
#pragma unroll
    for (int j = 0; j < OBS / 2; ++j) { ro[j] = prev[j]; rn[j] = nxt[j]; }
    const float2 *a = reinterpret_cast<const float2 *>(io.act_prev + i * ACT);
    float2 *ra = reinterpret_cast<float2 *>(io.r_act + row * ACT);
#pragma unroll
    for (int j = 0; j < ACT / 2; ++j) ra[j] = a[j];
    io.r_reward[row] = io.reward[i];
    io.r_done[row] = d;
  }
  float2 *cur = reinterpret_cast<float2 *>(io.cur + i * OBS);
#pragma unroll
  for (int j = 0; j < OBS / 2; ++j) cur[j] = make_float2(x[2 * j], x[2 * j + 1]);
  if (io.last_obs) {
    float2 *q = reinterpret_cast<float2 *>(io.last_obs + i * OBS);
#pragma unroll
    for (int j = 0; j < OBS / 2; ++j) q[j] = make_float2(x[2 * j], x[2 * j + 1]);
  }
}

// The Philox words of env i at the current tick: uniform a = 2 u - 1 (TB_SAC_UNIFORM), or Gaussian eps (TB_SAC_SAMPLE).
template <int ACT> __device__ __forceinline__ void sac_noise(const SacIO &io, int64_t i, float *v, bool gaussian) {
  constexpr int NR = (ACT + 3) / 4;
  uint32_t rr[4 * NR];
  const uint32_t tick = *io.tick;
#pragma unroll
  for (int j = 0; j < NR; ++j) philox4x32(io.seed, (uint64_t)(io.id_offset + i), tick, stream_word(kStreamSac, 0, j), rr + 4 * j);
#pragma unroll
  for (int o = 0; o < ACT; ++o) {
    if (!gaussian) {
      v[o] = 2.0f * u01<float>(rr[o]) - 1.0f;
    } else {  // Box-Muller on pair o / 2: cosine branch for even o, sine for odd (policy_kernel<12, 2>'s formula)
      const float u1 = ((float)(rr[2 * (o / 2)] >> 8) + 0.5f) * (1.0f / 16777216.0f), u2 = (float)(rr[2 * (o / 2) + 1] >> 8) * (1.0f / 16777216.0f);
      v[o] = sqrtf(-2.0f * logf(u1)) * ((o & 1) ? sinpif(2.0f * u2) : cospif(2.0f * u2));
    }
  }
}

template <int ACT> __device__ __forceinline__ void sac_store_act(const SacIO &io, int64_t i, const float *a) {
  float2 *q = reinterpret_cast<float2 *>(io.act + i * ACT);
#pragma unroll
  for (int j = 0; j < ACT / 2; ++j) q[j] = make_float2(a[2 * j], a[2 * j + 1]);
}

// Two launch shapes.  Fold only, or TB_SAC_UNIFORM: one thread per env, no dynamic shared memory.  With the network: a
// persistent grid of min(tiles, SMs) CTAs with SacLayout::Smem bytes of dynamic shared memory (one CTA per SM), each looping
// over 128-env tiles, one env per thread and per TMEM lane:
//   layer 1 float32 (no contraction, so torch restates it exactly), ReLU, rounded to BF16 into the A tile (128 x 256);
//   thread 0 issues 16 x tcgen05.mma (M 128, N 256, K 16) into 256 TMEM columns and commits to an mbarrier;
//   each warp reads its 32 lanes back (tcgen05.ld 32x32b), adds b2, ReLU, and forms both heads in float32;
//   clamp, noise, accurate tanhf.
// NORM: the instance of tb_sac_rollout with TB_SAC_VECNORM; the network's input is normalised in registers before layer 1 (the
// one-thread-per-env shape evaluates no network, so it is the same code in both instances).
// POP: the population instance (tb_set_sac_actors, agents > 1).  Tile t belongs to agent t * 128 / per_agent.  Each CTA runs a
// contiguous chunk of tiles instead of the stride loop, so that its tiles are agent-contiguous, and loads an agent's image
// into shared memory only when its next tile belongs to another agent than the image it holds: once per CTA while tiles <=
// SMs, and about once per agent boundary a chunk crosses beyond that.
template <int OBS, int ACT, bool NORM, bool POP>
__global__ void __launch_bounds__(kBlock, 1) sac_kernel(const __grid_constant__ SacIO io) {
  using L = SacLayout<OBS, ACT>;
  static_assert(OBS % 2 == 0 && ACT % 2 == 0, "observation and action rows are accessed as float2");
  extern __shared__ __align__(1024) uint8_t sac_smem[];
  pdl_wait();
  const int64_t n = io.n;
  if (!io.act || io.mode == TB_SAC_UNIFORM) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i < n) {
      float x[OBS];
      sac_fold<OBS, ACT>(io, i, x);
      if (io.act) {
        float a[ACT];
        sac_noise<ACT>(io, i, a, false);
        sac_store_act<ACT>(io, i, a);
      }
    }
    pdl_trigger();
    return;
  }
  uint8_t *W2 = sac_smem, *A = sac_smem + L::W2Bytes;
  float *S = reinterpret_cast<float *>(sac_smem + L::W2Bytes + L::ABytes);
  uint64_t *bar = reinterpret_cast<uint64_t *>(S + L::Small);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5;
  int64_t held = 0;  // POP: the agent whose image shared memory holds, first that of this CTA's first tile
  {
    const uint4 *src = io.w2;
    const float *small = io.small;
    if constexpr (POP) {
      held = (n + kBlock - 1) / kBlock * blockIdx.x / gridDim.x * kBlock / io.per_agent;
      src += held * io.image_w2;
      small += held * io.image_small;
    }
    uint4 *w = reinterpret_cast<uint4 *>(W2);
    for (int q = tid; q < L::W2Bytes / 16; q += kBlock) w[q] = src[q];
    for (int q = tid; q < L::Small; q += kBlock) S[q] = small[q];
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_slot)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // W2 written by plain stores, read by the tensor cores
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot, a_base = smem_u32(A), b_base = smem_u32(W2), bar_a = smem_u32(bar);
  const int64_t tiles = (n + kBlock - 1) / kBlock;
  uint32_t phase = 0;
  int64_t tile = blockIdx.x, last = tiles;
  if constexpr (POP) {  // this CTA's chunk of tiles [tile, last)
    tile = tiles * blockIdx.x / gridDim.x;
    last = tiles * (blockIdx.x + 1) / gridDim.x;
  }
  for (; tile < last; tile += POP ? 1 : gridDim.x, phase ^= 1u) {
    if (POP && tile * kBlock / io.per_agent != held) {
      // every warp is past its tcgen05.ld of the previous tile and every thread past its reads of S, and the previous MMA,
      // which read W2, has completed (the mbarrier wait); then the new image, and the proxy fence before the next MMA
      __syncthreads();
      held = tile * kBlock / io.per_agent;
      const uint4 *src = io.w2 + held * io.image_w2;
      const float *small = io.small + held * io.image_small;
      uint4 *w = reinterpret_cast<uint4 *>(W2);
      for (int q = tid; q < L::W2Bytes / 16; q += kBlock) w[q] = src[q];
      for (int q = tid; q < L::Small; q += kBlock) S[q] = small[q];
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncthreads();
    }
    const int64_t i = tile * kBlock + tid;
    const bool mine = i < n;
    float x[OBS];
#pragma unroll
    for (int c = 0; c < OBS; ++c) x[c] = 0.0f;
    if (mine) sac_fold<OBS, ACT>(io, i, x);
    if (NORM && mine && io.vn_norm_obs) {
#pragma unroll
      for (int c = 0; c < OBS; ++c) x[c] = vn_apply(x[c], io.vn_stats[c], io.vn_stats[OBS + c], io.vn_eps, io.vn_clip_obs);
    }
    // layer 1: acc = b1, then + W1[j][c] x[c] for c = 0 .. OBS - 1, each product and sum rounded (no fused multiply-add)
#pragma unroll 1
    for (int kc = 0; kc < L::H / 8; ++kc) {
      float h[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int j = kc * 8 + u;
        float acc = S[L::SB1 + j];
#pragma unroll
        for (int c = 0; c < OBS; ++c) acc = __fadd_rn(acc, __fmul_rn(S[L::SW1 + j * OBS + c], x[c]));
        h[u] = fmaxf(acc, 0.0f);
      }
      *reinterpret_cast<uint4 *>(A + umma_offset(tid, kc * 8, 128)) =
          make_uint4(bf16x2(h[0], h[1]), bf16x2(h[2], h[3]), bf16x2(h[4], h[5]), bf16x2(h[6], h[7]));
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int s = 0; s < L::H / 16; ++s) {
        const uint64_t ad = umma_desc(a_base + s * 2 * 16 * 128, 16 * 128, 128), bd = umma_desc(b_base + s * 2 * 32 * 128, 32 * 128, 128);
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(tmem),
                     "l"(ad), "l"(bd), "r"(kSacIdesc), "r"(s));
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_a) : "memory");
    }
    asm volatile("{\n.reg .pred P;\nSAC_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P, [%0], %1;\n@!P bra SAC_WAIT;\n}" ::"r"(bar_a),
                 "r"(phase) : "memory");
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    float mu[ACT], ls[ACT];
#pragma unroll
    for (int o = 0; o < ACT; ++o) { mu[o] = S[L::SMuB + o]; ls[o] = S[L::SLsB + o]; }
#pragma unroll 1
    for (int q = 0; q < L::H / 32; ++q) {
      uint32_t r[32];
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,"
          "%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
          : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
            "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
            "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
            "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
          : "r"(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(q * 32)));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int u = 0; u < 32; ++u) {
        const int j = q * 32 + u;
        const float h = fmaxf(__uint_as_float(r[u]) + S[L::SB2 + j], 0.0f);
#pragma unroll
        for (int o = 0; o < ACT; ++o) {
          mu[o] = fmaf(S[L::SMuW + o * L::H + j], h, mu[o]);
          ls[o] = fmaf(S[L::SLsW + o * L::H + j], h, ls[o]);
        }
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");  // the next tile's MMA overwrites these columns
    if (mine) {
      float a[ACT], eps[ACT];
      const bool sample = io.mode == TB_SAC_SAMPLE;
      if (sample) sac_noise<ACT>(io, i, eps, true);
#pragma unroll
      for (int o = 0; o < ACT; ++o) {
        const float l = fminf(fmaxf(ls[o], -20.0f), 2.0f);
        a[o] = tanhf(sample ? fmaf(expf(l), eps[o], mu[o]) : mu[o]);
      }
      sac_store_act<ACT>(io, i, a);
    }
  }
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem));
  pdl_trigger();
}

// tb_set_sac_actor: the caller's float32 vector -> W2 in BF16 at its canonical-layout offset, everything else to `small`.
// POP (tb_set_sac_actors): a flat grid of agents x kSacImageBlocks CTAs; CTA b converts row b / kSacImageBlocks into image
// b / kSacImageBlocks of w2 (H x H halves apart) and small (SacLayout::Small floats apart).
template <int OBS, int ACT> constexpr int kSacImageBlocks = (SacLayout<OBS, ACT>::Floats + 255) / 256;
template <int OBS, int ACT, bool POP>
__global__ void __launch_bounds__(256) sac_image_kernel(const float *p, uint16_t *w2, float *small) {
  using L = SacLayout<OBS, ACT>;
  if (POP) {
    const int agent = blockIdx.x / kSacImageBlocks<OBS, ACT>;
    p += (int64_t)agent * L::Floats; w2 += (int64_t)agent * L::H * L::H; small += (int64_t)agent * L::Small;
  }
  const int f = (POP ? blockIdx.x % kSacImageBlocks<OBS, ACT> : blockIdx.x) * 256 + threadIdx.x;
  if (f >= L::Floats) return;
  if (f < L::W2) small[f] = p[f];
  else if (f < L::B2) {
    const int e = f - L::W2;
    w2[umma_offset(e / L::H, e % L::H, L::H) / 2] = (uint16_t)(bf16x2(p[f], 0.0f) & 0xFFFFu);
  } else small[f - L::H * L::H] = p[f];
}

template <typename T, int KIND>
__global__ void __launch_bounds__(kBlock) reset_kernel(const __grid_constant__ Scene<T> sc, const __grid_constant__ StepIO io,
                                                       const double *init, const uint8_t *mask) {
  int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i >= io.n) return;
  if (mask && !mask[i]) return;
  T *base = static_cast<T *>(io.state);
  St<T> s;
  load_state(base, io.n, i, s);
  uint32_t ep = s.episode + 1;  // a fresh context holds episode = 0xffffffff
  T in[TB_INIT_WORDS];
  if (init) {
#pragma unroll
    for (int j = 0; j < TB_INIT_WORDS; ++j) in[j] = (T)init[i * TB_INIT_WORDS + j];
  } else {
    draw_init<T, KIND>(io.seed, (uint64_t)(io.id_offset + i), ep, in);
  }
  start_episode<T, KIND>(sc, s, in, ep, init == nullptr);
  store_state(base, io.n, i, s);
  if (io.pid) {
    T z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    store_pid(static_cast<T *>(io.pid), io.n, i, z);
  }
  if (io.obs) {
    float ob[12];
    pack_obs<T, KIND>(s, ob);
    store_obs<KIND>(io.obs, i, ob);
  }
}

// Scene::ball_vz: the vertical velocity of a ball after k contact-free substeps from rest, by the kernels' own arithmetic
// (ball_free_velocities, as in ctl_fast), so that a state materialised from the table is the state that was stepped
template <typename T> __global__ void ball_vz_kernel(const __grid_constant__ Scene<T> sc, T *out) {
  T bv[3] = {0, 0, 0}, bw[3] = {0, 0, 0};
  for (int k = 0; k < kBallVzEntries; ++k) {
    out[k] = bv[2];
    ball_free_velocities(sc, bv, bw);
  }
}

// Write pack 4 of every kStPristine env from the table and clear the bit (before the table changes: tb_set_param)
template <typename T> __global__ void materialise_kernel(const __grid_constant__ Scene<T> sc, T *base, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Pack<T> p7 = ld_pack(base, n, 7, i);
  int flags = (int)as_int(p7.z);
  if (!(flags & kStPristine)) return;
  St<T> s;
  s.flags = flags; s.step = (int)as_int(p7.y);
  materialise_ball(sc, s);
  st_pack(base, n, 4, i, Pack<T>{s.bv[0], s.bv[1], s.bv[2], s.bw[0]});
  base[((int64_t)7 * n + i) * 4 + 2] = int_as(T(), flags & ~kStPristine);
}

// canonical double [TB_STATE_WORDS] record <-> St<T> (a materialised state: no kStPristine, no stale pack 4)
template <typename T> __device__ __forceinline__ void state_to_record(const St<T> &s, double *o) {
  for (int j = 0; j < 3; ++j) {
    o[TB_S_RACKET_POS + j] = s.rp[j]; o[TB_S_RACKET_VEL + j] = s.rv[j]; o[TB_S_RACKET_ANGVEL + j] = s.rw[j];
    o[TB_S_BALL_POS + j] = s.bp[j]; o[TB_S_BALL_VEL + j] = s.bv[j]; o[TB_S_BALL_ANGVEL + j] = s.bw[j];
    o[TB_S_AUX + j] = s.aux[j];
  }
  for (int j = 0; j < 4; ++j) o[TB_S_RACKET_QUAT + j] = s.rq[j];
  o[TB_S_GOAL] = s.goal[0]; o[TB_S_GOAL + 1] = s.goal[1]; o[TB_S_D0] = s.d0; o[TB_S_RETURN] = s.ret;
  o[TB_S_STEP] = s.step; o[TB_S_FLAGS] = s.flags & kFlagDone; o[TB_S_EPISODE] = (double)(int32_t)s.episode;
}
template <typename T> __device__ __forceinline__ void record_to_state(const double *o, St<T> &s) {
  for (int j = 0; j < 3; ++j) {
    s.rp[j] = (T)o[TB_S_RACKET_POS + j]; s.rv[j] = (T)o[TB_S_RACKET_VEL + j]; s.rw[j] = (T)o[TB_S_RACKET_ANGVEL + j];
    s.bp[j] = (T)o[TB_S_BALL_POS + j]; s.bv[j] = (T)o[TB_S_BALL_VEL + j]; s.bw[j] = (T)o[TB_S_BALL_ANGVEL + j];
    s.aux[j] = (T)o[TB_S_AUX + j];
  }
  for (int j = 0; j < 4; ++j) s.rq[j] = (T)o[TB_S_RACKET_QUAT + j];
  s.goal[0] = (T)o[TB_S_GOAL]; s.goal[1] = (T)o[TB_S_GOAL + 1]; s.d0 = (T)o[TB_S_D0]; s.ret = (T)o[TB_S_RETURN];
  s.step = (int)o[TB_S_STEP]; s.flags = (int)o[TB_S_FLAGS] & kFlagDone; s.episode = (uint32_t)(int32_t)o[TB_S_EPISODE];
}

// canonical double [N, 32] record <-> packed state
template <typename T> __global__ void get_state_kernel(const __grid_constant__ Scene<T> sc, const T *base, int64_t n, double *out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  St<T> s;
  load_state(base, n, i, s);
  materialise_ball(sc, s);
  state_to_record(s, out + i * TB_STATE_WORDS);
}
template <typename T> __global__ void set_state_kernel(T *base, int64_t n, const double *in) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  St<T> s;
  record_to_state(in + i * TB_STATE_WORDS, s);
  store_state(base, n, i, s);
}

// ------------------------------------------------------------------------------------------------ tb_trace_step
// One thread per traced record: the record's env step taken as rollout_kernel takes it (env_substep until the step is
// complete), with the canonical record stored after every substep.  A trace is a diagnostic of a few envs, not a
// throughput path: a lane runs its flight alone, so a warp takes as long as its longest flight.
struct TraceIO {
  const double *states;
  const float *actions;
  int64_t count;
  int max_substeps;
  double *trace;  // [max_substeps, count, TB_STATE_WORDS]
  uint8_t *bits;  // [max_substeps, count] or nullptr
  int32_t *substeps;
  float *reward;
  uint8_t *done, *events;
};
constexpr int kTraceBlock = 128;
__device__ __forceinline__ void store_record(double *dst, const double *r) {
  double2 *p = reinterpret_cast<double2 *>(dst);
#pragma unroll
  for (int j = 0; j < TB_STATE_WORDS / 2; ++j) p[j] = make_double2(r[2 * j], r[2 * j + 1]);
}

template <typename T, int KIND>
__global__ void __launch_bounds__(kTraceBlock) trace_kernel(const __grid_constant__ Scene<T> sc, const __grid_constant__ TraceIO io) {
  const int64_t i = (int64_t)blockIdx.x * kTraceBlock + threadIdx.x;
  if (i >= io.count) return;
  St<T> s;
  record_to_state(io.states + i * TB_STATE_WORDS, s);
  float a[8];
  load_action<KIND>(io.actions, i, a);
  StepCtl c = {0, 0, 0, 0.0f, false};
  c.done = s.flags & kFlagDone;
  double r[TB_STATE_WORDS];
  int k = 0;
  bool fin = false;
#pragma unroll 1
  while (!fin) {
    int bits = 0;
    fin = env_substep<T, KIND>(sc, s, a, c, nullptr, &bits);
    if (fin) {
      s.ret += (T)c.reward;
      if (c.done) s.flags |= kFlagDone;
    }
    if (k < io.max_substeps) {  // a longer step still runs to its end: substeps, reward, done and events stay complete
      state_to_record(s, r);
      store_record(io.trace + ((int64_t)k * io.count + i) * TB_STATE_WORDS, r);
      if (io.bits) io.bits[(int64_t)k * io.count + i] = (uint8_t)bits;
    }
    ++k;
  }
  // the rest of the block repeats the final record (r holds it whenever k < max_substeps)
#pragma unroll 1
  for (int j = k; j < io.max_substeps; ++j) {
    store_record(io.trace + ((int64_t)j * io.count + i) * TB_STATE_WORDS, r);
    if (io.bits) io.bits[(int64_t)j * io.count + i] = 0;
  }
  io.substeps[i] = k;
  if (io.reward) io.reward[i] = c.reward;
  if (io.done) io.done[i] = c.done ? 1 : 0;
  if (io.events) io.events[i] = (uint8_t)c.events;
}

// ------------------------------------------------------------------------------------------------ tb_render
// One thread per pixel; a CTA covers kRenderBlock consecutive pixels (row-major) of one frame at a time and walks the frames
// blockIdx.y, blockIdx.y + gridDim.y, ...  Per frame, 71 threads stage what every ray of it shares: the racket's rotation,
// the shapes' centres relative to the eye, and the eye's offset c from every prism edge plane, formed in float64 from the
// record and rounded once (the rays then clip in float32).
constexpr int kRenderBlock = 256;
struct RenderIO {
  const double *states;
  int64_t count;
  uint8_t *rgb, *body;
  float *depth;
  int width, height;
  double eye[3];
  float f[3], r[3], u[3];  // view direction; r scaled by t W / H, u by t (the camera of tb_render)
  float light[3];          // TB_RENDER_LIGHT normalised
  float box_c[2][6];       // floor, net: ray_box's cb for this eye
};
__constant__ uint8_t k_render_color[6][3] = TB_RENDER_COLORS;
enum { kRfR = 0, kRfRp = 9, kRfOt = 12, kRfBall = 13, kRfGoal = 16, kRfGoalT = 19, kRfWords = 20 };

template <typename T, int KIND>
__global__ void __launch_bounds__(kRenderBlock) render_kernel(const __grid_constant__ Scene<T> sc, const __grid_constant__ RenderIO io) {
  constexpr bool kGoal = KIND == TB_ENV_SWING;
  __shared__ float s_rc[kRacketEdges], s_gc[kGoalEdges], s_f[kRfWords];
  const int64_t npix = (int64_t)io.width * io.height;
  const int64_t pix = (int64_t)blockIdx.x * kRenderBlock + threadIdx.x;
  const int px = (int)(pix % io.width), py = (int)(pix / io.width);
  float d[3];
  {
    const float a = (float)(2 * px + 1 - io.width) / (float)io.width, b = (float)(io.height - 2 * py - 1) / (float)io.height;
#pragma unroll
    for (int k = 0; k < 3; ++k) d[k] = io.f[k] + a * io.r[k] + b * io.u[k];
    const float inv = 1.f / sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) d[k] *= inv;
  }
  for (int64_t fr = blockIdx.y; fr < io.count; fr += gridDim.y) {
    const double *rec = io.states + fr * TB_STATE_WORDS;
    const int i = threadIdx.x;
    __syncthreads();  // the previous frame's rays are done with the staged words
    if (i <= kRacketEdges) {
      double R[9], rel[3], ol[3];
      quat_to_mat(rec + TB_S_RACKET_QUAT, R);
      for (int k = 0; k < 3; ++k) rel[k] = io.eye[k] - rec[TB_S_RACKET_POS + k];
      matT_vec(R, rel, ol);
      if (i < kRacketEdges) {
        const Edge<T> &e = sc.racket.e[i];
        s_rc[i] = (float)((ol[1] - (double)e.ax) * (double)e.nx + (ol[2] - (double)e.ay) * (double)e.ny);
      } else {
        for (int k = 0; k < 9; ++k) s_f[kRfR + k] = (float)R[k];
        for (int k = 0; k < 3; ++k) {
          s_f[kRfRp + k] = (float)-rel[k];
          s_f[kRfBall + k] = (float)(rec[TB_S_BALL_POS + k] - io.eye[k]);
        }
        s_f[kRfOt] = (float)ol[0];
        s_f[kRfGoal] = (float)(rec[TB_S_GOAL] - io.eye[0]);
        s_f[kRfGoal + 1] = (float)(rec[TB_S_GOAL + 1] - io.eye[1]);
        s_f[kRfGoal + 2] = (float)-io.eye[2];
        s_f[kRfGoalT] = (float)io.eye[2];
      }
    } else if (kGoal && i <= kRacketEdges + kGoalEdges) {
      const Edge<T> &e = sc.goal.e[i - kRacketEdges - 1];
      const double ou = io.eye[0] - rec[TB_S_GOAL], ov = io.eye[1] - rec[TB_S_GOAL + 1];
      s_gc[i - kRacketEdges - 1] = (float)((ou - (double)e.ax) * (double)e.nx + (ov - (double)e.ay) * (double)e.ny);
    }
    __syncthreads();
    if (pix >= npix) continue;
    float best = M<float>::inf(), n[3] = {0.f, 0.f, 0.f};
    int body = TB_BODY_NONE, face;
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const float s = ray_box(io.box_c[b], d, face);
      if (s < best) {
        best = s; body = b ? TB_BODY_NET : TB_BODY_COURT;
        n[0] = n[1] = n[2] = 0.f;
        n[face >> 1] = (face & 1) ? -1.f : 1.f;
      }
    }
    if (kGoal && !ray_skips(s_f + kRfGoal, (float)sc.goal.bound_radius, d, best)) {
      const float dl[3] = {d[2], d[0], d[1]};
      const float s = ray_prism(sc.goal, s_gc, s_f[kRfGoalT], dl, face);
      if (s < best) {
        best = s; body = TB_BODY_GOAL;
        if (face < 2) { n[0] = n[1] = 0.f; n[2] = face ? -1.f : 1.f; }
        else { n[0] = (float)sc.goal.e[face - 2].nx; n[1] = (float)sc.goal.e[face - 2].ny; n[2] = 0.f; }
      }
    }
    if (!ray_skips(s_f + kRfRp, (float)sc.racket.bound_radius, d, best)) {
      const float *R = s_f + kRfR;
      float dl[3];
      matT_vec(R, d, dl);
      const float s = ray_prism(sc.racket, s_rc, s_f[kRfOt], dl, face);
      if (s < best) {
        best = s; body = TB_BODY_RACKET;
        float nl[3] = {face == 0 ? 1.f : (face == 1 ? -1.f : 0.f), 0.f, 0.f};
        if (face >= 2) { nl[1] = (float)sc.racket.e[face - 2].nx; nl[2] = (float)sc.racket.e[face - 2].ny; }
        mat_vec(R, nl, n);
      }
    }
    {
      const float *c = s_f + kRfBall, r = (float)sc.ball_r;
      const float s = ray_sphere(c, r, d);
      if (s < best) {
        best = s; body = TB_BODY_BALL;
#pragma unroll
        for (int k = 0; k < 3; ++k) n[k] = (s * d[k] - c[k]) / r;
      }
    }
    const int64_t o = fr * npix + pix;
    if (io.depth) io.depth[o] = best;
    if (io.body) io.body[o] = (uint8_t)body;
    uint8_t *px_rgb = io.rgb + 3 * o;
    if (body == TB_BODY_NONE) {
      const uint8_t sky[3] = TB_RENDER_SKY;
      px_rgb[0] = sky[0]; px_rgb[1] = sky[1]; px_rgb[2] = sky[2];
    } else {
      float nl = n[0] * io.light[0] + n[1] * io.light[1] + n[2] * io.light[2];
      if (n[0] * d[0] + n[1] * d[1] + n[2] * d[2] > 0.f) nl = -nl;
      const float k = 0.35f + 0.65f * fmaxf(0.f, nl);
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) px_rgb[ch] = (uint8_t)floorf((float)k_render_color[body][ch] * k + 0.5f);
    }
  }
}

// ------------------------------------------------------------------------------------------------ host side
struct Params {  // order matches k_param_names
  double dt, gravity_z, lin_damping, ang_damping, max_coord_vel, rest_ball_racket, rest_ball_court, rest_ball_goal,
      fric_ball_racket, fric_ball_court, fric_ball_goal, contact_erp, linear_slop, rest_vel_threshold,
      solver_iterations, solver_residual, contact_threshold, hull_margin, box_margin, gyro_term, racket_scale, pid_kp,
      pid_ki, pid_kd, pid_max_force, pid_bias_z, pid_hit_z, shoot_start, shoot_frames, racket_court_contact, rest_racket_court,
      fric_racket_court;
};
static const char *k_param_names[] = {
    "dt", "gravity_z", "lin_damping", "ang_damping", "max_coord_vel", "rest_ball_racket", "rest_ball_court",
    "rest_ball_goal", "fric_ball_racket", "fric_ball_court", "fric_ball_goal", "contact_erp", "linear_slop",
    "rest_vel_threshold", "solver_iterations", "solver_residual", "contact_threshold", "hull_margin",
    "box_margin", "gyro_term", "racket_scale", "pid_kp", "pid_ki", "pid_kd", "pid_max_force", "pid_bias_z",
    "pid_hit_z", "shoot_start", "shoot_frames", "racket_court_contact", "rest_racket_court", "fric_racket_court"};
constexpr int kNumParams = sizeof(k_param_names) / sizeof(k_param_names[0]);
static_assert(sizeof(Params) == kNumParams * sizeof(double), "Params / name table mismatch");

static void params_default(Params &p) {
  p.dt = 1.0 / 240.0;          // fixed PyBullet time step [R]
  p.gravity_z = -9.81;         // swingracket_env.py:154
  p.lin_damping = 0.04;        // btMultiBody default, a = -v (k + k|v|) [R]
  p.ang_damping = 0.04;
  p.max_coord_vel = 100.0;
  p.rest_ball_racket = 0.9 * 0.9;  // racket.py:43 x objects.py:48
  p.rest_ball_court = 0.9 * 0.9;   // objects.py:29 x objects.py:48
  p.rest_ball_goal = 0.0;          // goal keeps Bullet's default restitution 0
  p.fric_ball_racket = 0.2 * 0.2;
  p.fric_ball_court = 0.2 * 0.2;
  p.fric_ball_goal = 0.2 * 0.5;
  p.contact_erp = 0.08;
  p.linear_slop = 1e-5;
  p.rest_vel_threshold = 0.2;
  p.solver_iterations = 50;
  p.solver_residual = 1e-7;
  p.contact_threshold = 0.02 * std::sqrt(3.0) * TB_BALL_RADIUS;
  p.hull_margin = TB_URDF_MARGIN;
  p.box_margin = TB_URDF_MARGIN;
  p.gyro_term = 1.0;
  p.racket_scale = 1.0;
  p.pid_kp = 3.0;   // racket.py:49-52
  p.pid_ki = 0.01;
  p.pid_kd = 0.1;
  p.pid_max_force = 10.0;
  p.pid_bias_z = 4.0;    // racket.py:110
  p.pid_hit_z = 1.5;     // tennisbot_env.py:106
  p.shoot_start = 0;     // tennisbot_env.py:118 (playground.py:99 shoots on frames 11 .. 49)
  p.shoot_frames = 5;    // BALL_SHOOT_FRAMES, tennisbot_env.py:21
  p.racket_court_contact = 0;        // 1: racket vs the court's floor box on the generic path (see Scene::racket_court)
  p.rest_racket_court = 0.9 * 0.9;   // racket.py:43 x objects.py:29
  p.fric_racket_court = 0.2 * 0.2;   // racket.py:44 x objects.py:30
}

// quad_edges: indices of the two outline edges that bound the quadrilateral of prism_inside_fast (its other two sides
// are the lines v = the lower and the upper end of those edges), or nullptr.  Both regions are verified against every edge
// line here and dropped if they do not clear them all.
template <typename T, int NE> static void build_prism(Prism<T, NE> &pr, const double (*v)[2], double half_thick, const int *quad_edges) {
  double r2 = 0, nx[NE], ny[NE];
  for (int i = 0; i < NE; ++i) {
    const double *a = v[i], *b = v[(i + 1) % NE];
    double ex = b[0] - a[0], ey = b[1] - a[1], l2 = ex * ex + ey * ey, il = 1.0 / std::sqrt(l2);
    pr.e[i].ax = (T)a[0]; pr.e[i].ay = (T)a[1]; pr.e[i].ex = (T)ex; pr.e[i].ey = (T)ey;
    pr.e[i].inv_len2 = (T)(1.0 / l2); pr.e[i].nx = (T)(ey * il); pr.e[i].ny = (T)(-ex * il);
    nx[i] = ey * il; ny[i] = -ex * il;
    double d2 = a[0] * a[0] + a[1] * a[1] + half_thick * half_thick;
    if (d2 > r2) r2 = d2;
  }
  pr.half_thick = (T)half_thick;
  pr.bound_radius = (T)std::sqrt(r2);
  const double shrink = sizeof(T) == 8 ? 1.0 - 1e-9 : 1.0 - 1e-4;
  {
    // ellipse: centred where the outline is widest (above the quadrilateral, if there is one), semi-axes out to the widest
    // point and up to the top, then scaled about its centre until it lies inside every edge's half plane
    double vlo = -1e30;
    if (quad_edges) vlo = std::fmax(std::fmax(v[quad_edges[0]][1], v[(quad_edges[0] + 1) % NE][1]), std::fmax(v[quad_edges[1]][1], v[(quad_edges[1] + 1) % NE][1]));
    double a0 = 0, c = 0, top = -1e30;
    for (int i = 0; i < NE; ++i) {
      if (v[i][1] < vlo) continue;
      if (std::fabs(v[i][0]) > a0) { a0 = std::fabs(v[i][0]); c = v[i][1]; }
      top = std::fmax(top, v[i][1]);
    }
    double b0 = top - c, s = 1e30;
    if (!(b0 > 0)) { b0 = a0; c = 0; }  // (a polygon symmetric about u as well, e.g. the goal's 32-gon: a circle)
    for (int i = 0; i < NE; ++i) {
      double off = (v[i][0] - 0.0) * nx[i] + (v[i][1] - c) * ny[i];
      double sup = std::sqrt(a0 * nx[i] * a0 * nx[i] + b0 * ny[i] * b0 * ny[i]);
      s = std::fmin(s, off / sup);
    }
    if (s > 0) {
      pr.in_c = (T)c; pr.in_inv_a = (T)(1.0 / (a0 * s * shrink)); pr.in_inv_b = (T)(1.0 / (b0 * s * shrink));
    } else {  // never inside
      pr.in_c = 0; pr.in_inv_a = (T)1e30; pr.in_inv_b = (T)1e30;
    }
    // the containing ellipse of the vertices at or above vlo (same centre and aspect), for prism_outside_fast
    double so = 0;
    for (int i = 0; i < NE; ++i) {
      if (v[i][1] < vlo) continue;
      double du = v[i][0] / a0, dv = (v[i][1] - c) / b0;
      so = std::fmax(so, std::sqrt(du * du + dv * dv));
    }
    pr.out_a = (T)(a0 * so / shrink); pr.out_b = (T)(b0 * so / shrink);
    pr.out_v = (T)vlo; pr.out_lo = (T)-1e30;
    pr.out_inv_a = pr.out_inv_b = 0;  // (set by build_scene once the rim is known)
  }
  {
    // coarse outline: walk the edges and keep one whenever the direction has turned by `turn` since the last one kept, and every
    // edge that is long (its neighbours' lines would meet far outside the outline); the smallest `turn` that fits the table
    double len[NE], med[NE], ang[NE];
    for (int i = 0; i < NE; ++i) {
      const double *a = v[i], *b = v[(i + 1) % NE];
      len[i] = med[i] = std::hypot(b[0] - a[0], b[1] - a[1]);
      ang[i] = std::atan2(b[1] - a[1], b[0] - a[0]);
    }
    std::sort(med, med + NE);
    const double long_edge = 1.5 * med[NE / 2];
    int keep[NE], nk = 0;
    for (double turn = 10.0; turn <= 180.0; turn += 1.0) {
      nk = 0;
      double last = 0;
      for (int i = 0; i < NE; ++i) {
        double d = nk ? std::remainder(ang[i] - last, 2 * M_PI) * (180.0 / M_PI) : 1e9;
        // (an edge before a long one is kept too when skipping it would leave more than `turn` to the long edge's predecessor)
        if (len[i] >= long_edge || std::fabs(d) >= turn) { keep[nk++] = i; last = ang[i]; }
      }
      if (nk <= kCoarseEdges) break;
    }
    if (nk == 0 || nk > kCoarseEdges) { nk = 0; for (int i = 0; i < NE && nk < kCoarseEdges; ++i) keep[nk++] = i; }  // (NE <= kCoarseEdges only)
    for (int k = 0; k < kCoarseEdges; ++k) {
      const int i = keep[k < nk ? k : 0];
      pr.c_ax[k] = (T)v[i][0]; pr.c_ay[k] = (T)v[i][1]; pr.c_nx[k] = (T)nx[i]; pr.c_ny[k] = (T)ny[i];
    }
  }
  pr.tz_lo = 1; pr.tz_hi = 0;
  for (int k = 0; k < 2; ++k) { pr.t_ax[k] = pr.t_ay[k] = 0; pr.t_nx[k] = pr.t_ny[k] = 0; }
  if (quad_edges) {
    const int e0 = quad_edges[0], e1 = quad_edges[1];
    double lo = std::fmax(std::fmin(v[e0][1], v[(e0 + 1) % NE][1]), std::fmin(v[e1][1], v[(e1 + 1) % NE][1]));
    double hi = std::fmin(std::fmax(v[e0][1], v[(e0 + 1) % NE][1]), std::fmax(v[e1][1], v[(e1 + 1) % NE][1]));
    const double eps = (hi - lo) * (1.0 - shrink);
    lo += eps; hi -= eps;
    // corners of the region: where the two edge lines meet v = lo and v = hi; all four must lie inside every edge line
    bool ok = hi > lo;
    for (int k = 0; k < 2 && ok; ++k) {
      const int e = quad_edges[k];
      for (int j = 0; j < 2 && ok; ++j) {
        const double vv = j ? hi : lo;
        if (std::fabs(nx[e]) < 1e-12) { ok = false; break; }
        const double uu = v[e][0] - (vv - v[e][1]) * ny[e] / nx[e];  // on the edge's line
        for (int i = 0; i < NE; ++i) ok = ok && (uu - v[i][0]) * nx[i] + (vv - v[i][1]) * ny[i] <= 1e-12;
      }
    }
    if (!ok) {  // no usable quadrilateral: the ellipse has to contain every vertex
      double so = 0;
      const double a0 = (double)pr.out_a, b0 = (double)pr.out_b, c = (double)pr.in_c;
      for (int i = 0; i < NE; ++i) {
        double du = v[i][0] / a0, dv = (v[i][1] - c) / b0;
        so = std::fmax(so, std::sqrt(du * du + dv * dv));
      }
      if (so > 1) { pr.out_a = (T)(a0 * so / shrink); pr.out_b = (T)(b0 * so / shrink); }
    }
    if (ok) {
      pr.out_lo = (T)std::fmin(std::fmin(v[e0][1], v[(e0 + 1) % NE][1]), std::fmin(v[e1][1], v[(e1 + 1) % NE][1]));
      pr.tz_lo = (T)lo; pr.tz_hi = (T)hi;
      for (int k = 0; k < 2; ++k) {
        const int e = quad_edges[k];
        pr.t_ax[k] = (T)v[e][0]; pr.t_ay[k] = (T)v[e][1]; pr.t_nx[k] = (T)nx[e]; pr.t_ny[k] = (T)ny[e];
      }
    }
  }
}

struct HostScene {  // double-precision master copy; Scene<T> is derived from it
  double racket_v[kRacketEdges][2], goal_v[kGoalEdges][2], racket_half_x, racket_inertia[3], com_z, swing_q[4], swing_off[3];
};
static void build_host_scene(const Params &p, HostScene &h) {
  double s = p.racket_scale, ymin = 1e30, ymax = -1e30, zmin = 1e30, zmax = -1e30;
  for (int i = 0; i < kRacketEdges; ++i) {
    double y = TB_RACKET_OUTLINE[i][0], z = TB_RACKET_OUTLINE[i][1];
    ymin = std::fmin(ymin, y); ymax = std::fmax(ymax, y); zmin = std::fmin(zmin, z); zmax = std::fmax(zmax, z);
    h.racket_v[i][0] = s * y;                      // COM frame = link frame shifted by the inertial origin
    h.racket_v[i][1] = s * (z - TB_RACKET_COM_Z);  // racket.urdf:18-19
  }
  h.racket_half_x = s * TB_RACKET_HALF_X;
  h.com_z = s * TB_RACKET_COM_Z;
  // Bullet recomputes the inertia from the compound's AABB (margin included) as a solid box [R]
  double m = p.hull_margin, ex = s * 2 * TB_RACKET_HALF_X + 2 * m, ey = s * (ymax - ymin) + 2 * m, ez = s * (zmax - zmin) + 2 * m;
  h.racket_inertia[0] = TB_RACKET_MASS / 12.0 * (ey * ey + ez * ez);
  h.racket_inertia[1] = TB_RACKET_MASS / 12.0 * (ex * ex + ez * ez);
  h.racket_inertia[2] = TB_RACKET_MASS / 12.0 * (ex * ex + ey * ey);
  // goal: PyBullet turns the URDF cylinder into a 32-gon prism, vertices (R sin, R cos) clockwise; store CCW
  for (int i = 0; i < kGoalEdges; ++i) {
    double th = 6.283185307179586476925286766559 * ((double)(kGoalEdges - 1 - i) / kGoalEdges);
    h.goal_v[i][0] = TB_GOAL_RADIUS * std::sin(th);
    h.goal_v[i][1] = TB_GOAL_RADIUS * std::cos(th);
  }
  // swing spawn: rpy (0, 0.5, 0) (swingracket_env.py:165) -> q = (0, sin .25, 0, cos .25); COM = base + R (0,0,com_z)
  double q[4] = {0, std::sin(0.25), 0, std::cos(0.25)};
  for (int i = 0; i < 4; ++i) h.swing_q[i] = q[i];
  double x = q[0], y = q[1], z = q[2], w = q[3];
  h.swing_off[0] = 2 * (x * z + y * w) * h.com_z;
  h.swing_off[1] = 2 * (y * z - x * w) * h.com_z;
  h.swing_off[2] = (1 - 2 * (x * x + y * y)) * h.com_z;
}
template <typename T> static void build_scene(const Params &p, Scene<T> &sc) {
  HostScene h;
  build_host_scene(p, h);
  std::memset(&sc, 0, sizeof sc);
  sc.dt = (T)p.dt; sc.gravity_z = (T)p.gravity_z; sc.lin_damping = (T)p.lin_damping; sc.ang_damping = (T)p.ang_damping;
  sc.max_coord_vel = (T)p.max_coord_vel;
  sc.rest_racket = (T)p.rest_ball_racket; sc.rest_court = (T)p.rest_ball_court; sc.rest_goal = (T)p.rest_ball_goal;
  sc.mu_racket = (T)p.fric_ball_racket; sc.mu_court = (T)p.fric_ball_court; sc.mu_goal = (T)p.fric_ball_goal;
  sc.erp = (T)p.contact_erp; sc.slop = (T)p.linear_slop; sc.rest_vel_threshold = (T)p.rest_vel_threshold;
  sc.solver_residual = (T)p.solver_residual; sc.contact_threshold = (T)p.contact_threshold;
  sc.hull_margin = (T)p.hull_margin; sc.box_margin = (T)p.box_margin; sc.gyro = (T)p.gyro_term;
  sc.pid_kp = (T)p.pid_kp; sc.pid_ki = (T)p.pid_ki; sc.pid_kd = (T)p.pid_kd; sc.pid_lim = (T)p.pid_max_force;
  sc.pid_bias_z = (T)p.pid_bias_z; sc.pid_hit_z = (T)p.pid_hit_z;
  sc.iters = (int)p.solver_iterations;
  sc.shoot_start = (int)p.shoot_start; sc.shoot_frames = (int)p.shoot_frames;
  sc.racket_court = p.racket_court_contact != 0; sc.rest_racket_court = (T)p.rest_racket_court; sc.mu_racket_court = (T)p.fric_racket_court;
  {
    T v = (T)p.max_coord_vel;
    unsigned long long bits = 0;
    std::memcpy(&bits, &v, sizeof v);
    sc.vmax_hi = sizeof(T) == 8 ? (unsigned)(bits >> 32) : (unsigned)bits;
  }
  sc.ball_r = (T)TB_BALL_RADIUS;
  sc.ball_inv_m = (T)(1.0 / TB_BALL_MASS);
  sc.ball_inv_i = (T)(1.0 / (0.4 * TB_BALL_MASS * TB_BALL_RADIUS * TB_BALL_RADIUS));  // sphere inertia recomputed [R]
  sc.racket_inv_m = (T)(1.0 / TB_RACKET_MASS);
  for (int i = 0; i < 3; ++i) { sc.racket_i[i] = (T)h.racket_inertia[i]; sc.racket_inv_i[i] = (T)(1.0 / h.racket_inertia[i]); }
  sc.com_z = (T)h.com_z;
  for (int i = 0; i < 4; ++i) sc.swing_q[i] = (T)h.swing_q[i];
  for (int i = 0; i < 3; ++i) sc.swing_off[i] = (T)h.swing_off[i];
  sc.floor_h[0] = (T)TB_FLOOR_HX; sc.floor_h[1] = (T)TB_FLOOR_HY; sc.floor_h[2] = (T)TB_FLOOR_HZ;
  sc.net_h[0] = (T)TB_NET_HX; sc.net_h[1] = (T)TB_NET_HY; sc.net_h[2] = (T)TB_NET_HZ;
  sc.goal_r = (T)TB_GOAL_RADIUS; sc.goal_hz = (T)TB_GOAL_HALF_Z;
  {
    // the racket's throat: the two long straight outline edges that run from the handle end up to the head (the edges
    // after vertex 0 and before the last vertex in the CCW outline, tb_scene_data.h)
    const int quad[2] = {0, kRacketEdges - 2};
    build_prism<T, kRacketEdges>(sc.racket, h.racket_v, h.racket_half_x, quad);
  }
  {
    double ay = 0, zlo = 1e30, zhi = -1e30;
    for (int i = 0; i < kRacketEdges; ++i) {
      ay = std::fmax(ay, std::fabs(h.racket_v[i][0]));
      zlo = std::fmin(zlo, h.racket_v[i][1]);
      zhi = std::fmax(zhi, h.racket_v[i][1]);
    }
    // rounded outward in T so the reject stays conservative after the conversion
    sc.racket_box[0] = (T)(ay * (1 + 1e-6)); sc.racket_box[1] = (T)(zlo - 1e-6); sc.racket_box[2] = (T)(zhi + 1e-6);
    sc.racket_obb[0] = (T)ay; sc.racket_obb[1] = (T)zlo; sc.racket_obb[2] = (T)zhi;
    double zm = std::fmax(std::fabs(zlo), std::fabs(zhi));
    sc.racket_obb_radius = (T)(std::sqrt(h.racket_half_x * h.racket_half_x + ay * ay + zm * zm) * (1 + 1e-6));
  }
  build_prism<T, kGoalEdges>(sc.goal, h.goal_v, TB_GOAL_HALF_Z, nullptr);
  {
    // fast-forward substep constants (ff_substep).  The three rejects are grown a little: they may only send a
    // substep into the exact tests for nothing, never past them.
    const double hack[3] = {-50.0, -2.0, -2.0};  // swingracket_env.py:135-141
    const double *I = h.racket_inertia;
    for (int i = 0; i < 3; ++i) {
      sc.ff_hack[i] = (T)(p.dt * hack[i] / TB_RACKET_MASS);
      sc.ff_gyro[i] = (T)(p.dt * p.gyro_term * (I[(i + 2) % 3] - I[(i + 1) % 3]) / I[i]);
    }
    sc.ff_dtg = (T)(p.dt * p.gravity_z);
    sc.ff_kl = (T)(p.dt * p.lin_damping);
    sc.ff_ka = (T)(p.dt * p.ang_damping);
    sc.ff_qx2 = (T)(0.25 * p.dt * p.dt);
    const double reach_r = TB_BALL_RADIUS + p.hull_margin + p.contact_threshold;
    const double reach_b = TB_BALL_RADIUS + p.box_margin + p.contact_threshold;
    const double grow = sizeof(T) == 8 ? 1e-9 : 1e-4;
    sc.ff_slab = (T)(h.racket_half_x + reach_r + grow);
    sc.ff_low_z = (T)(TB_FLOOR_HZ + p.contact_threshold + p.hull_margin + (double)sc.racket_obb_radius * (1 + 1e-6) + grow);
    sc.ff_ball_z = (T)(std::fmax(std::fmax(TB_FLOOR_HZ, TB_NET_HZ), TB_GOAL_HALF_Z) + std::fmax(reach_r, reach_b) + grow);
    auto hi_word = [](T v) {
      unsigned long long bits = 0;
      std::memcpy(&bits, &v, sizeof v);
      return sizeof(T) == 8 ? (unsigned)(bits >> 32) : (unsigned)bits;
    };
    sc.vmax2_hi = hi_word((T)(p.max_coord_vel * p.max_coord_vel));
    const double rr = (double)sc.racket.bound_radius + reach_r + grow, gr = TB_GOAL_RADIUS + reach_r + grow;
    sc.ffp_racket_r2 = (T)(rr * rr * (1 + 1e-6));
    sc.ffp_floor[0] = (T)(TB_FLOOR_HX + reach_b + grow); sc.ffp_floor[1] = (T)(TB_FLOOR_HY + reach_b + grow);
    sc.ffp_floor[2] = (T)(TB_FLOOR_HZ + reach_b + grow);
    sc.ffp_net[0] = (T)(TB_NET_HX + reach_b + grow); sc.ffp_net[1] = (T)(TB_NET_HY + reach_b + grow);
    sc.ffp_net[2] = (T)(TB_NET_HZ + reach_b + grow);
    sc.ffp_goal_z = (T)(TB_GOAL_HALF_Z + reach_r + grow);
    sc.ffp_goal_r2 = (T)(gr * gr * (1 + 1e-6));
    const double v9 = 0.9 * p.max_coord_vel;
    sc.ffp_a2 = (T)std::fmin(0.99 * 2.5e-3 / (0.25 * p.dt * p.dt), v9 * v9);
    sc.ffp_v2 = (T)(v9 * v9);
    sc.ffp_low = sc.floor_h[2] + sc.contact_threshold;  // formed in T like physics_step does
    sc.ffp_box[0] = (T)((double)sc.racket_box[0] + reach_r + grow); sc.ffp_box[1] = (T)((double)sc.racket_box[1] - reach_r - grow);
    sc.ffp_box[2] = (T)((double)sc.racket_box[2] + reach_r + grow);
    sc.ffp_rim = (T)(reach_r + grow);
    {
      // prism_outside_fast's ellipse must CONTAIN everything within `rim` of the containing ellipse E(a, b).  Growing both semi-
      // axes by rim is not enough (by the triangle inequality E(a + rim, b + rim) lies INSIDE the offset body, touching it on
      // the axes only): scale it by gamma = max over directions of (h_E + rim) / h_E', h = support function
      const double a = (double)sc.racket.out_a, b = (double)sc.racket.out_b, rim = (double)sc.ffp_rim;
      double gamma = 1.0;
      for (int k = 0; k <= 20000; ++k) {
        const double th = 1.5707963267948966 * k / 20000.0, c = std::cos(th), sn = std::sin(th);
        const double h = std::sqrt(a * a * c * c + b * b * sn * sn) + rim, hp = std::sqrt((a + rim) * (a + rim) * c * c + (b + rim) * (b + rim) * sn * sn);
        gamma = std::fmax(gamma, h / hp);
      }
      gamma *= 1.0 + 1e-6;  // (sampling of the maximum, conversion to T)
      sc.racket.out_inv_a = (T)(1.0 / (gamma * (a + rim)));
      sc.racket.out_inv_b = (T)(1.0 / (gamma * (b + rim)));
    }
    sc.ffl_inv_dt = (T)(1.0 / p.dt); sc.ffl_erp_dt = (T)(p.contact_erp / p.dt); sc.ffl_m = (T)TB_BALL_MASS;
    sc.ffl_jinv_t = (T)(1.0 / (1.0 / TB_BALL_MASS + TB_BALL_RADIUS * TB_BALL_RADIUS / (0.4 * TB_BALL_MASS * TB_BALL_RADIUS * TB_BALL_RADIUS)));
    sc.ffp_court[0] = sc.floor_h[0] + 1; sc.ffp_court[1] = sc.floor_h[1] + 1;
    sc.ffp_face[0] = (T)(TB_FLOOR_HX - p.box_margin - grow); sc.ffp_face[1] = (T)(TB_FLOOR_HY - p.box_margin - grow);
    sc.ffp_face[2] = (T)(TB_FLOOR_HZ - p.box_margin + grow);
  }
}

}  // namespace tb

// ================================================================================================ C ABI
using namespace tb;

static thread_local char g_err[512];
__attribute__((format(printf, 1, 2))) static int fail(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  std::vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return 1;
}
#define CU(call)                                                                          \
  do {                                                                                    \
    const cudaError_t e_ = (call);                                                        \
    if (e_ != cudaSuccess) return fail("%s failed: %s", #call, cudaGetErrorString(e_));  \
  } while (0)

// Device memory owned by a context: freed with it, and on the error paths that leave a buffer or a partly built group behind.
struct CudaFree { void operator()(void *p) const { cudaFree(p); } };
struct CudaFreeHost { void operator()(void *p) const { cudaFreeHost(p); } };
template <typename T> using DevPtr = std::unique_ptr<T, CudaFree>;
template <typename T> static cudaError_t dev_alloc(DevPtr<T> &p, size_t bytes) {
  void *raw = nullptr;
  const cudaError_t e = cudaMalloc(&raw, bytes);
  p.reset(static_cast<T *>(raw));
  return e;
}

// The groups allocated on first use.  Each is built in a local and moved into the context once all of it exists, so a call
// that fails part-way leaves the group absent and the next call builds it again.
struct EsBufs {               // per-env state of the ES rollout (see EsIO), from the first tb_es_begin*
  DevPtr<double> norm, n0, ret;
  DevPtr<float> hist, obs, term, rew, act;
  DevPtr<uint8_t> alive, done;
  DevPtr<unsigned> base;
  DevPtr<unsigned> stop;      // [N] see EsIO::stop
  DevPtr<double> master;      // [3, obs_dim] the generation's master normaliser (zeros for NULL)
  DevPtr<double> part;        // es_norm_partial_kernel's per-CTA moments
};
struct StagingBufs {          // device copies of the host-buffer entry points' arrays
  DevPtr<float> actions, obs, reward, term;
  DevPtr<uint8_t> done, events, mask;
};
struct SacActorBufs {         // tb_set_sac_actor / tb_set_sac_actors: the actors' images (see SacLayout)
  DevPtr<uint4> w2;           // [agents] W2, 128 KB each
  DevPtr<float> small;        // [agents] the other tensors
  int64_t cap = 0;            // images the buffers hold
  int64_t agents = 1;         // images the rollout uses: env i acts with image i / (N / agents)
};
struct SacBufs {              // tb_sac_begin: per-env staging between sac_kernel and the env step (see SacIO)
  DevPtr<float> cur, act, obs, term, rew;
  DevPtr<uint8_t> done;
  DevPtr<unsigned> base;
  DevPtr<uint8_t> pending;    // 1 from tb_sac_begin until a TB_SAC_VECNORM rollout with a training normaliser folds the reset
};
struct PolicyBufs {           // tb_set_policy / tb_set_policies
  DevPtr<float> params;       // [agents, tb_policy_floats(env_kind)] parameters
  DevPtr<float> act;          // [N, act_dim] clipped actions handed from policy_kernel to step_kernel
  int64_t params_cap = 0;     // floats params holds
  int64_t agents = 1;         // rows the rollout uses: env i acts with row i / (N / agents)
};
struct VecNormBufs {          // tb_set_vecnorm / tb_set_vecnorms (see VecNormIO)
  DevPtr<double> stats, ret, part;  // stats: [records][TB_VECNORM_WORDS(obs_dim)]
  DevPtr<float> raw;          // [N, obs_dim] raw observation handed from step_kernel to policy_kernel<.., true, ..>
  DevPtr<uint8_t> armed;
  int64_t stats_cap = 0, part_cap = 0;  // doubles stats and part hold
  int64_t records = 1;        // records attached: env i uses record i / (N / records)
};

struct tb_ctx {
  tb_config cfg;
  Params params;
  Scene<float> sc32;                         // the scene of the context's precision (rebuild)
  Scene<double> sc64;
  DevPtr<void> state;
  DevPtr<unsigned long long> stats;
  cudaStream_t own_stream = nullptr;
  StagingBufs staging;
  int64_t launches = 0;
  DevPtr<int> queue;                         // fast-forward work queue (env indices), num_envs entries
  DevPtr<int> queue_full, queue_ctl;
  DevPtr<unsigned long long> dq;             // the two dynamic queues of ff_kernel, dq_cap tagged slots each
  long long dq_cap = 0;
  DevPtr<unsigned> epoch;                    // device word, see StepIO
  DevPtr<unsigned long long> fault;          // device word, see StepIO
  std::unique_ptr<unsigned long long, CudaFreeHost> h_fault;  // the same word in mapped host memory (checked on entry of
                                                              // every call, no sync)
  unsigned long long *h_fault_dev = nullptr; // its device alias
  long long spin_limit = 0;                  // clock cycles, see StepIO (TB_FF_SPIN_LIMIT_MS, default 4000 ms)
  DevPtr<unsigned long long> queue_ctrs;     // two counter sets (kCtrWords each) used by alternate steps
  unsigned ff_grid = 0;                      // persistent grid of ff_kernel
  int ff_server_sm_stride = 0;               // see StepIO (set with the grid size, 0 = per-CTA roles)
  int step_resident = -1;                    // resident CTAs of step_kernel (its L2 prefetch distance)
  bool one_wave4 = false;                    // Tennisbot-v0: launch the 4-CTAs-per-SM build of step_kernel (see its MINB)
  int control_mode = TB_CONTROL_FORCE;
  DevPtr<void> pid;                          // controller memory, allocated by tb_set_control_mode(TB_CONTROL_PID)
  PolicyBufs policy;
  VecNormBufs vn;                            // the policy rollout's normaliser (tb_set_vecnorm), kept when detached
  tb_vecnorm vn_cfg{};                       // its configuration; vn_cfg.struct_size == 0: none attached
  SacActorBufs sac_actor;                   // SAC actor and ring (tb_set_sac_actor / tb_sac_begin / tb_sac_rollout)
  SacBufs sac;
  int sac_grid = 0;                          // persistent grid of sac_kernel: SMs
  // ES fitness rollout (tb_es_begin / tb_es_rollout); see EsIO
  int64_t es_individuals = 0;                // 0: no tb_es_begin yet
  DevPtr<float> es_w;                        // [floats][individuals], stream-ordered allocation
  int64_t es_w_cap = 0;                      // floats es_w holds
  EsBufs es;
  bool timing = false;                       // tb_set_kernel_timing
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  double ms_step = 0, ms_ff = 0;
  int64_t timed_steps = 0;

  // runs with the context's device current; the owners free the buffers after it, once the own stream has drained
  ~tb_ctx() {
    if (own_stream) { cudaStreamSynchronize(own_stream); cudaStreamDestroy(own_stream); }
    for (cudaEvent_t e : ev)
      if (e) cudaEventDestroy(e);
  }
};

struct DeviceGuard {
  int prev = -1;
  bool ok;
  explicit DeviceGuard(int dev) { ok = cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define GUARD(ctx)                                               \
  if (!(ctx)) return fail("context is NULL");                    \
  DeviceGuard guard_((ctx)->cfg.device);                         \
  if (!guard_.ok) return fail("cudaSetDevice failed")

template <int KIND> using Kind = std::integral_constant<int, KIND>;
// f(Kind<env_kind>()), or -1 for an unknown kind
template <typename F> static int with_kind(int env_kind, F &&f) {
  return env_kind == TB_ENV_SWING ? f(Kind<TB_ENV_SWING>()) : env_kind == TB_ENV_HIT ? f(Kind<TB_ENV_HIT>()) : -1;
}
// The one place a context's precision and env kind become the compile-time T and KIND of its kernels:
// f(Scene<T> &scene, T *state, Kind<KIND>()).
template <typename F> static int with_env(tb_ctx *c, F &&f) {
  if (c->cfg.precision == TB_F64)
    return with_kind(c->cfg.env_kind, [&](auto kind) { return f(c->sc64, static_cast<double *>(c->state.get()), kind); });
  return with_kind(c->cfg.env_kind, [&](auto kind) { return f(c->sc32, static_cast<float *>(c->state.get()), kind); });
}
// bytes of one state scalar
static size_t state_word(tb_ctx *c) { return with_env(c, [](auto &, auto *state, auto) { return (int)sizeof *state; }); }

// Every kernel launch of the library: plain, or with programmatic stream serialisation (pdl), counted and checked.
constexpr bool kPlain = false, kPdl = true;
template <typename... KArgs, typename... Args>
static int launch_smem(tb_ctx *c, bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                       Args &&...args) {
  if (pdl) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    CU(cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...));
  } else {
    kernel<<<grid, block, smem, stream>>>(std::forward<Args>(args)...);
  }
  c->launches++;
  CU(cudaGetLastError());
  return 0;
}
template <typename... KArgs, typename... Args>
static int launch(tb_ctx *c, bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args &&...args) {
  return launch_smem(c, pdl, kernel, grid, block, 0, stream, std::forward<Args>(args)...);
}

// A fast-forward launch of this context gave up on a wait (ff_give_up): its batch state is incomplete.  Sticky; every
// later call fails loudly instead of handing stale observations on.
static unsigned long long fault_word(const tb_ctx *c) { return *reinterpret_cast<volatile unsigned long long *>(c->h_fault.get()); }
static int check_fault(tb_ctx *c, const char *who) {
  const unsigned long long f = fault_word(c);
  if (!f) return 0;
  return fail("%s: an earlier fast-forward launch of this context timed out waiting on its work queues (code %llu); "
              "the batch state is incomplete - destroy the context", who, f);
}
// The scene of the context's precision and its ball_vz table, which is computed on the context's device (it must be current).
static int rebuild(tb_ctx *c) {
  return with_env(c, [c](auto &sc, auto *state, auto) {
    using T = std::remove_pointer_t<decltype(state)>;
    build_scene<T>(c->params, sc);
    DevPtr<T> d;
    CU(dev_alloc(d, kBallVzEntries * sizeof(T)));
    if (launch(c, kPlain, ball_vz_kernel<T>, 1, 1, nullptr, sc, d.get())) return 1;
    CU(cudaMemcpy(sc.ball_vz, d.get(), kBallVzEntries * sizeof(T), cudaMemcpyDeviceToHost));
    return 0;
  });
}
static unsigned grid_for(int64_t n, int block) { return (unsigned)((n + block - 1) / block); }
static StepIO make_io(tb_ctx *c) {
  StepIO io;
  std::memset(&io, 0, sizeof io);
  io.state = c->state.get(); io.n = c->cfg.num_envs; io.id_offset = c->cfg.env_id_offset; io.seed = c->cfg.seed;
  io.auto_reset = c->cfg.auto_reset; io.stats = c->stats.get(); io.k_steps = 1;
  io.pid = c->control_mode == TB_CONTROL_PID ? c->pid.get() : nullptr;
  return io;
}
// The env-step counter the policy noise and the ES history are keyed by (see StepIO::epoch).
static const unsigned *step_counter(tb_ctx *c) { return c->cfg.env_kind == TB_ENV_SWING ? c->epoch.get() : c->epoch.get() + 2; }

static int set_control_mode(tb_ctx *c, int mode) {
  if (mode != TB_CONTROL_FORCE && mode != TB_CONTROL_PID) return fail("tb_set_control_mode: unknown mode");
  if (mode == TB_CONTROL_PID && !c->pid) {
    const size_t bytes = (size_t)c->cfg.num_envs * 8 * state_word(c);
    DevPtr<void> pid;
    CU(dev_alloc(pid, bytes));
    CU(cudaMemset(pid.get(), 0, bytes));
    c->pid = std::move(pid);
  }
  c->control_mode = mode;
  return 0;
}

// ff_kernel is persistent: one CTA per resident slot (SMs x CTAs/SM from the occupancy calculator).
template <typename T> static int ff_grid_size(tb_ctx *c) {
  int per_sm = 0, sms = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ff_kernel<T>, kBlock, 0));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->cfg.device));
  int64_t resident = (int64_t)sms * (per_sm > 0 ? per_sm : 1);
  int64_t need = (c->cfg.num_envs + kBlock - 1) / kBlock;
  c->ff_grid = (unsigned)(need < resident ? need : resident);
  // server SMs every 12th: measured on B200 (1 Mi envs, f64) 2.46 ms per fast-forward launch, stride 8 2.59, 16 2.99,
  // per-CTA roles 2.60
  c->ff_server_sm_stride = need >= resident ? 12 : 0;
  return 0;
}
// CTAs of step_kernel that are resident at a time = how far ahead its L2 prefetch reaches.
template <typename T, int KIND> static int step_resident_ctas(tb_ctx *c) {
  int per_sm = 0, sms = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, step_kernel<T, KIND, false>, kBlock, 0));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->cfg.device));
  c->step_resident = sms * (per_sm > 0 ? per_sm : 1);
  if constexpr (KIND == TB_ENV_HIT) {  // see step_kernel's MINB
    int per_sm4 = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm4, step_kernel<T, TB_ENV_HIT, false, 4>, kBlock, 0));
    const int64_t grid = (c->cfg.num_envs + kBlock - 1) / kBlock;
    c->one_wave4 = per_sm4 > per_sm && grid > (int64_t)sms * per_sm && grid <= (int64_t)sms * per_sm4;
  }
  return 0;
}
static void fill_io(tb_ctx *c, StepIO &io) {
  io.queue = c->queue.get(); io.queue_full = c->queue_full.get(); io.queue_ctl = c->queue_ctl.get();
  io.fault = c->fault.get(); io.fault_host = c->h_fault_dev; io.spin_limit = c->spin_limit;
  io.server_sm_stride = c->ff_server_sm_stride;
  io.dq_full = c->dq.get(); io.dq_late = c->dq ? c->dq.get() + c->dq_cap : nullptr; io.dq_cap = c->dq_cap;
  io.epoch = c->epoch.get();  // (a slot written 2^32 steps ago with the same tag would have to survive untouched)
  io.queue_ctrs = c->queue_ctrs.get();
}
// One env step = step_kernel (+ ff_kernel for SwingRacket) on `stream`.
static int launch_step(tb_ctx *c, StepIO &io, cudaStream_t stream, bool stage = false) {
  fill_io(c, io);
  return with_env(c, [&](auto &sc, auto *state, auto kind) {
    using T = std::remove_pointer_t<decltype(state)>;
    const unsigned grid = grid_for(io.n, kBlock);
    if (c->timing) CU(cudaEventRecord(c->ev[0], stream));
    auto kernel = step_kernel<T, kind, true>;
    if (!stage) {
      if (c->step_resident < 0 && step_resident_ctas<T, kind>(c)) return 1;
      io.prefetch_ahead = c->step_resident;
      kernel = step_kernel<T, kind, false>;
      if constexpr (kind == TB_ENV_HIT) {
        if (c->one_wave4) { io.prefetch_ahead = 0; kernel = step_kernel<T, TB_ENV_HIT, false, 4>; }
      }
    }
    if (launch(c, kPdl, kernel, grid, kBlock, stream, sc, io)) return 1;
    if (c->timing) CU(cudaEventRecord(c->ev[1], stream));
    if constexpr (kind == TB_ENV_SWING) {
      if (!c->ff_grid && ff_grid_size<T>(c)) return 1;
      io.server_sm_stride = c->ff_server_sm_stride;
      if (launch(c, kPdl, ff_kernel<T>, c->ff_grid, kBlock, stream, sc, io)) return 1;
    }
    if (c->timing) {
      float a = 0, b = 0;
      CU(cudaEventRecord(c->ev[2], stream));
      CU(cudaEventSynchronize(c->ev[2]));
      CU(cudaEventElapsedTime(&a, c->ev[0], c->ev[1]));
      CU(cudaEventElapsedTime(&b, c->ev[1], c->ev[2]));
      c->ms_step += a; c->ms_ff += b; c->timed_steps++;
    }
    return 0;
  });
}
static int launch_reset(tb_ctx *c, const StepIO &io, const double *d_init, const uint8_t *d_mask, cudaStream_t stream) {
  return with_env(c, [&](auto &sc, auto *state, auto kind) {
    using T = std::remove_pointer_t<decltype(state)>;
    return launch(c, kPlain, reset_kernel<T, kind>, grid_for(io.n, kBlock), kBlock, stream, sc, io, d_init, d_mask);
  });
}

// CTAs of es_norm_partial_kernel and vecnorm_partial_kernel
static int64_t es_norm_blocks(int64_t n) { return (n + kBlock * kEsStatsPer - 1) / (kBlock * kEsStatsPer); }
// The normaliser's kernels: VecNormIO over the context's buffers, and f(VecNormIO, Kind<env_kind>())
static bool vecnorm_training(const tb_ctx *c) { return c->vn_cfg.struct_size && c->vn_cfg.training; }
static VecNormIO vecnorm_io(tb_ctx *c) {
  VecNormIO io;
  std::memset(&io, 0, sizeof io);
  io.stats = c->vn.stats.get(); io.ret = c->vn.ret.get(); io.part = c->vn.part.get(); io.armed = c->vn.armed.get();
  io.n = c->cfg.num_envs; io.gamma = c->vn_cfg.gamma; io.fold_obs = c->vn_cfg.training && c->vn_cfg.norm_obs;
  return io;
}
// Doubles of the partials buffer a pass over `records` records of num_envs / records envs each needs
static int64_t vecnorm_part_doubles(int64_t num_envs, int64_t records, int od) {
  return records * es_norm_blocks(num_envs / records) * (od + 1) * 3;
}
// One statistics pass (vecnorm_partial_kernel, and vecnorm_final_kernel when the context trains): the entry pass when
// io.reward is nullptr (copy obs to io.copy if set, fold it if *io.armed), else the step pass.  With A > 1 records, the
// segmented instances: still two launches, A es_norm_blocks(N / A) CTAs and A CTAs.
static int vecnorm_pass(tb_ctx *c, VecNormIO io, cudaStream_t s) {
  const int64_t records = c->vn.records;
  return with_kind(c->cfg.env_kind, [&](auto kind) {
    constexpr int O = Dims<kind>::obs;
    if (records == 1) {
      const int64_t blocks = es_norm_blocks(io.n);
      if (launch(c, kPlain, vecnorm_partial_kernel<O>, (unsigned)blocks, kBlock, s, io)) return 1;
      return vecnorm_training(c) ? launch(c, kPlain, vecnorm_final_kernel<O>, 1, kBlock, s, io, blocks) : 0;
    }
    io.n /= records;  // envs per record
    const int64_t blocks = es_norm_blocks(io.n);
    if (launch(c, kPlain, vecnorm_partial_kernel<O, true>, (unsigned)(records * blocks), kBlock, s, io)) return 1;
    return vecnorm_training(c) ? launch(c, kPlain, vecnorm_final_kernel<O, true>, (unsigned)records, kBlock, s, io, blocks) : 0;
  });
}
static int vecnorm_pass(tb_ctx *c, const float *obs, const float *reward, const uint8_t *done, cudaStream_t s) {
  VecNormIO io = vecnorm_io(c);
  io.obs = obs; io.reward = reward; io.done = done;
  io.copy = reward ? nullptr : c->vn.raw.get();
  return vecnorm_pass(c, io, s);
}

extern "C" {

const char *tb_last_error(void) { return g_err; }
int tb_abi_version(void) { return TB_ABI_VERSION; }
int tb_obs_dim(int kind) { return with_kind(kind, [](auto k) { return Dims<k>::obs; }); }
int tb_act_dim(int kind) { return with_kind(kind, [](auto k) { return Dims<k>::act; }); }
int tb_policy_floats(int kind) { return with_kind(kind, [](auto k) { return PolLayout<Dims<k>::obs, Dims<k>::act>::Floats; }); }
int tb_es_floats(int kind) { return with_kind(kind, [](auto k) { return EsLayout<Dims<k>::obs, Dims<k>::act>::Floats; }); }
int tb_sac_floats(int kind) { return with_kind(kind, [](auto k) { return SacLayout<Dims<k>::obs, Dims<k>::act>::Floats; }); }
int tb_num_params(void) { return kNumParams; }
const char *tb_param_name(int i) { return (i >= 0 && i < kNumParams) ? k_param_names[i] : nullptr; }

int tb_scene_constant(const char *name, int index, double *value) {
  if (!name || !value) return fail("tb_scene_constant: bad argument");
  Params p;
  params_default(p);
  HostScene h;
  build_host_scene(p, h);
#define SC(nm, v) if (std::strcmp(name, nm) == 0) { *value = (v); return 0; }
  SC("urdf_margin", TB_URDF_MARGIN) SC("ball_radius", TB_BALL_RADIUS) SC("ball_mass", TB_BALL_MASS)
  SC("racket_mass", TB_RACKET_MASS) SC("racket_com_z", TB_RACKET_COM_Z) SC("racket_half_x", TB_RACKET_HALF_X)
  SC("floor_hx", TB_FLOOR_HX) SC("floor_hy", TB_FLOOR_HY) SC("floor_hz", TB_FLOOR_HZ)
  SC("net_hx", TB_NET_HX) SC("net_hy", TB_NET_HY) SC("net_hz", TB_NET_HZ)
  SC("goal_radius", TB_GOAL_RADIUS) SC("goal_half_z", TB_GOAL_HALF_Z) SC("goal_sides", TB_GOAL_SIDES)
  SC("racket_outline_n", TB_RACKET_OUTLINE_N) SC("contact_threshold", p.contact_threshold)
#undef SC
  if (!std::strcmp(name, "racket_inertia") && index >= 0 && index < 3) { *value = h.racket_inertia[index]; return 0; }
  if (!std::strcmp(name, "racket_outline_y") && index >= 0 && index < kRacketEdges) { *value = TB_RACKET_OUTLINE[index][0]; return 0; }
  if (!std::strcmp(name, "racket_outline_z") && index >= 0 && index < kRacketEdges) { *value = TB_RACKET_OUTLINE[index][1]; return 0; }
  if (!std::strcmp(name, "goal_vertex_x") && index >= 0 && index < kGoalEdges) { *value = h.goal_v[index][0]; return 0; }
  if (!std::strcmp(name, "goal_vertex_y") && index >= 0 && index < kGoalEdges) { *value = h.goal_v[index][1]; return 0; }
  {  // regions of prism_inside_fast (COM frame), for the unit test that checks them against the outline
    static Scene<double> sd;  // (4 KB: not on the stack)
    build_scene<double>(p, sd);
    const double in_r[5] = {sd.racket.in_c, 1.0 / sd.racket.in_inv_a, 1.0 / sd.racket.in_inv_b, sd.racket.tz_lo, sd.racket.tz_hi};
    const double in_g[5] = {sd.goal.in_c, 1.0 / sd.goal.in_inv_a, 1.0 / sd.goal.in_inv_b, sd.goal.tz_lo, sd.goal.tz_hi};
    const double out_r[6] = {sd.racket.out_a, sd.racket.out_b, sd.racket.out_v, sd.racket.out_lo, sd.racket.out_inv_a, sd.racket.out_inv_b};
    if (!std::strcmp(name, "racket_outside") && index >= 0 && index < 6) { *value = out_r[index]; return 0; }
    if (!std::strcmp(name, "racket_rim")) { *value = sd.ffp_rim; return 0; }
    if (!std::strcmp(name, "racket_inside") && index >= 0 && index < 5) { *value = in_r[index]; return 0; }
    if (!std::strcmp(name, "goal_inside") && index >= 0 && index < 5) { *value = in_g[index]; return 0; }
    if (!std::strcmp(name, "racket_coarse_edge") && index >= 0 && index < 4 * kCoarseEdges) {  // (point u, v; outward normal u, v) per edge
      const double *t[4] = {sd.racket.c_ax, sd.racket.c_ay, sd.racket.c_nx, sd.racket.c_ny};
      *value = t[index & 3][index >> 2];
      return 0;
    }
    if (!std::strcmp(name, "racket_quad_edge") && index >= 0 && index < 8) {
      const double q[8] = {sd.racket.t_ax[0], sd.racket.t_ay[0], sd.racket.t_nx[0], sd.racket.t_ny[0], sd.racket.t_ax[1], sd.racket.t_ay[1], sd.racket.t_nx[1], sd.racket.t_ny[1]};
      *value = q[index];
      return 0;
    }
  }
  return fail("tb_scene_constant: unknown name or index '%s'", name);
}

int tb_create(const tb_config *cfg, tb_ctx **out) {
  if (!cfg || !out) return fail("tb_create: bad argument");
  if (cfg->struct_size != sizeof(tb_config)) return fail("tb_create: tb_config.struct_size mismatch");
  if (cfg->env_kind != TB_ENV_SWING && cfg->env_kind != TB_ENV_HIT) return fail("tb_create: unknown env_kind");
  if (cfg->precision != TB_F32 && cfg->precision != TB_F64) return fail("tb_create: unknown precision");
  if (cfg->num_envs <= 0 || cfg->num_envs > 0x7fffffffLL) return fail("tb_create: num_envs must be in [1, 2^31)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("tb_create: no CUDA device (this library has no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail("tb_create: device ordinal out of range");
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) return fail("tb_create: device is not sm_100 (library is built for sm_100a only)");
  DeviceGuard g(cfg->device);  // (declared first: the context's buffers are freed with its device current)
  if (!g.ok) return fail("tb_create: cudaSetDevice failed");
  std::unique_ptr<tb_ctx> c(new (std::nothrow) tb_ctx());
  if (!c) return fail("tb_create: out of memory");
  c->cfg = *cfg;
  params_default(c->params);
  if (rebuild(c.get())) return fail("tb_create: could not build the scene tables on the device");
  const int64_t n = cfg->num_envs;
  const size_t bytes = (size_t)n * kPacks * 4 * state_word(c.get());
  CU(dev_alloc(c->state, bytes));
  CU(dev_alloc(c->stats, TB_NUM_STATS * sizeof(unsigned long long)));
  CU(dev_alloc(c->queue_ctrs, 2 * kCtrWords * sizeof(unsigned long long)));
  if (cfg->env_kind == TB_ENV_SWING) {
    // every env is pushed to either dynamic queue at most kFfMaxVisits times per launch, + a ticket for every lane that may
    // end up waiting: ff_kernel's grid is at most ceil(n / 128) CTAs and never more than fit the device (<= 2048 CTAs of 128
    // threads on any sm_100 part)
    const long long ctas = (n + kBlock - 1) / kBlock;
    c->dq_cap = (long long)n * (kFfMaxVisits + 1) + (ctas < 2048 ? ctas : 2048) * kBlock;
    CU(dev_alloc(c->queue, (size_t)n * sizeof(int)));
    CU(dev_alloc(c->dq, (size_t)c->dq_cap * 2 * sizeof(unsigned long long)));
    CU(dev_alloc(c->queue_full, (size_t)n * sizeof(int)));
    CU(dev_alloc(c->queue_ctl, (size_t)n * sizeof(int)));
  }
  CU(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  const cudaStream_t s = c->own_stream;
  CU(cudaMemsetAsync(c->state.get(), 0, bytes, s));
  CU(cudaMemsetAsync(c->stats.get(), 0, TB_NUM_STATS * sizeof(unsigned long long), s));
  CU(cudaMemsetAsync(c->queue_ctrs.get(), 0, 2 * kCtrWords * sizeof(unsigned long long), s));
  CU(dev_alloc(c->fault, sizeof(unsigned long long)));
  CU(cudaMemsetAsync(c->fault.get(), 0, sizeof(unsigned long long), s));
  {
    void *h = nullptr;
    CU(cudaHostAlloc(&h, sizeof(unsigned long long), cudaHostAllocMapped));
    c->h_fault.reset(static_cast<unsigned long long *>(h));
  }
  *c->h_fault = 0;
  CU(cudaHostGetDevicePointer((void **)&c->h_fault_dev, c->h_fault.get(), 0));
  {
    const char *ms = std::getenv("TB_FF_SPIN_LIMIT_MS");
    double limit_ms = ms ? std::atof(ms) : 4000.0;
    if (!(limit_ms > 0)) limit_ms = 4000.0;
    c->spin_limit = (long long)(limit_ms * 1e-3 * (double)prop.clockRate * 1e3);  // clockRate is in kHz
  }
  CU(dev_alloc(c->epoch, 3 * sizeof(unsigned)));
  CU(cudaMemsetAsync(c->epoch.get(), 0, 3 * sizeof(unsigned), s));
  if (c->dq) CU(cudaMemsetAsync(c->dq.get(), 0, (size_t)c->dq_cap * 2 * sizeof(unsigned long long), s));  // tag 0 = no epoch
  // identity quaternion, episode = -1 so the first reset starts episode 0
  const size_t words = (size_t)n * TB_STATE_WORDS;
  std::unique_ptr<double[]> init(new (std::nothrow) double[words]());
  if (!init) return fail("tb_create: out of memory");
  for (size_t i = 0; i < (size_t)n; ++i) { init[i * TB_STATE_WORDS + TB_S_RACKET_QUAT + 3] = 1.0; init[i * TB_STATE_WORDS + TB_S_EPISODE] = -1.0; }
  DevPtr<double> d_init;
  CU(dev_alloc(d_init, words * sizeof(double)));
  CU(cudaMemcpyAsync(d_init.get(), init.get(), words * sizeof(double), cudaMemcpyHostToDevice, s));
  if (with_env(c.get(), [&](auto &, auto *state, auto) {
        using T = std::remove_pointer_t<decltype(state)>;
        return launch(c.get(), kPlain, set_state_kernel<T>, grid_for(n, 256), 256, s, state, n, d_init.get());
      }))
    return 1;
  CU(cudaStreamSynchronize(s));
  *out = c.release();
  return 0;
}

int tb_destroy(tb_ctx *c) {
  if (!c) return 0;
  DeviceGuard g(c->cfg.device);
  delete c;
  return 0;
}

int tb_set_param(tb_ctx *c, const char *name, double value) {
  if (!name) return fail("tb_set_param: bad argument");
  GUARD(c);
  double *slots = reinterpret_cast<double *>(&c->params);
  for (int i = 0; i < kNumParams; ++i)
    if (!std::strcmp(name, k_param_names[i])) {
      // envs whose ball velocity lives in the free-fall table (kStPristine) get it written out under the OLD parameters
      // first; a configuration call, so it simply waits for everything the device has in flight
      CU(cudaDeviceSynchronize());
      const int64_t n = c->cfg.num_envs;
      if (with_env(c, [&](auto &sc, auto *state, auto) {
            using T = std::remove_pointer_t<decltype(state)>;
            return launch(c, kPlain, materialise_kernel<T>, grid_for(n, 256), 256, c->own_stream, sc, state, n);
          }))
        return 1;
      CU(cudaStreamSynchronize(c->own_stream));
      slots[i] = value;
      if (rebuild(c)) return fail("tb_set_param: could not rebuild the scene tables on the device");
      return 0;
    }
  return fail("tb_set_param: unknown parameter '%s'", name);
}
int tb_set_control_mode(tb_ctx *c, int mode) {
  GUARD(c);
  return set_control_mode(c, mode);
}
int tb_get_param(tb_ctx *c, const char *name, double *value) {
  if (!c || !name || !value) return fail("tb_get_param: bad argument");
  const double *slots = reinterpret_cast<const double *>(&c->params);
  for (int i = 0; i < kNumParams; ++i)
    if (!std::strcmp(name, k_param_names[i])) { *value = slots[i]; return 0; }
  return fail("tb_get_param: unknown parameter '%s'", name);
}

static int reset_impl(tb_ctx *c, const double *d_init, const uint8_t *d_mask, float *d_obs, void *stream) {
  GUARD(c);
  if (check_fault(c, "tb_reset")) return 1;
  StepIO io = make_io(c);
  io.obs = d_obs;
  return launch_reset(c, io, d_init, d_mask, (cudaStream_t)stream);
}
// tb_reset / tb_reset_from with a normaliser in training: the reset envs' returns are zeroed, and a full reset arms the fold
static int vecnorm_reset(tb_ctx *c, const uint8_t *d_mask, void *stream) {
  if (!vecnorm_training(c)) return 0;
  return launch(c, kPlain, vecnorm_reset_kernel, grid_for(c->cfg.num_envs, kBlock), kBlock, (cudaStream_t)stream, vecnorm_io(c), d_mask);
}
int tb_reset(tb_ctx *c, const uint8_t *d_mask, float *d_obs, void *stream) {
  if (reset_impl(c, nullptr, d_mask, d_obs, stream)) return 1;
  return vecnorm_reset(c, d_mask, stream);
}
int tb_reset_from(tb_ctx *c, const double *d_init, const uint8_t *d_mask, float *d_obs, void *stream) {
  if (!d_init) return fail("tb_reset_from: d_init is NULL");
  if (reset_impl(c, d_init, d_mask, d_obs, stream)) return 1;
  return vecnorm_reset(c, d_mask, stream);
}

static int step_impl(tb_ctx *c, const float *d_actions, float *d_obs, float *d_reward, uint8_t *d_done,
                     float *d_terminal_obs, uint8_t *d_events, void *stream, bool stage) {
  GUARD(c);
  if (!d_actions || !d_obs || !d_reward || !d_done) return fail("tb_step: actions, obs, reward and done are required");
  if (check_fault(c, "tb_step")) return 1;
  StepIO io = make_io(c);
  io.actions = d_actions; io.obs = d_obs; io.reward = d_reward; io.done = d_done; io.term_obs = d_terminal_obs;
  io.events = d_events;
  return launch_step(c, io, (cudaStream_t)stream, stage);
}
int tb_step(tb_ctx *c, const float *d_actions, float *d_obs, float *d_reward, uint8_t *d_done, float *d_terminal_obs,
            uint8_t *d_events, void *stream) {
  return step_impl(c, d_actions, d_obs, d_reward, d_done, d_terminal_obs, d_events, stream, false);
}

int tb_rollout(tb_ctx *c, int action_mode, int k_steps, float *d_obs, float *d_reward_sum, int32_t *d_done_count, void *stream) {
  GUARD(c);
  if (action_mode != TB_ACT_RANDOM && !(action_mode == TB_ACT_TRACK && c->cfg.env_kind == TB_ENV_HIT))
    return fail("tb_rollout: unknown action mode (TB_ACT_TRACK is Tennisbot-v0's)");
  if (c->control_mode != TB_CONTROL_FORCE) return fail("tb_rollout: in-kernel random actions need TB_CONTROL_FORCE");
  if (k_steps < 0) return fail("tb_rollout: k_steps must be >= 0");
  StepIO io = make_io(c);
  io.k_steps = k_steps; io.action_mode = action_mode; io.obs = d_obs; io.reward_sum = d_reward_sum; io.done_count = d_done_count;
  return with_env(c, [&](auto &sc, auto *state, auto kind) {
    using T = std::remove_pointer_t<decltype(state)>;
    return launch(c, kPlain, rollout_kernel<T, kind>, grid_for(io.n, kBlock), kBlock, (cudaStream_t)stream, sc, io);
  });
}

// agents policy rows -> the library's buffer, grown when it holds fewer (cudaMalloc / cudaFree: not while capturing)
static int copy_policies(tb_ctx *c, const float *d_params, int64_t agents, cudaStream_t s) {
  const int64_t floats = agents * tb_policy_floats(c->cfg.env_kind);
  if (c->policy.params_cap < floats) {
    PolicyBufs p;
    CU(dev_alloc(p.params, (size_t)floats * sizeof(float)));
    if (c->policy.act) p.act = std::move(c->policy.act);
    else CU(dev_alloc(p.act, (size_t)c->cfg.num_envs * tb_act_dim(c->cfg.env_kind) * sizeof(float)));
    p.params_cap = floats;
    c->policy = std::move(p);
  }
  CU(cudaMemcpyAsync(c->policy.params.get(), d_params, (size_t)floats * sizeof(float), cudaMemcpyDeviceToDevice, s));
  c->policy.agents = agents;
  return 0;
}

int tb_set_policy(tb_ctx *c, const float *d_params, int64_t count, void *stream) {
  GUARD(c);
  const int64_t want = tb_policy_floats(c->cfg.env_kind);
  if (!d_params || count != want)
    return fail("tb_set_policy: expected tb_policy_floats(env_kind) = %lld floats in device memory, got %lld", (long long)want,
                (long long)count);
  return copy_policies(c, d_params, 1, (cudaStream_t)stream);
}

int tb_set_policies(tb_ctx *c, const float *d_params, int64_t agents, int64_t count, void *stream) {
  GUARD(c);
  const int64_t n = c->cfg.num_envs, floats = tb_policy_floats(c->cfg.env_kind);
  if (!d_params) return fail("tb_set_policies: d_params is NULL");
  if (agents < 1 || n % agents) return fail("tb_set_policies: agents must be >= 1 and divide num_envs = %lld, got %lld", (long long)n, (long long)agents);
  if (count != agents * floats)
    return fail("tb_set_policies: expected agents x tb_policy_floats(env_kind) = %lld x %lld floats, got %lld", (long long)agents,
                (long long)floats, (long long)count);
  if (check_fault(c, "tb_set_policies")) return 1;
  return copy_policies(c, d_params, agents, (cudaStream_t)stream);
}

int tb_policy_rollout_raw(tb_ctx *c, int k_steps, int deterministic, uint64_t noise_seed, float *d_obs, float *d_actions,
                          float *d_logp, float *d_value, float *d_reward, float *d_raw_reward, uint8_t *d_done, float *d_last_obs,
                          float *d_last_value, void *stream) {
  GUARD(c);
  if (!c->policy.params) return fail("tb_policy_rollout: no policy (tb_set_policy)");
  if (c->control_mode != TB_CONTROL_FORCE) return fail("tb_policy_rollout: the policy's actions are forces (TB_CONTROL_FORCE)");
  if (k_steps < 1 || !d_obs || !d_reward || !d_done || !d_last_obs) return fail("tb_policy_rollout: k_steps >= 1, obs, reward, done and last_obs are required");
  if (check_fault(c, "tb_policy_rollout")) return 1;
  const int64_t n = c->cfg.num_envs;
  const int od = tb_obs_dim(c->cfg.env_kind), ad = tb_act_dim(c->cfg.env_kind);
  // with a normaliser: policy_kernel<.., true> reads the raw observation from vn.raw (from d_last_obs after the last step)
  const bool vn = c->vn_cfg.struct_size != 0, train = vecnorm_training(c), pop = c->policy.agents > 1;
  if (vn && c->vn.records == 1 && pop)
    return fail("tb_policy_rollout: a normaliser (tb_set_vecnorm) keeps one record per context, so it cannot serve %lld agents "
                "(tb_set_policies); detach it or set one policy, or attach one record per agent (tb_set_vecnorms)",
                (long long)c->policy.agents);
  if (vn && c->vn.records != c->policy.agents)
    return fail("tb_policy_rollout: %lld policies (tb_set_policies) and %lld normaliser records (tb_set_vecnorms) differ; env i "
                "uses policy and record i / (N / agents), so the counts must be equal", (long long)c->policy.agents,
                (long long)c->vn.records);
  void (*kernel)(PolicyIO) = nullptr;
  with_kind(c->cfg.env_kind, [&](auto kind) {
    constexpr int O = Dims<kind>::obs, A = Dims<kind>::act;
    kernel = vn ? (pop ? policy_kernel<O, A, true, true> : policy_kernel<O, A, true, false>)
                : pop ? policy_kernel<O, A, false, true> : policy_kernel<O, A, false, false>;
    return 0;
  });
  cudaStream_t s = (cudaStream_t)stream;
  PolicyIO pio;
  std::memset(&pio, 0, sizeof pio);
  pio.params = c->policy.params.get(); pio.n = n; pio.id_offset = c->cfg.env_id_offset; pio.seed = noise_seed; pio.deterministic = deterministic;
  pio.act_env = c->policy.act.get(); pio.tick = step_counter(c); pio.envs_per_agent = n / c->policy.agents;
  if (vn) {
    pio.vn_stats = c->vn.stats.get(); pio.vn_clip_obs = c->vn_cfg.clip_obs; pio.vn_clip_reward = c->vn_cfg.clip_reward;
    pio.vn_eps = c->vn_cfg.epsilon; pio.vn_norm_obs = c->vn_cfg.norm_obs; pio.vn_norm_reward = c->vn_cfg.norm_reward;
    if (vecnorm_pass(c, d_obs, nullptr, nullptr, s)) return 1;  // d_obs[0] -> vn.raw, folded when armed
  }
  const unsigned grid = grid_for(n, kBlock);
  for (int t = 0; t < k_steps; ++t) {
    pio.obs = vn ? c->vn.raw.get() : d_obs + (size_t)t * n * od;
    pio.act_raw = d_actions ? d_actions + (size_t)t * n * ad : nullptr;
    pio.logp = d_logp ? d_logp + (size_t)t * n : nullptr;
    pio.value = d_value ? d_value + (size_t)t * n : nullptr;
    if (vn) { pio.vn_obs = d_obs + (size_t)t * n * od; pio.vn_reward = t ? d_reward + (size_t)(t - 1) * n : nullptr; }
    if (launch(c, kPdl, kernel, dim3(grid, 2), kBlock, s, pio)) return 1;
    StepIO io = make_io(c);
    io.actions = c->policy.act.get();
    io.obs = t + 1 < k_steps ? (vn ? c->vn.raw.get() : d_obs + (size_t)(t + 1) * n * od) : d_last_obs;
    io.reward = d_reward + (size_t)t * n; io.done = d_done + (size_t)t * n;
    if (launch_step(c, io, s)) return 1;
    if (d_raw_reward)  // the step's reward before the next policy launch normalises it in place (a copy, not a launch)
      CU(cudaMemcpyAsync(d_raw_reward + (size_t)t * n, io.reward, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (train && vecnorm_pass(c, io.obs, io.reward, io.done, s)) return 1;
  }
  if (d_last_value || vn) {  // bootstrap value of the observation the rollout ends with; the last step's normalised reward
    pio.obs = d_last_obs; pio.act_raw = nullptr; pio.act_env = nullptr; pio.logp = nullptr; pio.value = d_last_value;
    pio.vn_obs = nullptr; pio.vn_reward = vn ? d_reward + (size_t)(k_steps - 1) * n : nullptr;
    if (launch(c, kPdl, kernel, dim3(grid, 2), kBlock, s, pio)) return 1;
  }
  return 0;
}

int tb_policy_rollout(tb_ctx *c, int k_steps, int deterministic, uint64_t noise_seed, float *d_obs, float *d_actions, float *d_logp,
                      float *d_value, float *d_reward, uint8_t *d_done, float *d_last_obs, float *d_last_value, void *stream) {
  return tb_policy_rollout_raw(c, k_steps, deterministic, noise_seed, d_obs, d_actions, d_logp, d_value, d_reward, nullptr, d_done,
                               d_last_obs, d_last_value, stream);
}

// tb_set_vecnorm (who = "tb_set_vecnorm", agents = 1) and tb_set_vecnorms: `agents` records of one configuration
static int set_vecnorms(tb_ctx *c, const char *who, const tb_vecnorm *cfg, int64_t agents, const double *d_stats, void *stream) {
  GUARD(c);
  if (check_fault(c, who)) return 1;
  if (!cfg) { c->vn_cfg = tb_vecnorm{}; return 0; }
  const int64_t n = c->cfg.num_envs;
  if (agents < 1 || n % agents) return fail("%s: agents must be >= 1 and divide num_envs = %lld, got %lld", who, (long long)n, (long long)agents);
  if (cfg->struct_size != sizeof(tb_vecnorm)) return fail("%s: tb_vecnorm.struct_size mismatch", who);
  if (!(std::isfinite(cfg->clip_obs) && cfg->clip_obs > 0) || !(std::isfinite(cfg->clip_reward) && cfg->clip_reward > 0))
    return fail("%s: clip_obs and clip_reward must be finite and above 0", who);
  if (!(cfg->gamma >= 0 && cfg->gamma <= 1)) return fail("%s: gamma must be in [0, 1]", who);
  if (!(std::isfinite(cfg->epsilon) && cfg->epsilon > 0)) return fail("%s: epsilon must be finite and above 0", who);
  const int od = tb_obs_dim(c->cfg.env_kind), words = TB_VECNORM_WORDS(od);
  const bool rows = std::strcmp(who, "tb_set_vecnorm") != 0;  // tb_set_vecnorms' messages name the row
  cudaStream_t s = (cudaStream_t)stream;
  if (d_stats) {  // the records are read on the device: copy them back and check them first (synchronises `stream`)
    std::vector<double> h((size_t)(agents * words));
    CU(cudaMemcpyAsync(h.data(), d_stats, h.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    for (int64_t r = 0; r < agents; ++r)
      for (int i = 0; i < words; ++i) {
        const double v = h[(size_t)(r * words + i)];
        const bool count = i == 2 * od || i == 2 * od + 3, var = (i >= od && i < 2 * od) || i == 2 * od + 2;
        if (!std::isfinite(v) || (count && !(v > 0)) || (var && v < 0)) {
          if (rows)
            return fail("%s: stats[%lld][%d] = %g: counts must be above 0, variances at least 0, every entry finite", who,
                        (long long)r, i, v);
          return fail("%s: stats[%d] = %g: counts must be above 0, variances at least 0, every entry finite", who, i, v);
        }
      }
  }
  if (!c->vn.ret) {
    VecNormBufs b;
    CU(dev_alloc(b.ret, (size_t)n * sizeof(double)));
    CU(dev_alloc(b.raw, (size_t)n * od * sizeof(float)));
    CU(dev_alloc(b.armed, 1));
    c->vn = std::move(b);
  }
  // records and partials grow to the largest call (cudaMalloc / cudaFree: not while capturing)
  const int64_t stats_need = agents * words, part_need = vecnorm_part_doubles(n, agents, od);
  if (c->vn.stats_cap < stats_need) {
    DevPtr<double> p;
    CU(dev_alloc(p, (size_t)stats_need * sizeof(double)));
    c->vn.stats = std::move(p);
    c->vn.stats_cap = stats_need;
  }
  if (c->vn.part_cap < part_need) {
    DevPtr<double> p;
    CU(dev_alloc(p, (size_t)part_need * sizeof(double)));
    c->vn.part = std::move(p);
    c->vn.part_cap = part_need;
  }
  c->vn_cfg = *cfg;
  c->vn.records = agents;
  return with_kind(c->cfg.env_kind, [&](auto kind) {
    constexpr int O = Dims<kind>::obs;
    if (agents == 1)
      return launch(c, kPlain, vecnorm_init_kernel<O>, grid_for(n, kBlock), kBlock, s, vecnorm_io(c), d_stats);
    return launch(c, kPlain, vecnorm_init_records_kernel<O>, grid_for(std::max<int64_t>(n, stats_need), kBlock), kBlock, s,
                  vecnorm_io(c), d_stats, agents);
  });
}

int tb_set_vecnorm(tb_ctx *c, const tb_vecnorm *cfg, const double *d_stats, void *stream) {
  return set_vecnorms(c, "tb_set_vecnorm", cfg, 1, d_stats, stream);
}

int tb_set_vecnorms(tb_ctx *c, const tb_vecnorm *cfg, int64_t agents, const double *d_stats, void *stream) {
  return set_vecnorms(c, "tb_set_vecnorms", cfg, agents, d_stats, stream);
}

int tb_get_vecnorm(tb_ctx *c, double *d_stats, void *stream) {
  GUARD(c);
  if (!c->vn_cfg.struct_size) return fail("tb_get_vecnorm: no normaliser attached (tb_set_vecnorm)");
  if (c->vn.records != 1)
    return fail("tb_get_vecnorm: %lld records are attached; read them with tb_get_vecnorms", (long long)c->vn.records);
  if (!d_stats) return fail("tb_get_vecnorm: d_stats is NULL");
  const size_t bytes = TB_VECNORM_WORDS(tb_obs_dim(c->cfg.env_kind)) * sizeof(double);
  CU(cudaMemcpyAsync(d_stats, c->vn.stats.get(), bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int tb_get_vecnorms(tb_ctx *c, double *d_stats, int64_t agents, void *stream) {
  GUARD(c);
  if (!c->vn_cfg.struct_size) return fail("tb_get_vecnorms: no normaliser attached (tb_set_vecnorms)");
  if (agents != c->vn.records)
    return fail("tb_get_vecnorms: %lld records are attached, got agents = %lld", (long long)c->vn.records, (long long)agents);
  if (!d_stats) return fail("tb_get_vecnorms: d_stats is NULL");
  const size_t bytes = (size_t)agents * TB_VECNORM_WORDS(tb_obs_dim(c->cfg.env_kind)) * sizeof(double);
  CU(cudaMemcpyAsync(d_stats, c->vn.stats.get(), bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int tb_vecnorm_device_ptr(tb_ctx *c, double **d_records, int64_t *agents) {
  if (!c || !d_records || !agents) return fail("tb_vecnorm_device_ptr: bad argument");
  if (!c->vn_cfg.struct_size) return fail("tb_vecnorm_device_ptr: no normaliser attached (tb_set_vecnorms)");
  *d_records = c->vn.stats.get();
  *agents = c->vn.records;
  return 0;
}

int tb_vecnorm_apply(tb_ctx *c, const float *d_in, int64_t rows, int what, float *d_out, void *stream) {
  GUARD(c);
  if (!c->vn_cfg.struct_size) return fail("tb_vecnorm_apply: no normaliser attached (tb_set_vecnorm)");
  if (c->vn.records != 1)
    return fail("tb_vecnorm_apply: %lld records are attached (tb_set_vecnorms); it applies one", (long long)c->vn.records);
  if (what != TB_VECNORM_OBS && what != TB_VECNORM_REWARD) return fail("tb_vecnorm_apply: unknown what %d", what);
  const int od = tb_obs_dim(c->cfg.env_kind), width = what == TB_VECNORM_OBS ? od : 1;
  if (rows < 0 || rows > (int64_t)INT32_MAX * kBlock / width)  // (one thread per float, a grid of at most 2^31 - 1 CTAs)
    return fail("tb_vecnorm_apply: rows must be in 0 .. %lld, got %lld", (long long)((int64_t)INT32_MAX * kBlock / width),
                (long long)rows);
  if (rows > 0 && (!d_in || !d_out)) return fail("tb_vecnorm_apply: d_in and d_out are required");  // (an empty tensor's is NULL)
  if (check_fault(c, "tb_vecnorm_apply")) return 1;
  const tb_vecnorm &v = c->vn_cfg;
  const bool obs = what == TB_VECNORM_OBS;
  const int64_t count = rows * width;
  const unsigned grid = std::max<unsigned>(1u, grid_for(count, kBlock));  // one launch, rows = 0 included
  return with_kind(c->cfg.env_kind, [&](auto kind) {
    return launch(c, kPlain, vecnorm_apply_kernel<Dims<kind>::obs>, grid, kBlock, (cudaStream_t)stream, (const double *)c->vn.stats.get(),
                  d_in, d_out, count, (int)!obs, obs ? v.norm_obs : v.norm_reward, obs ? v.clip_obs : v.clip_reward, v.epsilon);
  });
}

static EsIO es_io(tb_ctx *c) {
  EsIO io;
  std::memset(&io, 0, sizeof io);
  io.w = c->es_w.get(); io.n = c->cfg.num_envs; io.individuals = c->es_individuals;
  io.repeats = c->es_individuals ? (int)(c->cfg.num_envs / c->es_individuals) : 0;
  io.norm = c->es.norm.get(); io.n0 = c->es.n0.get(); io.hist = c->es.hist.get(); io.ret = c->es.ret.get();
  io.alive = c->es.alive.get(); io.stop = c->es.stop.get();
  io.tick = step_counter(c);
  io.base = c->es.base.get();
  io.obs = c->es.obs.get(); io.term = c->es.term.get(); io.reward = c->es.rew.get(); io.done = c->es.done.get();
  return io;
}


// The checks tb_es_begin and tb_es_begin_noise share once the context is current, then the per-env state (once per context)
// and room for the population in es_w.
static int es_prepare(tb_ctx *c, const char *who, int64_t individuals, int64_t floats, cudaStream_t s) {
  const int64_t n = c->cfg.num_envs, want = tb_es_floats(c->cfg.env_kind);
  if (floats != want)
    return fail("%s: expected tb_es_floats(env_kind) = %lld floats per individual, got %lld", who, (long long)want, (long long)floats);
  if (n % individuals) return fail("%s: individuals (%lld) must divide num_envs (%lld)", who, (long long)individuals, (long long)n);
  if (individuals * floats > 0xffffffffLL)
    return fail("%s: individuals x floats must be below 2^32 (es_kernel indexes the population with 32 bits)", who);
  if (c->control_mode != TB_CONTROL_FORCE) return fail("%s: the GatedCNN's actions are forces (TB_CONTROL_FORCE)", who);
  if (check_fault(c, who)) return 1;
  if (!c->es.norm) {
    const size_t od = tb_obs_dim(c->cfg.env_kind), ad = tb_act_dim(c->cfg.env_kind);
    EsBufs e;
    CU(dev_alloc(e.norm, 2 * od * n * sizeof(double)));
    CU(dev_alloc(e.n0, od * sizeof(double)));
    CU(dev_alloc(e.ret, n * sizeof(double)));
    CU(dev_alloc(e.hist, TB_ES_HISTORY * od * n * sizeof(float)));
    CU(dev_alloc(e.obs, od * n * sizeof(float)));
    CU(dev_alloc(e.term, od * n * sizeof(float)));
    CU(dev_alloc(e.rew, n * sizeof(float)));
    CU(dev_alloc(e.act, ad * n * sizeof(float)));
    CU(dev_alloc(e.alive, n));
    CU(dev_alloc(e.done, n));
    CU(dev_alloc(e.base, sizeof(unsigned)));
    CU(dev_alloc(e.stop, n * sizeof(unsigned)));
    CU(dev_alloc(e.master, 3 * od * sizeof(double)));
    CU(dev_alloc(e.part, es_norm_blocks(n) * 3 * od * sizeof(double)));
    c->es = std::move(e);
  }
  if (c->es_w_cap < individuals * floats) {  // stream-ordered: a larger population does not synchronise either
    c->es_w_cap = 0;
    if (c->es_w) CU(cudaFreeAsync(c->es_w.release(), s));
    void *w = nullptr;
    CU(cudaMallocAsync(&w, (size_t)(individuals * floats) * sizeof(float), s));
    c->es_w.reset(static_cast<float *>(w));
    c->es_w_cap = individuals * floats;
  }
  return 0;
}

// Once es_w holds the population: reset every env, seed the normalisers from the master (kept for tb_es_normalizer_stats).
static int es_start(tb_ctx *c, int64_t individuals, const double *d_normalizer, cudaStream_t s) {
  const int64_t n = c->cfg.num_envs;
  const size_t master_bytes = (size_t)3 * tb_obs_dim(c->cfg.env_kind) * sizeof(double);
  if (d_normalizer) CU(cudaMemcpyAsync(c->es.master.get(), d_normalizer, master_bytes, cudaMemcpyDeviceToDevice, s));
  else CU(cudaMemsetAsync(c->es.master.get(), 0, master_bytes, s));
  StepIO io = make_io(c);
  io.obs = c->es.obs.get();
  if (launch_reset(c, io, nullptr, nullptr, s)) return 1;
  CU(cudaMemsetAsync(c->es.done.get(), 0, (size_t)n, s));  // the reset observation is the step obs the first action's trace shows
  c->es_individuals = individuals;
  const EsIO eio = es_io(c);
  return with_kind(c->cfg.env_kind, [&](auto kind) {
    return launch(c, kPlain, es_begin_kernel<Dims<kind>::obs>, grid_for(n, kBlock), kBlock, s, eio, d_normalizer);
  });
}

int tb_es_begin(tb_ctx *c, const float *d_weights, int64_t individuals, int64_t floats, const double *d_normalizer, void *stream) {
  if (!d_weights) return fail("tb_es_begin: d_weights is NULL");
  if (individuals < 1) return fail("tb_es_begin: individuals must be >= 1");
  GUARD(c);
  cudaStream_t s = (cudaStream_t)stream;
  if (es_prepare(c, "tb_es_begin", individuals, floats, s)) return 1;
  if (launch(c, kPlain, es_transpose_kernel, dim3((unsigned)((individuals + 31) / 32), (unsigned)((floats + 31) / 32)), dim3(32, 8), s,
             d_weights, individuals, (int)floats, c->es_w.get()))
    return 1;
  return es_start(c, individuals, d_normalizer, s);
}

int tb_es_begin_noise(tb_ctx *c, const float *d_theta, int64_t individuals, int64_t floats, float sigma, uint64_t noise_seed,
                      uint32_t generation, const double *d_normalizer, void *stream) {
  if (!d_theta) return fail("tb_es_begin_noise: d_theta is NULL");
  if (individuals < 1) return fail("tb_es_begin_noise: individuals must be >= 1");
  if (individuals % 2) return fail("tb_es_begin_noise: individuals must be even (antithetic pairs)");
  if (!(sigma > 0.0f) || !std::isfinite(sigma)) return fail("tb_es_begin_noise: sigma must be a finite number above 0");
  GUARD(c);
  const int64_t repeats = individuals > 0 && c->cfg.num_envs % individuals == 0 ? c->cfg.num_envs / individuals : 0;
  if (repeats && c->cfg.env_id_offset % (2 * repeats))
    return fail("tb_es_begin_noise: env_id_offset (%lld) must be a multiple of 2 x repeats (%lld), so a shard holds whole "
                "antithetic pairs", (long long)c->cfg.env_id_offset, (long long)(2 * repeats));
  cudaStream_t s = (cudaStream_t)stream;
  if (es_prepare(c, "tb_es_begin_noise", individuals, floats, s)) return 1;
  const int64_t pairs = individuals / 2, j0 = c->cfg.env_id_offset / (2 * repeats);
  if (launch(c, kPlain, es_perturb_kernel, dim3(grid_for(pairs, kBlock), (unsigned)((floats + 3) / 4)), kBlock, s, d_theta, pairs,
             (int)floats, sigma, noise_seed, generation, j0, c->es_w.get()))
    return 1;
  return es_start(c, individuals, d_normalizer, s);
}

int tb_es_noise_combine(tb_ctx *c, const int64_t *d_dirs, const float *d_coef, int64_t count, uint64_t noise_seed, uint32_t generation,
                        float *d_out, void *stream) {
  if (count < 0) return fail("tb_es_noise_combine: count must be >= 0");
  if (count > 0 && (!d_dirs || !d_coef)) return fail("tb_es_noise_combine: d_dirs and d_coef are required when count > 0");
  if (!d_out) return fail("tb_es_noise_combine: d_out is NULL");
  GUARD(c);
  if (check_fault(c, "tb_es_noise_combine")) return 1;
  const int floats = tb_es_floats(c->cfg.env_kind);
  return launch(c, kPlain, es_combine_kernel, (unsigned)((floats + 3) / 4), kBlock, (cudaStream_t)stream, d_dirs, d_coef, count,
                noise_seed, generation, floats, d_out);
}

int tb_es_normalizer_stats(tb_ctx *c, double *d_out, void *stream) {
  if (!d_out) return fail("tb_es_normalizer_stats: d_out is NULL");
  GUARD(c);
  if (!c->es_individuals) return fail("tb_es_normalizer_stats: no generation (call tb_es_begin or tb_es_begin_noise first)");
  if (check_fault(c, "tb_es_normalizer_stats")) return 1;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t blocks = es_norm_blocks(c->cfg.num_envs);
  const EsIO eio = es_io(c);
  const int od = tb_obs_dim(c->cfg.env_kind);
  if (with_kind(c->cfg.env_kind, [&](auto kind) {
        return launch(c, kPlain, es_norm_partial_kernel<Dims<kind>::obs>, (unsigned)blocks, kBlock, s, eio, c->es.master.get(),
                      c->es.part.get());
      }))
    return 1;
  return launch(c, kPlain, es_norm_final_kernel, (unsigned)od, kBlock, s, c->es.part.get(), blocks, od, c->es.master.get(), d_out);
}

int tb_es_rollout(tb_ctx *c, int k_steps, double *d_return, uint8_t *d_alive, float *d_obs, float *d_actions, float *d_reward,
                  uint8_t *d_done, void *stream) {
  if (k_steps < 1) return fail("tb_es_rollout: k_steps must be >= 1");
  if (!d_return || !d_alive) return fail("tb_es_rollout: d_return and d_alive are required");
  GUARD(c);
  if (!c->es_individuals) return fail("tb_es_rollout: no population (call tb_es_begin first)");
  if (c->control_mode != TB_CONTROL_FORCE) return fail("tb_es_rollout: the GatedCNN's actions are forces (TB_CONTROL_FORCE)");
  if (check_fault(c, "tb_es_rollout")) return 1;
  const int64_t n = c->cfg.num_envs;
  const int od = tb_obs_dim(c->cfg.env_kind), ad = tb_act_dim(c->cfg.env_kind);
  void (*kernel)(EsIO) = nullptr;
  with_kind(c->cfg.env_kind, [&](auto kind) { kernel = es_kernel<Dims<kind>::obs, Dims<kind>::act>; return 0; });
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned grid = grid_for(n, kBlock);
  EsIO eio = es_io(c);
  for (int t = 0; t <= k_steps; ++t) {  // launch t folds step t - 1 (t > 0) and acts for step t (t < K)
    eio.fold = t > 0;
    eio.act = t < k_steps ? c->es.act.get() : nullptr;
    eio.obs_trace = d_obs ? d_obs + (size_t)t * n * od : nullptr;
    eio.act_trace = d_actions && t < k_steps ? d_actions + (size_t)t * n * ad : nullptr;
    eio.rew_trace = d_reward && t > 0 ? d_reward + (size_t)(t - 1) * n : nullptr;
    eio.done_trace = d_done && t > 0 ? d_done + (size_t)(t - 1) * n : nullptr;
    eio.ret_out = t == k_steps ? d_return : nullptr;
    eio.alive_out = t == k_steps ? d_alive : nullptr;
    if (launch(c, kPdl, kernel, grid, kBlock, s, eio)) return 1;
    if (t == k_steps) break;
    StepIO io = make_io(c);
    io.actions = c->es.act.get(); io.obs = c->es.obs.get(); io.reward = c->es.rew.get(); io.done = c->es.done.get();
    io.term_obs = c->es.term.get();
    if (launch_step(c, io, s)) return 1;
  }
  return 0;
}

// agents actor rows -> the library's images, one launch; the buffers grow when they hold fewer (cudaMalloc / cudaFree: not
// while capturing).  agents = 1 is tb_set_sac_actor's launch.
static int convert_sac_actors(tb_ctx *c, const float *d_params, int64_t agents, cudaStream_t s) {
  const int64_t floats = tb_sac_floats(c->cfg.env_kind), small = floats - TB_SAC_HIDDEN * TB_SAC_HIDDEN;
  if (c->sac_actor.cap < agents) {
    SacActorBufs b;
    CU(dev_alloc(b.w2, (size_t)agents * TB_SAC_HIDDEN * TB_SAC_HIDDEN * 2));
    CU(dev_alloc(b.small, (size_t)(agents * small) * sizeof(float)));
    b.cap = agents;
    c->sac_actor = std::move(b);
  }
  c->sac_actor.agents = agents;
  uint16_t *w2 = reinterpret_cast<uint16_t *>(c->sac_actor.w2.get());
  return with_kind(c->cfg.env_kind, [&](auto kind) {
    constexpr int OBS = Dims<kind>::obs, ACT = Dims<kind>::act;
    if (agents == 1)
      return launch(c, kPlain, sac_image_kernel<OBS, ACT, false>, grid_for(floats, 256), 256, s, d_params, w2, c->sac_actor.small.get());
    return launch(c, kPlain, sac_image_kernel<OBS, ACT, true>, (unsigned)(agents * kSacImageBlocks<OBS, ACT>), 256, s, d_params, w2,
                  c->sac_actor.small.get());
  });
}

int tb_set_sac_actor(tb_ctx *c, const float *d_params, int64_t count, void *stream) {
  GUARD(c);
  const int64_t want = tb_sac_floats(c->cfg.env_kind);
  if (!d_params || count != want)
    return fail("tb_set_sac_actor: expected tb_sac_floats(env_kind) = %lld floats in device memory, got %lld", (long long)want,
                (long long)count);
  return convert_sac_actors(c, d_params, 1, (cudaStream_t)stream);
}

int tb_set_sac_actors(tb_ctx *c, const float *d_params, int64_t agents, int64_t count, void *stream) {
  GUARD(c);
  const int64_t n = c->cfg.num_envs, floats = tb_sac_floats(c->cfg.env_kind);
  if (!d_params) return fail("tb_set_sac_actors: d_params is NULL");
  if (agents < 1 || n % agents)
    return fail("tb_set_sac_actors: agents must be >= 1 and divide num_envs = %lld, got %lld", (long long)n, (long long)agents);
  if (count != agents * floats)
    return fail("tb_set_sac_actors: expected agents x tb_sac_floats(env_kind) = %lld x %lld floats, got %lld", (long long)agents,
                (long long)floats, (long long)count);
  if (agents > 1 && (n / agents) % kBlock)
    return fail("tb_set_sac_actors: with agents > 1, envs per agent (%lld / %lld = %lld) must be a multiple of %d: a %d-env "
                "tile multiplies against one actor's W2 image in shared memory, and two 128 KB images do not fit beside the A "
                "tile", (long long)n, (long long)agents, (long long)(n / agents), kBlock, kBlock);
  if (check_fault(c, "tb_set_sac_actors")) return 1;
  return convert_sac_actors(c, d_params, agents, (cudaStream_t)stream);
}

int tb_sac_begin(tb_ctx *c, void *stream) {
  GUARD(c);
  if (c->control_mode != TB_CONTROL_FORCE) return fail("tb_sac_begin: the actor's actions are forces (TB_CONTROL_FORCE)");
  if (!c->cfg.auto_reset) return fail("tb_sac_begin: the ring needs auto_reset = 1 (a done env starts its next episode in the step)");
  if (check_fault(c, "tb_sac_begin")) return 1;
  const size_t n = c->cfg.num_envs, od = tb_obs_dim(c->cfg.env_kind), ad = tb_act_dim(c->cfg.env_kind);
  if (!c->sac.cur) {
    SacBufs b;
    CU(dev_alloc(b.cur, od * n * sizeof(float)));
    CU(dev_alloc(b.obs, od * n * sizeof(float)));
    CU(dev_alloc(b.term, od * n * sizeof(float)));
    CU(dev_alloc(b.act, ad * n * sizeof(float)));
    CU(dev_alloc(b.rew, n * sizeof(float)));
    CU(dev_alloc(b.done, n));
    CU(dev_alloc(b.base, sizeof(unsigned)));
    CU(dev_alloc(b.pending, 1));
    c->sac = std::move(b);
  }
  if (!c->sac_grid) {  // (configuration calls, kept out of tb_sac_rollout so that it can be captured in any capture mode)
    CU(cudaDeviceGetAttribute(&c->sac_grid, cudaDevAttrMultiProcessorCount, c->cfg.device));
    if (with_kind(c->cfg.env_kind, [&](auto kind) {
          constexpr int OBS = Dims<kind>::obs, ACT = Dims<kind>::act, smem = SacLayout<OBS, ACT>::Smem;
          CU(cudaFuncSetAttribute(sac_kernel<OBS, ACT, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
          CU(cudaFuncSetAttribute(sac_kernel<OBS, ACT, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
          CU(cudaFuncSetAttribute(sac_kernel<OBS, ACT, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
          return 0;
        }))
      return 1;
  }
  cudaStream_t s = (cudaStream_t)stream;
  StepIO io = make_io(c);
  io.obs = c->sac.cur.get();
  if (launch_reset(c, io, nullptr, nullptr, s)) return 1;
  CU(cudaMemcpyAsync(c->sac.base.get(), step_counter(c), sizeof(unsigned), cudaMemcpyDeviceToDevice, s));
  CU(cudaMemsetAsync(c->sac.pending.get(), 1, 1, s));  // the next TB_SAC_VECNORM rollout folds the reset (SB3's reset())
  return 0;
}

int tb_sac_rollout(tb_ctx *c, int k_steps, int mode, uint64_t noise_seed, const tb_sac_ring *ring, float *d_last_obs, void *stream) {
  if (k_steps < 1) return fail("tb_sac_rollout: k_steps must be >= 1");
  const bool norm = (mode & TB_SAC_VECNORM) != 0;
  const int flags = mode;
  mode &= ~TB_SAC_VECNORM;
  if (mode != TB_SAC_SAMPLE && mode != TB_SAC_MEAN && mode != TB_SAC_UNIFORM) return fail("tb_sac_rollout: unknown mode %d", flags);
  if (ring) {
    if (ring->struct_size != sizeof(tb_sac_ring)) return fail("tb_sac_rollout: tb_sac_ring.struct_size mismatch");
    if (ring->slots < 1) return fail("tb_sac_rollout: ring slots must be >= 1");
    if (!ring->obs || !ring->act || !ring->reward || !ring->next_obs || !ring->done)
      return fail("tb_sac_rollout: every ring array (obs, act, reward, next_obs, done) is required");
  }
  GUARD(c);
  if (c->control_mode != TB_CONTROL_FORCE) return fail("tb_sac_rollout: the actor's actions are forces (TB_CONTROL_FORCE)");
  if (!c->cfg.auto_reset) return fail("tb_sac_rollout: the ring needs auto_reset = 1");
  if (!c->sac.cur) return fail("tb_sac_rollout: no tb_sac_begin on this context");
  if (mode != TB_SAC_UNIFORM && !c->sac_actor.w2) return fail("tb_sac_rollout: no actor (tb_set_sac_actor)");
  if (norm && !c->vn_cfg.struct_size) return fail("tb_sac_rollout: TB_SAC_VECNORM needs a normaliser (tb_set_vecnorm)");
  if (norm && c->vn.records != 1)
    return fail("tb_sac_rollout: TB_SAC_VECNORM uses one record, and %lld are attached (tb_set_vecnorms)", (long long)c->vn.records);
  if (norm && c->sac_actor.agents > 1)
    return fail("tb_sac_rollout: TB_SAC_VECNORM normalises with one record, and %lld actors are set (tb_set_sac_actors); a "
                "population of SAC actors has no per-agent normaliser: set one actor (tb_set_sac_actor) or drop the flag",
                (long long)c->sac_actor.agents);
  if (check_fault(c, "tb_sac_rollout")) return 1;
  const bool pop = c->sac_actor.agents > 1;
  const bool train = norm && vecnorm_training(c);
  const int64_t n = c->cfg.num_envs;
  cudaStream_t s = (cudaStream_t)stream;
  SacIO sio;
  std::memset(&sio, 0, sizeof sio);
  sio.w2 = c->sac_actor.w2.get(); sio.small = c->sac_actor.small.get(); sio.n = n; sio.id_offset = c->cfg.env_id_offset; sio.seed = noise_seed;
  sio.tick = step_counter(c); sio.base = c->sac.base.get(); sio.mode = mode; sio.act_prev = c->sac.act.get(); sio.cur = c->sac.cur.get();
  sio.obs = c->sac.obs.get(); sio.term = c->sac.term.get(); sio.reward = c->sac.rew.get(); sio.done = c->sac.done.get();
  if (ring) {
    sio.slots = ring->slots; sio.r_obs = ring->obs; sio.r_act = ring->act; sio.r_reward = ring->reward; sio.r_next = ring->next_obs;
    sio.r_done = ring->done;
  }
  if (norm) {
    sio.vn_stats = c->vn.stats.get(); sio.vn_clip_obs = c->vn_cfg.clip_obs; sio.vn_eps = c->vn_cfg.epsilon;
    sio.vn_norm_obs = c->vn_cfg.norm_obs;
  }
  if (pop) {
    sio.image_w2 = TB_SAC_HIDDEN * TB_SAC_HIDDEN * 2 / 16; sio.image_small = tb_sac_floats(c->cfg.env_kind) - TB_SAC_HIDDEN * TB_SAC_HIDDEN;
    sio.per_agent = n / c->sac_actor.agents;
  }
  if (train) {  // the entry pass: while tb_sac_begin's reset is pending, zero the returns and fold the current observation
    VecNormIO vio = vecnorm_io(c);
    vio.obs = c->sac.cur.get(); vio.armed = c->sac.pending.get();
    if (launch(c, kPlain, vecnorm_sac_entry_kernel, grid_for(n, kBlock), kBlock, s, vio)) return 1;
    if (vecnorm_pass(c, vio, s)) return 1;
  }
  return with_kind(c->cfg.env_kind, [&](auto kind) {
    constexpr int OBS = Dims<kind>::obs, ACT = Dims<kind>::act;
    auto kernel = norm ? sac_kernel<OBS, ACT, true, false> : pop ? sac_kernel<OBS, ACT, false, true> : sac_kernel<OBS, ACT, false, false>;
    constexpr int smem = SacLayout<OBS, ACT>::Smem;
    const int64_t tiles = (n + kBlock - 1) / kBlock;
    for (int t = 0; t <= k_steps; ++t) {  // launch t folds step t - 1 (t > 0) and acts for step t (t < K)
      sio.fold = t > 0;
      sio.act = t < k_steps ? c->sac.act.get() : nullptr;
      sio.last_obs = t == k_steps ? d_last_obs : nullptr;
      const bool net = sio.act && mode != TB_SAC_UNIFORM;
      const unsigned grid = net ? (unsigned)std::min<int64_t>(tiles, c->sac_grid) : (unsigned)tiles;
      if (launch_smem(c, kPdl, kernel, grid, kBlock, net ? smem : 0, s, sio)) return 1;
      if (t == k_steps) break;
      StepIO io = make_io(c);
      io.actions = c->sac.act.get(); io.obs = c->sac.obs.get(); io.reward = c->sac.rew.get(); io.done = c->sac.done.get();
      io.term_obs = c->sac.term.get();
      if (launch_step(c, io, s)) return 1;
      if (train && vecnorm_pass(c, io.obs, io.reward, io.done, s)) return 1;  // fold the step's raw observation and reward
    }
    return 0;
  });
}

int tb_render(tb_ctx *c, const tb_camera *cam, const double *d_states, int64_t count, uint8_t *d_rgb, float *d_depth,
              uint8_t *d_body, void *stream) {
  GUARD(c);
  if (!cam || !d_states || !d_rgb) return fail("tb_render: cam, d_states and d_rgb are required");
  if (count < 1) return fail("tb_render: count must be >= 1, got %lld", (long long)count);
  if (cam->struct_size != sizeof(tb_camera)) return fail("tb_render: tb_camera.struct_size mismatch");
  const int w = cam->width, h = cam->height;
  if (w < 1 || w > TB_RENDER_MAX_SIZE || h < 1 || h > TB_RENDER_MAX_SIZE)
    return fail("tb_render: width and height must be in 1 .. %d, got %d x %d", TB_RENDER_MAX_SIZE, w, h);
  if (!(std::isfinite(cam->fov_y_deg) && cam->fov_y_deg > 0 && cam->fov_y_deg < 180))
    return fail("tb_render: fov_y_deg must be a finite number in (0, 180), got %g", cam->fov_y_deg);
  double f[3], r[3], u[3];
  for (int k = 0; k < 3; ++k) f[k] = cam->target[k] - cam->eye[k];
  const double fl = std::sqrt(f[0] * f[0] + f[1] * f[1] + f[2] * f[2]);
  if (!(fl > 0)) return fail("tb_render: eye and target coincide");
  for (int k = 0; k < 3; ++k) f[k] /= fl;
  const double *up = cam->up;
  r[0] = f[1] * up[2] - f[2] * up[1]; r[1] = f[2] * up[0] - f[0] * up[2]; r[2] = f[0] * up[1] - f[1] * up[0];
  const double rl = std::sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]), ul = std::sqrt(up[0] * up[0] + up[1] * up[1] + up[2] * up[2]);
  if (!(rl > 1e-9 * ul) || !(ul > 0)) return fail("tb_render: up is parallel to the view direction");
  for (int k = 0; k < 3; ++k) r[k] /= rl;
  u[0] = r[1] * f[2] - r[2] * f[1]; u[1] = r[2] * f[0] - r[0] * f[2]; u[2] = r[0] * f[1] - r[1] * f[0];
  const int64_t px4 = (int64_t)w * h * 4;  // bytes of the largest output per frame (depth; rgb is 3)
  if (count > INT64_MAX / px4) return fail("tb_render: %lld frames of %d x %d overflow int64", (long long)count, w, h);
  if (check_fault(c, "tb_render")) return 1;
  RenderIO io;
  std::memset(&io, 0, sizeof io);
  io.states = d_states; io.count = count; io.rgb = d_rgb; io.depth = d_depth; io.body = d_body; io.width = w; io.height = h;
  const double t = std::tan(cam->fov_y_deg * (M_PI / 360.0)), light[3] = TB_RENDER_LIGHT;
  const double ll = std::sqrt(light[0] * light[0] + light[1] * light[1] + light[2] * light[2]);
  for (int k = 0; k < 3; ++k) {
    io.eye[k] = cam->eye[k];
    io.f[k] = (float)f[k]; io.r[k] = (float)(r[k] * t * w / h); io.u[k] = (float)(u[k] * t);
    io.light[k] = (float)(light[k] / ll);
  }
  const double boxes[2][3] = {{TB_FLOOR_HX, TB_FLOOR_HY, TB_FLOOR_HZ}, {TB_NET_HX, TB_NET_HY, TB_NET_HZ}};
  for (int b = 0; b < 2; ++b)
    for (int k = 0; k < 3; ++k) {
      io.box_c[b][2 * k] = (float)(cam->eye[k] - boxes[b][k]);
      io.box_c[b][2 * k + 1] = (float)(-cam->eye[k] - boxes[b][k]);
    }
  const dim3 grid((unsigned)(((int64_t)w * h + kRenderBlock - 1) / kRenderBlock), (unsigned)std::min<int64_t>(count, 65535));
  return with_env(c, [&](auto &sc, auto *state, auto kind) {
    using T = std::remove_pointer_t<decltype(state)>;
    return launch(c, kPlain, render_kernel<T, kind>, grid, kRenderBlock, (cudaStream_t)stream, sc, io);
  });
}

int tb_trace_max_substeps(int env_kind) {
  return with_kind(env_kind, [](auto kind) { return kind == TB_ENV_SWING ? TB_TRACE_MAX_SUBSTEPS : 1; });
}

int tb_trace_step(tb_ctx *c, const double *d_states, const float *d_actions, int64_t count, int32_t max_substeps,
                  double *d_trace, uint8_t *d_bits, int32_t *d_substeps, float *d_reward, uint8_t *d_done,
                  uint8_t *d_events, void *stream) {
  GUARD(c);
  if (!d_states || !d_actions || !d_trace || !d_substeps)
    return fail("tb_trace_step: d_states, d_actions, d_trace and d_substeps are required");
  if (count < 1) return fail("tb_trace_step: count must be >= 1, got %lld", (long long)count);
  const int bound = tb_trace_max_substeps(c->cfg.env_kind);
  if (max_substeps < 1 || max_substeps > bound)
    return fail("tb_trace_step: max_substeps must be in 1 .. %d for this env, got %d", bound, (int)max_substeps);
  if (c->control_mode == TB_CONTROL_PID)
    return fail("tb_trace_step: TB_CONTROL_PID contexts cannot be traced (the controller memory is not part of the record)");
  const int64_t rec = (int64_t)max_substeps * TB_STATE_WORDS * (int64_t)sizeof(double);  // bytes of one record's trace
  if (count > INT64_MAX / rec) return fail("tb_trace_step: %lld records x %d substeps overflow int64", (long long)count, (int)max_substeps);
  if (check_fault(c, "tb_trace_step")) return 1;
  TraceIO io;
  std::memset(&io, 0, sizeof io);
  io.states = d_states; io.actions = d_actions; io.count = count; io.max_substeps = max_substeps; io.trace = d_trace;
  io.bits = d_bits; io.substeps = d_substeps; io.reward = d_reward; io.done = d_done; io.events = d_events;
  return with_env(c, [&](auto &sc, auto *state, auto kind) {
    using T = std::remove_pointer_t<decltype(state)>;
    return launch(c, kPlain, trace_kernel<T, kind>, grid_for(count, kTraceBlock), kTraceBlock, (cudaStream_t)stream, sc, io);
  });
}

int tb_get_state(tb_ctx *c, double *d_state, void *stream) {
  GUARD(c);
  if (!d_state) return fail("tb_get_state: d_state is NULL");
  const int64_t n = c->cfg.num_envs;
  return with_env(c, [&](auto &sc, auto *state, auto) {
    using T = std::remove_pointer_t<decltype(state)>;
    return launch(c, kPlain, get_state_kernel<T>, grid_for(n, 256), 256, (cudaStream_t)stream, sc, state, n, d_state);
  });
}
int tb_set_state(tb_ctx *c, const double *d_state, void *stream) {
  GUARD(c);
  if (!d_state) return fail("tb_set_state: d_state is NULL");
  const int64_t n = c->cfg.num_envs;
  return with_env(c, [&](auto &, auto *state, auto) {
    using T = std::remove_pointer_t<decltype(state)>;
    return launch(c, kPlain, set_state_kernel<T>, grid_for(n, 256), 256, (cudaStream_t)stream, state, n, d_state);
  });
}

int tb_stats_device_ptr(tb_ctx *c, int64_t **d_stats) {
  if (!c || !d_stats) return fail("tb_stats_device_ptr: bad argument");
  *d_stats = reinterpret_cast<int64_t *>(c->stats.get());
  return 0;
}
int tb_read_stats(tb_ctx *c, int64_t *h_stats, int clear, void *stream) {
  GUARD(c);
  if (!h_stats) return fail("tb_read_stats: h_stats is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  CU(cudaMemcpyAsync(h_stats, c->stats.get(), TB_NUM_STATS * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  if (clear) CU(cudaMemsetAsync(c->stats.get(), 0, TB_NUM_STATS * sizeof(int64_t), s));
  CU(cudaStreamSynchronize(s));
  return check_fault(c, "tb_read_stats");  // never seen; a wait in ff_kernel gave up (kSpinLimit) and left envs unfinished
}

static int ensure_staging(tb_ctx *c) {
  if (c->staging.actions) return 0;
  const size_t n = (size_t)c->cfg.num_envs, od = (size_t)tb_obs_dim(c->cfg.env_kind), ad = (size_t)tb_act_dim(c->cfg.env_kind);
  StagingBufs b;
  CU(dev_alloc(b.actions, n * ad * sizeof(float)));
  CU(dev_alloc(b.obs, n * od * sizeof(float)));
  CU(dev_alloc(b.term, n * od * sizeof(float)));
  CU(dev_alloc(b.reward, n * sizeof(float)));
  CU(dev_alloc(b.done, n));
  CU(dev_alloc(b.events, n));
  CU(dev_alloc(b.mask, n));
  c->staging = std::move(b);
  return 0;
}

int tb_reset_host(tb_ctx *c, const uint8_t *h_mask, float *h_obs) {
  GUARD(c);
  if (ensure_staging(c)) return 1;
  const StagingBufs &b = c->staging;
  size_t n = (size_t)c->cfg.num_envs, od = (size_t)tb_obs_dim(c->cfg.env_kind);
  cudaStream_t s = c->own_stream;
  if (h_mask) CU(cudaMemcpyAsync(b.mask.get(), h_mask, n, cudaMemcpyHostToDevice, s));
  if (reset_impl(c, nullptr, h_mask ? b.mask.get() : nullptr, b.obs.get(), s)) return 1;
  if (h_obs) CU(cudaMemcpyAsync(h_obs, b.obs.get(), n * od * sizeof(float), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

// Device alias of a host buffer the kernels can address directly (pinned + mapped memory under unified virtual
// addressing: cudaHostAlloc / torch pin_memory), or nullptr for pageable memory.
static void *mapped_alias(const void *h) {
  if (!h) return nullptr;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, h) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

int tb_step_host(tb_ctx *c, const float *h_actions, float *h_obs, float *h_reward, uint8_t *h_done, float *h_terminal_obs,
                 uint8_t *h_events) {
  GUARD(c);
  if (!h_actions || !h_obs || !h_reward || !h_done) return fail("tb_step_host: actions, obs, reward and done are required");
  if (check_fault(c, "tb_step_host")) return 1;
  // Transport: zero copy for pinned buffers, staging for pageable ones and for pinned ones when TB_HOST_MODE=staging.
  // Measured on the B200 box, 1 Mi SwingRacket envs, per step averaged over episodes: zero copy 0.92 ms, staging 1.24 ms
  // (a sliced copy-engine pipeline: 1.19 ms).  The link carries 50 GB/s either way alone and 80-92 GB/s both ways at once
  // (0.63-0.68 ms for a step's 55.6 MB through the copy engines); a zero-copy light step is 0.77 ms (72 GB/s,
  // tools/e2e_paths_probe.py).  Reading the actions in place and copying only the results down was measured too: 0.93 ms
  // per light step.  Staging stays selectable because eight GPUs stepping at once measured 2.91e9 env-steps/s staged
  // against 2.71e9 zero copy: the host side of PCIe saturates, which the library cannot observe.
  const char *mode = std::getenv("TB_HOST_MODE");
  const bool staging = mode && !std::strcmp(mode, "staging");
  if (mode && *mode && !staging && std::strcmp(mode, "zero_copy"))
    return fail("tb_step_host: TB_HOST_MODE='%s' is neither zero_copy nor staging", mode);
  size_t n = (size_t)c->cfg.num_envs, od = (size_t)tb_obs_dim(c->cfg.env_kind), ad = (size_t)tb_act_dim(c->cfg.env_kind);
  cudaStream_t s = c->own_stream;
  if (!staging) {
    // Pinned buffers: the kernels read the actions from and write the results to host memory themselves.  The
    // two PCIe directions then run concurrently and overlap with the compute, instead of H2D -> kernels -> D2H.
    const float *za = (const float *)mapped_alias(h_actions);
    float *zo = (float *)mapped_alias(h_obs), *zr = (float *)mapped_alias(h_reward);
    uint8_t *zd = (uint8_t *)mapped_alias(h_done);
    float *zt = (float *)mapped_alias(h_terminal_obs);
    uint8_t *ze = (uint8_t *)mapped_alias(h_events);
    if (za && zo && zr && zd && (zt || !h_terminal_obs) && (ze || !h_events)) {
      if (step_impl(c, za, zo, zr, zd, zt, ze, s, true)) return 1;
      CU(cudaStreamSynchronize(s));
      return check_fault(c, "tb_step_host");
    }
  }
  if (ensure_staging(c)) return 1;
  const StagingBufs &b = c->staging;
  CU(cudaMemcpyAsync(b.actions.get(), h_actions, n * ad * sizeof(float), cudaMemcpyHostToDevice, s));
  if (tb_step(c, b.actions.get(), b.obs.get(), b.reward.get(), b.done.get(), h_terminal_obs ? b.term.get() : nullptr,
              h_events ? b.events.get() : nullptr, s))
    return 1;
  CU(cudaMemcpyAsync(h_obs, b.obs.get(), n * od * sizeof(float), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(h_reward, b.reward.get(), n * sizeof(float), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(h_done, b.done.get(), n, cudaMemcpyDeviceToHost, s));
  if (h_terminal_obs) CU(cudaMemcpyAsync(h_terminal_obs, b.term.get(), n * od * sizeof(float), cudaMemcpyDeviceToHost, s));
  if (h_events) CU(cudaMemcpyAsync(h_events, b.events.get(), n, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return check_fault(c, "tb_step_host");
}

int tb_set_kernel_timing(tb_ctx *c, int enabled) {
  GUARD(c);
  if (enabled && !c->ev[0])
    for (int i = 0; i < 3; ++i) CU(cudaEventCreate(&c->ev[i]));
  c->timing = enabled != 0;
  return 0;
}
int tb_get_kernel_timing(tb_ctx *c, double *ms_step_kernel, double *ms_ff_kernel, int64_t *steps) {
  if (!c || !ms_step_kernel || !ms_ff_kernel || !steps) return fail("tb_get_kernel_timing: bad argument");
  *ms_step_kernel = c->ms_step; *ms_ff_kernel = c->ms_ff; *steps = c->timed_steps;
  c->ms_step = c->ms_ff = 0; c->timed_steps = 0;
  return 0;
}

int tb_ff_diagnostics(tb_ctx *c, int64_t *h_out) {
  GUARD(c);
  if (!h_out) return fail("tb_ff_diagnostics: h_out is NULL");
  CU(cudaDeviceSynchronize());
  unsigned long long h[2 * kCtrWords];
  CU(cudaMemcpy(h, c->queue_ctrs.get(), sizeof h, cudaMemcpyDeviceToHost));
  // the set of the most recent step that entered the fast-forward: the one whose round count is non-zero and whose
  // twin was zeroed since (both non-zero cannot happen: every step_kernel zeroes the next step's set)
  const unsigned long long *s = h[kDRounds] ? h : h + kCtrWords;
  h_out[0] = (int64_t)s[kDRounds]; h_out[1] = (int64_t)s[kDFullEnvs]; h_out[2] = (int64_t)s[kDPhase];
  for (int i = 3; i < 15; ++i) h_out[i] = 0;  // (ff_kernel stores kDFinish = 0)
  const unsigned long long fault = fault_word(c);
  h_out[15] = (int64_t)(fault ? fault : s[kCError]);
  return 0;
}

int tb_launch_count(tb_ctx *c, int64_t *launches) {
  if (!c || !launches) return fail("tb_launch_count: bad argument");
  *launches = c->launches;
  return 0;
}

}  // extern "C"
