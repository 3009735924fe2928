// libdekf_b200.so: __global__ wrappers + the extern "C" boundary declared in include/dekf_b200.h.
// sm_100a only.  No CPU fallback: every entry point needs a live CUDA context.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/dekf_b200.h"
#include "estimator_core.cuh"
#include "host_setup.hpp"
#include "box_team.cuh"
#include "foot_team.cuh"
#include "foot_window.cuh"
#include "box_window.cuh"

namespace dekf {

// ------------------------------------------------------------------------------------------------
// kernels: one thread per estimator instance
// ------------------------------------------------------------------------------------------------
constexpr int kBlock = 128;
// resident CTAs per SM the small per-tick kernels are compiled for (register cap = 65536 / (128 * MINB)):
// 65,536 instances are 512 CTAs; 4 CTAs/SM (592 slots) run them in ONE wave instead of 1.15 / 1.73 (profiles/r01_tick_kernels.md)
#ifndef DEKF_MINB_EKF
#define DEKF_MINB_EKF 4
#endif
#ifndef DEKF_MINB_ASM
#define DEKF_MINB_ASM 4
#endif
#ifndef DEKF_MINB_INCR
#define DEKF_MINB_INCR 2  // the sweep stage needs the full register file: 128 registers spill 944 B and lose (33 vs 26 us)
#endif

__global__ void k_zero_i32(int32_t *p) { *p = 0; }

// Indices of the instances whose vo_flag is set, in arbitrary order (warp-aggregated append; *count must be 0 at launch).
__global__ void __launch_bounds__(256) k_vo_compact(const uint8_t *__restrict__ flag, int n, int32_t *__restrict__ list,
                                                    int32_t *__restrict__ count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool f = i < n && flag[i] != 0;
  const unsigned m = __ballot_sync(0xffffffffu, f);
  if (m == 0) return;
  const int lane = threadIdx.x & 31;
  int base = 0;
  if (lane == __ffs(m) - 1) base = atomicAdd(count, __popc(m));
  base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
  if (f) list[base + __popc(m & ((1u << lane) - 1u))] = i;
}

// PART (see ekf_tick): EKF_ALL = one launch does the whole tick; with a VO-carrying tick of a large batch the tick is two launches,
// EKF_REPLAY over the compacted list of the instances that received a pose (thread t handles list[t], t < *count) and EKF_UPDATE
// over all instances.
template <typename T, int PART = EKF_ALL>
__global__ void __launch_bounds__(kBlock, DEKF_MINB_EKF) k_ekf(const EkfConst<T> c, const Dims dm, const Buffers<T> b, const Inputs in,
                                                const Outputs out, int k, int32_t *status_state, int32_t *status_out,
                                                const int32_t *__restrict__ list, const int32_t *__restrict__ count) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (PART == EKF_REPLAY) {
    if (i >= *count) return;
    i = list[i];
  } else if (i >= dm.n) {
    return;
  }
  const int st = ekf_tick<T, PART>(c, dm, b, in, out, k, i);
  if (PART == EKF_UPDATE && in.vo_flag != nullptr && in.vo_flag[i]) return;  // the replay launch wrote this instance's status bits
  status_state[i] = st;  // b.status, or a ring slot when the EKF runs ahead of the MHE (dekf_run)
  if (status_out != nullptr) status_out[i] = st;
}

// quat_copy (dekf_run only): the tick's quaternion also goes to the per-step output array from here -- it used to be a
// device-to-device cudaMemcpyAsync per tick on the assembly stream, i.e. a copy-engine round trip in front of every solve
// VO synchronisation of the instances that carry a VO message, over the compacted list of those instances (thread t handles
// list[t], t < *count; a launch may be restricted to the instances of a tile range, like k_assemble).  Runs BEFORE k_assemble
// pushes the tick's sample; leaves its status bits in vo_stat for k_assemble<..., VOSPLIT = true> to pick up.
template <typename T>
__global__ void __launch_bounds__(kBlock) k_vo_sync(const MheConst<T> c, const Dims dm, const Buffers<T> b, const Inputs in,
                                                    const Outputs out, int Tk, const int32_t *__restrict__ list,
                                                    const int32_t *__restrict__ count, int i_lo, int i_hi, int32_t *__restrict__ vo_stat) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= *count) return;
  const int i = list[t];
  if (i < i_lo || i >= i_hi) return;
  vo_stat[i] = mhe_vo_sync<T>(c, dm, b, in, out, Tk, i, nullptr);
}

template <typename T, typename Model, bool VOSPLIT = false>
__global__ void __launch_bounds__(kBlock, DEKF_MINB_ASM) k_assemble(const MheConst<T> c, const Dims dm, const Buffers<T> b, const Inputs in,
                                                     const Outputs out, int Tk, const int32_t *prev_status, double *quat_copy,
                                                     const int32_t *vo_stat) {
  const int i = (blockIdx.x + dm.tile0) * blockDim.x + threadIdx.x;  // tile0: a launch may cover a tile range only (dekf_run, VO ticks)
  if (i >= dm.n) return;
  const int prev = (prev_status != nullptr) ? prev_status[i] : 0;  // this tick's EKF status bits (asked for first: not a stall at the end)
  double q[4];
#pragma unroll
  for (int f = 0; f < 4; ++f)
    q[f] = (in.quat != nullptr) ? in.quat[(size_t)f * dm.n + i] : (double)b.ekf_q[(size_t)f * dm.ns + i];
  if (quat_copy != nullptr) {
#pragma unroll
    for (int f = 0; f < 4; ++f) quat_copy[(size_t)f * dm.n + i] = q[f];
  }
  const int st = mhe_assemble<T, Model, true, VOSPLIT>(c, dm, b, in, out, Tk, i, q, vo_stat);
  tick_status(dm, b, Tk, i) = prev | st;
}

template <typename T>
__global__ void __launch_bounds__(kBlock) k_solve(const MheConst<T> c, const Dims dm, const Buffers<T> b, const Inputs in,
                                                  const Outputs out, int Tk, int32_t *status_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  int st = tick_status(dm, b, Tk, i);
  if (Tk >= 1) st |= mhe_solve<T>(c, dm, b, in, out, Tk, i);
  tick_status(dm, b, Tk, i) = st;
  if (status_out != nullptr) status_out[i] = st;
}

// incremental window solve (cfg.window_solve == DEKF_SOLVE_INCREMENTAL): restart the sweep at the first changed stage
template <typename T>
__global__ void __launch_bounds__(kBlock, DEKF_MINB_INCR) k_solve_incr(const MheConst<T> c, const Dims dm, const Buffers<T> b, const Inputs in,
                                                       const Outputs out, int Tk, int32_t *status_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  int st = tick_status(dm, b, Tk, i);
  if (Tk >= 1) st |= mhe_solve_incr<T>(c, dm, b, in, out, Tk, i);
  tick_status(dm, b, Tk, i) = st;
  if (status_out != nullptr) status_out[i] = st;
}
template <typename T>
__global__ void __launch_bounds__(kBlock) k_arrival_from_ckpt(const MheConst<T> c, const Dims dm, const Buffers<T> b, int Tk) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  arrival_from_checkpoint<T>(c, dm, b, Tk, i);
}

// state-constrained window solve (cfg.v_box_enable): marginalise + primal-dual active set on the block-tridiagonal QP
template <typename T>
__global__ void __launch_bounds__(kBlock) k_solve_box(const MheConst<T> c, const BoxConst bc, const Dims dm, const Buffers<T> b,
                                                      const BoxBuffers bb, const Inputs in, const Outputs out, int Tk,
                                                      int32_t *status_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  int st = tick_status(dm, b, Tk, i);
  if (Tk >= 1) st |= mhe_solve_box<T>(c, bc, dm, b, bb, in, out, Tk, i);
  tick_status(dm, b, Tk, i) = st;
  if (status_out != nullptr) status_out[i] = st;
}

// state-constrained window solve, team form (box_team.cuh): k_box_prior (one thread per instance: marginalisation +
// information-form prior) then k_box_team (9 lanes per instance, 3 instances per warp: the active-set iteration)
template <typename T>
__global__ void __launch_bounds__(kBlock) k_box_prior(const MheConst<T> c, const Dims dm, const Buffers<T> b, const BoxBuffers bb,
                                                      const BoxTeamBuffers tb, int Tk) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n || Tk < 1) return;
  const int st = box_team_prior<T>(c, dm, b, bb, tb, Tk, i);
  if (st) tick_status(dm, b, Tk, i) |= st;
}

constexpr int kTeamsPerWarp = 3, kTeamBlock = 64;  // 64-thread CTAs: finer tail of the 2.3-wave grid (128: 4.3 ms, 64: 4.0 ms, 32: 3.95 / foot 4.5 ms)
#ifndef DEKF_MINB_BOXTEAM
#define DEKF_MINB_BOXTEAM 8
#endif
template <typename T>
__global__ void __launch_bounds__(kTeamBlock, DEKF_MINB_BOXTEAM) k_box_team(const BoxConst bc, const Dims dm, const Buffers<T> b, const BoxBuffers bb,
                                                         const BoxTeamBuffers tb, const Inputs in, const Outputs out, int Tk,
                                                         int32_t *status_out) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int team = lane / 9;  // 3 = the five idle lanes of the warp
  const int r = lane - 9 * team, base = 9 * team;
  int i = warp * kTeamsPerWarp + team;
  const bool valid = team < kTeamsPerWarp && i < dm.n;
  if (i > dm.n - 1) i = dm.n - 1;  // idle teams shadow a real instance (loads only)
  const int n = dm.n;
  int st = 0;
  double xT = 0.0;
  if (Tk >= 1) {
    const int k0 = Tk < dm.N ? 0 : Tk - dm.N + 1;
    __shared__ T s_rec[kTeamBlock / 32 * 4][2 * REC_SIZE];  // per team (3 + the idle lanes' slot per warp): two stage records
    st = box_team_solve<T>(bc, dm, b, bb, tb, k0, Tk, i, valid, base, r, s_rec[(threadIdx.x >> 5) * 4 + team], xT);
    // getsolution(T) and the body-velocity read-out (DecentralEst.cpp:179-185)
    const unsigned bad = __ballot_sync(0xffffffffu, !(xT == xT) || !(xT - xT == 0.0));
    if ((bad >> base) & 0x1ffu) st |= ST_NONFINITE;
    const double v0 = bt_shfl(xT, base + 3), v1 = bt_shfl(xT, base + 4), v2 = bt_shfl(xT, base + 5);
    if (valid) {
      if (out.x != nullptr) out.x[(size_t)r * n + i] = xT;
      if (out.v_body != nullptr && r < 3) {
        const T *rec = b.win + (size_t)(Tk % dm.NW) * REC_SIZE * dm.ns + i;
        const double om0 = in.gyro[(size_t)0 * n + i], om1 = in.gyro[(size_t)1 * n + i], om2 = in.gyro[(size_t)2 * n + i];
        const double *lever = bc.lever;
        const double u0 = v0 + (om1 * lever[2] - om2 * lever[1]), u1 = v1 + (om2 * lever[0] - om0 * lever[2]),
                     u2 = v2 + (om0 * lever[1] - om1 * lever[0]);
        const double R0 = (double)rec[(size_t)(REC_R + r * 3 + 0) * dm.ns], R1 = (double)rec[(size_t)(REC_R + r * 3 + 1) * dm.ns],
                     R2 = (double)rec[(size_t)(REC_R + r * 3 + 2) * dm.ns];
        out.v_body[(size_t)r * n + i] = R0 * u0 + R1 * u1 + R2 * u2;
      }
    }
  }
  if (valid && r == 0) {
    if (Tk >= 1) bb.capped[i] = (st & ST_QP_MAXITER) ? 1 : 0;  // only box_team_solve sets ST_QP_MAXITER in st
    st |= tick_status(dm, b, Tk, i);
    tick_status(dm, b, Tk, i) = st;
    if (status_out != nullptr) status_out[i] = st;
  }
}

// leg_odom_type 1 (foot-position states): information-form window sweep / KF step, footstate.cuh
template <typename T, int L>
__global__ void __launch_bounds__(kBlock) k_solve_foot(const FootConst fc, const Dims dm, const Buffers<T> b, const FootBuffers fb,
                                                       const Inputs in, const Outputs out, int Tk, int32_t *status_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  int st = tick_status(dm, b, Tk, i);
  if (Tk >= 1 || fc.est_type == 1) st |= foot_solve<T, L>(fc, dm, b, fb, in, out, Tk, i);
  tick_status(dm, b, Tk, i) = st;
  if (status_out != nullptr) status_out[i] = st;
}
// the same with one WARP per instance (foot_team.cuh): rows of the 21 x 21 blocks in registers, shuffles between lanes
template <typename T, int L>
__global__ void __launch_bounds__(kTeamBlock) k_foot_team(const FootConst fc, const Dims dm, const Buffers<T> b, const FootBuffers fb,
                                                          const Inputs in, const Outputs out, int Tk, int32_t *status_out) {
  const int lane = threadIdx.x & 31;
  int i = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const bool valid = i < dm.n;
  if (!valid) i = dm.n - 1;  // idle warps shadow a real instance (loads only)
  int st = 0;
  if (Tk >= 1 || fc.est_type == 1) st = foot_team_solve<T, L>(fc, dm, b, fb, in, out, Tk, i, valid, lane);
  if (valid && lane == 0) {
    st |= tick_status(dm, b, Tk, i);
    tick_status(dm, b, Tk, i) = st;
    if (status_out != nullptr) status_out[i] = st;
  }
}
// smoothed window of the foot-state model (dekf_get_foot_window, foot_window.cuh): one warp per instance, two warps per CTA
// with the stage record, P_{k+1} and the transpose buffer of each warp in shared memory
constexpr int kFootWinBlock = 64;
template <int L, bool WX, bool WP, bool WC = false>
__global__ void __launch_bounds__(kFootWinBlock) k_foot_window(const FootConst fc, const Dims dm, const Buffers<double> b,
                                                               const FootBuffers fb, double *ring, int Tk, double *xout, double *Pout,
                                                               double *Cout) {
  __shared__ double sh[kFootWinBlock / 32][foot_win_smem_words<L>()];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i = (int)((size_t)blockIdx.x * (kFootWinBlock / 32) + w);
  if (i >= dm.n) return;  // whole warps only: no block-wide barrier follows
  foot_window_team<L, WX, WP, WC>(fc, dm, b, fb, ring, Tk, i, lane, sh[w], xout, Pout, Cout);
}
// C non-null (dekf_get_window_cross_cov): the lag-one blocks into C and, when P is non-null, the covariances into P (x unused)
template <int L>
void launch_foot_window(const FootConst &fc, const Dims &dm, const Buffers<double> &b, const FootBuffers &fb, double *ring, int Tk,
                        double *x, double *P, double *C, cudaStream_t stream) {
  const dim3 grid((dm.n + kFootWinBlock / 32 - 1) / (kFootWinBlock / 32));
  if (C && P)
    k_foot_window<L, false, true, true><<<grid, kFootWinBlock, 0, stream>>>(fc, dm, b, fb, ring, Tk, x, P, C);
  else if (C)
    k_foot_window<L, false, false, true><<<grid, kFootWinBlock, 0, stream>>>(fc, dm, b, fb, ring, Tk, x, P, C);
  else if (x && P)
    k_foot_window<L, true, true><<<grid, kFootWinBlock, 0, stream>>>(fc, dm, b, fb, ring, Tk, x, P, nullptr);
  else if (x)
    k_foot_window<L, true, false><<<grid, kFootWinBlock, 0, stream>>>(fc, dm, b, fb, ring, Tk, x, P, nullptr);
  else
    k_foot_window<L, false, true><<<grid, kFootWinBlock, 0, stream>>>(fc, dm, b, fb, ring, Tk, x, P, nullptr);
}
// window of a state-constrained handle (dekf_get_constrained_window, box_window.cuh): 9 lanes per instance, 3 instances per
// warp as in k_box_team; SOA: the serial solve's scratch [N][BOX_FAC][ns], else the team solve's [ns][N][BOX_TFAC]
// CROSS (dekf_get_window_cross_cov): the lag-one blocks into C and, when P is non-null, the covariances into P
template <bool SOA, bool CROSS = false>
__global__ void __launch_bounds__(kTeamBlock) k_box_window(const BoxConst bc, const Dims dm, const BoxBuffers bb, const double *fac,
                                                           int Tk, double *x, double *P, uint32_t *act, double *C) {
  __shared__ double sh[kTeamBlock / 32 * 4][BW_TEAM_WORDS];  // per team (3 + the idle lanes' slot per warp)
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int team = lane / 9;
  const int r = lane - 9 * team;
  int i = warp * kTeamsPerWarp + team;
  const bool valid = team < kTeamsPerWarp && i < dm.n;
  if (i > dm.n - 1) i = dm.n - 1;  // idle teams shadow a real instance (loads only)
  const BwLayout<SOA> lay = {fac, (size_t)dm.ns, dm.N};
  box_window_team<SOA, CROSS>(bc, dm, bb, lay, Tk, i, valid, r, sh[(threadIdx.x >> 5) * 4 + team], x, P, act, C);
}
// arrival cost of the foot-state model: (M_p, n_p) as the reference holds them (MheSrb.hpp:86-87)
__global__ void k_get_arrival_foot(const Dims dm, const FootBuffers fb, int ds, double *Mout, double *nout) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  int p = 0;
  for (int r = 0; r < ds; ++r)
    for (int c = 0; c <= r; ++c) {
      const double v = fb.arr_M[(size_t)(p++) * dm.ns + i];
      Mout[(size_t)(r * ds + c) * dm.n + i] = v;
      Mout[(size_t)(c * ds + r) * dm.n + i] = v;
    }
  for (int r = 0; r < ds; ++r) nout[(size_t)r * dm.n + i] = -fb.arr_m[(size_t)r * dm.ns + i];
}

// KF alternative (est_type 1): one predict + correct per tick instead of the window solve
template <typename T>
__global__ void __launch_bounds__(kBlock) k_kf(const MheConst<T> c, const Dims dm, const Buffers<T> b, const Inputs in,
                                               const Outputs out, int Tk, int32_t *status_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  int st = tick_status(dm, b, Tk, i);
  st |= kf_update<T>(c, dm, b, in, out, Tk, i);
  tick_status(dm, b, Tk, i) = st;
  if (status_out != nullptr) status_out[i] = st;
}

}  // namespace dekf
#include "solve_tma.cuh"
namespace dekf {

// whole tick in one launch (small batches: launch latency dominates)
template <typename T, typename Model>
__global__ void __launch_bounds__(kBlock) k_fused(const EkfConst<T> ec, const MheConst<T> mc, const Dims dm, const Buffers<T> b,
                                                  const Inputs in, const Outputs out, int k, int Tk, int32_t *status_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  int st = ekf_tick<T>(ec, dm, b, in, out, k, i);
  double q[4];
#pragma unroll
  for (int f = 0; f < 4; ++f) q[f] = (double)b.ekf_q[(size_t)f * dm.ns + i];
  st |= mhe_assemble<T, Model, false>(mc, dm, b, in, out, Tk, i, q);
  if (mc.est_type == 1)
    st |= kf_update<T>(mc, dm, b, in, out, Tk, i);
  else if (Tk >= 1 && mc.window_solve == 1)
    st |= mhe_solve_incr<T>(mc, dm, b, in, out, Tk, i, true);  // true: prefetch the stage records (few warps, latency-bound)
  else if (Tk >= 1)
    st |= mhe_solve<T>(mc, dm, b, in, out, Tk, i, true);
  tick_status(dm, b, Tk, i) = st;
  if (status_out != nullptr) status_out[i] = st;
}

// Whole tick in one launch, ROLE form (small batches, est_type 0, leg_odom_type 0): one CTA = 32 instances (lane = instance), one
// warp per ROLE, so that the pieces of a tick that do not depend on each other run side by side instead of one after the other in
// a single thread (k_fused: 53 us per batch-1 tick, two thirds of it in straight-line code that is fetched once per launch):
//   warp 0            front:  VO synchronisation (mhe_vo_sync) -> orientation EKF tick -> leg sums -> stage record of tick T
//   warps 1 .. NL     legs:   contact, kinematics and the leg-odometry statistic of ONE leg each (leg_statistic)
//   warp NL + 1       sweep:  window sweep over the stages T-N .. T-1 (they do not depend on this tick's sample), then the stage of
//                             tick T once the front warp has written its record, read-out of x_T
// The warps meet at three named barriers (non-aligned barrier.sync / barrier.arrive, one count per thread):
//   1: VO rows of the window are final (front -> sweep)   2: leg statistics are in shared memory (legs -> front)
//   3: the record of stage T is written (front -> sweep)
// Every operand and every operation is the one k_fused / the large-batch kernels use (same device functions, leg sums added in
// leg order), so the results are bit-identical (tests/test_gpu_parity.py::test_role_kernel_equals_fused_kernel).
__device__ __forceinline__ void role_bar_sync(int id, int cnt) { asm volatile("barrier.sync %0, %1;" ::"r"(id), "r"(cnt) : "memory"); }
__device__ __forceinline__ void role_bar_arrive(int id, int cnt) { asm volatile("barrier.arrive %0, %1;" ::"r"(id), "r"(cnt) : "memory"); }

template <typename T>
struct RoleStageSource : GlobalStageSource<T> {
  int jlast;  // ordinal of stage T in this sweep
  __device__ RoleStageSource(const Dims &dm_, const Buffers<T> &b_, int i_, int jl) : GlobalStageSource<T>(dm_, b_, i_, true), jlast(jl) {}
  __device__ __forceinline__ void acquire(int j) const {
    if (j == jlast) role_bar_sync(3, 64);
  }
};

template <typename T, typename Model>
__global__ void __launch_bounds__((Model::NLEG + 2) * 32, 1) k_fused_roles(const EkfConst<T> ec, const MheConst<T> mc, const Dims dm,
                                                                          const Buffers<T> b, const Inputs in, const Outputs out, int k,
                                                                          int Tk, int32_t *status_out) {
  constexpr int NL = Model::NLEG, NJ = Model::NJ;
  __shared__ T s_leg[NL][12][32];  // per leg: Qb (6), Qb beta (3), beta (3)
  __shared__ int s_contact[NL][32];
  __shared__ int s_status[32];
  const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  const int n = dm.n;
  const bool valid = i < n;
  if (role == 0) {
    int st = 0;
    if (valid) st = mhe_vo_sync<T>(mc, dm, b, in, out, Tk, i, nullptr);
    __threadfence_block();
    role_bar_arrive(1, 64);
    double q[4] = {1.0, 0.0, 0.0, 0.0};
    M3<T> R;
    V3<T> as = v3<T>(T(0), T(0), T(0));
    if (valid) {
      st |= ekf_tick<T>(ec, dm, b, in, out, k, i);
#pragma unroll
      for (int f = 0; f < 4; ++f) q[f] = (double)b.ekf_q[(size_t)f * dm.ns + i];
      // current sample (DecentralEst.cpp:867-879)
      R = quat_to_rot<T>((T)q[0], (T)q[1], (T)q[2], (T)q[3]);
      V3<T> ab;
#pragma unroll
      for (int f = 0; f < 3; ++f) ab[f] = (T)in.accel[(size_t)f * n + i];
      as = mul(R, ab);
      as[2] += T(-9.81);
    }
    role_bar_sync(2, (NL + 1) * 32);
    if (valid) {
      S3<T> Qb_sum;
#pragma unroll
      for (int f = 0; f < 6; ++f) Qb_sum.a[f] = T(0);
      V3<T> Qbeta_sum = v3<T>(T(0), T(0), T(0)), beta_swing = v3<T>(T(0), T(0), T(0));
      int n_swing = 0, contact_mask = 0;
#pragma unroll
      for (int leg = 0; leg < NL; ++leg) {  // leg order: the same sums as the serial loop of mhe_assemble
        const bool contact = s_contact[leg][lane] != 0;
        contact_mask |= (contact ? 1 : 0) << leg;
        if (contact) {
#pragma unroll
          for (int f = 0; f < 6; ++f) Qb_sum.a[f] += s_leg[leg][f][lane];
          Qbeta_sum = add(Qbeta_sum, v3<T>(s_leg[leg][6][lane], s_leg[leg][7][lane], s_leg[leg][8][lane]));
        } else {
          beta_swing = add(beta_swing, v3<T>(s_leg[leg][9][lane], s_leg[leg][10][lane], s_leg[leg][11][lane]));
          n_swing++;
        }
      }
      mhe_push_sample<T>(mc, dm, b, in, Tk, i, q, R, as, Qb_sum, Qbeta_sum, beta_swing, n_swing, contact_mask, NL);
    }
    s_status[lane] = st;
    __threadfence_block();
    role_bar_arrive(3, 64);
  } else if (role <= NL) {
    const int leg = role - 1;
    if (valid) {
      const bool contact = (in.foot_force[(size_t)leg * n + i] >= mc.thr);  // go1Sub.cpp:74, exact
      if (out.contact != nullptr) out.contact[(size_t)leg * n + i] = contact ? 1 : 0;
      T q[NJ], dq[NJ];
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        q[j] = (T)in.joint_pos[(size_t)(leg * NJ + j) * n + i];
        dq[j] = (T)in.joint_vel[(size_t)(leg * NJ + j) * n + i];
      }
      V3<T> om;
#pragma unroll
      for (int f = 0; f < 3; ++f) om[f] = (T)in.gyro[(size_t)f * n + i];
      V3<T> p, beta, Qbeta;
      T J[3 * NJ];
      S3<T> Qb;
      leg_statistic<T, Model>(mc, leg, q, dq, om, p, J, beta, Qb, Qbeta);
      s_contact[leg][lane] = contact ? 1 : 0;
#pragma unroll
      for (int f = 0; f < 6; ++f) s_leg[leg][f][lane] = Qb.a[f];
#pragma unroll
      for (int f = 0; f < 3; ++f) {
        s_leg[leg][6 + f][lane] = Qbeta[f];
        s_leg[leg][9 + f][lane] = beta[f];
      }
    }
    __threadfence_block();
    role_bar_arrive(2, (NL + 1) * 32);
  } else {
    role_bar_sync(1, 64);
    int st = 0;
    if (valid && Tk >= 1) {
      if (mc.window_solve == 1) {
        const int ks = incr_restart_stage(dm, b, Tk, i);
        RoleStageSource<T> src(dm, b, i, Tk - ks);
        st = mhe_solve_incr<T, RoleStageSource<T>>(mc, dm, b, in, out, Tk, i, src, ks);
      } else {
        const int k0 = (Tk < dm.N) ? 0 : Tk - dm.N;
        RoleStageSource<T> src(dm, b, i, Tk - k0);
        st = mhe_solve<T, RoleStageSource<T>>(mc, dm, b, in, out, Tk, i, src);
      }
    } else {
      role_bar_sync(3, 64);
    }
    if (valid) {
      st |= s_status[lane];
      tick_status(dm, b, Tk, i) = st;
      if (status_out != nullptr) status_out[i] = st;
    }
  }
}

template <typename T>
__global__ void k_init_state(const EkfConst<T> ec, const MheConst<T> mc, const Dims dm, const Buffers<T> b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  const int n = dm.ns;
#pragma unroll
  for (int f = 0; f < 4; ++f) b.ekf_q[(size_t)f * n + i] = ec.q0[f];
#pragma unroll
  for (int f = 0; f < 16; ++f) b.ekf_P[(size_t)f * n + i] = (f % 5 == 0) ? ec.P0[f / 5] : T(0);
#pragma unroll
  for (int f = 0; f < 45; ++f) b.arr_P[(size_t)f * n + i] = T(0);
  const int diag[3] = {0, 3, 5};
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    b.arr_P[(size_t)(0 + diag[f]) * n + i] = mc.P0[f];
    b.arr_P[(size_t)(6 + diag[f]) * n + i] = mc.P0[3 + f];
    b.arr_P[(size_t)(12 + diag[f]) * n + i] = mc.P0[6 + f];
  }
#pragma unroll
  for (int f = 0; f < 9; ++f) b.arr_x[(size_t)f * n + i] = T(0);
#pragma unroll
  for (int f = 0; f < 3; ++f) b.p_vo[(size_t)f * n + i] = 0.0;
  b.wp_count[i] = 0;
  b.pend_flag[i] = 0;
  b.status[i] = 0;
  b.status[(size_t)dm.ns + i] = 0;
}

// arrival cost getters: (P, x) -> dense 9x9 P, and (M_p, n_p) = (P^-1, -P^-1 x) (MheSrb.hpp:86-87)
template <typename T>
__global__ void k_get_arrival(const Dims dm, const Buffers<T> b, double *Pout, double *xout, int as_information) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  const int n = dm.n, ns = dm.ns;
  Cov9<T> P;
  load_cov(b.arr_P, ns, i, P);
  double A[81], x[9];
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      A[(0 + r) * 9 + 0 + c] = (double)P.pp(r, c);
      A[(3 + r) * 9 + 3 + c] = (double)P.vv(r, c);
      A[(6 + r) * 9 + 6 + c] = (double)P.bb(r, c);
      A[(0 + r) * 9 + 3 + c] = (double)P.pv(r, c);
      A[(3 + c) * 9 + 0 + r] = (double)P.pv(r, c);
      A[(0 + r) * 9 + 6 + c] = (double)P.pb(r, c);
      A[(6 + c) * 9 + 0 + r] = (double)P.pb(r, c);
      A[(3 + r) * 9 + 6 + c] = (double)P.vb(r, c);
      A[(6 + c) * 9 + 3 + r] = (double)P.vb(r, c);
    }
  for (int f = 0; f < 9; ++f) x[f] = (double)b.arr_x[(size_t)f * ns + i];
  if (as_information) {
    // Cholesky A = L L', M = A^-1 column by column, n_p = -M x
    double L[81];
    for (int j = 0; j < 9; ++j) {
      double d = A[j * 9 + j];
      for (int k = 0; k < j; ++k) d -= L[j * 9 + k] * L[j * 9 + k];
      d = sqrt(d);
      L[j * 9 + j] = d;
      for (int r = j + 1; r < 9; ++r) {
        double v = A[r * 9 + j];
        for (int k = 0; k < j; ++k) v -= L[r * 9 + k] * L[j * 9 + k];
        L[r * 9 + j] = v / d;
      }
    }
    double np[9];
    for (int f = 0; f < 9; ++f) np[f] = 0.0;
    for (int c = 0; c < 9; ++c) {
      double y[9];
      for (int r = 0; r < 9; ++r) {
        double v = (r == c) ? 1.0 : 0.0;
        for (int k = 0; k < r; ++k) v -= L[r * 9 + k] * y[k];
        y[r] = v / L[r * 9 + r];
      }
      for (int r = 8; r >= 0; --r) {
        double v = y[r];
        for (int k = r + 1; k < 9; ++k) v -= L[k * 9 + r] * y[k];
        y[r] = v / L[r * 9 + r];
      }
      for (int r = 0; r < 9; ++r) {
        Pout[(size_t)(r * 9 + c) * n + i] = y[r];
        np[r] -= y[r] * x[c];
      }
    }
    for (int f = 0; f < 9; ++f) xout[(size_t)f * n + i] = np[f];
  } else {
    for (int f = 0; f < 81; ++f) Pout[(size_t)f * n + i] = A[f];
    for (int f = 0; f < 9; ++f) xout[(size_t)f * n + i] = x[f];
  }
}

template <typename T>
__global__ void k_get_misc(const Dims dm, const Buffers<T> b, int Tk, double *p_vo, double *R_sb, double *ekfP) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  const int n = dm.n, ns = dm.ns;
  if (p_vo != nullptr)
    for (int f = 0; f < 3; ++f) p_vo[(size_t)f * n + i] = b.p_vo[(size_t)f * ns + i];
  if (R_sb != nullptr) {
    const T *rec = b.win + (size_t)(Tk % dm.NW) * REC_SIZE * ns + i;
    for (int f = 0; f < 9; ++f) R_sb[(size_t)f * n + i] = (double)rec[(size_t)(REC_R + f) * ns];
  }
  if (ekfP != nullptr)
    for (int f = 0; f < 16; ++f) ekfP[(size_t)f * n + i] = (double)b.ekf_P[(size_t)f * ns + i];
}

// incremental solve bookkeeping of the last tick: re-swept stages (T - restart stage) and how many of them carry a VO row
template <typename T>
__global__ void k_resweep_info(const Dims dm, const Buffers<T> b, int Tk, int32_t *depth, int32_t *n_vo) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  const int ks = incr_restart_stage(dm, b, Tk, i);
  int c = 0;
  for (int k = ks; k < Tk; ++k) c += b.win[((size_t)(k % dm.NW) * REC_SIZE + REC_FLAG) * dm.ns + i] != T(0);
  if (depth) depth[i] = Tk - ks;
  if (n_vo) n_vo[i] = c;
}

template <typename T>
__global__ void k_vo_count(const Dims dm, const Buffers<T> b, int Tk, int32_t *count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  int c = 0;
  const int k0 = (Tk >= dm.N) ? Tk - dm.N + 1 : 0;
  for (int k = k0; k < Tk; ++k) c += b.win[((size_t)(k % dm.NW) * REC_SIZE + REC_FLAG) * dm.ns + i] != T(0);
  count[i] = c;
}

// smoothed window of the last update(Tk) (dekf_get_window): one thread per instance, SoA loads coalesced over instances.
// FULL: the forward sweep from the arrival cost into the scratch ring scr [N][54][ns] runs first; otherwise the checkpoint ring
// of the incremental solve is read (one instantiation per mode: neither carries the other's registers).
template <typename T, bool FULL>
__global__ void __launch_bounds__(kBlock) k_window(const MheConst<T> c, const MheConst<double> c64, const Dims dm, const Buffers<T> b,
                                                   T *scr, int Tk, double *xout) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  mhe_window_smooth<T>(c, c64, dm, b, FULL ? scr : nullptr, Tk, i, xout, (size_t)dm.n);
}

// smoothed covariances of the window (dekf_get_window_cov): one thread per instance like k_window, which already sits at
// 250-255 registers; the 9x9 gain G and Sigma - P_{k+1}^s of each thread (126 doubles) live in shared memory instead, one
// column per thread so that a warp's accesses are conflict-free.  One-warp CTAs keep that area within the static limit.
// CROSS (dekf_get_window_cross_cov): also the lag-one blocks into cout, pout holding pslots blocks (window_cov_backward).
constexpr int kCovBlock = 32;
template <typename T, bool FULL, bool CROSS = false>
__global__ void __launch_bounds__(kCovBlock) k_window_cov(const MheConst<T> c, const MheConst<double> c64, const Dims dm,
                                                          const Buffers<T> b, T *scr, int Tk, double *pout, double *cout,
                                                          int pslots) {
  __shared__ double sh[126 * kCovBlock];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dm.n) return;
  mhe_window_cov<T, CROSS>(c, c64, dm, b, FULL ? scr : nullptr, Tk, i, pout, (size_t)dm.n, sh + threadIdx.x, kCovBlock, cout,
                           pslots);
}

}  // namespace dekf

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
using namespace dekf;

struct StageSet {
  double *in = nullptr;      // packed doubles (in_counts order)
  uint8_t *flag = nullptr;
  double *out = nullptr;     // quat4 x9 v_body3
  uint8_t *contact = nullptr;
  int32_t *status = nullptr;
};

// device staging of dekf_run_host: `cap` ticks of every stream
struct ChunkSet {
  int cap = 0;
  double *in = nullptr;      // gyro accel imu_time joint_pos joint_vel foot_force | vo_quat vo_time_pre vo_time_now vo_rel_p, each [cap][rows][n]
  float *in_f32 = nullptr;   // dekf_run_host_f32: gyro accel joint_pos joint_vel foot_force as float, each [cap][rows][n]
  int cap_f32 = 0;
  uint8_t *flag = nullptr;   // [cap][n]
  double *out = nullptr;     // quat [cap][4][n] | x [cap][9][n] | v_body [cap][3][n]
  float *out_f32 = nullptr;  // dekf_run_host_f32io: the same three arrays rounded to float (allocated on first use)
  int cap_out_f32 = 0;
  uint8_t *contact = nullptr;
  int32_t *status = nullptr;
};

struct dekf_handle {
  dekf_config cfg;
  Dims dm;
  int nl, nj, nq;
  int ds;  // state dimension 9 + 3 * leg_odom_type * num_legs (DecentralEst.cpp:20) == rows of outputs.x
  bool f32;
  EkfConst<double> ec64;
  MheConst<double> mc64;
  EkfConst<float> ec32;
  MheConst<float> mc32;
  Buffers<double> b64;
  Buffers<float> b32;
  BoxConst bc;
  BoxBuffers bb = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  double *row_V = nullptr;  // device copy of W^-1 (dekf_add_state_rows)
  BoxTeamBuffers tb = {nullptr, nullptr};
  bool box_team = true;           // team form of the constrained solve (DEKF_BOX_SERIAL=1 selects one thread per instance)
  bool foot_team = true;          // one warp per instance for the foot-state model (DEKF_FOOT_SERIAL=1: one thread per instance)
  FootConst fc;
  FootBuffers fb = {nullptr, nullptr, nullptr};  // leg_odom_type 1
  void *ckpt_mem = nullptr;       // incremental window solve: checkpoint ring
  void *win_scr = nullptr;        // dekf_get_window on a full re-sweep handle: filtered states [N][54][ns] (first use)
  double *foot_win_ring = nullptr;  // dekf_get_foot_window: stage factors [N-1][ns][FootWin<L>::W] (first use)
  double *cross_ring = nullptr;     // dekf_get_window_cross_cov without P on a 9-state handle: P_k^s, P_{k+1}^s [2][81][n]
  int32_t *resweep_mem = nullptr;
  void *slab = nullptr;
  size_t slab_bytes = 0;
  // device staging of the host-pointer entry points (set 1 and the copy streams only exist after dekf_run_host)
  StageSet stage[2];
  ChunkSet chunk[2];
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  // dekf_run: the EKF ticks run ahead of the MHE on their own stream through a small ring of quaternions / status words
  static constexpr int kAhead = 4;
  static constexpr int kMaxWays = 8;
  cudaStream_t s_ekf = nullptr, s_asm = nullptr;
  // solve streams: s_sol[0] carries every undivided solve; the full re-sweep of a large batch is cut into tile ranges, range r
  // runs on s_sol[r] (independent instances: range r of tick s+1 only waits for range r of tick s)
  cudaStream_t s_sol[kMaxWays] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_solw[kMaxWays][kAhead] = {};
  int solve_tile0 = 0, solve_tiles = -1;  // tile range of the next k_solve_tma launch (-1: the whole batch)
  int solve_slots = 0;                    // CTAs of k_solve_tma resident on the whole device (occupancy x SM count)
  int asm_tile0 = 0, asm_tiles = -1;      // tile range of the next k_assemble launch (-1: the whole batch)
  cudaStream_t s_asmw[kMaxWays] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // s_asmw[0] == s_asm
  cudaEvent_t ev_asmw[kMaxWays][kAhead] = {};  // assembly of tile range r of the tick in ring slot k is done
  cudaEvent_t ev_join = nullptr;
  double *quat_ring = nullptr;      // [kAhead][4][n]
  int32_t *status_ring = nullptr;   // [kAhead][n]
  cudaEvent_t ev_ekf[kAhead] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr;
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
  // debug taps
  double *tap_b_meas = nullptr, *tap_Q_meas = nullptr;
  int32_t *tap_vo = nullptr, *tap_ekf = nullptr;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int ekf_k = 0;    // EKF ticks done
  int next_T = 0;   // next MHE discrete time expected
  int64_t launches = 0;
  size_t extra_bytes = 0;
  CUtensorMap tmap;      // window ring as a 2-D tensor [NW*25][ns] (TMA box = one stage record of one tile)
  int fused_max = 4096;  // batches up to this size take the single fused launch (DEKF_FUSED_MAX_N at create)
  bool use_tma = true;   // window solve with TMA-staged stage tiles (DEKF_NO_TMA=1 at create: plain global loads)
  // tuning knobs, read ONCE in dekf_create (environment), never on the step path
  bool no_split = false;   // DEKF_NO_SPLIT=1: one k_solve_tma launch per tick in dekf_run
  bool no_asm_split = false; // DEKF_NO_ASM_SPLIT=1: VO ticks assemble the whole batch in one launch behind the whole previous solve
  int split_tiles_env = 0; // DEKF_SPLIT_TILES=<k>: size of the first tile range (0: the last full wave)
  int split_ways_env = 0;  // DEKF_SPLIT_WAYS=<w>: w equal tile ranges on w streams instead of the two-range split
  int host_chunk = 8;      // DEKF_HOST_CHUNK=<B>: ticks per copy of dekf_run_host
  bool host_ramp = true;   // DEKF_HOST_RAMP=0: every chunk of dekf_run_host is B ticks (no ramp at the ends of a call)
  bool ekf_serial = false;  // DEKF_EKF_SERIAL=1: no EKF launch of dekf_run overlaps a window solve (diagnosis tool, DESIGN.md section 10.1)
  // VO-carrying ticks of large batches compact the flagged instances and run the EKF replay and the VO synchronisation over that
  // list (ragged arrival: 3.9e8 -> 4.8e8 instance-steps/s; lock-step arrival: unchanged).  DEKF_VO_COMPACT=0: one launch each.
  bool vo_compact = true;
  int32_t *vo_stat = nullptr;  // [kAhead][n] status bits of k_vo_sync, picked up by k_assemble<..., VOSPLIT>
  int32_t *vo_list = nullptr, *vo_count = nullptr;  // [kAhead][n] / [kAhead]: instances flagged with a VO message, per ring slot
  int vo_slot = 0;             // ring slot of the tick being queued (dekf_run: s % kAhead; single ticks: 0)
  bool vo_list_valid = false;  // the list of vo_slot was built for the tick being queued (by its EKF launch)
  int run_pipeline_min = 256;  // DEKF_RUN_PIPELINE_MIN_N: see dekf_run
  int roles_max = 4096;    // DEKF_ROLES_MAX_N=<n>: batches up to n take the role form of the fused tick (0: always the serial form)
  int prio_mode = 0;       // DEKF_PRIO=<m>: stream priorities of dekf_run (0: all equal; 1: solve > assembly > EKF, round 1; 2: front kernels first)
  // small batches through the *_host entry points: one pinned, device-mapped host block; the kernel reads the tick's inputs
  // from it and writes the results into it over PCIe (no cudaMemcpy calls: the batch-1 tick is launch + kernel + sync)
  char *hmap = nullptr;
  size_t hmap_bytes = 0;
  // scratch of the host getters (dekf_get_host): allocated once, on first use
  double *get_scratch = nullptr;
  size_t get_scratch_bytes = 0;
  double *kf_Q = nullptr;  // [num_legs][6][n] per-leg Q_meas of the newest sample (cfg.kf_export_gain)
  double *asm_quat_copy = nullptr;  // dekf_run: where k_assemble also writes the tick's quaternion (per-step output)
  // optional per-kernel timing: an event pair around every launch, no host synchronisation until the read
  bool prof = false;
  struct ProfRec {
    cudaEvent_t e0, e1;
    int slot;
  };
  std::vector<ProfRec> prof_recs;   // pairs recorded since the last read
  std::vector<ProfRec> prof_free;   // recycled pairs
  double prof_ms[4] = {0, 0, 0, 0};
  int64_t prof_n[4] = {0, 0, 0, 0};
  std::string err;
};

namespace {

int alloc_stage_set(dekf_handle *h, StageSet &ss);
void free_stage_set(StageSet &ss);
int alloc_chunk_set(dekf_handle *h, ChunkSet &cs, int cap);
void free_chunk_set(ChunkSet &cs);

int fail(dekf_handle *h, int code, const char *what, cudaError_t ce = cudaSuccess) {
  if (h) {
    h->err = what;
    if (ce != cudaSuccess) {
      h->err += ": ";
      h->err += cudaGetErrorString(ce);
    }
  }
  return code;
}

#define CK(call)                                                 \
  do {                                                           \
    cudaError_t e_ = (call);                                     \
    if (e_ != cudaSuccess) return fail(h, DEKF_ECUDA, #call, e_); \
  } while (0)

inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

template <typename T>
size_t carve(Buffers<T> &b, const Dims &dm, char *base) {
  const StateSizes s = state_sizes(dm);
  size_t off = 0;
  auto take = [&](size_t count, size_t elt) {
    char *p = base ? base + off : nullptr;
    off += align_up(count * elt);
    return p;
  };
  b.ekf_q = (T *)take(s.ekf_q, sizeof(T));
  b.ekf_P = (T *)take(s.ekf_P, sizeof(T));
  b.ekf_hist = (T *)take(s.ekf_hist, sizeof(T));
  b.ekf_hist_time = (double *)take(s.ekf_hist_time, sizeof(double));
  b.arr_P = (T *)take(s.arr_P, sizeof(T));
  b.arr_x = (T *)take(s.arr_x, sizeof(T));
  b.win = (T *)take(s.win, sizeof(T));
  b.hist_time = (double *)take(s.hist_time, sizeof(double));
  b.hist_quat = (double *)take(s.hist_quat, sizeof(double));
  b.wp = (double *)take(s.wp, sizeof(double));
  b.wp_time = (double *)take(s.wp_time, sizeof(double));
  b.wp_count = (int32_t *)take(s.wp_count, sizeof(int32_t));
  b.p_vo = (double *)take(s.p_vo, sizeof(double));
  b.pend_flag = (uint8_t *)take(s.pend_flag, 1);
  b.pend = (double *)take(s.pend, sizeof(double));
  b.status = (int32_t *)take(s.status, sizeof(int32_t));
  b.ckpt = nullptr;
  b.resweep = nullptr;
  b.foot_leg = nullptr;
  return off;
}

inline int grid_for(int n) { return (n + kBlock - 1) / kBlock; }

// Event pair around one launch on the handle's stream; elapsed times are harvested by dekf_profile_read.
struct ProfScope {
  dekf_handle *h;
  dekf_handle::ProfRec rec;
  bool on;
  cudaStream_t st;
  ProfScope(dekf_handle *h_, int slot, cudaStream_t st_ = nullptr) : h(h_), on(h_->prof), st(st_ ? st_ : h_->stream) {
    if (!on) return;
    if (!h->prof_free.empty()) {
      rec = h->prof_free.back();
      h->prof_free.pop_back();
    } else if (cudaEventCreate(&rec.e0) != cudaSuccess || cudaEventCreate(&rec.e1) != cudaSuccess) {
      on = false;
      return;
    }
    rec.slot = slot;
    cudaEventRecord(rec.e0, st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(rec.e1, st);
    h->prof_recs.push_back(rec);
  }
};

Inputs to_inputs(const dekf_inputs *in) {
  Inputs r;
  r.gyro = in->gyro;
  r.accel = in->accel;
  r.imu_time = in->imu_time;
  r.joint_pos = in->joint_pos;
  r.joint_vel = in->joint_vel;
  r.foot_force = in->foot_force;
  r.vo_flag = in->vo_flag;
  r.vo_quat = in->vo_quat;
  r.vo_time_pre = in->vo_time_pre;
  r.vo_time_now = in->vo_time_now;
  r.vo_rel_p = in->vo_rel_p;
  r.quat = in->quat;
  return r;
}
Outputs to_outputs(const dekf_handle *h, const dekf_outputs *out) {
  Outputs r;
  std::memset(&r, 0, sizeof(r));
  if (out) {
    r.quat = out->quat;
    r.x = out->x;
    r.v_body = out->v_body;
    r.contact = out->contact;
  }
  r.dbg_b_meas = h->tap_b_meas;
  r.dbg_Q_meas = h->tap_Q_meas ? h->tap_Q_meas : h->kf_Q;  // kf_Q: cfg.kf_export_gain (K_KF_ getter)
  r.dbg_vo = h->tap_vo;
  r.dbg_ekf = h->tap_ekf;
  return r;
}

template <typename T, typename Model>
int launch_assemble(dekf_handle *h, const MheConst<T> &mc, const Buffers<T> &b, const Inputs &in, const Outputs &out,
                    int T_, const int32_t *acc) {
  {
    Dims adm = h->dm;
    adm.tile0 = h->asm_tiles >= 0 ? h->asm_tile0 : 0;
    const int grid = h->asm_tiles >= 0 ? h->asm_tiles : grid_for(h->dm.n);
    // large batches from T = 2 on (the VO latch of T = 0 / 1 is over): the VO synchronisation leaves k_assemble -- ticks
    // without a message skip it altogether, ticks with messages run it over the compacted list of the flagged instances
    const bool lean = T_ >= 2 && !h->cfg.debug_taps && h->dm.n > h->fused_max;  // k_assemble without the VO code is legal
    if (lean && h->vo_compact && in.vo_flag != nullptr) {
      int32_t *list = h->vo_list ? h->vo_list + (size_t)h->vo_slot * h->dm.n : nullptr, *count = h->vo_count ? h->vo_count + h->vo_slot : nullptr;
      if (!h->vo_list_valid || !list) {  // no EKF launch built the list for this tick (dekf_mhe_step on its own)
        if (!h->vo_list) {
          if (cudaMalloc((void **)&h->vo_list, (size_t)dekf_handle::kAhead * h->dm.n * sizeof(int32_t)) != cudaSuccess) return DEKF_ENOMEM;
          if (cudaMalloc((void **)&h->vo_stat, (size_t)dekf_handle::kAhead * h->dm.n * sizeof(int32_t)) != cudaSuccess) return DEKF_ENOMEM;
          if (cudaMalloc((void **)&h->vo_count, dekf_handle::kAhead * sizeof(int32_t)) != cudaSuccess) return DEKF_ENOMEM;
          h->extra_bytes += (size_t)dekf_handle::kAhead * (2 * h->dm.n + 1) * sizeof(int32_t);
        }
        list = h->vo_list + (size_t)h->vo_slot * h->dm.n;
        count = h->vo_count + h->vo_slot;
        k_zero_i32<<<1, 1, 0, h->stream>>>(count);
        k_vo_compact<<<(h->dm.n + 255) / 256, 256, 0, h->stream>>>(in.vo_flag, h->dm.n, list, count);
        h->vo_list_valid = true;
      }
      ProfScope ps(h, 1);
      const int i_lo = adm.tile0 * kBlock, i_hi = h->asm_tiles >= 0 ? (adm.tile0 + h->asm_tiles) * kBlock : h->dm.n;
      int32_t *vstat = h->vo_stat + (size_t)h->vo_slot * h->dm.n;
      k_vo_sync<T><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(mc, h->dm, b, in, out, T_, list, count, i_lo, i_hi, vstat);
      k_assemble<T, Model, true><<<grid, kBlock, 0, h->stream>>>(mc, adm, b, in, out, T_, acc, h->asm_quat_copy, vstat);
      h->launches++;
    } else if (lean && in.vo_flag == nullptr) {
      // a tick without any VO message: the VO synchronisation is a no-op for every instance -- the kernel without that code
      ProfScope ps(h, 1);
      k_assemble<T, Model, true><<<grid, kBlock, 0, h->stream>>>(mc, adm, b, in, out, T_, acc, h->asm_quat_copy, nullptr);
    } else {
      ProfScope ps(h, 1);
      k_assemble<T, Model><<<grid, kBlock, 0, h->stream>>>(mc, adm, b, in, out, T_, acc, h->asm_quat_copy, nullptr);
    }
  }
  h->launches++;
  return 0;
}
template <typename T>
void launch_box(dekf_handle *h, const MheConst<T> &mc, const Buffers<T> &b, const Inputs &in, const Outputs &out, int T_, int32_t *st) {
  if (!h->box_team) {
    k_solve_box<T><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(mc, h->bc, h->dm, b, h->bb, in, out, T_, st);
    return;
  }
  k_box_prior<T><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(mc, h->dm, b, h->bb, h->tb, T_);
  const int warps = (h->dm.n + kTeamsPerWarp - 1) / kTeamsPerWarp, wpb = kTeamBlock / 32;
  k_box_team<T><<<(warps + wpb - 1) / wpb, kTeamBlock, 0, h->stream>>>(h->bc, h->dm, b, h->bb, h->tb, in, out, T_, st);
  h->launches += 1;  // the caller counts one launch per window solve
}

template <typename T, typename Model>
int launch_fused(dekf_handle *h, const EkfConst<T> &ec, const MheConst<T> &mc, const Buffers<T> &b, const Inputs &in,
                 const Outputs &out, int k, int T_, int32_t *status) {
  {
    ProfScope ps(h, 2);
    // role form (one warp per piece of the tick) for the plain MHE; the KF alternative and tapped handles keep the serial form
    if (h->dm.n <= h->roles_max && h->cfg.est_type == 0 && !h->cfg.debug_taps)
      k_fused_roles<T, Model><<<(h->dm.n + 31) / 32, (Model::NLEG + 2) * 32, 0, h->stream>>>(ec, mc, h->dm, b, in, out, k, T_, status);
    else
      k_fused<T, Model><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(ec, mc, h->dm, b, in, out, k, T_, status);
  }
  h->launches++;
  return 0;
}

template <typename T>
int do_assemble(dekf_handle *h, const MheConst<T> &mc, const Buffers<T> &b, const Inputs &in, const Outputs &out, int T_,
                const int32_t *acc) {
  switch (h->cfg.robot) {
    case DEKF_ROBOT_GO1: return launch_assemble<T, Go1Model<T>>(h, mc, b, in, out, T_, acc);
    case DEKF_ROBOT_CASSIE: return launch_assemble<T, CassieModel<T>>(h, mc, b, in, out, T_, acc);
    case DEKF_ROBOT_POGOX: return launch_assemble<T, PogoXModel<T>>(h, mc, b, in, out, T_, acc);
  }
  return DEKF_EINVAL;
}
template <typename T>
int do_fused(dekf_handle *h, const EkfConst<T> &ec, const MheConst<T> &mc, const Buffers<T> &b, const Inputs &in,
             const Outputs &out, int k, int T_, int32_t *status) {
  switch (h->cfg.robot) {
    case DEKF_ROBOT_GO1: return launch_fused<T, Go1Model<T>>(h, ec, mc, b, in, out, k, T_, status);
    case DEKF_ROBOT_CASSIE: return launch_fused<T, CassieModel<T>>(h, ec, mc, b, in, out, k, T_, status);
    case DEKF_ROBOT_POGOX: return launch_fused<T, PogoXModel<T>>(h, ec, mc, b, in, out, k, T_, status);
  }
  return DEKF_EINVAL;
}

// DIAGNOSIS ONLY (DEKF_DBG_CARVEOUT=1, DESIGN.md section 10): every kernel of the large-batch tick asks for the maximum shared-memory
// carve-out, i.e. the smallest L1 -- the setting under which the transient deviation of section 10 shows up within a few ticks.
template <typename K>
static void prefer_max_shared(K kernel) {
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
}
template <typename T>
static void prefer_max_shared_all() {
  prefer_max_shared(k_ekf<T, EKF_ALL>);
  prefer_max_shared(k_ekf<T, EKF_REPLAY>);
  prefer_max_shared(k_ekf<T, EKF_UPDATE>);
  prefer_max_shared(k_vo_sync<T>);
  prefer_max_shared(k_assemble<T, Go1Model<T>, false>);
  prefer_max_shared(k_assemble<T, Go1Model<T>, true>);
  prefer_max_shared(k_solve_tma<T>);
  prefer_max_shared(k_solve_incr_tma<T>);
  prefer_max_shared(k_solve_incr<T>);
  prefer_max_shared(k_solve<T>);
}
int check_T(dekf_handle *h, int32_t T_) {
  if (T_ != h->next_T) return fail(h, DEKF_ESTATE, "T must advance by one per call starting at 0 (initialize) -- call dekf_reset to restart");
  return DEKF_OK;
}

int validate(const dekf_config *c, std::string &why) {
  if (c->abi_version != DEKF_ABI_VERSION) { why = "abi_version mismatch"; return DEKF_EINVAL; }
  if (c->n_instances < 1) { why = "n_instances < 1"; return DEKF_EINVAL; }
  if (c->N < 2 || c->N > 4096) { why = "N out of range"; return DEKF_EINVAL; }
  if (c->rate < 1 || c->ekf_rate < 1) { why = "rate < 1"; return DEKF_EINVAL; }
  if (c->precision != DEKF_FP64 && c->precision != DEKF_FP32) { why = "precision"; return DEKF_EINVAL; }
  if (c->robot < DEKF_ROBOT_GO1 || c->robot > DEKF_ROBOT_POGOX) { why = "robot"; return DEKF_EINVAL; }
  if (c->num_legs != robot_num_legs(c->robot)) { why = "num_legs does not match the robot model"; return DEKF_EINVAL; }
  if (c->leg_odom_type != 0 && c->leg_odom_type != 1) { why = "leg_odom_type must be 0 or 1"; return DEKF_EINVAL; }
  if (c->leg_odom_type == 1 && c->precision != DEKF_FP64) { why = "leg_odom_type 1 is carried in information form and needs DEKF_FP64"; return DEKF_EINVAL; }
  if (c->leg_odom_type == 1 && c->v_box_enable) { why = "v_box_enable is built for leg_odom_type 0 only"; return DEKF_EINVAL; }
  if (c->est_type != 0 && c->est_type != 1) { why = "est_type must be 0 (MHE) or 1 (KF alternative)"; return DEKF_EINVAL; }
  if (c->ekf_hist_depth < 4) { why = "ekf_hist_depth < 4"; return DEKF_EINVAL; }
  if (c->window_solve != DEKF_SOLVE_FULL && c->window_solve != DEKF_SOLVE_INCREMENTAL) { why = "window_solve"; return DEKF_EINVAL; }
  if (c->v_box_enable) {
    if (c->est_type != 0) { why = "v_box_enable needs est_type 0 (the KF alternative has no constraints)"; return DEKF_EINVAL; }
    for (int i = 0; i < 3; ++i)
      if (!(c->v_box_lo[i] < c->v_box_hi[i])) { why = "v_box_lo must be < v_box_hi"; return DEKF_EINVAL; }
  }
  if (c->x_box_mask) {
    if (c->x_box_mask & ~0x1ff) { why = "x_box_mask has 9 bits (p_s, v_s, accel bias)"; return DEKF_EINVAL; }
    if (c->est_type != 0 || c->leg_odom_type != 0) { why = "x_box_mask needs est_type 0 and leg_odom_type 0"; return DEKF_EINVAL; }
    for (int a = 0; a < 9; ++a)
      if (((c->x_box_mask >> a) & 1) && !(c->x_box_lo[a] < c->x_box_hi[a])) { why = "x_box_lo must be < x_box_hi"; return DEKF_EINVAL; }
  }
  return DEKF_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// extern "C"
// ------------------------------------------------------------------------------------------------
extern "C" {

int dekf_config_default_go1(dekf_config *cfg) {
  if (!cfg) return DEKF_EINVAL;
  fill_go1_defaults(cfg);
  return DEKF_OK;
}
int dekf_config_default_cassie(dekf_config *cfg) {
  if (!cfg) return DEKF_EINVAL;
  fill_go1_defaults(cfg);
  cfg->robot = DEKF_ROBOT_CASSIE;
  cfg->num_legs = 2;
  cfg->contact_effort_threshold = 150.0;
  cfg->p_ib[0] = cfg->p_ib[1] = cfg->p_ib[2] = 0.0;
  cfg->p_imu_2_opti[0] = cfg->p_imu_2_opti[1] = cfg->p_imu_2_opti[2] = 0.0;  // the Go1 mocap marker offset means nothing here
  return DEKF_OK;
}
int dekf_config_default_pogox(dekf_config *cfg) {
  if (!cfg) return DEKF_EINVAL;
  fill_go1_defaults(cfg);
  cfg->robot = DEKF_ROBOT_POGOX;
  cfg->num_legs = 1;
  cfg->contact_effort_threshold = 100.0;
  cfg->p_ib[0] = cfg->p_ib[1] = cfg->p_ib[2] = 0.0;
  cfg->p_imu_2_opti[0] = cfg->p_imu_2_opti[1] = cfg->p_imu_2_opti[2] = 0.0;
  return DEKF_OK;
}

int dekf_create(const dekf_config *cfg, dekf_handle **out) {
  if (!cfg || !out) return DEKF_EINVAL;
  *out = nullptr;
  dekf_handle *h = new (std::nothrow) dekf_handle();
  if (!h) return DEKF_ENOMEM;
  std::string why;
  int rc = validate(cfg, why);
  if (rc != DEKF_OK) {
    std::fprintf(stderr, "dekf_create: %s\n", why.c_str());
    delete h;
    return rc;
  }
  h->cfg = *cfg;
  h->dm = make_dims(*cfg);
  h->nl = robot_num_legs(cfg->robot);
  h->nj = robot_nj(cfg->robot);
  h->nq = h->nl * h->nj;
  h->ds = state_dim(*cfg);
  h->f32 = cfg->precision == DEKF_FP32;
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev <= 0 || cfg->device < 0 || cfg->device >= ndev) {
    std::fprintf(stderr, "dekf_create: no usable CUDA device (%s); there is no CPU fallback\n",
                 ce == cudaSuccess ? "bad ordinal" : cudaGetErrorString(ce));
    delete h;
    return DEKF_ENODEV;
  }
  if (cudaSetDevice(cfg->device) != cudaSuccess) {
    delete h;
    return DEKF_ENODEV;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major < 10) {
    std::fprintf(stderr, "dekf_create: device is not sm_100-class (this library carries sm_100a code only)\n");
    delete h;
    return DEKF_ENODEV;
  }
  if (const char *e = std::getenv("DEKF_FUSED_MAX_N")) h->fused_max = std::atoi(e);
  if (const char *e = std::getenv("DEKF_NO_TMA")) h->use_tma = std::atoi(e) == 0;
  if (const char *e = std::getenv("DEKF_NO_SPLIT")) h->no_split = std::atoi(e) != 0;
  if (const char *e = std::getenv("DEKF_SPLIT_TILES")) h->split_tiles_env = std::atoi(e);
  if (const char *e = std::getenv("DEKF_VO_COMPACT")) h->vo_compact = std::atoi(e) != 0;
  if (std::getenv("DEKF_EKF_SERIAL")) h->ekf_serial = true;
  if (std::getenv("DEKF_DBG_CARVEOUT")) {
    prefer_max_shared_all<double>();
    prefer_max_shared_all<float>();
    prefer_max_shared(k_vo_compact);
    prefer_max_shared(k_zero_i32);
  }
  if (const char *e = std::getenv("DEKF_RUN_PIPELINE_MIN_N")) h->run_pipeline_min = std::atoi(e);
  if (const char *e = std::getenv("DEKF_ROLES_MAX_N")) h->roles_max = std::atoi(e);
  if (const char *e = std::getenv("DEKF_NO_ASM_SPLIT")) h->no_asm_split = std::atoi(e) != 0;
  if (const char *e = std::getenv("DEKF_SPLIT_WAYS")) h->split_ways_env = std::atoi(e);
  if (const char *e = std::getenv("DEKF_PRIO")) h->prio_mode = std::atoi(e);
  if (const char *e = std::getenv("DEKF_HOST_RAMP")) h->host_ramp = std::atoi(e) != 0;
  if (const char *e = std::getenv("DEKF_HOST_CHUNK")) h->host_chunk = std::atoi(e) > 0 ? std::atoi(e) : 8;
  ce = cudaFuncSetAttribute(k_solve_tma<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_tma_smem_bytes<double>());
  if (ce == cudaSuccess)
    ce = cudaFuncSetAttribute(k_solve_tma<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_tma_smem_bytes<float>());
  if (ce == cudaSuccess)
    ce = cudaFuncSetAttribute(k_solve_incr_tma<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_tma_smem_bytes<double>());
  if (ce == cudaSuccess)
    ce = cudaFuncSetAttribute(k_solve_incr_tma<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_tma_smem_bytes<float>());
  if (ce != cudaSuccess) {
    std::fprintf(stderr, "dekf_create: cudaFuncSetAttribute(k_solve_tma): %s\n", cudaGetErrorString(ce));
    delete h;
    return DEKF_ECUDA;
  }
  h->ec64 = make_ekf_const<double>(*cfg);
  h->mc64 = make_mhe_const<double>(*cfg);
  h->ec32 = make_ekf_const<float>(*cfg);
  h->mc32 = make_mhe_const<float>(*cfg);
  h->slab_bytes = h->f32 ? carve<float>(h->b32, h->dm, nullptr) : carve<double>(h->b64, h->dm, nullptr);
  const size_t n = (size_t)cfg->n_instances;
  auto bail = [&](int code, const char *what, cudaError_t e) {
    std::fprintf(stderr, "dekf_create: %s: %s\n", what, cudaGetErrorString(e));
    dekf_destroy(h);
    return code;
  };
  if ((ce = cudaMalloc(&h->slab, h->slab_bytes)) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc(state)", ce);
  if ((ce = cudaMemsetAsync(h->slab, 0, h->slab_bytes, 0)) != cudaSuccess) return bail(DEKF_ECUDA, "memset", ce);
  if (h->f32)
    carve<float>(h->b32, h->dm, (char *)h->slab);
  else
    carve<double>(h->b64, h->dm, (char *)h->slab);
  if (h->use_tma) {
    // cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
    typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    ce = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (ce != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess) {
      std::fprintf(stderr, "dekf_create: cuTensorMapEncodeTiled is not available from this driver\n");
      dekf_destroy(h);
      return DEKF_ECUDA;
    }
    const size_t elt = h->f32 ? sizeof(float) : sizeof(double);
    void *base = h->f32 ? (void *)h->b32.win : (void *)h->b64.win;
    const cuuint64_t gdim[2] = {(cuuint64_t)h->dm.ns, (cuuint64_t)h->dm.NW * REC_SIZE};
    const cuuint64_t gstride[1] = {(cuuint64_t)h->dm.ns * elt};
    // one TMA box = the stage record of one pipeline's instances: a warp (32) with per-warp pipelines, else the CTA's tile
    const cuuint32_t box[2] = {(cuuint32_t)((h->f32 ? SolveCfg<float>::kPerWarp : SolveCfg<double>::kPerWarp) ? 32 : kTile), (cuuint32_t)REC_SIZE};
    const cuuint32_t estr[2] = {1, 1};
    CUresult cr = ((encode_fn)fn)(&h->tmap, h->f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, gdim,
                                  gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) {
      std::fprintf(stderr, "dekf_create: cuTensorMapEncodeTiled failed (%d)\n", (int)cr);
      dekf_destroy(h);
      return DEKF_ECUDA;
    }
  }
  h->extra_bytes = 0;
  if (h->mc64.window_solve == 1) {
    const size_t ns = (size_t)h->dm.ns, elt = h->f32 ? sizeof(float) : sizeof(double);
    const size_t ck = (size_t)h->dm.NW * 54 * ns * elt;
    if ((ce = cudaMalloc(&h->ckpt_mem, ck)) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc(checkpoint ring)", ce);
    if ((ce = cudaMalloc((void **)&h->resweep_mem, 2 * ns * sizeof(int32_t))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    if ((ce = cudaMemset(h->ckpt_mem, 0, ck)) != cudaSuccess) return bail(DEKF_ECUDA, "memset", ce);
    h->b64.ckpt = (double *)h->ckpt_mem;
    h->b32.ckpt = (float *)h->ckpt_mem;
    h->b64.resweep = h->b32.resweep = h->resweep_mem;
    h->extra_bytes += ck + 2 * ns * sizeof(int32_t);
  }
  h->fc = make_foot_const(*cfg);
  if (cfg->leg_odom_type == 1) {
    const size_t ns = (size_t)h->dm.ns, ds = (size_t)h->ds;
    const size_t leg = (size_t)h->dm.NW * foot_rec_size(h->nl) * ns * sizeof(double), am = ds * (ds + 1) / 2 * ns * sizeof(double);
    if ((ce = cudaMalloc((void **)&h->fb.leg, leg)) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc(foot ring)", ce);
    if ((ce = cudaMalloc((void **)&h->fb.arr_M, am)) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    if ((ce = cudaMalloc((void **)&h->fb.arr_m, ds * ns * sizeof(double))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    cudaMemset(h->fb.leg, 0, leg);
    cudaMemset(h->fb.arr_M, 0, am);
    cudaMemset(h->fb.arr_m, 0, ds * ns * sizeof(double));
    h->b64.foot_leg = h->fb.leg;
    h->extra_bytes += leg + am + ds * ns * sizeof(double);
  }
  h->bc = make_box_const(*cfg);
  {
    int sms = 0, per_sm = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
    if (h->f32)
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_solve_tma<float>, kTile, solve_tma_smem_bytes<float>());
    else
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_solve_tma<double>, kTile, solve_tma_smem_bytes<double>());
    h->solve_slots = sms * per_sm;
  }
  if (const char *e = std::getenv("DEKF_FOOT_SERIAL")) h->foot_team = std::atoi(e) == 0;
  if (h->bc.enable) {
    const size_t ns = (size_t)h->dm.ns;
    const size_t fac = (size_t)h->dm.N * BOX_FAC * ns * sizeof(double), act = (size_t)h->dm.NW * ns;
    if (h->bc.general) {  // bounds outside v_s: 18-bit masks, one thread per instance
      if ((ce = cudaMalloc((void **)&h->bb.act32, act * sizeof(uint32_t))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
      h->extra_bytes += act * sizeof(uint32_t);
      h->box_team = false;
    }
    if ((ce = cudaMalloc((void **)&h->bb.fac, fac)) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc(box factor scratch)", ce);
    if ((ce = cudaMalloc((void **)&h->bb.act, act)) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    if ((ce = cudaMalloc((void **)&h->bb.iters, ns * sizeof(int32_t))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    if ((ce = cudaMalloc((void **)&h->bb.nactive, ns * sizeof(int32_t))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    if ((ce = cudaMalloc((void **)&h->bb.capped, ns)) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    h->extra_bytes += fac + act + 2 * ns * sizeof(int32_t) + ns;
    if (const char *e = std::getenv("DEKF_BOX_SERIAL")) h->box_team = h->box_team && std::atoi(e) == 0;
    if (h->box_team) {
      const size_t tfac = (size_t)h->dm.N * BOX_TFAC * ns * sizeof(double);
      if ((ce = cudaMalloc((void **)&h->tb.prior, ns * BOX_PRIOR * sizeof(double))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
      if ((ce = cudaMalloc((void **)&h->tb.fac, tfac)) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc(box team scratch)", ce);
      h->extra_bytes += ns * BOX_PRIOR * sizeof(double) + tfac;
    }
  }
  if (cfg->debug_taps) {
    if ((ce = cudaMalloc((void **)&h->tap_b_meas, (size_t)3 * h->nl * n * sizeof(double))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    if ((ce = cudaMalloc((void **)&h->tap_Q_meas, (size_t)6 * h->nl * n * sizeof(double))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    if ((ce = cudaMalloc((void **)&h->tap_vo, (size_t)8 * n * sizeof(int32_t))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    if ((ce = cudaMalloc((void **)&h->tap_ekf, (size_t)3 * n * sizeof(int32_t))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    h->extra_bytes += (size_t)9 * h->nl * n * sizeof(double) + (size_t)11 * n * sizeof(int32_t);
  }
  if (cfg->kf_export_gain && cfg->est_type == 1 && cfg->leg_odom_type == 0 && !cfg->debug_taps) {
    if ((ce = cudaMalloc((void **)&h->kf_Q, (size_t)6 * h->nl * n * sizeof(double))) != cudaSuccess) return bail(DEKF_ENOMEM, "cudaMalloc", ce);
    h->extra_bytes += (size_t)6 * h->nl * n * sizeof(double);
  }
  if ((ce = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(DEKF_ECUDA, "cudaStreamCreate", ce);
  h->own_stream = true;
  if ((ce = cudaDeviceSynchronize()) != cudaSuccess) return bail(DEKF_ECUDA, "sync", ce);
  rc = dekf_reset(h);
  if (rc != DEKF_OK) {
    std::fprintf(stderr, "dekf_create: reset failed: %s\n", h->err.c_str());
    dekf_destroy(h);
    return rc;
  }
  *out = h;
  return DEKF_OK;
}

int dekf_destroy(dekf_handle *h) {
  if (!h) return DEKF_EINVAL;
  cudaSetDevice(h->cfg.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  cudaFree(h->slab);
  cudaFree(h->fb.leg);
  cudaFree(h->fb.arr_M);
  cudaFree(h->fb.arr_m);
  cudaFree(h->ckpt_mem);
  cudaFree(h->win_scr);
  cudaFree(h->foot_win_ring);
  cudaFree(h->cross_ring);
  cudaFree(h->resweep_mem);
  cudaFree(h->bb.fac);
  cudaFree(h->tb.prior);
  cudaFree(h->tb.fac);
  cudaFree(h->bb.act);
  cudaFree(h->bb.act32);
  cudaFree(h->bb.iters);
  cudaFree(h->bb.nactive);
  cudaFree(h->bb.capped);
  cudaFree(h->row_V);
  free_stage_set(h->stage[0]);
  free_stage_set(h->stage[1]);
  free_chunk_set(h->chunk[0]);
  free_chunk_set(h->chunk[1]);
  cudaFree(h->get_scratch);
  cudaFree(h->kf_Q);
  if (h->hmap) cudaFreeHost(h->hmap);
  if (h->s_ekf) cudaStreamDestroy(h->s_ekf);
  for (int r = 0; r < dekf_handle::kMaxWays; ++r)
    if (h->s_sol[r]) cudaStreamDestroy(h->s_sol[r]);
  for (int k = 0; k < dekf_handle::kAhead; ++k)
    for (int r = 0; r < dekf_handle::kMaxWays; ++r)
      if (h->ev_solw[r][k]) cudaEventDestroy(h->ev_solw[r][k]);
  if (h->s_asm) cudaStreamDestroy(h->s_asm);
  for (int r = 1; r < dekf_handle::kMaxWays; ++r)
    if (h->s_asmw[r]) cudaStreamDestroy(h->s_asmw[r]);
  for (int k = 0; k < dekf_handle::kAhead; ++k)
    for (int r = 0; r < dekf_handle::kMaxWays; ++r)
      if (h->ev_asmw[r][k]) cudaEventDestroy(h->ev_asmw[r][k]);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  cudaFree(h->quat_ring);
  cudaFree(h->status_ring);
  cudaFree(h->vo_list);
  cudaFree(h->vo_stat);
  cudaFree(h->vo_count);
  for (int k = 0; k < dekf_handle::kAhead; ++k) {
    if (h->ev_ekf[k]) cudaEventDestroy(h->ev_ekf[k]);
  }
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
  if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
  for (int k = 0; k < 2; ++k) {
    if (h->ev_h2d[k]) cudaEventDestroy(h->ev_h2d[k]);
    if (h->ev_comp[k]) cudaEventDestroy(h->ev_comp[k]);
    if (h->ev_d2h[k]) cudaEventDestroy(h->ev_d2h[k]);
  }
  cudaFree(h->tap_b_meas);
  cudaFree(h->tap_Q_meas);
  cudaFree(h->tap_vo);
  cudaFree(h->tap_ekf);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  for (auto &r : h->prof_recs) {
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
  }
  for (auto &r : h->prof_free) {
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
  }
  delete h;
  return DEKF_OK;
}

int dekf_reset(dekf_handle *h) {
  if (!h) return DEKF_EINVAL;
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemsetAsync(h->slab, 0, h->slab_bytes, h->stream));
  if (h->fb.arr_M) {
    CK(cudaMemsetAsync(h->fb.arr_M, 0, (size_t)h->ds * (h->ds + 1) / 2 * h->dm.ns * sizeof(double), h->stream));
    CK(cudaMemsetAsync(h->fb.arr_m, 0, (size_t)h->ds * h->dm.ns * sizeof(double), h->stream));
  }
  if (h->bb.act) {
    CK(cudaMemsetAsync(h->bb.act, 0, (size_t)h->dm.NW * h->dm.ns, h->stream));
    if (h->bb.act32) CK(cudaMemsetAsync(h->bb.act32, 0, (size_t)h->dm.NW * h->dm.ns * sizeof(uint32_t), h->stream));
    CK(cudaMemsetAsync(h->bb.iters, 0, (size_t)h->dm.ns * sizeof(int32_t), h->stream));
    CK(cudaMemsetAsync(h->bb.nactive, 0, (size_t)h->dm.ns * sizeof(int32_t), h->stream));
    CK(cudaMemsetAsync(h->bb.capped, 0, (size_t)h->dm.ns, h->stream));
  }
  if (h->f32)
    k_init_state<float><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->ec32, h->mc32, h->dm, h->b32);
  else
    k_init_state<double><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->ec64, h->mc64, h->dm, h->b64);
  h->launches++;
  CK(cudaGetLastError());
  h->ekf_k = 0;
  h->next_T = 0;
  return DEKF_OK;
}

int dekf_set_stream(dekf_handle *h, void *cuda_stream) {
  if (!h) return DEKF_EINVAL;
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  h->stream = (cudaStream_t)cuda_stream;
  h->own_stream = false;
  return DEKF_OK;
}
void *dekf_get_stream(dekf_handle *h) { return h ? (void *)h->stream : nullptr; }
const char *dekf_last_error(const dekf_handle *h) { return h ? h->err.c_str() : "null handle"; }
int dekf_num_joints(const dekf_handle *h) { return h ? h->nq : DEKF_EINVAL; }
int dekf_state_dim(const dekf_handle *h) { return h ? h->ds : DEKF_EINVAL; }
int64_t dekf_launch_count(const dekf_handle *h) { return h ? h->launches : 0; }
int64_t dekf_device_bytes(const dekf_handle *h) { return h ? (int64_t)(h->slab_bytes + h->extra_bytes) : 0; }

// one EKF tick of all instances on `stream`; status_state: where the tick's status bits are kept for the MHE to OR in
static int ekf_launch(dekf_handle *h, const dekf_inputs *in, const dekf_outputs *out, int32_t *status_state,
                      cudaStream_t stream) {
  const Inputs di = to_inputs(in);
  const Outputs dout = to_outputs(h, out);
  int32_t *st = out ? out->status : nullptr;
  const int g = grid_for(h->dm.n);
  int32_t *ss = status_state ? status_state : (h->f32 ? h->b32.status : h->b64.status);
  // A tick of a large batch that carries VO poses: compact the flagged instances, replay them densely, then the ordinary
  // update of everybody (ragged arrival: ~15 % of the instances are flagged on EVERY tick; one launch made every warp walk the
  // replay loop).  Lock-step arrival flags all instances: the replay launch then simply covers them all.
  const bool split = h->vo_compact && di.vo_flag != nullptr && !h->cfg.debug_taps && h->dm.n > h->fused_max;
  h->vo_list_valid = false;
  if (split) {
    if (!h->vo_list) {
      CK(cudaMalloc((void **)&h->vo_list, (size_t)dekf_handle::kAhead * h->dm.n * sizeof(int32_t)));
      CK(cudaMalloc((void **)&h->vo_stat, (size_t)dekf_handle::kAhead * h->dm.n * sizeof(int32_t)));
      CK(cudaMalloc((void **)&h->vo_count, dekf_handle::kAhead * sizeof(int32_t)));
      h->extra_bytes += (size_t)dekf_handle::kAhead * (2 * h->dm.n + 1) * sizeof(int32_t);
    }
    int32_t *list = h->vo_list + (size_t)h->vo_slot * h->dm.n, *count = h->vo_count + h->vo_slot;
    k_zero_i32<<<1, 1, 0, stream>>>(count);
    k_vo_compact<<<(h->dm.n + 255) / 256, 256, 0, stream>>>(di.vo_flag, h->dm.n, list, count);
    ProfScope ps(h, 0, stream);
    if (h->f32) {
      k_ekf<float, EKF_REPLAY><<<g, kBlock, 0, stream>>>(h->ec32, h->dm, h->b32, di, dout, h->ekf_k, ss, st, list, count);
      k_ekf<float, EKF_UPDATE><<<g, kBlock, 0, stream>>>(h->ec32, h->dm, h->b32, di, dout, h->ekf_k, ss, st, list, count);
    } else {
      k_ekf<double, EKF_REPLAY><<<g, kBlock, 0, stream>>>(h->ec64, h->dm, h->b64, di, dout, h->ekf_k, ss, st, list, count);
      k_ekf<double, EKF_UPDATE><<<g, kBlock, 0, stream>>>(h->ec64, h->dm, h->b64, di, dout, h->ekf_k, ss, st, list, count);
    }
    h->launches += 2;
    h->vo_list_valid = true;
  } else if (di.vo_flag == nullptr && !h->cfg.debug_taps) {
    // no VO pose on this tick: the update half alone IS the whole tick (no replay code in the kernel: no spill frame)
    ProfScope ps(h, 0, stream);
    if (h->f32)
      k_ekf<float, EKF_UPDATE><<<g, kBlock, 0, stream>>>(h->ec32, h->dm, h->b32, di, dout, h->ekf_k, ss, st, nullptr, nullptr);
    else
      k_ekf<double, EKF_UPDATE><<<g, kBlock, 0, stream>>>(h->ec64, h->dm, h->b64, di, dout, h->ekf_k, ss, st, nullptr, nullptr);
  } else {
    ProfScope ps(h, 0, stream);
    if (h->f32)
      k_ekf<float><<<g, kBlock, 0, stream>>>(h->ec32, h->dm, h->b32, di, dout, h->ekf_k, ss, st, nullptr, nullptr);
    else
      k_ekf<double><<<g, kBlock, 0, stream>>>(h->ec64, h->dm, h->b64, di, dout, h->ekf_k, ss, st, nullptr, nullptr);
  }
  h->launches++;
  CK(cudaGetLastError());
  h->ekf_k++;
  return DEKF_OK;
}

int dekf_ekf_step(dekf_handle *h, const dekf_inputs *in, const dekf_outputs *out) {
  if (!h || !in || !in->gyro || !in->accel || !in->imu_time) return fail(h, DEKF_EINVAL, "dekf_ekf_step: null input");
  if (in->vo_flag && (!in->vo_quat || !in->vo_time_now)) return fail(h, DEKF_EINVAL, "dekf_ekf_step: vo_flag without vo_quat/vo_time_now");
  CK(cudaSetDevice(h->cfg.device));
  h->vo_slot = 0;
  const int rc = ekf_launch(h, in, out, nullptr, h->stream);
  h->vo_list_valid = false;  // the list belonged to this EKF tick only
  return rc;
}

// phases: 1 = stage assembly, 2 = window solve, 3 = both (on h->stream)
static int mhe_step_impl(dekf_handle *h, int32_t T_, const dekf_inputs *in, const dekf_outputs *out, const int32_t *acc,
                         int phases = 3) {
  if (!in->gyro || !in->accel || !in->imu_time || !in->joint_pos || !in->joint_vel || !in->foot_force)
    return fail(h, DEKF_EINVAL, "dekf_mhe_step: null input");
  if (in->vo_flag && (!in->vo_time_pre || !in->vo_time_now || !in->vo_rel_p))
    return fail(h, DEKF_EINVAL, "dekf_mhe_step: vo_flag without vo_time_pre/vo_time_now/vo_rel_p");
  const Inputs di = to_inputs(in);
  const Outputs dout = to_outputs(h, out);
  int32_t *st = out ? out->status : nullptr;
  int rc;
  const bool tma = h->use_tma && T_ >= 1;
  const bool kf = h->cfg.est_type == 1;
  const int tiles = h->dm.ns / kTile;
  Dims rdm = h->dm;  // k_solve_tma may cover a tile range only (dekf_run splits the batch at the last full wave)
  rdm.tile0 = h->solve_tiles >= 0 ? h->solve_tile0 : 0;
  const int rtiles = h->solve_tiles >= 0 ? h->solve_tiles : tiles;
  // incremental solve on a tick that carries VO messages: TMA-staged re-sweep from the CTA's earliest restart stage
  const bool resweep_tick = h->mc64.window_solve == 1 && tma && T_ >= 2 && di.vo_flag != nullptr && !kf && !h->bc.enable &&
                            h->cfg.leg_odom_type == 0;
  if (phases & 1) {
    rc = h->f32 ? do_assemble<float>(h, h->mc32, h->b32, di, dout, T_, acc) : do_assemble<double>(h, h->mc64, h->b64, di, dout, T_, acc);
    if (rc) return fail(h, rc, "assemble");
    CK(cudaGetLastError());
  }
  if (!(phases & 2)) return DEKF_OK;
  if (h->f32) {
    ProfScope ps(h, resweep_tick ? 3 : 2);
    if (kf)
      k_kf<float><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->mc32, h->dm, h->b32, di, dout, T_, st);
    else if (h->bc.enable)
      launch_box<float>(h, h->mc32, h->b32, di, dout, T_, st);
    else if (resweep_tick)
      k_solve_incr_tma<float><<<tiles, kTile, solve_tma_smem_bytes<float>(), h->stream>>>(h->tmap, h->mc32, h->dm, h->b32, di, dout, T_, st);
    else if (h->mc32.window_solve == 1)
      k_solve_incr<float><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->mc32, h->dm, h->b32, di, dout, T_, st);
    else if (tma)
      k_solve_tma<float><<<rtiles, kTile, solve_tma_smem_bytes<float>(), h->stream>>>(h->tmap, h->mc32, rdm, h->b32, di, dout, T_, st);
    else
      k_solve<float><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->mc32, h->dm, h->b32, di, dout, T_, st);
  } else {
    ProfScope ps(h, resweep_tick ? 3 : 2);
    if (h->cfg.leg_odom_type == 1) {
      const int g = grid_for(h->dm.n);
      const int gt = (h->dm.n + kTeamBlock / 32 - 1) / (kTeamBlock / 32);  // one warp per instance
      if (h->foot_team && h->nl == 4)
        k_foot_team<double, 4><<<gt, kTeamBlock, 0, h->stream>>>(h->fc, h->dm, h->b64, h->fb, di, dout, T_, st);
      else if (h->foot_team && h->nl == 2)
        k_foot_team<double, 2><<<gt, kTeamBlock, 0, h->stream>>>(h->fc, h->dm, h->b64, h->fb, di, dout, T_, st);
      else if (h->foot_team)
        k_foot_team<double, 1><<<gt, kTeamBlock, 0, h->stream>>>(h->fc, h->dm, h->b64, h->fb, di, dout, T_, st);
      else if (h->nl == 4)
        k_solve_foot<double, 4><<<g, kBlock, 0, h->stream>>>(h->fc, h->dm, h->b64, h->fb, di, dout, T_, st);
      else if (h->nl == 2)
        k_solve_foot<double, 2><<<g, kBlock, 0, h->stream>>>(h->fc, h->dm, h->b64, h->fb, di, dout, T_, st);
      else
        k_solve_foot<double, 1><<<g, kBlock, 0, h->stream>>>(h->fc, h->dm, h->b64, h->fb, di, dout, T_, st);
    } else if (kf)
      k_kf<double><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->mc64, h->dm, h->b64, di, dout, T_, st);
    else if (h->bc.enable)
      launch_box<double>(h, h->mc64, h->b64, di, dout, T_, st);
    else if (resweep_tick)
      k_solve_incr_tma<double><<<tiles, kTile, solve_tma_smem_bytes<double>(), h->stream>>>(h->tmap, h->mc64, h->dm, h->b64, di, dout, T_, st);
    else if (h->mc64.window_solve == 1)
      k_solve_incr<double><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->mc64, h->dm, h->b64, di, dout, T_, st);
    else if (tma)
      k_solve_tma<double><<<rtiles, kTile, solve_tma_smem_bytes<double>(), h->stream>>>(h->tmap, h->mc64, rdm, h->b64, di, dout, T_, st);
    else
      k_solve<double><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->mc64, h->dm, h->b64, di, dout, T_, st);
  }
  h->launches++;
  CK(cudaGetLastError());
  h->next_T = T_ + 1;
  return DEKF_OK;
}

int dekf_mhe_step(dekf_handle *h, int32_t T_, const dekf_inputs *in, const dekf_outputs *out) {
  if (!h || !in) return fail(h, DEKF_EINVAL, "dekf_mhe_step: null argument");
  int rc = check_T(h, T_);
  if (rc) return rc;
  CK(cudaSetDevice(h->cfg.device));
  h->vo_slot = 0;
  h->vo_list_valid = false;  // stepped on its own: the assembly compacts this call's vo_flag itself
  return mhe_step_impl(h, T_, in, out, nullptr);
}

int dekf_step(dekf_handle *h, int32_t T_, const dekf_inputs *in, const dekf_outputs *out) {
  if (!h || !in) return fail(h, DEKF_EINVAL, "dekf_step: null argument");
  int rc = check_T(h, T_);
  if (rc) return rc;
  if (!in->gyro || !in->accel || !in->imu_time || !in->joint_pos || !in->joint_vel || !in->foot_force)
    return fail(h, DEKF_EINVAL, "dekf_step: null input");
  if (in->vo_flag && (!in->vo_quat || !in->vo_time_pre || !in->vo_time_now || !in->vo_rel_p))
    return fail(h, DEKF_EINVAL, "dekf_step: vo_flag without the VO arrays");
  CK(cudaSetDevice(h->cfg.device));
  dekf_inputs in2 = *in;
  in2.quat = nullptr;  // lock-step: the MHE consumes this tick's EKF quaternion
  if (h->dm.n <= h->fused_max && !h->bc.enable && h->cfg.leg_odom_type == 0) {
    const Inputs di = to_inputs(&in2);
    const Outputs dout = to_outputs(h, out);
    int32_t *st = out ? out->status : nullptr;
    if (h->f32)
      rc = do_fused<float>(h, h->ec32, h->mc32, h->b32, di, dout, h->ekf_k, T_, st);
    else
      rc = do_fused<double>(h, h->ec64, h->mc64, h->b64, di, dout, h->ekf_k, T_, st);
    if (rc) return fail(h, rc, "fused");
    CK(cudaGetLastError());
    h->ekf_k++;
    h->next_T = T_ + 1;
    return DEKF_OK;
  }
  dekf_outputs o_ekf;
  std::memset(&o_ekf, 0, sizeof(o_ekf));
  if (out) o_ekf.quat = out->quat;
  int32_t *slot = (h->f32 ? h->b32.status : h->b64.status) + (size_t)(T_ & 1) * h->dm.ns;  // tick_status(T_)
  h->vo_slot = 0;
  rc = ekf_launch(h, &in2, &o_ekf, slot, h->stream);
  if (rc) return rc;
  rc = mhe_step_impl(h, T_, &in2, out, slot);  // same vo_flag, same stream: the assembly reuses the EKF launch's list
  h->vo_list_valid = false;
  return rc;
}

int dekf_synchronize(dekf_handle *h) {
  if (!h) return DEKF_EINVAL;
  CK(cudaStreamSynchronize(h->stream));
  return DEKF_OK;
}

}  // extern "C"

// ---- host-pointer entry points --------------------------------------------------------------------------------
namespace {
enum HostKind { HK_STEP = 0, HK_MHE = 1, HK_EKF = 2 };
constexpr int kNumIn = 11;  // gyro accel imu_time joint_pos joint_vel foot_force | vo_quat vo_time_pre vo_time_now vo_rel_p | quat

void in_counts(const dekf_handle *h, size_t cnt[kNumIn]) {
  const size_t n = (size_t)h->dm.n;
  const size_t c[kNumIn] = {3 * n, 3 * n, n, (size_t)h->nq * n, (size_t)h->nq * n, (size_t)h->nl * n, 4 * n, n, n, 3 * n, 4 * n};
  for (int a = 0; a < kNumIn; ++a) cnt[a] = c[a];
}

int alloc_stage_set(dekf_handle *h, StageSet &ss) {
  if (ss.in) return DEKF_OK;
  const size_t n = (size_t)h->dm.n;
  size_t cnt[kNumIn], tot = 0;
  in_counts(h, cnt);
  for (int a = 0; a < kNumIn; ++a) tot += cnt[a];
  CK(cudaMalloc((void **)&ss.in, tot * sizeof(double)));
  CK(cudaMalloc((void **)&ss.flag, n));
  CK(cudaMalloc((void **)&ss.out, (size_t)(7 + h->ds) * n * sizeof(double)));
  CK(cudaMalloc((void **)&ss.contact, (size_t)h->nl * n));
  CK(cudaMalloc((void **)&ss.status, n * sizeof(int32_t)));
  h->extra_bytes += (tot + (size_t)(7 + h->ds) * n) * sizeof(double) + n + (size_t)h->nl * n + n * sizeof(int32_t);
  return DEKF_OK;
}
void free_chunk_set(ChunkSet &cs) {
  cudaFree(cs.in);
  cudaFree(cs.in_f32);
  cudaFree(cs.flag);
  cudaFree(cs.out);
  cudaFree(cs.contact);
  cudaFree(cs.status);
  cudaFree(cs.out_f32);
  cs = ChunkSet();
}
int alloc_chunk_set(dekf_handle *h, ChunkSet &cs, int cap) {
  if (cs.cap >= cap) return DEKF_OK;
  free_chunk_set(cs);
  const size_t n = (size_t)h->dm.n, c = (size_t)cap;
  const size_t in_rows = 16 + 2 * (size_t)h->nq + (size_t)h->nl;  // 3+3+1+nq+nq+nl + 4+1+1+3
  CK(cudaMalloc((void **)&cs.in, c * in_rows * n * sizeof(double)));
  CK(cudaMalloc((void **)&cs.flag, c * n));
  CK(cudaMalloc((void **)&cs.out, c * (size_t)(7 + h->ds) * n * sizeof(double)));
  CK(cudaMalloc((void **)&cs.contact, c * (size_t)h->nl * n));
  CK(cudaMalloc((void **)&cs.status, c * n * sizeof(int32_t)));
  cs.cap = cap;
  h->extra_bytes += c * ((in_rows + 7 + h->ds) * n * sizeof(double) + n + (size_t)h->nl * n + n * sizeof(int32_t));
  return DEKF_OK;
}
void free_stage_set(StageSet &ss) {
  cudaFree(ss.in);
  cudaFree(ss.flag);
  cudaFree(ss.out);
  cudaFree(ss.contact);
  cudaFree(ss.status);
  ss = StageSet();
}

// H2D copies of one tick's inputs on stream `st`; `din` receives the device pointers (NULL where the host gave NULL)
int stage_inputs(dekf_handle *h, const StageSet &ss, const dekf_inputs *in, cudaStream_t st, dekf_inputs *din) {
  const size_t n = (size_t)h->dm.n;
  size_t cnt[kNumIn];
  in_counts(h, cnt);
  const bool vo = in->vo_flag != nullptr;
  const double *src[kNumIn] = {in->gyro, in->accel, in->imu_time, in->joint_pos, in->joint_vel, in->foot_force,
                               vo ? in->vo_quat : nullptr, vo ? in->vo_time_pre : nullptr, vo ? in->vo_time_now : nullptr,
                               vo ? in->vo_rel_p : nullptr, in->quat};
  double *dst[kNumIn];
  size_t off = 0;
  for (int a = 0; a < kNumIn; ++a) {
    dst[a] = ss.in + off;
    off += cnt[a];
  }
  // host ranges that are contiguous in the packed order go as single copies
  int a = 0;
  while (a < kNumIn) {
    if (!src[a]) {
      ++a;
      continue;
    }
    int e = a;
    size_t total = cnt[a];
    while (e + 1 < kNumIn && src[e + 1] && src[e + 1] == src[e] + cnt[e]) {
      ++e;
      total += cnt[e];
    }
    CK(cudaMemcpyAsync(dst[a], src[a], total * sizeof(double), cudaMemcpyHostToDevice, st));
    a = e + 1;
  }
  if (vo) CK(cudaMemcpyAsync(ss.flag, in->vo_flag, n, cudaMemcpyHostToDevice, st));
  std::memset(din, 0, sizeof(*din));
  const double **dp[kNumIn] = {&din->gyro, &din->accel, &din->imu_time, &din->joint_pos, &din->joint_vel, &din->foot_force,
                               &din->vo_quat, &din->vo_time_pre, &din->vo_time_now, &din->vo_rel_p, &din->quat};
  for (int k = 0; k < kNumIn; ++k) *dp[k] = src[k] ? dst[k] : nullptr;
  din->vo_flag = vo ? ss.flag : nullptr;
  return DEKF_OK;
}

void stage_outputs(const dekf_handle *h, const StageSet &ss, const dekf_outputs *out, dekf_outputs *dout) {
  const size_t n = (size_t)h->dm.n;
  std::memset(dout, 0, sizeof(*dout));
  dout->quat = ss.out;
  dout->x = ss.out + 4 * n;
  dout->v_body = ss.out + (size_t)(4 + h->ds) * n;
  dout->contact = (out && out->contact) ? ss.contact : nullptr;
  dout->status = (out && out->status) ? ss.status : nullptr;
}

// D2H copies of one tick's results on stream `st` into the host arrays of `out` (+ step offset in elements of n)
int unstage_outputs(dekf_handle *h, const StageSet &ss, const dekf_outputs *out, size_t step, cudaStream_t st, int kind) {
  if (!out) return DEKF_OK;
  const size_t n = (size_t)h->dm.n;
  double *q = out->quat ? out->quat + step * 4 * n : nullptr;
  const size_t ds = (size_t)h->ds;
  double *x = (out->x && kind != HK_EKF) ? out->x + step * ds * n : nullptr;
  double *v = (out->v_body && kind != HK_EKF) ? out->v_body + step * 3 * n : nullptr;
  if (kind == HK_MHE) q = nullptr;
  if (q && x && v && x == q + 4 * n && v == x + ds * n) {
    CK(cudaMemcpyAsync(q, ss.out, (7 + ds) * n * sizeof(double), cudaMemcpyDeviceToHost, st));
  } else {
    if (q) CK(cudaMemcpyAsync(q, ss.out, 4 * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (x) CK(cudaMemcpyAsync(x, ss.out + 4 * n, ds * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (v) CK(cudaMemcpyAsync(v, ss.out + (4 + ds) * n, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, st));
  }
  if (out->contact && kind != HK_EKF)
    CK(cudaMemcpyAsync(out->contact + step * h->nl * n, ss.contact, (size_t)h->nl * n, cudaMemcpyDeviceToHost, st));
  if (out->status) CK(cudaMemcpyAsync(out->status + step * n, ss.status, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  return DEKF_OK;
}

int device_call(dekf_handle *h, int kind, int32_t T_, const dekf_inputs *din, const dekf_outputs *dout) {
  switch (kind) {
    case HK_STEP: return dekf_step(h, T_, din, dout);
    case HK_MHE: return dekf_mhe_step(h, T_, din, dout);
    default: return dekf_ekf_step(h, din, dout);
  }
}

// Small batches (n <= kZeroCopyMaxN): inputs are packed into a pinned, mapped host block the kernels read directly, results
// are written by the kernels into the same block: no copy engine round trips on the single-robot latency path.
constexpr int kZeroCopyMaxN = 256;
int host_call_zero_copy(dekf_handle *h, int kind, int32_t T_, const dekf_inputs *in, const dekf_outputs *out) {
  const size_t n = (size_t)h->dm.n, ds = (size_t)h->ds, nl = (size_t)h->nl;
  size_t cnt[kNumIn], tot = 0;
  in_counts(h, cnt);
  for (int a = 0; a < kNumIn; ++a) tot += cnt[a];
  const size_t out_d = (7 + ds) * n;
  const size_t bytes = (tot + out_d) * sizeof(double) + n * sizeof(int32_t) + n /*flag*/ + nl * n /*contact*/;
  if (h->hmap_bytes < bytes) {
    if (h->hmap) cudaFreeHost(h->hmap);
    h->hmap = nullptr;
    h->hmap_bytes = 0;
    CK(cudaHostAlloc((void **)&h->hmap, bytes, cudaHostAllocMapped));
    h->hmap_bytes = bytes;
  }
  double *hin = (double *)h->hmap, *hout = hin + tot;
  int32_t *hstatus = (int32_t *)(hout + out_d);
  uint8_t *hflag = (uint8_t *)(hstatus + n), *hcontact = hflag + n;
  const bool vo = in->vo_flag != nullptr;
  const double *src[kNumIn] = {in->gyro, in->accel, in->imu_time, in->joint_pos, in->joint_vel, in->foot_force,
                               vo ? in->vo_quat : nullptr, vo ? in->vo_time_pre : nullptr, vo ? in->vo_time_now : nullptr,
                               vo ? in->vo_rel_p : nullptr, in->quat};
  const double *dst[kNumIn];
  size_t off = 0;
  for (int a = 0; a < kNumIn; ++a) {
    dst[a] = src[a] ? hin + off : nullptr;
    if (src[a]) std::memcpy(hin + off, src[a], cnt[a] * sizeof(double));
    off += cnt[a];
  }
  if (vo) std::memcpy(hflag, in->vo_flag, n);
  dekf_inputs din;
  std::memset(&din, 0, sizeof(din));
  din.gyro = dst[0];
  din.accel = dst[1];
  din.imu_time = dst[2];
  din.joint_pos = dst[3];
  din.joint_vel = dst[4];
  din.foot_force = dst[5];
  din.vo_quat = dst[6];
  din.vo_time_pre = dst[7];
  din.vo_time_now = dst[8];
  din.vo_rel_p = dst[9];
  din.quat = dst[10];
  din.vo_flag = vo ? hflag : nullptr;
  dekf_outputs dout;
  std::memset(&dout, 0, sizeof(dout));
  dout.quat = hout;
  dout.x = hout + 4 * n;
  dout.v_body = hout + (4 + ds) * n;
  dout.contact = (out && out->contact) ? hcontact : nullptr;
  dout.status = (out && out->status) ? hstatus : nullptr;
  int rc = device_call(h, kind, T_, &din, &dout);
  if (rc) return rc;
  CK(cudaStreamSynchronize(h->stream));
  if (out) {
    if (out->quat && kind != HK_MHE) std::memcpy(out->quat, hout, 4 * n * sizeof(double));
    if (out->x && kind != HK_EKF) std::memcpy(out->x, hout + 4 * n, ds * n * sizeof(double));
    if (out->v_body && kind != HK_EKF) std::memcpy(out->v_body, hout + (4 + ds) * n, 3 * n * sizeof(double));
    if (out->contact && kind != HK_EKF) std::memcpy(out->contact, hcontact, nl * n);
    if (out->status) std::memcpy(out->status, hstatus, n * sizeof(int32_t));
  }
  return DEKF_OK;
}

int host_call(dekf_handle *h, int kind, int32_t T_, const dekf_inputs *in, const dekf_outputs *out) {
  if (!h || !in) return fail(h, DEKF_EINVAL, "host entry point: null argument");
  CK(cudaSetDevice(h->cfg.device));
  if (h->dm.n <= kZeroCopyMaxN && !h->cfg.debug_taps) return host_call_zero_copy(h, kind, T_, in, out);
  dekf_inputs din;
  dekf_outputs dout;
  int rc = alloc_stage_set(h, h->stage[0]);
  if (rc) return rc;
  rc = stage_inputs(h, h->stage[0], in, h->stream, &din);
  if (rc) return rc;
  stage_outputs(h, h->stage[0], out, &dout);
  rc = device_call(h, kind, T_, &din, &dout);
  if (rc) return rc;
  rc = unstage_outputs(h, h->stage[0], out, 0, h->stream, kind);
  if (rc) return rc;
  CK(cudaStreamSynchronize(h->stream));
  return DEKF_OK;
}

// rows of every input stream (elements per tick = rows * n)
void offset_inputs(const dekf_handle *h, const dekf_inputs *in, size_t s, bool vo, dekf_inputs *o) {
  const size_t n = (size_t)h->dm.n;
  auto at = [&](const double *p, size_t rows) { return p ? p + s * rows * n : nullptr; };
  std::memset(o, 0, sizeof(*o));
  o->gyro = at(in->gyro, 3);
  o->accel = at(in->accel, 3);
  o->imu_time = at(in->imu_time, 1);
  o->joint_pos = at(in->joint_pos, h->nq);
  o->joint_vel = at(in->joint_vel, h->nq);
  o->foot_force = at(in->foot_force, h->nl);
  o->quat = at(in->quat, 4);
  if (vo && in->vo_flag) {
    o->vo_flag = in->vo_flag + s * n;
    o->vo_quat = at(in->vo_quat, 4);
    o->vo_time_pre = at(in->vo_time_pre, 1);
    o->vo_time_now = at(in->vo_time_now, 1);
    o->vo_rel_p = at(in->vo_rel_p, 3);
  }
}
}  // namespace

extern "C" {

int dekf_step_host(dekf_handle *h, int32_t T_, const dekf_inputs *in, const dekf_outputs *out) {
  return host_call(h, HK_STEP, T_, in, out);
}
int dekf_mhe_step_host(dekf_handle *h, int32_t T_, const dekf_inputs *in, const dekf_outputs *out) {
  return host_call(h, HK_MHE, T_, in, out);
}
int dekf_ekf_step_host(dekf_handle *h, const dekf_inputs *in, const dekf_outputs *out) {
  return host_call(h, HK_EKF, 0, in, out);
}

int dekf_run(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs *in, const uint8_t *vo_steps, const dekf_outputs *out,
             int32_t out_per_step) {
  if (!h || !in || S < 0) return fail(h, DEKF_EINVAL, "dekf_run: bad argument");
  CK(cudaSetDevice(h->cfg.device));
  const size_t n = (size_t)h->dm.n;
  auto outputs_of = [&](int32_t s, dekf_outputs *os) {
    std::memset(os, 0, sizeof(*os));
    if (out && (out_per_step || s == S - 1)) {
      const size_t o = out_per_step ? (size_t)s : 0;
      os->quat = out->quat ? out->quat + o * 4 * n : nullptr;
      os->x = out->x ? out->x + o * (size_t)h->ds * n : nullptr;
      os->v_body = out->v_body ? out->v_body + o * 3 * n : nullptr;
      os->contact = out->contact ? out->contact + o * h->nl * n : nullptr;
      os->status = out->status ? out->status + o * n : nullptr;
    }
  };
  // small batches (one fused launch per tick) and tapped handles: plain tick loop.  Exception: a multi-tick call with the FULL
  // re-sweep on a few hundred to a few thousand instances is faster through the pipeline below, where the EKF and the assembly of
  // tick s+1 overlap the solve of tick s (measured at 512 ... 4,096 instances: 34.5-35.5 vs 43.3-45.3 us per tick; with the
  // incremental solve the single launch wins, 16.2 vs 18.8 us) -- same kernels' results either way, bit for bit
  const bool one_launch = h->dm.n <= h->fused_max && !h->bc.enable && h->cfg.leg_odom_type == 0;
  const bool rather_pipeline = one_launch && h->dm.n >= h->run_pipeline_min && h->mc64.window_solve == 0 && h->cfg.est_type == 0 && S >= 4;
  if ((one_launch && !rather_pipeline) || h->cfg.debug_taps || S < 2) {
    for (int32_t s = 0; s < S; ++s) {
      dekf_inputs is;
      offset_inputs(h, in, (size_t)s, !vo_steps || vo_steps[s], &is);
      dekf_outputs os;
      outputs_of(s, &os);
      const int rc = dekf_step(h, T0 + s, &is, &os);
      if (rc) return rc;
    }
    return DEKF_OK;
  }
  // Large batches: several streams.  The orientation EKF does not depend on the MHE, so its ticks run ahead (up to kAhead
  // ticks) on their own stream and hand each tick's quaternion / status word over through a ring.  The stage assembly of tick
  // s+1 does not depend on the window solve of tick s either (per-tick scratch words are double-buffered by tick parity, the
  // stage ring has one slot more than the window), unless tick s+1 inserts VO bounds into stages the solve of tick s is
  // reading: it runs one tick ahead on a second stream and is serialised behind the solve only on ticks that carry VO
  // messages.  The window solves run on one stream per tile range.  All streams have the SAME priority (DESIGN.md 4.1).
  constexpr int QA = dekf_handle::kAhead;
  int rc = check_T(h, T0);
  if (rc) return rc;
  if (!in->gyro || !in->accel || !in->imu_time || !in->joint_pos || !in->joint_vel || !in->foot_force)
    return fail(h, DEKF_EINVAL, "dekf_run: null input");
  if (in->vo_flag && (!in->vo_quat || !in->vo_time_pre || !in->vo_time_now || !in->vo_rel_p))
    return fail(h, DEKF_EINVAL, "dekf_run: vo_flag without the VO arrays");
  constexpr int MW = dekf_handle::kMaxWays;
  if (!h->s_ekf) {
    int lo = 0, hi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));  // lo = numerically largest = lowest priority
    // Stream priorities (DEKF_PRIO, measured in profiles/r02_pipeline.md).  Default: ALL EQUAL.  With the re-sweep cut into tile
    // ranges the solve streams always hold CTAs that are ready to run; under "solve first" the assembly of the next tick only got
    // SMs once the solves ran dry -- and the next solve then waited for that assembly: a bubble of one assembly per tick.
    int p_ekf = lo, p_asm = lo, p_sol = lo;
    if (h->prio_mode == 1) p_ekf = lo, p_asm = (lo + hi) / 2, p_sol = hi;  // round 1: solve first
    if (h->prio_mode == 2) p_ekf = hi, p_asm = hi, p_sol = lo;             // front kernels first
    CK(cudaStreamCreateWithPriority(&h->s_ekf, cudaStreamNonBlocking, p_ekf));
    CK(cudaStreamCreateWithPriority(&h->s_asm, cudaStreamNonBlocking, p_asm));
    // only the streams the tile ranges need (a process has a handful of hardware queues: streams beyond them share one and
    // serialise behind each other)
    const int nsol = h->split_ways_env >= 2 ? (h->split_ways_env < MW ? h->split_ways_env : MW) : 2;
    for (int r = 0; r < nsol; ++r) CK(cudaStreamCreateWithPriority(&h->s_sol[r], cudaStreamNonBlocking, p_sol));
    h->s_asmw[0] = h->s_asm;
    for (int r = 1; r < nsol; ++r) CK(cudaStreamCreateWithPriority(&h->s_asmw[r], cudaStreamNonBlocking, p_asm));
    CK(cudaMalloc((void **)&h->quat_ring, (size_t)QA * 4 * n * sizeof(double)));
    CK(cudaMalloc((void **)&h->status_ring, (size_t)QA * n * sizeof(int32_t)));
    h->extra_bytes += (size_t)QA * n * (4 * sizeof(double) + sizeof(int32_t));
    for (int k = 0; k < QA; ++k) {
      CK(cudaEventCreateWithFlags(&h->ev_ekf[k], cudaEventDisableTiming));
      for (int r = 0; r < MW; ++r) CK(cudaEventCreateWithFlags(&h->ev_solw[r][k], cudaEventDisableTiming));
      for (int r = 0; r < MW; ++r) CK(cudaEventCreateWithFlags(&h->ev_asmw[r][k], cudaEventDisableTiming));
    }
    CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
  }
  // the assembly may only run ahead of the solve where the solve is the plain window sweep (full or incremental)
  const bool asm_ahead = h->cfg.est_type == 0 && !h->bc.enable && h->cfg.leg_odom_type == 0 && !h->prof;
  // Full re-sweep with the TMA kernel: 65,536 instances are 512 tiles on 2 x 148 CTA slots = 1.73 waves.  The tick's solve is cut
  // into `ways` tile ranges, one launch per range on its own stream; the ranges are independent instances, so range r of tick
  // s + 1 starts as soon as range r of tick s is done and the partial wave of one tick overlaps the next tick instead of leaving
  // slots idle (DEKF_NO_SPLIT=1 disables; DEKF_SPLIT_WAYS / DEKF_SPLIT_TILES tune).
  int ways = 1, bound[MW + 1] = {0};
  {
    const int tiles = h->dm.ns / kTile, slots = h->solve_slots;
    if (asm_ahead && !h->no_split && h->use_tma && h->mc64.window_solve == 0 && slots > 0 && tiles > slots) {
      if (h->split_ways_env >= 2) {
        ways = h->split_ways_env < MW ? h->split_ways_env : MW;
        for (int r = 0; r < ways; ++r) bound[r] = (int)((int64_t)tiles * r / ways);
      } else if (tiles % slots != 0) {
        ways = 2;
        bound[1] = tiles / slots * slots;  // the last full wave
        if (h->split_tiles_env > 0 && h->split_tiles_env < tiles) bound[1] = h->split_tiles_env;
      }
    }
    bound[ways] = tiles;
  }
  // fork the internal streams off the caller-visible stream, join back at the end
  cudaStream_t user = h->stream;
  CK(cudaEventRecord(h->ev_fork, user));
  CK(cudaStreamWaitEvent(h->s_ekf, h->ev_fork, 0));
  CK(cudaStreamWaitEvent(h->s_asm, h->ev_fork, 0));
  for (int r = 0; r < ways; ++r) CK(cudaStreamWaitEvent(h->s_sol[r], h->ev_fork, 0));
  for (int r = 1; r < ways; ++r) CK(cudaStreamWaitEvent(h->s_asmw[r], h->ev_fork, 0));
  for (int32_t s = 0; s < S && rc == DEKF_OK; ++s) {
    const int slot = s % QA;
    dekf_inputs is;
    const bool vo_tick = (!vo_steps || vo_steps[s]) && in->vo_flag != nullptr;
    offset_inputs(h, in, (size_t)s, !vo_steps || vo_steps[s], &is);
    is.quat = nullptr;
    dekf_outputs os;
    outputs_of(s, &os);
    double *qslot = h->quat_ring + (size_t)slot * 4 * n;
    int32_t *sslot = h->status_ring + (size_t)slot * n;
    cudaError_t ce = cudaSuccess;
    if (s >= QA) {  // k_assemble of tick s-QA (every tile range of it) has consumed the slot
      for (int r = 0; r < ways && ce == cudaSuccess; ++r) ce = cudaStreamWaitEvent(h->s_ekf, h->ev_asmw[r][slot], 0);
    }
    dekf_outputs oe;
    std::memset(&oe, 0, sizeof(oe));
    oe.quat = qslot;
    h->vo_slot = slot;
    if (h->ekf_serial && s >= 1)  // diagnosis: no EKF launch overlaps a window solve
      for (int r = 0; r < ways && ce == cudaSuccess; ++r) ce = cudaStreamWaitEvent(h->s_ekf, h->ev_solw[r][(s - 1) % QA], 0);
    if (ce == cudaSuccess) rc = ekf_launch(h, &is, &oe, sslot, h->s_ekf);
    if (rc) break;
    if (ce == cudaSuccess) ce = cudaEventRecord(h->ev_ekf[slot], h->s_ekf);
    // ---- stage assembly of tick s.  Parity-buffered scratch + the spare ring slot allow ONE tick of lead: it waits for the solve
    // of tick s-2, and for the solve of tick s-1 too when this tick rewrites VO rows inside the window that solve is reading.
    // On such a tick the assembly is cut into the solve's tile ranges: range r only waits for range r of the previous solve and
    // releases range r of this tick's solve, so the other ranges keep the SMs busy meanwhile.
    is.quat = qslot;
    const bool asm_split = asm_ahead && ways > 1 && vo_tick && s >= 1 && T0 + s >= 2 && !h->no_asm_split;
    const int aways = asm_split ? ways : 1;
    for (int ra = 0; ra < aways && ce == cudaSuccess && rc == DEKF_OK; ++ra) {
      cudaStream_t sa = asm_ahead ? h->s_asmw[ra] : h->s_sol[0];
      ce = cudaStreamWaitEvent(sa, h->ev_ekf[slot], 0);
      if (asm_ahead) {
        for (int r = (asm_split ? ra : 0); r < (asm_split ? ra + 1 : ways) && ce == cudaSuccess; ++r) {
          if (s >= 1) ce = cudaStreamWaitEvent(sa, h->ev_asmw[r][(s - 1) % QA], 0);  // assembly of the previous tick (any stream)
          if (ce == cudaSuccess && s >= 2) ce = cudaStreamWaitEvent(sa, h->ev_solw[r][(s - 2) % QA], 0);
          if (ce == cudaSuccess && s >= 1 && vo_tick) ce = cudaStreamWaitEvent(sa, h->ev_solw[r][(s - 1) % QA], 0);
        }
      }
      if (ce != cudaSuccess) break;
      h->stream = sa;
      if (asm_split) {
        h->asm_tile0 = bound[ra];
        h->asm_tiles = bound[ra + 1] - bound[ra];
      }
      // the tick's quaternion leaves the ring slot BEFORE the slot is released to the EKF of tick s+QA (copying it on the
      // solve stream raced with that EKF tick whenever the solves lagged behind the assembly): k_assemble writes it out
      h->asm_quat_copy = os.quat;
      rc = mhe_step_impl(h, T0 + s, &is, &os, sslot, 1);
      h->asm_quat_copy = nullptr;
      h->asm_tiles = -1;
      h->stream = user;
      if (rc) break;
      for (int r = (asm_split ? ra : 0); r < (asm_split ? ra + 1 : ways) && ce == cudaSuccess; ++r)
        ce = cudaEventRecord(h->ev_asmw[r][slot], sa);
    }
    h->vo_list_valid = false;
    if (rc) break;
    if (ce != cudaSuccess) {
      rc = fail(h, DEKF_ECUDA, "dekf_run pipeline", ce);
      break;
    }
    // ---- window solve of tick s: one launch per tile range (tick 0 has no window sweep: one launch covers every instance)
    const bool split = ways > 1 && T0 + s >= 1;
    for (int r = 0; r < ways && ce == cudaSuccess && rc == DEKF_OK; ++r) {
      if (r == 0 || split) {
        if (asm_ahead) {
          for (int q = (split ? r : 0); q < (split ? r + 1 : ways) && ce == cudaSuccess; ++q)
            ce = cudaStreamWaitEvent(h->s_sol[r], h->ev_asmw[q][slot], 0);
        }
        if (ce != cudaSuccess) break;
        if (split) {
          h->solve_tile0 = bound[r];
          h->solve_tiles = bound[r + 1] - bound[r];
        }
        h->stream = h->s_sol[r];
        rc = mhe_step_impl(h, T0 + s, &is, &os, sslot, 2);
        h->stream = user;
        h->solve_tiles = -1;
        if (rc) break;
      } else {
        ce = cudaStreamWaitEvent(h->s_sol[r], h->ev_solw[0][slot], 0);  // undivided launch on s_sol[0]: keep the ranges ordered
      }
      if (ce == cudaSuccess) ce = cudaEventRecord(h->ev_solw[r][slot], h->s_sol[r]);
    }
    if (rc) break;
    if (ce != cudaSuccess) rc = fail(h, DEKF_ECUDA, "dekf_run pipeline", ce);
  }
  h->stream = user;
  // join the internal streams back into the caller-visible one; if any of this fails (or the loop failed), drain them
  // on the host so that nothing is in flight when the error is reported
  cudaError_t je = cudaSuccess;
  cudaStream_t internal[2 * MW + 2];
  int ni = 0;
  for (int r = 0; r < ways; ++r) internal[ni++] = h->s_sol[r];
  for (int r = 0; r < ways; ++r) internal[ni++] = h->s_asmw[r];
  internal[ni++] = h->s_ekf;
  for (int k = 0; k < ni && je == cudaSuccess; ++k) {
    je = cudaEventRecord(h->ev_join, internal[k]);
    if (je == cudaSuccess) je = cudaStreamWaitEvent(user, h->ev_join, 0);
  }
  if (je != cudaSuccess || rc != DEKF_OK) {
    for (int r = 0; r < MW; ++r)
      if (h->s_sol[r]) cudaStreamSynchronize(h->s_sol[r]);
    for (int r = 0; r < MW; ++r)
      if (h->s_asmw[r]) cudaStreamSynchronize(h->s_asmw[r]);
    cudaStreamSynchronize(h->s_ekf);
    cudaStreamSynchronize(user);
    if (rc == DEKF_OK) rc = fail(h, DEKF_ECUDA, "dekf_run: joining the internal streams", je);
  }
  return rc;
}

// float32 sensor streams -> the double staging arrays the kernels read (dekf_run_host_f32)
__global__ void __launch_bounds__(256) k_widen(const float *__restrict__ src, double *__restrict__ dst, size_t count) {
  for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += (size_t)gridDim.x * blockDim.x) dst[k] = (double)src[k];
}

__global__ void __launch_bounds__(256) k_narrow(const double *__restrict__ src, float *__restrict__ dst, size_t count) {
  for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += (size_t)gridDim.x * blockDim.x) dst[k] = (float)src[k];
}

// in: all-double host streams; inf (non-null: dekf_run_host_f32): the five sensor arrays as float, the rest from inf too;
// outf (non-null: dekf_run_host_f32io): quat / x / v_body leave the device as float, `out` then only carries contact / status
static int run_host_body(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs *in, const dekf_inputs_f32 *inf, const uint8_t *vo_steps,
                         const dekf_outputs *out, int32_t out_per_step, const dekf_outputs_f32 *outf);
static int run_host_impl(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs *in, const dekf_inputs_f32 *inf, const uint8_t *vo_steps,
                         const dekf_outputs *out, int32_t out_per_step, const dekf_outputs_f32 *outf = nullptr) {
  const int rc = run_host_body(h, T0, S, in, inf, vo_steps, out, out_per_step, outf);
  if (rc != DEKF_OK) {
    // an error return must not leave copies into / out of caller-owned host buffers in flight
    const std::string keep = h->err;
    if (h->s_h2d) cudaStreamSynchronize(h->s_h2d);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->s_d2h) cudaStreamSynchronize(h->s_d2h);
    h->err = keep;
  }
  return rc;
}
static int run_host_body(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs *in, const dekf_inputs_f32 *inf, const uint8_t *vo_steps,
                         const dekf_outputs *out, int32_t out_per_step, const dekf_outputs_f32 *outf) {
  CK(cudaSetDevice(h->cfg.device));
  const size_t n = (size_t)h->dm.n;
  // Ticks move in chunks of B: every field of the host streams is [S][rows][n], so B consecutive ticks of one field are
  // ONE contiguous copy (6 input copies + the VO arrays of the ticks that carry a message per chunk, 5 result copies per
  // chunk) and the chunk runs through dekf_run (EKF ticks ahead of the MHE).  Chunks are software-pipelined over three
  // streams and two device staging sets: H2D of chunk c+1 | kernels of chunk c | D2H of chunk c-1.
  int B = h->host_chunk;
  {
    const size_t per_tick = (size_t)(16 + 2 * h->nq + h->nl + 7 + h->ds) * 8 * n;
    const size_t cap = (size_t)384 << 20;  // staging budget per set
    if ((size_t)B * per_tick > cap) B = (int)(cap / per_tick);
  }
  if (B < 1) B = 1;
  if (B > S) B = S > 0 ? S : 1;
  int rc = alloc_chunk_set(h, h->chunk[0], B);
  if (rc) return rc;
  rc = alloc_chunk_set(h, h->chunk[1], B);
  if (rc) return rc;
  const size_t rows_f32 = 6 + 2 * (size_t)h->nq + (size_t)h->nl;  // gyro accel joint_pos joint_vel foot_force
  if (inf)
    for (int k = 0; k < 2; ++k)
      if (h->chunk[k].cap_f32 < h->chunk[k].cap) {
        cudaFree(h->chunk[k].in_f32);
        h->chunk[k].in_f32 = nullptr;
        CK(cudaMalloc((void **)&h->chunk[k].in_f32, (size_t)h->chunk[k].cap * rows_f32 * n * sizeof(float)));
        h->chunk[k].cap_f32 = h->chunk[k].cap;
        h->extra_bytes += (size_t)h->chunk[k].cap * rows_f32 * n * sizeof(float);
      }
  if (outf)
    for (int k = 0; k < 2; ++k)
      if (h->chunk[k].cap_out_f32 < h->chunk[k].cap) {
        cudaFree(h->chunk[k].out_f32);
        h->chunk[k].out_f32 = nullptr;
        CK(cudaMalloc((void **)&h->chunk[k].out_f32, (size_t)h->chunk[k].cap * (size_t)(7 + h->ds) * n * sizeof(float)));
        h->chunk[k].cap_out_f32 = h->chunk[k].cap;
        h->extra_bytes += (size_t)h->chunk[k].cap * (size_t)(7 + h->ds) * n * sizeof(float);
      }
  if (!h->s_h2d) {
    CK(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
      CK(cudaEventCreateWithFlags(&h->ev_h2d[k], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&h->ev_comp[k], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&h->ev_d2h[k], cudaEventDisableTiming));
    }
  }
  CK(cudaEventRecord(h->ev_comp[0], h->stream));  // order after whatever the caller queued on the handle's stream
  CK(cudaStreamWaitEvent(h->s_h2d, h->ev_comp[0], 0));
  CK(cudaStreamWaitEvent(h->s_d2h, h->ev_comp[0], 0));
  const size_t rows_in[6] = {3, 3, 1, (size_t)h->nq, (size_t)h->nq, (size_t)h->nl};
  const double *src_in[6] = {in->gyro, in->accel, in->imu_time, in->joint_pos, in->joint_vel, in->foot_force};
  const float *src_f32[6] = {inf ? inf->gyro : nullptr, inf ? inf->accel : nullptr, nullptr, inf ? inf->joint_pos : nullptr,
                             inf ? inf->joint_vel : nullptr, inf ? inf->foot_force : nullptr};
  const size_t rows_vo[4] = {4, 1, 1, 3};
  const double *src_vo[4] = {in->vo_quat, in->vo_time_pre, in->vo_time_now, in->vo_rel_p};
  // Chunk sizes ramp up (1, 2, 4, ... B) and down again at the end of the call: the first copy that nothing can overlap and the
  // last kernels + result copy that nothing overlaps either are ONE tick each instead of B ticks (DEKF_HOST_RAMP=0: all B).
  int c = 0, ramp = h->host_ramp ? 1 : B;
  for (int32_t s0 = 0, Bc = 0; s0 < S; s0 += Bc, ++c) {
    const int b = c & 1;
    Bc = ramp < B ? ramp : B;
    if (h->host_ramp && Bc > (S - s0 + 1) / 2) Bc = (S - s0 + 1) / 2;
    if (Bc > S - s0) Bc = S - s0;
    if (Bc < 1) Bc = 1;
    ramp = ramp * 2 < B ? ramp * 2 : B;
    ChunkSet &cs = h->chunk[b];
    const size_t cap = (size_t)cs.cap;
    if (c >= 2) CK(cudaStreamWaitEvent(h->s_h2d, h->ev_comp[b], 0));  // kernels of chunk c-2 are done with staging set b
    dekf_inputs din;
    std::memset(&din, 0, sizeof(din));
    const float *wsrc[6];
    double *wdst[6];
    size_t wcnt[6];
    int nw = 0;
    {
      double *d = cs.in;
      const double **dp[6] = {&din.gyro, &din.accel, &din.imu_time, &din.joint_pos, &din.joint_vel, &din.foot_force};
      float *df = cs.in_f32;
      nw = 0;
      for (int a = 0; a < 6; ++a) {
        const size_t cnt = (size_t)Bc * rows_in[a] * n;
        if (src_f32[a]) {  // half the PCIe bytes; widened on the COMPUTE stream below (a kernel on the copy stream would queue
                           // behind the running solves and stall the copies that follow it)
          CK(cudaMemcpyAsync(df, src_f32[a] + (size_t)s0 * rows_in[a] * n, cnt * sizeof(float), cudaMemcpyHostToDevice, h->s_h2d));
          wsrc[nw] = df;
          wdst[nw] = d;
          wcnt[nw++] = cnt;
          df += cap * rows_in[a] * n;
        } else {
          CK(cudaMemcpyAsync(d, src_in[a] + (size_t)s0 * rows_in[a] * n, cnt * sizeof(double), cudaMemcpyHostToDevice, h->s_h2d));
        }
        *dp[a] = d;
        d += cap * rows_in[a] * n;
      }
      bool any_vo = false;
      if (in->vo_flag) {
        const double **vp[4] = {&din.vo_quat, &din.vo_time_pre, &din.vo_time_now, &din.vo_rel_p};
        for (int a = 0; a < 4; ++a) {
          *vp[a] = d;
          for (int j = 0; j < Bc; ++j)
            if (!vo_steps || vo_steps[s0 + j]) {
              CK(cudaMemcpyAsync(d + (size_t)j * rows_vo[a] * n, src_vo[a] + (size_t)(s0 + j) * rows_vo[a] * n,
                                 rows_vo[a] * n * sizeof(double), cudaMemcpyHostToDevice, h->s_h2d));
              any_vo = true;
            }
          d += cap * rows_vo[a] * n;
        }
        for (int j = 0; j < Bc; ++j)
          if (!vo_steps || vo_steps[s0 + j])
            CK(cudaMemcpyAsync(cs.flag + (size_t)j * n, in->vo_flag + (size_t)(s0 + j) * n, n, cudaMemcpyHostToDevice, h->s_h2d));
        if (any_vo) din.vo_flag = cs.flag;
      }
    }
    CK(cudaEventRecord(h->ev_h2d[b], h->s_h2d));
    CK(cudaStreamWaitEvent(h->stream, h->ev_h2d[b], 0));
    if (c >= 2) CK(cudaStreamWaitEvent(h->stream, h->ev_d2h[b], 0));  // results of chunk c-2 have left staging set b
    for (int w = 0; w < nw; ++w) {
      k_widen<<<148 * 4, 256, 0, h->stream>>>(wsrc[w], wdst[w], wcnt[w]);
      h->launches++;
    }
    const bool last = s0 + Bc >= S;
    const bool want_out = out && (out_per_step || last);
    dekf_outputs dout;
    std::memset(&dout, 0, sizeof(dout));
    if (want_out) {
      dout.quat = cs.out;
      dout.x = cs.out + cap * 4 * n;
      dout.v_body = cs.out + cap * (size_t)(4 + h->ds) * n;
      dout.contact = out->contact ? cs.contact : nullptr;
      dout.status = out->status ? cs.status : nullptr;
    }
    // the chunk's own vo_steps mask (a tick whose VO arrays were not copied must not read them)
    rc = dekf_run(h, T0 + s0, Bc, &din, vo_steps ? vo_steps + s0 : nullptr, want_out ? &dout : nullptr, out_per_step ? 1 : 0);
    if (rc) return rc;
    if (want_out && outf) {  // one rounding to float32 on the device, behind the chunk's kernels
      const size_t cnt = (out_per_step ? (size_t)Bc : 1) * (size_t)(7 + h->ds) * n;
      // quat | x | v_body are contiguous in the staging set only when the chunk is full: narrow the three ranges
      const size_t k3[3] = {4, (size_t)h->ds, 3};
      const double *s3[3] = {dout.quat, dout.x, dout.v_body};
      size_t off = 0;
      for (int a = 0; a < 3; ++a) {
        const size_t c3 = (out_per_step ? (size_t)Bc : 1) * k3[a] * n;
        k_narrow<<<148 * 2, 256, 0, h->stream>>>(s3[a], cs.out_f32 + off, c3);
        h->launches++;
        off += cap * k3[a] * n;
      }
      (void)cnt;
    }
    CK(cudaEventRecord(h->ev_comp[b], h->stream));
    CK(cudaStreamWaitEvent(h->s_d2h, h->ev_comp[b], 0));
    if (want_out) {
      const size_t cnt = out_per_step ? (size_t)Bc : 1, so = out_per_step ? (size_t)s0 : 0;
      if (outf) {
        const float *fq = cs.out_f32, *fx = fq + cap * 4 * n, *fv = fx + cap * (size_t)h->ds * n;
        if (outf->quat) CK(cudaMemcpyAsync(outf->quat + so * 4 * n, fq, cnt * 4 * n * sizeof(float), cudaMemcpyDeviceToHost, h->s_d2h));
        if (outf->x) CK(cudaMemcpyAsync(outf->x + so * (size_t)h->ds * n, fx, cnt * (size_t)h->ds * n * sizeof(float), cudaMemcpyDeviceToHost, h->s_d2h));
        if (outf->v_body) CK(cudaMemcpyAsync(outf->v_body + so * 3 * n, fv, cnt * 3 * n * sizeof(float), cudaMemcpyDeviceToHost, h->s_d2h));
      } else {
        if (out->quat) CK(cudaMemcpyAsync(out->quat + so * 4 * n, dout.quat, cnt * 4 * n * sizeof(double), cudaMemcpyDeviceToHost, h->s_d2h));
        if (out->x) CK(cudaMemcpyAsync(out->x + so * (size_t)h->ds * n, dout.x, cnt * (size_t)h->ds * n * sizeof(double), cudaMemcpyDeviceToHost, h->s_d2h));
        if (out->v_body) CK(cudaMemcpyAsync(out->v_body + so * 3 * n, dout.v_body, cnt * 3 * n * sizeof(double), cudaMemcpyDeviceToHost, h->s_d2h));
      }
      if (out->contact) CK(cudaMemcpyAsync(out->contact + so * h->nl * n, cs.contact, cnt * h->nl * n, cudaMemcpyDeviceToHost, h->s_d2h));
      if (out->status) CK(cudaMemcpyAsync(out->status + so * n, cs.status, cnt * n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->s_d2h));
    }
    CK(cudaEventRecord(h->ev_d2h[b], h->s_d2h));
  }
  CK(cudaStreamSynchronize(h->s_h2d));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaStreamSynchronize(h->s_d2h));
  return DEKF_OK;
}

int dekf_run_host(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs *in, const uint8_t *vo_steps, const dekf_outputs *out,
                  int32_t out_per_step) {
  if (!h || !in || S < 0) return fail(h, DEKF_EINVAL, "dekf_run_host: bad argument");
  if (!in->gyro || !in->accel || !in->imu_time || !in->joint_pos || !in->joint_vel || !in->foot_force)
    return fail(h, DEKF_EINVAL, "dekf_run_host: null input");
  if (in->vo_flag && (!in->vo_quat || !in->vo_time_pre || !in->vo_time_now || !in->vo_rel_p))
    return fail(h, DEKF_EINVAL, "dekf_run_host: vo_flag without the VO arrays");
  return run_host_impl(h, T0, S, in, nullptr, vo_steps, out, out_per_step);
}

int dekf_run_host_f32(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs_f32 *inf, const uint8_t *vo_steps, const dekf_outputs *out,
                      int32_t out_per_step) {
  if (!h || !inf || S < 0) return fail(h, DEKF_EINVAL, "dekf_run_host_f32: bad argument");
  if (!inf->gyro || !inf->accel || !inf->imu_time || !inf->joint_pos || !inf->joint_vel || !inf->foot_force)
    return fail(h, DEKF_EINVAL, "dekf_run_host_f32: null input");
  if (inf->vo_flag && (!inf->vo_quat || !inf->vo_time_pre || !inf->vo_time_now || !inf->vo_rel_p))
    return fail(h, DEKF_EINVAL, "dekf_run_host_f32: vo_flag without the VO arrays");
  dekf_inputs in;  // the double fields; the five sensor arrays are taken from inf
  std::memset(&in, 0, sizeof(in));
  in.imu_time = inf->imu_time;
  in.vo_flag = inf->vo_flag;
  in.vo_quat = inf->vo_quat;
  in.vo_time_pre = inf->vo_time_pre;
  in.vo_time_now = inf->vo_time_now;
  in.vo_rel_p = inf->vo_rel_p;
  return run_host_impl(h, T0, S, &in, inf, vo_steps, out, out_per_step);
}

int dekf_run_host_f32io(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs_f32 *inf, const uint8_t *vo_steps,
                        const dekf_outputs_f32 *outf, int32_t out_per_step) {
  if (!h || !inf || !outf || S < 0) return fail(h, DEKF_EINVAL, "dekf_run_host_f32io: bad argument");
  if (!inf->gyro || !inf->accel || !inf->imu_time || !inf->joint_pos || !inf->joint_vel || !inf->foot_force)
    return fail(h, DEKF_EINVAL, "dekf_run_host_f32io: null input");
  if (inf->vo_flag && (!inf->vo_quat || !inf->vo_time_pre || !inf->vo_time_now || !inf->vo_rel_p))
    return fail(h, DEKF_EINVAL, "dekf_run_host_f32io: vo_flag without the VO arrays");
  dekf_inputs in;
  std::memset(&in, 0, sizeof(in));
  in.imu_time = inf->imu_time;
  in.vo_flag = inf->vo_flag;
  in.vo_quat = inf->vo_quat;
  in.vo_time_pre = inf->vo_time_pre;
  in.vo_time_now = inf->vo_time_now;
  in.vo_rel_p = inf->vo_rel_p;
  dekf_outputs out;  // contact / status keep their types; the three double arrays are replaced by outf's
  std::memset(&out, 0, sizeof(out));
  out.contact = outf->contact;
  out.status = outf->status;
  return run_host_impl(h, T0, S, &in, inf, vo_steps, &out, out_per_step, outf);
}

static int get_arrival(dekf_handle *h, double *P, double *x, int info) {
  if (!h || !P || !x) return fail(h, DEKF_EINVAL, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  if (h->cfg.leg_odom_type == 1) {
    if (!info) return fail(h, DEKF_EINVAL, "leg_odom_type 1 carries the arrival cost in information form: use dekf_get_arrival_cost");
    k_get_arrival_foot<<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->dm, h->fb, h->ds, P, x);
    h->launches++;
    CK(cudaGetLastError());
    return DEKF_OK;
  }
  if (h->mc64.window_solve == 1 && h->next_T >= 1) {  // marginalizeQP(T-N) on demand (see arrival_from_checkpoint)
    if (h->f32)
      k_arrival_from_ckpt<float><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->mc32, h->dm, h->b32, h->next_T - 1);
    else
      k_arrival_from_ckpt<double><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->mc64, h->dm, h->b64, h->next_T - 1);
    h->launches++;
  }
  if (h->f32)
    k_get_arrival<float><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->dm, h->b32, P, x, info);
  else
    k_get_arrival<double><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->dm, h->b64, P, x, info);
  h->launches++;
  CK(cudaGetLastError());
  return DEKF_OK;
}
int dekf_get_arrival_cost(dekf_handle *h, double *M_p, double *n_p) { return get_arrival(h, M_p, n_p, 1); }
int dekf_get_arrival_cov(dekf_handle *h, double *P, double *x) { return get_arrival(h, P, x, 0); }

static int get_misc(dekf_handle *h, double *p_vo, double *R, double *ekfP) {
  if (!h) return DEKF_EINVAL;
  CK(cudaSetDevice(h->cfg.device));
  const int Tk = h->next_T > 0 ? h->next_T - 1 : 0;
  if (h->f32)
    k_get_misc<float><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->dm, h->b32, Tk, p_vo, R, ekfP);
  else
    k_get_misc<double><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->dm, h->b64, Tk, p_vo, R, ekfP);
  h->launches++;
  CK(cudaGetLastError());
  return DEKF_OK;
}
int dekf_get_p_vo(dekf_handle *h, double *p) { return p ? get_misc(h, p, nullptr, nullptr) : DEKF_EINVAL; }
int dekf_get_R_sb(dekf_handle *h, double *R) { return R ? get_misc(h, nullptr, R, nullptr) : DEKF_EINVAL; }
int dekf_get_ekf_cov(dekf_handle *h, double *P) { return P ? get_misc(h, nullptr, nullptr, P) : DEKF_EINVAL; }

int dekf_get_window_vo_count(dekf_handle *h, int32_t *count) {
  if (!h || !count) return DEKF_EINVAL;
  CK(cudaSetDevice(h->cfg.device));
  const int Tk = h->next_T > 0 ? h->next_T - 1 : 0;
  if (h->f32)
    k_vo_count<float><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->dm, h->b32, Tk, count);
  else
    k_vo_count<double><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->dm, h->b64, Tk, count);
  h->launches++;
  CK(cudaGetLastError());
  return DEKF_OK;
}

int dekf_get_resweep_info(dekf_handle *h, int32_t *depth, int32_t *n_vo) {
  if (!h) return DEKF_EINVAL;
  if (h->mc64.window_solve != 1 || h->next_T < 2) return fail(h, DEKF_EINVAL, "dekf_get_resweep_info: needs DEKF_SOLVE_INCREMENTAL and T >= 1");
  CK(cudaSetDevice(h->cfg.device));
  if (h->f32)
    k_resweep_info<float><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->dm, h->b32, h->next_T - 1, depth, n_vo);
  else
    k_resweep_info<double><<<grid_for(h->dm.n), kBlock, 0, h->stream>>>(h->dm, h->b64, h->next_T - 1, depth, n_vo);
  h->launches++;
  CK(cudaGetLastError());
  return DEKF_OK;
}

int dekf_get_window(dekf_handle *h, double *x, int32_t *len) {
  if (!h) return DEKF_EINVAL;
  if (!x) return fail(h, DEKF_EINVAL, "dekf_get_window: null x");
  if (h->cfg.est_type != 0) return fail(h, DEKF_EINVAL, "dekf_get_window: est_type 1 (KF) has no window");
  if (h->cfg.leg_odom_type != 0) return fail(h, DEKF_EINVAL, "dekf_get_window: leg_odom_type 1 (foot states) is not supported");
  if (h->row_V != nullptr) return fail(h, DEKF_EINVAL, "dekf_get_window: not available after dekf_add_state_rows (constrained window)");
  if (h->cfg.v_box_enable || h->cfg.x_box_mask || h->bc.enable)
    return fail(h, DEKF_EINVAL, "dekf_get_window: not available with state bounds (v_box_enable / x_box_mask)");
  if (h->next_T < 2) return fail(h, DEKF_ESTATE, "dekf_get_window: needs a completed update(T >= 1)");
  CK(cudaSetDevice(h->cfg.device));
  const int Tk = h->next_T - 1, N = h->dm.N;
  void *scr = nullptr;
  if (h->mc64.window_solve == 0) {
    if (!h->win_scr) {
      const size_t bytes = (size_t)N * 54 * h->dm.ns * (h->f32 ? sizeof(float) : sizeof(double));
      CK(cudaMalloc(&h->win_scr, bytes));
      h->extra_bytes += bytes;
    }
    scr = h->win_scr;
  }
  // dekf_run joins its internal streams into h->stream before returning, so this launch is ordered after every tick
  const dim3 grid(grid_for(h->dm.n));
  if (h->f32 && scr)
    k_window<float, true><<<grid, kBlock, 0, h->stream>>>(h->mc32, h->mc64, h->dm, h->b32, (float *)scr, Tk, x);
  else if (h->f32)
    k_window<float, false><<<grid, kBlock, 0, h->stream>>>(h->mc32, h->mc64, h->dm, h->b32, nullptr, Tk, x);
  else if (scr)
    k_window<double, true><<<grid, kBlock, 0, h->stream>>>(h->mc64, h->mc64, h->dm, h->b64, (double *)scr, Tk, x);
  else
    k_window<double, false><<<grid, kBlock, 0, h->stream>>>(h->mc64, h->mc64, h->dm, h->b64, nullptr, Tk, x);
  h->launches++;
  CK(cudaGetLastError());
  if (len) *len = Tk + 1 < N ? Tk + 1 : N;
  return DEKF_OK;
}

int dekf_get_window_cov(dekf_handle *h, double *P, int32_t *len) {
  if (!h) return DEKF_EINVAL;
  if (!P) return fail(h, DEKF_EINVAL, "dekf_get_window_cov: null P");
  if (h->cfg.est_type != 0) return fail(h, DEKF_EINVAL, "dekf_get_window_cov: est_type 1 (KF) has no window");
  if (h->cfg.leg_odom_type != 0) return fail(h, DEKF_EINVAL, "dekf_get_window_cov: leg_odom_type 1 (foot states) is not supported");
  if (h->row_V != nullptr)
    return fail(h, DEKF_EINVAL, "dekf_get_window_cov: not available after dekf_add_state_rows (constrained window)");
  if (h->cfg.v_box_enable || h->cfg.x_box_mask || h->bc.enable)
    return fail(h, DEKF_EINVAL, "dekf_get_window_cov: not available with state bounds (v_box_enable / x_box_mask)");
  if (h->next_T < 2) return fail(h, DEKF_ESTATE, "dekf_get_window_cov: needs a completed update(T >= 1)");
  CK(cudaSetDevice(h->cfg.device));
  const int Tk = h->next_T - 1, N = h->dm.N;
  void *scr = nullptr;
  if (h->mc64.window_solve == 0) {  // the same scratch ring as dekf_get_window: each call rewrites it before reading it
    if (!h->win_scr) {
      const size_t bytes = (size_t)N * 54 * h->dm.ns * (h->f32 ? sizeof(float) : sizeof(double));
      CK(cudaMalloc(&h->win_scr, bytes));
      h->extra_bytes += bytes;
    }
    scr = h->win_scr;
  }
  const dim3 grid((h->dm.n + kCovBlock - 1) / kCovBlock);
  if (h->f32 && scr)
    k_window_cov<float, true><<<grid, kCovBlock, 0, h->stream>>>(h->mc32, h->mc64, h->dm, h->b32, (float *)scr, Tk, P, nullptr, 0);
  else if (h->f32)
    k_window_cov<float, false><<<grid, kCovBlock, 0, h->stream>>>(h->mc32, h->mc64, h->dm, h->b32, nullptr, Tk, P, nullptr, 0);
  else if (scr)
    k_window_cov<double, true><<<grid, kCovBlock, 0, h->stream>>>(h->mc64, h->mc64, h->dm, h->b64, (double *)scr, Tk, P, nullptr, 0);
  else
    k_window_cov<double, false><<<grid, kCovBlock, 0, h->stream>>>(h->mc64, h->mc64, h->dm, h->b64, nullptr, Tk, P, nullptr, 0);
  h->launches++;
  CK(cudaGetLastError());
  if (len) *len = Tk + 1 < N ? Tk + 1 : N;
  return DEKF_OK;
}

int dekf_get_foot_window(dekf_handle *h, double *x, double *P, int32_t *len) {
  if (!h) return DEKF_EINVAL;
  if (!x && !P) return fail(h, DEKF_EINVAL, "dekf_get_foot_window: x and P are both null");
  if (h->cfg.est_type != 0) return fail(h, DEKF_EINVAL, "dekf_get_foot_window: est_type 1 (KF) has no window");
  if (h->cfg.leg_odom_type != 1)
    return fail(h, DEKF_EINVAL, "dekf_get_foot_window: leg_odom_type 0 handle; use dekf_get_window / dekf_get_window_cov");
  if (h->next_T < 2) return fail(h, DEKF_ESTATE, "dekf_get_foot_window: needs a completed update(T >= 1)");
  CK(cudaSetDevice(h->cfg.device));
  const int Tk = h->next_T - 1, N = h->dm.N;
  if (!h->foot_win_ring) {  // every call rewrites the stages it reads
    const int W = h->nl == 4 ? FootWin<4>::W : (h->nl == 2 ? FootWin<2>::W : FootWin<1>::W);
    const size_t bytes = (size_t)(N > 1 ? N - 1 : 1) * h->dm.ns * W * sizeof(double);
    CK(cudaMalloc((void **)&h->foot_win_ring, bytes));
    h->extra_bytes += bytes;
  }
  // dekf_run joins its internal streams into h->stream before returning, so this launch is ordered after every tick
  if (h->nl == 4)
    launch_foot_window<4>(h->fc, h->dm, h->b64, h->fb, h->foot_win_ring, Tk, x, P, nullptr, h->stream);
  else if (h->nl == 2)
    launch_foot_window<2>(h->fc, h->dm, h->b64, h->fb, h->foot_win_ring, Tk, x, P, nullptr, h->stream);
  else
    launch_foot_window<1>(h->fc, h->dm, h->b64, h->fb, h->foot_win_ring, Tk, x, P, nullptr, h->stream);
  h->launches++;
  CK(cudaGetLastError());
  if (len) *len = Tk + 1 < N ? Tk + 1 : N;
  return DEKF_OK;
}

int dekf_get_constrained_window(dekf_handle *h, double *x, double *P, uint32_t *active, int32_t *len) {
  if (!h) return DEKF_EINVAL;
  if (!x && !P && !active) return fail(h, DEKF_EINVAL, "dekf_get_constrained_window: x, P and active are all null");
  if (!h->bc.enable)
    return fail(h, DEKF_EINVAL, "dekf_get_constrained_window: handle without state constraints; use dekf_get_window / dekf_get_window_cov");
  if (h->next_T < 2) return fail(h, DEKF_ESTATE, "dekf_get_constrained_window: needs a completed update(T >= 1)");
  CK(cudaSetDevice(h->cfg.device));
  const int Tk = h->next_T - 1, N = h->dm.N;
  const int warps = (h->dm.n + kTeamsPerWarp - 1) / kTeamsPerWarp, wpb = kTeamBlock / 32;
  const dim3 grid((warps + wpb - 1) / wpb);
  // dekf_run joins its internal streams into h->stream before returning, so this launch is ordered after every tick
  if (h->box_team)
    k_box_window<false><<<grid, kTeamBlock, 0, h->stream>>>(h->bc, h->dm, h->bb, h->tb.fac, Tk, x, P, active, nullptr);
  else
    k_box_window<true><<<grid, kTeamBlock, 0, h->stream>>>(h->bc, h->dm, h->bb, h->bb.fac, Tk, x, P, active, nullptr);
  h->launches++;
  CK(cudaGetLastError());
  if (len) *len = Tk + 1 < N ? Tk + 1 : N;
  return DEKF_OK;
}

int dekf_get_window_cross_cov(dekf_handle *h, double *P, double *C, int32_t *len) {
  if (!h) return DEKF_EINVAL;
  if (!C) return fail(h, DEKF_EINVAL, "dekf_get_window_cross_cov: null C");
  if (h->cfg.est_type != 0) return fail(h, DEKF_EINVAL, "dekf_get_window_cross_cov: est_type 1 (KF) has no window");
  if (h->next_T < 2) return fail(h, DEKF_ESTATE, "dekf_get_window_cross_cov: needs a completed update(T >= 1)");
  CK(cudaSetDevice(h->cfg.device));
  const int Tk = h->next_T - 1, N = h->dm.N;
  // dekf_run joins its internal streams into h->stream before returning, so these launches are ordered after every tick
  if (h->bc.enable) {  // state-constrained: the factor the last active-set solve left (box_window.cuh)
    const int warps = (h->dm.n + kTeamsPerWarp - 1) / kTeamsPerWarp, wpb = kTeamBlock / 32;
    const dim3 grid((warps + wpb - 1) / wpb);
    if (h->box_team)
      k_box_window<false, true><<<grid, kTeamBlock, 0, h->stream>>>(h->bc, h->dm, h->bb, h->tb.fac, Tk, nullptr, P, nullptr, C);
    else
      k_box_window<true, true><<<grid, kTeamBlock, 0, h->stream>>>(h->bc, h->dm, h->bb, h->bb.fac, Tk, nullptr, P, nullptr, C);
  } else if (h->cfg.leg_odom_type == 1) {  // foot states: the ring of dekf_get_foot_window, rewritten by every call
    if (!h->foot_win_ring) {
      const int W = h->nl == 4 ? FootWin<4>::W : (h->nl == 2 ? FootWin<2>::W : FootWin<1>::W);
      const size_t bytes = (size_t)(N > 1 ? N - 1 : 1) * h->dm.ns * W * sizeof(double);
      CK(cudaMalloc((void **)&h->foot_win_ring, bytes));
      h->extra_bytes += bytes;
    }
    if (h->nl == 4)
      launch_foot_window<4>(h->fc, h->dm, h->b64, h->fb, h->foot_win_ring, Tk, nullptr, P, C, h->stream);
    else if (h->nl == 2)
      launch_foot_window<2>(h->fc, h->dm, h->b64, h->fb, h->foot_win_ring, Tk, nullptr, P, C, h->stream);
    else
      launch_foot_window<1>(h->fc, h->dm, h->b64, h->fb, h->foot_win_ring, Tk, nullptr, P, C, h->stream);
  } else {  // 9-state: the RTS covariance pass reads P_{k+1}^s back from its output, so without P it runs on a two-block ring
    void *scr = nullptr;
    if (h->mc64.window_solve == 0) {  // the scratch ring of dekf_get_window
      if (!h->win_scr) {
        const size_t bytes = (size_t)N * 54 * h->dm.ns * (h->f32 ? sizeof(float) : sizeof(double));
        CK(cudaMalloc(&h->win_scr, bytes));
        h->extra_bytes += bytes;
      }
      scr = h->win_scr;
    }
    int pslots = N;
    if (!P) {
      if (!h->cross_ring) {
        const size_t bytes = 2 * 81 * (size_t)h->dm.n * sizeof(double);
        CK(cudaMalloc((void **)&h->cross_ring, bytes));
        h->extra_bytes += bytes;
      }
      P = h->cross_ring;
      pslots = 2;
    }
    const dim3 grid((h->dm.n + kCovBlock - 1) / kCovBlock);
    if (h->f32 && scr)
      k_window_cov<float, true, true><<<grid, kCovBlock, 0, h->stream>>>(h->mc32, h->mc64, h->dm, h->b32, (float *)scr, Tk, P, C, pslots);
    else if (h->f32)
      k_window_cov<float, false, true><<<grid, kCovBlock, 0, h->stream>>>(h->mc32, h->mc64, h->dm, h->b32, nullptr, Tk, P, C, pslots);
    else if (scr)
      k_window_cov<double, true, true><<<grid, kCovBlock, 0, h->stream>>>(h->mc64, h->mc64, h->dm, h->b64, (double *)scr, Tk, P, C, pslots);
    else
      k_window_cov<double, false, true><<<grid, kCovBlock, 0, h->stream>>>(h->mc64, h->mc64, h->dm, h->b64, nullptr, Tk, P, C, pslots);
  }
  h->launches++;
  CK(cudaGetLastError());
  if (len) *len = Tk + 1 < N ? Tk + 1 : N;
  return DEKF_OK;
}

int dekf_get_host(dekf_handle *h, int32_t what, void *host_out) {
  if (!h || !host_out) return fail(h, DEKF_EINVAL, "dekf_get_host: null argument");
  CK(cudaSetDevice(h->cfg.device));
  const size_t n = (size_t)h->dm.n;
  const size_t dsz = (size_t)h->ds;
  // DEKF_GET_BOX_WINDOW_ACTIVE: [N][n] uint32, half a double row each
  // DEKF_GET_WINDOW_C: [(N-1) * ds * ds][n], the lag-one blocks only
  const size_t rows[17] = {9, 3, dsz * dsz, dsz, 16, 1, dsz * dsz, dsz, 0, 9 * (size_t)h->dm.N, 81 * (size_t)h->dm.N,
                           dsz * (size_t)h->dm.N, dsz * dsz * (size_t)h->dm.N, 9 * (size_t)h->dm.N, 81 * (size_t)h->dm.N,
                           ((size_t)h->dm.N + 1) / 2, dsz * dsz * (size_t)(h->dm.N > 1 ? h->dm.N - 1 : 1)};
  if (what < 0 || what > DEKF_GET_WINDOW_C) return fail(h, DEKF_EINVAL, "dekf_get_host: unknown selector");
  // one scratch for the life of the handle (the 200 Hz node shells call this every tick)
  size_t need = (dsz * dsz + dsz + 6 * (size_t)h->nl) * n * sizeof(double);
  if (what == DEKF_GET_WINDOW_X && need < rows[DEKF_GET_WINDOW_X] * n * sizeof(double)) need = rows[DEKF_GET_WINDOW_X] * n * sizeof(double);
  if (what == DEKF_GET_WINDOW_P && need < rows[DEKF_GET_WINDOW_P] * n * sizeof(double)) need = rows[DEKF_GET_WINDOW_P] * n * sizeof(double);
  if (what >= DEKF_GET_FOOT_WINDOW_X && need < rows[what] * n * sizeof(double)) need = rows[what] * n * sizeof(double);
  if (h->get_scratch_bytes < need) {
    cudaFree(h->get_scratch);
    h->get_scratch = nullptr;
    h->get_scratch_bytes = 0;
    CK(cudaMalloc((void **)&h->get_scratch, need));
    h->get_scratch_bytes = need;
    h->extra_bytes += need;
  }
  double *d = h->get_scratch;
  if (what == DEKF_GET_KF_GAIN) {
    // K_KF_ = C_KF_ A_meas' C_meas^-1 (posterior form of DecentralEst.cpp:858): the 3 columns of leg i are C_KF_[:, v] Q_meas,i
    const double *Qsrc = h->tap_Q_meas ? h->tap_Q_meas : h->kf_Q;
    if (h->cfg.est_type != 1 || h->cfg.leg_odom_type != 0 || !Qsrc)
      return fail(h, DEKF_EINVAL, "DEKF_GET_KF_GAIN needs est_type 1, leg_odom_type 0 and cfg.kf_export_gain");
    int rc = dekf_get_arrival_cov(h, d, d + dsz * dsz * n);
    if (rc) return rc;
    const size_t L = (size_t)h->nl;
    std::vector<double> C(81 * n), Q(6 * L * n);
    CK(cudaMemcpyAsync(C.data(), d, 81 * n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(Q.data(), Qsrc, 6 * L * n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    double *K = (double *)host_out;
    const int sidx[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};
    for (size_t i = 0; i < n; ++i)
      for (size_t l = 0; l < L; ++l)
        for (int r = 0; r < 9; ++r)
          for (int c = 0; c < 3; ++c) {
            double v = 0.0;
            for (int k = 0; k < 3; ++k) v += C[(size_t)(r * 9 + 3 + k) * n + i] * Q[(l * 6 + sidx[k][c]) * n + i];
            K[((size_t)r * 3 * L + 3 * l + c) * n + i] = v;
          }
    return DEKF_OK;
  }
  int rc = DEKF_OK;
  const void *src = d;
  size_t bytes = rows[what] * n * sizeof(double);
  switch (what) {
    case DEKF_GET_R_SB: rc = dekf_get_R_sb(h, d); break;
    case DEKF_GET_P_VO: rc = dekf_get_p_vo(h, d); break;
    case DEKF_GET_ARRIVAL_M: rc = dekf_get_arrival_cost(h, d, d + dsz * dsz * n); break;
    case DEKF_GET_ARRIVAL_N:
      rc = dekf_get_arrival_cost(h, d, d + dsz * dsz * n);
      src = d + dsz * dsz * n;
      break;
    case DEKF_GET_EKF_COV: rc = dekf_get_ekf_cov(h, d); break;
    case DEKF_GET_ARRIVAL_COV: rc = dekf_get_arrival_cov(h, d, d + dsz * dsz * n); break;
    case DEKF_GET_ARRIVAL_MEAN:
      rc = dekf_get_arrival_cov(h, d, d + dsz * dsz * n);
      src = d + dsz * dsz * n;
      break;
    case DEKF_GET_WINDOW_X: {
      int32_t K = 0;
      rc = dekf_get_window(h, d, &K);
      bytes = (size_t)K * 9 * n * sizeof(double);
      break;
    }
    case DEKF_GET_WINDOW_P: {
      int32_t K = 0;
      rc = dekf_get_window_cov(h, d, &K);
      bytes = (size_t)K * 81 * n * sizeof(double);
      break;
    }
    case DEKF_GET_FOOT_WINDOW_X: {
      int32_t K = 0;
      rc = dekf_get_foot_window(h, d, nullptr, &K);
      bytes = (size_t)K * dsz * n * sizeof(double);
      break;
    }
    case DEKF_GET_FOOT_WINDOW_P: {
      int32_t K = 0;
      rc = dekf_get_foot_window(h, nullptr, d, &K);
      bytes = (size_t)K * dsz * dsz * n * sizeof(double);
      break;
    }
    case DEKF_GET_BOX_WINDOW_X: {
      int32_t K = 0;
      rc = dekf_get_constrained_window(h, d, nullptr, nullptr, &K);
      bytes = (size_t)K * 9 * n * sizeof(double);
      break;
    }
    case DEKF_GET_BOX_WINDOW_P: {
      int32_t K = 0;
      rc = dekf_get_constrained_window(h, nullptr, d, nullptr, &K);
      bytes = (size_t)K * 81 * n * sizeof(double);
      break;
    }
    case DEKF_GET_WINDOW_C: {
      int32_t K = 0;
      rc = dekf_get_window_cross_cov(h, nullptr, d, &K);
      bytes = (size_t)(K - 1) * dsz * dsz * n * sizeof(double);
      break;
    }
    case DEKF_GET_BOX_WINDOW_ACTIVE: {
      int32_t K = 0;
      rc = dekf_get_constrained_window(h, nullptr, nullptr, (uint32_t *)d, &K);
      bytes = (size_t)K * n * sizeof(uint32_t);
      break;
    }
    default:
      rc = dekf_get_window_vo_count(h, (int32_t *)d);
      bytes = n * sizeof(int32_t);
  }
  if (rc) return rc;
  CK(cudaMemcpyAsync(host_out, src, bytes, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return DEKF_OK;
}

int dekf_add_state_rows(dekf_handle *h, int32_t count, const double *a, const double *lb, const double *ub) {
  if (!h || count < 1 || count > 9 || !a || !lb || !ub) return fail(h, DEKF_EINVAL, "dekf_add_state_rows: bad argument");
  if (h->cfg.est_type != 0 || h->cfg.leg_odom_type != 0)
    return fail(h, DEKF_EINVAL, "dekf_add_state_rows: needs est_type 0 and leg_odom_type 0");
  if (h->next_T != 0 || h->ekf_k != 0) return fail(h, DEKF_ESTATE, "dekf_add_state_rows: call before the first step (or after dekf_reset)");
  CK(cudaSetDevice(h->cfg.device));
  double W[81], V[81], lo[9], hi[9];
  const int m = make_row_basis(h->cfg, count, a, lb, ub, W, V, lo, hi);
  if (m < 1) return fail(h, DEKF_EINVAL, "dekf_add_state_rows: rows (with the component bounds of the config) must be <= 9, linearly independent, lb < ub");
  const size_t ns = (size_t)h->dm.ns;
  const size_t fac = (size_t)h->dm.N * BOX_FAC * ns * sizeof(double), act = (size_t)h->dm.NW * ns;
  if (!h->bb.fac) {  // the handle was created without constraints: scratch of the one-thread-per-instance solve
    CK(cudaMalloc((void **)&h->bb.fac, fac));
    CK(cudaMalloc((void **)&h->bb.act, act));
    CK(cudaMalloc((void **)&h->bb.iters, ns * sizeof(int32_t)));
    CK(cudaMalloc((void **)&h->bb.nactive, ns * sizeof(int32_t)));
    CK(cudaMalloc((void **)&h->bb.capped, ns));
    h->extra_bytes += fac + act + 2 * ns * sizeof(int32_t) + ns;
  }
  if (!h->bb.act32) {
    CK(cudaMalloc((void **)&h->bb.act32, act * sizeof(uint32_t)));
    h->extra_bytes += act * sizeof(uint32_t);
  }
  if (!h->row_V) CK(cudaMalloc((void **)&h->row_V, 81 * sizeof(double)));
  CK(cudaMemcpyAsync(h->row_V, V, sizeof(V), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemsetAsync(h->bb.act, 0, act, h->stream));
  CK(cudaMemsetAsync(h->bb.act32, 0, act * sizeof(uint32_t), h->stream));
  CK(cudaMemsetAsync(h->bb.iters, 0, ns * sizeof(int32_t), h->stream));
  CK(cudaMemsetAsync(h->bb.nactive, 0, ns * sizeof(int32_t), h->stream));
  CK(cudaMemsetAsync(h->bb.capped, 0, ns, h->stream));
  CK(cudaStreamSynchronize(h->stream));  // V is a stack array
  h->bb.V = h->row_V;
  if (!h->bc.enable) h->bc = make_box_const(h->cfg);  // model constants of the information form (dt, noise weights, lever arm)
  h->bc.enable = 1;
  h->bc.general = 1;
  h->bc.nrows = m;
  h->bc.mask9 = (1 << m) - 1;
  for (int r = 0; r < 9; ++r) {
    h->bc.lo9[r] = r < m ? lo[r] : -1e300;
    h->bc.hi9[r] = r < m ? hi[r] : 1e300;
  }
  // the finite method (box_solve.cuh, phases 1-3) moves one bound per factorisation: give it room unless the config set a cap
  h->bc.max_iter = h->cfg.v_box_max_iter > 0 ? h->cfg.v_box_max_iter : 400;
  h->box_team = false;  // the team kernel knows the velocity box only
  return DEKF_OK;
}

int dekf_get_qp_info(dekf_handle *h, int32_t *iters, int32_t *n_active) {
  if (!h) return DEKF_EINVAL;
  if (!h->bc.enable) return fail(h, DEKF_EINVAL, "handle was created without v_box_enable");
  CK(cudaSetDevice(h->cfg.device));
  const size_t bytes = (size_t)h->dm.n * sizeof(int32_t);
  if (iters) CK(cudaMemcpyAsync(iters, h->bb.iters, bytes, cudaMemcpyDeviceToDevice, h->stream));
  if (n_active) CK(cudaMemcpyAsync(n_active, h->bb.nactive, bytes, cudaMemcpyDeviceToDevice, h->stream));
  return DEKF_OK;
}

int dekf_debug_taps(dekf_handle *h, double *b_meas, double *Q_meas, int32_t *vo_idx, int32_t *ekf_idx) {
  if (!h) return DEKF_EINVAL;
  if (!h->cfg.debug_taps) return fail(h, DEKF_EINVAL, "handle was created without debug_taps");
  CK(cudaSetDevice(h->cfg.device));
  const size_t n = (size_t)h->dm.n;
  if (b_meas) CK(cudaMemcpyAsync(b_meas, h->tap_b_meas, (size_t)3 * h->nl * n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  if (Q_meas) CK(cudaMemcpyAsync(Q_meas, h->tap_Q_meas, (size_t)6 * h->nl * n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  if (vo_idx) CK(cudaMemcpyAsync(vo_idx, h->tap_vo, 8 * n * sizeof(int32_t), cudaMemcpyDeviceToDevice, h->stream));
  if (ekf_idx) CK(cudaMemcpyAsync(ekf_idx, h->tap_ekf, 3 * n * sizeof(int32_t), cudaMemcpyDeviceToDevice, h->stream));
  return DEKF_OK;
}

int dekf_profile_enable(dekf_handle *h, int32_t enable) {
  if (!h) return DEKF_EINVAL;
  CK(cudaSetDevice(h->cfg.device));
  h->prof = enable != 0;
  return DEKF_OK;
}
int dekf_profile_read(dekf_handle *h, double *ms, int64_t *count) {
  if (!h || !ms || !count) return DEKF_EINVAL;
  CK(cudaStreamSynchronize(h->stream));
  for (auto &r : h->prof_recs) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.e0, r.e1) == cudaSuccess) {
      h->prof_ms[r.slot] += t;
      h->prof_n[r.slot]++;
    }
    h->prof_free.push_back(r);
  }
  h->prof_recs.clear();
  for (int k = 0; k < 4; ++k) {
    ms[k] = h->prof_ms[k];
    count[k] = h->prof_n[k];
    h->prof_ms[k] = 0;
    h->prof_n[k] = 0;
  }
  return DEKF_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// roofline denominators
// ------------------------------------------------------------------------------------------------
namespace {
template <typename T>
__global__ void __launch_bounds__(256) k_fma_peak(T *out, int iters, T a, T b) {
  // 16 independent FMA chains per thread keep the pipe full regardless of its latency
  T x[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) x[j] = (T)(threadIdx.x + j);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int j = 0; j < 16; ++j) x[j] = x[j] * a + b;
  }
  T s = (T)0;
#pragma unroll
  for (int j = 0; j < 16; ++j) s += x[j];
  if (s == (T)123456789) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <typename T>
int measure_fma(double *tflops) {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int blocks = sms * 8, threads = 256, iters = 4096;
  T *out = nullptr;
  if (cudaMalloc((void **)&out, (size_t)blocks * threads * sizeof(T)) != cudaSuccess) return DEKF_ENOMEM;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 6; ++rep) {
    cudaEventRecord(e0);
    k_fma_peak<T><<<blocks, threads>>>(out, iters, (T)1.0000001, (T)1e-7);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double fl = 2.0 * 16.0 * iters * (double)blocks * threads;
    if (rep > 0 && ms > 0.f) best = fmax(best, fl / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  *tflops = best;
  return cudaGetLastError() == cudaSuccess ? DEKF_OK : DEKF_ECUDA;
}
}  // namespace

extern "C" int dekf_measure_fma_peak(int32_t device, int32_t precision, double *tflops) {
  if (!tflops) return DEKF_EINVAL;
  if (cudaSetDevice(device) != cudaSuccess) return DEKF_ENODEV;
  return precision == DEKF_FP32 ? measure_fma<float>(tflops) : measure_fma<double>(tflops);
}

extern "C" int dekf_measure_copy_bw(int32_t device, double *gbs) {
  if (!gbs) return DEKF_EINVAL;
  if (cudaSetDevice(device) != cudaSuccess) return DEKF_ENODEV;
  const size_t bytes = (size_t)1 << 31;  // 2 GiB each way, far above the 126 MB L2
  void *a = nullptr, *b = nullptr;
  if (cudaMalloc(&a, bytes) != cudaSuccess) return DEKF_ENOMEM;
  if (cudaMalloc(&b, bytes) != cudaSuccess) {
    cudaFree(a);
    return DEKF_ENOMEM;
  }
  cudaMemset(a, 1, bytes);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 6; ++rep) {
    cudaEventRecord(e0);
    cudaMemcpyAsync(b, a, bytes, cudaMemcpyDeviceToDevice, 0);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms > 0.f) best = fmax(best, 2.0 * (double)bytes / (ms * 1e-3) / 1e9);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(a);
  cudaFree(b);
  *gbs = best;
  return cudaGetLastError() == cudaSuccess ? DEKF_OK : DEKF_ECUDA;
}
