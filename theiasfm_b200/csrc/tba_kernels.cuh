// tba_kernels.cuh -- sm_100a kernels of the bundle-adjustment engine.
//
// Replaces the arithmetic that ceres::Solve (called at
// src/theia/sfm/bundle_adjustment/bundle_adjuster.cc:205) performs for Theia's
// reprojection-error problem: residual/Jacobian evaluation, block accumulation,
// Schur elimination of the point blocks, SCHUR_JACOBI preconditioner and the
// implicit-Schur PCG matvec.  Layout and roofline per kernel: DESIGN.md section 4-5.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "tba_camera_models.cuh"
#include "tba_segments.h"
#include "tba_filter.cuh"
#include "tba_track_estimator.cuh"
#include "tba_two_view.cuh"

namespace tba {

constexpr int TILE = 256;   // observation slots per tile == threads per CTA
constexpr int MAXP = 256;   // max points per tile
constexpr int VB = 64;      // CTAs of the camera-space vector kernels (deterministic reductions)
constexpr int VT = 256;

// Device view of the packed problem.
struct DevProblem {
  int n_cam, n_group, n_pt, n_tiles;
  int ne;                      // n_cam * 6
  int ncs;                     // n_cam*6 + n_group*10 (camera-space vector length)
  int single_group;            // n_group == 1: block-reduce the intrinsics accumulations
  int loss_type; double loss_width;
  int ablate;                  // TBA_ABLATE (timing diagnostics of the matvec, results are WRONG when non-zero): bit0 no camera-side
                               // REDs, bit1 no x gather, bit2 no shared-intrinsics warp sums, bit3 no segmented reduction
  // parameters: current x and candidate
  double *ext, *intr, *pt, *ext_c, *intr_c, *pt_c;
  const int* cam_group; const int* group_model;
  double* cam_rec;             // [n_cam][kCamRec] for x
  double* cam_rec_c;           // ... for the candidate
  double* cam_s4;              // [n_cam][4] compact rotation scalars for x (cam_scalars)
  double* cam_s4_c;            // ... for the candidate
  // observation slots (tile-major, point-sorted)
  const int* slot_cam;         // -1 = padding
  const int* slot_pt;          // packed point id
  const uint8_t* slot_flags;   // bit0: all parameter blocks constant (Ceres fixed_cost)
  const int16_t* slot_run;     // (point, group) run index inside the tile
  const int* tile_pt_begin;    // [n_tiles + 1]
  const int* tile_nruns;       // [n_tiles]
  const uint8_t* tile_flags;   // [n_tiles] bit0: long tile (tracks > 32 observations; points may straddle warps)
  const double* xy;            // [tile][2][TILE]
  double* J;                   // [tile][NJ][TILE], NJ = 14 + 2 NI
  double* res;                 // [tile][2][TILE] robustified residuals
  // per point
  double* Hpp;                 // [n_pt][10] sym J_p^T J_p (unscaled)
  double* gp;                  // [n_pt][4]  J_p^T r
  double* Mp;                  // [n_pt][10] S_p (S_p Hpp S_p + D_p^2)^-1 S_p
  double* sp;                  // [n_pt][4] masked Jacobi scale
  double* dpt;                 // [n_pt][4] unscaled point delta
  const uint8_t* pt_const;
};

// ---------------------------------------------------------------- utilities
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

// Sum over the CTA (VT or TILE threads); result valid in thread 0.
__device__ __forceinline__ double block_sum(double v, double* s_red /*[32]*/) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) s_red[wid] = v;
  __syncthreads();
  double t = 0.0;
  if (wid == 0) {
    t = lane < (blockDim.x >> 5) ? s_red[lane] : 0.0;
    t = warp_sum(t);
  }
  return t;
}

// Segmented (by contiguous equal key) inclusive-from-the-right warp reduction:
// the FIRST lane of every run ends up holding the run's sum.
__device__ __forceinline__ double seg_reduce(double v, int key, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double ov = __shfl_down_sync(0xffffffffu, v, o);
    const int ok = __shfl_down_sync(0xffffffffu, key, o);
    if (lane + o < 32 && ok == key) v += ov;
  }
  return v;
}

// The same reduction when the run structure is known from a ballot of the run heads: lane + o belongs to lane's run iff
// lane + o <= run_last (runs are contiguous), so the key does not have to be shuffled along with every value -- 5 shuffles per
// reduced value instead of 10 (bit-identical sums: same additions in the same order).
__device__ __forceinline__ double seg_reduce_to(double v, int run_last, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double ov = __shfl_down_sync(0xffffffffu, v, o);
    if (lane + o <= run_last) v += ov;
  }
  return v;
}

// fp64 reduction into GLOBAL memory without a return value.  Written as the PTX `red` itself: left to the compiler, atomicAdd
// becomes ATOMG (with its round trip back to the SM) as soon as the kernel also contains a __threadfence -- the multi-GPU
// epilogue of k_schur_stream made every matvec 13 % slower that way (round 2, GPU call 4: RED wavefronts 0, ATOMG instead).
__device__ __forceinline__ void red_add(double* p, double v) {
#ifdef TBA_EMULATE
  atomicAdd(p, v);
#else
  asm volatile("red.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
#endif
}

// Transposed RED emission (default; TBA_TRED=0: lane-per-row REDs).  A lane-per-observation RED of an N-double camera row touches 32
// different 32-byte sectors per instruction (32 cameras), i.e. N x 32 sector operations at the L2 atomic units, which
// is what bounds these kernels (profiles/: k_precond_ext 88 % lts throughput at one sector operation per RED).  Here
// the warp first stages its 32 rows in shared memory ([32][N] doubles, lane-major) and then emits them element-major:
// instruction k covers elements 32k..32k+31 of the staged [32*N] array, so consecutive lanes add to consecutive doubles
// of the same row and one RED instruction covers about 32*8/32 = 8..11 sectors instead of 32 -- the same N RED
// instructions per warp, about a third of the sector operations.  sbase[o] = element offset of observation o's row in
// dst, < 0 for padding lanes.  The caller brackets the staging stores with __syncwarp().
template <int N>
__device__ __forceinline__ void warp_stage_row(double* __restrict__ stage, int* __restrict__ sbase, const double (&v)[N], int base, int lane) {
#pragma unroll
  for (int j = 0; j < N; ++j) stage[lane * N + j] = v[j];
  sbase[lane] = base;
}
template <int N>
__device__ __forceinline__ void warp_red_rows(double* __restrict__ dst, const double* __restrict__ stage, const int* __restrict__ sbase, int lane) {
#pragma unroll
  for (int k = 0; k < N; ++k) {
    const int e = k * 32 + lane;
    const int o = e / N;
    const int b = sbase[o];
    if (b >= 0) red_add(dst + (size_t)b + (e - o * N), stage[e]);
  }
}

// ------------------------------------------------------------ camera prep
// rec: the full [kCamRec] record (R | J_l) for the kernels that run rarely; s4 (optional): the four scalars the hot
// per-observation kernels gather instead (k_linearize, k_cost rebuild R and J_l from ext + s4 in registers).
__global__ void k_cam_prep(int n_cam, const double* __restrict__ ext, double* __restrict__ rec, double* __restrict__ s4 = nullptr) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < n_cam) cam_prep(ext + (size_t)c * 6 + 3, rec + (size_t)c * kCamRec, s4 ? s4 + (size_t)c * 4 : nullptr);
}
// The observing camera's parameters through vector gathers: ext[6] (3 x 128 bit) + s4[4] (2 x 128 bit), expanded in registers.
__device__ __forceinline__ void gather_camera(const double* __restrict__ ext, const double* __restrict__ s4, int cam, double Cw[6], double rec[kCamRec]) {
  const double2* e2 = reinterpret_cast<const double2*>(ext + (size_t)cam * 6);
  const double2 e0 = __ldg(e2), e1 = __ldg(e2 + 1), e3 = __ldg(e2 + 2);
  const double2* q2 = reinterpret_cast<const double2*>(s4 + (size_t)cam * 4);
  const double2 q0 = __ldg(q2), q1 = __ldg(q2 + 1);
  Cw[0] = e0.x; Cw[1] = e0.y; Cw[2] = e1.x; Cw[3] = e1.y; Cw[4] = e3.x; Cw[5] = e3.y;
  cam_rec_expand(e1.y, e3.x, e3.y, q0.x, q0.y, q1.x, q1.y, rec);
}

// ---------------------------------------------------- replicated scalar accumulators
// Sums that every warp of every tile adds into the SAME few addresses (shared-intrinsics gradient / matvec output,
// cost, ...) go to one of NREP replicas (row = warp id mod NREP) and are folded by k_fold afterwards: avoids the
// same-address serialisation of fp64 RED at L2 and keeps warps free of block-level barriers.
constexpr int NREP = 256;
constexpr int REPW = 32;  // columns: 0..9 intrinsics (a), 10..19 intrinsics (b), 20 cost, 21 fixed cost, 22 failed, 23 model cost change
__device__ __forceinline__ double* rep_row(double* rep) {
  return rep + (size_t)((blockIdx.x * (TILE / 32) + (threadIdx.x >> 5)) & (NREP - 1)) * REPW;
}
// dst_a[0..9] += column sums 0..9, dst_b[0..9] += columns 10..19, dst_s[0..3] += columns 20..23; replicas re-zeroed.
__global__ void k_fold(double* __restrict__ rep, double* __restrict__ dst_a, double* __restrict__ dst_b, double* __restrict__ dst_s) {
  const int j = threadIdx.x;
  if (j >= REPW) return;
  double v = 0.0;
  for (int r = 0; r < NREP; ++r) { v += rep[(size_t)r * REPW + j]; rep[(size_t)r * REPW + j] = 0.0; }
  if (j < 10) { if (dst_a) dst_a[j] += v; }
  else if (j < 20) { if (dst_b) dst_b[j - 10] += v; }
  else if (j < 24) { if (dst_s) dst_s[j - 20] += v; }
}

// Index of the first lane of the run (contiguous equal key) that `lane` belongs to, from the ballot of run heads.
__device__ __forceinline__ int run_head_lane(unsigned heads, int lane) { return 31 - __clz(heads & (0xffffffffu >> (31 - lane))); }

// Element (row k, lane) of the per-warp slice of a [tile][warp][rows][32] array.
__device__ __forceinline__ size_t wslice(int tile, int warp, int rows) { return ((size_t)tile * (TILE / 32) + warp) * rows * 32; }

// ---------------------------------------------------------- K1 linearise
// One thread per observation slot.  Writes the compact linearisation and the robustified residual
// ([tile][warp][NJ][32] / [tile][warp][2][32]: a warp's slice is contiguous), the per-point blocks, the camera-side
// gradient / squared column norms (fp64 RED to global) and cost / failure counters (replicas).
// Normal tiles: a point never straddles a warp -> per-point sums by warp-shuffle segmented reduction only, no
// block barrier.  Long tiles (tracks > 32 observations): combined across warps in shared memory.
template <uint32_t IMASK, bool EXT = false, bool TRED = false, int MINB = 1>
__global__ void __launch_bounds__(TILE, MINB) k_linearize(DevProblem P, double* __restrict__ g_cs, double* __restrict__ cn_cs,
                                                    double* __restrict__ rep) {
  constexpr int NI = popcount10(IMASK);
  constexpr int NJ = 14 + 2 * NI;
  __shared__ double s_acc[MAXP][14];
  const int tile = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool long_tile = (P.tile_flags[tile] & 1) != 0;
  const int p0 = P.tile_pt_begin[tile], npt = P.tile_pt_begin[tile + 1] - p0;
  if (long_tile) {
    for (int i = tid; i < npt * 14; i += TILE) (&s_acc[0][0])[i] = 0.0;
    __syncthreads();
  }
  const size_t slot = (size_t)tile * TILE + tid;
  const int cam = P.slot_cam[slot];
  const bool valid = cam >= 0;
  double cost = 0.0, fixed = 0.0, failed = 0.0;
  double Ja[6] = {0, 0, 0, 0, 0, 0}, Jw[6] = {0, 0, 0, 0, 0, 0}, Jh[2] = {0, 0}, r[2] = {0, 0};
  double Ji[2 * NI + 1];
#pragma unroll
  for (int j = 0; j < 2 * NI; ++j) Ji[j] = 0.0;
  int pl = -1 - lane, grp = 0;  // padding lanes: unique negative keys (each its own run)
  double h = 0.0;
  if (valid) {
    const int pt = P.slot_pt[slot];
    pl = pt - p0;
    grp = P.cam_group[cam];
    const double4 X = *reinterpret_cast<const double4*>(P.pt + (size_t)pt * 4);
    h = X.w;
    const double* xyw = P.xy + wslice(tile, warp, 2) + lane;
    const double x = xyw[0], y = xyw[32];
    double rho0 = 0.0;
    double Cw[6], rec[kCamRec];
    gather_camera(P.ext, P.cam_s4, cam, Cw, rec);
    const bool ok = linearize_obs_any<IMASK, EXT>(P.group_model[grp], Cw, rec,
                                         P.intr + (size_t)grp * 10, X.x, X.y, X.z, X.w, x, y, P.loss_type, P.loss_width,
                                         r, rho0, Ja, Jw, Jh, Ji);
    const bool is_fixed = (P.slot_flags[slot] & 1) != 0;
    if (!ok) failed = 1.0;
    else if (is_fixed) fixed = 0.5 * rho0;  // every block constant: Ceres removes the residual (fixed_cost)
    else cost = 0.5 * rho0;
    if (!ok || is_fixed) {
#pragma unroll
      for (int j = 0; j < 6; ++j) { Ja[j] = 0.0; Jw[j] = 0.0; }
      Jh[0] = Jh[1] = 0.0; r[0] = r[1] = 0.0;
#pragma unroll
      for (int j = 0; j < 2 * NI; ++j) Ji[j] = 0.0;
    }
  }
  // store the compact linearisation (each warp writes 256-byte rows of its own slice)
  {
    double* Jt = P.J + wslice(tile, warp, NJ) + lane;
#pragma unroll
    for (int j = 0; j < 6; ++j) Jt[j * 32] = Ja[j];
#pragma unroll
    for (int j = 0; j < 6; ++j) Jt[(6 + j) * 32] = Jw[j];
    Jt[12 * 32] = Jh[0];
    Jt[13 * 32] = Jh[1];
#pragma unroll
    for (int j = 0; j < 2 * NI; ++j) Jt[(14 + j) * 32] = Ji[j];
    double* rt = P.res + wslice(tile, warp, 2) + lane;
    rt[0] = r[0];
    rt[32] = r[1];
  }
  // per-point blocks: H_pp = J_p^T J_p (10, row-major upper), g_p = J_p^T r with J_p = [Ja | Jh]
  {
    const double jp0[4] = {Ja[0], Ja[1], Ja[2], Jh[0]}, jp1[4] = {Ja[3], Ja[4], Ja[5], Jh[1]};
    double acc[14];
    int n = 0;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = a; b < 4; ++b) acc[n++] = jp0[a] * jp0[b] + jp1[a] * jp1[b];
#pragma unroll
    for (int a = 0; a < 4; ++a) acc[10 + a] = jp0[a] * r[0] + jp1[a] * r[1];
    const int prev = __shfl_up_sync(0xffffffffu, pl, 1);
    const bool head = valid && (lane == 0 || prev != pl);
#pragma unroll
    for (int j = 0; j < 14; ++j) acc[j] = seg_reduce(acc[j], pl, lane);
    if (head) {
      if (long_tile) {
#pragma unroll
        for (int j = 0; j < 14; ++j) atomicAdd(&s_acc[pl][j], acc[j]);
      } else {
        double2* H2 = reinterpret_cast<double2*>(P.Hpp + (size_t)(p0 + pl) * 10);
#pragma unroll
        for (int j = 0; j < 5; ++j) H2[j] = make_double2(acc[2 * j], acc[2 * j + 1]);
        double2* G2 = reinterpret_cast<double2*>(P.gp + (size_t)(p0 + pl) * 4);
        G2[0] = make_double2(acc[10], acc[11]);
        G2[1] = make_double2(acc[12], acc[13]);
      }
    }
  }
  // camera-side gradient and squared column norms: J_c = [-h Ja | Jw]
  if (TRED && !long_tile) {
    // transposed RED emission: both 6-rows staged per warp in the (idle on normal tiles) s_acc area, emitted element-major
    double gv[6], cv[6];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double c0 = -h * Ja[j], c1 = -h * Ja[3 + j];
      gv[j] = c0 * r[0] + c1 * r[1];
      cv[j] = c0 * c0 + c1 * c1;
      gv[3 + j] = Jw[j] * r[0] + Jw[3 + j] * r[1];
      cv[3 + j] = Jw[j] * Jw[j] + Jw[3 + j] * Jw[3 + j];
    }
    static_assert(MAXP * 14 >= (TILE / 32) * (2 * 32 * 6 + 16), "s_acc too small for the TRED staging");
    double* stage = &s_acc[0][0] + warp * (2 * 32 * 6 + 16);
    int* sbase = reinterpret_cast<int*>(stage + 2 * 32 * 6);
    warp_stage_row<6>(stage, sbase, gv, valid ? cam * 6 : -1, lane);
    warp_stage_row<6>(stage + 32 * 6, sbase, cv, valid ? cam * 6 : -1, lane);
    __syncwarp();
    warp_red_rows<6>(g_cs, stage, sbase, lane);
    warp_red_rows<6>(cn_cs, stage + 32 * 6, sbase, lane);
  } else if (valid) {
    double* gc = g_cs + (size_t)cam * 6;
    double* cc = cn_cs + (size_t)cam * 6;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double c0 = -h * Ja[j], c1 = -h * Ja[3 + j];
      red_add(gc + j, c0 * r[0] + c1 * r[1]);
      red_add(cc + j, c0 * c0 + c1 * c1);
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      red_add(gc + 3 + j, Jw[j] * r[0] + Jw[3 + j] * r[1]);
      red_add(cc + 3 + j, Jw[j] * Jw[j] + Jw[3 + j] * Jw[3 + j]);
    }
  }
  double* rr = rep_row(rep);
  if (NI > 0) {
    if (P.single_group) {
#pragma unroll
      for (int j = 0; j < NI; ++j) {
        const double gsum = warp_sum(Ji[j] * r[0] + Ji[NI + j] * r[1]);
        const double csum = warp_sum(Ji[j] * Ji[j] + Ji[NI + j] * Ji[NI + j]);
        if (lane == 0) { red_add(rr + nth_bit(IMASK, j), gsum); red_add(rr + 10 + nth_bit(IMASK, j), csum); }
      }
    } else if (valid) {
#pragma unroll
      for (int j = 0; j < NI; ++j) {
        red_add(g_cs + P.ne + (size_t)grp * 10 + nth_bit(IMASK, j), Ji[j] * r[0] + Ji[NI + j] * r[1]);
        red_add(cn_cs + P.ne + (size_t)grp * 10 + nth_bit(IMASK, j), Ji[j] * Ji[j] + Ji[NI + j] * Ji[NI + j]);
      }
    }
  }
  {
    const double c = warp_sum(cost), f = warp_sum(fixed), e = warp_sum(failed);
    if (lane == 0) {
      red_add(rr + 20, c);
      if (f != 0.0) red_add(rr + 21, f);
      if (e != 0.0) red_add(rr + 22, e);
    }
  }
  if (long_tile) {
    __syncthreads();
    for (int i = tid; i < npt * 14; i += TILE) {
      const int p = i / 14, j = i - p * 14;
      if (j < 10) P.Hpp[(size_t)(p0 + p) * 10 + j] = s_acc[p][j];
      else P.gp[(size_t)(p0 + p) * 4 + (j - 10)] = s_acc[p][j];
    }
  }
}

// ------------------------------------------------------- K3 cost at candidate
template <bool EXT = false>
__global__ void __launch_bounds__(TILE) k_cost(DevProblem P, const double* __restrict__ ext, const double* __restrict__ s4,
                                               const double* __restrict__ intr, const double* __restrict__ pt,
                                               double* __restrict__ rep) {
  const int tile = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t slot = (size_t)tile * TILE + tid;
  const int cam = P.slot_cam[slot];
  double cost = 0.0, fixed = 0.0, failed = 0.0;
  if (cam >= 0) {
    const int p = P.slot_pt[slot], grp = P.cam_group[cam];
    const double4 X = *reinterpret_cast<const double4*>(pt + (size_t)p * 4);
    const double* xyw = P.xy + wslice(tile, warp, 2) + lane;
    double r0, r1;
    double Cw[6], rec[kCamRec];
    gather_camera(ext, s4, cam, Cw, rec);
    if (!reproject_any<EXT>(P.group_model[grp], Cw, rec, intr + (size_t)grp * 10, X.x, X.y,
                   X.z, X.w, xyw[0], xyw[32], r0, r1)) {
      failed = 1.0;
    } else {
      double rho[3];
      loss_evaluate(P.loss_type, P.loss_width, r0 * r0 + r1 * r1, rho);
      if (P.slot_flags[slot] & 1) fixed = 0.5 * rho[0]; else cost = 0.5 * rho[0];
    }
  }
  const double c = warp_sum(cost), f = warp_sum(fixed), e = warp_sum(failed);
  if (lane == 0) {
    double* rr = rep_row(rep);
    red_add(rr + 20, c);
    if (f != 0.0) red_add(rr + 21, f);
    if (e != 0.0) red_add(rr + 22, e);
  }
}

// ------------------------------------------ N1: post-BA track filter on the device-resident problem
// SetOutlierTracksToUnestimated (src/theia/sfm/set_outlier_tracks_to_unestimated.cc:62-136) for every packed point:
// status 1 = "bad reprojection" (a view sees the point at negative depth, or the mean squared reprojection error over
// the views exceeds max_sq_err), status 2 = "insufficient viewing angle" (no pair of unit rays X/h - C with
// dot < cos_min_angle: SufficientTriangulationAngle, triangulation.cc:236-250), 0 = keep.  The reference's loop
// "breaks" at the first negative depth, which only affects counters that are discarded for such a track, so the
// result does not depend on its (hash-map) view order.  One thread per point; mean_sq_err (optional) receives the
// mean squared reprojection error (ComputeStatisticsForTrack, select_good_tracks_for_bundle_adjustment.cc:79-108).
template <bool EXT>
__global__ void k_filter_tracks(DevProblem P, const long long* __restrict__ pt_slot, const int* __restrict__ pt_len, double max_sq_err,
                                double cos_min_angle, uint8_t* __restrict__ status, double* __restrict__ mean_sq_err) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= P.n_pt) return;
  FilterView V;
  V.ext = P.ext; V.cam_rec = P.cam_rec; V.intr = P.intr; V.pt = P.pt; V.xy = P.xy;
  V.slot_cam = P.slot_cam; V.cam_group = P.cam_group; V.group_model = P.group_model;
  double mean;
  status[k] = filter_track<EXT>(V, k, pt_slot[k], pt_len[k], max_sq_err, cos_min_angle, &mean);
  if (mean_sq_err) mean_sq_err[k] = mean;
}

// --------------------------------------------------------- N3: batched track estimation / per-track BA
// Unit viewing ray of every observation slot (Camera::PixelToUnitDepthRay, normalised): one thread per slot, coalesced
// reads of xy and writes of ray[slot/32][3][32]; the iterative undistortion makes this the arithmetic half of
// TrackEstimator::EstimateTrack, and it is observation-parallel.
__global__ void k_track_rays(DevProblem P, long long n_slots, double* __restrict__ ray) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  const int cam = P.slot_cam[s];
  if (cam < 0) return;
  const int grp = P.cam_group[cam];
  const long long wq = s >> 5;
  const int l = (int)(s & 31);
  double d[3];
  observation_ray(P.group_model[grp], P.cam_rec + (size_t)cam * kCamRec, P.intr + (size_t)grp * 10, P.xy[(size_t)(wq * 2) * 32 + l],
                  P.xy[(size_t)(wq * 2 + 1) * 32 + l], d);
  ray[(size_t)(wq * 3 + 0) * 32 + l] = d[0]; ray[(size_t)(wq * 3 + 1) * 32 + l] = d[1]; ray[(size_t)(wq * 3 + 2) * 32 + l] = d[2];
}

__device__ inline FilterView filter_view(const DevProblem& P) {
  FilterView V;
  V.ext = P.ext; V.cam_rec = P.cam_rec; V.intr = P.intr; V.pt = P.pt; V.xy = P.xy;
  V.slot_cam = P.slot_cam; V.cam_group = P.cam_group; V.group_model = P.group_model;
  return V;
}

// TrackEstimator::EstimateTrack for every non-constant packed point (one thread per point; thousands of independent
// 4-parameter problems).  cost2[k] = {initial, final} cost of the per-track BA (-1 when it did not run).
template <bool EXT>
__global__ void k_estimate_tracks(DevProblem P, const long long* __restrict__ pt_slot, const int* __restrict__ pt_len,
                                  const double* __restrict__ ray, TrackEstimatorOptions o, uint8_t* __restrict__ status,
                                  double* __restrict__ cost2) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= P.n_pt) return;
  if (P.pt_const[k]) { status[k] = kTrackSkipped; cost2[2 * k] = cost2[2 * k + 1] = -1.0; return; }
  const FilterView V = filter_view(P);
  double X[4] = {P.pt[(size_t)k * 4], P.pt[(size_t)k * 4 + 1], P.pt[(size_t)k * 4 + 2], P.pt[(size_t)k * 4 + 3]};
  PointLmResult lm;
  status[k] = estimate_track<EXT>(V, ray, pt_slot[k], pt_len[k], X, o, &lm);
  for (int j = 0; j < 4; ++j) P.pt[(size_t)k * 4 + j] = X[j];
  cost2[2 * k] = lm.initial_cost; cost2[2 * k + 1] = lm.final_cost;
}

// BundleAdjustTrack (bundle_adjustment.cc:96-107) for every non-constant packed point: LM on the point, cameras constant.
// status: Ceres termination type (0 CONVERGENCE, 1 NO_CONVERGENCE, 2 FAILURE), 255 = constant point (not adjusted).
template <bool EXT>
__global__ void k_adjust_tracks(DevProblem P, const long long* __restrict__ pt_slot, const int* __restrict__ pt_len, PointLmOptions o,
                                uint8_t* __restrict__ status, double* __restrict__ cost2) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= P.n_pt) return;
  if (P.pt_const[k]) { status[k] = kTrackSkipped; cost2[2 * k] = cost2[2 * k + 1] = -1.0; return; }
  const FilterView V = filter_view(P);
  double X[4] = {P.pt[(size_t)k * 4], P.pt[(size_t)k * 4 + 1], P.pt[(size_t)k * 4 + 2], P.pt[(size_t)k * 4 + 3]};
  const PointLmResult lm = point_lm<EXT>(V, pt_slot[k], pt_len[k], X, o);
  for (int j = 0; j < 4; ++j) P.pt[(size_t)k * 4 + j] = X[j];
  status[k] = (uint8_t)lm.termination;
  cost2[2 * k] = lm.initial_cost; cost2[2 * k + 1] = lm.final_cost;
}

// --------------------------------------------------------- N3: batched two-view bundle adjustment
// BundleAdjustTwoViews for many image pairs at once: one WARP runs the whole Levenberg-Marquardt of one pair
// (tba_two_view.cuh, WarpTeam): the passes over the pair's few hundred correspondences are strided over the 32 lanes, the
// 8x8 reduced system and every scalar are all-reduced by shuffles so that all lanes take the same decisions.  Pairs are
// independent: geometric verification hands over thousands of them.
struct TwoViewBatchDev {
  int n_pairs;
  const long long* off;       // [n_pairs + 1] into the correspondence arrays
  const double* ext1; double* ext2; double* k1; double* k2;
  const int* model1; const int* model2;
  const uint8_t* const1; const uint8_t* const2;  // constant_cameraN_intrinsics
  const double* xy1; const double* xy2;
  double* pt; double* sp; double* pt_c;
  uint8_t* inlier; double sq_max_error;   // optional post-BA inlier flags (nullptr: skipped)
};
template <bool EXT>
__global__ void k_two_view_ba(TwoViewBatchDev B, PointLmOptions o, uint8_t* __restrict__ termination, double* __restrict__ cost2,
                              int* __restrict__ iterations) {
  const int p = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);  // one warp per pair (WarpTeam)
  if (p >= B.n_pairs) return;                                                  // warp-uniform
  TwoViewPair P;
  const long long b = B.off[p];
  P.ext1 = B.ext1 + (size_t)p * 6; P.ext2 = B.ext2 + (size_t)p * 6; P.k1 = B.k1 + (size_t)p * 10; P.k2 = B.k2 + (size_t)p * 10;
  P.model1 = B.model1[p]; P.model2 = B.model2[p]; P.free_f1 = B.const1[p] ? 0 : 1; P.free_f2 = B.const2[p] ? 0 : 1;
  P.n = (int)(B.off[p + 1] - b);
  P.pt = B.pt + (size_t)b * 4; P.xy1 = B.xy1 + (size_t)b * 2; P.xy2 = B.xy2 + (size_t)b * 2; P.sp = B.sp + (size_t)b * 4; P.pt_c = B.pt_c + (size_t)b * 4;
  const PointLmResult r = two_view_lm<EXT, WarpTeam>(P, o);
  if (B.inlier != nullptr) {
    __syncwarp();  // lane 0's write-back of the refined camera values is visible to the warp
    two_view_inliers<EXT, WarpTeam>(P, B.sq_max_error, B.inlier + (size_t)b);
  }
  if ((threadIdx.x & 31) == 0) {
    termination[p] = (uint8_t)r.termination;
    cost2[2 * p] = r.initial_cost; cost2[2 * p + 1] = r.final_cost;
    iterations[p] = r.iterations;
  }
}

// --------------------------------------------------------- per-point blocks
// 4x4 SPD inverse through Cholesky (Ceres: InvertPSDMatrix, llt().solve(I)); returns false if not PD.
__device__ inline bool spd4_inverse(const double* A /*10 upper*/, double* Ainv /*10 upper*/) {
  // A index: (0,0)=0 (0,1)=1 (0,2)=2 (0,3)=3 (1,1)=4 (1,2)=5 (1,3)=6 (2,2)=7 (2,3)=8 (3,3)=9
  const double a00 = A[0], a01 = A[1], a02 = A[2], a03 = A[3], a11 = A[4], a12 = A[5], a13 = A[6], a22 = A[7], a23 = A[8], a33 = A[9];
  if (!(a00 > 0.0)) return false;
  const double l00 = sqrt(a00), i00 = 1.0 / l00;
  const double l10 = a01 * i00, l20 = a02 * i00, l30 = a03 * i00;
  const double d1 = a11 - l10 * l10;
  if (!(d1 > 0.0)) return false;
  const double l11 = sqrt(d1), i11 = 1.0 / l11;
  const double l21 = (a12 - l20 * l10) * i11, l31 = (a13 - l30 * l10) * i11;
  const double d2 = a22 - l20 * l20 - l21 * l21;
  if (!(d2 > 0.0)) return false;
  const double l22 = sqrt(d2), i22 = 1.0 / l22;
  const double l32 = (a23 - l30 * l20 - l31 * l21) * i22;
  const double d3 = a33 - l30 * l30 - l31 * l31 - l32 * l32;
  if (!(d3 > 0.0)) return false;
  const double l33 = sqrt(d3), i33 = 1.0 / l33;
  // M = L^-1 (lower)
  const double m10 = -l10 * i00 * i11;
  const double m21 = -l21 * i11 * i22;
  const double m32 = -l32 * i22 * i33;
  const double m20 = -(l20 * i00 + l21 * m10) * i22;
  const double m31 = -(l31 * i11 + l32 * m21) * i33;
  const double m30 = -(l30 * i00 + l31 * m10 + l32 * m20) * i33;
  // A^-1 = M^T M
  Ainv[0] = i00 * i00 + m10 * m10 + m20 * m20 + m30 * m30;
  Ainv[1] = m10 * i11 + m20 * m21 + m30 * m31;
  Ainv[2] = m20 * i22 + m30 * m32;
  Ainv[3] = m30 * i33;
  Ainv[4] = i11 * i11 + m21 * m21 + m31 * m31;
  Ainv[5] = m21 * i22 + m31 * m32;
  Ainv[6] = m31 * i33;
  Ainv[7] = i22 * i22 + m32 * m32;
  Ainv[8] = m32 * i33;
  Ainv[9] = i33 * i33;
  return true;
}

// Jacobi scale of the point columns (iteration 0): s = 1 / (1 + sqrt(colnorm2)), 0 on constant points.
__global__ void k_point_scale(DevProblem P, int use_scaling) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P.n_pt) return;
  const bool c = P.pt_const[p] != 0;
  const double* H = P.Hpp + (size_t)p * 10;
  const double d[4] = {H[0], H[4], H[7], H[9]};
#pragma unroll
  for (int j = 0; j < 4; ++j) P.sp[(size_t)p * 4 + j] = c ? 0.0 : (use_scaling ? 1.0 / (1.0 + sqrt(d[j])) : 1.0);
}

// M_p = S (S Hpp S + D^2)^-1 S with D^2 = clamp(s^2 diag(Hpp), lo, hi) / radius; flag[0] += 1 if a block is not PD.
// Also the max-norm of the (masked) point gradient into gmax partials.
__global__ void k_point_blocks(DevProblem P, double radius, double lo, double hi, double* __restrict__ flag) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P.n_pt) return;
  double* M = P.Mp + (size_t)p * 10;
  if (P.pt_const[p]) {
#pragma unroll
    for (int j = 0; j < 10; ++j) M[j] = 0.0;
    return;
  }
  const double* H = P.Hpp + (size_t)p * 10;
  const double4 s4 = *reinterpret_cast<const double4*>(P.sp + (size_t)p * 4);
  const double s[4] = {s4.x, s4.y, s4.z, s4.w};
  double A[10], Ai[10];
  int n = 0;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = a; b < 4; ++b) { A[n] = s[a] * H[n] * s[b]; ++n; }
  const int dg[4] = {0, 4, 7, 9};
#pragma unroll
  for (int a = 0; a < 4; ++a) A[dg[a]] += fmin(fmax(A[dg[a]], lo), hi) / radius;
  if (!spd4_inverse(A, Ai)) {
    atomicAdd(flag, 1.0);
#pragma unroll
    for (int j = 0; j < 10; ++j) M[j] = 0.0;
    return;
  }
  n = 0;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = a; b < 4; ++b) { M[n] = s[a] * Ai[n] * s[b]; ++n; }
}

__device__ __forceinline__ void sym4_mul(const double* __restrict__ M, const double t[4], double u[4]) {
  u[0] = M[0] * t[0] + M[1] * t[1] + M[2] * t[2] + M[3] * t[3];
  u[1] = M[1] * t[0] + M[4] * t[1] + M[5] * t[2] + M[6] * t[3];
  u[2] = M[2] * t[0] + M[5] * t[1] + M[7] * t[2] + M[8] * t[3];
  u[3] = M[3] * t[0] + M[6] * t[1] + M[8] * t[2] + M[9] * t[3];
}

// ---------------------------------------------------- TMA (bulk async copy) helpers
#ifdef TBA_EMULATE
// CPU emulation build (tests/emu/cuda_emu.h): the bulk copy is a memcpy by the issuing lane, the mbarrier a flag the other lanes
// poll (yielding to the fiber scheduler).
// *bar counts the completed phases: the issuing lane's sequence "expect_tx, bulk copy, bulk copy ..." runs without a yield in
// between, so a phase is complete as soon as its expect_tx is visible; wait(parity) passes once phase `parity` is over.
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t) { *bar = 0; }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t) { *bar += 1; }
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t*) { memcpy(dst, src, bytes); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { while ((*bar & 1u) == parity) emu_yield(); }
__device__ __forceinline__ void fence_proxy_async_smem() {}
#else
// cp.async.bulk global -> shared::cta completing on an mbarrier (SASS: UBLKCP + SYNCS.ARRIVE.TRANS64).
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Never a silent hang: a bulk copy that does not land within ~2 s (4e9 SM cycles) is a bug -- report it and abort the kernel
// (the launch then fails with a CUDA error that the engine returns to the caller).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000ll) {
      printf("tba: mbarrier wait timed out (block %d thread %d parity %u)\n", (int)blockIdx.x, (int)threadIdx.x, parity);
      __trap();
    }
  }
}

__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

#endif  // TBA_EMULATE

// --------------------------------------------- K2 implicit Schur complement
// MODE 0: y += F^T (I - E M E^T) F xs                (PCG matvec; ImplicitSchurComplement::RightMultiply)
// MODE 1: y += F^T (I - E M E^T) r                   (reduced rhs; ImplicitSchurComplement::ComputeRHS)
// MODE 2: dpt = -M E^T (r - F xs);  rep[23] += model cost change  (BackSubstitute + ComputeTrustRegionStep)
// All with the UNSCALED stored Jacobian; the Jacobi scaling lives in xs (= s .* x), M and the
// post-scaling of y (k_pcg_* kernels).  xs: camera-space vector [n_cam*6 | n_group*10].
//
// Every WARP is autonomous on a normal tile: lane 0 issues one TMA bulk copy of the warp's contiguous slice of the
// compact Jacobian (NJ x 32 doubles) [+ residuals] into the warp's shared-memory stage, completing on the warp's
// own mbarrier; meanwhile all lanes gather their camera's x block (3 x 128-bit loads) and the head lanes fetch
// M_p, so the gather latency overlaps the copy.  Per-point sums: warp-shuffle segmented reduction (a point's
// observations are contiguous lanes of ONE warp), u_p = M_p t_p on the head lane, broadcast back by shuffle.
// Camera-side sums: fp64 RED.ADD to global; shared-intrinsics sums: warp reduce + RED to a replica row.
// No block barrier on this path.  Long tiles (tracks > 32 observations) combine the per-point sums across warps in
// shared memory (two block barriers).  Dynamic shared memory: TILE * (NJ + 2) doubles.
template <uint32_t IMASK, int MODE, bool TRED = true>
__global__ void __launch_bounds__(TILE, (14 + 2 * popcount10(IMASK)) <= 20 ? 4 : 2) k_schur(DevProblem P, const double* __restrict__ xs, double* __restrict__ y,
                                                double* __restrict__ rep, const int* __restrict__ done_flag, int tile0) {
  constexpr int NI = popcount10(IMASK);
  constexpr int NJ = 14 + 2 * NI;
  constexpr int WS = (NJ + 2) * 32;  // doubles per warp stage
  if (done_flag != nullptr && *done_flag) return;
#ifdef TBA_EMULATE
  double* s_dyn = emu::dyn_smem<double>();
#else
  extern __shared__ __align__(128) double s_dyn[];
#endif
  __shared__ double s_t[MAXP][4];
  __shared__ __align__(8) uint64_t s_bar[TILE / 32];
  const int tile = tile0 + blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double* sJ = s_dyn + (size_t)warp * WS;  // [NJ][32]
  double* sR = sJ + NJ * 32;               // [2][32]
  if (lane == 0) {
    mbar_init(&s_bar[warp], 1);
    constexpr uint32_t jbytes = NJ * 32 * 8, rbytes = (MODE != 0) ? 2 * 32 * 8 : 0;
    mbar_expect_tx(&s_bar[warp], jbytes + rbytes);
    bulk_g2s(sJ, P.J + wslice(tile, warp, NJ), jbytes, &s_bar[warp]);
    if (MODE != 0) bulk_g2s(sR, P.res + wslice(tile, warp, 2), rbytes, &s_bar[warp]);
  }
  const bool long_tile = (P.tile_flags[tile] & 1) != 0;
  const int p0 = P.tile_pt_begin[tile], npt = P.tile_pt_begin[tile + 1] - p0;
  if (long_tile) {
    for (int i = tid; i < npt * 4; i += TILE) (&s_t[0][0])[i] = 0.0;
  }
  const size_t slot = (size_t)tile * TILE + tid;
  const int cam = P.slot_cam[slot];
  const bool valid = cam >= 0;
  int pl = -1 - lane, grp = 0;
  double h = 0.0;
  double2 xa = make_double2(0.0, 0.0), xb = xa, xc = xa;
  double xi[NI + 1];
  if (valid) {
    pl = P.slot_pt[slot] - p0;
    grp = (TRED && P.single_group) ? 0 : P.cam_group[cam];  // TRED: no 32-sector gather when one group owns everything
    h = P.pt[(size_t)(p0 + pl) * 4 + 3];
    if (MODE != 1) {
      const double2* x2 = reinterpret_cast<const double2*>(xs + (size_t)((MODE == 0 && (P.ablate & 2)) ? lane : cam) * 6);
      xa = __ldg(x2); xb = __ldg(x2 + 1); xc = __ldg(x2 + 2);
      if (NI > 0) {
        const double* xg = xs + P.ne + (size_t)grp * 10;
#pragma unroll
        for (int j = 0; j < NI; ++j) xi[j] = __ldg(xg + nth_bit(IMASK, j));
      }
    }
  }
  const int prev = __shfl_up_sync(0xffffffffu, pl, 1);
  const bool head = lane == 0 || prev != pl;
  const unsigned heads = __ballot_sync(0xffffffffu, head);
  // head lanes prefetch M_p (normal tiles)
  double2 m01 = make_double2(0.0, 0.0), m23 = m01, m45 = m01, m67 = m01, m89 = m01;
  if (!long_tile && head && valid) {
    const double2* M2 = reinterpret_cast<const double2*>(P.Mp + (size_t)(p0 + pl) * 10);
    m01 = __ldg(M2); m23 = __ldg(M2 + 1); m45 = __ldg(M2 + 2); m67 = __ldg(M2 + 3); m89 = __ldg(M2 + 4);
  }
  if (long_tile) __syncthreads();  // s_t zeroed
  __syncwarp();
  mbar_wait(&s_bar[warp], 0);  // this warp's slice landed in shared memory
  const double* Jt = sJ + lane;
#define JA(j) Jt[(j) * 32]
#define JW(j) Jt[(6 + (j)) * 32]
#define JH(j) Jt[(12 + (j)) * 32]
#define JI(j) Jt[(14 + (j)) * 32]
  double w0 = 0.0, w1 = 0.0, r0 = 0.0, r1 = 0.0;
  if (valid) {
    if (MODE != 0) { r0 = sR[lane]; r1 = sR[32 + lane]; }
    if (MODE != 1) {
      w0 = -h * (JA(0) * xa.x + JA(1) * xa.y + JA(2) * xb.x) + JW(0) * xb.y + JW(1) * xc.x + JW(2) * xc.y;
      w1 = -h * (JA(3) * xa.x + JA(4) * xa.y + JA(5) * xb.x) + JW(3) * xb.y + JW(4) * xc.x + JW(5) * xc.y;
#pragma unroll
      for (int j = 0; j < NI; ++j) { w0 += JI(j) * xi[j]; w1 += JI(NI + j) * xi[j]; }
    }
    if (MODE == 1) { w0 = r0; w1 = r1; }
    if (MODE == 2) { w0 = r0 - w0; w1 = r1 - w1; }
  }
  // t_p = sum_o J_p^T w,  J_p = [Ja | Jh]
  double t[4] = {0.0, 0.0, 0.0, 0.0};
  if (valid) {
    t[0] = JA(0) * w0 + JA(3) * w1; t[1] = JA(1) * w0 + JA(4) * w1; t[2] = JA(2) * w0 + JA(5) * w1;
    t[3] = JH(0) * w0 + JH(1) * w1;
  }
  if (MODE == 0 && (P.ablate & 8)) {
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) t[j] = seg_reduce(t[j], pl, lane);
  }
  double u0, u1, u2, u3;
  if (!long_tile) {
    u0 = m01.x * t[0] + m01.y * t[1] + m23.x * t[2] + m23.y * t[3];
    u1 = m01.y * t[0] + m45.x * t[1] + m45.y * t[2] + m67.x * t[3];
    u2 = m23.x * t[0] + m45.y * t[1] + m67.y * t[2] + m89.x * t[3];
    u3 = m23.y * t[0] + m67.x * t[1] + m89.x * t[2] + m89.y * t[3];
    if (MODE == 2 && head && valid) {
      double2* d = reinterpret_cast<double2*>(P.dpt + (size_t)(p0 + pl) * 4);
      d[0] = make_double2(-u0, -u1);
      d[1] = make_double2(-u2, -u3);
    }
    const int hl = run_head_lane(heads, lane);
    u0 = __shfl_sync(0xffffffffu, u0, hl); u1 = __shfl_sync(0xffffffffu, u1, hl);
    u2 = __shfl_sync(0xffffffffu, u2, hl); u3 = __shfl_sync(0xffffffffu, u3, hl);
  } else {
    if (head && valid) {
#pragma unroll
      for (int j = 0; j < 4; ++j) atomicAdd(&s_t[pl][j], t[j]);
    }
    __syncthreads();
    if (tid < npt) {
      const double tt[4] = {s_t[tid][0], s_t[tid][1], s_t[tid][2], s_t[tid][3]};
      double uu[4];
      sym4_mul(P.Mp + (size_t)(p0 + tid) * 10, tt, uu);
      s_t[tid][0] = uu[0]; s_t[tid][1] = uu[1]; s_t[tid][2] = uu[2]; s_t[tid][3] = uu[3];
      if (MODE == 2) {
        double* d = P.dpt + (size_t)(p0 + tid) * 4;
        d[0] = -uu[0]; d[1] = -uu[1]; d[2] = -uu[2]; d[3] = -uu[3];
      }
    }
    __syncthreads();
    u0 = u1 = u2 = u3 = 0.0;
    if (valid) { u0 = s_t[pl][0]; u1 = s_t[pl][1]; u2 = s_t[pl][2]; u3 = s_t[pl][3]; }
  }
  double z0 = 0.0, z1 = 0.0;
  if (valid) {
    z0 = w0 - (JA(0) * u0 + JA(1) * u1 + JA(2) * u2 + JH(0) * u3);
    z1 = w1 - (JA(3) * u0 + JA(4) * u1 + JA(5) * u2 + JH(1) * u3);
  }
  double* rr = rep_row(rep);
  if (MODE == 2) {
    // model residual m = J * step = -(F xs + E u) = -(r - z); contribution -m.(r + m/2)
    double mcc = 0.0;
    if (valid && !(P.slot_flags[slot] & 1)) {
      const double m0 = -(r0 - z0), m1 = -(r1 - z1);
      mcc = -(m0 * (r0 + 0.5 * m0) + m1 * (r1 + 0.5 * m1));
    }
    mcc = warp_sum(mcc);
    if (lane == 0) red_add(rr + 23, mcc);
    return;
  }
  if (TRED) {
    // camera-side contributions staged per warp and emitted element-major (warp_red_rows); TBA_TRED=0: one RED per lane and row element
    double yv[6];
#pragma unroll
    for (int j = 0; j < 3; ++j) yv[j] = valid ? -h * (JA(j) * z0 + JA(3 + j) * z1) : 0.0;
#pragma unroll
    for (int j = 0; j < 3; ++j) yv[3 + j] = valid ? JW(j) * z0 + JW(3 + j) * z1 : 0.0;
    double yi[NI + 1];
#pragma unroll
    for (int j = 0; j < NI; ++j) yi[j] = valid ? JI(j) * z0 + JI(NI + j) * z1 : 0.0;
    __syncwarp();  // every lane has finished reading the J slice: its first 6.5 rows are reused as staging [32][6] + 32 ints
    int* sbase = reinterpret_cast<int*>(sJ + 32 * 6);
    warp_stage_row<6>(sJ, sbase, yv, valid ? cam * 6 : -1, lane);
    __syncwarp();
    if (!(MODE == 0 && (P.ablate & 1))) warp_red_rows<6>(y, sJ, sbase, lane);
    if (NI > 0) {
      if (P.single_group) {
        if (MODE == 0 && (P.ablate & 4)) {
          double v = 0.0;
#pragma unroll
          for (int j = 0; j < NI; ++j) v += yi[j];
          if (v == 1.2345e300) red_add(rr, v);
        } else {
#pragma unroll
        for (int j = 0; j < NI; ++j) {
          const double v = warp_sum(yi[j]);
          if (lane == 0) red_add(rr + nth_bit(IMASK, j), v);
        }
        }
      } else if (valid) {
#pragma unroll
        for (int j = 0; j < NI; ++j) red_add(y + P.ne + (size_t)grp * 10 + nth_bit(IMASK, j), yi[j]);
      }
    }
    return;
  }
  if (valid) {
    double* yc = y + (size_t)cam * 6;
#pragma unroll
    for (int j = 0; j < 3; ++j) red_add(yc + j, -h * (JA(j) * z0 + JA(3 + j) * z1));
#pragma unroll
    for (int j = 0; j < 3; ++j) red_add(yc + 3 + j, JW(j) * z0 + JW(3 + j) * z1);
  }
  if (NI > 0) {
    if (P.single_group) {
#pragma unroll
      for (int j = 0; j < NI; ++j) {
        const double v = warp_sum(valid ? JI(j) * z0 + JI(NI + j) * z1 : 0.0);
        if (lane == 0) red_add(rr + nth_bit(IMASK, j), v);
      }
    } else if (valid) {
#pragma unroll
      for (int j = 0; j < NI; ++j) red_add(y + P.ne + (size_t)grp * 10 + nth_bit(IMASK, j), JI(j) * z0 + JI(NI + j) * z1);
    }
  }
#undef JA
#undef JW
#undef JH
#undef JI
}

// --------------------------------------------- fused matvec + all-reduce over NVLink peer memory (multi-GPU)
// Every rank owns an "inbox" [2][world][cap] in its own HBM that all peers can write (CUDA IPC / peer access).  After a grid
// barrier inside k_schur_stream<., 0> (its persistent CTAs are co-resident) every CTA STORES its slice of the rank's complete
// partial y into slot `rank` of every peer's inbox (buffer seq & 1) -- 16-byte stores over NVLink from all SMs, no separate
// collective launch -- and the CTA that finishes last releases flags[rank] = seq on every peer.  The consumer (k_pcg_a / k_pcg_reset_bz) acquires the `world` flags of its own
// inbox and sums the slots in rank order: the same bits on every rank (the replicated PCG state stays in lockstep) and
// run-to-run reproducible for a given world size.  Two buffers suffice: a rank can be at most one exchange ahead of a peer,
// because exchange k+1 needs the sums of exchange k, to which every peer contributed after it consumed exchange k-1.
struct P2pDev {
  int world = 1, rank = 0;
  unsigned long long seq = 0;
  size_t cap = 0;                        // doubles per slot
  double* const* inbox = nullptr;        // [world] base pointers of the ranks' inboxes (inbox[rank] is the local one)
  unsigned long long* const* flags = nullptr;  // [world] base pointers of the ranks' flag arrays ([world] each)
  int* ctr = nullptr;                    // local counters [2]: CTAs at the grid barrier / CTAs done pushing (zeroed before every matvec by k_pcg_c / k_pcg_reset_a)
};
#ifdef TBA_EMULATE
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) { *p = v; }
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) { return *p; }
__device__ __forceinline__ double ld_cg(const double* p) { return *p; }
#else
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ double ld_cg(const double* p) { return __ldcg(p); }
#endif
// Consumer side: wait for the `world` flags of the local inbox (threads 0 .. world-1), then a block barrier.
__device__ __forceinline__ void p2p_wait(const P2pDev& pp) {
  if ((int)threadIdx.x < pp.world) {
    const unsigned long long* f = pp.flags[pp.rank] + threadIdx.x;
#ifndef TBA_EMULATE
    const long long t0 = clock64();
#endif
    while (ld_acquire_sys(f) < pp.seq) {
#ifdef TBA_EMULATE
      emu_yield();
#else
      if (clock64() - t0 > 20000000000ll) { printf("tba: rank %d waited 10 s for the partial sums of rank %d (exchange %llu)\n", pp.rank, (int)threadIdx.x, pp.seq); __trap(); }
#endif
    }
  }
  __syncthreads();
}
__device__ __forceinline__ double p2p_sum(const P2pDev& pp, int i) {
  const double* base = pp.inbox[pp.rank] + (size_t)(pp.seq & 1ull) * pp.world * pp.cap + i;
  double v = 0.0;
  for (int q = 0; q < pp.world; ++q) v += ld_cg(base + (size_t)q * pp.cap);
  return v;
}

// --------------------------------------------- K2s: persistent streaming implicit Schur complement (round 2)
// Same three operators as k_schur (MODE 0 matvec, 1 reduced rhs, 2 back-substitution) over the NORMAL tiles, restructured
// around what the round-1 captures showed: the tile-per-CTA kernel is latency bound (one TMA round trip + two levels of
// dependent gathers per 32 observations and CTA lifetime), not bandwidth or issue bound.
//   * persistent CTAs (one per SM), every WARP owns a contiguous range of warp slices and a private ring of NS TMA stages:
//     one stage = the slice's compact Jacobian [NJ][32] (+ residuals [2][32]) + its camera / point index rows, fetched by
//     three or four cp.async.bulk copies that complete on the stage's mbarrier.  Slices i+1 .. i+NS-1 are in flight
//     while slice i is processed; the warp re-arms a stage as soon as it has consumed it (no block barrier anywhere);
//   * the camera-side gathers (x block of the observing camera, h and M_p of the point) of slice i+1 are issued BEFORE the
//     arithmetic of slice i and consumed one iteration later (software pipelining through registers);
//   * per-point sums by ballot-driven segmented shuffle reduction; camera-side sums staged in the consumed stage and emitted
//     element-major (warp_red_rows); sums shared by every observation (shared intrinsics, model cost change) are kept in
//     registers across the whole range and leave the warp once, at the end.
__device__ __forceinline__ int run_last_lane_dev(unsigned heads, int lane) {
#ifdef TBA_EMULATE
  return run_last_lane(heads, lane);
#else
  const unsigned above = lane >= 31 ? 0u : (heads & ~((2u << lane) - 1u));
  return above == 0u ? 31 : __ffs(above) - 2;
#endif
}

// element-major emission of staged [32][N] rows whose N elements go to the (non-contiguous) columns of IMASK
template <uint32_t IMASK, int N>
__device__ __forceinline__ void warp_red_rows_cols(double* __restrict__ dst, const double* __restrict__ stage, const int* __restrict__ sbase, int lane) {
#pragma unroll
  for (int k = 0; k < N; ++k) {
    const int e = k * 32 + lane;
    const int o = e / N, j = e - o * N;
    const int b = sbase[o];
    int col = 0;
#pragma unroll
    for (int q = 0; q < N; ++q) if (q == j) col = nth_bit(IMASK, q);
    if (b >= 0) red_add(dst + (size_t)b + col, stage[e]);
  }
}

template <uint32_t IMASK, int MODE>
struct StreamCfg {
  static constexpr int NI = popcount10(IMASK);
  static constexpr int NJ = 14 + 2 * NI;
  static constexpr int STG = NJ * 32 + (MODE != 0 ? 64 : 0) + 32;  // doubles per stage: J | [res] | cam ids (32 int) + point ids (32 int)
  static constexpr int NS = 3;                                      // ring depth
  // warps per CTA: what fits 220 KB of dynamic shared memory with NS stages, at most 12 (384 threads leave 168 registers per
  // thread: the software-pipelined gathers of the next slice live in registers next to the current slice's)
  static constexpr int NW = (220 * 1024 / (NS * STG * 8)) > 12 ? 12 : (220 * 1024 / (NS * STG * 8));
  static constexpr size_t SMEM = (size_t)NW * NS * STG * 8 + (size_t)NW * NS * 8;
};

template <uint32_t IMASK, int MODE>
__global__ void __launch_bounds__(StreamCfg<IMASK, MODE>::NW * 32, 1)
k_schur_stream(DevProblem P, const double* __restrict__ xs, double* __restrict__ y, double* __restrict__ rep,
               const int* __restrict__ done_flag, int n_slices, P2pDev pp) {
  using Cfg = StreamCfg<IMASK, MODE>;
  constexpr int NI = Cfg::NI, NJ = Cfg::NJ, STG = Cfg::STG, NS = Cfg::NS, NW = Cfg::NW;
  if (done_flag != nullptr && *done_flag) return;
#ifdef TBA_EMULATE
  double* s_dyn = emu::dyn_smem<double>();
#else
  extern __shared__ __align__(128) double s_dyn[];
#endif
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gw = blockIdx.x * NW + warp, GW = gridDim.x * NW;
  const int s_begin = (int)((long long)n_slices * gw / GW), s_end = (int)((long long)n_slices * (gw + 1) / GW);
  const bool active = s_begin < s_end;  // warp-uniform; idle warps fall through to the end (the multi-GPU epilogue has block barriers)
  double* ring = s_dyn + (size_t)warp * NS * STG;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_dyn + (size_t)NW * NS * STG) + warp * NS;
  constexpr uint32_t jbytes = NJ * 32 * 8, rbytes = (MODE != 0) ? 2 * 32 * 8 : 0;
  auto issue = [&](int stage, int slice) {  // lane 0 only
    double* st = ring + (size_t)stage * STG;
    mbar_expect_tx(&bars[stage], jbytes + rbytes + 256);
    bulk_g2s(st, P.J + (size_t)slice * NJ * 32, jbytes, &bars[stage]);
    if (MODE != 0) bulk_g2s(st + NJ * 32, P.res + (size_t)slice * 64, rbytes, &bars[stage]);
    int* idx = reinterpret_cast<int*>(st + NJ * 32 + (MODE != 0 ? 64 : 0));
    bulk_g2s(idx, P.slot_cam + (size_t)slice * 32, 128, &bars[stage]);
    bulk_g2s(idx + 32, P.slot_pt + (size_t)slice * 32, 128, &bars[stage]);
  };
  if (lane == 0 && active) {
#pragma unroll
    for (int k = 0; k < NS; ++k) mbar_init(&bars[k], 1);
#pragma unroll
    for (int k = 0; k < NS; ++k) if (s_begin + k < s_end) issue(k, s_begin + k);
  }
  __syncwarp();
  // intrinsics x of the single shared group: one uniform load for the whole kernel
  double xi_u[NI + 1];
  if (NI > 0 && MODE != 1 && P.single_group) {
#pragma unroll
    for (int j = 0; j < NI; ++j) xi_u[j] = __ldg(xs + P.ne + nth_bit(IMASK, j));
  }
  double yi_acc[NI + 1];  // shared-intrinsics sums of this lane over the whole range
#pragma unroll
  for (int j = 0; j < NI; ++j) yi_acc[j] = 0.0;
  double mcc_acc = 0.0;
  // ---- registers of the slice being prefetched ("n" = next)
  int cam_n = -1, pt_n = 0, grp_n = 0;
  unsigned heads_n = 0xffffffffu;
  double2 xa_n = make_double2(0.0, 0.0), xb_n = xa_n, xc_n = xa_n;
  double xi_n[NI + 1];
  double h_n = 0.0;
  double2 m01_n = xa_n, m23_n = xa_n, m45_n = xa_n, m67_n = xa_n, m89_n = xa_n;
  uint8_t flag_n = 0;
  auto prefetch = [&](int slice, int it) {
    const int stage = it % NS;
    mbar_wait(&bars[stage], (uint32_t)((it / NS) & 1));
    const int* idx = reinterpret_cast<const int*>(ring + (size_t)stage * STG + NJ * 32 + (MODE != 0 ? 64 : 0));
    cam_n = idx[lane];
    pt_n = idx[32 + lane];
    const bool valid = cam_n >= 0;
    const int key = valid ? pt_n : -1 - lane;
    const int prev = __shfl_up_sync(0xffffffffu, key, 1);
    const bool head = lane == 0 || prev != key;
    heads_n = __ballot_sync(0xffffffffu, head);
    if (valid) {
      h_n = __ldg(P.pt + (size_t)pt_n * 4 + 3);
      if (MODE != 1) {
        const double2* x2 = reinterpret_cast<const double2*>(xs + (size_t)((MODE == 0 && (P.ablate & 2)) ? lane : cam_n) * 6);
        xa_n = __ldg(x2); xb_n = __ldg(x2 + 1); xc_n = __ldg(x2 + 2);
      }
      if (NI > 0 && !P.single_group) {
        grp_n = __ldg(P.cam_group + cam_n);
        if (MODE != 1) {
          const double* xg = xs + P.ne + (size_t)grp_n * 10;
#pragma unroll
          for (int j = 0; j < NI; ++j) xi_n[j] = __ldg(xg + nth_bit(IMASK, j));
        }
      }
      if (head) {
        const double2* M2 = reinterpret_cast<const double2*>(P.Mp + (size_t)pt_n * 10);
        m01_n = __ldg(M2); m23_n = __ldg(M2 + 1); m45_n = __ldg(M2 + 2); m67_n = __ldg(M2 + 3); m89_n = __ldg(M2 + 4);
      }
      if (MODE == 2) flag_n = P.slot_flags[(size_t)slice * 32 + lane];
    }
  };
  if (active) prefetch(s_begin, 0);
  for (int s = s_begin, it = 0; s < s_end; ++s, ++it) {
    // ---- take over the prefetched registers, start the prefetch of the next slice
    const int cam = cam_n, pt = pt_n, grp = grp_n;
    const unsigned heads = heads_n;
    const double2 xa = xa_n, xb = xb_n, xc = xc_n, m01 = m01_n, m23 = m23_n, m45 = m45_n, m67 = m67_n, m89 = m89_n;
    const double h = h_n;
    const uint8_t flag = flag_n;
    double xi[NI + 1];
#pragma unroll
    for (int j = 0; j < NI; ++j) xi[j] = (NI > 0 && MODE != 1) ? (P.single_group ? xi_u[j] : xi_n[j]) : 0.0;
    const bool valid = cam >= 0;
    if (s + 1 < s_end) prefetch(s + 1, it + 1);
    // ---- slice s: its stage landed (waited for by its prefetch)
    const int stage = it % NS;
    double* sJ = ring + (size_t)stage * STG;
    const double* sR = sJ + NJ * 32;
    const double* Jt = sJ + lane;
#define JA(j) Jt[(j) * 32]
#define JW(j) Jt[(6 + (j)) * 32]
#define JH(j) Jt[(12 + (j)) * 32]
#define JI(j) Jt[(14 + (j)) * 32]
    double w0 = 0.0, w1 = 0.0, r0 = 0.0, r1 = 0.0;
    // the point rows of this lane in registers (each is used by both products); the camera rows are read where they are used
    double ja[6], jh[2];
#pragma unroll
    for (int j = 0; j < 6; ++j) ja[j] = JA(j);
    jh[0] = JH(0); jh[1] = JH(1);
    if (valid) {
      if (MODE != 0) { r0 = sR[lane]; r1 = sR[32 + lane]; }
      if (MODE != 1) {
        w0 = -h * (ja[0] * xa.x + ja[1] * xa.y + ja[2] * xb.x) + JW(0) * xb.y + JW(1) * xc.x + JW(2) * xc.y;
        w1 = -h * (ja[3] * xa.x + ja[4] * xa.y + ja[5] * xb.x) + JW(3) * xb.y + JW(4) * xc.x + JW(5) * xc.y;
#pragma unroll
        for (int j = 0; j < NI; ++j) { w0 += JI(j) * xi[j]; w1 += JI(NI + j) * xi[j]; }
      }
      if (MODE == 1) { w0 = r0; w1 = r1; }
      if (MODE == 2) { w0 = r0 - w0; w1 = r1 - w1; }
    }
    double t[4] = {0.0, 0.0, 0.0, 0.0};
    if (valid) {
      t[0] = ja[0] * w0 + ja[3] * w1; t[1] = ja[1] * w0 + ja[4] * w1; t[2] = ja[2] * w0 + ja[5] * w1;
      t[3] = jh[0] * w0 + jh[1] * w1;
    }
    if (!(MODE == 0 && (P.ablate & 8))) {
      const int last = run_last_lane_dev(heads, lane);
#pragma unroll
      for (int j = 0; j < 4; ++j) t[j] = seg_reduce_to(t[j], last, lane);
    }
    double u0 = m01.x * t[0] + m01.y * t[1] + m23.x * t[2] + m23.y * t[3];
    double u1 = m01.y * t[0] + m45.x * t[1] + m45.y * t[2] + m67.x * t[3];
    double u2 = m23.x * t[0] + m45.y * t[1] + m67.y * t[2] + m89.x * t[3];
    double u3 = m23.y * t[0] + m67.x * t[1] + m89.x * t[2] + m89.y * t[3];
    const bool head = (heads >> lane) & 1u;
    if (MODE == 2 && head && valid) {
      double2* d = reinterpret_cast<double2*>(P.dpt + (size_t)pt * 4);
      d[0] = make_double2(-u0, -u1);
      d[1] = make_double2(-u2, -u3);
    }
    const int hl = run_head_lane(heads, lane);
    u0 = __shfl_sync(0xffffffffu, u0, hl); u1 = __shfl_sync(0xffffffffu, u1, hl);
    u2 = __shfl_sync(0xffffffffu, u2, hl); u3 = __shfl_sync(0xffffffffu, u3, hl);
    double z0 = 0.0, z1 = 0.0;
    if (valid) {
      z0 = w0 - (ja[0] * u0 + ja[1] * u1 + ja[2] * u2 + jh[0] * u3);
      z1 = w1 - (ja[3] * u0 + ja[4] * u1 + ja[5] * u2 + jh[1] * u3);
    }
    if (MODE == 2) {
      // model residual m = J * step = -(F xs + E u) = -(r - z); contribution -m.(r + m/2)
      if (valid && !(flag & 1)) {
        const double m0 = -(r0 - z0), m1 = -(r1 - z1);
        mcc_acc += -(m0 * (r0 + 0.5 * m0) + m1 * (r1 + 0.5 * m1));
      }
    } else {
      double yv[6];
#pragma unroll
      for (int j = 0; j < 3; ++j) yv[j] = valid ? -h * (ja[j] * z0 + ja[3 + j] * z1) : 0.0;
#pragma unroll
      for (int j = 0; j < 3; ++j) yv[3 + j] = valid ? JW(j) * z0 + JW(3 + j) * z1 : 0.0;
      double yi[NI + 1];
#pragma unroll
      for (int j = 0; j < NI; ++j) yi[j] = valid ? JI(j) * z0 + JI(NI + j) * z1 : 0.0;
      __syncwarp();  // every lane has finished reading the J slice: its first rows are reused as staging [32][6] + 32 ints
      int* sbase = reinterpret_cast<int*>(sJ + 32 * 6);
      warp_stage_row<6>(sJ, sbase, yv, valid ? cam * 6 : -1, lane);
      __syncwarp();
      if (!(MODE == 0 && (P.ablate & 1))) warp_red_rows<6>(y, sJ, sbase, lane);
      if (NI > 0) {
        if (P.single_group) {
#pragma unroll
          for (int j = 0; j < NI; ++j) yi_acc[j] += yi[j];
        } else {
          // per-group intrinsics rows: staged behind the extrinsics rows ([32][NI] doubles + 32 ints) and emitted element-major
          static_assert(32 * 6 + 16 + 32 * NI + 16 <= NJ * 32, "stage too small for the intrinsics staging");
          double* si = sJ + 32 * 6 + 16;
          int* sibase = reinterpret_cast<int*>(si + 32 * NI);
          __syncwarp();
#pragma unroll
          for (int j = 0; j < NI; ++j) si[lane * NI + j] = yi[j];
          sibase[lane] = valid ? P.ne + grp * 10 : -1;
          __syncwarp();
          if (!(MODE == 0 && (P.ablate & 1))) warp_red_rows_cols<IMASK, (NI > 0 ? NI : 1)>(y, si, sibase, lane);
        }
      }
    }
#undef JA
#undef JW
#undef JH
#undef JI
    // ---- the stage is consumed: re-arm it for slice s + NS
    __syncwarp();
    if (lane == 0 && s + NS < s_end) {
      fence_proxy_async_smem();  // generic-proxy accesses of the stage (reads, staging stores) before the async-proxy refill
      issue(stage, s + NS);
    }
  }
  // ---- sums that leave the warp once
  double* rr = rep + (size_t)(gw & (NREP - 1)) * REPW;
  if (!active) {
  } else if (MODE == 2) {
    const double m = warp_sum(mcc_acc);
    if (lane == 0) red_add(rr + 23, m);
  } else if (NI > 0 && P.single_group) {
#pragma unroll
    for (int j = 0; j < NI; ++j) {
      const double v = warp_sum(yi_acc[j]);
      if (lane == 0) red_add(rr + nth_bit(IMASK, j), v);
    }
  }
  // ---- multi-GPU: grid barrier (the persistent CTAs are co-resident: one per SM), then EVERY CTA stores its slice of the
  // rank's complete partial y into slot `rank` of every peer's inbox; the CTA that finishes its stores last releases the flags
  if (MODE == 0 && pp.world > 1) {
    __shared__ int s_last;
    __threadfence();  // this thread's REDs are performed before its CTA is counted
    __syncthreads();
    if (threadIdx.x == 0) {
      atomicAdd(pp.ctr, 1);
#ifndef TBA_EMULATE
      const long long t0 = clock64();
      while (atomicAdd(pp.ctr, 0) < (int)gridDim.x) {
        if (clock64() - t0 > 4000000000ll) { printf("tba: grid barrier of the matvec timed out (block %d)\n", (int)blockIdx.x); __trap(); }
      }
#endif
    }
    __syncthreads();
    __threadfence();
    const size_t slot = ((size_t)(pp.seq & 1ull) * pp.world + pp.rank) * pp.cap;
    const bool fold = NI > 0 && P.single_group;
    if (fold && blockIdx.x == 0 && threadIdx.x < 10) {  // k_fold: replica columns 0..9 -> y[ne ..] (and to the peers), replicas re-zeroed
      double v = ld_cg(y + P.ne + threadIdx.x);
      for (int r = 0; r < NREP; ++r) { v += ld_cg(rep + (size_t)r * REPW + threadIdx.x); rep[(size_t)r * REPW + threadIdx.x] = 0.0; }
      y[P.ne + threadIdx.x] = v;
      for (int q = 0; q < pp.world; ++q) pp.inbox[q][slot + P.ne + threadIdx.x] = v;
    }
    // 16-byte stores of the extrinsics part (ne is even) and, with per-camera groups, of the intrinsics part
    const int n_push = fold ? P.ne : P.ncs;
    const int n2 = (n_push + 1) / 2;
    const int per = (n2 + (int)gridDim.x - 1) / (int)gridDim.x;
    const int i0 = (int)blockIdx.x * per, i1 = (i0 + per < n2) ? i0 + per : n2;
    for (int i = i0 + (int)threadIdx.x; i < i1; i += (int)blockDim.x) {
      const double a = ld_cg(y + 2 * i), b = 2 * i + 1 < n_push ? ld_cg(y + 2 * i + 1) : 0.0;
      for (int q = 0; q < pp.world; ++q) reinterpret_cast<double2*>(pp.inbox[q] + slot)[i] = make_double2(a, b);
    }
    // one system-scope fence per CTA, by the thread that counts the CTA in: the stores of the other threads happen before it
    // through the block barrier (fences are cumulative)
    __syncthreads();
    if (threadIdx.x == 0) { __threadfence_system(); s_last = atomicAdd(pp.ctr + 1, 1) == (int)gridDim.x - 1; }
    __syncthreads();
    if (s_last) {
      __threadfence_system();
      if ((int)threadIdx.x < pp.world) st_release_sys(pp.flags[threadIdx.x] + pp.rank, pp.seq);
    }
  }
}

// --------------------------------------------- K2p: everything the LM iteration needs from J besides the matvec, in ONE pass
// Fuses, over the normal tiles and with the streaming structure of k_schur_stream (per-warp TMA ring, pipelined gathers):
//   * the reduced right-hand side  y += F^T (I - E M E^T) r                          (k_schur MODE 1),
//   * the SCHUR_JACOBI extrinsics blocks  Sc[cam] += J_c^T Q_o J_c,  Q_o = I_2 - J_p M_p J_p^T   (k_precond_ext),
//   * the SCHUR_JACOBI intrinsics blocks  Si[g] += sum_o J_i^T J_i - sum_(p,g) W^T M_p W,  W = sum_{o in p and g} J_p^T J_i
//     (k_precond_intr; the per-(point, group) sums W by ballot-driven segmented shuffle reduction instead of shared-memory
//     atomics; with one shared group every lane keeps its share of Si in registers until the end of its range).
// Three sweeps over the 3.2 GB linearisation (5.7 ms at 20 M observations in round 1) become one.
// Long tiles keep the three tile kernels (engine: stage_prepare).
template <uint32_t IMASK>
struct PrepCfg {
  static constexpr int NI = popcount10(IMASK);
  static constexpr int NJ = 14 + 2 * NI;
  static constexpr int NSI = NI * (NI + 1) / 2;
  static constexpr int STG = NJ * 32 + 64 + 32;
  static constexpr int NS = 3;
  static constexpr int NWMAX = NI <= 4 ? 10 : 6;  // register budget: NI <= 4: 192 registers per thread, else 255
  static constexpr int NW = (216 * 1024 / (NS * STG * 8)) > NWMAX ? NWMAX : (216 * 1024 / (NS * STG * 8));
  static constexpr size_t SMEM = (size_t)NW * NS * STG * 8 + (size_t)NW * NS * 8 + (size_t)NW * (NSI + 1) * 8;
};

template <uint32_t IMASK>
__global__ void __launch_bounds__(PrepCfg<IMASK>::NW * 32, 1)
k_prepare_stream(DevProblem P, double* __restrict__ y, double* __restrict__ Sc, double* __restrict__ Si, double* __restrict__ rep, int n_slices) {
  using Cfg = PrepCfg<IMASK>;
  constexpr int NI = Cfg::NI, NJ = Cfg::NJ, STG = Cfg::STG, NS = Cfg::NS, NW = Cfg::NW, NSI = Cfg::NSI;
#ifdef TBA_EMULATE
  double* s_dyn = emu::dyn_smem<double>();
#else
  extern __shared__ __align__(128) double s_dyn[];
#endif
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gw = blockIdx.x * NW + warp, GW = gridDim.x * NW;
  const int s_begin = (int)((long long)n_slices * gw / GW), s_end = (int)((long long)n_slices * (gw + 1) / GW);
  double* ring = s_dyn + (size_t)warp * NS * STG;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_dyn + (size_t)NW * NS * STG) + warp * NS;
  double* s_si = s_dyn + (size_t)NW * NS * STG + (size_t)NW * NS;  // [NW][NSI + 1] end-of-kernel partials of the shared-group block
  constexpr uint32_t jbytes = NJ * 32 * 8, rbytes = 2 * 32 * 8;
  auto issue = [&](int stage, int slice) {  // lane 0 only
    double* st = ring + (size_t)stage * STG;
    mbar_expect_tx(&bars[stage], jbytes + rbytes + 256);
    bulk_g2s(st, P.J + (size_t)slice * NJ * 32, jbytes, &bars[stage]);
    bulk_g2s(st + NJ * 32, P.res + (size_t)slice * 64, rbytes, &bars[stage]);
    int* idx = reinterpret_cast<int*>(st + NJ * 32 + 64);
    bulk_g2s(idx, P.slot_cam + (size_t)slice * 32, 128, &bars[stage]);
    bulk_g2s(idx + 32, P.slot_pt + (size_t)slice * 32, 128, &bars[stage]);
  };
  if (lane == 0 && s_begin < s_end) {
#pragma unroll
    for (int k = 0; k < NS; ++k) mbar_init(&bars[k], 1);
#pragma unroll
    for (int k = 0; k < NS; ++k) if (s_begin + k < s_end) issue(k, s_begin + k);
  }
  __syncwarp();
  double yi_acc[NI + 1], si_acc[NSI + 1];
#pragma unroll
  for (int j = 0; j < NI; ++j) yi_acc[j] = 0.0;
#pragma unroll
  for (int j = 0; j < NSI; ++j) si_acc[j] = 0.0;
  // ---- registers of the slice being prefetched
  int cam_n = -1, pt_n = 0, grp_n = 0;
  unsigned heads_n = 0xffffffffu, rheads_n = 0xffffffffu;
  double h_n = 0.0;
  double2 m01_n = make_double2(0.0, 0.0), m23_n = m01_n, m45_n = m01_n, m67_n = m01_n, m89_n = m01_n;
  auto prefetch = [&](int it) {
    const int stage = it % NS;
    mbar_wait(&bars[stage], (uint32_t)((it / NS) & 1));
    const int* idx = reinterpret_cast<const int*>(ring + (size_t)stage * STG + NJ * 32 + 64);
    cam_n = idx[lane];
    pt_n = idx[32 + lane];
    const bool valid = cam_n >= 0;
    grp_n = 0;
    if (valid && NI > 0 && !P.single_group) grp_n = __ldg(P.cam_group + cam_n);
    const int key = valid ? pt_n : -1 - lane;
    const int prev = __shfl_up_sync(0xffffffffu, key, 1);
    const int prevg = __shfl_up_sync(0xffffffffu, grp_n, 1);
    const bool head = lane == 0 || prev != key;
    heads_n = __ballot_sync(0xffffffffu, head);
    rheads_n = __ballot_sync(0xffffffffu, head || prevg != grp_n);  // (point, group) runs
    if (valid) {
      h_n = __ldg(P.pt + (size_t)pt_n * 4 + 3);
      const double2* M2 = reinterpret_cast<const double2*>(P.Mp + (size_t)pt_n * 10);  // every lane: Q_o needs M_p
      m01_n = __ldg(M2); m23_n = __ldg(M2 + 1); m45_n = __ldg(M2 + 2); m67_n = __ldg(M2 + 3); m89_n = __ldg(M2 + 4);
    }
  };
  if (s_begin < s_end) prefetch(0);
  for (int s = s_begin, it = 0; s < s_end; ++s, ++it) {
    const int cam = cam_n, grp = grp_n;
    const unsigned heads = heads_n, rheads = rheads_n;
    const double M[10] = {m01_n.x, m01_n.y, m23_n.x, m23_n.y, m45_n.x, m45_n.y, m67_n.x, m67_n.y, m89_n.x, m89_n.y};
    const double h = h_n;
    const bool valid = cam >= 0;
    if (s + 1 < s_end) prefetch(it + 1);
    const int stage = it % NS;
    double* sJ = ring + (size_t)stage * STG;
    const double* sR = sJ + NJ * 32;
    const double* Jt = sJ + lane;
    double ja[6], jh[2], jw[6], ji[2 * NI + 1];
#pragma unroll
    for (int j = 0; j < 6; ++j) { ja[j] = Jt[j * 32]; jw[j] = Jt[(6 + j) * 32]; }
    jh[0] = Jt[12 * 32]; jh[1] = Jt[13 * 32];
#pragma unroll
    for (int j = 0; j < 2 * NI; ++j) ji[j] = Jt[(14 + j) * 32];
    double r0 = 0.0, r1 = 0.0;
    if (valid) { r0 = sR[lane]; r1 = sR[32 + lane]; }
    if (!valid) {
#pragma unroll
      for (int j = 0; j < 6; ++j) { ja[j] = 0.0; jw[j] = 0.0; }
      jh[0] = jh[1] = 0.0;
#pragma unroll
      for (int j = 0; j < 2 * NI; ++j) ji[j] = 0.0;
    }
    __syncwarp();  // every lane holds its rows: the stage is free for staging from here on
    const int last = run_last_lane_dev(heads, lane);
    const int hl = run_head_lane(heads, lane);
    // ---------------- reduced rhs (MODE 1 of k_schur): w = r
    {
      double t[4] = {ja[0] * r0 + ja[3] * r1, ja[1] * r0 + ja[4] * r1, ja[2] * r0 + ja[5] * r1, jh[0] * r0 + jh[1] * r1};
#pragma unroll
      for (int j = 0; j < 4; ++j) t[j] = seg_reduce_to(t[j], last, lane);
      double u[4];
      sym4_mul(M, t, u);
#pragma unroll
      for (int j = 0; j < 4; ++j) u[j] = __shfl_sync(0xffffffffu, u[j], hl);
      const double z0 = r0 - (ja[0] * u[0] + ja[1] * u[1] + ja[2] * u[2] + jh[0] * u[3]);
      const double z1 = r1 - (ja[3] * u[0] + ja[4] * u[1] + ja[5] * u[2] + jh[1] * u[3]);
      double yv[6];
#pragma unroll
      for (int j = 0; j < 3; ++j) { yv[j] = -h * (ja[j] * z0 + ja[3 + j] * z1); yv[3 + j] = jw[j] * z0 + jw[3 + j] * z1; }
      int* sbase = reinterpret_cast<int*>(sJ + 32 * 6);
      warp_stage_row<6>(sJ, sbase, yv, valid ? cam * 6 : -1, lane);
      __syncwarp();
      warp_red_rows<6>(y, sJ, sbase, lane);
      if (NI > 0) {
        if (P.single_group) {
#pragma unroll
          for (int j = 0; j < NI; ++j) yi_acc[j] += ji[j] * z0 + ji[NI + j] * z1;
        } else if (valid) {
#pragma unroll
          for (int j = 0; j < NI; ++j) red_add(y + P.ne + (size_t)grp * 10 + nth_bit(IMASK, j), ji[j] * z0 + ji[NI + j] * z1);
        }
      }
      __syncwarp();
    }
    // ---------------- extrinsics blocks: 21 entries per observation, staged and emitted in three groups of seven columns
    {
      const double jp0[4] = {ja[0], ja[1], ja[2], jh[0]}, jp1[4] = {ja[3], ja[4], ja[5], jh[1]};
      double m0[4], m1[4];
      sym4_mul(M, jp0, m0);
      sym4_mul(M, jp1, m1);
      const double q00 = 1.0 - (jp0[0] * m0[0] + jp0[1] * m0[1] + jp0[2] * m0[2] + jp0[3] * m0[3]);
      const double q01 = -(jp0[0] * m1[0] + jp0[1] * m1[1] + jp0[2] * m1[2] + jp0[3] * m1[3]);
      const double q11 = 1.0 - (jp1[0] * m1[0] + jp1[1] * m1[1] + jp1[2] * m1[2] + jp1[3] * m1[3]);
      double c0[6], c1[6];
#pragma unroll
      for (int j = 0; j < 3; ++j) { c0[j] = -h * ja[j]; c1[j] = -h * ja[3 + j]; c0[3 + j] = jw[j]; c1[3 + j] = jw[3 + j]; }
      double v[21];
      int n = 0;
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        const double qa0 = q00 * c0[a] + q01 * c1[a], qa1 = q01 * c0[a] + q11 * c1[a];
#pragma unroll
        for (int b = a; b < 6; ++b) { v[n] = qa0 * c0[b] + qa1 * c1[b]; ++n; }
      }
      int* sbase = reinterpret_cast<int*>(sJ + 32 * 7);
#pragma unroll
      for (int g3 = 0; g3 < 3; ++g3) {
        const double vv[7] = {v[7 * g3], v[7 * g3 + 1], v[7 * g3 + 2], v[7 * g3 + 3], v[7 * g3 + 4], v[7 * g3 + 5], v[7 * g3 + 6]};
        warp_stage_row<7>(sJ, sbase, vv, valid ? cam * 21 + 7 * g3 : -1, lane);
        __syncwarp();
        warp_red_rows<7>(Sc, sJ, sbase, lane);
        __syncwarp();
      }
    }
    // ---------------- intrinsics blocks
    if (NI > 0) {
      // W = sum over the (point, group) run of J_p^T J_i  (4 x NI), on the run's head lane
      const int rlast = run_last_lane_dev(rheads, lane);
      const bool rhead = (rheads >> lane) & 1u;
      double W[4 * NI + 1];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const double p0 = a < 3 ? ja[a] : jh[0], p1 = a < 3 ? ja[3 + a] : jh[1];
#pragma unroll
        for (int j = 0; j < NI; ++j) W[a * NI + j] = seg_reduce_to(p0 * ji[j] + p1 * ji[NI + j], rlast, lane);
      }
      double sub[NSI + 1];
#pragma unroll
      for (int j = 0; j < NSI; ++j) sub[j] = 0.0;
      if (rhead && valid) {
        double MW[4][NI + 1];
#pragma unroll
        for (int j = 0; j < NI; ++j) {
          const double t4[4] = {W[0 * NI + j], W[1 * NI + j], W[2 * NI + j], W[3 * NI + j]};
          double u4[4];
          sym4_mul(M, t4, u4);
          MW[0][j] = u4[0]; MW[1][j] = u4[1]; MW[2][j] = u4[2]; MW[3][j] = u4[3];
        }
        int n = 0;
#pragma unroll
        for (int a = 0; a < NI; ++a)
#pragma unroll
          for (int b = a; b < NI; ++b) {
            sub[n] = W[0 * NI + a] * MW[0][b] + W[1 * NI + a] * MW[1][b] + W[2 * NI + a] * MW[2][b] + W[3 * NI + a] * MW[3][b];
            ++n;
          }
      }
      int n = 0;
#pragma unroll
      for (int a = 0; a < NI; ++a)
#pragma unroll
        for (int b = a; b < NI; ++b) {
          const double acc = ji[a] * ji[b] + ji[NI + a] * ji[NI + b];  // 0 on padding lanes
          if (P.single_group) si_acc[n] += acc - sub[n];
          else if (valid) {
            const int ia = nth_bit(IMASK, a), ib = nth_bit(IMASK, b);
            const int idx = ia * 10 - ia * (ia - 1) / 2 + (ib - ia);
            red_add(Si + (size_t)grp * 55 + idx, acc - sub[n]);
          }
          ++n;
        }
    }
    __syncwarp();
    if (lane == 0 && s + NS < s_end) {
      fence_proxy_async_smem();
      issue(stage, s + NS);
    }
  }
  // ---- sums that leave the warp once
  if (NI > 0 && P.single_group) {
    double* rr = rep + (size_t)(gw & (NREP - 1)) * REPW;
#pragma unroll
    for (int j = 0; j < NI; ++j) {
      const double vsum = warp_sum(yi_acc[j]);
      if (lane == 0) red_add(rr + nth_bit(IMASK, j), vsum);
    }
#pragma unroll
    for (int j = 0; j < NSI; ++j) {
      const double vsum = warp_sum(si_acc[j]);
      if (lane == 0) s_si[warp * (NSI + 1) + j] = vsum;
    }
    __syncthreads();  // the only block barrier of the kernel: every thread reaches it (no early exit above)
    if ((int)threadIdx.x < NSI) {
      double vsum = 0.0;
      for (int w = 0; w < NW; ++w) vsum += s_si[w * (NSI + 1) + threadIdx.x];
      // position of entry n in the 10x10 upper triangle
      int n = 0, idx = 0;
      for (int a = 0; a < NI; ++a)
        for (int b = a; b < NI; ++b) {
          if (n == (int)threadIdx.x) { const int ia = nth_bit(IMASK, a), ib = nth_bit(IMASK, b); idx = ia * 10 - ia * (ia - 1) / 2 + (ib - ia); }
          ++n;
        }
      red_add(Si + idx, vsum);
    }
  }
}

// ------------------------------------------- SCHUR_JACOBI preconditioner blocks
// Extrinsics blocks: S_cc = sum_o J_c^T Q_o J_c with Q_o = I_2 - J_p M_p J_p^T (a view observes a track once).
// Sc: [n_cam][21] upper triangle, unscaled (scaling + D^2 + inversion in k_precond_finish).
template <uint32_t IMASK, bool TRED = false>
__global__ void __launch_bounds__(TILE) k_precond_ext(DevProblem P, double* __restrict__ Sc, int tile0) {
  constexpr int NI = popcount10(IMASK);
  constexpr int NJ = 14 + 2 * NI;
  const int tile = tile0 + blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t slot = (size_t)tile * TILE + tid;
  const int cam = P.slot_cam[slot];
  if (TRED) {
    // transposed RED emission: the 21 block entries of every observation staged per warp, emitted element-major
    __shared__ double s_stage[TILE / 32][32 * 21];
    __shared__ int s_base[TILE / 32][32];
    double v[21];
#pragma unroll
    for (int j = 0; j < 21; ++j) v[j] = 0.0;
    if (cam >= 0) {
      const double* Jt = P.J + wslice(tile, warp, NJ) + lane;
      double Ja[6], Jw[6], Jh[2];
#pragma unroll
      for (int j = 0; j < 6; ++j) Ja[j] = Jt[j * 32];
#pragma unroll
      for (int j = 0; j < 6; ++j) Jw[j] = Jt[(6 + j) * 32];
      Jh[0] = Jt[12 * 32];
      Jh[1] = Jt[13 * 32];
      const int pt = P.slot_pt[slot];
      const double h = P.pt[(size_t)pt * 4 + 3];
      const double* M = P.Mp + (size_t)pt * 10;
      const double jp0[4] = {Ja[0], Ja[1], Ja[2], Jh[0]}, jp1[4] = {Ja[3], Ja[4], Ja[5], Jh[1]};
      double m0[4], m1[4];
      sym4_mul(M, jp0, m0);
      sym4_mul(M, jp1, m1);
      const double q00 = 1.0 - (jp0[0] * m0[0] + jp0[1] * m0[1] + jp0[2] * m0[2] + jp0[3] * m0[3]);
      const double q01 = -(jp0[0] * m1[0] + jp0[1] * m1[1] + jp0[2] * m1[2] + jp0[3] * m1[3]);
      const double q11 = 1.0 - (jp1[0] * m1[0] + jp1[1] * m1[1] + jp1[2] * m1[2] + jp1[3] * m1[3]);
      double c0[6], c1[6];
#pragma unroll
      for (int j = 0; j < 3; ++j) { c0[j] = -h * Ja[j]; c1[j] = -h * Ja[3 + j]; c0[3 + j] = Jw[j]; c1[3 + j] = Jw[3 + j]; }
      int n = 0;
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        const double qa0 = q00 * c0[a] + q01 * c1[a], qa1 = q01 * c0[a] + q11 * c1[a];
#pragma unroll
        for (int b = a; b < 6; ++b) { v[n] = qa0 * c0[b] + qa1 * c1[b]; ++n; }
      }
    }
    warp_stage_row<21>(s_stage[warp], s_base[warp], v, cam >= 0 ? cam * 21 : -1, lane);
    __syncwarp();
    warp_red_rows<21>(Sc, s_stage[warp], s_base[warp], lane);
    return;
  }
  if (cam < 0) return;
  const double* Jt = P.J + wslice(tile, warp, NJ) + lane;
  double Ja[6], Jw[6], Jh[2];
#pragma unroll
  for (int j = 0; j < 6; ++j) Ja[j] = Jt[j * 32];
#pragma unroll
  for (int j = 0; j < 6; ++j) Jw[j] = Jt[(6 + j) * 32];
  Jh[0] = Jt[12 * 32];
  Jh[1] = Jt[13 * 32];
  const int pt = P.slot_pt[slot];
  const double h = P.pt[(size_t)pt * 4 + 3];
  const double* M = P.Mp + (size_t)pt * 10;
  const double jp0[4] = {Ja[0], Ja[1], Ja[2], Jh[0]}, jp1[4] = {Ja[3], Ja[4], Ja[5], Jh[1]};
  double m0[4], m1[4];
  sym4_mul(M, jp0, m0);
  sym4_mul(M, jp1, m1);
  const double q00 = 1.0 - (jp0[0] * m0[0] + jp0[1] * m0[1] + jp0[2] * m0[2] + jp0[3] * m0[3]);
  const double q01 = -(jp0[0] * m1[0] + jp0[1] * m1[1] + jp0[2] * m1[2] + jp0[3] * m1[3]);
  const double q11 = 1.0 - (jp1[0] * m1[0] + jp1[1] * m1[1] + jp1[2] * m1[2] + jp1[3] * m1[3]);
  double c0[6], c1[6];
#pragma unroll
  for (int j = 0; j < 3; ++j) { c0[j] = -h * Ja[j]; c1[j] = -h * Ja[3 + j]; c0[3 + j] = Jw[j]; c1[3 + j] = Jw[3 + j]; }
  double* S = Sc + (size_t)cam * 21;
  int n = 0;
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    const double qa0 = q00 * c0[a] + q01 * c1[a], qa1 = q01 * c0[a] + q11 * c1[a];
#pragma unroll
    for (int b = a; b < 6; ++b) { red_add(S + n, qa0 * c0[b] + qa1 * c1[b]); ++n; }
  }
}

// Intrinsics blocks: S_gg = sum_o J_i^T J_i - sum_(p,g) W^T M_p W, W = sum_{o in p and g} J_p^T J_i.
// Si: [n_group][55] upper triangle over the padded 10 parameter indices.  Dynamic smem: runs x 4 x NI doubles.
template <uint32_t IMASK>
__global__ void __launch_bounds__(TILE) k_precond_intr(DevProblem P, double* __restrict__ Si, int tile0) {
  constexpr int NI = popcount10(IMASK);
  constexpr int NJ = 14 + 2 * NI;
  constexpr int NW = 4 * NI;
  constexpr int NS = NI * (NI + 1) / 2;
#ifdef TBA_EMULATE
  double* s_w = emu::dyn_smem<double>();
#else
  extern __shared__ double s_w[];  // [nruns][NW] then [nruns] group ids (as int) and points
#endif
  __shared__ double s_red[32];
  const int tile = tile0 + blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nruns = P.tile_nruns[tile];
  int* s_grp = reinterpret_cast<int*>(s_w + (size_t)TILE * NW);
  int* s_pt = s_grp + TILE;
  for (int i = tid; i < nruns * NW; i += TILE) s_w[i] = 0.0;
  __syncthreads();
  const size_t slot = (size_t)tile * TILE + tid;
  const int cam = P.slot_cam[slot];
  const bool valid = cam >= 0;
  double acc[NS + 1];
#pragma unroll
  for (int j = 0; j < NS; ++j) acc[j] = 0.0;
  int grp = 0;
  if (valid) {
    const double* Jt = P.J + wslice(tile, warp, NJ) + lane;
    double jp0[4], jp1[4], Ji[2 * NI + 1];
#pragma unroll
    for (int j = 0; j < 3; ++j) { jp0[j] = Jt[j * 32]; jp1[j] = Jt[(3 + j) * 32]; }
    jp0[3] = Jt[12 * 32];
    jp1[3] = Jt[13 * 32];
#pragma unroll
    for (int j = 0; j < 2 * NI; ++j) Ji[j] = Jt[(14 + j) * 32];
    grp = P.cam_group[cam];
    const int run = P.slot_run[slot];
    if (run >= 0) {
      s_grp[run] = grp;
      s_pt[run] = P.slot_pt[slot];
      double* W = s_w + (size_t)run * NW;
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int j = 0; j < NI; ++j) atomicAdd(W + a * NI + j, jp0[a] * Ji[j] + jp1[a] * Ji[NI + j]);
    }
    int n = 0;
#pragma unroll
    for (int a = 0; a < NI; ++a)
#pragma unroll
      for (int b = a; b < NI; ++b) { acc[n] = Ji[a] * Ji[b] + Ji[NI + a] * Ji[NI + b]; ++n; }
  }
  __syncthreads();
  // per-run Schur term, handled by thread `run`
  int rgrp = grp;
  double sub[NS + 1];
#pragma unroll
  for (int j = 0; j < NS; ++j) sub[j] = 0.0;
  const bool has_run = tid < nruns;
  if (has_run) {
    rgrp = s_grp[tid];
    const double* W = s_w + (size_t)tid * NW;
    const double* M = P.Mp + (size_t)s_pt[tid] * 10;
    double MW[4][NI + 1];
#pragma unroll
    for (int j = 0; j < NI; ++j) {
      const double t[4] = {W[0 * NI + j], W[1 * NI + j], W[2 * NI + j], W[3 * NI + j]};
      double u[4];
      sym4_mul(M, t, u);
      MW[0][j] = u[0]; MW[1][j] = u[1]; MW[2][j] = u[2]; MW[3][j] = u[3];
    }
    int n = 0;
#pragma unroll
    for (int a = 0; a < NI; ++a)
#pragma unroll
      for (int b = a; b < NI; ++b) {
        sub[n] = W[0 * NI + a] * MW[0][b] + W[1 * NI + a] * MW[1][b] + W[2 * NI + a] * MW[2][b] + W[3 * NI + a] * MW[3][b];
        ++n;
      }
  }
  // accumulate into Si at padded parameter indices
  int n = 0;
#pragma unroll
  for (int a = 0; a < NI; ++a)
#pragma unroll
    for (int b = a; b < NI; ++b) {
      const int ia = nth_bit(IMASK, a), ib = nth_bit(IMASK, b);
      const int idx = ia * 10 - ia * (ia - 1) / 2 + (ib - ia);  // upper-triangle offset in a 10x10
      if (P.single_group) {
        const double v = block_sum(acc[n] - sub[n], s_red);
        if (tid == 0) red_add(Si + idx, v);
      } else {
        if (valid) red_add(Si + (size_t)grp * 55 + idx, acc[n]);
        if (has_run) red_add(Si + (size_t)rgrp * 55 + idx, -sub[n]);
      }
      ++n;
    }
}

// In-place Cholesky inverse of an n x n SPD matrix held in registers/local (row-major, n <= 10).
template <int N>
__device__ inline bool spd_inverse_n(double* A) {
  double L[N * N], Li[N * N];
#pragma unroll
  for (int i = 0; i < N; ++i)
#pragma unroll
    for (int j = 0; j <= i; ++j) {
      double s = A[i * N + j];
      for (int k = 0; k < j; ++k) s -= L[i * N + k] * L[j * N + k];
      if (i == j) { if (!(s > 0.0)) return false; L[i * N + i] = sqrt(s); }
      else L[i * N + j] = s / L[j * N + j];
    }
  for (int i = 0; i < N * N; ++i) Li[i] = 0.0;
  for (int j = 0; j < N; ++j) {
    Li[j * N + j] = 1.0 / L[j * N + j];
    for (int i = j + 1; i < N; ++i) {
      double s = 0.0;
      for (int k = j; k < i; ++k) s -= L[i * N + k] * Li[k * N + j];
      Li[i * N + j] = s / L[i * N + i];
    }
  }
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) {
      double s = 0.0;
      for (int k = (i > j ? i : j); k < N; ++k) s += Li[k * N + i] * Li[k * N + j];
      A[i * N + j] = s;
    }
  return true;
}

// Minv_c[c] = (s S_cc s + D^2)^-1 (identity on non-free coordinates); same for groups.
__global__ void k_precond_finish(DevProblem P, const double* __restrict__ Sc, const double* __restrict__ Si,
                                 const double* __restrict__ sm, const double* __restrict__ D2, double* __restrict__ Minv_c,
                                 double* __restrict__ Minv_i, double* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P.n_cam) {
    double A[36];
    const double* S = Sc + (size_t)i * 21;
    const double* s = sm + (size_t)i * 6;
    const double* d = D2 + (size_t)i * 6;
    int n = 0;
    for (int a = 0; a < 6; ++a)
      for (int b = a; b < 6; ++b) { const double v = s[a] * S[n] * s[b]; A[a * 6 + b] = v; A[b * 6 + a] = v; ++n; }
    for (int a = 0; a < 6; ++a) { if (s[a] != 0.0) A[a * 6 + a] += d[a]; else A[a * 6 + a] = 1.0; }
    if (!spd_inverse_n<6>(A)) { atomicAdd(flag, 1.0); for (int a = 0; a < 36; ++a) A[a] = (a % 7 == 0) ? 1.0 : 0.0; }
    for (int a = 0; a < 36; ++a) Minv_c[(size_t)i * 36 + a] = A[a];
  } else if (i < P.n_cam + P.n_group) {
    const int g = i - P.n_cam;
    double A[100];
    const double* S = Si + (size_t)g * 55;
    const double* s = sm + P.ne + (size_t)g * 10;
    const double* d = D2 + P.ne + (size_t)g * 10;
    int n = 0;
    for (int a = 0; a < 10; ++a)
      for (int b = a; b < 10; ++b) { const double v = s[a] * S[n] * s[b]; A[a * 10 + b] = v; A[b * 10 + a] = v; ++n; }
    for (int a = 0; a < 10; ++a) { if (s[a] != 0.0) A[a * 10 + a] += d[a]; else A[a * 10 + a] = 1.0; }
    if (!spd_inverse_n<10>(A)) { atomicAdd(flag, 1.0); for (int a = 0; a < 100; ++a) A[a] = (a % 11 == 0) ? 1.0 : 0.0; }
    for (int a = 0; a < 100; ++a) Minv_i[(size_t)g * 100 + a] = A[a];
  }
}

// ------------------------------------------------ camera-space vector kernels
// Jacobi scale (iteration 0) and LM diagonal; gradient max-norm partial.
//   sm = mask / (1 + sqrt(cn));  D2 = clamp(sm^2 cn, lo, hi) / radius on free coordinates.
__global__ void k_cs_scale(int ncs, const double* __restrict__ cn, const double* __restrict__ mask, int use_scaling,
                           double* __restrict__ sm) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ncs; i += gridDim.x * blockDim.x)
    sm[i] = mask[i] != 0.0 ? (use_scaling ? 1.0 / (1.0 + sqrt(cn[i])) : 1.0) : 0.0;
}
__global__ void k_cs_diag(int ncs, const double* __restrict__ cn, const double* __restrict__ sm, double radius, double lo,
                          double hi, double* __restrict__ D2) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ncs; i += gridDim.x * blockDim.x)
    D2[i] = sm[i] != 0.0 ? fmin(fmax(sm[i] * sm[i] * cn[i], lo), hi) / radius : 0.0;
}

// PCG state (ping-pong between kernels; see DESIGN.md section 5.4).
struct PcgState {
  double rho, last_rho, beta, alpha, pq, Q0, Q1, norm_b2;
  int iters;        // current (1-based) iteration
  int done;
  int status;       // 0 success/converged, 1 no convergence (max iters / indefinite: x still usable), 2 failure
  int pending_q;    // a Q-test is pending (part_Q holds x.(b+r) of iteration `iters`)
  int min_iters, max_iters;
  double eta;
};

__device__ __forceinline__ double sum_partials(const double* __restrict__ part, double* s_red) {
  // every CTA sums the VB partials in the same fixed order -> identical on all CTAs and all ranks
  double v = 0.0;
  if (threadIdx.x == 0) {
    for (int i = 0; i < VB; ++i) v += part[i];
    s_red[0] = v;
  }
  __syncthreads();
  v = s_red[0];
  __syncthreads();
  return v;
}

__device__ __forceinline__ bool zero_or_inf(double x) { return x == 0.0 || isinf(x); }

// b = sm .* y_rhs ; x = 0 ; r = b ; partial |b|^2
__global__ void __launch_bounds__(VT) k_pcg_init(int ncs, const double* __restrict__ yrhs, const double* __restrict__ sm,
                                                 double* __restrict__ b, double* __restrict__ x, double* __restrict__ r,
                                                 double* __restrict__ part) {
  __shared__ double s_red[32];
  double acc = 0.0;
  for (int i = blockIdx.x * VT + threadIdx.x; i < ncs; i += VB * VT) {
    const double v = sm[i] * yrhs[i];
    b[i] = v; x[i] = 0.0; r[i] = v;
    acc += v * v;
  }
  const double s = block_sum(acc, s_red);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}
__global__ void k_pcg_init_state(PcgState* st, const double* __restrict__ part, int min_iters, int max_iters, double eta) {
  double v = 0.0;
  for (int i = 0; i < VB; ++i) v += part[i];
  PcgState s;
  s.rho = 1.0; s.last_rho = 1.0; s.beta = 0.0; s.alpha = 0.0; s.pq = 0.0; s.Q0 = 0.0; s.Q1 = 0.0; s.norm_b2 = v;
  s.iters = 1; s.done = (v == 0.0) ? 1 : 0; s.status = 0; s.pending_q = 0;
  if (v == 0.0) s.iters = 0;
  s.min_iters = min_iters; s.max_iters = max_iters; s.eta = eta;
  *st = s;
}

// q = sm .* y + D2 .* p; partial pq = p.q  (kept for tba_debug_schur_matvec)
__global__ void __launch_bounds__(VT) k_pcg_v3(int ncs, const PcgState* __restrict__ in, const double* __restrict__ y,
                                               const double* __restrict__ sm, const double* __restrict__ D2,
                                               const double* __restrict__ p, double* __restrict__ q,
                                               double* __restrict__ part_pq) {
  __shared__ double s_red[32];
  if (in->done) return;
  double acc = 0.0;
  for (int i = blockIdx.x * VT + threadIdx.x; i < ncs; i += VB * VT) {
    const double qv = sm[i] * y[i] + D2[i] * p[i];
    q[i] = qv;
    acc += p[i] * qv;
  }
  const double s = block_sum(acc, s_red);
  if (threadIdx.x == 0) part_pq[blockIdx.x] = s;
}

// ---- round 2: three vector kernels per CG iteration instead of four (plus the separate fold) -------------------------------
//   C: [Q-test of the previous iteration]; rho, beta; p = z + beta p; xs = sm .* p; y = 0        (k_pcg_c)
//      matvec
//   A: [fold of the shared-intrinsics replica rows into y]; q = sm .* y + D2 .* p; partial p.q   (k_pcg_a)
//   B: alpha = rho / pq; x += alpha p; r -= alpha q; partial x.(b + r); z = Minv r; partial r.z  (k_pcg_b, per parameter block)
// The same operations in the same order as the round-1 sequence k_pcg_v1 .. v4; the partial sums of x.(b + r) are grouped per
// parameter block now (they were grouped per element stride), i.e. equal up to fp64 summation order.

// z = Minv r for one parameter block (camera: 6, intrinsics group: 10); returns r.z
__device__ __forceinline__ double pcg_precondition_block(const DevProblem& P, int blk, const double* __restrict__ Minv_c,
                                                         const double* __restrict__ Minv_i, const double* __restrict__ r,
                                                         double* __restrict__ z, int identity_precond) {
  double acc = 0.0;
  if (blk < P.n_cam) {
    const double* M = Minv_c + (size_t)blk * 36;
    const double* rr = r + (size_t)blk * 6;
    double* zz = z + (size_t)blk * 6;
    double rv[6];
#pragma unroll
    for (int a = 0; a < 6; ++a) rv[a] = rr[a];
#pragma unroll
    for (int a = 0; a < 6; ++a) {
      double s = rv[a];
      if (!identity_precond) {
        s = 0.0;
#pragma unroll
        for (int b = 0; b < 6; ++b) s += M[a * 6 + b] * rv[b];
      }
      zz[a] = s;
      acc += rv[a] * s;
    }
  } else {
    const int g = blk - P.n_cam;
    const double* M = Minv_i + (size_t)g * 100;
    const double* rr = r + P.ne + (size_t)g * 10;
    double* zz = z + P.ne + (size_t)g * 10;
    double rv[10];
#pragma unroll
    for (int a = 0; a < 10; ++a) rv[a] = rr[a];
#pragma unroll
    for (int a = 0; a < 10; ++a) {
      double s = rv[a];
      if (!identity_precond) {
        s = 0.0;
#pragma unroll
        for (int b = 0; b < 10; ++b) s += M[a * 10 + b] * rv[b];
      }
      zz[a] = s;
      acc += rv[a] * s;
    }
  }
  return acc;
}

__device__ __forceinline__ void pcg_q_test(PcgState& st, const double* __restrict__ part_Q, double* s_red) {
  if (!st.done && st.pending_q) {
    const double Q1 = -sum_partials(part_Q, s_red);
    const double zeta = st.iters * (Q1 - st.Q0) / Q1;
    st.Q1 = Q1;
    st.pending_q = 0;
    if (zeta < st.eta && st.iters >= st.min_iters) { st.done = 1; st.status = 0; }
    else {
      st.Q0 = Q1;
      if (st.iters >= st.max_iters) { st.done = 1; st.status = 1; }
      else st.iters += 1;
    }
  }
}

// The three phases as device functions on a PcgState held in registers (every CTA computes the same state from the same partial
// sums): the kernels k_pcg_c / k_pcg_a / k_pcg_b wrap one phase each, k_pcg_fused runs them back to back with grid barriers.
__device__ __forceinline__ void pcg_phase_c(int ncs, PcgState& st, const double* __restrict__ part_Q, const double* __restrict__ part_rho,
                                            const double* __restrict__ z, const double* __restrict__ sm, double* __restrict__ p,
                                            double* __restrict__ xs, double* __restrict__ y, int* __restrict__ zero_ctr, double* s_red) {
  if (zero_ctr != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { zero_ctr[0] = 0; zero_ctr[1] = 0; }  // barrier / completion counters of the next matvec
  pcg_q_test(st, part_Q, s_red);
  if (!st.done) {
    const double rho = sum_partials(part_rho, s_red);
    st.last_rho = st.rho;
    st.rho = rho;
    if (zero_or_inf(rho)) { st.done = 1; st.status = 2; }
    else if (st.iters > 1) {
      st.beta = rho / st.last_rho;
      if (zero_or_inf(st.beta)) { st.done = 1; st.status = 2; }
    } else st.beta = 0.0;
  }
  if (st.done) return;
  const bool first = st.iters == 1;
#pragma unroll 4
  for (int i = blockIdx.x * VT + threadIdx.x; i < ncs; i += VB * VT) {  // (unrolled: the loads of four trips in flight together)
    const double pv = first ? z[i] : z[i] + st.beta * p[i];
    p[i] = pv;
    xs[i] = sm[i] * pv;
    y[i] = 0.0;
  }
}
__global__ void __launch_bounds__(VT) k_pcg_c(int ncs, const PcgState* __restrict__ in, PcgState* __restrict__ out,
                                              const double* __restrict__ part_Q, const double* __restrict__ part_rho,
                                              const double* __restrict__ z, const double* __restrict__ sm, double* __restrict__ p,
                                              double* __restrict__ xs, double* __restrict__ y, int* __restrict__ done_flag, int* __restrict__ zero_ctr) {
  __shared__ double s_red[32];
  PcgState st = *in;
  pcg_phase_c(ncs, st, part_Q, part_rho, z, sm, p, xs, y, zero_ctr, s_red);
  if (blockIdx.x == 0 && threadIdx.x == 0) { *out = st; if (done_flag) *done_flag = st.done; }
}

// fold_rep != nullptr (one GPU, one shared intrinsics group): the replica rows of the matvec are folded into y[ne ..] here,
// in the fixed row order of k_fold, by every CTA (they all need the value) -- CTA 0 stores it and re-zeroes the replicas.
__device__ __forceinline__ void pcg_phase_a(int ncs, int ne, double* __restrict__ y, const double* __restrict__ sm,
                                            const double* __restrict__ D2, const double* __restrict__ p, double* __restrict__ q,
                                            double* __restrict__ part_pq, const double* __restrict__ fold_rep, const P2pDev& pp,
                                            double* s_red, double* s_fold) {
  if (pp.world > 1) p2p_wait(pp);  // the matvec of every rank has pushed its partial sums into the local inbox
  if (fold_rep != nullptr) {
    if (threadIdx.x < 10) {
      double v = y[ne + threadIdx.x];
      for (int r = 0; r < NREP; ++r) v += fold_rep[(size_t)r * REPW + threadIdx.x];
      s_fold[threadIdx.x] = v;
    }
    __syncthreads();
  }
  double acc = 0.0;
#pragma unroll 4
  for (int i = blockIdx.x * VT + threadIdx.x; i < ncs; i += VB * VT) {
    const double yv = pp.world > 1 ? p2p_sum(pp, i) : ((fold_rep != nullptr && i >= ne && i < ne + 10) ? s_fold[i - ne] : y[i]);
    const double qv = sm[i] * yv + D2[i] * p[i];
    q[i] = qv;
    acc += p[i] * qv;
  }
  const double s = block_sum(acc, s_red);
  if (threadIdx.x == 0) part_pq[blockIdx.x] = s;
}
__global__ void __launch_bounds__(VT) k_pcg_a(int ncs, int ne, const PcgState* __restrict__ in, double* __restrict__ y,
                                              const double* __restrict__ sm, const double* __restrict__ D2,
                                              const double* __restrict__ p, double* __restrict__ q, double* __restrict__ part_pq,
                                              const double* __restrict__ fold_rep, P2pDev pp) {
  __shared__ double s_red[32];
  __shared__ double s_fold[10];
  if (in->done) return;
  pcg_phase_a(ncs, ne, y, sm, D2, p, q, part_pq, fold_rep, pp, s_red, s_fold);
}
// (the replicas are re-zeroed by the kernel that runs after every CTA of k_pcg_a has read them: k_pcg_b)

__device__ __forceinline__ void pcg_phase_b(const DevProblem& P, PcgState& st, const double* __restrict__ part_pq,
                                            const double* __restrict__ p, const double* __restrict__ q, const double* __restrict__ b,
                                            double* __restrict__ x, double* __restrict__ r, double* __restrict__ z,
                                            const double* __restrict__ Minv_c, const double* __restrict__ Minv_i,
                                            double* __restrict__ part_Q, double* __restrict__ part_rho, int identity_precond, int first,
                                            double* __restrict__ zero_rep, double* s_red) {
  if (!first && !st.done) {
    const double pq = sum_partials(part_pq, s_red);
    st.pq = pq;
    if (pq <= 0.0 || isinf(pq)) { st.done = 1; st.status = 1; }
    else {
      st.alpha = st.rho / pq;
      if (isinf(st.alpha)) { st.done = 1; st.status = 2; }
      else st.pending_q = 1;
    }
  }
  if (zero_rep != nullptr && !first) {  // the replica columns folded by phase A
    for (int i = blockIdx.x * VT + threadIdx.x; i < NREP * 10; i += VB * VT) zero_rep[(size_t)(i / 10) * REPW + (i % 10)] = 0.0;
  }
  if (st.done) return;
  double accQ = 0.0, accR = 0.0;
  const int nblk = P.n_cam + P.n_group;
  for (int blk = blockIdx.x * VT + threadIdx.x; blk < nblk; blk += VB * VT) {
    const int i0 = blk < P.n_cam ? blk * 6 : P.ne + (blk - P.n_cam) * 10, n = blk < P.n_cam ? 6 : 10;
    if (!first) {
      for (int a = 0; a < n; ++a) {
        const int i = i0 + a;
        const double xv = x[i] + st.alpha * p[i];
        const double rv = r[i] - st.alpha * q[i];
        x[i] = xv; r[i] = rv;
        accQ += xv * (b[i] + rv);
      }
    }
    accR += pcg_precondition_block(P, blk, Minv_c, Minv_i, r, z, identity_precond);
  }
  const double sQ = block_sum(accQ, s_red);
  const double sR = block_sum(accR, s_red);
  if (threadIdx.x == 0) { if (!first) part_Q[blockIdx.x] = sQ; part_rho[blockIdx.x] = sR; }
}
__global__ void __launch_bounds__(VT) k_pcg_b(DevProblem P, const PcgState* __restrict__ in, PcgState* __restrict__ out,
                                              const double* __restrict__ part_pq, const double* __restrict__ p,
                                              const double* __restrict__ q, const double* __restrict__ b, double* __restrict__ x,
                                              double* __restrict__ r, double* __restrict__ z, const double* __restrict__ Minv_c,
                                              const double* __restrict__ Minv_i, double* __restrict__ part_Q,
                                              double* __restrict__ part_rho, int identity_precond, int first, double* __restrict__ zero_rep) {
  __shared__ double s_red[32];
  PcgState st = *in;
  pcg_phase_b(P, st, part_pq, p, q, b, x, r, z, Minv_c, Minv_i, part_Q, part_rho, identity_precond, first, zero_rep, s_red);
  if (blockIdx.x == 0 && threadIdx.x == 0) *out = st;
}

// ---- the three phases in ONE launch (one GPU kernel per CG iteration next to the matvec): A -> grid barrier -> B -> grid barrier
// -> C of the NEXT iteration.  VB CTAs of VT threads are co-resident on any device this engine runs on (the previous kernel of the
// stream has finished).  Sense-reversal barrier on bar[0] (arrivals) / bar[1] (generation), both zero before the first use; the
// partial sums written before a barrier are read behind it (fence by the arriving thread, cumulative through the block barrier).
// phase_mask: bit 0 = A, bit 1 = B, bit 2 = C (an iteration followed by a residual reset runs A|B only, the reset kernels, then C).
__device__ __forceinline__ void pcg_grid_barrier(int* bar) {
  __syncthreads();
  if (threadIdx.x == 0) {
    const int gen = *reinterpret_cast<volatile int*>(bar + 1);
    __threadfence();
    if (atomicAdd(bar, 1) == (int)gridDim.x - 1) {
      bar[0] = 0;
      __threadfence();
      atomicAdd(bar + 1, 1);
    } else {
#ifndef TBA_EMULATE
      const long long t0 = clock64();
      while (*reinterpret_cast<volatile int*>(bar + 1) == gen) {
        if (clock64() - t0 > 4000000000ll) { printf("tba: grid barrier of the fused PCG kernel timed out (block %d)\n", (int)blockIdx.x); __trap(); }
      }
#endif
    }
    __threadfence();
  }
  __syncthreads();
}
struct PcgVectors {
  const double *sm, *D2, *b, *Minv_c, *Minv_i;
  double *p, *q, *x, *r, *z, *xs, *y;
  double *part_pq, *part_Q, *part_rho;
  double* fold_rep;  // shared-intrinsics replica rows folded by phase A (one GPU), or nullptr
  int* zero_ctr;     // P2P counters of the next matvec, or nullptr
  int* bar;          // [2] grid barrier
  int identity_precond;
};
__global__ void __launch_bounds__(VT) k_pcg_fused(DevProblem P, const PcgState* __restrict__ in, PcgState* __restrict__ out, PcgVectors V,
                                                  int phase_mask, int first, P2pDev pp) {
  __shared__ double s_red[32];
  __shared__ double s_fold[10];
  PcgState st = *in;
  if (st.done) {  // the state travels on (the next kernel reads *out)
    if (blockIdx.x == 0 && threadIdx.x == 0) *out = st;
    return;
  }
  if (phase_mask & 1) {
    pcg_phase_a(P.ncs, P.ne, V.y, V.sm, V.D2, V.p, V.q, V.part_pq, V.fold_rep, pp, s_red, s_fold);
    if (phase_mask & 6) pcg_grid_barrier(V.bar);
  }
  if (phase_mask & 2) {
    pcg_phase_b(P, st, V.part_pq, V.p, V.q, V.b, V.x, V.r, V.z, V.Minv_c, V.Minv_i, V.part_Q, V.part_rho, V.identity_precond, first,
                (phase_mask & 1) ? V.fold_rep : nullptr, s_red);
    if (!st.done && (phase_mask & 4)) pcg_grid_barrier(V.bar);
  }
  if ((phase_mask & 4) && !st.done) pcg_phase_c(P.ncs, st, V.part_Q, V.part_rho, V.z, V.sm, V.p, V.xs, V.y, V.zero_ctr, s_red);
  if (blockIdx.x == 0 && threadIdx.x == 0) *out = st;
}

// Residual reset, second half, with the preconditioner applied to the fresh residual: r = b - (sm.*y + D2.*x); partial x.(b + r);
// z = Minv r; partial r.z (per parameter block)
__global__ void __launch_bounds__(VT) k_pcg_reset_bz(DevProblem P, const PcgState* __restrict__ in, double* __restrict__ y,
                                                     const double* __restrict__ sm, const double* __restrict__ D2,
                                                     const double* __restrict__ x, const double* __restrict__ b, double* __restrict__ r,
                                                     double* __restrict__ z, const double* __restrict__ Minv_c,
                                                     const double* __restrict__ Minv_i, double* __restrict__ part_Q,
                                                     double* __restrict__ part_rho, int identity_precond, const double* __restrict__ fold_rep, P2pDev pp) {
  __shared__ double s_red[32];
  __shared__ double s_fold[10];
  if (in->done) return;
  if (pp.world > 1) p2p_wait(pp);
  if (fold_rep != nullptr) {
    if (threadIdx.x < 10) {
      double v = y[P.ne + threadIdx.x];
      for (int rr = 0; rr < NREP; ++rr) v += fold_rep[(size_t)rr * REPW + threadIdx.x];
      s_fold[threadIdx.x] = v;
    }
    __syncthreads();
  }
  double accQ = 0.0, accR = 0.0;
  const int nblk = P.n_cam + P.n_group;
  for (int blk = blockIdx.x * VT + threadIdx.x; blk < nblk; blk += VB * VT) {
    const int i0 = blk < P.n_cam ? blk * 6 : P.ne + (blk - P.n_cam) * 10, n = blk < P.n_cam ? 6 : 10;
    for (int a = 0; a < n; ++a) {
      const int i = i0 + a;
      const double yv = pp.world > 1 ? p2p_sum(pp, i) : ((fold_rep != nullptr && i >= P.ne && i < P.ne + 10) ? s_fold[i - P.ne] : y[i]);
      const double rv = b[i] - (sm[i] * yv + D2[i] * x[i]);
      r[i] = rv;
      accQ += x[i] * (b[i] + rv);
    }
    accR += pcg_precondition_block(P, blk, Minv_c, Minv_i, r, z, identity_precond);
  }
  const double sQ = block_sum(accQ, s_red);
  const double sR = block_sum(accR, s_red);
  if (threadIdx.x == 0) { part_Q[blockIdx.x] = sQ; part_rho[blockIdx.x] = sR; }
}
__global__ void k_zero_rep_cols(double* __restrict__ rep) {  // re-zero the 10 folded replica columns (after k_pcg_reset_bz)
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < NREP * 10; i += gridDim.x * blockDim.x) rep[(size_t)(i / 10) * REPW + (i % 10)] = 0.0;
}

// Residual reset (every cg_residual_reset_period iterations): xs = sm .* x, y = 0 ... matvec ... r = b - (sm.*y + D2.*x)
__global__ void __launch_bounds__(VT) k_pcg_reset_a(int ncs, const PcgState* __restrict__ in, const double* __restrict__ x,
                                                    const double* __restrict__ sm, double* __restrict__ xs, double* __restrict__ y,
                                                    int* __restrict__ zero_ctr) {
  if (zero_ctr != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { zero_ctr[0] = 0; zero_ctr[1] = 0; }
  if (in->done) return;
  for (int i = blockIdx.x * VT + threadIdx.x; i < ncs; i += VB * VT) { xs[i] = sm[i] * x[i]; y[i] = 0.0; }
}
// Finalise a batch: run the pending Q-test so that `done`/`iters` are current, publish the flag.
__global__ void k_pcg_finalize(const PcgState* __restrict__ in, PcgState* __restrict__ out, const double* __restrict__ part_Q,
                               int* __restrict__ done_flag) {
  __shared__ double s_red[32];
  PcgState st = *in;
  if (!st.done && st.pending_q) {
    const double Q1 = -sum_partials(part_Q, s_red);
    const double zeta = st.iters * (Q1 - st.Q0) / Q1;
    st.Q1 = Q1;
    st.pending_q = 0;
    if (zeta < st.eta && st.iters >= st.min_iters) { st.done = 1; st.status = 0; }
    else {
      st.Q0 = Q1;
      if (st.iters >= st.max_iters) { st.done = 1; st.status = 1; }
      else st.iters += 1;
    }
  }
  if (threadIdx.x == 0) { *out = st; *done_flag = st.done; }
}
__global__ void k_set_flag(int* f, int v) { *f = v; }
__global__ void k_set_f64(double* p, double v) { *p = v; }

// xs = sm .* x (scaled solution -> unscaled), used before back-substitution
__global__ void k_cs_mul(int ncs, const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ o) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ncs; i += gridDim.x * blockDim.x) o[i] = a[i] * b[i];
}

// ------------------------------------------------- candidate / norms / gradient
// candidate = x + delta: cameras/intrinsics delta = -xs (xs = sm .* x_sol, zero on constant coordinates);
// points delta = dpt.  scal[4] += |delta|^2 (camera side, rank 0 only counts), scal[5] += |delta_pt|^2.
__global__ void k_candidate_cs(DevProblem P, const double* __restrict__ xs, double* __restrict__ scal, int count_norm) {
  __shared__ double s_red[32];
  double acc = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P.ncs; i += gridDim.x * blockDim.x) {
    const double d = -xs[i];
    if (i < P.ne) P.ext_c[i] = P.ext[i] + d; else P.intr_c[i - P.ne] = P.intr[i - P.ne] + d;
    acc += d * d;
  }
  const double s = block_sum(acc, s_red);
  if (threadIdx.x == 0 && count_norm) red_add(scal + 4, s);
}
__global__ void k_candidate_pt(DevProblem P, double* __restrict__ scal) {
  __shared__ double s_red[32];
  double acc = 0.0;
  for (size_t q = blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < (size_t)P.n_pt; q += (size_t)gridDim.x * blockDim.x) {  // one point per thread
    const bool cst = P.pt_const[q] != 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      double2 d = *reinterpret_cast<const double2*>(P.dpt + q * 4 + 2 * h);
      const double2 x = *reinterpret_cast<const double2*>(P.pt + q * 4 + 2 * h);
      if (cst) d = make_double2(0.0, 0.0);
      *reinterpret_cast<double2*>(P.pt_c + q * 4 + 2 * h) = make_double2(x.x + d.x, x.y + d.y);
      acc += d.x * d.x;
      acc += d.y * d.y;
    }
  }
  const double s = block_sum(acc, s_red);
  if (threadIdx.x == 0) red_add(scal + 5, s);
}

// |x|^2 over non-constant parameter blocks (ambient coordinates): scal[6] (camera side), scal[7] (points)
__global__ void k_xnorm(DevProblem P, const double* __restrict__ ext, const double* __restrict__ intr,
                        const double* __restrict__ pt, const double* __restrict__ blk_free /*[n_cam + n_group]*/,
                        double* __restrict__ scal, int count_cs) {
  __shared__ double s_red[32];
  double a_cs = 0.0, a_pt = 0.0;
  const size_t stride = (size_t)gridDim.x * blockDim.x, t0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (size_t i = t0; i < (size_t)P.ne; i += stride) if (blk_free[i / 6] != 0.0) a_cs += ext[i] * ext[i];
  for (size_t i = t0; i < (size_t)P.n_group * 10; i += stride) if (blk_free[P.n_cam + i / 10] != 0.0) a_cs += intr[i] * intr[i];
  for (size_t q = t0; q < (size_t)P.n_pt; q += stride) {
    const double2 a = *reinterpret_cast<const double2*>(pt + q * 4), b = *reinterpret_cast<const double2*>(pt + q * 4 + 2);
    if (!P.pt_const[q]) { a_pt += a.x * a.x; a_pt += a.y * a.y; a_pt += b.x * b.x; a_pt += b.y * b.y; }
  }
  const double s1 = block_sum(a_cs, s_red);
  const double s2 = block_sum(a_pt, s_red);
  if (threadIdx.x == 0) { if (count_cs) red_add(scal + 6, s1); red_add(scal + 7, s2); }
}

// max |g| over masked camera-space gradient -> gmax[0]; over free points -> gmax[1] (as ordered ints of the bit pattern)
__device__ __forceinline__ void atomic_max_double(double* addr, double v) {
  // v >= 0: the IEEE bit pattern is monotone
  atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}
// Gradient max norm in two steps around the all-reduce of the camera-side gradient: (1) this rank's points -> slot[0] (one slot per
// rank behind the linearisation scalars: after the SUM all-reduce every rank holds every rank's maximum), (2) the reduced camera-side
// gradient and the per-rank slots -> out[0].  Both by atomicMax on the bit pattern (targets zeroed by stage_linearize's memset).
__global__ void k_gradmax_pt(DevProblem P, double* __restrict__ slot) {
  double m = 0.0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < (size_t)P.n_pt; q += stride) {
    const double2 a = *reinterpret_cast<const double2*>(P.gp + q * 4), b = *reinterpret_cast<const double2*>(P.gp + q * 4 + 2);
    if (!P.pt_const[q]) m = fmax(fmax(m, fmax(fabs(a.x), fabs(a.y))), fmax(fabs(b.x), fabs(b.y)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.0) atomic_max_double(slot, m);
}
__global__ void k_gradmax_cs(int ncs, const double* __restrict__ g_cs, const double* __restrict__ mask, const double* __restrict__ slots,
                             int world, double* __restrict__ out) {
  double m = 0.0;
  const int t0 = blockIdx.x * blockDim.x + threadIdx.x;
  for (int i = t0; i < ncs; i += gridDim.x * blockDim.x) if (mask[i] != 0.0) m = fmax(m, fabs(g_cs[i]));
  if (t0 < world) m = fmax(m, slots[t0]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.0) atomic_max_double(out, m);
}

}  // namespace tba

#include "tba_inner.cuh"  // N4: observation passes of the inner iterations (uses DevProblem, block_sum, red_add from above)
