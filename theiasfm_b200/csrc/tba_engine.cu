// tba_engine.cu -- host side of the B200 bundle-adjustment engine + the C-ABI of
// include/theia_ba_b200.h.  Replaces ceres::Solve at
// src/theia/sfm/bundle_adjustment/bundle_adjuster.cc:205: a Levenberg-Marquardt
// trust-region loop (Ceres 1.14 TrustRegionMinimizer control flow, DESIGN.md section 3)
// whose every numerical stage is a CUDA kernel from tba_kernels.cuh.  The host
// only moves scalars.  No CPU fallback: every entry point fails with
// TBA_ERR_NO_DEVICE / TBA_ERR_CUDA when there is no usable GPU.
#include <dlfcn.h>
#include <nccl.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/theia_ba_b200.h"
#include "tba_kernels.cuh"
#include "tba_pack.h"
#include "tba_block_lm.h"

namespace tba {

// ------------------------------------------------------------------ NCCL (dlopen'ed)
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;  // optional (peer-memory setup)
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool load(std::string* err) {
    if (handle) return true;
#ifdef TBA_EMULATE
    const char* emu = getenv("TBA_EMU_NCCL");  // tests/emu/libemu_nccl.so (shared-memory stand-in, test infrastructure)
    const char* names[] = {emu ? emu : "libemu_nccl.so", "libemu_nccl.so"};
#else
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
#endif
    for (const char* n : names) {
      handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (handle) break;
    }
    if (!handle) { *err = std::string("cannot dlopen libnccl: ") + dlerror(); return false; }
    GetUniqueId = (decltype(GetUniqueId))dlsym(handle, "ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))dlsym(handle, "ncclCommInitRank");
    CommDestroy = (decltype(CommDestroy))dlsym(handle, "ncclCommDestroy");
    AllReduce = (decltype(AllReduce))dlsym(handle, "ncclAllReduce");
    GetErrorString = (decltype(GetErrorString))dlsym(handle, "ncclGetErrorString");
    AllGather = (decltype(AllGather))dlsym(handle, "ncclAllGather");
    if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllReduce || !GetErrorString) { *err = "libnccl is missing symbols"; return false; }
    return true;
  }
};
static NcclApi g_nccl;
static std::mutex g_nccl_mu;

// ------------------------------------------------------------------ device buffers
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  ~DevBuf() { release(); }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
  cudaError_t alloc(size_t count) {
    if (count <= n && p) return cudaSuccess;
    release();
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
};

}  // namespace tba

using namespace tba;

static_assert(TILE == kPackTile && MAXP == kPackMaxPoints, "tba_pack.h and tba_kernels.cuh disagree on the tile shape");

// A persistent kernel (one CTA per SM at most) with its launch shape.
template <class Fn>
struct PersistentKernel {
  Fn fn = nullptr;
  int nw = 0;       // warps per CTA
  size_t smem = 0;  // dynamic shared memory
};

// The kernel instantiations an uploaded problem runs, chosen once by tba_upload (select_kernels) from the intrinsics column set,
// the camera models and the switches read by tba_create.  The stages launch through it.
struct KernelSet {
  void (*linearize)(DevProblem, double*, double*, double*) = nullptr;
  // the implicit Schur operator by MODE (0 matvec, 1 reduced rhs, 2 back-substitution): tile per CTA, and streaming over the normal tiles
  void (*schur[3])(DevProblem, const double*, double*, double*, const int*, int) = {};
  size_t schur_smem = 0;
  PersistentKernel<void (*)(DevProblem, const double*, double*, double*, const int*, int, P2pDev)> schur_stream[3];
  PersistentKernel<void (*)(DevProblem, double*, double*, double*, double*, int)> prepare_stream;
  void (*precond_ext)(DevProblem, double*, int) = nullptr;
  void (*precond_intr)(DevProblem, double*, int) = nullptr;
  size_t precond_intr_smem = 0;
  void (*cost)(DevProblem, const double*, const double*, const double*, const double*, double*) = nullptr;
  void (*adjust_tracks)(DevProblem, const long long*, const int*, PointLmOptions, uint8_t*, double*) = nullptr;
  void (*filter_tracks)(DevProblem, const long long*, const int*, double, double, uint8_t*, double*) = nullptr;
  void (*estimate_tracks)(DevProblem, const long long*, const int*, const double*, TrackEstimatorOptions, uint8_t*, double*) = nullptr;
  void (*block_pass[2][2])(DevProblem, BlockPassArgs) = {};  // [KIND][COST_ONLY]
  int n_stream_tiles = 0;  // leading tiles the streaming kernels take: the normal tiles, or 0 when they are switched off
};

struct tba_context {
  int device = 0, rank = 0, world = 1;
  cudaStream_t stream = nullptr;
  ncclComm_t comm = nullptr;
  std::string err;
  bool uploaded = false;
  tba_options opt;
  int NI = 0, NJ = 14;  // stored intrinsics columns, Jacobian doubles per observation
  KernelSet ks;
  DevProblem P;
  int n_cam = 0, n_group = 0, n_pt = 0, n_tiles = 0;
  int64_t n_obs = 0, n_slots = 0;
  std::vector<int64_t> slot_orig;  // slot -> caller observation index (-1 padding); built on demand by the debug read-back
  HostPack pack;                   // host packing scratch + result of the last upload (kept: capacity and faulted-in pages are reused)
  int64_t launches = 0;
  double h2d_bytes = 0, d2h_bytes = 0;
  double setup_seconds = 0;
  int64_t n_free_cs = 0;  // free camera-space coordinates (global)
  int64_t n_free_pt = 0;  // free points on this rank
  int64_t n_free_pt_global = 0;
  int n_pt_caller = 0;
  // parameters and packed problem
  DevBuf<double> ext, intr, pt, ext_c, intr_c, pt_c, cam_rec, cam_rec_c, cam_s4, cam_s4_c, xy, J, res, Hpp, gp, Mp, sp, dpt;
  DevBuf<int> cam_group, group_model, slot_cam, slot_pt, tile_pt_begin, tile_nruns;
  DevBuf<uint8_t> slot_flags, pt_const, tile_flags;
  void* stage = nullptr;  // pinned host staging for the packed observation arrays
  size_t stage_cap = 0;
  int n_long_points = 0;
  DevBuf<int16_t> slot_run;
  DevBuf<long long> pt_slot;   // first slot of each packed point (track filter)
  DevBuf<int> pt_len;          // observations of each packed point
  DevBuf<double> pt_stat;      // per-point mean squared reprojection error (track filter output)
  // camera space: [g | cn | scal(16)] is one allreduce buffer
  DevBuf<double> lin;       // g_cs[ncs] | cn_cs[ncs] | scal[16]
  DevBuf<double> mask, blk_free, sm, D2, Sblk /*[n_cam*21 | n_group*55]*/, Minv_c, Minv_i;
  DevBuf<double> z2;  // z = Minv r of the PCG (z holds q = S p)
  int last_cg_iters = 6;  // CG iterations of the previous linear solve: size of the first enqueued batch
  DevBuf<double> b, x, r, p, z, xs, y, part /*3 x VB*/, gmax, flag, scal2 /*16*/, rep /*NREP x REPW*/;
  DevBuf<PcgState> st;      // [2]
  DevBuf<int> done_flag;
  DevBuf<int> pcg_bar;         // [2] grid barrier of k_pcg_fused (arrivals, generation)
  bool have_scale = false;
  // optional per-kernel timing (CUDA events on the engine stream)
  bool profiling = false;
  std::vector<cudaEvent_t> ev_pool;
  std::vector<std::pair<int, int>> ev_spans[8];  // 0: matvec, 1: linearize, 2: precond_ext, 3: precond_intr, 4: rhs, 5: back-substitution, 6: candidate cost, 7: fused prepare (rhs + both preconditioner block families) ; indices into ev_pool
  // set by tba_solve_multi (which sees the whole problem) before tba_upload: global per-camera observation counts and the
  // global number of free points, so that the upload needs no collective
  const double* preset_cnt_cam = nullptr;
  int64_t preset_free_pt = -1;
  // N4 inner iterations: host copies of the constness description and their device mirrors (allocated only when requested)
  std::vector<uint8_t> h_ext_const;
  std::vector<uint32_t> h_group_mask;
  std::vector<int> h_group_model;
  DevBuf<uint8_t> d_ext_const, d_blk_active;
  DevBuf<uint32_t> d_group_mask;
  DevBuf<double> d_blk_vals, d_blk_rec, d_blk_acc, d_inner_cost2;
  DevBuf<uint8_t> d_inner_status;
  int64_t inner_passes = 0;
  bool has_ext_models = false;  // some group uses FISHEYE / FOV / DIVISION_UNDISTORTION: EXT kernel instantiations
  bool exp_tred = true;     // transposed RED emission (warp_red_rows) in k_linearize / k_precond_ext / rhs / matvec; TBA_TRED=0: the round-1 lane-per-row REDs
  bool exp_lin_occ = true;  // k_linearize compiled for 3 CTAs/SM (80 registers, ~130 bytes of spills); TBA_LIN_OCC=2: 2 CTAs/SM, 128 registers
  double trace_pcg_gpu_ms = 0.0;  // TBA_TRACE_LM: device-side span of the PCG launches (first launch .. state copy), summed over a minimize
  bool pcg_fused = true;    // one vector kernel per CG iteration (k_pcg_fused, grid barriers between its phases); TBA_PCG=split: k_pcg_c / k_pcg_a / k_pcg_b
  bool stream_schur = true; // persistent streaming k_schur_stream over the normal tiles; TBA_MATVEC=tile: the tile-per-CTA k_schur everywhere
  // fused matvec + all-reduce over peer memory (P2pDev, tba_kernels.cuh): world > 1, every peer reachable, TBA_P2P != 0
  bool p2p_enabled = true, p2p_ok = false, p2p_use = false;
  size_t p2p_cap = 0;
  double* p2p_inbox = nullptr;                // local inbox [2][world][cap]
  unsigned long long* p2p_flags = nullptr;    // local flags [world]
  int* p2p_ctr = nullptr;
  std::vector<void*> p2p_opened;              // peer mappings opened with cudaIpcOpenMemHandle
  DevBuf<double*> p2p_inbox_ptrs;
  DevBuf<unsigned long long*> p2p_flag_ptrs;
  unsigned long long p2p_seq = 0;
  int n_sm = 148;
  int64_t real_matvecs = 0;  // matvec launches that did work (not early-exited after PCG convergence)
  double x_cost = 0, fixed_cost = 0;
  // host mirrors
  double* h_scal = nullptr;  // pinned [64]
  PcgState* h_st = nullptr;  // pinned
};

namespace {

void set_err(tba_context* c, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  c->err = buf;
}

#define CUDA_OK(c, expr)                                                                        \
  do {                                                                                          \
    cudaError_t e__ = (expr);                                                                   \
    if (e__ != cudaSuccess) {                                                                   \
      set_err(c, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(e__), __FILE__, __LINE__, #expr); \
      return TBA_ERR_CUDA;                                                                      \
    }                                                                                           \
  } while (0)

#define NCCL_OK(c, expr)                                                                        \
  do {                                                                                          \
    ncclResult_t r__ = (expr);                                                                  \
    if (r__ != ncclSuccess) {                                                                   \
      set_err(c, "NCCL error %s at %s:%d", g_nccl.GetErrorString(r__), __FILE__, __LINE__);     \
      return TBA_ERR_NCCL;                                                                      \
    }                                                                                           \
  } while (0)

// Every launch is checked: a rejected launch (bad configuration, missing shared-memory opt-in) must not turn into a
// silently skipped kernel.
#ifdef TBA_EMULATE  // CPU emulation build (tests/emu): blocks run one after the other, threads as fibers
#define LAUNCH(c, kern, grid, block, smem, ...)                                              \
  do {                                                                                       \
    if ((unsigned)(grid) == 0u) break; /* see the CUDA variant */                            \
    emu::launch((const void*)(kern), (unsigned)(grid), (unsigned)(block), (size_t)(smem), [&] { kern(__VA_ARGS__); }); \
    if (cudaGetLastError() != cudaSuccess) {                                                 \
      set_err(c, "kernel launch failed: invalid configuration at %s:%d (%s)", __FILE__, __LINE__, #kern); \
      return TBA_ERR_CUDA;                                                                   \
    }                                                                                        \
    (c)->launches++;                                                                         \
  } while (0)
#else
#define LAUNCH(c, kern, grid, block, smem, ...)                                                              \
  do {                                                                                                       \
    if ((unsigned)(grid) == 0u) break; /* nothing to do (empty problem / empty set): a 0-block launch is an error */ \
    kern<<<(grid), (block), (smem), (c)->stream>>>(__VA_ARGS__);                                             \
    const cudaError_t le__ = cudaPeekAtLastError();                                                          \
    if (le__ != cudaSuccess) {                                                                               \
      set_err(c, "kernel launch failed: %s at %s:%d (%s)", cudaGetErrorString(le__), __FILE__, __LINE__, #kern); \
      return TBA_ERR_CUDA;                                                                                   \
    }                                                                                                        \
    (c)->launches++;                                                                                         \
  } while (0)
#endif

int prof_begin(tba_context* c) {
  if (!c->profiling) return -1;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return -1;
  c->ev_pool.push_back(e);
  cudaEventRecord(e, c->stream);
  return (int)c->ev_pool.size() - 1;
}
void prof_end(tba_context* c, int which, int begin) {
  if (begin < 0) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  c->ev_pool.push_back(e);
  cudaEventRecord(e, c->stream);
  c->ev_spans[which].push_back({begin, (int)c->ev_pool.size() - 1});
}

// The intrinsics column set the kernels are compiled for: the first of these that covers every free intrinsics column.
const uint32_t kMasks[] = {0x000u, 0x001u, 0x061u, 0x0E1u, 0x07Fu, 0x3FFu};
uint32_t intrinsics_mask(uint32_t union_free) {
  for (uint32_t m : kMasks) if ((union_free & ~m) == 0) return m;
  return 0x3FFu;
}

int allreduce_sum(tba_context* c, double* buf, size_t n) {
  if (c->world == 1) return TBA_OK;
  NCCL_OK(c, g_nccl.AllReduce(buf, buf, n, ncclDouble, ncclSum, c->comm, c->stream));
  return TBA_OK;
}

double* lin_g(tba_context* c) { return c->lin.p; }
double* lin_cn(tba_context* c) { return c->lin.p + c->P.ncs; }
double* lin_scal(tba_context* c) { return c->lin.p + 2 * (size_t)c->P.ncs; }
// grid of the per-point / per-element streaming kernels (256 threads per CTA): enough CTAs to cover the latency of a dependent
// load chain (8 per SM), not more than the work
int small_grid(const tba_context* c, int64_t n_items) { return (int)std::max<int64_t>(1, std::min<int64_t>((n_items + 255) / 256, (int64_t)c->n_sm * 8)); }
// grid of the persistent streaming kernels: one CTA per SM at most, not more than the slices of 32 observations need
int persistent_grid(const tba_context* c, int nw, int n_slices) { return std::max(1, std::min(c->n_sm, (n_slices + nw - 1) / nw)); }

// scal layout: 0 cost, 1 fixed cost, 2 failed evals, 3 model cost change, 4 |delta_cs|^2, 5 |delta_pt|^2,
//              6 |x_cs|^2, 7 |x_pt|^2
int read_scal(tba_context* c, const double* dev, int n, double* out) {
  CUDA_OK(c, cudaMemcpyAsync(c->h_scal, dev, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  memcpy(out, c->h_scal, n * sizeof(double));
  return TBA_OK;
}
// Sums n doubles on the device over the ranks, then reads them to the host.
int allreduce_read(tba_context* c, double* dev, int n, double* out) {
  const int rc = allreduce_sum(c, dev, (size_t)n);
  return rc ? rc : read_scal(c, dev, n, out);
}
// Sums n host values over the ranks in place (through scal2): every rank gets the same values back.
int allreduce_host(tba_context* c, double* v, size_t n) {
  CUDA_OK(c, c->scal2.alloc(std::max<size_t>(n, 16)));
  CUDA_OK(c, cudaMemcpyAsync(c->scal2.p, v, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  const int rc = allreduce_sum(c, c->scal2.p, n);
  if (rc) return rc;
  CUDA_OK(c, cudaMemcpyAsync(v, c->scal2.p, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  return TBA_OK;
}

// ---- stages ---------------------------------------------------------------------------------
// Evaluate cost / residuals / compact Jacobian / gradient / column norms at x (and Jacobi scale at iteration 0).
// gmax != nullptr: also the gradient max norm (max |g| over the non-constant parameters), in the same all-reduce and the same
// device->host read as the cost -- one collective and one host synchronisation per linearisation instead of two each.
int stage_linearize(tba_context* c, double* cost, double* fixed, bool* ok, double* gmax = nullptr) {
  DevProblem& P = c->P;
  const size_t n_lin = 2 * (size_t)P.ncs + 16 + (size_t)c->world;  // [gradient | column norms | 16 scalars | one slot per rank]
  CUDA_OK(c, cudaMemsetAsync(c->lin.p, 0, n_lin * sizeof(double), c->stream));
  LAUNCH(c, k_cam_prep, (P.n_cam + 127) / 128, 128, 0, P.n_cam, P.ext, P.cam_rec, P.cam_s4);
  if (P.n_tiles > 0) {
    const int pb = prof_begin(c);
    LAUNCH(c, c->ks.linearize, P.n_tiles, TILE, 0, P, lin_g(c), lin_cn(c), c->rep.p);
    prof_end(c, 1, pb);
    LAUNCH(c, k_fold, 1, REPW, 0, c->rep.p, lin_g(c) + P.ne, lin_cn(c) + P.ne, lin_scal(c));
  }
  if (gmax && P.n_pt > 0) LAUNCH(c, k_gradmax_pt, small_grid(c, P.n_pt), 256, 0, P, lin_scal(c) + 16 + c->rank);
  int rc = allreduce_sum(c, c->lin.p, n_lin);
  if (rc) return rc;
  if (gmax) LAUNCH(c, k_gradmax_cs, VB, VT, 0, P.ncs, lin_g(c), c->mask.p, lin_scal(c) + 16, c->world, lin_scal(c) + 3);
  if (!c->have_scale) {
    LAUNCH(c, k_cs_scale, VB, VT, 0, P.ncs, lin_cn(c), c->mask.p, c->opt.jacobi_scaling, c->sm.p);
    if (P.n_pt > 0) LAUNCH(c, k_point_scale, (P.n_pt + 255) / 256, 256, 0, P, c->opt.jacobi_scaling);
    c->have_scale = true;
  }
  double s[4];
  rc = read_scal(c, lin_scal(c), 4, s);
  if (rc) return rc;
  *cost = s[0]; *fixed = s[1]; *ok = s[2] == 0.0;
  if (gmax) *gmax = s[3];
  return TBA_OK;
}

// ---- peer-memory setup for the fused matvec + all-reduce (collective: every rank calls it from tba_upload) -------------
void p2p_release(tba_context* c) {
#ifndef TBA_EMULATE
  for (void* q : c->p2p_opened) cudaIpcCloseMemHandle(q);
#endif
  c->p2p_opened.clear();
  if (c->p2p_inbox) cudaFree(c->p2p_inbox);
  if (c->p2p_flags) cudaFree(c->p2p_flags);
  if (c->p2p_ctr) cudaFree(c->p2p_ctr);
  c->p2p_inbox = nullptr; c->p2p_flags = nullptr; c->p2p_ctr = nullptr; c->p2p_cap = 0; c->p2p_ok = false;
}

#ifndef TBA_EMULATE
struct P2pInfo {
  long long pid;
  int device, ok;
  double* inbox;
  unsigned long long* flags;
  cudaIpcMemHandle_t h_inbox, h_flags;
};
#endif

// Allocates the inbox for `ncs` doubles per slot and exchanges the mappings.  On any failure on any rank every rank falls
// back to the NCCL all-reduce (p2p_ok = false); never an error.
int p2p_setup(tba_context* c, int ncs) {
#ifdef TBA_EMULATE
  (void)ncs; c->p2p_ok = false; return TBA_OK;  // the SIMT emulation has no peer mappings: NCCL stand-in
#else
  if (c->world == 1 || !c->p2p_enabled || g_nccl.AllGather == nullptr) { c->p2p_ok = false; return TBA_OK; }
  const size_t cap = ((size_t)ncs + 1) / 2 * 2;
  if (c->p2p_ok && cap <= c->p2p_cap) return TBA_OK;  // (ncs is a global property: every rank takes the same branch)
  p2p_release(c);
  const int W = c->world;
  int ok = 1;
  if (cudaMalloc(&c->p2p_inbox, 2 * (size_t)W * cap * sizeof(double)) != cudaSuccess) { c->p2p_inbox = nullptr; ok = 0; }
  if (cudaMalloc(&c->p2p_flags, (size_t)W * sizeof(unsigned long long)) != cudaSuccess) { c->p2p_flags = nullptr; ok = 0; }
  if (cudaMalloc(&c->p2p_ctr, 2 * sizeof(int)) != cudaSuccess) { c->p2p_ctr = nullptr; ok = 0; }
  cudaGetLastError();
  P2pInfo mine;
  memset(&mine, 0, sizeof mine);
  mine.pid = (long long)getpid(); mine.device = c->device; mine.inbox = c->p2p_inbox; mine.flags = c->p2p_flags;
  if (ok) {
    CUDA_OK(c, cudaMemsetAsync(c->p2p_flags, 0, (size_t)W * sizeof(unsigned long long), c->stream));
    CUDA_OK(c, cudaMemsetAsync(c->p2p_ctr, 0, 2 * sizeof(int), c->stream));
    if (cudaIpcGetMemHandle(&mine.h_inbox, c->p2p_inbox) != cudaSuccess || cudaIpcGetMemHandle(&mine.h_flags, c->p2p_flags) != cudaSuccess) { ok = 0; cudaGetLastError(); }
  }
  mine.ok = ok;
  // all-gather the descriptors (device buffers, NCCL)
  DevBuf<char> d_send, d_recv;
  CUDA_OK(c, d_send.alloc(sizeof(P2pInfo)));
  CUDA_OK(c, d_recv.alloc(sizeof(P2pInfo) * (size_t)W));
  CUDA_OK(c, cudaMemcpyAsync(d_send.p, &mine, sizeof mine, cudaMemcpyHostToDevice, c->stream));
  NCCL_OK(c, g_nccl.AllGather(d_send.p, d_recv.p, sizeof(P2pInfo), ncclChar, c->comm, c->stream));
  std::vector<P2pInfo> all((size_t)W);
  CUDA_OK(c, cudaMemcpyAsync(all.data(), d_recv.p, sizeof(P2pInfo) * (size_t)W, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  std::vector<double*> inbox((size_t)W, nullptr);
  std::vector<unsigned long long*> flags((size_t)W, nullptr);
  for (int q = 0; q < W && ok; ++q) {
    if (!all[q].ok) { ok = 0; break; }
    if (q == c->rank) { inbox[q] = c->p2p_inbox; flags[q] = c->p2p_flags; continue; }
    if (all[q].pid == mine.pid) {  // rank threads of one process (tba_solve_multi): plain peer access
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, c->device, all[q].device) != cudaSuccess || !can) { ok = 0; cudaGetLastError(); break; }
      const cudaError_t e = cudaDeviceEnablePeerAccess(all[q].device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { ok = 0; }
      cudaGetLastError();
      inbox[q] = all[q].inbox; flags[q] = all[q].flags;
    } else {                       // one process per GPU: CUDA IPC mappings (peer access enabled lazily by the runtime)
      void *pi = nullptr, *pf = nullptr;
      if (cudaIpcOpenMemHandle(&pi, all[q].h_inbox, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); break; }
      c->p2p_opened.push_back(pi);
      if (cudaIpcOpenMemHandle(&pf, all[q].h_flags, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); break; }
      c->p2p_opened.push_back(pf);
      inbox[q] = (double*)pi; flags[q] = (unsigned long long*)pf;
    }
  }
  // every rank must agree: the number of ranks that failed, summed over the ranks
  double failed = ok ? 0.0 : 1.0;
  const int rc = allreduce_host(c, &failed, 1);
  if (rc) return rc;
  if (failed != 0.0) { p2p_release(c); return TBA_OK; }
  CUDA_OK(c, c->p2p_inbox_ptrs.alloc((size_t)W));
  CUDA_OK(c, c->p2p_flag_ptrs.alloc((size_t)W));
  CUDA_OK(c, cudaMemcpyAsync(c->p2p_inbox_ptrs.p, inbox.data(), (size_t)W * sizeof(double*), cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(c->p2p_flag_ptrs.p, flags.data(), (size_t)W * sizeof(unsigned long long*), cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  c->p2p_cap = cap; c->p2p_seq = 0; c->p2p_ok = true;
  return TBA_OK;
#endif
}

P2pDev p2p_none() { return P2pDev(); }
// The descriptor of the NEXT exchange (advances the sequence number): the matvec launch and its consumer get the same one.
P2pDev p2p_next(tba_context* c) {
  P2pDev d;
  d.world = c->world; d.rank = c->rank; d.seq = ++c->p2p_seq; d.cap = c->p2p_cap;
  d.inbox = c->p2p_inbox_ptrs.p; d.flags = c->p2p_flag_ptrs.p; d.ctr = c->p2p_ctr;
  return d;
}

// One pass of the implicit Schur operator (mode 0 matvec, 1 reduced rhs, 2 back-substitution) over every tile: the persistent
// streaming kernel over the leading normal tiles, the tile-per-CTA kernel over the rest (the long tiles: tracks of 33..256
// observations).
int launch_schur(tba_context* c, int mode, const double* xs, double* y, const int* done, const P2pDev& pp = P2pDev()) {
  DevProblem& P = c->P;
  const KernelSet& k = c->ks;
  if (k.n_stream_tiles > 0) {
    const int n_slices = k.n_stream_tiles * (TILE / 32);
    const auto& s = k.schur_stream[mode];
    LAUNCH(c, s.fn, persistent_grid(c, s.nw, n_slices), s.nw * 32, s.smem, P, xs, y, c->rep.p, done, n_slices, pp);
  }
  const int rest = P.n_tiles - k.n_stream_tiles;
  if (rest > 0) LAUNCH(c, k.schur[mode], rest, TILE, k.schur_smem, P, xs, y, c->rep.p, done, k.n_stream_tiles);
  return TBA_OK;
}

// LM diagonal, per-point (E'E + D^2)^-1, SCHUR_JACOBI blocks, reduced rhs.  *ok=false if a block is not PD.
// defer_flag: do not wait for the "a point block / preconditioner block is not positive definite" flag here; stage_pcg reads it
// together with its own termination state (one host synchronisation less per LM iteration).
int stage_prepare(tba_context* c, double radius, bool* ok, bool defer_flag = false) {
  DevProblem& P = c->P;
  const tba_options& o = c->opt;
  const KernelSet& k = c->ks;
  CUDA_OK(c, cudaMemsetAsync(c->flag.p, 0, sizeof(double), c->stream));
  LAUNCH(c, k_cs_diag, VB, VT, 0, P.ncs, lin_cn(c), c->sm.p, radius, o.min_lm_diagonal, o.max_lm_diagonal, c->D2.p);
  if (P.n_pt > 0) LAUNCH(c, k_point_blocks, (P.n_pt + 255) / 256, 256, 0, P, radius, o.min_lm_diagonal, o.max_lm_diagonal, c->flag.p);
  const size_t nS = (size_t)P.n_cam * 21 + (size_t)P.n_group * 55;
  const bool precond = o.preconditioner_type != TBA_PRECOND_IDENTITY;
  // with a preconditioner the reduced rhs is accumulated behind the blocks ([blocks | flag | pad | rhs]): one memset and, on several
  // GPUs, ONE all-reduce for all of it
  const size_t y_off = (nS + 2) & ~(size_t)1;
  double* const yr = precond ? c->Sblk.p + y_off : c->y.p;
  if (precond) CUDA_OK(c, cudaMemsetAsync(c->Sblk.p, 0, (y_off + (size_t)P.ncs) * sizeof(double), c->stream));
  else CUDA_OK(c, cudaMemsetAsync(c->y.p, 0, (size_t)P.ncs * sizeof(double), c->stream));
  if (P.n_tiles > 0) {
    // normal tiles: ONE streaming pass over J for the reduced rhs and both families of SCHUR_JACOBI blocks (k_prepare_stream);
    // long tiles (and TBA_MATVEC=tile / IDENTITY preconditioner): the three tile kernels
    const int first_tile = precond ? k.n_stream_tiles : 0;
    if (first_tile > 0) {
      const int n_slices = first_tile * (TILE / 32);
      const int pb = prof_begin(c);
      LAUNCH(c, k.prepare_stream.fn, persistent_grid(c, k.prepare_stream.nw, n_slices), k.prepare_stream.nw * 32, k.prepare_stream.smem,
             P, yr, c->Sblk.p, c->Sblk.p + (size_t)P.n_cam * 21, c->rep.p, n_slices);
      prof_end(c, 7, pb);
    }
    const int rest = P.n_tiles - first_tile;
    if (rest > 0 && precond) {
      const int pb_ext = prof_begin(c);
      LAUNCH(c, k.precond_ext, rest, TILE, 0, P, c->Sblk.p, first_tile);
      prof_end(c, 2, pb_ext);
      if (c->NI > 0) {
        const int pb_intr = prof_begin(c);
        LAUNCH(c, k.precond_intr, rest, TILE, k.precond_intr_smem, P, c->Sblk.p + (size_t)P.n_cam * 21, first_tile);
        prof_end(c, 3, pb_intr);
      }
    }
    if (rest > 0) {
      const int pb_rhs = prof_begin(c);
      if (first_tile == 0) { const int rc1 = launch_schur(c, 1, nullptr, yr, nullptr); if (rc1) return rc1; }
      else LAUNCH(c, k.schur[1], rest, TILE, k.schur_smem, P, nullptr, yr, c->rep.p, nullptr, first_tile);
      prof_end(c, 4, pb_rhs);
    }
    if (P.single_group) LAUNCH(c, k_fold, 1, REPW, 0, c->rep.p, yr + P.ne, nullptr, nullptr);
  }
  if (precond) {
    // the not-positive-definite flag of k_point_blocks rides in the extra slot behind the blocks: one all-reduce less
    CUDA_OK(c, cudaMemcpyAsync(c->Sblk.p + nS, c->flag.p, sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    int rc = allreduce_sum(c, c->Sblk.p, y_off + (size_t)P.ncs);
    if (rc) return rc;
    CUDA_OK(c, cudaMemcpyAsync(c->flag.p, c->Sblk.p + nS, sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    LAUNCH(c, k_precond_finish, (P.n_cam + P.n_group + 63) / 64, 64, 0, P, c->Sblk.p, c->Sblk.p + (size_t)P.n_cam * 21, c->sm.p,
           c->D2.p, c->Minv_c.p, c->Minv_i.p, c->flag.p);
  }
  int rc = precond ? TBA_OK : allreduce_sum(c, c->y.p, P.ncs);
  if (rc) return rc;
  LAUNCH(c, k_pcg_init, VB, VT, 0, P.ncs, yr, c->sm.p, c->b.p, c->x.p, c->r.p, c->part.p);
  // the PD flag is summed over ranks so that every rank takes the same branch (with the preconditioner: done above)
  if (!precond) { rc = allreduce_sum(c, c->flag.p, 1); if (rc) return rc; }
  if (defer_flag) { *ok = true; return TBA_OK; }
  double f;
  rc = read_scal(c, c->flag.p, 1, &f);
  if (rc) return rc;
  *ok = f == 0.0;
  return TBA_OK;
}

const int* st_done(const PcgState* st) { return reinterpret_cast<const int*>(reinterpret_cast<const char*>(st) + offsetof(PcgState, done)); }

// The fused path is available when the whole problem runs through the streaming kernel (no long tiles, the default kernels).
bool p2p_matvec_possible(const tba_context* c) { return c->p2p_ok && c->p2p_use; }

// defer_fold: the caller folds the shared-intrinsics replica rows itself (k_pcg_a / k_pcg_reset_bz; one GPU only).
// pp (world > 1): the matvec kernel itself pushes the partial sums to the peers; no fold launch, no NCCL call.
int launch_matvec(tba_context* c, const int* done, bool defer_fold = false, const P2pDev& pp = P2pDev()) {
  DevProblem& P = c->P;
  if (P.n_tiles > 0) {
    const int pb = prof_begin(c);
    const int rc = launch_schur(c, 0, c->xs.p, c->y.p, done, pp);
    if (rc) return rc;
    prof_end(c, 0, pb);
    if (pp.world > 1) return TBA_OK;
    if (P.single_group && !defer_fold) LAUNCH(c, k_fold, 1, REPW, 0, c->rep.p, c->y.p + P.ne, nullptr, nullptr);
  }
  return allreduce_sum(c, c->y.p, P.ncs);
}

// ConjugateGradientsSolver::Solve on the reduced system; control flow on the device (PcgState),
// the host enqueues iterations in batches and polls the done flag.
// system_ok != nullptr: also fetch stage_prepare's deferred flag (false: the linear system was not usable, the result is void).
int stage_pcg(tba_context* c, int* iters, int* status, bool* system_ok = nullptr) {
  DevProblem& P = c->P;
  const tba_options& o = c->opt;
  double* part_rho = c->part.p;
  double* part_pq = c->part.p + VB;
  double* part_Q = c->part.p + 2 * VB;
  PcgState* st = c->st.p;
  static const bool trace = getenv("TBA_TRACE_LM") != nullptr;
  cudaEvent_t tev[2] = {nullptr, nullptr};
  if (trace) { cudaEventCreate(&tev[0]); cudaEventCreate(&tev[1]); cudaEventRecord(tev[0], c->stream); }
  LAUNCH(c, k_pcg_init_state, 1, 1, 0, st, c->part.p, o.min_linear_solver_iterations, o.max_linear_solver_iterations, o.eta);
  LAUNCH(c, k_set_flag, 1, 1, 0, c->done_flag.p, 0);
  if (c->n_free_cs == 0) {  // no reduced system: back-substitution only
    *iters = 0; *status = 0;
    CUDA_OK(c, cudaMemsetAsync(c->x.p, 0, (size_t)P.ncs * sizeof(double), c->stream));
    if (system_ok) { double f; const int rc = read_scal(c, c->flag.p, 1, &f); if (rc) return rc; *system_ok = f == 0.0; }
    return TBA_OK;
  }
  const int ident = o.preconditioner_type == TBA_PRECOND_IDENTITY;
  int cur = 0;  // index of the valid state
  int it = 0;
  // Three vector kernels per iteration (k_pcg_c, k_pcg_a, k_pcg_b; tba_kernels.cuh) around the matvec.  One GPU and one shared
  // intrinsics group: k_pcg_a folds the matvec's replica rows itself (no k_fold launch).  The host enqueues the number of
  // iterations the previous solve needed (+2) before it looks at the device-side state; surplus iterations early-exit.
  const bool fold_in_a = c->world == 1 && P.single_group && P.n_tiles > 0;
  double* fold_rep = fold_in_a ? c->rep.p : nullptr;
  const bool p2p = p2p_matvec_possible(c);  // multi-GPU: the matvec pushes its partial sums to the peers, k_pcg_a sums the inbox
  int* zero_ctr = p2p ? c->p2p_ctr : nullptr;
  // c->pcg_fused (default): ONE vector kernel per CG iteration -- phases A and B of iteration k and phase C of iteration k + 1 in
  // k_pcg_fused, grid barriers in between -- i.e. two launches per iteration with the matvec; TBA_PCG=split (and the SIMT emulation
  // build, which cannot run a grid barrier): the three kernels
  const bool fused = c->pcg_fused;
  PcgVectors V;
  V.sm = c->sm.p; V.D2 = c->D2.p; V.b = c->b.p; V.Minv_c = c->Minv_c.p; V.Minv_i = c->Minv_i.p;
  V.p = c->p.p; V.q = c->z.p; V.x = c->x.p; V.r = c->r.p; V.z = c->z2.p; V.xs = c->xs.p; V.y = c->y.p;
  V.part_pq = part_pq; V.part_Q = part_Q; V.part_rho = part_rho; V.fold_rep = fold_rep; V.zero_ctr = zero_ctr; V.bar = c->pcg_bar.p;
  V.identity_precond = ident;
  if (fused) {  // z = Minv r, rho (phase B, first) and phase C of iteration 1
    LAUNCH(c, k_pcg_fused, VB, VT, 0, P, st + cur, st + (cur ^ 1), V, 2 | 4, 1, p2p_none());
    cur ^= 1;
  } else {
    LAUNCH(c, k_pcg_b, VB, VT, 0, P, st + cur, st + (cur ^ 1), part_pq, c->p.p, c->z.p, c->b.p, c->x.p, c->r.p, c->z2.p, c->Minv_c.p, c->Minv_i.p,
           part_Q, part_rho, ident, 1, nullptr);
    cur ^= 1;
  }
  bool c_pending = !fused;  // phase C of the coming iteration still to be launched (split mode: always; fused: after a residual reset)
  int batch = std::max(4, std::min(c->last_cg_iters + 2, 64));
  for (;;) {
    for (int k = 0; k < batch; ++k) {
      ++it;
      if (c_pending) {
        LAUNCH(c, k_pcg_c, VB, VT, 0, P.ncs, st + cur, st + (cur ^ 1), part_Q, part_rho, c->z2.p, c->sm.p, c->p.p, c->xs.p, c->y.p, nullptr, zero_ctr);
        cur ^= 1;
      }
      // every kernel of an iteration (matvec included) early-exits through the device-side state
      const P2pDev pp = p2p ? p2p_next(c) : p2p_none();
      int rc = launch_matvec(c, st_done(st + cur), fold_in_a, pp);
      if (rc) return rc;
      const bool reset_now = o.cg_residual_reset_period > 0 && it % o.cg_residual_reset_period == 0;
      if (fused) {
        LAUNCH(c, k_pcg_fused, VB, VT, 0, P, st + cur, st + (cur ^ 1), V, reset_now ? (1 | 2) : (1 | 2 | 4), 0, pp);
        cur ^= 1;
        c_pending = reset_now;
      } else {
        LAUNCH(c, k_pcg_a, VB, VT, 0, P.ncs, P.ne, st + cur, c->y.p, c->sm.p, c->D2.p, c->p.p, c->z.p, part_pq, fold_rep, pp);
        LAUNCH(c, k_pcg_b, VB, VT, 0, P, st + cur, st + (cur ^ 1), part_pq, c->p.p, c->z.p, c->b.p, c->x.p, c->r.p, c->z2.p, c->Minv_c.p, c->Minv_i.p,
               part_Q, part_rho, ident, 0, fold_rep);
        cur ^= 1;
      }
      if (reset_now) {
        LAUNCH(c, k_pcg_reset_a, VB, VT, 0, P.ncs, st + cur, c->x.p, c->sm.p, c->xs.p, c->y.p, zero_ctr);
        const P2pDev pr = p2p ? p2p_next(c) : p2p_none();
        rc = launch_matvec(c, st_done(st + cur), fold_in_a, pr);
        if (rc) return rc;
        LAUNCH(c, k_pcg_reset_bz, VB, VT, 0, P, st + cur, c->y.p, c->sm.p, c->D2.p, c->x.p, c->b.p, c->r.p, c->z2.p, c->Minv_c.p, c->Minv_i.p,
               part_Q, part_rho, ident, fold_rep, pr);
        if (fold_in_a) LAUNCH(c, k_zero_rep_cols, 4, 256, 0, c->rep.p);
      }
    }
    LAUNCH(c, k_pcg_finalize, 1, 32, 0, st + cur, st + (cur ^ 1), part_Q, c->done_flag.p);
    cur ^= 1;
    CUDA_OK(c, cudaMemcpyAsync(c->h_st, st + cur, sizeof(PcgState), cudaMemcpyDeviceToHost, c->stream));
    if (system_ok) CUDA_OK(c, cudaMemcpyAsync(c->h_scal, c->flag.p, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (trace) cudaEventRecord(tev[1], c->stream);
    CUDA_OK(c, cudaStreamSynchronize(c->stream));
    if (trace) { float ms = 0; if (cudaEventElapsedTime(&ms, tev[0], tev[1]) == cudaSuccess) c->trace_pcg_gpu_ms += ms; cudaEventRecord(tev[0], c->stream); }
    if (system_ok) {
      *system_ok = c->h_scal[0] == 0.0;
      if (!*system_ok) { *iters = 0; *status = 0; return TBA_OK; }  // not positive definite: whatever the iterations did is discarded
    }
    if (c->h_st->done) break;
    if (it > o.max_linear_solver_iterations + batch) { set_err(c, "PCG did not terminate"); return TBA_ERR_CUDA; }
    batch = 4;
  }
  if (trace) { cudaEventDestroy(tev[0]); cudaEventDestroy(tev[1]); }
  c->last_cg_iters = c->h_st->iters;
  *iters = c->h_st->iters;
  *status = c->h_st->status;
  c->real_matvecs += c->h_st->iters + (o.cg_residual_reset_period > 0 ? c->h_st->iters / o.cg_residual_reset_period : 0);
  return TBA_OK;
}

// BackSubstitute + model cost change.
int stage_backsub(tba_context* c) {
  DevProblem& P = c->P;
  LAUNCH(c, k_cs_mul, VB, VT, 0, P.ncs, c->sm.p, c->x.p, c->xs.p);
  CUDA_OK(c, cudaMemsetAsync(c->scal2.p, 0, 16 * sizeof(double), c->stream));
  if (P.n_tiles > 0) {
    const int pb_bs = prof_begin(c);
    { const int rc2 = launch_schur(c, 2, c->xs.p, nullptr, nullptr); if (rc2) return rc2; }
    prof_end(c, 5, pb_bs);
    LAUNCH(c, k_fold, 1, REPW, 0, c->rep.p, nullptr, nullptr, c->scal2.p);
  }
  // candidate = x + delta, step norm
  LAUNCH(c, k_candidate_cs, VB, VT, 0, P, c->xs.p, c->scal2.p, c->rank == 0 ? 1 : 0);
  if (P.n_pt > 0) LAUNCH(c, k_candidate_pt, small_grid(c, P.n_pt), 256, 0, P, c->scal2.p);
  return TBA_OK;
}

// Cost at the candidate over every tile, added to scal2[0..2] = [cost, fixed, failed].  profile: record k_cost as span 6.
int launch_candidate_cost(tba_context* c, bool profile) {
  DevProblem& P = c->P;
  if (P.n_tiles == 0) return TBA_OK;
  const int pb = profile ? prof_begin(c) : -1;
  LAUNCH(c, c->ks.cost, P.n_tiles, TILE, 0, P, P.ext_c, P.cam_s4_c, P.intr_c, P.pt_c, c->rep.p);
  prof_end(c, 6, pb);
  LAUNCH(c, k_fold, 1, REPW, 0, c->rep.p, nullptr, nullptr, c->scal2.p);
  return TBA_OK;
}

// Cost at the candidate; scal2 then holds [cost, fixed, failed, mcc, |d_cs|^2, |d_pt|^2].
int stage_evaluate_candidate(tba_context* c, double* cand_cost, double* mcc, double* step_norm, bool* ok, double elapsed_s = 0.0,
                             double* elapsed_collective = nullptr, double* cand_xnorm = nullptr) {
  DevProblem& P = c->P;
  // multi-GPU: every branch of the LM loop must be taken by all ranks alike, the time-out included.  Rank 0's clock is the
  // clock: its elapsed time rides in slot 8 of this all-reduce (the other ranks add 0), so every rank reads the same value.
  if (c->world > 1) LAUNCH(c, k_set_f64, 1, 1, 0, c->scal2.p + 8, c->rank == 0 ? elapsed_s : 0.0);
  LAUNCH(c, k_cam_prep, (P.n_cam + 127) / 128, 128, 0, P.n_cam, P.ext_c, P.cam_rec_c, P.cam_s4_c);
  int rc = launch_candidate_cost(c, true);
  if (rc) return rc;
  // ||candidate|| over the non-constant blocks rides along (slots 6, 7): if the step is accepted it is the ||x|| the next
  // parameter-tolerance test needs -- no separate kernel + all-reduce + host round trip after the acceptance
  if (cand_xnorm) LAUNCH(c, k_xnorm, small_grid(c, std::max(P.n_pt, P.ne)), 256, 0, P, P.ext_c, P.intr_c, P.pt_c, c->blk_free.p, c->scal2.p, c->rank == 0 ? 1 : 0);
  double s[9];
  rc = allreduce_read(c, c->scal2.p, 9, s);
  if (rc) return rc;
  *ok = s[2] == 0.0;
  *cand_cost = s[0];
  *mcc = s[3];
  *step_norm = std::sqrt(s[4] + s[5]);
  if (cand_xnorm) *cand_xnorm = std::sqrt(s[6] + s[7]);
  if (elapsed_collective) *elapsed_collective = c->world > 1 ? s[8] : elapsed_s;
  return TBA_OK;
}

int stage_xnorm(tba_context* c, double* xn) {
  DevProblem& P = c->P;
  CUDA_OK(c, cudaMemsetAsync(c->scal2.p, 0, 16 * sizeof(double), c->stream));
  LAUNCH(c, k_xnorm, small_grid(c, std::max(P.n_pt, P.ne)), 256, 0, P, P.ext, P.intr, P.pt, c->blk_free.p, c->scal2.p, c->rank == 0 ? 1 : 0);
  double s[2];
  const int rc = allreduce_read(c, c->scal2.p + 6, 2, s);
  if (rc) return rc;
  *xn = std::sqrt(s[0] + s[1]);
  return TBA_OK;
}

void accept_candidate(tba_context* c) {
  DevProblem& P = c->P;
  std::swap(P.ext, P.ext_c);
  std::swap(P.intr, P.intr_c);
  std::swap(P.pt, P.pt_c);
  std::swap(P.cam_rec, P.cam_rec_c);
  std::swap(P.cam_s4, P.cam_s4_c);
}

// ---- N4: inner iterations -------------------------------------------------------------------------------
// The candidate buffers seen as "the problem": kernels that read P.ext / P.intr / P.pt / P.cam_rec then work on the candidate.
DevProblem candidate_view(const DevProblem& P) {
  DevProblem Q = P;
  Q.ext = P.ext_c; Q.intr = P.intr_c; Q.pt = P.pt_c; Q.cam_rec = P.cam_rec_c; Q.cam_s4 = P.cam_s4_c;
  return Q;
}

// One independent set (all cameras, or all intrinsics groups) of the coordinate descent: per-block LM state on the host in
// lockstep (tba_block_lm.h), observation passes on the device (k_block_pass).  Works on the candidate buffers in place.
template <int KIND>
int run_block_stage(tba_context* c) {
  DevProblem& P = c->P;
  constexpr int ND = block_dim(KIND), NA = block_acc(KIND);
  const int nb = KIND == kBlockCamera ? P.n_cam : P.n_group;
  if (nb == 0) return TBA_OK;  // (a rank without observations still takes part in the all-reduces below)
  const BlockLmOptions lo;
  const std::vector<double>& mask = c->pack.mask;  // 1 = free coordinate of a block that takes part in the problem
  std::vector<double> vals((size_t)nb * ND);
  double* dev_vals = KIND == kBlockCamera ? P.ext_c : P.intr_c;
  CUDA_OK(c, cudaMemcpyAsync(vals.data(), dev_vals, vals.size() * 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  std::vector<BlockLm> B((size_t)nb);
  std::vector<int> dims((size_t)nb, ND);
  int n_live = 0;
  for (int b = 0; b < nb; ++b) {
    bool fr[kBlkMaxN];
    const int N = KIND == kBlockCamera ? 6 : TBA_MODEL_NUM_PARAMETERS(c->h_group_model[b]);
    dims[b] = N;
    for (int j = 0; j < N; ++j) fr[j] = mask[(KIND == kBlockCamera ? (size_t)b * 6 : (size_t)P.ne + (size_t)b * 10) + j] != 0.0;
    block_lm_init(B[b], N, fr, &vals[(size_t)b * ND], lo);
    n_live += B[b].phase != kBlkDone;
  }
  if (n_live == 0) return TBA_OK;
  const int n_rep = (KIND == kBlockGroup && nb == 1) ? 256 : 1;
  CUDA_OK(c, c->d_blk_vals.alloc((size_t)nb * ND));
  CUDA_OK(c, c->d_blk_active.alloc((size_t)nb));
  CUDA_OK(c, c->d_blk_acc.alloc((size_t)n_rep * nb * NA));
  if (KIND == kBlockCamera) CUDA_OK(c, c->d_blk_rec.alloc((size_t)nb * kCamRec));
  std::vector<double> acc((size_t)n_rep * nb * NA);
  BlockPassArgs A;
  A.ext = KIND == kBlockCamera ? c->d_blk_vals.p : P.ext_c;
  A.rec = KIND == kBlockCamera ? c->d_blk_rec.p : P.cam_rec_c;
  A.intr = KIND == kBlockCamera ? P.intr_c : c->d_blk_vals.p;
  A.pt = P.pt_c;
  A.active = c->d_blk_active.p; A.ext_const = c->d_ext_const.p; A.group_const = c->d_group_mask.p;
  A.acc = c->d_blk_acc.p; A.n_rep = n_rep;
  auto exec = [&](int pass, const std::vector<uint8_t>& active, const std::vector<double>& pv, std::vector<double>& sum) -> int {
    CUDA_OK(c, cudaMemcpyAsync(c->d_blk_vals.p, pv.data(), pv.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(c, cudaMemcpyAsync(c->d_blk_active.p, active.data(), (size_t)nb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(c, cudaMemsetAsync(c->d_blk_acc.p, 0, acc.size() * 8, c->stream));
    if (KIND == kBlockCamera) LAUNCH(c, k_cam_prep, (nb + 127) / 128, 128, 0, nb, c->d_blk_vals.p, c->d_blk_rec.p, (double*)nullptr);
    if (P.n_tiles > 0) LAUNCH(c, c->ks.block_pass[KIND][pass != 0], P.n_tiles, TILE, 0, P, A);
    const int rc = allreduce_sum(c, c->d_blk_acc.p, acc.size());
    if (rc) return rc;
    CUDA_OK(c, cudaMemcpyAsync(acc.data(), c->d_blk_acc.p, acc.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(c, cudaStreamSynchronize(c->stream));
    c->h2d_bytes += (double)pv.size() * 8 + nb; c->d2h_bytes += (double)acc.size() * 8;
    c->inner_passes++;
    std::fill(sum.begin(), sum.end(), 0.0);
    for (int r = 0; r < n_rep; ++r) for (size_t i = 0; i < sum.size(); ++i) sum[i] += acc[(size_t)r * sum.size() + i];  // fixed order
    return TBA_OK;
  };
  {
    const int rc = block_lm_run_lockstep(B, dims, ND, NA, lo, exec);
    if (rc) return rc;
  }
  for (int b = 0; b < nb; ++b) for (int j = 0; j < dims[b]; ++j) vals[(size_t)b * ND + j] = B[b].x[j];
  CUDA_OK(c, cudaMemcpyAsync(dev_vals, vals.data(), vals.size() * 8, cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  return TBA_OK;
}

// CoordinateDescentMinimizer::Minimize on the candidate: extrinsics, then intrinsics groups, then points (Theia's reversed
// ordering, bundle_adjuster.cc:196-200), each block with Ceres' default per-block solver; then the cost there.
int stage_inner_iterations(tba_context* c, double* inner_cost, bool* ok) {
  DevProblem& P = c->P;
  int rc = run_block_stage<kBlockCamera>(c);
  if (rc) return rc;
  LAUNCH(c, k_cam_prep, (P.n_cam + 127) / 128, 128, 0, P.n_cam, P.ext_c, P.cam_rec_c, P.cam_s4_c);
  rc = run_block_stage<kBlockGroup>(c);
  if (rc) return rc;
  if (P.n_pt > 0) {
    PointLmOptions po;
    const BlockLmOptions lo;
    po.loss_type = c->opt.loss_function_type; po.loss_width = c->opt.robust_loss_width; po.max_num_iterations = lo.max_num_iterations;
    po.function_tolerance = lo.function_tolerance; po.gradient_tolerance = lo.gradient_tolerance; po.parameter_tolerance = lo.parameter_tolerance;
    po.initial_radius = lo.initial_radius; po.max_radius = lo.max_radius; po.min_radius = lo.min_radius; po.min_relative_decrease = lo.min_relative_decrease;
    po.min_diag = lo.min_diag; po.max_diag = lo.max_diag; po.jacobi_scaling = 1; po.max_consecutive_invalid = lo.max_consecutive_invalid;
    CUDA_OK(c, c->d_inner_status.alloc((size_t)P.n_pt));  // no-ops: sized at upload
    CUDA_OK(c, c->d_inner_cost2.alloc((size_t)P.n_pt * 2));
    const DevProblem Q = candidate_view(P);
    LAUNCH(c, c->ks.adjust_tracks, (P.n_pt + 63) / 64, 64, 0, Q, c->pt_slot.p, c->pt_len.p, po, c->d_inner_status.p, c->d_inner_cost2.p);
  }
  // cost at the refined candidate
  CUDA_OK(c, cudaMemsetAsync(c->scal2.p, 0, 3 * sizeof(double), c->stream));
  rc = launch_candidate_cost(c, false);
  if (rc) return rc;
  double s3[3];
  rc = allreduce_read(c, c->scal2.p, 3, s3);
  if (rc) return rc;
  *inner_cost = s3[0];
  *ok = s3[2] == 0.0;
  return TBA_OK;
}

// ||x - candidate|| over the non-constant blocks after the inner iterations (ParameterToleranceReached uses it).
int stage_step_norm(tba_context* c, double* step_norm) {
  DevProblem& P = c->P;
  CUDA_OK(c, cudaMemsetAsync(c->scal2.p + 4, 0, 2 * sizeof(double), c->stream));
  LAUNCH(c, k_xdiff, 256, 256, 0, P, c->blk_free.p, c->scal2.p, c->rank == 0 ? 1 : 0);
  double s2[2];
  const int rc = allreduce_read(c, c->scal2.p + 4, 2, s2);
  if (rc) return rc;
  *step_norm = std::sqrt(s2[0] + s2[1]);
  return TBA_OK;
}

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

void push_iter(tba_summary* s, const tba_iteration& it) {
  if (s->iterations && s->num_iterations < s->iterations_capacity) s->iterations[s->num_iterations] = it;
  s->num_iterations++;
}

int check_options(tba_context* c, const tba_options* o) {
  if (o->linear_solver_type < TBA_DENSE_NORMAL_CHOLESKY || o->linear_solver_type > TBA_ITERATIVE_SCHUR) {
    set_err(c, "linear_solver_type %d unsupported: the GPU engine implements ITERATIVE_SCHUR, and the exact solver types (DENSE_NORMAL_CHOLESKY, DENSE_QR, SPARSE_NORMAL_CHOLESKY, DENSE_SCHUR, SPARSE_SCHUR) as the same LM step solved to the fp64 floor; CGNR is not implemented", o->linear_solver_type);
    return TBA_ERR_UNSUPPORTED;
  }
  if (o->linear_solver_type == TBA_ITERATIVE_SCHUR && o->preconditioner_type != TBA_PRECOND_SCHUR_JACOBI && o->preconditioner_type != TBA_PRECOND_IDENTITY) { set_err(c, "preconditioner_type %d unsupported (SCHUR_JACOBI or IDENTITY)", o->preconditioner_type); return TBA_ERR_UNSUPPORTED; }
  if (o->loss_function_type < 0 || o->loss_function_type > 5) { set_err(c, "invalid loss function type %d", o->loss_function_type); return TBA_ERR_INVALID_ARGUMENT; }
  return TBA_OK;
}

// The kernels that depend on the intrinsics column set M.
template <uint32_t M>
void select_mask_kernels(const tba_context* c, KernelSet& k) {
  const bool tred = c->exp_tred;
  if (c->exp_lin_occ) k.linearize = tred ? k_linearize<M, false, true, 3> : k_linearize<M, false, false, 3>;
  else k.linearize = tred ? k_linearize<M, false, true> : k_linearize<M>;
  k.schur[0] = tred ? k_schur<M, 0, true> : k_schur<M, 0, false>;
  k.schur[1] = tred ? k_schur<M, 1, true> : k_schur<M, 1, false>;
  k.schur[2] = k_schur<M, 2, true>;  // back-substitution runs the TRED variant under either TBA_TRED setting
  k.schur_smem = (size_t)(14 + 2 * popcount10(M) + 2) * TILE * sizeof(double);
  k.schur_stream[0] = {k_schur_stream<M, 0>, StreamCfg<M, 0>::NW, StreamCfg<M, 0>::SMEM};
  k.schur_stream[1] = {k_schur_stream<M, 1>, StreamCfg<M, 1>::NW, StreamCfg<M, 1>::SMEM};
  k.schur_stream[2] = {k_schur_stream<M, 2>, StreamCfg<M, 2>::NW, StreamCfg<M, 2>::SMEM};
  k.prepare_stream = {k_prepare_stream<M>, PrepCfg<M>::NW, PrepCfg<M>::SMEM};
  k.precond_ext = tred ? k_precond_ext<M, true> : k_precond_ext<M>;
  k.precond_intr = k_precond_intr<M>;
  k.precond_intr_smem = (size_t)TILE * 4 * popcount10(M) * sizeof(double) + 2 * TILE * sizeof(int);
}

// Fills c->ks for an upload whose intrinsics column set is `imask` and opts its kernels in to the shared memory they launch with.
// The streaming kernels take the leading n_normal_tiles tiles unless TBA_MATVEC=tile or TBA_TRED=0 switched them off.
int select_kernels(tba_context* c, uint32_t imask, int n_normal_tiles) {
  KernelSet& k = c->ks;
  k = KernelSet();
  switch (imask) {  // the sets of kMasks
    case 0x000u: select_mask_kernels<0x000u>(c, k); break;
    case 0x001u: select_mask_kernels<0x001u>(c, k); break;
    case 0x061u: select_mask_kernels<0x061u>(c, k); break;
    case 0x0E1u: select_mask_kernels<0x0E1u>(c, k); break;
    case 0x07Fu: select_mask_kernels<0x07Fu>(c, k); break;
    default: select_mask_kernels<0x3FFu>(c, k); break;
  }
  // FISHEYE / FOV / DIVISION_UNDISTORTION (imask 0x3FF): the dual-number instantiations.  nvcc emits kernel templates in the order
  // of their first reference, and the code generated for the dual-number kernels that share device functions depends on that
  // order: keep k_linearize<0x3FF, true> the first kernel template this file names.
  const bool ext = c->has_ext_models;
  if (ext) k.linearize = k_linearize<0x3FFu, true>;
  k.cost = ext ? k_cost<true> : k_cost<false>;
  k.adjust_tracks = ext ? k_adjust_tracks<true> : k_adjust_tracks<false>;
  k.filter_tracks = ext ? k_filter_tracks<true> : k_filter_tracks<false>;
  k.estimate_tracks = ext ? k_estimate_tracks<true> : k_estimate_tracks<false>;
  k.block_pass[kBlockCamera][0] = ext ? k_block_pass<kBlockCamera, true, false> : k_block_pass<kBlockCamera, false, false>;
  k.block_pass[kBlockCamera][1] = ext ? k_block_pass<kBlockCamera, true, true> : k_block_pass<kBlockCamera, false, true>;
  k.block_pass[kBlockGroup][0] = ext ? k_block_pass<kBlockGroup, true, false> : k_block_pass<kBlockGroup, false, false>;
  k.block_pass[kBlockGroup][1] = ext ? k_block_pass<kBlockGroup, true, true> : k_block_pass<kBlockGroup, false, true>;
  k.n_stream_tiles = c->stream_schur && c->exp_tred ? n_normal_tiles : 0;
  if (c->NI > 0) CUDA_OK(c, cudaFuncSetAttribute(k.precond_intr, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.precond_intr_smem));
  for (int mode = 0; mode < 3; ++mode) {
    CUDA_OK(c, cudaFuncSetAttribute(k.schur[mode], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.schur_smem));
    CUDA_OK(c, cudaFuncSetAttribute(k.schur_stream[mode].fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.schur_stream[mode].smem));
  }
  CUDA_OK(c, cudaFuncSetAttribute(k.prepare_stream.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.prepare_stream.smem));
  return TBA_OK;
}

}  // namespace

// ============================================================================ C-ABI
extern "C" {

void tba_options_init(tba_options* o) {
  memset(o, 0, sizeof *o);
  o->loss_function_type = TBA_LOSS_TRIVIAL; o->robust_loss_width = 2.0;
  o->linear_solver_type = TBA_SPARSE_SCHUR; o->preconditioner_type = TBA_PRECOND_SCHUR_JACOBI;
  o->intrinsics_to_optimize = TBA_INTR_FOCAL_LENGTH | TBA_INTR_RADIAL_DISTORTION;
  o->num_threads = 1; o->max_num_iterations = 100; o->max_solver_time_in_seconds = 3600.0;
  o->use_inner_iterations = 1; o->function_tolerance = 1e-6; o->gradient_tolerance = 1e-10;
  o->parameter_tolerance = 1e-8; o->max_trust_region_radius = 1e12;
  o->initial_trust_region_radius = 1e4; o->min_trust_region_radius = 1e-32; o->min_relative_decrease = 1e-3;
  o->min_lm_diagonal = 1e-6; o->max_lm_diagonal = 1e32; o->eta = 1e-1;
  o->min_linear_solver_iterations = 0; o->max_linear_solver_iterations = 500; o->jacobi_scaling = 1;
  o->max_num_consecutive_invalid_steps = 5; o->cg_residual_reset_period = 10;
}

int tba_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

void tba_abi_sizes(int32_t* out /*[4]*/) {
  out[0] = (int32_t)sizeof(tba_options); out[1] = (int32_t)sizeof(tba_problem);
  out[2] = (int32_t)sizeof(tba_summary); out[3] = (int32_t)sizeof(tba_iteration);
}

int32_t tba_abi_size_two_view_batch(void) { return (int32_t)sizeof(tba_two_view_batch); }

int tba_nccl_unique_id(void* out_128_bytes) {
  std::lock_guard<std::mutex> lk(g_nccl_mu);
  std::string err;
  if (!g_nccl.load(&err)) return TBA_ERR_NCCL;
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return TBA_ERR_NCCL;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  memcpy(out_128_bytes, &id, 128);
  return TBA_OK;
}

int tba_create(int device, int rank, int world_size, const void* nccl_unique_id, tba_context** out) {
  if (!out || world_size < 1 || rank < 0 || rank >= world_size) return TBA_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  int n = tba_device_count();
  if (n <= 0 || device < 0 || device >= n) return TBA_ERR_NO_DEVICE;
  tba_context* c = new tba_context();
  c->device = device; c->rank = rank; c->world = world_size;
  tba_options_init(&c->opt);
  { const char* e = getenv("TBA_MATVEC"); c->stream_schur = !(e != nullptr && e[0] == 't'); }
  { const char* e = getenv("TBA_PCG"); c->pcg_fused = !(e != nullptr && e[0] == 's'); }
#ifdef TBA_EMULATE
  c->pcg_fused = false;  // the emulator runs the CTAs of a launch one after the other: no grid barrier (the three phases are the same device functions)
#endif
  { const char* e = getenv("TBA_P2P"); c->p2p_enabled = !(e != nullptr && e[0] == '0'); }
  // round 2: the transposed RED emission and the 3-CTA/SM linearise are the defaults (driver-measured 28.1 vs 31.9 ms per
  // LM iteration at 20 M observations, costs equal to 2e-8); TBA_TRED=0 / TBA_LIN_OCC=2 select the round-1 kernels
  { const char* e = getenv("TBA_LIN_OCC"); c->exp_lin_occ = !(e != nullptr && e[0] == '2'); }
  { const char* e = getenv("TBA_TRED"); c->exp_tred = !(e != nullptr && e[0] == '0'); }
  if (cudaSetDevice(device) != cudaSuccess || cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaMallocHost(&c->h_scal, 64 * sizeof(double)) != cudaSuccess || cudaMallocHost(&c->h_st, sizeof(PcgState)) != cudaSuccess) {
    delete c;
    return TBA_ERR_CUDA;
  }
  if (world_size > 1) {
    {
      // the lock covers only the dlopen: ncclCommInitRank blocks until every rank has called it, and the ranks of a
      // single-process multi-GPU group (tba_solve_multi) call tba_create concurrently from their own threads
      std::lock_guard<std::mutex> lk(g_nccl_mu);
      std::string err;
      if (!nccl_unique_id || !g_nccl.load(&err)) { tba_destroy(c); return TBA_ERR_NCCL; }
    }
    ncclUniqueId id;
    memcpy(&id, nccl_unique_id, 128);
    if (g_nccl.CommInitRank(&c->comm, world_size, id, rank) != ncclSuccess) { c->comm = nullptr; tba_destroy(c); return TBA_ERR_NCCL; }
  }
  *out = c;
  return TBA_OK;
}

void tba_destroy(tba_context* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  p2p_release(c);
  if (c->comm) g_nccl.CommDestroy(c->comm);
  if (c->stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); }
  if (c->h_scal) cudaFreeHost(c->h_scal);
  if (c->h_st) cudaFreeHost(c->h_st);
  if (c->stage) cudaFreeHost(c->stage);
  delete c;
}

const char* tba_last_error(tba_context* c) { return c ? c->err.c_str() : "null context"; }

void tba_shard_points(const int32_t* pt_num_obs, int32_t n_pt, int world_size, int rank, int32_t* begin, int32_t* end) {
  int64_t total = 0;
  for (int32_t i = 0; i < n_pt; ++i) total += pt_num_obs[i];
  auto cut = [&](int r) -> int32_t {
    if (r <= 0) return 0;
    if (r >= world_size) return n_pt;
    const int64_t target = total * r / world_size;
    int64_t cum = 0;
    for (int32_t i = 0; i < n_pt; ++i) { if (cum >= target) return i; cum += pt_num_obs[i]; }
    return n_pt;
  };
  *begin = cut(rank);
  *end = cut(rank + 1);
}

// --------------------------------------------------------------------------- upload / pack
int tba_upload(tba_context* c, const tba_options* options, const tba_problem* p) {
  if (!c || !options || !p) return TBA_ERR_INVALID_ARGUMENT;
  const double t0 = now_s();
  c->uploaded = false;
  int rc = check_options(c, options);
  if (rc) return rc;
  CUDA_OK(c, cudaSetDevice(c->device));
  c->opt = *options;
  if (options->linear_solver_type != TBA_ITERATIVE_SCHUR) {
    // Every factorising solver type (DENSE_QR / *_NORMAL_CHOLESKY on the full normal equations, *_SCHUR on the reduced
    // system) computes the SAME Levenberg-Marquardt step exactly; Schur elimination is an exact algebraic rewrite of it.
    // The exact Schur solver types (Theia's default, and what SetBundleAdjustmentOptions picks below 1000 views:
    // reconstruction_estimator_utils.cc:110-133) solve the SAME reduced system a Cholesky factorisation of S solves;
    // here it is solved by the preconditioned CG run until the quadratic model stops changing at fp64 resolution.
    c->opt.eta = 1e-13;
    c->opt.min_linear_solver_iterations = 0;
    c->opt.max_linear_solver_iterations = std::max(c->opt.max_linear_solver_iterations, 2000);
    c->opt.preconditioner_type = TBA_PRECOND_SCHUR_JACOBI;
  }
  const int nc = p->n_cam, ng = p->n_group, np = p->n_pt;
  const int64_t no = p->n_obs;
  if (nc < 0 || ng < 0 || np < 0 || no < 0) { set_err(c, "negative sizes"); return TBA_ERR_INVALID_ARGUMENT; }
  c->has_ext_models = false;
  for (int g = 0; g < ng; ++g) {
    if (TBA_MODEL_NUM_PARAMETERS(p->group_model[g]) < 0) {
      set_err(c, "camera intrinsics model %d of group %d is not a CameraIntrinsicsModelType (0..4)", p->group_model[g], g);
      return TBA_ERR_UNSUPPORTED;
    }
    if (p->group_model[g] >= TBA_MODEL_FISHEYE) c->has_ext_models = true;
  }
  for (int i = 0; i < nc; ++i) if (p->cam_group[i] < 0 || p->cam_group[i] >= ng) { set_err(c, "cam_group out of range"); return TBA_ERR_INVALID_ARGUMENT; }
  // ---- host packing (tba_pack.h: phases A-E, multi-threaded), into pinned staging memory
  // host threads of the pack: all hardware threads shared between the ranks of the box, at most 64 per rank
  const int T = std::max(1, std::min<int>(64, (int)std::thread::hardware_concurrency() / std::max(1, c->world)));
  HostPack& H = c->pack;
  c->slot_orig.clear();
  // TBA_UPLOAD_TRACE=1: host wall-clock of the phases of this call on stderr (where the end-to-end time of a solve goes)
  const bool trace = getenv("TBA_UPLOAD_TRACE") != nullptr;
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!trace) return;
    auto t = std::chrono::steady_clock::now();
    fprintf(stderr, "[tba_upload r%d] %-28s %8.2f ms\n", c->rank, what, std::chrono::duration<double, std::milli>(t - t_prev).count());
    t_prev = t;
  };
  pack_count_and_sort(p, T, &H);  // A, B, C
  lap("count_and_sort (A-C)");
  // rank-local validation errors (they depend on this rank's shard of the observations): in process-per-rank mode the
  // failing rank must still take part in the first collective below, where every rank learns about the failure and all
  // return together -- an early return here would leave the other ranks blocked in that all-reduce
  int local_err = TBA_OK;
  if (H.bad >= 0) { set_err(c, "observation %lld references camera %d / point %d out of range", (long long)H.bad, p->obs_cam[H.bad], p->obs_pt[H.bad]); local_err = TBA_ERR_INVALID_ARGUMENT; }
  else if (H.maxlen > TILE) { set_err(c, "track with %d observations exceeds the engine limit of %d per track", H.maxlen, TILE); local_err = TBA_ERR_UNSUPPORTED; }
  const bool collective_upload = c->world > 1 && c->preset_cnt_cam == nullptr;
  if (local_err != TBA_OK && !collective_upload) return local_err;
  if (local_err == TBA_OK) pack_points(p, &H);
  lap("pack_points");
  // ---- which blocks take part (blocks without residuals are not in the Ceres program)
  std::vector<double> cnt_c(nc, 0.0), cnt_g(ng, 0.0);
  if (local_err == TBA_OK) for (int i = 0; i < nc; ++i) { cnt_c[i] = H.cnt_cam[i]; cnt_g[p->cam_group[i]] += H.cnt_cam[i]; }
  c->n_free_pt = local_err == TBA_OK ? H.n_free_pt : 0;
  c->n_free_pt_global = c->n_free_pt;
  if (c->world > 1 && c->preset_cnt_cam != nullptr) {  // single-process multi-GPU: the caller counted over the whole problem
    std::fill(cnt_g.begin(), cnt_g.end(), 0.0);
    for (int i = 0; i < nc; ++i) { cnt_c[i] = c->preset_cnt_cam[i]; cnt_g[p->cam_group[i]] += cnt_c[i]; }
    c->n_free_pt_global = c->preset_free_pt;
  } else if (c->world > 1) {  // counts are global properties
    std::vector<double> tmp(cnt_c);
    tmp.insert(tmp.end(), cnt_g.begin(), cnt_g.end());
    tmp.push_back((double)c->n_free_pt);
    tmp.push_back(local_err != TBA_OK ? 1.0 : 0.0);  // number of ranks whose shard failed validation
    rc = allreduce_host(c, tmp.data(), tmp.size());
    if (rc) return rc;
    if (tmp.back() != 0.0) {  // some rank failed: every rank returns an error, nobody is left inside a collective
      if (local_err == TBA_OK) { set_err(c, "upload failed on %d other rank(s) (invalid observation indices or over-long track in their shard)", (int)tmp.back()); return TBA_ERR_INVALID_ARGUMENT; }
      return local_err;
    }
    std::copy(tmp.begin(), tmp.begin() + nc, cnt_c.begin());
    std::copy(tmp.begin() + nc, tmp.begin() + nc + ng, cnt_g.begin());
    c->n_free_pt_global = (int64_t)tmp[tmp.size() - 2];
  }
  pack_masks_and_tiles(p, cnt_c, cnt_g, &H);  // masks, D
  lap("masks_and_tiles (D)");
  const int ne = nc * 6, ncs = ne + ng * 10;
  const std::vector<double>& mask = H.mask;
  const std::vector<double>& blk_free = H.blk_free;
  std::vector<int>& tile_pt_begin = H.tile_pt_begin;
  std::vector<int>& tile_nruns = H.tile_nruns;
  std::vector<uint8_t>& tile_flags = H.tile_flags;
  c->n_free_cs = H.n_free_cs;
  const uint32_t imask = c->has_ext_models ? 0x3FFu : intrinsics_mask(H.union_free);  // other models: every intrinsics column stored
  c->NI = popcount10(imask);
  c->NJ = 14 + 2 * c->NI;
  const int npk = (int)H.pk2caller.size();
  const int n_long = H.n_long;
  const int n_tiles = H.n_tiles;
  const int64_t n_slots = H.n_slots;
  // E: fill the slot arrays (pinned staging), parallel over packed points
  const size_t stage_bytes = (size_t)n_slots * (4 + 4 + 2 + 1 + 16) + (size_t)npk * (32 + 1 + 8 + 4) + 10 * 256;
  if (c->stage_cap < stage_bytes) {
    if (c->stage) cudaFreeHost(c->stage);
    c->stage = nullptr; c->stage_cap = 0;
    CUDA_OK(c, cudaMallocHost(&c->stage, stage_bytes + stage_bytes / 8));
    c->stage_cap = stage_bytes + stage_bytes / 8;
  }
  uint8_t* sp8 = (uint8_t*)c->stage;
  auto carve = [&](size_t bytes) { uint8_t* r0 = sp8; sp8 += (bytes + 255) / 256 * 256; return r0; };
  double* h_xy = (double*)carve((size_t)n_slots * 16);
  double* h_pt = (double*)carve((size_t)npk * 32);
  int* h_slot_cam = (int*)carve((size_t)n_slots * 4);
  int* h_slot_pt = (int*)carve((size_t)n_slots * 4);
  int16_t* h_slot_run = (int16_t*)carve((size_t)n_slots * 2);
  uint8_t* h_slot_flags = carve((size_t)n_slots);
  uint8_t* h_pt_const = carve((size_t)npk);
  long long* h_pt_slot = (long long*)carve((size_t)npk * 8);
  int* h_pt_len = (int*)carve((size_t)npk * 4);
  lap("staging");
  PackDest d;
  d.xy = h_xy; d.pt = h_pt; d.slot_cam = h_slot_cam; d.slot_pt = h_slot_pt; d.slot_run = h_slot_run; d.slot_flags = h_slot_flags;
  d.pt_const = h_pt_const; d.slot_orig = nullptr;  // not part of the upload (see TBA_VEC_RESIDUALS in tba_debug_read)
  c->n_long_points = n_long;
  // ---- device allocation + H2D
  c->n_cam = nc; c->n_group = ng; c->n_pt = npk; c->n_pt_caller = np; c->n_tiles = n_tiles; c->n_obs = no; c->n_slots = n_slots;
  const int npd = npk;  // points on the device
  c->h2d_bytes = 0; c->d2h_bytes = 0; c->launches = 0;
#define ALLOC(buf, n) CUDA_OK(c, c->buf.alloc(n))
  ALLOC(ext, (size_t)ne); ALLOC(ext_c, (size_t)ne); ALLOC(intr, (size_t)ng * 10); ALLOC(intr_c, (size_t)ng * 10);
  ALLOC(pt, (size_t)npd * 4); ALLOC(pt_c, (size_t)npd * 4); ALLOC(cam_rec, (size_t)nc * kCamRec); ALLOC(cam_rec_c, (size_t)nc * kCamRec); ALLOC(cam_s4, (size_t)nc * 4); ALLOC(cam_s4_c, (size_t)nc * 4);
  ALLOC(xy, (size_t)n_slots * 2); ALLOC(J, (size_t)n_slots * c->NJ); ALLOC(res, (size_t)n_slots * 2);
  ALLOC(Hpp, (size_t)npd * 10); ALLOC(gp, (size_t)npd * 4); ALLOC(Mp, (size_t)npd * 10); ALLOC(sp, (size_t)npd * 4); ALLOC(dpt, (size_t)npd * 4);
  ALLOC(cam_group, (size_t)nc); ALLOC(group_model, (size_t)ng); ALLOC(slot_cam, (size_t)n_slots); ALLOC(slot_pt, (size_t)n_slots);
  ALLOC(tile_pt_begin, (size_t)n_tiles + 1); ALLOC(tile_nruns, (size_t)n_tiles); ALLOC(slot_flags, (size_t)n_slots);
  ALLOC(slot_run, (size_t)n_slots); ALLOC(pt_const, (size_t)npd); ALLOC(tile_flags, (size_t)n_tiles);
  ALLOC(pt_slot, (size_t)npd); ALLOC(pt_len, (size_t)npd); ALLOC(pt_stat, (size_t)npd);
  ALLOC(lin, 2 * (size_t)ncs + 16 + (size_t)std::max(1, c->world)); ALLOC(mask, (size_t)ncs); ALLOC(blk_free, (size_t)nc + ng); ALLOC(sm, (size_t)ncs); ALLOC(D2, (size_t)ncs);
  ALLOC(Sblk, (size_t)nc * 21 + (size_t)ng * 55 + 2 + (size_t)ncs); ALLOC(Minv_c, (size_t)nc * 36); ALLOC(Minv_i, (size_t)ng * 100);
  ALLOC(b, (size_t)ncs); ALLOC(x, (size_t)ncs); ALLOC(r, (size_t)ncs); ALLOC(p, (size_t)ncs); ALLOC(z, (size_t)ncs); ALLOC(z2, (size_t)ncs); ALLOC(xs, (size_t)ncs); ALLOC(y, (size_t)ncs);
  ALLOC(part, 3 * VB); ALLOC(gmax, 2); ALLOC(flag, 1); ALLOC(scal2, std::max<size_t>(16, (size_t)nc + ng)); ALLOC(st, 2); ALLOC(done_flag, 1); ALLOC(pcg_bar, 2); ALLOC(rep, (size_t)NREP * REPW);
#undef ALLOC
  lap("device alloc");
#define H2D(buf, src, n)                                                                                      \
  do {                                                                                                        \
    CUDA_OK(c, cudaMemcpyAsync(c->buf.p, (src), (n) * sizeof(*c->buf.p), cudaMemcpyHostToDevice, c->stream)); \
    c->h2d_bytes += (double)((n) * sizeof(*c->buf.p));                                                        \
  } while (0)
  H2D(ext, p->ext, (size_t)ne); H2D(intr, p->intr, (size_t)ng * 10);
  H2D(ext_c, p->ext, (size_t)ne); H2D(intr_c, p->intr, (size_t)ng * 10);
  H2D(cam_group, p->cam_group, (size_t)nc); H2D(group_model, p->group_model, (size_t)ng);
  H2D(tile_pt_begin, tile_pt_begin.data(), (size_t)n_tiles + 1); H2D(tile_nruns, tile_nruns.data(), (size_t)n_tiles);
  H2D(tile_flags, tile_flags.data(), (size_t)n_tiles);
  // the zero fills of the device-only buffers (3.4 GB for J) run on the GPU while the host fills the first chunk below
  CUDA_OK(c, cudaMemsetAsync(c->rep.p, 0, (size_t)NREP * REPW * sizeof(double), c->stream));
  CUDA_OK(c, cudaMemsetAsync(c->pcg_bar.p, 0, 2 * sizeof(int), c->stream));
  CUDA_OK(c, cudaMemsetAsync(c->J.p, 0, (size_t)n_slots * c->NJ * sizeof(double), c->stream));
  CUDA_OK(c, cudaMemsetAsync(c->dpt.p, 0, (size_t)npd * 4 * sizeof(double), c->stream));
  CUDA_OK(c, cudaMemsetAsync(c->Mp.p, 0, (size_t)npd * 10 * sizeof(double), c->stream));
  CUDA_OK(c, cudaMemsetAsync(c->Hpp.p, 0, (size_t)npd * 10 * sizeof(double), c->stream));
  CUDA_OK(c, cudaMemsetAsync(c->gp.p, 0, (size_t)npd * 4 * sizeof(double), c->stream));
  CUDA_OK(c, cudaMemsetAsync(c->Minv_c.p, 0, (size_t)nc * 36 * sizeof(double), c->stream));
  CUDA_OK(c, cudaMemsetAsync(c->Minv_i.p, 0, (size_t)ng * 100 * sizeof(double), c->stream));
  {
    // E: fill the slot arrays in pinned staging memory chunk by chunk (all host threads per chunk) and send every chunk on its
    // way as soon as it is filled: the copy of chunk k overlaps the filling of chunk k + 1
    int n_chunks = n_tiles >= 32768 ? 16 : n_tiles >= 8192 ? 8 : 1;  // (the last chunk's copy is what the final synchronisation waits for)
    if (const char* e = getenv("TBA_UPLOAD_CHUNKS")) n_chunks = std::max(1, std::min(atoi(e), std::max(1, n_tiles)));  // tests: small scenes too
#define H2D_RANGE(buf, src, off, n)                                                                                              \
  do {                                                                                                                           \
    if ((n) > 0) {                                                                                                               \
      CUDA_OK(c, cudaMemcpyAsync(c->buf.p + (off), (src) + (off), (n) * sizeof(*c->buf.p), cudaMemcpyHostToDevice, c->stream));  \
      c->h2d_bytes += (double)((n) * sizeof(*c->buf.p));                                                                         \
    }                                                                                                                            \
  } while (0)
    for (int ch = 0; ch < n_chunks; ++ch) {
      const int64_t t0 = (int64_t)n_tiles * ch / n_chunks, t1 = (int64_t)n_tiles * (ch + 1) / n_chunks;
      if (t1 <= t0) continue;
      pack_fill(p, H, T, d, t0, t1);
      const size_t s0 = (size_t)t0 * TILE, ns = (size_t)(t1 - t0) * TILE;
      const size_t q0 = (size_t)tile_pt_begin[t0], nq = (size_t)tile_pt_begin[t1] - q0;
      H2D_RANGE(slot_cam, h_slot_cam, s0, ns); H2D_RANGE(slot_pt, h_slot_pt, s0, ns);
      H2D_RANGE(slot_flags, h_slot_flags, s0, ns); H2D_RANGE(slot_run, h_slot_run, s0, ns);
      H2D_RANGE(xy, h_xy, s0 * 2, ns * 2);
      H2D_RANGE(pt, h_pt, q0 * 4, nq * 4); H2D_RANGE(pt_const, h_pt_const, q0, nq);
    }
#undef H2D_RANGE
    // the candidate copy of the points starts as a device-to-device copy (one trip over PCIe instead of two)
    if (npd > 0) CUDA_OK(c, cudaMemcpyAsync(c->pt_c.p, c->pt.p, (size_t)npd * 4 * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  }
  lap("fill (E) + H2D enqueue");
  parallel_for(npd, T, [&](int64_t k0, int64_t k1, int) {
    for (int64_t k = k0; k < k1; ++k) { h_pt_slot[k] = (long long)H.pt_slot[k]; h_pt_len[k] = H.cnt_pt[H.pk2caller[k]]; }
  });
  H2D(pt_slot, h_pt_slot, (size_t)npd); H2D(pt_len, h_pt_len, (size_t)npd);
  H2D(mask, mask.data(), (size_t)ncs); H2D(blk_free, blk_free.data(), (size_t)nc + ng);
#undef H2D
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  lap("tail + stream sync");
  DevProblem& P = c->P;
  P.n_cam = nc; P.n_group = ng; P.n_pt = npd; P.n_tiles = n_tiles; P.ne = ne; P.ncs = ncs; P.single_group = ng == 1;
  P.loss_type = options->loss_function_type; P.loss_width = options->robust_loss_width;
  P.ext = c->ext.p; P.intr = c->intr.p; P.pt = c->pt.p; P.ext_c = c->ext_c.p; P.intr_c = c->intr_c.p; P.pt_c = c->pt_c.p;
  P.cam_group = c->cam_group.p; P.group_model = c->group_model.p; P.cam_rec = c->cam_rec.p; P.cam_rec_c = c->cam_rec_c.p; P.cam_s4 = c->cam_s4.p; P.cam_s4_c = c->cam_s4_c.p;
  P.slot_cam = c->slot_cam.p; P.slot_pt = c->slot_pt.p; P.slot_flags = c->slot_flags.p; P.slot_run = c->slot_run.p;
  P.tile_pt_begin = c->tile_pt_begin.p; P.tile_nruns = c->tile_nruns.p; P.tile_flags = c->tile_flags.p; P.xy = c->xy.p; P.J = c->J.p; P.res = c->res.p;
  P.Hpp = c->Hpp.p; P.gp = c->gp.p; P.Mp = c->Mp.p; P.sp = c->sp.p; P.dpt = c->dpt.p; P.pt_const = c->pt_const.p;
  { const char* e = getenv("TBA_ABLATE"); P.ablate = e ? atoi(e) : 0; }  // timing diagnostics only (wrong results): see k_schur
  int n_normal_tiles = 0;  // tiles whose tracks fit a warp slice (they precede the long tiles)
  for (int t = 0; t < n_tiles; ++t) n_normal_tiles += (tile_flags[t] & 1) ? 0 : 1;
  rc = select_kernels(c, imask, n_normal_tiles);
  if (rc) return rc;
  {
    // multi-GPU: peer-memory inbox for the fused matvec + all-reduce; used only if EVERY rank runs its whole shard through the
    // streaming kernel (a rank with long tiles or without tiles would not push) -- agreed on collectively, here
    rc = p2p_setup(c, ncs);
    if (rc) return rc;
    c->p2p_use = false;
    if (c->world > 1 && c->p2p_ok) {
      double n_pushless = (c->ks.n_stream_tiles > 0 && c->ks.n_stream_tiles == n_tiles) ? 0.0 : 1.0;  // ranks that would not push
      rc = allreduce_host(c, &n_pushless, 1);
      if (rc) return rc;
      c->p2p_use = n_pushless == 0.0;
    }
  }
  c->have_scale = false;
  if (c->opt.use_inner_iterations) {
    c->h_ext_const.assign(p->ext_const, p->ext_const + nc);
    c->h_group_mask.assign(p->group_const_mask, p->group_const_mask + ng);
    c->h_group_model.assign(p->group_model, p->group_model + ng);
    CUDA_OK(c, c->d_ext_const.alloc((size_t)nc)); CUDA_OK(c, c->d_group_mask.alloc((size_t)ng));
    // every buffer the inner iterations use is allocated here, never inside tba_minimize (no cudaMalloc between collectives)
    CUDA_OK(c, c->d_blk_vals.alloc(std::max((size_t)nc * 6, (size_t)ng * 10)));
    CUDA_OK(c, c->d_blk_active.alloc((size_t)std::max(nc, ng)));
    CUDA_OK(c, c->d_blk_rec.alloc((size_t)nc * kCamRec));
    CUDA_OK(c, c->d_blk_acc.alloc(std::max((size_t)nc * block_acc(kBlockCamera), (size_t)(ng == 1 ? 256 : 1) * ng * block_acc(kBlockGroup))));
    CUDA_OK(c, c->d_inner_status.alloc((size_t)c->n_pt));
    CUDA_OK(c, c->d_inner_cost2.alloc((size_t)c->n_pt * 2));
    CUDA_OK(c, cudaMemcpyAsync(c->d_ext_const.p, p->ext_const, (size_t)nc, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(c, cudaMemcpyAsync(c->d_group_mask.p, p->group_const_mask, (size_t)ng * 4, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(c, cudaStreamSynchronize(c->stream));
  }
  c->uploaded = true;
  c->setup_seconds = now_s() - t0;
  return TBA_OK;
}

int tba_download(tba_context* c, tba_problem* p) {
  if (!c || !p || !c->uploaded) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  if (p->n_cam != c->n_cam || p->n_group != c->n_group || p->n_pt != c->n_pt_caller) { set_err(c, "download: problem shape differs from the uploaded one"); return TBA_ERR_INVALID_ARGUMENT; }
  // packed points come back through the pinned staging buffer of the upload (idle by now), then scatter to caller order
  std::vector<double> ptk_fallback;
  double* ptk = reinterpret_cast<double*>(c->stage);
  if (c->stage == nullptr || c->stage_cap < (size_t)c->n_pt * 32) { ptk_fallback.resize((size_t)c->n_pt * 4); ptk = ptk_fallback.data(); }
  CUDA_OK(c, cudaMemcpyAsync(p->ext, c->P.ext, (size_t)c->n_cam * 6 * 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(p->intr, c->P.intr, (size_t)c->n_group * 10 * 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(ptk, c->P.pt, (size_t)c->n_pt * 4 * 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  {
    const int T = std::max(1, std::min<int>(16, (int)std::thread::hardware_concurrency() / std::max(1, c->world)));
    const int* pk2caller = c->pack.pk2caller.data();
    double* dst = p->pt;
    parallel_for(c->n_pt, T, [=](int64_t b0, int64_t e0, int) {
      for (int64_t k = b0; k < e0; ++k) memcpy(dst + (size_t)pk2caller[k] * 4, ptk + (size_t)k * 4, 32);
    });
  }
  c->d2h_bytes += (double)c->n_cam * 48 + (double)c->n_group * 80 + (double)c->n_pt * 32;
  return TBA_OK;
}

// --------------------------------------------------------------------------- minimise
int tba_minimize(tba_context* c, tba_summary* s) {
  if (!c || !s || !c->uploaded) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  const tba_options& opt = c->opt;
  tba_iteration* itbuf = s->iterations;
  const int itcap = s->iterations_capacity;
  memset(s, 0, sizeof *s);
  s->iterations = itbuf; s->iterations_capacity = itcap;
  s->setup_time_in_seconds = c->setup_seconds;
  const double t1 = now_s();
  const int64_t launches0 = c->launches;
  cudaEvent_t ev0, ev1;
  CUDA_OK(c, cudaEventCreate(&ev0));
  CUDA_OK(c, cudaEventCreate(&ev1));
  int term = TBA_NO_CONVERGENCE;
  const char* msg = "";
  int rc = TBA_OK;
  double radius = opt.initial_trust_region_radius, decrease_factor = 2.0;
  double x_cost = 0, fixed = 0, xn = 0;
  bool ok = true;
  tba_iteration it;
  memset(&it, 0, sizeof it);
  int consecutive_invalid = 0;
  double elapsed = 0.0;  // collective view of the solver time (see the time-out test below)
  bool inner_enabled = opt.use_inner_iterations != 0;
  const double kInnerIterationTolerance = 1e-3;  // ceres::Solver::Options::inner_iteration_tolerance
  // TBA_TRACE_LM=1: host wall clock per stage (stream synchronised after each stage, which costs a little itself) on stderr at the
  // end of the call -- against the device times of tba_get_profile_stages this shows the launch / synchronisation / collective
  // overhead of each stage
  const bool trace = getenv("TBA_TRACE_LM") != nullptr;
  static const char* const kStageName[8] = {"linearize", "prepare", "pcg", "backsub", "evaluate", "accept+xnorm", "inner", "bookkeeping"};
  double tr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  double t_prev = now_s();
#define RCT(k, expr) do { rc = (expr); if (rc) goto fail; if (trace) { cudaStreamSynchronize(c->stream); const double t_now = now_s(); tr[k] += t_now - t_prev; t_prev = t_now; } } while (0)
  cudaEventRecord(ev0, c->stream);
  RCT(0, stage_linearize(c, &x_cost, &fixed, &ok, &it.gradient_max_norm));
  if (!ok) { term = TBA_FAILURE; msg = "Residual and Jacobian evaluation failed."; s->initial_cost = s->final_cost = -1; goto done; }
  s->initial_cost = x_cost + fixed;
  if (c->n_free_cs == 0 && c->n_free_pt_global == 0) {
    term = TBA_CONVERGENCE; msg = "Function tolerance reached. No non-constant parameter blocks found.";
    it.iteration = 0; it.cost = x_cost + fixed; it.step_is_valid = 1; it.step_is_successful = 1;
    push_iter(s, it);
    s->num_successful_steps = 1;
    s->final_cost = x_cost + fixed;
    goto done;
  }
  RCT(5, stage_xnorm(c, &xn));
  it.iteration = 0; it.step_is_valid = 1; it.step_is_successful = 1; it.cost = x_cost + fixed; it.trust_region_radius = radius;
  for (;;) {
    // FinalizeIterationAndCheckIfMinimizerCanContinue
    if (it.step_is_successful) s->num_successful_steps++; else s->num_unsuccessful_steps++;
    it.trust_region_radius = radius;
    cudaEventRecord(ev1, c->stream);
    cudaEventSynchronize(ev1);
    { float ms = 0; cudaEventElapsedTime(&ms, ev0, ev1); it.iteration_time_in_seconds = ms * 1e-3; }
    push_iter(s, it);
    if (opt.verbose && c->rank == 0)
      fprintf(stderr, "tba % 4d: f:% 3.12e d:% 3.2e g:% 3.2e h:% 3.2e rho:% 3.2e mu:% 3.2e li:% 3d t:% 3.2e\n", it.iteration, it.cost,
              it.cost_change, it.gradient_max_norm, it.step_norm, it.relative_decrease, it.trust_region_radius,
              it.linear_solver_iterations, it.iteration_time_in_seconds);
    // world > 1: `elapsed` is rank 0's clock as seen by every rank through the last candidate evaluation (a rank-local clock
    // here would let one rank leave the loop while the others enter the next iteration's all-reduces: deadlock)
    if ((c->world > 1 ? elapsed : now_s() - t1) > opt.max_solver_time_in_seconds) { term = TBA_NO_CONVERGENCE; msg = "Maximum solver time reached."; break; }
    if (it.iteration >= opt.max_num_iterations) { term = TBA_NO_CONVERGENCE; msg = "Maximum number of iterations reached."; break; }
    if (it.step_is_successful && it.gradient_max_norm <= opt.gradient_tolerance) { term = TBA_CONVERGENCE; msg = "Gradient tolerance reached."; break; }
    if (radius <= opt.min_trust_region_radius) { term = TBA_CONVERGENCE; msg = "Minimum trust region radius reached."; break; }
    cudaEventRecord(ev0, c->stream);
    const double prev_gmax = it.gradient_max_norm;
    const int prev_iter = it.iteration;
    memset(&it, 0, sizeof it);
    it.iteration = prev_iter + 1;
    // ComputeTrustRegionStep
    bool valid = true;
    int cg_iters = 0, cg_status = 0;
    double mcc = 0, cand = 0, step_norm = 0, cand_xn = -1.0;
    bool cand_ok = true;
    RCT(1, stage_prepare(c, radius, &valid, true));
    if (valid) {
      RCT(2, stage_pcg(c, &cg_iters, &cg_status, &valid));
      if (cg_status == 2) valid = false;
    }
    it.linear_solver_iterations = cg_iters;
    s->num_linear_solver_iterations += cg_iters;
    if (valid) {
      RCT(3, stage_backsub(c));
      RCT(4, stage_evaluate_candidate(c, &cand, &mcc, &step_norm, &cand_ok, now_s() - t1, &elapsed, &cand_xn));
      if (!std::isfinite(mcc) || !std::isfinite(step_norm)) valid = false;
      else valid = mcc > 0.0;
    }
    it.step_is_valid = valid;
    if (!valid) {  // HandleInvalidStep
      if (++consecutive_invalid >= opt.max_num_consecutive_invalid_steps) { term = TBA_FAILURE; msg = "Number of consecutive invalid steps more than Solver::Options::max_num_consecutive_invalid_steps"; break; }
      radius /= decrease_factor; decrease_factor *= 2.0;
      it.cost = x_cost + fixed; it.gradient_max_norm = prev_gmax; it.step_is_successful = 0;
      continue;
    }
    consecutive_invalid = 0;
    if (!cand_ok) cand = 1.7976931348623157e308;
    // DoInnerIterationsIfNeeded (N4)
    bool inner_useful = false, inner_ran = false;
    if (inner_enabled && cand_ok) {
      inner_ran = true;
      double inner_cost = 0;
      bool inner_ok = true;
      RCT(6, stage_inner_iterations(c, &inner_cost, &inner_ok));
      if (inner_ok) {
        mcc += cand - inner_cost;                       // the inner iterations' share is not credited to the trust-region step
        inner_useful = inner_cost < x_cost;
        inner_enabled = (1.0 - inner_cost / cand) > kInnerIterationTolerance;
        cand = inner_cost;
        RCT(6, stage_step_norm(c, &step_norm));
      } else {
        // Ceres returns before adopting inner_iteration_x_: restore the trust-region candidate
        RCT(3, stage_backsub(c));
        RCT(4, stage_evaluate_candidate(c, &cand, &mcc, &step_norm, &cand_ok));
      }
    }
    it.step_norm = step_norm;
    if (it.step_norm <= opt.parameter_tolerance * (xn + opt.parameter_tolerance)) { term = TBA_CONVERGENCE; msg = "Parameter tolerance reached."; break; }
    it.cost_change = x_cost - cand;
    if (std::fabs(it.cost_change) <= opt.function_tolerance * x_cost) { term = TBA_CONVERGENCE; msg = "Function tolerance reached."; break; }
    it.relative_decrease = it.cost_change / mcc;
    if (inner_useful || it.relative_decrease > opt.min_relative_decrease) {  // IsStepSuccessful / HandleSuccessfulStep
      if (trace) { const double t_now = now_s(); tr[7] += t_now - t_prev; t_prev = t_now; }
      accept_candidate(c);
      if (cand_xn >= 0.0 && !inner_ran) xn = cand_xn; else RCT(5, stage_xnorm(c, &xn));  // (the inner iterations move the candidate)
      RCT(0, stage_linearize(c, &x_cost, &fixed, &ok, &it.gradient_max_norm));
      if (!ok) { term = TBA_FAILURE; msg = "Residual and Jacobian evaluation failed."; break; }
      it.cost = x_cost + fixed;
      it.step_is_successful = 1;
      radius = radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * it.relative_decrease - 1.0, 3));
      radius = std::min(opt.max_trust_region_radius, radius);
      decrease_factor = 2.0;
    } else {  // HandleUnsuccessfulStep
      it.step_is_successful = 0; it.gradient_max_norm = prev_gmax;
      radius /= decrease_factor; decrease_factor *= 2.0;
      it.cost = cand + fixed;
    }
  }
  s->final_cost = x_cost + fixed;
done:
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  if (trace) {
    tr[7] += now_s() - t_prev;
    double total = 0;
    for (double v : tr) total += v;
    for (int k = 0; k < 8; ++k) fprintf(stderr, "[tba_minimize r%d] %-14s %9.3f ms  (%5.1f %%)\n", c->rank, kStageName[k], tr[k] * 1e3, 100.0 * tr[k] / std::max(total, 1e-30));
    fprintf(stderr, "[tba_minimize r%d] pcg, device-side span of its launches: %9.3f ms, CG iterations %d\n", c->rank, c->trace_pcg_gpu_ms, (int)s->num_linear_solver_iterations);
    c->trace_pcg_gpu_ms = 0.0;
  }
  s->termination_type = term;
  s->success = term != TBA_FAILURE;
  snprintf(s->message, sizeof s->message, "%s", msg);
  s->solve_time_in_seconds = now_s() - t1;
  s->num_kernel_launches = c->launches - launches0;
  s->h2d_bytes = c->h2d_bytes; s->d2h_bytes = c->d2h_bytes;
  c->x_cost = x_cost; c->fixed_cost = fixed;
  cudaEventDestroy(ev0); cudaEventDestroy(ev1);
  return TBA_OK;
fail:
  cudaEventDestroy(ev0); cudaEventDestroy(ev1);
  s->termination_type = TBA_FAILURE; s->success = 0;
  snprintf(s->message, sizeof s->message, "%s", c->err.c_str());
  return rc;
#undef RC
}

int tba_solve(tba_context* c, const tba_options* options, tba_problem* problem, tba_summary* summary) {
  if (!c || !options || !problem || !summary) return TBA_ERR_INVALID_ARGUMENT;
  int rc = tba_upload(c, options, problem);
  if (rc) { summary->success = 0; summary->termination_type = TBA_FAILURE; snprintf(summary->message, sizeof summary->message, "%s", c->err.c_str()); return rc; }
  rc = tba_minimize(c, summary);
  if (rc) return rc;
  const double t0 = now_s();
  rc = tba_download(c, problem);
  summary->solve_time_in_seconds += now_s() - t0;
  summary->d2h_bytes = c->d2h_bytes;
  return rc;
}

int tba_reset_parameters(tba_context* c, const tba_problem* p) {
  if (!c || !p || !c->uploaded) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  if (p->n_cam != c->n_cam || p->n_group != c->n_group || p->n_pt != c->n_pt_caller) { set_err(c, "reset: problem shape differs from the uploaded one"); return TBA_ERR_INVALID_ARGUMENT; }
  std::vector<double> ptk((size_t)c->n_pt * 4);
  for (int k = 0; k < c->n_pt; ++k) memcpy(&ptk[(size_t)k * 4], p->pt + (size_t)c->pack.pk2caller[k] * 4, 32);
  CUDA_OK(c, cudaMemcpyAsync(c->P.ext, p->ext, (size_t)c->n_cam * 48, cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(c->P.intr, p->intr, (size_t)c->n_group * 80, cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(c->P.pt, ptk.data(), (size_t)c->n_pt * 32, cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(c->P.ext_c, p->ext, (size_t)c->n_cam * 48, cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(c->P.intr_c, p->intr, (size_t)c->n_group * 80, cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(c->P.pt_c, ptk.data(), (size_t)c->n_pt * 32, cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  c->have_scale = false;
  return TBA_OK;
}

int tba_set_max_iterations(tba_context* c, int32_t max_num_iterations) {
  if (!c || max_num_iterations < 0) return TBA_ERR_INVALID_ARGUMENT;
  c->opt.max_num_iterations = max_num_iterations;
  return TBA_OK;
}

int tba_set_profiling(tba_context* c, int enable) {
  if (!c) return TBA_ERR_INVALID_ARGUMENT;
  cudaSetDevice(c->device);
  for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
  c->ev_pool.clear();
  for (auto& v : c->ev_spans) v.clear();
  c->real_matvecs = 0;
  c->profiling = enable != 0;
  return TBA_OK;
}

// out[0] = total ms in the Schur matvec kernel, out[1] = #launches, out[2] = total ms in linearize, out[3] = #launches,
// out[4] = observation slots, out[5] = valid observations, out[6] = packed points, out[7] = doubles stored per observation
int tba_get_profile(tba_context* c, double* out) {
  if (!c || !out) return TBA_ERR_INVALID_ARGUMENT;
  double stages[16];
  const int rc = tba_get_profile_stages(c, stages);
  if (rc) return rc;
  std::copy(stages, stages + 4, out);
  out[4] = (double)c->n_slots; out[5] = (double)c->n_obs; out[6] = (double)c->n_pt; out[7] = (double)c->NJ;
  return TBA_OK;
}

// Per-stage device times of the profiled minimise: out[2k] = total ms, out[2k + 1] = launches for stage k of
// {0 matvec, 1 linearize, 2 precond_ext, 3 precond_intr, 4 reduced rhs, 5 back-substitution, 6 candidate cost,
//  7 fused prepare (rhs + both preconditioner block families in one pass)}.
int tba_get_profile_stages(tba_context* c, double* out) {
  if (!c || !out) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  for (int w = 0; w < 8; ++w) {
    double tot = 0;
    for (auto& sp : c->ev_spans[w]) { float ms = 0; cudaEventElapsedTime(&ms, c->ev_pool[sp.first], c->ev_pool[sp.second]); tot += ms; }
    out[2 * w] = tot; out[2 * w + 1] = (double)c->ev_spans[w].size();
  }
  out[1] = (double)c->real_matvecs;  // early-exited launches (after convergence inside a batch) cost ~2 us and do no work
  return TBA_OK;
}

// --------------------------------------------------------------------------- N1: post-BA track filter
// SetOutlierTracksToUnestimated (set_outlier_tracks_to_unestimated.cc:62-136) on the device-resident problem (after
// tba_minimize / tba_solve on this context): status[q] for every CALLER point q: 0 keep, 1 bad reprojection (negative
// depth in some view, or mean squared reprojection error > max^2), 2 insufficient triangulation angle (also points
// without observations, whose ray list is empty).  mean_sq_error (optional, [n_pt]) receives the per-track mean squared
// reprojection error that ComputeStatisticsForTrack reports (NaN for points without observations).
int tba_filter_tracks(tba_context* c, double max_inlier_reprojection_error, double min_triangulation_angle_degrees,
                      uint8_t* status, double* mean_sq_error, int32_t* num_bad_reprojections, int32_t* num_insufficient_angles) {
  if (!c || !c->uploaded || !status) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  DevProblem& P = c->P;
  const double max_sq = max_inlier_reprojection_error * max_inlier_reprojection_error;
  const double cos_min = std::cos(min_triangulation_angle_degrees * 3.14159265358979323846 / 180.0);
  DevBuf<uint8_t> d_status;
  CUDA_OK(c, d_status.alloc((size_t)P.n_pt));
  // the per-camera rotation records must describe the CURRENT extrinsics
  LAUNCH(c, k_cam_prep, (P.n_cam + 127) / 128, 128, 0, P.n_cam, P.ext, P.cam_rec, P.cam_s4);
  if (P.n_pt > 0) {
    LAUNCH(c, c->ks.filter_tracks, (P.n_pt + 127) / 128, 128, 0, P, c->pt_slot.p, c->pt_len.p, max_sq, cos_min, d_status.p, c->pt_stat.p);
  }
  std::vector<uint8_t> hs((size_t)P.n_pt);
  std::vector<double> hm((size_t)P.n_pt);
  CUDA_OK(c, cudaMemcpyAsync(hs.data(), d_status.p, (size_t)P.n_pt, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(hm.data(), c->pt_stat.p, (size_t)P.n_pt * 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  int nb = 0, ni = 0;
  for (int q = 0; q < c->n_pt_caller; ++q) { status[q] = 2; if (mean_sq_error) mean_sq_error[q] = std::nan(""); }
  for (int k = 0; k < P.n_pt; ++k) { status[c->pack.pk2caller[k]] = hs[k]; if (mean_sq_error) mean_sq_error[c->pack.pk2caller[k]] = hm[k]; }
  for (int q = 0; q < c->n_pt_caller; ++q) { nb += status[q] == 1; ni += status[q] == 2; }
  if (num_bad_reprojections) *num_bad_reprojections = nb;
  if (num_insufficient_angles) *num_insufficient_angles = ni;
  return TBA_OK;
}

// --------------------------------------------------------------------------- N3: batched track estimation / per-track BA
namespace {
PointLmOptions point_lm_options(const tba_options& o) {
  PointLmOptions l;
  l.loss_type = o.loss_function_type; l.loss_width = o.robust_loss_width;
  l.max_num_iterations = o.max_num_iterations;
  l.function_tolerance = o.function_tolerance; l.gradient_tolerance = o.gradient_tolerance; l.parameter_tolerance = o.parameter_tolerance;
  l.initial_radius = o.initial_trust_region_radius; l.max_radius = o.max_trust_region_radius; l.min_radius = o.min_trust_region_radius;
  l.min_relative_decrease = o.min_relative_decrease; l.min_diag = o.min_lm_diagonal; l.max_diag = o.max_lm_diagonal;
  l.jacobi_scaling = o.jacobi_scaling; l.max_consecutive_invalid = o.max_num_consecutive_invalid_steps;
  return l;
}

// D2H of the per-packed-point outputs and scatter to caller order (points without observations are not packed).
int gather_track_outputs(tba_context* c, const uint8_t* d_status, const double* d_cost2, uint8_t fill, uint8_t* status, double* initial_cost,
                         double* final_cost) {
  const int npk = c->P.n_pt;
  std::vector<uint8_t> hs((size_t)npk);
  std::vector<double> hc((size_t)npk * 2);
  if (npk > 0) {
    CUDA_OK(c, cudaMemcpyAsync(hs.data(), d_status, (size_t)npk, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(c, cudaMemcpyAsync(hc.data(), d_cost2, (size_t)npk * 16, cudaMemcpyDeviceToHost, c->stream));
  }
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  for (int q = 0; q < c->n_pt_caller; ++q) {
    status[q] = fill;
    if (initial_cost) initial_cost[q] = -1.0;
    if (final_cost) final_cost[q] = -1.0;
  }
  for (int k = 0; k < npk; ++k) {
    const int q = c->pack.pk2caller[k];
    status[q] = hs[k];
    if (initial_cost) initial_cost[q] = hc[(size_t)2 * k];
    if (final_cost) final_cost[q] = hc[(size_t)2 * k + 1];
  }
  c->d2h_bytes += (double)npk * 17;
  return TBA_OK;
}
}  // namespace

int tba_adjust_tracks(tba_context* c, const tba_options* options, uint8_t* status, double* initial_cost, double* final_cost,
                      int32_t* num_failed) {
  if (!c || !c->uploaded || !options || !status) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  DevProblem& P = c->P;
  DevBuf<uint8_t> d_status;
  DevBuf<double> d_cost2;
  CUDA_OK(c, d_status.alloc((size_t)P.n_pt));
  CUDA_OK(c, d_cost2.alloc((size_t)P.n_pt * 2));
  LAUNCH(c, k_cam_prep, (P.n_cam + 127) / 128, 128, 0, P.n_cam, P.ext, P.cam_rec, P.cam_s4);
  if (P.n_pt > 0) {
    LAUNCH(c, c->ks.adjust_tracks, (P.n_pt + 63) / 64, 64, 0, P, c->pt_slot.p, c->pt_len.p, point_lm_options(*options), d_status.p, d_cost2.p);
  }
  const int rc = gather_track_outputs(c, d_status.p, d_cost2.p, kTrackSkipped, status, initial_cost, final_cost);
  if (rc) return rc;
  int nf = 0;
  for (int q = 0; q < c->n_pt_caller; ++q) nf += status[q] == TBA_FAILURE;
  if (num_failed) *num_failed = nf;
  return TBA_OK;
}

int tba_estimate_tracks(tba_context* c, const tba_options* ba_options, double max_acceptable_reprojection_error_pixels,
                        double min_triangulation_angle_degrees, int32_t bundle_adjustment, uint8_t* status, int32_t counts[5]) {
  if (!c || !c->uploaded || !ba_options || !status) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  DevProblem& P = c->P;
  TrackEstimatorOptions o;
  o.max_sq_reprojection_error = max_acceptable_reprojection_error_pixels * max_acceptable_reprojection_error_pixels;
  o.cos_min_angle = std::cos(min_triangulation_angle_degrees * 3.14159265358979323846 / 180.0);
  o.bundle_adjustment = bundle_adjustment ? 1 : 0;
  o.lm = point_lm_options(*ba_options);
  DevBuf<uint8_t> d_status;
  DevBuf<double> d_cost2;
  CUDA_OK(c, d_status.alloc((size_t)P.n_pt));
  CUDA_OK(c, d_cost2.alloc((size_t)P.n_pt * 2));
  LAUNCH(c, k_cam_prep, (P.n_cam + 127) / 128, 128, 0, P.n_cam, P.ext, P.cam_rec, P.cam_s4);
  // the rays live in the Jacobian store (NJ >= 14 doubles per slot; re-linearised by the next tba_minimize anyway)
  double* ray = P.J;
  if (c->n_slots > 0) LAUNCH(c, k_track_rays, (unsigned)((c->n_slots + 255) / 256), 256, 0, P, (long long)c->n_slots, ray);
  if (P.n_pt > 0) {
    LAUNCH(c, c->ks.estimate_tracks, (P.n_pt + 63) / 64, 64, 0, P, c->pt_slot.p, c->pt_len.p, ray, o, d_status.p, d_cost2.p);
  }
  // caller points without any observation: "view_ids.size() < 2" -> bad angle bucket
  const int rc = gather_track_outputs(c, d_status.p, d_cost2.p, kTrackBadAngle, status, nullptr, nullptr);
  if (rc) return rc;
  if (counts) {
    for (int j = 0; j < 5; ++j) counts[j] = 0;
    for (int q = 0; q < c->n_pt_caller; ++q)
      if (status[q] < 5) ++counts[status[q]];
  }
  return TBA_OK;
}

// --------------------------------------------------------------------------- N3: batched two-view BA
int tba_two_view_ba_batch(tba_context* c, tba_two_view_batch* b, uint8_t* termination, double* initial_cost, double* final_cost,
                          int32_t* iterations) {
  if (!c || !b || !termination || b->n_pairs < 0 || (b->n_pairs > 0 && !b->pair_off)) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  const int np = b->n_pairs;
  if (np == 0) return TBA_OK;
  const int64_t nc = b->pair_off[np];
  bool ext_models = false;
  for (int p = 0; p < np; ++p) {
    if (b->pair_off[p + 1] < b->pair_off[p] || b->pair_off[p] < 0) { set_err(c, "pair_off is not non-decreasing"); return TBA_ERR_INVALID_ARGUMENT; }
    if (TBA_MODEL_NUM_PARAMETERS(b->model1[p]) < 0 || TBA_MODEL_NUM_PARAMETERS(b->model2[p]) < 0) { set_err(c, "unknown camera model in pair %d", p); return TBA_ERR_UNSUPPORTED; }
    ext_models |= b->model1[p] >= TBA_MODEL_FISHEYE || b->model2[p] >= TBA_MODEL_FISHEYE;
  }
  DevBuf<long long> d_off;
  DevBuf<double> d_ext1, d_ext2, d_k1, d_k2, d_xy1, d_xy2, d_pt, d_sp, d_ptc, d_cost2;
  DevBuf<int> d_m1, d_m2, d_it;
  DevBuf<uint8_t> d_c1, d_c2, d_term;
  CUDA_OK(c, d_off.alloc((size_t)np + 1)); CUDA_OK(c, d_ext1.alloc((size_t)np * 6)); CUDA_OK(c, d_ext2.alloc((size_t)np * 6));
  CUDA_OK(c, d_k1.alloc((size_t)np * 10)); CUDA_OK(c, d_k2.alloc((size_t)np * 10)); CUDA_OK(c, d_m1.alloc((size_t)np)); CUDA_OK(c, d_m2.alloc((size_t)np));
  CUDA_OK(c, d_c1.alloc((size_t)np)); CUDA_OK(c, d_c2.alloc((size_t)np)); CUDA_OK(c, d_term.alloc((size_t)np)); CUDA_OK(c, d_cost2.alloc((size_t)np * 2));
  CUDA_OK(c, d_it.alloc((size_t)np));
  CUDA_OK(c, d_xy1.alloc((size_t)nc * 2)); CUDA_OK(c, d_xy2.alloc((size_t)nc * 2)); CUDA_OK(c, d_pt.alloc((size_t)nc * 4));
  CUDA_OK(c, d_sp.alloc((size_t)nc * 4)); CUDA_OK(c, d_ptc.alloc((size_t)nc * 4));
  std::vector<long long> h_off((size_t)np + 1);
  for (int p = 0; p <= np; ++p) h_off[p] = (long long)b->pair_off[p];
#define UP(dst, src, n) do { CUDA_OK(c, cudaMemcpyAsync((dst).p, (src), (size_t)(n) * sizeof(*(dst).p), cudaMemcpyHostToDevice, c->stream)); c->h2d_bytes += (double)((size_t)(n) * sizeof(*(dst).p)); } while (0)
  UP(d_off, h_off.data(), np + 1); UP(d_ext1, b->ext1, np * 6); UP(d_ext2, b->ext2, np * 6); UP(d_k1, b->intr1, np * 10); UP(d_k2, b->intr2, np * 10);
  UP(d_m1, b->model1, np); UP(d_m2, b->model2, np); UP(d_c1, b->constant_intrinsics1, np); UP(d_c2, b->constant_intrinsics2, np);
  UP(d_xy1, b->xy1, nc * 2); UP(d_xy2, b->xy2, nc * 2); UP(d_pt, b->points, nc * 4);
#undef UP
  TwoViewBatchDev B;
  B.n_pairs = np; B.off = d_off.p; B.ext1 = d_ext1.p; B.ext2 = d_ext2.p; B.k1 = d_k1.p; B.k2 = d_k2.p; B.model1 = d_m1.p; B.model2 = d_m2.p;
  B.const1 = d_c1.p; B.const2 = d_c2.p; B.xy1 = d_xy1.p; B.xy2 = d_xy2.p; B.pt = d_pt.p; B.sp = d_sp.p; B.pt_c = d_ptc.p;
  DevBuf<uint8_t> d_inl;
  B.inlier = nullptr; B.sq_max_error = b->final_max_reprojection_error_pixels * b->final_max_reprojection_error_pixels;
  if (b->inlier != nullptr) { CUDA_OK(c, d_inl.alloc((size_t)nc)); B.inlier = d_inl.p; }
  // SetSolverOptions of bundle_adjust_two_views.cc:54-69: everything but the solver type / iteration cap is Ceres' default
  PointLmOptions o;
  o.loss_type = TBA_LOSS_TRIVIAL; o.loss_width = 1.0; o.max_num_iterations = 200;
  o.function_tolerance = 1e-6; o.gradient_tolerance = 1e-10; o.parameter_tolerance = 1e-8;
  o.initial_radius = 1e4; o.max_radius = 1e16; o.min_radius = 1e-32; o.min_relative_decrease = 1e-3; o.min_diag = 1e-6; o.max_diag = 1e32;
  o.jacobi_scaling = 1; o.max_consecutive_invalid = 5;
  {
    auto kfn = ext_models ? k_two_view_ba<true> : k_two_view_ba<false>;
    LAUNCH(c, kfn, (np + 3) / 4, 128, 0, B, o, d_term.p, d_cost2.p, d_it.p);  // 4 warps = 4 pairs per CTA
  }
  std::vector<double> hc((size_t)np * 2);
  std::vector<int> hit((size_t)np);
  CUDA_OK(c, cudaMemcpyAsync(termination, d_term.p, (size_t)np, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(hc.data(), d_cost2.p, (size_t)np * 16, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(hit.data(), d_it.p, (size_t)np * 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(b->ext2, d_ext2.p, (size_t)np * 48, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(b->intr1, d_k1.p, (size_t)np * 80, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(b->intr2, d_k2.p, (size_t)np * 80, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(b->points, d_pt.p, (size_t)nc * 32, cudaMemcpyDeviceToHost, c->stream));
  if (b->inlier != nullptr) CUDA_OK(c, cudaMemcpyAsync(b->inlier, d_inl.p, (size_t)nc, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  c->d2h_bytes += (double)np * (1 + 16 + 4 + 48 + 160) + (double)nc * 32;
  for (int p = 0; p < np; ++p) {
    if (initial_cost) initial_cost[p] = hc[(size_t)2 * p];
    if (final_cost) final_cost[p] = hc[(size_t)2 * p + 1];
    if (iterations) iterations[p] = hit[p];
  }
  return TBA_OK;
}

// Pairs are independent: shard them over the devices of the box, one host thread and one (collective-free) context per device.
namespace {
std::mutex g_tv_mu;
std::vector<tba_context*> g_tv_ctx;
}  // namespace

int tba_two_view_ba_batch_multi(tba_two_view_batch* b, int n_devices, uint8_t* termination, double* initial_cost, double* final_cost,
                                int32_t* iterations) {
  if (!b || !termination || b->n_pairs < 0 || (b->n_pairs > 0 && !b->pair_off)) return TBA_ERR_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> lk(g_tv_mu);
  const int avail = tba_device_count();
  if (avail <= 0) return TBA_ERR_NO_DEVICE;
  if (n_devices <= 0 || n_devices > avail) n_devices = avail;
  n_devices = std::max(1, std::min(n_devices, std::max(b->n_pairs, 1)));
  while ((int)g_tv_ctx.size() < n_devices) {
    tba_context* cx = nullptr;
    const int rc = tba_create((int)g_tv_ctx.size(), 0, 1, nullptr, &cx);
    if (rc != TBA_OK) return rc;
    g_tv_ctx.push_back(cx);
  }
  const int np = b->n_pairs;
  if (np == 0) return TBA_OK;
  // contiguous ranges balanced by correspondence count
  std::vector<int> cut((size_t)n_devices + 1, np);
  cut[0] = 0;
  const int64_t total = b->pair_off[np] - b->pair_off[0];
  for (int d = 1, p = 0; d < n_devices; ++d) {
    const int64_t want = b->pair_off[0] + total * d / n_devices;
    while (p < np && b->pair_off[p] < want) ++p;
    cut[d] = std::max(p, cut[d - 1]);
  }
  std::vector<int> rcs((size_t)n_devices, TBA_OK);
  std::vector<std::thread> th;
  for (int d = 0; d < n_devices; ++d)
    th.emplace_back([&, d] {
      const int p0 = cut[d], p1 = cut[d + 1];
      if (p1 <= p0) return;
      std::vector<int64_t> off((size_t)(p1 - p0) + 1);
      const int64_t base = b->pair_off[p0];
      for (int p = p0; p <= p1; ++p) off[(size_t)(p - p0)] = b->pair_off[p] - base;
      tba_two_view_batch s = *b;
      s.n_pairs = p1 - p0; s.pair_off = off.data();
      s.ext1 = b->ext1 + (size_t)p0 * 6; s.ext2 = b->ext2 + (size_t)p0 * 6;
      s.intr1 = b->intr1 + (size_t)p0 * TBA_INTR_STRIDE; s.intr2 = b->intr2 + (size_t)p0 * TBA_INTR_STRIDE;
      s.model1 = b->model1 + p0; s.model2 = b->model2 + p0;
      s.constant_intrinsics1 = b->constant_intrinsics1 + p0; s.constant_intrinsics2 = b->constant_intrinsics2 + p0;
      s.xy1 = b->xy1 + (size_t)base * 2; s.xy2 = b->xy2 + (size_t)base * 2; s.points = b->points + (size_t)base * 4;
      s.inlier = b->inlier ? b->inlier + (size_t)base : nullptr;
      rcs[d] = tba_two_view_ba_batch(g_tv_ctx[d], &s, termination + p0, initial_cost ? initial_cost + p0 : nullptr,
                                     final_cost ? final_cost + p0 : nullptr, iterations ? iterations + p0 : nullptr);
    });
  for (auto& t : th) t.join();
  for (int d = 0; d < n_devices; ++d) if (rcs[d] != TBA_OK) return rcs[d];
  return TBA_OK;
}

// --------------------------------------------------------------------------- single-process multi-GPU
// The drop-in is called from ONE host thread (Theia's estimators); this entry point shards points + observations over
// n_devices GPUs of the box, runs one rank per device on its own host thread (each with its own context, stream and
// NCCL communicator) and gathers the result.  Contexts are cached for the life of the process.
namespace {
std::mutex g_multi_mu;
std::vector<tba_context*> g_multi_ctx;
}  // namespace

int tba_solve_multi(const tba_options* options, tba_problem* problem, tba_summary* summary, int n_devices) {
  if (!options || !problem || !summary) return TBA_ERR_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> lk(g_multi_mu);
  const int avail = tba_device_count();
  if (avail <= 0) return TBA_ERR_NO_DEVICE;
  if (n_devices <= 0 || n_devices > avail) n_devices = avail;
  if ((int)g_multi_ctx.size() != n_devices) {
    for (tba_context* cx : g_multi_ctx) tba_destroy(cx);
    g_multi_ctx.assign((size_t)n_devices, nullptr);
    unsigned char id[128];
    if (n_devices > 1 && tba_nccl_unique_id(id) != TBA_OK) { g_multi_ctx.clear(); return TBA_ERR_NCCL; }
    std::vector<int> rcs((size_t)n_devices, 0);
    std::vector<std::thread> th;
    for (int r = 0; r < n_devices; ++r) th.emplace_back([&, r] { rcs[r] = tba_create(r, r, n_devices, n_devices > 1 ? id : nullptr, &g_multi_ctx[r]); });
    for (auto& t : th) t.join();
    for (int r = 0; r < n_devices; ++r)
      if (rcs[r] != TBA_OK) { const int e = rcs[r]; for (tba_context* cx : g_multi_ctx) tba_destroy(cx); g_multi_ctx.clear(); return e; }
  }
  if (n_devices == 1) return tba_solve(g_multi_ctx[0], options, problem, summary);
  // shard ranges balanced by observation count
  const int np = problem->n_pt;
  for (int64_t i = 0; i < problem->n_obs; ++i)
    if (problem->obs_pt[i] < 0 || problem->obs_pt[i] >= np) return TBA_ERR_INVALID_ARGUMENT;
  for (int64_t i = 0; i < problem->n_obs; ++i)
    if (problem->obs_cam[i] < 0 || problem->obs_cam[i] >= problem->n_cam) return TBA_ERR_INVALID_ARGUMENT;
  std::vector<int32_t> cnt((size_t)np, 0);
  std::vector<double> cnt_cam((size_t)std::max(problem->n_cam, 1), 0.0);
  for (int64_t i = 0; i < problem->n_obs; ++i) { cnt[problem->obs_pt[i]]++; cnt_cam[problem->obs_cam[i]] += 1.0; }
  int64_t n_free_pt = 0;  // free points that have observations (the only ones in the program)
  for (int q = 0; q < np; ++q) n_free_pt += (cnt[q] > 0 && !problem->pt_const[q]) ? 1 : 0;
  std::mutex bar_mu;
  std::condition_variable bar_cv;
  int bar_count = 0;
  std::atomic<bool> failed(false);
  struct Shard { int32_t b = 0, e = 0; std::vector<double> ext, intr, pt, xy; std::vector<int32_t> cam, ptl; tba_summary s; int rc = 0; };
  std::vector<Shard> sh((size_t)n_devices);
  tba_iteration* itbuf = summary->iterations;
  const int itcap = summary->iterations_capacity;
  std::vector<std::thread> th;
  for (int r = 0; r < n_devices; ++r)
    th.emplace_back([&, r] {
      Shard& S = sh[r];
      tba_shard_points(cnt.data(), np, n_devices, r, &S.b, &S.e);
      S.ext.assign(problem->ext, problem->ext + (size_t)problem->n_cam * 6);
      S.intr.assign(problem->intr, problem->intr + (size_t)problem->n_group * 10);
      S.pt.assign(problem->pt + (size_t)S.b * 4, problem->pt + (size_t)S.e * 4);
      for (int64_t i = 0; i < problem->n_obs; ++i) {
        const int q = problem->obs_pt[i];
        if (q < S.b || q >= S.e) continue;
        S.cam.push_back(problem->obs_cam[i]); S.ptl.push_back(q - S.b);
        S.xy.push_back(problem->obs_xy[2 * i]); S.xy.push_back(problem->obs_xy[2 * i + 1]);
      }
      tba_problem p = *problem;
      p.ext = S.ext.data(); p.intr = S.intr.data(); p.pt = S.pt.data(); p.n_pt = S.e - S.b; p.pt_const = problem->pt_const + S.b;
      p.n_obs = (int64_t)S.cam.size(); p.obs_cam = S.cam.data(); p.obs_pt = S.ptl.data(); p.obs_xy = S.xy.data();
      memset(&S.s, 0, sizeof S.s);
      if (r == 0) { S.s.iterations = itbuf; S.s.iterations_capacity = itcap; }
      // tba_solve split in phases with a host barrier in between: every allocation (cudaMalloc / cudaMallocHost /
      // cudaFree of a grown buffer) of every rank happens while no NCCL kernel of this process is in flight, and a rank
      // whose upload failed keeps the others out of the collectives of tba_minimize
      tba_context* cx = g_multi_ctx[r];
      cx->preset_cnt_cam = cnt_cam.data(); cx->preset_free_pt = n_free_pt;
      S.rc = tba_upload(cx, options, &p);
      cx->preset_cnt_cam = nullptr; cx->preset_free_pt = -1;
      if (S.rc != TBA_OK) { failed.store(true); S.s.termination_type = TBA_FAILURE; snprintf(S.s.message, sizeof S.s.message, "%s", tba_last_error(cx)); }
      {
        std::unique_lock<std::mutex> bl(bar_mu);
        if (++bar_count == n_devices) bar_cv.notify_all();
        else bar_cv.wait(bl, [&] { return bar_count == n_devices; });
      }
      if (failed.load()) { if (S.rc == TBA_OK) S.rc = TBA_ERR_INVALID_ARGUMENT; return; }
      S.rc = tba_minimize(cx, &S.s);
      if (S.rc != TBA_OK) return;
      const double t0 = now_s();
      S.rc = tba_download(cx, &p);
      S.s.solve_time_in_seconds += now_s() - t0;
      S.s.d2h_bytes = cx->d2h_bytes;
    });
  for (auto& t : th) t.join();
  for (int r = 0; r < n_devices; ++r)
    if (sh[r].rc != TBA_OK) { *summary = sh[r].s; summary->iterations = itbuf; summary->iterations_capacity = itcap; return sh[r].rc; }
  memcpy(problem->ext, sh[0].ext.data(), (size_t)problem->n_cam * 48);
  memcpy(problem->intr, sh[0].intr.data(), (size_t)problem->n_group * 80);
  for (int r = 0; r < n_devices; ++r) memcpy(problem->pt + (size_t)sh[r].b * 4, sh[r].pt.data(), (size_t)(sh[r].e - sh[r].b) * 32);
  *summary = sh[0].s;
  for (int r = 1; r < n_devices; ++r) {
    summary->num_kernel_launches += sh[r].s.num_kernel_launches;
    summary->h2d_bytes += sh[r].s.h2d_bytes;
    summary->d2h_bytes += sh[r].s.d2h_bytes;
    summary->setup_time_in_seconds = std::max(summary->setup_time_in_seconds, sh[r].s.setup_time_in_seconds);
    summary->solve_time_in_seconds = std::max(summary->solve_time_in_seconds, sh[r].s.solve_time_in_seconds);
  }
  return TBA_OK;
}

// --------------------------------------------------------------------------- debug / test hooks
// Host-only: run the packing of tba_upload (world = 1) into caller buffers of capacity `cap_slots` slots /
// problem->n_pt points / cap_slots/256 + 1 tiles.  No CUDA call: usable (and tested) without a GPU.
// sizes_out = {n_tiles, n_slots, n_packed_points, n_long_points, NI, imask}.
int tba_debug_pack(const tba_problem* p, int64_t cap_slots, int64_t* sizes_out, int32_t* slot_cam, int32_t* slot_pt, int16_t* slot_run,
                   uint8_t* slot_flags, double* xy, int64_t* slot_orig, int32_t* pk2caller, int32_t* tile_pt_begin,
                   int32_t* tile_nruns, uint8_t* tile_flags, double* mask) {
  if (!p || !sizes_out) return TBA_ERR_INVALID_ARGUMENT;
  for (int i = 0; i < p->n_cam; ++i) if (p->cam_group[i] < 0 || p->cam_group[i] >= p->n_group) return TBA_ERR_INVALID_ARGUMENT;
  // one HostPack reused by every call, like the engine context's (tba_context::pack): the CPU tests, which call this with
  // problems of different shapes back to back, thereby also cover the reuse of its buffers
  static std::mutex mu;
  static HostPack H;
  std::lock_guard<std::mutex> lk(mu);
  pack_count_and_sort(p, 4, &H);
  if (H.bad >= 0) return TBA_ERR_INVALID_ARGUMENT;
  if (H.maxlen > TILE) return TBA_ERR_UNSUPPORTED;
  pack_points(p, &H);
  std::vector<double> cnt_c(p->n_cam, 0.0), cnt_g(p->n_group, 0.0);
  for (int i = 0; i < p->n_cam; ++i) { cnt_c[i] = H.cnt_cam[i]; cnt_g[p->cam_group[i]] += H.cnt_cam[i]; }
  pack_masks_and_tiles(p, cnt_c, cnt_g, &H);
  const uint32_t imask = intrinsics_mask(H.union_free);
  sizes_out[0] = H.n_tiles; sizes_out[1] = H.n_slots; sizes_out[2] = (int64_t)H.pk2caller.size(); sizes_out[3] = H.n_long;
  sizes_out[4] = popcount10(imask); sizes_out[5] = imask;
  if (H.n_slots > cap_slots) return TBA_ERR_INVALID_ARGUMENT;
  std::vector<double> pt((size_t)H.pk2caller.size() * 4);
  std::vector<uint8_t> ptc(H.pk2caller.size());
  for (int64_t s = 0; s < H.n_slots; ++s) slot_orig[s] = -1;
  PackDest d;
  d.xy = xy; d.pt = pt.data(); d.slot_cam = slot_cam; d.slot_pt = slot_pt; d.slot_run = slot_run; d.slot_flags = slot_flags;
  d.pt_const = ptc.data(); d.slot_orig = slot_orig;
  pack_fill(p, H, 4, d);
  for (size_t k = 0; k < H.pk2caller.size(); ++k) pk2caller[k] = H.pk2caller[k];
  for (int t = 0; t <= H.n_tiles; ++t) tile_pt_begin[t] = H.tile_pt_begin[t];
  for (int t = 0; t < H.n_tiles; ++t) { tile_nruns[t] = H.tile_nruns[t]; tile_flags[t] = H.tile_flags[t]; }
  for (size_t i = 0; i < H.mask.size(); ++i) mask[i] = H.mask[i];
  return TBA_OK;
}

int tba_debug_linearize(tba_context* c, double* cost) {
  if (!c || !c->uploaded) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  bool ok;
  double x, f;
  int rc = stage_linearize(c, &x, &f, &ok);
  if (rc) return rc;
  c->x_cost = x; c->fixed_cost = f;
  if (cost) *cost = x + f;
  return ok ? TBA_OK : TBA_ERR_INVALID_ARGUMENT;
}

int tba_debug_prepare_linear_system(tba_context* c, double radius) {
  if (!c || !c->uploaded) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  bool ok;
  int rc = stage_prepare(c, radius, &ok);
  if (rc) return rc;
  return ok ? TBA_OK : TBA_ERR_INVALID_ARGUMENT;
}

int tba_debug_schur_matvec(tba_context* c, const double* x_cam, const double* x_intr, double* y_cam, double* y_intr) {
  if (!c || !c->uploaded) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  DevProblem& P = c->P;
  // y = sm .* S_unscaled (sm .* x) + D2 .* x, using p as the input buffer
  CUDA_OK(c, cudaMemcpyAsync(c->p.p, x_cam, (size_t)P.ne * 8, cudaMemcpyHostToDevice, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(c->p.p + P.ne, x_intr, (size_t)P.n_group * 10 * 8, cudaMemcpyHostToDevice, c->stream));
  LAUNCH(c, k_cs_mul, VB, VT, 0, P.ncs, c->sm.p, c->p.p, c->xs.p);
  CUDA_OK(c, cudaMemsetAsync(c->y.p, 0, (size_t)P.ncs * 8, c->stream));
  LAUNCH(c, k_set_flag, 1, 1, 0, c->done_flag.p, 0);
  int rc = launch_matvec(c, c->done_flag.p);
  if (rc) return rc;
  LAUNCH(c, k_set_flag, 1, 1, 0, const_cast<int*>(st_done(c->st.p)), 0);
  LAUNCH(c, k_pcg_v3, VB, VT, 0, P.ncs, c->st.p, c->y.p, c->sm.p, c->D2.p, c->p.p, c->z.p, c->part.p + VB);
  CUDA_OK(c, cudaMemcpyAsync(y_cam, c->z.p, (size_t)P.ne * 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaMemcpyAsync(y_intr, c->z.p + P.ne, (size_t)P.n_group * 10 * 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_OK(c, cudaStreamSynchronize(c->stream));
  return TBA_OK;
}

int tba_debug_solve_linear_system(tba_context* c, int32_t* cg_iterations, double* model_cost_change) {
  if (!c || !c->uploaded) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  int iters = 0, status = 0;
  int rc = stage_pcg(c, &iters, &status);
  if (rc) return rc;
  rc = stage_backsub(c);
  if (rc) return rc;
  int r2 = allreduce_sum(c, c->scal2.p + 3, 1);
  if (r2) return r2;
  double s[8];
  rc = read_scal(c, c->scal2.p, 8, s);
  if (rc) return rc;
  if (cg_iterations) *cg_iterations = iters;
  if (model_cost_change) *model_cost_change = s[3];
  return status == 2 ? TBA_ERR_INVALID_ARGUMENT : TBA_OK;
}

int tba_debug_evaluate_step(tba_context* c, double* candidate_cost) {
  if (!c || !c->uploaded) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  DevProblem& P = c->P;
  CUDA_OK(c, cudaMemsetAsync(c->scal2.p, 0, 3 * sizeof(double), c->stream));
  LAUNCH(c, k_cam_prep, (P.n_cam + 127) / 128, 128, 0, P.n_cam, P.ext_c, P.cam_rec_c, P.cam_s4_c);
  int rc = launch_candidate_cost(c, false);
  if (rc) return rc;
  double s[3];
  rc = allreduce_read(c, c->scal2.p, 3, s);
  if (rc) return rc;
  if (candidate_cost) *candidate_cost = s[0] + s[1];
  return s[2] == 0.0 ? TBA_OK : TBA_ERR_INVALID_ARGUMENT;
}

int tba_debug_read(tba_context* c, int which, double* out, int64_t n) {
  if (!c || !c->uploaded || !out) return TBA_ERR_INVALID_ARGUMENT;
  CUDA_OK(c, cudaSetDevice(c->device));
  DevProblem& P = c->P;
  const int64_t ne = P.ne, ni = (int64_t)P.n_group * 10, np4 = (int64_t)P.n_pt * 4;
  std::vector<double> tmp, tmp2;
  auto fetch = [&](const double* dev, int64_t len, std::vector<double>& v) -> int {
    v.resize((size_t)len);
    CUDA_OK(c, cudaMemcpyAsync(v.data(), dev, (size_t)len * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(c, cudaStreamSynchronize(c->stream));
    return TBA_OK;
  };
  int rc = TBA_OK;
  switch (which) {
    case TBA_VEC_GRADIENT_CAM: case TBA_VEC_GRADIENT_INTR: case TBA_VEC_COLNORM2_CAM: case TBA_VEC_COLNORM2_INTR: {
      const bool grad = which == TBA_VEC_GRADIENT_CAM || which == TBA_VEC_GRADIENT_INTR;
      const bool cam = which == TBA_VEC_GRADIENT_CAM || which == TBA_VEC_COLNORM2_CAM;
      const int64_t len = cam ? ne : ni;
      if (n != len) return TBA_ERR_INVALID_ARGUMENT;
      if ((rc = fetch((grad ? lin_g(c) : lin_cn(c)) + (cam ? 0 : ne), len, tmp))) return rc;
      if ((rc = fetch(c->mask.p + (cam ? 0 : ne), len, tmp2))) return rc;
      for (int64_t i = 0; i < len; ++i) out[i] = tmp[i] * tmp2[i];
      return TBA_OK; }
    case TBA_VEC_GRADIENT_PT: case TBA_VEC_COLNORM2_PT: case TBA_VEC_STEP_PT: {
      if (n != (int64_t)c->n_pt_caller * 4) return TBA_ERR_INVALID_ARGUMENT;
      std::vector<uint8_t> pc((size_t)P.n_pt);
      CUDA_OK(c, cudaMemcpyAsync(pc.data(), c->pt_const.p, (size_t)P.n_pt, cudaMemcpyDeviceToHost, c->stream));
      memset(out, 0, (size_t)n * 8);
      if (which == TBA_VEC_COLNORM2_PT) {
        if ((rc = fetch(P.Hpp, (int64_t)P.n_pt * 10, tmp))) return rc;
        const int dg[4] = {0, 4, 7, 9};
        for (int64_t k = 0; k < P.n_pt; ++k) for (int j = 0; j < 4; ++j) out[(int64_t)c->pack.pk2caller[k] * 4 + j] = pc[k] ? 0.0 : tmp[k * 10 + dg[j]];
      } else {
        if ((rc = fetch(which == TBA_VEC_GRADIENT_PT ? P.gp : P.dpt, np4, tmp))) return rc;
        for (int64_t k = 0; k < P.n_pt; ++k) for (int j = 0; j < 4; ++j) out[(int64_t)c->pack.pk2caller[k] * 4 + j] = pc[k] ? 0.0 : tmp[k * 4 + j];
      }
      return TBA_OK; }
    case TBA_VEC_RESIDUALS: {
      if (n != c->n_obs * 2) return TBA_ERR_INVALID_ARGUMENT;
      if ((rc = fetch(P.res, c->n_slots * 2, tmp))) return rc;
      if ((int64_t)c->slot_orig.size() != c->n_slots) { c->slot_orig.resize((size_t)c->n_slots); pack_slot_orig(c->pack, 8, c->slot_orig.data()); }
      for (int64_t s = 0; s < c->n_slots; ++s) {
        const int64_t oi = c->slot_orig[s];
        if (oi < 0) continue;
        const int64_t wq = s / 32, l = s % 32;  // [tile][warp][2][32]
        out[2 * oi] = tmp[(size_t)(wq * 2 + 0) * 32 + l];
        out[2 * oi + 1] = tmp[(size_t)(wq * 2 + 1) * 32 + l];
      }
      return TBA_OK; }
    case TBA_VEC_SCHUR_RHS_CAM: if (n != ne) return TBA_ERR_INVALID_ARGUMENT; if ((rc = fetch(c->b.p, ne, tmp))) return rc; break;
    case TBA_VEC_SCHUR_RHS_INTR: if (n != ni) return TBA_ERR_INVALID_ARGUMENT; if ((rc = fetch(c->b.p + ne, ni, tmp))) return rc; break;
    case TBA_VEC_PRECOND_CAM: if (n != (int64_t)P.n_cam * 36) return TBA_ERR_INVALID_ARGUMENT; if ((rc = fetch(c->Minv_c.p, n, tmp))) return rc; break;
    case TBA_VEC_PRECOND_INTR: if (n != (int64_t)P.n_group * 100) return TBA_ERR_INVALID_ARGUMENT; if ((rc = fetch(c->Minv_i.p, n, tmp))) return rc; break;
    case TBA_VEC_STEP_CAM: case TBA_VEC_STEP_INTR: {
      const bool cam = which == TBA_VEC_STEP_CAM;
      const int64_t len = cam ? ne : ni;
      if (n != len) return TBA_ERR_INVALID_ARGUMENT;
      if ((rc = fetch(c->xs.p + (cam ? 0 : ne), len, tmp))) return rc;
      for (int64_t i = 0; i < len; ++i) out[i] = -tmp[i];
      return TBA_OK; }
    default: return TBA_ERR_INVALID_ARGUMENT;
  }
  memcpy(out, tmp.data(), (size_t)n * 8);
  return TBA_OK;
}

}  // extern "C"
