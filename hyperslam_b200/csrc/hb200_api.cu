// libhyperb200.so -- C-ABI (include/hyperb200.h) over the sm_100a kernels.
// Host-side bookkeeping mirrors what the reference's CeresOptimizer keeps in ceres::Problem
// (reference internal/hyper/optimizers/ceres/optimizer.cpp:189-382) but flattened: one set of
// device arrays per variable family and two factor lists.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

#include <cuda_runtime.h>
#include <dlfcn.h>

#include "../../include/hyperb200.h"
#include "hb200_bcr.cuh"
#include "hb200_calib.cuh"
#include "hb200_window.cuh"

using namespace hb;

namespace {

thread_local std::string g_error;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_error = buf;
  return code;
}

#define HB_CUDA(expr)                                                                                   \
  do {                                                                                                  \
    cudaError_t err__ = (expr);                                                                         \
    if (err__ != cudaSuccess) return fail(100 + static_cast<int>(err__), "%s: %s", #expr, cudaGetErrorString(err__)); \
  } while (0)

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) cap = n;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  // capacity for n elements, the first `keep` of them preserved (amortised doubling; device-to-device copy on `stream`)
  cudaError_t grow(size_t n, size_t keep, cudaStream_t stream) {
    if (n <= cap) return cudaSuccess;
    const size_t ncap = std::max<size_t>(n, cap + cap / 2 + 16);
    T* q = nullptr;
    cudaError_t e = cudaMalloc(&q, ncap * sizeof(T));
    if (e != cudaSuccess) return e;
    if (p && keep) e = cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (p) cudaFree(p);
    p = q; cap = ncap;
    return e;
  }
  void swap(DevBuf& o) { std::swap(p, o.p); std::swap(cap, o.cap); }
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }   // scratch buffers of the API calls do not leak on early error returns
};

void compute_basis(Basis* b, int k) {
  // Blending matrix of the uniform B-spline of order k and its cumulative form (DESIGN.md A.3).
  auto binom = [](int n, int r) { double v = 1; if (r < 0 || r > n) return 0.0; for (int i = 1; i <= r; ++i) v = v * (n - r + i) / i; return v; };
  double M[kMaxOrder][kMaxOrder];
  double fact = 1;
  for (int i = 2; i <= k - 1; ++i) fact *= i;
  for (int s = 0; s < k; ++s)
    for (int n = 0; n < k; ++n) {
      double sum = 0;
      for (int l = s; l <= k - 1; ++l) {
        double pw = 1;
        for (int i = 0; i < k - 1 - n; ++i) pw *= static_cast<double>(k - 1 - l);
        sum += ((l - s) % 2 ? -1.0 : 1.0) * binom(k, l - s) * pw;
      }
      M[s][n] = binom(k - 1, n) / fact * sum;
    }
  b->k = k;
  for (int j = 0; j < k; ++j)
    for (int n = 0; n < k; ++n) {
      double s = 0;
      for (int r = j; r < k; ++r) s += M[r][n];
      b->Mc[j * k + n] = s;
    }
}

// ---- NCCL, bound at run time ----------------------------------------------------------------------
// libnccl.so.2 is resolved with dlopen when the first communicator call is made: inside a torch process this is
// the copy torch already loaded (same SONAME), in a plain C++ host the system library.  Only the five entry
// points below are used; their prototypes are those of nccl.h 2.x (ncclUniqueId = 128 bytes by value,
// ncclDouble = 8, ncclSum = 0).
struct NcclUid { char internal[128]; };
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(NcclUid*) = nullptr;
  int (*CommInitRank)(void**, int, NcclUid, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;
int load_nccl() {
  if (g_nccl.lib) return 0;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* nm : names) { h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
  if (!h) return fail(300, "libnccl.so.2 not found: %s", dlerror());
  NcclApi a;
  a.lib = h;
  a.GetUniqueId = reinterpret_cast<int (*)(NcclUid*)>(dlsym(h, "ncclGetUniqueId"));
  a.CommInitRank = reinterpret_cast<int (*)(void**, int, NcclUid, int)>(dlsym(h, "ncclCommInitRank"));
  a.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclCommDestroy"));
  a.AllReduce = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(dlsym(h, "ncclAllReduce"));
  a.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(h, "ncclGetErrorString"));
  if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllReduce || !a.GetErrorString) return fail(300, "libnccl.so.2 lacks an expected symbol");
  g_nccl = a;
  return 0;
}
#define HB_NCCL(expr)                                                                                              \
  do {                                                                                                             \
    const int r__ = (expr);                                                                                        \
    if (r__ != 0) return fail(300 + r__, "%s: %s", #expr, g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "nccl error"); \
  } while (0)

}  // namespace

struct hb200_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  // side stream: the inertial / manifold factor kernels (and their J^T J) are independent of the visual ones and
  // run concurrently with them -- a fork / join inside the iteration (and inside its CUDA graph)
  cudaStream_t stream2 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_mid = nullptr;
  bool forked = false;
  // hb200_optimize on small windows: the five variable blocks travel as ONE pinned staging buffer each way
  double* h_stage = nullptr;
  size_t h_stage_cap = 0;
  DevBuf<double> d_stage;
  bool own_stream = false;
  bool use_graph = true;
  int num_sms = 0;
  long long launches = 0;
  long long launches_per_iteration = 0;
  long long iter_total = 0, snap_iter_total = 0;   // host mirror of SolverState.iteration (record ring index)
  int last_terminated = 0, last_performed = 0;     // outcome of the last hb200_iterate / hb200_optimize that fetched records
  double last_gmax = 0, last_step_norm = 0, last_x_norm = 0;

  // window state (index 0 = current, 1 = trial)
  int k = 0, K = 0, kb = 4, Kbg = 0, Kba = 0, C = 0, L = 0;
  Basis basis{}, bias_basis{};
  DevBuf<double> knots[2], bg[2], ba[2], grav[2], lms[2], tab[2];
  DevBuf<double> cams, imu, cam_tab, imu_tab;
  DevBuf<unsigned char> fixed;
  std::vector<unsigned char> h_knot_const;
  std::vector<double> h_knot_stamp, h_bg_stamp, h_ba_stamp;   // stamps the index maps of hb200_bind were computed from
  int gravity_const = 0, bias_const = 0;
  bool have_imu = false, have_gravity = false;
  double huber = 0.5, imu_scale = 1.6e-5, radius0 = 1e4;
  // ceres::Solver::Options termination tests (off: hb200_iterate runs exactly the requested number of iterations)
  bool term_enabled = false;
  double term_ftol = 1e-6, term_gtol = 1e-10, term_ptol = 1e-8, term_min_radius = 1e-32;

  // factors (host copies in user order; device copies in bound order)
  // visual list = pixel factors [0, Np) followed by bearing factors [Np, Np + Nb): both travel through the
  // same kernels and the same compact layout (kind flag in idx.w); manifold (pose) factors have their own.
  int Nv = 0, Ni = 0, Np = 0, Nb = 0, Nm = 0, P = 0;
  std::vector<double> h_p_stamp, h_p_pixel, h_b_stamp, h_b_bearing, h_m_stamp, h_m_meas, h_sensors;
  std::vector<int> h_p_cam, h_p_lm, h_b_cam, h_b_lm, h_m_sensor;
  std::vector<double> h_v_stamp, h_v_pixel, h_v_z, h_i_stamp, h_i_meas;
  std::vector<int> h_v_cam, h_v_lm;
  DevBuf<double> v_stamp, v_pixel, v_z, v_w, i_stamp, i_meas, m_stamp, m_meas, sensors;
  DevBuf<int> m_sensor;
  DevBuf<int2> m_idx;
  std::vector<int2> h_m_idx;
  double huber_bearing = 1.6e-3;   // reference optimizer.cpp:204
  DevBuf<int> v_cam, v_lm;
  DevBuf<int4> v_idx, i_idx;
  std::vector<int4> h_v_idx, h_i_idx;       // bound order
  std::vector<int> v_perm, i_perm;          // bound position -> user index
  DevBuf<int> seg_off, run_off, lm_off, lm_obs, d_invalid;
  // large windows: landmarks ordered by first knot base and cut into groups for schur_group_kernel
  DevBuf<int> lm_order, lm_group_off;
  int n_lm_groups = 0, schur_rt = 0;
  bool schur_groups = false;
  int nseg = 0, nruns = 0, max_rows = 6;
  int pix_splits = 1, imu_splits = 1, imu_splits_mma = 1;
  int beta = 3, min_beta = 0;   // min_beta: lower bound agreed across ranks (the packed layout must be identical everywhere)
  bool band_solver = true, band_smem = true, force_dense = false;
  DevBuf<double> band_ws;
  int band_chunk_cols = 0;       // !band_smem: block columns per shared-memory chunk view (per chain)
  size_t band_chunk_smem = 0;
  // long windows: multi-CTA block cyclic reduction instead of the single-CTA chain (hb200_bcr.cuh)
  bool use_bcr = false;
  BcrPlan bcr{};
  int bcr_ctas = 0;
  size_t bcr_smem = 0;
  DevBuf<double> bcr_ws;
  DevBuf<unsigned int> bcr_bar;
  DevBuf<long long> band_dbg;   // optional phase timings of band_solve_kernel (HB200_BAND_TIMING=1)
  bool bound = false;

  // device-side window bookkeeping (hb200_append_* / hb200_slide): the factor lists live on the device only, the host
  // mirrors above are refreshed on demand (sync_host_mirrors)
  bool device_managed = false;
  DevBuf<double> alt_stamp, alt_meas, alt_lms, alt_knots, alt_z;
  DevBuf<double2> alt_pixel;
  DevBuf<int4> alt_idx;
  DevBuf<int2> alt_midx;
  DevBuf<int> w_keep, w_pos, w_lkeep, w_lpos, w_cnt, w_scal;
  DevBuf<unsigned long long> w_last;
  // outputs
  DevBuf<double> v_r, v_Jp, v_Jl, i_r, i_Jp, i_wg, i_wa, i_Jg, m_r, m_Jp;
  DevBuf<double> cp_pix[2], cp_imu[2];
  int n_pix_blocks = 0, n_imu_blocks = 0, n_man_blocks = 0;   // manifold cost partials follow the inertial ones in cp_imu
  bool evaluated_J = false;
  // calibration-block Jacobians (on demand, hb200_factor_evaluate) and the reference-quirk switches
  int quirks = 0;
  bool calib_valid = false;
  std::vector<double> m_v_Jc, m_i_Jc, m_m_Jc;   // user order: [Np + Nb][2][14], [Ni][6][36], [Nm][6][6]
  // host mirror for hb200_factor_evaluate
  bool mirror_valid = false;
  std::vector<double> m_v_r, m_v_Jp, m_v_Jl, m_i_r, m_i_Jp, m_i_wg, m_i_wa, m_i_Jg, m_grav, m_b_r, m_b_Jp, m_b_Jl, m_m_r, m_m_Jp;

  // system (band-only packed storage, see SysLayout)
  int n = 0;
  SysLayout lay{};
  DevBuf<double> sys, D, Lw, Ldiag, dp, dl, Vinv, gl, Dl, lm_part, scal;
  DevBuf<int> spd;
  DevBuf<SolverState> st, records;
  int max_records = 64;
  int n_lm_blocks = 0;
  bool system_built = false;

  hb200_allreduce_fn allreduce = nullptr;
  void* allreduce_user = nullptr;
  // multi-GPU: one NCCL all-reduce of the packed system per iteration, enqueued from C on the context's stream
  // (graph-capturable); the step-acceptance scalars travel through peer memory inside accept_kernel
  void* nccl = nullptr;
  bool own_nccl = false;
  long long nccl_calls = 0, nccl_calls_per_iteration = 0;
  int nranks = 1, rank = 0;
  bool comm_warm = false;        // one eager all-reduce has run (NCCL's lazy setup is done: safe to capture)
  DevBuf<double> mbox;           // the peer arena: [mailbox | flags | partial system A | partial system B] (hb200_solve.cuh)
  long long arena_cap = 0;       // doubles per partial
  int peer_par = 0;              // arena half the NEXT iteration assembles into
  bool peer_reduce_wanted = true;
  DevBuf<unsigned long long> red_round;
  DevBuf<unsigned int> red_arrive;
  cudaGraph_t graph_b = nullptr;            // second capture of the iteration (arena half B)
  cudaGraphExec_t graph_exec_b = nullptr;
  bool graph_b_valid = false;
  bool peer_reduce() const { return nccl && peers_open && peer_reduce_wanted && lay.total <= arena_cap; }
  double* assembly() { return peer_reduce() ? mbox.p + kArenaParts + static_cast<long long>(peer_par) * arena_cap : sys.p; }
  DevBuf<unsigned long long> mbox_seq;
  DevBuf<double*> d_peers;
  std::vector<void*> peer_ptrs;  // cudaIpcOpenMemHandle mappings (own entry = mbox.p)
  bool peers_open = false;
  bool multi() const { return nccl != nullptr || allreduce != nullptr; }

  // profiling (hb200_profile_iteration)
  bool profiling = false;
  std::vector<cudaEvent_t> prof_events;
  std::vector<std::string> prof_names;
  size_t prof_used = 0;
  // snapshot
  DevBuf<double> snap_knots, snap_bg, snap_ba, snap_grav, snap_lms;
  DevBuf<SolverState> snap_st;
  bool have_snapshot = false;

  cudaGraph_t graph = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  bool graph_valid = false;

  int o_bg() const { return 6 * K; }
  int o_ba() const { return 6 * K + 3 * Kbg; }
  int o_g() const { return 6 * K + 3 * Kbg + 3 * Kba; }
  void invalidate() { graph_valid = false; system_built = false; evaluated_J = false; mirror_valid = false; calib_valid = false; }
};

namespace {

void prof_mark(hb200_ctx* c, const char* what) {
  if (!c->profiling) return;
  if (c->prof_used == c->prof_events.size()) { cudaEvent_t e; cudaEventCreate(&e); c->prof_events.push_back(e); c->prof_names.emplace_back(); }
  cudaEventRecord(c->prof_events[c->prof_used], c->stream);
  c->prof_names[c->prof_used] = what;
  c->prof_used += 1;
}

int check_launch(hb200_ctx* c, const char* what) {
  c->launches += 1;
  prof_mark(c, what);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(100 + static_cast<int>(e), "launch %s: %s", what, cudaGetErrorString(e));
  return 0;
}

#define HB_LAUNCH(ctx, what)                       \
  do {                                             \
    int rc__ = check_launch(ctx, what);            \
    if (rc__) return rc__;                         \
  } while (0)

// Launch on the context's stream as a PROGRAMMATIC dependent of the previous kernel in that stream: the grid may become
// resident while its predecessor still runs and blocks in pdl_wait() until the predecessor has completed (inside stream
// capture the edge becomes a programmatic graph dependency).  Only for kernels whose sole dependency is that predecessor
// and that call pdl_wait() first.  OFF by default: measured at cfg1 (profiles/r02_experiments.md) the step got slower
// (0.164 vs 0.155 ms) with the four single-dependency edges of the iteration (knot table -> factors, solve ->
// back-substitution -> trial factors -> accept) made programmatic; HB200_PDL=1 switches it on.
template <typename... KArgs, typename... Args>
cudaError_t launch_dependent(hb200_ctx* c, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args&&... args) {
  static const bool off = !(getenv("HB200_PDL") != nullptr && atoi(getenv("HB200_PDL")) != 0);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = c->stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = (off || c->profiling) ? 0 : 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

cudaStream_t side(hb200_ctx* c) { return c->forked ? c->stream2 : c->stream; }
int fork_side(hb200_ctx* c) {
  static const bool no_fork = getenv("HB200_NO_FORK") != nullptr;   // A/B switch for measurements
  if (c->profiling || c->forked || !c->stream2 || no_fork) return 0;   // the per-launch profile wants a serial timeline
  HB_CUDA(cudaEventRecord(c->ev_fork, c->stream));
  HB_CUDA(cudaStreamWaitEvent(c->stream2, c->ev_fork, 0));
  c->forked = true;
  return 0;
}
int join_side(hb200_ctx* c) {
  if (!c->forked) return 0;
  HB_CUDA(cudaEventRecord(c->ev_join, c->stream2));
  HB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
  c->forked = false;
  return 0;
}

int update_fixed(hb200_ctx* c) {
  c->n = 6 * c->K + 3 * c->Kbg + 3 * c->Kba + 2;
  std::vector<unsigned char> f(c->n, 0);
  for (int j = 0; j < c->K && j < static_cast<int>(c->h_knot_const.size()); ++j)
    if (c->h_knot_const[j]) for (int a = 0; a < 6; ++a) f[6 * j + a] = 1;
  if (c->bias_const) for (int a = c->o_bg(); a < c->o_g(); ++a) f[a] = 1;
  if (c->gravity_const) { f[c->o_g()] = 1; f[c->o_g() + 1] = 1; }
  HB_CUDA(c->fixed.ensure(c->n));
  HB_CUDA(cudaMemcpyAsync(c->fixed.p, f.data(), c->n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

// dense work copy of the reduced system: only the dense fallback solver and hb200_get_system need it
int ensure_dense(hb200_ctx* c) {
  const size_t n = c->n;
  const size_t T = (n + kCholNB - 1) / kCholNB;
  HB_CUDA(c->Lw.ensure((T * kCholNB + 1) * n));
  HB_CUDA(c->Ldiag.ensure(T * kCholNB * kCholNB));
  return 0;
}

int ensure_system(hb200_ctx* c) {
  const size_t n = c->n;
  // block half-bandwidth of the reduced pose system = longest landmark track in control points (>= k - 1)
  c->beta = std::max(std::max(c->k - 1, c->max_rows / 6 - 1), c->min_beta);
  c->beta = std::min(c->beta, std::max(c->K - 1, 0));
  c->lay = sys_layout(c->K, c->beta, c->n - 6 * c->K);
  HB_CUDA(c->sys.ensure(static_cast<size_t>(c->lay.total)));
  HB_CUDA(c->D.ensure(n));
  HB_CUDA(c->dp.ensure(n));
  HB_CUDA(c->dl.ensure(3 * static_cast<size_t>(std::max(c->L, 1))));
  HB_CUDA(c->Vinv.ensure(9 * static_cast<size_t>(std::max(c->L, 1))));
  HB_CUDA(c->gl.ensure(3 * static_cast<size_t>(std::max(c->L, 1))));
  HB_CUDA(c->Dl.ensure(3 * static_cast<size_t>(std::max(c->L, 1))));
  c->n_lm_blocks = (c->L + kLmWarps - 1) / kLmWarps;
  HB_CUDA(c->lm_part.ensure(5 * static_cast<size_t>(std::max(c->n_lm_blocks, 1))));
  HB_CUDA(c->scal.ensure(8));
  HB_CUDA(c->spd.ensure(1));
  HB_CUDA(c->records.ensure(c->max_records));
  // solver selection: block-banded + arrowhead unless the band is wide on a large system
  const size_t ws = band_workspace_doubles(c->K, c->beta, c->n - 6 * c->K) * sizeof(double);
  c->band_solver = !c->force_dense && ((c->n <= 512) || (12 * (c->beta + 1) <= 6 * c->K));
  c->band_smem = ws <= 220 * 1024;
  c->use_bcr = false;
  if (c->band_solver && !c->band_smem && 6 * c->beta <= kBcrMaxNb && c->n - 6 * c->K <= 54 && !getenv("HB200_NO_BCR")) {
    // the band does not fit one CTA's shared memory: cyclic reduction over super-blocks of beta control points
    const int m = c->n - 6 * c->K;
    const int nsb = (c->K + c->beta - 1) / c->beta;
    const int nctas = std::max(1, std::min(c->num_sms, (nsb + 1) / 2));
    const BcrPlan pl = bcr_plan(c->K, c->beta, m, nctas);
    const size_t nb = pl.nb;
    const size_t p1 = nb * (nb | 1) + nb + 1 + nb * (((2 * nb + m + 1 + 11) / 16) * 16 + 4) + static_cast<size_t>(m + 1) * m;
    const size_t p2 = 3 * nb * nb + 2 * nb * m + 2 * nb;
    const size_t mp = static_cast<size_t>((m + 5) / 6) * 6;
    const size_t p3 = mp * (mp | 1) + 3 * (mp + 1) + 8;                       // corner: padded matrix, reciprocal diagonal, rhs, solution
    const size_t p4 = nb * static_cast<size_t>(m + 1);                         // corner partials: staged Y_f | y
    const size_t p5 = 2 * (nb + 1) + 2 * nb + m + 2 + nb * (nb | 1);           // way back: rv, x, staged neighbours, L
    const size_t smem = std::max(std::max(p1, p2), std::max(p3, std::max(p4, p5))) * sizeof(double);
    if (smem <= 220 * 1024) {
      if (nctas != c->bcr_ctas || pl.total != c->bcr.total) {
        HB_CUDA(c->bcr_ws.ensure(static_cast<size_t>(pl.total)));
        HB_CUDA(c->bcr_bar.ensure(1));
        HB_CUDA(cudaMemsetAsync(c->bcr_bar.p, 0, sizeof(unsigned int), c->stream));   // the grid-barrier counter stays a multiple of the grid size
      }
      c->bcr = pl; c->bcr_ctas = nctas; c->bcr_smem = smem; c->use_bcr = true;
      HB_CUDA(cudaFuncSetAttribute(bcr_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    }
  }
  if (c->band_solver && !c->use_bcr) {
    if (c->band_smem) HB_CUDA(cudaFuncSetAttribute(band_solve_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ws)));
    else {
      // chunked factorisation: two shared-memory views of band_chunk_cols block columns (band + arrow + LI)
      const size_t colbytes = (static_cast<size_t>(6 + 6 * c->beta) * 6 + 6 * static_cast<size_t>(c->n - 6 * c->K + 1) + 48) * sizeof(double);
      const int fit = static_cast<int>((200 * 1024) / (2 * colbytes));
      c->band_chunk_cols = std::max(c->beta + 2, std::min(fit, c->K + c->beta));
      c->band_chunk_smem = 2 * colbytes * c->band_chunk_cols;
      // the chunk needs beta + 2 block columns: a wide band (landmark tracks of 17+ control points) or a wide arrow
      // leaves no band plan, and the dense cooperative Cholesky solves the window instead
      if (c->band_chunk_smem > 220 * 1024) c->band_solver = false;
      else {
        HB_CUDA(c->band_ws.ensure(ws / sizeof(double)));
        HB_CUDA(cudaFuncSetAttribute(band_solve_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(c->band_chunk_smem)));
      }
    }
  }
  HB_CUDA(c->band_ws.ensure(1));
  if (!c->band_solver) { int rc = ensure_dense(c); if (rc) return rc; }
  if (getenv("HB200_BAND_TIMING")) {
    HB_CUDA(c->band_dbg.ensure(72));
    long long variant = getenv("HB200_BCR_VARIANT") ? atoll(getenv("HB200_BCR_VARIANT")) : 0;
    HB_CUDA(cudaMemcpy(c->band_dbg.p + 71, &variant, sizeof(variant), cudaMemcpyHostToDevice));
  }
  // parallelism of the J^T J kernels: aim at ~2 CTAs per SM
  c->pix_splits = std::max(1, std::min((2 * c->num_sms + std::max(c->nseg, 1) - 1) / std::max(c->nseg, 1), std::max(1, c->Nv / (16 * std::max(c->nseg, 1)))));
  {
    static const int min_chunk = getenv("HB200_IMU_MIN_CHUNK") ? std::max(1, atoi(getenv("HB200_IMU_MIN_CHUNK"))) : 8;   // factors per CTA at least
    c->imu_splits = std::max(1, std::min((2 * c->num_sms + std::max(c->nruns, 1) - 1) / std::max(c->nruns, 1), std::max(1, c->Ni / (min_chunk * std::max(c->nruns, 1)))));
    // tensor-core kernel (large windows): ~6 CTAs per SM, at least two 8-factor chunks per CTA
    static const int per_sm = getenv("HB200_IMU_CTAS_PER_SM") ? std::max(1, atoi(getenv("HB200_IMU_CTAS_PER_SM"))) : 6;
    c->imu_splits_mma = std::max(1, std::min((per_sm * c->num_sms + std::max(c->nruns, 1) - 1) / std::max(c->nruns, 1), std::max(1, c->Ni / (16 * std::max(c->nruns, 1)))));
  }
  return 0;
}

int reset_solver_state(hb200_ctx* c) {
  SolverState s{};
  s.radius = c->radius0; s.decrease_factor = 2.0; s.spd = 1;
  HB_CUDA(c->st.ensure(1));
  HB_CUDA(cudaMemcpyAsync(c->st.p, &s, sizeof(s), cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->iter_total = 0;
  return 0;
}

// ---- kernel dispatch on (order, bias order) -------------------------------------------------
template <bool J>
PixelArgs pixel_args(hb200_ctx* c, int sel, bool accumulate) {
  PixelArgs a{};
  a.sys = accumulate ? c->assembly() : nullptr; a.lay = c->lay; a.tiles_per_cta = 1;
  a.n = c->Nv; a.stamp = c->v_stamp.p; a.pixel = reinterpret_cast<const double2*>(c->v_pixel.p); a.meas_z = c->v_z.p; a.idx = c->v_idx.p;
  a.tab = c->tab[sel].p; a.cam_tab = c->cam_tab.p; a.landmarks = c->lms[sel].p;
  a.r = J ? c->v_r.p : nullptr; a.Jp = c->v_Jp.p; a.Jl = c->v_Jl.p; a.w = c->v_w.p; a.cost_partial = c->cp_pix[J ? 0 : 1].p; a.huber = c->huber; a.huber_bearing = c->huber_bearing; a.K_knots = c->K;
  return a;
}
template <bool J>
InertialArgs inertial_args(hb200_ctx* c, int sel) {
  InertialArgs a{};
  a.n = c->Ni; a.stamp = c->i_stamp.p; a.meas = c->i_meas.p; a.idx = c->i_idx.p; a.tab = c->tab[sel].p; a.imu_tab = c->imu_tab.p;
  a.bg = c->bg[sel].p; a.ba = c->ba[sel].p; a.gravity = c->grav[sel].p;
  a.r = J ? c->i_r.p : nullptr; a.Jp = c->i_Jp.p; a.wg = c->i_wg.p; a.wa = c->i_wa.p; a.Jg = c->i_Jg.p;
  a.cost_partial = c->cp_imu[J ? 0 : 1].p; a.loss_scale = c->imu_scale;
  return a;
}
template <int K, bool J>
int launch_pixel(hb200_ctx* c, int sel, bool accumulate = false) {
  if (c->Nv == 0) return 0;
  PixelArgs a = pixel_args<J>(c, sel, accumulate);
  if (J && accumulate) {
    // optional (HB200_PIX_TILES): a CTA walks several consecutive tiles and flushes its J^T J accumulators once per knot base
    static const int tiles_env = getenv("HB200_PIX_TILES") ? atoi(getenv("HB200_PIX_TILES")) : 0;
    a.tiles_per_cta = tiles_env > 0 ? tiles_env : 1;   // measured on the 1 M-factor window: 1 tile 0.41 ms, 11 tiles 0.50 ms (fewer, longer CTAs lose more than the saved atomics win)
    const int grid = (c->n_pix_blocks + a.tiles_per_cta - 1) / a.tiles_per_cta;
    pixel_eval_kernel<K, J, J><<<grid, kEvalThreads, 0, c->stream>>>(a, c->basis);
  } else pixel_eval_kernel<K, J, false><<<c->n_pix_blocks, kEvalThreads, 0, c->stream>>>(a, c->basis);
  HB_LAUNCH(c, "pixel_eval_kernel");
  return 0;
}
template <int K, bool J>
int launch_inertial(hb200_ctx* c, int sel) {
  if (c->Ni == 0) return 0;
  const InertialArgs a = inertial_args<J>(c, sel);
  inertial_eval_kernel<K, 4, J><<<c->n_imu_blocks, kEvalThreads, J ? inertial_stash_bytes(K) : 0, side(c)>>>(a, c->basis, c->bias_basis);
  HB_LAUNCH(c, "inertial_eval_kernel");
  return 0;
}
// visual + inertial factors in one launch (both lists non-empty)
template <int K, bool J>
int launch_factors_merged(hb200_ctx* c, int sel, bool accumulate) {
  const PixelArgs pa = pixel_args<J>(c, sel, accumulate);
  const InertialArgs ia = inertial_args<J>(c, sel);
  const int blocks = c->n_pix_blocks + c->n_imu_blocks;
  const size_t smem = J ? inertial_stash_bytes(K) : 0;
  if (J && accumulate) HB_CUDA(launch_dependent(c, factor_eval_kernel<K, 4, J, J>, dim3(blocks), dim3(kEvalThreads), smem, pa, ia, c->basis, c->bias_basis, c->n_pix_blocks));
  else HB_CUDA(launch_dependent(c, factor_eval_kernel<K, 4, J, false>, dim3(blocks), dim3(kEvalThreads), smem, pa, ia, c->basis, c->bias_basis, c->n_pix_blocks));
  HB_LAUNCH(c, "factor_eval_kernel");
  return 0;
}
template <int K, bool J>
int launch_manifold(hb200_ctx* c, int sel) {
  if (c->Nm == 0) return 0;
  ManifoldArgs a{};
  a.n = c->Nm; a.stamp = c->m_stamp.p; a.meas = c->m_meas.p; a.idx = c->m_idx.p; a.tab = c->tab[sel].p; a.sensors = c->sensors.p;
  a.r = J ? c->m_r.p : nullptr; a.Jp = c->m_Jp.p; a.cost_partial = c->cp_imu[J ? 0 : 1].p + c->n_imu_blocks;
  manifold_eval_kernel<K, J><<<c->n_man_blocks, kEvalThreads, 0, side(c)>>>(a, c->basis);
  HB_LAUNCH(c, "manifold_eval_kernel");
  return 0;
}
int enqueue_manifold(hb200_ctx* c, bool want_J, int sel) {
  if (c->k == 4) return want_J ? launch_manifold<4, true>(c, sel) : launch_manifold<4, false>(c, sel);
  return want_J ? launch_manifold<6, true>(c, sel) : launch_manifold<6, false>(c, sel);
}

// keep_fork: leave the side stream forked on return (the caller enqueues more side-stream work and joins).
// clear_system: zero the packed reduced system in the knot-table launch; skip_prep: the table of state `sel` is
// already up to date (retract_kernel built the trial table).
int enqueue_evaluate(hb200_ctx* c, bool want_J, int sel, bool accumulate = false, bool keep_fork = false, bool clear_system = false,
                     bool skip_prep = false) {
  if (c->k != 4 && c->k != 6) return fail(-4, "spline order %d not supported (4 or 6)", c->k);
  if (!skip_prep) {
    const size_t nclear = clear_system ? static_cast<size_t>(c->lay.total) : 0;
    const int blocks = clear_system ? static_cast<int>(std::min<size_t>((nclear / 4 + 255) / 256, static_cast<size_t>(c->num_sms) * 4)) : (c->K + 255) / 256;
    prep_kernel<<<std::max(blocks, (c->K + 255) / 256), 256, 0, c->stream>>>(c->K, c->knots[sel].p, c->tab[sel].p, clear_system ? c->assembly() : nullptr, nclear);
    HB_LAUNCH(c, "prep_kernel");
  }
  int rc = 0;
  const bool J_any = want_J || accumulate;
  // Small windows are latency-bound: one launch for both factor families.  Large windows are throughput-bound: the
  // merged kernel would run the pixel CTAs at the inertial body's 255 registers, so the families stay separate.
  static const bool no_merge = getenv("HB200_NO_MERGE") != nullptr;   // profiling aid: one kernel per factor family
  if (c->Nv && c->Ni && !no_merge && c->n_pix_blocks + c->n_imu_blocks <= 4 * c->num_sms) {   // (also while profiling: same kernels as the graph)
    // visual and inertial factors side by side in one launch; pose factors (if any) on the side stream
    if (c->Nm && (rc = fork_side(c))) return rc;
    if (c->k == 4) rc = J_any ? launch_factors_merged<4, true>(c, sel, accumulate) : launch_factors_merged<4, false>(c, sel, false);
    else rc = J_any ? launch_factors_merged<6, true>(c, sel, accumulate) : launch_factors_merged<6, false>(c, sel, false);
    if (!rc) rc = enqueue_manifold(c, J_any, sel);
    // always join here: the inertial Jacobians were produced on the MAIN stream, so the J^T J kernels that follow
    // (enqueue_build) must not run on a still-forked side stream
    { const int rj = join_side(c); if (!rc) rc = rj; }
    return rc;
  }
  // visual factors on the main stream, inertial + manifold factors concurrently on the side stream
  if (c->Nv && (c->Ni || c->Nm) && (rc = fork_side(c))) return rc;
  if (accumulate) {   // fused path: pixel J^T J is accumulated by the factor kernel itself
    rc = (c->k == 4) ? launch_pixel<4, true>(c, sel, true) : launch_pixel<6, true>(c, sel, true);
    if (!rc) rc = (c->k == 4) ? launch_inertial<4, true>(c, sel) : launch_inertial<6, true>(c, sel);
    if (!rc) rc = enqueue_manifold(c, true, sel);
  } else {
    if (c->k == 4) { rc = want_J ? launch_pixel<4, true>(c, sel) : launch_pixel<4, false>(c, sel); if (!rc) rc = want_J ? launch_inertial<4, true>(c, sel) : launch_inertial<4, false>(c, sel); }
    else { rc = want_J ? launch_pixel<6, true>(c, sel) : launch_pixel<6, false>(c, sel); if (!rc) rc = want_J ? launch_inertial<6, true>(c, sel) : launch_inertial<6, false>(c, sel); }
    if (!rc) rc = enqueue_manifold(c, want_J, sel);
  }
  if (rc || !keep_fork) { const int rj = join_side(c); if (!rc) rc = rj; }
  return rc;
}

int enqueue_clear_system(hb200_ctx* c) {
  HB_CUDA(cudaMemsetAsync(c->assembly(), 0, static_cast<size_t>(c->lay.total) * sizeof(double), c->stream));
  prof_mark(c, "memset(system)");
  return 0;
}

// J^T J of the inertial / manifold factors and the cost sum on the side stream, the landmark Schur complement on
// the main stream: both accumulate into S with atomics (commutative), diag(J^T J) is kept apart from S, so nothing
// orders them.  after_eval_on_main: the factor Jacobians were produced by a launch on the MAIN stream (merged
// factor kernel), so the side stream is forked here rather than before the evaluation.
int enqueue_build(hb200_ctx* c, bool pixel_fused = false) {
  if (!pixel_fused) { int rc0 = enqueue_clear_system(c); if (rc0) return rc0; }
  if (c->Nv && !pixel_fused) {
    if (c->k == 4) pixel_hessian_kernel<4><<<c->nseg * c->pix_splits, kHessThreads, 0, c->stream>>>(c->seg_off.p, c->v_r.p, c->v_Jp.p, c->v_w.p, c->assembly(), c->lay, c->pix_splits);
    else pixel_hessian_kernel<6><<<c->nseg * c->pix_splits, kHessThreads, 0, c->stream>>>(c->seg_off.p, c->v_r.p, c->v_Jp.p, c->v_w.p, c->assembly(), c->lay, c->pix_splits);
    HB_LAUNCH(c, "pixel_hessian_kernel");
  }
  { const int rf = fork_side(c); if (rf) return rf; }   // (no-op when already forked or while profiling)
  if (c->Ni) {
    // large windows (>= 16 384 inertial factors): the augmented product on the FP64 tensor cores, ~6 CTAs per SM of 8-factor
    // chunks (1 M-factor window: 0.295 -> 0.16 ms); small windows: the scalar block-by-block kernel on short runs (cfg1, ~9
    // factors per CTA: 16.4 vs 18.3 us).  HB200_IMU_HESS=0 / 1 forces the scalar / tensor-core kernel (A/B switch)
    static const int hess_env = getenv("HB200_IMU_HESS") != nullptr ? atoi(getenv("HB200_IMU_HESS")) : -1;
    const bool scalar_hess = hess_env >= 0 ? hess_env == 0 : c->Ni < 16384;
    // (order 6 keeps the configuration it was measured with: 12-factor chunks, ~2 CTAs per SM -- order-6 window 0.045 ms; with
    // 8-factor chunks and ~6 CTAs per SM 0.053 ms)
    const int splits = (scalar_hess || c->k != 4) ? c->imu_splits : c->imu_splits_mma;
    const int grid = c->nruns * splits;
    if (scalar_hess) {
      if (c->k == 4)
        inertial_hessian_kernel<4, 4><<<grid, kHessThreads, 0, side(c)>>>(c->run_off.p, c->i_idx.p, c->i_r.p, c->i_Jp.p, c->i_wg.p, c->i_wa.p,
                                                                          c->i_Jg.p, c->imu_scale, c->assembly(), c->lay, c->o_bg(), c->o_ba(), c->o_g(), c->imu_splits);
      else
        inertial_hessian_kernel<6, 4><<<grid, kHessThreads, 0, side(c)>>>(c->run_off.p, c->i_idx.p, c->i_r.p, c->i_Jp.p, c->i_wg.p, c->i_wa.p,
                                                                          c->i_Jg.p, c->imu_scale, c->assembly(), c->lay, c->o_bg(), c->o_ba(), c->o_g(), c->imu_splits);
    } else {
      static const bool small_chunks = !(getenv("HB200_IMU_CH") != nullptr && atoi(getenv("HB200_IMU_CH")) != 8);   // 8-factor chunks (HB200_IMU_CH=16: 16 / 12)
#define HB_IMU_MMA(KK, CHH) inertial_hessian_mma_kernel<KK, 4, CHH><<<grid, kHessThreads, 0, side(c)>>>(c->run_off.p, c->i_idx.p, c->i_r.p, c->i_Jp.p, c->i_wg.p, c->i_wa.p, \
                                                    c->i_Jg.p, c->imu_scale, c->assembly(), c->lay, c->o_bg(), c->o_ba(), c->o_g(), splits)
      if (c->k == 4) { if (small_chunks) HB_IMU_MMA(4, 8); else HB_IMU_MMA(4, 16); }
      else HB_IMU_MMA(6, 12);
#undef HB_IMU_MMA
    }
    HB_LAUNCH(c, scalar_hess ? "inertial_hessian_kernel" : "inertial_hessian_mma_kernel");
  }
  if (c->Nm) {
    const int blocks = (c->Nm + kManWarps - 1) / kManWarps;
    if (c->k == 4) manifold_hessian_kernel<4><<<blocks, kManWarps * 32, 0, side(c)>>>(c->Nm, c->m_idx.p, c->m_r.p, c->m_Jp.p, c->assembly(), c->lay);
    else manifold_hessian_kernel<6><<<blocks, kManWarps * 32, 0, side(c)>>>(c->Nm, c->m_idx.p, c->m_r.p, c->m_Jp.p, c->assembly(), c->lay);
    HB_LAUNCH(c, "manifold_hessian_kernel");
  }
  if (c->forked) {   // the cost partials of the visual factors come from the main stream
    HB_CUDA(cudaEventRecord(c->ev_mid, c->stream));
    HB_CUDA(cudaStreamWaitEvent(c->stream2, c->ev_mid, 0));
  }
  cost_kernel<<<1, 256, 0, side(c)>>>(c->assembly(), c->lay, c->cp_pix[0].p, c->Nv ? c->n_pix_blocks : 0, c->cp_imu[0].p, c->n_imu_blocks + c->n_man_blocks);
  HB_LAUNCH(c, "cost_kernel");
  if (c->Nv && c->L && c->schur_groups) {
    const size_t smem = (3 * static_cast<size_t>(kSchurGroup) * (c->schur_rt + 1) + 3 * kSchurGroup + 4 * 3 * static_cast<size_t>(c->schur_rt)) * sizeof(double);
    if (c->k == 4)
      schur_group_kernel<4><<<c->n_lm_groups, kSchurGThreads, smem, c->stream>>>(c->lm_group_off.p, c->lm_order.p, c->lm_off.p, c->lm_obs.p, c->v_idx.p, c->v_r.p, c->v_Jp.p,
                                                                                 c->v_Jl.p, c->v_w.p, c->st.p, c->assembly(), c->lay, c->Vinv.p, c->gl.p, c->Dl.p, c->schur_rt);
    else
      schur_group_kernel<6><<<c->n_lm_groups, kSchurGThreads, smem, c->stream>>>(c->lm_group_off.p, c->lm_order.p, c->lm_off.p, c->lm_obs.p, c->v_idx.p, c->v_r.p, c->v_Jp.p,
                                                                                 c->v_Jl.p, c->v_w.p, c->st.p, c->assembly(), c->lay, c->Vinv.p, c->gl.p, c->Dl.p, c->schur_rt);
    HB_LAUNCH(c, "schur_group_kernel");
  } else if (c->Nv && c->L) {
    const size_t smem = 2 * 3 * static_cast<size_t>(c->max_rows) * sizeof(double);
    if (c->k == 4)
      schur_kernel<4><<<c->L, kSchurThreads, smem, c->stream>>>(c->lm_off.p, c->lm_obs.p, c->v_idx.p, c->v_r.p, c->v_Jp.p, c->v_Jl.p, c->v_w.p, c->st.p,
                                                                c->assembly(), c->lay, c->Vinv.p, c->gl.p, c->Dl.p, c->max_rows);
    else
      schur_kernel<6><<<c->L, kSchurThreads, smem, c->stream>>>(c->lm_off.p, c->lm_obs.p, c->v_idx.p, c->v_r.p, c->v_Jp.p, c->v_Jl.p, c->v_w.p, c->st.p,
                                                                c->assembly(), c->lay, c->Vinv.p, c->gl.p, c->Dl.p, c->max_rows);
    HB_LAUNCH(c, "schur_kernel");
  }
  return join_side(c);
}

// band-only raw system -> dense damped work copy Lw (dense fallback solver, hb200_get_system)
int enqueue_densify(hb200_ctx* c) {
  int rc = ensure_dense(c);
  if (rc) return rc;
  const size_t total = static_cast<size_t>(c->n + 1) * c->n;
  const int blocks = static_cast<int>(std::min<size_t>((total + 255) / 256, static_cast<size_t>(c->num_sms) * 8));
  densify_kernel<<<blocks, 256, 0, c->stream>>>(c->sys.p, c->lay, c->st.p, c->fixed.p, c->D.p, c->Lw.p, c->spd.p);
  HB_LAUNCH(c, "densify_kernel");
  return 0;
}

RetractArgs retract_args(hb200_ctx* c);
// Both solvers read the raw band-only system and apply LM damping + the constant-dof mask themselves (the band
// solver while it gathers, the dense fallback in densify_kernel);
// fuse_retract: the landmark back-substitution launch also retracts knots / biases / gravity (returns *fused)
int enqueue_solve(hb200_ctx* c, bool fuse_retract = false, bool* fused = nullptr) {
  if (c->use_bcr) {
    const double* sys = c->sys.p; SysLayout lay = c->lay; BcrPlan pl = c->bcr; double* ws = c->bcr_ws.p; unsigned int* bar = c->bcr_bar.p;
    double* x = c->dp.p; int* spd = c->spd.p; const SolverState* st = c->st.p; const unsigned char* fx = c->fixed.p; double* Dout = c->D.p;
    long long* dbg = c->band_dbg.p;
    void* args[] = {&sys, &lay, &pl, &ws, &bar, &x, &spd, &st, &fx, &Dout, &dbg};
    HB_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(bcr_solve_kernel), dim3(c->bcr_ctas), dim3(kBcrThreads), args, c->bcr_smem, c->stream));
    c->launches += 1;
    prof_mark(c, "bcr_solve_kernel");
  } else if (c->band_solver) {
    const SolverState* st = c->st.p;
    const unsigned char* fx = c->fixed.p;
    double* Dout = c->D.p;
    const size_t smem = c->band_smem ? band_workspace_doubles(c->K, c->beta, c->n - 6 * c->K) * sizeof(double) : 0;
    if (c->band_smem) band_solve_kernel<true><<<1, kBandThreads, smem, c->stream>>>(c->sys.p, c->lay, c->band_ws.p, c->dp.p, c->spd.p, c->band_dbg.p, st, fx, Dout, 0);
    else band_solve_kernel<false><<<1, kBandThreads, c->band_chunk_smem, c->stream>>>(c->sys.p, c->lay, c->band_ws.p, c->dp.p, c->spd.p, c->band_dbg.p, st, fx, Dout, c->band_chunk_cols);
    HB_LAUNCH(c, c->band_smem ? "band_solve_kernel" : "band_solve_kernel<chunked>");
  } else {
    { const int rd = enqueue_densify(c); if (rd) return rd; }
    int n = c->n;
    double* Lw = c->Lw.p; double* Ld = c->Ldiag.p; int* spd = c->spd.p;
    void* args[] = {&Lw, &Ld, &n, &spd};
    const int T = (n + kCholNB - 1) / kCholNB;
    const long long tiles = static_cast<long long>(T) * (T + 1) / 2 + T;
    int blocks = static_cast<int>(std::min<long long>(c->num_sms, std::max<long long>(1, (tiles + kCholWarps - 1) / kCholWarps)));
    HB_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(cholesky_kernel), dim3(blocks), dim3(kCholThreads), args, kCholSmem, c->stream));
    c->launches += 1;
    prof_mark(c, "cholesky_kernel");
    backsolve_kernel<<<1, 1024, 0, c->stream>>>(c->Lw.p, c->Ldiag.p, c->n, c->dp.p);
    HB_LAUNCH(c, "backsolve_kernel");
  }
  if (c->L) {
    if (c->Nv) {
      RetractArgs ra{};
      int extra = 0;
      if (fuse_retract) {
        ra = retract_args(c);
        extra = (std::max(std::max(c->K, 1), std::max(c->Kbg, c->Kba)) + kLmWarps * 32 - 1) / (kLmWarps * 32);
        if (fused) *fused = true;
      }
      if (c->k == 4)
        HB_CUDA(launch_dependent(c, lm_backsub_kernel<4>, dim3(c->n_lm_blocks + extra), dim3(kLmWarps * 32), 0, c->L, c->lm_off.p, c->lm_obs.p, c->v_idx.p, c->v_r.p, c->v_Jp.p, c->v_Jl.p, c->v_w.p,
                                 c->Vinv.p, c->gl.p, c->Dl.p, c->dp.p, c->dl.p, c->lm_part.p, c->lms[0].p, c->lms[1].p, c->n_lm_blocks, ra));
      else
        HB_CUDA(launch_dependent(c, lm_backsub_kernel<6>, dim3(c->n_lm_blocks + extra), dim3(kLmWarps * 32), 0, c->L, c->lm_off.p, c->lm_obs.p, c->v_idx.p, c->v_r.p, c->v_Jp.p, c->v_Jl.p, c->v_w.p,
                                 c->Vinv.p, c->gl.p, c->Dl.p, c->dp.p, c->dl.p, c->lm_part.p, c->lms[0].p, c->lms[1].p, c->n_lm_blocks, ra));
      HB_LAUNCH(c, "lm_backsub_kernel");
    } else {
      HB_CUDA(cudaMemsetAsync(c->dl.p, 0, 3 * static_cast<size_t>(c->L) * sizeof(double), c->stream));
      HB_CUDA(cudaMemsetAsync(c->lm_part.p, 0, 5 * static_cast<size_t>(c->n_lm_blocks) * sizeof(double), c->stream));
    }
  }
  return 0;
}

RetractArgs retract_args(hb200_ctx* c) {
  RetractArgs ra{};
  ra.K = c->K; ra.Kbg = c->Kbg; ra.Kba = c->Kba; ra.L = c->L;
  ra.dp = c->dp.p; ra.dl = c->dl.p; ra.knots = c->knots[0].p; ra.bg = c->bg[0].p; ra.ba = c->ba[0].p; ra.grav = c->grav[0].p; ra.lms = c->lms[0].p;
  ra.knots_t = c->knots[1].p; ra.bg_t = c->bg[1].p; ra.ba_t = c->ba[1].p; ra.grav_t = c->grav[1].p; ra.lms_t = c->lms[1].p; ra.tab_t = c->tab[1].p;
  ra.retract_landmarks = (c->L && !c->Nv) ? 1 : 0;
  return ra;
}
int enqueue_retract(hb200_ctx* c) {
  const int m = std::max(std::max(c->K, c->L), std::max(std::max(c->Kbg, c->Kba), 1));
  retract_kernel<<<(m + 127) / 128, 128, 0, c->stream>>>(retract_args(c));
  HB_LAUNCH(c, "retract_kernel");
  return 0;
}

int enqueue_scalars(hb200_ctx* c) {
  scalars_kernel<<<1, 256, 0, c->stream>>>(c->cp_pix[1].p, c->Nv ? c->n_pix_blocks : 0, c->cp_imu[1].p, c->n_imu_blocks + c->n_man_blocks, c->lm_part.p,
                                          (c->L && c->Nv) ? c->n_lm_blocks : 0, c->scal.p);
  HB_LAUNCH(c, "scalars_kernel");
  return 0;
}

TermArgs term_args(hb200_ctx* c) {
  TermArgs t{};
  t.enabled = c->term_enabled ? 1 : 0;
  t.function_tolerance = c->term_ftol; t.gradient_tolerance = c->term_gtol; t.parameter_tolerance = c->term_ptol; t.min_radius = c->term_min_radius;
  t.K = c->K; t.Kbg = c->Kbg; t.Kba = c->Kba;
  t.knots = c->knots[0].p; t.knots_t = c->knots[1].p; t.bg = c->bg[0].p; t.bg_t = c->bg[1].p; t.ba = c->ba[0].p; t.ba_t = c->ba[1].p;
  t.grav = c->grav[0].p; t.grav_t = c->grav[1].p;
  return t;
}

int enqueue_accept(hb200_ctx* c) {
  ScalarArgs sa{c->cp_pix[1].p, c->Nv ? c->n_pix_blocks : 0, c->cp_imu[1].p, c->n_imu_blocks + c->n_man_blocks, c->lm_part.p, (c->L && c->Nv) ? c->n_lm_blocks : 0};
  CommitArgs a{};
  const size_t counts[5] = {8 * static_cast<size_t>(c->K), 4 * static_cast<size_t>(c->Kbg), 4 * static_cast<size_t>(c->Kba), 3, 3 * static_cast<size_t>(c->L)};
  const double* srcs[5] = {c->knots[1].p, c->bg[1].p, c->ba[1].p, c->grav[1].p, c->lms[1].p};
  double* dsts[5] = {c->knots[0].p, c->bg[0].p, c->ba[0].p, c->grav[0].p, c->lms[0].p};
  size_t mx = 1, total = 0;
  for (int i = 0; i < 5; ++i) { a.count[i] = counts[i]; a.src[i] = srcs[i]; a.dst[i] = dsts[i]; mx = std::max(mx, counts[i]); total += counts[i]; }
  const bool fuse_commit = total <= 65536;   // small windows: one CTA commits the accepted state right away
  // scalars: summed inside this kernel on one GPU and, across GPUs, exchanged by it through peer memory; only the
  // fallbacks (callback hook, no peer mapping) run scalars_kernel + a second reduction before it
  const bool mailbox = c->nccl && c->peers_open;
  MailboxArgs mb{};
  mb.nranks = mailbox ? c->nranks : 1; mb.rank = c->rank; mb.peers = c->d_peers.p; mb.local = c->mbox.p; mb.seq = c->mbox_seq.p;
  HB_CUDA(launch_dependent(c, accept_kernel, dim3(1), dim3(kAcceptThreads), 0, c->sys.p, c->lay, c->scal.p, c->dp.p, c->D.p, c->fixed.p, c->st.p, c->spd.p, c->records.p, c->max_records,
                           (!c->multi() || mailbox) ? 1 : 0, sa, fuse_commit ? 1 : 0, a, mb, term_args(c)));
  HB_LAUNCH(c, "accept_kernel");
  if (!fuse_commit) {
    const int blocks = static_cast<int>(std::min<size_t>((mx + 255) / 256, static_cast<size_t>(c->num_sms) * 4));
    commit_kernel<<<blocks, 256, 0, c->stream>>>(c->st.p, a);
    HB_LAUNCH(c, "commit_kernel");
  }
  return 0;
}

// Sum of the packed partial systems over the ranks: ONE ncclAllReduce on the context's stream (capturable).
int enqueue_reduce_system(hb200_ctx* c) {
  if (c->peer_reduce()) {
    // fused barrier + reduction over peer memory (peer_reduce_kernel); the next iteration assembles into the other half
    PeerReduceArgs a{};
    a.nranks = c->nranks; a.rank = c->rank; a.peers = c->d_peers.p; a.local = c->mbox.p;
    a.part_offset = kArenaParts + static_cast<long long>(c->peer_par) * c->arena_cap; a.total = c->lay.total;
    a.out = c->sys.p; a.round = c->red_round.p; a.arrive = c->red_arrive.p; a.st = c->st.p;
    const long long pairs = c->lay.total / 2;
    const int grid = static_cast<int>(std::max<long long>(1, std::min<long long>(4LL * c->num_sms, (pairs + kReduceThreads - 1) / kReduceThreads)));
    peer_reduce_kernel<<<grid, kReduceThreads, 0, c->stream>>>(a);
    HB_LAUNCH(c, "peer_reduce_kernel");
    c->peer_par ^= 1;
    return 0;
  }
  if (c->nccl) {
    HB_NCCL(g_nccl.AllReduce(c->sys.p, c->sys.p, static_cast<size_t>(c->lay.total), /*ncclDouble*/ 8, /*ncclSum*/ 0, c->nccl, c->stream));
    c->nccl_calls += 1;
    prof_mark(c, "ncclAllReduce(system)");
  } else if (c->allreduce) {
    const int rc = c->allreduce(c->allreduce_user, c->sys.p, c->lay.total, c->stream);
    if (rc) return fail(200 + rc, "all-reduce callback failed (%d)", rc);
    prof_mark(c, "allreduce_callback(system)");
  }
  return 0;
}

// Trial-cost / model-decrease partials: fused into accept_kernel (one GPU: plain sums; NCCL + peer mapping: the
// mailbox exchange).  Fallbacks only: scalars_kernel + a 4-double reduction.
int enqueue_reduce_scalars(hb200_ctx* c) {
  if (!c->multi() || (c->nccl && c->peers_open)) return 0;
  int rc = enqueue_scalars(c);
  if (rc) return rc;
  if (c->nccl) {
    HB_NCCL(g_nccl.AllReduce(c->scal.p, c->scal.p, 8, 8, 0, c->nccl, c->stream));
    c->nccl_calls += 1;
    prof_mark(c, "ncclAllReduce(scalars)");
  } else {
    rc = c->allreduce(c->allreduce_user, c->scal.p, 8, c->stream);
    if (rc) return fail(200 + rc, "all-reduce callback failed (%d)", rc);
    prof_mark(c, "allreduce_callback(scalars)");
  }
  return 0;
}

// One LM iteration enqueued on the stream (graph-capturable unless the callback hook is in use).
int enqueue_iteration(hb200_ctx* c) {
  int rc = 0;
  // pixel J^T J: fused into the factor kernel (small windows: one launch less on the latency chain) or a separate
  // segment-wise pass over the Jacobians (large windows); HB200_FUSE=0/1 overrides the choice
  static const int fuse_env = getenv("HB200_FUSE") ? atoi(getenv("HB200_FUSE")) : -1;
  const bool fuse = fuse_env >= 0 ? fuse_env != 0 : true;
  if ((rc = enqueue_evaluate(c, true, 0, fuse, /*keep_fork=*/true, /*clear_system=*/fuse))) return rc;
  if ((rc = enqueue_build(c, fuse))) return rc;
  if ((rc = enqueue_reduce_system(c))) return rc;
  bool retracted = false;
  if ((rc = enqueue_solve(c, /*fuse_retract=*/true, &retracted))) return rc;
  if (!retracted && (rc = enqueue_retract(c))) return rc;   // (also builds the trial knot table)
  if ((rc = enqueue_evaluate(c, false, 1, false, false, false, /*skip_prep=*/true))) return rc;
  if ((rc = enqueue_reduce_scalars(c))) return rc;
  return enqueue_accept(c);
}

// The band layout depends on the longest landmark track of the LOCAL shard; the ranks agree on the maximum
// (one 4-byte ncclAllReduce(max) at bind / attach time, never on the iteration path).
int sync_layout(hb200_ctx* c) {
  if (!c->nccl || !c->bound) return 0;
  DevBuf<int> d;
  HB_CUDA(d.ensure(1));
  int v = c->beta;
  HB_CUDA(cudaMemcpyAsync(d.p, &v, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  HB_NCCL(g_nccl.AllReduce(d.p, d.p, 1, /*ncclInt32*/ 2, /*ncclMax*/ 2, c->nccl, c->stream));
  HB_CUDA(cudaMemcpyAsync(&v, d.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->comm_warm = true;
  if (v != c->beta) {
    c->min_beta = v;
    const int rc = ensure_system(c);
    if (rc) return rc;
    c->invalidate();
  }
  return 0;
}

int check_ready(hb200_ctx* c) {
  if (!c) return fail(-1, "null context");
  if (c->K == 0) return fail(-2, "spline not set");
  if (!c->bound) return fail(-2, "factors not bound (call hb200_bind)");
  if (c->Ni && (!c->have_imu || !c->have_gravity || c->Kbg == 0 || c->Kba == 0)) return fail(-2, "inertial factors need IMU calibration, bias splines and gravity");
  if (c->Nv && (c->C == 0 || c->L == 0)) return fail(-2, "pixel / bearing factors need cameras and landmarks");
  if (c->Nm && c->P == 0) return fail(-2, "manifold factors need pose sensors");
  return 0;
}

int ensure_placeholders(hb200_ctx* c) {
  // Kernels take these pointers even when a factor family is absent.
  for (int s = 0; s < 2; ++s) {
    HB_CUDA(c->bg[s].ensure(4)); HB_CUDA(c->ba[s].ensure(4)); HB_CUDA(c->grav[s].ensure(4)); HB_CUDA(c->lms[s].ensure(3));
    HB_CUDA(c->cp_pix[s].ensure(1)); HB_CUDA(c->cp_imu[s].ensure(1));
  }
  HB_CUDA(c->imu_tab.ensure(kImuStride)); HB_CUDA(c->cam_tab.ensure(kCamStride));
  HB_CUDA(c->v_z.ensure(1)); HB_CUDA(c->v_w.ensure(1)); HB_CUDA(c->sensors.ensure(7)); HB_CUDA(c->m_idx.ensure(1));
  return 0;
}

}  // namespace

extern "C" {

const char* hb200_last_error_string(void) { return g_error.c_str(); }

namespace {
int create_impl(const hb200_options* options, hb200_ctx* c) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) return fail(100 + static_cast<int>(e), "no CUDA device: %s (libhyperb200 has no CPU fallback)", cudaGetErrorString(e));
  c->device = options ? options->device : 0;
  if (c->device < 0 || c->device >= count) return fail(-1, "invalid device %d", c->device);
  HB_CUDA(cudaSetDevice(c->device));
  cudaDeviceProp prop{};
  HB_CUDA(cudaGetDeviceProperties(&prop, c->device));
  if (prop.major < 10) return fail(-5, "device sm_%d%d is not Blackwell (built for sm_100a only)", prop.major, prop.minor);
  c->num_sms = prop.multiProcessorCount;
  c->use_graph = options ? options->use_graph != 0 : true;
  c->force_dense = options ? (options->reserved & 1) != 0 : false;
  if (options && options->stream) { c->stream = static_cast<cudaStream_t>(options->stream); c->own_stream = false; }
  else { HB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)); c->own_stream = true; }
  HB_CUDA(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
  HB_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  HB_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
  HB_CUDA(cudaEventCreateWithFlags(&c->ev_mid, cudaEventDisableTiming));
  int rc = ensure_placeholders(c);
  if (rc) return rc;
  if (options && options->nccl_comm && (rc = hb200_set_nccl_comm(c, options->nccl_comm, options->nranks, options->rank))) return rc;
  HB_CUDA(cudaFuncSetAttribute(cholesky_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kCholSmem)));
  // the Jacobian passes of the inertial factors park their forward-sweep state in dynamic shared memory (41.5 KB at
  // order 4, 69 KB at order 6); together with the static scratch of the merged kernel that is above the 48 KB default
  HB_CUDA(cudaFuncSetAttribute(inertial_eval_kernel<4, 4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(inertial_stash_bytes(4))));
  HB_CUDA(cudaFuncSetAttribute(inertial_eval_kernel<6, 4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(inertial_stash_bytes(6))));
  HB_CUDA(cudaFuncSetAttribute(factor_eval_kernel<4, 4, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(inertial_stash_bytes(4))));
  HB_CUDA(cudaFuncSetAttribute(factor_eval_kernel<4, 4, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(inertial_stash_bytes(4))));
  HB_CUDA(cudaFuncSetAttribute(factor_eval_kernel<6, 4, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(inertial_stash_bytes(6))));
  HB_CUDA(cudaFuncSetAttribute(factor_eval_kernel<6, 4, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(inertial_stash_bytes(6))));
  return reset_solver_state(c);
}
}  // namespace

int hb200_create(const hb200_options* options, hb200_ctx** out) {
  if (!out) return fail(-1, "null output pointer");
  *out = nullptr;
  hb200_ctx* c = new hb200_ctx();
  const int rc = create_impl(options, c);
  if (rc) {
    const std::string keep = g_error;   // hb200_destroy must not clobber the message
    hb200_destroy(c);
    g_error = keep;
    return rc;
  }
  *out = c;
  return 0;
}

void hb200_destroy(hb200_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->stream2) cudaStreamSynchronize(c->stream2);
  for (size_t p = 0; p < c->peer_ptrs.size(); ++p)
    if (c->peer_ptrs[p] && c->peer_ptrs[p] != c->mbox.p) cudaIpcCloseMemHandle(c->peer_ptrs[p]);
  c->peer_ptrs.clear();
  // the captured iteration references the communicator: NCCL waits in ncclCommDestroy until such graphs are gone
  if (c->graph_exec) cudaGraphExecDestroy(c->graph_exec);
  if (c->graph) cudaGraphDestroy(c->graph);
  if (c->graph_exec_b) cudaGraphExecDestroy(c->graph_exec_b);
  if (c->graph_b) cudaGraphDestroy(c->graph_b);
  c->graph_exec = nullptr; c->graph = nullptr; c->graph_exec_b = nullptr; c->graph_b = nullptr;
  if (c->nccl && c->own_nccl && g_nccl.CommDestroy) g_nccl.CommDestroy(c->nccl);
  c->nccl = nullptr;
  for (cudaEvent_t e : c->prof_events) cudaEventDestroy(e);
  for (int s = 0; s < 2; ++s) { c->knots[s].release(); c->bg[s].release(); c->ba[s].release(); c->grav[s].release(); c->lms[s].release(); c->tab[s].release(); c->cp_pix[s].release(); c->cp_imu[s].release(); }
  c->cams.release(); c->imu.release(); c->cam_tab.release(); c->imu_tab.release(); c->fixed.release();
  c->v_stamp.release(); c->v_pixel.release(); c->i_stamp.release(); c->i_meas.release(); c->v_cam.release(); c->v_lm.release(); c->v_idx.release(); c->i_idx.release();
  c->v_z.release(); c->v_w.release(); c->m_stamp.release(); c->m_meas.release(); c->sensors.release(); c->m_sensor.release(); c->m_idx.release(); c->m_r.release(); c->m_Jp.release();
  c->seg_off.release(); c->run_off.release(); c->lm_off.release(); c->lm_obs.release(); c->d_invalid.release(); c->lm_order.release(); c->lm_group_off.release();
  c->v_r.release(); c->v_Jp.release(); c->v_Jl.release(); c->i_r.release(); c->i_Jp.release(); c->i_wg.release(); c->i_wa.release(); c->i_Jg.release();
  c->sys.release(); c->D.release(); c->Lw.release(); c->Ldiag.release(); c->dp.release(); c->dl.release(); c->Vinv.release(); c->gl.release(); c->Dl.release();
  c->band_ws.release(); c->band_dbg.release(); c->bcr_ws.release(); c->bcr_bar.release(); c->lm_part.release(); c->scal.release(); c->spd.release(); c->st.release(); c->records.release();
  c->snap_knots.release(); c->snap_bg.release(); c->snap_ba.release(); c->snap_grav.release(); c->snap_lms.release(); c->snap_st.release();
  if (c->h_stage) cudaFreeHost(c->h_stage);
  c->d_stage.release();
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->ev_mid) cudaEventDestroy(c->ev_mid);
  if (c->stream2) cudaStreamDestroy(c->stream2);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

int hb200_synchronize(hb200_ctx* c) {
  if (!c) return fail(-1, "null context");
  HB_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

void* hb200_stream(hb200_ctx* c) { return c ? c->stream : nullptr; }
long long hb200_launch_count(hb200_ctx* c) { return c ? c->launches : 0; }

int hb200_set_spline(hb200_ctx* c, int order, int K, const double* knots) {
  if (!c || !knots) return fail(-1, "null argument");
  if (order != 4 && order != 6) return fail(-4, "spline order %d not supported (4 or 6)", order);
  if (K < order) return fail(-1, "need at least %d knots, got %d", order, K);
  for (int j = 1; j < K; ++j)
    if (!(knots[8 * j + 7] > knots[8 * (j - 1) + 7])) return fail(-1, "knot stamps must be strictly increasing (knot %d)", j);
  {   // uniform B-spline (the reference only ever creates uniformly separated knots, abstract.cpp:89,128)
    const double dt0 = knots[8 + 7] - knots[7];
    for (int j = 2; j < K; ++j)
      if (std::fabs((knots[8 * j + 7] - knots[8 * (j - 1) + 7]) - dt0) > 1e-6 * dt0) return fail(-1, "knot stamps must be uniformly spaced (knot %d)", j);
  }
  HB_CUDA(cudaSetDevice(c->device));
  bool reshape = (order != c->k) || (K != c->K);
  // the index maps of hb200_bind follow from the stamps: a window shifted by one knot keeps K but needs a re-bind
  if (!reshape) for (int j = 0; j < K && !reshape; ++j) if (c->h_knot_stamp[j] != knots[8 * j + 7]) reshape = true;
  c->h_knot_stamp.resize(K);
  for (int j = 0; j < K; ++j) c->h_knot_stamp[j] = knots[8 * j + 7];
  c->k = order; c->K = K;
  compute_basis(&c->basis, order);
  for (int s = 0; s < 2; ++s) { HB_CUDA(c->knots[s].ensure(8 * static_cast<size_t>(K))); HB_CUDA(c->tab[s].ensure(static_cast<size_t>(K) * kTabStride)); }
  HB_CUDA(cudaMemcpyAsync(c->knots[0].p, knots, 8 * sizeof(double) * K, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if (reshape) { c->h_knot_const.assign(K, 0); c->bound = false; c->invalidate(); c->have_snapshot = false; int rc = update_fixed(c); if (rc) return rc; }
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  return 0;
}

int hb200_set_bias_splines(hb200_ctx* c, int order, int Kg, const double* gyro, int Ka, const double* accel) {
  if (!c || !gyro || !accel) return fail(-1, "null argument");
  if (order != 4) return fail(-4, "bias spline order %d not supported (4)", order);
  if (Kg < order || Ka < order) return fail(-1, "need at least %d bias knots", order);
  for (int w = 0; w < 2; ++w) {
    const double* b = w ? accel : gyro;
    const int Kb = w ? Ka : Kg;
    const double dt0 = b[4 + 3] - b[3];
    if (!(dt0 > 0)) return fail(-1, "bias knot stamps must be strictly increasing");
    for (int j = 2; j < Kb; ++j)
      if (std::fabs((b[4 * j + 3] - b[4 * (j - 1) + 3]) - dt0) > 1e-6 * dt0) return fail(-1, "bias knot stamps must be uniformly spaced (knot %d)", j);
  }
  HB_CUDA(cudaSetDevice(c->device));
  bool reshape = (Kg != c->Kbg) || (Ka != c->Kba);
  if (!reshape) {
    for (int j = 0; j < Kg && !reshape; ++j) if (c->h_bg_stamp[j] != gyro[4 * j + 3]) reshape = true;
    for (int j = 0; j < Ka && !reshape; ++j) if (c->h_ba_stamp[j] != accel[4 * j + 3]) reshape = true;
  }
  c->h_bg_stamp.resize(Kg); c->h_ba_stamp.resize(Ka);
  for (int j = 0; j < Kg; ++j) c->h_bg_stamp[j] = gyro[4 * j + 3];
  for (int j = 0; j < Ka; ++j) c->h_ba_stamp[j] = accel[4 * j + 3];
  c->kb = order; c->Kbg = Kg; c->Kba = Ka;
  compute_basis(&c->bias_basis, order);
  for (int s = 0; s < 2; ++s) { HB_CUDA(c->bg[s].ensure(4 * static_cast<size_t>(Kg))); HB_CUDA(c->ba[s].ensure(4 * static_cast<size_t>(Ka))); }
  HB_CUDA(cudaMemcpyAsync(c->bg[0].p, gyro, 4 * sizeof(double) * Kg, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->ba[0].p, accel, 4 * sizeof(double) * Ka, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if (reshape) { c->bound = false; c->invalidate(); c->have_snapshot = false; int rc = update_fixed(c); if (rc) return rc; }
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  return 0;
}

int hb200_set_gravity(hb200_ctx* c, const double* g) {
  if (!c || !g) return fail(-1, "null argument");
  HB_CUDA(cudaSetDevice(c->device));
  HB_CUDA(cudaMemcpyAsync(c->grav[0].p, g, 3 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->have_gravity = true;
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  return 0;
}

int hb200_set_cameras(hb200_ctx* c, int C, const double* cams) {
  if (!c || !cams || C <= 0) return fail(-1, "invalid cameras");
  HB_CUDA(cudaSetDevice(c->device));
  if (C != c->C) { c->bound = false; c->invalidate(); }
  c->C = C;
  HB_CUDA(c->cams.ensure(15 * static_cast<size_t>(C)));
  HB_CUDA(c->cam_tab.ensure(kCamStride * static_cast<size_t>(C)));
  HB_CUDA(cudaMemcpyAsync(c->cams.p, cams, 15 * sizeof(double) * C, cudaMemcpyHostToDevice, c->stream));
  calib_kernel<<<(C + 63) / 64, 64, 0, c->stream>>>(C, c->cams.p, c->cam_tab.p, nullptr, nullptr, 0);
  HB_LAUNCH(c, "calib_kernel");
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  return 0;
}

int hb200_set_imu(hb200_ctx* c, const double* imu) {
  if (!c || !imu) return fail(-1, "null argument");
  HB_CUDA(cudaSetDevice(c->device));
  HB_CUDA(c->imu.ensure(37));
  HB_CUDA(cudaMemcpyAsync(c->imu.p, imu, 37 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  calib_kernel<<<1, 64, 0, c->stream>>>(0, nullptr, nullptr, c->imu.p, c->imu_tab.p, c->quirks);
  HB_LAUNCH(c, "calib_kernel");
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->have_imu = true;
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  return 0;
}

int hb200_set_landmarks(hb200_ctx* c, int L, const double* xyz) {
  if (!c || (L > 0 && !xyz) || L < 0) return fail(-1, "invalid landmarks");
  HB_CUDA(cudaSetDevice(c->device));
  if (L != c->L) { c->bound = false; c->invalidate(); c->have_snapshot = false; }
  c->L = L;
  for (int s = 0; s < 2; ++s) HB_CUDA(c->lms[s].ensure(3 * static_cast<size_t>(std::max(L, 1))));
  if (L) HB_CUDA(cudaMemcpyAsync(c->lms[0].p, xyz, 3 * sizeof(double) * L, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  return 0;
}

int hb200_set_constant(hb200_ctx* c, const unsigned char* knot_constant, int gravity_constant, int bias_constant) {
  if (!c) return fail(-1, "null context");
  if (c->K == 0) return fail(-2, "spline not set");
  HB_CUDA(cudaSetDevice(c->device));
  if (knot_constant) c->h_knot_const.assign(knot_constant, knot_constant + c->K);
  else c->h_knot_const.assign(c->K, 0);
  c->gravity_const = gravity_constant; c->bias_const = bias_constant;
  c->system_built = false;
  return update_fixed(c);
}

int hb200_set_reference_quirks(hb200_ctx* c, int quirks) {
  if (!c) return fail(-1, "null context");
  if (quirks < 0 || quirks > 15) return fail(-1, "quirks is a bit mask in [0, 15]");
  HB_CUDA(cudaSetDevice(c->device));
  c->quirks = quirks;
  if (c->have_imu) {   // rebuild the derived IMU table with the Jacobian-side matrices of this variant
    calib_kernel<<<1, 64, 0, c->stream>>>(0, nullptr, nullptr, c->imu.p, c->imu_tab.p, c->quirks);
    HB_LAUNCH(c, "calib_kernel");
    HB_CUDA(cudaStreamSynchronize(c->stream));
  }
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  return 0;
}

int hb200_set_options(hb200_ctx* c, double huber_pixel, double imu_loss_scale, double radius) {
  if (!c) return fail(-1, "null context");
  if (!(huber_pixel > 0) || !(imu_loss_scale > 0) || !(radius > 0)) return fail(-1, "options must be positive");
  HB_CUDA(cudaSetDevice(c->device));
  if (huber_pixel != c->huber || imu_loss_scale != c->imu_scale) c->graph_valid = false;  // baked into kernel arguments
  c->huber = huber_pixel; c->imu_scale = imu_loss_scale; c->radius0 = radius;
  c->system_built = false; c->evaluated_J = false;
  return reset_solver_state(c);
}

namespace {
// visual list = pixel factors followed by bearing factors
void rebuild_visual(hb200_ctx* c) {
  const size_t Np = c->Np, Nb = c->Nb, N = Np + Nb;
  c->Nv = static_cast<int>(N);
  c->h_v_stamp.resize(N); c->h_v_cam.resize(N); c->h_v_lm.resize(N); c->h_v_pixel.resize(2 * N); c->h_v_z.assign(N, 0.0);
  std::copy(c->h_p_stamp.begin(), c->h_p_stamp.end(), c->h_v_stamp.begin());
  std::copy(c->h_p_cam.begin(), c->h_p_cam.end(), c->h_v_cam.begin());
  std::copy(c->h_p_lm.begin(), c->h_p_lm.end(), c->h_v_lm.begin());
  std::copy(c->h_p_pixel.begin(), c->h_p_pixel.end(), c->h_v_pixel.begin());
  for (size_t f = 0; f < Nb; ++f) {
    c->h_v_stamp[Np + f] = c->h_b_stamp[f]; c->h_v_cam[Np + f] = c->h_b_cam[f]; c->h_v_lm[Np + f] = c->h_b_lm[f];
    c->h_v_pixel[2 * (Np + f)] = c->h_b_bearing[3 * f]; c->h_v_pixel[2 * (Np + f) + 1] = c->h_b_bearing[3 * f + 1];
    c->h_v_z[Np + f] = c->h_b_bearing[3 * f + 2];
  }
  c->bound = false; c->invalidate();
}
}  // namespace

int hb200_set_pixel_factors(hb200_ctx* c, int n, const double* stamp, const int* camera, const int* landmark, const double* pixel) {
  if (!c || n < 0 || (n > 0 && (!stamp || !camera || !landmark || !pixel))) return fail(-1, "invalid pixel factors");
  c->Np = n;
  c->h_p_stamp.assign(stamp, stamp + n); c->h_p_cam.assign(camera, camera + n); c->h_p_lm.assign(landmark, landmark + n);
  c->h_p_pixel.assign(pixel, pixel + 2 * static_cast<size_t>(n));
  rebuild_visual(c);
  return 0;
}

int hb200_set_bearing_factors(hb200_ctx* c, int n, const double* stamp, const int* camera, const int* landmark, const double* bearing) {
  if (!c || n < 0 || (n > 0 && (!stamp || !camera || !landmark || !bearing))) return fail(-1, "invalid bearing factors");
  c->Nb = n;
  c->h_b_stamp.assign(stamp, stamp + n); c->h_b_cam.assign(camera, camera + n); c->h_b_lm.assign(landmark, landmark + n);
  c->h_b_bearing.assign(bearing, bearing + 3 * static_cast<size_t>(n));
  rebuild_visual(c);
  return 0;
}

int hb200_set_bearing_loss(hb200_ctx* c, double huber_bearing) {
  if (!c) return fail(-1, "null context");
  if (!(huber_bearing > 0)) return fail(-1, "options must be positive");
  if (huber_bearing != c->huber_bearing) c->graph_valid = false;
  c->huber_bearing = huber_bearing;
  c->system_built = false; c->evaluated_J = false;
  return 0;
}

int hb200_set_pose_sensors(hb200_ctx* c, int n, const double* T_bs) {
  if (!c || n < 0 || (n > 0 && !T_bs)) return fail(-1, "invalid pose sensors");
  HB_CUDA(cudaSetDevice(c->device));
  if (n != c->P) c->bound = false;
  c->P = n;
  c->h_sensors.assign(T_bs, T_bs + 7 * static_cast<size_t>(n));
  HB_CUDA(c->sensors.ensure(7 * static_cast<size_t>(std::max(n, 1))));
  if (n) HB_CUDA(cudaMemcpyAsync(c->sensors.p, c->h_sensors.data(), sizeof(double) * 7 * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->invalidate();
  return 0;
}

int hb200_set_manifold_factors(hb200_ctx* c, int n, const double* stamp, const int* sensor, const double* pose) {
  if (!c || n < 0 || (n > 0 && (!stamp || !sensor || !pose))) return fail(-1, "invalid manifold factors");
  c->Nm = n;
  c->h_m_stamp.assign(stamp, stamp + n); c->h_m_sensor.assign(sensor, sensor + n); c->h_m_meas.assign(pose, pose + 7 * static_cast<size_t>(n));
  c->bound = false; c->invalidate();
  return 0;
}

int hb200_set_inertial_factors(hb200_ctx* c, int n, const double* stamp, const double* meas) {
  if (!c || n < 0 || (n > 0 && (!stamp || !meas))) return fail(-1, "invalid inertial factors");
  c->Ni = n;
  c->h_i_stamp.assign(stamp, stamp + n); c->h_i_meas.assign(meas, meas + 6 * static_cast<size_t>(n));
  c->bound = false; c->invalidate();
  return 0;
}

}  // extern "C"

namespace {
// After hb200_append_* / hb200_slide the factor lists exist on the device only (bound order == list order from then
// on).  The host mirrors the copy-out calls and a later full hb200_bind need are refreshed here, on demand.  The visual
// list splits by kind (idx.w): the pixel factors keep their list order as user order, a bearing factor's user index is
// Np + its rank among the bearings; the manifold list is in user order as it stands.
int sync_host_mirrors(hb200_ctx* c) {
  if (!c->device_managed) return 0;
  HB_CUDA(cudaSetDevice(c->device));
  const size_t Nv = c->Nv, Ni = c->Ni, Nm = c->Nm;
  std::vector<double> st(Nv), px(2 * Nv), vz(Nv);
  c->h_v_idx.resize(Nv); c->h_i_idx.resize(Ni); c->h_i_stamp.resize(Ni); c->h_i_meas.resize(6 * Ni);
  c->h_m_idx.resize(Nm); c->h_m_stamp.resize(Nm); c->h_m_meas.resize(7 * Nm);
  if (Nv) {
    HB_CUDA(cudaMemcpyAsync(st.data(), c->v_stamp.p, sizeof(double) * Nv, cudaMemcpyDeviceToHost, c->stream));
    HB_CUDA(cudaMemcpyAsync(px.data(), c->v_pixel.p, sizeof(double) * 2 * Nv, cudaMemcpyDeviceToHost, c->stream));
    HB_CUDA(cudaMemcpyAsync(vz.data(), c->v_z.p, sizeof(double) * Nv, cudaMemcpyDeviceToHost, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->h_v_idx.data(), c->v_idx.p, sizeof(int4) * Nv, cudaMemcpyDeviceToHost, c->stream));
  }
  if (Ni) {
    HB_CUDA(cudaMemcpyAsync(c->h_i_stamp.data(), c->i_stamp.p, sizeof(double) * Ni, cudaMemcpyDeviceToHost, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->h_i_meas.data(), c->i_meas.p, sizeof(double) * 6 * Ni, cudaMemcpyDeviceToHost, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->h_i_idx.data(), c->i_idx.p, sizeof(int4) * Ni, cudaMemcpyDeviceToHost, c->stream));
  }
  if (Nm) {
    HB_CUDA(cudaMemcpyAsync(c->h_m_stamp.data(), c->m_stamp.p, sizeof(double) * Nm, cudaMemcpyDeviceToHost, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->h_m_meas.data(), c->m_meas.p, sizeof(double) * 7 * Nm, cudaMemcpyDeviceToHost, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->h_m_idx.data(), c->m_idx.p, sizeof(int2) * Nm, cudaMemcpyDeviceToHost, c->stream));
  }
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->h_p_stamp.clear(); c->h_p_pixel.clear(); c->h_p_cam.clear(); c->h_p_lm.clear();
  c->h_b_stamp.clear(); c->h_b_bearing.clear(); c->h_b_cam.clear(); c->h_b_lm.clear();
  for (size_t f = 0; f < Nv; ++f) {
    const int4 id = c->h_v_idx[f];
    if (id.w == 0) {
      c->h_p_stamp.push_back(st[f]); c->h_p_pixel.push_back(px[2 * f]); c->h_p_pixel.push_back(px[2 * f + 1]);
      c->h_p_cam.push_back(id.z); c->h_p_lm.push_back(id.y);
    } else {
      c->h_b_stamp.push_back(st[f]); c->h_b_bearing.push_back(px[2 * f]); c->h_b_bearing.push_back(px[2 * f + 1]); c->h_b_bearing.push_back(vz[f]);
      c->h_b_cam.push_back(id.z); c->h_b_lm.push_back(id.y);
    }
  }
  c->Np = static_cast<int>(c->h_p_stamp.size()); c->Nb = static_cast<int>(c->h_b_stamp.size());
  // user-order visual list (pixel factors, then bearing factors: what rebuild_visual assembles) and bound position -> user index
  c->h_v_stamp.resize(Nv); c->h_v_pixel.resize(2 * Nv); c->h_v_z.assign(Nv, 0.0); c->h_v_cam.resize(Nv); c->h_v_lm.resize(Nv);
  c->v_perm.resize(Nv);
  for (size_t f = 0, ip = 0, ib = 0; f < Nv; ++f) {
    const size_t u = (c->h_v_idx[f].w == 0) ? ip++ : c->Np + ib++;
    c->v_perm[f] = static_cast<int>(u);
    c->h_v_stamp[u] = st[f]; c->h_v_pixel[2 * u] = px[2 * f]; c->h_v_pixel[2 * u + 1] = px[2 * f + 1];
    c->h_v_cam[u] = c->h_v_idx[f].z; c->h_v_lm[u] = c->h_v_idx[f].y;
    if (c->h_v_idx[f].w) c->h_v_z[u] = vz[f];
  }
  c->h_m_sensor.resize(Nm);
  for (size_t f = 0; f < Nm; ++f) c->h_m_sensor[f] = c->h_m_idx[f].y;
  c->i_perm.resize(Ni); std::iota(c->i_perm.begin(), c->i_perm.end(), 0);
  c->device_managed = false;
  return 0;
}

// Incidence lists of the device-resident factor lists (landmark CSR, inertial runs, segment offsets, longest
// track) by counting + scan kernels, then everything hb200_bind derives from them.  One small read-back.
int rebuild_incidence_device(hb200_ctx* c) {
  const int Nv = c->Nv, Ni = c->Ni, Nm = c->Nm, L = c->L, K = c->K;
  c->nseg = K - c->k + 1;
  HB_CUDA(c->w_scal.ensure(8));
  HB_CUDA(cudaMemsetAsync(c->w_scal.p, 0, 8 * sizeof(int), c->stream));
  HB_CUDA(c->lm_off.ensure(static_cast<size_t>(L) + 2)); HB_CUDA(c->lm_obs.ensure(std::max(Nv, 1)));
  HB_CUDA(c->seg_off.ensure(static_cast<size_t>(c->nseg) + 2)); HB_CUDA(c->run_off.ensure(static_cast<size_t>(Ni) + 2));
  HB_CUDA(c->w_cnt.ensure(static_cast<size_t>(std::max(std::max(L, c->nseg), 1)) + 1));
  HB_CUDA(c->w_keep.ensure(std::max(std::max(Nv, Ni), 1))); HB_CUDA(c->w_pos.ensure(std::max(std::max(Nv, Ni), 1)));
  // landmark CSR
  HB_CUDA(cudaMemsetAsync(c->w_cnt.p, 0, sizeof(int) * (static_cast<size_t>(L) + 1), c->stream));
  if (Nv) { count_kernel<<<(Nv + 255) / 256, 256, 0, c->stream>>>(Nv, c->v_idx.p, 1, c->w_cnt.p); HB_LAUNCH(c, "count_kernel"); }
  scan_kernel<<<1, 1024, 0, c->stream>>>(c->w_cnt.p, L + 1, c->lm_off.p, c->w_scal.p + 0);
  HB_LAUNCH(c, "scan_kernel");
  HB_CUDA(cudaMemsetAsync(c->w_cnt.p, 0, sizeof(int) * (static_cast<size_t>(L) + 1), c->stream));
  if (Nv) {
    csr_fill_kernel<<<(Nv + 255) / 256, 256, 0, c->stream>>>(Nv, c->v_idx.p, c->lm_off.p, c->w_cnt.p, c->lm_obs.p);
    HB_LAUNCH(c, "csr_fill_kernel");
    csr_sort_kernel<<<(L + 127) / 128, 128, 0, c->stream>>>(L, c->lm_off.p, c->lm_obs.p, c->v_idx.p, c->k, c->w_scal.p + 1);
    HB_LAUNCH(c, "csr_sort_kernel");
  }
  // segment offsets of the visual list
  HB_CUDA(cudaMemsetAsync(c->w_cnt.p, 0, sizeof(int) * (static_cast<size_t>(c->nseg) + 1), c->stream));
  if (Nv) { count_kernel<<<(Nv + 255) / 256, 256, 0, c->stream>>>(Nv, c->v_idx.p, 0, c->w_cnt.p); HB_LAUNCH(c, "count_kernel"); }
  scan_kernel<<<1, 1024, 0, c->stream>>>(c->w_cnt.p, c->nseg + 1, c->seg_off.p, c->w_scal.p + 2);
  HB_LAUNCH(c, "scan_kernel");
  // inertial runs
  if (Ni) {
    run_flag_kernel<<<(Ni + 255) / 256, 256, 0, c->stream>>>(Ni, c->i_idx.p, c->w_keep.p);
    HB_LAUNCH(c, "run_flag_kernel");
    scan_kernel<<<1, 1024, 0, c->stream>>>(c->w_keep.p, Ni, c->w_pos.p, c->w_scal.p + 3);
    HB_LAUNCH(c, "scan_kernel");
  }
  int h[8];
  HB_CUDA(cudaMemcpyAsync(h, c->w_scal.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->max_rows = std::max(6 * c->k, h[1]);
  c->schur_groups = false;   // (the groups are cut on the host at hb200_bind; after device-side bookkeeping the per-landmark kernel runs)
  c->nruns = Ni ? h[3] : 0;
  if (Ni) { run_fill_kernel<<<(Ni + 255) / 256, 256, 0, c->stream>>>(Ni, c->w_keep.p, c->w_pos.p, c->nruns, c->run_off.p); HB_LAUNCH(c, "run_fill_kernel"); }
  else { const int z = 0; HB_CUDA(cudaMemcpyAsync(c->run_off.p, &z, sizeof(int), cudaMemcpyHostToDevice, c->stream)); }
  if (2 * 3 * static_cast<size_t>(c->max_rows) * sizeof(double) > 200 * 1024) return fail(-6, "landmark track spans %d control-point dofs; exceeds the Schur kernel's shared-memory tile", c->max_rows);
  // outputs and launch shapes (as hb200_bind)
  const size_t k = c->k;
  HB_CUDA(c->v_z.grow(std::max(Nv, 1), Nv, c->stream)); HB_CUDA(c->v_w.ensure(std::max(Nv, 1)));   // (v_z holds the bearings' third components)
  HB_CUDA(c->v_r.ensure(2 * static_cast<size_t>(std::max(Nv, 1)))); HB_CUDA(c->v_Jp.ensure(12 * k * std::max(Nv, 1))); HB_CUDA(c->v_Jl.ensure(6 * static_cast<size_t>(std::max(Nv, 1))));
  HB_CUDA(c->i_r.ensure(6 * static_cast<size_t>(std::max(Ni, 1)))); HB_CUDA(c->i_Jp.ensure(36 * k * std::max(Ni, 1)));
  HB_CUDA(c->i_wg.ensure(4 * static_cast<size_t>(std::max(Ni, 1)))); HB_CUDA(c->i_wa.ensure(4 * static_cast<size_t>(std::max(Ni, 1)))); HB_CUDA(c->i_Jg.ensure(12 * static_cast<size_t>(std::max(Ni, 1))));
  c->n_pix_blocks = (Nv + kEvalThreads - 1) / kEvalThreads;
  c->n_imu_blocks = (Ni + kEvalThreads - 1) / kEvalThreads;
  c->n_man_blocks = (Nm + kEvalThreads - 1) / kEvalThreads;
  HB_CUDA(c->m_r.ensure(6 * static_cast<size_t>(std::max(Nm, 1)))); HB_CUDA(c->m_Jp.ensure(36 * k * std::max(Nm, 1)));
  for (int s2 = 0; s2 < 2; ++s2) { HB_CUDA(c->cp_pix[s2].ensure(std::max(c->n_pix_blocks, 1))); HB_CUDA(c->cp_imu[s2].ensure(std::max(c->n_imu_blocks + c->n_man_blocks, 1))); }
  if (c->max_rows * 6 * sizeof(double) > 48 * 1024) {
    const int smem = static_cast<int>(2 * 3 * static_cast<size_t>(c->max_rows) * sizeof(double));
    HB_CUDA(cudaFuncSetAttribute(schur_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    HB_CUDA(cudaFuncSetAttribute(schur_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  }
  int rc = update_fixed(c);
  if (rc) return rc;
  if ((rc = ensure_system(c))) return rc;
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->bound = true;
  c->device_managed = true;
  c->invalidate();
  c->have_snapshot = false;
  return sync_layout(c);
}
}  // namespace

extern "C" {

int hb200_bind(hb200_ctx* c, int* num_invalid) {
  if (!c) return fail(-1, "null context");
  { const int rs = sync_host_mirrors(c); if (rs) return rs; }
  if (c->K == 0) return fail(-2, "spline not set");
  if (c->Ni && (c->Kbg == 0 || c->Kba == 0)) return fail(-2, "bias splines not set");
  if (c->Nv && (c->C == 0 || c->L == 0)) return fail(-2, "cameras / landmarks not set");
  if (c->Nm && c->P == 0) return fail(-2, "pose sensors not set");
  HB_CUDA(cudaSetDevice(c->device));
  const int Nv = c->Nv, Ni = c->Ni, Nm = c->Nm;
  HB_CUDA(c->d_invalid.ensure(1));
  HB_CUDA(cudaMemsetAsync(c->d_invalid.p, 0, sizeof(int), c->stream));
  HB_CUDA(c->v_stamp.ensure(std::max(Nv, 1))); HB_CUDA(c->v_pixel.ensure(2 * static_cast<size_t>(std::max(Nv, 1))));
  HB_CUDA(c->v_cam.ensure(std::max(Nv, 1))); HB_CUDA(c->v_lm.ensure(std::max(Nv, 1))); HB_CUDA(c->v_idx.ensure(std::max(Nv, 1)));
  HB_CUDA(c->v_z.ensure(std::max(Nv, 1))); HB_CUDA(c->v_w.ensure(std::max(Nv, 1)));
  HB_CUDA(c->m_stamp.ensure(std::max(Nm, 1))); HB_CUDA(c->m_meas.ensure(7 * static_cast<size_t>(std::max(Nm, 1)))); HB_CUDA(c->m_sensor.ensure(std::max(Nm, 1)));
  HB_CUDA(c->m_idx.ensure(std::max(Nm, 1)));
  c->h_m_idx.assign(Nm, make_int2(0, 0));
  HB_CUDA(c->i_stamp.ensure(std::max(Ni, 1))); HB_CUDA(c->i_meas.ensure(6 * static_cast<size_t>(std::max(Ni, 1)))); HB_CUDA(c->i_idx.ensure(std::max(Ni, 1)));
  c->h_v_idx.assign(Nv, make_int4(0, 0, 0, 0)); c->h_i_idx.assign(Ni, make_int4(0, 0, 0, 0));
  // pass 1: index maps in user order (device), a2/a4
  if (Nv) {
    HB_CUDA(cudaMemcpyAsync(c->v_stamp.p, c->h_v_stamp.data(), sizeof(double) * Nv, cudaMemcpyHostToDevice, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->v_cam.p, c->h_v_cam.data(), sizeof(int) * Nv, cudaMemcpyHostToDevice, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->v_lm.p, c->h_v_lm.data(), sizeof(int) * Nv, cudaMemcpyHostToDevice, c->stream));
    bind_pixel_kernel<<<(Nv + 127) / 128, 128, 0, c->stream>>>(Nv, c->v_stamp.p, c->v_cam.p, c->v_lm.p, c->knots[0].p, c->K, c->k, c->C, c->L, 0, c->v_idx.p, c->d_invalid.p);
    HB_LAUNCH(c, "bind_pixel_kernel");
    HB_CUDA(cudaMemcpyAsync(c->h_v_idx.data(), c->v_idx.p, sizeof(int4) * Nv, cudaMemcpyDeviceToHost, c->stream));
  }
  if (Ni) {
    HB_CUDA(cudaMemcpyAsync(c->i_stamp.p, c->h_i_stamp.data(), sizeof(double) * Ni, cudaMemcpyHostToDevice, c->stream));
    bind_inertial_kernel<<<(Ni + 127) / 128, 128, 0, c->stream>>>(Ni, c->i_stamp.p, c->knots[0].p, c->K, c->k, c->bg[0].p, c->Kbg, c->ba[0].p, c->Kba, c->kb,
                                                               c->i_idx.p, c->d_invalid.p);
    HB_LAUNCH(c, "bind_inertial_kernel");
    HB_CUDA(cudaMemcpyAsync(c->h_i_idx.data(), c->i_idx.p, sizeof(int4) * Ni, cudaMemcpyDeviceToHost, c->stream));
  }
  if (Nm) {
    HB_CUDA(cudaMemcpyAsync(c->m_stamp.p, c->h_m_stamp.data(), sizeof(double) * Nm, cudaMemcpyHostToDevice, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->m_meas.p, c->h_m_meas.data(), sizeof(double) * 7 * Nm, cudaMemcpyHostToDevice, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->m_sensor.p, c->h_m_sensor.data(), sizeof(int) * Nm, cudaMemcpyHostToDevice, c->stream));
    bind_manifold_kernel<<<(Nm + 127) / 128, 128, 0, c->stream>>>(Nm, c->m_stamp.p, c->m_sensor.p, c->knots[0].p, c->K, c->k, c->P, c->m_idx.p, c->d_invalid.p);
    HB_LAUNCH(c, "bind_manifold_kernel");
    HB_CUDA(cudaMemcpyAsync(c->h_m_idx.data(), c->m_idx.p, sizeof(int2) * Nm, cudaMemcpyDeviceToHost, c->stream));
  }
  int invalid = 0;
  HB_CUDA(cudaMemcpyAsync(&invalid, c->d_invalid.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if (num_invalid) *num_invalid = invalid;
  if (invalid) return fail(2, "%d factor(s) reference a stamp outside the spline's valid range or an invalid camera / landmark / sensor", invalid);
  for (int u = c->Np; u < Nv; ++u) c->h_v_idx[u].w = 1;   // bearing factors

  // pass 2: bound order = stable sort by knot base index (pixel) / (base, gyro base, accel base)
  c->v_perm.resize(Nv); std::iota(c->v_perm.begin(), c->v_perm.end(), 0);
  c->i_perm.resize(Ni); std::iota(c->i_perm.begin(), c->i_perm.end(), 0);
  {
    const std::vector<int4>& id = c->h_v_idx;
    if (!std::is_sorted(id.begin(), id.end(), [](const int4& a, const int4& b) { return a.x < b.x; }))
      std::stable_sort(c->v_perm.begin(), c->v_perm.end(), [&](int a, int b) { return id[a].x < id[b].x; });
    auto key = [](const int4& a, const int4& b) { return a.x != b.x ? a.x < b.x : (a.y != b.y ? a.y < b.y : a.z < b.z); };
    const std::vector<int4>& ii = c->h_i_idx;
    if (!std::is_sorted(ii.begin(), ii.end(), key)) std::stable_sort(c->i_perm.begin(), c->i_perm.end(), [&](int a, int b) { return key(ii[a], ii[b]); });
  }
  {
    std::vector<double> st(Nv), px(2 * static_cast<size_t>(Nv)), vz(Nv);
    std::vector<int4> id(Nv);
    for (int p = 0; p < Nv; ++p) { const int u = c->v_perm[p]; st[p] = c->h_v_stamp[u]; px[2 * p] = c->h_v_pixel[2 * u]; px[2 * p + 1] = c->h_v_pixel[2 * u + 1]; vz[p] = c->h_v_z[u]; id[p] = c->h_v_idx[u]; }
    c->h_v_idx = id;
    if (Nv) {
      HB_CUDA(cudaMemcpyAsync(c->v_stamp.p, st.data(), sizeof(double) * Nv, cudaMemcpyHostToDevice, c->stream));
      HB_CUDA(cudaMemcpyAsync(c->v_pixel.p, px.data(), sizeof(double) * 2 * Nv, cudaMemcpyHostToDevice, c->stream));
      HB_CUDA(cudaMemcpyAsync(c->v_z.p, vz.data(), sizeof(double) * Nv, cudaMemcpyHostToDevice, c->stream));
      HB_CUDA(cudaMemcpyAsync(c->v_idx.p, id.data(), sizeof(int4) * Nv, cudaMemcpyHostToDevice, c->stream));
    }
    std::vector<double> is(Ni), im(6 * static_cast<size_t>(Ni));
    std::vector<int4> iid(Ni);
    for (int p = 0; p < Ni; ++p) { const int u = c->i_perm[p]; is[p] = c->h_i_stamp[u]; for (int q = 0; q < 6; ++q) im[6 * p + q] = c->h_i_meas[6 * u + q]; iid[p] = c->h_i_idx[u]; }
    c->h_i_idx = iid;
    if (Ni) {
      HB_CUDA(cudaMemcpyAsync(c->i_stamp.p, is.data(), sizeof(double) * Ni, cudaMemcpyHostToDevice, c->stream));
      HB_CUDA(cudaMemcpyAsync(c->i_meas.p, im.data(), sizeof(double) * 6 * Ni, cudaMemcpyHostToDevice, c->stream));
      HB_CUDA(cudaMemcpyAsync(c->i_idx.p, iid.data(), sizeof(int4) * Ni, cudaMemcpyHostToDevice, c->stream));
    }
    HB_CUDA(cudaStreamSynchronize(c->stream));
  }
  // segment offsets (pixel), runs (inertial), landmark incidence (CSR)
  c->nseg = c->K - c->k + 1;
  std::vector<int> seg(c->nseg + 1, 0);
  for (int p = 0; p < Nv; ++p) seg[c->h_v_idx[p].x + 1] += 1;
  for (int s = 0; s < c->nseg; ++s) seg[s + 1] += seg[s];
  std::vector<int> runs;
  for (int p = 0; p < Ni; ++p) {
    const int4& a = c->h_i_idx[p];
    if (p == 0 || a.x != c->h_i_idx[p - 1].x || a.y != c->h_i_idx[p - 1].y || a.z != c->h_i_idx[p - 1].z) runs.push_back(p);
  }
  c->nruns = static_cast<int>(runs.size());
  runs.push_back(Ni);
  std::vector<int> off(c->L + 1, 0), obs(std::max(Nv, 1));
  for (int p = 0; p < Nv; ++p) off[c->h_v_idx[p].y + 1] += 1;
  for (int l = 0; l < c->L; ++l) off[l + 1] += off[l];
  {
    std::vector<int> cur(off.begin(), off.end() - 1);
    for (int p = 0; p < Nv; ++p) obs[cur[c->h_v_idx[p].y]++] = p;
  }
  c->max_rows = 6 * c->k;
  for (int l = 0; l < c->L; ++l)
    if (off[l + 1] > off[l]) c->max_rows = std::max(c->max_rows, 6 * (c->h_v_idx[obs[off[l + 1] - 1]].x + c->k - c->h_v_idx[obs[off[l]]].x));
  if (2 * 3 * static_cast<size_t>(c->max_rows) * sizeof(double) > 200 * 1024) return fail(-6, "landmark track spans %d control-point dofs; exceeds the Schur kernel's shared-memory tile", c->max_rows);
  HB_CUDA(c->seg_off.ensure(seg.size())); HB_CUDA(c->run_off.ensure(runs.size())); HB_CUDA(c->lm_off.ensure(off.size())); HB_CUDA(c->lm_obs.ensure(obs.size()));
  HB_CUDA(cudaMemcpyAsync(c->seg_off.p, seg.data(), sizeof(int) * seg.size(), cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->run_off.p, runs.data(), sizeof(int) * runs.size(), cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->lm_off.p, off.data(), sizeof(int) * off.size(), cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->lm_obs.p, obs.data(), sizeof(int) * obs.size(), cudaMemcpyHostToDevice, c->stream));
  {
    // landmark groups for the large-window Schur kernel: observed landmarks ordered by their first knot base, cut so that
    // a group has at most kSchurGroup members and its control-point rows fit one window of RT rows
    static const int min_lm = getenv("HB200_SCHUR_GROUP_MIN") ? atoi(getenv("HB200_SCHUR_GROUP_MIN")) : 8192;
    c->schur_groups = false;
    c->schur_rt = ((c->max_rows + 12 + 7) / 8) * 8;
    if (c->L >= min_lm && Nv) {
      std::vector<int> order;
      order.reserve(c->L);
      for (int l = 0; l < c->L; ++l) if (off[l + 1] > off[l]) order.push_back(l);
      auto first_base = [&](int l) { return c->h_v_idx[obs[off[l]]].x; };
      std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return first_base(a) < first_base(b); });
      std::vector<int> goff;
      const int win = c->schur_rt / 6;   // control points per window
      int glo = 0;
      for (size_t i = 0; i < order.size(); ++i) {
        const int l = order[i];
        const int lo = first_base(l), hi = c->h_v_idx[obs[off[l + 1] - 1]].x + c->k;
        if (goff.empty() || static_cast<int>(i) - goff.back() >= kSchurGroup || hi - glo > win) { goff.push_back(static_cast<int>(i)); glo = lo; }
      }
      c->n_lm_groups = static_cast<int>(goff.size());
      goff.push_back(static_cast<int>(order.size()));
      HB_CUDA(c->lm_order.ensure(std::max<size_t>(order.size(), 1))); HB_CUDA(c->lm_group_off.ensure(goff.size()));
      HB_CUDA(cudaMemcpyAsync(c->lm_order.p, order.data(), sizeof(int) * order.size(), cudaMemcpyHostToDevice, c->stream));
      HB_CUDA(cudaMemcpyAsync(c->lm_group_off.p, goff.data(), sizeof(int) * goff.size(), cudaMemcpyHostToDevice, c->stream));
      HB_CUDA(cudaStreamSynchronize(c->stream));
      c->schur_groups = c->n_lm_groups > 0;
      const size_t smem = (3 * static_cast<size_t>(kSchurGroup) * (c->schur_rt + 1) + 3 * kSchurGroup + 4 * 3 * static_cast<size_t>(c->schur_rt)) * sizeof(double);
      if (smem > 200 * 1024) c->schur_groups = false;
      else {
        HB_CUDA(cudaFuncSetAttribute(schur_group_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        HB_CUDA(cudaFuncSetAttribute(schur_group_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
      }
    }
  }
  // outputs
  const size_t k = c->k;
  HB_CUDA(c->v_r.ensure(2 * static_cast<size_t>(std::max(Nv, 1)))); HB_CUDA(c->v_Jp.ensure(12 * k * std::max(Nv, 1))); HB_CUDA(c->v_Jl.ensure(6 * static_cast<size_t>(std::max(Nv, 1))));
  HB_CUDA(c->i_r.ensure(6 * static_cast<size_t>(std::max(Ni, 1)))); HB_CUDA(c->i_Jp.ensure(36 * k * std::max(Ni, 1)));
  HB_CUDA(c->i_wg.ensure(4 * static_cast<size_t>(std::max(Ni, 1)))); HB_CUDA(c->i_wa.ensure(4 * static_cast<size_t>(std::max(Ni, 1)))); HB_CUDA(c->i_Jg.ensure(12 * static_cast<size_t>(std::max(Ni, 1))));
  c->n_pix_blocks = (Nv + kEvalThreads - 1) / kEvalThreads;
  c->n_imu_blocks = (Ni + kEvalThreads - 1) / kEvalThreads;
  c->n_man_blocks = (Nm + kEvalThreads - 1) / kEvalThreads;
  HB_CUDA(c->m_r.ensure(6 * static_cast<size_t>(std::max(Nm, 1)))); HB_CUDA(c->m_Jp.ensure(36 * k * std::max(Nm, 1)));
  for (int s = 0; s < 2; ++s) { HB_CUDA(c->cp_pix[s].ensure(std::max(c->n_pix_blocks, 1))); HB_CUDA(c->cp_imu[s].ensure(std::max(c->n_imu_blocks + c->n_man_blocks, 1))); }
  if (c->max_rows * 6 * sizeof(double) > 48 * 1024) {
    const int smem = static_cast<int>(2 * 3 * static_cast<size_t>(c->max_rows) * sizeof(double));
    HB_CUDA(cudaFuncSetAttribute(schur_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    HB_CUDA(cudaFuncSetAttribute(schur_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  }
  int rc = update_fixed(c);
  if (rc) return rc;
  rc = ensure_system(c);
  if (rc) return rc;
  if (c->schur_groups) {   // unobserved landmarks are not in any group: their blocks stay zero (no step)
    HB_CUDA(cudaMemsetAsync(c->Vinv.p, 0, sizeof(double) * 9 * static_cast<size_t>(std::max(c->L, 1)), c->stream));
    HB_CUDA(cudaMemsetAsync(c->gl.p, 0, sizeof(double) * 3 * static_cast<size_t>(std::max(c->L, 1)), c->stream));
    HB_CUDA(cudaMemsetAsync(c->Dl.p, 0, sizeof(double) * 3 * static_cast<size_t>(std::max(c->L, 1)), c->stream));
  }
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->bound = true;
  c->invalidate();
  return sync_layout(c);   // multi-GPU: all ranks adopt the widest band (collective when a communicator is attached)
}

int hb200_get_index_maps(hb200_ctx* c, int* pixel_base, int* inertial_base, int* gyro_bias_base, int* accel_bias_base) {
  if (!c || !c->bound) return fail(-2, "not bound");
  { const int rs = sync_host_mirrors(c); if (rs) return rs; }
  for (int p = 0; p < c->Nv; ++p) if (pixel_base && c->v_perm[p] < c->Np) pixel_base[c->v_perm[p]] = c->h_v_idx[p].x;
  for (int p = 0; p < c->Ni; ++p) {
    const int u = c->i_perm[p];
    if (inertial_base) inertial_base[u] = c->h_i_idx[p].x;
    if (gyro_bias_base) gyro_bias_base[u] = c->h_i_idx[p].y;
    if (accel_bias_base) accel_bias_base[u] = c->h_i_idx[p].z;
  }
  return 0;
}

int hb200_evaluate(hb200_ctx* c, int flags) {
  int rc = check_ready(c);
  if (rc) return rc;
  HB_CUDA(cudaSetDevice(c->device));
  const bool J = flags & HB200_EVAL_JACOBIANS;
  const int sel = (flags & HB200_EVAL_TRIAL) ? 1 : 0;
  rc = enqueue_evaluate(c, J, sel);
  if (rc) return rc;
  c->evaluated_J = J && sel == 0;   // a trial-state sweep overwrites the residual / Jacobian buffers
  c->mirror_valid = false; c->calib_valid = false; c->system_built = false;
  return 0;
}

int hb200_get_pixel_outputs(hb200_ctx* c, double* r, double* Jp, double* Jl) {
  if (!c || !c->bound) return fail(-2, "not bound");
  { const int rs = sync_host_mirrors(c); if (rs) return rs; }
  HB_CUDA(cudaSetDevice(c->device));
  const size_t N = c->Nv, w = 12 * static_cast<size_t>(c->k);
  std::vector<double> tr(2 * N), tJ(Jp ? w * N : 0), tl(Jl ? 6 * N : 0);
  if (N) {
    HB_CUDA(cudaMemcpyAsync(tr.data(), c->v_r.p, sizeof(double) * 2 * N, cudaMemcpyDeviceToHost, c->stream));
    if (Jp) HB_CUDA(cudaMemcpyAsync(tJ.data(), c->v_Jp.p, sizeof(double) * w * N, cudaMemcpyDeviceToHost, c->stream));
    if (Jl) HB_CUDA(cudaMemcpyAsync(tl.data(), c->v_Jl.p, sizeof(double) * 6 * N, cudaMemcpyDeviceToHost, c->stream));
  }
  HB_CUDA(cudaStreamSynchronize(c->stream));
  for (size_t p = 0; p < N; ++p) {
    const size_t u = c->v_perm[p];
    if (u >= static_cast<size_t>(c->Np)) continue;   // bearing factor
    if (r) { r[2 * u] = tr[2 * p]; r[2 * u + 1] = tr[2 * p + 1]; }
    if (Jp) std::memcpy(Jp + w * u, tJ.data() + w * p, sizeof(double) * w);
    if (Jl) std::memcpy(Jl + 6 * u, tl.data() + 6 * p, sizeof(double) * 6);
  }
  return 0;
}

int hb200_get_bearing_outputs(hb200_ctx* c, double* r, double* Jp, double* Jl) {
  if (!c || !c->bound) return fail(-2, "not bound");
  { const int rs = sync_host_mirrors(c); if (rs) return rs; }
  HB_CUDA(cudaSetDevice(c->device));
  const size_t N = c->Nv, w = 12 * static_cast<size_t>(c->k);
  if (c->Nb == 0) return 0;
  std::vector<double> tr(2 * N), tJ(Jp ? w * N : 0), tl(Jl ? 6 * N : 0);
  HB_CUDA(cudaMemcpyAsync(tr.data(), c->v_r.p, sizeof(double) * 2 * N, cudaMemcpyDeviceToHost, c->stream));
  if (Jp) HB_CUDA(cudaMemcpyAsync(tJ.data(), c->v_Jp.p, sizeof(double) * w * N, cudaMemcpyDeviceToHost, c->stream));
  if (Jl) HB_CUDA(cudaMemcpyAsync(tl.data(), c->v_Jl.p, sizeof(double) * 6 * N, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  for (size_t p = 0; p < N; ++p) {
    if (c->v_perm[p] < c->Np) continue;
    const size_t u = c->v_perm[p] - c->Np;   // first row of the 2-row slot carries the angular residual
    if (r) r[u] = tr[2 * p];
    if (Jp) std::memcpy(Jp + (w / 2) * u, tJ.data() + w * p, sizeof(double) * (w / 2));
    if (Jl) std::memcpy(Jl + 3 * u, tl.data() + 6 * p, sizeof(double) * 3);
  }
  return 0;
}

int hb200_get_manifold_outputs(hb200_ctx* c, double* r, double* Jp) {
  if (!c || !c->bound) return fail(-2, "not bound");
  HB_CUDA(cudaSetDevice(c->device));
  const size_t N = c->Nm, w = 36 * static_cast<size_t>(c->k);
  if (N == 0) return 0;
  if (r) HB_CUDA(cudaMemcpyAsync(r, c->m_r.p, sizeof(double) * 6 * N, cudaMemcpyDeviceToHost, c->stream));
  if (Jp) HB_CUDA(cudaMemcpyAsync(Jp, c->m_Jp.p, sizeof(double) * w * N, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int hb200_get_inertial_outputs(hb200_ctx* c, double* r, double* Jp, double* wg, double* wa, double* Jg) {
  if (!c || !c->bound) return fail(-2, "not bound");
  { const int rs = sync_host_mirrors(c); if (rs) return rs; }
  HB_CUDA(cudaSetDevice(c->device));
  const size_t N = c->Ni, w = 36 * static_cast<size_t>(c->k);
  std::vector<double> tr(6 * N), tJ(Jp ? w * N : 0), tg(wg ? 4 * N : 0), ta(wa ? 4 * N : 0), tG(Jg ? 12 * N : 0);
  if (N) {
    HB_CUDA(cudaMemcpyAsync(tr.data(), c->i_r.p, sizeof(double) * 6 * N, cudaMemcpyDeviceToHost, c->stream));
    if (Jp) HB_CUDA(cudaMemcpyAsync(tJ.data(), c->i_Jp.p, sizeof(double) * w * N, cudaMemcpyDeviceToHost, c->stream));
    if (wg) HB_CUDA(cudaMemcpyAsync(tg.data(), c->i_wg.p, sizeof(double) * 4 * N, cudaMemcpyDeviceToHost, c->stream));
    if (wa) HB_CUDA(cudaMemcpyAsync(ta.data(), c->i_wa.p, sizeof(double) * 4 * N, cudaMemcpyDeviceToHost, c->stream));
    if (Jg) HB_CUDA(cudaMemcpyAsync(tG.data(), c->i_Jg.p, sizeof(double) * 12 * N, cudaMemcpyDeviceToHost, c->stream));
  }
  HB_CUDA(cudaStreamSynchronize(c->stream));
  for (size_t p = 0; p < N; ++p) {
    const size_t u = c->i_perm[p];
    if (r) std::memcpy(r + 6 * u, tr.data() + 6 * p, sizeof(double) * 6);
    if (Jp) std::memcpy(Jp + w * u, tJ.data() + w * p, sizeof(double) * w);
    if (wg) std::memcpy(wg + 4 * u, tg.data() + 4 * p, sizeof(double) * 4);
    if (wa) std::memcpy(wa + 4 * u, ta.data() + 4 * p, sizeof(double) * 4);
    if (Jg) std::memcpy(Jg + 12 * u, tG.data() + 12 * p, sizeof(double) * 12);
  }
  return 0;
}

}  // extern "C"

namespace {
// rows of a tangent-space SE3 Jacobian [d/dtheta | d/drho] -> ambient [q(4) | p(3)] through the SE3JacobianAdapter
// (reference pixel.cpp:141, inertial.cpp:161): J_theta A_q(q) | J_rho
void tangent_to_ambient_se3(const double* Jt, int ld, int rows, const double* T, double* out /*rows x 7*/) {
  const double* q = T;
  const double Aq[12] = {2 * q[3], -2 * q[2], 2 * q[1], -2 * q[0], 2 * q[2], 2 * q[3], -2 * q[0], -2 * q[1], -2 * q[1], 2 * q[0], 2 * q[3], -2 * q[2]};
  for (int row = 0; row < rows; ++row) {
    const double* jt = Jt + static_cast<size_t>(ld) * row;
    double* o = out + 7 * row;
    for (int col = 0; col < 4; ++col) o[col] = jt[0] * Aq[col] + jt[1] * Aq[4 + col] + jt[2] * Aq[8 + col];
    o[4] = jt[3]; o[5] = jt[4]; o[6] = jt[5];
  }
}

// calibration-block Jacobians of every factor at the current state, mirrored to the host in user order
int ensure_calib_mirror(hb200_ctx* c) {
  HB_CUDA(cudaSetDevice(c->device));
  const size_t Nv = c->Nv, Ni = c->Ni, Nm = c->Nm;
  DevBuf<double> dv, di, dm;
  std::vector<double> tv(28 * Nv), ti(216 * Ni);
  c->m_v_Jc.assign(28 * Nv, 0.0); c->m_i_Jc.assign(216 * Ni, 0.0); c->m_m_Jc.assign(36 * Nm, 0.0);
  if (Nv) {
    HB_CUDA(dv.ensure(28 * Nv));
    const int blocks = static_cast<int>((Nv + kEvalThreads - 1) / kEvalThreads);
    if (c->k == 4) pixel_calib_kernel<4><<<blocks, kEvalThreads, 0, c->stream>>>(c->Nv, c->v_stamp.p, reinterpret_cast<const double2*>(c->v_pixel.p), c->v_z.p, c->v_idx.p, c->tab[0].p, c->cam_tab.p, c->lms[0].p, c->basis, dv.p);
    else pixel_calib_kernel<6><<<blocks, kEvalThreads, 0, c->stream>>>(c->Nv, c->v_stamp.p, reinterpret_cast<const double2*>(c->v_pixel.p), c->v_z.p, c->v_idx.p, c->tab[0].p, c->cam_tab.p, c->lms[0].p, c->basis, dv.p);
    HB_LAUNCH(c, "pixel_calib_kernel");
    HB_CUDA(cudaMemcpyAsync(tv.data(), dv.p, sizeof(double) * 28 * Nv, cudaMemcpyDeviceToHost, c->stream));
  }
  if (Ni) {
    HB_CUDA(di.ensure(216 * Ni));
    const int blocks = static_cast<int>((Ni + kEvalThreads - 1) / kEvalThreads);
    if (c->k == 4) inertial_calib_kernel<4><<<blocks, kEvalThreads, 0, c->stream>>>(c->Ni, c->i_stamp.p, c->i_idx.p, c->tab[0].p, c->imu.p, c->grav[0].p, c->basis, c->quirks, di.p);
    else inertial_calib_kernel<6><<<blocks, kEvalThreads, 0, c->stream>>>(c->Ni, c->i_stamp.p, c->i_idx.p, c->tab[0].p, c->imu.p, c->grav[0].p, c->basis, c->quirks, di.p);
    HB_LAUNCH(c, "inertial_calib_kernel");
    HB_CUDA(cudaMemcpyAsync(ti.data(), di.p, sizeof(double) * 216 * Ni, cudaMemcpyDeviceToHost, c->stream));
  }
  if (Nm) {
    HB_CUDA(dm.ensure(36 * Nm));
    const int blocks = static_cast<int>((Nm + kEvalThreads - 1) / kEvalThreads);
    if (c->k == 4) manifold_calib_kernel<4><<<blocks, kEvalThreads, 0, c->stream>>>(c->Nm, c->m_stamp.p, c->m_meas.p, c->m_idx.p, c->tab[0].p, c->sensors.p, c->basis, dm.p);
    else manifold_calib_kernel<6><<<blocks, kEvalThreads, 0, c->stream>>>(c->Nm, c->m_stamp.p, c->m_meas.p, c->m_idx.p, c->tab[0].p, c->sensors.p, c->basis, dm.p);
    HB_LAUNCH(c, "manifold_calib_kernel");
    HB_CUDA(cudaMemcpyAsync(c->m_m_Jc.data(), dm.p, sizeof(double) * 36 * Nm, cudaMemcpyDeviceToHost, c->stream));
  }
  HB_CUDA(cudaStreamSynchronize(c->stream));
  for (size_t p = 0; p < Nv; ++p) std::memcpy(&c->m_v_Jc[28 * static_cast<size_t>(c->v_perm[p])], &tv[28 * p], 28 * sizeof(double));   // pixel [0, Np), bearing after
  for (size_t p = 0; p < Ni; ++p) std::memcpy(&c->m_i_Jc[216 * static_cast<size_t>(c->i_perm[p])], &ti[216 * p], 216 * sizeof(double));
  c->calib_valid = true;
  return 0;
}
}  // namespace

extern "C" {

int hb200_factor_evaluate(hb200_ctx* c, int kind, int index, const double* const* parameters, double* residuals, double** jacobians) {
  if (!c || !c->bound) return fail(-2, "not bound");
  if (!c->evaluated_J) return fail(-2, "call hb200_evaluate(HB200_EVAL_JACOBIANS) first");
  if (!parameters || !residuals) return fail(-1, "null argument");
  if (!c->mirror_valid) {
    const size_t k = c->k;
    c->m_v_r.resize(2 * static_cast<size_t>(c->Np)); c->m_v_Jp.resize(12 * k * c->Np); c->m_v_Jl.resize(6 * static_cast<size_t>(c->Np));
    c->m_b_r.resize(c->Nb); c->m_b_Jp.resize(6 * k * c->Nb); c->m_b_Jl.resize(3 * static_cast<size_t>(c->Nb));
    c->m_m_r.resize(6 * static_cast<size_t>(c->Nm)); c->m_m_Jp.resize(36 * k * c->Nm);
    c->m_i_r.resize(6 * static_cast<size_t>(c->Ni)); c->m_i_Jp.resize(36 * k * c->Ni); c->m_i_wg.resize(4 * static_cast<size_t>(c->Ni));
    c->m_i_wa.resize(4 * static_cast<size_t>(c->Ni)); c->m_i_Jg.resize(12 * static_cast<size_t>(c->Ni)); c->m_grav.resize(3);
    int rc = hb200_get_pixel_outputs(c, c->m_v_r.data(), c->m_v_Jp.data(), c->m_v_Jl.data());
    if (rc) return rc;
    rc = hb200_get_inertial_outputs(c, c->m_i_r.data(), c->m_i_Jp.data(), c->m_i_wg.data(), c->m_i_wa.data(), c->m_i_Jg.data());
    if (rc) return rc;
    rc = hb200_get_bearing_outputs(c, c->m_b_r.data(), c->m_b_Jp.data(), c->m_b_Jl.data());
    if (rc) return rc;
    rc = hb200_get_manifold_outputs(c, c->m_m_r.data(), c->m_m_Jp.data());
    if (rc) return rc;
    HB_CUDA(cudaMemcpy(c->m_grav.data(), c->grav[0].p, 3 * sizeof(double), cudaMemcpyDeviceToHost));
    c->mirror_valid = true;
  }
  const int k = c->k, kb = c->kb;
  if (kind < HB200_PIXEL || kind > HB200_MANIFOLD) return fail(-1, "unknown factor kind %d", kind);
  if (jacobians && !c->calib_valid) {
    // calibration blocks requested?  (constant in the live configuration, so they are produced on demand only)
    const int first = k, count = (kind == HB200_INERTIAL) ? 5 : (kind == HB200_MANIFOLD ? 1 : 3);
    bool want = false;
    for (int b = 0; b < count; ++b) want = want || jacobians[first + b] != nullptr;
    if (want) { const int rc = ensure_calib_mirror(c); if (rc) return rc; }
  }
  const int nrs[4] = {2, 6, 1, 6};
  const int Ns[4] = {c->Np, c->Ni, c->Nb, c->Nm};
  const int nr = nrs[kind], N = Ns[kind];
  if (index < 0 || index >= N) return fail(-1, "factor index %d out of range", index);
  const double* rs[4] = {c->m_v_r.data(), c->m_i_r.data(), c->m_b_r.data(), c->m_m_r.data()};
  const double* Js[4] = {c->m_v_Jp.data(), c->m_i_Jp.data(), c->m_b_Jp.data(), c->m_m_Jp.data()};
  const double* r = rs[kind] + static_cast<size_t>(nr) * index;
  for (int i = 0; i < nr; ++i) residuals[i] = r[i];
  if (!jacobians) return 0;
  const double* Jp = Js[kind] + static_cast<size_t>(nr) * 6 * k * index;
  // state blocks: [J_theta * A_q(q_m) | J_rho | 0]  (ambient 8, row-major nr x 8)
  for (int m = 0; m < k; ++m) {
    if (!jacobians[m]) continue;
    const double* q = parameters[m];
    const double Aq[12] = {2 * q[3], -2 * q[2], 2 * q[1], -2 * q[0], 2 * q[2], 2 * q[3], -2 * q[0], -2 * q[1], -2 * q[1], 2 * q[0], 2 * q[3], -2 * q[2]};
    for (int row = 0; row < nr; ++row) {
      const double* jt = Jp + row * 6 * k + 6 * m;
      double* o = jacobians[m] + 8 * row;
      for (int col = 0; col < 4; ++col) o[col] = jt[0] * Aq[col] + jt[1] * Aq[4 + col] + jt[2] * Aq[8 + col];
      o[4] = jt[3]; o[5] = jt[4]; o[6] = jt[5]; o[7] = 0.0;
    }
  }
  if (kind == HB200_PIXEL || kind == HB200_BEARING) {
    const int sizes[4] = {7, 4, 4, 3};
    const double* Jl = (kind == HB200_PIXEL) ? &c->m_v_Jl[6 * static_cast<size_t>(index)] : &c->m_b_Jl[3 * static_cast<size_t>(index)];
    // calibration blocks (reference pixel.cpp:91-135,141; bearing.cpp:76): rows of [T_bs tangent 6 | intrinsics 4 | distortion 4]
    const double* Jc = &c->m_v_Jc[28 * static_cast<size_t>(kind == HB200_PIXEL ? index : c->Np + index)];
    const int coff[3] = {0, 6, 10};
    for (int b = 0; b < 4; ++b) {
      double* o = jacobians[k + b];
      if (!o) continue;
      if (b == 0) tangent_to_ambient_se3(Jc, 14, nr, parameters[k], o);
      else if (b < 3) { for (int row = 0; row < nr; ++row) for (int col = 0; col < sizes[b]; ++col) o[sizes[b] * row + col] = Jc[14 * row + coff[b] + col]; }
      else std::memcpy(o, Jl, 3 * nr * sizeof(double));
    }
  } else if (kind == HB200_MANIFOLD) {
    if (jacobians[k]) tangent_to_ambient_se3(&c->m_m_Jc[36 * static_cast<size_t>(index)], 6, 6, parameters[k], jacobians[k]);   // reference manifold.cpp:57
  } else {
    // reference inertial.cpp:155-194: rows of [T_bs tangent 6 | i_g 6 | i_a 6 | S_g 9 | X_a 9]
    const int sizes[5] = {7, 6, 6, 9, 9};
    const int coff[5] = {0, 6, 12, 18, 27};
    const double* Jc = &c->m_i_Jc[216 * static_cast<size_t>(index)];
    for (int b = 0; b < 5; ++b) {
      double* o = jacobians[k + b];
      if (!o) continue;
      if (b == 0) tangent_to_ambient_se3(Jc, 36, 6, parameters[k], o);
      else for (int row = 0; row < 6; ++row) for (int col = 0; col < sizes[b]; ++col) o[sizes[b] * row + col] = Jc[36 * row + coff[b] + col];
    }
    for (int m = 0; m < kb; ++m) {
      if (double* o = jacobians[k + 5 + m]) {
        std::fill(o, o + 24, 0.0);
        for (int a = 0; a < 3; ++a) o[4 * a + a] = c->m_i_wg[4 * static_cast<size_t>(index) + m];
      }
      if (double* o = jacobians[k + 5 + kb + m]) {
        std::fill(o, o + 24, 0.0);
        for (int a = 0; a < 3; ++a) o[4 * (3 + a) + a] = c->m_i_wa[4 * static_cast<size_t>(index) + m];
      }
    }
    if (double* o = jacobians[k + 5 + 2 * kb]) {
      // minimal-norm ambient Jacobian: J_tangent * PlusJacobian^T / |g|^2  (PlusJacobian^T PlusJacobian = |g|^2 I)
      const double* x = parameters[k + 5 + 2 * kb];
      const double sigma = x[0] * x[0] + x[1] * x[1];
      double v[3] = {x[0], x[1], 1.0}, beta = 0.0;
      if (sigma <= 2.220446049250313e-16) { if (x[2] < 0.0) beta = 2.0; }
      else {
        const double mu = std::sqrt(x[2] * x[2] + sigma);
        const double vp = (x[2] <= 0.0) ? (x[2] - mu) : (-sigma / (x[2] + mu));
        beta = 2.0 * vp * vp / (sigma + vp * vp);
        v[0] /= vp; v[1] /= vp;
      }
      const double nx = std::sqrt(sigma + x[2] * x[2]);
      double PJ[6];
      for (int cc = 0; cc < 2; ++cc) for (int rr = 0; rr < 3; ++rr) PJ[2 * rr + cc] = nx * ((rr == cc ? 1.0 : 0.0) - beta * v[cc] * v[rr]);
      const double* Jg = &c->m_i_Jg[12 * static_cast<size_t>(index)];
      for (int row = 0; row < 6; ++row)
        for (int col = 0; col < 3; ++col) o[3 * row + col] = (Jg[2 * row] * PJ[2 * col] + Jg[2 * row + 1] * PJ[2 * col + 1]) / (nx * nx);
    }
  }
  return 0;
}

int hb200_reduced_size(hb200_ctx* c) { return c ? 6 * c->K + 3 * c->Kbg + 3 * c->Kba + 2 : -1; }

int hb200_build_system(hb200_ctx* c) {
  int rc = check_ready(c);
  if (rc) return rc;
  if (!c->evaluated_J) return fail(-2, "call hb200_evaluate(HB200_EVAL_JACOBIANS) first");
  HB_CUDA(cudaSetDevice(c->device));
  if ((rc = enqueue_build(c))) return rc;
  if ((rc = enqueue_reduce_system(c))) return rc;
  c->system_built = true;
  return 0;
}

int hb200_get_system(hb200_ctx* c, double* S, double* b) {
  if (!c || !c->system_built) return fail(-2, "system not built");
  HB_CUDA(cudaSetDevice(c->device));
  const size_t n = c->n;
  { const int rc = enqueue_densify(c); if (rc) return rc; }   // dense, damped, masked -- what the solvers factor
  if (S) HB_CUDA(cudaMemcpyAsync(S, c->Lw.p, sizeof(double) * n * n, cudaMemcpyDeviceToHost, c->stream));
  if (b) HB_CUDA(cudaMemcpyAsync(b, c->Lw.p + static_cast<size_t>((n + 31) / 32) * 32 * n, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int hb200_solve(hb200_ctx* c) {
  if (!c || !c->system_built) return fail(-2, "system not built");
  HB_CUDA(cudaSetDevice(c->device));
  return enqueue_solve(c);
}

int hb200_get_delta(hb200_ctx* c, double* dp, double* dl) {
  if (!c || !c->bound) return fail(-2, "not bound");
  HB_CUDA(cudaSetDevice(c->device));
  if (dp) HB_CUDA(cudaMemcpyAsync(dp, c->dp.p, sizeof(double) * c->n, cudaMemcpyDeviceToHost, c->stream));
  if (dl && c->L) HB_CUDA(cudaMemcpyAsync(dl, c->dl.p, sizeof(double) * 3 * c->L, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

}  // extern "C"

namespace {

int iterate_enqueue(hb200_ctx* c, int iterations) {
  int rc = 0;
  for (int it = 0; it < iterations; ++it) {
    // the callback hook cannot be captured; with NCCL the first iteration runs eagerly (NCCL finishes its lazy
    // channel / buffer setup outside of a capture), every later one is a graph launch.  With the peer-memory
    // reduction the iteration exists twice: it assembles into arena half A or B by parity.
    const bool graph_ok = c->use_graph && !c->allreduce && (!c->nccl || c->comm_warm || c->peer_reduce());
    if (graph_ok) {
      const bool slot_b = c->peer_reduce() && c->peer_par == 1;
      cudaGraph_t& graph = slot_b ? c->graph_b : c->graph;
      cudaGraphExec_t& exec = slot_b ? c->graph_exec_b : c->graph_exec;
      bool& valid = slot_b ? c->graph_b_valid : c->graph_valid;
      if (!c->graph_valid) c->graph_b_valid = false;   // (invalidate() only knows the first slot)
      if (!valid) {
        if (exec) { cudaGraphExecDestroy(exec); exec = nullptr; }
        if (graph) { cudaGraphDestroy(graph); graph = nullptr; }
        const int par_before = c->peer_par;
        HB_CUDA(cudaStreamBeginCapture(c->stream, c->nccl ? cudaStreamCaptureModeRelaxed : cudaStreamCaptureModeThreadLocal));
        const long long before = c->launches, nccl_before = c->nccl_calls;
        rc = enqueue_iteration(c);
        cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
        c->launches = before;  // capture does not execute
        c->nccl_calls_per_iteration = c->nccl_calls - nccl_before;
        c->nccl_calls = nccl_before;
        c->peer_par = par_before;   // (enqueue_iteration toggled it: the toggle happens again at the launch below)
        if (rc) return rc;
        if (e != cudaSuccess) {
          if (!c->nccl) return fail(100 + static_cast<int>(e), "graph capture: %s", cudaGetErrorString(e));
          // a communicator that cannot be captured: fall back to direct launches for this context
          cudaGetLastError();
          c->use_graph = false; graph = nullptr;
          --it;
          continue;
        }
        HB_CUDA(cudaGraphInstantiate(&exec, graph, 0));
        valid = true;
        c->launches_per_iteration = 0;
        size_t nodes = 0;
        HB_CUDA(cudaGraphGetNodes(graph, nullptr, &nodes));
        cudaGraphNode_t* nd = new cudaGraphNode_t[nodes];
        HB_CUDA(cudaGraphGetNodes(graph, nd, &nodes));
        for (size_t i = 0; i < nodes; ++i) { cudaGraphNodeType t; if (cudaGraphNodeGetType(nd[i], &t) == cudaSuccess && t == cudaGraphNodeTypeKernel) c->launches_per_iteration += 1; }
        delete[] nd;
        c->launches_per_iteration -= c->nccl_calls_per_iteration;   // NCCL's kernel nodes are not this library's launches
        if (getenv("HB200_GRAPH_DEBUG")) {
          size_t edges = 0;
          cudaGraphGetEdges(graph, nullptr, nullptr, &edges);
          std::fprintf(stderr, "[hb200] iteration graph%s: %zu nodes (%lld own kernels, %lld NCCL), %zu edges\n", slot_b ? " (arena half B)" : "", nodes,
                       c->launches_per_iteration, c->nccl_calls_per_iteration, edges);
        }
      }
      HB_CUDA(cudaGraphLaunch(exec, c->stream));
      if (c->peer_reduce()) c->peer_par ^= 1;
      c->launches += c->launches_per_iteration;
      c->nccl_calls += c->nccl_calls_per_iteration;
    } else {
      if ((rc = enqueue_iteration(c))) return rc;
      if (c->nccl) c->comm_warm = true;
    }
  }
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  if (!c->term_enabled) c->iter_total += iterations;   // (with the termination tests on, the device counter is authoritative: pick_records)
  return 0;
}

// The device ring buffer of iteration records and the solver state, fetched in one batch (asynchronously); the
// records of the iterations PERFORMED since `it_before` are picked out after the synchronisation (with the
// termination tests on, fewer iterations than requested may have been performed).
struct RecordFetch {
  std::vector<SolverState> ring;
  SolverState st{};
};
int fetch_records(hb200_ctx* c, RecordFetch* f, SolverState* pinned = nullptr) {
  f->ring.resize(c->max_records);
  SolverState* dst = pinned ? pinned : f->ring.data();
  HB_CUDA(cudaMemcpyAsync(dst, c->records.p, sizeof(SolverState) * c->max_records, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaMemcpyAsync(pinned ? pinned + c->max_records : &f->st, c->st.p, sizeof(SolverState), cudaMemcpyDeviceToHost, c->stream));
  return 0;
}
// after the stream synchronisation: records of iterations it_before+1 .. st.iteration in order; returns their number
int pick_records(hb200_ctx* c, RecordFetch* f, long long it_before, int requested, std::vector<SolverState>* rec, const SolverState* pinned = nullptr) {
  if (pinned) { std::copy(pinned, pinned + c->max_records, f->ring.begin()); f->st = pinned[c->max_records]; }
  const long long it_after = f->st.iteration;
  const int performed = static_cast<int>(std::max<long long>(0, std::min<long long>(it_after - it_before, requested)));
  rec->resize(performed);
  for (int i = 0; i < performed; ++i) (*rec)[i] = f->ring[(it_before + i) % c->max_records];
  c->iter_total = it_after;
  c->last_terminated = f->st.terminated; c->last_performed = performed;
  c->last_gmax = f->st.gradient_max_norm; c->last_step_norm = f->st.step_norm; c->last_x_norm = f->st.x_norm;
  return performed;
}

void convert_records(const std::vector<SolverState>& rec, hb200_iteration* records) {
  for (size_t i = 0; i < rec.size(); ++i) {
    records[i].cost = rec[i].cost; records[i].cost_new = rec[i].cost_new; records[i].model_change = rec[i].model_change; records[i].rho = rec[i].rho;
    records[i].radius = rec[i].radius; records[i].accepted = rec[i].accepted; records[i].spd = rec[i].spd;
  }
}
}  // namespace

extern "C" {

int hb200_iterate(hb200_ctx* c, int iterations, hb200_iteration* records) {
  int rc = check_ready(c);
  if (rc) return rc;
  if (iterations < 0 || iterations > c->max_records) return fail(-1, "iterations must be in [0, %d]", c->max_records);
  HB_CUDA(cudaSetDevice(c->device));
  if (c->term_enabled) {   // a new call continues the trust region but starts with a clean termination state
    new_solve_kernel<<<1, 1, 0, c->stream>>>(c->st.p, c->radius0, 0);
    HB_LAUNCH(c, "new_solve_kernel");
  }
  const long long it_before = c->iter_total;
  if ((rc = iterate_enqueue(c, iterations))) return rc;
  if (iterations && (records || c->term_enabled)) {
    RecordFetch f;
    std::vector<SolverState> rec;
    if ((rc = fetch_records(c, &f))) return rc;
    HB_CUDA(cudaStreamSynchronize(c->stream));
    const int performed = pick_records(c, &f, it_before, iterations, &rec);
    if (records) {
      convert_records(rec, records);
      for (int i = performed; i < iterations; ++i) records[i] = hb200_iteration{};   // not performed: the solve terminated earlier
    }
  }
  return 0;
}

int hb200_optimize(hb200_ctx* c, int iterations, double* knots, double* gyro, double* accel, double* gravity, double* landmarks,
                   hb200_iteration* records) {
  int rc = check_ready(c);
  if (rc) return rc;
  if (iterations < 0 || iterations > c->max_records) return fail(-1, "iterations must be in [0, %d]", c->max_records);
  HB_CUDA(cudaSetDevice(c->device));
  // the blocks alias the caller's variables, stamps included: the bound index maps are only valid for the stamps
  // they were computed from (a slid window needs hb200_set_spline / hb200_slide + hb200_bind first)
  if (knots) for (int j = 0; j < c->K; ++j) if (knots[8 * j + 7] != c->h_knot_stamp[j]) return fail(-2, "knot %d: stamp differs from the bound window (re-bind after changing stamps)", j);
  if (gyro) for (int j = 0; j < c->Kbg; ++j) if (gyro[4 * j + 3] != c->h_bg_stamp[j]) return fail(-2, "gyroscope bias knot %d: stamp differs from the bound window", j);
  if (accel) for (int j = 0; j < c->Kba; ++j) if (accel[4 * j + 3] != c->h_ba_stamp[j]) return fail(-2, "accelerometer bias knot %d: stamp differs from the bound window", j);
  double* host[5] = {knots, (gyro && c->Kbg) ? gyro : nullptr, (accel && c->Kba) ? accel : nullptr, gravity, (landmarks && c->L) ? landmarks : nullptr};
  double* dev[5] = {c->knots[0].p, c->bg[0].p, c->ba[0].p, c->grav[0].p, c->lms[0].p};
  const size_t cnt[5] = {8 * static_cast<size_t>(c->K), 4 * static_cast<size_t>(c->Kbg), 4 * static_cast<size_t>(c->Kba), 3, 3 * static_cast<size_t>(c->L)};
  size_t off[5], total = 0;
  for (int i = 0; i < 5; ++i) { off[i] = total; if (host[i]) total += cnt[i]; }
  if (gravity) c->have_gravity = true;
  // Small windows: 11 small copies cost more than the iteration's kernels save; pack the blocks into one pinned
  // staging buffer (host memcpy, a few KB), one H2D, one segmented device copy -- and the mirror image back.
  const bool staged = total > 0 && total <= 8192;
  CommitArgs in{}, out{};
  if (staged) {
    if (c->h_stage_cap < total) {
      if (c->h_stage) cudaFreeHost(c->h_stage);
      c->h_stage = nullptr; c->h_stage_cap = 0;
      HB_CUDA(cudaMallocHost(&c->h_stage, sizeof(double) * 8192 + sizeof(SolverState) * (c->max_records + 1)));
      c->h_stage_cap = 8192;
    }
    HB_CUDA(c->d_stage.ensure(8192));
    for (int i = 0; i < 5; ++i) {
      const size_t n_i = host[i] ? cnt[i] : 0;
      if (n_i) std::memcpy(c->h_stage + off[i], host[i], sizeof(double) * n_i);
      in.count[i] = n_i; in.src[i] = c->d_stage.p + off[i]; in.dst[i] = dev[i];
      out.count[i] = n_i; out.src[i] = dev[i]; out.dst[i] = c->d_stage.p + off[i];
    }
    HB_CUDA(cudaMemcpyAsync(c->d_stage.p, c->h_stage, sizeof(double) * total, cudaMemcpyHostToDevice, c->stream));
    copy_segments_kernel<<<4, 256, 0, c->stream>>>(in);
    HB_LAUNCH(c, "copy_segments_kernel");
  } else {
    for (int i = 0; i < 5; ++i)
      if (host[i]) HB_CUDA(cudaMemcpyAsync(dev[i], host[i], sizeof(double) * cnt[i], cudaMemcpyHostToDevice, c->stream));
  }
  // every ceres::Solve starts from the initial trust-region radius and a clean termination state
  new_solve_kernel<<<1, 1, 0, c->stream>>>(c->st.p, c->radius0, 1);
  HB_LAUNCH(c, "new_solve_kernel");
  const long long it_before = c->iter_total;
  if ((rc = iterate_enqueue(c, iterations))) return rc;
  if (staged) {
    copy_segments_kernel<<<4, 256, 0, c->stream>>>(out);
    HB_LAUNCH(c, "copy_segments_kernel");
    HB_CUDA(cudaMemcpyAsync(c->h_stage, c->d_stage.p, sizeof(double) * total, cudaMemcpyDeviceToHost, c->stream));
  } else {
    for (int i = 0; i < 5; ++i)
      if (host[i]) HB_CUDA(cudaMemcpyAsync(host[i], dev[i], sizeof(double) * cnt[i], cudaMemcpyDeviceToHost, c->stream));
  }
  std::vector<SolverState> rec;
  RecordFetch fetch;
  SolverState* rec_pinned = staged ? reinterpret_cast<SolverState*>(c->h_stage + 8192) : nullptr;
  const bool want_records = (records && iterations) || c->term_enabled;
  if (want_records && (rc = fetch_records(c, &fetch, rec_pinned))) return rc;
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if (staged) {
    for (int i = 0; i < 5; ++i)
      if (host[i]) std::memcpy(host[i], c->h_stage + off[i], sizeof(double) * cnt[i]);
  }
  if (want_records) {
    const int performed = pick_records(c, &fetch, it_before, iterations, &rec, rec_pinned);
    if (records) {
      convert_records(rec, records);
      for (int i = performed; i < iterations; ++i) records[i] = hb200_iteration{};
    }
  }
  return 0;
}

int hb200_set_termination(hb200_ctx* c, double function_tolerance, double gradient_tolerance, double parameter_tolerance, double min_trust_region_radius) {
  if (!c) return fail(-1, "null context");
  c->term_ftol = function_tolerance; c->term_gtol = gradient_tolerance; c->term_ptol = parameter_tolerance; c->term_min_radius = min_trust_region_radius;
  c->term_enabled = function_tolerance > 0 || gradient_tolerance > 0 || parameter_tolerance > 0 || min_trust_region_radius > 0;
  c->graph_valid = false;   // baked into kernel arguments
  return 0;
}

int hb200_get_termination(hb200_ctx* c, int* type, int* iterations_performed, double* gradient_max_norm, double* step_norm, double* x_norm) {
  if (!c) return fail(-1, "null context");
  if (type) *type = c->last_terminated;
  if (iterations_performed) *iterations_performed = c->last_performed;
  if (gradient_max_norm) *gradient_max_norm = c->last_gmax;
  if (step_norm) *step_norm = c->last_step_norm;
  if (x_norm) *x_norm = c->last_x_norm;
  return 0;
}

int hb200_cost(hb200_ctx* c, double* cost) {
  int rc = check_ready(c);
  if (rc) return rc;
  if (!cost) return fail(-1, "null argument");
  HB_CUDA(cudaSetDevice(c->device));
  if ((rc = enqueue_evaluate(c, false, 0))) return rc;
  if ((rc = enqueue_scalars(c))) return rc;
  double s[4];
  HB_CUDA(cudaMemcpyAsync(s, c->scal.p, sizeof(s), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  *cost = s[0];
  return 0;
}

// FP64 throughput ceiling of the device (SURVEY.md 8d: "FP64 peak not in MEASURED_PEAKS.json -- measure"):
// 8 independent DFMA chains per thread, enough warps to hide the 8-cycle dependent latency.
__global__ void __launch_bounds__(256) hb200_fp64_peak_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
#pragma unroll 1
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
      x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
  }
  const double s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (s == 1.2345e300) out[0] = s;   // never true: keeps the chains alive
}

int hb200_measure_fp64_peak(hb200_ctx* c, double* tflops) {
  if (!c || !tflops) return fail(-1, "null argument");
  HB_CUDA(cudaSetDevice(c->device));
  DevBuf<double> d;
  HB_CUDA(d.ensure(1));
  cudaEvent_t e0, e1;
  HB_CUDA(cudaEventCreate(&e0)); HB_CUDA(cudaEventCreate(&e1));
  const int blocks = c->num_sms * 8, iters = 4096;
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    HB_CUDA(cudaEventRecord(e0, c->stream));
    hb200_fp64_peak_kernel<<<blocks, 256, 0, c->stream>>>(d.p, iters, 0.999999, 1e-7);
    HB_CUDA(cudaEventRecord(e1, c->stream));
    HB_CUDA(cudaStreamSynchronize(c->stream));
    float ms = 0;
    HB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 64.0 * iters * 256.0 * blocks;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *tflops = best;
  return 0;
}

__global__ void hb200_spin_kernel(long long cycles) {
  const long long t0 = clock64();
  while (clock64() - t0 < cycles) {}
}

int hb200_profile_iteration(hb200_ctx* c, int reps, int max_entries, char* names, double* ms, int* count) {
  int rc = check_ready(c);
  if (rc) return rc;
  if (reps == 0 || !names || !ms || !count) return fail(-1, "invalid argument");
  const bool reps_mode_evaluate = reps < 0;   // negative reps: profile the Evaluate sweep only
  if (reps < 0) reps = -reps;
  HB_CUDA(cudaSetDevice(c->device));
  std::vector<double> acc;
  std::vector<std::string> nm;
  for (int rep = 0; rep < reps; ++rep) {
    c->prof_used = 0;
    // keep the GPU busy while the host enqueues the whole iteration, so kernels run back to back
    hb200_spin_kernel<<<1, 1, 0, c->stream>>>(600000);
    c->profiling = true;
    prof_mark(c, "start");
    if (reps_mode_evaluate) rc = enqueue_evaluate(c, true, 0);   // the plain Evaluate sweep (hb200_evaluate), Jacobians materialised
    else rc = enqueue_iteration(c);
    c->profiling = false;
    if (rc) return rc;
    if (!reps_mode_evaluate) c->iter_total += 1;
    HB_CUDA(cudaStreamSynchronize(c->stream));
    if (rep == 0) { acc.assign(c->prof_used, 0.0); nm.assign(c->prof_names.begin(), c->prof_names.begin() + c->prof_used); }
    for (size_t i = 1; i < c->prof_used && i < acc.size(); ++i) {
      float t = 0;
      HB_CUDA(cudaEventElapsedTime(&t, c->prof_events[i - 1], c->prof_events[i]));
      acc[i] += t;
    }
  }
  int n_out = 0;
  for (size_t i = 1; i < acc.size() && n_out < max_entries; ++i, ++n_out) {
    std::snprintf(names + 32 * n_out, 32, "%s", nm[i].c_str());
    ms[n_out] = acc[i] / reps;
  }
  *count = n_out;
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  return 0;
}

int hb200_interpolate(hb200_ctx* c, int n, const double* stamps, double* pose, double* velocity, double* acceleration, int* num_invalid) {
  if (!c || n < 0 || (n > 0 && (!stamps || !pose))) return fail(-1, "invalid argument");
  if (c->K == 0) return fail(-2, "spline not set");
  HB_CUDA(cudaSetDevice(c->device));
  if (num_invalid) *num_invalid = 0;
  if (n == 0) return 0;
  DevBuf<double> d_t, d_p, d_v, d_a;
  HB_CUDA(d_t.ensure(n)); HB_CUDA(d_p.ensure(7 * static_cast<size_t>(n)));
  if (velocity) HB_CUDA(d_v.ensure(6 * static_cast<size_t>(n)));
  if (acceleration) HB_CUDA(d_a.ensure(6 * static_cast<size_t>(n)));
  HB_CUDA(c->d_invalid.ensure(1));
  HB_CUDA(cudaMemsetAsync(c->d_invalid.p, 0, sizeof(int), c->stream));
  HB_CUDA(cudaMemcpyAsync(d_t.p, stamps, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  prep_kernel<<<(c->K + 63) / 64, 64, 0, c->stream>>>(c->K, c->knots[0].p, c->tab[0].p, nullptr, 0);
  HB_LAUNCH(c, "prep_kernel");
  if (c->k == 4) interpolate_kernel<4><<<(n + 127) / 128, 128, 0, c->stream>>>(n, d_t.p, c->knots[0].p, c->tab[0].p, c->K, c->basis, d_p.p, d_v.p, d_a.p, c->d_invalid.p);
  else interpolate_kernel<6><<<(n + 127) / 128, 128, 0, c->stream>>>(n, d_t.p, c->knots[0].p, c->tab[0].p, c->K, c->basis, d_p.p, d_v.p, d_a.p, c->d_invalid.p);
  HB_LAUNCH(c, "interpolate_kernel");
  int bad = 0;
  HB_CUDA(cudaMemcpyAsync(pose, d_p.p, sizeof(double) * 7 * n, cudaMemcpyDeviceToHost, c->stream));
  if (velocity) HB_CUDA(cudaMemcpyAsync(velocity, d_v.p, sizeof(double) * 6 * n, cudaMemcpyDeviceToHost, c->stream));
  if (acceleration) HB_CUDA(cudaMemcpyAsync(acceleration, d_a.p, sizeof(double) * 6 * n, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaMemcpyAsync(&bad, c->d_invalid.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  cudaError_t e = cudaStreamSynchronize(c->stream);
  d_t.release(); d_p.release(); d_v.release(); d_a.release();
  if (e != cudaSuccess) return fail(100 + static_cast<int>(e), "interpolate: %s", cudaGetErrorString(e));
  if (num_invalid) *num_invalid = bad;
  return 0;
}

int hb200_debug_band_timing(hb200_ctx* c, long long* cycles /*[72]: 8 phase totals + 8 steps x 8 raw stamps*/) {
  if (!c || !c->band_dbg.p) return fail(-2, "set HB200_BAND_TIMING=1 before hb200_bind");
  HB_CUDA(cudaMemcpy(cycles, c->band_dbg.p, 72 * sizeof(long long), cudaMemcpyDeviceToHost));
  return 0;
}

int hb200_snapshot(hb200_ctx* c) {
  if (!c || c->K == 0) return fail(-2, "spline not set");
  HB_CUDA(cudaSetDevice(c->device));
  HB_CUDA(c->snap_knots.ensure(8 * static_cast<size_t>(c->K))); HB_CUDA(c->snap_bg.ensure(4 * static_cast<size_t>(std::max(c->Kbg, 1))));
  HB_CUDA(c->snap_ba.ensure(4 * static_cast<size_t>(std::max(c->Kba, 1)))); HB_CUDA(c->snap_grav.ensure(4)); HB_CUDA(c->snap_lms.ensure(3 * static_cast<size_t>(std::max(c->L, 1))));
  HB_CUDA(c->snap_st.ensure(1));
  HB_CUDA(cudaMemcpyAsync(c->snap_knots.p, c->knots[0].p, sizeof(double) * 8 * c->K, cudaMemcpyDeviceToDevice, c->stream));
  if (c->Kbg) HB_CUDA(cudaMemcpyAsync(c->snap_bg.p, c->bg[0].p, sizeof(double) * 4 * c->Kbg, cudaMemcpyDeviceToDevice, c->stream));
  if (c->Kba) HB_CUDA(cudaMemcpyAsync(c->snap_ba.p, c->ba[0].p, sizeof(double) * 4 * c->Kba, cudaMemcpyDeviceToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->snap_grav.p, c->grav[0].p, sizeof(double) * 3, cudaMemcpyDeviceToDevice, c->stream));
  if (c->L) HB_CUDA(cudaMemcpyAsync(c->snap_lms.p, c->lms[0].p, sizeof(double) * 3 * c->L, cudaMemcpyDeviceToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->snap_st.p, c->st.p, sizeof(SolverState), cudaMemcpyDeviceToDevice, c->stream));
  c->have_snapshot = true;
  c->snap_iter_total = c->iter_total;
  return 0;
}

int hb200_restore(hb200_ctx* c) {
  if (!c || !c->have_snapshot) return fail(-2, "no snapshot");
  HB_CUDA(cudaSetDevice(c->device));
  HB_CUDA(cudaMemcpyAsync(c->knots[0].p, c->snap_knots.p, sizeof(double) * 8 * c->K, cudaMemcpyDeviceToDevice, c->stream));
  if (c->Kbg) HB_CUDA(cudaMemcpyAsync(c->bg[0].p, c->snap_bg.p, sizeof(double) * 4 * c->Kbg, cudaMemcpyDeviceToDevice, c->stream));
  if (c->Kba) HB_CUDA(cudaMemcpyAsync(c->ba[0].p, c->snap_ba.p, sizeof(double) * 4 * c->Kba, cudaMemcpyDeviceToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->grav[0].p, c->snap_grav.p, sizeof(double) * 3, cudaMemcpyDeviceToDevice, c->stream));
  if (c->L) HB_CUDA(cudaMemcpyAsync(c->lms[0].p, c->snap_lms.p, sizeof(double) * 3 * c->L, cudaMemcpyDeviceToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->st.p, c->snap_st.p, sizeof(SolverState), cudaMemcpyDeviceToDevice, c->stream));
  c->iter_total = c->snap_iter_total;
  c->evaluated_J = false; c->system_built = false; c->mirror_valid = false; c->calib_valid = false;
  return 0;
}

int hb200_ingest_stereo(hb200_ctx* c, int n, const double* stamp, const int* camera0, const int* camera1, const double* pixel0,
                        const double* pixel1, double* bearing0, double* bearing1, double* landmark, int* num_invalid) {
  if (!c || n < 0) return fail(-1, "invalid arguments");
  if (c->K == 0 || c->C == 0) return fail(-2, "spline / cameras not set");
  if (c->k != 4 && c->k != 6) return fail(-4, "spline order %d not supported (4 or 6)", c->k);
  if (n > 0 && (!stamp || !camera0 || !camera1 || !pixel0 || !pixel1 || !bearing0 || !bearing1 || !landmark)) return fail(-1, "null argument");
  if (num_invalid) *num_invalid = 0;
  if (n == 0) return 0;
  HB_CUDA(cudaSetDevice(c->device));
  DevBuf<double> d_t, d_p0, d_p1, d_b0, d_b1, d_lm;
  DevBuf<int> d_c0, d_c1;
  const size_t N = static_cast<size_t>(n);
  HB_CUDA(d_t.ensure(N)); HB_CUDA(d_p0.ensure(2 * N)); HB_CUDA(d_p1.ensure(2 * N)); HB_CUDA(d_b0.ensure(3 * N)); HB_CUDA(d_b1.ensure(3 * N));
  HB_CUDA(d_lm.ensure(3 * N)); HB_CUDA(d_c0.ensure(N)); HB_CUDA(d_c1.ensure(N));
  HB_CUDA(c->d_invalid.ensure(1));
  HB_CUDA(cudaMemsetAsync(c->d_invalid.p, 0, sizeof(int), c->stream));
  HB_CUDA(cudaMemcpyAsync(d_t.p, stamp, sizeof(double) * N, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(d_c0.p, camera0, sizeof(int) * N, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(d_c1.p, camera1, sizeof(int) * N, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(d_p0.p, pixel0, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(d_p1.p, pixel1, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, c->stream));
  prep_kernel<<<(c->K + 63) / 64, 64, 0, c->stream>>>(c->K, c->knots[0].p, c->tab[0].p, nullptr, 0);
  HB_LAUNCH(c, "prep_kernel");
  if (c->k == 4) ingest_stereo_kernel<4><<<(n + 127) / 128, 128, 0, c->stream>>>(n, d_t.p, d_c0.p, d_c1.p, d_p0.p, d_p1.p, c->knots[0].p, c->tab[0].p, c->K, c->basis, c->cams.p, c->C, d_b0.p, d_b1.p, d_lm.p, c->d_invalid.p);
  else ingest_stereo_kernel<6><<<(n + 127) / 128, 128, 0, c->stream>>>(n, d_t.p, d_c0.p, d_c1.p, d_p0.p, d_p1.p, c->knots[0].p, c->tab[0].p, c->K, c->basis, c->cams.p, c->C, d_b0.p, d_b1.p, d_lm.p, c->d_invalid.p);
  HB_LAUNCH(c, "ingest_stereo_kernel");
  int bad = 0;
  HB_CUDA(cudaMemcpyAsync(bearing0, d_b0.p, sizeof(double) * 3 * N, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaMemcpyAsync(bearing1, d_b1.p, sizeof(double) * 3 * N, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaMemcpyAsync(landmark, d_lm.p, sizeof(double) * 3 * N, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaMemcpyAsync(&bad, c->d_invalid.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  d_t.release(); d_p0.release(); d_p1.release(); d_b0.release(); d_b1.release(); d_lm.release(); d_c0.release(); d_c1.release();
  if (num_invalid) *num_invalid = bad;
  return 0;
}

int hb200_get_state(hb200_ctx* c, double* knots, double* gyro, double* accel, double* gravity, double* landmarks) {
  if (!c) return fail(-1, "null context");
  HB_CUDA(cudaSetDevice(c->device));
  if (knots && c->K) HB_CUDA(cudaMemcpyAsync(knots, c->knots[0].p, sizeof(double) * 8 * c->K, cudaMemcpyDeviceToHost, c->stream));
  if (gyro && c->Kbg) HB_CUDA(cudaMemcpyAsync(gyro, c->bg[0].p, sizeof(double) * 4 * c->Kbg, cudaMemcpyDeviceToHost, c->stream));
  if (accel && c->Kba) HB_CUDA(cudaMemcpyAsync(accel, c->ba[0].p, sizeof(double) * 4 * c->Kba, cudaMemcpyDeviceToHost, c->stream));
  if (gravity) HB_CUDA(cudaMemcpyAsync(gravity, c->grav[0].p, sizeof(double) * 3, cudaMemcpyDeviceToHost, c->stream));
  if (landmarks && c->L) HB_CUDA(cudaMemcpyAsync(landmarks, c->lms[0].p, sizeof(double) * 3 * c->L, cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

// ---- device-side sliding-window bookkeeping (hb200_window.cuh) -----------------------------------------------
namespace {
int check_device_window(hb200_ctx* c) {
  if (!c) return fail(-1, "null context");
  if (!c->bound) return fail(-2, "bind the window first (hb200_bind)");
  return 0;
}

// the visual list's tail [Nv, Nv + n) after a bind on the device: kind check of the stamps / indices (rc 2), then the
// arrival order (rc 3).  The caller commits the new size only when both pass, so a rejected append changes nothing.
int check_visual_tail(hb200_ctx* c, int Nv, int n) {
  tail_sorted_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(Nv, n, c->v_idx.p, c->d_invalid.p + 1);
  HB_LAUNCH(c, "tail_sorted_kernel");
  int bad[2] = {0, 0};
  HB_CUDA(cudaMemcpyAsync(bad, c->d_invalid.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if (bad[0]) return fail(2, "%d appended factor(s) reference a stamp outside the spline's valid range or an invalid camera / landmark", bad[0]);
  if (bad[1]) return fail(3, "appended factors must arrive in stamp order (%d fall before the end of the list): use hb200_set_*_factors + hb200_bind", bad[1]);
  return 0;
}

// grow the visual list to Nv + n entries, the first Nv preserved (the buffers may move: the captured iteration goes)
int grow_visual(hb200_ctx* c, size_t Nv, size_t n) {
  c->graph_valid = false;
  HB_CUDA(c->v_stamp.grow(Nv + n, Nv, c->stream)); HB_CUDA(c->v_pixel.grow(2 * (Nv + n), 2 * Nv, c->stream));
  HB_CUDA(c->v_z.grow(Nv + n, Nv, c->stream)); HB_CUDA(c->v_idx.grow(Nv + n, Nv, c->stream));
  return 0;
}
}  // namespace

int hb200_append_knots(hb200_ctx* c, int count) {
  int rc = check_device_window(c);
  if (rc) return rc;
  if (count <= 0) return fail(-1, "count must be positive");
  HB_CUDA(cudaSetDevice(c->device));
  const int K = c->K;
  for (int s2 = 0; s2 < 2; ++s2) {
    HB_CUDA(c->knots[s2].grow(8 * static_cast<size_t>(K + count), s2 == 0 ? 8 * static_cast<size_t>(K) : 0, c->stream));
    HB_CUDA(c->tab[s2].ensure(static_cast<size_t>(K + count) * kTabStride));
  }
  append_knots_kernel<<<1, 32, 0, c->stream>>>(K, count, c->knots[0].p);
  HB_LAUNCH(c, "append_knots_kernel");
  std::vector<double> tail(8 * static_cast<size_t>(count));
  HB_CUDA(cudaMemcpyAsync(tail.data(), c->knots[0].p + 8 * static_cast<size_t>(K), sizeof(double) * tail.size(), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  for (int i = 0; i < count; ++i) { c->h_knot_stamp.push_back(tail[8 * i + 7]); c->h_knot_const.push_back(0); }
  c->K = K + count;
  if ((rc = update_fixed(c))) return rc;
  c->nseg = c->K - c->k + 1;
  HB_CUDA(c->seg_off.grow(static_cast<size_t>(c->nseg) + 2, static_cast<size_t>(c->nseg - count) + 1, c->stream));
  {   // the new segments hold no visual factor yet: their offsets equal the list length
    std::vector<int> fill(count, c->Nv);
    HB_CUDA(cudaMemcpyAsync(c->seg_off.p + (c->nseg - count) + 1, fill.data(), sizeof(int) * count, cudaMemcpyHostToDevice, c->stream));
  }
  if ((rc = ensure_system(c))) return rc;
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->invalidate(); c->have_snapshot = false;
  return sync_layout(c);
}

int hb200_append_landmarks(hb200_ctx* c, int n, const double* xyz) {
  int rc = check_device_window(c);
  if (rc) return rc;
  if (n <= 0 || !xyz) return fail(-1, "invalid landmarks");
  HB_CUDA(cudaSetDevice(c->device));
  const size_t L = c->L;
  for (int s2 = 0; s2 < 2; ++s2) HB_CUDA(c->lms[s2].grow(3 * (L + n), s2 == 0 ? 3 * L : 0, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->lms[0].p + 3 * L, xyz, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->L = static_cast<int>(L) + n;
  return rebuild_incidence_device(c);
}

int hb200_append_pixel_factors(hb200_ctx* c, int n, const double* stamp, const int* camera, const int* landmark, const double* pixel) {
  int rc = check_device_window(c);
  if (rc) return rc;
  if (n <= 0 || !stamp || !camera || !landmark || !pixel) return fail(-1, "invalid pixel factors");
  HB_CUDA(cudaSetDevice(c->device));
  const size_t Nv = c->Nv;
  if ((rc = grow_visual(c, Nv, n))) return rc;
  DevBuf<int> d_cam, d_lm;
  HB_CUDA(d_cam.ensure(n)); HB_CUDA(d_lm.ensure(n));
  HB_CUDA(c->d_invalid.ensure(2));
  HB_CUDA(cudaMemsetAsync(c->d_invalid.p, 0, 2 * sizeof(int), c->stream));
  HB_CUDA(cudaMemcpyAsync(c->v_stamp.p + Nv, stamp, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->v_pixel.p + 2 * Nv, pixel, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(d_cam.p, camera, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(d_lm.p, landmark, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
  bind_pixel_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(n, c->v_stamp.p + Nv, d_cam.p, d_lm.p, c->knots[0].p, c->K, c->k, c->C, c->L, 0, c->v_idx.p + Nv, c->d_invalid.p);
  HB_LAUNCH(c, "bind_pixel_kernel");
  if ((rc = check_visual_tail(c, static_cast<int>(Nv), n))) return rc;
  c->Nv = static_cast<int>(Nv) + n; c->Np += n;
  return rebuild_incidence_device(c);
}

int hb200_append_bearing_factors(hb200_ctx* c, int n, const double* stamp, const int* camera, const int* landmark, const double* bearing) {
  int rc = check_device_window(c);
  if (rc) return rc;
  if (n <= 0 || !stamp || !camera || !landmark || !bearing) return fail(-1, "invalid bearing factors");
  HB_CUDA(cudaSetDevice(c->device));
  const size_t Nv = c->Nv;
  if ((rc = grow_visual(c, Nv, n))) return rc;
  // [n][3] -> the visual list's (x, y) pairs + z column
  std::vector<double> xy(2 * static_cast<size_t>(n)), z(n);
  for (int f = 0; f < n; ++f) { xy[2 * f] = bearing[3 * f]; xy[2 * f + 1] = bearing[3 * f + 1]; z[f] = bearing[3 * f + 2]; }
  DevBuf<int> d_cam, d_lm;
  HB_CUDA(d_cam.ensure(n)); HB_CUDA(d_lm.ensure(n));
  HB_CUDA(c->d_invalid.ensure(2));
  HB_CUDA(cudaMemsetAsync(c->d_invalid.p, 0, 2 * sizeof(int), c->stream));
  HB_CUDA(cudaMemcpyAsync(c->v_stamp.p + Nv, stamp, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->v_pixel.p + 2 * Nv, xy.data(), sizeof(double) * 2 * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->v_z.p + Nv, z.data(), sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(d_cam.p, camera, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(d_lm.p, landmark, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
  bind_pixel_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(n, c->v_stamp.p + Nv, d_cam.p, d_lm.p, c->knots[0].p, c->K, c->k, c->C, c->L, 1, c->v_idx.p + Nv, c->d_invalid.p);
  HB_LAUNCH(c, "bind_pixel_kernel");
  if ((rc = check_visual_tail(c, static_cast<int>(Nv), n))) return rc;
  c->Nv = static_cast<int>(Nv) + n; c->Nb += n;
  return rebuild_incidence_device(c);
}

int hb200_append_manifold_factors(hb200_ctx* c, int n, const double* stamp, const int* sensor, const double* pose) {
  int rc = check_device_window(c);
  if (rc) return rc;
  if (n <= 0 || !stamp || !sensor || !pose) return fail(-1, "invalid manifold factors");
  if (c->P == 0) return fail(-2, "manifold factors need pose sensors (hb200_set_pose_sensors)");
  HB_CUDA(cudaSetDevice(c->device));
  const size_t Nm = c->Nm;
  c->graph_valid = false;   // (the buffers may move)
  HB_CUDA(c->m_stamp.grow(Nm + n, Nm, c->stream)); HB_CUDA(c->m_meas.grow(7 * (Nm + n), 7 * Nm, c->stream)); HB_CUDA(c->m_idx.grow(Nm + n, Nm, c->stream));
  HB_CUDA(c->m_sensor.ensure(n));
  HB_CUDA(c->d_invalid.ensure(2));
  HB_CUDA(cudaMemsetAsync(c->d_invalid.p, 0, 2 * sizeof(int), c->stream));
  HB_CUDA(cudaMemcpyAsync(c->m_stamp.p + Nm, stamp, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->m_meas.p + 7 * Nm, pose, sizeof(double) * 7 * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->m_sensor.p, sensor, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
  bind_manifold_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(n, c->m_stamp.p + Nm, c->m_sensor.p, c->knots[0].p, c->K, c->k, c->P, c->m_idx.p + Nm, c->d_invalid.p);
  HB_LAUNCH(c, "bind_manifold_kernel");
  tail_sorted_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(static_cast<int>(Nm), n, c->m_idx.p, c->d_invalid.p + 1);
  HB_LAUNCH(c, "tail_sorted_kernel");
  int bad[2] = {0, 0};
  HB_CUDA(cudaMemcpyAsync(bad, c->d_invalid.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if (bad[0]) return fail(2, "%d appended pose factor(s) reference a stamp outside the spline's valid range or an invalid sensor", bad[0]);
  if (bad[1]) return fail(3, "appended factors must arrive in stamp order (%d fall before the end of the list): use hb200_set_manifold_factors + hb200_bind", bad[1]);
  c->Nm = static_cast<int>(Nm) + n;
  return rebuild_incidence_device(c);
}

int hb200_append_stereo_tracks(hb200_ctx* c, int n, const double* stamp, const int* camera0, const int* camera1, const double* pixel0,
                               const double* pixel1, const int* landmark_in, int* landmark_out, int* num_new) {
  int rc = check_device_window(c);
  if (rc) return rc;
  if (n <= 0 || !stamp || !camera0 || !camera1 || !pixel0 || !pixel1 || !landmark_in) return fail(-1, "invalid stereo tracks");
  if (c->C == 0) return fail(-2, "cameras not set");
  if (c->k != 4 && c->k != 6) return fail(-4, "spline order %d not supported (4 or 6)", c->k);
  HB_CUDA(cudaSetDevice(c->device));
  const size_t N = n, Nv = c->Nv, L = c->L;
  // one H2D copy: [pixel0 2n | pixel1 2n | stamp n] doubles (the pixel pairs 16-byte aligned), then
  // [camera0 n | camera1 n | landmark_in n] ints
  const size_t nd = 5 * N, ni = 3 * N;
  std::vector<double> stage(nd + (ni + 1) / 2);
  std::memcpy(stage.data(), pixel0, sizeof(double) * 2 * N);
  std::memcpy(stage.data() + 2 * N, pixel1, sizeof(double) * 2 * N);
  std::memcpy(stage.data() + 4 * N, stamp, sizeof(double) * N);
  int* si = reinterpret_cast<int*>(stage.data() + nd);
  std::memcpy(si, camera0, sizeof(int) * N); std::memcpy(si + N, camera1, sizeof(int) * N); std::memcpy(si + 2 * N, landmark_in, sizeof(int) * N);
  DevBuf<double> d_in;
  DevBuf<int> d_flag, d_pos, d_out;   // d_out: [invalid, out of order, new landmarks | landmark_out n]
  HB_CUDA(d_in.ensure(stage.size())); HB_CUDA(d_flag.ensure(N)); HB_CUDA(d_pos.ensure(N)); HB_CUDA(d_out.ensure(3 + N));
  if ((rc = grow_visual(c, Nv, 2 * N))) return rc;
  for (int s2 = 0; s2 < 2; ++s2) HB_CUDA(c->lms[s2].grow(3 * (L + N), s2 == 0 ? 3 * L : 0, c->stream));
  HB_CUDA(cudaMemsetAsync(d_out.p, 0, 3 * sizeof(int), c->stream));
  HB_CUDA(cudaMemcpyAsync(d_in.p, stage.data(), sizeof(double) * stage.size(), cudaMemcpyHostToDevice, c->stream));
  const int* d_i = reinterpret_cast<const int*>(d_in.p + nd);
  stereo_new_flags_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(n, d_i + 2 * N, c->L, d_flag.p, d_out.p);
  HB_LAUNCH(c, "stereo_new_flags_kernel");
  scan_kernel<<<1, 1024, 0, c->stream>>>(d_flag.p, n, d_pos.p, d_out.p + 2);
  HB_LAUNCH(c, "scan_kernel");
  prep_kernel<<<(c->K + 63) / 64, 64, 0, c->stream>>>(c->K, c->knots[0].p, c->tab[0].p, nullptr, 0);
  HB_LAUNCH(c, "prep_kernel");
  const double2* q0 = reinterpret_cast<const double2*>(d_in.p);
  const double2* q1 = reinterpret_cast<const double2*>(d_in.p + 2 * N);
  double2* vpx = reinterpret_cast<double2*>(c->v_pixel.p);
  if (c->k == 4)
    append_stereo_tracks_kernel<4><<<(n + 127) / 128, 128, 0, c->stream>>>(n, d_in.p + 4 * N, q0, q1, d_i, d_i + N, d_i + 2 * N, d_pos.p, c->knots[0].p, c->tab[0].p, c->K, c->basis,
                                                                       c->cams.p, c->C, c->L, c->Nv, c->v_stamp.p, vpx, c->v_z.p, c->v_idx.p, c->lms[0].p, d_out.p + 3, d_out.p);
  else
    append_stereo_tracks_kernel<6><<<(n + 127) / 128, 128, 0, c->stream>>>(n, d_in.p + 4 * N, q0, q1, d_i, d_i + N, d_i + 2 * N, d_pos.p, c->knots[0].p, c->tab[0].p, c->K, c->basis,
                                                                       c->cams.p, c->C, c->L, c->Nv, c->v_stamp.p, vpx, c->v_z.p, c->v_idx.p, c->lms[0].p, d_out.p + 3, d_out.p);
  HB_LAUNCH(c, "append_stereo_tracks_kernel");
  tail_sorted_kernel<<<(2 * n + 127) / 128, 128, 0, c->stream>>>(static_cast<int>(Nv), 2 * n, c->v_idx.p, d_out.p + 1);
  HB_LAUNCH(c, "tail_sorted_kernel");
  std::vector<int> h(3 + N);
  HB_CUDA(cudaMemcpyAsync(h.data(), d_out.p, sizeof(int) * (3 + N), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if (h[0]) return fail(2, "%d stereo track(s) reference a stamp outside the spline's valid range, an invalid camera or a landmark slot outside [-1, L)", h[0]);
  if (h[1]) return fail(3, "appended factors must arrive in stamp order (%d fall before the end of the list): use hb200_set_bearing_factors + hb200_bind", h[1]);
  if (landmark_out) std::memcpy(landmark_out, h.data() + 3, sizeof(int) * N);
  if (num_new) *num_new = h[2];
  c->Nv = static_cast<int>(Nv + 2 * N); c->Nb += 2 * n; c->L = static_cast<int>(L) + h[2];
  return rebuild_incidence_device(c);
}

int hb200_append_inertial_factors(hb200_ctx* c, int n, const double* stamp, const double* meas) {
  int rc = check_device_window(c);
  if (rc) return rc;
  if (n <= 0 || !stamp || !meas) return fail(-1, "invalid inertial factors");
  if (!c->have_imu || c->Kbg == 0 || c->Kba == 0) return fail(-2, "inertial factors need IMU calibration and bias splines");
  HB_CUDA(cudaSetDevice(c->device));
  const size_t Ni = c->Ni;
  HB_CUDA(c->i_stamp.grow(Ni + n, Ni, c->stream)); HB_CUDA(c->i_meas.grow(6 * (Ni + n), 6 * Ni, c->stream)); HB_CUDA(c->i_idx.grow(Ni + n, Ni, c->stream));
  HB_CUDA(c->d_invalid.ensure(2));
  HB_CUDA(cudaMemsetAsync(c->d_invalid.p, 0, 2 * sizeof(int), c->stream));
  HB_CUDA(cudaMemcpyAsync(c->i_stamp.p + Ni, stamp, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaMemcpyAsync(c->i_meas.p + 6 * Ni, meas, sizeof(double) * 6 * n, cudaMemcpyHostToDevice, c->stream));
  bind_inertial_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(n, c->i_stamp.p + Ni, c->knots[0].p, c->K, c->k, c->bg[0].p, c->Kbg, c->ba[0].p, c->Kba, c->kb,
                                                             c->i_idx.p + Ni, c->d_invalid.p);
  HB_LAUNCH(c, "bind_inertial_kernel");
  tail_sorted_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(static_cast<int>(Ni), n, c->i_idx.p, c->d_invalid.p + 1);
  HB_LAUNCH(c, "tail_sorted_kernel");
  int bad[2] = {0, 0};
  HB_CUDA(cudaMemcpyAsync(bad, c->d_invalid.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if (bad[0]) return fail(2, "%d appended factor(s) reference a stamp outside the state or bias splines' valid range", bad[0]);
  if (bad[1]) return fail(3, "appended factors must arrive in stamp order (%d fall before the end of the list): use hb200_set_inertial_factors + hb200_bind", bad[1]);
  c->Ni = static_cast<int>(Ni) + n;
  return rebuild_incidence_device(c);
}

int hb200_slide(hb200_ctx* c, double lower_bound, int flags, hb200_slide_stats* stats) {
  int rc = check_device_window(c);
  if (rc) return rc;
  HB_CUDA(cudaSetDevice(c->device));
  const int Nv = c->Nv, Ni = c->Ni, Nm = c->Nm, L = c->L, K = c->K;
  // knot index of the last state element at or before the lower bound; the window keeps `left padding` elements in
  // front of the one that starts the lower bound's interval (reference optimizer.cpp:289: prev(upper_bound(lower), left_padding))
  int ub = static_cast<int>(std::upper_bound(c->h_knot_stamp.begin(), c->h_knot_stamp.end(), lower_bound) - c->h_knot_stamp.begin());
  const int begin = std::max(0, ub - 1 - (c->k - 1) / 2);
  const int last_const = ub - 1;   // knots 0 .. last_const have stamp <= lower bound
  HB_CUDA(c->w_scal.ensure(8));
  // [L_new, Nv_new, Ni_new, min base visual, min base inertial, min base manifold, bearing factors kept, Nm_new]
  int init[8] = {0, 0, 0, 0x7fffffff, 0x7fffffff, 0x7fffffff, 0, 0};
  HB_CUDA(cudaMemcpyAsync(c->w_scal.p, init, sizeof(init), cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(c->w_last.ensure(std::max(L, 1))); HB_CUDA(c->w_lkeep.ensure(std::max(L, 1) + 1)); HB_CUDA(c->w_lpos.ensure(std::max(L, 1) + 1));
  HB_CUDA(c->w_keep.ensure(std::max(std::max(Nv, Ni), 1))); HB_CUDA(c->w_pos.ensure(std::max(std::max(Nv, Ni), 1)));
  DevBuf<int> i_keep, i_pos, m_keep, m_pos;
  HB_CUDA(i_keep.ensure(std::max(Ni, 1))); HB_CUDA(i_pos.ensure(std::max(Ni, 1)));
  if (Nm) { HB_CUDA(m_keep.ensure(Nm)); HB_CUDA(m_pos.ensure(Nm)); }
  HB_CUDA(cudaMemsetAsync(c->w_last.p, 0, sizeof(unsigned long long) * std::max(L, 1), c->stream));
  if (Nv) { landmark_last_stamp_kernel<<<(Nv + 255) / 256, 256, 0, c->stream>>>(Nv, c->v_stamp.p, c->v_idx.p, c->w_last.p); HB_LAUNCH(c, "landmark_last_stamp_kernel"); }
  if (L) {
    landmark_keep_kernel<<<(L + 255) / 256, 256, 0, c->stream>>>(L, c->w_last.p, lower_bound, c->w_lkeep.p);
    HB_LAUNCH(c, "landmark_keep_kernel");
    scan_kernel<<<1, 1024, 0, c->stream>>>(c->w_lkeep.p, L, c->w_lpos.p, c->w_scal.p + 0);
    HB_LAUNCH(c, "scan_kernel");
  }
  if (Nv) {
    visual_keep_kernel<<<(Nv + 255) / 256, 256, 0, c->stream>>>(Nv, c->v_idx.p, c->w_lkeep.p, c->w_keep.p, c->w_scal.p + 3, c->w_scal.p + 6);
    HB_LAUNCH(c, "visual_keep_kernel");
    scan_kernel<<<1, 1024, 0, c->stream>>>(c->w_keep.p, Nv, c->w_pos.p, c->w_scal.p + 1);
    HB_LAUNCH(c, "scan_kernel");
  }
  if (Ni) {
    inertial_keep_kernel<<<(Ni + 255) / 256, 256, 0, c->stream>>>(Ni, c->i_idx.p, c->k, (flags & HB200_SLIDE_DROP_INERTIAL) ? last_const : -1, i_keep.p, c->w_scal.p + 4);
    HB_LAUNCH(c, "inertial_keep_kernel");
    scan_kernel<<<1, 1024, 0, c->stream>>>(i_keep.p, Ni, i_pos.p, c->w_scal.p + 2);
    HB_LAUNCH(c, "scan_kernel");
  }
  if (Nm) {
    manifold_keep_kernel<<<(Nm + 255) / 256, 256, 0, c->stream>>>(Nm, c->m_idx.p, c->k, (flags & HB200_SLIDE_DROP_POSE) ? last_const : -1, m_keep.p, c->w_scal.p + 5);
    HB_LAUNCH(c, "manifold_keep_kernel");
    scan_kernel<<<1, 1024, 0, c->stream>>>(m_keep.p, Nm, m_pos.p, c->w_scal.p + 7);
    HB_LAUNCH(c, "scan_kernel");
  }
  int h[8];
  HB_CUDA(cudaMemcpyAsync(h, c->w_scal.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  const int L_new = L ? h[0] : 0, Nv_new = Nv ? h[1] : 0, Ni_new = Ni ? h[2] : 0, Nm_new = Nm ? h[7] : 0, Nb_new = h[6];
  // state elements in front of `begin` go once no residual touches them (reference optimizer.cpp:331-341)
  int shift = std::min(std::min(begin, h[5]), std::min(h[3], h[4]));
  shift = std::max(0, std::min(shift, K - c->k));
  const int K_new = K - shift;
  // compaction into the alternate buffers, then swap
  HB_CUDA(c->alt_stamp.ensure(std::max(std::max(Nv_new, Ni_new), std::max(Nm_new, 1)))); HB_CUDA(c->alt_idx.ensure(std::max(std::max(Nv_new, Ni_new), 1)));
  HB_CUDA(c->alt_meas.ensure(std::max(6 * static_cast<size_t>(Ni_new), 7 * static_cast<size_t>(std::max(Nm_new, 1)))));
  HB_CUDA(c->alt_midx.ensure(std::max(Nm_new, 1)));
  HB_CUDA(c->alt_pixel.ensure(std::max(Nv_new, 1))); HB_CUDA(c->alt_z.ensure(std::max(Nv_new, 1)));
  if (Nv) {
    compact_visual_kernel<<<(Nv + 255) / 256, 256, 0, c->stream>>>(Nv, c->w_keep.p, c->w_pos.p, c->w_lpos.p, shift, c->v_stamp.p, reinterpret_cast<const double2*>(c->v_pixel.p),
                                                                  c->v_z.p, c->v_idx.p, c->alt_stamp.p, c->alt_pixel.p, c->alt_z.p, c->alt_idx.p);
    HB_LAUNCH(c, "compact_visual_kernel");
    // (v_pixel is a DevBuf<double>: copy the compacted pairs back instead of swapping differently typed buffers)
    HB_CUDA(cudaMemcpyAsync(c->v_pixel.p, c->alt_pixel.p, sizeof(double2) * Nv_new, cudaMemcpyDeviceToDevice, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->v_stamp.p, c->alt_stamp.p, sizeof(double) * Nv_new, cudaMemcpyDeviceToDevice, c->stream));
    if (c->Nb) HB_CUDA(cudaMemcpyAsync(c->v_z.p, c->alt_z.p, sizeof(double) * Nv_new, cudaMemcpyDeviceToDevice, c->stream));   // (read for bearings only)
    HB_CUDA(cudaMemcpyAsync(c->v_idx.p, c->alt_idx.p, sizeof(int4) * Nv_new, cudaMemcpyDeviceToDevice, c->stream));
  }
  if (Ni) {
    compact_inertial_kernel<<<(Ni + 255) / 256, 256, 0, c->stream>>>(Ni, i_keep.p, i_pos.p, shift, c->i_stamp.p, c->i_meas.p, c->i_idx.p, c->alt_stamp.p, c->alt_meas.p, c->alt_idx.p);
    HB_LAUNCH(c, "compact_inertial_kernel");
    HB_CUDA(cudaMemcpyAsync(c->i_stamp.p, c->alt_stamp.p, sizeof(double) * Ni_new, cudaMemcpyDeviceToDevice, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->i_meas.p, c->alt_meas.p, sizeof(double) * 6 * Ni_new, cudaMemcpyDeviceToDevice, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->i_idx.p, c->alt_idx.p, sizeof(int4) * Ni_new, cudaMemcpyDeviceToDevice, c->stream));
  }
  if (Nm) {
    compact_manifold_kernel<<<(Nm + 255) / 256, 256, 0, c->stream>>>(Nm, m_keep.p, m_pos.p, shift, c->m_stamp.p, c->m_meas.p, c->m_idx.p, c->alt_stamp.p, c->alt_meas.p, c->alt_midx.p);
    HB_LAUNCH(c, "compact_manifold_kernel");
    HB_CUDA(cudaMemcpyAsync(c->m_stamp.p, c->alt_stamp.p, sizeof(double) * Nm_new, cudaMemcpyDeviceToDevice, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->m_meas.p, c->alt_meas.p, sizeof(double) * 7 * Nm_new, cudaMemcpyDeviceToDevice, c->stream));
    HB_CUDA(cudaMemcpyAsync(c->m_idx.p, c->alt_midx.p, sizeof(int2) * Nm_new, cudaMemcpyDeviceToDevice, c->stream));
  }
  if (L) {
    HB_CUDA(c->alt_lms.ensure(3 * static_cast<size_t>(std::max(L_new, 1))));
    compact_landmarks_kernel<<<(L + 255) / 256, 256, 0, c->stream>>>(L, c->w_lkeep.p, c->w_lpos.p, c->lms[0].p, c->alt_lms.p);
    HB_LAUNCH(c, "compact_landmarks_kernel");
    HB_CUDA(cudaMemcpyAsync(c->lms[0].p, c->alt_lms.p, sizeof(double) * 3 * L_new, cudaMemcpyDeviceToDevice, c->stream));
  }
  if (shift) {
    HB_CUDA(c->alt_knots.ensure(8 * static_cast<size_t>(K_new)));
    shift_knots_kernel<<<(8 * K_new + 255) / 256, 256, 0, c->stream>>>(K_new, shift, c->knots[0].p, c->alt_knots.p);
    HB_LAUNCH(c, "shift_knots_kernel");
    HB_CUDA(cudaMemcpyAsync(c->knots[0].p, c->alt_knots.p, sizeof(double) * 8 * K_new, cudaMemcpyDeviceToDevice, c->stream));
  }
  HB_CUDA(cudaStreamSynchronize(c->stream));
  // host bookkeeping: sizes, stamps, constancy (elements at or before the lower bound: reference optimizer.cpp:322-328;
  // gravity once the window no longer covers the whole state range: reference abstract.cpp:57-61)
  c->h_knot_stamp.erase(c->h_knot_stamp.begin(), c->h_knot_stamp.begin() + shift);
  c->h_knot_const.assign(K_new, 0);
  for (int j = 0; j < K_new; ++j) c->h_knot_const[j] = c->h_knot_stamp[j] <= lower_bound ? 1 : 0;
  if (ub > 0) c->gravity_const = 1;
  c->K = K_new; c->L = L_new; c->Nv = Nv_new; c->Np = Nv_new - Nb_new; c->Nb = Nb_new; c->Ni = Ni_new; c->Nm = Nm_new;
  if (stats) {
    stats->knots_dropped = shift; stats->knots_constant = std::max(0, ub - shift); stats->landmarks_dropped = L - L_new;
    stats->visual_factors_dropped = Nv - Nv_new; stats->inertial_factors_dropped = Ni - Ni_new;
    stats->knots = K_new; stats->landmarks = L_new; stats->visual_factors = Nv_new; stats->inertial_factors = Ni_new;
  }
  return rebuild_incidence_device(c);
}

int hb200_factor_counts(hb200_ctx* c, int* pixel, int* bearing, int* inertial, int* manifold) {
  if (!c) return fail(-1, "null context");
  if (pixel) *pixel = c->Np;
  if (bearing) *bearing = c->Nb;
  if (inertial) *inertial = c->Ni;
  if (manifold) *manifold = c->Nm;
  return 0;
}

int hb200_window_sizes(hb200_ctx* c, int* knots, int* landmarks, int* visual_factors, int* inertial_factors) {
  if (!c) return fail(-1, "null context");
  if (knots) *knots = c->K;
  if (landmarks) *landmarks = c->L;
  if (visual_factors) *visual_factors = c->Nv;
  if (inertial_factors) *inertial_factors = c->Ni;
  return 0;
}

int hb200_set_allreduce(hb200_ctx* c, hb200_allreduce_fn fn, void* user) {
  if (!c) return fail(-1, "null context");
  if (fn && c->nccl) return fail(-2, "a NCCL communicator is attached; the callback hook is its replacement, not an addition");
  c->allreduce = fn; c->allreduce_user = user;
  c->graph_valid = false;
  return 0;
}

int hb200_comm_unique_id(char* id) {
  if (!id) return fail(-1, "null argument");
  int rc = load_nccl();
  if (rc) return rc;
  NcclUid u;
  HB_NCCL(g_nccl.GetUniqueId(&u));
  std::memcpy(id, u.internal, sizeof(u.internal));
  return 0;
}

int hb200_set_nccl_comm(hb200_ctx* c, void* comm, int nranks, int rank) {
  if (!c) return fail(-1, "null context");
  if (comm && (nranks < 1 || nranks > kMaxRanks || rank < 0 || rank >= nranks)) return fail(-1, "invalid rank %d of %d (at most %d ranks)", rank, nranks, kMaxRanks);
  if (comm && c->allreduce) return fail(-2, "the all-reduce callback hook is set; clear it first");
  if (comm) { int rc = load_nccl(); if (rc) return rc; }
  HB_CUDA(cudaSetDevice(c->device));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }   // it references the old communicator
  if (c->graph) { cudaGraphDestroy(c->graph); c->graph = nullptr; }
  if (c->graph_exec_b) { cudaGraphExecDestroy(c->graph_exec_b); c->graph_exec_b = nullptr; }
  if (c->graph_b) { cudaGraphDestroy(c->graph_b); c->graph_b = nullptr; }
  c->graph_valid = false; c->graph_b_valid = false;
  if (c->nccl && c->own_nccl) g_nccl.CommDestroy(c->nccl);
  c->nccl = comm; c->own_nccl = false;
  c->nranks = comm ? nranks : 1; c->rank = comm ? rank : 0;
  c->comm_warm = false; c->graph_valid = false;
  return sync_layout(c);
}

int hb200_comm_init_rank(hb200_ctx* c, int nranks, int rank, const char* id) {
  if (!c || !id) return fail(-1, "null argument");
  if (nranks < 1 || nranks > kMaxRanks || rank < 0 || rank >= nranks) return fail(-1, "invalid rank %d of %d (at most %d ranks)", rank, nranks, kMaxRanks);
  int rc = load_nccl();
  if (rc) return rc;
  HB_CUDA(cudaSetDevice(c->device));
  NcclUid u;
  std::memcpy(u.internal, id, sizeof(u.internal));
  void* comm = nullptr;
  HB_NCCL(g_nccl.CommInitRank(&comm, nranks, u, rank));
  rc = hb200_set_nccl_comm(c, comm, nranks, rank);
  if (rc) { g_nccl.CommDestroy(comm); return rc; }
  c->own_nccl = true;
  return 0;
}

int hb200_peer_handle(hb200_ctx* c, char* handle) {
  if (!c || !handle) return fail(-1, "null argument");
  HB_CUDA(cudaSetDevice(c->device));
  // the arena: mailbox + flag row + two partial-system halves (capacity HB200_PEER_ARENA_DOUBLES each, default 600 k doubles =
  // 4.8 MB: a K = 1000 window; larger systems fall back to ncclAllReduce)
  const long long cap = getenv("HB200_PEER_ARENA_DOUBLES") ? std::max(0LL, atoll(getenv("HB200_PEER_ARENA_DOUBLES"))) & ~1LL : 600000LL;
  const size_t arena = static_cast<size_t>(kArenaParts) + 2 * static_cast<size_t>(cap);
  HB_CUDA(c->mbox.ensure(arena));
  c->arena_cap = cap;
  HB_CUDA(c->mbox_seq.ensure(1)); HB_CUDA(c->red_round.ensure(1)); HB_CUDA(c->red_arrive.ensure(1));
  HB_CUDA(cudaMemsetAsync(c->mbox.p, 0, sizeof(double) * kArenaParts, c->stream));
  HB_CUDA(cudaMemsetAsync(c->mbox_seq.p, 0, sizeof(unsigned long long), c->stream));
  HB_CUDA(cudaMemsetAsync(c->red_round.p, 0, sizeof(unsigned long long), c->stream));
  HB_CUDA(cudaMemsetAsync(c->red_arrive.p, 0, sizeof(unsigned int), c->stream));
  c->peer_par = 0;
  c->peer_reduce_wanted = !(getenv("HB200_PEER_REDUCE") && atoi(getenv("HB200_PEER_REDUCE")) == 0);
  HB_CUDA(cudaStreamSynchronize(c->stream));
  cudaIpcMemHandle_t h;
  HB_CUDA(cudaIpcGetMemHandle(&h, c->mbox.p));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  std::memcpy(handle, &h, sizeof(h));
  return 0;
}

namespace {
void close_peers(hb200_ctx* c) {
  for (size_t p = 0; p < c->peer_ptrs.size(); ++p)
    if (c->peer_ptrs[p] && c->peer_ptrs[p] != c->mbox.p) cudaIpcCloseMemHandle(c->peer_ptrs[p]);
  c->peer_ptrs.clear();
  c->peers_open = false;
}
}  // namespace

int hb200_peer_connect(hb200_ctx* c, int nranks, int rank, const char* handles) {
  if (!c || !handles) return fail(-1, "null argument");
  if (!c->nccl || nranks != c->nranks || rank != c->rank) return fail(-2, "attach the communicator first (same nranks / rank)");
  if (!c->mbox.p) return fail(-2, "call hb200_peer_handle first");
  HB_CUDA(cudaSetDevice(c->device));
  close_peers(c);
  c->peer_ptrs.assign(nranks, nullptr);
  for (int p = 0; p < nranks; ++p) {
    if (p == rank) { c->peer_ptrs[p] = c->mbox.p; continue; }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handles + 64 * static_cast<size_t>(p), sizeof(h));
    void* ptr = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      close_peers(c);
      return fail(100 + static_cast<int>(e), "cudaIpcOpenMemHandle(rank %d): %s (the scalar exchange falls back to a second ncclAllReduce)", p, cudaGetErrorString(e));
    }
    c->peer_ptrs[p] = ptr;
  }
  HB_CUDA(c->d_peers.ensure(kMaxRanks));
  std::vector<double*> host(kMaxRanks, nullptr);
  for (int p = 0; p < nranks; ++p) host[p] = static_cast<double*>(c->peer_ptrs[p]);
  HB_CUDA(cudaMemcpyAsync(c->d_peers.p, host.data(), sizeof(double*) * kMaxRanks, cudaMemcpyHostToDevice, c->stream));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  c->peers_open = true;
  c->graph_valid = false;
  return 0;
}

int hb200_set_min_bandwidth(hb200_ctx* c, int beta) {
  if (!c || beta < 0) return fail(-1, "invalid argument");
  HB_CUDA(cudaSetDevice(c->device));
  c->min_beta = beta;
  if (c->bound) {
    HB_CUDA(cudaStreamSynchronize(c->stream));
    const int rc = ensure_system(c);
    if (rc) return rc;
    c->invalidate();
  }
  return 0;
}

int hb200_get_bandwidth(hb200_ctx* c, int* beta) {
  if (!c || !beta) return fail(-1, "null argument");
  if (!c->bound) return fail(-2, "not bound");
  *beta = c->beta;
  return 0;
}

int hb200_peer_disconnect(hb200_ctx* c) {
  if (!c) return fail(-1, "null context");
  HB_CUDA(cudaSetDevice(c->device));
  HB_CUDA(cudaStreamSynchronize(c->stream));
  close_peers(c);
  c->graph_valid = false;
  return 0;
}

int hb200_comm_info(hb200_ctx* c, int* nranks, int* rank, int* nccl, int* peer_mailbox, int* graph, long long* payload_doubles) {
  if (!c) return fail(-1, "null context");
  if (nranks) *nranks = c->nranks;
  if (rank) *rank = c->rank;
  if (nccl) *nccl = c->nccl ? 1 : 0;
  if (peer_mailbox) *peer_mailbox = (c->nccl && c->peers_open) ? (c->peer_reduce() ? 2 : 1) : 0;   // 2: the system reduction runs over peer memory too
  if (graph) *graph = (c->use_graph && !c->allreduce && c->graph_valid) ? 1 : 0;
  if (payload_doubles) *payload_doubles = c->bound ? c->lay.total : 0;
  return 0;
}

void* hb200_system_device_ptr(hb200_ctx* c, long long* count) {
  if (!c) return nullptr;
  if (count) *count = c->lay.total;
  return c->sys.p;
}

}  // extern "C"
