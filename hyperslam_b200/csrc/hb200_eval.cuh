// Factor evaluation kernels (sm_100a): knot table, index maps, stereo-pixel and inertial
// residual + Jacobian.  One factor per thread; a CTA's knot-table tile is staged to shared memory
// with one TMA bulk copy (cp.async.bulk + mbarrier).  Replaces, for a whole factor list at once,
//   ExteroceptiveCost::Evaluate           reference internal/hyper/optimizers/ceres/costs/exteroceptive.cpp:101-160
//   VisualPixelEvaluator<SE3>::evaluate   reference internal/hyper/optimizers/evaluators/pixel.cpp:16-146
//   InertialEvaluator<SE3>::evaluate      reference internal/hyper/optimizers/evaluators/inertial.cpp:13-205
//   AbstractState::evaluate (HyperState)  call sites pixel.cpp:74-75, inertial.cpp:93-94
// and projects Jacobians straight into the tangent space the Ceres manifolds would project them to
// (reference include/hyper/optimizers/ceres/manifolds/variables/wrapper.hpp:36-42).
#pragma once
#include "hb200_math.cuh"
#include "hb200_types.cuh"

namespace hb {

// ---------------------------------------------------------------------------------------------
// TMA (1-D bulk copy) + mbarrier helpers
// ---------------------------------------------------------------------------------------------
HB_DI uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
HB_DI void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
HB_DI void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
HB_DI void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
HB_DI void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
HB_DI void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// Stage knot-table rows [row_lo, row_lo + rows) into s_tab with one bulk copy.  Call from all threads.
HB_DI void stage_table(double* s_tab, uint64_t* bar, const double* g_tab, int row_lo, int rows) {
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t bytes = static_cast<uint32_t>(rows) * kTabStride * sizeof(double);
    mbar_expect_tx(bar, bytes);
    tma_load_1d(s_tab, g_tab + static_cast<size_t>(row_lo) * kTabStride, bytes, bar);
  }
  mbar_wait(bar, 0);
}

// Block-wide min / max of an int (blockDim.x <= 1024).
HB_DI void block_min_max(int v_min, int v_max, int* s_red /*2 ints*/, int* out_min, int* out_max) {
  if (threadIdx.x == 0) { s_red[0] = 0x7fffffff; s_red[1] = -0x7fffffff; }
  __syncthreads();
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    v_min = min(v_min, __shfl_xor_sync(0xffffffffu, v_min, o));
    v_max = max(v_max, __shfl_xor_sync(0xffffffffu, v_max, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicMin(&s_red[0], v_min); atomicMax(&s_red[1], v_max); }
  __syncthreads();
  *out_min = s_red[0];
  *out_max = s_red[1];
}

// ---------------------------------------------------------------------------------------------
// a2 / a4: knot base index of a stamp (bit-exact with the oracle's segment_base()).
// ---------------------------------------------------------------------------------------------
HB_DI int segment_base(const double* knots, int stride, int stamp_off, int K, int k, double t) {
  if (K < k) return -1;
  const double t0 = knots[stamp_off], t1 = knots[stride + stamp_off];
  long long j = static_cast<long long>(floor((t - t0) / (t1 - t0)));
  if (j < 0) j = 0;
  if (j > K - 2) j = K - 2;
  while (j > 0 && knots[static_cast<size_t>(j) * stride + stamp_off] > t) --j;
  while (j < K - 2 && knots[static_cast<size_t>(j + 1) * stride + stamp_off] <= t) ++j;
  if (!(knots[static_cast<size_t>(j) * stride + stamp_off] <= t && t < knots[static_cast<size_t>(j + 1) * stride + stamp_off])) return -1;
  const int base = static_cast<int>(j) - (k - 1) / 2;
  if (base < 0 || base + k - 1 > K - 1) return -1;
  return base;
}

// pixel and bearing factors share the visual list: `kind` (0 pixel, 1 bearing) goes to idx.w
__global__ void bind_pixel_kernel(int n, const double* __restrict__ stamp, const int* __restrict__ cam, const int* __restrict__ lm,
                                  const double* __restrict__ knots, int K, int k, int C, int L, int kind, int4* __restrict__ idx,
                                  int* __restrict__ num_invalid) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const int base = segment_base(knots, 8, 7, K, k, stamp[f]);
  const int c = cam[f], l = lm[f];
  idx[f] = make_int4(base, l, c, kind);
  if (base < 0 || c < 0 || c >= C || l < 0 || l >= L) atomicAdd(num_invalid, 1);
}

__global__ void bind_inertial_kernel(int n, const double* __restrict__ stamp, const double* __restrict__ knots, int K, int k,
                                     const double* __restrict__ bg, int Kbg, const double* __restrict__ ba, int Kba, int kb,
                                     int4* __restrict__ idx, int* __restrict__ num_invalid) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const double t = stamp[f];
  const int base = segment_base(knots, 8, 7, K, k, t);
  const int g = segment_base(bg, 4, 3, Kbg, kb, t);
  const int a = segment_base(ba, 4, 3, Kba, kb, t);
  idx[f] = make_int4(base, g, a, 0);
  if (base < 0 || g < 0 || a < 0) atomicAdd(num_invalid, 1);
}

// ---------------------------------------------------------------------------------------------
// Knot table: one thread per control point (a3, per-segment part shared by all factors).
// ---------------------------------------------------------------------------------------------
// One knot-table row from the control point's quaternion q, position p, stamp and the previous control
// point's quaternion qp (have_prev = false for row 0).
HB_DI void knot_table_row(const double* q, const double* p, double stamp, const double* qp, bool have_prev, double* __restrict__ row) {
  double R[9];
  quat_to_rot(q, R);
#pragma unroll
  for (int i = 0; i < 9; ++i) row[i] = R[i];
  row[9] = p[0]; row[10] = p[1]; row[11] = p[2];
  double d[3] = {0, 0, 0}, G[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  if (have_prev) {
    const double qc[4] = {-qp[0], -qp[1], -qp[2], qp[3]};
    double qr[4], Ji[9];
    quat_mul(qc, q, qr);
    quat_log(qr, d);
    so3_Jr_inv(d, Ji);
    m3_mult(Ji, R, G);
  }
  row[12] = d[0]; row[13] = d[1]; row[14] = d[2];
#pragma unroll
  for (int i = 0; i < 9; ++i) row[15 + i] = G[i];
  row[24] = stamp; row[25] = 0; row[26] = 0; row[27] = 0;
}

// clear / nclear: optional buffer zeroed by the same launch (the packed reduced system at the start of an
// iteration -- saves the separate memset node).
__global__ void prep_kernel(int K, const double* __restrict__ knots, double* __restrict__ tab, double* __restrict__ clear, size_t nclear) {
  pdl_launch_dependents();   // the factor kernel behind it may become resident now (it waits for this grid's completion)
  const size_t gid = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  for (size_t e = gid; e < nclear; e += static_cast<size_t>(gridDim.x) * blockDim.x) clear[e] = 0.0;
  const int j = static_cast<int>(gid);
  if (gid >= static_cast<size_t>(K)) return;
  const double* kn = knots + 8 * static_cast<size_t>(j);
  const double q[4] = {kn[0], kn[1], kn[2], kn[3]};
  double qp[4] = {0, 0, 0, 1};
  if (j > 0) { qp[0] = kn[-8]; qp[1] = kn[-7]; qp[2] = kn[-6]; qp[3] = kn[-5]; }
  knot_table_row(q, kn + 4, kn[7], qp, j > 0, tab + static_cast<size_t>(j) * kTabStride);
}

// Calibration tables (once per set_cameras / set_imu).
// quirks: reference-quirk switches of the inertial Jacobians (hb200_calib.cuh / oracle Quirks): the table carries the
// matrices the RESIDUAL uses and, separately, the ones the state / gravity JACOBIANS use (identical when quirks = 0).
__global__ void calib_kernel(int C, const double* __restrict__ cams, double* __restrict__ cam_tab, const double* __restrict__ imu,
                             double* __restrict__ imu_tab, int quirks) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < C) {
    const double* c = cams + 15 * t;
    double* o = cam_tab + kCamStride * t;
    double R[9];
    quat_to_rot(c, R);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) o[3 * i + j] = R[3 * j + i];  // R_sb = R_bs^T
    o[9] = c[4]; o[10] = c[5]; o[11] = c[6];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[12 + i] = c[7 + i];
  }
  if (t == 0 && imu != nullptr) {
    double R[9], Rsb[9];
    quat_to_rot(imu, R);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) Rsb[3 * i + j] = R[3 * j + i];
    const double* ig = imu + 7;
    const double* ia = imu + 13;
    const double Ig[9] = {ig[0], 0, 0, ig[3], ig[1], 0, ig[4], ig[5], ig[2]};
    const double Ia[9] = {ia[0], 0, 0, ia[3], ia[1], 0, ia[4], ia[5], ia[2]};
    double IgR[9], IaR[9];
    m3_mul(Ig, Rsb, IgR);
    m3_mul(Ia, Rsb, IaR);
#pragma unroll
    for (int i = 0; i < 9; ++i) { imu_tab[i] = Rsb[i]; imu_tab[12 + i] = IgR[i]; imu_tab[21 + i] = IaR[i]; }
    imu_tab[9] = imu[4]; imu_tab[10] = imu[5]; imu_tab[11] = imu[6];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        imu_tab[30 + 3 * i + j] = imu[19 + i + 3 * j];            // S_g row-major from column-major
        imu_tab[39 + 3 * i + j] = imu[28 + j + 3 * i] + imu[4 + j];  // lever arm c_i = X_a[:, i] + t_bs
        // Jacobian-side copies: (i) gyroscope intrinsics in the accelerometer rows (inertial.cpp:136,142,148),
        // (ii) no Jacobian of the S_g a_b_m term (:135,147), (v) lever arm without X_a (:142,148)
        imu_tab[48 + 3 * i + j] = (quirks & 1) ? IgR[3 * i + j] : IaR[3 * i + j];
        imu_tab[57 + 3 * i + j] = (quirks & 2) ? 0.0 : imu[19 + i + 3 * j];
        imu_tab[66 + 3 * i + j] = ((quirks & 8) ? 0.0 : imu[28 + j + 3 * i]) + imu[4 + j];
      }
    imu_tab[75] = 0.0;
  }
}

// ---------------------------------------------------------------------------------------------
// Basis evaluation (Horner), lam[0] = 1, lam[K] = 0.
// ---------------------------------------------------------------------------------------------
template <int K, bool DERIV>
HB_DI void basis_eval(const Basis& b, double u, double inv_dt, double* lam, double* lamd, double* lamdd) {
  lam[0] = 1.0; lam[K] = 0.0;
  if (DERIV) { lamd[0] = lamdd[0] = 0.0; lamd[K] = lamdd[K] = 0.0; }
#pragma unroll
  for (int j = 1; j < K; ++j) {
    double v = 0, d1 = 0, d2 = 0;
#pragma unroll
    for (int n = K - 1; n >= 0; --n) {
      if (DERIV) { d2 = d2 * u + 2.0 * d1; d1 = d1 * u + v; }
      v = v * u + b.Mc[j * K + n];
    }
    lam[j] = v;
    if (DERIV) { lamd[j] = d1 * inv_dt; lamdd[j] = d2 * inv_dt * inv_dt; }
  }
}

HB_DI double huber_rho(double s, double delta, double* weight) {
  if (s <= delta * delta) { *weight = 1.0; return s; }
  const double rt = sqrt(s);
  *weight = delta / rt;
  return 2.0 * delta * rt - delta * delta;
}

// ---------------------------------------------------------------------------------------------
// Pixel factor (a5 + a3 + a7..a10 fused).  T: table origin (row r at T + r*kTabStride).
// ---------------------------------------------------------------------------------------------
// 256-bit global store (SASS STG.E.256): p must be 32-byte aligned.  Writes whole 32 B sectors, so a
// thread-per-factor row store costs one L2 sector write per 32 B instead of two half-filled ones.
HB_DI void st_v4(double* p, double a, double b, double c, double d) {
  asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

// kind 0: pixel residual (reference pixel.cpp:16-146 + CartesianMetric); kind 1: bearing residual
// (reference bearing.cpp:14-79 + AngularMetric): r = [angle(p_s, z), 0], second Jacobian row zero, so a
// bearing factor travels through the same compact [2][6K] / [2][3] layout and the same J^T J / Schur code.
template <int K, bool WANT_J>
HB_DI void pixel_factor(const double* __restrict__ T, const Basis& B, int base, double t, double zx, double zy, double zz, int kind,
                        const double* __restrict__ cam, const double* __restrict__ lmk, double* r, double* __restrict__ Jp,
                        double* __restrict__ Jl) {
  constexpr int left = (K - 1) / 2;
  const double* row0 = T + static_cast<size_t>(base) * kTabStride;
  const double t0 = row0[left * kTabStride + 24], t1 = row0[(left + 1) * kTabStride + 24];
  const double inv_dt = 1.0 / (t1 - t0);
  const double u = (t - t0) * inv_dt;
  double lam[K + 1];
  basis_eval<K, false>(B, u, inv_dt, lam, nullptr, nullptr);

  double P[9], p[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) P[i] = row0[i];
  p[0] = row0[9]; p[1] = row0[10]; p[2] = row0[11];
  double M[(K - 1) * 9];
#pragma unroll
  for (int j = 1; j < K; ++j) {
    const double* rj = row0 + j * kTabStride;
    const double w[3] = {lam[j] * rj[12], lam[j] * rj[13], lam[j] * rj[14]};
    double A[9], Jr[9], Pn[9];
    so3_exp_and_Jr(w, A, WANT_J ? Jr : nullptr);
    m3_mul(P, A, Pn);
    if (WANT_J) {
      double G[9], JG[9], PJG[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) G[i] = rj[15 + i];
      m3_mul(Jr, G, JG);
      m3_mul(Pn, JG, PJG);
#pragma unroll
      for (int i = 0; i < 9; ++i) M[(j - 1) * 9 + i] = lam[j] * PJG[i];
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) P[i] = Pn[i];
#pragma unroll
    for (int c = 0; c < 3; ++c) p[c] += lam[j] * (rj[9 + c] - rj[9 + c - kTabStride]);
  }
  // p_s = R_sb (R^T (p_w - p) - t_bs)
  const double q[3] = {lmk[0] - p[0], lmk[1] - p[1], lmk[2] - p[2]};
  double pb[3], ps[3];
  m3_tvec(P, q, pb);
  const double pbt[3] = {pb[0] - cam[9], pb[1] - cam[10], pb[2] - cam[11]};
  m3_vec(cam, pbt, ps);
  double Jps[6];
  if (kind == 0) {
    const double iz = 1.0 / ps[2];
    const double x = ps[0] * iz, y = ps[1] * iz;
    const double cx = cam[12], cy = cam[13], fx = cam[14], fy = cam[15];
    const double k1 = cam[16], k2 = cam[17], p1 = cam[18], p2 = cam[19];
    const double r2 = x * x + y * y;
    const double rad = 1.0 + k1 * r2 + k2 * r2 * r2;
    const double dx = x * rad + 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x);
    const double dy = y * rad + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y;
    r[0] = fx * dx + cx - zx;
    r[1] = fy * dy + cy - zy;
    if (!WANT_J) return;
    const double g = k1 + 2.0 * k2 * r2;
    const double drx = 2.0 * x * g, dry = 2.0 * y * g;
    // J_r_n = diag(fx, fy) * d(distort)/dn
    const double a00 = fx * (rad + x * drx + 2.0 * p1 * y + 6.0 * p2 * x);
    const double a01 = fx * (x * dry + 2.0 * p1 * x + 2.0 * p2 * y);
    const double a10 = fy * (y * drx + 2.0 * p1 * x + 2.0 * p2 * y);
    const double a11 = fy * (rad + y * dry + 6.0 * p1 * y + 2.0 * p2 * x);
    // J_n_p = [iz 0 -x iz; 0 iz -y iz]
    Jps[0] = a00 * iz; Jps[1] = a01 * iz; Jps[2] = -(a00 * x + a01 * y) * iz;
    Jps[3] = a10 * iz; Jps[4] = a11 * iz; Jps[5] = -(a10 * x + a11 * y) * iz;
  } else {
    // theta = atan2(|p_s x z|, p_s . z);  d theta / d p_s = [c (z x n) - s z]^T / (|p_s|^2 |z|^2), n = (p_s x z)/s
    const double z[3] = {zx, zy, zz};
    double cr[3];
    cross(ps, z, cr);
    const double s = sqrt((cr[0] * cr[0] + cr[1] * cr[1] + cr[2] * cr[2])), c = (ps[0] * z[0] + ps[1] * z[1] + ps[2] * z[2]);
    r[0] = atan2(s, c);
    r[1] = 0.0;
    if (!WANT_J) return;
    Jps[0] = Jps[1] = Jps[2] = Jps[3] = Jps[4] = Jps[5] = 0.0;
    if (s > 1e-300) {
      const double is = 1.0 / s;
      const double nrm[3] = {cr[0] * is, cr[1] * is, cr[2] * is};
      double zn[3];
      cross(z, nrm, zn);
      const double iden = 1.0 / ((ps[0] * ps[0] + ps[1] * ps[1] + ps[2] * ps[2]) * (z[0] * z[0] + z[1] * z[1] + z[2] * z[2]));
#pragma unroll
      for (int i = 0; i < 3; ++i) Jps[i] = (c * zn[i] - s * z[i]) * iden;
    }
  }
  double Jpb[6], F[6], E[6];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) Jpb[3 * i + j] = Jps[3 * i] * cam[j] + Jps[3 * i + 1] * cam[3 + j] + Jps[3 * i + 2] * cam[6 + j];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) F[3 * i + j] = Jpb[3 * i] * P[3 * j] + Jpb[3 * i + 1] * P[3 * j + 1] + Jpb[3 * i + 2] * P[3 * j + 2];  // Jpb R^T
#pragma unroll
  for (int i = 0; i < 2; ++i) {  // E = F hat(q)
    E[3 * i] = F[3 * i + 1] * q[2] - F[3 * i + 2] * q[1];
    E[3 * i + 1] = F[3 * i + 2] * q[0] - F[3 * i] * q[2];
    E[3 * i + 2] = F[3 * i] * q[1] - F[3 * i + 1] * q[0];
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) Jl[i] = F[i];
  // E M_j (2x3 each)
  double EM[(K - 1) * 6];
#pragma unroll
  for (int j = 0; j < K - 1; ++j)
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int c = 0; c < 3; ++c)
        EM[j * 6 + 3 * i + c] = E[3 * i] * M[j * 9 + c] + E[3 * i + 1] * M[j * 9 + 3 + c] + E[3 * i + 2] * M[j * 9 + 6 + c];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    double row[6 * K];
#pragma unroll
    for (int m = 0; m < K; ++m) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double cur = (m == 0) ? E[3 * i + c] : EM[(m - 1) * 6 + 3 * i + c];
        const double nxt = (m + 1 < K) ? EM[m * 6 + 3 * i + c] : 0.0;
        row[6 * m + c] = cur - nxt;
        row[6 * m + 3 + c] = -(lam[m] - lam[m + 1]) * F[3 * i + c];
      }
    }
    double* out = Jp + i * 6 * K;   // 32-byte aligned: rows are 192 B (K=4) / 288 B (K=6)
#pragma unroll
    for (int g = 0; g < 6 * K / 4; ++g) st_v4(out + 4 * g, row[4 * g], row[4 * g + 1], row[4 * g + 2], row[4 * g + 3]);
  }
}

struct PixelArgs {
  int n;
  const double* stamp;
  const double2* pixel;    // pixel measurement, or the first two components of a bearing measurement
  const double* meas_z;    // third component of a bearing measurement (null when there are no bearing factors)
  const int4* idx;        // (base, landmark, camera, kind: 0 pixel / 1 bearing)
  const double* tab;      // knot table of the evaluated state
  const double* cam_tab;
  const double* landmarks;
  double* r;              // [n][2]
  double* Jp;             // [n][2][6K]
  double* Jl;             // [n][2][3]
  double* w;              // [n] robust-loss weight rho'(s) of each factor (written with the Jacobians)
  double* cost_partial;   // [gridDim.x]
  double huber;           // Huber delta of the pixel factors (reference optimizer.cpp:226)
  double huber_bearing;   // Huber delta of the bearing factors (reference optimizer.cpp:204)
  int K_knots;
  double* sys;            // packed band-only reduced system (SysLayout) to accumulate J^T J / J^T r into, or null
  SysLayout lay;
  int tiles_per_cta;      // consecutive 64-factor tiles one CTA of pixel_eval_kernel walks (large windows: its J^T J accumulators
                          // stay in registers across tiles of the same knot base, one flush per base instead of one per tile)
};

// J^T J / J^T r of up to 32 consecutive pixel factors [f0, f0 + cnt) of this CTA, accumulated into the
// lower triangle of S and into g with FP64 atomics.  Called right after the CTA wrote those factors'
// residuals and Jacobians, so the re-read hits L2.
//   * staging: thread = one Jacobian row (2 per factor), copied with 128-bit loads and scaled by sqrt(w);
//   * J^T J on the FP64 tensor cores (mma.sync m8n8k4 -> SASS DMMA.8x8x4): the 6K x 6K block is cut into 8 x 8
//     tiles (lower triangle only), the contraction runs over the rows of one knot base in steps of 4, rows
//     of other bases inside the sub-tile are masked to zero.  Fragments: lane l holds A[m = l/4][k = l%4] =
//     J[k][m] and B[k = l%4][n = l/4] = J[k][n] -- the same shared-memory access pattern -- and
//     C[m = l/4][n = 2 (l%4) + {0,1}].  This replaced a scalar 3x3-register-tile loop that executed ~9 000
//     instructions per warp (ncu smsp__inst_executed, profiles/) against ~1 400 for the factor evaluation itself.
// J^T J tiles / gradient entry a thread carries across the tiles of one knot base (registers)
template <int K>
struct PixelHessAcc {
  static constexpr int NB = 6 * K, NT = (NB + 7) / 8, NTILES = NT * (NT + 1) / 2, PER_WARP = (NTILES + 1) / 2;
  // row pitch of the staged Jacobian rows: the fragment loads touch word (k0 + l%4) * LD + l/4, conflict-free when
  // LD = 4 or 12 (mod 16); 6K = 24 -> 28.  (6K = 36 would need 44: 45 KB, over the static shared-memory limit -> 37)
  static constexpr int LD = (NB == 24) ? 28 : NB + 1;
  double c0[PER_WARP], c1[PER_WARP], g;
  int base;
};
template <int K>
HB_DI void pixel_hess_reset(PixelHessAcc<K>& acc, int base) {
#pragma unroll
  for (int q = 0; q < PixelHessAcc<K>::PER_WARP; ++q) { acc.c0[q] = 0.0; acc.c1[q] = 0.0; }
  acc.g = 0.0; acc.base = base;
}
template <int K>
HB_DI void pixel_hess_flush(const PixelArgs& a, const PixelHessAcc<K>& acc) {
  constexpr int NB = 6 * K, NTILES = PixelHessAcc<K>::NTILES;
  if (acc.base < 0) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, lm = lane >> 2, lk = lane & 3;
  double* S = a.sys;
  const int c0 = 6 * acc.base;
#pragma unroll
  for (int q = 0; q < PixelHessAcc<K>::PER_WARP; ++q) {
    const int tile = warp + 2 * q;
    if (tile >= NTILES) continue;
    int ti = 0;
    while ((ti + 1) * (ti + 2) / 2 <= tile) ++ti;
    const int tj = tile - ti * (ti + 1) / 2;
    const int rr = 8 * ti + lm, cc = 8 * tj + 2 * lk;
    if (rr < NB) {
      if (cc < NB && cc <= rr) atomicAdd(&S[sys_index(a.lay, c0 + rr, c0 + cc)], acc.c0[q]);
      if (cc + 1 < NB && cc + 1 <= rr) atomicAdd(&S[sys_index(a.lay, c0 + rr, c0 + cc + 1)], acc.c1[q]);
      // diag(J^T J) is accumulated on its own (the LM damping needs it BEFORE the Schur complement touches S)
      if (cc == rr) atomicAdd(&S[a.lay.oD + c0 + rr], acc.c0[q]);
      if (cc + 1 == rr) atomicAdd(&S[a.lay.oD + c0 + rr], acc.c1[q]);
    }
  }
  if (tid >= kEvalThreads - NB) atomicAdd(&S[a.lay.og + c0 + tid - (kEvalThreads - NB)], acc.g);
}

// lower-triangle tile number -> (tile row, tile column), compile time
__host__ __device__ constexpr int tile_row(int tile) { int ti = 0; while ((ti + 1) * (ti + 2) / 2 <= tile) ++ti; return ti; }
__host__ __device__ constexpr int tile_col(int tile) { return tile - tile_row(tile) * (tile_row(tile) + 1) / 2; }

// one k-step (4 Jacobian rows) of every tile warp W owns: the NT column fragments are loaded once and serve as A and B
// operand of all of them; the PER_WARP accumulators are independent, so the DMMAs of a step overlap
template <int K, int W>
HB_DI void pixel_hess_steps(PixelHessAcc<K>& acc, const double* sJ, int r_lo, int r_hi, int lm, int lk) {
  constexpr int NB = 6 * K, LD = PixelHessAcc<K>::LD, NT = PixelHessAcc<K>::NT, NTILES = PixelHessAcc<K>::NTILES;
#pragma unroll 1
  for (int k0 = r_lo; k0 < r_hi; k0 += 4) {   // rows come in pairs: r_lo, r_hi are even; the tail of a segment is masked
    const bool in = k0 + lk < r_hi;
    const double* p = sJ + (k0 + lk) * LD + lm;
    double fr[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) fr[t] = (in && (8 * t + 8 <= NB || 8 * t + lm < NB)) ? p[8 * t] : 0.0;
#pragma unroll
    for (int q = 0; q < PixelHessAcc<K>::PER_WARP; ++q) {
      const int tile = W + 2 * q;
      if (tile < NTILES) {
        const double av = fr[tile_row(W + 2 * q < NTILES ? W + 2 * q : 0)], bv = fr[tile_col(W + 2 * q < NTILES ? W + 2 * q : 0)];
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(acc.c0[q]), "+d"(acc.c1[q]) : "d"(av), "d"(bv));
      }
    }
  }
}

template <int K>
HB_DI void cta_pixel_hessian(const PixelArgs& a, int f0, int cnt, double* sJ /*[128][LD]*/, double* sr /*[128]*/, int* sseg /*[66]*/, PixelHessAcc<K>& acc) {
  constexpr int NB = 6 * K, LD = PixelHessAcc<K>::LD;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  __shared__ double s_sw[kEvalThreads];
  // per-factor scalars: sqrt(w), knot base, scaled residual
  int my_base = -1;
  if (tid < cnt) {
    const int f = f0 + tid;
    const double sw = sqrt(a.w[f]);
    const double2 rr = reinterpret_cast<const double2*>(a.r)[f];
    my_base = a.idx[f].x;
    s_sw[tid] = sw;
    sr[2 * tid] = sw * rr.x; sr[2 * tid + 1] = sw * rr.y;
  }
  // segments of equal knot base (bound order is sorted by base): factor t starts one iff its base differs from its
  // predecessor's; positions by ballot + popc (two warps), sseg[j] = first factor of segment j, sseg[nseg] = cnt
  const int prev = __shfl_up_sync(0xffffffffu, my_base, 1);
  __shared__ int s_edge[2], s_warp_cnt;
  if (lane == 31) s_edge[warp] = my_base;
  __syncthreads();   // (also: previous use of the scratch is complete; s_sw is visible)
  // staging: the CTA's 2 * cnt Jacobian rows are one contiguous run of global memory (just written: L2 hits) -- copied
  // cooperatively with coalesced 128-bit loads, scaled by sqrt(w) of their factor, pitch LD in shared memory
  {
    const double2* src = reinterpret_cast<const double2*>(a.Jp + static_cast<size_t>(f0) * 2 * NB);   // 16 B aligned
    const int total = cnt * NB;   // double2 elements
#pragma unroll 4
    for (int e = tid; e < total; e += kEvalThreads) {
      const double2 v = src[e];
      const int row = (2 * e) / NB, col = 2 * e - row * NB;   // NB is even: a pair never straddles two rows
      const double sw = s_sw[row >> 1];
      sJ[row * LD + col] = sw * v.x; sJ[row * LD + col + 1] = sw * v.y;
    }
  }
  const int before = (lane == 0) ? (warp == 0 ? -2 : s_edge[0]) : prev;
  const bool start = tid < cnt && my_base != before;
  const unsigned mask = __ballot_sync(0xffffffffu, start);
  if (warp == 0 && lane == 0) s_warp_cnt = __popc(mask);
  __syncthreads();
  const int pos = __popc(mask & ((1u << lane) - 1u)) + (warp ? s_warp_cnt : 0);
  if (start) sseg[pos] = tid;
  if (tid == 0) sseg[65] = 0;
  __syncthreads();
  if (warp == 1 && lane == 0) { const int n = s_warp_cnt + __popc(mask); sseg[n] = cnt; sseg[65] = n; }
  __syncthreads();
  const int nseg = sseg[65];
  const int lm = lane >> 2, lk = lane & 3;
  for (int j = 0; j < nseg; ++j) {
    const int r_lo = 2 * sseg[j], r_hi = 2 * sseg[j + 1];
    const int base = a.idx[f0 + sseg[j]].x;
    if (base != acc.base) { pixel_hess_flush<K>(a, acc); pixel_hess_reset<K>(acc, base); }   // (uniform across the CTA)
    if (warp == 0) pixel_hess_steps<K, 0>(acc, sJ, r_lo, r_hi, lm, lk);
    else pixel_hess_steps<K, 1>(acc, sJ, r_lo, r_hi, lm, lk);
    if (tid >= kEvalThreads - NB) {   // gradient: the last NB threads
      const int c = tid - (kEvalThreads - NB);
      double g0 = 0.0, g1 = 0.0;
      for (int row = r_lo; row < r_hi; row += 2) { g0 += sJ[row * LD + c] * sr[row]; g1 += sJ[(row + 1) * LD + c] * sr[row + 1]; }
      acc.g += g0 + g1;
    }
  }
}

// bid: the CTA's index within the pixel grid (the merged factor kernel offsets it)
template <int K, bool WANT_J, bool FUSE>
HB_DI void pixel_eval_body(const PixelArgs& a, const Basis& B, int bid0) {
  __shared__ __align__(16) double s_tab[kTileRows * kTabStride];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ int s_red[2];
  __shared__ double s_cost[kEvalThreads / 32];
  // scratch of the fused J^T J accumulation (the CTA's 64 factors = 128 Jacobian rows in one pass)
  __shared__ double s_J[FUSE ? 128 * PixelHessAcc<K>::LD : 1];
  __shared__ double s_r[FUSE ? 128 : 1];
  __shared__ int s_b[FUSE ? 66 : 1];
  const int T = (FUSE && a.tiles_per_cta > 1) ? a.tiles_per_cta : 1;
  PixelHessAcc<K> acc;
  if (FUSE) pixel_hess_reset<K>(acc, -1);
  for (int tt = 0; tt < T; ++tt) {
  const int bid = bid0 * T + tt;
  if (bid * kEvalThreads >= a.n) break;
  if (tt) __syncthreads();   // the previous tile's shared-memory state (table tile, mbarrier, J^T J scratch) is done with
  const int f = bid * kEvalThreads + threadIdx.x;
  const bool active = f < a.n;
  int4 id = make_int4(0, 0, 0, 0);
  if (active) id = a.idx[f];
  int bmin, bmax;
  block_min_max(active ? id.x : 0x7fffffff, active ? id.x : -0x7fffffff, s_red, &bmin, &bmax);
  const int rows = bmax - bmin + K;
  const bool staged = rows <= kTileRows;
  if (staged) stage_table(s_tab, &s_bar, a.tab, bmin, rows);
  double cost = 0.0;
  if (active) {
    const double t = a.stamp[f];
    const double2 z = a.pixel[f];
    const double* cam = a.cam_tab + kCamStride * id.z;
    const double* lmk = a.landmarks + 3 * static_cast<size_t>(id.y);
    double r[2];
    double* Jp = WANT_J ? a.Jp + static_cast<size_t>(f) * 12 * K : nullptr;
    double* Jl = WANT_J ? a.Jl + static_cast<size_t>(f) * 6 : nullptr;
    const double zz = (id.w != 0) ? a.meas_z[f] : 0.0;
    if (staged) pixel_factor<K, WANT_J>(s_tab - static_cast<ptrdiff_t>(bmin) * kTabStride, B, id.x, t, z.x, z.y, zz, id.w, cam, lmk, r, Jp, Jl);
    else pixel_factor<K, WANT_J>(a.tab, B, id.x, t, z.x, z.y, zz, id.w, cam, lmk, r, Jp, Jl);
    if (a.r) reinterpret_cast<double2*>(a.r)[f] = make_double2(r[0], r[1]);
    double wgt;
    cost = 0.5 * huber_rho(r[0] * r[0] + r[1] * r[1], (id.w != 0) ? a.huber_bearing : a.huber, &wgt);
    if (WANT_J) a.w[f] = wgt;
  }
  // deterministic block reduction of the cost
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cost += __shfl_xor_sync(0xffffffffu, cost, o);
  if ((threadIdx.x & 31) == 0) s_cost[threadIdx.x >> 5] = cost;
  __syncthreads();
  if (threadIdx.x == 0) {
    double c = 0;
    for (int w = 0; w < kEvalThreads / 32; ++w) c += s_cost[w];
    a.cost_partial[bid] = c;
  }
  if (FUSE && a.sys != nullptr) {
    // fused normal equations of this CTA's factors (residuals / Jacobians were written above; the barrier in the
    // cost reduction ordered them for the whole CTA)
    const int f_lo = bid * kEvalThreads;
    cta_pixel_hessian<K>(a, f_lo, min(kEvalThreads, a.n - f_lo), s_J, s_r, s_b, acc);
  }
  }   // tiles
  if (FUSE && a.sys != nullptr) pixel_hess_flush<K>(a, acc);
}

template <int K, bool WANT_J, bool FUSE = false>
__global__ void __launch_bounds__(kEvalThreads, (K == 4 && FUSE) ? 6 : 1) pixel_eval_kernel(PixelArgs a, Basis B) { pixel_eval_body<K, WANT_J, FUSE>(a, B, blockIdx.x); }

// ---------------------------------------------------------------------------------------------
// Inertial factor (a6 + a3 with value/velocity/acceleration Jacobian stacks fused).
// ---------------------------------------------------------------------------------------------
struct InertialArgs {
  int n;
  const double* stamp;
  const double* meas;      // [n][6]
  const int4* idx;         // (base, gyro bias base, accel bias base, -)
  const double* tab;
  const double* imu_tab;
  const double* bg;        // [Kbg][4]
  const double* ba;        // [Kba][4]
  const double* gravity;   // [3]
  double* r;               // [n][6]
  double* Jp;              // [n][6][6K]
  double* wg;              // [n][KB]
  double* wa;              // [n][KB]
  double* Jg;              // [n][6][2]
  double* cost_partial;
  double loss_scale;
};

// Ceres SphereManifold<3> plus-Jacobian (3x2): |x| (I - beta v v^T)[:, 0:2].
HB_DI void sphere_plus_jacobian(const double* x, double* J /*3x2*/) {
  const double sigma = x[0] * x[0] + x[1] * x[1];
  double v[3] = {x[0], x[1], 1.0};
  double beta = 0.0;
  const double xp = x[2];
  if (sigma <= 2.220446049250313e-16) {
    if (xp < 0.0) beta = 2.0;
  } else {
    const double mu = sqrt(xp * xp + sigma);
    const double vp = (xp <= 0.0) ? (xp - mu) : (-sigma / (xp + mu));
    beta = 2.0 * vp * vp / (sigma + vp * vp);
    v[0] /= vp; v[1] /= vp;
  }
  const double nx = sqrt(sigma + xp * xp);
#pragma unroll
  for (int c = 0; c < 2; ++c)
#pragma unroll
    for (int r = 0; r < 3; ++r) J[2 * r + c] = nx * ((r == c ? 1.0 : 0.0) - beta * v[c] * v[r]);
}

template <int K, int KB, bool WANT_J>
HB_DI void inertial_factor(const double* __restrict__ T, const Basis& B, const Basis& BB, int base, int gb, int ab, double t,
                           const double* __restrict__ z, const double* __restrict__ I, const double* __restrict__ bg,
                           const double* __restrict__ ba, const double* __restrict__ grav, double* r, double* __restrict__ Jp,
                           double* __restrict__ wg_out, double* __restrict__ wa_out, double* __restrict__ Jg,
                           double* __restrict__ stash /* shared memory, kInertialStash(K) doubles per thread, or null when !WANT_J */) {
  constexpr int left = (K - 1) / 2;
  const double* row0 = T + static_cast<size_t>(base) * kTabStride;
  const double t0 = row0[left * kTabStride + 24], t1 = row0[(left + 1) * kTabStride + 24];
  const double inv_dt = 1.0 / (t1 - t0);
  const double u = (t - t0) * inv_dt;
  double lam[K + 1], lamd[K + 1], lamdd[K + 1];
  basis_eval<K, true>(B, u, inv_dt, lam, lamd, lamdd);

  // ---- forward sweep: pose, body rates (Sommer et al. recursion) ----
  double P[9], pdd[3] = {0, 0, 0};
#pragma unroll
  for (int i = 0; i < 9; ++i) P[i] = row0[i];
  // What the backward sweep needs from step j -- A_j, lambda_j Jr(lambda_j d_j), A_j^T w, A_j^T wd, w_j: 27 doubles --
  // is parked in SHARED memory (slot s of this thread at stash[s * kEvalThreads]: conflict-free) instead of staying
  // live in registers across the residual and coefficient computations: with 81 (K = 4) / 135 (K = 6) more doubles
  // live the kernel sat at 255 registers and spilled 2.7 KB per thread, doubling its DRAM traffic.
  double w[3] = {0, 0, 0}, wd[3] = {0, 0, 0};
#pragma unroll 1
  for (int j = 1; j < K; ++j) {
    const double* rj = row0 + j * kTabStride;
    const double d[3] = {rj[12], rj[13], rj[14]};
    const double lw[3] = {lam[j] * d[0], lam[j] * d[1], lam[j] * d[2]};
    double Aj[9], Jr[9], Pn[9];
    so3_exp_and_Jr(lw, Aj, WANT_J ? Jr : nullptr);
    m3_mul(P, Aj, Pn);
#pragma unroll
    for (int i = 0; i < 9; ++i) P[i] = Pn[i];
    double aw[3], awd[3], wn[3], cr[3];
    m3_tvec(Aj, w, aw);
    m3_tvec(Aj, wd, awd);
#pragma unroll
    for (int c = 0; c < 3; ++c) wn[c] = aw[c] + lamd[j] * d[c];
    cross(wn, d, cr);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      wd[c] = awd[c] + lamd[j] * cr[c] + lamdd[j] * d[c];
      w[c] = wn[c];
      pdd[c] += lamdd[j] * (rj[9 + c] - rj[9 + c - kTabStride]);
    }
    if (WANT_J) {
      double* sj = stash + (j - 1) * 27 * kEvalThreads;
#pragma unroll
      for (int i = 0; i < 9; ++i) { sj[i * kEvalThreads] = Aj[i]; sj[(9 + i) * kEvalThreads] = lam[j] * Jr[i]; }
#pragma unroll
      for (int c = 0; c < 3; ++c) { sj[(18 + c) * kEvalThreads] = aw[c]; sj[(21 + c) * kEvalThreads] = awd[c]; sj[(24 + c) * kEvalThreads] = wn[c]; }
    }
  }
  // ---- bias splines (value + basis weights) ----
  double bgv[3] = {0, 0, 0}, bav[3] = {0, 0, 0};
  {
    constexpr int lb = (KB - 1) / 2;
    double lb_[KB + 1];
    const double* g0 = bg + 4 * static_cast<size_t>(gb);
    const double s0 = g0[4 * lb + 3], s1 = g0[4 * (lb + 1) + 3];
    basis_eval<KB, false>(BB, (t - s0) / (s1 - s0), 0.0, lb_, nullptr, nullptr);
#pragma unroll
    for (int m = 0; m < KB; ++m) {
      const double wv = lb_[m] - lb_[m + 1];
      if (WANT_J) wg_out[m] = wv;
#pragma unroll
      for (int c = 0; c < 3; ++c) bgv[c] += wv * g0[4 * m + c];
    }
    const double* a0 = ba + 4 * static_cast<size_t>(ab);
    const double u0 = a0[4 * lb + 3], u1 = a0[4 * (lb + 1) + 3];
    basis_eval<KB, false>(BB, (t - u0) / (u1 - u0), 0.0, lb_, nullptr, nullptr);
#pragma unroll
    for (int m = 0; m < KB; ++m) {
      const double wv = lb_[m] - lb_[m + 1];
      if (WANT_J) wa_out[m] = wv;
#pragma unroll
      for (int c = 0; c < 3; ++c) bav[c] += wv * a0[4 * m + c];
    }
  }
  // ---- residual (reference inertial.cpp:62-79) ----
  const double* Rsb = I;
  const double* IgR = I + 12;
  const double* IaR = I + 21;
  const double* Sg = I + 30;
  const double* lever = I + 39;  // row i = c_i
  const double* IlinR = I + 48;  // Jacobian-side matrices (== IaR, Sg, lever unless a reference quirk is switched on)
  const double* SgJ = I + 57;
  const double* leverJ = I + 66;
  const double gm[3] = {pdd[0] - grav[0], pdd[1] - grav[1], pdd[2] - grav[2]};
  double a_i[3], a_m[3];
  m3_tvec(P, gm, a_i);  // R^T (pdd - g) = A_lin - R_bw g
  double Fa[9];
  {
    const double ww = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) Fa[3 * i + j] = w[i] * w[j] - (i == j ? ww : 0.0);
    Fa[1] -= wd[2]; Fa[2] += wd[1]; Fa[3] += wd[2]; Fa[5] -= wd[0]; Fa[6] -= wd[1]; Fa[7] += wd[0];
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) a_m[i] = a_i[i] + Fa[3 * i] * lever[3 * i] + Fa[3 * i + 1] * lever[3 * i + 1] + Fa[3 * i + 2] * lever[3 * i + 2];
  {
    double t1v[3], t2v[3], t3v[3];
    m3_vec(IgR, w, t1v);
    m3_vec(Sg, a_m, t2v);
    m3_vec(IaR, a_m, t3v);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      r[c] = t1v[c] + t2v[c] + bgv[c] - z[c];
      r[3 + c] = t3v[c] + bav[c] - z[3 + c];
    }
  }
  if (!WANT_J) return;

  // ---- coefficient matrices: rows 0-2 gyro, 3-5 accel ----
  // d a_m / d theta = hat(a_i) R^T ; d a_m / d omega = Kw ; d a_m / d alpha = Kal ; d a_m / d pdd_w = R^T
  double Bm[9];  // hat(a_i) R^T
  {
    double Rt[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) Rt[3 * i + j] = P[3 * j + i];
    hat_mul(a_i, Rt, Bm);
  }
  double Kw[9], Kal[9];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double* c = leverJ + 3 * i;
    // row i of -(2 w^ c^ - c^ w^) ; (w^ c^) = c w^T - (w.c) I ; (c^ w^) = w c^T - (w.c) I
    const double wc = w[0] * c[0] + w[1] * c[1] + w[2] * c[2];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double wxcx = c[i] * w[j] - (i == j ? wc : 0.0);
      const double cxwx = w[i] * c[j] - (i == j ? wc : 0.0);
      Kw[3 * i + j] = -(2.0 * wxcx - cxwx);
    }
    // row i of -c^
    Kal[3 * i] = (i == 0) ? 0.0 : (i == 1 ? -c[2] : c[1]);
    Kal[3 * i + 1] = (i == 0) ? c[2] : (i == 1 ? 0.0 : -c[0]);
    Kal[3 * i + 2] = (i == 0) ? -c[1] : (i == 1 ? c[0] : 0.0);
  }
  // The 6 x 3 coefficient matrices [S_g ; I R_sb] {Bm, Kw, Kal} (+ I_g R_sb for the rate) are NOT materialised: with
  //   M_j = Bm TG_j + Kw XG_j + Kal YG_j      the block of step j is   [S_g M_j + I_g R_sb XG_j ; I_lin R_sb M_j]
  // -- 54 fewer live doubles across the backward sweep (the calibration matrices sit in shared memory) and six 3x3
  // products per step instead of nine 6x3x3 ones.
  double Cp[18];
  m3_mult(SgJ, P, &Cp[0]);  // S_g R^T
  m3_mult(IaR, P, &Cp[9]);  // I_a R_sb R^T (inertial.cpp:150,198 use I_a in every variant)
  (void)Rsb;
  // gravity tangent Jacobian: -(Cp) * PlusJacobian_sphere(g)   (6x2)
  {
    double PJ[6];
    sphere_plus_jacobian(grav, PJ);
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
      for (int c = 0; c < 2; ++c) Jg[2 * i + c] = -(Cp[3 * i] * PJ[c] + Cp[3 * i + 1] * PJ[2 + c] + Cp[3 * i + 2] * PJ[4 + c]);
  }
  // ---- backward sweep over j = K-1 .. 1 ----
  double Pc[9], QT[9], Z[9], Dprev[18];
#pragma unroll
  for (int i = 0; i < 9; ++i) { Pc[i] = P[i]; QT[i] = (i % 4 == 0) ? 1.0 : 0.0; Z[i] = 0.0; }
#pragma unroll
  for (int i = 0; i < 18; ++i) Dprev[i] = 0.0;
#pragma unroll 1   // one step's live set at a time: fully unrolled, the scheduler interleaved the steps and spilled 2.4 KB per thread
  for (int j = K - 1; j >= 1; --j) {
    const double* rj = row0 + j * kTabStride;
    const double d[3] = {rj[12], rj[13], rj[14]};
    const double* sj = stash + (j - 1) * 27 * kEvalThreads;
    double lj[9], atw[3], atwd[3], wat[3];
#pragma unroll
    for (int i = 0; i < 9; ++i) lj[i] = sj[(9 + i) * kEvalThreads];
#pragma unroll
    for (int c = 0; c < 3; ++c) { atw[c] = sj[(18 + c) * kEvalThreads]; atwd[c] = sj[(21 + c) * kEvalThreads]; wat[c] = sj[(24 + c) * kEvalThreads]; }
    double X[9], Y[9], tmp[9], tmp2[9];
    hat_mul(atw, lj, X);
#pragma unroll
    for (int i = 0; i < 3; ++i) X[4 * i] += lamd[j];
    hat_mul(atwd, lj, Y);
    hat_mul(d, X, tmp);
    hat(wat, tmp2);
#pragma unroll
    for (int i = 0; i < 9; ++i) Y[i] += lamd[j] * (tmp2[i] - tmp[i]);
#pragma unroll
    for (int i = 0; i < 3; ++i) Y[4 * i] += lamdd[j];
    double Xf[9], Yf[9], Tf[9];
    m3_mul(QT, X, Xf);
    m3_mul(Z, X, Yf);
    m3_mul(QT, Y, tmp);
#pragma unroll
    for (int i = 0; i < 9; ++i) Yf[i] += tmp[i];
    m3_mul(Pc, lj, Tf);
    double G[9], TG[9], XG[9], YG[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) G[i] = rj[15 + i];
    m3_mul(Tf, G, TG);
    m3_mul(Xf, G, XG);
    m3_mul(Yf, G, YG);
    double D[18];
    {
      double M[9], t9[9];
      m3_mul(Bm, TG, M);
      m3_mul(Kw, XG, t9);
#pragma unroll
      for (int i = 0; i < 9; ++i) M[i] += t9[i];
      m3_mul(Kal, YG, t9);
#pragma unroll
      for (int i = 0; i < 9; ++i) M[i] += t9[i];
      m3_mul(SgJ, M, &D[0]);
      m3_mul(IgR, XG, t9);
#pragma unroll
      for (int i = 0; i < 9; ++i) D[i] += t9[i];
      m3_mul(IlinR, M, &D[9]);
    }
    // block m = j : rotation = D_j - D_{j+1}, translation = (lamdd_m - lamdd_{m+1}) * Cp
    {
      const double wdd = lamdd[j] - lamdd[j + 1];
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        double2* out = reinterpret_cast<double2*>(Jp + i * 6 * K + 6 * j);
        out[0] = make_double2(D[3 * i] - Dprev[3 * i], D[3 * i + 1] - Dprev[3 * i + 1]);
        out[1] = make_double2(D[3 * i + 2] - Dprev[3 * i + 2], wdd * Cp[3 * i]);
        out[2] = make_double2(wdd * Cp[3 * i + 1], wdd * Cp[3 * i + 2]);
      }
    }
#pragma unroll
    for (int i = 0; i < 18; ++i) Dprev[i] = D[i];
    // Pc <- Pc A_j^T ; Z <- (Z - lamd_j QT d^) A_j^T ; QT <- QT A_j^T
    double Aj[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) Aj[i] = sj[i * kEvalThreads];
    m3_mult(Pc, Aj, tmp);
#pragma unroll
    for (int i = 0; i < 9; ++i) Pc[i] = tmp[i];
    mul_hat(QT, d, tmp);
#pragma unroll
    for (int i = 0; i < 9; ++i) tmp2[i] = Z[i] - lamd[j] * tmp[i];
    m3_mult(tmp2, Aj, Z);
    m3_mult(QT, Aj, tmp);
#pragma unroll
    for (int i = 0; i < 9; ++i) QT[i] = tmp[i];
  }
  // block m = 0 : rotation = [S_g ; I_lin R_sb] Bm - D_1
  {
    double Cth[18];
    m3_mul(SgJ, Bm, &Cth[0]);
    m3_mul(IlinR, Bm, &Cth[9]);
    const double wdd = lamdd[0] - lamdd[1];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      double2* out = reinterpret_cast<double2*>(Jp + i * 6 * K);
      out[0] = make_double2(Cth[3 * i] - Dprev[3 * i], Cth[3 * i + 1] - Dprev[3 * i + 1]);
      out[1] = make_double2(Cth[3 * i + 2] - Dprev[3 * i + 2], wdd * Cp[3 * i]);
      out[2] = make_double2(wdd * Cp[3 * i + 1], wdd * Cp[3 * i + 2]);
    }
  }
}

// dynamic shared memory of the Jacobian pass of the inertial factors (the merged factor kernel carries it too)
constexpr size_t inertial_stash_bytes(int K) { return static_cast<size_t>(27) * (K - 1) * kEvalThreads * sizeof(double); }

template <int K, int KB, bool WANT_J>
HB_DI void inertial_eval_body(const InertialArgs& a, const Basis& B, const Basis& BB, int bid) {
  extern __shared__ double s_dyn_eval[];
  double* stash = WANT_J ? s_dyn_eval + threadIdx.x : nullptr;
  __shared__ __align__(16) double s_tab[kTileRows * kTabStride];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ int s_red[2];
  __shared__ double s_cost[kEvalThreads / 32];
  __shared__ double s_imu[kImuStride];
  __shared__ double s_grav[3];
  for (int i = threadIdx.x; i < kImuStride; i += kEvalThreads) s_imu[i] = a.imu_tab[i];
  if (threadIdx.x < 3) s_grav[threadIdx.x] = a.gravity[threadIdx.x];
  const int f = bid * kEvalThreads + threadIdx.x;
  const bool active = f < a.n;
  int4 id = make_int4(0, 0, 0, 0);
  if (active) id = a.idx[f];
  int bmin, bmax;
  block_min_max(active ? id.x : 0x7fffffff, active ? id.x : -0x7fffffff, s_red, &bmin, &bmax);
  const int rows = bmax - bmin + K;
  const bool staged = rows <= kTileRows;
  if (staged) stage_table(s_tab, &s_bar, a.tab, bmin, rows);
  double cost = 0.0;
  if (active) {
    const double t = a.stamp[f];
    double z[6];
    {
      const double2* zp = reinterpret_cast<const double2*>(a.meas + 6 * static_cast<size_t>(f));
      const double2 z0 = zp[0], z1 = zp[1], z2 = zp[2];
      z[0] = z0.x; z[1] = z0.y; z[2] = z1.x; z[3] = z1.y; z[4] = z2.x; z[5] = z2.y;
    }
    double r[6];
    double* Jp = WANT_J ? a.Jp + static_cast<size_t>(f) * 36 * K : nullptr;
    double* wg = WANT_J ? a.wg + static_cast<size_t>(f) * KB : nullptr;
    double* wa = WANT_J ? a.wa + static_cast<size_t>(f) * KB : nullptr;
    double* Jg = WANT_J ? a.Jg + static_cast<size_t>(f) * 12 : nullptr;
    if (staged)
      inertial_factor<K, KB, WANT_J>(s_tab - static_cast<ptrdiff_t>(bmin) * kTabStride, B, BB, id.x, id.y, id.z, t, z, s_imu, a.bg, a.ba,
                                     s_grav, r, Jp, wg, wa, Jg, stash);
    else
      inertial_factor<K, KB, WANT_J>(a.tab, B, BB, id.x, id.y, id.z, t, z, s_imu, a.bg, a.ba, s_grav, r, Jp, wg, wa, Jg, stash);
    double s = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i) s += r[i] * r[i];
    cost = 0.5 * a.loss_scale * s;
    if (a.r) {
      double2* ro = reinterpret_cast<double2*>(a.r + 6 * static_cast<size_t>(f));
      ro[0] = make_double2(r[0], r[1]); ro[1] = make_double2(r[2], r[3]); ro[2] = make_double2(r[4], r[5]);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cost += __shfl_xor_sync(0xffffffffu, cost, o);
  if ((threadIdx.x & 31) == 0) s_cost[threadIdx.x >> 5] = cost;
  __syncthreads();
  if (threadIdx.x == 0) {
    double c = 0;
    for (int w = 0; w < kEvalThreads / 32; ++w) c += s_cost[w];
    a.cost_partial[bid] = c;
  }
}
template <int K, int KB, bool WANT_J>
__global__ void __launch_bounds__(kEvalThreads) inertial_eval_kernel(InertialArgs a, Basis B, Basis BB) { inertial_eval_body<K, KB, WANT_J>(a, B, BB, blockIdx.x); }

// Visual and inertial factors in ONE launch (they are independent): CTAs [0, n_pix_blocks) run the pixel / bearing
// body, the rest the inertial body.  At 12 k factors each of these kernels is a ~20 us latency-bound launch; side by
// side they cost the longer of the two.
template <int K, int KB, bool WANT_J, bool FUSE>
__global__ void __launch_bounds__(kEvalThreads) factor_eval_kernel(PixelArgs pa, InertialArgs ia, Basis B, Basis BB, int n_pix_blocks) {
  pdl_launch_dependents();
  pdl_wait();   // (launched as a programmatic dependent of the knot-table / retraction kernel on the iteration path)
  if (static_cast<int>(blockIdx.x) < n_pix_blocks) pixel_eval_body<K, WANT_J, FUSE>(pa, B, blockIdx.x);
  else inertial_eval_body<K, KB, WANT_J>(ia, B, BB, blockIdx.x - n_pix_blocks);
}


// ---------------------------------------------------------------------------------------------
// Manifold (pose) factor: prediction T_ws = T_wb (+) T_bs (reference
// internal/hyper/optimizers/evaluators/manifold.cpp:12-61), residual = ManifoldMetric<SE3> =
// [Log(R_ws R_z^T) | p_ws - p_z] (wired at reference optimizer.cpp:237, no loss).  Outputs r[6] and
// Jp[6][6K] on the control-point tangents.  Pose factors are few (priors, ground-truth poses), so the
// kernel reads the knot table straight from L2 -- no staging.
// ---------------------------------------------------------------------------------------------
struct ManifoldArgs {
  int n;
  const double* stamp;
  const double* meas;      // [n][7] = [q(4) | p(3)]
  const int2* idx;         // (base, sensor)
  const double* tab;
  const double* sensors;   // [P][7] = T_bs of each pose sensor
  double* r;               // [n][6]
  double* Jp;              // [n][6][6K]
  double* cost_partial;    // [gridDim.x]
};

__global__ void bind_manifold_kernel(int n, const double* __restrict__ stamp, const int* __restrict__ sensor, const double* __restrict__ knots, int K,
                                     int k, int P, int2* __restrict__ idx, int* __restrict__ num_invalid) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const int base = segment_base(knots, 8, 7, K, k, stamp[f]);
  const int s = sensor[f];
  idx[f] = make_int2(base, s);
  if (base < 0 || s < 0 || s >= P) atomicAdd(num_invalid, 1);
}

template <int K, bool WANT_J>
__global__ void __launch_bounds__(kEvalThreads) manifold_eval_kernel(ManifoldArgs a, Basis B) {
  __shared__ double s_cost[kEvalThreads / 32];
  constexpr int left = (K - 1) / 2;
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  double cost = 0.0;
  if (f < a.n) {
    const int2 id = a.idx[f];
    const double* row0 = a.tab + static_cast<size_t>(id.x) * kTabStride;
    const double t0 = row0[left * kTabStride + 24], t1 = row0[(left + 1) * kTabStride + 24];
    const double inv_dt = 1.0 / (t1 - t0);
    const double u = (a.stamp[f] - t0) * inv_dt;
    double lam[K + 1];
    basis_eval<K, false>(B, u, inv_dt, lam, nullptr, nullptr);
    double P[9], p[3];
#pragma unroll
    for (int i = 0; i < 9; ++i) P[i] = row0[i];
    p[0] = row0[9]; p[1] = row0[10]; p[2] = row0[11];
    double M[(K - 1) * 9];
#pragma unroll
    for (int j = 1; j < K; ++j) {
      const double* rj = row0 + j * kTabStride;
      const double w[3] = {lam[j] * rj[12], lam[j] * rj[13], lam[j] * rj[14]};
      double A[9], Jr[9], Pn[9];
      so3_exp_and_Jr(w, A, WANT_J ? Jr : nullptr);
      m3_mul(P, A, Pn);
      if (WANT_J) {
        double G[9], JG[9], PJG[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) G[i] = rj[15 + i];
        m3_mul(Jr, G, JG);
        m3_mul(Pn, JG, PJG);
#pragma unroll
        for (int i = 0; i < 9; ++i) M[(j - 1) * 9 + i] = lam[j] * PJG[i];
      }
#pragma unroll
      for (int i = 0; i < 9; ++i) P[i] = Pn[i];
#pragma unroll
      for (int c = 0; c < 3; ++c) p[c] += lam[j] * (rj[9 + c] - rj[9 + c - kTabStride]);
    }
    const double* T_bs = a.sensors + 7 * static_cast<size_t>(id.y);
    const double* z = a.meas + 7 * static_cast<size_t>(f);
    double Rbs[9], Rz[9], Rws[9], Rerr[9], Rt[3], q[4], th[3];
    quat_to_rot(T_bs, Rbs);
    quat_to_rot(z, Rz);
    m3_vec(P, T_bs + 4, Rt);
    m3_mul(P, Rbs, Rws);
    m3_mult(Rws, Rz, Rerr);
    rot_to_quat(Rerr, q);
    quat_log(q, th);
    double r[6] = {th[0], th[1], th[2], p[0] + Rt[0] - z[4], p[1] + Rt[1] - z[5], p[2] + Rt[2] - z[6]};
    if (a.r) {
#pragma unroll
      for (int i = 0; i < 6; ++i) a.r[6 * static_cast<size_t>(f) + i] = r[i];
    }
    cost = 0.5 * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2] + r[3] * r[3] + r[4] * r[4] + r[5] * r[5]);
    if (WANT_J) {
      const double nth[3] = {-th[0], -th[1], -th[2]};
      double A[9], H[9];
      so3_Jr_inv(nth, A);   // Jl^{-1}(theta) = Jr^{-1}(-theta)
      hat(Rt, H);
      double* out = a.Jp + static_cast<size_t>(f) * 36 * K;
#pragma unroll
      for (int m = 0; m < K; ++m) {
        double D[9], AD[9], HD[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) {
          const double cur = (m == 0) ? ((i % 4 == 0) ? 1.0 : 0.0) : M[(m - 1) * 9 + i];
          const double nxt = (m + 1 < K) ? M[m * 9 + i] : 0.0;
          D[i] = cur - nxt;   // d theta / d phi_m
        }
        m3_mul(A, D, AD);
        m3_mul(H, D, HD);
        const double wm = lam[m] - lam[m + 1];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            out[i * 6 * K + 6 * m + c] = AD[3 * i + c];
            out[i * 6 * K + 6 * m + 3 + c] = 0.0;
            out[(3 + i) * 6 * K + 6 * m + c] = -HD[3 * i + c];
            out[(3 + i) * 6 * K + 6 * m + 3 + c] = (i == c) ? wm : 0.0;
          }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cost += __shfl_xor_sync(0xffffffffu, cost, o);
  if ((threadIdx.x & 31) == 0) s_cost[threadIdx.x >> 5] = cost;
  __syncthreads();
  if (threadIdx.x == 0) {
    double c = 0;
    for (int w = 0; w < kEvalThreads / 32; ++w) c += s_cost[w];
    a.cost_partial[blockIdx.x] = c;
  }
}

// ---------------------------------------------------------------------------------------------
// Plain spline interpolation at arbitrary stamps (no Jacobians): pose [q|p], body velocity
// [omega | R^T pdot], body acceleration [alpha | R^T pddot].  Serves the reference's trajectory
// dump (reference apps/hyperslam/main.cpp:69-80: state->evaluate(StateQuery{stamp, kValueIndex})).
// ---------------------------------------------------------------------------------------------
template <int K>
__global__ void interpolate_kernel(int n, const double* __restrict__ stamps, const double* __restrict__ knots, const double* __restrict__ tab,
                                   int Kn, Basis B, double* __restrict__ pose, double* __restrict__ vel, double* __restrict__ acc,
                                   int* __restrict__ num_invalid) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const double t = stamps[f];
  const int base = segment_base(knots, 8, 7, Kn, K, t);
  if (base < 0) {
    atomicAdd(num_invalid, 1);
    for (int i = 0; i < 7; ++i) pose[7 * static_cast<size_t>(f) + i] = (i == 3) ? 1.0 : 0.0;
    if (vel) for (int i = 0; i < 6; ++i) vel[6 * static_cast<size_t>(f) + i] = 0.0;
    if (acc) for (int i = 0; i < 6; ++i) acc[6 * static_cast<size_t>(f) + i] = 0.0;
    return;
  }
  constexpr int left = (K - 1) / 2;
  const double* row0 = tab + static_cast<size_t>(base) * kTabStride;
  const double t0 = row0[left * kTabStride + 24], t1 = row0[(left + 1) * kTabStride + 24];
  const double inv_dt = 1.0 / (t1 - t0);
  double lam[K + 1], lamd[K + 1], lamdd[K + 1];
  basis_eval<K, true>(B, (t - t0) * inv_dt, inv_dt, lam, lamd, lamdd);
  const double* k0 = knots + 8 * static_cast<size_t>(base);
  double q[4] = {k0[0], k0[1], k0[2], k0[3]};
  double p[3] = {k0[4], k0[5], k0[6]}, pd[3] = {0, 0, 0}, pdd[3] = {0, 0, 0};
  double w[3] = {0, 0, 0}, wd[3] = {0, 0, 0};
#pragma unroll
  for (int j = 1; j < K; ++j) {
    const double* rj = row0 + j * kTabStride;
    const double d[3] = {rj[12], rj[13], rj[14]};
    const double lw[3] = {lam[j] * d[0], lam[j] * d[1], lam[j] * d[2]};
    double qe[4], qn[4], A[9], aw[3], awd[3], wn[3], cr[3];
    quat_exp(lw, qe);
    quat_mul(q, qe, qn);
#pragma unroll
    for (int i = 0; i < 4; ++i) q[i] = qn[i];
    so3_exp_and_Jr(lw, A, nullptr);
    m3_tvec(A, w, aw);
    m3_tvec(A, wd, awd);
#pragma unroll
    for (int c = 0; c < 3; ++c) wn[c] = aw[c] + lamd[j] * d[c];
    cross(wn, d, cr);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      wd[c] = awd[c] + lamd[j] * cr[c] + lamdd[j] * d[c];
      w[c] = wn[c];
      const double dp = rj[9 + c] - rj[9 + c - kTabStride];
      p[c] += lam[j] * dp; pd[c] += lamd[j] * dp; pdd[c] += lamdd[j] * dp;
    }
  }
  double* o = pose + 7 * static_cast<size_t>(f);
  o[0] = q[0]; o[1] = q[1]; o[2] = q[2]; o[3] = q[3]; o[4] = p[0]; o[5] = p[1]; o[6] = p[2];
  if (vel || acc) {
    double R[9], v[3], a[3];
    quat_to_rot(q, R);
    m3_tvec(R, pd, v);
    m3_tvec(R, pdd, a);
    if (vel) { double* ov = vel + 6 * static_cast<size_t>(f); ov[0] = w[0]; ov[1] = w[1]; ov[2] = w[2]; ov[3] = v[0]; ov[4] = v[1]; ov[5] = v[2]; }
    if (acc) { double* oa = acc + 6 * static_cast<size_t>(f); oa[0] = wd[0]; oa[1] = wd[1]; oa[2] = wd[2]; oa[3] = a[0]; oa[4] = a[1]; oa[5] = a[2]; }
  }
}

// ---------------------------------------------------------------------------------------------
// Ingest step in front of the hot path (SURVEY.md section 8f rank 4; reference
// internal/hyper/optimizers/abstract.cpp:186-264): per stereo track, the bearings of both views
// (C.convertPixelsToBearings, :221-223) and the triangulated landmark in the world frame
// (Camera::Triangulate(T_01, b0, b1), :252; T_w0.vectorPlus, :253) at the CURRENT state.  The two
// camera functions live in HyperSensors (not in the tree): pixel -> bearing inverts the
// radial-tangential model with Newton iterations on the evaluator's own forward model; Triangulate is
// the midpoint of the common perpendicular [INFERRED].  One track per thread.
// ---------------------------------------------------------------------------------------------
HB_DI void pixel_to_bearing(const double* __restrict__ cam /* raw [T_bs 7 | cx cy fx fy | k1 k2 p1 p2] */, double px, double py, double* b) {
  const double cx = cam[7], cy = cam[8], fx = cam[9], fy = cam[10];
  const double k1 = cam[11], k2 = cam[12], p1 = cam[13], p2 = cam[14];
  const double dx = (px - cx) / fx, dy = (py - cy) / fy;
  double x = dx, y = dy;
#pragma unroll 1
  for (int it = 0; it < 10; ++it) {
    const double r2 = x * x + y * y;
    const double rad = 1.0 + k1 * r2 + k2 * r2 * r2;
    const double ox = x * rad + 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x);
    const double oy = y * rad + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y;
    const double g = k1 + 2.0 * k2 * r2;
    const double drx = 2.0 * x * g, dry = 2.0 * y * g;
    const double j00 = rad + x * drx + 2.0 * p1 * y + 6.0 * p2 * x;
    const double j01 = x * dry + 2.0 * p1 * x + 2.0 * p2 * y;
    const double j10 = y * drx + 2.0 * p1 * x + 2.0 * p2 * y;
    const double j11 = rad + y * dry + 6.0 * p1 * y + 2.0 * p2 * x;
    const double e0 = ox - dx, e1 = oy - dy;
    const double idet = 1.0 / (j00 * j11 - j01 * j10);
    x -= (j11 * e0 - j01 * e1) * idet;
    y -= (-j10 * e0 + j00 * e1) * idet;
  }
  const double inv = rsqrt(x * x + y * y + 1.0);
  b[0] = x * inv; b[1] = y * inv; b[2] = inv;
}

// One stereo track: bearings b0 / b1 of both views and the triangulated world landmark lm at the state's pose at t.
// Returns the knot base of t, or -1 (outputs untouched) when the stamp or a camera index is invalid.  Shared by
// ingest_stereo_kernel and append_stereo_tracks_kernel (hb200_window.cuh); not inlined, so that both kernels run the
// same compiled code and produce the same bits (inlined, the two copies may contract multiply-adds differently).
template <int K>
__device__ __noinline__ int ingest_stereo_track(double t, int c0, int c1, double2 q0, double2 q1, const double* __restrict__ knots, const double* __restrict__ tab,
                              int Kn, const Basis& B, const double* __restrict__ cams, int C, double* b0, double* b1, double* lm) {
  const int base = segment_base(knots, 8, 7, Kn, K, t);
  if (base < 0 || c0 < 0 || c0 >= C || c1 < 0 || c1 >= C) return -1;
  // pose of the body at the stamp (value only)
  constexpr int left = (K - 1) / 2;
  const double* row0 = tab + static_cast<size_t>(base) * kTabStride;
  const double t0 = row0[left * kTabStride + 24], t1 = row0[(left + 1) * kTabStride + 24];
  const double inv_dt = 1.0 / (t1 - t0);
  double lam[K + 1];
  basis_eval<K, false>(B, (t - t0) * inv_dt, inv_dt, lam, nullptr, nullptr);
  double R[9], p[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = row0[i];
  p[0] = row0[9]; p[1] = row0[10]; p[2] = row0[11];
#pragma unroll
  for (int j = 1; j < K; ++j) {
    const double* rj = row0 + j * kTabStride;
    const double w[3] = {lam[j] * rj[12], lam[j] * rj[13], lam[j] * rj[14]};
    double A[9], Rn[9];
    so3_exp_and_Jr(w, A, nullptr);
    m3_mul(R, A, Rn);
#pragma unroll
    for (int i = 0; i < 9; ++i) R[i] = Rn[i];
#pragma unroll
    for (int c = 0; c < 3; ++c) p[c] += lam[j] * (rj[9 + c] - rj[9 + c - kTabStride]);
  }
  const double* ca = cams + 15 * static_cast<size_t>(c0);
  const double* cb = cams + 15 * static_cast<size_t>(c1);
  pixel_to_bearing(ca, q0.x, q0.y, b0);
  pixel_to_bearing(cb, q1.x, q1.y, b1);
  // T_01 = T_b0^-1 (+) T_b1: R_01 = R_b0^T R_b1, t_01 = R_b0^T (t_b1 - t_b0)
  double Ra[9], Rb[9], R01[9], d1[3], t01[3];
  quat_to_rot(ca, Ra);
  quat_to_rot(cb, Rb);
  m3_tmul(Ra, Rb, R01);
  const double dt[3] = {cb[4] - ca[4], cb[5] - ca[5], cb[6] - ca[6]};
  m3_tvec(Ra, dt, t01);
  m3_vec(R01, b1, d1);
  const double aa = b0[0] * b0[0] + b0[1] * b0[1] + b0[2] * b0[2], bb = b0[0] * d1[0] + b0[1] * d1[1] + b0[2] * d1[2];
  const double cc = d1[0] * d1[0] + d1[1] * d1[1] + d1[2] * d1[2];
  const double ee = b0[0] * t01[0] + b0[1] * t01[1] + b0[2] * t01[2], ff = d1[0] * t01[0] + d1[1] * t01[1] + d1[2] * t01[2];
  const double idet = 1.0 / (aa * cc - bb * bb);
  const double sa = (ee * cc - bb * ff) * idet, ub = (bb * ee - aa * ff) * idet;
  double p0[3], pb[3], pw[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) p0[i] = 0.5 * (sa * b0[i] + t01[i] + ub * d1[i]);
  // world point: p_w = R (R_b0 p_0 + t_b0) + p
  m3_vec(Ra, p0, pb);
  pb[0] += ca[4]; pb[1] += ca[5]; pb[2] += ca[6];
  m3_vec(R, pb, pw);
#pragma unroll
  for (int i = 0; i < 3; ++i) lm[i] = pw[i] + p[i];
  return base;
}

template <int K>
__global__ void ingest_stereo_kernel(int n, const double* __restrict__ stamps, const int* __restrict__ cam0, const int* __restrict__ cam1,
                                     const double* __restrict__ px0, const double* __restrict__ px1, const double* __restrict__ knots,
                                     const double* __restrict__ tab, int Kn, Basis B, const double* __restrict__ cams, int C,
                                     double* __restrict__ b0_out, double* __restrict__ b1_out, double* __restrict__ lm_out,
                                     int* __restrict__ num_invalid) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const double2 q0 = make_double2(px0[2 * static_cast<size_t>(f)], px0[2 * static_cast<size_t>(f) + 1]);
  const double2 q1 = make_double2(px1[2 * static_cast<size_t>(f)], px1[2 * static_cast<size_t>(f) + 1]);
  double b0[3] = {0.0, 0.0, 0.0}, b1[3] = {0.0, 0.0, 0.0}, lm[3] = {0.0, 0.0, 0.0};
  if (ingest_stereo_track<K>(stamps[f], cam0[f], cam1[f], q0, q1, knots, tab, Kn, B, cams, C, b0, b1, lm) < 0) atomicAdd(num_invalid, 1);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    b0_out[3 * static_cast<size_t>(f) + i] = b0[i];
    b1_out[3 * static_cast<size_t>(f) + i] = b1[i];
    lm_out[3 * static_cast<size_t>(f) + i] = lm[i];
  }
}

}  // namespace hb
