// Device-side sliding-window bookkeeping (sm_100a): what the reference does per message on its pointer graph --
// appending state elements by extrapolation (reference internal/hyper/optimizers/abstract.cpp:118-144), adding
// residual blocks (reference internal/hyper/optimizers/ceres/optimizer.cpp:189-274), dropping landmarks whose
// observation range left the window together with their residuals (optimizer.cpp:360-382), setting state elements
// at or before the window's lower bound constant and removing the ones no residual touches any more
// (optimizer.cpp:286-345) -- here on the flattened window that already lives in HBM: no host re-sort, no re-upload
// of the factor lists.  New factors arrive in stamp order, so appending keeps the bound order (sorted by knot base);
// removal is an order-preserving stream compaction; the incidence lists (landmark CSR, inertial runs, segment
// offsets) are rebuilt by counting + scan kernels.  Integer work: bit-exact against the host path by construction.
#pragma once
#include "hb200_eval.cuh"

namespace hb {

// ---- exclusive scan of n ints by ONE CTA of 1024 threads (chunk by chunk, carry in a register); total -> *total ----
__global__ void __launch_bounds__(1024) scan_kernel(const int* __restrict__ in, int n, int* __restrict__ out, int* __restrict__ total) {
  __shared__ int s_warp[32];
  __shared__ int s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int i = base + tid;
    const int v = (i < n) ? in[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int w = s_warp[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
      s_warp[lane] = w;
    }
    __syncthreads();
    const int carry = s_carry;
    const int incl = x + (warp ? s_warp[warp - 1] : 0) + carry;
    if (i < n) out[i] = incl - v;
    __syncthreads();
    if (tid == 1023) s_carry = incl;
    __syncthreads();
  }
  if (tid == 0) *total = s_carry;
}

// order-preserving key of a double for atomicMax (stamps are finite)
HB_DI unsigned long long stamp_key(double t) {
  const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(t));
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
HB_DI double stamp_from_key(unsigned long long k) {
  const unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double(static_cast<long long>(b));
}

// last observation stamp of every landmark (key 0 = never observed)
__global__ void landmark_last_stamp_kernel(int n, const double* __restrict__ stamp, const int4* __restrict__ idx, unsigned long long* __restrict__ last) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < n) atomicMax(&last[idx[f].y], stamp_key(stamp[f]));
}
// a landmark stays while its observation range intersects the window: last stamp >= lower bound (reference
// optimizer.cpp:366: !p_landmark->range().intersects(range) -> remove); unobserved landmarks are kept (just added)
__global__ void landmark_keep_kernel(int L, const unsigned long long* __restrict__ last, double lower, int* __restrict__ keep) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l < L) keep[l] = (last[l] == 0ull || stamp_from_key(last[l]) >= lower) ? 1 : 0;
}
// visual factors live and die with their landmark; min_base receives the smallest knot base among the kept ones,
// bearing_kept the number of kept bearing factors (kind 1)
__global__ void visual_keep_kernel(int n, const int4* __restrict__ idx, const int* __restrict__ lm_keep, int* __restrict__ keep, int* __restrict__ min_base,
                                   int* __restrict__ bearing_kept) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const int4 id = idx[f];
  const int k = lm_keep[id.y];
  keep[f] = k;
  if (k) atomicMin(min_base, id.x);
  if (k && id.w) atomicAdd(bearing_kept, 1);
}
// inertial factors: kept (the reference never removes them); with drop_base >= 0 those whose control points ALL lie
// at or before the lower bound (base + order - 1 <= drop_base: every block the residual moves with is constant) go
__global__ void inertial_keep_kernel(int n, const int4* __restrict__ idx, int order, int drop_base, int* __restrict__ keep, int* __restrict__ min_base) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const int k = (drop_base >= 0 && idx[f].x + order - 1 <= drop_base) ? 0 : 1;
  keep[f] = k;
  if (k) atomicMin(min_base, idx[f].x);
}

// pose priors (manifold factors): kept, as in the reference; with drop_base >= 0 the same rule as inertial_keep_kernel
__global__ void manifold_keep_kernel(int n, const int2* __restrict__ idx, int order, int drop_base, int* __restrict__ keep, int* __restrict__ min_base) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const int k = (drop_base >= 0 && idx[f].x + order - 1 <= drop_base) ? 0 : 1;
  keep[f] = k;
  if (k) atomicMin(min_base, idx[f].x);
}

// (z: third component of a bearing measurement; pixel factors carry 0 there)
__global__ void compact_visual_kernel(int n, const int* __restrict__ keep, const int* __restrict__ pos, const int* __restrict__ lm_pos, int knot_shift,
                                      const double* __restrict__ stamp, const double2* __restrict__ pixel, const double* __restrict__ z,
                                      const int4* __restrict__ idx, double* __restrict__ stamp_o, double2* __restrict__ pixel_o,
                                      double* __restrict__ z_o, int4* __restrict__ idx_o) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n || !keep[f]) return;
  const int p = pos[f];
  int4 id = idx[f];
  id.x -= knot_shift; id.y = lm_pos[id.y];
  stamp_o[p] = stamp[f]; pixel_o[p] = pixel[f]; z_o[p] = z[f]; idx_o[p] = id;
}
__global__ void compact_manifold_kernel(int n, const int* __restrict__ keep, const int* __restrict__ pos, int knot_shift, const double* __restrict__ stamp,
                                        const double* __restrict__ meas, const int2* __restrict__ idx, double* __restrict__ stamp_o,
                                        double* __restrict__ meas_o, int2* __restrict__ idx_o) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n || !keep[f]) return;
  const int p = pos[f];
  int2 id = idx[f];
  id.x -= knot_shift;
  stamp_o[p] = stamp[f]; idx_o[p] = id;
#pragma unroll
  for (int q = 0; q < 7; ++q) meas_o[7 * static_cast<size_t>(p) + q] = meas[7 * static_cast<size_t>(f) + q];
}
__global__ void compact_inertial_kernel(int n, const int* __restrict__ keep, const int* __restrict__ pos, int knot_shift, const double* __restrict__ stamp,
                                        const double* __restrict__ meas, const int4* __restrict__ idx, double* __restrict__ stamp_o,
                                        double* __restrict__ meas_o, int4* __restrict__ idx_o) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n || !keep[f]) return;
  const int p = pos[f];
  int4 id = idx[f];
  id.x -= knot_shift;
  stamp_o[p] = stamp[f]; idx_o[p] = id;
#pragma unroll
  for (int q = 0; q < 6; ++q) meas_o[6 * static_cast<size_t>(p) + q] = meas[6 * static_cast<size_t>(f) + q];
}
__global__ void compact_landmarks_kernel(int L, const int* __restrict__ keep, const int* __restrict__ pos, const double* __restrict__ xyz, double* __restrict__ xyz_o) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= L || !keep[l]) return;
  const int p = pos[l];
#pragma unroll
  for (int c = 0; c < 3; ++c) xyz_o[3 * static_cast<size_t>(p) + c] = xyz[3 * static_cast<size_t>(l) + c];
}
__global__ void shift_knots_kernel(int K_new, int shift, const double* __restrict__ knots, double* __restrict__ knots_o) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < 8 * K_new) knots_o[e] = knots[8 * shift + e];
}

// reference abstract.cpp:126-136: the new element and the current last one take the variable of the second to last;
// stamps continue at the knot separation
__global__ void append_knots_kernel(int K, int count, double* __restrict__ knots) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  const double dt = knots[8 * (K - 1) + 7] - knots[8 * (K - 2) + 7];
  for (int q = 0; q < 7; ++q) knots[8 * (K - 1) + q] = knots[8 * (K - 2) + q];
  for (int i = 0; i < count; ++i) {
    for (int q = 0; q < 7; ++q) knots[8 * (K + i) + q] = knots[8 * (K - 2) + q];
    knots[8 * (K + i) + 7] = knots[8 * (K - 1) + 7] + (i + 1) * dt;
  }
}

// ---- incidence lists -------------------------------------------------------------------------------------------
__global__ void count_kernel(int n, const int4* __restrict__ idx, int which /*0: base (x), 1: landmark (y)*/, int* __restrict__ cnt) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < n) atomicAdd(&cnt[which ? idx[f].y : idx[f].x], 1);
}
// fill the landmark CSR; within a landmark the observations must come in bound order (ascending factor index): the
// factor list is sorted by base, so a landmark's first / last observation give its control-point span
__global__ void csr_fill_kernel(int n, const int4* __restrict__ idx, const int* __restrict__ off, int* __restrict__ cursor, int* __restrict__ obs) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const int l = idx[f].y;
  obs[off[l] + atomicAdd(&cursor[l], 1)] = f;
}
__global__ void csr_sort_kernel(int L, const int* __restrict__ off, int* __restrict__ obs, const int4* __restrict__ idx, int order, int* __restrict__ max_rows) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= L) return;
  const int lo = off[l], hi = off[l + 1];
  for (int i = lo + 1; i < hi; ++i) {   // insertion sort: tracks are a handful of observations
    const int v = obs[i];
    int j = i - 1;
    while (j >= lo && obs[j] > v) { obs[j + 1] = obs[j]; --j; }
    obs[j + 1] = v;
  }
  if (hi > lo) atomicMax(max_rows, 6 * (idx[obs[hi - 1]].x + order - idx[obs[lo]].x));
}
// inertial runs: a run starts where (base, gyro bias base, accel bias base) changes
__global__ void run_flag_kernel(int n, const int4* __restrict__ idx, int* __restrict__ flag) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  int s = 1;
  if (f > 0) { const int4 a = idx[f], b = idx[f - 1]; s = (a.x != b.x || a.y != b.y || a.z != b.z) ? 1 : 0; }
  flag[f] = s;
}
__global__ void run_fill_kernel(int n, const int* __restrict__ flag, const int* __restrict__ pos, int nruns, int* __restrict__ run_off) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < n && flag[f]) run_off[pos[f]] = f;
  if (f == 0) run_off[nruns] = n;
}
// bound-order check of an appended tail: every new base must be >= the last old one and the tail itself ascending
// (Idx = int4 for the visual / inertial lists, int2 for the manifold list: the base is .x in all of them)
template <typename Idx>
__global__ void tail_sorted_kernel(int n_old, int n_new, const Idx* __restrict__ idx, int* __restrict__ bad) {
  const int f = n_old + blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_old + n_new || f == 0) return;
  if (idx[f].x < idx[f - 1].x) atomicAdd(bad, 1);
}

// ---- stereo tracks (reference abstract.cpp:243-260: process(VisualTracks)) ----------------------------------------
// "new landmark" flags of the tracks (landmark_in == -1); any other value must be an existing window slot
__global__ void stereo_new_flags_kernel(int n, const int* __restrict__ lm_in, int L, int* __restrict__ flag, int* __restrict__ num_invalid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int l = lm_in[i];
  flag[i] = (l == -1) ? 1 : 0;
  if (l < -1 || l >= L) atomicAdd(num_invalid, 1);
}
// One thread per track: bearings of both views and, for a new landmark, the triangulated point at the current state
// (ingest_stereo_track).  Writes the two bearing factors of track i -- camera0's at Nv + 2i, camera1's at Nv + 2i + 1 --
// straight into the grown visual list (kind 1), and a new landmark into slot L + new_pos[i] of `lms`.  lm_out[i]
// receives the slot the track's factors reference.  Invalid tracks are counted; the caller then discards the tail.
template <int K>
__global__ void append_stereo_tracks_kernel(int n, const double* __restrict__ stamp, const double2* __restrict__ px0, const double2* __restrict__ px1,
                                            const int* __restrict__ cam0, const int* __restrict__ cam1, const int* __restrict__ lm_in,
                                            const int* __restrict__ new_pos, const double* __restrict__ knots, const double* __restrict__ tab, int Kn, Basis B,
                                            const double* __restrict__ cams, int C, int L, int Nv, double* __restrict__ v_stamp, double2* __restrict__ v_pixel,
                                            double* __restrict__ v_z, int4* __restrict__ v_idx, double* __restrict__ lms, int* __restrict__ lm_out,
                                            int* __restrict__ num_invalid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double t = stamp[i];
  const int c0 = cam0[i], c1 = cam1[i], li = lm_in[i];
  const int l = (li == -1) ? L + new_pos[i] : li;
  double b0[3] = {0.0, 0.0, 0.0}, b1[3] = {0.0, 0.0, 0.0}, p[3] = {0.0, 0.0, 0.0};
  const int base = ingest_stereo_track<K>(t, c0, c1, px0[i], px1[i], knots, tab, Kn, B, cams, C, b0, b1, p);
  if (base < 0) atomicAdd(num_invalid, 1);
  const size_t f = static_cast<size_t>(Nv) + 2 * static_cast<size_t>(i);
  v_stamp[f] = t; v_pixel[f] = make_double2(b0[0], b0[1]); v_z[f] = b0[2]; v_idx[f] = make_int4(base, l, c0, 1);
  v_stamp[f + 1] = t; v_pixel[f + 1] = make_double2(b1[0], b1[1]); v_z[f + 1] = b1[2]; v_idx[f + 1] = make_int4(base, l, c1, 1);
  if (li == -1) {
#pragma unroll
    for (int q = 0; q < 3; ++q) lms[3 * static_cast<size_t>(l) + q] = p[q];
  }
  lm_out[i] = l;
}
}  // namespace hb
