// ba_kernels.cuh — device kernels of the bundle-adjustment hot path (FP64 throughout).
//
// What each kernel replaces in the reference (ceres = src/third_party/ceres-solver):
//   cam_prep_kernel     ceres/include/ceres/rotation.h:563-622 (AngleAxisRotatePoint) hoisted per pose:
//                       R(w) and dR/dw_k by forward-mode duals of the same expression
//   eval_kernel         openMVG/sfm/sfm_data_BA_ceres_camera_functor.hpp (5 models) +
//                       ceres autodiff (internal/autodiff.h:207-319) + HuberLoss (loss_function.cc:47-61)
//                       + Corrector (corrector.cc:41-155) + ProgramEvaluator::Evaluate
//                       (program_evaluator.h:138-285) + Jacobi column scaling
//                       (trust_region_minimizer.cc:239-253)
//   point_accum_kernel  SchurEliminator::ChunkDiagonalBlockAndGradient (schur_eliminator_impl.h:434-490)
//   colsum_kernel       SquaredColumnNorm / gradient for the camera+intrinsic columns
//   schur_kernel        SchurEliminator::Eliminate (schur_eliminator_impl.h:176-298, :374-410, :499-548)
//   pcg_kernel          ConjugateGradientsSolver::Solve (conjugate_gradients_solver.cc:66-245) with a
//                       block-Jacobi preconditioner, standing in for SimplicialLDLT (eigensparse.cc:45-143)
//   dense_solve_kernel  the same solve done directly (dense L D L' in one CTA) for <= 220 reduced unknowns;
//                       dense_assemble / coarse_invert / dense_apply: explicit inverse up to 640
//   backsub_kernel      SchurEliminator::BackSubstitute (schur_eliminator_impl.h:303-366)
//   model_kernel        model_cost_change (trust_region_minimizer.cc:402-405)
//   update3_kernel      Program::Plus + SubsetParameterization::Plus (program.cc:115-127)
#pragma once
#include "common.cuh"
#include <cooperative_groups.h>
#include <cfloat>

namespace omvg { namespace ba {

namespace cg = cooperative_groups;
constexpr int KI = OMVG_BA_INTR_STRIDE;   // 8

// ------------------------------------------------------------------------------ small helpers
template <int N> struct Dual { double a; double v[N]; };
template <int N> __device__ __forceinline__ Dual<N> dconst(double s) { Dual<N> d; d.a = s; for (int i = 0; i < N; ++i) d.v[i] = 0; return d; }
template <int N> __device__ __forceinline__ Dual<N> dvar(double s, int k) { Dual<N> d = dconst<N>(s); d.v[k] = 1.0; return d; }
template <int N> __device__ __forceinline__ Dual<N> operator+(const Dual<N> &f, const Dual<N> &g) { Dual<N> h; h.a = f.a + g.a; for (int i = 0; i < N; ++i) h.v[i] = f.v[i] + g.v[i]; return h; }
template <int N> __device__ __forceinline__ Dual<N> operator-(const Dual<N> &f, const Dual<N> &g) { Dual<N> h; h.a = f.a - g.a; for (int i = 0; i < N; ++i) h.v[i] = f.v[i] - g.v[i]; return h; }
template <int N> __device__ __forceinline__ Dual<N> operator*(const Dual<N> &f, const Dual<N> &g) { Dual<N> h; h.a = f.a * g.a; for (int i = 0; i < N; ++i) h.v[i] = f.a * g.v[i] + f.v[i] * g.a; return h; }
template <int N> __device__ __forceinline__ Dual<N> operator/(const Dual<N> &f, const Dual<N> &g) { Dual<N> h; const double gi = 1.0 / g.a, q = f.a * gi; h.a = q; for (int i = 0; i < N; ++i) h.v[i] = (f.v[i] - q * g.v[i]) * gi; return h; }
template <int N> __device__ __forceinline__ Dual<N> dsqrt(const Dual<N> &f) { Dual<N> h; h.a = sqrt(f.a); const double t = 1.0 / (2.0 * h.a); for (int i = 0; i < N; ++i) h.v[i] = t * f.v[i]; return h; }
template <int N> __device__ __forceinline__ Dual<N> dcos(const Dual<N> &f) { Dual<N> h; h.a = cos(f.a); const double s = -sin(f.a); for (int i = 0; i < N; ++i) h.v[i] = s * f.v[i]; return h; }
template <int N> __device__ __forceinline__ Dual<N> dsin(const Dual<N> &f) { Dual<N> h; h.a = sin(f.a); const double c = cos(f.a); for (int i = 0; i < N; ++i) h.v[i] = c * f.v[i]; return h; }

// deterministic block sum (fixed tree); result valid in thread 0
template <int THREADS> __device__ __forceinline__ double block_sum(double v, double *sh /* THREADS/32 */) {
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  double t = 0;
  if (threadIdx.x == 0) for (int i = 0; i < THREADS / 32; ++i) t += sh[i];
  return t;
}

// 3x3 SPD inverse through LLT (invert_psd_matrix.h:56-59). m = {a00,a10,a11,a20,a21,a22}
__device__ __forceinline__ bool inv3_spd(const double m[6], double inv[9]) {
  const double l00 = sqrt(m[0]), l10 = m[1] / l00, l20 = m[3] / l00;
  const double l11 = sqrt(m[2] - l10 * l10), l21 = (m[4] - l20 * l10) / l11;
  const double l22 = sqrt(m[5] - l20 * l20 - l21 * l21);
  if (!(l00 > 0.0 && l11 > 0.0 && l22 > 0.0) || !isfinite(l00) || !isfinite(l11) || !isfinite(l22)) return false;
  #pragma unroll
  for (int c = 0; c < 3; ++c) {
    double b0 = c == 0 ? 1.0 : 0.0, b1 = c == 1 ? 1.0 : 0.0, b2 = c == 2 ? 1.0 : 0.0;
    b0 /= l00; b1 = (b1 - l10 * b0) / l11; b2 = (b2 - l20 * b0 - l21 * b1) / l22;
    b2 /= l22; b1 = (b1 - l21 * b2) / l11; b0 = (b0 - l10 * b1 - l20 * b2) / l00;
    inv[0 * 3 + c] = b0; inv[1 * 3 + c] = b1; inv[2 * 3 + c] = b2;
  }
  return true;
}

// ------------------------------------------------------------------------------ per-pose rotation
// camR[p][9] row-major R(w); camdR[p][k][9] = dR/dw_k.  Same expression as AngleAxisRotatePoint:
// R = cos I + sin [w]x + (1-cos) w w^T with w = aa/theta;  theta^2 <= eps: R = I + [aa]x.
// camrec[p][22] = {R (9), Jr (9, row-major; column k = vee(R' dR_k), so dR_k X = R (Jr e_k x X)), t (3), pad}:
// the compact per-pose record the per-observation kernel gathers with 11 x 16-byte loads.
constexpr int CAMREC = 22;
__global__ void cam_prep_kernel(const double *__restrict__ poses, int n_poses, double *__restrict__ camR, double *__restrict__ camdR, double *__restrict__ camrec) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_poses) return;
  typedef Dual<3> D;
  D aa[3]; for (int k = 0; k < 3; ++k) aa[k] = dvar<3>(poses[6 * p + k], k);
  const D theta2 = aa[0] * aa[0] + aa[1] * aa[1] + aa[2] * aa[2];
  D R[9];
  if (theta2.a > DBL_EPSILON) {
    const D theta = dsqrt(theta2), c = dcos(theta), s = dsin(theta), ti = dconst<3>(1.0) / theta;
    const D w[3] = {aa[0] * ti, aa[1] * ti, aa[2] * ti};
    const D omc = dconst<3>(1.0) - c;
    // column j of R = R e_j = e_j c + (w x e_j) s + w (w_j) (1-c)
    for (int j = 0; j < 3; ++j) {
      D e[3] = {dconst<3>(j == 0), dconst<3>(j == 1), dconst<3>(j == 2)};
      const D wx[3] = {w[1] * e[2] - w[2] * e[1], w[2] * e[0] - w[0] * e[2], w[0] * e[1] - w[1] * e[0]};
      const D tmp = (w[0] * e[0] + w[1] * e[1] + w[2] * e[2]) * omc;
      for (int i = 0; i < 3; ++i) R[i * 3 + j] = e[i] * c + wx[i] * s + w[i] * tmp;
    }
  } else {
    for (int j = 0; j < 3; ++j) {
      D e[3] = {dconst<3>(j == 0), dconst<3>(j == 1), dconst<3>(j == 2)};
      const D wx[3] = {aa[1] * e[2] - aa[2] * e[1], aa[2] * e[0] - aa[0] * e[2], aa[0] * e[1] - aa[1] * e[0]};
      for (int i = 0; i < 3; ++i) R[i * 3 + j] = e[i] + wx[i];
    }
  }
  for (int i = 0; i < 9; ++i) { camR[9 * p + i] = R[i].a; for (int k = 0; k < 3; ++k) camdR[27 * p + 9 * k + i] = R[i].v[k]; }
  double *rec = camrec + (size_t)CAMREC * p;
  for (int i = 0; i < 9; ++i) rec[i] = R[i].a;
  for (int k = 0; k < 3; ++k) {
    double M[9];                                             // R' dR_k  (skew up to rounding)
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { double v = 0; for (int l = 0; l < 3; ++l) v += R[l * 3 + i].a * R[l * 3 + j].v[k]; M[i * 3 + j] = v; }
    rec[9 + 0 * 3 + k] = 0.5 * (M[7] - M[5]); rec[9 + 1 * 3 + k] = 0.5 * (M[2] - M[6]); rec[9 + 2 * 3 + k] = 0.5 * (M[3] - M[1]);
  }
  rec[18] = poses[6 * p + 3]; rec[19] = poses[6 * p + 4]; rec[20] = poses[6 * p + 5]; rec[21] = 0.0;
}

// ------------------------------------------------------------------------------ problem setup on the device
// (the caller's observation arrays are uploaded as they are; sorting by landmark, the per-pose lists and the
// range checks run here instead of on the host: at 1M observations the host version cost more than the solve)
__global__ void setup_check_kernel(const int *__restrict__ obs_view, const int *__restrict__ obs_point, long long n, int n_views, int n_points,
                                   int *__restrict__ keys, int *__restrict__ iota, int *__restrict__ bad) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n) return;
  const int v = obs_view[o], j = obs_point[o];
  if (v < 0 || v >= n_views || j < 0 || j >= n_points) { atomicMin(bad, (int)o); keys[o] = 0; } else keys[o] = j;
  iota[o] = (int)o;
}
__global__ void setup_gather_kernel(const int *__restrict__ perm, const int *__restrict__ obs_view, const int *__restrict__ view_pose, const int *__restrict__ view_intr,
                                    const double2 *__restrict__ xy, const double *__restrict__ w_in, const unsigned char *__restrict__ fl_in, long long n, int n_views,
                                    int *__restrict__ s_pose, int *__restrict__ s_intr, double2 *__restrict__ s_xy, double *__restrict__ s_w, unsigned char *__restrict__ s_fl,
                                    int *__restrict__ iota) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int o = perm[t]; int v = obs_view[o]; v = min(max(v, 0), n_views - 1);
  s_pose[t] = view_pose[v]; s_intr[t] = view_intr[v];
  if (xy) { s_xy[t] = xy[o]; if (s_w) s_w[t] = w_in[o]; if (s_fl) s_fl[t] = fl_in[o] ? 1 : 0; }
  iota[t] = (int)t;
}
// the per-observation payload (image positions, weights, flags) into landmark order; runs last in omvg_ba_create so that
// its 16 B/observation upload (a second stream) overlaps the sorts and the structure build
__global__ void setup_gather_xy_kernel(const int *__restrict__ perm, const double2 *__restrict__ xy, const double *__restrict__ w_in, const unsigned char *__restrict__ fl_in,
                                       long long n, double2 *__restrict__ s_xy, double *__restrict__ s_w, unsigned char *__restrict__ s_fl) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int o = perm[t];
  s_xy[t] = xy[o];
  if (s_w) s_w[t] = w_in[o];
  if (s_fl) s_fl[t] = fl_in[o] ? 1 : 0;
}
// segment starts of a sorted key array: start[k] = first t with key[t] >= k, start[n_keys] = n (empty keys included)
__global__ void setup_starts_kernel(const int *__restrict__ key, long long n, int n_keys, int *__restrict__ start) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n) return;
  const int lo = t == 0 ? -1 : key[t - 1], hi = t == n ? n_keys : key[t];
  for (int k = lo + 1; k <= hi; ++k) start[k] = (int)t;
}
// pt_single[j] = all observations of landmark j go through one intrinsic group; n_slow counts the landmarks the
// warp-per-landmark Schur kernel does not take (several groups, or more than 32 observations)
__global__ void setup_single_kernel(const int *__restrict__ s_intr, const int *__restrict__ pt_start, int n_points, unsigned char *__restrict__ pt_single,
                                    int *__restrict__ n_slow) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_points) return;
  unsigned char one = 1;
  for (int t = pt_start[j] + 1; t < pt_start[j + 1]; ++t) if (s_intr[t] != s_intr[pt_start[j]]) { one = 0; break; }
  pt_single[j] = one;
  const int K = pt_start[j + 1] - pt_start[j];
  if (K > 0 && (!one || K > 32)) atomicAdd(n_slow, 1);
}

// ------------------------------------------------------------------------------ outlier rejection on the resident scene
// RemoveOutliers_PixelResidualError (sfm/sfm_data_filters.cpp:40-73) on the device: an observation whose reprojection
// residual norm exceeds the threshold is removed (weight 0, counted); then a track left with fewer than min_len
// observations is removed as a whole (its observations are not counted, as in the reference).  Removed bits are
// returned in the CALLER's observation order.  Ground control points (fixed landmarks that were fixed at create) and
// observations that are already removed are left alone.
__global__ void reject_obs_kernel(const double *__restrict__ rnorm, double *__restrict__ obs_w, const int *__restrict__ obs_pt, const unsigned char *__restrict__ pt_gcp,
                                  long long n, double thr, const int *__restrict__ perm, unsigned *__restrict__ removed_bits, unsigned long long *__restrict__ counters) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool out = false;
  if (t < n && obs_w[t] != 0.0 && !(pt_gcp && pt_gcp[obs_pt[t]]) && rnorm[t] > thr) {
    obs_w[t] = 0.0; const int o = perm[t]; atomicOr(&removed_bits[o >> 5], 1u << (o & 31)); out = true;
  }
  const unsigned b = __ballot_sync(0xffffffffu, out);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(&counters[0], (unsigned long long)__popc(b));
}
// mode 0: tracks with fewer than min_len live observations; mode 1: tracks named by kill[] (the host-side angle test)
__global__ void reject_tracks_kernel(const int *__restrict__ pt_start, int n_points, double *__restrict__ obs_w, int min_len, const unsigned char *__restrict__ kill,
                                     const unsigned char *__restrict__ pt_gcp, const int *__restrict__ perm, unsigned *__restrict__ removed_bits,
                                     unsigned char *__restrict__ pt_fixed, unsigned *__restrict__ pt_mask, unsigned char *__restrict__ pt_removed,
                                     unsigned char *__restrict__ removed_now, unsigned long long *__restrict__ counters) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_points) return;
  if (removed_now) removed_now[j] = 0;
  if (pt_removed[j] || (pt_gcp && pt_gcp[j])) return;
  int alive = 0;
  for (int t = pt_start[j]; t < pt_start[j + 1]; ++t) alive += obs_w[t] != 0.0;
  const bool gone = kill ? kill[j] != 0 : alive < min_len;
  if (!gone) return;
  for (int t = pt_start[j]; t < pt_start[j + 1]; ++t) if (obs_w[t] != 0.0) { obs_w[t] = 0.0; const int o = perm[t]; atomicOr(&removed_bits[o >> 5], 1u << (o & 31)); }
  pt_removed[j] = 1; pt_fixed[j] = 1; pt_mask[j] = 0u;       // a removed track is no longer a parameter block
  if (removed_now) removed_now[j] = 1;
  atomicAdd(&counters[1], 1ull);
}
__global__ void fill_kernel(double *__restrict__ p, long long n, double v) { const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }
__global__ void fill_u32_kernel(unsigned *__restrict__ p, long long n, unsigned v) { const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }

// ------------------------------------------------------------------------------ residual / Jacobian
struct EvalArgs {
  const double *poses, *intr, *pts, *camR, *camdR, *camrec, *obs_xy;
  const int *intr_model, *obs_pose, *obs_intr, *obs_pt;
  long long n_obs;
  int use_loss; double huber_a;
  // outputs (component-major: comp * n_obs + obs)
  double *r, *Jp, *Jc, *Ji;
  double *cost_partial;
  double *rnorm;                            // optional: |r| (pixels, before weight and loss) per observation
  // optional per-observation weight / flags and fixed landmarks (ground control points, sfm_data_BA_ceres.cpp:398-452;
  // weight 0 removes an observation without rebuilding the structure: the outlier-rejection loop)
  const double *obs_w; const unsigned char *obs_flags; const unsigned char *pt_fixed;
  // scaling & masks
  const double *sc_pt, *sc_cam, *sc_intr;   // null => unscaled
  int kiu;                                  // intrinsic columns in use (max nparams over the groups)
  unsigned pose_mask;                       // bit k set => pose coordinate k is free
  const unsigned *intr_mask;                // per intrinsic: bit k set => parameter k is free
  int pts_free;
};

// distortion d(u; K) and its derivatives: dd[2][2] = d d/du, dk[2][5] = d d/dK[3..7]
__device__ __forceinline__ void distort(int model, const double *K, double x, double y, double &dx, double &dy,
                                        double dd[4], double dk[10], bool want_j) {
  for (int i = 0; i < 10; ++i) dk[i] = 0.0;
  if (model == OMVG_PINHOLE_CAMERA) { dx = x; dy = y; dd[0] = 1; dd[1] = 0; dd[2] = 0; dd[3] = 1; return; }
  const double r2 = x * x + y * y;
  if (model == OMVG_PINHOLE_CAMERA_RADIAL1 || model == OMVG_PINHOLE_CAMERA_RADIAL3 || model == OMVG_PINHOLE_CAMERA_BROWN) {
    const double k1 = K[3], k2 = model == OMVG_PINHOLE_CAMERA_RADIAL1 ? 0.0 : K[4], k3 = model == OMVG_PINHOLE_CAMERA_RADIAL1 ? 0.0 : K[5];
    const double r4 = r2 * r2, r6 = r4 * r2;
    const double rc = 1.0 + k1 * r2 + k2 * r4 + k3 * r6;
    const double drc = k1 + 2.0 * k2 * r2 + 3.0 * k3 * r4;      // d rc / d r2
    dx = x * rc; dy = y * rc;
    if (want_j) {
      dd[0] = rc + x * drc * 2.0 * x; dd[1] = x * drc * 2.0 * y;
      dd[2] = y * drc * 2.0 * x;      dd[3] = rc + y * drc * 2.0 * y;
      dk[0] = x * r2; dk[5] = y * r2;
      if (model != OMVG_PINHOLE_CAMERA_RADIAL1) { dk[1] = x * r4; dk[2] = x * r6; dk[6] = y * r4; dk[7] = y * r6; }
    }
    if (model == OMVG_PINHOLE_CAMERA_BROWN) {
      const double t1 = K[6], t2 = K[7];
      dx += t2 * (r2 + 2.0 * x * x) + 2.0 * t1 * x * y;
      dy += t1 * (r2 + 2.0 * y * y) + 2.0 * t2 * x * y;
      if (want_j) {
        dd[0] += t2 * (2.0 * x + 4.0 * x) + 2.0 * t1 * y; dd[1] += t2 * 2.0 * y + 2.0 * t1 * x;
        dd[2] += t1 * 2.0 * x + 2.0 * t2 * y;             dd[3] += t1 * (2.0 * y + 4.0 * y) + 2.0 * t2 * x;
        dk[3] = 2.0 * x * y; dk[4] = r2 + 2.0 * x * x;
        dk[8] = r2 + 2.0 * y * y; dk[9] = 2.0 * x * y;
      }
    }
    return;
  }
  // fisheye (sfm_data_BA_ceres_camera_functor.hpp:609-626)
  const double r = sqrt(r2);
  if (r > 1e-8) {
    const double th = atan(r), th2 = th * th, th3 = th2 * th, th4 = th2 * th2, th5 = th4 * th, th7 = th3 * th3 * th, th8 = th4 * th4, th9 = th8 * th;
    const double thd = th + K[3] * th3 + K[4] * th5 + K[5] * th7 + K[6] * th9;
    const double cd = thd / r;
    dx = x * cd; dy = y * cd;
    if (want_j) {
      const double dthd_dth = 1.0 + 3.0 * K[3] * th2 + 5.0 * K[4] * th4 + 7.0 * K[5] * th3 * th3 + 9.0 * K[6] * th8;
      const double dth_dr = 1.0 / (1.0 + r2);
      const double dcd_dr = (dthd_dth * dth_dr - cd) / r;         // d(thd/r)/dr
      const double gx = dcd_dr * x / r, gy = dcd_dr * y / r;      // d cd / dx, dy
      dd[0] = cd + x * gx; dd[1] = x * gy; dd[2] = y * gx; dd[3] = cd + y * gy;
      const double ir = 1.0 / r;
      dk[0] = x * th3 * ir; dk[1] = x * th5 * ir; dk[2] = x * th7 * ir; dk[3] = x * th9 * ir;
      dk[5] = y * th3 * ir; dk[6] = y * th5 * ir; dk[7] = y * th7 * ir; dk[8] = y * th9 * ir;
    }
  } else { dx = x; dy = y; dd[0] = 1; dd[1] = 0; dd[2] = 0; dd[3] = 1; }
}

constexpr int EVAL_THREADS = 128;
// EXT = false compiles the weight / flag / fixed-landmark handling out (the common problem has none)
template <bool WANT_J, int MINB, bool EXT>
__global__ void __launch_bounds__(EVAL_THREADS, MINB) eval_kernel(EvalArgs A) {
  __shared__ double sh[EVAL_THREADS / 32];
  // persistent grid-stride loop; the (DRAM-latency) index / observation loads of the NEXT observation are
  // issued before the current one is processed
  const long long stride = (long long)gridDim.x * EVAL_THREADS;
  long long o = (long long)blockIdx.x * EVAL_THREADS + threadIdx.x;
  double cost = 0.0;
  int ip = 0, iq = 0, j = 0; double2 xy = make_double2(0.0, 0.0);
  if (o < A.n_obs) { ip = __ldcs(A.obs_pose + o); iq = __ldcs(A.obs_intr + o); j = __ldcs(A.obs_pt + o); xy = __ldcs(reinterpret_cast<const double2 *>(A.obs_xy) + o); }
  while (o < A.n_obs) {
    const long long o_next = o + stride;
    int ipn = 0, iqn = 0, jn = 0; double2 xyn = make_double2(0.0, 0.0);
    if (o_next < A.n_obs) { ipn = __ldcs(A.obs_pose + o_next); iqn = __ldcs(A.obs_intr + o_next); jn = __ldcs(A.obs_pt + o_next); xyn = __ldcs(reinterpret_cast<const double2 *>(A.obs_xy) + o_next); }
    double R[CAMREC];
    { const double2 *rp = reinterpret_cast<const double2 *>(A.camrec + (size_t)CAMREC * ip);
      #pragma unroll
      for (int q = 0; q < CAMREC / 2; ++q) { const double2 v = __ldg(rp + q); R[2 * q] = v.x; R[2 * q + 1] = v.y; } }
    const double X0 = __ldg(A.pts + 3 * j), X1 = __ldg(A.pts + 3 * j + 1), X2 = __ldg(A.pts + 3 * j + 2);
    const double *T = R + 18;
    const double p0 = R[0] * X0 + R[1] * X1 + R[2] * X2 + T[0];
    const double p1 = R[3] * X0 + R[4] * X1 + R[5] * X2 + T[1];
    const double p2 = R[6] * X0 + R[7] * X1 + R[8] * X2 + T[2];
    const double wg = (EXT && A.obs_w) ? __ldcs(A.obs_w + o) : 1.0;   // WeightedCostFunction (functor.hpp:35-90)
    const bool dead = EXT && wg == 0.0;                        // removed observation: contributes exact zeros
    const bool safe = dead && WANT_J;                          // keep every Jacobian factor finite so that 0 * J == 0
    const double iz = safe ? 1.0 : 1.0 / p2, x = safe ? 0.0 : p0 * iz, y = safe ? 0.0 : p1 * iz;
    const double *K = A.intr + KI * iq;
    const int model = A.intr_model[iq];
    double dx, dy, dd[4], dk[10];
    double r0, r1, f;
    double gs[6];                                               // spherical: d(projection)/dp (2x3), unweighted
    const bool spherical = model == OMVG_CAMERA_SPHERICAL;
    if (spherical) {
      // ResidualErrorFunctor_Intrinsic_Spherical (functor.hpp:662-717): lon = atan2(x, z), lat = atan2(-y, |(x, z)|),
      // pixel = (lon, -lat) / 2pi * max(w, h) + (w, h) / 2.  K[0], K[1] carry the image size; there is no intrinsic block.
      for (int i = 0; i < 10; ++i) dk[i] = 0.0;
      dx = 0.0; dy = 0.0; f = 0.0; dd[0] = dd[1] = dd[2] = dd[3] = 0.0;
      const double rho2 = safe ? 1.0 : p0 * p0 + p2 * p2, rho = sqrt(rho2), n2 = rho2 + (safe ? 0.0 : p1 * p1);
      const double k = fmax(K[0], K[1]) / (2.0 * 3.14159265358979323846);
      r0 = (safe ? 0.0 : atan2(p0, p2)) * k + K[0] / 2.0 - xy.x;
      r1 = -(safe ? 0.0 : atan2(-p1, rho)) * k + K[1] / 2.0 - xy.y;
      if (WANT_J) {
        const double i2 = 1.0 / rho2, in2 = 1.0 / n2, ir = 1.0 / rho;
        gs[0] = k * p2 * i2; gs[1] = 0.0; gs[2] = -k * p0 * i2;                       // k * dlon/dp
        gs[3] = -k * p1 * p0 * ir * in2; gs[4] = k * rho * in2; gs[5] = -k * p1 * p2 * ir * in2;   // -k * dlat/dp
      }
    } else {
      distort(model, K, x, y, dx, dy, dd, dk, WANT_J);
      f = K[0];
      r0 = K[1] + dx * f - xy.x; r1 = K[2] + dy * f - xy.y;
    }
    if (!WANT_J && A.rnorm) A.rnorm[o] = sqrt(r0 * r0 + r1 * r1);
    if (EXT) { r0 = dead ? 0.0 : r0 * wg; r1 = dead ? 0.0 : r1 * wg; }
    const double s = r0 * r0 + r1 * r1;
    double rho0 = s, rho1 = 1.0;
    const double b = A.huber_a * A.huber_a;
    const bool lossy = A.use_loss && !(EXT && A.obs_flags && (A.obs_flags[o] & 1));   // GCP blocks carry no loss (:424)
    if (lossy && s > b) { const double rr = sqrt(s); rho0 = 2.0 * A.huber_a * rr - b; rho1 = fmax(DBL_MIN, A.huber_a / rr); }
    cost += 0.5 * rho0;
    if (WANT_J) {
      const double wl = sqrt(rho1);                             // Huber: rho'' <= 0 => r, J scaled by sqrt(rho')
      const double w = EXT ? wl * wg : wl;                      // Jacobian of the weighted residual
      const long long n = A.n_obs;
      __stcs(A.r + o, wl * r0); __stcs(A.r + n + o, wl * r1);
      // d r / d u = f * dd ; d u / d p = [[iz,0,-x iz],[0,iz,-y iz]]
      const double a00 = w * f * dd[0], a01 = w * f * dd[1], a10 = w * f * dd[2], a11 = w * f * dd[3];
      double g[6];                                              // d r / d p (2x3)
      g[0] = a00 * iz; g[1] = a01 * iz; g[2] = -(a00 * x + a01 * y) * iz;
      g[3] = a10 * iz; g[4] = a11 * iz; g[5] = -(a10 * x + a11 * y) * iz;
      if (spherical) {
        #pragma unroll
        for (int i = 0; i < 6; ++i) g[i] = w * gs[i];
      }
      // point block: g * R
      #pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double sc = (A.pts_free && !(EXT && A.pt_fixed && A.pt_fixed[j])) ? (A.sc_pt ? A.sc_pt[3 * j + c] : 1.0) : 0.0;
        __stcs(A.Jp + (0 * 3 + c) * n + o, sc * (g[0] * R[c] + g[1] * R[3 + c] + g[2] * R[6 + c]));
        __stcs(A.Jp + (1 * 3 + c) * n + o, sc * (g[3] * R[c] + g[4] * R[3 + c] + g[5] * R[6 + c]));
      }
      // pose block: rotation columns g * (dR_k X), translation columns g
      #pragma unroll
      for (int k = 0; k < 3; ++k) {
        // dR_k X = R (j_k x X), j_k = column k of Jr
        const double j0 = R[9 + k], j1 = R[12 + k], j2 = R[15 + k];
        const double v0 = j1 * X2 - j2 * X1, v1 = j2 * X0 - j0 * X2, v2 = j0 * X1 - j1 * X0;
        const double q0 = R[0] * v0 + R[1] * v1 + R[2] * v2;
        const double q1 = R[3] * v0 + R[4] * v1 + R[5] * v2;
        const double q2 = R[6] * v0 + R[7] * v1 + R[8] * v2;
        const double sc = ((A.pose_mask >> k) & 1) ? (A.sc_cam ? A.sc_cam[6 * ip + k] : 1.0) : 0.0;
        __stcs(A.Jc + (0 * 6 + k) * n + o, sc * (g[0] * q0 + g[1] * q1 + g[2] * q2));
        __stcs(A.Jc + (1 * 6 + k) * n + o, sc * (g[3] * q0 + g[4] * q1 + g[5] * q2));
        const double st = ((A.pose_mask >> (3 + k)) & 1) ? (A.sc_cam ? A.sc_cam[6 * ip + 3 + k] : 1.0) : 0.0;
        __stcs(A.Jc + (0 * 6 + 3 + k) * n + o, st * g[k]);
        __stcs(A.Jc + (1 * 6 + 3 + k) * n + o, st * g[3 + k]);
      }
      // intrinsic block: [f, ppx, ppy, K3..K7]
      const unsigned im = A.intr_mask[iq];
      double ji0[KI], ji1[KI];
      ji0[0] = w * dx; ji1[0] = w * dy; ji0[1] = spherical ? 0.0 : w; ji1[1] = 0.0; ji0[2] = 0.0; ji1[2] = spherical ? 0.0 : w;
      #pragma unroll
      for (int k = 0; k < 5; ++k) { ji0[3 + k] = w * f * dk[k]; ji1[3 + k] = w * f * dk[5 + k]; }
      #pragma unroll
      for (int k = 0; k < KI; ++k) {
        const double sc = ((im >> k) & 1) ? (A.sc_intr ? A.sc_intr[KI * iq + k] : 1.0) : 0.0;
        if (k < A.kiu) { __stcs(A.Ji + (0 * KI + k) * n + o, sc * ji0[k]); __stcs(A.Ji + (1 * KI + k) * n + o, sc * ji1[k]); }
      }
    }
    o = o_next; ip = ipn; iq = iqn; j = jn; xy = xyn;
  }
  const double t = block_sum<EVAL_THREADS>(cost, sh);
  if (threadIdx.x == 0) A.cost_partial[blockIdx.x] = t;
}

// ------------------------------------------------------------------------------ pose-centre priors
// PoseCenterConstraintCostFunction (sfm_data_BA_ceres.cpp:44-80), added with HuberLoss(a = fit^2) at :455-472:
// r = w .* (C - c0), C = -R' t.  A few hundred rows touching one pose block each: one block does them all.
struct PriorArgs {
  const double *poses, *camR, *camdR; const int *prior_pose; const double *center, *weight; int n; double huber_a;
  const double *sc_cam; unsigned pose_mask;
  double *rP, *JP;            // corrected residuals [n][3], Jacobians [n][3][6] (scaled, masked)
  double *cost_out;           // one partial
};
constexpr int PRIOR_THREADS = 128;
template <bool WANT_J>
__global__ void __launch_bounds__(PRIOR_THREADS) prior_eval_kernel(PriorArgs A) {
  __shared__ double sh[PRIOR_THREADS / 32];
  double cost = 0.0;
  for (int k = threadIdx.x; k < A.n; k += PRIOR_THREADS) {
    const int p = A.prior_pose[k];
    const double *R = A.camR + 9 * p, *t = A.poses + 6 * p + 3, *w = A.weight + 3 * k, *c0 = A.center + 3 * k;
    double r[3];
    #pragma unroll
    for (int i = 0; i < 3; ++i) r[i] = w[i] * (-(R[i] * t[0] + R[3 + i] * t[1] + R[6 + i] * t[2]) - c0[i]);
    const double s = r[0] * r[0] + r[1] * r[1] + r[2] * r[2], b = A.huber_a * A.huber_a;
    double rho0 = s, rho1 = 1.0;
    if (s > b) { const double rr = sqrt(s); rho0 = 2.0 * A.huber_a * rr - b; rho1 = fmax(DBL_MIN, A.huber_a / rr); }
    cost += 0.5 * rho0;
    if (WANT_J) {
      const double wl = sqrt(rho1);
      const double *dR = A.camdR + 27 * p;
      #pragma unroll
      for (int i = 0; i < 3; ++i) {
        A.rP[3 * k + i] = wl * r[i];
        #pragma unroll
        for (int c = 0; c < 6; ++c) {
          const double d = c < 3 ? -(dR[9 * c + i] * t[0] + dR[9 * c + 3 + i] * t[1] + dR[9 * c + 6 + i] * t[2]) : -R[3 * (c - 3) + i];
          const double sc = ((A.pose_mask >> c) & 1) ? (A.sc_cam ? A.sc_cam[6 * p + c] : 1.0) : 0.0;
          A.JP[18 * k + 6 * i + c] = sc * wl * w[i] * d;
        }
      }
    }
  }
  const double tsum = block_sum<PRIOR_THREADS>(cost, sh);
  if (threadIdx.x == 0) A.cost_out[0] = tsum;
}
// iteration 0: the Jacobi scale is known only after the unscaled column norms
__global__ void prior_scale_kernel(double *__restrict__ JP, const int *__restrict__ prior_pose, const double *__restrict__ sc_cam, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 18 * n) JP[i] *= sc_cam[6 * prior_pose[i / 18] + i % 6];
}
// adds the prior rows to the pose-diagonal blocks, column norms and gradient (run after cam_colsum_kernel)
__global__ void prior_accum_kernel(const double *__restrict__ JP, const double *__restrict__ rP, const int *__restrict__ prior_pose, int n,
                                   double *__restrict__ diag_cam, double *__restrict__ g_cam, double *__restrict__ FtF) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int p = prior_pose[k]; const double *J = JP + 18 * k, *r = rP + 3 * k;
  for (int a = 0; a < 6; ++a) {
    atomicAdd(g_cam + 6 * p + a, J[a] * r[0] + J[6 + a] * r[1] + J[12 + a] * r[2]);
    for (int b = 0; b < 6; ++b) {
      const double v = J[a] * J[b] + J[6 + a] * J[6 + b] + J[12 + a] * J[12 + b];
      atomicAdd(FtF + 36 * (size_t)p + a * 6 + b, v);
      if (a == b) atomicAdd(diag_cam + 6 * p + a, v);
    }
  }
}
// model-cost partial of the prior rows
__global__ void __launch_bounds__(PRIOR_THREADS) prior_model_kernel(const double *__restrict__ JP, const double *__restrict__ rP, const int *__restrict__ prior_pose, int n,
                                                                     const double *__restrict__ step_red, double *__restrict__ out) {
  __shared__ double sh[PRIOR_THREADS / 32];
  double v = 0.0;
  for (int k = threadIdx.x; k < n; k += PRIOR_THREADS) {
    const double *st = step_red + 6 * prior_pose[k];
    for (int i = 0; i < 3; ++i) { double m = 0; for (int c = 0; c < 6; ++c) m += JP[18 * k + 6 * i + c] * st[c]; v += -m * (rP[3 * k + i] + m / 2.0); }
  }
  const double t = block_sum<PRIOR_THREADS>(v, sh);
  if (threadIdx.x == 0) out[0] = t;
}

// fixed-order final reduction of per-block partials -> out[0]
__global__ void reduce_partials_kernel(const double *__restrict__ part, int n, double *__restrict__ out) {
  __shared__ double sh[32];
  double v = 0; for (int i = threadIdx.x; i < n; i += 1024) v += part[i];
  const double t = block_sum<1024>(v, sh);
  if (threadIdx.x == 0) out[0] = t;
}

// ------------------------------------------------------------------------------ column sums
// per point: EtE (6 unique: 00,10,11,20,21,22), Etb (3) and, for points whose observations all use one
// intrinsic group (pt_single), EtFi = sum_obs Jp' Ji (3 x KI) from the (scaled) blocks.
__global__ void point_accum_kernel(const double *__restrict__ Jp, const double *__restrict__ Ji, const double *__restrict__ r, const int *__restrict__ pt_start,
                                   const unsigned char *__restrict__ pt_single, int n_points, long long n, int kiu, double *__restrict__ EtE, double *__restrict__ Etb,
                                   double *__restrict__ EtFi, double *__restrict__ diag_pt) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_points) return;
  double e00 = 0, e10 = 0, e11 = 0, e20 = 0, e21 = 0, e22 = 0, b0 = 0, b1 = 0, b2 = 0;
  double fi[3 * KI];
  #pragma unroll
  for (int k = 0; k < 3 * KI; ++k) fi[k] = 0.0;
  const bool single = pt_single[j] != 0;
  for (long long o = pt_start[j]; o < pt_start[j + 1]; ++o) {
    #pragma unroll
    for (int row = 0; row < 2; ++row) {
      const double a = Jp[(row * 3 + 0) * n + o], b = Jp[(row * 3 + 1) * n + o], c = Jp[(row * 3 + 2) * n + o], rr = r[row * n + o];
      e00 += a * a; e10 += b * a; e11 += b * b; e20 += c * a; e21 += c * b; e22 += c * c;
      b0 += a * rr; b1 += b * rr; b2 += c * rr;
      if (single) {
        #pragma unroll
        for (int k = 0; k < KI; ++k) { const double v = k < kiu ? Ji[(row * KI + k) * n + o] : 0.0; fi[k] += a * v; fi[KI + k] += b * v; fi[2 * KI + k] += c * v; }
      }
    }
  }
  double *E = EtE + 6 * (size_t)j; E[0] = e00; E[1] = e10; E[2] = e11; E[3] = e20; E[4] = e21; E[5] = e22;
  diag_pt[3 * (size_t)j] = e00; diag_pt[3 * (size_t)j + 1] = e11; diag_pt[3 * (size_t)j + 2] = e22;       // squared column norms
  Etb[3 * (size_t)j] = b0; Etb[3 * (size_t)j + 1] = b1; Etb[3 * (size_t)j + 2] = b2;
  #pragma unroll
  for (int k = 0; k < 3 * KI; ++k) EtFi[(size_t)j * 3 * KI + k] = fi[k];
}

// per pose (one CTA of CCS_THREADS): Fc'Fc (6x6, full), squared column norms (its diagonal) and gradient Fc'r over the
// pose's observation list — fixed order (lane, then warp), no atomics.  One warp per pose left 7 warps per SM at 1000
// poses and a 16-deep chain of dependent gathers: 82 us at 1000 cameras, 43 us at 10.
constexpr int CCS_THREADS = 128;
__global__ void __launch_bounds__(CCS_THREADS) cam_colsum_kernel(const double *__restrict__ Jc, const double *__restrict__ r, const int *__restrict__ cam_start,
                                  const int *__restrict__ cam_obs, int n_poses, long long n, double *__restrict__ diag_cam,
                                  double *__restrict__ g_cam, double *__restrict__ FtF) {
  __shared__ double sh[CCS_THREADS / 32][27];
  const int p = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (p >= n_poses) return;
  double m[21], g[6] = {0, 0, 0, 0, 0, 0};
  #pragma unroll
  for (int k = 0; k < 21; ++k) m[k] = 0.0;
  for (int t = cam_start[p] + threadIdx.x; t < cam_start[p + 1]; t += CCS_THREADS) {
    const long long o = cam_obs[t];
    const double r0 = r[o], r1 = r[n + o];
    double a[6], b[6];
    #pragma unroll
    for (int k = 0; k < 6; ++k) { a[k] = Jc[k * n + o]; b[k] = Jc[(6 + k) * n + o]; g[k] += a[k] * r0 + b[k] * r1; }
    int q = 0;
    #pragma unroll
    for (int i = 0; i < 6; ++i)
      #pragma unroll
      for (int k = 0; k <= i; ++k) m[q++] += a[i] * a[k] + b[i] * b[k];
  }
  #pragma unroll
  for (int k = 0; k < 21; ++k) { for (int o = 16; o > 0; o >>= 1) m[k] += __shfl_down_sync(0xffffffffu, m[k], o); }
  #pragma unroll
  for (int k = 0; k < 6; ++k) { for (int o = 16; o > 0; o >>= 1) g[k] += __shfl_down_sync(0xffffffffu, g[k], o); }
  if (lane == 0) {
    #pragma unroll
    for (int k = 0; k < 21; ++k) sh[warp][k] = m[k];
    #pragma unroll
    for (int k = 0; k < 6; ++k) sh[warp][21 + k] = g[k];
  }
  __syncthreads();
  if (threadIdx.x < 27) {
    double v = 0.0;
    #pragma unroll
    for (int w = 0; w < CCS_THREADS / 32; ++w) v += sh[w][threadIdx.x];
    sh[0][threadIdx.x] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int q = 0;
    for (int i = 0; i < 6; ++i) for (int k = 0; k <= i; ++k) { FtF[36 * (size_t)p + i * 6 + k] = sh[0][q]; FtF[36 * (size_t)p + k * 6 + i] = sh[0][q]; ++q; }
    for (int k = 0; k < 6; ++k) { diag_cam[6 * p + k] = FtF[36 * (size_t)p + k * 6 + k]; g_cam[6 * p + k] = sh[0][21 + k]; }
  }
}

// per intrinsic group: Fi'Fi (KI x KI, full), its diagonal and the gradient Fi'r, reduced in fixed order
// (chunks x blocks, then a final pass): part[q][chunk][80] = {64 FiFi, 8 g, 8 unused}
constexpr int ICS_THREADS = 256;
constexpr int ICS_W = 80;
// KIU = number of intrinsic columns in use (3 pinhole .. 8 Brown): only those products are formed, which keeps the
// kernel at a few dozen registers (the generic 8-column version needed 166 and ran one CTA per SM: 105 us)
template <int KIU>
__global__ void __launch_bounds__(ICS_THREADS) intr_colsum_kernel(const double *__restrict__ Ji, const double *__restrict__ r, const int *__restrict__ obs_intr,
                                   long long n, int chunks, double *__restrict__ part) {
  __shared__ double sh[ICS_THREADS / 32];
  const int q = blockIdx.y, chunk = blockIdx.x;
  constexpr int NM = KIU * (KIU + 1) / 2;
  double m[NM], g[KIU];
  #pragma unroll
  for (int k = 0; k < NM; ++k) m[k] = 0;
  #pragma unroll
  for (int k = 0; k < KIU; ++k) g[k] = 0;
  const long long per = (n + chunks - 1) / chunks, lo = per * chunk, hi = lo + per < n ? lo + per : n;
  for (long long o = lo + threadIdx.x; o < hi; o += ICS_THREADS) {
    const bool mine = __ldcs(obs_intr + o) == q;
    const double r0 = __ldcs(r + o), r1 = __ldcs(r + n + o);
    double a[KIU], b[KIU];
    #pragma unroll
    for (int k = 0; k < KIU; ++k) { a[k] = __ldcs(Ji + k * n + o); b[k] = __ldcs(Ji + (KI + k) * n + o); }
    if (!mine) continue;
    #pragma unroll
    for (int k = 0; k < KIU; ++k) g[k] += a[k] * r0 + b[k] * r1;
    int t = 0;
    #pragma unroll
    for (int i = 0; i < KIU; ++i)
      #pragma unroll
      for (int k = 0; k <= i; ++k) m[t++] += a[i] * a[k] + b[i] * b[k];
  }
  double *dst = part + ((size_t)q * chunks + chunk) * ICS_W;
  for (int e = threadIdx.x; e < ICS_W; e += ICS_THREADS) dst[e] = 0.0;
  __syncthreads();
  int t = 0;
  #pragma unroll
  for (int i = 0; i < KIU; ++i)
    #pragma unroll
    for (int k = 0; k <= i; ++k) {
      const double v = block_sum<ICS_THREADS>(m[t++], sh);
      if (threadIdx.x == 0) { dst[i * KI + k] = v; dst[k * KI + i] = v; }
    }
  #pragma unroll
  for (int k = 0; k < KIU; ++k) { const double v = block_sum<ICS_THREADS>(g[k], sh); if (threadIdx.x == 0) dst[64 + k] = v; }
}
// one CTA per (intrinsic group, element): strided partial sums over the chunks, then a fixed-order block reduction
__global__ void __launch_bounds__(128) intr_colsum_final_kernel(const double *__restrict__ part, int chunks, int n_intr, double *__restrict__ diag_intr, double *__restrict__ g_intr,
                                         double *__restrict__ FiFi) {
  __shared__ double sh[4];
  const int q = blockIdx.x / 72, e = blockIdx.x % 72;
  double v = 0;
  for (int c = threadIdx.x; c < chunks; c += 128) v += part[((size_t)q * chunks + c) * ICS_W + e];
  v = block_sum<128>(v, sh);
  if (threadIdx.x != 0) return;
  if (e < 64) { FiFi[(size_t)q * 64 + e] = v; if (e / KI == e % KI) diag_intr[q * KI + e / KI] = v; }
  else g_intr[q * KI + (e - 64)] = v;
}
__global__ void make_scale_kernel(const double *__restrict__ n2, int n, double *__restrict__ scale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) scale[i] = 1.0 / (1.0 + sqrt(n2[i]));
}
// apply the just-computed column scaling to the unscaled J of iteration 0 (ScaleColumns, :253)
__global__ void scale_J_kernel(double *__restrict__ Jp, double *__restrict__ Jc, double *__restrict__ Ji, const int *__restrict__ obs_pose,
                               const int *__restrict__ obs_intr, const int *__restrict__ obs_pt, long long n, int kiu,
                               const double *__restrict__ sc_pt, const double *__restrict__ sc_cam, const double *__restrict__ sc_intr) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (o >= n) return;
  const int ip = obs_pose[o], iq = obs_intr[o], j = obs_pt[o];
  for (int row = 0; row < 2; ++row) {
    for (int c = 0; c < 3; ++c) Jp[(row * 3 + c) * n + o] *= sc_pt[3 * j + c];
    for (int c = 0; c < 6; ++c) Jc[(row * 6 + c) * n + o] *= sc_cam[6 * ip + c];
    for (int c = 0; c < kiu; ++c) Ji[(row * KI + c) * n + o] *= sc_intr[KI * iq + c];
  }
}
// g_unscaled = g_scaled / scale ; then max |g| over free columns (gradient_max_norm)


// ------------------------------------------------------------------------------ reduced system
// Camera-pair structure: bitmap[nc][words] (bit b of row a set <=> S block (a,b) exists),
// wprefix[nc][words] = #bits of the row before that word, rowptr[nc+1].
struct Bsr { const unsigned *bitmap; const int *wprefix; const int *rowptr; int words; };
__device__ __forceinline__ int bsr_find(const Bsr &B, int a, int b) {
  const size_t w = (size_t)a * B.words + (b >> 5);
  return B.rowptr[a] + B.wprefix[w] + __popc(B.bitmap[w] & ((1u << (b & 31)) - 1u));
}
__global__ void bitmap_mark_kernel(const int *__restrict__ obs_pose, const int *__restrict__ obs_pt, const int *__restrict__ pt_start,
                                   long long n, unsigned *__restrict__ bitmap, int words) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (o >= n) return;
  const int a = obs_pose[o], j = obs_pt[o];
  for (long long u = pt_start[j]; u < pt_start[j + 1]; ++u) { const int b = obs_pose[u]; atomicOr(&bitmap[(size_t)a * words + (b >> 5)], 1u << (b & 31)); }
}
__global__ void bitmap_rowcount_kernel(const unsigned *__restrict__ bitmap, int nc, int words, int *__restrict__ wprefix, int *__restrict__ rowcount) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x; if (a >= nc) return;
  int c = 0; for (int w = 0; w < words; ++w) { wprefix[(size_t)a * words + w] = c; c += __popc(bitmap[(size_t)a * words + w]); }
  rowcount[a] = c;
}
__global__ void bitmap_cols_kernel(const unsigned *__restrict__ bitmap, const int *__restrict__ rowptr, int nc, int words, int *__restrict__ cols) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x; if (a >= nc) return;
  int k = rowptr[a];
  for (int w = 0; w < words; ++w) { unsigned m = bitmap[(size_t)a * words + w]; while (m) { const int b = __ffs(m) - 1; m &= m - 1; cols[k++] = w * 32 + b; } }
}

struct SchurArgs {
  const double *r, *Jp, *Jc, *Ji, *EtE, *Etb, *EtFi, *lmD_pt;
  const int *obs_pose, *obs_intr, *obs_pt, *pt_start; const unsigned char *pt_single;
  const double *FtF, *FiFi, *g_cam, *g_intr;
  long long n; int n_poses, n_intr, pts_free, kiu;
  int skip_fast;   // schur_kernel: leave the landmarks the split Schur step handles (pt_single and <= 32 observations) alone
  Bsr bsr;
  double *Scc;      // [nnzb][36]
  double *Sci;      // [KI*n_intr][6*n_poses]
  double *Sii;      // [KI*n_intr][KI*n_intr]
  double *rhs;      // [6*n_poses + KI*n_intr]
  double *Einv;     // [n_points][9]  (written by the thread of the point's first observation)
  int *fail;
};

// Radius-independent part of the reduced system, computed once per Jacobian evaluation without atomics
// (cam_colsum / intr_colsum): Scc(p,p) = Fc'Fc, Sii(q,q) = Fi'Fi, rhs = [Fc'r ; Fi'r].  S must be zeroed first.
// With the points eliminated schur_gather_kernel writes all of Scc, Fc'Fc included, and Scc is left alone here.
__global__ void s_init_kernel(SchurArgs A) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int nc36 = 36 * A.n_poses, ni64 = 64 * A.n_intr, nred = 6 * A.n_poses + KI * A.n_intr;
  if (i < nc36 && !A.pts_free) { const int p = i / 36; A.Scc[36 * (size_t)bsr_find(A.bsr, p, p) + i % 36] = A.FtF[i]; }
  if (i < ni64) { const int q = i / 64, e = i % 64; A.Sii[(size_t)(KI * q + e / KI) * (KI * A.n_intr) + KI * q + e % KI] = A.FiFi[i]; }
  if (i < nred) A.rhs[i] = i < 6 * A.n_poses ? A.g_cam[i] : A.g_intr[i - 6 * A.n_poses];
}

// One thread per observation t.  Adds the point-elimination terms  -(E'F)' (E'E + D^2)^-1 (E'F)  and the
// same-observation border term Fi'Fc.  Camera-pair blocks are visited for cam(u) >= cam(t) and the term goes to both
// (cam(t), cam(u)) and its transpose: it adds to what schur_gather_kernel wrote, which is both triangles.  Everything
// hot (the intrinsics corner, its right-hand side) is reduced per point first so that no address sees more than ~one
// atomic per point.
constexpr int SCHUR_THREADS = 128;
__global__ void __launch_bounds__(SCHUR_THREADS) schur_kernel(SchurArgs A) {
  __shared__ double s_ii[KI * KI + KI];
  __shared__ int s_q0;
  const long long t = (long long)blockIdx.x * SCHUR_THREADS + threadIdx.x;
  const long long n = A.n;
  if (threadIdx.x < KI * KI + KI) s_ii[threadIdx.x] = 0.0;
  if (threadIdx.x == 0) s_q0 = A.obs_intr[(long long)blockIdx.x * SCHUR_THREADS];
  __syncthreads();
  const int q0 = s_q0;
  const int nred_c = 6 * A.n_poses, ni8 = KI * A.n_intr;
  bool mine = t < n;
  if (mine && A.skip_fast && A.pts_free) { const int j = A.obs_pt[t]; mine = !(A.pt_single[j] != 0 && A.pt_start[j + 1] - A.pt_start[j] <= 32); }
  if (mine) {
    const int j = A.obs_pt[t], ct = A.obs_pose[t], qt = A.obs_intr[t];
    double jc[12], ji[2 * KI], jp[6];
    #pragma unroll
    for (int k = 0; k < 12; ++k) jc[k] = A.Jc[k * n + t];
    #pragma unroll
    for (int k = 0; k < 2 * KI; ++k) ji[k] = (k % KI) < A.kiu ? A.Ji[k * n + t] : 0.0;
    #pragma unroll
    for (int k = 0; k < 6; ++k) jp[k] = A.Jp[k * n + t];
    double *sci_row0 = A.Sci + (size_t)(KI * qt) * nred_c + 6 * ct;
    if (!A.pts_free) {
      #pragma unroll
      for (int a = 0; a < KI; ++a) {
        if (ji[a] == 0.0 && ji[KI + a] == 0.0) continue;
        #pragma unroll
        for (int b = 0; b < 6; ++b) atomicAdd(&sci_row0[(size_t)a * nred_c + b], ji[a] * jc[b] + ji[KI + a] * jc[6 + b]);
      }
    } else {
      double inv[9], ie[3], m[6];
      const double *E = A.EtE + 6 * (size_t)j;
      const double d0 = A.lmD_pt[3 * j], d1 = A.lmD_pt[3 * j + 1], d2 = A.lmD_pt[3 * j + 2];
      m[0] = E[0] + d0 * d0; m[1] = E[1]; m[2] = E[2] + d1 * d1; m[3] = E[3]; m[4] = E[4]; m[5] = E[5] + d2 * d2;
      const bool ok = inv3_spd(m, inv);
      if (!ok) atomicExch(A.fail, 1);
      const double *eb = A.Etb + 3 * (size_t)j;
      #pragma unroll
      for (int a = 0; a < 3; ++a) ie[a] = inv[a * 3] * eb[0] + inv[a * 3 + 1] * eb[1] + inv[a * 3 + 2] * eb[2];
      const bool first = t == A.pt_start[j];
      if (first) { for (int a = 0; a < 9; ++a) A.Einv[9 * (size_t)j + a] = inv[a]; }
      double efc[18];                                          // E'Fc of this observation (3x6)
      #pragma unroll
      for (int a = 0; a < 3; ++a)
        #pragma unroll
        for (int c = 0; c < 6; ++c) efc[a * 6 + c] = jp[a] * jc[c] + jp[3 + a] * jc[6 + c];
      // rhs_c -= (E'Fc)' (Einv E'b)
      #pragma unroll
      for (int c = 0; c < 6; ++c) atomicAdd(&A.rhs[6 * ct + c], -(efc[c] * ie[0] + efc[6 + c] * ie[1] + efc[12 + c] * ie[2]));
      const bool single = A.pt_single[j] != 0;
      if (single) {
        // border with the point-summed E'Fi:  Sci(qt; ct) += Fi'Fc - (Einv E'Fi_pt)' E'Fc
        const double *fi = A.EtFi + (size_t)j * 3 * KI;
        #pragma unroll
        for (int a = 0; a < KI; ++a) {
          const double f0 = fi[a], f1 = fi[KI + a], f2 = fi[2 * KI + a];
          if (f0 == 0.0 && f1 == 0.0 && f2 == 0.0 && ji[a] == 0.0 && ji[KI + a] == 0.0) continue;   // constant parameter
          const double g0 = inv[0] * f0 + inv[1] * f1 + inv[2] * f2, g1 = inv[3] * f0 + inv[4] * f1 + inv[5] * f2, g2 = inv[6] * f0 + inv[7] * f1 + inv[8] * f2;
          #pragma unroll
          for (int b = 0; b < 6; ++b)
            atomicAdd(&sci_row0[(size_t)a * nred_c + b], ji[a] * jc[b] + ji[KI + a] * jc[6 + b] - (g0 * efc[b] + g1 * efc[6 + b] + g2 * efc[12 + b]));
          if (first) {                                          // once per point: corner and its right-hand side
            const double rv = -(f0 * ie[0] + f1 * ie[1] + f2 * ie[2]);
            if (qt == q0) atomicAdd(&s_ii[KI * KI + a], rv); else atomicAdd(&A.rhs[nred_c + KI * qt + a], rv);
            #pragma unroll
            for (int b = 0; b < KI; ++b) {
              const double v = -(g0 * fi[b] + g1 * fi[KI + b] + g2 * fi[2 * KI + b]);
              if (v == 0.0) continue;
              if (qt == q0) atomicAdd(&s_ii[a * KI + b], v); else atomicAdd(&A.Sii[(size_t)(KI * qt + a) * ni8 + KI * qt + b], v);
            }
          }
        }
      }
      double gt_c[18];                                         // Einv * E'Fc_t
      #pragma unroll
      for (int a = 0; a < 3; ++a)
        #pragma unroll
        for (int c = 0; c < 6; ++c) gt_c[a * 6 + c] = inv[a * 3] * efc[c] + inv[a * 3 + 1] * efc[6 + c] + inv[a * 3 + 2] * efc[12 + c];
      double gt_i[3 * KI];
      if (!single) {                                           // general (rare) path: per-observation-pair border terms
        #pragma unroll
        for (int a = 0; a < KI; ++a) {
          const double e0 = jp[0] * ji[a] + jp[3] * ji[KI + a], e1 = jp[1] * ji[a] + jp[4] * ji[KI + a], e2 = jp[2] * ji[a] + jp[5] * ji[KI + a];
          gt_i[a] = inv[0] * e0 + inv[1] * e1 + inv[2] * e2; gt_i[KI + a] = inv[3] * e0 + inv[4] * e1 + inv[5] * e2; gt_i[2 * KI + a] = inv[6] * e0 + inv[7] * e1 + inv[8] * e2;
          const double rv = -(e0 * ie[0] + e1 * ie[1] + e2 * ie[2]);
          if (rv != 0.0) atomicAdd(&A.rhs[nred_c + KI * qt + a], rv);
          if (ji[a] == 0.0 && ji[KI + a] == 0.0) continue;
          #pragma unroll
          for (int b = 0; b < 6; ++b) atomicAdd(&sci_row0[(size_t)a * nred_c + b], ji[a] * jc[b] + ji[KI + a] * jc[6 + b]);
        }
      }
      for (long long u = A.pt_start[j]; u < A.pt_start[j + 1]; ++u) {
        const int cu = A.obs_pose[u];
        if (cu < ct && single) continue;
        double up[6], uc[12], efu[18];
        #pragma unroll
        for (int k = 0; k < 6; ++k) up[k] = A.Jp[k * n + u];
        #pragma unroll
        for (int k = 0; k < 12; ++k) uc[k] = A.Jc[k * n + u];
        #pragma unroll
        for (int a = 0; a < 3; ++a)
          #pragma unroll
          for (int c = 0; c < 6; ++c) efu[a * 6 + c] = up[a] * uc[c] + up[3 + a] * uc[6 + c];
        if (cu >= ct) {                                        // Scc(ct, cu) -= (Einv E'Fc_t)' E'Fc_u, and Scc(cu, ct) its transpose
          double *blk = A.Scc + 36 * (size_t)bsr_find(A.bsr, ct, cu);
          double *blt = cu > ct ? A.Scc + 36 * (size_t)bsr_find(A.bsr, cu, ct) : nullptr;
          #pragma unroll
          for (int a = 0; a < 6; ++a)
            #pragma unroll
            for (int b = 0; b < 6; ++b) {
              const double v = -(gt_c[a] * efu[b] + gt_c[6 + a] * efu[6 + b] + gt_c[12 + a] * efu[12 + b]);
              atomicAdd(&blk[a * 6 + b], v);
              if (blt) atomicAdd(&blt[b * 6 + a], v);
            }
        }
        if (!single) {
          const int qu = A.obs_intr[u];
          #pragma unroll
          for (int a = 0; a < KI; ++a) {
            if (gt_i[a] == 0.0 && gt_i[KI + a] == 0.0 && gt_i[2 * KI + a] == 0.0) continue;
            #pragma unroll
            for (int b = 0; b < 6; ++b) atomicAdd(&A.Sci[(size_t)(KI * qt + a) * nred_c + 6 * cu + b], -(gt_i[a] * efu[b] + gt_i[KI + a] * efu[6 + b] + gt_i[2 * KI + a] * efu[12 + b]));
            #pragma unroll
            for (int b = 0; b < KI; ++b) {
              const double ui0 = b < A.kiu ? A.Ji[b * n + u] : 0.0, ui1 = b < A.kiu ? A.Ji[(KI + b) * n + u] : 0.0;
              const double e0 = up[0] * ui0 + up[3] * ui1, e1 = up[1] * ui0 + up[4] * ui1, e2 = up[2] * ui0 + up[5] * ui1;
              const double v = gt_i[a] * e0 + gt_i[KI + a] * e1 + gt_i[2 * KI + a] * e2;
              if (v != 0.0) atomicAdd(&A.Sii[(size_t)(KI * qt + a) * ni8 + KI * qu + b], -v);
            }
          }
        }
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < KI * KI + KI) {
    const double v = s_ii[threadIdx.x];
    if (v != 0.0) {
      if (threadIdx.x < KI * KI) atomicAdd(&A.Sii[(size_t)(KI * q0 + threadIdx.x / KI) * ni8 + KI * q0 + threadIdx.x % KI], v);
      else atomicAdd(&A.rhs[nred_c + KI * q0 + (threadIdx.x - KI * KI)], v);
    }
  }
}

constexpr int CORNER_REPS = 64;

// ---- Schur step for the common landmark (all its observations through one intrinsic group, at most 32 of them), in
// two kernels:
//   schur_stage_kernel  : thread per observation (coalesced component-major loads), per-observation border / rhs
//                         terms, writes GE[obs] = { Einv E'Fc (18), E'Fc (18) }  (288 B per observation)
//   schur_gather_kernel : warp per upper block of Scc, sums the block's terms from GE over the pair lists built at
//                         create and stores the block and its transpose once (no atomics, fixed order)
// KIU = intrinsic columns in use (3 pinhole .. 8 Brown): the generic 8-column body kept 16 Jacobian and 24 EtFi values
// live per thread (162 registers, 3 CTAs per SM, 17 % of the warps active, 5x off its DRAM time).  The 36 doubles of an
// observation's {E^-1 E'F, E'F} record go through shared memory so that a warp writes its 32 records (9 KB, contiguous)
// with full 256-byte stores instead of 36 scattered 8-byte stores per lane.
constexpr int GE_LD = 37;                            // padded record stride in shared memory (conflict-free for both phases)
template <int KIU>
__global__ void __launch_bounds__(SCHUR_THREADS, 5) schur_stage_kernel(SchurArgs A, double *__restrict__ GE, double *__restrict__ corner_rep) {
  // The intrinsics corner (and its rhs) of group q0 is hit once per landmark: accumulate into CORNER_REPS replicas
  // with native FP64 REDs (shared-memory double atomics are CAS loops: they cost 0.3 ms here) and fold them after.
  __shared__ double ge_s[SCHUR_THREADS / 32][32 * GE_LD];
  const long long t = (long long)blockIdx.x * SCHUR_THREADS + threadIdx.x;
  const long long n = A.n;
  const int nred_c = 6 * A.n_poses, ni8 = KI * A.n_intr;
  const int q0 = A.obs_intr[0];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double *s_ii = corner_rep + (size_t)(blockIdx.x % CORNER_REPS) * (KI * KI + KI);
  double *gs = ge_s[warp] + lane * GE_LD;
  bool mine = t < n;
  int j = 0;
  if (mine) { j = A.obs_pt[t]; const int K = A.pt_start[j + 1] - A.pt_start[j]; mine = A.pt_single[j] != 0 && K <= 32; }
  if (mine) {
    const int ct = A.obs_pose[t], qt = A.obs_intr[t];
    double inv[9], ie[3], m[6];
    { const double *E = A.EtE + 6 * (size_t)j;
      const double d0 = A.lmD_pt[3 * j], d1 = A.lmD_pt[3 * j + 1], d2 = A.lmD_pt[3 * j + 2];
      m[0] = E[0] + d0 * d0; m[1] = E[1]; m[2] = E[2] + d1 * d1; m[3] = E[3]; m[4] = E[4]; m[5] = E[5] + d2 * d2; }
    if (!inv3_spd(m, inv)) atomicExch(A.fail, 1);
    { const double *eb = A.Etb + 3 * (size_t)j;
      #pragma unroll
      for (int a = 0; a < 3; ++a) ie[a] = inv[a * 3] * eb[0] + inv[a * 3 + 1] * eb[1] + inv[a * 3 + 2] * eb[2]; }
    const bool first = t == A.pt_start[j];
    if (first) { for (int a = 0; a < 9; ++a) A.Einv[9 * (size_t)j + a] = inv[a]; }
    double jc[12], jp[6];
    #pragma unroll
    for (int k = 0; k < 12; ++k) jc[k] = A.Jc[k * n + t];
    #pragma unroll
    for (int k = 0; k < 6; ++k) jp[k] = A.Jp[k * n + t];
    // E'F (3 x 6) and E^-1 E'F: the record for the pair walk.  Staged in shared memory (written to GE below) and read
    // back from there by the border terms, so that the 18 + 18 values are not live in registers next to jc / inv.
    { double efc[18];
      #pragma unroll
      for (int a = 0; a < 3; ++a)
        #pragma unroll
        for (int c = 0; c < 6; ++c) efc[a * 6 + c] = jp[a] * jc[c] + jp[3 + a] * jc[6 + c];
      #pragma unroll
      for (int a = 0; a < 3; ++a)
        #pragma unroll
        for (int c = 0; c < 6; ++c) {
          gs[a * 6 + c] = inv[a * 3] * efc[c] + inv[a * 3 + 1] * efc[6 + c] + inv[a * 3 + 2] * efc[12 + c];
          gs[18 + a * 6 + c] = efc[a * 6 + c];
        } }
    __syncwarp(__activemask());
    const double *ef = gs + 18;
    #pragma unroll
    for (int c = 0; c < 6; ++c) atomicAdd(&A.rhs[6 * ct + c], -(ef[c] * ie[0] + ef[6 + c] * ie[1] + ef[12 + c] * ie[2]));
    double *sci_row0 = A.Sci + (size_t)(KI * qt) * nred_c + 6 * ct;
    const double *fi = A.EtFi + (size_t)j * 3 * KI;
    #pragma unroll
    for (int a = 0; a < KIU; ++a) {
      const double f0 = fi[a], f1 = fi[KI + a], f2 = fi[2 * KI + a];
      const double ji0 = A.Ji[a * n + t], ji1 = A.Ji[(KI + a) * n + t];
      if (f0 == 0.0 && f1 == 0.0 && f2 == 0.0 && ji0 == 0.0 && ji1 == 0.0) continue;   // constant parameter
      const double g0 = inv[0] * f0 + inv[1] * f1 + inv[2] * f2, g1 = inv[3] * f0 + inv[4] * f1 + inv[5] * f2, g2 = inv[6] * f0 + inv[7] * f1 + inv[8] * f2;
      #pragma unroll
      for (int b = 0; b < 6; ++b)
        atomicAdd(&sci_row0[(size_t)a * nred_c + b], ji0 * jc[b] + ji1 * jc[6 + b] - (g0 * ef[b] + g1 * ef[6 + b] + g2 * ef[12 + b]));
      if (first) {
        const double rv = -(f0 * ie[0] + f1 * ie[1] + f2 * ie[2]);
        if (qt == q0) atomicAdd(&s_ii[KI * KI + a], rv); else atomicAdd(&A.rhs[nred_c + KI * qt + a], rv);
        #pragma unroll
        for (int b = 0; b < KIU; ++b) {
          const double v = -(g0 * fi[b] + g1 * fi[KI + b] + g2 * fi[2 * KI + b]);
          if (v == 0.0) continue;
          if (qt == q0) atomicAdd(&s_ii[a * KI + b], v); else atomicAdd(&A.Sii[(size_t)(KI * qt + a) * ni8 + KI * qt + b], v);
        }
      }
    }
  } else {
    #pragma unroll
    for (int k = 0; k < 36; ++k) gs[k] = 0.0;         // (records of landmarks the general kernel handles are not read)
  }
  __syncwarp();
  // the warp's 32 records are contiguous in GE: 36 coalesced 256-byte stores
  { const long long t0 = (long long)blockIdx.x * SCHUR_THREADS + 32 * warp;
    const long long nrec = n - t0 < 32 ? n - t0 : 32;
    if (nrec > 0) {
      double *dst = GE + 36 * (size_t)t0;
      #pragma unroll 4
      for (int e = lane; e < 36 * (int)nrec; e += 32) dst[e] = ge_s[warp][(e / 36) * GE_LD + e % 36];
    } }
}
// folds the corner replicas of schur_stage_kernel into Sii / rhs of group q0 (fixed order)
__global__ void corner_fold_kernel(const double *__restrict__ corner_rep, const int *__restrict__ obs_intr, int n_poses, int n_intr, double *__restrict__ Sii, double *__restrict__ rhs) {
  const int e = threadIdx.x; if (e >= KI * KI + KI) return;
  const int q0 = obs_intr[0], ni8 = KI * n_intr;
  double v = 0; for (int rp2 = 0; rp2 < CORNER_REPS; ++rp2) v += corner_rep[(size_t)rp2 * (KI * KI + KI) + e];
  if (v == 0.0) return;
  if (e < KI * KI) atomicAdd(&Sii[(size_t)(KI * q0 + e / KI) * ni8 + KI * q0 + e % KI], v);
  else atomicAdd(&rhs[6 * n_poses + KI * q0 + (e - KI * KI)], v);
}
// ---- pair lists of schur_gather_kernel, built once per context (omvg_ba_create).  An entry is one term of the
// split Schur step: a landmark j the warp-per-landmark step takes (pt_single, 1..32 observations) and two of its
// observations t, u with cam(t) <= cam(u), t = u included.  Entries are grouped by the upper Scc block (cam(t), cam(u)),
// in the order of the work list (wpos), and kept in landmark order inside a group (stable radix sort).  Observation
// weights, fixed and removed landmarks do not change the lists: GE carries them.
__device__ __forceinline__ bool pair_fast(const int *__restrict__ pt_start, const unsigned char *__restrict__ pt_single, int j, int &t0, int &K) {
  t0 = pt_start[j]; K = pt_start[j + 1] - t0;
  return pt_single[j] != 0 && K >= 1 && K <= 32;
}
__global__ void pair_count_kernel(const int *__restrict__ pt_start, const unsigned char *__restrict__ pt_single, const int *__restrict__ obs_pose,
                                  int n_points, long long *__restrict__ count) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x; if (j > n_points) return;
  long long cnt = 0; int t0, K;
  if (j < n_points && pair_fast(pt_start, pt_single, j, t0, K))
    for (int t = 0; t < K; ++t) { const int ct = obs_pose[t0 + t]; for (int u = 0; u < K; ++u) cnt += obs_pose[t0 + u] >= ct; }
  count[j] = cnt;                                    // count[n_points] = 0: the exclusive scan then ends in the total
}
__global__ void pair_fill_kernel(const int *__restrict__ pt_start, const unsigned char *__restrict__ pt_single, const int *__restrict__ obs_pose,
                                 int n_points, const long long *__restrict__ offs, Bsr B, const int *__restrict__ wpos,
                                 int *__restrict__ key, unsigned long long *__restrict__ pair) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x; if (j >= n_points) return;
  int t0, K; if (!pair_fast(pt_start, pt_single, j, t0, K)) return;
  long long o = offs[j];
  for (int t = 0; t < K; ++t) {
    const int ct = obs_pose[t0 + t];
    for (int u = 0; u < K; ++u) {
      const int cu = obs_pose[t0 + u]; if (cu < ct) continue;
      key[o] = wpos[bsr_find(B, ct, cu)];
      pair[o] = ((unsigned long long)(unsigned)(t0 + u) << 32) | (unsigned)(t0 + t);   // int2 {t, u}
      ++o;
    }
  }
}

// Scc(a, b) for every upper block (a <= b) of the work list and its transpose:  Fc'Fc (a = b)  -  sum over the block's
// entries of (Einv E'Fc_t)' E'Fc_u, each entry read from the GE records of schur_stage_kernel.  One warp per block; lane l
// takes entries l, l + 32, ... and accumulates all 36 elements in registers (18 16-byte loads per entry per lane, against
// 12 8-byte loads per entry per WARP lane if lanes split the block's elements), then the 32 partial blocks are reduced by
// a fixed shuffle tree.  Every block is written, empty ones included, so Scc needs no zeroing; with no landmark on the
// per-observation path the result does not depend on scheduling.
constexpr int GATHER_THREADS = 128;
__global__ void __launch_bounds__(GATHER_THREADS) schur_gather_kernel(const double *__restrict__ GE, const int *__restrict__ gstart, const int2 *__restrict__ pairs,
                                                                      const int *__restrict__ gblk, const int *__restrict__ gblkT, int nwork,
                                                                      const int *__restrict__ brow, const double *__restrict__ FtF, double *__restrict__ Scc) {
  const int w = (int)(((long long)blockIdx.x * GATHER_THREADS + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (w >= nwork) return;                           // (whole warps: nwork is a warp count)
  double acc[36];
  #pragma unroll
  for (int i = 0; i < 36; ++i) acc[i] = 0.0;
  const int e1 = gstart[w + 1];
  for (int e = gstart[w] + lane; e < e1; e += 32) {
    const int2 pr = pairs[e];
    const double2 *g2 = reinterpret_cast<const double2 *>(GE + 36 * (size_t)pr.x);        // Einv E'Fc_t (3 x 6)
    const double2 *f2 = reinterpret_cast<const double2 *>(GE + 36 * (size_t)pr.y + 18);   // E'Fc_u (3 x 6)
    double g[18], f[18];
    #pragma unroll
    for (int k = 0; k < 9; ++k) { const double2 v = g2[k]; g[2 * k] = v.x; g[2 * k + 1] = v.y; }
    #pragma unroll
    for (int k = 0; k < 9; ++k) { const double2 v = f2[k]; f[2 * k] = v.x; f[2 * k + 1] = v.y; }
    #pragma unroll
    for (int a = 0; a < 3; ++a)
      #pragma unroll
      for (int r = 0; r < 6; ++r)
        #pragma unroll
        for (int c = 0; c < 6; ++c) acc[r * 6 + c] = fma(g[a * 6 + r], f[a * 6 + c], acc[r * 6 + c]);
  }
  // reduce-scatter over lane bits 4 and 3 (36 -> 18 -> 9 elements per lane), then a butterfly over bits 2..0: the 8
  // lanes of group q = lane >> 3 hold the block's elements 9q .. 9q + 8, summed over all 32 lanes
  double h[18], v[9];
  { const bool up = lane & 16;
    #pragma unroll
    for (int i = 0; i < 18; ++i) { const double keep = up ? acc[18 + i] : acc[i], send = up ? acc[i] : acc[18 + i]; h[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16); } }
  { const bool up = lane & 8;
    #pragma unroll
    for (int i = 0; i < 9; ++i) { const double keep = up ? h[9 + i] : h[i], send = up ? h[i] : h[9 + i]; v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8); } }
  #pragma unroll
  for (int m = 4; m >= 1; m >>= 1)
    #pragma unroll
    for (int i = 0; i < 9; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], m);
  const int s = lane & 7, q = lane >> 3;
  double x = v[0];
  #pragma unroll
  for (int i = 1; i < 8; ++i) if (s == i) x = v[i];
  const int eu = gblk[w], el = gblkT[w];
  const double *ftf = FtF + 36 * (size_t)brow[eu];
  auto put = [&](int idx, double sum) {
    if (eu == el) { Scc[36 * (size_t)eu + idx] = ftf[idx] - sum; return; }
    Scc[36 * (size_t)eu + idx] = -sum;
    Scc[36 * (size_t)el + (idx % 6) * 6 + idx / 6] = -sum;
  };
  put(9 * q + s, x);
  if (s == 0) put(9 * q + 8, v[8]);
}

// S diag += D^2 (free columns) / = 1 (masked columns); block-Jacobi preconditioner Minv_c = inv(diag block)
__global__ void finish_cam_kernel(double *__restrict__ Scc, Bsr B, const double *__restrict__ lmD_cam, unsigned pose_mask, int n_poses,
                                  double *__restrict__ Minv, int *__restrict__ fail, int need_inverse) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x; if (p >= n_poses) return;
  double *blk = Scc + 36 * (size_t)bsr_find(B, p, p);
  double M[36];
  for (int k = 0; k < 6; ++k) { if ((pose_mask >> k) & 1) blk[k * 6 + k] += lmD_cam[6 * p + k] * lmD_cam[6 * p + k]; else blk[k * 6 + k] = 1.0; }
  if (!need_inverse) return;                          // direct solve (dense_solve_kernel): no preconditioner
  for (int k = 0; k < 36; ++k) M[k] = blk[k];
  // Cholesky 6x6 in place (lower), then inverse via forward/back substitution of unit vectors
  for (int k = 0; k < 6; ++k) {
    double d = M[k * 6 + k]; for (int q = 0; q < k; ++q) d -= M[k * 6 + q] * M[k * 6 + q];
    if (!(d > 0.0) || !isfinite(d)) { atomicExch(fail, 2); return; }
    d = sqrt(d); M[k * 6 + k] = d;
    for (int i = k + 1; i < 6; ++i) { double s = M[i * 6 + k]; for (int q = 0; q < k; ++q) s -= M[i * 6 + q] * M[k * 6 + q]; M[i * 6 + k] = s / d; }
  }
  for (int c = 0; c < 6; ++c) {
    double b[6]; for (int i = 0; i < 6; ++i) b[i] = i == c ? 1.0 : 0.0;
    for (int i = 0; i < 6; ++i) { double s = b[i]; for (int q = 0; q < i; ++q) s -= M[i * 6 + q] * b[q]; b[i] = s / M[i * 6 + i]; }
    for (int i = 5; i >= 0; --i) { double s = b[i]; for (int q = i + 1; q < 6; ++q) s -= M[q * 6 + i] * b[q]; b[i] = s / M[i * 6 + i]; }
    for (int i = 0; i < 6; ++i) Minv[36 * (size_t)p + i * 6 + c] = b[i];
  }
}
// intrinsics corner: add D^2 / identity, dense Cholesky inverse by one thread block (ni*8 <= 256)
__global__ void finish_intr_kernel(double *__restrict__ Sii, const double *__restrict__ lmD_intr, const unsigned *__restrict__ intr_mask,
                                   int ni8, double *__restrict__ Minv_i, double *__restrict__ work, int *__restrict__ fail, int need_inverse) {
  // LM diagonal / identity rows: one thread per row (off-diagonal zeroing first, diagonals after the barrier)
  for (int i = threadIdx.x; i < ni8; i += blockDim.x) {
    const bool free_ = (intr_mask[i / KI] >> (i % KI)) & 1;
    if (!free_) for (int k = 0; k < ni8; ++k) { Sii[(size_t)i * ni8 + k] = 0.0; Sii[(size_t)k * ni8 + i] = 0.0; }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < ni8; i += blockDim.x) {
    const bool free_ = (intr_mask[i / KI] >> (i % KI)) & 1;
    if (free_) Sii[(size_t)i * ni8 + i] += lmD_intr[i] * lmD_intr[i]; else Sii[(size_t)i * ni8 + i] = 1.0;
  }
  __syncthreads();
  // the block-Jacobi preconditioner of the single-vector PCG (used when more than 32 intrinsic columns are free):
  // Minv_i[q] = inverse of the KI x KI diagonal block of group q (constant coordinates are identity rows), one thread each
  if (!need_inverse) return;
  const int n_intr = ni8 / KI;
  for (int q = threadIdx.x; q < n_intr; q += blockDim.x) {
    double M[KI * KI];
    for (int a = 0; a < KI; ++a) for (int b = 0; b < KI; ++b) M[a * KI + b] = Sii[(size_t)(KI * q + a) * ni8 + KI * q + b];
    bool ok = true;
    for (int k = 0; k < KI; ++k) {
      double d = M[k * KI + k]; for (int p = 0; p < k; ++p) d -= M[k * KI + p] * M[k * KI + p];
      if (!(d > 0.0) || !isfinite(d)) { ok = false; break; }
      d = sqrt(d); M[k * KI + k] = d;
      for (int i = k + 1; i < KI; ++i) { double t = M[i * KI + k]; for (int p = 0; p < k; ++p) t -= M[i * KI + p] * M[k * KI + p]; M[i * KI + k] = t / d; }
    }
    if (!ok) { atomicExch(fail, 3); continue; }
    for (int c = 0; c < KI; ++c) {
      double b[KI]; for (int i = 0; i < KI; ++i) b[i] = i == c ? 1.0 : 0.0;
      for (int i = 0; i < KI; ++i) { double t = b[i]; for (int p = 0; p < i; ++p) t -= M[i * KI + p] * b[p]; b[i] = t / M[i * KI + i]; }
      for (int i = KI - 1; i >= 0; --i) { double t = b[i]; for (int p = i + 1; p < KI; ++p) t -= M[p * KI + i] * b[p]; b[i] = t / M[i * KI + i]; }
      for (int i = 0; i < KI; ++i) Minv_i[(size_t)q * KI * KI + i * KI + c] = b[i];
    }
  }
  (void)work;
}


// ------------------------------------------------------------------------------ small reduced systems: direct solve
// Up to DENSE_MAX unknowns (37 cameras with one shared intrinsic group) the reduced system  [Scc Sci'; Sci Sii] z = rhs
// is solved exactly, as Ceres does (schur_complement_solver.cc: dense / sparse Cholesky), by ONE CTA: the lower triangle
// is assembled packed in shared memory, factored as L D L' (right-looking, columns kept unscaled so that a step needs
// one barrier and no square root) and solved by one warp with shuffles.  An iterative solve is pure latency at this
// size: the single-CTA PCG took 254 us per solve at 10 cameras and 420 us at 50, this takes a few tens of us.
// A non-positive pivot raises `fail` (the LM loop treats the step as invalid, like a failed Cholesky in Ceres).
constexpr int DENSE_MAX = 220;                      // (n (n + 1) / 2 + (3 + DENSE_NB) n) doubles <= 227 KB of shared memory
constexpr int DENSE_NB = 8;                         // panel width of the blocked factorisation
__global__ void __launch_bounds__(1024) dense_solve_kernel(const double *__restrict__ Scc, const int *__restrict__ rowptr, const int *__restrict__ cols,
                                                          const double *__restrict__ Sci, const double *__restrict__ Sii, const double *__restrict__ rhs,
                                                          int n_poses, int ni8, double *__restrict__ z, int *__restrict__ fail, double *__restrict__ out,
                                                          unsigned long long *__restrict__ tim) {
  extern __shared__ double dsm[];
  unsigned long long tlast = 0; if (tim && threadIdx.x == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tlast));
#define DENSE_LAP(k) do { if (tim && threadIdx.x == 0) { unsigned long long now_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now_)); tim[k] += now_ - tlast; tlast = now_; } } while (0)
  const int nc6 = 6 * n_poses, n = nc6 + ni8;
  double *L = dsm;                                   // packed lower triangle, row i at i (i + 1) / 2
  double *y = L + n * (n + 1) / 2;                   // right-hand side / solution
  double *invd = y + n;                              // 1 / d_k
  double *acc = invd + n;                            // backward substitution: sum_{k>i} c_ki x_k
  double *Lp = acc + n;                              // [n][DENSE_NB] multipliers l_ic = c_ic / d_c of the current panel
  __shared__ int bad;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  if (tid == 0) bad = 0;
  for (int i = tid; i < n * (n + 1) / 2; i += nt) L[i] = 0.0;
  for (int i = tid; i < n; i += nt) { y[i] = rhs[i]; acc[i] = 0.0; }
  for (int i = tid; i < n * DENSE_NB; i += nt) Lp[i] = 0.0;
  __syncthreads();
  // camera-camera blocks (both triangles are stored; take b <= a), one warp per block row
  for (int a = warp; a < n_poses; a += nwarps)
    for (int e = rowptr[a]; e < rowptr[a + 1]; ++e) {
      const int b = cols[e]; if (b > a) break;
      const double *blk = Scc + 36 * (size_t)e;
      for (int k = lane; k < 36; k += 32) { const int i = 6 * a + k / 6, j = 6 * b + k % 6; if (j <= i) L[i * (i + 1) / 2 + j] = blk[k]; }
    }
  for (int q = warp; q < ni8; q += nwarps) {
    double *row = L + (nc6 + q) * (nc6 + q + 1) / 2;
    for (int k = lane; k < nc6; k += 32) row[k] = Sci[(size_t)q * nc6 + k];
    for (int k = lane; k <= q; k += 32) row[nc6 + k] = Sii[(size_t)q * ni8 + k];
  }
  __syncthreads();
  DENSE_LAP(0);
  // L D L', right-looking, DENSE_NB columns per panel.  Column k of L keeps the UNSCALED c_ik = l_ik d_k, the diagonal d_k.
  // Panel: one barrier per column, a handful of elements per thread (the columns of the panel right of it, the multiplier
  // l_ic into Lp, the right-hand side: y is eliminated along with the columns).  Trailing matrix: ONE pass per panel,
  // L[i][j] -= sum_c Lp[i][c] c_jc with the eight c_jc of a column in registers — a rank-1 update per column moved
  // 24 bytes of shared memory per element and column and ran at the shared-memory bandwidth (291 us at n = 188).
  const int ty = warp, tx = lane;                    // requires 1024 threads
  bool ok = true;
  for (int k0 = 0; k0 < n && ok; k0 += DENSE_NB) {
    const int nb = n - k0 < DENSE_NB ? n - k0 : DENSE_NB;
    for (int c = 0; c < nb; ++c) {
      const int kc = k0 + c;
      const double dk = L[kc * (kc + 1) / 2 + kc];
      if (!(dk > 0.0) || !isfinite(dk)) { ok = false; break; }            // (uniform: every thread reads the same dk)
      const double inv = __drcp_rn(dk);
      if (tid == 0) invd[kc] = inv;
      const double yk = y[kc];
      const int nrows = n - kc - 1, ncols = nb - c;
      for (int p = tid; p < nrows * ncols; p += nt) {
        const int r = p / ncols, sl = c + p % ncols, i = kc + 1 + r;
        const double li = L[i * (i + 1) / 2 + kc] * inv;
        if (sl == c) { Lp[i * DENSE_NB + c] = li; y[i] -= li * yk; }
        else { const int j = k0 + sl; if (j <= i) L[i * (i + 1) / 2 + j] -= li * L[j * (j + 1) / 2 + kc]; }
      }
      __syncthreads();
    }
    const int t0 = k0 + nb;
    if (ok && t0 < n) {
      for (int j = t0 + ((tx - t0) & 31); j < n; j += 32) {
        double cj[DENSE_NB];
        #pragma unroll
        for (int c = 0; c < DENSE_NB; ++c) cj[c] = c < nb ? L[j * (j + 1) / 2 + k0 + c] : 0.0;
        for (int i = j + ((ty - j) & 31); i < n; i += 32) {
          const double *__restrict__ lp = Lp + i * DENSE_NB;
          double a = L[i * (i + 1) / 2 + j];
          #pragma unroll
          for (int c = 0; c < DENSE_NB; ++c) a -= lp[c] * cj[c];
          L[i * (i + 1) / 2 + j] = a;
        }
      }
      __syncthreads();
    }
  }
  if (!ok) { if (tid == 0) { atomicExch(fail, 4); out[0] = 0.0; out[1] = 0.0; out[2] = 0.0; } for (int i = tid; i < n; i += nt) z[i] = 0.0; return; }
  DENSE_LAP(1);
  // y now holds w = L^-1 b.  Backward: x_i = (w_i - sum_{k>i} c_ki x_k) / d_i, 32 unknowns at a time from the bottom: one
  // warp solves the 32 x 32 triangle (lane = unknown, one shuffle per step, row k of L is contiguous), then every thread
  // adds the block's contribution to the accumulators of the rows above it.
  for (int b1 = n; b1 > 0; b1 -= 32) {
    const int b0 = b1 > 32 ? b1 - 32 : 0, mrows = b1 - b0;
    if (warp == 0) {
      const int i = b0 + lane;
      const bool mine = lane < mrows;
      double a = mine ? acc[i] : 0.0; const double w = mine ? y[i] : 0.0, idv = mine ? invd[i] : 0.0;
      for (int kk = mrows - 1; kk >= 0; --kk) {
        const double xc = (w - a) * idv;                                   // final for lane kk at this step
        const double xk = __shfl_sync(0xffffffffu, xc, kk);
        if (lane == kk) y[i] = xk;
        if (lane < kk) a += L[(b0 + kk) * (b0 + kk + 1) / 2 + i] * xk;
      }
    }
    __syncthreads();
    if (tid < b0) {
      double a0 = 0.0, a1 = 0.0;
      int k = b0;
      for (; k + 1 < b1; k += 2) { a0 += L[k * (k + 1) / 2 + tid] * y[k]; a1 += L[(k + 1) * (k + 2) / 2 + tid] * y[k + 1]; }
      if (k < b1) a0 += L[k * (k + 1) / 2 + tid] * y[k];
      acc[tid] += a0 + a1;
    }
    __syncthreads();
  }
  DENSE_LAP(2);
  for (int i = tid; i < n; i += nt) z[i] = y[i];
  if (tid == 0) { out[0] = 0.0; out[1] = 0.0; out[2] = 0.0; }
#undef DENSE_LAP
  (void)bad;
}

// ------------------------------------------------------------------------------ PCG (cooperative)
// aggregates of the two-level preconditioner (see PCG v3 below)
struct Coarse { const int *agg_of, *agg_start, *agg_cams; int ng, nw, nco; };
struct PcgArgs {
  const double *Scc; const int *rowptr, *cols; const double *Sci, *Sii, *rhs, *Minv_c, *Minv_i;
  int n_poses, ni8;
  double *z, *res, *p, *w, *zeta;          // length nred = 6 n_poses + ni8
  double *part;                            // [3][gridDim.x] partial sums
  double tol; int max_iter;
  double *out;                             // [0]=iterations, [1]=final relative residual, [2]=|b|
  // optional two-level part of the preconditioner on the camera rows (the gauge modes leave the intrinsics alone, so
  // the coarse space of PCG v3 is the coarse space of the full system too): M^-1 = blockdiag^-1 + Wa (Wa' Scc Wa)^-1 Wa'
  const double *W; Coarse C; const double *Einv; double *Cv, *Yv;   // W == nullptr: block-Jacobi only
};

__device__ __forceinline__ double grid_sum(cg::grid_group &grid, double v, double *part, double *sh) {
  const double t = block_sum<256>(v, sh);
  if (threadIdx.x == 0) part[blockIdx.x] = t;
  grid.sync();
  double s = 0;
  for (int i = 0; i < (int)gridDim.x; ++i) s += part[i];     // same order in every thread: deterministic
  return s;
}

// y = S x for the rows owned by this block; returns this thread's partial of x'y (lane 0 of each warp holds it)
__device__ __forceinline__ double spmv_rows(const PcgArgs &A, const double *__restrict__ x, double *__restrict__ y) {
  const int lane = threadIdx.x & 31, warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const int nc6 = 6 * A.n_poses;
  double dot = 0;
  for (int a = warp; a < A.n_poses; a += nwarps) {
    double acc[6] = {0, 0, 0, 0, 0, 0};
    for (int e = A.rowptr[a] + lane; e < A.rowptr[a + 1]; e += 32) {
      const double *blk = A.Scc + 36 * (size_t)e; const double *xb = x + 6 * A.cols[e];
      #pragma unroll
      for (int i = 0; i < 6; ++i)
        #pragma unroll
        for (int k = 0; k < 6; ++k) acc[i] += blk[i * 6 + k] * xb[k];
    }
    // border: + Sci' x_i   (column block of camera a)
    for (int q = lane; q < A.ni8; q += 32) {
      const double xi = x[nc6 + q]; const double *row = A.Sci + (size_t)q * nc6 + 6 * a;
      #pragma unroll
      for (int i = 0; i < 6; ++i) acc[i] += row[i] * xi;
    }
    #pragma unroll
    for (int i = 0; i < 6; ++i) { for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_down_sync(0xffffffffu, acc[i], o); }
    if (lane == 0) { for (int i = 0; i < 6; ++i) { y[6 * a + i] = acc[i]; dot += acc[i] * x[6 * a + i]; } }
  }
  // intrinsic rows: y_i = Sci x_c + Sii x_i   (one warp per row)
  for (int q = warp; q < A.ni8; q += nwarps) {
    double acc = 0;
    const double *row = A.Sci + (size_t)q * nc6;
    for (int k = lane; k < nc6; k += 32) acc += row[k] * x[k];
    for (int k = lane; k < A.ni8; k += 32) acc += A.Sii[(size_t)q * A.ni8 + k] * x[nc6 + k];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if (lane == 0) { y[nc6 + q] = acc; dot += acc * x[nc6 + q]; }
  }
  return dot;
}

// zeta = Minv r for this block's rows; returns partial r'zeta.  Minv_i is block diagonal: [n_intr][KI*KI].
// With a coarse space (A.W != nullptr) two extra grid-wide steps come first: Cv = Wa' r_c, Yv = Einv Cv.
__device__ __forceinline__ double precond_rows(cg::grid_group &grid, const PcgArgs &A, const double *__restrict__ r, double *__restrict__ zeta) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31, gwarp = tid >> 5, nwarps = nt >> 5;
  const int nc6 = 6 * A.n_poses;
  const bool coarse = A.W != nullptr && A.C.nco > 0;
  if (coarse) {
    const int nw = A.C.nw, nco = A.C.nco;
    for (int g = gwarp; g < A.C.ng; g += nwarps) {
      const int c0 = A.C.agg_start[g], ne = 6 * (A.C.agg_start[g + 1] - c0);
      for (int m = 0; m < nw; ++m) {
        double v = 0;
        for (int idx = lane; idx < ne; idx += 32) { const size_t e = 6 * (size_t)A.C.agg_cams[c0 + idx / 6] + idx % 6; v += A.W[(size_t)m * nc6 + e] * r[e]; }
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) A.Cv[g * nw + m] = v;
      }
    }
    grid.sync();
    for (int row = gwarp; row < nco; row += nwarps) {
      const double *er = A.Einv + (size_t)row * nco;
      double v = 0; for (int k = lane; k < nco; k += 32) v += er[k] * __ldcg(A.Cv + k);
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) A.Yv[row] = v;
    }
    grid.sync();
  }
  double dot = 0;
  for (int i = tid; i < nc6; i += nt) {
    const int a = i / 6, k = i % 6; const double *M = A.Minv_c + 36 * (size_t)a + 6 * k; const double *rb = r + 6 * a;
    double v = M[0] * rb[0] + M[1] * rb[1] + M[2] * rb[2] + M[3] * rb[3] + M[4] * rb[4] + M[5] * rb[5];
    if (coarse) { const double *y = A.Yv + A.C.agg_of[a] * A.C.nw; for (int m = 0; m < A.C.nw; ++m) v += A.W[(size_t)m * nc6 + i] * __ldcg(y + m); }
    zeta[i] = v; dot += v * r[i];
  }
  for (int q = tid; q < A.ni8; q += nt) {
    const double *M = A.Minv_i + (size_t)(q / KI) * KI * KI + (q % KI) * KI; const double *rb = r + nc6 + (q / KI) * KI;
    double v = 0;
    #pragma unroll
    for (int k = 0; k < KI; ++k) v += M[k] * rb[k];
    zeta[nc6 + q] = v; dot += v * r[nc6 + q];
  }
  return dot;
}

__global__ void __launch_bounds__(256) pcg_kernel(PcgArgs A) {
  cg::grid_group grid = cg::this_grid();
  __shared__ double sh[8];
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  const int nred = 6 * A.n_poses + A.ni8;
  double *P0 = A.part, *P1 = A.part + gridDim.x, *P2 = A.part + 2 * gridDim.x;
  double bb = 0;
  for (int i = tid; i < nred; i += nt) { A.z[i] = 0.0; const double b = A.rhs[i]; A.res[i] = b; bb += b * b; }
  const double bnorm2 = grid_sum(grid, bb, P0, sh);
  double rz = grid_sum(grid, precond_rows(grid, A, A.res, A.zeta), P1, sh);
  for (int i = tid; i < nred; i += nt) A.p[i] = A.zeta[i];
  grid.sync();
  int it = 0; double rr = bnorm2;
  if (bnorm2 > 0.0) {
    for (it = 1; it <= A.max_iter; ++it) {
      const double pw = grid_sum(grid, spmv_rows(A, A.p, A.w), P0, sh);
      const double alpha = rz / pw;
      double rr_l = 0;
      for (int i = tid; i < nred; i += nt) { A.z[i] += alpha * A.p[i]; const double rn = A.res[i] - alpha * A.w[i]; A.res[i] = rn; rr_l += rn * rn; }
      rr = grid_sum(grid, rr_l, P2, sh);
      if (!(rr > A.tol * A.tol * bnorm2)) break;
      const double rz_new = grid_sum(grid, precond_rows(grid, A, A.res, A.zeta), P1, sh);
      const double beta = rz_new / rz; rz = rz_new;
      for (int i = tid; i < nred; i += nt) A.p[i] = A.zeta[i] + beta * A.p[i];
      grid.sync();
    }
  }
  if (tid == 0) { A.out[0] = (double)(it > A.max_iter ? A.max_iter : it); A.out[1] = bnorm2 > 0 ? sqrt(rr / bnorm2) : 0.0; A.out[2] = sqrt(bnorm2); }
}

// ------------------------------------------------------------------------------ block-PCG (pcg3 / pcg5): common parts
// Two-level preconditioned block-PCG on the camera-camera part of the reduced system, with the
// (small, dense) intrinsics border removed by block elimination:
//     [Scc Sci'] [zc]   [bc]        Scc Y = [bc | Sci'] (1 + ni8 right-hand sides, solved together)
//     [Sci Sii ] [zi] = [bi]   =>   (Sii - Sci Y2) zi = bi - Sci y1 ;  zc = y1 - Y2 zi
// Preconditioner: M^-1 = blockdiag(Scc_pp)^-1 + W (W' Scc W)^-1 W', where the columns of W are the
// (<= 7) gauge generators of the scene (3 translations, scale, 3 rotations) expressed in the scaled
// camera coordinates.  Those are exactly the eigenvectors LM damping leaves at ~1/radius; with them
// in the coarse space the preconditioned spectrum is radius-independent (cond ~ 3-4), so ~20-30
// iterations reach 1e-10 where block-Jacobi alone needs > 1000.
constexpr int MAXW = 7;
constexpr int MAXRHS = 1 + 32;     // bc + up to 32 free intrinsic columns handled by block elimination

// gauge generators, camera part, scaled:  W[m][6p+k] = g_m[6p+k] / scale[6p+k] (0 on constant coordinates)
__global__ void gauge_kernel(const double *__restrict__ poses, const double *__restrict__ camR, const double *__restrict__ camdR,
                             const double *__restrict__ sc_cam, unsigned pose_mask, int n_poses, unsigned gen_mask, int nw, double *__restrict__ W) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x; if (p >= n_poses) return;
  const double *R = camR + 9 * p, *dR = camdR + 27 * p, *t = poses + 6 * p + 3;
  double g[7][6];
  for (int m = 0; m < 7; ++m) for (int k = 0; k < 6; ++k) g[m][k] = 0.0;
  for (int a = 0; a < 3; ++a) for (int i = 0; i < 3; ++i) g[a][3 + i] = -R[i * 3 + a];        // X += e_a : dt = -R e_a
  for (int i = 0; i < 3; ++i) g[3][3 + i] = t[i];                                             // X *= (1+s): dt = t
  // X -> (I + [e_a]x) X : R' = R (I - [e_a]x), t' = t.  Solve sum_k dR_k dw_k = -R [e_a]x (least squares, exact)
  double AtA[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int k = 0; k < 3; ++k) for (int l = 0; l < 3; ++l) { double v = 0; for (int i = 0; i < 9; ++i) v += dR[9 * k + i] * dR[9 * l + i]; AtA[k * 3 + l] = v; }
  const double m6[6] = {AtA[0], AtA[3], AtA[4], AtA[6], AtA[7], AtA[8]};
  double inv[9];
  if (inv3_spd(m6, inv)) {
    for (int a = 0; a < 3; ++a) {
      double B[9];                                      // -R [e_a]x ; ([e]x)_{lj}: column j = e x e_j
      for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) {
        // [e_a]x = [[0,-e2,e1],[e2,0,-e0],[-e1,e0,0]]
        double v = 0;
        for (int l = 0; l < 3; ++l) {
          double ex = 0;
          if (l == 0 && j == 1) ex = -(a == 2); if (l == 0 && j == 2) ex = (a == 1);
          if (l == 1 && j == 0) ex = (a == 2);  if (l == 1 && j == 2) ex = -(a == 0);
          if (l == 2 && j == 0) ex = -(a == 1); if (l == 2 && j == 1) ex = (a == 0);
          v += R[i * 3 + l] * ex;
        }
        B[i * 3 + j] = -v;
      }
      double Atb[3];
      for (int k = 0; k < 3; ++k) { double v = 0; for (int i = 0; i < 9; ++i) v += dR[9 * k + i] * B[i]; Atb[k] = v; }
      for (int k = 0; k < 3; ++k) g[4 + a][k] = inv[k * 3] * Atb[0] + inv[k * 3 + 1] * Atb[1] + inv[k * 3 + 2] * Atb[2];
    }
  }
  int row = 0;
  for (int m = 0; m < 7; ++m) {
    if (!((gen_mask >> m) & 1)) continue;
    for (int k = 0; k < 6; ++k) W[(size_t)row * 6 * n_poses + 6 * p + k] = ((pose_mask >> k) & 1) ? g[m][k] / sc_cam[6 * p + k] : 0.0;
    ++row;
  }
  (void)nw;
}

struct Pcg2Args {
  const double *Scc; const int *rowptr, *cols; const double *Sci, *Sii, *rhs, *Minv_c;
  const double *W;            // [nw][nc6]
  const unsigned *intr_mask;  // free intrinsic parameters (block elimination columns)
  int n_poses, ni8, nw;
  double *X, *Rv, *Pv, *Wv, *Zv;   // [nrhs][nc6] each
  double *AW;                 // not read by pcg3 / pcg5 (left null); kept so that their parameter layout, and code, stay as measured
  double *part;               // [gridDim.x][PCG2_V] partial reductions
  double *z;                  // out: reduced step [nc6 + ni8]
  double tol; int max_iter;
  double *out;                // [0]=iterations, [1]=max relative residual, [2]=|bc|
};
constexpr int PCG2_V = 320;   // max reduction width: nrhs*(1+nw) <= 33*8 = 264, border 32*33 handled in chunks
constexpr int PCG2_THREADS = 256;

constexpr int PCG3_NCO_MAX = 1024;          // coarse dimension bound (aggregation keeps 7 * n_aggregates below it)
struct Pcg2Smem {
  double wpart[PCG2_THREADS / 32][PCG2_V];   // per-warp partials
  double bv[PCG2_V], tot[PCG2_V];
  double Einv[MAXW * MAXW];
  double alpha[MAXRHS], beta[MAXRHS], rz[MAXRHS], bb[MAXRHS], zi[MAXRHS];
  double T[32][33];
  int rhs_col[MAXRHS];
  unsigned char done[MAXRHS];
  int nrhs, all_done; double worst;
};

// warp-reduce v; lane 0 ADDS it into this warp's slot idx (slots are zeroed by vsum_begin)
template <class SM> __device__ __forceinline__ void warp_acc(SM &S, double v, int idx) {
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) S.wpart[threadIdx.x >> 5][idx] += v;
}
template <class SM> __device__ __forceinline__ void vsum_begin(SM &S, int V) {
  for (int i = threadIdx.x; i < V * (PCG2_THREADS / 32); i += PCG2_THREADS) S.wpart[i / V][i % V] = 0.0;
  __syncthreads();
}
// block partials -> global -> grid.sync -> fixed-order totals in S.tot[0..V) (identical in every block).
// Cross-block sum: one warp per value, lanes stride over the blocks (5 loads each at 148 blocks), then a
// fixed butterfly — the same order in every block, hence bitwise identical totals everywhere.
template <class SM> __device__ __forceinline__ void vsum_end(cg::grid_group &grid, SM &S, int V, double *part) {
  __syncthreads();
  if (gridDim.x == 1) {                      // single-CTA solve (pcg5 with one aggregate): a block barrier is the grid barrier
    for (int i = threadIdx.x; i < V; i += PCG2_THREADS) { double t = 0; for (int w = 0; w < PCG2_THREADS / 32; ++w) t += S.wpart[w][i]; S.tot[i] = t; }
    __threadfence_block();
    __syncthreads();
    return;
  }
  for (int i = threadIdx.x; i < V; i += PCG2_THREADS) { double t = 0; for (int w = 0; w < PCG2_THREADS / 32; ++w) t += S.wpart[w][i]; part[(size_t)blockIdx.x * PCG2_V + i] = t; }
  grid.sync();
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, nb = (int)gridDim.x;
  for (int i = wib; i < V; i += PCG2_THREADS / 32) {
    double t = 0;
    for (int b = lane; b < nb; b += 32) t += part[(size_t)b * PCG2_V + i];
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) S.tot[i] = t;
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------ PCG v3 (aggregated coarse space)
// Same block elimination of the intrinsics border as above, but the coarse space of the two-level
// preconditioner is piecewise: the cameras are partitioned into aggregates (<= ~16 graph neighbours,
// built on the host from the camera-pair structure) and every aggregate carries its own copy of the
// <= 7 gauge generators.  Long camera chains drift by slowly varying similarity transforms — exactly
// what piecewise-rigid coarse functions capture — so the iteration count stays ~30-70 from 10 to
// 1000+ cameras where the single global gauge space needs 500-900 (measured, tools/ notes in DESIGN.md).
//   M^-1 = blockdiag(Scc_pp)^-1 + Wa (Wa' Scc Wa)^-1 Wa',   Wa[(g,m)] = W[m] restricted to aggregate g.

// E += Wa' Scc Wa, one thread per S block (a,b): the nw x nw coupling of aggregates g(a), g(b)
__global__ void coarse_assemble_kernel(const double *__restrict__ Scc, const int *__restrict__ brow, const int *__restrict__ cols, int nnzb,
                                       const double *__restrict__ W, int n_poses, Coarse C, double *__restrict__ E) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x; if (e >= nnzb) return;
  const int a = brow[e], b = cols[e];
  const size_t nc6 = 6 * (size_t)n_poses;
  double blk[36];
  #pragma unroll
  for (int i = 0; i < 36; ++i) blk[i] = Scc[36 * (size_t)e + i];
  const int ga = C.agg_of[a], gb = C.agg_of[b];
  for (int m2 = 0; m2 < C.nw; ++m2) {
    double wb[6], sw[6];
    #pragma unroll
    for (int k = 0; k < 6; ++k) wb[k] = W[m2 * nc6 + 6 * b + k];
    #pragma unroll
    for (int i = 0; i < 6; ++i) { double v = 0;
      #pragma unroll
      for (int k = 0; k < 6; ++k) v += blk[i * 6 + k] * wb[k];
      sw[i] = v; }
    for (int m1 = 0; m1 < C.nw; ++m1) {
      double v = 0;
      #pragma unroll
      for (int i = 0; i < 6; ++i) v += W[m1 * nc6 + 6 * a + i] * sw[i];
      if (v != 0.0) atomicAdd(&E[(size_t)(ga * C.nw + m1) * C.nco + gb * C.nw + m2], v);
    }
  }
}

// Coarse operator inverse by blocked Gauss-Jordan, in place, ONE cooperative kernel.  A blocked Cholesky with an
// explicit triangular inverse serialises on that inverse (one CTA per block column; 2.46 vs 1.0 ms, DESIGN.md §4.3);
// Gauss-Jordan does twice the flops but every pivot step is a rank-32 update of the WHOLE matrix — 196 independent
// 64x64 tiles — between two grid syncs:
//   phase 1 (every CTA): B = inv(A_KK) redundantly in shared memory; slices of  Cold = A[:,K] (copy),
//                        H = B A[K,:],  Gn = -A[:,K] B  into scratch
//   phase 2 (tiles):     A_ij <- A_ij - Cold_i H_j  (i,j not in K);  A_Kj <- H_j;  A_iK <- Gn_i;  A_KK <- B
// A is symmetrised (+ tiny ridge) first; SPD input needs no pivoting (every pivot block is a Schur complement).
constexpr int CT = 64;           // output tile
constexpr int GJ_B = 32;
__device__ __forceinline__ unsigned long long gtimer2() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define GJ_LAP(k) do { if (tim && tid == 0) { const unsigned long long now_ = gtimer2(); tim[k] += now_ - tlast; tlast = now_; } } while (0)
// Measured per inversion at n = 875 (28 pivot steps, us): pivot-block inverse 533, slices 64, tiles 172, grid syncs 145.
// The 32 sequential pivots of a block (an FP64 reciprocal and two barriers each) are the critical path; a one-warp
// register-resident variant with shuffle broadcasts was twice slower (1050 us) and was dropped.
__global__ void __launch_bounds__(256, 2) coarse_invert_kernel(double *__restrict__ A, int n, double *__restrict__ tmp, int *__restrict__ fail, unsigned long long *__restrict__ tim) {
  cg::grid_group grid = cg::this_grid();
  __shared__ double Bs[GJ_B][GJ_B + 1];
  __shared__ double As[CT][GJ_B + 1];
  __shared__ double Hs[GJ_B][CT + 1];
  __shared__ double s_red[8];
  __shared__ double s_row[GJ_B], s_col[GJ_B];
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  double *Cold = tmp, *H = tmp + (size_t)GJ_B * n, *Gn = tmp + 2 * (size_t)GJ_B * n;     // [n][32], [32][n], [n][32]
  // ridge = 1e-15 * max diagonal (every CTA computes it: no extra sync)
  { double mx = 0; for (int i = threadIdx.x; i < n; i += blockDim.x) mx = fmax(mx, A[(size_t)i * n + i]);
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = mx;
    __syncthreads();
    mx = 0; for (int w = 0; w < 8; ++w) mx = fmax(mx, s_red[w]);
    const double ridge = 1e-15 * mx;
    grid.sync();                                           // everyone has read the diagonal before it changes
    for (long long idx = tid; idx < (long long)n * n; idx += nt) {
      const int i = (int)(idx / n), j = (int)(idx % n);
      if (j < i) { const double v = 0.5 * (A[(size_t)i * n + j] + A[(size_t)j * n + i]); A[(size_t)i * n + j] = v; A[(size_t)j * n + i] = v; }
      else if (j == i) A[idx] += ridge;
    } }
  grid.sync();
  const int mt = (n + CT - 1) / CT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  unsigned long long tlast = tim ? gtimer2() : 0ull;
  for (int k0 = 0; k0 < n; k0 += GJ_B) {
    const int nb = min(GJ_B, n - k0);
    // ---- phase 1: B = inv(A_KK), identity-padded to 32.  Gauss-Jordan by ONE warp: lane r keeps row r in registers,
    // the pivot row goes through shared memory (one broadcast LDS per element) — no block barrier inside the 32
    // sequential pivots (the 256-thread version paid two __syncthreads and an FP64 reciprocal per pivot: 19 us per block)
    if (threadIdx.x < 32) {
      const int r = threadIdx.x;
      double b[GJ_B];
      #pragma unroll
      for (int c2 = 0; c2 < GJ_B; ++c2) b[c2] = (r < nb && c2 < nb) ? __ldcg(A + (size_t)(k0 + r) * n + k0 + c2) : (r == c2 ? 1.0 : 0.0);
      #pragma unroll
      for (int k = 0; k < GJ_B; ++k) {
        if (r == k) {
          #pragma unroll
          for (int c2 = 0; c2 < GJ_B; ++c2) s_row[c2] = b[c2];
        }
        __syncwarp();
        const double piv = s_row[k];
        if (!(piv > 0.0) || !isfinite(piv)) { if (r == 0 && blockIdx.x == 0) atomicExch(fail, 4); }
        const double ip = __drcp_rn(piv);                  // (1.0 / piv compiles to the same reciprocal plus a slow-path division)
        const double f = b[k];
        if (r == k) {
          #pragma unroll
          for (int c2 = 0; c2 < GJ_B; ++c2) b[c2] = c2 == k ? ip : b[c2] * ip;
        } else {
          const double fi = f * ip;
          #pragma unroll
          for (int c2 = 0; c2 < GJ_B; ++c2) b[c2] = c2 == k ? -fi : b[c2] - fi * s_row[c2];
        }
        __syncwarp();
      }
      #pragma unroll
      for (int c2 = 0; c2 < GJ_B; ++c2) Bs[r][c2] = b[c2];
    }
    __syncthreads();
    // slices of Cold / H / Gn
    GJ_LAP(0);
    // (all 32 operand loads of a slice element are issued before the first FMA: L1 is cold after a grid sync and a
    // dependent L2 round trip costs ~0.5 us; Bs is identity-padded, so out-of-range pivots contribute zeros)
    for (long long idx = tid; idx < (long long)n * GJ_B; idx += nt) {
      const int i = (int)(idx >> 5), q = (int)(idx & 31);
      double av[GJ_B];
      #pragma unroll
      for (int p2 = 0; p2 < GJ_B; ++p2) av[p2] = p2 < nb ? __ldcg(A + (size_t)i * n + k0 + p2) : 0.0;
      double g = 0.0;
      #pragma unroll
      for (int p2 = 0; p2 < GJ_B; ++p2) g += av[p2] * Bs[p2][q];
      Cold[idx] = q < nb ? __ldcg(A + (size_t)i * n + k0 + q) : 0.0;
      Gn[idx] = q < nb ? -g : 0.0;
    }
    for (long long idx = tid; idx < (long long)n * GJ_B; idx += nt) {
      const int q = (int)(idx / n), j = (int)(idx % n);
      double av[GJ_B];
      #pragma unroll
      for (int p2 = 0; p2 < GJ_B; ++p2) av[p2] = p2 < nb ? __ldcg(A + (size_t)(k0 + p2) * n + j) : 0.0;
      double h = 0.0;
      #pragma unroll
      for (int p2 = 0; p2 < GJ_B; ++p2) h += Bs[q][p2] * av[p2];
      H[idx] = q < nb ? h : 0.0;
    }
    GJ_LAP(1);
    grid.sync();
    GJ_LAP(2);
    // ---- phase 2: tiles
    for (int t = blockIdx.x; t < mt * mt; t += gridDim.x) {
      const int i0 = (t / mt) * CT, j0 = (t % mt) * CT;
      __syncthreads();
      for (int idx = threadIdx.x; idx < CT * GJ_B; idx += 256) { const int r = idx >> 5, q = idx & 31; As[r][q] = i0 + r < n ? Cold[(size_t)(i0 + r) * GJ_B + q] : 0.0; }
      for (int idx = threadIdx.x; idx < CT * GJ_B; idx += 256) { const int q = idx / CT, c2 = idx % CT; Hs[q][c2] = j0 + c2 < n ? H[(size_t)q * n + j0 + c2] : 0.0; }
      __syncthreads();
      double acc[4][4], aold[4][4];                            // the tile's old values are fetched under the product
      #pragma unroll
      for (int p2 = 0; p2 < 4; ++p2)
        #pragma unroll
        for (int q = 0; q < 4; ++q) {
          acc[p2][q] = 0.0;
          const int r = i0 + ty + 16 * p2, c2 = j0 + tx + 16 * q;
          aold[p2][q] = (r < n && c2 < n) ? __ldcg(A + (size_t)r * n + c2) : 0.0;
        }
      #pragma unroll 8
      for (int kk = 0; kk < GJ_B; ++kk) {
        double av[4], bv[4];
        #pragma unroll
        for (int p2 = 0; p2 < 4; ++p2) { av[p2] = As[ty + 16 * p2][kk]; bv[p2] = Hs[kk][tx + 16 * p2]; }
        #pragma unroll
        for (int p2 = 0; p2 < 4; ++p2)
          #pragma unroll
          for (int q = 0; q < 4; ++q) acc[p2][q] += av[p2] * bv[q];
      }
      #pragma unroll
      for (int p2 = 0; p2 < 4; ++p2)
        #pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int r = i0 + ty + 16 * p2, c2 = j0 + tx + 16 * q;
          if (r >= n || c2 >= n) continue;
          const bool rk = r >= k0 && r < k0 + nb, ck = c2 >= k0 && c2 < k0 + nb;
          double v;
          if (rk) v = ck ? Bs[r - k0][c2 - k0] : Hs[r - k0][tx + 16 * q];
          else v = ck ? Gn[(size_t)r * GJ_B + (c2 - k0)] : aold[p2][q] - acc[p2][q];
          A[(size_t)r * n + c2] = v;
        }
    }
    GJ_LAP(3);
    grid.sync();
    GJ_LAP(4);
  }
}

struct Pcg3Args {
  Pcg2Args base;          // Scc, Sci, Sii, rhs, Minv_c, W, intr_mask, X/Rv/Pv/Wv/Zv, part, z, tol, max_iter, out
  Coarse C;
  const double *Einv;     // [nco][nco]
  double *Cv;             // [MAXRHS][nco] coarse residuals  W_a' r
  double *Yv;             // [MAXRHS][nco] coarse corrections Einv c
  double *Pv2;            // second direction buffer (ping-pong with base.Pv)
  unsigned long long *tim; // optional (OMVG_BA_PCG_TIMING): ns spent by CTA 0 in [coarse, z, spmv, update, other]
};
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define PCG_LAP(k) do { if (P.tim && tid == 0) { const unsigned long long now_ = gtimer(); P.tim[k] += now_ - tlast; tlast = now_; } } while (0)

// 32-byte read-only load (LDG.E.256, sm_100): a 6x6 block is 9 of these instead of 36 8-byte loads, which at the
// 288-byte lane stride cost one L1 wavefront per lane per instruction (the SpMV was L1-wavefront bound)
__device__ __forceinline__ void ldg256(const double *p, double &a, double &b, double &c, double &d) {
  asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
// w_j = Scc p_j with p_j = z_j + beta_j * pold_j formed ON THE FLY for the gathered columns (so the
// direction update needs no grid sync of its own); the owner warp of row a stores p_j(a) into pnew and
// accumulates p_j.w_j over its rows into this warp's reduction slot j.
__device__ __forceinline__ void spmv_pcg(const Pcg2Args &A, Pcg2Smem &S, const double *__restrict__ Z, const double *__restrict__ Pold,
                                         double *__restrict__ Pnew, double *__restrict__ Wv, int nv) {
  const int lane = threadIdx.x & 31, warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const size_t nc6 = 6 * (size_t)A.n_poses;
  for (int a = warp; a < A.n_poses; a += nwarps) {
    for (int j0 = 0; j0 < nv; j0 += 4) {
      double acc[4][6];
      #pragma unroll
      for (int j = 0; j < 4; ++j)
        #pragma unroll
        for (int i = 0; i < 6; ++i) acc[j][i] = 0.0;
      for (int e = A.rowptr[a] + lane; e < A.rowptr[a + 1]; e += 32) {
        const double *blk = A.Scc + 36 * (size_t)e; const int cb = 6 * A.cols[e];
        double b[36];
        #pragma unroll
        for (int i = 0; i < 9; ++i) ldg256(blk + 4 * i, b[4 * i], b[4 * i + 1], b[4 * i + 2], b[4 * i + 3]);
        #pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j0 + j < nv && !S.done[j0 + j]) {
            const size_t off = (size_t)(j0 + j) * nc6 + cb; const double bt = S.beta[j0 + j];
            // the 6-vectors are 48 contiguous, 16-byte aligned bytes: three 16-byte loads each instead of six 8-byte
            // ones (at a 48-byte lane stride every load instruction costs one L1 wavefront per lane)
            const double2 *zp = reinterpret_cast<const double2 *>(Z + off), *pp = reinterpret_cast<const double2 *>(Pold + off);
            const double2 z0 = zp[0], z1 = zp[1], z2 = zp[2], q0 = pp[0], q1 = pp[1], q2 = pp[2];
            const double xv[6] = {z0.x + bt * q0.x, z0.y + bt * q0.y, z1.x + bt * q1.x, z1.y + bt * q1.y, z2.x + bt * q2.x, z2.y + bt * q2.y};
            #pragma unroll
            for (int i = 0; i < 6; ++i)
              #pragma unroll
              for (int k = 0; k < 6; ++k) acc[j][i] += b[i * 6 + k] * xv[k];
          }
        }
      }
      #pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (j0 + j < nv && !S.done[j0 + j]) {
          #pragma unroll
          for (int i = 0; i < 6; ++i) { double v = acc[j][i]; for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o); acc[j][i] = v; }
          if (lane == 0) {
            const size_t off = (size_t)(j0 + j) * nc6 + 6 * (size_t)a; const double bt = S.beta[j0 + j];
            double d = 0;
            for (int i = 0; i < 6; ++i) { const double pv = Z[off + i] + bt * Pold[off + i]; Pnew[off + i] = pv; Wv[off + i] = acc[j][i]; d += acc[j][i] * pv; }
            S.wpart[threadIdx.x >> 5][j0 + j] += d;
          }
        }
      }
    }
  }
}

__global__ void __launch_bounds__(PCG2_THREADS) pcg3_kernel(Pcg3Args P) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ unsigned char pcg2_smem_raw[];
  Pcg2Smem &S = *reinterpret_cast<Pcg2Smem *>(pcg2_smem_raw);
  const Pcg2Args &A = P.base; const Coarse &C = P.C;
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31, gwarp = tid >> 5, nwarps = nt >> 5;
  const size_t nc6 = 6 * (size_t)A.n_poses;
  const int nw = C.nw, nco = C.nco;
  if (threadIdx.x == 0) {
    int n = 1; S.rhs_col[0] = -1;
    for (int q = 0; q < A.ni8; ++q) if ((A.intr_mask[q / KI] >> (q % KI)) & 1) { if (n < MAXRHS) S.rhs_col[n++] = q; }
    S.nrhs = n;
  }
  __syncthreads();
  const int nrhs = S.nrhs;
  double *Pcur = A.Pv, *Pnext = P.Pv2;
  // ---- init (aggregate-owned elements): X = 0, P = 0, R = B, |b|^2, coarse residual
  vsum_begin(S, nrhs);
  // (aggregate, right-hand side) pairs are the unit of work of the vector phases: ng * nrhs warp tasks
  for (int task = gwarp; task < C.ng * nrhs; task += nwarps) {
    const int g = task / nrhs, j = task - g * nrhs;
    const int c0 = C.agg_start[g], ne = 6 * (C.agg_start[g + 1] - c0);
    {
      const double *src = j == 0 ? A.rhs : A.Sci + (size_t)S.rhs_col[j] * nc6;
      double v = 0;
      double cm[MAXW];
      #pragma unroll
      for (int m = 0; m < MAXW; ++m) cm[m] = 0.0;
      for (int idx = lane; idx < ne; idx += 32) {
        const size_t e = 6 * (size_t)C.agg_cams[c0 + idx / 6] + idx % 6; const double b = src[e];
        A.X[j * nc6 + e] = 0.0; Pcur[j * nc6 + e] = 0.0; A.Rv[j * nc6 + e] = b; v += b * b;
        #pragma unroll
        for (int m = 0; m < MAXW; ++m) if (m < nw) cm[m] += A.W[m * nc6 + e] * b;
      }
      warp_acc(S, v, j);
      #pragma unroll
      for (int m = 0; m < MAXW; ++m) if (m < nw) {
        double cv = cm[m]; for (int o = 16; o > 0; o >>= 1) cv += __shfl_xor_sync(0xffffffffu, cv, o);
        if (lane == 0) P.Cv[(size_t)j * nco + g * nw + m] = cv;
      }
    }
  }
  vsum_end(grid, S, nrhs, A.part);
  if (threadIdx.x < nrhs) { const int j = threadIdx.x; S.bb[j] = S.tot[j]; S.done[j] = !(S.tot[j] > 0.0); S.alpha[j] = 0; S.beta[j] = 0; S.rz[j] = 0; }
  if (threadIdx.x == 0) { S.worst = 0; S.all_done = 0; }
  __syncthreads();
  int it = 0;
  unsigned long long tlast = P.tim ? gtimer() : 0ull;
  for (;;) {
    // (y) coarse solve  Y_j = Einv C_j, one row per warp.  The phase is pure latency (L1 is cold after a grid sync,
    // every operand comes from L2): the right-hand sides are staged once per CTA in shared memory and each lane
    // issues ALL its row loads back to back before the first FMA (the naive k-loop paid one L2 round trip per
    // 5 loads: 13 us per iteration).
    if (nco > 0) {
      double *sCv = reinterpret_cast<double *>(pcg2_smem_raw + sizeof(Pcg2Smem));     // [4][PCG3_NCO_MAX]
      for (int j0 = 0; j0 < nrhs; j0 += 4) {
        const int nj = min(4, nrhs - j0);
        for (int kc = 0; kc < nco; kc += PCG3_NCO_MAX) {       // (one chunk unless the coarse space exceeds 1024)
          const int nk = min(PCG3_NCO_MAX, nco - kc);
          { double tv[4][(PCG3_NCO_MAX + PCG2_THREADS - 1) / PCG2_THREADS];      // all loads in flight before the first store
            #pragma unroll
            for (int j = 0; j < 4; ++j)
              #pragma unroll
              for (int q = 0; q < (PCG3_NCO_MAX + PCG2_THREADS - 1) / PCG2_THREADS; ++q) { const int k = threadIdx.x + PCG2_THREADS * q; tv[j][q] = (j < nj && k < nk) ? __ldcg(P.Cv + (size_t)(j0 + j) * nco + kc + k) : 0.0; }
            #pragma unroll
            for (int j = 0; j < 4; ++j)
              #pragma unroll
              for (int q = 0; q < (PCG3_NCO_MAX + PCG2_THREADS - 1) / PCG2_THREADS; ++q) { const int k = threadIdx.x + PCG2_THREADS * q; if (k < nk) sCv[j * PCG3_NCO_MAX + k] = tv[j][q]; } }
          __syncthreads();
          PCG_LAP(6);
          for (int row = gwarp; row < nco; row += nwarps) {
            const double *er = P.Einv + (size_t)row * nco + kc;
            double ev[PCG3_NCO_MAX / 32];
            #pragma unroll
            for (int q = 0; q < PCG3_NCO_MAX / 32; ++q) { const int k = lane + 32 * q; ev[q] = k < nk ? __ldcg(er + k) : 0.0; }
            double acc[4] = {0, 0, 0, 0};
            #pragma unroll
            for (int q = 0; q < PCG3_NCO_MAX / 32; ++q) { const int k = lane + 32 * q;
              if (k < nk) {
                #pragma unroll
                for (int j = 0; j < 4; ++j) if (j < nj) acc[j] += ev[q] * sCv[j * PCG3_NCO_MAX + k]; } }
            #pragma unroll
            for (int j = 0; j < 4; ++j) {
              double v = acc[j]; for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
              if (lane == 0 && j < nj) { double *dst = P.Yv + (size_t)(j0 + j) * nco + row; *dst = kc == 0 ? v : *dst + v; }
            }
          }
          __syncthreads();
          PCG_LAP(7);
        }
      }
      grid.sync();
    }
    PCG_LAP(0);
    // (b) z = Minv r + Wa y ;  r'z
    vsum_begin(S, nrhs);
    for (int task = gwarp; task < C.ng * nrhs; task += nwarps) {
      const int g = task / nrhs, j = task - g * nrhs;
      const int c0 = C.agg_start[g], ne = 6 * (C.agg_start[g + 1] - c0);
      {
        if (S.done[j]) continue;
        double y[MAXW];
        #pragma unroll
        for (int m = 0; m < MAXW; ++m) y[m] = m < nw ? P.Yv[(size_t)j * nco + g * nw + m] : 0.0;
        double rzp = 0;
        for (int idx = lane; idx < ne; idx += 32) {
          const size_t cam = C.agg_cams[c0 + idx / 6]; const int k = idx % 6; const size_t e = 6 * cam + k;
          const double *rb = A.Rv + j * nc6 + 6 * cam;
          const double2 *M2 = reinterpret_cast<const double2 *>(A.Minv_c + 36 * cam + 6 * k), *r2 = reinterpret_cast<const double2 *>(rb);   // 16-byte loads
          const double2 m0 = M2[0], m1 = M2[1], m2 = M2[2], b0 = r2[0], b1 = r2[1], b2 = r2[2];
          double zz = m0.x * b0.x + m0.y * b0.y + m1.x * b1.x + m1.y * b1.y + m2.x * b2.x + m2.y * b2.y;
          #pragma unroll
          for (int m = 0; m < MAXW; ++m) if (m < nw) zz += A.W[m * nc6 + e] * y[m];
          A.Zv[j * nc6 + e] = zz; rzp += zz * rb[k];
        }
        warp_acc(S, rzp, j);
      }
    }
    vsum_end(grid, S, nrhs, A.part);
    if (threadIdx.x < nrhs) { const int j = threadIdx.x; if (!S.done[j]) { const double rzn = S.tot[j]; S.beta[j] = it == 0 ? 0.0 : rzn / S.rz[j]; S.rz[j] = rzn; } }
    __syncthreads();
    PCG_LAP(1);
    if (it >= A.max_iter) break;
    // (c+d) p = z + beta p (on the fly) ; w = Scc p ; p'w
    vsum_begin(S, nrhs);
    spmv_pcg(A, S, A.Zv, Pcur, Pnext, A.Wv, nrhs);
    vsum_end(grid, S, nrhs, A.part);
    PCG_LAP(2);
    { double *t2 = Pcur; Pcur = Pnext; Pnext = t2; }
    if (threadIdx.x < nrhs) { const int j = threadIdx.x; S.alpha[j] = S.done[j] ? 0.0 : S.rz[j] / S.tot[j]; }
    __syncthreads();
    // (e) x += alpha p ; r -= alpha w ; |r|^2 ; coarse residual of the new r
    vsum_begin(S, nrhs);
    for (int task = gwarp; task < C.ng * nrhs; task += nwarps) {
      const int g = task / nrhs, j = task - g * nrhs;
      const int c0 = C.agg_start[g], ne = 6 * (C.agg_start[g + 1] - c0);
      {
        if (S.done[j]) continue;
        const double al = S.alpha[j]; double v = 0;
        double cm[MAXW];
        #pragma unroll
        for (int m = 0; m < MAXW; ++m) cm[m] = 0.0;
        for (int idx = lane; idx < ne; idx += 32) {
          const size_t e = 6 * (size_t)C.agg_cams[c0 + idx / 6] + idx % 6;
          A.X[j * nc6 + e] += al * Pcur[j * nc6 + e];
          const double rn = A.Rv[j * nc6 + e] - al * A.Wv[j * nc6 + e]; A.Rv[j * nc6 + e] = rn; v += rn * rn;
          #pragma unroll
          for (int m = 0; m < MAXW; ++m) if (m < nw) cm[m] += A.W[m * nc6 + e] * rn;
        }
        warp_acc(S, v, j);
        #pragma unroll
        for (int m = 0; m < MAXW; ++m) if (m < nw) {
          double cv = cm[m]; for (int o = 16; o > 0; o >>= 1) cv += __shfl_xor_sync(0xffffffffu, cv, o);
          if (lane == 0) P.Cv[(size_t)j * nco + g * nw + m] = cv;
        }
      }
    }
    vsum_end(grid, S, nrhs, A.part);                // its grid.sync publishes Cv as well
    PCG_LAP(3);
    ++it;
    if (threadIdx.x == 0) {
      int ad = 1; double wmax = 0;
      for (int j = 0; j < nrhs; ++j) if (!S.done[j]) { const double rel2 = S.tot[j] / S.bb[j]; wmax = fmax(wmax, rel2); if (!(rel2 > A.tol * A.tol)) S.done[j] = 1; else ad = 0; }
      S.all_done = ad; S.worst = wmax;
    }
    __syncthreads();
    if (S.all_done) break;
  }
  // ---- border: (Sii - Sci Y2) zi = bi - Sci y1 ; zc = y1 - Y2 zi
  PCG_LAP(4);
  const int k = nrhs - 1;
  if (k > 0) {
    for (int a = 0; a < k; ++a) {
      vsum_begin(S, k + 1);
      const double *row = A.Sci + (size_t)S.rhs_col[1 + a] * nc6;
      for (int b = 0; b <= k; ++b) {
        const double *x = A.X + (size_t)(b == k ? 0 : 1 + b) * nc6;
        double v = 0; for (size_t i = tid; i < nc6; i += nt) v += row[i] * x[i];
        warp_acc(S, v, b);
      }
      vsum_end(grid, S, k + 1, A.part);
      if (threadIdx.x <= k) {
        const int b = threadIdx.x;
        if (b < k) S.T[a][b] = A.Sii[(size_t)S.rhs_col[1 + a] * A.ni8 + S.rhs_col[1 + b]] - S.tot[b];
        else S.T[a][k] = A.rhs[nc6 + S.rhs_col[1 + a]] - S.tot[k];
      }
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      for (int a = 0; a < k; ++a) for (int b = a + 1; b < k; ++b) { const double m = 0.5 * (S.T[a][b] + S.T[b][a]); S.T[a][b] = m; S.T[b][a] = m; }
      for (int c = 0; c < k; ++c) {
        int piv = c; for (int r2 = c + 1; r2 < k; ++r2) if (fabs(S.T[r2][c]) > fabs(S.T[piv][c])) piv = r2;
        if (piv != c) for (int q = 0; q <= k; ++q) { const double t2 = S.T[c][q]; S.T[c][q] = S.T[piv][q]; S.T[piv][q] = t2; }
        for (int r2 = c + 1; r2 < k; ++r2) { const double f = S.T[r2][c] / S.T[c][c]; for (int q = c; q <= k; ++q) S.T[r2][q] -= f * S.T[c][q]; }
      }
      for (int c = k - 1; c >= 0; --c) { double sacc = S.T[c][k]; for (int q = c + 1; q < k; ++q) sacc -= S.T[c][q] * S.zi[q]; S.zi[c] = sacc / S.T[c][c]; }
    }
    __syncthreads();
  }
  for (size_t i = tid; i < nc6; i += nt) { double v = A.X[i]; for (int a = 0; a < k; ++a) v -= A.X[(size_t)(1 + a) * nc6 + i] * S.zi[a]; A.z[i] = v; }
  for (int q = tid; q < A.ni8; q += nt) { double v = 0; for (int a = 0; a < k; ++a) if (S.rhs_col[1 + a] == q) v = S.zi[a]; A.z[nc6 + q] = v; }
  PCG_LAP(5);
  if (tid == 0) { A.out[0] = (double)it; A.out[1] = sqrt(S.worst); A.out[2] = sqrt(S.bb[0]); }
}

// ------------------------------------------------------------------------------ PCG v5 (shared-memory resident)
// The v3 iteration is four grid-wide phases of three or four DEPENDENT L2 round trips each (every vector element a
// CTA touches was last written by another SM): ~26 us per iteration at 1000 cameras for ~0.3 us of arithmetic.
// Here CTA g owns aggregate g for the whole solve and keeps everything it owns in shared memory: its slices of
// x, r, p, z, w for up to 4 right-hand sides, its block-Jacobi inverses, its gauge vectors, the coarse residual and
// (as far as they fit: ~110 KB) the S blocks of its camera rows.  Per iteration only this crosses the chip:
//   [A] read  alpha-partials + Wa'w of all aggregates (one L2 trip)   write  z of its cameras, r'z / |r|^2 partials
//   [B] read  beta-partials + z, p of the neighbour cameras (one trip) write  p of its cameras, p'w partials, Wa'w
// i.e. two grid barriers and two L2 round trips; the coarse solve (its nw rows of Einv, fetched into registers in the
// shadow of the Wa'w read), the block-Jacobi step, the vector updates and the SpMV arithmetic are local.
// The coarse residual of the new r is not recomputed but updated, c_new = c - alpha Wa'w, with Wa'w formed during the
// SpMV and published by the same barrier as p'w.  Same stopping rule and iteration count as v3.
constexpr int PCG5_NR = 4;            // right-hand sides held in shared memory (1 + free intrinsic columns)
constexpr int PCG5_MC = 21;           // cameras per aggregate (aggregation keeps them <= ~16; 2000-camera scenes reach 17-20)
constexpr int PCG5_ST = ((PCG5_MC * 6 + 31) / 32) * 32;   // per-rhs thread stride: a warp never straddles two right-hand sides
constexpr int PCG5_BS = 37;           // padded block stride (doubles): lane-per-block reads without 4-way bank conflicts
constexpr int PCG5_NB = 112;          // neighbour cameras of an aggregate (union of the columns of its rows) staged per iteration
constexpr int PCG5_PS = PCG5_NR * 6 + 1;   // doubles per staged neighbour (4 rhs x 6, +1 pad: lanes hit different banks)
// reduction / control block of pcg5: at most 2 * PCG5_NR values per reduction (Pcg2Smem is sized for 33 right-hand sides
// x 8 generators and would cost 36 KB of the shared memory the S-block cache wants)
struct Pcg5Red {
  double wpart[PCG2_THREADS / 32][2 * PCG5_NR + 8];
  double tot[2 * PCG5_NR + 8];
  double alpha[PCG5_NR + 1], beta[PCG5_NR + 1], rz[PCG5_NR + 1], bb[PCG5_NR + 1], zi[PCG5_NR + 1];
  double T[PCG5_NR + 1][PCG5_NR + 2];
  int rhs_col[PCG5_NR + 1];
  unsigned char done[PCG5_NR + 4];
  int nrhs, all_done; double worst;
};
struct Pcg5Smem {
  double x[PCG5_NR][PCG5_MC * 6], r[PCG5_NR][PCG5_MC * 6], p[PCG5_NR][PCG5_MC * 6], z[PCG5_NR][PCG5_MC * 6], w[PCG5_NR][PCG5_MC * 6];
  double minv[PCG5_MC][36], wg[MAXW][PCG5_MC * 6];
  double y[MAXW][PCG5_NR], aw[PCG2_THREADS / 32][PCG5_NR][MAXW], wrow[PCG2_THREADS / 32][PCG5_NR][6], drow[PCG2_THREADS / 32][PCG5_NR * 6];
  int cams[PCG5_MC], rowstart[PCG5_MC + 1], rowptr0[PCG5_MC], nbl[PCG5_NB];
  int ncam, nb_cached, nnb;
};
__global__ void __launch_bounds__(PCG2_THREADS) pcg5_kernel(Pcg3Args P, double *__restrict__ Cg, double *__restrict__ AW, int nb_cache,
                                                                const int *__restrict__ nb_start, const int *__restrict__ nb_list, const unsigned short *__restrict__ blk_lcol) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ unsigned char pcg2_smem_raw[];
  Pcg5Red &S = *reinterpret_cast<Pcg5Red *>(pcg2_smem_raw);
  Pcg5Smem &L = *reinterpret_cast<Pcg5Smem *>(pcg2_smem_raw + sizeof(Pcg5Red));
  double *sCv = reinterpret_cast<double *>(pcg2_smem_raw + sizeof(Pcg5Red) + sizeof(Pcg5Smem));      // [PCG5_NR][PCG3_NCO_MAX]
  double *sPN = sCv + PCG5_NR * PCG3_NCO_MAX;                                                         // [PCG5_NB][PCG5_PS] p = z + beta p of the neighbours
  double *sS = sPN + PCG5_NB * PCG5_PS;                                                               // [nb_cache][PCG5_BS]
  unsigned short *sCol = reinterpret_cast<unsigned short *>(sS + (size_t)nb_cache * PCG5_BS);         // [nb_cache] position of the block's column in the neighbour list
  const Pcg2Args &A = P.base; const Coarse &C = P.C;
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  constexpr int NWARP = PCG2_THREADS / 32;
  const size_t nc6 = 6 * (size_t)A.n_poses;
  const int nw = C.nw, nco = C.nco;
  const int g = blockIdx.x;                       // the aggregate this CTA owns (CTAs beyond ng only take part in the barriers)
  const bool own = g < C.ng;
  if (threadIdx.x == 0) {
    int n = 1; S.rhs_col[0] = -1;
    for (int q = 0; q < A.ni8; ++q) if ((A.intr_mask[q / KI] >> (q % KI)) & 1) { if (n < PCG5_NR) S.rhs_col[n++] = q; }
    S.nrhs = n;
    const int c0 = own ? C.agg_start[g] : 0; L.ncam = own ? C.agg_start[g + 1] - c0 : 0;
    int nb = 0;
    for (int ci = 0; ci < L.ncam; ++ci) { const int a = C.agg_cams[c0 + ci]; L.cams[ci] = a; L.rowstart[ci] = nb; L.rowptr0[ci] = A.rowptr[a]; nb += A.rowptr[a + 1] - A.rowptr[a]; }
    L.rowstart[L.ncam] = nb; L.nb_cached = min(nb, nb_cache);
  }
  __syncthreads();
  const int nrhs = S.nrhs, ncam = L.ncam, ne = 6 * ncam;
  double *Pcur = A.Pv, *Pnext = P.Pv2;
  { const int nb0 = own ? nb_start[g] : 0; const int nnb = own ? nb_start[g + 1] - nb0 : 0;
    if (threadIdx.x == 0) L.nnb = nnb;
    for (int i = threadIdx.x; i < nnb; i += PCG2_THREADS) L.nbl[i] = nb_list[nb0 + i]; }
  __syncthreads();
  // ---- load what this CTA owns: block-Jacobi inverses, gauge vectors, S blocks of its rows
  for (int i = threadIdx.x; i < ncam * 36; i += PCG2_THREADS) L.minv[i / 36][i % 36] = A.Minv_c[36 * (size_t)L.cams[i / 36] + i % 36];
  for (int i = threadIdx.x; i < nw * ne; i += PCG2_THREADS) { const int m = i / ne, idx = i % ne; L.wg[m][idx] = A.W[m * nc6 + 6 * (size_t)L.cams[idx / 6] + idx % 6]; }
  for (int ci = 0; ci < ncam; ++ci) {
    const int nbr = L.rowstart[ci + 1] - L.rowstart[ci];
    for (int i = threadIdx.x; i < nbr * 36; i += PCG2_THREADS) {
      const int lb = L.rowstart[ci] + i / 36;
      if (lb < nb_cache) sS[(size_t)lb * PCG5_BS + i % 36] = A.Scc[36 * (size_t)(L.rowptr0[ci] + i / 36) + i % 36];
    }
    for (int i = threadIdx.x; i < nbr; i += PCG2_THREADS) { const int lb = L.rowstart[ci] + i; if (lb < nb_cache) sCol[lb] = blk_lcol[L.rowptr0[ci] + i]; }
  }
  // ---- init: x = 0, p = 0, w = 0, r = b, |b|^2, coarse residual of this aggregate -> Cg, p (global) = 0
  vsum_begin(S, nrhs);
  for (int t = threadIdx.x; t < nrhs * PCG5_ST; t += PCG2_THREADS) {
    const int j = t / PCG5_ST, idx = t % PCG5_ST;                       // (PCG5_ST is a multiple of 32: a warp never straddles two right-hand sides)
    double v = 0;
    if (idx < ne) {
      const size_t e = 6 * (size_t)L.cams[idx / 6] + idx % 6;
      const double b = (j == 0 ? A.rhs : A.Sci + (size_t)S.rhs_col[j] * nc6)[e];
      L.x[j][idx] = 0.0; L.p[j][idx] = 0.0; L.w[j][idx] = 0.0; L.r[j][idx] = b; v = b * b;
      Pcur[j * nc6 + e] = 0.0;
    }
    warp_acc(S, v, j);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nrhs * nw; i += PCG2_THREADS) {
    const int j = i / nw, m = i % nw;
    double cv = 0; for (int idx = 0; idx < ne; ++idx) cv += L.wg[m][idx] * L.r[j][idx];
    if (own) { Cg[(size_t)j * nco + g * nw + m] = cv; AW[(size_t)j * nco + g * nw + m] = 0.0; }
  }
  vsum_end(grid, S, nrhs, A.part);
  if (threadIdx.x < nrhs) { const int j = threadIdx.x; S.bb[j] = S.tot[j]; S.done[j] = !(S.tot[j] > 0.0); S.alpha[j] = 0; S.beta[j] = 0; S.rz[j] = 0; }
  if (threadIdx.x == 0) { S.worst = 0; S.all_done = 0; }
  for (int i = threadIdx.x; i < nrhs * nco; i += PCG2_THREADS) sCv[(i / nco) * PCG3_NCO_MAX + i % nco] = __ldcg(Cg + (size_t)(i / nco) * nco + i % nco);
  __syncthreads();
  int it = 0;
  unsigned long long tlast = P.tim ? gtimer() : 0ull;
  for (;;) {
    // ================================================================= [A]
    vsum_begin(S, 2 * nrhs);
    { // coarse step: this aggregate's rows of Einv go to registers while Wa'w of all aggregates arrives
      double ev[PCG3_NCO_MAX / 32];
      const bool yrow = own && wib < nw && nco > 0;
      if (yrow) {
        const double *er = P.Einv + (size_t)(g * nw + wib) * nco;
        #pragma unroll
        for (int q = 0; q < PCG3_NCO_MAX / 32; ++q) { const int k = lane + 32 * q; ev[q] = k < nco ? __ldcg(er + k) : 0.0; }
      }
      if (it > 0) {                                              // all loads in flight before the first use: ONE L2 round trip
        double awv[PCG5_NR][PCG3_NCO_MAX / PCG2_THREADS];
        #pragma unroll
        for (int j = 0; j < PCG5_NR; ++j)
          #pragma unroll
          for (int q = 0; q < PCG3_NCO_MAX / PCG2_THREADS; ++q) { const int k2 = threadIdx.x + PCG2_THREADS * q; awv[j][q] = (j < nrhs && k2 < nco) ? __ldcg(AW + (size_t)j * nco + k2) : 0.0; }
        #pragma unroll
        for (int j = 0; j < PCG5_NR; ++j)
          #pragma unroll
          for (int q = 0; q < PCG3_NCO_MAX / PCG2_THREADS; ++q) { const int k2 = threadIdx.x + PCG2_THREADS * q; if (j < nrhs && k2 < nco) sCv[j * PCG3_NCO_MAX + k2] -= S.alpha[j] * awv[j][q]; }
      }
      __syncthreads();
      PCG_LAP(0);
      if (yrow) {
        double acc[PCG5_NR] = {0, 0, 0, 0};
        #pragma unroll
        for (int q = 0; q < PCG3_NCO_MAX / 32; ++q) { const int k = lane + 32 * q;
          if (k < nco) {
            #pragma unroll
            for (int j = 0; j < PCG5_NR; ++j) if (j < nrhs) acc[j] += ev[q] * sCv[j * PCG3_NCO_MAX + k]; } }
        #pragma unroll
        for (int j = 0; j < PCG5_NR; ++j) {
          double v = acc[j]; for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
          if (lane == 0 && j < nrhs) L.y[wib][j] = v;
        }
      }
      __syncthreads();
      PCG_LAP(1);
    }
    // local: x += alpha p ; r -= alpha w ; |r|^2
    for (int t = threadIdx.x; t < nrhs * PCG5_ST; t += PCG2_THREADS) {
      const int j = t / PCG5_ST, idx = t % PCG5_ST;
      double rr = 0;
      if (idx < ne && !S.done[j]) {
        const double al = S.alpha[j];
        L.x[j][idx] += al * L.p[j][idx];
        const double rn = L.r[j][idx] - al * L.w[j][idx]; L.r[j][idx] = rn; rr = rn * rn;
      }
      warp_acc(S, rr, nrhs + j);
    }
    __syncthreads();
    // local: z = Minv r + Wa y ; r'z ; z of the own cameras is published for the neighbours' SpMV
    for (int t = threadIdx.x; t < nrhs * PCG5_ST; t += PCG2_THREADS) {
      const int j = t / PCG5_ST, idx = t % PCG5_ST;
      double rz = 0;
      if (idx < ne && !S.done[j]) {
        const int ci = idx / 6, k = idx % 6;
        const double *M = L.minv[ci] + 6 * k, *rb = L.r[j] + 6 * ci;
        double zz = M[0] * rb[0] + M[1] * rb[1] + M[2] * rb[2] + M[3] * rb[3] + M[4] * rb[4] + M[5] * rb[5];
        if (nco > 0) for (int m = 0; m < nw; ++m) zz += L.wg[m][idx] * L.y[m][j];
        L.z[j][idx] = zz; rz = zz * rb[k];
        A.Zv[j * nc6 + 6 * (size_t)L.cams[ci] + k] = zz;
      }
      warp_acc(S, rz, j);
    }
    PCG_LAP(2);
    vsum_end(grid, S, 2 * nrhs, A.part);
    PCG_LAP(3);
    if (threadIdx.x < nrhs) { const int j = threadIdx.x; if (!S.done[j]) { const double rzn = S.tot[j]; S.beta[j] = it == 0 ? 0.0 : rzn / S.rz[j]; S.rz[j] = rzn; } }
    __syncthreads();
    if (threadIdx.x == 0) {
      int ad = 1; double wmax = 0;
      for (int j = 0; j < nrhs; ++j) if (!S.done[j]) { const double rel2 = S.tot[nrhs + j] / S.bb[j]; wmax = fmax(wmax, rel2); if (!(rel2 > A.tol * A.tol)) S.done[j] = 1; else ad = 0; }
      S.all_done = ad; if (it > 0) S.worst = wmax;
    }
    __syncthreads();
    if (S.all_done || it >= A.max_iter) break;
    // ================================================================= [B]  w = Scc (z + beta p) ; p'w ; Wa' w
    vsum_begin(S, nrhs);
    for (int i = threadIdx.x; i < NWARP * PCG5_NR * MAXW; i += PCG2_THREADS) (&L.aw[0][0][0])[i] = 0.0;
    // p = z + beta p of every neighbour camera, gathered ONCE per iteration (each is used by up to ncam rows)
    { constexpr int NQ = (PCG5_NB * PCG5_NR * 3 + PCG2_THREADS - 1) / PCG2_THREADS;
      const int total = L.nnb * nrhs * 3, per = nrhs * 3;
      double2 zz[NQ], pp[NQ];
      #pragma unroll
      for (int q = 0; q < NQ; ++q) {                              // every load issued before the first use: ONE L2 round trip
        const int t = threadIdx.x + PCG2_THREADS * q;
        zz[q] = make_double2(0.0, 0.0); pp[q] = zz[q];
        if (t < total) {
          const int u = t / per, rj = t - u * per, j = rj / 3, h = rj - 3 * j;
          if (!S.done[j]) {
            const size_t off = (size_t)j * nc6 + 6 * (size_t)L.nbl[u] + 2 * h;
            zz[q] = __ldcg(reinterpret_cast<const double2 *>(A.Zv + off)); pp[q] = __ldcg(reinterpret_cast<const double2 *>(Pcur + off));
          }
        }
      }
      #pragma unroll
      for (int q = 0; q < NQ; ++q) {
        const int t = threadIdx.x + PCG2_THREADS * q;
        if (t < total) {
          const int u = t / per, rj = t - u * per, j = rj / 3, h = rj - 3 * j;
          if (!S.done[j]) { const double bt = S.beta[j]; sPN[u * PCG5_PS + j * 6 + 2 * h] = zz[q].x + bt * pp[q].x; sPN[u * PCG5_PS + j * 6 + 2 * h + 1] = zz[q].y + bt * pp[q].y; }
        }
      } }
    PCG_LAP(6);
    __syncthreads();
    for (int ci = wib; ci < ncam; ci += NWARP) {
      const int a = L.cams[ci];
      double acc[PCG5_NR][6];
      #pragma unroll
      for (int j = 0; j < PCG5_NR; ++j)
        #pragma unroll
        for (int i = 0; i < 6; ++i) acc[j][i] = 0.0;
      const int nbr = L.rowstart[ci + 1] - L.rowstart[ci];
      for (int e = lane; e < nbr; e += 32) {
        const int lb = L.rowstart[ci] + e;
        double b[36]; int lc;
        if (lb < nb_cache) {
          const double *blk = sS + (size_t)lb * PCG5_BS;
          #pragma unroll
          for (int i = 0; i < 36; ++i) b[i] = blk[i];
          lc = sCol[lb];
        } else {
          const double *blk = A.Scc + 36 * (size_t)(L.rowptr0[ci] + e);
          #pragma unroll
          for (int i = 0; i < 9; ++i) ldg256(blk + 4 * i, b[4 * i], b[4 * i + 1], b[4 * i + 2], b[4 * i + 3]);
          lc = blk_lcol[L.rowptr0[ci] + e];
        }
        const double *pn = sPN + lc * PCG5_PS;
        #pragma unroll
        for (int j = 0; j < PCG5_NR; ++j) {
          if (j < nrhs && !S.done[j]) {
            double xv[6];
            #pragma unroll
            for (int k2 = 0; k2 < 6; ++k2) xv[k2] = pn[j * 6 + k2];
            #pragma unroll
            for (int i = 0; i < 6; ++i)
              #pragma unroll
              for (int k2 = 0; k2 < 6; ++k2) acc[j][i] += b[i * 6 + k2] * xv[k2];
          }
        }
      }
      // row totals -> lane 0 -> shared memory, then the per-element tail runs on 24 / 28 lanes instead of one
      #pragma unroll
      for (int j = 0; j < PCG5_NR; ++j) {
        if (j < nrhs && !S.done[j]) {
          #pragma unroll
          for (int i = 0; i < 6; ++i) { double v = acc[j][i]; for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o); if (lane == 0) L.wrow[wib][j][i] = v; }
        }
      }
      __syncwarp();
      if (lane < PCG5_NR * 6) {                                   // lane = (j, i): p = z + beta p, w, p'w partial
        const int j = lane / 6, i = lane - 6 * j;
        double d = 0.0;
        if (j < nrhs && !S.done[j]) {
          const double bt = S.beta[j], wv = L.wrow[wib][j][i];
          const double pv = L.z[j][6 * ci + i] + bt * L.p[j][6 * ci + i];
          L.p[j][6 * ci + i] = pv; L.w[j][6 * ci + i] = wv; d = wv * pv;
          Pnext[(size_t)j * nc6 + 6 * (size_t)a + i] = pv;
        }
        L.drow[wib][lane] = d;
      }
      __syncwarp();
      if (lane < PCG5_NR) { const int j = lane; if (j < nrhs && !S.done[j]) { double d = 0; for (int i = 0; i < 6; ++i) d += L.drow[wib][6 * j + i]; S.wpart[wib][j] += d; } }
      if (lane < PCG5_NR * MAXW) {                                // lane = (j, m): Wa' w of this row
        const int j = lane / MAXW, m = lane - MAXW * j;
        if (j < nrhs && m < nw && !S.done[j]) { double t2 = 0; for (int i = 0; i < 6; ++i) t2 += L.wg[m][6 * ci + i] * L.wrow[wib][j][i]; L.aw[wib][j][m] += t2; }
      }
      __syncwarp();
    }
    PCG_LAP(7);
    __syncthreads();
    if (own)
      for (int i = threadIdx.x; i < nrhs * nw; i += PCG2_THREADS) {
        const int j = i / nw, m = i % nw;
        if (!S.done[j]) { double t2 = 0; for (int w2 = 0; w2 < NWARP; ++w2) t2 += L.aw[w2][j][m]; AW[(size_t)j * nco + g * nw + m] = t2; }
      }
    PCG_LAP(4);
    vsum_end(grid, S, nrhs, A.part);              // its grid.sync also publishes p of the own cameras and Wa'w
    PCG_LAP(5);
    { double *t2 = Pcur; Pcur = Pnext; Pnext = t2; }
    if (threadIdx.x < nrhs) { const int j = threadIdx.x; S.alpha[j] = S.done[j] ? 0.0 : S.rz[j] / S.tot[j]; }
    __syncthreads();
    ++it;
  }
  // ---- the solutions leave shared memory; then the border as in v3
  for (int t = threadIdx.x; t < nrhs * PCG5_ST; t += PCG2_THREADS) { const int j = t / PCG5_ST, idx = t % PCG5_ST; if (idx < ne) A.X[j * nc6 + 6 * (size_t)L.cams[idx / 6] + idx % 6] = L.x[j][idx]; }
  grid.sync();
  const int k = nrhs - 1;
  if (k > 0) {
    for (int a = 0; a < k; ++a) {
      vsum_begin(S, k + 1);
      const double *row = A.Sci + (size_t)S.rhs_col[1 + a] * nc6;
      for (int b = 0; b <= k; ++b) {
        const double *x = A.X + (size_t)(b == k ? 0 : 1 + b) * nc6;
        double v = 0; for (size_t i = tid; i < nc6; i += nt) v += row[i] * __ldcg(x + i);
        warp_acc(S, v, b);
      }
      vsum_end(grid, S, k + 1, A.part);
      if (threadIdx.x <= k) {
        const int b = threadIdx.x;
        if (b < k) S.T[a][b] = A.Sii[(size_t)S.rhs_col[1 + a] * A.ni8 + S.rhs_col[1 + b]] - S.tot[b];
        else S.T[a][k] = A.rhs[nc6 + S.rhs_col[1 + a]] - S.tot[k];
      }
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      for (int a = 0; a < k; ++a) for (int b = a + 1; b < k; ++b) { const double m = 0.5 * (S.T[a][b] + S.T[b][a]); S.T[a][b] = m; S.T[b][a] = m; }
      for (int c = 0; c < k; ++c) {
        int piv = c; for (int r2 = c + 1; r2 < k; ++r2) if (fabs(S.T[r2][c]) > fabs(S.T[piv][c])) piv = r2;
        if (piv != c) for (int q = 0; q <= k; ++q) { const double t2 = S.T[c][q]; S.T[c][q] = S.T[piv][q]; S.T[piv][q] = t2; }
        for (int r2 = c + 1; r2 < k; ++r2) { const double f = S.T[r2][c] / S.T[c][c]; for (int q = c; q <= k; ++q) S.T[r2][q] -= f * S.T[c][q]; }
      }
      for (int c = k - 1; c >= 0; --c) { double sacc = S.T[c][k]; for (int q = c + 1; q < k; ++q) sacc -= S.T[c][q] * S.zi[q]; S.zi[c] = sacc / S.T[c][c]; }
    }
    __syncthreads();
  }
  for (size_t i = tid; i < nc6; i += nt) { double v = __ldcg(A.X + i); for (int a = 0; a < k; ++a) v -= __ldcg(A.X + (size_t)(1 + a) * nc6 + i) * S.zi[a]; A.z[i] = v; }
  for (int q = tid; q < A.ni8; q += nt) { double v = 0; for (int a = 0; a < k; ++a) if (S.rhs_col[1 + a] == q) v = S.zi[a]; A.z[nc6 + q] = v; }
  if (tid == 0) { A.out[0] = (double)it; A.out[1] = sqrt(S.worst); A.out[2] = sqrt(S.bb[0]); }
}

// ------------------------------------------------------------------------------ back substitution
// y_pt = Einv (Etb - sum_obs EtFc z_c + EtFi z_i) ; step = -y  (levenberg_marquardt_strategy.cc:120)
__global__ void backsub_kernel(const double *__restrict__ Jp, const double *__restrict__ Jc, const double *__restrict__ Ji,
                               const double *__restrict__ Etb, const double *__restrict__ Einv, const int *__restrict__ obs_pose,
                               const int *__restrict__ obs_intr, const int *__restrict__ pt_start, int n_points, int n_poses, long long n, int kiu,
                               const double *__restrict__ z, int pts_free, double *__restrict__ step_pt) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x; if (j >= n_points) return;
  if (!pts_free || pt_start[j] == pt_start[j + 1]) { step_pt[3 * j] = step_pt[3 * j + 1] = step_pt[3 * j + 2] = 0.0; return; }
  double b0 = Etb[3 * (size_t)j], b1 = Etb[3 * (size_t)j + 1], b2 = Etb[3 * (size_t)j + 2];
  for (long long o = pt_start[j]; o < pt_start[j + 1]; ++o) {
    const double *zc = z + 6 * obs_pose[o]; const double *zi = z + 6 * n_poses + KI * obs_intr[o];
    double f0 = 0, f1 = 0;                                    // F z for the two residual rows
    #pragma unroll
    for (int k = 0; k < 6; ++k) { f0 += Jc[k * n + o] * zc[k]; f1 += Jc[(6 + k) * n + o] * zc[k]; }
    #pragma unroll
    for (int k = 0; k < KI; ++k) if (k < kiu) { f0 += Ji[k * n + o] * zi[k]; f1 += Ji[(KI + k) * n + o] * zi[k]; }
    b0 -= Jp[0 * n + o] * f0 + Jp[3 * n + o] * f1; b1 -= Jp[1 * n + o] * f0 + Jp[4 * n + o] * f1; b2 -= Jp[2 * n + o] * f0 + Jp[5 * n + o] * f1;
  }
  const double *I = Einv + 9 * (size_t)j;
  step_pt[3 * j] = -(I[0] * b0 + I[1] * b1 + I[2] * b2); step_pt[3 * j + 1] = -(I[3] * b0 + I[4] * b1 + I[5] * b2); step_pt[3 * j + 2] = -(I[6] * b0 + I[7] * b1 + I[8] * b2);
}
// Coalesced form (default): thread per OBSERVATION computes its E'F z 3-vector with contiguous component-major
// loads; observations are sorted by landmark, so a segmented warp scan sums each landmark's run and the last lane
// of a run adds it to acc[landmark] (one atomic per landmark per warp).  backsub_point_kernel finishes
// step = -Einv (Etb - acc) in place.  The thread-per-landmark kernel above re-fetched every sector ~4x (280 us).
__global__ void backsub_obs_kernel(const double *__restrict__ Jp, const double *__restrict__ Jc, const double *__restrict__ Ji,
                                   const int *__restrict__ obs_pose, const int *__restrict__ obs_intr, const int *__restrict__ obs_pt,
                                   int n_poses, long long n, int kiu, const double *__restrict__ z, double *__restrict__ acc) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool valid = o < n;
  int j = -1; double v0 = 0, v1 = 0, v2 = 0;
  if (valid) {
    j = obs_pt[o];
    const double *zc = z + 6 * obs_pose[o]; const double *zi = z + 6 * n_poses + KI * obs_intr[o];
    double f0 = 0, f1 = 0;
    #pragma unroll
    for (int k = 0; k < 6; ++k) { f0 += __ldcs(Jc + k * n + o) * zc[k]; f1 += __ldcs(Jc + (6 + k) * n + o) * zc[k]; }
    #pragma unroll
    for (int k = 0; k < KI; ++k) if (k < kiu) { f0 += __ldcs(Ji + k * n + o) * zi[k]; f1 += __ldcs(Ji + (KI + k) * n + o) * zi[k]; }
    v0 = __ldcs(Jp + 0 * n + o) * f0 + __ldcs(Jp + 3 * n + o) * f1;
    v1 = __ldcs(Jp + 1 * n + o) * f0 + __ldcs(Jp + 4 * n + o) * f1;
    v2 = __ldcs(Jp + 2 * n + o) * f0 + __ldcs(Jp + 5 * n + o) * f1;
  }
  #pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int jv = __shfl_up_sync(0xffffffffu, j, off);
    const double a0 = __shfl_up_sync(0xffffffffu, v0, off), a1 = __shfl_up_sync(0xffffffffu, v1, off), a2 = __shfl_up_sync(0xffffffffu, v2, off);
    if (lane >= off && jv == j) { v0 += a0; v1 += a1; v2 += a2; }
  }
  const int jn = __shfl_down_sync(0xffffffffu, j, 1);
  if (valid && (lane == 31 || jn != j)) { atomicAdd(acc + 3 * (size_t)j, v0); atomicAdd(acc + 3 * (size_t)j + 1, v1); atomicAdd(acc + 3 * (size_t)j + 2, v2); }
}
__global__ void backsub_point_kernel(const double *__restrict__ Etb, const double *__restrict__ Einv, const int *__restrict__ pt_start, int n_points,
                                     int pts_free, double *__restrict__ step_pt /* in: acc, out: step */) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x; if (j >= n_points) return;
  if (!pts_free || pt_start[j] == pt_start[j + 1]) { step_pt[3 * j] = step_pt[3 * j + 1] = step_pt[3 * j + 2] = 0.0; return; }
  const double b0 = Etb[3 * (size_t)j] - step_pt[3 * j], b1 = Etb[3 * (size_t)j + 1] - step_pt[3 * j + 1], b2 = Etb[3 * (size_t)j + 2] - step_pt[3 * j + 2];
  const double *I = Einv + 9 * (size_t)j;
  step_pt[3 * j] = -(I[0] * b0 + I[1] * b1 + I[2] * b2); step_pt[3 * j + 1] = -(I[3] * b0 + I[4] * b1 + I[5] * b2); step_pt[3 * j + 2] = -(I[6] * b0 + I[7] * b1 + I[8] * b2);
}

__global__ void negate_kernel(const double *__restrict__ z, int n, double *__restrict__ step) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) step[i] = -z[i]; }

// model_cost_change partials: - m . (r + m/2), m = J step    (trust_region_minimizer.cc:402-405)
constexpr int MODEL_THREADS = 128;
__global__ void __launch_bounds__(MODEL_THREADS) model_kernel(const double *__restrict__ r, const double *__restrict__ Jp, const double *__restrict__ Jc, const double *__restrict__ Ji,
                             const int *__restrict__ obs_pose, const int *__restrict__ obs_intr, const int *__restrict__ obs_pt, long long n, int n_poses, int kiu,
                             const double *__restrict__ step_pt, const double *__restrict__ step_red, double *__restrict__ part) {
  __shared__ double sh[MODEL_THREADS / 32];
  const long long o = (long long)blockIdx.x * MODEL_THREADS + threadIdx.x;
  double v = 0;
  if (o < n) {
    const double *sp = step_pt + 3 * obs_pt[o], *sc = step_red + 6 * obs_pose[o], *si = step_red + 6 * n_poses + KI * obs_intr[o];
    #pragma unroll
    for (int row = 0; row < 2; ++row) {
      double m = 0;
      #pragma unroll
      for (int k = 0; k < 3; ++k) m += Jp[(row * 3 + k) * n + o] * sp[k];
      #pragma unroll
      for (int k = 0; k < 6; ++k) m += Jc[(row * 6 + k) * n + o] * sc[k];
      #pragma unroll
      for (int k = 0; k < KI; ++k) if (k < kiu) m += Ji[(row * KI + k) * n + o] * si[k];
      v += -m * (r[row * n + o] + m / 2.0);
    }
  }
  const double t = block_sum<MODEL_THREADS>(v, sh);
  if (threadIdx.x == 0) part[blockIdx.x] = t;
}

// candidate = x + step * scale on free coordinates; partials of |delta|^2 (ambient) and |x|^2


// ------------------------------------------------------------------------------ mid-size reduced systems: explicit inverse
// Between DENSE_MAX and DENSE2_MAX = 640 unknowns (36 .. ~105 cameras) the reduced system is still too small for the PCG to be
// anything but latency (21 iterations of 20 us at 50 cameras) and too large for one CTA's shared memory: it is assembled
// dense in global memory, inverted in place by the blocked Gauss-Jordan kernel that already inverts the coarse operator
// (coarse_invert_kernel: all SMs, one rank-32 update of every tile per pivot block) and applied to the right-hand side.
__global__ void dense_assemble_kernel(const double *__restrict__ Scc, const int *__restrict__ brow, const int *__restrict__ cols, int nnzb,
                                      const double *__restrict__ Sci, const double *__restrict__ Sii, int n_poses, int ni8, double *__restrict__ A) {
  const int nc6 = 6 * n_poses, n = nc6 + ni8;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nt = (long long)gridDim.x * blockDim.x;
  for (long long t = tid; t < 36ll * nnzb; t += nt) {                 // camera-camera blocks (both triangles are stored)
    const int e = (int)(t / 36), k = (int)(t % 36);
    A[(size_t)(6 * brow[e] + k / 6) * n + 6 * cols[e] + k % 6] = Scc[t];
  }
  for (long long t = tid; t < (long long)ni8 * nc6; t += nt) {        // border and its transpose
    const int q = (int)(t / nc6), k = (int)(t % nc6);
    const double v = Sci[t];
    A[(size_t)(nc6 + q) * n + k] = v; A[(size_t)k * n + nc6 + q] = v;
  }
  for (long long t = tid; t < (long long)ni8 * ni8; t += nt) A[(size_t)(nc6 + t / ni8) * n + nc6 + t % ni8] = Sii[t];
}
// z = Ainv rhs (one warp per row)
__global__ void dense_apply_kernel(const double *__restrict__ Ainv, const double *__restrict__ rhs, int n, double *__restrict__ z, double *__restrict__ out) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row == 0 && lane == 0) { out[0] = 0.0; out[1] = 0.0; out[2] = 0.0; }
  if (row >= n) return;
  const double *a = Ainv + (size_t)row * n;
  double v = 0.0;
  for (int k = lane; k < n; k += 32) v += a[k] * rhs[k];
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) z[row] = v;
}

// ------------------------------------------------------------------------------ merged small launches
// The LM loop used to issue ~50 launches per iteration, half of them a few microseconds of work on one vector each
// (three parameter blocks x {update, two reductions}, three gradient maxima, three LM diagonals, four memsets).  One
// launch per group, blockIdx.y selecting the parameter block; the arithmetic and the reduction orders are unchanged.
struct UpdSeg { const double *x, *step, *scale; int n, stride; unsigned uniform_mask; const unsigned *block_mask; double *cand; };
struct Upd3 { UpdSeg s[3]; };
// part[seg][gridDim.x] = |step * scale|^2 partials, part[3 + seg][gridDim.x] = |x|^2 partials (seg: points, poses, intrinsics)
__global__ void update3_kernel(Upd3 U, double *__restrict__ part) {
  __shared__ double sh[8];
  const UpdSeg &S = U.s[blockIdx.y];
  double ds = 0, xs = 0;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < S.n; i += gridDim.x * 256) {
    const int blk = i / S.stride, k = i % S.stride;
    const unsigned m = S.block_mask ? S.block_mask[blk] : S.uniform_mask;
    const double xv = S.x[i];
    double d = 0;
    if ((m >> k) & 1) d = S.step[i] * S.scale[i];
    S.cand[i] = xv + d;
    ds += d * d;
    if (m != 0) xs += xv * xv;                                // constant blocks are not part of the reduced program
  }
  const double a = block_sum<256>(ds, sh); const double b = block_sum<256>(xs, sh);
  if (threadIdx.x == 0) { part[blockIdx.y * gridDim.x + blockIdx.x] = a; part[(3 + blockIdx.y) * gridDim.x + blockIdx.x] = b; }
}
// out[b] = sum of part[b][0..n) (block b; same order as reduce_partials_kernel)
__global__ void reduce_multi_kernel(const double *__restrict__ part, int n, double *__restrict__ out) {
  __shared__ double sh[32];
  const double *p = part + (size_t)blockIdx.x * n;
  double v = 0; for (int i = threadIdx.x; i < n; i += 1024) v += p[i];
  const double t = block_sum<1024>(v, sh);
  if (threadIdx.x == 0) out[blockIdx.x] = t;
}
struct Vec3Seg { const double *a, *b; int n; };
struct Vec3 { Vec3Seg s[3]; };
__global__ void grad_max3_kernel(Vec3 V, double *__restrict__ part) {          // a = gradient, b = scale
  __shared__ double sh[8];
  const Vec3Seg &S = V.s[blockIdx.y];
  double m = 0;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < S.n; i += gridDim.x * 256) m = fmax(m, fabs(S.a[i] / S.b[i]));
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) { for (int i = 1; i < 8; ++i) m = fmax(m, sh[i]); part[blockIdx.y * gridDim.x + blockIdx.x] = m; }
}
struct Diag3Seg { const double *diag; double *lmD; int n; };
struct Diag3 { Diag3Seg s[3]; };
// lmD = sqrt(clamp(diag, lo, hi) / radius)   (levenberg_marquardt_strategy.cc:75-87)
__global__ void lm_diag3_kernel(Diag3 D, double lo, double hi, double radius) {
  const Diag3Seg &S = D.s[blockIdx.y];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S.n; i += gridDim.x * blockDim.x) S.lmD[i] = sqrt(fmin(fmax(S.diag[i], lo), hi) / radius);
}
struct Zero4 { double *p[4]; long long n[4]; };
__global__ void zero4_kernel(Zero4 Z) {
  double *p = Z.p[blockIdx.y]; const long long n = Z.n[blockIdx.y];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = 0.0;
}

}}  // namespace omvg::ba
