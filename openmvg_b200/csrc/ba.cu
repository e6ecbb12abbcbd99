// ba.cu — host side of the bundle-adjustment hot path: problem packing, device structures and the
// Levenberg-Marquardt controller that mirrors Ceres 1.13's TrustRegionMinimizer +
// LevenbergMarquardtStrategy (reference: src/third_party/ceres-solver/internal/ceres/
// trust_region_minimizer.cc:66-119,226-279,355-424,667-786; levenberg_marquardt_strategy.cc:65-160;
// trust_region_step_evaluator.cc:51-59) as configured by openMVG
// (src/openMVG/sfm/sfm_data_BA_ceres.cpp:242-253,275-305,321-344,394-395,477-493).
// All arithmetic runs in the kernels of ba_kernels.cuh; the host only takes the accept/reject and
// termination decisions from a handful of scalars read back once per LM iteration.
#include "ba_kernels.cuh"
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <memory>
#include <chrono>
#include <vector>

using namespace omvg;
using namespace omvg::ba;

namespace {

enum Slot { S_COST = 0, S_MODEL, S_STEP2_PT, S_STEP2_POSE, S_STEP2_INTR, S_X2_PT, S_X2_POSE, S_X2_INTR,
            S_GMAX_PT, S_GMAX_CAM, S_GMAX_INTR, S_PCG_IT, S_PCG_RES, S_PCG_B, S_CAND_COST, S_COUNT = 16 };

int model_nparams(int m) {     // size of the Ceres parameter block = getParams().size()
  switch (m) { case 1: return 3; case 2: return 4; case 3: return 6; case 4: return 8; case 5: return 7; case OMVG_CAMERA_SPHERICAL: return 0; default: return -1; }
}
int model_ndata(int m) { return m == OMVG_CAMERA_SPHERICAL ? 2 : model_nparams(m); }   // doubles of the slot the kernels read

template <typename T> struct DevBuf {
  T *p = nullptr; size_t n = 0;
  int alloc(size_t count) { release(); n = count; if (!count) return OMVG_OK; OMVG_CUDA(pool_malloc(reinterpret_cast<void **>(&p), count * sizeof(T))); return OMVG_OK; }
  void release() { if (p) pool_free(p); p = nullptr; n = 0; }
  ~DevBuf() { release(); }
};

}  // namespace

// stream / events / pinned scalars of a context: creating and destroying them costs ~2.5 ms per Adjust, so
// released sets are kept per device and reused (omvg_trim_cache() frees them)
struct CtxRes { cudaStream_t stream = nullptr, stream2 = nullptr; cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr}; double *h_scal = nullptr; };
struct ResPool { std::mutex mu; std::vector<CtxRes> free_[16]; };
static ResPool &res_pool() { static ResPool p; return p; }

struct omvg_ba_ctx {
  int device = 0, n_sms = 0;
  cudaStream_t stream = nullptr, stream2 = nullptr;   // stream2: payload upload under the structure build (omvg_ba_create)
  cudaEvent_t ev_up = nullptr;
  int nc = 0, ni = 0, np = 0, nv = 0; long long no = 0;
  int ni8 = 0, nred = 0, words = 0, nnzb = 0, eval_blocks = 0, eval_grid = 0, kiu = KI, gj_grid = 0, ics_chunks = 64;
  std::vector<int> perm;                    // sorted position -> caller's observation index (fetched on first use)
  DevBuf<int> d_perm;
  std::vector<int> h_intr_model;
  // parameters: [0] current, [1] candidate, init = copy at create
  DevBuf<double> pose[2], intr[2], pt[2], pose0, intr0, pt0;
  DevBuf<int> intr_model, obs_pose, obs_intr, obs_pt, pt_start, cam_start, cam_obs;
  DevBuf<double> obs_xy;
  DevBuf<double> r, Jp, Jc, Ji, camR[2], camdR, camrec[2];
  DevBuf<double> sc_pt, sc_cam, sc_intr, diag_pt, diag_cam, diag_intr, lmD_pt, lmD_cam, lmD_intr, g_cam, g_intr;
  DevBuf<double> EtE, Etb, EtFi, FtF, FiFi, Einv, step_pt, step_red;
  DevBuf<unsigned char> pt_single;
  DevBuf<unsigned> bitmap, intr_mask; DevBuf<int> wprefix, rowptr, cols;
  DevBuf<double> Scc, Sci, Sii, rhs, Minv_c, Minv_i, work_i;
  DevBuf<double> z, res, pvec, w, zeta, pcg_part;
  DevBuf<double> gW, bX, bR, bP, bW, bZ, pcg2_part;   // two-level block-PCG workspaces
  DevBuf<int> agg_of, agg_start, agg_cams, brow, nb_start, nb_list; DevBuf<unsigned short> blk_lcol; int nb_max = 0;   // neighbour lists of the aggregates (pcg5)
  DevBuf<double> cE, cT, cCv, cYv, cCv2, cAW, bP2; int ng = 0, agg_maxsize = 0;   // cE: coarse operator, inverted in place
  DevBuf<double> dA, dT;                             // dense reduced system / scratch of its in-place inverse (mid-size scenes)
  DevBuf<double> part, part2, part3, icol_part, scal;
  DevBuf<int> fail;
  DevBuf<unsigned long long> pcg_tim;
  DevBuf<double> corner_rep;
  DevBuf<double> GE;                        // per observation { Einv E'Fc, E'Fc } of the split Schur step
  DevBuf<unsigned long long> pairs; DevBuf<int> gstart, gblk, gblkT; int nwork = 0;   // pair lists of schur_gather_kernel
  // optional extensions: GCP weights / flags / fixed landmarks, pose-centre priors
  DevBuf<double> obs_w; DevBuf<unsigned char> obs_flags, pt_fixed; DevBuf<unsigned> pt_mask;
  DevBuf<unsigned char> pt_gcp, pt_removed, pt_now; DevBuf<unsigned> rej_bits; DevBuf<unsigned long long> rej_cnt;   // outlier rejection (omvg_ba_reject_outliers)
  bool reject_ready = false;
  int n_slow = 0;                           // landmarks left to the per-observation Schur kernel
  bool has_ext = false; int npri = 0; double prior_huber_a = 0; DevBuf<int> prior_pose; DevBuf<double> prior_center, prior_weight, rP, JP;
  double *h_scal = nullptr;                 // pinned
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evj0 = nullptr, evj1 = nullptr;
  long long launches = 0;
};

namespace {

#define LAUNCH_CHECK() OMVG_CUDA(cudaGetLastError())

// OMVG_BA_TIMING=1: host wall-clock of the phases around the solve (where the end-to-end time goes)
struct PhaseTimer {
  bool on = getenv("OMVG_BA_TIMING") != nullptr; const char *what;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  explicit PhaseTimer(const char *w) : what(w) {}
  void lap(const char *name) { if (!on) return; const auto t1 = std::chrono::steady_clock::now(); fprintf(stderr, "[omvg_ba timing] %s/%s %.3f ms\n", what, name, std::chrono::duration<double, std::milli>(t1 - t0).count()); t0 = t1; }
};

int validate(const omvg_ba_problem *P) {
  if (!P) return fail(OMVG_E_ARG, "null problem");
  if (P->n_poses < 1 || P->n_intrinsics < 1 || P->n_points < 1 || P->n_views < 1 || P->n_obs < 1) return fail(OMVG_E_ARG, "bad sizes (need >=1 pose, intrinsic, point, view, observation)");
  if (!P->poses || !P->intrinsics || !P->intr_model || (!P->points && P->n_points) || !P->view_pose || !P->view_intr) return fail(OMVG_E_ARG, "null array");
  if (P->n_obs && (!P->obs_view || !P->obs_point || !P->obs_xy)) return fail(OMVG_E_ARG, "null observation array");
  if (P->n_obs >= (1ll << 31)) return fail(OMVG_E_UNSUPPORTED, "more than 2^31 observations");
  for (int q = 0; q < P->n_intrinsics; ++q) if (model_nparams(P->intr_model[q]) < 0)
    return fail(OMVG_E_UNSUPPORTED, "camera model %d is not implemented on the GPU path", P->intr_model[q]);
  for (int v = 0; v < P->n_views; ++v)
    if (P->view_pose[v] < 0 || P->view_pose[v] >= P->n_poses || P->view_intr[v] < 0 || P->view_intr[v] >= P->n_intrinsics) return fail(OMVG_E_ARG, "view %d out of range", v);
  // (observation indices are range-checked on the device by setup_check_kernel)
  if (P->n_priors < 0 || (P->n_priors > 0 && (!P->prior_pose || !P->prior_center || !P->prior_weight))) return fail(OMVG_E_ARG, "bad pose-centre prior arrays");
  for (int k = 0; k < P->n_priors; ++k) if (P->prior_pose[k] < 0 || P->prior_pose[k] >= P->n_poses) return fail(OMVG_E_ARG, "prior %d: pose out of range", k);
  if (P->n_priors > 0 && !(P->prior_huber_a >= 0.0)) return fail(OMVG_E_ARG, "prior_huber_a must be >= 0");
  // the camera-pair bitmap takes n_poses^2 / 8 bytes (+ 4x that for its prefix counts): 131072 poses = 10.7 GB of the 180
  if (P->n_poses > 131072) return fail(OMVG_E_UNSUPPORTED, "more than 131072 poses (camera-pair bitmap)");
  // dense border Sci [8 n_intr][6 n_poses] doubles and corner Sii [8 n_intr]^2: keep both under 16 GB
  if ((double)P->n_intrinsics * 8.0 * ((double)P->n_poses * 6.0 + (double)P->n_intrinsics * 8.0) * 8.0 > 16e9)
    return fail(OMVG_E_UNSUPPORTED, "%d intrinsic groups x %d poses: the dense intrinsics border would exceed 16 GB", P->n_intrinsics, P->n_poses);
  return OMVG_OK;
}

template <typename T> int upload(DevBuf<T> &b, const T *h, size_t n, cudaStream_t s) {
  int rc = b.alloc(n); if (rc) return rc;
  if (n) OMVG_CUDA(cudaMemcpyAsync(b.p, h, n * sizeof(T), cudaMemcpyHostToDevice, s));
  return OMVG_OK;
}

int reduce_to(omvg_ba_ctx *c, const double *part, int n, int slot) {
  reduce_partials_kernel<<<1, 1024, 0, c->stream>>>(part, n, c->scal.p + slot); LAUNCH_CHECK(); c->launches++; return OMVG_OK;
}

struct Masks { unsigned pose_mask; std::vector<unsigned> intr_mask; int pts_free; };

// sfm_data_BA_ceres.cpp:275-305 (poses), 321-344 + Camera_Pinhole*.hpp subsetParameterization, 394-395
Masks make_masks(const omvg_ba_ctx *c, const omvg_ba_options *o) {
  Masks m; m.pts_free = o->structure_opt != 0;
  if (o->extrinsics_opt == 1) m.pose_mask = 0;
  else if (o->extrinsics_opt == 4) m.pose_mask = 0x38;      // ADJUST_TRANSLATION: rotation constant
  else if (o->extrinsics_opt == 2) m.pose_mask = 0x07;      // ADJUST_ROTATION: translation constant
  else m.pose_mask = 0x3f;
  m.intr_mask.assign(c->ni, 0);
  for (int q = 0; q < c->ni; ++q) {
    if (o->intrinsics_opt & 1) continue;                    // NONE
    const int k = model_nparams(c->h_intr_model[q]);
    unsigned mm = 0;
    for (int i = 0; i < k; ++i) {
      bool constant = (i == 0) ? !(o->intrinsics_opt & 2) : (i <= 2 ? !(o->intrinsics_opt & 4) : !(o->intrinsics_opt & 8));
      if (!constant) mm |= 1u << i;
    }
    m.intr_mask[q] = mm;
  }
  return m;
}

int eval_cost(omvg_ba_ctx *c, const omvg_ba_options *o, int which, int slot) {
  cam_prep_kernel<<<(c->nc + 127) / 128, 128, 0, c->stream>>>(c->pose[which].p, c->nc, c->camR[which].p, c->camdR.p, c->camrec[which].p); LAUNCH_CHECK();
  // NB: cam_prep overwrites camdR; the cost-only pass is always followed by a full evaluation before
  // camdR is read again (accepted step) or the current pose's camdR is not needed (J is materialised).
  EvalArgs A{}; A.poses = c->pose[which].p; A.intr = c->intr[which].p; A.pts = c->pt[which].p; A.camR = c->camR[which].p; A.camdR = c->camdR.p; A.camrec = c->camrec[which].p;
  A.obs_xy = c->obs_xy.p; A.intr_model = c->intr_model.p; A.obs_pose = c->obs_pose.p; A.obs_intr = c->obs_intr.p; A.obs_pt = c->obs_pt.p;
  A.n_obs = c->no; A.use_loss = o->use_loss; A.huber_a = o->huber_a; A.cost_partial = c->part.p;
  A.obs_w = c->obs_w.p; A.obs_flags = c->obs_flags.p; A.pt_fixed = c->pt_fixed.p;
  if (c->has_ext) eval_kernel<false, 8, true><<<c->eval_grid, EVAL_THREADS, 0, c->stream>>>(A);
  else eval_kernel<false, 8, false><<<c->eval_grid, EVAL_THREADS, 0, c->stream>>>(A);
  LAUNCH_CHECK();
  c->launches += 2;
  if (c->npri) {
    PriorArgs PA{}; PA.poses = c->pose[which].p; PA.camR = c->camR[which].p; PA.camdR = c->camdR.p; PA.prior_pose = c->prior_pose.p; PA.center = c->prior_center.p; PA.weight = c->prior_weight.p;
    PA.n = c->npri; PA.huber_a = c->prior_huber_a; PA.cost_out = c->part.p + c->eval_grid;
    prior_eval_kernel<false><<<1, PRIOR_THREADS, 0, c->stream>>>(PA); LAUNCH_CHECK(); c->launches++;
  }
  return reduce_to(c, c->part.p, c->eval_grid + (c->npri ? 1 : 0), slot);
}

int colsums(omvg_ba_ctx *c) {
  point_accum_kernel<<<(c->np + 127) / 128, 128, 0, c->stream>>>(c->Jp.p, c->Ji.p, c->r.p, c->pt_start.p, c->pt_single.p, c->np, c->no, c->kiu, c->EtE.p, c->Etb.p, c->EtFi.p, c->diag_pt.p); LAUNCH_CHECK();
  cam_colsum_kernel<<<c->nc, CCS_THREADS, 0, c->stream>>>(c->Jc.p, c->r.p, c->cam_start.p, c->cam_obs.p, c->nc, c->no, c->diag_cam.p, c->g_cam.p, c->FtF.p); LAUNCH_CHECK();
  if (c->npri) { prior_accum_kernel<<<(c->npri + 127) / 128, 128, 0, c->stream>>>(c->JP.p, c->rP.p, c->prior_pose.p, c->npri, c->diag_cam.p, c->g_cam.p, c->FtF.p); LAUNCH_CHECK(); c->launches++; }
  const int chunks = c->ics_chunks;
  { const dim3 g(chunks, c->ni);
    switch (c->kiu) {          // columns in use = max getParams() size over the intrinsic groups (3, 4, 6, 7 or 8)
      case 3: intr_colsum_kernel<3><<<g, ICS_THREADS, 0, c->stream>>>(c->Ji.p, c->r.p, c->obs_intr.p, c->no, chunks, c->icol_part.p); break;
      case 4: intr_colsum_kernel<4><<<g, ICS_THREADS, 0, c->stream>>>(c->Ji.p, c->r.p, c->obs_intr.p, c->no, chunks, c->icol_part.p); break;
      case 6: intr_colsum_kernel<6><<<g, ICS_THREADS, 0, c->stream>>>(c->Ji.p, c->r.p, c->obs_intr.p, c->no, chunks, c->icol_part.p); break;
      case 7: intr_colsum_kernel<7><<<g, ICS_THREADS, 0, c->stream>>>(c->Ji.p, c->r.p, c->obs_intr.p, c->no, chunks, c->icol_part.p); break;
      default: intr_colsum_kernel<8><<<g, ICS_THREADS, 0, c->stream>>>(c->Ji.p, c->r.p, c->obs_intr.p, c->no, chunks, c->icol_part.p); break;
    } }
  LAUNCH_CHECK();
  intr_colsum_final_kernel<<<c->ni * 72, 128, 0, c->stream>>>(c->icol_part.p, chunks, c->ni, c->diag_intr.p, c->g_intr.p, c->FiFi.p); LAUNCH_CHECK();
  c->launches += 4; return OMVG_OK;
}

// full evaluation at parameter set `which`: cost, corrected r and J (scaled), column sums, gradient max
int eval_jac(omvg_ba_ctx *c, const omvg_ba_options *o, const Masks &m, int which, bool &have_scale, bool time_it) {
  cam_prep_kernel<<<(c->nc + 127) / 128, 128, 0, c->stream>>>(c->pose[which].p, c->nc, c->camR[which].p, c->camdR.p, c->camrec[which].p); LAUNCH_CHECK();
  EvalArgs A{}; A.poses = c->pose[which].p; A.intr = c->intr[which].p; A.pts = c->pt[which].p; A.camR = c->camR[which].p; A.camdR = c->camdR.p; A.camrec = c->camrec[which].p;
  A.obs_xy = c->obs_xy.p; A.intr_model = c->intr_model.p; A.obs_pose = c->obs_pose.p; A.obs_intr = c->obs_intr.p; A.obs_pt = c->obs_pt.p;
  A.n_obs = c->no; A.use_loss = o->use_loss; A.huber_a = o->huber_a; A.r = c->r.p; A.Jp = c->Jp.p; A.Jc = c->Jc.p; A.Ji = c->Ji.p;
  A.cost_partial = c->part.p; A.kiu = c->kiu; A.pose_mask = m.pose_mask; A.intr_mask = c->intr_mask.p; A.pts_free = m.pts_free;
  A.obs_w = c->obs_w.p; A.obs_flags = c->obs_flags.p; A.pt_fixed = c->pt_fixed.p;
  if (have_scale) { A.sc_pt = c->sc_pt.p; A.sc_cam = c->sc_cam.p; A.sc_intr = c->sc_intr.p; }
  if (time_it) OMVG_CUDA(cudaEventRecord(c->evj0, c->stream));
  if (c->has_ext) eval_kernel<true, 4, true><<<c->eval_grid, EVAL_THREADS, 0, c->stream>>>(A);
  else eval_kernel<true, 4, false><<<c->eval_grid, EVAL_THREADS, 0, c->stream>>>(A);
  LAUNCH_CHECK();
  if (time_it) OMVG_CUDA(cudaEventRecord(c->evj1, c->stream));
  c->launches += 2;
  if (c->npri) {
    PriorArgs PA{}; PA.poses = c->pose[which].p; PA.camR = c->camR[which].p; PA.camdR = c->camdR.p; PA.prior_pose = c->prior_pose.p; PA.center = c->prior_center.p; PA.weight = c->prior_weight.p;
    PA.n = c->npri; PA.huber_a = c->prior_huber_a; PA.sc_cam = have_scale ? c->sc_cam.p : nullptr; PA.pose_mask = m.pose_mask; PA.rP = c->rP.p; PA.JP = c->JP.p; PA.cost_out = c->part.p + c->eval_grid;
    prior_eval_kernel<true><<<1, PRIOR_THREADS, 0, c->stream>>>(PA); LAUNCH_CHECK(); c->launches++;
  }
  int rc = reduce_to(c, c->part.p, c->eval_grid + (c->npri ? 1 : 0), S_COST); if (rc) return rc;
  if (!have_scale) {        // iteration 0: Jacobi scaling from the unscaled J (trust_region_minimizer.cc:239-253)
    if ((rc = colsums(c))) return rc;
    make_scale_kernel<<<(3 * c->np + 255) / 256, 256, 0, c->stream>>>(c->diag_pt.p, 3 * c->np, c->sc_pt.p); LAUNCH_CHECK();
    make_scale_kernel<<<(6 * c->nc + 255) / 256, 256, 0, c->stream>>>(c->diag_cam.p, 6 * c->nc, c->sc_cam.p); LAUNCH_CHECK();
    make_scale_kernel<<<(c->ni8 + 255) / 256, 256, 0, c->stream>>>(c->diag_intr.p, c->ni8, c->sc_intr.p); LAUNCH_CHECK();
    scale_J_kernel<<<(unsigned)((c->no + 255) / 256), 256, 0, c->stream>>>(c->Jp.p, c->Jc.p, c->Ji.p, c->obs_pose.p, c->obs_intr.p, c->obs_pt.p, c->no, c->kiu,
                                                                          c->sc_pt.p, c->sc_cam.p, c->sc_intr.p); LAUNCH_CHECK();
    if (c->npri) { prior_scale_kernel<<<(18 * c->npri + 127) / 128, 128, 0, c->stream>>>(c->JP.p, c->prior_pose.p, c->sc_cam.p, c->npri); LAUNCH_CHECK(); c->launches++; }
    c->launches += 4; have_scale = true;
  }
  if ((rc = colsums(c))) return rc;
  // gradient max norm (unscaled): g = J_scaled' r / scale
  const int gb = 64;
  Vec3 GV{}; GV.s[0] = Vec3Seg{c->Etb.p, c->sc_pt.p, m.pts_free ? 3 * c->np : 0}; GV.s[1] = Vec3Seg{c->g_cam.p, c->sc_cam.p, 6 * c->nc}; GV.s[2] = Vec3Seg{c->g_intr.p, c->sc_intr.p, c->ni8};
  grad_max3_kernel<<<dim3(gb, 3), 256, 0, c->stream>>>(GV, c->part2.p); LAUNCH_CHECK();     // part2[3][64], read back by read_scalars
  c->launches += 1;
  return OMVG_OK;
}

// gauge generators for the coarse space of the two-level preconditioner (needs camR/camdR of the CURRENT poses,
// i.e. must run right after eval_jac and before any cost-only evaluation of a candidate)
int make_gauge(omvg_ba_ctx *c, const Masks &m, int &nw) {
  unsigned gen = 0;
  if (m.pts_free) {
    if ((m.pose_mask & 0x38u) == 0x38u) gen |= 0x0fu;       // translations + scale move t
    if ((m.pose_mask & 0x07u) == 0x07u) gen |= 0x70u;       // rotations move the angle-axis
  }
  nw = __builtin_popcount(gen);
  if (nw == 0) return OMVG_OK;
  gauge_kernel<<<(c->nc + 63) / 64, 64, 0, c->stream>>>(c->pose[0].p, c->camR[0].p, c->camdR.p, c->sc_cam.p, m.pose_mask, c->nc, gen, nw, c->gW.p); LAUNCH_CHECK();
  c->launches++; return OMVG_OK;
}

int read_scalars(omvg_ba_ctx *c) {
  OMVG_CUDA(cudaMemcpyAsync(c->h_scal, c->scal.p, S_COUNT * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(c->h_scal + S_COUNT, c->part2.p, 3 * 64 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(c->h_scal + S_COUNT + 192, c->fail.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  return OMVG_OK;
}
double host_gmax(const omvg_ba_ctx *c) { double m = 0; for (int i = 0; i < 192; ++i) m = std::max(m, c->h_scal[S_COUNT + i]); return m; }

int build_structure(omvg_ba_ctx *c) {
  c->words = (c->nc + 31) / 32;
  int rc;
  if ((rc = c->bitmap.alloc((size_t)c->nc * c->words))) return rc;
  if ((rc = c->wprefix.alloc((size_t)c->nc * c->words))) return rc;
  if ((rc = c->rowptr.alloc(c->nc + 1))) return rc;
  OMVG_CUDA(cudaMemsetAsync(c->bitmap.p, 0, (size_t)c->nc * c->words * 4, c->stream));
  // every pose owns its diagonal block even without observations
  std::vector<unsigned> diagbits((size_t)c->nc * c->words, 0u);
  for (int a = 0; a < c->nc; ++a) diagbits[(size_t)a * c->words + (a >> 5)] |= 1u << (a & 31);
  OMVG_CUDA(cudaMemcpyAsync(c->bitmap.p, diagbits.data(), diagbits.size() * 4, cudaMemcpyHostToDevice, c->stream));
  if (c->no) { bitmap_mark_kernel<<<(unsigned)((c->no + 255) / 256), 256, 0, c->stream>>>(c->obs_pose.p, c->obs_pt.p, c->pt_start.p, c->no, c->bitmap.p, c->words); LAUNCH_CHECK(); }
  DevBuf<int> rowcount; if ((rc = rowcount.alloc(c->nc))) return rc;
  bitmap_rowcount_kernel<<<(c->nc + 127) / 128, 128, 0, c->stream>>>(c->bitmap.p, c->nc, c->words, c->wprefix.p, rowcount.p); LAUNCH_CHECK();
  std::vector<int> hc(c->nc), hp(c->nc + 1, 0);
  OMVG_CUDA(cudaMemcpyAsync(hc.data(), rowcount.p, c->nc * 4, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  for (int a = 0; a < c->nc; ++a) hp[a + 1] = hp[a] + hc[a];
  c->nnzb = hp[c->nc];
  OMVG_CUDA(cudaMemcpyAsync(c->rowptr.p, hp.data(), (c->nc + 1) * 4, cudaMemcpyHostToDevice, c->stream));
  if ((rc = c->cols.alloc(c->nnzb))) return rc;
  bitmap_cols_kernel<<<(c->nc + 127) / 128, 128, 0, c->stream>>>(c->bitmap.p, c->rowptr.p, c->nc, c->words, c->cols.p); LAUNCH_CHECK();
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  c->launches += 3;
  // ---- aggregates for the coarse space of the PCG preconditioner: greedy over the camera graph
  std::vector<int> hcols(c->nnzb), brow(c->nnzb);
  OMVG_CUDA(cudaMemcpy(hcols.data(), c->cols.p, (size_t)c->nnzb * 4, cudaMemcpyDeviceToHost));
  for (int a = 0; a < c->nc; ++a) for (int e = hp[a]; e < hp[a + 1]; ++e) brow[e] = a;
  int agg_max = std::max(8, (7 * c->nc + 1023) / 1024);     // coarse dimension 7*nc/agg_max <= ~1024
  // up to 600 cameras aggregates of 6 still fit one CTA per aggregate and a coarse inverse of <= 600^2 is cheap: fewer PCG
  // iterations for the same price (measured: 500 cameras 8.38 -> 7.68 ms per solve, 200 cameras 4.68 -> 4.62; at 1000
  // cameras aggregates of 6 or 7 would exceed / just fit the 148 CTAs of the shared-memory PCG: 14.4 / 12.3 against 12.1 ms)
  if (c->nc <= 600) agg_max = 6;
  if (const char *e = getenv("OMVG_BA_AGG")) agg_max = std::max(agg_max > 8 ? agg_max : 2, atoi(e));
  // Greedy aggregation of the camera graph: a seed takes the unaggregated cameras closest to it in index, first among its
  // neighbours, then among the neighbours of the cameras it already took, until the aggregate is full.  (Filling from the
  // seed's own neighbours only left holes — e.g. a stride pattern where camera a+11 is no neighbour of a — and with them
  // ~25 % more aggregates than 7 nc / 1024 allows: 182 instead of 143 at 2000 cameras.)
  std::vector<int> agg_of(c->nc, -1), agg_size;
  { std::vector<char> seen(c->nc, 0); std::vector<int> touched;
    for (int a = 0; a < c->nc; ++a) {
      if (agg_of[a] >= 0) continue;
      const int g = (int)agg_size.size(); agg_of[a] = g; int cnt = 1;
      std::vector<std::pair<int, int>> heap;                    // min-heap on (index distance to the seed, camera)
      auto cmp = [](const std::pair<int, int> &x, const std::pair<int, int> &y) { return x > y; };
      touched.clear(); seen[a] = 1; touched.push_back(a);
      auto push = [&](int x) {
        for (int e = hp[x]; e < hp[x + 1]; ++e) { const int b = hcols[e];
          if (!seen[b] && agg_of[b] < 0) { seen[b] = 1; touched.push_back(b); heap.emplace_back(std::abs(b - a), b); std::push_heap(heap.begin(), heap.end(), cmp); } } };
      push(a);
      while (!heap.empty() && cnt < agg_max) {
        std::pop_heap(heap.begin(), heap.end(), cmp); const int b = heap.back().second; heap.pop_back();
        agg_of[b] = g; ++cnt; push(b);
      }
      for (int t : touched) seen[t] = 0;
      agg_size.push_back(cnt);
    } }
  // aggregates of at most half the target size (singletons cannot carry 7 independent generators) join their smallest
  // neighbouring aggregate, preferably one that stays within what pcg5 holds in shared memory
  { std::vector<std::vector<int>> mem(agg_size.size());
    for (int a = 0; a < c->nc; ++a) mem[agg_of[a]].push_back(a);
    std::vector<int> order(agg_size.size()); for (size_t g = 0; g < order.size(); ++g) order[g] = (int)g;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return mem[x].size() < mem[y].size(); });
    int live = (int)agg_size.size();
    for (int g : order) {
      if (mem[g].empty() || (int)mem[g].size() * 2 > agg_max || live <= 1) continue;
      int tgt = -1, tgt_any = -1;
      for (int a : mem[g]) for (int e = hp[a]; e < hp[a + 1]; ++e) { const int h = agg_of[hcols[e]];
        if (h == g) continue;
        if (tgt_any < 0 || mem[h].size() < mem[tgt_any].size() || (mem[h].size() == mem[tgt_any].size() && h < tgt_any)) tgt_any = h;
        if ((int)(mem[h].size() + mem[g].size()) <= PCG5_MC && (tgt < 0 || mem[h].size() < mem[tgt].size() || (mem[h].size() == mem[tgt].size() && h < tgt))) tgt = h; }
      if (tgt < 0) tgt = mem[g].size() == 1 ? tgt_any : -1;       // a singleton must go somewhere
      if (tgt < 0 && mem[g].size() == 1) { const int a = mem[g][0]; tgt = agg_of[a == 0 ? (c->nc > 1 ? 1 : 0) : a - 1]; if (tgt == g) tgt = -1; }
      if (tgt < 0) continue;
      for (int a : mem[g]) { agg_of[a] = tgt; mem[tgt].push_back(a); }
      mem[g].clear(); --live;
    }
    for (size_t g = 0; g < agg_size.size(); ++g) agg_size[g] = (int)mem[g].size(); }
  std::vector<int> remap(agg_size.size(), -1); int ng = 0;
  for (size_t g = 0; g < agg_size.size(); ++g) if (agg_size[g] > 0) remap[g] = ng++;
  std::vector<int> agg_start(ng + 1, 0), agg_cams(c->nc);
  for (int a = 0; a < c->nc; ++a) { agg_of[a] = remap[agg_of[a]]; agg_start[agg_of[a] + 1]++; }
  for (int g = 0; g < ng; ++g) agg_start[g + 1] += agg_start[g];
  { std::vector<int> cur(agg_start.begin(), agg_start.end() - 1); for (int a = 0; a < c->nc; ++a) agg_cams[cur[agg_of[a]]++] = a; }
  c->ng = ng;
  c->agg_maxsize = 0; for (int gq = 0; gq < ng; ++gq) c->agg_maxsize = std::max(c->agg_maxsize, agg_start[gq + 1] - agg_start[gq]);
  if (getenv("OMVG_BA_TIMING")) fprintf(stderr, "[omvg_ba structure] %d poses, %d S blocks, %d aggregates (target %d, largest %d)\n", c->nc, c->nnzb, ng, agg_max, c->agg_maxsize);
  if ((rc = upload(c->agg_of, agg_of.data(), c->nc, c->stream))) return rc;
  if ((rc = upload(c->agg_start, agg_start.data(), ng + 1, c->stream))) return rc;
  if ((rc = upload(c->agg_cams, agg_cams.data(), c->nc, c->stream))) return rc;
  if ((rc = upload(c->brow, brow.data(), c->nnzb, c->stream))) return rc;
  // neighbour cameras of every aggregate (the union of the S-block columns of its rows) and, per S block, the position
  // of its column in the list of its row's aggregate: pcg5 gathers each neighbour's vectors ONCE per iteration
  { std::vector<int> nb_start(ng + 1, 0), nb_list; std::vector<unsigned short> lcol(c->nnzb, 0); std::vector<int> mark(c->nc, -1);
    c->nb_max = 0;
    for (int g = 0; g < ng; ++g) {
      const int first = (int)nb_list.size();
      for (int t = agg_start[g]; t < agg_start[g + 1]; ++t) { const int a = agg_cams[t];
        for (int e = hp[a]; e < hp[a + 1]; ++e) { const int b = hcols[e]; if (mark[b] < first) { mark[b] = (int)nb_list.size(); nb_list.push_back(b); } lcol[e] = (unsigned short)std::min(65535, mark[b] - first); } }
      nb_start[g + 1] = (int)nb_list.size(); c->nb_max = std::max(c->nb_max, nb_start[g + 1] - first);
    }
    if ((rc = upload(c->nb_start, nb_start.data(), ng + 1, c->stream))) return rc;
    if ((rc = upload(c->nb_list, nb_list.data(), nb_list.size(), c->stream))) return rc;
    if ((rc = upload(c->blk_lcol, lcol.data(), lcol.size(), c->stream))) return rc;
    OMVG_CUDA(cudaStreamSynchronize(c->stream)); }
  const size_t nco_max = (size_t)ng * MAXW;
  if ((rc = c->cE.alloc(nco_max * nco_max))) return rc;
  if ((rc = c->cT.alloc(3 * (size_t)GJ_B * nco_max))) return rc;   // Gauss-Jordan scratch: Cold / H / Gn
  if ((rc = c->cCv.alloc((size_t)MAXRHS * nco_max))) return rc;
  if ((rc = c->cYv.alloc((size_t)MAXRHS * nco_max))) return rc;
  if ((rc = c->cCv2.alloc((size_t)MAXRHS * nco_max + 1)) || (rc = c->cAW.alloc((size_t)MAXRHS * nco_max + 1))) return rc;
  if ((rc = c->bP2.alloc((size_t)MAXRHS * 6 * c->nc))) return rc;
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  return c->Scc.alloc((size_t)c->nnzb * 36);
}

// Pair lists of schur_gather_kernel (see pair_fill_kernel).  Work list: the diagonal blocks first (one entry per
// observation of the camera: the longest lists start first), then the upper off-diagonal blocks row by row, so that the
// rows in flight share their landmarks' GE records in L2.
int build_pair_lists(omvg_ba_ctx *c) {
  int rc;
  std::vector<int> hp(c->nc + 1), hcols(c->nnzb);
  OMVG_CUDA(cudaMemcpyAsync(hp.data(), c->rowptr.p, (c->nc + 1) * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(hcols.data(), c->cols.p, (size_t)c->nnzb * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  auto find = [&](int a, int b) { return (int)(std::lower_bound(hcols.begin() + hp[a], hcols.begin() + hp[a + 1], b) - hcols.begin()); };
  std::vector<int> wpos(c->nnzb, -1), gblk, gblkT;
  for (int a = 0; a < c->nc; ++a) { const int e = find(a, a); wpos[e] = (int)gblk.size(); gblk.push_back(e); gblkT.push_back(e); }
  for (int a = 0; a < c->nc; ++a)
    for (int e = hp[a]; e < hp[a + 1]; ++e) if (hcols[e] > a) { wpos[e] = (int)gblk.size(); gblk.push_back(e); gblkT.push_back(find(hcols[e], a)); }
  c->nwork = (int)gblk.size();
  cudaStream_t s = c->stream;
  DevBuf<int> d_wpos;
  if ((rc = upload(c->gblk, gblk.data(), gblk.size(), s)) || (rc = upload(c->gblkT, gblkT.data(), gblkT.size(), s)) || (rc = upload(d_wpos, wpos.data(), wpos.size(), s))) return rc;
  DevBuf<long long> cnt, offs; DevBuf<unsigned char> tmp;
  if ((rc = cnt.alloc(c->np + 1)) || (rc = offs.alloc(c->np + 1)) || (rc = c->gstart.alloc(c->nwork + 1))) return rc;
  pair_count_kernel<<<(c->np + 256) / 256, 256, 0, s>>>(c->pt_start.p, c->pt_single.p, c->obs_pose.p, c->np, cnt.p); LAUNCH_CHECK();
  size_t tb = 0;
  OMVG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, cnt.p, offs.p, c->np + 1, s));
  if ((rc = tmp.alloc(tb))) return rc;
  OMVG_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb, cnt.p, offs.p, c->np + 1, s));
  long long total = 0;
  OMVG_CUDA(cudaMemcpyAsync(&total, offs.p + c->np, sizeof total, cudaMemcpyDeviceToHost, s));
  OMVG_CUDA(cudaStreamSynchronize(s));
  if (total > std::numeric_limits<int>::max()) return fail(OMVG_E_UNSUPPORTED, "%lld camera-pair terms of the Schur complement (at most 2^31 - 1)", total);
  const int n = (int)total;
  if (n > 0) {
    DevBuf<int> k0, k1; DevBuf<unsigned long long> p0;
    if ((rc = k0.alloc(n)) || (rc = k1.alloc(n)) || (rc = p0.alloc(n)) || (rc = c->pairs.alloc(n))) return rc;
    pair_fill_kernel<<<(c->np + 255) / 256, 256, 0, s>>>(c->pt_start.p, c->pt_single.p, c->obs_pose.p, c->np, offs.p, Bsr{c->bitmap.p, c->wprefix.p, c->rowptr.p, c->words}, d_wpos.p, k0.p, p0.p); LAUNCH_CHECK();
    int kbits = 1; while ((1ll << kbits) < c->nwork) ++kbits;
    size_t sb = 0;
    OMVG_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sb, k0.p, k1.p, p0.p, c->pairs.p, n, 0, kbits, s));
    if (sb > tmp.n && (rc = tmp.alloc(sb))) return rc;
    sb = tmp.n;
    OMVG_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, sb, k0.p, k1.p, p0.p, c->pairs.p, n, 0, kbits, s));
    setup_starts_kernel<<<(unsigned)((n + 256) / 256), 256, 0, s>>>(k1.p, n, c->nwork, c->gstart.p); LAUNCH_CHECK();
    OMVG_CUDA(cudaStreamSynchronize(s));               // the temporaries are released at the end of this scope
    c->launches += 2;
  } else {
    OMVG_CUDA(cudaMemsetAsync(c->gstart.p, 0, (c->nwork + 1) * sizeof(int), s));
    OMVG_CUDA(cudaStreamSynchronize(s));
  }
  c->launches += 1;
  if (getenv("OMVG_BA_TIMING")) fprintf(stderr, "[omvg_ba structure] %d upper S blocks, %d pair-list entries (%.1f MB)\n", c->nwork, n, n * 8e-6);
  return OMVG_OK;
}

}  // namespace

extern "C" {

void omvg_trim_cache(void) {
  omvg::pool_trim();
  ResPool &rp = res_pool(); std::lock_guard<std::mutex> g(rp.mu);
  int cur = 0; cudaGetDevice(&cur);
  for (int d = 0; d < 16; ++d) { if (rp.free_[d].empty()) continue; cudaSetDevice(d);
    for (CtxRes &r : rp.free_[d]) { cudaFreeHost(r.h_scal); for (cudaEvent_t e : r.ev) cudaEventDestroy(e); cudaStreamDestroy(r.stream); cudaStreamDestroy(r.stream2); }
    rp.free_[d].clear(); }
  cudaSetDevice(cur);
}

void omvg_ba_default_options(omvg_ba_options *o) {
  if (!o) return;
  std::memset(o, 0, sizeof *o);
  o->intrinsics_opt = 14; o->extrinsics_opt = 6; o->structure_opt = 1; o->use_loss = 1; o->huber_a = 16.0;
  o->max_num_iterations = 50; o->max_consecutive_invalid_steps = 5;
  o->function_tolerance = 1e-6; o->gradient_tolerance = 1e-10; o->parameter_tolerance = 1e-8;
  o->initial_radius = 1e4; o->max_radius = 1e16; o->min_radius = 1e-32; o->min_relative_decrease = 1e-3;
  o->min_lm_diagonal = 1e-6; o->max_lm_diagonal = 1e32;
  o->pcg_tolerance = 1e-8; o->pcg_max_iterations = 2000; o->verbose = 0;
}

int omvg_ba_create(omvg_ba_ctx **out, int device, const omvg_ba_problem *P) {
  if (!out) return fail(OMVG_E_ARG, "null ctx");
  PhaseTimer tm("create");
  int rc = validate(P); if (rc) return rc;
  tm.lap("validate");
  int n = 0; OMVG_CUDA(cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) return fail(OMVG_E_CUDA, "no CUDA device %d (found %d)", device, n);
  int cc_major = 0, cc_minor = 0, n_sms = 0;                 // attributes: cudaGetDeviceProperties costs milliseconds
  OMVG_CUDA(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, device));
  OMVG_CUDA(cudaDeviceGetAttribute(&cc_minor, cudaDevAttrComputeCapabilityMinor, device));
  OMVG_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, device));
  if (cc_major != 10) return fail(OMVG_E_CUDA, "device %d is sm_%d%d; this library is sm_100a only", device, cc_major, cc_minor);
  OMVG_CUDA(cudaSetDevice(device));
  omvg_ba_ctx *c = new omvg_ba_ctx; c->device = device; c->n_sms = n_sms;
  std::unique_ptr<omvg_ba_ctx, void (*)(omvg_ba_ctx *)> guard(c, [](omvg_ba_ctx *x) { omvg_ba_destroy(x); });
  { CtxRes r; bool have = false;
    { ResPool &rp = res_pool(); std::lock_guard<std::mutex> g(rp.mu); auto &v = rp.free_[device & 15]; if (!v.empty()) { r = v.back(); v.pop_back(); have = true; } }
    if (!have) {
      OMVG_CUDA(cudaStreamCreateWithFlags(&r.stream, cudaStreamNonBlocking));
      OMVG_CUDA(cudaStreamCreateWithFlags(&r.stream2, cudaStreamNonBlocking));
      for (int i = 0; i < 4; ++i) OMVG_CUDA(cudaEventCreate(&r.ev[i]));
      OMVG_CUDA(cudaEventCreateWithFlags(&r.ev[4], cudaEventDisableTiming));
      OMVG_CUDA(cudaMallocHost(&r.h_scal, (S_COUNT + 192 + 2) * sizeof(double)));
    }
    c->stream = r.stream; c->stream2 = r.stream2; c->ev0 = r.ev[0]; c->ev1 = r.ev[1]; c->evj0 = r.ev[2]; c->evj1 = r.ev[3]; c->ev_up = r.ev[4]; c->h_scal = r.h_scal; }
  c->nc = P->n_poses; c->ni = P->n_intrinsics; c->np = P->n_points; c->nv = P->n_views; c->no = P->n_obs;
  c->ni8 = KI * c->ni; c->nred = 6 * c->nc + c->ni8; c->eval_blocks = (int)std::max<long long>(1, (c->no + EVAL_THREADS - 1) / EVAL_THREADS);
  c->eval_grid = std::min(c->eval_blocks, c->n_sms * (getenv("OMVG_BA_EVAL_WAVES") ? atoi(getenv("OMVG_BA_EVAL_WAVES")) : 4));   // persistent grid-stride evaluation
  tm.lap("stream+events+pinned");
  c->h_intr_model.assign(P->intr_model, P->intr_model + c->ni);
  c->kiu = 3; for (int q = 0; q < c->ni; ++q) c->kiu = std::max(c->kiu, model_nparams(P->intr_model[q]));   // (>= 3: the column-sum kernels are instantiated for 3, 4, 6, 7, 8)
  const long long no = c->no;
  // intrinsics with the unused tail zeroed (so block norms only see real parameters)
  std::vector<double> h_intr((size_t)c->ni8, 0.0);
  for (int q = 0; q < c->ni; ++q) for (int k = 0; k < model_ndata(P->intr_model[q]); ++k) h_intr[KI * q + k] = P->intrinsics[KI * q + k];
  cudaStream_t s = c->stream;
#define UP(buf, ptr, cnt) if ((rc = upload(buf, ptr, (size_t)(cnt), s))) return rc
  UP(c->pose0, P->poses, 6 * c->nc); UP(c->intr0, h_intr.data(), c->ni8); UP(c->pt0, P->points, 3 * (size_t)c->np);
  UP(c->intr_model, P->intr_model, c->ni);
  // ---- observations: upload as given, then sort by landmark / build the per-pose lists on the device
  // the image positions / weights / flags (16-25 B per observation) are only needed by the last gather: their upload runs on
  // a second stream under the sorts and the structure build (pinned host buffers; pageable ones are staged synchronously)
  DevBuf<double> raw_xy, raw_w; DevBuf<unsigned char> raw_fl;
  { DevBuf<int> raw_view, raw_point, d_view_pose, d_view_intr, keys, iota, keys2, bad; DevBuf<unsigned char> cubtmp;
    UP(raw_view, P->obs_view, no); UP(raw_point, P->obs_point, no);
    UP(d_view_pose, P->view_pose, c->nv); UP(d_view_intr, P->view_intr, c->nv);
    if ((rc = upload(raw_xy, P->obs_xy, (size_t)(2 * no), c->stream2))) return rc;
    if (P->obs_weight) { if ((rc = upload(raw_w, P->obs_weight, (size_t)no, c->stream2))) return rc; if ((rc = c->obs_w.alloc(no))) return rc; }
    if (P->obs_no_loss) { if ((rc = upload(raw_fl, P->obs_no_loss, (size_t)no, c->stream2))) return rc; if ((rc = c->obs_flags.alloc(no))) return rc; }
    OMVG_CUDA(cudaEventRecord(c->ev_up, c->stream2));
    if (tm.on) { cudaStreamSynchronize(s); cudaStreamSynchronize(c->stream2); }
    tm.lap("uploads");
    if ((rc = keys.alloc(no)) || (rc = iota.alloc(no)) || (rc = keys2.alloc(no)) || (rc = bad.alloc(1))) return rc;
    if ((rc = c->d_perm.alloc(no)) || (rc = c->obs_pose.alloc(no)) || (rc = c->obs_intr.alloc(no)) || (rc = c->obs_pt.alloc(no)) || (rc = c->obs_xy.alloc(2 * no))) return rc;
    if ((rc = c->pt_start.alloc(c->np + 1)) || (rc = c->cam_start.alloc(c->nc + 1)) || (rc = c->cam_obs.alloc(no)) || (rc = c->pt_single.alloc(c->np))) return rc;
    const int h_big = 0x7fffffff; OMVG_CUDA(cudaMemcpyAsync(bad.p, &h_big, sizeof(int), cudaMemcpyHostToDevice, s));
    const unsigned gb = (unsigned)((no + 255) / 256);
    setup_check_kernel<<<gb, 256, 0, s>>>(raw_view.p, raw_point.p, no, c->nv, c->np, keys.p, iota.p, bad.p); LAUNCH_CHECK();
    int pbits = 1; while ((1ll << pbits) < c->np) ++pbits;
    int cbits = 1; while ((1ll << cbits) < c->nc) ++cbits;
    size_t tb1 = 0, tb2 = 0;                                  // stable LSD radix sorts (CUB): by landmark, then by pose
    OMVG_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb1, keys.p, c->obs_pt.p, iota.p, c->d_perm.p, (int)no, 0, pbits, s));
    OMVG_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb2, c->obs_pose.p, keys2.p, iota.p, c->cam_obs.p, (int)no, 0, cbits, s));
    if ((rc = cubtmp.alloc(std::max(tb1, tb2)))) return rc;
    size_t tb = cubtmp.n;
    OMVG_CUDA(cub::DeviceRadixSort::SortPairs(cubtmp.p, tb, keys.p, c->obs_pt.p, iota.p, c->d_perm.p, (int)no, 0, pbits, s));
    setup_gather_kernel<<<gb, 256, 0, s>>>(c->d_perm.p, raw_view.p, d_view_pose.p, d_view_intr.p, nullptr, nullptr, nullptr, no, c->nv,
                                           c->obs_pose.p, c->obs_intr.p, nullptr, nullptr, nullptr, iota.p); LAUNCH_CHECK();
    setup_starts_kernel<<<(unsigned)((no + 256) / 256), 256, 0, s>>>(c->obs_pt.p, no, c->np, c->pt_start.p); LAUNCH_CHECK();
    tb = cubtmp.n;
    OMVG_CUDA(cub::DeviceRadixSort::SortPairs(cubtmp.p, tb, c->obs_pose.p, keys2.p, iota.p, c->cam_obs.p, (int)no, 0, cbits, s));
    setup_starts_kernel<<<(unsigned)((no + 256) / 256), 256, 0, s>>>(keys2.p, no, c->nc, c->cam_start.p); LAUNCH_CHECK();
    DevBuf<int> slow; if ((rc = slow.alloc(1))) return rc;
    OMVG_CUDA(cudaMemsetAsync(slow.p, 0, sizeof(int), s));
    setup_single_kernel<<<(c->np + 255) / 256, 256, 0, s>>>(c->obs_intr.p, c->pt_start.p, c->np, c->pt_single.p, slow.p); LAUNCH_CHECK();
    int h_bad = 0; OMVG_CUDA(cudaMemcpyAsync(&h_bad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    OMVG_CUDA(cudaMemcpyAsync(&c->n_slow, slow.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    OMVG_CUDA(cudaStreamSynchronize(s));                      // the temporaries above are released at the end of this scope
    c->launches += 9;
    if (h_bad != h_big) return fail(OMVG_E_ARG, "observation %d out of range", h_bad);
    tm.lap("device sort / lists");
  }
  if (P->point_fixed) {
    std::vector<unsigned> pm(c->np); for (int j = 0; j < c->np; ++j) pm[j] = P->point_fixed[j] ? 0u : 7u;
    UP(c->pt_fixed, P->point_fixed, c->np); UP(c->pt_mask, pm.data(), c->np);
  }
  c->has_ext = P->obs_weight || P->obs_no_loss || P->point_fixed;
  c->npri = P->n_priors; c->prior_huber_a = P->prior_huber_a;
  if (c->npri) { UP(c->prior_pose, P->prior_pose, c->npri); UP(c->prior_center, P->prior_center, 3 * c->npri); UP(c->prior_weight, P->prior_weight, 3 * c->npri); }
#undef UP
#define AL(buf, cnt) if ((rc = buf.alloc((size_t)(cnt)))) return rc
  for (int w = 0; w < 2; ++w) { AL(c->pose[w], 6 * c->nc); AL(c->intr[w], c->ni8); AL(c->pt[w], 3 * (size_t)c->np); AL(c->camR[w], 9 * c->nc); AL(c->camrec[w], (size_t)CAMREC * c->nc); }
  AL(c->camdR, 27 * c->nc);
  AL(c->r, 2 * no); AL(c->Jp, 6 * no); AL(c->Jc, 12 * no); AL(c->Ji, 2 * KI * no);
  AL(c->sc_pt, 3 * (size_t)c->np); AL(c->sc_cam, 6 * c->nc); AL(c->sc_intr, c->ni8);
  AL(c->diag_pt, 3 * (size_t)c->np); AL(c->diag_cam, 6 * c->nc); AL(c->diag_intr, c->ni8);
  AL(c->lmD_pt, 3 * (size_t)c->np); AL(c->lmD_cam, 6 * c->nc); AL(c->lmD_intr, c->ni8); AL(c->g_cam, 6 * c->nc); AL(c->g_intr, c->ni8);
  AL(c->EtFi, 3 * KI * (size_t)c->np); AL(c->FtF, 36 * (size_t)c->nc); AL(c->FiFi, 64 * (size_t)c->ni);
  AL(c->EtE, 6 * (size_t)c->np); AL(c->Etb, 3 * (size_t)c->np); AL(c->Einv, 9 * (size_t)c->np); AL(c->step_pt, 3 * (size_t)c->np); AL(c->step_red, c->nred);
  AL(c->intr_mask, c->ni);
  AL(c->Sci, (size_t)c->ni8 * 6 * c->nc); AL(c->Sii, (size_t)c->ni8 * c->ni8); AL(c->rhs, c->nred); AL(c->Minv_c, 36 * (size_t)c->nc); AL(c->Minv_i, (size_t)c->ni * KI * KI);
  AL(c->work_i, (size_t)c->ni8 * c->ni8 + c->ni8);
  AL(c->gW, (size_t)MAXW * 6 * c->nc);
  AL(c->bX, (size_t)MAXRHS * 6 * c->nc); AL(c->bR, (size_t)MAXRHS * 6 * c->nc); AL(c->bP, (size_t)MAXRHS * 6 * c->nc); AL(c->bW, (size_t)MAXRHS * 6 * c->nc); AL(c->bZ, (size_t)MAXRHS * 6 * c->nc);
  AL(c->pcg2_part, (size_t)c->n_sms * PCG2_V);
  AL(c->z, c->nred); AL(c->res, c->nred); AL(c->pvec, c->nred); AL(c->w, c->nred); AL(c->zeta, c->nred); AL(c->pcg_part, 3 * (size_t)c->n_sms * 2);
  if (c->npri) { AL(c->rP, 3 * c->npri); AL(c->JP, 18 * c->npri); }
  AL(c->part, std::max(c->eval_blocks, 1024) + 2); AL(c->part2, 1024); AL(c->part3, 1024); c->ics_chunks = (int)std::max<long long>(1, std::min<long long>(4ll * c->n_sms / std::max(1, c->ni), (c->no + 2047) / 2048));
  AL(c->icol_part, (size_t)c->ni * c->ics_chunks * ICS_W); AL(c->scal, S_COUNT); AL(c->fail, 1);
#undef AL
  OMVG_CUDA(cudaMemsetAsync(c->scal.p, 0, S_COUNT * sizeof(double), s));
  tm.lap("allocations");
  if ((rc = build_structure(c))) return rc;
  tm.lap("structure");
  if ((rc = build_pair_lists(c))) return rc;
  tm.lap("pair lists");
  OMVG_CUDA(cudaStreamWaitEvent(s, c->ev_up, 0));
  setup_gather_xy_kernel<<<(unsigned)((no + 255) / 256), 256, 0, s>>>(c->d_perm.p, reinterpret_cast<const double2 *>(raw_xy.p), raw_w.p, raw_fl.p, no,
                                                                  reinterpret_cast<double2 *>(c->obs_xy.p), c->obs_w.p, c->obs_flags.p); LAUNCH_CHECK();
  c->launches++;
  if ((rc = omvg_ba_reset(c))) return rc;
  OMVG_CUDA(cudaStreamSynchronize(s));
  guard.release();
  *out = c; return OMVG_OK;
}

int omvg_ba_reset(omvg_ba_ctx *c) {
  if (!c) return fail(OMVG_E_ARG, "null ctx");
  OMVG_CUDA(cudaSetDevice(c->device));
  OMVG_CUDA(cudaMemcpyAsync(c->pose[0].p, c->pose0.p, 6 * c->nc * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(c->intr[0].p, c->intr0.p, c->ni8 * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  if (c->np) OMVG_CUDA(cudaMemcpyAsync(c->pt[0].p, c->pt0.p, 3 * (size_t)c->np * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  return OMVG_OK;
}

int omvg_ba_destroy(omvg_ba_ctx *c) {
  if (!c) return OMVG_OK;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->stream2) cudaStreamSynchronize(c->stream2);
  CtxRes r; r.stream = c->stream; r.stream2 = c->stream2; r.ev[0] = c->ev0; r.ev[1] = c->ev1; r.ev[2] = c->evj0; r.ev[3] = c->evj1; r.ev[4] = c->ev_up; r.h_scal = c->h_scal;
  const int dev = c->device & 15;
  delete c;                                   // DevBuf destructors hand device memory back to the pool
  if (r.stream && r.stream2 && r.ev[4] && r.h_scal) { ResPool &rp = res_pool(); std::lock_guard<std::mutex> g(rp.mu); rp.free_[dev].push_back(r); }
  else { if (r.h_scal) cudaFreeHost(r.h_scal); for (cudaEvent_t e : r.ev) if (e) cudaEventDestroy(e); if (r.stream) cudaStreamDestroy(r.stream); }
  return OMVG_OK;
}

int omvg_ba_download(omvg_ba_ctx *c, double *poses, double *intrinsics, double *points) {
  if (!c) return fail(OMVG_E_ARG, "null ctx");
  OMVG_CUDA(cudaSetDevice(c->device));
  if (poses) OMVG_CUDA(cudaMemcpyAsync(poses, c->pose[0].p, 6 * c->nc * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  std::vector<double> hi(c->ni8);
  if (intrinsics) OMVG_CUDA(cudaMemcpyAsync(hi.data(), c->intr[0].p, c->ni8 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  if (points && c->np) OMVG_CUDA(cudaMemcpyAsync(points, c->pt[0].p, 3 * (size_t)c->np * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  if (intrinsics) for (int q = 0; q < c->ni; ++q) for (int k = 0; k < model_nparams(c->h_intr_model[q]); ++k) intrinsics[KI * q + k] = hi[KI * q + k];
  return OMVG_OK;
}

int omvg_ba_run(omvg_ba_ctx *c, const omvg_ba_options *O, omvg_ba_summary *sum) {
  if (!c || !O || !sum) return fail(OMVG_E_ARG, "null argument");
  OMVG_CUDA(cudaSetDevice(c->device));
  std::memset(sum, 0, sizeof *sum);
  const Masks m = make_masks(c, O);
  OMVG_CUDA(cudaMemcpyAsync(c->intr_mask.p, m.intr_mask.data(), c->ni * sizeof(unsigned), cudaMemcpyHostToDevice, c->stream));
  OMVG_CUDA(cudaMemsetAsync(c->fail.p, 0, sizeof(int), c->stream));
  const long long launches0 = c->launches;
  OMVG_CUDA(cudaEventRecord(c->ev0, c->stream));
  int rc; bool have_scale = false;
  double jac_ms = 0; long long jac_launches = 0;
  auto account_jac = [&]() { float ms = 0; cudaEventSynchronize(c->evj1); cudaEventElapsedTime(&ms, c->evj0, c->evj1); jac_ms += ms; ++jac_launches; };

  if ((rc = eval_jac(c, O, m, 0, have_scale, true))) return rc;
  // small reduced systems are solved directly by one CTA (dense_solve_kernel): no gauge / coarse space / PCG
  const int dense_max = getenv("OMVG_BA_DENSE_MAX") ? std::min(DENSE_MAX, atoi(getenv("OMVG_BA_DENSE_MAX"))) : DENSE_MAX;
  const bool use_dense1 = 6 * c->nc + c->ni8 <= dense_max;                      // one CTA, shared memory
  const int dense2_max = getenv("OMVG_BA_DENSE2_MAX") ? std::min(1024, atoi(getenv("OMVG_BA_DENSE2_MAX"))) : 640;
  const bool use_dense2 = !use_dense1 && 6 * c->nc + c->ni8 <= dense2_max;      // explicit inverse by the blocked Gauss-Jordan kernel
  const bool use_dense = use_dense1 || use_dense2;
  int nw = 0;
  if (!use_dense && (rc = make_gauge(c, m, nw))) return rc;
  int n_free_intr = 0; for (unsigned mm : m.intr_mask) n_free_intr += __builtin_popcount(mm);
  // up to 32 free intrinsic columns: block elimination of the intrinsics border (pcg5, else pcg3); otherwise pcg_kernel
  const bool use_pcg3 = n_free_intr <= MAXRHS - 1 && c->nc >= 2 && !getenv("OMVG_BA_PCG1");
  // the per-observation kernels gather pose records (176 B x n_poses) and points through L1: give them all of it
  OMVG_CUDA(cudaFuncSetAttribute(eval_kernel<true, 4, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
  OMVG_CUDA(cudaFuncSetAttribute(eval_kernel<false, 8, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
  OMVG_CUDA(cudaFuncSetAttribute(eval_kernel<true, 4, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
  OMVG_CUDA(cudaFuncSetAttribute(eval_kernel<false, 8, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
  OMVG_CUDA(cudaFuncSetAttribute(pcg3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(Pcg2Smem) + 4 * PCG3_NCO_MAX * sizeof(double))));
  if ((rc = read_scalars(c))) return rc;
  account_jac();
  double x_cost = c->h_scal[S_COST];
  double gmax = host_gmax(c);
  sum->initial_cost = x_cost;
  double radius = O->initial_radius, decrease_factor = 2.0;
  int iteration = 0, n_success = 0, n_fail = 0, n_invalid = 0, termination = 3;
  double x_norm = -1.0;                                   // trust_region_minimizer.cc Init(): "x_norm_ = -1"
  bool step_is_successful = true, failure = false;
  double reference_cost = x_cost, accumulated_reference = 0.0, current_cost = x_cost;
  long long pcg_total = 0;
  int coarse_age = -1; double last_pcg_its = 0, fresh_pcg_its = 1e30; bool fresh_pending = false;
  static const int coarse_every = getenv("OMVG_BA_COARSE_EVERY") ? std::max(1, atoi(getenv("OMVG_BA_COARSE_EVERY"))) : 3;
  if (!c->gj_grid) {                                        // as many co-resident CTAs as the tile count can use
    int per_sm = 1; OMVG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, coarse_invert_kernel, 256, 0));
    c->gj_grid = c->n_sms * std::max(1, std::min(per_sm, 2));
  }

  for (;;) {
    if (step_is_successful) ++n_success; else ++n_fail;
    if (iteration >= O->max_num_iterations) { termination = 3; break; }
    if (step_is_successful && gmax <= O->gradient_tolerance) { termination = 2; break; }
    if (radius <= O->min_radius) { termination = 4; break; }
    ++iteration;
    // ---- LM diagonal (levenberg_marquardt_strategy.cc:75-87); diag_* always belong to the current J
    { Diag3 DG{}; DG.s[0] = Diag3Seg{c->diag_pt.p, c->lmD_pt.p, 3 * c->np}; DG.s[1] = Diag3Seg{c->diag_cam.p, c->lmD_cam.p, 6 * c->nc}; DG.s[2] = Diag3Seg{c->diag_intr.p, c->lmD_intr.p, c->ni8};
      const int nb = std::max(1, std::min(2 * c->n_sms, (3 * c->np + 255) / 256));
      lm_diag3_kernel<<<dim3(nb, 3), 256, 0, c->stream>>>(DG, O->min_lm_diagonal, O->max_lm_diagonal, radius); LAUNCH_CHECK(); }
    // ---- reduced camera system
    if (m.pts_free && !c->corner_rep.p) { if ((rc = c->corner_rep.alloc((size_t)CORNER_REPS * (KI * KI + KI)))) return rc; }
    { Zero4 Z{}; Z.p[0] = c->Scc.p; Z.n[0] = m.pts_free ? 0 : (long long)c->nnzb * 36;     // (schur_gather_kernel writes all of Scc)
      Z.p[1] = c->Sci.p; Z.n[1] = (long long)c->Sci.n; Z.p[2] = c->Sii.p; Z.n[2] = (long long)c->Sii.n;
      Z.p[3] = m.pts_free ? c->corner_rep.p : c->rhs.p; Z.n[3] = m.pts_free ? (long long)c->corner_rep.n : 0;     // (rhs is fully written by s_init_kernel)
      const long long zmax = std::max(std::max(Z.n[0], Z.n[1]), std::max(Z.n[2], Z.n[3]));
      const int nb = (int)std::max<long long>(1, std::min<long long>(4 * c->n_sms, (zmax + 255) / 256));
      zero4_kernel<<<dim3(nb, 4), 256, 0, c->stream>>>(Z); LAUNCH_CHECK(); }
    SchurArgs SA{}; SA.r = c->r.p; SA.Jp = c->Jp.p; SA.Jc = c->Jc.p; SA.Ji = c->Ji.p; SA.EtE = c->EtE.p; SA.Etb = c->Etb.p; SA.EtFi = c->EtFi.p; SA.lmD_pt = c->lmD_pt.p; SA.pt_single = c->pt_single.p; SA.FtF = c->FtF.p; SA.FiFi = c->FiFi.p; SA.g_cam = c->g_cam.p; SA.g_intr = c->g_intr.p;
    SA.obs_pose = c->obs_pose.p; SA.obs_intr = c->obs_intr.p; SA.obs_pt = c->obs_pt.p; SA.pt_start = c->pt_start.p; SA.n = c->no; SA.n_poses = c->nc; SA.n_intr = c->ni;
    SA.pts_free = m.pts_free; SA.kiu = c->kiu; SA.bsr = Bsr{c->bitmap.p, c->wprefix.p, c->rowptr.p, c->words}; SA.Scc = c->Scc.p; SA.Sci = c->Sci.p; SA.Sii = c->Sii.p; SA.rhs = c->rhs.p;
    SA.Einv = c->Einv.p; SA.fail = c->fail.p;
    { const int ninit = std::max(std::max(36 * c->nc, 64 * c->ni), c->nred); s_init_kernel<<<(ninit + 255) / 256, 256, 0, c->stream>>>(SA); LAUNCH_CHECK(); }
    if (m.pts_free) {
      if (!c->GE.p) { if ((rc = c->GE.alloc(36 * (size_t)c->no))) return rc; }
      { const unsigned sg = (unsigned)((c->no + SCHUR_THREADS - 1) / SCHUR_THREADS);
#define STAGE(K) schur_stage_kernel<K><<<sg, SCHUR_THREADS, 0, c->stream>>>(SA, c->GE.p, c->corner_rep.p)
        switch (c->kiu) {        // intrinsic columns in use (as for the column sums)
          case 3: STAGE(3); break;
          case 4: STAGE(4); break;
          case 6: STAGE(6); break;
          case 7: STAGE(7); break;
          default: STAGE(8); break;
        }
#undef STAGE
      }
      LAUNCH_CHECK();
      corner_fold_kernel<<<1, 96, 0, c->stream>>>(c->corner_rep.p, c->obs_intr.p, c->nc, c->ni, c->Sii.p, c->rhs.p); LAUNCH_CHECK(); c->launches++;
      schur_gather_kernel<<<(unsigned)(((long long)c->nwork * 32 + GATHER_THREADS - 1) / GATHER_THREADS), GATHER_THREADS, 0, c->stream>>>(
          c->GE.p, c->gstart.p, reinterpret_cast<const int2 *>(c->pairs.p), c->gblk.p, c->gblkT.p, c->nwork, c->brow.p, c->FtF.p, c->Scc.p); LAUNCH_CHECK();
      c->launches += 2;
      SA.skip_fast = 1;
    }
    // the remaining landmarks (several intrinsic groups, more than 32 observations) add to the gathered Scc: after it
    if (!m.pts_free || c->n_slow > 0) { schur_kernel<<<(unsigned)((c->no + SCHUR_THREADS - 1) / SCHUR_THREADS), SCHUR_THREADS, 0, c->stream>>>(SA); LAUNCH_CHECK(); }
    c->launches += 1;
    finish_cam_kernel<<<(c->nc + 63) / 64, 64, 0, c->stream>>>(c->Scc.p, SA.bsr, c->lmD_cam.p, m.pose_mask, c->nc, c->Minv_c.p, c->fail.p, use_dense ? 0 : 1); LAUNCH_CHECK();
    finish_intr_kernel<<<1, 256, 0, c->stream>>>(c->Sii.p, c->lmD_intr.p, c->intr_mask.p, c->ni8, c->Minv_i.p, c->work_i.p, c->fail.p, (use_pcg3 || use_dense) ? 0 : 1); LAUNCH_CHECK();
    // ---- PCG on S z = rhs
    PcgArgs PA{}; PA.Scc = c->Scc.p; PA.rowptr = c->rowptr.p; PA.cols = c->cols.p; PA.Sci = c->Sci.p; PA.Sii = c->Sii.p; PA.rhs = c->rhs.p; PA.Minv_c = c->Minv_c.p; PA.Minv_i = c->Minv_i.p;
    PA.n_poses = c->nc; PA.ni8 = c->ni8; PA.z = c->z.p; PA.res = c->res.p; PA.p = c->pvec.p; PA.w = c->w.p; PA.zeta = c->zeta.p; PA.part = c->pcg_part.p;
    PA.tol = O->pcg_tolerance; PA.max_iter = O->pcg_max_iterations; PA.out = c->scal.p + S_PCG_IT;
    // ---- coarse operator of the two-level preconditioner (aggregated gauge space), shared by the PCG variants.
    // It is only a preconditioner: a slightly stale E^-1 (previous LM step, radius/3) costs a few extra PCG
    // iterations (measured 38->40, 42->49, 43->43) but saves its O(nco^3) setup, so it is refreshed every
    // `coarse_every` LM steps (measured at 1000 cameras, ms per solve: every step 17.9, 2: 16.0, 3: 15.2, 5: 15.9),
    // or earlier if the last solve needed 1.5x the iterations seen right after a refresh.
    const bool use_coarse = !use_dense && nw > 0 && c->nc >= 2;
    const Coarse CO{c->agg_of.p, c->agg_start.p, c->agg_cams.p, c->ng, nw, use_coarse ? c->ng * nw : 0};
    if (use_coarse) {
      const int nco = CO.nco;
      const bool refresh = nco > 0 && (coarse_age < 0 || coarse_age >= coarse_every || last_pcg_its > 1.5 * fresh_pcg_its + 5);
      if (refresh) { coarse_age = 0; fresh_pending = true; }
      ++coarse_age;
      if (refresh) {
        OMVG_CUDA(cudaMemsetAsync(c->cE.p, 0, (size_t)nco * nco * sizeof(double), c->stream));
        coarse_assemble_kernel<<<(c->nnzb + 127) / 128, 128, 0, c->stream>>>(c->Scc.p, c->brow.p, c->cols.p, c->nnzb, c->gW.p, c->nc, CO, c->cE.p); LAUNCH_CHECK();
        // blocked Gauss-Jordan, in place: cE becomes E^-1
        double *Ep = c->cE.p, *Tp = c->cT.p; int nn = nco; int *fp = c->fail.p;
        static const bool gj_timing = getenv("OMVG_BA_GJ_TIMING") != nullptr;
        unsigned long long *tp = nullptr;
        if (gj_timing) { if (!c->pcg_tim.p) { if ((rc = c->pcg_tim.alloc(8))) return rc; } OMVG_CUDA(cudaMemsetAsync(c->pcg_tim.p, 0, 64, c->stream)); tp = c->pcg_tim.p; }
        void *cargs[] = {&Ep, &nn, &Tp, &fp, &tp};
        const int mt = (nco + CT - 1) / CT;                   // no more CTAs than 64x64 tiles: a small coarse space pays for fewer barrier participants
        const int gj = std::max(1, std::min(c->gj_grid, mt * mt));
        OMVG_CUDA(cudaLaunchCooperativeKernel((void *)coarse_invert_kernel, dim3(gj), dim3(256), cargs, 0, c->stream));
        if (gj_timing) { unsigned long long h[8]; OMVG_CUDA(cudaMemcpyAsync(h, c->pcg_tim.p, 64, cudaMemcpyDeviceToHost, c->stream)); OMVG_CUDA(cudaStreamSynchronize(c->stream));
          fprintf(stderr, "[omvg_ba gj timing] us: pivot inverse %.1f slices %.1f sync %.1f tiles %.1f sync %.1f (n %d, %d CTAs)\n", h[0] * 1e-3, h[1] * 1e-3, h[2] * 1e-3, h[3] * 1e-3, h[4] * 1e-3, nco, c->gj_grid); }
        c->launches += 2;
      }
    }
    if (use_dense2) {
      int nd = 6 * c->nc + c->ni8;
      if (!c->dA.p) { if ((rc = c->dA.alloc((size_t)nd * nd)) || (rc = c->dT.alloc(3 * (size_t)GJ_B * nd))) return rc; }
      OMVG_CUDA(cudaMemsetAsync(c->dA.p, 0, (size_t)nd * nd * sizeof(double), c->stream));
      dense_assemble_kernel<<<std::max(1, std::min(4 * c->n_sms, (36 * c->nnzb + 255) / 256)), 256, 0, c->stream>>>(c->Scc.p, c->brow.p, c->cols.p, c->nnzb, c->Sci.p, c->Sii.p, c->nc, c->ni8, c->dA.p); LAUNCH_CHECK();
      double *Ap = c->dA.p, *Tp = c->dT.p; int *fp = c->fail.p; unsigned long long *tp = nullptr;
      void *cargs[] = {&Ap, &nd, &Tp, &fp, &tp};
      const int mt = (nd + CT - 1) / CT;
      OMVG_CUDA(cudaLaunchCooperativeKernel((void *)coarse_invert_kernel, dim3(std::max(1, std::min(c->gj_grid, mt * mt))), dim3(256), cargs, 0, c->stream));
      dense_apply_kernel<<<(nd * 32 + 255) / 256, 256, 0, c->stream>>>(c->dA.p, c->rhs.p, nd, c->z.p, c->scal.p + S_PCG_IT); LAUNCH_CHECK();
      c->launches += 3;
    } else
    if (use_dense1) {
      const int nd = 6 * c->nc + c->ni8;
      const size_t dsm = ((size_t)nd * (nd + 1) / 2 + (3 + DENSE_NB) * (size_t)nd) * sizeof(double);
      OMVG_CUDA(cudaFuncSetAttribute(dense_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsm));
      static const bool dense_timing = getenv("OMVG_BA_DENSE_TIMING") != nullptr;
      unsigned long long *tp = nullptr;
      if (dense_timing) { if (!c->pcg_tim.p) { if ((rc = c->pcg_tim.alloc(8))) return rc; } OMVG_CUDA(cudaMemsetAsync(c->pcg_tim.p, 0, 64, c->stream)); tp = c->pcg_tim.p; }
      dense_solve_kernel<<<1, 1024, dsm, c->stream>>>(c->Scc.p, c->rowptr.p, c->cols.p, c->Sci.p, c->Sii.p, c->rhs.p, c->nc, c->ni8, c->z.p, c->fail.p, c->scal.p + S_PCG_IT, tp); LAUNCH_CHECK();
      if (dense_timing) { unsigned long long h[8]; OMVG_CUDA(cudaMemcpyAsync(h, c->pcg_tim.p, 64, cudaMemcpyDeviceToHost, c->stream)); OMVG_CUDA(cudaStreamSynchronize(c->stream));
        fprintf(stderr, "[omvg_ba dense timing] n %d us: assemble %.1f factor %.1f backward %.1f\n", nd, h[0] * 1e-3, h[1] * 1e-3, h[2] * 1e-3); }
    } else
    if (use_pcg3) {
      Pcg2Args P2{}; P2.Scc = c->Scc.p; P2.rowptr = c->rowptr.p; P2.cols = c->cols.p; P2.Sci = c->Sci.p; P2.Sii = c->Sii.p; P2.rhs = c->rhs.p; P2.Minv_c = c->Minv_c.p;
      P2.W = c->gW.p; P2.intr_mask = c->intr_mask.p; P2.n_poses = c->nc; P2.ni8 = c->ni8; P2.nw = nw; P2.X = c->bX.p; P2.Rv = c->bR.p; P2.Pv = c->bP.p; P2.Wv = c->bW.p; P2.Zv = c->bZ.p;
      P2.part = c->pcg2_part.p; P2.z = c->z.p; P2.tol = O->pcg_tolerance; P2.max_iter = O->pcg_max_iterations; P2.out = c->scal.p + S_PCG_IT;
      Pcg3Args P3{}; P3.base = P2; P3.C = CO; P3.C.nco = c->ng * nw; P3.Einv = c->cE.p; P3.Cv = c->cCv.p; P3.Yv = c->cYv.p; P3.Pv2 = c->bP2.p;
      static const bool pcg_timing = getenv("OMVG_BA_PCG_TIMING") != nullptr;
      if (pcg_timing) { if (!c->pcg_tim.p) { if ((rc = c->pcg_tim.alloc(8))) return rc; } OMVG_CUDA(cudaMemsetAsync(c->pcg_tim.p, 0, 64, c->stream)); P3.tim = c->pcg_tim.p; }
      // pcg5: shared-memory resident, aggregate-owned (2 barriers + 2 L2 round trips per iteration).  Needs one CTA per
      // aggregate, <= 4 right-hand sides (1 + free intrinsic columns) and aggregates of <= 16 cameras; else pcg3.
      const int nrhs_host = 1 + n_free_intr;
      if (nrhs_host <= PCG5_NR && c->ng <= c->n_sms && c->agg_maxsize <= PCG5_MC && c->nb_max <= PCG5_NB && P3.C.nco <= PCG3_NCO_MAX) {
        const size_t fixed = sizeof(Pcg5Red) + sizeof(Pcg5Smem) + (size_t)PCG5_NR * PCG3_NCO_MAX * sizeof(double) + (size_t)PCG5_NB * PCG5_PS * sizeof(double);
        static const int smem_max = [] { int v = 0, dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev); return v; }();
        const int nb_cache = (int)std::max<long long>(0, ((long long)smem_max - (long long)fixed - 2048) /   /* (static shared memory of the kernel + slack) */ (long long)(PCG5_BS * sizeof(double) + sizeof(unsigned short)));
        const size_t smem = fixed + (size_t)nb_cache * (PCG5_BS * sizeof(double) + sizeof(unsigned short)) + 16;
        OMVG_CUDA(cudaFuncSetAttribute(pcg5_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        double *cg2 = c->cCv2.p, *aw = c->cAW.p; int nbc = nb_cache; const int *nbs = c->nb_start.p, *nbl = c->nb_list.p; const unsigned short *lc = c->blk_lcol.p;
        void *args[] = {&P3, &cg2, &aw, &nbc, &nbs, &nbl, &lc};
        // one CTA per aggregate and no more: idle CTAs would only add participants to the two barriers of every iteration
        OMVG_CUDA(cudaLaunchCooperativeKernel((void *)pcg5_kernel, dim3(std::max(1, c->ng)), dim3(PCG2_THREADS), args, smem, c->stream));
        if (pcg_timing) { unsigned long long h[8]; OMVG_CUDA(cudaMemcpyAsync(h, c->pcg_tim.p, 64, cudaMemcpyDeviceToHost, c->stream)); OMVG_CUDA(cudaStreamSynchronize(c->stream));
          fprintf(stderr, "[omvg_ba pcg5 timing] us: A wait-AW %.1f y %.1f local %.1f reduce %.1f | B gather %.1f rows %.1f publish %.1f reduce %.1f (cache %d blocks)\n", h[0] * 1e-3, h[1] * 1e-3, h[2] * 1e-3, h[3] * 1e-3, h[6] * 1e-3, h[7] * 1e-3, h[4] * 1e-3, h[5] * 1e-3, nb_cache); }
      } else {
        void *args[] = {&P3};
        OMVG_CUDA(cudaLaunchCooperativeKernel((void *)pcg3_kernel, dim3(c->n_sms), dim3(PCG2_THREADS), args, sizeof(Pcg2Smem) + 4 * PCG3_NCO_MAX * sizeof(double), c->stream));
        if (pcg_timing) { unsigned long long h[8]; OMVG_CUDA(cudaMemcpyAsync(h, c->pcg_tim.p, 64, cudaMemcpyDeviceToHost, c->stream)); OMVG_CUDA(cudaStreamSynchronize(c->stream));
          fprintf(stderr, "[omvg_ba pcg timing] us: coarse (stage %.1f rows %.1f sync %.1f) z %.1f spmv %.1f update %.1f tail %.1f border %.1f\n", h[6] * 1e-3, h[7] * 1e-3, h[0] * 1e-3, h[1] * 1e-3, h[2] * 1e-3, h[3] * 1e-3, h[4] * 1e-3, h[5] * 1e-3); }
      }
    } else {
      // more than 32 free intrinsic columns (e.g. one intrinsic group per image), a single pose, or OMVG_BA_PCG1: PCG on the
      // whole reduced system [Scc Sci'; Sci Sii] with the aggregated coarse space on the camera rows (when there is one) and
      // block-Jacobi on the intrinsics
      if (use_coarse) { PA.W = c->gW.p; PA.C = CO; PA.Einv = c->cE.p; PA.Cv = c->cCv.p; PA.Yv = c->cYv.p; }
      void *args[] = {&PA}; OMVG_CUDA(cudaLaunchCooperativeKernel((void *)pcg_kernel, dim3(c->n_sms), dim3(256), args, 0, c->stream));
    }
    // ---- back substitution, step = -y
    if (!m.pts_free) {
      backsub_kernel<<<(c->np + 127) / 128, 128, 0, c->stream>>>(c->Jp.p, c->Jc.p, c->Ji.p, c->Etb.p, c->Einv.p, c->obs_pose.p, c->obs_intr.p, c->pt_start.p, c->np, c->nc, c->no, c->kiu,
                                                               c->z.p, m.pts_free, c->step_pt.p); LAUNCH_CHECK();
    } else {
      OMVG_CUDA(cudaMemsetAsync(c->step_pt.p, 0, 3 * (size_t)c->np * sizeof(double), c->stream));
      backsub_obs_kernel<<<(unsigned)((c->no + 255) / 256), 256, 0, c->stream>>>(c->Jp.p, c->Jc.p, c->Ji.p, c->obs_pose.p, c->obs_intr.p, c->obs_pt.p, c->nc, c->no, c->kiu, c->z.p, c->step_pt.p); LAUNCH_CHECK();
      backsub_point_kernel<<<(c->np + 255) / 256, 256, 0, c->stream>>>(c->Etb.p, c->Einv.p, c->pt_start.p, c->np, m.pts_free, c->step_pt.p); LAUNCH_CHECK();
      c->launches++;
    }
    negate_kernel<<<(c->nred + 255) / 256, 256, 0, c->stream>>>(c->z.p, c->nred, c->step_red.p); LAUNCH_CHECK();
    // ---- model cost change
    model_kernel<<<c->eval_blocks, MODEL_THREADS, 0, c->stream>>>(c->r.p, c->Jp.p, c->Jc.p, c->Ji.p, c->obs_pose.p, c->obs_intr.p, c->obs_pt.p, c->no, c->nc, c->kiu, c->step_pt.p, c->step_red.p, c->part.p); LAUNCH_CHECK();
    c->launches += 9;
    if (c->npri) { prior_model_kernel<<<1, PRIOR_THREADS, 0, c->stream>>>(c->JP.p, c->rP.p, c->prior_pose.p, c->npri, c->step_red.p, c->part.p + c->eval_blocks); LAUNCH_CHECK(); c->launches++; }
    if ((rc = reduce_to(c, c->part.p, c->eval_blocks + (c->npri ? 1 : 0), S_MODEL))) return rc;
    // ---- candidate = Plus(x, step * scale)
    const int ub = 64;
    auto update_all = [&]() -> int {       // candidate = Plus(x, step * scale) for the three parameter blocks; |step|^2 and |x|^2 into S_STEP2_* / S_X2_*
      Upd3 U{};
      U.s[0] = UpdSeg{c->pt[0].p, c->step_pt.p, c->sc_pt.p, 3 * c->np, 3, m.pts_free ? 7u : 0u, m.pts_free ? c->pt_mask.p : nullptr, c->pt[1].p};
      U.s[1] = UpdSeg{c->pose[0].p, c->step_red.p, c->sc_cam.p, 6 * c->nc, 6, m.pose_mask, nullptr, c->pose[1].p};
      U.s[2] = UpdSeg{c->intr[0].p, c->step_red.p + 6 * c->nc, c->sc_intr.p, c->ni8, KI, 0u, c->intr_mask.p, c->intr[1].p};
      update3_kernel<<<dim3(ub, 3), 256, 0, c->stream>>>(U, c->part3.p); LAUNCH_CHECK();
      static_assert(S_STEP2_POSE == S_STEP2_PT + 1 && S_STEP2_INTR == S_STEP2_PT + 2 && S_X2_PT == S_STEP2_PT + 3 && S_X2_POSE == S_STEP2_PT + 4 && S_X2_INTR == S_STEP2_PT + 5, "slot order");
      reduce_multi_kernel<<<6, 1024, 0, c->stream>>>(c->part3.p, ub, c->scal.p + S_STEP2_PT); LAUNCH_CHECK();
      c->launches += 2; return OMVG_OK;
    };
    if ((rc = update_all())) return rc;
    if ((rc = eval_cost(c, O, 1, S_CAND_COST))) return rc;
    if ((rc = read_scalars(c))) return rc;
    const double *h = c->h_scal;
    pcg_total += (long long)h[S_PCG_IT];
    last_pcg_its = h[S_PCG_IT]; if (fresh_pending) { fresh_pcg_its = last_pcg_its; fresh_pending = false; }
    int failflag; std::memcpy(&failflag, c->h_scal + S_COUNT + 192, sizeof(int));
    const double model_cost_change = h[S_MODEL];
    bool finite_step = std::isfinite(h[S_STEP2_PT]) && std::isfinite(h[S_STEP2_POSE]) && std::isfinite(h[S_STEP2_INTR]) && std::isfinite(model_cost_change);
    const bool solved = failflag == 0 && finite_step;
    if (failflag) OMVG_CUDA(cudaMemsetAsync(c->fail.p, 0, sizeof(int), c->stream));
    if (O->verbose) fprintf(stderr, "[omvg_ba] it %d cost %.12e cand %.12e model %.6e radius %.3e pcg %d res %.2e\n", iteration, x_cost, h[S_CAND_COST], model_cost_change, radius, (int)h[S_PCG_IT], h[S_PCG_RES]);
    if (!solved || !(model_cost_change > 0.0)) {            // HandleInvalidStep (:429-462)
      if (++n_invalid >= O->max_consecutive_invalid_steps) { failure = true; termination = -1; break; }
      radius = radius / decrease_factor; decrease_factor *= 2.0;
      step_is_successful = false; continue;
    }
    n_invalid = 0;
    const double candidate_cost = h[S_CAND_COST];
    const double step_norm = std::sqrt(h[S_STEP2_PT] + h[S_STEP2_POSE] + h[S_STEP2_INTR]);
    if (step_norm <= O->parameter_tolerance * (x_norm + O->parameter_tolerance)) { termination = 1; break; }
    const double cost_change = x_cost - candidate_cost;
    if (std::fabs(cost_change) <= O->function_tolerance * x_cost) { termination = 0; break; }
    const double rel = (current_cost - candidate_cost) / model_cost_change;
    const double hist = (reference_cost - candidate_cost) / (accumulated_reference + model_cost_change);
    const double rho = std::max(rel, hist);
    if (rho > O->min_relative_decrease) {                    // HandleSuccessfulStep (:767-780)
      std::swap(c->pose[0].p, c->pose[1].p); std::swap(c->intr[0].p, c->intr[1].p); std::swap(c->pt[0].p, c->pt[1].p); std::swap(c->camR[0].p, c->camR[1].p); std::swap(c->camrec[0].p, c->camrec[1].p);
      // |x| of the accepted iterate = sqrt(|x_old|^2 ...) is not reusable: recompute from the candidate norms
      if ((rc = eval_jac(c, O, m, 0, have_scale, true))) return rc;
      if (!use_dense && (rc = make_gauge(c, m, nw))) return rc;
      // x_norm of the new x: update3_kernel measures |x| of its input: one more pass over the new x
      if ((rc = update_all())) return rc;     // (the gradient maxima of eval_jac sit in part2, the norm partials in part3)
      if ((rc = read_scalars(c))) return rc;
      account_jac();
      x_cost = c->h_scal[S_COST]; gmax = host_gmax(c);
      x_norm = std::sqrt(c->h_scal[S_X2_PT] + c->h_scal[S_X2_POSE] + c->h_scal[S_X2_INTR]);
      step_is_successful = true;
      radius = radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * rho - 1.0, 3)); radius = std::min(O->max_radius, radius);
      decrease_factor = 2.0;
      current_cost = candidate_cost; reference_cost = candidate_cost; accumulated_reference = 0.0;
    } else {                                                  // HandleUnsuccessfulStep (:782-786)
      step_is_successful = false;
      radius = radius / decrease_factor; decrease_factor *= 2.0;
    }
  }
  OMVG_CUDA(cudaEventRecord(c->ev1, c->stream));
  OMVG_CUDA(cudaEventSynchronize(c->ev1));
  float ms = 0; OMVG_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  sum->final_cost = x_cost; sum->iterations = n_success + n_fail; sum->successful_steps = n_success; sum->unsuccessful_steps = n_fail;
  sum->lm_steps = iteration; sum->termination = termination; sum->usable = failure ? 0 : 1; sum->pcg_iterations = pcg_total;
  sum->kernel_launches = c->launches - launches0; sum->device_ms = ms; sum->jacobian_ms = jac_ms; sum->jacobian_launches = jac_launches;
  return failure ? fail(OMVG_E_NUMERIC, "bundle adjustment failed: %d consecutive invalid steps", n_invalid) : OMVG_OK;
}

// AngleAxisToRotationMatrix (ceres/include/ceres/rotation.h:377-420), row-major
static void aa_to_R(const double *aa, double R[9]) {
  const double theta2 = aa[0] * aa[0] + aa[1] * aa[1] + aa[2] * aa[2];
  if (theta2 > std::numeric_limits<double>::epsilon()) {
    const double theta = std::sqrt(theta2), wx = aa[0] / theta, wy = aa[1] / theta, wz = aa[2] / theta;
    const double c = std::cos(theta), s = std::sin(theta), k = 1.0 - c;
    R[0] = c + wx * wx * k;      R[1] = wx * wy * k - wz * s; R[2] = wy * s + wx * wz * k;
    R[3] = wz * s + wx * wy * k; R[4] = c + wy * wy * k;      R[5] = -wx * s + wy * wz * k;
    R[6] = -wy * s + wx * wz * k; R[7] = wx * s + wy * wz * k; R[8] = c + wz * wz * k;
  } else {
    R[0] = 1; R[1] = -aa[2]; R[2] = aa[1]; R[3] = aa[2]; R[4] = 1; R[5] = -aa[0]; R[6] = -aa[1]; R[7] = aa[0]; R[8] = 1;
  }
}

// Adjust's write-back rules (sfm_data_BA_ceres.cpp:528-568) applied to the caller's flat arrays: poses only if
// extrinsics were refined, ADJUST_ROTATION keeps the pose CENTRE (t = -R_new C_old), intrinsics only if intrinsics
// were refined, points as they are on the device.  `poses` / `intrinsics` hold the caller's previous values on entry.
int omvg_ba_writeback(omvg_ba_ctx *c, const omvg_ba_options *O, double *poses, double *intrinsics, double *points) {
  if (!c || !O) return fail(OMVG_E_ARG, "null argument");
  std::vector<double> np_(poses ? (size_t)6 * c->nc : 0), ni_(intrinsics ? (size_t)KI * c->ni : 0);
  if (intrinsics) std::memcpy(ni_.data(), intrinsics, ni_.size() * sizeof(double));
  int rc = omvg_ba_download(c, poses ? np_.data() : nullptr, intrinsics ? ni_.data() : nullptr, points);
  if (rc) return rc;
  if (poses && O->extrinsics_opt != 1) {
    for (int p = 0; p < c->nc; ++p) {
      double *dst = poses + 6 * p; const double *src = np_.data() + 6 * p;
      if (O->extrinsics_opt == 2) {
        double Ro[9], Rn[9], C[3];
        aa_to_R(dst, Ro); aa_to_R(src, Rn);
        for (int i = 0; i < 3; ++i) C[i] = -(Ro[0 * 3 + i] * dst[3] + Ro[1 * 3 + i] * dst[4] + Ro[2 * 3 + i] * dst[5]);
        for (int i = 0; i < 3; ++i) dst[i] = src[i];
        for (int i = 0; i < 3; ++i) dst[3 + i] = -(Rn[i * 3] * C[0] + Rn[i * 3 + 1] * C[1] + Rn[i * 3 + 2] * C[2]);
      } else {
        for (int i = 0; i < 6; ++i) dst[i] = src[i];
      }
    }
  }
  if (intrinsics && !(O->intrinsics_opt & 1)) std::memcpy(intrinsics, ni_.data(), ni_.size() * sizeof(double));
  return OMVG_OK;
}

int omvg_ba_solve(omvg_ba_problem *P, const omvg_ba_options *O, omvg_ba_summary *sum) {
  omvg_ba_options def; if (!O) { omvg_ba_default_options(&def); O = &def; }
  omvg_ba_summary local; if (!sum) sum = &local;
  PhaseTimer tm("solve");
  omvg_ba_ctx *c = nullptr;
  int rc = omvg_ba_create(&c, O->device, P); if (rc) return rc;
  tm.lap("create");
  rc = omvg_ba_run(c, O, sum);
  tm.lap("run");
  if (rc == OMVG_OK) rc = omvg_ba_writeback(c, O, P->poses, P->intrinsics, P->points);   // state is copied back only when usable (solver.cc:445-448)
  tm.lap("download+write-back");
  omvg_ba_destroy(c);
  tm.lap("destroy");
  return rc;
}

// Reprojection residual norms (pixels) of every observation at the current device parameters, in the
// caller's observation order — what RemoveOutliers_PixelResidualError (sfm/sfm_data_filters.cpp:40-73)
// recomputes on the host after every Adjust of the BA / reject loop (sequential_SfM.cpp:205-211).
static int ensure_perm(omvg_ba_ctx *c) {
  if (!c->perm.empty() || !c->no) return OMVG_OK;
  c->perm.resize(c->no);
  OMVG_CUDA(cudaMemcpyAsync(c->perm.data(), c->d_perm.p, (size_t)c->no * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  return OMVG_OK;
}

int omvg_ba_residual_norms(omvg_ba_ctx *c, double *norms) {
  if (!c || !norms) return fail(OMVG_E_ARG, "null argument");
  OMVG_CUDA(cudaSetDevice(c->device));
  { const int prc = ensure_perm(c); if (prc) return prc; }
  omvg_ba_options O; omvg_ba_default_options(&O); O.use_loss = 0;
  cam_prep_kernel<<<(c->nc + 127) / 128, 128, 0, c->stream>>>(c->pose[0].p, c->nc, c->camR[0].p, c->camdR.p, c->camrec[0].p); LAUNCH_CHECK();
  EvalArgs A{}; A.poses = c->pose[0].p; A.intr = c->intr[0].p; A.pts = c->pt[0].p; A.camR = c->camR[0].p; A.camdR = c->camdR.p; A.camrec = c->camrec[0].p;
  A.obs_xy = c->obs_xy.p; A.intr_model = c->intr_model.p; A.obs_pose = c->obs_pose.p; A.obs_intr = c->obs_intr.p; A.obs_pt = c->obs_pt.p;
  A.n_obs = c->no; A.use_loss = 0; A.huber_a = O.huber_a; A.cost_partial = c->part.p; A.rnorm = c->r.p;   // r is scratch between solves
  eval_kernel<false, 8, false><<<c->eval_grid, EVAL_THREADS, 0, c->stream>>>(A); LAUNCH_CHECK();   // (weights deliberately not applied: pixels)
  c->launches += 2;
  std::vector<double> h(c->no);
  OMVG_CUDA(cudaMemcpyAsync(h.data(), c->r.p, (size_t)c->no * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  for (long long t = 0; t < c->no; ++t) norms[c->perm[t]] = h[t];
  return OMVG_OK;
}

// Replaces the per-observation weights of a resident problem (caller's observation order).  Weight 0
// removes the observation exactly (zero residual and Jacobian rows) while the sparsity structure stays
// a superset: the BA -> RemoveOutliers_PixelResidualError -> BA loop (sequential_SfM.cpp:1226-1243,
// sfm_filters.hpp:49-79) runs without rebuilding or re-uploading the scene.
int omvg_ba_set_obs_weights(omvg_ba_ctx *c, const double *w) {
  if (!c || !w) return fail(OMVG_E_ARG, "null argument");
  OMVG_CUDA(cudaSetDevice(c->device));
  { const int prc = ensure_perm(c); if (prc) return prc; }
  std::vector<double> s_w(c->no);
  for (long long t = 0; t < c->no; ++t) { const double v = w[c->perm[t]]; if (!(v >= 0.0) || !std::isfinite(v)) return fail(OMVG_E_ARG, "weight %d is negative or not finite", c->perm[t]); s_w[t] = v; }
  if (!c->obs_w.p) { int rc = c->obs_w.alloc(c->no); if (rc) return rc; }
  c->has_ext = true;
  OMVG_CUDA(cudaMemcpyAsync(c->obs_w.p, s_w.data(), (size_t)c->no * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  return OMVG_OK;
}

// Device-side RemoveOutliers_PixelResidualError (sfm/sfm_data_filters.cpp:40-73) + the track-length rule, and the
// removal of tracks named by the caller (the angle test of badTrackRejector, sequential_SfM.cpp:1237-1243, is host
// geometry): observations get weight 0 (exact removal, structure unchanged), removed tracks become constant blocks.
static int ensure_reject_state(omvg_ba_ctx *c) {
  if (c->reject_ready) return OMVG_OK;
  int rc;
  const unsigned gb = (unsigned)((c->no + 255) / 256), gp = (unsigned)((c->np + 255) / 256);
  if ((rc = c->pt_gcp.alloc(c->np)) || (rc = c->pt_removed.alloc(c->np)) || (rc = c->pt_now.alloc(c->np)) || (rc = c->rej_bits.alloc((size_t)(c->no + 31) / 32 + 1)) || (rc = c->rej_cnt.alloc(2))) return rc;
  if (c->pt_fixed.p) OMVG_CUDA(cudaMemcpyAsync(c->pt_gcp.p, c->pt_fixed.p, c->np, cudaMemcpyDeviceToDevice, c->stream));   // fixed at create = control points
  else OMVG_CUDA(cudaMemsetAsync(c->pt_gcp.p, 0, c->np, c->stream));
  OMVG_CUDA(cudaMemsetAsync(c->pt_removed.p, 0, c->np, c->stream));
  if (!c->obs_w.p) { if ((rc = c->obs_w.alloc(c->no))) return rc; fill_kernel<<<gb, 256, 0, c->stream>>>(c->obs_w.p, c->no, 1.0); LAUNCH_CHECK(); c->launches++; }
  if (!c->pt_fixed.p) { if ((rc = c->pt_fixed.alloc(c->np))) return rc; OMVG_CUDA(cudaMemsetAsync(c->pt_fixed.p, 0, c->np, c->stream)); }
  if (!c->pt_mask.p) { if ((rc = c->pt_mask.alloc(c->np))) return rc; fill_u32_kernel<<<gp, 256, 0, c->stream>>>(c->pt_mask.p, c->np, 7u); LAUNCH_CHECK(); c->launches++; }
  c->has_ext = true; c->reject_ready = true;
  return OMVG_OK;
}

static int reject_finish(omvg_ba_ctx *c, uint32_t *obs_removed_bits, uint8_t *point_removed, int64_t *n_outliers, int64_t *n_tracks) {
  unsigned long long h[2] = {0, 0};
  OMVG_CUDA(cudaMemcpyAsync(h, c->rej_cnt.p, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  if (obs_removed_bits) OMVG_CUDA(cudaMemcpyAsync(obs_removed_bits, c->rej_bits.p, ((size_t)(c->no + 31) / 32) * 4, cudaMemcpyDeviceToHost, c->stream));
  if (point_removed) OMVG_CUDA(cudaMemcpyAsync(point_removed, c->pt_now.p, c->np, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  if (n_outliers) *n_outliers = (int64_t)h[0];
  if (n_tracks) *n_tracks = (int64_t)h[1];
  return OMVG_OK;
}

int omvg_ba_reject_outliers(omvg_ba_ctx *c, double threshold_px, int32_t min_track_length, uint32_t *obs_removed_bits, uint8_t *point_removed,
                            int64_t *n_outliers, int64_t *n_tracks) {
  if (!c) return fail(OMVG_E_ARG, "null ctx");
  if (!(threshold_px >= 0.0) || min_track_length < 0) return fail(OMVG_E_ARG, "bad threshold / track length");
  OMVG_CUDA(cudaSetDevice(c->device));
  int rc = ensure_reject_state(c); if (rc) return rc;
  OMVG_CUDA(cudaMemsetAsync(c->rej_bits.p, 0, c->rej_bits.n * 4, c->stream));
  OMVG_CUDA(cudaMemsetAsync(c->rej_cnt.p, 0, 16, c->stream));
  // |r| in pixels at the current parameters (no weight, no loss): r is scratch between solves
  cam_prep_kernel<<<(c->nc + 127) / 128, 128, 0, c->stream>>>(c->pose[0].p, c->nc, c->camR[0].p, c->camdR.p, c->camrec[0].p); LAUNCH_CHECK();
  EvalArgs A{}; A.poses = c->pose[0].p; A.intr = c->intr[0].p; A.pts = c->pt[0].p; A.camR = c->camR[0].p; A.camdR = c->camdR.p; A.camrec = c->camrec[0].p;
  A.obs_xy = c->obs_xy.p; A.intr_model = c->intr_model.p; A.obs_pose = c->obs_pose.p; A.obs_intr = c->obs_intr.p; A.obs_pt = c->obs_pt.p;
  A.n_obs = c->no; A.use_loss = 0; A.huber_a = 16.0; A.cost_partial = c->part.p; A.rnorm = c->r.p;
  eval_kernel<false, 8, false><<<c->eval_grid, EVAL_THREADS, 0, c->stream>>>(A); LAUNCH_CHECK();
  reject_obs_kernel<<<(unsigned)((c->no + 255) / 256), 256, 0, c->stream>>>(c->r.p, c->obs_w.p, c->obs_pt.p, c->pt_gcp.p, c->no, threshold_px, c->d_perm.p, c->rej_bits.p, c->rej_cnt.p); LAUNCH_CHECK();
  reject_tracks_kernel<<<(c->np + 127) / 128, 128, 0, c->stream>>>(c->pt_start.p, c->np, c->obs_w.p, min_track_length, nullptr, c->pt_gcp.p, c->d_perm.p, c->rej_bits.p,
                                                                 c->pt_fixed.p, c->pt_mask.p, c->pt_removed.p, c->pt_now.p, c->rej_cnt.p); LAUNCH_CHECK();
  c->launches += 4;
  return reject_finish(c, obs_removed_bits, point_removed, n_outliers, n_tracks);
}

int omvg_ba_remove_points(omvg_ba_ctx *c, const uint8_t *point_mask, uint32_t *obs_removed_bits, int64_t *n_tracks) {
  if (!c || !point_mask) return fail(OMVG_E_ARG, "null argument");
  OMVG_CUDA(cudaSetDevice(c->device));
  int rc = ensure_reject_state(c); if (rc) return rc;
  DevBuf<unsigned char> kill; if ((rc = kill.alloc(c->np))) return rc;
  OMVG_CUDA(cudaMemcpyAsync(kill.p, point_mask, c->np, cudaMemcpyHostToDevice, c->stream));
  OMVG_CUDA(cudaMemsetAsync(c->rej_bits.p, 0, c->rej_bits.n * 4, c->stream));
  OMVG_CUDA(cudaMemsetAsync(c->rej_cnt.p, 0, 16, c->stream));
  reject_tracks_kernel<<<(c->np + 127) / 128, 128, 0, c->stream>>>(c->pt_start.p, c->np, c->obs_w.p, 0, kill.p, c->pt_gcp.p, c->d_perm.p, c->rej_bits.p,
                                                                 c->pt_fixed.p, c->pt_mask.p, c->pt_removed.p, c->pt_now.p, c->rej_cnt.p); LAUNCH_CHECK();
  c->launches++;
  return reject_finish(c, obs_removed_bits, nullptr, nullptr, n_tracks);      // (synchronises: `kill` may be released)
}

// Makes the current (refined) parameters the state omvg_ba_reset() returns to: the next run of the
// BA / reject loop starts from the previous solution.
int omvg_ba_commit(omvg_ba_ctx *c) {
  if (!c) return fail(OMVG_E_ARG, "null ctx");
  OMVG_CUDA(cudaSetDevice(c->device));
  OMVG_CUDA(cudaMemcpyAsync(c->pose0.p, c->pose[0].p, 6 * c->nc * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(c->intr0.p, c->intr[0].p, c->ni8 * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(c->pt0.p, c->pt[0].p, 3 * (size_t)c->np * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  return OMVG_OK;
}

int omvg_ba_debug_eval(omvg_ba_ctx *c, const omvg_ba_options *O, double *cost, double *r, double *J_intr, double *J_pose, double *J_point) {
  if (!c || !O) return fail(OMVG_E_ARG, "null argument");
  OMVG_CUDA(cudaSetDevice(c->device));
  { const int prc = ensure_perm(c); if (prc) return prc; }
  Masks m = make_masks(c, O);
  OMVG_CUDA(cudaMemcpyAsync(c->intr_mask.p, m.intr_mask.data(), c->ni * sizeof(unsigned), cudaMemcpyHostToDevice, c->stream));
  // unscaled evaluation (intrinsic columns >= kiu are never written: present them as zeros)
  OMVG_CUDA(cudaMemsetAsync(c->Ji.p, 0, c->Ji.n * sizeof(double), c->stream));
  cam_prep_kernel<<<(c->nc + 127) / 128, 128, 0, c->stream>>>(c->pose[0].p, c->nc, c->camR[0].p, c->camdR.p, c->camrec[0].p); LAUNCH_CHECK();
  EvalArgs A{}; A.poses = c->pose[0].p; A.intr = c->intr[0].p; A.pts = c->pt[0].p; A.camR = c->camR[0].p; A.camdR = c->camdR.p; A.camrec = c->camrec[0].p;
  A.obs_xy = c->obs_xy.p; A.intr_model = c->intr_model.p; A.obs_pose = c->obs_pose.p; A.obs_intr = c->obs_intr.p; A.obs_pt = c->obs_pt.p;
  A.n_obs = c->no; A.use_loss = O->use_loss; A.huber_a = O->huber_a; A.r = c->r.p; A.Jp = c->Jp.p; A.Jc = c->Jc.p; A.Ji = c->Ji.p;
  A.cost_partial = c->part.p; A.kiu = c->kiu; A.pose_mask = m.pose_mask; A.intr_mask = c->intr_mask.p; A.pts_free = m.pts_free;
  A.obs_w = c->obs_w.p; A.obs_flags = c->obs_flags.p; A.pt_fixed = c->pt_fixed.p;      // (prior rows are not part of this dump)
  eval_kernel<true, 4, true><<<c->eval_grid, EVAL_THREADS, 0, c->stream>>>(A); LAUNCH_CHECK();
  int rc = reduce_to(c, c->part.p, c->eval_grid, S_COST); if (rc) return rc;
  c->launches += 2;
  const long long n = c->no;
  std::vector<double> hr(2 * n), hp(6 * n), hc(12 * n), hi(2 * KI * n); double hcost = 0;
  OMVG_CUDA(cudaMemcpyAsync(hr.data(), c->r.p, hr.size() * 8, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(hp.data(), c->Jp.p, hp.size() * 8, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(hc.data(), c->Jc.p, hc.size() * 8, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(hi.data(), c->Ji.p, hi.size() * 8, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(&hcost, c->scal.p + S_COST, 8, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  if (cost) *cost = hcost;
  for (long long t = 0; t < n; ++t) {
    const long long o = c->perm[t];
    for (int row = 0; row < 2; ++row) {
      if (r) r[2 * o + row] = hr[row * n + t];
      if (J_point) for (int k = 0; k < 3; ++k) J_point[(o * 2 + row) * 3 + k] = hp[(row * 3 + k) * n + t];
      if (J_pose) for (int k = 0; k < 6; ++k) J_pose[(o * 2 + row) * 6 + k] = hc[(row * 6 + k) * n + t];
      if (J_intr) for (int k = 0; k < KI; ++k) J_intr[(o * 2 + row) * KI + k] = hi[(row * KI + k) * n + t];
    }
  }
  return OMVG_OK;
}

}  // extern "C"
