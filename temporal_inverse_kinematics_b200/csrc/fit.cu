// Fit SMPL-X body poses to observed keypoints: damped Gauss-Newton (Levenberg-Marquardt) per frame with an analytic
// Jacobian of the keypoint forward of keypoints.cu.  One warp per frame, several frames per CTA, the model tables staged
// once per CTA in shared memory.  Per frame f the unknowns are x = (theta (66) [, tau (3)]) and the cost is
//
//   E(x) = sum_k w_k |kp_k(theta, beta, tau) - y_k|^2 + lambda |theta - theta0|^2.
//
// A warp keeps everything of its frame in its own slice of shared memory:
//   - the forward: local rotations (22), FK of the 55-joint tree level by level (joints of one tree depth per pass),
//     landmark rest positions (shape + pose blend, one lane per landmark coordinate) and skinning, residuals r = kp - y;
//   - the Jacobian (3n x 72 rows, lanes over (point, joint) pairs, only ancestors written):
//       joint point k, proper ancestor j:   dkp_k/dtheta_j = -[t_k - t_j]x Rg_j Jr(theta_j)
//       landmark l, joint j:                 sum_{m: j <= m} w_lm (-[x_lm - t_j]x Rg_j Jr(theta_j))
//                                            + (sum_m w_lm Rg_m) d(offset_l)/dtheta_j   (pose blend, j >= 1)
//       translation:                         I;
//   - H = J^T W J + lambda I (packed lower triangle, lanes over 4x4 tiles) and g = J^T W r + lambda (theta - theta0);
//   - the damped system (H + mu diag(H)) delta = -g by a warp Cholesky on the packed triangle (which overwrites J: J is
//     rebuilt after every accepted step) and two substitutions; then one forward at the candidate.
// Every loop and reduction of a frame runs in an order fixed by the frame's own data and lane ids, so a frame's result
// does not depend on the other frames of the call or on its warp slot.
#include <string.h>

#include <algorithm>

#include "fit_device.cuh"

namespace tik {

__global__ void __launch_bounds__(kFitMaxWarps * 32)
fit_keypoints_kernel(const __grid_constant__ FitParams p) {
  extern __shared__ __align__(16) float fit_sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int L = p.n_lm, B = p.n_betas, n = p.n_sel, R = 3 * n;
  const bool has_pd = p.lm_pd != nullptr && L > 0;
  const FitSmem sm = fit_smem(n, L, B, has_pd);
  FitCta c;
  c.pd = has_pd ? fit_sm + sm.pd : nullptr;
  c.jt = fit_sm + sm.jt; c.jd = fit_sm + sm.jd; c.lmt = fit_sm + sm.lmt; c.lmd = fit_sm + sm.lmd; c.w = fit_sm + sm.w;
  c.anc = reinterpret_cast<const unsigned long long*>(fit_sm + sm.anc);
  {
    float* pd = fit_sm + sm.pd;
    if (has_pd)
      for (int i = tid; i < 3 * L * kFitFeat; i += blockDim.x) pd[i] = __ldg(p.lm_pd + (int64_t)(i / kFitFeat) * (kFitJ - 1) * 9 + i % kFitFeat);
    for (int i = tid; i < kFitJ * 3; i += blockDim.x) fit_sm[sm.jt + i] = __ldg(p.jt + i);
    for (int i = tid; i < kFitJ * 3 * B; i += blockDim.x) fit_sm[sm.jd + i] = __ldg(p.jd + i);
    for (int i = tid; i < 3 * L; i += blockDim.x) fit_sm[sm.lmt + i] = __ldg(p.lm_t + i);
    for (int i = tid; i < 3 * L * B; i += blockDim.x) fit_sm[sm.lmd + i] = __ldg(p.lm_d + i);
    for (int i = tid; i < L * kFitJ; i += blockDim.x) {    // dense skinning weights: repeated joints add up
      const int l = i / kFitJ, j = i % kFitJ;
      float w = 0.f;
      for (int k = 0; k < p.kmax; ++k)
        if (__ldg(p.skin_idx + l * p.kmax + k) == j) w += __ldg(p.skin_w + l * p.kmax + k);
      fit_sm[sm.w + i] = w;
    }
    unsigned long long* anc = reinterpret_cast<unsigned long long*>(fit_sm + sm.anc);
    for (int i = tid; i < kFitJ; i += blockDim.x) anc[i] = p.anc[i];
  }
  __syncthreads();

  float* base = fit_sm + sm.cta + warp * sm.warp;
  FitWarp s;
  s.U = base + sm.U; s.H = base + sm.H; s.g = base + sm.g; s.b = base + sm.b; s.x = base + sm.x; s.x0 = base + sm.x0;
  s.xc = base + sm.xc; s.y = base + sm.y; s.wr = base + sm.wr; s.res = base + sm.res; s.beta = base + sm.beta;
  s.rest = base + sm.rest; s.psh = base + sm.psh; s.p = base + sm.p; s.v = base + sm.v; s.Rl = base + sm.Rl;
  s.Rg = base + sm.Rg; s.t = base + sm.t; s.M = base + sm.M; s.D = base + sm.D;

  for (int64_t f = (int64_t)blockIdx.x * p.warps + warp; f < p.F; f += (int64_t)gridDim.x * p.warps) {
    // ---- the frame's inputs
    for (int i = lane; i < kFitPose; i += 32) s.x[i] = s.x0[i] = __ldg(p.init_pose + f * kFitPose + i);
    if (lane < kFitPitch - kFitPose) {
      const int c3 = lane;
      s.x[kFitPose + c3] = (c3 < 3 && p.transl != nullptr) ? __ldg(p.transl + f * 3 + c3) : 0.f;
      s.x0[kFitPose + c3] = 0.f;
    }
    for (int i = lane; i < R; i += 32) {
      s.y[i] = __ldg(p.target + f * R + i);
      s.wr[i] = p.weights == nullptr ? 1.f : __ldg(p.weights + (p.weights_per_frame ? f * n : 0) + i / 3);
    }
    if (lane < B)
      s.beta[lane] = p.betas == nullptr ? 0.f : __ldg(p.betas + (p.betas_per_frame ? f * B : 0) + lane);
    __syncwarp();
    for (int i = lane; i < kFitJ * 3; i += 32) {
      float v = c.jt[i];
      for (int k = 0; k < B; ++k) v = fmaf(c.jd[i * B + k], s.beta[k], v);
      s.rest[i] = v;
    }
    for (int i = lane; i < 3 * L; i += 32) {
      float v = c.lmt[i];
      for (int k = 0; k < B; ++k) v = fmaf(c.lmd[i * B + k], s.beta[k], v);
      s.psh[i] = v;
    }
    __syncwarp();

    // ---- Levenberg-Marquardt with the fixed schedule: accept on a strictly lower cost
    const float E0 = fit_forward(p, c, s, s.x, lane);
    float E = E0, mu = 1e-3f;
    const bool finite = isfinite(E0);
    if (finite && p.n_iter > 0) {
      fit_normal_equations(p, c, s, lane);
      for (int it = 0; it < p.n_iter; ++it) {
        bool accept = false;
        if (fit_solve(p, s, mu, lane)) {
          for (int i = lane; i < kFitPitch; i += 32) s.xc[i] = s.x[i] + (i < p.P ? s.b[i] : 0.f);
          __syncwarp();
          const float Ec = fit_forward(p, c, s, s.xc, lane);
          accept = Ec < E;
          if (accept) E = Ec;
        }
        if (accept) {
          for (int i = lane; i < kFitPitch; i += 32) s.x[i] = s.xc[i];
          __syncwarp();
          mu = fmaxf(mu / 10.f, 1e-7f);
          if (it + 1 < p.n_iter) fit_normal_equations(p, c, s, lane);
        } else {
          mu = fminf(mu * 10.f, 1e7f);
        }
      }
    }
    for (int i = lane; i < kFitPose; i += 32) p.pose_out[f * kFitPose + i] = s.x[i];
    if (p.transl_out != nullptr && lane < 3) p.transl_out[f * 3 + lane] = s.x[kFitPose + lane];
    if (p.cost != nullptr && lane == 0) {
      p.cost[f * 2] = E0;
      p.cost[f * 2 + 1] = finite ? E : __int_as_float(0x7fc00000);
    }
    __syncwarp();
  }
}

}  // namespace tik

extern "C" int tik_fit_keypoints(const TikKeypointModel* m, const float* target_dev, const float* weights_dev,
                                 int weights_per_frame, const float* init_pose_dev, const float* betas_dev,
                                 int betas_per_frame, const float* transl_dev, int fit_transl, const int32_t* select_host,
                                 int n_select, float prior_weight, int n_iter, int64_t F, float* pose_out_dev,
                                 float* transl_out_dev, float* cost_dev, void* stream) {
  using namespace tik;
  const char* fn = "fit_keypoints";
  TIK_CHECK_ARG(m != nullptr, "%s: null model", fn);
  const int B = m->n_betas, L = m->n_landmarks;
  if (int rc = fit_check_model(m, fn)) return rc;
  if (int rc = fit_check_weights(weights_dev, weights_per_frame, fn)) return rc;
  TIK_CHECK_ARG(betas_per_frame == 0 || betas_per_frame == 1, "fit_keypoints: betas_per_frame=%d must be 0 or 1", betas_per_frame);
  TIK_CHECK_ARG(!(betas_per_frame && betas_dev == nullptr && B > 0), "fit_keypoints: per-frame betas need betas_dev");
  FitParams p;
  memset(&p, 0, sizeof(p));
  if (int rc = fit_check_solver(m, fit_transl, select_host, n_select, prior_weight, n_iter, F, &p, fn)) return rc;
  if (F == 0) return TIK_OK;
  TIK_CHECK_ARG(target_dev != nullptr && init_pose_dev != nullptr && pose_out_dev != nullptr, "fit_keypoints: null pointer");
  const bool use_betas = B > 0 && betas_dev != nullptr;
  const int64_t R = 3 * (int64_t)n_select;
  const void* ins[5] = {target_dev, weights_dev, init_pose_dev, use_betas ? betas_dev : nullptr, transl_dev};
  const int64_t in_n[5] = {F * R, weights_per_frame ? F * n_select : n_select, F * kFitPose,
                           betas_per_frame ? F * B : B, F * 3};
  const void* outs[3] = {pose_out_dev, transl_out_dev, cost_dev};
  const int64_t out_n[3] = {F * kFitPose, F * 3, F * 2};
  for (int o = 0; o < 3; ++o) {
    for (int i = 0; i < 5; ++i)
      TIK_CHECK_ARG(!fit_overlap(outs[o], out_n[o], ins[i], in_n[i]), "fit_keypoints: output %d overlaps input %d", o, i);
    for (int o2 = o + 1; o2 < 3; ++o2)
      TIK_CHECK_ARG(!fit_overlap(outs[o], out_n[o], outs[o2], out_n[o2]), "fit_keypoints: outputs %d and %d overlap", o, o2);
  }

  fit_model_params(m, &p);
  p.target = target_dev; p.weights = weights_dev; p.init_pose = init_pose_dev;
  p.betas = use_betas ? betas_dev : nullptr; p.transl = transl_dev;
  p.pose_out = pose_out_dev; p.transl_out = transl_out_dev; p.cost = cost_dev;
  p.F = F;
  p.n_betas = use_betas ? B : 0;          // no betas: the shape directions are not read at all
  p.weights_per_frame = weights_dev != nullptr ? weights_per_frame : 0;
  p.betas_per_frame = use_betas ? betas_per_frame : 0;

  // The model tables never need more than B = 16 directions; size the launch by the call's own shapes.
  const bool has_pd = p.lm_pd != nullptr && L > 0;
  if (!use_betas) { p.jd = nullptr; p.lm_d = nullptr; }
  const FitSmem sm = fit_smem(n_select, L, p.n_betas, has_pd);
  cudaStream_t s = (cudaStream_t)stream;
  int dev = 0, sms = 148, optin = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  TIK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  TIK_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const int64_t cta_bytes = 4 * (int64_t)sm.cta, warp_bytes = 4 * (int64_t)sm.warp;
  const int warps = (int)std::min<int64_t>(kFitMaxWarps, (optin - cta_bytes) / warp_bytes);
  TIK_CHECK_ARG(warps >= 1, "fit_keypoints: %lld bytes of shared memory per frame do not fit", (long long)warp_bytes);
  p.warps = warps;
  static bool attr_set[64] = {};
  if (!attr_set[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(fit_keypoints_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
    attr_set[dev & 63] = true;
  }
  const size_t smem = (size_t)(cta_bytes + warps * warp_bytes);
  int per_sm = 1;
  TIK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fit_keypoints_kernel, warps * 32, smem));
  const int64_t blocks = std::min<int64_t>(ceil_div(F, warps), (int64_t)sms * std::max(1, per_sm));
  fit_keypoints_kernel<<<(unsigned)blocks, warps * 32, smem, s>>>(p);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}
