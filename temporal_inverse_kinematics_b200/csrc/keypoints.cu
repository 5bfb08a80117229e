// Body keypoints straight from SMPL-X poses: the 55 FK joints and the landmark vertices of smplx's VertexJointSelector
// (nose, eyes, ears), without skinning the mesh.  One thread per frame, one launch per call:
//
//   1. pose blend of the landmarks: offset[3L] = sum_j posedirs_lm[:, 9(j-1)+e] (R_j - I)[e], one joint at a time
//      (Rodrigues of joint j, nine features, 9 x kRows FMAs with the posedirs rows read from shared memory as
//      broadcast float4); the 486 features are never stored;
//   2. rest skeleton of this frame's betas: rest_j = Jt_j + Jd_j . beta (Jt, Jd broadcast from shared memory);
//   3. FK over the compile-time SMPL-X tree (fk_bulk_kernel's recipe: fully unrolled, transforms in registers).  Not
//      pruned: a run-time skip of unneeded joints kept every transform live across the branches and put them in local
//      memory (2 KB of spills per thread); the whole tree fits in registers;
//   4. at each skinning joint j, v_l += w_lj (G_j (p_l - rest_j) + t_j) with p_l = lm_template + lm_dirs . beta +
//      offset_l: the lbs_skin_kernel formula sum_k w_k A_{j_k} p_l, A_j = [G_j | t_j - G_j rest_j], summed per joint;
//   5. the requested points (+ transl) into the frame's output row.
//
// Rodrigues runs twice per joint (blend pass and FK pass): keeping 54 rotations per thread would cost 2 KB of shared
// memory per frame.  Tiles of 64 contiguous frames come in (poses, per-frame betas, transl) and go out (points) through
// shared memory by cp.async.bulk; a ragged last tile or unaligned arrays are staged with ordinary loads and stores.
#include <string.h>

#include <algorithm>

#include "fk_device.cuh"

namespace tik {

constexpr int kKpJ = 55;
constexpr int kKpFeat = (kKpJ - 1) * 9;          // 486 pose features
constexpr int kKpFrames = 64;                    // frames per tile = threads per CTA
constexpr int kKpPoints = kKpJ + TIK_LBS_MAX_LANDMARKS;
constexpr int kKpWPitch = kKpJ + 1;              // dense landmark skinning weights [l][j]

struct KpParams {
  const float* jt; const float* jd;
  const float* lm_t; const float* lm_d; const float* lm_pd;
  const int32_t* skin_idx; const float* skin_w;
  const float* pose; const float* betas; const float* transl; float* out;
  int64_t F;
  int n_betas, n_lm, kmax, pose_J, n_rot, betas_per_frame, n_select, bulk;
  unsigned long long sel_mask;                   // joints written to the output
  int8_t slot[kKpPoints];                        // first output slot of each point, -1: not selected
  int8_t dup[TIK_KP_MAX_SELECT];                 // slot s repeats slot dup[s] (-1: written directly)
};

// Shared-memory layout in floats; every region starts on a 16-byte boundary (bulk-copy destinations, float4 reads).
struct KpSmem { int pd, jt, jd, dt, dd, lmt, lmd, w, bsh, pose, bet, tr, out, scr, scr_ld, total; };
__host__ __device__ inline KpSmem kp_smem(int rows, int nb, int pose_J, int n_lm, int n_betas, int n_select) {
  auto up = [](int n) { return (n + 3) / 4 * 4; };
  const int nbs = nb > 0 ? nb : 1;
  KpSmem s;
  int o = 0;
  s.pd = o;   o += up(kKpFeat * rows);
  s.jt = o;   o += up(kKpJ * 3);
  s.jd = o;   o += up(kKpJ * 3 * nbs);
  s.dt = o;   o += up(kKpJ * 3);
  s.dd = o;   o += up(kKpJ * 3 * nbs);
  s.lmt = o;  o += up(TIK_LBS_MAX_LANDMARKS * 3);
  s.lmd = o;  o += up(TIK_LBS_MAX_LANDMARKS * 3 * nbs);
  s.w = o;    o += up(TIK_LBS_MAX_LANDMARKS * kKpWPitch);
  s.bsh = o;  o += up(nbs);
  s.pose = o; o += up(kKpFrames * pose_J * 3);
  s.bet = o;  o += up(kKpFrames * n_betas);
  s.tr = o;   o += up(kKpFrames * 3);
  s.out = o;  o += up(kKpFrames * n_select * 3);
  s.scr_ld = 6 * n_lm + 1;                       // per frame: p_l then v_l; odd pitch
  s.scr = o;  o += up(kKpFrames * s.scr_ld);
  s.total = o;
  return s;
}

// kRows: posedirs rows held (3L padded to a multiple of 4, 16 for L <= 5, 24 for L <= 8); kNB: betas held (0: none,
// zero padded to 10 or 16).
template <int kRows, int kNB>
__global__ void __launch_bounds__(kKpFrames)
body_keypoints_kernel(const __grid_constant__ KpParams p) {
  constexpr int kL = kRows / 3;                  // landmarks held in registers
  constexpr int kR4 = kRows / 4;
  constexpr int kNBs = kNB > 0 ? kNB : 1;
  extern __shared__ __align__(16) float kp_sm[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ unsigned long long s_skin;
  const int tid = threadIdx.x;
  const int L = p.n_lm, B = p.n_betas;
  const bool has_pd = p.lm_pd != nullptr && L > 0;
  const KpSmem sm = kp_smem(kRows, kNB, p.pose_J, L, p.betas_per_frame ? B : 0, p.n_select);
  float* sPD = kp_sm + sm.pd;
  float* sJt = kp_sm + sm.jt;
  float* sJd = kp_sm + sm.jd;
  float* sDt = kp_sm + sm.dt;
  float* sDd = kp_sm + sm.dd;
  float* sLmt = kp_sm + sm.lmt;
  float* sLmd = kp_sm + sm.lmd;
  float* sW = kp_sm + sm.w;
  float* sBsh = kp_sm + sm.bsh;
  float* sPose = kp_sm + sm.pose;
  float* sBet = kp_sm + sm.bet;
  float* sTr = kp_sm + sm.tr;
  float* sOut = kp_sm + sm.out;
  float* sScr = kp_sm + sm.scr;

  // ---- model tables, once per CTA
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
    s_skin = 0ull;
  }
  for (int i = tid; i < kKpFeat * kRows; i += kKpFrames) {
    const int col = i / kRows, r = i % kRows;
    sPD[i] = (has_pd && r < 3 * L) ? __ldg(p.lm_pd + (int64_t)r * kKpFeat + col) : 0.f;
  }
  for (int i = tid; i < kKpJ * 3; i += kKpFrames) sJt[i] = __ldg(p.jt + i);
  for (int i = tid; i < kKpJ * 3 * kNB; i += kKpFrames) {
    const int k = i % kNBs;
    sJd[i] = k < B ? __ldg(p.jd + (i / kNBs) * B + k) : 0.f;
  }
  for (int i = tid; i < L * 3; i += kKpFrames) sLmt[i] = __ldg(p.lm_t + i);
  for (int i = tid; i < L * 3 * kNB; i += kKpFrames) {
    const int k = i % kNBs;
    sLmd[i] = k < B ? __ldg(p.lm_d + (i / kNBs) * B + k) : 0.f;
  }
  for (int i = tid; i < L * kKpJ; i += kKpFrames) {             // dense weights: repeated joints add up
    const int l = i / kKpJ, j = i % kKpJ;
    float w = 0.f;
    for (int k = 0; k < p.kmax; ++k)
      if (__ldg(p.skin_idx + l * p.kmax + k) == j) w += __ldg(p.skin_w + l * p.kmax + k);
    sW[l * kKpWPitch + j] = w;
  }
  __syncthreads();
  // parent offsets of Jt and Jd; the joint loop is unrolled so that every parent index is a compile-time constant
  static_assert(3 * (1 + kNB) <= kKpFrames, "one thread per offset entry of a joint");
#pragma unroll
  for (int j = 0; j < kKpJ; ++j) {
    constexpr int kNone = -1;
    const int par = f60_parent(j);
    if (tid < 3) {
      sDt[j * 3 + tid] = sJt[j * 3 + tid] - (par == kNone ? 0.f : sJt[par * 3 + tid]);
    } else if (tid < 3 * (1 + kNB)) {
      const int q = tid - 3;                                     // (c, k) of the joint's 3 x kNB block
      sDd[j * 3 * kNBs + q] = sJd[j * 3 * kNBs + q] - (par == kNone ? 0.f : sJd[par * 3 * kNBs + q]);
    }
  }
  if (kNB > 0 && !p.betas_per_frame && tid < kNB) sBsh[tid] = (p.betas != nullptr && tid < B) ? __ldg(p.betas + tid) : 0.f;
  __syncthreads();
  if (tid < kKpJ) {
    bool used = false;
    for (int l = 0; l < L; ++l) used |= sW[l * kKpWPitch + tid] != 0.f;
    if (used) atomicOr(&s_skin, 1ull << tid);
  }
  __syncthreads();
  const unsigned long long skin = s_skin, sel = p.sel_mask;
  const int prow = p.pose_J * 3, orow = p.n_select * 3;
  const int nbf = p.betas_per_frame ? B : 0;
  const bool has_tr = p.transl != nullptr;

  const int64_t n_tiles = (p.F + kKpFrames - 1) / kKpFrames;
  uint32_t phase = 0;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t f0 = tile * kKpFrames;
    const int nf = (int)min((int64_t)kKpFrames, p.F - f0);
    const bool bulk = p.bulk && nf == kKpFrames;
    if (tid == 0) tma_store_wait_read0();                        // the previous tile's points have left sOut
    if (bulk) {
      if (tid == 0) {
        fence_proxy_async_smem();
        const uint32_t bp = kKpFrames * prow * 4, bb = kKpFrames * nbf * 4, bt = has_tr ? kKpFrames * 12 : 0;
        mbar_expect_tx(&bar, bp + bb + bt);
        bulk_load_1d(sPose, p.pose + f0 * prow, bp, &bar);
        if (bb) bulk_load_1d(sBet, p.betas + f0 * nbf, bb, &bar);
        if (bt) bulk_load_1d(sTr, p.transl + f0 * 3, bt, &bar);
      }
      mbar_wait(&bar, phase);
      phase ^= 1u;
    } else {
      __syncthreads();
      for (int i = tid; i < nf * prow; i += kKpFrames) sPose[i] = __ldg(p.pose + f0 * prow + i);
      for (int i = tid; i < nf * nbf; i += kKpFrames) sBet[i] = __ldg(p.betas + f0 * nbf + i);
      if (has_tr)
        for (int i = tid; i < nf * 3; i += kKpFrames) sTr[i] = __ldg(p.transl + f0 * 3 + i);
      __syncthreads();
    }

    if (tid < nf) {
      const float* aa = sPose + tid * prow;
      float* orow_s = sOut + tid * orow;
      float* scr = sScr + tid * sm.scr_ld;
      const float* brow = p.betas_per_frame ? sBet + tid * B : sBsh;
      float beta[kNBs];
#pragma unroll
      for (int k = 0; k < kNBs; ++k) beta[k] = (kNB > 0 && k < (p.betas_per_frame ? B : kNB)) ? brow[k] : 0.f;
      const float tx = has_tr ? sTr[tid * 3] : 0.f, ty = has_tr ? sTr[tid * 3 + 1] : 0.f, tz = has_tr ? sTr[tid * 3 + 2] : 0.f;

      // ---- 1. landmark pose blend
      float acc[kRows];
#pragma unroll
      for (int r = 0; r < kRows; ++r) acc[r] = 0.f;
      if (has_pd) {
        const float4* pd4 = reinterpret_cast<const float4*>(sPD);
#pragma unroll 1
        for (int j = 1; j < p.n_rot; ++j) {
          float R[9];
          rodrigues_q_fast(aa[j * 3], aa[j * 3 + 1], aa[j * 3 + 2], R);
          R[0] -= 1.f; R[4] -= 1.f; R[8] -= 1.f;
          const float4* col = pd4 + (j - 1) * 9 * kR4;
#pragma unroll
          for (int e = 0; e < 9; ++e)
#pragma unroll
            for (int q = 0; q < kR4; ++q) {
              const float4 w = col[e * kR4 + q];
              acc[4 * q] = fmaf(w.x, R[e], acc[4 * q]);
              acc[4 * q + 1] = fmaf(w.y, R[e], acc[4 * q + 1]);
              acc[4 * q + 2] = fmaf(w.z, R[e], acc[4 * q + 2]);
              acc[4 * q + 3] = fmaf(w.w, R[e], acc[4 * q + 3]);
            }
        }
      }
      // shaped + blended landmark rest positions p_l, skinned sums v_l = 0
#pragma unroll
      for (int l = 0; l < kL; ++l) {
        if (l < L) {
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            float v = sLmt[l * 3 + c];
#pragma unroll
            for (int k = 0; k < kNB; ++k) v = fmaf(sLmd[(l * 3 + c) * kNB + k], beta[k], v);
            scr[l * 3 + c] = v + acc[l * 3 + c];
            scr[3 * L + l * 3 + c] = 0.f;
          }
        }
      }

      // ---- 2-4. rest skeleton, FK, skinning
      float GR[kKpJ][9], Gt[kKpJ][3];
#pragma unroll
      for (int j = 0; j < kKpJ; ++j) {
        {
          float R[9];
          if (j < p.n_rot) {
            rodrigues_q_fast(aa[j * 3], aa[j * 3 + 1], aa[j * 3 + 2], R);
          } else {
#pragma unroll
            for (int k = 0; k < 9; ++k) R[k] = (k % 4 == 0) ? 1.f : 0.f;
          }
          float d[3];                                              // offset to the parent (root: rest position)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            float v = sDt[j * 3 + c];
#pragma unroll
            for (int k = 0; k < kNB; ++k) v = fmaf(sDd[(j * 3 + c) * kNB + k], beta[k], v);
            d[c] = v;
          }
          const int par = f60_parent(j);
          if (par < 0) {
#pragma unroll
            for (int k = 0; k < 9; ++k) GR[j][k] = R[k];
            Gt[j][0] = d[0]; Gt[j][1] = d[1]; Gt[j][2] = d[2];
          } else {
#pragma unroll
            for (int r = 0; r < 3; ++r) {
#pragma unroll
              for (int c = 0; c < 3; ++c)
                GR[j][r * 3 + c] = GR[par][r * 3] * R[c] + GR[par][r * 3 + 1] * R[3 + c] + GR[par][r * 3 + 2] * R[6 + c];
              Gt[j][r] = GR[par][r * 3] * d[0] + GR[par][r * 3 + 1] * d[1] + GR[par][r * 3 + 2] * d[2] + Gt[par][r];
            }
          }
          if ((sel >> j) & 1ull) {
            float* o = orow_s + p.slot[j] * 3;
            o[0] = Gt[j][0] + tx; o[1] = Gt[j][1] + ty; o[2] = Gt[j][2] + tz;
          }
          if ((skin >> j) & 1ull) {
            float r[3];                                            // absolute rest position of the skinning joint
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              float v = sJt[j * 3 + c];
#pragma unroll
              for (int k = 0; k < kNB; ++k) v = fmaf(sJd[(j * 3 + c) * kNB + k], beta[k], v);
              r[c] = v;
            }
#pragma unroll 1
            for (int l = 0; l < L; ++l) {                         // v_l += w_lj (G_j (p_l - rest_j) + t_j)
              const float w = sW[l * kKpWPitch + j];
              if (w != 0.f) {
                const float qx = scr[l * 3] - r[0], qy = scr[l * 3 + 1] - r[1], qz = scr[l * 3 + 2] - r[2];
                float* v = scr + 3 * L + l * 3;
                v[0] = fmaf(w, fmaf(GR[j][0], qx, fmaf(GR[j][1], qy, fmaf(GR[j][2], qz, Gt[j][0]))), v[0]);
                v[1] = fmaf(w, fmaf(GR[j][3], qx, fmaf(GR[j][4], qy, fmaf(GR[j][5], qz, Gt[j][1]))), v[1]);
                v[2] = fmaf(w, fmaf(GR[j][6], qx, fmaf(GR[j][7], qy, fmaf(GR[j][8], qz, Gt[j][2]))), v[2]);
              }
            }
          }
        }
      }

      // ---- 5. landmark points, then repeated selections
      for (int l = 0; l < L; ++l) {
        const int s = p.slot[kKpJ + l];
        if (s >= 0) {
          float* o = orow_s + s * 3;
          const float* v = scr + 3 * L + l * 3;
          o[0] = v[0] + tx; o[1] = v[1] + ty; o[2] = v[2] + tz;
        }
      }
      for (int s = 0; s < p.n_select; ++s) {
        const int d = p.dup[s];
        if (d >= 0) {
          orow_s[s * 3] = orow_s[d * 3]; orow_s[s * 3 + 1] = orow_s[d * 3 + 1]; orow_s[s * 3 + 2] = orow_s[d * 3 + 2];
        }
      }
    }

    if (bulk) {
      fence_proxy_async_smem();                                  // st.shared -> visible to the bulk store
      __syncthreads();
      if (tid == 0) {
        bulk_store_1d(p.out + f0 * orow, sOut, (uint32_t)(kKpFrames * orow * 4));
        tma_store_commit();
      }
    } else {
      __syncthreads();
      for (int i = tid; i < nf * orow; i += kKpFrames) p.out[f0 * orow + i] = sOut[i];
      __syncthreads();
    }
  }
  if (tid == 0) tma_store_wait0();
}

template <int kRows, int kNB>
static int launch_keypoints(const KpParams& p, int sms, cudaStream_t s) {
  auto kern = body_keypoints_kernel<kRows, kNB>;
  static bool attr_set[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  const int smax = (int)sizeof(float) *
                   kp_smem(kRows, kNB, 60, kRows / 3, TIK_KP_MAX_BETAS, TIK_KP_MAX_SELECT).total;
  if (!attr_set[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smax));
    attr_set[dev & 63] = true;
  }
  const size_t smem = sizeof(float) *
                      (size_t)kp_smem(kRows, kNB, p.pose_J, p.n_lm, p.betas_per_frame ? p.n_betas : 0, p.n_select).total;
  int per_sm = 1;
  TIK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kKpFrames, smem));
  const int64_t n_tiles = ceil_div(p.F, kKpFrames);
  const int64_t blocks = std::min<int64_t>(n_tiles, (int64_t)sms * std::max(1, per_sm));
  kern<<<(unsigned)blocks, kKpFrames, smem, s>>>(p);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}

}  // namespace tik

extern "C" int tik_body_keypoints(const TikKeypointModel* m, const float* pose_dev, int pose_J, const float* betas_dev,
                                  int betas_per_frame, const float* transl_dev, const int32_t* select_host, int n_select,
                                  int64_t F, float* out_dev, void* stream) {
  using namespace tik;
  TIK_CHECK_ARG(m != nullptr, "keypoints: null model");
  const int B = m->n_betas, L = m->n_landmarks;
  TIK_CHECK_ARG(B >= 0 && B <= TIK_KP_MAX_BETAS, "keypoints: n_betas=%d outside [0,%d]", B, TIK_KP_MAX_BETAS);
  TIK_CHECK_ARG(L >= 0 && L <= TIK_LBS_MAX_LANDMARKS, "keypoints: n_landmarks=%d outside [0,%d]", L, TIK_LBS_MAX_LANDMARKS);
  TIK_CHECK_ARG(m->joint_template_dev != nullptr && (m->joint_dirs_dev != nullptr) == (B > 0),
                "keypoints: joint_template_dev must be set and joint_dirs_dev set iff n_betas > 0");
  if (L > 0) {
    TIK_CHECK_ARG(m->kmax >= 1 && m->kmax <= kKpJ, "keypoints: kmax=%d outside [1,%d]", m->kmax, kKpJ);
    TIK_CHECK_ARG(m->lm_template_dev && m->lm_skin_idx_dev && m->lm_skin_w_dev && (m->lm_dirs_dev != nullptr) == (B > 0),
                  "keypoints: landmark arrays missing (lm_dirs_dev must be set iff n_betas > 0)");
  }
  TIK_CHECK_ARG(pose_J == 22 || pose_J == kKpJ || pose_J == 60, "keypoints: pose_J=%d must be 22, 55 or 60", pose_J);
  TIK_CHECK_ARG(betas_per_frame == 0 || betas_per_frame == 1, "keypoints: betas_per_frame=%d must be 0 or 1", betas_per_frame);
  TIK_CHECK_ARG(!(betas_per_frame && betas_dev == nullptr && B > 0), "keypoints: per-frame betas need betas_dev");
  TIK_CHECK_ARG(n_select >= 1 && n_select <= TIK_KP_MAX_SELECT, "keypoints: n_select=%d outside [1,%d]", n_select, TIK_KP_MAX_SELECT);
  TIK_CHECK_ARG(select_host != nullptr, "keypoints: null select_host");
  TIK_CHECK_ARG(F >= 0, "negative frame count");
  KpParams p;
  memset(&p, 0, sizeof(p));
  for (int i = 0; i < kKpPoints; ++i) p.slot[i] = -1;
  for (int s = 0; s < n_select; ++s) {
    const int q = select_host[s];
    TIK_CHECK_ARG(q >= 0 && q < kKpJ + L, "keypoints: select[%d]=%d outside [0,%d)", s, q, kKpJ + L);
    p.dup[s] = p.slot[q] >= 0 ? p.slot[q] : -1;
    if (p.slot[q] < 0) p.slot[q] = (int8_t)s;
    if (q < kKpJ) p.sel_mask |= 1ull << q;
  }
  if (F == 0) return TIK_OK;
  TIK_CHECK_ARG(pose_dev != nullptr && out_dev != nullptr, "null pointer");
  const bool use_betas = B > 0 && betas_dev != nullptr;
  p.jt = m->joint_template_dev; p.jd = m->joint_dirs_dev;
  p.lm_t = m->lm_template_dev; p.lm_d = m->lm_dirs_dev; p.lm_pd = m->lm_posedirs_dev;
  p.skin_idx = m->lm_skin_idx_dev; p.skin_w = m->lm_skin_w_dev;
  p.pose = pose_dev; p.betas = use_betas ? betas_dev : nullptr; p.transl = transl_dev; p.out = out_dev;
  p.F = F;
  p.n_betas = B; p.n_lm = L; p.kmax = L > 0 ? m->kmax : 0; p.pose_J = pose_J; p.n_rot = std::min(pose_J, kKpJ);
  p.betas_per_frame = use_betas ? betas_per_frame : 0;
  p.n_select = n_select;
  const uintptr_t per_frame = (uintptr_t)pose_dev | (uintptr_t)out_dev | (uintptr_t)transl_dev |
                              (p.betas_per_frame ? (uintptr_t)betas_dev : 0);
  p.bulk = (per_frame & 15) == 0;
  cudaStream_t s = (cudaStream_t)stream;
  int dev = 0, sms = 148;
  TIK_CUDA(cudaGetDevice(&dev));
  TIK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int nb = use_betas ? (B <= 10 ? 10 : 16) : 0;
  if (L <= 5) {
    if (nb == 0) return launch_keypoints<16, 0>(p, sms, s);
    if (nb == 10) return launch_keypoints<16, 10>(p, sms, s);
    return launch_keypoints<16, 16>(p, sms, s);
  }
  if (nb == 0) return launch_keypoints<24, 0>(p, sms, s);
  if (nb == 10) return launch_keypoints<24, 10>(p, sms, s);
  return launch_keypoints<24, 16>(p, sms, s);
}
