// Device code of the keypoint fit shared by fit.cu (tik_fit_keypoints) and fit_shape.cu (tik_fit_keypoints_shape):
// the parameter block, the shared-memory layout of a frame, and the forward, normal equations and damped solve of one
// frame by one warp.  See fit.cu for the algorithm.
#pragma once
#include <math.h>

#include <algorithm>

#include "fk_device.cuh"

namespace tik {

constexpr int kFitJ = 55;
constexpr int kFitBody = 22;                              // joints with unknown rotations (0..21)
constexpr int kFitPose = 3 * kFitBody;                    // 66
constexpr int kFitMaxP = kFitPose + 3;                    // + translation
constexpr int kFitPitch = 72;                             // row pitch of J and length of the x vectors: 18 tiles of 4
constexpr int kFitTri = kFitMaxP * (kFitMaxP + 1) / 2;    // packed lower triangle of the 69 x 69 system
constexpr int kFitFeat = (kFitBody - 1) * 9;              // pose-blend features of joints 1..21
constexpr int kFitMaxWarps = 8;
constexpr int kFitMaxLevels = 16;

struct FitParams {
  const float* jt; const float* jd;
  const float* lm_t; const float* lm_d; const float* lm_pd;
  const int32_t* skin_idx; const float* skin_w;
  const float* target; const float* weights; const float* init_pose; const float* betas; const float* transl;
  float* pose_out; float* transl_out; float* cost;
  int64_t F;
  int n_betas, n_lm, kmax, n_sel, weights_per_frame, betas_per_frame, P, n_iter, warps, n_levels;
  float prior;
  unsigned long long anc[kFitJ];                          // bit a of anc[j]: joint a is j or an ancestor of j
  int8_t par[kFitJ];
  int8_t order[kFitJ];                                    // joints sorted by tree depth
  int8_t level[kFitMaxLevels + 1];                        // order[level[d] .. level[d+1]) have depth d
  int8_t sel[TIK_KP_MAX_SELECT];                          // point index of each selected point
};

// Shared-memory layout in floats, every region 16-byte aligned: CTA tables, then one slice per warp.
struct FitSmem {
  int pd, jt, jd, lmt, lmd, w, anc, cta;                  // CTA tables (offsets from 0)
  int U, H, g, b, x, x0, xc, y, wr, res, beta, rest, psh, p, v, Rl, Rg, t, M, D, warp;   // offsets in a warp slice
};
__host__ __device__ inline FitSmem fit_smem(int n_sel, int L, int B, bool has_pd) {
  auto up = [](int n) { return (n + 3) / 4 * 4; };
  FitSmem s;
  int o = 0;
  s.pd = o;   o += up(has_pd ? 3 * L * kFitFeat : 0);
  s.jt = o;   o += up(kFitJ * 3);
  s.jd = o;   o += up(kFitJ * 3 * B);
  s.lmt = o;  o += up(3 * L);
  s.lmd = o;  o += up(3 * L * B);
  s.w = o;    o += up(L * kFitJ);
  s.anc = o;  o += up(2 * kFitJ);
  s.cta = o;
  const int R = 3 * n_sel;
  o = 0;
  s.U = o;    o += up(R * kFitPitch > kFitTri ? R * kFitPitch : kFitTri);   // J, then the factor of the damped system
  s.H = o;    o += up(kFitTri);
  s.g = o;    o += kFitPitch;
  s.b = o;    o += kFitPitch;
  s.x = o;    o += kFitPitch;
  s.x0 = o;   o += kFitPitch;
  s.xc = o;   o += kFitPitch;
  s.y = o;    o += up(R);
  s.wr = o;   o += up(R);
  s.res = o;  o += up(R);
  s.beta = o; o += up(TIK_KP_MAX_BETAS);
  s.rest = o; o += up(kFitJ * 3);
  s.psh = o;  o += up(3 * L);
  s.p = o;    o += up(3 * L);
  s.v = o;    o += up(3 * L);
  s.Rl = o;   o += up(kFitBody * 9);
  s.Rg = o;   o += up(kFitJ * 9);
  s.t = o;    o += up(kFitJ * 3);
  s.M = o;    o += up(kFitBody * 9);
  s.D = o;    o += up(has_pd ? (kFitBody - 1) * 27 : 0);
  s.warp = o;
  return s;
}

struct FitCta { const float *pd, *jt, *jd, *lmt, *lmd, *w; const unsigned long long* anc; };
struct FitWarp { float *U, *H, *g, *b, *x, *x0, *xc, *y, *wr, *res, *beta, *rest, *psh, *p, *v, *Rl, *Rg, *t, *M, *D; };

// The CTA staging and per-frame loads of fit_keypoints_kernel, for the kernels of fit_shape.cu.  fit_keypoints_kernel
// keeps its own inline copy: calling these instead changes its register allocation (101 -> 99) and so its code.
// Stages the model tables of a CTA in shared memory (the caller synchronises the CTA before reading them).
__device__ __forceinline__ FitCta fit_stage_cta(const FitParams& p, const FitSmem& sm, float* fit_sm, bool has_pd) {
  const int tid = threadIdx.x, L = p.n_lm, B = p.n_betas;
  FitCta c;
  c.pd = has_pd ? fit_sm + sm.pd : nullptr;
  c.jt = fit_sm + sm.jt; c.jd = fit_sm + sm.jd; c.lmt = fit_sm + sm.lmt; c.lmd = fit_sm + sm.lmd; c.w = fit_sm + sm.w;
  c.anc = reinterpret_cast<const unsigned long long*>(fit_sm + sm.anc);
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
  return c;
}

__device__ __forceinline__ FitWarp fit_warp_slice(float* base, const FitSmem& sm) {
  FitWarp s;
  s.U = base + sm.U; s.H = base + sm.H; s.g = base + sm.g; s.b = base + sm.b; s.x = base + sm.x; s.x0 = base + sm.x0;
  s.xc = base + sm.xc; s.y = base + sm.y; s.wr = base + sm.wr; s.res = base + sm.res; s.beta = base + sm.beta;
  s.rest = base + sm.rest; s.psh = base + sm.psh; s.p = base + sm.p; s.v = base + sm.v; s.Rl = base + sm.Rl;
  s.Rg = base + sm.Rg; s.t = base + sm.t; s.M = base + sm.M; s.D = base + sm.D;
  return s;
}

// theta0 of frame f into x and x0, its translation (or 0) into x; x0 is 0 past the pose.
__device__ __forceinline__ void fit_load_start(const FitParams& p, const FitWarp& s, int64_t f, int lane) {
  for (int i = lane; i < kFitPose; i += 32) s.x[i] = s.x0[i] = __ldg(p.init_pose + f * kFitPose + i);
  if (lane < kFitPitch - kFitPose) {
    const int c3 = lane;
    s.x[kFitPose + c3] = (c3 < 3 && p.transl != nullptr) ? __ldg(p.transl + f * 3 + c3) : 0.f;
    s.x0[kFitPose + c3] = 0.f;
  }
}

// Targets y and per-row weights of frame f.
__device__ __forceinline__ void fit_load_targets(const FitParams& p, const FitWarp& s, int64_t f, int lane) {
  const int n = p.n_sel, R = 3 * n;
  for (int i = lane; i < R; i += 32) {
    s.y[i] = __ldg(p.target + f * R + i);
    s.wr[i] = p.weights == nullptr ? 1.f : __ldg(p.weights + (p.weights_per_frame ? f * n : 0) + i / 3);
  }
}

// Rest joints Jt + Jd beta and landmark rest points lm_t + lm_d beta of the betas in s.beta.
__device__ __forceinline__ void fit_shape_rest(const FitParams& p, const FitCta& c, const FitWarp& s, int lane) {
  const int L = p.n_lm, B = p.n_betas;
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
}

__device__ __forceinline__ float fit_warp_sum(float v) {
  // xor butterfly: every lane ends with the same bits (each step adds the same two partial sums on both sides)
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int tri(int i) { return i * (i + 1) / 2; }

// Keypoints of the pose xv (theta, tau), residuals and cost; leaves the frame's FK state (Rl, Rg, t, p) in shared memory.
static __device__ float fit_forward(const FitParams& p, const FitCta& c, const FitWarp& s, const float* xv, int lane) {
  const int L = p.n_lm, R = 3 * p.n_sel;
  if (lane < kFitBody) {
    float Rm[9];
    rodrigues_q_fast(xv[lane * 3], xv[lane * 3 + 1], xv[lane * 3 + 2], Rm);
#pragma unroll
    for (int e = 0; e < 9; ++e) s.Rl[lane * 9 + e] = Rm[e];
  }
  __syncwarp();
  for (int d = 0; d < p.n_levels; ++d) {
    for (int i = p.level[d] + lane; i < p.level[d + 1]; i += 32) {
      const int j = p.order[i], par = p.par[j];
      float* G = s.Rg + j * 9;
      float* tj = s.t + j * 3;
      if (par < 0) {
#pragma unroll
        for (int e = 0; e < 9; ++e) G[e] = s.Rl[j * 9 + e];
        tj[0] = s.rest[j * 3]; tj[1] = s.rest[j * 3 + 1]; tj[2] = s.rest[j * 3 + 2];
      } else {
        const float* GP = s.Rg + par * 9;
        const float* tp = s.t + par * 3;
        const float d0 = s.rest[j * 3] - s.rest[par * 3], d1 = s.rest[j * 3 + 1] - s.rest[par * 3 + 1],
                    d2 = s.rest[j * 3 + 2] - s.rest[par * 3 + 2];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          if (j < kFitBody) {
            const float* Rm = s.Rl + j * 9;
#pragma unroll
            for (int cc = 0; cc < 3; ++cc)
              G[r * 3 + cc] = GP[r * 3] * Rm[cc] + GP[r * 3 + 1] * Rm[3 + cc] + GP[r * 3 + 2] * Rm[6 + cc];
          } else {
            G[r * 3] = GP[r * 3]; G[r * 3 + 1] = GP[r * 3 + 1]; G[r * 3 + 2] = GP[r * 3 + 2];
          }
          tj[r] = GP[r * 3] * d0 + GP[r * 3 + 1] * d1 + GP[r * 3 + 2] * d2 + tp[r];
        }
      }
    }
    __syncwarp();
  }
  if (lane < 3 * L) {                                      // landmark rest positions: shape + pose blend
    float acc = 0.f;
    if (c.pd != nullptr) {
      const float* row = c.pd + lane * kFitFeat;
      for (int j = 1; j < kFitBody; ++j)
#pragma unroll
        for (int e = 0; e < 9; ++e)
          acc = fmaf(row[(j - 1) * 9 + e], s.Rl[j * 9 + e] - (e % 4 == 0 ? 1.f : 0.f), acc);
    }
    s.p[lane] = s.psh[lane] + acc;
  }
  __syncwarp();
  if (lane < 3 * L) {                                      // skinning: v_l = sum_m w_lm (Rg_m (p_l - rest_m) + t_m)
    const int l = lane / 3, cc = lane % 3;
    float v = 0.f;
    for (int m = 0; m < kFitJ; ++m) {
      const float w = c.w[l * kFitJ + m];
      if (w != 0.f) {
        const float qx = s.p[l * 3] - s.rest[m * 3], qy = s.p[l * 3 + 1] - s.rest[m * 3 + 1],
                    qz = s.p[l * 3 + 2] - s.rest[m * 3 + 2];
        const float* G = s.Rg + m * 9 + cc * 3;
        v = fmaf(w, fmaf(G[0], qx, fmaf(G[1], qy, fmaf(G[2], qz, s.t[m * 3 + cc]))), v);
      }
    }
    s.v[lane] = v;
  }
  __syncwarp();
  float e = 0.f, pr = 0.f;
  for (int i = lane; i < R; i += 32) {
    const int k = i / 3, cc = i % 3, q = p.sel[k];
    const float kp = (q < kFitJ ? s.t[q * 3 + cc] : s.v[(q - kFitJ) * 3 + cc]) + xv[kFitPose + cc];
    const float r = kp - s.y[i];
    s.res[i] = r;
    e = fmaf(s.wr[i] * r, r, e);
  }
  for (int i = lane; i < kFitPose; i += 32) {
    const float dl = xv[i] - s.x0[i];
    pr = fmaf(dl, dl, pr);
  }
  const float E = fit_warp_sum(e) + p.prior * fit_warp_sum(pr);
  __syncwarp();
  return E;
}

// J at the point of the last forward (x), then H (packed, lambda on the pose diagonal) and g.
static __device__ void fit_normal_equations(const FitParams& p, const FitCta& c, const FitWarp& s, int lane) {
  const int n = p.n_sel, R = 3 * n, P = p.P;
  const bool has_pd = c.pd != nullptr;
  if (lane < kFitBody) {
    // right Jacobian of the exponential map at theta_j, M_j = Rg_j Jr, and D_j,a = R_j [Jr e_a]x for the pose blend
    const float a0 = s.x[lane * 3], a1 = s.x[lane * 3 + 1], a2 = s.x[lane * 3 + 2];
    const float phi2 = a0 * a0 + a1 * a1 + a2 * a2;
    float ca, cb;                                          // Jr = I - ca [a]x + cb [a]x^2
    if (phi2 < 0.04f) {
      ca = 0.5f - phi2 * (1.f / 24.f - phi2 * (1.f / 720.f));
      cb = 1.f / 6.f - phi2 * (1.f / 120.f - phi2 * (1.f / 5040.f));
    } else {
      const float phi = sqrtf(phi2), sh = sinf(0.5f * phi);
      ca = 2.f * sh * sh / phi2;
      cb = (phi - sinf(phi)) / (phi2 * phi);
    }
    const float K[9] = {0.f, -a2, a1, a2, 0.f, -a0, -a1, a0, 0.f};
    float Jr[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) {
        const float k2 = K[r * 3] * K[cc] + K[r * 3 + 1] * K[3 + cc] + K[r * 3 + 2] * K[6 + cc];
        Jr[r * 3 + cc] = (r == cc ? 1.f : 0.f) - ca * K[r * 3 + cc] + cb * k2;
      }
    const float* G = s.Rg + lane * 9;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc)
        s.M[lane * 9 + r * 3 + cc] = G[r * 3] * Jr[cc] + G[r * 3 + 1] * Jr[3 + cc] + G[r * 3 + 2] * Jr[6 + cc];
    if (has_pd && lane >= 1) {
      const float* Rm = s.Rl + lane * 9;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const float u0 = Jr[a], u1 = Jr[3 + a], u2 = Jr[6 + a];
        const float S[9] = {0.f, -u2, u1, u2, 0.f, -u0, -u1, u0, 0.f};
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int cc = 0; cc < 3; ++cc)
            s.D[(lane - 1) * 27 + a * 9 + r * 3 + cc] = Rm[r * 3] * S[cc] + Rm[r * 3 + 1] * S[3 + cc] + Rm[r * 3 + 2] * S[6 + cc];
      }
    }
  }
  float4* U4 = reinterpret_cast<float4*>(s.U);
  for (int i = lane; i < R * (kFitPitch / 4); i += 32) U4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncwarp();
  for (int pi = lane; pi < n * kFitBody; pi += 32) {
    const int k = pi / kFitBody, j = pi % kFitBody, q = p.sel[k];
    const float* Mj = s.M + j * 9;
    float blk[9];
    bool nz = false;
    if (q < kFitJ) {
      if (q != j && ((c.anc[q] >> j) & 1ull)) {            // joint point below j: rotation about t_j
        const float d0 = s.t[q * 3] - s.t[j * 3], d1 = s.t[q * 3 + 1] - s.t[j * 3 + 1], d2 = s.t[q * 3 + 2] - s.t[j * 3 + 2];
#pragma unroll
        for (int a = 0; a < 3; ++a) {                      // column a: M_a x d
          const float m0 = Mj[a], m1 = Mj[3 + a], m2 = Mj[6 + a];
          blk[a] = m1 * d2 - m2 * d1; blk[3 + a] = m2 * d0 - m0 * d2; blk[6 + a] = m0 * d1 - m1 * d0;
        }
        nz = true;
      }
    } else {
      const int l = q - kFitJ;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, A[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const float* pl = s.p + l * 3;
      for (int m = 0; m < kFitJ; ++m) {
        const float w = c.w[l * kFitJ + m];
        if (w == 0.f) continue;
        const float* G = s.Rg + m * 9;
        if (has_pd)
#pragma unroll
          for (int e = 0; e < 9; ++e) A[e] = fmaf(w, G[e], A[e]);
        if ((c.anc[m] >> j) & 1ull) {                      // x_lm - t_j for every skinning joint m below (or at) j
          const float qx = pl[0] - s.rest[m * 3], qy = pl[1] - s.rest[m * 3 + 1], qz = pl[2] - s.rest[m * 3 + 2];
          s0 = fmaf(w, fmaf(G[0], qx, fmaf(G[1], qy, fmaf(G[2], qz, s.t[m * 3]))) - s.t[j * 3], s0);
          s1 = fmaf(w, fmaf(G[3], qx, fmaf(G[4], qy, fmaf(G[5], qz, s.t[m * 3 + 1]))) - s.t[j * 3 + 1], s1);
          s2 = fmaf(w, fmaf(G[6], qx, fmaf(G[7], qy, fmaf(G[8], qz, s.t[m * 3 + 2]))) - s.t[j * 3 + 2], s2);
        }
      }
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const float m0 = Mj[a], m1 = Mj[3 + a], m2 = Mj[6 + a];
        blk[a] = m1 * s2 - m2 * s1; blk[3 + a] = m2 * s0 - m0 * s2; blk[6 + a] = m0 * s1 - m1 * s0;
      }
      if (has_pd && j >= 1) {                              // (sum_m w_lm Rg_m) . d offset_l / d theta_j
        const float* D = s.D + (j - 1) * 27;
        float dp[9];
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) {
          const float* row = c.pd + (l * 3 + cc) * kFitFeat + (j - 1) * 9;
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            float v = 0.f;
#pragma unroll
            for (int e = 0; e < 9; ++e) v = fmaf(row[e], D[a * 9 + e], v);
            dp[cc * 3 + a] = v;
          }
        }
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int a = 0; a < 3; ++a)
            blk[r * 3 + a] += A[r * 3] * dp[a] + A[r * 3 + 1] * dp[3 + a] + A[r * 3 + 2] * dp[6 + a];
      }
      nz = true;
    }
    if (nz)
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int a = 0; a < 3; ++a) s.U[(3 * k + r) * kFitPitch + 3 * j + a] = blk[r * 3 + a];
  }
  if (P > kFitPose)
    for (int i = lane; i < R; i += 32) s.U[i * kFitPitch + kFitPose + i % 3] = 1.f;
  __syncwarp();

  // H: lanes over the 4x4 tiles of the lower triangle, rows in order
  const int nt = (P + 3) / 4, ntiles = nt * (nt + 1) / 2;
  for (int ti = lane; ti < ntiles; ti += 32) {
    int I = 0;
    while (tri(I + 1) <= ti) ++I;
    const int Jc = ti - tri(I);
    float acc[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) acc[e] = 0.f;
    for (int r = 0; r < R; ++r) {
      const float wr = s.wr[r];
      const float4 a4 = *reinterpret_cast<const float4*>(s.U + r * kFitPitch + 4 * I);
      const float4 b4 = *reinterpret_cast<const float4*>(s.U + r * kFitPitch + 4 * Jc);
      const float wa[4] = {wr * a4.x, wr * a4.y, wr * a4.z, wr * a4.w}, bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u * 4 + v] = fmaf(wa[u], bb[v], acc[u * 4 + v]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int i = 4 * I + u, j = 4 * Jc + v;
        if (j <= i && i < P) s.H[tri(i) + j] = acc[u * 4 + v] + (i == j && i < kFitPose ? p.prior : 0.f);
      }
  }
  for (int a = lane; a < P; a += 32) {
    float acc = 0.f;
    for (int r = 0; r < R; ++r) acc = fmaf(s.wr[r] * s.U[r * kFitPitch + a], s.res[r], acc);
    s.g[a] = acc + (a < kFitPose ? p.prior * (s.x[a] - s.x0[a]) : 0.f);
  }
  __syncwarp();
}

// (H + mu diag(H)) delta = -g by Cholesky in U; delta in b.  false: a pivot was not positive (or not finite).
static __device__ bool fit_solve(const FitParams& p, const FitWarp& s, float mu, int lane) {
  const int P = p.P;
  float* A = s.U;
  for (int i = lane; i < tri(P); i += 32) A[i] = s.H[i];
  for (int i = lane; i < P; i += 32) s.b[i] = -s.g[i];
  __syncwarp();
  for (int i = lane; i < P; i += 32) A[tri(i) + i] = fmaf(mu, s.H[tri(i) + i], s.H[tri(i) + i]);
  __syncwarp();
  for (int k = 0; k < P; ++k) {
    const float d = A[tri(k) + k];
    if (!(d > 0.f) || !(d < INFINITY)) return false;      // same value in every lane: the warp leaves together
    const float lk = sqrtf(d);
    __syncwarp();
    for (int i = k + 1 + lane; i < P; i += 32) A[tri(i) + k] /= lk;
    if (lane == 0) A[tri(k) + k] = lk;
    __syncwarp();
    for (int i = k + 1 + lane; i < P; i += 32) {
      const float lik = A[tri(i) + k];
      float* row = A + tri(i);
      int jk = tri(k + 1) + k;
      for (int j = k + 1; j <= i; ++j) {
        row[j] = fmaf(-lik, A[jk], row[j]);
        jk += j + 1;
      }
    }
    __syncwarp();
  }
  for (int k = 0; k < P; ++k) {                            // L y = -g
    const float yk = s.b[k] / A[tri(k) + k];
    __syncwarp();
    for (int i = k + 1 + lane; i < P; i += 32) s.b[i] = fmaf(-A[tri(i) + k], yk, s.b[i]);
    if (lane == 0) s.b[k] = yk;
    __syncwarp();
  }
  for (int k = P - 1; k >= 0; --k) {                       // L^T delta = y
    const float dk = s.b[k] / A[tri(k) + k];
    __syncwarp();
    for (int i = lane; i < k; i += 32) s.b[i] = fmaf(-A[tri(k) + i], dk, s.b[i]);
    if (lane == 0) s.b[k] = dk;
    __syncwarp();
  }
  return true;
}

// ---- host side shared by the two entry points; fn names the entry point in error messages

static bool fit_overlap(const void* a, int64_t na, const void* b, int64_t nb) {
  if (a == nullptr || b == nullptr || na <= 0 || nb <= 0) return false;
  const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
  return x < y + (uintptr_t)nb * 4 && y < x + (uintptr_t)na * 4;
}

static int fit_check_model(const TikKeypointModel* m, const char* fn) {
  const int B = m->n_betas, L = m->n_landmarks;
  TIK_CHECK_ARG(B >= 0 && B <= TIK_KP_MAX_BETAS, "%s: n_betas=%d outside [0,%d]", fn, B, TIK_KP_MAX_BETAS);
  TIK_CHECK_ARG(L >= 0 && L <= TIK_LBS_MAX_LANDMARKS, "%s: n_landmarks=%d outside [0,%d]", fn, L, TIK_LBS_MAX_LANDMARKS);
  TIK_CHECK_ARG(m->joint_template_dev != nullptr && (m->joint_dirs_dev != nullptr) == (B > 0),
                "%s: joint_template_dev must be set and joint_dirs_dev set iff n_betas > 0", fn);
  if (L > 0) {
    TIK_CHECK_ARG(m->kmax >= 1 && m->kmax <= kFitJ, "%s: kmax=%d outside [1,%d]", fn, m->kmax, kFitJ);
    TIK_CHECK_ARG(m->lm_template_dev && m->lm_skin_idx_dev && m->lm_skin_w_dev && (m->lm_dirs_dev != nullptr) == (B > 0),
                  "%s: landmark arrays missing (lm_dirs_dev must be set iff n_betas > 0)", fn);
  }
  return TIK_OK;
}

static int fit_check_weights(const float* weights_dev, int weights_per_frame, const char* fn) {
  TIK_CHECK_ARG(weights_per_frame == 0 || weights_per_frame == 1, "%s: weights_per_frame=%d must be 0 or 1", fn,
                weights_per_frame);
  TIK_CHECK_ARG(!(weights_per_frame && weights_dev == nullptr), "%s: per-frame weights need weights_dev", fn);
  return TIK_OK;
}

// The solver's arguments; fills the selection, P, n_iter and the prior of p.
static int fit_check_solver(const TikKeypointModel* m, int fit_transl, const int32_t* select_host, int n_select,
                            float prior_weight, int n_iter, int64_t F, FitParams* p, const char* fn) {
  const int L = m->n_landmarks;
  TIK_CHECK_ARG(fit_transl == 0 || fit_transl == 1, "%s: fit_transl=%d must be 0 or 1", fn, fit_transl);
  TIK_CHECK_ARG(n_select >= 1 && n_select <= TIK_KP_MAX_SELECT, "%s: n_select=%d outside [1,%d]", fn, n_select,
                TIK_KP_MAX_SELECT);
  TIK_CHECK_ARG(select_host != nullptr, "%s: null select_host", fn);
  TIK_CHECK_ARG(prior_weight > 0.f && prior_weight < INFINITY, "%s: prior_weight=%g must be positive and finite", fn,
                (double)prior_weight);
  TIK_CHECK_ARG(n_iter >= 0, "%s: n_iter=%d must be >= 0", fn, n_iter);
  TIK_CHECK_ARG(F >= 0, "%s: negative frame count", fn);
  for (int s = 0; s < n_select; ++s) {
    const int q = select_host[s];
    TIK_CHECK_ARG(q >= 0 && q < kFitJ + L, "%s: select[%d]=%d outside [0,%d)", fn, s, q, kFitJ + L);
    p->sel[s] = (int8_t)q;
  }
  p->n_sel = n_select;
  p->P = fit_transl ? kFitMaxP : kFitPose;
  p->n_iter = n_iter; p->prior = prior_weight;
  return TIK_OK;
}

// The model's arrays and the tree tables: ancestors (parents precede children), depth order.
static void fit_model_params(const TikKeypointModel* m, FitParams* p) {
  const int L = m->n_landmarks;
  p->jt = m->joint_template_dev; p->jd = m->joint_dirs_dev;
  p->lm_t = m->lm_template_dev; p->lm_d = m->lm_dirs_dev; p->lm_pd = m->lm_posedirs_dev;
  p->skin_idx = m->lm_skin_idx_dev; p->skin_w = m->lm_skin_w_dev;
  p->n_lm = L; p->kmax = L > 0 ? m->kmax : 0;
  int depth[kFitJ], maxd = 0;
  for (int j = 0; j < kFitJ; ++j) {
    const int par = f60_parent(j);
    p->par[j] = (int8_t)par;
    p->anc[j] = (par < 0 ? 0ull : p->anc[par]) | (1ull << j);
    depth[j] = par < 0 ? 0 : depth[par] + 1;
    maxd = std::max(maxd, depth[j]);
  }
  p->n_levels = maxd + 1;
  int o = 0;
  for (int d = 0; d <= maxd; ++d) {
    p->level[d] = (int8_t)o;
    for (int j = 0; j < kFitJ; ++j)
      if (depth[j] == d) p->order[o++] = (int8_t)j;
  }
  p->level[maxd + 1] = (int8_t)o;
}

}  // namespace tik
