// Fit one body shape per sequence: Levenberg-Marquardt over the betas of each sequence and the poses (and
// translations) of its frames, with the arrow-shaped normal equations solved by a Schur complement.  Sequence s has the
// frames [frame_start[s], frame_start[s+1]) and the cost
//
//   E_s = sum_{f in s} [ sum_k w_fk |kp_k(theta_f, beta_s, tau_f) - y_fk|^2 + lambda |theta_f - theta0_f|^2 ]
//         + lambda_beta |beta_s|^2.
//
// Per frame the pose block H_f (P x P, P = 66 or 69), g_f, the coupling C_f = J_x^T W J_beta (P x B), H_bb,f =
// J_beta^T W J_beta and g_b,f = J_beta^T W r are built by one warp with the forward, Jacobian and Cholesky of
// fit_device.cuh; the beta columns of J are
//   joint point k:  dt_k/dbeta = jd_root + sum_{m on the path root -> k, m != root} Rg_par(m) (jd_m - jd_par(m))
//   landmark l:     dv_l/dbeta = sum_m w_lm (Rg_m (lm_d_l - jd_m) + dt_m/dbeta).
// One iteration is four launches, with no host synchronisation (mu_s, E_s and the accept flags live in the workspace):
//   1. frame kernel (warp per frame): after an accepted step (or on the first pass) the forward and J at (x_f, beta_s)
//      and the blocks above, stored in the workspace; after a rejection the stored blocks are read back.  Then
//      L L^T = H_f + mu_s diag(H_f), b_f = -(H_f + mu D_f)^-1 g_f (fit_solve), Z = L^-1 C_f, S_f = H_bb,f - Z^T Z,
//      Y_f = L^-T Z = (H_f + mu D_f)^-1 C_f and r_f = g_b,f - Y_f^T g_f;
//   2. sequence kernel (CTA per sequence): the sums of S_f, r_f and diag(H_bb,f) in fp64, in an order fixed by the
//      frame's index in its sequence, and the fp64 Cholesky of
//        (sum S_f + lambda_beta I + mu diag(sum H_bb,f + lambda_beta I)) dbeta = -(sum r_f + lambda_beta beta);
//   3. candidate kernel (warp per frame): dx_f = b_f - Y_f dbeta, the forward at (x_f + dx_f, beta_s + dbeta), its cost;
//   4. accept kernel (CTA per sequence): the candidate cost in fp64 and the schedule of fit_keypoints per sequence.
// Nothing depends on where a sequence sits in the batch: a frame's work reads only its own data and its sequence's
// state, and every sum over a sequence runs in an order fixed by frame indices within the sequence.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "fit_device.cuh"

namespace tik {

constexpr int kShapeMaxB = TIK_KP_MAX_BETAS;
constexpr int kShapeSeqThreads = 640;                    // sequence kernel: chunks of frames x record entries
constexpr int kShapeAccThreads = 256;                    // accept kernel: a power of two (tree reduction)

struct ShapeSeq {                                        // state of one sequence in the workspace
  double E, E0;                                          // current and initial cost
  float beta[kShapeMaxB], dbeta[kShapeMaxB];
  float mu;
  int live;                                              // the initial cost is finite
  int acc;                                               // the last candidate was accepted
  int ok;                                                // the last solve had positive pivots
};

// Per-frame workspace arrays; strides in floats.
struct ShapeWs {
  float *H, *g, *C, *hb, *Y, *b, *x, *xc, *rec, *cost;
  int32_t* seq;
  ShapeSeq* st;
  int ht, hbs, recs;                                     // strides of H, of [H_bb | g_b] and of the Schur record
};

struct ShapeParams {
  FitParams f;                                           // model, inputs, selection, P, prior; f.n_betas = B
  ShapeWs w;
  const int64_t* frame_start;
  int64_t n_seqs;
  const float* betas_init;
  float* betas_out;
  float beta_prior;
};

__host__ __device__ inline int shape_up4(int n) { return (n + 3) / 4 * 4; }
__host__ __device__ inline int shape_tri(int n) { return n * (n + 1) / 2; }

// Extra per-warp regions of the frame kernel behind fit_smem's slice: J_beta (R x B), C / Z / Y (B columns of pitch
// kFitPitch), H_bb (B x B), g_b and a B-vector for the substitutions.
struct ShapeSmem { int jb, cz, hb, gb, tmp, warp; };
__host__ __device__ inline ShapeSmem shape_smem(const FitSmem& f, int n_sel, int B) {
  ShapeSmem s;
  int o = f.warp;
  s.jb = o;  o += shape_up4(3 * n_sel * B);
  s.cz = o;  o += B * kFitPitch;
  s.hb = o;  o += shape_up4(B * B);
  s.gb = o;  o += kShapeMaxB;
  s.tmp = o; o += kShapeMaxB;
  s.warp = o;
  return s;
}

// The warp slice of the kernels that only run the forward (start and candidate): no J, H, g, b, M or D.
__host__ __device__ inline FitSmem shape_fwd_smem(int n_sel, int L, int B, bool has_pd) {
  FitSmem s = fit_smem(n_sel, L, B, has_pd);             // the CTA tables as the fit stages them
  const int R = 3 * n_sel;
  int o = 0;
  s.U = s.H = s.g = s.b = s.M = s.D = 0;                 // never touched by fit_forward
  s.x = o;    o += kFitPitch;
  s.x0 = o;   o += kFitPitch;
  s.xc = o;   o += kFitPitch;
  s.y = o;    o += shape_up4(R);
  s.wr = o;   o += shape_up4(R);
  s.res = o;  o += shape_up4(R);
  s.beta = o; o += shape_up4(TIK_KP_MAX_BETAS);
  s.rest = o; o += shape_up4(kFitJ * 3);
  s.psh = o;  o += shape_up4(3 * L);
  s.p = o;    o += shape_up4(3 * L);
  s.v = o;    o += shape_up4(3 * L);
  s.Rl = o;   o += shape_up4(kFitBody * 9);
  s.Rg = o;   o += shape_up4(kFitJ * 9);
  s.t = o;    o += shape_up4(kFitJ * 3);
  s.warp = o;
  return s;
}

__device__ __forceinline__ void shape_range(const ShapeParams& p, int64_t s, int64_t* f0, int64_t* f1) {
  const int64_t F = p.f.F;
  const int64_t a = std::min<int64_t>(std::max<int64_t>(p.frame_start[s], 0), F);
  *f0 = a;
  *f1 = std::min<int64_t>(std::max<int64_t>(p.frame_start[s + 1], a), F);
}

// Sequence of frame f: the last s with frame_start[s] <= f, in [0, n_seqs) whatever the table holds.
__device__ __forceinline__ int64_t shape_seq_of(const ShapeParams& p, int64_t f) {
  int64_t lo = 0, hi = p.n_seqs - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) / 2;
    if (__ldg(p.frame_start + mid) <= f) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// beta of the sequence state (plus dbeta when cand) into s.beta, then the frame's rest points.
__device__ __forceinline__ void shape_frame_rest(const ShapeParams& p, const FitCta& c, const FitWarp& s, const ShapeSeq& q,
                                                 bool cand, int lane) {
  if (lane < p.f.n_betas) s.beta[lane] = cand ? q.beta[lane] + q.dbeta[lane] : q.beta[lane];
  __syncwarp();
  fit_shape_rest(p.f, c, s, lane);
  __syncwarp();
}

// J_beta (R x B, row-major) of the selected points at the last forward.  The joint derivatives dt/dbeta (55*3 x B)
// are built level by level in U and H, which are free until fit_normal_equations and hold >= 2 * kFitTri floats.
__device__ void shape_beta_jacobian(const FitParams& p, const FitCta& c, const FitWarp& s, float* Jb, int lane) {
  const int B = p.n_betas, n = p.n_sel;
  float* dT = s.U;
  for (int d = 0; d < p.n_levels; ++d) {
    const int j0 = p.level[d], nj = p.level[d + 1] - j0;
    for (int t = lane; t < nj * B; t += 32) {
      const int j = p.order[j0 + t / B], b = t % B, par = p.par[j];
      if (par < 0) {
#pragma unroll
        for (int r = 0; r < 3; ++r) dT[(j * 3 + r) * B + b] = c.jd[(j * 3 + r) * B + b];
      } else {
        const float* G = s.Rg + par * 9;
        const float e0 = c.jd[(j * 3) * B + b] - c.jd[(par * 3) * B + b];
        const float e1 = c.jd[(j * 3 + 1) * B + b] - c.jd[(par * 3 + 1) * B + b];
        const float e2 = c.jd[(j * 3 + 2) * B + b] - c.jd[(par * 3 + 2) * B + b];
#pragma unroll
        for (int r = 0; r < 3; ++r)
          dT[(j * 3 + r) * B + b] = fmaf(G[r * 3], e0, fmaf(G[r * 3 + 1], e1, fmaf(G[r * 3 + 2], e2, dT[(par * 3 + r) * B + b])));
      }
    }
    __syncwarp();
  }
  for (int t = lane; t < n * B; t += 32) {
    const int k = t / B, b = t % B, q = p.sel[k];
    float v[3];
    if (q < kFitJ) {
#pragma unroll
      for (int r = 0; r < 3; ++r) v[r] = dT[(q * 3 + r) * B + b];
    } else {
      const int l = q - kFitJ;
      v[0] = v[1] = v[2] = 0.f;
      for (int m = 0; m < kFitJ; ++m) {
        const float w = c.w[l * kFitJ + m];
        if (w == 0.f) continue;
        const float* G = s.Rg + m * 9;
        const float e0 = c.lmd[(l * 3) * B + b] - c.jd[(m * 3) * B + b];
        const float e1 = c.lmd[(l * 3 + 1) * B + b] - c.jd[(m * 3 + 1) * B + b];
        const float e2 = c.lmd[(l * 3 + 2) * B + b] - c.jd[(m * 3 + 2) * B + b];
#pragma unroll
        for (int r = 0; r < 3; ++r)
          v[r] = fmaf(w, fmaf(G[r * 3], e0, fmaf(G[r * 3 + 1], e1, fmaf(G[r * 3 + 2], e2, dT[(m * 3 + r) * B + b]))), v[r]);
      }
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) Jb[(3 * k + r) * B + b] = v[r];
  }
  __syncwarp();
}

// C = J_x^T W J_beta (column b at Cz + b * kFitPitch), H_bb = J_beta^T W J_beta (symmetric, B x B), g_b = J_beta^T W r.
__device__ void shape_coupling(const FitParams& p, const FitWarp& s, const float* Jb, float* Cz, float* hb, float* gb,
                               int lane) {
  const int B = p.n_betas, R = 3 * p.n_sel, P = p.P;
  for (int t = lane; t < P * B; t += 32) {
    const int b = t / P, a = t % P;
    float acc = 0.f;
    for (int r = 0; r < R; ++r) acc = fmaf(s.wr[r] * s.U[r * kFitPitch + a], Jb[r * B + b], acc);
    Cz[b * kFitPitch + a] = acc;
  }
  for (int t = lane; t < shape_tri(B); t += 32) {
    int a = 0;
    while (shape_tri(a + 1) <= t) ++a;
    const int b = t - shape_tri(a);
    float acc = 0.f;
    for (int r = 0; r < R; ++r) acc = fmaf(s.wr[r] * Jb[r * B + a], Jb[r * B + b], acc);
    hb[a * B + b] = acc;
    hb[b * B + a] = acc;
  }
  for (int b = lane; b < B; b += 32) {
    float acc = 0.f;
    for (int r = 0; r < R; ++r) acc = fmaf(s.wr[r] * Jb[r * B + b], s.res[r], acc);
    gb[b] = acc;
  }
  __syncwarp();
}

// Z <- L^-1 Z (forward) or L^-T Z (back) for the B columns of Z, L the packed factor of fit_solve; per column the
// arithmetic of fit_solve's substitutions.
__device__ void shape_substitute(const float* A, float* Z, float* tmp, int P, int B, bool back, int lane) {
  for (int s = 0; s < P; ++s) {
    const int k = back ? P - 1 - s : s;
    const float lkk = A[tri(k) + k];
    if (lane < B) tmp[lane] = Z[lane * kFitPitch + k] / lkk;
    __syncwarp();
    const int m = back ? k : P - 1 - k;                  // rows left to update: [0, k) or (k, P)
    for (int t = lane; t < m * B; t += 32) {
      const int cc = t / m, i = back ? t % m : k + 1 + t % m;
      const float l = back ? A[tri(k) + i] : A[tri(i) + k];
      Z[cc * kFitPitch + i] = fmaf(-l, tmp[cc], Z[cc * kFitPitch + i]);
    }
    if (lane < B) Z[lane * kFitPitch + k] = tmp[lane];
    __syncwarp();
  }
}

__global__ void shape_seq_init_kernel(const __grid_constant__ ShapeParams p) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= p.n_seqs) return;
  ShapeSeq& q = p.w.st[s];
  for (int b = 0; b < kShapeMaxB; ++b) {
    q.beta[b] = (b < p.f.n_betas && p.betas_init != nullptr) ? p.betas_init[s * p.f.n_betas + b] : 0.f;
    q.dbeta[b] = 0.f;
  }
  q.mu = 1e-3f;
  q.live = q.acc = q.ok = 0;
  q.E = q.E0 = 0.0;
}

// Start (cand = false: x from the inputs) or candidate (cand = true: x + dx at beta + dbeta): the forward and the frame cost.
template <bool cand>
__global__ void __launch_bounds__(kFitMaxWarps * 32)
shape_forward_kernel(const __grid_constant__ ShapeParams p) {
  extern __shared__ __align__(16) float fit_sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = blockDim.x >> 5;
  const FitParams& fp = p.f;
  const bool has_pd = fp.lm_pd != nullptr && fp.n_lm > 0;
  const FitSmem sm = shape_fwd_smem(fp.n_sel, fp.n_lm, fp.n_betas, has_pd);
  const FitCta c = fit_stage_cta(fp, sm, fit_sm, has_pd);
  __syncthreads();
  const FitWarp s = fit_warp_slice(fit_sm + sm.cta + warp * sm.warp, sm);
  const int B = fp.n_betas, P = fp.P;
  for (int64_t f = (int64_t)blockIdx.x * warps + warp; f < fp.F; f += (int64_t)gridDim.x * warps) {
    int64_t sq;
    if (!cand) {
      sq = shape_seq_of(p, f);
      if (lane == 0) p.w.seq[f] = (int32_t)sq;
    } else {
      sq = p.w.seq[f];
    }
    const ShapeSeq& q = p.w.st[sq];
    if (cand && !(q.live && q.ok)) continue;
    fit_load_start(fp, s, f, lane);                      // x0; x = the inputs' start
    fit_load_targets(fp, s, f, lane);
    if (cand) {
      const float* x = p.w.x + f * kFitPitch;
      const float* bv = p.w.b + f * kFitPitch;
      const float* Y = p.w.Y + f * (int64_t)(B * kFitPitch);
      for (int i = lane; i < kFitPitch; i += 32) {
        float d = 0.f;
        if (i < P) {
          d = bv[i];
          for (int k = 0; k < B; ++k) d = fmaf(-Y[k * kFitPitch + i], q.dbeta[k], d);
        }
        s.xc[i] = x[i] + d;
      }
    }
    shape_frame_rest(p, c, s, q, cand, lane);
    const float* xv = cand ? s.xc : s.x;
    const float E = fit_forward(fp, c, s, xv, lane);
    float* xo = (cand ? p.w.xc : p.w.x) + f * kFitPitch;
    for (int i = lane; i < kFitPitch; i += 32) xo[i] = xv[i];
    if (lane == 0) p.w.cost[f] = E;
    __syncwarp();
  }
}

// Phase 1: the damped frame blocks and their Schur contributions.
__global__ void __launch_bounds__(kFitMaxWarps * 32)
shape_frame_kernel(const __grid_constant__ ShapeParams p, int first) {
  extern __shared__ __align__(16) float fit_sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = blockDim.x >> 5;
  const FitParams& fp = p.f;
  const bool has_pd = fp.lm_pd != nullptr && fp.n_lm > 0;
  const int B = fp.n_betas, P = fp.P, TB = shape_tri(B);
  const FitSmem sm = fit_smem(fp.n_sel, fp.n_lm, B, has_pd);
  const ShapeSmem xs = shape_smem(sm, fp.n_sel, B);
  const FitCta c = fit_stage_cta(fp, sm, fit_sm, has_pd);
  __syncthreads();
  float* base = fit_sm + sm.cta + warp * xs.warp;
  const FitWarp s = fit_warp_slice(base, sm);
  float *Jb = base + xs.jb, *Cz = base + xs.cz, *hb = base + xs.hb, *gb = base + xs.gb, *tmp = base + xs.tmp;
  const ShapeWs& w = p.w;
  for (int64_t f = (int64_t)blockIdx.x * warps + warp; f < fp.F; f += (int64_t)gridDim.x * warps) {
    const ShapeSeq& q = w.st[w.seq[f]];
    if (!q.live) continue;
    float* Hw = w.H + f * w.ht;
    float* gw = w.g + f * kFitPitch;
    float* Cw = w.C + f * (int64_t)(B * kFitPitch);
    float* hw = w.hb + f * w.hbs;
    if (first || q.acc) {                                // new point: forward, J, blocks
      float* xw = w.x + f * kFitPitch;
      const float* src = first ? xw : w.xc + f * kFitPitch;
      fit_load_start(fp, s, f, lane);                    // x0 (x is replaced below)
      fit_load_targets(fp, s, f, lane);
      __syncwarp();
      for (int i = lane; i < kFitPitch; i += 32) {
        const float v = src[i];
        s.x[i] = v;
        xw[i] = v;
      }
      shape_frame_rest(p, c, s, q, false, lane);
      fit_forward(fp, c, s, s.x, lane);
      shape_beta_jacobian(fp, c, s, Jb, lane);
      fit_normal_equations(fp, c, s, lane);
      shape_coupling(fp, s, Jb, Cz, hb, gb, lane);
      for (int i = lane; i < tri(P); i += 32) Hw[i] = s.H[i];
      for (int i = lane; i < P; i += 32) gw[i] = s.g[i];
      for (int i = lane; i < B * kFitPitch; i += 32) Cw[i] = Cz[i];
      for (int i = lane; i < B * B; i += 32) hw[i] = hb[i];
      for (int i = lane; i < B; i += 32) hw[B * B + i] = gb[i];
    } else {                                             // rejected: only mu changed
      for (int i = lane; i < tri(P); i += 32) s.H[i] = Hw[i];
      for (int i = lane; i < P; i += 32) s.g[i] = gw[i];
      for (int i = lane; i < B * kFitPitch; i += 32) Cz[i] = Cw[i];
      for (int i = lane; i < B * B; i += 32) hb[i] = hw[i];
      for (int i = lane; i < B; i += 32) gb[i] = hw[B * B + i];
    }
    __syncwarp();
    float* rec = w.rec + f * w.recs;
    if (!fit_solve(fp, s, q.mu, lane)) {
      if (lane == 0) rec[TB + 2 * B] = 1.f;              // a pivot failed: the sequence rejects this step
      __syncwarp();
      continue;
    }
    shape_substitute(s.U, Cz, tmp, P, B, false, lane);   // Z = L^-1 C
    for (int t = lane; t < TB; t += 32) {                // S_f = H_bb - Z^T Z (lower triangle, rows in order)
      int a = 0;
      while (shape_tri(a + 1) <= t) ++a;
      const int b = t - shape_tri(a);
      float v = hb[a * B + b];
      for (int i = 0; i < P; ++i) v = fmaf(-Cz[a * kFitPitch + i], Cz[b * kFitPitch + i], v);
      rec[t] = v;
    }
    __syncwarp();
    shape_substitute(s.U, Cz, tmp, P, B, true, lane);    // Y = L^-T Z = (H + mu D)^-1 C
    for (int b = lane; b < B; b += 32) {
      float v = gb[b];
      for (int i = 0; i < P; ++i) v = fmaf(-Cz[b * kFitPitch + i], s.g[i], v);
      rec[TB + b] = v;                                   // r_f = g_b - C^T (H + mu D)^-1 g
      rec[TB + B + b] = hb[b * B + b];
    }
    if (lane == 0) rec[TB + 2 * B] = 0.f;
    float* Yw = w.Y + f * (int64_t)(B * kFitPitch);
    float* bw = w.b + f * kFitPitch;
    for (int i = lane; i < B * kFitPitch; i += 32) Yw[i] = Cz[i];
    for (int i = lane; i < kFitPitch; i += 32) bw[i] = i < P ? s.b[i] : 0.f;
    __syncwarp();
  }
}

// Phase 2: per sequence, the fp64 sums of the frame records and the B x B solve for dbeta.
__global__ void __launch_bounds__(kShapeSeqThreads)
shape_seq_kernel(const __grid_constant__ ShapeParams p) {
  __shared__ double part[kShapeSeqThreads];
  __shared__ double tot[kShapeSeqThreads];
  const int64_t sq = blockIdx.x;
  ShapeSeq& q = p.w.st[sq];
  if (!q.live) return;
  const int B = p.f.n_betas, TB = shape_tri(B), Q = p.w.recs, K = kShapeSeqThreads / Q;
  const int tid = threadIdx.x, e = tid % Q, ch = tid / Q;
  int64_t f0, f1;
  shape_range(p, sq, &f0, &f1);
  double acc = 0.0;
  if (ch < K && e <= TB + 2 * B)
    for (int64_t f = f0 + ch; f < f1; f += K) acc += (double)p.w.rec[f * Q + e];
  part[tid] = acc;
  __syncthreads();
  if (tid < Q) {
    double v = 0.0;
    for (int k = 0; k < K; ++k) v += part[k * Q + tid];
    tot[tid] = v;
  }
  __syncthreads();
  if (tid != 0) return;
  double M[kShapeMaxB * kShapeMaxB], rhs[kShapeMaxB];
  const double lb = p.beta_prior;
  for (int a = 0; a < B; ++a) {
    for (int b = 0; b <= a; ++b) M[a * B + b] = tot[shape_tri(a) + b];
    M[a * B + a] += lb + (double)q.mu * (tot[TB + B + a] + lb);
    rhs[a] = -(tot[TB + a] + lb * (double)q.beta[a]);
  }
  bool ok = tot[TB + 2 * B] == 0.0;
  for (int k = 0; k < B && ok; ++k) {                    // Cholesky, lower triangle in place
    double d = M[k * B + k];
    for (int j = 0; j < k; ++j) d -= M[k * B + j] * M[k * B + j];
    if (!(d > 0.0) || !(d < INFINITY)) { ok = false; break; }
    const double lk = sqrt(d);
    M[k * B + k] = lk;
    for (int i = k + 1; i < B; ++i) {
      double v = M[i * B + k];
      for (int j = 0; j < k; ++j) v -= M[i * B + j] * M[k * B + j];
      M[i * B + k] = v / lk;
    }
  }
  if (ok) {
    for (int k = 0; k < B; ++k) {
      double v = rhs[k];
      for (int j = 0; j < k; ++j) v -= M[k * B + j] * rhs[j];
      rhs[k] = v / M[k * B + k];
    }
    for (int k = B - 1; k >= 0; --k) {
      double v = rhs[k];
      for (int j = k + 1; j < B; ++j) v -= M[j * B + k] * rhs[j];
      rhs[k] = v / M[k * B + k];
    }
    for (int k = 0; k < B; ++k) q.dbeta[k] = (float)rhs[k];
  }
  q.ok = ok;
}

// Sum over the sequence's frames of w.cost in fp64: thread t takes frames f0 + t, f0 + t + T, ..., then a fixed tree.
__device__ double shape_cost_sum(const ShapeParams& p, int64_t sq, double* red) {
  int64_t f0, f1;
  shape_range(p, sq, &f0, &f1);
  const int tid = threadIdx.x;
  double acc = 0.0;
  for (int64_t f = f0 + tid; f < f1; f += kShapeAccThreads) acc += (double)p.w.cost[f];
  red[tid] = acc;
  __syncthreads();
  for (int o = kShapeAccThreads / 2; o > 0; o >>= 1) {
    if (tid < o) red[tid] += red[tid + o];
    __syncthreads();
  }
  return red[0];
}

// Start (init = 1): E0 of every sequence.  Step (init = 0): accept or reject the candidate (phase 4).
__global__ void __launch_bounds__(kShapeAccThreads)
shape_accept_kernel(const __grid_constant__ ShapeParams p, int init) {
  __shared__ double red[kShapeAccThreads];
  const int64_t sq = blockIdx.x;
  ShapeSeq& q = p.w.st[sq];
  const int B = p.f.n_betas;
  if (!init && !(q.live && q.ok)) {
    if (threadIdx.x == 0 && q.live) { q.acc = 0; q.mu = fminf(q.mu * 10.f, 1e7f); }
    return;
  }
  const double sum = shape_cost_sum(p, sq, red);
  if (threadIdx.x != 0) return;
  float bc[kShapeMaxB];
  double pr = 0.0;
  for (int k = 0; k < B; ++k) {
    bc[k] = init ? q.beta[k] : q.beta[k] + q.dbeta[k];
    pr += (double)bc[k] * (double)bc[k];
  }
  const double E = sum + (double)p.beta_prior * pr;
  if (init) {
    q.E = q.E0 = E;
    q.live = isfinite(E);
    return;
  }
  if (E < q.E) {
    q.E = E;
    for (int k = 0; k < B; ++k) q.beta[k] = bc[k];
    q.acc = 1;
    q.mu = fmaxf(q.mu / 10.f, 1e-7f);
  } else {
    q.acc = 0;
    q.mu = fminf(q.mu * 10.f, 1e7f);
  }
}

// The poses and translations of the last accepted point, then the betas and costs of every sequence.
__global__ void shape_output_kernel(const __grid_constant__ ShapeParams p, float* pose_out, float* transl_out, float* cost) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, F = p.f.F, B = p.f.n_betas;
  if (i < F * kFitMaxP) {
    const int64_t f = i / kFitMaxP;
    const int a = (int)(i % kFitMaxP);
    const ShapeSeq& q = p.w.st[p.w.seq[f]];
    const float v = (q.acc ? p.w.xc : p.w.x)[f * kFitPitch + a];
    if (a < kFitPose) pose_out[f * kFitPose + a] = v;
    else if (transl_out != nullptr) transl_out[f * 3 + a - kFitPose] = v;
    return;
  }
  const int64_t sq = i - F * kFitMaxP;
  if (sq >= p.n_seqs) return;
  const ShapeSeq& q = p.w.st[sq];
  for (int k = 0; k < B; ++k) p.betas_out[sq * B + k] = q.beta[k];
  if (cost != nullptr) {
    cost[sq * 2] = (float)q.E0;
    cost[sq * 2 + 1] = q.live ? (float)q.E : __int_as_float(0x7fc00000);
  }
}

// Workspace layout: per-frame arrays, then the sequence states; every array 256-byte aligned.
struct ShapeLayout { int64_t H, g, C, hb, Y, b, x, xc, rec, cost, seq, st, total; int ht, hbs, recs; };
static ShapeLayout shape_layout(int B, int P, int64_t F, int64_t S) {
  ShapeLayout l;
  l.ht = shape_up4(shape_tri(P));
  l.hbs = shape_up4(B * B + B);
  l.recs = shape_up4(shape_tri(B) + 2 * B + 1);
  int64_t o = 0;
  auto take = [&](int64_t bytes) { const int64_t at = o; o += (bytes + 255) / 256 * 256; return at; };
  l.H = take(4 * F * l.ht);
  l.g = take(4 * F * kFitPitch);
  l.C = take(4 * F * B * kFitPitch);
  l.hb = take(4 * F * l.hbs);
  l.Y = take(4 * F * B * kFitPitch);
  l.b = take(4 * F * kFitPitch);
  l.x = take(4 * F * kFitPitch);
  l.xc = take(4 * F * kFitPitch);
  l.rec = take(4 * F * l.recs);
  l.cost = take(4 * F);
  l.seq = take(4 * F);
  l.st = take((int64_t)sizeof(ShapeSeq) * S);
  l.total = o;
  return l;
}

}  // namespace tik

extern "C" int tik_fit_keypoints_shape_workspace_bytes(const TikKeypointModel* m, int n_select, int fit_transl, int64_t F,
                                                       int64_t n_seqs, int64_t* bytes) {
  using namespace tik;
  const char* fn = "fit_keypoints_shape";
  TIK_CHECK_ARG(m != nullptr && bytes != nullptr, "%s: null model or bytes", fn);
  TIK_CHECK_ARG(m->n_betas >= 1 && m->n_betas <= TIK_KP_MAX_BETAS, "%s: n_betas=%d outside [1,%d]", fn, m->n_betas,
                TIK_KP_MAX_BETAS);
  TIK_CHECK_ARG(n_select >= 1 && n_select <= TIK_KP_MAX_SELECT, "%s: n_select=%d outside [1,%d]", fn, n_select,
                TIK_KP_MAX_SELECT);
  TIK_CHECK_ARG(fit_transl == 0 || fit_transl == 1, "%s: fit_transl=%d must be 0 or 1", fn, fit_transl);
  TIK_CHECK_ARG(F >= 0 && n_seqs >= 0 && n_seqs <= F && (n_seqs >= 1) == (F >= 1),
                "%s: n_seqs=%lld for F=%lld (every sequence needs a frame)", fn, (long long)n_seqs, (long long)F);
  *bytes = F == 0 ? 0 : shape_layout(m->n_betas, fit_transl ? kFitMaxP : kFitPose, F, n_seqs).total;
  return TIK_OK;
}

extern "C" int tik_fit_keypoints_shape(const TikKeypointModel* m, const float* target_dev, const float* weights_dev,
                                       int weights_per_frame, const float* init_pose_dev, const float* transl_dev,
                                       int fit_transl, const int64_t* frame_start_dev, int64_t n_seqs,
                                       const float* betas_init_dev, float shape_prior_weight, const int32_t* select_host,
                                       int n_select, float prior_weight, int n_iter, int64_t F, void* workspace_dev,
                                       int64_t workspace_bytes, float* pose_out_dev, float* transl_out_dev,
                                       float* betas_out_dev, float* cost_dev, void* stream) {
  using namespace tik;
  const char* fn = "fit_keypoints_shape";
  TIK_CHECK_ARG(m != nullptr, "%s: null model", fn);
  if (int rc = fit_check_model(m, fn)) return rc;
  const int B = m->n_betas, L = m->n_landmarks;
  TIK_CHECK_ARG(B >= 1, "%s: the model has no shape directions (n_betas = 0)", fn);
  if (int rc = fit_check_weights(weights_dev, weights_per_frame, fn)) return rc;
  ShapeParams p;
  memset(&p, 0, sizeof(p));
  if (int rc = fit_check_solver(m, fit_transl, select_host, n_select, prior_weight, n_iter, F, &p.f, fn)) return rc;
  TIK_CHECK_ARG(shape_prior_weight > 0.f && shape_prior_weight < INFINITY,
                "%s: shape_prior_weight=%g must be positive and finite", fn, (double)shape_prior_weight);
  TIK_CHECK_ARG(n_seqs >= 0 && n_seqs <= F && (n_seqs >= 1) == (F >= 1),
                "%s: n_seqs=%lld for F=%lld (every sequence needs a frame)", fn, (long long)n_seqs, (long long)F);
  if (F == 0) return TIK_OK;
  TIK_CHECK_ARG(target_dev != nullptr && init_pose_dev != nullptr && frame_start_dev != nullptr && pose_out_dev != nullptr &&
                betas_out_dev != nullptr && workspace_dev != nullptr, "%s: null pointer", fn);
  const ShapeLayout lay = shape_layout(B, p.f.P, F, n_seqs);
  TIK_CHECK_ARG(workspace_bytes >= lay.total, "%s: workspace of %lld bytes, %lld needed", fn, (long long)workspace_bytes,
                (long long)lay.total);
  TIK_CHECK_ARG((uintptr_t)workspace_dev % 256 == 0, "%s: workspace_dev must be 256-byte aligned", fn);
  const int64_t R = 3 * (int64_t)n_select;
  const void* ins[6] = {target_dev, weights_dev, init_pose_dev, transl_dev, frame_start_dev, betas_init_dev};
  const int64_t in_n[6] = {F * R, weights_per_frame ? F * n_select : n_select, F * kFitPose, F * 3, 2 * (n_seqs + 1),
                           n_seqs * B};
  const void* outs[5] = {pose_out_dev, transl_out_dev, betas_out_dev, cost_dev, workspace_dev};
  const int64_t out_n[5] = {F * kFitPose, F * 3, n_seqs * B, n_seqs * 2, lay.total / 4};
  for (int o = 0; o < 5; ++o) {
    for (int i = 0; i < 6; ++i)
      TIK_CHECK_ARG(!fit_overlap(outs[o], out_n[o], ins[i], in_n[i]), "%s: output %d overlaps input %d", fn, o, i);
    for (int o2 = o + 1; o2 < 5; ++o2)
      TIK_CHECK_ARG(!fit_overlap(outs[o], out_n[o], outs[o2], out_n[o2]), "%s: outputs %d and %d overlap", fn, o, o2);
  }

  fit_model_params(m, &p.f);
  p.f.target = target_dev; p.f.weights = weights_dev; p.f.init_pose = init_pose_dev; p.f.transl = transl_dev;
  p.f.F = F;
  p.f.n_betas = B;
  p.f.weights_per_frame = weights_dev != nullptr ? weights_per_frame : 0;
  char* ws = (char*)workspace_dev;
  p.w.H = (float*)(ws + lay.H); p.w.g = (float*)(ws + lay.g); p.w.C = (float*)(ws + lay.C); p.w.hb = (float*)(ws + lay.hb);
  p.w.Y = (float*)(ws + lay.Y); p.w.b = (float*)(ws + lay.b); p.w.x = (float*)(ws + lay.x); p.w.xc = (float*)(ws + lay.xc);
  p.w.rec = (float*)(ws + lay.rec); p.w.cost = (float*)(ws + lay.cost); p.w.seq = (int32_t*)(ws + lay.seq);
  p.w.st = (ShapeSeq*)(ws + lay.st);
  p.w.ht = lay.ht; p.w.hbs = lay.hbs; p.w.recs = lay.recs;
  p.frame_start = frame_start_dev; p.n_seqs = n_seqs; p.betas_init = betas_init_dev; p.betas_out = betas_out_dev;
  p.beta_prior = shape_prior_weight;

  const bool has_pd = p.f.lm_pd != nullptr && L > 0;
  const FitSmem fsm = fit_smem(n_select, L, B, has_pd);
  const ShapeSmem xsm = shape_smem(fsm, n_select, B);
  const FitSmem vsm = shape_fwd_smem(n_select, L, B, has_pd);
  cudaStream_t s = (cudaStream_t)stream;
  int dev = 0, sms = 148, optin = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  TIK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  TIK_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const int64_t cta_bytes = 4 * (int64_t)fsm.cta;
  const int64_t frame_warp = 4 * (int64_t)xsm.warp, fwd_warp = 4 * (int64_t)vsm.warp;
  const int fw = (int)std::min<int64_t>(kFitMaxWarps, (optin - cta_bytes) / frame_warp);
  const int vw = (int)std::min<int64_t>(kFitMaxWarps, (optin - cta_bytes) / fwd_warp);
  TIK_CHECK_ARG(fw >= 1, "%s: %lld bytes of shared memory per frame do not fit", fn, (long long)frame_warp);
  static bool attr_set[64] = {};
  if (!attr_set[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(shape_frame_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
    TIK_CUDA(cudaFuncSetAttribute(shape_forward_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
    TIK_CUDA(cudaFuncSetAttribute(shape_forward_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
    attr_set[dev & 63] = true;
  }
  const size_t fsmem = (size_t)(cta_bytes + fw * frame_warp), vsmem = (size_t)(cta_bytes + vw * fwd_warp);
  int fper = 1, vper = 1;
  TIK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fper, shape_frame_kernel, fw * 32, fsmem));
  TIK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&vper, shape_forward_kernel<true>, vw * 32, vsmem));
  const unsigned fblocks = (unsigned)std::min<int64_t>(ceil_div(F, fw), (int64_t)sms * std::max(1, fper));
  const unsigned vblocks = (unsigned)std::min<int64_t>(ceil_div(F, vw), (int64_t)sms * std::max(1, vper));
  const unsigned S = (unsigned)n_seqs;

  shape_seq_init_kernel<<<(unsigned)ceil_div(n_seqs, 128), 128, 0, s>>>(p);
  shape_forward_kernel<false><<<vblocks, vw * 32, vsmem, s>>>(p);
  shape_accept_kernel<<<S, kShapeAccThreads, 0, s>>>(p, 1);
  for (int it = 0; it < n_iter; ++it) {
    shape_frame_kernel<<<fblocks, fw * 32, fsmem, s>>>(p, it == 0);
    shape_seq_kernel<<<S, kShapeSeqThreads, 0, s>>>(p);
    shape_forward_kernel<true><<<vblocks, vw * 32, vsmem, s>>>(p);
    shape_accept_kernel<<<S, kShapeAccThreads, 0, s>>>(p, 0);
  }
  shape_output_kernel<<<(unsigned)ceil_div(F * kFitMaxP + n_seqs, 256), 256, 0, s>>>(p, pose_out_dev, transl_out_dev,
                                                                                       cost_dev);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}
