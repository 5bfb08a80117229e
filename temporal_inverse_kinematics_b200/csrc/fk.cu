// Body forward kinematics: one warp per frame, one lane per joint.
//
//   G_0 = [R_0 | j_0],  G_i = G_parent(i) . [R_i | j_i - j_parent(i)],  joint_i = translation of G_i (+ transl)
//
// Replaces the joint output of common/smpl_util.py:67-70 (third-party smplx forward; SURVEY.md 8c).
// The chain is evaluated by pointer jumping over the kinematic tree: in round r every lane composes
// its accumulated transform with that of its 2^r-th ancestor, fetched with warp shuffles, so a tree
// of depth D needs ceil(log2(D+1)) rounds of 12 shuffles (3 for the 22-joint SMPL-X body, depth 7)
// instead of one round per tree level.  Inputs/outputs are staged per warp through shared memory so
// that global traffic is contiguous.  HBM-bound: 264 B in, 264 + 792 B out per frame (aa in,
// joints + local rotmats out).
#include <string.h>

#include <stdlib.h>

#include <algorithm>

#include "tik_common.cuh"
#include "umma_ptx.cuh"
#include "fk_device.cuh"

namespace tik {

struct FkParams {
  float rest[TIK_MAX_JOINTS * 3];  // offset to parent (root: rest position), precomputed on host
  int8_t parent[TIK_MAX_JOINTS];
  int J;
  int rounds;
};

constexpr int kFkWarps = 8;

__device__ __forceinline__ void rodrigues_q(float ax, float ay, float az, float* R) {
  // common/geometry.py:22-65
  float ex = ax + 1e-8f, ey = ay + 1e-8f, ez = az + 1e-8f;
  float ang = sqrtf(ex * ex + ey * ey + ez * ez);
  float ia = 1.0f / ang;
  float nx = ax * ia, ny = ay * ia, nz = az * ia;
  float s, c;
  sincosf(ang * 0.5f, &s, &c);
  float w = c, x = s * nx, y = s * ny, z = s * nz;
  float iq = rsqrtf(w * w + x * x + y * y + z * z);   // quaternion re-normalisation (quat2mat, geometry.py:49)
  w *= iq; x *= iq; y *= iq; z *= iq;
  float w2 = w * w, x2 = x * x, y2 = y * y, z2 = z * z;
  float wx = w * x, wy = w * y, wz = w * z, xy = x * y, xz = x * z, yz = y * z;
  R[0] = w2 + x2 - y2 - z2; R[1] = 2.f * xy - 2.f * wz;   R[2] = 2.f * wy + 2.f * xz;
  R[3] = 2.f * wz + 2.f * xy; R[4] = w2 - x2 + y2 - z2;   R[5] = 2.f * yz - 2.f * wx;
  R[6] = 2.f * xz - 2.f * wy; R[7] = 2.f * wx + 2.f * yz; R[8] = w2 - x2 - y2 + z2;
}

template <bool kRotIn>
__global__ void __launch_bounds__(kFkWarps * 32)
fk_kernel(const float* __restrict__ pose, const float* __restrict__ transl, float* __restrict__ joints,
          float* __restrict__ localR, float* __restrict__ globalR, int64_t F, const __grid_constant__ FkParams p) {
  constexpr int IN = kRotIn ? 9 : 3;
  __shared__ __align__(16) float s_io[kFkWarps][32 * 9];     // this kernel serves J <= 32 (one lane per joint)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int J = p.J;
  const bool active = lane < J;
  const int par0 = active ? p.parent[lane] : -1;
  const float dx = active ? p.rest[lane * 3 + 0] : 0.f;
  const float dy = active ? p.rest[lane * 3 + 1] : 0.f;
  const float dz = active ? p.rest[lane * 3 + 2] : 0.f;
  float* st = s_io[warp];
  const int64_t warps_total = (int64_t)gridDim.x * kFkWarps;

  for (int64_t f = (int64_t)blockIdx.x * kFkWarps + warp; f < F; f += warps_total) {
    // ---- coalesced load of this frame's pose into the warp's staging row
    const float* gp = pose + f * (int64_t)J * IN;
    for (int i = lane; i < J * IN; i += 32) st[i] = __ldg(gp + i);
    __syncwarp();
    float R[9];
    if (active) {
      if (kRotIn) {
#pragma unroll
        for (int k = 0; k < 9; ++k) R[k] = st[lane * 9 + k];
      } else {
        rodrigues_q(st[lane * 3], st[lane * 3 + 1], st[lane * 3 + 2], R);
      }
    } else {
#pragma unroll
      for (int k = 0; k < 9; ++k) R[k] = (k % 4 == 0) ? 1.f : 0.f;
    }
    __syncwarp();
    if (localR != nullptr) {
      if (active) {
#pragma unroll
        for (int k = 0; k < 9; ++k) st[lane * 9 + k] = R[k];
      }
      __syncwarp();
      float* go = localR + f * (int64_t)J * 9;
      for (int i = lane; i < J * 9; i += 32) go[i] = st[i];
      __syncwarp();
    }
    // ---- pointer jumping
    float tx = dx, ty = dy, tz = dz;
    int anc = par0;
    for (int r = 0; r < p.rounds; ++r) {
      const int src = anc < 0 ? lane : anc;
      float A[9], ax, ay, az;
#pragma unroll
      for (int k = 0; k < 9; ++k) A[k] = __shfl_sync(0xffffffffu, R[k], src);
      ax = __shfl_sync(0xffffffffu, tx, src);
      ay = __shfl_sync(0xffffffffu, ty, src);
      az = __shfl_sync(0xffffffffu, tz, src);
      const int anc2 = __shfl_sync(0xffffffffu, anc, src);
      if (anc >= 0) {
        float ntx = A[0] * tx + A[1] * ty + A[2] * tz + ax;
        float nty = A[3] * tx + A[4] * ty + A[5] * tz + ay;
        float ntz = A[6] * tx + A[7] * ty + A[8] * tz + az;
        float N[9];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int j = 0; j < 3; ++j) N[i * 3 + j] = A[i * 3] * R[j] + A[i * 3 + 1] * R[3 + j] + A[i * 3 + 2] * R[6 + j];
#pragma unroll
        for (int k = 0; k < 9; ++k) R[k] = N[k];
        tx = ntx; ty = nty; tz = ntz;
        anc = anc2;
      }
    }
    if (transl != nullptr) {
      tx += __ldg(transl + f * 3 + 0);
      ty += __ldg(transl + f * 3 + 1);
      tz += __ldg(transl + f * 3 + 2);
    }
    // ---- coalesced stores
    if (active) { st[lane * 3] = tx; st[lane * 3 + 1] = ty; st[lane * 3 + 2] = tz; }
    __syncwarp();
    float* gj = joints + f * (int64_t)J * 3;
    for (int i = lane; i < J * 3; i += 32) gj[i] = st[i];
    __syncwarp();
    if (globalR != nullptr) {
      if (active) {
#pragma unroll
        for (int k = 0; k < 9; ++k) st[lane * 9 + k] = R[k];
      }
      __syncwarp();
      float* gg = globalR + f * (int64_t)J * 9;
      for (int i = lane; i < J * 9; i += 32) gg[i] = st[i];
      __syncwarp();
    }
  }
}


// ------------------------------------------------------------------------------------------------
// Specialisation for the tree that is actually on the path: the 22-joint SMPL-X body
// (parents -1,0,0,0,1,2,3,4,5,6,7,8,9,9,9,12,13,14,16,17,18,19).  The shuffle kernel above spends ~450 warp
// instructions per frame (32 lanes march through every level), which caps it near 2 G frames/s; here one
// THREAD owns one frame and walks the tree as fully unrolled straight-line code (compile-time parents, so every
// transform lives in registers; ~70 warp-instructions per frame), which puts the kernel back on the HBM roofline.
// A CTA stages 64 frames through shared memory so that all global traffic is contiguous 128-bit accesses; a
// thread's pose row is overwritten in place by its joint positions.
constexpr int kB22 = 22;
constexpr int kB22Threads = 128;
__device__ constexpr int kB22Parent[kB22] = {-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19};
constexpr int kB22ParentHost[kB22] = {-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19};

struct Fk22Params { float rest[kB22 * 3]; };   // offset to parent (root: rest position)

template <bool kRotIn, bool kLocalOut>
__global__ void __launch_bounds__(kB22Threads)
fk_body22_kernel(const float* __restrict__ pose, const float* __restrict__ transl, float* __restrict__ joints,
                 float* __restrict__ localR, int64_t F, const __grid_constant__ Fk22Params p) {
  constexpr int IN = kRotIn ? 9 : 3;
  constexpr int IO_LD = kB22 * IN + 1;          // odd row pitch: conflict-free per-thread rows
  constexpr int ROT_LD = kB22 * 9 + 1;
  extern __shared__ __align__(16) float fk_smem[];
  float* s_io = fk_smem;                         // [64][IO_LD]: pose in, joints out (first 66 floats of the row)
  float* s_rot = fk_smem + kB22Threads * IO_LD;  // [64][ROT_LD]: local rotations out (aa input only)
  const int tid = threadIdx.x;
  const int64_t tiles = (F + kB22Threads - 1) / kB22Threads;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t f0 = tile * kB22Threads;
    const int nf = (int)min((int64_t)kB22Threads, F - f0);
    // ---- coalesced load: nf * 22 * IN floats, contiguous in global memory
    const float* gp = pose + f0 * (kB22 * IN);
    const int n_in = nf * kB22 * IN;
    // consecutive threads -> consecutive floats: 128 B per warp-load, consecutive shared-memory banks
#pragma unroll 8
    for (int i = tid; i < n_in; i += kB22Threads) s_io[i / (kB22 * IN) * IO_LD + i % (kB22 * IN)] = __ldg(gp + i);
    __syncthreads();
    if (tid < nf) {
      float* row = s_io + tid * IO_LD;
      float GR[kB22][9];
      float Gt[kB22][3];
#pragma unroll
      for (int j = 0; j < kB22; ++j) {
        float R[9];
        if (kRotIn) {
#pragma unroll
          for (int k = 0; k < 9; ++k) R[k] = row[j * 9 + k];
        } else {
          rodrigues_q(row[j * 3], row[j * 3 + 1], row[j * 3 + 2], R);
          if (kLocalOut) {
#pragma unroll
            for (int k = 0; k < 9; ++k) s_rot[tid * ROT_LD + j * 9 + k] = R[k];
          }
        }
        const float dx = p.rest[j * 3], dy = p.rest[j * 3 + 1], dz = p.rest[j * 3 + 2];
        const int par = kB22Parent[j];
        if (par < 0) {
#pragma unroll
          for (int k = 0; k < 9; ++k) GR[j][k] = R[k];
          Gt[j][0] = dx; Gt[j][1] = dy; Gt[j][2] = dz;
        } else {
          const float* A = GR[par];
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) GR[j][a * 3 + b] = A[a * 3] * R[b] + A[a * 3 + 1] * R[3 + b] + A[a * 3 + 2] * R[6 + b];
          Gt[j][0] = A[0] * dx + A[1] * dy + A[2] * dz + Gt[par][0];
          Gt[j][1] = A[3] * dx + A[4] * dy + A[5] * dz + Gt[par][1];
          Gt[j][2] = A[6] * dx + A[7] * dy + A[8] * dz + Gt[par][2];
        }
      }
      float tx = 0.f, ty = 0.f, tz = 0.f;
      if (transl != nullptr) {
        tx = __ldg(transl + (f0 + tid) * 3); ty = __ldg(transl + (f0 + tid) * 3 + 1); tz = __ldg(transl + (f0 + tid) * 3 + 2);
      }
      // the pose row is dead now: overwrite it with the joint positions
#pragma unroll
      for (int j = 0; j < kB22; ++j) {
        row[j * 3] = Gt[j][0] + tx; row[j * 3 + 1] = Gt[j][1] + ty; row[j * 3 + 2] = Gt[j][2] + tz;
      }
    }
    __syncthreads();
    // ---- coalesced stores
    float* gj = joints + f0 * (kB22 * 3);
    const int n_out = nf * kB22 * 3;
#pragma unroll 8
    for (int i = tid; i < n_out; i += kB22Threads) gj[i] = s_io[i / 66 * IO_LD + i % 66];
    if (kLocalOut) {
      float* gr = localR + f0 * (kB22 * 9);
#pragma unroll 8
      for (int i = tid; i < nf * 198; i += kB22Threads) gr[i] = s_rot[i / 198 * ROT_LD + i % 198];
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// Trees of up to 64 joints (the full 55-joint SMPL-X skeleton: body + jaw + eyes + 2 x 15 finger joints, plus rigid
// landmark pseudo-joints such as nose / ears hanging off the head with identity rotation; SURVEY.md 8f row 3,
// common/smpl_util.py:61-69, data_amass.py:176-218).  One warp per frame; the warp keeps every joint's global
// transform in shared memory and walks the tree LEVEL BY LEVEL (host-sorted order), one lane per joint of the level,
// so a level costs one pass however many joints it holds (11 levels for SMPL-X).  All global traffic is staged
// through the warp's shared-memory rows and is contiguous.
constexpr int kTreeMaxJ = 64;
constexpr int kTreeWarps = 4;
constexpr int kTreeMaxLevels = 24;

struct FkTreeParams {
  float rest[kTreeMaxJ * 3];        // offset to parent (root: rest position)
  int8_t parent[kTreeMaxJ];
  uint8_t order[kTreeMaxJ];         // joints sorted by tree level
  uint8_t level_start[kTreeMaxLevels + 1];
  int32_t n_levels, J;
};

template <bool kRotIn>
__global__ void __launch_bounds__(kTreeWarps * 32)
fk_tree_kernel(const float* __restrict__ pose, const float* __restrict__ transl, float* __restrict__ joints,
               float* __restrict__ localR, float* __restrict__ globalR, int64_t F, const __grid_constant__ FkTreeParams p) {
  constexpr int IN = kRotIn ? 9 : 3;
  __shared__ __align__(16) float s_R[kTreeWarps][kTreeMaxJ * 9];     // pose in, then local rotations
  __shared__ __align__(16) float s_G[kTreeWarps][kTreeMaxJ * 12];    // global [R | t] per joint
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int J = p.J;
  float* sr = s_R[warp];
  float* sg = s_G[warp];
  const int64_t warps_total = (int64_t)gridDim.x * kTreeWarps;
  for (int64_t f = (int64_t)blockIdx.x * kTreeWarps + warp; f < F; f += warps_total) {
    const float* gp = pose + f * (int64_t)J * IN;
    for (int i = lane; i < J * IN; i += 32) sr[i] = __ldg(gp + i);
    __syncwarp();
    if (!kRotIn) {
      // axis-angle -> rotation matrix, two joints per lane; inputs are read before any 9-float row is written
      float R0[9], R1[9];
      const int j0 = lane, j1 = lane + 32;
      if (j0 < J) rodrigues_q(sr[j0 * 3], sr[j0 * 3 + 1], sr[j0 * 3 + 2], R0);
      if (j1 < J) rodrigues_q(sr[j1 * 3], sr[j1 * 3 + 1], sr[j1 * 3 + 2], R1);
      __syncwarp();
      if (j0 < J) {
#pragma unroll
        for (int k = 0; k < 9; ++k) sr[j0 * 9 + k] = R0[k];
      }
      if (j1 < J) {
#pragma unroll
        for (int k = 0; k < 9; ++k) sr[j1 * 9 + k] = R1[k];
      }
      __syncwarp();
    }
    if (localR != nullptr) {
      float* go = localR + f * (int64_t)J * 9;
      for (int i = lane; i < J * 9; i += 32) go[i] = sr[i];
    }
    float tx = 0.f, ty = 0.f, tz = 0.f;
    if (transl != nullptr) { tx = __ldg(transl + f * 3); ty = __ldg(transl + f * 3 + 1); tz = __ldg(transl + f * 3 + 2); }
    for (int l = 0; l < p.n_levels; ++l) {
      for (int q = p.level_start[l] + lane; q < p.level_start[l + 1]; q += 32) {
        const int j = p.order[q];
        const int par = p.parent[j];
        const float* R = sr + j * 9;
        const float dx = p.rest[j * 3], dy = p.rest[j * 3 + 1], dz = p.rest[j * 3 + 2];
        float* G = sg + j * 12;
        if (par < 0) {
#pragma unroll
          for (int k = 0; k < 9; ++k) G[k] = R[k];
          G[9] = dx + tx; G[10] = dy + ty; G[11] = dz + tz;
        } else {
          const float* A = sg + par * 12;
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) G[a * 3 + b] = A[a * 3] * R[b] + A[a * 3 + 1] * R[3 + b] + A[a * 3 + 2] * R[6 + b];
          G[9] = A[0] * dx + A[1] * dy + A[2] * dz + A[9];
          G[10] = A[3] * dx + A[4] * dy + A[5] * dz + A[10];
          G[11] = A[6] * dx + A[7] * dy + A[8] * dz + A[11];
        }
      }
      __syncwarp();
    }
    float* gj = joints + f * (int64_t)J * 3;
    for (int i = lane; i < J * 3; i += 32) gj[i] = sg[(i / 3) * 12 + 9 + i % 3];
    if (globalR != nullptr) {
      float* gg = globalR + f * (int64_t)J * 9;
      for (int i = lane; i < J * 9; i += 32) gg[i] = sg[(i / 9) * 12 + i % 9];
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// Thread-per-frame specialisation for the full SMPL-X skeleton + face landmarks (60 joints, the tree of
// smpl_util.SyntheticBodyModel(skeleton='full')): same idea as fk_body22_kernel -- compile-time parents, fully unrolled,
// every live transform in registers (at most the current chain: a wrist stays live while its 15 finger joints are
// walked) -- ~5x fewer warp instructions per frame than the level-order kernel above.  Axis-angle in, joints out.
// The device-side parent table is f60_parent (fk_device.cuh).
constexpr int kF60Threads = 64;
constexpr int kF60ParentHost[kF60] = {-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 15, 15, 15,
                                      20, 25, 26, 20, 28, 29, 20, 31, 32, 20, 34, 35, 20, 37, 38,
                                      21, 40, 41, 21, 43, 44, 21, 46, 47, 21, 49, 50, 21, 52, 53, 15, 15, 15, 15, 15};
struct Fk60Params { float rest[kF60 * 3]; };

__global__ void __launch_bounds__(kF60Threads)
fk_full60_kernel(const float* __restrict__ pose, const float* __restrict__ transl, float* __restrict__ joints, int64_t F,
                 const __grid_constant__ Fk60Params p) {
  constexpr int LD = kF60 * 3 + 1;                 // odd row pitch: conflict-free per-thread rows
  extern __shared__ __align__(16) float fk_smem[];
  float* s_io = fk_smem;                           // [64][LD]: pose in, joints out
  const int tid = threadIdx.x;
  const int64_t tiles = (F + kF60Threads - 1) / kF60Threads;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t f0 = tile * kF60Threads;
    const int nf = (int)min((int64_t)kF60Threads, F - f0);
    const float* gp = pose + f0 * (kF60 * 3);
    const int n_io = nf * kF60 * 3;
#pragma unroll 8
    for (int i = tid; i < n_io; i += kF60Threads) s_io[i / (kF60 * 3) * LD + i % (kF60 * 3)] = __ldg(gp + i);
    __syncthreads();
    if (tid < nf) {
      float* row = s_io + tid * LD;
      float GR[kF60][9];
      float Gt[kF60][3];
#pragma unroll
      for (int j = 0; j < kF60; ++j) {
        float R[9];
        rodrigues_q(row[j * 3], row[j * 3 + 1], row[j * 3 + 2], R);
        const float dx = p.rest[j * 3], dy = p.rest[j * 3 + 1], dz = p.rest[j * 3 + 2];
        constexpr int kNone = -1;
        const int par = f60_parent(j);
        if (par == kNone) {
#pragma unroll
          for (int k = 0; k < 9; ++k) GR[j][k] = R[k];
          Gt[j][0] = dx; Gt[j][1] = dy; Gt[j][2] = dz;
        } else {
          const float* A = GR[par];
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) GR[j][a * 3 + b] = A[a * 3] * R[b] + A[a * 3 + 1] * R[3 + b] + A[a * 3 + 2] * R[6 + b];
          Gt[j][0] = A[0] * dx + A[1] * dy + A[2] * dz + Gt[par][0];
          Gt[j][1] = A[3] * dx + A[4] * dy + A[5] * dz + Gt[par][1];
          Gt[j][2] = A[6] * dx + A[7] * dy + A[8] * dz + Gt[par][2];
        }
      }
      float tx = 0.f, ty = 0.f, tz = 0.f;
      if (transl != nullptr) {
        tx = __ldg(transl + (f0 + tid) * 3); ty = __ldg(transl + (f0 + tid) * 3 + 1); tz = __ldg(transl + (f0 + tid) * 3 + 2);
      }
#pragma unroll
      for (int j = 0; j < kF60; ++j) { row[j * 3] = Gt[j][0] + tx; row[j * 3 + 1] = Gt[j][1] + ty; row[j * 3 + 2] = Gt[j][2] + tz; }
    }
    __syncthreads();
    float* gj = joints + f0 * (kF60 * 3);
#pragma unroll 8
    for (int i = tid; i < n_io; i += kF60Threads) gj[i] = s_io[i / (kF60 * 3) * LD + i % (kF60 * 3)];
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// Bulk-async pipelined thread-per-frame FK (axis-angle in, joints out) for the compile-time trees: the 22-joint
// SMPL-X body (the tree on the IK path) and the 60-joint full skeleton.
//
// The thread-per-frame kernels above are instruction-bound on their own staging: every float goes global -> register
// -> shared, shared -> register -> global with index arithmetic (~1200 of ~3600 thread-instructions per frame), and
// load / compute / store are serial phases per CTA.  Here a tile of kFrames frames is ONE contiguous block of global
// memory (kFrames * J * 12 bytes), so a producer thread moves it with a single cp.async.bulk (1-D TMA) into one of
// kStages shared-memory buffers, the compute threads overwrite their pose row in place with the joint positions
// (joint j's output occupies exactly the floats of joint j's input), and the producer sends the buffer back with a
// single bulk store.  Load of tile i+1, compute of tile i and store of tile i-1 overlap; the compute threads issue
// no global-memory instructions at all.  Rows are read / written as 8-byte (J = 22: row pitch 264 B) or 16-byte
// (J = 60: 720 B) vectors, both bank-conflict free at those pitches.  sin / cos / rsqrt use the SFU intrinsics
// (abs error ~5e-7 on |x| < pi, far inside the 1e-4 parity bar): precise sincosf costs ~40 instructions and a
// local-memory slow path per joint.
struct TreeBody22 {
  static constexpr int J = 22, VEC = 2;
  __host__ __device__ static constexpr int parent(int j) {
    constexpr int P[22] = {-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19};
    return P[j];
  }
};
struct TreeFull60 {
  static constexpr int J = 60, VEC = 4;
  __host__ __device__ static constexpr int parent(int j) { return f60_parent(j); }
};
template <int J> struct RestParams { float rest[J * 3]; };   // offset to parent (root: rest position)

template <int VEC> struct VecT;
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

template <class Tree, int kFrames, int kStages>
__global__ void __launch_bounds__(kFrames + 32)
fk_bulk_kernel(const float* __restrict__ pose, const float* __restrict__ transl, float* __restrict__ joints, int64_t n_tiles,
               const __grid_constant__ RestParams<Tree::J> p) {
  constexpr int J = Tree::J, ROW = J * 3, VEC = Tree::VEC, G = VEC;       // G joints = 3 vectors of VEC floats
  static_assert(J % G == 0 && (ROW * 4) % (VEC * 4) == 0, "row must split into whole vector groups");
  constexpr uint32_t kTileBytes = (uint32_t)kFrames * ROW * 4;
  static_assert(kTileBytes % 16 == 0, "bulk copies move multiples of 16 bytes");
  using V = typename VecT<VEC>::type;
  extern __shared__ __align__(128) uint8_t fk_bulk_smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(fk_bulk_smem + (size_t)kStages * kTileBytes);
  uint64_t* done = full + kStages;
  const int tid = threadIdx.x;
  if (tid == 0) {
#pragma unroll
    for (int b = 0; b < kStages; ++b) { mbar_init(&full[b], 1); mbar_init(&done[b], kFrames); }
    fence_barrier_init();
  }
  __syncthreads();
  const int64_t first = blockIdx.x, stride = gridDim.x;
  const int64_t n_my = first < n_tiles ? (n_tiles - first + stride - 1) / stride : 0;

  if (tid >= kFrames) {
    // ---- producer: one thread issues every bulk load and bulk store of this CTA
    if (tid == kFrames) {
      for (int64_t i = 0; i < n_my; ++i) {
        const int b = (int)(i % kStages);
        uint8_t* buf = fk_bulk_smem + (size_t)b * kTileBytes;
        if (i >= kStages) {                                  // the buffer's previous tile has been computed: send it out
          mbar_wait(&done[b], (uint32_t)((i / kStages) - 1) & 1u);
          bulk_store_1d(joints + (first + (i - kStages) * stride) * (int64_t)(kFrames * ROW), buf, kTileBytes);
          tma_store_commit();
          tma_store_wait_read0();                            // shared memory has been read: the buffer may be refilled
        }
        mbar_expect_tx(&full[b], kTileBytes);
        bulk_load_1d(buf, pose + (first + i * stride) * (int64_t)(kFrames * ROW), kTileBytes, &full[b]);
      }
      for (int64_t i = n_my > kStages ? n_my - kStages : 0; i < n_my; ++i) {
        const int b = (int)(i % kStages);
        mbar_wait(&done[b], (uint32_t)(i / kStages) & 1u);
        bulk_store_1d(joints + (first + i * stride) * (int64_t)(kFrames * ROW), fk_bulk_smem + (size_t)b * kTileBytes, kTileBytes);
        tma_store_commit();
      }
      tma_store_wait0();
    }
    return;
  }

  // ---- compute: thread tid owns frame tid of every tile
  for (int64_t i = 0; i < n_my; ++i) {
    const int b = (int)(i % kStages);
    mbar_wait(&full[b], (uint32_t)(i / kStages) & 1u);
    V* row = reinterpret_cast<V*>(fk_bulk_smem + (size_t)b * kTileBytes + (size_t)tid * ROW * 4);
    float tx = 0.f, ty = 0.f, tz = 0.f;
    if (transl != nullptr) {
      const int64_t f = (first + i * stride) * kFrames + tid;
      tx = __ldg(transl + f * 3); ty = __ldg(transl + f * 3 + 1); tz = __ldg(transl + f * 3 + 2);
    }
    float GR[J][9];
    float Gt[J][3];
#pragma unroll
    for (int g = 0; g < J / G; ++g) {
      float a[3 * G];
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const V v = row[g * 3 + q];
        const float* vf = reinterpret_cast<const float*>(&v);
#pragma unroll
        for (int e = 0; e < VEC; ++e) a[q * VEC + e] = vf[e];
      }
#pragma unroll
      for (int q = 0; q < G; ++q) {
        const int j = g * G + q;
        float R[9];
        rodrigues_q_fast(a[q * 3], a[q * 3 + 1], a[q * 3 + 2], R);
        const float dx = p.rest[j * 3], dy = p.rest[j * 3 + 1], dz = p.rest[j * 3 + 2];
        const int par = Tree::parent(j);
        if (par < 0) {
#pragma unroll
          for (int k = 0; k < 9; ++k) GR[j][k] = R[k];
          Gt[j][0] = dx; Gt[j][1] = dy; Gt[j][2] = dz;
        } else {
          const float* A = GR[par];
#pragma unroll
          for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c) GR[j][r * 3 + c] = A[r * 3] * R[c] + A[r * 3 + 1] * R[3 + c] + A[r * 3 + 2] * R[6 + c];
          Gt[j][0] = A[0] * dx + A[1] * dy + A[2] * dz + Gt[par][0];
          Gt[j][1] = A[3] * dx + A[4] * dy + A[5] * dz + Gt[par][1];
          Gt[j][2] = A[6] * dx + A[7] * dy + A[8] * dz + Gt[par][2];
        }
        a[q * 3] = Gt[j][0] + tx; a[q * 3 + 1] = Gt[j][1] + ty; a[q * 3 + 2] = Gt[j][2] + tz;
      }
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        V v;
        float* vf = reinterpret_cast<float*>(&v);
#pragma unroll
        for (int e = 0; e < VEC; ++e) vf[e] = a[q * VEC + e];
        row[g * 3 + q] = v;
      }
    }
    fence_proxy_async_smem();          // this thread's st.shared -> visible to the bulk store (async proxy)
    mbar_arrive(&done[b]);
  }
}

// Launches the bulk kernel on the whole tiles of the batch; returns the number of frames it covered.
template <class Tree, int kFrames, int kStages>
static int launch_fk_bulk(const float* pose, const float* transl, float* joints, int64_t F, const float* rest_off,
                          cudaStream_t s, int64_t* covered) {
  constexpr size_t smem = (size_t)kStages * kFrames * Tree::J * 12 + 2 * kStages * sizeof(uint64_t);
  auto kern = fk_bulk_kernel<Tree, kFrames, kStages>;
  static bool attr_set[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (!attr_set[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    TIK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr_set[dev & 63] = true;
  }
  const int64_t n_tiles = F / kFrames;
  *covered = n_tiles * kFrames;
  if (n_tiles == 0) return TIK_OK;
  RestParams<Tree::J> p;
  for (int i = 0; i < Tree::J * 3; ++i) p.rest[i] = rest_off[i];
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(16, (227 * 1024) / (smem + 1024)));
  int64_t blocks = std::min<int64_t>(n_tiles, (int64_t)148 * per_sm);
  kern<<<(unsigned)blocks, kFrames + 32, smem, s>>>(pose, transl, joints, n_tiles, p);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}

static int fk_bulk_cfg() {
  static int v = -2;
  if (v == -2) { const char* e = getenv("TIK_FK_BULK"); v = e ? atoi(e) : 0; }
  return v;      // -1: off (staged kernels above); 0: default; 1..3: alternative tile / stage shapes (tools/hbm_bench.py)
}

template <bool kRotIn, bool kLocalOut>
static int launch_body22(const float* pose, const float* transl, float* joints, float* localR, int64_t F,
                         const Fk22Params& p, cudaStream_t s) {
  constexpr int IN = kRotIn ? 9 : 3;
  const size_t smem = sizeof(float) * ((size_t)kB22Threads * (kB22 * IN + 1) + (kLocalOut ? (size_t)kB22Threads * (kB22 * 9 + 1) : 0));
  static bool attr_set[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (!attr_set[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(fk_body22_kernel<kRotIn, kLocalOut>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    TIK_CUDA(cudaFuncSetAttribute(fk_body22_kernel<kRotIn, kLocalOut>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr_set[dev & 63] = true;
  }
  int64_t blocks = ceil_div(F, kB22Threads);
  const int64_t cap = 148 * 12;
  if (blocks > cap) blocks = cap;
  fk_body22_kernel<kRotIn, kLocalOut><<<(unsigned)blocks, kB22Threads, smem, s>>>(pose, transl, joints, localR, F, p);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}
}  // namespace tik

extern "C" int tik_fk_body(const float* pose_dev, int pose_is_rotmat, const float* rest_host,
                           const int32_t* parents_host, int J, const float* transl_dev, float* joints_dev,
                           float* local_R_dev, float* global_R_dev, int64_t F, void* stream) {
  using namespace tik;
  TIK_CHECK_ARG(J >= 1 && J <= TIK_MAX_JOINTS, "J=%d outside [1,%d]", J, TIK_MAX_JOINTS);
  TIK_CHECK_ARG(F >= 0, "negative frame count");
  if (F == 0) return TIK_OK;
  TIK_CHECK_ARG(pose_dev && rest_host && parents_host && joints_dev, "null pointer");
  FkParams p;
  int depth[TIK_MAX_JOINTS], maxd = 0;
  for (int i = 0; i < J; ++i) {
    int par = parents_host[i];
    TIK_CHECK_ARG(par < i && par >= -1, "parents[%d]=%d must be -1 or an earlier joint", i, par);
    p.parent[i] = (int8_t)par;
    depth[i] = par < 0 ? 0 : depth[par] + 1;
    if (depth[i] > maxd) maxd = depth[i];
    for (int k = 0; k < 3; ++k)
      p.rest[i * 3 + k] = par < 0 ? rest_host[i * 3 + k] : rest_host[i * 3 + k] - rest_host[par * 3 + k];
  }
  for (int i = J; i < TIK_MAX_JOINTS; ++i) { p.parent[i] = -1; p.rest[i * 3] = p.rest[i * 3 + 1] = p.rest[i * 3 + 2] = 0.f; }
  cudaStream_t s = (cudaStream_t)stream;
  // fast path: the SMPL-X body tree (the one on the IK path), no global rotations requested
  bool body22 = J == kB22 && global_R_dev == nullptr && (!pose_is_rotmat || local_R_dev == nullptr);
  for (int i = 0; body22 && i < J; ++i) body22 = parents_host[i] == kB22ParentHost[i];
  if (body22 && (((uintptr_t)pose_dev | (uintptr_t)joints_dev | (uintptr_t)local_R_dev) & 15) == 0) {
    Fk22Params q;
    for (int i = 0; i < kB22 * 3; ++i) q.rest[i] = p.rest[i];
    if (pose_is_rotmat) return launch_body22<true, false>(pose_dev, transl_dev, joints_dev, nullptr, F, q, s);
    if (local_R_dev) {
      // local rotations are an element-wise conversion: the streaming Rodrigues kernel (81 % of the HBM peak) writes
      // them; the joints come from the joints-only kernel below (a fused variant needs 792 more bytes of shared
      // memory per frame and measured 2.3x slower, profiles/r1_notes.md)
      int rc = launch_batch_rodrigues(pose_dev, local_R_dev, F * kB22, s);
      if (rc != TIK_OK) return rc;
    }
    // joints from axis-angle: bulk-async pipelined kernel on the whole tiles, staged kernel on the remainder
    int64_t done_frames = 0;
    const int cfg = fk_bulk_cfg();
    if (cfg >= 0) {
      int rc = cfg == 1   ? launch_fk_bulk<TreeBody22, 64, 3>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames)
               : cfg == 2 ? launch_fk_bulk<TreeBody22, 128, 2>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames)
               : cfg == 3 ? launch_fk_bulk<TreeBody22, 64, 2>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames)
                          : launch_fk_bulk<TreeBody22, 128, 3>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames);
      if (rc != TIK_OK) return rc;
      if (done_frames == F) return TIK_OK;
    }
    return launch_body22<false, false>(pose_dev + done_frames * (kB22 * 3), transl_dev ? transl_dev + done_frames * 3 : nullptr,
                                       joints_dev + done_frames * (kB22 * 3), nullptr, F - done_frames, q, s);
  }
  if (J == kF60 && !pose_is_rotmat && local_R_dev == nullptr && global_R_dev == nullptr) {
    bool full60 = true;
    for (int i = 0; full60 && i < J; ++i) full60 = parents_host[i] == kF60ParentHost[i];
    if (full60) {
      int64_t done_frames = 0;
      const int cfg = fk_bulk_cfg();
      if (cfg >= 0 && (((uintptr_t)pose_dev | (uintptr_t)joints_dev) & 15) == 0) {
        int rc = cfg == 1   ? launch_fk_bulk<TreeFull60, 32, 3>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames)
                 : cfg == 2 ? launch_fk_bulk<TreeFull60, 64, 3>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames)
                 : cfg == 3 ? launch_fk_bulk<TreeFull60, 32, 2>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames)
                 : cfg == 4 ? launch_fk_bulk<TreeFull60, 64, 2>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames)
                 : cfg == 5 ? launch_fk_bulk<TreeFull60, 128, 1>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames)
                 : cfg == 6 ? launch_fk_bulk<TreeFull60, 32, 1>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames)
                            // default: ONE buffer per CTA, four CTAs per SM.  720 B per frame in place means ~315 frames per SM whatever
                            // the shape; single-buffered CTAs put all of them under compute threads (8 warps instead of 4) and
                            // overlap each other's load / compute / store phases: 0.68 of the HBM peak against 0.48-0.55 with
                            // two buffers per CTA (cfg 4), 0.67 with 128 frames x 1 (cfg 5), 0.48 with 32 x 1 (cfg 6).
                            : launch_fk_bulk<TreeFull60, 64, 1>(pose_dev, transl_dev, joints_dev, F, p.rest, s, &done_frames);
        if (rc != TIK_OK) return rc;
        if (done_frames == F) return TIK_OK;
        pose_dev += done_frames * (kF60 * 3);
        joints_dev += done_frames * (kF60 * 3);
        if (transl_dev) transl_dev += done_frames * 3;
        F -= done_frames;
      }
      Fk60Params q;
      for (int i = 0; i < kF60 * 3; ++i) q.rest[i] = p.rest[i];
      const size_t smem = sizeof(float) * (size_t)kF60Threads * (kF60 * 3 + 1);
      static bool attr_set[64] = {};
      int dev = 0;
      TIK_CUDA(cudaGetDevice(&dev));
      if (!attr_set[dev & 63]) {
        TIK_CUDA(cudaFuncSetAttribute(fk_full60_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        attr_set[dev & 63] = true;
      }
      int64_t blocks = ceil_div(F, kF60Threads);
      if (blocks > 148 * 16) blocks = 148 * 16;
      fk_full60_kernel<<<(unsigned)blocks, kF60Threads, smem, s>>>(pose_dev, transl_dev, joints_dev, F, q);
      TIK_LAUNCH_CHECK();
      return TIK_OK;
    }
  }
  if (J > 32) {
    FkTreeParams q;
    memset(&q, 0, sizeof(q));
    q.J = J;
    int nl = 0;
    for (int i = 0; i < J; ++i) { q.parent[i] = p.parent[i]; for (int k = 0; k < 3; ++k) q.rest[i * 3 + k] = p.rest[i * 3 + k]; }
    TIK_CHECK_ARG(maxd + 1 <= kTreeMaxLevels, "kinematic tree deeper than %d levels", kTreeMaxLevels);
    int pos = 0;
    for (int l = 0; l <= maxd; ++l) {
      q.level_start[l] = (uint8_t)pos;
      for (int i = 0; i < J; ++i) if (depth[i] == l) q.order[pos++] = (uint8_t)i;
      nl = l + 1;
    }
    q.level_start[nl] = (uint8_t)pos;
    q.n_levels = nl;
    int64_t blocks = ceil_div(F, kTreeWarps);
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (pose_is_rotmat)
      fk_tree_kernel<true><<<(unsigned)blocks, kTreeWarps * 32, 0, s>>>(pose_dev, transl_dev, joints_dev, local_R_dev, global_R_dev, F, q);
    else
      fk_tree_kernel<false><<<(unsigned)blocks, kTreeWarps * 32, 0, s>>>(pose_dev, transl_dev, joints_dev, local_R_dev, global_R_dev, F, q);
    TIK_LAUNCH_CHECK();
    return TIK_OK;
  }
  p.J = J;
  p.rounds = 0;
  while ((1 << p.rounds) < maxd + 1) ++p.rounds;
  int sms = 148;
  int64_t blocks = ceil_div(F, kFkWarps);
  int64_t cap = (int64_t)sms * 8 * 4;   // persistent-ish: grid-stride over frames
  if (blocks > cap) blocks = cap;
  if (pose_is_rotmat)
    fk_kernel<true><<<(unsigned)blocks, kFkWarps * 32, 0, s>>>(pose_dev, transl_dev, joints_dev, local_R_dev, global_R_dev, F, p);
  else
    fk_kernel<false><<<(unsigned)blocks, kFkWarps * 32, 0, s>>>(pose_dev, transl_dev, joints_dev, local_R_dev, global_R_dev, F, p);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}
