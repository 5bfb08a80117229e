// Rotation-representation conversions, fp32, HBM-bandwidth bound.
//
// One thread per rotation; each CTA stages its 256 rotations through shared memory so that
// global traffic is fully coalesced 128-bit loads/stores even though a rotation is 3, 6 or 9
// floats.  Precise libm (no fast-math): parity target is 1e-4 max-abs against the reference
// formulas, cited per function.
#include <algorithm>

#include "tik_common.cuh"
#include "umma_ptx.cuh"

namespace tik {

constexpr int kConvThreads = 256;

template <int IN, int OUT, class F>
__device__ __forceinline__ void staged_map(const float* __restrict__ in, float* __restrict__ out, int64_t M, F f) {
  __shared__ __align__(16) float s_in[kConvThreads * IN];
  __shared__ __align__(16) float s_out[kConvThreads * OUT];
  const int64_t base = (int64_t)blockIdx.x * kConvThreads;
  const int n = (int)min((int64_t)kConvThreads, M - base);
  const float* gin = in + base * IN;
  float* gout = out + base * OUT;
  if (n == kConvThreads) {
    const float4* g4 = reinterpret_cast<const float4*>(gin);
    float4* s4 = reinterpret_cast<float4*>(s_in);
#pragma unroll
    for (int i = threadIdx.x; i < kConvThreads * IN / 4; i += kConvThreads) s4[i] = __ldg(g4 + i);
  } else {
    for (int i = threadIdx.x; i < n * IN; i += kConvThreads) s_in[i] = gin[i];
  }
  __syncthreads();
  if ((int)threadIdx.x < n) {
    float a[IN], r[OUT];
#pragma unroll
    for (int k = 0; k < IN; ++k) a[k] = s_in[threadIdx.x * IN + k];
    f(a, r);
#pragma unroll
    for (int k = 0; k < OUT; ++k) s_out[threadIdx.x * OUT + k] = r[k];
  }
  __syncthreads();
  if (n == kConvThreads) {
    float4* g4 = reinterpret_cast<float4*>(gout);
    const float4* s4 = reinterpret_cast<const float4*>(s_out);
#pragma unroll
    for (int i = threadIdx.x; i < kConvThreads * OUT / 4; i += kConvThreads) g4[i] = s4[i];
  } else {
    for (int i = threadIdx.x; i < n * OUT; i += kConvThreads) gout[i] = s_out[i];
  }
}

// Bulk-async pipelined variant of staged_map for the whole 256-rotation tiles of a batch (the staged kernel above
// keeps the remainder).  A tile's input and output are contiguous blocks of global memory, so ONE producer thread
// moves them with cp.async.bulk (1-D TMA) through a ring of kStages shared-memory buffer pairs and the 256 compute
// threads issue no global-memory instructions: the staged version spent about a quarter of its instructions on
// staging and ran load / compute / store as serial phases per CTA (ncu: issue-bound at 55-73 % issue utilisation
// with DRAM at 50-65 %, profiles/r2_hbm_kernels.md).
constexpr int kConvStages = 4;

__device__ __forceinline__ void conv_bulk_load(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void conv_bulk_store(void* dst, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(dst), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}

template <int IN, int OUT, class F>
__device__ __forceinline__ void bulk_map(const float* __restrict__ in, float* __restrict__ out, int64_t n_tiles, F f) {
  constexpr uint32_t kInBytes = kConvThreads * IN * 4, kOutBytes = kConvThreads * OUT * 4;
  extern __shared__ __align__(128) uint8_t conv_smem[];
  uint8_t* in_bufs = conv_smem;
  uint8_t* out_bufs = conv_smem + (size_t)kConvStages * kInBytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(out_bufs + (size_t)kConvStages * kOutBytes);
  uint64_t* done = full + kConvStages;
  const int tid = threadIdx.x;
  if (tid == 0) {
#pragma unroll
    for (int b = 0; b < kConvStages; ++b) { mbar_init(&full[b], 1); mbar_init(&done[b], kConvThreads); }
    fence_barrier_init();
  }
  __syncthreads();
  const int64_t first = blockIdx.x, stride = gridDim.x;
  const int64_t n_my = first < n_tiles ? (n_tiles - first + stride - 1) / stride : 0;
  if (tid >= kConvThreads) {
    if (tid == kConvThreads) {
      auto load = [&](int64_t t) {
        const int b = (int)(t % kConvStages);
        mbar_expect_tx(&full[b], kInBytes);
        conv_bulk_load(in_bufs + (size_t)b * kInBytes, in + (first + t * stride) * (int64_t)(kConvThreads * IN), kInBytes, &full[b]);
      };
      for (int64_t t = 0; t < n_my && t < kConvStages; ++t) load(t);
      for (int64_t j = 0; j < n_my; ++j) {
        const int b = (int)(j % kConvStages);
        mbar_wait(&done[b], (uint32_t)(j / kConvStages) & 1u);                 // tile j computed: its output buffer is complete
        conv_bulk_store(out + (first + j * stride) * (int64_t)(kConvThreads * OUT), out_bufs + (size_t)b * kOutBytes, kOutBytes);
        tma_store_commit();
        if (j >= 1) {
          // the PREVIOUS tile's store has read its shared-memory buffer (one tile of slack for the producer): that
          // buffer pair may take the tile kStages ahead of it
          tma_store_wait_read1();
          if (j - 1 + kConvStages < n_my) load(j - 1 + kConvStages);
        }
      }
      tma_store_wait0();
    }
    return;
  }
  for (int64_t i = 0; i < n_my; ++i) {
    const int b = (int)(i % kConvStages);
    mbar_wait(&full[b], (uint32_t)(i / kConvStages) & 1u);
    const float* si = reinterpret_cast<const float*>(in_bufs + (size_t)b * kInBytes) + tid * IN;
    float* so = reinterpret_cast<float*>(out_bufs + (size_t)b * kOutBytes) + tid * OUT;
    float a[IN], r[OUT];
    if constexpr (IN % 2 == 0) {       // even row pitch: 8-byte loads are bank-conflict free where 4-byte ones are 2-way
#pragma unroll
      for (int k = 0; k < IN / 2; ++k) {
        const float2 v = reinterpret_cast<const float2*>(si)[k];
        a[2 * k] = v.x; a[2 * k + 1] = v.y;
      }
    } else {
#pragma unroll
      for (int k = 0; k < IN; ++k) a[k] = si[k];
    }
    f(a, r);
#pragma unroll
    for (int k = 0; k < OUT; ++k) so[k] = r[k];
    fence_proxy_async_smem();          // st.shared -> visible to the bulk store (async proxy)
    mbar_arrive(&done[b]);
  }
}

// common/geometry.py:330-344 -- a1 = (x0,x2,x4), a2 = (x1,x3,x5); R columns = b1,b2,b3.
__device__ __forceinline__ void rot6d_one(const float* x, float* R) {
  float a1x = x[0], a1y = x[2], a1z = x[4], a2x = x[1], a2y = x[3], a2z = x[5];
  // one reciprocal per normalisation instead of three divisions (the kernels were issue-bound, profiles/r2_hbm_kernels.md)
  float i1 = 1.0f / fmaxf(sqrtf(a1x * a1x + a1y * a1y + a1z * a1z), 1e-6f);
  float b1x = a1x * i1, b1y = a1y * i1, b1z = a1z * i1;
  float d = b1x * a2x + b1y * a2y + b1z * a2z;
  float ux = a2x - d * b1x, uy = a2y - d * b1y, uz = a2z - d * b1z;
  float i2 = 1.0f / fmaxf(sqrtf(ux * ux + uy * uy + uz * uz), 1e-6f);
  float b2x = ux * i2, b2y = uy * i2, b2z = uz * i2;
  float b3x = b1y * b2z - b1z * b2y, b3y = b1z * b2x - b1x * b2z, b3z = b1x * b2y - b1y * b2x;
  R[0] = b1x; R[1] = b2x; R[2] = b3x;
  R[3] = b1y; R[4] = b2y; R[5] = b3y;
  R[6] = b1z; R[7] = b2z; R[8] = b3z;
}

// common/kornia_geometry_conversion.py:125-201
__device__ __forceinline__ void aa_kornia_one(const float* a, float* R) {
  float rx = a[0], ry = a[1], rz = a[2];
  float t2 = rx * rx + ry * ry + rz * rz;
  if (t2 > 1e-6f) {
    float th = sqrtf(t2);
    float inv = 1.0f / (th + 1e-6f);
    float wx = rx * inv, wy = ry * inv, wz = rz * inv;
    float s, c;
    sincosf(th, &s, &c);
    float k = 1.0f - c;
    R[0] = c + wx * wx * k;       R[1] = wx * wy * k - wz * s;  R[2] = wy * s + wx * wz * k;
    R[3] = wz * s + wx * wy * k;  R[4] = c + wy * wy * k;       R[5] = -wx * s + wy * wz * k;
    R[6] = -wy * s + wx * wz * k; R[7] = wx * s + wy * wz * k;  R[8] = c + wz * wz * k;
  } else {
    R[0] = 1.f; R[1] = -rz; R[2] = ry;
    R[3] = rz;  R[4] = 1.f; R[5] = -rx;
    R[6] = -ry; R[7] = rx;  R[8] = 1.f;
  }
}

// common/geometry.py:22-65 (batch_rodrigues + quat2mat)
__device__ __forceinline__ void rodrigues_one(const float* a, float* R) {
  float ex = a[0] + 1e-8f, ey = a[1] + 1e-8f, ez = a[2] + 1e-8f;
  float ang = sqrtf(ex * ex + ey * ey + ez * ez);
  float ia = 1.0f / ang;
  float nx = a[0] * ia, ny = a[1] * ia, nz = a[2] * ia;
  float s, c;
  sincosf(ang * 0.5f, &s, &c);
  float w = c, x = s * nx, y = s * ny, z = s * nz;
  float iq = rsqrtf(w * w + x * x + y * y + z * z);
  w *= iq; x *= iq; y *= iq; z *= iq;
  float w2 = w * w, x2 = x * x, y2 = y * y, z2 = z * z;
  float wx = w * x, wy = w * y, wz = w * z, xy = x * y, xz = x * z, yz = y * z;
  R[0] = w2 + x2 - y2 - z2; R[1] = 2.f * xy - 2.f * wz;   R[2] = 2.f * wy + 2.f * xz;
  R[3] = 2.f * wz + 2.f * xy; R[4] = w2 - x2 + y2 - z2;   R[5] = 2.f * yz - 2.f * wx;
  R[6] = 2.f * xz - 2.f * wy; R[7] = 2.f * wx + 2.f * yz; R[8] = w2 - x2 - y2 + z2;
}

// atan2(y, x) for x >= 0 (or NaN): |error| <= 1.1e-7 rad (degree-8 minimax-style fit of atan(z)/z in z^2 on [0,1],
// checked against float64 on 200,001 points in fp32 arithmetic; tools/fit_atan.py).  libm's atan2f costs ~60
// instructions with divergent paths; this is ~20, branch-free.
__device__ __forceinline__ float atan2_xpos(float y, float x) {
  const float ay = fabsf(y);
  const float mx = fmaxf(ay, x), mn = fminf(ay, x);
  const float z = mx > 0.0f ? __fdividef(mn, mx) : (mx == 0.0f ? 0.0f : mx);     // NaN propagates
  const float u = z * z;
  float p = 0.0028340641874819994f;
  p = fmaf(p, u, -0.016005029901862144f);
  p = fmaf(p, u, 0.042587608098983765f);
  p = fmaf(p, u, -0.07495445758104324f);
  p = fmaf(p, u, 0.10636754333972931f);
  p = fmaf(p, u, -0.14202570915222168f);
  p = fmaf(p, u, 0.19992484152317047f);
  p = fmaf(p, u, -0.3333306610584259f);
  p = fmaf(p, u, 1.0f);
  float r = z * p;
  r = ay > x ? 1.5707963267948966f - r : r;
  r = (x != x || y != y) ? x + y : r;                   // fmaxf / fminf drop NaNs: put them back as atan2f would
  return copysignf(r, y);
}

// common/geometry.py:100-150 (w,x,y,z).  The reference picks atan2(-s, -q0) when q0 < 0 and atan2(s, q0) otherwise:
// one atan2 of sign-flipped arguments, whose second argument is never negative.
__device__ __forceinline__ void quat_to_aa(float q0, float q1, float q2, float q3, float* aa) {
  const float s2 = q1 * q1 + q2 * q2 + q3 * q3;
  const float rs = rsqrtf(s2);
  const float s = s2 * rs;                              // sqrt(s2) for s2 > 0 (s2 == 0 takes the k = 2 branch below)
  const bool neg = q0 < 0.0f;
  const float two_theta = 2.0f * atan2_xpos(neg ? -s : s, neg ? -q0 : q0);
  const float k = s2 > 0.0f ? two_theta * rs : 2.0f;
  aa[0] = q1 * k; aa[1] = q2 * k; aa[2] = q3 * k;
}

// common/geometry.py:37-65 quat2mat: (w,x,y,z), normalised first
__device__ __forceinline__ void quat2mat_one(const float* q, float* R) {
  float w = q[0], x = q[1], y = q[2], z = q[3];
  const float iq = rsqrtf(w * w + x * x + y * y + z * z);
  w *= iq; x *= iq; y *= iq; z *= iq;
  const float w2 = w * w, x2 = x * x, y2 = y * y, z2 = z * z;
  const float wx = w * x, wy = w * y, wz = w * z, xy = x * y, xz = x * z, yz = y * z;
  R[0] = w2 + x2 - y2 - z2; R[1] = 2.f * xy - 2.f * wz;   R[2] = 2.f * wy + 2.f * xz;
  R[3] = 2.f * wz + 2.f * xy; R[4] = w2 - x2 + y2 - z2;   R[5] = 2.f * yz - 2.f * wx;
  R[6] = 2.f * xz - 2.f * wy; R[7] = 2.f * wx + 2.f * yz; R[8] = w2 - x2 - y2 + z2;
}

// common/geometry.py:68-97,153-233: four-case selection on the transposed matrix, NaN -> 0.
// The ncu capture of round 2 (profiles/r2_hbm_kernels.md) showed the first version issue-bound (306 instructions per
// rotation: four divergent cases, two atan2f, five precise divisions): the cases are now selects over shared sums, the
// common factor 0.5 / sqrt(t) is one rsqrt (same inf / NaN behaviour as q / sqrt(t) * 0.5 for t <= 0).
__device__ __forceinline__ void rotmat_to_quat_one(const float* R, float* q);
__device__ __forceinline__ void rotmat_to_aa_one(const float* R, float* aa) {
  float q[4];
  rotmat_to_quat_one(R, q);
  quat_to_aa(q[0], q[1], q[2], q[3], aa);
#pragma unroll
  for (int k = 0; k < 3; ++k)
    if (isnan(aa[k])) aa[k] = 0.f;
}
// common/geometry.py:153-233 rotation_matrix_to_quaternion -> (w,x,y,z)
__device__ __forceinline__ void rotmat_to_quat_one(const float* R, float* q) {
  // m = R^T
  const float m00 = R[0], m01 = R[3], m02 = R[6];
  const float m10 = R[1], m11 = R[4], m12 = R[7];
  const float m20 = R[2], m21 = R[5], m22 = R[8];
  const bool d2 = m22 < 1e-6f, d01 = m00 > m11, d0n1 = m00 < -m11;
  const bool c0 = d2 && d01, c1 = d2 && !d01, c2 = !d2 && d0n1;           // else: c3
  const float s01 = m01 + m10, s20 = m20 + m02, s12 = m12 + m21;
  const float a12 = m12 - m21, a20 = m20 - m02, a01 = m01 - m10;
  const float t = c0 ? 1.f + m00 - m11 - m22 : c1 ? 1.f - m00 + m11 - m22 : c2 ? 1.f - m00 - m11 + m22 : 1.f + m00 + m11 + m22;
  float q0 = c0 ? a12 : c1 ? a20 : c2 ? a01 : t;
  float q1 = c0 ? t : c1 ? s01 : c2 ? s20 : a12;
  float q2 = c0 ? s01 : c1 ? t : c2 ? s12 : a20;
  float q3 = c0 ? s20 : c1 ? s12 : c2 ? t : a01;
  const float h = 0.5f * rsqrtf(t);
  q[0] = q0 * h; q[1] = q1 * h; q[2] = q2 * h; q[3] = q3 * h;
}

// common/kornia_geometry_conversion.py:204-307,396-439: (x,y,z,w) quaternion read as (w,x,y,z).
__device__ __forceinline__ void rotmat_to_aa_kornia_quirk_one(const float* R, float* aa) {
  const float tiny = 1.17549435e-38f;
  float m00 = R[0], m01 = R[1], m02 = R[2], m10 = R[3], m11 = R[4], m12 = R[5], m20 = R[6], m21 = R[7], m22 = R[8];
  float tr = m00 + m11 + m22;
  float qx, qy, qz, qw;
  if (tr > 0.f) {
    float sq = sqrtf(tr + 1.0f) * 2.f, dn = fmaxf(sq, tiny);
    qw = 0.25f * sq; qx = (m21 - m12) / dn; qy = (m02 - m20) / dn; qz = (m10 - m01) / dn;
  } else if (m00 > m11 && m00 > m22) {
    float sq = sqrtf(1.0f + m00 - m11 - m22 + 1e-8f) * 2.f, dn = fmaxf(sq, tiny);
    qw = (m21 - m12) / dn; qx = 0.25f * sq; qy = (m01 + m10) / dn; qz = (m02 + m20) / dn;
  } else if (m11 > m22) {
    float sq = sqrtf(1.0f + m11 - m00 - m22 + 1e-8f) * 2.f, dn = fmaxf(sq, tiny);
    qw = (m02 - m20) / dn; qx = (m01 + m10) / dn; qy = 0.25f * sq; qz = (m12 + m21) / dn;
  } else {
    float sq = sqrtf(1.0f + m22 - m00 - m11 + 1e-8f) * 2.f, dn = fmaxf(sq, tiny);
    qw = (m10 - m01) / dn; qx = (m02 + m20) / dn; qy = (m12 + m21) / dn; qz = 0.25f * sq;
  }
  quat_to_aa(qx, qy, qz, qw, aa);   // the quirk: element 0 (= x) is treated as cos(theta/2)
}

__global__ void __launch_bounds__(kConvThreads) rot6d_kernel(const float* in, float* out, int64_t M) {
  staged_map<6, 9>(in, out, M, [](const float* a, float* r) { rot6d_one(a, r); });
}
__global__ void __launch_bounds__(kConvThreads) aa_kornia_kernel(const float* in, float* out, int64_t M) {
  staged_map<3, 9>(in, out, M, [](const float* a, float* r) { aa_kornia_one(a, r); });
}
__global__ void __launch_bounds__(kConvThreads) rodrigues_kernel(const float* in, float* out, int64_t M) {
  staged_map<3, 9>(in, out, M, [](const float* a, float* r) { rodrigues_one(a, r); });
}
__global__ void __launch_bounds__(kConvThreads) rotmat_to_aa_kernel(const float* in, float* out, int64_t M, int quirk) {
  if (quirk)
    staged_map<9, 3>(in, out, M, [](const float* a, float* r) { rotmat_to_aa_kornia_quirk_one(a, r); });
  else
    staged_map<9, 3>(in, out, M, [](const float* a, float* r) { rotmat_to_aa_one(a, r); });
}

__global__ void __launch_bounds__(kConvThreads + 32) rot6d_bulk_kernel(const float* in, float* out, int64_t n_tiles) {
  bulk_map<6, 9>(in, out, n_tiles, [](const float* a, float* r) { rot6d_one(a, r); });
}
__global__ void __launch_bounds__(kConvThreads + 32) aa_kornia_bulk_kernel(const float* in, float* out, int64_t n_tiles) {
  bulk_map<3, 9>(in, out, n_tiles, [](const float* a, float* r) { aa_kornia_one(a, r); });
}
__global__ void __launch_bounds__(kConvThreads + 32) rodrigues_bulk_kernel(const float* in, float* out, int64_t n_tiles) {
  bulk_map<3, 9>(in, out, n_tiles, [](const float* a, float* r) { rodrigues_one(a, r); });
}
__global__ void __launch_bounds__(kConvThreads + 32) rotmat_to_aa_bulk_kernel(const float* in, float* out, int64_t n_tiles, int quirk) {
  if (quirk)
    bulk_map<9, 3>(in, out, n_tiles, [](const float* a, float* r) { rotmat_to_aa_kornia_quirk_one(a, r); });
  else
    bulk_map<9, 3>(in, out, n_tiles, [](const float* a, float* r) { rotmat_to_aa_one(a, r); });
}

__global__ void __launch_bounds__(kConvThreads) quat2mat_kernel(const float* in, float* out, int64_t M) {
  staged_map<4, 9>(in, out, M, [](const float* a, float* r) { quat2mat_one(a, r); });
}
__global__ void __launch_bounds__(kConvThreads) rotmat_to_quat_kernel(const float* in, float* out, int64_t M) {
  staged_map<9, 4>(in, out, M, [](const float* a, float* r) { rotmat_to_quat_one(a, r); });
}
__global__ void __launch_bounds__(kConvThreads) quat_to_aa_kernel(const float* in, float* out, int64_t M) {
  staged_map<4, 3>(in, out, M, [](const float* a, float* r) { quat_to_aa(a[0], a[1], a[2], a[3], r); });
}

template <class K>
static int launch_staged(K kernel, const void* in, void* out, int64_t M, cudaStream_t s) {
  TIK_CHECK_ARG(M >= 0, "negative count");
  if (M == 0) return TIK_OK;
  TIK_CHECK_ARG(in && out, "null pointer");
  TIK_CHECK_ARG((((uintptr_t)in | (uintptr_t)out) & 15) == 0, "pointers must be 16-byte aligned");
  const int64_t blocks = ceil_div(M, kConvThreads);
  TIK_CHECK_ARG(blocks < (1ll << 31), "too many rotations for one launch");
  kernel<<<(unsigned)blocks, kConvThreads, 0, s>>>((const float*)in, (float*)out, M);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}

static bool conv_bulk_enabled() {
  static int v = -1;
  if (v < 0) v = getenv("TIK_NO_CONV_BULK") ? 0 : 1;
  return v != 0;
}

// whole 256-rotation tiles -> the bulk-pipelined kernel (persistent CTAs); the remainder (and small batches) -> the
// staged kernel
template <int IN, int OUT, class KB, class K, class... Args>
static int launch_conv(KB bulk_kernel, K kernel, const void* in, void* out, int64_t M, cudaStream_t s, Args... extra) {
  TIK_CHECK_ARG(M >= 0, "negative count");
  if (M == 0) return TIK_OK;
  TIK_CHECK_ARG(in && out, "null pointer");
  TIK_CHECK_ARG((((uintptr_t)in | (uintptr_t)out) & 15) == 0, "pointers must be 16-byte aligned");
  const float* fin = (const float*)in;
  float* fout = (float*)out;
  const int64_t n_tiles = M / kConvThreads;
  if (conv_bulk_enabled() && n_tiles >= 148) {
    constexpr size_t smem = (size_t)kConvStages * kConvThreads * (IN + OUT) * 4 + 2 * kConvStages * sizeof(uint64_t);
    // function attributes are per (kernel, device); several kernels share this template instantiation
    static const void* attr_kernel[16] = {};
    static uint64_t attr_devs[16] = {};
    int dev = 0;
    TIK_CUDA(cudaGetDevice(&dev));
    int slot = 0;
    while (slot < 15 && attr_kernel[slot] && attr_kernel[slot] != (const void*)bulk_kernel) ++slot;
    if (attr_kernel[slot] != (const void*)bulk_kernel || !(attr_devs[slot] >> (dev & 63) & 1)) {
      TIK_CUDA(cudaFuncSetAttribute(bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      TIK_CUDA(cudaFuncSetAttribute(bulk_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      if (attr_kernel[slot] != (const void*)bulk_kernel) { attr_kernel[slot] = (const void*)bulk_kernel; attr_devs[slot] = 0; }
      attr_devs[slot] |= 1ull << (dev & 63);
    }
    const int per_sm = (int)std::min<size_t>(7, (227 * 1024) / (smem + 1024));     // 288 threads per CTA, 2048 per SM
    const int64_t blocks = std::min<int64_t>(n_tiles, (int64_t)148 * per_sm);
    bulk_kernel<<<(unsigned)blocks, kConvThreads + 32, smem, s>>>(fin, fout, n_tiles, extra...);
    TIK_LAUNCH_CHECK();
    const int64_t covered = n_tiles * kConvThreads;
    fin += covered * IN;
    fout += covered * OUT;
    M -= covered;
    if (M == 0) return TIK_OK;
  }
  int64_t blocks = ceil_div(M, kConvThreads);
  TIK_CHECK_ARG(blocks < (1ll << 31), "too many rotations for one launch");
  kernel<<<(unsigned)blocks, kConvThreads, 0, s>>>(fin, fout, M, extra...);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}

// Per-frame mean of overlapping window predictions, one window per frame (inference.window_mean, reference
// inference.py:56-67), for every sequence of a ragged batch in one launch.  One thread per output value (euclidean) or
// per joint (rotation).  The sums run over o = -h..h in ascending order from 0 and end in one IEEE division by the
// count: the operation order of inference._window_sum followed by acc / cnt, so the euclidean mean is bit-identical
// to the per-sequence torch route, and the rotation mean goes through the same device functions as tik_batch_rodrigues,
// tik_rot6d_to_rotmat and tik_rotmat_to_aa.
template <int MODE>
__global__ void __launch_bounds__(kConvThreads) window_mean_kernel(const float* __restrict__ preds, long long frames, int T_out,
                                                                 int D, const int64_t* __restrict__ frame_start, long long n_seqs,
                                                                 int h, float* __restrict__ out) {
  const int per_frame = MODE == TIK_MEAN_ROTATION ? D / 3 : D;
  const long long e = (long long)blockIdx.x * kConvThreads + threadIdx.x;
  if (e >= frames * per_frame) return;
  const long long j = e / per_frame;
  const int d = (int)(e - j * per_frame) * (MODE == TIK_MEAN_ROTATION ? 3 : 1);
  // sequence of frame j: the last s with frame_start[s] <= j; indices clamped to [0, frames) against malformed tables
  long long lo = 0, hi = n_seqs - 1;
  while (lo < hi) {
    const long long mid = (lo + hi + 1) >> 1;
    if (__ldg(frame_start + mid) <= j) lo = mid; else hi = mid - 1;
  }
  const long long f0 = min(max((long long)__ldg(frame_start + lo), 0ll), frames - 1);
  const long long F = min(max((long long)__ldg(frame_start + lo + 1), f0 + 1), frames) - f0;
  const long long i = j - f0;
  float cnt = 0.f;
  if (MODE == TIK_MEAN_EUCLIDEAN) {
    float acc = 0.f;
    for (int o = -h; o <= h; ++o) {
      const long long src = i - o;
      if (src < 0 || src >= F) continue;
      acc += __ldg(preds + ((f0 + src) * T_out + o + h) * D + d);
      cnt += 1.f;
    }
    out[j * D + d] = __fdiv_rn(acc, cnt);
  } else {
    float acc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = 0.f;
    for (int o = -h; o <= h; ++o) {
      const long long src = i - o;
      if (src < 0 || src >= F) continue;
      const float* p = preds + ((f0 + src) * T_out + o + h) * D + d;
      const float a[3] = {__ldg(p), __ldg(p + 1), __ldg(p + 2)};
      float R[9];
      rodrigues_one(a, R);
#pragma unroll
      for (int k = 0; k < 9; ++k) acc[k] += R[k];
      cnt += 1.f;
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = __fdiv_rn(acc[k], cnt);
    const float x6[6] = {acc[0], acc[1], acc[3], acc[4], acc[6], acc[7]};   // first two columns, row by row (x6 of window_mean)
    float R[9], aa[3];
    rot6d_one(x6, R);
    rotmat_to_aa_one(R, aa);
#pragma unroll
    for (int k = 0; k < 3; ++k) out[j * D + d + k] = aa[k];
  }
}

// h = 0: every frame takes its own window's first prediction (preds[:, 0]) in both modes
__global__ void __launch_bounds__(kConvThreads) window_first_kernel(const float* __restrict__ preds, long long frames, int T_out,
                                                                  int D, float* __restrict__ out) {
  const long long e = (long long)blockIdx.x * kConvThreads + threadIdx.x;
  if (e >= frames * D) return;
  const long long j = e / D;
  out[e] = __ldg(preds + j * T_out * D + (e - j * D));
}

int launch_batch_rodrigues(const float* aa, float* R9, int64_t M, cudaStream_t s) {
  return launch_conv<3, 9>(rodrigues_bulk_kernel, rodrigues_kernel, aa, R9, M, s);
}

}  // namespace tik

extern "C" {
int tik_rot6d_to_rotmat(const float* x6, float* R, int64_t M, void* stream) {
  return tik::launch_conv<6, 9>(tik::rot6d_bulk_kernel, tik::rot6d_kernel, x6, R, M, (cudaStream_t)stream);
}
int tik_aa_to_rotmat(const float* aa, float* R, int64_t M, void* stream) {
  return tik::launch_conv<3, 9>(tik::aa_kornia_bulk_kernel, tik::aa_kornia_kernel, aa, R, M, (cudaStream_t)stream);
}
int tik_batch_rodrigues(const float* aa, float* R9, int64_t M, void* stream) {
  return tik::launch_conv<3, 9>(tik::rodrigues_bulk_kernel, tik::rodrigues_kernel, aa, R9, M, (cudaStream_t)stream);
}
int tik_quat_to_rotmat(const float* q, float* R, int64_t M, void* stream) {
  return tik::launch_staged(tik::quat2mat_kernel, q, R, M, (cudaStream_t)stream);
}
int tik_rotmat_to_quat(const float* R, float* q, int64_t M, void* stream) {
  return tik::launch_staged(tik::rotmat_to_quat_kernel, R, q, M, (cudaStream_t)stream);
}
int tik_quat_to_aa(const float* q, float* aa, int64_t M, void* stream) {
  return tik::launch_staged(tik::quat_to_aa_kernel, q, aa, M, (cudaStream_t)stream);
}
int tik_rotmat_to_aa(const float* R, float* aa, int64_t M, int kornia_quirk, void* stream) {
  return tik::launch_conv<9, 3>(tik::rotmat_to_aa_bulk_kernel, tik::rotmat_to_aa_kernel, R, aa, M, (cudaStream_t)stream, kornia_quirk);
}
int tik_window_mean(const float* preds, int64_t frames, int T_out, int D, const int64_t* frame_start, int64_t n_seqs,
                    int h, int mode, float* out, void* stream) {
  using namespace tik;
  TIK_CHECK_ARG(preds && out && frame_start, "window mean: null preds, out or frame_start pointer");
  TIK_CHECK_ARG(n_seqs >= 1, "window mean: n_seqs = %lld, need >= 1", (long long)n_seqs);
  TIK_CHECK_ARG(frames >= 0 && T_out >= 1 && D >= 1, "window mean: bad shape frames=%lld T_out=%d D=%d", (long long)frames, T_out, D);
  TIK_CHECK_ARG(mode == TIK_MEAN_EUCLIDEAN || mode == TIK_MEAN_ROTATION, "window mean: unknown mode %d", mode);
  TIK_CHECK_ARG(h >= 0 && 2 * h + 1 <= T_out, "window mean: h_w_size = %d needs 2h+1 <= T_out = %d predictions per window", h, T_out);
  TIK_CHECK_ARG(mode != TIK_MEAN_ROTATION || D % 3 == 0, "window mean: rotation mode needs D divisible by 3, got %d", D);
  if (frames == 0) return TIK_OK;
  const int per_frame = (mode == TIK_MEAN_ROTATION && h > 0) ? D / 3 : D;
  const int64_t blocks = ceil_div(frames * per_frame, kConvThreads);
  TIK_CHECK_ARG(blocks < (1ll << 31), "window mean: too many frames for one launch");
  cudaStream_t s = (cudaStream_t)stream;
  if (h == 0)
    window_first_kernel<<<(unsigned)blocks, kConvThreads, 0, s>>>(preds, (long long)frames, T_out, D, out);
  else if (mode == TIK_MEAN_EUCLIDEAN)
    window_mean_kernel<TIK_MEAN_EUCLIDEAN><<<(unsigned)blocks, kConvThreads, 0, s>>>(preds, (long long)frames, T_out, D, frame_start,
                                                                                     (long long)n_seqs, h, out);
  else
    window_mean_kernel<TIK_MEAN_ROTATION><<<(unsigned)blocks, kConvThreads, 0, s>>>(preds, (long long)frames, T_out, D, frame_start,
                                                                                    (long long)n_seqs, h, out);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}
}
