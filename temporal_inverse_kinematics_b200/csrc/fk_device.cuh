// Device pieces shared by the thread-per-frame FK kernels (fk.cu) and the keypoint kernel (keypoints.cu): the
// compile-time SMPL-X tree, the SFU Rodrigues, and 1-D bulk copies between global and shared memory.
#pragma once
#include "tik_common.cuh"
#include "umma_ptx.cuh"

namespace tik {

// parents of the 55 SMPL-X joints followed by the five face landmarks hanging off the head (60-joint full skeleton)
constexpr int kF60 = 60;
__host__ __device__ constexpr int f60_parent(int j) {
  constexpr int P[kF60] = {-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 15, 15, 15,
                           20, 25, 26, 20, 28, 29, 20, 31, 32, 20, 34, 35, 20, 37, 38,
                           21, 40, 41, 21, 43, 44, 21, 46, 47, 21, 49, 50, 21, 52, 53, 15, 15, 15, 15, 15};
  return P[j];
}

__device__ __forceinline__ void bulk_load_1d(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_store_1d(void* dst, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(dst), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void rodrigues_q_fast(float ax, float ay, float az, float* R) {
  // common/geometry.py:22-65 with SFU sin / cos / rsqrt
  float ex = ax + 1e-8f, ey = ay + 1e-8f, ez = az + 1e-8f;
  float n2 = ex * ex + ey * ey + ez * ez;
  float ia = rsqrtf(n2);
  float ang = n2 * ia;
  float nx = ax * ia, ny = ay * ia, nz = az * ia;
  float s, c;
  __sincosf(ang * 0.5f, &s, &c);
  float w = c, x = s * nx, y = s * ny, z = s * nz;
  float iq = rsqrtf(w * w + x * x + y * y + z * z);   // quaternion re-normalisation (quat2mat, geometry.py:49)
  w *= iq; x *= iq; y *= iq; z *= iq;
  float w2 = w * w, x2 = x * x, y2 = y * y, z2 = z * z;
  float wx = w * x, wy = w * y, wz = w * z, xy = x * y, xz = x * z, yz = y * z;
  R[0] = w2 + x2 - y2 - z2; R[1] = 2.f * (xy - wz);       R[2] = 2.f * (wy + xz);
  R[3] = 2.f * (wz + xy);   R[4] = w2 - x2 + y2 - z2;     R[5] = 2.f * (yz - wx);
  R[6] = 2.f * (xz - wy);   R[7] = 2.f * (wx + yz);       R[8] = w2 - x2 - y2 + z2;
}

}  // namespace tik
