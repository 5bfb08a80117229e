// Linear blend skinning of an SMPL-X mesh: the vertex half of smplx.lbs.lbs (published SMPL-X formulation, restated in
// oracle/lbs_port.py) on top of tik_fk_body's joints and rotations.  Per chunk of frames:
//   1. lbs_prep_kernel: pose features (R_local[1:] - I) straight into the GEMM's K-contiguous (F_chunk, 512) operand,
//      relative transforms A_j = [G_j | t_j - G_j rest_j] (F_chunk, 55, 12) fp32, posed joints + transl.
//   2. pose blend offsets = posedirs (3V_pad, 512) . features^T on the existing implicit-GEMM kernels (3xTF32 for fp32,
//      tcgen05 bf16 for bf16), transposed so that the frames are the GEMM's columns: the zero bias row is F_chunk floats
//      and the ring keeps its stages (the natural orientation has c_out = 3V_pad and a 126 KB bias table).
//   3. lbs_skin_kernel: v = (sum_k w_k A_{j_k}) (v_shaped + offset) + transl, the chunk's transforms in shared memory,
//      offsets read back from L2, vertices written row-contiguous.
#include <stdlib.h>

#include <algorithm>

#include "tik_common.cuh"

namespace tik {

constexpr int kLbsJ = 55;
constexpr int kLbsFeat = (kLbsJ - 1) * 9;      // 486 pose features
constexpr int kLbsK = 512;                     // feature columns, zero padded to whole 64-wide K chunks
constexpr int kPrepThreads = 256;
constexpr int kSkinFt = 32;                    // frames per skin tile: one per lane
constexpr int kSkinVt = 32;                    // vertices per skin tile: four per warp
constexpr int kSkinThreads = 256;
constexpr int kApitch = kSkinFt + 1;           // shared transforms [55*12][33]: conflict-free transposed fill
constexpr int kOpitch = kSkinVt * 3 + 1;       // shared output tile [32 frames][97]
// shared memory of the skin kernel: transforms, transl, output tile, then the vertex tile's skinning table and v_shaped
constexpr size_t kSkinSmemFixed = sizeof(float) * ((size_t)kLbsJ * 12 * kApitch + kSkinFt * 3 + (size_t)kSkinFt * kOpitch + kSkinVt * 3);
static size_t skin_smem(int kmax) { return kSkinSmemFixed + (size_t)kSkinVt * kmax * 8; }
// Frames per chunk: the largest multiple of 64 whose fp32 offsets (3V_pad x chunk x 4 B) fit 32 MB, in [64, 1024] and no
// more than F needs: 256 at V = 10,475, where the offsets stay in L2 next to posedirs (32 MB bf16, 64 MB fp32) for the
// skin kernel.  Measured on a B200 (tools/bench_mesh.py, DESIGN.md section 9): 128 / 256 / 512 frames per chunk take
// 12.6 / 10.7 / 12.6 ms (fp32) and 10.5 / 8.7 / 11.0 ms (bf16) for 16,384 frames -- 128 pays twice the launches and
// per-launch tails, 512 makes the skin kernel's offset reads miss L2.  TIK_LBS_CHUNK (a multiple of 64) overrides it for
// such measurements.
constexpr int64_t kLbsOffsetsBudget = 32ll << 20;
constexpr int kLbsMaxChunk = 1024;

static int64_t lbs_rows_pad(int V) { return ceil_div(3ll * V, 128) * 128; }

static int lbs_chunk(const TikLbsModel* m, int64_t F) {
  int64_t fc = (kLbsOffsetsBudget / (lbs_rows_pad(m->V) * 4)) / 64 * 64;
  if (const char* e = getenv("TIK_LBS_CHUNK")) {
    const int want = atoi(e);
    if (want >= 64 && want % 64 == 0) fc = want;
  }
  fc = std::max<int64_t>(64, std::min<int64_t>(fc, kLbsMaxChunk));
  return (int)std::min<int64_t>(fc, ceil_div(std::max<int64_t>(F, 1), 64) * 64);
}

struct LbsWorkspace { void* feat; float* A; float* offsets; float* bias; int64_t bytes; };

static LbsWorkspace lbs_layout(const TikLbsModel* m, int dtype, int fc, char* base) {
  auto up = [](int64_t b) { return (b + 255) / 256 * 256; };
  LbsWorkspace w;
  int64_t off = 0;
  w.feat = base + off;
  off += up((int64_t)fc * kLbsK * (dtype == TIK_BF16 ? 2 : 4));
  w.A = reinterpret_cast<float*>(base + off);
  off += up((int64_t)fc * kLbsJ * 12 * 4);
  w.offsets = reinterpret_cast<float*>(base + off);
  off += up(lbs_rows_pad(m->V) * fc * 4);
  w.bias = reinterpret_cast<float*>(base + off);
  off += up((int64_t)fc * 4);
  w.bytes = off;
  return w;
}

template <class T> __device__ __forceinline__ T to_op(float v);
template <> __device__ __forceinline__ float to_op<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 to_op<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// One grid-stride pass over the chunk's (fc, 512) feature operand; the first fc threads also zero the GEMM's bias row and
// the first nf * 55 threads write the frame's relative transform and posed joint (+ transl) of one joint.
template <class T>
__global__ void __launch_bounds__(kPrepThreads) lbs_prep_kernel(const float* __restrict__ joints, const float* __restrict__ local_R,
                                                                const float* __restrict__ global_R, int fk_J,
                                                                const float* __restrict__ rest, const float* __restrict__ transl,
                                                                int nf, int fc, T* __restrict__ feat, float* __restrict__ A,
                                                                float* __restrict__ bias, float* __restrict__ joints_out, int jo_J) {
  const int64_t n_feat = (int64_t)fc * kLbsK;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_feat; i += (int64_t)gridDim.x * blockDim.x) {
    const int f = (int)(i / kLbsK), col = (int)(i % kLbsK);
    float v = 0.f;
    if (f < nf && col < kLbsFeat) {                     // smplx order: column 9 (j - 1) + 3 a + b of (R_j - I)
      const int e = col % 9;
      v = __ldg(local_R + ((int64_t)f * fk_J + 1) * 9 + col) - (e == 0 || e == 4 || e == 8 ? 1.f : 0.f);
    }
    feat[i] = to_op<T>(v);
    if (i < fc) bias[i] = 0.f;
    if (i < (int64_t)nf * kLbsJ) {
      const int ff = (int)(i / kLbsJ), j = (int)(i % kLbsJ);
      const float* G = global_R + ((int64_t)ff * fk_J + j) * 9;
      const float* t = joints + ((int64_t)ff * fk_J + j) * 3;
      const float r0 = __ldg(rest + j * 3), r1 = __ldg(rest + j * 3 + 1), r2 = __ldg(rest + j * 3 + 2);
      float* a = A + i * 12;
#pragma unroll
      for (int row = 0; row < 3; ++row) {
        const float g0 = __ldg(G + row * 3), g1 = __ldg(G + row * 3 + 1), g2 = __ldg(G + row * 3 + 2), tr = __ldg(t + row);
        a[row * 4] = g0;
        a[row * 4 + 1] = g1;
        a[row * 4 + 2] = g2;
        a[row * 4 + 3] = tr - (g0 * r0 + g1 * r1 + g2 * r2);
        if (joints_out != nullptr && j < jo_J)
          joints_out[((int64_t)ff * jo_J + j) * 3 + row] = tr + (transl ? __ldg(transl + (int64_t)ff * 3 + row) : 0.f);
      }
    }
  }
}

struct LbsLandmarks { int n; int vid[TIK_LBS_MAX_LANDMARKS]; };

// Block = one 32-frame tile of the chunk x a strided set of 32-vertex tiles.  Lane = frame, so the offsets of one vertex
// coordinate are one coalesced 128 B row of the (3V_pad, fc) GEMM output and the transforms are read from shared memory
// without conflicts; results go through a shared tile so that each frame's 32 vertices are stored as 384 contiguous bytes.
__global__ void __launch_bounds__(kSkinThreads, 2) lbs_skin_kernel(
    const float* __restrict__ offsets, int fc, const float* __restrict__ v_shaped, const int32_t* __restrict__ skin_idx,
    const float* __restrict__ skin_w, int kmax, int V, const float* __restrict__ A, const float* __restrict__ transl,
    int nf, int n_ftiles, int vsplit, float* __restrict__ verts, float* __restrict__ joints_out, int jo_J,
    const LbsLandmarks lm) {
  extern __shared__ __align__(16) float lbs_smem[];
  float* sA = lbs_smem;                               // [(j * 12 + e) * 33 + frame]
  float* sT = sA + kLbsJ * 12 * kApitch;              // [frame * 3 + c]
  float* sO = sT + kSkinFt * 3;                       // [frame * 97 + vertex * 3 + c]
  const int ft = blockIdx.x % n_ftiles, vs = blockIdx.x / n_ftiles;
  const int f0 = ft * kSkinFt;
  const int nft = min(kSkinFt, nf - f0);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < nft * kLbsJ * 12; i += kSkinThreads) {
    const int f = i / (kLbsJ * 12), r = i % (kLbsJ * 12);
    sA[r * kApitch + f] = __ldg(A + (int64_t)(f0 + f) * kLbsJ * 12 + r);
  }
  for (int i = tid; i < kSkinFt * 3; i += kSkinThreads)
    sT[i] = (transl != nullptr && i < nft * 3) ? __ldg(transl + (int64_t)f0 * 3 + i) : 0.f;
  __syncthreads();
  const int n_vt = (V + kSkinVt - 1) / kSkinVt;
  const bool lane_on = lane < nft;
  const float tx = sT[lane * 3], ty = sT[lane * 3 + 1], tz = sT[lane * 3 + 2];
  float* sV = sO + kSkinFt * kOpitch;                 // [vertex * 3 + c] v_shaped of the vertex tile
  float* sW = sV + kSkinVt * 3;                       // [vertex * kmax + k] skinning weights of the vertex tile
  int32_t* sI = reinterpret_cast<int32_t*>(sW + kSkinVt * kmax);   // and their joints
  for (int vt = vs; vt < n_vt; vt += vsplit) {
    const int v0 = vt * kSkinVt;
    const int nv = min(kSkinVt, V - v0);
    // the tile's table and rest vertices in one coalesced pass, so that no warp waits on a dependent global load below
    for (int i = tid; i < nv * kmax; i += kSkinThreads) {
      sI[i] = __ldg(skin_idx + (int64_t)v0 * kmax + i);
      sW[i] = __ldg(skin_w + (int64_t)v0 * kmax + i);
    }
    if (tid < nv * 3) sV[tid] = __ldg(v_shaped + (int64_t)v0 * 3 + tid);
    float off[kSkinVt / 8][3];
#pragma unroll
    for (int q = 0; q < kSkinVt / 8; ++q) {           // all twelve offset loads of the warp in flight at once
      const int v = v0 + warp + 8 * q;
      const float* orow = offsets + (int64_t)v * 3 * fc + f0 + lane;
      const bool ok = v < V && lane_on;
#pragma unroll
      for (int c = 0; c < 3; ++c) off[q][c] = ok ? __ldg(orow + c * fc) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < kSkinVt / 8; ++q) {
      const int vl = warp + 8 * q, v = v0 + vl;
      if (v >= V || !lane_on) continue;
      const float px = sV[vl * 3] + off[q][0], py = sV[vl * 3 + 1] + off[q][1], pz = sV[vl * 3 + 2] + off[q][2];
      float T[12];
#pragma unroll
      for (int e = 0; e < 12; ++e) T[e] = 0.f;
      for (int k = 0; k < kmax; ++k) {
        const int j = sI[vl * kmax + k];
        const float w = sW[vl * kmax + k];
        const float* a = sA + j * 12 * kApitch + lane;
#pragma unroll
        for (int e = 0; e < 12; ++e) T[e] = fmaf(w, a[e * kApitch], T[e]);
      }
      const float ox = fmaf(T[0], px, fmaf(T[1], py, fmaf(T[2], pz, T[3]))) + tx;
      const float oy = fmaf(T[4], px, fmaf(T[5], py, fmaf(T[6], pz, T[7]))) + ty;
      const float oz = fmaf(T[8], px, fmaf(T[9], py, fmaf(T[10], pz, T[11]))) + tz;
      float* so = sO + lane * kOpitch + vl * 3;
      so[0] = ox; so[1] = oy; so[2] = oz;
      for (int k = 0; k < lm.n; ++k)                   // face landmark joints are mesh vertices (smplx VertexJointSelector)
        if (lm.vid[k] == v && joints_out != nullptr) {
          float* jo = joints_out + ((int64_t)(f0 + lane) * jo_J + kLbsJ + k) * 3;
          jo[0] = ox; jo[1] = oy; jo[2] = oz;
        }
    }
    __syncthreads();
    for (int i = tid; i < nft * kSkinVt * 3; i += kSkinThreads) {
      const int f = i / (kSkinVt * 3), c = i % (kSkinVt * 3);
      if (c < nv * 3) verts[((int64_t)(f0 + f) * V + v0) * 3 + c] = sO[f * kOpitch + c];
    }
    __syncthreads();
  }
}

static int lbs_check_model(const TikLbsModel* m) {
  TIK_CHECK_ARG(m != nullptr, "null model");
  TIK_CHECK_ARG(m->V >= 1 && m->J == kLbsJ, "lbs: V=%d must be >= 1 and J=%d must be %d", m->V, m->J, kLbsJ);
  TIK_CHECK_ARG(m->kmax >= 1 && m->kmax <= kLbsJ, "lbs: kmax=%d outside [1,%d]", m->kmax, kLbsJ);
  TIK_CHECK_ARG(m->n_landmarks >= 0 && m->n_landmarks <= TIK_LBS_MAX_LANDMARKS, "lbs: n_landmarks=%d outside [0,%d]",
                m->n_landmarks, TIK_LBS_MAX_LANDMARKS);
  for (int k = 0; k < m->n_landmarks; ++k)
    TIK_CHECK_ARG(m->landmark_vid[k] >= 0 && m->landmark_vid[k] < m->V, "lbs: landmark vertex %d outside [0,%d)", m->landmark_vid[k], m->V);
  TIK_CHECK_ARG(m->v_shaped_dev && m->rest_joints_dev && m->posedirs_dev && m->skin_idx_dev && m->skin_w_dev, "lbs: null model pointer");
  TIK_CHECK_ARG(3ll * m->V <= (1ll << 30), "lbs: V=%d too large", m->V);
  return TIK_OK;
}

}  // namespace tik

extern "C" int tik_lbs_workspace_bytes(const TikLbsModel* m, int dtype, int64_t F, int64_t* bytes) {
  using namespace tik;
  int rc = lbs_check_model(m);
  if (rc != TIK_OK) return rc;
  TIK_CHECK_ARG(dtype == TIK_F32 || dtype == TIK_BF16, "bad dtype %d", dtype);
  TIK_CHECK_ARG(F >= 0 && bytes != nullptr, "lbs: bad arguments");
  *bytes = lbs_layout(m, dtype, lbs_chunk(m, F), nullptr).bytes;
  return TIK_OK;
}

extern "C" int tik_lbs(const TikLbsModel* m, int dtype, const float* joints_dev, const float* local_R_dev,
                       const float* global_R_dev, int fk_J, const float* transl_dev, int64_t F, void* workspace_dev,
                       int64_t workspace_bytes, float* verts_dev, float* joints_out_dev, int joints_out_J, void* stream) {
  using namespace tik;
  int rc = lbs_check_model(m);
  if (rc != TIK_OK) return rc;
  TIK_CHECK_ARG(dtype == TIK_F32 || dtype == TIK_BF16, "bad dtype %d", dtype);
  TIK_CHECK_ARG(F >= 0, "negative frame count");
  TIK_CHECK_ARG(fk_J >= kLbsJ && fk_J <= TIK_MAX_JOINTS, "lbs: fk_J=%d outside [%d,%d]", fk_J, kLbsJ, TIK_MAX_JOINTS);
  TIK_CHECK_ARG(joints_out_dev == nullptr || (joints_out_J >= 1 && joints_out_J <= kLbsJ) || joints_out_J == kLbsJ + m->n_landmarks,
                "lbs: joints_out_J=%d must be in [1,%d] or %d", joints_out_J, kLbsJ, kLbsJ + m->n_landmarks);
  if (F == 0) return TIK_OK;
  TIK_CHECK_ARG(joints_dev && local_R_dev && global_R_dev && verts_dev && workspace_dev, "null pointer");
  const int fc = lbs_chunk(m, F);
  const LbsWorkspace ws = lbs_layout(m, dtype, fc, reinterpret_cast<char*>(workspace_dev));
  if (workspace_bytes < ws.bytes) {
    set_error("lbs: workspace of %lld bytes, %lld needed", (long long)workspace_bytes, (long long)ws.bytes);
    return TIK_ERR_WORKSPACE;
  }
  TIK_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace_dev) & 255) == 0 && (reinterpret_cast<uintptr_t>(m->posedirs_dev) & 15) == 0,
                "lbs: workspace must be 256-byte and posedirs 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  static bool attr_set[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (!attr_set[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(lbs_skin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)skin_smem(kLbsJ)));
    attr_set[dev & 63] = true;
  }
  int sms = 148;
  TIK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int64_t rows = lbs_rows_pad(m->V);
  LbsLandmarks lm;
  lm.n = joints_out_J == kLbsJ + m->n_landmarks ? m->n_landmarks : 0;
  for (int k = 0; k < TIK_LBS_MAX_LANDMARKS; ++k) lm.vid[k] = k < lm.n ? m->landmark_vid[k] : -1;
  // Every chunk hands the GEMM the same descriptor (the ragged last chunk keeps fc columns, its pad rows are zero), so the
  // bf16 path prepares its tensor maps once.
  TikRowGemm g;
  memset(&g, 0, sizeof(g));
  g.n_slabs = 1;
  g.slabs[0].a_dev = m->posedirs_dev; g.slabs[0].c = kLbsK; g.slabs[0].t_in = (int32_t)rows; g.slabs[0].t_mul = 1; g.slabs[0].t_off = 0;
  g.w_dev = ws.feat; g.bias_dev = ws.bias; g.bias_per_node = 0;
  g.nv = 1; g.v = 1; g.t_out = (int32_t)rows; g.c_out = fc; g.c_out_valid = fc;
  g.act = TIK_ACT_NONE; g.res_kind = TIK_RES_NONE; g.out_dev = ws.offsets; g.out_layout = TIK_OUT_ROWS_F32;
  const int n_vt = (int)ceil_div(m->V, kSkinVt);
  for (int64_t c0 = 0; c0 < F; c0 += fc) {
    const int nf = (int)std::min<int64_t>(fc, F - c0);
    const float* jc = joints_dev + c0 * fk_J * 3;
    const float* lc = local_R_dev + c0 * fk_J * 9;
    const float* gc = global_R_dev + c0 * fk_J * 9;
    const float* tc = transl_dev ? transl_dev + c0 * 3 : nullptr;
    float* joc = joints_out_dev ? joints_out_dev + c0 * joints_out_J * 3 : nullptr;
    const unsigned prep_blocks = (unsigned)std::min<int64_t>(ceil_div((int64_t)fc * kLbsK, kPrepThreads), (int64_t)sms * 8);
    if (dtype == TIK_BF16)
      lbs_prep_kernel<__nv_bfloat16><<<prep_blocks, kPrepThreads, 0, s>>>(jc, lc, gc, fk_J, m->rest_joints_dev, tc, nf, fc,
          reinterpret_cast<__nv_bfloat16*>(ws.feat), ws.A, ws.bias, joc, joints_out_J);
    else
      lbs_prep_kernel<float><<<prep_blocks, kPrepThreads, 0, s>>>(jc, lc, gc, fk_J, m->rest_joints_dev, tc, nf, fc,
          reinterpret_cast<float*>(ws.feat), ws.A, ws.bias, joc, joints_out_J);
    TIK_LAUNCH_CHECK();
    rc = dtype == TIK_BF16 ? rowgemm_bf16(&g, s) : rowgemm_f32(&g, s);
    if (rc != TIK_OK) return rc;
    // two resident blocks per SM (kmax <= 32) over (frame tiles x vertex slices): each block stages its 32 frames' transforms once
    // and reuses them for every vertex tile of its slice
    const int n_ftiles = (int)ceil_div(nf, kSkinFt);
    const int vsplit = (int)std::max<int64_t>(1, std::min<int64_t>(n_vt, ceil_div(2ll * sms, n_ftiles)));
    lbs_skin_kernel<<<(unsigned)(n_ftiles * vsplit), kSkinThreads, skin_smem(m->kmax), s>>>(
        ws.offsets, fc, m->v_shaped_dev, m->skin_idx_dev, m->skin_w_dev, m->kmax, m->V, ws.A, tc, nf, n_ftiles, vsplit,
        verts_dev + c0 * m->V * 3, joc, joints_out_J, lm);
    TIK_LAUNCH_CHECK();
  }
  return TIK_OK;
}
