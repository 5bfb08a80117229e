// Stem of the ST-GCN backbone: everything block 0 does to the raw 3-channel keypoints, in one pass.
//
//   X0 = data_bn(x)                                             st_gcn_aaai18.py:119-125 (channel index v*C+c)
//   H0[n,w,t,:] = relu( Wg' . (sum_v A^[k,v,w] X0[n,t,v,:]) + b1[w,:] )   gconv_origin.py:56-65 + tcn.0/tcn.1
//   R0[n,w,t',:] = Wr'[w] . x[n, s*t', w, :]                    residual 1x1 conv + BN (st_gcn_aaai18.py:198-204),
//                                                               data_bn scale folded into Wr', constants into the
//                                                               temporal conv's per-node bias
//
// Input is the reference's (N,T,V,Cin) fp32 layout; outputs are node-major (N,V,T,Cout) so that the temporal
// convolution's TMA boxes are dense.  HBM-bound: Cin*4*V B in, 2 * V*Cout*sizeof(T) B out per frame.
// One CTA handles kStemFrames frames of one clip; each thread produces 8 consecutive channels (one 16 B store).
#include <algorithm>

#include "tik_common.cuh"

namespace tik {

constexpr int kStemFrames = 32;
constexpr int kStemThreads = 288;   // >= 2 x 17 nodes x 8 channel groups (Cout = 64)
constexpr int kStemMaxV = 32;
constexpr int kStemMaxKC = 40;  // K * Cin

template <class T> __device__ __forceinline__ void store8(T* p, const float* a);
template <> __device__ __forceinline__ void store8<float>(float* p, const float* a) {
  reinterpret_cast<float4*>(p)[0] = make_float4(a[0], a[1], a[2], a[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(a[4], a[5], a[6], a[7]);
}
template <> __device__ __forceinline__ void store8<__nv_bfloat16>(__nv_bfloat16* p, const float* a) {
  uint4 t;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&t);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(a[2 * i], a[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = t;
}

// Thread t owns one (node w, 8-channel group g) pair for the whole CTA: its 8 x K*Cin weights, 8 biases and
// 8 x Cin residual weights live in registers, and it walks the CTA's frames writing one 16-byte vector per frame
// and tensor (consecutive frames of one node are consecutive 2*Cout-byte rows of the node-major output).
constexpr int kStemMaxKCReg = 16;  // register-resident weights: K*Cin <= 16 (IK model: 1 x 3 -> KCR = 4; spatial K=5 -> 15)

template <class OutT, int KCR, int CINR>
__global__ void __launch_bounds__(kStemThreads, (KCR <= 4 ? 3 : 1))
stem_gcn_kernel(const float* __restrict__ x, const float* __restrict__ in_scale, const float* __restrict__ in_shift,
                const float* __restrict__ agg, const float* __restrict__ w, const float* __restrict__ bias,
                OutT* __restrict__ out, const float* __restrict__ res_w, OutT* __restrict__ res_out, int res_stride,
                int T, int V, int Cin, int K, int Cout, int relu, const TikWindowing win, long long win_n0, const WinSeqs seqs,
                long long n_clips) {
  extern __shared__ __align__(16) float smem[];
  const int KC = K * Cin, VC = V * Cin;
  float* s_raw = smem;                                // [frames][V*Cin] raw input
  float* s_bn = s_raw + kStemFrames * VC;             // [frames][V*Cin] after data_bn
  float* s_a = s_bn + kStemFrames * VC;               // [frames][V][K*Cin] aggregated data_bn(x)
  float* s_agg = s_a + kStemFrames * V * KC;          // [K][V][V]
  const int tiles_t = (T + kStemFrames - 1) / kStemFrames;
  const int cg = Cout / 8;
  const int pairs = V * cg;                           // (node, channel group) pairs
  const int slots = kStemThreads / pairs > 0 ? kStemThreads / pairs : 1;
  const int pid = threadIdx.x % pairs, slot = threadIdx.x / pairs;
  const int wv = pid / cg, c0 = (pid - wv * cg) * 8;
  const bool worker = slot < slots && threadIdx.x < slots * pairs;

  // per-thread constants (registers)
  float wreg[KCR][8], breg[8], rreg[CINR][8];
#pragma unroll
  for (int kc = 0; kc < KCR; ++kc)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      wreg[kc][j] = (worker && kc < KC) ? __ldg(w + (size_t)(c0 + j) * KC + kc) : 0.f;
      if (kc < CINR) rreg[kc][j] = (worker && res_w != nullptr && kc < Cin) ? __ldg(res_w + ((size_t)wv * Cout + c0 + j) * Cin + kc) : 0.f;
    }
#pragma unroll
  for (int j = 0; j < 8; ++j) breg[j] = worker ? __ldg(bias + wv * Cout + c0 + j) : 0.f;
  for (int i = threadIdx.x; i < K * V * V; i += kStemThreads) s_agg[i] = __ldg(agg + i);
  const int T_res = (T - 1) / res_stride + 1;

  for (int64_t tile = blockIdx.x; tile < (int64_t)n_clips * tiles_t; tile += gridDim.x) {
    const int64_t n = tile / tiles_t;
    const int t0 = (int)(tile - n * tiles_t) * kStemFrames;
    const int nf = min(kStemFrames, T - t0);
    __syncthreads();                                  // previous tile's readers are done with the staging arrays
    // clip n is window win_n0 + n of the input; root-centred on 0.5*(kp[a]+kp[b]) (InferenceDataset, data_amass.py:232-235)
    const WinClip clip = win_clip(win, seqs, win_n0 + (long long)n);
    for (int i = threadIdx.x; i < nf * VC; i += kStemThreads) {
      const int vc = i % VC;
      const float* fr = x + win_frame(clip, t0 + i / VC) * VC;
      float raw = __ldg(fr + vc);
      if (win.root_a >= 0) {
        const int c = vc % Cin;
        raw -= 0.5f * (__ldg(fr + win.root_a * Cin + c) + __ldg(fr + win.root_b * Cin + c));
      }
      s_raw[i] = raw;
      s_bn[i] = fmaf(raw, __ldg(in_scale + vc), __ldg(in_shift + vc));
    }
    __syncthreads();
    // aggregated input: a[f][w][k*Cin+ci] = sum_v agg[k][v][w] * data_bn(x)[f][v][ci]
    for (int i = threadIdx.x; i < nf * V * KC; i += kStemThreads) {
      const int kc = i % KC, w2 = (i / KC) % V, f = i / (KC * V);
      const int k = kc / Cin, ci = kc - k * Cin;
      float acc = 0.f;
      for (int v = 0; v < V; ++v) acc = fmaf(s_agg[(k * V + v) * V + w2], s_bn[f * VC + v * Cin + ci], acc);
      s_a[i] = acc;
    }
    __syncthreads();
    if (worker) {
      OutT* orow = out + ((n * V + wv) * (int64_t)T + t0) * Cout + c0;
      OutT* rrow = res_out != nullptr ? res_out + ((n * V + wv) * (int64_t)T_res) * Cout + c0 : nullptr;
      for (int f = slot; f < nf; f += slots) {
        const float* a = s_a + (f * V + wv) * KC;
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = breg[j];
#pragma unroll
        for (int kc = 0; kc < KCR; ++kc) {
          if (kc < KC) {
            const float av = a[kc];
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = fmaf(wreg[kc][j], av, acc[j]);
          }
        }
        if (relu) {
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = fmaxf(acc[j], 0.f);
        }
        store8<OutT>(orow + (int64_t)f * Cout, acc);
        if (rrow != nullptr && ((t0 + f) % res_stride) == 0) {
          float r[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) r[j] = 0.f;
#pragma unroll
          for (int ci = 0; ci < CINR; ++ci) {
            if (ci < Cin) {
              const float xv = s_raw[f * VC + wv * Cin + ci];
#pragma unroll
              for (int j = 0; j < 8; ++j) r[j] = fmaf(rreg[ci][j], xv, r[j]);
            }
          }
          store8<OutT>(rrow + (int64_t)((t0 + f) / res_stride) * Cout, r);
        }
      }
    }
  }
}

template <class T>
static int launch_stem(const float* x, const float* sc, const float* sh, const float* agg, const float* w,
                       const float* bias, void* out, const float* res_w, void* res_out, int res_stride, int64_t N,
                       int Tn, int V, int Cin, int K, int Cout, int relu, const TikWindowing& win, int64_t win_n0, const WinSeqs& seqs,
                       cudaStream_t s) {
  const size_t KC = (size_t)K * Cin;
  size_t smem = sizeof(float) * (2 * (size_t)kStemFrames * V * Cin + (size_t)kStemFrames * V * KC + (size_t)K * V * V);
  TIK_CHECK_ARG(KC <= (size_t)kStemMaxKCReg, "stem: K*Cin=%zu > %d is not instantiated", KC, kStemMaxKCReg);
  TIK_CHECK_ARG(V * (Cout / 8) <= kStemThreads, "stem: V*Cout/8 = %d exceeds the CTA size", V * (Cout / 8));
  TIK_CHECK_ARG(smem <= 200 * 1024, "stem shared memory %zu too large", smem);
  static bool attr_set[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (!attr_set[dev & 63]) {   // per device (and per template instantiation: the static is per T)
    TIK_CUDA(cudaFuncSetAttribute(stem_gcn_kernel<T, 4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    TIK_CUDA(cudaFuncSetAttribute(stem_gcn_kernel<T, 16, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_set[dev & 63] = true;
  }
  int64_t tiles = N * ceil_div(Tn, kStemFrames);
  const unsigned gx = (unsigned)std::min<int64_t>(tiles, 148 * 3);       // persistent CTAs: weights loaded once
  if (KC <= 4 && Cin <= 4)
    stem_gcn_kernel<T, 4, 4><<<gx, kStemThreads, smem, s>>>(x, sc, sh, agg, w, bias, reinterpret_cast<T*>(out), res_w,
                                                          reinterpret_cast<T*>(res_out), res_stride, Tn, V, Cin, K, Cout, relu, win,
                                                          (long long)win_n0, seqs, (long long)N);
  else
    stem_gcn_kernel<T, 16, 8><<<gx, kStemThreads, smem, s>>>(x, sc, sh, agg, w, bias, reinterpret_cast<T*>(out), res_w,
                                                          reinterpret_cast<T*>(res_out), res_stride, Tn, V, Cin, K, Cout, relu, win,
                                                          (long long)win_n0, seqs, (long long)N);
  TIK_LAUNCH_CHECK();
  return TIK_OK;
}

}  // namespace tik

extern "C" int tik_stem_gcn(int dtype, const float* x, const float* in_scale, const float* in_shift, const float* agg,
                            const float* w, const float* bias, void* out, const float* res_w, void* res_out,
                            int res_stride, int64_t N, int T, int V, int Cin, int K, int Cout, int relu, void* stream) {
  return tik::stem_gcn_impl(dtype, x, in_scale, in_shift, agg, w, bias, out, res_w, res_out, res_stride, N, T, V, Cin, K, Cout,
                            relu, tik::plain_windowing(N, T), 0, tik::WinSeqs{}, (cudaStream_t)stream);
}

// The windowing comes from the caller's entry point, which has checked it (or built it: plain_windowing).
int tik::stem_gcn_impl(int dtype, const float* x, const float* in_scale, const float* in_shift, const float* agg,
                       const float* w, const float* bias, void* out, const float* res_w, void* res_out,
                       int res_stride, int64_t N, int T, int V, int Cin, int K, int Cout, int relu,
                       const TikWindowing& win, int64_t win_n0, const WinSeqs& seqs, cudaStream_t s) {
  using namespace tik;
  TIK_CHECK_ARG(x && in_scale && in_shift && agg && w && bias && out, "null pointer");
  TIK_CHECK_ARG(N >= 0 && T > 0 && V > 0 && V <= kStemMaxV && Cin > 0 && K > 0 && K <= 5 && K * Cin <= kStemMaxKC &&
                    Cout > 0 && Cout % 8 == 0,
                "stem: unsupported shape N=%lld T=%d V=%d Cin=%d K=%d Cout=%d", (long long)N, T, V, Cin, K, Cout);
  TIK_CHECK_ARG((res_w == nullptr) == (res_out == nullptr), "stem: res_w and res_out go together");
  TIK_CHECK_ARG(res_w == nullptr || res_stride >= 1, "stem: bad residual stride");
  if (N == 0) return TIK_OK;
  if (dtype == TIK_F32)
    return launch_stem<float>(x, in_scale, in_shift, agg, w, bias, out, res_w, res_out, res_stride, N, T, V, Cin, K, Cout, relu, win, win_n0, seqs, s);
  if (dtype == TIK_BF16)
    return launch_stem<__nv_bfloat16>(x, in_scale, in_shift, agg, w, bias, out, res_w, res_out, res_stride, N, T, V, Cin, K, Cout, relu, win, win_n0, seqs, s);
  set_error("bad dtype %d", dtype);
  return TIK_ERR_INVALID;
}
