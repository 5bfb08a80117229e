// Shared helpers for libtik.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/tik.h"

namespace tik {

void set_error(const char* fmt, ...);

#define TIK_CHECK_ARG(cond, ...)                 \
  do {                                           \
    if (!(cond)) {                               \
      ::tik::set_error(__VA_ARGS__);             \
      return TIK_ERR_INVALID;                    \
    }                                            \
  } while (0)

#define TIK_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      ::tik::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return TIK_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

// launch check without host synchronisation (SURVEY.md section 8b "Error conventions")
#define TIK_LAUNCH_CHECK()                                                               \
  do {                                                                                   \
    cudaError_t e_ = cudaPeekAtLastError();                                              \
    if (e_ != cudaSuccess) {                                                             \
      ::tik::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
      (void)cudaGetLastError();                                                          \
      return TIK_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Programmatic dependent launch: a kernel launched this way may start (and run its prologue: barrier init, tensor-
// memory allocation, constant operands to TMEM / shared memory) while its predecessor in the stream is still draining;
// it must execute pdl_wait() before it touches anything the predecessor wrote.  Captured as a programmatic edge in
// CUDA graphs.  TIK_NO_PDL=1 falls back to ordinary stream order.
bool pdl_enabled();
template <class... KArgs, class... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid, 1, 1);
  cfg.blockDim = dim3(block, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

// Per-launch options the plan sets before each tensor-core launch (thread-local; read when the launch fills its
// parameters).  rev: walk the tiles from the last to the first -- consecutive kernels alternate, so each starts on the
// part of its input the previous kernel wrote last, which is still in L2.
struct LaunchOpts { int rev; };
LaunchOpts& launch_opts();

// Every run reads its input through a TikWindowing.  A batch of N clips of T frames is window mode over its own N*T
// frames with stride T and no root: clip n, frame t reads frame n*T + t, which is always inside [0, N*T - 1], so the
// clamp never applies and the loaded address is that of the (N,T,V,C) layout.
static inline TikWindowing plain_windowing(int64_t N, int T) { return TikWindowing{N * T, 0, T, -1, -1}; }

// The packed-sequence tables of a ragged batch (TikSeqBatch), or n_seqs == 0 for one sequence spanning all
// win.frames frames.
struct WinSeqs { const int64_t* frame_start; const int64_t* window_start; long long n_seqs; };
static inline WinSeqs win_seqs(const TikSeqBatch& b) {
  return WinSeqs{b.frame_start_dev, b.window_start_dev, (long long)b.n_seqs};
}

// Host checks of a caller's windowing that need no plan.
static inline int check_windowing(const TikWindowing* win, const char* who) {
  TIK_CHECK_ARG(win != nullptr, "%s: null windowing", who);
  TIK_CHECK_ARG(win->frames > 0 && win->stride >= 1, "%s: windowing needs frames > 0 and stride >= 1", who);
  TIK_CHECK_ARG((win->root_a < 0) == (win->root_b < 0), "%s: root_a and root_b must both be set or both be negative", who);
  return TIK_OK;
}

// Host checks of a ragged-batch window call that need no plan (the tables themselves live on the device).
static inline int check_seq_windows(const TikWindowing* win, const TikSeqBatch* seqs, int64_t n_windows, const char* who) {
  TIK_CHECK_ARG(win != nullptr && seqs != nullptr, "%s: null windowing or sequence batch", who);
  TIK_CHECK_ARG(seqs->n_seqs >= 1, "%s: n_seqs = %lld, need >= 1", who, (long long)seqs->n_seqs);
  TIK_CHECK_ARG(seqs->frame_start_dev && seqs->window_start_dev, "%s: null frame_start or window_start table", who);
  TIK_CHECK_ARG(n_windows >= 0, "%s: n_windows = %lld < 0", who, (long long)n_windows);
  return check_windowing(win, who);
}

// One window's frames: frame t reads packed frame f0 + clamp(base + t, 0, last).
struct WinClip { long long base, f0, last; };

#ifdef __CUDACC__
// Looked up once per window (global window index g): the sequence is the last s with window_start[s] <= g (a binary
// search, ceil(log2 S) + 1 loads), so sequences without windows are skipped.  Indices read from the tables are
// clamped to the packed buffer: a malformed table gives wrong frames, never a read outside [0, win.frames).
// Without tables: base = g*stride + offset, f0 = 0, last = frames - 1 (one sequence, or a plain batch of clips).
__device__ __forceinline__ WinClip win_clip(const TikWindowing& win, const WinSeqs& sq, long long g) {
  if (sq.n_seqs <= 0) return WinClip{g * win.stride + win.offset, 0, win.frames - 1};
  long long lo = 0, hi = sq.n_seqs - 1;
  while (lo < hi) {
    const long long mid = (lo + hi + 1) >> 1;
    if (__ldg(sq.window_start + mid) <= g) lo = mid; else hi = mid - 1;
  }
  const long long n = g - (long long)__ldg(sq.window_start + lo), frames = win.frames;
  const long long f0 = min(max((long long)__ldg(sq.frame_start + lo), 0ll), frames - 1);
  const long long f1 = min(max((long long)__ldg(sq.frame_start + lo + 1), f0 + 1), frames);
  return WinClip{n * win.stride + win.offset, f0, f1 - f0 - 1};
}
// Packed frame of frame t of the window: the edge padding of sample_window (mmskeleton/datasets/data_amass.py:18-42)
// inside the window's own sequence.
__device__ __forceinline__ long long win_frame(const WinClip& c, long long t) {
  const long long fi = c.base + t;
  return c.f0 + (fi < 0 ? 0 : (fi >= c.last ? c.last : fi));
}
#endif

// fp32 implicit-GEMM arguments (stgcn_simt.cu rowgemm_f32_kernel, rowgemm_tf32.cu): TikRowGemm with the K offsets resolved
struct F32Slab { const float* a; int c, t_in, t_mul, t_off, koff; };
struct F32Args {
  F32Slab slabs[TIK_MAX_SLABS];
  int n_slabs;
  const float* w; int ktot;
  const float* bias; int bias_per_node;
  int64_t rows; int v, t_out, c_out, c_out_valid;
  int act; float slope;
  int res_kind; const void* res; const float* res_w; int res_cin, res_t_mul, res_t_in;
  float* out; int out_layout;
  // n / t_out and n / v for n < 2^31 as (n * magic) >> shift (rowgemm_tf32.cu: ~100 integer divisions per tile row otherwise)
  unsigned long long div_t_magic, div_v_magic; int div_t_shift, div_v_shift;
  // optional: the weights already split into their TF32 parts (tf32_split_weights; the plan does it once per weight
  // version in its workspace), both (c_out, ktot) like w.  nullptr: the kernel splits W on the way, like the activations.
  const float* w_big; const float* w_small;
};
bool rowgemm_tf32_supported(const F32Args& a);
int rowgemm_tf32_launch(const F32Args& a, cudaStream_t s);

// internal entry points shared between translation units
int rowgemm_f32(const TikRowGemm* d, cudaStream_t s);
int rowgemm_f32_presplit(const TikRowGemm* d, const float* w_big, const float* w_small, cudaStream_t s);
int tf32_split_weights(const float* w, float* big, float* small, int64_t n, cudaStream_t s);
int rowgemm_bf16(const TikRowGemm* d, cudaStream_t s);
int launch_batch_rodrigues(const float* aa, float* R9, int64_t M, cudaStream_t s);
int stem_gcn_impl(int dtype, const float* x, const float* in_scale, const float* in_shift, const float* agg,
                  const float* w, const float* bias, void* out, const float* res_w, void* res_out,
                  int res_stride, int64_t N, int T, int V, int Cin, int K, int Cout, int relu,
                  const TikWindowing& win, int64_t win_n0, const WinSeqs& seqs, cudaStream_t s);

}  // namespace tik
