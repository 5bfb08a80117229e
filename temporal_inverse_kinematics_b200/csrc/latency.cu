// Latency plan: the WHOLE PoseRegressor forward (pose_trainer.py:94-133 = StgGcn18 backbone,
// st_gcn_aaai18.py:113-133, + Linear / LeakyReLU / Linear head) for a handful of clips as ONE persistent
// cooperative kernel.
//
// The throughput plan (plan.cu) is 19-25 dependent launches of kernels built to stream millions of rows; for one
// 64-frame window (1088 rows) each of them is a few microseconds of work behind a launch, a prologue (barrier
// init, TMEM allocation, weights to tensor memory) and a drain: 370-430 us per window, launch-bound
// (BASELINE.json configs[4], profiles/r1_notes.md).  Here every layer is a *phase* of one kernel: 148 CTAs x 256
// threads stay resident, split the phase's output tiles between them, and meet at a grid-wide barrier
// (cooperative launch => co-residency is guaranteed).  Activations ping-pong through a few hundred KB of
// workspace that never leaves L2; the fp32 BN-folded weights (12.7 MB) are L2-resident across calls.
//
// Arithmetic is fp32 FMA on CUDA cores with the SAME packed fp32 algebra as the 1e-4 parity path
// (engine.PackedNet("fp32"), SURVEY.md Appendix B): at 0.5 GFLOP per window the tensor pipe buys nothing, and the
// latency path inherits fp32 accuracy.  Phases (K = 1 adjacency partition, the IK model):
//   stem      data_bn + block-0 graph conv + BN + ReLU, and block-0's residual branch
//   gemm      implicit GEMM over K-slabs (temporal taps, residual 1x1 conv), optional on-the-fly adjacency
//             aggregation of the A operand (the einsum of gconv_origin.py:63 moved in front of the 1x1 conv),
//             bias (per node), identity residual, ReLU
//   gemv      the head's two Linear layers (<= 32 rows): one warp per output column, lanes split K
#include <cooperative_groups.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "tik_common.cuh"

namespace cg = cooperative_groups;

namespace tik {

constexpr int kLatThreads = 256;
constexpr int kLatKC = 32;            // K chunk of the tiled GEMM
constexpr int kLatCB = 32;            // output columns per tile
constexpr int kLatMaxV = 32;
constexpr int kLatMaxPhases = 3 * TIK_MAX_BLOCKS + 4;

struct LatSlab { const float* a; int c, t_in, t_mul, t_off, koff; };

// non-zero adjacency entries per destination node, built on the host (plan creation)
struct alignas(16) LatNbr {
  float w[kLatMaxV][kLatMaxV];
  uint8_t v[kLatMaxV][kLatMaxV];
  int deg[kLatMaxV];
};

struct alignas(16) LatPhase {
  int kind;                     // 0 stem, 1 gemm, 2 gemv
  // ---- gemm / gemv
  LatSlab slabs[TIK_MAX_SLABS];
  int n_slabs;
  int nbr;                      // graph convolution: index of the block's neighbour table (adjacency A^), else -1:
                                //   H[(n,w,t)] = sum_v A^[v][w] Z[(n,v,t)]
  const float* w; int ktot;
  const float* bias; int bias_per_node;
  int v, t_out, c_out, c_out_valid;      // rows = N * v * t_out  (head: v = 1, t_out = T')
  int act; float slope;
  const float* res;             // identity residual, node-major (rows, c_out), or null
  float* out; int out_layout;   // out == nullptr: the caller's poses pointer
  int rb;                       // tile rows (16 or 32)
  // ---- stem
  const float *in_scale, *in_shift, *agg0, *w0, *b0, *res_w;
  float *h0, *r0;
  int T, V, Cin, Cout, res_stride;
};

struct LatParams {
  const LatPhase* phases;
  const LatNbr* nbr;            // one neighbour table per block
  int n_phases, n_nbr;
  const float* x;               // (frames,V,Cin) input read through win: clip n is window n
  float* poses;
  int64_t N;
  TikWindowing win;
  WinSeqs seqs;                 // ragged batch tables (n_seqs == 0: none)
  unsigned long long* times;    // debug: [CTA][2 * phases] %globaltimer at the start and at the end of every phase's work (or null)
};

// ------------------------------------------------------------------------------------------------ stem phase
// One CTA per frame: the frame's V x Cin keypoints go to shared memory (root-centred, data_bn applied), V x Cin
// threads aggregate them over the adjacency, then every thread produces output channels from shared memory.  All
// global loads of a frame are issued at once (the first version walked the adjacency per thread with a dependent
// load per neighbour).
struct LatStemSmem { float raw[kLatMaxV * 8], bn[kLatMaxV * 8], a[kLatMaxV * 8]; };

__device__ void lat_stem(const LatPhase& ph, const LatParams& p, LatStemSmem& sm) {
  const int V = ph.V, Cin = ph.Cin, Cout = ph.Cout, T = ph.T;
  const int VC = V * Cin;
  const int T_res = (T - 1) / ph.res_stride + 1;
  const int tid = threadIdx.x;
  const int64_t frames = p.N * (int64_t)T;
  for (int64_t f = blockIdx.x; f < frames; f += gridDim.x) {
    const int64_t n = f / T;
    const int t = (int)(f - n * T);
    const float* fr = p.x + win_frame(win_clip(p.win, p.seqs, n), t) * (int64_t)VC;
    __syncthreads();                                   // the previous frame's readers are done
    if (tid < VC) {
      float raw = __ldg(fr + tid);
      if (p.win.root_a >= 0) {
        const int ci = tid % Cin;
        raw -= 0.5f * (__ldg(fr + p.win.root_a * Cin + ci) + __ldg(fr + p.win.root_b * Cin + ci));
      }
      sm.raw[tid] = raw;
      sm.bn[tid] = fmaf(raw, __ldg(ph.in_scale + tid), __ldg(ph.in_shift + tid));
    }
    __syncthreads();
    if (tid < VC) {
      const int w = tid / Cin, ci = tid - w * Cin;
      float acc = 0.f;
      for (int v = 0; v < V; ++v) acc = fmaf(__ldg(ph.agg0 + v * V + w), sm.bn[v * Cin + ci], acc);
      sm.a[tid] = acc;
    }
    __syncthreads();
    for (int o = tid; o < V * Cout; o += kLatThreads) {
      const int w = o / Cout, c = o - w * Cout;
      float acc = __ldg(ph.b0 + o);
      for (int ci = 0; ci < Cin; ++ci) acc = fmaf(__ldg(ph.w0 + (size_t)c * Cin + ci), sm.a[w * Cin + ci], acc);
      ph.h0[((n * V + w) * (int64_t)T + t) * Cout + c] = fmaxf(acc, 0.f);
      if (ph.r0 != nullptr && (t % ph.res_stride) == 0) {
        float r = 0.f;
        for (int ci = 0; ci < Cin; ++ci) r = fmaf(__ldg(ph.res_w + (size_t)o * Cin + ci), sm.raw[w * Cin + ci], r);
        ph.r0[((n * V + w) * (int64_t)T_res + t / ph.res_stride) * Cout + c] = r;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ gemm phase
constexpr int kLatKCH = 128;          // K chunk staged per pipeline step (four float4 per thread and operand): one
constexpr int kLatKV = kLatKCH / 32;  // chunk of FMAs covers the L2 latency of the next chunk's loads
constexpr int kLatPitch = kLatKCH + 4;   // operand row pitch (floats): 16-byte aligned rows, 4-bank skew per row

struct LatSmem {
  float ab[(32 + kLatCB) * kLatPitch];  // A tile [RB][pitch] then B tile [32][pitch], k contiguous; reused for the
                                        // cross-warp reduction (8 warps x RB x 32 partial sums)
  float Cs[32][kLatCB + 1];             // reduced tile (the Z tile of the graph-convolution epilogue)
};

// Implicit GEMM tile of RB rows x 32 columns by 256 threads.  Shared-memory bandwidth, not FMA rate, bounds a small
// tile (the first version read 1.5 operands per FMA: 3 us per 128-wide K chunk), so the K range of a chunk is SPLIT
// OVER THE 8 WARPS: every warp owns whole groups of 4 consecutive k, keeps a full RB x 32 partial tile in registers
// ((RB/4) x 4 per lane, rows ly + 4i, columns lx + 8j: conflict-free float4 operand reads along k, 8 LDS.128 per 64
// FMAs), and the warps' partial tiles meet once per tile in shared memory (fixed summation order: deterministic).
// The K loop is software pipelined: the global loads of chunk i+1 are issued before the FMAs of chunk i.
//
// FRAME = false (temporal convolution, residual slabs): rows are consecutive node-major rows (nv, t); a slab's source
//   row is (nv, t * t_mul + t_off), zero outside [0, t_in).
// FRAME = true (graph convolution): a tile is ONE frame (n, t) = the V rows (n, v, t); the tile computes
//   Z = X . Wg^T for its V nodes and the epilogue aggregates over the adjacency, H[w] = sum_v A^[v,w] Z[v] + b[w]
//   (the reference's own order, gconv_origin.py:59-63), through shared memory -- ONE small aggregation per tile.
template <int RB, bool FRAME>
__device__ void lat_gemm(const LatPhase& ph, const LatParams& p, LatSmem& sm, const LatNbr* nbr) {
  constexpr int MI = RB / 4;                          // rows per lane
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int ly = lane >> 3, lx = lane & 7;
  const int V = ph.v;
  const int64_t rows = p.N * V * (int64_t)ph.t_out;
  const int64_t row_tiles = FRAME ? p.N * (int64_t)ph.t_out : (rows + RB - 1) / RB;
  const int col_tiles = (ph.c_out + kLatCB - 1) / kLatCB;
  float* As = sm.ab;
  float* Bs = sm.ab + RB * kLatPitch;
  // loaders: tile row (or column) lr = tid / 8, channels k0 + 32 h + lk .. +3
  const int lr = tid >> 3, lk = (tid & 7) * 4;
  float* out = ph.out != nullptr ? ph.out : p.poses;
  int n_chunks = 0;
  for (int s = 0; s < ph.n_slabs; ++s) n_chunks += (ph.slabs[s].c + kLatKCH - 1) / kLatKCH;
  for (int64_t item = blockIdx.x; item < row_tiles * col_tiles; item += gridDim.x) {
    const int64_t rt = item / col_tiles;
    const int col0 = (int)(item - rt * col_tiles) * kLatCB;
    float acc[MI][4];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    // the loader's row
    bool row_ok;
    int64_t g_nv;
    int g_t;
    if (FRAME) {
      const int64_t n = rt / ph.t_out;
      g_t = (int)(rt - n * ph.t_out);
      row_ok = lr < V;
      g_nv = n * V + (row_ok ? lr : 0);
    } else {
      const int64_t grow = rt * RB + lr;
      row_ok = lr < RB && grow < rows;
      g_nv = row_ok ? grow / ph.t_out : 0;
      g_t = row_ok ? (int)(grow % ph.t_out) : 0;
    }
    const bool col_ok = (col0 + lr) < ph.c_out;
    const float* wbase = ph.w + (int64_t)(col0 + lr) * ph.ktot;

    float4 a4[kLatKV], b4[kLatKV];
    int cs = 0, ck0 = 0;                              // slab / k0 of the chunk held in the registers
    auto issue = [&](int s, int k0) {                 // global loads of chunk (s, k0) -> registers, nothing consumed here
      const LatSlab sl = ph.slabs[s];
      const int ts = g_t * sl.t_mul + sl.t_off;
      const bool a_ok = row_ok && ts >= 0 && ts < sl.t_in;
      // activations were written earlier in THIS kernel by other SMs: ordinary loads (ordered by the grid barrier),
      // never the non-coherent read-only path; weights are constants (__ldg)
      const float* arow = sl.a + (g_nv * sl.t_in + (a_ok ? ts : 0)) * (int64_t)sl.c;
#pragma unroll
      for (int h = 0; h < kLatKV; ++h) {
        const int k = k0 + 32 * h + lk;               // channel counts are multiples of 4
        a4[h] = (a_ok && k < sl.c) ? *reinterpret_cast<const float4*>(arow + k) : make_float4(0.f, 0.f, 0.f, 0.f);
        b4[h] = (col_ok && k < sl.c) ? __ldg(reinterpret_cast<const float4*>(wbase + sl.koff + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    issue(0, 0);
    for (int ch = 0; ch < n_chunks; ++ch) {
      const int klen = min(kLatKCH, ph.slabs[cs].c - ck0);       // multiple of 4
      __syncthreads();
#pragma unroll
      for (int h = 0; h < kLatKV; ++h) {
        if (lr < RB) *reinterpret_cast<float4*>(As + lr * kLatPitch + 32 * h + lk) = a4[h];
        *reinterpret_cast<float4*>(Bs + lr * kLatPitch + 32 * h + lk) = b4[h];
      }
      __syncthreads();
      if (ch + 1 < n_chunks) {
        ck0 += kLatKCH;
        if (ck0 >= ph.slabs[cs].c) { ++cs; ck0 = 0; }
        issue(cs, ck0);
      }
      for (int kk = 4 * warp; kk < klen; kk += 32) {   // this warp's groups of 4 consecutive k
        float4 av[MI], bv[4];
#pragma unroll
        for (int i = 0; i < MI; ++i) av[i] = *reinterpret_cast<const float4*>(As + (ly + 4 * i) * kLatPitch + kk);
#pragma unroll
        for (int j = 0; j < 4; ++j) bv[j] = *reinterpret_cast<const float4*>(Bs + (lx + 8 * j) * kLatPitch + kk);
#pragma unroll
        for (int i = 0; i < MI; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j)
            acc[i][j] = fmaf(av[i].x, bv[j].x, fmaf(av[i].y, bv[j].y, fmaf(av[i].z, bv[j].z, fmaf(av[i].w, bv[j].w, acc[i][j]))));
      }
    }
    // ---- the 8 warps' partial tiles meet in shared memory (the operand tiles are dead), summed in warp order
    __syncthreads();
    float* red = sm.ab;                                // [8][RB][32 + 1]
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) red[(warp * RB + ly + 4 * i) * (kLatCB + 1) + lx + 8 * j] = acc[i][j];
    __syncthreads();
    for (int o = tid; o < RB * kLatCB; o += kLatThreads) {
      const int r = o / kLatCB, c = o - r * kLatCB;
      float v = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) v += red[(w * RB + r) * (kLatCB + 1) + c];
      sm.Cs[r][c] = v;
    }
    __syncthreads();
    if (FRAME) {
      // ---- adjacency aggregation of the Z tile + per-node bias + ReLU, coalesced row stores
      const int64_t n = rt / ph.t_out;
      for (int o = tid; o < V * kLatCB; o += kLatThreads) {
        const int w = o / kLatCB, cc = o - w * kLatCB;
        const int c = col0 + cc;
        if (c >= ph.c_out) continue;
        float val = __ldg(ph.bias + w * ph.c_out + c);
        const int d = nbr->deg[w];
        for (int j = 0; j < d; ++j) val = fmaf(nbr->w[w][j], sm.Cs[nbr->v[w][j]][cc], val);
        if (ph.act == TIK_ACT_RELU) val = fmaxf(val, 0.f);
        out[((n * V + w) * (int64_t)ph.t_out + g_t) * ph.c_out + c] = val;
      }
    } else {
      // ---- epilogue: bias (per node), identity residual, activation, layout
      for (int o = tid; o < RB * kLatCB; o += kLatThreads) {
        const int rr = o / kLatCB, cc = o - rr * kLatCB;
        const int64_t r = rt * RB + rr;
        const int c = col0 + cc;
        if (r >= rows || c >= ph.c_out) continue;
        const int64_t nv = r / ph.t_out;
        const int t = (int)(r % ph.t_out);
        const int node = (int)(nv % V);
        const int64_t n = nv / V;
        float val = sm.Cs[rr][cc] + __ldg(ph.bias + (ph.bias_per_node ? node * ph.c_out : 0) + c);
        if (ph.res != nullptr) val += ph.res[r * ph.c_out + c];
        if (ph.act == TIK_ACT_RELU) val = fmaxf(val, 0.f);
        else if (ph.act == TIK_ACT_LEAKY) val = val > 0.f ? val : val * ph.slope;
        if (ph.out_layout == TIK_OUT_NODE_MAJOR) out[r * ph.c_out + c] = val;
        else if (ph.out_layout == TIK_OUT_TIME_MAJOR) out[((n * ph.t_out + t) * V + node) * (int64_t)ph.c_out + c] = val;
        else if (c < ph.c_out_valid) out[r * ph.c_out_valid + c] = val;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ gemv phase
// Head layers: rows = N * T' <= 32.  A CTA owns a few output columns; its 8 warps are (column, K split) pairs, the
// lanes stride K in float4 steps (coalesced weight reads; the few A rows come from L1/L2) with 4 K steps of loads in
// flight and 4 rows of accumulators at a time; warp-shuffle reduction, then the K splits meet in shared memory.
__device__ void lat_gemv(const LatPhase& ph, const LatParams& p, float* red /* [8 warps][4 rows] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int kWarps = kLatThreads / 32;
  const int rows = (int)(p.N * ph.t_out);
  const int K = ph.ktot;
  const float* __restrict__ A = ph.slabs[0].a;
  float* out = ph.out != nullptr ? ph.out : p.poses;
  const int ld_out = ph.out_layout == TIK_OUT_ROWS_F32 ? ph.c_out_valid : ph.c_out;
  int cols_per_cta = (ph.c_out_valid + gridDim.x - 1) / gridDim.x;
  int ksplit = 1;
  while (ksplit * 2 * cols_per_cta <= kWarps) ksplit *= 2;                   // 1, 2, 4 or 8 warps per column
  cols_per_cta = kWarps / ksplit;
  const int my_col = warp / ksplit, my_split = warp - my_col * ksplit;
  const int kspan = ((K / 4 + ksplit - 1) / ksplit) * 4;                        // K range of one split (multiple of 4)
  const int k_lo = my_split * kspan, k_hi = min(K, k_lo + kspan);
  for (int c0 = blockIdx.x * cols_per_cta; c0 < ph.c_out_valid; c0 += gridDim.x * cols_per_cta) {
    const int c = c0 + my_col;
    const bool c_ok = c < ph.c_out_valid;
    const float* __restrict__ wrow = ph.w + (size_t)(c_ok ? c : 0) * K;
    for (int r0 = 0; r0 < rows; r0 += 4) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      if (c_ok) {
        for (int kb = k_lo + lane * 4; kb < k_hi; kb += 4 * 128) {
          float4 w4[4], a4[4][4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int k = kb + u * 128;
            const bool ok = k < k_hi;
            w4[u] = ok ? __ldg(reinterpret_cast<const float4*>(wrow + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int r = 0; r < 4; ++r)   // written by the previous phase: ordinary loads, not __ldg
              a4[r][u] = ok ? *reinterpret_cast<const float4*>(A + (size_t)(r0 + r) * K + k) : make_float4(0.f, 0.f, 0.f, 0.f);   // buffers hold a multiple of 4 rows
          }
#pragma unroll
          for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int r = 0; r < 4; ++r)
              acc[r] = fmaf(a4[r][u].x, w4[u].x, fmaf(a4[r][u].y, w4[u].y, fmaf(a4[r][u].z, w4[u].z, fmaf(a4[r][u].w, w4[u].w, acc[r]))));
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int off = 16; off > 0; off >>= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], off);
      }
      __syncthreads();
      if (lane < 4) red[warp * 4 + lane] = lane == 0 ? acc[0] : lane == 1 ? acc[1] : lane == 2 ? acc[2] : acc[3];
      __syncthreads();
      if (my_split == 0 && lane < 4 && c_ok && r0 + lane < rows) {
        float val = __ldg(ph.bias + c);
        for (int q = 0; q < ksplit; ++q) val += red[(warp + q) * 4 + lane];     // fixed order: deterministic
        if (ph.act == TIK_ACT_RELU) val = fmaxf(val, 0.f);
        else if (ph.act == TIK_ACT_LEAKY) val = val > 0.f ? val : val * ph.slope;
        out[(size_t)(r0 + lane) * ld_out + c] = val;
      }
    }
  }
}

static_assert(sizeof(LatPhase) % 16 == 0 && sizeof(LatNbr) % 16 == 0, "descriptors are staged as uint4");

// dynamic shared memory: [LatSmem][LatStemSmem][phases][neighbour tables]
__host__ __device__ constexpr size_t lat_smem_bytes(int n_phases, int n_nbr) {
  return sizeof(LatSmem) + sizeof(LatStemSmem) + (size_t)n_phases * sizeof(LatPhase) + (size_t)n_nbr * sizeof(LatNbr);
}

__global__ void __launch_bounds__(kLatThreads) stgcn_latency_kernel(const __grid_constant__ LatParams p) {
  extern __shared__ __align__(16) uint8_t lat_smem[];
  LatSmem& sm = *reinterpret_cast<LatSmem*>(lat_smem);
  LatStemSmem& sm_stem = *reinterpret_cast<LatStemSmem*>(lat_smem + sizeof(LatSmem));
  LatPhase* s_ph = reinterpret_cast<LatPhase*>(lat_smem + sizeof(LatSmem) + sizeof(LatStemSmem));
  LatNbr* s_nbr = reinterpret_cast<LatNbr*>(s_ph + p.n_phases);
  cg::grid_group grid = cg::this_grid();
  // every phase descriptor and neighbour table -> shared memory, once: no descriptor fetch on a phase's critical path
  {
    const int n4 = (int)((p.n_phases * sizeof(LatPhase)) / 16), m4 = (int)((p.n_nbr * sizeof(LatNbr)) / 16);
    for (int i = threadIdx.x; i < n4; i += kLatThreads) reinterpret_cast<uint4*>(s_ph)[i] = __ldg(reinterpret_cast<const uint4*>(p.phases) + i);
    for (int i = threadIdx.x; i < m4; i += kLatThreads) reinterpret_cast<uint4*>(s_nbr)[i] = __ldg(reinterpret_cast<const uint4*>(p.nbr) + i);
    __syncthreads();
  }
  for (int i = 0; i < p.n_phases; ++i) {
    if (p.times != nullptr && threadIdx.x == 0) {
      unsigned long long tnow;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(tnow));
      p.times[(size_t)blockIdx.x * 2 * p.n_phases + 2 * i] = tnow;
    }
    const LatPhase& ph = s_ph[i];
    if (ph.kind == 0) lat_stem(ph, p, sm_stem);
    else if (ph.kind == 2) lat_gemv(ph, p, sm.ab);
    else if (ph.nbr >= 0) lat_gemm<32, true>(ph, p, sm, s_nbr + ph.nbr);
    else lat_gemm<16, false>(ph, p, sm, nullptr);
    if (p.times != nullptr) {
      __syncthreads();
      if (threadIdx.x == 0) {
        unsigned long long tnow;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(tnow));
        p.times[(size_t)blockIdx.x * 2 * p.n_phases + 2 * i + 1] = tnow;
      }
    }
    if (i + 1 < p.n_phases) grid.sync();
  }
}

}  // namespace tik

// ------------------------------------------------------------------------------------------------ host side
struct TikLatencyPlan {
  TikNet net;
  int64_t n_max;
  int T, T_out;
  int n_phases;
  tik::LatPhase* phases_dev;
  const tik::LatNbr* nbr_dev;
  int n_nbr;
  size_t smem;
  int grid;
  unsigned long long* times_dev;   // debug (tik_debug_latency_times)
};

namespace tik {

static int lat_out_frames(int t, int stride) { return (t - 1) / stride + 1; }
static int64_t lat_align(int64_t v) { return (v + 255) / 256 * 256; }

struct LatLayout { int64_t off_x[2], off_h, off_r0, off_feat, off_z, off_phases, off_nbr, total; };

static int lat_check(const TikNet* net, int64_t n_max, int T) {
  TIK_CHECK_ARG(net && n_max >= 1 && T >= 1, "latency plan: bad arguments");
  TIK_CHECK_ARG(net->K == 1, "latency plan: K=%d adjacency partitions (only the uniform strategy, K=1, is built)", net->K);
  TIK_CHECK_ARG(net->V >= 1 && net->V <= kLatMaxV && net->c_in >= 1 && net->c_in <= 8, "latency plan: V=%d c_in=%d unsupported", net->V, net->c_in);
  TIK_CHECK_ARG(net->n_blocks >= 2 && net->n_blocks <= TIK_MAX_BLOCKS, "latency plan: n_blocks=%d", net->n_blocks);
  TIK_CHECK_ARG(net->head_hidden > 0 && net->head_out > 0, "latency plan needs the regressor head");
  TIK_CHECK_ARG(net->head_hidden % 4 == 0, "latency plan: head hidden width must be a multiple of 4");
  for (int i = 0; i < net->n_blocks; ++i) {
    const TikBlock& b = net->blocks[i];
    TIK_CHECK_ARG(b.c_out % 8 == 0 && b.kt >= 1 && (b.kt % 2) == 1 && b.kt + 1 <= TIK_MAX_SLABS && b.stride >= 1, "latency plan: block %d shape", i);
    TIK_CHECK_ARG(!b.res_as_slab, "latency plan takes the fp32 packing (no identity K-slabs)");
    TIK_CHECK_ARG(i > 0 || b.res_kind == TIK_RES_NONE || b.res_kind == TIK_RES_STEM, "latency plan: block 0 residual");
  }
  int t = T;
  for (int i = 0; i < net->n_blocks; ++i) t = lat_out_frames(t, net->blocks[i].stride);
  TIK_CHECK_ARG(n_max * t <= 32, "latency plan: N*T' = %lld rows exceed the head's 32-row limit", (long long)(n_max * t));
  return TIK_OK;
}

static void lat_layout(const TikNet* net, int64_t n, int T, LatLayout* L, int* t_final) {
  const int64_t V = net->V;
  int t = T;
  int64_t x = 0, h = 0, r0 = 0;
  for (int i = 0; i < net->n_blocks; ++i) {
    const TikBlock& b = net->blocks[i];
    h = std::max<int64_t>(h, V * t * b.c_out);
    t = lat_out_frames(t, b.stride);
    if (i == 0 && b.res_kind == TIK_RES_STEM) r0 = V * t * b.c_out;
    x = std::max<int64_t>(x, V * t * b.c_out);
  }
  *t_final = t;
  int64_t off = 0;
  L->off_x[0] = off; off = lat_align(off + x * n * 4);
  L->off_x[1] = off; off = lat_align(off + x * n * 4);
  L->off_h = off; off = lat_align(off + h * n * 4);
  L->off_r0 = off; off = lat_align(off + r0 * n * 4);
  const int64_t head_rows = (n * t + 3) / 4 * 4;             // the head kernels read rows in groups of 4
  L->off_feat = off; off = lat_align(off + V * net->blocks[net->n_blocks - 1].c_out * head_rows * 4);
  L->off_z = off; off = lat_align(off + (int64_t)net->head_hidden * head_rows * 4);
  L->off_phases = off; off = lat_align(off + (int64_t)sizeof(LatPhase) * kLatMaxPhases);
  L->off_nbr = off; off = lat_align(off + (int64_t)sizeof(LatNbr) * net->n_blocks);
  L->total = off;
}

}  // namespace tik

extern "C" {

int tik_stgcn_latency_workspace_bytes(const TikNet* net, int64_t n_max, int T, int64_t* bytes) {
  using namespace tik;
  int rc = lat_check(net, n_max, T);
  if (rc != TIK_OK) return rc;
  TIK_CHECK_ARG(bytes != nullptr, "null pointer");
  LatLayout L;
  int tf;
  lat_layout(net, n_max, T, &L, &tf);
  *bytes = L.total;
  return TIK_OK;
}

int tik_stgcn_latency_create(const TikNet* net, int64_t n_max, int T, void* workspace, int64_t ws_bytes, TikLatencyPlan** out) {
  using namespace tik;
  int rc = lat_check(net, n_max, T);
  if (rc != TIK_OK) return rc;
  TIK_CHECK_ARG(out != nullptr, "null pointer");
  LatLayout L;
  int tf;
  lat_layout(net, n_max, T, &L, &tf);
  if (!workspace || ws_bytes < L.total) {
    set_error("latency plan: workspace of %lld bytes is smaller than the %lld bytes needed", (long long)ws_bytes, (long long)L.total);
    return TIK_ERR_WORKSPACE;
  }
  TIK_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "latency plan: workspace must be 256-byte aligned");
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  float* xbuf[2] = {reinterpret_cast<float*>(ws + L.off_x[0]), reinterpret_cast<float*>(ws + L.off_x[1])};
  float* hbuf = reinterpret_cast<float*>(ws + L.off_h);
  float* r0buf = reinterpret_cast<float*>(ws + L.off_r0);
  float* feat = reinterpret_cast<float*>(ws + L.off_feat);
  float* zbuf = reinterpret_cast<float*>(ws + L.off_z);
  std::vector<LatPhase> ph;
  const int V = net->V;
  int t = T, cur = 0;
  // neighbour lists of every block's A * edge_importance
  std::vector<LatNbr> nbr(net->n_blocks);
  {
    std::vector<float> a((size_t)V * V);
    for (int i = 0; i < net->n_blocks; ++i) {
      TIK_CUDA(cudaMemcpy(a.data(), net->blocks[i].agg_dev, a.size() * sizeof(float), cudaMemcpyDeviceToHost));
      memset(&nbr[i], 0, sizeof(LatNbr));
      for (int w = 0; w < V; ++w) {
        int d = 0;
        for (int v = 0; v < V; ++v)
          if (a[(size_t)v * V + w] != 0.f) { nbr[i].w[w][d] = a[(size_t)v * V + w]; nbr[i].v[w][d] = (uint8_t)v; ++d; }
        nbr[i].deg[w] = d;
      }
    }
    TIK_CUDA(cudaMemcpy(ws + L.off_nbr, nbr.data(), nbr.size() * sizeof(LatNbr), cudaMemcpyHostToDevice));
    TIK_CUDA(cudaMemset(ws + L.off_feat, 0, (size_t)(L.off_phases - L.off_feat)));      // padded head rows read as zeros
  }
  const LatNbr* nbr_dev = reinterpret_cast<const LatNbr*>(ws + L.off_nbr);
  auto rb_for = [&](int64_t rows_per_clip, int c_out) {
    // 16-row tiles while 32-row tiles would leave most of the 148 CTAs without work (one clip)
    const int64_t tiles32 = ((rows_per_clip + 31) / 32) * ((c_out + kLatCB - 1) / kLatCB);
    return tiles32 >= 148 ? 32 : 16;
  };
  for (int i = 0; i < net->n_blocks; ++i) {
    const TikBlock& b = net->blocks[i];
    const int pad = (b.kt - 1) / 2;
    const int t_o = lat_out_frames(t, b.stride);
    const bool last = i == net->n_blocks - 1;
    LatPhase g;
    if (i == 0) {
      memset(&g, 0, sizeof(g));
      g.kind = 0; g.nbr = -1;
      g.in_scale = net->in_scale_dev; g.in_shift = net->in_shift_dev; g.agg0 = b.agg_dev;
      g.w0 = reinterpret_cast<const float*>(b.w_gcn_dev); g.b0 = b.b_gcn_dev;
      g.res_w = b.res_kind == TIK_RES_STEM ? b.w_res_stem_dev : nullptr;
      g.h0 = hbuf; g.r0 = b.res_kind == TIK_RES_STEM ? r0buf : nullptr;
      g.T = t; g.V = V; g.Cin = b.c_in; g.Cout = b.c_out; g.res_stride = b.stride;
      ph.push_back(g);
    } else {
      memset(&g, 0, sizeof(g));
      g.kind = 1;
      g.n_slabs = 1;
      g.slabs[0] = {xbuf[cur], b.c_in, t, 1, 0, 0};
      g.nbr = i;
      g.w = reinterpret_cast<const float*>(b.w_gcn_dev); g.ktot = b.c_in;
      g.bias = b.b_gcn_dev; g.bias_per_node = 1;
      g.v = V; g.t_out = t; g.c_out = b.c_out; g.c_out_valid = b.c_out;
      g.act = TIK_ACT_RELU; g.out = hbuf; g.out_layout = TIK_OUT_NODE_MAJOR;
      g.rb = rb_for((int64_t)V * t, b.c_out);
      ph.push_back(g);
    }
    LatPhase c;
    memset(&c, 0, sizeof(c));
    c.kind = 1;
    c.nbr = -1;
    int ns = 0, koff = 0;
    for (int dt = 0; dt < b.kt; ++dt) { c.slabs[ns++] = {hbuf, b.c_out, t, b.stride, dt - pad, koff}; koff += b.c_out; }
    if (b.res_kind == TIK_RES_CONV) { c.slabs[ns++] = {xbuf[cur], b.c_in, t, b.stride, 0, koff}; koff += b.c_in; }
    c.n_slabs = ns;
    c.w = reinterpret_cast<const float*>(b.w_tcn_dev); c.ktot = koff;
    c.bias = b.b_tcn_dev; c.bias_per_node = (i == 0 && b.res_kind == TIK_RES_STEM) ? 1 : 0;
    c.v = V; c.t_out = t_o; c.c_out = b.c_out; c.c_out_valid = b.c_out;
    c.act = TIK_ACT_RELU;
    if (b.res_kind == TIK_RES_IDENTITY) c.res = xbuf[cur];
    else if (b.res_kind == TIK_RES_STEM) c.res = r0buf;
    const int nxt = (i == 0) ? 0 : cur ^ 1;
    c.out = last ? feat : xbuf[nxt];
    c.out_layout = last ? TIK_OUT_TIME_MAJOR : TIK_OUT_NODE_MAJOR;
    c.rb = rb_for((int64_t)V * t_o, b.c_out);
    ph.push_back(c);
    cur = nxt;
    t = t_o;
  }
  const int c_last = net->blocks[net->n_blocks - 1].c_out;
  TIK_CHECK_ARG((V * c_last) % 4 == 0, "latency plan: feature width must be a multiple of 4");
  LatPhase h1;
  memset(&h1, 0, sizeof(h1));
  h1.kind = 2; h1.n_slabs = 1; h1.nbr = -1;
  h1.slabs[0] = {feat, V * c_last, 0, 1, 0, 0};
  h1.w = reinterpret_cast<const float*>(net->w1_dev); h1.ktot = V * c_last;
  h1.bias = net->b1_dev; h1.v = 1; h1.t_out = tf; h1.c_out = net->head_hidden; h1.c_out_valid = net->head_hidden;
  h1.act = TIK_ACT_LEAKY; h1.slope = net->leaky_slope; h1.out = zbuf; h1.out_layout = TIK_OUT_NODE_MAJOR;
  ph.push_back(h1);
  LatPhase h2 = h1;
  h2.slabs[0] = {zbuf, net->head_hidden, 0, 1, 0, 0};
  h2.w = reinterpret_cast<const float*>(net->w2_dev); h2.ktot = net->head_hidden;
  h2.bias = net->b2_dev; h2.c_out = net->head_out; h2.c_out_valid = net->head_out;
  h2.act = TIK_ACT_NONE; h2.out = nullptr; h2.out_layout = TIK_OUT_ROWS_F32;
  ph.push_back(h2);
  TIK_CHECK_ARG((int)ph.size() <= kLatMaxPhases, "latency plan: too many phases");
  TIK_CUDA(cudaMemcpy(ws + L.off_phases, ph.data(), ph.size() * sizeof(LatPhase), cudaMemcpyHostToDevice));
  int dev = 0, sms = 148, coop = 0, per_sm = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  TIK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  TIK_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
  if (!coop) { set_error("latency plan: the device does not support cooperative launches"); return TIK_ERR_UNSUPPORTED; }
  const size_t smem = lat_smem_bytes((int)ph.size(), net->n_blocks);
  TIK_CHECK_ARG(smem <= 200 * 1024, "latency plan: %zu bytes of shared memory (too many blocks)", smem);
  TIK_CUDA(cudaFuncSetAttribute(stgcn_latency_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  TIK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, stgcn_latency_kernel, kLatThreads, smem));
  if (per_sm < 1) { set_error("latency plan: kernel does not fit on an SM"); return TIK_ERR_UNSUPPORTED; }
  TikLatencyPlan* P = new TikLatencyPlan();
  P->net = *net; P->n_max = n_max; P->T = T; P->T_out = tf;
  P->n_phases = (int)ph.size();
  P->phases_dev = reinterpret_cast<LatPhase*>(ws + L.off_phases);
  P->nbr_dev = nbr_dev; P->n_nbr = net->n_blocks; P->smem = smem;
  // one CTA per SM by default: every grid barrier costs one round over 148 arrivals (TIK_LAT_CTAS_PER_SM=2 for experiments)
  int want = 1;
  if (const char* e = getenv("TIK_LAT_CTAS_PER_SM")) want = atoi(e);
  P->grid = sms * std::max(1, std::min(per_sm, want));
  P->times_dev = nullptr;
  *out = P;
  return TIK_OK;
}

// Every run of a latency plan: clip n of the N clips is window n of x read through win (the entry point has checked
// win itself, or built it for a plain batch).  Every argument check of the three entry points is here.
static int lat_run(TikLatencyPlan* P, const float* x, const TikWindowing& win, const tik::WinSeqs& seqs, int64_t N, float* poses,
                   void* stream) {
  using namespace tik;
  TIK_CHECK_ARG(P != nullptr, "latency plan: null plan");
  TIK_CHECK_ARG(x && poses, "latency plan: null input or poses pointer");
  TIK_CHECK_ARG(N >= 0 && N <= P->n_max, "latency plan: N = %lld outside [0, n_max = %lld]", (long long)N, (long long)P->n_max);
  TIK_CHECK_ARG(win.root_a < P->net.V && win.root_b < P->net.V, "latency plan: root keypoints (%d, %d) must be < V = %d",
                win.root_a, win.root_b, P->net.V);
  if (N == 0) return TIK_OK;
  LatParams p;
  p.phases = P->phases_dev; p.n_phases = P->n_phases; p.nbr = P->nbr_dev; p.n_nbr = P->n_nbr;
  p.x = x; p.poses = poses; p.N = N; p.win = win; p.seqs = seqs; p.times = P->times_dev;
  void* args[] = {&p};
  TIK_CUDA(cudaLaunchCooperativeKernel((const void*)stgcn_latency_kernel, dim3((unsigned)P->grid), dim3(kLatThreads), args, P->smem, (cudaStream_t)stream));
  return TIK_OK;
}

int tik_stgcn_latency_run(TikLatencyPlan* plan, const float* x_dev, int64_t N, float* poses_dev, void* stream) {
  return lat_run(plan, x_dev, tik::plain_windowing(N, plan ? plan->T : 0), tik::WinSeqs{}, N, poses_dev, stream);
}

int tik_stgcn_latency_run_windows(TikLatencyPlan* plan, const float* seq_dev, const TikWindowing* win, int64_t n_windows,
                                  float* poses_dev, void* stream) {
  int rc = tik::check_windowing(win, "latency plan");
  return rc != TIK_OK ? rc : lat_run(plan, seq_dev, *win, tik::WinSeqs{}, n_windows, poses_dev, stream);
}

int tik_stgcn_latency_run_seq_windows(TikLatencyPlan* plan, const float* seq_dev, const TikWindowing* win,
                                      const TikSeqBatch* seqs, int64_t n_windows, float* poses_dev, void* stream) {
  int rc = tik::check_seq_windows(win, seqs, n_windows, "latency plan");
  return rc != TIK_OK ? rc : lat_run(plan, seq_dev, *win, tik::win_seqs(*seqs), n_windows, poses_dev, stream);
}

int tik_stgcn_latency_phases(const TikLatencyPlan* plan) { return plan ? plan->n_phases : 0; }

int tik_debug_latency_times(TikLatencyPlan* plan, void* dev_buf) {
  if (!plan) return TIK_ERR_INVALID;
  plan->times_dev = reinterpret_cast<unsigned long long*>(dev_buf);
  return TIK_OK;
}

void tik_stgcn_latency_destroy(TikLatencyPlan* plan) { delete plan; }

}  // extern "C"
