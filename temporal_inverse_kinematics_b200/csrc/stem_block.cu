// The whole first ST-GCN block in ONE kernel (bf16 tensor-core path):
//
//   X0 = data_bn(x)                                                    st_gcn_aaai18.py:119-125
//   H0[n,w,t,:] = relu( Wg' . (sum_v A^[v,w] X0[n,t,v,:]) + b1[w,:] )    gconv_origin.py:56-65 + tcn.0/tcn.1
//   R0[n,w,t,:] = Wr' . (s0[w,:] * x[n,t,w,:])                          residual 1x1 conv + BN (st_gcn_aaai18.py:198-204)
//   Y0[n,w,t,:] = relu( sum_dt Wt'[dt] . H0[n,w,t+dt-1,:] + R0 + b2[w,:] )   tcn.2-4 + residual + ReLU (:205-214)
//
// Neither H0 nor R0 ever reaches HBM (the two-kernel path writes and re-reads both: 2.2 GB per 4096 clips); the
// kernel reads the raw (N,T,V,3) fp32 keypoints and writes the node-major bf16 block output.
//
// A tile is lo = min(T, 13) output frames x V nodes of one clip, computed from 15 input frames (one halo frame each
// side; rows past lo + 1 are zero).  Rows are node-major inside the tile, h = v*15 + l (V <= 17: at most 255 rows = two
// 128-row MMA tiles), so a temporal tap is a
// shift of the A operand by one 128-byte shared-memory row and a tap at a tile edge never crosses a node boundary
// into a valid output row.
//   builders (8 warps, SIMT): data_bn, adjacency aggregation and the residual's scaled input, written as ONE
//            16-wide K slice per row: [agg_hi | agg_lo | xs_hi | xs_lo | 0] (bf16 hi/lo split: the inputs keep
//            ~16 bits of mantissa), double buffered;
//   MMA A:   Hpre = slice . Wg'^T (H0 pre-activation) and RD = slice . Wr'^T (R0): one K=16 tcgen05.mma each per 128 rows;
//   mid pass (8 warps): Hpre + b1 -> ReLU -> zero outside the clip (the temporal conv pads H0, not x) -> bf16
//            -> shared memory in the 128B-swizzled K-major layout;
//   MMA 3:   RD += sum_dt H0[h + dt - 1] . Wt'[dt]^T -- accumulates ON TOP of R0 in tensor memory, so the
//            residual costs nothing;
//   final pass (8 other warps): RD + b2 -> ReLU -> bf16 -> staging (aliases the H0 tile) -> 4-D TMA store.
// Two tiles are in flight (TMEM: 2 x 128 columns of Hpre, 2 x 128 of RD): the epilogue warps run tile i+1's mid pass and tile i's final
// pass concurrently, while the tensor pipe executes tile i's temporal taps.
#include <string.h>

#include <algorithm>
#include <vector>

#include "tik_common.cuh"
#include "umma_prepared.h"
#include "umma_ptx.cuh"

namespace tik {

constexpr int kSbL = 15;                            // frames per tile incl. halo (V * kSbL <= 256 rows = two 128-row MMA tiles)
constexpr int kSbLoMax = kSbL - 2;                 // output frames per tile (T = 64: 5 tiles of 13 instead of 6 of 12)
constexpr int kSbCout = 64;
constexpr int kSbEpiWarps = 16, kSbBuildWarps = 8;
constexpr int kSbThreads = 64 + 32 * kSbEpiWarps + 32 * kSbBuildWarps;   // 832
constexpr int kSbTile = 16384;                      // 128 rows x 128 B
constexpr int kSbHBytes = 1024 + 2 * kSbTile + 1024;   // 8 guard rows + 256 rows + 8 guard rows
constexpr int kSbMaxV = 256 / kSbL;                // V * kSbL <= 256
// shared-memory map (bytes from the 1024-aligned base)
constexpr int kSbOffW16 = 0;                        // stacked [Wg' ; Wr'] : 128 rows x 64 K
constexpr int kSbOffWt = kSbOffW16 + kSbTile;       // 3 taps x (64 rows x 64 K)
constexpr int kSbOffA0 = kSbOffWt + 3 * 8192;       // 2 buffers x 2 MMA tiles
constexpr int kSbOffH = kSbOffA0 + 4 * kSbTile;     // 2 buffers
constexpr int kSbOffBias1 = kSbOffH + 2 * kSbHBytes;
constexpr int kSbBiasLd = kSbCout + 4;               // padded pitch: rows of different nodes start in different banks
constexpr int kSbOffBias2 = kSbOffBias1 + kSbMaxV * kSbBiasLd * 4;
constexpr int kSbOffAs = kSbOffBias2 + kSbMaxV * kSbBiasLd * 4;           // As[u][v][c] = A^[u,v] * s0[u,c]   (V*V*Cin fp32)
constexpr int kSbNbrLd = 20;                        // neighbour list pitch (ints): lists are read 4 entries at a time
constexpr int kSbAsLd = 20 * 4 + 4;                 // weight row pitch (floats) for CIN <= 4: 16-byte aligned, odd multiple of 4 banks
constexpr int kSbOffNbr = kSbOffAs + kSbMaxV * kSbAsLd * 4;             // per node: source-node offsets of the non-zero A^[u,v], zero padded
constexpr int kSbOffCnt = kSbOffNbr + kSbMaxV * kSbNbrLd * 4;           // per node: number of 4-entry groups
constexpr int kSbOffCst = kSbOffCnt + kSbMaxV * 4 + 8;         // cst[v][c] = sum_u A^[u,v] o0[u,c]; sum[v][c] = sum_u As; scale[v][c]
constexpr int kSbRawBufs = 3;                                           // raw keypoint tiles in flight (cp.async)
constexpr int kSbOffRaw = kSbOffCst + 3 * kSbMaxV * 4 * 4;              // kSbRawBufs x 14 x V*Cin fp32
constexpr int kSbOffBar = (kSbOffRaw + kSbRawBufs * kSbL * kSbMaxV * 4 * 4 + 15) / 16 * 16;
constexpr int kSbSmemBytes = kSbOffBar + 256 + 1024;

struct StemBlockParams {
  CUtensorMap map_w16, map_wt, map_out;
  const float* x;
  const float* in_scale; const float* in_shift; const float* agg;
  const float* bias1;                       // (V, 64)
  const float* bias2; int32_t bias2_per_node;
  int32_t n_clips, T, V, lo, tiles_t;       // lo = output frames per tile, tiles_t = ceil(T / lo)
  TikWindowing win; long long win_n0;
  WinSeqs seqs;                             // ragged batch tables (n_seqs == 0: none)
};

__device__ __forceinline__ uint32_t bf16_bits(float v) { return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v)); }

template <int CIN>
__global__ void __launch_bounds__(kSbThreads, 1) stem_block_kernel(const __grid_constant__ StemBlockParams p) {
  static_assert(4 * CIN <= 16, "hi/lo slices of the aggregated and the scaled input must fit one K=16 step");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; pointer arithmetic on the shared base keeps the address space (LDS / STS, not generic LD / ST)
  uint8_t* s_w16 = smem + kSbOffW16;
  uint8_t* s_wt = smem + kSbOffWt;
  uint8_t* s_a0 = smem + kSbOffA0;
  uint8_t* s_h = smem + kSbOffH;
  float* s_bias1 = reinterpret_cast<float*>(smem + kSbOffBias1);
  float* s_bias2 = reinterpret_cast<float*>(smem + kSbOffBias2);
  float* s_as = reinterpret_cast<float*>(smem + kSbOffAs);
  int* s_nbr = reinterpret_cast<int*>(smem + kSbOffNbr);   // [v][k] = u_k * CIN, padded with 0 (weight 0) to a multiple of 4
  int* s_cnt4 = reinterpret_cast<int*>(smem + kSbOffCnt);  // [v] = groups of 4 neighbours
  float* s_cst = reinterpret_cast<float*>(smem + kSbOffCst);
  float* s_sum = s_cst + kSbMaxV * 4;
  float* s_scale = s_sum + kSbMaxV * 4;
  float* s_rawbuf = reinterpret_cast<float*>(smem + kSbOffRaw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kSbOffBar);
  uint64_t* w_full = bars;                  // [1]
  uint64_t* a0_full = bars + 1;             // [2] builders -> MMA
  uint64_t* a0_empty = bars + 3;            // [2] MMA A has read the slice
  uint64_t* da_full = bars + 5;             // [2] MMA A done -> mid pass
  uint64_t* h_full = bars + 7;              // [2] mid pass wrote H0 -> MMA 3
  uint64_t* d3_full = bars + 9;             // [2] MMA 3 done -> final pass
  uint64_t* tmem_empty = bars + 11;         // [2] final pass has read the accumulators
  uint64_t* stage_full = bars + 13;         // [2] final pass wrote the staging tile -> store
  uint64_t* h_empty = bars + 15;            // [2] store has read the staging tile (aliases H0)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 17);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int V = p.V, VC = V * CIN;
  const int n_tiles = p.n_clips * p.tiles_t;
  const int my_tiles = n_tiles > (int)blockIdx.x ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.map_w16); tma_prefetch_desc(&p.map_wt); tma_prefetch_desc(&p.map_out); }
  if (warp == 1 && lane == 0) {
    mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a0_full[i], kSbBuildWarps); mbar_init(&a0_empty[i], 1); mbar_init(&da_full[i], 1);
      mbar_init(&h_full[i], kSbEpiWarps / 2); mbar_init(&d3_full[i], 1); mbar_init(&tmem_empty[i], kSbEpiWarps / 2);
      mbar_init(&stage_full[i], kSbEpiWarps / 2); mbar_init(&h_empty[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  for (int i = threadIdx.x; i < V * kSbCout; i += kSbThreads) {
    const int bi = (i / kSbCout) * kSbBiasLd + (i % kSbCout);
    s_bias1[bi] = __ldg(p.bias1 + i);
    s_bias2[bi] = __ldg(p.bias2 + (p.bias2_per_node ? i : (i % kSbCout)));
  }
  // data_bn folded into the aggregation:  sum_u A^[u,v] (s0[u,c] x[u,c] + o0[u,c]) = sum_u As[v,u,c] x[u,c] + cst[v,c]
  // and only the non-zero adjacency entries are visited (the skeleton graph is sparse): compacted per target node v
  if (threadIdx.x < V) {
    const int v = threadIdx.x;
    int cnt = 0;
    for (int u = 0; u < V; ++u) {
      const float a = __ldg(p.agg + u * V + v);
      if (a != 0.f) {
        s_nbr[v * kSbNbrLd + cnt] = u * CIN;
        for (int c = 0; c < CIN; ++c) s_as[v * kSbAsLd + cnt * CIN + c] = a * __ldg(p.in_scale + u * CIN + c);
        ++cnt;
      }
    }
    const int cnt4 = (cnt + 3) / 4;
    for (int k = cnt; k < cnt4 * 4; ++k) {                   // padding entries: node 0 with weight 0
      s_nbr[v * kSbNbrLd + k] = 0;
      for (int c = 0; c < CIN; ++c) s_as[v * kSbAsLd + k * CIN + c] = 0.f;
    }
    s_cnt4[v] = cnt4;
  }
  for (int i = threadIdx.x; i < VC; i += kSbThreads) {
    const int v = i / CIN, c = i - v * CIN;
    float cst = 0.f, sum = 0.f;
    for (int u = 0; u < V; ++u) {
      const float a = __ldg(p.agg + u * V + v);
      cst = fmaf(a, __ldg(p.in_shift + u * CIN + c), cst);
      sum = fmaf(a, __ldg(p.in_scale + u * CIN + c), sum);
    }
    s_cst[i] = cst; s_sum[i] = sum; s_scale[i] = __ldg(p.in_scale + i);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();                                               // tables above are constants; x may come from a previous kernel

  if (warp == 0) {
    // ===================== weights (once) + TMA store issuer =====================
    if (lane == 0) {
      mbar_expect_tx(w_full, (uint32_t)(kSbTile + 3 * 8192));
      tma_load_2d(s_w16, &p.map_w16, w_full, 0, 0);
      for (int dt = 0; dt < 3; ++dt) tma_load_2d(s_wt + dt * 8192, &p.map_wt, w_full, dt * kSbCout, 0);
      for (int it = 0; it < my_tiles; ++it) {
        const int tile = (int)blockIdx.x + it * (int)gridDim.x;
        const int n = tile / p.tiles_t, tt = tile - n * p.tiles_t;
        const int b = it & 1;
        mbar_wait(&stage_full[b], (uint32_t)((it >> 1) & 1));
        tma_store_4d(&p.map_out, s_h + (size_t)b * kSbHBytes + 1024, 0, tt * p.lo, 0, n);
        tma_store_commit();
        tma_store_wait_read0();
        mbar_arrive(&h_empty[b]);
      }
      tma_store_wait0();
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (warp-uniform loop, lane 0 issues) =====================
    constexpr uint32_t idesc = make_idesc_bf16(128, kSbCout);
    const bool leader = lane == 0;
    mbar_wait(w_full, 0);
    const uint32_t w16_u32 = smem_u32(s_w16), wt_u32 = smem_u32(s_wt), a0_u32 = smem_u32(s_a0), h_u32 = smem_u32(s_h);
    // TMEM: Hpre[b][j] at columns b*128 + j*64 (read by the mid pass), RD[b][j] at 256 + b*128 + j*64 (R0, then the
    // temporal taps accumulate on top; read by the final pass).  Separate lifetimes: the next tile's H0 GEMM never
    // waits for the previous final pass.
    auto issue_ah = [&](int it) {
      const int b = it & 1;
      mbar_wait(&a0_full[b], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      if (leader) {
#pragma unroll
        for (int j = 0; j < 2; ++j)
          umma_bf16(tmem_base + (uint32_t)(b * 128 + j * 64), make_smem_desc_kmajor_sw128(a0_u32 + (uint32_t)(b * 2 + j) * kSbTile),
                    make_smem_desc_kmajor_sw128(w16_u32), idesc, 0u);
        umma_commit(&da_full[b]);
      }
      __syncwarp();
    };
    auto issue_ar = [&](int it) {
      const int b = it & 1;
      mbar_wait(&tmem_empty[b], (uint32_t)(((it >> 1) & 1) ^ 1));
      tc_fence_after();
      if (leader) {
#pragma unroll
        for (int j = 0; j < 2; ++j)
          umma_bf16(tmem_base + (uint32_t)(256 + b * 128 + j * 64), make_smem_desc_kmajor_sw128(a0_u32 + (uint32_t)(b * 2 + j) * kSbTile),
                    make_smem_desc_kmajor_sw128(w16_u32 + 64u * 128u), idesc, 0u);
        umma_commit(&a0_empty[b]);
      }
      __syncwarp();
    };
    if (my_tiles > 0) { issue_ah(0); issue_ar(0); }
    for (int it = 0; it < my_tiles; ++it) {
      const int b = it & 1;
      if (it + 1 < my_tiles) issue_ah(it + 1);
      mbar_wait(&h_full[b], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      if (leader) {
        const uint32_t hb = h_u32 + (uint32_t)b * kSbHBytes + 1024u;
#pragma unroll
        for (int dt = 0; dt < 3; ++dt) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const uint32_t arow = hb + (uint32_t)(128 * j + dt - 1) * 128u;     // may start 128 B below the tile: guard rows
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem_base + (uint32_t)(256 + b * 128 + j * 64), make_smem_desc_kmajor_sw128(arow + (uint32_t)k * 32u),
                        make_smem_desc_kmajor_sw128(wt_u32 + (uint32_t)dt * 8192u + (uint32_t)k * 32u), idesc, 1u);
          }
        }
        umma_commit(&d3_full[b]);
      }
      __syncwarp();
      if (it + 1 < my_tiles) issue_ar(it + 1);
    }
  } else if (warp < 2 + kSbEpiWarps / 2) {
    // ===================== mid group (8 warps): Hpre + b1 -> ReLU -> bf16 H0 tile in shared memory =====================
    const int lane_grp = warp & 3;
    const int half = (warp - 2) >> 2;                     // 32-column half of the 64 channels
    const int i_row = lane_grp * 32 + lane;
    const uint32_t lane_off = (uint32_t)(lane_grp * 32) << 16;
    for (int it = 0; it < my_tiles; ++it) {
      const int b = it & 1;
      const uint32_t ph = (uint32_t)((it >> 1) & 1);
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const int tt = tile % p.tiles_t;
      const int t_first = tt * p.lo - 1;                  // frame of tile row l = 0
      mbar_wait(&da_full[b], ph);
      tc_fence_after();
      mbar_wait(&h_empty[b], ph ^ 1);                     // the store that read this buffer as a staging tile is done
      uint8_t* hb = s_h + (size_t)b * kSbHBytes + 1024;
#pragma unroll
      for (int j = 0; j < 2; ++j) {                       // one 128-row MMA tile at a time: 32 live accumulator registers
        uint32_t a[32];
        tmem_ld16(tmem_base + lane_off + (uint32_t)(b * 128 + j * 64 + half * 32), a);
        tmem_ld16(tmem_base + lane_off + (uint32_t)(b * 128 + j * 64 + half * 32 + 16), a + 16);
        tmem_ld_wait();
        const int h = 128 * j + i_row;
        const int v = h / kSbL, l = h - v * kSbL;
        const int t = t_first + l;
        const bool ok = v < V && t >= 0 && t < p.T;
        const float* bias = s_bias1 + (v < V ? v : 0) * kSbBiasLd + half * 32;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 b0 = *reinterpret_cast<const float4*>(bias + 8 * q);
          const float4 b1 = *reinterpret_cast<const float4*>(bias + 8 * q + 4);
          uint4 u;
          u.x = pack_bf16x2_relu(__uint_as_float(a[8 * q + 0]) + b0.x, __uint_as_float(a[8 * q + 1]) + b0.y);
          u.y = pack_bf16x2_relu(__uint_as_float(a[8 * q + 2]) + b0.z, __uint_as_float(a[8 * q + 3]) + b0.w);
          u.z = pack_bf16x2_relu(__uint_as_float(a[8 * q + 4]) + b1.x, __uint_as_float(a[8 * q + 5]) + b1.y);
          u.w = pack_bf16x2_relu(__uint_as_float(a[8 * q + 6]) + b1.z, __uint_as_float(a[8 * q + 7]) + b1.w);
          if (!ok) u = make_uint4(0, 0, 0, 0);            // temporal zero padding applies to H0
          *reinterpret_cast<uint4*>(hb + (size_t)h * 128 + (((half * 4 + q) ^ (h & 7)) << 4)) = u;
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&h_full[b]);
    }
  } else if (warp < 2 + kSbEpiWarps) {
    // ===================== final group (8 warps): RD + b2 -> ReLU -> bf16 -> staging tile (aliases H0) =====================
    const int lane_grp = warp & 3;
    const int half = (warp - 2 - kSbEpiWarps / 2) >> 2;
    const int i_row = lane_grp * 32 + lane;
    const uint32_t lane_off = (uint32_t)(lane_grp * 32) << 16;
    for (int it = 0; it < my_tiles; ++it) {
      const int b = it & 1;
      mbar_wait(&d3_full[b], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      uint8_t* stage = s_h + (size_t)b * kSbHBytes + 1024;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        uint32_t a[32];
        tmem_ld16(tmem_base + lane_off + (uint32_t)(256 + b * 128 + j * 64 + half * 32), a);
        tmem_ld16(tmem_base + lane_off + (uint32_t)(256 + b * 128 + j * 64 + half * 32 + 16), a + 16);
        tmem_ld_wait();
        if (j == 1) {                                      // both accumulator tiles are in registers / already staged
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[b]);
        }
        const int h = 128 * j + i_row;
        const int v = h / kSbL, l = h - v * kSbL;
        if (v < V && l >= 1 && l <= p.lo) {
          const int srow = v * p.lo + l - 1;
          const float* bias = s_bias2 + v * kSbBiasLd + half * 32;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 b0 = *reinterpret_cast<const float4*>(bias + 8 * q);
            const float4 b1 = *reinterpret_cast<const float4*>(bias + 8 * q + 4);
            uint4 u;
            u.x = pack_bf16x2_relu(__uint_as_float(a[8 * q + 0]) + b0.x, __uint_as_float(a[8 * q + 1]) + b0.y);
            u.y = pack_bf16x2_relu(__uint_as_float(a[8 * q + 2]) + b0.z, __uint_as_float(a[8 * q + 3]) + b0.w);
            u.z = pack_bf16x2_relu(__uint_as_float(a[8 * q + 4]) + b1.x, __uint_as_float(a[8 * q + 5]) + b1.y);
            u.w = pack_bf16x2_relu(__uint_as_float(a[8 * q + 6]) + b1.z, __uint_as_float(a[8 * q + 7]) + b1.w);
            *reinterpret_cast<uint4*>(stage + (size_t)srow * 128 + (((half * 4 + q) ^ (srow & 7)) << 4)) = u;
          }
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&stage_full[b]);
    }
  } else {
    // ===================== builders: raw keypoints -> one K=16 operand slice per tile row =====================
    // Raw frames arrive through 4-byte cp.async copies two tiles ahead (the 204-byte frames are not 16-byte aligned,
    // so no bulk copy); one thread then builds one tile row.
    constexpr int NB = 32 * kSbBuildWarps;
    const int tid = threadIdx.x - 32 * (2 + kSbEpiWarps);
    // this thread's (at most 3) elements of a raw tile: frame l and offset vc inside the frame never change
    int el_l[3], el_vc[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int idx = tid + k * NB;
      el_l[k] = idx < kSbL * VC ? idx / VC : -1;
      el_vc[k] = idx - (idx / VC) * VC;
    }
    auto prefetch = [&](int it) {
      if (it < my_tiles) {
        const int tile = (int)blockIdx.x + it * (int)gridDim.x;
        const int n = tile / p.tiles_t, tt = tile - n * p.tiles_t;
        const int t_first = tt * p.lo - 1;
        const uint32_t dst = smem_u32(s_rawbuf + (it % kSbRawBufs) * (kSbL * kSbMaxV * 4)) + (uint32_t)tid * 4u;
        const WinClip clip = win_clip(p.win, p.seqs, p.win_n0 + (long long)n);   // clip n is window win_n0 + n of the input
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          if (el_l[k] >= 0) {
            const int t = t_first + el_l[k];
            const bool ok = t >= 0 && t < p.T;
            const float* src = ok ? p.x + win_frame(clip, t) * VC + el_vc[k] : p.x;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst + (uint32_t)(k * NB) * 4u), "l"(src), "r"(ok ? 4 : 0) : "memory");
          }
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    prefetch(0);
    prefetch(1);
    for (int it = 0; it < my_tiles; ++it) {
      const int b = it & 1;
      prefetch(it + 2);
      asm volatile("cp.async.wait_group 2;" ::: "memory");
      named_bar_sync(3, NB);                                // every thread's copies of tile `it` have landed
      const float* raw = s_rawbuf + (it % kSbRawBufs) * (kSbL * kSbMaxV * 4);
      mbar_wait(&a0_empty[b], (uint32_t)(((it >> 1) & 1) ^ 1));
      const int h = tid;
      if (h < V * kSbL) {
        const int v = h / kSbL, l = h - v * kSbL;
        const float* fr = raw + l * VC;
        float root[CIN], agg[CIN], xs[CIN];
#pragma unroll
        for (int c = 0; c < CIN; ++c) {
          // window mode: root-centred on 0.5*(kp[a]+kp[b]) (data_amass.py:232-235)
          root[c] = p.win.root_a >= 0 ? 0.5f * (fr[p.win.root_a * CIN + c] + fr[p.win.root_b * CIN + c]) : 0.f;
          agg[c] = s_cst[v * CIN + c] - root[c] * s_sum[v * CIN + c];
          xs[c] = (fr[v * CIN + c] - root[c]) * s_scale[v * CIN + c];
        }
        // four neighbours per step: one 16-byte load of their offsets, then independent weight / value loads, so the
        // shared-memory latencies overlap instead of chaining (the port is contended by the running tap MMAs)
        const int cnt4 = s_cnt4[v];
        for (int g4 = 0; g4 < cnt4; ++g4) {
          const int4 off = *reinterpret_cast<const int4*>(s_nbr + v * kSbNbrLd + 4 * g4);
          const float* wv = s_as + v * kSbAsLd + 4 * g4 * CIN;
          const int o[4] = {off.x, off.y, off.z, off.w};
          float w[4][CIN], xv[4][CIN];
#pragma unroll
          for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int c = 0; c < CIN; ++c) { w[k][c] = wv[k * CIN + c]; xv[k][c] = fr[o[k] + c]; }
#pragma unroll
          for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int c = 0; c < CIN; ++c) agg[c] = fmaf(w[k][c], xv[k][c], agg[c]);
        }
        // slots: [agg_hi(CIN) | agg_lo(CIN) | xs_hi(CIN) | xs_lo(CIN) | 0...]
        uint32_t e[16];
#pragma unroll
        for (int s = 0; s < 16; ++s) e[s] = 0;
#pragma unroll
        for (int c = 0; c < CIN; ++c) {
          const __nv_bfloat16 ah = __float2bfloat16_rn(agg[c]);
          const __nv_bfloat16 xh = __float2bfloat16_rn(xs[c]);
          e[c] = (uint32_t)__bfloat16_as_ushort(ah);
          e[CIN + c] = bf16_bits(agg[c] - __bfloat162float(ah));
          e[2 * CIN + c] = (uint32_t)__bfloat16_as_ushort(xh);
          e[3 * CIN + c] = bf16_bits(xs[c] - __bfloat162float(xh));
        }
        uint8_t* row = s_a0 + (size_t)(b * 2 + (h >> 7)) * kSbTile + (size_t)(h & 127) * 128;
        const uint4 p0 = make_uint4(e[0] | (e[1] << 16), e[2] | (e[3] << 16), e[4] | (e[5] << 16), e[6] | (e[7] << 16));
        const uint4 p1 = make_uint4(e[8] | (e[9] << 16), e[10] | (e[11] << 16), e[12] | (e[13] << 16), e[14] | (e[15] << 16));
        *reinterpret_cast<uint4*>(row + ((0 ^ (h & 7)) << 4)) = p0;
        *reinterpret_cast<uint4*>(row + ((1 ^ (h & 7)) << 4)) = p1;
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&a0_full[b]);
      named_bar_sync(3, NB);                                // the raw buffer is refilled by the next prefetch
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ host side
struct StemBlockPrepared {
  StemBlockParams p;
  int cin;
  int64_t cap;
};

bool stem_block_supported(const TikNet* net, int dtype) {
  if (dtype != TIK_BF16 || net->n_blocks < 1) return false;
  const TikBlock& b = net->blocks[0];
  return net->K == 1 && net->c_in == 3 && b.c_out == kSbCout && b.kt == 3 && b.stride == 1 && net->V <= kSbMaxV &&
         (b.res_kind == TIK_RES_NONE || (b.res_kind == TIK_RES_STEM && b.w_res_stem_dev));
}

int64_t stem_block_workspace_bytes() { return kSbTile; }

int stem_block_prepare(const TikNet* net, void* w16_dev, void* out, int64_t n_clips, int T, StemBlockPrepared** outp) {
  TIK_CHECK_ARG(stem_block_supported(net, TIK_BF16) && w16_dev && out && n_clips > 0 && T > 0, "stem block: unsupported configuration");
  TIK_CHECK_ARG(n_clips * ceil_div(T, kSbLoMax) < (1ll << 31), "stem block: too many tiles");
  const TikBlock& b = net->blocks[0];
  const int V = net->V, cin = net->c_in;
  // stacked weights [Wg' ; Wr'] against the operand slots [agg_hi | agg_lo | xs_hi | xs_lo]
  std::vector<float> wg((size_t)kSbCout * cin), s0((size_t)V * cin), wrs;
  cudaError_t ce = cudaMemcpy(wg.data(), b.w_gcn_dev, wg.size() * 4, cudaMemcpyDeviceToHost);
  if (ce == cudaSuccess) ce = cudaMemcpy(s0.data(), net->in_scale_dev, s0.size() * 4, cudaMemcpyDeviceToHost);
  if (ce == cudaSuccess && b.res_kind == TIK_RES_STEM) {
    wrs.resize((size_t)V * kSbCout * cin);
    ce = cudaMemcpy(wrs.data(), b.w_res_stem_dev, wrs.size() * 4, cudaMemcpyDeviceToHost);
  }
  if (ce != cudaSuccess) { set_error("stem block: weight download failed: %s", cudaGetErrorString(ce)); return TIK_ERR_CUDA; }
  std::vector<__nv_bfloat16> w16((size_t)128 * 64, __float2bfloat16_rn(0.f));
  for (int co = 0; co < kSbCout; ++co)
    for (int c = 0; c < cin; ++c) {
      const __nv_bfloat16 g = __float2bfloat16_rn(wg[(size_t)co * cin + c]);
      w16[(size_t)co * 64 + c] = g;
      w16[(size_t)co * 64 + cin + c] = g;
      if (!wrs.empty()) {
        // w_res_stem[v] = Wr' * s0[v]  ->  Wr' from the node with the largest |s0[v, c]| (zero scale everywhere: no contribution)
        int vb = 0;
        for (int v = 1; v < V; ++v)
          if (fabsf(s0[(size_t)v * cin + c]) > fabsf(s0[(size_t)vb * cin + c])) vb = v;
        const float sc = s0[(size_t)vb * cin + c];
        const float wr = sc != 0.f ? (float)((double)wrs[((size_t)vb * kSbCout + co) * cin + c] / (double)sc) : 0.f;
        const __nv_bfloat16 r = __float2bfloat16_rn(wr);
        w16[(size_t)(64 + co) * 64 + 2 * cin + c] = r;
        w16[(size_t)(64 + co) * 64 + 3 * cin + c] = r;
      }
    }
  ce = cudaMemcpy(w16_dev, w16.data(), w16.size() * 2, cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) { set_error("stem block: weight upload failed: %s", cudaGetErrorString(ce)); return TIK_ERR_CUDA; }

  StemBlockPrepared* g = new StemBlockPrepared();
  StemBlockParams& p = g->p;
  memset(&p, 0, sizeof(p));
  g->cin = cin; g->cap = n_clips;
  p.in_scale = net->in_scale_dev; p.in_shift = net->in_shift_dev; p.agg = b.agg_dev;
  p.bias1 = b.b_gcn_dev; p.bias2 = b.b_tcn_dev; p.bias2_per_node = b.res_kind == TIK_RES_STEM ? 1 : 0;
  p.T = T; p.V = V;
  p.lo = T < kSbLoMax ? T : kSbLoMax;
  p.tiles_t = (T + p.lo - 1) / p.lo;
  int rc;
  {
    uint64_t dims[2] = {64, 128};
    uint64_t strides[1] = {128};
    uint32_t box[2] = {64, 128};
    rc = encode_bf16_map(&p.map_w16, w16_dev, 2, dims, strides, box);
  }
  if (rc == TIK_OK) {
    const uint64_t ktot = (uint64_t)3 * kSbCout + (b.res_as_slab ? kSbCout : 0);
    uint64_t dims[2] = {ktot, (uint64_t)kSbCout};
    uint64_t strides[1] = {ktot * 2};
    uint32_t box[2] = {64, (uint32_t)kSbCout};
    rc = encode_bf16_map(&p.map_wt, b.w_tcn_dev, 2, dims, strides, box);
  }
  if (rc == TIK_OK) {
    uint64_t dims[4] = {(uint64_t)kSbCout, (uint64_t)T, (uint64_t)V, (uint64_t)n_clips};
    uint64_t strides[3] = {(uint64_t)kSbCout * 2, (uint64_t)kSbCout * 2 * T, (uint64_t)kSbCout * 2 * T * V};
    uint32_t box[4] = {64, (uint32_t)p.lo, (uint32_t)V, 1};
    rc = encode_bf16_map(&p.map_out, out, 4, dims, strides, box);
  }
  if (rc != TIK_OK) { delete g; return rc; }
  *outp = g;
  return TIK_OK;
}

int stem_block_launch(StemBlockPrepared* g, const float* x, int64_t n_clips, const TikWindowing& win, int64_t win_n0,
                      const WinSeqs& seqs, cudaStream_t s) {
  TIK_CHECK_ARG(g && x && n_clips <= g->cap, "stem block: n_clips exceeds the prepared capacity");
  if (n_clips <= 0) return TIK_OK;
  StemBlockParams p = g->p;
  p.x = x; p.n_clips = (int32_t)n_clips;
  p.win = win;
  p.win_n0 = (long long)win_n0;
  p.seqs = seqs;
  static bool attr_done[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (!attr_done[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(stem_block_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSbSmemBytes));
    attr_done[dev & 63] = true;
  }
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t tiles = n_clips * p.tiles_t;
  const unsigned grid = (unsigned)std::min<int64_t>(tiles, sms);
  TIK_CUDA(launch_pdl(stem_block_kernel<3>, grid, kSbThreads, (size_t)kSbSmemBytes, s, p));
  return TIK_OK;
}

void stem_block_free(StemBlockPrepared* g) { delete g; }

}  // namespace tik
