// Fused graph convolution on tcgen05: adjacency aggregation + 1x1 channel GEMM + BN + ReLU in ONE kernel.
//
//   H[n,w,t,:] = relu( Wg' . ( sum_v A^[v,w] X[n,v,t,:] ) + b1[w,:] )          (K = 1 partition)
//
// Replaces the aggregate kernel + channel GEMM pair (gconv_origin.py:56-65 with the einsum moved in front of the
// conv, st_gcn_aaai18.py:178-179), i.e. two full activation passes through HBM per block.
//
// A tile is f <= 7 frames x 17 nodes of one clip (<= 119 rows, row r = v*f + t_local; f = gcn_fused_frames(T, Cin)), fetched
// as ONE 4-D TMA box (64 channels, f frames, 17 nodes, 1 clip) per 64-channel slab of the node-major activations.
//   MMA 1 (aggregation as a dense block-structured GEMM):   D1[128 x Cin] = Abd[128 x 128] . Xtile[128 x Cin]
//          Abd[(w,t),(v,t')] = A^[v,w] * delta(t,t'), bf16, K-major, resident in shared memory;
//          the X tile is used in place as the MN-major B operand (rows = K, channels contiguous).
//   mid pass: 8 warps move D1 TMEM -> registers -> bf16 -> the SAME shared-memory tile, now a K-major A operand.
//   MMA 2 (channel mix):                                      D2[128 x Cout] = Xagg[128 x Cin] . Wg'[Cout x Cin]^T
//   final pass: D2 + bias[node] -> ReLU -> bf16 -> swizzled staging -> 4-D TMA store (box clipped at the clip end).
// The dense Abd multiply costs 128/Cout of the channel GEMM in tensor time, far less than a round trip of the
// aggregated tensor through HBM.  Warp roles: warp 0 TMA producer, warp 1 MMA issuer, 8 mid-pass warps and 8
// final-pass warps (TMEM lane group x column half each), so tile i+1's mid pass overlaps tile i's final pass; D1 is
// double buffered in tensor memory, D2 too when 2*(Cin+Cout) <= 512 columns.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "tik_common.cuh"
#include "umma_ptx.cuh"

namespace tik {

constexpr int kGfGroupWarps = 8;                  // warps per epilogue group (mid pass / final pass)
constexpr int kGfThreads = 64 + 32 * 2 * kGfGroupWarps;
constexpr int kGfTile = 16384;                     // one 128-row x 64-channel swizzled slab
constexpr int kGfSmemBudget = 225 * 1024;
constexpr int kGfMaxBufs = 8;                      // input tiles in flight: the kernel is HBM-latency bound otherwise
constexpr int kGwMaxBufs = 16;                     // gcn_wide_kernel: 64-channel input slabs in flight

struct GcnFusedParams {
  CUtensorMap map_x, map_out, map_w;
  int32_t n_clips, T, V, ttg, tiles_t;   // ttg = frames per tile (gcn_fused_frames(T, cin) <= 7)
  int32_t xbufs;                          // input tiles in flight
  int32_t sbufs;                          // staging tiles (2: the store of tile i-1 may still be reading while tile i is staged)
  int32_t halves;                         // gcn_wide_kernel: CTAs per tile (output-channel split)
  int32_t xslab;                          // gcn_wide_kernel: bytes between input slabs of the ring
  const __nv_bfloat16* w;                 // gcn_wide_kernel: (Cout, Cin) weights, copied to tensor memory
  int32_t off_w, off_x, off_stage, off_bias, off_bar;
  const float* bias;                      // (V, COUT)
  const __nv_bfloat16* abd;               // (128, 128) row-major block-structured adjacency, copied to tensor memory
  int32_t relu;
  int32_t rev;                            // LaunchOpts: clips walked last to first
};

template <int CIN, int COUT>
__global__ void __launch_bounds__(kGfThreads, 1) gcn_fused_kernel(const __grid_constant__ GcnFusedParams p) {
  constexpr int KC1 = CIN / 64;                       // 64-channel slabs of the input
  constexpr int KC2 = COUT / 64;
  // tensor memory: [Abd 64 columns][D1 x ND1, CIN columns each; the bf16 Xagg of a tile overwrites its D1][D2 x ND2]
  constexpr int ND1 = (64 + 2 * CIN + COUT) <= 512 ? 2 : 1;
  constexpr int ND2 = (64 + ND1 * CIN + 2 * COUT) <= 512 ? 2 : 1;
  constexpr int TMEM_NEED = 64 + ND1 * CIN + ND2 * COUT;
  constexpr int TMEM_COLS = TMEM_NEED <= 128 ? 128 : (TMEM_NEED <= 256 ? 256 : 512);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; pointer arithmetic on the shared base keeps the address space (LDS / STS, not generic LD / ST)
  uint8_t* s_w = smem + p.off_w;                      // KC1 slabs of COUT rows x 128 B
  uint8_t* s_x = smem + p.off_x;                      // xbufs x KC1 slabs
  uint8_t* s_stage = smem + p.off_stage;              // KC2 slabs
  float* s_bias = reinterpret_cast<float*>(smem + p.off_bias);
  uint64_t* x_full = reinterpret_cast<uint64_t*>(smem + p.off_bar);   // [kGfMaxBufs]
  uint64_t* x_empty = x_full + kGfMaxBufs;            // [kGfMaxBufs]
  uint64_t* w_full = x_empty + kGfMaxBufs;
  uint64_t* d1_full = w_full + 1;                     // [2] aggregation MMA done -> mid group
  uint64_t* xagg_full = d1_full + 2;                  // [2] mid group rewrote the tile as bf16 Xagg -> channel MMA
  uint64_t* d2_full = xagg_full + 2;                  // [2] channel MMA done -> final group
  uint64_t* d2_empty = d2_full + 2;                   // [2] final group has read D2
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d2_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = p.n_clips * p.tiles_t;
  const int my_tiles = n_tiles > (int)blockIdx.x ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int rows_valid = p.ttg * p.V;                 // rows the TMA box fills (<= 128)
  const uint32_t x_bytes = (uint32_t)(KC1 * rows_valid * 128);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.map_x); tma_prefetch_desc(&p.map_out); tma_prefetch_desc(&p.map_w);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kGfMaxBufs; ++i) { mbar_init(&x_full[i], 1); mbar_init(&x_empty[i], 1); }
    mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&d1_full[i], 1); mbar_init(&xagg_full[i], kGfGroupWarps); mbar_init(&d2_full[i], 1); mbar_init(&d2_empty[i], kGfGroupWarps);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  // bias rows are padded by 4 floats: a warp holds rows of ~5 different nodes, and rows COUT*4 bytes apart would all
  // start in the same bank (measured: 36 % of the shared-memory wavefronts were bank conflicts)
  for (int i = threadIdx.x; i < p.V * COUT; i += kGfThreads) s_bias[(i / COUT) * (COUT + 4) + (i % COUT)] = __ldg(p.bias + i);
  // rows the TMA box never writes must not hold NaN bit patterns (they meet zero columns of Abd in MMA 1)
  {
    const int pad_rows = 128 - rows_valid;
    const int total16 = p.xbufs * KC1 * pad_rows * 8;
    for (int i = threadIdx.x; i < total16; i += kGfThreads) {
      const int piece = i & 7, rr = (i >> 3) % pad_rows, slab = (i >> 3) / pad_rows;
      *reinterpret_cast<uint4*>(s_x + (size_t)slab * kGfTile + (size_t)(rows_valid + rr) * 128 + piece * 16) = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_abd = tmem_base, tmem_d1 = tmem_base + 64, tmem_d2 = tmem_base + 64 + ND1 * CIN;
  // ---- block-structured adjacency -> tensor memory (once per CTA): the A operand of every aggregation MMA
  if (warp >= 2 && warp < 6) {
    const int r = (warp & 3) * 32 + lane;
    const uint4* arow = reinterpret_cast<const uint4*>(p.abd + (size_t)r * 128);
    uint4 v[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = __ldg(arow + u);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const uint32_t w8[8] = {v[2 * u].x, v[2 * u].y, v[2 * u].z, v[2 * u].w, v[2 * u + 1].x, v[2 * u + 1].y, v[2 * u + 1].z, v[2 * u + 1].w};
      tmem_st8(tmem_abd + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(8 * u), w8);
    }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();                                               // adjacency / weights / bias are constants; X comes from the previous kernel

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_expect_tx(w_full, (uint32_t)(KC1 * COUT * 128));
      for (int kc = 0; kc < KC1; ++kc) tma_load_2d(s_w + (size_t)kc * COUT * 128, &p.map_w, w_full, kc * 64, 0);
      int b = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int nf = tile / p.tiles_t, tt = tile - nf * p.tiles_t;
        const int n = p.rev ? p.n_clips - 1 - nf : nf;
        const int t0 = min(tt * p.ttg, p.T - p.ttg);          // the last tile of a clip is shifted back, never out of range
        mbar_wait(&x_empty[b], phase ^ 1);
        mbar_expect_tx(&x_full[b], x_bytes);
        for (int kc = 0; kc < KC1; ++kc)
          tma_load_4d(s_x + ((size_t)b * KC1 + kc) * kGfTile, &p.map_x, &x_full[b], kc * 64, t0, 0, n);
        if (++b == p.xbufs) { b = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // Warp-uniform loop, lane 0 issues.  The aggregation MMA of tile i+1 goes out before the channel MMA of tile i
    // (D1 is double buffered), so the mid group can start on tile i+1 while the final group drains tile i.
    constexpr uint32_t idesc1 = make_idesc_bf16(128, CIN) | (1u << 16);   // B operand MN-major
    constexpr uint32_t idesc2 = make_idesc_bf16(128, COUT);
    const bool leader = lane == 0;
    mbar_wait(w_full, 0);
    const uint32_t w_u32 = smem_u32(s_w), x_u32 = smem_u32(s_x);
    // MMA 1: D1 = Abd (tensor memory) . Xtile (shared memory, MN-major B); the X buffer is free as soon as it has run
    auto issue_mma1 = [&](uint32_t xb, int s1, int buf) {
      if (leader) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const uint64_t db = make_smem_desc_mnmajor_sw128(xb + (uint32_t)k * 2048u, (uint32_t)kGfTile);
          umma_bf16_ts(tmem_d1 + (uint32_t)(s1 * CIN), tmem_abd + (uint32_t)(8 * k), db, idesc1, k != 0 ? 1u : 0u);
        }
        umma_commit(&d1_full[s1]);
        umma_commit(&x_empty[buf]);
      }
      __syncwarp();
    };
    int b = 0; uint32_t phase = 0;
    if (my_tiles > 0) {
      mbar_wait(&x_full[0], 0);
      tc_fence_after();
      issue_mma1(x_u32, 0, 0);
    }
    // With two D1 buffers and two X buffers the aggregation MMA of tile it+1 goes out before the channel MMA of tile
    // it, so the mid group works on tile it+1 while the final group drains tile it.
    const bool early = ND1 == 2 && p.xbufs >= 2;
    for (int it = 0; it < my_tiles; ++it) {
      const int s1 = ND1 == 2 ? (it & 1) : 0;
      const int s2 = ND2 == 2 ? (it & 1) : 0;
      int nb = b + 1; uint32_t nphase = phase;
      if (nb == p.xbufs) { nb = 0; nphase ^= 1; }
      if (early && it + 1 < my_tiles) {
        mbar_wait(&x_full[nb], nphase);
        tc_fence_after();
        issue_mma1(x_u32 + (uint32_t)nb * (uint32_t)(KC1 * kGfTile), s1 ^ 1, nb);
      }
      // ---- MMA 2: D2 = Xagg (tensor memory, written over D1 by the mid group) . Wg^T (shared memory)
      mbar_wait(&xagg_full[it & 1], (uint32_t)((it >> 1) & 1));
      mbar_wait(&d2_empty[s2], (uint32_t)(((ND2 == 2 ? (it >> 1) : it) & 1) ^ 1));   // that accumulator has been read
      tc_fence_after();
      if (leader) {
#pragma unroll
        for (int kc = 0; kc < KC1; ++kc) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t db = make_smem_desc_kmajor_sw128(w_u32 + (uint32_t)kc * (COUT * 128) + (uint32_t)k * 32u);
            // channels c0 = kc*64 + k*16 live at column half*(CIN/2) + (c0 - half*(CIN/2)) / 2 of this tile's D1 (mid group)
            constexpr int HC = CIN / 2;
            const int c0 = kc * 64 + k * 16;
            const int xcol = (c0 / HC) * HC + (c0 % HC) / 2;
            umma_bf16_ts(tmem_d2 + (uint32_t)(s2 * COUT), tmem_d1 + (uint32_t)(s1 * CIN + xcol), db, idesc2, (kc | k) != 0 ? 1u : 0u);
          }
        }
        umma_commit(&d2_full[s2]);
      }
      __syncwarp();
      if (!early && it + 1 < my_tiles) {                     // D1 / Xagg of this tile is dead once MMA 2 above has run (in order)
        mbar_wait(&x_full[nb], nphase);
        tc_fence_after();
        issue_mma1(x_u32 + (uint32_t)nb * (uint32_t)(KC1 * kGfTile), ND1 == 2 ? (s1 ^ 1) : 0, nb);
      }
      b = nb; phase = nphase;
    }
  } else if (warp < 2 + kGfGroupWarps) {
    // ===================== mid group (8 warps): D1 (fp32) -> Xagg (bf16 pairs), in place in tensor memory =====================
    // Xagg is the A operand of MMA 2 (TS mode): it never touches shared memory.  Thread = tile row x column half; each
    // half packs into the first half of ITS OWN source columns (channels [h*CW1, +CW1) -> columns h*CW1 + [0, CW1/2)),
    // so no thread overwrites data another thread still has to load.
    constexpr int CW1 = CIN / 2;
    const int lane_grp = warp & 3;
    const int half = (warp - 2) >> 2;
    const uint32_t lane_off = (uint32_t)(lane_grp * 32) << 16;
    for (int it = 0; it < my_tiles; ++it) {
      const int s1 = ND1 == 2 ? (it & 1) : 0;
      mbar_wait(&d1_full[s1], (uint32_t)((ND1 == 2 ? (it >> 1) : it) & 1));
      tc_fence_after();
      uint32_t a[CW1];
#pragma unroll
      for (int i = 0; i < CW1 / 16; ++i) tmem_ld16(tmem_d1 + lane_off + (uint32_t)(s1 * CIN + half * CW1 + 16 * i), a + 16 * i);
      tmem_ld_wait();
#pragma unroll
      for (int q = 0; q < CW1 / 16; ++q) {                   // 16 fp32 columns -> 8 packed columns per store
        uint32_t w8[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) w8[e] = pack_bf16x2(__uint_as_float(a[16 * q + 2 * e]), __uint_as_float(a[16 * q + 2 * e + 1]));
        tmem_st8(tmem_d1 + lane_off + (uint32_t)(s1 * CIN + half * CW1 + 8 * q), w8);   // inside this thread's own source columns
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&xagg_full[it & 1]);
    }
  } else {
    // ===================== final group (8 warps): D2 + bias -> ReLU -> bf16 -> staging -> TMA store =====================
    constexpr int CW2 = COUT / 2;                            // columns per thread
    constexpr int SUB = CW2 > 64 ? 64 : CW2;                 // columns per register pass
    const int lane_grp = warp & 3;
    const int half = (warp - 2 - kGfGroupWarps) >> 2;
    const int r = lane_grp * 32 + lane;
    const int node = r / p.ttg;                              // tile row r = node * ttg + t_local
    const float* bias = s_bias + (node < p.V ? node : 0) * (COUT + 4) + half * CW2;
    const uint32_t lane_off = (uint32_t)(lane_grp * 32) << 16;
    const bool issuer = threadIdx.x == 32 * (2 + kGfGroupWarps);
    for (int it = 0; it < my_tiles; ++it) {
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const int nf = tile / p.tiles_t, tt = tile - nf * p.tiles_t;
      const int n = p.rev ? p.n_clips - 1 - nf : nf;
      const int t0 = min(tt * p.ttg, p.T - p.ttg);
      const int s2 = ND2 == 2 ? (it & 1) : 0;
      uint8_t* stage = s_stage + (size_t)((p.sbufs == 2) ? (it & 1) : 0) * (KC2 * kGfTile);
      if (issuer) {                                          // the store that last read this staging tile has finished reading it
        if (p.sbufs == 2) tma_store_wait_read1(); else tma_store_wait_read0();
      }
      mbar_wait(&d2_full[s2], (uint32_t)((ND2 == 2 ? (it >> 1) : it) & 1));
      tc_fence_after();
#pragma unroll
      for (int sub = 0; sub < CW2 / SUB; ++sub) {
        uint32_t a[SUB];
#pragma unroll
        for (int i = 0; i < SUB / 16; ++i)
          tmem_ld16(tmem_d2 + lane_off + (uint32_t)(s2 * COUT + half * CW2 + sub * SUB + 16 * i), a + 16 * i);
        tmem_ld_wait();
        if (sub == CW2 / SUB - 1) {                          // accumulator fully in registers: hand it back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&d2_empty[s2]);
        }
        if (sub == 0) named_bar_sync(1, 32 * kGfGroupWarps); // staging tile free (issuer passed wait_read)
#pragma unroll
        for (int q = 0; q < SUB / 8; ++q) {
          const float4 b0 = *reinterpret_cast<const float4*>(bias + sub * SUB + 8 * q);
          const float4 b1 = *reinterpret_cast<const float4*>(bias + sub * SUB + 8 * q + 4);
          const float v0 = __uint_as_float(a[8 * q + 0]) + b0.x, v1 = __uint_as_float(a[8 * q + 1]) + b0.y;
          const float v2 = __uint_as_float(a[8 * q + 2]) + b0.z, v3 = __uint_as_float(a[8 * q + 3]) + b0.w;
          const float v4 = __uint_as_float(a[8 * q + 4]) + b1.x, v5 = __uint_as_float(a[8 * q + 5]) + b1.y;
          const float v6 = __uint_as_float(a[8 * q + 6]) + b1.z, v7 = __uint_as_float(a[8 * q + 7]) + b1.w;
          uint4 u;
          if (p.relu) { u.x = pack_bf16x2_relu(v0, v1); u.y = pack_bf16x2_relu(v2, v3); u.z = pack_bf16x2_relu(v4, v5); u.w = pack_bf16x2_relu(v6, v7); }
          else { u.x = pack_bf16x2(v0, v1); u.y = pack_bf16x2(v2, v3); u.z = pack_bf16x2(v4, v5); u.w = pack_bf16x2(v6, v7); }
          const int col = half * CW2 + sub * SUB + 8 * q;
          const int j = (col & 63) >> 3;
          *reinterpret_cast<uint4*>(stage + (size_t)(col >> 6) * kGfTile + (size_t)r * 128 + ((j ^ (r & 7)) << 4)) = u;
        }
      }
      fence_proxy_async_smem();
      named_bar_sync(2, 32 * kGfGroupWarps);
      if (issuer) {
        for (int c = 0; c < KC2; ++c) tma_store_4d(&p.map_out, stage + (size_t)c * kGfTile, c * 64, t0, 0, n);
        tma_store_commit();
      }
    }
    if (issuer) tma_store_wait0();
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ 64-channel inputs: two tiles per pass
// At Cin = 64 a tile is only 16 KB and the single MMA-issuing thread (8 aggregation MMAs of N = 64, ~65 cycles each, plus
// the barrier hand-offs) bounds the kernel well above its HBM time.  Two tiles that share the adjacency are therefore
// aggregated by ONE set of N = 128 MMAs -- their X boxes sit in adjacent 16 KB slabs, exactly the layout of a
// 128-channel tile -- and only the channel GEMM runs per tile (its A operand is that tile's half of the TMEM-resident
// aggregate).  Half the aggregation MMAs, half the hand-offs per tile.
template <int COUT>
__global__ void __launch_bounds__(kGfThreads, 1) gcn_fused_pair_kernel(const __grid_constant__ GcnFusedParams p) {
  constexpr int KC2 = COUT / 64;
  constexpr int ND1 = (64 + 2 * 128 + 2 * COUT) <= 512 ? 2 : 1;
  constexpr int ND2 = (64 + ND1 * 128 + 4 * COUT) <= 512 ? 2 : 1;
  constexpr int TMEM_NEED = 64 + ND1 * 128 + ND2 * 2 * COUT;
  constexpr int TMEM_COLS = TMEM_NEED <= 256 ? 256 : 512;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; pointer arithmetic on the shared base keeps the address space (LDS / STS, not generic LD / ST)
  uint8_t* s_w = smem + p.off_w;                      // COUT rows x 128 B
  uint8_t* s_x = smem + p.off_x;                      // xbufs stages x 2 slabs (tile A, tile B)
  uint8_t* s_stage = smem + p.off_stage;              // 2 staging tiles (A, B) of KC2 slabs
  float* s_bias = reinterpret_cast<float*>(smem + p.off_bias);
  uint64_t* x_full = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* x_empty = x_full + kGfMaxBufs;
  uint64_t* w_full = x_empty + kGfMaxBufs;
  uint64_t* d1_full = w_full + 1;
  uint64_t* xagg_full = d1_full + 2;
  uint64_t* d2_full = xagg_full + 2;
  uint64_t* d2_empty = d2_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d2_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = p.n_clips * p.tiles_t;
  const int n_pairs = (n_tiles + 1) / 2;
  const int my_pairs = n_pairs > (int)blockIdx.x ? (n_pairs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int rows_valid = p.ttg * p.V;
  const uint32_t x_bytes = (uint32_t)(rows_valid * 128);

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.map_x); tma_prefetch_desc(&p.map_out); tma_prefetch_desc(&p.map_w); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kGfMaxBufs; ++i) { mbar_init(&x_full[i], 1); mbar_init(&x_empty[i], 1); }
    mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&d1_full[i], 1); mbar_init(&xagg_full[i], kGfGroupWarps); mbar_init(&d2_full[i], 1); mbar_init(&d2_empty[i], kGfGroupWarps);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  for (int i = threadIdx.x; i < p.V * COUT; i += kGfThreads) s_bias[(i / COUT) * (COUT + 4) + (i % COUT)] = __ldg(p.bias + i);
  {
    const int pad_rows = 128 - rows_valid;
    const int total16 = p.xbufs * 2 * pad_rows * 8;
    for (int i = threadIdx.x; i < total16; i += kGfThreads) {
      const int piece = i & 7, rr = (i >> 3) % pad_rows, slab = (i >> 3) / pad_rows;
      *reinterpret_cast<uint4*>(s_x + (size_t)slab * kGfTile + (size_t)(rows_valid + rr) * 128 + piece * 16) = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_abd = tmem_base, tmem_d1 = tmem_base + 64, tmem_d2 = tmem_base + 64 + ND1 * 128;
  if (warp >= 2 && warp < 6) {
    const int r = (warp & 3) * 32 + lane;
    const uint4* arow = reinterpret_cast<const uint4*>(p.abd + (size_t)r * 128);
    uint4 v[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = __ldg(arow + u);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const uint32_t w8[8] = {v[2 * u].x, v[2 * u].y, v[2 * u].z, v[2 * u].w, v[2 * u + 1].x, v[2 * u + 1].y, v[2 * u + 1].z, v[2 * u + 1].w};
      tmem_st8(tmem_abd + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(8 * u), w8);
    }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();                                               // adjacency / weights / bias are constants; X comes from the previous kernel

  // tile coordinates of pair `it`, slot h (a trailing odd tile is loaded twice and stored once)
  auto tile_of = [&](int it, int h, int& n, int& t0, bool& valid) {
    int tile = 2 * ((int)blockIdx.x + it * (int)gridDim.x) + h;
    valid = tile < n_tiles;
    if (!valid) tile = n_tiles - 1;
    n = tile / p.tiles_t;
    const int tt = tile - n * p.tiles_t;
    t0 = min(tt * p.ttg, p.T - p.ttg);
    if (p.rev) n = p.n_clips - 1 - n;
  };

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_expect_tx(w_full, (uint32_t)(COUT * 128));
      tma_load_2d(s_w, &p.map_w, w_full, 0, 0);
      int b = 0; uint32_t phase = 0;
      for (int it = 0; it < my_pairs; ++it) {
        mbar_wait(&x_empty[b], phase ^ 1);
        mbar_expect_tx(&x_full[b], 2 * x_bytes);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          int n, t0; bool valid;
          tile_of(it, h, n, t0, valid);
          tma_load_4d(s_x + ((size_t)b * 2 + h) * kGfTile, &p.map_x, &x_full[b], 0, t0, 0, n);
        }
        if (++b == p.xbufs) { b = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc1 = make_idesc_bf16(128, 128) | (1u << 16);   // both tiles at once; B operand MN-major
    constexpr uint32_t idesc2 = make_idesc_bf16(128, COUT);
    const bool leader = lane == 0;
    mbar_wait(w_full, 0);
    const uint32_t w_u32 = smem_u32(s_w), x_u32 = smem_u32(s_x);
    auto issue_mma1 = [&](uint32_t xb, int s1, int buf) {
      if (leader) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const uint64_t db = make_smem_desc_mnmajor_sw128(xb + (uint32_t)k * 2048u, (uint32_t)kGfTile);
          umma_bf16_ts(tmem_d1 + (uint32_t)(s1 * 128), tmem_abd + (uint32_t)(8 * k), db, idesc1, k != 0 ? 1u : 0u);
        }
        umma_commit(&d1_full[s1]);
        umma_commit(&x_empty[buf]);
      }
      __syncwarp();
    };
    int b = 0; uint32_t phase = 0;
    if (my_pairs > 0) {
      mbar_wait(&x_full[0], 0);
      tc_fence_after();
      issue_mma1(x_u32, 0, 0);
    }
    const bool early = ND1 == 2 && p.xbufs >= 2;
    for (int it = 0; it < my_pairs; ++it) {
      const int s1 = ND1 == 2 ? (it & 1) : 0;
      const int s2 = ND2 == 2 ? (it & 1) : 0;
      int nb = b + 1; uint32_t nphase = phase;
      if (nb == p.xbufs) { nb = 0; nphase ^= 1; }
      if (early && it + 1 < my_pairs) {
        mbar_wait(&x_full[nb], nphase);
        tc_fence_after();
        issue_mma1(x_u32 + (uint32_t)nb * (uint32_t)(2 * kGfTile), s1 ^ 1, nb);
      }
      mbar_wait(&xagg_full[it & 1], (uint32_t)((it >> 1) & 1));
      mbar_wait(&d2_empty[s2], (uint32_t)(((ND2 == 2 ? (it >> 1) : it) & 1) ^ 1));
      tc_fence_after();
      if (leader) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {                        // tile h: its 64 aggregated channels are bf16 pairs at D1 columns h*64 + [0, 32)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t db = make_smem_desc_kmajor_sw128(w_u32 + (uint32_t)k * 32u);
            umma_bf16_ts(tmem_d2 + (uint32_t)(s2 * 2 * COUT + h * COUT), tmem_d1 + (uint32_t)(s1 * 128 + h * 64 + k * 8), db, idesc2, k != 0 ? 1u : 0u);
          }
        }
        umma_commit(&d2_full[s2]);
      }
      __syncwarp();
      if (!early && it + 1 < my_pairs) {
        mbar_wait(&x_full[nb], nphase);
        tc_fence_after();
        issue_mma1(x_u32 + (uint32_t)nb * (uint32_t)(2 * kGfTile), ND1 == 2 ? (s1 ^ 1) : 0, nb);
      }
      b = nb; phase = nphase;
    }
  } else if (warp < 2 + kGfGroupWarps) {
    // ===================== mid group: D1 (fp32, both tiles) -> bf16 pairs in place (column half = tile) =====================
    const int lane_grp = warp & 3;
    const int half = (warp - 2) >> 2;
    const uint32_t lane_off = (uint32_t)(lane_grp * 32) << 16;
    for (int it = 0; it < my_pairs; ++it) {
      const int s1 = ND1 == 2 ? (it & 1) : 0;
      mbar_wait(&d1_full[s1], (uint32_t)((ND1 == 2 ? (it >> 1) : it) & 1));
      tc_fence_after();
      uint32_t a[64];
#pragma unroll
      for (int i = 0; i < 4; ++i) tmem_ld16(tmem_d1 + lane_off + (uint32_t)(s1 * 128 + half * 64 + 16 * i), a + 16 * i);
      tmem_ld_wait();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t w8[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) w8[e] = pack_bf16x2(__uint_as_float(a[16 * q + 2 * e]), __uint_as_float(a[16 * q + 2 * e + 1]));
        tmem_st8(tmem_d1 + lane_off + (uint32_t)(s1 * 128 + half * 64 + 8 * q), w8);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&xagg_full[it & 1]);
    }
  } else {
    // ===================== final group: both tiles' D2 + bias -> ReLU -> bf16 -> staging A / B -> TMA stores =====================
    constexpr int CW2 = COUT / 2;
    const int lane_grp = warp & 3;
    const int half = (warp - 2 - kGfGroupWarps) >> 2;
    const int r = lane_grp * 32 + lane;
    const int node = r / p.ttg;
    const float* bias = s_bias + (node < p.V ? node : 0) * (COUT + 4) + half * CW2;
    const uint32_t lane_off = (uint32_t)(lane_grp * 32) << 16;
    const bool issuer = threadIdx.x == 32 * (2 + kGfGroupWarps);
    for (int it = 0; it < my_pairs; ++it) {
      const int s2 = ND2 == 2 ? (it & 1) : 0;
      if (issuer) tma_store_wait_read0();                    // both staging tiles of the previous pair have been read
      mbar_wait(&d2_full[s2], (uint32_t)((ND2 == 2 ? (it >> 1) : it) & 1));
      tc_fence_after();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t a[CW2];
#pragma unroll
        for (int i = 0; i < CW2 / 16; ++i)
          tmem_ld16(tmem_d2 + lane_off + (uint32_t)(s2 * 2 * COUT + h * COUT + half * CW2 + 16 * i), a + 16 * i);
        tmem_ld_wait();
        if (h == 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&d2_empty[s2]);
        }
        if (h == 0) named_bar_sync(1, 32 * kGfGroupWarps);   // staging tiles free (issuer passed wait_read)
        uint8_t* stage = s_stage + (size_t)h * (KC2 * kGfTile);
#pragma unroll
        for (int q = 0; q < CW2 / 8; ++q) {
          const float4 b0 = *reinterpret_cast<const float4*>(bias + 8 * q);
          const float4 b1 = *reinterpret_cast<const float4*>(bias + 8 * q + 4);
          const float v0 = __uint_as_float(a[8 * q + 0]) + b0.x, v1 = __uint_as_float(a[8 * q + 1]) + b0.y;
          const float v2 = __uint_as_float(a[8 * q + 2]) + b0.z, v3 = __uint_as_float(a[8 * q + 3]) + b0.w;
          const float v4 = __uint_as_float(a[8 * q + 4]) + b1.x, v5 = __uint_as_float(a[8 * q + 5]) + b1.y;
          const float v6 = __uint_as_float(a[8 * q + 6]) + b1.z, v7 = __uint_as_float(a[8 * q + 7]) + b1.w;
          uint4 u;
          if (p.relu) { u.x = pack_bf16x2_relu(v0, v1); u.y = pack_bf16x2_relu(v2, v3); u.z = pack_bf16x2_relu(v4, v5); u.w = pack_bf16x2_relu(v6, v7); }
          else { u.x = pack_bf16x2(v0, v1); u.y = pack_bf16x2(v2, v3); u.z = pack_bf16x2(v4, v5); u.w = pack_bf16x2(v6, v7); }
          const int col = half * CW2 + 8 * q;
          const int j = (col & 63) >> 3;
          *reinterpret_cast<uint4*>(stage + (size_t)(col >> 6) * kGfTile + (size_t)r * 128 + ((j ^ (r & 7)) << 4)) = u;
        }
      }
      fence_proxy_async_smem();
      named_bar_sync(2, 32 * kGfGroupWarps);
      if (issuer) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          int n, t0; bool valid;
          tile_of(it, h, n, t0, valid);
          if (valid)
            for (int c = 0; c < KC2; ++c) tma_store_4d(&p.map_out, s_stage + (size_t)h * (KC2 * kGfTile) + (size_t)c * kGfTile, c * 64, t0, 0, n);
        }
        tma_store_commit();
      }
    }
    if (issuer) tma_store_wait0();
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ wide inputs (Cin = 256): weights in tensor memory
// A 256-channel tile (64 KB) plus its 256 x 256 weights (128 KB) and a staging tile do not fit one SM, so the last block ran
// as two aggregation-only launches + a plain channel GEMM (three activation passes, 274 us at B = 4096).  This kernel does
// it in one pass, TRANSPOSED: output channels on the 128 accumulator lanes, tile rows (node, frame) on the columns.
//   * the weights are the TMEM-resident A operand (TS mode): 128 output channels x 256 input channels = 128 columns,
//     loaded once per CTA; the output channels are split over NH = Cout / 128 CTAs (CTA parity = channel half; adjacent
//     CTAs work on the same tile at the same time, the second reader hits L2);
//   * MMA a: Z^T[128 ch x N] = Wg'[128 x 256] . Xtile^T -- aggregation and channel mix commute, and with Cin = Cout the
//     channel GEMM first costs nothing extra; the X slabs are the B operand exactly as TMA delivers them (rows x 64
//     channels, K-major), N = tile rows rounded up to 16 (80 for the 68 rows of a 4-frame tile, not 128);
//   * mid: Z^T fp32 -> bf16 pairs in place in tensor memory (it is the A operand of the next MMA: no shared memory);
//   * MMA b: D^T[128 ch x N] = Z^T . Abd^T, Abd (128 x 128, K-major) resident in shared memory;
//   * final: D^T + bias[node][ch] -> ReLU -> bf16 -> transposed into the row-major staging tile -> 4-D TMA store.
// Shared-memory traffic per tile drops from ~300 KB (SS-mode 128 x 128 x 16 MMAs read 8 KB each; Z went through shared
// memory) to ~150 KB, the MMA work from 1344 to 840 cycles; what is left is the HBM time of one read + one write.
// History: aggregation first in 64-channel quarters (four MMA -> register pass -> MMA hand-offs per tile): 348 us;
// channel GEMM first in SS mode with Z staged through shared memory: 171 us (shared-memory bandwidth bound).
// Tiles hold at most 5 frames here (N <= 96: two Z^T and two D^T accumulators of 96 columns beside the 128 weight columns).
constexpr int kGwAcc = 96;                          // tensor-memory columns per accumulator
template <int NQ>
__global__ void __launch_bounds__(kGfThreads, 1) gcn_wide_kernel(const __grid_constant__ GcnFusedParams p) {
  constexpr int CO = 128;                             // output channels per CTA = accumulator lanes
  constexpr int TMEM_COLS = 512;                      // [W 128][Z^T 2 x 96][D^T 2 x 96]
  static_assert(NQ * 32 == 128, "256 input channels as bf16 pairs fill 128 columns");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_abd = smem + p.off_w;                    // 2 slabs of 128 rows x 64 K (the map_w box)
  uint8_t* s_x = smem + p.off_x;                      // xbufs slabs (64 channels of one tile each), p.xslab bytes apart
  uint8_t* s_stage = smem + p.off_stage;              // 2 staging tiles of 2 slabs of 16 * n_groups rows (stores are unconditional)
  float* s_bias = reinterpret_cast<float*>(smem + p.off_bias);   // [node][128]
  uint64_t* x_full = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* x_empty = x_full + kGwMaxBufs;
  uint64_t* abd_full = x_empty + kGwMaxBufs;
  uint64_t* da_full = abd_full + 1;                   // [2] channel GEMM done -> mid group
  uint64_t* z_full = da_full + 2;                     // [2] mid group packed Z^T -> aggregation MMA
  uint64_t* d2_full = z_full + 2;                     // [2] aggregation done -> final group
  uint64_t* d2_empty = d2_full + 2;                   // [2] final group has read D^T
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d2_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int NH = p.halves;                            // CTAs per tile (gridDim.x is a multiple of it)
  const int half_out = (int)blockIdx.x % NH;
  const int first_tile = (int)blockIdx.x / NH, tile_step = (int)gridDim.x / NH;
  const int n_tiles = p.n_clips * p.tiles_t;
  const int my_tiles = n_tiles > first_tile ? (n_tiles - first_tile + tile_step - 1) / tile_step : 0;
  const int rows_valid = p.ttg * p.V;
  const int n_groups = (rows_valid + 15) >> 4;        // 16-row groups = K-steps of the aggregation; N = 16 * n_groups <= 96
  const uint32_t x_bytes = (uint32_t)(rows_valid * 128);

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.map_x); tma_prefetch_desc(&p.map_out); tma_prefetch_desc(&p.map_w); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kGwMaxBufs; ++i) { mbar_init(&x_full[i], 1); mbar_init(&x_empty[i], 1); }
    mbar_init(abd_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&da_full[i], 1); mbar_init(&z_full[i], kGfGroupWarps); mbar_init(&d2_full[i], 1); mbar_init(&d2_empty[i], kGfGroupWarps);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  for (int i = threadIdx.x; i < p.V * CO; i += kGfThreads)
    s_bias[i] = __ldg(p.bias + (size_t)(i / CO) * (CO * NH) + half_out * CO + (i % CO));
  {
    // Input slabs are only as long as a tile has rows (rounded up to the 8-row swizzle atom), so that many are in flight.
    // The MMA reads N = 16 * n_groups rows, i.e. up to 15 rows past a slab's end into the next slab (for the last one: into
    // the staging tiles); those become columns of Z^T that only meet zero columns of Abd, so they merely have to be FINITE:
    // bf16 activations are, and the ring and the staging tiles are zeroed once here (a slab that is never filled, or not
    // yet, holds whatever the previous kernel left).
    const int n16 = p.xbufs * (p.xslab >> 4) + 4 * n_groups * 128;   // ring + 2 staging tiles of 2 slabs, contiguous
    for (int i = threadIdx.x; i < n16; i += kGfThreads) reinterpret_cast<uint4*>(s_x)[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_w = tmem_base, tmem_z = tmem_base + 128, tmem_d2 = tmem_base + 128 + 2 * kGwAcc;
  // ---- this CTA's 128 x 256 weight slice -> tensor memory: lane = output channel, column j = input channels 2j, 2j+1
  if (warp >= 2 && warp < 6) {
    const int c = (warp & 3) * 32 + lane;
    const uint4* wrow = reinterpret_cast<const uint4*>(p.w + (size_t)(half_out * CO + c) * (NQ * 64));
#pragma unroll
    for (int u = 0; u < NQ * 4; ++u) {                // 16 input channels = 8 columns per step
      const uint4 v0 = __ldg(wrow + 2 * u), v1 = __ldg(wrow + 2 * u + 1);
      const uint32_t w8[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
      tmem_st8(tmem_w + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(8 * u), w8);
    }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();

  auto tile_of = [&](int it, int& n, int& t0) {
    const int tile = first_tile + it * tile_step;
    n = tile / p.tiles_t;
    t0 = min((tile - n * p.tiles_t) * p.ttg, p.T - p.ttg);
    if (p.rev) n = p.n_clips - 1 - n;
  };

  if (warp == 0) {
    // ===================== TMA producer: Abd once, then one 64-channel slab per step =====================
    if (lane == 0) {
      mbar_expect_tx(abd_full, 2u * kGfTile);
      tma_load_2d(s_abd, &p.map_w, abd_full, 0, 0);
      tma_load_2d(s_abd + kGfTile, &p.map_w, abd_full, 64, 0);
      int b = 0; uint32_t phase = 0;
      for (int it = 0; it < my_tiles; ++it) {
        int n, t0;
        tile_of(it, n, t0);
        for (int q = 0; q < NQ; ++q) {
          mbar_wait(&x_empty[b], phase ^ 1);
          mbar_expect_tx(&x_full[b], x_bytes);
          tma_load_4d(s_x + (size_t)b * p.xslab, &p.map_x, &x_full[b], q * 64, t0, 0, n);
          if (++b == p.xbufs) { b = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: the whole warp runs the loop, one elected lane issues (umma_*_w) =====================
    // With N <= 96 an MMA is <= 48 tensor cycles, so this role is bound by how fast it can issue.  Run under `if (lane ==
    // 0)` every tcgen05 instruction was wrapped in a uniformisation loop (~8 instructions; ~500 dependent scalar
    // instructions per tile: 2800 cycles per tile with the tensor pipe 31 % active and no barrier ever spinning).
    // Descriptors are one 64-bit add from two bases; ring indices are running counters.
    {
      const uint32_t idesc = make_idesc_bf16(128, 16 * n_groups);
      mbar_wait(abd_full, 0);
      // the start-address field (bits 0..13, 16-byte units) never overflows: shared-memory addresses are < 256 KB
      const uint64_t dx0 = make_smem_desc_kmajor_sw128(smem_u32(s_x));
      const uint64_t dabd0 = make_smem_desc_kmajor_sw128(smem_u32(s_abd));
      const uint32_t xstep = (uint32_t)(p.xslab >> 4);
      int b = 0; uint32_t xphase = 0;
      auto mma_a = [&](int s) {                        // Z^T = W . X^T into accumulator s (its last reader, MMA b of two tiles ago, was issued earlier)
        const uint32_t dcol = tmem_z + (uint32_t)(s * kGwAcc);
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          mbar_wait(&x_full[b], xphase);
          tc_fence_after();
          const uint64_t dx = dx0 + (uint64_t)((uint32_t)b * xstep);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ts_w(dcol, tmem_w + (uint32_t)(q * 32 + k * 8), dx + (uint64_t)(2 * k), idesc, (q | k) != 0 ? 1u : 0u);
          umma_commit_w(&x_empty[b]);
          if (++b == p.xbufs) { b = 0; xphase ^= 1; }
        }
        umma_commit_w(&da_full[s]);
      };
      if (my_tiles > 0) mma_a(0);
      for (int t = 0; t < my_tiles; ++t) {
        const int s = t & 1;
        const uint32_t par = (uint32_t)((t >> 1) & 1);
        if (t + 1 < my_tiles) mma_a(s ^ 1);
        mbar_wait(&z_full[s], par);
        mbar_wait(&d2_empty[s], par ^ 1);
        tc_fence_after();
        for (int j = 0; j < n_groups; ++j)             // rows 16j..16j+15 of the tile: Z^T columns 16j.. (packed into 8), Abd K-columns 16j..
          umma_bf16_ts_w(tmem_d2 + (uint32_t)(s * kGwAcc), tmem_z + (uint32_t)(s * kGwAcc + 16 * j),
                         dabd0 + (uint64_t)((j >> 2) * (kGfTile >> 4) + (j & 3) * 2), idesc, j != 0 ? 1u : 0u);
        umma_commit_w(&d2_full[s]);
      }
    }
  } else if (warp < 2 + kGfGroupWarps) {
    // ===================== mid group: Z^T fp32 -> bf16 pairs, in place (16 columns -> the first 8 of the same 16) =====================
    // Warp (lane group, half) takes the 16-column groups half, half + 2, half + 4 (N <= 96: at most three).
    const int lane_grp = warp & 3;
    const int half = (warp - 2) >> 2;
    const uint32_t lane_off = (uint32_t)(lane_grp * 32) << 16;
    for (int t = 0; t < my_tiles; ++t) {
      const int s = t & 1;
      const uint32_t col = tmem_z + lane_off + (uint32_t)(s * kGwAcc + 16 * half);
      mbar_wait(&da_full[s], (uint32_t)((t >> 1) & 1));
      tc_fence_after();
      uint32_t a[3][16];
#pragma unroll
      for (int i = 0; i < 3; ++i)
        if (half + 2 * i < n_groups) tmem_ld16(col + 32 * i, a[i]);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 3; ++i)
        if (half + 2 * i < n_groups) {
          uint32_t w8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) w8[e] = pack_bf16x2(__uint_as_float(a[i][2 * e]), __uint_as_float(a[i][2 * e + 1]));
          tmem_st8(col + 32 * i, w8);
        }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&z_full[s]);
    }
  } else {
    // ===================== final group: D^T + bias -> ReLU -> bf16 -> transposed staging -> TMA store =====================
    const int lane_grp = warp & 3;
    const int half = (warp - 2 - kGfGroupWarps) >> 2;
    const int c = lane_grp * 32 + lane;                // this thread's output channel (within the CTA's 128)
    const uint32_t lane_off = (uint32_t)(lane_grp * 32) << 16;
    const bool issuer = threadIdx.x == 32 * (2 + kGfGroupWarps);
    // Row n of a tile is always the same node, and this thread always the same channel: its bias values live in registers.
    float bias_r[3][16];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int row = 16 * (half + 2 * i) + j;
        bias_r[i][j] = row < rows_valid ? s_bias[(row / p.ttg) * CO + c] : 0.f;
      }
    // staging address of (row n, channel c): slab c/64, 128-byte rows, 16-byte chunks XOR-swizzled with the row (n & 7 = j & 7).
    // Slabs have 16 * n_groups rows, so every row of a group is stored without a bounds test (the TMA store reads the valid
    // ones); the eight swizzle variants are base registers, (group, row) is an immediate offset of the store.
    const bool relu = p.relu != 0;
    const uint32_t sslab = (uint32_t)n_groups * 2048u;
    const uint32_t c_off = smem_u32(s_stage) + (uint32_t)(c >> 6) * sslab + (uint32_t)(c & 7) * 2u + (uint32_t)(16 * half) * 128u;
    const uint32_t c_chunk = (uint32_t)((c & 63) >> 3);
    for (int t = 0; t < my_tiles; ++t) {
      int n, t0;
      tile_of(t, n, t0);
      const int s = t & 1;
      uint8_t* stage = s_stage + (size_t)s * (2 * sslab);
      uint32_t base8[8];
#pragma unroll
      for (int m = 0; m < 8; ++m) base8[m] = c_off + (uint32_t)s * (2u * sslab) + ((c_chunk ^ (uint32_t)m) << 4);
      if (issuer) tma_store_wait_read1();              // the store of tile t-2 has read this staging tile
      mbar_wait(&d2_full[s], (uint32_t)((t >> 1) & 1));
      tc_fence_after();
      const uint32_t col = tmem_d2 + lane_off + (uint32_t)(s * kGwAcc + 16 * half);
      named_bar_sync(1, 32 * kGfGroupWarps);           // the issuer has passed its wait: the staging tile is free
#pragma unroll
      for (int i = 0; i < 3; ++i)                      // one 16-row group at a time: 48 bias registers leave room for 16 accumulators
        if (half + 2 * i < n_groups) {
          uint32_t a[16];
          tmem_ld16(col + 32 * i, a);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float v = __uint_as_float(a[j]) + bias_r[i][j];
            v = relu ? fmaxf(v, 0.f) : v;
            const uint16_t h16 = __bfloat16_as_ushort(__float2bfloat16_rn(v));
            asm volatile("st.shared.b16 [%0], %1;" ::"r"(base8[j & 7] + (uint32_t)((32 * i + j) * 128)), "h"(h16) : "memory");
          }
        }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&d2_empty[s]);        // the accumulator has been read
      fence_proxy_async_smem();
      named_bar_sync(2, 32 * kGfGroupWarps);
      if (issuer) {
        for (int h = 0; h < 2; ++h) tma_store_4d(&p.map_out, stage + (size_t)h * sslab, half_out * CO + h * 64, t0, 0, n);
        tma_store_commit();
      }
    }
    if (issuer) tma_store_wait0();
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int encode_bf16_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides, const uint32_t* box) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* q = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess || !q) {
      set_error("cuTensorMapEncodeTiled not available from the driver");
      return TIK_ERR_CUDA;
    }
    fn = reinterpret_cast<EncodeTiledFn>(q);
  }
  const uint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (fused gcn) failed with CUresult %d", (int)r);
    return TIK_ERR_CUDA;
  }
  return TIK_OK;
}

struct GcnFusedPrepared {
  GcnFusedParams p;
  int cin, cout, smem_bytes;
  bool pair;                               // Cin = 64: two tiles per aggregation pass (gcn_fused_pair_kernel)
  bool wide;                               // Cin = 256: quarter-streamed inputs, output channels split over two CTAs (gcn_wide_kernel)
};
constexpr int kGwCo = 128;                 // output channels per CTA of the wide kernel

// Frames per tile: at most 7 (7 x 17 nodes = 119 of the 128 MMA rows); the 256-channel kernel keeps tile rows on the
// accumulator columns, at most 5 frames (85 rows -> N = 96).  Balanced over the tiles of a clip so that the last tile
// re-does as few frames as possible (T=16: 3 tiles of 6, not 7+7+shifted 7; T=8: 2 tiles of 4).
int gcn_fused_frames(int T, int cin) {
  const int max_frames = cin == 256 ? 5 : 7;
  const int tiles = (T + max_frames - 1) / max_frames;
  return (T + tiles - 1) / tiles;
}

bool gcn_fused_supported(int cin, int cout, int V, int K) {
  if (K != 1 || V * 7 > 128 || V < 1) return false;
  return (cin == 64 && (cout == 64 || cout == 128)) || (cin == 128 && (cout == 128 || cout == 256)) ||
         (cin == 256 && cout == 256);                                          // gcn_wide_kernel
}

int gcn_fused_prepare(const void* x, const void* abd, const void* w, const float* bias, void* out, int64_t n_clips, int T, int V,
                      int cin, int cout, int relu, GcnFusedPrepared** outp) {
  TIK_CHECK_ARG(gcn_fused_supported(cin, cout, V, 1), "fused gcn: unsupported shape cin=%d cout=%d V=%d", cin, cout, V);
  TIK_CHECK_ARG(x && abd && w && bias && out && n_clips > 0 && T > 0, "fused gcn: bad arguments");
  GcnFusedPrepared* g = new GcnFusedPrepared();
  GcnFusedParams& p = g->p;
  memset(&p, 0, sizeof(p));
  g->cin = cin; g->cout = cout;
  p.n_clips = (int32_t)n_clips; p.T = T; p.V = V;
  p.ttg = gcn_fused_frames(T, cin);
  p.tiles_t = (T + p.ttg - 1) / p.ttg;
  p.bias = bias; p.relu = relu; p.abd = reinterpret_cast<const __nv_bfloat16*>(abd);
  int rc = TIK_OK;
  {
    uint64_t dims[4] = {(uint64_t)cin, (uint64_t)T, (uint64_t)V, (uint64_t)n_clips};
    uint64_t strides[3] = {(uint64_t)cin * 2, (uint64_t)cin * 2 * T, (uint64_t)cin * 2 * T * V};
    uint32_t box[4] = {64, (uint32_t)p.ttg, (uint32_t)V, 1};
    rc = encode_bf16_map(&p.map_x, x, 4, dims, strides, box);
  }
  if (rc == TIK_OK) {
    uint64_t dims[4] = {(uint64_t)cout, (uint64_t)T, (uint64_t)V, (uint64_t)n_clips};
    uint64_t strides[3] = {(uint64_t)cout * 2, (uint64_t)cout * 2 * T, (uint64_t)cout * 2 * T * V};
    uint32_t box[4] = {64, (uint32_t)p.ttg, (uint32_t)V, 1};
    rc = encode_bf16_map(&p.map_out, out, 4, dims, strides, box);
  }
  if (rc == TIK_OK && cin == 256) {                        // wide kernel: weights go to tensor memory, the 2-D map fetches Abd
    uint64_t dims[2] = {128, 128};
    uint64_t strides[1] = {128 * 2};
    uint32_t box[2] = {64, 128};
    rc = encode_bf16_map(&p.map_w, abd, 2, dims, strides, box);
    p.w = reinterpret_cast<const __nv_bfloat16*>(w);
  } else if (rc == TIK_OK) {
    uint64_t dims[2] = {(uint64_t)cin, (uint64_t)cout};
    uint64_t strides[1] = {(uint64_t)cin * 2};
    uint32_t box[2] = {64, (uint32_t)cout};
    rc = encode_bf16_map(&p.map_w, w, 2, dims, strides, box);
  }
  if (rc != TIK_OK) { delete g; return rc; }
  g->wide = cin == 256;
  if (g->wide) {
    // Abd 32 KB + two staging tiles of two slabs + bias [node][128]; the rest is the ring of input slabs
    p.halves = cout / kGwCo;
    const int bias_bytes = (V * kGwCo * 4 + 1023) / 1024 * 1024;
    p.sbufs = 2;
    p.xslab = (p.ttg * V + 7) / 8 * 1024;
    const int sslab = (p.ttg * V + 15) / 16 * 2048;        // staging slab: rows rounded up to the 16-row groups
    const int fixed = 2 * kGfTile + 4 * sslab + bias_bytes + 512;
    p.xbufs = std::min((kGfSmemBudget - fixed) / p.xslab, kGwMaxBufs);
    if (const char* e = getenv("TIK_GCN_WIDE_XBUFS")) p.xbufs = std::max(1, std::min(p.xbufs, atoi(e)));
    p.off_w = 0;                           // Abd
    p.off_x = 2 * kGfTile;
    p.off_stage = p.off_x + p.xbufs * p.xslab;
    p.off_bias = p.off_stage + 4 * sslab;
    p.off_bar = p.off_bias + bias_bytes;
    g->smem_bytes = p.off_bar + 512 + 1024;
    g->pair = false;
    *outp = g;
    return TIK_OK;
  }
  const int kc1 = cin / 64, kc2 = cout / 64;
  const int w_bytes = kc1 * cout * 128;
  const int bias_bytes = (V * (cout + 4) * 4 + 1023) / 1024 * 1024;
  // 64 -> 128 would need 576 TMEM columns to keep D1 double buffered as a pair; single-buffered it is slower (360 vs 324 us)
  g->pair = cin == 64 && cout == 64;
  const int stage_tiles = g->pair ? 2 : 1;                // input tiles per ring stage
  // two staging tiles when at least three input stages still fit beside them (measured: input depth matters more);
  // the pair kernel always stages both of its tiles
  p.sbufs = 2;
  int fixed = w_bytes + p.sbufs * kc2 * kGfTile + bias_bytes + 256;
  if (!g->pair && (kGfSmemBudget - fixed) / (kc1 * kGfTile) < 3) {
    p.sbufs = 1;
    fixed = w_bytes + kc2 * kGfTile + bias_bytes + 256;
  }
  p.xbufs = (kGfSmemBudget - fixed) / (stage_tiles * kc1 * kGfTile);
  if (p.xbufs > kGfMaxBufs) p.xbufs = kGfMaxBufs;
  if (p.xbufs < 1) {
    delete g;
    set_error("fused gcn: shared memory plan does not fit");
    return TIK_ERR_UNSUPPORTED;
  }
  p.off_w = 0;
  p.off_x = p.off_w + (w_bytes + 1023) / 1024 * 1024;
  p.off_stage = p.off_x + p.xbufs * stage_tiles * kc1 * kGfTile;
  p.off_bias = p.off_stage + p.sbufs * kc2 * kGfTile;
  p.off_bar = p.off_bias + bias_bytes;
  g->smem_bytes = p.off_bar + 256 + 1024;
  *outp = g;
  return TIK_OK;
}

template <int CIN, int COUT>
static int gf_launch_variant(const GcnFusedPrepared* g, unsigned grid, cudaStream_t s) {
  static bool attr_done[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (!attr_done[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(gcn_fused_kernel<CIN, COUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGfSmemBudget + 2048));
    TIK_CUDA(cudaFuncSetAttribute(gcn_fused_kernel<CIN, COUT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr_done[dev & 63] = true;
  }
  TIK_CUDA(launch_pdl(gcn_fused_kernel<CIN, COUT>, grid, kGfThreads, (size_t)g->smem_bytes, s, g->p));
  return TIK_OK;
}

template <int COUT>
static int gf_launch_pair(const GcnFusedPrepared* g, unsigned grid, cudaStream_t s) {
  static bool attr_done[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (!attr_done[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(gcn_fused_pair_kernel<COUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGfSmemBudget + 2048));
    TIK_CUDA(cudaFuncSetAttribute(gcn_fused_pair_kernel<COUT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr_done[dev & 63] = true;
  }
  TIK_CUDA(launch_pdl(gcn_fused_pair_kernel<COUT>, grid, kGfThreads, (size_t)g->smem_bytes, s, g->p));
  return TIK_OK;
}

static int gf_launch_wide(const GcnFusedPrepared* g, unsigned grid, cudaStream_t s) {
  static bool attr_done[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (!attr_done[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(gcn_wide_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGfSmemBudget + 2048));
    TIK_CUDA(cudaFuncSetAttribute(gcn_wide_kernel<4>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr_done[dev & 63] = true;
  }
  TIK_CUDA(launch_pdl(gcn_wide_kernel<4>, grid, kGfThreads, (size_t)g->smem_bytes, s, g->p));
  return TIK_OK;
}

int gcn_fused_launch(GcnFusedPrepared* g, int64_t n_clips, cudaStream_t s) {
  GcnFusedParams& p = g->p;
  const int32_t cap = p.n_clips;
  if (n_clips <= 0) return TIK_OK;
  TIK_CHECK_ARG(n_clips <= cap, "fused gcn: n_clips exceeds the prepared capacity");
  const int32_t saved = p.n_clips;
  p.n_clips = (int32_t)n_clips;            // tiles only over the valid clips (tensor maps keep the full capacity)
  p.rev = launch_opts().rev;
  int sms = 148;
  { int dev = 0; if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); }
  const int64_t tiles = n_clips * p.tiles_t;
  const unsigned grid = (unsigned)std::min<int64_t>(g->pair ? (tiles + 1) / 2 : tiles, sms);
  int rc;
  if (g->wide) {                           // CTA parity = output-channel half: the grid is a multiple of the split
    const int64_t want = tiles * p.halves, cap_ctas = sms / p.halves * p.halves;
    rc = gf_launch_wide(g, (unsigned)std::min<int64_t>(want, cap_ctas), s);
  } else if (g->pair && g->cout == 64) rc = gf_launch_pair<64>(g, grid, s);
  else if (g->pair && g->cout == 128) rc = gf_launch_pair<128>(g, grid, s);
  else if (g->cin == 64 && g->cout == 128) rc = gf_launch_variant<64, 128>(g, grid, s);
  else if (g->cin == 128 && g->cout == 128) rc = gf_launch_variant<128, 128>(g, grid, s);
  else rc = gf_launch_variant<128, 256>(g, grid, s);
  p.n_clips = saved;
  return rc;
}

void gcn_fused_free(GcnFusedPrepared* g) { delete g; }

}  // namespace tik

extern "C" int tik_gcn_fused(const void* x_dev, const void* abd_dev, const void* w_dev, const float* bias_dev, void* out_dev,
                             int64_t N, int T, int V, int Cin, int Cout, int relu, void* stream) {
  using namespace tik;
  GcnFusedPrepared* g = nullptr;
  int rc = gcn_fused_prepare(x_dev, abd_dev, w_dev, bias_dev, out_dev, N, T, V, Cin, Cout, relu, &g);
  if (rc != TIK_OK) return rc;
  rc = gcn_fused_launch(g, N, (cudaStream_t)stream);
  gcn_fused_free(g);
  return rc;
}
