// bf16 implicit-GEMM on Blackwell tensor cores (tcgen05.mma + TMEM accumulators, TMA-fed), persistent.
//
//   out[row, :] = act( sum_slabs A_s[row_s, :] . W[:, slab]^T + bias + residual )
//
// A "row" is (row group nv = clip*V + node, frame t).  Because activations are node-major
// (NV, T, C), the rows a 128-row MMA tile needs from one slab form a 3-D box
// (64 channels, TT frames, VV row groups) of the source tensor, so every A operand -- including the
// time-shifted taps of the (kt x 1) temporal convolution, its stride-2 sub-sampling and its zero
// padding at clip ends -- is ONE cp.async.bulk.tensor load: the shift is the box start coordinate,
// the stride is the tensor map's elementStrides and the padding is TMA out-of-bounds zero fill.
// The box lands in shared memory in the 128-byte-swizzled K-major layout that the UMMA shared-memory
// descriptor consumes directly.
//
// Persistent kernel, one CTA per SM, static round-robin tile schedule.  Warp roles (640 threads):
//   warp 0     TMA producer: streams A chunks (and W chunks when the weights do not fit) through a ring whose stages
//              hold 1, 2 or 4 K chunks each (one barrier hand-off per stage), running ahead across tile boundaries;
//   warp 1     MMA issuer (warp-uniform loop, one lane issues): 4 x tcgen05.mma (M=128, N=BN, K=16) per 64-channel
//              chunk into one of two TMEM accumulators, tcgen05.commit frees ring stages / publishes the accumulator;
//   warps 2-17 epilogue (TMEM lane group x column quarter): tcgen05.ld up front, accumulator handed back at once,
//              bias / activation / bf16 -> 128B-swizzled staging tile, overlapped with the next tile's main loop;
//   warp 18    TMA-store warp: one cp.async.bulk.tensor store per 64-column slab, two staging tiles in flight.
// When (c_out x K_total) bf16 weights fit beside the ring they are loaded into shared memory once per CTA
// and stay resident for all its tiles (they are the larger half of the per-tile operand bytes otherwise).
//
// Serves: BN-folded 1x1 channel GEMM of ConvTemporalGraphical (gconv_origin.py:59) after the adjacency
// aggregation, the temporal convolution + residual + BN + ReLU of StGcnBlock (st_gcn_aaai18.py:177-214)
// and both Linear layers of the head (pose_trainer.py:89-92).
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "tik_common.cuh"
#include "umma_prepared.h"
#include "umma_ptx.cuh"

namespace tik {

constexpr int kTileM = 128;
constexpr int kChunkK = 64;                       // bf16 elements per K chunk = one 128 B swizzle row
constexpr int kABytes = kTileM * kChunkK * 2;     // 16 KB
constexpr int kEpiWarps = 16;                     // four warps per TMEM lane group, each takes a quarter of the columns
constexpr int kUmmaThreads = 64 + 32 * kEpiWarps + 32;   // + one TMA-store warp
constexpr int kMaxStages = 12;
constexpr int kSmemBudget = 225 * 1024;

struct UmmaParams {
  CUtensorMap map_a[TIK_MAX_SLABS];
  CUtensorMap map_w;
  CUtensorMap map_out;             // node-major output (c_out, t_out, nv) for the TMA-store epilogue
  int32_t tma_store, off_stage;    // epilogue stages the tile in swizzled smem and stores it with TMA
  int32_t stage_bufs;              // 1 or 2 staging tiles
  int32_t n_slabs;
  int32_t chunks[TIK_MAX_SLABS];   // c_s / 64
  int32_t t_mul[TIK_MAX_SLABS];
  int32_t t_off[TIK_MAX_SLABS];
  int32_t total_chunks;
  int32_t tt, vv, tiles_t;         // tile = tt frames x vv row groups
  int32_t a_box_bytes;             // tt*vv*128
  int32_t n_tiles_n;               // c_out / BN
  int64_t tiles_m;                 // ceil(nv/vv) * tiles_t
  int32_t stages, w_resident;
  int32_t group;                   // K chunks per ring stage: one full/empty barrier hand-off per `group` chunks
  int32_t off_ring, off_bias, off_bar;   // byte offsets in the 1024-aligned dynamic shared memory
  int32_t bias_rows;
  int64_t nv;
  int32_t v, t_out, c_out, c_out_valid;
  const float* bias; int32_t bias_per_node;
  int32_t act; float slope;
  int32_t res_kind; const void* res; const float* res_w; int32_t res_cin, res_t_mul, res_t_in;
  void* out; int32_t out_layout;
  int32_t ts;                      // weights stationary in tensor memory (rowgemm_ts_kernel)
  const __nv_bfloat16* w_gmem;     // ts: (c_out, ktot) row-major weights
  int32_t ktot;
  int32_t rev;                     // LaunchOpts: tiles walked last to first
};

__device__ __forceinline__ float apply_act(float v, int act, float slope) {
  if (act == TIK_ACT_RELU) return fmaxf(v, 0.f);
  if (act == TIK_ACT_LEAKY) return v > 0.f ? v : v * slope;
  return v;
}

template <int BN, int ACT>
__global__ void __launch_bounds__(kUmmaThreads, 1) rowgemm_umma_kernel(const __grid_constant__ UmmaParams p) {
  constexpr int kBBytes = BN * kChunkK * 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; pointer arithmetic on the shared base keeps the address space (LDS / STS, not generic LD / ST)
  uint8_t* w_res = smem;                                    // resident weights: total_chunks x (BN x 64) tiles
  uint8_t* ring = smem + p.off_ring;
  float* s_bias = reinterpret_cast<float*>(smem + p.off_bias);
  uint8_t* s_stage = smem + p.off_stage;                    // BN/64 regions of 128 rows x 128 B (swizzled)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tmem_full = empty_bar + kMaxStages;             // [2]
  uint64_t* tmem_empty = tmem_full + 2;                     // [2]
  uint64_t* w_full = tmem_empty + 2;
  uint64_t* stage_full = w_full + 1;                        // [2] staging tile written by the 16 epilogue warps
  uint64_t* stage_empty = stage_full + 2;                   // [2] staging tile read by the TMA store
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stage_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int stages = p.stages;
  const int chunk_bytes = kABytes + (p.w_resident ? 0 : kBBytes);
  const int stage_bytes = p.group * chunk_bytes;
  const int num_tiles = (int)(p.tiles_m * p.n_tiles_n);
  const int g0 = (int)blockIdx.x, gstep = (int)gridDim.x;
  auto tile_of = [&](int g) -> int { return p.rev ? num_tiles - 1 - g : g; };

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.n_slabs; ++s) tma_prefetch_desc(&p.map_a[s]);
    tma_prefetch_desc(&p.map_w);
    if (p.tma_store) tma_prefetch_desc(&p.map_out);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], kEpiWarps); }
    mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&stage_full[i], kEpiWarps); mbar_init(&stage_empty[i], 1); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<2 * BN>(tmem_slot);
  // per-node tables are stored with a 4-float pad per row (rows c_out*4 bytes apart would share their first bank)
  for (int i = threadIdx.x; i < p.bias_rows * p.c_out; i += kUmmaThreads) s_bias[(i / p.c_out) * (p.c_out + 4) + (i % p.c_out)] = __ldg(p.bias + i);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();                                  // the next kernel may begin its own prologue
  pdl_wait();                                               // everything below reads what the previous kernel wrote

  if (warp == 0) {
    // ===================== TMA producer =====================
    // The whole warp runs the loop (warp-uniform control flow keeps addresses / coordinates in uniform registers);
    // lane 0 issues.
    const bool leader = lane == 0;
    if (p.w_resident && leader) {
      mbar_expect_tx(w_full, (uint32_t)(p.total_chunks * kBBytes));
      for (int kc = 0; kc < p.total_chunks; ++kc) tma_load_2d(w_res + (size_t)kc * kBBytes, &p.map_w, w_full, kc * kChunkK, 0);
    }
    const uint32_t tx_bytes = (uint32_t)(p.a_box_bytes + (p.w_resident ? 0 : kBBytes));
    const int group = p.group, total_chunks = p.total_chunks;
    int stage = 0; uint32_t phase = 0;
    for (int g = g0; g < num_tiles; g += gstep) {
      const int tile = tile_of(g);
      const int tm = tile / p.n_tiles_n;
      const int n0 = (tile - tm * p.n_tiles_n) * BN;
      const int tile_nv = tm / p.tiles_t;
      const int t0 = (tm - tile_nv * p.tiles_t) * p.tt;
      const int nv0 = tile_nv * p.vv;
      int kw = 0, j = 0;                                   // j = position of this chunk inside its stage
      for (int s = 0; s < p.n_slabs; ++s) {
        const int ts = t0 * p.t_mul[s] + p.t_off[s];
        const int nc = p.chunks[s];
        for (int c = 0; c < nc; ++c, ++kw) {
          if (j == 0) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            const int in_stage = min(group, total_chunks - kw);
            if (leader) mbar_expect_tx(&full_bar[stage], tx_bytes * (uint32_t)in_stage);
          }
          uint8_t* sa = ring + (size_t)stage * stage_bytes + (size_t)j * chunk_bytes;
          if (leader) {
            tma_load_3d(sa, &p.map_a[s], &full_bar[stage], c * kChunkK, ts, nv0);
            if (!p.w_resident) tma_load_2d(sa + kABytes, &p.map_w, &full_bar[stage], kw * kChunkK, n0);
          }
          __syncwarp();
          if (++j == group || kw + 1 == total_chunks) {
            j = 0;
            if (++stage == stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // Warp-uniform loop, one lane issues tcgen05.mma / tcgen05.commit.
    constexpr uint32_t idesc = make_idesc_bf16(kTileM, BN);
    const bool leader = lane == 0;
    if (p.w_resident) mbar_wait(w_full, 0);
    const uint32_t ring_u32 = smem_u32(ring), wres_u32 = smem_u32(w_res);
    const uint64_t desc_hi = make_smem_desc_kmajor_sw128(0);          // everything but the start address
    int stage = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    const int total_chunks = p.total_chunks, group = p.group;
    for (int g = g0; g < num_tiles; g += gstep) {
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);        // epilogue has drained this accumulator
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
      for (int kc = 0; kc < total_chunks; kc += group) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const int in_stage = min(group, total_chunks - kc);
        for (int j = 0; j < in_stage; ++j) {
          const uint32_t sa = ring_u32 + (uint32_t)stage * (uint32_t)stage_bytes + (uint32_t)j * (uint32_t)chunk_bytes;
          const uint32_t sb = p.w_resident ? wres_u32 + (uint32_t)(kc + j) * (uint32_t)kBBytes : sa + kABytes;
          // descriptor = constant high part | (address >> 4); +2 per 16-element (32 B) K step inside the swizzled row
          const uint64_t da = desc_hi | (uint64_t)((sa >> 4) & 0x3FFF);
          const uint64_t db = desc_hi | (uint64_t)((sb >> 4) & 0x3FFF);
          if (leader) {
#pragma unroll
            for (int k = 0; k < kChunkK / 16; ++k)
              umma_bf16(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kc | j | k) != 0 ? 1u : 0u);
          }
        }
        if (leader) umma_commit(&empty_bar[stage]);        // frees this ring slot once the MMAs have read it
        __syncwarp();
        if (++stage == stages) { stage = 0; phase ^= 1; }
      }
      if (leader) umma_commit(&tmem_full[acc]);          // accumulator complete -> epilogue
      __syncwarp();
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else if (warp == 2 + kEpiWarps) {
    // ===================== TMA-store warp =====================
    // Takes the store issue and its completion waits off the epilogue warps' critical path.
    if (lane == 0 && p.tma_store) {
      const int ntn = p.n_tiles_n, tiles_t = p.tiles_t;
      int sbuf = 0; uint32_t sphase = 0;
      int prev = -1;
      for (int g = g0; g < num_tiles; g += gstep) {
      const int tile = tile_of(g);
        const int tm = tile / ntn;
        const int n0 = (tile - tm * ntn) * BN;
        const int tile_nv = tm / tiles_t, tile_t = tm - tile_nv * tiles_t;
        mbar_wait(&stage_full[sbuf], sphase);
        for (int c = 0; c < BN / 64; ++c)
          tma_store_3d(&p.map_out, s_stage + ((size_t)sbuf * (BN / 64) + c) * kABytes, n0 + c * 64, tile_t * p.tt, tile_nv * p.vv);
        tma_store_commit();
        if (p.stage_bufs == 2) {
          tma_store_wait_read1();                           // every store but the newest has finished reading smem
          if (prev >= 0) mbar_arrive(&stage_empty[prev]);
          prev = sbuf;
          if (++sbuf == 2) { sbuf = 0; sphase ^= 1; }
        } else {
          tma_store_wait_read0();
          mbar_arrive(&stage_empty[0]);
          sphase ^= 1;
        }
      }
      tma_store_wait0();
    }
  } else {
    // ===================== epilogue =====================
    // 16 warps: TMEM lane group (warp & 3) x column quarter; thread = one tile row x BN/4 columns.
    constexpr int CW = BN / 4;
    const int lane_grp = warp & 3;               // TMEM lanes [32*lane_grp, +32) are accessible to this warp
    const int cq = (warp - 2) >> 2;              // column quarter
    const int r = lane_grp * 32 + lane;          // tile row == TMEM lane
    const int nv_l = r / p.tt, t_l = r - nv_l * p.tt;
    const bool use_res = p.res_kind == TIK_RES_IDENTITY;
    const int ntn = p.n_tiles_n, tiles_t = p.tiles_t;
    int acc = 0; uint32_t acc_phase = 0;
    int sbuf = 0; uint32_t sphase = 0;
    for (int g = g0; g < num_tiles; g += gstep) {
      const int tile = tile_of(g);
      const int tm = tile / ntn;
      const int n0 = (tile - tm * ntn) * BN;
      const int tile_nv = tm / tiles_t, tile_t = tm - tile_nv * tiles_t;
      const int t = tile_t * p.tt + t_l;
      const int nv = tile_nv * p.vv + nv_l;
      const bool valid = (nv_l < p.vv) && (nv < (int)p.nv) && (t < p.t_out);
      const int n = nv / p.v, node = nv - n * p.v;
      const int64_t row = (int64_t)nv * p.t_out + t;
      const int cb = cq * CW;                    // first column (within the tile) this thread handles
      const float* bias = s_bias + (p.bias_per_node ? node * (p.c_out + 4) : 0) + n0 + cb;
      const __nv_bfloat16* res_row = (valid && use_res) ? reinterpret_cast<const __nv_bfloat16*>(p.res) + row * p.c_out + n0 + cb : nullptr;
      int64_t out_off;
      if (p.out_layout == TIK_OUT_NODE_MAJOR) out_off = row * p.c_out + n0 + cb;
      else if (p.out_layout == TIK_OUT_TIME_MAJOR) out_off = (((int64_t)n * p.t_out + t) * p.v + node) * (int64_t)p.c_out + n0 + cb;
      else out_off = row * p.c_out_valid + n0 + cb;
      uint8_t* stage_row = s_stage + (size_t)sbuf * (BN / 64) * kABytes + (size_t)r * 128;

      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN + cb) + ((uint32_t)(lane_grp * 32) << 16);
      uint32_t a[CW];
#pragma unroll
      for (int i = 0; i < CW / 16; ++i) tmem_ld16(tmem_d + (uint32_t)(16 * i), a + 16 * i);
      tmem_ld_wait();
      // the accumulator now lives in registers: hand the TMEM buffer back to the MMA warp right away
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      // the store issued from this staging tile (stage_bufs tiles ago) must have finished reading it
      if (p.tma_store) mbar_wait(&stage_empty[sbuf], sphase ^ 1);
      if (valid || p.tma_store) {
#pragma unroll
        for (int q = 0; q < CW / 8; ++q) {       // 8 columns = one 16-byte bf16 piece
          const float4 b0 = *reinterpret_cast<const float4*>(bias + 8 * q);
          const float4 b1 = *reinterpret_cast<const float4*>(bias + 8 * q + 4);
          float v[8] = {__uint_as_float(a[8 * q + 0]) + b0.x, __uint_as_float(a[8 * q + 1]) + b0.y,
                        __uint_as_float(a[8 * q + 2]) + b0.z, __uint_as_float(a[8 * q + 3]) + b0.w,
                        __uint_as_float(a[8 * q + 4]) + b1.x, __uint_as_float(a[8 * q + 5]) + b1.y,
                        __uint_as_float(a[8 * q + 6]) + b1.z, __uint_as_float(a[8 * q + 7]) + b1.w};
          if (res_row != nullptr) {              // slow path (scattered 16 B loads); the plan folds residuals into a K-slab
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(res_row + 8 * q));
            const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = __bfloat1622float2(h[e]);
              v[2 * e] += f.x;
              v[2 * e + 1] += f.y;
            }
          }
          if (ACT == TIK_ACT_LEAKY) {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = v[e] > 0.f ? v[e] : v[e] * p.slope;
          }
          if (p.out_layout == TIK_OUT_ROWS_F32) {
            float* o = reinterpret_cast<float*>(p.out) + out_off + 8 * q;
#pragma unroll
            for (int e = 0; e < 8; ++e)
              if (valid && n0 + cb + 8 * q + e < p.c_out_valid) o[e] = (ACT == TIK_ACT_RELU) ? fmaxf(v[e], 0.f) : v[e];
          } else {
            uint4 u;
            if (ACT == TIK_ACT_RELU) {
              u.x = pack_bf16x2_relu(v[0], v[1]); u.y = pack_bf16x2_relu(v[2], v[3]);
              u.z = pack_bf16x2_relu(v[4], v[5]); u.w = pack_bf16x2_relu(v[6], v[7]);
            } else {
              u.x = pack_bf16x2(v[0], v[1]); u.y = pack_bf16x2(v[2], v[3]);
              u.z = pack_bf16x2(v[4], v[5]); u.w = pack_bf16x2(v[6], v[7]);
            }
            if (p.tma_store) {
              // 16 B piece j of this row's 128 B line in 64-column region (cb+8q)/64, at its 128B-swizzle position
              const int col = cb + 8 * q;
              const int j = (col & 63) >> 3;
              *reinterpret_cast<uint4*>(stage_row + (size_t)(col >> 6) * kABytes + ((j ^ (r & 7)) << 4)) = u;
            } else if (valid) {
              *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + out_off + 8 * q) = u;
            }
          }
        }
      }
      if (p.tma_store) {
        fence_proxy_async_smem();                           // st.shared -> visible to the TMA (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(&stage_full[sbuf]);      // 16 warps -> the store warp issues the tile
        if (p.stage_bufs == 2) { if (++sbuf == 2) { sbuf = 0; sphase ^= 1; } } else { sphase ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<2 * BN>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ weight-stationary variant
// Same implicit GEMM computed TRANSPOSED with the weights as the tensor-memory-resident A operand:
//
//   D^T[c_out (TMEM lanes), tile rows (TMEM columns)] = W[c_out x K] (TMEM) . A_tile[rows x K]^T (shared memory)
//
// The SS form above reads a 128 x 16 weight slice from shared memory for every MMA (and streams the weights through
// the ring again for every tile when they do not fit beside it); at N <= 128 that operand traffic, not the tensor
// pipe, is what saturates the 128 B/clk shared-memory port.  Here the weights are written to tensor memory once per
// CTA (c_out <= 128 lanes x K/2 columns, bf16 pairs) and only the activation tile is read from shared memory.
// The accumulator comes out channel-major (lane = output channel, column = tile row), so the epilogue adds a
// per-lane bias and transposes through the swizzled staging tile with 2-byte stores (one 64-byte run per warp
// instruction).  Eligible: c_out == 128 (at 64 the padded lanes cost more than the saved weight reads), K <= 512,
// per-channel bias, node-major TMA-stored output.
template <int ACT>
__global__ void __launch_bounds__(kUmmaThreads, 1) rowgemm_ts_kernel(const __grid_constant__ UmmaParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; pointer arithmetic on the shared base keeps the address space (LDS / STS, not generic LD / ST)
  uint8_t* ring = smem + p.off_ring;
  uint8_t* s_stage = smem + p.off_stage;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tmem_full = empty_bar + kMaxStages;             // [2]
  uint64_t* tmem_empty = tmem_full + 2;                     // [2]
  uint64_t* w_full = tmem_empty + 2;                        // unused here
  uint64_t* stage_full = w_full + 1;                        // [2]
  uint64_t* stage_empty = stage_full + 2;                   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stage_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int stages = p.stages, group = p.group, total_chunks = p.total_chunks;
  const int stage_bytes = group * kABytes;
  const int n_tiles = (int)p.tiles_m;
  const int regions = p.c_out / 64;                         // 64-channel staging regions

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.n_slabs; ++s) tma_prefetch_desc(&p.map_a[s]);
    tma_prefetch_desc(&p.map_out);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], kEpiWarps); }
    for (int i = 0; i < 2; ++i) { mbar_init(&stage_full[i], kEpiWarps); mbar_init(&stage_empty[i], 1); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_w = tmem_base;                        // K/2 columns of bf16 pairs, lane = output channel
  const uint32_t tmem_acc = tmem_base + 256;                // 2 x 128 fp32 columns
  // ---- weights -> tensor memory (once per CTA): the 16 epilogue warps share the work, four per TMEM lane quadrant,
  // each taking a quarter of the K range (a warp can only write the lanes of its own quadrant)
  if (warp >= 2 && warp < 2 + kEpiWarps) {
    const int co = (warp & 3) * 32 + lane;
    const int part = (warp - 2) >> 2;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const uint4* wrow = reinterpret_cast<const uint4*>(p.w_gmem + (size_t)(co < p.c_out ? co : 0) * p.ktot);
    const int n16 = p.ktot / 16;                            // 16 bf16 = 8 packed columns per store; 4 stores per batch of loads
    for (int k8 = part * 4; k8 < n16; k8 += 16) {
      uint4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = co < p.c_out ? __ldg(wrow + 2 * k8 + u) : make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t r[8] = {v[2 * u].x, v[2 * u].y, v[2 * u].z, v[2 * u].w, v[2 * u + 1].x, v[2 * u + 1].y, v[2 * u + 1].z, v[2 * u + 1].w};
        tmem_st8(tmem_w + lane_off + (uint32_t)(8 * (k8 + u)), r);
      }
    }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();                                               // weights are constants; activations come from the previous kernel

  if (warp == 0) {
    // ===================== TMA producer: activation chunks only =====================
    const bool leader = lane == 0;
    int stage = 0; uint32_t phase = 0;
    for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
      const int tile = p.rev ? n_tiles - 1 - ti : ti;
      const int tile_nv = tile / p.tiles_t;
      const int t0 = (tile - tile_nv * p.tiles_t) * p.tt;
      const int nv0 = tile_nv * p.vv;
      int kw = 0, j = 0;
      for (int s = 0; s < p.n_slabs; ++s) {
        const int ts = t0 * p.t_mul[s] + p.t_off[s];
        const int nc = p.chunks[s];
        for (int c = 0; c < nc; ++c, ++kw) {
          if (j == 0) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (leader) mbar_expect_tx(&full_bar[stage], (uint32_t)p.a_box_bytes * (uint32_t)min(group, total_chunks - kw));
          }
          if (leader)
            tma_load_3d(ring + (size_t)stage * stage_bytes + (size_t)j * kABytes, &p.map_a[s], &full_bar[stage], c * kChunkK, ts, nv0);
          __syncwarp();
          if (++j == group || kw + 1 == total_chunks) {
            j = 0;
            if (++stage == stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The state of the NEXT barrier this thread will need (next ring stage, or the next tile's accumulator) is
    // polled with a non-blocking test_wait before the current stage's MMAs are issued, so the poll's round trip
    // overlaps the issue; in steady state the blocking wait is never entered.
    constexpr uint32_t idesc = make_idesc_bf16(128, kTileM);   // M = 128 channel lanes (zero rows beyond c_out), N = tile rows
    const bool leader = lane == 0;
    const uint32_t ring_u32 = smem_u32(ring);
    const uint64_t desc_hi = make_smem_desc_kmajor_sw128(0);
    const int stages_per_tile = (total_chunks + group - 1) / group;
    int stage = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    bool full_ready = false, acc_ready = false;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      if (!acc_ready) mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tc_fence_after();
      const bool last_tile = tile + (int)gridDim.x >= n_tiles;
      const uint32_t tmem_d = tmem_acc + (uint32_t)(acc * kTileM);
      int sidx = 0;
      for (int kc = 0; kc < total_chunks; kc += group, ++sidx) {
        if (!full_ready) mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        int nstage = stage + 1; uint32_t nphase = phase;
        if (nstage == stages) { nstage = 0; nphase ^= 1; }
        const bool last_stage = sidx + 1 == stages_per_tile;
        // early polls for what comes next
        const bool poll_full = !(last_stage && last_tile);
        bool nfull = false, nacc = false;
        if (poll_full) nfull = mbar_test_wait(&full_bar[nstage], nphase);
        if (last_stage && !last_tile) nacc = mbar_test_wait(&tmem_empty[acc ^ 1], (acc == 1 ? acc_phase ^ 1 : acc_phase) ^ 1);
        const int in_stage = min(group, total_chunks - kc);
        for (int j = 0; j < in_stage; ++j) {
          const uint32_t sa = ring_u32 + (uint32_t)stage * (uint32_t)stage_bytes + (uint32_t)j * (uint32_t)kABytes;
          const uint64_t db = desc_hi | (uint64_t)((sa >> 4) & 0x3FFF);
          if (leader) {
#pragma unroll
            for (int k = 0; k < kChunkK / 16; ++k)
              umma_bf16_ts(tmem_d, tmem_w + (uint32_t)((kc + j) * 32 + k * 8), db + (uint64_t)(2 * k), idesc, (kc | j | k) != 0 ? 1u : 0u);
          }
        }
        if (leader) umma_commit(&empty_bar[stage]);
        __syncwarp();
        stage = nstage; phase = nphase;
        full_ready = nfull; acc_ready = nacc;
      }
      if (leader) umma_commit(&tmem_full[acc]);
      __syncwarp();
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else if (warp == 2 + kEpiWarps) {
    // ===================== TMA-store warp =====================
    if (lane == 0) {
      int sbuf = 0; uint32_t sphase = 0;
      int prev = -1;
      for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
        const int tile = p.rev ? n_tiles - 1 - ti : ti;
        const int tile_nv = tile / p.tiles_t, tile_t = tile - tile_nv * p.tiles_t;
        mbar_wait(&stage_full[sbuf], sphase);
        for (int c = 0; c < regions; ++c)
          tma_store_3d(&p.map_out, s_stage + ((size_t)sbuf * regions + c) * kABytes, c * 64, tile_t * p.tt, tile_nv * p.vv);
        tma_store_commit();
        if (p.stage_bufs == 2) {
          tma_store_wait_read1();
          if (prev >= 0) mbar_arrive(&stage_empty[prev]);
          prev = sbuf;
          if (++sbuf == 2) { sbuf = 0; sphase ^= 1; }
        } else {
          tma_store_wait_read0();
          mbar_arrive(&stage_empty[0]);
          sphase ^= 1;
        }
      }
      tma_store_wait0();
    }
  } else {
    // ===================== epilogue: 16 warps = TMEM lane group (32 channels) x 32-row quarter =====================
    // The accumulator is channel-major.  tcgen05.ld.16x256b hands each thread mma-style fragments (two adjacent tile
    // rows of one channel per register pair); packed to bf16x2 they are exactly the fragments stmatrix.trans wants,
    // which writes them transposed: 16-byte pieces of 8 consecutive channels per tile row, at the piece's 128B-swizzle
    // position (every lane supplies the address of one piece).
    const int lane_grp = warp & 3;
    const int rq = (warp - 2) >> 2;                         // tile rows [32*rq, +32)
    const bool grp_ok = lane_grp * 32 < p.c_out;
    float bias[2][2];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int co = lane_grp * 32 + 16 * h + 8 * u + (lane >> 2);
        bias[h][u] = co < p.c_out ? __ldg(p.bias + co) : 0.f;
      }
    // stmatrix address role of this lane: matrix i = lane/8 -> rows +8*(i/2), channel piece +(i%2); row k = lane%8
    const int a_row = ((lane >> 4) & 1) * 8 + (lane & 7);
    const int a_piece = (lane >> 3) & 1;
    int acc = 0; uint32_t acc_phase = 0;
    int sbuf = 0; uint32_t sphase = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      uint32_t a[2][16];
#pragma unroll
      for (int h = 0; h < 2; ++h)
        tmem_ld_16x256b_x4(tmem_acc + ((uint32_t)(lane_grp * 32 + 16 * h) << 16) + (uint32_t)(acc * kTileM + rq * 32), a[h]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      mbar_wait(&stage_empty[sbuf], sphase ^ 1);
      if (grp_ok) {
        const uint32_t st_u32 = smem_u32(s_stage + (size_t)sbuf * regions * kABytes);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int co0 = lane_grp * 32 + 16 * h;
          const uint32_t piece = (uint32_t)(((co0 & 63) >> 3) + a_piece);
          const uint32_t region = st_u32 + (uint32_t)(co0 >> 6) * kABytes;
#pragma unroll
          for (int pr = 0; pr < 2; ++pr) {                  // two 8-row blocks per stmatrix.x4
            uint32_t m[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {                   // q = 2*(row block) + (channel half)
              float v0 = __uint_as_float(a[h][8 * pr + 2 * q]) + bias[h][q & 1];
              float v1 = __uint_as_float(a[h][8 * pr + 2 * q + 1]) + bias[h][q & 1];
              if (ACT == TIK_ACT_LEAKY) { v0 = v0 > 0.f ? v0 : v0 * p.slope; v1 = v1 > 0.f ? v1 : v1 * p.slope; }
              m[q] = (ACT == TIK_ACT_RELU) ? pack_bf16x2_relu(v0, v1) : pack_bf16x2(v0, v1);
            }
            const int r = rq * 32 + pr * 16 + a_row;
            stmatrix_x4_trans(region + (uint32_t)r * 128u + ((piece ^ (uint32_t)(r & 7)) << 4), m[0], m[1], m[2], m[3]);
          }
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&stage_full[sbuf]);
      if (p.stage_bufs == 2) { if (++sbuf == 2) { sbuf = 0; sphase ^= 1; } } else { sphase ^= 1; }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
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
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !p) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return nullptr;
  }
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

static int encode_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box, const uint32_t* estr) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return TIK_ERR_CUDA;
  TIK_CHECK_ARG(((uintptr_t)base & 15) == 0, "TMA base address must be 16-byte aligned");
  // A strided (stride-2) box over 128-byte rows skips every other row: do not let L2 promotion fetch the skipped rows
  const bool skip_rows = rank > 1 && estr[1] > 1 && strides_bytes[0] <= 128;
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  skip_rows ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d dims %llu,%llu,%llu box %u,%u,%u)", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)(rank > 2 ? dims[2] : 0),
              box[0], box[1], rank > 2 ? box[2] : 0);
    return TIK_ERR_CUDA;
  }
  return TIK_OK;
}

static int64_t align_up_i(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

struct UmmaPrepared {
  UmmaParams p;
  int bn;
  int smem_bytes;
  int64_t nv_capacity;
};

static int num_sms() {
  static int sms[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (!sms[dev & 63]) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    sms[dev & 63] = v;
  }
  return sms[dev & 63];
}

template <int BN, int ACT>
static int launch_variant(const UmmaParams& p, int smem_bytes, unsigned grid, cudaStream_t s) {
  static int attr_done[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (attr_done[dev & 63] < smem_bytes) {   // the attribute is per device
    TIK_CUDA(cudaFuncSetAttribute(rowgemm_umma_kernel<BN, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget + 2048));
    TIK_CUDA(cudaFuncSetAttribute(rowgemm_umma_kernel<BN, ACT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr_done[dev & 63] = kSmemBudget + 2048;
  }
  TIK_CUDA(launch_pdl(rowgemm_umma_kernel<BN, ACT>, grid, kUmmaThreads, (size_t)smem_bytes, s, p));
  return TIK_OK;
}

int umma_prepare(const TikRowGemm* d, int64_t nv_capacity, UmmaPrepared** out) {
  TIK_CHECK_ARG(d->c_out % 64 == 0, "bf16 path: c_out=%d must be a multiple of 64", d->c_out);
  TIK_CHECK_ARG(nv_capacity >= d->nv && nv_capacity > 0, "nv capacity");
  if (d->res_kind == TIK_RES_STEM) {
    set_error("bf16 path: TIK_RES_STEM is only implemented by the fp32 kernel (the stem kernel precomputes that branch)");
    return TIK_ERR_UNSUPPORTED;
  }
  UmmaPrepared* u = new UmmaPrepared();
  UmmaParams& p = u->p;
  memset(&p, 0, sizeof(p));
  int ktot = 0, max_mul = 1;
  for (int i = 0; i < d->n_slabs; ++i) {
    const TikSlab& sl = d->slabs[i];
    if (!(sl.a_dev && sl.c > 0 && sl.c % 64 == 0 && sl.t_in > 0 && sl.t_mul >= 1 && sl.t_mul <= 8)) {
      delete u;
      set_error("bf16 path: slab %d malformed (c=%d must be a multiple of 64, t_mul=%d in [1,8])", i, sl.c, sl.t_mul);
      return TIK_ERR_INVALID;
    }
    ktot += sl.c;
    if (sl.t_mul > max_mul) max_mul = sl.t_mul;
  }
  int tt = d->t_out < kTileM ? d->t_out : kTileM;
  if (tt * max_mul > 256) tt = 256 / max_mul;     // TMA box extent limit
  int vv = kTileM / tt;
  p.tt = tt; p.vv = vv; p.tiles_t = (int)ceil_div(d->t_out, tt);
  p.a_box_bytes = tt * vv * kChunkK * 2;
  p.n_slabs = d->n_slabs;
  p.total_chunks = ktot / 64;
  for (int i = 0; i < d->n_slabs; ++i) {
    const TikSlab& sl = d->slabs[i];
    p.chunks[i] = sl.c / 64; p.t_mul[i] = sl.t_mul; p.t_off[i] = sl.t_off;
    uint64_t dims[3] = {(uint64_t)sl.c, (uint64_t)sl.t_in, (uint64_t)nv_capacity};
    uint64_t strides[2] = {(uint64_t)sl.c * 2, (uint64_t)sl.c * 2 * (uint64_t)sl.t_in};
    uint32_t box[3] = {(uint32_t)kChunkK, (uint32_t)(tt * sl.t_mul), (uint32_t)vv};
    uint32_t estr[3] = {1, (uint32_t)sl.t_mul, 1};
    int rc = encode_map(&p.map_a[i], sl.a_dev, 3, dims, strides, box, estr);
    if (rc != TIK_OK) { delete u; return rc; }
  }
  u->bn = d->c_out % 256 == 0 ? 256 : (d->c_out % 128 == 0 ? 128 : 64);
  if (const char* e = getenv("TIK_UMMA_BN")) {          // tuning hook: narrower N tiles for the 256-column layers
    const int want = atoi(e);
    if ((want == 128 || want == 64) && want < u->bn && d->c_out % want == 0) u->bn = want;
  }
  p.n_tiles_n = d->c_out / u->bn;
  {
    uint64_t dims[2] = {(uint64_t)ktot, (uint64_t)d->c_out};
    uint64_t strides[1] = {(uint64_t)ktot * 2};
    uint32_t box[2] = {(uint32_t)kChunkK, (uint32_t)u->bn};
    uint32_t estr[2] = {1, 1};
    int rc = encode_map(&p.map_w, d->w_dev, 2, dims, strides, box, estr);
    if (rc != TIK_OK) { delete u; return rc; }
  }
  // shared-memory plan: [resident W][ring][bias][barriers]
  const int b_bytes = u->bn * kChunkK * 2;
  const int bias_rows = d->bias_per_node ? d->v : 1;
  const int bias_bytes = (int)align_up_i(bias_rows * (d->c_out + 4) * 4, 16);
  const int bar_bytes = 256;
  const int w_bytes = p.total_chunks * b_bytes;
  p.tma_store = (d->out_layout == TIK_OUT_NODE_MAJOR && d->out_dev != nullptr) ? 1 : 0;
  // smem policy: a deep A ring matters most (>= 4 stages), then resident weights, then a second staging tile
  const int one_stage_tile = p.tma_store ? (u->bn / 64) * kABytes : 0;
  // Ring stages hold `group` K chunks each: the producer -> MMA -> producer barrier round trip (~650 cycles on the
  // MMA thread) is paid once per stage, so small-N layers need several chunks per stage to stay HBM-bound.
  int w_res = 0, stages = 0, sbufs = 1, group = 1;
  auto ring_chunks = [&](int wres, int sb) {
    const int fixed_ = bias_bytes + bar_bytes + sb * one_stage_tile;
    return wres ? (kSmemBudget - fixed_ - w_bytes) / kABytes : (kSmemBudget - fixed_) / (kABytes + b_bytes);
  };
  // Pick (weights resident?, staging tiles, chunks per stage) by a cost model fitted to whole-batch B200 timings
  // (tools/umma_probe.py grp): barrier hand-offs per tile cost ~400 cycles each, and the activation stream needs
  // ~8 chunks (128 KB) in flight per SM to cover HBM latency.
  const char* env_g = getenv("TIK_UMMA_GROUP");     // tuning hooks (tools/umma_probe.py)
  const char* env_o = getenv("TIK_UMMA_OPT");
  const int options[4][2] = {{1, 2}, {1, 1}, {0, 2}, {0, 1}};
  int best_score = INT32_MAX;
  for (int o = 0; o < 4; ++o) {
    const int wres = options[o][0], sb = options[o][1];
    if (wres && p.n_tiles_n != 1) continue;
    if (env_o && o != atoi(env_o)) continue;
    const int fit = ring_chunks(wres, sb);
    for (int g = 4; g >= 1; g >>= 1) {
      if (env_g && g != atoi(env_g)) continue;
      if (g > 1 && g > p.total_chunks) continue;
      int st = fit / g;
      if (st < 2) continue;
      if (st > kMaxStages) st = kMaxStages;
      const int inflight = std::min(st * g, 8);
      const int handoffs = (p.total_chunks + g - 1) / g;
      const int score = handoffs * 400 + 24000 / inflight + (wres ? 0 : 200) + (sb == 2 ? 0 : 100);
      if (score < best_score) { best_score = score; w_res = wres; sbufs = sb; group = g; stages = st; }
    }
  }
  // Weight-stationary kernel (weights in tensor memory, see rowgemm_ts_kernel): the whole ring is activations.
  p.ts = (p.tma_store && (d->c_out == 128 || d->c_out == 64) && ktot <= 512 && !d->bias_per_node && d->res_kind == TIK_RES_NONE && !getenv("TIK_NO_TS")) ? 1 : 0;
  if (p.ts) {
    best_score = INT32_MAX;
    for (int sb = 2; sb >= 1; --sb) {
      const int fit = (kSmemBudget - bar_bytes - bias_bytes - sb * one_stage_tile) / kABytes;
      for (int g = 4; g >= 1; g >>= 1) {
        if (env_g && g != atoi(env_g)) continue;
        if (g > 1 && g > p.total_chunks) continue;
        int st = fit / g;
        if (st < 2) continue;
        if (st > kMaxStages) st = kMaxStages;
        const int score = ((p.total_chunks + g - 1) / g) * 400 + 24000 / std::min(st * g, 8) + (sb == 2 ? 0 : 100);
        if (score < best_score) { best_score = score; w_res = 1; sbufs = sb; group = g; stages = st; }
      }
    }
  }
  p.group = group;
  p.stage_bufs = sbufs;
  const int stage_out_bytes = sbufs * one_stage_tile;
  if (stages < 2) {
    delete u;
    if (env_o || env_g) set_error("bf16 path: no shared-memory plan with TIK_UMMA_OPT=%s TIK_UMMA_GROUP=%s fits this GEMM (c_out=%d, %d K chunks)",
                                  env_o ? env_o : "-", env_g ? env_g : "-", d->c_out, p.total_chunks);
    else set_error("bf16 path: bias table too large for shared memory");
    return TIK_ERR_UNSUPPORTED;
  }
  p.w_resident = w_res; p.stages = stages;
  p.off_ring = (w_res && !p.ts) ? w_bytes : 0;
  p.off_stage = p.off_ring + stages * group * (kABytes + (w_res ? 0 : b_bytes));
  p.off_bias = p.off_stage + stage_out_bytes;
  p.off_bar = p.off_bias + bias_bytes;
  if (p.tma_store) {
    uint64_t dims[3] = {(uint64_t)d->c_out, (uint64_t)d->t_out, (uint64_t)nv_capacity};
    uint64_t strides[2] = {(uint64_t)d->c_out * 2, (uint64_t)d->c_out * 2 * (uint64_t)d->t_out};
    uint32_t box[3] = {(uint32_t)kChunkK, (uint32_t)tt, (uint32_t)vv};
    uint32_t estr[3] = {1, 1, 1};
    int rc = encode_map(&p.map_out, d->out_dev, 3, dims, strides, box, estr);
    if (rc != TIK_OK) { delete u; return rc; }
  }
  p.bias_rows = bias_rows;
  p.w_gmem = reinterpret_cast<const __nv_bfloat16*>(d->w_dev); p.ktot = ktot;
  u->smem_bytes = p.off_bar + bar_bytes + 1024;
  u->nv_capacity = nv_capacity;
  *out = u;
  return TIK_OK;
}

int umma_launch(UmmaPrepared* u, const TikRowGemm* d, cudaStream_t s) {
  UmmaParams& p = u->p;
  TIK_CHECK_ARG(d->nv <= u->nv_capacity, "nv exceeds prepared capacity");
  p.nv = d->nv; p.v = d->v; p.t_out = d->t_out; p.c_out = d->c_out; p.c_out_valid = d->c_out_valid;
  p.bias = d->bias_dev; p.bias_per_node = d->bias_per_node;
  p.act = d->act; p.slope = d->slope;
  p.res_kind = d->res_kind; p.res = d->res_dev; p.res_w = d->res_w_dev;
  p.res_cin = d->res_cin; p.res_t_mul = d->res_t_mul; p.res_t_in = d->res_t_in;
  p.out = d->out_dev; p.out_layout = d->out_layout;
  p.rev = launch_opts().rev;
  if (d->nv == 0 || d->t_out == 0) return TIK_OK;
  p.tiles_m = ceil_div(d->nv, p.vv) * ceil_div(d->t_out, p.tt);
  p.tiles_t = (int)ceil_div(d->t_out, p.tt);
  const int64_t tiles = p.tiles_m * p.n_tiles_n;
  const unsigned grid = (unsigned)std::min<int64_t>(tiles, num_sms());
  TIK_CHECK_ARG(tiles < (1ll << 31), "too many tiles");
#define TIK_LAUNCH_BN(BN_)                                                                          \
  do {                                                                                              \
    if (d->act == TIK_ACT_RELU) return launch_variant<BN_, TIK_ACT_RELU>(p, u->smem_bytes, grid, s);    \
    if (d->act == TIK_ACT_LEAKY) return launch_variant<BN_, TIK_ACT_LEAKY>(p, u->smem_bytes, grid, s);  \
    return launch_variant<BN_, TIK_ACT_NONE>(p, u->smem_bytes, grid, s);                              \
  } while (0)
  if (p.ts) {
    static int ts_attr[64] = {};
    int dev = 0;
    TIK_CUDA(cudaGetDevice(&dev));
    if (!ts_attr[dev & 63]) {
      TIK_CUDA(cudaFuncSetAttribute(rowgemm_ts_kernel<TIK_ACT_RELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget + 2048));
      TIK_CUDA(cudaFuncSetAttribute(rowgemm_ts_kernel<TIK_ACT_LEAKY>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget + 2048));
      TIK_CUDA(cudaFuncSetAttribute(rowgemm_ts_kernel<TIK_ACT_NONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget + 2048));
      ts_attr[dev & 63] = 1;
    }
    TIK_CHECK_ARG(d->res_kind == TIK_RES_NONE && !d->bias_per_node, "weight-stationary kernel: residual / per-node bias changed after prepare");
    if (d->act == TIK_ACT_RELU) TIK_CUDA(launch_pdl(rowgemm_ts_kernel<TIK_ACT_RELU>, grid, kUmmaThreads, (size_t)u->smem_bytes, s, p));
    else if (d->act == TIK_ACT_LEAKY) TIK_CUDA(launch_pdl(rowgemm_ts_kernel<TIK_ACT_LEAKY>, grid, kUmmaThreads, (size_t)u->smem_bytes, s, p));
    else TIK_CUDA(launch_pdl(rowgemm_ts_kernel<TIK_ACT_NONE>, grid, kUmmaThreads, (size_t)u->smem_bytes, s, p));
    return TIK_OK;
  }
  if (u->bn == 64) TIK_LAUNCH_BN(64);
  if (u->bn == 128) TIK_LAUNCH_BN(128);
  TIK_LAUNCH_BN(256);
#undef TIK_LAUNCH_BN
}

void umma_free(UmmaPrepared* u) { delete u; }

// One-shot calls (tik_rowgemm: the per-module forwards and the iterative head's per-iteration layers) used to encode
// their tensor maps and pick their shared-memory policy on EVERY call (~100-200 us of host work, more than the kernel
// at small sizes).  Prepared launches are now kept in a small LRU keyed by the full descriptor (every pointer, shape
// and flag) and the device: a call with the same tensors at the same addresses -- what a loop over PyTorch's caching
// allocator produces -- re-uses its tensor maps.
int rowgemm_bf16(const TikRowGemm* d, cudaStream_t s) {
  struct Entry { TikRowGemm key; int dev; UmmaPrepared* u; uint64_t used; };
  static std::mutex mu;
  static std::vector<Entry> cache;
  static uint64_t tick = 0;
  constexpr size_t kCap = 32;
  // no rows: a no-op, as on the fp32 path (umma_prepare would reject the empty tensor maps)
  if (d->nv == 0) return TIK_OK;
  // tuning / A-B switches are read at prepare time: with any of them set (tools, the variant tests) nothing is cached
  if (getenv("TIK_UMMA_GROUP") || getenv("TIK_UMMA_OPT") || getenv("TIK_UMMA_BN") || getenv("TIK_NO_TS") ||
      getenv("TIK_NO_ROWGEMM_CACHE")) {
    UmmaPrepared* u = nullptr;
    int rc = umma_prepare(d, d->nv, &u);
    if (rc != TIK_OK) return rc;
    rc = umma_launch(u, d, s);
    umma_free(u);
    return rc;
  }
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  const TikRowGemm key = *d;                                // compared field-wise below (padding bytes are unspecified)
  std::lock_guard<std::mutex> lock(mu);
  auto same = [](const TikRowGemm& a, const TikRowGemm& b) {
    if (a.n_slabs != b.n_slabs || a.w_dev != b.w_dev || a.bias_dev != b.bias_dev || a.bias_per_node != b.bias_per_node || a.nv != b.nv ||
        a.v != b.v || a.t_out != b.t_out || a.c_out != b.c_out || a.c_out_valid != b.c_out_valid || a.act != b.act || a.slope != b.slope ||
        a.res_kind != b.res_kind || a.res_dev != b.res_dev || a.res_w_dev != b.res_w_dev || a.res_cin != b.res_cin ||
        a.res_t_mul != b.res_t_mul || a.res_t_in != b.res_t_in || a.out_dev != b.out_dev || a.out_layout != b.out_layout)
      return false;
    for (int i = 0; i < a.n_slabs; ++i)
      if (a.slabs[i].a_dev != b.slabs[i].a_dev || a.slabs[i].c != b.slabs[i].c || a.slabs[i].t_in != b.slabs[i].t_in ||
          a.slabs[i].t_mul != b.slabs[i].t_mul || a.slabs[i].t_off != b.slabs[i].t_off)
        return false;
    return true;
  };
  for (auto& e : cache)
    if (e.dev == dev && same(e.key, key)) {
      e.used = ++tick;
      return umma_launch(e.u, d, s);
    }
  UmmaPrepared* u = nullptr;
  int rc = umma_prepare(d, d->nv, &u);
  if (rc != TIK_OK) return rc;
  if (cache.size() >= kCap) {
    size_t lru = 0;
    for (size_t i = 1; i < cache.size(); ++i)
      if (cache[i].used < cache[lru].used) lru = i;
    umma_free(cache[lru].u);
    cache.erase(cache.begin() + (long)lru);
  }
  cache.push_back({key, dev, u, ++tick});
  return umma_launch(u, d, s);
}

}  // namespace tik
