// Temporal convolution + identity residual + BN + ReLU of a stride-1 ST-GCN block (st_gcn_aaai18.py:181-214),
// weight-stationary, with every activation row brought into shared memory ONCE.
//
// The general implicit GEMM (stgcn_umma.cu) loads one TMA box per temporal tap, i.e. the H tensor enters shared
// memory three times (twice from L2).  Measured with the same kernel fed one tensor four times: it stays at
// ~5.7 TB/s of L2 -> shared-memory fill with DRAM at 2.8 TB/s, so the fill, not HBM, binds these layers.
// Here a tile is G whole row groups (clip x node) with a one-frame halo on each side:
//   rows j*(T+2) + (t+1),  t = -1 .. T        (the halo rows are TMA out-of-bounds zero fill = the conv's zero padding)
// and the three taps are the SAME shared-memory tile read at row offsets 0, 1, 2 (a K-major 128B-swizzled operand may
// start at any 128-byte row: DESIGN.md §3 (iii)).  As in rowgemm_ts_kernel the GEMM is computed transposed,
//   D^T[c_out (TMEM lanes), n (TMEM columns)] = sum_taps W_tap (TMEM) . Htile[n + tap, :]^T  +  I . Xtile[n + 1, :]^T
// with the BN-folded weights (and the identity block that carries the residual) written once per CTA into tensor
// memory, N = the tile's rows rounded up to 16; output column n = j*(T+2) + t is valid for t < T.
// One ring stage = one tile (all of its 64-channel chunks): one barrier hand-off per tile.
// Long clips are cut into SEGMENTS of L frames: a tile is then G row groups x (L + 2) frames starting at frame t0 - 1;
// the halo rows of an interior segment are the neighbouring segment's real frames (same TMA box, other start
// coordinate), only the clip ends are out-of-bounds zero fill.  T = 64 at 128 channels thereby runs with the T = 32
// tile shape (3 x 34 rows, N = 112) instead of one 66-row group per tile (N = 80): 370 -> ~295 us per launch.
//
// Measured (B=4096): b1 (64 ch, T=64) 410 us (SS, per-tap boxes) -> 324 (TS, per-tap boxes) -> 297 us here; b3/b4
// (128 ch, T=32) 397 -> 338 -> 288 us = 5.8 TB/s of DRAM traffic, 89 % of the copy peak.  The channel-major accumulator
// is transposed by the epilogue with tcgen05.ld.16x256b fragments + stmatrix.trans; a first version with 2-byte
// shared-memory stores was instruction-bound and 2x slower than the kernels it replaces.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "tik_common.cuh"
#include "umma_prepared.h"
#include "umma_ptx.cuh"

namespace tik {

constexpr int kThEpiWarps = 16;
constexpr int kThThreads = 64 + 32 * kThEpiWarps + 32;     // producer, MMA, 16 epilogue warps, store warp
constexpr int kThMaxStages = 6;
constexpr int kThSmemBudget = 225 * 1024;

struct TcnHaloParams {
  CUtensorMap map_h, map_x, map_out;
  const __nv_bfloat16* w;        // (c_out, ktot) row-major: [tap 0 | tap 1 | tap 2 | identity]
  const float* bias;             // (c_out)
  int32_t ktot, c, c_out;        // c = channels of H and X (= c_out)
  int32_t T, R, G, N;            // T frames per clip, R = L + 2 rows per row group and tile, G row groups per tile, N = MMA columns (multiple of 16)
  int32_t L, segs;               // segment length (frames of a row group per tile) and segments per row group
  int32_t acc_stride;            // TMEM columns between the two accumulators
  int32_t kc;                    // 64-channel chunks of H (= of X)
  int32_t chunk_bytes, stage_bytes, stages;
  int32_t region_bytes, stage_bufs, off_stage, off_bar;
  int64_t nv;
  int32_t n_tiles;
  int32_t rev;                   // LaunchOpts: tiles walked last to first
};

__global__ void __launch_bounds__(kThThreads, 1) tcn_halo_kernel(const __grid_constant__ TcnHaloParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; pointer arithmetic on the shared base keeps the address space (LDS / STS, not generic LD / ST)
  uint8_t* ring = smem;
  uint8_t* s_stage = smem + p.off_stage;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* empty_bar = full_bar + kThMaxStages;
  uint64_t* tmem_full = empty_bar + kThMaxStages;           // [2]
  uint64_t* tmem_empty = tmem_full + 2;                     // [2]
  uint64_t* stage_full = tmem_empty + 2;                    // [2]
  uint64_t* stage_empty = stage_full + 2;                   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stage_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = p.n_tiles;
  const int regions = p.c_out / 64;
  const int chunks = 2 * p.kc;                              // H chunks, then X chunks

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.map_h); tma_prefetch_desc(&p.map_x); tma_prefetch_desc(&p.map_out); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < p.stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], kThEpiWarps);
      mbar_init(&stage_full[i], kThEpiWarps); mbar_init(&stage_empty[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_w = tmem_base;                        // ktot/2 columns of bf16 pairs, lane = output channel
  const uint32_t tmem_acc = tmem_base + (uint32_t)(p.ktot / 2);
  // ---- weights -> tensor memory (once per CTA; zero rows beyond c_out): the 16 epilogue warps share the work, four
  // per TMEM lane quadrant, each taking a quarter of the K range
  if (warp >= 2 && warp < 2 + kThEpiWarps) {
    const int co = (warp & 3) * 32 + lane;
    const int part = (warp - 2) >> 2;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const uint4* wrow = reinterpret_cast<const uint4*>(p.w + (size_t)(co < p.c_out ? co : 0) * p.ktot);
    const int n16 = p.ktot / 16;
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
  pdl_wait();                                               // weights are constants; H and X come from the previous kernels

  if (warp == 0) {
    // ===================== TMA producer: one stage = one tile =====================
    if (lane == 0) {
      const uint32_t box_bytes = (uint32_t)(p.G * p.R * 128);
      int stage = 0; uint32_t phase = 0;
      for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
        const int tile = p.rev ? n_tiles - 1 - ti : ti;
        const int nv0 = (tile / p.segs) * p.G;
        const int t0 = (tile % p.segs) * p.L;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        mbar_expect_tx(&full_bar[stage], box_bytes * (uint32_t)chunks);
        uint8_t* dst = ring + (size_t)stage * p.stage_bytes;
        for (int c = 0; c < p.kc; ++c) tma_load_3d(dst + (size_t)c * p.chunk_bytes, &p.map_h, &full_bar[stage], c * 64, t0 - 1, nv0);
        for (int c = 0; c < p.kc; ++c) tma_load_3d(dst + (size_t)(p.kc + c) * p.chunk_bytes, &p.map_x, &full_bar[stage], c * 64, t0 - 1, nv0);
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (warp-uniform loop, lane 0 issues) =====================
    const uint32_t idesc = make_idesc_bf16(128, p.N);        // M = 128 channel lanes, N = tile rows
    const bool leader = lane == 0;
    const uint32_t ring_u32 = smem_u32(ring);
    const uint64_t desc_hi = make_smem_desc_kmajor_sw128(0);
    int stage = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      const uint32_t tmem_d = tmem_acc + (uint32_t)(acc * p.acc_stride);
      const uint32_t sbase = ring_u32 + (uint32_t)stage * (uint32_t)p.stage_bytes;
      if (leader) {
        uint32_t first = 0;
        for (int c = 0; c < p.kc; ++c) {                    // H chunk c serves all three taps as row-shifted views
          const uint32_t sb = sbase + (uint32_t)c * (uint32_t)p.chunk_bytes;
#pragma unroll
          for (int tap = 0; tap < 3; ++tap) {
            const uint64_t db = desc_hi | (uint64_t)(((sb + (uint32_t)tap * 128u) >> 4) & 0x3FFF);
            const uint32_t wa = tmem_w + (uint32_t)((tap * p.c + c * 64) / 2);
#pragma unroll
            for (int k = 0; k < 4; ++k) { umma_bf16_ts(tmem_d, wa + (uint32_t)(k * 8), db + (uint64_t)(2 * k), idesc, first); first = 1; }
          }
        }
        for (int c = 0; c < p.kc; ++c) {                    // residual: identity block against the centre rows of X
          const uint32_t sb = sbase + (uint32_t)(p.kc + c) * (uint32_t)p.chunk_bytes + 128u;
          const uint64_t db = desc_hi | (uint64_t)((sb >> 4) & 0x3FFF);
          const uint32_t wa = tmem_w + (uint32_t)((3 * p.c + c * 64) / 2);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16_ts(tmem_d, wa + (uint32_t)(k * 8), db + (uint64_t)(2 * k), idesc, 1u);
        }
        umma_commit(&empty_bar[stage]);
        umma_commit(&tmem_full[acc]);
      }
      __syncwarp();
      if (++stage == p.stages) { stage = 0; phase ^= 1; }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else if (warp == 2 + kThEpiWarps) {
    // ===================== TMA-store warp =====================
    if (lane == 0) {
      int sbuf = 0; uint32_t sphase = 0;
      int prev = -1;
      for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
        const int tile = p.rev ? n_tiles - 1 - ti : ti;
        mbar_wait(&stage_full[sbuf], sphase);
        for (int c = 0; c < regions; ++c)
          tma_store_3d(&p.map_out, s_stage + ((size_t)sbuf * regions + c) * p.region_bytes, c * 64, (tile % p.segs) * p.L, (tile / p.segs) * p.G);
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
    // ===================== epilogue: 16 warps = TMEM lane group (32 channels) x interleaved 16-column chunks =====================
    // Channel-major accumulator -> row-major bf16 staging through tcgen05.ld.16x256b fragments and stmatrix.trans
    // (see rowgemm_ts_kernel).  Every lane supplies the address of one 16-byte piece; pieces of halo columns go to a
    // scratch sink.
    constexpr int kMaxChunks = 3;                           // N <= 192 columns -> at most 3 chunks of 16 per warp
    const int lane_grp = warp & 3;
    const int rq = (warp - 2) >> 2;
    const bool grp_ok = lane_grp * 32 < p.c_out;
    float bias[2][2];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int co = lane_grp * 32 + 16 * h + 8 * u + (lane >> 2);
        bias[h][u] = co < p.c_out ? __ldg(p.bias + co) : 0.f;
      }
    const int a_col = ((lane >> 4) & 1) * 8 + (lane & 7);   // column inside a 16-column chunk whose piece this lane addresses
    const int a_piece = (lane >> 3) & 1;
    const uint32_t sink = smem_u32(smem + p.off_bar + 256) + (uint32_t)lane * 16u;
    const int n_chunks16 = p.N / 16;
    int acc = 0; uint32_t acc_phase = 0;
    int sbuf = 0; uint32_t sphase = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      uint32_t a[kMaxChunks][2][8];
#pragma unroll
      for (int q = 0; q < kMaxChunks; ++q) {
        const int ch = rq + 4 * q;
        if (ch < n_chunks16) {
#pragma unroll
          for (int h = 0; h < 2; ++h)
            tmem_ld_16x256b_x2(tmem_acc + ((uint32_t)(lane_grp * 32 + 16 * h) << 16) + (uint32_t)(acc * p.acc_stride + ch * 16), a[q][h]);
        }
      }
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);          // accumulator is in registers: hand it back right away
      mbar_wait(&stage_empty[sbuf], sphase ^ 1);
      if (grp_ok) {
        const uint32_t st_u32 = smem_u32(s_stage + (size_t)sbuf * regions * p.region_bytes);
#pragma unroll
        for (int q = 0; q < kMaxChunks; ++q) {
          const int ch = rq + 4 * q;
          if (ch < n_chunks16) {
            const int n = ch * 16 + a_col;                  // column n = j*R + t  ->  row group j, frame t
            const int j = n / p.R, t = n - j * p.R;
            const bool ok = j < p.G && t < p.L;
            const int r = j * p.L + t;                      // staging row
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int co0 = lane_grp * 32 + 16 * h;
              const uint32_t piece = (uint32_t)(((co0 & 63) >> 3) + a_piece);
              uint32_t m[4];
#pragma unroll
              for (int u = 0; u < 4; ++u)                   // u = 2*(8-column block) + (channel half)
                m[u] = pack_bf16x2_relu(__uint_as_float(a[q][h][2 * u]) + bias[h][u & 1], __uint_as_float(a[q][h][2 * u + 1]) + bias[h][u & 1]);
              const uint32_t addr = ok ? st_u32 + (uint32_t)(co0 >> 6) * (uint32_t)p.region_bytes + (uint32_t)r * 128u + ((piece ^ (uint32_t)(r & 7)) << 4)
                                       : sink;
              stmatrix_x4_trans(addr, m[0], m[1], m[2], m[3]);
            }
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
struct TcnHaloPrepared {
  TcnHaloParams p;
  int smem_bytes;
  int64_t nv_cap;
};

bool tcn_halo_supported(int c, int c_out, int kt, int stride, int T, bool identity_slab) {
  if (!(identity_slab && kt == 3 && stride == 1 && c == c_out && (c_out == 64 || c_out == 128))) return false;
  (void)T;                                                   // any T: long clips are cut into segments
  return true;
}

// Segment length.  The whole clip (the tuned shapes: T = 32 at 128 channels, T = 64 at 64 channels) unless cutting it
// fills the MMA columns clearly better or the clip does not fit a tile at all.  Candidates are the divisors of T (no
// ragged last segment); score = valid rows per MMA column minus a charge for the two halo rows every segment re-loads.
static int tcn_halo_segment(int T, int n_max) {
  auto score = [&](int L) {
    const int G = n_max / (L + 2);
    if (G < 1) return -1.0;
    const int N = (G * (L + 2) + 15) / 16 * 16;
    return (double)G * L / N - 0.5 * (2.0 / L - 2.0 / T);
  };
  int best = T + 2 <= n_max ? T : 0;
  double best_s = best ? score(T) + 0.03 : -1.0;             // hysteresis: leave the whole-clip shape only for a clear win
  for (int L = std::min(T - 1, n_max - 2); L >= 8; --L) {
    if (T % L) continue;
    const double sc = score(L);
    if (sc > best_s + 1e-9) { best_s = sc; best = L; }
  }
  return best ? best : std::min(T, n_max - 2);               // no divisor fits: ragged last segment (TMA clips it)
}

int tcn_halo_prepare(const void* h, const void* x, const void* w, const float* bias, void* out, int64_t nv_cap, int T, int c,
                     TcnHaloPrepared** outp) {
  TIK_CHECK_ARG(h && x && w && bias && out && nv_cap > 0 && tcn_halo_supported(c, c, 3, 1, T, true), "halo temporal conv: unsupported shape");
  TcnHaloPrepared* g = new TcnHaloPrepared();
  TcnHaloParams& p = g->p;
  memset(&p, 0, sizeof(p));
  p.w = reinterpret_cast<const __nv_bfloat16*>(w); p.bias = bias;
  p.c = c; p.c_out = c; p.ktot = 4 * c; p.kc = c / 64;
  const int n_max = ((512 - p.ktot / 2) / 2) / 32 * 32;   // two accumulators beside the weights, 32-column pitch
  p.T = T;
  p.L = tcn_halo_segment(T, std::min(n_max, 256));
  if (const char* e = getenv("TIK_HALO_SEG")) { const int l = atoi(e); if (l >= 1 && l <= T && l + 2 <= n_max) p.L = l; }
  p.segs = (T + p.L - 1) / p.L;
  p.R = p.L + 2;
  p.G = n_max / p.R;
  if ((int64_t)p.G > nv_cap) p.G = (int)nv_cap;
  p.N = (p.G * p.R + 15) / 16 * 16;
  p.acc_stride = (p.N + 31) / 32 * 32;
  p.chunk_bytes = p.N * 128;
  if (p.chunk_bytes % 1024) p.chunk_bytes = (p.chunk_bytes / 1024 + 1) * 1024;
  p.stage_bytes = 2 * p.kc * p.chunk_bytes;
  p.region_bytes = (p.G * p.L * 128 + 1023) / 1024 * 1024;
  const int regions = c / 64;
  p.stage_bufs = 2;
  p.stages = (kThSmemBudget - 768 - p.stage_bufs * regions * p.region_bytes) / p.stage_bytes;
  if (p.stages > kThMaxStages) p.stages = kThMaxStages;
  if (p.stages < 2) { delete g; set_error("halo temporal conv: shared-memory plan does not fit"); return TIK_ERR_UNSUPPORTED; }
  p.off_stage = p.stages * p.stage_bytes;
  p.off_bar = p.off_stage + p.stage_bufs * regions * p.region_bytes;
  g->smem_bytes = p.off_bar + 256 + 512 + 1024;            // barriers, stmatrix sink, alignment slack
  g->nv_cap = nv_cap;
  int rc;
  {
    uint64_t dims[3] = {(uint64_t)c, (uint64_t)T, (uint64_t)nv_cap};
    uint64_t strides[2] = {(uint64_t)c * 2, (uint64_t)c * 2 * T};
    uint32_t box[3] = {64, (uint32_t)p.R, (uint32_t)p.G};
    rc = encode_bf16_map(&p.map_h, h, 3, dims, strides, box);
    if (rc == TIK_OK) rc = encode_bf16_map(&p.map_x, x, 3, dims, strides, box);
    uint32_t obox[3] = {64, (uint32_t)p.L, (uint32_t)p.G};
    if (rc == TIK_OK) rc = encode_bf16_map(&p.map_out, out, 3, dims, strides, obox);
  }
  if (rc != TIK_OK) { delete g; return rc; }
  *outp = g;
  return TIK_OK;
}

int tcn_halo_launch(TcnHaloPrepared* g, int64_t nv, cudaStream_t s) {
  TIK_CHECK_ARG(g && nv <= g->nv_cap, "halo temporal conv: nv exceeds the prepared capacity");
  if (nv <= 0) return TIK_OK;
  TcnHaloParams p = g->p;
  p.nv = nv;
  p.n_tiles = (int32_t)((nv + p.G - 1) / p.G) * p.segs;
  p.rev = launch_opts().rev;
  static bool attr_done[64] = {};
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  if (!attr_done[dev & 63]) {
    TIK_CUDA(cudaFuncSetAttribute(tcn_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kThSmemBudget + 2048));
    attr_done[dev & 63] = true;
  }
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const unsigned grid = (unsigned)std::min<int64_t>(p.n_tiles, sms);
  TIK_CUDA(launch_pdl(tcn_halo_kernel, grid, kThThreads, (size_t)g->smem_bytes, s, p));
  return TIK_OK;
}

void tcn_halo_free(TcnHaloPrepared* g) { delete g; }

}  // namespace tik
