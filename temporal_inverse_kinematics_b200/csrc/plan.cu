// Whole-network launch plan: PoseRegressor.forward (pose_trainer.py:94-133) =
// StgGcn18 backbone (st_gcn_aaai18.py:113-133) + Linear/LeakyReLU/Linear head, as a fixed sequence of
// kernels over caller-owned workspace.
//
// The backbone runs n_chunk clips at a time so that the per-layer activations of a chunk stay resident in
// the 126 MB L2 between producer and consumer kernels; the last block writes its (N,T',V*C) features into a
// batch-level buffer and the two head GEMMs then run ONCE over up to n_max clips (a per-chunk head would be
// a handful of CTAs on a 148-SM part).
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "tik_common.cuh"
#include "umma_prepared.h"

namespace tik {

static thread_local char g_err[512] = "";

bool pdl_enabled() {
  static int v = -1;
  if (v < 0) v = getenv("TIK_NO_PDL") ? 0 : 1;
  return v != 0;
}

LaunchOpts& launch_opts() {
  static thread_local LaunchOpts o = {0};
  return o;
}
// Serpentine tile order (tik_common.cuh LaunchOpts): TIK_SERPENTINE = 0 | 1.
// Measured on one box, three alternating rounds (tools/ab_env.sh, profiles/r2_ab_serpentine.log), sum of the 17 network
// launches of a configs[2] step: serpentine 3653-3658 us vs 3672-3700 us (on by default).
static int serpentine_enabled() {           // read per run (two getenv calls): tests and A/B tools flip it inside one process
  const char* e = getenv("TIK_SERPENTINE");
  return e ? atoi(e) : 1;
}

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static int out_frames(int t, int stride) { return (t - 1) / stride + 1; }
static int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

struct Step {
  enum Kind { STEM = 0, AGG = 1, GEMM = 2, FUSED_GCN = 3, STEM_BLOCK = 4, TCN_HALO = 5 } kind;
  GcnFusedPrepared* fused = nullptr;
  StemBlockPrepared* stem_block = nullptr;
  TcnHaloPrepared* halo = nullptr;
  double fused_flops_per_clip = 0;
  TikRowGemm g;               // GEMM
  UmmaPrepared* prep = nullptr;
  const void* src = nullptr;  // AGG input
  void* dst = nullptr;        // STEM / AGG output
  void* dst2 = nullptr;       // STEM residual output
  int t = 0, c = 0;
  const TikBlock* blk = nullptr;
  bool out_is_feat = false;   // GEMM: writes the batch-level feature buffer at the chunk's offset
  bool out_is_poses = false;  // GEMM: writes the caller's poses pointer
  int k_identity = 0;         // GEMM: K columns that only carry an identity residual (not algorithmic FLOPs)
  const float* w_big = nullptr;   // fp32 GEMM: the weights split into their TF32 parts once per plan (rowgemm_tf32.cu)
  const float* w_small = nullptr;
};

}  // namespace tik

struct TikPlan {
  TikNet net;
  int dtype;
  int64_t n_chunk, n_max;
  int T, T_out;
  size_t es;                  // element size of activations
  std::vector<tik::Step> chunk_steps, batch_steps;
  uint8_t* feat = nullptr;    // (n_max, T', V*C_last) activation dtype
  int64_t feat_elems_per_clip = 0;
  int c_last = 0;
  ~TikPlan() {
    for (auto* v : {&chunk_steps, &batch_steps})
      for (auto& s : *v)
      {
        if (s.prep) tik::umma_free(s.prep);
        if (s.fused) tik::gcn_fused_free(s.fused);
        if (s.stem_block) tik::stem_block_free(s.stem_block);
        if (s.halo) tik::tcn_halo_free(s.halo);
      }
  }
};

namespace tik {

struct WsLayout {
  int64_t off_x0, off_x1, off_agg, off_h, off_r0, off_feat, off_z, off_abd, off_w16, off_wsplit, total_bytes;
};

static int check_net(const TikNet* net, int dtype) {
  TIK_CHECK_ARG(net != nullptr, "null net");
  TIK_CHECK_ARG(dtype == TIK_F32 || dtype == TIK_BF16, "bad dtype %d", dtype);
  TIK_CHECK_ARG(net->n_blocks >= 1 && net->n_blocks <= TIK_MAX_BLOCKS, "n_blocks=%d", net->n_blocks);
  TIK_CHECK_ARG(net->V >= 1 && net->V <= 32 && net->K >= 1 && net->K <= 5, "V=%d K=%d unsupported", net->V, net->K);
  TIK_CHECK_ARG(net->c_in >= 1 && net->c_in <= 8 && net->c_in * net->K <= 16, "stem needs c_in <= 8 and K*c_in <= 16 (got c_in=%d K=%d)", net->c_in, net->K);
  TIK_CHECK_ARG(net->blocks[0].c_in == net->c_in, "block 0 c_in mismatch");
  const int cmul = dtype == TIK_BF16 ? 64 : 8;
  for (int i = 0; i < net->n_blocks; ++i) {
    const TikBlock& b = net->blocks[i];
    TIK_CHECK_ARG(b.kt >= 1 && (b.kt % 2) == 1 && b.kt + 1 <= TIK_MAX_SLABS, "block %d: temporal kernel %d unsupported", i, b.kt);
    TIK_CHECK_ARG(!b.res_as_slab || dtype == TIK_BF16, "block %d: res_as_slab is a tensor-core packing", i);
    TIK_CHECK_ARG(b.stride >= 1 && b.stride <= 8, "block %d: stride %d", i, b.stride);
    TIK_CHECK_ARG(b.c_out % cmul == 0, "block %d: c_out=%d must be a multiple of %d for this dtype", i, b.c_out, cmul);
    if (i > 0) {
      TIK_CHECK_ARG(b.c_in == net->blocks[i - 1].c_out, "block %d: c_in does not chain", i);
      TIK_CHECK_ARG(b.res_kind == TIK_RES_NONE || b.res_kind == TIK_RES_IDENTITY || b.res_kind == TIK_RES_CONV, "block %d: res_kind", i);
    } else {
      TIK_CHECK_ARG(b.res_kind == TIK_RES_NONE || b.res_kind == TIK_RES_STEM, "block 0: residual must be none or stem-conv");
      TIK_CHECK_ARG(b.res_kind != TIK_RES_STEM || (b.c_in <= 8 && b.w_res_stem_dev), "block 0: stem residual needs c_in <= 8");
    }
    TIK_CHECK_ARG(b.agg_dev && b.w_gcn_dev && b.b_gcn_dev && b.w_tcn_dev && b.b_tcn_dev, "block %d: null weight pointer", i);
  }
  if (net->head_hidden > 0) {
    TIK_CHECK_ARG(net->w1_dev && net->b1_dev && net->w2_dev && net->b2_dev && net->head_out > 0, "head pointers");
    TIK_CHECK_ARG(net->head_hidden % cmul == 0, "head hidden=%d must be a multiple of %d", net->head_hidden, cmul);
  }
  return TIK_OK;
}

static void ws_layout(const TikNet* net, int dtype, int64_t n, int64_t n_max, int T, WsLayout* L, int* t_out_final) {
  const int64_t V = net->V;
  int t = T;
  int64_t x = 0, a = 0, h = 0, r0 = 0;
  for (int i = 0; i < net->n_blocks; ++i) {
    const TikBlock& b = net->blocks[i];
    if (i > 0) {
      x = std::max<int64_t>(x, V * t * b.c_in);
      a = std::max<int64_t>(a, (int64_t)net->K * V * t * b.c_in);
    }
    h = std::max<int64_t>(h, V * t * b.c_out);
    t = out_frames(t, b.stride);
    if (i == 0 && b.res_kind == TIK_RES_STEM) r0 = V * t * b.c_out;
    if (i + 1 < net->n_blocks) x = std::max<int64_t>(x, V * t * b.c_out);
  }
  *t_out_final = t;
  const int64_t es = dtype == TIK_BF16 ? 2 : 4;
  const int64_t feat = V * t * net->blocks[net->n_blocks - 1].c_out;
  const int64_t z = net->head_hidden > 0 ? (int64_t)t * net->head_hidden : 0;
  int64_t off = 0;
  L->off_x0 = off; off = align_up(off + x * n * es, 1024);
  L->off_x1 = off; off = align_up(off + x * n * es, 1024);
  L->off_agg = off; off = align_up(off + a * n * es, 1024);
  L->off_h = off; off = align_up(off + h * n * es, 1024);
  L->off_r0 = off; off = align_up(off + r0 * n * es, 1024);
  L->off_feat = off; off = align_up(off + feat * n_max * es, 1024);
  L->off_z = off; off = align_up(off + z * n_max * es, 1024);
  L->off_abd = off; off = align_up(off + (int64_t)net->n_blocks * 128 * 128 * 2, 1024);
  L->off_w16 = off; off = align_up(off + stem_block_workspace_bytes(), 1024);
  L->off_wsplit = off;                                                       // fp32 plans: every GEMM's weights as TF32 big / small parts
  if (dtype == TIK_F32) {
    int64_t w_elems = 0;
    for (int i = 0; i < net->n_blocks; ++i) {          // only the 64-column GEMMs read pre-split weights (rowgemm_tf32.cu)
      const TikBlock& b = net->blocks[i];
      if (b.c_out <= 64) w_elems += align_up((int64_t)b.c_out * net->K * b.c_in, 256) + align_up((int64_t)b.c_out * (b.kt * b.c_out + b.c_in), 256);
    }
    if (net->head_hidden > 0 && net->head_hidden <= 64) w_elems += align_up((int64_t)net->head_hidden * V * net->blocks[net->n_blocks - 1].c_out, 256);
    if (net->head_hidden > 0 && net->head_out <= 64) w_elems += align_up((int64_t)net->head_out * net->head_hidden, 256);
    off = align_up(off + 2 * w_elems * 4, 1024);
  }
  L->total_bytes = off;
}

// Clip k of the n clips of this step is window win_n0 + k of x read through win (the stem steps; the other steps read
// the workspace).
static int run_step(TikPlan* P, Step& st, const float* x, int64_t n, int64_t clip_off, float* poses, cudaStream_t s,
                    const TikWindowing& win, int64_t win_n0, const WinSeqs& seqs) {
  const TikNet& net = P->net;
  const int V = net.V;
  if (st.kind == Step::STEM) {
    const TikBlock& b = *st.blk;
    return stem_gcn_impl(P->dtype, x, net.in_scale_dev, net.in_shift_dev, b.agg_dev, reinterpret_cast<const float*>(b.w_gcn_dev),
                         b.b_gcn_dev, st.dst, st.dst2 ? b.w_res_stem_dev : nullptr, st.dst2, b.stride, n, st.t, V, b.c_in, net.K,
                         b.c_out, 1, win, win_n0, seqs, s);
  }
  if (st.kind == Step::AGG) {
    // planes are spaced for a full chunk (the tensor maps are baked for n_chunk clips)
    return tik_aggregate(P->dtype, st.src, st.blk->agg_dev, st.dst, P->n_chunk, st.t, V, st.c, net.K, s);
  }
  if (st.kind == Step::FUSED_GCN) return gcn_fused_launch(st.fused, n, s);
  if (st.kind == Step::STEM_BLOCK) return stem_block_launch(st.stem_block, x, n, win, win_n0, seqs, s);
  if (st.kind == Step::TCN_HALO) return tcn_halo_launch(st.halo, n * V, s);
  TikRowGemm g = st.g;
  if (g.v == 1) {             // head: rows = n * T'
    g.t_out = (int32_t)(n * P->T_out);
    g.slabs[0].t_in = g.t_out;
  } else {
    g.nv = n * V;
  }
  if (st.out_is_feat) g.out_dev = P->feat + clip_off * P->feat_elems_per_clip * (int64_t)P->es;
  if (st.out_is_poses) g.out_dev = poses;
  return P->dtype == TIK_BF16 ? umma_launch(st.prep, &g, s) : rowgemm_f32_presplit(&g, st.w_big, st.w_small, s);
}

// Every run of a plan: clip n of the N clips is window n of x read through win.  The entry points check win itself (or
// build it for a plain batch: plain_windowing); every other argument check of the four of them is here.
static int run_impl(TikPlan* P, const float* x, const TikWindowing& win, const WinSeqs& seqs, int64_t N, float* poses,
                    void* feat_out, cudaStream_t s, std::vector<cudaEvent_t>* events = nullptr,
                    std::vector<std::pair<Step*, int64_t>>* trace = nullptr) {
  TIK_CHECK_ARG(P != nullptr, "plan: null plan");
  TIK_CHECK_ARG(x != nullptr, "plan: null input pointer");
  TIK_CHECK_ARG(N >= 0, "plan: N = %lld < 0", (long long)N);
  TIK_CHECK_ARG(win.root_a < P->net.V && win.root_b < P->net.V, "plan: root keypoints (%d, %d) must be < V = %d",
                win.root_a, win.root_b, P->net.V);
  TIK_CHECK_ARG(P->net.head_hidden == 0 || poses, "plan: poses pointer required");
  const TikNet& net = P->net;
  auto mark = [&](Step* st, int64_t n) -> int {
    if (!events) return TIK_OK;
    cudaEvent_t e;
    TIK_CUDA(cudaEventCreate(&e));
    TIK_CUDA(cudaEventRecord(e, s));
    events->push_back(e);
    if (st) trace->push_back({st, n});
    return TIK_OK;
  };
  const int serp = serpentine_enabled();
  for (int64_t b0 = 0; b0 < N; b0 += P->n_max) {
    const int64_t nb = std::min<int64_t>(P->n_max, N - b0);
    for (int64_t n0 = 0; n0 < nb; n0 += P->n_chunk) {
      const int64_t n = std::min<int64_t>(P->n_chunk, nb - n0);
      int k = 0;
      for (auto& st : P->chunk_steps) {
        int rc = mark(&st, n);
        if (rc != TIK_OK) return rc;
        launch_opts() = {serp ? (k & 1) : 0};              // consecutive kernels walk the clips in opposite directions
        rc = run_step(P, st, x, n, n0, nullptr, s, win, b0 + n0, seqs);
        launch_opts() = {0};
        if (rc != TIK_OK) return rc;
        ++k;
      }
    }
    int k = (int)P->chunk_steps.size();
    for (auto& st : P->batch_steps) {
      int rc = mark(&st, nb);
      if (rc != TIK_OK) return rc;
      launch_opts() = {serp && nb <= P->n_chunk ? (k & 1) : 0};   // several chunks: the features were not written in one sweep
      rc = run_step(P, st, nullptr, nb, 0, poses ? poses + b0 * (int64_t)P->T_out * net.head_out : nullptr, s, win, 0, seqs);
      launch_opts() = {0};
      if (rc != TIK_OK) return rc;
      ++k;
    }
    if (feat_out) {
      TIK_CUDA(cudaMemcpyAsync(reinterpret_cast<uint8_t*>(feat_out) + b0 * P->feat_elems_per_clip * (int64_t)P->es, P->feat,
                               (size_t)(nb * P->feat_elems_per_clip) * P->es, cudaMemcpyDeviceToDevice, s));
    }
  }
  return mark(nullptr, 0);
}

}  // namespace tik

extern "C" {

int tik_version(void) { return 104; }
const char* tik_last_error(void) { return tik::g_err; }

int tik_check_device(void) {
  using namespace tik;
  int dev = 0;
  TIK_CUDA(cudaGetDevice(&dev));
  int major = 0;
  TIK_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) {
    set_error("libtik.so is built for sm_100a only; device %d has compute capability major %d", dev, major);
    return TIK_ERR_UNSUPPORTED;
  }
  return TIK_OK;
}

int tik_stgcn_out_frames(const TikNet* net, int T) {
  if (!net || T < 1) return -1;
  int t = T;
  for (int i = 0; i < net->n_blocks; ++i) t = tik::out_frames(t, net->blocks[i].stride);
  return t;
}

int tik_stgcn_workspace_bytes(const TikNet* net, int dtype, int64_t n_chunk, int64_t n_max, int T, int64_t* bytes) {
  using namespace tik;
  int rc = check_net(net, dtype);
  if (rc != TIK_OK) return rc;
  TIK_CHECK_ARG(n_chunk >= 1 && n_max >= n_chunk && T >= 1 && bytes, "bad arguments");
  WsLayout L;
  int tf;
  ws_layout(net, dtype, n_chunk, n_max, T, &L, &tf);
  *bytes = L.total_bytes;
  return TIK_OK;
}

int tik_stgcn_plan_create(const TikNet* net, int dtype, int64_t n_chunk, int64_t n_max, int T, void* workspace,
                          int64_t ws_bytes, TikPlan** plan_out) {
  using namespace tik;
  int rc = check_net(net, dtype);
  if (rc != TIK_OK) return rc;
  TIK_CHECK_ARG(n_chunk >= 1 && n_max >= n_chunk && T >= 1 && plan_out, "bad arguments");
  WsLayout L;
  int tf;
  ws_layout(net, dtype, n_chunk, n_max, T, &L, &tf);
  if (!workspace || ws_bytes < L.total_bytes) {
    set_error("workspace of %lld bytes is smaller than the %lld bytes this plan needs", (long long)ws_bytes, (long long)L.total_bytes);
    return TIK_ERR_WORKSPACE;
  }
  TIK_CHECK_ARG(((uintptr_t)workspace & 1023) == 0, "workspace must be 1024-byte aligned");
  TIK_CHECK_ARG(n_max * tf < (1ll << 31), "n_max * T' too large for one head launch");
  TikPlan* P = new TikPlan();
  P->net = *net; P->dtype = dtype; P->n_chunk = n_chunk; P->n_max = n_max; P->T = T; P->T_out = tf;
  P->es = dtype == TIK_BF16 ? 2 : 4;
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  void* xbuf[2] = {ws + L.off_x0, ws + L.off_x1};
  void* agg = ws + L.off_agg;
  void* hbuf = ws + L.off_h;
  void* r0buf = ws + L.off_r0;
  void* zbuf = ws + L.off_z;
  P->feat = ws + L.off_feat;
  const int V = net->V, K = net->K;
  const int64_t nv = n_chunk * V;
  int t = T;
  int cur = 0;   // xbuf[cur] holds the input of the next block (from block 1 on)
  for (int i = 0; i < net->n_blocks; ++i) {
    const TikBlock& b = P->net.blocks[i];
    const int pad = (b.kt - 1) / 2;
    const int t_o = out_frames(t, b.stride);
    const bool last = i == net->n_blocks - 1;
    if (i == 0 && net->n_blocks > 1 && stem_block_supported(net, dtype) && !getenv("TIK_NO_STEM_BLOCK")) {
      // the whole first block in one kernel: neither H0 nor the residual branch touches HBM
      Step s; s.kind = Step::STEM_BLOCK; s.blk = &b; s.t = t;
      int rcs = stem_block_prepare(&P->net, ws + L.off_w16, xbuf[0], n_chunk, t, &s.stem_block);
      if (rcs != TIK_OK) { delete P; return rcs; }
      s.fused_flops_per_clip = 2.0 * V * t * (double)b.c_out * (K * b.c_in + b.kt * b.c_out + (b.res_kind == TIK_RES_STEM ? b.c_in : 0));
      P->chunk_steps.push_back(s);
      cur = 0;
      t = t_o;
      continue;
    }
    if (i == 0) {
      Step s; s.kind = Step::STEM; s.dst = hbuf; s.t = t; s.blk = &b;
      s.dst2 = b.res_kind == TIK_RES_STEM ? r0buf : nullptr;
      P->chunk_steps.push_back(s);
    } else if (dtype == TIK_BF16 && gcn_fused_supported(b.c_in, b.c_out, V, K) && !getenv("TIK_NO_FUSED_GCN")) {
      // aggregation + channel GEMM in one kernel: build the block-structured bf16 operand Abd in the workspace
      const int f = gcn_fused_frames(t, b.c_in);
      std::vector<float> a_host((size_t)V * V);
      cudaError_t ce = cudaMemcpy(a_host.data(), b.agg_dev, a_host.size() * sizeof(float), cudaMemcpyDeviceToHost);
      std::vector<__nv_bfloat16> abd_host(128 * 128, __float2bfloat16_rn(0.f));
      for (int w = 0; w < V; ++w)
        for (int v = 0; v < V; ++v)
          for (int q = 0; q < f; ++q) abd_host[(size_t)(w * f + q) * 128 + (v * f + q)] = __float2bfloat16_rn(a_host[(size_t)v * V + w]);
      void* abd_dev = ws + L.off_abd + (int64_t)i * 128 * 128 * 2;
      if (ce == cudaSuccess) ce = cudaMemcpy(abd_dev, abd_host.data(), abd_host.size() * 2, cudaMemcpyHostToDevice);
      if (ce != cudaSuccess) { set_error("plan: Abd upload failed: %s", cudaGetErrorString(ce)); delete P; return TIK_ERR_CUDA; }
      Step s; s.kind = Step::FUSED_GCN; s.blk = &b; s.t = t;
      int rcf = gcn_fused_prepare(xbuf[cur], abd_dev, b.w_gcn_dev, b.b_gcn_dev, hbuf, n_chunk, t, V, b.c_in, b.c_out, 1, &s.fused);
      if (rcf != TIK_OK) { delete P; return rcf; }
      s.fused_flops_per_clip = 2.0 * V * t * (double)b.c_in * b.c_out;
      P->chunk_steps.push_back(s);
    } else {
      Step s; s.kind = Step::AGG; s.src = xbuf[cur]; s.dst = agg; s.t = t; s.c = b.c_in; s.blk = &b;
      P->chunk_steps.push_back(s);
      Step g; g.kind = Step::GEMM; memset(&g.g, 0, sizeof(g.g));
      g.g.n_slabs = K;
      for (int k = 0; k < K; ++k)
        g.g.slabs[k] = {reinterpret_cast<uint8_t*>(agg) + (int64_t)k * nv * t * b.c_in * P->es, b.c_in, t, 1, 0};
      g.g.w_dev = b.w_gcn_dev; g.g.bias_dev = b.b_gcn_dev; g.g.bias_per_node = 1;
      g.g.nv = nv; g.g.v = V; g.g.t_out = t; g.g.c_out = b.c_out; g.g.c_out_valid = b.c_out;
      g.g.act = TIK_ACT_RELU; g.g.res_kind = TIK_RES_NONE;
      g.g.out_dev = hbuf; g.g.out_layout = TIK_OUT_NODE_MAJOR;
      P->chunk_steps.push_back(g);
    }
    if (dtype == TIK_BF16 && !last && b.res_kind == TIK_RES_IDENTITY &&
        tcn_halo_supported(b.c_in, b.c_out, b.kt, b.stride, t, b.res_as_slab != 0) && !getenv("TIK_NO_TCN_HALO")) {
      // stride-1 block with an identity residual: one halo tile serves all three taps (tcn_halo.cu)
      const int nxt_h = (i == 0) ? 0 : cur ^ 1;
      Step hs; hs.kind = Step::TCN_HALO; hs.blk = &b; hs.t = t;
      int rch = tcn_halo_prepare(hbuf, xbuf[cur], b.w_tcn_dev, b.b_tcn_dev, xbuf[nxt_h], nv, t, b.c_out, &hs.halo);
      if (rch != TIK_OK) { delete P; return rch; }
      hs.fused_flops_per_clip = 2.0 * V * t * (double)b.c_out * (b.kt * b.c_out);
      P->chunk_steps.push_back(hs);
      cur = nxt_h;
      t = t_o;
      continue;
    }
    Step c; c.kind = Step::GEMM; memset(&c.g, 0, sizeof(c.g));
    int ns = 0;
    for (int dt = 0; dt < b.kt; ++dt) c.g.slabs[ns++] = {hbuf, b.c_out, t, b.stride, dt - pad};
    if (b.res_kind == TIK_RES_CONV) c.g.slabs[ns++] = {xbuf[cur], b.c_in, t, b.stride, 0};
    if (b.res_as_slab && b.res_kind == TIK_RES_IDENTITY) { c.g.slabs[ns++] = {xbuf[cur], b.c_out, t_o, 1, 0}; c.k_identity = b.c_out; }
    if (b.res_as_slab && b.res_kind == TIK_RES_STEM) { c.g.slabs[ns++] = {r0buf, b.c_out, t_o, 1, 0}; c.k_identity = b.c_out; }
    c.g.n_slabs = ns;
    c.g.w_dev = b.w_tcn_dev; c.g.bias_dev = b.b_tcn_dev; c.g.bias_per_node = (b.res_kind == TIK_RES_STEM) ? 1 : 0;
    c.g.nv = nv; c.g.v = V; c.g.t_out = t_o; c.g.c_out = b.c_out; c.g.c_out_valid = b.c_out;
    c.g.act = TIK_ACT_RELU;
    if (b.res_as_slab) c.g.res_kind = TIK_RES_NONE;
    else if (b.res_kind == TIK_RES_IDENTITY) { c.g.res_kind = TIK_RES_IDENTITY; c.g.res_dev = xbuf[cur]; }
    else if (b.res_kind == TIK_RES_STEM) { c.g.res_kind = TIK_RES_IDENTITY; c.g.res_dev = r0buf; }   // precomputed by the stem
    else c.g.res_kind = TIK_RES_NONE;
    const int nxt = (i == 0) ? 0 : cur ^ 1;
    if (last) {
      c.g.out_dev = nullptr; c.out_is_feat = true; c.g.out_layout = TIK_OUT_TIME_MAJOR;
      P->c_last = b.c_out;
    } else {
      c.g.out_dev = xbuf[nxt]; c.g.out_layout = TIK_OUT_NODE_MAJOR;
    }
    P->chunk_steps.push_back(c);
    cur = nxt;
    t = t_o;
  }
  P->feat_elems_per_clip = (int64_t)tf * V * P->c_last;
  if (net->head_hidden > 0) {
    const int feat_c = V * P->c_last;
    const int32_t rows = (int32_t)(n_max * tf);
    Step h1; h1.kind = Step::GEMM; memset(&h1.g, 0, sizeof(h1.g));
    h1.g.n_slabs = 1;
    h1.g.slabs[0] = {P->feat, feat_c, rows, 1, 0};
    h1.g.w_dev = net->w1_dev; h1.g.bias_dev = net->b1_dev; h1.g.bias_per_node = 0;
    h1.g.nv = 1; h1.g.v = 1; h1.g.t_out = rows; h1.g.c_out = net->head_hidden; h1.g.c_out_valid = net->head_hidden;
    h1.g.act = TIK_ACT_LEAKY; h1.g.slope = net->leaky_slope; h1.g.res_kind = TIK_RES_NONE;
    h1.g.out_dev = zbuf; h1.g.out_layout = TIK_OUT_NODE_MAJOR;
    P->batch_steps.push_back(h1);
    Step h2; h2.kind = Step::GEMM; memset(&h2.g, 0, sizeof(h2.g));
    h2.g.n_slabs = 1;
    h2.g.slabs[0] = {zbuf, net->head_hidden, rows, 1, 0};
    h2.g.w_dev = net->w2_dev; h2.g.bias_dev = net->b2_dev; h2.g.bias_per_node = 0;
    h2.g.nv = 1; h2.g.v = 1; h2.g.t_out = rows;
    h2.g.c_out = dtype == TIK_BF16 ? (int)align_up(net->head_out, 64) : net->head_out;
    h2.g.c_out_valid = net->head_out;
    h2.g.act = TIK_ACT_NONE; h2.g.res_kind = TIK_RES_NONE;
    h2.g.out_dev = nullptr; h2.out_is_poses = true; h2.g.out_layout = TIK_OUT_ROWS_F32;
    P->batch_steps.push_back(h2);
  }
  if (dtype == TIK_BF16) {
    for (auto* v : {&P->chunk_steps, &P->batch_steps})
      for (auto& s : *v) {
        if (s.kind != Step::GEMM) continue;
        TikRowGemm g = s.g;
        if (!g.out_dev) g.out_dev = P->feat;    // placeholder, overridden at launch
        int rc2 = umma_prepare(&g, g.nv, &s.prep);
        if (rc2 != TIK_OK) { delete P; return rc2; }
      }
  }
  if (dtype == TIK_F32 && !getenv("TIK_NO_TF32_PRESPLIT")) {
    // weights are constants of the plan (a weight update re-creates it): split them into TF32 parts once
    float* wsp = reinterpret_cast<float*>(ws + L.off_wsplit);
    for (auto* v : {&P->chunk_steps, &P->batch_steps})
      for (auto& s : *v) {
        if (s.kind != Step::GEMM || s.g.c_out > 64) continue;   // only the 64-column kernel reads pre-split weights (rowgemm_tf32.cu)
        int64_t ktot = 0;
        for (int k = 0; k < s.g.n_slabs; ++k) ktot += s.g.slabs[k].c;
        const int64_t n = align_up((int64_t)s.g.c_out * ktot, 256);
        if ((reinterpret_cast<uint8_t*>(wsp + 2 * n) - ws) > L.total_bytes) break;      // ws_layout's bound covers every GEMM; never overrun
        int rc3 = tf32_split_weights(reinterpret_cast<const float*>(s.g.w_dev), wsp, wsp + n, (int64_t)s.g.c_out * ktot, 0);
        if (rc3 != TIK_OK) { delete P; return rc3; }
        s.w_big = wsp; s.w_small = wsp + n;
        wsp += 2 * n;
      }
    cudaError_t ce = cudaStreamSynchronize(0);
    if (ce != cudaSuccess) { set_error("plan: weight split failed: %s", cudaGetErrorString(ce)); delete P; return TIK_ERR_CUDA; }
  }
  *plan_out = P;
  return TIK_OK;
}

int tik_stgcn_plan_run(TikPlan* P, const float* x, int64_t N, float* poses, void* feat_out, void* stream) {
  using namespace tik;
  return run_impl(P, x, plain_windowing(N, P ? P->T : 0), WinSeqs{}, N, poses, feat_out, (cudaStream_t)stream);
}

int tik_stgcn_plan_run_windows(TikPlan* P, const float* seq, const TikWindowing* win, int64_t n_windows, float* poses,
                               void* feat_out, void* stream) {
  using namespace tik;
  int rc = check_windowing(win, "plan");
  return rc != TIK_OK ? rc : run_impl(P, seq, *win, WinSeqs{}, n_windows, poses, feat_out, (cudaStream_t)stream);
}

int tik_stgcn_plan_run_seq_windows(TikPlan* P, const float* seq, const TikWindowing* win, const TikSeqBatch* seqs,
                                   int64_t n_windows, float* poses, void* feat_out, void* stream) {
  using namespace tik;
  int rc = check_seq_windows(win, seqs, n_windows, "plan");
  return rc != TIK_OK ? rc : run_impl(P, seq, *win, win_seqs(*seqs), n_windows, poses, feat_out, (cudaStream_t)stream);
}

int tik_stgcn_plan_profile(TikPlan* P, const float* x, int64_t N, float* poses, void* stream, double* ms_by_kind,
                           int64_t* launches_by_kind, double* flops_gemm) {
  using namespace tik;
  TIK_CHECK_ARG(ms_by_kind && launches_by_kind && flops_gemm, "plan profile: null output pointer");
  std::vector<cudaEvent_t> ev;
  std::vector<std::pair<Step*, int64_t>> trace;
  cudaStream_t s = (cudaStream_t)stream;
  int rc = run_impl(P, x, plain_windowing(N, P ? P->T : 0), WinSeqs{}, N, poses, nullptr, s, &ev, &trace);
  if (rc != TIK_OK) return rc;
  TIK_CUDA(cudaStreamSynchronize(s));
  for (int k = 0; k < 3; ++k) { ms_by_kind[k] = 0; launches_by_kind[k] = 0; }
  *flops_gemm = 0;
  for (size_t i = 0; i < trace.size(); ++i) {
    float ms = 0;
    TIK_CUDA(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
    Step& st = *trace[i].first;
    const int64_t n = trace[i].second;
    const int kind = (st.kind == Step::FUSED_GCN || st.kind == Step::STEM_BLOCK || st.kind == Step::TCN_HALO) ? (int)Step::GEMM : (int)st.kind;   // tensor-core family
    ms_by_kind[kind] += ms;
    launches_by_kind[kind] += 1;
    if (getenv("TIK_PLAN_TRACE")) {
      static const char* names[] = {"stem", "aggregate", "gemm", "fused_gcn", "stem_block", "tcn_halo"};
      int ktot = 0;
      for (int q = 0; q < st.g.n_slabs && st.kind == Step::GEMM; ++q) ktot += st.g.slabs[q].c;
      fprintf(stderr, "tik trace: step %2zu %-9s clips=%lld K=%d c_out=%d t_out=%d  %.1f us\n", i, names[st.kind], (long long)n, ktot,
              st.kind == Step::GEMM ? st.g.c_out : st.c, st.kind == Step::GEMM ? st.g.t_out : st.t, ms * 1e3);
    }
    if (st.kind == Step::FUSED_GCN || st.kind == Step::STEM_BLOCK || st.kind == Step::TCN_HALO) *flops_gemm += st.fused_flops_per_clip * (double)n;
    if (st.kind == Step::GEMM) {
      double ktot = -st.k_identity;
      for (int q = 0; q < st.g.n_slabs; ++q) ktot += st.g.slabs[q].c;
      const double rows = st.g.v == 1 ? (double)n * P->T_out : (double)n * P->net.V * st.g.t_out;
      *flops_gemm += 2.0 * rows * ktot * st.g.c_out_valid;
    }
  }
  for (auto e : ev) cudaEventDestroy(e);
  return TIK_OK;
}

int64_t tik_stgcn_plan_launches(const TikPlan* P, int64_t N) {
  if (!P || N <= 0) return 0;
  int64_t total = 0;
  for (int64_t b0 = 0; b0 < N; b0 += P->n_max) {
    const int64_t nb = std::min<int64_t>(P->n_max, N - b0);
    total += ((nb + P->n_chunk - 1) / P->n_chunk) * (int64_t)P->chunk_steps.size() + (int64_t)P->batch_steps.size();
  }
  return total;
}

void tik_stgcn_plan_destroy(TikPlan* P) { delete P; }

}  // extern "C"
