// Prepared (tensor maps encoded once) launches of the tcgen05 implicit GEMM.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "tik_common.cuh"

namespace tik {
struct UmmaPrepared;
// Encodes the TMA tensor maps for `d` with room for nv_capacity row groups (host-only work).
int umma_prepare(const TikRowGemm* d, int64_t nv_capacity, UmmaPrepared** out);
// Launch with the current nv / bias / residual / output fields of `d` (slab tensors are those baked at prepare time).
int umma_launch(UmmaPrepared* u, const TikRowGemm* d, cudaStream_t s);
void umma_free(UmmaPrepared* u);
struct GcnFusedPrepared;
bool gcn_fused_supported(int cin, int cout, int V, int K);
int gcn_fused_frames(int T, int cin); // frames per tile = the block size of the Abd operand
int gcn_fused_prepare(const void* x, const void* abd, const void* w, const float* bias, void* out, int64_t n_clips, int T, int V,
                      int cin, int cout, int relu, GcnFusedPrepared** outp);
int gcn_fused_launch(GcnFusedPrepared* g, int64_t n_clips, cudaStream_t s);
void gcn_fused_free(GcnFusedPrepared* g);
// 128B-swizzled bf16 tiled tensor map (rank <= 5, unit element strides), defined in gcn_fused.cu
int encode_bf16_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides, const uint32_t* box);
struct StemBlockPrepared;
// Whole first ST-GCN block (data_bn + graph conv + temporal conv + residual) in one kernel; stem_block.cu
bool stem_block_supported(const TikNet* net, int dtype);
int64_t stem_block_workspace_bytes();
int stem_block_prepare(const TikNet* net, void* w16_dev, void* out, int64_t n_clips, int T, StemBlockPrepared** outp);
int stem_block_launch(StemBlockPrepared* g, const float* x, int64_t n_clips, const TikWindowing& win, int64_t win_n0,
                      const WinSeqs& seqs, cudaStream_t s);
void stem_block_free(StemBlockPrepared* g);
struct TcnHaloPrepared;
// Stride-1 temporal conv + identity residual, weight-stationary, each activation row loaded once; tcn_halo.cu
bool tcn_halo_supported(int c, int c_out, int kt, int stride, int T, bool identity_slab);
int tcn_halo_prepare(const void* h, const void* x, const void* w, const float* bias, void* out, int64_t nv_cap, int T, int c,
                     TcnHaloPrepared** outp);
int tcn_halo_launch(TcnHaloPrepared* g, int64_t nv, cudaStream_t s);
void tcn_halo_free(TcnHaloPrepared* g);
}  // namespace tik
