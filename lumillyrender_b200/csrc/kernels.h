// kernels.h — host-callable launchers of the kernels in kernels.cu
#pragma once
#include "device_scene.h"

namespace lr {
// the render kernel (persistent.cuh).  *next_unit must be 0 on `stream` before the launch.
cudaError_t launch_render_persistent(const DevScene& sc, const DevParams& p, bool has_ggx, bool count, float* out_sum, float* out_sumsq,
                                     unsigned long long* counters, unsigned int* next_unit, int sm_count, cudaStream_t stream);
#define LR_DECL_INST(name)                                                                                              \
  cudaError_t name(const DevScene& sc, const DevParams& p, bool count, float* out_sum, float* out_sumsq,                \
                   unsigned long long* counters, unsigned int* next_unit, int sm_count, cudaStream_t stream);
LR_DECL_INST(launch_persistent_i0_t0_g0) LR_DECL_INST(launch_persistent_i0_t1_g0)
LR_DECL_INST(launch_persistent_i1_t0_g0) LR_DECL_INST(launch_persistent_i1_t1_g0)
LR_DECL_INST(launch_persistent_i0_t0_g1) LR_DECL_INST(launch_persistent_i0_t1_g1)
LR_DECL_INST(launch_persistent_i1_t0_g1) LR_DECL_INST(launch_persistent_i1_t1_g1)
#undef LR_DECL_INST
cudaError_t launch_reduce_splits(float* dst, const float* partial, size_t n, int splits, cudaStream_t stream);
cudaError_t launch_scale(float* dst, size_t n, float divisor, cudaStream_t stream);
// lr_render_multi: the per-device sum buffers (peer pointers), added in order by one kernel on the first device
constexpr int kMaxPeers = 8;
struct PeerBuffers { const float* p[kMaxPeers]; int count; };
cudaError_t launch_reduce_peers(float* dst, const PeerBuffers& src, size_t n, float divisor, cudaStream_t stream);
// lr_multi_film: each pixel from the buffer of the device that owns its tile (shard_of_tile / shard_device), / divisor if > 0
cudaError_t launch_gather_shards(float* dst, const PeerBuffers& src, int crop_w, int crop_h, int n_shards, float divisor, cudaStream_t stream);
cudaError_t launch_primary(const DevScene& sc, float u, float v, float ua, float va, int* prim, float* t, cudaStream_t stream);
cudaError_t launch_aov(const DevScene& sc, const DevParams& p, int kind, float* out, cudaStream_t stream);
cudaError_t launch_rays(const DevScene& sc, long long n, const float* org, const float* dir, int* prim, float* t, float* nout,
                        bool render_query, cudaStream_t stream);

cudaError_t launch_read_bw(const float4* buf, size_t n4, int iters, int blocks, float* sink, cudaStream_t stream);
}  // namespace lr
