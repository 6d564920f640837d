// nlm_tiled_launch.cuh -- launcher template of the tiled kernel.  The instantiations are spread over
// several translation units (ndnlm_tiled_g*.cu, one per instances_g*.inc) so they compile in parallel.
#pragma once
#include <atomic>

#include "nlm_tiled.cuh"

typedef cudaError_t (*tiled_launch_fn)(const CUtensorMap&, const ndnlm::DevParams&, const void*, void*, int*, int grid,
                                       size_t smem, cudaStream_t);

// T = float: staged cube / internal output are float4 per voxel group; T = double: 4 doubles (32 bytes).
template <typename T, int NV4, int FW, int FX, int FR, int L, int NWARPS, int CH, bool NEFF, bool HALF = false, bool DH = false,
          bool PERSIST = false>
cudaError_t launch_tiled(const CUtensorMap& tmap, const ndnlm::DevParams& P, const void* padded_, void* out_,
                         int* err, int grid, size_t smem, cudaStream_t st) {
    using V4 = typename ndnlm::Elem<T>::V4;
    const V4* padded = static_cast<const V4*>(padded_);
    V4* out = static_cast<V4*>(out_);
    auto kern = ndnlm::nlm_tiled_kernel<T, NV4, FW, FX, FR, L, NWARPS, CH, NEFF, HALF, DH, PERSIST>;
    // the opt-in to > 48 KB dynamic shared memory is a per-device function attribute
    static std::atomic<bool> opted_in[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || !opted_in[dev].load()) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) opted_in[dev].store(true);
    }
    if constexpr (PERSIST) {   // `grid` is the number of tiles: one CTA per SM walks them (the box fills its shared memory)
        int sms = 0;
        e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return e;
        if (grid > sms) grid = sms;
    }
    kern<<<grid, NWARPS * 32, smem, st>>>(tmap, P, padded, out, err);
    return cudaGetLastError();
}
