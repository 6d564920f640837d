// Explicit instantiations of the tiled kernel, group 7 (instances_g7.inc: persistent CTAs); see nlm_tiled_launch.cuh.
#include "nlm_tiled_launch.cuh"

#define TILED_INSTP(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                \
    template cudaError_t launch_tiled<float, NV4, FW, FX, FR, L, NW, CH, NEFF, false, false, true>(   \
        const CUtensorMap&, const ndnlm::DevParams&, const void*, void*, int*, int, size_t, cudaStream_t);
#include "instances_g7.inc"
