// nlm_common.cuh -- shared device/host definitions for libndnlm (sm_100a only).
//
// Vocabulary follows the reference (jnhansen/nd, nd/_filters.pyx): a *voxel* p, its *search
// window* q in p+[-r,r]^3, the *patch* d in [-f,f]^3, *variables* v.  Internally the three
// array axes are assigned three ROLES:
//     W  slowest axis of the staged cube; one warp per W row inside a CTA tile; patch sum
//        along W goes through a shared-memory exchange,
//     R  register axis: every thread owns a column of L consecutive voxels along R,
//     X  fastest axis: one lane per voxel, patch sum along X by warp shuffles.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>

#ifndef NDNLM_TILE_PROBE
#define NDNLM_TILE_PROBE 0   // 1 (development): one warp of the tiled kernel records clock64() at the phase boundaries of
                             //    every tile into DevParams::probe (tools/dev_tile_probe.py)
#endif

#ifndef __CUDA_ARCH__
#define NDNLM_HOST_SIDE 1
#endif

namespace ndnlm {

constexpr int ROLE_W = 0, ROLE_R = 1, ROLE_X = 2;

// Geometry + constants handed to every kernel (role order).
struct DevParams {
    int n[3];          // interior extent            (W, R, X)
    int rad[3];        // search radius r
    int fr[3];         // patch radius f
    int pad[3];        // r + f
    int pd[3];         // padded extent n + 2 pad
    int V;             // true number of variables
    int nv4;           // float4 groups per voxel (tiled layout), ceil(V/4)
    // tiled kernel
    int g[3];          // warp grid
    int t[3];          // valid tile extent
    int b[3];          // shared-memory box extent
    int tiles[3];      // number of tiles
    int npass;         // passes over the W search range (each keeps only its rows in shared memory)
    int ntw_pass;      // W offsets per pass
    float c1, c2;      // w = exp2(-max(D*c1 - c2, 0)),  D = raw patch sum of squared differences
    // generic kernel (double precision constants, reference arithmetic)
    double inv_norm;   // 1 / (V * prod(2f+1))          (nd/_filters.pyx:337)
    double two_sigma2; // 2 sigma^2                      (:391)
    double inv_h2;     // 1 / h^2                        (:391)
    double n_eff;      // < 0: self weight = max weight  (:406-413)
    int zero_dist;     // reference_compiled semantics with some f_i > 0 (SURVEY F1)
    int use_ldg_loader;// debugging: fill the tile with plain loads instead of TMA
#if NDNLM_TILE_PROBE
    unsigned long long* probe;   // [tile][8]: clock64() at the tile's phase boundaries, slot 7 the SM id
    int probe_cap;               // tiles the buffer holds
#endif
};

__host__ __device__ inline int reflect_index(int i, int n) {
    // reference `_idx`, EDGE_MODE_REFLECT (nd/_filters.pyx:34-40): one reflection, no edge repeat.
    if (i < 0) return -i;
    if (i >= n) return 2 * n - 2 - i;
    return i;
}

}  // namespace ndnlm
