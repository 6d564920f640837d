// ndnlm.cu -- C ABI (include/ndnlm.h) over the sm_100a non-local-means kernels.
//
// Replaces nd/_filters.pyx::_pixelwise_nlmeans_3d (reference nd/_filters.pyx:317-420) behind the
// call site nd/filters.py:462-463.  See include/ndnlm.h for the contract of every entry point.
#include "../../include/ndnlm.h"

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "nlm_common.cuh"
#include "nlm_boxmean.cuh"
#include "nlm_generic.cuh"
#include "nlm_staging.cuh"
using namespace ndnlm;

// ------------------------------------------------------------------------------------------
// errors, launch accounting
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t e_ = (expr);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return fail(NDNLM_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// This library links its own (static) CUDA runtime, whose "current device" is separate from the caller's
// runtime (PyTorch ships another libcudart).  Every launching entry point therefore binds the device that
// OWNS the buffers it was given and restores the previous one on exit; launching on the wrong device would
// make TMA read peer memory and never complete.
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(const void* ptr) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
            cudaGetLastError();
            ok = false;
            return;
        }
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; }
        if (prev != attr.device && cudaSetDevice(attr.device) != cudaSuccess) ok = false;
        if (prev == attr.device) prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};
#define GUARD_DEVICE(ptr)                                                                    \
    DeviceGuard guard_(ptr);                                                                 \
    if (!guard_.ok) return fail(NDNLM_EINVAL, "%s is not a CUDA device pointer", #ptr)

static inline unsigned blocks_for(long long total, int threads) { return unsigned((total + threads - 1) / threads); }

// ------------------------------------------------------------------------------------------
// tiled-kernel instantiation table
// ------------------------------------------------------------------------------------------
#include "nlm_tiled_launch.cuh"

struct TiledInst {
    int elem;           // bytes per element of the staged cube the kernel computes in: 4 (float) or 8 (double)
    int minb;           // CTAs per SM the kernel is compiled for (__launch_bounds__ min blocks)
    bool half;          // the last variable group carries at most two variables (V = 5, 6): its upper lanes are skipped
    bool dh;            // double-duty halo warps (nlm_tiled.cuh, TiledCfg): nwarps warps cover nwarps + fw rows
    bool persist;       // persistent CTAs (nlm_tiled.cuh, TiledCfg): one W pass, next box loaded during the epilogue
    int nv4, fw, fx, fr, L, nwarps, ch;
    bool neff;
    size_t exch_bytes;
    tiled_launch_fn launch;
    const char* name;
};

// The instantiations live in ndnlm_tiled_g*.cu (explicit instantiation definitions); here they are only declared.
#define TILED_INST(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                        \
    extern template cudaError_t launch_tiled<float, NV4, FW, FX, FR, L, NW, CH, NEFF>(                        \
        const CUtensorMap&, const ndnlm::DevParams&, const void*, void*, int*, int, size_t, cudaStream_t);
#define TILED_INST64(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                      \
    extern template cudaError_t launch_tiled<double, NV4, FW, FX, FR, L, NW, CH, NEFF>(                       \
        const CUtensorMap&, const ndnlm::DevParams&, const void*, void*, int*, int, size_t, cudaStream_t);
#define TILED_INSTH(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                       \
    extern template cudaError_t launch_tiled<float, NV4, FW, FX, FR, L, NW, CH, NEFF, true>(                  \
        const CUtensorMap&, const ndnlm::DevParams&, const void*, void*, int*, int, size_t, cudaStream_t);
#define TILED_INSTD(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                       \
    extern template cudaError_t launch_tiled<float, NV4, FW, FX, FR, L, NW, CH, NEFF, false, true>(           \
        const CUtensorMap&, const ndnlm::DevParams&, const void*, void*, int*, int, size_t, cudaStream_t);
#define TILED_INSTD64(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                     \
    extern template cudaError_t launch_tiled<double, NV4, FW, FX, FR, L, NW, CH, NEFF, false, true>(          \
        const CUtensorMap&, const ndnlm::DevParams&, const void*, void*, int*, int, size_t, cudaStream_t);
#define TILED_INSTP(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                       \
    extern template cudaError_t launch_tiled<float, NV4, FW, FX, FR, L, NW, CH, NEFF, false, false, true>(   \
        const CUtensorMap&, const ndnlm::DevParams&, const void*, void*, int*, int, size_t, cudaStream_t);
#include "instances_g0.inc"
#include "instances_g1.inc"
#include "instances_g2.inc"
#include "instances_g3.inc"
#include "instances_g4.inc"
#include "instances_g5.inc"
#include "instances_g6.inc"
#include "instances_g7.inc"
#undef TILED_INST
#undef TILED_INST64
#undef TILED_INSTH
#undef TILED_INSTD
#undef TILED_INSTD64
#undef TILED_INSTP

#define TILED_INSTD64(NV4, FW, FX, FR, L, NW, CH, NEFF)                                              \
    {                                                                                                \
        8, 1, false, true, false, NV4, FW, FX, FR, L, NW, CH, NEFF, TiledCfg<double, NV4, FW, FX, FR, L, NW, CH, NEFF, true>::EXCH_BYTES, \
            launch_tiled<double, NV4, FW, FX, FR, L, NW, CH, NEFF, false, true>,                     \
            "nlm_tiled<double,nv4=" #NV4 ",f=(" #FW "," #FR "," #FX "),L=" #L ",warps=" #NW "(dh),ch=" #CH ",neff=" #NEFF ">" \
    },

#define TILED_INSTD(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                \
    {                                                                                                \
        4, 1, false, true, false, NV4, FW, FX, FR, L, NW, CH, NEFF, TiledCfg<float, NV4, FW, FX, FR, L, NW, CH, NEFF, true>::EXCH_BYTES, \
            launch_tiled<float, NV4, FW, FX, FR, L, NW, CH, NEFF, false, true>,                      \
            "nlm_tiled<nv4=" #NV4 ",f=(" #FW "," #FR "," #FX "),L=" #L ",warps=" #NW "(dh),ch=" #CH ",neff=" #NEFF ">" \
    },
#define TILED_INSTH(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                \
    {                                                                                                \
        4, tiled_min_blocks<float, NV4, FW, L, NW>(), true, false, false, NV4, FW, FX, FR, L, NW, CH, NEFF, TiledCfg<float, NV4, FW, FX, FR, L, NW, CH, NEFF>::EXCH_BYTES, \
            launch_tiled<float, NV4, FW, FX, FR, L, NW, CH, NEFF, true>,                             \
            "nlm_tiled<nv4=" #NV4 "(half),f=(" #FW "," #FR "," #FX "),L=" #L ",warps=" #NW ",ch=" #CH ",neff=" #NEFF ">" \
    },
#define TILED_INST(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                 \
    {                                                                                                \
        4, tiled_min_blocks<float, NV4, FW, L, NW>(), false, false, false, NV4, FW, FX, FR, L, NW, CH, NEFF, TiledCfg<float, NV4, FW, FX, FR, L, NW, CH, NEFF>::EXCH_BYTES, \
            launch_tiled<float, NV4, FW, FX, FR, L, NW, CH, NEFF>,                                   \
            "nlm_tiled<nv4=" #NV4 ",f=(" #FW "," #FR "," #FX "),L=" #L ",warps=" #NW ",ch=" #CH ",neff=" #NEFF ">" \
    },
#define TILED_INSTP(NV4, FW, FX, FR, L, NW, CH, NEFF)                                                \
    {                                                                                                \
        4, 1, false, false, true, NV4, FW, FX, FR, L, NW, CH, NEFF, TiledCfg<float, NV4, FW, FX, FR, L, NW, CH, NEFF, false, true>::EXCH_BYTES, \
            launch_tiled<float, NV4, FW, FX, FR, L, NW, CH, NEFF, false, false, true>,               \
            "nlm_tiled<nv4=" #NV4 ",f=(" #FW "," #FR "," #FX "),L=" #L ",warps=" #NW "(persist),ch=" #CH ",neff=" #NEFF ">" \
    },
#define TILED_INST64(NV4, FW, FX, FR, L, NW, CH, NEFF)                                               \
    {                                                                                                \
        8, 1, false, false, false, NV4, FW, FX, FR, L, NW, CH, NEFF, TiledCfg<double, NV4, FW, FX, FR, L, NW, CH, NEFF>::EXCH_BYTES, \
            launch_tiled<double, NV4, FW, FX, FR, L, NW, CH, NEFF>,                                  \
            "nlm_tiled<double,nv4=" #NV4 ",f=(" #FW "," #FR "," #FX "),L=" #L ",warps=" #NW ",ch=" #CH ",neff=" #NEFF ">" \
    },

// Candidates are tried in order; the first whose shared-memory box fits is used.
static const TiledInst g_tiled[] = {
#include "instances_g0.inc"
#include "instances_g1.inc"
#include "instances_g2.inc"
#include "instances_g3.inc"
#include "instances_g4.inc"
#include "instances_g5.inc"
#include "instances_g6.inc"
#include "instances_g7.inc"
};
#undef TILED_INST
#undef TILED_INST64
#undef TILED_INSTH
#undef TILED_INSTD
#undef TILED_INSTD64
#undef TILED_INSTP
static const int g_ntiled = int(sizeof(g_tiled) / sizeof(g_tiled[0]));

// ------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------
struct ndnlm_plan {
    int64_t shape[4];
    uint32_t r[3], f[3];
    double sigma, h, n_eff;
    int semantics, dtype;
    int perm[3];        // role -> user axis
    DevParams P;
    int kernel;         // NDNLM_KERNEL_GENERIC / NDNLM_KERNEL_TILED
    int inst;           // index into g_tiled
    int vec_bytes;      // tiled layout: bytes per staged voxel group, 16 (float4) or 32 (4 doubles)
    int boxmean;        // reference_compiled fast path (nlm_boxmean.cuh): staged like the tiled kernel, inst == -1
    int threads, grid;
    size_t smem;
    int elem_bytes;
    size_t padded_bytes, out_bytes;
    double flops_per_voxel;
    int64_t n_offsets;
    char name[96];
};

static const size_t kMaxSmem = 232448;   // 227 KB per CTA on sm_100a
#ifndef NDNLM_DH_MIN_FW
#define NDNLM_DH_MIN_FW 2                // float32: double-duty-halo-warp instantiations are preferred from this W patch radius on
#endif

static int largest_divisor_leq(int n, int cap) {
    int best = 1;
    for (int d = 1; d <= n; ++d)
        if (n % d == 0 && d <= cap) best = d;
    return best;
}

// Try to configure tiled instantiation `ti` for the plan's geometry; returns true if it fits.
static bool configure_tiled(ndnlm_plan* pl, const TiledInst& ti, int elem) {
    DevParams& P = pl->P;
    if (ti.elem != elem || ti.nv4 != P.nv4) return false;
    if (ti.half && P.V > 4 * ti.nv4 - 2) return false;
    if (ti.fw != P.fr[0] || ti.fr != P.fr[1] || ti.fx != P.fr[2]) return false;
    if (ti.neff != (pl->n_eff >= 0)) return false;
    const int txw = 32 - 2 * ti.fx;
    int gw, gr, gx;
    if (ti.fw > 0) {
        gw = ti.dh ? ti.nwarps + ti.fw : ti.nwarps;     // W rows of the CTA tile (patch-halo rows included)
        gr = gx = 1;
    } else {
        gw = largest_divisor_leq(ti.nwarps, P.n[0] < 1 ? 1 : P.n[0]);
        const int rem = ti.nwarps / gw;
        gx = 1;
        for (int d = 1; d <= rem; ++d)
            if (rem % d == 0 && (long long)(d - 1) * txw < P.n[2] && d * txw + 2 * ti.fx + 2 * P.rad[2] <= 256) gx = d;
        gr = rem / gx;
    }
    P.g[0] = gw; P.g[1] = gr; P.g[2] = gx;
    P.t[0] = gw - 2 * ti.fw; P.t[1] = gr * ti.L; P.t[2] = gx * txw;
    if (P.t[0] < 1) return false;
    // W search range in passes: the fewest passes whose box fits shared memory
    const int ntw = 2 * P.rad[0] + 1;
    bool fits = false;
    size_t smem = 0;
    // kernels compiled for two CTAs per SM first look for a pass count whose box lets two CTAs share the SM's shared memory;
    // persistent CTAs need the whole W search range in one box
    size_t cap = ti.minb > 1 ? (kMaxSmem / ti.minb - 1024) : kMaxSmem;
    for (int attempt = 0; attempt < 2 && !fits; ++attempt, cap = kMaxSmem)
    for (int npass = 1; npass <= (ti.persist ? 1 : ntw) && !fits; ++npass) {
        const int per = (ntw + npass - 1) / npass;
        P.npass = (ntw + per - 1) / per;
        P.ntw_pass = per;
        P.b[0] = gw + per - 1;
        P.b[1] = gr * ti.L + 2 * ti.fr + 2 * P.rad[1];
        P.b[1] |= 1;   // odd R pitch in shared memory: conflict-free LDS.128 across lanes (R is the fastest axis)
        P.b[2] = gx * txw + 2 * ti.fx + 2 * P.rad[2];
        bool ok = true;
        for (int k = 0; k < 3; ++k)
            if (P.b[k] > 256) ok = false;
        const size_t plane = ((size_t(P.b[0]) * P.b[1] * P.b[2] + 7) / 8) * 8;
        smem = size_t(ti.nv4) * plane * (4 * size_t(elem)) + ti.exch_bytes + 16 + 16 * size_t(ti.fw > 0 ? gw : ti.nwarps);
        fits = ok && smem <= cap;
    }
    if (!fits) return false;
    long long tiles = 1;
    for (int k = 0; k < 3; ++k) {
        P.tiles[k] = (P.n[k] + P.t[k] - 1) / P.t[k];
        tiles *= P.tiles[k];
    }
    if (tiles > 0x7fffffffLL) return false;
    pl->smem = smem;
    pl->threads = ti.nwarps * 32;
    pl->grid = int(tiles);
    return true;
}

extern "C" int ndnlm_plan_create(ndnlm_plan_t** out_plan, const int64_t shape[4], const uint32_t r[3],
                                 const uint32_t f[3], double sigma, double h, double n_eff, int semantics,
                                 int dtype, int kernel) {
    return ndnlm_plan_create_roles(out_plan, shape, r, f, sigma, h, n_eff, semantics, dtype, kernel, nullptr);
}

extern "C" int ndnlm_plan_create_roles(ndnlm_plan_t** out_plan, const int64_t shape[4], const uint32_t r[3],
                                       const uint32_t f[3], double sigma, double h, double n_eff, int semantics,
                                       int dtype, int kernel, const int32_t* role_axis) {
    if (!out_plan || !shape || !r || !f) return fail(NDNLM_EINVAL, "null argument");
    if (role_axis) {
        int seen = 0;
        for (int k = 0; k < 3; ++k)
            if (role_axis[k] >= 0 && role_axis[k] <= 2) seen |= 1 << role_axis[k];
        if (seen != 7) return fail(NDNLM_EINVAL, "role_axis must be a permutation of (0, 1, 2)");
    }
    *out_plan = nullptr;
    if (dtype != NDNLM_F32 && dtype != NDNLM_F64)
        return fail(NDNLM_EDTYPE, "No matching signature found (only float32 / float64 data is supported)");
    if (semantics != NDNLM_AS_WRITTEN && semantics != NDNLM_REFERENCE_COMPILED)
        return fail(NDNLM_EINVAL, "unknown semantics %d", semantics);
    for (int a = 0; a < 4; ++a)
        if (shape[a] < 1 || shape[a] > 0x3fffffff) return fail(NDNLM_EINVAL, "shape[%d]=%lld out of range", a, (long long)shape[a]);
    for (int a = 0; a < 3; ++a) {
        if ((int64_t)r[a] + (int64_t)f[a] > shape[a] - 1)
            return fail(NDNLM_ERADIUS, "r[%d]+f[%d]=%u exceeds N-1=%lld: a single reflection is undefined there", a, a,
                        r[a] + f[a], (long long)shape[a] - 1);
    }
    if (!(h != 0.0)) return fail(NDNLM_EINVAL, "h must be non-zero");
    if (n_eff >= 0 && n_eff == 1.0) return fail(NDNLM_EINVAL, "n_eff == 1 divides by zero in find_weight");

    ndnlm_plan* pl = new ndnlm_plan();
    memset(pl, 0, sizeof(*pl));
    for (int a = 0; a < 4; ++a) pl->shape[a] = shape[a];
    for (int a = 0; a < 3; ++a) { pl->r[a] = r[a]; pl->f[a] = f[a]; }
    pl->sigma = sigma; pl->h = h; pl->n_eff = n_eff; pl->semantics = semantics; pl->dtype = dtype;

    // ---- role assignment.  It must NOT depend on the extent of axis 0, so that slabs / shards cut along
    //      axis 0 (the usual 'y') run exactly the same arithmetic as the whole cube:
    //        3 filtered axes: W = axis 0, X = the wider of axes 1 and 2 (tie: 2), R = the other;
    //        2 filtered axes: the unfiltered axis is W; X = the later filtered axis unless only axis 0 is left, R = the other;
    //        1 filtered axis: X = it; R, W = the rest (R the later one);   none: X = 2, R = 1, W = 0.
    bool active[3];
    int nact = 0;
    for (int a = 0; a < 3; ++a) { active[a] = (r[a] > 0 || f[a] > 0); nact += active[a]; }
    int ax = 2, ar = 1, aw = 0;
    if (nact == 3) {
        aw = 0;
        ax = (shape[1] > shape[2]) ? 1 : 2;
        ar = 3 - ax;
    } else if (nact == 2) {
        for (int a = 0; a < 3; ++a) if (!active[a]) aw = a;
        int first = -1, second = -1;
        for (int a = 0; a < 3; ++a) if (active[a]) { if (first < 0) first = a; else second = a; }
        if (first == 0) { ax = second; ar = 0; }                       // axis 0 goes to the register role
        else { ax = (shape[first] > shape[second]) ? first : second; ar = first + second - ax; }
    } else if (nact == 1) {
        for (int a = 0; a < 3; ++a) if (active[a]) ax = a;
        ar = -1;
        for (int a = 2; a >= 0; --a) if (a != ax && ar < 0) ar = a;
        aw = 3 - ax - ar;
    }
    if (role_axis) {   // roles fixed by the caller: every shard of one array must use the layout of the whole
        aw = role_axis[ROLE_W]; ar = role_axis[ROLE_R]; ax = role_axis[ROLE_X];
    }
    pl->perm[ROLE_W] = aw; pl->perm[ROLE_R] = ar; pl->perm[ROLE_X] = ax;

    DevParams& P = pl->P;
    int n_a = 0;
    long long K = 1;
    for (int role = 0; role < 3; ++role) {
        const int a = pl->perm[role];
        P.n[role] = int(shape[a]);
        P.rad[role] = int(r[a]);
        P.fr[role] = int(f[a]);
        P.pad[role] = int(r[a] + f[a]);
        P.pd[role] = P.n[role] + 2 * P.pad[role];
        n_a += f[a] > 0;
        K *= 2 * (long long)r[a] + 1;
    }
    K -= 1;
    const int V = int(shape[3]);
    P.V = V;
    P.nv4 = (V + 3) / 4;
    const double norm = double(V) * (2.0 * f[0] + 1) * (2.0 * f[1] + 1) * (2.0 * f[2] + 1);
    P.inv_norm = 1.0 / norm;
    P.two_sigma2 = 2.0 * sigma * sigma;
    P.inv_h2 = 1.0 / (h * h);
    P.n_eff = n_eff;
    const double log2e = 1.4426950408889634;
    P.c1 = float(log2e / (norm * h * h));
    P.c2 = float(2.0 * sigma * sigma * log2e / (h * h));
    P.zero_dist = (semantics == NDNLM_REFERENCE_COMPILED) && (f[0] > 0 || f[1] > 0 || f[2] > 0);
    {
        const char* env = getenv("NDNLM_LOADER");
        P.use_ldg_loader = (env && strcmp(env, "ldg") == 0) ? 1 : 0;
    }
    pl->n_offsets = K;
    pl->flops_per_voxel = double(K) * (5.0 * V + 2.0 * n_a + 6.0 + (n_eff >= 0 ? 2.0 : 0.0)) + 3.0 * V + 3.0;

    // ---- kernel selection ----
    pl->kernel = NDNLM_KERNEL_GENERIC;
    pl->inst = -1;
    // float64 data runs on the tiled kernel only on explicit request (NDNLM_KERNEL_TILED): the cube is then staged as
    // float32 and the result widened back -- north_star's fp32 compute, ~1e-6 from the reference's float64 result.
    // float64 data: the float64 instantiations of the tiled kernel (the reference's own float64 arithmetic) by default;
    // NDNLM_KERNEL_TILED asks for the float32 instantiations instead (the cube is staged as float32 and the result
    // widened back: north_star's fp32 compute, ~1e-6 from the float64 result); NDNLM_KERNEL_TILED_F64 insists on float64.
    const bool tiled_ok = !P.zero_dist && K > 0;
    const int elem = (dtype == NDNLM_F64 && kernel != NDNLM_KERNEL_TILED) ? 8 : 4;
    if (kernel == NDNLM_KERNEL_TILED_F64 && dtype != NDNLM_F64) {
        delete pl;
        return fail(NDNLM_EINVAL, "NDNLM_KERNEL_TILED_F64 needs float64 data");
    }
    pl->vec_bytes = 4 * elem;
    if (kernel != NDNLM_KERNEL_GENERIC && tiled_ok) {
        const char* venv = getenv("NDNLM_TILED_VARIANT");   // tuning aid: force one instantiation
        const int forced = venv ? atoi(venv) : -1;
        // Three rounds over the table: the double-duty-halo-warp instantiations (instances_g6.inc) first where they are
        // enabled (by default for patch radius f_W >= NDNLM_DH_MIN_FW and for float64; NDNLM_DH=0 / 1 disables /
        // enables all of them), then the persistent-CTA instantiations (instances_g7.inc; NDNLM_PERSIST=0 disables
        // them), then everything else in file order.
        const char* denv = getenv("NDNLM_DH");
        const char* penv = getenv("NDNLM_PERSIST");
        const bool use_persist = penv ? atoi(penv) != 0 : true;
        for (int round = 0; round < 3 && pl->inst < 0; ++round) {
            for (int i = 0; i < g_ntiled; ++i) {
                if (forced >= 0 && i != forced) continue;
                // measured (profiles/r2_dh_experiment*.txt): float32 +15 % with four halo rows (f_W = 2), -1 % with two
                // (f_W = 1: that kernel is bound by the shared-memory pipe, not by latency); float64 +9 % / +24 %
                const bool use_dh = denv ? atoi(denv) != 0 : (g_tiled[i].fw >= NDNLM_DH_MIN_FW || g_tiled[i].elem == 8);
                const int group = g_tiled[i].dh ? 0 : g_tiled[i].persist ? 1 : 2;
                if (forced < 0 && (group != round || (g_tiled[i].dh && !use_dh) || (g_tiled[i].persist && !use_persist))) continue;
                if (configure_tiled(pl, g_tiled[i], elem)) {
                    pl->kernel = NDNLM_KERNEL_TILED;
                    pl->inst = i;
                    break;
                }
            }
        }
    }
    // reference_compiled semantics with some f_i > 0 and the default self weight is a reflect box mean (SURVEY.md F1):
    // separable HBM-bound fast path on the tiled staging layout
    if (kernel != NDNLM_KERNEL_GENERIC && dtype == NDNLM_F32 && P.zero_dist && n_eff < 0 && K > 0 && boxmean_supported(P)) {
        pl->kernel = NDNLM_KERNEL_TILED;
        pl->boxmean = 1;
        pl->vec_bytes = 16;
    }
    if ((kernel == NDNLM_KERNEL_TILED || kernel == NDNLM_KERNEL_TILED_F64) && pl->kernel != NDNLM_KERNEL_TILED) {
        delete pl;
        return fail(NDNLM_EINVAL, "no tiled-kernel instantiation for this configuration (dtype/V/f pattern/shared memory)");
    }
    const long long voxels = (long long)shape[0] * shape[1] * shape[2];
    const long long pvox = (long long)P.pd[0] * P.pd[1] * P.pd[2];
    if (pl->kernel == NDNLM_KERNEL_TILED) {
        pl->elem_bytes = pl->vec_bytes / 4;
        pl->padded_bytes = size_t(pvox) * P.nv4 * pl->vec_bytes;
        pl->out_bytes = size_t(voxels) * P.nv4 * pl->vec_bytes;
        if (pl->boxmean) {
            pl->threads = 256;
            pl->grid = 0;
            pl->smem = 0;
            snprintf(pl->name, sizeof(pl->name), "nlm_boxmean<ringW=%d,ringX=%d,rR=%d>[zero_dist]", boxmean_ring_for(P.rad[0]),
                     boxmean_ring_for(P.rad[2]), P.rad[1]);
        } else {
            snprintf(pl->name, sizeof(pl->name), "%s[passes=%d]", g_tiled[pl->inst].name, P.npass);
        }
    } else {
        pl->elem_bytes = (dtype == NDNLM_F64) ? 8 : 4;
        pl->padded_bytes = size_t(pvox) * V * pl->elem_bytes;
        pl->out_bytes = size_t(voxels) * V * pl->elem_bytes;
        pl->threads = 256;
        pl->grid = int(blocks_for(voxels, 256));
        pl->smem = 0;
        memset(P.g, 0, sizeof(P.g)); memset(P.t, 0, sizeof(P.t)); memset(P.b, 0, sizeof(P.b));
        memset(P.tiles, 0, sizeof(P.tiles));
        snprintf(pl->name, sizeof(pl->name), "nlm_generic<%s>%s", dtype == NDNLM_F64 ? "double" : "float",
                 P.zero_dist ? "[zero_dist]" : "");
    }
    *out_plan = pl;
    return NDNLM_OK;
}

extern "C" void ndnlm_plan_destroy(ndnlm_plan_t* plan) { delete plan; }

extern "C" int ndnlm_plan_info(const ndnlm_plan_t* pl, ndnlm_info_t* info) {
    if (!pl || !info) return fail(NDNLM_EINVAL, "null argument");
    memset(info, 0, sizeof(*info));
    info->kernel = pl->kernel;
    for (int k = 0; k < 3; ++k) {
        info->role_axis[k] = pl->perm[k];
        info->n[k] = pl->P.n[k];
        info->pad[k] = pl->P.pad[k];
        info->padded[k] = pl->P.pd[k];
        info->tile[k] = pl->P.t[k];
        info->box[k] = pl->P.b[k];
        info->warps[k] = pl->P.g[k];
    }
    info->vp = pl->kernel == NDNLM_KERNEL_TILED ? pl->P.nv4 * 4 : pl->P.V;
    info->threads = pl->threads;
    info->grid = pl->grid;
    info->smem_bytes = int(pl->smem);
    info->elem_bytes = pl->elem_bytes;
    info->n_offsets = pl->n_offsets;
    info->voxels = pl->shape[0] * pl->shape[1] * pl->shape[2];
    info->flops_per_voxel = pl->flops_per_voxel;
    info->padded_bytes = pl->padded_bytes;
    info->out_bytes = pl->out_bytes;
    snprintf(info->kernel_name, sizeof(info->kernel_name), "%s", pl->name);
    return NDNLM_OK;
}

// ------------------------------------------------------------------------------------------
// stage / unstage / halo
// ------------------------------------------------------------------------------------------
static void fill_stage_params(const ndnlm_plan* pl, const int64_t strides[4], StageParams& S) {
    for (int k = 0; k < 3; ++k) {
        S.n[k] = pl->P.n[k];
        S.pad[k] = pl->P.pad[k];
        S.pd[k] = pl->P.pd[k];
        S.rstride[k] = strides[pl->perm[k]];
    }
    S.vstride = strides[3];
    S.V = pl->P.V;
    S.nv4 = pl->P.nv4;
    S.halo_role = -1;
    S.lo_halo = S.hi_halo = 0;
}

static int role_of_axis(const ndnlm_plan* pl, int axis) {
    for (int k = 0; k < 3; ++k)
        if (pl->perm[k] == axis) return k;
    return -1;
}

extern "C" int ndnlm_stage(const ndnlm_plan_t* pl, const void* arr, const int64_t arr_strides[4], void* padded,
                           int shard_axis, int lo_edge, int hi_edge, void* stream) {
    if (!pl || !arr || !arr_strides || !padded) return fail(NDNLM_EINVAL, "null argument");
    GUARD_DEVICE(padded);
    cudaStream_t st = (cudaStream_t)stream;
    StageParams S;
    fill_stage_params(pl, arr_strides, S);
    if (shard_axis >= 0) {
        if (shard_axis > 2) return fail(NDNLM_EINVAL, "shard_axis must be -1..2");
        S.halo_role = role_of_axis(pl, shard_axis);
        if (lo_edge < NDNLM_EDGE_REFLECT || lo_edge > NDNLM_EDGE_SOURCE || hi_edge < NDNLM_EDGE_REFLECT ||
            hi_edge > NDNLM_EDGE_SOURCE)
            return fail(NDNLM_EINVAL, "unknown edge mode");
        S.lo_halo = lo_edge;
        S.hi_halo = hi_edge;
    }
    const long long pvox = (long long)S.pd[0] * S.pd[1] * S.pd[2];
    static const bool legacy_stage = getenv("NDNLM_STAGE") && strcmp(getenv("NDNLM_STAGE"), "legacy") == 0;   // debugging aid
    const long long xr_plane = (long long)S.pd[1] * S.pd[2];
    if (pl->kernel == NDNLM_KERNEL_TILED && !legacy_stage && xr_plane < (1LL << 31)) {
        // row-blocked staging kernel; one vector load per voxel when the caller's layout allows it
        const size_t vb = size_t(pl->vec_bytes);
        const bool same_type = (pl->dtype == NDNLM_F64) == (pl->vec_bytes == 32);
        bool vec = same_type && S.V % 4 == 0 && S.vstride == 1 && (reinterpret_cast<uintptr_t>(arr) % vb) == 0;
        for (int k = 0; k < 3; ++k)
            if (S.pd[k] > 1 && S.rstride[k] % 4 != 0) vec = false;
        const unsigned wblocks = unsigned((S.pd[0] + STAGE_ROWS - 1) / STAGE_ROWS);
        const dim3 grid(unsigned((xr_plane + 255) / 256), wblocks < 65535u ? wblocks : 65535u, unsigned(S.nv4));
#define NDNLM_STAGE_ROWS(TIN, V4, VEC) \
        stage_tiled_rows_kernel<TIN, V4, VEC><<<grid, 256, 0, st>>>(S, (const TIN*)arr, (V4*)padded, wblocks)
        if (pl->vec_bytes == 32) {
            if (vec) NDNLM_STAGE_ROWS(double, double4v, true); else NDNLM_STAGE_ROWS(double, double4v, false);
        } else if (pl->dtype == NDNLM_F64) {
            NDNLM_STAGE_ROWS(double, float4, false);
        } else {
            if (vec) NDNLM_STAGE_ROWS(float, float4, true); else NDNLM_STAGE_ROWS(float, float4, false);
        }
#undef NDNLM_STAGE_ROWS
    } else if (pl->kernel == NDNLM_KERNEL_TILED) {
        const long long total = pvox * S.nv4;
        if (pl->vec_bytes == 32)
            stage_tiled_kernel<double, double4v><<<blocks_for(total, 256), 256, 0, st>>>(S, (const double*)arr, (double4v*)padded);
        else if (pl->dtype == NDNLM_F64)
            stage_tiled_kernel<double, float4><<<blocks_for(total, 256), 256, 0, st>>>(S, (const double*)arr, (float4*)padded);
        else
            stage_tiled_kernel<float, float4><<<blocks_for(total, 256), 256, 0, st>>>(S, (const float*)arr, (float4*)padded);
    } else if (pl->dtype == NDNLM_F64) {
        const long long total = pvox * S.V;
        stage_generic_kernel<double><<<blocks_for(total, 256), 256, 0, st>>>(S, (const double*)arr, (double*)padded);
    } else {
        const long long total = pvox * S.V;
        stage_generic_kernel<float><<<blocks_for(total, 256), 256, 0, st>>>(S, (const float*)arr, (float*)padded);
    }
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return NDNLM_OK;
}

// The internal output of the tiled kernels is [q][W][X][R] vectors of 4 variables.  With exactly 4 variables of the
// compute type and a caller array whose strides spell that order, it IS the caller's array.
extern "C" int ndnlm_output_is_native(const ndnlm_plan_t* pl, const int64_t out_strides[4]) {
    if (!pl || !out_strides || pl->kernel != NDNLM_KERNEL_TILED) return 0;
    const DevParams& P = pl->P;
    if (P.V != 4 || P.nv4 != 1) return 0;
    if ((pl->dtype == NDNLM_F64) != (pl->vec_bytes == 32)) return 0;      // float64 data computed in float32
    const int order[3] = {ROLE_R, ROLE_X, ROLE_W};                          // fastest first, behind the variables
    long long expect = 4;
    if (out_strides[3] != 1) return 0;
    for (int k = 0; k < 3; ++k) {
        const int role = order[k];
        if (P.n[role] > 1 && out_strides[pl->perm[role]] != expect) return 0;
        expect *= P.n[role];
    }
    return 1;
}

extern "C" int ndnlm_unstage(const ndnlm_plan_t* pl, const void* internal, void* output, const int64_t out_strides[4],
                             void* stream) {
    if (!pl || !internal || !output || !out_strides) return fail(NDNLM_EINVAL, "null argument");
    GUARD_DEVICE(internal);
    cudaStream_t st = (cudaStream_t)stream;
    StageParams S;
    fill_stage_params(pl, out_strides, S);
    const long long vox = (long long)S.n[0] * S.n[1] * S.n[2];
    if (pl->kernel == NDNLM_KERNEL_TILED) {
        if (pl->vec_bytes == 32)
            unstage_tiled_kernel<double, double4v><<<blocks_for(vox * S.nv4, 256), 256, 0, st>>>(S, (const double4v*)internal, (double*)output);
        else if (pl->dtype == NDNLM_F64)
            unstage_tiled_kernel<double, float4><<<blocks_for(vox * S.nv4, 256), 256, 0, st>>>(S, (const float4*)internal, (double*)output);
        else
            unstage_tiled_kernel<float, float4><<<blocks_for(vox * S.nv4, 256), 256, 0, st>>>(S, (const float4*)internal, (float*)output);
    } else if (pl->dtype == NDNLM_F64) {
        unstage_generic_kernel<double><<<blocks_for(vox * S.V, 256), 256, 0, st>>>(S, (const double*)internal, (double*)output);
    } else {
        unstage_generic_kernel<float><<<blocks_for(vox * S.V, 256), 256, 0, st>>>(S, (const float*)internal, (float*)output);
    }
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return NDNLM_OK;
}

// The padded cube as [outer][pd_hr][inner] in units of `unit` bytes.
static void halo_geometry(const ndnlm_plan* pl, int role, long long& outer, long long& inner, int& unit) {
    const DevParams& P = pl->P;
    // memory order of the roles, slowest first: tiled [q][W][X][R], generic [W][R][X][V]
    const int tiled_order[3] = {ROLE_W, ROLE_X, ROLE_R};
    const int generic_order[3] = {ROLE_W, ROLE_R, ROLE_X};
    const int* order;
    if (pl->kernel == NDNLM_KERNEL_TILED) {
        unit = pl->vec_bytes;
        outer = P.nv4;
        inner = 1;
        order = tiled_order;
    } else {
        unit = pl->elem_bytes;
        outer = 1;
        inner = P.V;
        order = generic_order;
    }
    int pos = 0;
    while (order[pos] != role) ++pos;
    for (int k = 0; k < pos; ++k) outer *= P.pd[order[k]];
    for (int k = pos + 1; k < 3; ++k) inner *= P.pd[order[k]];
}

extern "C" size_t ndnlm_halo_bytes(const ndnlm_plan_t* pl, int axis) {
    if (!pl || axis < 0 || axis > 2) return 0;
    const int role = role_of_axis(pl, axis);
    long long outer, inner;
    int unit;
    halo_geometry(pl, role, outer, inner, unit);
    return size_t(outer) * size_t(pl->P.pad[role]) * size_t(inner) * size_t(unit);
}

template <bool PACK>
static int halo_copy(const ndnlm_plan* pl, void* padded, int axis, int side, void* msg, cudaStream_t st) {
    if (!pl || !padded || !msg) return fail(NDNLM_EINVAL, "null argument");
    if (axis < 0 || axis > 2 || side < 0 || side > 1) return fail(NDNLM_EINVAL, "bad axis/side");
    GUARD_DEVICE(padded);
    const int role = role_of_axis(pl, axis);
    const DevParams& P = pl->P;
    const long long rows = P.pad[role];
    if (rows == 0) return NDNLM_OK;
    if (P.n[role] < rows) return fail(NDNLM_EINVAL, "shard has fewer interior rows (%d) than the halo (%lld)", P.n[role], rows);
    long long outer, inner;
    int unit;
    halo_geometry(pl, role, outer, inner, unit);
    long long first;
    if (PACK) first = side == 0 ? rows : P.n[role];          // my first / last `pad` interior rows
    else      first = side == 0 ? 0 : rows + P.n[role];      // my lower / upper pad rows
    const long long total = outer * rows * inner;
    if (unit == 32)
        halo_copy_kernel<double4v, PACK><<<blocks_for(total, 256), 256, 0, st>>>((double4v*)padded, (double4v*)msg, outer, P.pd[role], inner, first, rows);
    else if (unit == 16)
        halo_copy_kernel<float4, PACK><<<blocks_for(total, 256), 256, 0, st>>>((float4*)padded, (float4*)msg, outer, P.pd[role], inner, first, rows);
    else if (unit == 8)
        halo_copy_kernel<double, PACK><<<blocks_for(total, 256), 256, 0, st>>>((double*)padded, (double*)msg, outer, P.pd[role], inner, first, rows);
    else
        halo_copy_kernel<float, PACK><<<blocks_for(total, 256), 256, 0, st>>>((float*)padded, (float*)msg, outer, P.pd[role], inner, first, rows);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return NDNLM_OK;
}

extern "C" int ndnlm_halo_pack(const ndnlm_plan_t* pl, const void* padded, int axis, int side, void* msg, void* stream) {
    return halo_copy<true>(pl, const_cast<void*>(padded), axis, side, msg, (cudaStream_t)stream);
}
extern "C" int ndnlm_halo_unpack(const ndnlm_plan_t* pl, void* padded, int axis, int side, const void* msg, void* stream) {
    return halo_copy<false>(pl, padded, axis, side, const_cast<void*>(msg), (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------
// run
// ------------------------------------------------------------------------------------------
typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static encode_tiled_fn get_encode_fn() {
    static encode_tiled_fn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (encode_tiled_fn)p;
    });
    return fn;
}

#if NDNLM_TILE_PROBE
// Development builds only (-DNDNLM_TILE_PROBE=1, tools/dev_tile_probe.py): the device buffer of [tile][8] uint64 the next
// tiled-kernel launches record their tile timelines into; cap = 0 stops recording.
static unsigned long long* g_probe = nullptr;
static int g_probe_cap = 0;
extern "C" int ndnlm_tile_probe(void* buf, int cap) {
    g_probe = static_cast<unsigned long long*>(buf);
    g_probe_cap = buf ? cap : 0;
    return NDNLM_OK;
}
#endif

extern "C" size_t ndnlm_scratch_bytes(const ndnlm_plan_t* pl) {
    if (!pl || !pl->boxmean) return 0;
    const DevParams& P = pl->P;
    return boxmean_scratch_rows(P) * P.n[1] * P.n[2] * P.nv4 * sizeof(float4);
}

extern "C" int ndnlm_run(const ndnlm_plan_t* pl, const void* padded, void* out_internal, int32_t* err_flag, void* stream) {
    return ndnlm_run_scratch(pl, padded, out_internal, err_flag, nullptr, stream);
}

extern "C" int ndnlm_run_scratch(const ndnlm_plan_t* pl, const void* padded, void* out_internal, int32_t* err_flag,
                                 void* scratch, void* stream) {
    if (!pl || !padded || !out_internal || !err_flag) return fail(NDNLM_EINVAL, "null argument");
    GUARD_DEVICE(padded);
    cudaStream_t st = (cudaStream_t)stream;
    const DevParams& P = pl->P;
    if (pl->kernel == NDNLM_KERNEL_TILED && pl->boxmean) {
        float4* inter = (float4*)scratch;
        if (!inter) CUDA_TRY(cudaMallocAsync((void**)&inter, ndnlm_scratch_bytes(pl), st));
        int nl = 0;
        cudaError_t e = boxmean_run(P, (const float4*)padded, (float4*)out_internal, inter, st, &nl);
        g_launches += nl;
        if (!scratch) cudaFreeAsync(inter, st);
        if (e != cudaSuccess) return fail(NDNLM_ECUDA, "box-mean kernels failed to launch: %s", cudaGetErrorString(e));
    } else if (pl->kernel == NDNLM_KERNEL_TILED) {
        const TiledInst& ti = g_tiled[pl->inst];
        CUtensorMap tmap;
        memset(&tmap, 0, sizeof(tmap));
        if (!P.use_ldg_loader) {
            encode_tiled_fn enc = get_encode_fn();
            if (!enc) return fail(NDNLM_ECUDA, "cuTensorMapEncodeTiled is not available from the driver");
            // padded cube [q][W][X][R] as a 5-D tensor of floats / doubles (v, r, x, w, q), innermost first
            const cuuint64_t vb = (cuuint64_t)pl->vec_bytes;
            const cuuint64_t gdim[5] = {4, (cuuint64_t)P.pd[1], (cuuint64_t)P.pd[2], (cuuint64_t)P.pd[0], (cuuint64_t)P.nv4};
            const cuuint64_t gstr[4] = {vb, (cuuint64_t)P.pd[1] * vb, (cuuint64_t)P.pd[1] * P.pd[2] * vb,
                                        (cuuint64_t)P.pd[1] * P.pd[2] * P.pd[0] * vb};
            const cuuint32_t box[5] = {4, (cuuint32_t)P.b[1], (cuuint32_t)P.b[2], (cuuint32_t)P.b[0], 1};
            const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
            CUresult cr = enc(&tmap, pl->vec_bytes == 32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<void*>(padded), gdim, gstr, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (cr != CUDA_SUCCESS) return fail(NDNLM_ECUDA, "cuTensorMapEncodeTiled failed with CUresult %d", int(cr));
        }
#if NDNLM_TILE_PROBE
        DevParams PP = P;
        PP.probe = g_probe;
        PP.probe_cap = g_probe_cap;
        cudaError_t e = ti.launch(tmap, PP, padded, out_internal, err_flag, pl->grid, pl->smem, st);
#else
        cudaError_t e = ti.launch(tmap, P, padded, out_internal, err_flag, pl->grid, pl->smem, st);
#endif
        g_launches++;
        if (e != cudaSuccess) return fail(NDNLM_ECUDA, "tiled kernel launch failed: %s", cudaGetErrorString(e));
    } else if (pl->dtype == NDNLM_F64) {
        nlm_generic_kernel<double><<<pl->grid, 256, 0, st>>>(P, (const double*)padded, (double*)out_internal, err_flag);
        g_launches++;
        CUDA_TRY(cudaGetLastError());
    } else {
        nlm_generic_kernel<float><<<pl->grid, 256, 0, st>>>(P, (const float*)padded, (float*)out_internal, err_flag);
        g_launches++;
        CUDA_TRY(cudaGetLastError());
    }
    return NDNLM_OK;
}

// ------------------------------------------------------------------------------------------
// one-call apply
// ------------------------------------------------------------------------------------------
static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

extern "C" size_t ndnlm_workspace_bytes(const ndnlm_plan_t* pl) {
    if (!pl) return 0;
    return align256(pl->padded_bytes) + align256(pl->out_bytes) + 256 + align256(ndnlm_scratch_bytes(pl));
}

extern "C" int ndnlm_apply(const ndnlm_plan_t* pl, const void* arr, const int64_t arr_strides[4], void* output,
                           const int64_t out_strides[4], void* workspace, void* stream) {
    if (!pl || !workspace) return fail(NDNLM_EINVAL, "null argument");
    GUARD_DEVICE(workspace);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* ws = (unsigned char*)workspace;
    void* padded = ws;
    void* internal = ws + align256(pl->padded_bytes);
    int32_t* flag = (int32_t*)(ws + align256(pl->padded_bytes) + align256(pl->out_bytes));
    CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(int32_t), st));
    int rc = ndnlm_stage(pl, arr, arr_strides, padded, -1, NDNLM_EDGE_REFLECT, NDNLM_EDGE_REFLECT, stream);
    if (rc) return rc;
    void* scratch = ndnlm_scratch_bytes(pl) ? (void*)(ws + align256(pl->padded_bytes) + align256(pl->out_bytes) + 256) : nullptr;
    if (output && out_strides && ndnlm_output_is_native(pl, out_strides) &&
        (reinterpret_cast<uintptr_t>(output) % size_t(pl->vec_bytes)) == 0) {
        rc = ndnlm_run_scratch(pl, padded, output, flag, scratch, stream);      // the kernels write the caller's array
        if (rc) return rc;
    } else {
        rc = ndnlm_run_scratch(pl, padded, internal, flag, scratch, stream);
        if (rc) return rc;
        rc = ndnlm_unstage(pl, internal, output, out_strides, stream);
        if (rc) return rc;
    }
    int32_t hflag = 0;
    CUDA_TRY(cudaMemcpyAsync(&hflag, flag, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (hflag & NDNLM_FLAG_NOSOLUTION) return fail(NDNLM_ENOSOLUTION, "No solution");
    if (hflag & NDNLM_FLAG_UNDERFLOW)
        return fail(NDNLM_WUNDERFLOW, "at some voxels every neighbour weight is below the float32 range (< 2^-126): they were "
                                      "left unfiltered; use float64 data / the generic kernel, or a larger h");
    return NDNLM_OK;
}

// ------------------------------------------------------------------------------------------
// synthetic data, misc
// ------------------------------------------------------------------------------------------
extern "C" int ndnlm_synth_cube(float* out, int64_t ny_local, int64_t nx, int64_t nt, int32_t V, int64_t y_offset,
                                uint64_t seed, void* stream) {
    if (!out || ny_local < 1 || nx < 1 || nt < 1 || V < 1) return fail(NDNLM_EINVAL, "bad argument");
    GUARD_DEVICE(out);
    const long long total = (long long)ny_local * nx * nt;
    synth_cube_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(out, ny_local, nx, nt, V, y_offset, seed);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return NDNLM_OK;
}

// FP32 FMA-chain microbenchmark: the measured CUDA-core peak of THIS device under load, the
// denominator beside the nominal SMs*128*2*clock figure (SURVEY.md 8(d)).
__global__ void __launch_bounds__(1024) fp32_peak_kernel(float* out, float a, float b, int iters) {
    float r[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) r[i] = threadIdx.x * 0.001f + i;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = fmaf(r[i], a, b);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += r[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

extern "C" int ndnlm_measure_fp32_peak(double* tflops, double seconds, int device, void* stream) {
    if (!tflops) return fail(NDNLM_EINVAL, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    int dev = device, sms = 0, prev = 0;
    CUDA_TRY(cudaGetDevice(&prev));
    CUDA_TRY(cudaSetDevice(dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    float* out = nullptr;
    CUDA_TRY(cudaMalloc(&out, sizeof(float) * size_t(sms) * 2 * 1024));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int iters = 1 << 15;
    double best = 0.0, elapsed = 0.0;
    for (int rep = 0; rep < 1000 && (rep < 3 || elapsed < seconds); ++rep) {
        CUDA_TRY(cudaEventRecord(e0, st));
        fp32_peak_kernel<<<sms * 2, 1024, 0, st>>>(out, 1.0001f, 0.5f, iters);
        CUDA_TRY(cudaEventRecord(e1, st));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        const double fl = 2.0 * 16.0 * double(iters) * double(sms) * 2.0 * 1024.0;
        if (rep > 0 && fl / (ms * 1e-3) > best) best = fl / (ms * 1e-3);
        elapsed += ms * 1e-3;
        g_launches++;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    cudaSetDevice(prev);
    *tflops = best * 1e-12;
    return NDNLM_OK;
}

extern "C" int64_t ndnlm_launch_count(void) { return g_launches.load(); }
extern "C" const char* ndnlm_last_error(void) { return g_err; }
extern "C" const char* ndnlm_version(void) { return "ndnlm 0.1 (sm_100a)"; }
