// ndflt.cu -- C ABI (include/ndflt.h) of the sibling filters: N-D and 1-D correlation kernels that restate
// scipy.ndimage's NI_Correlate / NI_Correlate1D operation by operation (see the header for the algorithm and
// the reference call sites nd/filters.py:260-268 and :370-378).  HBM-bound streaming kernels: one thread per
// output element, threads run along the axis with the smallest output stride (coalesced stores), neighbours
// come through L1/L2; an interior fast path skips the boundary-extension index math.
#include "../../include/ndflt.h"
#include "../../include/ndnlm.h"

#include <atomic>
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <vector>

#include <cuda_runtime.h>

static thread_local char g_flt_err[512] = "";
static std::atomic<long long> g_flt_launches{0};

static int flt_fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_flt_err, sizeof(g_flt_err), fmt, ap);
    va_end(ap);
    return code;
}
#define FLT_CUDA_TRY(expr)                                                                          \
    do {                                                                                            \
        cudaError_t e_ = (expr);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return flt_fail(NDNLM_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// The library carries its own static CUDA runtime: bind the device that owns the buffers (see ndnlm.cu).
struct FltDeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit FltDeviceGuard(const void* ptr) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
            cudaGetLastError();
            ok = false;
            return;
        }
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != attr.device && cudaSetDevice(attr.device) != cudaSuccess) ok = false;
        if (prev == attr.device) prev = -1;
    }
    ~FltDeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// Stream-ordered scratch buffer that is released on every exit path (including failed launches).
struct AsyncBuf {
    void* p = nullptr;
    cudaStream_t st;
    explicit AsyncBuf(cudaStream_t s) : st(s) {}
    cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes ? bytes : 1, st); }
    ~AsyncBuf() {
        if (p) cudaFreeAsync(p, st);
    }
};

namespace ndflt {

// NI_ExtendLine (scipy ni_support.c): index of the element that position i (outside [0, n)) stands for;
// -1 = the constant `cval`.  One reflection / wrap covers every kernel that is not longer than the axis; only
// longer kernels take the modulo path.
__host__ __device__ inline long long extend_index(long long i, long long n, int mode) {
    if (i >= 0 && i < n) return i;
    switch (mode) {
        case NDFLT_MODE_REFLECT: {           // d c b a | a b c d | d c b a
            if (n <= 1) return 0;
            const long long once = i < 0 ? -i - 1 : 2 * n - 1 - i;
            if (once >= 0 && once < n) return once;
            const long long p = 2 * n;
            long long m = i % p;
            if (m < 0) m += p;
            return m < n ? m : p - 1 - m;
        }
        case NDFLT_MODE_MIRROR: {            // d c b | a b c d | c b a
            if (n <= 1) return 0;
            const long long once = i < 0 ? -i : 2 * n - 2 - i;
            if (once >= 0 && once < n) return once;
            const long long p = 2 * n - 2;
            long long m = i % p;
            if (m < 0) m += p;
            return m < n ? m : p - m;
        }
        case NDFLT_MODE_WRAP: {              // a b c d | a b c d | a b c d
            if (n <= 1) return 0;
            const long long once = i < 0 ? i + n : i - n;
            if (once >= 0 && once < n) return once;
            long long m = i % n;
            if (m < 0) m += n;
            return m;
        }
        case NDFLT_MODE_NEAREST:
            return i < 0 ? 0 : n - 1;
        default:
            return -1;
    }
}

struct Geometry {
    long long shape[4], istr[4], ostr[4];
    int ord[4];            // axes from the fastest-running thread index to the slowest
    long long total;
    int mode;
    double cval;
};

__device__ __forceinline__ void decompose(const Geometry& G, long long lin, long long (&idx)[4]) {
    if (G.total <= 0xffffffffLL) {          // 32-bit divisions are several times cheaper than 64-bit ones
        unsigned l = unsigned(lin);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int a = G.ord[k];
            const unsigned n = unsigned(G.shape[a]);
            const unsigned q = l / n;
            idx[a] = l - q * n;
            l = q;
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int a = G.ord[k];
        const long long n = G.shape[a];
        idx[a] = lin % n;
        lin /= n;
    }
}

struct Tap {
    int off[4];            // offset of the tap from the output position, per axis
    long long lin;         // the same as an element offset in the input (interior fast path)
    double w;
};

// ---- N-D correlation (NI_Correlate) ----------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
correlate_nd_kernel(const Geometry G, const T* __restrict__ in, T* __restrict__ out, const Tap* __restrict__ taps,
                    const int ntaps, const int4 omin, const int4 omax) {
    const long long lin = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (lin >= G.total) return;
    long long idx[4];
    decompose(G, lin, idx);
    const int lo[4] = {omin.x, omin.y, omin.z, omin.w}, hi[4] = {omax.x, omax.y, omax.z, omax.w};
    bool interior = true;
    long long base = 0, obase = 0;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        interior = interior && (idx[a] + lo[a] >= 0) && (idx[a] + hi[a] < G.shape[a]);
        base += idx[a] * G.istr[a];
        obase += idx[a] * G.ostr[a];
    }
    double tmp = 0.0;
    if (interior) {
        for (int t = 0; t < ntaps; ++t) {
            const double v = double(__ldg(in + base + __ldg(&taps[t].lin)));
            tmp = __dadd_rn(tmp, __dmul_rn(v, __ldg(&taps[t].w)));
        }
    } else {
        for (int t = 0; t < ntaps; ++t) {
            long long src = 0;
            bool inside = true;
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const long long j = extend_index(idx[a] + taps[t].off[a], G.shape[a], G.mode);
                inside = inside && j >= 0;
                src += j * G.istr[a];
            }
            const double v = inside ? double(__ldg(in + src)) : G.cval;
            tmp = __dadd_rn(tmp, __dmul_rn(v, __ldg(&taps[t].w)));
        }
    }
    out[obase] = T(tmp);
}

// ---- 1-D correlation (NI_Correlate1D) ---------------------------------------------------------------
// SYM: 1 symmetric, -1 antisymmetric, 0 general.  w points at the kernel centre (w[-size1 .. size2]).
template <typename T, int SYM>
__global__ void __launch_bounds__(256)
correlate_1d_kernel(const Geometry G, const T* __restrict__ in, T* __restrict__ out, const double* __restrict__ wbuf,
                    const int axis, const int size1, const int size2, const int origin) {
    const long long lin = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (lin >= G.total) return;
    long long idx[4];
    decompose(G, lin, idx);
    long long base = 0, obase = 0;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        base += idx[a] * G.istr[a];
        obase += idx[a] * G.ostr[a];
    }
    const long long n = G.shape[axis], st = G.istr[axis];
    const long long l = idx[axis] - origin;               // tap j reads position l + j
    const T* line = in + (base - idx[axis] * st);           // element 0 of this line
    const double* w = wbuf + size1;
    const bool interior = (l - size1 >= 0) && (l + size2 < n);
    auto at = [&](const int j) -> double {
        if (interior) return double(__ldg(line + (l + j) * st));
        const long long k = extend_index(l + j, n, G.mode);
        return k >= 0 ? double(__ldg(line + k * st)) : G.cval;
    };
    double tmp;
    if (SYM != 0) {
        tmp = __dmul_rn(at(0), __ldg(w));
        for (int j = -size1; j < 0; ++j) {
            const double a = at(j), b = at(-j);
            const double s = SYM > 0 ? __dadd_rn(a, b) : __dsub_rn(a, b);
            tmp = __dadd_rn(tmp, __dmul_rn(s, __ldg(w + j)));
        }
    } else {
        tmp = __dmul_rn(at(size2), __ldg(w + size2));
        for (int j = -size1; j < size2; ++j) tmp = __dadd_rn(tmp, __dmul_rn(at(j), __ldg(w + j)));
    }
    out[obase] = T(tmp);
}

}  // namespace ndflt
#include "ndflt_tiled.cuh"
using namespace ndflt;

// C-contiguous (row-major) layout of both arrays?  (extent-1 axes may carry any stride)
static bool is_contiguous(const int64_t shape[4], const int64_t strides[4]) {
    long long expect = 1;
    for (int a = 3; a >= 0; --a) {
        if (shape[a] != 1 && strides[a] != expect) return false;
        expect *= shape[a];
    }
    return true;
}

// Tile geometry of the [outer][n][inner] view around axis `s`; false if the grid would not fit.
static bool make_tile(TileGeom& T, const int64_t shape[4], int s, int taps_along_s, int mode, double cval) {
    T.outer = 1;
    T.inner = 1;
    for (int a = 0; a < s; ++a) T.outer *= shape[a];
    for (int a = s + 1; a < 4; ++a) T.inner *= shape[a];
    T.n = shape[s];
    if (T.inner > 0xffffffffLL) return false;
    T.TI = int(T.inner < TILE_THREADS ? T.inner : TILE_THREADS);
    T.RP = TILE_THREADS / T.TI;
    int rows = 4 * taps_along_s;                       // rows per CTA: re-read overhead (rows + taps) / rows
    rows = rows < 16 ? 16 : (rows > 64 ? 64 : rows);
    T.U = (rows + T.RP - 1) / T.RP;
    const long long nbi = (T.inner + T.TI - 1) / T.TI, nbn = (T.n + (long long)T.RP * T.U - 1) / ((long long)T.RP * T.U);
    if (nbi * nbn * T.outer > 0x7fffffffLL) return false;
    T.nbi = unsigned(nbi);
    T.nbn = unsigned(nbn);
    T.mode = mode;
    T.cval = cval;
    return true;
}

static int fill_geometry(Geometry& G, const int64_t shape[4], const int64_t in_strides[4], const int64_t out_strides[4],
                         int mode, double cval) {
    G.total = 1;
    for (int a = 0; a < 4; ++a) {
        if (shape[a] < 1 || shape[a] > 0x7fffffffLL) return flt_fail(NDNLM_EINVAL, "shape[%d]=%lld out of range", a, (long long)shape[a]);
        G.shape[a] = shape[a];
        G.istr[a] = in_strides[a];
        G.ostr[a] = out_strides[a];
        G.total *= shape[a];
    }
    if (mode < NDFLT_MODE_REFLECT || mode > NDFLT_MODE_WRAP) return flt_fail(NDNLM_EINVAL, "unknown boundary mode %d", mode);
    G.mode = mode;
    G.cval = cval;
    // thread order: smallest output stride first (extent-1 axes last)
    int ax[4] = {0, 1, 2, 3};
    for (int i = 0; i < 4; ++i)
        for (int j = i + 1; j < 4; ++j) {
            auto key = [&](int a) { return shape[a] == 1 ? (long long)0x7fffffffffffffffLL : llabs((long long)out_strides[a]); };
            if (key(ax[j]) < key(ax[i]) || (key(ax[j]) == key(ax[i]) && ax[j] > ax[i])) {
                const int t = ax[i]; ax[i] = ax[j]; ax[j] = t;
            }
        }
    for (int k = 0; k < 4; ++k) G.ord[k] = ax[k];
    return NDNLM_OK;
}

static inline unsigned flt_blocks(long long total) { return unsigned((total + 255) / 256); }

// Dense 2-D footprints: instantiations for 3x3, 3x5, 5x3, 5x5, 7x7 (U = 16 consecutive rows per thread).
constexpr int DENSE_U = 16;
template <typename T, int KH, int KW>
static int launch_dense2d_t(const TileGeom& TG, const Dense2dGeom& D, const void* in, void* out, const double* weights,
                            cudaStream_t st) {
    TileGeom G = TG;
    G.U = DENSE_U;
    const long long nbn = (G.n + (long long)G.RP * DENSE_U - 1) / ((long long)G.RP * DENSE_U);
    if (G.outer * nbn * G.nbi > 0x7fffffffLL) return 1;
    G.nbn = unsigned(nbn);
    AsyncBuf wbuf(st);
    FLT_CUDA_TRY(wbuf.alloc(sizeof(double) * KH * KW));
    double* dw = (double*)wbuf.p;
    FLT_CUDA_TRY(cudaMemcpyAsync(dw, weights, sizeof(double) * KH * KW, cudaMemcpyHostToDevice, st));
    correlate_2d_slide_kernel<T, KH, KW, DENSE_U><<<unsigned(G.outer * G.nbn * G.nbi), TILE_THREADS, 0, st>>>(
        G, D, (const T*)in, (T*)out, dw);
    g_flt_launches++;
    FLT_CUDA_TRY(cudaGetLastError());
    return NDNLM_OK;
}
static int launch_dense2d(int dtype, int kh, int kw, const TileGeom& TG, const Dense2dGeom& D, const void* in, void* out,
                          const double* weights, cudaStream_t st) {
#define NDFLT_DENSE(KH, KW)                                                                             \
    if (kh == KH && kw == KW)                                                                           \
        return dtype == NDFLT_F64 ? launch_dense2d_t<double, KH, KW>(TG, D, in, out, weights, st)       \
                                  : launch_dense2d_t<float, KH, KW>(TG, D, in, out, weights, st);
    NDFLT_DENSE(3, 3)
    NDFLT_DENSE(3, 5)
    NDFLT_DENSE(5, 3)
    NDFLT_DENSE(5, 5)
    NDFLT_DENSE(7, 7)
#undef NDFLT_DENSE
    return 1;
}

// Dense 3 x 3 x 3 footprints over the tiled axis and two trailing axes.
template <typename T>
static int launch_dense3d_t(const TileGeom& TG, const Dense3dGeom& D, const void* in, void* out, const double* weights,
                            cudaStream_t st) {
    constexpr int U3 = 8;
    TileGeom G = TG;
    G.U = U3;
    const long long nbn = (G.n + (long long)G.RP * U3 - 1) / ((long long)G.RP * U3);
    if (G.outer * nbn * G.nbi > 0x7fffffffLL) return 1;
    G.nbn = unsigned(nbn);
    AsyncBuf wbuf(st);
    FLT_CUDA_TRY(wbuf.alloc(sizeof(double) * 27));
    double* dw = (double*)wbuf.p;
    FLT_CUDA_TRY(cudaMemcpyAsync(dw, weights, sizeof(double) * 27, cudaMemcpyHostToDevice, st));
    correlate_3d_slide_kernel<T, 3, 3, 3, U3><<<unsigned(G.outer * G.nbn * G.nbi), TILE_THREADS, 0, st>>>(
        G, D, (const T*)in, (T*)out, dw);
    g_flt_launches++;
    FLT_CUDA_TRY(cudaGetLastError());
    return NDNLM_OK;
}

extern "C" int ndflt_correlate(const void* in, void* out, const int64_t shape[4], const int64_t in_strides[4],
                               const int64_t out_strides[4], int dtype, const double* weights, const int64_t kshape[4],
                               const int64_t origin[4], int mode, double cval, void* stream) {
    if (!in || !out || !shape || !in_strides || !out_strides || !weights || !kshape || !origin)
        return flt_fail(NDNLM_EINVAL, "null argument");
    if (dtype != NDFLT_F32 && dtype != NDFLT_F64) return flt_fail(NDNLM_EDTYPE, "only float32 / float64 data is supported");
    FltDeviceGuard guard(out);
    if (!guard.ok) return flt_fail(NDNLM_EINVAL, "out is not a CUDA device pointer");
    Geometry G;
    int rc = fill_geometry(G, shape, in_strides, out_strides, mode, cval);
    if (rc) return rc;
    long long ksz = 1;
    for (int a = 0; a < 4; ++a) {
        if (kshape[a] < 1 || kshape[a] > 4096) return flt_fail(NDNLM_EINVAL, "kernel shape[%d]=%lld out of range", a, (long long)kshape[a]);
        // scipy `_invalid_origin`: -(lenw // 2) <= origin <= (lenw - 1) // 2
        if (origin[a] < -(kshape[a] / 2) || origin[a] > (kshape[a] - 1) / 2)
            return flt_fail(NDNLM_EINVAL, "Invalid origin; origin must satisfy -(weights.shape[k] // 2) <= origin[k] <= (weights.shape[k]-1) // 2");
        ksz *= kshape[a];
    }
    if (ksz > (1 << 22)) return flt_fail(NDNLM_EINVAL, "kernel too large");
    std::vector<Tap> taps;
    int lo[4] = {0, 0, 0, 0}, hi[4] = {0, 0, 0, 0};
    long long k = 0;
    for (long long k0 = 0; k0 < kshape[0]; ++k0)
        for (long long k1 = 0; k1 < kshape[1]; ++k1)
            for (long long k2 = 0; k2 < kshape[2]; ++k2)
                for (long long k3 = 0; k3 < kshape[3]; ++k3, ++k) {
                    const double w = weights[k];
                    if (!(fabs(w) > DBL_EPSILON)) continue;      // NI_Correlate keeps only the footprint |w| > eps
                    Tap t;
                    const long long kk[4] = {k0, k1, k2, k3};
                    t.lin = 0;
                    const bool first = taps.empty();
                    for (int a = 0; a < 4; ++a) {
                        t.off[a] = int(kk[a] - kshape[a] / 2 - origin[a]);
                        t.lin += (long long)t.off[a] * in_strides[a];
                        lo[a] = first ? t.off[a] : (t.off[a] < lo[a] ? t.off[a] : lo[a]);
                        hi[a] = first ? t.off[a] : (t.off[a] > hi[a] ? t.off[a] : hi[a]);
                    }
                    t.w = w;
                    taps.push_back(t);
                }
    cudaStream_t st = (cudaStream_t)stream;
    // ---- fast path: contiguous arrays, footprint small enough for shared memory ----
    int s_axis = 3;
    for (int a = 3; a >= 0; --a)
        if (kshape[a] > 1) s_axis = a;
    TileGeom TG;
    // ---- fastest path: dense KH x KW footprint over the tiled axis and ONE trailing axis ----
    {
        int x_axis = -1, nk = 0;
        for (int a = 0; a < 4; ++a)
            if (kshape[a] > 1) { ++nk; if (a != s_axis) x_axis = a; }
        const bool dense = (long long)taps.size() == ksz;
        if (dense && nk == 2 && x_axis > s_axis && is_contiguous(shape, in_strides) && is_contiguous(shape, out_strides) &&
            make_tile(TG, shape, s_axis, int(kshape[s_axis]), mode, cval)) {
            Dense2dGeom D;
            D.dimx = unsigned(shape[x_axis]);
            long long xs = 1;
            for (int a = x_axis + 1; a < 4; ++a) xs *= shape[a];
            D.xs = unsigned(xs);
            D.oy = int(origin[s_axis]);
            D.ox = int(origin[x_axis]);
            int rc2 = launch_dense2d(dtype, int(kshape[s_axis]), int(kshape[x_axis]), TG, D, in, out, weights, st);
            if (rc2 <= 0) return rc2;                                   // 0 done, < 0 error, > 0 no instantiation
        }
        // dense 3 x 3 x 3 over the tiled axis and TWO trailing axes
        int ax3[3], n3 = 0;
        for (int a = 0; a < 4; ++a)
            if (kshape[a] > 1 && n3 < 3) ax3[n3++] = a;
        if (dense && nk == 3 && kshape[ax3[0]] == 3 && kshape[ax3[1]] == 3 && kshape[ax3[2]] == 3 &&
            is_contiguous(shape, in_strides) && is_contiguous(shape, out_strides) && make_tile(TG, shape, ax3[0], 3, mode, cval)) {
            Dense3dGeom D;
            long long xs = 1, ts = 1;
            for (int a = ax3[1] + 1; a < 4; ++a) xs *= shape[a];
            for (int a = ax3[2] + 1; a < 4; ++a) ts *= shape[a];
            D.dimx = unsigned(shape[ax3[1]]); D.xs = unsigned(xs);
            D.dimt = unsigned(shape[ax3[2]]); D.ts = unsigned(ts);
            D.oy = int(origin[ax3[0]]); D.ox = int(origin[ax3[1]]); D.ot = int(origin[ax3[2]]);
            int rc3 = dtype == NDFLT_F64 ? launch_dense3d_t<double>(TG, D, in, out, weights, st)
                                         : launch_dense3d_t<float>(TG, D, in, out, weights, st);
            if (rc3 <= 0) return rc3;
        }
    }
    if (!taps.empty() && taps.size() <= size_t(MAX_SMEM_TAPS) && is_contiguous(shape, in_strides) &&
        is_contiguous(shape, out_strides) && s_axis < 3 && make_tile(TG, shape, s_axis, hi[s_axis] - lo[s_axis] + 1, mode, cval)) {
        TrailGeom R;
        memset(&R, 0, sizeof(R));
        R.ntrail = 3 - s_axis;
        long long str = 1;
        for (int a = 3; a > s_axis; --a) {
            const int k = a - s_axis - 1;
            R.dim[k] = unsigned(shape[a]);
            R.str[k] = str;
            R.lo[k] = lo[a];
            R.hi[k] = hi[a];
            str *= shape[a];
        }
        R.slo = lo[s_axis];
        R.shi = hi[s_axis];
        std::vector<TiledTap> tt(taps.size());
        for (size_t i = 0; i < taps.size(); ++i) {
            tt[i].w = taps[i].w;
            tt[i].ds = taps[i].off[s_axis];
            tt[i].lin = (long long)taps[i].off[s_axis] * TG.inner;
            for (int k = 0; k < 3; ++k) tt[i].dt[k] = 0;
            for (int k = 0; k < R.ntrail; ++k) {
                tt[i].dt[k] = taps[i].off[s_axis + 1 + k];
                tt[i].lin += (long long)tt[i].dt[k] * R.str[k];
            }
        }
        AsyncBuf tbuf(st);
        FLT_CUDA_TRY(tbuf.alloc(tt.size() * sizeof(TiledTap)));
        TiledTap* dtt = (TiledTap*)tbuf.p;
        FLT_CUDA_TRY(cudaMemcpyAsync(dtt, tt.data(), tt.size() * sizeof(TiledTap), cudaMemcpyHostToDevice, st));
        const unsigned grid = unsigned(TG.outer * TG.nbn * TG.nbi);
        if (dtype == NDFLT_F64)
            correlate_nd_tiled_kernel<double><<<grid, TILE_THREADS, 0, st>>>(TG, R, (const double*)in, (double*)out, dtt, int(tt.size()));
        else
            correlate_nd_tiled_kernel<float><<<grid, TILE_THREADS, 0, st>>>(TG, R, (const float*)in, (float*)out, dtt, int(tt.size()));
        g_flt_launches++;
        FLT_CUDA_TRY(cudaGetLastError());
        return NDNLM_OK;
    }
    AsyncBuf gbuf(st);
    FLT_CUDA_TRY(gbuf.alloc(taps.size() * sizeof(Tap)));
    Tap* dtaps = (Tap*)gbuf.p;
    if (!taps.empty()) FLT_CUDA_TRY(cudaMemcpyAsync(dtaps, taps.data(), taps.size() * sizeof(Tap), cudaMemcpyHostToDevice, st));
    // (pageable source: cudaMemcpyAsync returns once the host buffer has been staged, so `taps` may go out of scope)
    const int4 omin = make_int4(lo[0], lo[1], lo[2], lo[3]), omax = make_int4(hi[0], hi[1], hi[2], hi[3]);
    if (dtype == NDFLT_F64)
        correlate_nd_kernel<double><<<flt_blocks(G.total), 256, 0, st>>>(G, (const double*)in, (double*)out, dtaps, int(taps.size()), omin, omax);
    else
        correlate_nd_kernel<float><<<flt_blocks(G.total), 256, 0, st>>>(G, (const float*)in, (float*)out, dtaps, int(taps.size()), omin, omax);
    g_flt_launches++;
    FLT_CUDA_TRY(cudaGetLastError());
    return NDNLM_OK;
}

template <typename T, int SYM>
static void launch_1d_fast(const TileGeom& TG, const void* in, void* out, const double* dw, int size1, int size2, int origin,
                           cudaStream_t st) {
    if (TG.inner == 1) {
        constexpr int U = 4;
        const long long total = TG.outer * TG.n;
        const unsigned grid = unsigned((total + TILE_THREADS * U - 1) / (TILE_THREADS * U));
        correlate_1d_rows_kernel<T, SYM, U><<<grid, TILE_THREADS, 0, st>>>(total, unsigned(TG.n), (const T*)in, (T*)out, dw, size1,
                                                                          size2, origin, TG.mode, TG.cval);
    } else {
        const unsigned grid = unsigned(TG.outer * TG.nbn * TG.nbi);
        correlate_1d_tiled_kernel<T, SYM><<<grid, TILE_THREADS, 0, st>>>(TG, (const T*)in, (T*)out, dw, size1, size2, origin);
    }
}

// Register sliding-window kernels for symmetric / antisymmetric kernels of half-width 1..8 (Gaussian sigma <= 2 with the
// default truncation, boxcar-like 1-D kernels); U = 32 consecutive rows per thread.
constexpr int SLIDE_U = 32;
template <typename T, int SYM, int S1>
static void launch_slide(const TileGeom& TG, const void* in, void* out, const double* dw, int origin, cudaStream_t st) {
    TileGeom G = TG;
    G.U = SLIDE_U;
    G.nbn = unsigned((G.n + (long long)G.RP * SLIDE_U - 1) / ((long long)G.RP * SLIDE_U));
    const unsigned grid = unsigned(G.outer * G.nbn * G.nbi);
    correlate_1d_slide_kernel<T, SYM, S1, SLIDE_U><<<grid, TILE_THREADS, 0, st>>>(G, (const T*)in, (T*)out, dw, origin);
}
template <typename T, int SYM>
static bool try_slide(const TileGeom& TG, const void* in, void* out, const double* dw, int size1, int size2, int origin,
                      cudaStream_t st) {
    if (TG.inner == 1 || size1 != size2 || size1 < 1 || size1 > 8) return false;
    if (TG.outer * ((TG.n + (long long)TG.RP * SLIDE_U - 1) / ((long long)TG.RP * SLIDE_U)) * TG.nbi > 0x7fffffffLL) return false;
    switch (size1) {
        case 1: launch_slide<T, SYM, 1>(TG, in, out, dw, origin, st); break;
        case 2: launch_slide<T, SYM, 2>(TG, in, out, dw, origin, st); break;
        case 3: launch_slide<T, SYM, 3>(TG, in, out, dw, origin, st); break;
        case 4: launch_slide<T, SYM, 4>(TG, in, out, dw, origin, st); break;
        case 5: launch_slide<T, SYM, 5>(TG, in, out, dw, origin, st); break;
        case 6: launch_slide<T, SYM, 6>(TG, in, out, dw, origin, st); break;
        case 7: launch_slide<T, SYM, 7>(TG, in, out, dw, origin, st); break;
        default: launch_slide<T, SYM, 8>(TG, in, out, dw, origin, st); break;
    }
    return true;
}

// Fastest-axis passes through shared memory (kernels up to 129 taps).
template <typename T, int SYM, int S1>
static void launch_rows_smem(const RowsGeom& RG, size_t smem, const void* in, void* out, const double* dw, int size1, int size2,
                             int origin, cudaStream_t st) {
    const unsigned grid = unsigned(((RG.lines + RG.LN - 1) / RG.LN) * RG.nbc);
    correlate_1d_rows_smem_kernel<T, SYM, S1><<<grid, TILE_THREADS, smem, st>>>(RG, (const T*)in, (T*)out, dw, size1, size2, origin);
}
template <typename T, int SYM>
static bool try_rows_smem(const TileGeom& TG, const void* in, void* out, const double* dw, int size1, int size2, int origin,
                          cudaStream_t st) {
    const int nw = size1 + size2 + 1;
    if (TG.inner != 1 || nw > 129 || TG.n > 0x7fffffffLL) return false;
    RowsGeom RG;
    RG.lines = TG.outer;
    RG.n = unsigned(TG.n);
    RG.CW = int(TG.n < 256 ? TG.n : 256);
    RG.pitch = RG.CW + nw - 1;
    int ln = 2048 / RG.CW;                                           // ~8 outputs per thread
    const int cap = int((40960 - 8 * nw) / (8 * RG.pitch));          // <= 40 KB of shared memory
    ln = ln < cap ? ln : cap;
    if (ln < 1) return false;
    if ((long long)ln > RG.lines) ln = int(RG.lines);
    RG.LN = ln;
    RG.nbc = unsigned((TG.n + RG.CW - 1) / RG.CW);
    if (((RG.lines + RG.LN - 1) / RG.LN) * RG.nbc > 0x7fffffffLL) return false;
    RG.mode = TG.mode;
    RG.cval = TG.cval;
    const size_t smem = size_t(RG.LN) * RG.pitch * 8 + size_t(nw) * 8;
    if constexpr (SYM != 0) {                                        // general kernels only take the S1 = 0 form
        if (size1 == size2 && size1 >= 1 && size1 <= 8) {
            switch (size1) {
                case 1: launch_rows_smem<T, SYM, 1>(RG, smem, in, out, dw, size1, size2, origin, st); break;
                case 2: launch_rows_smem<T, SYM, 2>(RG, smem, in, out, dw, size1, size2, origin, st); break;
                case 3: launch_rows_smem<T, SYM, 3>(RG, smem, in, out, dw, size1, size2, origin, st); break;
                case 4: launch_rows_smem<T, SYM, 4>(RG, smem, in, out, dw, size1, size2, origin, st); break;
                case 5: launch_rows_smem<T, SYM, 5>(RG, smem, in, out, dw, size1, size2, origin, st); break;
                case 6: launch_rows_smem<T, SYM, 6>(RG, smem, in, out, dw, size1, size2, origin, st); break;
                case 7: launch_rows_smem<T, SYM, 7>(RG, smem, in, out, dw, size1, size2, origin, st); break;
                default: launch_rows_smem<T, SYM, 8>(RG, smem, in, out, dw, size1, size2, origin, st); break;
            }
            return true;
        }
    }
    launch_rows_smem<T, SYM, 0>(RG, smem, in, out, dw, size1, size2, origin, st);
    return true;
}

template <typename T>
static void launch_1d_fast_sym(int sym, const TileGeom& TG, const void* in, void* out, const double* dw, int size1, int size2,
                               int origin, cudaStream_t st) {
    if (sym > 0 && try_slide<T, 1>(TG, in, out, dw, size1, size2, origin, st)) return;
    if (sym < 0 && try_slide<T, -1>(TG, in, out, dw, size1, size2, origin, st)) return;
    if (sym > 0 && try_rows_smem<T, 1>(TG, in, out, dw, size1, size2, origin, st)) return;
    if (sym < 0 && try_rows_smem<T, -1>(TG, in, out, dw, size1, size2, origin, st)) return;
    if (sym == 0 && try_rows_smem<T, 0>(TG, in, out, dw, size1, size2, origin, st)) return;
    if (sym > 0) launch_1d_fast<T, 1>(TG, in, out, dw, size1, size2, origin, st);
    else if (sym < 0) launch_1d_fast<T, -1>(TG, in, out, dw, size1, size2, origin, st);
    else launch_1d_fast<T, 0>(TG, in, out, dw, size1, size2, origin, st);
}

template <typename T>
static void launch_1d(int sym, const Geometry& G, const void* in, void* out, const double* dw, int axis, int size1, int size2,
                      int origin, cudaStream_t st) {
    const unsigned nb = flt_blocks(G.total);
    if (sym > 0)
        correlate_1d_kernel<T, 1><<<nb, 256, 0, st>>>(G, (const T*)in, (T*)out, dw, axis, size1, size2, origin);
    else if (sym < 0)
        correlate_1d_kernel<T, -1><<<nb, 256, 0, st>>>(G, (const T*)in, (T*)out, dw, axis, size1, size2, origin);
    else
        correlate_1d_kernel<T, 0><<<nb, 256, 0, st>>>(G, (const T*)in, (T*)out, dw, axis, size1, size2, origin);
}

extern "C" int ndflt_correlate1d(const void* in, void* out, const int64_t shape[4], const int64_t in_strides[4],
                                 const int64_t out_strides[4], int dtype, int axis, const double* weights,
                                 int64_t nweights, int64_t origin, int mode, double cval, void* stream) {
    if (!in || !out || !shape || !in_strides || !out_strides || !weights) return flt_fail(NDNLM_EINVAL, "null argument");
    if (dtype != NDFLT_F32 && dtype != NDFLT_F64) return flt_fail(NDNLM_EDTYPE, "only float32 / float64 data is supported");
    if (axis < 0 || axis > 3) return flt_fail(NDNLM_EINVAL, "axis must be 0..3");
    if (nweights < 1 || nweights > (1 << 20)) return flt_fail(NDNLM_EINVAL, "no filter weights given");
    if (origin < -(nweights / 2) || origin > (nweights - 1) / 2)
        return flt_fail(NDNLM_EINVAL, "Invalid origin; origin must satisfy -(len(weights) // 2) <= origin <= (len(weights)-1) // 2");
    FltDeviceGuard guard(out);
    if (!guard.ok) return flt_fail(NDNLM_EINVAL, "out is not a CUDA device pointer");
    Geometry G;
    int rc = fill_geometry(G, shape, in_strides, out_strides, mode, cval);
    if (rc) return rc;
    const int size1 = int(nweights / 2), size2 = int(nweights - size1 - 1);
    // symmetry test of NI_Correlate1D
    int sym = 0;
    if (nweights & 1) {
        sym = 1;
        for (int i = 1; i <= size1; ++i)
            if (fabs(weights[i + size1] - weights[size1 - i]) > DBL_EPSILON) { sym = 0; break; }
        if (sym == 0) {
            sym = -1;
            for (int i = 1; i <= size1; ++i)
                if (fabs(weights[size1 + i] + weights[size1 - i]) > DBL_EPSILON) { sym = 0; break; }
        }
    }
    cudaStream_t st = (cudaStream_t)stream;
    AsyncBuf wbuf(st);
    FLT_CUDA_TRY(wbuf.alloc(size_t(nweights) * sizeof(double)));
    double* dw = (double*)wbuf.p;
    FLT_CUDA_TRY(cudaMemcpyAsync(dw, weights, size_t(nweights) * sizeof(double), cudaMemcpyHostToDevice, st));
    TileGeom TG;
    const bool fast = nweights <= MAX_SMEM_WEIGHTS && is_contiguous(shape, in_strides) && is_contiguous(shape, out_strides) &&
                      shape[axis] <= 0xffffffffLL && make_tile(TG, shape, axis, int(nweights), mode, cval) &&
                      (TG.inner > 1 || (TG.outer * TG.n + TILE_THREADS * 4 - 1) / (TILE_THREADS * 4) <= 0x7fffffffLL);
    if (fast) {
        if (dtype == NDFLT_F64) launch_1d_fast_sym<double>(sym, TG, in, out, dw, size1, size2, int(origin), st);
        else launch_1d_fast_sym<float>(sym, TG, in, out, dw, size1, size2, int(origin), st);
    } else if (dtype == NDFLT_F64) {
        launch_1d<double>(sym, G, in, out, dw, axis, size1, size2, int(origin), st);
    } else {
        launch_1d<float>(sym, G, in, out, dw, axis, size1, size2, int(origin), st);
    }
    g_flt_launches++;
    FLT_CUDA_TRY(cudaGetLastError());
    return NDNLM_OK;
}

extern "C" int64_t ndflt_launch_count(void) { return g_flt_launches.load(); }
extern "C" const char* ndflt_last_error(void) { return g_flt_err; }
