// nlm_tiled.cuh -- the TMA-tiled fp32 non-local-means kernel for sm_100a.
//
// Replaces the voxel / search-window / patch loops of the reference
// (nd/_filters.pyx:351-420) for float32 data.  One CTA owns a (TW, TR, TX) tile of voxels:
//
//   * the reflect-padded input box (tile + halo r+f per axis) is brought into shared memory
//     by ONE TMA tensor copy per variable group (cp.async.bulk.tensor.5d, mbarrier completion);
//   * a warp is one W row x 32 X positions; a thread owns a column of L voxels along R
//     (centre values, the neighbour window and all accumulators live in registers);
//   * per search offset t: pointwise squared differences over the variables (packed
//     FADD2/FMUL2/FFMA2), then a separable box sum over the patch: along R in registers,
//     along X by warp shuffles, along W through a shared-memory exchange between warps;
//     all sums are DIRECT (2f+1)-term sums in a fixed order, so a voxel's result does not
//     depend on where its tile or shard starts;
//   * weight w = exp2(-max(D*c1 - c2, 0)) (one FFMA, one NaN-propagating max, one MUFU.EX2),
//     then acc += w * neighbour (FFMA2), S += w, M = max(M, w) [, Q += w*w];
//   * weight sums are folded into float64 once per W-offset row (fp64-accumulated weight sums).
//
// No tensor cores: the path is not a dense contraction.  The binding unit is the FP32 pipe
// (128 lane-ops/clk/SM, profiles/r1_pipe_microbench.txt).
//
// The kernel is templated on the element type T.  T = float is the path described above.  T = double is the
// reference's float64 arithmetic (fused `floating` = double, nd/_filters.pyx:320-321: differences, squares, patch
// sums, weights with a double-precision exp, weighted sums all in float64) on the same tiles: 32-byte voxels
// (4 doubles), plain FP64 instructions instead of the packed f32x2 ones, half the warps per CTA.
#pragma once
#include <type_traits>

#include "nlm_common.cuh"

#ifndef NDNLM_KEEP_OWN
#define NDNLM_KEEP_OWN 0   // 1: keep my own exchanged sums in registers instead of re-reading them from shared memory
#endif
#ifndef NDNLM_DEBUG_CTA_SYNC
#define NDNLM_DEBUG_CTA_SYNC 0   // 1: replace the neighbour-only mbarrier protocol of the W exchange by two CTA barriers per
                                 //    chunk (slow; lets compute-sanitizer's racecheck, which does not model remote mbarrier
                                 //    arrivals, verify the data flow itself)
#endif
#ifndef NDNLM_NO_PAIRED
#define NDNLM_NO_PAIRED 0   // 1 (tuning experiment): plain 3-term column sums instead of the pair-sharing variant
#endif
#ifndef NDNLM_FOLD_T
#define NDNLM_FOLD_T double   // type of the second-level weight-sum accumulators
#endif

namespace ndnlm {

constexpr unsigned FULL_MASK = 0xffffffffu;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "NDNLM_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra NDNLM_DONE;\n"
        "bra NDNLM_WAIT;\n"
        "NDNLM_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// One 5-D TMA tile load: coordinates (v, r, x, w, q) in elements of the padded cube.
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                            int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}

// max that PROPAGATES NaN, like the reference's `0 > x ? 0 : x` (nd/_filters.c:3604-3609).
__device__ __forceinline__ float fmax_nan(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float2 lo2(const float4& v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi2(const float4& v) { return make_float2(v.z, v.w); }

// ---- element-type traits: float -> float4 / float2 with packed f32x2 arithmetic, double -> 4 / 2 doubles ----
struct alignas(32) double4v { double x, y, z, w; };
__device__ __forceinline__ double2 lo2(const double4v& v) { return make_double2(v.x, v.y); }
__device__ __forceinline__ double2 hi2(const double4v& v) { return make_double2(v.z, v.w); }

template <typename T> struct Elem;
template <> struct Elem<float> {
    using V4 = float4;
    using P2 = float2;
    static constexpr CUtensorMapDataType tma_type = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
};
template <> struct Elem<double> {
    using V4 = double4v;
    using P2 = double2;
    static constexpr CUtensorMapDataType tma_type = CU_TENSOR_MAP_DATA_TYPE_FLOAT64;
};
__device__ __forceinline__ float2 mk2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ double2 mk2(double a, double b) { return make_double2(a, b); }
__device__ __forceinline__ float4 mk4(float a, float b, float c, float d) { return make_float4(a, b, c, d); }
__device__ __forceinline__ double4v mk4(double a, double b, double c, double d) { double4v v; v.x = a; v.y = b; v.z = c; v.w = d; return v; }
__device__ __forceinline__ float2 padd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 pmul(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 pfma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ double2 padd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 pmul(double2 a, double2 b) { return make_double2(a.x * b.x, a.y * b.y); }
__device__ __forceinline__ double2 pfma(double2 a, double2 b, double2 c) { return make_double2(fma(a.x, b.x, c.x), fma(a.y, b.y, c.y)); }
__device__ __forceinline__ float2 pneg(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ double2 pneg(double2 a) { return make_double2(-a.x, -a.y); }
// NaN-propagating max(x, 0) like the reference's `0 > x ? 0 : x`
__device__ __forceinline__ float clamp0_nan(float x) { return fmax_nan(x, 0.f); }
__device__ __forceinline__ double clamp0_nan(double x) { return (0.0 > x) ? 0.0 : x; }
// weight from the scaled, clamped exponent argument: float: exp2(-t) (t carries log2 e), double: exp(-t)
__device__ __forceinline__ float weight_of(float t) { return ex2_approx(-t); }
__device__ __forceinline__ double weight_of(double t) { return exp(-t); }
__device__ __forceinline__ float tmax(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double tmax(double a, double b) { return fmax(a, b); }

// Direct (2F+1)-term sum along the register column, fixed order.
template <int F, int L, typename T>
__device__ __forceinline__ void column_box_sum(const T (&s)[L + 2 * F], T (&o)[L]) {
    if constexpr (F == 0) {
#pragma unroll
        for (int i = 0; i < L; ++i) o[i] = s[i];
    } else if constexpr (F == 1) {
#pragma unroll
        for (int i = 0; i < L; ++i) o[i] = (s[i] + s[i + 1]) + s[i + 2];
    } else if constexpr (F == 2) {
        T a[L + 3];
#pragma unroll
        for (int i = 0; i < L + 3; ++i) a[i] = s[i] + s[i + 1];
#pragma unroll
        for (int i = 0; i < L; ++i) o[i] = (a[i] + a[i + 2]) + s[i + 4];
    } else {
#pragma unroll
        for (int i = 0; i < L; ++i) {
            T t = s[i];
#pragma unroll
            for (int d = 1; d <= 2 * F; ++d) t += s[i + d];
            o[i] = t;
        }
    }
}

// F == 1 variant that shares the middle pair between two neighbouring outputs: 3 adds per 2 outputs
// instead of 4.  The association depends on the parity of the output index inside the column, so it is
// only used where the R axis is never cut by slabs / shards (three filtered axes: W is axis 0).
template <int L, typename T>
__device__ __forceinline__ void column_box_sum_paired(const T (&s)[L + 2], T (&o)[L]) {
#pragma unroll
    for (int k = 0; k < L / 2; ++k) {
        const T m = s[2 * k + 1] + s[2 * k + 2];
        o[2 * k] = s[2 * k] + m;
        o[2 * k + 1] = m + s[2 * k + 3];
    }
}

// (2F+1)-term sum across lanes in a fixed order that depends only on the lane-relative position
// (lane x gets x-F..x+F).  F == 2 uses pair sums: ((v[x-2]+v[x-1]) + (v[x]+v[x+1])) + v[x+2], 3 shuffles.
template <int F>
__device__ __forceinline__ float lane_box_sum(float v) {
    if constexpr (F == 0) {
        return v;
    } else if constexpr (F == 1) {
        const float a = __shfl_up_sync(FULL_MASK, v, 1);
        const float b = __shfl_down_sync(FULL_MASK, v, 1);
        return (a + v) + b;
    } else if constexpr (F == 2) {
        const float pair = v + __shfl_down_sync(FULL_MASK, v, 1);
        const float left = __shfl_up_sync(FULL_MASK, pair, 2);
        const float right = __shfl_down_sync(FULL_MASK, v, 2);
        return (left + pair) + right;
    } else {
        float t = v;
#pragma unroll
        for (int d = 1; d <= F; ++d) {
            const float a = __shfl_up_sync(FULL_MASK, v, d);
            const float b = __shfl_down_sync(FULL_MASK, v, d);
            t += a + b;
        }
        return t;
    }
}

// Call fn(integral_constant<int, nj>, bool_constant<centre>) for the runtime (uniform) nj in 1..MAXJ.
template <int MAXJ, typename Fn>
__device__ __forceinline__ void dispatch_chunk(const int nj, const bool centre, Fn&& fn) {
    if constexpr (MAXJ >= 1) {
        if (nj == MAXJ) {
            if (centre) fn(std::integral_constant<int, MAXJ>{}, std::true_type{});
            else        fn(std::integral_constant<int, MAXJ>{}, std::false_type{});
        } else {
            dispatch_chunk<MAXJ - 1>(nj, centre, fn);
        }
    }
}

// The same for two values at once (a register pair): the adds are packed FADD2.
template <int F, typename P2>
__device__ __forceinline__ P2 lane_box_sum2(const P2 v) {
    auto up = [](const P2 a, const int d) {
        return mk2(__shfl_up_sync(FULL_MASK, a.x, d), __shfl_up_sync(FULL_MASK, a.y, d));
    };
    auto down = [](const P2 a, const int d) {
        return mk2(__shfl_down_sync(FULL_MASK, a.x, d), __shfl_down_sync(FULL_MASK, a.y, d));
    };
    if constexpr (F == 0) {
        return v;
    } else if constexpr (F == 1) {
        const P2 a = up(v, 1), b = down(v, 1);
        return padd(padd(a, v), b);
    } else if constexpr (F == 2) {
        const P2 pair = padd(v, down(v, 1));
        const P2 left = up(pair, 2), right = down(v, 2);
        return padd(padd(left, pair), right);
    } else {
        P2 t = v;
#pragma unroll
        for (int d = 1; d <= F; ++d) t = padd(t, padd(up(v, d), down(v, d)));
        return t;
    }
}

// DH ("double-duty halo warps", FW > 0 only): the 2 FW patch-halo rows of a CTA tile only run phase A (squared
// differences, R / X sums, publish) -- about half the work of a row that also weighs and accumulates.  With one warp per
// row they leave their warp scheduler under-used and occupy 2 FW of the NWARPS register-file slots.  With DH each of FW
// halo WARPS serves TWO halo rows (one above, one below the valid rows; it keeps no accumulators, so the second centre
// column fits its registers): NWARPS warps then cover NWARPS + FW rows, NWARPS - FW of them valid.
// PERSIST: persistent CTAs (one per SM) that walk tiles blockIdx.x + k gridDim.x, keep the whole W search range in
// shared memory (one pass), read the centre column from it and load the next tile's box while the finished tile runs its
// epilogue.  The W exchange then only holds the TXW valid lanes of a row: the sums of the X-halo lanes are never read.
template <typename T, int NV4, int FW, int FX, int FR, int L, int NWARPS, int CH, bool NEFF, bool DH = false,
          bool PERSIST = false>
struct TiledCfg {
    static constexpr int E = L + 2 * FR;      // column elements including the patch halo
    static constexpr int WN = E + CH - 1;     // neighbour window elements per chunk of CH R-offsets
    static constexpr int TXW = 32 - 2 * FX;   // valid lanes per warp
    static constexpr int THREADS = NWARPS * 32;
    static constexpr int NROWS = DH ? NWARPS + FW : NWARPS;   // W rows of the CTA tile, patch-halo rows included
    static constexpr int EXW = PERSIST ? TXW : 32;             // exchange slots per row and R-offset
    static constexpr size_t EXCH_BYTES = FW > 0 ? size_t(CH) * NROWS * (L / 2) * EXW * sizeof(typename Elem<T>::P2) : 0;
};

// HALF: the last variable group holds at most two real variables (V = 5 or 6 of 8): its upper two lanes are zero
// padding, and every load, difference, square and accumulation on them is skipped (64-bit instead of 128-bit
// shared-memory loads, 3 instead of 4 packed operations per voxel pair, a quarter fewer registers for that group).
// Small-footprint instantiations (float, one variable group, L <= 4) are compiled for several CTAs per SM -- 4 for the
// 4-warp kernels of 2-D images / batch axes, 2 for the 8-warp fallbacks: 2-D images have few offsets per tile, so the
// TMA wait and the epilogue of one CTA should overlap the arithmetic of the others.
template <typename T, int NV4, int FW, int L, int NWARPS>
constexpr int tiled_min_blocks() {
    return (sizeof(T) == 4 && NV4 == 1 && L <= 4 && NWARPS <= 4) ? 4 : (sizeof(T) == 4 && NV4 == 1 && L <= 4 && NWARPS <= 8) ? 2 : 1;
}

template <typename T, int NV4, int FW, int FX, int FR, int L, int NWARPS, int CH, bool NEFF, bool HALF = false, bool DH = false,
          bool PERSIST = false>
__global__ void __launch_bounds__(NWARPS * 32, tiled_min_blocks<T, NV4, FW, L, NWARPS>())
nlm_tiled_kernel(const __grid_constant__ CUtensorMap tmap, const DevParams P,
                 const typename Elem<T>::V4* __restrict__ padded, typename Elem<T>::V4* __restrict__ out,
                 int* __restrict__ err) {
    using Cfg = TiledCfg<T, NV4, FW, FX, FR, L, NWARPS, CH, NEFF, DH, PERSIST>;
    using V4 = typename Elem<T>::V4;
    using P2 = typename Elem<T>::P2;
    constexpr bool F64 = sizeof(T) == 8;
    static_assert(L % 2 == 0, "L must be even (outputs are exchanged in pairs)");
    static_assert(!DH || (FW > 0 && NWARPS >= 3 * FW + 1), "double-duty halo warps need a W patch axis");
    static_assert(!PERSIST || (!F64 && !HALF && !DH && FW > 0 && L == 4), "persistent CTAs: float32, L = 4, W patch axis");
    constexpr int E = Cfg::E, TXW = Cfg::TXW;
    constexpr int NROWS = Cfg::NROWS;                      // W rows of the tile (== NWARPS unless DH)

    // Shared memory: the padded box as [q][BW][BX][BRP] float4 -- R is the FASTEST axis and its
    // pitch BRP is odd, so a thread's column / neighbour window is a run of consecutive float4
    // (immediate LDS offsets) and the 8 lanes of an LDS.128 phase hit 8 distinct 16-B bank groups.
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int BW = P.b[0], BRP = P.b[1], BX = P.b[2];
    const int plane = ((BW * BRP * BX + 7) >> 3) << 3;   // float4 per variable group, 128-B multiple
    V4* tile = reinterpret_cast<V4*>(smem_raw);
    P2* exch = reinterpret_cast<P2*>(smem_raw + size_t(NV4) * plane * sizeof(V4));
    uint64_t* mbar =
        reinterpret_cast<uint64_t*>(smem_raw + size_t(NV4) * plane * sizeof(V4) + Cfg::EXCH_BYTES);
    // Neighbour-only synchronisation of the W exchange (no CTA-wide barrier in the hot loop):
    //   full[w]   every row that warp w reads has published its sums for the current chunk (one arrival per
    //             source row, so a reader waits ONCE)
    //   empty[w]  every warp that reads warp w's sums has finished with them              (one arrival per reader)
    uint64_t* mbar_full = mbar + 1;
    uint64_t* mbar_empty = mbar + 1 + NROWS;

    // PERSIST: this CTA's tk-th tile is tile_id = blockIdx.x + tk gridDim.x, in the order of the one-tile-per-CTA launch
    [[maybe_unused]] const int ntiles = P.tiles[0] * P.tiles[1] * P.tiles[2];
    [[maybe_unused]] int tile_id = blockIdx.x, tk = 0;
    [[maybe_unused]] uint32_t xpar_carry = 0;   // exchange parity at the end of the previous tile
#if NDNLM_TILE_PROBE
#define NDNLM_PROBE(slot)                                                                         \
    do {                                                                                          \
        if (threadIdx.x == 32 * FW && tile_id < P.probe_cap) P.probe[size_t(tile_id) * 8 + (slot)] = clock64(); \
    } while (0)
#else
#define NDNLM_PROBE(slot) do {} while (0)
#endif
    do {
    NDNLM_PROBE(0);
    int bid = PERSIST ? tile_id : int(blockIdx.x);
    const int tileX = bid % P.tiles[2];
    bid /= P.tiles[2];
    const int tileR = bid % P.tiles[1];
    const int tileW = bid / P.tiles[1];
    const int w0 = tileW * P.t[0], r0 = tileR * P.t[1], x0 = tileX * P.t[2];
#if NDNLM_TILE_PROBE
    if (threadIdx.x == 32 * FW && tile_id < P.probe_cap) {
        unsigned sm;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
        P.probe[size_t(tile_id) * 8 + 7] = sm;
    }
#endif
    // ---- stage the padded box (tile + halo r+f) into shared memory ----
    if (!PERSIST || tk == 0) {
    if (threadIdx.x == 0) {
        mbar_init(mbar, 1);
        if constexpr (FW > 0) {
            for (int w = 0; w < NROWS; ++w) {
                int readers = 0;   // valid rows within FW rows of w, other than w itself
                for (int d = -FW; d <= FW; ++d)
                    if (d != 0 && w + d >= FW && w + d < NROWS - FW) ++readers;
                int sources = 0;   // rows within FW of w, other than w itself (the rows w reads)
                for (int d = -FW; d <= FW; ++d)
                    if (d != 0 && w + d >= 0 && w + d < NROWS) ++sources;
                mbar_init(mbar_full + w, sources);                         // "every row I read is published"
                mbar_init(mbar_empty + w, readers > 0 ? readers : 1);      // "every reader of my row is done"
            }
        }
        fence_mbar_init();
    }
    __syncthreads();
    }
    // The W search range [-rW, rW] is covered in P.npass passes of P.ntw_pass offsets each; a pass keeps
    // only the rows it needs in shared memory (BW = rows of the CTA + ntw_pass - 1), which is what lets
    // more warps fit beside the exchange buffer.  Pass `p` starts at padded row w0 + p * ntw_pass.
    auto load_pass = [&](const int pass) {
        const int wbase = w0 + pass * P.ntw_pass;
        if (!P.use_ldg_loader) {
            if (threadIdx.x == 0) {
                mbar_arrive_expect_tx(mbar, uint32_t(NV4) * uint32_t(BW * BRP * BX) * uint32_t(sizeof(V4)));
#pragma unroll
                for (int q = 0; q < NV4; ++q) tma_load_5d(tile + size_t(q) * plane, &tmap, mbar, 0, r0, x0, wbase, q);
            }
            mbar_wait(mbar, uint32_t(pass & 1));
        } else {
            const int box = BW * BRP * BX;
            for (int i = threadIdx.x; i < NV4 * box; i += blockDim.x) {
                const int q = i / box;
                int rem = i - q * box;
                const int br = rem % BRP;
                rem /= BRP;
                const int bx = rem % BX;
                const int bw = rem / BX;
                const int gw = wbase + bw, gr = r0 + br, gx = x0 + bx;
                V4 v = mk4(T(0), T(0), T(0), T(0));
                if (gw < P.pd[0] && gr < P.pd[1] && gx < P.pd[2])
                    v = padded[((size_t(q) * P.pd[0] + gw) * P.pd[2] + gx) * P.pd[1] + gr];
                tile[size_t(q) * plane + (bw * BX + bx) * BRP + br] = v;
            }
            __syncthreads();
        }
    };

    // ---- warp / lane roles ----
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gxw = (FW > 0) ? 1 : P.g[2], grw = (FW > 0) ? 1 : P.g[1];
    const int wx = wid % gxw;
    const int wr = (wid / gxw) % grw;
    // W row inside the CTA tile.  DH: warps 0 .. NWARPS-FW-1 own the valid rows FW .. NROWS-FW-1, halo warp k (the last
    // FW warps) owns the halo rows k (above) and NROWS-FW+k (below)
    const int ww = DH ? (wid >= NWARPS - FW ? wid - (NWARPS - FW) : wid + FW) : wid / (gxw * grw);
    const int lx = wx * TXW + lane + P.rad[2];
    const int lr0 = wr * L + P.rad[1];
    const bool wvalid = (FW == 0) || (ww >= FW && ww < NROWS - FW);
    const int xw = DH ? ww : wid;                          // my row's index among the exchange slots / mbarriers

    // centre column: read once, straight from the padded cube (R is the fastest axis there too); PERSIST: from the box
    V4 c[NV4][E];
    if constexpr (!PERSIST) {
        const int gw = w0 + ww + P.rad[0], gx = x0 + lx;      // padded coordinates of this thread's column
        const bool inb = gw < P.pd[0] && gx < P.pd[2];
#pragma unroll
        for (int q = 0; q < NV4; ++q)
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const int gr = r0 + lr0 + e;
                if constexpr (HALF) {
                    const V4* src = padded + ((size_t(q) * P.pd[0] + gw) * P.pd[2] + gx) * P.pd[1] + gr;
                    if (!(inb && gr < P.pd[1])) {
                        c[q][e] = mk4(T(0), T(0), T(0), T(0));
                    } else if (q == NV4 - 1) {
                        const P2 t = *reinterpret_cast<const P2*>(src);
                        c[q][e] = mk4(t.x, t.y, T(0), T(0));
                    } else {
                        c[q][e] = *src;
                    }
                } else {
                    c[q][e] = (inb && gr < P.pd[1])
                                  ? padded[((size_t(q) * P.pd[0] + gw) * P.pd[2] + gx) * P.pd[1] + gr]
                                  : mk4(T(0), T(0), T(0), T(0));
                }
            }
    }

    P2 acc_lo[NV4][L], acc_hi[NV4][L];
    P2 S2[L / 2], Q2[L / 2];
    T M[L];
    NDNLM_FOLD_T Sd[L], Qd[L];
#pragma unroll
    for (int o = 0; o < L; ++o) {
#pragma unroll
        for (int q = 0; q < NV4; ++q) {
            acc_lo[q][o] = mk2(T(0), T(0));
            acc_hi[q][o] = mk2(T(0), T(0));
        }
        M[o] = T(0);
        Sd[o] = 0;
        Qd[o] = 0;
    }

#pragma unroll
    for (int o2 = 0; o2 < L / 2; ++o2) {
        S2[o2] = mk2(T(0), T(0));
        Q2[o2] = mk2(T(0), T(0));
    }
    const int rW = P.rad[0], rR = P.rad[1], rX = P.rad[2];
    // exponent argument t = D c1 - c2: float carries log2(e) (exp2 path), double is the reference's
    // (D / norm - 2 sigma^2) / h^2 (nd/_filters.pyx:388-391)
    const T c1s = F64 ? T(P.inv_norm * P.inv_h2) : T(P.c1);
    const T c2s = F64 ? T(P.two_sigma2 * P.inv_h2) : T(P.c2);
    const P2 c1 = mk2(c1s, c1s);
    const P2 nc2 = mk2(-c2s, -c2s);
    P2* const ex_own = exch + (xw * (L / 2)) * 32 + lane;     // + (j*NWARPS*(L/2) + o2)*32
    constexpr int EX_J = NROWS * (L / 2) * 32;                      // float2 stride between R-offsets j
    constexpr int EX_ROW = (L / 2) * 32;                            // float2 stride between W rows (FW>0: 1 warp/row)
    // L == 4 layout [j][row][slot] float4.  PERSIST: slots are the valid lanes only; the X-halo lanes store nothing and read
    // their neighbour's slot (their sums, weights and accumulators are never used)
    constexpr int EXW = Cfg::EXW;
    [[maybe_unused]] V4* const ex_own4 =
        reinterpret_cast<V4*>(exch) + xw * EXW + (PERSIST ? min(max(lane - FX, 0), TXW - 1) : lane);
    [[maybe_unused]] constexpr int EX_J4 = NROWS * EXW;             // float4 stride between R-offsets j
    [[maybe_unused]] const bool ex_store = !PERSIST || (lane >= FX && lane < 32 - FX);
    uint32_t xpar = PERSIST ? xpar_carry : 0;                       // parity of the current exchange round
    static_assert(FW == 0 || NROWS >= 2 * FW + 2, "every row needs at least one reader");

    // One chunk of NJ consecutive R-offsets [ch0, ch0+NJ).  NJ is a compile-time constant so the body is
    // straight-line code the scheduler can interleave freely.  CENTRE: the chunk contains the centre
    // voxel itself (tw = tx = 0 and ch0 <= 0 < ch0+NJ), whose offset must be skipped -- rare slow path.
    auto chunk = [&](auto nj_tag, auto centre_tag, const V4* nb, const int ch0) {
        constexpr int NJ = decltype(nj_tag)::value;
        constexpr bool CENTRE = decltype(centre_tag)::value;
        constexpr int WNJ = E + NJ - 1;
        if constexpr (CENTRE && FW > 0 && !NDNLM_DEBUG_CTA_SYNC) mbar_wait(mbar_empty + xw, xpar ^ 1);
        [[maybe_unused]] P2 own[NDNLM_KEEP_OWN != 0 ? NJ : 1][L / 2];

        V4 n[NV4][WNJ];
#pragma unroll
        for (int k = 0; k < WNJ; ++k) {
#pragma unroll
            for (int q = 0; q < NV4; ++q) {
                if constexpr (HALF) {
                    if (q == NV4 - 1) {
                        const P2 t = *reinterpret_cast<const P2*>(nb + size_t(q) * plane + k);
                        n[q][k] = mk4(t.x, t.y, T(0), T(0));
                    } else {
                        n[q][k] = nb[size_t(q) * plane + k];
                    }
                } else {
                    n[q][k] = nb[size_t(q) * plane + k];
                }
            }
        }

        auto weigh = [&](const P2 (&D)[L / 2], const int j) {
#pragma unroll
            for (int o2 = 0; o2 < L / 2; ++o2) {
                const P2 t = pfma(D[o2], c1, nc2);
                const T w0_ = weight_of(clamp0_nan(t.x));
                const T w1_ = weight_of(clamp0_nan(t.y));
                const int o = 2 * o2;
                const P2 w2 = mk2(w0_, w1_);
                S2[o2] = padd(S2[o2], w2);
                M[o] = tmax(M[o], w0_);
                M[o + 1] = tmax(M[o + 1], w1_);
                if constexpr (NEFF) Q2[o2] = pfma(w2, w2, Q2[o2]);
                const P2 w0b = mk2(w0_, w0_), w1b = mk2(w1_, w1_);
#pragma unroll
                for (int q = 0; q < NV4; ++q) {
                    if constexpr (HALF) {
                        acc_lo[q][o] = pfma(w0b, lo2(n[q][o + FR + j]), acc_lo[q][o]);
                        acc_lo[q][o + 1] = pfma(w1b, lo2(n[q][o + 1 + FR + j]), acc_lo[q][o + 1]);
                        if (q != NV4 - 1) {
                            acc_hi[q][o] = pfma(w0b, hi2(n[q][o + FR + j]), acc_hi[q][o]);
                            acc_hi[q][o + 1] = pfma(w1b, hi2(n[q][o + 1 + FR + j]), acc_hi[q][o + 1]);
                        }
                    } else {
                        acc_lo[q][o] = pfma(w0b, lo2(n[q][o + FR + j]), acc_lo[q][o]);
                        acc_hi[q][o] = pfma(w0b, hi2(n[q][o + FR + j]), acc_hi[q][o]);
                        acc_lo[q][o + 1] = pfma(w1b, lo2(n[q][o + 1 + FR + j]), acc_lo[q][o + 1]);
                        acc_hi[q][o + 1] = pfma(w1b, hi2(n[q][o + 1 + FR + j]), acc_hi[q][o + 1]);
                    }
                }
            }
        };

        // ---- phase A: squared differences, box sums along R (registers) and X (shuffles) ----
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            if constexpr (CENTRE) {
                if (ch0 + j == 0) continue;   // p == q is excluded (nd/_filters.pyx:368-369)
            }
            T s[E];
#pragma unroll
            for (int e = 0; e < E; ++e) {
                P2 sq;
#pragma unroll
                for (int q = 0; q < NV4; ++q) {
                    if constexpr (HALF) {
                        const P2 d0 = padd(lo2(c[q][e]), pneg(lo2(n[q][e + j])));
                        sq = (q == 0) ? pmul(d0, d0) : pfma(d0, d0, sq);
                        if (q != NV4 - 1) {
                            const P2 d1 = padd(hi2(c[q][e]), pneg(hi2(n[q][e + j])));
                            sq = pfma(d1, d1, sq);
                        }
                    } else {
                        const P2 d0 = padd(lo2(c[q][e]), pneg(lo2(n[q][e + j])));
                        const P2 d1 = padd(hi2(c[q][e]), pneg(hi2(n[q][e + j])));
                        sq = (q == 0) ? pmul(d0, d0) : pfma(d0, d0, sq);
                        sq = pfma(d1, d1, sq);
                    }
                }
                s[e] = sq.x + sq.y;
            }
            T pr[L];
            if constexpr (FR == 1 && FW > 0 && !NDNLM_NO_PAIRED) column_box_sum_paired<L>(s, pr);
            else column_box_sum<FR, L>(s, pr);
            P2 px[L / 2];
#pragma unroll
            for (int o2 = 0; o2 < L / 2; ++o2) px[o2] = lane_box_sum2<FX>(mk2(pr[2 * o2], pr[2 * o2 + 1]));
            if constexpr (FW == 0) {
                weigh(px, j);
            } else {
                // before the first store of this chunk: my readers must be done with the previous round
                // (on a fresh barrier the wait for the "previous" parity returns at once)
                if constexpr (!CENTRE && !NDNLM_DEBUG_CTA_SYNC) {
                    if (j == 0) mbar_wait(mbar_empty + xw, xpar ^ 1);
                }
                if constexpr (L == 4) {
                    // one 16-B store / load per row and offset: [j][row][lane] float4
                    if (ex_store) ex_own4[j * EX_J4] = mk4(px[0].x, px[0].y, px[1].x, px[1].y);
                } else {
#pragma unroll
                    for (int o2 = 0; o2 < L / 2; ++o2) ex_own[j * EX_J + o2 * 32] = px[o2];
                }
                if constexpr (NDNLM_KEEP_OWN != 0) {
#pragma unroll
                    for (int o2 = 0; o2 < L / 2; ++o2) own[j][o2] = px[o2];
                }
            }
        }

        // ---- phase B: box sum along W through shared memory, then weights ----
        if constexpr (FW > 0) {
            __syncwarp();
            if constexpr (NDNLM_DEBUG_CTA_SYNC) __syncthreads();
            // release: my sums are published -- tell every valid row that reads them (lanes 0..2FW-1, one each)
            if (!NDNLM_DEBUG_CTA_SYNC && lane < 2 * FW) {
                const int d = (lane < FW) ? lane - FW : lane - FW + 1;
                if (xw + d >= FW && xw + d < NROWS - FW) mbar_arrive(mbar_full + xw + d);
            }
            if (wvalid) {
                if constexpr (!NDNLM_DEBUG_CTA_SYNC) mbar_wait(mbar_full + xw, xpar);   // acquire: all rows I read are published
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    if constexpr (CENTRE) {
                        if (ch0 + j == 0) continue;
                    }
                    P2 D[L / 2];
                    if constexpr (L == 4) {
                        V4 t = ex_own4[j * EX_J4 - FW * EXW];
                        D[0] = mk2(t.x, t.y);
                        D[1] = mk2(t.z, t.w);
#pragma unroll
                        for (int d = -FW + 1; d <= FW; ++d) {
                            if (NDNLM_KEEP_OWN != 0 && d == 0) {
                                D[0] = padd(D[0], own[j][0]);
                                D[1] = padd(D[1], own[j][1]);
                            } else {
                                t = ex_own4[j * EX_J4 + d * EXW];
                                D[0] = padd(D[0], mk2(t.x, t.y));
                                D[1] = padd(D[1], mk2(t.z, t.w));
                            }
                        }
                    } else {
#pragma unroll
                        for (int o2 = 0; o2 < L / 2; ++o2) {
                            P2 t = ex_own[j * EX_J + o2 * 32 - FW * EX_ROW];
#pragma unroll
                            for (int d = -FW + 1; d <= FW; ++d) {
                                if (NDNLM_KEEP_OWN != 0 && d == 0) t = padd(t, own[j][o2]);
                                else t = padd(t, ex_own[j * EX_J + o2 * 32 + d * EX_ROW]);
                            }
                            D[o2] = t;
                        }
                    }
                    weigh(D, j);
                }
                __syncwarp();
                if (!NDNLM_DEBUG_CTA_SYNC && lane < 2 * FW) {         // done reading the neighbour rows
                    const int d = (lane < FW) ? lane - FW : lane - FW + 1;
                    mbar_arrive(mbar_empty + xw + d);
                }
            }
            if constexpr (NDNLM_DEBUG_CTA_SYNC) __syncthreads();
            xpar ^= 1;
        }
    };

    // The R-offset range [-rR, rR] is cut into chunks of CH; all chunks of a step are full except the last.
    // When the whole range fits ONE chunk (2 rR + 1 <= CH, e.g. cfg3: 5 offsets) the chunk size is hoisted
    // out of the offset loops, so the hot loop contains no dispatch at all.
    auto fold_weight_sums = [&]() {
#pragma unroll
        for (int o2 = 0; o2 < L / 2; ++o2) {
            Sd[2 * o2] += NDNLM_FOLD_T(S2[o2].x);
            Sd[2 * o2 + 1] += NDNLM_FOLD_T(S2[o2].y);
            S2[o2] = mk2(T(0), T(0));
            if constexpr (NEFF) {
                Qd[2 * o2] += NDNLM_FOLD_T(Q2[o2].x);
                Qd[2 * o2 + 1] += NDNLM_FOLD_T(Q2[o2].y);
                Q2[o2] = mk2(T(0), T(0));
            }
        }
    };
    const int nR = 2 * rR + 1;
    if constexpr (DH) {
        if (ww < FW) {
            // ---- a double-duty halo warp: phase A only, for its two rows ww (above the valid rows) and ww2 (below) ----
            // It keeps no accumulators (their registers hold the second centre column), runs the same sweep over passes
            // and offsets as the other warps with the same CTA barriers (one per pass change, those of load_pass), and
            // leaves before the epilogue.  The arithmetic is phase A of `chunk` above, expression by expression: the
            // sums a halo row publishes must not depend on which kind of warp computed them.
            const int ww2 = NROWS - FW + ww;
            V4 c2[NV4][E];
            {
                const int gw = w0 + ww2 + P.rad[0], gx = x0 + lx;
                const bool inb = gw < P.pd[0] && gx < P.pd[2];
#pragma unroll
                for (int q = 0; q < NV4; ++q)
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        const int gr = r0 + lr0 + e;
                        c2[q][e] = (inb && gr < P.pd[1])
                                       ? padded[((size_t(q) * P.pd[0] + gw) * P.pd[2] + gx) * P.pd[1] + gr]
                                       : mk4(T(0), T(0), T(0), T(0));
                    }
            }
            static_assert(!DH || !HALF, "no half-group variant of the double-duty halo warps");
            auto halo_chunk = [&](auto nj_tag, auto centre_tag, const V4 (&cc)[NV4][E], const int hrow, const uint32_t par,
                                  const V4* nb, const int ch0) {
                constexpr int NJ = decltype(nj_tag)::value;
                constexpr bool CENTRE = decltype(centre_tag)::value;
                constexpr int WNJ = E + NJ - 1;
                V4 n[NV4][WNJ];
#pragma unroll
                for (int k = 0; k < WNJ; ++k)
#pragma unroll
                    for (int q = 0; q < NV4; ++q) n[q][k] = nb[size_t(q) * plane + k];
                // my readers must be done with the previous round before its slots are overwritten
                if constexpr (!NDNLM_DEBUG_CTA_SYNC) mbar_wait(mbar_empty + hrow, par ^ 1);
                [[maybe_unused]] P2* const ex = exch + (hrow * (L / 2)) * 32 + lane;
                [[maybe_unused]] V4* const ex4 = reinterpret_cast<V4*>(exch) + hrow * 32 + lane;
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    if constexpr (CENTRE) {
                        if (ch0 + j == 0) continue;
                    }
                    T s[E];
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        P2 sq;
#pragma unroll
                        for (int q = 0; q < NV4; ++q) {
                            const P2 d0 = padd(lo2(cc[q][e]), pneg(lo2(n[q][e + j])));
                            const P2 d1 = padd(hi2(cc[q][e]), pneg(hi2(n[q][e + j])));
                            sq = (q == 0) ? pmul(d0, d0) : pfma(d0, d0, sq);
                            sq = pfma(d1, d1, sq);
                        }
                        s[e] = sq.x + sq.y;
                    }
                    T pr[L];
                    if constexpr (FR == 1 && !NDNLM_NO_PAIRED) column_box_sum_paired<L>(s, pr);
                    else column_box_sum<FR, L>(s, pr);
                    P2 px[L / 2];
#pragma unroll
                    for (int o2 = 0; o2 < L / 2; ++o2) px[o2] = lane_box_sum2<FX>(mk2(pr[2 * o2], pr[2 * o2 + 1]));
                    if constexpr (L == 4) {
                        ex4[j * EX_J4] = mk4(px[0].x, px[0].y, px[1].x, px[1].y);
                    } else {
#pragma unroll
                        for (int o2 = 0; o2 < L / 2; ++o2) ex[j * EX_J + o2 * 32] = px[o2];
                    }
                }
                __syncwarp();
                if (!NDNLM_DEBUG_CTA_SYNC && lane < 2 * FW) {      // published: tell every valid row that reads this one
                    const int d = (lane < FW) ? lane - FW : lane - FW + 1;
                    if (hrow + d >= FW && hrow + d < NROWS - FW) mbar_arrive(mbar_full + hrow + d);
                }
            };
            uint32_t hpar = 0;
            const int drow = (ww2 - ww) * BX * BRP;
            for (int pass = 0; pass < P.npass; ++pass) {
                const int twa = -rW + pass * P.ntw_pass;
                const int twb = min(rW, twa + P.ntw_pass - 1);
                if (pass > 0) __syncthreads();
                load_pass(pass);
                for (int tw = twa; tw <= twb; ++tw) {
                    for (int tx = -rX; tx <= rX; ++tx) {
                        const V4* nb0 = tile + ((ww + tw - twa) * BX + lx + tx) * BRP + lr0;
                        const bool centre_step = (tw == 0) & (tx == 0);
                        for (int ch0 = -rR; ch0 <= rR; ch0 += CH) {
                            const int nj = min(CH, rR - ch0 + 1);                        // uniform
                            const bool centre = centre_step && ch0 <= 0 && ch0 + nj > 0;
                            dispatch_chunk<CH>(nj, centre, [&](auto nj_tag, auto centre_tag) {
                                halo_chunk(nj_tag, centre_tag, c, ww, hpar, nb0 + ch0, ch0);
                                halo_chunk(nj_tag, centre_tag, c2, ww2, hpar, nb0 + drow + ch0, ch0);
                            });
                            if constexpr (NDNLM_DEBUG_CTA_SYNC) {      // the two CTA barriers of `chunk` in that mode
                                __syncthreads();
                                __syncthreads();
                            }
                            hpar ^= 1;
                        }
                    }
                }
            }
            return;
        }
    }
    for (int pass = 0; pass < (PERSIST ? 1 : P.npass); ++pass) {
        const int twa = -rW + pass * P.ntw_pass;
        const int twb = min(rW, twa + P.ntw_pass - 1);
        if (pass > 0) {                    // every warp is done with the previous pass's rows
            NDNLM_PROBE(2);
            __syncthreads();
            NDNLM_PROBE(3);
        }
        if constexpr (PERSIST) {
            // the box of every tile but the first was requested at the end of the previous tile
            if (tk > 0 && !P.use_ldg_loader) mbar_wait(mbar, uint32_t(tk & 1));
            else load_pass(0);
        } else {
            load_pass(pass);
        }
        NDNLM_PROBE(pass == 0 ? 1 : 4);
        if constexpr (PERSIST) {
            // one pass: every row of the tile, halo rows included, is in the box (padded row w0 + ww + rW is box row ww + rW)
            const V4* cs = tile + ((ww + rW) * BX + lx) * BRP + lr0;
#pragma unroll
            for (int q = 0; q < NV4; ++q)
#pragma unroll
                for (int e = 0; e < E; ++e) c[q][e] = cs[size_t(q) * plane + e];
        }
        if (nR <= CH) {
            dispatch_chunk<CH>(nR, false, [&](auto nj_tag, auto) {
                for (int tw = twa; tw <= twb; ++tw) {
                    for (int tx = -rX; tx <= rX; ++tx) {
                        const V4* nb0 = tile + ((ww + tw - twa) * BX + lx + tx) * BRP + lr0 - rR;
                        if ((tw == 0) & (tx == 0)) chunk(nj_tag, std::true_type{}, nb0, -rR);
                        else chunk(nj_tag, std::false_type{}, nb0, -rR);
                    }
                    fold_weight_sums();   // fp32 partial weight sums of this W-offset row -> float64
                }
            });
        } else {
            for (int tw = twa; tw <= twb; ++tw) {
                for (int tx = -rX; tx <= rX; ++tx) {
                    const V4* nb0 = tile + ((ww + tw - twa) * BX + lx + tx) * BRP + lr0;
                    const bool centre_step = (tw == 0) & (tx == 0);
                    for (int ch0 = -rR; ch0 <= rR; ch0 += CH) {
                        const int nj = min(CH, rR - ch0 + 1);                        // uniform
                        const bool centre = centre_step && ch0 <= 0 && ch0 + nj > 0;
                        dispatch_chunk<CH>(nj, centre, [&](auto nj_tag, auto centre_tag) {
                            chunk(nj_tag, centre_tag, nb0 + ch0, ch0);
                        });
                    }
                }
                fold_weight_sums();
            }
        }
    }

    NDNLM_PROBE(5);
    if constexpr (PERSIST) {
        // The box is dead once every warp is here: request the next tile's box now, so that it lands while this tile runs
        // its epilogue (registers and global memory only).  Every exchange round of this tile is complete as well.
        __syncthreads();
        NDNLM_PROBE(3);
        xpar_carry = xpar;
        const int next = tile_id + int(gridDim.x);
        if (threadIdx.x == 0 && next < ntiles && !P.use_ldg_loader) {
            int nb = next;
            const int nx0 = (nb % P.tiles[2]) * P.t[2];
            nb /= P.tiles[2];
            const int nr0 = (nb % P.tiles[1]) * P.t[1], nw0 = (nb / P.tiles[1]) * P.t[0];
            mbar_arrive_expect_tx(mbar, uint32_t(NV4) * uint32_t(BW * BRP * BX) * uint32_t(sizeof(V4)));
#pragma unroll
            for (int q = 0; q < NV4; ++q) tma_load_5d(tile + size_t(q) * plane, &tmap, mbar, 0, nr0, nx0, nw0, q);
        }
    }

    // ---- epilogue: self weight, normalise, store (nd/_filters.pyx:405-420) ----
    const int gw_ = w0 + ww - FW;
    const int gx_ = x0 + wx * TXW + lane - FX;
    if (wvalid && lane >= FX && lane < 32 - FX && gw_ < P.n[0] && gx_ < P.n[2]) {
        V4* po = out + (size_t(gw_) * P.n[2] + gx_) * P.n[1] + (r0 + wr * L);   // out is [q][W][X][R]
        const size_t oplane = size_t(P.n[0]) * P.n[1] * P.n[2];
#pragma unroll
        for (int o = 0; o < L; ++o) {
            const int gr_ = r0 + wr * L + o;
            if (gr_ >= P.n[1]) continue;
            double ws;
            // Every neighbour weight below 2^-126 flushes to zero in fp32 (ex2.approx.ftz): the float64 weights of the
            // reference would still be positive there.  Such a voxel is left unfiltered (self weight 1) and reported
            // through bit 1 of the flag instead of silently producing 0 / 0 (DESIGN.md 5, domain note).
            const bool underflow = (double(Sd[o]) == 0.0);
            if (underflow) atomicOr(err, 2);
            if constexpr (NEFF) {
                const double n_ = P.n_eff, Sx = double(Sd[o]), Qx = double(Qd[o]);
                if (underflow) {
                    ws = 1.0;
                } else {
                    if (n_ - 1.0 > Sx * Sx / Qx) atomicOr(err, 1);   // find_weight: 'No solution' (:310-311)
                    ws = (Sx + sqrt(n_ * Sx * Sx - n_ * n_ * Qx + n_ * Qx)) / (n_ - 1.0);
                }
            } else {
                ws = (M[o] == T(0)) ? 1.0 : double(M[o]);
            }
            const double tot = double(Sd[o]) + ws;
#pragma unroll
            for (int q = 0; q < NV4; ++q) {
                const V4 cc = c[q][o + FR];
                V4 res;
                // weighted_sum has the data type in the reference and is rounded after the self term (:419)
                res.x = T(double(T(double(acc_lo[q][o].x) + ws * double(cc.x))) / tot);
                res.y = T(double(T(double(acc_lo[q][o].y) + ws * double(cc.y))) / tot);
                if constexpr (HALF) {
                    if (q == NV4 - 1) {
                        res.z = T(0);
                        res.w = T(0);
                    } else {
                        res.z = T(double(T(double(acc_hi[q][o].x) + ws * double(cc.z))) / tot);
                        res.w = T(double(T(double(acc_hi[q][o].y) + ws * double(cc.w))) / tot);
                    }
                } else {
                    res.z = T(double(T(double(acc_hi[q][o].x) + ws * double(cc.z))) / tot);
                    res.w = T(double(T(double(acc_hi[q][o].y) + ws * double(cc.w))) / tot);
                }
                po[q * oplane + o] = res;
            }
        }
    }
#if NDNLM_TILE_PROBE
    __syncwarp();
#endif
    NDNLM_PROBE(6);
    tile_id += int(gridDim.x);
    ++tk;
    } while (PERSIST && tile_id < ntiles);
#undef NDNLM_PROBE
}

}  // namespace ndnlm
