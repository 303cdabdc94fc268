// knn_grid.cu — a4, the production k-nearest-neighbour search: EXACT, but over a uniform cell grid instead of all M
// inputs.  Same contract and same bit-exact result as the brute-force kernels of knn.cu (and as the oracle):
// distance = ((dx*dx+dy*dy)+dz*dz) in non-fused fp32, order = (distance ascending, index ascending), first k.
//
// Replaces k_nearest_neighbor_kernel.cu:8-112 (one thread per query scanning every input, local-memory insertion
// sort).  The reference's call sites search small neighbourhoods in clouds of 256..8192 points (pointconv.py:46,
// pwc3d_core.py:81, RPEFlow_core.py:329-331, models/utils.py:148), so almost all of the M distance evaluations of a
// brute-force scan are wasted.
//
//   build  (one CTA per cloud)  bounding box -> cubic cells of side H sized for ~max(2,k/2) points per cell ->
//                               shared-memory histogram -> scan -> points scattered into cell order (x,y,z,index).
//                               The same kernel sorts 3-D QUERIES into the inputs' cells, so the 32 queries of a
//                               warp look at the same few cells (their candidate loads coalesce into broadcasts).
//   query  (one thread per query)  scan the (2r+1)^D block of cells around the query's cell with a sorted
//                               k-list in registers; stop when the k-th best is provably final, else double r
//                               and rescan; a block that covers the whole grid IS the brute-force scan.
//
// Why the early stop is exact.  cell(x) = clamp(floor(fl(fl(x - lo) * inv_h))) is monotone in x, so a point whose
// cell lies beyond a face of the scanned block is farther from the query than R = (distance from the query to that
// face's plane lo + j*H) - delta along that axis, where delta bounds the rounding in the cell computation (relative
// 2^-24 per operation on magnitudes <= extent + a few H; delta = 2^-19 * (extent + 16 H) is > 30x that).  Its fp32
// distance is therefore >= R^2 * (1 - 5u), u = 2^-24 being the rounding of each of the five fp32 operations on
// non-negative terms.  If the k-th best distance found so far is STRICTLY below thr = R^2 * (1 - 2^-20) (fp64,
// rounded down), with R the minimum over the faces that have cells behind them, no unseen point can enter the
// list or tie with it, so the list equals the brute-force answer.  Within the scanned block the list is ordered by the full (distance, index) key, so the order in
// which cells (and the atomically scattered points inside a cell) are visited does not matter.
#include <math_constants.h>

#include "common.cuh"

namespace b200 {

constexpr int KG_CELLS_MAX = 16384;     // cells per cloud (64 KB shared-memory histogram in the build kernel)
constexpr int KG_GMAX = 1024;           // cells per axis
constexpr int KG_BUILD_THREADS = 1024;
constexpr int KG_QUERY_THREADS = 128;
constexpr int KG_STEP = 4;              // candidates per lane per lock-step iteration of the batched query (votes amortised)

struct KnnGridParams {                  // 48 bytes per cloud, written by the build kernel
    float lo[3];
    float inv_h;
    int G[3];
    int cells;
    double H;                           // cell side as the cell function sees it: 1 / (double)inv_h
    double delta;                       // bound on the rounding of the cell function, see the header comment
};

__device__ __forceinline__ int kg_cell(float x, float lo, float inv_h, int G) {
    const int c = __float2int_rd(__fmul_rn(__fsub_rn(x, lo), inv_h));      // NaN -> 0; saturates
    return min(max(c, 0), G - 1);
}

template <int D>
__device__ __forceinline__ int kg_cell_index(const KnnGridParams& p, float x, float y, float z) {
    const int cx = kg_cell(x, p.lo[0], p.inv_h, p.G[0]);
    const int cy = kg_cell(y, p.lo[1], p.inv_h, p.G[1]);
    const int cz = D == 3 ? kg_cell(z, p.lo[2], p.inv_h, p.G[2]) : 0;
    return (cz * p.G[1] + cy) * p.G[0] + cx;
}

// ---- build: bounding box + cell geometry (make_params) -> histogram -> scan -> scatter ---------------------------
template <int D>
__global__ void __launch_bounds__(KG_BUILD_THREADS)
knn_grid_build_kernel(const float* __restrict__ pts, int M, int sp, int sd, int ctarget, int make_params,
                      KnnGridParams* __restrict__ params, int* __restrict__ cell_start, float4* __restrict__ sorted) {
    // coordinate d of point i is pts[i * sp + d * sd]: (sp, sd) = (D, 1) for point-major [M,D] clouds (the extension entry,
    // k_nearest_neighbor.cpp:6) and (1, M) for the channel-first [D,M] clouds every model call site passes (wrapper.py:119)
    extern __shared__ int s_hist[];                      // [cells + 1]
    __shared__ float s_red[2 * 3][32];
    __shared__ int s_warp_tot[32];
    __shared__ KnnGridParams s_p;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pts += (size_t)b * M * D;

    if (make_params) {
        float mn[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, mx[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
        for (int i = tid; i < M; i += KG_BUILD_THREADS) {
#pragma unroll
            for (int d = 0; d < D; ++d) {
                const float v = __ldg(pts + (size_t)i * sp + (size_t)d * sd);
                mn[d] = fminf(mn[d], v);                 // fminf/fmaxf drop NaNs
                mx[d] = fmaxf(mx[d], v);
            }
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                mn[d] = fminf(mn[d], __shfl_xor_sync(FULL, mn[d], o));
                mx[d] = fmaxf(mx[d], __shfl_xor_sync(FULL, mx[d], o));
            }
            if (lane == 0) { s_red[d][warp] = mn[d]; s_red[3 + d][warp] = mx[d]; }
        }
        __syncthreads();
        if (tid == 0) {
            KnnGridParams p;
            double ext[3] = {0.0, 0.0, 0.0}, vol = 1.0, maxext = 0.0;
            int nd = 0;
            for (int d = 0; d < 3; ++d) { p.lo[d] = 0.0f; p.G[d] = 1; }
            for (int d = 0; d < D; ++d) {
                float lo = CUDART_INF_F, hi = -CUDART_INF_F;
                for (int w = 0; w < KG_BUILD_THREADS / 32; ++w) { lo = fminf(lo, s_red[d][w]); hi = fmaxf(hi, s_red[3 + d][w]); }
                const double e = (double)hi - (double)lo;
                p.lo[d] = isfinite(lo) ? lo : 0.0f;
                if (isfinite(e) && e > 0.0) { ext[d] = e; vol *= e; maxext = fmax(maxext, e); ++nd; }
            }
            p.inv_h = 0.0f;                              // one cell: every query scans everything
            if (nd > 0 && isfinite(vol) && vol > 0.0) {
                const double ntarget = fmax(1.0, (double)M / (double)ctarget);
                double h = pow(vol / ntarget, 1.0 / nd);
                for (int iter = 0; iter < 200; ++iter) {
                    const float ih = (float)(1.0 / h);
                    if (!(ih > 0.0f) || !isfinite(ih)) break;
                    long long total = 1;
                    int g[3] = {1, 1, 1};
                    for (int d = 0; d < D; ++d) {
                        g[d] = ext[d] > 0.0 ? (int)fmin((double)KG_GMAX, floor(ext[d] * (double)ih) + 1.0) : 1;
                        total *= g[d];
                    }
                    if (total <= KG_CELLS_MAX) {
                        p.inv_h = ih;
                        for (int d = 0; d < 3; ++d) p.G[d] = g[d];
                        break;
                    }
                    h *= 1.25;
                }
            }
            p.cells = p.G[0] * p.G[1] * p.G[2];
            p.H = p.inv_h > 0.0f ? 1.0 / (double)p.inv_h : 0.0;
            p.delta = ldexp(maxext + 16.0 * p.H, -19);
            s_p = p;
            params[b] = p;
        }
    } else if (tid == 0) {
        s_p = params[b];
    }
    __syncthreads();
    const KnnGridParams p = s_p;
    const int cells = p.cells;

    for (int c = tid; c <= cells; c += KG_BUILD_THREADS) s_hist[c] = 0;
    __syncthreads();
    for (int i = tid; i < M; i += KG_BUILD_THREADS) {
        const float x = __ldg(pts + (size_t)i * sp), y = __ldg(pts + (size_t)i * sp + sd);
        const float z = D == 3 ? __ldg(pts + (size_t)i * sp + 2 * (size_t)sd) : 0.0f;
        atomicAdd(&s_hist[kg_cell_index<D>(p, x, y, z)], 1);
    }
    __syncthreads();

    // exclusive scan of s_hist[0..cells): each thread owns a run of consecutive cells
    const int per = (cells + KG_BUILD_THREADS - 1) / KG_BUILD_THREADS;
    const int c0 = min(tid * per, cells), c1 = min(c0 + per, cells);
    int run = 0;
    for (int c = c0; c < c1; ++c) run += s_hist[c];
    int incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int v = s_warp_tot[lane], iv = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(FULL, iv, o);
            if (lane >= o) iv += u;
        }
        s_warp_tot[lane] = iv - v;                       // exclusive warp offsets
    }
    __syncthreads();
    int off = s_warp_tot[warp] + incl - run;
    for (int c = c0; c < c1; ++c) {
        const int n = s_hist[c];
        s_hist[c] = off;
        off += n;
    }
    if (tid == KG_BUILD_THREADS - 1) s_hist[cells] = M;
    __syncthreads();
    if (cell_start) {
        int* cs = cell_start + (size_t)b * (KG_CELLS_MAX + 1);
        for (int c = tid; c <= cells; c += KG_BUILD_THREADS) cs[c] = s_hist[c];
    }
    __syncthreads();
    float4* out = sorted + (size_t)b * M;
    for (int i = tid; i < M; i += KG_BUILD_THREADS) {    // s_hist now serves as the per-cell write cursor
        const float x = __ldg(pts + (size_t)i * sp), y = __ldg(pts + (size_t)i * sp + sd);
        const float z = D == 3 ? __ldg(pts + (size_t)i * sp + 2 * (size_t)sd) : 0.0f;
        const int pos = atomicAdd(&s_hist[kg_cell_index<D>(p, x, y, z)], 1);
        out[pos] = make_float4(x, y, z, __int_as_float(i));
    }
}

// ---- query ---------------------------------------------------------------------------------------------------
// One thread per query.  The k-list lives in KMAX registers as 64-bit keys (distance bits << 32 | index): distances
// are >= +0, so unsigned key order IS the (distance, index) order, and a NaN/inf distance can never beat the
// (inf, 0) key of an empty slot.  When k < KMAX the first KMAX-k slots hold key 0, which nothing can displace, so
// every register index is static.
constexpr u64 KG_EMPTY = (u64)0x7f800000u << 32;         // (distance +inf, index 0): k_nearest_neighbor.cpp:16 zero-initialises

__device__ __forceinline__ void kg_cswap(u64& a, u64& b) {           // a <- min, b <- max
    const bool sw = b < a;
    const u64 t = sw ? b : a;
    b = sw ? a : b;
    a = t;
}

template <int N>
__device__ __forceinline__ void kg_bitonic_sort(u64 (&a)[N]) {       // ascending, fully unrolled network
#pragma unroll
    for (int k = 2; k <= N; k <<= 1)
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1)
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const int l = i ^ j;
                if (l > i) {
                    if ((i & k) == 0) kg_cswap(a[i], a[l]);
                    else kg_cswap(a[l], a[i]);
                }
            }
}

// L (sorted) <- the N smallest of L and a sorted batch: elementwise min against the reversed batch leaves a bitonic
// sequence holding exactly those N keys; log2(N) half-cleaner stages sort it.
template <int N>
__device__ __forceinline__ void kg_merge_sorted(u64 (&L)[N], const u64 (&batch)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) L[i] = batch[N - 1 - i] < L[i] ? batch[N - 1 - i] : L[i];
#pragma unroll
    for (int j = N >> 1; j > 0; j >>= 1)
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const int l = i ^ j;
            if (l > i) kg_cswap(L[i], L[l]);
        }
}

template <int KMAX>
__device__ __forceinline__ void kg_insert(u64 (&L)[KMAX], u64 key) {
#pragma unroll
    for (int s = 0; s < KMAX; ++s) {                     // bubble through: the list stays sorted
        const bool lt = key < L[s];
        const u64 t = lt ? L[s] : key;
        L[s] = lt ? key : L[s];
        key = t;
    }
}

struct KgQuery {
    float qx, qy, qz;
    int orig, cx, cy, cz;
    bool live;
};

template <int D>
__device__ __forceinline__ KgQuery kg_load_query(const KnnGridParams& p, const float4* __restrict__ sorted_q,
                                                 const float* __restrict__ raw_q, int qsp, int qsd, int b, int t, int Q) {
    KgQuery q;
    q.live = t < Q;
    q.qx = q.qy = q.qz = 0.0f;
    q.orig = t;
    if (q.live) {
        if (sorted_q) {
            const float4 v = __ldg(sorted_q + (size_t)b * Q + t);
            q.qx = v.x; q.qy = v.y; q.qz = v.z; q.orig = __float_as_int(v.w);
        } else {
            const float* v = raw_q + (size_t)b * Q * D + (size_t)t * qsp;
            q.qx = __ldg(v); q.qy = __ldg(v + qsd);
            if (D == 3) q.qz = __ldg(v + 2 * (size_t)qsd);
        }
    }
    q.cx = kg_cell(q.qx, p.lo[0], p.inv_h, p.G[0]);
    q.cy = kg_cell(q.qy, p.lo[1], p.inv_h, p.G[1]);
    q.cz = D == 3 ? kg_cell(q.qz, p.lo[2], p.inv_h, p.G[2]) : 0;
    return q;
}

// Largest fp32 value T such that a k-th best distance < T proves the search of the (2r+1)^D block final: every
// unseen point lies beyond one of the block's faces, i.e. farther than R = (distance from the query to the nearest
// face that has cells behind it) - delta along that axis; its fp32 distance is >= R^2 (1 - 5u).
template <int D>
__device__ __forceinline__ float kg_bound(const KnnGridParams& p, const KgQuery& q, int r) {
    double R = CUDART_INF;
    const float qc[3] = {q.qx, q.qy, q.qz};
    const int cc[3] = {q.cx, q.cy, q.cz};
#pragma unroll
    for (int d = 0; d < D; ++d) {
        if (cc[d] - r > 0) R = fmin(R, (double)qc[d] - ((double)p.lo[d] + (double)(cc[d] - r) * p.H));
        if (cc[d] + r < p.G[d] - 1) R = fmin(R, ((double)p.lo[d] + (double)(cc[d] + r + 1) * p.H) - (double)qc[d]);
    }
    R -= p.delta;
    if (!(R > 0.0) || !(R * R > 1e-30)) return 0.0f;     // below that fp32 products go subnormal: no relative bound
    if (!isfinite(R)) return CUDART_INF_F;               // no face has cells behind it: the block is the whole grid
    return __double2float_rd(R * R * (1.0 - 9.5367431640625e-07));
}

template <int D>
__device__ __forceinline__ u64 kg_key(const KgQuery& q, const float4& pt) {
    const float d = D == 3 ? sqdist3_rule(q.qx, q.qy, q.qz, pt.x, pt.y, pt.z) : sqdist2_rule(q.qx, q.qy, pt.x, pt.y);
    return ((u64)__float_as_uint(d) << 32) | (u64)(unsigned)__float_as_int(pt.w);
}

template <int KMAX>
__device__ __forceinline__ void kg_store(const u64 (&L)[KMAX], int64_t* __restrict__ o, int k) {
#pragma unroll
    for (int s = 0; s < KMAX; ++s)
        if (s >= KMAX - k) o[s - (KMAX - k)] = (int64_t)(unsigned)(L[s] & 0xffffffffull);
}

// Small k (KMAX <= 8): plain nested loops over the block's rows of cells, insert on the spot.
template <int D, int KMAX>
__global__ void __launch_bounds__(KG_QUERY_THREADS)
knn_grid_query_kernel(const float4* __restrict__ sorted_pts, const int* __restrict__ cell_start,
                      const KnnGridParams* __restrict__ params, const float4* __restrict__ sorted_q,
                      const float* __restrict__ raw_q, int qsp, int qsd, int64_t* __restrict__ out, int M, int Q, int k) {
    __shared__ KnnGridParams s_p;
    const int b = blockIdx.y, t = blockIdx.x * KG_QUERY_THREADS + threadIdx.x;
    if (threadIdx.x == 0) s_p = params[b];
    __syncthreads();
    const KgQuery q = kg_load_query<D>(s_p, sorted_q, raw_q, qsp, qsd, b, t, Q);
    if (!q.live) return;
    sorted_pts += (size_t)b * M;
    const int* cs = cell_start + (size_t)b * (KG_CELLS_MAX + 1);
    const int Gx = s_p.G[0], Gy = s_p.G[1], Gz = s_p.G[2];

    u64 L[KMAX];
    for (int r = 1;; r <<= 1) {
#pragma unroll
        for (int s = 0; s < KMAX; ++s) L[s] = s < KMAX - k ? 0ull : KG_EMPTY;
        const int x0 = max(q.cx - r, 0), x1 = min(q.cx + r, Gx - 1);
        const int y0 = max(q.cy - r, 0), y1 = min(q.cy + r, Gy - 1);
        const int z0 = D == 3 ? max(q.cz - r, 0) : 0, z1 = D == 3 ? min(q.cz + r, Gz - 1) : 0;
        for (int z = z0; z <= z1; ++z) {
            for (int y = y0; y <= y1; ++y) {
                const int rowbase = (z * Gy + y) * Gx;
                const int e = __ldg(cs + rowbase + x1 + 1);
                int c = __ldg(cs + rowbase + x0);                          // cells x0..x1 of a row are contiguous
                for (; c + KG_STEP <= e; c += KG_STEP) {                   // KG_STEP loads in flight per thread
                    float4 pt[KG_STEP];
#pragma unroll
                    for (int j = 0; j < KG_STEP; ++j) pt[j] = __ldg(sorted_pts + c + j);
#pragma unroll
                    for (int j = 0; j < KG_STEP; ++j) {
                        const u64 key = kg_key<D>(q, pt[j]);
                        if (key < L[KMAX - 1]) kg_insert<KMAX>(L, key);
                    }
                }
                for (; c < e; ++c) {
                    const u64 key = kg_key<D>(q, __ldg(sorted_pts + c));
                    if (key < L[KMAX - 1]) kg_insert<KMAX>(L, key);
                }
            }
        }
        const bool whole = x0 == 0 && y0 == 0 && z0 == 0 && x1 == Gx - 1 && y1 == Gy - 1 && z1 == Gz - 1;
        const float kth = __uint_as_float((unsigned)(L[KMAX - 1] >> 32));
        if (whole || kth < kg_bound<D>(s_p, q, r)) break;
    }
    kg_store<KMAX>(L, out + ((size_t)b * Q + q.orig) * k, k);
}

// Large k (KMAX = 16, 32): inserting into a sorted register list costs ~6*KMAX instructions and only a few lanes
// need it at any one candidate.  Candidates that beat the lane's current k-th best are parked in a per-lane
// shared-memory batch instead; when some lane's batch is full (and at the end of the block) the whole warp sorts
// its batches with a bitonic network and merges them into the lists — every lane busy, ~12*KMAX compare-swaps per
// KMAX parked candidates.  A parked candidate that is no longer good enough simply loses the merge.
// The warp walks the candidates in lock-step (each lane through its own rows of cells, KG_STEP candidates per step
// with their loads in flight together) so that it stays converged for the drains; a drain starts as soon as some
// lane's batch could overflow in the next step.
template <int D, int KMAX>
__global__ void __launch_bounds__(KG_QUERY_THREADS)
knn_grid_query_batched_kernel(const float4* __restrict__ sorted_pts, const int* __restrict__ cell_start,
                              const KnnGridParams* __restrict__ params, const float4* __restrict__ sorted_q,
                              const float* __restrict__ raw_q, int qsp, int qsd, int64_t* __restrict__ out, int M, int Q, int k) {
    __shared__ u64 s_batch[KMAX][KG_QUERY_THREADS];
    __shared__ KnnGridParams s_p;
    const int b = blockIdx.y, t = blockIdx.x * KG_QUERY_THREADS + threadIdx.x;
    if (threadIdx.x == 0) s_p = params[b];
    __syncthreads();
    const KgQuery q = kg_load_query<D>(s_p, sorted_q, raw_q, qsp, qsd, b, t, Q);   // dead lanes follow the warp with no candidates
    sorted_pts += (size_t)b * M;
    const int* cs = cell_start + (size_t)b * (KG_CELLS_MAX + 1);
    const int Gx = s_p.G[0], Gy = s_p.G[1], Gz = s_p.G[2];

    u64 L[KMAX];
#pragma unroll
    for (int s = 0; s < KMAX; ++s) L[s] = KG_EMPTY;
    bool done = !q.live;
    for (int r = 1;; r <<= 1) {
        const int x0 = max(q.cx - r, 0), x1 = min(q.cx + r, Gx - 1);
        const int y0 = max(q.cy - r, 0), y1 = min(q.cy + r, Gy - 1);
        const int z0 = D == 3 ? max(q.cz - r, 0) : 0, z1 = D == 3 ? min(q.cz + r, Gz - 1) : 0;
        if (!done) {                                     // finished lanes keep their list and offer no candidates
#pragma unroll
            for (int s = 0; s < KMAX; ++s) L[s] = s < KMAX - k ? 0ull : KG_EMPTY;
        }
        // A pass only counts if its k-th best ends up strictly below the stop bound of this block; candidates at or
        // beyond the bound cannot be part of such a result, so the bound also caps the parking threshold from the
        // start (a pass that finds fewer than k candidates under it fails the test below and the block doubles).
        const float bound = kg_bound<D>(s_p, q, r);
        const u64 bkey = (u64)__float_as_uint(bound) << 32;
        u64 thr = L[KMAX - 1] < bkey ? L[KMAX - 1] : bkey;
        // rows of cells: the query's own row first (it fills the list with near points, so most later candidates
        // fail the threshold test), then the others in storage order
        int y = y0, z = done ? z1 + 1 : z0, c = 0, e = 0, nb = 0;
        bool home = !done;
        while (true) {
            while (c >= e && (home || z <= z1)) {        // next non-empty row (cells x0..x1 of a row are contiguous)
                const int ry = home ? q.cy : y, rz = home ? q.cz : z;
                const bool skip = !home && ry == q.cy && rz == q.cz;
                const int rowbase = (rz * Gy + ry) * Gx;
                if (!skip) {
                    c = __ldg(cs + rowbase + x0);
                    e = __ldg(cs + rowbase + x1 + 1);
                }
                if (home) home = false;
                else if (++y > y1) { y = y0; ++z; }
            }
            const bool active = c < e;
            if (!__any_sync(FULL, active)) break;
            {                                            // up to KG_STEP candidates of this lane's row per warp step
                const int n = active ? min(e - c, KG_STEP) : 0;
                float4 pt[KG_STEP];
#pragma unroll
                for (int j = 0; j < KG_STEP; ++j)
                    if (j < n) pt[j] = __ldg(sorted_pts + c + j);
#pragma unroll
                for (int j = 0; j < KG_STEP; ++j)
                    if (j < n) {
                        const u64 key = kg_key<D>(q, pt[j]);
                        if (key < thr) s_batch[nb++][threadIdx.x] = key;
                    }
                c += n;
            }
            if (__any_sync(FULL, nb > KMAX - KG_STEP)) {  // the next step may park KG_STEP more
                u64 batch[KMAX];
#pragma unroll
                for (int j = 0; j < KMAX; ++j) batch[j] = j < nb ? s_batch[j][threadIdx.x] : ~0ull;
                kg_bitonic_sort<KMAX>(batch);
                kg_merge_sorted<KMAX>(L, batch);
                nb = 0;
                thr = L[KMAX - 1] < bkey ? L[KMAX - 1] : bkey;
            }
        }
        if (__any_sync(FULL, nb > 0)) {
            u64 batch[KMAX];
#pragma unroll
            for (int j = 0; j < KMAX; ++j) batch[j] = j < nb ? s_batch[j][threadIdx.x] : ~0ull;
            kg_bitonic_sort<KMAX>(batch);
            kg_merge_sorted<KMAX>(L, batch);
        }
        if (!done) {
            const bool whole = x0 == 0 && y0 == 0 && z0 == 0 && x1 == Gx - 1 && y1 == Gy - 1 && z1 == Gz - 1;
            const float kth = __uint_as_float((unsigned)(L[KMAX - 1] >> 32));
            done = whole || kth < bound;
        }
        if (__all_sync(FULL, done)) break;
    }
    if (q.live) kg_store<KMAX>(L, out + ((size_t)b * Q + q.orig) * k, k);
}

struct KnnGridScratch {
    KnnGridParams* params;
    int* cell_start;
    float4* sorted_pts;
    float4* sorted_q;
    int64_t total;
};
static KnnGridScratch kg_carve(void* base, int B, int M, int Q, int D) {
    KnnGridScratch s;
    int64_t off = 0;
    auto take = [&](int64_t bytes) {
        char* ptr = base ? static_cast<char*>(base) + off : nullptr;
        off += (bytes + 255) & ~int64_t(255);
        return ptr;
    };
    s.sorted_pts = reinterpret_cast<float4*>(take((int64_t)B * M * 16));
    s.sorted_q = D == 3 ? reinterpret_cast<float4*>(take((int64_t)B * Q * 16)) : nullptr;
    s.cell_start = reinterpret_cast<int*>(take((int64_t)B * (KG_CELLS_MAX + 1) * 4));
    s.params = reinterpret_cast<KnnGridParams*>(take((int64_t)B * sizeof(KnnGridParams)));
    s.total = off;
    return s;
}

template <int D, int KMAX>
static void kg_launch_query(const KnnGridScratch& s, const float* query, int qsp, int qsd, int64_t* idx, int B, int M, int Q, int k,
                            cudaStream_t st) {
    dim3 grid(ceil_div(Q, KG_QUERY_THREADS), B);
    if constexpr (KMAX >= 16)
        knn_grid_query_batched_kernel<D, KMAX><<<grid, KG_QUERY_THREADS, 0, st>>>(s.sorted_pts, s.cell_start, s.params, s.sorted_q,
                                                                                  query, qsp, qsd, idx, M, Q, k);
    else
        knn_grid_query_kernel<D, KMAX><<<grid, KG_QUERY_THREADS, 0, st>>>(s.sorted_pts, s.cell_start, s.params, s.sorted_q, query,
                                                                          qsp, qsd, idx, M, Q, k);
}

template <int D>
static cudaError_t kg_run(const float* input, const float* query, int64_t* idx, const KnnGridScratch& s, int B, int M, int Q,
                          int k, bool channel_first, cudaStream_t st) {
    const int isp = channel_first ? 1 : D, isd = channel_first ? M : 1;      // strides of the input cloud
    const int qsp = channel_first ? 1 : D, qsd = channel_first ? Q : 1;      // ... and of the queries
    const size_t smem = (size_t)(KG_CELLS_MAX + 1) * sizeof(int);
    cudaError_t e = cudaFuncSetAttribute(knn_grid_build_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int ctarget = k / 2 < 2 ? 2 : (k / 2 > 16 ? 16 : k / 2);
    if (k >= 16 && M <= 2048) ctarget = M <= 1024 ? 16 : 12;    // small clouds: coarser cells (self search 1024 pts, k = 16: 122 -> 89 us; 2048 pts: 202 -> 183 us)
    knn_grid_build_kernel<D><<<B, KG_BUILD_THREADS, smem, st>>>(input, M, isp, isd, ctarget, 1, s.params, s.cell_start, s.sorted_pts);
    KnnGridScratch q = s;
    if (s.sorted_q) {
        if (query == input && Q == M) q.sorted_q = s.sorted_pts;    // self search: the inputs' cell order is the queries'
        else                                                         // queries into the inputs' cells (no cell table needed)
            knn_grid_build_kernel<D><<<B, KG_BUILD_THREADS, smem, st>>>(query, Q, qsp, qsd, ctarget, 0, s.params, nullptr, s.sorted_q);
    }
    if (k == 1) kg_launch_query<D, 1>(q, query, qsp, qsd, idx, B, M, Q, k, st);
    else if (k <= 4) kg_launch_query<D, 4>(q, query, qsp, qsd, idx, B, M, Q, k, st);
    else if (k <= 8) kg_launch_query<D, 8>(q, query, qsp, qsd, idx, B, M, Q, k, st);
    else if (k <= 16) kg_launch_query<D, 16>(q, query, qsp, qsd, idx, B, M, Q, k, st);
    else kg_launch_query<D, 32>(q, query, qsp, qsd, idx, B, M, Q, k, st);
    return cudaGetLastError();
}

}  // namespace b200

extern "C" int64_t b200_knn_scratch_bytes(int B, int M, int Q, int D, int k) {
    (void)k;
    if (B < 0 || M < 0 || Q < 0) return 0;
    return b200::kg_carve(nullptr, B, M, Q, D).total;
}

static int knn_grid_entry(const float* input_xyz, const float* query_xyz, int64_t* idx, void* scratch, int64_t scratch_bytes, int B,
                          int M, int Q, int D, int k, bool channel_first, b200_stream_t stream);

extern "C" int b200_knn_grid(const float* input_xyz, const float* query_xyz, int64_t* idx, void* scratch,
                             int64_t scratch_bytes, int B, int M, int Q, int D, int k, b200_stream_t stream) {
    return knn_grid_entry(input_xyz, query_xyz, idx, scratch, scratch_bytes, B, M, Q, D, k, false, stream);
}

extern "C" int b200_knn_grid_cf(const float* input_xyz, const float* query_xyz, int64_t* idx, void* scratch,
                                int64_t scratch_bytes, int B, int M, int Q, int D, int k, b200_stream_t stream) {
    return knn_grid_entry(input_xyz, query_xyz, idx, scratch, scratch_bytes, B, M, Q, D, k, true, stream);
}

static int knn_grid_entry(const float* input_xyz, const float* query_xyz, int64_t* idx, void* scratch, int64_t scratch_bytes, int B,
                          int M, int Q, int D, int k, bool channel_first, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0 || Q == 0) || (input_xyz && query_xyz && idx && scratch), "b200_knn_grid: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(D == 2 || D == 3, "b200_knn_grid: D must be 2 or 3 (got %d)", D);
    B200_REQUIRE(k >= 1 && k <= 32, "b200_knn_grid: k must be in [1,32] (got %d); the reference kernel has 32 slots", k);
    B200_REQUIRE(B >= 0 && M >= 1 && Q >= 0, "b200_knn_grid: bad sizes B=%d M=%d Q=%d", B, M, Q);
    B200_REQUIRE(B <= 65535, "b200_knn_grid: B=%d exceeds gridDim.y", B);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 255) == 0, "b200_knn_grid: scratch must be 256-byte aligned");
    const KnnGridScratch s = kg_carve(scratch, B, M, Q, D);
    B200_REQUIRE(scratch_bytes >= s.total, "b200_knn_grid: scratch too small (%lld < %lld bytes)", (long long)scratch_bytes,
                 (long long)s.total);
    if (B == 0 || Q == 0) return B200_OK;
    const cudaError_t e = D == 2 ? kg_run<2>(input_xyz, query_xyz, idx, s, B, M, Q, k, channel_first, as_stream(stream))
                                 : kg_run<3>(input_xyz, query_xyz, idx, s, B, M, Q, k, channel_first, as_stream(stream));
    if (e != cudaSuccess) return cuda_fail(e, "b200_knn_grid");
    return B200_OK;
}
