// fps.cu — a3: furthest point sampling.
//
// Replaces models/csrc/furthest_point_sampling/furthest_point_sampling_kernel.cu:34-85 (one 1024-thread CTA
// per cloud; every iteration re-loads all points from global memory, read-modify-writes a global distance
// array, then does a 10-level shared-memory tree argmax with five __syncthreads).
//
// Here the points AND their running distances live in registers for the whole kernel, so an iteration is
// pure ALU work followed by a two-level warp argmax:
//   per thread : PPT points: d = ((dx*dx+dy*dy)+dz*dz) (non-fused), dist = min(dist, d), running (max, index)
//   per warp   : redux.sync.max on the distance bits, then redux.sync.min on the indices that hold that max
//   per CTA    : lane 0 of each warp -> shared slot; ONE __syncthreads; every warp repeats the two redux on
//                the <=32 slots, so every thread knows the winner without a second barrier (slots are
//                double-buffered by iteration parity).
// Clouds larger than 8192 points (config 5: 32768) are split over a thread-block cluster of CS CTAs; each CTA
// publishes {key, x, y, z} of its local winner into every peer's shared memory (DSMEM) and one cluster
// barrier per iteration replaces the global round trip.
//
// Exactness (SURVEY §8a): start at index 0, distances start at 1e10, ties -> LOWEST index.  Equal to the
// reference torch fallback models/csrc/wrapper.py:83-96 bit for bit.
#include <cooperative_groups.h>

#include "fps_common.cuh"

namespace cg = cooperative_groups;

namespace b200 {

struct FpsSlot {               // what a CTA publishes to its cluster peers each iteration
    unsigned long long key;    // (distance bits << 32) | (0xFFFFFFFF - index): max key = max distance, then min index
    float x, y, z, pad;
};

constexpr int FPS_PPT = 16, FPS_T = 512;               // points per thread, threads per CTA: 8192 points per CTA

template <int CS>
__global__ void __launch_bounds__(FPS_T, 1)
fps_kernel(const float* __restrict__ xyz, int64_t* __restrict__ out, int N, int S, float negzero) {
    constexpr int PPT = FPS_PPT, T = FPS_T, NW = T / 32;
    __shared__ unsigned s_d[2][32], s_i[2][32];
    __shared__ __align__(16) FpsSlot s_slot[2][CS];
    extern __shared__ float s_pts[];                     // xyz of this CTA's chunk

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rank = (int)cg::this_cluster().block_rank(), cloud = blockIdx.x / CS;
    const int chunk = (N + CS - 1) / CS;
    const int lo = rank * chunk, hi = min(N, lo + chunk);
    const float* P = xyz + (size_t)cloud * N * 3;

    float px[PPT], py[PPT], pz[PPT], dist[PPT];
#pragma unroll
    for (int i = 0; i < PPT; ++i) {
        const int gi = lo + i * T + tid;
        const bool ok = gi < hi;
        px[i] = ok ? __ldg(P + (size_t)gi * 3 + 0) : 0.0f;
        py[i] = ok ? __ldg(P + (size_t)gi * 3 + 1) : 0.0f;
        pz[i] = ok ? __ldg(P + (size_t)gi * 3 + 2) : 0.0f;
        dist[i] = ok ? 1e10f : 0.0f;                     // padding never beats a real point (index tie-break below)
        if (ok) {
            s_pts[(i * T + tid) * 3 + 0] = px[i];
            s_pts[(i * T + tid) * 3 + 1] = py[i];
            s_pts[(i * T + tid) * 3 + 2] = pz[i];
        }
    }
    cg::this_cluster().sync();

    unsigned cur = 0;
    float cx = __ldg(P + 0), cy = __ldg(P + 1), cz = __ldg(P + 2);
    int64_t* o = out + (size_t)cloud * S;

    for (int s = 0; s < S; ++s) {
        if (rank == 0 && tid == 0) o[s] = (int64_t)cur;
        if (s == S - 1) break;

        // Running argmax over this thread's points.  Only the slot number is tracked in the loop (SEL with an
        // immediate); padding slots hold distance 0 and an index >= hi, so they lose every tie to a real point.
        // Two points per FADD2/FFMA2 (non-fused rule kept, see sqr2).
        float bd = -1.0f;
        int bslot = 0;
        const u64 nz = pack2(negzero, negzero);
        const u64 c2x = pack2(cx, cx), c2y = pack2(cy, cy), c2z = pack2(cz, cz);
#pragma unroll
        for (int i = 0; i < PPT; i += 2) {
            float d0, d1;
            unpack2(sqdist_pair<3>(pack2(px[i], px[i + 1]), pack2(py[i], py[i + 1]), pack2(pz[i], pz[i + 1]),
                                   c2x, c2y, c2z, nz), d0, d1);
            dist[i] = fminf(dist[i], d0);
            dist[i + 1] = fminf(dist[i + 1], d1);
            if (dist[i] > bd) { bd = dist[i]; bslot = i; }                      // increasing index, strict '>': lowest index wins
            if (dist[i + 1] > bd) { bd = dist[i + 1]; bslot = i + 1; }
        }
        const unsigned bi = (unsigned)(lo + bslot * T + tid);
        const unsigned db = __float_as_uint(bd);         // distances are >= +0: the bit pattern orders like the value
        const unsigned wmax = __reduce_max_sync(FULL, db);
        const unsigned widx = __reduce_min_sync(FULL, db == wmax ? bi : 0xFFFFFFFFu);
        const int par = s & 1;
        if (lane == 0) { s_d[par][warp] = wmax; s_i[par][warp] = widx; }
        __syncthreads();

        cg::cluster_group cluster = cg::this_cluster();
        if (warp == 0) {
            const unsigned vd = lane < NW ? s_d[par][lane] : 0u;
            const unsigned vi = lane < NW ? s_i[par][lane] : 0xFFFFFFFFu;
            const unsigned gmax = __reduce_max_sync(FULL, vd);
            const unsigned gidx = __reduce_min_sync(FULL, vd == gmax ? vi : 0xFFFFFFFFu);
            if (lane < CS) {                             // lane r writes this CTA's winner into peer r's slot
                FpsSlot v;
                v.key = ((unsigned long long)gmax << 32) | (unsigned long long)(0xFFFFFFFFu - gidx);
                const int li = (int)gidx - lo;              // < PPT*T even for a padding slot (never the global winner)
                v.x = s_pts[li * 3 + 0]; v.y = s_pts[li * 3 + 1]; v.z = s_pts[li * 3 + 2]; v.pad = 0.0f;
                FpsSlot* dst = cluster.map_shared_rank(&s_slot[par][rank], lane);
                *dst = v;
            }
        }
        cluster.sync();                                  // release our DSMEM stores / acquire the peers'
        FpsSlot w = s_slot[par][0];
#pragma unroll
        for (int r = 1; r < CS; ++r) {
            const FpsSlot c = s_slot[par][r];
            if (c.key > w.key) w = c;
        }
        cur = 0xFFFFFFFFu - (unsigned)(w.key & 0xFFFFFFFFull);
        cx = w.x; cy = w.y; cz = w.z;
    }
    cg::this_cluster().sync();                           // no CTA may exit while peers can still write its smem
}

// ---- pruned variant (one CTA per cloud, N <= 8192) --------------------------------------------------------------------
// The scan above touches every point in every iteration, and at one cloud per SM that IS the cost: 2.1 G distance
// updates per 64 clouds, ~72 % of the SM's issue slots.  But an update only changes dist[i] when the new centre is
// closer to point i than every earlier sample, which after a few hundred samples is true for a few percent of the
// cloud.  So the points are first sorted along a Morton curve (one bitonic sort in shared memory per cloud), which
// makes every group of 32 consecutive points — one register "row" of a warp: the i-th point of each lane — a
// compact bucket with a bounding box and a cached (max distance, lowest index holding it).  Per iteration lane i of
// a warp tests row i: it evaluates the distance rule on the gap vector from the centre to the row's box,
//     g = max(fl(lo - c), fl(c - hi), 0) per axis,   d_box = ((gx*gx + gy*gy) + gz*gz)   (same non-fused fp32 ops);
// fp32 subtraction, multiplication and addition are monotone, so d_box <= the rule's distance of EVERY point in the
// box, and d_box >= the row's cached max proves that no dist[] of the row changes: the row is skipped, its cache
// stays valid.  Rows that fail the test are updated exactly as in the full scan and their cache is recomputed with
// two redux.  The running distances are therefore bit-identical to the full scan's at every iteration, and with the
// (max distance, lowest original index) argmax so is every output index (tests: vs the oracle).  The box test is
// fps_common.cuh::fps_box_dist, shared with the cluster scan of fps_large.cu.

__device__ __forceinline__ unsigned fps_spread5(unsigned v) {         // 5 bits -> every third bit
    return (v & 1u) | ((v & 2u) << 2) | ((v & 4u) << 4) | ((v & 8u) << 6) | ((v & 16u) << 8);
}

// SM = true: the sorted coordinates live in SHARED memory instead of registers (only the running distances stay in
// registers), so the kernel fits 64 registers and 112 KB and TWO clouds share an SM: an iteration is a latency chain that
// leaves the SM mostly idle, and with more clouds than SMs (batch > 74 on a B200) the second wave costs nothing extra.
// Visited rows (a few per iteration after pruning) read their coordinates with three conflict-free LDS.  Same arithmetic,
// same results.
template <int PPT, int FP_T, bool SM>
__global__ void __launch_bounds__(FP_T, SM ? 2 : 1)
fps_pruned_kernel(const float* __restrict__ xyz, int64_t* __restrict__ out, int N, int S) {
    constexpr int NP = PPT * FP_T, NW = FP_T / 32, RS = NW * 32;     // RS: slots between consecutive rows of a thread
    static_assert(PPT % 4 == 0 && PPT <= 32 && NP <= 8192, "rows are tested by lanes and visited in groups of four");
    __shared__ unsigned s_key_static[SM ? 1 : NP];       // sort keys, then the original index of every sorted slot
    extern __shared__ __align__(16) unsigned char fps_dyn[];          // SM: [keys -> x | y | z | idx16]
    unsigned* s_key = SM ? reinterpret_cast<unsigned*>(fps_dyn) : s_key_static;
    float* s_x = reinterpret_cast<float*>(fps_dyn);      // aliases the keys: written after every key has been read
    float* s_y = s_x + NP;
    float* s_z = s_y + NP;
    unsigned short* s_i16 = reinterpret_cast<unsigned short*>(s_z + NP);
    __shared__ float s_red[6][NW];
    __shared__ unsigned s_d[2][NW], s_i[2][NW];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* P = xyz + (size_t)blockIdx.x * N * 3;

    // bounding box of the cloud (NaNs dropped by fminf/fmaxf)
    float mn[3] = {3.0e38f, 3.0e38f, 3.0e38f}, mx[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
    for (int i = tid; i < N; i += FP_T)
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const float v = __ldg(P + (size_t)i * 3 + d);
            mn[d] = fminf(mn[d], v);
            mx[d] = fmaxf(mx[d], v);
        }
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        mn[d] = fps_unorder(__reduce_min_sync(FULL, fps_orderable(mn[d])));
        mx[d] = fps_unorder(__reduce_max_sync(FULL, fps_orderable(mx[d])));
        if (lane == 0) { s_red[d][warp] = mn[d]; s_red[3 + d][warp] = mx[d]; }
    }
    __syncthreads();
    float ext = 0.0f;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
#pragma unroll
        for (int w = 0; w < NW; ++w) { mn[d] = fminf(mn[d], s_red[d][w]); mx[d] = fmaxf(mx[d], s_red[3 + d][w]); }
        ext = fmaxf(ext, mx[d] - mn[d]);
    }
    const float scale = (ext > 0.0f && ext < 3.0e38f) ? 31.99f / ext : 0.0f;     // cubic cells: 32 per longest axis
    // Morton keys (any grouping is correct; this one makes the rows compact)
    for (int i = tid; i < NP; i += FP_T) {
        unsigned key = 0xFFFFFFFFu;                      // padding sorts to the end
        if (i < N) {
            unsigned code = 0;
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                const int c = (int)((__ldg(P + (size_t)i * 3 + d) - mn[d]) * scale);   // NaN -> 0
                code |= fps_spread5((unsigned)min(max(c, 0), 31)) << d;
            }
            key = (code << 13) | (unsigned)i;
        }
        s_key[i] = key;
    }
    __syncthreads();
    for (int k = 2; k <= NP; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < NP / 2; t += FP_T) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), l = i | j;
                const unsigned a = s_key[i], b = s_key[l];
                if ((a > b) == ((i & k) == 0)) { s_key[i] = b; s_key[l] = a; }
            }
            __syncthreads();
        }

    // registers: row i of this thread = sorted slot (i*NW + warp)*32 + lane, i.e. bucket i*NW + warp — neighbouring
    // buckets (the ones a new centre activates together) belong to different warps, so the visits spread over the CTA
    float px[SM ? 1 : PPT], py[SM ? 1 : PPT], pz[SM ? 1 : PPT], dist[PPT];
    const int base = warp * 32 + lane;
    unsigned* my_idx = s_key + base;                     // my_idx[i*RS]: original index of row i's point (0xFFFFFFFF: none)
    float lox = 0.f, loy = 0.f, loz = 0.f, hix = 0.f, hiy = 0.f, hiz = 0.f, rmax_d = 0.0f;
    unsigned rmax_i = 0xFFFFFFFFu;
    bool rstale = false;                                 // rmax_i is recomputed lazily, only for a row that holds the warp's max
#pragma unroll
    for (int i = 0; i < PPT; ++i) {
        const unsigned key = my_idx[i * RS];
        const bool ok = key != 0xFFFFFFFFu;
        const unsigned oi = ok ? (key & 8191u) : 0xFFFFFFFFu;
        const float x = ok ? __ldg(P + (size_t)oi * 3 + 0) : 0.0f;
        const float y = ok ? __ldg(P + (size_t)oi * 3 + 1) : 0.0f;
        const float z = ok ? __ldg(P + (size_t)oi * 3 + 2) : 0.0f;
        if (SM) { s_y[i * RS + base] = y; s_z[i * RS + base] = z; s_i16[i * RS + base] = (unsigned short)(ok ? oi : 0xFFFFu); }
        else { px[i] = x; py[i] = y; pz[i] = z; }
        dist[i] = ok ? 1e10f : 0.0f;
        // row box over the lanes that hold a point; an empty row gets (+big, -big): its gap is huge, it is never visited
        const float bx0 = fps_unorder(__reduce_min_sync(FULL, fps_orderable(ok ? x : 3.0e38f)));
        const float by0 = fps_unorder(__reduce_min_sync(FULL, fps_orderable(ok ? y : 3.0e38f)));
        const float bz0 = fps_unorder(__reduce_min_sync(FULL, fps_orderable(ok ? z : 3.0e38f)));
        const float bx1 = fps_unorder(__reduce_max_sync(FULL, fps_orderable(ok ? x : -3.0e38f)));
        const float by1 = fps_unorder(__reduce_max_sync(FULL, fps_orderable(ok ? y : -3.0e38f)));
        const float bz1 = fps_unorder(__reduce_max_sync(FULL, fps_orderable(ok ? z : -3.0e38f)));
        const unsigned any = __reduce_min_sync(FULL, oi);
        if (lane == i) {
            lox = bx0; loy = by0; loz = bz0; hix = bx1; hiy = by1; hiz = bz1;
            rmax_d = any != 0xFFFFFFFFu ? 1e10f : 0.0f;
            rmax_i = any;
        }
    }
    __syncthreads();                                     // every key has been read before the slots are rewritten
    if (SM) {
#pragma unroll
        for (int i = 0; i < PPT; ++i) {                  // x goes where the keys were
            const unsigned oi = s_i16[i * RS + base];
            s_x[i * RS + base] = oi != 0xFFFFu ? __ldg(P + (size_t)oi * 3 + 0) : 0.0f;
        }
    } else {
#pragma unroll
        for (int i = 0; i < PPT; ++i) {
            const unsigned key = my_idx[i * RS];
            my_idx[i * RS] = key != 0xFFFFFFFFu ? (key & 8191u) : 0xFFFFFFFFu;
        }
    }
    __syncwarp();                                        // a thread only ever reads its own slots again

    unsigned cur = 0;
    float cx = __ldg(P + 0), cy = __ldg(P + 1), cz = __ldg(P + 2);
    int64_t* o = out + (size_t)blockIdx.x * S;
    for (int s = 0; s < S; ++s) {
        if (tid == 0) o[s] = (int64_t)cur;
        if (s == S - 1) break;

        // which rows can change?  lane i answers for row i
        const float dbox = fps_box_dist(lox, loy, loz, hix, hiy, hiz, cx, cy, cz);
        const unsigned mask = __ballot_sync(FULL, lane < PPT && fps_box_may_change(dbox, rmax_d));
#pragma unroll
        for (int g4 = 0; g4 < PPT; g4 += 4) {
            if (((mask >> g4) & 0xFu) == 0u) continue;   // warp-uniform
#pragma unroll
            for (int i = g4; i < g4 + 4; ++i) {
                if (!((mask >> i) & 1u)) continue;       // warp-uniform
                const float d = SM ? sqdist3_rule(s_x[i * RS + base], s_y[i * RS + base], s_z[i * RS + base], cx, cy, cz)
                                   : sqdist3_rule(px[SM ? 0 : i], py[SM ? 0 : i], pz[SM ? 0 : i], cx, cy, cz);
                dist[i] = fminf(dist[i], d);
                const unsigned m = __reduce_max_sync(FULL, __float_as_uint(dist[i]));   // >= +0: bit order = value order
                if (lane == i) { rmax_d = __uint_as_float(m); rstale = true; }
            }
        }
        const unsigned vd = lane < PPT ? __float_as_uint(rmax_d) : 0u;
        const unsigned wmax = __reduce_max_sync(FULL, vd);
        const unsigned need = __ballot_sync(FULL, lane < PPT && vd == wmax && rstale);
        if (need) {                                      // usually one row: lowest original index among its maxima
#pragma unroll
            for (int g4 = 0; g4 < PPT; g4 += 4) {
                if (((need >> g4) & 0xFu) == 0u) continue;
#pragma unroll
                for (int i = g4; i < g4 + 4; ++i) {
                    if (!((need >> i) & 1u)) continue;
                    const unsigned mine = SM ? (s_i16[i * RS + base] == 0xFFFFu ? 0xFFFFFFFFu : (unsigned)s_i16[i * RS + base]) : my_idx[SM ? 0 : i * RS];
                    const unsigned mi = __reduce_min_sync(FULL, __float_as_uint(dist[i]) == wmax ? mine : 0xFFFFFFFFu);
                    if (lane == i) { rmax_i = mi; rstale = false; }
                }
            }
        }
        const unsigned widx = __reduce_min_sync(FULL, (lane < PPT && vd == wmax) ? rmax_i : 0xFFFFFFFFu);
        const int par = s & 1;
        if (lane == 0) { s_d[par][warp] = wmax; s_i[par][warp] = widx; }
        __syncthreads();
        const unsigned qd = lane < NW ? s_d[par][lane] : 0u;
        const unsigned qi = lane < NW ? s_i[par][lane] : 0xFFFFFFFFu;
        const unsigned gmax = __reduce_max_sync(FULL, qd);
        cur = __reduce_min_sync(FULL, qd == gmax ? qi : 0xFFFFFFFFu);
        cx = __ldg(P + (size_t)cur * 3 + 0);
        cy = __ldg(P + (size_t)cur * 3 + 1);
        cz = __ldg(P + (size_t)cur * 3 + 2);
    }
}

template <int PPT, int FP_T, bool SM = false>
static cudaError_t launch_fps_pruned(const float* xyz, int64_t* idx, int B, int N, int S, cudaStream_t st) {
    size_t smem = 0;
    if (SM) {
        smem = (size_t)PPT * FP_T * (3 * sizeof(float) + sizeof(unsigned short));
        cudaError_t e = cudaFuncSetAttribute(fps_pruned_kernel<PPT, FP_T, SM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(fps_pruned_kernel<PPT, FP_T, SM>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
    }
    fps_pruned_kernel<PPT, FP_T, SM><<<B, FP_T, smem, st>>>(xyz, idx, N, S);
    return cudaGetLastError();
}

static cudaError_t dispatch_pruned(const float* xyz, int64_t* idx, int B, int N, int S, cudaStream_t st) {
    if (N <= 1024) return launch_fps_pruned<4, 256>(xyz, idx, B, N, S, st);
    if (N <= 2048) return launch_fps_pruned<4, 512>(xyz, idx, B, N, S, st);
    if (N <= 4096) return launch_fps_pruned<8, 512>(xyz, idx, B, N, S, st);
    // more clouds than SMs: two clouds per SM (coordinates in shared memory) instead of a second wave
    if (B > sm_count()) return launch_fps_pruned<16, 512, true>(xyz, idx, B, N, S, st);
    return launch_fps_pruned<16, 512>(xyz, idx, B, N, S, st);
}

template <int CS>
static cudaError_t launch_fps(const float* xyz, int64_t* idx, int B, int N, int S, cudaStream_t st) {
    auto kern = fps_kernel<CS>;
    const size_t smem = (size_t)FPS_PPT * FPS_T * 3 * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(B * CS);
    cfg.blockDim = dim3(FPS_T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, xyz, idx, N, S, -0.0f);
}

}  // namespace b200

// Largest cloud b200_fps takes (the 8-CTA cluster holds 8 x 8192 points in registers); above it b200_fps returns
// B200_ENOSUP and the host layer calls b200_fps_large.  A variant build may lower it to 8192 to time the pruned cluster
// scan against fps_kernel<CS> on the same clouds (profiles/build_variant.sh; DESIGN §4).
#ifndef B200_FPS_CLUSTER_MAX_N
#define B200_FPS_CLUSTER_MAX_N 65536
#endif
static_assert(B200_FPS_CLUSTER_MAX_N >= 8192 && B200_FPS_CLUSTER_MAX_N <= 65536, "b200_fps: 8192 <= cluster limit <= 65536");

extern "C" int b200_fps(const float* xyz, int64_t* idx, int B, int N, int n_samples, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0) || (xyz && idx), "b200_fps: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && n_samples >= 1, "b200_fps: bad sizes B=%d n_samples=%d", B, n_samples);
    B200_REQUIRE(N > n_samples, "b200_fps: need N > n_samples (N=%d, n_samples=%d) as models/csrc/wrapper.py:98", N, n_samples);
    if (N > B200_FPS_CLUSTER_MAX_N) {
        set_error("b200_fps: N=%d exceeds %d points per cloud (8-CTA cluster x 8192); b200_fps_large takes any N",
                  N, B200_FPS_CLUSTER_MAX_N);
        return B200_ENOSUP;
    }
    if (B == 0) return B200_OK;
    cudaStream_t st = as_stream(stream);
    // one CTA per cloud up to 8192 points; above, the smallest cluster whose CTAs hold the cloud in registers
    cudaError_t e;
    if (N <= 8192) e = dispatch_pruned(xyz, idx, B, N, n_samples, st);
    else if (N <= 16384) e = launch_fps<2>(xyz, idx, B, N, n_samples, st);
    else if (N <= 32768) e = launch_fps<4>(xyz, idx, B, N, n_samples, st);
    else e = launch_fps<8>(xyz, idx, B, N, n_samples, st);
    if (e != cudaSuccess) return cuda_fail(e, "b200_fps");
    return B200_OK;
}
