// fps_large.cu — a3 for clouds of any size: furthest point sampling as a pruned scan over one thread-block cluster per
// cloud, with caller scratch.  Serves b200_fps_large (every N > n_samples); the library's own routing sends clouds of
// more than 65536 points here (ops._furthest_point_sampling_cuda), where b200_fps, whose cluster holds the cloud in
// registers, stops.
//
// Replaces models/csrc/furthest_point_sampling/furthest_point_sampling_kernel.cu:34-85 for those clouds: the reference's
// one 1024-thread CTA keeps its running distances in the global `dists_temp` and scans all N of them per iteration.
//
// Prep (many CTAs per cloud, 4 launches + 1 memset):
//   fps_large_bbox_kernel     bounding box with order-independent atomic min/max on the monotone uint image of each bound
//   fps_large_hist_kernel     Morton bucket of every point (b bits per axis, 2^(3b) >= N/8 buckets) -> counts
//   fps_large_scan_kernel     exclusive scan of the counts (one CTA per cloud)
//   fps_large_scatter_kernel  atomic cursor per bucket -> sorted SoA x | y | z | original index
// knn_grid's cell order is not reused: its cells hold ~k/2 points in raster order, so 32 consecutive sorted points are
// strips across the cloud, not compact rows.
//
// Why the sort cannot change a pick.  The order of the points inside a bucket depends on the order in which the scatter
// kernel's atomics land and may differ from run to run.  The layout only decides which points share a row (and so which
// rows the box test can skip); the running distances are updated with the same rule for every point a skip does not
// prove unchanged, and the argmax is taken over (distance, LOWEST ORIGINAL INDEX), so the picks are those of the full
// scan for any layout.
//
// Iteration (fps_large_kernel, a cluster of FPSL_CS = 8 CTAs of 512 threads per cloud).  The sorted slots are cut into
// rows of 32 points and groups of 32 rows; CTA r of the cluster owns a contiguous range of `gpc` groups.  Rows and
// groups each keep a bounding box and a cached (max running distance, lowest original index holding it).  Per
// iteration:
//   A  each thread tests its groups with fps_box_dist (fps_common.cuh, the test of fps.cu's pruned kernel one level
//      up) and appends the ones that may change to a shared list;
//   B  a warp per listed group: lane i tests row i; for every row that may change, the 32 lanes update the row's 32
//      running distances (sqdist3_rule, fminf), and two redux give the row's new (max, lowest index); the row cache
//      and then the group cache are rewritten;
//   C  the CTA winner is the (max, lowest index) over its group caches (redux per warp, one __syncthreads, redux);
//      lanes 0..CS-1 of warp 0 write {key, x, y, z} into every peer's slot (DSMEM); one cluster.sync; every thread
//      reduces the CS slots to the next centre.
// A group whose box passes the test proves all its rows unchanged (its box contains theirs and its cached max is their
// maximum), so the work of an iteration scales with the rows a centre can reach, plus one test per group (N/8192
// per thread of the cluster), not with N.
//
// Where the data lives.  Group caches, the active list, row caches and the points (x, y, z, running distance, index:
// 20 B per slot) are kept in the CTA's shared memory when its share fits (21.5 KB per group: clouds of up to 81920
// points); otherwise the points and row caches stay in the L2-resident scratch and only the group caches and the list
// are in shared memory (36 B per group: clouds of up to ~52 M points); beyond that they move to scratch too.  The kernel reaches all of them through
// generic pointers, so there is one kernel and one arithmetic.
//
// Safety: synchronisation only inside a cluster (clusters of different clouds may run in waves); the kernel ends with a
// cluster barrier, so no CTA exits while a peer can still write its shared memory; all offsets are size_t.  Non-finite
// coordinates finish and give indices in [0, N): they never enter a box, NaN distances never lower a running
// distance, and padding slots (distance 0, index 0xFFFFFFFF) lose every tie to a real point.
//
// ptxas (sm_100a, -O3): fps_large_kernel 84 registers, 656 B static shared memory + fpsl_smem_bytes(gpc, level) dynamic
// (215 KB at gpc = 10, level 2); prep kernels 26-32 registers; no stack, no spills.
#include <cooperative_groups.h>

#include <algorithm>

#include "fps_common.cuh"

namespace cg = cooperative_groups;

namespace b200 {

constexpr int FPSL_CS = 8;                   // portable cluster size
constexpr int FPSL_T = 512, FPSL_NW = FPSL_T / 32;
constexpr int FPSL_GP = 1024;                // points per group (32 rows of 32)
constexpr int FPSL_PREP_T = 256;

struct __align__(16) FpsBox {                // row or group cache: 32 bytes
    float lox, loy, loz, dmax;               // dmax: the largest running distance of the box's points
    float hix, hiy, hiz;
    unsigned imax;                           // lowest original index holding dmax (0xFFFFFFFF: no point)
};

struct FpsLargeSlot {                        // what a CTA publishes to its cluster peers each iteration
    unsigned long long key;                  // (distance bits << 32) | (0xFFFFFFFF - index)
    float x, y, z, pad;
};

// ---- scratch layout (per cloud, every array 256-byte aligned) ----------------------------------------------------------
struct FpsLargeLayout {
    int bits, gpc;                           // Morton bits per axis; groups per CTA
    size_t slots, buckets;                   // padded slots per cloud (gpc * CS * 1024); 2^(3*bits)
    size_t off_x, off_y, off_z, off_d, off_i, off_rows, off_groups, off_act, cloud_bytes;   // within a cloud's block
    size_t off_hist, off_bbox, total;        // counts + boxes of all clouds (zeroed by one memset) after the B blocks
};

static inline size_t al256(size_t v) { return (v + 255) & ~(size_t)255; }

static FpsLargeLayout fps_large_layout(int B, int N) {
    FpsLargeLayout L{};
    int b = 1;
    while (b < 7 && ((size_t)1 << (3 * b)) * 8 < (size_t)N) ++b;              // >= N/8 buckets: ~8 points per bucket
    L.bits = b;
    L.buckets = (size_t)1 << (3 * b);
    const size_t groups = ((size_t)N + FPSL_GP - 1) / FPSL_GP;
    L.gpc = (int)((groups + FPSL_CS - 1) / FPSL_CS);
    L.slots = (size_t)L.gpc * FPSL_CS * FPSL_GP;
    size_t o = 0;
    L.off_x = o; o += al256(L.slots * 4);
    L.off_y = o; o += al256(L.slots * 4);
    L.off_z = o; o += al256(L.slots * 4);
    L.off_d = o; o += al256(L.slots * 4);
    L.off_i = o; o += al256(L.slots * 4);
    L.off_rows = o; o += al256(L.slots / 32 * sizeof(FpsBox));
    L.off_groups = o; o += al256(L.slots / FPSL_GP * sizeof(FpsBox));
    L.off_act = o; o += al256(L.slots / FPSL_GP * sizeof(unsigned));
    L.cloud_bytes = o;
    L.off_hist = (size_t)B * o;
    L.off_bbox = L.off_hist + al256((size_t)B * L.buckets * 4);
    L.total = L.off_bbox + al256((size_t)B * 6 * 4);
    return L;
}

// ---- prep -------------------------------------------------------------------------------------------------------------
// bbox[cloud*6 + d] = max over points of ~orderable(x_d) (i.e. the min), bbox[cloud*6 + 3 + d] = max of orderable(x_d);
// both start at 0 (the memset), so the result does not depend on the order the atomics land in.
__global__ void __launch_bounds__(FPSL_PREP_T)
fps_large_bbox_kernel(const float* __restrict__ xyz, unsigned* __restrict__ bbox, int N) {
    const float* P = xyz + (size_t)blockIdx.y * N * 3;
    float mn[3] = {3.0e38f, 3.0e38f, 3.0e38f}, mx[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
    for (size_t i = (size_t)blockIdx.x * FPSL_PREP_T + threadIdx.x; i < (size_t)N; i += (size_t)gridDim.x * FPSL_PREP_T)
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const float v = __ldg(P + i * 3 + d);                               // fminf/fmaxf drop NaNs
            mn[d] = fminf(mn[d], v);
            mx[d] = fmaxf(mx[d], v);
        }
    unsigned* bb = bbox + (size_t)blockIdx.y * 6;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const unsigned lo = __reduce_max_sync(FULL, ~fps_orderable(mn[d]));
        const unsigned hi = __reduce_max_sync(FULL, fps_orderable(mx[d]));
        if ((threadIdx.x & 31) == 0) { atomicMax(bb + d, lo); atomicMax(bb + 3 + d, hi); }
    }
}

__device__ __forceinline__ unsigned fps_spread7(unsigned v) {          // 7 bits -> every third bit
    unsigned r = 0;
#pragma unroll
    for (int k = 0; k < 7; ++k) r |= ((v >> k) & 1u) << (3 * k);
    return r;
}

__device__ __forceinline__ unsigned fps_large_bucket(const float* p, const unsigned* bb, int bits) {
    float mn[3], ext = 0.0f;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        mn[d] = fps_unorder(~bb[d]);
        ext = fmaxf(ext, fps_unorder(bb[3 + d]) - mn[d]);
    }
    const int cells = 1 << bits;
    const float scale = (ext > 0.0f && ext < 3.0e38f) ? ((float)cells - 0.01f) / ext : 0.0f;   // cubic cells
    unsigned code = 0;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const int c = (int)__fmul_rn(__fsub_rn(p[d], mn[d]), scale);           // NaN -> 0; same bucket in both passes
        code |= fps_spread7((unsigned)min(max(c, 0), cells - 1)) << d;
    }
    return code;
}

__global__ void __launch_bounds__(FPSL_PREP_T)
fps_large_hist_kernel(const float* __restrict__ xyz, unsigned* __restrict__ hist, const unsigned* __restrict__ bbox,
                      int N, int bits) {
    const float* P = xyz + (size_t)blockIdx.y * N * 3;
    unsigned* H = hist + (size_t)blockIdx.y * ((size_t)1 << (3 * bits));
    const unsigned* bb = bbox + (size_t)blockIdx.y * 6;
    for (size_t i = (size_t)blockIdx.x * FPSL_PREP_T + threadIdx.x; i < (size_t)N; i += (size_t)gridDim.x * FPSL_PREP_T) {
        const float p[3] = {__ldg(P + i * 3 + 0), __ldg(P + i * 3 + 1), __ldg(P + i * 3 + 2)};
        atomicAdd(H + fps_large_bucket(p, bb, bits), 1u);
    }
}

// Exclusive scan of one cloud's counts, in place: thread t owns a contiguous chunk of buckets / 1024 counts.
__global__ void __launch_bounds__(1024)
fps_large_scan_kernel(unsigned* __restrict__ hist, int bits) {
    __shared__ unsigned s_w[32];
    const size_t nb = (size_t)1 << (3 * bits);
    unsigned* H = hist + (size_t)blockIdx.x * nb;
    const size_t per = (nb + 1023) / 1024, lo = min(nb, threadIdx.x * per), hi = min(nb, lo + per);
    unsigned sum = 0;
    for (size_t i = lo; i < hi; ++i) sum += H[i];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned v = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned w = s_w[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(FULL, wi, o);
            if (lane >= o) wi += v;
        }
        s_w[lane] = wi - w;
    }
    __syncthreads();
    unsigned run = s_w[warp] + incl - sum;
    for (size_t i = lo; i < hi; ++i) { const unsigned c = H[i]; H[i] = run; run += c; }
}

__global__ void __launch_bounds__(FPSL_PREP_T)
fps_large_scatter_kernel(const float* __restrict__ xyz, unsigned char* __restrict__ scratch, FpsLargeLayout L, int N) {
    const float* P = xyz + (size_t)blockIdx.y * N * 3;
    unsigned* H = reinterpret_cast<unsigned*>(scratch + L.off_hist) + (size_t)blockIdx.y * L.buckets;
    const unsigned* bb = reinterpret_cast<const unsigned*>(scratch + L.off_bbox) + (size_t)blockIdx.y * 6;
    unsigned char* C = scratch + (size_t)blockIdx.y * L.cloud_bytes;
    float* sx = reinterpret_cast<float*>(C + L.off_x);
    float* sy = reinterpret_cast<float*>(C + L.off_y);
    float* sz = reinterpret_cast<float*>(C + L.off_z);
    unsigned* si = reinterpret_cast<unsigned*>(C + L.off_i);
    for (size_t i = (size_t)blockIdx.x * FPSL_PREP_T + threadIdx.x; i < (size_t)N; i += (size_t)gridDim.x * FPSL_PREP_T) {
        const float p[3] = {__ldg(P + i * 3 + 0), __ldg(P + i * 3 + 1), __ldg(P + i * 3 + 2)};
        const unsigned pos = atomicAdd(H + fps_large_bucket(p, bb, L.bits), 1u);   // real points fill slots [0, N)
        sx[pos] = p[0]; sy[pos] = p[1]; sz[pos] = p[2]; si[pos] = (unsigned)i;
    }
}

// ---- iteration --------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long fps_key(float d, unsigned i) {
    return ((unsigned long long)__float_as_uint(d) << 32) | (unsigned long long)(0xFFFFFFFFu - i);
}

// smem_level: 2 = groups, rows, points and list in shared memory; 1 = groups and list; 0 = nothing (all in scratch).
__host__ __device__ constexpr size_t fpsl_smem_bytes(int gpc, int level) {
    return level == 0 ? 0
         : (size_t)gpc * (sizeof(FpsBox) + sizeof(unsigned)) +
               (level == 2 ? (size_t)gpc * 32 * sizeof(FpsBox) + (size_t)gpc * FPSL_GP * 5 * 4 : 0);
}

__global__ void __launch_bounds__(FPSL_T, 1)
fps_large_kernel(const float* __restrict__ xyz, int64_t* __restrict__ out, unsigned char* __restrict__ scratch,
                 FpsLargeLayout L, int N, int S, int smem_level) {
    constexpr int T = FPSL_T, NW = FPSL_NW, CS = FPSL_CS;
    __shared__ unsigned s_d[2][NW], s_i[2][NW];
    __shared__ __align__(16) FpsLargeSlot s_slot[2][CS];
    __shared__ int s_nact;
    extern __shared__ __align__(16) unsigned char fpsl_dyn[];

    cg::cluster_group cluster = cg::this_cluster();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rank = (int)cluster.block_rank(), cloud = blockIdx.x / CS;
    const int gpc = L.gpc, rpc = gpc * 32, npc = gpc * FPSL_GP;                // groups, rows, slots of this CTA
    const size_t base = (size_t)rank * npc;                                    // first slot of this CTA in the cloud
    const float* P = xyz + (size_t)cloud * N * 3;
    unsigned char* C = scratch + (size_t)cloud * L.cloud_bytes;

    // this CTA's slice of every array, in scratch or in shared memory
    float* px = reinterpret_cast<float*>(C + L.off_x) + base;
    float* py = reinterpret_cast<float*>(C + L.off_y) + base;
    float* pz = reinterpret_cast<float*>(C + L.off_z) + base;
    float* pd = reinterpret_cast<float*>(C + L.off_d) + base;
    unsigned* pi = reinterpret_cast<unsigned*>(C + L.off_i) + base;
    FpsBox* rows = reinterpret_cast<FpsBox*>(C + L.off_rows) + (size_t)rank * rpc;
    FpsBox* grp = reinterpret_cast<FpsBox*>(C + L.off_groups) + (size_t)rank * gpc;
    unsigned* act = reinterpret_cast<unsigned*>(C + L.off_act) + (size_t)rank * gpc;
    if (smem_level >= 1) {                                                     // layout: fpsl_smem_bytes
        unsigned char* q = fpsl_dyn;
        grp = reinterpret_cast<FpsBox*>(q); q += (size_t)gpc * sizeof(FpsBox);
        if (smem_level == 2) {
            rows = reinterpret_cast<FpsBox*>(q); q += (size_t)rpc * sizeof(FpsBox);
            float* sx = reinterpret_cast<float*>(q); q += (size_t)npc * 4;
            float* sy = reinterpret_cast<float*>(q); q += (size_t)npc * 4;
            float* sz = reinterpret_cast<float*>(q); q += (size_t)npc * 4;
            float* sd = reinterpret_cast<float*>(q); q += (size_t)npc * 4;
            unsigned* sidx = reinterpret_cast<unsigned*>(q); q += (size_t)npc * 4;
            for (int j = tid; j < npc; j += T) {
                const bool ok = base + j < (size_t)N;
                sx[j] = ok ? px[j] : 0.0f; sy[j] = ok ? py[j] : 0.0f; sz[j] = ok ? pz[j] : 0.0f;
                sidx[j] = ok ? pi[j] : 0xFFFFFFFFu;
            }
            px = sx; py = sy; pz = sz; pd = sd; pi = sidx;
            __syncthreads();
        }
        act = reinterpret_cast<unsigned*>(q);
    }

    // initial state: running distances 1e10 (padding 0), row boxes and caches, then group boxes and caches
    for (int r = warp; r < rpc; r += NW) {
        const int j = r * 32 + lane;
        const bool ok = base + j < (size_t)N;
        const float x = ok ? px[j] : 0.0f, y = ok ? py[j] : 0.0f, z = ok ? pz[j] : 0.0f;
        const unsigned oi = ok ? pi[j] : 0xFFFFFFFFu;
        pd[j] = ok ? 1e10f : 0.0f;
        if (!ok) { px[j] = 0.0f; py[j] = 0.0f; pz[j] = 0.0f; pi[j] = 0xFFFFFFFFu; }   // scratch padding holds old bytes
        FpsBox b;
        b.lox = fps_unorder(__reduce_min_sync(FULL, fps_orderable(ok ? x : 3.0e38f)));
        b.loy = fps_unorder(__reduce_min_sync(FULL, fps_orderable(ok ? y : 3.0e38f)));
        b.loz = fps_unorder(__reduce_min_sync(FULL, fps_orderable(ok ? z : 3.0e38f)));
        b.hix = fps_unorder(__reduce_max_sync(FULL, fps_orderable(ok ? x : -3.0e38f)));
        b.hiy = fps_unorder(__reduce_max_sync(FULL, fps_orderable(ok ? y : -3.0e38f)));
        b.hiz = fps_unorder(__reduce_max_sync(FULL, fps_orderable(ok ? z : -3.0e38f)));
        b.imax = __reduce_min_sync(FULL, oi);
        b.dmax = b.imax != 0xFFFFFFFFu ? 1e10f : 0.0f;
        if (lane == 0) rows[r] = b;                                            // an empty row: (+big, -big), never visited
    }
    __syncthreads();
    for (int g = tid; g < gpc; g += T) {
        FpsBox b = rows[g * 32];
        for (int i = 1; i < 32; ++i) {
            const FpsBox r = rows[g * 32 + i];
            b.lox = fminf(b.lox, r.lox); b.loy = fminf(b.loy, r.loy); b.loz = fminf(b.loz, r.loz);
            b.hix = fmaxf(b.hix, r.hix); b.hiy = fmaxf(b.hiy, r.hiy); b.hiz = fmaxf(b.hiz, r.hiz);
            if (fps_key(r.dmax, r.imax) > fps_key(b.dmax, b.imax)) { b.dmax = r.dmax; b.imax = r.imax; }
        }
        grp[g] = b;
    }
    if (tid == 0) s_nact = 0;
    cluster.sync();                                                            // peers are running before any DSMEM store

    unsigned cur = 0;
    float cx = __ldg(P + 0), cy = __ldg(P + 1), cz = __ldg(P + 2);
    int64_t* o = out + (size_t)cloud * S;
    for (int s = 0; s < S; ++s) {
        if (rank == 0 && tid == 0) o[s] = (int64_t)cur;
        if (s == S - 1) break;

        // A: groups the centre may reach -> act[]
        for (int g0 = 0; g0 < gpc; g0 += T) {
            const int g = g0 + tid;
            bool may = false;
            if (g < gpc) {
                const FpsBox b = grp[g];
                may = fps_box_may_change(fps_box_dist(b.lox, b.loy, b.loz, b.hix, b.hiy, b.hiz, cx, cy, cz), b.dmax);
            }
            const unsigned m = __ballot_sync(FULL, may);
            int at = 0;
            if (lane == 0 && m) at = atomicAdd(&s_nact, __popc(m));
            at = __shfl_sync(FULL, at, 0);
            if (may) act[at + __popc(m & ((1u << lane) - 1u))] = (unsigned)g;
        }
        __syncthreads();
        const int nact = s_nact;

        // B: a warp per listed group; lane i holds row i's cache
        for (int a = warp; a < nact; a += NW) {
            const int g = (int)act[a], r = g * 32 + lane;
            FpsBox rb = rows[r];
            const float dbox = fps_box_dist(rb.lox, rb.loy, rb.loz, rb.hix, rb.hiy, rb.hiz, cx, cy, cz);
            const unsigned vis = __ballot_sync(FULL, fps_box_may_change(dbox, rb.dmax));
            for (unsigned m = vis; m; m &= m - 1) {                                // warp-uniform
                const int i = __ffs(m) - 1;
                const int j = (g * 32 + i) * 32 + lane;
                const float old = pd[j];
                const float nd = fminf(old, sqdist3_rule(px[j], py[j], pz[j], cx, cy, cz));
                if (nd != old) pd[j] = nd;
                const unsigned mx = __reduce_max_sync(FULL, __float_as_uint(nd));   // >= +0: bit order = value order
                const unsigned mi = __reduce_min_sync(FULL, __float_as_uint(nd) == mx ? pi[j] : 0xFFFFFFFFu);
                if (lane == i) { rb.dmax = __uint_as_float(mx); rb.imax = mi; }
            }
            if ((vis >> lane) & 1u) { rows[r].dmax = rb.dmax; rows[r].imax = rb.imax; }
            const unsigned gm = __reduce_max_sync(FULL, __float_as_uint(rb.dmax));
            const unsigned gi = __reduce_min_sync(FULL, __float_as_uint(rb.dmax) == gm ? rb.imax : 0xFFFFFFFFu);
            if (lane == 0) { grp[g].dmax = __uint_as_float(gm); grp[g].imax = gi; }
        }
        __syncthreads();

        // C: CTA winner over the group caches, then the cluster exchange
        unsigned long long best = 0;
        for (int g = tid; g < gpc; g += T) {
            const FpsBox b = grp[g];
            const unsigned long long k = fps_key(b.dmax, b.imax);
            best = k > best ? k : best;
        }
        const unsigned bd = (unsigned)(best >> 32), bi = 0xFFFFFFFFu - (unsigned)best;
        const unsigned wmax = __reduce_max_sync(FULL, bd);
        const unsigned widx = __reduce_min_sync(FULL, bd == wmax ? bi : 0xFFFFFFFFu);
        const int par = s & 1;
        if (lane == 0) { s_d[par][warp] = wmax; s_i[par][warp] = widx; }
        if (tid == 0) s_nact = 0;                                              // every thread has read it (barrier above)
        __syncthreads();
        if (warp == 0) {
            const unsigned vd = lane < NW ? s_d[par][lane] : 0u;
            const unsigned vi = lane < NW ? s_i[par][lane] : 0xFFFFFFFFu;
            const unsigned gmax = __reduce_max_sync(FULL, vd);
            const unsigned gidx = __reduce_min_sync(FULL, vd == gmax ? vi : 0xFFFFFFFFu);
            if (lane < CS) {                                                   // lane r writes this CTA's winner into peer r
                const bool real = gidx < (unsigned)N;                          // a CTA of padding only has no winner
                FpsLargeSlot v;
                v.key = fps_key(__uint_as_float(gmax), gidx);
                v.x = real ? __ldg(P + (size_t)gidx * 3 + 0) : 0.0f;
                v.y = real ? __ldg(P + (size_t)gidx * 3 + 1) : 0.0f;
                v.z = real ? __ldg(P + (size_t)gidx * 3 + 2) : 0.0f;
                v.pad = 0.0f;
                *cluster.map_shared_rank(&s_slot[par][rank], lane) = v;
            }
        }
        cluster.sync();                                                        // release our DSMEM stores / acquire the peers'
        FpsLargeSlot w = s_slot[par][0];
#pragma unroll
        for (int r = 1; r < CS; ++r) {
            const FpsLargeSlot c = s_slot[par][r];
            if (c.key > w.key) w = c;
        }
        cur = 0xFFFFFFFFu - (unsigned)(w.key & 0xFFFFFFFFull);
        cx = w.x; cy = w.y; cz = w.z;
    }
    cluster.sync();                                                            // no CTA may exit while peers can still write its smem
}

static int fps_large_smem_budget() {                                             // opt-in shared memory per block
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
        return 0;
    return v - 2048;                                                            // the kernel's static shared memory
}

}  // namespace b200

extern "C" int64_t b200_fps_scratch_bytes(int B, int N) {
    if (B < 0 || N < 1) return -1;
    return (int64_t)b200::fps_large_layout(B, N).total;
}

extern "C" int b200_fps_large(const float* xyz, int64_t* idx, void* scratch, int64_t scratch_bytes, int B, int N,
                              int n_samples, b200_stream_t stream) {
    using namespace b200;
    B200_REQUIRE((B == 0) || (xyz && idx && scratch), "b200_fps_large: null pointer");   // empty calls carry null pointers
    B200_REQUIRE(B >= 0 && n_samples >= 1, "b200_fps_large: bad sizes B=%d n_samples=%d", B, n_samples);
    B200_REQUIRE(N > n_samples, "b200_fps_large: need N > n_samples (N=%d, n_samples=%d) as models/csrc/wrapper.py:98", N,
                 n_samples);
    if (B == 0) return B200_OK;
    const FpsLargeLayout L = fps_large_layout(B, N);
    B200_REQUIRE(scratch_bytes >= (int64_t)L.total, "b200_fps_large: scratch too small (%lld < %lld bytes)",
                 (long long)scratch_bytes, (long long)L.total);
    B200_REQUIRE(((uintptr_t)scratch & 255) == 0, "b200_fps_large: scratch must be 256-byte aligned");
    B200_REQUIRE(B <= 65535, "b200_fps_large: B=%d clouds exceed the prep grid (65535)", B);
    cudaStream_t st = as_stream(stream);
    unsigned char* sc = static_cast<unsigned char*>(scratch);
    unsigned* hist = reinterpret_cast<unsigned*>(sc + L.off_hist);
    unsigned* bbox = reinterpret_cast<unsigned*>(sc + L.off_bbox);

    B200_CUDA(cudaMemsetAsync(hist, 0, L.total - L.off_hist, st));            // counts and boxes of every cloud
    const int per_cloud = (int)std::min<int64_t>(((int64_t)N + FPSL_PREP_T * 8 - 1) / (FPSL_PREP_T * 8), 1024);
    const dim3 pg(per_cloud, B);
    fps_large_bbox_kernel<<<pg, FPSL_PREP_T, 0, st>>>(xyz, bbox, N);
    fps_large_hist_kernel<<<pg, FPSL_PREP_T, 0, st>>>(xyz, hist, bbox, N, L.bits);
    fps_large_scan_kernel<<<B, 1024, 0, st>>>(hist, L.bits);
    fps_large_scatter_kernel<<<pg, FPSL_PREP_T, 0, st>>>(xyz, sc, L, N);
    B200_LAUNCH_CHECK("b200_fps_large (prep)");

    const int budget = fps_large_smem_budget();
    const int level = fpsl_smem_bytes(L.gpc, 2) <= (size_t)budget ? 2 : fpsl_smem_bytes(L.gpc, 1) <= (size_t)budget ? 1 : 0;
    const size_t smem = fpsl_smem_bytes(L.gpc, level);
    cudaError_t e = cudaFuncSetAttribute(fps_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "b200_fps_large");
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)B * FPSL_CS);
    cfg.blockDim = dim3(FPSL_T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = FPSL_CS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, fps_large_kernel, xyz, idx, sc, L, N, n_samples, level);
    if (e != cudaSuccess) return cuda_fail(e, "b200_fps_large");
    return B200_OK;
}
