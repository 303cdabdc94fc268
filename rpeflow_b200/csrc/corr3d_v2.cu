// corr3d_v2.cu — a5 passes 2 and 3, second generation: warp-specialised tcgen05 pipelines in which EVERY per-(row, channel)
// contraction runs on the tensor cores, because ncu showed both first-generation kernels to be bound by instruction issue
// (1837 / 1316 thread-instructions per row at C = 32, tensor pipe < 5 % busy) — not by the MMAs, HBM or L2.
//
// Replaces models/pwc3d_core.py:91-101 (pass 2: cost_mlp layer 2, weight_net2, mul + sum over the neighbours) and
// :106-115 (pass 3: weight_net1, mul + sum over the self-neighbours).  What moved onto tcgen05.mma compared with
// corr3d_tc.cu / corr3d.cu:
//   * relu(bc + Wc.hid), the last weight-net layer (8 FMAs + 3 LDS per row and channel before): one K = 8 MMA group
//     into a second accumulator, D_w[128 x C] = HID[128 x 8] . Wc^T;
//   * both biases: a constant [1,1,0,..] K-slice in the A tile against [b_hi, b_lo, 0,..] in the B tile, so the epilogue
//     is lrelu(D) * relu(D_w) and nothing else;
//   * pass 3 altogether (it had no MMA at all).
// Structure of both kernels: CTA = 8 worker warps + 1 MMA warp, persistent over (sample, tile) items.
//   workers   meta (neighbour index, offset, weight-net hidden layer), produce (operand tiles into a 2-deep
//             shared-memory ring, K-major, 128-byte swizzle; 3xTF32 = hi/lo split), epilogue (tcgen05.ld, activation,
//             sum over the 16 neighbour rows by recursive halving, store).  Thread t <-> row t & 127.
//   MMA warp  one lane waits for "full" mbarriers, issues tcgen05.mma / tcgen05.commit; it never produces, so its
//             ~70 cycles per MMA issue are off the workers' critical path (r1 clock64 trace, DESIGN.md).
//   W2        pre-split into its swizzled shared-memory image once per call (corr3d_v2_prep_kernel) and brought in by
//             cp.async.bulk (one thread, zero per-thread instructions) — resident when it is a single K block.
// The accumulators are double-buffered in tensor memory when 4*C <= 512 columns, so the epilogue of tile t overlaps
// the MMAs of tile t+1; produce(t+1) is issued before epilogue(t).
#include <algorithm>

#include "corr3d_common.cuh"
#include "sm100_async.cuh"

#ifdef V2_TRACE
// debug builds only (profiles/build_variant.sh trace "-DV2_TRACE"): clock64 stamps of CTA 0's first worker thread per tile
__device__ long long v2_trace_buf[8 * 512];
extern "C" __attribute__((visibility("default"))) int b200_debug_read_v2_trace(long long* host, int n) {
    return (int)cudaMemcpyFromSymbol(host, v2_trace_buf, sizeof(long long) * n);
}
#define V2_STAMP(slot) do { if (blockIdx.x == 0 && tid == 0 && lt < 512) v2_trace_buf[lt * 8 + (slot)] = clock64(); } while (0)
#else
#define V2_STAMP(slot) do { } while (0)
#endif

namespace b200 {

constexpr int V2_ROWS = 128, V2_KB = 32, V2_K = 16;
constexpr int V2_TILE = V2_ROWS * 128;                  // one 128-row operand tile: 16 KB

// ---- weight images (once per call) ---------------------------------------------------------------------------------
// W2img  [nkb][hi|lo][C rows x 128 B]  : W2[o][kb*32 .. +32) split into TF32 hi/lo, in the swizzled layout of the B tile
// wcimg  [C rows x 128 B]              : chunks 0,1 = Wc_hi[o][0..7]; 2,3 = Wc_lo[o][0..7]; 4 = (bc_hi, bc_lo, 0, 0);
//                                        6 = (bias2_hi, bias2_lo, 0, 0)   (bias2 = cost_mlp's b2, or null for pass 3)
__global__ void corr3d_v2_prep_kernel(const float* __restrict__ W2, const float* __restrict__ Wc, const float* __restrict__ bc,
                                      const float* __restrict__ bias2, float* __restrict__ W2img, float* __restrict__ wcimg, int C) {
    const int nkb = C / V2_KB;
    const int n_w2 = W2img ? C * C : 0;
    const int total = n_w2 + C * 32;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        if (e < n_w2) {
            const int o = e / C, c = e - o * C, kb = c / V2_KB, cl = c - kb * V2_KB;
            const float v = __ldg(W2 + e), hi = tf32_hi(v);
            const size_t base = (size_t)kb * 2 * C * 32;                     // floats per K block: 2 tiles of C rows x 32 floats
            const uint32_t off = (sw128(o, cl >> 2) >> 2) + (cl & 3);
            W2img[base + off] = hi;
            W2img[base + (size_t)C * 32 + off] = v - hi;
        } else {
            const int r = e - n_w2, o = r >> 5, f = r & 31, q = f >> 2, w = f & 3;
            float v = 0.0f;
            if (q < 2) v = tf32_hi(__ldg(Wc + (size_t)o * 8 + f));
            else if (q < 4) { const float x = __ldg(Wc + (size_t)o * 8 + (f - 8)); v = x - tf32_hi(x); }
            else if (q == 4 && w < 2) { const float x = __ldg(bc + o); v = w == 0 ? tf32_hi(x) : x - tf32_hi(x); }
            else if (q == 6 && w < 2 && bias2) { const float x = __ldg(bias2 + o); v = w == 0 ? tf32_hi(x) : x - tf32_hi(x); }
            wcimg[(sw128(o, q) >> 2) + w] = v;
        }
        (void)nkb;
    }
}

// ---- shared-memory plan --------------------------------------------------------------------------------------------
struct V2Smem {
    int a[2], w[2];          // ring stages: A tile pair (hi | lo, 32 KB) and, when W2 is streamed, its K block (hi | lo)
    int hid[2];              // HID tiles (per accumulator buffer): chunks 0,1 hid_hi; 2,3 hid_lo; 4 = ones
    int wres, wc;            // resident W2 (single K block) and the Wc / bias image
    int w1c, wn, meta_j, meta_d, stagebuf, bars, total;
    int wbytes;              // bytes of one W2 K block (hi + lo)
};
__host__ __device__ inline V2Smem v2_layout(int C, bool with_w2, bool with_stagebuf, int depth) {
    V2Smem L;
    int off = 0;
    const bool resident = with_w2 && C == V2_KB;
    L.wbytes = with_w2 ? 2 * C * 128 : 0;
    for (int s = 0; s < 2; ++s) { L.a[s] = off; off += (with_w2 && s < depth) ? 2 * V2_TILE : 0; }
    for (int s = 0; s < 2; ++s) { L.w[s] = off; off += (with_w2 && !resident && s < depth) ? L.wbytes : 0; }
    for (int s = 0; s < 2; ++s) { L.hid[s] = off; off += s < depth ? V2_TILE : 0; }
    L.wres = off;   off += resident ? L.wbytes : 0;
    L.wc = off;     off += C * 128;                         // C % 8 == 0 -> 1024-aligned
    L.w1c = off;    off += with_w2 ? 3 * C * 4 : 0;
    L.wn = off;     off += WN_FLOATS * 4;
    L.meta_j = off; off += 2 * 256 * 4;                     // pass 2: s_j[128]; pass 3: one private slot per (tile parity, thread)
    L.meta_d = off; off += V2_ROWS * 16;
    L.stagebuf = off; off += with_stagebuf ? C * 33 * 4 : 0;
    off = (off + 15) & ~15;
    L.bars = off;   off += 128;                             // full[2], empty[2], acc_full[2], acc_empty[2], wres, tmem slot
    L.total = off;
    return L;
}

// weight-net hidden layer, split over the two threads of a row: this thread computes outputs [4*half, 4*half+4)
__device__ __forceinline__ void v2_hidden_half(const float* s_wn, float dx, float dy, float dz, int half, float (&out)[4]) {
    const float4* w4 = reinterpret_cast<const float4*>(s_wn);
    float wa[24], h1[8];
#pragma unroll
    for (int i = 0; i < 6; ++i) { const float4 v = w4[i]; wa[4 * i] = v.x; wa[4 * i + 1] = v.y; wa[4 * i + 2] = v.z; wa[4 * i + 3] = v.w; }
    const float4 ba0 = w4[6], ba1 = w4[7];
    const float bav[8] = {ba0.x, ba0.y, ba0.z, ba0.w, ba1.x, ba1.y, ba1.z, ba1.w};
#pragma unroll
    for (int o = 0; o < 8; ++o) {                           // same operation order as weight_net_hidden
        float s = bav[o];
        s = fmaf(wa[o * 3 + 0], dx, s);
        s = fmaf(wa[o * 3 + 1], dy, s);
        s = fmaf(wa[o * 3 + 2], dz, s);
        h1[o] = fmaxf(s, 0.0f);
    }
    const float4 bb = w4[24 + half];
    const float bbv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int o = 4 * half + u;
        const float4 r0 = w4[8 + 2 * o], r1 = w4[9 + 2 * o];
        float s = bbv[u];
        s = fmaf(r0.x, h1[0], s); s = fmaf(r0.y, h1[1], s); s = fmaf(r0.z, h1[2], s); s = fmaf(r0.w, h1[3], s);
        s = fmaf(r1.x, h1[4], s); s = fmaf(r1.y, h1[5], s); s = fmaf(r1.z, h1[6], s); s = fmaf(r1.w, h1[7], s);
        out[u] = fmaxf(s, 0.0f);
    }
}

// sum the 16 rows of a point (16 consecutive lanes) for 16 columns by recursive halving; lane m ends with column m
__device__ __forceinline__ float v2_reduce16(float (&v)[16], int m) {
#pragma unroll
    for (int h = 8, n = 8; h >= 1; h >>= 1, n >>= 1) {
        const bool up = (m & h) != 0;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            if (t < n) {
                const float keep = up ? v[n + t] : v[t];
                const float send = up ? v[t] : v[n + t];
                v[t] = keep + __shfl_xor_sync(FULL, send, h);
            }
        }
    }
    return v[0];
}

// the whole hidden layer by one thread (4 worker warps: one thread per row)
__device__ __forceinline__ void v2_hidden_full(const float* s_wn, float dx, float dy, float dz, float (&out)[8]) {
    weight_net_hidden_s(s_wn, dx, dy, dz, out);
}

// =====================================================================================================================
// pass 2: P[b,i,:] = sum_{j in knn12(i)} relu(weight_net2(d)) * lrelu(W2 . lrelu(A1_i + G2_j + W1c.d) + b2)
// NW = worker warps (4: one thread per row, thin CTAs that overlap each other on an SM; 8: two threads per row),
// DEPTH = stages of the operand ring / HID buffers (2 also double-buffers the accumulators when 4*C <= 512 columns).
// =====================================================================================================================
template <int NW, int DEPTH>
__global__ void __launch_bounds__(NW * 32 + 32, NW == 4 ? 4 : 1)
corr3d_v2_stage1_kernel(const float* __restrict__ xyz1, const float* __restrict__ xyz2, const int64_t* __restrict__ knn12,
                        const float* __restrict__ A1, const float* __restrict__ G2, const float* __restrict__ W2img,
                        const float* __restrict__ wcimg, const float* __restrict__ W1cT, const float* __restrict__ Wa,
                        const float* __restrict__ ba, const float* __restrict__ Wb, const float* __restrict__ bb,
                        float* __restrict__ P, int C, int N1, int N2, int B, uint32_t tmem_cols, int nbuf) {
    constexpr int NWT = NW * 32;                            // worker threads
    extern __shared__ uint8_t v2_smem_raw[];
    const uint32_t sbase = (smem_u32(v2_smem_raw) + 1023u) & ~1023u;
    uint8_t* gbase = v2_smem_raw + (sbase - smem_u32(v2_smem_raw));
    const V2Smem L = v2_layout(C, true, false, DEPTH);
    float* s_w1c = reinterpret_cast<float*>(gbase + L.w1c);
    float* s_wn = reinterpret_cast<float*>(gbase + L.wn);
    int* s_j = reinterpret_cast<int*>(gbase + L.meta_j);
    float4* s_d = reinterpret_cast<float4*>(gbase + L.meta_d);
    const uint32_t bars = sbase + L.bars;
    const uint32_t bar_wres = bars + 64, tmem_slot = bars + 72;
#define bar_full(s) (bars + 8u * (s))
#define bar_empty(s) (bars + 16u + 8u * (s))
#define bar_accf(s) (bars + 32u + 8u * (s))
#define bar_acce(s) (bars + 48u + 8u * (s))
#define HID_OFF(i) (L.hid[0] + (int)(i) * V2_TILE)
#define A_OFF(i) (L.a[0] + (int)(i) * 2 * V2_TILE)
#define W_OFF(i) (L.w[0] + (int)(i) * L.wbytes)
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + L.bars + 72);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nkb = C / V2_KB;
    const bool resident = nkb == 1;
    const uint32_t tiles = (uint32_t)(N1 + 7) / 8u;         // tiles per sample: 8 points x 16 neighbours = 128 rows
    const uint32_t items = (uint32_t)B * tiles;             // < 2^31 (checked on the host)

    if (tid == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar_full(s), NWT);
            mbar_init(bar_empty(s), 1);
            mbar_init(bar_accf(s), 1);
            mbar_init(bar_acce(s), NWT);
        }
        mbar_init(bar_wres, 1);
        mbar_init_fence();
    }
    if (warp == NW) {
        tmem_alloc(tmem_slot, tmem_cols);
    }
    if (tid < NWT) {
        for (int e = tid; e < 3 * C; e += NWT) s_w1c[e] = __ldg(W1cT + e);
        weight_net_stage(s_wn, Wa, ba, Wb, bb, tid, NWT);
        // constant part of the HID tiles: chunk 4 = (1, 1, 0, 0), everything else zero until meta writes chunks 0..3
        for (int e = tid; e < DEPTH * V2_ROWS * 8; e += NWT) {
            const int buf = e / (V2_ROWS * 8), r = (e >> 3) & (V2_ROWS - 1), q = e & 7;
            *reinterpret_cast<float4*>(gbase + HID_OFF(buf) + sw128(r, q)) = q == 4 ? make_float4(1.0f, 1.0f, 0.0f, 0.0f) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
        for (int e = tid; e < C * 8; e += NWT)              // Wc / bias image: already in tile layout
            reinterpret_cast<float4*>(gbase + L.wc)[e] = __ldg(reinterpret_cast<const float4*>(wcimg) + e);
        fence_proxy_async();
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot_ptr;
    const uint32_t idesc = umma_idesc_tf32(V2_ROWS, C);

    if (warp == NW) {
        // =============================== MMA warp ===============================
        if (lane == 0) {
            if (resident) {
                mbar_arrive_expect_tx(bar_wres, (uint32_t)L.wbytes);
                bulk_g2s(sbase + L.wres, W2img, (uint32_t)L.wbytes, bar_wres);
                mbar_wait(bar_wres, 0);
            }
            uint32_t it = 0, lt = 0;                        // ring items / tiles handled by this CTA so far
            for (uint32_t item = blockIdx.x; item < items; item += gridDim.x, ++lt) {
                const uint32_t buf = nbuf == 2 ? (lt & 1u) : 0u, use = nbuf == 2 ? (lt >> 1) : lt;
                const uint32_t acc = tmem + buf * 2u * (uint32_t)C, accw = acc + (uint32_t)C;
                const uint32_t wc = sbase + L.wc, hid = sbase + HID_OFF(lt % DEPTH);
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const uint32_t s = it % DEPTH, ph = it / DEPTH;
                    mbar_wait(bar_full(s), ph & 1u);
                    tcgen05_fence_after();
                    if (kb == 0) {
                        if (use >= 1) {                     // the epilogue that last read this accumulator pair is done
                            mbar_wait(bar_acce(buf), (use - 1) & 1u);
                            tcgen05_fence_after();
                        }
                        // weights: D_w = hid_hi.Wc_hi + hid_hi.Wc_lo + hid_lo.Wc_hi + 1.(bc_hi, bc_lo)
                        umma_tf32(accw, umma_desc_sw128(hid), umma_desc_sw128(wc), idesc, 0u);
                        umma_tf32(accw, umma_desc_sw128(hid), umma_desc_sw128(wc + 32), idesc, 1u);
                        umma_tf32(accw, umma_desc_sw128(hid + 32), umma_desc_sw128(wc), idesc, 1u);
                        umma_tf32(accw, umma_desc_sw128(hid + 64), umma_desc_sw128(wc + 64), idesc, 1u);
                        // main accumulator starts from the bias b2
                        umma_tf32(acc, umma_desc_sw128(hid + 64), umma_desc_sw128(wc + 96), idesc, 0u);
                    }
                    const uint32_t a_hi = sbase + A_OFF(s), a_lo = a_hi + V2_TILE;
                    const uint32_t w_hi = resident ? sbase + L.wres : sbase + W_OFF(s), w_lo = w_hi + (uint32_t)C * 128u;
#pragma unroll
                    for (int ks = 0; ks < V2_KB / 8; ++ks) {
                        const uint64_t ah = umma_desc_sw128(a_hi + ks * 32), wh = umma_desc_sw128(w_hi + ks * 32);
                        umma_tf32(acc, ah, wh, idesc, 1u);
                        umma_tf32(acc, ah, umma_desc_sw128(w_lo + ks * 32), idesc, 1u);
                        umma_tf32(acc, umma_desc_sw128(a_lo + ks * 32), wh, idesc, 1u);
                    }
                    umma_commit(bar_empty(s));
                    if (kb == nkb - 1) umma_commit(bar_accf(buf));
                }
            }
        }
        __syncwarp();
    } else {
        // =============================== worker warps ===============================
        const int row = tid & (V2_ROWS - 1), half = tid >> 7;
        const int lq = warp & 3, ch = warp >> 2;            // TMEM lane quarter / which share of the 16-column chunks
        const int m = lane & 15;
        uint32_t it = 0;

        // Fat CTAs (NW = 8, one or two per SM): loads are issued as early as their addresses are known, because nothing
        // else hides their latency (ncu r2: 57 % of the stall samples were long-scoreboard waits, one exposed round trip
        // per step) — the neighbour index of the NEXT tile is fetched while this tile is being produced, the A1 / G2 rows of
        // a K block are all requested before the first is used, and the next K block's rows before this one is converted.
        // Thin CTAs (NW = 4, several per SM) overlap each other instead and keep the register count low.
        constexpr bool DEEP = NW == 8;
        int64_t jpre = 0;
        uint32_t jpre_item = 0xffffffffu;
        auto fetch_j = [&](uint32_t item) {
            const uint32_t b = item / tiles, i0 = (item - b * tiles) * 8u;
            const int i = min((int)i0 + (row >> 4), N1 - 1);
            jpre = __ldg(knn12 + ((size_t)b * N1 + i) * V2_K + (row & 15));
            jpre_item = item;
        };
        constexpr int STEPS = 1024 / NWT, GROUP = 4;
        auto convert = [&](const float4& a, const float4& g, int r, int q, const float4& wx, const float4& wy, const float4& wz,
                           uint8_t* a_hi, uint8_t* a_lo) {
            const float4 d = s_d[r];
            float4 v;
            v.x = leaky01(a.x + g.x + fmaf(wz.x, d.z, fmaf(wy.x, d.y, wx.x * d.x)));
            v.y = leaky01(a.y + g.y + fmaf(wz.y, d.z, fmaf(wy.y, d.y, wx.y * d.x)));
            v.z = leaky01(a.z + g.z + fmaf(wz.z, d.z, fmaf(wy.z, d.y, wx.z * d.x)));
            v.w = leaky01(a.w + g.w + fmaf(wz.w, d.z, fmaf(wy.w, d.y, wx.w * d.x)));
            const float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
            const uint32_t off = sw128((uint32_t)r, (uint32_t)q);
            *reinterpret_cast<float4*>(a_hi + off) = hi;
            *reinterpret_cast<float4*>(a_lo + off) = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
        };
        auto produce = [&](uint32_t item, uint32_t lt) {
            const uint32_t b = item / tiles;
            const int i0 = (int)(item - b * tiles) * 8;
            V2_STAMP(0);
            // ---- meta: thread(s) of a row: neighbour index, offset, weight-net hidden layer
            {
                const int i = min(i0 + (row >> 4), N1 - 1);
                if (jpre_item != item) fetch_j(item);
                int64_t j = jpre;
                j = j < 0 ? 0 : (j >= N2 ? N2 - 1 : j);
                const float x2 = __ldg(xyz2 + ((size_t)b * 3 + 0) * N2 + j), y2 = __ldg(xyz2 + ((size_t)b * 3 + 1) * N2 + j),
                            z2 = __ldg(xyz2 + ((size_t)b * 3 + 2) * N2 + j);
                const float x1 = __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + i), y1 = __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + i),
                            z1 = __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + i);
                if (DEEP && item + gridDim.x < items) fetch_j(item + gridDim.x);   // in flight until the next produce()
                const float dx = x2 - x1, dy = y2 - y1, dz = z2 - z1;
#ifdef V2_TRACE
                if (dx == 123456.0f) s_d[row].w = dx;     // make the stamp below wait for the loads
                V2_STAMP(1);
#endif
                uint8_t* hid = gbase + HID_OFF(lt % DEPTH);
                if (NW == 8) {                              // two threads per row: `half` selects four of the eight outputs
                    float hd[4];
                    v2_hidden_half(s_wn, dx, dy, dz, half, hd);
                    named_bar_sync<1, NWT>();                  // every produce() read of the previous tile's s_j / s_d is done
                    const float4 hi = make_float4(tf32_hi(hd[0]), tf32_hi(hd[1]), tf32_hi(hd[2]), tf32_hi(hd[3]));
                    *reinterpret_cast<float4*>(hid + sw128(row, half)) = hi;
                    *reinterpret_cast<float4*>(hid + sw128(row, 2 + half)) = make_float4(hd[0] - hi.x, hd[1] - hi.y, hd[2] - hi.z, hd[3] - hi.w);
                } else {
                    float hd[8];
                    v2_hidden_full(s_wn, dx, dy, dz, hd);
                    named_bar_sync<1, NWT>();
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        const float4 hi = make_float4(tf32_hi(hd[4 * u]), tf32_hi(hd[4 * u + 1]), tf32_hi(hd[4 * u + 2]), tf32_hi(hd[4 * u + 3]));
                        *reinterpret_cast<float4*>(hid + sw128(row, u)) = hi;
                        *reinterpret_cast<float4*>(hid + sw128(row, 2 + u)) =
                            make_float4(hd[4 * u] - hi.x, hd[4 * u + 1] - hi.y, hd[4 * u + 2] - hi.z, hd[4 * u + 3] - hi.w);
                    }
                }
                // (the HID tile of this buffer is free: the MMAs of the tile that used it last were waited for by an
                // epilogue that precedes this call in every worker's program order)
                if (half == 0) { s_j[row] = (int)j; s_d[row] = make_float4(dx, dy, dz, 0.0f); }
                named_bar_sync<1, NWT>();
            }
            V2_STAMP(2);
            // ---- K blocks: this thread handles chunk q = tid & 7 of rows (step * NWT + tid) >> 3
            const int q = tid & 7;
            const float* a_base = A1 + (size_t)b * N1 * C + 4 * q;
            const float* g_base = G2 + (size_t)b * N2 * C + 4 * q;
            if (DEEP) {
                int a_off[STEPS], g_off[STEPS];             // element offsets: < 2^31 (a sample's A1 / G2 is N * C floats)
#pragma unroll
                for (int step = 0; step < STEPS; ++step) {
                    const int r = (step * NWT + tid) >> 3;
                    a_off[step] = min(i0 + (r >> 4), N1 - 1) * C;
                    g_off[step] = s_j[r] * C;
                }
                float4 a[STEPS], g[STEPS];
#pragma unroll
                for (int step = 0; step < STEPS; ++step) {
                    a[step] = __ldg(reinterpret_cast<const float4*>(a_base + a_off[step]));
                    g[step] = __ldg(reinterpret_cast<const float4*>(g_base + g_off[step]));
                }
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const uint32_t s = it % DEPTH, ph = it / DEPTH;
                    float4 an[STEPS], gn[STEPS];
                    if (kb + 1 < nkb) {
#pragma unroll
                        for (int step = 0; step < STEPS; ++step) {
                            an[step] = __ldg(reinterpret_cast<const float4*>(a_base + a_off[step] + (kb + 1) * V2_KB));
                            gn[step] = __ldg(reinterpret_cast<const float4*>(g_base + g_off[step] + (kb + 1) * V2_KB));
                        }
                    }
                    if (ph >= 1) mbar_wait(bar_empty(s), (ph - 1) & 1u);
                    uint8_t* a_hi = gbase + A_OFF(s);
                    uint8_t* a_lo = a_hi + V2_TILE;
                    if (!resident && tid == 0) {
                        mbar_arrive_expect_tx(bar_full(s), (uint32_t)L.wbytes);
                        bulk_g2s(sbase + W_OFF(s), W2img + (size_t)kb * 2 * C * 32, (uint32_t)L.wbytes, bar_full(s));
                    }
                    const int c0 = kb * V2_KB + 4 * q;
                    const float4 wx = *reinterpret_cast<const float4*>(s_w1c + c0);
                    const float4 wy = *reinterpret_cast<const float4*>(s_w1c + C + c0);
                    const float4 wz = *reinterpret_cast<const float4*>(s_w1c + 2 * C + c0);
#pragma unroll
                    for (int step = 0; step < STEPS; ++step) convert(a[step], g[step], (step * NWT + tid) >> 3, q, wx, wy, wz, a_hi, a_lo);
                    fence_proxy_async();
                    if (!(!resident && tid == 0)) mbar_arrive(bar_full(s));   // thread 0's arrival was the expect_tx one
                    if (kb + 1 < nkb) {
#pragma unroll
                        for (int step = 0; step < STEPS; ++step) { a[step] = an[step]; g[step] = gn[step]; }
                    }
                }
            } else {
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const uint32_t s = it % DEPTH, ph = it / DEPTH;
                    if (ph >= 1) mbar_wait(bar_empty(s), (ph - 1) & 1u);
                    uint8_t* a_hi = gbase + A_OFF(s);
                    uint8_t* a_lo = a_hi + V2_TILE;
                    if (!resident && tid == 0) {
                        mbar_arrive_expect_tx(bar_full(s), (uint32_t)L.wbytes);
                        bulk_g2s(sbase + W_OFF(s), W2img + (size_t)kb * 2 * C * 32, (uint32_t)L.wbytes, bar_full(s));
                    }
                    const int c0 = kb * V2_KB + 4 * q;
                    const float4 wx = *reinterpret_cast<const float4*>(s_w1c + c0);
                    const float4 wy = *reinterpret_cast<const float4*>(s_w1c + C + c0);
                    const float4 wz = *reinterpret_cast<const float4*>(s_w1c + 2 * C + c0);
#pragma unroll
                    for (int s0 = 0; s0 < STEPS; s0 += GROUP) {          // GROUP row pairs in flight, then converted
                        float4 a[GROUP], g[GROUP];
#pragma unroll
                        for (int u = 0; u < GROUP; ++u) {
                            const int r = ((s0 + u) * NWT + tid) >> 3;
                            a[u] = __ldg(reinterpret_cast<const float4*>(a_base + min(i0 + (r >> 4), N1 - 1) * C + kb * V2_KB));
                            g[u] = __ldg(reinterpret_cast<const float4*>(g_base + s_j[r] * C + kb * V2_KB));
                        }
#pragma unroll
                        for (int u = 0; u < GROUP; ++u) convert(a[u], g[u], ((s0 + u) * NWT + tid) >> 3, q, wx, wy, wz, a_hi, a_lo);
                    }
                    fence_proxy_async();
                    if (!(!resident && tid == 0)) mbar_arrive(bar_full(s));
                }
            }
            V2_STAMP(3);
        };

        auto epilogue = [&](uint32_t item, uint32_t lt) {
            const uint32_t b = item / tiles;
            const int i0 = (int)(item - b * tiles) * 8;
            const uint32_t buf = nbuf == 2 ? (lt & 1u) : 0u, use = nbuf == 2 ? (lt >> 1) : lt;
            V2_STAMP(4);
            mbar_wait(bar_accf(buf), use & 1u);
            tcgen05_fence_after();
            V2_STAMP(5);
            const uint32_t acc = tmem + buf * 2u * (uint32_t)C + ((uint32_t)(lq * 32) << 16);
            const int pt = i0 + lq * 2 + (lane >> 4);
            float* prow = P + ((size_t)b * N1 + min(pt, N1 - 1)) * C;
            for (int cb = ch * 16; cb < C; cb += 16 * (NW / 4)) {   // the warps of a lane quarter take alternate 16-column chunks
                uint32_t rm[16], rw[16];
                tmem_ld(acc + (uint32_t)cb, rm);
                tmem_ld(acc + (uint32_t)(C + cb), rw);
                tmem_ld_wait();
                float v[16];
#pragma unroll
                for (int c = 0; c < 16; ++c) v[c] = leaky01(__uint_as_float(rm[c])) * fmaxf(__uint_as_float(rw[c]), 0.0f);
                const float tot = v2_reduce16(v, m);
                if (pt < N1) prow[cb + m] = tot;
            }
            tcgen05_fence_before();
            mbar_arrive(bar_acce(buf));
            V2_STAMP(6);
        };

        // software pipeline over this CTA's tiles: with two accumulator buffers the operands of tile t+1 are produced
        // before the epilogue of tile t (its MMAs overlap the epilogue); with one buffer the epilogue comes first
        // (the MMAs of tile t+1 cannot start before it anyway — producing ahead would deadlock the ring).
        uint32_t cur = blockIdx.x, lt = 0;
        if (cur < items) produce(cur, 0);
        while (cur < items) {
            const uint32_t nxt = cur + gridDim.x;
            if (nbuf == 2) {
                if (nxt < items) produce(nxt, lt + 1);
                epilogue(cur, lt);
            } else {
                epilogue(cur, lt);
                if (nxt < items) produce(nxt, lt + 1);
            }
            cur = nxt;
            ++lt;
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    if (warp == NW) tmem_dealloc(tmem, tmem_cols);
}

// =====================================================================================================================
// pass 3: out[b,:,i] = sum_{j in knn11(i)} relu(weight_net1(xyz1_j - xyz1_i)) * P[b,j,:]
// An item = 32 consecutive points of one sample (4 tiles of 128 rows); results go through a [C][33] shared-memory tile
// so that the channel-first output is written as 128-byte runs.  4 worker warps (one thread per row) and one HID buffer /
// accumulator: thin CTAs, up to 4 of which overlap each other on an SM.
// =====================================================================================================================
__global__ void __launch_bounds__(160, 4)
corr3d_v2_stage2_kernel(const float* __restrict__ xyz1, const int64_t* __restrict__ knn11, const float* __restrict__ P,
                        const float* __restrict__ wcimg, const float* __restrict__ Wa, const float* __restrict__ ba,
                        const float* __restrict__ Wb, const float* __restrict__ bb, float* __restrict__ out, int C, int N1, int B,
                        uint32_t tmem_cols) {
    constexpr int NW = 4, NWT = 128;
    extern __shared__ uint8_t v2_smem_raw[];
    const uint32_t sbase = (smem_u32(v2_smem_raw) + 1023u) & ~1023u;
    uint8_t* gbase = v2_smem_raw + (sbase - smem_u32(v2_smem_raw));
    const V2Smem L = v2_layout(C, false, true, 1);
    float* s_wn = reinterpret_cast<float*>(gbase + L.wn);
    float* s_out = reinterpret_cast<float*>(gbase + L.stagebuf);
    const uint32_t bars = sbase + L.bars;
    const uint32_t tmem_slot = bars + 72;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + L.bars + 72);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t groups = (uint32_t)(N1 + 31) / 32u;      // items per sample
    const uint32_t items = (uint32_t)B * groups;            // < 2^31 (checked on the host)

    if (tid == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar_full(s), NWT);
            mbar_init(bar_accf(s), 1);
            mbar_init(bar_acce(s), NWT);
        }
        mbar_init_fence();
    }
    if (warp == NW) {
        tmem_alloc(tmem_slot, tmem_cols);
    }
    if (tid < NWT) {
        weight_net_stage(s_wn, Wa, ba, Wb, bb, tid, NWT);
        for (int e = tid; e < V2_ROWS * 8; e += NWT) {
            const int r = e >> 3, q = e & 7;
            *reinterpret_cast<float4*>(gbase + HID_OFF(0) + sw128(r, q)) = q == 4 ? make_float4(1.0f, 1.0f, 0.0f, 0.0f) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
        for (int e = tid; e < C * 8; e += NWT)
            reinterpret_cast<float4*>(gbase + L.wc)[e] = __ldg(reinterpret_cast<const float4*>(wcimg) + e);
        fence_proxy_async();
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot_ptr;
    const uint32_t idesc = umma_idesc_tf32(V2_ROWS, C);

    // tiles are numbered consecutively over this CTA's items: tile lt is the lt-th use of the one HID buffer / accumulator
    if (warp == NW) {
        if (lane == 0) {
            uint32_t lt = 0;
            for (uint32_t item = blockIdx.x; item < items; item += gridDim.x) {
                for (int t4 = 0; t4 < 4; ++t4, ++lt) {
                    mbar_wait(bar_full(0), lt & 1u);
                    tcgen05_fence_after();
                    if (lt >= 1) {
                        mbar_wait(bar_acce(0), (lt - 1) & 1u);
                        tcgen05_fence_after();
                    }
                    const uint32_t accw = tmem, wc = sbase + L.wc, hid = sbase + HID_OFF(0);
                    umma_tf32(accw, umma_desc_sw128(hid), umma_desc_sw128(wc), idesc, 0u);
                    umma_tf32(accw, umma_desc_sw128(hid), umma_desc_sw128(wc + 32), idesc, 1u);
                    umma_tf32(accw, umma_desc_sw128(hid + 32), umma_desc_sw128(wc), idesc, 1u);
                    umma_tf32(accw, umma_desc_sw128(hid + 64), umma_desc_sw128(wc + 64), idesc, 1u);
                    umma_commit(bar_accf(0));
                }
            }
        }
        __syncwarp();
    } else {
        const int row = tid & (V2_ROWS - 1);
        // ch is 0 in every worker warp; the kernel's register allocation (12 bytes of spill instead of 16) depends on it
        const int lq = warp & 3, ch = warp >> 2, m = lane & 15;

        // The tile sequence of this CTA: tile g = (item = blockIdx.x + (g / 4) * gridDim.x, quarter g % 4).
        // Loads are issued as early as their addresses are known (nothing else hides their latency at 1-3 CTAs per SM):
        // the neighbour index of tile g+2 is fetched during tile g, the P rows of a tile's first column chunk are
        // requested before the wait for its accumulator, later chunks one chunk ahead.
        auto tile_pos = [&](uint32_t g, int& b, int& i0) -> bool {
            const uint32_t item = blockIdx.x + (g >> 2) * gridDim.x;
            if (item >= items) return false;
            const uint32_t bb = item / groups;
            b = (int)bb;
            i0 = (int)(item - bb * groups) * 32 + (int)(g & 3u) * 8;
            return true;
        };
        auto fetch_j = [&](uint32_t g) -> int64_t {
            int b, i0;
            if (!tile_pos(g, b, i0)) return 0;
            const int i = min(i0 + (row >> 4), N1 - 1);
            return __ldg(knn11 + ((size_t)b * N1 + i) * V2_K + (row & 15));
        };
        // The HID buffer may be overwritten once the MMAs of the previous tile are complete: they are, because that
        // tile's epilogue (which waited for bar_accf) precedes this call in program order of every worker.
        auto meta = [&](int b, int i0, int64_t jraw) -> int {
            const int i = min(i0 + (row >> 4), N1 - 1);
            int64_t j = jraw;
            j = j < 0 ? 0 : (j >= N1 ? N1 - 1 : j);
            const float dx = __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + j) - __ldg(xyz1 + ((size_t)b * 3 + 0) * N1 + i);
            const float dy = __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + j) - __ldg(xyz1 + ((size_t)b * 3 + 1) * N1 + i);
            const float dz = __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + j) - __ldg(xyz1 + ((size_t)b * 3 + 2) * N1 + i);
            uint8_t* hid = gbase + HID_OFF(0);
            float hd[8];
            v2_hidden_full(s_wn, dx, dy, dz, hd);
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const float4 hi = make_float4(tf32_hi(hd[4 * u]), tf32_hi(hd[4 * u + 1]), tf32_hi(hd[4 * u + 2]), tf32_hi(hd[4 * u + 3]));
                *reinterpret_cast<float4*>(hid + sw128(row, u)) = hi;
                *reinterpret_cast<float4*>(hid + sw128(row, 2 + u)) =
                    make_float4(hd[4 * u] - hi.x, hd[4 * u + 1] - hi.y, hd[4 * u + 2] - hi.z, hd[4 * u + 3] - hi.w);
            }
            fence_proxy_async();
            mbar_arrive(bar_full(0));
            return (int)j;
        };
        auto load_p = [&](const float* prow, int cb, float4 (&p4)[4]) {
#pragma unroll
            for (int u = 0; u < 4; ++u) p4[u] = __ldg(reinterpret_cast<const float4*>(prow + cb) + u);
        };
        auto epilogue = [&](uint32_t g, const float* prow, float4 (&p4)[4]) {
            mbar_wait(bar_accf(0), g & 1u);
            tcgen05_fence_after();
            const uint32_t accw = tmem + ((uint32_t)(lq * 32) << 16);
            const int ptl = (int)(g & 3u) * 8 + lq * 2 + (lane >> 4);   // point index inside the 32-point item
            for (int cb = ch * 16; cb < C; cb += 16) {
                uint32_t rw[16];
                tmem_ld(accw + (uint32_t)cb, rw);
                float4 pn[4];
                if (cb + 16 < C) load_p(prow, cb + 16, pn);
                tmem_ld_wait();
                float v[16];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    v[4 * u + 0] = fmaxf(__uint_as_float(rw[4 * u + 0]), 0.0f) * p4[u].x;
                    v[4 * u + 1] = fmaxf(__uint_as_float(rw[4 * u + 1]), 0.0f) * p4[u].y;
                    v[4 * u + 2] = fmaxf(__uint_as_float(rw[4 * u + 2]), 0.0f) * p4[u].z;
                    v[4 * u + 3] = fmaxf(__uint_as_float(rw[4 * u + 3]), 0.0f) * p4[u].w;
                }
                const float tot = v2_reduce16(v, m);
                s_out[(cb + m) * 33 + ptl] = tot;
                if (cb + 16 < C) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) p4[u] = pn[u];
                }
            }
            tcgen05_fence_before();
            mbar_arrive(bar_acce(0));
        };

        const uint32_t ntiles = blockIdx.x < items ? ((items - 1u - blockIdx.x) / gridDim.x + 1u) * 4u : 0u;
        if (ntiles > 0) {
            // prologue: tile 0's meta, indices of tiles 1 and 2 in flight
            int b = 0, i0 = 0, bn = 0, in0 = 0;
            tile_pos(0, b, i0);
            int64_t jraw1 = fetch_j(1);
            int jcur = meta(b, i0, fetch_j(0));
            int64_t jraw2 = fetch_j(2);
            for (uint32_t g = 0; g < ntiles; ++g) {
                const bool more = g + 1 < ntiles;
                if (more) tile_pos(g + 1, bn, in0);
                const float* prow = P + ((size_t)b * N1 + jcur) * C;
                float4 p4[4];
                load_p(prow, ch * 16, p4);                  // requested before the accumulator wait
                epilogue(g, prow, p4);
                int jnext = 0;
                if (more) {                                 // with one buffer the next tile's HID can only be written after this epilogue
                    jnext = meta(bn, in0, jraw1);
                    jraw1 = jraw2;
                    jraw2 = fetch_j(g + 3);
                }
                jcur = jnext;
                if ((g & 3u) == 3u) {                       // the [C][33] tile of this 32-point item is complete
                    named_bar_sync<1, NWT>();
                    const int g0 = i0 - 24;
                    for (int e = tid; e < 32 * C; e += NWT) {
                        const int o = e >> 5, pt = e & 31;
                        if (g0 + pt < N1) out[((size_t)b * C + o) * N1 + g0 + pt] = s_out[o * 33 + pt];
                    }
                    named_bar_sync<1, NWT>();                  // ... and read before the next item overwrites it
                }
                b = bn; i0 = in0;
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    if (warp == NW) tmem_dealloc(tmem, tmem_cols);
}

// =====================================================================================================================
// pass 1: the two per-point halves of cost_mlp's first layer (pwc3d_core.py:91-93 after factorising the concat):
//   A1[b,i,:] = W1[:, 0:C] . feat1[b,:,i] + b1        G2[b,j,:] = W1[:, C:2C] . feat2[b,:,j]
// Channel-first features in, POINT-MAJOR rows out (the layout pass 2 gathers).  The first generation was a 64x64x16
// shared-memory SIMT GEMM at 4.3 instructions per FMA (K is only 32..192): 0.86 ms per step, a quarter of the whole op.
// Here: tile = 128 points, thread = point: 32 coalesced channel loads per K block, TF32 hi/lo split, one swizzled
// 128-byte row per thread into the A tile; tcgen05.mma (3xTF32) against the pre-split W image; epilogue = tcgen05.ld,
// + bias, 128-bit row stores.  4 worker warps + 1 MMA warp, 2-deep ring, accumulators double-buffered when 2*C <= 512.
// blockIdx.y = 0: A1 (feat1, bias), 1: G2 (feat2, no bias).
// =====================================================================================================================
__global__ void __launch_bounds__(160, 2)
corr3d_v2_linear_kernel(const float* __restrict__ feat1, const float* __restrict__ feat2, const float* __restrict__ W1img,
                        const float* __restrict__ b1, float* __restrict__ A1, float* __restrict__ G2, int C, int N1, int N2, int B,
                        uint32_t tmem_cols, int nbuf) {
    constexpr int NW = 4, NWT = 128, DEPTH = 2;
    extern __shared__ uint8_t v2_smem_raw[];
    const uint32_t sbase = (smem_u32(v2_smem_raw) + 1023u) & ~1023u;
    uint8_t* gbase = v2_smem_raw + (sbase - smem_u32(v2_smem_raw));
    const int which = blockIdx.y;
    const float* X = which ? feat2 : feat1;
    float* out = which ? G2 : A1;
    const int N = which ? N2 : N1;
    const int nkb = C / V2_KB;
    const int wbytes = 2 * C * 128;
    // smem: [A stage 0 | A stage 1] (32 KB each: hi | lo), [W stage 0 | W stage 1], bias[C], barriers
    const int a_off = 0, w_off = 2 * 2 * V2_TILE, bias_off = w_off + 2 * wbytes, bars_off = (bias_off + C * 4 + 15) & ~15;
    float* s_bias = reinterpret_cast<float*>(gbase + bias_off);
    const uint32_t bars = sbase + bars_off;
    const uint32_t tmem_slot = bars + 72;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + bars_off + 72);
    const float* Wimg = W1img + (size_t)which * 2 * C * C;          // [nkb][hi|lo][C x 32 floats] per half

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t tiles = (uint32_t)(N + V2_ROWS - 1) / V2_ROWS;
    const uint32_t items = (uint32_t)B * tiles;

    if (tid == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar_full(s), NWT);
            mbar_init(bar_empty(s), 1);
            mbar_init(bar_accf(s), 1);
            mbar_init(bar_acce(s), NWT);
        }
        mbar_init_fence();
    }
    if (warp == NW) {
        tmem_alloc(tmem_slot, tmem_cols);
    }
    for (int e = tid; e < C; e += blockDim.x) s_bias[e] = (which == 0 && b1) ? __ldg(b1 + e) : 0.0f;
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot_ptr;
    const uint32_t idesc = umma_idesc_tf32(V2_ROWS, C);

    if (warp == NW) {
        if (lane == 0) {
            uint32_t it = 0, lt = 0;
            for (uint32_t item = blockIdx.x; item < items; item += gridDim.x, ++lt) {
                const uint32_t buf = nbuf == 2 ? (lt & 1u) : 0u, use = nbuf == 2 ? (lt >> 1) : lt;
                const uint32_t acc = tmem + buf * (uint32_t)C;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const uint32_t s = it % DEPTH, ph = it / DEPTH;
                    mbar_wait(bar_full(s), ph & 1u);
                    tcgen05_fence_after();
                    if (kb == 0 && use >= 1) {
                        mbar_wait(bar_acce(buf), (use - 1) & 1u);
                        tcgen05_fence_after();
                    }
                    const uint32_t a_hi = sbase + a_off + s * 2 * V2_TILE, a_lo = a_hi + V2_TILE;
                    const uint32_t w_hi = sbase + w_off + s * wbytes, w_lo = w_hi + (uint32_t)C * 128u;
#pragma unroll
                    for (int ks = 0; ks < V2_KB / 8; ++ks) {
                        const uint64_t ah = umma_desc_sw128(a_hi + ks * 32), wh = umma_desc_sw128(w_hi + ks * 32);
                        umma_tf32(acc, ah, wh, idesc, (kb | ks) != 0);
                        umma_tf32(acc, ah, umma_desc_sw128(w_lo + ks * 32), idesc, 1u);
                        umma_tf32(acc, umma_desc_sw128(a_lo + ks * 32), wh, idesc, 1u);
                    }
                    umma_commit(bar_empty(s));
                    if (kb == nkb - 1) umma_commit(bar_accf(buf));
                }
            }
        }
        __syncwarp();
    } else {
        const int row = tid;                                // point inside the tile = TMEM lane (warp w owns lanes 32w..32w+31)
        uint32_t it = 0;
        auto produce = [&](uint32_t item) {
            const uint32_t b = item / tiles;
            const int n = min((int)(item - b * tiles) * V2_ROWS + row, N - 1);
            const float* x = X + (size_t)b * C * N + n;
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const uint32_t s = it % DEPTH, ph = it / DEPTH;
                float v[V2_KB];
#pragma unroll
                for (int c = 0; c < V2_KB; ++c) v[c] = __ldg(x + (size_t)(kb * V2_KB + c) * N);      // coalesced over the warp's points
                if (ph >= 1) mbar_wait(bar_empty(s), (ph - 1) & 1u);
                if (tid == 0) {
                    mbar_arrive_expect_tx(bar_full(s), (uint32_t)wbytes);
                    bulk_g2s(sbase + w_off + s * wbytes, Wimg + (size_t)kb * 2 * C * 32, (uint32_t)wbytes, bar_full(s));
                }
                uint8_t* a_hi = gbase + a_off + s * 2 * V2_TILE;
                uint8_t* a_lo = a_hi + V2_TILE;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float4 hi = make_float4(tf32_hi(v[4 * q]), tf32_hi(v[4 * q + 1]), tf32_hi(v[4 * q + 2]), tf32_hi(v[4 * q + 3]));
                    const uint32_t off = sw128((uint32_t)row, (uint32_t)q);
                    *reinterpret_cast<float4*>(a_hi + off) = hi;
                    *reinterpret_cast<float4*>(a_lo + off) = make_float4(v[4 * q] - hi.x, v[4 * q + 1] - hi.y, v[4 * q + 2] - hi.z, v[4 * q + 3] - hi.w);
                }
                fence_proxy_async();
                if (tid != 0) mbar_arrive(bar_full(s));
            }
        };
        auto epilogue = [&](uint32_t item, uint32_t lt) {
            const uint32_t b = item / tiles;
            const int n = (int)(item - b * tiles) * V2_ROWS + row;
            const uint32_t buf = nbuf == 2 ? (lt & 1u) : 0u, use = nbuf == 2 ? (lt >> 1) : lt;
            mbar_wait(bar_accf(buf), use & 1u);
            tcgen05_fence_after();
            const uint32_t acc = tmem + buf * (uint32_t)C + ((uint32_t)(warp * 32) << 16);
            float* orow = out + ((size_t)b * N + min(n, N - 1)) * C;
            for (int cb = 0; cb < C; cb += 16) {
                uint32_t r[16];
                tmem_ld(acc + (uint32_t)cb, r);
                tmem_ld_wait();
                if (n < N) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const float4 bb = *reinterpret_cast<const float4*>(s_bias + cb + 4 * u);
                        *reinterpret_cast<float4*>(orow + cb + 4 * u) =
                            make_float4(__uint_as_float(r[4 * u]) + bb.x, __uint_as_float(r[4 * u + 1]) + bb.y,
                                        __uint_as_float(r[4 * u + 2]) + bb.z, __uint_as_float(r[4 * u + 3]) + bb.w);
                    }
                }
            }
            tcgen05_fence_before();
            mbar_arrive(bar_acce(buf));
        };
        uint32_t cur = blockIdx.x, lt = 0;
        if (cur < items) produce(cur);
        while (cur < items) {
            const uint32_t nxt = cur + gridDim.x;
            if (nbuf == 2) {
                if (nxt < items) produce(nxt);
                epilogue(cur, lt);
            } else {
                epilogue(cur, lt);
                if (nxt < items) produce(nxt);
            }
            cur = nxt;
            ++lt;
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    if (warp == NW) tmem_dealloc(tmem, tmem_cols);
}

// W1 [C, 2C+3] -> two swizzled images (columns 0..C-1 and C..2C-1), each [nkb][hi|lo][C rows x 32 floats]
__global__ void corr3d_v2_prep_w1_kernel(const float* __restrict__ W1, float* __restrict__ W1img, int C) {
    const int Kin = 2 * C + 3, total = 2 * C * C;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int which = e / (C * C), r = e - which * C * C, o = r / C, c = r - o * C, kb = c / V2_KB, cl = c - kb * V2_KB;
        const float v = __ldg(W1 + (size_t)o * Kin + which * C + c), hi = tf32_hi(v);
        float* img = W1img + (size_t)which * 2 * C * C + (size_t)kb * 2 * C * 32;
        const uint32_t off = (sw128(o, cl >> 2) >> 2) + (cl & 3);
        img[off] = hi;
        img[(size_t)C * 32 + off] = v - hi;
    }
}

// ---- host side -----------------------------------------------------------------------------------------------------
struct V2Config { int nw, depth; };
static V2Config v2_config(int C) {
    // Pass 2: thin CTAs (4 worker warps, one stage; 2-4 of them overlap each other on an SM) or fat ones (8 worker warps,
    // 2-deep ring, hoisted loads; the overlap is inside the one CTA an SM can hold).  Measured at batch 74
    // (profiles/r2_notes.md): thin wins while >= 2 CTAs fit (C <= 128), fat wins pass 2 at C = 192.  Pass 3 is always thin.
    return C > 128 ? V2Config{8, 2} : V2Config{4, 1};
}

bool corr3d_v2_eligible(int C, int k, int precision) {
    if (precision != 2) return false;                      // 3xTF32 only (the default; precision 1 keeps the first-generation kernel)
    if (k != V2_K || C % 32 != 0 || C < 32 || C > 192) return false;
    return v2_layout(C, true, false, v2_config(C).depth).total + 1024 <= 227 * 1024 && v2_layout(C, false, true, 1).total + 1024 <= 227 * 1024;
}

static uint32_t pow2_cols(int need) {
    uint32_t c = 32;
    while ((int)c < need) c <<= 1;
    return c;
}

template <typename K>
static cudaError_t v2_prepare(K kern, int threads, size_t smem, uint32_t cols, int* ctas_per_sm) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    // without this the driver picks the smallest carve-out that fits ONE CTA and co-residency is lost
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    // CTAs per SM from first principles (registers are allocated per warp in units of 256; 1 KB of shared memory is
    // reserved per CTA; 228 KB per SM).  cudaOccupancyMaxActiveBlocksPerMultiprocessor answered 1 for every variant
    // of these kernels on the r2 box while ncu reported 2-4 resident CTAs, so it is not used.
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess) return e;
    const int warps = (threads + 31) / 32;
    const int regs_per_warp = ((fa.numRegs * 32 + 255) / 256) * 256;
    int n = std::min(std::min(65536 / (regs_per_warp * warps), (int)((228 * 1024) / (smem + fa.sharedSizeBytes + 1024))), 2048 / threads);
    n = std::min(n, (int)(512 / cols));                    // tensor memory: 512 columns per SM
    *ctas_per_sm = std::max(n, 1);
    return cudaSuccess;
}

cudaError_t corr3d_v2_run(const float* xyz1, const float* feat1, const float* xyz2, const float* feat2, const int64_t* knn12,
                          const int64_t* knn11, const Corr3dScratch& s, const b200_corr3d_weights* w, float* out, int B, int C, int N1,
                          int N2, cudaStream_t st) {
    if ((long long)B * ((N1 + 7) / 8) >= (1ll << 31)) return cudaErrorInvalidValue;     // 32-bit item counters in the kernels
    float* W2img = s.v2_W2img;
    float* wc2 = s.v2_wcimg;                    // weight_net2 + b2 (pass 2)
    float* wc1 = s.v2_wcimg + (size_t)C * 32;   // weight_net1 (pass 3)
    corr3d_v2_prep_kernel<<<ceil_div(C * C + C * 32, 256), 256, 0, st>>>(w->W2, w->n2_Wc, w->n2_bc, w->b2, W2img, wc2, C);
    corr3d_v2_prep_kernel<<<ceil_div(C * 32, 256), 256, 0, st>>>(nullptr, w->n1_Wc, w->n1_bc, nullptr, nullptr, wc1, C);
    corr3d_v2_prep_w1_kernel<<<ceil_div(2 * C * C, 256), 256, 0, st>>>(w->W1, s.v2_W1img, C);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;

    // ---- pass 1
    {
        const int nbuf = 2 * C <= 512 ? 2 : 1;
        const uint32_t cols = pow2_cols(nbuf * C);
        const size_t smem = (size_t)(2 * 2 * V2_TILE + 2 * 2 * C * 128 + C * 4 + 16 + 128) + 1024;
        int per_sm = 1;
        e = v2_prepare(corr3d_v2_linear_kernel, 160, smem, cols, &per_sm);
        if (e != cudaSuccess) return e;
        const long long items = (long long)B * ((std::max(N1, N2) + V2_ROWS - 1) / V2_ROWS);
        const int gx = (int)std::max<long long>(1, std::min<long long>(items, ((long long)sm_count() * per_sm + 1) / 2));
        corr3d_v2_linear_kernel<<<dim3(gx, 2), 160, smem, st>>>(feat1, feat2, s.v2_W1img, w->b1, s.A1, s.G2, C, N1, N2, B, cols, nbuf);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    // ---- pass 2
    {
        const V2Config c = v2_config(C);
        const int nbuf = (c.depth == 2 && 4 * C <= 512) ? 2 : 1;
        const size_t smem = (size_t)v2_layout(C, true, false, c.depth).total + 1024;
        const uint32_t cols = pow2_cols(nbuf * 2 * C);
        const int threads = c.nw * 32 + 32;
        const long long items = (long long)B * ((N1 + 7) / 8);
        int per_sm = 1;
#define V2_LAUNCH1(NW, DEPTH)                                                                                                       \
    do {                                                                                                                            \
        e = v2_prepare(corr3d_v2_stage1_kernel<NW, DEPTH>, threads, smem, cols, &per_sm);                                           \
        if (e != cudaSuccess) return e;                                                                                             \
        const int grid = (int)std::min<long long>(items, (long long)sm_count() * per_sm);                                           \
        corr3d_v2_stage1_kernel<NW, DEPTH><<<grid, threads, smem, st>>>(xyz1, xyz2, knn12, s.A1, s.G2, W2img, wc2, s.W1cT, w->n2_Wa, \
                                                                       w->n2_ba, w->n2_Wb, w->n2_bb, s.P, C, N1, N2, B, cols, nbuf); \
    } while (0)
        if (c.nw == 8) V2_LAUNCH1(8, 2);
        else V2_LAUNCH1(4, 1);
#undef V2_LAUNCH1
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    // ---- pass 3
    {
        const size_t smem = (size_t)v2_layout(C, false, true, 1).total + 1024;
        const uint32_t cols = pow2_cols(C);
        const long long items = (long long)B * ((N1 + 31) / 32);
        int per_sm = 1;
        e = v2_prepare(corr3d_v2_stage2_kernel, 160, smem, cols, &per_sm);
        if (e != cudaSuccess) return e;
        const int grid = (int)std::min<long long>(items, (long long)sm_count() * per_sm);
        corr3d_v2_stage2_kernel<<<grid, 160, smem, st>>>(xyz1, knn11, s.P, wc1, w->n1_Wa, w->n1_ba, w->n1_Wb, w->n1_bb, out, C, N1, B,
                                                         cols);
    }
    return cudaGetLastError();
}

}  // namespace b200
