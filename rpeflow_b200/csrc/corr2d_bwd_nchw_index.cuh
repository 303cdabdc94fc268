// corr2d_bwd_nchw_index.cuh — every address corr2d_bwd_nchw.cu forms, as host-and-device inline functions.
//
// The kernel takes its tile origin, its cp.async pieces (source offset, in-image predicate, shared-memory slot) and its
// output offsets from here, and tests/corr2d_bwd_nchw_audit.cpp walks the same functions on the CPU for every piece of
// every tile: sources inside the tensor (zero-filled pieces point at its base), 16-byte pieces 4-float aligned, and
// every output element written exactly once.  Plain C++ (no CUDA headers) so that a host compiler can include it.
#pragma once
#include <stddef.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define BN_HD __host__ __device__ __forceinline__
#define BN_CE __host__ __device__ constexpr
#else
#define BN_HD inline
#define BN_CE constexpr
#endif

namespace b200 {
namespace bn {

constexpr int TH = 8, TW = 32, P = 8, CC = 32, CB = 8, MD = 4, ND = 9;
constexpr int HR = TH + 2 * MD, HC = TW + 2 * MD;   // 16 x 40 halo
constexpr int HP = 44;                              // halo row pitch (floats): 11 sixteen-byte units, odd
constexpr int GP = 36;                              // grad_out row pitch (floats): 9 sixteen-byte units, odd
constexpr int THREADS = 128;
constexpr int H_FLOATS = CC * HR * HP;              // partner halo [32 ch][16 rows][44]: 22528 floats
constexpr int G_FLOATS = ND * TH * GP;              // grad_out planes of one row offset [9][8][36]: 2592 floats
constexpr size_t SMEM = (size_t)(2 * G_FLOATS + H_FLOATS) * sizeof(float);   // 110,848 B: two CTAs per SM

// ALIGNED: W % 4 == 0 and every pointer 16-byte aligned -> 16-byte halo pieces and float4 stores; otherwise 4-byte
// pieces and scalar stores.  WHICH = 1 stages grad_out unshifted (16-byte pieces when ALIGNED), WHICH = 2 pre-shifted
// by each plane's own displacement (always 4-byte pieces).
template <bool ALIGNED> BN_CE int halo_width() { return ALIGNED ? 4 : 1; }
template <bool ALIGNED> BN_CE int halo_pieces() { return CC * HR * HC / halo_width<ALIGNED>(); }
template <int WHICH, bool ALIGNED> BN_CE int grad_width() { return (WHICH == 1 && ALIGNED) ? 4 : 1; }
template <int WHICH, bool ALIGNED> BN_CE int grad_pieces() { return ND * TH * TW / grad_width<WHICH, ALIGNED>(); }

struct Tile {
    int b, y0, x0;
};
BN_HD Tile tile_of(int tile, int tiles_x, int tiles_y) {
    const int tx = tile % tiles_x;
    tile /= tiles_x;
    return Tile{tile / tiles_y, (tile % tiles_y) * TH, tx * TW};
}

struct Piece {
    int dst;       // float offset in the destination buffer (halo or one grad_out buffer)
    size_t src;    // float offset from the tensor's base; 0 for a zero-filled piece
    bool in;       // false: the piece is zero-filled (outside the image or a channel >= C)
};

// Partner halo piece e of channel chunk c0: channel ch, halo row, halo column col (a 4-column run when ALIGNED).
template <bool ALIGNED>
BN_HD Piece halo_piece(int e, Tile t, int c0, int C, int H, int W) {
    constexpr int PW = halo_width<ALIGNED>(), PR = HC / PW;
    const int col = (e % PR) * PW, row = (e / PR) % HR, ch = e / (PR * HR);
    const int gy = t.y0 + row - MD, gx = t.x0 + col - MD, c = c0 + ch;
    const bool in = gy >= 0 && gy < H && gx >= 0 && gx < W && c < C;   // ALIGNED: W % 4 == 0, a run is in or out whole
    return Piece{(ch * HR + row) * HP + col, in ? (((size_t)t.b * C + c) * H + gy) * W + gx : 0, in};
}

// grad_out piece e for partner row offset pdy: slot pdx holds plane t(pdy, pdx); for WHICH = 2 the plane of the mirrored
// displacement, read at (y - dy, x - dx), so that both gradients walk the halo with the same offsets.
template <int WHICH, bool ALIGNED>
BN_HD Piece grad_piece(int e, int pdy, Tile t, int H, int W) {
    constexpr int PW = grad_width<WHICH, ALIGNED>(), PR = TW / PW;
    const int i = (e % PR) * PW, rr = (e / PR) % TH, pdx = e / (PR * TH);
    int plane_t, gy, gx;
    if (WHICH == 1) {
        plane_t = pdy * ND + pdx;
        gy = t.y0 + rr;
        gx = t.x0 + i;
    } else {
        const int dyi = ND - 1 - pdy, dxi = ND - 1 - pdx;
        plane_t = dyi * ND + dxi;
        gy = t.y0 + rr - (dyi - MD);
        gx = t.x0 + i - (dxi - MD);
    }
    const bool in = gy >= 0 && gy < H && gx >= 0 && gx < W;
    return Piece{(pdx * TH + rr) * GP + i, in ? (((size_t)t.b * ND * ND + plane_t) * H + gy) * W + gx : 0, in};
}

// Thread -> (channel group = warp, tile row, 8-pixel strip); the 8 lanes of an LDS.128 phase are 8 rows of one strip.
BN_HD int thread_cg(int tid) { return tid >> 5; }
BN_HD int thread_row(int tid) { return tid & 7; }
BN_HD int thread_strip(int tid) { return (tid & 31) >> 3; }

// Shared-memory reads of thread tid at row offset pdy: the 16 halo columns of channel c (of its 8), and the 8 grad_out
// values of column offset pdx.  Both start 16-byte aligned.
BN_HD int halo_read(int tid, int c, int pdy) {
    return ((thread_cg(tid) * CB + c) * HR + thread_row(tid) + pdy) * HP + thread_strip(tid) * P;
}
BN_HD int grad_read(int tid, int pdx) { return (pdx * TH + thread_row(tid)) * GP + thread_strip(tid) * P; }

// Output element (channel ch, pixel (y, x)) of sample b, NCHW.
BN_HD size_t out_offset(int b, int ch, int y, int x, int C, int H, int W) {
    return (((size_t)b * C + ch) * H + y) * W + x;
}

}  // namespace bn
}  // namespace b200
