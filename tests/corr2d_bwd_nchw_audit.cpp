// Address audit of corr2d_bwd_nchw.cu: walks, on the CPU, every cp.async piece, shared-memory read and output store
// that the kernel forms through corr2d_bwd_nchw_index.cuh, for each shape "B C H W" given on the command line, both
// gradients and every ALIGNED value the host can select for it.  Prints one line per failure and exits 1 if any.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "corr2d_bwd_nchw_index.cuh"

using namespace b200::bn;

static long failures = 0;
#define EXPECT(cond, ...)                                                \
    do {                                                                 \
        if (!(cond) && failures++ < 20) {                                \
            std::printf("FAIL B=%d C=%d H=%d W=%d WHICH=%d ALIGNED=%d: ", B, C, H, W, WHICH, (int)ALIGNED); \
            std::printf(__VA_ARGS__);                                    \
            std::printf("\n");                                           \
        }                                                                \
    } while (0)

template <int WHICH, bool ALIGNED>
static void audit(int B, int C, int H, int W) {
    const size_t n_in = (size_t)B * C * H * W, n_g = (size_t)B * ND * ND * H * W;
    const int tiles_x = (W + TW - 1) / TW, tiles_y = (H + TH - 1) / TH;
    std::vector<unsigned char> written(n_in, 0);
    for (int tile = 0; tile < B * tiles_x * tiles_y; ++tile) {
        const Tile t = tile_of(tile, tiles_x, tiles_y);
        EXPECT(t.b >= 0 && t.b < B && t.y0 >= 0 && t.y0 < H && t.x0 >= 0 && t.x0 < W, "tile %d origin", tile);
        for (int c0 = 0; c0 < C; c0 += CC) {
            constexpr int HW_ = halo_width<ALIGNED>();
            for (int e = 0; e < halo_pieces<ALIGNED>(); ++e) {
                const Piece p = halo_piece<ALIGNED>(e, t, c0, C, H, W);
                EXPECT(p.dst >= 0 && p.dst + HW_ <= H_FLOATS, "halo piece %d dst %d", e, p.dst);
                EXPECT(p.src + HW_ <= n_in, "halo piece %d src %zu of %zu", e, p.src, n_in);
                EXPECT(p.in || p.src == 0, "zero-filled halo piece %d not at the base", e);
                if (HW_ == 4) EXPECT(p.src % 4 == 0 && p.dst % 4 == 0, "halo piece %d misaligned", e);
            }
            constexpr int GW = grad_width<WHICH, ALIGNED>();
            for (int pdy = 0; pdy < ND; ++pdy)
                for (int e = 0; e < grad_pieces<WHICH, ALIGNED>(); ++e) {
                    const Piece p = grad_piece<WHICH, ALIGNED>(e, pdy, t, H, W);
                    EXPECT(p.dst >= 0 && p.dst + GW <= G_FLOATS, "grad piece %d dst %d", e, p.dst);
                    EXPECT(p.src + GW <= n_g, "grad piece %d src %zu of %zu", e, p.src, n_g);
                    EXPECT(p.in || p.src == 0, "zero-filled grad piece %d not at the base", e);
                    if (GW == 4) EXPECT(p.src % 4 == 0 && p.dst % 4 == 0, "grad piece %d misaligned", e);
                }
            for (int tid = 0; tid < THREADS; ++tid) {
                for (int pdy = 0; pdy < ND; ++pdy)
                    for (int c = 0; c < CB; ++c) {
                        const int r = halo_read(tid, c, pdy);
                        EXPECT(r % 4 == 0 && r >= 0 && r + 2 * P <= H_FLOATS, "halo read %d", r);
                    }
                for (int pdx = 0; pdx < ND; ++pdx) {
                    const int r = grad_read(tid, pdx);
                    EXPECT(r % 4 == 0 && r >= 0 && r + P <= G_FLOATS, "grad read %d", r);
                }
                const int y = t.y0 + thread_row(tid), x = t.x0 + thread_strip(tid) * P;
                if (y >= H) continue;
                for (int c = 0; c < CB; ++c) {
                    const int ch = c0 + thread_cg(tid) * CB + c;
                    if (ch >= C) continue;
                    const size_t o = out_offset(t.b, ch, y, x, C, H, W);
                    if (ALIGNED) {
                        for (int m = 0; m < P / 4; ++m) {
                            if (x + 4 * m >= W) continue;
                            EXPECT(x + 4 * m + 4 <= W && (o + 4 * m) % 4 == 0 && o + 4 * m + 4 <= n_in, "float4 store at %zu", o);
                            for (int j = 4 * m; j < 4 * m + 4; ++j)
                                if (o + j < n_in) ++written[o + j];
                        }
                    } else {
                        for (int j = 0; j < P; ++j) {
                            if (x + j >= W) continue;
                            EXPECT(o + j < n_in, "store at %zu of %zu", o + j, n_in);
                            if (o + j < n_in) ++written[o + j];
                        }
                    }
                }
            }
        }
    }
    size_t bad = 0;
    for (size_t i = 0; i < n_in; ++i) bad += written[i] != 1;
    EXPECT(bad == 0, "%zu output elements not written exactly once", bad);
}

int main(int argc, char** argv) {
    if ((argc - 1) % 4 != 0 || argc == 1) {
        std::fprintf(stderr, "usage: %s B C H W [B C H W ...]\n", argv[0]);
        return 2;
    }
    int shapes = 0;
    for (int a = 1; a + 3 < argc; a += 4, ++shapes) {
        const int B = std::atoi(argv[a]), C = std::atoi(argv[a + 1]), H = std::atoi(argv[a + 2]), W = std::atoi(argv[a + 3]);
        audit<1, false>(B, C, H, W);
        audit<2, false>(B, C, H, W);
        if (W % 4 == 0) {
            audit<1, true>(B, C, H, W);
            audit<2, true>(B, C, H, W);
        }
    }
    std::printf("%d shapes, %ld failures\n", shapes, failures);
    return failures ? 1 : 0;
}
