/* Plain-C consumer of p2p_project_view_list_tables: a flat list that mixes integer-roll yaws and yaws that are not
 * integer column rolls, in one call.
 *   gcc -std=c99 -Wall -Iinclude tests/c_fractional_list.c -o c_fractional_list -L<dir> -lp2p_b200 -Wl,-rpath,<dir>
 *   ./c_fractional_list Wp Hp W H fov out.bin     (writes 4 * H * W * 3 bytes: views (0, 60), (33.3, 60), (90, 120),
 *                                                  (33.3, 120); the two 33.3 views share one column table)
 * The panorama is the LCG pattern of tests/c_abi_smoke.c. */
#include <stdio.h>
#include <stdlib.h>

#include "p2p.h"

#define CHECK(call)                                                                 \
    do {                                                                            \
        int rc_ = (call);                                                           \
        if (rc_ != P2P_OK) {                                                        \
            fprintf(stderr, "%s -> %d (%s): %s\n", #call, rc_, p2p_status_string(rc_), \
                    ctx ? p2p_last_error(ctx) : "");                                \
            return 2;                                                               \
        }                                                                           \
    } while (0)

int main(int argc, char **argv) {
    p2p_ctx *ctx = NULL;
    if (argc != 7) {
        fprintf(stderr, "usage: %s Wp Hp W H fov out.bin\n", argv[0]);
        return 1;
    }
    const int Wp = atoi(argv[1]), Hp = atoi(argv[2]), W = atoi(argv[3]), H = atoi(argv[4]), fov = atoi(argv[5]);
    const double yaws[4] = {0.0, 33.3, 90.0, 33.3};
    const double pitches[4] = {60.0, 60.0, 120.0, 120.0};
    const int n_views = 4;
    size_t i, n = (size_t)Wp * Hp * 3, out_bytes = (size_t)n_views * W * H * 3;
    unsigned char *pano = (unsigned char *)malloc(n);
    unsigned char *out = (unsigned char *)malloc(out_bytes);
    int32_t *ix = (int32_t *)malloc(sizeof(int32_t) * (size_t)Wp), *fx = (int32_t *)malloc(sizeof(int32_t) * (size_t)Wp);
    int32_t shifts[4];
    const int32_t *ixs[4] = {NULL, NULL, NULL, NULL}, *fxs[4] = {NULL, NULL, NULL, NULL};
    p2p_pitch_consts pc[4];
    unsigned int s = 12345u;
    int k;
    FILE *f;
    if (!pano || !out || !ix || !fx) return 1;
    for (i = 0; i < n; ++i) {
        s = s * 1664525u + 1013904223u;
        pano[i] = (unsigned char)(s >> 24);
    }
    CHECK(p2p_create(0, 1, &ctx));
    for (k = 0; k < n_views; ++k) {
        CHECK(p2p_pitch_constants((double)fov, pitches[k], W, &pc[k]));
        if (yaws[k] == 33.3) {
            CHECK(p2p_yaw_table(Wp, yaws[k], ix, fx, &shifts[k]));   /* shift -1: not an integer roll */
            if (shifts[k] >= 0) return 4;
            ixs[k] = ix;
            fxs[k] = fx;
        } else {
            int32_t *tix = (int32_t *)malloc(sizeof(int32_t) * (size_t)Wp), *tfx = (int32_t *)malloc(sizeof(int32_t) * (size_t)Wp);
            if (!tix || !tfx) return 1;
            CHECK(p2p_yaw_table(Wp, yaws[k], tix, tfx, &shifts[k]));
            free(tix);
            free(tfx);
            if (shifts[k] < 0) return 4;
        }
    }
    CHECK(p2p_upload_pano(ctx, 0, pano, Wp, Hp, (size_t)Wp * 3));
    CHECK(p2p_project_view_list_tables(ctx, 0, n_views, shifts, ixs, fxs, pc, W, H, 0, H, out, 0));
    CHECK(p2p_sync(ctx, 0));
    f = fopen(argv[6], "wb");
    if (!f) return 5;
    fwrite(out, 1, out_bytes, f);
    fclose(f);
    p2p_destroy(ctx);
    free(pano); free(out); free(ix); free(fx);
    return 0;
}
