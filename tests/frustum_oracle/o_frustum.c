/* o_frustum.c -- CPU restatement of mr_terrain_cull_frustum: the checker the frustum-cull tests compare the GPU with.
 * Test infrastructure, not product: built with -ffp-contract=off (every float operation rounded on its own) into
 * libmr_oracle_frustum.so and loaded by tests/_frustum_oracle.py.  It stands beside the reference oracle under oracle/,
 * which it does not change: the compaction below is mr_o_terrain_cull's, with the frustum test as the visibility bit. */
#include <stddef.h>
#include <stdint.h>
#include "../../include/myrenderer_b200.h"

int mr_o_frustum_visible(const float view_proj[16], const float p0[4], const float p1[4]);
int mr_o_terrain_cull_frustum(const float* bbox, uint32_t n, uint32_t tile_rows, uint32_t tile_cols, const float view_proj[16],
                              uint32_t* visible_out, uint32_t* visible_ids_out, uint32_t* idx_out, uint64_t counts_out[2]);

/* The six-plane frustum test of mr_terrain_cull_frustum (NEW SPEC: the reference has no frustum test), literally as the
 * header states it: planes R3+R0, R3-R0, R3+R1, R3-R1, R2, R3-R2 from the rows R_i = (m[i], m[4+i], m[8+i], m[12+i]);
 * per plane the p-vertex (hi where the coefficient is >= 0, else lo) and s = ((a*px + b*py) + c*pz) + d, each operation
 * rounded (-ffp-contract=off); culled iff s < 0 for some plane.  Returns 1 if the box is kept. */
int mr_o_frustum_visible(const float view_proj[16], const float p0[4], const float p1[4]) {
    float pl[6][4];
    int j, k;
    for (j = 0; j < 4; ++j) {
        const float r0 = view_proj[4 * j], r1 = view_proj[4 * j + 1], r2 = view_proj[4 * j + 2], r3 = view_proj[4 * j + 3];
        pl[0][j] = r3 + r0;
        pl[1][j] = r3 - r0;
        pl[2][j] = r3 + r1;
        pl[3][j] = r3 - r1;
        pl[4][j] = r2;
        pl[5][j] = r3 - r2;
    }
    for (k = 0; k < 6; ++k) {
        const float a = pl[k][0], b = pl[k][1], c = pl[k][2], d = pl[k][3];
        const float px = a >= 0.0f ? p1[0] : p0[0];
        const float py = b >= 0.0f ? p1[1] : p0[1];
        const float pz = c >= 0.0f ? p1[2] : p0[2];
        const float ax = a * px, by = b * py, cz = c * pz;
        const float s1 = ax + by, s2 = s1 + cz, s = s2 + d;
        if (s < 0.0f) return 0;
    }
    return 1;
}

/* mr_o_terrain_cull (oracle/o_terrain.c) with mr_o_frustum_visible as the test: the same compaction and outputs */
int mr_o_terrain_cull_frustum(const float* bbox, uint32_t n, uint32_t tile_rows, uint32_t tile_cols, const float view_proj[16],
                              uint32_t* visible_out, uint32_t* visible_ids_out, uint32_t* idx_out, uint64_t counts_out[2]) {
    uint32_t tiles_r, tiles_c, t, nvis = 0;
    uint64_t nidx = 0;
    if (!bbox || n < 2 || !tile_rows || !tile_cols) return MR_E_BADARG;
    tiles_r = (n - 1u + tile_rows - 1u) / tile_rows;
    tiles_c = (n - 1u + tile_cols - 1u) / tile_cols;
    for (t = 0; t < tiles_r * tiles_c; ++t) {
        int vis = mr_o_frustum_visible(view_proj, bbox + 8u * (size_t)t, bbox + 8u * (size_t)t + 4u);
        if (visible_out) visible_out[t] = vis ? 1u : 0u;
        if (vis) {
            uint32_t tr = t / tiles_c, tc = t % tiles_c, r0 = tr * tile_rows, c0 = tc * tile_cols, r, c;
            uint32_t qr = tile_rows < n - 1u - r0 ? tile_rows : n - 1u - r0;
            uint32_t qc = tile_cols < n - 1u - c0 ? tile_cols : n - 1u - c0;
            if (visible_ids_out) visible_ids_out[nvis] = t;
            ++nvis;
            for (r = r0; r < r0 + qr; ++r)
                for (c = c0; c < c0 + qc; ++c) {
                    if (idx_out) {
                        uint32_t i00 = r * n + c;
                        uint32_t* o = idx_out + nidx;
                        o[0] = i00 + n; o[1] = i00; o[2] = i00 + n + 1u; o[3] = i00 + n + 1u; o[4] = i00; o[5] = i00 + 1u;
                    }
                    nidx += 6u;
                }
        }
    }
    if (counts_out) {
        counts_out[0] = nvis;
        counts_out[1] = nidx;
    }
    return MR_OK;
}
