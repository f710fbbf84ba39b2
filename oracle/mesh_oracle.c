/* TEST INFRASTRUCTURE ONLY -- serial C restatement of the marching-cubes export (instance_nerf_b200/csrc/mesh.cu,
 * include/inerf_b200.h "mesh export"): the same table header, the same fp32 arithmetic in the same order (built with
 * -ffp-contract=off; no product here may be contracted into an fma, so none is written) and the same output order.
 *
 * oracle_mesh: counts[0..1] = (V, F); verts / tris (may be NULL) receive the mesh when they are non-NULL. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include "mc_table.h"

int oracle_mesh(const float *v, uint32_t X, uint32_t Y, uint32_t Z, const float *bbox, float iso, int32_t *counts, float *verts,
                int32_t *tris) {
    const uint32_t n[3] = {X, Y, Z};
    const size_t YZ = (size_t)Y * Z, N = (size_t)X * YZ;
    const size_t stride[3] = {YZ, Z, 1};
    uint8_t *mask = calloc(N, 1), *cs = calloc(N, 1);
    int32_t *first = malloc(N * sizeof(int32_t));
    if (!mask || !cs || !first) { free(mask); free(cs); free(first); return -1; }
    float lo[3], ext[3];
    for (int a = 0; a < 3; a++) { lo[a] = bbox[a]; ext[a] = bbox[3 + a] - bbox[a]; }

    int64_t nv = 0, nt = 0;
    for (uint32_t i = 0; i < X; i++)
        for (uint32_t j = 0; j < Y; j++)
            for (uint32_t k = 0; k < Z; k++) {
                const size_t e = i * YZ + (size_t)j * Z + k;
                const uint32_t c[3] = {i, j, k};
                const int in0 = v[e] > iso;
                uint8_t m = 0;
                for (int a = 0; a < 3; a++)
                    if (c[a] + 1 < n[a] && in0 != (v[e + stride[a]] > iso)) m |= (uint8_t)(1u << a);
                mask[e] = m;
                first[e] = (int32_t)nv;
                if (verts) {
                    float p[3];
                    for (int d = 0; d < 3; d++) p[d] = lo[d] + ((float)c[d] / (float)n[d]) * ext[d];
                    for (int a = 0; a < 3; a++) {
                        if (!(m >> a & 1)) continue;
                        const float va = v[e], vb = v[e + stride[a]];
                        const float t = fminf(fmaxf((iso - va) / (vb - va), 0.f), 1.f);
                        const float s = (float)c[a] + t;
                        float *q = verts + (size_t)(nv + __builtin_popcount(m & ((1u << a) - 1))) * 3;
                        for (int d = 0; d < 3; d++) q[d] = d == a ? lo[d] + (s / (float)n[d]) * ext[d] : p[d];
                    }
                }
                nv += __builtin_popcount(m);
                if (i + 1 < X && j + 1 < Y && k + 1 < Z) {
                    uint32_t cc = 0;
                    for (uint32_t corner = 0; corner < 8; corner++)
                        cc |= (uint32_t)(v[e + (corner & 1) * YZ + (corner >> 1 & 1) * Z + (corner >> 2 & 1)] > iso) << corner;
                    cs[e] = (uint8_t)cc;
                    nt += MC_TRI_COUNT[cc];
                }
            }
    counts[0] = (int32_t)nv;
    counts[1] = (int32_t)nt;
    if (tris) {
        size_t o = 0;
        for (size_t e = 0; e < N; e++)
            for (int q = 0; q < 3 * MC_TRI_COUNT[cs[e]]; q++) {
                const int ed = MC_TRI_TABLE[cs[e]][q], axis = ed >> 2, a = MC_EDGE_CORNERS[ed][0];
                const size_t owner = e + (a & 1) * YZ + (a >> 1 & 1) * (size_t)Z + (a >> 2 & 1);
                tris[o++] = first[owner] + __builtin_popcount(mask[owner] & ((1u << axis) - 1));
            }
    }
    free(mask); free(cs); free(first);
    return 0;
}
