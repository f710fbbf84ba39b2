// Cell -> sample point of the occupancy-grid update (nerf/mask_renderer.py:455-548), shared by the point kernel of
// occupancy.cu and the fused density sweep of field_fused.cu.
//
// The reference builds, per cascade c, `xyzs = 2 * coords.float() / (G - 1) - 1`, scales it by the PYTHON double
// `bound_c - half_grid_size` (rounded to fp32 when it meets the tensor) and adds `(rand * 2 - 1) * half_grid_size`
// (mask_renderer.py:480-487, 516-524).  occ_point() evaluates exactly those fp32 operations in that order; the two
// per-cascade scalars are computed on the host in double and rounded once (OccPoints::scale / hgs).
#pragma once
#include "common.cuh"
#include "march_device.cuh"

namespace occ {

struct OccPoints {
    const int32_t* cells;   // [C * per_cascade] Morton cell indices, or NULL: cell j of every cascade (full sweep, per_cascade = G^3)
    const float* noise;     // [C * per_cascade, 3] in [0, 1), or NULL: counter-based generator keyed by `seed`
    unsigned long long seed;
    uint32_t per_cascade, G, C;
    float scale[16];        // (float)(bound_c - bound_c / G), bound_c = min(2^c, bound)
    float hgs[16];          // (float)(bound_c / G)
};

// fills `o` for C cascades of a G^3 grid (host side; defined in occupancy.cu); INERF_OK or an argument error
int make_points(OccPoints* o, uint32_t C, uint32_t G, float bound, const int32_t* cells, uint32_t per_cascade, const float* noise, uint64_t seed);

// exclusive scan, in place, of `n_segments` consecutive runs of `per_segment` int32 block counts; the total of segment s goes
// to totals[s] (one launch on `st`, defined in occupancy.cu; also the compaction behind inerf_extract_volume)
int scan_block_counts(int32_t* counts, uint32_t per_segment, uint32_t n_segments, int32_t* totals, cudaStream_t st);

// splitmix64 finaliser over (seed, counter): 64 well-mixed bits per call, no state, no memory traffic
__device__ __forceinline__ unsigned long long mix64(unsigned long long seed, unsigned long long counter) {
    unsigned long long z = seed + (counter + 1ull) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
// three uniforms in [0, 1) with 21 bits each from one 64-bit draw
__device__ __forceinline__ void uniform3(unsigned long long seed, unsigned long long counter, float u[3]) {
    const unsigned long long z = mix64(seed, counter);
#pragma unroll
    for (int d = 0; d < 3; d++) u[d] = (float)((uint32_t)(z >> (21 * d)) & 0x1FFFFFu) * (1.0f / 2097152.0f);
}
// uniform integer in [0, n) (multiply-shift; bias < 2^-32 * n)
__device__ __forceinline__ uint32_t uniform_below(unsigned long long seed, unsigned long long counter, uint32_t n) {
    return (uint32_t)(((mix64(seed, counter) >> 32) * (unsigned long long)n) >> 32);
}

// sample s of the sweep -> point (fp32, the reference's operation order) and its flat cell index c * G^3 + morton
__device__ __forceinline__ void occ_point(const OccPoints& o, uint32_t s, float xyz[3], uint32_t& flat_index) {
    const uint32_t c = s / o.per_cascade;
    const uint32_t m = o.cells ? (uint32_t)__ldg(o.cells + s) : s - c * o.per_cascade;
    const uint32_t coord[3] = {march::morton3D_dec(m), march::morton3D_dec(m >> 1), march::morton3D_dec(m >> 2)};
    float u[3];
    if (o.noise) { u[0] = __ldg(o.noise + (size_t)s * 3); u[1] = __ldg(o.noise + (size_t)s * 3 + 1); u[2] = __ldg(o.noise + (size_t)s * 3 + 2); }
    else uniform3(o.seed, s, u);
    const float gm1 = (float)(o.G - 1);
#pragma unroll
    for (int d = 0; d < 3; d++) {
        const float unit = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, (float)coord[d]), gm1), 1.0f);   // 2 * coords.float() / (G - 1) - 1
        const float jit = __fmul_rn(__fsub_rn(__fmul_rn(u[d], 2.0f), 1.0f), o.hgs[c]);            // (rand * 2 - 1) * half_grid_size
        xyz[d] = __fadd_rn(__fmul_rn(unit, o.scale[c]), jit);
    }
    flat_index = c * o.G * o.G * o.G + m;
}

}  // namespace occ
