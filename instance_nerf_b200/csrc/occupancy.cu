// Occupancy-grid EMA update + bitfield packing without host round trips (sm_100a).
//
// Replaces the tail of NeRFMaskRenderer.update_extra_state
// (nerf/mask_renderer.py:532-540): boolean-mask indexing, torch.maximum, a
// .item() sync for the mean, then packbits (raymarching.cu:267-289).  Here:
//   launch 1: grid = max(grid * decay, tmp) where both >= 0, and the sum of
//             clamp(grid, 0) reduced in double into sum_out[0];
//   launch 2: thresh = min(sum / n_cells, density_thresh) read on the device,
//             bits packed 32 cells per thread.
// Both are pure streaming kernels: 16.125 B per cell, float4 loads.
//
// The front of the update -- which cells are re-sampled and where inside each cell (mask_renderer.py:466-527) -- is device
// code as well: the reference's meshgrid / randint / nonzero / index_put sequence (5 nested Python loops, two host syncs)
// becomes cell-index kernels below plus a point generator shared with the fused density sweep (occupancy_device.cuh,
// field_fused.cu), and mark_untrained_grid (mask_renderer.py:389-452) is one thread per cell looping over the cameras.
#include "occupancy_device.cuh"

namespace {

using occ::OccPoints;

__global__ void __launch_bounds__(256) k_fill(float* __restrict__ p, uint32_t n, float v) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = v;
}

// sweep sample s -> xyzs[s] and its flat cell index (the modular density path and the parity tests; the fused sweep
// generates the same points inside its gather warps)
__global__ void __launch_bounds__(256) k_occ_points(OccPoints o, uint32_t n, float* __restrict__ xyzs, int32_t* __restrict__ flat) {
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < n; s += gridDim.x * blockDim.x) {
        float xyz[3];
        uint32_t idx;
        occ::occ_point(o, s, xyz, idx);
        xyzs[(size_t)s * 3] = xyz[0]; xyzs[(size_t)s * 3 + 1] = xyz[1]; xyzs[(size_t)s * 3 + 2] = xyz[2];
        flat[s] = (int32_t)idx;
    }
}

// ---- partial update: which cells (mask_renderer.py:498-513) ---------------------------------------------------------
// Per cascade N uniformly random cells + N cells drawn with replacement from the currently occupied ones
// (density_grid[c] > 0).  The reference materialises `nonzero` (host sync for its size) and indexes it; here the occupied
// cells are compacted IN ORDER (= torch.nonzero order) by count -> scan -> write with the sizes left on the device.
constexpr uint32_t kOccBlock = 1024;

__global__ void __launch_bounds__(kOccBlock) k_occ_count(const float* __restrict__ grid, uint32_t cells_per_cascade, uint32_t blocks_per_cascade,
                                                         int32_t* __restrict__ block_counts) {
    const uint32_t c = blockIdx.y, b = blockIdx.x, i = b * kOccBlock + threadIdx.x;
    const bool occ_cell = i < cells_per_cascade && grid[(size_t)c * cells_per_cascade + i] > 0.f;
    const int total = __syncthreads_count(occ_cell);
    if (threadIdx.x == 0) block_counts[c * blocks_per_cascade + b] = total;
}

// one CTA per cascade: exclusive scan of its block counts in place, total -> n_occ[c]
__global__ void __launch_bounds__(1024) k_occ_scan(int32_t* __restrict__ block_counts, uint32_t blocks_per_cascade, int32_t* __restrict__ n_occ) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t carry_s;
    int32_t* bc = block_counts + (size_t)blockIdx.x * blocks_per_cascade;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (uint32_t base = 0; base < blocks_per_cascade; base += 1024) {
        const uint32_t n = base + threadIdx.x;
        const uint32_t v = n < blocks_per_cascade ? (uint32_t)bc[n] : 0u;
        uint32_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += up; }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const uint32_t ws = warp_sums[lane];
            uint32_t wi = ws;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t up = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= (uint32_t)o) wi += up; }
            warp_sums[lane] = wi - ws;
        }
        __syncthreads();
        const uint32_t excl = carry_s + warp_sums[warp] + incl - v;
        if (n < blocks_per_cascade) bc[n] = (int32_t)excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) n_occ[blockIdx.x] = (int32_t)carry_s;
}

__global__ void __launch_bounds__(kOccBlock) k_occ_compact(const float* __restrict__ grid, uint32_t cells_per_cascade, uint32_t blocks_per_cascade,
                                                           const int32_t* __restrict__ block_offsets, int32_t* __restrict__ occ_list) {
    __shared__ uint32_t warp_base[32];
    const uint32_t c = blockIdx.y, b = blockIdx.x, i = b * kOccBlock + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool occ_cell = i < cells_per_cascade && grid[(size_t)c * cells_per_cascade + i] > 0.f;
    const uint32_t bal = __ballot_sync(0xffffffffu, occ_cell);
    if (lane == 0) warp_base[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
        const uint32_t v = warp_base[lane];
        uint32_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += up; }
        warp_base[lane] = incl - v;
    }
    __syncthreads();
    if (occ_cell) {
        const uint32_t pos = (uint32_t)block_offsets[c * blocks_per_cascade + b] + warp_base[warp] + __popc(bal & ((1u << lane) - 1u));
        occ_list[(size_t)c * cells_per_cascade + pos] = (int32_t)i;
    }
}

// cells[c, 0:N] = uniform cells, cells[c, N:2N] = occupied picks.  Injected draws (parity tests): `uniform_cells` [C, N]
// Morton indices, `occ_picks` [C, N] positions in the ordered occupied list (what torch.randint(0, n_occ) returns).
// A cascade without an occupied cell repeats its uniform cells (the reference raises on randint(0, 0)).
__global__ void __launch_bounds__(256) k_occ_pick(const int32_t* __restrict__ occ_list, const int32_t* __restrict__ n_occ, uint32_t cells_per_cascade,
                                                  uint32_t N, uint32_t C, const int32_t* __restrict__ uniform_cells,
                                                  const int32_t* __restrict__ occ_picks, unsigned long long seed, int32_t* __restrict__ cells) {
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < C * N; t += gridDim.x * blockDim.x) {
        const uint32_t c = t / N, j = t - c * N;
        const uint32_t u = uniform_cells ? (uint32_t)uniform_cells[t] : occ::uniform_below(seed, 2ull * t, cells_per_cascade);
        const uint32_t n = (uint32_t)n_occ[c];
        uint32_t o = u;
        if (n > 0) {
            const uint32_t r = occ_picks ? min((uint32_t)occ_picks[t], n - 1u) : occ::uniform_below(seed, 2ull * t + 1ull, n);
            o = (uint32_t)occ_list[(size_t)c * cells_per_cascade + r];
        }
        cells[(size_t)c * 2 * N + j] = (int32_t)u;
        cells[(size_t)c * 2 * N + N + j] = (int32_t)o;
    }
}

// ---- mark_untrained_grid (mask_renderer.py:389-452) ------------------------------------------------------------------
// One thread per (cascade, cell); the camera poses ([B, 4, 4] c2w, row-major) are staged through shared memory 64 at a
// time.  cam = (p - t) @ R evaluated as an FMA chain over the world axes; a cell nobody sees gets density -1.
struct MarkParams {
    float scale[16], hgs2[16];   // (float)(bound_c - bound_c / G), (float)(2 * bound_c / G)
    float kx, ky;                 // (float)(cx / fx), (float)(cy / fy)
};
__global__ void __launch_bounds__(256) k_mark_untrained(const float* __restrict__ poses, uint32_t B, MarkParams mp, uint32_t C, uint32_t G,
                                                        float* __restrict__ grid, uint32_t* __restrict__ n_marked) {
    __shared__ float P[64][12];
    const uint32_t cells = G * G * G;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = t < C * cells;
    const uint32_t c = live ? t / cells : 0, m = live ? t - c * cells : 0;
    const float gm1 = (float)(G - 1);
    float w[3];
    const uint32_t coord[3] = {march::morton3D_dec(m), march::morton3D_dec(m >> 1), march::morton3D_dec(m >> 2)};
#pragma unroll
    for (int d = 0; d < 3; d++) w[d] = __fmul_rn(__fsub_rn(__fdiv_rn(__fmul_rn(2.0f, (float)coord[d]), gm1), 1.0f), mp.scale[c]);
    bool seen = false;
    for (uint32_t head = 0; head < B; head += 64) {
        const uint32_t nb = min(64u, B - head);
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < nb * 12; i += blockDim.x) {
            const uint32_t b = i / 12, e = i - b * 12;   // rows 0..2 of the 4x4 matrix: R | t
            P[b][e] = poses[(size_t)(head + b) * 16 + e];
        }
        __syncthreads();
        if (live && !seen) {
            for (uint32_t b = 0; b < nb; b++) {
                const float vx = __fsub_rn(w[0], P[b][3]), vy = __fsub_rn(w[1], P[b][7]), vz = __fsub_rn(w[2], P[b][11]);
                const float cx_ = __fmaf_rn(vz, P[b][8], __fmaf_rn(vy, P[b][4], __fmul_rn(vx, P[b][0])));
                const float cy_ = __fmaf_rn(vz, P[b][9], __fmaf_rn(vy, P[b][5], __fmul_rn(vx, P[b][1])));
                const float cz_ = __fmaf_rn(vz, P[b][10], __fmaf_rn(vy, P[b][6], __fmul_rn(vx, P[b][2])));
                // `cx / fx * cam_z + half_grid_size * 2`: a multiply kernel, then an add kernel -- two roundings, no FMA
                if (cz_ > 0.f && fabsf(cx_) < __fadd_rn(__fmul_rn(mp.kx, cz_), mp.hgs2[c]) && fabsf(cy_) < __fadd_rn(__fmul_rn(mp.ky, cz_), mp.hgs2[c])) { seen = true; break; }
            }
        }
    }
    if (live && !seen) grid[t] = -1.0f;
    const uint32_t cnt = __syncthreads_count(live && !seen);
    if (n_marked && threadIdx.x == 0 && cnt) atomicAdd(n_marked, cnt);
}

static void fill_cascades(float bound, uint32_t C, uint32_t G, float* scale, float* hgs, double hgs_mul) {
    for (uint32_t c = 0; c < 16; c++) {
        const double bc = c < C ? ((double)(1u << c) < (double)bound ? (double)(1u << c) : (double)bound) : 0.0;
        const double h = bc / (double)G;
        scale[c] = (float)(bc - h);
        hgs[c] = (float)(h * hgs_mul);
    }
}

__global__ void __launch_bounds__(256) k_occ_ema(float* __restrict__ grid, const float* __restrict__ tmp, uint32_t n, float decay,
                                                 double* __restrict__ sum_out) {
    double local = 0.0;
    const uint32_t n4 = n >> 2;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
        float4 g = reinterpret_cast<float4*>(grid)[i];
        const float4 t = __ldg(reinterpret_cast<const float4*>(tmp) + i);
        if (g.x >= 0 && t.x >= 0) g.x = fmaxf(__fmul_rn(g.x, decay), t.x);
        if (g.y >= 0 && t.y >= 0) g.y = fmaxf(__fmul_rn(g.y, decay), t.y);
        if (g.z >= 0 && t.z >= 0) g.z = fmaxf(__fmul_rn(g.z, decay), t.z);
        if (g.w >= 0 && t.w >= 0) g.w = fmaxf(__fmul_rn(g.w, decay), t.w);
        reinterpret_cast<float4*>(grid)[i] = g;
        local += (double)fmaxf(g.x, 0.f) + (double)fmaxf(g.y, 0.f) + (double)fmaxf(g.z, 0.f) + (double)fmaxf(g.w, 0.f);
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3u)) {
        const uint32_t i = (n & ~3u) + threadIdx.x;
        float g = grid[i];
        const float t = tmp[i];
        if (g >= 0 && t >= 0) g = fmaxf(__fmul_rn(g, decay), t);
        grid[i] = g;
        local += (double)fmaxf(g, 0.f);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    __shared__ double warp_part[8];
    if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0;
        for (int i = 0; i < 8; i++) s += warp_part[i];
        atomicAdd(sum_out, s);
    }
}

__global__ void __launch_bounds__(256) k_occ_pack(const float* __restrict__ grid, uint32_t n_cells, const double* __restrict__ sum_in,
                                                  float density_thresh, uint8_t* __restrict__ bitfield, float* __restrict__ mean_out) {
    const float mean = (float)(sum_in[0] / (double)n_cells);
    const float thresh = fminf(mean, density_thresh);
    if (mean_out && blockIdx.x == 0 && threadIdx.x == 0) mean_out[0] = mean;
    const uint32_t nwords = n_cells >> 5;
    for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += gridDim.x * blockDim.x) {
        const float4* g = reinterpret_cast<const float4*>(grid) + (size_t)w * 8;
        uint32_t bits = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const float4 v = __ldg(g + i);
            bits |= (uint32_t)(v.x > thresh) << (i * 4 + 0);
            bits |= (uint32_t)(v.y > thresh) << (i * 4 + 1);
            bits |= (uint32_t)(v.z > thresh) << (i * 4 + 2);
            bits |= (uint32_t)(v.w > thresh) << (i * 4 + 3);
        }
        reinterpret_cast<uint32_t*>(bitfield)[w] = bits;
    }
}

}  // namespace

extern "C" int inerf_occupancy_ema(float* density_grid, const float* tmp_grid, uint32_t n_cells, float decay, double* sum_out,
                                   void* stream) {
    if (n_cells == 0) return INERF_OK;
    INERF_REQUIRE(density_grid); INERF_REQUIRE(tmp_grid); INERF_REQUIRE(sum_out);
    if (((uintptr_t)density_grid & 15u) || ((uintptr_t)tmp_grid & 15u)) return INERF_ERR_ALIGN;
    const unsigned int blocks = min(div_up(max(n_cells >> 2, 1u), 256), (unsigned int)(kNumSMs * 8));
    k_occ_ema<<<blocks, 256, 0, (cudaStream_t)stream>>>(density_grid, tmp_grid, n_cells, decay, sum_out);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

extern "C" int inerf_occupancy_pack(const float* density_grid, uint32_t n_cells, const double* sum_in, float density_thresh,
                                    uint8_t* bitfield, float* mean_out, void* stream) {
    if (n_cells == 0) return INERF_OK;
    if (n_cells & 31u) return INERF_ERR_SIZE;  // C * H^3 is a multiple of 32 for every H >= 4
    INERF_REQUIRE(density_grid); INERF_REQUIRE(sum_in); INERF_REQUIRE(bitfield);
    if (((uintptr_t)density_grid & 15u) || ((uintptr_t)bitfield & 3u)) return INERF_ERR_ALIGN;
    const unsigned int blocks = min(div_up(n_cells >> 5, 256), (unsigned int)(kNumSMs * 8));
    k_occ_pack<<<blocks, 256, 0, (cudaStream_t)stream>>>(density_grid, n_cells, sum_in, density_thresh, bitfield, mean_out);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

// ---- sweep points, cell sampling, untrained-cell marking ---------------------------------------------------------------------

namespace occ {
int make_points(OccPoints* o, uint32_t C, uint32_t G, float bound, const int32_t* cells, uint32_t per_cascade, const float* noise, uint64_t seed) {
    if (C == 0 || C > 16 || G < 2 || G > 1024 || (G & (G - 1)) || !(bound > 0.f) || per_cascade == 0) return INERF_ERR_SIZE;
    if ((uint64_t)C * per_cascade >= 0x7fffffffull || (uint64_t)C * G * G * G >= 0x7fffffffull) return INERF_ERR_SIZE;
    if (cells == nullptr && per_cascade != G * G * G) return INERF_ERR_SIZE;   // a full sweep visits every cell once
    o->cells = cells; o->noise = noise; o->seed = seed; o->per_cascade = per_cascade; o->G = G; o->C = C;
    fill_cascades(bound, C, G, o->scale, o->hgs, 1.0);
    return INERF_OK;
}

int scan_block_counts(int32_t* counts, uint32_t per_segment, uint32_t n_segments, int32_t* totals, cudaStream_t st) {
    k_occ_scan<<<n_segments, 1024, 0, st>>>(counts, per_segment, totals);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}
}  // namespace occ

extern "C" int inerf_occupancy_points(uint32_t C, uint32_t G, float bound, const int32_t* cells, uint32_t per_cascade, const float* noise,
                                      uint64_t seed, float* xyzs, int32_t* flat_index, void* stream) {
    OccPoints o;
    if (int e = occ::make_points(&o, C, G, bound, cells, per_cascade, noise, seed)) return e;
    INERF_REQUIRE(xyzs); INERF_REQUIRE(flat_index);
    const uint32_t n = C * per_cascade;
    k_occ_points<<<min(div_up(n, 256), (unsigned int)(kNumSMs * 8)), 256, 0, (cudaStream_t)stream>>>(o, n, xyzs, flat_index);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

extern "C" int inerf_fill_f32(float* p, uint32_t n, float value, void* stream) {
    if (n == 0) return INERF_OK;
    INERF_REQUIRE(p);
    k_fill<<<min(div_up(n, 256), (unsigned int)(kNumSMs * 8)), 256, 0, (cudaStream_t)stream>>>(p, n, value);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

extern "C" size_t inerf_occupancy_sample_scratch_ints(uint32_t C, uint32_t G) {
    const uint64_t cells = (uint64_t)G * G * G;
    return (size_t)(C * cells + (uint64_t)C * ((cells + kOccBlock - 1) / kOccBlock) + C);   // occupied list | block counts | n_occ
}

extern "C" int inerf_occupancy_sample_cells(const float* density_grid, uint32_t C, uint32_t G, uint32_t N, const int32_t* uniform_cells,
                                            const int32_t* occ_picks, uint64_t seed, int32_t* cells, int32_t* scratch, void* stream) {
    if (C == 0 || C > 16 || G < 2 || G > 1024 || (G & (G - 1)) || N == 0) return INERF_ERR_SIZE;
    const uint64_t cpc64 = (uint64_t)G * G * G;
    if (C * cpc64 >= 0x7fffffffull || (uint64_t)C * 2 * N >= 0x7fffffffull) return INERF_ERR_SIZE;
    INERF_REQUIRE(density_grid); INERF_REQUIRE(cells); INERF_REQUIRE(scratch);
    const uint32_t cpc = (uint32_t)cpc64, bpc = (cpc + kOccBlock - 1) / kOccBlock;
    int32_t* occ_list = scratch;
    int32_t* block_counts = scratch + (size_t)C * cpc;
    int32_t* n_occ = block_counts + (size_t)C * bpc;
    cudaStream_t st = (cudaStream_t)stream;
    k_occ_count<<<dim3(bpc, C), kOccBlock, 0, st>>>(density_grid, cpc, bpc, block_counts);
    INERF_LAUNCH_CHECK();
    if (int e = occ::scan_block_counts(block_counts, bpc, C, n_occ, st)) return e;
    k_occ_compact<<<dim3(bpc, C), kOccBlock, 0, st>>>(density_grid, cpc, bpc, block_counts, occ_list);
    INERF_LAUNCH_CHECK();
    k_occ_pick<<<min(div_up((unsigned long long)C * N, 256), (unsigned int)(kNumSMs * 8)), 256, 0, st>>>(occ_list, n_occ, cpc, N, C, uniform_cells,
                                                                                                   occ_picks, seed, cells);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

extern "C" int inerf_mark_untrained_grid(const float* poses, uint32_t B, float fx, float fy, float cx, float cy, uint32_t C, uint32_t G,
                                         float bound, float* density_grid, uint32_t* n_marked, void* stream) {
    if (C == 0 || C > 16 || G < 2 || G > 1024 || (G & (G - 1)) || !(bound > 0.f) || fx == 0.f || fy == 0.f) return INERF_ERR_SIZE;
    if ((uint64_t)C * G * G * G >= 0x7fffffffull) return INERF_ERR_SIZE;
    INERF_REQUIRE(density_grid);
    if (B) INERF_REQUIRE(poses);
    MarkParams mp;
    fill_cascades(bound, C, G, mp.scale, mp.hgs2, 2.0);
    mp.kx = (float)((double)cx / (double)fx);
    mp.ky = (float)((double)cy / (double)fy);
    const uint32_t n = C * G * G * G;
    k_mark_untrained<<<div_up(n, 256), 256, 0, (cudaStream_t)stream>>>(poses, B, mp, C, G, density_grid, n_marked);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}
