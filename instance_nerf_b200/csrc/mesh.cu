// Marching cubes on the GPU: a float volume v[X,Y,Z] (C order) -> a triangle mesh of the surface v = iso, in the geometry of
// inerf_volume_points (sample (i,j,k) at lo + (i,j,k) / (X,Y,Z) * (hi - lo)).  DESIGN section 4.9.
//
// Three passes over the samples, in tiles of kMcBlock consecutive samples (C order, so every load of v is coalesced along Z):
//   k_mc_count  per sample: the crossing-edge mask of the three lattice edges it owns (+x, +y, +z) and the case of the cube
//               whose lower corner it is; per tile: the vertex and triangle totals.  occ::scan_block_counts turns the two
//               total rows into exclusive tile offsets and leaves (V, F) on the device.
//   k_mc_verts  per sample: its first vertex index (tile offset + in-tile scan), kept for the triangle pass, and its vertices.
//   k_mc_tris   per cube: its triangles, each edge resolved to the vertex of the sample that owns it.
// Every output position is a prefix sum over C order: no atomics, the same bytes on every run.
#include "common.cuh"
#include "occupancy_device.cuh"

#define MC_TABLE_ATTR static __device__ const
#include "mc_table.h"

namespace {

constexpr uint32_t kMcBlock = 1024;

struct McGeom {
    uint32_t n[3];     // X, Y, Z
    uint32_t YZ;       // Y * Z
    uint32_t n_smp;    // X * Y * Z
    uint32_t n_blk;    // tiles of kMcBlock samples
};

__device__ __forceinline__ void mc_coords(const McGeom& g, uint32_t e, uint32_t c[3]) {
    c[2] = e % g.n[2];
    const uint32_t t = e / g.n[2];
    c[1] = t % g.n[1]; c[0] = t / g.n[1];
}

// Exclusive prefix of x over the CTA's threads in thread order, and the CTA total.  sm: 33 words of shared memory.
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t x, uint32_t* sm, uint32_t& total) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += up; }
    if (lane == 31) sm[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint32_t ws = sm[lane];
        uint32_t wi = ws;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t up = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= (uint32_t)o) wi += up; }
        sm[lane] = wi - ws;
        if (lane == 31) sm[32] = wi;
    }
    __syncthreads();
    const uint32_t r = sm[warp] + incl - x;
    total = sm[32];
    __syncthreads();   // sm is reused by the next tile
    return r;
}

// info[e] = crossing-edge mask (bit a: the edge from sample e along axis a) | case << 3 (0 when e is not a cube's lower corner)
__global__ void __launch_bounds__(kMcBlock) k_mc_count(const float* __restrict__ v, McGeom g, float iso, int32_t* __restrict__ info,
                                                       int32_t* __restrict__ counts) {
    __shared__ uint8_t tri_count[256];
    __shared__ uint32_t sm[33];
    if (threadIdx.x < 256) tri_count[threadIdx.x] = MC_TRI_COUNT[threadIdx.x];
    __syncthreads();
    for (uint32_t b = blockIdx.x; b < g.n_blk; b += gridDim.x) {
        const uint32_t e = b * kMcBlock + threadIdx.x;
        uint32_t mask = 0, cs = 0;
        if (e < g.n_smp) {
            uint32_t c[3];
            mc_coords(g, e, c);
            const bool hx = c[0] + 1 < g.n[0], hy = c[1] + 1 < g.n[1], hz = c[2] + 1 < g.n[2];
            const float* p = v + e;
            const uint32_t in0 = __ldg(p) > iso;
            const uint32_t inx = hx && __ldg(p + g.YZ) > iso, iny = hy && __ldg(p + g.n[2]) > iso, inz = hz && __ldg(p + 1) > iso;
            mask = (uint32_t)(hx && in0 != inx) | (uint32_t)(hy && in0 != iny) << 1 | (uint32_t)(hz && in0 != inz) << 2;
            if (hx && hy && hz) {
                cs = in0 | inx << 1 | iny << 2 | inz << 4
                   | (uint32_t)(__ldg(p + g.YZ + g.n[2]) > iso) << 3 | (uint32_t)(__ldg(p + g.YZ + 1) > iso) << 5
                   | (uint32_t)(__ldg(p + g.n[2] + 1) > iso) << 6 | (uint32_t)(__ldg(p + g.YZ + g.n[2] + 1) > iso) << 7;
            }
            info[e] = (int32_t)(mask | cs << 3);
        }
        uint32_t nv, nt;
        block_excl_scan(__popc(mask), sm, nv);
        block_excl_scan(tri_count[cs], sm, nt);
        if (threadIdx.x == 0) { counts[b] = (int32_t)nv; counts[g.n_blk + b] = (int32_t)nt; }
    }
}

// Vertex of sample e on its edge along axis a: s = c_a + t, t = clamp((iso - va) / (vb - va), 0, 1) (NaN -> 0), then the
// voxel-point formula with s for c_a.  fp32, one IEEE op each, in this order (the C oracle repeats it).
__global__ void __launch_bounds__(kMcBlock) k_mc_verts(const float* __restrict__ v, McGeom g, float lx, float ly, float lz, float ex,
                                                       float ey, float ez, float iso, const int32_t* __restrict__ info,
                                                       const int32_t* __restrict__ vert_offsets, int32_t* __restrict__ first_vert,
                                                       float* __restrict__ verts) {
    __shared__ uint32_t sm[33];
    const float lo[3] = {lx, ly, lz}, ext[3] = {ex, ey, ez};
    for (uint32_t b = blockIdx.x; b < g.n_blk; b += gridDim.x) {
        const uint32_t e = b * kMcBlock + threadIdx.x;
        const uint32_t mask = e < g.n_smp ? (uint32_t)info[e] & 7u : 0u;
        uint32_t total;
        uint32_t o = (uint32_t)vert_offsets[b] + block_excl_scan(__popc(mask), sm, total);
        if (mask) {
            first_vert[e] = (int32_t)o;   // read only where a crossing edge refers to it
            uint32_t c[3];
            mc_coords(g, e, c);
            float p[3];
#pragma unroll
            for (int d = 0; d < 3; d++) p[d] = __fadd_rn(lo[d], __fmul_rn(__fdiv_rn((float)c[d], (float)g.n[d]), ext[d]));
            const float va = __ldg(v + e);
            const uint32_t stride[3] = {g.YZ, g.n[2], 1u};
#pragma unroll
            for (int a = 0; a < 3; a++) {
                if (!(mask >> a & 1u)) continue;
                const float vb = __ldg(v + e + stride[a]);
                const float t = fminf(fmaxf(__fdiv_rn(__fsub_rn(iso, va), __fsub_rn(vb, va)), 0.f), 1.f);
                const float s = __fadd_rn((float)c[a], t);
                float* q = verts + (size_t)o * 3;
#pragma unroll
                for (int d = 0; d < 3; d++) q[d] = d == a ? __fadd_rn(lo[d], __fmul_rn(__fdiv_rn(s, (float)g.n[d]), ext[d])) : p[d];
                o++;
            }
        }
    }
}

__global__ void __launch_bounds__(kMcBlock) k_mc_tris(McGeom g, const int32_t* __restrict__ info, const int32_t* __restrict__ tri_offsets,
                                                      const int32_t* __restrict__ first_vert, int32_t* __restrict__ tris) {
    __shared__ int8_t table[256][16];
    __shared__ uint8_t tri_count[256];
    __shared__ uint32_t owner_off[12];   // edge -> offset of the sample that owns it
    __shared__ uint32_t sm[33];
    for (uint32_t i = threadIdx.x; i < 256 * 16; i += kMcBlock) table[i >> 4][i & 15] = MC_TRI_TABLE[i >> 4][i & 15];
    if (threadIdx.x < 256) tri_count[threadIdx.x] = MC_TRI_COUNT[threadIdx.x];
    if (threadIdx.x < 12) {
        const uint32_t a = MC_EDGE_CORNERS[threadIdx.x][0];
        owner_off[threadIdx.x] = (a & 1u) * g.YZ + (a >> 1 & 1u) * g.n[2] + (a >> 2 & 1u);
    }
    __syncthreads();
    for (uint32_t b = blockIdx.x; b < g.n_blk; b += gridDim.x) {
        const uint32_t e = b * kMcBlock + threadIdx.x;
        const uint32_t cs = e < g.n_smp ? (uint32_t)info[e] >> 3 : 0u;
        const uint32_t nt = tri_count[cs];
        uint32_t total;
        const size_t o = (size_t)(uint32_t)tri_offsets[b] + block_excl_scan(nt, sm, total);
        for (uint32_t k = 0; k < 3 * nt; k++) {
            const uint32_t ed = (uint32_t)table[cs][k], axis = ed >> 2;
            const uint32_t owner = e + owner_off[ed];
            const uint32_t below = (uint32_t)__ldg(info + owner) & ((1u << axis) - 1u);   // the owner's vertices on lower axes come first
            tris[o * 3 + k] = __ldg(first_vert + owner) + __popc(below);
        }
    }
}

// Every axis 2..2048 and X*Y*Z < 2^31, as the voxel grid; and V <= 3 X Y Z, F <= 5 (X-1)(Y-1)(Z-1) below 2^31 so that every
// vertex / triangle index and the device counts fit int32.
int make_mc(McGeom* g, uint32_t X, uint32_t Y, uint32_t Z) {
    const uint32_t n[3] = {X, Y, Z};
    for (int a = 0; a < 3; a++) {
        if (n[a] < 2 || n[a] > 2048) return INERF_ERR_SIZE;
        g->n[a] = n[a];
    }
    const uint64_t smp = (uint64_t)X * Y * Z, cubes = (uint64_t)(X - 1) * (Y - 1) * (Z - 1);
    if (smp >= (1ull << 31) || 3 * smp >= (1ull << 31) || 5 * cubes >= (1ull << 31)) return INERF_ERR_SIZE;
    g->YZ = Y * Z;
    g->n_smp = (uint32_t)smp;
    g->n_blk = div_up(smp, kMcBlock);
    return INERF_OK;
}

unsigned int mc_grid(const McGeom& g) {
    const unsigned int cap = (unsigned int)device_sm_count() * 2;   // 2 CTAs of 1024 threads fill an SM
    return g.n_blk < cap ? g.n_blk : cap;
}

}  // namespace

// per-sample info | per-sample first vertex | vertex tile counts | triangle tile counts
extern "C" size_t inerf_mesh_scratch_ints(uint32_t X, uint32_t Y, uint32_t Z) {
    McGeom g;
    if (make_mc(&g, X, Y, Z)) return 0;
    return (size_t)2 * g.n_smp + (size_t)2 * g.n_blk;
}

extern "C" int inerf_mesh_count(const float* v, uint32_t X, uint32_t Y, uint32_t Z, float iso, int32_t* scratch, int32_t* counts,
                                void* stream) {
    McGeom g;
    if (int e = make_mc(&g, X, Y, Z)) return e;
    INERF_REQUIRE(v); INERF_REQUIRE(scratch); INERF_REQUIRE(counts);
    cudaStream_t st = (cudaStream_t)stream;
    int32_t* tile_counts = scratch + (size_t)2 * g.n_smp;
    k_mc_count<<<mc_grid(g), kMcBlock, 0, st>>>(v, g, iso, scratch, tile_counts);
    INERF_LAUNCH_CHECK();
    return occ::scan_block_counts(tile_counts, g.n_blk, 2, counts, st);
}

extern "C" int inerf_mesh_emit(const float* v, uint32_t X, uint32_t Y, uint32_t Z, const float* bbox_host, float iso, int32_t* scratch,
                               float* verts, int32_t* tris, void* stream) {
    McGeom g;
    if (int e = make_mc(&g, X, Y, Z)) return e;
    INERF_REQUIRE(v); INERF_REQUIRE(bbox_host); INERF_REQUIRE(scratch); INERF_REQUIRE(verts); INERF_REQUIRE(tris);
    float lo[3], ext[3];
    for (int a = 0; a < 3; a++) {
        lo[a] = bbox_host[a];
        const float hi = bbox_host[3 + a];
        if (!isfinite(lo[a]) || !isfinite(hi) || !(hi > lo[a])) return INERF_ERR_SIZE;
        ext[a] = hi - lo[a];
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int32_t* info = scratch;
    int32_t* first_vert = scratch + g.n_smp;
    const int32_t* tile_offsets = scratch + (size_t)2 * g.n_smp;
    k_mc_verts<<<mc_grid(g), kMcBlock, 0, st>>>(v, g, lo[0], lo[1], lo[2], ext[0], ext[1], ext[2], iso, info, tile_offsets, first_vert, verts);
    INERF_LAUNCH_CHECK();
    k_mc_tris<<<mc_grid(g), kMcBlock, 0, st>>>(g, info, tile_offsets + g.n_blk, first_vert, tris);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}
