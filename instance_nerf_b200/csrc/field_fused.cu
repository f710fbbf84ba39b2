// inerf_field_forward: NeRFNetwork.forward (nerf/network_mask.py:119-158) as ONE persistent kernel.
//
// Per 128-sample tile: both hash encoders gathered straight into UMMA operand tiles in shared memory
// (no [B,32] activation ever touches HBM), SH degree 4, then sigma-net, colour-net and mask-net as a chain
// of tcgen05.mma (fp16 x fp16 -> fp32 in TMEM) with TMEM->register epilogues that apply ReLU / exp / sigmoid
// and write the next layer's operand tile.  Weights (< 40 KB fp16) stay resident in shared memory for the
// life of the CTA.  (The first version -- two lock-step 256-thread CTAs per SM that overlapped gathers and MMAs only across
// CTAs -- took 3.78 ms for 7.8 M samples against 2.05 ms for the warp-specialised kernel below and was removed; DESIGN.md 4.2.)
#include <vector>

#include "field_device.cuh"
#include "occupancy_device.cuh"

namespace {

using namespace field;

// ---- gather and MLP chain as concurrent roles of ONE CTA per SM -----------------------------------------------------------
// The structure is the render kernel's (render_fused.cu) without its marcher and compositor: 16 gather warps (thread = sample
// row x 4 of the 16 levels, 64 registers) fill one of two operand stages while 8 chain warps (96 registers) run the tcgen05
// chain of the previous tile and store its results; the gather warps never wait for an epilogue.
constexpr uint32_t kWsChainT = 256, kWsGatherT = 512, kWsThreads = kWsChainT + kWsGatherT, kWsStages = 2;

struct WsCtrl {
    uint64_t a_full[kWsStages], a_empty[kWsStages], mma_bar;
    uint32_t tmem_slot;
    LevelGeom lg[16];
};
struct WsSmem {
    static constexpr uint32_t A = 0;
    static constexpr uint32_t W = A + kWsStages * kStageBytes;
    static __host__ __device__ uint32_t ctrl(uint32_t K) { return (W + weight_layout(K).total + 15u) & ~15u; }
    static __host__ __device__ uint32_t bytes(uint32_t K) { return ctrl(K) + (uint32_t)sizeof(WsCtrl) + 16u; }
};

// The CTA of the three per-sample field kernels (k_field_forward_ws, k_occupancy_density, k_extract_volume).  What differs
// between them is a Job:
//   rows(desc)                  the number of rows, read once per CTA
//   point(s, p)                 gather warps: the point of row s < rows
//   sh_row(s, smem, a_ci, row)  gather warps: the SH16 columns of the colour-net input of row s (nothing for density only)
//   tile(...)                   chain warps: the chain over one gathered stage (mlp_chain or sigma_chain, which releases the
//                               stage), then the stores of rows row0 .. row0 + 127 below n
// A parameter struct that a job indexes at run time (OccPoints' per-cascade arrays) is a __grid_constant__ kernel parameter held
// by reference: a copy inside the job would go to local memory.
template <typename Job>
__device__ __forceinline__ void ws_field_cta(const inerf_field_desc desc, const Job& job) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t K = desc.K;
    WsCtrl* ctl = reinterpret_cast<WsCtrl*>(smem + WsSmem::ctrl(K));
    const uint32_t tid = threadIdx.x;
    load_weights(smem, WsSmem::W, desc.weights, K);
    init_levels(ctl->lg, desc.offsets, desc.L, desc.S, desc.H, tid);
    if (tid == 0) {
        for (uint32_t i = 0; i < kWsStages; i++) { umma::mbar_init(&ctl->a_full[i], kWsGatherT / 32); umma::mbar_init(&ctl->a_empty[i], 1); }
        umma::mbar_init(&ctl->mma_bar, 1);
        umma::mbar_fence_init();
    }
    if (tid < 32) umma::tmem_alloc<kTmemCols>(&ctl->tmem_slot);
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem_base = ctl->tmem_slot;
    const uint32_t n = job.rows(desc);
    const uint32_t num_tiles = (n + kTile - 1) / kTile;

    if (tid < kWsChainT) {
        // ------------------------------------------------------------------------------------------------ chain --
        umma::reg_alloc<96>();
        uint32_t phase = 0, it = 0;
        auto chain_sync = [] { umma::named_sync<1, kWsChainT>(); };
        for (uint32_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
            const uint32_t sa = it % kWsStages;
            umma::mbar_wait(&ctl->a_full[sa], (it / kWsStages) & 1u);
            const uint32_t a_es = WsSmem::A + sa * kStageBytes;
            const ChainBufs bufs{a_es, a_es + kBytesEs, a_es + kBytesEs + kBytesCi, WsSmem::W};
            job.tile(desc, smem, bufs, tmem_base, &ctl->mma_bar, phase, &ctl->a_empty[sa], chain_sync, tile * kTile, n, tid);
            umma::fence_before_sync();
            chain_sync();   // TMEM and the chain's hidden tiles are reused by the next tile
        }
    } else {
        // ----------------------------------------------------------------------------------------------- gather --
        umma::reg_dealloc<64>();
        const uint32_t gt = tid - kWsChainT, row = gt & (kTile - 1), quarter = gt >> 7;
        const float inv2b = __fdiv_rn(1.0f, __fmul_rn(2.0f, desc.bound));
        const uint2* table = reinterpret_cast<const uint2*>(desc.table_packed);
        uint32_t it = 0;
        for (uint32_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
            const uint32_t sa = it % kWsStages;
            if (it >= kWsStages) umma::mbar_wait(&ctl->a_empty[sa], ((it / kWsStages) - 1u) & 1u);
            const uint32_t s = tile * kTile + row;
            if (s < n) {   // rows past the end keep stale operands: their outputs are never stored
                const uint32_t a_es = WsSmem::A + sa * kStageBytes, a_ci = a_es + kBytesEs, a_mi = a_ci + kBytesCi;
                float p[3], x01[3];
                job.point(s, p);
                bool oob = false;
#pragma unroll
                for (int d = 0; d < 3; d++) {
                    x01[d] = __fmul_rn(__fadd_rn(p[d], desc.bound), inv2b);  // grid.py:149
                    oob |= (x01[d] < 0.f || x01[d] > 1.f);
                }
                if (quarter == 0) job.sh_row(s, smem, a_ci, row);
                encode4(x01, oob, quarter * 4, ctl->lg, table, smem, a_es, a_mi, row);
            }
            umma::fence_async_smem();
            __syncwarp();
            if ((gt & 31u) == 0) umma::mbar_arrive(&ctl->a_full[sa]);   // one arrival per gather warp
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (tid < 32) umma::tmem_dealloc<kTmemCols>(tmem_base);
}

// ---- field forward: a sample stream (xyzs, dirs) -> sigma / rgb / logits, and for training the saved net inputs -------------
struct ForwardJob {
    const float* xyzs;
    const float* dirs;
    uint32_t B_rows;
    float* sigmas;
    float* rgbs;
    float* masks;
    uint4* x0_save;
    uint4* xs_save;

    __device__ __forceinline__ uint32_t rows(const inerf_field_desc& desc) const {   // rows past *n_valid: padding
        return desc.n_valid ? min(B_rows, (uint32_t)max(0, __ldg(desc.n_valid))) : B_rows;
    }
    __device__ __forceinline__ void point(uint32_t s, float p[3]) const {
#pragma unroll
        for (int d = 0; d < 3; d++) p[d] = __ldg(xyzs + (size_t)s * 3 + d);
    }
    __device__ __forceinline__ void sh_row(uint32_t s, uint8_t* smem, uint32_t a_ci, uint32_t row) const {
        sh16_to_smem(__ldg(dirs + (size_t)s * 3), __ldg(dirs + (size_t)s * 3 + 1), __ldg(dirs + (size_t)s * 3 + 2), smem, a_ci, row);
    }
    template <typename Sync>
    __device__ __forceinline__ void tile(const inerf_field_desc& desc, uint8_t* smem, const ChainBufs& bufs, uint32_t tmem_base, uint64_t* mma_bar,
                                         uint32_t& phase, uint64_t* release, Sync&& chain_sync, uint32_t row0, uint32_t B, uint32_t tid) const {
        const uint32_t K = desc.K, Kp = weight_layout(K).Kp;
        const uint32_t warp = tid >> 5, lane = tid & 31;
        const bool with_masks = masks != nullptr;
        const uint32_t orow = row0 + (warp & 3u) * 32u + lane;
        const float sigma = mlp_chain(smem, bufs, tmem_base, mma_bar, phase, K, desc.density_scale, with_masks, tid, release, chain_sync, [&](float) {
            // training: keep the mask-net input row (32 mask-table features | 15 geo | 0, fp16) for the backward pass.  The row's
            // owner wrote the geo columns itself a moment ago, and the stage is only released after the layer-0 MMAs.
            if (x0_save != nullptr && warp < 4 && orow < B) {
#pragma unroll
                for (uint32_t c = 0; c < 6; c++)
                    x0_save[(size_t)orow * 6 + c] = *reinterpret_cast<const uint4*>(smem + bufs.a_mi + umma::tile_off(tid, c * 8, kLBO, sbo_of(48)));
            }
            // stage-1 training: keep the inputs of BOTH nets -- 32 sigma-table features | SH16, geo15, 0 (fp16 [.,64])
            if (xs_save != nullptr && warp < 4 && orow < B) {
#pragma unroll
                for (uint32_t c = 0; c < 4; c++) {
                    xs_save[(size_t)orow * 8 + c] = *reinterpret_cast<const uint4*>(smem + bufs.a_es + umma::tile_off(tid, c * 8, kLBO, sbo_of(32)));
                    xs_save[(size_t)orow * 8 + 4 + c] = *reinterpret_cast<const uint4*>(smem + bufs.a_ci + umma::tile_off(tid, c * 8, kLBO, sbo_of(32)));
                }
            }
        });
        if (warp < 4) {
            float rgb[3];
            epilogue_rgb(tmem_base, rgb, tid);
            if (orow < B) {
                sigmas[orow] = sigma;
                rgbs[(size_t)orow * 3] = rgb[0]; rgbs[(size_t)orow * 3 + 1] = rgb[1]; rgbs[(size_t)orow * 3 + 2] = rgb[2];
            }
        }
        if (with_masks) {
            const uint32_t chunks = Kp / 16, c_begin = (warp >> 2) ? (chunks + 1) / 2 : 0, c_end = (warp >> 2) ? chunks : (chunks + 1) / 2;
            for (uint32_t c = c_begin; c < c_end; c++) {
                uint32_t v[16];
                umma::tmem_ld16(tmem_base + D_d + (((warp & 3u) * 32u) << 16) + c * 16, v);
                umma::tmem_ld_wait();
                if (orow < B) {
                    float* out = masks + (size_t)orow * K + c * 16;
                    if ((K & 3u) == 0 && c * 16 + 16 <= K) {
#pragma unroll
                        for (int i = 0; i < 4; i++)
                            reinterpret_cast<float4*>(out)[i] = make_float4(__half2float(__float2half_rn(__uint_as_float(v[4 * i]))),
                                                                            __half2float(__float2half_rn(__uint_as_float(v[4 * i + 1]))),
                                                                            __half2float(__float2half_rn(__uint_as_float(v[4 * i + 2]))),
                                                                            __half2float(__float2half_rn(__uint_as_float(v[4 * i + 3]))));
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; i++)
                            if (c * 16 + i < K) out[i] = __half2float(__float2half_rn(__uint_as_float(v[i])));
                    }
                }
            }
        }
    }
};

__global__ void __launch_bounds__(kWsThreads, 1) k_field_forward_ws(inerf_field_desc desc, const float* __restrict__ xyzs,
                                                                    const float* __restrict__ dirs, uint32_t B_rows,
                                                                    float* __restrict__ sigmas, float* __restrict__ rgbs,
                                                                    float* __restrict__ masks, uint4* __restrict__ x0_save,
                                                                    uint4* __restrict__ xs_save) {
    ws_field_cta(desc, ForwardJob{xyzs, dirs, B_rows, sigmas, rgbs, masks, x0_save, xs_save});
}

// ---- occupancy-grid density sweep (update_extra_state, nerf/mask_renderer.py:466-527) ------------------------------------
// tmp_grid[c, cell] = density(jittered point of the cell) * density_scale for every sample of the sweep, in ONE launch with
// the role structure above: the gather warps make each point from its cell id (Morton decode, cascade scale, jitter --
// occupancy_device.cuh) instead of reading a sample stream, the chain warps run the sigma-net only and scatter the result to
// the cell.  The reference goes through meshgrid / morton3D / rand_like / two table casts / encode / 2 GEMMs / index_put per
// (block, cascade) from 5 nested Python loops.
struct OccJob {
    const occ::OccPoints& pts;
    uint32_t n;
    float* tmp_grid;

    __device__ __forceinline__ uint32_t rows(const inerf_field_desc&) const { return n; }
    __device__ __forceinline__ void point(uint32_t s, float p[3]) const {
        uint32_t flat;
        occ::occ_point(pts, s, p, flat);
    }
    __device__ __forceinline__ void sh_row(uint32_t, uint8_t*, uint32_t, uint32_t) const {}
    template <typename Sync>
    __device__ __forceinline__ void tile(const inerf_field_desc& desc, uint8_t* smem, const ChainBufs& bufs, uint32_t tmem_base, uint64_t* mma_bar,
                                         uint32_t& phase, uint64_t* release, Sync&& chain_sync, uint32_t row0, uint32_t, uint32_t tid) const {
        const float sigma = sigma_chain(smem, bufs, tmem_base, mma_bar, phase, desc.K, tid, release, chain_sync);
        const uint32_t s = row0 + tid;
        if (tid < kTile && s < n) {
            const uint32_t c = s / pts.per_cascade;
            const uint32_t m = pts.cells ? (uint32_t)__ldg(pts.cells + s) : s - c * pts.per_cascade;
            tmp_grid[(size_t)c * pts.G * pts.G * pts.G + m] = __fmul_rn(sigma, desc.density_scale);   // `sigmas *= self.density_scale`
        }
    }
};

__global__ void __launch_bounds__(kWsThreads, 1) k_occupancy_density(inerf_field_desc desc, const __grid_constant__ occ::OccPoints pts, uint32_t n,
                                                                     float* __restrict__ tmp_grid) {
    ws_field_cta(desc, OccJob{pts, n, tmp_grid});
}

// ---- volume extraction (inerf_volume_points / inerf_extract_volume) ---------------------------------------------------------
// The fields on an X x Y x Z voxel grid in the geometry of inerf_project_labels.  Voxels are enumerated in C order, so a tile
// of the fused kernel is 128 consecutive voxels along Z and a voxel's index in that order is its output index (coalesced stores,
// no padding rows; the 4 x 4 x 8-brick alternative and its open A/B: DESIGN.md 4.8).
struct VolGeom {
    float lo[3], ext[3];   // bbox lo, hi - lo (fp32)
    uint32_t n[3];         // X, Y, Z
    uint32_t n_vox;        // X * Y * Z
    // occupancy grid (bits == NULL: every voxel is live); the fields of march::Walk that cell_index reads
    const uint8_t* bits;
    float bound, rbound, Hf, Hm1, H3;
    uint32_t H3i;
    int C;
};

// C-order index -> voxel (i, j, k)
__device__ __forceinline__ void vol_voxel(const VolGeom& g, uint32_t e, uint32_t v[3]) {
    v[2] = e % g.n[2];
    const uint32_t t = e / g.n[2];
    v[1] = t % g.n[1]; v[0] = t / g.n[1];
}

// p = lo + ((float)i / (float)X) * (hi - lo) per axis (grid_pts_coord, project_3d_masks.py:72-83)
__device__ __forceinline__ void vol_point(const VolGeom& g, const uint32_t v[3], float p[3]) {
#pragma unroll
    for (int d = 0; d < 3; d++) p[d] = __fadd_rn(g.lo[d], __fmul_rn(__fdiv_rn((float)v[d], (float)g.n[d]), g.ext[d]));
}

// the occupancy bit the marcher tests for a sample at p with dt = 0 (march::Walk::eval_cell; p lies inside [-bound, bound]^3)
__device__ __forceinline__ bool vol_live(const VolGeom& g, const float p[3]) {
    if (g.bits == nullptr) return true;
    const int level = march::clamped_exponent(fmaxf(fabsf(p[0]), fmaxf(fabsf(p[1]), fabsf(p[2]))), g.C);
    float mip_bound;
    int nx, ny, nz;
    const uint32_t idx = march::cell_index(p[0], p[1], p[2], level, g.bound, g.rbound, g.Hf, g.Hm1, g.H3i, g.H3, mip_bound, nx, ny, nz);
    return (__ldg(g.bits + (idx >> 3)) >> (idx & 7u)) & 1u;
}

__global__ void __launch_bounds__(256) k_volume_points(VolGeom g, float* __restrict__ xyzs, uint8_t* __restrict__ occupied) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < g.n_vox; i += gridDim.x * blockDim.x) {
        uint32_t v[3];
        float p[3];
        vol_voxel(g, i, v);
        vol_point(g, v, p);
        xyzs[(size_t)i * 3] = p[0]; xyzs[(size_t)i * 3 + 1] = p[1]; xyzs[(size_t)i * 3 + 2] = p[2];
        if (occupied) occupied[i] = vol_live(g, p) ? 1 : 0;
    }
}

// Occupancy pre-pass (bitfield != NULL): count -> scan (occ::scan_block_counts) -> compact, as inerf_occupancy_sample_cells.
// The compaction writes the indices of the live voxels in order and the zero outputs of the empty ones.  Both passes evaluate
// each voxel's point and cell (a few dozen ALU ops and one L2-resident byte) rather than keep a flag per voxel in HBM.
constexpr uint32_t kVolBlock = 1024;

__device__ __forceinline__ bool vol_index_live(const VolGeom& g, uint32_t e) {
    if (e >= g.n_vox) return false;
    uint32_t v[3];
    float p[3];
    vol_voxel(g, e, v);
    vol_point(g, v, p);
    return vol_live(g, p);
}

__global__ void __launch_bounds__(kVolBlock) k_vol_count(VolGeom g, int32_t* __restrict__ block_counts) {
    const bool live = vol_index_live(g, blockIdx.x * kVolBlock + threadIdx.x);
    const int total = __syncthreads_count(live);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kVolBlock) k_vol_compact(VolGeom g, const int32_t* __restrict__ block_offsets, int32_t* __restrict__ live_ids,
                                                           float* __restrict__ sigma, float* __restrict__ rgb, int32_t* __restrict__ label) {
    __shared__ uint32_t warp_base[32];
    const uint32_t e = blockIdx.x * kVolBlock + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool live = vol_index_live(g, e);
    const uint32_t bal = __ballot_sync(0xffffffffu, live);
    if (lane == 0) warp_base[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
        const uint32_t c = warp_base[lane];
        uint32_t incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += up; }
        warp_base[lane] = incl - c;
    }
    __syncthreads();
    if (live) {
        live_ids[(uint32_t)block_offsets[blockIdx.x] + warp_base[warp] + __popc(bal & ((1u << lane) - 1u))] = (int32_t)e;
    } else if (e < g.n_vox) {
        if (sigma) sigma[e] = 0.f;
        if (rgb) { rgb[(size_t)e * 3] = 0.f; rgb[(size_t)e * 3 + 1] = 0.f; rgb[(size_t)e * 3 + 2] = 0.f; }
        if (label) label[e] = 0;
    }
}

// The fused extraction: the per-sample field CTA with a voxel front and an argmax epilogue.  The gather warps turn row s into a
// voxel (live_ids[s], or voxel s when every voxel is evaluated) and its point, and gather both tables and the SH row of the one
// view direction; the chain warps run the full mlp_chain (mask-net only when labels are wanted); warps 0..3, which own TMEM
// lanes 0..127, take sigma, rgb and the argmax over the Kp logit columns and store sigma / rgb / label.  Nothing [n, K]-shaped
// leaves the SM.  With live_ids the tile loop stops at the device-side live count (*n_live_in), the way desc.n_valid bounds
// the training forward.
struct ExtractJob {
    VolGeom g;
    const int32_t* live_ids;
    const int32_t* n_live_in;
    float vx, vy, vz, sigma_thresh;
    float* sigma_out;
    float* rgb_out;
    int32_t* label_out;
    int32_t* n_live_out;

    __device__ __forceinline__ uint32_t rows(const inerf_field_desc&) const {   // block 0 also reports the count
        const uint32_t n = live_ids ? (uint32_t)max(0, __ldg(n_live_in)) : g.n_vox;
        if (n_live_out && blockIdx.x == 0 && threadIdx.x == 0) *n_live_out = (int32_t)n;
        return n;
    }
    __device__ __forceinline__ void point(uint32_t s, float p[3]) const {
        uint32_t v[3];
        vol_voxel(g, live_ids ? (uint32_t)__ldg(live_ids + s) : s, v);
        vol_point(g, v, p);
    }
    __device__ __forceinline__ void sh_row(uint32_t, uint8_t* smem, uint32_t a_ci, uint32_t row) const { sh16_to_smem(vx, vy, vz, smem, a_ci, row); }
    template <typename Sync>
    __device__ __forceinline__ void tile(const inerf_field_desc& desc, uint8_t* smem, const ChainBufs& bufs, uint32_t tmem_base, uint64_t* mma_bar,
                                         uint32_t& phase, uint64_t* release, Sync&& chain_sync, uint32_t row0, uint32_t n, uint32_t tid) const {
        const uint32_t K = desc.K, Kp = weight_layout(K).Kp;
        const uint32_t warp = tid >> 5;
        const bool with_masks = label_out != nullptr;
        const float sigma = mlp_chain(smem, bufs, tmem_base, mma_bar, phase, K, desc.density_scale, with_masks, tid, release, chain_sync, [](float) {});
        if (warp < 4) {   // thread tid owns tile row tid
            float rgb[3];
            epilogue_rgb(tmem_base, rgb, tid);
            uint32_t arg = 0;
            if (with_masks) {
                // argmax over the fp16-rounded logits inerf_field_forward stores; the lowest index wins a tie
                float best = 0.f;
                for (uint32_t c = 0; c < Kp / 16; c++) {
                    uint32_t v[16];
                    umma::tmem_ld16(tmem_base + D_d + ((warp * 32u) << 16) + c * 16, v);
                    umma::tmem_ld_wait();
#pragma unroll
                    for (uint32_t i = 0; i < 16; i++) {
                        const uint32_t k = c * 16 + i;
                        const float l = __half2float(__float2half_rn(__uint_as_float(v[i])));
                        if (k < K && (k == 0 || l > best)) { best = l; arg = k; }
                    }
                }
            }
            const uint32_t s = row0 + tid;
            if (s < n) {
                const uint32_t o = live_ids ? (uint32_t)__ldg(live_ids + s) : s;
                if (sigma_out) sigma_out[o] = sigma;
                if (rgb_out) { rgb_out[(size_t)o * 3] = rgb[0]; rgb_out[(size_t)o * 3 + 1] = rgb[1]; rgb_out[(size_t)o * 3 + 2] = rgb[2]; }
                if (label_out) label_out[o] = sigma >= sigma_thresh ? (int32_t)arg + 1 : 0;
            }
        }
    }
};

__global__ void __launch_bounds__(kWsThreads, 1) k_extract_volume(inerf_field_desc desc, VolGeom g, const int32_t* __restrict__ live_ids,
                                                                  const int32_t* __restrict__ n_live_in, float vx, float vy, float vz,
                                                                  float sigma_thresh, float* __restrict__ sigma_out, float* __restrict__ rgb_out,
                                                                  int32_t* __restrict__ label_out, int32_t* __restrict__ n_live_out) {
    ws_field_cta(desc, ExtractJob{g, live_ids, n_live_in, vx, vy, vz, sigma_thresh, sigma_out, rgb_out, label_out, n_live_out});
}

// fp32 / fp16 embeddings of both encoders -> interleaved fp16 (sigma.c0, sigma.c1, mask.c0, mask.c1), one pass
template <typename T>
__global__ void k_pack_tables(const T* __restrict__ es, const T* __restrict__ em, uint64_t n, uint2* __restrict__ out) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        __half2 a, b;
        if constexpr (std::is_same<T, float>::value) {
            const float2 fa = reinterpret_cast<const float2*>(es)[i], fb = reinterpret_cast<const float2*>(em)[i];
            a = __floats2half2_rn(fa.x, fa.y); b = __floats2half2_rn(fb.x, fb.y);
        } else {
            a = reinterpret_cast<const __half2*>(es)[i]; b = reinterpret_cast<const __half2*>(em)[i];
        }
        out[i] = make_uint2(h2_bits(a), h2_bits(b));
    }
}

int validate_desc(const inerf_field_desc* d) {
    INERF_REQUIRE(d);
    INERF_REQUIRE(d->table_packed); INERF_REQUIRE(d->offsets); INERF_REQUIRE(d->weights);
    if (d->L != 16 || d->K == 0 || d->K > 64 || d->H == 0 || !(d->bound > 0.f)) return INERF_ERR_UNSUPPORTED;
    if (((uintptr_t)d->weights & 15u) || ((uintptr_t)d->table_packed & 7u)) return INERF_ERR_ALIGN;
    return INERF_OK;
}

// host-side checks of a volume request and its geometry (bits != NULL: with the occupancy grid C x H^3)
int make_vol(VolGeom* g, const float* bbox, uint32_t X, uint32_t Y, uint32_t Z, float bound, const uint8_t* bits, uint32_t C, uint32_t H) {
    INERF_REQUIRE(bbox);
    const uint32_t n[3] = {X, Y, Z};
    for (int a = 0; a < 3; a++) {
        if (n[a] == 0 || n[a] > 2048) return INERF_ERR_SIZE;
        const float lo = bbox[a], hi = bbox[3 + a];
        if (!(hi > lo) || !(lo >= -bound) || !(hi <= bound)) return INERF_ERR_SIZE;
        g->lo[a] = lo;
        g->ext[a] = hi - lo;
        g->n[a] = n[a];
    }
    if ((uint64_t)X * Y * Z >= (1ull << 31)) return INERF_ERR_SIZE;
    g->n_vox = X * Y * Z;
    g->bits = bits;
    g->bound = bound;
    g->rbound = 1.0f / bound;
    if (bits) {   // the marcher's grid: C cascades of H^3 cells, H a power of two with 10-bit Morton coordinates
        if (C == 0 || C > 16 || H < 2 || H > 1024 || (H & (H - 1)) || (uint64_t)C * H * H * H >= (1ull << 32)) return INERF_ERR_SIZE;
        g->C = (int)C;
        g->Hf = (float)H;
        g->Hm1 = (float)(H - 1);
        g->H3 = (float)(H * H * H);
        g->H3i = ((uint64_t)C * H * H * H <= (1ull << 24)) ? H * H * H : 0u;
    }
    return INERF_OK;
}

}  // namespace

namespace field {
int validate(const inerf_field_desc* d) { return validate_desc(d); }
}

extern "C" int inerf_field_pack_tables(const void* emb_sigma, const void* emb_mask, int dtype, uint64_t n_entries, void* packed,
                                       void* stream) {
    INERF_REQUIRE(emb_sigma); INERF_REQUIRE(emb_mask); INERF_REQUIRE(packed);
    if (n_entries == 0) return INERF_OK;
    if (((uintptr_t)packed & 7u) || ((uintptr_t)emb_sigma & 7u) || ((uintptr_t)emb_mask & 7u)) return INERF_ERR_ALIGN;
    const unsigned grid = 8 * kNumSMs;
    if (dtype == INERF_F32) k_pack_tables<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)emb_sigma, (const float*)emb_mask, n_entries, (uint2*)packed);
    else if (dtype == INERF_F16) k_pack_tables<__half><<<grid, 256, 0, (cudaStream_t)stream>>>((const __half*)emb_sigma, (const __half*)emb_mask, n_entries, (uint2*)packed);
    else return INERF_ERR_UNSUPPORTED;
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

extern "C" size_t inerf_field_weights_bytes(uint32_t K) { return (K == 0 || K > 64) ? 0 : field::weight_layout(K).total; }

static int field_forward_impl(const inerf_field_desc* desc, const float* xyzs, const float* dirs, uint32_t B, float* sigmas, float* rgbs,
                              float* masks, void* x0_save, void* stream, void* xs_save = nullptr) {
    if (int e = validate_desc(desc)) return e;
    if (B == 0) return INERF_OK;
    INERF_REQUIRE(xyzs); INERF_REQUIRE(dirs); INERF_REQUIRE(sigmas); INERF_REQUIRE(rgbs);
    if (x0_save && (((uintptr_t)x0_save & 15u) || masks == nullptr)) return INERF_ERR_ALIGN;
    if (xs_save && ((uintptr_t)xs_save & 15u)) return INERF_ERR_ALIGN;
    return launch_persistent(k_field_forward_ws, B, kWsThreads, WsSmem::bytes(desc->K), (cudaStream_t)stream, *desc, xyzs, dirs, B, sigmas, rgbs,
                             masks, (uint4*)x0_save, (uint4*)xs_save);
}

extern "C" int inerf_occupancy_density(const inerf_field_desc* desc, uint32_t C, uint32_t G, const int32_t* cells, uint32_t per_cascade,
                                       const float* noise, uint64_t seed, float* tmp_grid, void* stream) {
    if (int e = validate_desc(desc)) return e;
    occ::OccPoints pts;
    if (int e = occ::make_points(&pts, C, G, desc->bound, cells, per_cascade, noise, seed)) return e;
    INERF_REQUIRE(tmp_grid);
    const uint32_t n = C * per_cascade;
    return launch_persistent(k_occupancy_density, n, kWsThreads, WsSmem::bytes(desc->K), (cudaStream_t)stream, *desc, pts, n, tmp_grid);
}

extern "C" int inerf_field_forward(const inerf_field_desc* desc, const float* xyzs, const float* dirs, uint32_t B, float* sigmas,
                                   float* rgbs, float* masks, void* stream) {
    return field_forward_impl(desc, xyzs, dirs, B, sigmas, rgbs, masks, nullptr, stream);
}

extern "C" int inerf_field_forward_train(const inerf_field_desc* desc, const float* xyzs, const float* dirs, uint32_t B, float* sigmas,
                                         float* rgbs, float* masks, void* x0_save, void* stream) {
    INERF_REQUIRE(x0_save);
    return field_forward_impl(desc, xyzs, dirs, B, sigmas, rgbs, masks, x0_save, stream);
}

// Stage-1 (RGB-sigma) training forward: sigma / rgb as inerf_field_forward with the instance head off, plus the saved inputs of
// the sigma and colour nets for inerf_field_backward_rgb.
extern "C" int inerf_field_forward_train_rgb(const inerf_field_desc* desc, const float* xyzs, const float* dirs, uint32_t B, float* sigmas,
                                             float* rgbs, void* xs_save, void* stream) {
    INERF_REQUIRE(xs_save);
    return field_forward_impl(desc, xyzs, dirs, B, sigmas, rgbs, nullptr, nullptr, stream, xs_save);
}

extern "C" int inerf_volume_points(const float* bbox_host, uint32_t X, uint32_t Y, uint32_t Z, const uint8_t* bitfield, uint32_t C, uint32_t H,
                                   float bound, float* xyzs, uint8_t* occupied, void* stream) {
    if (!(bound > 0.f)) return INERF_ERR_SIZE;
    VolGeom g;
    if (int e = make_vol(&g, bbox_host, X, Y, Z, bound, bitfield, C, H)) return e;
    INERF_REQUIRE(xyzs);
    k_volume_points<<<min(div_up((unsigned long long)X * Y * Z, 256), (unsigned int)(kNumSMs * 8)), 256, 0, (cudaStream_t)stream>>>(g, xyzs, occupied);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

// live ids (one per enumerated voxel) | block counts of the pre-pass | live count
extern "C" size_t inerf_extract_scratch_ints(uint32_t X, uint32_t Y, uint32_t Z) {
    if (X == 0 || Y == 0 || Z == 0 || X > 2048 || Y > 2048 || Z > 2048 || (uint64_t)X * Y * Z >= (1ull << 31)) return 0;
    const uint64_t n = (uint64_t)X * Y * Z;
    return (size_t)(n + (n + kVolBlock - 1) / kVolBlock + 1);
}

extern "C" int inerf_extract_volume(const inerf_field_desc* desc, const float* bbox_host, uint32_t X, uint32_t Y, uint32_t Z, const uint8_t* bitfield,
                                    uint32_t C, uint32_t H, const float* view_dir_host, float sigma_thresh, float* sigma, float* rgb, int32_t* label,
                                    int32_t* scratch, int32_t* n_live, void* stream) {
    if (int e = validate_desc(desc)) return e;   // K >= 1: a label request always has logits to take the argmax of
    VolGeom g;
    if (int e = make_vol(&g, bbox_host, X, Y, Z, desc->bound, bitfield, C, H)) return e;
    if (sigma == nullptr && rgb == nullptr && label == nullptr) return INERF_ERR_NULL;
    if (rgb) INERF_REQUIRE(view_dir_host);
    if (bitfield) INERF_REQUIRE(scratch);
    const float vd[3] = {view_dir_host ? view_dir_host[0] : 0.f, view_dir_host ? view_dir_host[1] : 0.f, view_dir_host ? view_dir_host[2] : 1.f};
    cudaStream_t st = (cudaStream_t)stream;
    const int32_t* live_ids = nullptr;
    const int32_t* n_live_in = nullptr;
    if (bitfield) {
        const uint32_t nblk = div_up(g.n_vox, kVolBlock);
        int32_t* counts = scratch + g.n_vox;
        k_vol_count<<<nblk, kVolBlock, 0, st>>>(g, counts);
        INERF_LAUNCH_CHECK();
        if (int e = occ::scan_block_counts(counts, nblk, 1, counts + nblk, st)) return e;
        k_vol_compact<<<nblk, kVolBlock, 0, st>>>(g, counts, scratch, sigma, rgb, label);
        INERF_LAUNCH_CHECK();
        live_ids = scratch;
        n_live_in = counts + nblk;
    }
    return launch_persistent(k_extract_volume, g.n_vox, kWsThreads, WsSmem::bytes(desc->K), st, *desc, g, live_ids, n_live_in, vd[0], vd[1], vd[2],
                             sigma_thresh, sigma, rgb, label, n_live);
}
