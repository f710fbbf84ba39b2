// inerf_field_backward_mask: backward of the instance head for the instance-field training stage, ONE persistent launch.
//
// In that stage (MaskTrainer, nerf/utils.py:1242-1246) the sigma / colour nets and their table are frozen; the trainable
// part is mask_net (47->64->64->K, network_mask.py:84-92) and encoder_mask's hash table.  Given dL/dlogits per sample
// (what composite_rays_with_masks_train_backward produces, raymarching.cu:828-940) the reference runs, through autograd,
// 6 cuBLAS GEMMs + 2 ReLU-backward kernels + 1 cat-backward + kernel_grid_backward (gridencoder.cu:245-337) + a
// whole-table zero + cast.  Here, per 128-sample tile and all on tcgen05 (fp16 operands, fp32 accumulators in TMEM):
//
//   recompute  H1 = relu(X0 W0^T), H2 = relu(H1 W1^T)          (X0 = saved mask-net input row, fp16 [.,48])
//   dX chain   dH2 = (dY W2) . [H2>0],  dH1 = (dH2 W1) . [H1>0],  dF = dH1 W0[:, :32]
//   dW         [dY|dH2]^T [H2|H1] -> dW2, dW1 ;  [dH1|0]^T X0 -> dW0    accumulated ACROSS tiles in TMEM (the operand tiles
//              are read as MN-major, so no transposed copies are written); one atomicAdd pass per CTA at the end
//   scatter    dF (32 feature grads / sample) -> 16 levels x 8 corners float2 atomics into the fp32 table gradient.
//
// Gradients w.r.t. the geo features (X0 columns 32..46) are not produced: sigma_net is frozen in this stage.
#include <cstring>

#include "field_device.cuh"

namespace {

using namespace field;

struct BwdWeights {   // byte offsets inside the packed backward blob (all B operands, K-major)
    static constexpr uint32_t w0 = 0;                  // [64 x 48]  W0[o][j]            (recompute layer 0)
    static constexpr uint32_t w1 = w0 + 64 * 48 * 2;   // [64 x 64]  W1[o][j]            (recompute layer 1)
    static constexpr uint32_t w2t = w1 + 64 * 64 * 2;  // [64 x 64]  (n=j, k=o) = W2[o][j], o >= K zero
    static constexpr uint32_t w1t = w2t + 64 * 64 * 2; // [64 x 64]  (n=j, k=o) = W1[o][j]
    static constexpr uint32_t w0t = w1t + 64 * 64 * 2; // [32 x 64]  (n=j, k=o) = W0[o][j], j < 32 (mask-table features only)
    static constexpr uint32_t total = w0t + 32 * 64 * 2;
};

struct BSmem {
    static constexpr uint32_t TG = 0;                      // [128 x 128]  dY (64, cols >= K zero) | dH2 (64)
    static constexpr uint32_t TH = TG + kTile * 128 * 2;   // [128 x 128]  H2 (64) | H1 (64)
    static constexpr uint32_t TG2 = TH + kTile * 128 * 2;  // [128 x 128]  dH1 (64) | zeros (64)
    static constexpr uint32_t TX = TG2 + kTile * 128 * 2;  // [128 x 48]   X0
    static constexpr uint32_t W = TX + kTile * 48 * 2;
    static constexpr uint32_t DF = W + BwdWeights::total;      // 2 x [128 x 32] fp32: dF handed from the chain to the scatter warps
    static constexpr uint32_t MISC = DF + 2 * kTile * 32 * 4; // LevelGeom[16] | mbarrier | tmem slot | df_full[2] | df_empty[2]
    static constexpr uint32_t bytes = MISC + 16 * sizeof(LevelGeom) + 64;
};
// Scatter role: 16 warps, thread = (row, 4 levels), with setmaxnreg 104 (chain) / 64 (scatter) -- inside the CTA's own
// 768 x 80 register allocation, which is all setmaxnreg can redistribute (a 112 / 72 split exceeds it and hangs in
// setmaxnreg.inc, DESIGN.md section 4.4).  Measured on B200 for 7.8 M samples: 8 scatter warps x 8 levels at 127 registers
// 5.02 ms -> 16 warps 4.79 ms -> + 16-byte REDs for x-neighbour pairs 4.24 ms.
constexpr uint32_t kBwdChainT = 256, kBwdScatterT = 512, kBwdThreads = kBwdChainT + kBwdScatterT;
constexpr uint32_t kScatLevels = 16 / (kBwdScatterT / kTile);   // levels per scatter thread
// scatter thread (row, q) owns levels q, q + 4, q + 8, q + 12
__host__ __device__ constexpr uint32_t scat_level(uint32_t q, uint32_t li) { return q + li * (16 / kScatLevels); }
constexpr uint32_t kBwdRegsChain = 104, kBwdRegsScatter = 64;
static_assert(kBwdChainT * kBwdRegsChain + kBwdScatterT * kBwdRegsScatter <= kBwdThreads * 80, "setmaxnreg budget exceeds the CTA's allocation");
constexpr uint32_t kSbo128 = sbo_of(128), kSbo64 = sbo_of(64), kSbo48 = sbo_of(48);
// TMEM columns (512 allocated: one CTA per SM)
constexpr uint32_t T_a = 0, T_b = 64, T_x = 128, T_w1 = 160, T_w0 = 288, kBwdTmemCols = 512;

struct BwdParams {
    const float* xyzs;          // [B, 3]
    const uint4* x0;            // fp16 [B, 48] as 6 x 16 B per row
    const float* grad_logits;   // [B, K]
    uint32_t B;
    float2* grad_table;         // fp32 [T, 2] (encoder_mask.embeddings.grad), accumulated
    float* grad_w0;             // [64, 47]
    float* grad_w1;             // [64, 64]
    float* grad_w2;             // [K, 64]
    const void* weights;        // packed backward blob
};

// 32 TMEM columns -> ReLU -> fp16 -> 4 chunks of a 128-column tile; returns the 32 "value > 0" bits
__device__ __forceinline__ uint32_t epi_relu32(uint32_t taddr, uint8_t* smem, uint32_t tile_off0, uint32_t row, uint32_t col0) {
    uint32_t v[2][16];
    umma::tmem_ld16(taddr, v[0]);
    umma::tmem_ld16(taddr + 16, v[1]);
    umma::tmem_ld_wait();
    uint32_t mask = 0;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        uint32_t p[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            p[i] = cvt_relu_f16x2(__uint_as_float(v[h][2 * i]), __uint_as_float(v[h][2 * i + 1]));
            mask |= ((p[i] & 0xffffu) ? 1u : 0u) << (h * 16 + 2 * i);
            mask |= ((p[i] >> 16) ? 1u : 0u) << (h * 16 + 2 * i + 1);
        }
        const uint32_t k = col0 + h * 16;
        *reinterpret_cast<uint4*>(smem + tile_off0 + umma::tile_off(row, k, kLBO, kSbo128)) = make_uint4(p[0], p[1], p[2], p[3]);
        *reinterpret_cast<uint4*>(smem + tile_off0 + umma::tile_off(row, k + 8, kLBO, kSbo128)) = make_uint4(p[4], p[5], p[6], p[7]);
    }
    return mask;
}

// same, into a tile whose 8-row groups are `sbo` bytes apart
__device__ __forceinline__ uint32_t epi_relu_to(uint32_t taddr, uint8_t* smem, uint32_t tile_off0, uint32_t sbo, uint32_t row, uint32_t col0) {
    uint32_t v[2][16];
    umma::tmem_ld16(taddr, v[0]);
    umma::tmem_ld16(taddr + 16, v[1]);
    umma::tmem_ld_wait();
    uint32_t mask = 0;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        uint32_t p[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            p[i] = cvt_relu_f16x2(__uint_as_float(v[h][2 * i]), __uint_as_float(v[h][2 * i + 1]));
            mask |= ((p[i] & 0xffffu) ? 1u : 0u) << (h * 16 + 2 * i);
            mask |= ((p[i] >> 16) ? 1u : 0u) << (h * 16 + 2 * i + 1);
        }
        const uint32_t k = col0 + h * 16;
        *reinterpret_cast<uint4*>(smem + tile_off0 + umma::tile_off(row, k, kLBO, sbo)) = make_uint4(p[0], p[1], p[2], p[3]);
        *reinterpret_cast<uint4*>(smem + tile_off0 + umma::tile_off(row, k + 8, kLBO, sbo)) = make_uint4(p[4], p[5], p[6], p[7]);
    }
    return mask;
}

// 32 TMEM columns . mask -> fp16 -> 4 chunks of a 128-column tile
__device__ __forceinline__ void epi_masked32(uint32_t taddr, uint32_t mask, uint8_t* smem, uint32_t tile_off0, uint32_t row, uint32_t col0) {
    uint32_t v[2][16];
    umma::tmem_ld16(taddr, v[0]);
    umma::tmem_ld16(taddr + 16, v[1]);
    umma::tmem_ld_wait();
#pragma unroll
    for (int h = 0; h < 2; h++) {
        uint32_t p[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const float a = ((mask >> (h * 16 + 2 * i)) & 1u) ? __uint_as_float(v[h][2 * i]) : 0.f;
            const float b = ((mask >> (h * 16 + 2 * i + 1)) & 1u) ? __uint_as_float(v[h][2 * i + 1]) : 0.f;
            p[i] = h2_bits(__floats2half2_rn(a, b));
        }
        const uint32_t k = col0 + h * 16;
        *reinterpret_cast<uint4*>(smem + tile_off0 + umma::tile_off(row, k, kLBO, kSbo128)) = make_uint4(p[0], p[1], p[2], p[3]);
        *reinterpret_cast<uint4*>(smem + tile_off0 + umma::tile_off(row, k + 8, kLBO, kSbo128)) = make_uint4(p[4], p[5], p[6], p[7]);
    }
}

// ---- scatter role (shared by the instance-stage and the stage-1 backward kernels) ------------------------------------------------
// 16 warps, thread = (row, 4 interleaved levels): takes the 32 feature gradients of a sample from the double-buffered fp32 tile
// the chain warps fill and adds w * g to the 8 corners of each of its levels in the fp32 table gradient.
__device__ __forceinline__ void scatter_role(const inerf_field_desc& desc, const float* __restrict__ xyzs, float2* __restrict__ grad_table,
                                             const LevelGeom* lg, const uint8_t* df_tiles, uint64_t* df_full, uint64_t* df_empty,
                                             uint32_t num_tiles, uint32_t B_eff, uint32_t rt) {
    const uint32_t lane = rt & 31, row = rt & (kTile - 1), half = rt >> 7;
    const float inv2b = __fdiv_rn(1.0f, __fmul_rn(2.0f, desc.bound));
    uint32_t it = 0;
    for (uint32_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
        const uint32_t s = tile * kTile + row;
        const bool live = s < B_eff;
        const uint32_t db = it & 1u;
        umma::mbar_wait(&df_full[db], (it >> 1) & 1u);
        uint32_t v[2 * kScatLevels];
        {
            // levels interleaved over the scatter threads (scat_level): every warp gets run-reduced coarse levels AND RED-heavy fine
            // ones.  With contiguous level groups only the 8 warps of the fine levels issued REDs, at 46 % of the measured RED
            // rate, while the other 8 warps waited: 3.74 -> 3.66 ms; without any scatter the kernel takes 1.28 ms (DESIGN.md 4.4).
            const float* src = reinterpret_cast<const float*>(df_tiles) + db * (kTile * 32) + row;
#pragma unroll
            for (uint32_t li = 0; li < kScatLevels; li++) {
                v[2 * li] = __float_as_uint(src[(2 * scat_level(half, li)) * kTile]);
                v[2 * li + 1] = __float_as_uint(src[(2 * scat_level(half, li) + 1) * kTile]);
            }
        }
        umma::mbar_arrive(&df_empty[db]);   // the values are in registers: the chain may refill this buffer
        {
            // Consecutive rows of a tile are consecutive samples of the same ray (the stream is sorted by ray and by t), so on the
            // coarse levels whole runs of lanes fall into the SAME cell: left alone, their atomics serialise on a handful of
            // addresses in L2.  Levels 0..7 (threads of half 0) therefore reduce each run inside the warp first -- segmented
            // reduction towards the run's first lane, bounded by the next run head -- and only run heads issue atomics.
            float x01[3] = {2.f, 2.f, 2.f};
            if (live) {
#pragma unroll
                for (int d = 0; d < 3; d++) x01[d] = __fmul_rn(__fadd_rn(__ldg(xyzs + (size_t)s * 3 + d), desc.bound), inv2b);
            }
            const bool ok = live && !(x01[0] < 0.f || x01[0] > 1.f || x01[1] < 0.f || x01[1] > 1.f || x01[2] < 0.f || x01[2] > 1.f);
#pragma unroll
            for (uint32_t li = 0; li < kScatLevels; li++) {
                float g0 = ok ? __uint_as_float(v[2 * li]) : 0.f, g1 = ok ? __uint_as_float(v[2 * li + 1]) : 0.f;
                const uint32_t level = scat_level(half, li);
                const LevelGeom g = lg[level];
                uint32_t idx[8];
                float w[8];
                float xs[3] = {ok ? x01[0] : 0.f, ok ? x01[1] : 0.f, ok ? x01[2] : 0.f};
                level_corners(xs, g, idx, w);
                float2* base = grad_table + g.offset;
                if (level < 8) {   // levels 0..7 (warp-uniform)
                    // run heads: first lane, or a lane whose cell differs from the previous lane's (corner 0 and corner 7
                    // together identify the cell; a hash collision only splits or merges runs of identical addresses)
                    const uint32_t p0 = __shfl_up_sync(0xffffffffu, idx[0], 1), p7 = __shfl_up_sync(0xffffffffu, idx[7], 1);
                    const bool head = lane == 0 || p0 != idx[0] || p7 != idx[7];
                    const uint32_t heads = __ballot_sync(0xffffffffu, head);
                    const uint32_t after = lane == 31 ? 0u : (heads >> (lane + 1));
                    const uint32_t next_head = after ? (lane + 1 + (uint32_t)__ffs(after) - 1u) : 32u;
                    float a0[8], a1[8];
#pragma unroll
                    for (uint32_t c = 0; c < 8; c++) { a0[c] = __fmul_rn(w[c], g0); a1[c] = __fmul_rn(w[c], g1); }
#pragma unroll
                    for (uint32_t off = 1; off < 32; off <<= 1) {
                        const bool take = lane + off < next_head;
#pragma unroll
                        for (uint32_t c = 0; c < 8; c++) {
                            const float o0 = __shfl_down_sync(0xffffffffu, a0[c], off), o1 = __shfl_down_sync(0xffffffffu, a1[c], off);
                            if (take) { a0[c] += o0; a1[c] += o1; }
                        }
                    }
                    if (head) {
#pragma unroll
                        for (uint32_t c = 0; c < 8; c++)
                            if (a0[c] != 0.f || a1[c] != 0.f) atomicAdd(base + idx[c], make_float2(a0[c], a1[c]));
                    }
                } else if (g0 != 0.f || g1 != 0.f) {
                    // x-neighbour corners (2i, 2i+1) sit in one 16-byte aligned slot whenever the cell's x index is even (prime[0] = 1:
                    // entry a and a ^ 1): one 16-byte RED instead of two 8-byte ones (-11 % kernel time on B200)
#pragma unroll
                    for (uint32_t c = 0; c < 8; c += 2) {
                        const float2 va = make_float2(__fmul_rn(w[c], g0), __fmul_rn(w[c], g1));
                        const float2 vb = make_float2(__fmul_rn(w[c + 1], g0), __fmul_rn(w[c + 1], g1));
                        if ((idx[c] ^ idx[c + 1]) == 1u) {
                            const bool odd = idx[c] & 1u;
                            atomicAdd(reinterpret_cast<float4*>(base + (idx[c] & ~1u)),
                                      odd ? make_float4(vb.x, vb.y, va.x, va.y) : make_float4(va.x, va.y, vb.x, vb.y));
                        } else {
                            atomicAdd(base + idx[c], va);
                            atomicAdd(base + idx[c + 1], vb);
                        }
                    }
                }
            }
        }
    }
}

// ---- CTA of the two backward kernels --------------------------------------------------------------------------------------------
// Shared memory (Sm = BSmem or RSm): operand tiles [0, Sm::W), the packed weight blob (kWeightBytes) at Sm::W, the dF tiles at
// Sm::DF and at Sm::MISC: LevelGeom[16] | MMA mbarrier | TMEM slot | df_full[2] | df_empty[2].  512 TMEM columns.
struct BwdCta {
    LevelGeom* lg;
    uint64_t* bar;        // MMA completion (chain role)
    uint64_t* df_full;    // [2] dF tile written by the chain role
    uint64_t* df_empty;   // [2] dF tile read by the scatter role
    uint32_t tmem;
    uint32_t phase;       // of `bar`

    __device__ __forceinline__ void wait_mma() {
        __syncwarp();
        umma::mbar_wait(bar, phase);
        phase ^= 1u;
        umma::fence_after_sync();
    }
    // generic-proxy tile writes -> visible to the next MMAs (barrier over the chain role only)
    __device__ __forceinline__ void publish() const {
        umma::fence_async_smem();
        umma::fence_before_sync();
        umma::named_sync<1, kBwdChainT>();
    }
};

template <typename Sm, uint32_t kWeightBytes>
__device__ __forceinline__ BwdCta bwd_cta_setup(uint8_t* smem, const inerf_field_desc& desc, const void* weights, uint32_t tid) {
    LevelGeom* lg = reinterpret_cast<LevelGeom*>(smem + Sm::MISC);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + Sm::MISC + 16 * sizeof(LevelGeom));
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + Sm::MISC + 16 * sizeof(LevelGeom) + 8);
    uint64_t* df_full = reinterpret_cast<uint64_t*>(smem + Sm::MISC + 16 * sizeof(LevelGeom) + 16);
    uint64_t* df_empty = df_full + 2;

    // zero the operand tiles once: padding columns that no stage writes stay zero for the whole launch
    for (uint32_t i = tid; i < Sm::W / 16; i += kBwdThreads) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
    {
        const uint4* wsrc = reinterpret_cast<const uint4*>(weights);
        uint4* wdst = reinterpret_cast<uint4*>(smem + Sm::W);
        for (uint32_t i = tid; i < kWeightBytes / 16; i += kBwdThreads) wdst[i] = __ldg(wsrc + i);
    }
    init_levels(lg, desc.offsets, desc.L, desc.S, desc.H, tid);
    if (tid == 0) {
        umma::mbar_init(bar, 1);
        for (int i = 0; i < 2; i++) { umma::mbar_init(&df_full[i], kBwdChainT); umma::mbar_init(&df_empty[i], kBwdScatterT); }
        umma::mbar_fence_init();
    }
    if (tid < 32) umma::tmem_alloc<kBwdTmemCols>(tmem_slot);
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    return BwdCta{lg, bar, df_full, df_empty, *tmem_slot, 0u};
}

__device__ __forceinline__ void bwd_cta_teardown(uint32_t tmem, uint32_t tid) {
    umma::fence_before_sync();
    __syncthreads();
    if (tid < 32) umma::tmem_dealloc<kBwdTmemCols>(tmem);
}

// Two roles per CTA: the CHAIN warps (threads 0..255) run the tcgen05 recompute / dX / dW chain of tile i + 1 while the SCATTER
// warps (threads 256..511) push tile i's feature gradients into the table gradient.  The scatter is bound by the rate at
// which an SM retires RED lanes (~1 per clock); run back to back with the chain (the first version of this kernel) it left
// the tensor pipe and the LSU idle in turns.  dF travels through a double-buffered fp32 tile in shared memory.
__global__ void __launch_bounds__(kBwdThreads, 1) k_field_backward_mask(inerf_field_desc desc, BwdParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t K = desc.K, tid = threadIdx.x;
    // TG2's right half and dY's padding columns stay zero
    BwdCta cta = bwd_cta_setup<BSmem, BwdWeights::total>(smem, desc, p.weights, tid);
    const uint32_t tmem = cta.tmem;
    const uint32_t sbase = umma::smem_u32(smem);

    const bool chain_role = tid < kBwdChainT;
    const uint32_t rt = chain_role ? tid : tid - kBwdChainT;      // thread index inside the role
    const uint32_t warp = rt >> 5, lane = rt & 31;
    const uint32_t row = rt & (kTile - 1), half = rt >> 7;
    const uint32_t lane_base = ((warp & 3u) * 32u) << 16;
    const uint32_t B_eff = desc.n_valid ? min(p.B, (uint32_t)max(0, __ldg(desc.n_valid))) : p.B;   // rows past *n_valid are padding
    const uint32_t num_tiles = (B_eff + kTile - 1) / kTile;
    uint32_t tiles_done = 0;
    const bool issue_warp = tid < 32;   // one elected lane of warp 0 issues the MMAs (uniform branch for the compiler)

    if (chain_role) {
    umma::reg_alloc<kBwdRegsChain>();
    // The tile's inputs -- X0 (96 B / row) and dL/dlogits (4K B / row) -- are PREFETCHED into registers one tile ahead (issued
    // right after the first MMAs of the current tile), so their ~1 us of HBM latency is off the chain's critical path (the chain
    // alone took 5.7 us per tile, DESIGN.md 4.4).  16-byte loads; thread (row, half) takes the 8-column logit chunks half,
    // half + 2 (K <= 32 needs no more; further chunks of a wider head are loaded in place).  Columns >= K of the dY tile are
    // never written: they keep the zeros of the initial clear.
    const uint32_t nch = (K + 7u) >> 3;                     // 8-column chunks of dY that carry data
    const bool vec_ok = (K & 3u) == 0 && (((uintptr_t)p.grad_logits) & 15u) == 0;
    uint4 px[3];
    float4 pg[4];
    auto prefetch = [&](uint32_t tile_n) {
        const uint32_t sn = tile_n * kTile + row;
        const bool live_n = tile_n < num_tiles && sn < B_eff;
#pragma unroll
        for (uint32_t c = 0; c < 3; c++) px[c] = live_n ? __ldg(p.x0 + (size_t)sn * 6 + half * 3 + c) : make_uint4(0u, 0u, 0u, 0u);
        const float4* g4 = reinterpret_cast<const float4*>(p.grad_logits + (size_t)sn * K);
#pragma unroll
        for (uint32_t j = 0; j < 2; j++) {
            const uint32_t chunk = half + 2 * j;
            const bool ok0 = vec_ok && live_n && chunk * 8 < K, ok1 = vec_ok && live_n && chunk * 8 + 4 < K;
            pg[2 * j] = ok0 ? __ldg(g4 + chunk * 2) : make_float4(0.f, 0.f, 0.f, 0.f);
            pg[2 * j + 1] = ok1 ? __ldg(g4 + chunk * 2 + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    prefetch(blockIdx.x);
    for (uint32_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, tiles_done++) {
        const uint32_t s = tile * kTile + row;
        const bool live = s < B_eff;
        // ---- S0: X0 and dY rows -> operand tiles --------------------------------------------------------------
#pragma unroll
        for (uint32_t c = 0; c < 3; c++)
            *reinterpret_cast<uint4*>(smem + BSmem::TX + umma::tile_off(row, (half * 3 + c) * 8, kLBO, kSbo48)) = px[c];
        if (vec_ok) {
#pragma unroll
            for (uint32_t j = 0; j < 2; j++) {
                const uint32_t chunk = half + 2 * j;
                if (chunk < nch)
                    *reinterpret_cast<uint4*>(smem + BSmem::TG + umma::tile_off(row, chunk * 8, kLBO, kSbo128)) =
                        make_uint4(h2_bits(__floats2half2_rn(pg[2 * j].x, pg[2 * j].y)), h2_bits(__floats2half2_rn(pg[2 * j].z, pg[2 * j].w)),
                                   h2_bits(__floats2half2_rn(pg[2 * j + 1].x, pg[2 * j + 1].y)), h2_bits(__floats2half2_rn(pg[2 * j + 1].z, pg[2 * j + 1].w)));
            }
        }
        {   // chunks the prefetch does not cover: K > 32, or a K / alignment the 16-byte loads cannot serve
            const float* g = p.grad_logits + (size_t)s * K;
            for (uint32_t chunk = vec_ok ? 4u + half : half; chunk < nch; chunk += 2) {
                const uint32_t k0 = chunk * 8;
                uint32_t q[4];
#pragma unroll
                for (uint32_t i = 0; i < 4; i++) {
                    const uint32_t ka = k0 + 2 * i;
                    const float a = (live && ka < K) ? __ldg(g + ka) : 0.f;
                    const float b = (live && ka + 1 < K) ? __ldg(g + ka + 1) : 0.f;
                    q[i] = h2_bits(__floats2half2_rn(a, b));
                }
                *reinterpret_cast<uint4*>(smem + BSmem::TG + umma::tile_off(row, k0, kLBO, kSbo128)) = make_uint4(q[0], q[1], q[2], q[3]);
            }
        }
        cta.publish();
        // ---- S1: H1 pre-activation and dY W2 -----------------------------------------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, BSmem::TX, kSbo48, BSmem::W + BwdWeights::w0, kSbo48, 48, 64, tmem + T_a);
            issue_gemm2(sbase, BSmem::TG, kSbo128, BSmem::W + BwdWeights::w2t, kSbo64, 64, 64, tmem + T_b);
            umma::commit(cta.bar);
        }
        prefetch(tile + gridDim.x);   // next tile's inputs: in flight during the four MMA stages of this one
        cta.wait_mma();
        const uint32_t mask1 = epi_relu32(tmem + T_a + lane_base + half * 32, smem, BSmem::TH, row, 64 + half * 32);   // H1 -> TH[:, 64:128]
        cta.publish();
        // ---- S2: H2 pre-activation; dH2 = (dY W2) . [H2 > 0] ---------------------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, BSmem::TH + 8 * kLBO, kSbo128, BSmem::W + BwdWeights::w1, kSbo64, 64, 64, tmem + T_a);
            umma::commit(cta.bar);
        }
        cta.wait_mma();
        const uint32_t mask2 = epi_relu32(tmem + T_a + lane_base + half * 32, smem, BSmem::TH, row, half * 32);        // H2 -> TH[:, 0:64]
        epi_masked32(tmem + T_b + lane_base + half * 32, mask2, smem, BSmem::TG, row, 64 + half * 32);                 // dH2 -> TG[:, 64:128]
        cta.publish();
        // ---- S3: dH1 = (dH2 W1) . [H1 > 0] --------------------------------------------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, BSmem::TG + 8 * kLBO, kSbo128, BSmem::W + BwdWeights::w1t, kSbo64, 64, 64, tmem + T_b);
            umma::commit(cta.bar);
        }
        cta.wait_mma();
        epi_masked32(tmem + T_b + lane_base + half * 32, mask1, smem, BSmem::TG2, row, half * 32);                     // dH1 -> TG2[:, 0:64]
        cta.publish();
        // ---- S4: dF = dH1 W0[:, :32]; weight gradients accumulate across tiles ------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, BSmem::TG2, kSbo128, BSmem::W + BwdWeights::w0t, kSbo64, 64, 32, tmem + T_x);
            issue_gemm_tn(sbase, BSmem::TG, kSbo128, BSmem::TH, kSbo128, 128, tmem + T_w1, tiles_done > 0);
            issue_gemm_tn(sbase, BSmem::TG2, kSbo128, BSmem::TX, kSbo48, 48, tmem + T_w0, tiles_done > 0);
            umma::commit(cta.bar);
        }
        cta.wait_mma();
        // ---- hand dF (32 feature gradients / sample, fp32, [column][row] so that neither side has bank conflicts) to the scatter warps
        {
            const uint32_t db = tiles_done & 1u;
            if (tiles_done >= 2) umma::mbar_wait(&cta.df_empty[db], ((tiles_done >> 1) - 1u) & 1u);
            uint32_t v[16];
            umma::tmem_ld16(tmem + T_x + lane_base + half * 16, v);
            umma::tmem_ld_wait();
            float* dst = reinterpret_cast<float*>(smem + BSmem::DF) + db * (kTile * 32) + (half * 16) * kTile + row;
#pragma unroll
            for (int i = 0; i < 16; i++) dst[i * kTile] = __uint_as_float(v[i]);
            umma::mbar_arrive(&cta.df_full[db]);
        }
        umma::fence_before_sync();
        umma::named_sync<1, kBwdChainT>();   // TMEM accumulators T_a/T_b/T_x and the operand tiles are reused by the next tile
    }

    // ---- weight gradients of this CTA: TMEM -> global (fp32 atomics) ------------------------------------------------
    {
        const uint32_t q = warp & 3u, m = q * 32u + lane;   // TMEM lane = row of [dY|dH2]^T resp. [dH1|0]^T
        if (q < 2 && half == 0) {            // dW2[o = m][j], lanes 0..63, columns 0..63 of T_w1
            for (uint32_t c = 0; c < 64; c += 16) {
                uint32_t v[16];
                umma::tmem_ld16(tmem + T_w1 + lane_base + c, v);
                umma::tmem_ld_wait();
                if (m < K)
#pragma unroll
                    for (int j = 0; j < 16; j++) atomicAdd(p.grad_w2 + (size_t)m * 64 + c + j, __uint_as_float(v[j]));
            }
        } else if (q >= 2 && half == 1) {    // dW1[o = m - 64][j], lanes 64..127, columns 64..127 of T_w1
            for (uint32_t c = 0; c < 64; c += 16) {
                uint32_t v[16];
                umma::tmem_ld16(tmem + T_w1 + lane_base + 64 + c, v);
                umma::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; j++) atomicAdd(p.grad_w1 + (size_t)(m - 64) * 64 + c + j, __uint_as_float(v[j]));
            }
        }
        if (q < 2) {                         // dW0[o = m][j], lanes 0..63, columns 0..47 of T_w0 (j = 47 is X0's zero padding)
            const uint32_t c_begin = half ? 32u : 0u, c_end = half ? 48u : 32u;
            for (uint32_t c = c_begin; c < c_end; c += 16) {
                uint32_t v[16];
                umma::tmem_ld16(tmem + T_w0 + lane_base + c, v);
                umma::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; j++)
                    if (c + j < 47) atomicAdd(p.grad_w0 + (size_t)m * 47 + c + j, __uint_as_float(v[j]));
            }
        }
    }
    } else {
    umma::reg_dealloc<kBwdRegsScatter>();
    scatter_role(desc, p.xyzs, p.grad_table, cta.lg, smem + BSmem::DF, cta.df_full, cta.df_empty, num_tiles, B_eff, rt);
    }
    bwd_cta_teardown(tmem, tid);
}

// =================================================================================================================================
// inerf_field_backward_rgb: backward of the stage-1 (RGB-sigma) field -- sigma_net (32->64->16) and color_net (32->64->64->3) with
// the sigma hash table (Trainer.train_step, nerf/utils.py:536-632; network.py:96-127 through autograd: 10 cuBLAS GEMMs, 3
// ReLU-backward kernels, sigmoid / trunc_exp backward, cat / slice backward, kernel_grid_backward, whole-table zero + cast).
// Per 128-sample tile, all on tcgen05 (fp16 operands as autocast rounds them, fp32 accumulators in TMEM):
//
//   recompute  Hs = relu(E Ws0^T), Hc1 = relu(Ci Wc0^T), Hc2 = relu(Hc1 Wc1^T)        (E, Ci = saved net inputs, fp16 [.,64])
//   colour     dP = fp16(g_rgb) . rgb (1 - rgb);  dHc2 = (dP Wc2) . [Hc2>0];  dHc1 = (dHc2 Wc1) . [Hc1>0];  dCi = dHc1 Wc0
//   sigma      dO = [fp16(g_sigma * clamp(sigma, e^-15, e^15)) | dCi[:, 16:31]];  dHs = (dO Ws1) . [Hs>0];  dE = dHs Ws0
//   dW         [dHc2|dHc1]^T [Hc1|Ci] -> dWc1, dWc0 ;  [dHs|dP|dO]^T [E|Hc2|Hs] -> dWs0, dWc2, dWs1   (diagonal blocks of two
//              M = 128 products whose operands are the tiles above read MN-major; accumulated ACROSS tiles in TMEM)
//   scatter    dE (32 feature gradients / sample) -> the fp32 sigma-table gradient (scatter_role).
struct RgbBwdWeights {   // byte offsets inside the packed blob (B operands, K-major)
    static constexpr uint32_t ws0 = 0;                    // [64 x 32]  Ws0[o][j]
    static constexpr uint32_t wc0 = ws0 + 64 * 32 * 2;    // [64 x 32]  Wc0[o][j], j = 31 zero
    static constexpr uint32_t wc1 = wc0 + 64 * 32 * 2;    // [64 x 64]  Wc1[o][j]
    static constexpr uint32_t wc2t = wc1 + 64 * 64 * 2;   // [64 x 16]  (n=j, k=o) = Wc2[o][j], o >= 3 zero
    static constexpr uint32_t wc1t = wc2t + 64 * 16 * 2;  // [64 x 64]  (n=j, k=o) = Wc1[o][j]
    static constexpr uint32_t wc0t = wc1t + 64 * 64 * 2;  // [32 x 64]  (n=j, k=o) = Wc0[o][j], j = 31 zero
    static constexpr uint32_t ws1t = wc0t + 32 * 64 * 2;  // [64 x 16]  (n=j, k=o) = Ws1[o][j]
    static constexpr uint32_t ws0t = ws1t + 64 * 16 * 2;  // [32 x 64]  (n=j, k=o) = Ws0[o][j]
    static constexpr uint32_t total = ws0t + 32 * 64 * 2;
};
struct RSm {   // operand tiles: column ranges of four wide K-major tiles, so that the dW products read them whole
    static constexpr uint32_t GA = 0;                        // [128 x 128]  dHc2 (64) | dHc1 (64)
    static constexpr uint32_t HA = GA + kTile * 128 * 2;     // [128 x 96]   Hc1 (64) | Ci (32)
    static constexpr uint32_t GB = HA + kTile * 96 * 2;      // [128 x 128]  dHs (64) | dP (16) | 0 (16) | dO (16) | 0 (16)
    static constexpr uint32_t HB = GB + kTile * 128 * 2;     // [128 x 160]  E (32) | Hc2 (64) | Hs (64)
    static constexpr uint32_t W = HB + kTile * 160 * 2;
    static constexpr uint32_t DF = W + RgbBwdWeights::total;
    static constexpr uint32_t MISC = DF + 2 * kTile * 32 * 4;
    static constexpr uint32_t bytes = MISC + 16 * sizeof(LevelGeom) + 64;
};
constexpr uint32_t kSbo96 = sbo_of(96), kSbo160 = sbo_of(160), kSbo32 = sbo_of(32), kSbo16 = sbo_of(16);
// TMEM columns: three 64-wide working accumulators, one 32-wide, and the two weight-gradient products
constexpr uint32_t R_a = 0, R_b = 64, R_c = 128, R_x = 192, R_w1 = 224, R_w2 = 320;   // R_w1: 96 columns, R_w2: 160 columns
static_assert(R_w2 + 160 <= kBwdTmemCols, "TMEM plan");
static_assert(RSm::bytes <= 227 * 1024, "shared memory plan");

struct RgbBwdParams {
    const float* xyzs;          // [B, 3]
    const uint4* xs;            // fp16 [B, 64] = E (32) | Ci (32), 8 x 16 B per row
    const float* sigmas;        // [B]   forward output (unscaled)
    const float* rgbs;          // [B, 3] forward output
    const float* grad_sigmas;   // [B]
    const float* grad_rgbs;     // [B, 3]
    uint32_t B;
    float2* grad_table;         // fp32 [T, 2] (encoder.embeddings.grad), accumulated
    float* grad_ws0;            // [64, 32]
    float* grad_ws1;            // [16, 64]
    float* grad_wc0;            // [64, 31]
    float* grad_wc1;            // [64, 64]
    float* grad_wc2;            // [3, 64]
    const void* weights;        // packed blob (RgbBwdWeights)
};

__global__ void __launch_bounds__(kBwdThreads, 1) k_field_backward_rgb(inerf_field_desc desc, RgbBwdParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t tid = threadIdx.x;
    // the padding columns of GB (and dP's columns 3..15) stay zero
    BwdCta cta = bwd_cta_setup<RSm, RgbBwdWeights::total>(smem, desc, p.weights, tid);
    const uint32_t tmem = cta.tmem;
    const uint32_t sbase = umma::smem_u32(smem);

    const bool chain_role = tid < kBwdChainT;
    const uint32_t rt = chain_role ? tid : tid - kBwdChainT;
    const uint32_t warp = rt >> 5, lane = rt & 31;
    const uint32_t row = rt & (kTile - 1), half = rt >> 7;
    const uint32_t lane_base = ((warp & 3u) * 32u) << 16;
    const uint32_t B_eff = desc.n_valid ? min(p.B, (uint32_t)max(0, __ldg(desc.n_valid))) : p.B;
    const uint32_t num_tiles = (B_eff + kTile - 1) / kTile;
    uint32_t tiles_done = 0;
    const bool issue_warp = tid < 32;   // one elected lane of warp 0 issues the MMAs (uniform branch for the compiler)
    constexpr uint32_t Wb = RSm::W;

    if (chain_role) {
    umma::reg_alloc<kBwdRegsChain>();
    // inputs of the next tile prefetched into registers (as in k_field_backward_mask): thread (row, 0) takes E and the colour
    // head's (g_rgb, rgb), thread (row, 1) takes Ci and the density head's (g_sigma, sigma)
    uint4 px[4];
    float pf[6];
    auto prefetch = [&](uint32_t tile_n) {
        const uint32_t sn = tile_n * kTile + row;
        const bool live_n = tile_n < num_tiles && sn < B_eff;
#pragma unroll
        for (uint32_t c = 0; c < 4; c++) px[c] = live_n ? __ldg(p.xs + (size_t)sn * 8 + half * 4 + c) : make_uint4(0u, 0u, 0u, 0u);
        if (half == 0) {
#pragma unroll
            for (uint32_t c = 0; c < 3; c++) {
                pf[c] = live_n ? __ldg(p.grad_rgbs + (size_t)sn * 3 + c) : 0.f;
                pf[3 + c] = live_n ? __ldg(p.rgbs + (size_t)sn * 3 + c) : 0.f;
            }
        } else {
            pf[0] = live_n ? __ldg(p.grad_sigmas + sn) : 0.f;
            pf[1] = live_n ? __ldg(p.sigmas + sn) : 0.f;
        }
    };
    prefetch(blockIdx.x);
    for (uint32_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, tiles_done++) {
        // ---- S0: saved inputs and the head gradients -> operand tiles ---------------------------------------------------
        uint32_t dh0_bits = 0;   // fp16 gradient of the sigma-net's output 0 (thread (row, 1))
        if (half == 0) {
#pragma unroll
            for (uint32_t c = 0; c < 4; c++)
                *reinterpret_cast<uint4*>(smem + RSm::HB + umma::tile_off(row, c * 8, kLBO, kSbo160)) = px[c];          // E -> HB[:, 0:32]
            // sigmoid backward as autocast runs it: the incoming gradient is cast to fp16, g * (1 - y) * y in fp32, ONE rounding
            float dp[3];
#pragma unroll
            for (uint32_t c = 0; c < 3; c++) {
                const float g16 = __half2float(__float2half_rn(pf[c])), y = pf[3 + c];
                dp[c] = __fmul_rn(__fmul_rn(g16, __fsub_rn(1.0f, y)), y);
            }
            *reinterpret_cast<uint4*>(smem + RSm::GB + umma::tile_off(row, 64, kLBO, kSbo128)) =
                make_uint4(h2_bits(__floats2half2_rn(dp[0], dp[1])), h2_bits(__floats2half2_rn(dp[2], 0.f)), 0u, 0u);    // dP -> GB[:, 64:72]
        } else {
#pragma unroll
            for (uint32_t c = 0; c < 4; c++)
                *reinterpret_cast<uint4*>(smem + RSm::HA + umma::tile_off(row, 64 + c * 8, kLBO, kSbo96)) = px[c];      // Ci -> HA[:, 64:96]
            // trunc_exp backward (activation.py:13-17): g * exp(clamp(x, -15, 15)) in fp32, then the cast back to the fp16 activation
            const float e = fminf(fmaxf(pf[1], 3.0590232e-07f), 3269017.4f);
            dh0_bits = (uint32_t)__half_as_ushort(__float2half_rn(__fmul_rn(pf[0], e)));
        }
        cta.publish();
        // ---- S1: Hs, Hc1 pre-activations; dP Wc2 ---------------------------------------------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, RSm::HB, kSbo160, Wb + RgbBwdWeights::ws0, kSbo32, 32, 64, tmem + R_a);
            issue_gemm2(sbase, RSm::HA + 8 * kLBO, kSbo96, Wb + RgbBwdWeights::wc0, kSbo32, 32, 64, tmem + R_b);
            issue_gemm2(sbase, RSm::GB + 8 * kLBO, kSbo128, Wb + RgbBwdWeights::wc2t, kSbo16, 16, 64, tmem + R_c);
            umma::commit(cta.bar);
        }
        prefetch(tile + gridDim.x);
        cta.wait_mma();
        const uint32_t mask_s = epi_relu_to(tmem + R_a + lane_base + half * 32, smem, RSm::HB, kSbo160, row, 96 + half * 32);    // Hs  -> HB[:, 96:160]
        const uint32_t mask_c1 = epi_relu_to(tmem + R_b + lane_base + half * 32, smem, RSm::HA, kSbo96, row, half * 32);        // Hc1 -> HA[:, 0:64]
        cta.publish();
        // ---- S2: Hc2 pre-activation; dHc2 = (dP Wc2) . [Hc2 > 0] --------------------------------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, RSm::HA, kSbo96, Wb + RgbBwdWeights::wc1, kSbo64, 64, 64, tmem + R_a);
            umma::commit(cta.bar);
        }
        cta.wait_mma();
        const uint32_t mask_c2 = epi_relu_to(tmem + R_a + lane_base + half * 32, smem, RSm::HB, kSbo160, row, 32 + half * 32);   // Hc2 -> HB[:, 32:96]
        epi_masked32(tmem + R_c + lane_base + half * 32, mask_c2, smem, RSm::GA, row, half * 32);                               // dHc2 -> GA[:, 0:64]
        cta.publish();
        // ---- S3: dHc1 = (dHc2 Wc1) . [Hc1 > 0] ----------------------------------------------------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, RSm::GA, kSbo128, Wb + RgbBwdWeights::wc1t, kSbo64, 64, 64, tmem + R_b);
            umma::commit(cta.bar);
        }
        cta.wait_mma();
        epi_masked32(tmem + R_b + lane_base + half * 32, mask_c1, smem, RSm::GA, row, 64 + half * 32);                          // dHc1 -> GA[:, 64:128]
        cta.publish();
        // ---- S4: dCi = dHc1 Wc0; the density head's output gradient dO = [dh0 | dgeo15] ----------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, RSm::GA + 8 * kLBO, kSbo128, Wb + RgbBwdWeights::wc0t, kSbo64, 64, 32, tmem + R_x);
            umma::commit(cta.bar);
        }
        cta.wait_mma();
        if (half == 1) {   // columns 16..31 of dCi: geo15 (column 31 is the zero padding of Ci)
            uint32_t v[16];
            umma::tmem_ld16(tmem + R_x + lane_base + 16, v);
            umma::tmem_ld_wait();
            uint32_t q[8];
            q[0] = dh0_bits | ((uint32_t)__half_as_ushort(__float2half_rn(__uint_as_float(v[0]))) << 16);
#pragma unroll
            for (int i = 1; i < 8; i++) q[i] = h2_bits(__floats2half2_rn(__uint_as_float(v[2 * i - 1]), __uint_as_float(v[2 * i])));
            *reinterpret_cast<uint4*>(smem + RSm::GB + umma::tile_off(row, 96, kLBO, kSbo128)) = make_uint4(q[0], q[1], q[2], q[3]);
            *reinterpret_cast<uint4*>(smem + RSm::GB + umma::tile_off(row, 104, kLBO, kSbo128)) = make_uint4(q[4], q[5], q[6], q[7]);
        }
        cta.publish();
        // ---- S5: dHs = (dO Ws1) . [Hs > 0] ---------------------------------------------------------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, RSm::GB + 12 * kLBO, kSbo128, Wb + RgbBwdWeights::ws1t, kSbo16, 16, 64, tmem + R_a);
            umma::commit(cta.bar);
        }
        cta.wait_mma();
        epi_masked32(tmem + R_a + lane_base + half * 32, mask_s, smem, RSm::GB, row, half * 32);                                // dHs -> GB[:, 0:64]
        cta.publish();
        // ---- S6: dE = dHs Ws0; weight gradients accumulate across tiles ----------------------------------------------------------
        if (issue_warp && umma::elect_one()) {
            umma::fence_after_sync();
            issue_gemm2(sbase, RSm::GB, kSbo128, Wb + RgbBwdWeights::ws0t, kSbo64, 64, 32, tmem + R_x);
            issue_gemm_tn(sbase, RSm::GA, kSbo128, RSm::HA, kSbo96, 96, tmem + R_w1, tiles_done > 0);
            issue_gemm_tn(sbase, RSm::GB, kSbo128, RSm::HB, kSbo160, 160, tmem + R_w2, tiles_done > 0);
            umma::commit(cta.bar);
        }
        cta.wait_mma();
        {
            const uint32_t db = tiles_done & 1u;
            if (tiles_done >= 2) umma::mbar_wait(&cta.df_empty[db], ((tiles_done >> 1) - 1u) & 1u);
            uint32_t v[16];
            umma::tmem_ld16(tmem + R_x + lane_base + half * 16, v);
            umma::tmem_ld_wait();
            float* dst = reinterpret_cast<float*>(smem + RSm::DF) + db * (kTile * 32) + (half * 16) * kTile + row;
#pragma unroll
            for (int i = 0; i < 16; i++) dst[i * kTile] = __uint_as_float(v[i]);
            umma::mbar_arrive(&cta.df_full[db]);
        }
        umma::fence_before_sync();
        umma::named_sync<1, kBwdChainT>();
    }

    // ---- weight gradients of this CTA: TMEM -> global (fp32 atomics).  Lane m of R_w1 / R_w2 = column m of GA / GB. ------------
    if (tiles_done > 0) {
        const uint32_t q = warp & 3u, m = q * 32u + lane;
        auto flush = [&](uint32_t tcol, uint32_t ncols, float* dst, uint32_t ld, uint32_t r, uint32_t c_lim, bool row_ok) {
            for (uint32_t c = 0; c < ncols; c += 16) {
                uint32_t v[16];
                umma::tmem_ld16(tmem + tcol + lane_base + c, v);
                umma::tmem_ld_wait();
                if (row_ok)
#pragma unroll
                    for (int j = 0; j < 16; j++)
                        if (c + j < c_lim) atomicAdd(dst + (size_t)r * ld + c + j, __uint_as_float(v[j]));
            }
        };
        if (half == 0) {
            if (q < 2) flush(R_w1, 64, p.grad_wc1, 64, m, 64, true);                       // dWc1[o = m][j]        lanes 0..63,   HA cols 0..63
            else flush(R_w1 + 64, 32, p.grad_wc0, 31, m - 64, 31, true);                   // dWc0[o = m - 64][j]   lanes 64..127, HA cols 64..94
        } else {
            if (q < 2) flush(R_w2, 32, p.grad_ws0, 32, m, 32, true);                       // dWs0[o = m][j]        lanes 0..63,   HB cols 0..31
            else if (q == 2) flush(R_w2 + 32, 64, p.grad_wc2, 64, m - 64, 64, m - 64 < 3); // dWc2[o = m - 64][j]   lanes 64..66,  HB cols 32..95
            else flush(R_w2 + 96, 64, p.grad_ws1, 64, m - 96, 64, m - 96 < 16);            // dWs1[o = m - 96][j]   lanes 96..111, HB cols 96..159
        }
    }
    } else {
    umma::reg_dealloc<kBwdRegsScatter>();
    scatter_role(desc, p.xyzs, p.grad_table, cta.lg, smem + RSm::DF, cta.df_full, cta.df_empty, num_tiles, B_eff, rt);
    }
    bwd_cta_teardown(tmem, tid);
}

// ---- weight packing: fp32 nn.Linear matrices -> the fp16 operand blobs of the field kernels ---------------------------------
// Each blob is written down once, as a list of PackJobs (one per operand tile).  The host packers (CPU pointers) and
// k_pack_weights (DEVICE pointers, no host round trip: the trainable weights change every optimizer step) apply the same
// element rule, pack_value.
struct PackJob {
    const float* W;        // fp32 [n_out, n_in] row-major (nn.Linear layout)
    uint32_t n_out, n_in;  // logical shape of W
    uint32_t Npad, Kpad;   // operand tile shape [Npad x Kpad]
    uint32_t dst;          // byte offset inside the blob
    uint32_t transpose;    // 0: (n, k) = W[n][k]; 1: (n, k) = W[k][n]
    uint32_t n_lim;        // rows of the tile that carry data (others zero)
};
struct PackJobs {
    PackJob j[13];
    uint32_t n;
    void add(const float* W, uint32_t n_out, uint32_t n_in, uint32_t Npad, uint32_t Kpad, uint32_t dst, uint32_t tr, uint32_t n_lim) {
        j[n++] = PackJob{W, n_out, n_in, Npad, Kpad, dst, tr, n_lim};
    }
};

// element (n, k) of job J's tile; zero outside W
__host__ __device__ __forceinline__ float pack_value(const PackJob& J, uint32_t n, uint32_t k) {
    float v = 0.f;
    if (!J.transpose) { if (n < J.n_out && k < J.n_in) v = J.W[(size_t)n * J.n_in + k]; }
    else if (k < J.n_out && n < J.n_in && n < J.n_lim) v = J.W[(size_t)k * J.n_in + n];
    return v;
}

__global__ void k_pack_weights(PackJobs jobs, uint8_t* fwd, uint8_t* bwd, uint32_t n_fwd) {
    for (uint32_t ji = blockIdx.y; ji < jobs.n; ji += gridDim.y) {
        const PackJob J = jobs.j[ji];
        uint8_t* out = (ji < n_fwd ? fwd : bwd) + J.dst;
        const uint32_t total = J.Npad * J.Kpad;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
            const uint32_t n = i / J.Kpad, k = i % J.Kpad;
            *reinterpret_cast<__half*>(out + umma::tile_off(n, k, kLBO, sbo_of(J.Kpad))) = __float2half_rn(pack_value(J, n, k));
        }
    }
}

// every element of every tile: the jobs of a blob cover it, so no byte keeps what was there before
void pack_on_host(const PackJobs& jobs, uint8_t* blob) {
    for (uint32_t ji = 0; ji < jobs.n; ji++) {
        const PackJob& J = jobs.j[ji];
        for (uint32_t n = 0; n < J.Npad; n++)
            for (uint32_t k = 0; k < J.Kpad; k++) {
                const __half h = __float2half_rn(pack_value(J, n, k));
                memcpy(blob + J.dst + umma::tile_off(n, k, kLBO, sbo_of(J.Kpad)), &h, 2);
            }
    }
}

// the forward blob (field::weight_layout): sigma-net, colour-net, mask-net
void add_forward_layers(PackJobs& jobs, const float* sigma0, const float* sigma1, const float* color0, const float* color1, const float* color2,
                        const float* mask0, const float* mask1, const float* mask2, uint32_t K) {
    const WeightLayout wl = weight_layout(K);
    jobs.add(sigma0, 64, 32, 64, 32, wl.s0, 0, 64);
    jobs.add(sigma1, 16, 64, 16, 64, wl.s1, 0, 16);
    jobs.add(color0, 64, 31, 64, 32, wl.c0, 0, 64);
    jobs.add(color1, 64, 64, 64, 64, wl.c1, 0, 64);
    jobs.add(color2, 3, 64, 16, 64, wl.c2, 0, 16);
    jobs.add(mask0, 64, 47, 64, 48, wl.m0, 0, 64);
    jobs.add(mask1, 64, 64, 64, 64, wl.m1, 0, 64);
    jobs.add(mask2, K, 64, wl.Kp, 64, wl.m2, 0, wl.Kp);
}

// the mask-head backward blob (BwdWeights)
void add_mask_bwd_layers(PackJobs& jobs, const float* mask0, const float* mask1, const float* mask2, uint32_t K) {
    jobs.add(mask0, 64, 47, 64, 48, BwdWeights::w0, 0, 64);
    jobs.add(mask1, 64, 64, 64, 64, BwdWeights::w1, 0, 64);
    jobs.add(mask2, K, 64, 64, 64, BwdWeights::w2t, 1, 64);
    jobs.add(mask1, 64, 64, 64, 64, BwdWeights::w1t, 1, 64);
    jobs.add(mask0, 64, 47, 32, 64, BwdWeights::w0t, 1, 32);
}

}  // namespace

extern "C" int inerf_field_pack_weights(const float* sigma0, const float* sigma1, const float* color0, const float* color1,
                                        const float* color2, const float* mask0, const float* mask1, const float* mask2, uint32_t K,
                                        void* packed_host) {
    if (K == 0 || K > 64) return INERF_ERR_SIZE;
    INERF_REQUIRE(sigma0); INERF_REQUIRE(sigma1); INERF_REQUIRE(color0); INERF_REQUIRE(color1); INERF_REQUIRE(color2);
    INERF_REQUIRE(mask0); INERF_REQUIRE(mask1); INERF_REQUIRE(mask2); INERF_REQUIRE(packed_host);
    PackJobs jobs{};
    add_forward_layers(jobs, sigma0, sigma1, color0, color1, color2, mask0, mask1, mask2, K);
    pack_on_host(jobs, static_cast<uint8_t*>(packed_host));
    return INERF_OK;
}

// Device-side equivalent of inerf_field_pack_weights (+ inerf_field_pack_weights_bwd when packed_bwd != NULL):
// all pointers are DEVICE pointers, one launch, no synchronisation.
extern "C" int inerf_field_pack_weights_device(const float* sigma0, const float* sigma1, const float* color0, const float* color1,
                                               const float* color2, const float* mask0, const float* mask1, const float* mask2, uint32_t K,
                                               void* packed_fwd, void* packed_bwd, void* stream) {
    if (K == 0 || K > 64) return INERF_ERR_SIZE;
    INERF_REQUIRE(sigma0); INERF_REQUIRE(sigma1); INERF_REQUIRE(color0); INERF_REQUIRE(color1); INERF_REQUIRE(color2);
    INERF_REQUIRE(mask0); INERF_REQUIRE(mask1); INERF_REQUIRE(mask2); INERF_REQUIRE(packed_fwd);
    PackJobs jobs{};
    add_forward_layers(jobs, sigma0, sigma1, color0, color1, color2, mask0, mask1, mask2, K);
    const uint32_t n_fwd = jobs.n;
    if (packed_bwd) add_mask_bwd_layers(jobs, mask0, mask1, mask2, K);
    k_pack_weights<<<dim3(4, jobs.n), 256, 0, (cudaStream_t)stream>>>(jobs, (uint8_t*)packed_fwd, (uint8_t*)packed_bwd, n_fwd);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

extern "C" size_t inerf_field_bwd_weights_bytes(void) { return BwdWeights::total; }

extern "C" int inerf_field_pack_weights_bwd(const float* mask0, const float* mask1, const float* mask2, uint32_t K, void* packed_host) {
    if (K == 0 || K > 64) return INERF_ERR_SIZE;
    INERF_REQUIRE(mask0); INERF_REQUIRE(mask1); INERF_REQUIRE(mask2); INERF_REQUIRE(packed_host);
    PackJobs jobs{};
    add_mask_bwd_layers(jobs, mask0, mask1, mask2, K);
    pack_on_host(jobs, static_cast<uint8_t*>(packed_host));
    return INERF_OK;
}

extern "C" int inerf_field_backward_mask(const inerf_field_desc* desc, const void* weights_bwd, const float* xyzs, const void* x0,
                                         const float* grad_logits, uint32_t B, float* grad_table, float* grad_w0, float* grad_w1,
                                         float* grad_w2, void* stream) {
    if (int e = field::validate(desc)) return e;
    if (B == 0) return INERF_OK;
    INERF_REQUIRE(weights_bwd); INERF_REQUIRE(xyzs); INERF_REQUIRE(x0); INERF_REQUIRE(grad_logits);
    INERF_REQUIRE(grad_table); INERF_REQUIRE(grad_w0); INERF_REQUIRE(grad_w1); INERF_REQUIRE(grad_w2);
    if (((uintptr_t)weights_bwd & 15u) || ((uintptr_t)x0 & 15u) || ((uintptr_t)grad_table & 7u)) return INERF_ERR_ALIGN;
    const BwdParams p{xyzs, (const uint4*)x0, grad_logits, B, (float2*)grad_table, grad_w0, grad_w1, grad_w2, weights_bwd};
    return launch_persistent(k_field_backward_mask, B, kBwdThreads, BSmem::bytes, (cudaStream_t)stream, *desc, p);
}

// ---- stage-1 (RGB-sigma) backward ------------------------------------------------------------------------------------------
extern "C" size_t inerf_field_rgb_bwd_weights_bytes(void) { return RgbBwdWeights::total; }

// fp32 nn.Linear matrices (DEVICE) -> the operand blob of inerf_field_backward_rgb (DEVICE), one launch on `stream`
extern "C" int inerf_field_pack_weights_rgb_bwd_device(const float* sigma0, const float* sigma1, const float* color0, const float* color1,
                                                       const float* color2, void* packed_bwd, void* stream) {
    INERF_REQUIRE(sigma0); INERF_REQUIRE(sigma1); INERF_REQUIRE(color0); INERF_REQUIRE(color1); INERF_REQUIRE(color2);
    INERF_REQUIRE(packed_bwd);
    if ((uintptr_t)packed_bwd & 15u) return INERF_ERR_ALIGN;
    PackJobs jobs{};
    jobs.add(sigma0, 64, 32, 64, 32, RgbBwdWeights::ws0, 0, 64);
    jobs.add(color0, 64, 31, 64, 32, RgbBwdWeights::wc0, 0, 64);
    jobs.add(color1, 64, 64, 64, 64, RgbBwdWeights::wc1, 0, 64);
    jobs.add(color2, 3, 64, 64, 16, RgbBwdWeights::wc2t, 1, 64);
    jobs.add(color1, 64, 64, 64, 64, RgbBwdWeights::wc1t, 1, 64);
    jobs.add(color0, 64, 31, 32, 64, RgbBwdWeights::wc0t, 1, 32);
    jobs.add(sigma1, 16, 64, 64, 16, RgbBwdWeights::ws1t, 1, 64);
    jobs.add(sigma0, 64, 32, 32, 64, RgbBwdWeights::ws0t, 1, 32);
    k_pack_weights<<<dim3(4, jobs.n), 256, 0, (cudaStream_t)stream>>>(jobs, nullptr, (uint8_t*)packed_bwd, 0);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

extern "C" int inerf_field_backward_rgb(const inerf_field_desc* desc, const void* weights_bwd, const float* xyzs, const void* xs,
                                        const float* sigmas, const float* rgbs, const float* grad_sigmas, const float* grad_rgbs, uint32_t B,
                                        float* grad_table, float* grad_ws0, float* grad_ws1, float* grad_wc0, float* grad_wc1,
                                        float* grad_wc2, void* stream) {
    if (int e = field::validate(desc)) return e;
    if (B == 0) return INERF_OK;
    INERF_REQUIRE(weights_bwd); INERF_REQUIRE(xyzs); INERF_REQUIRE(xs); INERF_REQUIRE(sigmas); INERF_REQUIRE(rgbs);
    INERF_REQUIRE(grad_sigmas); INERF_REQUIRE(grad_rgbs); INERF_REQUIRE(grad_table);
    INERF_REQUIRE(grad_ws0); INERF_REQUIRE(grad_ws1); INERF_REQUIRE(grad_wc0); INERF_REQUIRE(grad_wc1); INERF_REQUIRE(grad_wc2);
    if (((uintptr_t)weights_bwd & 15u) || ((uintptr_t)xs & 15u) || ((uintptr_t)grad_table & 15u)) return INERF_ERR_ALIGN;
    const RgbBwdParams p{xyzs, (const uint4*)xs, sigmas, rgbs, grad_sigmas, grad_rgbs, B, (float2*)grad_table,
                         grad_ws0, grad_ws1, grad_wc0, grad_wc1, grad_wc2, weights_bwd};
    return launch_persistent(k_field_backward_rgb, B, kBwdThreads, RSm::bytes, (cudaStream_t)stream, *desc, p);
}
