// Device-side building blocks of the fused instance field (shared by field_fused.cu, render_fused.cu and
// train_fused.cu): hash-grid gathers for both tables straight into UMMA operand tiles, SH degree 4, and the
// tcgen05 MLP chain with its TMEM epilogues.
//
// Arithmetic contract (nerf/network_mask.py:119-158 under torch autocast, the reference's `-O` preset):
//   * hash encode: weights fp32, every product rounded to fp16, accumulated in fp16 (gridencoder.cu:161-185);
//   * every nn.Linear: fp16 operands, fp32 accumulation (TMEM), ONE rounding of the output to fp16;
//   * sigma = exp(float(h0)) in fp32 (activation.py:5-18), rgb = fp16(sigmoid(float(h))), logits = fp16 values.
//
// Table layout: the two encoders (encoder.embeddings, encoder_mask.embeddings) share level geometry, so the
// kernels read ONE interleaved fp16 table, 8 bytes per entry = (sigma.c0, sigma.c1, mask.c0, mask.c1), built by
// inerf_field_pack_tables.  One 8-byte gather per corner serves both encoders and halves the L2 sector traffic.
#pragma once
#include "common.cuh"
#include "umma.cuh"

namespace field {

constexpr int kTile = 128;        // samples per tile = TMEM lanes = UMMA M
constexpr int kThreads = 256;     // chain group: 8 warps, epilogues split by column half
constexpr uint32_t kLBO = 128;    // K-direction core-matrix stride (bytes)

// ---- packed weight blob (fp16, UMMA B-operand layout, see inerf_field_pack_weights) ----
struct WeightLayout {
    uint32_t s0, s1, c0, c1, c2, m0, m1, m2, total, Kp;
};
__host__ __device__ inline WeightLayout weight_layout(uint32_t K) {
    WeightLayout w;
    w.Kp = (K + 15u) & ~15u;
    w.s0 = 0;                       // [64 x 32]
    w.s1 = w.s0 + 64 * 32 * 2;      // [16 x 64]
    w.c0 = w.s1 + 16 * 64 * 2;      // [64 x 32]   (31 inputs + 1 zero column)
    w.c1 = w.c0 + 64 * 32 * 2;      // [64 x 64]
    w.c2 = w.c1 + 64 * 64 * 2;      // [16 x 64]   (3 outputs + 13 zero rows)
    w.m0 = w.c2 + 16 * 64 * 2;      // [64 x 48]   (47 inputs + 1 zero column)
    w.m1 = w.m0 + 64 * 48 * 2;      // [64 x 64]
    w.m2 = w.m1 + 64 * 64 * 2;      // [Kp x 64]
    w.total = w.m2 + w.Kp * 64 * 2;
    return w;
}

// ---- level geometry -----------------------------------------------------------------------
struct LevelGeom {
    float scale;
    uint32_t r1;       // resolution + 1
    uint32_t offset;   // first entry of the level
    uint32_t size;     // entries in the level
    uint32_t mode;     // 0 dense (index < size, never wraps), 1 hashed with power-of-two size (mask), 2 hashed generic (%)
    uint32_t mask;     // size - 1 (mode 1)
    uint32_t r1sq;     // r1 * r1 (mode 0)
    uint32_t pad;
};

// Operand-tile byte offsets of one pipeline stage + the weight blob (the hidden activations live in tensor memory).
struct ChainBufs {
    uint32_t a_es;   // [128 x 32] sigma-table features
    uint32_t a_ci;   // [128 x 32] SH16 | geo15 | 0
    uint32_t a_mi;   // [128 x 48] mask-table features 32 | geo15 | 0
    uint32_t w;      // weight blob
};
constexpr uint32_t kBytesEs = kTile * 32 * 2, kBytesCi = kTile * 32 * 2, kBytesMi = kTile * 48 * 2, kBytesH = kTile * 64 * 2;
constexpr uint32_t kStageBytes = kBytesEs + kBytesCi + kBytesMi;   // what the gather warps produce per tile (28 KB)
constexpr uint32_t sbo_of(uint32_t kdim) { return (kdim / 8) * 128; }

// TMEM column plan (fp32 accumulators)
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t D_a = 0;     // 64: sigma hidden / colour hidden
constexpr uint32_t D_b = 64;    // 64: mask hidden
constexpr uint32_t D_c = 128;   // 16: sigma-net output / rgb
constexpr uint32_t D_d = 144;   // up to 64: logits
// hidden activations as tcgen05 A operands IN TENSOR MEMORY (fp16 pairs, 32 columns per 64-wide layer): the epilogue of layer
// i writes them with tcgen05.st and the MMAs of layer i + 1 read them there -- they never touch shared memory
constexpr uint32_t A_h1 = 208;  // 32: sigma hidden, then colour hidden
constexpr uint32_t A_h2 = 240;  // 32: mask hidden
// (render kernel) the gathered INPUT tiles as tensor-memory operands too, two stages of 56 columns: sigma-table features 16 |
// SH 8 + geo 8 | mask-table features 16 + geo 8 (fp16 pairs)
constexpr uint32_t T_stage0 = 272, kStageCols = 56, S_es = 0, S_ci = 16, S_mi = 32;

__device__ __forceinline__ uint32_t pack_half2(__half a, __half b) {
    return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
}
__device__ __forceinline__ uint32_t h2_bits(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ __half2 bits_h2(uint32_t u) { return *reinterpret_cast<__half2*>(&u); }

// (lo, hi) fp32 -> packed fp16x2, round-to-nearest-even, ReLU folded into the conversion (relu commutes with rounding)
__device__ __forceinline__ uint32_t cvt_relu_f16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// level geometry exactly as the op-level kernel (gridencode.cu level_geom / gridencoder.cu:137-139)
__device__ __forceinline__ void init_levels(LevelGeom* lg, const int32_t* __restrict__ offsets, uint32_t L, float S, uint32_t H,
                                            uint32_t tid) {
    if (tid < L) {
        const uint32_t l = tid;
        LevelGeom g;
        g.offset = (uint32_t)offsets[l];
        g.size = (uint32_t)(offsets[l + 1] - offsets[l]);
        g.scale = __fmaf_rn(exp2f(__fmul_rn((float)l, S)), (float)H, -1.0f);
        const uint32_t resolution = (uint32_t)ceilf(g.scale) + 1;
        g.r1 = resolution + 1;
        g.r1sq = g.r1 * g.r1;
        // gridencoder.cu:66-84: the dense stride survives all three dimensions iff r1^3 <= size
        const bool dense = (g.r1 <= g.size) && (g.r1sq <= g.size) && ((uint64_t)g.r1sq * g.r1 <= g.size);
        g.mode = dense ? 0u : (((g.size & (g.size - 1)) == 0) ? 1u : 2u);
        g.mask = g.size - 1;
        g.pad = 0;
        lg[l] = g;
    }
}

// Class of the 4 consecutive levels [l0, l0 + 4) a gather thread encodes: all dense, all hashed with a power-of-two size
// (the hash-grid preset: levels 0..3 dense, 4..15 hashed), or mixed.  The levels of a gather warp are fixed, so the branch on
// the class is warp-uniform and the dense and hashed quarters run straight-line code without a mode branch per level.
constexpr uint32_t kLevelsMixed = 0, kLevelsDense = 1, kLevelsHashed = 2;
__device__ __forceinline__ uint32_t level_class4(const LevelGeom* lg, uint32_t l0) {
    const uint32_t m0 = lg[l0].mode, m1 = lg[l0 + 1].mode, m2 = lg[l0 + 2].mode, m3 = lg[l0 + 3].mode;
    if ((m0 | m1 | m2 | m3) == 0u) return kLevelsDense;
    if (m0 == 1u && m1 == 1u && m2 == 1u && m3 == 1u) return kLevelsHashed;
    return kLevelsMixed;
}

// (a ^ b) & m as one three-input LOP3 (left to itself the compiler forms x ^ y ^ z per corner and masks it separately)
__device__ __forceinline__ uint32_t xor_and(uint32_t a, uint32_t b, uint32_t m) {
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0x28;" : "=r"(r) : "r"(a), "r"(b), "r"(m));
    return r;
}

// Corner indices (relative to the level's first entry) and trilinear weights of one point at one level.
// w fp32 = (wx * wy) * wz in the reference's order (gridencoder.cu:161-185 / :283-301).
// kMode: the level's mode when the caller knows it (0 dense, 1 hashed with a power-of-two size); -1 reads g.mode.
template <int kMode = -1>
__device__ __forceinline__ void level_corners(const float x01[3], const LevelGeom& g, uint32_t idx[8], float w[8]) {
    float fr[3];
    uint32_t pg[3];
#pragma unroll
    for (int d = 0; d < 3; d++) {
        const float pos = __fmaf_rn(x01[d], g.scale, 0.5f);
        const float fl = floorf(pos);
        pg[d] = (uint32_t)fl;
        fr[d] = __fsub_rn(pos, fl);
    }
    const float wx[2] = {__fsub_rn(1.0f, fr[0]), fr[0]};
    const float wy[2] = {__fsub_rn(1.0f, fr[1]), fr[1]};
    const float wz[2] = {__fsub_rn(1.0f, fr[2]), fr[2]};
    // one warp-uniform branch per level (dense levels never wrap, hashed levels have power-of-two sizes)
    const uint32_t mode = kMode < 0 ? g.mode : (uint32_t)kMode;
    if (mode == 0) {
        const uint32_t y0 = pg[1] * g.r1, y1 = y0 + g.r1, z0 = pg[2] * g.r1sq, z1 = z0 + g.r1sq;
        const uint32_t b00 = pg[0] + y0 + z0, b10 = pg[0] + y1 + z0, b01 = pg[0] + y0 + z1, b11 = pg[0] + y1 + z1;
        idx[0] = b00; idx[1] = b00 + 1u; idx[2] = b10; idx[3] = b10 + 1u;
        idx[4] = b01; idx[5] = b01 + 1u; idx[6] = b11; idx[7] = b11 + 1u;
    } else {
        const uint32_t x0 = pg[0], x1 = pg[0] + 1u;
        const uint32_t y0 = pg[1] * 2654435761u, y1 = y0 + 2654435761u, z0 = pg[2] * 805459861u, z1 = z0 + 805459861u;
        const uint32_t h00 = y0 ^ z0, h10 = y1 ^ z0, h01 = y0 ^ z1, h11 = y1 ^ z1;
        idx[0] = xor_and(x0, h00, g.mask); idx[1] = xor_and(x1, h00, g.mask); idx[2] = xor_and(x0, h10, g.mask); idx[3] = xor_and(x1, h10, g.mask);
        idx[4] = xor_and(x0, h01, g.mask); idx[5] = xor_and(x1, h01, g.mask); idx[6] = xor_and(x0, h11, g.mask); idx[7] = xor_and(x1, h11, g.mask);
        if (kMode < 0 && mode == 2) {   // hashed level whose size is not a power of two (never produced by grid.py's level table; kept exact)
            idx[0] = (x0 ^ h00) % g.size; idx[1] = (x1 ^ h00) % g.size; idx[2] = (x0 ^ h10) % g.size; idx[3] = (x1 ^ h10) % g.size;
            idx[4] = (x0 ^ h01) % g.size; idx[5] = (x1 ^ h01) % g.size; idx[6] = (x0 ^ h11) % g.size; idx[7] = (x1 ^ h11) % g.size;
        }
    }
    const float w00 = __fmul_rn(wx[0], wy[0]), w10 = __fmul_rn(wx[1], wy[0]), w01 = __fmul_rn(wx[0], wy[1]), w11 = __fmul_rn(wx[1], wy[1]);
    w[0] = __fmul_rn(w00, wz[0]); w[1] = __fmul_rn(w10, wz[0]); w[2] = __fmul_rn(w01, wz[0]); w[3] = __fmul_rn(w11, wz[0]);
    w[4] = __fmul_rn(w00, wz[1]); w[5] = __fmul_rn(w10, wz[1]); w[6] = __fmul_rn(w01, wz[1]); w[7] = __fmul_rn(w11, wz[1]);
}

// One level of one point from the interleaved table: returns (sigma-table half2, mask-table half2) bit patterns.
// Per corner: product rounded to fp16; fp16 accumulation.
// __hadd2 (one rounding of the exact sum) equals the reference's half(float(acc) + float(p)): fp32 carries
// 24 >= 2*11+2 bits, so the double rounding is innocuous.
template <int kMode = -1>
__device__ __forceinline__ void encode_level(const float x01[3], const LevelGeom& g, const uint2* __restrict__ table, uint32_t& out_s,
                                             uint32_t& out_m) {
    uint32_t idx[8];
    float w[8];
    level_corners<kMode>(x01, g, idx, w);
    // Addresses: the entry index offset + idx is formed in 32 bits -- it is below offsets[L], an int32 -- so a corner costs one
    // 32-bit add and one widening shift-add onto the table base, not a 64-bit add of level base and index.  The x-neighbour of a
    // dense corner is the next entry (idx[c + 1] = idx[c] + 1 never wraps): the same address + 8 bytes, an immediate offset of
    // the load.
    const uint2* ptr[8];
    const uint32_t mode = kMode < 0 ? g.mode : (uint32_t)kMode;
#pragma unroll
    for (uint32_t c = 0; c < 8; c += 2) {
        ptr[c] = table + (g.offset + idx[c]);
        ptr[c + 1] = mode == 0 ? ptr[c] + 1 : table + (g.offset + idx[c + 1]);
    }
    uint2 v[8];
    // One 8-byte gather per corner.  (Tried and rejected on B200: fetching the x-neighbour with one aligned 16-byte gather when
    // it is entry a^1 -- 23 % fewer L1 sectors but LDG.128 scatters cost as many data-pipe wavefronts, +6 % time; DESIGN.md 4.1.)
    // (Also rejected on B200: L1::no_allocate for the finest levels -- 9.5 -> 14.5 ms per c2 frame: the x-neighbour of a corner
    // is fetched by the next instruction of the same thread and hits the line the first one allocated.)
#pragma unroll
    for (uint32_t c = 0; c < 8; c++) v[c] = __ldg(ptr[c]);
    __half2 as = __float2half2_rn(0.f), am = as;
#pragma unroll
    for (uint32_t c = 0; c < 8; c++) {
        const float2 fs = __half22float2(bits_h2(v[c].x));
        const float2 fm = __half22float2(bits_h2(v[c].y));
        // packed fp32 multiply (FMUL2, sm_100): same round-to-nearest products, half the multiply issue slots (-0.2 ms / c2 frame)
        const float2 ww = make_float2(w[c], w[c]);
        const float2 ps = __fmul2_rn(ww, fs), pm = __fmul2_rn(ww, fm);
        as = __hadd2(as, __floats2half2_rn(ps.x, ps.y));
        am = __hadd2(am, __floats2half2_rn(pm.x, pm.y));
    }
    out_s = h2_bits(as);
    out_m = h2_bits(am);
}

// Encode 4 consecutive levels [l0, l0+4) of one point, the 4 + 4 packed feature pairs returned in registers.
// (The class is read from shared memory per call: held in a register across the render kernel's tile loop it costs the
// 64-register gather warps a spill.)
__device__ __forceinline__ void encode4_regs(const float x01[3], bool oob, uint32_t l0, const LevelGeom* __restrict__ lg,
                                             const uint2* __restrict__ table, uint32_t (&fs)[4], uint32_t (&fm)[4]) {
    const uint32_t cls = level_class4(lg, l0);
    if (cls == kLevelsHashed) {
#pragma unroll
        for (uint32_t li = 0; li < 4; li++) encode_level<1>(x01, lg[l0 + li], table, fs[li], fm[li]);
    } else if (cls == kLevelsDense) {
#pragma unroll
        for (uint32_t li = 0; li < 4; li++) encode_level<0>(x01, lg[l0 + li], table, fs[li], fm[li]);
    } else {
#pragma unroll
        for (uint32_t li = 0; li < 4; li++) encode_level(x01, lg[l0 + li], table, fs[li], fm[li]);
    }
#pragma unroll
    for (uint32_t li = 0; li < 4; li++)
        if (oob) { fs[li] = 0u; fm[li] = 0u; }
}

// Same, stored as one 16-byte core-matrix row chunk per table of the shared-memory operand stage.
__device__ __forceinline__ void encode4(const float x01[3], bool oob, uint32_t l0, const LevelGeom* __restrict__ lg,
                                        const uint2* __restrict__ table, uint8_t* smem, uint32_t a_es, uint32_t a_mi, uint32_t row) {
    uint32_t fs[4], fm[4];
    encode4_regs(x01, oob, l0, lg, table, fs, fm);
    const uint32_t k0 = l0 * 2;
    *reinterpret_cast<uint4*>(smem + a_es + umma::tile_off(row, k0, kLBO, sbo_of(32))) = make_uint4(fs[0], fs[1], fs[2], fs[3]);
    *reinterpret_cast<uint4*>(smem + a_mi + umma::tile_off(row, k0, kLBO, sbo_of(48))) = make_uint4(fm[0], fm[1], fm[2], fm[3]);
}

// SH degree 4 (same polynomials as shencode.cu) rounded to fp16 into A_ci columns 0..15
__device__ __forceinline__ void sh16_pack(float x, float y, float z, uint32_t (&p)[8]) {
    float o[16];
    const float xy = x * y, xz = x * z, yz = y * z, x2 = x * x, y2 = y * y, z2 = z * z;
    o[0] = 0.28209479177387814f;
    o[1] = -0.48860251190291987f * y;
    o[2] = 0.48860251190291987f * z;
    o[3] = -0.48860251190291987f * x;
    o[4] = 1.0925484305920792f * xy;
    o[5] = -1.0925484305920792f * yz;
    o[6] = 0.94617469575755997f * z2 - 0.31539156525251999f;
    o[7] = -1.0925484305920792f * xz;
    o[8] = 0.54627421529603959f * x2 - 0.54627421529603959f * y2;
    o[9] = 0.59004358992664352f * y * (-3.0f * x2 + y2);
    o[10] = 2.8906114426405538f * xy * z;
    o[11] = 0.45704579946446572f * y * (1.0f - 5.0f * z2);
    o[12] = 0.3731763325901154f * z * (5.0f * z2 - 3.0f);
    o[13] = 0.45704579946446572f * x * (1.0f - 5.0f * z2);
    o[14] = 1.4453057213202769f * z * (x2 - y2);
    o[15] = 0.59004358992664352f * x * (-x2 + 3.0f * y2);
#pragma unroll
    for (int i = 0; i < 8; i++) p[i] = pack_half2(__float2half_rn(o[2 * i]), __float2half_rn(o[2 * i + 1]));
}
__device__ __forceinline__ void sh16_to_smem(float x, float y, float z, uint8_t* smem, uint32_t a_ci, uint32_t row) {
    uint32_t p[8];
    sh16_pack(x, y, z, p);
    *reinterpret_cast<uint4*>(smem + a_ci + umma::tile_off(row, 0, kLBO, sbo_of(32))) = make_uint4(p[0], p[1], p[2], p[3]);
    *reinterpret_cast<uint4*>(smem + a_ci + umma::tile_off(row, 8, kLBO, sbo_of(32))) = make_uint4(p[4], p[5], p[6], p[7]);
}

// ---- MMA issue (one thread) -------------------------------------------------------------------
// D[128 x N] (+)= A[128 x Kdim] * B[N x Kdim]^T ; A at smem+a_off (sbo_of(Kdim)), B at smem+b_off (sbo_of(Kdim))
__device__ __forceinline__ void issue_gemm(uint32_t smem_base, uint32_t a_off, uint32_t b_off, uint32_t Kdim, uint32_t N,
                                           uint32_t tmem_d) {
    const uint32_t idesc = umma::make_idesc_f16(128, N);
    const uint32_t hi = umma::desc_hi(sbo_of(Kdim));
    const uint32_t a_lo = umma::desc_lo(smem_base + a_off, kLBO), b_lo = umma::desc_lo(smem_base + b_off, kLBO);
#pragma unroll
    for (uint32_t k = 0; k < Kdim / 16; k++) umma::mma_f16_lohi(tmem_d, a_lo + k * (2 * kLBO >> 4), hi, b_lo + k * (2 * kLBO >> 4), hi, idesc, k > 0);
}

// A operand in tensor memory (columns tmem_a .. tmem_a + Kdim / 2), B [N x Kdim] in shared memory
__device__ __forceinline__ void issue_gemm_ts(uint32_t tmem_a, uint32_t smem_base, uint32_t b_off, uint32_t Kdim, uint32_t N, uint32_t tmem_d) {
    const uint32_t idesc = umma::make_idesc_f16(128, N);
    const uint32_t hi = umma::desc_hi(sbo_of(Kdim));
    const uint32_t b_lo = umma::desc_lo(smem_base + b_off, kLBO);
#pragma unroll
    for (uint32_t k = 0; k < Kdim / 16; k++) umma::mma_f16_ts(tmem_d, tmem_a + k * 8, b_lo + k * (2 * kLBO >> 4), hi, idesc, k > 0);
}

// general form: separate core-matrix row-group strides for A and B (operands that are column ranges of wider tiles)
__device__ __forceinline__ void issue_gemm2(uint32_t smem_base, uint32_t a_off, uint32_t sbo_a, uint32_t b_off, uint32_t sbo_b, uint32_t Kdim,
                                            uint32_t N, uint32_t tmem_d) {
    const uint32_t idesc = umma::make_idesc_f16(128, N);
    const uint32_t a_hi = umma::desc_hi(sbo_a), b_hi = umma::desc_hi(sbo_b);
    const uint32_t a_lo = umma::desc_lo(smem_base + a_off, kLBO), b_lo = umma::desc_lo(smem_base + b_off, kLBO);
#pragma unroll
    for (uint32_t k = 0; k < Kdim / 16; k++) umma::mma_f16_lohi(tmem_d, a_lo + k * (2 * kLBO >> 4), a_hi, b_lo + k * (2 * kLBO >> 4), b_hi, idesc, k > 0);
}
// D[128 x N] (+)= A^T * B, the reduction running over the 128 ROWS (samples) of two K-major tiles: A is [128 x 128 cols]
// (row-group stride sbo_a), B is [128 x N cols] (sbo_b).  The tiles are read as MN-major operands: same bytes, descriptor
// LBO = row-group stride, SBO = 128 (validated by scripts/probe/umma_probe_t.cu).
__device__ __forceinline__ void issue_gemm_tn(uint32_t smem_base, uint32_t a_off, uint32_t sbo_a, uint32_t b_off, uint32_t sbo_b, uint32_t N,
                                              uint32_t tmem_d, bool accumulate) {
    const uint32_t idesc = umma::make_idesc_f16(128, N) | (1u << 15) | (1u << 16);   // a_major = b_major = MN
    const uint32_t hi = umma::desc_hi(128);
    const uint32_t a_lo = umma::desc_lo(smem_base + a_off, sbo_a), b_lo = umma::desc_lo(smem_base + b_off, sbo_b);
#pragma unroll
    for (uint32_t k = 0; k < kTile / 16; k++)
        umma::mma_f16_lohi(tmem_d, a_lo + k * (2 * sbo_a >> 4), hi, b_lo + k * (2 * sbo_b >> 4), hi, idesc, accumulate || k > 0);
}

// ---- epilogues (chain group: 8 warps; warp w owns TMEM lanes 32*(w&3).., column half w>>2) ---------
// 64-wide hidden layer: TMEM accumulators -> fp16 round -> ReLU -> the next layer's A operand IN TENSOR MEMORY: columns
// tmem_a + 16 * (warp >> 2) .. + 16 of this thread's lane hold its 32 fp16 values as 16 packed pairs.  The caller waits
// (tmem_st_wait) before the group barrier.
__device__ __forceinline__ void epilogue_hidden_tmem(uint32_t tmem_d, uint32_t tmem_a, uint32_t tid) {
    const uint32_t warp = tid >> 5;
    const uint32_t lane_base = ((warp & 3u) * 32u) << 16, half = warp >> 2;
    uint32_t v[2][16];
    umma::tmem_ld16(tmem_d + lane_base + half * 32u, v[0]);
    umma::tmem_ld16(tmem_d + lane_base + half * 32u + 16u, v[1]);
    umma::tmem_ld_wait();
    uint32_t p[16];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        p[i] = cvt_relu_f16x2(__uint_as_float(v[0][2 * i]), __uint_as_float(v[0][2 * i + 1]));
        p[8 + i] = cvt_relu_f16x2(__uint_as_float(v[1][2 * i]), __uint_as_float(v[1][2 * i + 1]));
    }
    umma::tmem_st16(tmem_a + lane_base + half * 16u, p);
}

// sigma-net output (16 columns): h0 -> sigma (returned, valid for warps 0..3), geo15 -> A_ci[:,16:32] and A_mi[:,32:48]
__device__ __forceinline__ float epilogue_sigma(uint32_t tmem_base, uint8_t* smem, const ChainBufs& b, float density_scale, uint32_t tid) {
    const uint32_t warp = tid >> 5, lane = tid & 31;
    float sigma = 0.f;
    if (warp < 4) {
        const uint32_t row = warp * 32u + lane;
        uint32_t v[16];
        umma::tmem_ld16(tmem_base + D_c + ((warp * 32u) << 16), v);
        umma::tmem_ld_wait();
        __half h[16];
#pragma unroll
        for (int i = 0; i < 16; i++) h[i] = __float2half_rn(__uint_as_float(v[i]));
        sigma = __fmul_rn(expf(__half2float(h[0])), density_scale);
        const __half z = __float2half_rn(0.f);
        const uint4 g0 = make_uint4(pack_half2(h[1], h[2]), pack_half2(h[3], h[4]), pack_half2(h[5], h[6]), pack_half2(h[7], h[8]));
        const uint4 g1 = make_uint4(pack_half2(h[9], h[10]), pack_half2(h[11], h[12]), pack_half2(h[13], h[14]), pack_half2(h[15], z));
        *reinterpret_cast<uint4*>(smem + b.a_ci + umma::tile_off(row, 16, kLBO, sbo_of(32))) = g0;
        *reinterpret_cast<uint4*>(smem + b.a_ci + umma::tile_off(row, 24, kLBO, sbo_of(32))) = g1;
        *reinterpret_cast<uint4*>(smem + b.a_mi + umma::tile_off(row, 32, kLBO, sbo_of(48))) = g0;
        *reinterpret_cast<uint4*>(smem + b.a_mi + umma::tile_off(row, 40, kLBO, sbo_of(48))) = g1;
    }
    return sigma;
}

// Same with the geo columns going to the TENSOR-MEMORY input stage (`stage` = its first column): A_ci columns 8..15, A_mi 16..23
__device__ __forceinline__ float epilogue_sigma_tmem(uint32_t tmem_base, uint32_t stage, float density_scale, uint32_t tid) {
    const uint32_t warp = tid >> 5;
    float sigma = 0.f;
    if (warp < 4) {
        uint32_t v[16];
        umma::tmem_ld16(tmem_base + D_c + ((warp * 32u) << 16), v);
        umma::tmem_ld_wait();
        __half h[16];
#pragma unroll
        for (int i = 0; i < 16; i++) h[i] = __float2half_rn(__uint_as_float(v[i]));
        sigma = __fmul_rn(expf(__half2float(h[0])), density_scale);
        const __half z = __float2half_rn(0.f);
        const uint32_t g[8] = {pack_half2(h[1], h[2]), pack_half2(h[3], h[4]), pack_half2(h[5], h[6]), pack_half2(h[7], h[8]),
                               pack_half2(h[9], h[10]), pack_half2(h[11], h[12]), pack_half2(h[13], h[14]), pack_half2(h[15], z)};
        umma::tmem_st8(stage + ((warp * 32u) << 16) + S_ci + 8, g);
        umma::tmem_st8(stage + ((warp * 32u) << 16) + S_mi + 16, g);
    }
    return sigma;
}

// colour output: 3 of 16 columns -> fp16 round -> sigmoid (fp32) -> fp16 round.  Valid for warps 0..3.
__device__ __forceinline__ void epilogue_rgb(uint32_t tmem_base, float rgb[3], uint32_t tid) {
    const uint32_t warp = tid >> 5;
    uint32_t v[16];
    umma::tmem_ld16(tmem_base + D_c + (((warp & 3u) * 32u) << 16), v);
    umma::tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const float h = __half2float(__float2half_rn(__uint_as_float(v[i])));
        rgb[i] = __half2float(__float2half_rn(__fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-h)))));
    }
}

// The whole MLP chain for one 128-sample tile whose encoder features / SH are already in shared memory and visible
// to the async proxy.  Executed by the 256 threads of the chain group (`tid` = index inside the group, thread 0 issues).
// `sync()` is a barrier over exactly those 256 threads.  After the layer-0 colour/mask MMAs have been issued the
// issuer commits to `release_bar` (if not null): the gathered operand tiles may then be overwritten.
// After return: D_c holds the colour pre-activations, D_d the logits (if with_masks); returns sigma for warps 0..3.
// `on_sigma(sigma)` runs in every thread right after the sigma-net epilogue and before the next barrier.
// kInTmem: the input tiles are tensor-memory operands as well (`in_stage` = first column of the stage, render kernel).
template <bool kInTmem = false, typename Sync, typename OnSigma>
__device__ __forceinline__ float mlp_chain(uint8_t* smem, const ChainBufs& b, uint32_t tmem_base, uint64_t* bar, uint32_t& phase, uint32_t K,
                                           float density_scale, bool with_masks, uint32_t tid, uint64_t* release_bar, Sync&& sync,
                                           OnSigma&& on_sigma, uint32_t in_stage = 0) {
    const uint32_t sbase = umma::smem_u32(smem);
    const WeightLayout wl = weight_layout(K);
    const bool issue_warp = tid < 32;   // warp 0 of the chain group; one elected lane issues
    // sigma layer 0
    if (issue_warp && umma::elect_one()) {
        umma::fence_after_sync();
        if (kInTmem) issue_gemm_ts(in_stage + S_es, sbase, b.w + wl.s0, 32, 64, tmem_base + D_a);
        else issue_gemm(sbase, b.a_es, b.w + wl.s0, 32, 64, tmem_base + D_a);
        umma::commit(bar);
    }
    __syncwarp();
    umma::mbar_wait(bar, phase); phase ^= 1u;
    umma::fence_after_sync();
    epilogue_hidden_tmem(tmem_base + D_a, tmem_base + A_h1, tid);
    umma::tmem_st_wait(); umma::fence_before_sync();
    sync();
    // sigma layer 1
    if (issue_warp && umma::elect_one()) {
        umma::fence_after_sync();
        issue_gemm_ts(tmem_base + A_h1, sbase, b.w + wl.s1, 64, 16, tmem_base + D_c);
        umma::commit(bar);
    }
    __syncwarp();
    umma::mbar_wait(bar, phase); phase ^= 1u;
    umma::fence_after_sync();
    const float sigma = kInTmem ? epilogue_sigma_tmem(tmem_base, in_stage, density_scale, tid) : epilogue_sigma(tmem_base, smem, b, density_scale, tid);
    on_sigma(sigma);
    if (kInTmem) umma::tmem_st_wait(); else umma::fence_async_smem();
    umma::fence_before_sync();
    sync();
    // colour layer 0 + mask layer 0
    if (issue_warp && umma::elect_one()) {
        umma::fence_after_sync();
        if (kInTmem) {
            issue_gemm_ts(in_stage + S_ci, sbase, b.w + wl.c0, 32, 64, tmem_base + D_a);
            if (with_masks) issue_gemm_ts(in_stage + S_mi, sbase, b.w + wl.m0, 48, 64, tmem_base + D_b);
        } else {
            issue_gemm(sbase, b.a_ci, b.w + wl.c0, 32, 64, tmem_base + D_a);
            if (with_masks) issue_gemm(sbase, b.a_mi, b.w + wl.m0, 48, 64, tmem_base + D_b);
        }
        umma::commit(bar);
        if (release_bar) umma::commit(release_bar);
    }
    __syncwarp();
    umma::mbar_wait(bar, phase); phase ^= 1u;
    umma::fence_after_sync();
    epilogue_hidden_tmem(tmem_base + D_a, tmem_base + A_h1, tid);
    if (with_masks) epilogue_hidden_tmem(tmem_base + D_b, tmem_base + A_h2, tid);
    umma::tmem_st_wait(); umma::fence_before_sync();
    sync();
    // colour layer 1 + mask layer 1
    if (issue_warp && umma::elect_one()) {
        umma::fence_after_sync();
        issue_gemm_ts(tmem_base + A_h1, sbase, b.w + wl.c1, 64, 64, tmem_base + D_a);
        if (with_masks) issue_gemm_ts(tmem_base + A_h2, sbase, b.w + wl.m1, 64, 64, tmem_base + D_b);
        umma::commit(bar);
    }
    __syncwarp();
    umma::mbar_wait(bar, phase); phase ^= 1u;
    umma::fence_after_sync();
    epilogue_hidden_tmem(tmem_base + D_a, tmem_base + A_h1, tid);
    if (with_masks) epilogue_hidden_tmem(tmem_base + D_b, tmem_base + A_h2, tid);
    umma::tmem_st_wait(); umma::fence_before_sync();
    sync();
    // colour layer 2 + mask layer 2
    if (issue_warp && umma::elect_one()) {
        umma::fence_after_sync();
        issue_gemm_ts(tmem_base + A_h1, sbase, b.w + wl.c2, 64, 16, tmem_base + D_c);
        if (with_masks) issue_gemm_ts(tmem_base + A_h2, sbase, b.w + wl.m2, 64, wl.Kp, tmem_base + D_d);
        umma::commit(bar);
    }
    __syncwarp();
    umma::mbar_wait(bar, phase); phase ^= 1u;
    umma::fence_after_sync();
    return sigma;
}

// Density only (NeRFNetwork.density, nerf/network_mask.py:160-178, as the occupancy-grid update calls it): the sigma-net
// half of the chain above -- 32 -> 64 ReLU -> 16, sigma = exp(fp16(h0)) in fp32, unscaled.  Returns sigma for warps 0..3.
// The gathered stage is released (commit to `release_bar`) as soon as the layer-0 MMAs have been issued.
template <typename Sync>
__device__ __forceinline__ float sigma_chain(uint8_t* smem, const ChainBufs& b, uint32_t tmem_base, uint64_t* bar, uint32_t& phase, uint32_t K,
                                             uint32_t tid, uint64_t* release_bar, Sync&& sync) {
    const uint32_t sbase = umma::smem_u32(smem);
    const WeightLayout wl = weight_layout(K);
    const bool issue_warp = tid < 32;   // warp 0 of the chain group; one elected lane issues
    if (issue_warp && umma::elect_one()) {
        umma::fence_after_sync();
        issue_gemm(sbase, b.a_es, b.w + wl.s0, 32, 64, tmem_base + D_a);
        umma::commit(bar);
        if (release_bar) umma::commit(release_bar);
    }
    __syncwarp();
    umma::mbar_wait(bar, phase); phase ^= 1u;
    umma::fence_after_sync();
    epilogue_hidden_tmem(tmem_base + D_a, tmem_base + A_h1, tid);
    umma::tmem_st_wait(); umma::fence_before_sync();
    sync();
    if (issue_warp && umma::elect_one()) {
        umma::fence_after_sync();
        issue_gemm_ts(tmem_base + A_h1, sbase, b.w + wl.s1, 64, 16, tmem_base + D_c);
        umma::commit(bar);
    }
    __syncwarp();
    umma::mbar_wait(bar, phase); phase ^= 1u;
    umma::fence_after_sync();
    float sigma = 0.f;
    const uint32_t warp = tid >> 5;
    if (warp < 4) {
        uint32_t v[16];
        umma::tmem_ld16(tmem_base + D_c + ((warp * 32u) << 16), v);
        umma::tmem_ld_wait();
        sigma = expf(__half2float(__float2half_rn(__uint_as_float(v[0]))));
    }
    return sigma;
}

// weights -> smem (all threads of the CTA)
__device__ __forceinline__ void load_weights(uint8_t* smem, uint32_t w_off, const void* weights, uint32_t K) {
    const WeightLayout wl = weight_layout(K);
    const uint4* wsrc = reinterpret_cast<const uint4*>(weights);
    uint4* wdst = reinterpret_cast<uint4*>(smem + w_off);
    for (uint32_t i = threadIdx.x; i < wl.total / 16; i += blockDim.x) wdst[i] = __ldg(wsrc + i);
}

int validate(const inerf_field_desc* d);

// Host: launch a persistent field kernel -- one CTA per SM, or one per tile when there are fewer tiles of `rows` -- with `smem`
// bytes of dynamic shared memory.  The attribute is per device and cheap to set, so every launch sets it.
template <typename... P, typename... A>
inline int launch_persistent(void (*kernel)(P...), uint32_t rows, uint32_t threads, uint32_t smem, cudaStream_t stream, A... args) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const uint32_t num_tiles = (rows + kTile - 1) / kTile, sms = (uint32_t)device_sm_count();
    kernel<<<num_tiles < sms ? num_tiles : sms, threads, smem, stream>>>(args...);
    INERF_LAUNCH_CHECK();
    return INERF_OK;
}

}  // namespace field
