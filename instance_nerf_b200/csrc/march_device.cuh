// Occupancy-grid DDA shared by the marching kernels (raymarch.cu) and the fused renderer (render_fused.cu).
// See raymarch.cu for the float-semantics contract (explicit round-to-nearest intrinsics where nvcc
// contracts the reference's expressions; bit-identical sample stream to raymarching.cu:311-480, 958-1063).
#pragma once
#include "common.cuh"

namespace march {

constexpr float kSqrt3 = 1.7320508075688772f;

// ---- Morton (raymarching.cu:56-81) -----------------------------------------
__host__ __device__ __forceinline__ uint32_t expand_bits(uint32_t v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
__host__ __device__ __forceinline__ uint32_t morton3D_enc(uint32_t x, uint32_t y, uint32_t z) {
    return expand_bits(x) | (expand_bits(y) << 1) | (expand_bits(z) << 2);
}
__host__ __device__ __forceinline__ uint32_t morton3D_dec(uint32_t x) {
    x = x & 0x49249249u;
    x = (x | (x >> 2)) & 0xc30c30c3u;
    x = (x | (x >> 4)) & 0x0f00f00fu;
    x = (x | (x >> 8)) & 0xff0000ffu;
    x = (x | (x >> 16)) & 0x0000ffffu;
    return x;
}

// frexpf exponent clamped to [0, C-1] (raymarching.cu:42-54).  For the clamped
// result the biased-exponent field is enough: zero / denormals give <= 0.
__device__ __forceinline__ int clamped_exponent(float mx, int C) {
    const int e = (int)((__float_as_uint(mx) >> 23) & 0xffu) - 126;
    return min(C - 1, max(0, e));
}

// Occupancy cell of point (x, y, z) at cascade `level` (raymarching.cu:1022-1033): the cell coordinates n (also returned,
// with mip_bound = min(2^level, bound), for the DDA's exit test) and the bitfield index level * H^3 + morton(n).  Two latency
// cuts that are exact: 1 / mip_bound is a power of two (exponent arithmetic) unless the cascade is clipped to `bound`
// (precomputed quotient rbound), and the index is formed in integers whenever the reference's float expression is exact,
// i.e. C * H^3 <= 2^24 (H3i != 0).  Shared by Walk::eval_cell and the volume extraction (field_fused.cu).
__device__ __forceinline__ uint32_t cell_index(float x, float y, float z, int level, float bound, float rbound, float Hf, float Hm1,
                                               uint32_t H3i, float H3, float& mip_bound, int& nx, int& ny, int& nz) {
    const float pow2 = __uint_as_float((uint32_t)(127 + level) << 23);
    const bool clipped = !(pow2 <= bound);   // fminf(2^level, bound) picks bound
    mip_bound = clipped ? bound : pow2;
    const float mip_rbound = clipped ? rbound : __uint_as_float((uint32_t)(127 - level) << 23);
    const float hH = __fmul_rn(0.5f, Hf);
    nx = (int)clampf(__fmul_rn(__fmaf_rn(x, mip_rbound, 1.0f), hH), 0.0f, Hm1);
    ny = (int)clampf(__fmul_rn(__fmaf_rn(y, mip_rbound, 1.0f), hH), 0.0f, Hm1);
    nz = (int)clampf(__fmul_rn(__fmaf_rn(z, mip_rbound, 1.0f), hH), 0.0f, Hm1);
    return H3i ? (uint32_t)level * H3i + morton3D_enc(nx, ny, nz) : (uint32_t)__fmaf_rn((float)level, H3, (float)morton3D_enc(nx, ny, nz));
}

struct Walk {
    float ox, oy, oz, dx, dy, dz, rdx, rdy, rdz;
    float sx, sy, sz;  // 0.5 * sign(d)
    float bound, dt_gamma, dt_min, dt_max, rH, H3, Hf, Hm1, far;
    float rbound;      // 1 / bound (for the cascade whose extent is clipped to `bound`)
    uint32_t H3i;      // H^3; 0 = the cell index does not fit a float exactly (C * H^3 > 2^24): keep the float expression
    int C;
    const uint8_t* __restrict__ grid;
    // render-kernel accelerators (results identical to reading grid[] directly):
    //  * `coarse`: shared-memory bitmap, one bit per aligned 4x4x4 block of cells (= 64 consecutive Morton
    //    indices = one 8-byte word of the bitfield), 0 = the whole block is empty -> no global load;
    //  * the last 8-byte word read is kept in registers (consecutive samples mostly stay inside one block).
    const uint32_t* coarse = nullptr;
    unsigned long long cword = 0ull;
    uint32_t cblk = 0xffffffffu;

    bool words = true;   // the bitfield may be read as aligned 8-byte words (set by init)

    __device__ __forceinline__ bool occupied_cached(uint32_t index) {
        if (!words) return (grid[index >> 3] >> (index & 7u)) & 1u;
        const uint32_t blk = index >> 6;
        if (coarse != nullptr && !((coarse[blk >> 5] >> (blk & 31u)) & 1u)) return false;
        if (blk != cblk) {
            cword = __ldg(reinterpret_cast<const unsigned long long*>(grid) + blk);
            cblk = blk;
        }
        return (cword >> (index & 63u)) & 1ull;
    }

    __device__ __forceinline__ void init(const float* __restrict__ o, const float* __restrict__ d,
                                         const uint8_t* __restrict__ g, float bound_, float dt_gamma_,
                                         uint32_t max_steps, uint32_t C_, uint32_t H, float far_) {
        ox = o[0]; oy = o[1]; oz = o[2];
        dx = d[0]; dy = d[1]; dz = d[2];
        rdx = __fdiv_rn(1.0f, dx); rdy = __fdiv_rn(1.0f, dy); rdz = __fdiv_rn(1.0f, dz);
        sx = copysignf(0.5f, dx); sy = copysignf(0.5f, dy); sz = copysignf(0.5f, dz);
        bound = bound_; dt_gamma = dt_gamma_;
        Hf = (float)H; Hm1 = (float)(H - 1);
        rH = __fdiv_rn(1.0f, Hf);
        H3 = (float)(H * H * H);
        dt_min = __fdiv_rn(2.0f * kSqrt3, (float)max_steps);                                   // :345
        dt_max = __fdiv_rn(__fmul_rn(2.0f * kSqrt3, (float)(1 << (C_ - 1))), Hf);              // :346
        far = far_; C = (int)C_; grid = g;
        rbound = __fdiv_rn(1.0f, bound_);
        H3i = ((uint64_t)C_ * H * H * H <= (1ull << 24)) ? H * H * H : 0u;
        words = (((uintptr_t)g & 7u) == 0) && (((uint64_t)C_ * H * H * H) & 63u) == 0;
        cblk = 0xffffffffu;
    }
    __device__ __forceinline__ float step_size(float t) const { return clampf(__fmul_rn(t, dt_gamma), dt_min, dt_max); }

    // One DDA walk (raymarching.cu:359-400 / :427-479 / :1008-1062): the reference's loop, one eval_cell per visited cell.
    // WRITE: false = count only, true = write samples.  `ts` (optional, count pass): the parameter t of every sample is
    // recorded there, so that the samples can later be expanded in parallel without a second walk.
    template <bool WRITE>
    __device__ __forceinline__ uint32_t run(float t, uint32_t limit, float* __restrict__ xyzs, float* __restrict__ dirs,
                                            float* __restrict__ deltas, float* __restrict__ ts = nullptr) {
        uint32_t step = 0;
        float last_t = t;
        while (t < far && step < limit) {
            float x, y, z, dt, tt;
            const float t_sample = t;
            if (eval_cell(t, x, y, z, dt, tt)) {   // occupied: t has been advanced past the sample
                if (ts) ts[step] = t_sample;
                if (WRITE) {
                    xyzs[0] = x; xyzs[1] = y; xyzs[2] = z;
                    dirs[0] = dx; dirs[1] = dy; dirs[2] = dz;
                    deltas[0] = dt;
                    deltas[1] = __fsub_rn(t, last_t);
                    last_t = t;
                    xyzs += 3; dirs += 3; deltas += 2;
                }
                step++;
            } else {
                do { t = __fadd_rn(t, step_size(t)); } while (t < tt);
            }
        }
        return step;
    }

    // ONE cell evaluation of the DDA at parameter t (used by the render kernel's per-lane state machine).
    // Occupied: returns true with the sample (x, y, z, dt) and t advanced past it.  Empty: returns false with `tt` = the
    // parameter at which the ray leaves this cell; the caller then does `do { t += step_size(t); } while (t < tt);`.
    // Same values as run() / the reference (the cell lookup is cell_index above).
    __device__ __forceinline__ bool eval_cell(float& t, float& x, float& y, float& z, float& dt, float& tt) {
        x = clampf(__fmaf_rn(t, dx, ox), -bound, bound);
        y = clampf(__fmaf_rn(t, dy, oy), -bound, bound);
        z = clampf(__fmaf_rn(t, dz, oz), -bound, bound);
        dt = step_size(t);
        const float mx = fmaxf(fabsf(x), fmaxf(fabsf(y), fabsf(z)));
        const float md = __fmul_rn(__fmul_rn(dt, Hf), 0.5f);
        const int level = max(clamped_exponent(mx, C), clamped_exponent(md, C));
        float mip_bound;
        int nx, ny, nz;
        const uint32_t index = cell_index(x, y, z, level, bound, rbound, Hf, Hm1, H3i, H3, mip_bound, nx, ny, nz);
        if (occupied_cached(index)) {
            t = __fadd_rn(t, dt);
            return true;
        }
        const float tx = __fmul_rn(__fmaf_rn(__fmaf_rn(__fmul_rn(__fadd_rn(__fadd_rn((float)nx, 0.5f), sx), rH), 2.0f, -1.0f), mip_bound, -x), rdx);
        const float ty = __fmul_rn(__fmaf_rn(__fmaf_rn(__fmul_rn(__fadd_rn(__fadd_rn((float)ny, 0.5f), sy), rH), 2.0f, -1.0f), mip_bound, -y), rdy);
        const float tz = __fmul_rn(__fmaf_rn(__fmaf_rn(__fmul_rn(__fadd_rn(__fadd_rn((float)nz, 0.5f), sz), rH), 2.0f, -1.0f), mip_bound, -z), rdz);
        tt = __fadd_rn(t, fmaxf(0.0f, fminf(tx, fminf(ty, tz))));
        return false;
    }
};


}  // namespace march
