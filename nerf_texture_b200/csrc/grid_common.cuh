// grid_common.cuh — level table, index arithmetic and the lane-pair gather of the multi-resolution grid encoder,
// shared by grid.cu (stand-alone encoder) and field.cu (encoder fused with the MLPs).
#pragma once

#include "common.cuh"

namespace ntx {

constexpr int kFieldMaxLevels = 32;      // levels the fused kernels (field.cu, texture_field.cu) keep in their shared level table

// ---------------------------------------------------------------------------------------------------- level table
struct GridLevel {
    float scale;         // exp2f(level*S)*H - 1                      gridencoder.cu:126
    uint32_t res;        // ceil(scale)+1                              :127
    uint32_t hs;         // hashmap_size = offsets[l+1]-offsets[l]     :125
    uint32_t offset;     // offsets[l]
    uint32_t sy, sz;     // dense strides of y and z (0 if that dimension is dropped by the early loop exit, :60)
    uint32_t use_hash;   // gridtype==0 && stride>hashmap_size         :67
    uint32_t mask;       // hs-1 if hs is a power of two else 0 (then a real modulo is used)
};

__device__ __forceinline__ float level_scale(uint32_t level, float S, uint32_t H) {
    // written exactly as the reference writes it so that nvcc contracts it the same way (one FMA after exp2f)
    return exp2f(level * S) * H - 1.0f;
}

template <uint32_t D>
__device__ __forceinline__ GridLevel make_level(const int* __restrict__ offsets, uint32_t level, float S, uint32_t H,
                                                uint32_t gridtype, bool align) {
    GridLevel g;
    g.scale = level_scale(level, S, H);
    g.res = (uint32_t)ceilf(g.scale) + 1;
    g.offset = (uint32_t)offsets[level];
    g.hs = (uint32_t)offsets[level + 1] - g.offset;
    const uint32_t R = align ? g.res : g.res + 1;
    uint32_t stride = 1;  // uint32 wrap-around on purpose: mirrors get_grid_index (:56-63)
    g.sy = g.sz = 0;
    // d = 0 is always taken (stride 1 <= hs)
    stride *= R;
    if (D > 1 && stride <= g.hs) { g.sy = stride; stride *= R; if (D > 2 && stride <= g.hs) { g.sz = stride; stride *= R; } }
    g.use_hash = (gridtype == 0 && stride > g.hs) ? 1u : 0u;
    g.mask = ((g.hs & (g.hs - 1)) == 0) ? g.hs - 1 : 0u;
    return g;
}

__device__ __forceinline__ uint32_t wrap_index(const GridLevel& g, uint32_t index) {
    return g.mask ? (index & g.mask) : (index % g.hs);
}

template <uint32_t D>
__device__ __forceinline__ uint32_t corner_index(const GridLevel& g, const uint32_t* p) {
    uint32_t index;
    if (g.use_hash) {
        index = p[0];  // primes[0] == 1
        if (D > 1) index ^= p[1] * 2654435761u;
        if (D > 2) index ^= p[2] * 805459861u;
    } else {
        index = p[0];
        if (D > 1) index += p[1] * g.sy;
        if (D > 2) index += p[2] * g.sz;
    }
    return wrap_index(g, index);
}

// out-of-line so that the compiler keeps the (almost never taken) modulo behind a real branch instead of if-converting a
// 20-instruction integer division into every corner of every level
static __device__ __noinline__ uint32_t slow_umod(uint32_t a, uint32_t b) { return a % b; }

// ---------------------------------------------------------------------------------------------------- lane-pair gather
// per-level record of the pair gather: 32 bytes = two LDS.128, with the level's table pointer resolved once per CTA so that
// a corner address is a single IMAD.WIDE (index * elem + base)
struct PairLevel {
    float scale;
    uint32_t hs, sy, sz;
    const void* base;      // grid + offset * 2
    uint32_t mask;
    uint32_t kind;         // bit 0: hashed, power-of-two table, scale < 2^22 (the hot path of the fine levels)
                           // bit 1: dense (all three strides taken: plain x + y*R + z*R^2 addressing, a wrap needs a coordinate == R)
                           // bit 2: use_hash (for the generic path, taken when neither fast bit is set)
    __device__ __forceinline__ uint32_t use_hash() const { return kind >> 2; }
};
template <typename scalar_t>
__device__ __forceinline__ PairLevel make_pair_level(const GridLevel& g, const scalar_t* __restrict__ grid) {
    PairLevel q;
    q.scale = g.scale; q.hs = g.hs; q.sy = g.sy; q.sz = g.sz; q.mask = g.mask;
    q.base = grid + (size_t)g.offset * 2;
    q.kind = (g.use_hash && g.mask && g.scale < 4194304.0f) ? 1u : 0u;
    // sy = R, sz = R^2; the level is a plain dense R^3 block iff the third stride was taken and R^3 fits the level
    if (!g.use_hash && g.sz != 0 && (uint64_t)g.sz * g.sy <= g.hs && g.scale < 4194304.0f) q.kind |= 2u;
    q.kind |= g.use_hash << 2;
    return q;
}

// D = 3, C = 2.  Raw table element = 2 scalars: u32 for half2, u64 for float2.
template <typename scalar_t> struct Elem2;
template <> struct Elem2<__half> {
    using raw = uint32_t;
    using accum = __half2;
    // plain read-only loads: L1::no_allocate on the big hashed levels was measured 2-4x SLOWER (profiles/r01_summary.md)
    static __device__ __forceinline__ raw load(const void* p) { return __ldg(reinterpret_cast<const raw*>(p)); }
    static __device__ __forceinline__ raw xchg(raw v) { return __shfl_xor_sync(0xffffffffu, v, 1); }
    static __device__ __forceinline__ accum zero() { return __floats2half2_rn(0.f, 0.f); }
    static __device__ __forceinline__ void add(accum& r, float w, raw v) {
        // reference (c10::Half): p = half(w * float(g)); r = half(float(r) + float(p)).  The second step equals one
        // correctly-rounded fp16 add for every pair of finite halves (checked exhaustively, tests/test_oracle_cpu.py),
        // so HADD2 does both channels in one instruction.
        const float2 f = half2_bits_to_float2(v);
        r = __hadd2(r, __floats2half2_rn(w * f.x, w * f.y));
    }
    static __device__ __forceinline__ raw pack(const accum& r) { return *reinterpret_cast<const uint32_t*>(&r); }
};
template <> struct Elem2<float> {
    using raw = uint64_t;
    struct accum { float a, b; };
    static __device__ __forceinline__ raw load(const void* p) { return __ldg(reinterpret_cast<const unsigned long long*>(p)); }
    static __device__ __forceinline__ raw xchg(raw v) { return __shfl_xor_sync(0xffffffffu, v, 1); }
    static __device__ __forceinline__ accum zero() { return {0.f, 0.f}; }
    static __device__ __forceinline__ void add(accum& r, float w, raw v) {
        const float lo = __uint_as_float((uint32_t)v), hi = __uint_as_float((uint32_t)(v >> 32));
        r.a = __fmaf_rn(w, lo, r.a);
        r.b = __fmaf_rn(w, hi, r.b);
    }
    static __device__ __forceinline__ raw pack(const accum& r) { return (uint64_t)__float_as_uint(r.a) | ((uint64_t)__float_as_uint(r.b) << 32); }
};

// 0: out of range (features 0, gridencoder.cu:112-121), 1: live, 2: a coordinate is NaN (features NaN, loads suppressed)
__device__ __forceinline__ uint32_t sample_class(float x, float y, float z) {
    const bool inside = (x >= 0 && x <= 1) && (y >= 0 && y <= 1) && (z >= 0 && z <= 1);   // false for NaN
    const bool nan = (x != x) || (y != y) || (z != z);
    return inside ? 1u : (nan ? 2u : 0u);
}
template <typename raw> __device__ __forceinline__ raw nan_features();
template <> __device__ __forceinline__ uint32_t nan_features<uint32_t>() { return 0x7fff7fffu; }                 // two fp16 NaNs
template <> __device__ __forceinline__ uint64_t nan_features<uint64_t>() { return 0x7fc000007fc00000ull; }     // two fp32 NaNs

// A lane pair (lanes 2i, 2i+1) owns one sample; lane p (= lane & 1) gathers the four corners whose x bit is p.
// Processes the 4 consecutive levels lv[0..3]; on return lane p holds the finished features of levels 2p and 2p+1
// (packed[0], packed[1]), accumulated over the 8 corners in exactly the reference's order and rounding.
// Must be called by all 32 lanes of the warp (uses shuffles).  `live` = sample valid and inside [0,1]^3; coordinates of
// non-live samples must have been forced to 0 by the caller (their loads then hit entry 0 of each level and are discarded).
// Callers classify with sample_class(): a NaN coordinate is NOT live (its corner indices would be arbitrary 32-bit values and
// the dense-level fast path could read outside the table) but, as in the reference — whose `x < 0 || x > 1` test lets NaN
// through and whose weights then are NaN (gridencoder.cu:110-121) — its features come out as NaN, not as zeros.
template <typename scalar_t>
__device__ __forceinline__ void pair_gather4(const float x, const float y, const float z, const bool live, const uint32_t p, const PairLevel* __restrict__ lv,
                                             const float half_off,
                                             typename Elem2<scalar_t>::raw packed[2]) {
    using E = Elem2<scalar_t>;
    using raw = typename E::raw;
    raw v[4][4];
    float fx[4], fy[4], fz[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const PairLevel g = lv[j];
        const float px = __fmaf_rn(x, g.scale, half_off), py = __fmaf_rn(y, g.scale, half_off), pz = __fmaf_rn(z, g.scale, half_off);
        const raw* gl = static_cast<const raw*>(g.base);
        if (g.kind & 1u) {           // hashed level, power-of-two table: the hot path for fine levels
            // floor of a non-negative float < 2^22 without the quarter-rate FRND/F2I: px + 2^23 rounded down has floor(px)
            // in its mantissa, and subtracting 2^23 again is exact  (same values as floorf / (uint32_t) below)
            const float bx = __fadd_rd(px, 8388608.0f), by = __fadd_rd(py, 8388608.0f), bz = __fadd_rd(pz, 8388608.0f);
            fx[j] = px - (bx - 8388608.0f); fy[j] = py - (by - 8388608.0f); fz[j] = pz - (bz - 8388608.0f);
            const uint32_t cx = (__float_as_uint(bx) - 0x4b000000u) + p;
            const uint32_t ty0 = (__float_as_uint(by) - 0x4b000000u) * 2654435761u, ty1 = ty0 + 2654435761u;
            const uint32_t tz0 = (__float_as_uint(bz) - 0x4b000000u) * 805459861u, tz1 = tz0 + 805459861u;
            const uint32_t a0 = cx ^ ty0, a1 = cx ^ ty1;
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const uint32_t index = (((c & 1) ? a1 : a0) ^ ((c & 2) ? tz1 : tz0)) & g.mask;
                v[j][c] = E::load(gl + index);
            }
        } else if (g.kind & 2u) {    // dense coarse level: plain 3-D addressing
            const float bx = __fadd_rd(px, 8388608.0f), by = __fadd_rd(py, 8388608.0f), bz = __fadd_rd(pz, 8388608.0f);
            fx[j] = px - (bx - 8388608.0f); fy[j] = py - (by - 8388608.0f); fz[j] = pz - (bz - 8388608.0f);
            uint32_t i00 = (__float_as_uint(bx) - 0x4b000000u) + p + (__float_as_uint(by) - 0x4b000000u) * g.sy + (__float_as_uint(bz) - 0x4b000000u) * g.sz;
            uint32_t i01 = i00 + g.sy, i10 = i00 + g.sz, i11 = i01 + g.sz;
            // with align_corners a coordinate of exactly 1.0 makes the far corner index R: the reference then wraps modulo
            // the level size (gridencoder.cu:71).  i11 is the largest of the four, so one test covers them all.
            if (__builtin_expect(i11 >= g.hs, 0)) {
                i00 = i00 >= g.hs ? (g.mask ? (i00 & g.mask) : slow_umod(i00, g.hs)) : i00;
                i01 = i01 >= g.hs ? (g.mask ? (i01 & g.mask) : slow_umod(i01, g.hs)) : i01;
                i10 = i10 >= g.hs ? (g.mask ? (i10 & g.mask) : slow_umod(i10, g.hs)) : i10;
                i11 = g.mask ? (i11 & g.mask) : slow_umod(i11, g.hs);
            }
            v[j][0] = E::load(gl + i00);
            v[j][1] = E::load(gl + i01);
            v[j][2] = E::load(gl + i10);
            v[j][3] = E::load(gl + i11);
        } else {
            const float flx = floorf(px), fly = floorf(py), flz = floorf(pz);
            fx[j] = px - flx; fy[j] = py - fly; fz[j] = pz - flz;
            const uint32_t cx = (uint32_t)flx + p, iy = (uint32_t)fly, iz = (uint32_t)flz;
            uint32_t ty0, ty1, tz0, tz1;
            if (g.use_hash()) { ty0 = iy * 2654435761u; ty1 = ty0 + 2654435761u; tz0 = iz * 805459861u; tz1 = tz0 + 805459861u; }
            else { ty0 = iy * g.sy; ty1 = ty0 + g.sy; tz0 = iz * g.sz; tz1 = tz0 + g.sz; }
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const uint32_t ty = (c & 1) ? ty1 : ty0, tz = (c & 2) ? tz1 : tz0;
                uint32_t index = g.use_hash() ? (cx ^ ty ^ tz) : (cx + ty + tz);
                // dense levels only leave [0, hs) when a coordinate is exactly 1.0 (corner res) — rare, keep it a branch
                if (__builtin_expect(index >= g.hs, 0)) index = g.mask ? (index & g.mask) : slow_umod(index, g.hs);
                v[j][c] = E::load(gl + index);
            }
        }
    }
    // lane p accumulates levels 2p and 2p+1 of the batch; it needs the partner's corners of those levels
    raw o[2][4];
#pragma unroll
    for (int jj = 0; jj < 2; jj++)
#pragma unroll
        for (int c = 0; c < 4; c++) o[jj][c] = E::xchg(p ? v[jj][c] : v[2 + jj][c]);
#pragma unroll
    for (int jj = 0; jj < 2; jj++) {
        const float wfx = p ? fx[2 + jj] : fx[jj], wfy = p ? fy[2 + jj] : fy[jj], wfz = p ? fz[2 + jj] : fz[jj];
        const float wx0 = 1 - wfx, wy0 = 1 - wfy, wz0 = 1 - wfz;
        // reference order: idx = bx + 2*by + 4*bz, w = ((1*wx)*wy)*wz   (gridencoder.cu:146-167)
        const float w00 = wx0 * wy0, w10 = wfx * wy0, w01 = wx0 * wfy, w11 = wfx * wfy;
        typename E::accum r = E::zero();
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const float wz = (c & 2) ? wfz : wz0;
            const raw mine = p ? v[2 + jj][c] : v[jj][c];
            const raw x0v = p ? o[jj][c] : mine;   // corner with x bit 0
            const raw x1v = p ? mine : o[jj][c];   // corner with x bit 1
            E::add(r, ((c & 1) ? w01 : w00) * wz, x0v);
            E::add(r, ((c & 1) ? w11 : w10) * wz, x1v);
        }
        packed[jj] = live ? E::pack(r) : (raw)0;
    }
}

}  // namespace ntx
