// mlp_tile.cuh — building blocks of the tcgen05 fully-fused MLP, shared by mlp.cu (stand-alone FFMLP) and field.cu
// (hash-grid -> MLP -> SH -> MLP in one kernel).
//
// A CTA owns a 128-row batch tile = the M dimension of one UMMA (M=128, cta_group::1).  Activations [128 x K] and
// weights [N x K] (the reference's row-major [out,in] matrices, ffmlp.cu:632, are exactly "N x K, K-major") sit in
// shared memory in the no-swizzle core-matrix layout; accumulators [128 x N] fp32 live in TMEM; one thread issues
// the K/16 tcgen05.mma of a layer, commits to an mbarrier, and the epilogue warps pull the tile out of TMEM, apply the
// activation, round to fp16 (the reference keeps activations in fp16 between layers too) and write the next layer's
// A operand back to shared memory.  Nothing but the first input and the final 16-wide output touches global memory.
#pragma once

#include "common.cuh"
#include "tc05.cuh"

namespace ntx {

constexpr uint32_t kTileRows = 128;

// byte offset of fp16 element (r, k) in a [rows x Kdim] K-major no-swizzle tile (Kdim multiple of 8)
__device__ __forceinline__ uint32_t kmajor_off(uint32_t r, uint32_t k, uint32_t Kdim) {
    return (r >> 3) * (Kdim * 16u) + (k >> 3) * 128u + (r & 7u) * 16u + (k & 7u) * 2u;
}
// byte offset of the 16-byte chunk (r, kc) — kc indexes groups of 8 halfs
__device__ __forceinline__ uint32_t kmajor_chunk_off(uint32_t r, uint32_t kc, uint32_t Kdim) {
    return (r >> 3) * (Kdim * 16u) + kc * 128u + (r & 7u) * 16u;
}

// copy a row-major [rows x Kdim] fp16 matrix from global memory into the core-matrix layout (all threads of the CTA)
__device__ __forceinline__ void load_matrix_kmajor(uint8_t* smem_dst, const __half* __restrict__ src, uint32_t rows, uint32_t Kdim,
                                                   uint32_t tid, uint32_t nthreads) {
    const uint32_t kchunks = Kdim >> 3, total = rows * kchunks;
    for (uint32_t c = tid; c < total; c += nthreads) {
        const uint32_t r = c / kchunks, kc = c - r * kchunks;
        const uint4 v = *reinterpret_cast<const uint4*>(src + (size_t)r * Kdim + kc * 8);
        *reinterpret_cast<uint4*>(smem_dst + kmajor_chunk_off(r, kc, Kdim)) = v;
    }
}
// same, streaming source (batch rows are read exactly once)
__device__ __forceinline__ void load_rows_kmajor_stream(uint8_t* smem_dst, const __half* __restrict__ src, uint32_t rows, uint32_t rows_valid,
                                                        uint32_t Kdim, uint32_t tid, uint32_t nthreads) {
    const uint32_t kchunks = Kdim >> 3, total = rows * kchunks;
    for (uint32_t c = tid; c < total; c += nthreads) {
        const uint32_t r = c / kchunks, kc = c - r * kchunks;
        const uint4 v = (r < rows_valid) ? ld_stream_u4(src + (size_t)r * Kdim + kc * 8) : make_uint4(0u, 0u, 0u, 0u);  // ragged last tile
        *reinterpret_cast<uint4*>(smem_dst + kmajor_chunk_off(r, kc, Kdim)) = v;
    }
}

// D[128 x N] = A[128 x Kdim] . W[N x Kdim]^T   — issued by one thread
__device__ __forceinline__ void issue_layer(uint32_t a_smem, uint32_t w_smem, uint32_t Kdim, uint32_t N, uint32_t tmem_d) {
    const uint32_t idesc = tc::idesc_f16_f32(kTileRows, N);
    const uint32_t sbo = Kdim * 16u;
    for (uint32_t ks = 0; ks < (Kdim >> 4); ks++) {
        const uint64_t da = tc::smem_desc_kmajor_noswz(a_smem + ks * 256u, 128u, sbo);
        const uint64_t db = tc::smem_desc_kmajor_noswz(w_smem + ks * 256u, 128u, sbo);
        tc::mma_f16_ss(tmem_d, da, db, idesc, ks > 0 ? 1u : 0u);
    }
}

// Everything the issuing lane needs for the MMAs of one layer whose A operand is in tensor memory, precomputed once per CTA
// (field.cu, texture_field.cu): the layer is two LDS.128 + the UTCHMMAs instead of a descriptor build on the consumers' critical path.
struct StageMma {
    uint32_t b_lo[4];      // low words of the weight (B operand) descriptors of the K = 16 steps
    uint32_t b_hi;         // their common high word (SBO, descriptor version)
    uint32_t idesc;        // instruction descriptor (M = 128, N)
    uint32_t ksteps;       // 2 (a 32-wide input) or 4 (64-wide)
    uint32_t pad;
};
static_assert(sizeof(StageMma) == 32, "StageMma is two 16-byte loads");
// weights W [N x Kdim] K-major at shared address w, Kdim = 32 or 64
__device__ __forceinline__ StageMma stage_mma(uint32_t w, uint32_t Kdim, uint32_t N) {
    StageMma m;
    m.ksteps = Kdim >> 4;
    m.idesc = tc::idesc_f16_f32(kTileRows, N);
    m.b_hi = 0; m.pad = 0;
    for (uint32_t ks = 0; ks < 4; ks++) {
        const uint64_t d = tc::smem_desc_kmajor_noswz(w + (ks < m.ksteps ? ks : 0u) * 256u, 128u, Kdim * 16u);
        m.b_lo[ks] = (uint32_t)d;
        m.b_hi = (uint32_t)(d >> 32);
    }
    return m;
}
// issue layer st from its table entry: A = the operand columns in tensor memory (8 per K = 16 step)
__device__ __forceinline__ void issue_stage_ts(const StageMma* __restrict__ table, uint32_t st, uint32_t tmem_a, uint32_t tmem_acc) {
    const uint4 lo = *reinterpret_cast<const uint4*>(table[st].b_lo);
    const uint4 meta = *reinterpret_cast<const uint4*>(&table[st].b_hi);        // b_hi, idesc, ksteps, pad
    const uint64_t hi = (uint64_t)meta.x << 32;
    tc::mma_f16_ts(tmem_acc, tmem_a, hi | lo.x, meta.y, 0u);
    tc::mma_f16_ts(tmem_acc, tmem_a + 8u, hi | lo.y, meta.y, 1u);
    if (meta.z == 4u) {
        tc::mma_f16_ts(tmem_acc, tmem_a + 16u, hi | lo.z, meta.y, 1u);
        tc::mma_f16_ts(tmem_acc, tmem_a + 24u, hi | lo.w, meta.y, 1u);
    }
}

// activation ids of the reference (ffmlp.cu:22-33); applied to the fp16-rounded pre-activation like utils.h:425-470
__device__ __forceinline__ float mlp_activation(uint32_t act, float x) {
    constexpr float K_ACT = 10.0f;
    switch (act) {
        case 0: return x * (float)(x > 0.0f);                    // ReLU as x*(x>0): NaN-propagating like the reference
        case 1: return expf(x);
        case 2: return sinf(x);
        case 3: return 1.0f / (1.0f + expf(-x));
        case 4: { const float t = x * K_ACT; return 0.5f * (t + sqrtf(t * t + 4)) / K_ACT; }
        case 5: return logf(expf(x * K_ACT) + 1.0f) / K_ACT;
        default: return x;
    }
}
__device__ __forceinline__ uint32_t act_pack2(uint32_t act, uint32_t a_bits, uint32_t b_bits) {
    // accumulator (fp32) -> fp16 -> activation in fp32 -> fp16, two lanes at a time
    if (act == 0) {
        // the reference rounds to fp16 and then applies ReLU as x * (x > 0) (NaN-propagating; negative x gives -0).
        // cvt.rn.relu does clamp + round + pack in ONE instruction (F2FP.RELU); clamping before rounding gives the same
        // value, NaN still propagates, and only the sign of a zero differs, which nothing downstream can observe.
        uint32_t r;
        asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(b_bits)), "f"(__uint_as_float(a_bits)));
        return r;
    }
    const __half2 h = __floats2half2_rn(__uint_as_float(a_bits), __uint_as_float(b_bits));
    if (act >= 6) return *reinterpret_cast<const uint32_t*>(&h);
    const float2 f = __half22float2(h);
    return float2_to_half2_bits(mlp_activation(act, f.x), mlp_activation(act, f.y));
}

}  // namespace ntx
