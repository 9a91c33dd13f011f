// field.cu — the whole per-sample field of nerf/network_ff.py:85-101 in ONE kernel (fp16 inference):
//
//   xyz -> [0,1]^3 -> hash-grid gather (L levels x 2 features, fp16 table, lane-pair gather of grid_common.cuh)
//       -> sigma MLP  (2L -> 64 -> .. -> 16)  on tcgen05      -> sigma = exp(h[0]) * density_scale
//   dir -> SH degree 4 (16) ++ h[1..15] ++ 0  = 32
//       -> colour MLP (32 -> 64 -> .. -> 16)  on tcgen05      -> rgb = sigmoid(h[0..2])
//
// The reference runs this as 4 extension calls + ~10 torch glue kernels with every intermediate (features 64 B, padded
// copies, geo_feat, SH 64 B, concatenated colour input 64 B ...) making a round trip through HBM (SURVEY.md 3.2).
// Here a CTA owns 128-sample tiles and is warp-specialised:
//   * 12 producer warps gather features straight into the shared-memory A operand of the first UMMA.  A warp (16 lane
//     pairs) takes 16-row slices of the CTA's tile sequence round-robin, so the producers run up to kStages tiles ahead;
//     the feature tile is handed back as soon as the first MMA has read it;
//   * 4 consumer warps (one per TMEM lane quarter) run the two MLPs: one elected thread issues the tcgen05.mma of a layer; the
//     warps pull the fp32 accumulator out of tensor memory (tcgen05.ld), apply ReLU, round to fp16 and write the tile straight
//     back into tensor memory (tcgen05.st) as the A operand of the next layer's MMA (A-from-TMEM form).  Hidden activations,
//     geo_feat and the SH basis never exist in shared memory: no STS, no generic->async proxy fence in the layer chain, and the
//     16 KB activation buffer of round 1 is gone (the gather's throughput follows the L1 capacity the carve-out leaves);
//   * the MMA -> epilogue chain is 7 dependent stages per tile, one tile per CTA in flight (two resident CTAs per SM interleave
//     their chains); the consumer loop is written for kCtx tiles in flight, but ping-pong between two TMEM contexts measured
//     slower in both rounds (see kCtx);
//   * shared memory is kept small on purpose: weights 36 KB + the producer->consumer feature ring.
// Only xyz/dir (24 B) come in and sigma/rgb (16 B) go out per sample.
#include "grid_common.cuh"
#include "mlp_tile.cuh"
#include "sh_poly.cuh"

namespace ntx {

#ifndef NTX_FIELD_PRODUCERS       // development sweeps: NTX_NVCC_EXTRA="-DNTX_FIELD_PRODUCERS=8 -DNTX_FIELD_STAGES=2"
#define NTX_FIELD_PRODUCERS 12
#endif
#ifndef NTX_FIELD_STAGES
#define NTX_FIELD_STAGES 3
#endif
constexpr int kConsumerWarps = 4;   // one per TMEM lane quarter
constexpr int kProducerWarps = NTX_FIELD_PRODUCERS;
constexpr int kTaskRows = 16;                                            // rows one producer warp gathers at a time
constexpr int kTasksPerTile = 8;                                         // kTileRows / kTaskRows
constexpr int kFieldThreads = 32 * (kConsumerWarps + kProducerWarps);   // 512
constexpr int kFW = 64;          // hidden width of both MLPs
constexpr int kColorIn = 32;     // SH(16) + geo_feat(15) + zero pad (network_ff.py:42,95-97)
constexpr int kStages = NTX_FIELD_STAGES;       // feature tiles in the producer -> consumer ring
#ifndef NTX_FIELD_CTX
#define NTX_FIELD_CTX 1
#endif
// Tiles a CTA's consumers keep in flight (TMEM contexts they alternate between).  2 measured SLOWER again in round 2, although with
// the activations in tensor memory a second context no longer costs shared memory: frame 6.48 -> 8.05 ms, cfg2 coherent 201 -> 252 us,
// MLP chain alone 124 -> 147 us (profiles/r02_summary.md) — the chain's time is the TMEM -> register read of the accumulators
// (32 KB per hidden layer at ~64 B/clk per SM), which a second context shares instead of hiding.  The loop below stays generic.
constexpr int kCtx = NTX_FIELD_CTX;
constexpr uint32_t kOpndCol = 64;      // fp16 A operand [128 x 64] of the next layer: 32 columns behind the fp32 accumulator [128 x 64]
constexpr uint32_t kCtxCols = 96;      // accumulator + operand columns of one context
constexpr uint32_t kFieldTmemCols = kCtx == 1 ? 128 : 256;   // kCtx * kCtxCols rounded up to a power of two

struct FieldPlan {
    uint32_t k0;                 // sigma-net input width = 2L
    uint32_t ws_bytes, wc_bytes; // weight bytes of the two nets
    uint32_t ws_off, wc_off, a0_off, lv_off, misc_off, total;
    uint32_t a0_stage;
};
__host__ __device__ inline FieldPlan field_plan(uint32_t L, uint32_t ns, uint32_t nc) {
    FieldPlan p;
    p.k0 = 2 * L;
    p.ws_bytes = 2u * (kFW * p.k0 + (ns - 1) * kFW * kFW + 16u * kFW);
    p.wc_bytes = 2u * (kFW * kColorIn + (nc - 1) * kFW * kFW + 16u * kFW);
    p.ws_off = 0;
    p.wc_off = p.ws_off + p.ws_bytes;
    p.a0_stage = kTileRows * p.k0 * 2u;
    p.a0_off = (p.wc_off + p.wc_bytes + 127u) & ~127u;
    p.lv_off = p.a0_off + kStages * p.a0_stage;
    p.misc_off = p.lv_off + (uint32_t)sizeof(PairLevel) * kFieldMaxLevels;
    p.total = p.misc_off + 512u;      // barriers + TMEM slot (128 B) | per-stage MMA parameter table (384 B)
    return p;
}

// development probes (-DNTX_DEV_PROBES, tools/field_probe.py): cycle accounting of one producer and one consumer warp per CTA
#ifdef NTX_DEV_PROBES
__device__ unsigned long long g_probe[8];   // consumer: wait_full, wait_mma, epilogue | - | producer: wait_empty, gather, loads | CTAs
#define PROBE_DECL unsigned long long pr_t = clock64(), pr_acc[3] = {0, 0, 0};
#define PROBE_MARK(i) { const unsigned long long n_ = clock64(); pr_acc[i] += n_ - pr_t; pr_t = n_; }
#define PROBE_FLUSH(base) { for (int i_ = 0; i_ < 3; i_++) atomicAdd(&g_probe[(base) + i_], pr_acc[i_]); }
#else
#define PROBE_DECL
#define PROBE_MARK(i) {}
#define PROBE_FLUSH(base) {}
#endif

__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(32 * kConsumerWarps) : "memory"); }

// hidden-layer epilogue: warp q owns TMEM lanes 32q.. (= tile rows): accumulator columns -> ReLU -> fp16 -> operand columns,
// 32 accumulator columns per pass (the kernel lives in 64 registers per thread)
__device__ __forceinline__ void field_hidden_epilogue(uint32_t acc, uint32_t opnd) {
#pragma unroll
    for (int h = 0; h < kFW; h += 32) {
        uint32_t v[32], o[16];
        tc::tmem_ld_x32(acc + h, v);
        tc::tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; j++) o[j] = act_pack2(0, v[2 * j], v[2 * j + 1]);
        tc::tmem_st_x16(opnd + (h >> 1), o);
    }
}

// consumer stage st (0 .. ns+nc+1) = "MMA st has completed -> epilogue".  Layer table (weights in the order the nets store them):
//   st = 0          a0 [128 x 2L] . Ws0^T -> 64      hidden epilogue          (issued when the feature tile arrives)
//   st = 1..ns-1    h . Ws(st)^T          -> 64      hidden epilogue
//   st = ns         h . Ws_out^T          -> 16      sigma + colour-net input
//   st = ns+1       h [128 x 32] . Wc0^T  -> 64      hidden epilogue
//   st = ns+2..ns+nc                      -> 64      hidden epilogue
//   st = ns+nc+1    h . Wc_out^T          -> 16      rgb
// The MMAs of stage st come from a StageMma table (mlp_tile.cuh) precomputed once per CTA: between the consumers' barrier and the
// first UTCHMMA of a stage the round-2 build spent ~50 uniform-datapath instructions assembling descriptors (SASS) — on the critical
// path of every stage, issued by one warp while the other three wait, next to twelve gathering warps.
__device__ __forceinline__ StageMma make_stage_mma(uint32_t st, uint32_t ns, uint32_t nc, uint32_t K0, uint32_t ws_addr, uint32_t wc_addr) {
    uint32_t w, Kdim, N;
    if (st <= ns) { w = ws_addr + kFW * K0 * 2u + (st - 1) * (kFW * kFW * 2u); Kdim = kFW; N = st == ns ? 16u : (uint32_t)kFW; }
    else if (st == ns + 1) { w = wc_addr; Kdim = kColorIn; N = kFW; }
    else { w = wc_addr + kFW * kColorIn * 2u + (st - ns - 2) * (kFW * kFW * 2u); Kdim = kFW; N = st == ns + nc + 1 ? 16u : (uint32_t)kFW; }
    return stage_mma(w, Kdim, N);
}

// What a row is: MODE_ROWS  = a row of xyz/dirs (the ntx_ngp_field_forward contract, optionally through a row list);
//                 MODE_DENSITY = a cell of the occupancy grid (density-grid maintenance, see DensityArgs);
//                 MODE_RAYS  = an entry (sample row, ray) of the device-driven frame's live list: the marcher stores only the
//                              sample's ray parameter t and the field kernel rebuilds xyz = clamp(o + t d) with the marcher's own
//                              expression (raymarching.cu:362-364) and takes the view direction from the ray — 12 instead of 32
//                              bytes per sample leave the marcher, and xyz/dirs never exist in HBM.
constexpr int MODE_ROWS = 0, MODE_DENSITY = 1, MODE_RAYS = 2;
struct RayArgs {
    const int2* live;       // [n_live] (sample row, ray index)
    const float* ts;        // [rows] ray parameter of the sample at that row
    const float* rays_o;    // [N,3]
    const float* rays_d;    // [N,3]
};

// Density-grid maintenance mode (NeRFRenderer.update_extra_state, renderer.py:567-635): the samples are the cells of one cascade of
// the occupancy grid — positions are generated in the kernel from the cell's Morton index exactly as the reference's torch code
// computes them — only the sigma net runs, and sigma * density_scale lands in tmp_grid[cell].
struct DensityArgs {
    const int* cells;     // nullable: Morton index of slot i (partial update, renderer.py:603-625); null: slot i is cell i (full update)
    const float* noise;   // nullable: uniform [0,1) jitter, [.,3]; row = slot (cells given) or x-major meshgrid index of the cell (full update)
    uint32_t H;           // grid size
    float inv_hm1;        // fp32 1 / (H - 1)
    float scale;          // fp32 (bound_c - half_grid_size)
    float hgs;            // fp32 half_grid_size = bound_c / H
    float* tmp;           // tmp_grid of this cascade [H^3]
};
__device__ __forceinline__ uint32_t compact_bits3(uint32_t x) {      // raymarching.cu:75-83
    x = x & 0x49249249u;
    x = (x | (x >> 2)) & 0xc30c30c3u;
    x = (x | (x >> 4)) & 0x0f00f00fu;
    x = (x | (x >> 8)) & 0xff0000ffu;
    x = (x | (x >> 16)) & 0x0000ffffu;
    return x;
}

template <int MODE>
__global__ void __launch_bounds__(kFieldThreads, 2) ngp_field_kernel(
    const float* __restrict__ xyz, const float* __restrict__ dirs, const float* __restrict__ deltas, const uint32_t M_arg, const int* __restrict__ M_dev,
    const int* __restrict__ rows, const float bound, const __half* __restrict__ table, const int* __restrict__ offsets, const uint32_t L, const float S, const uint32_t H, const bool align,
    const __half* __restrict__ w_sigma, const __half* __restrict__ w_color, const uint32_t ns, const uint32_t nc, const float density_scale,
    float* __restrict__ sigmas, float* __restrict__ rgbs, const uint32_t dbg, const DensityArgs dens, const RayArgs rays) {
    constexpr bool DENSITY = MODE == MODE_DENSITY, RAYS = MODE == MODE_RAYS;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t M = M_dev ? (uint32_t)*M_dev : M_arg;     // device-driven frames: the sample count of this launch lives on the device
    const FieldPlan plan = field_plan(L, ns, nc);
    uint8_t* ws_smem = smem + plan.ws_off;
    uint8_t* wc_smem = smem + plan.wc_off;
    uint8_t* a0_smem = smem + plan.a0_off;   // kStages tiles
    PairLevel* lv = reinterpret_cast<PairLevel*>(smem + plan.lv_off);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + plan.misc_off);        // [kStages] producers -> consumer
    uint64_t* empty_bar = full_bar + kStages;                                      // [kStages] consumer (MMA completion) -> producers
    uint64_t* mma_bar = empty_bar + kStages;                                       // [kCtx] layer done -> consumer warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_bar + kCtx);
    StageMma* stage_table = reinterpret_cast<StageMma*>(smem + plan.misc_off + 128u);   // [ns + nc + 2] (entry 0 unused)

    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t K0 = plan.k0;

    // ---- one-time setup (all 16 warps) ---------------------------------------------------------------------------
    if (tid == 0) {
        for (int s = 0; s < kStages; s++) { tc::mbar_init(&full_bar[s], kTasksPerTile); tc::mbar_init(&empty_bar[s], 1); }
        for (int c = 0; c < kCtx; c++) tc::mbar_init(&mma_bar[c], 1);
        tc::fence_mbar_init();
    }
    if (warp == 0) tc::tmem_alloc<kFieldTmemCols>(tmem_slot);
    if (tid >= 32 && tid < 32 + ns + nc + 2 && tid > 32) stage_table[tid - 32] = make_stage_mma(tid - 32, ns, nc, plan.k0, tc::smem_u32(ws_smem), tc::smem_u32(wc_smem));
    if (tid < L) lv[tid] = make_pair_level(make_level<3>(offsets, tid, S, H, /*gridtype=*/0, align), table);
    {
        const __half* w = w_sigma; uint8_t* dst = ws_smem;
        load_matrix_kmajor(dst, w, kFW, K0, tid, kFieldThreads); w += (size_t)kFW * K0; dst += (size_t)kFW * K0 * 2;
        for (uint32_t k = 0; k + 1 < ns; k++) { load_matrix_kmajor(dst, w, kFW, kFW, tid, kFieldThreads); w += kFW * kFW; dst += kFW * kFW * 2; }
        load_matrix_kmajor(dst, w, 16, kFW, tid, kFieldThreads);
        w = w_color; dst = wc_smem;
        load_matrix_kmajor(dst, w, kFW, kColorIn, tid, kFieldThreads); w += kFW * kColorIn; dst += kFW * kColorIn * 2;
        for (uint32_t k = 0; k + 1 < nc; k++) { load_matrix_kmajor(dst, w, kFW, kFW, tid, kFieldThreads); w += kFW * kFW; dst += kFW * kFW * 2; }
        load_matrix_kmajor(dst, w, 16, kFW, tid, kFieldThreads);
    }
    tc::fence_proxy_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t ntiles = ceil_div<uint32_t>(M, kTileRows);

    if (warp >= kConsumerWarps) {
        // =============================== PRODUCERS: gather ===========================================================
        const uint32_t pw = warp - kConsumerWarps;             // 0..11
        const uint32_t p = lane & 1u;                          // which x corner this lane gathers
        const float half_off = align ? 0.0f : 0.5f;
        // GridEncoder.forward: inputs = (inputs + bound) / (2 * bound) (grid.py:143).  torch's CUDA true-division by a Python
        // scalar multiplies by the fp32 reciprocal (BinaryDivTrueKernel.cu), so do exactly that.
        const float inv2b = 1.0f / (2.0f * bound);
        PROBE_DECL
        for (uint32_t task = pw;; task += kProducerWarps) {
            const uint32_t k = task / kTasksPerTile;            // k-th tile of this CTA
            const uint32_t tile = blockIdx.x + k * gridDim.x;
            if (tile >= ntiles) break;
            const uint32_t s = k % kStages, use = k / kStages;
            const uint32_t srow = (task % kTasksPerTile) * kTaskRows + (lane >> 1);   // row of this lane pair inside the tile
            const uint32_t bi = tile * kTileRows + srow;
            const bool valid = bi < M;
            const uint32_t b = (MODE == MODE_ROWS && valid && rows) ? (uint32_t)rows[bi] : bi;     // optional row list
            float x = 0.f, y = 0.f, z = 0.f;
            bool skip = !valid;
            if (DENSITY) {
                if (valid) {
                    // xyzs = 2 * coords.float() / (H - 1) - 1; cas_xyzs = xyzs * (bound_c - hgs) [+ (rand * 2 - 1) * hgs]   (renderer.py:590-598)
                    // — one rounding per torch op (a division by a Python scalar is a multiplication by its fp32 reciprocal)
                    const uint32_t cell = dens.cells ? (uint32_t)dens.cells[bi] : bi;
                    const uint32_t c3[3] = {compact_bits3(cell), compact_bits3(cell >> 1), compact_bits3(cell >> 2)};
                    const size_t nrow = dens.cells ? (size_t)bi : ((size_t)c3[0] * dens.H + c3[1]) * dens.H + c3[2];
                    float v[3];
#pragma unroll
                    for (int d = 0; d < 3; d++) {
                        v[d] = __fmul_rn(__fsub_rn(__fmul_rn(__fmul_rn(2.0f, (float)c3[d]), dens.inv_hm1), 1.0f), dens.scale);
                        if (dens.noise) v[d] = __fadd_rn(v[d], __fmul_rn(__fsub_rn(__fmul_rn(dens.noise[nrow * 3 + d], 2.0f), 1.0f), dens.hgs));
                    }
                    x = __fmul_rn(__fadd_rn(v[0], bound), inv2b);
                    y = __fmul_rn(__fadd_rn(v[1], bound), inv2b);
                    z = __fmul_rn(__fadd_rn(v[2], bound), inv2b);
                }
            } else if (RAYS) {
                if (valid) {
                    const int2 e = rays.live[bi];
                    const float t = rays.ts[e.x];
                    const float* o = rays.rays_o + (size_t)e.y * 3;
                    const float* d = rays.rays_d + (size_t)e.y * 3;
                    // the marcher's sample position, written exactly like probe()/locate() in raymarch.cu (and raymarching.cu:362-364)
                    // so that the compiler contracts it the same way: clamp(o + t * d, -bound, bound)
                    const float sx = fminf(bound, fmaxf(-bound, o[0] + t * d[0]));
                    const float sy = fminf(bound, fmaxf(-bound, o[1] + t * d[1]));
                    const float sz = fminf(bound, fmaxf(-bound, o[2] + t * d[2]));
                    x = __fmul_rn(__fadd_rn(sx, bound), inv2b);
                    y = __fmul_rn(__fadd_rn(sy, bound), inv2b);
                    z = __fmul_rn(__fadd_rn(sz, bound), inv2b);
                }
            } else if (valid) {
                x = __fmul_rn(__fadd_rn(xyz[(size_t)b * 3], bound), inv2b);
                y = __fmul_rn(__fadd_rn(xyz[(size_t)b * 3 + 1], bound), inv2b);
                z = __fmul_rn(__fadd_rn(xyz[(size_t)b * 3 + 2], bound), inv2b);
                if (deltas && deltas[(size_t)b * 2] == 0.0f) skip = true;  // sentinel slot of march_rays
            }
            const uint32_t cls = skip ? 0u : sample_class(x, y, z);
            const bool live = cls == 1u;
            if (!live) { x = 0.f; y = 0.f; z = 0.f; }  // keeps the (discarded) loads of dead lanes in bounds
            PROBE_MARK(2)
            tc::mbar_wait_relaxed(&empty_bar[s], (use & 1u) ^ 1u, 256u);   // slot free? (first use of a slot passes immediately)
            PROBE_MARK(0)
            uint8_t* a0 = a0_smem + s * plan.a0_stage;
            for (uint32_t l0 = 0; l0 < L; l0 += 4) {
                uint32_t packed[2];
#ifdef NTX_DEV_PROBES
                if (dbg & 1u) { packed[0] = packed[1] = 0; } else
#endif
                pair_gather4<__half>(x, y, z, live, p, lv + l0, half_off, packed);
                if (cls == 2u) { packed[0] = packed[1] = nan_features<uint32_t>(); }   // NaN coordinate: NaN features like the reference
                // lane p owns levels l0+2p, l0+2p+1 -> 4 consecutive halfs (8 bytes) of the row
                const uint32_t kcol = 2 * (l0 + 2 * p);
                *reinterpret_cast<uint2*>(a0 + kmajor_off(srow, kcol, K0)) = make_uint2(packed[0], packed[1]);
            }
            tc::fence_proxy_async_smem();          // my generic-proxy writes -> visible to the tensor core's async proxy
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&full_bar[s]);
            PROBE_MARK(1)
        }
        if (pw == 0 && lane == 0) PROBE_FLUSH(4)
    } else {
        // =============================== CONSUMERS: the two MLPs, activations resident in tensor memory =============
        // kCtx tiles (contexts) in flight: each has its own accumulator + operand columns and its own MMA barrier; with kCtx = 2 the
        // four warps alternate between them stage by stage (one tile's MMA under the other tile's epilogue).
        const uint32_t ws_addr = tc::smem_u32(ws_smem), wc_addr = tc::smem_u32(wc_smem);
        const uint32_t quarter = warp, row = quarter * 32 + lane;
        const uint32_t nst = DENSITY ? ns + 1 : ns + nc + 2;      // density mode: the sigma net only
        uint32_t ph[kCtx] = {};
        PROBE_DECL
        for (uint32_t k0 = 0;; k0 += kCtx) {
            if (blockIdx.x + k0 * gridDim.x >= ntiles) break;
            uint32_t b[kCtx], aux[kCtx];                  // output row | ray index (MODE_RAYS)
            bool has[kCtx], ok[kCtx], dead[kCtx];
            float dxs[kCtx], dys[kCtx], dzs[kCtx];        // view direction of the row (its SH basis is evaluated between the two nets): loaded
                                                          // when the tile starts — a load issued at the stage that needs it sits on the chain's
                                                          // critical path (measured: frame 6.48 -> 7.36 ms)
#pragma unroll
            for (int c = 0; c < kCtx; c++) {
                const uint32_t k = k0 + c, tile = blockIdx.x + k * gridDim.x;
                has[c] = tile < ntiles;
                b[c] = tile * kTileRows + row; aux[c] = 0; ok[c] = false; dead[c] = false;
                if (!has[c]) continue;
                const uint32_t s = k % kStages, use = k / kStages;
                ok[c] = b[c] < M;                         // this thread's row exists (ragged last tile)
                if (DENSITY) { if (ok[c] && dens.cells) b[c] = (uint32_t)dens.cells[b[c]]; }
                else if (RAYS) {
                    if (ok[c]) { const int2 e = rays.live[b[c]]; b[c] = (uint32_t)e.x; aux[c] = (uint32_t)e.y; }   // sigma / rgb go to the sample's slot row
                } else if (ok[c] && rows) b[c] = (uint32_t)rows[b[c]];
                dead[c] = MODE == MODE_ROWS && (!ok[c] || (deltas && deltas[(size_t)b[c] * 2] == 0.0f));
                dxs[c] = dys[c] = dzs[c] = 0.f;
                if (!DENSITY && ok[c]) {
                    const float* d = RAYS ? rays.rays_d + (size_t)aux[c] * 3 : dirs + (size_t)b[c] * 3;
                    dxs[c] = d[0]; dys[c] = d[1]; dzs[c] = d[2];
                }
                PROBE_MARK(2)
                // Only the issuing warp waits for the feature tile: nobody else reads it, and a consumer warp still polling
                // full_bar[s] after the slot has been released below could see the producers complete the NEXT phase of that
                // barrier and wait forever on a parity that has come round again.
                if (warp == 0) { tc::mbar_wait(&full_bar[s], use & 1u); tc::tc_fence_after_sync(); }
                PROBE_MARK(0)
#ifdef NTX_DEV_PROBES
                if (dbg & 2u) {   // producer-only timing: release the slot at once, skip both MLPs
                    if (tid == 0) tc::mbar_arrive(&empty_bar[s]);
                    if (ok[c] && sigmas) { st_stream_f32(sigmas + b[c], 0.f); for (int q = 0; q < 3; q++) st_stream_f32(rgbs + (size_t)b[c] * 3 + q, 0.f); }
                    has[c] = false;
                    continue;
                }
#endif
                if (warp == 0 && tc::elect_one()) {
                    issue_layer(tc::smem_u32(a0_smem + s * plan.a0_stage), ws_addr, K0, kFW, tmem_base + c * kCtxCols);
                    tc::mma_commit(&mma_bar[c]);
                    tc::mma_commit(&empty_bar[s]);   // the feature tile is free again as soon as this MMA has read it
                }
            }
            for (uint32_t st = 0; st < nst; st++) {
#pragma unroll
                for (int c = 0; c < kCtx; c++) {
                    if (!has[c]) continue;
                    const uint32_t acc_all = tmem_base + c * kCtxCols, opnd_all = acc_all + kOpndCol;        // MMA addresses (all 128 lanes)
                    const uint32_t acc = acc_all + ((quarter * 32u) << 16), opnd = opnd_all + ((quarter * 32u) << 16);   // this warp's lanes
                    const float dx = dxs[c], dy = dys[c], dz = dzs[c];
                    tc::mbar_wait(&mma_bar[c], ph[c]); ph[c] ^= 1;
                    PROBE_MARK(1)
                    tc::tc_fence_after_sync();
                    if (st == ns) {
                        uint32_t v[16];
                        tc::tmem_ld_x16(acc, v);
                        tc::tmem_wait_ld();
                        // h = fp16(W2 . a)   (FFMLP output is fp16); sigma = trunc_exp(h[0]) = exp(float(h[0]))   (network_ff.py:88)
                        uint32_t hb[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) hb[j] = float2_to_half2_bits(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
                        const float h0 = __low2float(*reinterpret_cast<const __half2*>(&hb[0]));
                        if (DENSITY) {
                            // sigmas = trunc_exp(h[..., 0]); sigmas *= density_scale; tmp_grid[cas, indices] = sigmas   (network_ff.py:113, renderer.py:600-602)
                            if (ok[c]) dens.tmp[b[c]] = __fmul_rn(expf(h0), density_scale);
                        } else {
                            if (ok[c]) st_stream_f32(sigmas + b[c], dead[c] ? 0.0f : density_scale * expf(h0));
                            // colour-net input [128 x 32] = SH(dir) ++ h[1..15] ++ 0   (network_ff.py:93-97) -> 16 operand columns.
                            // SH in fp32, rounded to fp16 when it enters the fp16 MLP.
                            uint32_t o[16];
                            {
                                float sh[16];
                                sh_basis<4, false>(dx, dy, dz, sh, nullptr, nullptr, nullptr);
#pragma unroll
                                for (int j = 0; j < 8; j++) o[j] = float2_to_half2_bits(sh[2 * j], sh[2 * j + 1]);
                            }
#pragma unroll
                            for (int j = 0; j < 7; j++) o[8 + j] = __byte_perm(hb[j], hb[j + 1], 0x5432);
                            o[15] = __byte_perm(hb[7], 0u, 0x5432);
                            tc::tmem_st_x16(opnd, o);
                        }
                    } else if (st + 1 == nst) {
                        uint32_t v[8];
                        tc::tmem_ld_x8(acc, v);
                        tc::tmem_wait_ld();
                        if (ok[c]) {
#pragma unroll
                            for (int q = 0; q < 3; q++) {
                                // rgb = sigmoid(h) evaluated on the fp16 output in fp32 and rounded back to fp16 (torch.sigmoid on a half tensor)
                                const float hc = __half2float(__float2half_rn(__uint_as_float(v[q])));
                                const float sg = 1.0f / (1.0f + expf(-hc));
                                st_stream_f32(rgbs + (size_t)b[c] * 3 + q, dead[c] ? 0.0f : __half2float(__float2half_rn(sg)));
                            }
                        }
                    } else {
                        field_hidden_epilogue(acc, opnd);
                    }
                    // epilogue done by all four warps: this tile's next layer may read the operand columns and overwrite the
                    // accumulator (after the last stage: the next tile of this context may)
                    tc::tmem_wait_st(); tc::tc_fence_before_sync(); consumer_sync();
                    if (st + 1 < nst && warp == 0 && tc::elect_one()) {
                        tc::tc_fence_after_sync();
                        issue_stage_ts(stage_table, st + 1, opnd_all, acc_all);
                        tc::mma_commit(&mma_bar[c]);
                    }
                    PROBE_MARK(2)
                }
            }
        }
        if (tid == 0) PROBE_FLUSH(0)
    }

    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<kFieldTmemCols>(tmem_base);
#ifdef NTX_DEV_PROBES
    if (tid == 0) atomicAdd(&g_probe[7], 1ull);
#endif
}

}  // namespace ntx

using namespace ntx;

// development probes (only in builds with -DNTX_DEV_PROBES; tools/field_probe.py): NTX_FIELD_DEBUG bit 0 = producers skip the
// gather, bit 1 = consumers skip the MLPs; ntx_dev_probe_read returns the cycle accounting.  Product builds always pass 0
// and the branches do not exist.
#ifdef NTX_DEV_PROBES
extern "C" int ntx_dev_probe_read(unsigned long long* out8, int reset) {
    if (cudaMemcpyFromSymbol(out8, g_probe, sizeof(unsigned long long) * 8) != cudaSuccess) return NTX_ERR_CUDA;
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_probe, z, sizeof(z)); }
    return NTX_OK;
}
#endif
static uint32_t dev_probe_flags() {
#ifdef NTX_DEV_PROBES
    const char* e = getenv("NTX_FIELD_DEBUG");
    return e ? (uint32_t)atoi(e) : 0u;
#else
    return 0u;
#endif
}

extern "C" int ntx_ngp_field_forward(const float* xyz, const float* dirs, const float* deltas, uint32_t M, float bound, const void* embeddings_f16,
                                     const int* offsets, uint32_t L, float S, uint32_t H, int align_corners, const void* w_sigma_f16,
                                     const void* w_color_f16, float density_scale, float* sigmas, float* rgbs, ntx_stream_t stream) {
    return launch_ngp_field(xyz, dirs, deltas, M, nullptr, nullptr, bound, embeddings_f16, offsets, L, S, H, align_corners, w_sigma_f16, w_color_f16, density_scale, sigmas,
                            rgbs, reinterpret_cast<cudaStream_t>(stream));
}

// M = upper bound of the sample count (sizes the grid); M_dev (nullable, device) = the actual count, read by the kernel;
// rows (nullable, device) = indices of the rows to evaluate (then M counts list entries)
template <int MODE>
static int launch_field_kernel(const float* xyz, const float* dirs, const float* deltas, uint32_t M, const int* M_dev, const int* rows, float bound,
                               const void* embeddings_f16, const int* offsets, uint32_t L, float S, uint32_t H, int align_corners, const void* w_sigma_f16,
                               const void* w_color_f16, float density_scale, float* sigmas, float* rgbs, const DensityArgs& dens, const RayArgs& rays, cudaStream_t stream) {
    const uint32_t ns = 2, nc = 3;  // FFMLP(num_layers=2) and FFMLP(num_layers=3): nerf/network_ff.py:31-49
    const FieldPlan plan = field_plan(L, ns, nc);
    static int occ_dev[kMaxDevices] = {};
    static uint32_t configured_dev[kMaxDevices] = {};
    int& occ = occ_dev[current_device()];
    uint32_t& configured = configured_dev[current_device()];
    if (plan.total > configured) {
        if (cudaFuncSetAttribute(ngp_field_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.total) != cudaSuccess) {
            cudaGetLastError();
            set_error("ngp_field_forward: cannot reserve %u bytes of shared memory", plan.total);
            return NTX_ERR_CUDA;
        }
        configured = plan.total;
        occ = 0;
    }
    if (!occ) {
        occ = resident_ctas_per_sm((const void*)ngp_field_kernel<MODE>, kFieldThreads, plan.total, kFieldTmemCols);
        if (tunables().field_ctas > 0) occ = std::min(occ, tunables().field_ctas);
    }
    const int sms = device_sm_count();
    const uint32_t ntiles = ceil_div<uint32_t>(M, kTileRows);
    const uint32_t grid = std::min<uint32_t>(ntiles, (uint32_t)(occ * sms));
    ngp_field_kernel<MODE><<<grid, kFieldThreads, plan.total, stream>>>(
        xyz, dirs, deltas, M, M_dev, rows, bound, static_cast<const __half*>(embeddings_f16), offsets, L, S, H, align_corners != 0,
        static_cast<const __half*>(w_sigma_f16), static_cast<const __half*>(w_color_f16), ns, nc, density_scale, sigmas, rgbs, dev_probe_flags(), dens, rays);
    return check_launch(MODE == MODE_DENSITY ? "density_grid_query" : "ngp_field_forward");
}

int ntx::launch_ngp_field(const float* xyz, const float* dirs, const float* deltas, uint32_t M, const int* M_dev, const int* rows, float bound,
                          const void* embeddings_f16,
                          const int* offsets, uint32_t L, float S, uint32_t H, int align_corners, const void* w_sigma_f16, const void* w_color_f16,
                          float density_scale, float* sigmas, float* rgbs, cudaStream_t stream) {
    NTX_REQUIRE(xyz && dirs && embeddings_f16 && offsets && w_sigma_f16 && w_color_f16 && sigmas && rgbs, NTX_ERR_INVALID_ARGUMENT, "ngp_field_forward: null pointer");
    NTX_REQUIRE(L >= 8 && L <= kFieldMaxLevels && L % 8 == 0, NTX_ERR_UNSUPPORTED, "ngp_field_forward: num_levels must be 8, 16, 24 or 32 (got %u)", L);
    NTX_REQUIRE(((uintptr_t)w_sigma_f16 & 15) == 0 && ((uintptr_t)w_color_f16 & 15) == 0, NTX_ERR_INVALID_ARGUMENT, "ngp_field_forward: weights must be 16-byte aligned");
    NTX_REQUIRE(bound > 0, NTX_ERR_INVALID_ARGUMENT, "ngp_field_forward: bound must be positive");
    if (M == 0) return NTX_OK;
    return launch_field_kernel<MODE_ROWS>(xyz, dirs, deltas, M, M_dev, rows, bound, embeddings_f16, offsets, L, S, H, align_corners, w_sigma_f16, w_color_f16,
                                          density_scale, sigmas, rgbs, DensityArgs{}, RayArgs{}, stream);
}

// sigma * density_scale of `n_cells` occupancy-grid cells of ONE cascade -> tmp_grid_cascade[cell]  (see DensityArgs)
int ntx::launch_density_query(uint32_t n_cells, const int* cells, const float* noise, uint32_t grid_size, float cascade_bound, float bound, const void* embeddings_f16,
                              const int* offsets, uint32_t L, float S, uint32_t H, int align_corners, const void* w_sigma_f16, float density_scale,
                              float* tmp_grid_cascade, cudaStream_t stream) {
    NTX_REQUIRE(embeddings_f16 && offsets && w_sigma_f16 && tmp_grid_cascade, NTX_ERR_INVALID_ARGUMENT, "update_density_grid: null pointer");
    NTX_REQUIRE(L >= 8 && L <= kFieldMaxLevels && L % 8 == 0, NTX_ERR_UNSUPPORTED, "update_density_grid: num_levels must be 8, 16, 24 or 32 (got %u)", L);
    NTX_REQUIRE(((uintptr_t)w_sigma_f16 & 15) == 0, NTX_ERR_INVALID_ARGUMENT, "update_density_grid: weights must be 16-byte aligned");
    NTX_REQUIRE(bound > 0 && cascade_bound > 0 && grid_size >= 2 && grid_size <= 1024, NTX_ERR_INVALID_ARGUMENT, "update_density_grid: bad bound / grid size");
    if (n_cells == 0) return NTX_OK;
    DensityArgs d;
    d.cells = cells; d.noise = noise; d.H = grid_size;
    d.inv_hm1 = 1.0f / (float)(grid_size - 1);
    const double hgs = (double)cascade_bound / (double)grid_size;       // Python floats (renderer.py:592-594), rounded to fp32 when they meet the tensor
    d.scale = (float)((double)cascade_bound - hgs);
    d.hgs = (float)hgs;
    d.tmp = tmp_grid_cascade;
    // the colour net is not evaluated in this mode; its shared-memory slot is filled from the sigma weights (any valid pointer)
    return launch_field_kernel<MODE_DENSITY>(nullptr, nullptr, nullptr, n_cells, nullptr, nullptr, bound, embeddings_f16, offsets, L, S, H, align_corners, w_sigma_f16,
                                             w_sigma_f16, density_scale, nullptr, nullptr, d, RayArgs{}, stream);
}

// the device-driven frame: rows = the marcher's live list (sample row, ray); M_dev = its length on the device
int ntx::launch_ngp_field_rays(const int2* live, const int* n_live_dev, uint32_t M_bound, const float* ts, const float* rays_o, const float* rays_d, float bound,
                               const void* embeddings_f16, const int* offsets, uint32_t L, float S, uint32_t H, int align_corners, const void* w_sigma_f16,
                               const void* w_color_f16, float density_scale, float* sigmas, float* rgbs, cudaStream_t stream) {
    NTX_REQUIRE(live && n_live_dev && ts && rays_o && rays_d && embeddings_f16 && offsets && w_sigma_f16 && w_color_f16 && sigmas && rgbs, NTX_ERR_INVALID_ARGUMENT,
                "render_rays(field): null pointer");
    NTX_REQUIRE(L >= 8 && L <= kFieldMaxLevels && L % 8 == 0, NTX_ERR_UNSUPPORTED, "ngp_field_forward: num_levels must be 8, 16, 24 or 32 (got %u)", L);
    NTX_REQUIRE(((uintptr_t)w_sigma_f16 & 15) == 0 && ((uintptr_t)w_color_f16 & 15) == 0, NTX_ERR_INVALID_ARGUMENT, "ngp_field_forward: weights must be 16-byte aligned");
    NTX_REQUIRE(bound > 0, NTX_ERR_INVALID_ARGUMENT, "ngp_field_forward: bound must be positive");
    if (M_bound == 0) return NTX_OK;
    RayArgs r;
    r.live = live; r.ts = ts; r.rays_o = rays_o; r.rays_d = rays_d;
    return launch_field_kernel<MODE_RAYS>(nullptr, nullptr, nullptr, M_bound, n_live_dev, nullptr, bound, embeddings_f16, offsets, L, S, H, align_corners, w_sigma_f16,
                                          w_color_f16, density_scale, sigmas, rgbs, DensityArgs{}, r, stream);
}
