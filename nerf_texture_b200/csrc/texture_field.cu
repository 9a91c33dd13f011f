// texture_field.cu — NeRFNetwork.density(x) of the product's model (nerf/network_curvedfield.py:412-433) in ONE kernel (fp16 inference):
//
//   xyz -> MeshProjector.project (tools/map.py:414-433)                        -> p_sur, sdf, h_mask = |sdf| < threshold
//       -> texture grid at (p_sur + bound) / (2 bound)  (map.py:563, 623: L levels x 2 features, fp16 table, all levels hashed)
//       ++ FreqEncoder(sdf) = [sdf, sin(2^0 sdf), cos(2^0 sdf), .., sin(2^11 sdf), cos(2^11 sdf)]   (tools/encoding.py:5-43; map.py:584, 643)
//       -> sigma_net (network_curvedfield.py:416): tcnn FullyFusedMLP, ReLU, one hidden layer of 32, input zero-padded to 16s
//       -> h [16] fp16;  sigma = h_mask ? exp(float(h[0])) : 0;  geo_feat = h[1:]                   (network_curvedfield.py:417-422)
//
// The composed path is a projection launch, a grid launch, ~30 torch kernels for the frequency encoding, concatenation and padding,
// an MLP launch and the exp / where — with p_sur, sdf, the features and the 48-wide input making round trips through HBM.  Here
// only xyz (12 B) comes in and sigma + h (36 B) go out per sample.  A CTA owns 128-sample tiles and is warp-specialised like the
// fused field kernel (field.cu):
//   * producer warps: a lane projects ONE sample (mesh_project.cuh, the per-query body of ntx_mesh_project — a divergent pointer
//     chase with its neighbour list in registers), forms the sample's frequency encoding and writes it into its row of the K-major
//     A tile in shared memory; then the warp's lane pairs gather the texture grid for its 32 samples, 16 at a time (the lane-pair
//     gather of grid_common.cuh), into the same rows;
//   * 4 consumer warps (one per TMEM lane quarter) run the two layers on tcgen05 — [128 x K0] . W1^T -> 32 (A in shared memory),
//     ReLU / fp16 back into tensor memory, [128 x 32] . W2^T -> 16 (A in tensor memory) — and the epilogue: h rounded to fp16,
//     sigma = exp(h0) in fp32, masked.
// The kernel's time is the projection's (ntx_mesh_project alone is ~3.4 ms per 2^20 samples, the MLP ~40 us): the split between
// producers and consumers is chosen for the projection's occupancy (DESIGN §4.10).
#include "grid_common.cuh"
#include "mesh_project.cuh"
#include "mlp_tile.cuh"

namespace ntx {

#ifndef NTX_TF_PRODUCERS          // development sweeps: NTX_NVCC_EXTRA="-DNTX_TF_PRODUCERS=12 -DNTX_TF_MIN_CTAS=2"
#define NTX_TF_PRODUCERS 28
#endif
#ifndef NTX_TF_MIN_CTAS
#define NTX_TF_MIN_CTAS 1
#endif
constexpr int kTfConsumerWarps = 4;                                       // one per TMEM lane quarter
constexpr int kTfTasksPerTile = kTileRows / 32;                           // a producer warp fills 32 rows (one per lane) at a time
// Launch shape per neighbour-list length.  K <= 8 (what the product's model uses): 28 producer warps + 4 consumers = 1024 threads at
// 64 registers, one CTA per SM — the most projecting warps a 64-register kernel can have.  K <= 16 needs more than 64 registers for its
// list (it spills at 64): 12 producers, one CTA of 512 threads.  The ring has a slot for every tile the producers can be filling plus
// the one the consumers are working on.
template <int K> struct TfCfg {
    static constexpr int kProducers = K <= 8 ? NTX_TF_PRODUCERS : 12;
    static constexpr int kMinCtas = K <= 8 ? NTX_TF_MIN_CTAS : 1;
    static constexpr int kThreads = 32 * (kTfConsumerWarps + kProducers);
    static constexpr int kStages = kProducers / kTfTasksPerTile + 1;
};
constexpr uint32_t kTfHidden = 32;                                        // sigma_net's n_neurons (network_curvedfield.py:171-180)
constexpr uint32_t kTfFreq = 25;                                          // FreqEncoder(input_dim=1, multires=12).output_dim
constexpr uint32_t kTfOpndCol = 32;                                       // fp16 hidden operand [128 x 32] behind the fp32 accumulator [128 x 32]
constexpr uint32_t kTfTmemCols = 64;

// sigma_net's input width: 2L grid features + 25 frequency values, zero-padded to a multiple of 16 (the tcnn shim's padded_in)
__host__ __device__ inline uint32_t tf_in_dim(uint32_t L) { return (2u * L + kTfFreq + 15u) & ~15u; }

struct TfPlan {
    uint32_t k0;                          // tf_in_dim(L)
    uint32_t w1_off, w2_off, a_off, a_stage, mask_off, lv_off, misc_off, total;
};
constexpr uint32_t kTfMaxStages = 16;
__host__ __device__ inline TfPlan tf_plan(uint32_t L, uint32_t stages) {
    TfPlan p;
    p.k0 = tf_in_dim(L);
    p.w1_off = 0;                                         // W1 [32 x K0] K-major
    p.w2_off = kTfHidden * p.k0 * 2u;                     // W2 [16 x 32] K-major
    p.a_off = (p.w2_off + 16u * kTfHidden * 2u + 127u) & ~127u;
    p.a_stage = kTileRows * p.k0 * 2u;
    p.mask_off = p.a_off + stages * p.a_stage;         // h_mask of every row of a stage (u8)
    p.lv_off = p.mask_off + stages * kTileRows;
    p.misc_off = p.lv_off + (uint32_t)sizeof(PairLevel) * kFieldMaxLevels;
    p.total = p.misc_off + 320u;                          // barriers + TMEM slot | the output layer's StageMma (at +288)
    return p;
}

__device__ __forceinline__ void tf_consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(32 * kTfConsumerWarps) : "memory"); }

template <int K>
__global__ void __launch_bounds__(TfCfg<K>::kThreads, TfCfg<K>::kMinCtas) texture_field_density_kernel(
    const float* __restrict__ xyz, const uint32_t N, const int k_want, const float r2, const float dir_vec_wdist, const float h_threshold,
    const mesh::MeshView m, const float bound, const __half* __restrict__ table, const int* __restrict__ offsets, const uint32_t L, const float S,
    const uint32_t H, const bool align, const __half* __restrict__ w_sigma, float* __restrict__ sigma, __half* __restrict__ h_out) {
    constexpr int kTfStages = TfCfg<K>::kStages, kTfProducerWarps = TfCfg<K>::kProducers, kTfThreads = TfCfg<K>::kThreads;
    static_assert(2 * kTfStages * 8 + 8 + 4 <= 288 && kTfStages <= (int)kTfMaxStages, "barriers overlap the StageMma");
    extern __shared__ __align__(1024) uint8_t smem[];
    const TfPlan plan = tf_plan(L, kTfStages);
    const uint32_t K0 = plan.k0;
    uint8_t* w1_smem = smem + plan.w1_off;
    uint8_t* w2_smem = smem + plan.w2_off;
    uint8_t* a_smem = smem + plan.a_off;
    uint8_t* mask_smem = smem + plan.mask_off;
    PairLevel* lv = reinterpret_cast<PairLevel*>(smem + plan.lv_off);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + plan.misc_off);    // [kTfStages] producers -> consumers
    uint64_t* empty_bar = full_bar + kTfStages;                                // [kTfStages] consumers (tile done) -> producers
    uint64_t* mma_bar = empty_bar + kTfStages;                                 // layer done -> consumer warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_bar + 1);
    StageMma* out_layer = reinterpret_cast<StageMma*>(smem + plan.misc_off + 288u);

    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    // ---- one-time setup ----------------------------------------------------------------------------------------------
    if (tid == 0) {
        for (int s = 0; s < kTfStages; s++) { tc::mbar_init(&full_bar[s], kTfTasksPerTile); tc::mbar_init(&empty_bar[s], 1); }
        tc::mbar_init(mma_bar, 1);
        tc::fence_mbar_init();
    }
    if (warp == 0) tc::tmem_alloc<kTfTmemCols>(tmem_slot);
    if (tid == 32) *out_layer = stage_mma(tc::smem_u32(w2_smem), kTfHidden, 16u);
    // pair_gather4 takes levels in groups of 4: the slots past L repeat level 0 (their features are never stored)
    if (tid < ((L + 3u) & ~3u)) lv[tid] = make_pair_level(make_level<3>(offsets, tid < L ? tid : 0u, S, H, /*gridtype=*/0, align), table);
    load_matrix_kmajor(w1_smem, w_sigma, kTfHidden, K0, tid, kTfThreads);
    load_matrix_kmajor(w2_smem, w_sigma + (size_t)kTfHidden * K0, 16, kTfHidden, tid, kTfThreads);
    tc::fence_proxy_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t ntiles = ceil_div<uint32_t>(N, kTileRows);

    if (warp >= kTfConsumerWarps) {
        // =============================== PRODUCERS: project, encode, gather ==========================================
        const uint32_t pw = warp - kTfConsumerWarps;
        const uint32_t p = lane & 1u;                          // which x corner this lane gathers
        const float half_off = align ? 0.0f : 0.5f;
        // GridEncoder.forward: (inputs + bound) / (2 * bound) (grid.py:143) — torch multiplies by the fp32 reciprocal (see field.cu)
        const float inv2b = 1.0f / (2.0f * bound);
        for (uint32_t task = pw;; task += kTfProducerWarps) {
            const uint32_t k = task / kTfTasksPerTile;            // k-th tile of this CTA
            const uint32_t tile = blockIdx.x + k * gridDim.x;
            if (tile >= ntiles) break;
            const uint32_t s = k % kTfStages, use = k / kTfStages;
            const uint32_t row0 = (task % kTfTasksPerTile) * 32u;  // this warp's 32 rows of the tile
            const uint32_t bi = tile * kTileRows + row0 + lane;
            const bool valid = bi < N;
            float ps[3] = {0.f, 0.f, 0.f}, sdf = 0.f;
            if (valid) {
                float x[3];
                mesh::load3(xyz, bi, x);
                const mesh::Projection pr = mesh::project_query<K>(x, k_want, r2, dir_vec_wdist, m);
                ps[0] = pr.p_sur[0]; ps[1] = pr.p_sur[1]; ps[2] = pr.p_sur[2];
                sdf = pr.sdf;
            }
            const bool in_shell = valid && fabsf(sdf) < h_threshold;     // h_mask (map.py:429-431); NaN -> false, as in torch
            float gx = __fmul_rn(__fadd_rn(ps[0], bound), inv2b);
            float gy = __fmul_rn(__fadd_rn(ps[1], bound), inv2b);
            float gz = __fmul_rn(__fadd_rn(ps[2], bound), inv2b);
            const uint32_t cls = valid ? sample_class(gx, gy, gz) : 0u;  // casts that miss may leave the box: zero features
            if (cls != 1u) { gx = 0.f; gy = 0.f; gz = 0.f; }             // keeps the (discarded) loads of dead lanes in bounds
            // FreqEncoder (tools/encoding.py:32-43): input * freq with freq = 2^i (exact) through torch's sin / cos = sinf / cosf (not the
            // fast intrinsics), then cat -> fp32 and the MLP's cast to fp16.  z[j] = fp16 pair (2j, 2j+1) of [sdf, sin0, cos0, ..., cos11, 0]
            uint32_t z[13];
            {
                float prev = sdf;
#pragma unroll
                for (int i = 0; i < 12; i++) {
                    const float a = __fmul_rn(sdf, (float)(1 << i));
                    const float sn = sinf(a), cs = cosf(a);
                    z[i] = float2_to_half2_bits(prev, sn);
                    prev = cs;
                }
                z[12] = float2_to_half2_bits(prev, 0.0f);
            }
            tc::mbar_wait_relaxed(&empty_bar[s], (use & 1u) ^ 1u, 256u);   // slot free? (first use of a slot passes immediately)
            uint8_t* a = a_smem + s * plan.a_stage;
            mask_smem[s * kTileRows + row0 + lane] = in_shell ? 1 : 0;
#pragma unroll
            for (int j = 0; j < 13; j++) *reinterpret_cast<uint32_t*>(a + kmajor_off(row0 + lane, 2u * L + 2u * j, K0)) = z[j];
            for (uint32_t c = 2u * L + 26u; c < K0; c += 2u) *reinterpret_cast<uint32_t*>(a + kmajor_off(row0 + lane, c, K0)) = 0u;
            // texture grid: lane pair i gathers row row0 + 16 h + i
#pragma unroll 1
            for (uint32_t h = 0; h < 2; h++) {
                const uint32_t src = h * 16u + (lane >> 1);
                const float qx = __shfl_sync(0xffffffffu, gx, src), qy = __shfl_sync(0xffffffffu, gy, src), qz = __shfl_sync(0xffffffffu, gz, src);
                const uint32_t qcls = __shfl_sync(0xffffffffu, cls, src);
                for (uint32_t l0 = 0; l0 < L; l0 += 4) {
                    uint32_t packed[2];
                    pair_gather4<__half>(qx, qy, qz, qcls == 1u, p, lv + l0, half_off, packed);
                    if (qcls == 2u) { packed[0] = packed[1] = nan_features<uint32_t>(); }   // NaN coordinate: NaN features like the reference
                    const uint32_t lvl = l0 + 2u * p;                // lane p owns levels lvl, lvl + 1 -> 4 consecutive halfs of the row
                    uint8_t* dst = a + kmajor_off(row0 + src, 2u * lvl, K0);
                    if (lvl + 1u < L) *reinterpret_cast<uint2*>(dst) = make_uint2(packed[0], packed[1]);
                    else if (lvl < L) *reinterpret_cast<uint32_t*>(dst) = packed[0];
                }
            }
            tc::fence_proxy_async_smem();          // my generic-proxy writes -> visible to the tensor core's async proxy
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&full_bar[s]);
        }
    } else {
        // =============================== CONSUMERS: sigma_net on tcgen05, epilogue ====================================
        const uint32_t quarter = warp, row = quarter * 32 + lane;
        const uint32_t acc_all = tmem_base, opnd_all = tmem_base + kTfOpndCol;          // MMA addresses (all 128 lanes)
        const uint32_t acc = acc_all + ((quarter * 32u) << 16), opnd = opnd_all + ((quarter * 32u) << 16);   // this warp's lanes
        uint32_t ph = 0;
        for (uint32_t k = 0;; k++) {
            const uint32_t tile = blockIdx.x + k * gridDim.x;
            if (tile >= ntiles) break;
            const uint32_t s = k % kTfStages, use = k / kTfStages;
            // only the issuing warp waits for the tile (see field.cu); the others learn of it through the layer barrier + tf_consumer_sync
            if (warp == 0) {
                tc::mbar_wait(&full_bar[s], use & 1u);
                tc::tc_fence_after_sync();
                if (tc::elect_one()) {
                    issue_layer(tc::smem_u32(a_smem + s * plan.a_stage), tc::smem_u32(w1_smem), K0, kTfHidden, acc_all);
                    tc::mma_commit(mma_bar);
                }
                __syncwarp();
            }
            // hidden layer: ReLU, fp16, back into tensor memory as the A operand of the output layer
            tc::mbar_wait(mma_bar, ph); ph ^= 1;
            tc::tc_fence_after_sync();
            {
                uint32_t v[32], o[16];
                tc::tmem_ld_x32(acc, v);
                tc::tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 16; j++) o[j] = act_pack2(0, v[2 * j], v[2 * j + 1]);
                tc::tmem_st_x16(opnd, o);
            }
            tc::tmem_wait_st(); tc::tc_fence_before_sync(); tf_consumer_sync();
            if (warp == 0 && tc::elect_one()) {
                tc::tc_fence_after_sync();
                issue_stage_ts(out_layer, 0, opnd_all, acc_all);
                tc::mma_commit(mma_bar);
            }
            tc::mbar_wait(mma_bar, ph); ph ^= 1;
            tc::tc_fence_after_sync();
            {
                uint32_t v[16];
                tc::tmem_ld_x16(acc, v);
                tc::tmem_wait_ld();
                const uint32_t b = tile * kTileRows + row;
                if (b < N) {
                    // h = fp16(W2 . a) (the MLP's output is fp16); sigma = trunc_exp(h[..., 0]) = exp(float(h0)), where(h_mask, sigma, 0)
                    uint32_t hb[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) hb[j] = float2_to_half2_bits(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
                    const float h0 = __low2float(*reinterpret_cast<const __half2*>(&hb[0]));
                    st_stream_f32(sigma + b, mask_smem[s * kTileRows + row] ? expf(h0) : 0.0f);
                    st_stream_u4(h_out + (size_t)b * 16, make_uint4(hb[0], hb[1], hb[2], hb[3]));
                    st_stream_u4(h_out + (size_t)b * 16 + 8, make_uint4(hb[4], hb[5], hb[6], hb[7]));
                }
            }
            // tile done by all four warps: its A stage and masks may be refilled, its accumulator overwritten
            tc::tc_fence_before_sync(); tf_consumer_sync();
            if (tid == 0) tc::mbar_arrive(&empty_bar[s]);
        }
    }

    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<kTfTmemCols>(tmem_base);
}

template <int K>
static int launch_texture_field(uint32_t N, const float* xyz, uint32_t k_want, float r2, float dir_vec_wdist, float h_threshold, const mesh::MeshView& m,
                                float bound, const void* table, const int* offsets, uint32_t L, float S, uint32_t H, int align_corners,
                                const void* w_sigma, float* sigma, void* h_out, cudaStream_t stream) {
    auto kern = texture_field_density_kernel<K>;
    const TfPlan plan = tf_plan(L, TfCfg<K>::kStages);
    static int occ_dev[kMaxDevices] = {};
    static uint32_t configured_dev[kMaxDevices] = {};
    int& occ = occ_dev[current_device()];
    uint32_t& configured = configured_dev[current_device()];
    if (plan.total > configured) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.total) != cudaSuccess) {
            cudaGetLastError();
            set_error("ntx_texture_field_density: cannot reserve %u bytes of shared memory", plan.total);
            return NTX_ERR_CUDA;
        }
        configured = plan.total;
        occ = 0;
    }
    if (!occ) occ = resident_ctas_per_sm((const void*)kern, TfCfg<K>::kThreads, plan.total, kTfTmemCols);
    const uint32_t ntiles = ceil_div<uint32_t>(N, kTileRows);
    const uint32_t grid = std::min<uint32_t>(ntiles, (uint32_t)(occ * device_sm_count()));
    kern<<<grid, TfCfg<K>::kThreads, plan.total, stream>>>(xyz, N, (int)k_want, r2, dir_vec_wdist, h_threshold, m, bound, static_cast<const __half*>(table), offsets, L, S, H,
                                                   align_corners != 0, static_cast<const __half*>(w_sigma), sigma, static_cast<__half*>(h_out));
    return check_launch("ntx_texture_field_density");
}

}  // namespace ntx

using namespace ntx;

extern "C" int ntx_texture_field_density(const void* mesh, const float* vertex_normals, const float* xyz, uint32_t N, uint32_t K, float r,
                                         float dir_vec_wdist, float h_threshold, float bound, const void* embeddings_f16, const int* offsets,
                                         uint32_t L, float S, uint32_t H, int align_corners, const void* w_sigma_f16, float* sigma, void* h_f16,
                                         ntx_stream_t stream) {
    // everything that needs no device first: these checks run without a GPU
    NTX_REQUIRE(K >= 1 && K <= 16, NTX_ERR_INVALID_ARGUMENT, "ntx_texture_field_density: K must be in 1..16, got %u", K);
    NTX_REQUIRE(L >= 1 && L <= (uint32_t)kFieldMaxLevels, NTX_ERR_INVALID_ARGUMENT, "ntx_texture_field_density: L must be in 1..%d, got %u", kFieldMaxLevels, L);
    NTX_REQUIRE(r > 0.0f, NTX_ERR_INVALID_ARGUMENT, "ntx_texture_field_density: r must be positive");
    NTX_REQUIRE(bound > 0.0f, NTX_ERR_INVALID_ARGUMENT, "ntx_texture_field_density: bound must be positive");
    NTX_REQUIRE(mesh != nullptr, NTX_ERR_INVALID_ARGUMENT, "ntx_texture_field_density: not a mesh handle");
    mesh::MeshHandle* h = mesh::checked(mesh, "ntx_texture_field_density");
    if (!h) return NTX_ERR_INVALID_ARGUMENT;
    NTX_REQUIRE(h->n_triangles > 0, NTX_ERR_INVALID_ARGUMENT, "ntx_texture_field_density: the mesh has no triangles");
    if (N == 0) return NTX_OK;
    NTX_REQUIRE(vertex_normals && xyz && embeddings_f16 && offsets && w_sigma_f16 && sigma && h_f16, NTX_ERR_INVALID_ARGUMENT,
                "ntx_texture_field_density: null pointer");
    NTX_REQUIRE(((uintptr_t)w_sigma_f16 & 15) == 0 && ((uintptr_t)h_f16 & 15) == 0, NTX_ERR_INVALID_ARGUMENT,
                "ntx_texture_field_density: w_sigma and h must be 16-byte aligned");
    const mesh::MeshView m = mesh::mesh_view(h, vertex_normals);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const float r2 = r * r;
    if (K <= 8)
        return launch_texture_field<8>(N, xyz, K, r2, dir_vec_wdist, h_threshold, m, bound, embeddings_f16, offsets, L, S, H, align_corners, w_sigma_f16, sigma, h_f16, st);
    return launch_texture_field<16>(N, xyz, K, r2, dir_vec_wdist, h_threshold, m, bound, embeddings_f16, offsets, L, S, H, align_corners, w_sigma_f16, sigma, h_f16, st);
}
