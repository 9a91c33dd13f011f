/* ntx.h — C ABI of libntx.so: B200 (sm_100a) kernels for NeRF-Texture's per-ray-sample hot path.
 *
 * Every entry point is `extern "C"`, takes plain device pointers + sizes + a cudaStream_t, allocates
 * nothing, does not synchronise the stream (one exception: ntx_render_rays, see there) and returns 0 on success or a negative ntx_status (no exceptions cross
 * the ABI; ntx_last_error() gives the message of the calling thread's last failure).  The caller owns all
 * buffers, exactly like the reference's natives, which write into caller-allocated tensors and return void.
 * The device is the current CUDA context's.  Calls on distinct streams are thread-safe.
 *
 * Each function names the reference interface it replaces (paths relative to yihua7/NeRF-Texture).
 * The Python packages gridencoder / ffmlp / shencoder / raymarching shipped in nerf_texture_b200/compat bind
 * these with ctypes; INTEGRATION.md shows the binding a reference maintainer would add.
 */
#ifndef NTX_H_
#define NTX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* ntx_stream_t; /* == cudaStream_t */

typedef enum {
    NTX_OK = 0,
    NTX_ERR_INVALID_ARGUMENT = -1, /* reference: TORCH_CHECK / std::runtime_error -> RuntimeError in Python */
    NTX_ERR_UNSUPPORTED = -2,      /* e.g. "GridEncoding: C must be 1, 2, 4, or 8." (gridencoder.cu:355) */
    NTX_ERR_CUDA = -3,             /* launch / runtime failure (the reference never checks: SURVEY F8) */
    NTX_ERR_WORKSPACE = -4
} ntx_status;

typedef enum { NTX_F32 = 0, NTX_F16 = 1, NTX_F64 = 2 } ntx_dtype;

/* layouts of the [levels x samples x features] grid tensors */
typedef enum {
    NTX_LAYOUT_LBC = 0, /* [L,B,C]: the reference kernel's layout (gridencoder.cu:362) */
    NTX_LAYOUT_BLC = 1  /* [B,L*C]: what grid_encode() returns after its permute (grid.py:52) — no extra copy */
} ntx_grid_layout;

const char* ntx_last_error(void);
int ntx_version(void);
/* 1 if the library was built with sm_100a SASS and the current device is CC 10.x */
int ntx_device_ok(void);

/* ------------------------------------------------------------------------------------------------ gridencoder
 * replaces grid_encode_forward / grid_encode_backward (gridencoder/src/gridencoder.h:12-13, gridencoder.cu:419,444)
 *   inputs      [B,D] f32 in [0,1]           embeddings [n_entries,C] dtype      offsets [L+1] i32
 *   outputs     [L,B,C] or [B,L*C] dtype     dy_dx [B, L*D*C] dtype (only if calc_grad_inputs)
 *   S = log2(per_level_scale) as f32, H = base resolution, gridtype 0 hash / 1 tiled.
 * D in {2,3}, C in {1,2,4,8}; anything else -> NTX_ERR_UNSUPPORTED (reference: std::runtime_error). */
int ntx_grid_encode_forward(const float* inputs, const void* embeddings, const int* offsets, void* outputs,
                            uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H,
                            int calc_grad_inputs, void* dy_dx, uint32_t gridtype, int align_corners,
                            int dtype, int out_layout, ntx_stream_t stream);
/*   grad [L,B,C] or [B,L*C] dtype;  grad_embeddings [n_entries,C] dtype, zero-initialised by the caller (grid.py:74);
 *   grad_inputs [B,D] dtype (only if calc_grad_inputs; needs the dy_dx saved by the forward) */
int ntx_grid_encode_backward(const void* grad, const float* inputs, const void* embeddings, const int* offsets,
                             void* grad_embeddings, uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H,
                             int calc_grad_inputs, const void* dy_dx, void* grad_inputs, uint32_t gridtype,
                             int align_corners, int dtype, int grad_layout, ntx_stream_t stream);
/* test hooks: the per-level `scale` the device computes (gridencoder.cu:126) and the integer corner-index
 * stream of one level, idx[b*2^D + corner] (0xffffffff for out-of-range samples) */
int ntx_grid_level_scales(float S, uint32_t H, uint32_t L, float* scales_out, ntx_stream_t stream);
int ntx_grid_debug_indices(const float* inputs, const int* offsets, uint32_t B, uint32_t D, uint32_t level, float S,
                           uint32_t H, uint32_t gridtype, int align_corners, uint32_t* idx_out, ntx_stream_t stream);

/* ------------------------------------------------------------------------------------------------ ffmlp
 * replaces ffmlp_forward / ffmlp_inference / ffmlp_backward / allocate_splitk / free_splitk
 * (ffmlp/src/ffmlp.h:8-14, ffmlp.cu:635,673,749,721,732).  All tensors fp16.
 *   inputs [B,input_dim]   weights flat [hidden*input_dim + (num_layers-1)*hidden*hidden + output_dim*hidden],
 *   each matrix row-major [out,in] (ffmlp.cu:632)   outputs [B,output_dim]   output_dim <= 16 is padded to 16
 *   by the caller (ffmlp.py:118).  The reference needs B % 128 == 0 (ffmlp.py:157 pads with zero rows); here any B works,
 *   the kernel masks the ragged last 128-row tile.
 *   forward_buffer [num_layers,B,hidden] (training), backward_buffer likewise.  activation ids: ffmlp.cu:22-33.
 * hidden_dim in {16,32,64,128,256} (ffmlp.cu:652-659), as long as all weight matrices + one 128-row activation tile fit
 * the SM's 227 KB of shared memory; anything else -> NTX_ERR_UNSUPPORTED. */
int ntx_ffmlp_forward(const void* inputs, const void* weights, uint32_t B, uint32_t input_dim, uint32_t output_dim,
                      uint32_t hidden_dim, uint32_t num_layers, uint32_t activation, uint32_t output_activation,
                      void* forward_buffer, void* outputs, ntx_stream_t stream);
int ntx_ffmlp_inference(const void* inputs, const void* weights, uint32_t B, uint32_t input_dim, uint32_t output_dim,
                        uint32_t hidden_dim, uint32_t num_layers, uint32_t activation, uint32_t output_activation,
                        void* inference_buffer /* unused, may be NULL */, void* outputs, ntx_stream_t stream);
/* workspace: fp32 scratch for the weight-gradient reduction, ntx_ffmlp_backward_workspace_bytes() bytes */
size_t ntx_ffmlp_backward_workspace_bytes(uint32_t input_dim, uint32_t output_dim, uint32_t hidden_dim, uint32_t num_layers);
int ntx_ffmlp_backward(const void* grad, const void* inputs, const void* weights, const void* forward_buffer,
                       uint32_t B, uint32_t input_dim, uint32_t output_dim, uint32_t hidden_dim, uint32_t num_layers,
                       uint32_t activation, uint32_t output_activation, int calc_grad_inputs, void* backward_buffer,
                       void* grad_inputs, void* grad_weights, void* workspace, ntx_stream_t stream);
/* kept for drop-in parity with ffmlp.py:126,133 — the B200 path needs no side streams; both are no-ops */
int ntx_allocate_splitk(size_t size);
int ntx_free_splitk(void);

/* ------------------------------------------------------------------------------------------------ shencoder
 * replaces sh_encode_forward / sh_encode_backward (shencoder/src/shencoder.h:10,13, shencoder.cu:402,421).  fp32 only
 * (the Python wrapper forces fp32: sphere_harmonics.py:16).  inputs [B,3], outputs [B,C*C], dy_dx [B,3*C*C], C in 1..8. */
int ntx_sh_encode_forward(const float* inputs, float* outputs, uint32_t B, uint32_t D, uint32_t C,
                          int calc_grad_inputs, float* dy_dx, ntx_stream_t stream);
/* grad_inputs [B,3] is ACCUMULATED into (shencoder.cu:377); the caller zero-fills it (sphere_harmonics.py:50) */
int ntx_sh_encode_backward(const float* grad, const float* inputs, uint32_t B, uint32_t D, uint32_t C,
                           const float* dy_dx, float* grad_inputs, ntx_stream_t stream);

/* ------------------------------------------------------------------------------------------------ raymarching
 * replaces the natives of raymarching/src/raymarching.h:7-20 (fp32 / int32 / uint8 only; the Python wrappers cast
 * everything to fp32: raymarching.py custom_fwd(cast_inputs=torch.float32)). */
int ntx_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N, float min_near,
                           float* nears, float* fars, ntx_stream_t stream);
int ntx_polar_from_ray(const float* rays_o, const float* rays_d, float radius, uint32_t N, float* coords, ntx_stream_t stream);
int ntx_morton3D(const int* coords, uint32_t N, int* indices, ntx_stream_t stream);
int ntx_morton3D_invert(const int* indices, uint32_t N, int* coords, ntx_stream_t stream);
int ntx_packbits(const float* grid, uint32_t N, float density_thresh, uint8_t* bitfield, ntx_stream_t stream);

/* march_rays_train (raymarching.cu:485) and, with rays_ts != NULL, march_rays_train_differentiable (:680).
 * counter [2] i32 = {samples, rays}: ADDED to, like the reference's atomicAdd; the caller zeroes it (renderer.py:367).
 * Segments are allocated by an ordered scan, so rays[] rows and sample offsets come out in ascending ray order — a
 * deterministic member of the reference's (atomic, arbitrary-order) outcome set.
 * workspace: ntx_march_rays_train_workspace_bytes(N) bytes, zero on first use (the kernel leaves it zeroed). */
size_t ntx_march_rays_train_workspace_bytes(uint32_t N);
int ntx_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound, float dt_gamma,
                         uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M, const float* nears,
                         const float* fars, float* xyzs, float* dirs, float* deltas, float* rays_ts, int* rays,
                         int* counter, uint32_t perturb, void* workspace, ntx_stream_t stream);
int ntx_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* deltas, const int* rays,
                                     uint32_t M, uint32_t N, float* weights_sum, float* depth, float* image,
                                     ntx_stream_t stream);
int ntx_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_image, const float* sigmas,
                                      const float* rgbs, const float* deltas, const int* rays, const float* weights_sum,
                                      const float* image, uint32_t M, uint32_t N, float* grad_sigmas, float* grad_rgbs,
                                      ntx_stream_t stream);
/* inference loop body (raymarching.cu:1009,1107,1137).  xyzs/dirs/deltas must be zero-filled by the caller for slots
 * that are not written (raymarching.py:389-391) unless zero_fill != 0, in which case the kernel writes the zeros itself
 * (saves three memsets per loop iteration; M_padded = rows of xyzs/dirs/deltas). */
int ntx_march_rays(uint32_t n_alive, uint32_t n_step, const int* rays_alive, const float* rays_t, const float* rays_o,
                   const float* rays_d, float bound, float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H,
                   const uint8_t* grid, const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                   uint32_t perturb, int zero_fill, uint32_t M_padded, const uint8_t* occupancy_mip /* nullable */, ntx_stream_t stream);
/* Optional accelerator of march_rays: a conservative (dilated) 4x4x4-cell mip of the occupancy bit-field.  With it the marcher
 * stops walking a ray through empty space as soon as no occupied voxel can be reached any more; the emitted samples are
 * unchanged (such a ray emits nothing further and is marked dead by composite_rays whatever t it stops at).
 * mip: ntx_occupancy_mip_bytes(C,H) bytes; rebuild whenever the bit-field changes.  H must be a power of two >= 16. */
size_t ntx_occupancy_mip_bytes(uint32_t C, uint32_t H);
int ntx_build_occupancy_mip(const uint8_t* grid, uint32_t C, uint32_t H, uint8_t* mip, ntx_stream_t stream);
/* composite_rays (raymarching.cu:1021-1104).  One extension over the reference: a slot with deltas == (0, -t), t > 0, is the
 * "paused" marker the marcher of ntx_render_rays writes (walk_budget): the ray stops compositing there but stays alive with
 * rays_t = t.  The reference's marcher (and ntx_march_rays) only ever writes (0, 0) into unused slots, for which the behaviour
 * is the reference's: rays_t = -1. */
int ntx_composite_rays(uint32_t n_alive, uint32_t n_step, const int* rays_alive, float* rays_t, const float* sigmas,
                       const float* rgbs, const float* deltas, float* weights_sum, float* depth, float* image,
                       ntx_stream_t stream);
/* compact_rays: survivors (rays_t_old >= 0) are written in ascending slot order (warp-ballot + block scan + chained
 * look-back); alive_counter [1] is ADDED to.  workspace: ntx_compact_rays_workspace_bytes(n_alive), zero on first use. */
size_t ntx_compact_rays_workspace_bytes(uint32_t n_alive);
int ntx_compact_rays(uint32_t n_alive, int* rays_alive, const int* rays_alive_old, float* rays_t, const float* rays_t_old,
                     int* alive_counter, void* workspace, ntx_stream_t stream);

/* ------------------------------------------------------------------------------------------------ fused field
 * One launch for nerf/network_ff.py:85-101 in fp16 inference mode:
 *   x01 = (xyz+bound)/(2 bound) -> hash-grid (D=3, C=2, L<=16, fp16 table) -> FFMLP(2L -> 64 -> 16) -> sigma = exp(h0)*density_scale
 *   SH(dirs, degree 4) ++ h[1..15] ++ 0 -> FFMLP(32 -> 64 -> 64 -> 16)[:3] -> sigmoid -> rgb
 * Features, hidden activations and geo_feat never leave the SM (smem / TMEM); the two MLPs run on tcgen05.
 * xyz, dirs [M,3] f32; sigmas [M] f32; rgbs [M,3] f32.  Rows whose deltas (optional, [M,2]) are 0 are skipped. */
int ntx_ngp_field_forward(const float* xyz, const float* dirs, const float* deltas /* nullable */, uint32_t M, float bound,
                          const void* embeddings_f16, const int* offsets, uint32_t L, float S, uint32_t H,
                          int align_corners, const void* w_sigma_f16, const void* w_color_f16, float density_scale,
                          float* sigmas, float* rgbs, ntx_stream_t stream);

/* ------------------------------------------------------------------------------------------------ whole frame
 * The inference branch of NeRFRenderer.run_cuda (nerf/renderer.py:436-489) as ONE call: near_far_from_aabb, then per
 * iteration compact_rays -> march_rays -> field -> composite_rays, with exactly the reference's bookkeeping
 * (n_step = clamp(N // n_alive, 1, 8), samples padded to 128, step += n_step, stop at n_alive == 0 or step >= max_steps).
 * The reference reads n_alive back with a blocking .item() every iteration (renderer.py:469); here the loop state lives on
 * the device (the kernels read n_alive / n_step from it), grids are sized from a bound that lags two iterations behind
 * through a pinned host mailbox, and the launching thread never lets the stream run dry.  Results are bit-identical to
 * calling the individual entry points in the reference's order.
 *   sample_budget, max_n_step: samples per iteration n_step = clamp(sample_budget // n_alive, 1, max_n_step).  (0, 0) = (N, 8) is
 *     the reference's schedule.  The image does not depend on the schedule (a ray's samples are composited in the same order and
 *     stop at the same sample; only how many iterations that takes, and how many samples past an opaque ray's stop are evaluated
 *     and discarded, changes), so a B200 with memory to spare can run e.g. (4N, 32) and cut the number of iterations.
 *     Exceptions: perturb != 0 (the reference jitters t once per march_rays call, so the schedule is part of the random
 *     realisation) and rays that need more than max_steps samples (the step budget is checked once per iteration).
 *   walk_budget: 0 = the reference's iteration structure.  > 0: after the first iteration a ray that has crossed this many empty
 *     voxels in one march without filling its n_step slots pauses (sentinel (0, -t), see raymarch.cu) and carries on in the next
 *     iteration from exactly that t: same samples, same image, but a launch no longer lasts as long as its longest walk.
 *     With walk_budget > 0 and an occupancy mip the mip is consulted once per ray before the loop: rays that cannot reach an occupied
 *     cell start dead (they would emit nothing and be dropped by the first composite_rays) and the others' `far` is shortened to the
 *     end of their last maybe-occupied stretch; wide schedules (max_n_step > 8) round n_step down to a multiple of 4.
 *     A ray that never pauses may then take up to max_steps + pause allowance samples where the reference truncates at max_steps
 *     (only reachable when a ray crosses more than max_steps occupied lattice points); pass walk_budget = 0 where that cap matters.
 *   rays_o, rays_d [N,3] f32; aabb [6] f32 (device); grid = density bit-field; occupancy_mip nullable (ntx_build_occupancy_mip)
 *   weights_sum [N], depth [N], image [N,3] f32: overwritten (image WITHOUT the background term, like composite_rays)
 *   workspace: ntx_render_rays_workspace_bytes(N, sample_budget) bytes of device memory, 256-byte aligned
 *   host_mailbox: max_steps + 2*H*C + 8 ints of pinned, device-mapped host memory (cudaHostAlloc / torch pin_memory)
 *   sample_counter: nullable device counter, incremented by the number of samples marched (statistics)
 *   stats_out: nullable host pointer to 2 uint32: [0] loop iterations that had rays alive, [1] kernels launched by this call
 *   kernel_ms_out: nullable host pointer to 2 floats.  When given, every march and field launch of the frame is bracketed by
 *     CUDA events on `stream`, the call synchronises the stream at the end and returns [0] the summed march-kernel time and
 *     [1] the summed field-kernel time in ms (bench.py's roofline; costs a few event records, do not use in production).
 * The call waits on its own run-ahead events (the ABI's one exception to "does not synchronise") and serialises concurrent callers
 * on the same device with a per-device mutex (its events are per-device state); calls on different devices do not interact. */
size_t ntx_render_rays_workspace_bytes(uint32_t N, uint32_t sample_budget);
int ntx_render_rays(const float* rays_o, const float* rays_d, uint32_t N, const float* aabb, float min_near, float bound,
                    float dt_gamma, uint32_t max_steps, uint32_t perturb, uint32_t sample_budget, uint32_t max_n_step,
                    uint32_t walk_budget, uint32_t C, uint32_t H, const uint8_t* grid,
                    const uint8_t* occupancy_mip, const void* embeddings_f16, const int* offsets, uint32_t L, float S,
                    uint32_t base_resolution, int align_corners, const void* w_sigma_f16, const void* w_color_f16,
                    float density_scale, float* weights_sum, float* depth, float* image, void* workspace,
                    int* host_mailbox, unsigned long long* sample_counter, uint32_t* stats_out, float* kernel_ms_out,
                    ntx_stream_t stream);

/* Epilogue of a ray-sharded frame (BASELINE config 4): rank r rendered the interleaved tiles k = r, r + world, ... (tile rays each)
 * into a planar block [weights_sum (n_max) | depth (n_max) | rgb (3 n_max)] f32; `gathered` = the world blocks after ONE all-gather.
 * Puts every ray back at its image position and adds the background term image + (1 - weights_sum) * bg (renderer.py:485).
 * world = 1: the single-GPU epilogue. */
int ntx_unshard_frame(const float* gathered, uint32_t world, uint32_t n_max, uint32_t tile, uint32_t N, float bg,
                      float* image, float* depth, float* weights_sum, ntx_stream_t stream);

/* The same epilogue fused with the exchange: `peers_dev` is a DEVICE array of `world` pointers, entry r = this rank's NVLink mapping of
 * rank r's planar block buffer (symmetric memory: cudaIpc / torch.distributed._symmetric_memory buffer_ptrs_dev); the block of this
 * frame starts `offset_floats` into each buffer.  The kernel reads the peers' blocks in place while it un-permutes — no all-gather, no
 * staging copy.  The caller must order it after a cross-rank barrier (all blocks written) and must not overwrite a block before every
 * rank has passed the next barrier (double-buffer the blocks). */
int ntx_unshard_frame_peers(const void* peers_dev, size_t offset_floats, uint32_t world, uint32_t n_max, uint32_t tile,
                            uint32_t N, float bg, float* image, float* depth, float* weights_sum, ntx_stream_t stream);

/* ------------------------------------------------------------------------------------------------ density-grid maintenance
 * The density-grid half of NeRFRenderer.update_extra_state (nerf/renderer.py:567-647) as one launch chain, no host round trip:
 *   tmp_grid = -1; for every cascade: query sigma * density_scale at the grid cells (positions generated in the kernel from the
 *   cells' Morton indices exactly as renderer.py:590-598 computes them, hash-grid gather + sigma MLP fused: the field kernel in
 *   density mode) -> tmp_grid[cas, cell]; density_grid[valid] = max(density_grid[valid] * decay, tmp_grid[valid]);
 *   mean_density = mean(clamp(density_grid, min=0)); packbits(density_grid, min(mean_density, density_thresh)) -> density_bitfield.
 *   density_grid [C, H^3] f32 (in/out, Morton order per cascade), density_bitfield [C*H^3/8] u8 (out), H a power of two
 *   cells: nullable [C, n_cells] i32 Morton indices (the partial update of renderer.py:603-625; duplicates: one of the writers wins, as
 *     in the reference's index_put); null = every cell of every cascade (full update), n_cells ignored
 *   noise: nullable uniform [0,1) jitter `torch.rand_like(cas_xyzs)` (renderer.py:597), [C, n, 3] f32: row = list position when
 *     `cells` is given, else the x-major meshgrid index (x*H + y)*H + z of the cell; null = cell centres
 *   workspace: ntx_update_density_grid_workspace_bytes(C, H) bytes, 256-byte aligned
 *   stats_out: device [2] f32 = {mean_density, the threshold used}
 * Field parameters as in ntx_ngp_field_forward (only the sigma net is evaluated). */
size_t ntx_update_density_grid_workspace_bytes(uint32_t C, uint32_t H);
int ntx_update_density_grid(float* density_grid, uint8_t* density_bitfield, uint32_t C, uint32_t H, float bound,
                            float density_scale, float decay, float density_thresh, const void* embeddings_f16,
                            const int* offsets, uint32_t L, float S, uint32_t base_resolution, int align_corners,
                            const void* w_sigma_f16, const int* cells, uint32_t n_cells, const float* noise,
                            int force_full_grid, void* workspace, float* stats_out, ntx_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------------------
 * Mesh front end of the texture field (SURVEY §8 f3): what MeshProjector.project (tools/map.py:414-433) does per sample —
 * K nearest mesh vertices (frnn.frnn_grid_points, tools/map.py:396,456) -> coarse normal (tools/map.py:454-500) -> two nearest-hit ray
 * casts along +-normal (external/RayTracer) -> surface point, signed distance, face.
 *
 * ntx_mesh_create replaces `_raytracing.create_raytracer(vertices, triangles)` (external/RayTracer/src/bindings.cpp:17,
 * src/raytracer.cu:21-41) AND the grid frnn builds on its first call (tools/map.py:396): HOST arrays `vertices` [n_vertices,3] f32 and
 * `triangles` [n_triangles,3] i32 (n_triangles may be 0: neighbour queries only) -> an opaque handle that owns the two search trees on
 * the CURRENT device.  Non-finite vertices and out-of-range indices -> NTX_ERR_INVALID_ARGUMENT.  Unlike the reference wrapper
 * (raytracer.py:17-24) meshes of <= 8 triangles need no padding.  The call synchronises (cudaMalloc + cudaMemcpy), like the reference's.
 * ntx_mesh_info: out6 = {n_vertices, n_triangles, triangle-tree nodes, its depth, vertex-tree nodes, its depth}. */
int ntx_mesh_create(const float* vertices, uint32_t n_vertices, const int32_t* triangles, uint32_t n_triangles, void** mesh_out);
int ntx_mesh_destroy(void* mesh);
int ntx_mesh_info(const void* mesh, uint32_t* out6);

/* `RayTracer::trace` (external/RayTracer/include/raytracing/raytracer.h:20, src/bvh.cu:695-721): for each ray the nearest triangle hit
 * with 0 <= t < 10 (MAX_DIST, bvh.cu:36) by the formula of triangle.cuh:27-39.
 *   rays_o, rays_d [N,3] f32 (device) -> depth [N] = t or 10, positions [N,3] = o + depth * d, normals [N,3] = unit face normal or 0,
 *   face_idx [N] i64 = index into `triangles`; a MISS LEAVES face_idx UNTOUCHED (the reference's wrapper pre-fills -1, raytracer.py:37).
 *   positions may alias rays_o and normals rays_d (the wrapper's inplace=True).
 * The result is that of an exhaustive scan over the triangles in index order (ties in t: lowest index); every product and sum of the
 * hit formula is rounded separately.  The reference's own binary may differ in the last bits where nvcc fused multiply-adds. */
int ntx_mesh_trace(const void* mesh, const float* rays_o, const float* rays_d, float* positions, float* normals, float* depth,
                   int64_t* face_idx, uint32_t N, ntx_stream_t stream);

/* frnn.frnn_grid_points(queries[None], vertices[None], K=K, r=r, return_sorted=True) for one batch element: the K nearest mesh
 * vertices with squared distance < r*r, ascending (ties: lowest index).  dists [N,K] f32 SQUARED distances, idxs [N,K] i64; both
 * padded with -1 when fewer than K vertices are in range.  1 <= K <= 32. */
int ntx_mesh_knn(const void* mesh, const float* queries, uint32_t N, uint32_t K, float r, float* dists, int64_t* idxs, ntx_stream_t stream);

/* MeshProjector.project(xyz, K) up to its two torch one-liners on the outputs (tbn = self.tbn[face_idx], h_mask = |sdf| < threshold),
 * fused into one kernel: per sample the K-neighbour list stays in registers, the coarse normal of knn(use_dir_vec=True,
 * weighting='Shepard', dir_vec_wdist) is formed from `vertex_normals` [n_vertices,3] f32 (device) and both casts run back to back.
 *   -> p_sur [N,3], sdf [N] (-depth_inner if depth_inner < depth_outer else depth_outer), normal [N,3], face_idx [N] i64 (-1: neither
 *   cast hit anything within 10).  1 <= K <= 16; the mesh must have triangles.
 * Queries are independent and may come in any order; the kernels run one thread per query, so a batch whose neighbours in memory are
 * neighbours in space is up to 1.6x faster (nerf_texture_b200/mesh.py orders batches of 2^19 or more along a Morton curve). */
int ntx_mesh_project(const void* mesh, const float* vertex_normals, const float* xyz, uint32_t N, uint32_t K, float r, float dir_vec_wdist,
                     float* p_sur, float* sdf, float* normal, int64_t* face_idx, ntx_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------------------
 * Fused texture-field density: NeRFNetwork.density(x) of the product's model (nerf/network_curvedfield.py:412-433) in fp16 inference,
 * for the configuration main.py trains (MeshFeatureField with hash=True, prob_model=False, no imported texture; sigma_net = tcnn
 * FullyFusedMLP, ReLU, one hidden layer of 32 neurons, no output activation), as ONE kernel:
 *   MeshProjector.project(xyz, K) as in ntx_mesh_project (tools/map.py:414-433) -> p_sur, sdf
 *   x_embed = texture grid at (p_sur + bound) / (2 bound)  (tools/map.py:563,623; D = 3, C = 2, L levels, every level hashed, fp16 table
 *             as under autocast; out-of-range coordinates — casts that miss may leave the box — give zero features, like the reference)
 *   z_embed = FreqEncoder(sdf) = [sdf, sin(2^i sdf), cos(2^i sdf) for i = 0..11]  (tools/encoding.py:5-43, get_encoder('frequency', multires=12))
 *   h = sigma_net(cat(x_embed, z_embed) zero-padded to 16*ceil((2L+25)/16), rounded to fp16)  (tools/map.py:719, network_curvedfield.py:416)
 *   sigma = |sdf| < h_threshold ? exp(float(h[0])) : 0        (trunc_exp + torch.where, network_curvedfield.py:417-421)
 *   h_threshold = min(MeshProjector.depth_threshold, MeshFeatureField.h_threshold) as fp32 (tools/map.py:429-431)
 *   mesh, vertex_normals, K, r, dir_vec_wdist as in ntx_mesh_project; embeddings_f16, offsets, L, S, H, align_corners as in
 *   ntx_ngp_field_forward.  w_sigma_f16: the tinycudann shim's flat parameters [32 x in | 16 x 32] fp16, each matrix row-major [out,in].
 *   xyz [N,3] f32 -> sigma [N] f32, h_f16 [N,16] fp16 (geo_feat = h[:, 1:]).  w_sigma_f16 and h_f16 16-byte aligned.
 * Every sample gets h, also those outside the shell (sigma 0) and those whose casts miss (sdf = 10).  A null or triangle-less mesh,
 * K outside 1..16 or L outside 1..32 -> NTX_ERR_INVALID_ARGUMENT (checked before the device is touched, except the triangle count);
 * N = 0 is a no-op.  Queries are independent: like ntx_mesh_project, a batch in Morton order runs faster.
 * Measured on one B200 (1000 W power limit), 2^20 samples around a 230 K-triangle mesh: 5.54 ms, against 4.74 ms for the same computation
 * composed from the drop-in operators — not yet faster, see DESIGN.md §4.10 (profiles/r03_texture_field.txt). */
int ntx_texture_field_density(const void* mesh, const float* vertex_normals, const float* xyz, uint32_t N, uint32_t K, float r,
                              float dir_vec_wdist, float h_threshold, float bound, const void* embeddings_f16, const int* offsets,
                              uint32_t L, float S, uint32_t H, int align_corners, const void* w_sigma_f16, float* sigma, void* h_f16,
                              ntx_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NTX_H_ */
