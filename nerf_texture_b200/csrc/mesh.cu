// mesh.cu — the mesh front end of the texture field (SURVEY §8 f3) behind the C ABI: nearest ray/triangle hits
// (external/RayTracer, `RayTracer.trace`), K nearest mesh vertices (frnn.frnn_grid_points at tools/map.py:396,456) and the whole of
// MeshProjector.project (tools/map.py:414-433) as ONE kernel per batch of samples.
//
// Trees in the 64-byte two-box node format of mesh_bvh.cuh, read through the read-only path (the trees of the reference's meshes —
// 10^4..10^6 triangles, <= 100 MB — live in the 126 MB L2 after the first wave; one 4 x LDG.128 node fetch decides both children).
// One thread per query: neighbouring samples of a camera ray walk nearly the same nodes, and the per-thread state (a 64-entry
// stack in local memory, the K-entry neighbour list in registers) is small.  Two other mappings were built, verified bit-exact and
// measured slower on B200 (DESIGN.md, "Tried and lost"; profiles/r02_mesh_ab_*): lanes pulling queries from a per-warp chunk, and
// 8 lanes per query on an 8-wide tree.
#include "mesh_build.h"
#include "mesh_project.cuh"

#include <mutex>
#include <new>

namespace ntx {
namespace mesh {

static void free_handle(MeshHandle* h) {
    if (!h) return;
    cudaFree(h->tri_nodes); cudaFree(h->tris); cudaFree(h->pt_nodes); cudaFree(h->pts); cudaFree(h->vertices);
    h->magic = 0;
    delete h;
}

template <typename T>
static bool upload(T** dst, const std::vector<T>& src) {
    *dst = nullptr;
    const size_t bytes = std::max<size_t>(src.size(), 1) * sizeof(T);
    if (cudaMalloc((void**)dst, bytes) != cudaSuccess) return false;
    if (!src.empty() && cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) return false;
    return true;
}

// bvh.cu:695-721 raytrace_kernel.  positions may alias rays_o and normals rays_d (raytracer.py:52-54 `inplace`): a thread reads its
// ray before it writes anything.
__global__ void __launch_bounds__(128) mesh_trace_kernel(uint32_t N, const float* rays_o, const float* rays_d, float* positions, float* normals,
                                                         float* depth, long long* face_idx, const Node* __restrict__ nodes,
                                                         const Tri* __restrict__ tris, float slack) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    float ro[3], rd[3];
    load3(rays_o, i, ro);
    load3(rays_d, i, rd);
    const Hit h = trace_one(nodes, tris, ro, rd, slack);
    depth[i] = h.t;
    for (int k = 0; k < 3; k++) positions[3 * (size_t)i + k] = NTX_ADD(ro[k], NTX_MUL(h.t, rd[k]));
    float n[3] = {0.0f, 0.0f, 0.0f};
    if (h.face >= 0) {
        Tri tr;
        fetch_tri(tris, h.slot, tr);
        tri_normal(tr, n);
        face_idx[i] = h.face;   // a miss leaves the caller's value (the reference pre-fills -1, raytracer.py:37)
    }
    for (int k = 0; k < 3; k++) normals[3 * (size_t)i + k] = n[k];
}

template <int K>
__global__ void __launch_bounds__(128) mesh_knn_kernel(uint32_t N, const float* queries, float r2, int k_want, const Node* __restrict__ nodes,
                                                       const Point* __restrict__ pts, float* dists, long long* idxs) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    float q[3];
    load3(queries, i, q);
    float bd[K];
    int bi[K];
    knn_one<K>(nodes, pts, q, r2, k_want, bd, bi);
    const size_t row = (size_t)i * k_want;
#pragma unroll
    for (int s = 0; s < K; s++) {
        if (s >= K - k_want) {
            const bool ok = knn_slot_valid(bi[s]);
            dists[row + s - (K - k_want)] = ok ? bd[s] : -1.0f;
            idxs[row + s - (K - k_want)] = ok ? bi[s] : -1;
        }
    }
}

// MeshProjector.project, one thread per sample (project_query)
template <int K>
__global__ void __launch_bounds__(128) mesh_project_kernel(uint32_t N, const float* xyz, int k_want, float r2, float dir_vec_wdist, const MeshView m,
                                                           float* p_sur, float* sdf, float* normal_out, long long* face_idx) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    float x[3];
    load3(xyz, i, x);
    const Projection p = project_query<K>(x, k_want, r2, dir_vec_wdist, m);
    for (int c = 0; c < 3; c++) {
        p_sur[3 * (size_t)i + c] = p.p_sur[c];
        normal_out[3 * (size_t)i + c] = p.normal[c];
    }
    sdf[i] = p.sdf;
    face_idx[i] = p.face;
}

}  // namespace mesh
}  // namespace ntx

using namespace ntx;
using namespace ntx::mesh;

extern "C" {

int ntx_mesh_create(const float* vertices, uint32_t n_vertices, const int32_t* triangles, uint32_t n_triangles, void** mesh_out) {
    NTX_REQUIRE(mesh_out != nullptr, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_create: mesh_out is null");
    *mesh_out = nullptr;
    NTX_REQUIRE(vertices != nullptr && n_vertices > 0, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_create: no vertices");
    NTX_REQUIRE(n_triangles == 0 || triangles != nullptr, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_create: triangles is null");
    NTX_REQUIRE(n_vertices < (1u << 27) && n_triangles < (1u << 27), NTX_ERR_UNSUPPORTED, "ntx_mesh_create: more than 2^27 primitives");
    BuildResult tri_tree, pt_tree;
    std::vector<Tri> tris;
    std::vector<Point> pts;
    NTX_REQUIRE(build_triangle_tree(vertices, n_vertices, triangles, n_triangles, tri_tree, tris), NTX_ERR_INVALID_ARGUMENT,
                "ntx_mesh_create: non-finite vertex or triangle index out of range");
    NTX_REQUIRE(build_point_tree(vertices, n_vertices, pt_tree, pts), NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_create: non-finite vertex");
    NTX_REQUIRE(tri_tree.depth < kStackDepth && pt_tree.depth < kStackDepth, NTX_ERR_UNSUPPORTED, "ntx_mesh_create: tree deeper than %d", kStackDepth);
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (uint32_t i = 0; i < n_vertices; i++)
        for (int k = 0; k < 3; k++) { lo[k] = std::min(lo[k], vertices[3 * (size_t)i + k]); hi[k] = std::max(hi[k], vertices[3 * (size_t)i + k]); }
    MeshHandle* h = new (std::nothrow) MeshHandle();
    NTX_REQUIRE(h != nullptr, NTX_ERR_CUDA, "ntx_mesh_create: out of host memory");
    std::memset(h, 0, sizeof(*h));
    h->magic = kMeshMagic;
    cudaGetDevice(&h->device);
    h->n_vertices = n_vertices; h->n_triangles = n_triangles;
    h->tri_nodes_n = (uint32_t)tri_tree.nodes.size(); h->pt_nodes_n = (uint32_t)pt_tree.nodes.size();
    h->tri_depth = tri_tree.depth; h->pt_depth = pt_tree.depth;
    h->slack = 1e-5f * std::max(hi[0] - lo[0], std::max(hi[1] - lo[1], hi[2] - lo[2]));
    std::vector<float> verts(vertices, vertices + 3 * (size_t)n_vertices);
    const bool ok = upload(&h->tri_nodes, tri_tree.nodes) && upload(&h->tris, tris) && upload(&h->pt_nodes, pt_tree.nodes) && upload(&h->pts, pts) &&
                    upload(&h->vertices, verts);
    if (!ok) {
        set_error("ntx_mesh_create: %s", cudaGetErrorString(cudaGetLastError()));
        free_handle(h);
        return NTX_ERR_CUDA;
    }
    *mesh_out = h;
    return NTX_OK;
}

int ntx_mesh_destroy(void* mesh) {
    if (!mesh) return NTX_OK;
    MeshHandle* h = (MeshHandle*)mesh;
    NTX_REQUIRE(h->magic == kMeshMagic, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_destroy: not a mesh handle");
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(h->device);
    free_handle(h);
    if (prev >= 0) cudaSetDevice(prev);
    return NTX_OK;
}

int ntx_mesh_info(const void* mesh, uint32_t* out6) {
    const MeshHandle* h = (const MeshHandle*)mesh;
    NTX_REQUIRE(h && h->magic == kMeshMagic && out6, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_info: not a mesh handle");
    out6[0] = h->n_vertices; out6[1] = h->n_triangles; out6[2] = h->tri_nodes_n; out6[3] = h->tri_depth; out6[4] = h->pt_nodes_n; out6[5] = h->pt_depth;
    return NTX_OK;
}

int ntx_mesh_trace(const void* mesh, const float* rays_o, const float* rays_d, float* positions, float* normals, float* depth, int64_t* face_idx,
                   uint32_t N, ntx_stream_t stream) {
    MeshHandle* h = checked(mesh, "ntx_mesh_trace");
    if (!h) return NTX_ERR_INVALID_ARGUMENT;
    if (N == 0) return NTX_OK;
    NTX_REQUIRE(rays_o && rays_d && positions && normals && depth && face_idx, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_trace: null pointer");
    const uint32_t block = (uint32_t)tunables().mesh_block;
    mesh_trace_kernel<<<ceil_div(N, block), block, 0, (cudaStream_t)stream>>>(N, rays_o, rays_d, positions, normals, depth, (long long*)face_idx,
                                                                          h->tri_nodes, h->tris, h->slack);
    return check_launch("ntx_mesh_trace");
}

int ntx_mesh_knn(const void* mesh, const float* queries, uint32_t N, uint32_t K, float r, float* dists, int64_t* idxs, ntx_stream_t stream) {
    MeshHandle* h = checked(mesh, "ntx_mesh_knn");
    if (!h) return NTX_ERR_INVALID_ARGUMENT;
    NTX_REQUIRE(K >= 1 && K <= 32, NTX_ERR_UNSUPPORTED, "ntx_mesh_knn: K must be in 1..32, got %u", K);
    NTX_REQUIRE(r > 0.0f, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_knn: r must be positive");
    if (N == 0) return NTX_OK;
    NTX_REQUIRE(queries && dists && idxs, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_knn: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const float r2 = r * r;
    const uint32_t block = (uint32_t)tunables().mesh_block;
    const dim3 grid(ceil_div(N, block));
    if (K <= 8) {
        mesh_knn_kernel<8><<<grid, block, 0, st>>>(N, queries, r2, (int)K, h->pt_nodes, h->pts, dists, (long long*)idxs);
    } else if (K <= 16) {
        mesh_knn_kernel<16><<<grid, block, 0, st>>>(N, queries, r2, (int)K, h->pt_nodes, h->pts, dists, (long long*)idxs);
    } else {
        mesh_knn_kernel<32><<<grid, block, 0, st>>>(N, queries, r2, (int)K, h->pt_nodes, h->pts, dists, (long long*)idxs);
    }
    return check_launch("ntx_mesh_knn");
}

int ntx_mesh_project(const void* mesh, const float* vertex_normals, const float* xyz, uint32_t N, uint32_t K, float r, float dir_vec_wdist,
                     float* p_sur, float* sdf, float* normal, int64_t* face_idx, ntx_stream_t stream) {
    MeshHandle* h = checked(mesh, "ntx_mesh_project");
    if (!h) return NTX_ERR_INVALID_ARGUMENT;
    NTX_REQUIRE(K >= 1 && K <= 16, NTX_ERR_UNSUPPORTED, "ntx_mesh_project: K must be in 1..16, got %u", K);
    NTX_REQUIRE(r > 0.0f, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_project: r must be positive");
    NTX_REQUIRE(h->n_triangles > 0, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_project: the mesh has no triangles");
    if (N == 0) return NTX_OK;
    NTX_REQUIRE(vertex_normals && xyz && p_sur && sdf && normal && face_idx, NTX_ERR_INVALID_ARGUMENT, "ntx_mesh_project: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const float r2 = r * r;
    const uint32_t block = (uint32_t)tunables().mesh_block;
    const dim3 grid(ceil_div(N, block));
    const MeshView m = mesh_view(h, vertex_normals);
    if (K <= 8) {
        mesh_project_kernel<8><<<grid, block, 0, st>>>(N, xyz, (int)K, r2, dir_vec_wdist, m, p_sur, sdf, normal, (long long*)face_idx);
    } else {
        mesh_project_kernel<16><<<grid, block, 0, st>>>(N, xyz, (int)K, r2, dir_vec_wdist, m, p_sur, sdf, normal, (long long*)face_idx);
    }
    return check_launch("ntx_mesh_project");
}

}  // extern "C"
