// mesh_project.cuh — the mesh handle and the per-query body of MeshProjector.project (tools/map.py:414-433), shared by mesh.cu
// (ntx_mesh_project: one thread per query, results to global memory) and texture_field.cu (the projection feeds the texture-grid
// gather of the same thread without leaving its registers).
#pragma once

#include "common.cuh"
#include "mesh_bvh.cuh"

namespace ntx {
namespace mesh {

constexpr uint32_t kMeshMagic = 0x4d53484eu;

struct MeshHandle {
    uint32_t magic;
    int device;
    uint32_t n_vertices, n_triangles;
    uint32_t tri_nodes_n, pt_nodes_n, tri_depth, pt_depth;
    float slack;          // pruning slack of trace_one: 1e-5 of the mesh's largest extent
    Node* tri_nodes;
    Tri* tris;
    Node* pt_nodes;
    Point* pts;
    float* vertices;      // [n_vertices, 3] in the caller's order (the fused projection gathers neighbours by index)
};

// the handle behind an ABI pointer, or null (message set) if it is not one or lives on another device
static inline MeshHandle* checked(const void* mesh, const char* who) {
    MeshHandle* h = (MeshHandle*)mesh;
    if (!h || h->magic != kMeshMagic) { set_error("%s: not a mesh handle", who); return nullptr; }
    int dev = -1;
    cudaGetDevice(&dev);
    if (dev != h->device) { set_error("%s: the mesh lives on device %d, the current device is %d", who, h->device, dev); return nullptr; }
    return h;
}

__device__ __forceinline__ void load3(const float* p, uint32_t i, float* v) {
    v[0] = p[3 * (size_t)i]; v[1] = p[3 * (size_t)i + 1]; v[2] = p[3 * (size_t)i + 2];
}

__device__ __forceinline__ float norm3(const float* v) { return sqrtf(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); }

// tools/map.py:454-500 (knn with use_dir_vec=True, weighting='Shepard'): the terms one neighbour contributes.  The arithmetic is plain
// fp32 (the reference's is a chain of ~30 torch kernels over [N,K,3] temporaries whose reduction order is not specified — parity is to
// tolerance there, see the tests).  sums = {mean_dir[3], normal_test[3], weighted normals[3], weight sum}
__device__ __forceinline__ void neighbour_terms(const float* x, bool ok, float d2, int idx, const float* __restrict__ vertices,
                                                const float* __restrict__ vertex_normals, uint32_t n_vertices, float* sums) {
    // fewer than K vertices in the radius: frnn pads with -1, which torch's indexing wraps to the last vertex, sqrt(-1) = NaN (:458)
    const uint32_t j = ok ? (uint32_t)idx : n_vertices - 1;
    const float dis = ok ? sqrtf(d2) : NAN;
    float vn[3], dvo[3];
    for (int c = 0; c < 3; c++) { vn[c] = __ldg(vertex_normals + 3 * (size_t)j + c); dvo[c] = x[c] - __ldg(vertices + 3 * (size_t)j + c); }
    const float len = norm3(dvo) + 1e-5f;                 // :461
    const float w = 1.0f / (dis + 1e-7f);                 // :474 and :487 (Shepard): the same weight twice
    const float nl = norm3(vn) + 1e-5f;                   // :497
    for (int c = 0; c < 3; c++) {
        sums[c] += w * (dvo[c] / len);                    // :476
        sums[3 + c] += vn[c];                             // :477
        sums[6 + c] += (vn[c] / nl) * w;                  // :498 before the division by the weight sum
    }
    sums[9] += w;
}

__device__ __forceinline__ void finish_normal(float* sums, int k_want, float dir_vec_wdist, float* n) {
    float* mean_dir = sums;
    float* ntest = sums + 3;
    float* acc = sums + 6;
    float wsum = sums[9];
    for (int c = 0; c < 3; c++) ntest[c] /= (float)k_want;
    if (mean_dir[0] * ntest[0] + mean_dir[1] * ntest[1] + mean_dir[2] * ntest[2] < 0.0f)
        for (int c = 0; c < 3; c++) mean_dir[c] = -mean_dir[c];  // :478
    {
        const float len = norm3(mean_dir) + 1e-5f;                // :479
        for (int c = 0; c < 3; c++) mean_dir[c] /= len;
        const float w = 1.0f / (fmaxf(dir_vec_wdist, 1e-5f) + 1e-7f);   // :481-482, :487
        const float nl = norm3(mean_dir) + 1e-5f;                 // :497 (normalised a second time, as the reference does)
        for (int c = 0; c < 3; c++) acc[c] += (mean_dir[c] / nl) * w;
        wsum += w;
    }
    for (int c = 0; c < 3; c++) acc[c] /= wsum;                   // :496
    const float len = norm3(acc) + 1e-5f;                         // :499
    for (int c = 0; c < 3; c++) n[c] = acc[c] / len;
}

// What the projection needs of a mesh, as kernel arguments
struct MeshView {
    const float* __restrict__ vertices;
    const float* __restrict__ vertex_normals;
    uint32_t n_vertices;
    const Node* __restrict__ pt_nodes;
    const Point* __restrict__ pts;
    const Node* __restrict__ tri_nodes;
    const Tri* __restrict__ tris;
    float slack;
};
inline MeshView mesh_view(const MeshHandle* h, const float* vertex_normals) {
    return MeshView{h->vertices, vertex_normals, h->n_vertices, h->pt_nodes, h->pts, h->tri_nodes, h->tris, h->slack};
}

struct Projection {
    float p_sur[3];
    float sdf;
    float normal[3];
    int face;             // -1: neither cast hit anything within kMaxDist
};

// MeshProjector.project for one sample x: the neighbour list never leaves the registers, both casts run back to back
template <int K>
__device__ __forceinline__ Projection project_query(const float* x, int k_want, float r2, float dir_vec_wdist, const MeshView& m) {
    float bd[K];
    int bi[K];
    knn_one<K>(m.pt_nodes, m.pts, x, r2, k_want, bd, bi);
    float sums[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int s = 0; s < K; s++)
        if (s >= K - k_want) neighbour_terms(x, knn_slot_valid(bi[s]), bd[s], bi[s], m.vertices, m.vertex_normals, m.n_vertices, sums);
    float n[3], nn[3];
    finish_normal(sums, k_want, dir_vec_wdist, n);
    for (int c = 0; c < 3; c++) nn[c] = -n[c];
    const Hit h1 = trace_one(m.tri_nodes, m.tris, x, n, m.slack);       // :419 inner
    const Hit h2 = trace_one(m.tri_nodes, m.tris, x, nn, m.slack);      // :420 outer
    // :421-425
    Projection p;
    const bool cond = h1.t < h2.t;                                     // :421
    const float t = cond ? h1.t : h2.t;
    for (int c = 0; c < 3; c++) {
        p.p_sur[c] = NTX_ADD(x[c], NTX_MUL(t, cond ? n[c] : -n[c]));   // :422
        p.normal[c] = n[c];
    }
    p.sdf = cond ? -h1.t : h2.t;                                       // :423
    p.face = cond ? h1.face : h2.face;                                 // :425
    return p;
}

}  // namespace mesh
}  // namespace ntx
