// trace.h — host-side entry points of the traversal kernels and the GPU BVH builder.
#pragma once
#include "common.cuh"

namespace rtx {

// Drains a ray queue (see common.cuh for the queue layout).  n is read from *n_ptr on the device when n_ptr is
// non-null (wavefront queues), else n_fixed.  `cursor` = two device words owned by this launch, zero on entry and left zero (the kernel's
// last CTA resets them: no memset per launch).  grid_share = number of traversal
// launches expected to run concurrently (each gets 1/grid_share of the machine's resident CTAs).  order / n_heavy_ptr / cap: the queue's
// trace order (wavefront.h RayQueue): slot indices, *n_heavy_ptr expensive rays from entry 0 upwards, the others from entry cap-1 downwards.
// vis_pid / vis (any-hit only): instead of writing hit_inst, an occluded ray j stores 0 to vis[vis_pid[j]] (the wavefront's per-path visibility).
// vis_pid / vmask (any-hit only): an occluded ray j sets bit (vis_pid[j] & 15) of vmask[vis_pid[j] >> 4] (the occlusion masks of the ReSTIR reuse passes).
cudaError_t launch_trace(const SceneAS& S, const float4* o_tmin, const float4* d_tmax, const uint32_t* n_ptr, uint32_t n_fixed,
                         unsigned int* cursor, float4* hit_a, uint32_t* hit_inst, bool any_hit, TraceStats* stats,
                         cudaStream_t stream, int grid_share = 1, const uint32_t* order = nullptr, const uint32_t* n_heavy_ptr = nullptr,
                         uint32_t cap = 0, const uint32_t* vis_pid = nullptr, float* vis = nullptr, uint32_t* vmask = nullptr);

struct Bvh8 {
    uint4* nodes = nullptr;     // 5 x uint4 per node
    float4* prims = nullptr;    // PRIM_F4 x float4 per primitive, in leaf order
    uint32_t n_nodes = 0, n_prims = 0;
    float lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};   // padded bounds of everything inside
    float build_ms = 0.0f;
    float sah_cost = 0.0f;      // SAH cost of the wide tree relative to the root area (c_node = 1, c_prim = 0.3)
    // nodes are emitted level by level (children always behind their parent): level k = [level_start[k], level_start[k + 1])
    uint32_t level_start[48] = {0}; uint32_t n_levels = 0;
};

// BLAS over an indexed triangle list (vertex stride 28 B, position first).  Returns device allocations owned by the caller.
cudaError_t build_blas(const uint8_t* d_vertices, uint32_t n_vertices, const uint32_t* d_indices, uint32_t n_tris,
                       Bvh8* out, cudaStream_t stream);
// TLAS over instance records (4 x float4 each, already in device memory) with world-space boxes lo/hi (float4 each).
cudaError_t build_tlas(const float4* d_inst_recs, const float4* d_box_lo, const float4* d_box_hi, uint32_t n_instances,
                       Bvh8* out, cudaStream_t stream);
void free_bvh(Bvh8* b);
// Per-frame TLAS update when the whole TLAS is one node (n_instances <= the leaf size): rewrites out->nodes / out->prims in place,
// stream-ordered, no allocation, no host synchronisation.  d_ctr = 256 B of device scratch.
// Per-frame TLAS REFIT (rdn/Renderer.cpp:594, TopLevelASGenerator update path): keeps the topology of the last build, copies the new instance
// records into leaf order and recomputes every node's origin, exponents and quantised child boxes bottom-up, one launch per level.
// Stream-ordered, no allocation, no host synchronisation.  Valid while the instance count is the one the TLAS was built for.
cudaError_t refit_tlas(const float4* d_inst_recs, const float4* d_box_lo, const float4* d_box_hi, uint32_t n_instances, Bvh8* inout,
                       cudaStream_t stream);
bool tlas_fits_one_node(uint32_t n_instances);
cudaError_t update_tlas_one_node(const float4* d_inst_recs, const float4* d_box_lo, const float4* d_box_hi, uint32_t n_instances, Bvh8* out,
                                 void* d_ctr, cudaStream_t stream);

// Fills instance records + world boxes from descs/props (device arrays) and per-model BLAS bounds.
struct BlasBounds { float lo[3]; float hi[3]; const uint8_t* verts; uint32_t n_verts; };   // verts: the model's 28-B vertex buffer
cudaError_t launch_instance_records(const rtx_instance_desc* d_descs, const rtx_instance_props* d_props, const BlasBounds* d_bounds,
                                    uint32_t n, float4* d_recs, float4* d_lo, float4* d_hi, unsigned int* d_scratch6 /* 6 words per instance */,
                                    cudaStream_t stream);

// BLAS REFIT over new vertex positions (DXR PERFORM_UPDATE; same vertex count and index buffer as the build): keeps the topology, child
// order and leaf order of the build, rewrites the triangle records from the vertices and recomputes every node bottom-up, one launch per
// level, with the builder's padding (2^-15 of the NEW bounds) and outward quantisation.  The padded model bounds go to inout's table
// entries d_ref / d_bounds (when non-null) and to d_out6 (6 floats, device).  inout->lo / hi are NOT updated (the host copy is the
// caller's: it copies d_out6 back).  Stream-ordered, no allocation, no host synchronisation.  d_scratch = 256 B of device scratch.
cudaError_t refit_blas(const uint8_t* d_vertices, const uint32_t* d_indices, uint32_t n_tris, Bvh8* inout, void* d_scratch, BlasRef* d_ref,
                       BlasBounds* d_bounds, float* d_out6, cudaStream_t stream);

}  // namespace rtx
