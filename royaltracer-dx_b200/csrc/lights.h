// lights.h — the emissive-triangle list (binding t6) built on the device from the scene as it is now: CollectEmissiveTriangles +
// CreateEmissiveTrianglesBuffer (rdn/Renderer.cpp:2123-2243), record for record the bytes of the host mirror collect_emissive
// (host/Renderer.cpp) over the same vertices.
#pragma once
#include <vector>

#include "shade.cuh"

namespace rtx {

struct LightBuffers {
    // the emissive index: which triangles of each model are emitters (three equal face-vertex ids of a material with Ke0+Ke1+Ke2 > 0);
    // model m's ones in index order from tris[base[m]], base[m] = the triangles of the models before m
    uint32_t* tris = nullptr; size_t cap_tris = 0;
    uint8_t* flags = nullptr; size_t cap_flags = 0;
    uint32_t* d_base = nullptr; uint32_t* d_count = nullptr; size_t cap_models = 0;
    void* select_tmp = nullptr; size_t cap_select_tmp = 0;
    std::vector<uint32_t> count;            // host copy of d_count
    // per collect, grow-only
    unsigned long long* keys = nullptr; unsigned long long* keys_sorted = nullptr; float* cdf = nullptr; size_t cap_records = 0;
    uint32_t* inst_base = nullptr; size_t cap_inst = 0;
    void* sort_tmp = nullptr; size_t cap_sort_tmp = 0;
    float* d_total = nullptr;
};

// Rebuilds the emissive index of `models` (host copies of the per-model records, S.models is not read) from S's material ids and
// materials.  Synchronises the stream (L.count is read back); may allocate.
cudaError_t lights_build_index(LightBuffers& L, const std::vector<ModelRef>& models, const SceneData& S, cudaStream_t stream,
                               uint64_t* launches);
// Writes the n records (n = the sum of L.count over the models of the n_instances instances S.inst_model names, n > 0) to out, on the
// stream.  Allocates only when n or n_instances exceed every earlier call's; otherwise neither allocates nor synchronises.
cudaError_t lights_collect(LightBuffers& L, const SceneData& S, uint32_t n_instances, uint32_t n, rtx_light_triangle* out,
                           cudaStream_t stream, uint64_t* launches);
void lights_free(LightBuffers& L);

}  // namespace rtx
