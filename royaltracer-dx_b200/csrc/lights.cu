// lights.cu — the emissive-triangle list on the device (rtx_collect_emissive_triangles).  Bit-identical to the host mirror
// collect_emissive (host/Renderer.cpp, built with -ffp-contract=off; this file with -fmad=false and explicit _rn operations):
//   1. k_light_inst_base   per instance, the index of its first record (exclusive sum of its model's emissive count)
//   2. k_light_keys        per record in collection order (instance, then triangle index order): its weight (triangle_weight's operations)
//                          and the key (~bits(weight)) << 32 | collection index.  weight is in [+0, +inf] (0.5 * sqrt of a sum of squares
//                          times a positive mean), so ascending keys = descending weights with ties in collection order: std::stable_sort
//   3. radix sort of the keys (cub, plumbing)
//   4. k_light_sums        the two sequential float sums of the host (total, then the running sum of weight / total) as one dependent
//                          chain each on one thread, fed from shared memory by the block's other warps
//   5. k_light_write       the 80-byte records in sorted order
#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "lights.h"

namespace rtx {

// material id of face-vertex slot s and that material's Ke, with the shading kernels' out-of-range rule (ClosestHit, fetch_material_head)
__device__ __forceinline__ uint32_t light_material_id(const SceneData& S, uint32_t s) {
    return s < S.n_material_ids ? S.material_ids[s] : 0u;
}
__device__ __forceinline__ float3 light_ke(const SceneData& S, uint32_t id) {
    if (id >= S.n_materials) return make_float3(0.0f, 0.0f, 0.0f);
    const float* ke = S.materials[id].Ke;
    return make_float3(ke[0], ke[1], ke[2]);
}

__global__ void k_light_flags(SceneData S, uint32_t mat_offset, uint32_t n_tris, uint8_t* __restrict__ flags) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tris) return;
    const uint32_t s = mat_offset + 3u * t;
    const uint32_t m0 = light_material_id(S, s), m1 = light_material_id(S, s + 1u), m2 = light_material_id(S, s + 2u);
    const float3 ke = light_ke(S, m0);
    flags[t] = m0 == m1 && m0 == m2 && __fadd_rn(__fadd_rn(ke.x, ke.y), ke.z) > 0.0f;
}

__global__ void __launch_bounds__(1024) k_light_inst_base(const uint32_t* __restrict__ inst_model, uint32_t n_inst,
                                                          const uint32_t* __restrict__ count, uint32_t* __restrict__ base) {
    typedef cub::BlockScan<uint32_t, 1024> Scan;
    __shared__ typename Scan::TempStorage tmp;
    uint32_t run = 0;
    for (uint32_t b = 0; b < n_inst; b += 1024) {
        const uint32_t i = b + threadIdx.x;
        const uint32_t v = i < n_inst ? count[inst_model[i]] : 0u;
        uint32_t ex, agg;
        Scan(tmp).ExclusiveSum(v, ex, agg);
        if (i < n_inst) base[i] = run + ex;
        run += agg;
        __syncthreads();
    }
}

struct LightTri { float p[3][3]; float3 ke; uint32_t inst; };

// record j of the collection order: the instance whose records hold j (the last i with inst_base[i] <= j), its model's emissive triangle
__device__ __forceinline__ LightTri light_tri(const SceneData& S, const uint32_t* __restrict__ inst_base, uint32_t n_inst,
                                              const uint32_t* __restrict__ tris, const uint32_t* __restrict__ tri_base, uint32_t j) {
    uint32_t lo = 0, hi = n_inst;
    while (hi - lo > 1u) {
        const uint32_t mid = (lo + hi) >> 1;
        if (inst_base[mid] <= j) lo = mid; else hi = mid;
    }
    LightTri r;
    r.inst = lo;
    const uint32_t m = S.inst_model[lo];
    const ModelRef M = S.models[m];
    const uint32_t t = tris[tri_base[m] + (j - inst_base[lo])];
#pragma unroll
    for (int v = 0; v < 3; v++) {
        const float* q = reinterpret_cast<const float*>(M.verts + (size_t)M.idx[3u * t + v] * 28u);
        r.p[v][0] = q[0]; r.p[v][1] = q[1]; r.p[v][2] = q[2];
    }
    r.ke = light_ke(S, light_material_id(S, M.mat_offset + 3u * t));
    return r;
}

// triangle_weight (host/Renderer.cpp; rdn/Renderer.cpp:2217-2233) operation for operation
__device__ __forceinline__ float light_weight(const LightTri& r) {
    float e1[3], e2[3];
#pragma unroll
    for (int k = 0; k < 3; k++) { e1[k] = __fsub_rn(r.p[1][k], r.p[0][k]); e2[k] = __fsub_rn(r.p[2][k], r.p[0][k]); }
    const float c0 = __fsub_rn(__fmul_rn(e1[1], e2[2]), __fmul_rn(e1[2], e2[1]));
    const float c1 = __fsub_rn(__fmul_rn(e1[2], e2[0]), __fmul_rn(e1[0], e2[2]));
    const float c2 = __fsub_rn(__fmul_rn(e1[0], e2[1]), __fmul_rn(e1[1], e2[0]));
    const float d = __fadd_rn(__fadd_rn(__fmul_rn(c0, c0), __fmul_rn(c1, c1)), __fmul_rn(c2, c2));
    const float area = __fmul_rn(0.5f, __fsqrt_rn(d));
    return __fmul_rn(area, __fdiv_rn(__fadd_rn(__fadd_rn(r.ke.x, r.ke.y), r.ke.z), 3.0f));
}

__device__ __forceinline__ float key_weight(unsigned long long key) { return __uint_as_float(~(uint32_t)(key >> 32)); }

__global__ void k_light_keys(SceneData S, const uint32_t* __restrict__ inst_base, uint32_t n_inst, const uint32_t* __restrict__ tris,
                             const uint32_t* __restrict__ tri_base, uint32_t n, unsigned long long* __restrict__ keys) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const float w = light_weight(light_tri(S, inst_base, n_inst, tris, tri_base, j));
    keys[j] = ((unsigned long long)(~__float_as_uint(w)) << 32) | j;
}

// The host's two sums over the sorted weights, `total += w` and then `cum += w / total`, are sequential binary32 additions: thread 0
// runs each as one dependent chain over a shared-memory chunk while warps 1.. stage the next chunk (and, for the second chain, divide
// and write back the previous chunk's running sums).  Chunks are padded with +0, which leaves both sums unchanged (neither is ever -0).
static constexpr int SUM_THREADS = 256, SUM_CHUNK = 2048, SUM_LOADERS = SUM_THREADS - 32;

__device__ __forceinline__ float chain(float* b, float acc, bool keep_running_sums) {
    float4* b4 = reinterpret_cast<float4*>(b);
#pragma unroll 8
    for (int k = 0; k < SUM_CHUNK / 4; k++) {
        const float4 v = b4[k];
        float4 r;
        acc = __fadd_rn(acc, v.x); r.x = acc;
        acc = __fadd_rn(acc, v.y); r.y = acc;
        acc = __fadd_rn(acc, v.z); r.z = acc;
        acc = __fadd_rn(acc, v.w); r.w = acc;
        if (keep_running_sums) b4[k] = r;
    }
    return acc;
}

__global__ void __launch_bounds__(SUM_THREADS) k_light_sums(const unsigned long long* __restrict__ keys, uint32_t n, float* __restrict__ cdf,
                                                            float* __restrict__ d_total) {
    __shared__ __align__(16) float buf[2][SUM_CHUNK];
    __shared__ float s_total;
    const uint32_t nc = (n + SUM_CHUNK - 1) / SUM_CHUNK;
    const int lt = (int)threadIdx.x - 32;       // >= 0: a staging thread
    auto stage = [&](uint32_t c, bool divide, float total) {
        for (int k = lt; k < SUM_CHUNK; k += SUM_LOADERS) {
            const uint32_t j = c * SUM_CHUNK + k;
            float w = 0.0f;
            if (j < n) { w = key_weight(keys[j]); if (divide) w = __fdiv_rn(w, total); }
            buf[c & 1][k] = w;
        }
    };
    auto store = [&](uint32_t c) {
        for (int k = lt; k < SUM_CHUNK; k += SUM_LOADERS) {
            const uint32_t j = c * SUM_CHUNK + k;
            if (j < n) cdf[j] = buf[c & 1][k];
        }
    };
    float acc = 0.0f;
    if (lt >= 0) stage(0, false, 0.0f);
    __syncthreads();
    for (uint32_t c = 0; c < nc; c++) {
        if (threadIdx.x == 0) acc = chain(buf[c & 1], acc, false);
        else if (lt >= 0 && c + 1 < nc) stage(c + 1, false, 0.0f);
        __syncthreads();
    }
    if (threadIdx.x == 0) { s_total = acc; *d_total = acc; }
    __syncthreads();
    const float total = s_total;
    acc = 0.0f;
    if (lt >= 0) stage(0, true, total);
    __syncthreads();
    for (uint32_t c = 0; c < nc; c++) {
        if (threadIdx.x == 0) acc = chain(buf[c & 1], acc, true);
        else if (lt >= 0) {
            if (c > 0) store(c - 1);
            if (c + 1 < nc) stage(c + 1, true, total);      // (the buffer just stored)
        }
        __syncthreads();
    }
    if (lt >= 0 && nc) store(nc - 1);
}

__global__ void k_light_write(SceneData S, const uint32_t* __restrict__ inst_base, uint32_t n_inst, const uint32_t* __restrict__ tris,
                              const uint32_t* __restrict__ tri_base, uint32_t n, const unsigned long long* __restrict__ keys,
                              const float* __restrict__ cdf, const float* __restrict__ d_total, rtx_light_triangle* __restrict__ out) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const unsigned long long key = keys[j];
    const LightTri r = light_tri(S, inst_base, n_inst, tris, tri_base, (uint32_t)key);
    const float total = *d_total;
    const float c = j + 1 == n ? 1.0f : cdf[j];         // CollectEmissiveTriangles forces the last entry to 1
    float4* o = reinterpret_cast<float4*>(out + j);
    o[0] = make_float4(r.p[0][0], r.p[0][1], r.p[0][2], c);
    o[1] = make_float4(r.p[1][0], r.p[1][1], r.p[1][2], __uint_as_float(r.inst));
    o[2] = make_float4(r.p[2][0], r.p[2][1], r.p[2][2], __fdiv_rn(key_weight(key), total));
    o[3] = make_float4(r.ke.x, r.ke.y, r.ke.z, __uint_as_float(n));
    o[4] = make_float4(total, 0.0f, 0.0f, 0.0f);
}

// device buffers of at least n elements each, grown together (grow-only); buffers that grow are freed behind everything queued on the stream
template <int K>
static cudaError_t grow(void* const (&p)[K], const size_t (&elem)[K], size_t* cap, size_t n, cudaStream_t stream) {
    bool have = true;
    for (int i = 0; i < K; i++) have = have && *(void**)p[i];
    if (have && *cap >= n) return cudaSuccess;
    if (*cap) {
        const cudaError_t e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) return e;
    }
    *cap = 0;
    const size_t k = n ? n : 1;
    for (int i = 0; i < K; i++) {
        void** q = (void**)p[i];
        if (*q) { cudaFree(*q); *q = nullptr; }
        const cudaError_t e = cudaMalloc(q, k * elem[i]);
        if (e != cudaSuccess) return e;
    }
    *cap = k;
    return cudaSuccess;
}
#define LCK(x) do { const cudaError_t e__ = (x); if (e__ != cudaSuccess) return e__; } while (0)

cudaError_t lights_build_index(LightBuffers& L, const std::vector<ModelRef>& models, const SceneData& S, cudaStream_t stream,
                               uint64_t* launches) {
    const size_t nm = models.size();
    std::vector<uint32_t> base(nm ? nm : 1, 0u);
    size_t total = 0, max_tris = 0;
    for (size_t m = 0; m < nm; m++) { base[m] = (uint32_t)total; total += models[m].n_tris; max_tris = std::max(max_tris, (size_t)models[m].n_tris); }
    LCK(grow<1>({&L.tris}, {4}, &L.cap_tris, total, stream));
    LCK(grow<1>({&L.flags}, {1}, &L.cap_flags, max_tris, stream));
    LCK(grow<2>({&L.d_base, &L.d_count}, {4, 4}, &L.cap_models, nm, stream));
    thrust::counting_iterator<uint32_t> ids(0);
    size_t tmp_bytes = 0;
    LCK(cub::DeviceSelect::Flagged(nullptr, tmp_bytes, ids, L.flags, L.tris, L.d_count, (int)max_tris, stream));
    LCK(grow<1>({&L.select_tmp}, {1}, &L.cap_select_tmp, tmp_bytes, stream));
    LCK(cudaMemsetAsync(L.d_count, 0, L.cap_models * sizeof(uint32_t), stream));
    LCK(cudaMemcpyAsync(L.d_base, base.data(), base.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    for (size_t m = 0; m < nm; m++) {
        const uint32_t nt = models[m].n_tris;
        if (!nt) continue;
        k_light_flags<<<(nt + 255) / 256, 256, 0, stream>>>(S, models[m].mat_offset, nt, L.flags);
        LCK(cudaGetLastError());
        size_t bytes = L.cap_select_tmp;
        LCK(cub::DeviceSelect::Flagged(L.select_tmp, bytes, ids, L.flags, L.tris + base[m], L.d_count + m, (int)nt, stream));
        *launches += 2;
    }
    L.count.assign(nm, 0u);
    if (nm) LCK(cudaMemcpyAsync(L.count.data(), L.d_count, nm * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    return cudaStreamSynchronize(stream);       // (also keeps `base` alive until its copy has been made)
}

cudaError_t lights_collect(LightBuffers& L, const SceneData& S, uint32_t n_inst, uint32_t n, rtx_light_triangle* out, cudaStream_t stream,
                           uint64_t* launches) {
    LCK(grow<3>({&L.keys, &L.keys_sorted, &L.cdf}, {8, 8, 4}, &L.cap_records, n, stream));
    LCK(grow<1>({&L.inst_base}, {4}, &L.cap_inst, n_inst, stream));
    if (!L.d_total) LCK(cudaMalloc((void**)&L.d_total, sizeof(float)));
    size_t sort_bytes = 0;
    LCK(cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, L.keys, L.keys_sorted, (int)n, 0, 64, stream));
    LCK(grow<1>({&L.sort_tmp}, {1}, &L.cap_sort_tmp, sort_bytes, stream));
    sort_bytes = L.cap_sort_tmp;
    k_light_inst_base<<<1, 1024, 0, stream>>>(S.inst_model, n_inst, L.d_count, L.inst_base);
    k_light_keys<<<(n + 255) / 256, 256, 0, stream>>>(S, L.inst_base, n_inst, L.tris, L.d_base, n, L.keys);
    LCK(cudaGetLastError());
    LCK(cub::DeviceRadixSort::SortKeys(L.sort_tmp, sort_bytes, L.keys, L.keys_sorted, (int)n, 0, 64, stream));
    k_light_sums<<<1, SUM_THREADS, 0, stream>>>(L.keys_sorted, n, L.cdf, L.d_total);
    k_light_write<<<(n + 255) / 256, 256, 0, stream>>>(S, L.inst_base, n_inst, L.tris, L.d_base, n, L.keys_sorted, L.cdf, L.d_total, out);
    *launches += 5;
    return cudaGetLastError();
}

void lights_free(LightBuffers& L) {
    void* p[] = {L.tris, L.flags, L.d_base, L.d_count, L.select_tmp, L.keys, L.keys_sorted, L.cdf, L.inst_base, L.sort_tmp, L.d_total};
    for (void* q : p) if (q) cudaFree(q);
    L = LightBuffers();
}

}  // namespace rtx
