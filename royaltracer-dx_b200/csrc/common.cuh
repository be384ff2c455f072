// common.cuh — shared declarations of the sm_100a engine (device structs, error handling).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/rtx_b200.h"

namespace rtx {

void set_error(const std::string& s);

#define RTX_CK(call)                                                                           \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            char b__[512];                                                                     \
            snprintf(b__, sizeof b__, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            rtx::set_error(b__);                                                               \
            return RTX_ERR_CUDA;                                                               \
        }                                                                                      \
    } while (0)

// shaders/Common_v7.hlsl:1-3, Miss_v7.hlsl:7
#define RTX_PI_REF 3.1415f
#define RTX_S_BIAS 0.00002f
#define RTX_EPS 0.000001f
#define RTX_MISS_ID 4294967294u

// ---- acceleration structure (DESIGN.md §"Data layout in HBM") ------------------------------------
// 80-B compressed 8-wide node, stored as 5 x uint4:
//   n0 = (px, py, pz, ex | ey<<8 | ez<<16 | imask<<24)
//   n1 = (child_base, prim_base, WI = imask << 24 | W, 0)
//   n2 = (qlo_x[0..3], qlo_x[4..7], qlo_y[0..3], qlo_y[4..7])
//   n3 = (qlo_z[0..3], qlo_z[4..7], qhi_x[0..3], qhi_x[4..7])
//   n4 = (qhi_y[0..3], qhi_y[4..7], qhi_z[0..3], qhi_z[4..7])
// W: leaf child in slot s holds c (1..3) primitives <=> bits 3s .. 3s+c-1 set; the node's primitives are stored densely from prim_base in
// bit order, so the primitive behind bit b is prim_base + popc(W & ((1 << b) - 1)).  imask bit s <=> slot s is an inner child; the inner
// children are stored densely from child_base in slot order.  An empty slot has neither.
// 48-B triangle = 3 x float4: (v0.xyz, bits(prim)), (v1.xyz, 0), (v2.xyz, 0).
// 64-B instance record = 4 x float4: rows 0..2 of world->object (from objectToWorldInverse), (blas, instance, 0, 0).
struct alignas(16) BlasRef {
    const uint4* nodes;
    const float4* tris;
    float lo[3], hi[3];   // padded object-space bounds of the model: an instance whose object-space ray misses them is not entered
    float pad_[2];
};

struct SceneAS {
    const uint4* tlas_nodes;
    const float4* inst_recs;
    const BlasRef* blas;
    uint32_t n_instances;
    uint32_t one_bits;    // 0x3F800000, passed as a run-time value: keeps it in a register so that the byte->float PRMT of the node test takes its
                          // selector as an immediate (with the constant folded in, ptxas re-materialised a selector register per PRMT: 43 extra
                          // IMAD.U32 per node test)
    unsigned int* overflow;   // per-context word raised when a traversal stack overflows (checked and cleared by the API, api.cu check_overflow)
    int num_sms;          // of the context's device: sizes the persistent traversal grid (trace.cu launch_trace)
};

// Ray queue entry layout (SoA): o_tmin[j] = (o.xyz, tmin), d_tmax[j] = (d.xyz, tmax).
// Hit record (20 B/ray): hit_a[j] = (t, b1, b2, bits(prim)); hit_inst[j] = instance (0xFFFFFFFF = miss).

struct TraceStats {
    unsigned long long nodes, tris, insts;
    unsigned long long replays;     // shading stages: paths replayed with IEEE operations (wavefront.cu)
};

}  // namespace rtx
