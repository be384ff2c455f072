// wave_dev.cuh — device helpers shared by the wavefront stages (wavefront.cu) and the ReSTIR reuse passes (restir.cu).
#pragma once
#include "wavefront.h"

namespace rtx {

struct StateView {
    float4* base; uint32_t n;
    uint2* seed;          // the path's RNG state in its own 8-byte plane: every stage updates it, and as the .w of two float4 planes it cost a
                          // 32-byte read and a 32-byte write per path and stage to move 8 bytes (E0 stages only; nullptr elsewhere)
    __device__ __forceinline__ float4& at(int plane, uint32_t pid) const { return base[(size_t)plane * n + pid]; }
    // The path state is STREAMED: each stage reads a plane once and the next reader is a launch later, ~0.5 GB per k_gi_step launch.
    // ld / stt use the evict-first cache policy (ld.global.cs / st.global.cs) so that this traffic does not push the BVH, which every
    // traversal launch re-reads at random, out of the L2: closest-hit launches -2.7 %, C2 pass -1.3 % (profiles/r02_l2_policy_ab.txt).
    __device__ __forceinline__ float4 ld(int plane, uint32_t pid) const { return __ldcs(&at(plane, pid)); }
    __device__ __forceinline__ void stt(int plane, uint32_t pid, float4 v) const { __stcs(&at(plane, pid), v); }
    __device__ __forceinline__ uint2 ld_seed(uint32_t pid) const { return __ldcs(&seed[pid]); }
    __device__ __forceinline__ void st_seed(uint32_t pid, uint2 v) const { __stcs(&seed[pid], v); }
};

// queue entries and hit records a shading stage consumes (read once)
template <typename T> __device__ __forceinline__ T ld_stream(const T* p) { return __ldcs(p); }

// Which paths a part (path range) of a pass owns: the contiguous range [p0, p0 + np), or — chunk != 0 — every parts-th chunk of `chunk`
// consecutive paths (a few image rows), so that concurrent parts see the same mix of the image and finish together.  k = index in the part.
struct PartMap {
    uint32_t p0, chunk, parts, h;
    __device__ __forceinline__ uint32_t path(uint32_t k) const { return chunk ? ((k / chunk) * parts + h) * chunk + (k % chunk) : p0 + k; }
};

__device__ __forceinline__ f3 xyz(float4 v) { return mk3(v.x, v.y, v.z); }
__device__ __forceinline__ float4 f4(f3 v, float w) { return make_float4(v.x, v.y, v.z, w); }
__device__ __forceinline__ float4 f4u(f3 v, uint32_t w) { return make_float4(v.x, v.y, v.z, __uint_as_float(w)); }

// Warp-level queue compaction: one atomicAdd per warp claims a contiguous run of slots.  Must be reached by all 32 lanes.
__device__ __forceinline__ void push_ray(const RayQueue& q, bool emit, f3 o, float tmin, f3 d, float tmax, uint32_t pid) {
    const unsigned mask = __ballot_sync(0xffffffffu, emit);
    if (mask == 0u) return;
    const unsigned lane = threadIdx.x & 31u;
    const int leader = __ffs(mask) - 1;
    unsigned base = 0;
    if ((int)lane == leader) base = atomicAdd(q.count, (unsigned)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (emit) {
        const unsigned slot = base + __popc(mask & ((1u << lane) - 1u));
        q.o_tmin[slot] = f4(o, tmin);
        q.d_tmax[slot] = f4(d, tmax);
        q.pid[slot] = pid;
    }
}

// Cost class of a ray: does its segment cross the bounds of the scene's large instances?  Only the ORDER of a queue depends on it (every
// path draws its own random numbers, results do not depend on queue order), so the slab test may be approximate.
__device__ __forceinline__ bool ray_is_heavy(const SceneData& S, f3 o, float tmin, f3 d, float tmax) {
    if (!S.heavy_valid) return true;
    float ix, iy, iz;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ix) : "f"(d.x));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iy) : "f"(d.y));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iz) : "f"(d.z));
    const float ax = (S.heavy_lo[0] - o.x) * ix, bx = (S.heavy_hi[0] - o.x) * ix;
    const float ay = (S.heavy_lo[1] - o.y) * iy, by = (S.heavy_hi[1] - o.y) * iy;
    const float az = (S.heavy_lo[2] - o.z) * iz, bz = (S.heavy_hi[2] - o.z) * iz;
    const float tn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), tmin));
    const float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), tmax));
    return !(tn > tf);            // NaN (a direction component of 0 inside the slab) counts as heavy
}

// Trace order of a queue (wavefront.h RayQueue): heavy rays are recorded from entry 0 upwards, the others from entry cap-1 downwards.
// A warp claims its queue slots and its order entries with ONE round of atomics: lane k performs the k-th of {count, n_heavy, n_light}
// of the first queue and, in push_ray_pair, of the second (six dependent round trips to the L2 per warp before; ncu showed 7 % of
// k_gi_step's stall samples on them at 3 of 32 lanes).  Both must be reached by all 32 lanes.
__device__ __forceinline__ void store_ray(const RayQueue& q, unsigned slot, f3 o, float tmin, f3 d, float tmax, uint32_t pid) {
    q.o_tmin[slot] = f4(o, tmin);
    q.d_tmax[slot] = f4(d, tmax);
    q.pid[slot] = pid;
}

// order entries only, for rays whose slots are already fixed (k_generate: slot = index within the part)
__device__ __forceinline__ void record_order(const RayQueue& q, unsigned mask, bool emit, bool heavy, unsigned slot) {
    const unsigned full = 0xffffffffu, lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
    const unsigned mh = __ballot_sync(full, emit && heavy), ml = mask & ~mh;
    const unsigned v = lane == 0u ? __popc(mh) : (lane == 1u ? __popc(ml) : 0u);
    unsigned r = 0;
    if (v) r = atomicAdd(lane == 0u ? q.n_heavy : q.n_light, v);
    const unsigned bh = __shfl_sync(full, r, 0), bl = __shfl_sync(full, r, 1);
    if (emit) q.order[heavy ? bh + __popc(mh & below) : q.cap - 1u - (bl + __popc(ml & below))] = slot;
}

__device__ __forceinline__ void push_ray2(const RayQueue& q, bool emit, bool heavy, f3 o, float tmin, f3 d, float tmax, uint32_t pid) {
    const unsigned full = 0xffffffffu, lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
    const unsigned mask = __ballot_sync(full, emit);
    if (mask == 0u) return;
    const bool ord = q.order != nullptr;
    const unsigned mh = __ballot_sync(full, emit && heavy), ml = mask & ~mh;
    unsigned* p = lane == 0u ? q.count : (lane == 1u ? q.n_heavy : q.n_light);
    const unsigned v = lane == 0u ? __popc(mask) : (!ord || lane > 2u ? 0u : (lane == 1u ? __popc(mh) : __popc(ml)));
    unsigned r = 0;
    if (v) r = atomicAdd(p, v);
    const unsigned slot = __shfl_sync(full, r, 0) + __popc(mask & below);
    const unsigned bh = __shfl_sync(full, r, 1), bl = __shfl_sync(full, r, 2);
    if (emit) {
        store_ray(q, slot, o, tmin, d, tmax, pid);
        if (ord) q.order[heavy ? bh + __popc(mh & below) : q.cap - 1u - (bl + __popc(ml & below))] = slot;
    }
}

__device__ __forceinline__ void push_ray_pair(const RayQueue& qa, bool ea, bool ha, f3 oa, float tmina, f3 da, float tmaxa,
                                              const RayQueue& qb, bool eb, bool hb, f3 ob, float tminb, f3 db, float tmaxb, uint32_t pid) {
    const unsigned full = 0xffffffffu, lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
    const unsigned ma = __ballot_sync(full, ea), mb = __ballot_sync(full, eb);
    if ((ma | mb) == 0u) return;
    const bool orda = qa.order != nullptr, ordb = qb.order != nullptr;
    const unsigned mha = __ballot_sync(full, ea && ha), mla = ma & ~mha, mhb = __ballot_sync(full, eb && hb), mlb = mb & ~mhb;
    unsigned* p = qa.count; unsigned v = 0;
    switch (lane) {
        case 0: v = __popc(ma); break;
        case 1: p = qa.n_heavy; v = orda ? __popc(mha) : 0u; break;
        case 2: p = qa.n_light; v = orda ? __popc(mla) : 0u; break;
        case 3: p = qb.count; v = __popc(mb); break;
        case 4: p = qb.n_heavy; v = ordb ? __popc(mhb) : 0u; break;
        case 5: p = qb.n_light; v = ordb ? __popc(mlb) : 0u; break;
        default: break;
    }
    unsigned r = 0;
    if (v) r = atomicAdd(p, v);
    const unsigned sa = __shfl_sync(full, r, 0) + __popc(ma & below), bha = __shfl_sync(full, r, 1), bla = __shfl_sync(full, r, 2);
    const unsigned sb = __shfl_sync(full, r, 3) + __popc(mb & below), bhb = __shfl_sync(full, r, 4), blb = __shfl_sync(full, r, 5);
    if (ea) {
        store_ray(qa, sa, oa, tmina, da, tmaxa, pid);
        if (orda) qa.order[ha ? bha + __popc(mha & below) : qa.cap - 1u - (bla + __popc(mla & below))] = sa;
    }
    if (eb) {
        store_ray(qb, sb, ob, tminb, db, tmaxb, pid);
        if (ordb) qb.order[hb ? bhb + __popc(mhb & below) : qb.cap - 1u - (blb + __popc(mlb & below))] = sb;
    }
}

}  // namespace rtx
