// traverse.cuh — closest-hit / any-hit traversal of the two-level compressed 8-wide BVH.
//
// Replaces the fixed-function TraceRay of the reference (no source exists: D3D12 driver + RT cores;
// call sites shaders/Pass_init_di_v7.hlsl:91-99, Sampler_v7.hlsl:86-104,223-229,428-434,
// Path_Sampler_v7.hlsl:45-52,271-283).  Contract (SURVEY.md §8a T3/T4):
//   * opaque triangles, no culling (two-sided), instance mask 0xFF;
//   * a triangle is hit iff TMin < t < TMax (strict), t measured along the un-renormalised object-space
//     direction so it equals the world-space parameter;
//   * closest hit = lexicographic minimum of (t, instance, primitive) — traversal-order independent;
//   * any-hit returns as soon as one triangle is hit.
// The ray/triangle test is the watertight edge-function test; its operation order is part of the contract
// (hit IDs are compared bit-exactly against the CPU oracle).  Box tests only have to be conservative.
//
// Instruction-level notes (ncu, profiles/r01_trace_hotspots_*.txt): the kernel is issue-bound, so the inner loops
// are written for instruction count and for the fma/alu pipe split of sm_100 —
//   * quantised plane bytes become floats with ONE byte-permute each (1 + q*2^-15 in the mantissa), the small extra
//     rounding this costs is covered by widening the slab interval by 2^-23 |A|;
//   * the Woop axis permutation uses predicated selects from a one-hot mask (no branches, no register copies);
//   * leaving a BLAS is detected by the stack depth (no sentinel entry, no pop loop).
#pragma once
#include "common.cuh"

namespace rtx {

#define RTX_STACK_SIZE 40
// A full stack drops the entry (no memory fault) and raises the context's overflow word (SceneAS::overflow): every API call that hands
// results to the caller checks it, fails with RTX_ERR_STATE and clears it (api.cu check_overflow).  rtx_set_instances also rejects a
// TLAS + BLAS pair whose level counts could exceed the stack before anything is traced.
#define RTX_PUSH(v)                                                   \
    do {                                                              \
        if (sp < RTX_STACK_SIZE) stack[sp++] = (v);                   \
        else *S.overflow = 1u;                                        \
    } while (0)

// byte I of x as the float 1 + q*2^-15 (0x3F80qq00: one byte permute with `one` = 0x3F800000); intersect_node() scales it back
template <int I>
__device__ __forceinline__ float plane_byte(uint32_t x, uint32_t one) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(x), "r"(one), "n"(0x7604 | (I << 4)));
    return __uint_as_float(d);
}

struct RaySpace {          // the ray in the space currently traversed + derived constants
    float ox, oy, oz;
    float ix, iy, iz;      // approximate reciprocal direction, clamped away from 0 (box tests only: conservative, not reproducible)
    float Sx, Sy, Sz;      // watertight shear constants (BLAS space only)
    uint32_t ksel;         // one-hot axis selectors: bit (3a + c) set iff k_a == c, a = 0 (kx), 1 (ky), 2 (kz)
    uint32_t octinv4;      // (dx>=0 | dy>=0 <<1 | dz>=0 <<2) * 0x01010101
};

__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// box-test part: origin, reciprocal direction, octant
__device__ __forceinline__ void setup_box(RaySpace& r, float ox, float oy, float oz, float dx, float dy, float dz) {
    r.ox = ox; r.oy = oy; r.oz = oz;
    const float tiny = 1e-20f;
    r.ix = rcp_approx(fabsf(dx) > tiny ? dx : copysignf(tiny, dx));
    r.iy = rcp_approx(fabsf(dy) > tiny ? dy : copysignf(tiny, dy));
    r.iz = rcp_approx(fabsf(dz) > tiny ? dz : copysignf(tiny, dz));
    // octant from the SIGN BITS, consistent with copysignf above: a component that is exactly -0 gets a huge negative reciprocal and
    // must pick the far/near planes of a negative direction (with `d >= 0` it was paired with the positive ones and the slab test
    // culled every box — tests/test_gpu_parity.py::test_trace_edge_cases)
    const uint32_t oct = ((__float_as_uint(dx) >> 31) ^ 1u) | (((__float_as_uint(dy) >> 31) ^ 1u) << 1) | (((__float_as_uint(dz) >> 31) ^ 1u) << 2);
    r.octinv4 = oct * 0x01010101u;
}
// triangle-test part (same rule as the oracle: first maximum in x,y,z order; swap kx,ky if d[kz] < 0;
// Sz = 1/d[kz] (IEEE), Sx = d[kx]*Sz, Sy = d[ky]*Sz)
__device__ __forceinline__ float fsel(bool p, float a, float b) {   // p ? a : b as one predicated select (never a branch)
    float d;
    asm("{ .reg .pred q; setp.ne.u32 q, %3, 0; selp.f32 %0, %1, %2, q; }" : "=f"(d) : "f"(a), "f"(b), "r"((uint32_t)p));
    return d;
}
__device__ __forceinline__ void setup_tri(RaySpace& r, float dx, float dy, float dz) {
    const float ax = fabsf(dx), ay = fabsf(dy), az = fabsf(dz);
    const bool yg = ay > ax;
    const bool zg = az > fmaxf(ax, ay);                   // first maximum in x,y,z order (NaN-free inputs)
    const uint32_t kz = zg ? 2u : (yg ? 1u : 0u);
    const float dkz = fsel(zg, dz, fsel(yg, dy, dx));
    float dkx = fsel(zg, dx, fsel(yg, dz, dy));           // kx = kz + 1 (mod 3), ky = kz + 2 (mod 3)
    float dky = fsel(zg, dy, fsel(yg, dx, dz));
    uint32_t kx = (kz == 2u) ? 0u : kz + 1u, ky = (kx == 2u) ? 0u : kx + 1u;
    const bool sw = dkz < 0.0f;
    const float t0 = fsel(sw, dky, dkx), t1 = fsel(sw, dkx, dky);
    const uint32_t k0 = sw ? ky : kx, k1 = sw ? kx : ky;
    r.ksel = (1u << k0) | (8u << k1) | (64u << kz);
    r.Sz = 1.0f / dkz;
    r.Sx = t0 * r.Sz;
    r.Sy = t1 * r.Sz;
}

// (v[kx], v[ky], v[kz]) for the three vertices at once: 6 mask tests + 18 predicated selects, no branches.
__device__ __forceinline__ void permute_axes(uint32_t ksel, float ax, float ay, float az, float bx, float by, float bz, float cx, float cy,
                                             float cz, float& Ax, float& Ay, float& Az, float& Bx, float& By, float& Bz, float& Cx,
                                             float& Cy, float& Cz) {
    asm("{\n\t"
        ".reg .pred x0, x1, y0, y1, z0, z1;\n\t"
        ".reg .b32 m;\n\t"
        ".reg .f32 t;\n\t"
        "and.b32 m, %18, 1;   setp.ne.u32 x0, m, 0;\n\t"
        "and.b32 m, %18, 2;   setp.ne.u32 x1, m, 0;\n\t"
        "and.b32 m, %18, 8;   setp.ne.u32 y0, m, 0;\n\t"
        "and.b32 m, %18, 16;  setp.ne.u32 y1, m, 0;\n\t"
        "and.b32 m, %18, 64;  setp.ne.u32 z0, m, 0;\n\t"
        "and.b32 m, %18, 128; setp.ne.u32 z1, m, 0;\n\t"
        "selp.f32 t, %10, %11, x1; selp.f32 %0, %9, t, x0;\n\t"
        "selp.f32 t, %10, %11, y1; selp.f32 %1, %9, t, y0;\n\t"
        "selp.f32 t, %10, %11, z1; selp.f32 %2, %9, t, z0;\n\t"
        "selp.f32 t, %13, %14, x1; selp.f32 %3, %12, t, x0;\n\t"
        "selp.f32 t, %13, %14, y1; selp.f32 %4, %12, t, y0;\n\t"
        "selp.f32 t, %13, %14, z1; selp.f32 %5, %12, t, z0;\n\t"
        "selp.f32 t, %16, %17, x1; selp.f32 %6, %15, t, x0;\n\t"
        "selp.f32 t, %16, %17, y1; selp.f32 %7, %15, t, y0;\n\t"
        "selp.f32 t, %16, %17, z1; selp.f32 %8, %15, t, z0;\n\t"
        "}"
        : "=f"(Ax), "=f"(Ay), "=f"(Az), "=f"(Bx), "=f"(By), "=f"(Bz), "=f"(Cx), "=f"(Cy), "=f"(Cz)
        : "f"(ax), "f"(ay), "f"(az), "f"(bx), "f"(by), "f"(bz), "f"(cx), "f"(cy), "f"(cz), "r"(ksel));
}

// Watertight ray/triangle test; identical operation order to oracle/rtx_oracle.cpp tri_test().
__device__ __forceinline__ bool tri_test(const RaySpace& r, float4 a, float4 b, float4 c, float tmin, float tmax,
                                         float& t, float& b1, float& b2) {
    float Akx, Aky, Akz, Bkx, Bky, Bkz, Ckx, Cky, Ckz;
    permute_axes(r.ksel, a.x - r.ox, a.y - r.oy, a.z - r.oz, b.x - r.ox, b.y - r.oy, b.z - r.oz, c.x - r.ox, c.y - r.oy, c.z - r.oz,
                 Akx, Aky, Akz, Bkx, Bky, Bkz, Ckx, Cky, Ckz);
    float Ax = Akx - r.Sx * Akz, Ay = Aky - r.Sy * Akz;
    float Bx = Bkx - r.Sx * Bkz, By = Bky - r.Sy * Bkz;
    float Cx = Ckx - r.Sx * Ckz, Cy = Cky - r.Sy * Ckz;
    float U = Cx * By - Cy * Bx;
    float V = Ax * Cy - Ay * Cx;
    float W = Bx * Ay - By * Ax;
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        U = (float)(__dsub_rn(__dmul_rn((double)Cx, (double)By), __dmul_rn((double)Cy, (double)Bx)));
        V = (float)(__dsub_rn(__dmul_rn((double)Ax, (double)Cy), __dmul_rn((double)Ay, (double)Cx)));
        W = (float)(__dsub_rn(__dmul_rn((double)Bx, (double)Ay), __dmul_rn((double)By, (double)Ax)));
    }
    const bool neg = (U < 0.0f) | (V < 0.0f) | (W < 0.0f);
    const bool pos = (U > 0.0f) | (V > 0.0f) | (W > 0.0f);
    float det = (U + V) + W;
    if ((neg & pos) | (det == 0.0f)) return false;
    float Az = r.Sz * Akz, Bz = r.Sz * Bkz, Cz = r.Sz * Ckz;
    float T = (U * Az + V * Bz) + W * Cz;
    float rcp = 1.0f / det;
    float tt = T * rcp;
    if (!(tt > tmin && tt < tmax)) return false;
    t = tt; b1 = V * rcp; b2 = W * rcp;
    return true;
}

// Intersects the 8 quantised child boxes of one node; returns the hit mask in the traversal's group format:
// bits 24..31 = hit inner children at bit 24 + (slot ^ octinv) (front-to-back priority), bits 0..23 = the triangle bits of the hit leaf
// children (child j owns bits 3j..3j+2, unary count).
// The node carries WI = imask << 24 | W (common.cuh), so a hit child j contributes WI & C_j with a compile-time C_j: ONE predicated
// LOP3 per child.  The octant permutation of the inner byte is one shared-memory table look-up per node (perm[o][h]: bit s of h -> bit
// s ^ o).  (Before: per-child meta bytes that needed 2 extractions, a variable shift and an OR per child plus the meta decoding,
// ~56 instructions per node against ~14.)
__device__ __forceinline__ uint32_t intersect_node(const RaySpace& r, uint4 n0, uint4 n1, uint4 n2, uint4 n3, uint4 n4,
                                                   float tmin, float tmax, uint32_t one, const uint8_t* __restrict__ perm) {
    const float px = __uint_as_float(n0.x), py = __uint_as_float(n0.y), pz = __uint_as_float(n0.z);
    const uint32_t e = n0.w;
    const float ax = __uint_as_float((e & 0xffu) << 23) * r.ix;
    const float ay = __uint_as_float(((e >> 8) & 0xffu) << 23) * r.iy;
    const float az = __uint_as_float(((e >> 16) & 0xffu) << 23) * r.iz;
    // plane = p + q * 2^e  ->  t = F(q) * A + B with F(q) = 1 + q/2^15 the float plane_byte() builds, A = 2^15 a, B = b - A.
    const float SC = 32768.0f;
    const float ax2 = ax * SC, ay2 = ay * SC, az2 = az * SC;
    const float bx = (px - r.ox) * r.ix - ax2, by = (py - r.oy) * r.iy - ay2, bz = (pz - r.oz) * r.iz - az2;
    // the rounding of (b - 2^15 a) is up to 2^-9 of a grid cell: widen the slab interval by 2^-23 |A| (= 2^-8 cell) instead
    const float w = 1.1920929e-7f, fx = fabsf(ax2), fy = fabsf(ay2), fz = fabsf(az2);
    const float bxn = __fmaf_rn(fx, -w, bx), bxf = __fmaf_rn(fx, w, bx), byn = __fmaf_rn(fy, -w, by), byf = __fmaf_rn(fy, w, by);
    const float bzn = __fmaf_rn(fz, -w, bz), bzf = __fmaf_rn(fz, w, bz);
    const bool nx = !(r.octinv4 & 1u), ny = !(r.octinv4 & 2u), nz = !(r.octinv4 & 4u);
    const uint32_t WI = n1.z;
    uint32_t acc = 0;
#define RTX_CHILD(H, J)                                                                                      \
        {                                                                                                    \
            float t0x = __fmaf_rn(plane_byte<J>(xn, one), ax2, bxn);                                         \
            float t0y = __fmaf_rn(plane_byte<J>(yn, one), ay2, byn);                                         \
            float t0z = __fmaf_rn(plane_byte<J>(zn, one), az2, bzn);                                         \
            float t1x = __fmaf_rn(plane_byte<J>(xf, one), ax2, bxf);                                         \
            float t1y = __fmaf_rn(plane_byte<J>(yf, one), ay2, byf);                                         \
            float t1z = __fmaf_rn(plane_byte<J>(zf, one), az2, bzf);                                         \
            float tn = fmaxf(fmaxf(t0x, t0y), fmaxf(t0z, tmin));                                             \
            float tf = fminf(fminf(t1x, t1y), fminf(t1z, tmax));                                             \
            asm("{ .reg .pred p; setp.le.f32 p, %1, %2; @p lop3.b32 %0, %3, %4, %0, 0xEA; }"                 \
                : "+r"(acc) : "f"(tn), "f"(tf), "r"(WI), "n"((7u << (3 * (4 * H + J))) | (1u << (24 + 4 * H + J)))); \
        }
#define RTX_HALF(H, QLOX, QLOY, QLOZ, QHIX, QHIY, QHIZ)                                                      \
    {                                                                                                        \
        const uint32_t xn = nx ? QHIX : QLOX, xf = nx ? QLOX : QHIX;                                         \
        const uint32_t yn = ny ? QHIY : QLOY, yf = ny ? QLOY : QHIY;                                         \
        const uint32_t zn = nz ? QHIZ : QLOZ, zf = nz ? QLOZ : QHIZ;                                         \
        RTX_CHILD(H, 0) RTX_CHILD(H, 1) RTX_CHILD(H, 2) RTX_CHILD(H, 3)                                      \
    }
    RTX_HALF(0, n2.x, n2.z, n3.x, n3.z, n4.x, n4.z)
    RTX_HALF(1, n2.y, n2.w, n3.y, n3.w, n4.y, n4.w)
#undef RTX_HALF
#undef RTX_CHILD
    const uint32_t P = perm[((r.octinv4 & 7u) << 8) | (acc >> 24)];
    return (acc & 0x00ffffffu) | (P << 24);
}

// bit s of h -> bit s ^ o, for all 8 octants o: the front-to-back order of the inner children (filled once per CTA)
__device__ __forceinline__ void fill_perm_table(uint8_t* perm, unsigned tid, unsigned nthreads) {
    for (unsigned i = tid; i < 2048u; i += nthreads) {
        const unsigned o = i >> 8, h = i & 255u;
        unsigned p = 0;
        for (unsigned b = 0; b < 8u; b++)
            if (h & (1u << b)) p |= 1u << (b ^ o);
        perm[i] = (uint8_t)p;
    }
}

// index of the primitive behind leaf bit `bit` of a node whose valid-primitive mask is W (primitives are stored densely in bit order)
__device__ __forceinline__ uint32_t leaf_prim_index(uint32_t W, uint32_t bit) { return __popc(W & ~(0xffffffffu << bit)); }

// ---- per-ray traversal state ------------------------------------------------------------------------------------------------------
// Hot state lives in registers (Trav); state that is touched a few times per ray lives in shared memory (TravCold), one float4 slot per
// thread and array, so that the kernel fits 64 registers = 8 resident CTAs per SM.
struct Trav {
    float ox, oy, oz;           // ray origin in the space currently traversed
    float ix, iy, iz;           // approximate reciprocal direction (box tests only)
    uint32_t octinv4;
    float tmin, tmax;
    float ht;                   // closest hit so far (t), tmax when there is none
    uint32_t hinst;             // its instance, 0xFFFFFFFF = none
    const uint4* nodes; const float4* prims;
    uint2 G;
    uint32_t cur_inst;
    int sp;
    int blas_sp;                // stack depth at which the current BLAS was entered; -1 while in the TLAS
};

struct TravCold {               // this thread's slots
    float4* wo;                 // world-space origin, bits(ray index)
    float4* wd;                 // world-space direction, -
    float4* hit;                // b1, b2, bits(prim), -
    float4* tri;                // Sx, Sy, Sz, bits(ksel): the watertight shear constants of the BLAS being traversed
};

__device__ __forceinline__ void load_box(const Trav& T, RaySpace& r) {
    r.ox = T.ox; r.oy = T.oy; r.oz = T.oz; r.ix = T.ix; r.iy = T.iy; r.iz = T.iz; r.octinv4 = T.octinv4;
}
__device__ __forceinline__ void store_box(Trav& T, const RaySpace& r) {
    T.ox = r.ox; T.oy = r.oy; T.oz = r.oz; T.ix = r.ix; T.iy = r.iy; T.iz = r.iz; T.octinv4 = r.octinv4;
}

__device__ __forceinline__ void trav_init(Trav& T, const TravCold& C, const SceneAS& S, float4 o_tmin, float4 d_tmax, uint32_t j) {
    *C.wo = make_float4(o_tmin.x, o_tmin.y, o_tmin.z, __uint_as_float(j));
    *C.wd = d_tmax;
    *C.hit = make_float4(0.0f, 0.0f, __uint_as_float(0xFFFFFFFFu), 0.0f);
    T.tmin = o_tmin.w; T.tmax = d_tmax.w;
    RaySpace r;
    setup_box(r, o_tmin.x, o_tmin.y, o_tmin.z, d_tmax.x, d_tmax.y, d_tmax.z);
    store_box(T, r);
    T.ht = d_tmax.w; T.hinst = 0xFFFFFFFFu;
    T.nodes = S.tlas_nodes; T.prims = S.inst_recs;
    T.G = make_uint2(0u, 0x80000000u);
    T.cur_inst = 0; T.sp = 0; T.blas_sp = -1;
}

// ---- phase-scheduled traversal -------------------------------------------------------------------------------------
// A step of one ray is: (N) intersect one node (or take a parked instance-leaf group from the stack), then (T) test the triangles of the
// hit leaf children or (I) enter one instance, then (P) pop when the current group is used up.
// ncu on C3 (profiles/r01_s4_*): with all of that in one per-lane step, the triangle loop ran at 2.3 of 32 lanes and the instance entry at
// 4.5 — a lane meets a triangle leaf on one node visit in nine and an instance on one in six, yet with 23 active lanes nearly every
// iteration of the warp paid for all three code paths.  Here a lane that finds triangles or an instance leaf PARKS (keeps
// (leaf_base, leaf_bits, leaf_W) in registers) and the warp runs T / I only when enough lanes are parked, or when too few lanes are left
// with node work (trace.cu).  A parked lane does nothing in between, so every ray still executes exactly the same sequence of steps and
// the results are bit-identical.
// (Measured alternatives, all slower: one triangle per step with the leaf group kept in registers; pending leaf groups parked on the
// stack; warp-cooperative triangle tests through a shared-memory pair list, -5 % on C2 / +4 % on C3 against the per-lane step;
// prefetch.global.L1 of a parked lane's first primitive, -2 %.)
enum { PEND_NONE = 0, PEND_TRI = 1, PEND_INST = 2 };

// (N).  Leaves (leaf_base, leaf_bits, leaf_W) != 0 when the lane has leaf work.
template <bool ANY_HIT, bool STATS>
__device__ __forceinline__ void trav_node(Trav& T, const SceneAS& S, const uint8_t* perm, uint2* stack, uint32_t& leaf_base, uint32_t& leaf_bits,
                                          uint32_t& leaf_W, unsigned int* c_nodes) {
    uint2 G = T.G;
    int sp = T.sp;
    if (G.y & 0xff000000u) {
        const uint32_t bit = 31u - __clz(G.y);
        G.y &= ~(1u << bit);
        const uint32_t imask = G.y & 0xffu;   // low byte carries the node's imask for relative indexing
        if (G.y & 0xff000000u) RTX_PUSH(G);
        const uint32_t slot = (bit - 24u) ^ (T.octinv4 & 0xffu);
        const uint32_t rel = __popc(imask & ~(0xffffffffu << slot));
        const uint4* np = T.nodes + (size_t)(G.x + rel) * 5;
        const uint4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3), n4 = __ldg(np + 4);
        if (STATS) (*c_nodes)++;
        RaySpace r;
        load_box(T, r);
        const uint32_t hm = intersect_node(r, n0, n1, n2, n3, n4, T.tmin, ANY_HIT ? T.tmax : T.ht, S.one_bits, perm);
        G.x = n1.x;
        G.y = (hm & 0xff000000u) | (n0.w >> 24);
        leaf_base = n1.y;
        leaf_bits = hm & 0x00ffffffu;
        leaf_W = n1.z;
    } else {                                   // an instance-leaf group that was parked on the stack (dense bits)
        leaf_base = G.x; leaf_bits = G.y; leaf_W = 0x00ffffffu;
        G = make_uint2(0u, 0u);
    }
    T.G = G; T.sp = sp;
}

// (T).  Returns true (ANY_HIT only) when a triangle was hit.
template <bool ANY_HIT, bool STATS>
__device__ __forceinline__ bool trav_tris(Trav& T, const TravCold& C, uint32_t leaf_base, uint32_t leaf_bits, uint32_t leaf_W, unsigned int* c_tris) {
    const float4 ts = *C.tri;
    RaySpace r;
    r.ox = T.ox; r.oy = T.oy; r.oz = T.oz; r.Sx = ts.x; r.Sy = ts.y; r.Sz = ts.z; r.ksel = __float_as_uint(ts.w);
    while (leaf_bits != 0u) {
        const uint32_t bit = 31u - __clz(leaf_bits);
        leaf_bits &= ~(1u << bit);
        const float4* tp = T.prims + (size_t)(leaf_base + leaf_prim_index(leaf_W, bit)) * 3;
        const float4 a = __ldg(tp), b = __ldg(tp + 1), c = __ldg(tp + 2);
        if (STATS) (*c_tris)++;
        float t, b1, b2;
        if (tri_test(r, a, b, c, T.tmin, T.tmax, t, b1, b2)) {
            if (ANY_HIT) return true;
            const uint32_t prim = __float_as_uint(a.w);
            // closest hit = lexicographic minimum of (t, instance, primitive)
            bool better = T.hinst == 0xFFFFFFFFu || t < T.ht;
            if (!better && t == T.ht)
                better = T.cur_inst < T.hinst || (T.cur_inst == T.hinst && prim < __float_as_uint(C.hit->z));
            if (better) {
                T.ht = t; T.hinst = T.cur_inst;
                *C.hit = make_float4(b1, b2, a.w, 0.0f);
            }
        }
    }
    return false;
}

// (I)  Takes the next instance leaf of the parked group.  The ray is transformed into the instance's object space and first tested against
// the model's object-space bounds (the world box of a rotated instance is up to sqrt(3) larger per axis than the geometry): on a miss the
// lane stays where it is (returns false; leaf_bits holds what is left of the group) and saves the shear set-up (an IEEE divide), the fetch
// and test of the BLAS root node and a stack round trip.
template <bool ANY_HIT, bool STATS>
__device__ __forceinline__ bool trav_enter_instance(Trav& T, const TravCold& C, const SceneAS& S, uint2* stack, uint32_t leaf_base,
                                                    uint32_t& leaf_bits, uint32_t leaf_W, unsigned int* c_insts) {
    const uint32_t bit = 31u - __clz(leaf_bits);
    leaf_bits &= ~(1u << bit);
    const float4* ip = T.prims + (size_t)(leaf_base + leaf_prim_index(leaf_W, bit)) * 4;
    const float4 r0 = __ldg(ip), r1 = __ldg(ip + 1), r2 = __ldg(ip + 2), r3 = __ldg(ip + 3);
    if (STATS) (*c_insts)++;
    const BlasRef* bp = S.blas + __float_as_uint(r3.x);
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(bp)), b1 = __ldg(reinterpret_cast<const float4*>(bp) + 1);
    const float2 b2 = __ldg(reinterpret_cast<const float2*>(bp) + 4);
    const float4 wo = *C.wo, wd = *C.wd;
    const float tox = ((r0.x * wo.x + r0.y * wo.y) + r0.z * wo.z) + r0.w * 1.0f;
    const float toy = ((r1.x * wo.x + r1.y * wo.y) + r1.z * wo.z) + r1.w * 1.0f;
    const float toz = ((r2.x * wo.x + r2.y * wo.y) + r2.z * wo.z) + r2.w * 1.0f;
    const float tdx = ((r0.x * wd.x + r0.y * wd.y) + r0.z * wd.z) + r0.w * 0.0f;
    const float tdy = ((r1.x * wd.x + r1.y * wd.y) + r1.z * wd.z) + r1.w * 0.0f;
    const float tdz = ((r2.x * wd.x + r2.y * wd.y) + r2.z * wd.z) + r2.w * 0.0f;
    RaySpace r;
    setup_box(r, tox, toy, toz, tdx, tdy, tdz);
    {   // slab test against (lo, hi) = (b1.x, b1.y, b1.z), (b1.w, b2.x, b2.y); conservative like the node test (approximate reciprocal
        // against bounds padded by 2^-15 of the model's scale)
        const float ax = (b1.x - tox) * r.ix, bx = (b1.w - tox) * r.ix;
        const float ay = (b1.y - toy) * r.iy, by = (b2.x - toy) * r.iy;
        const float az = (b1.z - toz) * r.iz, bz = (b2.y - toz) * r.iz;
        const float tn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), T.tmin));
        const float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), ANY_HIT ? T.tmax : T.ht));
        // widened by a relative 2^-20 on either side for the rounding of the reciprocal and the products (a few 2^-23 of t)
        if (!(tn * 0.999999f <= tf * 1.000001f) && !(tn <= tf)) return false;
    }
    uint2 G = T.G;
    int sp = T.sp;
    if (leaf_bits) {                       // park the other instance leaves with their bits made dense
        uint32_t dense = 0u, lb = leaf_bits;
        do {
            const uint32_t b = 31u - __clz(lb);
            lb &= ~(1u << b);
            dense |= 1u << leaf_prim_index(leaf_W, b);
        } while (lb);
        RTX_PUSH(make_uint2(leaf_base, dense));
    }
    if (G.y & 0xff000000u) RTX_PUSH(G);
    T.blas_sp = sp;
    setup_tri(r, tdx, tdy, tdz);
    store_box(T, r);
    *C.tri = make_float4(r.Sx, r.Sy, r.Sz, __uint_as_float(r.ksel));
    T.nodes = reinterpret_cast<const uint4*>(__float_as_uint(b0.x) | ((unsigned long long)__float_as_uint(b0.y) << 32));
    T.prims = reinterpret_cast<const float4*>(__float_as_uint(b0.z) | ((unsigned long long)__float_as_uint(b0.w) << 32));
    T.cur_inst = __float_as_uint(r3.y);
    T.G = make_uint2(0u, 0x80000000u); T.sp = sp;
    return true;
}

// (P) pops the next group when the current one is used up; returns true when the ray is finished
__device__ __forceinline__ bool trav_pop(Trav& T, const TravCold& C, const SceneAS& S, uint2* stack) {
    if ((T.G.y & 0xff000000u) == 0u) {
        int sp = T.sp;
        if (sp == T.blas_sp) {                 // the BLAS is exhausted: back to the TLAS / world space
            const float4 wo = *C.wo, wd = *C.wd;
            RaySpace r;
            setup_box(r, wo.x, wo.y, wo.z, wd.x, wd.y, wd.z);
            store_box(T, r);
            T.nodes = S.tlas_nodes; T.prims = S.inst_recs; T.blas_sp = -1;
        }
        if (sp == 0) return true;
        T.G = stack[--sp];
        T.sp = sp;
    }
    return false;
}

}  // namespace rtx
