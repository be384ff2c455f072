// bvh_build.cu — GPU builder of the compressed 8-wide BVH (BLAS over triangles, TLAS over instances).
//
// Replaces ID3D12GraphicsCommandList4::BuildRaytracingAccelerationStructure as driven by
// rdn/nv_helpers_dx12/BottomLevelASGenerator.cpp:97-117,235 and TopLevelASGenerator.cpp:181-199,240
// (the reference only describes geometry to the driver; the driver's builder has no source).
//
// Pipeline (all on the context stream, no host data structures):
//   1. primitive boxes + scene bounds        (k_tri_boxes, atomics on order-preserving uints)
//   2. 63-bit Morton codes of box centres     (k_morton)  + radix sort (cub::DeviceRadixSort — plumbing)
//   3. binary hierarchy by parallel locally-ordered clustering over the sorted order (k_ploc_*): every round each cluster
//      finds the neighbour (+-16 positions) with the smallest merged surface area; mutual pairs merge.  Each merge also
//      fills the node's table of the SAH dynamic programme (cost of covering the subtree with 1..7 wide-node roots)
//   4. SAH-optimal collapse to 8-wide nodes (k_collapse, one launch per tree level): follows the programme's decisions
//      (which subtrees become leaves of <= 3 primitives, how the 8 child slots are split); children are assigned to
//      octant slots so that (slot ^ ray octant) is a front-to-back order; boxes are quantised to 8 bits per plane
//      in the node's local power-of-two grid.
// Boxes are padded by 2^-15 of the model's coordinate scale so that the (bit-exact, contract-defining)
// ray/triangle test never reports a hit the conservative box tests culled.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "trace.h"

namespace rtx {

#define CKE(call)                            \
    do {                                     \
        cudaError_t e__ = (call);            \
        if (e__ != cudaSuccess) return e__;  \
    } while (0)

// primitives per leaf child: 3 triangles in a BLAS; ONE instance in the TLAS, so that every instance sits behind its own quantised box and a
// ray only enters the instances whose boxes it hits (with up to 3 instances per leaf box the C3 scene entered 2.69 instances per ray, and the
// one-node TLAS of C2 put both instances behind one box: 2.000)
#define MAX_LEAF 3          // the largest leaf any instantiation uses (array bounds)
#define SINGLE_NODE_MAX 8   // n <= 8 primitives: one node, one primitive per child slot

struct BuildCounters {
    unsigned int nodes, prims, tasks_out, hier_nodes;
    unsigned int bounds[6];   // order-preserving encodings: lo xyz (min), hi xyz (max)
};

__device__ __forceinline__ unsigned int enc_f(float f) {
    unsigned int b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __host__ __forceinline__ float dec_f(unsigned int e) {
    unsigned int b = (e & 0x80000000u) ? (e & 0x7fffffffu) : ~e;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    float f; memcpy(&f, &b, 4); return f;
#endif
}

// the padding of every primitive box: 2^-15 of the largest absolute coordinate of the reduced bounds
__device__ __forceinline__ float leaf_pad(const BuildCounters* c) {
    float s = 0.0f;
    for (int k = 0; k < 6; k++) s = fmaxf(s, fabsf(dec_f(c->bounds[k])));
    return s * 3.0517578125e-5f + 1e-30f;
}

__global__ void k_init_counters(BuildCounters* c) {
    c->nodes = 1; c->prims = 0; c->tasks_out = 0; c->hier_nodes = 0;
    c->bounds[0] = c->bounds[1] = c->bounds[2] = 0xffffffffu;
    c->bounds[3] = c->bounds[4] = c->bounds[5] = 0u;
}

__device__ __forceinline__ void reduce_bounds(BuildCounters* c, float lx, float ly, float lz, float hx, float hy, float hz, bool valid) {
    unsigned int v[6];
    v[0] = valid ? enc_f(lx) : 0xffffffffu; v[1] = valid ? enc_f(ly) : 0xffffffffu; v[2] = valid ? enc_f(lz) : 0xffffffffu;
    v[3] = valid ? enc_f(hx) : 0u; v[4] = valid ? enc_f(hy) : 0u; v[5] = valid ? enc_f(hz) : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 3; k++) v[k] = min(v[k], __shfl_xor_sync(0xffffffffu, v[k], o));
#pragma unroll
        for (int k = 3; k < 6; k++) v[k] = max(v[k], __shfl_xor_sync(0xffffffffu, v[k], o));
    }
    if ((threadIdx.x & 31) == 0) {
        for (int k = 0; k < 3; k++) atomicMin(&c->bounds[k], v[k]);
        for (int k = 3; k < 6; k++) atomicMax(&c->bounds[k], v[k]);
    }
}

__global__ void k_tri_boxes(const uint8_t* __restrict__ verts, const uint32_t* __restrict__ idx, uint32_t n,
                            float4* __restrict__ lo, float4* __restrict__ hi, BuildCounters* c) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = t < n;
    float lx = 0, ly = 0, lz = 0, hx = 0, hy = 0, hz = 0;
    if (valid) {
        const float* a = (const float*)(verts + (size_t)idx[3 * t] * 28);
        const float* b = (const float*)(verts + (size_t)idx[3 * t + 1] * 28);
        const float* d = (const float*)(verts + (size_t)idx[3 * t + 2] * 28);
        lx = fminf(a[0], fminf(b[0], d[0])); hx = fmaxf(a[0], fmaxf(b[0], d[0]));
        ly = fminf(a[1], fminf(b[1], d[1])); hy = fmaxf(a[1], fmaxf(b[1], d[1]));
        lz = fminf(a[2], fminf(b[2], d[2])); hz = fmaxf(a[2], fmaxf(b[2], d[2]));
        lo[t] = make_float4(lx, ly, lz, 0.0f);
        hi[t] = make_float4(hx, hy, hz, 0.0f);
    }
    reduce_bounds(c, lx, ly, lz, hx, hy, hz, valid);
}

__global__ void k_box_bounds(const float4* __restrict__ lo, const float4* __restrict__ hi, uint32_t n, BuildCounters* c) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = t < n;
    float4 l = valid ? lo[t] : make_float4(0, 0, 0, 0), h = valid ? hi[t] : make_float4(0, 0, 0, 0);
    reduce_bounds(c, l.x, l.y, l.z, h.x, h.y, h.z, valid);
}

__device__ __forceinline__ unsigned long long expand21(unsigned long long v) {
    v &= 0x1fffffull;
    v = (v | v << 32) & 0x1f00000000ffffull;
    v = (v | v << 16) & 0x1f0000ff0000ffull;
    v = (v | v << 8) & 0x100f00f00f00f00full;
    v = (v | v << 4) & 0x10c30c30c30c30c3ull;
    v = (v | v << 2) & 0x1249249249249249ull;
    return v;
}

__global__ void k_morton(const float4* __restrict__ lo, const float4* __restrict__ hi, uint32_t n, const BuildCounters* c,
                         unsigned long long* __restrict__ keys, uint32_t* __restrict__ vals) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    float blx = dec_f(c->bounds[0]), bly = dec_f(c->bounds[1]), blz = dec_f(c->bounds[2]);
    float ex = dec_f(c->bounds[3]) - blx, ey = dec_f(c->bounds[4]) - bly, ez = dec_f(c->bounds[5]) - blz;
    float4 l = lo[t], h = hi[t];
    float cx = 0.5f * (l.x + h.x), cy = 0.5f * (l.y + h.y), cz = 0.5f * (l.z + h.z);
    float fx = ex > 0.0f ? (cx - blx) / ex : 0.0f, fy = ey > 0.0f ? (cy - bly) / ey : 0.0f, fz = ez > 0.0f ? (cz - blz) / ez : 0.0f;
    unsigned long long qx = (unsigned long long)fminf(fmaxf(fx * 2097152.0f, 0.0f), 2097151.0f);
    unsigned long long qy = (unsigned long long)fminf(fmaxf(fy * 2097152.0f, 0.0f), 2097151.0f);
    unsigned long long qz = (unsigned long long)fminf(fmaxf(fz * 2097152.0f, 0.0f), 2097151.0f);
    keys[t] = (expand21(qx) << 2) | (expand21(qy) << 1) | expand21(qz);
    vals[t] = t;
}

// ---- binary hierarchy by parallel locally-ordered clustering (PLOC) over the Morton-sorted primitives.
// Node ids: leaf j (sorted position) -> j, inner nodes -> n + k in creation order.  Every merge also fills the node's
// table of the surface-area-heuristic dynamic programme that later picks the optimal 8-wide collapse:
//   C(m,1) = min(C_leaf(m), C_inner(m)),  C(m,i) = min(C_dist(m,i), C(m,i-1)),
//   C_inner(m) = A_m * c_node + C_dist(m,8),  C_dist(m,j) = min_k C(left,k) + C(right,j-k),  C_leaf(m) = A_m * P_m * c_prim (P_m <= 3)
#ifndef PLOC_RADIUS
#define PLOC_RADIUS 16
#endif
#define C_NODE 1.0f
#ifndef C_PRIM
#define C_PRIM 0.9f      // relative cost of a primitive test (swept 0.15 .. 2.5 on C2 / C3 / C5: profiles/r02_sah_prim_cost_sweep.txt)
#endif

struct Hier {
    float4* nlo; float4* nhi;       // boxes of all 2n-1 nodes
    int2* child;                    // inner nodes
    int* cnt;                       // primitives under an inner node
    float* cost;                    // 7 floats per inner node: C(m,1..7)
    unsigned char* dec;             // 8 bytes per inner node: [0] = 1 if C(m,1) is a leaf; [j-1], j=2..8: best k of C_dist(m,j),
                                    //   bit 7 set (j <= 7) if C(m,j) = C(m,j-1) (use fewer roots)
    int n;
};

__device__ __forceinline__ float box_area(float4 l, float4 h) {
    float dx = h.x - l.x, dy = h.y - l.y, dz = h.z - l.z;
    return 2.0f * (dx * dy + dy * dz + dz * dx);
}

__global__ void k_leaf_boxes(const float4* __restrict__ plo, const float4* __restrict__ phi, const uint32_t* __restrict__ vals, int n,
                             float4* __restrict__ nlo, float4* __restrict__ nhi, int* __restrict__ clusters, const BuildCounters* c) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const float pad = leaf_pad(c);
    const uint32_t p = vals[j];
    float4 l = plo[p], h = phi[p];
    nlo[j] = make_float4(l.x - pad, l.y - pad, l.z - pad, 0.0f);
    nhi[j] = make_float4(h.x + pad, h.y + pad, h.z + pad, 0.0f);
    clusters[j] = j;
}

__global__ void k_ploc_nn(const int* __restrict__ clusters, int nc, const float4* __restrict__ nlo, const float4* __restrict__ nhi,
                          int* __restrict__ nn) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nc) return;
    const int ci = clusters[i];
    const float4 l = nlo[ci], h = nhi[ci];
    float best = INFINITY; int bj = -1; unsigned bh = 0xffffffffu;
    const int j0 = max(0, i - PLOC_RADIUS), j1 = min(nc - 1, i + PLOC_RADIUS);
    for (int j = j0; j <= j1; j++) {
        if (j == i) continue;
        const int cj = clusters[j];
        const float4 l2 = nlo[cj], h2 = nhi[cj];
        const float4 ul = make_float4(fminf(l.x, l2.x), fminf(l.y, l2.y), fminf(l.z, l2.z), 0.0f);
        const float4 uh = make_float4(fmaxf(h.x, h2.x), fmaxf(h.y, h2.y), fmaxf(h.z, h2.z), 0.0f);
        const float a = box_area(ul, uh);
        // Equal areas (regular grids) are ordered by a symmetric hash of the pair: a strict total order on pairs, so the
        // smallest pair of every neighbourhood is mutual and ties cannot form long one-directional chains.
        unsigned hp = (unsigned)min(ci, cj) * 0x9E3779B1u ^ (unsigned)max(ci, cj) * 0x85EBCA77u;
        hp ^= hp >> 15; hp *= 0x2C1B3C6Du; hp ^= hp >> 12;
        if (a < best || (a == best && hp < bh)) { best = a; bj = j; bh = hp; }
    }
    nn[i] = bj;
}

__device__ __forceinline__ void node_costs(const Hier& H, int id, float out[7]) {
    if (id < H.n) {                       // single primitive: a leaf whatever the budget
        const float c = box_area(H.nlo[id], H.nhi[id]) * C_PRIM;
        for (int i = 0; i < 7; i++) out[i] = c;
    } else {
        const float* c = H.cost + (size_t)(id - H.n) * 7;
        for (int i = 0; i < 7; i++) out[i] = c[i];
    }
}

template <int MAXL>
__global__ void k_ploc_merge(const int* __restrict__ clusters, int nc, const int* __restrict__ nn, Hier H, BuildCounters* ctr,
                             int* __restrict__ out_val, int* __restrict__ valid) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nc) return;
    const int j = nn[i];
    const int a = clusters[i];
    if (j >= 0 && nn[j] == i) {
        if (i < j) {
            const int b = clusters[j];
            const int k = (int)atomicAdd(&ctr->hier_nodes, 1u);
            const int id = H.n + k;
            const float4 la = H.nlo[a], ha = H.nhi[a], lb = H.nlo[b], hb = H.nhi[b];
            const float4 l = make_float4(fminf(la.x, lb.x), fminf(la.y, lb.y), fminf(la.z, lb.z), 0.0f);
            const float4 h = make_float4(fmaxf(ha.x, hb.x), fmaxf(ha.y, hb.y), fmaxf(ha.z, hb.z), 0.0f);
            H.nlo[id] = l; H.nhi[id] = h;
            H.child[k] = make_int2(a, b);
            const int pa = a < H.n ? 1 : H.cnt[a - H.n], pb = b < H.n ? 1 : H.cnt[b - H.n];
            const int P = pa + pb;
            H.cnt[k] = P;
            // SAH dynamic programme
            float ca[7], cb[7];
            node_costs(H, a, ca); node_costs(H, b, cb);
            const float A = box_area(l, h);
            float dist[9]; unsigned char dk[9];
            for (int jj = 2; jj <= 8; jj++) {
                float best = INFINITY; int bk = 1;
                for (int kk = 1; kk < jj; kk++) {
                    if (kk > 7 || jj - kk > 7) continue;
                    const float c = ca[kk - 1] + cb[jj - kk - 1];
                    if (c < best) { best = c; bk = kk; }
                }
                dist[jj] = best; dk[jj] = (unsigned char)bk;
            }
            float* C = H.cost + (size_t)k * 7;
            unsigned char* D = H.dec + (size_t)k * 8;
            const float c_leaf = (P <= MAXL) ? A * (float)P * C_PRIM : INFINITY;
            const float c_inner = A * C_NODE + dist[8];
            C[0] = fminf(c_leaf, c_inner);
            D[0] = (c_leaf <= c_inner) ? 1 : 0;
            D[7] = dk[8];
            for (int ii = 2; ii <= 7; ii++) {
                if (C[ii - 2] <= dist[ii]) { C[ii - 1] = C[ii - 2]; D[ii - 1] = (unsigned char)(dk[ii] | 0x80u); }
                else { C[ii - 1] = dist[ii]; D[ii - 1] = dk[ii]; }
            }
            out_val[i] = id; valid[i] = 1;
        } else {
            out_val[i] = -1; valid[i] = 0;
        }
    } else {
        out_val[i] = a; valid[i] = 1;
    }
}

__global__ void k_ploc_compact(const int* __restrict__ out_val, const int* __restrict__ valid, const int* __restrict__ pos, int nc,
                               int* __restrict__ clusters_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nc) return;
    if (valid[i]) clusters_out[pos[i]] = out_val[i];
}

// ---- collapse to 8-wide compressed nodes
struct CollapseArgs {
    Hier H;
    const uint32_t* vals;
    uint4* out_nodes; float4* out_prims;
    BuildCounters* ctr;
};

struct TriSource {       // 3 x float4 per primitive
    const uint8_t* verts; const uint32_t* idx;
    __device__ __forceinline__ void write(float4* dst, uint32_t prim) const {
        const float* a = (const float*)(verts + (size_t)idx[3 * prim] * 28);
        const float* b = (const float*)(verts + (size_t)idx[3 * prim + 1] * 28);
        const float* d = (const float*)(verts + (size_t)idx[3 * prim + 2] * 28);
        dst[0] = make_float4(a[0], a[1], a[2], __uint_as_float(prim));
        dst[1] = make_float4(b[0], b[1], b[2], 0.0f);
        dst[2] = make_float4(d[0], d[1], d[2], 0.0f);
    }
};
struct RecSource {       // 4 x float4 per primitive
    const float4* recs;
    __device__ __forceinline__ void write(float4* dst, uint32_t prim) const {
        for (int k = 0; k < 4; k++) dst[k] = recs[(size_t)prim * 4 + k];
    }
};

__device__ __forceinline__ int exp_for_extent(float ext) {
    // smallest e with 255 * 2^e >= ext (conservatively one step larger when in doubt); biased into [1,254]
    float q = ext / 255.0f;
    int e = 0;
    if (q > 0.0f) { frexpf(q, &e); } else e = -126;
    int biased = e + 127;
    return max(1, min(254, biased));
}

// sorted positions of the (<= MAX_LEAF) primitives under node id
__device__ __forceinline__ int collect_prims(const Hier& H, int id, int out[MAX_LEAF]) {
    int n = 0; int st[4]; int sp = 0; st[sp++] = id;
    while (sp) {
        const int m = st[--sp];
        if (m < H.n) { if (n < MAX_LEAF) out[n++] = m; }
        else { const int2 c = H.child[m - H.n]; st[sp++] = c.y; st[sp++] = c.x; }
    }
    return n;
}

template <int PRIM_F4, typename Source>
__device__ void emit_node(const CollapseArgs& A, const Source& src, const int* cid, const bool* is_leaf, int cnt, float4 plo, float4 phi,
                          uint32_t out_idx, uint2* tasks_out) {
    const Hier& H = A.H;
    // slot assignment: greedy on cost[c][s] = dot(centre_c - centre_parent, sign vector of s)
    float ccx[8], ccy[8], ccz[8];
    const float pcx = 0.5f * (plo.x + phi.x), pcy = 0.5f * (plo.y + phi.y), pcz = 0.5f * (plo.z + phi.z);
    for (int c = 0; c < cnt; c++) {
        float4 l = H.nlo[cid[c]], h = H.nhi[cid[c]];
        ccx[c] = 0.5f * (l.x + h.x) - pcx; ccy[c] = 0.5f * (l.y + h.y) - pcy; ccz[c] = 0.5f * (l.z + h.z) - pcz;
    }
    int slot_child[8];
    for (int s = 0; s < 8; s++) slot_child[s] = -1;
    unsigned child_done = 0, slot_done = 0;
    for (int it = 0; it < cnt; it++) {
        float best = -INFINITY; int bc = -1, bs = -1;
        for (int c = 0; c < cnt; c++) {
            if (child_done & (1u << c)) continue;
            for (int s = 0; s < 8; s++) {
                if (slot_done & (1u << s)) continue;
                float cost = ((s & 1) ? ccx[c] : -ccx[c]) + ((s & 2) ? ccy[c] : -ccy[c]) + ((s & 4) ? ccz[c] : -ccz[c]);
                if (cost > best) { best = cost; bc = c; bs = s; }
            }
        }
        slot_child[bs] = bc; child_done |= 1u << bc; slot_done |= 1u << bs;
    }
    unsigned imask = 0; int n_inner = 0, n_prims = 0;
    int cnt_of[8];
    for (int s = 0; s < 8; s++) {
        cnt_of[s] = 0;
        int c = slot_child[s];
        if (c < 0) continue;
        int id = cid[c];
        if (!is_leaf[c]) { imask |= 1u << s; n_inner++; }
        else { cnt_of[s] = (id < H.n) ? 1 : H.cnt[id - H.n]; n_prims += cnt_of[s]; }
    }
    const uint32_t child_base = n_inner ? atomicAdd(&A.ctr->nodes, (unsigned)n_inner) : 0u;
    const uint32_t prim_base = n_prims ? atomicAdd(&A.ctr->prims, (unsigned)n_prims) : 0u;
    const uint32_t task_base = n_inner ? atomicAdd(&A.ctr->tasks_out, (unsigned)n_inner) : 0u;
    const int ex = exp_for_extent(phi.x - plo.x), ey = exp_for_extent(phi.y - plo.y), ez = exp_for_extent(phi.z - plo.z);
    const float sx = __uint_as_float((unsigned)ex << 23), sy = __uint_as_float((unsigned)ey << 23), sz = __uint_as_float((unsigned)ez << 23);
    unsigned char qlo[3][8], qhi[3][8];
    unsigned W = 0;                          // unary primitive count of leaf child s at bits 3s..3s+2
    int inner_rank = 0, prim_off = 0;
    for (int s = 0; s < 8; s++) {
        for (int a = 0; a < 3; a++) { qlo[a][s] = 0; qhi[a][s] = 0; }
        int c = slot_child[s];
        if (c < 0) continue;
        int id = cid[c];
        float4 l = H.nlo[id], h = H.nhi[id];
        const float lov[3] = {l.x, l.y, l.z}, hiv[3] = {h.x, h.y, h.z}, pv[3] = {plo.x, plo.y, plo.z}, sv[3] = {sx, sy, sz};
        for (int a = 0; a < 3; a++) {
            int ql = (int)floorf((lov[a] - pv[a]) / sv[a]);
            int qh = (int)ceilf((hiv[a] - pv[a]) / sv[a]);
            ql = max(0, min(255, ql)); qh = max(0, min(255, qh));
            while (ql > 0 && pv[a] + (float)ql * sv[a] > lov[a]) ql--;
            while (qh < 255 && pv[a] + (float)qh * sv[a] < hiv[a]) qh++;
            qlo[a][s] = (unsigned char)ql; qhi[a][s] = (unsigned char)qh;
        }
        if (imask & (1u << s)) {
            tasks_out[task_base + inner_rank] = make_uint2((unsigned)id, child_base + inner_rank);
            inner_rank++;
        } else {
            int pr[MAX_LEAF];
            const int pc = collect_prims(H, id, pr);
            W |= ((1u << pc) - 1u) << (3 * s);
            for (int k = 0; k < pc; k++)
                src.write(A.out_prims + (size_t)(prim_base + prim_off + k) * PRIM_F4, A.vals[pr[k]]);
            prim_off += pc;
        }
    }
    auto pack4 = [](const unsigned char* b) { return (unsigned)b[0] | ((unsigned)b[1] << 8) | ((unsigned)b[2] << 16) | ((unsigned)b[3] << 24); };
    uint4* o = A.out_nodes + (size_t)out_idx * 5;
    o[0] = make_uint4(__float_as_uint(plo.x), __float_as_uint(plo.y), __float_as_uint(plo.z),
                      (unsigned)ex | ((unsigned)ey << 8) | ((unsigned)ez << 16) | (imask << 24));
    o[1] = make_uint4(child_base, prim_base, W | (imask << 24), 0u);
    o[2] = make_uint4(pack4(qlo[0]), pack4(qlo[0] + 4), pack4(qlo[1]), pack4(qlo[1] + 4));
    o[3] = make_uint4(pack4(qlo[2]), pack4(qlo[2] + 4), pack4(qhi[0]), pack4(qhi[0] + 4));
    o[4] = make_uint4(pack4(qhi[1]), pack4(qhi[1] + 4), pack4(qhi[2]), pack4(qhi[2] + 4));
}

// One wide node per task: follow the dynamic programme's decisions from the task's hierarchy node with a budget of 8 roots.
template <int PRIM_F4, typename Source>
__global__ void k_collapse(CollapseArgs A, Source src, const uint2* __restrict__ tasks_in, unsigned n_in, uint2* tasks_out) {
    unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_in) return;
    const Hier& H = A.H;
    const uint2 task = tasks_in[t];
    const int root = (int)task.x;
    int cid[8]; bool leaf[8]; int cnt = 0;
    int st_node[16], st_budget[16]; int sp = 0;
    {
        const int2 ch = H.child[root - H.n];
        const int k = H.dec[(size_t)(root - H.n) * 8 + 7] & 0x7f;
        st_node[sp] = ch.y; st_budget[sp++] = 8 - k;
        st_node[sp] = ch.x; st_budget[sp++] = k;
    }
    while (sp) {
        const int m = st_node[--sp]; int j = st_budget[sp];
        if (m < H.n) { cid[cnt] = m; leaf[cnt++] = true; continue; }
        const unsigned char* D = H.dec + (size_t)(m - H.n) * 8;
        while (j >= 2 && j <= 7 && (D[j - 1] & 0x80u)) j--;        // C(m,j) = C(m,j-1)
        if (j == 1) { cid[cnt] = m; leaf[cnt++] = (D[0] != 0); continue; }
        const int k = D[j - 1] & 0x7f;
        const int2 ch = H.child[m - H.n];
        st_node[sp] = ch.y; st_budget[sp++] = j - k;
        st_node[sp] = ch.x; st_budget[sp++] = k;
    }
    emit_node<PRIM_F4, Source>(A, src, cid, leaf, cnt, H.nlo[root], H.nhi[root], task.y, tasks_out);
}

// n <= SINGLE_NODE_MAX: one node, primitive i alone in child slot i behind its own quantised box
template <int PRIM_F4, typename Source>
__global__ void k_single_node(Source src, const float4* __restrict__ plo, const float4* __restrict__ phi, int n, uint4* out_nodes,
                              float4* out_prims, BuildCounters* c) {
    if (threadIdx.x || blockIdx.x) return;
    const float pad = leaf_pad(c);
    float l[3] = {INFINITY, INFINITY, INFINITY}, h[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = 0; i < n; i++) {
        const float4 a = plo[i], b = phi[i];
        l[0] = fminf(l[0], a.x - pad); l[1] = fminf(l[1], a.y - pad); l[2] = fminf(l[2], a.z - pad);
        h[0] = fmaxf(h[0], b.x + pad); h[1] = fmaxf(h[1], b.y + pad); h[2] = fmaxf(h[2], b.z + pad);
    }
    int e[3]; float sv[3];
    for (int a = 0; a < 3; a++) { e[a] = exp_for_extent(h[a] - l[a]); sv[a] = __uint_as_float((unsigned)e[a] << 23); }
    unsigned char qlo[3][8], qhi[3][8];
    unsigned W = 0;
    for (int i = 0; i < 8; i++) {
        for (int a = 0; a < 3; a++) { qlo[a][i] = 0; qhi[a][i] = 0; }
        if (i >= n) continue;
        W |= 1u << (3 * i);
        src.write(out_prims + (size_t)i * PRIM_F4, (uint32_t)i);
        const float4 a4 = plo[i], b4 = phi[i];
        const float lov[3] = {a4.x - pad, a4.y - pad, a4.z - pad}, hiv[3] = {b4.x + pad, b4.y + pad, b4.z + pad};
        for (int a = 0; a < 3; a++) {
            int ql = (int)floorf((lov[a] - l[a]) / sv[a]);
            int qh = (int)ceilf((hiv[a] - l[a]) / sv[a]);
            ql = max(0, min(255, ql)); qh = max(0, min(255, qh));
            while (ql > 0 && l[a] + (float)ql * sv[a] > lov[a]) ql--;
            while (qh < 255 && l[a] + (float)qh * sv[a] < hiv[a]) qh++;
            qlo[a][i] = (unsigned char)ql; qhi[a][i] = (unsigned char)qh;
        }
    }
    auto pack4 = [](const unsigned char* b) { return (unsigned)b[0] | ((unsigned)b[1] << 8) | ((unsigned)b[2] << 16) | ((unsigned)b[3] << 24); };
    out_nodes[0] = make_uint4(__float_as_uint(l[0]), __float_as_uint(l[1]), __float_as_uint(l[2]), (unsigned)e[0] | ((unsigned)e[1] << 8) | ((unsigned)e[2] << 16));
    out_nodes[1] = make_uint4(0u, 0u, W, 0u);
    out_nodes[2] = make_uint4(pack4(qlo[0]), pack4(qlo[0] + 4), pack4(qlo[1]), pack4(qlo[1] + 4));
    out_nodes[3] = make_uint4(pack4(qlo[2]), pack4(qlo[2] + 4), pack4(qhi[0]), pack4(qhi[0] + 4));
    out_nodes[4] = make_uint4(pack4(qhi[1]), pack4(qhi[1] + 4), pack4(qhi[2]), pack4(qhi[2] + 4));
    c->nodes = 1; c->prims = (unsigned)n;
}

struct Scratch {
    void* p = nullptr;
    ~Scratch() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 16); }
};
// all the scratch of one build in ONE allocation, carved up front (a build used to make 20 cudaMallocs)
struct Arena {
    char* base = nullptr; size_t used = 0, cap = 0;
    ~Arena() { if (base) cudaFree(base); }
    static size_t pad(size_t b) { return (b + 255) & ~(size_t)255; }
    cudaError_t reserve(size_t bytes) { cap = bytes; return cudaMalloc((void**)&base, bytes ? bytes : 256); }
    void* take(size_t bytes) { void* p = base + used; used += pad(bytes); return used <= cap ? p : nullptr; }
};

template <int PRIM_F4, int MAXL, typename Source>
static cudaError_t build_generic(const float4* d_plo, const float4* d_phi, uint32_t n, Source src, BuildCounters* d_ctr, Bvh8* out,
                                 cudaStream_t stream) {
    const int TB = 256;
    auto grid = [&](size_t k) { return (unsigned)((k + TB - 1) / TB); };
    const uint32_t max_nodes = n <= SINGLE_NODE_MAX ? 1u : n;
    Scratch nodes_s, prims_s;
    CKE(nodes_s.alloc((size_t)max_nodes * 80));
    CKE(prims_s.alloc((size_t)n * PRIM_F4 * 16));
    uint4* d_nodes = (uint4*)nodes_s.p;
    float4* d_prims = (float4*)prims_s.p;
    BuildCounters h_ctr;
    out->sah_cost = 0.0f;

    if (n <= SINGLE_NODE_MAX) {
        out->n_levels = 1; out->level_start[0] = 0; out->level_start[1] = 1;
        k_single_node<PRIM_F4, Source><<<1, 32, 0, stream>>>(src, d_plo, d_phi, (int)n, d_nodes, d_prims, d_ctr);
    } else {
        size_t tmp_bytes = 0, tmp2_bytes = 0;
        CKE(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                            (uint32_t*)nullptr, (uint32_t*)nullptr, (int)n, 0, 63, stream));
        CKE(cub::DeviceScan::ExclusiveSum(nullptr, tmp2_bytes, (int*)nullptr, (int*)nullptr, (int)n, stream));
        struct Buf { void* p; };
        Arena arena;
        const size_t sizes[] = {(size_t)n * 8, (size_t)n * 8, (size_t)n * 4, (size_t)n * 4, (size_t)n * 8, (size_t)n * 4, (size_t)n * 28, (size_t)n * 8,
                                (size_t)2 * n * 16, (size_t)2 * n * 16, (size_t)n * 4, (size_t)n * 4, (size_t)n * 4, (size_t)n * 4, (size_t)n * 4,
                                (size_t)n * 4, (size_t)n * 8, (size_t)n * 8, tmp_bytes, tmp2_bytes};
        size_t total = 0;
        for (size_t b : sizes) total += Arena::pad(b);
        CKE(arena.reserve(total));
        Buf keys_a{arena.take(sizes[0])}, keys_b{arena.take(sizes[1])}, vals_a{arena.take(sizes[2])}, vals_b{arena.take(sizes[3])},
            child_s{arena.take(sizes[4])}, cnt_s{arena.take(sizes[5])}, cost_s{arena.take(sizes[6])}, dec_s{arena.take(sizes[7])},
            nlo_s{arena.take(sizes[8])}, nhi_s{arena.take(sizes[9])}, cl_a{arena.take(sizes[10])}, cl_b{arena.take(sizes[11])},
            nn_s{arena.take(sizes[12])}, val_s{arena.take(sizes[13])}, valid_s{arena.take(sizes[14])}, pos_s{arena.take(sizes[15])},
            tasks_a{arena.take(sizes[16])}, tasks_b{arena.take(sizes[17])}, tmp_s{arena.take(sizes[18])}, tmp2_s{arena.take(sizes[19])};
        k_morton<<<grid(n), TB, 0, stream>>>(d_plo, d_phi, n, d_ctr, (unsigned long long*)keys_a.p, (uint32_t*)vals_a.p);
        CKE(cub::DeviceRadixSort::SortPairs(tmp_s.p, tmp_bytes, (unsigned long long*)keys_a.p, (unsigned long long*)keys_b.p,
                                            (uint32_t*)vals_a.p, (uint32_t*)vals_b.p, (int)n, 0, 63, stream));
        Hier H;
        H.nlo = (float4*)nlo_s.p; H.nhi = (float4*)nhi_s.p; H.child = (int2*)child_s.p; H.cnt = (int*)cnt_s.p;
        H.cost = (float*)cost_s.p; H.dec = (unsigned char*)dec_s.p; H.n = (int)n;
        int* cin = (int*)cl_a.p; int* cout = (int*)cl_b.p;
        k_leaf_boxes<<<grid(n), TB, 0, stream>>>(d_plo, d_phi, (uint32_t*)vals_b.p, (int)n, H.nlo, H.nhi, cin, d_ctr);
        int nc = (int)n;
        while (nc > 1) {
            k_ploc_nn<<<grid(nc), TB, 0, stream>>>(cin, nc, H.nlo, H.nhi, (int*)nn_s.p);
            k_ploc_merge<MAXL><<<grid(nc), TB, 0, stream>>>(cin, nc, (int*)nn_s.p, H, d_ctr, (int*)val_s.p, (int*)valid_s.p);
            CKE(cub::DeviceScan::ExclusiveSum(tmp2_s.p, tmp2_bytes, (int*)valid_s.p, (int*)pos_s.p, nc, stream));
            k_ploc_compact<<<grid(nc), TB, 0, stream>>>((int*)val_s.p, (int*)valid_s.p, (int*)pos_s.p, nc, cout);
            CKE(cudaMemcpyAsync(&h_ctr, d_ctr, sizeof h_ctr, cudaMemcpyDeviceToHost, stream));
            CKE(cudaStreamSynchronize(stream));
            const int merged = (int)h_ctr.hier_nodes;
            const int nc_new = (int)n - merged;
            if (nc_new >= nc) return cudaErrorUnknown;          // no progress: cannot happen (the closest pair is always mutual)
            nc = nc_new;
            int* t = cin; cin = cout; cout = t;
        }
        int root = 0;
        CKE(cudaMemcpyAsync(&root, cin, sizeof(int), cudaMemcpyDeviceToHost, stream));
        CKE(cudaStreamSynchronize(stream));
        float root_cost[7];
        CKE(cudaMemcpy(root_cost, H.cost + (size_t)(root - (int)n) * 7, sizeof root_cost, cudaMemcpyDeviceToHost));
        float4 rl, rh;
        CKE(cudaMemcpy(&rl, H.nlo + root, 16, cudaMemcpyDeviceToHost)); CKE(cudaMemcpy(&rh, H.nhi + root, 16, cudaMemcpyDeviceToHost));
        const float ra = 2.0f * ((rh.x - rl.x) * (rh.y - rl.y) + (rh.y - rl.y) * (rh.z - rl.z) + (rh.z - rl.z) * (rh.x - rl.x));
        out->sah_cost = ra > 0.0f ? root_cost[0] / ra : 0.0f;
        CollapseArgs A;
        A.H = H; A.vals = (uint32_t*)vals_b.p; A.out_nodes = d_nodes; A.out_prims = d_prims; A.ctr = d_ctr;
        uint2 root_task = make_uint2((unsigned)root, 0u);
        CKE(cudaMemcpyAsync(tasks_a.p, &root_task, sizeof root_task, cudaMemcpyHostToDevice, stream));
        unsigned n_in = 1;
        uint2* tin = (uint2*)tasks_a.p; uint2* tout = (uint2*)tasks_b.p;
        out->n_levels = 1; out->level_start[0] = 0; out->level_start[1] = 1;
        while (n_in > 0) {
            k_collapse<PRIM_F4, Source><<<grid(n_in), TB, 0, stream>>>(A, src, tin, n_in, tout);
            CKE(cudaMemcpyAsync(&h_ctr, d_ctr, sizeof h_ctr, cudaMemcpyDeviceToHost, stream));
            CKE(cudaStreamSynchronize(stream));
            if (h_ctr.tasks_out > 0 && out->n_levels < 47u) { out->n_levels++; out->level_start[out->n_levels] = h_ctr.nodes; }
            n_in = h_ctr.tasks_out;
            CKE(cudaMemsetAsync(&d_ctr->tasks_out, 0, sizeof(unsigned), stream));
            uint2* t = tin; tin = tout; tout = t;
        }
        CKE(cudaGetLastError());
    }
    CKE(cudaMemcpyAsync(&h_ctr, d_ctr, sizeof h_ctr, cudaMemcpyDeviceToHost, stream));
    CKE(cudaStreamSynchronize(stream));
    CKE(cudaGetLastError());
    out->n_nodes = h_ctr.nodes; out->n_prims = h_ctr.prims;
    // right-size the node array (child indices are relative to the array start, so a plain copy is valid)
    CKE(cudaMalloc((void**)&out->nodes, (size_t)out->n_nodes * 80));
    CKE(cudaMemcpyAsync(out->nodes, d_nodes, (size_t)out->n_nodes * 80, cudaMemcpyDeviceToDevice, stream));
    out->prims = d_prims; prims_s.p = nullptr;
    float s = 0.0f;
    for (int k = 0; k < 6; k++) s = fmaxf(s, fabsf(dec_f(h_ctr.bounds[k])));
    const float pad = s * 3.0517578125e-5f + 1e-30f;
    for (int k = 0; k < 3; k++) { out->lo[k] = dec_f(h_ctr.bounds[k]) - pad; out->hi[k] = dec_f(h_ctr.bounds[3 + k]) + pad; }
    CKE(cudaStreamSynchronize(stream));
    return cudaSuccess;
}

cudaError_t build_blas(const uint8_t* d_vertices, uint32_t n_vertices, const uint32_t* d_indices, uint32_t n_tris, Bvh8* out,
                       cudaStream_t stream) {
    (void)n_vertices;
    cudaEvent_t e0, e1;
    CKE(cudaEventCreate(&e0)); CKE(cudaEventCreate(&e1));
    CKE(cudaEventRecord(e0, stream));
    Scratch plo, phi, ctr;
    CKE(plo.alloc((size_t)n_tris * 16)); CKE(phi.alloc((size_t)n_tris * 16)); CKE(ctr.alloc(sizeof(BuildCounters)));
    k_init_counters<<<1, 1, 0, stream>>>((BuildCounters*)ctr.p);
    if (n_tris) k_tri_boxes<<<(n_tris + 255) / 256, 256, 0, stream>>>(d_vertices, d_indices, n_tris, (float4*)plo.p, (float4*)phi.p, (BuildCounters*)ctr.p);
    TriSource src{d_vertices, d_indices};
    cudaError_t e = build_generic<3, 3, TriSource>((float4*)plo.p, (float4*)phi.p, n_tris, src, (BuildCounters*)ctr.p, out, stream);
    if (e == cudaSuccess) {
        cudaEventRecord(e1, stream); cudaEventSynchronize(e1);
        cudaEventElapsedTime(&out->build_ms, e0, e1);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return e;
}

cudaError_t build_tlas(const float4* d_inst_recs, const float4* d_box_lo, const float4* d_box_hi, uint32_t n_instances, Bvh8* out,
                       cudaStream_t stream) {
    Scratch ctr;
    CKE(ctr.alloc(sizeof(BuildCounters)));
    k_init_counters<<<1, 1, 0, stream>>>((BuildCounters*)ctr.p);
    if (n_instances) k_box_bounds<<<(n_instances + 255) / 256, 256, 0, stream>>>(d_box_lo, d_box_hi, n_instances, (BuildCounters*)ctr.p);
    RecSource src{d_inst_recs};
    return build_generic<4, 1, RecSource>(d_box_lo, d_box_hi, n_instances, src, (BuildCounters*)ctr.p, out, stream);
}

// ---- TLAS refit ------------------------------------------------------------------------------------------------------
// leaf order of the instance records: prims[k] (4 x float4) carries its instance id in .w.y
__global__ void k_refit_prims(const float4* __restrict__ recs, uint32_t n_prims, float4* __restrict__ prims) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_prims) return;
    const uint32_t inst = __float_as_uint(prims[4 * k + 3].y);
    for (int r = 0; r < 4; r++) prims[4 * k + r] = recs[4 * (size_t)inst + r];
}

// the box a node's quantised planes describe (a conservative superset of everything below it)
__device__ __forceinline__ void node_box(const uint4* np, float lo[3], float hi[3]) {
    const uint4 n0 = np[0], n1 = np[1], n2 = np[2], n3 = np[3], n4 = np[4];
    const float p[3] = {__uint_as_float(n0.x), __uint_as_float(n0.y), __uint_as_float(n0.z)};
    const float sc[3] = {__uint_as_float((n0.w & 0xffu) << 23), __uint_as_float(((n0.w >> 8) & 0xffu) << 23), __uint_as_float(((n0.w >> 16) & 0xffu) << 23)};
    const uint32_t qlo[3][2] = {{n2.x, n2.y}, {n2.z, n2.w}, {n3.x, n3.y}}, qhi[3][2] = {{n3.z, n3.w}, {n4.x, n4.y}, {n4.z, n4.w}};
    const uint32_t WI = n1.z;
    for (int a = 0; a < 3; a++) { lo[a] = INFINITY; hi[a] = -INFINITY; }
    for (int s = 0; s < 8; s++) {
        if (!((WI >> (24 + s)) & 1u) && !((WI >> (3 * s)) & 7u)) continue;     // empty slot
        for (int a = 0; a < 3; a++) {
            const float ql = (float)((qlo[a][s >> 2] >> (8 * (s & 3))) & 0xffu), qh = (float)((qhi[a][s >> 2] >> (8 * (s & 3))) & 0xffu);
            lo[a] = fminf(lo[a], p[a] + ql * sc[a]); hi[a] = fmaxf(hi[a], p[a] + qh * sc[a]);
        }
    }
}

// Leaf-box sources of the refit: the box of the primitive record in leaf slot `slot`, folded into l / h.
struct InstLeafBoxes {   // TLAS: the instance's (already padded) world box, found through the instance id in .w.y of the record
    const float4* prims; const float4* box_lo; const float4* box_hi;
    __device__ __forceinline__ void fold(uint32_t slot, float l[3], float h[3]) const {
        const uint32_t inst = __float_as_uint(prims[4 * (size_t)slot + 3].y);
        const float4 a = box_lo[inst], b = box_hi[inst];
        l[0] = fminf(l[0], a.x); l[1] = fminf(l[1], a.y); l[2] = fminf(l[2], a.z);
        h[0] = fmaxf(h[0], b.x); h[1] = fmaxf(h[1], b.y); h[2] = fmaxf(h[2], b.z);
    }
};
struct TriLeafBoxes {    // BLAS: the refitted triangle record, padded as k_tri_boxes + k_leaf_boxes / k_single_node pad a triangle
    const float4* prims; const BuildCounters* ctr;
    __device__ __forceinline__ void fold(uint32_t slot, float l[3], float h[3]) const {
        const float pad = leaf_pad(ctr);
        const float4 a = prims[3 * (size_t)slot], b = prims[3 * (size_t)slot + 1], d = prims[3 * (size_t)slot + 2];
        l[0] = fminf(l[0], fminf(a.x, fminf(b.x, d.x)) - pad); h[0] = fmaxf(h[0], fmaxf(a.x, fmaxf(b.x, d.x)) + pad);
        l[1] = fminf(l[1], fminf(a.y, fminf(b.y, d.y)) - pad); h[1] = fmaxf(h[1], fmaxf(a.y, fmaxf(b.y, d.y)) + pad);
        l[2] = fminf(l[2], fminf(a.z, fminf(b.z, d.z)) - pad); h[2] = fmaxf(h[2], fmaxf(a.z, fmaxf(b.z, d.z)) + pad);
    }
};

// one thread per node of one level: child boxes from the refitted children (inner) or the leaf source (leaves), then the same
// origin / exponent / outward quantisation as emit_node.  Topology, child order and primitive order stay those of the build.
template <typename Leaves>
__global__ void k_refit_level(uint4* __restrict__ nodes, uint32_t first, uint32_t count, Leaves leaves) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    uint4* np = nodes + (size_t)(first + t) * 5;
    const uint4 n0 = np[0], n1 = np[1];
    const uint32_t WI = n1.z, imask = WI >> 24, W = WI & 0x00ffffffu;
    float clo[8][3], chi[8][3];
    bool used[8];
    float plo[3] = {INFINITY, INFINITY, INFINITY}, phi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int s = 0; s < 8; s++) {
        used[s] = false;
        if ((imask >> s) & 1u) {
            const uint32_t child = n1.x + __popc(imask & ((1u << s) - 1u));
            node_box(nodes + (size_t)child * 5, clo[s], chi[s]);
            used[s] = true;
        } else if ((W >> (3 * s)) & 7u) {
            for (int a = 0; a < 3; a++) { clo[s][a] = INFINITY; chi[s][a] = -INFINITY; }
            for (int k = 0; k < 3; k++) {
                if (!((W >> (3 * s + k)) & 1u)) continue;
                leaves.fold(n1.y + __popc(W & ((1u << (3 * s + k)) - 1u)), clo[s], chi[s]);
            }
            used[s] = true;
        }
        if (used[s]) for (int a = 0; a < 3; a++) { plo[a] = fminf(plo[a], clo[s][a]); phi[a] = fmaxf(phi[a], chi[s][a]); }
    }
    int e[3]; float sv[3];
    for (int a = 0; a < 3; a++) { e[a] = exp_for_extent(phi[a] - plo[a]); sv[a] = __uint_as_float((unsigned)e[a] << 23); }
    unsigned char qlo[3][8], qhi[3][8];
    for (int s = 0; s < 8; s++) {
        for (int a = 0; a < 3; a++) { qlo[a][s] = 0; qhi[a][s] = 0; }
        if (!used[s]) continue;
        for (int a = 0; a < 3; a++) {
            int ql = (int)floorf((clo[s][a] - plo[a]) / sv[a]);
            int qh = (int)ceilf((chi[s][a] - plo[a]) / sv[a]);
            ql = max(0, min(255, ql)); qh = max(0, min(255, qh));
            while (ql > 0 && plo[a] + (float)ql * sv[a] > clo[s][a]) ql--;
            while (qh < 255 && plo[a] + (float)qh * sv[a] < chi[s][a]) qh++;
            qlo[a][s] = (unsigned char)ql; qhi[a][s] = (unsigned char)qh;
        }
    }
    auto pack4 = [](const unsigned char* b) { return (unsigned)b[0] | ((unsigned)b[1] << 8) | ((unsigned)b[2] << 16) | ((unsigned)b[3] << 24); };
    np[0] = make_uint4(__float_as_uint(plo[0]), __float_as_uint(plo[1]), __float_as_uint(plo[2]),
                       (unsigned)e[0] | ((unsigned)e[1] << 8) | ((unsigned)e[2] << 16) | (n0.w & 0xff000000u));
    np[2] = make_uint4(pack4(qlo[0]), pack4(qlo[0] + 4), pack4(qlo[1]), pack4(qlo[1] + 4));
    np[3] = make_uint4(pack4(qlo[2]), pack4(qlo[2] + 4), pack4(qhi[0]), pack4(qhi[0] + 4));
    np[4] = make_uint4(pack4(qhi[1]), pack4(qhi[1] + 4), pack4(qhi[2]), pack4(qhi[2] + 4));
}

// one launch per level, deepest first: a node reads the boxes of its inner children, refitted by the launch before
template <typename Leaves>
static cudaError_t refit_levels(Bvh8* b, Leaves leaves, cudaStream_t stream) {
    for (int lv = (int)b->n_levels - 1; lv >= 0; lv--) {
        const uint32_t first = b->level_start[lv], count = b->level_start[lv + 1] - first;
        if (count) k_refit_level<Leaves><<<(count + 127) / 128, 128, 0, stream>>>(b->nodes, first, count, leaves);
    }
    return cudaGetLastError();
}

cudaError_t refit_tlas(const float4* d_inst_recs, const float4* d_box_lo, const float4* d_box_hi, uint32_t n_instances, Bvh8* b,
                       cudaStream_t stream) {
    if (!b->nodes || !b->prims || b->n_prims != n_instances || b->n_levels == 0u || b->level_start[b->n_levels] != b->n_nodes)
        return cudaErrorInvalidValue;
    k_refit_prims<<<(n_instances + 255) / 256, 256, 0, stream>>>(d_inst_recs, n_instances, b->prims);
    return refit_levels(b, InstLeafBoxes{b->prims, d_box_lo, d_box_hi}, stream);
}

// ---- BLAS refit (DXR PERFORM_UPDATE) ---------------------------------------------------------------------------------
// leaf order of the triangle records: prims[3k] carries its primitive id in .w (TriSource::write).  Rewrites each record from the new
// vertices and folds its box into the model bounds (the reduction of k_tri_boxes: the padding of the level pass needs them).
__global__ void k_refit_tris(const uint8_t* __restrict__ verts, const uint32_t* __restrict__ idx, uint32_t n, float4* __restrict__ prims,
                             BuildCounters* c) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = k < n;
    float lx = 0, ly = 0, lz = 0, hx = 0, hy = 0, hz = 0;
    if (valid) {
        float4* r = prims + 3 * (size_t)k;
        TriSource{verts, idx}.write(r, __float_as_uint(r[0].w));
        const float4 a = r[0], b = r[1], d = r[2];
        lx = fminf(a.x, fminf(b.x, d.x)); hx = fmaxf(a.x, fmaxf(b.x, d.x));
        ly = fminf(a.y, fminf(b.y, d.y)); hy = fmaxf(a.y, fmaxf(b.y, d.y));
        lz = fminf(a.z, fminf(b.z, d.z)); hz = fmaxf(a.z, fmaxf(b.z, d.z));
    }
    reduce_bounds(c, lx, ly, lz, hx, hy, hz, valid);
}

// the padded model bounds (build_generic's out->lo / hi) into the model's table entries, when they exist, and into out6
__global__ void k_refit_tables(const BuildCounters* c, BlasRef* ref, BlasBounds* bb, float* out6) {
    const float pad = leaf_pad(c);
    for (int k = 0; k < 3; k++) {
        const float l = dec_f(c->bounds[k]) - pad, h = dec_f(c->bounds[3 + k]) + pad;
        out6[k] = l; out6[3 + k] = h;
        if (ref) { ref->lo[k] = l; ref->hi[k] = h; }
        if (bb) { bb->lo[k] = l; bb->hi[k] = h; }
    }
}

cudaError_t refit_blas(const uint8_t* d_vertices, const uint32_t* d_indices, uint32_t n_tris, Bvh8* b, void* d_scratch, BlasRef* d_ref,
                       BlasBounds* d_bounds, float* d_out6, cudaStream_t stream) {
    static_assert(sizeof(BuildCounters) <= 256, "refit_blas: scratch too small");
    if (!b->nodes || !b->prims || b->n_prims != n_tris || b->n_levels == 0u || b->level_start[b->n_levels] != b->n_nodes)
        return cudaErrorInvalidValue;
    if (n_tris == 0) return cudaSuccess;
    BuildCounters* ctr = (BuildCounters*)d_scratch;
    k_init_counters<<<1, 1, 0, stream>>>(ctr);
    k_refit_tris<<<(n_tris + 255) / 256, 256, 0, stream>>>(d_vertices, d_indices, n_tris, b->prims, ctr);
    const cudaError_t e = refit_levels(b, TriLeafBoxes{b->prims, ctr}, stream);
    if (e != cudaSuccess) return e;
    k_refit_tables<<<1, 1, 0, stream>>>(ctr, d_ref, d_bounds, d_out6);
    return cudaGetLastError();
}

bool tlas_fits_one_node(uint32_t n_instances) { return n_instances >= 1u && n_instances <= (uint32_t)SINGLE_NODE_MAX; }

cudaError_t update_tlas_one_node(const float4* d_inst_recs, const float4* d_box_lo, const float4* d_box_hi, uint32_t n_instances, Bvh8* out,
                                 void* d_ctr, cudaStream_t stream) {
    if (!tlas_fits_one_node(n_instances) || !out->nodes || !out->prims) return cudaErrorInvalidValue;
    static_assert(sizeof(BuildCounters) <= 256, "update_tlas_one_node: scratch too small");
    BuildCounters* ctr = (BuildCounters*)d_ctr;
    k_init_counters<<<1, 1, 0, stream>>>(ctr);
    k_box_bounds<<<(n_instances + 255) / 256, 256, 0, stream>>>(d_box_lo, d_box_hi, n_instances, ctr);
    RecSource src{d_inst_recs};
    k_single_node<4, RecSource><<<1, 32, 0, stream>>>(src, d_box_lo, d_box_hi, (int)n_instances, out->nodes, out->prims, ctr);
    out->n_nodes = 1; out->n_prims = n_instances;
    return cudaGetLastError();
}

void free_bvh(Bvh8* b) {
    if (b->nodes) cudaFree(b->nodes);
    if (b->prims) cudaFree(b->prims);
    b->nodes = nullptr; b->prims = nullptr; b->n_nodes = b->n_prims = 0;
}

// ---- instance records: rows of world->object from objectToWorldInverse (binding t3, Renderer.cpp:2091-2121) and the
// world box of each instance (8 corners of the padded BLAS box through the desc's 3x4 objectToWorld).
__global__ void k_instance_records(const rtx_instance_desc* __restrict__ descs, const rtx_instance_props* __restrict__ props,
                                   const BlasBounds* __restrict__ bounds, uint32_t n, float4* __restrict__ recs,
                                   float4* __restrict__ lo, float4* __restrict__ hi) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* m = props[i].objectToWorldInverse;
    recs[4 * i + 0] = make_float4(m[0], m[4], m[8], m[12]);
    recs[4 * i + 1] = make_float4(m[1], m[5], m[9], m[13]);
    recs[4 * i + 2] = make_float4(m[2], m[6], m[10], m[14]);
    const uint32_t blas = (uint32_t)descs[i].blas;
    recs[4 * i + 3] = make_float4(__uint_as_float(blas), __uint_as_float(i), 0.0f, 0.0f);
    const BlasBounds b = bounds[blas];
    float l[3] = {INFINITY, INFINITY, INFINITY}, h[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int k = 0; k < 8; k++) {
        float x = (k & 1) ? b.hi[0] : b.lo[0], y = (k & 2) ? b.hi[1] : b.lo[1], z = (k & 4) ? b.hi[2] : b.lo[2];
        for (int r = 0; r < 3; r++) {
            const float* t = descs[i].transform[r];
            float v = t[0] * x + t[1] * y + t[2] * z + t[3];
            l[r] = fminf(l[r], v); h[r] = fmaxf(h[r], v);
        }
    }
    float s = 0.0f;
    for (int r = 0; r < 3; r++) s = fmaxf(s, fmaxf(fabsf(l[r]), fabsf(h[r])));
    const float pad = s * 3.0517578125e-5f + 1e-30f;
    lo[i] = make_float4(l[0] - pad, l[1] - pad, l[2] - pad, 0.0f);
    hi[i] = make_float4(h[0] + pad, h[1] + pad, h[2] + pad, 0.0f);
}

// Tight world boxes: the extent of the instance's TRANSFORMED VERTICES instead of the 8 corners of its object-space box.
// For a rotated instance the corner box is up to sqrt(3) larger per axis than the geometry; C3 (1000 rotated instances)
// entered 4.4 instances per ray with corner boxes.  TIGHT_CHUNKS CTAs per instance share its vertices (the per-frame TLAS update of
// the 0.5 M-vertex C2 mesh took 1.1 ms with one CTA per instance) and fold their partial extents with order-preserving atomics;
// every vertex of the model's buffer is taken (a superset of the referenced ones, so the box stays conservative); same 2^-15 padding.
#define TIGHT_CHUNKS 64
__global__ void k_tight_init(uint32_t n, unsigned int* __restrict__ acc) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 6u * n) acc[i] = (i % 6u) < 3u ? 0xffffffffu : 0u;
}
__global__ void __launch_bounds__(256)
k_instance_tight_boxes(const rtx_instance_desc* __restrict__ descs, const BlasBounds* __restrict__ bounds, uint32_t n,
                       unsigned int* __restrict__ acc) {
    const uint32_t i = blockIdx.x;          // instance in grid.x (up to 2^31-1), vertex chunk in grid.y
    if (i >= n) return;
    const BlasBounds b = bounds[(uint32_t)descs[i].blas];
    if (blockIdx.y * 256u >= b.n_verts) return;
    float t[3][4];
    for (int r = 0; r < 3; r++) for (int c = 0; c < 4; c++) t[r][c] = descs[i].transform[r][c];
    float l[3] = {INFINITY, INFINITY, INFINITY}, h[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (uint32_t v = blockIdx.y * 256u + threadIdx.x; v < b.n_verts; v += gridDim.y * 256u) {
        const float* p = reinterpret_cast<const float*>(b.verts + (size_t)v * 28);
        const float x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
        for (int r = 0; r < 3; r++) {
            const float w = t[r][0] * x + t[r][1] * y + t[r][2] * z + t[r][3];
            l[r] = fminf(l[r], w); h[r] = fmaxf(h[r], w);
        }
    }
    __shared__ float sl[3][8], sh[3][8];
    for (int r = 0; r < 3; r++) {
        for (int o = 16; o > 0; o >>= 1) { l[r] = fminf(l[r], __shfl_xor_sync(0xffffffffu, l[r], o)); h[r] = fmaxf(h[r], __shfl_xor_sync(0xffffffffu, h[r], o)); }
        if ((threadIdx.x & 31) == 0) { sl[r][threadIdx.x >> 5] = l[r]; sh[r][threadIdx.x >> 5] = h[r]; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int r = 0; r < 3; r++) {
            for (int w = 0; w < 8; w++) { l[r] = fminf(l[r], sl[r][w]); h[r] = fmaxf(h[r], sh[r][w]); }
            atomicMin(&acc[6 * i + r], enc_f(l[r]));
            atomicMax(&acc[6 * i + 3 + r], enc_f(h[r]));
        }
    }
}
__global__ void k_tight_finish(uint32_t n, const unsigned int* __restrict__ acc, float4* __restrict__ lo, float4* __restrict__ hi) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float l[3], h[3];
    for (int r = 0; r < 3; r++) { l[r] = dec_f(acc[6 * i + r]); h[r] = dec_f(acc[6 * i + 3 + r]); }
    float s = 0.0f;
    for (int r = 0; r < 3; r++) s = fmaxf(s, fmaxf(fabsf(l[r]), fabsf(h[r])));
    const float pad = s * 3.0517578125e-5f + 1e-30f;
    // never larger than the corner box already written by k_instance_records
    const float4 cl = lo[i], ch = hi[i];
    lo[i] = make_float4(fmaxf(l[0] - pad, cl.x), fmaxf(l[1] - pad, cl.y), fmaxf(l[2] - pad, cl.z), 0.0f);
    hi[i] = make_float4(fminf(h[0] + pad, ch.x), fminf(h[1] + pad, ch.y), fminf(h[2] + pad, ch.z), 0.0f);
}

cudaError_t launch_instance_records(const rtx_instance_desc* d_descs, const rtx_instance_props* d_props, const BlasBounds* d_bounds,
                                    uint32_t n, float4* d_recs, float4* d_lo, float4* d_hi, unsigned int* d_scratch6, cudaStream_t stream) {
    if (n) {
        k_instance_records<<<(n + 127) / 128, 128, 0, stream>>>(d_descs, d_props, d_bounds, n, d_recs, d_lo, d_hi);
        if (d_scratch6) {
            k_tight_init<<<(6 * n + 255) / 256, 256, 0, stream>>>(n, d_scratch6);
            k_instance_tight_boxes<<<dim3(n, TIGHT_CHUNKS), 256, 0, stream>>>(d_descs, d_bounds, n, d_scratch6);
            k_tight_finish<<<(n + 255) / 256, 256, 0, stream>>>(n, d_scratch6, d_lo, d_hi);
        }
    }
    return cudaGetLastError();
}

}  // namespace rtx
