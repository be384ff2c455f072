// trace.cu — persistent-thread traversal kernels (the `extend` and `connect` stages of the wavefront).
//
// One launch drains a whole ray queue: the grid is sized to the machine (148 SMs x resident CTAs), and every
// warp pulls batches of consecutive rays from a global cursor with one atomic per refill.  A warp refills its
// idle lanes as soon as fewer than FETCH_THRESHOLD lanes are still traversing, so long-running incoherent rays do
// not strand the other 31 lanes (B200 has no RT cores; warp-execution efficiency is the second-order term after
// memory latency — see DESIGN.md §Kernels).
#include <algorithm>
using std::max;

#include "trace.h"
#include "traverse.cuh"

namespace rtx {

#ifndef TRACE_BLOCK
#define TRACE_BLOCK 128
#endif
#ifndef RTX_TRACE_MINB
#define RTX_TRACE_MINB (1024 / TRACE_BLOCK)   // resident CTAs per SM the register budget is set for (64 registers, 1024 threads)
#endif
#ifndef FETCH_THRESHOLD
#define FETCH_THRESHOLD 24     // refill the warp's idle lanes when fewer than this many lanes are still traversing
#endif
#ifndef RTX_SCHED_DEFAULT
#define RTX_SCHED_DEFAULT 0x060808   // th_tri | th_inst << 8 | th_node << 16: run the triangle (instance) phase when >= th lanes are parked,
#endif                               // or whenever fewer than th_node lanes have node work left (sweep: profiles/r01_s4_sched_sweep.txt)

// rays are read once and hit records are read a launch later: evict-first loads / stores (__ldcs / __stcs), so that the launch's own
// streaming traffic does not push the BVH out of the L2 (wave_dev.cuh StateView::ld has the numbers)

template <bool ANY_HIT, bool STATS>
__global__ void __launch_bounds__(TRACE_BLOCK, RTX_TRACE_MINB)
trace_kernel(SceneAS S, const float4* __restrict__ o_tmin, const float4* __restrict__ d_tmax,
             const uint32_t* __restrict__ n_ptr, uint32_t n_fixed, unsigned int* __restrict__ cursor,
             float4* __restrict__ hit_a, uint32_t* __restrict__ hit_inst, TraceStats* st, int fetch_th, int sched,
             const uint32_t* __restrict__ order, const uint32_t* __restrict__ n_heavy_ptr, uint32_t cap,
             const uint32_t* __restrict__ vis_pid, float* __restrict__ vis, uint32_t* __restrict__ vmask) {
    // trace order (wavefront.h RayQueue): claim k -> slot order[k] (k < n_heavy) or order[cap-1-(k-n_heavy)]: expensive rays first
    const uint32_t n = n_ptr ? *n_ptr : n_fixed;
    const uint32_t n_heavy = order ? *n_heavy_ptr : 0u;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    uint2 stack[RTX_STACK_SIZE];
    __shared__ uint8_t s_perm[2048];
    __shared__ float4 s_cold[4][TRACE_BLOCK];
    fill_perm_table(s_perm, threadIdx.x, blockDim.x);
    __syncthreads();
    const TravCold C = {&s_cold[0][threadIdx.x], &s_cold[1][threadIdx.x], &s_cold[2][threadIdx.x], &s_cold[3][threadIdx.x]};
    Trav T;
    uint32_t pend = PEND_NONE, leaf_base = 0u, leaf_bits = 0u, leaf_W = 0u;    // a parked leaf group (traverse.cuh)
    const int th_tri = sched & 0xff, th_inst = (sched >> 8) & 0xff, th_node = (sched >> 16) & 0xff;
    bool active = false;
    bool exhausted = (S.n_instances == 0u);
    // Ray claims: a warp claims EXACTLY the rays its idle lanes need, when they need them (one atomic per refill).  Claiming 32 at a time
    // plus one chunk ahead (to hide the atomic's latency) left ~48 unstarted rays in every warp's private pool when the cursor ran out:
    // at 1080p 11 % of a queue sat in private pools while other warps already idled ("queue found drained" 434 .. 547 us of a 638 us
    // launch, profiles/r01_s4_trace_timeline.txt).  Exact claims: closest-hit launches -3.3 % on C2, -4.6 % on C3 (profiles/r02_*).
    unsigned int c_nodes = 0, c_tris = 0, c_insts = 0;

#ifdef RTX_TRACE_TIMELINE
    unsigned long long tl_t0, tl_tex = 0, tl_rays = 0; unsigned tl_steps = 0, tl_drain_steps = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tl_t0));
#endif
    for (;;) {
        // ---- refill idle lanes from the queue
        const unsigned idle = __ballot_sync(0xffffffffu, !active);
        if (idle && !exhausted) {
            const uint32_t need = (uint32_t)__popc(idle);
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(cursor, need);
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base + need >= n) {
                exhausted = true;                                // this claim took the last rays (or came too late)
#ifdef RTX_TRACE_TIMELINE
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tl_tex));
#endif
            }
            const uint32_t mine = base + (uint32_t)__popc(idle & lt_mask);
            if (!active && mine < n) {
                const uint32_t slot = order ? __ldg(order + (mine < n_heavy ? mine : cap - 1u - (mine - n_heavy))) : mine;
                trav_init(T, C, S, __ldcs(o_tmin + slot), __ldcs(d_tmax + slot), slot);
                active = true;
            }
        }
        const unsigned act = __ballot_sync(0xffffffffu, active);
        if (act == 0u) {
            if (exhausted) break;
            continue;
        }
        // ---- traverse until too few lanes are left (or to the end once the queue is drained)
        const int threshold = exhausted ? 1 : fetch_th;
        do {
            if (active && pend == PEND_NONE) {
                trav_node<ANY_HIT, STATS>(T, S, s_perm, stack, leaf_base, leaf_bits, leaf_W, &c_nodes);
                if (leaf_bits) pend = T.blas_sp >= 0 ? PEND_TRI : PEND_INST;
            }
            const unsigned m_tri = __ballot_sync(0xffffffffu, pend == PEND_TRI), m_inst = __ballot_sync(0xffffffffu, pend == PEND_INST);
            const unsigned m_node = __ballot_sync(0xffffffffu, active && pend == PEND_NONE);
            const bool flush = __popc(m_node) < th_node;
            const bool do_tri = m_tri && (flush || __popc(m_tri) >= th_tri);       // warp-uniform
            const bool do_inst = m_inst && (flush || __popc(m_inst) >= th_inst);
            // ONE divergent region for the three kinds of lanes, so that their instruction streams can interleave (a lane that pops does
            // not wait for the triangle loads of its neighbours); the pop/finish tail is therefore written out in both branches
#define RTX_FINISH(FOUND)                                                                                      \
            {                                                                                                  \
                bool done;                                                                                     \
                if (ANY_HIT && (FOUND)) { T.hinst = T.cur_inst; done = true; }                                 \
                else done = trav_pop(T, C, S, stack);                                                          \
                if (done) {                                                                                    \
                    active = false;                                                                            \
                    RTX_WRITE_RESULT                                                                           \
                }                                                                                              \
            }
#define RTX_WRITE_RESULT                                                                                       \
            {                                                                                                  \
                const uint32_t j = __float_as_uint(C.wo->w);                                                   \
                if (!ANY_HIT) { const float4 h = *C.hit; __stcs(hit_a + j, make_float4(T.ht, h.x, h.y, h.z)); } \
                /* any-hit with a visibility array: an occluded ray clears its path's entry (no scatter kernel) */ \
                if (ANY_HIT && vis) { if (T.hinst != 0xFFFFFFFFu) vis[__ldg(vis_pid + j)] = 0.0f; }            \
                /* ... or sets bit (pid & 15) of word pid >> 4 of an occlusion mask (the ReSTIR reuse passes) */   \
                else if (ANY_HIT && vmask) {                                                                   \
                    if (T.hinst != 0xFFFFFFFFu) { const uint32_t pid = __ldg(vis_pid + j); atomicOr(&vmask[pid >> 4], 1u << (pid & 15u)); } \
                }                                                                                              \
                else __stcs(hit_inst + j, T.hinst);                                                            \
            }
            if (pend == PEND_TRI) {
                if (do_tri) {
                    const bool found = trav_tris<ANY_HIT, STATS>(T, C, leaf_base, leaf_bits, leaf_W, &c_tris);
                    pend = PEND_NONE;
                    RTX_FINISH(found)
                }
            } else if (pend == PEND_INST) {
                if (do_inst) {
                    const bool entered = trav_enter_instance<ANY_HIT, STATS>(T, C, S, stack, leaf_base, leaf_bits, leaf_W, &c_insts);
                    if (entered) pend = PEND_NONE;
                    else if (leaf_bits == 0u) {          // every instance of the group rejected: back to the node work (pop if the group is used up)
                        pend = PEND_NONE;
                        RTX_FINISH(false)
                    }                                    // else: stays parked with the remaining instance leaves
                }
            } else if (active) {
                RTX_FINISH(false)
            }
#undef RTX_FINISH
#undef RTX_WRITE_RESULT
#ifdef RTX_TRACE_TIMELINE
            tl_steps++; if (exhausted) tl_drain_steps++;
#endif
        } while (__popc(__ballot_sync(0xffffffffu, active)) >= threshold);
    }
#ifdef RTX_TRACE_TIMELINE
    {
        unsigned long long tl_t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tl_t1));
        const unsigned wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
        if (lane == 0 && (wid % 37u) == 0u && n > 100000u)
            printf("TL %u n %u start %llu exhausted_at %llu end %llu steps %u drain_steps %u\n", wid, n, tl_t0 % 100000000ull,
                   tl_tex ? tl_tex - tl_t0 : 0ull, tl_t1 - tl_t0, tl_steps, tl_drain_steps);
    }
#endif
    if (S.n_instances == 0u) {   // empty scene: everything misses
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
            if (!ANY_HIT) hit_a[i] = make_float4(__ldg(d_tmax + i).w, 0.0f, 0.0f, __uint_as_float(0xFFFFFFFFu));
            if (!(ANY_HIT && (vis || vmask))) hit_inst[i] = 0xFFFFFFFFu;
        }
    }
    // the last CTA to finish leaves the cursor at 0 for the next launch (cursor[1] counts finished CTAs and wraps to 0 by itself)
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicInc(cursor + 1, gridDim.x - 1u) == gridDim.x - 1u) { cursor[0] = 0u; __threadfence(); }
    }
    if (STATS) {
        atomicAdd(&st->nodes, (unsigned long long)c_nodes);
        atomicAdd(&st->tris, (unsigned long long)c_tris);
        atomicAdd(&st->insts, (unsigned long long)c_insts);
    }
}

cudaError_t launch_trace(const SceneAS& S, const float4* o_tmin, const float4* d_tmax, const uint32_t* n_ptr, uint32_t n_fixed,
                         unsigned int* cursor, float4* hit_a, uint32_t* hit_inst, bool any_hit, TraceStats* stats,
                         cudaStream_t stream, int grid_share, const uint32_t* order, const uint32_t* n_heavy_ptr, uint32_t cap,
                         const uint32_t* vis_pid, float* vis, uint32_t* vmask) {
    // `cursor` = two words, both 0 between launches: [0] the ray cursor, [1] the count of finished CTAs; the last CTA of a launch
    // resets [0] (and atomicInc wraps [1]), so no memset precedes the launch.
    const int sms = S.num_sms > 0 ? S.num_sms : 148;
    // persistent: the resident CTAs of the machine, or this launch's share of them when several traversals run concurrently
    // (wave_render_pass: the parts' kernels are then co-resident and one part's drain phase overlaps the other's work)
    const int grid = max(sms, sms * RTX_TRACE_MINB / max(grid_share, 1));
    // (run-time kernel arguments on purpose: folded into compile-time constants they reschedule most of trace_kernel's SASS)
    const int fetch_th = FETCH_THRESHOLD, sched = RTX_SCHED_DEFAULT;
    if (stats) {
        if (any_hit) trace_kernel<true, true><<<grid, TRACE_BLOCK, 0, stream>>>(S, o_tmin, d_tmax, n_ptr, n_fixed, cursor, hit_a, hit_inst, stats, fetch_th, sched, order, n_heavy_ptr, cap, vis_pid, vis, vmask);
        else trace_kernel<false, true><<<grid, TRACE_BLOCK, 0, stream>>>(S, o_tmin, d_tmax, n_ptr, n_fixed, cursor, hit_a, hit_inst, stats, fetch_th, sched, order, n_heavy_ptr, cap, vis_pid, vis, vmask);
    } else {
        if (any_hit) trace_kernel<true, false><<<grid, TRACE_BLOCK, 0, stream>>>(S, o_tmin, d_tmax, n_ptr, n_fixed, cursor, hit_a, hit_inst, nullptr, fetch_th, sched, order, n_heavy_ptr, cap, vis_pid, vis, vmask);
        else trace_kernel<false, false><<<grid, TRACE_BLOCK, 0, stream>>>(S, o_tmin, d_tmax, n_ptr, n_fixed, cursor, hit_a, hit_inst, nullptr, fetch_th, sched, order, n_heavy_ptr, cap, vis_pid, vis, vmask);
    }
    return cudaGetLastError();
}

}  // namespace rtx
