// wavefront.h — host interface of the wavefront stages (generate / shade / connect / accumulate).
#pragma once
#include "common.cuh"
#include "shade.cuh"
#include "trace.h"

namespace rtx {

// Structure-of-arrays path state: NSTATE float4 planes of n_paths entries each (DESIGN.md §"Data layout in HBM").
enum StatePlane {
    SP_X1 = 0,      // x1.xyz (payload.hitPosition), bits(mID)
    SP_N1,          // payload.hitNormal.xyz, -  (legacy estimator: bits(seed.x))
    SP_O,           // o = -direction, -  (legacy estimator: bits(seed.y))
    SP_DI_X2,       // reservoir.x2, w_sum
    SP_DI_N2,       // reservoir.n2, f_g
    SP_DI_L2,       // reservoir.L2 (binary16 values), -
    SP_DI_R,        // ReconnectDI(x1,n1,x2,n2,L2,o) vector, -
    SP_GI_XN,       // reservoir_GI.xn, - (k_finalize: w_sum after the visibility test)
    SP_GI_NN,       // reservoir_GI.nn, -
    SP_GI_E3,       // reservoir_GI.E3 (binary16 values), -
    SP_ORIGIN,      // path origin, pdf of the BSDF ray in flight
    SP_ACC_F,       // acc_f incl. the ray in flight, -  (legacy estimator: colour, pdf)
    SP_ACC_FR,      // acc_f_reconnection incl. the ray in flight, -
    SP_SH1,         // x1_shadow, flag (1 = a reservoir winner exists)
    SP_SH2,         // x2_shadow, -
    SP_RESULT,      // per-sample radiance C, flag (1 = sampling path: finalize computes C)
    SP_GI_SC,       // scalars of the GI reservoir, updated every bounce: w_sum, acc_pdf, 1 = a sample was accepted, -
    NSTATE
};

// Ray queue: slots are claimed in emission order (warp-compacted, so the path ids of a queue stay in pixel order and the shading stages'
// structure-of-arrays state accesses stay coalesced).  A queue can carry a TRACE ORDER beside it (wave_dev.cuh push_ray2): order[] holds
// slot indices, those of rays expected to be expensive ("heavy": their segment crosses the bounds of the scene's large instances) from
// entry 0 upwards, the others from entry cap-1 downwards.  The persistent traversal kernel claims order entries front to back, i.e. it
// starts the long rays first and the queue runs out among the short ones (longest-processing-time-first: what the last-started long rays
// leave behind was a third of a 1080p launch); hit records land in the ray's own slot.  order == nullptr: traced in slot order.
// (Filling the QUEUE itself from both ends was measured first: traversal -12 %, but the shading stage then reads its state at a fifth of
// the density for the heavy rays: k_gi_step 3.66 -> 6.05 ms per C2 pass; an array-of-structures state made that order-independent at
// 4.15 ms and cost the streaming stages 3x — profiles/r02_lpt_queue_layouts.txt.)
struct RayQueue {
    float4* o_tmin; float4* d_tmax; uint32_t* pid; uint32_t* count;   // count lives on the device
    uint32_t* order; uint32_t* n_heavy; uint32_t* n_light; uint32_t cap;
};

#define WAVE_MAX_PARTS 4
// One lane's pass buffers (api.cu: a context has two).  gPermanentData and gOutput belong to the context.
struct WaveBuffers {
    uint32_t n_paths = 0;
    int parts = 2;                     // path ranges of a pass that run concurrently on separate streams (wave_render_pass)
    cudaStream_t aux[WAVE_MAX_PARTS - 1] = {}; cudaEvent_t ev_fork = nullptr, ev_join[WAVE_MAX_PARTS - 1] = {};
    // the DI visibility rays of a part are traced on a side stream, beside the part's indirect bounces (they are only read by k_finalize):
    // their persistent CTAs take the SM slots the closest-hit launches leave idle while their last long rays drain
    cudaStream_t aux_sh[WAVE_MAX_PARTS] = {}; cudaEvent_t ev_sh_fork[WAVE_MAX_PARTS] = {}, ev_sh_join[WAVE_MAX_PARTS] = {};
    float4* state = nullptr;           // NSTATE * n_paths
    uint2* seeds = nullptr;            // n_paths: RNG state (StateView::seed)
    RayQueue q[2];                     // closest-hit ray queues (ping-pong)
    RayQueue sq[2];                    // shadow queues: [0] DI visibility, [1] GI reservoir winner
    float4* hit_a = nullptr; uint32_t* hit_inst = nullptr;    // hit records of the queue just traced
    float* vis_di = nullptr; float* vis_gi = nullptr;         // per path, 1 = visible
    uint32_t* counts = nullptr;        // 4 queue counters + scratch
    unsigned int* cursor = nullptr;    // 4 words per part (launch_trace)
    unsigned long long* ray_counters = nullptr;   // [0] closest, [1] shadow, [2] paths
    uint32_t* first_sample = nullptr;  // device word: the sample index of the pass being rendered (k_generate reads it)
    // CUDA graph of a pass (wavefront.cu wave_render_pass): replayed while the configuration (graph_key) stays what was captured
    struct GraphSlot { cudaGraphExec_t exec = nullptr; uint64_t launches = 0, last_used = 0; unsigned char key[512] = {}; };
    bool use_graph = true, have_last_key = false; GraphSlot graphs[4]; uint64_t graph_clock = 0;
    unsigned char last_key[512] = {};
    float4* accum = nullptr;           // gPermanentData, borrowed from the context (wave_free leaves it alone)
    rtx_camera_params* cam = nullptr;  // b0 (device copy)
    float* debug = nullptr;            // 64 floats
};

// the pass buffers for spp samples of a width x height frame, accumulating into `accum`
cudaError_t wave_alloc(WaveBuffers* B, float4* accum, uint32_t width, uint32_t height, uint32_t spp);
void wave_free(WaveBuffers* B);

#define WAVE_MAX_EVENTS 96
// stage kinds of rtx_last_pass_stage_ms (include/rtx_b200.h RTX_STAGE_*)
enum StageKind { SK_GENERATE = 0, SK_CLOSEST, SK_ANY, SK_SHADE_PRIMARY, SK_DI_FINISH, SK_GI_STEP, SK_SCATTER, SK_FINALIZE, SK_ACCUMULATE, SK_COUNT };
struct PassTiming {
    cudaEvent_t ev[WAVE_MAX_EVENTS] = {};   // [0],[1] bracket the pass; with stage_timing, ev[2+i] is recorded before launch i
    unsigned char kind[WAVE_MAX_EVENTS] = {};
    int n_marks = 0;
    bool stage_timing = false;
    TraceStats* stats = nullptr;       // non-null: use the counting traversal variant
};

// One DispatchRays-equivalent: samples [first_sample, first_sample + spp) of every pixel.
// reduce: null, or the event of a multi-GPU reduce that may still read gPermanentData (the final k_accumulate waits for it).
// parts_override > 0: that many path ranges instead of B.parts.  defer_accumulate: everything but the final k_accumulate (the caller
// launches wave_accumulate itself, behind whatever has to touch gPermanentData first: api.cu pipelines consecutive passes that way).
cudaError_t wave_render_pass(WaveBuffers& B, const SceneData& S, const SceneAS& AS, uint32_t first_sample, uint32_t spp,
                             cudaStream_t stream, uint64_t* launches, PassTiming* timing, cudaEvent_t reduce, bool accumulate = true,
                             int parts_override = 0, bool defer_accumulate = false);
// the same stage sequence built with fast math (wavefront.cu compiled with -DRTX_FAST_MATH): RTX_FLAG_FAST_MATH
namespace fast {
cudaError_t wave_render_pass(WaveBuffers& B, const SceneData& S, const SceneAS& AS, uint32_t first_sample, uint32_t spp,
                             cudaStream_t stream, uint64_t* launches, PassTiming* timing, cudaEvent_t reduce, bool accumulate = true,
                             int parts_override = 0, bool defer_accumulate = false);
}
// The reference's legacy estimator (include/RayGen.hlsl + include/Hit.hlsl) as a wavefront: legacy.cu.  S.bounces caps the path length.
cudaError_t wave_render_pass_legacy(WaveBuffers& B, const SceneData& S, const SceneAS& AS, uint32_t first_sample, uint32_t spp,
                                    cudaStream_t stream, uint64_t* launches, PassTiming* timing);
// wave_alloc / wave_free and the functions below are compiled once (wave_common.cu), whichever build rendered the pass.
cudaError_t wave_accumulate(WaveBuffers& B, uint32_t npx, uint32_t spp, cudaStream_t stream);   // k_accumulate over SP_RESULT
// gOutput (RGBA8) of the accumulation buffer `accum`
cudaError_t wave_resolve(const float4* accum, uint8_t* output, uint32_t n_pixels, cudaStream_t stream, uint64_t* launches);
cudaError_t wave_selftest_dmath(cudaStream_t stream, unsigned long long* host_out, uint32_t n_out);
cudaError_t wave_debug_pixel(WaveBuffers& B, const SceneData& S, uint32_t x, uint32_t y, cudaStream_t stream, float* host_out64);

}  // namespace rtx
