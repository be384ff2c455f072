/* rtx_b200.h — C ABI of the B200-native wavefront path tracer that replaces the DXR seam of
 * ML200/RoyalTracer-DX (reference paths relative to /root/reference/Pathtracer/).
 *
 * The reference has no plugin/FFI API; the seam is the DXR pipeline interface between
 * rdn/Renderer.cpp (host) and the shader set (SURVEY.md §8b).  Each entry point below names the
 * reference interface it replaces.  All structs are byte-compatible with the reference's GPU
 * structs.  Conventions: extern "C", plain pointers and sizes, integer status (0 = OK) plus
 * rtx_last_error(); a context is not thread-safe (one caller thread, like the reference's
 * WM_PAINT-driven loop, rdn/Win32Application.cpp:100-104); the caller owns every host pointer,
 * the library copies on upload and owns all device memory.  There is no CPU fallback: every
 * entry point that computes fails with RTX_ERR_CUDA if no sm_100 device is usable.
 */
#ifndef RTX_B200_H
#define RTX_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int32_t rtx_status;
#define RTX_OK            0
#define RTX_ERR_ARG       1   /* bad argument (the reference helpers throw std::logic_error) */
#define RTX_ERR_CUDA      2   /* CUDA runtime failure (reference: ThrowIfFailed, rdn/DXSampleHelper.h:17-23) */
#define RTX_ERR_STATE     3   /* call order violated (e.g. render before instances are set) */

typedef struct rtx_ctx rtx_ctx;

/* S1  src/Components/Vertex.h:25-35 == shaders/Common_v7.hlsl:100-103 (28 B) */
typedef struct { float position[3]; float normal_material[4]; } rtx_vertex;
/* S4  src/Components/Vertex.h:14-23 == shaders/Common_v7.hlsl:53-60 (128 B) */
typedef struct { float Kd[4]; float Ks[3]; float Ni; float Ke[3]; float pad0; float Pr_Pm_Ps_Pc[4]; float LUT[16]; } rtx_material;
/* S6  rdn/Renderer.h:275-282 == shaders/Common_v7.hlsl:76-84 (384 B), raw XMMATRIX memory */
typedef struct { float objectToWorld[16], objectToWorldInverse[16], prevObjectToWorld[16], prevObjectToWorldInverse[16],
                 objectToWorldNormal[16], prevObjectToWorldNormal[16]; } rtx_instance_props;
/* S7  rdn/Renderer.h:113-124 == shaders/Common_v7.hlsl:86-97 (80 B) */
typedef struct { float x[3]; float cdf; float y[3]; uint32_t instanceID; float z[3]; float weight;
                 float emission[3]; uint32_t triCount; float total_weight; float pad0[3]; } rtx_light_triangle;
/* S8  shaders/Pass_init_di_v7.hlsl:36-45, filled by rdn/Renderer.cpp:1722-1768 (padded to 512 B) */
typedef struct { float view[16], projection[16], viewI[16], projectionI[16], prevView[16], prevProjection[16];
                 float time; float pad[31]; } rtx_camera_params;
/* T2  D3D12_RAYTRACING_INSTANCE_DESC as filled by rdn/nv_helpers_dx12/TopLevelASGenerator.cpp:181-199 (64 B):
 * 3x4 row-major objectToWorld, InstanceID:24|InstanceMask:8, InstanceContributionToHitGroupIndex:24|Flags:8,
 * and the BLAS handle (here: the model id returned by rtx_upload_model). */
typedef struct { float transform[3][4]; uint32_t instance_id_mask; uint32_t hit_group_flags; uint64_t blas; } rtx_instance_desc;
/* RayDesc (HLSL) and the closest-hit result (InstanceID(), PrimitiveIndex(), RayTCurrent(), barycentrics) */
typedef struct { float origin[3]; float tmin; float direction[3]; float tmax; } rtx_ray;
typedef struct { float t, u, v; uint32_t prim; uint32_t inst; } rtx_hit;      /* inst == 0xFFFFFFFF: miss */

#define RTX_FLAG_JITTER          1u  /* 2 RandomFloat draws before anything else (legacy include/RayGen.hlsl:84-85) */
#define RTX_FLAG_LAMBERT_ONLY    2u  /* strategy probabilities forced to (1,0) (BASELINE config C1) */
#define RTX_FLAG_LEGACY_RR       16u /* rtx_render_pass runs the reference's legacy estimator (include/RayGen.hlsl:60-137 + include/Hit.hlsl:
                                       * RIS-10 NEE with one shadow ray per bounce, MIS on emitter hits, Russian roulette after depth 3);
                                       * cfg.bounces (<= 60) caps the number of closest-hit rays per path */
#define RTX_FLAG_FAST_MATH       32u /* rtx_render_pass (estimator E0) runs the shading stages built with FMA contraction and approximate
                                       * division / sqrt / rsqrt / sincos (-use_fast_math): ~19 % faster on BASELINE config C2, no longer
                                       * bit-identical to the CPU oracle — paths diverge at discrete decisions; the converged image agrees within
                                       * the tolerance tests/test_gpu_parity.py::test_fast_math_mode_converges_to_the_exact_image states.
                                       * Default (flag clear): every float operation in IEEE binary32 source order, bit-exact parity. */
#define RTX_FLAG_RESTIR          8u  /* allocate the reservoir / sample buffers u2..u7 (rdn/Renderer.cpp:1331-1577) for rtx_render_frame */

/* Compile-time #defines of shaders/Common_v7.hlsl:1-28 that BASELINE configs vary, as runtime fields. */
typedef struct {
    uint32_t struct_size;       /* sizeof(rtx_config) */
    int32_t  device;            /* CUDA ordinal */
    uint32_t width, height;     /* rdn/Main.cpp:25 (1920x1080) */
    uint32_t bounces;           /* Common_v7.hlsl:11, default 3 */
    uint32_t nee_samples;       /* Common_v7.hlsl:8,  default 4 */
    uint32_t nee_samples_di;    /* Common_v7.hlsl:9,  default 4 */
    uint32_t flags;             /* RTX_FLAG_*; rtx_create rejects any other bit */
    uint32_t samples_per_pass;  /* paths in flight per DispatchRays-equivalent = W*H*samples_per_pass (>=1) */
    void*    stream;            /* cudaStream_t to run on, NULL = context-owned stream */
} rtx_config;

typedef struct {
    uint64_t closest_rays, shadow_rays, paths;   /* TraceRay-equivalents actually issued since the last reset */
    uint64_t kernel_launches;                    /* launches of this library's own kernels */
    uint64_t nodes_visited, tris_tested, instances_entered;   /* only counted by rtx_trace_stats */
    uint64_t shading_replays;    /* paths the shading stages re-ran with guarded IEEE operations (RTX_OPT_TRACE_STATS only) */
} rtx_counters;

typedef struct {
    uint32_t n_nodes, n_tris;        /* 80-B nodes / 48-B triangles in the BLAS */
    uint64_t bytes;
    float    sah_cost;
    float    build_ms;
} rtx_blas_info;

const char* rtx_last_error(void);
/* replaces Renderer::OnInit's device/pipeline/buffer creation (rdn/Renderer.cpp:44-103, 1026-1188) */
rtx_status rtx_create(const rtx_config* cfg, rtx_ctx** out);
void       rtx_destroy(rtx_ctx*);
/* replaces CreateBottomLevelAS + BuildRaytracingAccelerationStructure (rdn/Renderer.cpp:771-823,
 * nv_helpers_dx12/BottomLevelASGenerator.cpp:97-117,235): one opaque indexed triangle geometry, stride 28.
 * material_id_offset = the model's offset into the global materialIDs (the reference smuggles it as a float in
 * vertex.normal.w, shaders/Hit_v7.hlsl:16-17). */
rtx_status rtx_upload_model(rtx_ctx*, const rtx_vertex* v, uint32_t n_vertices, const uint32_t* indices, uint32_t n_indices,
                            uint32_t material_id_offset, uint32_t* model_id_out);
rtx_status rtx_blas_info_get(rtx_ctx*, uint32_t model_id, rtx_blas_info* out);
/* Deforming meshes (DXR: a BLAS built with ALLOW_UPDATE, then PERFORM_UPDATE): new vertex data for an uploaded model — same vertex
 * count, same index buffer, same material_id_offset (topology changes go through rtx_upload_model).  Both modes update everything
 * derived from the vertices: the model's vertex buffer in place, its triangle records, its node boxes or a new BVH, its closest-hit
 * attribute records, its object-space bounds in the per-model tables, the world boxes of its instances and the TLAS (one-node rewrite,
 * refit or rebuild as rtx_set_instances chooses, over the instance list already set; without instances only the model is updated).
 * Leaf boxes are padded as the builder pads them (2^-15 of the largest absolute coordinate of the NEW bounds), so hits stay those of
 * the brute-force definition in both modes.
 * Stream order: like every entry point, ordered after all passes already queued (pipelined ones included); work queued after the call
 * sees the new geometry, captured pass graphs included (no recapture).  The call does not reset the accumulation (only a view change
 * does) and does not touch the emissive-triangle list: a caller that deforms an emissive model collects and sets it again.
 * Errors: RTX_ERR_ARG before any device work for a null context, an unknown model, a vertex count that differs from the upload, an
 * unknown mode, a null pointer with a nonzero count, and (_device) memory that is not device or managed memory of cfg.device.
 * RTX_UPDATE_REBUILD re-runs the traversal-stack depth check of rtx_set_instances and returns RTX_ERR_STATE as it does. */
#define RTX_UPDATE_REFIT   0u  /* keep the BVH topology, recompute every node box bottom-up (DXR PERFORM_UPDATE).  Child order stays that of
                                * the build: after a large deformation traversal gets slower, not wrong (RTX_UPDATE_REBUILD restores it) */
#define RTX_UPDATE_REBUILD 1u  /* full build over the new positions into new buffers, swapped in for the old ones (restores tree quality);
                                * the old buffers are freed once the stream has passed every user; synchronises the host */
/* from host memory (the call may synchronise the host, like rtx_upload_model) */
rtx_status rtx_update_model(rtx_ctx*, uint32_t model_id, const rtx_vertex* v, uint32_t n_vertices, uint32_t mode);
/* from a device buffer of n_vertices * 28 bytes on the context's device, copied on the context stream.  With RTX_UPDATE_REFIT the call
 * neither synchronises the host nor allocates: the per-frame path of an animated mesh.  The bounds the refit computes are copied back
 * behind an event and read before their next host use (rtx_set_instances, rtx_upload_model's table rebuild, rtx_blas_info_get), which
 * then waits for the refit. */
rtx_status rtx_update_model_device(rtx_ctx*, uint32_t model_id, const void* d_vertices, uint32_t n_vertices, uint32_t mode);
/* binding t4 (rdn/Renderer.cpp:1274-1282) and t5 */
rtx_status rtx_set_material_ids(rtx_ctx*, const uint32_t* ids, uint32_t n);
rtx_status rtx_set_materials(rtx_ctx*, const rtx_material* m, uint32_t n);
/* replaces CreateTopLevelAS / per-frame refit (rdn/Renderer.cpp:831-886,594) and binding t3 (:2091-2121) */
rtx_status rtx_set_instances(rtx_ctx*, const rtx_instance_desc* descs, const rtx_instance_props* props, uint32_t n);
/* binding t6 (rdn/Renderer.cpp:2237-2280) */
rtx_status rtx_set_emissive_triangles(rtx_ctx*, const rtx_light_triangle* l, uint32_t n);
/* binding b0 (rdn/Renderer.cpp:1722-1768); a view change resets the accumulation (Pass_spat_di_v7.hlsl:407-423) */
rtx_status rtx_set_camera(rtx_ctx*, const rtx_camera_params*);
/* replaces the DispatchRays sequence (rdn/Renderer.cpp:611-673): renders samples [first_sample, first_sample+n_samples)
 * of every pixel with estimator E0 and accumulates them (gPermanentData).  Asynchronous and ordered on the context stream: work
 * queued there before the call is seen by the pass, work queued there after the call runs after the pass.  Calls that directly follow
 * each other (and whole frames rtx_set_instances -> rtx_set_camera -> rtx_render_pass -> rtx_read_output_async on a TLAS of <= 8
 * instances) overlap on internal streams; gPermanentData receives them in call order, the results are bit-identical to running them
 * one after the other (RTX_OPT_PASS_PIPELINE, RTX_OPT_FRAME_PIPELINE). */
rtx_status rtx_render_pass(rtx_ctx*, uint32_t first_sample, uint32_t n_samples);
/* One frame of the reference's dispatch sequence (rdn/Renderer.cpp:611-673): DispatchRays RayGen (pass 1, 1 spp, sample
 * index = frame_index) -> RayGen2 (temporal reuse against last frame's reservoirs, reprojected with prevView/prevProjection
 * of rtx_set_camera and prevObjectToWorld of rtx_set_instances) -> RayGen3 (spatial reuse, final shade, accumulation).
 * Needs RTX_FLAG_RESTIR and samples_per_pass == 1.  rtx_reset_restir zero-fills the reservoir history. */
rtx_status rtx_render_frame(rtx_ctx*, uint32_t frame_index);
rtx_status rtx_reset_restir(rtx_ctx*);
/* debug: the *_last reservoir / sample buffers after a frame, 40 floats per pixel (layout: csrc/restir.cu k_restir_dump) */
rtx_status rtx_read_restir(rtx_ctx*, float* out40_per_pixel);
rtx_status rtx_reset_accum(rtx_ctx*);
rtx_status rtx_synchronize(rtx_ctx*);
/* gPermanentData (u1): float4 per pixel, row-major; gOutput slice 0 (u0): RGBA8 */
rtx_status rtx_read_accum(rtx_ctx*, float* host_out);
rtx_status rtx_read_output(rtx_ctx*, uint8_t* rgba8_out);
/* the same without stalling the caller (the reference blocks on its fence every frame, rdn/Renderer.cpp:717-735; a host that keeps
 * one frame in flight overlaps the read-back of frame k with the rendering of frame k+1): resolve + D2H copy are enqueued and the
 * call returns; rtx_wait_output blocks until the image of the last rtx_read_output_async is complete in rgba8_out (pinned memory
 * for a truly asynchronous copy).  rgba8_out must stay valid until then. */
rtx_status rtx_read_output_async(rtx_ctx*, uint8_t* rgba8_out);
rtx_status rtx_wait_output(rtx_ctx*);
/* multi-GPU: the accumulation buffer rtx_read_output* resolves — a device buffer of W*H float4 owned by the caller, typically the
 * destination of the per-pass reduce on rank 0 (SURVEY.md 8e: "rank 0 then runs F20's divide + sRGB"); NULL = the context's own buffer */
rtx_status rtx_set_resolve_source(rtx_ctx*, const void* d_accum_float4);
/* device pointer of gPermanentData, for the per-pass NCCL reduce over NVLink (SURVEY.md §8e) */
rtx_status rtx_accum_device_ptr(rtx_ctx*, void** out);
/* Multi-GPU (SURVEY.md 8e; the reference is single-GPU): the scene is replicated, every rank renders its own samples of the full frame
 * and the accumulation buffers are combined by ONE ncclReduce(sum, fp32, W*H*4, root 0) per progressive pass over NVLink.
 * rtx_comm_unique_id: 128 bytes from ncclGetUniqueId on one rank, handed to the others by the host.  rtx_comm_init: collective;
 * afterwards rank 0's rtx_read_output* resolve the reduced sum.  rtx_reduce_accum: queues the reduce behind everything rendered so far
 * on a side stream; the render stream does not wait (the next pass overlaps it, only its final accumulation waits for the reduce to
 * have read gPermanentData).  NCCL is bound at run time (dlopen of libnccl.so.2). */
rtx_status rtx_comm_unique_id(void* out128);
rtx_status rtx_comm_init(rtx_ctx*, const void* unique_id128, int rank, int world);
rtx_status rtx_reduce_accum(rtx_ctx*);
rtx_status rtx_read_reduced_accum(rtx_ctx*, float* host_out);   /* rank 0: the sum over ranks, float4 per pixel */
rtx_status rtx_comm_destroy(rtx_ctx*);
/* raw TraceRay (T3 closest / T4 any-hit): host buffers, or device buffers with _device */
rtx_status rtx_trace(rtx_ctx*, const rtx_ray* rays, uint32_t n, rtx_hit* out, int any_hit);
rtx_status rtx_trace_device(rtx_ctx*, const void* d_rays, uint32_t n, void* d_hits, int any_hit);
/* like rtx_trace_device but also counts nodes / triangles / instances visited (roofline's B_ray) */
rtx_status rtx_trace_stats(rtx_ctx*, const void* d_rays, uint32_t n, void* d_hits, int any_hit);
rtx_status rtx_get_counters(rtx_ctx*, rtx_counters* out);
rtx_status rtx_reset_counters(rtx_ctx*);
/* device time in ms of the traversal kernels / all kernels of the last rtx_render_pass (CUDA events on the ctx stream) */
rtx_status rtx_last_pass_ms(rtx_ctx*, float* trace_ms, float* total_ms);
/* the same per stage kind (needs RTX_OPT_STAGE_TIMING): ms_by_stage[RTX_STAGE_*] summed over the launches of the last pass */
#define RTX_STAGE_GENERATE 0
#define RTX_STAGE_CLOSEST 1
#define RTX_STAGE_ANY 2
#define RTX_STAGE_SHADE_PRIMARY 3
#define RTX_STAGE_DI_FINISH 4
#define RTX_STAGE_GI_STEP 5
#define RTX_STAGE_SCATTER 6
#define RTX_STAGE_FINALIZE 7
#define RTX_STAGE_ACCUMULATE 8
#define RTX_STAGE_COUNT 9
rtx_status rtx_last_pass_stage_ms(rtx_ctx*, float* ms_by_stage, uint32_t n_stages, float* total_ms);
/* runtime options.  RTX_OPT_TRACE_STATS: closest-hit traversals of rtx_render_pass also count nodes/triangles/instances
 * (instrumented kernel variant: for the roofline's B_ray, never for timed runs), and the shading stages count the paths they
 * replay with guarded IEEE operations (rtx_counters.shading_replays).  RTX_OPT_STAGE_TIMING: record CUDA events
 * around every traversal launch of a pass so that rtx_last_pass_ms can report the traversal share.
 * RTX_OPT_PASS_PARTS: 1..4 path ranges of a pass that run concurrently on separate CUDA streams (default 2; the image
 * does not depend on it; passes with per-launch events, statistics or ReSTIR reuse always run as one part). */
#define RTX_OPT_TRACE_STATS   1u
#define RTX_OPT_STAGE_TIMING  2u
#define RTX_OPT_PASS_PARTS    3u
#define RTX_OPT_TLAS_REBUILD  4u   /* 1: rtx_set_instances always rebuilds the TLAS; 0 (default): it refits the last build when the instance
                                    * list still names the same models (rdn/Renderer.cpp:594 refits every frame) */
/* launch tuning of the traversal kernels (0 = built-in default, the measured optimum; csrc/trace.cu): */
#define RTX_OPT_TRACE_FETCH_TH 5u  /* a warp refills its idle lanes when fewer than this many lanes are still traversing (default 24) */
#define RTX_OPT_TRACE_SCHED    6u  /* phase scheduling thresholds th_tri | th_inst << 8 | th_node << 16 (default 0x060808) */
#define RTX_OPT_TRACE_WAVES    7u  /* persistent grid = SMs x resident CTAs x waves (default 1) */
#define RTX_OPT_QUEUE_LPT       8u  /* 1 (default): closest-hit queues are traced longest-processing-time-first (rays that cross the bounds of the
                                    * scene's large instances before the others); 0: in emission order.  The image does not depend on it. */
#define RTX_OPT_TRACE_CTAS      9u  /* resident CTAs per SM of the persistent traversal grid (0 = default: all the register budget allows) */
#define RTX_OPT_PASS_GRAPH     10u  /* 1 (default): a pass of a static configuration is captured once into a CUDA graph and replayed; 0: plain launches */
#define RTX_OPT_SHADOW_OVERLAP 11u  /* 1 (default): the DI visibility rays of a pass are traced on a side stream beside the indirect bounces; 0: in sequence */
#define RTX_OPT_PART_ROWS      12u  /* concurrent path ranges own interleaved chunks of this many image rows: 0 = contiguous ranges, 1..64, 0xffffffff (default) = chosen per frame size */
#define RTX_OPT_PASS_PIPELINE  13u  /* 1 (default): rtx_render_pass calls that directly follow each other overlap (two sets of pass buffers, accumulation in call order: bit-identical); 0: one pass at a time */
#define RTX_OPT_FRAME_PIPELINE 14u  /* 1 (default): a per-frame loop rtx_set_instances (<= 8 instances, same models) -> rtx_set_camera -> rtx_render_pass -> rtx_read_output_async keeps two sets of per-frame state and overlaps consecutive frames (bit-identical); 0: one frame at a time */
rtx_status rtx_set_option(rtx_ctx*, uint32_t option, uint32_t value);
/* debug: per-pixel record of one sample in the layout of the oracle's orc_debug_pixel (64 floats) */
rtx_status rtx_debug_pixel(rtx_ctx*, uint32_t x, uint32_t y, float* out64);
/* self-test of the device arithmetic (csrc/dmath.cuh): compares every hand-scheduled fast path with the IEEE-754
 * operation it restates over ALL 2^32 binary32 bit patterns on the device.  mismatches_out[0] = d_rsqrt vs 1/sqrt; [2..6] = the
 * unguarded fast paths (result or range flag wrong): sqrt, rcp, rsqrt, a/b on 2^34 pairs, a/3 and a/pi on every a. */
rtx_status rtx_selftest_dmath(rtx_ctx*, uint64_t* mismatches_out, uint32_t n_out);

#ifdef __cplusplus
}
#endif
#endif
