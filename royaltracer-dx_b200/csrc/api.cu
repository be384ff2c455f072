// api.cu — the C ABI (include/rtx_b200.h): context, scene upload, acceleration-structure builds, render passes.
// Plays the role of the DXR runtime + pipeline state behind rdn/Renderer.cpp's calls (SURVEY.md §8b).
#include <dlfcn.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "restir.h"
#include <stdlib.h>

#include "trace.h"
#include "wavefront.h"

namespace rtx {
static thread_local std::string g_err;
void set_error(const std::string& s) { g_err = s; }
}  // namespace rtx

using namespace rtx;

struct ModelRec {
    uint8_t* d_verts = nullptr; uint32_t* d_idx = nullptr; float4* d_shade = nullptr;
    uint32_t n_verts = 0, n_tris = 0, mat_offset = 0;
    Bvh8 bvh;
    // a refit leaves the new padded bounds on the device; their copy lands in this pinned block (6 floats) behind rtx_ctx::ev_bounds and
    // reaches bvh.lo / hi before the next host use of them (sync_host_bounds)
    float* h_bounds = nullptr; bool bounds_pending = false;
};

struct rtx_ctx {
    rtx_config cfg;
    cudaStream_t stream = nullptr; bool own_stream = false;
    std::vector<ModelRec> models;
    uint32_t* d_material_ids = nullptr; uint32_t n_material_ids = 0;
    rtx_material* d_materials = nullptr; uint32_t n_materials = 0;
    // The per-frame instance state (rdn/Renderer.cpp:594: the TLAS is refitted every frame) of the n_instances instances.  Its buffers
    // are kept between calls and the host arrays go through a ring of two pinned staging blocks, so that rtx_set_instances neither
    // allocates nor synchronises.  fs[0] grows on demand; fs[1] is lane 1's set of a pipelined frame loop (below), allocated once for
    // SINGLE_NODE_INSTANCES.
    struct FrameSet {
        rtx_instance_desc* d_descs = nullptr; rtx_instance_props* d_props = nullptr; uint32_t* d_inst_model = nullptr;
        float4* d_inst_recs = nullptr; float4 *d_box_lo = nullptr, *d_box_hi = nullptr; unsigned int* d_box6 = nullptr;
        size_t cap = 0;                     // instances the arrays above are sized for (d_inst_recs: 4 float4, d_box6: 6 words each)
        Bvh8 tlas; size_t tlas_cap = 0;     // instance records tlas.prims has room for
        void* d_tlas_ctr = nullptr;         // 256 B of TLAS build scratch
    } fs[2];
    uint32_t n_instances = 0;
    std::vector<uint32_t> tlas_models;      // instance -> model of the TLAS currently built (a refit needs the same)
    bool force_tlas_rebuild = false;        // RTX_OPT_TLAS_REBUILD: rebuild instead of refitting
    struct Stage { void* p = nullptr; size_t cap = 0; cudaEvent_t ev = nullptr; bool pending = false; } stage[2];
    int stage_i = 0;
    cudaStream_t copy_stream = nullptr; cudaEvent_t ev_resolved = nullptr, ev_copied = nullptr; bool copy_pending = false;
    BlasRef* d_blas = nullptr; BlasBounds* d_bounds = nullptr; ModelRef* d_model_refs = nullptr; uint32_t n_tables = 0;
    rtx_light_triangle* d_lights = nullptr; uint32_t n_lights = 0;
    rtx_camera_params cam; bool have_cam = false;
    WaveBuffers wb; bool wb_ready = false;
    RestirBuffers rs; bool rs_ready = false;
    float4* d_trace_o = nullptr; float4* d_trace_d = nullptr; float4* d_trace_ha = nullptr; uint32_t* d_trace_hi = nullptr;
    rtx_hit* d_trace_out = nullptr; uint32_t trace_cap = 0;
    TraceStats* d_stats = nullptr;
    void* d_refit = nullptr;                // 256 B: BLAS refit scratch (BuildCounters), the refitted bounds at byte 128
    cudaEvent_t ev_bounds = nullptr; bool bounds_pending = false;   // behind the last refit's bounds copy (ModelRec::h_bounds)
    unsigned int* d_overflow = nullptr;     // raised by a traversal whose stack overflowed (SceneAS::overflow); checked + cleared by check_overflow
    unsigned int* h_overflow = nullptr;     // pinned copy written behind every asynchronous read-back (rtx_wait_output looks at it)
    void* d_trace_rays = nullptr; size_t cap_trace_rays = 0; void* d_trace_hits = nullptr; size_t cap_trace_hits = 0;   // rtx_trace staging
    size_t cap_material_ids = 0, cap_materials = 0, cap_lights = 0;
    int num_sms = 148, fetch_th = 0, sched = 0, waves = 0, ctas_per_sm = 0;     // traversal launch tuning (0 = the built-in defaults, trace.cu)
    // multi-GPU (rtx_comm_init): one NCCL reduce of gPermanentData per progressive pass, on the side stream (SURVEY.md 8e)
    void* comm = nullptr; int comm_rank = 0, comm_world = 1;
    float4* d_total = nullptr;              // root only: the sum over ranks; rtx_read_output* resolve it
    cudaEvent_t ev_pass = nullptr, ev_reduced = nullptr;
    float heavy_lo[3] = {0, 0, 0}, heavy_hi[3] = {0, 0, 0}; bool heavy_valid = false, lpt = true;   // SceneData::heavy_* (queue order only)
    uint64_t launches = 0;
    PassTiming timing;
    bool trace_stats = false;
    bool pass_timed = false;
    // Pipelined passes (RTX_OPT_PASS_PIPELINE): rtx_render_pass calls that follow each other with no other call in between alternate
    // between two sets of pass buffers ("lanes": wb and wb2) on two private streams, each pass as ONE path range, so that the start and
    // the tail of a pass overlap the middle of the other one.  gPermanentData is shared: the k_accumulate launches are chained through
    // ev_acc in call order, so the sums are bit-identical to passes run one after the other.  The API stays stream-ordered: a lane
    // starts behind ev_state (whatever other entry points queued on the caller's stream), and the caller's stream is made to wait for
    // every pass's accumulation (no host wait).  The first pass after any other call runs as before (B.parts path ranges on the
    // caller's stream).
    // Pipelined FRAMES (RTX_OPT_FRAME_PIPELINE): a per-frame loop in the reference's order — rtx_set_instances, rtx_set_camera,
    // rtx_render_pass, rtx_read_output_async — with a TLAS that fits one node (<= 8 instances: BASELINE config C2) keeps two sets of the
    // per-frame state (fs[0] and fs[1], and the camera blocks), one per lane: the calls of frame k+1 write the set of the lane frame k-1
    // used and queue on that lane's stream, so frame k+1 starts under the tail of frame k.  Every other call pattern takes the plain
    // path above (enter() first copies fs[1] back into fs[0] if it is the newer one).
    bool frame_pipeline = true, frame_seq_ok = false, resolve_pending = false;
    cudaEvent_t ev_fset = nullptr; bool fset_pending = false;       // behind the last fast rtx_set_instances / rtx_set_camera on a lane stream
    int pending_lane = -1;              // >= 0: the fast rtx_set_instances of this frame prepared that lane
    int cur_set = 0;                    // which set of per-frame instance state (fs) is the newest
    int lane_read_set[2] = {0, 0};      // the set the last pass of each lane read
    int cam_version = 0, cam_block_version[2] = {0, 0};   // the camera blocks of the two lanes (wb.cam, wb2.cam) against the latest rtx_set_camera
    WaveBuffers wb2; bool wb2_ready = false, wb2_refused = false;
    cudaStream_t lane_stream[2] = {nullptr, nullptr}; cudaEvent_t ev_acc[2] = {nullptr, nullptr}, ev_state = nullptr;
    PassTiming timing2;
    bool pipeline = true, in_sequence = false, main_dirty = true, reduce_pending = false;
    int last_lane = 0;
};

static rtx_status fail(rtx_status code, const char* msg) { set_error(msg); return code; }

// Every entry point except rtx_render_pass, rtx_reduce_accum and rtx_synchronize starts here: the device is made current, and a sequence of pipelined
// passes ends (the caller's stream already waits for every pass queued so far; what this call queues there is ordered before the
// passes that follow through ev_state).
static rtx_status sync_frame_state(rtx_ctx* c);
static rtx_status enter(rtx_ctx* c) {
    RTX_CK(cudaSetDevice(c->cfg.device));
    c->in_sequence = false; c->main_dirty = true; c->frame_seq_ok = false; c->pending_lane = -1;
    if (c->fset_pending) { RTX_CK(cudaStreamWaitEvent(c->stream, c->ev_fset, 0)); c->fset_pending = false; }   // a prepared frame that was never rendered
    return sync_frame_state(c);
}
#define RTX_ENTER(c) do { const rtx_status e__ = enter(c); if (e__ != RTX_OK) return e__; } while (0)

extern "C" const char* rtx_last_error(void) { return g_err.c_str(); }

extern "C" void rtx_destroy(rtx_ctx* c);
extern "C" rtx_status rtx_comm_destroy(rtx_ctx* c);
static rtx_status create_resources(rtx_ctx* c) {
    if (c->cfg.stream) c->stream = (cudaStream_t)c->cfg.stream;
    else { RTX_CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)); c->own_stream = true; }
    for (int i = 0; i < WAVE_MAX_EVENTS; i++) RTX_CK(cudaEventCreate(&c->timing.ev[i]));
    for (int i = 0; i < 2; i++) RTX_CK(cudaEventCreate(&c->timing2.ev[i]));
    for (int i = 0; i < 2; i++) RTX_CK(cudaEventCreateWithFlags(&c->ev_acc[i], cudaEventDisableTiming));
    RTX_CK(cudaEventCreateWithFlags(&c->ev_state, cudaEventDisableTiming));
    RTX_CK(cudaEventCreateWithFlags(&c->ev_fset, cudaEventDisableTiming));
    for (int i = 0; i < 2; i++) RTX_CK(cudaStreamCreateWithFlags(&c->lane_stream[i], cudaStreamNonBlocking));
    RTX_CK(cudaMalloc((void**)&c->d_stats, sizeof(TraceStats)));
    RTX_CK(cudaMemset(c->d_stats, 0, sizeof(TraceStats)));
    RTX_CK(cudaMalloc((void**)&c->d_overflow, sizeof(unsigned int)));
    RTX_CK(cudaMemset(c->d_overflow, 0, sizeof(unsigned int)));
    RTX_CK(cudaMallocHost((void**)&c->h_overflow, sizeof(unsigned int)));
    *c->h_overflow = 0u;
    RTX_CK(cudaMalloc(&c->d_refit, 256));
    RTX_CK(cudaEventCreateWithFlags(&c->ev_bounds, cudaEventDisableTiming));
    return RTX_OK;
}

extern "C" rtx_status rtx_create(const rtx_config* cfg, rtx_ctx** out) {
    if (!cfg || !out) return fail(RTX_ERR_ARG, "rtx_create: null argument");
    if (cfg->struct_size != sizeof(rtx_config)) return fail(RTX_ERR_ARG, "rtx_create: rtx_config.struct_size mismatch");
    if (cfg->width == 0 || cfg->height == 0) return fail(RTX_ERR_ARG, "rtx_create: zero-sized image");
    if (cfg->flags & ~(RTX_FLAG_JITTER | RTX_FLAG_LAMBERT_ONLY | RTX_FLAG_RESTIR | RTX_FLAG_LEGACY_RR | RTX_FLAG_FAST_MATH))
        return fail(RTX_ERR_ARG, "rtx_create: unknown flags (valid: RTX_FLAG_JITTER | RTX_FLAG_LAMBERT_ONLY | RTX_FLAG_RESTIR | RTX_FLAG_LEGACY_RR | RTX_FLAG_FAST_MATH)");
    // every path range owns a block of 128 queue counters of which the indirect queues take 5 + bounces (wavefront.cu); the legacy
    // estimator keeps its per-bounce bookkeeping in 64 slots (legacy.cu)
    if ((cfg->flags & RTX_FLAG_LEGACY_RR) ? cfg->bounces > 60u : cfg->bounces > 120u)
        return fail(RTX_ERR_ARG, "rtx_create: bounces out of range (<= 120, <= 60 with RTX_FLAG_LEGACY_RR)");
    int ndev = 0;
    RTX_CK(cudaGetDeviceCount(&ndev));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(RTX_ERR_CUDA, "rtx_create: no such CUDA device (no CPU fallback exists)");
    RTX_CK(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    RTX_CK(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major < 10) return fail(RTX_ERR_CUDA, "rtx_create: kernels are built for sm_100a only");
    rtx_ctx* c = new rtx_ctx();
    c->cfg = *cfg;
    if (c->cfg.samples_per_pass == 0) c->cfg.samples_per_pass = 1;
    c->num_sms = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
    memset(&c->cam, 0, sizeof c->cam);
    const rtx_status st = create_resources(c);
    if (st != RTX_OK) { const std::string keep = g_err; rtx_destroy(c); g_err = keep; return st; }     // nothing leaks on a failed create
    *out = c;
    return RTX_OK;
}

static void free_tables(rtx_ctx* c) {
    if (c->d_blas) cudaFree(c->d_blas);
    if (c->d_bounds) cudaFree(c->d_bounds);
    if (c->d_model_refs) cudaFree(c->d_model_refs);
    c->d_blas = nullptr; c->d_bounds = nullptr; c->d_model_refs = nullptr; c->n_tables = 0;
}

static void free_frame_set(rtx_ctx::FrameSet& f) {
    void* p[] = {f.d_descs, f.d_props, f.d_inst_model, f.d_inst_recs, f.d_box_lo, f.d_box_hi, f.d_box6, f.d_tlas_ctr};
    for (void* q : p) if (q) cudaFree(q);
    free_bvh(&f.tlas);
}

extern "C" void rtx_destroy(rtx_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->cfg.device);
    for (int i = 0; i < 2; i++) if (c->lane_stream[i]) cudaStreamSynchronize(c->lane_stream[i]);
    if (c->stream) cudaStreamSynchronize(c->stream);
    rtx_comm_destroy(c);
    for (auto& m : c->models) {
        if (m.d_verts) cudaFree(m.d_verts); if (m.d_idx) cudaFree(m.d_idx); if (m.d_shade) cudaFree(m.d_shade); free_bvh(&m.bvh);
        if (m.h_bounds) cudaFreeHost(m.h_bounds);
    }
    void* ptrs[] = {c->d_material_ids, c->d_materials, c->d_lights, c->d_trace_o, c->d_trace_d, c->d_trace_ha, c->d_trace_hi,
                    c->d_trace_out, c->d_stats, c->d_overflow, c->d_trace_rays, c->d_trace_hits, c->d_refit};
    for (void* p : ptrs) if (p) cudaFree(p);
    if (c->h_overflow) cudaFreeHost(c->h_overflow);
    for (auto& f : c->fs) free_frame_set(f);
    free_tables(c);
    if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
    if (c->ev_resolved) cudaEventDestroy(c->ev_resolved);
    if (c->ev_copied) cudaEventDestroy(c->ev_copied);
    for (auto& sg : c->stage) { if (sg.p) cudaFreeHost(sg.p); if (sg.ev) cudaEventDestroy(sg.ev); }
    if (c->wb2_ready) wave_free_lane(&c->wb2);
    if (c->wb_ready) wave_free(&c->wb);
    if (c->rs_ready) restir_free(&c->rs);
    for (int i = 0; i < WAVE_MAX_EVENTS; i++) if (c->timing.ev[i]) cudaEventDestroy(c->timing.ev[i]);
    for (int i = 0; i < 2; i++) { if (c->timing2.ev[i]) cudaEventDestroy(c->timing2.ev[i]); if (c->ev_acc[i]) cudaEventDestroy(c->ev_acc[i]); }
    if (c->ev_state) cudaEventDestroy(c->ev_state);
    if (c->ev_fset) cudaEventDestroy(c->ev_fset);
    if (c->ev_bounds) cudaEventDestroy(c->ev_bounds);
    for (int i = 0; i < 2; i++) if (c->lane_stream[i]) cudaStreamDestroy(c->lane_stream[i]);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

// host array -> device buffer; the buffer is reallocated only when it has to grow (*cap, in elements; nullptr = always fresh)
template <typename T>
static rtx_status upload(T** dptr, const T* host, size_t n, cudaStream_t s, size_t* cap = nullptr) {
    const size_t want = n ? n : 1;
    if (!*dptr || !cap || *cap < want) {
        if (*dptr) { RTX_CK(cudaStreamSynchronize(s)); cudaFree(*dptr); *dptr = nullptr; }
        RTX_CK(cudaMalloc((void**)dptr, want * sizeof(T)));
        if (cap) *cap = want;
    }
    if (n) RTX_CK(cudaMemcpyAsync(*dptr, host, n * sizeof(T), cudaMemcpyHostToDevice, s));
    RTX_CK(cudaStreamSynchronize(s));       // the caller's (pageable) array may be reused as soon as the call returns
    return RTX_OK;
}

// closest-hit attribute records (shade.cuh ModelRef::shade): positions and normals of a triangle's three vertices in one 80-byte record
__global__ void k_shade_records(const uint8_t* __restrict__ verts, const uint32_t* __restrict__ idx, uint32_t n_tris, float4* __restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tris) return;
    const float* a = reinterpret_cast<const float*>(verts + (size_t)idx[3 * t] * 28);
    const float* b = reinterpret_cast<const float*>(verts + (size_t)idx[3 * t + 1] * 28);
    const float* d = reinterpret_cast<const float*>(verts + (size_t)idx[3 * t + 2] * 28);
    float4* o = out + (size_t)t * 5;
    o[0] = make_float4(a[0], a[1], a[2], a[3]);
    o[1] = make_float4(b[0], b[1], b[2], a[4]);
    o[2] = make_float4(d[0], d[1], d[2], a[5]);
    o[3] = make_float4(b[3], b[4], b[5], 0.0f);
    o[4] = make_float4(d[3], d[4], d[5], 0.0f);
}

extern "C" rtx_status rtx_upload_model(rtx_ctx* c, const rtx_vertex* v, uint32_t nv, const uint32_t* idx, uint32_t ni,
                                       uint32_t material_id_offset, uint32_t* model_id_out) {
    if (!c || (!v && nv) || (!idx && ni)) return fail(RTX_ERR_ARG, "rtx_upload_model: null argument");
    if (ni % 3) return fail(RTX_ERR_ARG, "rtx_upload_model: index count is not a multiple of 3");
    for (uint32_t i = 0; i < ni; i++) if (idx[i] >= nv) return fail(RTX_ERR_ARG, "rtx_upload_model: index out of range");
    RTX_ENTER(c);
    ModelRec m;
    m.n_verts = nv; m.n_tris = ni / 3; m.mat_offset = material_id_offset;
    rtx_status st;
    if ((st = upload((rtx_vertex**)&m.d_verts, v, nv, c->stream)) != RTX_OK) return st;
    if ((st = upload(&m.d_idx, idx, ni, c->stream)) != RTX_OK) return st;
    RTX_CK(build_blas(m.d_verts, nv, m.d_idx, m.n_tris, &m.bvh, c->stream));
    RTX_CK(cudaMalloc((void**)&m.d_shade, (size_t)(m.n_tris ? m.n_tris : 1) * 80));
    RTX_CK(cudaMallocHost((void**)&m.h_bounds, 6 * sizeof(float)));
    if (m.n_tris) k_shade_records<<<(m.n_tris + 255) / 256, 256, 0, c->stream>>>(m.d_verts, m.d_idx, m.n_tris, m.d_shade);
    RTX_CK(cudaGetLastError());
    c->launches += 9;
    c->models.push_back(m);
    // the per-model tables are rebuilt by the next rtx_set_instances; until then there is no valid TLAS (rendering or tracing in
    // between returns RTX_ERR_STATE instead of handing freed tables to the kernels)
    free_tables(c);
    c->n_instances = 0; c->tlas_models.clear();
    if (model_id_out) *model_id_out = (uint32_t)c->models.size() - 1;
    return RTX_OK;
}

// The host copies of the bounds that refits left on the device (ModelRec::h_bounds) become bvh.lo / hi.  Every host use of a model's
// bounds goes through here first: a stale copy would put the old bounds back into d_blas and the traversal would cull real hits.
static rtx_status sync_host_bounds(rtx_ctx* c) {
    if (!c->bounds_pending) return RTX_OK;
    RTX_CK(cudaEventSynchronize(c->ev_bounds));
    for (ModelRec& m : c->models) {
        if (!m.bounds_pending) continue;
        for (int k = 0; k < 3; k++) { m.bvh.lo[k] = m.h_bounds[k]; m.bvh.hi[k] = m.h_bounds[3 + k]; }
        m.bounds_pending = false;
    }
    c->bounds_pending = false;
    return RTX_OK;
}

extern "C" rtx_status rtx_blas_info_get(rtx_ctx* c, uint32_t model_id, rtx_blas_info* out) {
    if (!c || !out || model_id >= c->models.size()) return fail(RTX_ERR_ARG, "rtx_blas_info_get: bad argument");
    RTX_CK(cudaSetDevice(c->cfg.device));
    const rtx_status st = sync_host_bounds(c);
    if (st != RTX_OK) return st;
    const ModelRec& m = c->models[model_id];
    out->n_nodes = m.bvh.n_nodes; out->n_tris = m.bvh.n_prims;
    out->bytes = (uint64_t)m.bvh.n_nodes * 80 + (uint64_t)m.bvh.n_prims * 48;
    out->sah_cost = m.bvh.sah_cost; out->build_ms = m.bvh.build_ms;
    return RTX_OK;
}

extern "C" rtx_status rtx_set_material_ids(rtx_ctx* c, const uint32_t* ids, uint32_t n) {
    if (!c || (!ids && n)) return fail(RTX_ERR_ARG, "rtx_set_material_ids: null argument");
    RTX_ENTER(c);
    c->n_material_ids = n;
    return upload(&c->d_material_ids, ids, n, c->stream, &c->cap_material_ids);
}

extern "C" rtx_status rtx_set_materials(rtx_ctx* c, const rtx_material* m, uint32_t n) {
    if (!c || (!m && n)) return fail(RTX_ERR_ARG, "rtx_set_materials: null argument");
    RTX_ENTER(c);
    c->n_materials = n;
    return upload(&c->d_materials, m, n, c->stream, &c->cap_materials);
}

// a model's entries of d_blas and d_bounds, padding zeroed
static void table_entries(const ModelRec& m, BlasRef* br, BlasBounds* bb) {
    memset(br, 0, sizeof *br); memset(bb, 0, sizeof *bb);
    br->nodes = m.bvh.nodes; br->tris = m.bvh.prims;
    for (int k = 0; k < 3; k++) { bb->lo[k] = br->lo[k] = m.bvh.lo[k]; bb->hi[k] = br->hi[k] = m.bvh.hi[k]; }
    bb->verts = m.d_verts; bb->n_verts = m.n_verts;
}

static rtx_status ensure_tables(rtx_ctx* c) {
    if (c->d_blas && c->n_tables == c->models.size()) return RTX_OK;
    const rtx_status sb = sync_host_bounds(c);
    if (sb != RTX_OK) return sb;
    free_tables(c);
    const size_t n = c->models.size();
    std::vector<BlasRef> br(n); std::vector<BlasBounds> bb(n); std::vector<ModelRef> mr(n);
    for (size_t i = 0; i < n; i++) {
        const ModelRec& m = c->models[i];
        table_entries(m, &br[i], &bb[i]);
        mr[i].verts = m.d_verts; mr[i].idx = m.d_idx; mr[i].mat_offset = m.mat_offset; mr[i].n_tris = m.n_tris; mr[i].shade = m.d_shade;
    }
    rtx_status st;
    if ((st = upload(&c->d_blas, br.data(), n, c->stream)) != RTX_OK) return st;
    if ((st = upload(&c->d_bounds, bb.data(), n, c->stream)) != RTX_OK) return st;
    if ((st = upload(&c->d_model_refs, mr.data(), n, c->stream)) != RTX_OK) return st;
    c->n_tables = (uint32_t)n;
    return RTX_OK;
}

// device buffer of at least n elements; reallocated (cudaFree synchronises) only when it has to grow
template <typename T>
static rtx_status reserve(T** dptr, size_t* cap, size_t n) {
    if (*dptr && *cap >= n) return RTX_OK;
    if (*dptr) { cudaFree(*dptr); *dptr = nullptr; }
    RTX_CK(cudaMalloc((void**)dptr, (n ? n : 1) * sizeof(T)));
    *cap = n ? n : 1;
    return RTX_OK;
}

// the caller's arrays are copied into a pinned staging block (the library copies on upload, S-rows ownership) and from there to the
// device on `s`; the block is reused two calls later, after the event recorded behind its H2D copies
static rtx_status stage_instances(rtx_ctx* c, const rtx_instance_desc* descs, const rtx_instance_props* props, uint32_t n,
                                  rtx_instance_desc* d_descs, rtx_instance_props* d_props, uint32_t* d_inst_model, cudaStream_t s) {
    rtx_ctx::Stage& sg = c->stage[c->stage_i]; c->stage_i ^= 1;
    if (!sg.ev) RTX_CK(cudaEventCreateWithFlags(&sg.ev, cudaEventDisableTiming));
    if (sg.pending) { RTX_CK(cudaEventSynchronize(sg.ev)); sg.pending = false; }
    const size_t b_descs = (size_t)n * sizeof(rtx_instance_desc), b_props = (size_t)n * sizeof(rtx_instance_props), b_im = (size_t)n * 4;
    if (sg.cap < b_descs + b_props + b_im) {
        if (sg.p) cudaFreeHost(sg.p);
        sg.cap = b_descs + b_props + b_im + 4096;
        RTX_CK(cudaMallocHost(&sg.p, sg.cap));
    }
    if (n) {
        uint8_t* h = (uint8_t*)sg.p;
        memcpy(h, descs, b_descs); memcpy(h + b_descs, props, b_props);
        uint32_t* im = (uint32_t*)(h + b_descs + b_props);
        for (uint32_t i = 0; i < n; i++) im[i] = (uint32_t)descs[i].blas;
        RTX_CK(cudaMemcpyAsync(d_descs, h, b_descs, cudaMemcpyHostToDevice, s));
        RTX_CK(cudaMemcpyAsync(d_props, h + b_descs, b_props, cudaMemcpyHostToDevice, s));
        RTX_CK(cudaMemcpyAsync(d_inst_model, im, b_im, cudaMemcpyHostToDevice, s));
        RTX_CK(cudaEventRecord(sg.ev, s)); sg.pending = true;
    }
    return RTX_OK;
}

static bool lane_buffers(rtx_ctx* c);

// the per-instance arrays of f for at least n instances; all of them are reallocated together (cudaFree synchronises), only when they
// have to grow
static cudaError_t reserve_instances(rtx_ctx::FrameSet& f, size_t n) {
    if (f.d_descs && f.cap >= n) return cudaSuccess;
    const size_t k = n ? n : 1;
    void** p[] = {(void**)&f.d_descs, (void**)&f.d_props, (void**)&f.d_inst_model, (void**)&f.d_inst_recs, (void**)&f.d_box_lo,
                  (void**)&f.d_box_hi, (void**)&f.d_box6};
    const size_t bytes[] = {sizeof(rtx_instance_desc), sizeof(rtx_instance_props), 4, 64, 16, 16, 24};      // per instance
    f.cap = 0;
    for (int i = 0; i < 7; i++) {
        if (*p[i]) { cudaFree(*p[i]); *p[i] = nullptr; }
        const cudaError_t e = cudaMalloc(p[i], k * bytes[i]);
        if (e != cudaSuccess) return e;
    }
    f.cap = k;
    return cudaSuccess;
}

static const size_t SINGLE_NODE_INSTANCES = 8;      // the largest TLAS that is one node (bvh_build.cu tlas_fits_one_node)
// lane 1's set of per-frame state (<= 8 instances); false (the frame is not pipelined) when it cannot be allocated
static bool ensure_frame_set(rtx_ctx* c) {
    rtx_ctx::FrameSet& f = c->fs[1];
    if (f.tlas_cap) return true;
    const size_t n = SINGLE_NODE_INSTANCES;
    cudaError_t e = reserve_instances(f, n);
    if (e == cudaSuccess && !f.d_tlas_ctr) e = cudaMalloc(&f.d_tlas_ctr, 256);
    if (e == cudaSuccess && !f.tlas.nodes) e = cudaMalloc((void**)&f.tlas.nodes, 80);
    if (e == cudaSuccess && !f.tlas.prims) e = cudaMalloc((void**)&f.tlas.prims, n * 64);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }      // (freed by rtx_destroy)
    f.tlas_cap = n;
    return true;
}
// fs[0] becomes the newest set again (copied from fs[1] on the caller's stream, which is behind every pass); box6 and the TLAS scratch
// hold nothing between calls
static rtx_status sync_frame_state(rtx_ctx* c) {
    if (c->cur_set == 0) return RTX_OK;
    rtx_ctx::FrameSet &d = c->fs[0], &f = c->fs[1];
    const size_t n = c->n_instances;
    const cudaMemcpyKind k = cudaMemcpyDeviceToDevice;
    RTX_CK(cudaMemcpyAsync(d.d_descs, f.d_descs, n * sizeof(rtx_instance_desc), k, c->stream));
    RTX_CK(cudaMemcpyAsync(d.d_props, f.d_props, n * sizeof(rtx_instance_props), k, c->stream));
    RTX_CK(cudaMemcpyAsync(d.d_inst_model, f.d_inst_model, n * 4, k, c->stream));
    RTX_CK(cudaMemcpyAsync(d.d_inst_recs, f.d_inst_recs, n * 64, k, c->stream));
    RTX_CK(cudaMemcpyAsync(d.d_box_lo, f.d_box_lo, n * 16, k, c->stream));
    RTX_CK(cudaMemcpyAsync(d.d_box_hi, f.d_box_hi, n * 16, k, c->stream));
    RTX_CK(cudaMemcpyAsync(d.tlas.nodes, f.tlas.nodes, 80, k, c->stream));
    RTX_CK(cudaMemcpyAsync(d.tlas.prims, f.tlas.prims, n * 64, k, c->stream));
    c->cur_set = 0;
    return RTX_OK;
}
// is the call part of a per-frame loop that can be pipelined?  (the previous frame ended with rtx_render_pass [+ read-back] and nothing else)
static bool frame_fast_ok(rtx_ctx* c) {
    return c->pipeline && c->frame_pipeline && c->frame_seq_ok && c->wb_ready &&
           !(c->cfg.flags & (RTX_FLAG_LEGACY_RR | RTX_FLAG_RESTIR)) && !c->timing.stage_timing && !c->trace_stats &&
           (uint64_t)c->cfg.width * c->cfg.height * c->cfg.samples_per_pass >= 65536u && lane_buffers(c) && ensure_frame_set(c);
}

// Instance records, world boxes and TLAS of the n instances in f.d_descs / d_props (of the models c->tlas_models), on stream s, after
// the instance list or a model's geometry changed.
static rtx_status update_instance_state(rtx_ctx* c, rtx_ctx::FrameSet& f, uint32_t n, bool same_models, cudaStream_t s) {
    cudaError_t e = launch_instance_records(f.d_descs, f.d_props, c->d_bounds, n, f.d_inst_recs, f.d_box_lo, f.d_box_hi, f.d_box6, s);
    if (e == cudaSuccess && n) {
        if (!f.d_tlas_ctr) RTX_CK(cudaMalloc(&f.d_tlas_ctr, 256));
        if (tlas_fits_one_node(n) && f.tlas.nodes && f.tlas_cap >= n) {
            // a TLAS of one node is rewritten in place: no allocation, no host synchronisation (the per-frame path of BASELINE config C2)
            e = update_tlas_one_node(f.d_inst_recs, f.d_box_lo, f.d_box_hi, n, &f.tlas, f.d_tlas_ctr, s);
        } else if (f.tlas.nodes && f.tlas.n_prims == n && same_models && !c->force_tlas_rebuild) {
            // same instances of the same models as the last build: REFIT (what the reference does every frame, rdn/Renderer.cpp:594)
            e = refit_tlas(f.d_inst_recs, f.d_box_lo, f.d_box_hi, n, &f.tlas, s);
        } else {
            RTX_CK(cudaStreamSynchronize(s));
            free_bvh(&f.tlas);
            e = build_tlas(f.d_inst_recs, f.d_box_lo, f.d_box_hi, n, &f.tlas, s);
            f.tlas_cap = e == cudaSuccess ? f.tlas.n_prims : 0;
        }
        // The traversal stack (RTX_STACK_SIZE = 40 entries per ray) holds at most one entry per level of the node path being descended
        // plus one parked instance-leaf group per TLAS level: reject a TLAS + BLAS pair that could overflow it before anything is traced
        // (the kernels still raise the context's overflow word if it ever happens, check_overflow).
        uint32_t blas_levels = 0;
        for (uint32_t i = 0; i < n; i++) blas_levels = std::max(blas_levels, c->models[c->tlas_models[i]].bvh.n_levels);
        if (e == cudaSuccess && 2u * f.tlas.n_levels + blas_levels + 2u > 40u)
            return fail(RTX_ERR_STATE, "TLAS + BLAS too deep for the traversal stack (RTX_STACK_SIZE)");
    }
    c->launches += 6;
    RTX_CK(e);
    return RTX_OK;
}

extern "C" rtx_status rtx_set_instances(rtx_ctx* c, const rtx_instance_desc* descs, const rtx_instance_props* props, uint32_t n) {
    if (!c || ((!descs || !props) && n)) return fail(RTX_ERR_ARG, "rtx_set_instances: null argument");
    RTX_CK(cudaSetDevice(c->cfg.device));
    for (uint32_t i = 0; i < n; i++) {
        if (descs[i].blas >= c->models.size()) return fail(RTX_ERR_ARG, "rtx_set_instances: instance references an unknown model");
        if (c->models[descs[i].blas].n_tris == 0) return fail(RTX_ERR_ARG, "rtx_set_instances: instance of an empty model");
    }
    rtx_status st;
    if ((st = sync_host_bounds(c)) != RTX_OK) return st;
    {   // bounds of the "heavy" instances (BLAS with >= 1/4 of the largest BLAS's triangles): rays crossing them go to the front of the
        // wavefront's queues (wavefront.h RayQueue), and the bounds of everything: the classification is only worth its atomics when it
        // separates something (in a scene whose instances are all of one size every ray that hits anything is "heavy": C3 lost 2 % to
        // it).  Corner boxes through the desc's objectToWorld: conservative, host arithmetic only.
        uint32_t max_tris = 0;
        for (uint32_t i = 0; i < n; i++) max_tris = std::max(max_tris, c->models[descs[i].blas].n_tris);
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        float slo[3] = {INFINITY, INFINITY, INFINITY}, shi[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (uint32_t i = 0; i < n; i++) {
            const ModelRec& m = c->models[descs[i].blas];
            const bool heavy = (uint64_t)m.n_tris * 4u >= max_tris;
            for (int k = 0; k < 8; k++) {
                const float x = (k & 1) ? m.bvh.hi[0] : m.bvh.lo[0], y = (k & 2) ? m.bvh.hi[1] : m.bvh.lo[1], z = (k & 4) ? m.bvh.hi[2] : m.bvh.lo[2];
                for (int r = 0; r < 3; r++) {
                    const float* t = descs[i].transform[r];
                    const float v = t[0] * x + t[1] * y + t[2] * z + t[3];
                    if (heavy) { lo[r] = fminf(lo[r], v); hi[r] = fmaxf(hi[r], v); }
                    slo[r] = fminf(slo[r], v); shi[r] = fmaxf(shi[r], v);
                }
            }
        }
        const float vh = (hi[0] - lo[0]) * (hi[1] - lo[1]) * (hi[2] - lo[2]), vs = (shi[0] - slo[0]) * (shi[1] - slo[1]) * (shi[2] - slo[2]);
        c->heavy_valid = n > 0 && lo[0] <= hi[0] && vh < 0.5f * vs;
        for (int r = 0; r < 3; r++) { c->heavy_lo[r] = lo[r]; c->heavy_hi[r] = hi[r]; }
    }
    bool same_models = c->tlas_models.size() == n;
    for (uint32_t i = 0; same_models && i < n; i++) same_models = c->tlas_models[i] == (uint32_t)descs[i].blas;
    rtx_ctx::FrameSet& f0 = c->fs[0];
    if (same_models && tlas_fits_one_node(n) && f0.tlas.nodes && f0.tlas.n_prims == n && f0.tlas_cap >= n && c->n_instances == n &&
        !c->force_tlas_rebuild && c->d_blas && c->n_tables == c->models.size() && frame_fast_ok(c)) {
        // the per-frame path of a pipelined frame loop: the state set of the lane this frame will render on, on that lane's stream
        const int L = 1 - c->last_lane;
        rtx_ctx::FrameSet& f = c->fs[L];
        const cudaStream_t s_ = c->lane_stream[L];
        if (c->main_dirty) { RTX_CK(cudaEventRecord(c->ev_state, c->stream)); c->main_dirty = false; }
        RTX_CK(cudaStreamWaitEvent(s_, c->ev_state, 0));
        RTX_CK(cudaStreamWaitEvent(s_, c->ev_acc[L], 0));                                        // the last pass of this lane ...
        if (c->lane_read_set[1 - L] == L) RTX_CK(cudaStreamWaitEvent(s_, c->ev_acc[1 - L], 0));   // ... and of the other one if it read this set
        if (L) { Bvh8 t = f0.tlas; t.nodes = f.tlas.nodes; t.prims = f.tlas.prims; f.tlas = t; }  // set 0's counts, levels, bounds
        if ((st = stage_instances(c, descs, props, n, f.d_descs, f.d_props, f.d_inst_model, s_)) != RTX_OK) return st;
        if ((st = update_instance_state(c, f, n, same_models, s_)) != RTX_OK) return st;
        RTX_CK(cudaEventRecord(c->ev_fset, s_)); c->fset_pending = true;
        c->pending_lane = L; c->cur_set = L;
        return RTX_OK;
    }
    RTX_ENTER(c);
    if ((st = ensure_tables(c)) != RTX_OK) return st;
    RTX_CK(reserve_instances(f0, n));
    if ((st = stage_instances(c, descs, props, n, f0.d_descs, f0.d_props, f0.d_inst_model, c->stream)) != RTX_OK) return st;
    c->n_instances = n;
    if (n) {
        c->tlas_models.resize(n);
        for (uint32_t i = 0; i < n; i++) c->tlas_models[i] = (uint32_t)descs[i].blas;
    }
    return update_instance_state(c, f0, n, same_models, c->stream);
}

// New vertex positions (and normals) for an uploaded model: everything derived from the vertices follows on the context stream — the
// vertex buffer in place, the closest-hit attribute records, the triangle records and node boxes (REFIT) or a new BVH (REBUILD), the
// model's d_blas / d_bounds entries, the instance world boxes and the TLAS.
static rtx_status update_model(rtx_ctx* c, uint32_t id, const void* v, uint32_t nv, uint32_t mode, bool device) {
    RTX_ENTER(c);
    ModelRec& m = c->models[id];
    const bool tables = c->d_blas && c->n_tables == c->models.size();
    rtx_status st;
    if (nv) RTX_CK(cudaMemcpyAsync(m.d_verts, v, (size_t)nv * sizeof(rtx_vertex), device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
    if (m.n_tris) k_shade_records<<<(m.n_tris + 255) / 256, 256, 0, c->stream>>>(m.d_verts, m.d_idx, m.n_tris, m.d_shade);
    RTX_CK(cudaGetLastError());
    c->launches += 1;
    if (mode == RTX_UPDATE_REFIT) {
        float* d_out6 = (float*)((char*)c->d_refit + 128);
        RTX_CK(refit_blas(m.d_verts, m.d_idx, m.n_tris, &m.bvh, c->d_refit, tables ? c->d_blas + id : nullptr, tables ? c->d_bounds + id : nullptr,
                          d_out6, c->stream));
        if (m.n_tris) {
            RTX_CK(cudaMemcpyAsync(m.h_bounds, d_out6, 6 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
            RTX_CK(cudaEventRecord(c->ev_bounds, c->stream));
            m.bounds_pending = c->bounds_pending = true;
            c->launches += 3 + m.bvh.n_levels;
        }
    } else {
        if ((st = sync_host_bounds(c)) != RTX_OK) return st;      // (a pending copy would overwrite the new build's bounds)
        Bvh8 nb;
        const cudaError_t e = build_blas(m.d_verts, m.n_verts, m.d_idx, m.n_tris, &nb, c->stream);
        if (e != cudaSuccess) { free_bvh(&nb); RTX_CK(e); }
        Bvh8 old = m.bvh;
        m.bvh = nb;
        if (tables) {       // in place: captured pass graphs hold the d_blas pointer
            BlasRef br; BlasBounds bb;
            table_entries(m, &br, &bb);
            RTX_CK(cudaMemcpyAsync(c->d_blas + id, &br, sizeof br, cudaMemcpyHostToDevice, c->stream));
            RTX_CK(cudaMemcpyAsync(c->d_bounds + id, &bb, sizeof bb, cudaMemcpyHostToDevice, c->stream));
        }
        // the build synchronised the stream, which is behind every pass queued before this call: nothing reads the old BVH any more
        RTX_CK(cudaStreamSynchronize(c->stream));
        free_bvh(&old);
        c->launches += 9;
    }
    if (c->n_instances && (st = update_instance_state(c, c->fs[0], c->n_instances, true, c->stream)) != RTX_OK) return st;
    if (!device) {
        RTX_CK(cudaStreamSynchronize(c->stream));
        return sync_host_bounds(c);
    }
    return RTX_OK;
}

static rtx_status check_update_args(rtx_ctx* c, uint32_t id, const void* v, uint32_t nv, uint32_t mode, const char* name) {
    if (!c) return fail(RTX_ERR_ARG, (std::string(name) + ": null context").c_str());
    if (id >= c->models.size()) return fail(RTX_ERR_ARG, (std::string(name) + ": unknown model").c_str());
    if (nv != c->models[id].n_verts) return fail(RTX_ERR_ARG, (std::string(name) + ": vertex count differs from the model's upload").c_str());
    if (mode != RTX_UPDATE_REFIT && mode != RTX_UPDATE_REBUILD) return fail(RTX_ERR_ARG, (std::string(name) + ": unknown mode").c_str());
    if (!v && nv) return fail(RTX_ERR_ARG, (std::string(name) + ": null vertex pointer").c_str());
    return RTX_OK;
}

extern "C" rtx_status rtx_update_model(rtx_ctx* c, uint32_t model_id, const rtx_vertex* v, uint32_t nv, uint32_t mode) {
    const rtx_status st = check_update_args(c, model_id, v, nv, mode, "rtx_update_model");
    if (st != RTX_OK) return st;
    return update_model(c, model_id, v, nv, mode, false);
}

extern "C" rtx_status rtx_update_model_device(rtx_ctx* c, uint32_t model_id, const void* d_v, uint32_t nv, uint32_t mode) {
    const rtx_status st = check_update_args(c, model_id, d_v, nv, mode, "rtx_update_model_device");
    if (st != RTX_OK) return st;
    if (nv) {
        cudaPointerAttributes a;
        memset(&a, 0, sizeof a);
        const cudaError_t e = cudaPointerGetAttributes(&a, d_v);
        if (e != cudaSuccess) cudaGetLastError();
        if (e != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != c->cfg.device)
            return fail(RTX_ERR_ARG, "rtx_update_model_device: the vertices are not device memory of the context's device");
    }
    return update_model(c, model_id, d_v, nv, mode, true);
}

extern "C" rtx_status rtx_set_emissive_triangles(rtx_ctx* c, const rtx_light_triangle* l, uint32_t n) {
    if (!c || (!l && n)) return fail(RTX_ERR_ARG, "rtx_set_emissive_triangles: null argument");
    RTX_ENTER(c);
    c->n_lights = n;
    if (n == 0) {   // an out-of-bounds read of t6 returns zeros (SURVEY.md Appendix C.3): keep one zero record
        rtx_light_triangle z; memset(&z, 0, sizeof z);
        return upload(&c->d_lights, &z, 1, c->stream, &c->cap_lights);
    }
    return upload(&c->d_lights, l, n, c->stream, &c->cap_lights);
}

static rtx_status ensure_wave(rtx_ctx* c) {
    if (c->wb_ready) return RTX_OK;
    RTX_CK(wave_alloc(&c->wb, c->cfg.width, c->cfg.height, c->cfg.samples_per_pass));
    c->wb_ready = true;
    return RTX_OK;
}

extern "C" rtx_status rtx_set_camera(rtx_ctx* c, const rtx_camera_params* cam) {
    if (!c || !cam) return fail(RTX_ERR_ARG, "rtx_set_camera: null argument");
    RTX_CK(cudaSetDevice(c->cfg.device));
    const int fast_lane = c->pending_lane;       // >= 0: the camera of a pipelined frame (its rtx_set_instances chose the lane)
    rtx_status st;
    if (fast_lane < 0) {
        RTX_ENTER(c);
        if ((st = ensure_wave(c)) != RTX_OK) return st;
    }
    // Pass_spat_di_v7.hlsl:407-423: any element of view differing from the previous view by more than s_bias resets the accumulation
    // The shader compares view with prevView of the SAME constant buffer; a host that does not maintain prevView (all zeros, or a copy of
    // view) is covered by also comparing with the view of the previous call.
    bool different = !c->have_cam;
    for (int i = 0; i < 16 && !different; i++) {
        if (fabsf(cam->view[i] - cam->prevView[i]) > RTX_S_BIAS) different = true;
        if (c->have_cam && fabsf(cam->view[i] - c->cam.view[i]) > RTX_S_BIAS) different = true;
    }
    c->cam = *cam; c->have_cam = true;
    c->cam_version++;
    if (fast_lane >= 0) {
        const cudaStream_t s_ = c->lane_stream[fast_lane];      // (already behind ev_state and the lane's last pass: rtx_set_instances)
        RTX_CK(cudaMemcpyAsync(fast_lane ? c->wb2.cam : c->wb.cam, &c->cam, sizeof c->cam, cudaMemcpyHostToDevice, s_));
        c->cam_block_version[fast_lane] = c->cam_version;
        if (different) {        // the reset lands between the previous frame's accumulation (and resolve) and this frame's
            RTX_CK(cudaStreamWaitEvent(s_, c->ev_acc[1 - fast_lane], 0));
            if (c->resolve_pending) RTX_CK(cudaStreamWaitEvent(s_, c->ev_resolved, 0));
            RTX_CK(cudaMemsetAsync(c->wb.accum, 0, (size_t)c->cfg.width * c->cfg.height * 16, s_));
        }
        RTX_CK(cudaEventRecord(c->ev_fset, s_)); c->fset_pending = true;
        return RTX_OK;
    }
    RTX_CK(cudaMemcpyAsync(c->wb.cam, &c->cam, sizeof c->cam, cudaMemcpyHostToDevice, c->stream));
    c->cam_block_version[0] = c->cam_version;       // (lane 1's block is brought up to date when a pass runs there)
    if (different) RTX_CK(cudaMemsetAsync(c->wb.accum, 0, (size_t)c->cfg.width * c->cfg.height * 16, c->stream));
    return RTX_OK;      // the 512-B copy from pageable memory is staged by the driver before the call returns
}

// the bindings of a pass that reads set `set` of the per-frame instance state
static SceneData scene_data(rtx_ctx* c, int set = 0) {
    SceneData S;
    memset(&S, 0, sizeof S);            // (padding bytes too: the wavefront compares these structs bytewise to reuse a captured pass)
    S.models = c->d_model_refs; S.inst_model = c->fs[set].d_inst_model; S.props = c->fs[set].d_props;
    S.material_ids = c->d_material_ids; S.n_material_ids = c->n_material_ids;
    S.materials = c->d_materials; S.n_materials = c->n_materials;
    S.lights = c->d_lights;
    S.cfg_flags = c->cfg.flags; S.bounces = c->cfg.bounces; S.nee_samples = c->cfg.nee_samples; S.nee_samples_di = c->cfg.nee_samples_di;
    S.width = c->cfg.width; S.height = c->cfg.height;
    for (int r = 0; r < 3; r++) { S.heavy_lo[r] = c->heavy_lo[r]; S.heavy_hi[r] = c->heavy_hi[r]; }
    S.heavy_valid = c->heavy_valid && c->lpt ? 1u : 0u;
    return S;
}

static SceneAS make_as(rtx_ctx* c, int set = 0) {
    SceneAS a;
    memset(&a, 0, sizeof a);            // (padding bytes too: the wavefront compares these structs bytewise to reuse a captured pass)
    const Bvh8& tl = c->fs[set].tlas;
    a.tlas_nodes = tl.nodes; a.inst_recs = tl.prims; a.blas = c->d_blas; a.n_instances = c->n_instances;
    a.one_bits = 0x3F800000u;
    a.overflow = c->d_overflow;
    a.num_sms = c->num_sms; a.fetch_th = c->fetch_th; a.sched = c->sched; a.waves = c->waves; a.ctas_per_sm = c->ctas_per_sm;
    return a;
}

// Reads the context's overflow word behind everything queued on the stream; a raised word fails the call ONCE and is cleared, so that
// the context is usable again after the offending scene has been replaced.
static rtx_status check_overflow(rtx_ctx* c) {
    unsigned int flag = 0;
    RTX_CK(cudaMemcpyAsync(&flag, c->d_overflow, sizeof flag, cudaMemcpyDeviceToHost, c->stream));
    RTX_CK(cudaStreamSynchronize(c->stream));
    if (flag) {
        RTX_CK(cudaMemsetAsync(c->d_overflow, 0, sizeof flag, c->stream));
        c->main_dirty = true; c->in_sequence = false;       // the passes that follow start behind the clear
        return fail(RTX_ERR_STATE, "traversal stack overflow (BVH deeper than RTX_STACK_SIZE): the results of this pass are invalid");
    }
    return RTX_OK;
}

// the second set of pass buffers, allocated when first needed and only if it takes less than a quarter of the free device memory
static bool lane_buffers(rtx_ctx* c) {
    if (c->wb2_ready) return true;
    if (c->wb2_refused || !c->wb_ready) return false;
    size_t free_b = 0, total_b = 0;
    const size_t need = (size_t)c->wb.n_paths * 480u;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || need > free_b / 4) { c->wb2_refused = true; return false; }
    c->wb2 = WaveBuffers();
    if (wave_alloc_lane(&c->wb2, c->wb, c->cfg.width, c->cfg.height, c->cfg.samples_per_pass) != cudaSuccess) {
        cudaGetLastError();
        wave_free_lane(&c->wb2); c->wb2_refused = true;
        return false;
    }
    c->wb2_ready = true;
    return true;
}

extern "C" rtx_status rtx_render_pass(rtx_ctx* c, uint32_t first_sample, uint32_t n_samples) {
    if (!c) return fail(RTX_ERR_ARG, "rtx_render_pass: null context");
    if (!c->have_cam) return fail(RTX_ERR_STATE, "rtx_render_pass: camera not set");
    if (!c->n_instances || !c->fs[0].tlas.nodes) return fail(RTX_ERR_STATE, "rtx_render_pass: no instances");
    if (!c->d_materials || !c->d_material_ids) return fail(RTX_ERR_STATE, "rtx_render_pass: materials not set");
    RTX_CK(cudaSetDevice(c->cfg.device));
    rtx_status st;
    if (!c->d_lights && (st = rtx_set_emissive_triangles(c, nullptr, 0)) != RTX_OK) return st;
    if ((st = ensure_wave(c)) != RTX_OK) return st;
    const uint32_t npx = c->cfg.width * c->cfg.height;
    // pipelined passes (see rtx_ctx): the estimator E0 without per-launch instrumentation, frames large enough to be cut into path ranges
    const bool eligible = c->pipeline && !(c->cfg.flags & (RTX_FLAG_LEGACY_RR | RTX_FLAG_RESTIR)) &&
                          !c->timing.stage_timing && !c->trace_stats && (uint64_t)npx * c->cfg.samples_per_pass >= 65536u && lane_buffers(c);
    uint32_t done = 0;
    while (done < n_samples) {
        const uint32_t spp = std::min(c->cfg.samples_per_pass, n_samples - done);
        c->timing.stats = c->trace_stats ? c->d_stats : nullptr;
        // whatever other entry points queued on the caller's stream (camera, instances, uploads, clears) is ordered before the passes of
        // both lanes through ev_state, recorded BEFORE this pass is queued (a lane never waits for the other lane's pass)
        if (c->main_dirty) { RTX_CK(cudaEventRecord(c->ev_state, c->stream)); c->main_dirty = false; }
        if (c->pending_lane >= 0 && !eligible) RTX_ENTER(c);          // (cannot happen: the fast calls test the same conditions)
        const int frame_lane = eligible ? c->pending_lane : -1;       // >= 0: a frame prepared by the fast rtx_set_instances [+ rtx_set_camera]
        if (!(eligible && (c->in_sequence || frame_lane >= 0))) {
            // the first pass after any other call: B.parts path ranges on the caller's stream, accumulation included
            const SceneData S = scene_data(c);
            const SceneAS AS = make_as(c);
            if (c->cam_block_version[0] != c->cam_version) {
                RTX_CK(cudaMemcpyAsync(c->wb.cam, &c->cam, sizeof c->cam, cudaMemcpyHostToDevice, c->stream));
                c->cam_block_version[0] = c->cam_version;
            }
            if (c->cfg.flags & RTX_FLAG_LEGACY_RR) RTX_CK(wave_render_pass_legacy(c->wb, S, AS, first_sample + done, spp, c->stream, &c->launches, &c->timing));
            else if (c->cfg.flags & RTX_FLAG_FAST_MATH) RTX_CK(fast::wave_render_pass(c->wb, S, AS, first_sample + done, spp, c->stream, &c->launches, &c->timing));
            else RTX_CK(wave_render_pass(c->wb, S, AS, first_sample + done, spp, c->stream, &c->launches, &c->timing));
            RTX_CK(cudaEventRecord(c->ev_acc[0], c->stream));
            c->last_lane = 0; c->lane_read_set[0] = 0;
        } else {
            // a pass that directly follows another (or a pipelined frame): the other lane, one path range, its accumulation behind the
            // previous pass's
            const int lane = frame_lane >= 0 ? frame_lane : 1 - c->last_lane;
            const int set = frame_lane >= 0 ? frame_lane : c->cur_set;       // the per-frame state it reads
            const SceneData S = scene_data(c, set);
            const SceneAS AS = make_as(c, set);
            WaveBuffers& B = lane ? c->wb2 : c->wb;
            PassTiming& T = lane ? c->timing2 : c->timing;
            const cudaStream_t st_ = c->lane_stream[lane];
            RTX_CK(cudaStreamWaitEvent(st_, c->ev_state, 0));
            RTX_CK(cudaStreamWaitEvent(st_, c->ev_acc[lane], 0));           // the previous pass in these buffers (it may have run on the caller's stream)
            if (lane) {
                B.shadow_overlap = c->wb.shadow_overlap; B.part_rows = c->wb.part_rows;
                if (!c->wb.use_graph) B.use_graph = false;
                T.stage_timing = false; T.stats = nullptr;
            }
            if (c->cam_block_version[lane] != c->cam_version) {              // the lane's camera block lags behind the last rtx_set_camera
                RTX_CK(cudaMemcpyAsync(B.cam, &c->cam, sizeof c->cam, cudaMemcpyHostToDevice, st_));
                c->cam_block_version[lane] = c->cam_version;
            }
            if (c->cfg.flags & RTX_FLAG_FAST_MATH) RTX_CK(fast::wave_render_pass(B, S, AS, first_sample + done, spp, st_, &c->launches, &T, true, 1, true));
            else RTX_CK(wave_render_pass(B, S, AS, first_sample + done, spp, st_, &c->launches, &T, true, 1, true));
            RTX_CK(cudaStreamWaitEvent(st_, c->ev_acc[1 - lane], 0));                         // gPermanentData += in call order
            if (c->reduce_pending) RTX_CK(cudaStreamWaitEvent(st_, c->ev_reduced, 0));        // a pending multi-GPU reduce still reads it
            if (c->resolve_pending) RTX_CK(cudaStreamWaitEvent(st_, c->ev_resolved, 0));      // ... or the resolve of the previous frame
            RTX_CK(wave_accumulate(B, npx, spp, st_));
            c->launches += 1;
            RTX_CK(cudaEventRecord(c->ev_acc[lane], st_));
            RTX_CK(cudaStreamWaitEvent(c->stream, c->ev_acc[lane], 0));     // stream-ordered API: the caller's stream sees the pass as done
            c->last_lane = lane; c->lane_read_set[lane] = set;
        }
        c->in_sequence = true; c->pending_lane = -1; c->fset_pending = false;
        done += spp;
    }
    c->pass_timed = true;
    c->frame_seq_ok = true;         // a frame loop may go on from here (rtx_read_output_async / rtx_wait_output keep it, enter() ends it)
    return RTX_OK;
}

static rtx_status ensure_restir(rtx_ctx* c) {
    if (!(c->cfg.flags & RTX_FLAG_RESTIR)) return fail(RTX_ERR_STATE, "ReSTIR entry point on a context created without RTX_FLAG_RESTIR");
    if (c->cfg.samples_per_pass != 1) return fail(RTX_ERR_STATE, "RTX_FLAG_RESTIR needs samples_per_pass == 1 (one sample per frame, as the reference)");
    if (c->rs_ready) return RTX_OK;
    RTX_CK(restir_alloc(&c->rs, c->cfg.width, c->cfg.height));
    RTX_CK(restir_clear(c->rs, c->stream));
    c->rs_ready = true;
    return RTX_OK;
}

extern "C" rtx_status rtx_render_frame(rtx_ctx* c, uint32_t frame_index) {
    if (!c) return fail(RTX_ERR_ARG, "rtx_render_frame: null context");
    if (!c->have_cam) return fail(RTX_ERR_STATE, "rtx_render_frame: camera not set");
    if (!c->n_instances || !c->fs[0].tlas.nodes) return fail(RTX_ERR_STATE, "rtx_render_frame: no instances");
    if (!c->d_materials || !c->d_material_ids) return fail(RTX_ERR_STATE, "rtx_render_frame: materials not set");
    RTX_ENTER(c);
    rtx_status st;
    if (!c->d_lights && (st = rtx_set_emissive_triangles(c, nullptr, 0)) != RTX_OK) return st;
    if ((st = ensure_wave(c)) != RTX_OK) return st;
    if ((st = ensure_restir(c)) != RTX_OK) return st;
    const SceneData S = scene_data(c);
    const SceneAS AS = make_as(c);
    c->timing.stats = c->trace_stats ? c->d_stats : nullptr;
    if (c->wb.wait_before_accumulate) RTX_CK(cudaStreamWaitEvent(c->stream, c->wb.wait_before_accumulate, 0));   // a pending reduce reads gPermanentData
    RTX_CK(wave_render_pass(c->wb, S, AS, frame_index, 1, c->stream, &c->launches, &c->timing, false));     // RayGen
    RTX_CK(restir_store_pass1(c->rs, c->wb, S, c->stream, &c->launches));
    RTX_CK(restir_reuse_passes(c->rs, c->wb, S, AS, frame_index, c->stream, &c->launches));                 // RayGen2, RayGen3
    c->pass_timed = true;
    return RTX_OK;
}

extern "C" rtx_status rtx_reset_restir(rtx_ctx* c) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_restir(c)) != RTX_OK) return st;
    RTX_CK(restir_clear(c->rs, c->stream));
    return RTX_OK;
}

extern "C" rtx_status rtx_read_restir(rtx_ctx* c, float* out) {
    if (!c || !out) return fail(RTX_ERR_ARG, "rtx_read_restir: null argument");
    RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_restir(c)) != RTX_OK) return st;
    RTX_CK(restir_dump(c->rs, c->stream, out));
    return RTX_OK;
}

extern "C" rtx_status rtx_reset_accum(rtx_ctx* c) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_wave(c)) != RTX_OK) return st;
    RTX_CK(cudaMemsetAsync(c->wb.accum, 0, (size_t)c->cfg.width * c->cfg.height * 16, c->stream));
    return RTX_OK;
}

extern "C" rtx_status rtx_synchronize(rtx_ctx* c) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    RTX_CK(cudaSetDevice(c->cfg.device));       // (not through enter(): waiting changes no state, a pipelined sequence of passes goes on after it)
    RTX_CK(cudaStreamSynchronize(c->stream));   // the caller's stream is behind every pass queued so far
    return check_overflow(c);
}

extern "C" rtx_status rtx_read_accum(rtx_ctx* c, float* host_out) {
    if (!c || !host_out) return fail(RTX_ERR_ARG, "rtx_read_accum: null argument");
    RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_wave(c)) != RTX_OK) return st;
    RTX_CK(cudaMemcpyAsync(host_out, c->wb.accum, (size_t)c->cfg.width * c->cfg.height * 16, cudaMemcpyDeviceToHost, c->stream));
    RTX_CK(cudaStreamSynchronize(c->stream));
    return check_overflow(c);
}

extern "C" rtx_status rtx_read_output(rtx_ctx* c, uint8_t* rgba8_out) {
    if (!c || !rgba8_out) return fail(RTX_ERR_ARG, "rtx_read_output: null argument");
    RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_wave(c)) != RTX_OK) return st;
    const uint32_t npx = c->cfg.width * c->cfg.height;
    if (c->copy_pending) { RTX_CK(cudaEventSynchronize(c->ev_copied)); c->copy_pending = false; }
    if (c->comm && c->ev_reduced) RTX_CK(cudaStreamWaitEvent(c->stream, c->ev_reduced, 0));      // the reduced buffer must be complete
    RTX_CK(wave_resolve(c->wb, npx, c->stream, &c->launches));
    RTX_CK(cudaMemcpyAsync(rgba8_out, c->wb.output, (size_t)npx * 4, cudaMemcpyDeviceToHost, c->stream));
    return check_overflow(c);       // synchronises the stream
}

static rtx_status ensure_side_stream(rtx_ctx* c) {
    if (c->copy_stream) return RTX_OK;
    RTX_CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    RTX_CK(cudaEventCreateWithFlags(&c->ev_resolved, cudaEventDisableTiming));
    RTX_CK(cudaEventCreateWithFlags(&c->ev_copied, cudaEventDisableTiming));
    return RTX_OK;
}

// Resolve + read-back without stalling the caller: the D2H copy runs on a side stream behind the resolve kernel, the next frame's
// kernels overlap it.  rtx_wait_output blocks until the image of the LAST rtx_read_output_async call is in rgba8_out.
// With a communicator (rtx_comm_init) the root resolves the REDUCED buffer, and the resolve itself runs on the side stream behind the
// reduce: the render stream never waits for NCCL, the next pass overlaps reduce + resolve + copy.
extern "C" rtx_status rtx_read_output_async(rtx_ctx* c, uint8_t* rgba8_out) {
    if (!c || !rgba8_out) return fail(RTX_ERR_ARG, "rtx_read_output_async: null argument");
    RTX_CK(cudaSetDevice(c->cfg.device));
    // a read-back right after a pass keeps a pipelined sequence alive: the resolve below runs on the caller's stream, which is behind the
    // pass, and the next pass's accumulation waits for it (ev_resolved); from anywhere else it is an ordinary call
    const bool keep = c->in_sequence && c->frame_seq_ok;
    if (!keep) RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_wave(c)) != RTX_OK) return st;
    if ((st = ensure_side_stream(c)) != RTX_OK) return st;
    const uint32_t npx = c->cfg.width * c->cfg.height;
    if (c->comm && c->comm_rank == 0 && c->wb.resolve_source == c->d_total) {
        // side stream order: reduce(k) -> resolve(k) -> copy(k) -> reduce(k+1) ...: nothing else touches d_total or gOutput
        RTX_CK(wave_resolve(c->wb, npx, c->copy_stream, &c->launches));
    } else {
        if (c->copy_pending) RTX_CK(cudaStreamWaitEvent(c->stream, c->ev_copied, 0));      // gOutput is rewritten by the resolve below
        RTX_CK(wave_resolve(c->wb, npx, c->stream, &c->launches));
        RTX_CK(cudaEventRecord(c->ev_resolved, c->stream));
        RTX_CK(cudaStreamWaitEvent(c->copy_stream, c->ev_resolved, 0));
        c->resolve_pending = true;
    }
    RTX_CK(cudaMemcpyAsync(rgba8_out, c->wb.output, (size_t)npx * 4, cudaMemcpyDeviceToHost, c->copy_stream));
    RTX_CK(cudaMemcpyAsync(c->h_overflow, c->d_overflow, sizeof(unsigned int), cudaMemcpyDeviceToHost, c->copy_stream));   // for rtx_wait_output
    RTX_CK(cudaEventRecord(c->ev_copied, c->copy_stream));
    c->copy_pending = true;
    return RTX_OK;
}

// Multi-GPU hosts: rank 0 resolves the REDUCED accumulation buffer (a device float4-per-pixel buffer it owns, e.g. the destination of the
// per-pass ncclReduce) instead of this context's private partial sum.  nullptr restores the context's own buffer.
extern "C" rtx_status rtx_set_resolve_source(rtx_ctx* c, const void* d_accum_float4) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_wave(c)) != RTX_OK) return st;
    c->wb.resolve_source = (const float4*)d_accum_float4;
    return RTX_OK;
}

extern "C" rtx_status rtx_wait_output(rtx_ctx* c) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    RTX_CK(cudaSetDevice(c->cfg.device));
    if (c->copy_pending) {
        RTX_CK(cudaEventSynchronize(c->ev_copied));
        c->copy_pending = false;
        if (*c->h_overflow) {
            *c->h_overflow = 0u;
            RTX_CK(cudaMemsetAsync(c->d_overflow, 0, sizeof(unsigned int), c->stream));
            return fail(RTX_ERR_STATE, "traversal stack overflow (BVH deeper than RTX_STACK_SIZE): the image just read back is invalid");
        }
    }
    return RTX_OK;
}

extern "C" rtx_status rtx_accum_device_ptr(rtx_ctx* c, void** out) {
    if (!c || !out) return fail(RTX_ERR_ARG, "rtx_accum_device_ptr: null argument");
    RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_wave(c)) != RTX_OK) return st;
    *out = c->wb.accum;
    return RTX_OK;
}

// rays arrive as rtx_ray (o, tmin, d, tmax) = two float4 per ray, AoS; the kernels want two SoA planes.
__global__ void k_split_rays(const float4* __restrict__ rays, uint32_t n, float4* __restrict__ o, float4* __restrict__ d) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    o[i] = rays[2 * i]; d[i] = rays[2 * i + 1];
}
__global__ void k_pack_hits(const float4* __restrict__ ha, const uint32_t* __restrict__ hi, uint32_t n, int any_hit, const float4* __restrict__ d,
                            rtx_hit* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    rtx_hit h;
    if (any_hit) { h.t = 0.0f; h.u = 0.0f; h.v = 0.0f; h.prim = 0xFFFFFFFFu; h.inst = hi[i] == 0xFFFFFFFFu ? 0xFFFFFFFFu : 0u; }
    else {
        const float4 a = ha[i];
        h.inst = hi[i];
        if (h.inst == 0xFFFFFFFFu) { h.t = d[i].w; h.u = h.v = 0.0f; h.prim = 0xFFFFFFFFu; }
        else { h.t = a.x; h.u = a.y; h.v = a.z; h.prim = __float_as_uint(a.w); }
    }
    out[i] = h;
}

static rtx_status ensure_trace_cap(rtx_ctx* c, uint32_t n) {
    if (n <= c->trace_cap) return RTX_OK;
    void* ptrs[] = {c->d_trace_o, c->d_trace_d, c->d_trace_ha, c->d_trace_hi};
    for (void* p : ptrs) if (p) cudaFree(p);
    c->d_trace_o = c->d_trace_d = c->d_trace_ha = nullptr; c->d_trace_hi = nullptr; c->trace_cap = 0;
    RTX_CK(cudaMalloc((void**)&c->d_trace_o, (size_t)n * 16));
    RTX_CK(cudaMalloc((void**)&c->d_trace_d, (size_t)n * 16));
    RTX_CK(cudaMalloc((void**)&c->d_trace_ha, (size_t)n * 16));
    RTX_CK(cudaMalloc((void**)&c->d_trace_hi, (size_t)n * 4));
    c->trace_cap = n;
    return RTX_OK;
}

static rtx_status trace_device_impl(rtx_ctx* c, const void* d_rays, uint32_t n, void* d_hits, int any_hit, bool stats) {
    if (!c || (!d_rays && n) || (!d_hits && n)) return fail(RTX_ERR_ARG, "rtx_trace: null argument");
    if (!c->n_instances || !c->fs[0].tlas.nodes) return fail(RTX_ERR_STATE, "rtx_trace: no instances");
    if (n == 0) return RTX_OK;
    RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_trace_cap(c, n)) != RTX_OK) return st;
    static_assert(sizeof(rtx_ray) == 32, "rtx_ray must be 32 bytes");
    const unsigned grid = (n + 255) / 256;
    k_split_rays<<<grid, 256, 0, c->stream>>>((const float4*)d_rays, n, c->d_trace_o, c->d_trace_d);
    // the cursor word of part 0 of the wavefront buffers
    if (!c->wb_ready) { if ((st = ensure_wave(c)) != RTX_OK) return st; }
    RTX_CK(launch_trace(make_as(c), c->d_trace_o, c->d_trace_d, nullptr, n, c->wb.cursor, c->d_trace_ha, c->d_trace_hi, any_hit != 0,
                        stats ? c->d_stats : nullptr, c->stream));
    k_pack_hits<<<grid, 256, 0, c->stream>>>(c->d_trace_ha, c->d_trace_hi, n, any_hit, c->d_trace_d, (rtx_hit*)d_hits);
    c->launches += 3;
    RTX_CK(cudaGetLastError());
    return RTX_OK;
}

extern "C" rtx_status rtx_trace_device(rtx_ctx* c, const void* d_rays, uint32_t n, void* d_hits, int any_hit) {
    return trace_device_impl(c, d_rays, n, d_hits, any_hit, false);
}
extern "C" rtx_status rtx_trace_stats(rtx_ctx* c, const void* d_rays, uint32_t n, void* d_hits, int any_hit) {
    return trace_device_impl(c, d_rays, n, d_hits, any_hit, true);
}

extern "C" rtx_status rtx_trace(rtx_ctx* c, const rtx_ray* rays, uint32_t n, rtx_hit* out, int any_hit) {
    if (!c || (!rays && n) || (!out && n)) return fail(RTX_ERR_ARG, "rtx_trace: null argument");
    if (n == 0) return RTX_OK;
    RTX_ENTER(c);
    rtx_status rs;       // staging buffers are kept between calls and only grow
    if ((rs = reserve((uint8_t**)&c->d_trace_rays, &c->cap_trace_rays, (size_t)n * sizeof(rtx_ray))) != RTX_OK) return rs;
    if ((rs = reserve((uint8_t**)&c->d_trace_hits, &c->cap_trace_hits, (size_t)n * sizeof(rtx_hit))) != RTX_OK) return rs;
    void* d_rays = c->d_trace_rays; void* d_hits = c->d_trace_hits;
    RTX_CK(cudaMemcpyAsync(d_rays, rays, (size_t)n * sizeof(rtx_ray), cudaMemcpyHostToDevice, c->stream));
    rtx_status st = trace_device_impl(c, d_rays, n, d_hits, any_hit, false);
    if (st == RTX_OK) {
        cudaError_t e = cudaMemcpyAsync(out, d_hits, (size_t)n * sizeof(rtx_hit), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) { set_error(cudaGetErrorString(e)); st = RTX_ERR_CUDA; }
    }
    if (st != RTX_OK) return st;
    return check_overflow(c);
}

// ---- multi-GPU: the single collective of the path (SURVEY.md 8e) behind the C ABI ---------------------------------------------------
// NCCL is bound at run time (dlopen): a process that already carries NCCL (PyTorch's bundled copy) keeps exactly one instance, a plain
// C++ host gets the system libnccl.so.2.  Prototypes restated from nccl.h (ncclUniqueId = 128 opaque bytes, passed by value).
namespace {
struct NcclId { char internal[128]; };
struct NcclApi {
    int (*GetUniqueId)(NcclId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*Reduce)(const void*, void*, size_t, int, int, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool ok = false; std::string err;
};
NcclApi& nccl() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);       // the copy the process already loaded, if any
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) { api.err = std::string("NCCL not found: ") + dlerror(); return; }
        api.GetUniqueId = (int (*)(NcclId*))dlsym(h, "ncclGetUniqueId");
        api.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(h, "ncclCommInitRank");
        api.Reduce = (int (*)(const void*, void*, size_t, int, int, int, void*, cudaStream_t))dlsym(h, "ncclReduce");
        api.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
        api.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
        api.ok = api.GetUniqueId && api.CommInitRank && api.Reduce && api.CommDestroy;
        if (!api.ok) api.err = "NCCL symbols missing";
    });
    return api;
}
rtx_status nccl_fail(const char* what, int code) {
    NcclApi& n = nccl();
    set_error(std::string(what) + ": " + (n.GetErrorString ? n.GetErrorString(code) : "NCCL error"));
    return RTX_ERR_CUDA;
}
}  // namespace

extern "C" rtx_status rtx_comm_unique_id(void* out128) {
    if (!out128) return fail(RTX_ERR_ARG, "rtx_comm_unique_id: null argument");
    NcclApi& n = nccl();
    if (!n.ok) return fail(RTX_ERR_STATE, n.err.c_str());
    NcclId id;
    const int r = n.GetUniqueId(&id);
    if (r != 0) return nccl_fail("ncclGetUniqueId", r);
    memcpy(out128, &id, sizeof id);
    return RTX_OK;
}

extern "C" rtx_status rtx_comm_destroy(rtx_ctx* c) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    if (!c->comm) return RTX_OK;
    cudaSetDevice(c->cfg.device);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    nccl().CommDestroy(c->comm);
    c->comm = nullptr; c->comm_world = 1; c->comm_rank = 0;
    if (c->wb_ready) { if (c->wb.resolve_source == c->d_total) c->wb.resolve_source = nullptr; c->wb.wait_before_accumulate = nullptr; }
    c->reduce_pending = false;
    if (c->d_total) { cudaFree(c->d_total); c->d_total = nullptr; }
    if (c->ev_pass) { cudaEventDestroy(c->ev_pass); c->ev_pass = nullptr; }
    if (c->ev_reduced) { cudaEventDestroy(c->ev_reduced); c->ev_reduced = nullptr; }
    return RTX_OK;
}

// Collective over all ranks of the job (one context per GPU, one process or thread per context).  unique_id128 comes from
// rtx_comm_unique_id on one rank and reaches the others through the host's own channel (a file, MPI, torch.distributed ...).
extern "C" rtx_status rtx_comm_init(rtx_ctx* c, const void* unique_id128, int rank, int world) {
    if (!c || !unique_id128 || world < 1 || rank < 0 || rank >= world) return fail(RTX_ERR_ARG, "rtx_comm_init: bad argument");
    if (c->comm) return fail(RTX_ERR_STATE, "rtx_comm_init: the context already has a communicator");
    NcclApi& n = nccl();
    if (!n.ok) return fail(RTX_ERR_STATE, n.err.c_str());
    RTX_ENTER(c);
    rtx_status st;
    if ((st = ensure_wave(c)) != RTX_OK) return st;
    if ((st = ensure_side_stream(c)) != RTX_OK) return st;
    NcclId id; memcpy(&id, unique_id128, sizeof id);
    const int r = n.CommInitRank(&c->comm, world, id, rank);
    if (r != 0) { c->comm = nullptr; return nccl_fail("ncclCommInitRank", r); }
    c->comm_rank = rank; c->comm_world = world;
    RTX_CK(cudaEventCreateWithFlags(&c->ev_pass, cudaEventDisableTiming));
    RTX_CK(cudaEventCreateWithFlags(&c->ev_reduced, cudaEventDisableTiming));
    if (rank == 0) {
        const size_t bytes = (size_t)c->cfg.width * c->cfg.height * 16;
        RTX_CK(cudaMalloc((void**)&c->d_total, bytes));
        RTX_CK(cudaMemsetAsync(c->d_total, 0, bytes, c->stream));
        c->wb.resolve_source = c->d_total;          // "rank 0 then runs F20's divide + sRGB" on the sum
    }
    return RTX_OK;
}

// One ncclReduce(sum, fp32, W*H*4, root 0) straight from gPermanentData into the root's reduced buffer (no staging copy), queued on the
// side stream behind everything rendered so far.  The render stream goes on immediately; only the NEXT accumulation (the last kernel of
// the next pass, which rewrites gPermanentData) waits for the reduce to have read it.
extern "C" rtx_status rtx_reduce_accum(rtx_ctx* c) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    if (!c->comm) return fail(RTX_ERR_STATE, "rtx_reduce_accum: no communicator (rtx_comm_init)");
    RTX_CK(cudaSetDevice(c->cfg.device));
    // (not through enter(): a reduce between two passes does not end a pipelined sequence; the caller's stream is behind every pass)
    RTX_CK(cudaEventRecord(c->ev_pass, c->stream));
    RTX_CK(cudaStreamWaitEvent(c->copy_stream, c->ev_pass, 0));
    const size_t count = (size_t)c->cfg.width * c->cfg.height * 4;
    const int r = nccl().Reduce(c->wb.accum, c->comm_rank == 0 ? (void*)c->d_total : (void*)c->wb.accum, count, /*ncclFloat32*/ 7, /*ncclSum*/ 0, 0,
                                c->comm, c->copy_stream);
    if (r != 0) return nccl_fail("ncclReduce", r);
    RTX_CK(cudaEventRecord(c->ev_reduced, c->copy_stream));
    c->wb.wait_before_accumulate = c->ev_reduced;
    c->reduce_pending = true;
    return RTX_OK;
}

// the root's reduced accumulation buffer (float4 per pixel), complete up to the last rtx_reduce_accum
extern "C" rtx_status rtx_read_reduced_accum(rtx_ctx* c, float* host_out) {
    if (!c || !host_out) return fail(RTX_ERR_ARG, "rtx_read_reduced_accum: null argument");
    if (!c->comm || c->comm_rank != 0) return fail(RTX_ERR_STATE, "rtx_read_reduced_accum: only on rank 0 of a communicator");
    RTX_CK(cudaSetDevice(c->cfg.device));
    RTX_CK(cudaMemcpyAsync(host_out, c->d_total, (size_t)c->cfg.width * c->cfg.height * 16, cudaMemcpyDeviceToHost, c->copy_stream));
    RTX_CK(cudaStreamSynchronize(c->copy_stream));
    return RTX_OK;
}

extern "C" rtx_status rtx_get_counters(rtx_ctx* c, rtx_counters* out) {
    if (!c || !out) return fail(RTX_ERR_ARG, "rtx_get_counters: null argument");
    RTX_ENTER(c);
    memset(out, 0, sizeof *out);
    RTX_CK(cudaStreamSynchronize(c->stream));
    if (c->wb_ready) {
        unsigned long long h[8];
        RTX_CK(cudaMemcpy(h, c->wb.ray_counters, sizeof h, cudaMemcpyDeviceToHost));
        out->closest_rays = h[0]; out->shadow_rays = h[1]; out->paths = h[2];
        if (c->wb2_ready) {
            RTX_CK(cudaMemcpy(h, c->wb2.ray_counters, sizeof h, cudaMemcpyDeviceToHost));
            out->closest_rays += h[0]; out->shadow_rays += h[1]; out->paths += h[2];
        }
    }
    TraceStats ts;
    RTX_CK(cudaMemcpy(&ts, c->d_stats, sizeof ts, cudaMemcpyDeviceToHost));
    out->nodes_visited = ts.nodes; out->tris_tested = ts.tris; out->instances_entered = ts.insts;
    out->shading_replays = ts.replays;
    out->kernel_launches = c->launches;
    return RTX_OK;
}

extern "C" rtx_status rtx_reset_counters(rtx_ctx* c) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    RTX_ENTER(c);
    RTX_CK(cudaStreamSynchronize(c->stream));
    if (c->wb_ready) RTX_CK(cudaMemset(c->wb.ray_counters, 0, 64));
    if (c->wb2_ready) RTX_CK(cudaMemset(c->wb2.ray_counters, 0, 64));
    RTX_CK(cudaMemset(c->d_stats, 0, sizeof(TraceStats)));
    c->launches = 0;
    return RTX_OK;
}

static rtx_status stage_ms(rtx_ctx* c, float* by_kind, float* total) {
    if (!c->pass_timed) return fail(RTX_ERR_STATE, "rtx_last_pass_ms: no pass rendered yet");
    RTX_CK(cudaSetDevice(c->cfg.device));
    for (int k = 0; k < SK_COUNT; k++) by_kind[k] = 0.0f;
    if (c->last_lane == 1) {        // the last pass ran on the second lane (pipelined passes carry no per-launch events)
        RTX_CK(cudaEventSynchronize(c->timing2.ev[1]));
        RTX_CK(cudaEventElapsedTime(total, c->timing2.ev[0], c->timing2.ev[1]));
        return RTX_OK;
    }
    RTX_CK(cudaEventSynchronize(c->timing.ev[1]));
    RTX_CK(cudaEventElapsedTime(total, c->timing.ev[0], c->timing.ev[1]));
    for (int i = 0; i < c->timing.n_marks; i++) {
        float d = 0.0f;
        cudaEvent_t next = (i + 1 < c->timing.n_marks) ? c->timing.ev[3 + i] : c->timing.ev[1];
        RTX_CK(cudaEventElapsedTime(&d, c->timing.ev[2 + i], next));
        by_kind[c->timing.kind[i]] += d;
    }
    return RTX_OK;
}

extern "C" rtx_status rtx_last_pass_ms(rtx_ctx* c, float* trace_ms, float* total_ms) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    float k[SK_COUNT], t = 0.0f;
    rtx_status st = stage_ms(c, k, &t);
    if (st != RTX_OK) return st;
    if (total_ms) *total_ms = t;
    if (trace_ms) *trace_ms = k[SK_CLOSEST];
    return RTX_OK;
}

extern "C" rtx_status rtx_last_pass_stage_ms(rtx_ctx* c, float* ms_by_stage, uint32_t n_stages, float* total_ms) {
    if (!c || !ms_by_stage) return fail(RTX_ERR_ARG, "rtx_last_pass_stage_ms: null argument");
    float k[SK_COUNT], t = 0.0f;
    rtx_status st = stage_ms(c, k, &t);
    if (st != RTX_OK) return st;
    for (uint32_t i = 0; i < n_stages; i++) ms_by_stage[i] = i < (uint32_t)SK_COUNT ? k[i] : 0.0f;
    if (total_ms) *total_ms = t;
    return RTX_OK;
}

extern "C" rtx_status rtx_set_option(rtx_ctx* c, uint32_t option, uint32_t value) {
    if (!c) return fail(RTX_ERR_ARG, "null context");
    RTX_ENTER(c);
    if (option == RTX_OPT_TRACE_STATS) c->trace_stats = value != 0;
    else if (option == RTX_OPT_STAGE_TIMING) c->timing.stage_timing = value != 0;
    else if (option == RTX_OPT_TLAS_REBUILD) c->force_tlas_rebuild = value != 0;
    else if (option == RTX_OPT_PASS_PARTS) {
        if (value < 1u || value > (uint32_t)WAVE_MAX_PARTS) return fail(RTX_ERR_ARG, "rtx_set_option: RTX_OPT_PASS_PARTS must be 1..4");
        c->wb.parts = (int)value;
    }
    else if (option == RTX_OPT_TRACE_FETCH_TH) { if (value > 32u) return fail(RTX_ERR_ARG, "rtx_set_option: RTX_OPT_TRACE_FETCH_TH must be 0..32"); c->fetch_th = (int)value; }
    else if (option == RTX_OPT_TRACE_SCHED) c->sched = (int)(value & 0xffffffu);
    else if (option == RTX_OPT_TRACE_WAVES) { if (value > 8u) return fail(RTX_ERR_ARG, "rtx_set_option: RTX_OPT_TRACE_WAVES must be 0..8"); c->waves = (int)value; }
    else if (option == RTX_OPT_QUEUE_LPT) c->lpt = value != 0;
    else if (option == RTX_OPT_PASS_GRAPH) { c->wb.use_graph = value != 0; c->wb2.use_graph = value != 0; }
    else if (option == RTX_OPT_SHADOW_OVERLAP) c->wb.shadow_overlap = value != 0;
    else if (option == RTX_OPT_PASS_PIPELINE) c->pipeline = value != 0;
    else if (option == RTX_OPT_FRAME_PIPELINE) c->frame_pipeline = value != 0;
    else if (option == RTX_OPT_PART_ROWS) { if (value > 64u && value != 0xffffffffu) return fail(RTX_ERR_ARG, "rtx_set_option: RTX_OPT_PART_ROWS must be 0..64 or 0xffffffff (automatic)"); c->wb.part_rows = value == 0xffffffffu ? -1 : (int)value; }
    else if (option == RTX_OPT_TRACE_CTAS) { if (value > 32u) return fail(RTX_ERR_ARG, "rtx_set_option: RTX_OPT_TRACE_CTAS must be 0..32"); c->ctas_per_sm = (int)value; }
    else return fail(RTX_ERR_ARG, "rtx_set_option: unknown option");
    return RTX_OK;
}

extern "C" rtx_status rtx_selftest_dmath(rtx_ctx* c, uint64_t* out, uint32_t n_out) {
    if (!c || !out || n_out == 0) return fail(RTX_ERR_ARG, "rtx_selftest_dmath: bad argument");
    RTX_ENTER(c);
    unsigned long long h[8] = {0};
    RTX_CK(wave_selftest_dmath(c->stream, h, 8));
    for (uint32_t i = 0; i < n_out; i++) out[i] = i < 8 ? (uint64_t)h[i] : 0;
    return RTX_OK;
}

extern "C" rtx_status rtx_debug_pixel(rtx_ctx* c, uint32_t x, uint32_t y, float* out64) {
    if (!c || !out64 || !c->wb_ready) return fail(RTX_ERR_ARG, "rtx_debug_pixel: bad argument");
    if (x >= c->cfg.width || y >= c->cfg.height) return fail(RTX_ERR_ARG, "rtx_debug_pixel: pixel out of range");
    RTX_ENTER(c);
    SceneData S; memset(&S, 0, sizeof S); S.width = c->cfg.width; S.height = c->cfg.height;
    RTX_CK(wave_debug_pixel(c->wb, S, x, y, c->stream, out64));
    return RTX_OK;
}
