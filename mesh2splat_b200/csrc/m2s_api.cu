// m2s_api.cu — C-ABI implementation (include/m2s.h) over the kernels in m2s_kernels.cu.
// Host orchestration only: context, device-resident scene, launches, counter read-back.
// There is deliberately NO CPU compute path: without a CUDA device every entry point fails.
#include <algorithm>
#include <cmath>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/m2s.h"
#include "m2s_device.cuh"
#include "m2s_prepass.cuh"
#include "m2s_render.cuh"

namespace m2s {
int convert_warps_per_cta(int layout);
size_t tri_frag_bytes(int layout);
cudaError_t convert_configure(int layout, int* raster_blocks_per_sm, int* fragment_blocks_per_sm);
cudaError_t convert_launch(int layout, const ConvertArgs& args, int raster_grid, int fragment_grid, cudaStream_t stream, cudaEvent_t mid);
cudaError_t gather_wait_launch(const unsigned long long* xch, uint32_t world, unsigned long long epoch, unsigned long long gcap,
                               unsigned long long* total_global, uint32_t* status, cudaStream_t stream);
cudaError_t mip_groups_launch(uint32_t* arena, const DTexture& t, uint32_t g0, uint32_t g1, cudaStream_t stream);
cudaError_t vrange_launch(const float4* tris, uint32_t first, uint32_t count, const DRange* ranges, uint32_t nranges, const DPrim* prims,
                          uint32_t ntex, int* minmax, cudaStream_t stream);
cudaError_t vrange_publish_launch(int* minmax, uint32_t ntex, int* host, unsigned long long* host_tag, unsigned long long tag, cudaStream_t stream);
cudaError_t ply_rows_launch(const void* ref96, unsigned long long count, const unsigned long long* d_count,
                            uint32_t format, float mult, void* rows, cudaStream_t stream);
// host-side helpers implemented in m2s_host.cpp
void set_error(const std::string& msg);
}  // namespace m2s

using namespace m2s;

#define M2S_EXPORT extern "C" __attribute__((visibility("default")))

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                          \
            return (_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver) ? M2S_E_NOGPU : M2S_E_CUDA; \
        }                                                                                           \
    } while (0)

struct VRangeSlot {        // v-range reduction of one pipeline chunk: device buffer + pinned host copy + "copy done" event
    int* d_minmax = nullptr;     // [2 * ntex]: sortable-int min | max of v per texture, then 1 non-finite flag (armed: see vrange_publish_kernel)
    int* h_minmax = nullptr;     // pinned + mapped: written by the publish kernel, followed (8-byte aligned) by the tag
    int* h_minmax_dev = nullptr; // its device view
    unsigned long long* h_tag = nullptr;      // host view of the tag
    unsigned long long* h_tag_dev = nullptr;
    unsigned long long tag = 0;               // the tag the current reduction will publish
    cudaEvent_t ev = nullptr;    // recorded behind the publish kernel (error path: a failed launch never writes the tag)
};
struct m2s_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    uint32_t* d_sched = nullptr;             // 8 x 128 B (one scheduler word per cache line)
    unsigned long long* d_counter = nullptr; // running fragment counter
    unsigned long long* d_total = nullptr;   // published count
    uint32_t* d_nitems = nullptr;            // work items queued by the last raster launch
    uint32_t* d_prepass_valid = nullptr;     // counter of the synchronous m2s_prepass
    unsigned long long* h_total = nullptr;   // pinned
    uint32_t* h_status = nullptr;            // pinned + mapped: raised by device-side waits that timed out (fused gather)
    uint32_t* d_status = nullptr;            // its device view
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_mid = nullptr;
    cudaEvent_t ev_r[4] = {};                // timing of the synchronous sort / splat (created on first use)
    // convert_host pipeline: a second stream for the downloads, per-chunk counts and events
    static constexpr int kMaxChunks = 8;
    cudaStream_t stream2 = nullptr;
    cudaStream_t stream3 = nullptr;              // uploads of the host pipeline: the copy engine keeps going while chunk kernels run
    cudaStream_t up = nullptr;                   // stream triangle chunks are uploaded on (= stream, or stream3 inside the pipeline)
    // the host pipeline keeps TWO copy engines busy in the upload direction (one stream delivers 35 GB/s on these boxes, two
    // 51 GB/s: scripts/pcie_probe.py) and never puts a kernel between two copies of a stream (a copy behind a kernel of
    // its own stream waits for it: with the v-range and mip kernels on the copy stream every chunk cost ~40 us of bubbles)
    cudaStream_t stream4 = nullptr;              // texture rows
    cudaStream_t stream5 = nullptr;              // v-range reductions and their 8-byte results
    cudaStream_t tex_up = nullptr;               // stream texture rows are uploaded on (= up, or stream4 inside the pipeline)
    cudaStream_t mip = nullptr;                  // stream their mip rows are generated on (= tex_up, or the compute stream inside the pipeline)
    cudaStream_t aux = nullptr;                  // stream the v-range reductions run on (= up, or stream5 inside the pipeline)
    cudaEvent_t ev_tri[kMaxChunks] = {};         // "chunk c's triangles are resident"
    cudaEvent_t ev_up[kMaxChunks] = {};          // "chunk c's texture rows are resident"
    cudaEvent_t ev_alloc = nullptr;
    unsigned long long* d_chunk_tot = nullptr;   // [kMaxChunks]
    unsigned long long* h_chunk_tot = nullptr;   // pinned + mapped: {count, tag} per chunk, written by the raster kernel
    unsigned long long host_seq = 0;             // tag generator
    // file writer: two pinned staging buffers (download of block i overlaps the write of block i-1)
    static constexpr size_t kStageBytes = 32u << 20;
    unsigned char* h_stage[2] = {nullptr, nullptr};
    cudaEvent_t ev_chunk[kMaxChunks] = {};
    VRangeSlot vr[kMaxChunks];        // v-range reductions of the host pipeline (lazy texture upload)
    uint32_t vr_ntex = 0;                    // textures the slots are sized for
    bool vr_dirty = false;                   // a pipeline was abandoned half way: the device copies must be re-armed
    static constexpr int kLayouts = 5;
    int blocks_per_sm[kLayouts] = {};       // raster kernel (persistent)
    int frag_blocks_per_sm[kLayouts] = {};  // fragment kernel
    unsigned long long epoch = 0;            // pairs up the ranks' calls of the fused gather
    bool dirty = true;                       // scheduler state needs a memset before the next launch
    // scratch owned by the context (grown on demand)
    void* d_out = nullptr;      size_t out_bytes = 0;       // convert_host output
    unsigned long long* d_keys = nullptr; size_t keys_bytes = 0;
    // intermediates between the raster and the fragment kernel
    void* d_trifrag = nullptr;  size_t trifrag_bytes = 0;   // TriRec per triangle of the shard
    void* d_items = nullptr;    size_t items_bytes = 0;     // FragItem queue
};

struct m2s_dscene {
    float4* d_tris = nullptr;
    uint64_t ntri = 0;
    DRange* d_ranges = nullptr;
    uint32_t nranges = 0;
    DPrim* d_prims = nullptr;
    uint32_t nprims = 0;
    DTexture* d_texs = nullptr;
    uint32_t* d_arena = nullptr;  // all mip chains of all textures
    uint32_t ntex = 0;
    std::vector<DTexture> h_texs;
    std::vector<void*> allocs;
    // lazily uploaded textures (host pipeline): level-0 rows travel in groups of kTexGroupRows rows, each group brings
    // its own rows of the mip levels 1..4 with it (a group of 16 rows is closed under the 2x2 box filter)
    std::vector<const uint8_t*> h_rgba;              // host images (valid for the duration of the call that uploads lazily)
    std::vector<std::vector<uint8_t>> present;       // per texture, per row group: already on the device
    uint64_t h2d_bytes = 0;                          // payload copied host -> device for this scene so far
};
constexpr uint32_t kTexGroupRows = 16;               // = 2^M2S_MAX_MIP_LEVEL

static unsigned long long* g_trace = nullptr;  // debugging aid for M2S_TRACE builds (scripts/trace_raster.py)
extern "C" __attribute__((visibility("default"))) void m2s_debug_set_trace(void* p) { g_trace = (unsigned long long*)p; }

// Context scratch grows on the stream that will USE it: the free of the old block is ordered after the kernels
// already enqueued there, the new block is ready before the next one.  (A caller that alternates between streams
// without synchronising them must not share one context: documented in m2s.h.)
static m2s_status grow(m2s_ctx* ctx, void** p, size_t* have, size_t need, cudaStream_t stream = nullptr) {
    if (*have >= need) return M2S_OK;
    if (!stream) stream = ctx->stream;
    if (*p) CUDA_TRY(cudaFreeAsync(*p, stream));
    *p = nullptr; *have = 0;
    CUDA_TRY(cudaMallocAsync(p, need + need / 4, stream));  // 25 % head room: density sweeps do not reallocate at every step
    *have = need + need / 4;
    return M2S_OK;
}

// ---- housekeeping ---------------------------------------------------------------------------
M2S_EXPORT int m2s_version(void) { return M2S_VERSION; }

M2S_EXPORT const char* m2s_status_string(m2s_status s) {
    switch (s) {
        case M2S_OK: return "ok";
        case M2S_E_INVALID: return "invalid argument";
        case M2S_E_NOGPU: return "no CUDA device";
        case M2S_E_CUDA: return "CUDA error";
        case M2S_E_CAPACITY: return "output capacity exceeded";
        case M2S_E_IO: return "I/O error";
        case M2S_E_FORMAT: return "unsupported or malformed input";
    }
    return "unknown";
}

M2S_EXPORT uint32_t m2s_record_stride(uint32_t layout) {
    switch (layout) {
        case M2S_LAYOUT_REF96: return 96;
        case M2S_LAYOUT_PACKED56: return 56;
        case M2S_LAYOUT_PLY_STANDARD: return 248;
        case M2S_LAYOUT_PLY_PBR: return 76;
        case M2S_LAYOUT_PLY_COMPRESSED: return 48;
    }
    return 0;
}

M2S_EXPORT uint64_t m2s_reference_capacity(uint32_t R, uint32_t primitive_count) {
    const uint64_t mc = primitive_count ? primitive_count : 1;
    return std::min<uint64_t>((uint64_t)R * R * 6ull * mc, M2S_REFERENCE_MAX_GAUSSIANS);
}

M2S_EXPORT void m2s_params_default(m2s_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->resolution = 520;  // int(16 + 0.5 * (1024 - 16)): ImGuiUI.cpp:512 with the default quality
    p->gaussian_std = 0.65f;
    p->layout = M2S_LAYOUT_REF96;
}

M2S_EXPORT m2s_status m2s_ctx_create(int device, m2s_ctx** out) {
    if (!out) { set_error("m2s_ctx_create: out is NULL"); return M2S_E_INVALID; }
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        set_error(std::string("no CUDA device available: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0"));
        return M2S_E_NOGPU;
    }
    if (device < 0 || device >= n) { set_error("m2s_ctx_create: bad device index"); return M2S_E_INVALID; }
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { set_error("mesh2splat_b200 kernels are built for sm_100a only"); return M2S_E_NOGPU; }
    m2s_ctx* c = new m2s_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    cudaMemPool_t pool;
    CUDA_TRY(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t thresh = UINT64_MAX;  // keep freed blocks cached: uploads in steady state never hit cudaMalloc
    CUDA_TRY(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thresh));
    CUDA_TRY(cudaMalloc(&c->d_sched, 8 * 128));
    CUDA_TRY(cudaMalloc(&c->d_counter, sizeof(unsigned long long)));
    CUDA_TRY(cudaMalloc(&c->d_total, sizeof(unsigned long long)));
    CUDA_TRY(cudaMalloc(&c->d_nitems, sizeof(uint32_t)));
    CUDA_TRY(cudaMallocHost(&c->h_total, sizeof(unsigned long long)));
    CUDA_TRY(cudaHostAlloc(&c->h_status, sizeof(uint32_t), cudaHostAllocMapped));
    *c->h_status = 0;
    CUDA_TRY(cudaHostGetDevicePointer((void**)&c->d_status, c->h_status, 0));
    CUDA_TRY(cudaEventCreate(&c->ev0));
    CUDA_TRY(cudaEventCreate(&c->ev1));
    CUDA_TRY(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&c->stream3, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&c->stream4, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&c->stream5, cudaStreamNonBlocking));
    c->up = c->tex_up = c->mip = c->aux = c->stream;
    for (int i = 0; i < m2s_ctx::kMaxChunks; ++i) CUDA_TRY(cudaEventCreateWithFlags(&c->ev_tri[i], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&c->ev_alloc, cudaEventDisableTiming));
    for (int i = 0; i < m2s_ctx::kMaxChunks; ++i) CUDA_TRY(cudaEventCreateWithFlags(&c->ev_up[i], cudaEventDisableTiming));
    CUDA_TRY(cudaMalloc(&c->d_chunk_tot, m2s_ctx::kMaxChunks * sizeof(unsigned long long)));
    CUDA_TRY(cudaHostAlloc(&c->h_chunk_tot, 2 * m2s_ctx::kMaxChunks * sizeof(unsigned long long), cudaHostAllocMapped));
    std::memset(c->h_chunk_tot, 0, 2 * m2s_ctx::kMaxChunks * sizeof(unsigned long long));
    for (int i = 0; i < m2s_ctx::kMaxChunks; ++i) CUDA_TRY(cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming));
    for (int l = 0; l < m2s_ctx::kLayouts; ++l) {
        CUDA_TRY(convert_configure(l, &c->blocks_per_sm[l], &c->frag_blocks_per_sm[l]));
        if (c->blocks_per_sm[l] < 1 || c->frag_blocks_per_sm[l] < 1) { set_error("conversion kernel does not fit on this device"); return M2S_E_CUDA; }
    }
    *out = c;
    return M2S_OK;
}

M2S_EXPORT void m2s_ctx_destroy(m2s_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->d_out) cudaFreeAsync(c->d_out, c->stream);
    if (c->d_keys) cudaFreeAsync(c->d_keys, c->stream);
    if (c->d_trifrag) cudaFreeAsync(c->d_trifrag, c->stream);
    if (c->d_items) cudaFreeAsync(c->d_items, c->stream);
    cudaStreamSynchronize(c->stream);
    if (c->d_prepass_valid) cudaFree(c->d_prepass_valid);
    cudaFree(c->d_sched); cudaFree(c->d_counter); cudaFree(c->d_total); cudaFree(c->d_nitems);
    cudaFreeHost(c->h_total);
    if (c->h_status) cudaFreeHost(c->h_status);
    cudaFree(c->d_chunk_tot); cudaFreeHost(c->h_chunk_tot);
    for (int i = 0; i < 2; ++i) if (c->h_stage[i]) cudaFreeHost(c->h_stage[i]);
    for (auto& v : c->vr) { if (v.d_minmax) cudaFree(v.d_minmax); if (v.h_minmax) cudaFreeHost(v.h_minmax); if (v.ev) cudaEventDestroy(v.ev); }
    for (int i = 0; i < m2s_ctx::kMaxChunks; ++i) if (c->ev_chunk[i]) cudaEventDestroy(c->ev_chunk[i]);
    cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1); if (c->ev_mid) cudaEventDestroy(c->ev_mid);
    for (cudaEvent_t e : c->ev_r) if (e) cudaEventDestroy(e);
    if (c->stream2) cudaStreamDestroy(c->stream2);
    if (c->stream3) cudaStreamDestroy(c->stream3);
    if (c->stream4) cudaStreamDestroy(c->stream4);
    if (c->stream5) cudaStreamDestroy(c->stream5);
    for (int i = 0; i < m2s_ctx::kMaxChunks; ++i) if (c->ev_tri[i]) cudaEventDestroy(c->ev_tri[i]);
    if (c->ev_alloc) cudaEventDestroy(c->ev_alloc);
    for (int i = 0; i < m2s_ctx::kMaxChunks; ++i) if (c->ev_up[i]) cudaEventDestroy(c->ev_up[i]);
    cudaStreamDestroy(c->stream);
    delete c;
}

M2S_EXPORT int m2s_ctx_device(const m2s_ctx* c) { return c ? c->device : -1; }
// Device-side conditions the enqueue-only entry points cannot return: call after synchronising the stream.
M2S_EXPORT m2s_status m2s_ctx_status(m2s_ctx* c) {
    if (!c) { set_error("m2s_ctx_status: ctx is NULL"); return M2S_E_INVALID; }
    const uint32_t v = __atomic_exchange_n(c->h_status, 0u, __ATOMIC_ACQ_REL);
    if (v == 0) return M2S_OK;
    if (v == kStatusSplatCapacity) {
        set_error("m2s_splat_enqueue: the quads touch more (tile, quad) pairs than max_pairs; the G-buffer was left cleared");
        return M2S_E_CAPACITY;
    }
    c->dirty = true;
    set_error(std::string("fused gather: a peer rank did not publish its ") + ((v & 1u) ? "count" : "completion flag") +
              " within 2 s (did every rank call m2s_convert_gather_enqueue the same number of times?)");
    return M2S_E_CUDA;
}
M2S_EXPORT int m2s_ctx_sm_count(const m2s_ctx* c) { return c ? c->sm_count : 0; }

// ---- inputs ---------------------------------------------------------------------------------
M2S_EXPORT m2s_status m2s_compute_bboxes(const float* tris, m2s_primitive* prims, uint32_t nprim, int cumulative) {
    if ((!tris && nprim) || (!prims && nprim)) { set_error("m2s_compute_bboxes: NULL input"); return M2S_E_INVALID; }
    // SceneManager.cpp:476-477,514-520,527 — minBB/maxBB live outside the mesh loop
    float mn[3] = {3.402823466e+38f, 3.402823466e+38f, 3.402823466e+38f};
    float mx[3] = {-3.402823466e+38f, -3.402823466e+38f, -3.402823466e+38f};
    for (uint32_t p = 0; p < nprim; ++p) {
        if (!cumulative)
            for (int c = 0; c < 3; ++c) { mn[c] = 3.402823466e+38f; mx[c] = -3.402823466e+38f; }
        const uint64_t a = prims[p].first_triangle, b = a + prims[p].triangle_count;
        for (uint64_t t = a; t < b; ++t)
            for (int k = 0; k < 3; ++k)
                for (int c = 0; c < 3; ++c) {
                    const float v = tris[t * M2S_FLOATS_PER_TRIANGLE + M2S_FLOATS_PER_VERTEX * k + c];
                    mn[c] = std::min(mn[c], v);
                    mx[c] = std::max(mx[c], v);
                }
        for (int c = 0; c < 3; ++c) { prims[p].bbox_min[c] = mn[c]; prims[p].bbox_max[c] = mx[c]; }
    }
    return M2S_OK;
}

static uint32_t mip_levels(uint32_t w, uint32_t h) {
    uint32_t m = std::max(w, h), q = 0;
    while ((m >> (q + 1)) != 0) ++q;
    return std::min<uint32_t>(q, M2S_MAX_MIP_LEVEL) + 1;
}

M2S_EXPORT void m2s_scene_free(m2s_ctx* ctx, m2s_dscene* s) {
    if (!s) return;
    if (ctx) {
        cudaSetDevice(ctx->device);
        for (void* p : s->allocs) cudaFreeAsync(p, ctx->stream);
    }
    delete s;
}

// rows [g0, g1) x kTexGroupRows of texture t: one contiguous H2D copy, then the rows of levels 1.. that they determine
struct MipRun { uint32_t t, g0, g1; };   // levels 1.. of the row groups [g0, g1) of texture t are still to be generated
static m2s_status upload_texture_groups(m2s_ctx* ctx, m2s_dscene* d, uint32_t t, uint32_t g0, uint32_t g1, std::vector<MipRun>* deferred = nullptr) {
    const DTexture& dt = d->h_texs[t];
    const uint32_t H = dt.h[0], W = dt.w[0];
    const uint32_t r0 = g0 * kTexGroupRows, r1 = std::min<uint32_t>(H, g1 * kTexGroupRows);
    if (r0 >= r1) return M2S_OK;
    CUDA_TRY(cudaMemcpyAsync(d->d_arena + dt.off[0] + (size_t)r0 * W, d->h_rgba[t] + (size_t)r0 * W * 4, (size_t)(r1 - r0) * W * 4,
                             cudaMemcpyHostToDevice, ctx->tex_up));
    // level-l row j needs level-(l-1) rows 2j, 2j+1: inside the same 16-row group — all levels in one launch; inside the
    // host pipeline the launch is left to the caller (on the compute stream, behind an event: no kernel on the copy stream)
    const uint32_t ge = std::min<uint32_t>(g1, (H + kTexGroupRows - 1) / kTexGroupRows);
    if (deferred) deferred->push_back({t, g0, ge});
    else CUDA_TRY(mip_groups_launch(d->d_arena, dt, g0, ge, ctx->tex_up));
    for (uint32_t g = g0; g < g1 && g < d->present[t].size(); ++g) d->present[t][g] = 1;
    d->h2d_bytes += (uint64_t)(r1 - r0) * W * 4;
    return M2S_OK;
}

// Which texture rows can the triangles [lo, hi) sample?  The v-range per texture is reduced ON THE GPU from the triangles
// already uploaded (vrange_launch: the host would have to stream the same 144 B/triangle through one core — ~1 ms for
// the bench scene), copied back (8 bytes per texture) and turned into 16-row groups here: +-3 groups cover the
// footprints of all five mip levels (level l reaches 2^(l+1) level-0 rows beyond the sample point, plus the drift of
// non-power-of-two chains) and the REPEAT wrap at both ends; a range whose v spans a whole period (or is not finite)
// takes the whole image.
static float sortable_to_float(int i) { i ^= (i >> 31) & 0x7fffffff; float f; std::memcpy(&f, &i, 4); return f; }

static m2s_status vrange_enqueue(m2s_ctx* ctx, m2s_dscene* d, uint64_t lo, uint64_t hi, int slot);
// `idle` (optional) is called while the host waits for the reduction: the host pipeline enqueues ready downloads there
template <class Idle>
static m2s_status upload_groups_from_vrange(m2s_ctx* ctx, m2s_dscene* d, int slot, Idle idle, std::vector<MipRun>* deferred = nullptr) {
    const uint32_t nt = d->ntex;
    if (!nt) return M2S_OK;
    for (uint32_t spin = 0;; ++spin) {
        if (__atomic_load_n(ctx->vr[slot].h_tag, __ATOMIC_ACQUIRE) == ctx->vr[slot].tag) break;   // the values are ordered before the tag
        if ((spin & 255u) == 255u) {  // a failed launch never writes the tag: ask the stream now and then
            const cudaError_t q = cudaEventQuery(ctx->vr[slot].ev);
            if (q == cudaSuccess) { if (__atomic_load_n(ctx->vr[slot].h_tag, __ATOMIC_ACQUIRE) == ctx->vr[slot].tag) break; }
            else if (q != cudaErrorNotReady) { set_error(std::string("v-range reduction: ") + cudaGetErrorString(q)); return M2S_E_CUDA; }
        }
        const cudaError_t ie = idle();
        if (ie != cudaSuccess) { set_error(std::string("convert_host download: ") + cudaGetErrorString(ie)); return M2S_E_CUDA; }
    }
    const int* mm = ctx->vr[slot].h_minmax;
    const bool finite = mm[2 * nt] == 0;
    for (uint32_t t = 0; t < nt; ++t) {
        if (mm[t] > mm[nt + t]) continue;  // no triangle of the range samples this texture
        const uint32_t ng = (uint32_t)d->present[t].size();
        std::vector<uint8_t> need(ng, 0);
        const float vmin = sortable_to_float(mm[t]), vmax = sortable_to_float(mm[nt + t]);
        const float fl = std::floor(vmin);
        if (!finite || !(vmax - fl <= 1.0f) || ng <= 8) std::fill(need.begin(), need.end(), 1);  // v = 1.0 exactly wraps to the first rows (modulo below)
        else {
            const float H = (float)d->h_texs[t].h[0];
            const long long ra = (long long)std::floor((vmin - fl) * H) - 1, rb = (long long)std::floor((vmax - fl) * H) + 1;
            const long long ga = ra / (long long)kTexGroupRows - 3 - (ra < 0), gb = rb / (long long)kTexGroupRows + 3;
            if (gb - ga + 1 >= (long long)ng) std::fill(need.begin(), need.end(), 1);
            else for (long long g = ga; g <= gb; ++g) need[(size_t)(((g % ng) + ng) % ng)] = 1;  // REPEAT: wraps at both ends
        }
        for (uint32_t g = 0; g < ng;) {
            if (!need[g] || d->present[t][g]) { ++g; continue; }
            uint32_t e = g;
            while (e < ng && need[e] && !d->present[t][e]) ++e;
            m2s_status st = upload_texture_groups(ctx, d, t, g, e, deferred);
            if (st != M2S_OK) return st;
            g = e;
        }
    }
    return M2S_OK;
}

// enqueue on the context stream: reduce the v-range of triangles [lo, hi) (already on the device) per texture, copy it
// to the slot's pinned buffer, record the slot's event
static m2s_status vrange_enqueue(m2s_ctx* ctx, m2s_dscene* d, uint64_t lo, uint64_t hi, int slot) {
    const uint32_t nt = d->ntex;
    if (!nt) return M2S_OK;
    if (ctx->vr_ntex != nt) {  // (re)size and arm every slot: the armed layout (min block | max block | flag) depends on the texture count
        for (auto& v : ctx->vr) {
            if (v.d_minmax) { cudaFree(v.d_minmax); v.d_minmax = nullptr; }
            if (v.h_minmax) { cudaFreeHost(v.h_minmax); v.h_minmax = nullptr; }
        }
        ctx->vr_ntex = 0;
        for (auto& v : ctx->vr) {
            const size_t nints = 2 * (size_t)nt + 1, tag_off = (nints * sizeof(int) + 7) & ~(size_t)7;
            CUDA_TRY(cudaMalloc(&v.d_minmax, nints * sizeof(int)));
            std::vector<int> arm(nints, 0);
            for (size_t i = 0; i < nt; ++i) { arm[i] = 0x7f7f7f7f; arm[nt + i] = (int)0x80808080; }
            CUDA_TRY(cudaMemcpy(v.d_minmax, arm.data(), nints * sizeof(int), cudaMemcpyHostToDevice));
            CUDA_TRY(cudaHostAlloc(&v.h_minmax, tag_off + 8, cudaHostAllocMapped));
            std::memset(v.h_minmax, 0, tag_off + 8);
            CUDA_TRY(cudaHostGetDevicePointer((void**)&v.h_minmax_dev, v.h_minmax, 0));
            v.h_tag = reinterpret_cast<unsigned long long*>(reinterpret_cast<unsigned char*>(v.h_minmax) + tag_off);
            v.h_tag_dev = reinterpret_cast<unsigned long long*>(reinterpret_cast<unsigned char*>(v.h_minmax_dev) + tag_off);
            if (!v.ev) CUDA_TRY(cudaEventCreateWithFlags(&v.ev, cudaEventDisableTiming));
        }
        ctx->vr_ntex = nt;
    }
    VRangeSlot& v = ctx->vr[slot];
    // min <- 0x7f7f7f7f (above every finite float's key), max <- 0x80808080 (below), flag <- 0
    // d_minmax is armed (at allocation, then by every publish kernel); a conversion that failed in between re-arms it
    if (ctx->vr_dirty) {
        for (auto& w : ctx->vr) {
            CUDA_TRY(cudaMemsetAsync(w.d_minmax, 0x7f, nt * sizeof(int), ctx->aux));
            CUDA_TRY(cudaMemsetAsync(w.d_minmax + nt, 0x80, nt * sizeof(int), ctx->aux));
            CUDA_TRY(cudaMemsetAsync(w.d_minmax + 2 * nt, 0, sizeof(int), ctx->aux));
        }
        ctx->vr_dirty = false;
    }
    if (hi > lo)
        CUDA_TRY(vrange_launch(d->d_tris, (uint32_t)lo, (uint32_t)(hi - lo), d->d_ranges, d->nranges, d->d_prims, nt, v.d_minmax, ctx->aux));
    v.tag = ++ctx->host_seq;
    CUDA_TRY(vrange_publish_launch(v.d_minmax, nt, v.h_minmax_dev, v.h_tag_dev, v.tag, ctx->aux));
    CUDA_TRY(cudaEventRecord(v.ev, ctx->aux));
    return M2S_OK;
}

// first_tris < triangle_count: only that many triangles are copied here (the caller streams the rest into
// d_tris itself, interleaved with its launches) and the stream is not synchronised.
// lazy_tex: the images are NOT copied here; the caller brings in the row groups its triangle ranges sample with
// ensure_textures_for_range (m2s_convert_host pipelines them with the triangle chunks, m2s_scene_upload_range
// uploads what one shard needs).
static m2s_status scene_upload_impl(m2s_ctx* ctx, const m2s_scene* sc, m2s_dscene** out, uint64_t first_tris, bool sync,
                                    uint64_t tri_offset = 0, bool lazy_tex = false) {
    if (!ctx || !sc || !out) { set_error("m2s_scene_upload: NULL argument"); return M2S_E_INVALID; }
    *out = nullptr;
    if (sc->triangle_count && !sc->triangles) { set_error("m2s_scene_upload: triangles is NULL"); return M2S_E_INVALID; }
    if (sc->triangle_count >= (1ull << 32) - 64) { set_error("m2s_scene_upload: too many triangles (< 2^32 supported)"); return M2S_E_INVALID; }
    if ((sc->primitive_count && !sc->primitives) || (sc->texture_count && !sc->textures)) {
        set_error("m2s_scene_upload: primitive/texture table is NULL"); return M2S_E_INVALID;
    }
    // primitive ranges: inside the triangle list, pairwise disjoint
    std::vector<DRange> ranges;
    std::vector<DPrim> prims(sc->primitive_count);
    for (uint32_t p = 0; p < sc->primitive_count; ++p) {
        const m2s_primitive& src = sc->primitives[p];
        if (src.first_triangle + src.triangle_count > sc->triangle_count) {
            set_error("m2s_scene_upload: primitive range exceeds the triangle list"); return M2S_E_INVALID;
        }
        const int32_t ti[3] = {src.albedo_texture, src.normal_texture, src.metallic_roughness_texture};
        for (int m = 0; m < 3; ++m) {
            if (ti[m] >= (int32_t)sc->texture_count) { set_error("m2s_scene_upload: texture index out of range"); return M2S_E_INVALID; }
            prims[p].tex[m] = ti[m] < 0 ? -1 : ti[m];
        }
        for (int c = 0; c < 3; ++c) { prims[p].bmin[c] = src.bbox_min[c]; prims[p].bmax[c] = src.bbox_max[c]; }
        for (int c = 0; c < 4; ++c) prims[p].factor[c] = src.base_color_factor[c];
        prims[p].pad = 0;
        if (src.triangle_count)
            ranges.push_back({(uint32_t)src.first_triangle, (uint32_t)(src.first_triangle + src.triangle_count), p, 0});
    }
    std::sort(ranges.begin(), ranges.end(), [](const DRange& a, const DRange& b) { return a.first < b.first; });
    for (size_t i = 1; i < ranges.size(); ++i)
        if (ranges[i].first < ranges[i - 1].end) { set_error("m2s_scene_upload: primitive triangle ranges overlap"); return M2S_E_INVALID; }
    for (uint32_t t = 0; t < sc->texture_count; ++t)
        if (!sc->textures[t].rgba || !sc->textures[t].width || !sc->textures[t].height ||
            sc->textures[t].width > 32768 || sc->textures[t].height > 32768) {
            set_error("m2s_scene_upload: bad texture"); return M2S_E_INVALID;
        }

    CUDA_TRY(cudaSetDevice(ctx->device));
    m2s_dscene* d = new m2s_dscene();
    auto fail = [&](m2s_status st) { m2s_scene_free(ctx, d); return st; };
#define UP_TRY(expr)                                                                 \
    do {                                                                             \
        cudaError_t _e = (expr);                                                     \
        if (_e != cudaSuccess) {                                                     \
            set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));           \
            return fail(M2S_E_CUDA);                                                 \
        }                                                                            \
    } while (0)
    auto dalloc = [&](void** p, size_t bytes) -> cudaError_t {
        cudaError_t e = cudaMallocAsync(p, std::max<size_t>(bytes, 16), ctx->stream);
        if (e == cudaSuccess) d->allocs.push_back(*p);
        return e;
    };
    d->ntri = sc->triangle_count;
    UP_TRY(dalloc((void**)&d->d_tris, sc->triangle_count * (size_t)kTriBytes));
    if (sc->triangle_count && tri_offset < sc->triangle_count && first_tris)  // triangles [tri_offset, tri_offset + first_tris)
        UP_TRY(cudaMemcpyAsync(reinterpret_cast<unsigned char*>(d->d_tris) + tri_offset * (size_t)kTriBytes,
                               reinterpret_cast<const unsigned char*>(sc->triangles) + tri_offset * (size_t)kTriBytes,
                               std::min<uint64_t>(first_tris, sc->triangle_count - tri_offset) * (size_t)kTriBytes, cudaMemcpyHostToDevice, ctx->stream));
    if (sc->triangle_count && tri_offset < sc->triangle_count && first_tris)
        d->h2d_bytes += std::min<uint64_t>(first_tris, sc->triangle_count - tri_offset) * (uint64_t)kTriBytes;
    d->nranges = (uint32_t)ranges.size();
    UP_TRY(dalloc((void**)&d->d_ranges, ranges.size() * sizeof(DRange)));
    if (!ranges.empty())
        UP_TRY(cudaMemcpyAsync(d->d_ranges, ranges.data(), ranges.size() * sizeof(DRange), cudaMemcpyHostToDevice, ctx->stream));
    d->nprims = sc->primitive_count;
    UP_TRY(dalloc((void**)&d->d_prims, prims.size() * sizeof(DPrim)));
    if (!prims.empty())
        UP_TRY(cudaMemcpyAsync(d->d_prims, prims.data(), prims.size() * sizeof(DPrim), cudaMemcpyHostToDevice, ctx->stream));
    // textures: ONE arena for all mip chains (levels addressed by 32-bit texel offsets); levels 1..
    // are built on the GPU
    d->ntex = sc->texture_count;
    d->h_texs.resize(sc->texture_count);
    size_t arena_texels = 64;
    for (uint32_t t = 0; t < sc->texture_count; ++t) {
        DTexture& dt = d->h_texs[t];
        std::memset(&dt, 0, sizeof(dt));
        dt.nlevels = mip_levels(sc->textures[t].width, sc->textures[t].height);
        uint32_t w = sc->textures[t].width, h = sc->textures[t].height;
        for (uint32_t l = 0; l < (uint32_t)kMaxLevels; ++l) {
            if (l < dt.nlevels) {
                dt.w[l] = (uint16_t)w; dt.h[l] = (uint16_t)h;
                if (arena_texels + (size_t)w * h >= (1ull << 32)) { set_error("m2s_scene_upload: textures exceed the 16 GiB arena"); return fail(M2S_E_INVALID); }
                dt.off[l] = (uint32_t)arena_texels;
                arena_texels += (size_t)w * h;
                arena_texels = (arena_texels + 63) & ~(size_t)63;  // 256-byte aligned levels
                w = std::max(1u, w / 2); h = std::max(1u, h / 2);
            } else { dt.w[l] = dt.w[dt.nlevels - 1]; dt.h[l] = dt.h[dt.nlevels - 1]; dt.off[l] = dt.off[dt.nlevels - 1]; }
        }
    }
    UP_TRY(dalloc((void**)&d->d_arena, arena_texels * 4));
    d->h_rgba.resize(sc->texture_count);
    d->present.resize(sc->texture_count);
    for (uint32_t t = 0; t < sc->texture_count; ++t) {
        const uint32_t ngroups = (d->h_texs[t].h[0] + kTexGroupRows - 1) / kTexGroupRows;
        d->h_rgba[t] = sc->textures[t].rgba;
        d->present[t].assign(ngroups, 0);
        if (!lazy_tex) {
            m2s_status st = upload_texture_groups(ctx, d, t, 0, ngroups);
            if (st != M2S_OK) return fail(st);
        }
    }
    UP_TRY(dalloc((void**)&d->d_texs, d->h_texs.size() * sizeof(DTexture)));
    if (!d->h_texs.empty())
        UP_TRY(cudaMemcpyAsync(d->d_texs, d->h_texs.data(), d->h_texs.size() * sizeof(DTexture), cudaMemcpyHostToDevice, ctx->stream));
    if (sync) UP_TRY(cudaStreamSynchronize(ctx->stream));
#undef UP_TRY
    *out = d;
    return M2S_OK;
}

M2S_EXPORT m2s_status m2s_scene_upload(m2s_ctx* ctx, const m2s_scene* sc, m2s_dscene** out) {
    return scene_upload_impl(ctx, sc, out, UINT64_MAX, true);
}


M2S_EXPORT uint64_t m2s_scene_h2d_bytes(const m2s_dscene* s) { return s ? s->h2d_bytes : 0; }

M2S_EXPORT m2s_status m2s_scene_read_mip(m2s_ctx* ctx, const m2s_dscene* s, uint32_t texture, uint32_t level, uint8_t* dst,
                                         uint32_t* width, uint32_t* height) {
    if (!ctx || !s || !dst) { set_error("m2s_scene_read_mip: NULL argument"); return M2S_E_INVALID; }
    if (texture >= s->ntex || level >= s->h_texs[texture].nlevels) { set_error("m2s_scene_read_mip: out of range"); return M2S_E_INVALID; }
    const DTexture& t = s->h_texs[texture];
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaMemcpyAsync(dst, s->d_arena + t.off[level], (size_t)t.w[level] * t.h[level] * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (width) *width = t.w[level];
    if (height) *height = t.h[level];
    return M2S_OK;
}

// ---- the hot path -----------------------------------------------------------------------------
static uint64_t effective_cap(const m2s_dscene* s, const m2s_params* p, uint64_t out_capacity) {
    uint64_t cap = p->max_gaussians;
    if (cap == 0) cap = (p->flags & M2S_FLAG_UNCAPPED) ? out_capacity : m2s_reference_capacity(p->resolution, s->nprims);
    return std::min(cap, out_capacity);
}

static m2s_status convert_enqueue_impl(m2s_ctx* ctx, const m2s_dscene* s, const m2s_params* p, void* d_out, uint64_t out_capacity,
                                       uint64_t* d_keys, uint64_t* d_total, void* stream_, const m2s_peers* peers,
                                       const unsigned long long* prev_totals = nullptr, uint32_t nprev = 0,
                                       unsigned long long* host_total = nullptr, unsigned long long host_tag = 0, cudaEvent_t mid = nullptr) {
    if (!ctx || !s || !p) { set_error("m2s_convert: NULL argument"); return M2S_E_INVALID; }
    if (p->resolution < 1 || p->resolution > 4096) { set_error("m2s_convert: resolution must be in 1..4096"); return M2S_E_INVALID; }
    if (p->layout > M2S_LAYOUT_PLY_COMPRESSED) { set_error("m2s_convert: unknown layout"); return M2S_E_INVALID; }
    if (!peers && !d_out && out_capacity) { set_error("m2s_convert: output buffer is NULL"); return M2S_E_INVALID; }
    if (peers) {
        if (peers->world < 1 || peers->world > M2S_MAX_PEERS || peers->rank >= peers->world) { set_error("m2s_convert_gather: bad world/rank"); return M2S_E_INVALID; }
        if (p->layout > M2S_LAYOUT_PACKED56) { set_error("m2s_convert_gather: layouts REF96 and PACKED56 only"); return M2S_E_INVALID; }
        for (uint32_t r = 0; r < peers->world; ++r)
            if (!peers->out[r] || !peers->xch[r] || (reinterpret_cast<uintptr_t>(peers->out[r]) & 15u)) { set_error("m2s_convert_gather: NULL or misaligned peer buffer"); return M2S_E_INVALID; }
    }
    if (!(p->gaussian_std > 0.0f) && p->layout != M2S_LAYOUT_REF96) { set_error("m2s_convert: gaussian_std must be > 0"); return M2S_E_INVALID; }
    uint64_t first = std::min<uint64_t>(p->first_triangle, s->ntri);
    uint64_t count = p->triangle_count;
    if (count == 0 || first + count > s->ntri) count = s->ntri - first;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : ctx->stream;
    const uint64_t cap = effective_cap(s, p, out_capacity);
    const int klayout = (int)p->layout;  // every layout, the .ply rows included, is written by the fragment kernel itself
    void* kout = d_out;
    if (reinterpret_cast<uintptr_t>(kout) & 15u) { set_error("m2s_convert: the output buffer must be 16-byte aligned"); return M2S_E_INVALID; }
    const int grid = ctx->sm_count * ctx->blocks_per_sm[klayout];
    // work-unit size: as large as 32 triangles, but small enough that every warp of the grid gets the
    // same number of units (a 70 k-triangle mesh is only ~1 unit of 32 per resident warp)
    uint64_t unit_tris, n_units;
    {
        const uint64_t warps = (uint64_t)grid * convert_warps_per_cta(klayout);
        const uint64_t rounds = std::max<uint64_t>(1, (count + warps * kUnitTris - 1) / (warps * kUnitTris));
        unit_tris = (count + warps * rounds - 1) / (warps * rounds);
        unit_tris = std::min<uint64_t>(std::max<uint64_t>(unit_tris, 1), kUnitTris);
        n_units = (count + unit_tris - 1) / unit_tris;
    }
    // work-item granularity: ~8 items per SM at the expected output (O(2 R^2) fragments) so that small conversions
    // still spread over the GPU, at most 2048 fragments; an oversized row block (<= 32 rows x R pixels) takes at most
    // kMaxSplit queue slots
    uint32_t item_max = (uint32_t)std::min<uint64_t>(kItemMaxFrags, (2ull * p->resolution * p->resolution) / ((uint64_t)ctx->sm_count * 8));
    item_max = std::max<uint32_t>({item_max, 64u, (32u * p->resolution + kMaxSplit - 1) / kMaxSplit});
    item_max = std::min<uint32_t>((item_max + 31u) & ~31u, kItemMaxFrags);
    const uint32_t flush_frags = std::max<uint32_t>(32u, item_max / 2);
    // item queue: a warp stops taking slots once it has seen the counter pass the cap, so live items cover disjoint
    // output ranges below it: per unit one item of small triangles and one end-of-unit item, cap/32 items closed by
    // 32 non-empty blocks, cap/flush closed by their fragment count, cap/item_max pieces of oversized blocks; plus
    // ONE reservation per raster warp that may straddle the cap (< 2 kMaxSplit + kStashItems slots).  The queue
    // cannot overflow.
    const uint64_t raster_warps = (uint64_t)grid * convert_warps_per_cta(klayout);
    const uint64_t queue_cap = std::min<uint64_t>(2 * n_units + cap / 32 + cap / flush_frags + cap / item_max +
                                                  raster_warps * (2ull * kMaxSplit + kStashItems) + 64, (1u << 24) - 1);
    {   // scratch between the two kernels (grown on demand, kept by the context)
        m2s_status st = grow(ctx, &ctx->d_trifrag, &ctx->trifrag_bytes, std::max<uint64_t>(count, 1) * tri_frag_bytes(klayout), stream);
        if (st == M2S_OK) st = grow(ctx, &ctx->d_items, &ctx->items_bytes, queue_cap * sizeof(FragItem), stream);
        if (st != M2S_OK) return st;
    }
    if (ctx->dirty) {
        CUDA_TRY(cudaMemsetAsync(ctx->d_sched, 0, 8 * 128, stream));
        CUDA_TRY(cudaMemsetAsync(ctx->d_counter, 0, sizeof(unsigned long long), stream));
        ctx->dirty = false;
    }
    ConvertArgs a;
    std::memset(&a, 0, sizeof(a));
    a.tris = s->d_tris;
    a.tri_first = (uint32_t)first;
    a.tri_count = (uint32_t)count;
    a.ranges = s->d_ranges; a.nranges = s->nranges;
    a.prims = s->d_prims; a.nprims = s->nprims; a.texs = s->d_texs; a.tex_base = s->d_arena; a.ntex = s->ntex;
    a.R = p->resolution;
    a.row_begin = std::min(p->row_begin, p->resolution);
    a.row_end = (p->row_end == 0 || p->row_end > p->resolution) ? p->resolution : p->row_end;
    a.half_R = (float)p->resolution * 0.5f;
    a.mult = p->gaussian_std / (float)p->resolution;
    a.log_sz = logf(1e-7f * a.mult);
    a.tri_frag = (unsigned char*)ctx->d_trifrag;
    a.items = (FragItem*)ctx->d_items;
    a.queue_cap = (uint32_t)queue_cap;
    a.item_max_frags = item_max;
    a.flush_frags = flush_frags;
    a.n_items_out = ctx->d_nitems;
    a.out = (uint8_t*)kout;
    a.cap = cap;
    a.keys = (unsigned long long*)d_keys;
    a.counter = ctx->d_counter;
    // fused gather: the raster kernel's count stays local, the global total goes to d_total after the wait
    a.total_out = (peers && peers->world > 1) ? ctx->d_total : (d_total ? (unsigned long long*)d_total : ctx->d_total);
    a.prev_totals = prev_totals;
    a.nprev = nprev;
    a.host_total = host_total;
    a.host_tag = host_tag;
    a.sched = ctx->d_sched;
    a.unit_tris = (uint32_t)unit_tris;
    a.n_units = (uint32_t)n_units;
    a.trace = g_trace;
    if (peers && peers->world > 1) {
        a.world = peers->world; a.rank = peers->rank;
        for (uint32_t r = 0; r < peers->world; ++r) { a.peer_out[r] = (uint8_t*)peers->out[r]; a.peer_xch[r] = (unsigned long long*)peers->xch[r]; }
        a.epoch = ++ctx->epoch;
        a.gcap = out_capacity;
        a.status = ctx->d_status;
    }
    const int fgrid = ctx->sm_count * ctx->frag_blocks_per_sm[klayout];
    cudaError_t e = convert_launch(klayout, a, grid, fgrid, stream, mid);
    if (e != cudaSuccess) { ctx->dirty = true; set_error(std::string("convert launch: ") + cudaGetErrorString(e)); return M2S_E_CUDA; }
    if (peers && peers->world > 1)
        CUDA_TRY(gather_wait_launch((const unsigned long long*)peers->xch[peers->rank], peers->world, a.epoch, out_capacity,
                                    (unsigned long long*)d_total, ctx->d_status, stream));
    return M2S_OK;
}

M2S_EXPORT m2s_status m2s_convert_enqueue(m2s_ctx* ctx, const m2s_dscene* s, const m2s_params* p, void* d_out,
                                          uint64_t out_capacity, uint64_t* d_keys, uint64_t* d_total, void* stream_) {
    return convert_enqueue_impl(ctx, s, p, d_out, out_capacity, d_keys, d_total, stream_, nullptr);
}

M2S_EXPORT m2s_status m2s_convert_gather_enqueue(m2s_ctx* ctx, const m2s_dscene* s, const m2s_params* p, const m2s_peers* peers,
                                                 uint64_t out_capacity, uint64_t* d_total_global, void* stream_) {
    if (!peers) { set_error("m2s_convert_gather: peers is NULL"); return M2S_E_INVALID; }
    if (peers->world <= 1)  // degenerate: plain conversion into the local final buffer
        return convert_enqueue_impl(ctx, s, p, peers->out[0], out_capacity, nullptr, d_total_global, stream_, nullptr);
    return convert_enqueue_impl(ctx, s, p, nullptr, out_capacity, nullptr, d_total_global, stream_, peers);
}

M2S_EXPORT m2s_status m2s_convert(m2s_ctx* ctx, const m2s_dscene* s, const m2s_params* p, void* d_out, uint64_t out_capacity,
                                  uint64_t* d_keys, m2s_result* res) {
    if (!ctx) { set_error("m2s_convert: ctx is NULL"); return M2S_E_INVALID; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    m2s_status st = m2s_convert_enqueue(ctx, s, p, d_out, out_capacity, d_keys, nullptr, ctx->stream);
    if (st != M2S_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(ctx->h_total, ctx->d_total, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { ctx->dirty = true; set_error(std::string("convert: ") + cudaGetErrorString(e)); return M2S_E_CUDA; }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    const uint64_t cap = effective_cap(s, p, out_capacity);
    const uint64_t total = *ctx->h_total;
    if (res) { res->total = total; res->cap = cap; res->written = std::min(total, cap); res->device_ms = ms; }
    if (total > cap) {
        char buf[160];
        std::snprintf(buf, sizeof(buf), "m2s_convert: %llu gaussians generated, capacity %llu", (unsigned long long)total, (unsigned long long)cap);
        set_error(buf);
        return M2S_E_CAPACITY;
    }
    return M2S_OK;
}

// Measurement aid: one conversion with an event between the two kernels (no programmatic dependent launch, so they do
// not overlap): the per-kernel shares of the step, measured live instead of read from a profile.
M2S_EXPORT m2s_status m2s_convert_timed(m2s_ctx* ctx, const m2s_dscene* s, const m2s_params* p, void* d_out, uint64_t out_capacity,
                                        float* raster_ms, float* fragment_ms) {
    if (!ctx) { set_error("m2s_convert_timed: ctx is NULL"); return M2S_E_INVALID; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (!ctx->ev_mid) CUDA_TRY(cudaEventCreate(&ctx->ev_mid));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    m2s_status st = convert_enqueue_impl(ctx, s, p, d_out, out_capacity, nullptr, nullptr, ctx->stream, nullptr, nullptr, 0, nullptr, 0, ctx->ev_mid);
    if (st != M2S_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { ctx->dirty = true; set_error(std::string("convert_timed: ") + cudaGetErrorString(e)); return M2S_E_CUDA; }
    float a = 0.f, b = 0.f;
    cudaEventElapsedTime(&a, ctx->ev0, ctx->ev_mid);
    cudaEventElapsedTime(&b, ctx->ev_mid, ctx->ev1);
    if (raster_ms) *raster_ms = a;
    if (fragment_ms) *fragment_ms = b;
    return M2S_OK;
}

// Upload only the maps a layout consumes: PACKED56 carries neither normal nor metallic/roughness, the
// standard .ply row no metallic/roughness — their texels would cross PCIe for nothing.
struct SlimScene {
    std::vector<m2s_primitive> prims;
    std::vector<m2s_texture> texs;
    m2s_scene scene;
    SlimScene(const m2s_scene* sc, uint32_t layout) : prims(sc->primitives, sc->primitives + sc->primitive_count), scene(*sc) {
        const bool need_normal = layout != M2S_LAYOUT_PACKED56;
        const bool need_mr = layout == M2S_LAYOUT_REF96 || layout == M2S_LAYOUT_PLY_PBR || layout == M2S_LAYOUT_PLY_COMPRESSED;
        std::vector<int32_t> remap(sc->texture_count, -1);
        auto use = [&](int32_t& idx, bool needed) {
            if (idx < 0 || !needed || (uint32_t)idx >= sc->texture_count) { if (idx >= 0 && (uint32_t)idx < sc->texture_count) idx = -1; return; }
            if (remap[idx] < 0) { remap[idx] = (int32_t)texs.size(); texs.push_back(sc->textures[idx]); }
            idx = remap[idx];
        };
        for (auto& pr : prims) { use(pr.albedo_texture, true); use(pr.normal_texture, need_normal); use(pr.metallic_roughness_texture, need_mr); }
        scene.primitives = prims.data();
        scene.textures = texs.data();
        scene.texture_count = (uint32_t)texs.size();
    }
};

// One shard of a scene: the triangles [first, first + count) (at their global indices) and only the texture rows they
// can sample, only the maps `layout` consumes — what one rank of a multi-GPU conversion needs on its device.
M2S_EXPORT m2s_status m2s_scene_upload_range(m2s_ctx* ctx, const m2s_scene* sc, uint32_t layout, uint64_t first_triangle,
                                             uint64_t triangle_count, m2s_dscene** out) {
    if (!ctx || !sc || !out) { set_error("m2s_scene_upload_range: NULL argument"); return M2S_E_INVALID; }
    if (layout > M2S_LAYOUT_PLY_COMPRESSED) { set_error("m2s_scene_upload_range: unknown layout"); return M2S_E_INVALID; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    SlimScene slim(sc, layout);
    const uint64_t first = std::min<uint64_t>(first_triangle, sc->triangle_count);
    uint64_t count = triangle_count;
    if (count == 0 || first + count > sc->triangle_count) count = sc->triangle_count - first;
    m2s_dscene* ds = nullptr;
    m2s_status st = scene_upload_impl(ctx, &slim.scene, &ds, count, false, first, true);
    if (st != M2S_OK) return st;
    st = vrange_enqueue(ctx, ds, first, first + count, 0);
    if (st == M2S_OK) st = upload_groups_from_vrange(ctx, ds, 0, [] { return cudaSuccess; });
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (st == M2S_OK && e != cudaSuccess) { set_error(std::string("m2s_scene_upload_range: ") + cudaGetErrorString(e)); st = M2S_E_CUDA; }
    if (st != M2S_OK) { m2s_scene_free(ctx, ds); return st; }
    *out = ds;
    return M2S_OK;
}

M2S_EXPORT m2s_status m2s_convert_host(m2s_ctx* ctx, const m2s_scene* sc, const m2s_params* p, void* h_out, uint64_t out_capacity,
                                       uint64_t* h_keys, m2s_result* res) {
    if (!ctx || !sc || !p || (!h_out && out_capacity)) { set_error("m2s_convert_host: NULL argument"); return M2S_E_INVALID; }
    const uint32_t stride = m2s_record_stride(p->layout);
    if (!stride) { set_error("m2s_convert_host: unknown layout"); return M2S_E_INVALID; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    SlimScene slim_holder(sc, p->layout);
    const m2s_scene& slim = slim_holder.scene;
    // Pipeline (REF96 / PACKED56, meshes large enough to split): the triangle range is cut into chunks; chunk c's
    // records are appended after chunk c-1's on the device (fragment kernel: prev_totals) and start crossing
    // PCIe on a second stream while chunk c+1 is still being uploaded and converted — H2D and D2H overlap.
    uint64_t first = std::min<uint64_t>(p->first_triangle, sc->triangle_count);
    uint64_t count = p->triangle_count;
    if (count == 0 || first + count > sc->triangle_count) count = sc->triangle_count - first;
    int nchunks = 1;
    if (count >= 16384) {  // every layout: the fragment kernel appends after the earlier chunks' records itself
        // every chunk shortens the tail (the last chunk's kernels and download) and costs ~25 us of kernel latency on the
        // compute stream, hidden behind the uploads; chunks of >= 8 k triangles keep the GPU filled
        nchunks = (int)std::max<uint64_t>(2, std::min<uint64_t>(4, count / 16384));
        if (const char* e = std::getenv("M2S_HOST_CHUNKS")) nchunks = std::max(1, std::min(m2s_ctx::kMaxChunks, std::atoi(e)));
    }
    const uint64_t per = (count + nchunks - 1) / nchunks;
    m2s_dscene* ds = nullptr;
    // Pipeline: (1) the triangle chunks go up back to back, each followed by a reduction of its v-range per texture and
    // a 8-byte-per-texture copy back; (2) per chunk, as soon as its v-range is on the host: the texture row groups it
    // samples (not yet resident) go up, the two kernels are enqueued; (3) a chunk's records start crossing PCIe on a
    // second stream as soon as its count has arrived (zero-copy, from the raster kernel's last CTA) while later chunks
    // are still being uploaded and converted.  The first records exist after ~1/nchunks of the upload; a shard
    // (first_triangle/triangle_count) never uploads texture rows it does not sample.
    m2s_status st = scene_upload_impl(ctx, &slim, &ds, 0, false, first, true);
    if (st != M2S_OK) return st;
    st = grow(ctx, &ctx->d_out, &ctx->out_bytes, std::max<uint64_t>(out_capacity, 1) * stride);
    if (st == M2S_OK && h_keys) st = grow(ctx, (void**)&ctx->d_keys, &ctx->keys_bytes, std::max<uint64_t>(out_capacity, 1) * 8);
    if (st != M2S_OK) { cudaStreamSynchronize(ctx->stream); m2s_scene_free(ctx, ds); return st; }
    m2s_result r;
    std::memset(&r, 0, sizeof(r));
    const uint64_t cap = effective_cap(ds, p, out_capacity);
    auto fail_with = [&](m2s_status code) {
        cudaStreamSynchronize(ctx->stream3); cudaStreamSynchronize(ctx->stream4); cudaStreamSynchronize(ctx->stream5);
        cudaStreamSynchronize(ctx->stream); cudaStreamSynchronize(ctx->stream2);
        ctx->dirty = true; ctx->vr_dirty = true;
        m2s_scene_free(ctx, ds);
        return code;
    };
    auto bail = [&](const char* what, cudaError_t e) {
        set_error(std::string(what) + ": " + cudaGetErrorString(e));
        return fail_with(M2S_E_CUDA);
    };
    static const bool host_trace = std::getenv("M2S_HOST_TRACE") != nullptr;  // debug: phase times on stderr
    const auto t_start = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_start).count(); };
    cudaError_t e = cudaEventRecord(ctx->ev0, ctx->stream);
    if (e != cudaSuccess) return bail("convert_host", e);
    // uploads run on their own stream (behind the allocations and table copies made above on the context stream): the
    // copy engine streams triangles and texture rows continuously while the chunks' kernels run on the context stream
    e = cudaEventRecord(ctx->ev_alloc, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream3, ctx->ev_alloc, 0);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream4, ctx->ev_alloc, 0);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream5, ctx->ev_alloc, 0);
    if (e != cudaSuccess) return bail("convert_host", e);
    // triangles on one copy stream, texture rows on another (two copy engines: 51 instead of 35 GB/s), the v-range
    // reductions on a third, the mip rows on the compute stream: no copy ever queues behind a kernel
    struct UpGuard { m2s_ctx* c; ~UpGuard() { c->up = c->tex_up = c->mip = c->aux = c->stream; } } up_guard{ctx};
    ctx->up = ctx->stream3; ctx->tex_up = ctx->stream4; ctx->aux = ctx->stream5; ctx->mip = ctx->stream;
    uint64_t lo_[m2s_ctx::kMaxChunks], hi_[m2s_ctx::kMaxChunks];
    int planned = 0, uploaded = 0;
    for (int c = 0; c < nchunks; ++c) {
        const uint64_t lo = first + (uint64_t)c * per, hi = std::min(first + count, lo + per);
        if (lo >= hi && c > 0) break;
        lo_[c] = lo; hi_[c] = hi;
        ++planned;
    }
    // (1) triangle chunk c goes up (its own copy stream), followed by the reduction of its v-range per texture (a kernel behind
    // "chunk c is resident" on the aux stream, results through mapped memory)
    auto upload_tris = [&](int c) -> m2s_status {
        cudaError_t e1 = cudaSuccess;
        if (hi_[c] > lo_[c]) {
            e1 = cudaMemcpyAsync(reinterpret_cast<unsigned char*>(ds->d_tris) + lo_[c] * (size_t)kTriBytes,
                                 reinterpret_cast<const unsigned char*>(sc->triangles) + lo_[c] * (size_t)kTriBytes,
                                 (hi_[c] - lo_[c]) * (size_t)kTriBytes, cudaMemcpyHostToDevice, ctx->up);
            ds->h2d_bytes += (hi_[c] - lo_[c]) * (uint64_t)kTriBytes;
        }
        if (e1 == cudaSuccess) e1 = cudaEventRecord(ctx->ev_tri[c], ctx->up);
        if (e1 == cudaSuccess) e1 = cudaStreamWaitEvent(ctx->aux, ctx->ev_tri[c], 0);
        if (e1 != cudaSuccess) { set_error(std::string("convert_host upload: ") + cudaGetErrorString(e1)); return M2S_E_CUDA; }
        return vrange_enqueue(ctx, ds, lo_[c], hi_[c], c);
    };
    // look-ahead: triangle chunks (and their v-range reductions) queued ahead of the chunk whose texture rows go up: the
    // first records exist after ~lookahead/nchunks of the triangles and 1/nchunks of the texture rows (the downloads, 36 MB
    // at 55 GB/s, are the longest leg of the call: they must start early).  Measured on the bench scene
    // (profiles/r02_e2e_pipeline.txt): 4 chunks / look-ahead 2: 1.08 ms; 8 / 3: 1.09; every triangle chunk queued up front:
    // 1.14-1.16 (first records at 0.34 ms instead of 0.20); every copy cut in halves over two streams (two streams deliver
    // 51 GB/s against 35 for one when they carry 13 MB each — not with 1 MB pieces beside a running download): 1.23
    int lookahead = 2;
    if (const char* e = std::getenv("M2S_HOST_LOOKAHEAD")) lookahead = std::max(1, std::atoi(e));
    for (; uploaded < std::min(planned, lookahead); ++uploaded) {
        st = upload_tris(uploaded);
        if (st != M2S_OK) return fail_with(st);
    }
    unsigned long long tags[m2s_ctx::kMaxChunks] = {};
    uint64_t base = 0, written = 0;
    int next_dl = 0;
    // enqueue the downloads of the chunks whose counts have arrived (in order); block: wait for them
    auto downloads = [&](int upto, bool block) -> cudaError_t {
        while (next_dl < upto) {
            const int c = next_dl;
            volatile unsigned long long* slot = ctx->h_chunk_tot + 2 * c;
            for (;;) {
                if (__atomic_load_n(&ctx->h_chunk_tot[2 * c + 1], __ATOMIC_ACQUIRE) == tags[c]) break;  // count is ordered before the tag
                if (!block) return cudaSuccess;
                const cudaError_t q = cudaEventQuery(ctx->ev_chunk[c]);
                if (q == cudaSuccess) break;             // finished: the tag is there
                if (q != cudaErrorNotReady) return q;
            }
            if (__atomic_load_n(&ctx->h_chunk_tot[2 * c + 1], __ATOMIC_ACQUIRE) != tags[c]) return cudaErrorUnknown;
            const uint64_t tot = slot[0];
            if (host_trace) std::fprintf(stderr, "[m2s host] chunk %d rasterised at %.0f us (%llu records)\n", c, since(), (unsigned long long)tot);
            const uint64_t room = cap > base ? cap - base : 0, w = std::min(tot, room);
            if (w) {
                cudaError_t e2 = cudaStreamWaitEvent(ctx->stream2, ctx->ev_chunk[c], 0);
                if (e2 == cudaSuccess)
                    e2 = cudaMemcpyAsync(reinterpret_cast<unsigned char*>(h_out) + base * stride,
                                         reinterpret_cast<const unsigned char*>(ctx->d_out) + base * stride, w * stride,
                                         cudaMemcpyDeviceToHost, ctx->stream2);
                if (e2 == cudaSuccess && h_keys)
                    e2 = cudaMemcpyAsync(h_keys + base, ctx->d_keys + base, w * 8, cudaMemcpyDeviceToHost, ctx->stream2);
                if (e2 != cudaSuccess) return e2;
            }
            base += tot;
            written += w;
            ++next_dl;
        }
        return cudaSuccess;
    };
    int launched = 0;
    for (int c = 0; c < planned; ++c) {  // (2)
        std::vector<MipRun> runs;
        const double t_it0 = host_trace ? since() : 0.0;
        st = upload_groups_from_vrange(ctx, ds, c, [&] { return downloads(launched, false); }, &runs);  // (3) while waiting: whatever is ready
        if (st != M2S_OK) return fail_with(st);
        const double t_it1 = host_trace ? since() : 0.0;
        e = cudaEventRecord(ctx->ev_up[c], ctx->tex_up);   // chunk c's texture rows are resident (level 0)
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ctx->ev_up[c], 0);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ctx->ev_tri[c], 0);
        if (e != cudaSuccess) return bail("convert_host", e);
        for (const MipRun& r : runs) {   // their mip rows: on the compute stream, right before the kernels that sample them
            e = mip_groups_launch(ds->d_arena, ds->h_texs[r.t], r.g0, r.g1, ctx->stream);
            if (e != cudaSuccess) return bail("convert_host mips", e);
        }
        if (uploaded < planned) {  // the next look-ahead chunk
            st = upload_tris(uploaded++);
            if (st != M2S_OK) return fail_with(st);
        }
        m2s_params pc = *p;
        pc.first_triangle = lo_[c];
        pc.triangle_count = hi_[c] - lo_[c];
        unsigned long long* h_dev = nullptr;  // device view of the mapped count slot
        e = cudaHostGetDevicePointer((void**)&h_dev, ctx->h_chunk_tot + 2 * c, 0);
        if (e != cudaSuccess) return bail("convert_host", e);
        tags[c] = ++ctx->host_seq;
        if (hi_[c] > lo_[c]) {
            st = convert_enqueue_impl(ctx, ds, &pc, ctx->d_out, out_capacity, h_keys ? (uint64_t*)ctx->d_keys : nullptr,
                                      (uint64_t*)(ctx->d_chunk_tot + c), ctx->stream, nullptr, ctx->d_chunk_tot, (uint32_t)c,
                                      h_dev, tags[c]);
            if (st != M2S_OK) return fail_with(st);
        } else {  // empty range: nothing to launch, the count is zero
            e = cudaMemsetAsync(ctx->d_chunk_tot + c, 0, sizeof(unsigned long long), ctx->stream);
            if (e != cudaSuccess) return bail("convert_host", e);
            ctx->h_chunk_tot[2 * c] = 0;
            __atomic_store_n(&ctx->h_chunk_tot[2 * c + 1], tags[c], __ATOMIC_RELEASE);
        }
        e = cudaEventRecord(ctx->ev_chunk[c], ctx->stream);
        if (e != cudaSuccess) return bail("convert_host", e);
        ++launched;
        const double t_it2 = host_trace ? since() : 0.0;
        e = downloads(launched, false);  // (3) whatever is ready
        if (e != cudaSuccess) return bail("convert_host download", e);
        if (host_trace) std::fprintf(stderr, "[m2s host] chunk %d: v-range wait + rows enqueued %.0f us, tris/mips/kernels enqueued %.0f us, downloads %.0f us (at %.0f us)\n",
                                     c, t_it1 - t_it0, t_it2 - t_it1, since() - t_it2, since());
    }
    e = cudaEventRecord(ctx->ev1, ctx->stream);
    if (e != cudaSuccess) return bail("convert_host", e);
    if (host_trace) std::fprintf(stderr, "[m2s host] enqueued %d chunks at %.0f us\n", launched, since());
    e = downloads(launched, true);
    if (e != cudaSuccess) return bail("convert_host download", e);
    e = cudaStreamSynchronize(ctx->stream2);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream3);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream4);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream5);
    if (e != cudaSuccess) return bail("convert_host download", e);
    if (host_trace) std::fprintf(stderr, "[m2s host] downloads done at %.0f us\n", since());
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    r.total = base; r.cap = cap; r.written = written; r.device_ms = ms;
    st = M2S_OK;
    if (base > cap) {
        char buf[160];
        std::snprintf(buf, sizeof(buf), "m2s_convert: %llu gaussians generated, capacity %llu", (unsigned long long)base, (unsigned long long)cap);
        set_error(buf);
        st = M2S_E_CAPACITY;
    }
    if (res) *res = r;
    m2s_scene_free(ctx, ds);
    return st;
}

// ---- scene -> .ply file: rows encoded on the GPU, streamed to disk through two pinned buffers -------------
// (SceneManager::exportPly + parsers.cpp::savePlyVector write 4 bytes at a time from one thread)
namespace m2s {
m2s_status convert_scene_to_ply(m2s_ctx* ctx, const m2s_scene* sc, const m2s_params* p, const char* path, m2s_result* res) {
    if (!ctx || !sc || !p || !path) { set_error("convert_scene_to_ply: NULL argument"); return M2S_E_INVALID; }
    if (p->layout < M2S_LAYOUT_PLY_STANDARD || p->layout > M2S_LAYOUT_PLY_COMPRESSED) { set_error("convert_scene_to_ply: a .ply row layout is required"); return M2S_E_INVALID; }
    const uint32_t format = p->layout - M2S_LAYOUT_PLY_STANDARD;
    const uint32_t stride = m2s_record_stride(p->layout);
    CUDA_TRY(cudaSetDevice(ctx->device));
    SlimScene slim(sc, p->layout);
    m2s_dscene* ds = nullptr;
    m2s_status st = scene_upload_impl(ctx, &slim.scene, &ds, UINT64_MAX, false);
    if (st != M2S_OK) return st;
    const uint64_t cap = p->max_gaussians ? p->max_gaussians : m2s_reference_capacity(p->resolution, sc->primitive_count);
    st = grow(ctx, &ctx->d_out, &ctx->out_bytes, std::max<uint64_t>(cap, 1) * stride);
    if (st != M2S_OK) { cudaStreamSynchronize(ctx->stream); m2s_scene_free(ctx, ds); return st; }
    m2s_result r;
    std::memset(&r, 0, sizeof(r));
    st = m2s_convert(ctx, ds, p, ctx->d_out, cap, nullptr, &r);  // synchronises; r.written rows are in d_out
    m2s_scene_free(ctx, ds);
    if (res) *res = r;
    if (st != M2S_OK && st != M2S_E_CAPACITY) return st;
    for (int i = 0; i < 2; ++i)
        if (!ctx->h_stage[i]) CUDA_TRY(cudaMallocHost(&ctx->h_stage[i], m2s_ctx::kStageBytes));
    FILE* f = std::fopen(path, "wb");
    if (!f) { set_error(std::string("cannot open ") + path); return M2S_E_IO; }
    char hdr[4096];
    const size_t hn = m2s_ply_header(format, r.written, hdr, sizeof(hdr));
    bool ok = std::fwrite(hdr, 1, hn, f) == hn;
    const size_t rows_per_block = m2s_ctx::kStageBytes / stride;
    const uint64_t nblocks = (r.written + rows_per_block - 1) / rows_per_block;
    cudaError_t e = cudaSuccess;
    auto block_bytes = [&](uint64_t b) { return (size_t)std::min<uint64_t>(rows_per_block, r.written - b * rows_per_block) * stride; };
    for (uint64_t b = 0; b <= nblocks && ok && e == cudaSuccess; ++b) {
        if (b < nblocks) {  // start the download of block b ...
            e = cudaMemcpyAsync(ctx->h_stage[b & 1], reinterpret_cast<const unsigned char*>(ctx->d_out) + b * rows_per_block * stride,
                                block_bytes(b), cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaEventRecord(ctx->ev_chunk[b & 1], ctx->stream);
        }
        if (b > 0 && e == cudaSuccess) {  // ... and write block b-1 while it crosses PCIe
            e = cudaEventSynchronize(ctx->ev_chunk[(b - 1) & 1]);
            if (e == cudaSuccess) ok = std::fwrite(ctx->h_stage[(b - 1) & 1], 1, block_bytes(b - 1), f) == block_bytes(b - 1);
        }
    }
    cudaStreamSynchronize(ctx->stream);
    ok = (std::fclose(f) == 0) && ok;
    if (e != cudaSuccess) { set_error(std::string("convert_scene_to_ply download: ") + cudaGetErrorString(e)); return M2S_E_CUDA; }
    if (!ok) { set_error(std::string("short write to ") + path); return M2S_E_IO; }
    return st;
}
}  // namespace m2s

// ---- outputs ----------------------------------------------------------------------------------
M2S_EXPORT m2s_status m2s_ply_encode(m2s_ctx* ctx, const void* d_ref96, uint64_t count, uint32_t format, float mult, void* d_rows,
                                     void* stream_) {
    if (!ctx || (count && (!d_ref96 || !d_rows))) { set_error("m2s_ply_encode: NULL argument"); return M2S_E_INVALID; }
    if (format > 2) format = 0;  // savePlyVector default branch (parsers.cpp:646-648)
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(ply_rows_launch(d_ref96, count, nullptr, format, mult, d_rows, stream_ ? (cudaStream_t)stream_ : ctx->stream));
    return M2S_OK;
}


// ---- the viewer prepass (SURVEY 8 f-4): GaussiansPrepass::execute + gaussianSplattingPrepassCS.glsl ----------------
static bool invert4(const double m[16], double inv[16]) {   // column-major, cofactors
    inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
    inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
    inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
    inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
    inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
    inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
    inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
    inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
    inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
    inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
    inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
    inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
    inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
    inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
    inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
    inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
    const double det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
    if (det == 0.0) return false;
    for (int k = 0; k < 16; ++k) inv[k] /= det;
    return true;
}

M2S_EXPORT m2s_status m2s_prepass_enqueue(m2s_ctx* ctx, const void* d_records, uint64_t count, const uint64_t* d_count,
                                          const m2s_prepass_params* p, void* d_quads, float* d_depths, uint32_t* d_valid, void* stream_) {
    if (!ctx || !p || !d_valid || (count && (!d_records || !d_quads || !d_depths))) { set_error("m2s_prepass: NULL argument"); return M2S_E_INVALID; }
    if (p->layout != M2S_LAYOUT_REF96 && p->layout != M2S_LAYOUT_PACKED56) { set_error("m2s_prepass: layouts REF96 and PACKED56 only"); return M2S_E_INVALID; }
    if (p->render_mode == 3 || p->render_mode > 6) { set_error("m2s_prepass: render modes 0-2 and 4-6 only"); return M2S_E_INVALID; }
    if (count >= (1ull << 32)) { set_error("m2s_prepass: too many gaussians (< 2^32 supported)"); return M2S_E_INVALID; }
    if ((reinterpret_cast<uintptr_t>(d_quads) & 15u) || (reinterpret_cast<uintptr_t>(d_records) & 15u)) {
        set_error("m2s_prepass: the record and quad buffers must be 16-byte aligned"); return M2S_E_INVALID;
    }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : ctx->stream;
    PrepassArgs a;
    std::memset(&a, 0, sizeof(a));
    std::memcpy(a.V, p->world_to_view, 64); std::memcpy(a.P, p->view_to_clip, 64); std::memcpy(a.M, p->model_to_world, 64);
    double M[16], Mi[16];
    for (int k = 0; k < 16; ++k) M[k] = p->model_to_world[k];
    if (!invert4(M, Mi)) { set_error("m2s_prepass: model_to_world is singular"); return M2S_E_INVALID; }
    for (int c = 0; c < 4; ++c) for (int r = 0; r < 4; ++r) a.Nmat[c * 4 + r] = (float)Mi[r * 4 + c];   // transpose(inverse(M))
    {   // inverse(mat3(M)): rows of M's upper 3x3
        const double m00 = M[0], m01 = M[4], m02 = M[8], m10 = M[1], m11 = M[5], m12 = M[9], m20 = M[2], m21 = M[6], m22 = M[10];
        const double det = m00 * (m11 * m22 - m12 * m21) - m01 * (m10 * m22 - m12 * m20) + m02 * (m10 * m21 - m11 * m20);
        if (det == 0.0) { set_error("m2s_prepass: model_to_world has a singular rotation part"); return M2S_E_INVALID; }
        const double i = 1.0 / det;
        a.Ninv[0] = (float)((m11 * m22 - m12 * m21) * i); a.Ninv[3] = (float)((m02 * m21 - m01 * m22) * i); a.Ninv[6] = (float)((m01 * m12 - m02 * m11) * i);
        a.Ninv[1] = (float)((m12 * m20 - m10 * m22) * i); a.Ninv[4] = (float)((m00 * m22 - m02 * m20) * i); a.Ninv[7] = (float)((m02 * m10 - m00 * m12) * i);
        a.Ninv[2] = (float)((m10 * m21 - m11 * m20) * i); a.Ninv[5] = (float)((m01 * m20 - m00 * m21) * i); a.Ninv[8] = (float)((m00 * m11 - m01 * m10) * i);
    }
    const double l0 = M[0] * M[0] + M[1] * M[1] + M[2] * M[2] + M[3] * M[3], l1 = M[4] * M[4] + M[5] * M[5] + M[6] * M[6] + M[7] * M[7];
    a.mscale2[0] = (float)l0; a.mscale2[1] = (float)l0; a.mscale2[2] = (float)l1;   // (|M[0]|, |M[0]|, |M[1]|) squared — sic (:96)
    a.res[0] = p->resolution[0]; a.res[1] = p->resolution[1]; a.near_far[0] = p->near_far[0]; a.near_far[1] = p->near_far[1];
    a.std_dev = p->std_dev; a.render_mode = p->render_mode; a.layout = p->layout == M2S_LAYOUT_REF96 ? 0u : 1u;
    a.count = count; a.d_count = (const unsigned long long*)d_count;
    a.records = (const unsigned char*)d_records; a.quads = (float4*)d_quads; a.depths = d_depths; a.valid = d_valid;
    CUDA_TRY(cudaMemsetAsync(d_valid, 0, sizeof(uint32_t), stream));
    CUDA_TRY(prepass_launch(a, stream));
    return M2S_OK;
}

M2S_EXPORT m2s_status m2s_prepass(m2s_ctx* ctx, const void* d_records, uint64_t count, const m2s_prepass_params* p, void* d_quads,
                                  float* d_depths, uint32_t* valid) {
    if (!ctx) { set_error("m2s_prepass: ctx is NULL"); return M2S_E_INVALID; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (!ctx->d_prepass_valid) CUDA_TRY(cudaMalloc(&ctx->d_prepass_valid, sizeof(uint32_t)));
    m2s_status st = m2s_prepass_enqueue(ctx, d_records, count, nullptr, p, d_quads, d_depths, ctx->d_prepass_valid, ctx->stream);
    if (st != M2S_OK) return st;
    uint32_t v = 0;
    CUDA_TRY(cudaMemcpyAsync(&v, ctx->d_prepass_valid, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (valid) *valid = v;
    return M2S_OK;
}

// ---- depth sort (SURVEY 8 f-5) and splatting pass (f-6): RadixSortPass + GaussianSplattingPass ----------------------
static inline bool misaligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) != 0; }

static m2s_status timing_events(m2s_ctx* ctx) {
    for (cudaEvent_t& e : ctx->ev_r)
        if (!e) CUDA_TRY(cudaEventCreate(&e));
    return M2S_OK;
}

M2S_EXPORT m2s_status m2s_sort_quads_enqueue(m2s_ctx* ctx, const void* d_quads, const float* d_depths, uint64_t count,
                                             const uint32_t* d_count, void* d_sorted_quads, uint32_t* d_order, void* stream_) {
    if (!ctx || (count && (!d_quads || !d_depths || !d_sorted_quads))) { set_error("m2s_sort_quads: NULL argument"); return M2S_E_INVALID; }
    if (count >= (1ull << 32)) { set_error("m2s_sort_quads: too many quads (< 2^32 supported)"); return M2S_E_INVALID; }
    if (misaligned16(d_quads) || misaligned16(d_sorted_quads) || misaligned16(d_depths) || misaligned16(d_order)) {
        set_error("m2s_sort_quads: every buffer must be 16-byte aligned"); return M2S_E_INVALID;
    }
    if (count == 0) return M2S_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : ctx->stream;
    SortArgs a;
    std::memset(&a, 0, sizeof(a));
    a.quads = (const float4*)d_quads; a.depths = d_depths; a.count = count; a.d_count = d_count;
    a.sorted = (float4*)d_sorted_quads; a.order = d_order;
    a.temp_bytes = sort_temp_bytes(count);
    const size_t n4 = ((size_t)count * 4 + 255) & ~(size_t)255;   // 256-byte aligned sub-buffers
    unsigned char* scratch = nullptr;
    CUDA_TRY(cudaMallocAsync((void**)&scratch, 4 * n4 + a.temp_bytes, stream));   // the context's stream-ordered pool
    a.keys[0] = (uint32_t*)scratch; a.keys[1] = (uint32_t*)(scratch + n4);
    a.vals[0] = (uint32_t*)(scratch + 2 * n4); a.vals[1] = (uint32_t*)(scratch + 3 * n4);
    a.temp = scratch + 4 * n4;
    const cudaError_t e = sort_launch(a, stream);
    CUDA_TRY(cudaFreeAsync(scratch, stream));
    CUDA_TRY(e);
    return M2S_OK;
}

M2S_EXPORT m2s_status m2s_sort_quads(m2s_ctx* ctx, const void* d_quads, const float* d_depths, uint64_t count, void* d_sorted_quads,
                                     uint32_t* d_order, float* device_ms) {
    if (!ctx) { set_error("m2s_sort_quads: ctx is NULL"); return M2S_E_INVALID; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    m2s_status st = timing_events(ctx);
    if (st != M2S_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev_r[0], ctx->stream));
    st = m2s_sort_quads_enqueue(ctx, d_quads, d_depths, count, nullptr, d_sorted_quads, d_order, ctx->stream);
    if (st != M2S_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev_r[1], ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (device_ms) CUDA_TRY(cudaEventElapsedTime(device_ms, ctx->ev_r[0], ctx->ev_r[1]));
    return M2S_OK;
}

static m2s_status splat_validate(m2s_ctx* ctx, const void* d_sorted_quads, uint64_t count, const m2s_splat_params* p, const m2s_gbuffer* gb) {
    if (!ctx || !p || !gb || (count && !d_sorted_quads) || !gb->position || !gb->normal || !gb->albedo || !gb->depth || !gb->metallic_roughness) {
        set_error("m2s_splat: NULL argument"); return M2S_E_INVALID;
    }
    if (p->width < 1 || p->width > 4096 || p->height < 1 || p->height > 4096) { set_error("m2s_splat: width and height must be 1..4096"); return M2S_E_INVALID; }
    if (p->render_mode == 3 || p->render_mode > 6) { set_error("m2s_splat: render modes 0-2 and 4-6 only"); return M2S_E_INVALID; }
    if (count >= (1ull << 32)) { set_error("m2s_splat: too many quads (< 2^32 supported)"); return M2S_E_INVALID; }
    if (misaligned16(d_sorted_quads) || misaligned16(gb->position) || misaligned16(gb->normal) || misaligned16(gb->albedo) ||
        misaligned16(gb->depth) || misaligned16(gb->metallic_roughness)) {
        set_error("m2s_splat: the quads and the G-buffer images must be 16-byte aligned"); return M2S_E_INVALID;
    }
    return M2S_OK;
}

static void splat_args(m2s_ctx* ctx, const void* d_sorted_quads, uint64_t count, const uint32_t* d_count, const m2s_splat_params* p,
                       const m2s_gbuffer* gb, SplatArgs& a) {
    std::memset(&a, 0, sizeof(a));
    a.quads = (const float4*)d_sorted_quads; a.count = count; a.d_count = d_count;
    a.width = (int)p->width; a.height = (int)p->height; a.mode = p->render_mode;
    a.tiles_x = (a.width + kSplatTile - 1) / kSplatTile; a.tiles_y = (a.height + kSplatTile - 1) / kSplatTile;
    a.position = (uint2*)gb->position; a.normal = (uint2*)gb->normal; a.depth = (uint2*)gb->depth;
    a.albedo = (uint32_t*)gb->albedo; a.metallic_roughness = (uint32_t*)gb->metallic_roughness;
    a.status = ctx->d_status;
}

static inline size_t up256(size_t b) { return (b + 255) & ~(size_t)255; }

// scratch of the per-quad stage: records, tile counts, their scan, CUB temporary storage
static m2s_status splat_alloc_prepare(SplatArgs& a, cudaStream_t stream, unsigned char** block) {
    const size_t n = a.count ? a.count : 1;
    const size_t tb = splat_scan_temp_bytes(n);
    const size_t b_rec = up256(n * splat_rec_bytes()), b_tiles = up256(n * 4), b_incl = up256(n * 8);
    CUDA_TRY(cudaMallocAsync((void**)block, b_rec + b_tiles + b_incl + tb, stream));
    a.rec = *block; a.tiles = (uint32_t*)(*block + b_rec); a.incl = (unsigned long long*)(*block + b_rec + b_tiles);
    a.temp = *block + b_rec + b_tiles + b_incl; a.temp_bytes = tb;
    return M2S_OK;
}
// scratch of the pair stage: keys and values (double-buffered), tile ranges, CUB temporary storage
static m2s_status splat_alloc_finish(SplatArgs& a, uint64_t max_pairs, cudaStream_t stream, unsigned char** block) {
    const int tiles = a.tiles_x * a.tiles_y;
    const size_t mp = max_pairs ? max_pairs : 1;
    const size_t tb = splat_sort_temp_bytes(mp, tiles);
    const size_t b_pair = up256(mp * 4), b_ranges = up256((size_t)tiles * 8);
    CUDA_TRY(cudaMallocAsync((void**)block, 4 * b_pair + b_ranges + tb, stream));
    for (int k = 0; k < 2; ++k) { a.keys[k] = (uint32_t*)(*block + k * b_pair); a.vals[k] = (uint32_t*)(*block + (2 + k) * b_pair); }
    a.ranges = (uint2*)(*block + 4 * b_pair);
    a.temp = *block + 4 * b_pair + b_ranges; a.temp_bytes = tb;
    a.max_pairs = max_pairs;
    return M2S_OK;
}

M2S_EXPORT m2s_status m2s_splat_enqueue(m2s_ctx* ctx, const void* d_sorted_quads, uint64_t count, const uint32_t* d_count,
                                        const m2s_splat_params* p, const m2s_gbuffer* gb, uint64_t max_pairs, void* stream_) {
    m2s_status st = splat_validate(ctx, d_sorted_quads, count, p, gb);
    if (st != M2S_OK) return st;
    if (max_pairs >= (1ull << 31)) { set_error("m2s_splat_enqueue: max_pairs must be below 2^31"); return M2S_E_INVALID; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : ctx->stream;
    SplatArgs a;
    splat_args(ctx, d_sorted_quads, count, d_count, p, gb, a);
    unsigned char *b0 = nullptr, *b1 = nullptr;
    if ((st = splat_alloc_prepare(a, stream, &b0)) != M2S_OK) return st;
    cudaError_t e = splat_prepare(a, stream);
    if (e == cudaSuccess) {
        if ((st = splat_alloc_finish(a, max_pairs, stream, &b1)) != M2S_OK) { cudaFreeAsync(b0, stream); return st; }
        e = splat_finish(a, stream);
        CUDA_TRY(cudaFreeAsync(b1, stream));
    }
    CUDA_TRY(cudaFreeAsync(b0, stream));
    CUDA_TRY(e);
    return M2S_OK;
}

M2S_EXPORT m2s_status m2s_splat(m2s_ctx* ctx, const void* d_sorted_quads, uint64_t count, const uint32_t* d_count,
                                const m2s_splat_params* p, const m2s_gbuffer* gb, uint64_t* pairs, float* device_ms) {
    m2s_status st = splat_validate(ctx, d_sorted_quads, count, p, gb);
    if (st != M2S_OK) return st;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if ((st = timing_events(ctx)) != M2S_OK) return st;
    cudaStream_t stream = ctx->stream;
    SplatArgs a;
    splat_args(ctx, d_sorted_quads, count, d_count, p, gb, a);
    unsigned char *b0 = nullptr, *b1 = nullptr;
    if ((st = splat_alloc_prepare(a, stream, &b0)) != M2S_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev_r[0], stream));
    cudaError_t e = splat_prepare(a, stream);
    unsigned long long total = 0;
    if (e == cudaSuccess && count) e = cudaMemcpyAsync(ctx->h_total, a.incl + count - 1, 8, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaEventRecord(ctx->ev_r[1], stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e == cudaSuccess && count) total = *ctx->h_total;
    if (e == cudaSuccess && total >= (1ull << 31)) {
        cudaFreeAsync(b0, stream);
        set_error("m2s_splat: more than 2^31 (tile, quad) pairs"); return M2S_E_CAPACITY;
    }
    if (e == cudaSuccess) {
        if ((st = splat_alloc_finish(a, total, stream, &b1)) != M2S_OK) { cudaFreeAsync(b0, stream); return st; }
        e = cudaEventRecord(ctx->ev_r[2], stream);
        if (e == cudaSuccess) e = splat_finish(a, stream);
        if (e == cudaSuccess) e = cudaEventRecord(ctx->ev_r[3], stream);
        CUDA_TRY(cudaFreeAsync(b1, stream));
    }
    CUDA_TRY(cudaFreeAsync(b0, stream));
    CUDA_TRY(e);
    CUDA_TRY(cudaStreamSynchronize(stream));
    if (pairs) *pairs = total;
    if (device_ms) {
        float t0 = 0.f, t1 = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&t0, ctx->ev_r[0], ctx->ev_r[1]));
        CUDA_TRY(cudaEventElapsedTime(&t1, ctx->ev_r[2], ctx->ev_r[3]));
        *device_ms = t0 + t1;
    }
    return M2S_OK;
}
