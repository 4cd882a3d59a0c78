/* m2s.h — C ABI of the B200-native mesh -> 3D-gaussian-splat conversion path.
 *
 * This is the drop-in boundary for ONE path of electronicarts/mesh2splat: the
 * conversion pass.  Every entry point names the reference interface it stands
 * in for (paths relative to the reference tree):
 *
 *   reference                                                  here
 *   ---------------------------------------------------------  ----------------------------
 *   SceneManager::setupMeshBuffers + glUtils::generateTextures  m2s_scene_upload
 *     (src/utils/SceneManager.cpp:468-576,
 *      src/utils/glUtils.cpp:252-317)
 *   ConversionPass::execute / ::conversion                      m2s_convert, m2s_convert_enqueue,
 *     (src/renderer/renderPasses/ConversionPass.cpp:9-117)      m2s_convert_host
 *     + converter{VS,GS,FS}.glsl + SSBO atomic append
 *   SceneManager::exportPly + parsers::savePlyVector            m2s_ply_encode, m2s_ply_write
 *   GaussiansPrepass::execute + gaussianSplattingPrepassCS.glsl  m2s_prepass, m2s_prepass_enqueue
 *     (src/utils/SceneManager.cpp:651-678,
 *      src/parsers/parsers.cpp:232-316,339-428,431-514,631-651)
 *   SceneManager::loadModel -> execute -> exportPly             m2s_convert_file
 *     (src/utils/SceneManager.hpp:18-20)
 *   RadixSortPass::execute + radixSortPrepass.glsl              m2s_sort_quads, m2s_sort_quads_enqueue
 *     + radixSortGather.glsl + glu::RadixSort
 *     (src/renderer/renderPasses/RadixSortPass.cpp:8-90,
 *      thirdParty/RadixSort.hpp:1393-1530)
 *   GaussianSplattingPass::execute + gaussianSplatting{VS,PS}   m2s_splat, m2s_splat_enqueue
 *     .glsl into the G-buffer
 *     (src/renderer/renderPasses/GaussianSplattingPass.cpp:37-97,
 *      src/renderer/renderer.cpp:329-379)
 *
 * Plain pointers and sizes only; no C++/torch types.  All functions return an
 * m2s_status; m2s_last_error() gives the thread-local message of the last
 * failure.  The library has NO CPU fallback: without a usable CUDA device every
 * compute entry point fails with M2S_E_NOGPU.
 */
#ifndef M2S_H
#define M2S_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define M2S_VERSION 100 /* 0.1.0 */

typedef enum m2s_status {
    M2S_OK = 0,
    M2S_E_INVALID = 1,  /* bad argument */
    M2S_E_NOGPU = 2,    /* no CUDA device / driver */
    M2S_E_CUDA = 3,     /* CUDA runtime error (message in m2s_last_error) */
    M2S_E_CAPACITY = 4, /* more gaussians generated than the output holds; result.total has the
                           true count (the reference silently discards: converterFS.glsl:48-51) */
    M2S_E_IO = 5,
    M2S_E_FORMAT = 6    /* malformed .glb / unsupported feature */
} m2s_status;

/* Output record layouts (stride in bytes = m2s_record_stride(layout)). */
typedef enum m2s_layout {
    /* 6 x float4, bit-compatible with GaussianDataSSBO (src/utils/utils.hpp:145-152) /
     * GaussianVertex (converterFS.glsl:21-28): position.xyz1 | color.rgba | scale.xyz0 (raw) |
     * normal.xyz0 | rotation (w,x,y,z) | pbr (metallic, roughness, 0, 1). */
    M2S_LAYOUT_REF96 = 0,
    /* 14 floats: xyz | rot (w,x,y,z) | log(scale*sigma/R) xyz | SH0 rgb | opacity logit — the values
     * parsers.cpp:469-511 derives from the SSBO record, minus normal and f_rest. */
    M2S_LAYOUT_PACKED56 = 1,
    /* one row of the three .ply bodies the reference writes (format 0/1/2 of savePlyVector) */
    M2S_LAYOUT_PLY_STANDARD = 2,   /* 62 floats = 248 B, parsers.cpp:431-514 */
    M2S_LAYOUT_PLY_PBR = 3,        /* 19 floats =  76 B, parsers.cpp:232-316 */
    M2S_LAYOUT_PLY_COMPRESSED = 4  /* 48 B,               parsers.cpp:339-428 */
} m2s_layout;

enum {
    M2S_FLAG_NONE = 0,
    /* cap = min(6*R*R*primitive_count, 7 000 000) exactly as ConversionPass.cpp:21-24 when
     * max_gaussians == 0 (default).  With this flag and max_gaussians == 0 the cap is only the
     * capacity of the output buffer handed in. */
    M2S_FLAG_UNCAPPED = 1u << 0
};

#define M2S_FLOATS_PER_VERTEX 12u   /* pos3 normal3 tangent4 uv2: the live part of the reference's
                                       17-float vertex (SceneManager.cpp:484-512) */
#define M2S_FLOATS_PER_TRIANGLE 36u /* 144 B */
#define M2S_MAX_MIP_LEVEL 4u        /* GL_TEXTURE_MAX_LEVEL 4, glUtils.cpp:313 */
#define M2S_REFERENCE_MAX_GAUSSIANS 7000000u /* MAX_GAUSSIANS_TO_SORT, RenderPass.hpp:8 */

/* RGBA8 image, row 0 first, exactly the bytes tinygltf hands to glTexImage2D
 * (glUtils.cpp:292-303); wrap REPEAT, trilinear, levels 0..4 generated on upload. */
typedef struct m2s_texture {
    const uint8_t* rgba;
    uint32_t width, height;
} m2s_texture;

/* One glTF primitive = one utils::Mesh = one glDrawArrays of the reference
 * (ConversionPass.cpp:70-117). */
typedef struct m2s_primitive {
    uint64_t first_triangle;
    uint64_t triangle_count;
    float bbox_min[3];           /* u_bboxMin (ConversionPass.cpp:111) */
    float bbox_max[3];           /* u_bboxMax */
    float base_color_factor[4];  /* u_materialFactor (ConversionPass.cpp:110) */
    int32_t albedo_texture;      /* index into m2s_scene.textures, -1 = hasAlbedoMap 0 */
    int32_t normal_texture;
    int32_t metallic_roughness_texture;
    int32_t reserved;
} m2s_primitive;

typedef struct m2s_scene {
    /* triangle soup, world space, M2S_FLOATS_PER_TRIANGLE floats per triangle:
     * 3 x { position xyz, normal xyz, tangent xyzw, uv } */
    const float* triangles;
    uint64_t triangle_count;
    const m2s_primitive* primitives;
    uint32_t primitive_count;
    const m2s_texture* textures;
    uint32_t texture_count;
} m2s_scene;

typedef struct m2s_params {
    uint32_t resolution;    /* R = resolutionTarget (ConversionPass.cpp:45): 1..4096 */
    float gaussian_std;     /* sigma (main.cpp:26 default 0.65); used by every layout but REF96 */
    uint64_t max_gaussians; /* 0 = reference rule (see M2S_FLAG_UNCAPPED) */
    uint32_t layout;        /* m2s_layout */
    uint32_t flags;
    /* shard of the flattened triangle list this call converts (multi-GPU: one contiguous range
     * per rank); triangle_count == 0 means "to the end" */
    uint64_t first_triangle;
    uint64_t triangle_count;
    /* pixel-row band of the R x R grid this call rasterises: rows [row_begin, row_end); row_end == 0 means
     * "to R".  Lets a multi-GPU plan split meshes made of a few huge triangles (SURVEY 8e: "split very large
     * triangles by pixel-row bands"): every rank takes all triangles but only its rows. */
    uint32_t row_begin;
    uint32_t row_end;
} m2s_params;

typedef struct m2s_result {
    uint64_t total;    /* fragments generated = the reference's numberOfGaussians
                          (may exceed capacity, ConversionPass.cpp:56-59) */
    uint64_t written;  /* records actually stored = min(total, cap) */
    uint64_t cap;      /* effective cap applied */
    float device_ms;   /* device time of the conversion kernel(s), CUDA events */
} m2s_result;

typedef struct m2s_ctx m2s_ctx;       /* one per GPU; externally synchronised */
typedef struct m2s_dscene m2s_dscene; /* device-resident scene (triangles, primitive table, mip chains) */

/* ---- housekeeping ------------------------------------------------------------------------- */
int m2s_version(void);
const char* m2s_last_error(void);
const char* m2s_status_string(m2s_status s);
uint32_t m2s_record_stride(uint32_t layout);
/* min(6*R*R*max(1,primitive_count), 7 000 000): ConversionPass.cpp:21-24 */
uint64_t m2s_reference_capacity(uint32_t resolution, uint32_t primitive_count);
void m2s_params_default(m2s_params* p);

m2s_status m2s_ctx_create(int device, m2s_ctx** out);
void m2s_ctx_destroy(m2s_ctx* ctx);
int m2s_ctx_device(const m2s_ctx* ctx);
/* Conditions raised on the device that an enqueue-only call cannot return: a fused-gather wait that timed out after
 * 2 s because a peer never published (M2S_E_CUDA), or an m2s_splat_enqueue whose quads touched more (tile, quad) pairs
 * than its max_pairs (M2S_E_CAPACITY).  M2S_OK if neither; clears the condition.  Call after synchronising. */
m2s_status m2s_ctx_status(m2s_ctx* ctx);
int m2s_ctx_sm_count(const m2s_ctx* ctx);

/* ---- inputs: replaces setupMeshBuffers + generateTextures ---------------------------------- */
/* Fills primitives[i].bbox_{min,max} from the triangle positions.  cumulative != 0 reproduces
 * the reference, where primitive k gets the union bbox of primitives 0..k
 * (SceneManager.cpp:476-477,514-520,527); 0 gives each primitive its own box. Host-only. */
m2s_status m2s_compute_bboxes(const float* triangles, m2s_primitive* primitives,
                              uint32_t primitive_count, int cumulative);

/* Copies triangles + primitive table + textures to the device and builds mip levels 1..4
 * (2x2 box, round-to-nearest) on the GPU.  Host pointers may be pageable. */
m2s_status m2s_scene_upload(m2s_ctx* ctx, const m2s_scene* scene, m2s_dscene** out);
/* One shard of a scene (multi-GPU: one contiguous triangle range per rank): copies the triangles
 * [first_triangle, first_triangle + triangle_count) to their global positions and, of the maps `layout` consumes, only
 * the texture rows those triangles can sample (16-row groups incl. their mip rows, REPEAT wrap and all five levels'
 * footprints considered).  Converting any triangle outside the range with the returned scene is undefined. */
m2s_status m2s_scene_upload_range(m2s_ctx* ctx, const m2s_scene* scene, uint32_t layout, uint64_t first_triangle,
                                  uint64_t triangle_count, m2s_dscene** out);
/* Payload bytes copied host -> device for this scene so far (triangles + texture rows); accounting for benchmarks. */
uint64_t m2s_scene_h2d_bytes(const m2s_dscene* scene);
/* The enqueue stream of the last conversion that used the scene must be idle (scratch and scene memory are
 * stream-ordered allocations of the context stream). */
void m2s_scene_free(m2s_ctx* ctx, m2s_dscene* scene);
/* Copies one generated mip level (RGBA8, tightly packed) back to the host; for parity tests. */
m2s_status m2s_scene_read_mip(m2s_ctx* ctx, const m2s_dscene* scene, uint32_t texture,
                              uint32_t level, uint8_t* dst, uint32_t* width, uint32_t* height);

/* ---- the hot path: replaces ConversionPass::execute ---------------------------------------- */
/* Enqueue-only form.  d_out: device buffer of out_capacity records; d_keys: optional device
 * array of out_capacity uint64 (fragment identity: triangle << 24 | y << 12 | x), may be NULL;
 * d_total: device uint64 receiving the fragment count; stream: cudaStream_t (NULL = context
 * stream).  Nothing is synchronised. */
m2s_status m2s_convert_enqueue(m2s_ctx* ctx, const m2s_dscene* scene, const m2s_params* params,
                               void* d_out, uint64_t out_capacity, uint64_t* d_keys,
                               uint64_t* d_total, void* stream);
/* enqueue + wait + read the counter back (the glFinish + counter readback of
 * ConversionPass.cpp:54-59).  Returns M2S_E_CAPACITY if total > cap (records up to cap are valid). */
m2s_status m2s_convert(m2s_ctx* ctx, const m2s_dscene* scene, const m2s_params* params,
                       void* d_out, uint64_t out_capacity, uint64_t* d_keys, m2s_result* result);
/* Measurement aid (not part of the reference's surface): one conversion on the context stream with an event between
 * the two kernels (which then do not overlap) — the per-kernel times of the step, for bench.py's roofline. */
m2s_status m2s_convert_timed(m2s_ctx* ctx, const m2s_dscene* scene, const m2s_params* params,
                             void* d_out, uint64_t out_capacity, float* raster_ms, float* fragment_ms);
/* Host-buffer form: upload scene, convert, download records (and keys if h_keys != NULL).
 * Everything a caller holding CPU data pays for.  Only the maps the layout consumes are uploaded, and of those only
 * the texture rows the converted triangle range can sample.  With >= 16384 triangles the call is pipelined: the
 * triangle range is converted in chunks (each bringing its triangles and texture rows with it) whose records are
 * appended on the device, and each chunk's download overlaps the next chunk's upload and kernels (pass pinned host
 * memory to benefit; M2S_HOST_CHUNKS=n overrides the chunk count, 1 = unpipelined).  The cap and the returned total
 * behave as in one launch. */
m2s_status m2s_convert_host(m2s_ctx* ctx, const m2s_scene* scene, const m2s_params* params,
                            void* h_out, uint64_t out_capacity, uint64_t* h_keys,
                            m2s_result* result);

/* ---- multi-GPU: conversion fused with the gather ------------------------------------------------
 * One process per GPU; rank r converts its own triangle range (params->first_triangle/triangle_count)
 * and its fragment kernel stores the records straight into the final buffer of EVERY rank (peer
 * memory over NVLink) at the rank-major global offset — the "single all-gather" of the conversion
 * result without a separate collective pass or a host round trip.  Buffers come from any allocator
 * that maps peer memory into each process (torch symmetric memory, cudaIpc*, cuMem*).
 * xch[p]: rank p's exchange block, M2S_MAX_PEERS*4 uint64, zeroed once before first use.
 * Every rank must make the same sequence of calls (an epoch counter pairs them up).  Layouts REF96 and
 * PACKED56.  d_total_global (device, optional) receives the number of records in the final buffer
 * once all ranks' records have landed; work enqueued after this call on `stream` sees the full buffer. */
#define M2S_MAX_PEERS 8
typedef struct m2s_peers {
    uint32_t world, rank;
    void* out[M2S_MAX_PEERS];
    uint64_t* xch[M2S_MAX_PEERS];
} m2s_peers;
m2s_status m2s_convert_gather_enqueue(m2s_ctx* ctx, const m2s_dscene* scene, const m2s_params* params,
                                      const m2s_peers* peers, uint64_t out_capacity, uint64_t* d_total_global,
                                      void* stream);

/* ---- outputs: replaces exportPly / savePlyVector -------------------------------------------- */
/* ASCII header of format 0/1/2 for `count` vertices; returns bytes written (excl. NUL) or the
 * needed size if dst is too small. */
size_t m2s_ply_header(uint32_t format, uint64_t count, char* dst, size_t dst_size);
/* GPU encoder: REF96 device records -> .ply body rows on the device (format 0/1/2). */
m2s_status m2s_ply_encode(m2s_ctx* ctx, const void* d_ref96, uint64_t count, uint32_t format,
                          float scale_multiplier, void* d_rows, void* stream);
/* Host writer: REF96 host records -> file, byte-identical to parsers::savePlyVector. */
m2s_status m2s_ply_write(const char* path, const void* h_ref96, uint64_t count, uint32_t format,
                         float scale_multiplier);

/* ---- file-level surface: loadModel -> execute -> exportPly --------------------------------- */
/* .glb -> host scene: SceneManager::parseGltfFile + setupMeshBuffers (bbox rule) + loadTextures
 * (src/utils/SceneManager.cpp:195-459,468-649): scene-graph world transforms, de-indexing, flat
 * normal / per-face tangent fallbacks, one primitive per glTF primitive, RGBA8 images.
 * cumulative_bbox != 0 keeps the reference's running-union bbox. */
typedef struct m2s_hscene m2s_hscene;
m2s_status m2s_glb_load(const char* glb_path, int cumulative_bbox, m2s_hscene** out);
const m2s_scene* m2s_hscene_view(const m2s_hscene* scene);
/* "<mesh name or 'mesh'>_<counter>" exactly as utils::Mesh::name (SceneManager.cpp:305-307) */
const char* m2s_hscene_primitive_name(const m2s_hscene* scene, uint32_t primitive);
void m2s_hscene_free(m2s_hscene* scene);

/* loadModel -> ConversionPass::execute -> exportPly in one call (the batch loop of
 * guiRendererConcreteMediator.cpp:146-193): capacity = the reference rule, .ply rows encoded on the GPU and
 * streamed to disk through two pinned buffers.  ply_format as exportPly's exportFormat (0 standard,
 * 1 PBR, 2 compressed; anything else = 0).  M2S_E_CAPACITY: the file holds the `cap` valid records. */
m2s_status m2s_convert_file(m2s_ctx* ctx, const char* glb_path, uint32_t resolution,
                            float gaussian_std, uint32_t ply_format, const char* ply_path,
                            m2s_result* result);

/* ---- the step after the path in the reference's frame graph: the viewer prepass (SURVEY 8 f-4) ----------------
 * GaussiansPrepass::execute (src/renderer/renderPasses/GaussiansPrepass.cpp:8-55) + gaussianSplattingPrepassCS.glsl
 * :58-204: per gaussian — model/view/clip transform, frustum cull (1.05 w), 3-D covariance from scale and rotation,
 * EWA projection to a 2-D conic (+0.3 low-pass), screen-space axes, atomic append of one QuadNdcTransformation (96 B:
 * gaussianMean2dNdc, quadScaleNdc, color, conic (.w = view depth), normal (.w = pbr.x), wsPos (.w = pbr.y)) and of the
 * view-space depth the radix sort keys on.  Matrices are column-major (glm::mat4).  Input records:
 *   M2S_LAYOUT_REF96     the reference's GaussianVertex, u_format 0 (scale * std_dev, normal through the normal matrix)
 *   M2S_LAYOUT_PACKED56  a standard 3DGS gaussian as the reference loads it from a .ply without PBR values, u_format 1
 *                        (scale = exp(log_scale), colour = SH0 * C0 + 0.5, alpha = sigmoid(opacity), normal = the
 *                        shortest axis, pbr = 0)
 * Not reproduced: the mesh depth test (u_depthTestMesh: needs the viewer's mesh depth pre-pass) and render mode 3 (debug
 * colours from the invocation id).  Output order is unspecified, as in the reference (atomic arrival order). */
typedef struct m2s_prepass_params {
    float world_to_view[16];   /* renderContext.viewMat */
    float view_to_clip[16];    /* renderContext.projMat */
    float model_to_world[16];  /* renderContext.modelMat */
    float resolution[2];       /* renderContext.rendererResolution */
    float near_far[2];
    float std_dev;             /* gaussianStd / resolutionTarget (GaussiansPrepass.cpp:18) */
    uint32_t render_mode;      /* 0 (or 6) colour, 1 depth, 2 normal; 4, 5: colour and opacity 0 (the shader's if-chain
                                  sets none), for the splatting pass's overdraw and metallic-roughness modes */
    uint32_t layout;           /* M2S_LAYOUT_REF96 or M2S_LAYOUT_PACKED56 */
    uint32_t reserved;
} m2s_prepass_params;
#define M2S_QUAD_BYTES 96u
/* Enqueue-only: d_quads holds `count` x 96 B, d_depths `count` floats, d_valid one uint32 (zeroed by the call, then the
 * number of surviving gaussians).  d_count (optional): device-side count that overrides `count` downwards (the
 * counter of a conversion that was only enqueued). */
m2s_status m2s_prepass_enqueue(m2s_ctx* ctx, const void* d_records, uint64_t count, const uint64_t* d_count,
                               const m2s_prepass_params* params, void* d_quads, float* d_depths, uint32_t* d_valid,
                               void* stream);
/* Synchronous variant on the context stream; *valid receives the counter. */
m2s_status m2s_prepass(m2s_ctx* ctx, const void* d_records, uint64_t count, const m2s_prepass_params* params,
                       void* d_quads, float* d_depths, uint32_t* valid);

/* ---- the passes after the prepass: depth sort (SURVEY 8 f-5) and splatting into the G-buffer (f-6) ----------------
 * RadixSortPass::execute (src/renderer/renderPasses/RadixSortPass.cpp:8-90, radixSortPrepass.glsl, radixSortGather.glsl,
 * thirdParty/RadixSort.hpp:1393-1530): key = floatBitsToUint(view depth) with no sign fix-up, value = prepass index;
 * the stable ascending order of the 32-bit keys over the prepass arrival order (survivors have negative view z: nearest
 * first); the gather moves each 96-byte quad to its sorted place.  d_count (optional): the prepass's d_valid, a device
 * count that overrides `count` downwards, so convert -> prepass -> sort -> splat needs no host round trip.  d_order
 * (optional) receives the prepass index of every sorted quad.  Scratch comes from the context's stream-ordered pool. */
m2s_status m2s_sort_quads_enqueue(m2s_ctx* ctx, const void* d_quads, const float* d_depths, uint64_t count,
                                  const uint32_t* d_count, void* d_sorted_quads, uint32_t* d_order, void* stream);
/* Synchronous variant on the context stream; device_ms (optional) receives the device time. */
m2s_status m2s_sort_quads(m2s_ctx* ctx, const void* d_quads, const float* d_depths, uint64_t count, void* d_sorted_quads,
                          uint32_t* d_order, float* device_ms);

/* GaussianSplattingPass::execute (GaussianSplattingPass.cpp:37-97) + gaussianSplattingVS.glsl + gaussianSplattingPS.glsl
 * into the 5-target G-buffer of Renderer::createGBuffer (renderer.cpp:329-379): every sorted quad is two triangles over
 * the corners (-1,-1), (-1,1), (1,1), (1,-1), rasterised into a width x height viewport with no depth test and no culling;
 * per fragment g = exp(-0.5 a dx^2 - 0.5 c dy^2 - b dx dy) and
 *   position = (wsPos, 1) g               RGBA16F
 *   normal   = (normal, opacity) g        RGBA16F
 *   albedo   = (rgb a, a) g               RGBA8    (render mode 4, overdraw: (.01, .005, 0, .01))
 *   depth    = (d, d, d, a g), d = z g    RGBA16F
 *   metallic_roughness = (m, r, 0, 1) g   RGBA8
 * blended front to back with ONE_MINUS_DST_ALPHA, ONE per target (mode 4: ONE, ONE) and converted to the storage format
 * after every fragment; the targets start cleared to 0.  Choices GL leaves to the implementation are listed in DESIGN.md
 * section 2.  Not reproduced: mode 3 (debug colours of the prepass) and the lighting of mode 6 (which writes the same
 * G-buffer as mode 0). */
typedef struct m2s_splat_params {
    uint32_t width, height;   /* renderContext.rendererResolution: 1..4096 each */
    uint32_t render_mode;     /* 0, 1, 2, 4, 5 or 6 */
    uint32_t reserved;
} m2s_splat_params;
/* Device images, row-major, row 0 = the bottom row (GL's window origin, as glReadPixels returns it).  position, normal and
 * depth hold half4 per pixel, albedo and metallic_roughness uchar4; every pointer 16-byte aligned. */
typedef struct m2s_gbuffer {
    void* position;
    void* normal;
    void* albedo;
    void* depth;
    void* metallic_roughness;
} m2s_gbuffer;
/* Non-lit composite of the deferred pass (gaussianSplattingDeferredPS.glsl:120-131) is a read of one target: mode 5 shows
 * (metallic_roughness.rg, 0, 1), every other mode but 6 (albedo.rgb, 1). */
/* Enqueue-only: d_sorted_quads holds `count` x 96 B (d_count as for the sort).  max_pairs: capacity of the (tile, quad) pair
 * scratch, 16 x 16 pixel tiles; the radix sort of the pairs runs over all max_pairs entries.  If the quads touch more
 * pairs, the G-buffer is left cleared and m2s_ctx_status reports M2S_E_CAPACITY. */
m2s_status m2s_splat_enqueue(m2s_ctx* ctx, const void* d_sorted_quads, uint64_t count, const uint32_t* d_count,
                             const m2s_splat_params* params, const m2s_gbuffer* gbuffer, uint64_t max_pairs, void* stream);
/* Synchronous variant on the context stream: counts the pairs, reads the count back and sizes the scratch exactly.
 * pairs and device_ms (both optional) receive the pair count and the device time of the pass. */
m2s_status m2s_splat(m2s_ctx* ctx, const void* d_sorted_quads, uint64_t count, const uint32_t* d_count,
                     const m2s_splat_params* params, const m2s_gbuffer* gbuffer, uint64_t* pairs, float* device_ms);

#ifdef __cplusplus
}
#endif
#endif /* M2S_H */
