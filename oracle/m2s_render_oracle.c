/* m2s_render_oracle.c — CPU restatement of the viewer passes after the prepass (SURVEY 8 f-5, f-6).
 *
 * TEST INFRASTRUCTURE ONLY, like m2s_oracle.c: nothing under mesh2splat_b200/ may include, link or call this file.
 *
 *   depth sort       src/renderer/renderPasses/RadixSortPass.cpp:8-90, radixSortPrepass.glsl, radixSortGather.glsl,
 *                    thirdParty/RadixSort.hpp:1393-1530: the stable ascending order of floatBitsToUint(depth)
 *   splatting pass   src/renderer/renderPasses/GaussianSplattingPass.cpp:37-97, gaussianSplattingVS.glsl,
 *                    gaussianSplattingPS.glsl, G-buffer src/renderer/renderer.cpp:329-379
 * The fixed-function parts are restated from the OpenGL 4.6 core spec: 14.6.1 (polygon rasterisation with the rule
 * m2s_oracle.c's orc_triangle_setup follows for the conversion: 8 sub-pixel bits, pixel centres, top-left ownership,
 * +-8192-pixel guard band — here for a W x H viewport), 17.3.6 (blending) and the conversions of 2.3.4 / 8.24
 * (f32 -> f16 round to nearest even, f32 -> unorm8 rint(clamp(f) * 255), unorm8 -> f32 u / 255).
 *
 * Pinning: the vertex and fragment shader arithmetic is checked bit for bit against the reference's own
 * gaussianSplattingVS/PS.glsl compiled as C++ (oracle/build_render.py, tests/golden/ref_splat_vectors.npz).
 *
 * Arithmetic: fp32, one rounding per operation (build with -ffp-contract=off), GLM's operation order.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_API __attribute__((visibility("default")))

typedef struct orc_setup {
    int32_t X[3], Y[3]; /* window coords, 8 sub-pixel bits */
    int64_t area2;      /* signed doubled area in fixed point; 0 => no fragments */
    int32_t valid;      /* 0 if a coordinate is NaN/inf or beyond the guard band (never rasterised) */
    /* sign-normalised edge functions at pixel (i,j): E_k = A_k i + B_k j + C_k >= 0 inside */
    int64_t A[3], B[3], C[3];
    int32_t incl[3];    /* edge owns its E==0 samples (top-left rule) */
    int32_t x0, y0, x1, y1; /* inclusive candidate pixel box, empty if x1<x0 or y1<y0 */
} orc_setup;

static inline int64_t floor_div256(int64_t v) { return v >> 8; } /* arithmetic shift = floor */

/* Rasteriser set-up of one triangle in normalised device coordinates for a W x H viewport at the origin (GL 4.6 14.6.1 /
 * 13.8.1): xw = ndc*W/2 + W/2, snapped to 1/256 pixel; sign-normalised edge functions, top-left ownership, candidate pixel
 * box clamped to the viewport.  Fills the window-space fields of s; returns 1 if the triangle can produce fragments. */
static int orc_raster_setup(const float ndx[3], const float ndy[3], uint32_t W, uint32_t H, orc_setup* s) {
    const float hw = (float)W * 0.5f, hh = (float)H * 0.5f;
    s->valid = 1;
    for (int k = 0; k < 3; ++k) {
        float xw = ndx[k] * hw + hw, yw = ndy[k] * hh + hh;
        if (!isfinite(xw) || !isfinite(yw) || fabsf(xw) > 8192.0f || fabsf(yw) > 8192.0f) { s->valid = 0; xw = yw = 0.0f; }
        s->X[k] = (int32_t)lrintf(xw * 256.0f);
        s->Y[k] = (int32_t)lrintf(yw * 256.0f);
    }
    if (!s->valid) { s->area2 = 0; s->x1 = -1; s->y1 = -1; return 0; }
    int64_t area2 = (int64_t)(s->X[1] - s->X[0]) * (s->Y[2] - s->Y[0]) - (int64_t)(s->X[2] - s->X[0]) * (s->Y[1] - s->Y[0]);
    s->area2 = area2;
    if (area2 == 0) { s->x1 = -1; s->y1 = -1; return 0; }
    const int64_t sg = area2 < 0 ? -1 : 1;
    for (int k = 0; k < 3; ++k) {
        int a = (k + 1) % 3, b = (k + 2) % 3;
        int64_t dx = s->X[b] - s->X[a], dy = s->Y[b] - s->Y[a];
        s->A[k] = sg * (-dy * 256);
        s->B[k] = sg * (dx * 256);
        s->C[k] = sg * (dx * (128 - (int64_t)s->Y[a]) - dy * (128 - (int64_t)s->X[a]));
        s->incl[k] = (s->A[k] > 0) || (s->A[k] == 0 && s->B[k] > 0);
    }
    int32_t xmin = s->X[0], xmax = s->X[0], ymin = s->Y[0], ymax = s->Y[0];
    for (int k = 1; k < 3; ++k) {
        if (s->X[k] < xmin) xmin = s->X[k];
        if (s->X[k] > xmax) xmax = s->X[k];
        if (s->Y[k] < ymin) ymin = s->Y[k];
        if (s->Y[k] > ymax) ymax = s->Y[k];
    }
    int64_t x0 = floor_div256((int64_t)xmin + 127), x1 = floor_div256((int64_t)xmax - 128);
    int64_t y0 = floor_div256((int64_t)ymin + 127), y1 = floor_div256((int64_t)ymax - 128);
    if (x0 < 0) x0 = 0;
    if (y0 < 0) y0 = 0;
    if (x1 > (int64_t)W - 1) x1 = (int64_t)W - 1;
    if (y1 > (int64_t)H - 1) y1 = (int64_t)H - 1;
    s->x0 = (int32_t)x0; s->x1 = (int32_t)x1; s->y0 = (int32_t)y0; s->y1 = (int32_t)y1;
    return (x1 >= x0 && y1 >= y0) ? 1 : 0;
}

static inline int orc_inside(const orc_setup* s, int i, int j, int64_t E[3]) {
    for (int k = 0; k < 3; ++k) {
        E[k] = s->A[k] * i + s->B[k] * j + s->C[k];
        if (E[k] < 0 || (E[k] == 0 && !s->incl[k])) return 0;
    }
    return 1;
}

/* ------------------------------------------------------------------------------------------ */
/* viewer: depth sort (SURVEY 8 f-5)                                                            */
/* ------------------------------------------------------------------------------------------ */
/* order[i] = prepass index of the i-th quad in the stable ascending order of floatBitsToUint(depths) (LSD radix sort,
 * 4 passes of 8 bits: stable, as glu::RadixSort is). */
ORC_API void orc_sort_quads(const float* depths, uint32_t n, uint32_t* order) {
    uint32_t* keys = (uint32_t*)malloc((size_t)(n ? n : 1) * 4 * 3);
    uint32_t *k2 = keys + n, *o2 = keys + 2 * (size_t)n;
    memcpy(keys, depths, (size_t)n * 4);
    for (uint32_t i = 0; i < n; ++i) order[i] = i;
    uint32_t *ka = keys, *kb = k2, *oa = order, *ob = o2;
    for (int pass = 0; pass < 4; ++pass) {
        size_t cnt[257] = {0};
        const int sh = pass * 8;
        for (uint32_t i = 0; i < n; ++i) ++cnt[((ka[i] >> sh) & 255u) + 1];
        for (int b = 0; b < 256; ++b) cnt[b + 1] += cnt[b];
        for (uint32_t i = 0; i < n; ++i) {
            const size_t d = cnt[(ka[i] >> sh) & 255u]++;
            kb[d] = ka[i]; ob[d] = oa[i];
        }
        uint32_t* t = ka; ka = kb; kb = t;
        t = oa; oa = ob; ob = t;
    }
    /* four passes: the result is back in `order` */
    free(keys);
}

/* ------------------------------------------------------------------------------------------ */
/* viewer: splatting pass (SURVEY 8 f-6)                                                        */
/* ------------------------------------------------------------------------------------------ */
/* the varyings of gaussianSplattingVS.glsl (constant over the quad) */
typedef struct {
    float sx, sy, ocx, ocy, ocz, cr, cg, cb, op, nx, ny, nz, wx, wy, wz, dep, m0, m1;
} orc_vary;

/* quad: 24 floats (QuadNdcTransformation): mean, quadScale, color, conic (.w depth), normal (.w pbr.x), wsPos (.w pbr.y).
 * Corners (GaussianSplattingPass.cpp:10-15) in NDC: gl_Position = (mean.xy + (v.x * qs.xy + v.y * qs.zw), 0, 1). */
static void splat_vs(const float* q, float W, float H, float cx[4], float cy[4], orc_vary* v) {
    static const float vx[4] = {-1.0f, -1.0f, 1.0f, 1.0f}, vy[4] = {-1.0f, 1.0f, 1.0f, -1.0f};
    for (int c = 0; c < 4; ++c) {
        cx[c] = q[0] + (vx[c] * q[4] + vy[c] * q[6]);
        cy[c] = q[1] + (vx[c] * q[5] + vy[c] * q[7]);
    }
    v->sx = (q[0] + 1.0f) * 0.5f * W; v->sy = (q[1] + 1.0f) * 0.5f * H;
    v->ocx = -0.5f * q[12]; v->ocy = -q[13]; v->ocz = -0.5f * q[14];
    v->cr = q[8] * q[11]; v->cg = q[9] * q[11]; v->cb = q[10] * q[11]; v->op = q[11];
    v->nx = q[16]; v->ny = q[17]; v->nz = q[18]; v->wx = q[20]; v->wy = q[21]; v->wz = q[22];
    v->dep = q[15]; v->m0 = q[19]; v->m1 = q[23];
}

/* gaussianSplattingPS.glsl at gl_FragCoord (fx, fy): out = position, normal, albedo, depth, metallic-roughness (5 x 4) */
static void splat_ps(const orc_vary* v, float fx, float fy, uint32_t mode, float out[20]) {
    const float dx = v->sx - fx, dy = v->sy - fy;
    const float t0 = v->ocx * (dx * dx), t1 = v->ocz * (dy * dy), t2 = v->ocy * (dx * dy);   /* dot(out_conic.xzy, ...) */
    const float g = expf((t0 + t1) + t2);
    out[0] = v->wx * g; out[1] = v->wy * g; out[2] = v->wz * g; out[3] = 1.0f * g;
    out[4] = v->nx * g; out[5] = v->ny * g; out[6] = v->nz * g; out[7] = v->op * g;
    if (mode == 4) { out[8] = 0.01f; out[9] = 0.005f; out[10] = 0.0f; out[11] = 0.01f; }
    else { out[8] = v->cr * g; out[9] = v->cg * g; out[10] = v->cb * g; out[11] = v->op * g; }
    const float d = v->dep * g;
    out[12] = d; out[13] = d; out[14] = d; out[15] = v->op * g;
    out[16] = v->m0 * g; out[17] = v->m1 * g; out[18] = 0.0f * g; out[19] = 1.0f * g;
}

/* For the golden vectors: the 4 corners' gl_Position and the shader outputs at n fragment positions (frag_xy: n x 2). */
ORC_API void orc_splat_vertex(const float* quad, float W, float H, float corners[16]) {
    float cx[4], cy[4];
    orc_vary v;
    splat_vs(quad, W, H, cx, cy, &v);
    for (int c = 0; c < 4; ++c) { corners[4 * c] = cx[c]; corners[4 * c + 1] = cy[c]; corners[4 * c + 2] = 0.0f; corners[4 * c + 3] = 1.0f; }
}
ORC_API void orc_splat_fragments(const float* quad, float W, float H, uint32_t mode, const float* frag_xy, uint32_t n, float* out) {
    float cx[4], cy[4];
    orc_vary v;
    splat_vs(quad, W, H, cx, cy, &v);
    for (uint32_t i = 0; i < n; ++i) splat_ps(&v, frag_xy[2 * i], frag_xy[2 * i + 1], mode, out + 20 * (size_t)i);
}

static inline float cl01(float x) { return fminf(fmaxf(x, 0.0f), 1.0f); }
/* GL 4.6 17.3.6 blend into a float16 target (src * factor + dst, or src + dst for ONE, ONE), stored with round to nearest even */
static inline _Float16 blend_h(float s, float f, _Float16 d, int one) { return (_Float16)(one ? s + (float)d : s * f + (float)d); }
/* ... into an RGBA8 unorm target: source, destination and factor clamped to [0, 1] first; stored as rint(clamp(r) * 255) */
static inline uint8_t blend_u(float s, float f, uint8_t d, int one) {
    const float df = (float)d / 255.0f;
    const float r = one ? cl01(s) + df : cl01(s) * f + df;
    return (uint8_t)rintf(cl01(r) * 255.0f);
}

typedef struct { orc_setup t[2]; int ok[2]; orc_vary v; } orc_squad;

/* GaussianSplattingPass into a cleared W x H G-buffer (row 0 = bottom row): quads (n x 24 floats) in draw order, each two
 * triangles (0,1,2), (0,2,3); ONE_MINUS_DST_ALPHA, ONE per target (mode 4: ONE, ONE).  Targets: (H, W, 4) each. */
ORC_API void orc_splat(const float* quads, uint32_t n, uint32_t W, uint32_t H, uint32_t mode, _Float16* pos, _Float16* nrm, uint8_t* alb,
                       _Float16* dep, uint8_t* mr) {
    const size_t npx = (size_t)W * H * 4;
    memset(pos, 0, npx * 2); memset(nrm, 0, npx * 2); memset(dep, 0, npx * 2); memset(alb, 0, npx); memset(mr, 0, npx);
    const int one = mode == 4;
    const uint32_t kChunk = 1u << 16, kBand = 16;
    orc_squad* sq = (orc_squad*)malloc(sizeof(orc_squad) * kChunk);
    for (uint32_t c0 = 0; c0 < n; c0 += kChunk) {
        const uint32_t cn = n - c0 < kChunk ? n - c0 : kChunk;
        #pragma omp parallel for schedule(static)
        for (uint32_t i = 0; i < cn; ++i) {
            float cx[4], cy[4];
            splat_vs(quads + 24 * (size_t)(c0 + i), (float)W, (float)H, cx, cy, &sq[i].v);
            for (int t = 0; t < 2; ++t) {
                const float tx[3] = {cx[0], cx[1 + t], cx[2 + t]}, ty[3] = {cy[0], cy[1 + t], cy[2 + t]};
                memset(&sq[i].t[t], 0, sizeof(orc_setup));
                sq[i].ok[t] = orc_raster_setup(tx, ty, W, H, &sq[i].t[t]);
            }
        }
        /* row bands are independent: every band applies the chunk's quads in draw order */
        #pragma omp parallel for schedule(dynamic)
        for (uint32_t b0 = 0; b0 < H; b0 += kBand) {
            const int b1 = (int)(b0 + kBand < H ? b0 + kBand : H) - 1;
            for (uint32_t i = 0; i < cn; ++i) {
                for (int t = 0; t < 2; ++t) {
                    const orc_setup* s = &sq[i].t[t];
                    if (!sq[i].ok[t] || s->y1 < (int)b0 || s->y0 > b1) continue;
                    const int ya = s->y0 > (int)b0 ? s->y0 : (int)b0, yb = s->y1 < b1 ? s->y1 : b1;
                    for (int y = ya; y <= yb; ++y)
                        for (int x = s->x0; x <= s->x1; ++x) {
                            int64_t E[3];
                            if (!orc_inside(s, x, y, E)) continue;
                            float o[20];
                            splat_ps(&sq[i].v, (float)x + 0.5f, (float)y + 0.5f, mode, o);
                            const size_t p = ((size_t)y * W + x) * 4;
                            const float fp = 1.0f - (float)pos[p + 3], fn = 1.0f - (float)nrm[p + 3], fd = 1.0f - (float)dep[p + 3];
                            const float fa = cl01(1.0f - (float)alb[p + 3] / 255.0f), fm = cl01(1.0f - (float)mr[p + 3] / 255.0f);
                            for (int k = 0; k < 4; ++k) {
                                pos[p + k] = blend_h(o[k], fp, pos[p + k], one);
                                nrm[p + k] = blend_h(o[4 + k], fn, nrm[p + k], one);
                                alb[p + k] = blend_u(o[8 + k], fa, alb[p + k], one);
                                dep[p + k] = blend_h(o[12 + k], fd, dep[p + k], one);
                                mr[p + k] = blend_u(o[16 + k], fm, mr[p + k], one);
                            }
                        }
                }
            }
        }
    }
    free(sq);
}
