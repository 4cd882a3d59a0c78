// m2s_render.cu — the two passes after the prepass in the reference's frame graph (SURVEY 8 f-5, f-6):
//   RadixSortPass (src/renderer/renderPasses/RadixSortPass.cpp:8-90, radixSortPrepass.glsl, radixSortGather.glsl,
//     thirdParty/RadixSort.hpp:1393-1530): key = floatBitsToUint(view depth), value = prepass index, a stable LSD radix
//     sort, then the gather of the 96-byte quads into depth order.
//   GaussianSplattingPass (GaussianSplattingPass.cpp:37-97, gaussianSplattingVS.glsl, gaussianSplattingPS.glsl, G-buffer
//     renderer.cpp:329-379): every sorted quad is two triangles (0,1,2), (0,2,3) rasterised into a W x H viewport with the
//     GL rules of m2s_span.cuh; each fragment evaluates the gaussian and is blended front to back (ONE_MINUS_DST_ALPHA, ONE;
//     overdraw mode 4: ONE, ONE) into five targets, each converted to its storage format after every fragment.
//
// Shape of the splat: a tile rasteriser.  (1) One thread per quad: both triangles' exact set-up and the 16 x 16 tiles
// their boxes touch; (2) a scan gives every quad its slot for (tile, quad) pairs; (3) a stable radix sort on the tile id
// bits only keeps the depth order inside each tile; (4) one CTA per tile, one thread per pixel: the tile's quads are
// staged in shared memory in batches of 256, every thread tests its pixel against both triangles (the integer edge
// functions, no second coverage rule) and blends the five targets in registers.  Blend arithmetic is fp32 with separate
// multiplies and adds (no FMA), as in the oracle.  The only early exit is the exact one: every pixel of the tile holds
// alpha == 1 in all five targets (a further fragment adds src * 0) and every remaining quad has finite values with a
// conic that keeps exp() finite.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda_fp16.h>
#include "m2s_render.cuh"
#include "m2s_span.cuh"

namespace m2s {

// ---------------------------------------------------------------------------------------------------------------------
// depth sort
// ---------------------------------------------------------------------------------------------------------------------
__global__ void sort_keys_kernel(const float* __restrict__ depths, unsigned long long count, const uint32_t* d_count,
                                 uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const unsigned long long n = d_count ? min(count, (unsigned long long)*d_count) : count;
    // entries past the device count sort last: all-ones keys, and among equal keys their indices are the largest
    keys[i] = i < n ? __float_as_uint(depths[i]) : 0xffffffffu;
    vals[i] = (uint32_t)i;
}

__global__ void sort_gather_kernel(const float4* __restrict__ quads, unsigned long long count, const uint32_t* d_count,
                                   const uint32_t* __restrict__ vals, float4* __restrict__ sorted, uint32_t* __restrict__ order) {
    const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;   // one float4 of the output
    const unsigned long long n = d_count ? min(count, (unsigned long long)*d_count) : count;
    if (t >= n * 6) return;
    const unsigned long long q = t / 6, part = t - q * 6;
    const uint32_t src = __ldg(vals + q);
    sorted[t] = __ldg(quads + (size_t)src * 6 + part);
    if (order && part == 0) order[q] = src;
}

size_t sort_temp_bytes(unsigned long long count) {
    size_t bytes = 0;
    cub::DoubleBuffer<uint32_t> k(nullptr, nullptr), v(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, k, v, (int)count, 0, 32);
    return bytes;
}

cudaError_t sort_launch(const SortArgs& a, cudaStream_t stream) {
    if (a.count == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((a.count + 255) / 256);
    sort_keys_kernel<<<blocks, 256, 0, stream>>>(a.depths, a.count, a.d_count, a.keys[0], a.vals[0]);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    cub::DoubleBuffer<uint32_t> k(a.keys[0], a.keys[1]), v(a.vals[0], a.vals[1]);
    size_t bytes = a.temp_bytes;
    e = cub::DeviceRadixSort::SortPairs(a.temp, bytes, k, v, (int)a.count, 0, 32, stream);
    if (e != cudaSuccess) return e;
    const unsigned long long threads = a.count * 6;
    sort_gather_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(a.quads, a.count, a.d_count, v.Current(), a.sorted, a.order);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------------
// splat: per quad set-up
// ---------------------------------------------------------------------------------------------------------------------
struct __align__(16) SplatRec {     // 112 B per sorted quad
    long long C[2][3];              // E'_k at the centre of pixel (0, 0), ownership bias folded in
    int A[2][3], B[2][3];
    unsigned short tx0, ty0, tx1, ty1;   // tiles the two triangles' boxes touch
    uint32_t flags;                 // bit t: triangle t can emit fragments; bit 2: "tame" (see below)
    uint32_t pad_;
};
static_assert(sizeof(SplatRec) == 112, "SplatRec layout");
constexpr uint32_t kTame = 4u;

size_t splat_rec_bytes() { return sizeof(SplatRec); }

__device__ __forceinline__ bool finite4(float4 v) { return isfinite(v.x) && isfinite(v.y) && isfinite(v.z) && isfinite(v.w); }

__global__ void splat_setup_kernel(const SplatArgs a) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.count) return;
    const unsigned long long n = a.d_count ? min(a.count, (unsigned long long)*a.d_count) : a.count;
    uint32_t tiles = 0;
    if (i < n) {
        const float4* q = a.quads + i * 6;
        const float4 mean = __ldg(q), qs = __ldg(q + 1);
        // gaussianSplattingVS.glsl: gl_Position = (mean.xy + (v.x * quadScale.xy + v.y * quadScale.zw), 0, 1) over the corners
        // (-1,-1), (-1,1), (1,1), (1,-1) (GaussianSplattingPass.cpp:10-15); the products are by +-1 and exact
        const float vx[4] = {-1.f, -1.f, 1.f, 1.f}, vy[4] = {-1.f, 1.f, 1.f, -1.f};
        float cx[4], cy[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            cx[c] = __fadd_rn(mean.x, __fadd_rn(__fmul_rn(vx[c], qs.x), __fmul_rn(vy[c], qs.z)));
            cy[c] = __fadd_rn(mean.y, __fadd_rn(__fmul_rn(vx[c], qs.y), __fmul_rn(vy[c], qs.w)));
        }
        SplatRec r;
        r.flags = 0; r.pad_ = 0;
        int bx0 = 1 << 30, by0 = 1 << 30, bx1 = -1, by1 = -1;
#pragma unroll
        for (int t = 0; t < 2; ++t) {   // indices (0,1,2), (0,2,3) (GaussianSplattingPass.cpp:17-20)
            const float tx[3] = {cx[0], cx[1 + t], cx[2 + t]}, ty[3] = {cy[0], cy[1 + t], cy[2 + t]};
            RowState rs;
            int x0, y0, h;
            if (viewport_triangle_setup(tx, ty, a.width, a.height, rs, x0, y0, h)) {
                r.flags |= 1u << t;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    r.C[t][k] = rs.E[k] - (long long)rs.A[k] * x0 - (long long)rs.B[k] * y0;
                    r.A[t][k] = rs.A[k]; r.B[t][k] = rs.B[k];
                }
                bx0 = min(bx0, x0); by0 = min(by0, y0); bx1 = max(bx1, x0 + rs.w - 1); by1 = max(by1, y0 + h - 1);
            } else {
#pragma unroll
                for (int k = 0; k < 3; ++k) { r.C[t][k] = -1; r.A[t][k] = 0; r.B[t][k] = 0; }
            }
        }
        if (r.flags) {
            r.tx0 = (unsigned short)(bx0 / kSplatTile); r.ty0 = (unsigned short)(by0 / kSplatTile);
            r.tx1 = (unsigned short)(bx1 / kSplatTile); r.ty1 = (unsigned short)(by1 / kSplatTile);
            tiles = (uint32_t)(r.tx1 - r.tx0 + 1) * (uint32_t)(r.ty1 - r.ty0 + 1);
            // "tame": every value the fragment shader reads is finite and the conic is positive semi-definite with a margin,
            // so g = exp(.) stays finite at every pixel and a fragment over a saturated pixel adds exactly src * 0
            const float4 col = __ldg(q + 2), con = __ldg(q + 3), nrm = __ldg(q + 4), ws = __ldg(q + 5);
            const double ca = con.x, cb = con.y, cc = con.z;
            if (isfinite(mean.x) && isfinite(mean.y) && finite4(col) && finite4(con) && finite4(nrm) && finite4(ws) && ca >= 0.0 &&
                cc >= 0.0 && cb * cb <= 0.999 * ca * cc)
                r.flags |= kTame;
        } else {
            r.tx0 = r.ty0 = 1; r.tx1 = r.ty1 = 0;
        }
        reinterpret_cast<SplatRec*>(a.rec)[i] = r;
    }
    a.tiles[i] = tiles;
}

size_t splat_scan_temp_bytes(unsigned long long count) {
    size_t bytes = 0;
    cub::DeviceScan::InclusiveSum(nullptr, bytes, (const uint32_t*)nullptr, (unsigned long long*)nullptr, (int)count);
    return bytes;
}

static int tile_bits(int tiles) {   // bits of the largest key: tile ids and the padding key `tiles`
    int b = 1;
    while ((1 << b) <= tiles) ++b;
    return b;
}

size_t splat_sort_temp_bytes(unsigned long long max_pairs, int tiles) {
    size_t bytes = 0;
    cub::DoubleBuffer<uint32_t> k(nullptr, nullptr), v(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, k, v, (int)max_pairs, 0, tile_bits(tiles));
    return bytes;
}

cudaError_t splat_prepare(const SplatArgs& a, cudaStream_t stream) {
    if (a.count == 0) return cudaSuccess;
    splat_setup_kernel<<<(unsigned)((a.count + 255) / 256), 256, 0, stream>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    size_t bytes = a.temp_bytes;
    return cub::DeviceScan::InclusiveSum(a.temp, bytes, a.tiles, a.incl, (int)a.count, stream);
}

// ---------------------------------------------------------------------------------------------------------------------
// splat: pairs, tile ranges
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long pair_total(const SplatArgs& a) { return a.count ? a.incl[a.count - 1] : 0ull; }

__global__ void splat_pad_kernel(const SplatArgs a) {   // pairs past the total sort last (key = number of tiles)
    const unsigned long long total = pair_total(a);
    const uint32_t pad = (uint32_t)(a.tiles_x * a.tiles_y);
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.max_pairs;
         i += (unsigned long long)gridDim.x * blockDim.x)
        if (i >= total) { a.keys[0][i] = pad; a.vals[0][i] = 0; }
    if (blockIdx.x == 0 && threadIdx.x == 0 && total > a.max_pairs && a.status) {
        atomicOr(a.status, kStatusSplatCapacity);   // zero-copy memory: seen by m2s_ctx_status after the stream is synchronised
        __threadfence_system();
    }
}

__global__ void splat_emit_kernel(const SplatArgs a) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.count || pair_total(a) > a.max_pairs) return;
    const uint32_t n = a.tiles[i];
    if (!n) return;
    const SplatRec& r = reinterpret_cast<const SplatRec*>(a.rec)[i];
    unsigned long long o = a.incl[i] - n;
    for (int ty = r.ty0; ty <= r.ty1; ++ty)
        for (int tx = r.tx0; tx <= r.tx1; ++tx, ++o) { a.keys[0][o] = (uint32_t)(ty * a.tiles_x + tx); a.vals[0][o] = (uint32_t)i; }
}

__global__ void splat_ranges_kernel(const SplatArgs a, const uint32_t* __restrict__ keys) {
    const unsigned long long total = pair_total(a);
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (total > a.max_pairs || i >= total) return;
    const uint32_t t = keys[i];
    if (i == 0 || keys[i - 1] != t) a.ranges[t].x = (uint32_t)i;
    if (i + 1 == total || keys[i + 1] != t) a.ranges[t].y = (uint32_t)(i + 1);
}

// ---------------------------------------------------------------------------------------------------------------------
// splat: per tile blend
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kBatch = kSplatTile * kSplatTile;   // quads staged per round = threads per CTA

struct SQuad {                      // one staged quad: both triangles relative to the tile origin + the shader's inputs
    long long E[6];                 // E'_k at the tile origin, triangle t = k / 3
    int A[6], B[6];
    float sx, sy;                   // out_screen
    float ocx, ocy, ocz;            // out_conic
    float cr, cg, cb, op;           // out_color (premultiplied), out_opacity
    float nx, ny, nz;               // out_normal
    float wx, wy, wz;               // out_wsPos
    float dep;                      // out_depth
    float m0, m1;                   // metallicRoughness
    uint32_t flags;
};

__device__ __forceinline__ float clamp01(float x) { return fminf(fmaxf(x, 0.0f), 1.0f); }
__device__ __forceinline__ float to_half(float x) { return __half2float(__float2half_rn(x)); }
// GL blend into a float16 target: src * factor + dst (factor ONE_MINUS_DST_ALPHA of this target, or ONE), stored as f16
__device__ __forceinline__ float blend_h(float s, float f, float d, bool one) { return to_half(one ? __fadd_rn(s, d) : __fadd_rn(__fmul_rn(s, f), d)); }
// ... into an RGBA8 unorm target: source, destination and factor clamped to [0, 1] (GL 4.6 17.3.6), rint(clamp(r) * 255)
__device__ __forceinline__ uint32_t blend_u(float s, float f, float d, bool one) {
    const float r = one ? __fadd_rn(clamp01(s), d) : __fadd_rn(__fmul_rn(clamp01(s), f), d);
    return (uint32_t)__float2int_rn(__fmul_rn(clamp01(r), 255.0f));
}
__device__ __forceinline__ uint2 pack_half4(const float v[4]) {
    const __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], v[3]);
    return make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}

__global__ void __launch_bounds__(kBatch, 2) splat_tile_kernel(const SplatArgs a, const uint32_t* __restrict__ vals) {
    __shared__ SQuad sq[kBatch];
    __shared__ float u8f[256];      // unorm8 -> f32: u / 255
    const int tid = threadIdx.x, lx = tid % kSplatTile, ly = tid / kSplatTile;
    const int tile = blockIdx.x, tx = tile % a.tiles_x, ty = tile / a.tiles_x;
    const int px = tx * kSplatTile + lx, py = ty * kSplatTile + ly;
    const bool inside = px < a.width && py < a.height;
    u8f[tid] = __fdiv_rn((float)tid, 255.0f);
    const bool over = pair_total(a) > a.max_pairs;
    const uint2 range = over ? make_uint2(0, 0) : a.ranges[tile];
    const bool one = a.mode == 4;
    const float fx = (float)px + 0.5f, fy = (float)py + 0.5f;   // gl_FragCoord.xy
    float pos[4] = {0, 0, 0, 0}, nrm[4] = {0, 0, 0, 0}, dep[4] = {0, 0, 0, 0};
    uint32_t alb[4] = {0, 0, 0, 0}, mr[4] = {0, 0, 0, 0};
    bool check_exit = !one;
    __syncthreads();
    for (uint32_t b0 = range.x; b0 < range.y; b0 += kBatch) {
        if (check_exit) {   // exact early exit (see the file comment)
            const bool sat = !inside || (pos[3] == 1.0f && nrm[3] == 1.0f && dep[3] == 1.0f && alb[3] == 255u && mr[3] == 255u);
            if (__syncthreads_and(sat)) {
                bool wild = false;
                for (uint32_t j = b0 + tid; j < range.y; j += kBatch)
                    wild |= !(reinterpret_cast<const SplatRec*>(a.rec)[vals[j]].flags & kTame);
                if (!__syncthreads_or(wild)) break;
                check_exit = false;   // a wild quad is still to come: blend everything
            }
        }
        const uint32_t nb = min((uint32_t)kBatch, range.y - b0);
        __syncthreads();
        if ((uint32_t)tid < nb) {
            const uint32_t qi = vals[b0 + tid];
            const SplatRec& r = reinterpret_cast<const SplatRec*>(a.rec)[qi];
            const float4* q = a.quads + (size_t)qi * 6;
            const float4 mean = __ldg(q), col = __ldg(q + 2), con = __ldg(q + 3), nn = __ldg(q + 4), ws = __ldg(q + 5);
            SQuad& s = sq[tid];
            const int ox = tx * kSplatTile, oy = ty * kSplatTile;
#pragma unroll
            for (int t = 0; t < 2; ++t)
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const int A = r.A[t][k], B = r.B[t][k];
                    s.E[t * 3 + k] = r.C[t][k] + (long long)A * ox + (long long)B * oy;
                    s.A[t * 3 + k] = A; s.B[t * 3 + k] = B;
                }
            s.flags = r.flags;
            // gaussianSplattingVS.glsl: out_screen = (mean.xy + 1) * 0.5 * u_resolution, out_conic = (-0.5 a, -b, -0.5 c),
            // out_color = color.rgb * color.a, metallicRoughness = (normal.w, wsPos.w)
            s.sx = __fmul_rn(__fmul_rn(__fadd_rn(mean.x, 1.0f), 0.5f), (float)a.width);
            s.sy = __fmul_rn(__fmul_rn(__fadd_rn(mean.y, 1.0f), 0.5f), (float)a.height);
            s.ocx = __fmul_rn(-0.5f, con.x); s.ocy = -con.y; s.ocz = __fmul_rn(-0.5f, con.z);
            s.cr = __fmul_rn(col.x, col.w); s.cg = __fmul_rn(col.y, col.w); s.cb = __fmul_rn(col.z, col.w); s.op = col.w;
            s.nx = nn.x; s.ny = nn.y; s.nz = nn.z; s.wx = ws.x; s.wy = ws.y; s.wz = ws.z; s.dep = con.w; s.m0 = nn.w; s.m1 = ws.w;
        }
        __syncthreads();
        if (inside) {
            for (uint32_t j = 0; j < nb; ++j) {
                const SQuad& s = sq[j];
                for (int t = 0; t < 2; ++t) {
                    if (!(s.flags & (1u << t))) continue;
                    const int k0 = t * 3;
                    if (s.E[k0] + (long long)s.A[k0] * lx + (long long)s.B[k0] * ly < 0 ||
                        s.E[k0 + 1] + (long long)s.A[k0 + 1] * lx + (long long)s.B[k0 + 1] * ly < 0 ||
                        s.E[k0 + 2] + (long long)s.A[k0 + 2] * lx + (long long)s.B[k0 + 2] * ly < 0)
                        continue;
                    // gaussianSplattingPS.glsl
                    const float dx = __fsub_rn(s.sx, fx), dy = __fsub_rn(s.sy, fy);
                    const float al = __fadd_rn(__fadd_rn(__fmul_rn(s.ocx, __fmul_rn(dx, dx)), __fmul_rn(s.ocz, __fmul_rn(dy, dy))),
                                               __fmul_rn(s.ocy, __fmul_rn(dx, dy)));
                    const float g = expf(al);
                    const float sp[4] = {__fmul_rn(s.wx, g), __fmul_rn(s.wy, g), __fmul_rn(s.wz, g), g};
                    const float sn[4] = {__fmul_rn(s.nx, g), __fmul_rn(s.ny, g), __fmul_rn(s.nz, g), __fmul_rn(s.op, g)};
                    const float dd = __fmul_rn(s.dep, g);
                    const float sd[4] = {dd, dd, dd, __fmul_rn(s.op, g)};
                    const float sa[4] = {one ? 0.01f : __fmul_rn(s.cr, g), one ? 0.005f : __fmul_rn(s.cg, g), one ? 0.0f : __fmul_rn(s.cb, g),
                                         one ? 0.01f : __fmul_rn(s.op, g)};
                    const float sm[4] = {__fmul_rn(s.m0, g), __fmul_rn(s.m1, g), __fmul_rn(0.0f, g), g};
                    const float fp = __fsub_rn(1.0f, pos[3]), fn = __fsub_rn(1.0f, nrm[3]), fd = __fsub_rn(1.0f, dep[3]);
                    const float fa = clamp01(__fsub_rn(1.0f, u8f[alb[3]])), fm = clamp01(__fsub_rn(1.0f, u8f[mr[3]]));
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        pos[c] = blend_h(sp[c], fp, pos[c], one);
                        nrm[c] = blend_h(sn[c], fn, nrm[c], one);
                        dep[c] = blend_h(sd[c], fd, dep[c], one);
                        alb[c] = blend_u(sa[c], fa, u8f[alb[c]], one);
                        mr[c] = blend_u(sm[c], fm, u8f[mr[c]], one);
                    }
                }
            }
        }
    }
    if (!inside) return;
    const size_t o = (size_t)py * a.width + px;
    a.position[o] = pack_half4(pos);
    a.normal[o] = pack_half4(nrm);
    a.depth[o] = pack_half4(dep);
    a.albedo[o] = alb[0] | (alb[1] << 8) | (alb[2] << 16) | (alb[3] << 24);
    a.metallic_roughness[o] = mr[0] | (mr[1] << 8) | (mr[2] << 16) | (mr[3] << 24);
}

cudaError_t splat_finish(const SplatArgs& a, cudaStream_t stream) {
    const int tiles = a.tiles_x * a.tiles_y;
    cudaError_t e = cudaMemsetAsync(a.ranges, 0, (size_t)tiles * sizeof(uint2), stream);
    if (e != cudaSuccess) return e;
    const uint32_t* sorted_vals = a.vals[0];
    if (a.count && a.max_pairs) {
        const unsigned pad_blocks = (unsigned)min((a.max_pairs + 255) / 256, 4096ull);
        splat_pad_kernel<<<pad_blocks, 256, 0, stream>>>(a);
        splat_emit_kernel<<<(unsigned)((a.count + 255) / 256), 256, 0, stream>>>(a);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        cub::DoubleBuffer<uint32_t> k(a.keys[0], a.keys[1]), v(a.vals[0], a.vals[1]);
        size_t bytes = a.temp_bytes;
        e = cub::DeviceRadixSort::SortPairs(a.temp, bytes, k, v, (int)a.max_pairs, 0, tile_bits(tiles), stream);
        if (e != cudaSuccess) return e;
        splat_ranges_kernel<<<(unsigned)((a.max_pairs + 255) / 256), 256, 0, stream>>>(a, k.Current());
        sorted_vals = v.Current();
    } else if (a.count) {
        splat_pad_kernel<<<1, 32, 0, stream>>>(a);   // raises the capacity condition if there are pairs
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    splat_tile_kernel<<<tiles, kBatch, 0, stream>>>(a, sorted_vals);
    return cudaGetLastError();
}

}  // namespace m2s
