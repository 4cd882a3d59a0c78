// m2s_render.cuh — arguments of the viewer's depth sort and splatting pass (m2s_render.cu), filled by the C-ABI host code
// (m2s_api.cu).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace m2s {

constexpr int kSplatTile = 16;                       // 16 x 16 pixels per tile, one CTA per tile, one thread per pixel
constexpr uint32_t kStatusSplatCapacity = 4u;        // context status bit: more (tile, quad) pairs than the scratch holds

// depth sort: stable ascending order of floatBitsToUint(depth) over the prepass arrival order, then the gather
struct SortArgs {
    const float4* quads;            // count x 6
    const float* depths;
    unsigned long long count;       // capacity of the inputs
    const uint32_t* d_count;        // optional device count (<= count)
    float4* sorted;                 // count x 6
    uint32_t* order;                // optional
    // scratch (count each) + CUB temporary storage
    uint32_t* keys[2];
    uint32_t* vals[2];
    void* temp;
    size_t temp_bytes;
};
size_t sort_temp_bytes(unsigned long long count);
cudaError_t sort_launch(const SortArgs& a, cudaStream_t stream);

struct SplatArgs {
    const float4* quads;            // sorted quads, count x 6
    unsigned long long count;
    const uint32_t* d_count;        // optional device count (<= count)
    int width, height;
    uint32_t mode;
    int tiles_x, tiles_y;
    unsigned long long max_pairs;
    // G-buffer: row 0 = bottom row
    uint2* position;                // half4
    uint2* normal;                  // half4
    uint32_t* albedo;               // uchar4
    uint2* depth;                   // half4
    uint32_t* metallic_roughness;   // uchar4
    uint32_t* status;               // context status word (mapped pinned host memory)
    // scratch
    void* rec;                      // count x SplatRec
    uint32_t* tiles;                // count: tiles each quad touches
    unsigned long long* incl;       // count: inclusive scan of `tiles`; incl[count - 1] = number of pairs
    uint32_t* keys[2];              // max_pairs each: tile id
    uint32_t* vals[2];              // max_pairs each: sorted quad index
    uint2* ranges;                  // tiles_x * tiles_y: [begin, end) of each tile's pairs
    void* temp;
    size_t temp_bytes;
};
size_t splat_rec_bytes();
size_t splat_scan_temp_bytes(unsigned long long count);
size_t splat_sort_temp_bytes(unsigned long long max_pairs, int tiles);
// Per quad set-up, tile counts and their scan: afterwards incl[count - 1] holds the number of (tile, quad) pairs.
cudaError_t splat_prepare(const SplatArgs& a, cudaStream_t stream);
// Pairs, their stable sort by tile, tile ranges and the per-tile blend into the G-buffer.  More pairs than max_pairs:
// the G-buffer is cleared and kStatusSplatCapacity is raised.
cudaError_t splat_finish(const SplatArgs& a, cudaStream_t stream);

}  // namespace m2s
