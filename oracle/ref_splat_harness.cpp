// ref_splat_harness.cpp — hosts the REFERENCE's splatting shaders on the CPU (TEST INFRASTRUCTURE).
//
// oracle/build_render.py rewrites src/shaders/rendering/gaussianSplattingVS.glsl and gaussianSplattingPS.glsl into
// oracle/_ref/splatVS.inc and splatPS.inc (qualifier / layout / literal / swizzle token rewrites only) and this file gives
// them the GLSL environment they expect: GLM types (the reference's vendored copy), the vertex attributes, gl_Position,
// gl_FragCoord and the five colour outputs.  Nothing here restates the shaders' arithmetic.  The varyings are flat over a
// quad (every corner computes the same values), so the fragment shader reads those of the first corner.
#define GLM_FORCE_SWIZZLE   // .xy() / .zw() / .rgb() / .xzy() swizzle functions
#include <cmath>
#include <cstdint>
#include <cstring>
#include <glm/glm.hpp>

#define REF_API extern "C" __attribute__((visibility("default")))

namespace refvs {
using namespace glm;
static vec4 gl_Position;
#include "splatVS.inc"
}  // namespace refvs

namespace refps {
using namespace glm;
static vec4 gl_FragCoord;
#include "splatPS.inc"
}  // namespace refps

// quad: 24 floats (QuadNdcTransformation); frag_xy: n x 2 (gl_FragCoord.xy); corners: 4 x 4 (gl_Position of the corners
// (-1,-1), (-1,1), (1,1), (1,-1), GaussianSplattingPass.cpp:10-15); out: n x 5 x 4 (gPosition, gNormal, gAlbedo, gDepth,
// gMetallicRoughness).
REF_API void ref_splat(const float* quad, float width, float height, int render_mode, const float* frag_xy, uint32_t n, float* corners,
                       float* out) {
    static const float vx[4] = {-1.0f, -1.0f, 1.0f, 1.0f}, vy[4] = {-1.0f, 1.0f, 1.0f, -1.0f};
    refvs::u_resolution = glm::vec2(width, height);
    std::memcpy(&refvs::gaussianMean2Ndc, quad, 16); std::memcpy(&refvs::quadScaleNdc, quad + 4, 16);
    std::memcpy(&refvs::color, quad + 8, 16); std::memcpy(&refvs::conic, quad + 12, 16);
    std::memcpy(&refvs::normal, quad + 16, 16); std::memcpy(&refvs::gaussianWsPos, quad + 20, 16);
    for (int c = 3; c >= 0; --c) {   // corner 0 last: its varyings are the ones passed on
        refvs::vertexPos = glm::vec4(vx[c], vy[c], 0.0f, 1.0f);
        refvs::main();
        std::memcpy(corners + 4 * c, &refvs::gl_Position, 16);
    }
    refps::out_color = refvs::out_color; refps::out_opacity = refvs::out_opacity; refps::out_screen = refvs::out_screen;
    refps::out_conic = refvs::out_conic; refps::out_normal = refvs::out_normal; refps::out_wsPos = refvs::out_wsPos;
    refps::out_depth = refvs::out_depth; refps::metallicRoughness = refvs::metallicRoughness;
    refps::u_resolution = glm::vec2(width, height); refps::u_renderMode = render_mode;
    for (uint32_t i = 0; i < n; ++i) {
        refps::gl_FragCoord = glm::vec4(frag_xy[2 * i], frag_xy[2 * i + 1], 0.0f, 1.0f);
        refps::main();
        std::memcpy(out + 20 * (size_t)i, &refps::gPosition, 16);
        std::memcpy(out + 20 * (size_t)i + 4, &refps::gNormal, 16);
        std::memcpy(out + 20 * (size_t)i + 8, &refps::gAlbedo, 16);
        std::memcpy(out + 20 * (size_t)i + 12, &refps::gDepth, 16);
        std::memcpy(out + 20 * (size_t)i + 16, &refps::gMetallicRoughness, 16);
    }
}
