// m2s_span.cuh — exact coverage of one pixel row of a triangle's candidate box as an interval.
//
// The rasteriser's rule (GL 4.6 14.6.1, restated in oracle/m2s_oracle.c): pixel (x, y) of the box is covered iff
// E'_k(x, y) = E_k(x, y) - (edge k owns its zero set ? 0 : 1) >= 0 for the three sign-normalised integer edge
// functions E_k = A_k x + B_k y + C_k.  For a fixed row the covered set is the intersection of three half-lines,
// i.e. ONE interval [xl, xl + n): it is computed here with three estimated divisions, each corrected by exact
// int64 evaluations, so the result is bit-identical to testing every pixel centre — at O(1) per row instead
// of O(width).  Used by raster_kernel (to count) and fragment_kernel (to enumerate); also compiled for the host
// by tests/test_span_host.py (g++), which checks it against the brute-force per-pixel test.
#pragma once
#include <cmath>
#include <cstdint>

#if defined(__CUDACC__)
#define M2S_HD __host__ __device__ __forceinline__
#else
#define M2S_HD inline
#endif

namespace m2s {

struct RowState {   // one triangle, relative to the origin (x0, y0) of its candidate box
    long long E[3]; // E'_k at the box origin (ownership bias folded in: covered <=> all E' >= 0)
    int A[3];       // dE_k/dx per pixel
    int B[3];       // dE_k/dy per pixel
    int w;          // box width in pixels (1..4096)
};

M2S_HD float span_quot(long long num, int den) {  // estimate of num / den, num >= 0, den > 0
#if defined(__CUDA_ARCH__)
    return __fdividef(__ll2float_rn(num), __int2float_rn(den));
#else
    return (float)num / (float)den;
#endif
}

// Row `yrel` (0-based inside the box): returns the number of covered pixels, xl = first covered column.
M2S_HD uint32_t span_row(const RowState& s, int yrel, int& xl) {
    int lo = 0, hi = s.w - 1;
    const float wlim = (float)s.w + 2.0f;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k < 3; ++k) {
        const long long D = s.E[k] + (long long)s.B[k] * yrel;  // E'_k at column 0 of this row
        const int A = s.A[k];
        if (A == 0) {
            if (D < 0) hi = -1;
        } else if (A > 0) {             // covered for x >= ceil(-D / A)
            if (D < 0) {
                const float qf = span_quot(-D, A);
                if (!(qf < wlim)) hi = -1;      // the boundary lies right of the box (also catches inf/NaN)
                else {
                    int x = (int)qf;
                    long long e = D + (long long)A * x;
                    while (e < 0) { ++x; e += A; }                     // exact fix-up of the estimate
                    while (x > 0 && e - A >= 0) { --x; e -= A; }
                    lo = lo > x ? lo : x;
                }
            }
        } else {                        // covered for x <= floor(D / -A)
            if (D < 0) hi = -1;
            else {
                const float qf = span_quot(D, -A);
                if (qf < wlim) {                // else: no constraint inside the box
                    int x = (int)qf + 1;
                    long long e = D + (long long)A * x;
                    while (e < 0) { --x; e -= A; }                     // A < 0: stepping left raises e
                    while (e + A >= 0) { ++x; e += A; }
                    hi = hi < x ? hi : x;
                }
            }
        }
    }
    xl = lo;
    return hi >= lo ? (uint32_t)(hi - lo + 1) : 0u;
}

// The same rule for one pixel of the box: (xrel, yrel) relative to the box origin.
M2S_HD bool span_covers(const RowState& s, int xrel, int yrel) {
    bool in = true;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k < 3; ++k) in = in && s.E[k] + (long long)s.A[k] * xrel + (long long)s.B[k] * yrel >= 0;
    return in;
}

// fp32 operations without contraction, on the device and on the host (built with -ffp-contract=off there)
M2S_HD float span_mul(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
M2S_HD float span_add(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
// Rasteriser set-up of one triangle given in normalised device coordinates (w = 1) for a W x H viewport at the origin
// (GL 4.6 13.8.1, 14.6.1): xw = ndc * W/2 + W/2 in fp32 without contraction, snapped to 1/256 pixel; sign-normalised
// edge functions with top-left ownership folded in; candidate box clamped to the viewport (which is also the clip:
// GL clips to |x|, |y| <= w, exactly the pixels inside the viewport).  A corner that is not finite or lies beyond
// the 8192-pixel guard band (the conversion's guard; the int32 edge steps need it) drops the triangle.  Returns false
// if it cannot emit a fragment; else rs (relative to the box origin (x0, y0)) and the box height h.
M2S_HD bool viewport_triangle_setup(const float ndx[3], const float ndy[3], int W, int H, RowState& rs, int& x0, int& y0, int& h) {
    const float hw = (float)W * 0.5f, hh = (float)H * 0.5f;
    int X[3], Y[3];
    bool valid = true;
    for (int k = 0; k < 3; ++k) {
        const float xw = span_add(span_mul(ndx[k], hw), hw), yw = span_add(span_mul(ndy[k], hh), hh);
        if (!(xw >= -8192.0f && xw <= 8192.0f) || !(yw >= -8192.0f && yw <= 8192.0f)) valid = false;   // also rejects NaN
        X[k] = valid ? (int)rintf(span_mul(xw, 256.0f)) : 0;
        Y[k] = valid ? (int)rintf(span_mul(yw, 256.0f)) : 0;
    }
    if (!valid) return false;
    const long long area2 = (long long)(X[1] - X[0]) * (Y[2] - Y[0]) - (long long)(X[2] - X[0]) * (Y[1] - Y[0]);
    if (area2 == 0) return false;
    int xmin = X[0], xmax = X[0], ymin = Y[0], ymax = Y[0];
    for (int k = 1; k < 3; ++k) {
        xmin = X[k] < xmin ? X[k] : xmin; xmax = X[k] > xmax ? X[k] : xmax;
        ymin = Y[k] < ymin ? Y[k] : ymin; ymax = Y[k] > ymax ? Y[k] : ymax;
    }
    int bx0 = (xmin + 127) >> 8, bx1 = (xmax - 128) >> 8, by0 = (ymin + 127) >> 8, by1 = (ymax - 128) >> 8;
    bx0 = bx0 < 0 ? 0 : bx0; by0 = by0 < 0 ? 0 : by0;
    bx1 = bx1 > W - 1 ? W - 1 : bx1; by1 = by1 > H - 1 ? H - 1 : by1;
    if (bx1 < bx0 || by1 < by0) return false;
    const int sg = area2 < 0 ? -1 : 1;
    for (int k = 0; k < 3; ++k) {
        const int va = (k + 1) % 3, vb = (k + 2) % 3;
        const int dx = X[vb] - X[va], dy = Y[vb] - Y[va];
        const int A = sg * (-dy * 256), B = sg * (dx * 256);
        const long long C = (long long)sg * ((long long)dx * (128 - Y[va]) - (long long)dy * (128 - X[va]));
        const bool owns = A > 0 || (A == 0 && B > 0);
        rs.E[k] = C + (long long)A * bx0 + (long long)B * by0 - (owns ? 0 : 1);
        rs.A[k] = A; rs.B[k] = B;
    }
    rs.w = bx1 - bx0 + 1;
    x0 = bx0; y0 = by0; h = by1 - by0 + 1;
    return true;
}

}  // namespace m2s
