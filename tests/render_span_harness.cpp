// render_span_harness.cpp — the splatting kernel's triangle set-up (m2s_span.cuh: viewport_triangle_setup + span_covers)
// compiled for the host.  Built and run by tests/test_render_span_host.py (g++), which compares its coverage with the oracle's.
// stdin: W H n, then n quads as 6 floats (mean.xy, quadScale.xyzw); stdout: per quad, the number of covered pixels of each
// triangle followed by the covered pixel indices (y * W + x) of both triangles in order.
#include <cstdio>
#include <vector>
#include "../mesh2splat_b200/csrc/m2s_span.cuh"

int main() {
    int W, H, n;
    if (std::scanf("%d %d %d", &W, &H, &n) != 3) return 1;
    for (int i = 0; i < n; ++i) {
        float q[6];
        for (float& v : q) if (std::scanf("%f", &v) != 1) return 1;
        const float vx[4] = {-1.f, -1.f, 1.f, 1.f}, vy[4] = {-1.f, 1.f, 1.f, -1.f};
        float cx[4], cy[4];
        for (int c = 0; c < 4; ++c) {
            cx[c] = m2s::span_add(q[0], m2s::span_add(m2s::span_mul(vx[c], q[2]), m2s::span_mul(vy[c], q[4])));
            cy[c] = m2s::span_add(q[1], m2s::span_add(m2s::span_mul(vx[c], q[3]), m2s::span_mul(vy[c], q[5])));
        }
        std::vector<long> px;
        long cnt[2] = {0, 0};
        for (int t = 0; t < 2; ++t) {
            const float tx[3] = {cx[0], cx[1 + t], cx[2 + t]}, ty[3] = {cy[0], cy[1 + t], cy[2 + t]};
            m2s::RowState rs;
            int x0, y0, h;
            if (!m2s::viewport_triangle_setup(tx, ty, W, H, rs, x0, y0, h)) continue;
            for (int y = 0; y < h; ++y)
                for (int x = 0; x < rs.w; ++x)
                    if (m2s::span_covers(rs, x, y)) { ++cnt[t]; px.push_back((long)(y0 + y) * W + x0 + x); }
        }
        std::printf("%ld %ld", cnt[0], cnt[1]);
        for (long p : px) std::printf(" %ld", p);
        std::printf("\n");
    }
    return 0;
}
