// shipsim_render.cu -- debug rendering of ONE selected env to an RGB image (SURVEY.md §8 f4).
// Replaces, for inspection purposes, ShipGame.render (game.py:197-229: blue background, pymunk debug-draw of the
// shapes, a circle per lidar ray at the point the ray reached, a yellow circle on the ship's position) and
// ShipGame.get_screen (game.py:133-138), the `rgb_array` mode ShipEnv.metadata promises (ship_env.py:18).
// One thread per pixel, analytic point-in-shape tests against the same fp32 planes the step kernels use; nothing here
// is on the hot path.
#include "shipsim_device.cuh"
#include "shipsim_launch.h"

namespace shipsim {

__global__ void __launch_bounds__(256) render_kernel(const __grid_constant__ StepParams p, int e, int img_w, int img_h, uint8_t *rgb)
{
    const int px = blockIdx.x * blockDim.x + threadIdx.x, py = blockIdx.y * blockDim.y + threadIdx.y;
    if (px >= img_w || py >= img_h) return;
    // pixel centre -> world; screen y points down (ShipGame.invert_p, game.py)
    const float wx = (px + 0.5f) * p.W / (float)img_w;
    const float wy = p.H - (py + 0.5f) * p.H / (float)img_h;

    EnvRegs r;
    float4 l0, l1, l2, g0, g1, g2;
    load_env(p, e, r, l0, l1, l2, g0, g1, g2);
    // lidar[0..9] in state planes 2-4, lidar[10..] in the appended planes (shipsim_state_bytes)
    auto reading = [&](int j) {
        if (j >= kBeams) {
            const float4 v = p.state[(size_t)(kPlanes + (j - kBeams) / 4) * p.N + e];
            const int c = (j - kBeams) & 3;
            return c == 0 ? v.x : (c == 1 ? v.y : (c == 2 ? v.z : v.w));
        }
        const float lid[kBeams] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w, l2.x, l2.y};
        return lid[j];
    };
    float2 g[kGoals];
    unpack_goals(g0, g1, g2, g);

    uchar3 col = make_uchar3(0, 0, 200);                                 // screen.fill((0, 0, 200))
    // river banks (static polygons)
    const float4 *rec = p.bank + (size_t)r.scen * p.scen_stride4;
    const float4 hdr = __ldg(rec + 4);
    for (int b = 0; b < 2; ++b) {
        const int nb = __float_as_int(b ? hdr.w : hdr.z);
        bool inside = nb > 0;
        for (int i = 0; i < nb; ++i) {
            const float4 ed = __ldg(rec + kBankHeader4 + b * p.maxv + i);    // nx, ny, v_i
            if (ed.x * (wx - ed.z) + ed.y * (wy - ed.w) > 0.f) inside = false;
        }
        if (inside) col = make_uchar3(110, 110, 110);
    }
    // remaining goals (radius-5 circles)
    for (int k = 0; k < kGoals; ++k) {
        const float dx = wx - g[k].x, dy = wy - g[k].y;
        if (((r.alive >> k) & 1) && dx * dx + dy * dy <= p.goal_r * p.goal_r) col = make_uchar3(0, 200, 0);
    }
    // the ship's hull
    float s, c;
    sincos_fast(r.th, s, c);
    {
        const float ux = wx - r.x, uy = wy - r.y;
        const float qx = ux * c + uy * s, qy = -ux * s + uy * c;           // body frame
        bool inside = true;
#pragma unroll
        for (int j = 0; j < kShipVerts; ++j)
            if (p.ship_nx[j] * (qx - p.ship_lx[j]) + p.ship_ny[j] * (qy - p.ship_ly[j]) > 0.f) inside = false;
        if (inside) col = make_uchar3(255, 255, 255);
    }
    // lidar: a circle of radius 10 where each ray ended -- red at the sticky reading of a ray that has hit, green at
    // the full ray length otherwise (game.py:206-222)
    {
        float minx = 0.f, maxx = 0.f, miny = 0.f, maxy = 0.f;               // models.py:51-54: origin = corner + half the world AABB
#pragma unroll
        for (int j = 1; j < kShipVerts; ++j) {
            const float hx = p.ship_lx[j] * c - p.ship_ly[j] * s, hy = p.ship_lx[j] * s + p.ship_ly[j] * c;
            minx = fminf(minx, hx); maxx = fmaxf(maxx, hx); miny = fminf(miny, hy); maxy = fmaxf(maxy, hy);
        }
        const float ox = r.x + 0.5f * (maxx - minx), oy = r.y + 0.5f * (maxy - miny);
        for (int j = 0; j < p.n_beams; ++j) {             // one marker per ray of the fan
            const float dirx = c * p.ray_cw[j] - s * p.ray_sw[j], diry = s * p.ray_cw[j] + c * p.ray_sw[j];
            const float v = reading(j);
            const bool hit = v >= 0.f && v < p.lidar_len;
            const float len = hit ? v : p.lidar_len;
            const float dx = wx - (ox + len * dirx), dy = wy - (oy + len * diry);
            if (dx * dx + dy * dy <= 100.f) col = hit ? make_uchar3(255, 0, 0) : make_uchar3(0, 255, 0);
        }
    }
    // pygame.draw.circle(screen, (255, 255, 0), player.position, 10)
    {
        const float dx = wx - r.x, dy = wy - r.y;
        if (dx * dx + dy * dy <= 100.f) col = make_uchar3(255, 255, 0);
    }
    uint8_t *o = rgb + ((size_t)py * img_w + px) * 3;
    o[0] = col.x; o[1] = col.y; o[2] = col.z;
}

cudaError_t launch_render(const StepParams &p, int e, int img_w, int img_h, uint8_t *rgb, cudaStream_t stream)
{
    const dim3 block(32, 8), grid((img_w + 31) / 32, (img_h + 7) / 8);
    render_kernel<<<grid, block, 0, stream>>>(p, e, img_w, img_h, rgb);
    return cudaGetLastError();
}

}  // namespace shipsim
