// shipsim_scengen.cu -- scenario generation and bank packing ON THE DEVICE (SURVEY.md §8 f2).
//
// gen_scenarios_kernel restates the reference's reset path in double precision, one thread per scenario:
//   game_map.gen_river_poly (ship_gym/game_map.py:22-73)  ->  pm.Poly's convex hull (models.py:180, cpConvexHull tol 0)
//   ->  ShipGame.gen_goal_path (game.py:300-330) with its two fat (r = 10) horizontal segment queries per goal.
// The reference draws from CPython's Mersenne Twister (random.gauss / random.randint) and numpy's (np.random.uniform);
// those streams cannot be reproduced on a GPU, so draws come from Philox4x32-10 keyed by (seed, scenario): the
// DISTRIBUTIONS are the reference's (tests compare against the host generator, which is pinned to the reference's
// fixtures), the individual maps are not.
// pack_bank_kernel then derives, from the fp32-rounded vertices, the scenario records (fp32 planes, double planes,
// header) of every bank, generated here or loaded from the host; the reach grid and spawn rows follow in
// shipsim_kernels.cu.  Everything is enqueued on the caller's stream: a bank can be regenerated between rollouts without
// a host round trip.
#include "shipsim_device.cuh"
#include "shipsim_launch.h"

namespace shipsim {

namespace {

struct Rng {
    unsigned long long seed, key;
    unsigned ctr;
    __device__ uint4 next() { return philox4x32_10(seed, key, ctr++, 7u); }
    __device__ double uniform()            // [0, 1) with 53 random bits
    {
        const uint4 r = next();
        return (double)((((unsigned long long)r.x << 32) | r.y) >> 11) * (1.0 / 9007199254740992.0);
    }
    __device__ double gauss(double mu, double sigma)   // random.gauss(mu, sigma): Box-Muller, one value per call
    {
        const uint4 r = next();
        const double u1 = ((double)((((unsigned long long)r.x << 32) | r.y) >> 11) + 1.0) * (1.0 / 9007199254740992.0);   // (0, 1]
        const double u2 = (double)((((unsigned long long)r.z << 32) | r.w) >> 11) * (1.0 / 9007199254740992.0);
        return mu + sigma * sqrt(-2.0 * log(u1)) * cos(6.283185307179586476925 * u2);
    }
    __device__ int randint(int lo, int hi)  // random.randint(lo, hi): inclusive
    {
        const uint4 r = next();
        return lo + (int)__umulhi(r.x, (unsigned)(hi - lo + 1));
    }
};

constexpr int kMaxPts = kMaxHull + 2;

// Andrew's monotone chain: CCW hull, collinear points dropped, first vertex = min x then min y (cpConvexHull, tol 0)
__device__ int convex_hull(double (*pts)[2], int n, double (*out)[2])
{
    for (int i = 1; i < n; ++i) {           // insertion sort by (x, y)
        const double px = pts[i][0], py = pts[i][1];
        int j = i - 1;
        while (j >= 0 && (pts[j][0] > px || (pts[j][0] == px && pts[j][1] > py))) { pts[j + 1][0] = pts[j][0]; pts[j + 1][1] = pts[j][1]; --j; }
        pts[j + 1][0] = px; pts[j + 1][1] = py;
    }
    int m = 0;
    for (int i = 0; i < n; ++i)             // drop exact duplicates
        if (m == 0 || pts[i][0] != pts[m - 1][0] || pts[i][1] != pts[m - 1][1]) { pts[m][0] = pts[i][0]; pts[m][1] = pts[i][1]; ++m; }
    n = m;
    if (n < 3) { for (int i = 0; i < n; ++i) { out[i][0] = pts[i][0]; out[i][1] = pts[i][1]; } return n; }
    double h[2 * kMaxPts][2];
    int k = 0;
    for (int i = 0; i < n; ++i) {
        while (k >= 2 && (h[k - 1][0] - h[k - 2][0]) * (pts[i][1] - h[k - 2][1]) - (h[k - 1][1] - h[k - 2][1]) * (pts[i][0] - h[k - 2][0]) <= 0.0) --k;
        h[k][0] = pts[i][0]; h[k][1] = pts[i][1]; ++k;
    }
    const int lower = k + 1;
    for (int i = n - 2; i >= 0; --i) {
        while (k >= lower && (h[k - 1][0] - h[k - 2][0]) * (pts[i][1] - h[k - 2][1]) - (h[k - 1][1] - h[k - 2][1]) * (pts[i][0] - h[k - 2][0]) <= 0.0) --k;
        h[k][0] = pts[i][0]; h[k][1] = pts[i][1]; ++k;
    }
    --k;
    for (int i = 0; i < k; ++i) { out[i][0] = h[i][0]; out[i][1] = h[i][1]; }
    return k;
}

// cpPolyShapePointQuery: signed distance, negative inside
__device__ double poly_point_distance(const double (*v)[2], int n, double px, double py)
{
    bool outside = false;
    double best = 1.0e300;
    for (int i = 0; i < n; ++i) {
        const int j = i == 0 ? n - 1 : i - 1;
        const double ax = v[j][0], ay = v[j][1], bx = v[i][0], by = v[i][1];
        const double ex = bx - ax, ey = by - ay, ln = sqrt(ex * ex + ey * ey);
        if ((ey / ln) * (px - bx) + (-ex / ln) * (py - by) > 0.0) outside = true;
        const double dx = ax - bx, dy = ay - by;
        double t = (dx * (px - bx) + dy * (py - by)) / (dx * dx + dy * dy);
        t = fmin(fmax(t, 0.0), 1.0);
        const double cx = bx + dx * t - px, cy = by + dy * t - py;
        best = fmin(best, sqrt(cx * cx + cy * cy));
    }
    return outside ? best : -best;
}

// x of cpShapeSegmentQuery(hull, a, b, r).point for a horizontal segment; returns false when the query misses
// (cpPolyShapeSegmentQuery incl. the bevelled vertices; game.py:322-323 uses r = 10)
__device__ bool fat_segment_hit_x(const double (*v)[2], int n, double ax, double ay, double bx, double by, double r, double &hit_x)
{
    if (poly_point_distance(v, n, ax, ay) <= r) { hit_x = bx; return true; }     // alpha = 0: `point` stays at the segment end
    bool hit = false;
    double alpha = 1.0;
    for (int i = 0; i < n; ++i) {
        const int j = i == 0 ? n - 1 : i - 1;
        const double ex = v[i][0] - v[j][0], ey = v[i][1] - v[j][1], ln = sqrt(ex * ex + ey * ey);
        const double nx = ey / ln, ny = -ex / ln;
        const double an = ax * nx + ay * ny;
        const double d = an - (v[i][0] * nx + v[i][1] * ny) - r;
        if (d < 0.0) continue;
        const double bn = bx * nx + by * ny;
        const double t = d / fmax(an - bn, 2.2250738585072014e-308);
        if (t < 0.0 || t > 1.0) continue;
        const double qx = ax + (bx - ax) * t, qy = ay + (by - ay) * t;
        const double along = nx * qy - ny * qx;
        if (nx * v[j][1] - ny * v[j][0] <= along && along <= nx * v[i][1] - ny * v[i][0]) { hit = true; hit_x = qx - nx * r; alpha = t; }
    }
    for (int i = 0; i < n; ++i) {           // bevelled vertices (CircleSegmentQuery)
        const double dax = ax - v[i][0], day = ay - v[i][1], dbx = bx - v[i][0], dby = by - v[i][1];
        const double daa = dax * dax + day * day, dab = dax * dbx + day * dby, dbb = dbx * dbx + dby * dby;
        const double qa = daa - 2.0 * dab + dbb, qb = dab - daa;
        const double det = qb * qb - qa * (daa - r * r);
        if (det >= 0.0 && qa != 0.0) {
            const double t = (-qb - sqrt(det)) / qa;
            if (0.0 <= t && t <= 1.0 && t < alpha) {
                const double mx = dax + (dbx - dax) * t, my = day + (dby - day) * t;
                const double ln = sqrt(mx * mx + my * my);
                hit = true; hit_x = ax + (bx - ax) * t - (mx / ln) * r; alpha = t;
            }
        }
    }
    return hit;
}

// space.segment_query(a, b, r, filter)[0].point.x over the static bank shapes in insertion order; the spatial index
// only offers shapes whose box the THIN segment crosses
__device__ bool first_bank_hit(const double (*h0)[2], int n0, const double (*h1)[2], int n1, double ax, double ay, double bx,
                               double r, double &hit_x)
{
    for (int b = 0; b < 2; ++b) {
        const double (*v)[2] = b ? h1 : h0;
        const int n = b ? n1 : n0;
        double l = 1e300, rt = -1e300, bo = 1e300, tp = -1e300;
        for (int i = 0; i < n; ++i) { l = fmin(l, v[i][0]); rt = fmax(rt, v[i][0]); bo = fmin(bo, v[i][1]); tp = fmax(tp, v[i][1]); }
        if (ay < bo || ay > tp || fmax(ax, bx) < l || fmin(ax, bx) > rt) continue;
        if (fat_segment_hit_x(v, n, ax, ay, bx, ay, r, hit_x)) return true;
    }
    return false;
}

}  // namespace

__global__ void __launch_bounds__(64) gen_scenarios_kernel(unsigned long long seed, int n_scen, double W, double H, int map_N,
                                                           double width_frac, double *hull_xy /*[S][2][kMaxHull][2]*/,
                                                           int *hull_n /*[S][2]*/, double *goals /*[S][5][2]*/)
{
    const int sidx = blockIdx.x * blockDim.x + threadIdx.x;
    if (sidx >= n_scen) return;
    Rng rng{seed, (unsigned long long)sidx, 0u};
    // ---- game_map.gen_river_poly (game_map.py:22-73)
    const double y_start = -100.0, y_delta = (H * 1.2 - y_start) / map_N, bank_width = width_frac * W / 2.0;
    double hull[2][kMaxPts][2];
    int hn[2];
    for (int b = 0; b < 2; ++b) {
        const double x_min = b ? W - bank_width : 0.0, x_max = b ? W : bank_width;
        const double centre = x_min + (x_max - x_min);           // the reference's `x_middle` evaluates to x_max (:48)
        double pts[kMaxPts][2];
        for (int i = 1; i <= map_N; ++i) {
            double x = 0.0, y = 0.0;
            for (int t = 0; t < 1000; ++t) {                     // redraw BOTH while x is outside [x_min, x_max] (:50-63)
                x = rng.gauss(centre, 50.0);
                y = y_start + rng.gauss(y_delta * i, 20.0);
                if (x_min <= x && x <= x_max) break;
            }
            pts[i - 1][0] = x; pts[i - 1][1] = y;
        }
        pts[map_N][0] = b ? W : 0.0; pts[map_N][1] = H;          // the two outer-wall corners (:68, :71)
        pts[map_N + 1][0] = b ? W : 0.0; pts[map_N + 1][1] = 0.0;
        hn[b] = convex_hull(pts, map_N + 2, hull[b]);            // pm.Poly convexifies (models.py:180)
    }
    // ---- ShipGame.gen_goal_path (game.py:300-330)
    const double gy_delta = H / (kGoals + 1);
    for (int i = 1; i <= kGoals; ++i) {
        const double y = gy_delta * i + (double)rng.randint(-20, 20);
        double left = 0.0, right = 0.0, x;
        const bool okl = first_bank_hit(hull[0], hn[0], hull[1], hn[1], W / 2.0, y, 0.0, 10.0, left);
        const bool okr = first_bank_hit(hull[0], hn[0], hull[1], hn[1], W / 2.0, y, W, 10.0, right);
        if (!okl || !okr) x = (W / 2.0) * i + (double)rng.randint(-50, 50);        // the `except` branch (:328-330)
        else { const double lo = left + 60.0, hi = right - 60.0; x = lo + (hi - lo) * rng.uniform(); }   // np.random.uniform(lo, hi)
        goals[((size_t)sidx * kGoals + (i - 1)) * 2 + 0] = x;
        goals[((size_t)sidx * kGoals + (i - 1)) * 2 + 1] = y;
    }
    for (int b = 0; b < 2; ++b) {
        hull_n[sidx * 2 + b] = hn[b];
        double *o = hull_xy + ((size_t)sidx * 2 + b) * kMaxHull * 2;
        for (int i = 0; i < kMaxHull; ++i) { o[2 * i] = i < hn[b] ? hull[b][i][0] : 0.0; o[2 * i + 1] = i < hn[b] ? hull[b][i][1] : 0.0; }
    }
}

// maximum hull size over all banks (the step kernel's edge stride and SAT lane layout depend on it)
__global__ void max_hull_kernel(const int *hull_n, int n, int *out)
{
    int m = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) m = max(m, hull_n[i]);
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// The only writer of the scenario records (the fp32 records and the EdgeD planes; layout in shipsim_device.cuh) of every
// bank, loaded or generated; one thread per scenario.  `stride4` / `maxv` are the layout of the fp32 bank, and hull_xy
// holds `maxv` vertices per hull.  hull_xy is rounded to fp32 IN PLACE so that the reach-grid build that follows sees the
// polygon the kernels represent.  The squared edge length is two rounded products and a rounded sum, never a DFMA: the
// planes are then those plain double arithmetic gives (the float64 oracle is compiled with -ffp-contract=off).
__global__ void __launch_bounds__(128) pack_bank_kernel(double *hull_xy, const int *hull_n, const double *goals, int n_scen,
                                                        int maxv, int stride4, float4 *bank, EdgeD *edges)
{
    const int sidx = blockIdx.x * blockDim.x + threadIdx.x;
    if (sidx >= n_scen) return;
    float4 *rec = bank + (size_t)sidx * stride4;
    for (int b = 0; b < 2; ++b) {
        double *v = hull_xy + ((size_t)sidx * 2 + b) * maxv * 2;
        const int n = hull_n[sidx * 2 + b];
        double l = 1e300, bo = 1e300, r = -1e300, t = -1e300;
        for (int i = 0; i < n; ++i) {           // (not fmin / fmax: a tie such as -0 against +0 keeps the earlier vertex)
            const double x = (double)(float)v[2 * i], y = (double)(float)v[2 * i + 1];
            v[2 * i] = x; v[2 * i + 1] = y;
            l = x < l ? x : l; r = r < x ? x : r; bo = y < bo ? y : bo; t = t < y ? y : t;
        }
        rec[b] = make_float4(__double2float_rd(l), __double2float_rd(bo), __double2float_ru(r), __double2float_ru(t));
        float4 *E = rec + kBankHeader4 + b * maxv;
        EdgeD *ED = edges + ((size_t)sidx * 2 + b) * kMaxHull;
        for (int i = 0; i < n; ++i) {
            const int j = i == 0 ? n - 1 : i - 1;
            const double ex = v[2 * i] - v[2 * j], ey = v[2 * i + 1] - v[2 * j + 1];
            const double ln = sqrt(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)));
            E[i] = make_float4((float)(ey / ln), (float)(-ex / ln), (float)v[2 * i], (float)v[2 * i + 1]);
            EdgeD e;
            e.set_normal(ey / ln, -ex / ln); e.vx = (float)v[2 * i]; e.vy = (float)v[2 * i + 1]; e.len = (float)ln;
            e.pad = __int_as_float(b * kMaxHull + i);
            ED[i] = e;
        }
    }
    const double *g = goals + (size_t)sidx * 10;
    rec[2] = make_float4((float)g[0], (float)g[1], (float)g[2], (float)g[3]);
    rec[3] = make_float4((float)g[4], (float)g[5], (float)g[6], (float)g[7]);
    rec[4] = make_float4((float)g[8], (float)g[9], __int_as_float(hull_n[sidx * 2]), __int_as_float(hull_n[sidx * 2 + 1]));
}

cudaError_t launch_max_hull(const int *hull_n, int n, int *out, cudaStream_t stream)
{
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(int), stream);
    if (e != cudaSuccess) return e;
    max_hull_kernel<<<1, 256, 0, stream>>>(hull_n, n, out);
    return cudaGetLastError();
}

cudaError_t launch_gen_scenarios(unsigned long long seed, int n_scen, double W, double H, int map_N, double width_frac, double *hull_xy,
                                 int *hull_n, double *goals, cudaStream_t stream)
{
    gen_scenarios_kernel<<<(n_scen + 63) / 64, 64, 0, stream>>>(seed, n_scen, W, H, map_N, width_frac, hull_xy, hull_n, goals);
    return cudaGetLastError();
}

cudaError_t launch_pack_bank(double *hull_xy, const int *hull_n, const double *goals, int n_scen, int maxv, int stride4, float4 *bank,
                             EdgeD *edges, cudaStream_t stream)
{
    pack_bank_kernel<<<(n_scen + 127) / 128, 128, 0, stream>>>(hull_xy, hull_n, goals, n_scen, maxv, stride4, bank, edges);
    return cudaGetLastError();
}

}  // namespace shipsim
