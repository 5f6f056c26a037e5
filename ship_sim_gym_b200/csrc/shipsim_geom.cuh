// shipsim_geom.cuh -- pieces shared by the step kernels (serial-in-time step_kernel and the time-parallel
// window_kernel): action fetch, hull AABB, reach-grid lookup, two-float plane evaluation, ray-vs-plane test, the plane
// phase with its candidate staging, the ray query against a plane row (cooperative and serial), and the stores of a
// frame, of the state and of the statistics.  The lidar and plane work of both kernels runs through these functions on
// the same inputs.  What each kernel still spells out itself -- the integration, the goal tests, reward / done and the
// separating-axis passes (whose lane layouts differ) -- performs the same operations in the same order.  Together that
// makes their results bit-identical (tests/test_gpu_window.py).
#pragma once
#include "shipsim_device.cuh"

namespace shipsim {

// Action words are read once, never again by this SM: streaming loads (__ldcs), so that they do not displace the
// reach-grid and plane records in L1.
// actions[k][e]: `ap` walks down this env's column (stride = one row of the action tensor, in bytes)
__device__ __forceinline__ int load_action(const StepParams &p, const char *ap, int k, long long gid)
{
    switch (p.action_dtype) {
        case 0: return __ldcs(reinterpret_cast<const int *>(ap));
        case 1: return (int)__ldcs(reinterpret_cast<const long long *>(ap));
        case 2: return (int)__ldcs(reinterpret_cast<const unsigned char *>(ap));
        default: return random_action(p, gid, p.step0 + (unsigned)k);
    }
}

// actions[k][e] by row index: the base pointer stays in the constant bank (no per-lane pointer to keep or spill)
__device__ __forceinline__ int load_action_at(const StepParams &p, size_t idx, int k, long long gid)
{
    switch (p.action_dtype) {
        case 0: return __ldcs(reinterpret_cast<const int *>(p.actions) + idx);
        case 1: return (int)__ldcs(reinterpret_cast<const long long *>(p.actions) + idx);
        case 2: return (int)__ldcs(reinterpret_cast<const unsigned char *>(p.actions) + idx);
        default: return random_action(p, gid, p.step0 + (unsigned)k);
    }
}

// One bank-normal axis of the separating-axis test: does plane `ed` of the bank have the whole ship (rotated hull
// rx/ry about the body origin bx/by) strictly in front of it?
__device__ __forceinline__ bool bank_axis_separates(const float4 ed, const float (&rx)[kShipVerts], const float (&ry)[kShipVerts],
                                                    float bx, float by)
{
    float m = fmaf(ed.x, rx[0], __fmul_rn(ed.y, ry[0]));
#pragma unroll
    for (int j = 1; j < kShipVerts; ++j) m = fminf(m, fmaf(ed.x, rx[j], __fmul_rn(ed.y, ry[j])));
    const float base = fmaf(ed.x, bx - ed.z, __fmul_rn(ed.y, by - ed.w));
    return base + m > 0.f;
}

// half extents of the rotated hull's AABB (cpPolyShapeCacheData): the lidar origin is the body origin plus these
// (models.py:51-53).  Hull vertex 0 is the body origin.
__device__ __forceinline__ void hull_half_extents(const StepParams &p, float c, float s, float &hx, float &hy)
{
    float minx = 0.f, maxx = 0.f, miny = 0.f, maxy = 0.f;
#pragma unroll
    for (int j = 1; j < kShipVerts; ++j) {
        const float wx = fmaf(p.ship_lx[j], c, -__fmul_rn(p.ship_ly[j], s));
        const float wy = fmaf(p.ship_lx[j], s, __fmul_rn(p.ship_ly[j], c));
        minx = fminf(minx, wx); maxx = fmaxf(maxx, wx); miny = fminf(miny, wy); maxy = fmaxf(maxy, wy);
    }
    hx = __fmul_rn(0.5f, __fadd_rn(maxx, -minx));
    hy = __fmul_rn(0.5f, __fadd_rn(maxy, -miny));
}

// Reach-grid cell of the lidar origin (ox, oy): which bank edges a ray starting there can touch at all.
__device__ __forceinline__ uint4 load_cell(const StepParams &p, int scen, float ox, float oy)
{
    int ix = __float2int_rd((ox - p.gridp.x0) * p.gridp.inv_cx);
    int iy = __float2int_rd((oy - p.gridp.y0) * p.gridp.inv_cy);
    ix = min(max(ix, 0), kGridN - 1);
    iy = min(max(iy, 0), kGridN - 1);
    return __ldg(p.grid + ((size_t)scen * kGridN + iy) * kGridN + ix);
}

// The same lookup as an asynchronous copy into shared memory (LDGSTS): no destination register, so the 16-byte cell does
// not sit in four registers from the moment its pose is known until the next step looks at it, and no register
// scoreboard is tied up by an L2 round trip (ncu: with a plain load, an unrelated instruction of the copy-out that
// happened to share the load's scoreboard slot waited out the whole round trip: 7.7 % of the stall samples).
__device__ __forceinline__ void fetch_cell_async(const StepParams &p, int scen, float ox, float oy, unsigned smem_dst)
{
    int ix = __float2int_rd((ox - p.gridp.x0) * p.gridp.inv_cx);
    int iy = __float2int_rd((oy - p.gridp.y0) * p.gridp.inv_cy);
    ix = min(max(ix, 0), kGridN - 1);
    iy = min(max(iy, 0), kGridN - 1);
    cp_async16_s(smem_dst, p.grid + ((size_t)scen * kGridN + iy) * kGridN + ix);
}

// A candidate plane seen from the ray origin (ox, oy) = (x + hx, y + hy): d = n.(o - v_i), ta = cross(n, o - v_i), with
// the two-float normal of the record.  The difference o - v_i is formed in fp32 from fp32 inputs (exact when the two are
// within a factor of two of each other, otherwise good to 1e-5 at map scale -- below what the fp32 pose itself carries).
struct PlaneEval { float d, ta, nx, ny, len; };

__device__ __forceinline__ PlaneEval eval_plane_rec(const float4 nn, const float4 ev, float x, float y, float hx, float hy)
{
    const float qx = __fadd_rn(__fadd_rn(x, -ev.x), hx), qy = __fadd_rn(__fadd_rn(y, -ev.y), hy);     // origin - v_i
    PlaneEval o;
    o.d = __fadd_rn(fmaf(nn.x, qx, __fmul_rn(nn.y, qy)), fmaf(nn.z, qx, __fmul_rn(nn.w, qy)));
    o.ta = __fadd_rn(fmaf(nn.x, qy, -__fmul_rn(nn.y, qx)), fmaf(nn.z, qy, -__fmul_rn(nn.w, qx)));
    o.nx = nn.x;
    o.ny = nn.y;
    o.len = ev.z;
    return o;
}

__device__ __forceinline__ PlaneEval eval_plane(const EdgeD *E, float x, float y, float hx, float hy)
{
    return eval_plane_rec(__ldg(reinterpret_cast<const float4 *>(E)), __ldg(reinterpret_cast<const float4 *>(E) + 1), x, y, hx, hy);
}

__device__ __forceinline__ float rcp_approx(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// One ray (direction dir, length L) against one candidate plane: cpPolyShapeSegmentQuery's loop body.  nxl / nyl =
// -L * n.  The reference computes t = d / max(an - bn, DBL_MIN) and rejects t outside [0, 1]: with d >= 0 that is
// an - bn > 0 and d <= an - bn (d == 0 with the ray leaving the plane can only yield the origin itself, which the
// edge-extent test or the inside test has already decided).  `val` = |hit - origin|.
__device__ __forceinline__ bool ray_vs_plane(float d, float ta, float nxl, float nyl, float len, float dirx, float diry, float L, float &val)
{
    // (every product / sum spelled out: which operand pairs the compiler fuses would otherwise differ between the two
    // kernels that inline this, and their results are compared bit for bit)
    const float denom = fmaf(nxl, dirx, __fmul_rn(nyl, diry));            // an - bn
    const float cr = fmaf(nxl, diry, -__fmul_rn(nyl, dirx));              // -L * cross(n, dir)
    const float t = __fmul_rn(d, rcp_approx(denom));
    const float tang = fmaf(-t, cr, ta);                                  // cross(n, hit - v_i)
    val = __fmul_rn(t, L);
    return d >= 0.f && denom > 0.f && d <= denom && tang >= -len && tang <= 0.f;
}

// direction of ray (rc, rs) = (cos, sin of its body-frame angle) for a hull heading (c, s)
__device__ __forceinline__ void ray_dir(float c, float s, float rc, float rs, float &dirx, float &diry)
{
    dirx = fmaf(c, rc, -__fmul_rn(s, rs));
    diry = fmaf(s, rc, __fmul_rn(c, rs));
}

constexpr int kMaxCand = 4;                  // candidate planes a scratch row holds (more -> serial ray query)
constexpr int kScr4 = 1 + 2 * kMaxCand;      // scratch row: header + two float4 per plane (odd stride: conflict-free)
constexpr int kRowPlane0 = 1;                // row index of the first plane
// header.z bits
constexpr int kHdrIn0 = 1 << 8, kHdrIn1 = 1 << 9, kHdrBig = 1 << 10;

// One candidate plane at one pose (x, y, c, s; hx, hy = half extents of the hull's AABB): what the lidar of the next step
// and the ship-vs-bank pre-test of this step need from it.
struct PlaneOut { float d, ta, nxl, nyl, len; bool out, sep, keep; };

template <bool WITH_SAT>
__device__ __forceinline__ PlaneOut plane_at_pose(const StepParams &p, const float4 nn, const float4 ev, float x, float y, float hx,
                                                  float hy, float c, float s)
{
    const float L = p.lidar_len;
    const PlaneEval pe = eval_plane_rec(nn, ev, x, y, hx, hy);
    PlaneOut o;
    o.d = pe.d; o.ta = pe.ta; o.nxl = __fmul_rn(-L, pe.nx); o.nyl = __fmul_rn(-L, pe.ny); o.len = pe.len;
    o.out = pe.d > 0.f;
    // the normal in the body frame, where both the hull and the ray fan are constant
    const float bnx = fmaf(pe.nx, c, __fmul_rn(pe.ny, s)), bny = fmaf(pe.ny, c, -__fmul_rn(pe.nx, s));
    o.sep = false;
    if (WITH_SAT) {
        // does this bank plane have the whole ship in front of it?  n.(hull vertex j - v_i) = d - n.h + (R^T n).l_j
        // (vertex 0 is the body origin)
        float m = 0.f;
#pragma unroll
        for (int j = 1; j < kShipVerts; ++j) m = fminf(m, fmaf(bnx, p.ship_lx[j], __fmul_rn(bny, p.ship_ly[j])));
        o.sep = __fadd_rn(__fadd_rn(pe.d, -fmaf(pe.nx, hx, __fmul_rn(pe.ny, hy))), m) > 0.f;
    }
    // Can any ray of the fan reach this plane at all?  A ray hits only if 0 <= d <= -L n.dir (ray_vs_plane), and over
    // the fan -n.dir <= cos(max(0, angle(-n, fan axis) - half spread)).  Planes that fail (with a margin far above
    // fp32 rounding) are left out of the row: fewer planes per ray, and often no ray pass for the env at all.
    const float cm = -fmaf(bnx, p.fan_cx, __fmul_rn(bny, p.fan_cy));
    float reach = 1.f;
    if (cm < p.fan_cos)                                                                   // a bound: approx is plenty
        reach = fmaf(cm, p.fan_cos, __fmul_rn(sqrt_approx(fmaxf(fmaf(-cm, cm, 1.f), 0.f)), p.fan_sin));
    o.keep = pe.d >= 0.f && pe.d <= fmaf(__fmul_rn(L, reach), 1.0001f, 1.0e-3f);
    return o;
}

// Where a row of float4 (a plane row, a frame, the statistics accumulators) lives.  step_kernel names its shared memory
// by 32-bit shared address (RowSmem; see "shared memory by address" in shipsim_device.cuh); window_kernel by generic
// pointers into its shared arrays, and the scenario-upload and frame kernels write rows to global memory (RowPtr).  The
// pieces below are written once against either and compile to each kernel's own addressing.
struct RowPtr {
    float4 *p;
    __device__ __forceinline__ void st(int i, float4 v) const { p[i] = v; }
    __device__ __forceinline__ float4 ld(int i) const { return p[i]; }
    __device__ __forceinline__ float2 ld2(int i) const { return *reinterpret_cast<const float2 *>(p + i); }
    __device__ __forceinline__ float ldf(int j) const { return reinterpret_cast<const float *>(p)[j]; }   // float j
    __device__ __forceinline__ void cp_async(int i, const float4 *src) const { cp_async16(p + i, src); }
};
struct RowSmem {
    unsigned a;
    __device__ __forceinline__ void st(int i, float4 v) const { sts4(a + 16u * (unsigned)i, v); }
    __device__ __forceinline__ float4 ld(int i) const { return lds4(a + 16u * (unsigned)i); }
    __device__ __forceinline__ float2 ld2(int i) const { return lds2(a + 16u * (unsigned)i); }
    __device__ __forceinline__ float ldf(int j) const { return lds1(a + 4u * (unsigned)j); }
    __device__ __forceinline__ void cp_async(int i, const float4 *src) const { cp_async16_s(a + 16u * (unsigned)i, src); }
};

// The observation frame of a state (ShipEnv.__add_states, ship_env.py:79-113): pose, rudder, nearest goal (gx, gy) and
// lidar[0..9] as the state planes hold them (l0, l1, l2.xy).
template <class ROW>
__device__ __forceinline__ void store_frame(const ROW f, const EnvRegs &r, float gx, float gy, float4 l0, float4 l1, float4 l2)
{
    f.st(0, make_float4(r.x, r.y, (float)r.rudder, r.th));
    f.st(1, make_float4(gx, gy, l0.x, l0.y));
    f.st(2, make_float4(l0.z, l0.w, l1.x, l1.y));
    f.st(3, make_float4(l1.z, l1.w, l2.x, l2.y));
}

// The env's state planes from r and the lidar readings of frame f (the newest: it holds the sticky readings).
template <class ROW>
__device__ __forceinline__ void store_env_frame(const StepParams &p, int e, const EnvRegs &r, const ROW f)
{
    const float4 l1 = f.ld(1), l2 = f.ld(2), l3 = f.ld(3);
    store_env(p, e, r, make_float4(l1.z, l1.w, l2.x, l2.y), make_float4(l2.z, l2.w, l3.x, l3.y), l3.z, l3.w);
}

// The warp's eight statistics accumulators (warp_stats) -> the slot row of this CTA: one red.add per non-zero value.
template <class ROW>
__device__ __forceinline__ void flush_stats(const StepParams &p, int lane, const ROW stat)
{
    __syncwarp();
    if (p.stats && lane < 8) {
        const float v = stat.ldf(lane);
        if (v != 0.f) atomicAdd(p.stats + (size_t)(blockIdx.x % kStatSlots) * kStatLen + lane, (double)v);
    }
}

// Copies the raw records of a staged cell's candidate planes (cell.w: up to kMaxCand record indices, 0xff = none) into
// raw[2i], raw[2i+1] (cp.async: they land while the caller does other work; plane_phase<..., STAGED> reads them).
template <class ROW>
__device__ __forceinline__ void stage_candidates(const StepParams &p, int scen, const uint4 cell, const ROW raw)
{
    const float4 *E4 = reinterpret_cast<const float4 *>(p.edges_d + (size_t)scen * (2 * kMaxHull));
#pragma unroll
    for (int n = 0; n < kMaxCand; ++n) {
        const unsigned idx = (cell.w >> (8 * n)) & 0xffu;
        if (idx != 0xffu) {
            raw.cp_async(2 * n, E4 + 2 * idx);
            raw.cp_async(2 * n + 1, E4 + 2 * idx + 1);
        }
    }
}

// One ray of the fan (body-frame direction rc, rs) against an env's plane row: cpPolyShapeSegmentQuery over the row's
// planes, later accepted planes overwriting earlier ones; an origin inside a bank reads L (alpha = 0, `point` stays at
// the ray end).  LiDAR.query: the first bank (list order) that reports a hit wins.  Returns the reading, < 0 for none.
template <class ROW>
__device__ __forceinline__ float ray_vs_row(const ROW row, float rc, float rs, float L)
{
    const float4 hdr = row.ld(0);
    float dirx, diry;
    ray_dir(hdr.x, hdr.y, rc, rs, dirx, diry);
    const int hz = __float_as_int(hdr.z);
    const int n = hz & 0xff;
    float v0 = -1.f, v1 = -1.f;                     // hit distance per bank (< 0: none)
#pragma unroll 1
    for (int i = 0; i < n; ++i) {
        const float4 e0 = row.ld(kRowPlane0 + 2 * i);
        const float2 e1 = row.ld2(kRowPlane0 + 1 + 2 * i);
        float val;
        const bool ok = ray_vs_plane(e0.x, e0.y, e0.z, e0.w, e1.x, dirx, diry, L, val);
        if (ok && e1.y == 0.f) v0 = val;
        if (ok && e1.y != 0.f) v1 = val;
    }
    if (hz & kHdrIn0) v0 = L;
    if (hz & kHdrIn1) v1 = L;
    return v0 >= 0.f ? v0 : v1;
}

// Plane phase for one env at pose (x, y, c, s): fills the env's scratch row for the next lidar query and returns,
// when WITH_SAT, bit b set <=> bank b is near and none of its candidate planes has the whole ship in front of it
// (=> the full separating-axis pass has to decide).  Scratch row:
//   [0]      c, s, bits(n | in0<<8 | in1<<9 | big<<10), 0
//   [1+2i]   d, ta, -L*nx, -L*ny        [2+2i]  len, bank (0.f / 1.f), 0, 0
//   big row (more than kMaxCand planes would have to be kept; rays are then cast serially by the owner lane):
//   [1]      x, y, hx, hy               [2]     bits(scen), bits(m0), bits(m1), bits(flags)
// STAGED: the raw record of candidate i has already been copied (cp.async) into raw[2i], raw[2i+1]; the record carries
// its own index (bank * kMaxHull + edge) in `pad`, so the candidate masks need not be walked again (only cells with at
// most kMaxCand candidates are staged).
// A cell may name more than kMaxCand candidates (long banks of short edges: the hard map): all of them are evaluated
// -- the separating-plane pre-test and the inside test want every one -- and since the fan-reach cull drops about half,
// the row usually still holds what the rays can reach.  Only when a (kMaxCand+1)-th plane would have to be kept does
// the env fall back to the big row.
// (Round 2 also tried this phase warp-cooperatively -- the (env, candidate) pairs of a whole warp laid out by a prefix
// sum and evaluated one per lane: 7-12 % fewer instructions, but longer dependent chains and more live registers; it
// measured 1 % faster at 1M envs and 4 % slower on the two latency-bound shapes.  profiles/r02_b_coop_plane_phase.md.)
template <bool WITH_SAT, bool STAGED, class ROW>
__device__ __forceinline__ unsigned plane_phase(const StepParams &p, float x, float y, float hx, float hy, float c, float s, int scen,
                                                const uint4 cell, const ROW row, const ROW raw)
{
    unsigned m0 = cell.x, m1 = cell.y;
    const unsigned near = ((m0 != 0u || (cell.z & 1u)) ? 1u : 0u) | ((m1 != 0u || (cell.z & 2u)) ? 2u : 0u);
    const int ncand = (int)((cell.z >> 8) & 0xffu);
    const EdgeD *E = p.edges_d + (size_t)scen * (2 * kMaxHull);
    unsigned outm = 0u, sepm = 0u;
    int nk = 0;                                  // planes kept for the ray pass
    float4 nn_next = make_float4(0.f, 0.f, 0.f, 0.f), ev_next = nn_next;
    if (!STAGED && ncand > 0) {
        int idx;
        if (m0) { idx = __ffs(m0) - 1; m0 &= m0 - 1u; } else { idx = kMaxHull + __ffs(m1) - 1; m1 &= m1 - 1u; }
        nn_next = __ldg(reinterpret_cast<const float4 *>(E + idx));
        ev_next = __ldg(reinterpret_cast<const float4 *>(E + idx) + 1);
    }
#pragma unroll 1
    for (int n = 0; n < ncand; ++n) {
        float4 nn, ev;
        if (STAGED) {
            nn = raw.ld(2 * n);
            ev = raw.ld(2 * n + 1);
        } else {                                 // the next record is asked for before this one is evaluated
            nn = nn_next; ev = ev_next;
            if (n + 1 < ncand) {
                int idx;
                if (m0) { idx = __ffs(m0) - 1; m0 &= m0 - 1u; } else { idx = kMaxHull + __ffs(m1) - 1; m1 &= m1 - 1u; }
                nn_next = __ldg(reinterpret_cast<const float4 *>(E + idx));
                ev_next = __ldg(reinterpret_cast<const float4 *>(E + idx) + 1);
            }
        }
        const bool bank1 = __float_as_int(ev.w) >= kMaxHull;
        const unsigned bbit = bank1 ? 2u : 1u;
        const PlaneOut o = plane_at_pose<WITH_SAT>(p, nn, ev, x, y, hx, hy, c, s);
        if (o.out) outm |= bbit;
        if (o.sep) sepm |= bbit;
        if (o.keep) {
            if (!STAGED && nk == kMaxCand) {     // the row is full: big row (the masks are the cell's, not the walked ones)
                row.st(0, make_float4(c, s, __int_as_float(kHdrBig), 0.f));
                row.st(1, make_float4(x, y, hx, hy));
                row.st(2, make_float4(__int_as_float(scen), __uint_as_float(cell.x), __uint_as_float(cell.y), __uint_as_float(cell.z)));
                return near & ~sepm;            // what has been proven separated stays proven
            }
            row.st(kRowPlane0 + 2 * nk, make_float4(o.d, o.ta, o.nxl, o.nyl));
            row.st(kRowPlane0 + 1 + 2 * nk, make_float4(o.len, bank1 ? 1.f : 0.f, 0.f, 0.f));
            ++nk;
        }
    }
    // cpShapeSegmentQuery: start point inside the shape => alpha = 0 and `point` stays at the ray end
    const unsigned inm = cell.z & 3u & ~outm;
    row.st(0, make_float4(c, s, __int_as_float(nk | (int)(inm << 8)), 0.f));
    return near & ~sepm;
}

// The plane phase for cells that name more candidates than are staged, out of line: it walks the candidate masks and
// reads the records from global memory.  (Inlined into the window kernel it cost registers the hot path needs.)
static __device__ __noinline__ unsigned plane_phase_unstaged(const StepParams &p, float x, float y, float hx, float hy, float c, float s,
                                                             int scen, const uint4 cell, float4 *row)
{
    return plane_phase<true, false>(p, x, y, hx, hy, c, s, scen, cell, RowPtr{row}, RowPtr{nullptr});
}

// Serial LiDAR.query of one env by one lane: only for rows that more than kMaxCand planes would have to be kept in.
static __device__ __noinline__ void ray_query_serial(const StepParams &p, const float4 *row, float *lid)
{
    const float L = p.lidar_len;
    const float4 h = row[0], a = row[1], b4 = row[2];
    const float c = h.x, s = h.y;
    const int scen = __float_as_int(b4.x);
    const unsigned masks[2] = {__float_as_uint(b4.y), __float_as_uint(b4.z)};
    const unsigned flags = __float_as_uint(b4.w);
    const EdgeD *E = p.edges_d + (size_t)scen * (2 * kMaxHull);
    unsigned pend = (1u << kBeams) - 1u;
    for (int b = 0; b < 2; ++b) {
        bool out = false;
        unsigned hitm = 0u;
        float v[kBeams];
        for (unsigned m = masks[b]; m; m &= m - 1u) {
            const PlaneEval pe = eval_plane(E + b * kMaxHull + (__ffs(m) - 1), a.x, a.y, a.z, a.w);
            out = out || (pe.d > 0.f);
#pragma unroll
            for (int j = 0; j < kBeams; ++j) {
                float dirx, diry;
                ray_dir(c, s, p.ray_c[j], p.ray_s[j], dirx, diry);
                float val;
                if (ray_vs_plane(pe.d, pe.ta, __fmul_rn(-L, pe.nx), __fmul_rn(-L, pe.ny), pe.len, dirx, diry, L, val)) { v[j] = val; hitm |= 1u << j; }
            }
        }
        const bool inside = ((flags >> b) & 1u) && !out;
#pragma unroll
        for (int j = 0; j < kBeams; ++j)
            if ((pend >> j) & 1u) {
                if (inside) lid[j] = L;
                else if ((hitm >> j) & 1u) lid[j] = v[j];
            }
        pend &= inside ? 0u : ~hitm;
    }
}

// The same query for a fan of p.n_beams rays (the wide step kernel), ray by ray: the planes are evaluated again for
// every ray (the same arithmetic on the same inputs, so every ray sees exactly the values the loop above would), which
// keeps no per-ray array -- 32 of them would live in local memory.  Per ray: the first bank (list order) that is hit or
// holds the origin decides; within a bank the last accepted plane wins.
static __device__ __noinline__ void ray_query_serial_wide(const StepParams &p, const float4 *row, float *lid)
{
    const float L = p.lidar_len;
    const float4 h = row[0], a = row[1], b4 = row[2];
    const float c = h.x, s = h.y;
    const int scen = __float_as_int(b4.x);
    const unsigned masks[2] = {__float_as_uint(b4.y), __float_as_uint(b4.z)};
    const unsigned flags = __float_as_uint(b4.w);
    const EdgeD *E = p.edges_d + (size_t)scen * (2 * kMaxHull);
    for (int j = 0; j < p.n_beams; ++j) {
        float dirx, diry;
        ray_dir(c, s, p.ray_cw[j], p.ray_sw[j], dirx, diry);
        for (int b = 0; b < 2; ++b) {
            bool out = false, hit = false;
            float v = 0.f;
            for (unsigned m = masks[b]; m; m &= m - 1u) {
                const PlaneEval pe = eval_plane(E + b * kMaxHull + (__ffs(m) - 1), a.x, a.y, a.z, a.w);
                out = out || (pe.d > 0.f);
                float val;
                if (ray_vs_plane(pe.d, pe.ta, __fmul_rn(-L, pe.nx), __fmul_rn(-L, pe.ny), pe.len, dirx, diry, L, val)) { v = val; hit = true; }
            }
            if (((flags >> b) & 1u) && !out) { lid[j] = L; break; }
            if (hit) { lid[j] = v; break; }
        }
    }
}

}  // namespace shipsim
