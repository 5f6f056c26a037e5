// shipsim_device.cuh -- device-side data layout and per-env transition pieces for the fused step kernel.
//
// New code, written for sm_100a.  It implements the transition spec of SURVEY.md Appendix A, which restates
// ShipEnv.step (ship_gym/ship_env.py:136-156) and everything it reaches (game.py:140-153,185-195,232-257,
// 333-349; models.py:39-76,129-146) plus the Chipmunk2D routines the reference delegates to.  fp32 state,
// hull planes rebuilt in double where conditioning demands it.
//
// Execution model: G lanes cooperate on one env (G = 1, 2, 4, 8, 16 or 32; 32/G envs per warp).  The lanes of a
// group hold IDENTICAL copies of the env's scalar state, so the cheap serial parts (integrator, reward, done) are
// computed redundantly with no communication, regular loops (bank edges) are strided over the group, and the
// irregular heavy parts (ray-vs-live-edge tests, separating-axis tests) are executed by the WHOLE WARP for one
// needy env at a time (loop over a ballot), which keeps control flow warp-uniform: the first thread-per-env
// kernel ran with 7-9 of 32 lanes active (ncu, profiles/r01_v1_*.txt) because every lane took its own path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <cstdio>

namespace shipsim {

constexpr int kGoals = 5;
constexpr int kBeams = 10;         // the reference's fan: the tuned kernels' compile-time beam count
constexpr int kMaxBeams = 32;      // widest fan (one warp lane per ray)
constexpr int kFrame = 16;
constexpr int kPlanes = 8;
constexpr int kShipVerts = 5;
constexpr int kStatSlots = 128;     // replicated accumulator rows (one 128-byte line each) to spread atomics
constexpr int kStatLen = 16;
constexpr int kBankHeader4 = 6;     // float4s before the edge records of a scenario
constexpr int kMaxHull = 32;        // SHIPSIM_MAX_HULL: fixed stride of the double-plane records
constexpr int kGridN = 32;          // the reach grid has kGridN x kGridN cells per scenario
constexpr unsigned kFull = 0xffffffffu;

// Plane of one bank edge as the lidar and the plane phase see it (32 bytes = two 16-byte loads).  A lidar reading is
// d / (-n.dir): an error of d is amplified by 1/cos(incidence), and an fp32 normal (6e-8 rad) swings d by 6e-5 over a
// 1000-unit edge, so the unit normal is kept to 48 bits as an unevaluated sum of two floats (hi + lo, "double-float"):
// n.q then costs two fp32 FMAs per term instead of a trip through the FP64 pipe and six conversions.  (Round 1 stored the
// normal as doubles; the double evaluation held ~24 registers at its peak, which is what made the warp-cooperative
// plane phase spill at 96 registers -- and spills are ruinous in a kernel whose L1 is almost all shared memory.)
// Built from the SAME fp32-rounded vertices the fp32 records carry.
struct EdgeD {
    float nxh, nyh;                 // outward unit normal of the edge v_{i-1} -> v_i, leading parts
    float nxl, nyl;                 // ... and what is left of the double value: n = (nxh + nxl, nyh + nyl)
    float vx, vy;                   // v_i
    float len;                      // |v_i - v_{i-1}|
    float pad;                      // bits: the record's own index, bank * kMaxHull + i

    __host__ __device__ void set_normal(double nx, double ny)
    {
        nxh = (float)nx; nxl = (float)(nx - (double)nxh);
        nyh = (float)ny; nyl = (float)(ny - (double)nyh);
    }
};

// Reach grid: one uint4 per cell.  x / y: bit i set <=> edge i of bank 0 / 1 comes within max(lidar length, cell
// diagonal) (+ margin) of the cell, i.e. the superset of edges a ray starting anywhere in the cell can touch;
// z: bit b set <=> the cell may intersect the interior of bank b (then "origin inside the bank" <=> no candidate
// plane has the origin in front of it; clear => the origin is certainly outside); w: reserved.
// Border cells are unbounded (they stand for everything beyond the grid).
struct GridParams {
    float x0, y0;                   // lower-left corner of cell (0,0)
    float inv_cx, inv_cy;           // 1 / cell size
};

// Scenario record (float4 units): [0] aabb bank0 (l,b,r,t)  [1] aabb bank1  [2] goal0.xy goal1.xy
// [3] goal2.xy goal3.xy  [4] goal4.xy, bits(n0), bits(n1)  [5] reserved; then per bank b, edge i < n_b:
// [6 + b*maxv + i] = nx, ny, v_i.x, v_i.y
// Plane i is the edge v_{i-1} -> v_i with outward unit normal n (Chipmunk's cpSplittingPlane {v0 = v_i, n}).
// All plane tests are evaluated RELATIVE to the vertex (n.(p - v_i)), never as n.p - n.v_i: world coordinates
// are O(1000) and fp32 would lose ~1e-4 to cancellation; differences of nearby points are (nearly) exact.

struct StepParams {
    float4 *state;               // [kPlanes][N]
    const float4 *bank;          // packed scenario records
    const EdgeD *edges_d;        // [n_scen][2][kMaxHull] two-float planes
    const uint4 *grid;           // [n_scen][kGridN*kGridN] reach grid
    const float4 *spawn_rows;    // [n_scen][1 + 2*kMaxCand] plane-phase output at the spawn pose
    GridParams gridp;
    const void *actions;         // [K][N]
    float4 *obs;                 // [K][N][4*history]
    float *reward;               // [K][N]
    uint8_t *done;               // [K][N]
    double *stats;               // [kStatSlots][kStatLen]
    unsigned long long seed;
    long long env_id_offset;
    int N, K;
    int action_dtype, history, auto_reset, max_steps;
    int n_scen, maxv, scen_stride4;   // maxv = edge stride of the fp32 records
    int hull_max;                     // largest hull in the bank (SAT pass lane layout)
    int pick_base, pick_count;        // fresh-maps mode (pick_count > 0, a power of two): resets pick from this slice of the bank
    unsigned step0;              // global step counter at launch (random-action stream)
    float W, H, dt, damping;
    float lidar_len;
    float acc_dt;                // thrust/mass*dt        (cpBodyUpdateVelocity: v += f*m_inv*dt)
    float ang_dt;                // thrust/moment*dt      (w += t*i_inv*dt, t = -rudder*thrust)
    float goal_r, step_penalty, spawn_x, spawn_y;
    float ray_c[kBeams], ray_s[kBeams];              // cos/sin of radians(90 - spread/2 + i*spread/n) (models.py:48-49,62)
    float fan_cx, fan_cy, fan_cos, fan_sin;          // body-frame axis of the ray fan, cos/sin of its half opening
    float ship_lx[kShipVerts], ship_ly[kShipVerts];  // body-frame hull, CCW (models.py:6,88 through cpConvexHull)
    float ship_nx[kShipVerts], ship_ny[kShipVerts];  // body-frame outward normal of edge j-1 -> j
    float ship_off[kShipVerts];                      // ship_n[j] . ship_l[j]: offset of the hull's plane j (rotation invariant)
    float ship_aabb[4];                                // body-frame l,b,r,t of the hull
    float goal_cull_r2;                              // (max |hull vertex| + goal radius)^2: bounding circle about the body origin
    // episode log (shipsim_episode_log_bind; log_count == nullptr: off, and the kernels run their log-free instantiation)
    float4 *log_rows;                                // [log_cap][log_row4]
    int4 *log_meta;                                  // [log_cap][2] = SHIPSIM_EP_K .. SHIPSIM_EP_CALL
    int *log_count;
    int log_cap, log_row4;                           // log_row4 = float4 per record row (4 * the config's history)
    int log_k0;                                      // added to the step index (the chunk offset of shipsim_step_host)
    int log_call;                                    // sequence number of the step call
    // lidar fans other than the reference's 10 beams (the wide step kernel; appended so that the fields above keep their
    // parameter offsets in the tuned kernels)
    int n_beams;                                     // 1 .. kMaxBeams
    float ray_cw[kMaxBeams], ray_sw[kMaxBeams];      // the whole fan's ray table (entries past n_beams: unused)
    // weighted scenario picks (shipsim_scenario_weights; pick_cdf == nullptr: uniform picks, and the step kernels run their
    // pick-free instantiation).
    // Appended for the same reason as the beam fields.  Built on the stream by build_pick_table_kernel.
    const unsigned *pick_cdf;                        // [n_scen + 1]: inclusive prefix sums of the weights, then the total (0: uniform)
    const unsigned *pick_guide;                      // [n_scen + 1]: first i with cdf[i] > floor(j * total / n_scen); [n_scen] = n_scen - 1
    // chained launches (shipsim_step_chained): per-env tickets, [N] each, owned by the handle and zeroed at
    // shipsim_bind_state.  started[e] counts the chained launches that have claimed env e, done[e] those that have
    // stored its state.  Appended for the same reason as the beam fields.
    unsigned *chain_started, *chain_done;
};

// State planes [kPlanes, kPlanes + extra_lidar_planes(n)) hold lidar[10 .. n-1], four readings per plane.
__host__ __device__ __forceinline__ int extra_lidar_planes(int n_beams) { return n_beams > kBeams ? (n_beams - kBeams + 3) / 4 : 0; }

// SHIPSIM_END_* (include/shipsim.h)
constexpr int kEndCollision = 1, kEndAllGoals = 2, kEndOob = 4, kEndTimeout = 8, kEndGoal = 16;

__device__ __forceinline__ int end_bits(bool colliding, bool all_goals, bool oob, bool timeout, bool goal_reached)
{
    return (colliding ? kEndCollision : 0) | (all_goals ? kEndAllGoals : 0) | (oob ? kEndOob : 0) | (timeout ? kEndTimeout : 0)
           | (goal_reached ? kEndGoal : 0);
}

// Episode log: one atomic per warp reserves the slots of the lanes in `m` (a ballot; non-zero, warp-uniform), which are
// handed out in lane order.  Returns this lane's slot (meaningful where its bit of m is set).
__device__ __forceinline__ unsigned log_reserve(const StepParams &p, int lane, unsigned m)
{
    const int src = __ffs(m) - 1;
    unsigned base = 0u;
    if (lane == src) base = (unsigned)atomicAdd(p.log_count, __popc(m));
    base = __shfl_sync(0xffffffffu, base, src);
    return base + (unsigned)__popc(m & ((1u << lane) - 1u));
}

// the record's metadata (the caller writes the row: its last `4 * history` float4 of log_rows[slot])
__device__ __forceinline__ void log_meta(const StepParams &p, unsigned slot, int k, int e, int steps, float ret, int end, int scen, int ep)
{
    int4 *m = p.log_meta + (size_t)slot * 2;
    m[0] = make_int4(p.log_k0 + k, e, steps, __float_as_int(ret));
    m[1] = make_int4(end, scen, ep, p.log_call);
}

struct EnvRegs {
    float x, y, th, vx, vy, w, ret;
    int rudder, alive, steps, scen, episode;
};

// ---------------------------------------------------------------------------------------------- Philox4x32-10
__device__ __forceinline__ uint4 philox4x32_10(unsigned long long seed, unsigned long long ctr_lo, unsigned c2, unsigned c3)
{
    unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
    unsigned c0 = (unsigned)ctr_lo, c1 = (unsigned)(ctr_lo >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

// Which scenario an env's next episode plays (ShipGame.reset builds a new level every time, game.py:271-272).  Finite bank:
// a uniform draw keyed by (seed, global env id, episode) -- an integer hash (three multiply-xorshift rounds per word, the
// "triple32" finaliser), not Philox: a pick sits on the reset path of both kernels, where the ten Philox rounds were 6 %
// of the window kernel's instructions (profiles/r02_*), and nothing but uniformity and independence of the sharding
// is asked of it.  Fresh-maps mode (shipsim_fresh_maps): the bank is regenerated slice by slice behind the envs; resets
// pick from the slice generated last, walking it with a per-env offset and odd stride, so that an env never meets the
// same map twice (a slice is retired before the walk could wrap: see fresh_tick).
__device__ __forceinline__ unsigned mix32(unsigned x)
{
    x ^= x >> 17; x *= 0xed5ad4bbu; x ^= x >> 11; x *= 0xac4c1b51u; x ^= x >> 15; x *= 0x31848babu; x ^= x >> 14;
    return x;
}
// everything of a pick but the episode number (constant per env)
__device__ __forceinline__ unsigned pick_key(const StepParams &p, long long gid)
{
    unsigned k = mix32((unsigned)p.seed ^ 0x9E3779B9u);
    k = mix32(k ^ (unsigned)(p.seed >> 32));
    k = mix32(k ^ (unsigned)(unsigned long long)gid);
    return mix32(k ^ (unsigned)((unsigned long long)gid >> 32));
}
// Weighted pick from the hash h (shipsim_scenario_weights): with t = umulhi(h, total), the first i with cdf[i] > t.  The
// answer lies in [guide[j], guide[j + 1]] for the bucket j = umulhi(h, n_scen) (floor(j * total / n) <= t <
// floor((j + 1) * total / n) + 1), so a binary search over that range ends it: a run of zero weights costs no linear scan.
// With equal weights w the pick is floor(umulhi(h, n * w) / w) == umulhi(h, n), the uniform pick; total == 0 (all weights
// zero, or a sum of 2^32 or more) falls back to it as well.
__device__ __forceinline__ int pick_weighted(const StepParams &p, unsigned h)
{
    const unsigned n = (unsigned)p.n_scen;
    const unsigned j = __umulhi(h, n);
    const unsigned total = __ldg(p.pick_cdf + n);
    unsigned lo = __ldg(p.pick_guide + j), hi = __ldg(p.pick_guide + j + 1);
    if (total == 0u) return (int)j;
    const unsigned t = __umulhi(h, total);
    while (lo < hi) {
        const unsigned mid = (lo + hi) >> 1;
        if (__ldg(p.pick_cdf + mid) > t) hi = mid;
        else lo = mid + 1u;
    }
    return (int)lo;
}
// PICK: weighted picks (p.pick_cdf != nullptr).  The step kernels take it as a template flag, like the episode log's LOG,
// so that their weight-free instantiations are the kernels as they were.
template <bool PICK>
__device__ __forceinline__ int pick_scenario_keyed(const StepParams &p, unsigned key, int episode)
{
    if (p.pick_count > 0) {
        const unsigned stride = mix32(key ^ 0x5bd1e995u) | 1u;
        return p.pick_base + (int)((key + (unsigned)episode * stride) & (unsigned)(p.pick_count - 1));
    }
    const unsigned h = mix32(key + (unsigned)episode * 0x9E3779B9u);
    if (PICK) return pick_weighted(p, h);
    return (int)__umulhi(h, (unsigned)p.n_scen);
}
template <bool PICK>
__device__ __forceinline__ int pick_scenario(const StepParams &p, long long gid, int episode)
{
    return pick_scenario_keyed<PICK>(p, pick_key(p, gid), episode);
}

__device__ __forceinline__ int random_action(const StepParams &p, long long gid, unsigned step)
{
    const uint4 r = philox4x32_10(p.seed, (unsigned long long)gid, step, 1u);
    return (int)__umulhi(r.x, 3u);
}

// ---------------------------------------------------------------------------------------------- sin / cos
// One sincos per env-step sits on the loop-carried critical path (pose -> overlap tests -> done -> reset -> pose).
// Cody-Waite reduction by pi/2 (3 constants, exact for |x| < ~1e5, which bounds any reachable angle:
// |w| <= ~1.4 rad/s * dt over at most max_steps steps) + the usual minimax polynomials on [-pi/4, pi/4];
// ~1 ulp, no local-memory slow path in the hot loop (libdevice's Payne-Hanek branch is kept for huge angles).
// never taken in practice: kept out of the loop body (returns by value -- pointers would pin sin / cos to local memory)
static __device__ __noinline__ float2 sincos_huge(float x)
{
    float sn, cs;
    sincosf(x, &sn, &cs);
    return make_float2(sn, cs);
}

__device__ __forceinline__ void sincos_fast(float x, float &sn, float &cs)
{
    if (fabsf(x) > 1.0e5f) { const float2 v = sincos_huge(x); sn = v.x; cs = v.y; return; }
    const float q = rintf(x * 0.636619772367581343f);          // 2/pi
    float r = fmaf(q, -1.57079601287841796875f, x);
    r = fmaf(q, -3.1391647326017846353352069854736e-07f, r);
    r = fmaf(q, -5.3903029534742383771844745924903e-15f, r);
    const int n = (int)q;
    const float r2 = r * r;
    float sp = fmaf(r2, -1.95152959e-4f, 8.33216087e-3f);
    sp = fmaf(sp, r2, -1.66666546e-1f);
    sp = fmaf(sp * r2, r, r);
    float cp = fmaf(r2, 2.44331571e-5f, -1.38873163e-3f);
    cp = fmaf(cp, r2, 4.16666457e-2f);
    cp = fmaf(cp, r2, -0.5f);
    cp = fmaf(cp, r2, 1.0f);
    const float s1 = (n & 1) ? cp : sp;
    const float c1 = (n & 1) ? sp : cp;
    sn = (n & 2) ? -s1 : s1;
    cs = ((n + 1) & 2) ? -c1 : c1;
}

// ---------------------------------------------------------------------------------------------- state I/O
__device__ __forceinline__ int pack_bits(int rudder, int alive, int steps)
{
    return ((rudder / 5 + 2) & 7) | ((alive & 31) << 3) | (steps << 8);
}

// goals travel as the three raw float4 planes (g0 = goal0.xy goal1.xy, g1 = goal2.xy goal3.xy, g2 = goal4.xy, -, -)
__device__ __forceinline__ void load_env(const StepParams &p, int e, EnvRegs &r, float4 &l0, float4 &l1, float4 &l2, float4 &g0,
                                         float4 &g1, float4 &g2)
{
    const float4 *s = p.state;
    const size_t N = (size_t)p.N;
    const float4 a = s[0 * N + e], b = s[1 * N + e];
    l0 = s[2 * N + e]; l1 = s[3 * N + e]; l2 = s[4 * N + e];       // lidar[0..9], bits(scenario), bits(episode)
    g0 = s[5 * N + e]; g1 = s[6 * N + e]; g2 = s[7 * N + e];
    r.x = a.x; r.y = a.y; r.th = a.z; r.vx = a.w;
    r.vy = b.x; r.w = b.y; r.ret = b.z;
    const int bits = __float_as_int(b.w);
    r.rudder = ((bits & 7) - 2) * 5; r.alive = (bits >> 3) & 31; r.steps = bits >> 8;
    r.scen = __float_as_int(l2.z); r.episode = __float_as_int(l2.w);
}

__device__ __forceinline__ void store_env(const StepParams &p, int e, const EnvRegs &r, float4 l0, float4 l1, float l8, float l9)
{
    float4 *s = p.state;
    const size_t N = (size_t)p.N;
    s[0 * N + e] = make_float4(r.x, r.y, r.th, r.vx);
    s[1 * N + e] = make_float4(r.vy, r.w, r.ret, __int_as_float(pack_bits(r.rudder, r.alive, r.steps)));
    s[2 * N + e] = l0;
    s[3 * N + e] = l1;
    s[4 * N + e] = make_float4(l8, l9, __int_as_float(r.scen), __int_as_float(r.episode));
}

__device__ __forceinline__ void store_goals(const StepParams &p, int e, float4 g0, float4 g1, float4 g2)   // goals only change on reset
{
    float4 *s = p.state;
    const size_t N = (size_t)p.N;
    s[5 * N + e] = g0; s[6 * N + e] = g1; s[7 * N + e] = make_float4(g2.x, g2.y, 0.f, 0.f);
}

// ---------------------------------------------------------------------------------------------- chained launches
// Programmatic dependent launch (PTX griddepcontrol): launch_dependents lets the next launch of the stream start once
// every CTA of this one has executed it (or exited); wait blocks until the previous launch has completed and its
// memory is visible.  Both are no-ops in a launch without the programmatic-serialization attribute.
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ unsigned long long global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// A chained env waits this long at most for its previous launch: far beyond any launch a caller would make (a CTA of
// the headline runs for under half a millisecond), so only a broken ticket sequence reaches it, and then the kernel
// traps with a message instead of holding the GPU forever.
constexpr unsigned long long kChainWaitNs = 120ull * 1000000000ull;

static __device__ __noinline__ void chain_stuck(int e, unsigned ticket, unsigned done)
{
    printf("shipsim: chained launch, env %d: ticket %u still waits after %llu s (done = %u)\n", e, ticket, kChainWaitNs / 1000000000ull, done);
    __trap();
}

// Spin until the launch that holds ticket - 1 of env e has stored the env's state: done[e] - ticket >= 0 (wrap-safe),
// acquire at gpu scope so that the state loads after it see that launch's stores.
__device__ __forceinline__ void chain_await(const unsigned *done, unsigned ticket, int e)
{
    unsigned d;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(d) : "l"(done) : "memory");
    if ((int)(d - ticket) >= 0) return;
    const unsigned long long t0 = global_ns();
    unsigned ns = 64;
    for (;;) {
        __nanosleep(ns);
        if (ns < 1024) ns <<= 1;
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(d) : "l"(done) : "memory");
        if ((int)(d - ticket) >= 0) return;
        if (global_ns() - t0 > kChainWaitNs) chain_stuck(e, ticket, d);
    }
}

// Publish that the env's state for ticket `ticket` is stored (release at gpu scope).  max, not a plain store: the counter
// stays monotonic even if a caller races chained launches of one handle across streams.
__device__ __forceinline__ void chain_release(unsigned *done, unsigned ticket)
{
    asm volatile("red.release.gpu.global.max.u32 [%0], %1;" :: "l"(done), "r"(ticket + 1u) : "memory");
}

// ShipGame.reset + ShipEnv.reset for one env (game.py:260-277, ship_env.py:171-184); the goals come from the bank
// record of `scen` (float4 2..4) and are handled by the caller.
__device__ __forceinline__ void reset_env(const StepParams &p, EnvRegs &r, int scen, int episode)
{
    r.x = p.spawn_x; r.y = p.spawn_y; r.th = 0.f; r.vx = 0.f; r.vy = 0.f; r.w = 0.f; r.ret = 0.f;
    r.rudder = 0; r.alive = (1 << kGoals) - 1; r.steps = 0; r.scen = scen; r.episode = episode;
}

// ShipGame.closest_goal (game.py:333-349): first strict minimum wins; (-1,-1) when none (ship_env.py:103-107)
__device__ __forceinline__ void closest_goal(const float2 (&g)[kGoals], int alive, float x, float y, float &gx, float &gy)
{
    float best = 3.0e38f;
    gx = -1.f; gy = -1.f;
#pragma unroll
    for (int k = 0; k < kGoals; ++k) {
        const float dx = g[k].x - x, dy = g[k].y - y;
        const float d2 = dx * dx + dy * dy;
        const bool take = ((alive >> k) & 1) && d2 < best;
        if (take) { best = d2; gx = g[k].x; gy = g[k].y; }
    }
}

__device__ __forceinline__ void unpack_goals(float4 g0, float4 g1, float4 g2, float2 (&g)[kGoals])
{
    g[0] = make_float2(g0.x, g0.y); g[1] = make_float2(g0.z, g0.w); g[2] = make_float2(g1.x, g1.y);
    g[3] = make_float2(g1.z, g1.w); g[4] = make_float2(g2.x, g2.y);
}

// The goals of scenario `scen`: bank record float4 2..4 (what the state's goal planes g0..g2 hold), unpacked into g.
// (The nearest-goal search is left to the caller: window_kernel issues more loads and the next pick in between.)
__device__ __forceinline__ void scenario_goals(const StepParams &p, int scen, float4 &g0, float4 &g1, float4 &g2, float2 (&g)[kGoals])
{
    const float4 *rec = p.bank + (size_t)scen * p.scen_stride4;
    g0 = __ldg(rec + 2); g1 = __ldg(rec + 3); g2 = __ldg(rec + 4);
    unpack_goals(g0, g1, g2, g);
}

// Circle-vs-poly contact (CircleToPoly): distance(goal centre, ship polygon) <= goal radius, evaluated in the
// body frame where the hull is constant.  cpPolyShapePointQuery semantics: inside => negative distance.
__device__ __forceinline__ bool goal_culled(const StepParams &p, float qx, float qy)
{
    const float rr = p.goal_r;
    return qx < p.ship_aabb[0] - rr || qx > p.ship_aabb[2] + rr || qy < p.ship_aabb[1] - rr || qy > p.ship_aabb[3] + rr;
}

__device__ __forceinline__ bool goal_touches_ship(const StepParams &p, float qx, float qy)
{
    bool outside = false;
    float best = 3.0e38f;
#pragma unroll
    for (int j = 0; j < kShipVerts; ++j) {
        const int j0 = (j + kShipVerts - 1) % kShipVerts;
        const float ax = p.ship_lx[j0], ay = p.ship_ly[j0], bx = p.ship_lx[j], by = p.ship_ly[j];
        outside = outside || (p.ship_nx[j] * (qx - bx) + p.ship_ny[j] * (qy - by) > 0.f);
        const float ex = ax - bx, ey = ay - by;                       // cpClosetPointOnSegment
        float t = __fdividef(ex * (qx - bx) + ey * (qy - by), ex * ex + ey * ey);
        t = fminf(fmaxf(t, 0.f), 1.f);
        const float cx = bx + ex * t - qx, cy = by + ey * t - qy;
        best = fminf(best, cx * cx + cy * cy);
    }
    return !outside || best <= p.goal_r * p.goal_r;
}

// The same contact test with the clear cases settled first: the largest signed distance m of the goal centre to the
// hull's edge lines decides "centre well inside the hull" (m < -eps: contact) and "farther than the goal radius from
// some edge line" (m > r + eps: no contact, the true distance is at least m); eps = 1e-3 is orders of magnitude above
// fp32 rounding at these magnitudes, so both shortcuts agree with the full test, which decides everything else.
__device__ __forceinline__ bool goal_contact(const StepParams &p, float qx, float qy)
{
    float m = -3.0e38f;
#pragma unroll
    for (int j = 0; j < kShipVerts; ++j)
        m = fmaxf(m, p.ship_nx[j] * (qx - p.ship_lx[j]) + p.ship_ny[j] * (qy - p.ship_ly[j]));
    if (m < -1.0e-3f) return true;
    if (m > p.goal_r + 1.0e-3f) return false;
    return !goal_culled(p, qx, qy) && goal_touches_ship(p, qx, qy);
}

__device__ __forceinline__ void prefetch_l2(const void *ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); }
__device__ __forceinline__ void prefetch_l1(const void *ptr) { asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr)); }

// ---------------------------------------------------------------------------------------------- shared memory by address
// On sm_100 an access to a __shared__ array is LDS [reg + UR], where the uniform register holds the CTA's shared
// window base, 0x400 + (CgaCtaId << 24): ptxas rebuilds it with an S2UR wherever it runs out of uniform registers, and
// in these kernels that special-register read was the hottest stall of the loop (ncu: 14 % of the samples on one of
// them).  The hot loops therefore address shared memory through a 32-bit shared-space address that is computed once
// and kept in an ordinary register, with explicit ld.shared / st.shared.  (asm volatile: these keep their order among
// themselves and relative to __syncwarp, which is all the kernels rely on.)
__device__ __forceinline__ unsigned smem_addr(const void *ptr) { return (unsigned)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ float4 lds4(unsigned a)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint4 lds4u(unsigned a)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ float2 lds2(unsigned a)
{
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ float lds1(unsigned a)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ unsigned lds_u8(unsigned a)
{
    unsigned v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts4(unsigned a, float4 v)
{
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts2(unsigned a, float2 v) { asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(a), "f"(v.x), "f"(v.y) : "memory"); }
__device__ __forceinline__ void sts1(unsigned a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_u8(unsigned a, unsigned v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

// 16-byte asynchronous global -> shared copy (LDGSTS): no register staging, completes in the background
__device__ __forceinline__ void cp_async16_s(unsigned smem_dst, const void *gmem_src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) { cp_async16_s(smem_addr(smem_dst), gmem_src); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Episode statistics of one step for a whole warp: counters by ballot + popc, the two sums (episode return and length of
// the envs that finished) by visiting the few finished lanes.  Lane 0 adds the totals to the warp's eight accumulators
// (shared-space address `stat`): plain shared-memory read-modify-write, no atomics (measured: the shared atomics cost 4 %
// of the stall samples).
__device__ __forceinline__ void warp_stats(unsigned stat, int lane, bool counted, bool goal_reached, bool done, bool colliding, bool oob,
                                           bool timeout, bool all_goals, float ep_return, int ep_steps)
{
    const unsigned gm = __ballot_sync(kFull, counted && goal_reached);
    const unsigned dm = __ballot_sync(kFull, counted && done);
    if ((gm | dm) == 0u) return;                                    // warp-uniform
    const unsigned cm = __ballot_sync(kFull, counted && done && colliding), om = __ballot_sync(kFull, counted && done && oob);
    const unsigned tm = __ballot_sync(kFull, counted && done && timeout), am = __ballot_sync(kFull, counted && done && all_goals);
    float rsum = 0.f, ssum = 0.f;
    for (unsigned m = dm; m; m &= m - 1u) {
        const int src = __ffs(m) - 1;
        rsum += __shfl_sync(kFull, ep_return, src);
        ssum += (float)__shfl_sync(kFull, ep_steps, src);
    }
    if (lane == 0) {
        float4 a = lds4(stat), b = lds4(stat + 16);
        a.x += (float)__popc(dm); a.y += rsum; a.z += ssum; a.w += (float)__popc(gm);
        b.x += (float)__popc(cm); b.y += (float)__popc(om); b.z += (float)__popc(tm); b.w += (float)__popc(am);
        sts4(stat, a); sts4(stat + 16, b);
    }
}

__device__ __forceinline__ float sqrt_approx(float x)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

}  // namespace shipsim
