// shipsim_kernels.cu -- the fused ShipEnv step kernel (K env-steps per launch), reset, stats and bank-build kernels.
// sm_100a only.  See shipsim_device.cuh for the data layout and the reference lines each piece restates.
//
// Execution model.  G lanes cooperate on one env (G = 1..32, 32/G envs per warp); the lanes of a group hold
// identical copies of the env's scalar state.  Per-env work that is regular runs per lane; the irregular geometry is
// done in two ways that keep control flow warp-uniform no matter how few envs of a warp are near a bank:
//   * plane phase (owner lane): the reach grid names the few bank edges near the env; their planes are evaluated in
//     double at the new pose, which at once (a) settles the ship-vs-bank test for all but touching cases and (b) leaves
//     in shared memory everything the NEXT step's lidar needs;
//   * ray pass (whole warp): three needy envs at a time, one lane per (env, ray), reading those planes;
//   * SAT pass (whole warp, rare): 32/lps envs at a time, one lane per (env, bank edge).
// The loop is rotated: an iteration starts with the pose already integrated, so that the grid cell of the pose an
// iteration works on was requested a whole iteration earlier.
#include "shipsim_geom.cuh"
#include "shipsim_launch.h"

#include <atomic>

namespace shipsim {

// Grids that fill the machine (one lane per env, >= 1,184 CTAs of 128 envs' worth): CTA size and CTAs per SM to aim
// for.  Registers per thread follow from the pair: 128 x 5 -> 96, 64 x 9 -> 112, 128 x 4 / 64 x 8 -> 128.  Spills are
// ruinous here (the L1 that would catch them is almost entirely carved out as shared memory), so the shape is chosen
// as the most warps per SM that still compile without any.
constexpr int kBigThreads = 128, kBigMinBlocks = 5;
// All other grids: CTA size, and CTAs of kThreads threads per SM to aim for (launch_g)
constexpr int kSmallThreads = 64, kMinBlocks = 4;

constexpr float kDeadGoal = 3.0e19f;        // coordinate of a goal that has been taken: its squared distance is +inf

// MINB = CTAs per SM the register allocation aims for: 5 (96 registers) pays off only when the grid is large enough
// to fill them, otherwise 4 (128 registers, less rematerialisation).
//
// Shared memory: ONE array; every env has one block of EB4 float4 (odd stride: the 128-bit accesses of a warp's envs
// are conflict-free) holding its observation tile row, its plane row and its goals at compile-time offsets, addressed
// from a single per-lane byte offset.  (Round 1 kept seven arrays with their own index arithmetic; at 96 registers the
// compiler rebuilt those indices from threadIdx / blockIdx inside the loop: 12 % of the instructions, and an S2R
// stall that was the hottest sample of the kernel.  The offsets are laundered through an empty asm so that they stay
// in their registers.)
// LOG: write the episode log (shipsim_episode_log_bind).  The log-free kernel is a separate instantiation: its registers
// and spills are those of the kernel before the log existed (-Xptxas -v).
// PICK: weighted scenario picks (shipsim_scenario_weights), a separate instantiation for the same reason.
// NB: lidar capacity.  kBeams (10) is the tuned kernel of the reference's fan, with the beam count a compile-time constant;
// kMaxBeams (32) is the wide kernel: a 32-reading frame slot, p.n_beams (1..32) rays at run time, and its shared memory
// allocated dynamically (StepLayout::BYTES; the G = 1 blocks exceed the 48 KB of a static allocation).  Everything else --
// physics, goals, SAT, reward / done, reset, statistics, episode log -- is this one body of code for both.
template <int G, int HIST, int NB, int THREADS>
struct StepLayout {
    static constexpr bool WIDE = NB != kBeams;
    static constexpr int EPW = 32 / G;                      // envs per warp
    static constexpr int FR4 = WIDE ? 10 : 4;               // float4 per frame slot: 6 + NB floats, rounded up
    static constexpr int OBS4 = FR4 * HIST;                 // float4 per tile row
    static constexpr int RAW = OBS4 + kScr4 + 3;
    static constexpr int EB4 = (RAW + (G > 1 ? 2 * kMaxCand : 0)) | 1;
    static constexpr int WX4 = EPW * EB4;
    static constexpr int RAYN = WIDE ? kMaxBeams : kBeams;  // ray table entries
    static constexpr int WB4 = WX4 + 4 + RAYN / 2;
    static constexpr int BYTES = THREADS / 32 * WB4 * 16;
};

template <int G, int HIST, int NB, int THREADS>
__device__ __forceinline__ float4 *step_smem()
{
    if constexpr (NB == kBeams) {
        __shared__ float4 smem[StepLayout<G, HIST, NB, THREADS>::BYTES / 16];
        return smem;
    } else {
        extern __shared__ float4 smem_dyn[];
        return smem_dyn;
    }
}

template <int G, int HIST, int MINB, int THREADS, bool LOG, int NB, bool PICK>
__global__ void __launch_bounds__(THREADS, MINB) step_kernel(const __grid_constant__ StepParams p)
{
    using LY = StepLayout<G, HIST, NB, THREADS>;
    constexpr bool WIDE = LY::WIDE;
    constexpr int EPW = 32 / G;                 // envs per warp
    constexpr int FR4 = LY::FR4;                // float4 per frame slot
    constexpr int OBS4 = LY::OBS4;              // float4 per tile row
    constexpr int NF = OBS4 - FR4;              // float4 index of the newest frame inside the tile row
    // ray pass: two passes (six envs) per loop trip in the 128-register build (grids that do not fill the machine are
    // latency bound: +4 % on the hard map at 65,536 envs); the 96-register build has no room for it (-1 % at 1M envs)
    constexpr int kRayPassUnroll = MINB * THREADS <= 512 ? 2 : 1;       // (512 threads per SM = the 128-register builds)
    constexpr int CF = 4 * NF;                  // float offset of the newest frame inside the tile row
    constexpr int NW = THREADS / 32;
    // env block: [0, OBS4) tile row = [older frame | newest frame] (lidar slots = the sticky readings);
    // [SCR, SCR + kScr4) plane row; [GOL, GOL + 3) goals (taken goals hold kDeadGoal)
    constexpr int SCR = OBS4, GOL = OBS4 + kScr4;
    // [RAW, RAW + 2 * kMaxCand): raw candidate-plane records (cp.async targets) -- only with G > 1 (few envs per CTA),
    // where they are requested at the top of the iteration; with G = 1 that would cost 16 KB, so they land in the plane
    // row itself once the ray pass has finished with it
    constexpr int RAW = LY::RAW;
    constexpr int EB4 = LY::EB4;
    // warp block: the env blocks, then 2 float4 of ray-pass list, 2 of statistics, RAYN / 2 of ray directions
    // (cos[RAYN], sin[RAYN])
    constexpr int WX4 = LY::WX4;
    constexpr int RAYN = LY::RAYN;
    constexpr int SRC = WX4, STA = WX4 + 2, RAY = WX4 + 4;
    constexpr int WB4 = LY::WB4;
    // the last float4 of an env block exists only to make the stride odd: it is the landing slot of fetch_cell_async
    constexpr int CEL = EB4 - 1;
    static_assert(CEL >= RAW + (G > 1 ? 2 * kMaxCand : 0), "the cell slot must not overlap the block's contents");
    float4 *const smem = step_smem<G, HIST, NB, THREADS>();
    const int nb = WIDE ? p.n_beams : kBeams;  // rays of the fan

    // Everything a lane needs to find its data -- lane, warp, shared-memory offsets, output indices -- follows from ONE
    // value, the env index e, by a mask, a shift or a multiply-add; e itself is laundered (a shuffle from the own lane:
    // an identity the assembler cannot see through) so that nothing is rebuilt from the special registers inside the loop.
    int e = (blockIdx.x * NW + (threadIdx.x >> 5)) * EPW + (threadIdx.x & 31) / G;
    int lane;
    if (G == 1) {
        e = __shfl_sync(kFull, e, threadIdx.x & 31);
        lane = e & 31;
    } else {
        lane = threadIdx.x & 31;
        lane = __shfl_sync(kFull, lane, lane);
        e = __shfl_sync(kFull, e, lane);
    }
    const int grp = lane / G, gl = lane % G;
    // Shared memory is addressed by 32-bit shared-space addresses held in ordinary registers (see "shared memory by
    // address" in shipsim_device.cuh): eb = this env's block (laundered like e), wb = this warp's block, one
    // multiply-add away.
    unsigned eb = smem_addr(smem) + (unsigned)(((e / EPW) & (NW - 1)) * WB4 + grp * EB4) * 16u;   // (blockIdx.x * NW is a multiple of NW)
    eb = __shfl_sync(kFull, eb, lane);
    const unsigned wb = eb - (unsigned)(grp * EB4) * 16u;
    const bool valid = e < p.N;
    const bool leader = valid && gl == 0;
#define EA(i) (eb + 16u * (unsigned)(i))                     /* address of float4 i of this env's block */
#define WA(env, i) (wb + (unsigned)(env) * (EB4 * 16u) + 16u * (unsigned)(i))
    const float L = p.lidar_len;

    if (lane < RAYN) {                                              // ray direction table (body frame), one per warp
        sts1(wb + RAY * 16 + 4 * lane, WIDE ? p.ray_cw[lane] : p.ray_c[lane]);
        sts1(wb + RAY * 16 + 4 * RAYN + 4 * lane, WIDE ? p.ray_sw[lane] : p.ray_s[lane]);
    }
    if (lane < 8) sts1(wb + STA * 16 + 4 * lane, 0.f);
    if (!valid && gl == 0) sts4(EA(SCR), make_float4(1.f, 0.f, 0.f, 0.f));      // idle groups: a defined heading for the shadow lanes

    EnvRegs r;
    {
        float4 l0, l1, l2, g0, g1, g2;
        load_env(p, valid ? e : p.N - 1, r, l0, l1, l2, g0, g1, g2);   // lanes of idle groups shadow the last env; they never store
        float2 g[kGoals];
        unpack_goals(g0, g1, g2, g);
        float gx, gy;
        closest_goal(g, r.alive, r.x, r.y, gx, gy);
        if (gl == 0) {
#pragma unroll
            for (int i = 0; i < kGoals; ++i) if (!((r.alive >> i) & 1)) g[i] = make_float2(kDeadGoal, kDeadGoal);
            sts4(EA(GOL), make_float4(g[0].x, g[0].y, g[1].x, g[1].y));
            sts4(EA(GOL + 1), make_float4(g[2].x, g[2].y, g[3].x, g[3].y));
            // .z, .w: the goals-alive mask and the episode number live here, not in registers (a taken goal and a reset are
            // the only things that touch them)
            sts4(EA(GOL + 2), make_float4(g[4].x, g[4].y, __int_as_float(r.alive), __int_as_float(r.episode)));
            store_frame(RowSmem{EA(NF)}, r, gx, gy, l0, l1, l2);    // newest frame of the resident tile = frame of the current state
            if (WIDE) {                         // lidar[10 ..] from the appended state planes: float4 q of them = tile float4 NF + 4 + q
                const int nx = extra_lidar_planes(nb);
                for (int q = 0; q < nx; ++q) sts4(EA(NF + 4 + q), p.state[(size_t)(kPlanes + q) * p.N + (valid ? e : p.N - 1)]);
            }
        }
    }
    float c, s, hx, hy;
    sincos_fast(r.th, s, c);
    hull_half_extents(p, c, s, hx, hy);
    // (G > 1: the lanes of a group share the env's block.  One lane fetches / writes, and wherever another lane's read and
    // the leader's write of the same word are not already separated by a warp synchronisation, one is placed -- all of them
    // compile away for G = 1.  compute-sanitizer racecheck: profiles/r02_x_sanitize.txt)
    if (G == 1 || gl == 0) fetch_cell_async(p, r.scen, r.x + hx, r.y + hy, EA(CEL));
    __syncwarp();                                // ray table, statistics and tile initialisation (all per warp) are in place

    // Iteration k >= 0 is env-step k and starts with the pose ALREADY integrated (cpBodyUpdatePosition of step k);
    // iteration -1 only runs the plane phase at the loaded pose and the first integration.
#pragma unroll 1
    for (int k = -1; k < p.K; ++k) {
        const bool live = k >= 0;
        bool done = false, do_reset = false, goal_reached = false;
        float reward = 0.f, gx = -1.f, gy = -1.f;
        if (live) {
            // this step's action: asked for first, looked at after the lidar pass (kept in a register across the loop it was
            // the one value the 96-register build spilled -- and a spilled prefetch is a synchronous load)
            const int a = load_action_at(p, (size_t)k * p.N + min(e, p.N - 1), k, p.env_id_offset + e);   // (idle lanes read the last env's)
            // previous frame <- newest frame of the last step / reset (SURVEY.md App. A note N2); lidar stays in place
            if (HIST == 2 && gl == 0) {
                if (!WIDE) {
                    const float4 f0 = lds4(EA(4)), f1 = lds4(EA(5)), f2 = lds4(EA(6)), f3 = lds4(EA(7));
                    sts4(EA(0), f0); sts4(EA(1), f1); sts4(EA(2), f2); sts4(EA(3), f3);
                } else {                        // the float4 that hold the 6 + n values of a frame
                    const int f4 = (6 + nb + 3) >> 2;
#pragma unroll
                    for (int i = 0; i < FR4; ++i) if (i < f4) sts4(EA(i), lds4(EA(FR4 + i)));
                }
            }

            // ---- LiDAR.query (models.py:39-76) at the PRE-integration pose (game.py:193 precedes :194): the plane
            // rows hold that pose's planes.  Up to three needy envs per pass, lanes 0-9 / 10-19 / 20-29 = their rays
            // (the wide kernel: 32 / n envs per pass, lanes [n * slot, n * slot + n) = the rays of slot `slot`).
            const float4 h0 = lds4(EA(SCR));    // header of the pose the step starts from: its trig, and what its lidar needs
            const int hz_own = __float_as_int(h0.z);
            const bool big = leader && (hz_own & kHdrBig);
            const bool wants = leader && (hz_own & 0x3ff) != 0;
            const unsigned need = __ballot_sync(kFull, wants);
            if (HIST == 2) __syncwarp();        // the frame copy has read the old readings before any lane overwrites them
            if (big) {                          // (rare: generic pointers are good enough)
                float4 *blk = smem + ((e / EPW) & (NW - 1)) * WB4 + grp * EB4;
                if (WIDE) ray_query_serial_wide(p, blk + SCR, reinterpret_cast<float *>(blk) + CF + 6);
                else ray_query_serial(p, blk + SCR, reinterpret_cast<float *>(blk) + CF + 6);
            }
            if (need) {
                // needy envs, compacted: entry q of the warp's list = the env slot of the q-th needy env
                if (wants) sts_u8(wb + SRC * 16 + __popc(need & ((1u << lane) - 1u)), (unsigned)grp);
                __syncwarp();
                const int cnt = __popc(need);
                const int rslot = lane / nb, rj = lane - rslot * nb;        // env slot 0..2 of the pass (lanes 30, 31 idle), ray
                const int rpp = WIDE ? 32 / nb : 3;                         // envs per pass
                const float ray_c = lds1(wb + RAY * 16 + 4 * rj), ray_s = lds1(wb + RAY * 16 + 4 * RAYN + 4 * rj);     // (lanes of a ray: broadcast)
#pragma unroll kRayPassUnroll
                for (int q = rslot; q < cnt; q += rpp) {        // lanes 30, 31 (rslot 3) only keep the others company
                    if (rslot < rpp) {
                        const unsigned ra = WA(lds_u8(wb + SRC * 16 + q), 0);      // the env's block
                        const float v = ray_vs_row(RowSmem{ra + SCR * 16}, ray_c, ray_s, L);
                        if (v >= 0.f) sts1(ra + 4 * (CF + 6 + rj), v);          // misses keep the old reading (sticky vals, models.py:71)
                    }
                }
            }

            // ---- ShipGame.handle_discrete_action (game.py:140-153); Ship.move_forward / rotate (models.py:129-146)
            // The rudder angle lives in the tile, as the third value of the newest frame (exact: a small integer in fp32).
            float dvx = 0.f, dvy = 0.f, dw = 0.f;
            const unsigned rud_slot = EA(NF) + 8;
            const float rud = lds1(rud_slot);
            if (G > 1) __syncwarp();            // every lane has the old angle before the leader stores the new one
            if (a == 0) {                       // thrust along the heading the step starts from
                dvx = -p.acc_dt * h0.y; dvy = p.acc_dt * h0.x; dw = -p.ang_dt * rud;
            }
            else if (a == 1) { if (gl == 0) sts1(rud_slot, fmaxf(rud - 5.f, -10.f)); }
            else if (a == 2) { if (gl == 0) sts1(rud_slot, fminf(rud + 5.f, 10.f)); }
            // ---- cpBodyUpdateVelocity: v = v*damping + f/m*dt, w = w*damping + t/I*dt.  Nothing between here and the next
            // cpBodyUpdatePosition looks at the velocities (the overlap tests below work on the pose), so they are
            // advanced at once instead of carrying the three force terms across the cooperative passes.
            r.vx = r.vx * p.damping + dvx;
            r.vy = r.vy * p.damping + dvy;
            r.w = r.w * p.damping + dw;
        }
        __syncwarp();                           // the plane rows have been read (thrust heading, ray pass): they may be rewritten

        // the reach-grid cell of the integrated pose was asked for an iteration ago (asynchronous copy): it names the
        // candidate planes, whose raw records are now copied global -> shared the same way -- with G = 1 into the plane
        // row itself, which the ray pass has finished with, otherwise into the env's own staging area
        cp_async_wait_all();
        if (G > 1) __syncwarp();                // the leader's copy has landed before the group's other lanes look
        const uint4 cell = lds4u(EA(CEL));
        const bool near_any = leader && (cell.x | cell.y | (cell.z & 3u)) != 0u;
        const bool staged = near_any && ((cell.z >> 8) & 0xffu) <= (unsigned)kMaxCand;
        const RowSmem raw{G > 1 ? EA(RAW) : EA(SCR + 1)};
        if (staged) stage_candidates(p, r.scen, cell, raw);
        bool all_goals = false;
        if (live) {     // (while the candidate planes are in flight)
            // ---- goals (collide_goal, game.py:243-257) and the nearest remaining goal (closest_goal, game.py:333-349).
            // The squared distance to the body origin serves both the nearest-goal search and a bounding-circle cull;
            // only goals inside the circle are rotated into the body frame for the exact circle-vs-hull test.  Taken
            // goals sit at kDeadGoal: their distance is +inf, so neither the cull nor the search needs the alive mask.
            float2 g[kGoals];
            float gd2[kGoals];
            {
                const float4 ga = lds4(EA(GOL)), gb = lds4(EA(GOL + 1));
                const float2 gc = lds2(EA(GOL + 2));
                g[0] = make_float2(ga.x, ga.y); g[1] = make_float2(ga.z, ga.w); g[2] = make_float2(gb.x, gb.y);
                g[3] = make_float2(gb.z, gb.w); g[4] = gc;
            }
            if (G > 1) __syncwarp();            // every lane has the goals before the leader retires one
            unsigned cand = 0u;
#pragma unroll
            for (int i = 0; i < kGoals; ++i) {
                const float ux = g[i].x - r.x, uy = g[i].y - r.y;
                gd2[i] = ux * ux + uy * uy;
                if (gd2[i] <= p.goal_cull_r2) cand |= 1u << i;
            }
            if (!valid) cand = 0u;
            float took = 0.f;                   // (a float: as a bool set inside the loop this flag was spilled to local memory)
#pragma unroll 1
            while (cand) {                      // rarely more than one trip
                const int i = __ffs(cand) - 1;
                cand &= cand - 1u;
                float ux = g[0].x, uy = g[0].y;
#pragma unroll
                for (int j = 1; j < kGoals; ++j) if (i == j) { ux = g[j].x; uy = g[j].y; }
                ux -= r.x; uy -= r.y;
                const float qx = ux * c + uy * s, qy = -ux * s + uy * c;
                if (goal_contact(p, qx, qy)) {
                    took = 1.f;
#pragma unroll
                    for (int j = 0; j < kGoals; ++j) if (i == j) gd2[j] = __int_as_float(0x7f800000);
                    if (gl == 0) {
                        sts2(EA(GOL) + 8 * i, make_float2(kDeadGoal, kDeadGoal));
                        sts1(EA(GOL + 2) + 8, __int_as_float(__float_as_int(lds1(EA(GOL + 2) + 8)) & ~(1 << i)));
                    }
                }
            }
            goal_reached = took != 0.f;
            float best = 3.0e38f;
#pragma unroll
            for (int i = 0; i < kGoals; ++i)
                if (gd2[i] < best) { best = gd2[i]; gx = g[i].x; gy = g[i].y; }
            all_goals = !(best < 3.0e38f);            // every goal taken: no finite distance left

        }
        // ---- plane phase at the integrated pose: next step's lidar planes + this step's ship-vs-bank pre-test
        cp_async_wait_all();
        unsigned ask = 0u;
        if (leader) {
            if (staged) ask = plane_phase<true, true>(p, r.x, r.y, hx, hy, c, s, r.scen, cell, RowSmem{EA(SCR)}, raw);
            else if (near_any) ask = plane_phase<true, false>(p, r.x, r.y, hx, hy, c, s, r.scen, cell, RowSmem{EA(SCR)}, RowSmem{0u});
            else sts4(EA(SCR), make_float4(c, s, 0.f, 0.f));
        }

        if (live) {
            // ---- overlap test at the new pose -> begin callback collide_ship (game.py:232-241)
            bool colliding = false;
            {
                // Separating-axis test for the envs the plane phase could not settle.  Contact <=> no separating axis
                // among the edge normals of both convex polygons (touching counts: GJK distance <= 0).
                unsigned needs = __ballot_sync(kFull, ask != 0u);
                if (needs) {
                    const int lps_sh = p.hull_max <= 8 ? 3 : (p.hull_max <= 16 ? 4 : 5);    // log2(lanes per env slot)
                    const int lps = 1 << lps_sh, nslots = 32 >> lps_sh;
                    const int sslot = lane >> lps_sh, sel = lane & (lps - 1);
                    const unsigned slotmask = lps == 32 ? kFull : (((1u << lps) - 1u) << (sslot * lps));
                    while (needs) {
                        int src = -1, myslot = -1;
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            if (q < nslots && needs) {
                                const int t = __ffs(needs) - 1;
                                needs &= needs - 1u;
                                if (sslot == q) src = t;
                                if (t / G == grp) myslot = q;
                            }
                        }
                        const bool act_env = src >= 0;
                        const int srcl2 = act_env ? src : lane;
                        const float bx = __shfl_sync(kFull, r.x, srcl2), by = __shfl_sync(kFull, r.y, srcl2);
                        const float bc = __shfl_sync(kFull, c, srcl2), bs = __shfl_sync(kFull, s, srcl2);
                        const unsigned bsa = __shfl_sync(kFull, (unsigned)r.scen | (ask << 28), srcl2);
                        const float4 *rec = p.bank + (size_t)(bsa & 0x0fffffffu) * p.scen_stride4;
                        const float4 hdr = __ldg(rec + 4);
                        const float4 *bE = rec + kBankHeader4;
                        // the edge records of both banks are requested together with the header: their addresses do not
                        // depend on it (every slot below maxv exists), so one memory round trip serves the whole pass
                        float4 edb[2];
#pragma unroll
                        for (int b = 0; b < 2; ++b) {
                            edb[b] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (act_env && ((bsa >> (28 + b)) & 1u) && sel < p.maxv) edb[b] = __ldg(bE + b * p.maxv + sel);
                        }
                        float rx[kShipVerts], ry[kShipVerts];
#pragma unroll
                        for (int j = 0; j < kShipVerts; ++j) {
                            rx[j] = p.ship_lx[j] * bc - p.ship_ly[j] * bs;
                            ry[j] = p.ship_lx[j] * bs + p.ship_ly[j] * bc;
                        }
                        bool coll = false;
#pragma unroll
                        for (int b = 0; b < 2; ++b) {
                            const bool do_b = act_env && ((bsa >> (28 + b)) & 1u) && !coll;
                            const int nb = __float_as_int(b ? hdr.w : hdr.z);
                            const bool actl = do_b && sel < nb;
                            const float4 ed = edb[b];
                            const unsigned sb = __ballot_sync(kFull, actl && bank_axis_separates(ed, rx, ry, bx, by));   // a bank edge normal separates
                            bool sep = (sb & slotmask) != 0u;
                            if (__ballot_sync(kFull, do_b && !sep)) {                           // else try the ship's edge normals
#pragma unroll
                                for (int j = 0; j < kShipVerts; ++j) {
                                    const float nx = p.ship_nx[j] * bc - p.ship_ny[j] * bs;
                                    const float ny = p.ship_nx[j] * bs + p.ship_ny[j] * bc;
                                    const float pr = actl ? nx * (ed.z - bx) + ny * (ed.w - by) : 3.0e38f;
                                    // axis j separates <=> no bank vertex of the slot reaches the hull's plane j
                                    const unsigned reach = __ballot_sync(kFull, pr <= p.ship_off[j]);
                                    sep = sep || (reach & slotmask) == 0u;
                                }
                            }
                            if (do_b && !sep) coll = true;
                        }
                        const unsigned res = __ballot_sync(kFull, coll);
                        if (myslot >= 0 && ((res >> (myslot * lps)) & 1u)) colliding = true;
                    }
                }
            }

            // ---- ShipEnv.determine_reward (ship_env.py:62-77): collision alone does not change the value (Q12)
            const bool oob = (r.x < 0.f) || (r.x > p.W) || (r.y < 0.f) || (r.y > p.H);
            reward = goal_reached ? 1.f : (oob ? -1.f : p.step_penalty);
            r.ret += reward;
            r.steps += 1;
            const bool timeout = (r.steps >= p.max_steps);
            done = colliding || all_goals || oob || timeout;             // ship_env.py:115-134

            warp_stats(wb + STA * 16, lane, leader, goal_reached, done, colliding, oob, timeout, all_goals, r.ret, r.steps);
            do_reset = done && p.auto_reset;
            if (LOG) {
                // episode log: the terminal row -- the previous frame and the newest one completed with this step's pose,
                // rudder, nearest remaining goal and sticky lidar, i.e. what the frame block below writes without a reset --
                // and the episode's numbers, before the reset replaces them
                const unsigned lm = __ballot_sync(kFull, leader && done);
                if (lm) {
                    const unsigned slot = log_reserve(p, lane, lm);
                    if (leader && done && slot < (unsigned)p.log_cap) {
                        if (!WIDE) {
                            float4 *row = p.log_rows + (size_t)slot * p.log_row4 + (p.log_row4 - OBS4);
                            if (HIST == 2) { row[0] = lds4(EA(0)); row[1] = lds4(EA(1)); row[2] = lds4(EA(2)); row[3] = lds4(EA(3)); }
                            const float4 f1 = lds4(EA(OBS4 - 3));
                            row[OBS4 - 4] = make_float4(r.x, r.y, lds1(EA(OBS4 - 4) + 8), r.th);
                            row[OBS4 - 3] = make_float4(gx, gy, f1.z, f1.w);
                            row[OBS4 - 2] = lds4(EA(OBS4 - 2));
                            row[OBS4 - 1] = lds4(EA(OBS4 - 1));
                        } else {                // dense rows of (6 + n) * HIST floats
                            const int F = 6 + nb;
                            float *row = reinterpret_cast<float *>(p.log_rows) + (size_t)slot * (F * HIST);
                            if (HIST == 2) {
                                for (int i = 0; i < F; ++i) row[i] = lds1(EA(0) + 4 * i);
                                row += F;
                            }
                            row[0] = r.x; row[1] = r.y; row[2] = lds1(EA(NF) + 8); row[3] = r.th; row[4] = gx; row[5] = gy;
                            for (int i = 6; i < F; ++i) row[i] = lds1(EA(NF) + 4 * i);
                        }
                        log_meta(p, slot, k, e, r.steps, r.ret, end_bits(colliding, all_goals, oob, timeout, goal_reached), r.scen,
                                 __float_as_int(lds1(EA(GOL + 2) + 12)));
                    }
                }
            }
            int ep_g = 0;
            if (G > 1) {                        // read by every lane while the warp is converged, before the leader stores the next one
                ep_g = __float_as_int(lds1(EA(GOL + 2) + 12)) + 1;
                __syncwarp();
            }
            if (do_reset) {
                const int ep = G > 1 ? ep_g : __float_as_int(lds1(EA(GOL + 2) + 12)) + 1;    // (only a reset needs the episode number: kept in shared memory)
                reset_env(p, r, pick_scenario<PICK>(p, p.env_id_offset + e, ep), ep);
                c = 1.f; s = 0.f;
                hx = 0.5f * (p.ship_aabb[2] - p.ship_aabb[0]); hy = 0.5f * (p.ship_aabb[3] - p.ship_aabb[1]);
                {
                    float4 rg0, rg1, rg2;
                    float2 gn[kGoals];
                    scenario_goals(p, r.scen, rg0, rg1, rg2, gn);
                    closest_goal(gn, r.alive, r.x, r.y, gx, gy);
                    if (gl == 0) {
                        sts4(EA(GOL), rg0); sts4(EA(GOL + 1), rg1);
                        sts4(EA(GOL + 2), make_float4(rg2.x, rg2.y, __int_as_float((1 << kGoals) - 1), __int_as_float(ep)));
                    }
                    // the goal planes of the state change only here: written at once (a "goals changed" flag carried
                    // to the end of the kernel had been spilled to local memory and reloaded every iteration)
                    if (leader) store_goals(p, e, rg0, rg1, rg2);
                }
                if (gl == 0) {              // the spawn pose's planes were evaluated when the scenario was loaded
                    const float4 *sp = p.spawn_rows + (size_t)r.scen * kScr4;
                    const float4 h0 = __ldg(sp);
                    const int hn = __float_as_int(h0.z);
                    const int nrow = (hn & kHdrBig) ? 2 : 2 * (hn & 0xff);
                    sts4(EA(SCR), h0);
                    for (int i = 1; i <= nrow; ++i) sts4(EA(SCR + i), __ldg(sp + i));
                }
            }
        }
        if (live && gl == 0) {
            // ---- this step's observation frame.  The leader completes the newest frame in the resident tile (the lidar
            // slots are already there) BEFORE the pose moves on, so that no copy of this step's pose has to be kept.
            if (do_reset) {                                     // ship_env.py:180-184: [-1 x 16 | reset frame], vals = -1
                const float4 neg = make_float4(-1.f, -1.f, -1.f, -1.f);
                if (HIST == 2) {
#pragma unroll
                    for (int i = 0; i < FR4; ++i) sts4(EA(i), neg);
                }
                sts4(EA(NF), make_float4(r.x, r.y, 0.f, r.th));             // rudder 0 (models.py:108)
                sts4(EA(NF + 1), make_float4(gx, gy, -1.f, -1.f));
#pragma unroll
                for (int i = 2; i < FR4; ++i) sts4(EA(NF + i), neg);
            } else {                            // the rudder slot already holds this step's angle
                sts2(EA(NF), make_float2(r.x, r.y));
                sts1(EA(NF) + 12, r.th);
                sts2(EA(NF + 1), make_float2(gx, gy));
            }
        }
        // ---- cpSpaceStep of the NEXT step, positions first (cpBodyUpdatePosition).  Done before this step's copy-out
        // so that the grid cell of the new pose is requested as early as possible: it is consumed an iteration later.
        if (k + 1 < p.K) {
            r.x += r.vx * p.dt;
            r.y += r.vy * p.dt;
            r.th += r.w * p.dt;
            sincos_fast(r.th, s, c);
            hull_half_extents(p, c, s, hx, hy);
            if (G == 1 || gl == 0) fetch_cell_async(p, r.scen, r.x + hx, r.y + hy, EA(CEL));
        }
        if (live) {
            // ---- outputs: obs rows of the warp's envs are contiguous in global memory, so the tile is copied out with
            // fully coalesced 128-bit streaming stores.
            __syncwarp();
            if (WIDE) {
                // Rows of R = (6 + n) * HIST floats are dense in global memory and in general not 16-byte aligned, so the
                // warp's EPW rows go out as one run of 32-bit streaming stores, lane l taking floats l, l + 32, ... of
                // it.  (row, col) of a lane's float moves on by 32 floats per round: 32 / R rows and 32 % R columns.
                // A store is real iff it lies before the end of this step's rows (as below).
                if (p.obs) {
                    const int F = 6 + nb, R = F * HIST;
                    const int drow = 32 / R, dcol = 32 - drow * R;
                    int row = lane / R, col = lane - row * R;
                    float *o = reinterpret_cast<float *>(p.obs) + ((size_t)k * p.N + (e - grp)) * R + lane;
                    const float *o_end = reinterpret_cast<const float *>(p.obs) + (size_t)(k + 1) * p.N * R;
#pragma unroll 1
                    for (int i = lane; i < EPW * R; i += 32) {
                        // tile float of row column col: the older frame's F values, then the newest frame's
                        const int tc = col < F ? col : col + (4 * FR4 - F);
                        if (o < o_end) __stcs(o, lds1(WA(row, 0) + 4u * (unsigned)tc));
                        o += 32;
                        row += drow; col += dcol;
                        if (col >= R) { col -= R; ++row; }
                    }
                }
            } else if (p.obs && lane < EPW * OBS4) {
                // lane -> (row lane / OBS4, column lane % OBS4), each further round moves 32 / OBS4 rows down.  A round is
                // real iff its row belongs to an env of this batch, i.e. iff its address lies before the end of this step's
                // rows (tested against the step's end pointer, which moves with k: a loop-invariant row limit was hoisted,
                // spilled and reloaded from local memory right here in every iteration)
                const unsigned cp_src = WA(lane / OBS4, lane % OBS4);
                float4 *o = p.obs + ((size_t)k * p.N + (e - grp)) * OBS4 + lane;
                const float4 *o_end = p.obs + (size_t)(k + 1) * p.N * OBS4;
#pragma unroll
                for (int i = 0; i < (EPW * OBS4 >= 32 ? EPW * OBS4 / 32 : 1); ++i)
                    if (o + i * 32 < o_end) __stcs(o + i * 32, lds4(cp_src + i * (32 / OBS4) * (EB4 * 16)));
            }
            if (leader) {
                const size_t row = (size_t)k * p.N + e;
                if (p.reward) p.reward[row] = reward;
                if (p.done) p.done[row] = done ? 1 : 0;
            }
        }
        __syncwarp();                           // copy-out done and plane rows complete before the next iteration
    }
    // the loop leaves the pose of the last step in r (no integration after it)
    if (leader) {
        r.episode = __float_as_int(lds1(EA(GOL + 2) + 12));
        r.alive = __float_as_int(lds1(EA(GOL + 2) + 8));
        r.rudder = (int)lds1(EA(NF) + 8);
        store_env_frame(p, e, r, RowSmem{EA(NF)});
        if (WIDE) {
            const int nx = extra_lidar_planes(nb);
            for (int q = 0; q < nx; ++q) p.state[(size_t)(kPlanes + q) * p.N + e] = lds4(EA(NF + 4 + q));
        }
    }
    flush_stats(p, lane, RowSmem{wb + STA * 16});
#undef EA
#undef WA
}

// plane phase at the spawn pose of every scenario (what a reset env starts from), one thread per scenario
__global__ void __launch_bounds__(128) build_spawn_rows_kernel(const __grid_constant__ StepParams p, float4 *rows)
{
    const int sidx = blockIdx.x * blockDim.x + threadIdx.x;
    if (sidx >= p.n_scen) return;
    float4 *row = rows + (size_t)sidx * kScr4;
    for (int i = 0; i < kScr4; ++i) row[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    const float hx = 0.5f * (p.ship_aabb[2] - p.ship_aabb[0]), hy = 0.5f * (p.ship_aabb[3] - p.ship_aabb[1]);
    const uint4 cell = load_cell(p, sidx, p.spawn_x + hx, p.spawn_y + hy);
    if ((cell.x | cell.y | (cell.z & 3u)) != 0u) plane_phase<false, false>(p, p.spawn_x, p.spawn_y, hx, hy, 1.f, 0.f, sidx, cell, RowPtr{row}, RowPtr{nullptr});
    else row[0] = make_float4(1.f, 0.f, 0.f, 0.f);
}

// ------------------------------------------------------------------------------------------------------------
// reach-grid build kernel: one thread per (scenario, cell), double precision.  Runs once per scenario upload.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double point_rect_dist(double px, double py, double x0, double y0, double x1, double y1)
{
    const double dx = fmax(fmax(x0 - px, px - x1), 0.0), dy = fmax(fmax(y0 - py, py - y1), 0.0);
    return sqrt(dx * dx + dy * dy);
}

__device__ __forceinline__ double point_seg_dist(double px, double py, double ax, double ay, double bx, double by)
{
    const double ex = bx - ax, ey = by - ay;
    const double den = ex * ex + ey * ey;
    double t = den > 0.0 ? ((px - ax) * ex + (py - ay) * ey) / den : 0.0;
    t = fmin(fmax(t, 0.0), 1.0);
    const double dx = px - (ax + t * ex), dy = py - (ay + t * ey);
    return sqrt(dx * dx + dy * dy);
}

// distance between the segment a-b and the axis-aligned rectangle [x0,x1] x [y0,y1] (0 when they intersect)
__device__ double seg_rect_dist(double ax, double ay, double bx, double by, double x0, double y0, double x1, double y1)
{
    {   // Liang-Barsky: does any part of the segment lie inside the rectangle?
        double t0 = 0.0, t1 = 1.0;
        const double dx = bx - ax, dy = by - ay;
        const double pp[4] = {-dx, dx, -dy, dy};
        const double qq[4] = {ax - x0, x1 - ax, ay - y0, y1 - ay};
        bool inside = true;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (pp[i] == 0.0) { if (qq[i] < 0.0) inside = false; }
            else {
                const double t = qq[i] / pp[i];
                if (pp[i] < 0.0) t0 = fmax(t0, t); else t1 = fmin(t1, t);
            }
        }
        if (inside && t0 <= t1) return 0.0;
    }
    double d = fmin(point_rect_dist(ax, ay, x0, y0, x1, y1), point_rect_dist(bx, by, x0, y0, x1, y1));
    d = fmin(d, point_seg_dist(x0, y0, ax, ay, bx, by));
    d = fmin(d, point_seg_dist(x1, y0, ax, ay, bx, by));
    d = fmin(d, point_seg_dist(x0, y1, ax, ay, bx, by));
    d = fmin(d, point_seg_dist(x1, y1, ax, ay, bx, by));
    return d;
}

__global__ void __launch_bounds__(256) build_grid_kernel(const double *hull_xy, const int *hull_n, int n_scen, int maxv_in,
                                                         double gx0, double gy0, double cw, double ch, double reach,
                                                         double touch_margin, uint4 *grid)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)n_scen * kGridN * kGridN) return;
    const int s = (int)(t / (kGridN * kGridN)), cidx = (int)(t % (kGridN * kGridN));
    const int ix = cidx % kGridN, iy = cidx / kGridN;
    const double kBig = 1.0e12;
    const bool border = ix == 0 || iy == 0 || ix == kGridN - 1 || iy == kGridN - 1;
    const double x0 = ix == 0 ? -kBig : gx0 + ix * cw, x1 = ix == kGridN - 1 ? kBig : gx0 + (ix + 1) * cw;
    const double y0 = iy == 0 ? -kBig : gy0 + iy * ch, y1 = iy == kGridN - 1 ? kBig : gy0 + (iy + 1) * ch;
    // a finite point of the cell (used when no edge comes near: the cell is then entirely inside or outside)
    const double px = ix == 0 ? x1 : x0, py = iy == 0 ? y1 : y0;
    unsigned masks[2] = {0u, 0u}, flags = 0u;
    for (int b = 0; b < 2; ++b) {
        const double *v = hull_xy + ((size_t)s * 2 + b) * maxv_in * 2;
        const int n = hull_n[s * 2 + b];
        bool touch = false, pin = true;
        for (int i = 0; i < n; ++i) {
            const int j = i == 0 ? n - 1 : i - 1;
            const double ax = v[2 * j], ay = v[2 * j + 1], bx = v[2 * i], by = v[2 * i + 1];
            const double d = seg_rect_dist(ax, ay, bx, by, x0, y0, x1, y1);
            if (d <= reach) masks[b] |= 1u << i;
            if (d <= touch_margin) touch = true;
            // outward normal of a CCW loop is (ey, -ex): p is inside iff it is behind every plane
            if ((by - ay) * (px - bx) - (bx - ax) * (py - by) > 0.0) pin = false;
        }
        if (touch || pin) {
            flags |= 1u << b;
            if (border) masks[b] = n >= 32 ? kFull : ((1u << n) - 1u);      // unbounded cell: the inside test needs every plane
        }
    }
    // w: the first (up to) four candidates as bytes, bank * kMaxHull + edge, in the order the plane phase evaluates them
    // (bank 0 first, ascending edge index); 0xff = none.  z bits 8..15: the number of candidates.
    unsigned list = 0xffffffffu;
    int cnt = 0;
    for (int b = 0; b < 2; ++b)
        for (unsigned m = masks[b]; m; m &= m - 1u) {
            if (cnt < 4) list = (list & ~(0xffu << (8 * cnt))) | ((unsigned)(b * kMaxHull + (__ffs(m) - 1)) << (8 * cnt));
            ++cnt;
        }
    grid[t] = make_uint4(masks[0], masks[1], flags | ((unsigned)cnt << 8), list);
}

// ------------------------------------------------------------------------------------------------------------
// reset kernel: ShipEnv.reset for the masked envs (ship_env.py:171-184)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) reset_kernel(const __grid_constant__ StepParams p, const uint8_t *mask,
                                                    const int *scenario, int first, float4 *obs)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.N) return;
    if (mask && !mask[e]) return;
    EnvRegs r;
    float4 l0, l1, l2, g0, g1, g2;
    load_env(p, e, r, l0, l1, l2, g0, g1, g2);
    const int ep = first ? 0 : r.episode + 1;
    int scen = scenario ? scenario[e] : p.pick_cdf ? pick_scenario<true>(p, p.env_id_offset + e, ep) : pick_scenario<false>(p, p.env_id_offset + e, ep);
    scen = min(max(scen, 0), p.n_scen - 1);       // caller-supplied ids index the bank: never out of range (the host layer raises first)
    reset_env(p, r, scen, ep);
    float2 g[kGoals];
    float gx, gy;
    scenario_goals(p, scen, g0, g1, g2, g);
    closest_goal(g, r.alive, r.x, r.y, gx, gy);
    const float4 neg4 = make_float4(-1.f, -1.f, -1.f, -1.f);      // models.py:36: LiDAR.vals start at -1
    store_env(p, e, r, neg4, neg4, -1.f, -1.f);
    for (int q = 0; q < extra_lidar_planes(p.n_beams); ++q) p.state[(size_t)(kPlanes + q) * p.N + e] = neg4;
    store_goals(p, e, g0, g1, g2);
    if (obs) {                                  // rows of (6 + n) * history floats: [-1 x (6 + n) | x, y, 0, 0, gx, gy, -1 x n]
        const int F = 6 + p.n_beams;
        float *o = reinterpret_cast<float *>(obs) + (size_t)e * F * p.history;
        if (p.history == 2) {
            for (int i = 0; i < F; ++i) o[i] = -1.f;
            o += F;
        }
        o[0] = r.x; o[1] = r.y; o[2] = 0.f; o[3] = 0.f; o[4] = gx; o[5] = gy;
        for (int i = 6; i < F; ++i) o[i] = -1.f;
    }
}

// After a bank swap (shipsim_load_scenarios / shipsim_generate_scenarios on a live handle) a stored scenario id may
// exceed the new bank: fold it into range so that no kernel indexes bank / grid / edges_d / spawn_rows out of bounds.
// (The env keeps its old goals until its next reset; the host layer resets the whole batch after a swap.)
__global__ void __launch_bounds__(256) clamp_scenarios_kernel(float4 *state, int N, int n_scen)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    float4 *q = state + (size_t)4 * N + e;
    const int scen = __float_as_int(q->z);
    if (scen < 0 || scen >= n_scen) q->z = __int_as_float((int)((unsigned)scen % (unsigned)n_scen));
}

// the observation frame of the CURRENT state of every env (ShipEnv.__add_states, ship_env.py:79-113): what the next
// step will report as its "previous" frame.  Used by shipsim_step_host, which ships frames and rebuilds the history.
__global__ void __launch_bounds__(256) frame_kernel(const __grid_constant__ StepParams p, float4 *out)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.N) return;
    EnvRegs r;
    float4 l0, l1, l2, g0, g1, g2;
    load_env(p, e, r, l0, l1, l2, g0, g1, g2);
    float2 g[kGoals];
    unpack_goals(g0, g1, g2, g);
    float gx, gy;
    closest_goal(g, r.alive, r.x, r.y, gx, gy);
    store_frame(RowPtr{out + (size_t)e * 4}, r, gx, gy, l0, l1, l2);
}

// ------------------------------------------------------------------------------------------------------------
// Lossless compaction of a chunk of frames for the host path (shipsim_step_host): 64 + 5 bytes per env-step shrink to
// ~20, which is what crosses PCIe.  Between consecutive frames of an env the pose changes every step, everything else
// rarely: rudder / reward / done are a handful of states, the nearest goal switches now and then, a lidar reading only
// when its ray hits.  Per env-step the kernel emits one 16-byte record
//     { x, y, angle, word }    word = rudder code | reward code << 3 | done << 5 | change mask << 8
// (change mask: bit j set <=> slot 4 + j of the frame -- gx, gy, lidar 0..9 -- differs bitwise from the env's previous
// frame) and appends the changed values to a variable-length stream; off[k][block] = where the values of the 32 envs
// of a block start at step k (the blocks' order in the stream is whatever the atomics made it: the table is the truth).
// One warp per (step, 32-env block), blocks blk0 and up (the envs below 32 * blk0 go home as complete rows by DMA:
// history_rows_kernel).  The host rebuilds the frames exactly (shipsim_host.cpp: expand_delta_rows).
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) compact_frames_kernel(const float4 *frames, const float4 *prev0, const float *rew, const uint8_t *done,
                                                             int N, int blk0, int kc, float step_penalty, uint4 *rec, unsigned *off, float *var,
                                                             unsigned var_cap, unsigned *counter)
{
    const int lane = threadIdx.x & 31;
    const int nblk = (N + 31) / 32, nb = nblk - blk0;
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= (long long)kc * nb) return;
    const int k = (int)(w / nb), blk = blk0 + (int)(w % nb);
    const int e = blk * 32 + lane;
    const bool valid = e < N;
    unsigned mask = 0u;
    float vals[12];
    uint4 r = make_uint4(0u, 0u, 0u, 0u);
    if (valid) {
        const float4 *f = frames + ((size_t)k * N + e) * 4;
        const float4 *q = k > 0 ? f - (size_t)N * 4 : prev0 + (size_t)e * 4;
        const float4 f0 = f[0], f1 = f[1], f2 = f[2], f3 = f[3];
        const float4 q1 = q[1], q2 = q[2], q3 = q[3];
        const float nv[12] = {f1.x, f1.y, f1.z, f1.w, f2.x, f2.y, f2.z, f2.w, f3.x, f3.y, f3.z, f3.w};
        const float ov[12] = {q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w, q3.x, q3.y, q3.z, q3.w};
#pragma unroll
        for (int j = 0; j < 12; ++j) {
            vals[j] = nv[j];
            if (__float_as_uint(nv[j]) != __float_as_uint(ov[j])) mask |= 1u << j;
        }
        const float rw = rew[(size_t)k * N + e];
        const unsigned rcode = rw == 1.f ? 1u : (rw == -1.f ? 2u : (rw == step_penalty ? 0u : 3u));     // 3 never happens
        const unsigned rud = (unsigned)((int)f0.z / 5 + 2) & 7u;
        r = make_uint4(__float_as_uint(f0.x), __float_as_uint(f0.y), __float_as_uint(f0.w),
                       rud | (rcode << 3) | ((done[(size_t)k * N + e] ? 1u : 0u) << 5) | (mask << 8));
        rec[(size_t)k * N + e] = r;
    }
    const int n = __popc(mask);
    int incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += v;
    }
    const int total = __shfl_sync(kFull, incl, 31);
    unsigned base = 0u;
    if (lane == 0) {
        base = total ? atomicAdd(counter, (unsigned)total) : 0u;
        off[(size_t)k * nblk + blk] = base;
    }
    base = __shfl_sync(kFull, base, 0);
    unsigned at = base + (unsigned)(incl - n);
#pragma unroll
    for (int j = 0; j < 12; ++j)
        if ((mask >> j) & 1u) {
            if (at < var_cap) var[at] = vals[j];        // (beyond the capacity: dropped; the host sees counter > capacity)
            ++at;
        }
}

// Complete observation rows [previous frame | frame] of the envs [0, nd) for a chunk of frames (ship_env.py:112-113;
// 16 x -1 as the previous frame of a step that ended an episode under auto-reset, ship_env.py:180-184): the part of the
// host path's output that travels as plain rows by DMA while the host threads expand the compacted part.  One thread per
// quarter frame; rows[kc][nd][32].
__global__ void __launch_bounds__(256) history_rows_kernel(const float4 *frames, const float4 *prev0, const uint8_t *done, int N, int nd,
                                                           int kc, int cut, float4 *rows)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)kc * nd * 4) return;
    const int q = (int)(t & 3);
    const long long ke = t >> 2;
    const int k = (int)(ke / nd), e = (int)(ke % nd);
    const size_t at = ((size_t)k * N + e) * 4 + q;
    const float4 cur = frames[at];
    float4 prev = k > 0 ? frames[at - (size_t)N * 4] : prev0[(size_t)e * 4 + q];
    if (cut && done[(size_t)k * N + e]) prev = make_float4(-1.f, -1.f, -1.f, -1.f);
    float4 *o = rows + (size_t)ke * 8 + q;
    __stcs(o, prev);
    __stcs(o + 4, cur);
}

// Episode log on the frames-only path of shipsim_step_host, where the step kernel runs in its one-frame mode and puts the
// terminal frame into the second half of a record's row: the first half, the env's previous frame, comes from the chunk's
// frames (prev0 = the frames before the chunk's first step).  One thread per record slot; only the records of call
// `call` whose step lies in this chunk are touched.
__global__ void __launch_bounds__(256) log_prev_frames_kernel(const float4 *frames, const float4 *prev0, int N, int k0, int kc, int call,
                                                              float4 *rows, const int4 *meta, const int *count, int cap)
{
    const int n = min(*count, cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int4 m0 = meta[2 * (size_t)i], m1 = meta[2 * (size_t)i + 1];
        if (m1.w != call || m0.x < k0 || m0.x >= k0 + kc) continue;
        const int kk = m0.x - k0, e = m0.y;
        const float4 *src = kk > 0 ? frames + ((size_t)(kk - 1) * N + e) * 4 : prev0 + (size_t)e * 4;
#pragma unroll
        for (int q = 0; q < 4; ++q) rows[(size_t)i * 8 + q] = src[q];
    }
}

// stats slots -> out[kStatLen]; one warp per statistic column
__global__ void stats_reduce_kernel(double *slots, double *out, int clear)
{
    const int col = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double acc = 0.0;
    for (int s = lane; s < kStatSlots; s += 32) {
        acc += slots[s * kStatLen + col];
        if (clear) slots[s * kStatLen + col] = 0.0;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(kFull, acc, off);
    if (lane == 0) out[col] = acc;
}

// Table of the weighted scenario picks (pick_weighted) from w[n]: cdf[0, n) = inclusive prefix sums, cdf[n] = total, and
// guide[j] = first i with cdf[i] > floor(j * total / n), guide[n] = n - 1.  A total of 0 or of 2^32 and more is stored as
// 0 ("uniform"), and the rest is left as it was.  One CTA walks the bank a tile at a time (banks reach 2^28 maps): the
// total in 64 bits first, then per tile a block-wide scan, and element i hands its guide entries -- the j with
// floor(j * total / n) in [cdf[i - 1], cdf[i]), i.e. j in [ceil(cdf[i - 1] * n / total), ceil(cdf[i] * n / total)) -- to
// its whole warp to write, so that one heavy weight does not leave a single thread filling most of the guide.
constexpr int kPickThreads = 1024;
__global__ void __launch_bounds__(kPickThreads) build_pick_table_kernel(const unsigned *w, int n, unsigned *cdf, unsigned *guide)
{
    __shared__ unsigned long long s_sum[kPickThreads / 32];
    __shared__ unsigned s_scan[kPickThreads / 32];
    __shared__ unsigned s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned long long acc = 0ull;
    for (int i = tid; i < n; i += kPickThreads) acc += __ldg(w + i);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(kFull, acc, off);
    if (lane == 0) s_sum[warp] = acc;
    __syncthreads();
    if (warp == 0) {
        acc = s_sum[lane];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(kFull, acc, off);
        if (lane == 0) { s_sum[0] = acc; s_carry = 0u; }
    }
    __syncthreads();
    const unsigned long long total = s_sum[0];
    if (total == 0ull || total >= (1ull << 32)) {
        if (tid == 0) cdf[n] = 0u;
        return;
    }
    if (tid == 0) { cdf[n] = (unsigned)total; guide[n] = (unsigned)(n - 1); }
    for (int base = 0; base < n; base += kPickThreads) {
        const int i = base + tid;
        const unsigned v = i < n ? __ldg(w + i) : 0u;
        unsigned x = v;                                          // inclusive scan within the warp ...
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const unsigned y = __shfl_up_sync(kFull, x, off);
            if (lane >= off) x += y;
        }
        if (lane == 31) s_scan[warp] = x;
        __syncthreads();
        if (warp == 0) {                                         // ... of the warp totals ...
            unsigned s = s_scan[lane];
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const unsigned y = __shfl_up_sync(kFull, s, off);
                if (lane >= off) s += y;
            }
            s_scan[lane] = s;
        }
        __syncthreads();
        const unsigned incl = s_carry + (warp ? s_scan[warp - 1] : 0u) + x;     // ... and of the tiles before (< 2^32)
        const unsigned excl = incl - v;
        __syncthreads();                                         // every thread has read s_carry and s_scan
        if (tid == kPickThreads - 1) s_carry = incl;
        if (i < n) cdf[i] = incl;
        unsigned j0 = 0u, j1 = 0u;
        if (i < n) {
            j0 = (unsigned)(((unsigned long long)excl * (unsigned)n + total - 1ull) / total);
            j1 = (unsigned)(((unsigned long long)incl * (unsigned)n + total - 1ull) / total);
        }
        for (unsigned m = __ballot_sync(kFull, j1 > j0); m; m &= m - 1u) {
            const int src = __ffs(m) - 1;
            const unsigned a = __shfl_sync(kFull, j0, src), b = __shfl_sync(kFull, j1, src);
            const unsigned val = (unsigned)(base + warp * 32 + src);
            for (unsigned k = a + lane; k < b; k += 32u) guide[k] = val;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// launch wrappers (called from the C ABI)
// ------------------------------------------------------------------------------------------------------------
template <int G, int HIST, int MB, int T, int NB>
static cudaError_t launch_gh(const StepParams &p, int blocks, cudaStream_t stream)
{
    void (*const kern)(StepParams) =
        p.log_count ? (p.pick_cdf ? step_kernel<G, HIST, MB, T, true, NB, true> : step_kernel<G, HIST, MB, T, true, NB, false>)
                    : (p.pick_cdf ? step_kernel<G, HIST, MB, T, false, NB, true> : step_kernel<G, HIST, MB, T, false, NB, false>);
    if constexpr (NB == kBeams) {
        kern<<<blocks, T, 0, stream>>>(p);
    } else {
        // the wide kernel's shared memory is dynamic: up to 68 KB per CTA (G = 1, 128 threads, HISTORY_SIZE 2), beyond the
        // 48 KB a launch gets without asking -- the opt-in is made once per instantiation and device
        constexpr int bytes = StepLayout<G, HIST, NB, T>::BYTES;
        if (bytes > 48 * 1024) {
            static std::atomic<unsigned long long> opted[4] = {};
            const int which = (p.log_count ? 1 : 0) + (p.pick_cdf ? 2 : 0);
            int dev = 0;
            cudaError_t err = cudaGetDevice(&dev);
            if (err != cudaSuccess) return err;
            const unsigned long long bit = 1ull << (dev & 63);
            if (!(opted[which].load() & bit)) {
                err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
                if (err != cudaSuccess) return err;
                opted[which].fetch_or(bit);
            }
        }
        kern<<<blocks, T, bytes, stream>>>(p);
    }
    return cudaSuccess;
}

template <int G, int NB>
static cudaError_t launch_g(const StepParams &p, cudaStream_t stream, LaunchShape *shape)
{
    const int envs_per_cta = kThreads / G;
    int blocks = (p.N + envs_per_cta - 1) / envs_per_cta;
    int threads = kThreads;
    bool launched = false;
    cudaError_t err = cudaSuccess;
    if constexpr (G == 1) {
        if (blocks >= 148 * 8) {
            threads = kBigThreads;
            blocks = (p.N + threads - 1) / threads;
            if (p.history == 2) err = launch_gh<G, 2, kBigMinBlocks, kBigThreads, NB>(p, blocks, stream);
            else err = launch_gh<G, 1, kBigMinBlocks, kBigThreads, NB>(p, blocks, stream);
            launched = true;
        }
    }
    if (!launched) {
        // Grids that do not fill the machine: 64-thread CTAs (same 16 warps per SM at 128 registers), so that the few
        // CTAs spread evenly -- 65,536 envs are 512 CTAs of 128 threads, 3.46 per SM: every SM waits for the ones that got 4
        constexpr int T = kSmallThreads, MB = kMinBlocks * kThreads / kSmallThreads;
        threads = T;
        blocks = (p.N + T / G - 1) / (T / G);
        if (p.history == 2) err = launch_gh<G, 2, MB, T, NB>(p, blocks, stream);
        else err = launch_gh<G, 1, MB, T, NB>(p, blocks, stream);
    }
    if (shape) { shape->lanes_per_env = G; shape->threads = threads; shape->blocks = blocks; shape->window = 1; }
    return err != cudaSuccess ? err : cudaGetLastError();
}

template <int NB>
static cudaError_t launch_step_nb(const StepParams &p, int lanes_per_env, cudaStream_t stream, LaunchShape *shape)
{
    switch (lanes_per_env) {
        case 1: return launch_g<1, NB>(p, stream, shape);
        case 2: return launch_g<2, NB>(p, stream, shape);
        case 4: return launch_g<4, NB>(p, stream, shape);
        case 8: return launch_g<8, NB>(p, stream, shape);
        case 16: return launch_g<16, NB>(p, stream, shape);
        case 32: return launch_g<32, NB>(p, stream, shape);
        default: return cudaErrorInvalidValue;
    }
}

// the reference's 10-beam fan runs the tuned kernels; every other beam count (1..32) the wide ones
cudaError_t launch_step(const StepParams &p, int lanes_per_env, cudaStream_t stream, LaunchShape *shape)
{
    if (p.n_beams == kBeams) return launch_step_nb<kBeams>(p, lanes_per_env, stream, shape);
    if (p.n_beams < 1 || p.n_beams > kMaxBeams) return cudaErrorInvalidValue;
    return launch_step_nb<kMaxBeams>(p, lanes_per_env, stream, shape);
}

cudaError_t launch_reset(const StepParams &p, const uint8_t *mask, const int *scenario, int first, float4 *obs,
                         cudaStream_t stream)
{
    const int threads = 256;
    reset_kernel<<<(p.N + threads - 1) / threads, threads, 0, stream>>>(p, mask, scenario, first, obs);
    return cudaGetLastError();
}

cudaError_t launch_clamp_scenarios(float4 *state, int N, int n_scen, cudaStream_t stream)
{
    clamp_scenarios_kernel<<<(N + 255) / 256, 256, 0, stream>>>(state, N, n_scen);
    return cudaGetLastError();
}

cudaError_t launch_compact_frames(const float4 *frames, const float4 *prev0, const float *rew, const uint8_t *done, int N, int env0, int kc,
                                  float step_penalty, uint4 *rec, unsigned *off, float *var, unsigned var_cap, unsigned *counter,
                                  cudaStream_t stream)
{
    const long long warps = (long long)kc * ((N + 31) / 32 - env0 / 32);
    if (warps <= 0) return cudaSuccess;
    compact_frames_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, stream>>>(frames, prev0, rew, done, N, env0 / 32, kc, step_penalty,
                                                                                   rec, off, var, var_cap, counter);
    return cudaGetLastError();
}

cudaError_t launch_history_rows(const float4 *frames, const float4 *prev0, const uint8_t *done, int N, int nd, int kc, int cut, float4 *rows,
                                cudaStream_t stream)
{
    const long long threads = (long long)kc * nd * 4;
    if (threads <= 0) return cudaSuccess;
    history_rows_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(frames, prev0, done, N, nd, kc, cut, rows);
    return cudaGetLastError();
}

cudaError_t launch_frame(const StepParams &p, float4 *out, cudaStream_t stream)
{
    frame_kernel<<<(p.N + 255) / 256, 256, 0, stream>>>(p, out);
    return cudaGetLastError();
}

cudaError_t launch_build_grid(const double *hull_xy, const int *hull_n, int n_scen, int maxv_in, double gx0, double gy0,
                              double cw, double ch, double reach, double touch_margin, uint4 *grid, cudaStream_t stream)
{
    const long long total = (long long)n_scen * kGridN * kGridN;
    build_grid_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(hull_xy, hull_n, n_scen, maxv_in, gx0, gy0, cw, ch,
                                                                          reach, touch_margin, grid);
    return cudaGetLastError();
}

cudaError_t launch_build_spawn_rows(const StepParams &p, float4 *rows, cudaStream_t stream)
{
    build_spawn_rows_kernel<<<(p.n_scen + 127) / 128, 128, 0, stream>>>(p, rows);
    return cudaGetLastError();
}

cudaError_t launch_log_prev_frames(const StepParams &p, const float4 *frames, const float4 *prev0, int k0, int kc, cudaStream_t stream)
{
    const int blocks = p.log_cap < 1184 * 256 ? (p.log_cap + 255) / 256 : 1184;
    log_prev_frames_kernel<<<blocks, 256, 0, stream>>>(frames, prev0, p.N, k0, kc, p.log_call, p.log_rows, p.log_meta, p.log_count, p.log_cap);
    return cudaGetLastError();
}

cudaError_t launch_build_pick_table(const unsigned *weights, int n_scen, unsigned *table, cudaStream_t stream)
{
    build_pick_table_kernel<<<1, kPickThreads, 0, stream>>>(weights, n_scen, table, table + n_scen + 1);
    return cudaGetLastError();
}

cudaError_t launch_stats_reduce(double *slots, double *out, int clear, cudaStream_t stream)
{
    stats_reduce_kernel<<<1, 32 * kStatLen, 0, stream>>>(slots, out, clear);
    return cudaGetLastError();
}

}  // namespace shipsim
