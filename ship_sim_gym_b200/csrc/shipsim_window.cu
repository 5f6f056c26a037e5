// shipsim_window.cu -- time-parallel ("window") variant of the fused ShipEnv step kernel, for latency-bound batches.
// sm_100a only.  Same transition as step_kernel (shipsim_kernels.cu; SURVEY.md Appendix A), same helper functions
// (shipsim_geom.cuh), bit-identical results (tests/test_gpu_window.py).
//
// Why.  With few envs per SM (4,096 envs = 28 per SM) a K-step rollout is a chain of K dependent iterations and the
// machine idles on instruction latency.  But only the cheap part of a step is sequential: the rigid-body recurrence
// (cpBodyUpdatePosition / cpBodyUpdateVelocity: ~10 flops) and the rudder clamp.  Everything expensive -- the lidar
// query, the ship-vs-bank overlap test, the goal tests, the observation frame -- is a pure function of one pose and
// feeds back into the trajectory only through `done` (auto-reset).  So, when the actions of the rollout are known up
// front (they are: shipsim_step takes the whole [K][N] action tensor), T consecutive steps of one env are SPECULATED:
//   1. the sequential part runs as two short scans executed by every lane of the env's group in lockstep (no
//      divergence, no waiting): rudder / angular velocity / angle from pre-decoded actions, then ONE sincos per lane,
//      then velocity / position with the thrust terms broadcast through shared memory; the group's first lane drops
//      each step's result into shared memory and lane t = lane % T picks up the pose of "its" step;
//   2. lane t does the pose-dependent work of step t -- reach-grid lookup, plane phase, goal tests, out-of-bounds --
//      and the cooperative ray / separating-axis passes run over (env, step) pairs instead of envs;
//   3. the sequential leftovers are resolved without loops over steps where possible: goals taken (one ballot per
//      goal), episode return (ordered per-lane prefix, same rounding as the serial kernel), sticky lidar readings
//      (models.py:71: a miss keeps the last hit -- per ray, the latest hitting lane at or before t, by ballot + clz);
//   4. the window is cut after the first `done`: steps beyond it are discarded, the env resets and the next window
//      starts from the reset state (episodes last ~48 steps on the default map, so a window of 16 commits 13.9 steps
//      on average).
// A warp holds E = 32/T envs; envs of a warp advance independently (each has its own step cursor k0).
//
// Shared memory per env: the plane-phase rows live in a ring of T+1 slots -- slot cb is the "carry", the planes of the
// last committed step (or of the reset), i.e. what step k0's lidar looks at; slot cb+1+t belongs to speculated step t;
// committing n steps just advances cb by n.  The observation frames sit in T+1 linear slots: slot 0 is the carry frame
// (rewritten after every window by the lane of the last committed step), slot 1+t the frame of step t, so that the
// copy-out addresses are compile-time offsets.
//   1. uses a log2(T)-round prefix for the integer rudder recurrence (clamped additions compose), not a T-step chain;
//   2. runs the separating-axis test per env group on the earliest undecided step and, with auto-reset, drops the steps
//      behind the first done; lidar queries are cast for committed steps only.
#include "shipsim_geom.cuh"
#include "shipsim_launch.h"

namespace shipsim {

constexpr int kWinThreads = 32;      // one-warp CTAs: a latency-bound batch is a few thousand warps, spread them evenly over the SMs (64 -> 32 threads: 0.460 -> 0.458 ms on the headline, -1.8 % at 2,048 envs)

// LOG: write the episode log (shipsim_episode_log_bind).  The log-free kernel is a separate instantiation: its registers
// and spills are those of the kernel before the log existed (-Xptxas -v; this kernel sits at the 128-register wall).
// PICK: weighted scenario picks (shipsim_scenario_weights), a separate instantiation for the same reason.
// CHAIN: a chained launch (shipsim_step_chained, log-free only).  Back-to-back launches of one handle each last as long
// as their slowest warp (a launch of the headline: CTA ends spread from 0.30 to 0.44 ms, a sixth of the warp-slot time
// idle), so a chained launch starts while the previous one still runs and each env waits for its own previous launch
// only, through two tickets per env:
//   * start: the env-group leader takes t = started[e]++, then -- once every ticket of the CTA is taken -- the CTA lets
//     the next launch start (griddepcontrol.launch_dependents), and the leader waits until done[e] reaches t before the
//     env's state is loaded;
//   * end: after the state, goal, obs, reward and done stores and the statistics flush, done[e] = max(done[e], t + 1)
//     with release semantics; then griddepcontrol.wait, so that launch N + 1 completes after launch N and everything
//     later on the stream sees both (by then N is long done: it costs nothing in steady state).
// Deadlock-free: a waiting CTA waits only for tickets taken earlier; a ticket is taken only by a CTA that is already
// running; that CTA waits only on smaller tickets; and launch N + 1 starts only after every CTA of launch N has triggered,
// i.e. is resident.  So the CTA that holds the smallest outstanding ticket is running and waits for nobody.
template <int T, int HIST, bool LOG, bool PICK, bool CHAIN>
__global__ void __launch_bounds__(kWinThreads, 512 / kWinThreads) window_kernel(const __grid_constant__ StepParams p)
{
    // The two physics scans are unrolled over the whole window when it is short (every load that feeds the chains is
    // then issued ahead of them: 4 -> 16 iterations per trip took the headline from 0.458 to 0.449 ms), by 4 for the
    // longest window (T = 32 fully unrolled is 9 % SLOWER at 2,048 envs: code size).
    constexpr int kScanUnroll = T <= 16 ? T : 4;
    constexpr int E = 32 / T;                   // envs per warp
    constexpr int NW = kWinThreads / 32;
    constexpr int OBS4 = 4 * HIST;              // float4 per obs row
    constexpr int NS = T + 1;                   // ring slots per env
    constexpr int FS4 = 5;                      // float4 per frame slot (4 used; odd stride: conflict-free)
    constexpr int FR4 = NS * FS4;               // float4 per env frame ring
    constexpr int SC4 = NS * kScr4;             // float4 per env plane-row ring
    constexpr float kMiss = -2.f;               // "this ray did not hit at this step" until the sticky scan resolves it
    __shared__ float4 s_frame[NW * E * FR4];
    __shared__ float4 s_scr[NW * E * SC4];
    __shared__ float2 s_goal[NW * E * kGoals];
    __shared__ float4 s_rf[NW * E * 2];         // reset frame, first two float4 (the rest is -1)
    __shared__ float4 s_ph[NW * 32 * 2];        // physics scan -> lanes: (th, w, bits(rudder), -) and (x, y, vx, vy) per step
    // lanes -> scans: every lane's torque term, thrust pair and reward, read back by its group as LDS.128 broadcasts
    // (4 torque terms, 2 thrust pairs or 4 rewards per load instead of one shuffle per value)
    __shared__ float4 s_dw[NW * 8], s_dv[NW * 16], s_rw[NW * 8];
    __shared__ int4 s_env[NW * E];              // per env, for the copy-out: step cursor, committed steps, (carry slot of the plane ring), reset?
    __shared__ float s_ray[2 * 32];
    __shared__ unsigned s_src[NW][32];          // ray pass: compacted (plane row | frame offset) of the needy steps
    __shared__ __align__(16) float s_stat[NW][8];   // (warp_stats reads and writes it as two float4)
    __shared__ unsigned s_ticket[CHAIN ? NW * E : 1];   // CHAIN: the ticket of each env of the CTA

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int el = lane / T, t = lane % T;
    const int gbase = el * T;                   // first lane of this env's group
    const unsigned segmask = T == 32 ? kFull : (((1u << T) - 1u) << gbase);
    const int warp_env0 = (blockIdx.x * NW + warp) * E;
    const int e = warp_env0 + el;
    const bool valid = e < p.N;
    const int ec = valid ? e : p.N - 1;         // lanes of idle groups shadow the last env; they never store
    const int wfr0 = warp * E * FR4, wsc0 = warp * E * SC4;
    const int fr0 = wfr0 + el * FR4, sc0 = wsc0 + el * SC4;
    const int goal0 = (warp * E + el) * kGoals;
    const int rf0 = (warp * E + el) * 2;
    const float L = p.lidar_len;
    const long long gid = p.env_id_offset + e;
#define stat (s_stat[warp])
    const unsigned stat_s = smem_addr(s_stat[warp]);
    auto ring = [](int s) { return s >= NS ? s - NS : s; };

    // lane roles in the cooperative passes (as in step_kernel)
    const int rslot = lane / kBeams;
    const int rj = lane - rslot * kBeams;
    if (threadIdx.x < 32) {
        s_ray[threadIdx.x] = p.ray_c[threadIdx.x % kBeams];
        s_ray[32 + threadIdx.x] = p.ray_s[threadIdx.x % kBeams];
    }
    if (lane < 8) stat[lane] = 0.f;
    // separating-axis pass: one step per env group at a time, lane t takes bank edges t, t + T, ...
    const int epl = (p.hull_max + T - 1) / T;

    const size_t act_esize = p.action_dtype == 1 ? 8 : (p.action_dtype == 2 ? 1 : 4);
    const char *act0 = reinterpret_cast<const char *>(p.actions) + (size_t)ec * act_esize;
    const size_t act_stride = (size_t)p.N * act_esize;

    if constexpr (CHAIN) {
        const bool lead = valid && t == 0;
        // (the shared store waits for the atomic's result: the CTA triggers with all its tickets taken)
        if (lead) s_ticket[warp * E + el] = atomicAdd(p.chain_started + e, 1u);
        __syncwarp();
        griddep_launch_dependents();
        if (lead) chain_await(p.chain_done + e, s_ticket[warp * E + el], e);
        __syncwarp();
    }

    EnvRegs r;
    int cb = 0;                                 // ring slot of the carry
    int k0 = 0;                                 // this env's next step
    bool goals_dirty = false;
    float c0, s0;                               // trig of the pose step k0 starts from
    {
        float4 l0, l1, l2, g0, g1, g2;
        load_env(p, ec, r, l0, l1, l2, g0, g1, g2);
        float2 g[kGoals];
        unpack_goals(g0, g1, g2, g);
        float gx, gy;
        closest_goal(g, r.alive, r.x, r.y, gx, gy);
        sincos_fast(r.th, s0, c0);
        if (t == 0) {
#pragma unroll
            for (int i = 0; i < kGoals; ++i) s_goal[goal0 + i] = g[i];
            store_frame(RowPtr{s_frame + fr0}, r, gx, gy, l0, l1, l2);     // carry frame = frame of the current state
            float hx, hy;                       // carry row = planes of the current pose
            hull_half_extents(p, c0, s0, hx, hy);
            const uint4 cell = load_cell(p, r.scen, r.x + hx, r.y + hy);
            float4 *row = s_scr + sc0;
            if ((cell.x | cell.y | (cell.z & 3u)) != 0u) plane_phase<false, false>(p, r.x, r.y, hx, hy, c0, s0, r.scen, cell, RowPtr{row}, RowPtr{nullptr});
            else row[0] = make_float4(c0, s0, 0.f, 0.f);
        }
    }
    // Actions are held one window ahead: a_my = action of step k0 + t, a_nx = action of step k0 + T + t.  After a window
    // that commits n steps the next window's actions are n lanes further along this pair (two shuffles); only the n
    // lanes at the far end load anything, and what they load is not looked at before the end of the next window.
    // The scenario of the NEXT episode depends only on (seed, env id, episode number): it is drawn an episode ahead, so
    // that at a reset the Philox rounds are not in front of the loads of the new scenario's goals and spawn row, and
    // every window pulls those few lines towards L1 in case it ends in a reset.
    constexpr int SPL = (kScr4 + T - 1) / T;    // spawn-row float4s per lane
    const unsigned pkey = pick_key(p, gid);
    int next_scen = pick_scenario_keyed<PICK>(p, pkey, r.episode + 1);
    int a_my = 3, a_nx = 3;
    if (valid && t < p.K) a_my = load_action(p, act0 + (size_t)t * act_stride, t, gid);
    if (valid && T + t < p.K) a_nx = load_action(p, act0 + (size_t)(T + t) * act_stride, T + t, gid);
    __syncthreads();

#pragma unroll 1
    while (true) {
        const int nvalid = valid ? min(T, p.K - k0) : 0;        // steps this env still has, capped by the window
        if (__ballot_sync(kFull, nvalid > 0) == 0u) break;
        const bool active = t < nvalid;
        // (Pays only for the longest window, where an SM holds few envs and a reset's loads are fully exposed: at 2,048 envs
        // +6 %; with T <= 16 the twelve prefetches and their addresses cost more than they hide: -1.2 % on the headline.)
        if (T >= 32 && p.auto_reset) {
#pragma unroll
            for (int i = 0; i < (3 + kScr4 + T - 1) / T; ++i) {
                const int q = t + i * T;
                if (q < 3) prefetch_l1(p.bank + (size_t)next_scen * p.scen_stride4 + 2 + q);
                else if (q < 3 + kScr4) prefetch_l1(p.spawn_rows + (size_t)next_scen * kScr4 + (q - 3));
            }
        }

        // ---- 1. the sequential part, T steps: handle_discrete_action (game.py:140-153), cpBodyUpdatePosition,
        // cpBodyUpdateVelocity -- the same operations in the same order as step_kernel, split so that as little as
        // possible is serial.  Every lane of the group runs the scans in lockstep (no divergence, no waiting); the
        // group's first lane drops each step's result into shared memory and lane t picks up step t.
        float mx, my, mth, mc, ms;
        int mrud;
        {
            float4 *ph = s_ph + (warp * 32 + gbase) * 2;
            // scan 1a: the rudder (Ship.rotate / clamp_rudder, models.py:136-146) is an integer recurrence
            // rud <- clamp(rud + inc, -10, 10).  Clamped additions are closed under composition --
            // min(max(r + a, lo), hi) followed by (a', lo', hi') is (a + a', max(lo + a', lo'), min(max(hi + a', lo'), hi'))
            // -- so the T rudder values of the window come from a log2(T)-round prefix over (a, lo, hi) instead of a
            // T-step chain; integers, hence exact.
            int rud_t;                                  // rudder after the action of step t
            {
                int fa = a_my == 1 ? -5 : (a_my == 2 ? 5 : 0), flo = -10, fhi = 10;
#pragma unroll
                for (int off = 1; off < T; off <<= 1) {
                    const int pa = __shfl_up_sync(kFull, fa, off, T), plo = __shfl_up_sync(kFull, flo, off, T),
                              phi = __shfl_up_sync(kFull, fhi, off, T);
                    if (t >= off) {                     // earlier steps first (pa, plo, phi), then this lane's
                        const int na = pa + fa, nlo = max(plo + fa, flo), nhi = min(max(phi + fa, flo), fhi);
                        fa = na; flo = nlo; fhi = nhi;
                    }
                }
                rud_t = min(max(r.rudder + fa, flo), fhi);
            }
            // scan 1b: angular velocity and angle.  Thrust (action 0) leaves the rudder alone, so the torque term of
            // step t uses rud_t; it is rounded to fp32 before the fused multiply-add, exactly as in step_kernel.
            {
                reinterpret_cast<float *>(s_dw)[warp * 32 + lane] = a_my == 0 ? -p.ang_dt * (float)rud_t : 0.f;
                __syncwarp();
                const float4 *dw4 = s_dw + (warp * 32 + gbase) / 4;
                float th = r.th, w = r.w;
                float2 *po = reinterpret_cast<float2 *>(ph);
#pragma unroll 1
                for (int i0 = 0; i0 < T; i0 += kScanUnroll) {
                    float dw[kScanUnroll];                      // the trip's torque terms, all loaded ahead of the chain
#pragma unroll
                    for (int j = 0; j < kScanUnroll; j += 4) {
                        const float4 d = dw4[(i0 + j) / 4];
                        dw[j] = d.x; dw[j + 1] = d.y; dw[j + 2] = d.z; dw[j + 3] = d.w;
                    }
#pragma unroll
                    for (int u = 0; u < kScanUnroll; ++u) {
                        th += w * p.dt;
                        w = w * p.damping + dw[u];
                        if (t == 0) *po = make_float2(th, w);
                        po += 4;
                    }
                }
            }
            __syncwarp();
            {
                const float2 v = *reinterpret_cast<const float2 *>(ph + 2 * t);
                mth = v.x; mrud = rud_t;
            }
            sincos_fast(mth, ms, mc);                   // one sincos per lane instead of T per lane
            // thrust of step t acts along the heading the step STARTS from: the trig of step t-1 (or of the carry)
            float pc = __shfl_up_sync(kFull, mc, 1, T), ps = __shfl_up_sync(kFull, ms, 1, T);
            if (t == 0) { pc = c0; ps = s0; }
            float2 dv_t = make_float2(0.f, 0.f);
            if (a_my == 0) dv_t = make_float2(-p.acc_dt * ps, p.acc_dt * pc);
            reinterpret_cast<float2 *>(s_dv)[warp * 32 + lane] = dv_t;
            __syncwarp();
            // scan 2: velocity and position, x and y as one pair.  x += vx * dt and vx = vx * damping + dvx each compile to
            // one contracted fma; __ffma2_rn (FFMA2) does two of them in one issue slot, each element rounded exactly as
            // by the scalar fma, so the results stay bit for bit those of step_kernel.  (ptxas does not pair scalar fmas.)
            {
                const float4 *dv4 = s_dv + (warp * 32 + gbase) / 2;
                const float2 dt2 = make_float2(p.dt, p.dt), damp2 = make_float2(p.damping, p.damping);
                float2 xy = make_float2(r.x, r.y), v = make_float2(r.vx, r.vy);
                unsigned po = smem_addr(ph + 1);
#pragma unroll 1
                for (int i0 = 0; i0 < T; i0 += kScanUnroll) {
                    float2 dv[kScanUnroll];                     // the trip's thrust terms, all loaded ahead of the chain
#pragma unroll
                    for (int j = 0; j < kScanUnroll; j += 2) {
                        const float4 d = dv4[(i0 + j) / 2];
                        dv[j] = make_float2(d.x, d.y); dv[j + 1] = make_float2(d.z, d.w);
                    }
#pragma unroll
                    for (int u = 0; u < kScanUnroll; ++u) {
                        xy = __ffma2_rn(v, dt2, xy);
                        v = __ffma2_rn(v, damp2, dv[u]);
                        // (two 8-byte stores that ptxas cannot merge: a 16-byte one wants (xy, v) in one register
                        // quad and costs four moves a step)
                        if (t == 0) { sts2(po, xy); sts2(po + 8, v); }
                        po += 32;
                    }
                }
            }
            __syncwarp();
            {
                const float4 v = ph[2 * t + 1];
                mx = v.x; my = v.y;
            }
        }

        // ---- 2. pose-dependent work of step t at (mx, my, mth): reach-grid cell, candidate planes staged by cp.async
        const int myslot_ring = ring(cb + 1 + t);
        float4 *myrow = s_scr + sc0 + myslot_ring * kScr4;
        float4 *myfr = s_frame + fr0 + (1 + t) * FS4;    // frames: slot 0 = carry, slot 1 + t = step t (no ring)
        float hx = 0.f, hy = 0.f;
        uint4 cell = make_uint4(0u, 0u, 0u, 0xffffffffu);
        if (active) {
            hull_half_extents(p, mc, ms, hx, hy);
            cell = load_cell(p, r.scen, mx + hx, my + hy);
        }

        // goals (collide_goal, game.py:243-257): which goals does the hull touch at this pose?  (whether they are
        // still alive is settled by the scan below)
        float2 g[kGoals];
        float gd2[kGoals];
        unsigned touch = 0u, cand = 0u;
        {
#pragma unroll
            for (int i = 0; i < kGoals; ++i) {
                g[i] = s_goal[goal0 + i];
                const float ux = g[i].x - mx, uy = g[i].y - my;
                gd2[i] = ux * ux + uy * uy;
            }
#pragma unroll
            for (int i = 0; i < kGoals; ++i)
                if (active && ((r.alive >> i) & 1) && gd2[i] <= p.goal_cull_r2) cand |= 1u << i;
        }
        // this step's lidar slots: "no hit" until the ray pass says otherwise
        reinterpret_cast<float2 *>(myfr + 1)[1] = make_float2(kMiss, kMiss);
        myfr[2] = make_float4(kMiss, kMiss, kMiss, kMiss);
        myfr[3] = make_float4(kMiss, kMiss, kMiss, kMiss);

        const bool near_any = active && (cell.x | cell.y | (cell.z & 3u)) != 0u;
        const bool staged = near_any && ((cell.z >> 8) & 0xffu) <= (unsigned)kMaxCand;
        if (staged) stage_candidates(p, r.scen, cell, RowPtr{myrow + 1});
        const bool oob = (mx < 0.f) || (mx > p.W) || (my < 0.f) || (my > p.H);
        // (while the candidate planes are in flight: the exact goal tests and everything that follows from them)
#pragma unroll 1
        while (cand) {
            const int i = __ffs(cand) - 1;
            cand &= cand - 1u;
            const float2 gi = s_goal[goal0 + i];
            const float ux = gi.x - mx, uy = gi.y - my;
            const float qx = fmaf(ux, mc, __fmul_rn(uy, ms)), qy = fmaf(uy, mc, -__fmul_rn(ux, ms));
            if (goal_contact(p, qx, qy)) touch |= 1u << i;
        }

        // ---- 3a. goals taken so far in the window: prefix OR of the touch masks (one ballot per goal: taken before /
        // up to step t <=> an earlier / this-or-earlier lane of the env touches it)
        unsigned inc = 0u, exc = 0u;
        {
            const unsigned below = segmask & ((1u << lane) - 1u), upto = segmask & ((2u << lane) - 1u);
#pragma unroll
            for (int i = 0; i < kGoals; ++i) {
                const unsigned m = __ballot_sync(kFull, (touch >> i) & 1u);
                if (m & below) exc |= 1u << i;
                if (m & upto) inc |= 1u << i;
            }
        }
        const int alive_prev = r.alive & ~(int)exc, alive_t = r.alive & ~(int)inc;
        const bool goal_reached = (alive_prev & (int)touch) != 0;
        const int steps_t = r.steps + t + 1;
        const bool all_goals = alive_t == 0;
        const bool timeout = steps_t >= p.max_steps;
        // With auto-reset the window is cut after the env's first done step, so nothing behind the first step that is done
        // for a reason already known (no goals left, out of bounds, step cap) can be committed: such steps need neither
        // the overlap test nor a lidar query.  (A ship that has run into a bank keeps ploughing through it for the rest of
        // the speculated window: before this cut those steps were a third of the separating-axis work.)
        const bool prune = p.auto_reset != 0;
        bool open_step = true;
        {
            const unsigned cd = __ballot_sync(kFull, active && (all_goals || oob || timeout)) & segmask;
            if (prune && cd != 0u && lane > __ffs(cd) - 1) open_step = false;
        }


        // ---- plane phase at pose t: lidar planes of step t+1 + ship-vs-bank pre-test of step t
        cp_async_wait_all();
        unsigned ask = 0u;
        if (staged) {
            ask = plane_phase<true, true>(p, mx, my, hx, hy, mc, ms, r.scen, cell, RowPtr{myrow}, RowPtr{myrow + 1});
        } else if (near_any) {                  // more candidates than are staged: evaluated straight from global memory
            ask = plane_phase_unstaged(p, mx, my, hx, hy, mc, ms, r.scen, cell, myrow);
        } else if (active) {
            myrow[0] = make_float4(mc, ms, 0.f, 0.f);
        }
        __syncwarp();

        // ---- overlap test at the new pose -> collide_ship (game.py:232-241): separating-axis pass for the steps the
        // plane phase could not settle.  Every env group works on its own earliest open step (one lane per bank edge,
        // strided when the hull has more edges than the group has lanes); a collision closes all later steps of the env.
        bool colliding = false;
        bool asking = ask != 0u && open_step;
        {
            unsigned needs;
            while ((needs = __ballot_sync(kFull, asking)) != 0u) {
                const unsigned mine = needs & segmask;
                const bool act_env = mine != 0u;
                const int src = act_env ? __ffs(mine) - 1 : lane;
                const float bx = __shfl_sync(kFull, mx, src), by = __shfl_sync(kFull, my, src);
                const float bc = __shfl_sync(kFull, mc, src), bs = __shfl_sync(kFull, ms, src);
                const unsigned bask = __shfl_sync(kFull, ask, src);
                const float4 *rec = p.bank + (size_t)r.scen * p.scen_stride4;
                const float4 hdr = __ldg(rec + 4);
                const float4 *bE = rec + kBankHeader4;
                float rx[kShipVerts], ry[kShipVerts];
#pragma unroll
                for (int j = 0; j < kShipVerts; ++j) {
                    rx[j] = p.ship_lx[j] * bc - p.ship_ly[j] * bs;
                    ry[j] = p.ship_lx[j] * bs + p.ship_ly[j] * bc;
                }
                bool coll = false;
#pragma unroll 1
                for (int b = 0; b < 2; ++b) {
                    const bool do_b = act_env && ((bask >> b) & 1u) && !coll;
                    const int nb = __float_as_int(b ? hdr.w : hdr.z);
                    const float4 *bEb = bE + b * p.maxv;
                    // a bank edge normal separates?  (lane t of the group takes edges t, t + T, ...)
                    bool lsep = false;
#pragma unroll 1
                    for (int u = 0; u < epl; ++u) {
                        const int idx = t + u * T;
                        if (do_b && idx < nb) lsep = lsep || bank_axis_separates(__ldg(bEb + idx), rx, ry, bx, by);
                    }
                    const unsigned sb = __ballot_sync(kFull, lsep);
                    bool sep = (sb & segmask) != 0u;
                    if (__ballot_sync(kFull, do_b && !sep)) {                   // else try the ship's edge normals
                        float pr[kShipVerts];
#pragma unroll
                        for (int j = 0; j < kShipVerts; ++j) pr[j] = 3.0e38f;
#pragma unroll 1
                        for (int u = 0; u < epl; ++u) {
                            const int idx = t + u * T;
                            if (do_b && idx < nb) {
                                const float4 ed = __ldg(bEb + idx);
#pragma unroll
                                for (int j = 0; j < kShipVerts; ++j) {
                                    const float nx = p.ship_nx[j] * bc - p.ship_ny[j] * bs;
                                    const float ny = p.ship_nx[j] * bs + p.ship_ny[j] * bc;
                                    pr[j] = fminf(pr[j], nx * (ed.z - bx) + ny * (ed.w - by));
                                }
                            }
                        }
#pragma unroll
                        for (int j = 0; j < kShipVerts; ++j) {      // axis j separates <=> no bank vertex reaches the hull's plane j
                            const unsigned reach = __ballot_sync(kFull, pr[j] <= p.ship_off[j]);
                            sep = sep || (reach & segmask) == 0u;
                        }
                    }
                    if (do_b && !sep) coll = true;
                }
                if (act_env && lane == src) { asking = false; colliding = coll; }
                if (coll && prune) asking = false;                              // the env is done at step src: later steps are moot
            }
        }

        // ShipEnv.determine_reward (ship_env.py:62-77) / is_done (ship_env.py:115-134)
        const float reward = goal_reached ? 1.f : (oob ? -1.f : p.step_penalty);
        const bool done = colliding || all_goals || oob || timeout;
        // cut the window after the first done step (auto-reset): everything speculated beyond it is discarded
        const unsigned dmask = __ballot_sync(kFull, active && done) & segmask;
        const bool do_reset = p.auto_reset && dmask != 0u;
        const int ncommit = do_reset ? __ffs(dmask) - gbase : nvalid;
        const bool commit = t < ncommit;

        // The actions of the next window, now: after a window that commits n steps they are n lanes further along the
        // (a_my, a_nx) pair, and the lanes at the far end load theirs.  Done here, as soon as n is known, and not at the end
        // of the iteration: the compiler waits for every outstanding load at the loop's back edge, so a load issued there
        // was paid in full at the top of every window (4.5 % of the stall samples, ncu); from here it has the ray pass, the
        // frame and the copy-out to land behind.
        {
            const int sh = t + ncommit;                             // (ncommit <= T)
            const int m1 = __shfl_sync(kFull, a_my, sh, T), m2 = __shfl_sync(kFull, a_nx, sh, T);    // lane (sh mod T) of the group
            a_my = sh < T ? m1 : m2;
            a_nx = m2;
            if (sh >= T) {
                const int kk = k0 + ncommit + T + t;
                a_nx = (valid && kk < p.K) ? load_action(p, act0 + (size_t)kk * act_stride, kk, gid) : 3;
            }
            // two windows ahead: pull the action rows into L2 (longest window only: -1.2 % on the headline with T = 16)
            if (T >= 32 && p.action_dtype != 3 && valid && k0 + ncommit + 2 * T + t < p.K) prefetch_l2(act0 + (size_t)(k0 + ncommit + 2 * T + t) * act_stride);
        }


        // ---- LiDAR.query (models.py:39-76) of step t at its PRE-integration pose = the pose of step t-1 (ring slot
        // cb + t; the carry for t = 0), for the steps that are committed.  Up to three needy steps per pass, lanes 0-9 /
        // 10-19 / 20-29 = their rays.
        {
            const int srcrow = sc0 + ring(cb + t) * kScr4;
            const int hz_own = commit ? __float_as_int(s_scr[srcrow].z) : 0;
            const bool big = (hz_own & kHdrBig) != 0;
            const bool wants = (hz_own & 0x3ff) != 0;
            const unsigned need = __ballot_sync(kFull, wants);
            if (big) ray_query_serial(p, s_scr + srcrow, reinterpret_cast<float *>(myfr) + 6);
            if (need) {
                if (wants) s_src[warp][__popc(need & ((1u << lane) - 1u))] =
                    (unsigned)(srcrow - wsc0) | ((unsigned)((fr0 - wfr0 + (1 + t) * FS4) * 4 + 6) << 16);
                __syncwarp();
                const int cnt = __popc(need);
                const float ray_c = s_ray[lane], ray_s = s_ray[32 + lane];
#pragma unroll 1
                for (int q = rslot; q < cnt; q += 3) {
                    if (rslot < 3) {
                        const unsigned sw = s_src[warp][q];
                        const float v = ray_vs_row(RowPtr{s_scr + wsc0 + (int)(sw & 0xffffu)}, ray_c, ray_s, L);
                        if (v >= 0.f) reinterpret_cast<float *>(s_frame + wfr0)[(sw >> 16) + rj] = v;
                    }
                }
            }
        }

        // episode return after step t: ordered sum (lane t adds the rewards of steps 0..t one by one), same rounding
        // as one step at a time
        float my_ret = r.ret;
        reinterpret_cast<float *>(s_rw)[warp * 32 + lane] = reward;
        __syncwarp();
        {
            const float4 *rw4 = s_rw + (warp * 32 + gbase) / 4;
            float rv[T];
#pragma unroll
            for (int j = 0; j < T; j += 4) {
                const float4 d = rw4[j / 4];
                rv[j] = d.x; rv[j + 1] = d.y; rv[j + 2] = d.z; rv[j + 3] = d.w;
            }
#pragma unroll
            for (int i = 0; i < T; ++i)
                if (i <= t) my_ret += rv[i];
        }
        warp_stats(stat_s, lane, commit, goal_reached, done, colliding, oob, timeout, all_goals, my_ret, steps_t);
        // this step's frame: pose, rudder, nearest remaining goal (closest_goal, game.py:333-349), and the lidar
        // readings.  Sticky readings (models.py:71): a ray that missed keeps the reading of the last step at which it
        // hit -- the latest hit at or before step t inside the window (found with a ballot per ray), else the carry's.
        __syncwarp();                           // ray pass results are in the frame slots
        {
            float gx = -1.f, gy = -1.f, best = 3.0e38f;
#pragma unroll
            for (int i = 0; i < kGoals; ++i)
                if (((alive_t >> i) & 1) && gd2[i] < best) { best = gd2[i]; gx = g[i].x; gy = g[i].y; }
            float h[kBeams], cv[kBeams];
            {
                const float4 *cf = s_frame + fr0;
                const float2 a0 = reinterpret_cast<const float2 *>(cf + 1)[1];
                const float4 a1 = cf[2], a2 = cf[3];
                cv[0] = a0.x; cv[1] = a0.y; cv[2] = a1.x; cv[3] = a1.y; cv[4] = a1.z; cv[5] = a1.w;
                cv[6] = a2.x; cv[7] = a2.y; cv[8] = a2.z; cv[9] = a2.w;
                const float2 b0 = reinterpret_cast<const float2 *>(myfr + 1)[1];
                const float4 b1 = myfr[2], b2 = myfr[3];
                h[0] = b0.x; h[1] = b0.y; h[2] = b1.x; h[3] = b1.y; h[4] = b1.z; h[5] = b1.w;
                h[6] = b2.x; h[7] = b2.y; h[8] = b2.z; h[9] = b2.w;
            }
            const unsigned upto = segmask & ((2u << lane) - 1u);       // lanes of this env at steps <= t
#pragma unroll
            for (int j = 0; j < kBeams; ++j) {
                const unsigned m = __ballot_sync(kFull, h[j] != kMiss) & upto;
                const float v = __shfl_sync(kFull, h[j], 31 - __clz(m));     // m == 0: lane 31's value, not used
                h[j] = m ? v : cv[j];
            }
            myfr[0] = make_float4(mx, my, (float)mrud, mth);
            myfr[1] = make_float4(gx, gy, h[0], h[1]);
            myfr[2] = make_float4(h[2], h[3], h[4], h[5]);
            myfr[3] = make_float4(h[6], h[7], h[8], h[9]);
        }

        // ---- 4. the state the next window starts from: after the last committed step (the scans left it in shared
        // memory), or the reset
        const int srcl = gbase + max(ncommit, 1) - 1;
        EnvRegs rn;
        {
            const float4 *ph = s_ph + (warp * 32 + srcl) * 2;
            const float4 v0 = ph[0], v1 = ph[1];
            rn.th = v0.x; rn.w = v0.y;
            rn.x = v1.x; rn.y = v1.y; rn.vx = v1.z; rn.vy = v1.w;
        }
        rn.rudder = __shfl_sync(kFull, mrud, srcl);
        rn.ret = __shfl_sync(kFull, my_ret, srcl);
        rn.alive = __shfl_sync(kFull, alive_t, srcl);
        rn.steps = r.steps + ncommit; rn.scen = r.scen; rn.episode = r.episode;
        float c0n = __shfl_sync(kFull, mc, srcl), s0n = __shfl_sync(kFull, ms, srcl);
        if (t == 0) s_env[warp * E + el] = make_int4(k0, ncommit, cb, (int)do_reset);
        float4 spv[SPL];                                            // the new scenario's spawn row, lane t holds entries t, t + T, ...
        if (do_reset) {                                             // ShipEnv.reset (ship_env.py:171-184)
            const int ep = r.episode + 1;
            reset_env(p, rn, next_scen, ep);
            c0n = 1.f; s0n = 0.f;
            const float4 *sp = p.spawn_rows + (size_t)rn.scen * kScr4;
            float4 rg0, rg1, rg2;
            float2 gn[kGoals];
            scenario_goals(p, rn.scen, rg0, rg1, rg2, gn);
#pragma unroll
            for (int i = 0; i < SPL; ++i) if (t + i * T < kScr4) spv[i] = __ldg(sp + t + i * T);
            next_scen = pick_scenario_keyed<PICK>(p, pkey, ep + 1);
            float rgx, rgy;
            closest_goal(gn, rn.alive, rn.x, rn.y, rgx, rgy);
            if (t == 0) {
#pragma unroll
                for (int i = 0; i < kGoals; ++i) s_goal[goal0 + i] = gn[i];
                s_rf[rf0] = make_float4(rn.x, rn.y, 0.f, 0.f);
                s_rf[rf0 + 1] = make_float4(rgx, rgy, -1.f, -1.f);
            }
            goals_dirty = true;
        }
        __syncwarp();

        // ---- outputs of the committed steps.  Obs row of step t = [frame t-1 | frame t] = frame slots (t, t + 1);
        // OBS4 lanes per row, 32/OBS4 rows per store instruction, 128-bit streaming stores, no loop: a window has at
        // most T rows per env.
        if (p.obs) {
            constexpr int RPR = 32 / OBS4;                          // rows per store instruction
            constexpr int NIT = (T + RPR - 1) / RPR;
            const float4 neg = make_float4(-1.f, -1.f, -1.f, -1.f);
            const int col = lane % OBS4, r0 = lane / OBS4;
            const int half = HIST == 2 ? (col >> 2) : 1, q = col & 3;
            const size_t rstride = (size_t)p.N * OBS4 * RPR;        // float4 between the rows of consecutive stores
#pragma unroll
            for (int elr = 0; elr < E; ++elr) {
                const int4 ev = s_env[warp * E + elr];              // k0, committed, -, reset
                const float4 *fb = s_frame + wfr0 + elr * FR4 + (r0 + half) * FS4 + q;
                float4 *o = p.obs + ((size_t)(ev.x + r0) * p.N + (warp_env0 + elr)) * OBS4 + col;
                const int nplain = ev.w ? ev.y - 1 : ev.y;          // the last committed row of an env that resets is special
#pragma unroll
                for (int it = 0; it < NIT; ++it) {
                    if (r0 + it * RPR < nplain) __stcs(o, fb[it * RPR * FS4]);
                    o += rstride;
                }
                if (ev.w && r0 == 0) {                              // ship_env.py:180-184: [-1 x 16 | reset frame], vals = -1
                    const float4 rfv = (half == 0 || q >= 2) ? neg : s_rf[(warp * E + elr) * 2 + q];
                    __stcs(p.obs + ((size_t)(ev.x + nplain) * p.N + (warp_env0 + elr)) * OBS4 + col, rfv);
                }
            }
        }
        if (commit) {
            const size_t row = (size_t)(k0 + t) * p.N + e;
            if (p.reward) p.reward[row] = reward;
            if (p.done) p.done[row] = done ? 1 : 0;
        }
        if (LOG) {
            // episode log: the lane of the window's first done step writes the terminal row -- frame slots t and t + 1,
            // complete since the sticky-lidar scan, not yet overwritten by the reset below -- and the episode's numbers
            // (r is still the finished episode's state)
            const bool mine = do_reset && t == ncommit - 1;
            const unsigned lm = __ballot_sync(kFull, mine);
            if (lm) {
                const unsigned slot = log_reserve(p, lane, lm);
                if (mine && slot < (unsigned)p.log_cap) {
                    float4 *row = p.log_rows + (size_t)slot * p.log_row4 + (p.log_row4 - OBS4);
                    const float4 *fp = myfr - (HIST - 1) * FS4;
#pragma unroll
                    for (int h = 0; h < HIST; ++h)
#pragma unroll
                        for (int i = 0; i < 4; ++i) row[4 * h + i] = fp[h * FS4 + i];
                    log_meta(p, slot, k0 + t, e, steps_t, my_ret, end_bits(colliding, all_goals, oob, timeout, goal_reached), r.scen, r.episode);
                }
            }
        }
        __syncwarp();                           // rows and frames have been read: the carry may move

        if (ncommit > 0) {
            const int ncb = ring(cb + ncommit);
            const float4 negc = make_float4(-1.f, -1.f, -1.f, -1.f);
            if (do_reset) {                     // carry := reset frame + the spawn pose's planes (built at scenario upload)
                if (t == 0) {
                    float4 *f = s_frame + fr0;
                    f[0] = s_rf[rf0]; f[1] = s_rf[rf0 + 1]; f[2] = negc; f[3] = negc;
                }
                float4 *row = s_scr + sc0 + ncb * kScr4;            // the whole row: entries past its planes are never read
#pragma unroll
                for (int i = 0; i < SPL; ++i) if (t + i * T < kScr4) row[t + i * T] = spv[i];
            } else if (t == ncommit - 1) {      // carry := the frame of the last committed step
                float4 *f = s_frame + fr0;
                f[0] = myfr[0]; f[1] = myfr[1]; f[2] = myfr[2]; f[3] = myfr[3];
            }
            cb = ncb;
            r = rn; c0 = c0n; s0 = s0n;
            k0 += ncommit;
        }
        __syncwarp();
    }

    if (valid && t == 0) {
        store_env_frame(p, e, r, RowPtr{s_frame + fr0});
        if (goals_dirty) {
            const float2 a0 = s_goal[goal0], a1 = s_goal[goal0 + 1], a2 = s_goal[goal0 + 2], a3 = s_goal[goal0 + 3], a4 = s_goal[goal0 + 4];
            store_goals(p, e, make_float4(a0.x, a0.y, a1.x, a1.y), make_float4(a2.x, a2.y, a3.x, a3.y), make_float4(a4.x, a4.y, 0.f, 0.f));
        }
    }
    flush_stats(p, lane, RowPtr{reinterpret_cast<float4 *>(s_stat[warp])});
    if constexpr (CHAIN) {
        __threadfence();
        __syncwarp();
        if (valid && t == 0) chain_release(p.chain_done + e, s_ticket[warp * E + el]);
        griddep_wait();
    }
#undef stat
}

// A chained launch: programmatic stream serialization lets it start before the previous kernel of the stream has
// completed (as soon as that kernel's CTAs have all executed griddepcontrol.launch_dependents).
static cudaError_t launch_pdl(void (*kernel)(StepParams), const StepParams &p, int blocks, cudaStream_t stream)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks);
    cfg.blockDim = dim3(kWinThreads);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, p);
}

template <int T, bool PICK>
static cudaError_t launch_th(const StepParams &p, int blocks, cudaStream_t stream, bool chain)
{
    if (chain) return launch_pdl(p.history == 2 ? window_kernel<T, 2, false, PICK, true> : window_kernel<T, 1, false, PICK, true>, p, blocks, stream);
    if (p.log_count) {
        if (p.history == 2) window_kernel<T, 2, true, PICK, false><<<blocks, kWinThreads, 0, stream>>>(p);
        else window_kernel<T, 1, true, PICK, false><<<blocks, kWinThreads, 0, stream>>>(p);
    } else {
        if (p.history == 2) window_kernel<T, 2, false, PICK, false><<<blocks, kWinThreads, 0, stream>>>(p);
        else window_kernel<T, 1, false, PICK, false><<<blocks, kWinThreads, 0, stream>>>(p);
    }
    return cudaGetLastError();
}

template <int T>
static cudaError_t launch_t(const StepParams &p, cudaStream_t stream, LaunchShape *shape, bool chain)
{
    const int envs_per_cta = (kWinThreads / 32) * (32 / T);
    const int blocks = (p.N + envs_per_cta - 1) / envs_per_cta;
    if (shape) { shape->lanes_per_env = T; shape->threads = kWinThreads; shape->blocks = blocks; shape->window = T; }
    return p.pick_cdf ? launch_th<T, true>(p, blocks, stream, chain) : launch_th<T, false>(p, blocks, stream, chain);
}

cudaError_t launch_window(const StepParams &p, int window, cudaStream_t stream, LaunchShape *shape, bool chain)
{
    if (chain && (p.log_count || !p.chain_started || !p.chain_done)) return cudaErrorInvalidValue;
    switch (window) {
        case 4: return launch_t<4>(p, stream, shape, chain);
        case 8: return launch_t<8>(p, stream, shape, chain);
        case 16: return launch_t<16>(p, stream, shape, chain);
        case 32: return launch_t<32>(p, stream, shape, chain);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace shipsim
