// shipsim_policy.cu -- the policy half of an on-device rollout step (BASELINE configs[4]: policy + envs on one GPU, no host
// round trip per step): stable-baselines' MlpPolicy as the reference trains it (train/stable_baselines/ppo.py:88 --
// separate tanh trunks 32 -> 64 -> 64 for the policy and the value function, heads of 3 and 1) evaluated for a whole
// batch of envs, with the categorical sample taken by Gumbel-max from noise the caller drew for the whole rollout.
// One launch per step instead of the 7 torch kernels (3 addmm, 2 tanh, add, argmax) the loop needed: at 16,384 envs every
// one of those runs for a few microseconds and the loop was launch bound (59 of 66 us per step).
//
// fp32 SIMT, FMA in ascending input order.  No tensor cores: 0.4 GFLOP per step is ~6 us of the FP32 pipes, and the
// results stay within 1e-5 of the fp32 torch module (bf16 / tf32 operands would not).
//
// One CTA per SM, 16 warps = 8 tile slots x 2 trunks; a tile = 16 envs (four warps per scheduler hide the shared-memory
// latency of the register-tiled products better than two: 18.0 -> 16.4 us at 16,384 envs, -10 % at 65,536).  The weights (50 KB) are copied into shared memory
// ONCE per CTA by cp.async while the observation tiles are loaded.  (Reading them through L1 cost every 4-input block of
// the loops an L2 round trip: 40 % of the kernel's cycles were long-scoreboard stalls, ncu; an L1 prefetch did not help.)
// Each layer is a small SGEMM with a 4 x 8 register tile per thread (4 envs x 8 hidden units: lane = unit group * 4 +
// env group): per input k a thread reads 4 activations (k-major tile, one 128-bit load) and 8 weights (two), conflict-free,
// and issues 32 FMAs.  (The very first version gave every
// thread one hidden unit and broadcast the activations: a 128-bit broadcast load still costs four wavefronts, and the
// kernel ran at the shared-memory rate.)
#include "shipsim_device.cuh"
#include "shipsim_launch.h"

#include <algorithm>
#include <atomic>

namespace shipsim {

constexpr int kPolD = 32, kPolH = 64, kPolA = 3;      // inputs, hidden units per trunk, actions
constexpr int kPolE = 16;                             // envs per tile
constexpr int kPolT = 8;                              // register tile: kPolM envs x kPolT units per thread
constexpr int kPolM = kPolE / 4;                      // (4 env groups per warp)

// tanh(x) = 1 - 2 / (exp(2x) + 1) on the special-function unit (ex2.approx + rcp.approx: 7 instructions, |error| < 4e-7,
// saturates correctly at both ends) instead of libdevice's two-branch tanhf.
__device__ __forceinline__ float tanh_sfu(float x) { return 1.f - __fdividef(2.f, __expf(2.f * x) + 1.f); }

// acc[m][n] += sum_k act[k][e0 + m] * w[k * ldw + n], k < K: act = k-major shared-memory tile (row = kPolE floats), w = shared memory
template <int K>
__device__ __forceinline__ void tile_gemm(float (&acc)[kPolM][kPolT], const float *act, const float *w, int ldw)
{
    static_assert(kPolM == 4 || kPolM == 8, "one or two 128-bit activation loads per input");
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
        float x[kPolM];
        {
            const float4 xa = *reinterpret_cast<const float4 *>(act + k * kPolE);
            x[0] = xa.x; x[1] = xa.y; x[2] = xa.z; x[3] = xa.w;
            if (kPolM == 8) {
                const float4 xb = *reinterpret_cast<const float4 *>(act + k * kPolE + 4);
                x[kPolM - 4] = xb.x; x[kPolM - 3] = xb.y; x[kPolM - 2] = xb.z; x[kPolM - 1] = xb.w;
            }
        }
        const float4 ca = *reinterpret_cast<const float4 *>(w + k * ldw), cb = *reinterpret_cast<const float4 *>(w + k * ldw + 4);
        const float c[kPolT] = {ca.x, ca.y, ca.z, ca.w, cb.x, cb.y, cb.z, cb.w};
#pragma unroll
        for (int m = 0; m < kPolM; ++m)
#pragma unroll
            for (int n = 0; n < kPolT; ++n) acc[m][n] = fmaf(x[m], c[n], acc[m][n]);
    }
}

constexpr int kPolSlots = 8;                                          // tiles a CTA works on at once
// the two warps of a slot meet at the slot's own named barrier: slots do not wait for each other (CTA-wide barriers were
// 20 % of the kernel's stall cycles, ncu: four slots at different points of their tiles, a slot without a tile idling)
__device__ __forceinline__ void slot_sync(int slot) { asm volatile("bar.sync %0, 64;" ::"r"(slot + 1) : "memory"); }
constexpr int kPolW1 = kPolD * 2 * kPolH, kPolW2 = 2 * kPolH * kPolH, kPolW3 = 2 * kPolH * 4;      // floats
constexpr int kPolTile = kPolD * kPolE + 2 * (2 * kPolH * kPolE) + kPolE * 4;                       // x | h1 | h2 | heads, floats per slot
constexpr size_t kPolSmem = (size_t)(kPolW1 + kPolW2 + kPolW3 + kPolSlots * kPolTile) * sizeof(float);

__global__ void __launch_bounds__(64 * kPolSlots, 1) mlp_policy_kernel(const float *__restrict__ obs, int n, const float *__restrict__ w1,
                                                                       const float *__restrict__ b1, const float *__restrict__ w2,
                                                                       const float *__restrict__ b2, const float *__restrict__ w3,
                                                                       const float *__restrict__ b3, const float *__restrict__ noise,
                                                                       float *__restrict__ out, long long *__restrict__ actions)
{
    extern __shared__ __align__(16) float smem[];
    float *s_w1 = smem, *s_w2 = s_w1 + kPolW1, *s_w3 = s_w2 + kPolW2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int slot = warp >> 1, trunk = warp & 1;                       // even warps: policy trunk, odd warps: value trunk
    const int st = tid & 63;                                            // thread index inside the slot
    float *s_x = s_w3 + kPolW3 + slot * kPolTile;                       // [k][env]
    float *s_h1 = s_x + kPolD * kPolE, *s_h2 = s_h1 + 2 * kPolH * kPolE;    // [unit][env], both trunks
    float *s_o = s_h2 + 2 * kPolH * kPolE;
    const int eg = lane & 3, ug = lane >> 2;                            // env group (8 envs), unit group (8 units of the trunk)

    // weights -> shared memory, asynchronously (all of it in flight at once)
    for (int q = tid; q < kPolW1 / 4; q += 64 * kPolSlots) cp_async16(s_w1 + 4 * q, w1 + 4 * q);
    for (int q = tid; q < kPolW2 / 4; q += 64 * kPolSlots) cp_async16(s_w2 + 4 * q, w2 + 4 * q);
    for (int q = tid; q < kPolW3 / 4; q += 64 * kPolSlots) cp_async16(s_w3 + 4 * q, w3 + 4 * q);

    const int ntiles = (n + kPolE - 1) / kPolE;
    const int u0 = trunk * kPolH + ug * kPolT;                          // this thread's first hidden unit (of 128)
    // tiles are dealt round-robin over (pass, slot, CTA): with 512 tiles on 148 SMs every CTA gets 3 or 4
    for (int tile0 = blockIdx.x; tile0 < ntiles; tile0 += gridDim.x * kPolSlots) {                  // (uniform over the CTA)
        const int tile = tile0 + slot * gridDim.x;
        const bool live = tile < ntiles;
        const int e0 = tile * kPolE;
        const int ne = live ? min(kPolE, n - e0) : 0;
        // observations of the slot's envs, transposed into the k-major tile (rows beyond the batch: zeros)
        if (live) {
            for (int q = st; q < kPolE * kPolD / 4; q += 64) {
                const int row = q / (kPolD / 4), k4 = (q % (kPolD / 4)) * 4;
                const float4 v = row < ne ? __ldg(reinterpret_cast<const float4 *>(obs + (size_t)e0 * kPolD) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
                s_x[(k4 + 0) * kPolE + row] = v.x; s_x[(k4 + 1) * kPolE + row] = v.y; s_x[(k4 + 2) * kPolE + row] = v.z; s_x[(k4 + 3) * kPolE + row] = v.w;
            }
        }
        if (tile0 == (int)blockIdx.x) {                                 // first pass: the weights must have landed (all threads fetched them)
            cp_async_wait_all();
            __syncthreads();
        } else if (live) slot_sync(slot);                               // later passes: the slot's tile is complete
        if (!live) continue;                                            // (a slot without a tile in this pass has none in any later one)
        float acc[kPolM][kPolT];
        auto init = [&](const float *bias) {
            const float4 ba = __ldg(reinterpret_cast<const float4 *>(bias + u0)), bb = __ldg(reinterpret_cast<const float4 *>(bias + u0) + 1);
            const float b[kPolT] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int m = 0; m < kPolM; ++m)
#pragma unroll
                for (int nn = 0; nn < kPolT; ++nn) acc[m][nn] = b[nn];
        };
        auto store_tanh = [&](float *dst) {                             // dst[unit][env]: kPolM consecutive envs per unit, 128-bit stores
#pragma unroll
            for (int nn = 0; nn < kPolT; ++nn) {
                float4 *d = reinterpret_cast<float4 *>(dst + (u0 + nn) * kPolE + eg * kPolM);
#pragma unroll
                for (int q = 0; q < kPolM / 4; ++q)
                    d[q] = make_float4(tanh_sfu(acc[4 * q][nn]), tanh_sfu(acc[4 * q + 1][nn]), tanh_sfu(acc[4 * q + 2][nn]), tanh_sfu(acc[4 * q + 3][nn]));
            }
        };
        {
            // layer 1: h1 = tanh(b1 + x W1)          (w1: [32][128], observation scale folded in)
            init(b1);
            tile_gemm<kPolD>(acc, s_x + eg * kPolM, s_w1 + u0, 2 * kPolH);
            store_tanh(s_h1);
            __syncwarp();                                               // layer 2 of a trunk reads only what its own warp wrote
            // layer 2, block diagonal: a trunk's units see only that trunk's 64 activations          (w2: [2][64][64])
            init(b2);
            tile_gemm<kPolH>(acc, s_h1 + trunk * kPolH * kPolE + eg * kPolM, s_w2 + trunk * kPolH * kPolH + ug * kPolT, kPolH);
            store_tanh(s_h2);
        }
        slot_sync(slot);
        {
            // heads: thread (o, e) -- o < 3: logit o from the policy trunk, o = 3: value from the value trunk          (w3: [128][4])
#pragma unroll
            for (int r = 0; r < (4 * kPolE) / 64; ++r) {
                const int e = st % kPolE, o = st / kPolE + (64 / kPolE) * r;
                const int base = o == kPolA ? kPolH : 0;
                float a = __ldg(b3 + o);
#pragma unroll 8
                for (int i = 0; i < kPolH; ++i) a = fmaf(s_h2[(base + i) * kPolE + e], s_w3[(base + i) * 4 + o], a);
                s_o[e * 4 + o] = a;
            }
        }
        slot_sync(slot);
        if (st < ne) {
            const float4 o4 = *reinterpret_cast<const float4 *>(s_o + st * 4);
            *reinterpret_cast<float4 *>(out + (size_t)(e0 + st) * 4) = o4;
            // categorical sample by Gumbel-max: argmax_o (logit_o + noise_o), first maximum wins
            const float *nz = noise + (size_t)(e0 + st) * kPolA;
            const float z0 = o4.x + __ldg(nz), z1 = o4.y + __ldg(nz + 1), z2 = o4.z + __ldg(nz + 2);
            int arg = 0;
            float best = z0;
            if (z1 > best) { best = z1; arg = 1; }
            if (z2 > best) { arg = 2; }
            actions[e0 + st] = arg;
        }
        slot_sync(slot);                                                // (s_o and the tiles are reused by the next pass)
    }
    cp_async_wait_all();
}

// Per-map scoring of a rollout's steps (gae_kernel<true>, shipsim_gae_scored).  Appended after the unscored kernel's
// parameters, which the unscored instantiation never reads, so that instantiation keeps its parameter offsets and its code.
struct GaeScoring {
    const float4 *plane4;        // state plane 4 of the bound state: .z = bits(scenario) of the episode each env plays now
    int *step_scen;              // [T][N]: in, the scenario of the episode that ended at (t, e) or -1; out, the scenario of every step
    double *scores;              // [n_scen + 1][3] (SHIPSIM_SCORE_*), added into; row n_scen: steps of no known scenario
    int n_scen;
};

// Generalised advantage estimation over a finished rollout, as PPO2's runner computes it (the reference trains with
// stable-baselines PPO2: train/stable_baselines/ppo.py:88,104): adv[t] = delta[t] + gamma * lam * nonterminal[t] * adv[t + 1],
// delta[t] = r[t] + gamma * V[t + 1] * nonterminal[t] - V[t], returns = adv + V.  One thread per env walks its T steps
// backwards (coalesced across envs): one launch instead of ~T + 8 elementwise torch kernels.
//
// SCORE: the same walk also attributes every step to its map and sums Prioritized Level Replay's value-loss scores per map.
// Going backwards, the steps after an env's last done belong to the episode it plays now (the bound state); a done at t
// starts, going backwards, the episode that ended at t, whose map scatter_records_kernel put into step_scen[t].  Per run
// of steps on one map the count, sum max(adv, 0) and sum |adv| stay in registers (double) and are flushed with double
// atomics when the map changes and at the end -- so the table's last bits depend on the order in which the atomics land.
// adv and ret are computed by the same operations in the same order as without SCORE.
template <bool SCORE>
__global__ void __launch_bounds__(256) gae_kernel(const float *__restrict__ rew, const float *__restrict__ val, const unsigned char *__restrict__ done,
                                                  int T, int N, float gamma, float gl, float *__restrict__ adv, float *__restrict__ ret, GaeScoring sc)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    int seg = 0, steps = 0;
    double pos = 0.0, mag = 0.0;
    auto flush = [&]() {
        if (steps) {
            double *s = sc.scores + (size_t)(seg >= 0 && seg < sc.n_scen ? seg : sc.n_scen) * 3;
            atomicAdd(s + 0, (double)steps);
            atomicAdd(s + 1, pos);
            atomicAdd(s + 2, mag);
        }
        steps = 0; pos = 0.0; mag = 0.0;
    };
    if (SCORE) seg = __float_as_int(sc.plane4[e].z);
    float last = 0.f, vnext = __ldg(val + (size_t)T * N + e);
    for (int t = T - 1; t >= 0; --t) {
        const size_t i = (size_t)t * N + e;
        const bool d = done[i];
        const float nt = d ? 0.f : 1.f, v = __ldg(val + i);
        const float delta = __ldg(rew + i) + gamma * vnext * nt - v;
        last = delta + gl * nt * last;
        adv[i] = last;
        ret[i] = last + v;
        vnext = v;
        if (SCORE) {
            if (d) {                                                    // step t belongs to the episode that ended at t
                const int s = sc.step_scen[i];
                if (s != seg) { flush(); seg = s; }
            }
            sc.step_scen[i] = seg;
            ++steps;
            pos += (double)fmaxf(last, 0.f);
            mag += (double)fabsf(last);
        }
    }
    if (SCORE) flush();
}

// One thread per episode-log record (slots < min(*count, cap)): the record of call c, step k within it, env e, scenario s
// is rollout step t = (c - call0) * steps_per_call + k, and step_scen[t][e] = s.  Records outside the rollout (t, e or s
// out of range) are skipped.
__global__ void __launch_bounds__(256) scatter_records_kernel(const int4 *__restrict__ meta, const int *__restrict__ count, int cap, int call0,
                                                              int steps_per_call, int T, int N, int n_scen, int *__restrict__ step_scen)
{
    const int n = min(*count, cap);
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
        const int4 a = meta[2 * (size_t)r], b = meta[2 * (size_t)r + 1];      // {k, env, length, return}, {end, scenario, episode, call}
        const int k = a.x, env = a.y, s = b.y;
        const long long t = (long long)(b.w - call0) * steps_per_call + k;
        if (k < 0 || k >= steps_per_call || t < 0 || t >= T || env < 0 || env >= N || s < 0 || s >= n_scen) continue;
        step_scen[t * N + env] = s;
    }
}

cudaError_t launch_gae(const float *rew, const float *val, const unsigned char *done, int T, int N, float gamma, float lam, float *adv, float *ret,
                       cudaStream_t stream)
{
    if (T <= 0 || N <= 0) return cudaSuccess;
    gae_kernel<false><<<(N + 255) / 256, 256, 0, stream>>>(rew, val, done, T, N, gamma, gamma * lam, adv, ret, GaeScoring{});
    return cudaGetLastError();
}

cudaError_t launch_gae_scored(const float *rew, const float *val, const unsigned char *done, int T, int N, float gamma, float lam, float *adv,
                              float *ret, const int4 *log_meta, const int *log_count, int log_cap, int call0, int steps_per_call,
                              const float4 *plane4, int n_scen, int *step_scen, double *scores, cudaStream_t stream)
{
    if (T <= 0 || N <= 0) return cudaSuccess;
    cudaError_t err = cudaMemsetAsync(step_scen, 0xff, (size_t)T * N * sizeof(int), stream);         // -1: no record
    if (err != cudaSuccess) return err;
    if (log_cap > 0) {
        const int blocks = std::min((log_cap + 255) / 256, 1184);
        scatter_records_kernel<<<blocks, 256, 0, stream>>>(log_meta, log_count, log_cap, call0, steps_per_call, T, N, n_scen, step_scen);
        if ((err = cudaGetLastError()) != cudaSuccess) return err;
    }
    gae_kernel<true><<<(N + 255) / 256, 256, 0, stream>>>(rew, val, done, T, N, gamma, gamma * lam, adv, ret,
                                                          GaeScoring{plane4, step_scen, scores, n_scen});
    return cudaGetLastError();
}

cudaError_t launch_mlp_policy(const float *obs, int n, const float *w1, const float *b1, const float *w2, const float *b2, const float *w3,
                              const float *b3, const float *noise, float *out, long long *actions, cudaStream_t stream)
{
    if (n <= 0) return cudaSuccess;
    // the opt-in into more than 48 KB of dynamic shared memory holds for one device, and the SM count is one device's: both
    // are kept per device (a process may run collectors on several GPUs, from several threads).  The count is published
    // after the opt-in succeeded; a thread that still reads 0 repeats both, which is harmless.
    static std::atomic<int> sms_of[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    int sms = dev < 64 ? sms_of[dev].load() : 0;
    if (!sms) {
        e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(mlp_policy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPolSmem);
        if (e != cudaSuccess) return e;
        if (dev < 64) sms_of[dev].store(sms);
    }
    const int ntiles = (n + kPolE - 1) / kPolE;
    const int blocks = std::min(sms, ntiles);
    mlp_policy_kernel<<<blocks, 64 * kPolSlots, kPolSmem, stream>>>(obs, n, w1, b1, w2, b2, w3, b3, noise, out, actions);
    return cudaGetLastError();
}

}  // namespace shipsim
