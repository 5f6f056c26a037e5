// shipsim_abi.cu -- the C ABI of libshipsim.so (include/shipsim.h): handle management, scenario packing,
// parameter derivation and kernel launches.  Host-side C++; no torch types anywhere.
#include "../../include/shipsim.h"
#include "shipsim_device.cuh"
#include "shipsim_launch.h"
#include "shipsim_host.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <string>
#include <vector>

using namespace shipsim;

// Small persistent worker pool for the host half of shipsim_step_host (assembling observation histories from frames
// while later chunks are still crossing PCIe).  run(n, fn) calls fn(i) for i in [0, n) on the workers + the caller.
class HostPool {
public:
    explicit HostPool(int n_threads)
    {
        for (int i = 0; i < n_threads; ++i) workers_.emplace_back([this] { loop(); });
    }
    ~HostPool()
    {
        { std::lock_guard<std::mutex> lk(m_); quit_ = true; ++gen_; }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
    }
    void run(int n, const std::function<void(int)> &fn) { start(n, fn); finish(); }
    // start(): the workers begin on fn(0..n-1) and the caller carries on; finish(): the caller joins in and waits for all
    void start(int n, const std::function<void(int)> &fn)
    {
        {
            std::lock_guard<std::mutex> lk(m_);
            fn_ = &fn; n_ = n; next_.store(0); pending_ = (int)workers_.size(); ++gen_;
        }
        cv_.notify_all();
    }
    void finish()
    {
        drain();
        std::unique_lock<std::mutex> lk(m_);
        done_cv_.wait(lk, [this] { return pending_ == 0; });
    }
    int size() const { return (int)workers_.size() + 1; }

private:
    void drain() { for (int i; (i = next_.fetch_add(1)) < n_;) (*fn_)(i); }
    void loop()
    {
        unsigned seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return gen_ != seen; });
                seen = gen_;
                if (quit_) return;
            }
            drain();
            { std::lock_guard<std::mutex> lk(m_); --pending_; }
            done_cv_.notify_one();
        }
    }
    std::vector<std::thread> workers_;
    std::mutex m_;
    std::condition_variable cv_, done_cv_;
    const std::function<void(int)> *fn_ = nullptr;
    std::atomic<int> next_{0};
    int n_ = 0, pending_ = 0;
    unsigned gen_ = 0;
    bool quit_ = false;
};

struct shipsim_handle {
    shipsim_config cfg;
    int device = 0;
    StepParams p;
    float4 *d_bank = nullptr;
    EdgeD *d_edges = nullptr;
    uint4 *d_grid = nullptr;
    float4 *d_spawn = nullptr;
    double *d_gen_xy = nullptr, *d_gen_goals = nullptr;   // raw output of the device scenario generator (for read-back)
    int *d_gen_n = nullptr;
    int gen_count = 0;
    float ship_reach = 0.f;                  // bound on the distance of any hull point from the lidar origin
    int lanes = 1;
    int window = 1;                          // steps of one env speculated together (1 = the serial-in-time kernel)
    // staging for shipsim_step_host (allocated on first use, sized for the largest K seen)
    int32_t *d_act = nullptr; float *d_obs = nullptr; float *d_rew = nullptr; uint8_t *d_done = nullptr;
    int stage_K = 0;
    cudaStream_t copy_stream = nullptr;      // shipsim_step_host: results of chunk i go home while chunk i+1 is computed
    static constexpr int kMaxChunks = 64;
    cudaEvent_t chunk_done[kMaxChunks] = {}, copy_done[kMaxChunks] = {}, trace0 = nullptr, trace_mid[kMaxChunks] = {};
    float4 *d_frame0 = nullptr;
    // compacted wire format of the host path (compact_frames_kernel / expand_delta_rows)
    uint4 *d_rec = nullptr;                  // [K][N] records
    unsigned *d_off = nullptr, *d_count = nullptr;   // [K][N/32] value offsets; one counter per chunk
    uint32_t *h_rec = nullptr, *h_off = nullptr, *h_count = nullptr;     // pinned mirrors
    float *h_var = nullptr, *d_var = nullptr;   // the changed values (a dense stream per chunk), host mirror and device buffer
    double var_density = 2.0;                // floats per env-step the speculative D2H copy of a chunk's values is sized for
    cudaStream_t aux_stream = nullptr;       // actions of chunks 1.. go up here; the (rare) rest of a chunk's values comes down
    cudaEvent_t act_up = nullptr;
    float *h_cur = nullptr;                  // one frame per env: the decoder's running state
    size_t rec_cap = 0, var_cap = 0, cur_cap = 0;
    int var_per_step = 0;                    // capacity of the value stream, floats per env-step
    // the envs [0, dma_envs) go home as complete rows by DMA, the others compacted + expanded by the host threads
    float *d_rows = nullptr;                 // [K][dma_envs][32]
    size_t rows_cap = 0;
    int dma_envs = -1;                       // -1: not chosen yet
    int dma_for_n = 0, dma_for_k = 0;
    int dma_step = 0, dma_dir = 1;           // the split climbs towards the shorter call: step size and direction
    double dma_last_t = 0.0;                 // seconds per env-step of the previous call
    // fresh-maps mode (shipsim_fresh_maps): the device-generated bank is regenerated a quarter at a time behind the envs
    struct {
        bool on = false, pending = false;
        int map_N = 0;
        float width_frac = 0.f;
        uint64_t seed = 0;
        int period = 0;                      // resets of period p pick from quarter p % 4
        long long steps = 0;                 // env-steps (per env) since the period began
        int max_steps = 0;                   // the longest episode cap seen: a period lasts at least that many steps
        int generation[4] = {0, 0, 0, 0};    // how many times each quarter has been regenerated
        cudaStream_t stream = nullptr;
        cudaEvent_t period_begin = nullptr, gen_done = nullptr;
    } fresh;
    const void *zc_host[4] = {nullptr, nullptr, nullptr, nullptr};     // the last tiny call's buffers and their device aliases
    void *zc_dev[4] = {nullptr, nullptr, nullptr, nullptr};
    HostPool *pool = nullptr;
    int64_t last_h2d = 0, last_d2h = 0;      // bytes the last shipsim_step_host moved over PCIe
    int64_t launches = 0;
    int32_t calls = 0;                       // shipsim_step / shipsim_step_host calls so far (SHIPSIM_EP_CALL)
    LaunchShape shape{1, kThreads, 0, 1};
};

static thread_local std::string g_err;

static int fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}

#define CU(expr)                                                                                      \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess)                                                                        \
            return fail(SHIPSIM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));       \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

extern "C" int shipsim_abi_version(void) { return SHIPSIM_ABI_VERSION; }
extern "C" const char *shipsim_last_error(void) { return g_err.c_str(); }

extern "C" int shipsim_config_default(shipsim_config *c)
{
    if (!c) return fail(SHIPSIM_ERR_ARG, "cfg is NULL");
    std::memset(c, 0, sizeof(*c));
    c->struct_size = (int32_t)sizeof(shipsim_config);
    c->num_envs = 1;
    c->bounds_w = 600.f; c->bounds_h = 600.f;                 // config.py:24
    c->dt = 1.0f;                                             // SPEED 10 * base_dt 0.1 (config.py:23, game.py:27)
    c->damping = (float)std::pow(0.4, 1.0);                   // game.py:270
    c->max_steps = 1000; c->history = 2;                      // config.py:15-16
    c->auto_reset = 1;
    c->lidar_beams = SHIPSIM_N_BEAMS; c->lidar_spread_deg = 90.f; c->lidar_distance = 100.f;   // models.py:29
    c->ship_w = 2.f; c->ship_h = 3.f;                         // game.py:275
    c->mass = 5.f; c->thrust = 100.f;                         // models.py:87,107
    c->goal_radius = 5.f; c->step_penalty = -0.01f; c->spawn_y = 25.f;   // game.py:82, ship_env.py:13, game.py:274
    c->lanes_per_env = 0;
    c->steps_in_flight = 0;
    c->host_threads = 0;
    return SHIPSIM_OK;
}

// ---- small double-precision geometry helpers (host) --------------------------------------------------------
namespace {
struct P2 { double x, y; };

// Convex hull, CCW, collinear points dropped, first vertex = min-x then min-y: what pm.Poly does to the
// vertex list it is given (models.py:96,180 -> cpPolyShapeInit -> cpConvexHull tol 0).
std::vector<P2> convex_hull_ccw(std::vector<P2> pts)
{
    std::sort(pts.begin(), pts.end(), [](const P2 &a, const P2 &b) { return a.x < b.x || (a.x == b.x && a.y < b.y); });
    pts.erase(std::unique(pts.begin(), pts.end(), [](const P2 &a, const P2 &b) { return a.x == b.x && a.y == b.y; }), pts.end());
    const int n = (int)pts.size();
    if (n < 3) return pts;
    std::vector<P2> h(2 * n);
    int k = 0;
    auto turn = [](const P2 &o, const P2 &a, const P2 &b) { return (a.x - o.x) * (b.y - o.y) - (a.y - o.y) * (b.x - o.x); };
    for (int i = 0; i < n; ++i) { while (k >= 2 && turn(h[k - 2], h[k - 1], pts[i]) <= 0) --k; h[k++] = pts[i]; }
    for (int i = n - 2, t = k + 1; i >= 0; --i) { while (k >= t && turn(h[k - 2], h[k - 1], pts[i]) <= 0) --k; h[k++] = pts[i]; }
    h.resize(k - 1);
    return h;
}

// cpMomentForPoly about the body origin (models.py:89)
double moment_for_poly(double m, const std::vector<P2> &v)
{
    double s1 = 0, s2 = 0;
    const int n = (int)v.size();
    for (int i = 0; i < n; ++i) {
        const P2 a = v[i], b = v[(i + 1) % n];
        const double cr = b.x * a.y - b.y * a.x;
        s1 += cr * (a.x * a.x + a.y * a.y + a.x * b.x + a.y * b.y + b.x * b.x + b.y * b.y);
        s2 += cr;
    }
    return m * s1 / (6.0 * s2);
}

float round_down(double v) { float f = (float)v; return (double)f > v ? std::nextafterf(f, -INFINITY) : f; }
float round_up(double v) { float f = (float)v; return (double)f < v ? std::nextafterf(f, INFINITY) : f; }
}  // namespace

static int derive_params(shipsim_handle *h)
{
    const shipsim_config &c = h->cfg;
    StepParams &p = h->p;
    std::memset(&p, 0, sizeof(p));
    p.seed = c.seed; p.env_id_offset = c.env_id_offset; p.N = c.num_envs;
    p.history = c.history; p.auto_reset = c.auto_reset; p.max_steps = c.max_steps;
    p.W = c.bounds_w; p.H = c.bounds_h; p.dt = c.dt; p.damping = c.damping;
    p.lidar_len = c.lidar_distance;
    p.goal_r = c.goal_radius; p.step_penalty = c.step_penalty;
    p.spawn_x = c.bounds_w / 2.f; p.spawn_y = c.spawn_y;
    // ship hull: SHIP_TEMPLATE (models.py:6) scaled by (width, height), convexified like pm.Poly does
    const double tpl[5][2] = {{0, 0}, {0, 10}, {5, 15}, {10, 10}, {10, 0}};
    std::vector<P2> raw;
    for (auto &t : tpl) raw.push_back({t[0] * c.ship_w, t[1] * c.ship_h});
    const double moment = moment_for_poly(c.mass, raw);
    std::vector<P2> hull = convex_hull_ccw(raw);
    if ((int)hull.size() != kShipVerts || hull[0].x != 0.0 || hull[0].y != 0.0)
        return fail(SHIPSIM_ERR_ARG, "ship_w / ship_h must be positive");
    double l = 1e300, b = 1e300, r = -1e300, t = -1e300;
    for (int j = 0; j < kShipVerts; ++j) {
        const P2 a = hull[(j + kShipVerts - 1) % kShipVerts], v = hull[j];
        const double ex = v.x - a.x, ey = v.y - a.y, ln = std::sqrt(ex * ex + ey * ey);
        p.ship_lx[j] = (float)v.x; p.ship_ly[j] = (float)v.y;
        p.ship_nx[j] = (float)(ey / ln); p.ship_ny[j] = (float)(-ex / ln);
        p.ship_off[j] = (float)((ey / ln) * v.x + (-ex / ln) * v.y);
        l = std::min(l, v.x); r = std::max(r, v.x); b = std::min(b, v.y); t = std::max(t, v.y);
    }
    p.ship_aabb[0] = (float)l; p.ship_aabb[1] = (float)b; p.ship_aabb[2] = (float)r; p.ship_aabb[3] = (float)t;
    double rmax = 0;
    for (auto &v : hull) rmax = std::max(rmax, std::sqrt(v.x * v.x + v.y * v.y));
    p.goal_cull_r2 = (float)((rmax + c.goal_radius) * (rmax + c.goal_radius) * 1.0001);
    h->ship_reach = (float)(2.0 * rmax);
    p.acc_dt = (float)((double)c.thrust / c.mass * c.dt);
    p.ang_dt = (float)((double)c.thrust / moment * c.dt);
    // lidar fan (models.py:48-49,62)
    const double deg = 3.14159265358979323846 / 180.0;
    const double delta = ((double)c.lidar_spread_deg / c.lidar_beams) * deg;
    const double start = (90.0 - (double)c.lidar_spread_deg / 2.0) * deg;
    const int nb = c.lidar_beams;
    p.n_beams = nb;
    for (int i = 0; i < kBeams; ++i) { p.ray_c[i] = (float)std::cos(start + delta * i); p.ray_s[i] = (float)std::sin(start + delta * i); }
    for (int i = 0; i < kMaxBeams; ++i) { p.ray_cw[i] = (float)std::cos(start + delta * i); p.ray_sw[i] = (float)std::sin(start + delta * i); }
    {
        // the fan-reach cull: the fan's axis and half opening (a single ray: half width 0)
        const double mid = start + delta * (nb - 1) * 0.5, half = std::fabs(delta) * (nb - 1) * 0.5;
        p.fan_cx = (float)std::cos(mid); p.fan_cy = (float)std::sin(mid);
        p.fan_cos = (float)std::cos(half); p.fan_sin = (float)std::sin(half);
        // A fan of half-width >= 180 degrees covers every direction: the bound of plane_at_pose,
        // cos(max(0, angle - half)), is then 1.  cos/sin(half) would wrap around and bound it too low (dropping planes
        // that rays hit), so the cull is switched off: with fan_cos = -1 the bound is 1 (or more) for every plane.
        if (half >= 3.14159265358979323846) { p.fan_cos = -1.f; p.fan_sin = 0.f; }
    }
    // reach grid: kGridN x kGridN cells over the bounds plus a pad (the ray origin of a live env lies within
    // [0, W + ship extent]); the border cells are unbounded
    const double pad = 32.0;
    p.gridp.x0 = (float)(-pad); p.gridp.y0 = (float)(-pad);
    p.gridp.inv_cx = (float)(kGridN / (c.bounds_w + 2.0 * pad));
    p.gridp.inv_cy = (float)(kGridN / (c.bounds_h + 2.0 * pad));
    return SHIPSIM_OK;
}

extern "C" int shipsim_create(const shipsim_config *cfg, int device, shipsim_t **out)
{
    if (!cfg || !out) return fail(SHIPSIM_ERR_ARG, "cfg/out is NULL");
    if (cfg->struct_size != (int32_t)sizeof(shipsim_config)) return fail(SHIPSIM_ERR_ARG, "shipsim_config size mismatch (ABI version?)");
    if (cfg->num_envs < 1) return fail(SHIPSIM_ERR_ARG, "num_envs must be >= 1");
    if (cfg->history < 1) return fail(SHIPSIM_ERR_ARG, "history_size must be greater than zero");   // ship_env.py:46-47
    if (cfg->host_threads < 0) return fail(SHIPSIM_ERR_ARG, "host_threads must be >= 0");
    if (cfg->history > 2) return fail(SHIPSIM_ERR_UNSUPPORTED, "history > 2 is assembled by the host layer from 1-frame observations");
    if (cfg->lidar_beams < 1 || cfg->lidar_beams > kMaxBeams) return fail(SHIPSIM_ERR_ARG, "lidar_beams must be in [1, 32]");
    if (!(cfg->dt > 0.f) || !(cfg->bounds_w > 0.f) || !(cfg->bounds_h > 0.f) || !(cfg->lidar_distance > 0.f) || cfg->max_steps < 1
        || cfg->max_steps >= (1 << 22))
        return fail(SHIPSIM_ERR_ARG, "dt, bounds, lidar_distance must be positive and 1 <= max_steps < 2^22");
    // the ship and goal knobs: a zero mass would give a zero moment and infinite accelerations, a zero scale no hull
    if (!(cfg->mass > 0.f) || !std::isfinite(cfg->mass) || !(cfg->ship_w > 0.f) || !std::isfinite(cfg->ship_w)
        || !(cfg->ship_h > 0.f) || !std::isfinite(cfg->ship_h))
        return fail(SHIPSIM_ERR_ARG, "mass, ship_w and ship_h must be positive and finite");
    if (!(cfg->goal_radius >= 0.f) || !std::isfinite(cfg->goal_radius))
        return fail(SHIPSIM_ERR_ARG, "goal_radius must be >= 0 and finite");
    if (!std::isfinite(cfg->thrust) || !std::isfinite(cfg->lidar_spread_deg) || !std::isfinite(cfg->spawn_y)
        || !std::isfinite(cfg->step_penalty))
        return fail(SHIPSIM_ERR_ARG, "thrust, lidar_spread_deg, spawn_y and step_penalty must be finite");
    {
        const int g = cfg->lanes_per_env;
        if (g != 0 && g != 1 && g != 2 && g != 4 && g != 8 && g != 16 && g != 32)
            return fail(SHIPSIM_ERR_ARG, "lanes_per_env must be 0 (auto), 1, 2, 4, 8, 16 or 32");
        const int w = cfg->steps_in_flight;
        if (w != 0 && w != 1 && w != 4 && w != 8 && w != 16 && w != 32)
            return fail(SHIPSIM_ERR_ARG, "steps_in_flight must be 0 (auto), 1 (off), 4, 8, 16 or 32");
        if (w > 1 && cfg->lidar_beams != SHIPSIM_N_BEAMS)
            return fail(SHIPSIM_ERR_UNSUPPORTED, "steps_in_flight > 1 (the time-parallel kernel) needs lidar_beams = 10");
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SHIPSIM_ERR_CUDA, "no CUDA device: libshipsim has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(SHIPSIM_ERR_ARG, "bad device index");
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(SHIPSIM_ERR_CUDA, "libshipsim is built for sm_100a (B200) only");
    shipsim_handle *h = new shipsim_handle();
    h->cfg = *cfg;
    h->device = device;
    const int rc = derive_params(h);
    if (rc != SHIPSIM_OK) { delete h; return rc; }
    if (cfg->lanes_per_env) {
        h->lanes = cfg->lanes_per_env;
    } else {
        // Auto (measured on B200, profiles/r01_c_sweep_envs_x_lanes.log): batches that fill the machine are issue bound
        // and run one lane per env; small batches are latency bound, so lanes are spent on the cooperative passes --
        // but not beyond 8 per env, since every lane of a group repeats the env's scalar work.
        const int n = cfg->num_envs;
        const int g = n < 8192 ? 8 : (n < 24576 ? 4 : (n < 49152 ? 2 : 1));
        h->lanes = g;
    }
    if (cfg->steps_in_flight) {
        h->window = cfg->steps_in_flight;
    } else {
        // Auto (measured on B200, profiles/r01_k_sweep_window.log): batches too small to fill the machine are bound by
        // the latency of one dependent step after another; the window kernel speculates several steps of an env at
        // once (shipsim_window.cu).  The window is as long as still lets every warp be resident at once (16 warps of
        // 128 registers per SM x 148 SMs = 2,368 warps of 32 / T envs); beyond 32,768 envs the serial-in-time kernel
        // is faster.  An explicit lanes_per_env asks for the serial-in-time kernel.
        const int n = cfg->num_envs;
        // Fans other than 10 beams have no time-parallel kernel: the serial-in-time one runs them at every size.
        h->window = (cfg->lanes_per_env || n > SHIPSIM_WINDOW_AUTO_MAX_ENVS || cfg->lidar_beams != SHIPSIM_N_BEAMS)
                        ? 1 : (n <= 2368 ? 32 : (n <= 4736 ? 16 : 8));
    }
    *out = h;
    return SHIPSIM_OK;
}

extern "C" int shipsim_destroy(shipsim_t *h)
{
    if (!h) return SHIPSIM_OK;
    DeviceGuard g(h->device);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for (auto &ev : h->chunk_done) if (ev) cudaEventDestroy(ev);
    for (auto &ev : h->copy_done) if (ev) cudaEventDestroy(ev);
    if (h->trace0) cudaEventDestroy(h->trace0);
    for (auto &ev : h->trace_mid) if (ev) cudaEventDestroy(ev);
    if (h->fresh.stream) cudaStreamDestroy(h->fresh.stream);
    if (h->fresh.period_begin) cudaEventDestroy(h->fresh.period_begin);
    if (h->fresh.gen_done) cudaEventDestroy(h->fresh.gen_done);
    if (h->h_rec) cudaFreeHost(h->h_rec);
    if (h->h_off) cudaFreeHost(h->h_off);
    if (h->h_count) cudaFreeHost(h->h_count);
    if (h->h_var) cudaFreeHost(h->h_var);
    if (h->h_cur) cudaFreeHost(h->h_cur);
    cudaFree(h->d_rec); cudaFree(h->d_off); cudaFree(h->d_count); cudaFree(h->d_rows); cudaFree(h->d_var);
    if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
    if (h->act_up) cudaEventDestroy(h->act_up);
    cudaFree(h->d_frame0);
    delete h->pool;
    cudaFree(h->d_bank); cudaFree(h->d_edges); cudaFree(h->d_grid); cudaFree(h->d_spawn); cudaFree(h->d_act);
    cudaFree(h->d_gen_xy); cudaFree(h->d_gen_goals); cudaFree(h->d_gen_n); cudaFree(h->d_obs); cudaFree(h->d_rew); cudaFree(h->d_done);
    delete h;
    return SHIPSIM_OK;
}

extern "C" int shipsim_load_scenarios(shipsim_t *h, const double *hull_xy, const int32_t *hull_n, const double *goals_xy,
                                      int32_t n_scen, int32_t maxv)
{
    if (!h || !hull_xy || !hull_n || !goals_xy) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    if (n_scen < 1 || maxv < 3) return fail(SHIPSIM_ERR_ARG, "need n_scenarios >= 1 and maxv >= 3");
    int dev_maxv = 0;
    for (int i = 0; i < n_scen * 2; ++i) {
        if (hull_n[i] < 3 || hull_n[i] > maxv || hull_n[i] > SHIPSIM_MAX_HULL)
            return fail(SHIPSIM_ERR_ARG, "hull vertex count out of range [3, min(maxv, 32)]");
        dev_maxv = std::max(dev_maxv, (int)hull_n[i]);
    }
    const int stride4 = kBankHeader4 + 2 * dev_maxv;
    std::vector<float4> host((size_t)n_scen * stride4, make_float4(0.f, 0.f, 0.f, 0.f));
    std::vector<EdgeD> edges((size_t)n_scen * 2 * kMaxHull);
    std::memset(edges.data(), 0, edges.size() * sizeof(EdgeD));
    // the device geometry is the fp32-rounded polygon: every derived quantity (fp32 planes, double planes, reach
    // grid) is computed in double from the ROUNDED vertices, so the representations agree with each other
    std::vector<double> rxy((size_t)n_scen * 2 * dev_maxv * 2, 0.0);
    for (int s = 0; s < n_scen; ++s) {
        float4 *rec = host.data() + (size_t)s * stride4;
        for (int b = 0; b < 2; ++b) {
            const double *vin = hull_xy + ((size_t)s * 2 + b) * maxv * 2;
            double *v = rxy.data() + ((size_t)s * 2 + b) * dev_maxv * 2;
            const int n = hull_n[s * 2 + b];
            for (int i = 0; i < 2 * n; ++i) v[i] = (double)(float)vin[i];
            double l = 1e300, bo = 1e300, r = -1e300, t = -1e300, area2 = 0;
            for (int i = 0; i < n; ++i) {
                const double ax = v[2 * ((i + n - 1) % n)], ay = v[2 * ((i + n - 1) % n) + 1], bx = v[2 * i], by = v[2 * i + 1];
                area2 += ax * by - ay * bx;
                l = std::min(l, bx); r = std::max(r, bx); bo = std::min(bo, by); t = std::max(t, by);
            }
            if (!(area2 > 0)) return fail(SHIPSIM_ERR_ARG, "bank hulls must be convex and counter-clockwise");
            rec[b] = make_float4(round_down(l), round_down(bo), round_up(r), round_up(t));
            float4 *E = rec + kBankHeader4 + b * dev_maxv;
            EdgeD *ED = edges.data() + ((size_t)s * 2 + b) * kMaxHull;
            for (int i = 0; i < n; ++i) {
                const double ax = v[2 * ((i + n - 1) % n)], ay = v[2 * ((i + n - 1) % n) + 1], bx = v[2 * i], by = v[2 * i + 1];
                const double ex = bx - ax, ey = by - ay, ln = std::sqrt(ex * ex + ey * ey);
                if (!(ln > 0)) return fail(SHIPSIM_ERR_ARG, "degenerate hull edge");
                E[i] = make_float4((float)(ey / ln), (float)(-ex / ln), (float)bx, (float)by);   // cpvrperp: outward for CCW
                ED[i].set_normal(ey / ln, -ex / ln); ED[i].vx = (float)bx; ED[i].vy = (float)by; ED[i].len = (float)ln;
                { const int self = b * kMaxHull + i; std::memcpy(&ED[i].pad, &self, 4); }
            }
        }
        const double *g = goals_xy + (size_t)s * 10;
        rec[2] = make_float4((float)g[0], (float)g[1], (float)g[2], (float)g[3]);
        rec[3] = make_float4((float)g[4], (float)g[5], (float)g[6], (float)g[7]);
        float4 g2 = make_float4((float)g[8], (float)g[9], 0.f, 0.f);
        const int n0 = hull_n[s * 2], n1 = hull_n[s * 2 + 1];
        std::memcpy(&g2.z, &n0, 4); std::memcpy(&g2.w, &n1, 4);
        rec[4] = g2;
    }
    if (n_scen >= (1 << 28)) return fail(SHIPSIM_ERR_ARG, "too many scenarios");
    DeviceGuard g(h->device);
    float4 *d = nullptr;
    EdgeD *de = nullptr;
    uint4 *dg = nullptr;
    float4 *dsp = nullptr;
    double *dxy = nullptr;
    int *dn = nullptr;
    const size_t grid_cells = (size_t)n_scen * kGridN * kGridN;
    auto cleanup = [&]() { cudaFree(d); cudaFree(de); cudaFree(dg); cudaFree(dsp); cudaFree(dxy); cudaFree(dn); };
    cudaError_t e = cudaMalloc(&d, host.size() * sizeof(float4));
    if (e == cudaSuccess) e = cudaMalloc(&de, edges.size() * sizeof(EdgeD));
    if (e == cudaSuccess) e = cudaMalloc(&dg, grid_cells * sizeof(uint4));
    if (e == cudaSuccess) e = cudaMalloc(&dsp, (size_t)n_scen * (1 + 2 * 4) * sizeof(float4)   /* kScr4, shipsim_geom.cuh */);
    if (e == cudaSuccess) e = cudaMalloc(&dxy, rxy.size() * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&dn, (size_t)n_scen * 2 * sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpy(d, host.data(), host.size() * sizeof(float4), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(de, edges.data(), edges.size() * sizeof(EdgeD), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dxy, rxy.data(), rxy.size() * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dn, hull_n, (size_t)n_scen * 2 * sizeof(int), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        // reach grid, built on the device in double (one thread per cell)
        const double pad = -(double)h->p.gridp.x0;
        const double cw = ((double)h->cfg.bounds_w + 2.0 * pad) / kGridN, ch = ((double)h->cfg.bounds_h + 2.0 * pad) / kGridN;
        const double margin = 0.05 + 1e-4 * std::max((double)h->cfg.bounds_w, (double)h->cfg.bounds_h);
        // the cell is looked up at the LIDAR ORIGIN, and its masks also decide "bank not near => no ship-vs-bank test":
        // the reach must cover the hull as seen from that origin (every hull point lies within 2 * max |hull vertex|)
        const double reach = std::max({(double)h->cfg.lidar_distance, (double)h->ship_reach, std::sqrt(cw * cw + ch * ch)}) + margin;
        e = launch_build_grid(dxy, dn, n_scen, dev_maxv, (double)h->p.gridp.x0, (double)h->p.gridp.y0, cw, ch, reach, margin, dg, 0);
    }
    if (e == cudaSuccess) {
        // plane phase at the spawn pose of every scenario (what an env that is reset inside the kernel starts from)
        StepParams q = h->p;
        q.bank = d; q.edges_d = de; q.grid = dg; q.n_scen = n_scen; q.maxv = dev_maxv; q.scen_stride4 = stride4; q.hull_max = dev_maxv;
        e = launch_build_spawn_rows(q, dsp, 0);
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();           // also: no launch may still be reading the old bank
    if (e != cudaSuccess) { cleanup(); return fail(SHIPSIM_ERR_CUDA, cudaGetErrorString(e)); }
    cudaFree(dxy); cudaFree(dn);
    cudaFree(h->d_bank); cudaFree(h->d_edges); cudaFree(h->d_grid); cudaFree(h->d_spawn);
    h->d_bank = d; h->d_edges = de; h->d_grid = dg; h->d_spawn = dsp;
    h->p.bank = d; h->p.edges_d = de; h->p.grid = dg; h->p.spawn_rows = dsp;
    const int old_n = h->p.n_scen;
    h->p.n_scen = n_scen; h->p.maxv = dev_maxv; h->p.scen_stride4 = stride4; h->p.hull_max = dev_maxv;
    h->fresh.on = false; h->fresh.pending = false; h->p.pick_base = 0; h->p.pick_count = 0;     // (a host bank cannot be regenerated)
    h->launches += 2;
    if (h->p.state && n_scen < old_n) {      // live envs may hold ids of the old, larger bank
        CU(launch_clamp_scenarios(h->p.state, h->cfg.num_envs, n_scen, 0));
        CU(cudaDeviceSynchronize());
        h->launches++;
    }
    return SHIPSIM_OK;
}

// ---- scenario generation on the device (SURVEY.md §8 f2) ------------------------------------------------------
extern "C" int shipsim_generate_scenarios(shipsim_t *h, int32_t n_scen, uint64_t seed, int32_t map_N, float width_frac, void *stream)
{
    if (!h) return fail(SHIPSIM_ERR_ARG, "handle is NULL");
    if (n_scen < 1 || n_scen >= (1 << 28)) return fail(SHIPSIM_ERR_ARG, "n_scenarios out of range");
    if (map_N < 1 || map_N > kMaxHull - 2) return fail(SHIPSIM_ERR_ARG, "map_N must be in [1, 30] (two wall corners are added; hulls hold 32 vertices)");
    if (!(width_frac > 0.f) || !(width_frac <= 1.f)) return fail(SHIPSIM_ERR_ARG, "width_frac must be in (0, 1]");
    DeviceGuard g(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int maxv = kMaxHull, stride4 = kBankHeader4 + 2 * maxv;
    float4 *d = nullptr, *dsp = nullptr;
    EdgeD *de = nullptr;
    uint4 *dg = nullptr;
    double *dxy = nullptr, *dgo = nullptr;
    int *dn = nullptr, *dmax = nullptr;
    auto cleanup = [&]() { cudaFree(d); cudaFree(de); cudaFree(dg); cudaFree(dsp); cudaFree(dxy); cudaFree(dgo); cudaFree(dn); cudaFree(dmax); };
    cudaError_t e = cudaMalloc(&d, (size_t)n_scen * stride4 * sizeof(float4));
    if (e == cudaSuccess) e = cudaMalloc(&de, (size_t)n_scen * 2 * kMaxHull * sizeof(EdgeD));
    if (e == cudaSuccess) e = cudaMalloc(&dg, (size_t)n_scen * kGridN * kGridN * sizeof(uint4));
    if (e == cudaSuccess) e = cudaMalloc(&dsp, (size_t)n_scen * (1 + 2 * 4) * sizeof(float4)   /* kScr4, shipsim_geom.cuh */);
    if (e == cudaSuccess) e = cudaMalloc(&dxy, (size_t)n_scen * 2 * kMaxHull * 2 * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&dgo, (size_t)n_scen * 10 * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&dn, (size_t)n_scen * 2 * sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc(&dmax, sizeof(int));
    if (e == cudaSuccess) e = cudaMemsetAsync(d, 0, (size_t)n_scen * stride4 * sizeof(float4), s);
    if (e == cudaSuccess) e = cudaMemsetAsync(de, 0, (size_t)n_scen * 2 * kMaxHull * sizeof(EdgeD), s);
    if (e == cudaSuccess) e = launch_gen_scenarios(seed, n_scen, h->cfg.bounds_w, h->cfg.bounds_h, map_N, width_frac, dxy, dn, dgo, s);
    if (e == cudaSuccess) e = launch_max_hull(dn, n_scen * 2, dmax, s);
    if (e == cudaSuccess) e = launch_pack_bank(dxy, dn, dgo, n_scen, maxv, stride4, d, de, s);
    if (e == cudaSuccess) {
        const double pad = -(double)h->p.gridp.x0;
        const double cw = ((double)h->cfg.bounds_w + 2.0 * pad) / kGridN, ch = ((double)h->cfg.bounds_h + 2.0 * pad) / kGridN;
        const double margin = 0.05 + 1e-4 * std::max((double)h->cfg.bounds_w, (double)h->cfg.bounds_h);
        // the cell is looked up at the LIDAR ORIGIN, and its masks also decide "bank not near => no ship-vs-bank test":
        // the reach must cover the hull as seen from that origin (every hull point lies within 2 * max |hull vertex|)
        const double reach = std::max({(double)h->cfg.lidar_distance, (double)h->ship_reach, std::sqrt(cw * cw + ch * ch)}) + margin;
        e = launch_build_grid(dxy, dn, n_scen, kMaxHull, (double)h->p.gridp.x0, (double)h->p.gridp.y0, cw, ch, reach, margin, dg, s);
    }
    int hull_max = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&hull_max, dmax, sizeof(int), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);          // 4-byte read-back: the SAT pass lane layout depends on it
    if (e == cudaSuccess) {
        StepParams q = h->p;
        q.bank = d; q.edges_d = de; q.grid = dg; q.n_scen = n_scen; q.maxv = maxv; q.scen_stride4 = stride4; q.hull_max = hull_max;
        e = launch_build_spawn_rows(q, dsp, s);
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();            // no launch may still be reading the old bank
    if (e != cudaSuccess) { cleanup(); return fail(SHIPSIM_ERR_CUDA, cudaGetErrorString(e)); }
    cudaFree(dmax);
    cudaFree(h->d_bank); cudaFree(h->d_edges); cudaFree(h->d_grid); cudaFree(h->d_spawn);
    cudaFree(h->d_gen_xy); cudaFree(h->d_gen_goals); cudaFree(h->d_gen_n);
    h->d_bank = d; h->d_edges = de; h->d_grid = dg; h->d_spawn = dsp;
    h->d_gen_xy = dxy; h->d_gen_goals = dgo; h->d_gen_n = dn; h->gen_count = n_scen;
    h->fresh.on = false; h->fresh.pending = false; h->fresh.map_N = map_N; h->fresh.width_frac = width_frac; h->fresh.seed = seed;
    h->p.pick_base = 0; h->p.pick_count = 0;
    h->p.bank = d; h->p.edges_d = de; h->p.grid = dg; h->p.spawn_rows = dsp;
    const int old_n = h->p.n_scen;
    h->p.n_scen = n_scen; h->p.maxv = maxv; h->p.scen_stride4 = stride4; h->p.hull_max = hull_max;
    h->launches += 5;
    if (h->p.state && n_scen < old_n) {
        CU(launch_clamp_scenarios(h->p.state, h->cfg.num_envs, n_scen, s));
        CU(cudaStreamSynchronize(s));
        h->launches++;
    }
    return SHIPSIM_OK;
}

extern "C" int shipsim_read_scenarios(shipsim_t *h, double *host_hull_xy, int32_t *host_hull_n, double *host_goals)
{
    if (!h || !host_hull_xy || !host_hull_n || !host_goals) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    if (!h->d_gen_xy) return fail(SHIPSIM_ERR_STATE, "no device-generated bank: call shipsim_generate_scenarios first");
    DeviceGuard g(h->device);
    const size_t S = (size_t)h->gen_count;
    CU(cudaMemcpy(host_hull_xy, h->d_gen_xy, S * 2 * kMaxHull * 2 * sizeof(double), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(host_hull_n, h->d_gen_n, S * 2 * sizeof(int), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(host_goals, h->d_gen_goals, S * 10 * sizeof(double), cudaMemcpyDeviceToHost));
    return SHIPSIM_OK;
}

// ---- fresh maps (SURVEY.md section 8 f2; ShipGame.reset builds a new level every time: game.py:271-272) -------------
// The device-generated bank is cut into four slices.  Resets of period p (a period = at least max_steps env-steps, so
// every episode that began in it ends before the next period does) pick from slice p % 4; slice (p + 1) % 4 -- last
// picked from in period p - 3, drained during p - 2 -- is regenerated with a new seed on a side stream while period p
// runs.  No map is played after the period following the one it was picked in, and none comes back.
static uint64_t fresh_seed(uint64_t seed, int period) { return seed + 0x9E3779B97F4A7C15ull * (uint64_t)(period + 1); }

static int fresh_regenerate(shipsim_t *h, int slice, uint64_t seed)
{
    const int q = h->gen_count / 4;
    const int maxv = kMaxHull, stride4 = kBankHeader4 + 2 * maxv;
    const size_t s0 = (size_t)slice * q;
    cudaStream_t gs = h->fresh.stream;
    double *dxy = h->d_gen_xy + s0 * 2 * kMaxHull * 2, *dgo = h->d_gen_goals + s0 * 10;
    int *dn = h->d_gen_n + s0 * 2;
    float4 *d = h->d_bank + s0 * stride4, *dsp = h->d_spawn + s0 * (1 + 2 * 4);
    EdgeD *de = h->d_edges + s0 * 2 * kMaxHull;
    uint4 *dg = h->d_grid + s0 * kGridN * kGridN;
    CU(cudaMemsetAsync(d, 0, (size_t)q * stride4 * sizeof(float4), gs));
    CU(cudaMemsetAsync(de, 0, (size_t)q * 2 * kMaxHull * sizeof(EdgeD), gs));
    CU(launch_gen_scenarios(seed, q, h->cfg.bounds_w, h->cfg.bounds_h, h->fresh.map_N, h->fresh.width_frac, dxy, dn, dgo, gs));
    CU(launch_pack_bank(dxy, dn, dgo, q, maxv, stride4, d, de, gs));
    const double pad = -(double)h->p.gridp.x0;
    const double cw = ((double)h->cfg.bounds_w + 2.0 * pad) / kGridN, ch = ((double)h->cfg.bounds_h + 2.0 * pad) / kGridN;
    const double margin = 0.05 + 1e-4 * std::max((double)h->cfg.bounds_w, (double)h->cfg.bounds_h);
    const double reach = std::max({(double)h->cfg.lidar_distance, (double)h->ship_reach, std::sqrt(cw * cw + ch * ch)}) + margin;
    CU(launch_build_grid(dxy, dn, q, kMaxHull, (double)h->p.gridp.x0, (double)h->p.gridp.y0, cw, ch, reach, margin, dg, gs));
    StepParams sp = h->p;
    sp.bank = d; sp.edges_d = de; sp.grid = dg; sp.n_scen = q;
    CU(launch_build_spawn_rows(sp, dsp, gs));
    h->launches += 4;
    return SHIPSIM_OK;
}

// called before every step launch: moves on to the next period when the current one has lasted long enough
static int fresh_tick(shipsim_t *h, int K, cudaStream_t s)
{
    auto &f = h->fresh;
    if (!f.on) return SHIPSIM_OK;
    f.max_steps = std::max(f.max_steps, h->cfg.max_steps);
    if (f.steps >= f.max_steps) {
        f.period++;
        f.steps = 0;
        const int q = h->gen_count / 4, slice = f.period % 4;
        if (f.pending) {                                 // this period's slice was regenerated while the last one ran
            CU(cudaStreamWaitEvent(s, f.gen_done, 0));
            f.pending = false;
        }
        h->p.pick_base = slice * q;
        if (f.period + 1 >= 4) {                         // the slice after this one has been played: new maps for it
            const int nxt = (f.period + 1) % 4;
            CU(cudaEventRecord(f.period_begin, s));      // every launch that could still read it precedes this point
            CU(cudaStreamWaitEvent(f.stream, f.period_begin, 0));
            const int rc = fresh_regenerate(h, nxt, fresh_seed(f.seed, f.period + 1));
            if (rc) return rc;
            CU(cudaEventRecord(f.gen_done, f.stream));
            f.generation[nxt]++;
            f.pending = true;
        }
    }
    f.steps += K;
    return SHIPSIM_OK;
}

extern "C" int shipsim_fresh_maps(shipsim_t *h, int32_t enable)
{
    if (!h) return fail(SHIPSIM_ERR_ARG, "handle is NULL");
    DeviceGuard g(h->device);
    auto &f = h->fresh;
    if (!enable) {
        if (f.on) CU(cudaStreamSynchronize(f.stream));
        f.on = false; f.pending = false;
        h->p.pick_base = 0; h->p.pick_count = 0;
        return SHIPSIM_OK;
    }
    if (!h->d_gen_xy || h->p.bank != h->d_bank || h->gen_count != h->p.n_scen)
        return fail(SHIPSIM_ERR_STATE, "fresh maps need a device-generated bank: call shipsim_generate_scenarios first");
    const int q = h->gen_count / 4;
    if (h->gen_count % 4 != 0 || q < 1 || (q & (q - 1)) != 0)
        return fail(SHIPSIM_ERR_ARG, "fresh maps need a bank of 4 * 2^k scenarios");
    if (!h->cfg.auto_reset) return fail(SHIPSIM_ERR_STATE, "fresh maps need auto_reset (an env that is never reset would outlive its map)");
    if (!f.stream) {
        CU(cudaStreamCreateWithFlags(&f.stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&f.period_begin, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&f.gen_done, cudaEventDisableTiming));
    }
    f.on = true; f.pending = false; f.period = 0; f.steps = 0; f.max_steps = h->cfg.max_steps;
    for (int &gen : f.generation) gen = 0;
    h->p.pick_base = 0; h->p.pick_count = q;
    h->p.hull_max = std::max(h->p.hull_max, std::min(kMaxHull, f.map_N + 2));   // regenerated hulls: at most map_N + 2 vertices
    return SHIPSIM_OK;
}

extern "C" int shipsim_fresh_info(const shipsim_t *h, int32_t *info)
{
    if (!h || !info) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    info[0] = h->fresh.on ? 1 : 0; info[1] = h->fresh.period; info[2] = h->p.pick_base; info[3] = h->p.pick_count;
    for (int i = 0; i < 4; ++i) info[4 + i] = h->fresh.generation[i];
    return SHIPSIM_OK;
}

extern "C" int shipsim_set_max_steps(shipsim_t *h, int32_t max_steps)
{
    if (!h) return fail(SHIPSIM_ERR_ARG, "handle is NULL");
    if (max_steps < 1 || max_steps >= (1 << 22)) return fail(SHIPSIM_ERR_ARG, "need 1 <= max_steps < 2^22");
    h->cfg.max_steps = max_steps;
    h->p.max_steps = max_steps;
    return SHIPSIM_OK;
}

static int state_planes(const shipsim_t *h) { return kPlanes + extra_lidar_planes(h->cfg.lidar_beams); }
static int frame_floats(const shipsim_t *h) { return 6 + h->cfg.lidar_beams; }      // ShipEnv.n_states (ship_env.py:43)

extern "C" size_t shipsim_state_bytes(const shipsim_t *h) { return h ? (size_t)h->cfg.num_envs * state_planes(h) * sizeof(float4) : 0; }
extern "C" size_t shipsim_stats_bytes(const shipsim_t *) { return (size_t)kStatSlots * kStatLen * sizeof(double); }

extern "C" int shipsim_bind_state(shipsim_t *h, void *dev_state, void *dev_stats, void *stream)
{
    if (!h || !dev_state || !dev_stats) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    if (((uintptr_t)dev_state & 15) || ((uintptr_t)dev_stats & 7)) return fail(SHIPSIM_ERR_ARG, "state must be 16-byte aligned");
    DeviceGuard g(h->device);
    h->p.state = (float4 *)dev_state;
    h->p.stats = (double *)dev_stats;
    CU(cudaMemsetAsync(dev_stats, 0, shipsim_stats_bytes(h), (cudaStream_t)stream));
    return SHIPSIM_OK;
}

static int ready(const shipsim_t *h)
{
    if (!h) return fail(SHIPSIM_ERR_ARG, "handle is NULL");
    if (!h->p.bank) return fail(SHIPSIM_ERR_STATE, "shipsim_load_scenarios has not been called");
    if (!h->p.state) return fail(SHIPSIM_ERR_STATE, "shipsim_bind_state has not been called");
    return SHIPSIM_OK;
}

extern "C" int shipsim_reset(shipsim_t *h, const uint8_t *dev_mask, const int32_t *dev_scenario, int first, float *dev_obs, void *stream)
{
    const int rc = ready(h);
    if (rc) return rc;
    DeviceGuard g(h->device);
    CU(launch_reset(h->p, dev_mask, dev_scenario, first, (float4 *)dev_obs, (cudaStream_t)stream));
    h->launches++;
    return SHIPSIM_OK;
}

extern "C" int shipsim_episode_log_bind(shipsim_t *h, float *dev_rows, int32_t *dev_meta, int32_t capacity, int32_t *dev_count)
{
    if (!h) return fail(SHIPSIM_ERR_ARG, "handle is NULL");
    StepParams &p = h->p;
    if (capacity == 0) {
        p.log_rows = nullptr; p.log_meta = nullptr; p.log_count = nullptr; p.log_cap = 0; p.log_row4 = 0;
        return SHIPSIM_OK;
    }
    if (!h->cfg.auto_reset) return fail(SHIPSIM_ERR_STATE, "the episode log needs auto_reset (without it the caller sees the terminal rows)");
    if (capacity < 0 || !dev_rows || !dev_meta || !dev_count) return fail(SHIPSIM_ERR_ARG, "NULL buffer or capacity < 0");
    if (((uintptr_t)dev_rows & 15) || ((uintptr_t)dev_meta & 15) || ((uintptr_t)dev_count & 3))
        return fail(SHIPSIM_ERR_ARG, "dev_rows / dev_meta must be 16-byte aligned");
    DeviceGuard g(h->device);
    // rows and metadata may sit in page-locked host memory (written over PCIe): the kernels need its device alias
    auto device_alias = [](void *ptr) {
        cudaPointerAttributes attr{};
        const bool host = cudaPointerGetAttributes(&attr, ptr) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer;
        cudaGetLastError();
        return host ? attr.devicePointer : ptr;
    };
    {
        cudaPointerAttributes attr{};
        const bool dev = cudaPointerGetAttributes(&attr, dev_count) == cudaSuccess && attr.type == cudaMemoryTypeDevice;
        cudaGetLastError();
        if (!dev) return fail(SHIPSIM_ERR_ARG, "dev_count must be device memory (it is the target of device atomics)");
    }
    p.log_rows = (float4 *)device_alias(dev_rows);
    p.log_meta = (int4 *)device_alias(dev_meta);
    p.log_count = (int *)dev_count;
    p.log_cap = capacity;
    p.log_row4 = 4 * h->cfg.history;         // (the wide kernel's rows are dense: (6 + lidar_beams) * history floats)
    return SHIPSIM_OK;
}

static int step_impl(shipsim_t *h, const void *dev_actions, int action_dtype, int32_t K, float *dev_obs, float *dev_reward,
                     uint8_t *dev_done, void *stream, int history)
{
    const int rc = ready(h);
    if (rc) return rc;
    if (K < 1) return fail(SHIPSIM_ERR_ARG, "K must be >= 1");
    if (action_dtype < 0 || action_dtype > 3) return fail(SHIPSIM_ERR_ARG, "bad action_dtype");
    if (action_dtype != SHIPSIM_ACTION_RANDOM && !dev_actions) return fail(SHIPSIM_ERR_ARG, "dev_actions is NULL");
    // (the tuned 10-beam kernel stores rows as float4; the wide kernel's rows are dense floats)
    if ((uintptr_t)dev_obs & (h->cfg.lidar_beams == SHIPSIM_N_BEAMS ? 15 : 3))
        return fail(SHIPSIM_ERR_ARG, h->cfg.lidar_beams == SHIPSIM_N_BEAMS ? "dev_obs must be 16-byte aligned" : "dev_obs must be 4-byte aligned");
    DeviceGuard g(h->device);
    {
        const int rcf = fresh_tick(h, K, (cudaStream_t)stream);
        if (rcf) return rcf;
    }
    StepParams p = h->p;
    p.actions = dev_actions; p.action_dtype = action_dtype; p.K = K;
    p.obs = (float4 *)dev_obs; p.reward = dev_reward; p.done = dev_done;
    p.history = history;
    // the window kernel needs the actions of the whole rollout up front and at least one full window of steps
    if (h->window > 1 && K >= h->window) CU(launch_window(p, h->window, (cudaStream_t)stream, &h->shape));
    else CU(launch_step(p, h->lanes, (cudaStream_t)stream, &h->shape));
    h->p.step0 += (unsigned)K;
    h->launches++;
    return SHIPSIM_OK;
}

extern "C" int shipsim_step(shipsim_t *h, const void *dev_actions, int action_dtype, int32_t K, float *dev_obs, float *dev_reward,
                            uint8_t *dev_done, void *stream)
{
    if (h) { h->p.log_call = h->calls++; h->p.log_k0 = 0; }
    return step_impl(h, dev_actions, action_dtype, K, dev_obs, dev_reward, dev_done, stream, h ? h->p.history : 1);
}

extern "C" int shipsim_step_host(shipsim_t *h, const int32_t *host_actions, int32_t K, float *host_obs, float *host_reward,
                                 uint8_t *host_done, void *stream)
{
    const int rc = ready(h);
    if (rc) return rc;
    if (K < 1 || !host_actions) return fail(SHIPSIM_ERR_ARG, "K must be >= 1 and host_actions non-NULL");
    DeviceGuard g(h->device);
    h->p.log_call = h->calls++;
    h->p.log_k0 = 0;
    const size_t N = (size_t)h->cfg.num_envs;
    const size_t n = N * K;
    // With HISTORY_SIZE = 2 an observation is [frame of the previous step | frame of this step] (ship_env.py:112-113):
    // half of every row repeats the row before it, and between consecutive frames of an env little changes besides the
    // pose.  The kernel runs in its one-frame mode.  The caller's rows are then produced by two engines at once, because
    // either alone is the bottleneck (PCIe at ~55 GB/s for 128-byte rows; the host cores' stores for the expansion):
    //  * envs [0, nd): complete rows are put together on the device (history_rows_kernel) and DMA-ed straight into the
    //    caller's buffer (when it is page-locked);
    //  * envs [nd, N): a kernel turns the frames into 16-byte records + a stream of changed values (~20 bytes per
    //    env-step instead of 64 + 5) and host threads rebuild the rows -- reset observations included;
    // chunk by chunk, while later chunks are still being computed.  nd follows the measured balance of the two.
    // (Small calls -- a gym-style caller stepping a handful of envs one step at a time -- are latency bound: for them the
    // kernel writes complete rows and everything, copies included, goes through the caller's stream with one wait.)
    const bool small = n < ((size_t)1 << 16);
    // Tiny calls with page-locked buffers (the gym facade: one env, one step): no copies at all -- the kernel reads the
    // actions from the caller's memory and writes rows, rewards and done flags straight into it (mapped pinned memory;
    // a few hundred bytes over PCIe), one launch and one wait.
    const size_t F = (size_t)frame_floats(h);                       // floats per frame
    if (n * F * h->cfg.history * sizeof(float) <= ((size_t)1 << 16) && host_obs && host_reward && host_done) {
        auto mapped = [&](const void *ptr, void **dev) {
            cudaPointerAttributes attr{};
            const bool ok = cudaPointerGetAttributes(&attr, ptr) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer;
            cudaGetLastError();
            if (ok) *dev = attr.devicePointer;
            return ok;
        };
        void *da = nullptr, *dobs = nullptr, *dr = nullptr, *dd = nullptr;
        bool all = false;
        if (h->zc_host[0] == host_actions && h->zc_host[1] == host_obs && h->zc_host[2] == host_reward && h->zc_host[3] == host_done) {
            da = h->zc_dev[0]; dobs = h->zc_dev[1]; dr = h->zc_dev[2]; dd = h->zc_dev[3];
            all = da != nullptr;
        } else if (mapped(host_actions, &da) && mapped(host_obs, &dobs) && mapped(host_reward, &dr) && mapped(host_done, &dd)) {
            h->zc_host[0] = host_actions; h->zc_host[1] = host_obs; h->zc_host[2] = host_reward; h->zc_host[3] = host_done;
            h->zc_dev[0] = da; h->zc_dev[1] = dobs; h->zc_dev[2] = dr; h->zc_dev[3] = dd;
            all = true;
        } else {
            h->zc_host[0] = host_actions; h->zc_host[1] = host_obs; h->zc_host[2] = host_reward; h->zc_host[3] = host_done;
            h->zc_dev[0] = h->zc_dev[1] = h->zc_dev[2] = h->zc_dev[3] = nullptr;                 // (remembered as not mapped)
        }
        if (all) {
            const int rc2 = step_impl(h, da, SHIPSIM_ACTION_I32, K, (float *)dobs, (float *)dr, (uint8_t *)dd, stream, h->cfg.history);
            if (rc2) return rc2;
            h->last_h2d = (int64_t)(n * sizeof(int32_t));
            h->last_d2h = (int64_t)(n * (F * h->cfg.history * sizeof(float) + 5));
            CU(cudaStreamSynchronize((cudaStream_t)stream));
            return SHIPSIM_OK;
        }
    }
    // (the compacted wire format is that of 16-float frames: other fans take the plain copies)
    const bool frames_only = h->cfg.history == 2 && host_obs != nullptr && !small && h->cfg.lidar_beams == SHIPSIM_N_BEAMS;
    int nd = 0;                                                      // envs [0, nd) by DMA (frames_only)
    bool adaptive = false;
    if (K > h->stage_K) {
        cudaFree(h->d_act); cudaFree(h->d_obs); cudaFree(h->d_rew); cudaFree(h->d_done);
        h->d_act = nullptr; h->d_obs = nullptr; h->d_rew = nullptr; h->d_done = nullptr; h->stage_K = 0;
        CU(cudaMalloc(&h->d_act, n * sizeof(int32_t)));
        CU(cudaMalloc(&h->d_obs, n * F * h->cfg.history * sizeof(float)));
        CU(cudaMalloc(&h->d_rew, n * sizeof(float)));
        CU(cudaMalloc(&h->d_done, n));
        h->stage_K = K;
    }
    cudaStream_t s = (cudaStream_t)stream;
    if (!h->copy_stream) {
        CU(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        const unsigned evf = std::getenv("SHIPSIM_HOST_TRACE") ? cudaEventDefault : cudaEventDisableTiming;
        for (auto &ev : h->chunk_done) CU(cudaEventCreateWithFlags(&ev, evf));
        for (auto &ev : h->copy_done) CU(cudaEventCreateWithFlags(&ev, evf));
        CU(cudaEventCreateWithFlags(&h->trace0, evf));
        CU(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&h->act_up, cudaEventDisableTiming));
        if (std::getenv("SHIPSIM_HOST_TRACE")) for (auto &ev : h->trace_mid) CU(cudaEventCreate(&ev));
    }
    int n_chunks = small ? 1 : (K >= 64 ? 16 : (K >= 8 ? 8 : 1));
    if (const char *ev = std::getenv("SHIPSIM_HOST_CHUNKS")) n_chunks = std::max(1, std::min({atoi(ev), (int)shipsim_handle::kMaxChunks, (int)K}));
    int kbeg[shipsim_handle::kMaxChunks + 1];
    for (int c = 0; c <= n_chunks; ++c) kbeg[c] = (int)((int64_t)K * c / n_chunks);
    const size_t nblk = (N + 31) / 32;
    for (int c = 0; c < n_chunks; ++c)
        if (kbeg[c + 1] <= kbeg[c]) return fail(SHIPSIM_ERR_ARG, "internal: empty chunk");
    if (frames_only) {
        // Value stream: room for all 12 variable slots of every env-step (measured need on the default map: 0.9), so
        // that it cannot overflow; untouched pages of the mapping cost nothing.
        h->var_per_step = 12;
        if (n > h->rec_cap) {
            cudaFree(h->d_rec); cudaFree(h->d_off); cudaFree(h->d_count);
            if (h->h_rec) cudaFreeHost(h->h_rec);
            if (h->h_off) cudaFreeHost(h->h_off);
            if (h->h_count) cudaFreeHost(h->h_count);
            if (h->h_var) cudaFreeHost(h->h_var);
            cudaFree(h->d_var); h->d_var = nullptr;
            h->d_rec = nullptr; h->d_off = nullptr; h->d_count = nullptr; h->h_rec = nullptr; h->h_off = nullptr; h->h_count = nullptr;
            h->h_var = nullptr; h->rec_cap = 0;
            CU(cudaMalloc(&h->d_rec, n * sizeof(uint4)));
            CU(cudaMalloc(&h->d_off, (size_t)K * nblk * sizeof(unsigned)));
            CU(cudaMalloc(&h->d_count, shipsim_handle::kMaxChunks * sizeof(unsigned)));
            CU(cudaHostAlloc(&h->h_rec, n * sizeof(uint4), cudaHostAllocDefault));
            CU(cudaHostAlloc(&h->h_off, (size_t)K * nblk * sizeof(unsigned), cudaHostAllocDefault));
            CU(cudaHostAlloc(&h->h_count, shipsim_handle::kMaxChunks * sizeof(unsigned), cudaHostAllocDefault));
            CU(cudaHostAlloc(&h->h_var, n * h->var_per_step * sizeof(float), cudaHostAllocDefault));
            CU(cudaMalloc(&h->d_var, n * h->var_per_step * sizeof(float)));
            h->rec_cap = n;
        }
        if (N > h->cur_cap) {
            if (h->h_cur) cudaFreeHost(h->h_cur);
            h->h_cur = nullptr; h->cur_cap = 0;
            CU(cudaHostAlloc(&h->h_cur, N * kFrame * sizeof(float), cudaHostAllocDefault));
            h->cur_cap = N;
        }
        if (!h->d_frame0) CU(cudaMalloc(&h->d_frame0, N * kFrame * sizeof(float)));
        if (!h->pool) {
            int nt = std::max(1, std::min(16, (int)std::thread::hardware_concurrency()));
            if (h->cfg.host_threads > 0) nt = std::min(h->cfg.host_threads, 256);
            if (const char *ev = std::getenv("SHIPSIM_HOST_THREADS")) nt = std::max(1, atoi(ev));
            h->pool = new HostPool(nt - 1);
        }
        CU(launch_frame(h->p, h->d_frame0, s));
        CU(cudaMemsetAsync(h->d_count, 0, shipsim_handle::kMaxChunks * sizeof(unsigned), s));
        h->launches++;
        // how many envs travel as complete rows
        cudaPointerAttributes attr{};
        const bool pinned = cudaPointerGetAttributes(&attr, host_obs) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        cudaGetLastError();
        const char *fixed = std::getenv("SHIPSIM_HOST_DMA_ENVS");
        if (!pinned) nd = 0;
        else if (fixed) nd = std::max(0, std::min(atoi(fixed), (int)N));
        else if (n < ((size_t)1 << 18)) nd = 0;                       // (small calls are latency bound either way)
        else {
            adaptive = true;
            if (h->dma_envs < 0 || h->dma_for_n != (int)N || h->dma_for_k != K) {
                // First guess.  With a core per ~4 GB/s of rows the host threads alone are the faster engine, and DMA
                // writes landing next to their streaming stores slow both (B200 box, 16 cores: 6.4 ms per 4,096 x 1,000
                // call with the host threads alone, 8-10 ms with any share by DMA; profiles/r02_e2e_sweep.log); with few
                // cores per GPU the copy engine has to carry most of it.
                const int thr = h->pool->size();
                h->dma_envs = thr >= 8 ? 0 : (int)((double)N * 50.0 / (50.0 + 9.0 * thr));
                h->dma_for_n = (int)N; h->dma_for_k = K;
                h->dma_step = std::max(32, (int)(N / 8) / 32 * 32);
                h->dma_dir = 1;
                h->dma_last_t = 0.0;
            }
            nd = h->dma_envs;
        }
        nd = nd >= (int)N ? (int)N : (nd / 32) * 32;
        if ((size_t)nd * K > h->rows_cap) {
            cudaFree(h->d_rows);
            h->d_rows = nullptr; h->rows_cap = 0;
            CU(cudaMalloc(&h->d_rows, (size_t)nd * K * 2 * kFrame * sizeof(float)));
            h->rows_cap = (size_t)nd * K;
        }
    }
    const bool trace = std::getenv("SHIPSIM_HOST_TRACE") != nullptr;
    if (trace) CU(cudaEventRecord(h->trace0, s));
    h->last_h2d = (int64_t)(n * sizeof(int32_t));                   // (the actions go up chunk by chunk, ahead of the chunk's kernel)
    h->last_d2h = 0;
    // The rollout is cut into chunks of steps: while chunk i+1 is being computed on the caller's stream, the results
    // of chunk i travel to the host on the copy stream and chunk i-1 is being expanded by the host threads.
    const size_t row_full = F * h->cfg.history;                     // floats per complete row; chunk regions of d_obs are sized for it
    float *d_var = h->d_var;
    if (const char *ev = std::getenv("SHIPSIM_HOST_VAR_DENSITY")) h->var_density = atof(ev);      // (test hook: 0 forces the fetch-the-rest path)
    size_t spec[shipsim_handle::kMaxChunks] = {};                    // floats of each chunk's value stream copied down unasked
    // Every host thread owns a contiguous range of env blocks for the whole call (the running frames of its envs stay in its
    // cache) and walks the chunks as their records arrive: no barrier between chunks.  Whoever finds the next chunk missing
    // polls its event.  The threads are started BEFORE the stream work is issued (launching 16 chunks of kernels and copies
    // takes the calling thread ~1 ms, a fifth of the call), and the calling thread joins them when it is done.
    const bool expand = frames_only && nd < (int)N;
    const bool cut = h->cfg.auto_reset != 0;
    const size_t blk0 = (size_t)nd / 32;
    const int jobs = expand ? (int)std::min<size_t>(nblk - blk0, (size_t)h->pool->size()) : 0;
    std::atomic<int> ready{0};                                       // chunks whose records are in host memory
    std::atomic<int> issued{0};                                      // chunks whose copies (and event) are in the copy stream
    std::atomic<int> bad{0};
    std::mutex poll, fix;
    bool fixed[shipsim_handle::kMaxChunks] = {};
    std::atomic<long long> extra_d2h{0};
    const int dev = h->device;
    const std::function<void(int)> worker = [&](int j) {
        cudaSetDevice(dev);
        const size_t b0 = blk0 + (nblk - blk0) * (size_t)j / jobs, b1 = blk0 + (nblk - blk0) * (size_t)(j + 1) / jobs;
        for (int c = 0; c < n_chunks; ++c) {
            while (ready.load(std::memory_order_acquire) <= c) {
                if (bad.load(std::memory_order_relaxed)) return;
                if (poll.try_lock()) {
                    const int r = ready.load(std::memory_order_relaxed);
                    if (r <= c && r < issued.load(std::memory_order_acquire)) {      // (an event not yet recorded by this call reads as complete)
                        const cudaError_t q = cudaEventQuery(h->copy_done[r]);
                        if (q == cudaSuccess) ready.store(r + 1, std::memory_order_release);
                        else if (q != cudaErrorNotReady) bad.store((int)q);
                    }
                    poll.unlock();
                }
#if defined(__x86_64__)
                __builtin_ia32_pause();
#endif
            }
            const int k0 = kbeg[c], kc = kbeg[c + 1] - kbeg[c];
            const size_t off = (size_t)k0 * N;
            if (h->h_count[c] > spec[c]) {                       // the speculative copy fell short: one thread fetches the rest
                std::lock_guard<std::mutex> lk(fix);
                if (!fixed[c]) {
                    const size_t at = off * h->var_per_step + spec[c];
                    cudaError_t q = cudaMemcpyAsync(h->h_var + at, d_var + at, (h->h_count[c] - spec[c]) * sizeof(float), cudaMemcpyDeviceToHost,
                                                    h->aux_stream);
                    if (q == cudaSuccess) q = cudaStreamSynchronize(h->aux_stream);
                    if (q != cudaSuccess) { bad.store((int)q); return; }
                    extra_d2h.fetch_add((long long)(h->h_count[c] - spec[c]) * (long long)sizeof(float));
                    fixed[c] = true;
                }
            }
            expand_delta_rows(host_obs + off * row_full, host_reward ? host_reward + off : nullptr, host_done ? host_done + off : nullptr,
                              h->h_rec + off * 4, h->h_off + (size_t)k0 * nblk, h->h_var + off * h->var_per_step, h->h_cur, kc, N, b0, b1,
                              h->cfg.step_penalty, cut, 2);
        }
    };
    using clk = std::chrono::steady_clock;
    const auto t_begin = clk::now();
    if (expand) h->pool->start(jobs, worker);
    const int rc_issue = [&]() -> int {
        const float4 *prev_frames = h->d_frame0;                        // the frames the next chunk's first step is compared with
        for (int c = 0; c < n_chunks; ++c) {
            const int k0 = kbeg[c], kc = kbeg[c + 1] - kbeg[c];
            if (kc <= 0) continue;
            const size_t off = (size_t)k0 * N;
            const int hist_c = frames_only ? 1 : h->cfg.history;
            float *d_chunk = h->d_obs + off * row_full;
            if (c == 0) {
                // the first chunk's actions go up ahead of its kernel; the rest follows on another stream while it runs
                CU(cudaMemcpyAsync(h->d_act, host_actions, (size_t)kc * N * sizeof(int32_t), cudaMemcpyHostToDevice, s));
                if (n_chunks > 1) {
                    CU(cudaEventRecord(h->act_up, s));                   // (orders the copy behind whatever the caller's stream did before)
                    CU(cudaStreamWaitEvent(h->aux_stream, h->act_up, 0));
                    CU(cudaMemcpyAsync(h->d_act + (size_t)kc * N, host_actions + (size_t)kc * N, (n - (size_t)kc * N) * sizeof(int32_t),
                                       cudaMemcpyHostToDevice, h->aux_stream));
                    CU(cudaEventRecord(h->act_up, h->aux_stream));
                }
            } else if (c == 1) CU(cudaStreamWaitEvent(s, h->act_up, 0));
            h->p.log_k0 = k0;                                       // episode-log records carry the step index within the call
            const int rc2 = step_impl(h, h->d_act + off, SHIPSIM_ACTION_I32, kc, d_chunk, h->d_rew + off, h->d_done + off, stream, hist_c);
            h->p.log_k0 = 0;
            if (rc2) return rc2;
            if (frames_only && h->p.log_count && h->cfg.history == 2) {     // the one-frame kernel logged the terminal frame only
                CU(launch_log_prev_frames(h->p, (const float4 *)d_chunk, prev_frames, k0, kc, s));
                h->launches++;
            }
            if (trace) CU(cudaEventRecord(h->trace_mid[c], s));
            if (frames_only) {
                if (nd < (int)N) {
                    CU(launch_compact_frames((const float4 *)d_chunk, prev_frames, h->d_rew + off, h->d_done + off, (int)N, nd, kc, h->cfg.step_penalty,
                                             h->d_rec + off, h->d_off + (size_t)k0 * nblk, d_var + off * h->var_per_step,
                                             (unsigned)std::min<size_t>((size_t)kc * N * h->var_per_step, 0xffffffffu), h->d_count + c, s));
                    h->launches++;
                }
                if (nd > 0) {
                    CU(launch_history_rows((const float4 *)d_chunk, prev_frames, h->d_done + off, (int)N, nd, kc, h->cfg.auto_reset != 0,
                                           (float4 *)(h->d_rows + (size_t)k0 * nd * row_full), s));
                    h->launches++;
                }
                prev_frames = (const float4 *)d_chunk + ((size_t)(kc - 1) * N) * 4;
            }
            cudaStream_t cs = h->copy_stream;
            if (small) cs = s;                                      // one stream, no event hops
            else {
                CU(cudaEventRecord(h->chunk_done[c], s));
                CU(cudaStreamWaitEvent(h->copy_stream, h->chunk_done[c], 0));
            }
            if (frames_only) {
                if (nd < (int)N) {
                    if (c == 0) {
                        CU(cudaMemcpyAsync(h->h_cur, h->d_frame0, N * kFrame * sizeof(float), cudaMemcpyDeviceToHost, h->copy_stream));
                        h->last_d2h += (int64_t)(N * kFrame * sizeof(float));
                    }
                    if (nd == 0) CU(cudaMemcpyAsync(h->h_rec + off * 4, h->d_rec + off, (size_t)kc * N * sizeof(uint4), cudaMemcpyDeviceToHost, h->copy_stream));
                    else CU(cudaMemcpy2DAsync(h->h_rec + (off + nd) * 4, N * sizeof(uint4), h->d_rec + off + nd, N * sizeof(uint4), (N - nd) * sizeof(uint4),
                                              kc, cudaMemcpyDeviceToHost, h->copy_stream));
                    CU(cudaMemcpyAsync(h->h_off + (size_t)k0 * nblk, h->d_off + (size_t)k0 * nblk, (size_t)kc * nblk * sizeof(unsigned),
                                       cudaMemcpyDeviceToHost, h->copy_stream));
                    CU(cudaMemcpyAsync(h->h_count + c, h->d_count + c, sizeof(unsigned), cudaMemcpyDeviceToHost, h->copy_stream));
                    // the values: how many there are is only known on the device, so a size that has been enough so far goes
                    // down unasked (a host thread fetches the rest in the rare case that it was not)
                    spec[c] = std::min((size_t)kc * N * h->var_per_step, (size_t)((double)kc * (N - nd) * h->var_density) + 1024);
                    CU(cudaMemcpyAsync(h->h_var + off * h->var_per_step, d_var + off * h->var_per_step, spec[c] * sizeof(float),
                                       cudaMemcpyDeviceToHost, h->copy_stream));
                    h->last_d2h += (int64_t)kc * (N - nd) * sizeof(uint4) + (int64_t)kc * nblk * sizeof(unsigned) + sizeof(unsigned)
                                   + (int64_t)spec[c] * sizeof(float);
                }
                CU(cudaEventRecord(h->copy_done[c], h->copy_stream));       // what the host threads wait for
                issued.store(c + 1, std::memory_order_release);
                if (nd > 0) {
                    const size_t w = (size_t)nd * row_full * sizeof(float);
                    CU(cudaMemcpy2DAsync(host_obs + off * row_full, N * row_full * sizeof(float), h->d_rows + (size_t)k0 * nd * row_full, w, w, kc,
                                         cudaMemcpyDeviceToHost, h->copy_stream));
                    if (host_reward) CU(cudaMemcpy2DAsync(host_reward + off, N * sizeof(float), h->d_rew + off, N * sizeof(float), nd * sizeof(float), kc,
                                                          cudaMemcpyDeviceToHost, h->copy_stream));
                    if (host_done) CU(cudaMemcpy2DAsync(host_done + off, N, h->d_done + off, N, nd, kc, cudaMemcpyDeviceToHost, h->copy_stream));
                    h->last_d2h += (int64_t)kc * nd * (row_full * sizeof(float) + (host_reward ? 4 : 0) + (host_done ? 1 : 0));
                }
                continue;
            } else {
                h->last_d2h += (int64_t)kc * N * ((host_reward ? 4 : 0) + (host_done ? 1 : 0));
                if (host_obs) {
                    h->last_d2h += (int64_t)kc * N * row_full * sizeof(float);
                    CU(cudaMemcpyAsync(host_obs + off * row_full, d_chunk, (size_t)kc * N * row_full * sizeof(float), cudaMemcpyDeviceToHost, cs));
                }
                if (host_reward) CU(cudaMemcpyAsync(host_reward + off, h->d_rew + off, (size_t)kc * N * sizeof(float), cudaMemcpyDeviceToHost, cs));
                if (host_done) CU(cudaMemcpyAsync(host_done + off, h->d_done + off, (size_t)kc * N, cudaMemcpyDeviceToHost, cs));
            }
            if (!small) CU(cudaEventRecord(h->copy_done[c], h->copy_stream));
        }
        return SHIPSIM_OK;
    }();
    if (expand) {
        if (rc_issue) bad.store(-1);
        h->pool->finish();
    }
    if (rc_issue) return rc_issue;
    if (expand) {
        if (bad.load()) return fail(SHIPSIM_ERR_CUDA, std::string("copy stream: ") + cudaGetErrorString((cudaError_t)bad.load()));
        h->last_d2h += extra_d2h.load();
        double dens = 0.0;
        for (int c = 0; c < n_chunks; ++c) dens = std::max(dens, (double)h->h_count[c] / ((double)(kbeg[c + 1] - kbeg[c]) * (double)(N - nd)));
        h->var_density = std::max(0.9 * h->var_density, std::min(12.0, 1.25 * dens + 0.25));       // follows the need up at once, down slowly
    }
    if (!small) CU(cudaStreamSynchronize(h->copy_stream));
    CU(cudaStreamSynchronize(s));
    if (trace && !small) {
        std::fprintf(stderr, "step_host trace (ms since the call's first stream op): host done %.2f\n",
                     std::chrono::duration<double, std::milli>(clk::now() - t_begin).count());
        for (int c = 0; c < n_chunks; ++c) {
            float a = 0.f, b = 0.f;
            cudaEventElapsedTime(&a, h->trace0, h->chunk_done[c]);
            cudaEventElapsedTime(&b, h->trace0, h->copy_done[c]);
            float m = 0.f;
            cudaEventElapsedTime(&m, h->trace0, h->trace_mid[c]);
            std::fprintf(stderr, "  chunk %2d: step kernel done %.2f  compaction done %.2f  records home %.2f\n", c, m, a, b);
        }
    }
    if (adaptive) {
        // The split for the next call climbs towards the shorter call: keep going while the time per env-step improves, turn
        // round (with half the step) when it gets worse, stay when it no longer changes.
        const double t = std::chrono::duration<double>(clk::now() - t_begin).count() / (double)n;
        if (h->dma_last_t > 0.0 && t > h->dma_last_t * 1.015) {
            h->dma_dir = -h->dma_dir;
            h->dma_step = std::max(32, h->dma_step / 2 / 32 * 32);
        }
        if (h->dma_last_t == 0.0 || t < h->dma_last_t * 0.985 || t > h->dma_last_t * 1.015)
            h->dma_envs = std::max(0, std::min((int)N, nd + h->dma_dir * h->dma_step));
        h->dma_last_t = t;
    }
    return SHIPSIM_OK;
}

extern "C" int shipsim_mlp_policy_forward(const float *dev_obs, int32_t num_envs, const float *dev_w1, const float *dev_b1, const float *dev_w2,
                                          const float *dev_b2, const float *dev_w3, const float *dev_b3, const float *dev_noise, float *dev_out,
                                          int64_t *dev_actions, void *stream)
{
    if (!dev_obs || !dev_w1 || !dev_b1 || !dev_w2 || !dev_b2 || !dev_w3 || !dev_b3 || !dev_noise || !dev_out || !dev_actions || num_envs < 1)
        return fail(SHIPSIM_ERR_ARG, "NULL buffer or num_envs < 1");
    if (((uintptr_t)dev_obs & 15) != 0) return fail(SHIPSIM_ERR_ARG, "dev_obs must be 16-byte aligned");
    CU(launch_mlp_policy(dev_obs, num_envs, dev_w1, dev_b1, dev_w2, dev_b2, dev_w3, dev_b3, dev_noise, dev_out, (long long *)dev_actions,
                         (cudaStream_t)stream));
    return SHIPSIM_OK;
}

extern "C" int shipsim_gae(const float *dev_rewards, const float *dev_values, const uint8_t *dev_dones, int32_t n_steps, int32_t num_envs, float gamma,
                           float lam, float *dev_adv, float *dev_returns, void *stream)
{
    if (!dev_rewards || !dev_values || !dev_dones || !dev_adv || !dev_returns || n_steps < 1 || num_envs < 1)
        return fail(SHIPSIM_ERR_ARG, "NULL buffer or bad sizes");
    CU(launch_gae(dev_rewards, dev_values, dev_dones, n_steps, num_envs, gamma, lam, dev_adv, dev_returns, (cudaStream_t)stream));
    return SHIPSIM_OK;
}

extern "C" int shipsim_host_traffic(const shipsim_t *h, int64_t *h2d_bytes, int64_t *d2h_bytes)
{
    if (!h) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    if (h2d_bytes) *h2d_bytes = h->last_h2d;
    if (d2h_bytes) *d2h_bytes = h->last_d2h;
    return SHIPSIM_OK;
}

extern "C" int shipsim_host_threads(const shipsim_t *h, int32_t *n_threads)
{
    if (!h || !n_threads) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    *n_threads = h->pool ? h->pool->size() : 0;
    return SHIPSIM_OK;
}

extern "C" int shipsim_expand_delta(float *host_obs, float *host_reward, uint8_t *host_done, const uint32_t *host_rec, const uint32_t *host_off,
                                    const float *host_var, float *host_cur, int32_t n_steps, int64_t num_envs, float step_penalty,
                                    int32_t cut_on_done, int32_t history)
{
    if (!host_rec || !host_off || !host_var || !host_cur || n_steps < 0 || num_envs < 1 || (history != 1 && history != 2))
        return fail(SHIPSIM_ERR_ARG, "NULL buffer or bad sizes");
    expand_delta_rows(host_obs, host_reward, host_done, host_rec, host_off, host_var, host_cur, n_steps, (size_t)num_envs, 0,
                      ((size_t)num_envs + 31) / 32, step_penalty, cut_on_done != 0, history);
    return SHIPSIM_OK;
}

extern "C" int shipsim_assemble_history(float *host_obs, const float *host_frames, const uint8_t *host_cut, int64_t n_rows, int64_t num_envs)
{
    if (!host_obs || !host_frames || n_rows < 0 || num_envs < 1) return fail(SHIPSIM_ERR_ARG, "NULL buffer or bad sizes");
    assemble_history_rows(host_obs, host_frames, host_cut, 0, (size_t)n_rows, (size_t)num_envs);
    return SHIPSIM_OK;
}

extern "C" int shipsim_stats_read(shipsim_t *h, double *dev_out, int clear, void *stream)
{
    const int rc = ready(h);
    if (rc) return rc;
    if (!dev_out) return fail(SHIPSIM_ERR_ARG, "dev_out is NULL");
    DeviceGuard g(h->device);
    CU(launch_stats_reduce(h->p.stats, dev_out, clear, (cudaStream_t)stream));
    h->launches++;
    return SHIPSIM_OK;
}

extern "C" int shipsim_set_state(shipsim_t *h, const float *pose, const int32_t *ints, const float *lidar, const float *goals,
                                 const float *ep_return)
{
    const int rc = ready(h);
    if (rc) return rc;
    if (!pose || !ints || !lidar || !goals || !ep_return) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    const size_t N = (size_t)h->cfg.num_envs;
    const int nb = h->cfg.lidar_beams, planes = state_planes(h);
    std::vector<float4> st(N * planes);
    for (size_t e = 0; e < N; ++e) {
        // lidar[e][lidar_beams]; readings past the fan (planes 2-4 of a fan of fewer than 10 beams) hold -1
        float l[kBeams + 4 * ((kMaxBeams - kBeams) / 4 + 1)];
        for (int j = 0; j < (int)(sizeof(l) / sizeof(l[0])); ++j) l[j] = j < nb ? lidar[e * nb + j] : -1.f;
        const float *q = pose + e * 6, *gl = goals + e * 10;
        const int32_t *in = ints + e * 5;
        if (in[0] % 5 != 0 || in[0] < -10 || in[0] > 10) return fail(SHIPSIM_ERR_ARG, "rudder must be in {-10,-5,0,5,10}");
        if (in[3] < 0 || in[3] >= h->p.n_scen) return fail(SHIPSIM_ERR_ARG, "scenario id out of range");
        const int bits = ((in[0] / 5 + 2) & 7) | ((in[1] & 31) << 3) | (in[2] << 8);
        float fb, fs, fe;
        std::memcpy(&fb, &bits, 4); std::memcpy(&fs, &in[3], 4); std::memcpy(&fe, &in[4], 4);
        st[0 * N + e] = make_float4(q[0], q[1], q[2], q[3]);
        st[1 * N + e] = make_float4(q[4], q[5], ep_return[e], fb);
        st[2 * N + e] = make_float4(l[0], l[1], l[2], l[3]);
        st[3 * N + e] = make_float4(l[4], l[5], l[6], l[7]);
        st[4 * N + e] = make_float4(l[8], l[9], fs, fe);
        st[5 * N + e] = make_float4(gl[0], gl[1], gl[2], gl[3]);
        st[6 * N + e] = make_float4(gl[4], gl[5], gl[6], gl[7]);
        st[7 * N + e] = make_float4(gl[8], gl[9], 0.f, 0.f);
        for (int pl = kPlanes; pl < planes; ++pl) {
            const float *x = l + kBeams + 4 * (pl - kPlanes);
            st[pl * N + e] = make_float4(x[0], x[1], x[2], x[3]);
        }
    }
    DeviceGuard g(h->device);
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(h->p.state, st.data(), st.size() * sizeof(float4), cudaMemcpyHostToDevice));
    return SHIPSIM_OK;
}

extern "C" int shipsim_get_state(shipsim_t *h, float *pose, int32_t *ints, float *lidar, float *goals, float *ep_return)
{
    const int rc = ready(h);
    if (rc) return rc;
    const size_t N = (size_t)h->cfg.num_envs;
    const int nb = h->cfg.lidar_beams, planes = state_planes(h);
    std::vector<float4> st(N * planes);
    DeviceGuard g(h->device);
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(st.data(), h->p.state, st.size() * sizeof(float4), cudaMemcpyDeviceToHost));
    for (size_t e = 0; e < N; ++e) {
        const float4 a = st[0 * N + e], b = st[1 * N + e], l0 = st[2 * N + e], l1 = st[3 * N + e], l2 = st[4 * N + e];
        const float4 g0 = st[5 * N + e], g1 = st[6 * N + e], g2 = st[7 * N + e];
        int bits, scen, ep;
        std::memcpy(&bits, &b.w, 4); std::memcpy(&scen, &l2.z, 4); std::memcpy(&ep, &l2.w, 4);
        if (pose) { float *q = pose + e * 6; q[0] = a.x; q[1] = a.y; q[2] = a.z; q[3] = a.w; q[4] = b.x; q[5] = b.y; }
        if (ep_return) ep_return[e] = b.z;
        if (ints) { int32_t *in = ints + e * 5; in[0] = ((bits & 7) - 2) * 5; in[1] = (bits >> 3) & 31; in[2] = bits >> 8; in[3] = scen; in[4] = ep; }
        if (lidar) {
            float l[kBeams + 4 * ((kMaxBeams - kBeams) / 4 + 1)] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w, l2.x, l2.y};
            for (int pl = kPlanes; pl < planes; ++pl) {
                const float4 x = st[pl * N + e];
                float *d = l + kBeams + 4 * (pl - kPlanes);
                d[0] = x.x; d[1] = x.y; d[2] = x.z; d[3] = x.w;
            }
            std::memcpy(lidar + e * nb, l, nb * sizeof(float));
        }
        if (goals) { float *gl = goals + e * 10; gl[0] = g0.x; gl[1] = g0.y; gl[2] = g0.z; gl[3] = g0.w; gl[4] = g1.x; gl[5] = g1.y; gl[6] = g1.z; gl[7] = g1.w; gl[8] = g2.x; gl[9] = g2.y; }
    }
    return SHIPSIM_OK;
}

extern "C" int shipsim_render(shipsim_t *h, int32_t env_index, int32_t width, int32_t height, uint8_t *dev_rgb, void *stream)
{
    const int rc = ready(h);
    if (rc) return rc;
    if (env_index < 0 || env_index >= h->cfg.num_envs) return fail(SHIPSIM_ERR_ARG, "env_index out of range");
    if (width < 1 || height < 1 || !dev_rgb) return fail(SHIPSIM_ERR_ARG, "bad image size / NULL buffer");
    DeviceGuard g(h->device);
    CU(launch_render(h->p, env_index, width, height, dev_rgb, (cudaStream_t)stream));
    return SHIPSIM_OK;
}

extern "C" int shipsim_launch_count(const shipsim_t *h, int64_t *out)
{
    if (!h || !out) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    *out = h->launches;
    return SHIPSIM_OK;
}

extern "C" int shipsim_launch_shape(const shipsim_t *h, int32_t *lanes, int32_t *threads, int32_t *ctas)
{
    if (!h) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    if (lanes) *lanes = h->shape.lanes_per_env;
    if (threads) *threads = h->shape.threads;
    if (ctas) *ctas = h->shape.blocks;
    return SHIPSIM_OK;
}

extern "C" int shipsim_launch_window(const shipsim_t *h, int32_t *steps_in_flight)
{
    if (!h || !steps_in_flight) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    *steps_in_flight = h->shape.window;
    return SHIPSIM_OK;
}
