// shipsim_abi.cu -- the C ABI of libshipsim.so (include/shipsim.h): handle management, scenario packing,
// parameter derivation and kernel launches.  Host-side C++; no torch types anywhere.
#include "../../include/shipsim.h"
#include "shipsim_geom.cuh"
#include "shipsim_launch.h"
#include "shipsim_host.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

using namespace shipsim;

// Small persistent worker pool for the host half of shipsim_step_host (assembling observation histories from frames
// while later chunks are still crossing PCIe): fn(i) for i in [0, n) runs on the workers + the caller.
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

namespace {
// ---- owned CUDA resources ----------------------------------------------------------------------------------------
// Move-only owner of one CUDA handle, released with Release when the owner dies or takes another handle.  size_ is the
// element count of an allocation (Buffer).
template <class H, cudaError_t (*Release)(H)>
class Owned {
public:
    Owned() = default;
    Owned(Owned &&o) noexcept : h_(std::exchange(o.h_, H{})), size_(std::exchange(o.size_, 0)) {}
    Owned &operator=(Owned &&o) noexcept { if (this != &o) { reset(); std::swap(h_, o.h_); std::swap(size_, o.size_); } return *this; }
    ~Owned() { reset(); }
    void reset() { if (h_) Release(std::exchange(h_, H{})); size_ = 0; }
    H *out() { reset(); return &h_; }                 // where the call that creates the next handle writes it
    operator H() const { return h_; }

protected:
    H h_{};
    size_t size_ = 0;
};
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;
using Event = Owned<cudaEvent_t, cudaEventDestroy>;

// Buffer of T that grows on demand: ensure(count) frees the old allocation, then allocates the new one; if that fails,
// the capacity is 0 and the CUDA error is returned.
template <class T, cudaError_t (*Alloc)(void **, size_t), cudaError_t (*Release)(void *)>
struct Buffer : Owned<void *, Release> {
    cudaError_t ensure(size_t count)
    {
        if (count <= this->size_) return cudaSuccess;
        const cudaError_t e = Alloc(this->out(), count * sizeof(T));
        if (e == cudaSuccess) this->size_ = count;
        return e;
    }
    operator T *() const { return static_cast<T *>(this->h_); }
};
template <class T> using DeviceBuf = Buffer<T, cudaMalloc, cudaFree>;
template <class T> using PinnedBuf = Buffer<T, cudaMallocHost, cudaFreeHost>;

// One scenario bank on the device, in the layout the kernels read it with.
struct Bank {
    DeviceBuf<float4> rec;                   // [n_scen][stride4] packed scenario records
    DeviceBuf<EdgeD> edges;                  // [n_scen][2][kMaxHull] two-float planes
    DeviceBuf<uint4> grid;                   // [n_scen][kGridN * kGridN] reach grid
    DeviceBuf<float4> spawn;                 // [n_scen][kScr4] plane rows at the spawn pose
    DeviceBuf<unsigned> pick;                // [2][n_scen + 1] weighted-pick table (cdf, guide): shipsim_scenario_weights
    int n_scen = 0, maxv = 0, stride4 = 0, hull_max = 0;
    bool generated = false;                  // by shipsim_generate_scenarios: fresh maps may regenerate it in place

    cudaError_t alloc(int n, int edge_stride)
    {
        n_scen = n; maxv = edge_stride; stride4 = kBankHeader4 + 2 * edge_stride;
        cudaError_t e = rec.ensure((size_t)n * stride4);
        if (e == cudaSuccess) e = edges.ensure((size_t)n * 2 * kMaxHull);
        if (e == cudaSuccess) e = grid.ensure((size_t)n * kGridN * kGridN);
        if (e == cudaSuccess) e = spawn.ensure((size_t)n * kScr4);
        if (e == cudaSuccess) e = pick.ensure(2 * ((size_t)n + 1));
        return e;
    }
};

// Raw output of the device scenario generator: double hull vertices ([n][2][kMaxHull][2]), hull sizes and goals.
struct Generated {
    DeviceBuf<double> xy, goals;
    DeviceBuf<int> n;
    int count = 0;
};

constexpr int kMaxChunks = 64;               // shipsim_step_host cuts a call into at most this many chunks of steps

// The share of a frames-only shipsim_step_host call that goes home as complete rows by DMA: envs [0, envs).  The host
// threads expand the others.
struct DmaSplit {
    int envs = -1;                           // -1: not chosen yet
    int for_n = 0, for_k = 0;
    int step = 0, dir = 1;                   // the split climbs towards the shorter call: step size and direction
    double last_t = 0.0;                     // seconds per env-step of the previous call

    int choose(int N, int K, int threads)
    {
        if (envs < 0 || for_n != N || for_k != K) {
            // First guess.  With a core per ~4 GB/s of rows the host threads alone are the faster engine, and DMA
            // writes landing next to their streaming stores slow both (B200 box, 16 cores: 6.4 ms per 4,096 x 1,000
            // call with the host threads alone, 8-10 ms with any share by DMA; profiles/r02_e2e_sweep.log); with few
            // cores per GPU the copy engine has to carry most of it.
            envs = threads >= 8 ? 0 : (int)((double)N * 50.0 / (50.0 + 9.0 * threads));
            for_n = N; for_k = K; step = std::max(32, N / 8 / 32 * 32); dir = 1; last_t = 0.0;
        }
        return envs;
    }
    // Keep going while the time per env-step improves, turn round (with half the step) when it gets worse, stay when it
    // no longer changes.  `nd` is the split this call ran with, `t` its seconds per env-step.
    void update(int N, int nd, double t)
    {
        if (last_t > 0.0 && t > last_t * 1.015) {
            dir = -dir;
            step = std::max(32, step / 2 / 32 * 32);
        }
        if (last_t == 0.0 || t < last_t * 0.985 || t > last_t * 1.015) envs = std::max(0, std::min(N, nd + dir * step));
        last_t = t;
    }
};

}  // namespace

struct shipsim_handle {
    shipsim_config cfg;
    int device = 0;
    StepParams p;
    Bank bank;                               // the bank the kernels read
    Generated gen;                           // the last shipsim_generate_scenarios (for read-back)
    struct { double cw, ch, margin, reach; } grid_geom;   // of the reach grid's cells (derive_params, launch_build_grid)
    int lanes = 1;
    int window = 1;                          // steps of one env speculated together (1 = the serial-in-time kernel)
    // staging for shipsim_step_host (allocated on first use, sized for the largest K seen)
    DeviceBuf<int32_t> d_act; DeviceBuf<float> d_obs; DeviceBuf<float> d_rew; DeviceBuf<uint8_t> d_done;
    Stream copy_stream;                      // shipsim_step_host: results of chunk i go home while chunk i+1 is computed
    Event chunk_done[kMaxChunks], copy_done[kMaxChunks];
    int chunk_events = -1;                   // -1: not created yet; else whether they time (for a trace)
    Event trace0, trace_mid[kMaxChunks];     // created by the first call that asks for a trace
    DeviceBuf<float4> d_frame0;
    // compacted wire format of the host path (compact_frames_kernel / expand_delta_rows)
    DeviceBuf<uint4> d_rec;                  // [K][N] records
    DeviceBuf<unsigned> d_off, d_count;      // [K][N/32] value offsets; one counter per chunk
    PinnedBuf<uint32_t> h_rec, h_off, h_count;   // pinned mirrors
    PinnedBuf<float> h_var;                  // the changed values (a dense stream per chunk), host mirror ...
    DeviceBuf<float> d_var;                  // ... and device buffer
    double var_density = 2.0;                // floats per env-step the speculative D2H copy of a chunk's values is sized for
    Stream aux_stream;                       // actions of chunks 1.. go up here; the (rare) rest of a chunk's values comes down
    Event act_up;
    PinnedBuf<float> h_cur;                  // one frame per env: the decoder's running state
    DeviceBuf<float> d_rows;                 // [K][dma envs][32]: the complete rows that go home by DMA
    DmaSplit dma;
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
        Stream stream;
        Event period_begin, gen_done;
    } fresh;
    const void *zc_host[4] = {nullptr, nullptr, nullptr, nullptr};     // the last tiny call's buffers and their device aliases
    void *zc_dev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::unique_ptr<HostPool> pool;
    int64_t last_h2d = 0, last_d2h = 0;      // bytes the last shipsim_step_host moved over PCIe
    int64_t launches = 0;
    int32_t calls = 0;                       // shipsim_step / shipsim_step_host calls so far (SHIPSIM_EP_CALL)
    // chained launches (shipsim_step_chained)
    DeviceBuf<unsigned> chain_tickets;       // [2][N]: started, done (bound and zeroed with the state)
    bool chain_open = false;                 // the handle's last enqueue was a window launch on chain_stream ...
    cudaStream_t chain_stream = nullptr;
    uint64_t chain_seq = 0;                  // ... and g_enqueues has not moved since
    int64_t chained = 0;                     // chained launches so far
    LaunchShape shape{1, kThreads, 0, 1};
    __attribute__((visibility("hidden"))) ~shipsim_handle() = default;     // (not one of the library's exported symbols)
};

static thread_local std::string g_err;

// Every ABI call that enqueues work (or changes what a launch reads) moves this counter, so that a chained launch also
// sees work that another handle put on the stream in between -- e.g. two handles alternating on one stream and writing
// one output buffer: overlapping those launches would race.
static std::atomic<uint64_t> g_enqueues{0};

// The next step call of the handle starts a new chain.
static void unchain(shipsim_t *h)
{
    if (h) h->chain_open = false;
    g_enqueues.fetch_add(1, std::memory_order_relaxed);
}

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
// the same for a shipsim status: a failure is passed on
#define TRY(expr)                                                                                     \
    do {                                                                                              \
        const int _rc = (expr);                                                                       \
        if (_rc != SHIPSIM_OK) return _rc;                                                            \
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
    // The grid is built in double: cell size, touch margin and the reach of a cell's masks.  The cell is looked up at the
    // LIDAR ORIGIN, and its masks also decide "bank not near => no ship-vs-bank test": the reach must cover the hull as
    // seen from that origin (every hull point lies within 2 * max |hull vertex|, taken in fp32).
    auto &gg = h->grid_geom;
    gg.cw = ((double)c.bounds_w + 2.0 * pad) / kGridN;
    gg.ch = ((double)c.bounds_h + 2.0 * pad) / kGridN;
    gg.margin = 0.05 + 1e-4 * std::max((double)c.bounds_w, (double)c.bounds_h);
    gg.reach = std::max({(double)c.lidar_distance, (double)(float)(2.0 * rmax), std::sqrt(gg.cw * gg.cw + gg.ch * gg.ch)}) + gg.margin;
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
    delete h;                                // (the owners release the handle's resources on its device)
    return SHIPSIM_OK;
}

// The reach grid (one thread per cell, in double) and the plane rows at the spawn pose (what an env that is reset inside
// the kernel starts from) of the scenarios [s0, s0 + n) of bank b, from their double hull vertices: hull_stride per hull,
// hull_xy and hull_n start at scenario s0.
static cudaError_t build_reach_tables(const shipsim_t *h, const Bank &b, size_t s0, int n, const double *hull_xy, const int *hull_n,
                                      int hull_stride, cudaStream_t s)
{
    const auto &gg = h->grid_geom;
    uint4 *grid = b.grid + s0 * kGridN * kGridN;
    const cudaError_t e = launch_build_grid(hull_xy, hull_n, n, hull_stride, (double)h->p.gridp.x0, (double)h->p.gridp.y0, gg.cw, gg.ch,
                                            gg.reach, gg.margin, grid, s);
    if (e != cudaSuccess) return e;
    StepParams q = h->p;
    q.bank = b.rec + s0 * b.stride4; q.edges_d = b.edges + s0 * 2 * kMaxHull; q.grid = grid; q.n_scen = n;
    q.maxv = b.maxv; q.scen_stride4 = b.stride4; q.hull_max = b.hull_max;
    return launch_build_spawn_rows(q, b.spawn + s0 * kScr4, s);
}

// Make `b` the bank the kernels read; the device is idle, so no launch still reads the old one.  A new bank leaves
// fresh-maps mode, and live envs may hold scenario ids of an old, larger bank: those are folded into range.
static int install(shipsim_t *h, Bank &&b, cudaStream_t s)
{
    const int old_n = h->p.n_scen;
    h->bank = std::move(b);
    const Bank &nb = h->bank;
    StepParams &p = h->p;
    p.bank = nb.rec; p.edges_d = nb.edges; p.grid = nb.grid; p.spawn_rows = nb.spawn;
    p.n_scen = nb.n_scen; p.maxv = nb.maxv; p.scen_stride4 = nb.stride4; p.hull_max = nb.hull_max;
    h->fresh.on = false; h->fresh.pending = false; p.pick_base = 0; p.pick_count = 0;
    p.pick_cdf = nullptr; p.pick_guide = nullptr;              // weights belong to the old bank
    if (p.state && nb.n_scen < old_n) {
        CU(launch_clamp_scenarios(p.state, h->cfg.num_envs, nb.n_scen, s));
        CU(cudaStreamSynchronize(s));
        h->launches++;
    }
    return SHIPSIM_OK;
}

extern "C" int shipsim_load_scenarios(shipsim_t *h, const double *hull_xy, const int32_t *hull_n, const double *goals_xy,
                                      int32_t n_scen, int32_t maxv)
{
    unchain(h);
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
    Bank b;
    DeviceBuf<double> dxy;
    DeviceBuf<int> dn;
    CU(b.alloc(n_scen, dev_maxv));
    CU(dxy.ensure(rxy.size()));
    CU(dn.ensure((size_t)n_scen * 2));
    CU(cudaMemcpy(b.rec, host.data(), host.size() * sizeof(float4), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(b.edges, edges.data(), edges.size() * sizeof(EdgeD), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dxy, rxy.data(), rxy.size() * sizeof(double), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dn, hull_n, (size_t)n_scen * 2 * sizeof(int), cudaMemcpyHostToDevice));
    b.hull_max = dev_maxv;
    CU(build_reach_tables(h, b, 0, n_scen, dxy, dn, dev_maxv, 0));
    CU(cudaDeviceSynchronize());                                 // also: no launch may still be reading the old bank
    h->launches += 2;
    return install(h, std::move(b), 0);
}

// ---- scenario generation on the device (SURVEY.md §8 f2) ------------------------------------------------------
extern "C" int shipsim_generate_scenarios(shipsim_t *h, int32_t n_scen, uint64_t seed, int32_t map_N, float width_frac, void *stream)
{
    unchain(h);
    if (!h) return fail(SHIPSIM_ERR_ARG, "handle is NULL");
    if (n_scen < 1 || n_scen >= (1 << 28)) return fail(SHIPSIM_ERR_ARG, "n_scenarios out of range");
    if (map_N < 1 || map_N > kMaxHull - 2) return fail(SHIPSIM_ERR_ARG, "map_N must be in [1, 30] (two wall corners are added; hulls hold 32 vertices)");
    if (!(width_frac > 0.f) || !(width_frac <= 1.f)) return fail(SHIPSIM_ERR_ARG, "width_frac must be in (0, 1]");
    DeviceGuard g(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    Bank b;
    Generated gen;
    DeviceBuf<int> dmax;
    CU(b.alloc(n_scen, kMaxHull));
    CU(gen.xy.ensure((size_t)n_scen * 2 * kMaxHull * 2));
    CU(gen.goals.ensure((size_t)n_scen * 10));
    CU(gen.n.ensure((size_t)n_scen * 2));
    CU(dmax.ensure(1));
    CU(cudaMemsetAsync(b.rec, 0, (size_t)n_scen * b.stride4 * sizeof(float4), s));
    CU(cudaMemsetAsync(b.edges, 0, (size_t)n_scen * 2 * kMaxHull * sizeof(EdgeD), s));
    CU(launch_gen_scenarios(seed, n_scen, h->cfg.bounds_w, h->cfg.bounds_h, map_N, width_frac, gen.xy, gen.n, gen.goals, s));
    CU(launch_max_hull(gen.n, n_scen * 2, dmax, s));
    CU(launch_pack_bank(gen.xy, gen.n, gen.goals, n_scen, b.maxv, b.stride4, b.rec, b.edges, s));
    CU(cudaMemcpyAsync(&b.hull_max, dmax, sizeof(int), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));                                // 4-byte read-back: the SAT pass lane layout depends on it
    CU(build_reach_tables(h, b, 0, n_scen, gen.xy, gen.n, kMaxHull, s));
    CU(cudaDeviceSynchronize());                                 // no launch may still be reading the old bank
    h->launches += 5;
    b.generated = true;
    gen.count = n_scen;
    h->gen = std::move(gen);
    h->fresh.map_N = map_N; h->fresh.width_frac = width_frac; h->fresh.seed = seed;
    return install(h, std::move(b), s);
}

extern "C" int shipsim_read_scenarios(shipsim_t *h, double *host_hull_xy, int32_t *host_hull_n, double *host_goals)
{
    unchain(h);
    if (!h || !host_hull_xy || !host_hull_n || !host_goals) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    if (!h->gen.count) return fail(SHIPSIM_ERR_STATE, "no device-generated bank: call shipsim_generate_scenarios first");
    DeviceGuard g(h->device);
    const size_t S = (size_t)h->gen.count;
    CU(cudaMemcpy(host_hull_xy, h->gen.xy, S * 2 * kMaxHull * 2 * sizeof(double), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(host_hull_n, h->gen.n, S * 2 * sizeof(int), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(host_goals, h->gen.goals, S * 10 * sizeof(double), cudaMemcpyDeviceToHost));
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
    const Bank &b = h->bank;
    const int q = b.n_scen / 4;
    const size_t s0 = (size_t)slice * q;
    cudaStream_t gs = h->fresh.stream;
    double *dxy = h->gen.xy + s0 * 2 * kMaxHull * 2, *dgo = h->gen.goals + s0 * 10;
    int *dn = h->gen.n + s0 * 2;
    float4 *d = b.rec + s0 * b.stride4;
    EdgeD *de = b.edges + s0 * 2 * kMaxHull;
    CU(cudaMemsetAsync(d, 0, (size_t)q * b.stride4 * sizeof(float4), gs));
    CU(cudaMemsetAsync(de, 0, (size_t)q * 2 * kMaxHull * sizeof(EdgeD), gs));
    CU(launch_gen_scenarios(seed, q, h->cfg.bounds_w, h->cfg.bounds_h, h->fresh.map_N, h->fresh.width_frac, dxy, dn, dgo, gs));
    CU(launch_pack_bank(dxy, dn, dgo, q, b.maxv, b.stride4, d, de, gs));
    CU(build_reach_tables(h, b, s0, q, dxy, dn, kMaxHull, gs));
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
        const int q = h->bank.n_scen / 4, slice = f.period % 4;
        if (f.pending) {                                 // this period's slice was regenerated while the last one ran
            CU(cudaStreamWaitEvent(s, f.gen_done, 0));
            f.pending = false;
        }
        h->p.pick_base = slice * q;
        if (f.period + 1 >= 4) {                         // the slice after this one has been played: new maps for it
            const int nxt = (f.period + 1) % 4;
            CU(cudaEventRecord(f.period_begin, s));      // every launch that could still read it precedes this point
            CU(cudaStreamWaitEvent(f.stream, f.period_begin, 0));
            TRY(fresh_regenerate(h, nxt, fresh_seed(f.seed, f.period + 1)));
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
    unchain(h);
    if (!h) return fail(SHIPSIM_ERR_ARG, "handle is NULL");
    DeviceGuard g(h->device);
    auto &f = h->fresh;
    if (!enable) {
        if (f.on) CU(cudaStreamSynchronize(f.stream));
        f.on = false; f.pending = false;
        h->p.pick_base = 0; h->p.pick_count = 0;
        return SHIPSIM_OK;
    }
    Bank &b = h->bank;
    if (h->p.pick_cdf) return fail(SHIPSIM_ERR_STATE, "fresh maps replay no map: turn scenario weights off first (shipsim_scenario_weights NULL)");
    if (!b.generated) return fail(SHIPSIM_ERR_STATE, "fresh maps need a device-generated bank: call shipsim_generate_scenarios first");
    const int q = b.n_scen / 4;
    if (b.n_scen % 4 != 0 || q < 1 || (q & (q - 1)) != 0)
        return fail(SHIPSIM_ERR_ARG, "fresh maps need a bank of 4 * 2^k scenarios");
    if (!h->cfg.auto_reset) return fail(SHIPSIM_ERR_STATE, "fresh maps need auto_reset (an env that is never reset would outlive its map)");
    if (!f.stream || !f.period_begin || !f.gen_done) {
        CU(cudaStreamCreateWithFlags(f.stream.out(), cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(f.period_begin.out(), cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(f.gen_done.out(), cudaEventDisableTiming));
    }
    f.on = true; f.pending = false; f.period = 0; f.steps = 0; f.max_steps = h->cfg.max_steps;
    for (int &gen : f.generation) gen = 0;
    h->p.pick_base = 0; h->p.pick_count = q;
    b.hull_max = std::max(b.hull_max, std::min(kMaxHull, f.map_N + 2));       // regenerated hulls: at most map_N + 2 vertices
    h->p.hull_max = b.hull_max;
    return SHIPSIM_OK;
}

extern "C" int shipsim_fresh_info(const shipsim_t *h, int32_t *info)
{
    if (!h || !info) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    info[0] = h->fresh.on ? 1 : 0; info[1] = h->fresh.period; info[2] = h->p.pick_base; info[3] = h->p.pick_count;
    for (int i = 0; i < 4; ++i) info[4 + i] = h->fresh.generation[i];
    return SHIPSIM_OK;
}

extern "C" int shipsim_scenario_weights(shipsim_t *h, const uint32_t *dev_weights, void *stream)
{
    unchain(h);
    if (!h) return fail(SHIPSIM_ERR_ARG, "handle is NULL");
    if (!h->p.bank) return fail(SHIPSIM_ERR_STATE, "shipsim_load_scenarios has not been called");
    if (!dev_weights) {
        h->p.pick_cdf = nullptr; h->p.pick_guide = nullptr;
        return SHIPSIM_OK;
    }
    if (h->fresh.on) return fail(SHIPSIM_ERR_STATE, "scenario weights replay maps: fresh maps are on (shipsim_fresh_maps 0 first)");
    DeviceGuard g(h->device);
    Bank &b = h->bank;
    CU(launch_build_pick_table(dev_weights, b.n_scen, b.pick, (cudaStream_t)stream));
    h->launches++;
    h->p.pick_cdf = b.pick; h->p.pick_guide = b.pick + b.n_scen + 1;
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
    unchain(h);
    if (!h || !dev_state || !dev_stats) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    if (((uintptr_t)dev_state & 15) || ((uintptr_t)dev_stats & 7)) return fail(SHIPSIM_ERR_ARG, "state must be 16-byte aligned");
    DeviceGuard g(h->device);
    const size_t N = (size_t)h->cfg.num_envs;
    CU(h->chain_tickets.ensure(2 * N));
    CU(cudaMemsetAsync(h->chain_tickets, 0, 2 * N * sizeof(unsigned), (cudaStream_t)stream));
    h->p.chain_started = h->chain_tickets;
    h->p.chain_done = h->chain_tickets + N;
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
    unchain(h);
    TRY(ready(h));
    DeviceGuard g(h->device);
    CU(launch_reset(h->p, dev_mask, dev_scenario, first, (float4 *)dev_obs, (cudaStream_t)stream));
    h->launches++;
    return SHIPSIM_OK;
}

// What the runtime knows of a pointer: its memory type and, for page-locked host memory that is mapped, its device alias.
// Memory the runtime does not know reads as unregistered; the error of that query is cleared, so no later call sees it.
struct PtrInfo {
    cudaMemoryType type;
    void *alias;
};
static PtrInfo pointer_info(const void *ptr)
{
    cudaPointerAttributes attr{};
    const bool ok = cudaPointerGetAttributes(&attr, ptr) == cudaSuccess;
    cudaGetLastError();
    if (!ok) return {cudaMemoryTypeUnregistered, nullptr};
    return {attr.type, attr.type == cudaMemoryTypeHost ? attr.devicePointer : nullptr};
}

extern "C" int shipsim_episode_log_bind(shipsim_t *h, float *dev_rows, int32_t *dev_meta, int32_t capacity, int32_t *dev_count)
{
    unchain(h);
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
    if (pointer_info(dev_count).type != cudaMemoryTypeDevice)
        return fail(SHIPSIM_ERR_ARG, "dev_count must be device memory (it is the target of device atomics)");
    // rows and metadata may sit in page-locked host memory (written over PCIe): the kernels need its device alias
    const PtrInfo rows = pointer_info(dev_rows), meta = pointer_info(dev_meta);
    p.log_rows = (float4 *)(rows.alias ? rows.alias : dev_rows);
    p.log_meta = (int4 *)(meta.alias ? meta.alias : dev_meta);
    p.log_count = (int *)dev_count;
    p.log_cap = capacity;
    p.log_row4 = 4 * h->cfg.history;         // (the wide kernel's rows are dense: (6 + lidar_beams) * history floats)
    return SHIPSIM_OK;
}

static int step_impl(shipsim_t *h, const void *dev_actions, int action_dtype, int32_t K, float *dev_obs, float *dev_reward,
                     uint8_t *dev_done, void *stream, int history, bool chain = false)
{
    TRY(ready(h));
    if (K < 1) return fail(SHIPSIM_ERR_ARG, "K must be >= 1");
    if (action_dtype < 0 || action_dtype > 3) return fail(SHIPSIM_ERR_ARG, "bad action_dtype");
    if (action_dtype != SHIPSIM_ACTION_RANDOM && !dev_actions) return fail(SHIPSIM_ERR_ARG, "dev_actions is NULL");
    // (the tuned 10-beam kernel stores rows as float4; the wide kernel's rows are dense floats)
    if ((uintptr_t)dev_obs & (h->cfg.lidar_beams == SHIPSIM_N_BEAMS ? 15 : 3))
        return fail(SHIPSIM_ERR_ARG, h->cfg.lidar_beams == SHIPSIM_N_BEAMS ? "dev_obs must be 16-byte aligned" : "dev_obs must be 4-byte aligned");
    DeviceGuard g(h->device);
    h->chain_open = false;                   // (until this launch is enqueued)
    TRY(fresh_tick(h, K, (cudaStream_t)stream));
    StepParams p = h->p;
    p.actions = dev_actions; p.action_dtype = action_dtype; p.K = K;
    p.obs = (float4 *)dev_obs; p.reward = dev_reward; p.done = dev_done;
    p.history = history;
    // the window kernel needs the actions of the whole rollout up front and at least one full window of steps
    const bool window = h->window > 1 && K >= h->window;
    if (window) CU(launch_window(p, h->window, (cudaStream_t)stream, &h->shape, chain));
    else CU(launch_step(p, h->lanes, (cudaStream_t)stream, &h->shape));
    h->p.step0 += (unsigned)K;
    h->launches++;
    h->chained += chain;
    h->chain_open = window;
    h->chain_stream = (cudaStream_t)stream;
    h->chain_seq = g_enqueues.fetch_add(1, std::memory_order_relaxed) + 1;
    return SHIPSIM_OK;
}

extern "C" int shipsim_step(shipsim_t *h, const void *dev_actions, int action_dtype, int32_t K, float *dev_obs, float *dev_reward,
                            uint8_t *dev_done, void *stream)
{
    if (h) { h->p.log_call = h->calls++; h->p.log_k0 = 0; }
    return step_impl(h, dev_actions, action_dtype, K, dev_obs, dev_reward, dev_done, stream, h ? h->p.history : 1);
}

// Whether this window launch may overlap the handle's previous one: that launch was the last work any handle enqueued
// and it went to the same stream, the configuration is one the CHAIN kernels cover (log-free, 10 beams, no fresh maps:
// their bank regeneration runs on a side stream), and the stream is not being captured (a graph has no previous launch
// to overlap).
static bool chainable(const shipsim_t *h, int32_t K, cudaStream_t s)
{
    if (!h->chain_open || h->chain_stream != s || h->chain_seq != g_enqueues.load(std::memory_order_relaxed)) return false;
    if (!(h->window > 1 && K >= h->window) || h->cfg.lidar_beams != SHIPSIM_N_BEAMS || h->p.log_count || h->fresh.on) return false;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(s, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusNone;
}

extern "C" int shipsim_step_chained(shipsim_t *h, const void *dev_actions, int action_dtype, int32_t K, float *dev_obs,
                                    float *dev_reward, uint8_t *dev_done, void *stream)
{
    if (!h) return shipsim_step(h, dev_actions, action_dtype, K, dev_obs, dev_reward, dev_done, stream);
    const bool chain = h->p.state && chainable(h, K, (cudaStream_t)stream);
    h->p.log_call = h->calls++;
    h->p.log_k0 = 0;
    return step_impl(h, dev_actions, action_dtype, K, dev_obs, dev_reward, dev_done, stream, h->p.history, chain);
}

// ---- shipsim_step_host ------------------------------------------------------------------------------------------------
// With HISTORY_SIZE = 2 an observation is [frame of the previous step | frame of this step] (ship_env.py:112-113): half
// of every row repeats the row before it, and between consecutive frames of an env little changes besides the pose.
// Three regimes, by size:
//  * zero copy: tiny calls with page-locked buffers (the gym facade: one env, one step) -- the kernel reads the actions
//    from the caller's memory and writes rows, rewards and done flags straight into it (mapped pinned memory), one
//    launch and one wait;
//  * plain copies of complete rows.  Small calls are latency bound: everything goes through the caller's stream;
//  * frames only: the kernel runs in its one-frame mode, and the caller's rows are produced by two engines at once,
//    because either alone is the bottleneck (PCIe at ~55 GB/s for 128-byte rows; the host cores' stores for the
//    expansion).  Envs [0, nd): complete rows are put together on the device (history_rows_kernel) and DMA-ed straight
//    into the caller's buffer (when it is page-locked).  Envs [nd, N): a kernel turns the frames into 16-byte records + a
//    stream of changed values (~20 bytes per env-step instead of 64 + 5) and host threads rebuild the rows -- reset
//    observations included.  nd follows the measured balance of the two (DmaSplit).
// The last two cut the rollout into chunks of steps: while chunk i+1 is being computed on the caller's stream, the
// results of chunk i travel to the host on the copy stream (and chunk i-1 is being expanded by the host threads).

// Room in the value stream for all 12 variable slots of every env-step (measured need on the default map: 0.9), so that
// it cannot overflow; untouched pages of the mapping cost nothing.
constexpr int kVarPerStep = 12;

// One chunked shipsim_step_host call
struct HostCall {
    const int32_t *actions;
    float *obs, *reward;                     // (any output may be NULL: it is then not copied back)
    uint8_t *done;
    cudaStream_t s;                          // the caller's stream
    int K;
    size_t N, n, row_full;                   // envs, env-steps, floats per complete row
    bool small, trace;
    int n_chunks = 1, kbeg[kMaxChunks + 1] = {};   // chunk c holds the steps [kbeg[c], kbeg[c + 1])
    bool adaptive = false;                   // frames only: the DMA split nd is DmaSplit's choice
    int nd = 0;

    int kc(int ci) const { return kbeg[ci + 1] - kbeg[ci]; }
    size_t off(int ci) const { return (size_t)kbeg[ci] * N; }     // the chunk's first env-step
};

// Chunk ci of a chunked call: its actions go up (the first chunk's ahead of its kernel, the rest on the aux stream while
// it runs) and its steps are launched on the caller's stream with `hist` frames per row.
static int step_chunk(shipsim_t *h, const HostCall &c, int ci, int hist)
{
    if (ci == 0) {
        CU(cudaMemcpyAsync(h->d_act, c.actions, (size_t)c.kc(0) * c.N * sizeof(int32_t), cudaMemcpyHostToDevice, c.s));
        if (c.n_chunks > 1) {
            CU(cudaEventRecord(h->act_up, c.s));                 // (orders the copy behind whatever the caller's stream did before)
            CU(cudaStreamWaitEvent(h->aux_stream, h->act_up, 0));
            CU(cudaMemcpyAsync(h->d_act + c.off(1), c.actions + c.off(1), (c.n - c.off(1)) * sizeof(int32_t), cudaMemcpyHostToDevice,
                               h->aux_stream));
            CU(cudaEventRecord(h->act_up, h->aux_stream));
        }
    } else if (ci == 1) CU(cudaStreamWaitEvent(c.s, h->act_up, 0));
    h->p.log_k0 = c.kbeg[ci];                                    // episode-log records carry the step index within the call
    const size_t off = c.off(ci);
    const int rc = step_impl(h, h->d_act + off, SHIPSIM_ACTION_I32, c.kc(ci), h->d_obs + off * c.row_full, h->d_rew + off, h->d_done + off,
                             c.s, hist);
    h->p.log_k0 = 0;
    return rc;
}

static int step_plain_copies(shipsim_t *h, const HostCall &c)
{
    for (int ci = 0; ci < c.n_chunks; ++ci) {
        const size_t off = c.off(ci), rows = (size_t)c.kc(ci) * c.N;
        TRY(step_chunk(h, c, ci, h->cfg.history));
        if (c.trace) CU(cudaEventRecord(h->trace_mid[ci], c.s));
        cudaStream_t cs = c.s;                                  // small: one stream, no event hops
        if (!c.small) {
            cs = h->copy_stream;
            CU(cudaEventRecord(h->chunk_done[ci], c.s));
            CU(cudaStreamWaitEvent(h->copy_stream, h->chunk_done[ci], 0));
        }
        h->last_d2h += (int64_t)rows * ((c.reward ? 4 : 0) + (c.done ? 1 : 0));
        if (c.obs) {
            h->last_d2h += (int64_t)(rows * c.row_full * sizeof(float));
            CU(cudaMemcpyAsync(c.obs + off * c.row_full, h->d_obs + off * c.row_full, rows * c.row_full * sizeof(float), cudaMemcpyDeviceToHost, cs));
        }
        if (c.reward) CU(cudaMemcpyAsync(c.reward + off, h->d_rew + off, rows * sizeof(float), cudaMemcpyDeviceToHost, cs));
        if (c.done) CU(cudaMemcpyAsync(c.done + off, h->d_done + off, rows, cudaMemcpyDeviceToHost, cs));
        if (!c.small) CU(cudaEventRecord(h->copy_done[ci], h->copy_stream));
    }
    return SHIPSIM_OK;
}

// The buffers of the compacted wire format, the host threads, and the first frame of every env; then how many envs
// travel as complete rows.
static int frames_setup(shipsim_t *h, HostCall &c)
{
    const size_t N = c.N, n = c.n, nblk = (N + 31) / 32;
    CU(h->d_rec.ensure(n));
    CU(h->d_off.ensure((size_t)c.K * nblk));
    CU(h->d_count.ensure(kMaxChunks));
    CU(h->h_rec.ensure(n * 4));
    CU(h->h_off.ensure((size_t)c.K * nblk));
    CU(h->h_count.ensure(kMaxChunks));
    CU(h->h_var.ensure(n * kVarPerStep));
    CU(h->d_var.ensure(n * kVarPerStep));
    CU(h->h_cur.ensure(N * kFrame));
    CU(h->d_frame0.ensure(N * kFrame / 4));
    if (!h->pool) {
        int nt = std::max(1, std::min(16, (int)std::thread::hardware_concurrency()));
        if (h->cfg.host_threads > 0) nt = std::min(h->cfg.host_threads, 256);
        if (const char *ev = std::getenv("SHIPSIM_HOST_THREADS")) nt = std::max(1, atoi(ev));
        h->pool = std::make_unique<HostPool>(nt - 1);
    }
    CU(launch_frame(h->p, h->d_frame0, c.s));
    CU(cudaMemsetAsync(h->d_count, 0, kMaxChunks * sizeof(unsigned), c.s));
    h->launches++;
    const char *fixed = std::getenv("SHIPSIM_HOST_DMA_ENVS");
    int nd;
    if (pointer_info(c.obs).type != cudaMemoryTypeHost) nd = 0;
    else if (fixed) nd = std::max(0, std::min(atoi(fixed), (int)N));
    else if (n < ((size_t)1 << 18)) nd = 0;                         // (small calls are latency bound either way)
    else {
        c.adaptive = true;
        nd = h->dma.choose((int)N, c.K, h->pool->size());
    }
    c.nd = nd >= (int)N ? (int)N : (nd / 32) * 32;
    CU(h->d_rows.ensure((size_t)c.nd * c.K * 2 * kFrame));
    return SHIPSIM_OK;
}

// The stream work of a frames-only call, chunk by chunk: step kernel, compaction and/or complete rows, and the copies home.
// `issued` counts the chunks whose copies (and copy_done event) are in the copy stream; spec[c] = floats of chunk c's
// value stream copied down unasked.
static int issue_frames(shipsim_t *h, const HostCall &c, size_t *spec, std::atomic<int> &issued)
{
    const size_t N = c.N, nblk = (N + 31) / 32, row_full = c.row_full;
    const int nd = c.nd;
    const bool expand = nd < (int)N;
    cudaStream_t s = c.s;
    const float4 *prev_frames = h->d_frame0;                     // the frames the next chunk's first step is compared with
    for (int ci = 0; ci < c.n_chunks; ++ci) {
        const int k0 = c.kbeg[ci], kc = c.kc(ci);
        const size_t off = c.off(ci);
        const float4 *frames = (const float4 *)(h->d_obs + off * row_full);
        TRY(step_chunk(h, c, ci, 1));
        if (h->p.log_count) {                                    // the one-frame kernel logged the terminal frame only
            CU(launch_log_prev_frames(h->p, frames, prev_frames, k0, kc, s));
            h->launches++;
        }
        if (c.trace) CU(cudaEventRecord(h->trace_mid[ci], s));
        if (expand) {
            CU(launch_compact_frames(frames, prev_frames, h->d_rew + off, h->d_done + off, (int)N, nd, kc, h->cfg.step_penalty, h->d_rec + off,
                                     h->d_off + (size_t)k0 * nblk, h->d_var + off * kVarPerStep,
                                     (unsigned)std::min<size_t>((size_t)kc * N * kVarPerStep, 0xffffffffu), h->d_count + ci, s));
            h->launches++;
        }
        if (nd > 0) {
            CU(launch_history_rows(frames, prev_frames, h->d_done + off, (int)N, nd, kc, h->cfg.auto_reset != 0,
                                   (float4 *)(h->d_rows + (size_t)k0 * nd * row_full), s));
            h->launches++;
        }
        prev_frames = frames + ((size_t)(kc - 1) * N) * 4;
        CU(cudaEventRecord(h->chunk_done[ci], s));
        CU(cudaStreamWaitEvent(h->copy_stream, h->chunk_done[ci], 0));
        if (expand) {
            if (ci == 0) {
                CU(cudaMemcpyAsync(h->h_cur, h->d_frame0, N * kFrame * sizeof(float), cudaMemcpyDeviceToHost, h->copy_stream));
                h->last_d2h += (int64_t)(N * kFrame * sizeof(float));
            }
            if (nd == 0) CU(cudaMemcpyAsync(h->h_rec + off * 4, h->d_rec + off, (size_t)kc * N * sizeof(uint4), cudaMemcpyDeviceToHost, h->copy_stream));
            else CU(cudaMemcpy2DAsync(h->h_rec + (off + nd) * 4, N * sizeof(uint4), h->d_rec + off + nd, N * sizeof(uint4), (N - nd) * sizeof(uint4),
                                      kc, cudaMemcpyDeviceToHost, h->copy_stream));
            CU(cudaMemcpyAsync(h->h_off + (size_t)k0 * nblk, h->d_off + (size_t)k0 * nblk, (size_t)kc * nblk * sizeof(unsigned),
                               cudaMemcpyDeviceToHost, h->copy_stream));
            CU(cudaMemcpyAsync(h->h_count + ci, h->d_count + ci, sizeof(unsigned), cudaMemcpyDeviceToHost, h->copy_stream));
            // the values: how many there are is only known on the device, so a size that has been enough so far goes
            // down unasked (a host thread fetches the rest in the rare case that it was not)
            spec[ci] = std::min((size_t)kc * N * kVarPerStep, (size_t)((double)kc * (N - nd) * h->var_density) + 1024);
            CU(cudaMemcpyAsync(h->h_var + off * kVarPerStep, h->d_var + off * kVarPerStep, spec[ci] * sizeof(float), cudaMemcpyDeviceToHost,
                               h->copy_stream));
            h->last_d2h += (int64_t)kc * (N - nd) * sizeof(uint4) + (int64_t)kc * nblk * sizeof(unsigned) + sizeof(unsigned)
                           + (int64_t)spec[ci] * sizeof(float);
        }
        CU(cudaEventRecord(h->copy_done[ci], h->copy_stream));          // what the host threads wait for
        issued.store(ci + 1, std::memory_order_release);
        if (nd > 0) {
            const size_t w = (size_t)nd * row_full * sizeof(float);
            CU(cudaMemcpy2DAsync(c.obs + off * row_full, N * row_full * sizeof(float), h->d_rows + (size_t)k0 * nd * row_full, w, w, kc,
                                 cudaMemcpyDeviceToHost, h->copy_stream));
            if (c.reward) CU(cudaMemcpy2DAsync(c.reward + off, N * sizeof(float), h->d_rew + off, N * sizeof(float), nd * sizeof(float), kc,
                                               cudaMemcpyDeviceToHost, h->copy_stream));
            if (c.done) CU(cudaMemcpy2DAsync(c.done + off, N, h->d_done + off, N, nd, kc, cudaMemcpyDeviceToHost, h->copy_stream));
            h->last_d2h += (int64_t)kc * nd * (row_full * sizeof(float) + (c.reward ? 4 : 0) + (c.done ? 1 : 0));
        }
    }
    return SHIPSIM_OK;
}

static int step_frames_only(shipsim_t *h, const HostCall &c)
{
    const size_t N = c.N, nblk = (N + 31) / 32;
    const int nd = c.nd;
    size_t spec[kMaxChunks] = {};
    // Every host thread owns a contiguous range of env blocks for the whole call (the running frames of its envs stay in its
    // cache) and walks the chunks as their records arrive: no barrier between chunks.  Whoever finds the next chunk missing
    // polls its event.  The threads are started BEFORE the stream work is issued (launching 16 chunks of kernels and copies
    // takes the calling thread ~1 ms, a fifth of the call), and the calling thread joins them when it is done.
    const bool expand = nd < (int)N;
    const size_t blk0 = (size_t)nd / 32;
    const int jobs = expand ? (int)std::min<size_t>(nblk - blk0, (size_t)h->pool->size()) : 0;
    std::atomic<int> ready{0};                                   // chunks whose records are in host memory
    std::atomic<int> issued{0};                                  // chunks whose copies (and event) are in the copy stream
    std::atomic<int> bad{0};
    std::mutex poll, fix;
    bool fixed[kMaxChunks] = {};
    std::atomic<long long> extra_d2h{0};
    const std::function<void(int)> worker = [&](int j) {
        cudaSetDevice(h->device);
        const size_t b0 = blk0 + (nblk - blk0) * (size_t)j / jobs, b1 = blk0 + (nblk - blk0) * (size_t)(j + 1) / jobs;
        for (int ci = 0; ci < c.n_chunks; ++ci) {
            while (ready.load(std::memory_order_acquire) <= ci) {
                if (bad.load(std::memory_order_relaxed)) return;
                if (poll.try_lock()) {
                    const int r = ready.load(std::memory_order_relaxed);
                    if (r <= ci && r < issued.load(std::memory_order_acquire)) {     // (an event not yet recorded by this call reads as complete)
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
            const size_t off = c.off(ci);
            if (h->h_count[ci] > spec[ci]) {                     // the speculative copy fell short: one thread fetches the rest
                std::lock_guard<std::mutex> lk(fix);
                if (!fixed[ci]) {
                    const size_t at = off * kVarPerStep + spec[ci];
                    cudaError_t q = cudaMemcpyAsync(h->h_var + at, h->d_var + at, (h->h_count[ci] - spec[ci]) * sizeof(float), cudaMemcpyDeviceToHost,
                                                    h->aux_stream);
                    if (q == cudaSuccess) q = cudaStreamSynchronize(h->aux_stream);
                    if (q != cudaSuccess) { bad.store((int)q); return; }
                    extra_d2h.fetch_add((long long)(h->h_count[ci] - spec[ci]) * (long long)sizeof(float));
                    fixed[ci] = true;
                }
            }
            expand_delta_rows(c.obs + off * c.row_full, c.reward ? c.reward + off : nullptr, c.done ? c.done + off : nullptr, h->h_rec + off * 4,
                              h->h_off + (size_t)c.kbeg[ci] * nblk, h->h_var + off * kVarPerStep, h->h_cur, c.kc(ci), N, b0, b1,
                              h->cfg.step_penalty, h->cfg.auto_reset != 0, 2);
        }
    };
    if (expand) h->pool->start(jobs, worker);
    const int rc_issue = issue_frames(h, c, spec, issued);
    if (!expand) return rc_issue;
    if (rc_issue) bad.store(-1);
    h->pool->finish();
    if (rc_issue) return rc_issue;
    if (bad.load()) return fail(SHIPSIM_ERR_CUDA, std::string("copy stream: ") + cudaGetErrorString((cudaError_t)bad.load()));
    h->last_d2h += extra_d2h.load();
    double dens = 0.0;
    for (int ci = 0; ci < c.n_chunks; ++ci) dens = std::max(dens, (double)h->h_count[ci] / ((double)c.kc(ci) * (double)(N - nd)));
    h->var_density = std::max(0.9 * h->var_density, std::min(12.0, 1.25 * dens + 0.25));       // follows the need up at once, down slowly
    return SHIPSIM_OK;
}

static int step_host_impl(shipsim_t *h, const int32_t *host_actions, int32_t K, float *host_obs, float *host_reward,
                          uint8_t *host_done, void *stream)
{
    TRY(ready(h));
    if (K < 1 || !host_actions) return fail(SHIPSIM_ERR_ARG, "K must be >= 1 and host_actions non-NULL");
    DeviceGuard g(h->device);
    h->p.log_call = h->calls++;
    h->p.log_k0 = 0;
    const size_t N = (size_t)h->cfg.num_envs, n = N * K, row_full = (size_t)frame_floats(h) * h->cfg.history;
    cudaStream_t s = (cudaStream_t)stream;
    if (n * row_full * sizeof(float) <= ((size_t)1 << 16) && host_obs && host_reward && host_done) {
        // zero copy, when all four buffers are mapped page-locked memory (the aliases of the last call's are remembered)
        const void *host[4] = {host_actions, host_obs, host_reward, host_done};
        if (!std::equal(host, host + 4, h->zc_host)) {
            std::copy(host, host + 4, h->zc_host);
            for (int i = 0; i < 4; ++i)
                if (!(h->zc_dev[i] = pointer_info(host[i]).alias)) { std::fill(h->zc_dev, h->zc_dev + 4, nullptr); break; }
        }
        if (h->zc_dev[0]) {
            void *const *dev = h->zc_dev;
            TRY(step_impl(h, dev[0], SHIPSIM_ACTION_I32, K, (float *)dev[1], (float *)dev[2], (uint8_t *)dev[3], s, h->cfg.history));
            h->last_h2d = (int64_t)(n * sizeof(int32_t));
            h->last_d2h = (int64_t)(n * (row_full * sizeof(float) + 5));
            CU(cudaStreamSynchronize(s));
            return SHIPSIM_OK;
        }
    }
    // the chunked regimes: staging buffers, the copy and aux streams and the per-chunk events.  A trace reads the times
    // of the chunk events, so they are created with timing while calls ask for a trace (without, which is cheaper, else).
    const bool small = n < ((size_t)1 << 16), trace = std::getenv("SHIPSIM_HOST_TRACE") != nullptr;
    CU(h->d_act.ensure(n));
    CU(h->d_obs.ensure(n * row_full));
    CU(h->d_rew.ensure(n));
    CU(h->d_done.ensure(n));
    if (!h->act_up) {                                               // (the last of the three to be created)
        CU(cudaStreamCreateWithFlags(h->copy_stream.out(), cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(h->aux_stream.out(), cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(h->act_up.out(), cudaEventDisableTiming));
    }
    if (h->chunk_events != (int)trace) {
        for (auto &ev : h->chunk_done) CU(cudaEventCreateWithFlags(ev.out(), trace ? cudaEventDefault : cudaEventDisableTiming));
        for (auto &ev : h->copy_done) CU(cudaEventCreateWithFlags(ev.out(), trace ? cudaEventDefault : cudaEventDisableTiming));
        h->chunk_events = (int)trace;
    }
    if (trace && !h->trace0) {                                      // (trace0 is created last)
        for (auto &ev : h->trace_mid) CU(cudaEventCreate(ev.out()));
        CU(cudaEventCreate(h->trace0.out()));
    }
    HostCall c{host_actions, host_obs, host_reward, host_done, s, K, N, n, row_full, small, trace};
    c.n_chunks = small ? 1 : (K >= 64 ? 16 : (K >= 8 ? 8 : 1));
    if (const char *ev = std::getenv("SHIPSIM_HOST_CHUNKS")) c.n_chunks = std::max(1, std::min({atoi(ev), kMaxChunks, (int)K}));
    for (int ci = 0; ci <= c.n_chunks; ++ci) c.kbeg[ci] = (int)((int64_t)K * ci / c.n_chunks);
    for (int ci = 0; ci < c.n_chunks; ++ci)
        if (c.kc(ci) <= 0) return fail(SHIPSIM_ERR_ARG, "internal: empty chunk");
    // (the compacted wire format is that of 16-float frames: other fans take the plain copies)
    const bool frames_only = h->cfg.history == 2 && host_obs != nullptr && !small && h->cfg.lidar_beams == SHIPSIM_N_BEAMS;
    if (frames_only) TRY(frames_setup(h, c));
    if (trace) CU(cudaEventRecord(h->trace0, s));
    h->last_h2d = (int64_t)(n * sizeof(int32_t));                // (the actions go up chunk by chunk, ahead of the chunk's kernel)
    h->last_d2h = 0;
    if (const char *ev = std::getenv("SHIPSIM_HOST_VAR_DENSITY")) h->var_density = atof(ev);      // (test hook: 0 forces the fetch-the-rest path)
    using clk = std::chrono::steady_clock;
    const auto t_begin = clk::now();
    TRY(frames_only ? step_frames_only(h, c) : step_plain_copies(h, c));
    if (!small) CU(cudaStreamSynchronize(h->copy_stream));
    CU(cudaStreamSynchronize(s));
    if (trace && !small) {
        std::fprintf(stderr, "step_host trace (ms since the call's first stream op): host done %.2f\n",
                     std::chrono::duration<double, std::milli>(clk::now() - t_begin).count());
        for (int ci = 0; ci < c.n_chunks; ++ci) {
            float a = 0.f, b = 0.f, m = 0.f;
            cudaEventElapsedTime(&a, h->trace0, h->chunk_done[ci]);
            cudaEventElapsedTime(&b, h->trace0, h->copy_done[ci]);
            cudaEventElapsedTime(&m, h->trace0, h->trace_mid[ci]);
            std::fprintf(stderr, "  chunk %2d: step kernel done %.2f  compaction done %.2f  records home %.2f\n", ci, m, a, b);
        }
    }
    if (c.adaptive) h->dma.update((int)N, c.nd, std::chrono::duration<double>(clk::now() - t_begin).count() / (double)n);
    return SHIPSIM_OK;
}

extern "C" int shipsim_step_host(shipsim_t *h, const int32_t *host_actions, int32_t K, float *host_obs, float *host_reward,
                                 uint8_t *host_done, void *stream)
{
    const int rc = step_host_impl(h, host_actions, K, host_obs, host_reward, host_done, stream);
    unchain(h);                              // (its window launches, if any, are no anchor for a chain)
    return rc;
}

extern "C" int shipsim_mlp_policy_forward(const float *dev_obs, int32_t num_envs, const float *dev_w1, const float *dev_b1, const float *dev_w2,
                                          const float *dev_b2, const float *dev_w3, const float *dev_b3, const float *dev_noise, float *dev_out,
                                          int64_t *dev_actions, void *stream)
{
    unchain(nullptr);
    if (!dev_obs || !dev_w1 || !dev_b1 || !dev_w2 || !dev_b2 || !dev_w3 || !dev_b3 || !dev_noise || !dev_out || !dev_actions || num_envs < 1)
        return fail(SHIPSIM_ERR_ARG, "NULL buffer or num_envs < 1");
    // the kernel moves these in 16-byte units (cp.async of the weights, float4 loads and stores) and the actions as int64
    const struct { const void *p; uintptr_t mask; const char *msg; } aligned[] = {
        {dev_obs, 15, "dev_obs must be 16-byte aligned"}, {dev_w1, 15, "dev_w1 must be 16-byte aligned"},
        {dev_b1, 15, "dev_b1 must be 16-byte aligned"},   {dev_w2, 15, "dev_w2 must be 16-byte aligned"},
        {dev_b2, 15, "dev_b2 must be 16-byte aligned"},   {dev_w3, 15, "dev_w3 must be 16-byte aligned"},
        {dev_out, 15, "dev_out must be 16-byte aligned"}, {dev_actions, 7, "dev_actions must be 8-byte aligned"}};
    for (const auto &a : aligned)
        if (((uintptr_t)a.p & a.mask) != 0) return fail(SHIPSIM_ERR_ARG, a.msg);
    CU(launch_mlp_policy(dev_obs, num_envs, dev_w1, dev_b1, dev_w2, dev_b2, dev_w3, dev_b3, dev_noise, dev_out, (long long *)dev_actions,
                         (cudaStream_t)stream));
    return SHIPSIM_OK;
}

extern "C" int shipsim_gae(const float *dev_rewards, const float *dev_values, const uint8_t *dev_dones, int32_t n_steps, int32_t num_envs, float gamma,
                           float lam, float *dev_adv, float *dev_returns, void *stream)
{
    unchain(nullptr);
    if (!dev_rewards || !dev_values || !dev_dones || !dev_adv || !dev_returns || n_steps < 1 || num_envs < 1)
        return fail(SHIPSIM_ERR_ARG, "NULL buffer or bad sizes");
    CU(launch_gae(dev_rewards, dev_values, dev_dones, n_steps, num_envs, gamma, lam, dev_adv, dev_returns, (cudaStream_t)stream));
    return SHIPSIM_OK;
}

extern "C" int shipsim_gae_scored(shipsim_t *h, const float *dev_rewards, const float *dev_values, const uint8_t *dev_dones, int32_t n_steps,
                                  float gamma, float lam, int32_t call0, int32_t steps_per_call, float *dev_adv, float *dev_returns,
                                  int32_t *dev_step_scenario, double *dev_scores, void *stream)
{
    unchain(h);
    TRY(ready(h));
    if (!h->cfg.auto_reset) return fail(SHIPSIM_ERR_STATE, "level scores need auto_reset (they attribute steps through the episode log)");
    if (!h->p.log_count) return fail(SHIPSIM_ERR_STATE, "level scores need the episode log: call shipsim_episode_log_bind first");
    if (!dev_rewards || !dev_values || !dev_dones || !dev_adv || !dev_returns || !dev_step_scenario || !dev_scores || n_steps < 1 || steps_per_call < 1)
        return fail(SHIPSIM_ERR_ARG, "NULL buffer or bad sizes");
    if (((uintptr_t)dev_scores & 7) || ((uintptr_t)dev_step_scenario & 3))
        return fail(SHIPSIM_ERR_ARG, "dev_scores must be 8-byte and dev_step_scenario 4-byte aligned");
    DeviceGuard g(h->device);
    const StepParams &p = h->p;
    CU(launch_gae_scored(dev_rewards, dev_values, dev_dones, n_steps, h->cfg.num_envs, gamma, lam, dev_adv, dev_returns, p.log_meta, p.log_count,
                         p.log_cap, call0, steps_per_call, p.state + (size_t)4 * h->cfg.num_envs, p.n_scen, (int *)dev_step_scenario, dev_scores,
                         (cudaStream_t)stream));
    h->launches += 2;
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
    unchain(h);
    TRY(ready(h));
    if (!dev_out) return fail(SHIPSIM_ERR_ARG, "dev_out is NULL");
    DeviceGuard g(h->device);
    CU(launch_stats_reduce(h->p.stats, dev_out, clear, (cudaStream_t)stream));
    h->launches++;
    return SHIPSIM_OK;
}

// An env's state as the floats of its planes (plane-major, 4 per plane): pose [0, 6), episode return 6, packed rudder /
// alive / steps 7, lidar[0, 10) from 8, scenario 18 and episode 19 (int bits), goals [20, 30), 0 at 30 and 31, then
// lidar[10 ..) from 32.  Readings past the fan hold -1.
constexpr int kStateFloats = 4 * (kPlanes + (kMaxBeams - kBeams + 3) / 4);
static int lidar_slot(int j) { return j < kBeams ? 8 + j : 4 * kPlanes + j - kBeams; }

extern "C" int shipsim_set_state(shipsim_t *h, const float *pose, const int32_t *ints, const float *lidar, const float *goals,
                                 const float *ep_return)
{
    unchain(h);
    TRY(ready(h));
    if (!pose || !ints || !lidar || !goals || !ep_return) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    const size_t N = (size_t)h->cfg.num_envs;
    const int nb = h->cfg.lidar_beams, planes = state_planes(h);
    std::vector<float4> st(N * planes);
    for (size_t e = 0; e < N; ++e) {
        const int32_t *in = ints + e * 5;
        if (in[0] % 5 != 0 || in[0] < -10 || in[0] > 10) return fail(SHIPSIM_ERR_ARG, "rudder must be in {-10,-5,0,5,10}");
        if (in[3] < 0 || in[3] >= h->p.n_scen) return fail(SHIPSIM_ERR_ARG, "scenario id out of range");
        const int bits = ((in[0] / 5 + 2) & 7) | ((in[1] & 31) << 3) | (in[2] << 8);
        float f[kStateFloats] = {};
        std::copy(pose + e * 6, pose + e * 6 + 6, f);
        f[6] = ep_return[e];
        std::memcpy(f + 7, &bits, 4);
        std::memcpy(f + 18, in + 3, 8);
        std::copy(goals + e * 10, goals + e * 10 + 10, f + 20);
        for (int j = 0; j < kBeams + 4 * (planes - kPlanes); ++j) f[lidar_slot(j)] = j < nb ? lidar[e * nb + j] : -1.f;
        for (int pl = 0; pl < planes; ++pl) std::memcpy(&st[pl * N + e], f + 4 * pl, sizeof(float4));
    }
    DeviceGuard g(h->device);
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(h->p.state, st.data(), st.size() * sizeof(float4), cudaMemcpyHostToDevice));
    return SHIPSIM_OK;
}

extern "C" int shipsim_get_state(shipsim_t *h, float *pose, int32_t *ints, float *lidar, float *goals, float *ep_return)
{
    unchain(h);
    TRY(ready(h));
    const size_t N = (size_t)h->cfg.num_envs;
    const int nb = h->cfg.lidar_beams, planes = state_planes(h);
    std::vector<float4> st(N * planes);
    DeviceGuard g(h->device);
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(st.data(), h->p.state, st.size() * sizeof(float4), cudaMemcpyDeviceToHost));
    for (size_t e = 0; e < N; ++e) {
        float f[kStateFloats];
        for (int pl = 0; pl < planes; ++pl) std::memcpy(f + 4 * pl, &st[pl * N + e], sizeof(float4));
        int bits;
        std::memcpy(&bits, f + 7, 4);
        if (pose) std::copy(f, f + 6, pose + e * 6);
        if (ep_return) ep_return[e] = f[6];
        if (ints) {
            int32_t *in = ints + e * 5;
            in[0] = ((bits & 7) - 2) * 5; in[1] = (bits >> 3) & 31; in[2] = bits >> 8;
            std::memcpy(in + 3, f + 18, 8);
        }
        if (lidar) for (int j = 0; j < nb; ++j) lidar[e * nb + j] = f[lidar_slot(j)];
        if (goals) std::copy(f + 20, f + 30, goals + e * 10);
    }
    return SHIPSIM_OK;
}

extern "C" int shipsim_render(shipsim_t *h, int32_t env_index, int32_t width, int32_t height, uint8_t *dev_rgb, void *stream)
{
    unchain(h);
    TRY(ready(h));
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

extern "C" int shipsim_chained_count(const shipsim_t *h, int64_t *out)
{
    if (!h || !out) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    *out = h->chained;
    return SHIPSIM_OK;
}

extern "C" int shipsim_launch_window(const shipsim_t *h, int32_t *steps_in_flight)
{
    if (!h || !steps_in_flight) return fail(SHIPSIM_ERR_ARG, "NULL argument");
    *steps_in_flight = h->shape.window;
    return SHIPSIM_OK;
}
