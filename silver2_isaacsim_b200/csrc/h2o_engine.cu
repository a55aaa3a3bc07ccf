// h2o_engine.cu -- host side of libh2o_b200.so: handle, parameter upload, kernel
// dispatch, CUDA-graph rollouts, host-buffer pipeline, DLPack validation.  The C ABI is
// declared in include/h2o.h and include/h2o_dlpack.h (which cite the reference interfaces).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/h2o_dlpack.h"
#include "h2o_kernels.cuh"

using namespace h2o;

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local std::string g_last_error;

static int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                           \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            return fail(H2O_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),    \
                        __FILE__, __LINE__);                                                     \
    } while (0)

// ---------------------------------------------------------------------------
// engine
// ---------------------------------------------------------------------------
static constexpr uint32_t H2O_MAGIC = 0x48324f42u;  // "H2OB"
static constexpr int HOST_PIPE_STREAMS = 3;

struct h2o_engine {
    uint32_t magic = H2O_MAGIC;
    int device = 0;
    int dtype = H2O_F32;
    int64_t n = 0;
    size_t esz = 4;
    double rho = 1025.0, grav = 9.81;
    double current[3] = {0.0, 0.0, 0.0};  // uniform water current
    double surface_z = 0.0;               // flat water surface height
    int param_mode = -1;  // -1 unset, PARAM_TABLE, PARAM_PER_BODY
    void* coeff = nullptr;
    int64_t coeff_rows = 0;
    int32_t* slot_type = nullptr;
    int n_slots = 0, n_types = 0;
    void* prev = nullptr;
    double* stats = nullptr;
    uint32_t* redo_bitmap = nullptr;  // one bit per body, all zero between launches (tile kernel, deferred-list overflow)
    bool stats_on = false;
    int bodies_per_robot = 0;
    int quat_order = H2O_QUAT_XYZW;
    int kernel_choice = H2O_KERNEL_AUTO;
    int last_kernel = 0;
    int64_t launches = 0;
    int sm_count = 148;
    int tile_cfg = 0;          // 0 = default configuration of the dtype
    void* am_dense = nullptr;  // (am_types, 6, 6) dense added-mass matrices in the engine dtype, or nullptr
    int32_t* am_slot_type = nullptr;
    int am_types = 0, am_slots = 0;
    const void* surface_eta = nullptr;  // (n,) per-body surface heights, borrowed, or nullptr = flat
    double* wave_tab = nullptr;    // (MAX_WAVE_COMPONENTS, WAVE_STRIDE) wave table, first n_waves rows in use
    double* wave_clock = nullptr;  // the wave field's clock (one double, device)
    int n_waves = 0;               // 0 = no wave field
    double wave_depth = INFINITY;
    int wave_slope = 0;            // 1: with a wave field, bodies are tested against the surface's tangent plane
    int fluid_inertia = 0;         // 1: Froude-Krylov force and added mass on the fluid-relative acceleration
    const double* env_cond = nullptr;  // (n / bodies_per_env, ENV_STRIDE) per-env conditions, borrowed, or nullptr
    long long bodies_per_env = 0;
    GridArgs grid{};  // current grid (borrowed values, dims and geometry); grid.vals == nullptr = none
    long long* robot_offsets = nullptr;  // (n_robots_var + 1,) body offsets of unequal robots, or nullptr
    long long n_robots_var = 0;
    int max_ctas_per_sm = 0;   // 0 = as many as fit
    int warp_compat = 0;       // components entry point reproduces the Warp twin's deviations
    int robot_cfg = -1;        // -1 = pick the CTA size by lane utilisation (tuning override: 0,1,2)
    int rollout_free_bodies = 0;  // 1: rollouts integrate the bound state between steps (free bodies)
    double rollout_gravity = 9.81;
    int last_ctas_per_sm = 0;
    int last_overlap = 0;      // 1: the last tile launch was captured to start while the previous grid drains
    // bound tensors
    bool bound = false;
    int b_layout = LAYOUT_SPLIT;
    const void *b_pos = nullptr, *b_quat = nullptr, *b_lin = nullptr, *b_ang = nullptr;
    void *b_f = nullptr, *b_t = nullptr, *b_w = nullptr;
    // rollout graph
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graph_exec = nullptr;
    int graph_steps = 0;
    int64_t graph_launches_per_replay = 0;
    // host pipeline
    void* hp_dev[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // pos quat lin ang F T W
    void* hp_pin[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t hp_dev_bytes[4] = {0, 0, 0, 0}, hp_pin_bytes[4] = {0, 0, 0, 0};
    cudaStream_t hp_stream[HOST_PIPE_STREAMS] = {nullptr, nullptr, nullptr};
    cudaEvent_t hp_event = nullptr;
    int last_host_path = 0;  // 1 = zero-copy (kernel on the pinned host buffers), 2 = staged chunk pipeline
    cudaStream_t capture_stream = nullptr;  // graph capture never runs on the caller's (maybe legacy) stream
    int no_fallback = 0;       // study knob (H2O_NO_FALLBACK=1): flagged bodies keep their fast-path result
    bool dry_run = false;  // launch helpers do their one-time attribute / occupancy set-up and count, but launch nothing
};

// A captured rollout bakes in device pointers (coefficients, slot maps, dense added mass, robot offsets)
// and constants (rho, g, environment, quaternion order, statistics flag, kernel / tile choice).  Every
// setter that changes one of them drops the graph; h2o_launch_rollout then reports NOT_CONFIGURED until
// h2o_capture_rollout is called again, instead of replaying kernels over freed or stale memory.
static void invalidate_graph(h2o_engine* e)
{
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
    if (e->graph) { cudaGraphDestroy(e->graph); e->graph = nullptr; }
    e->graph_steps = 0;
    e->graph_launches_per_replay = 0;
}

static WaveArgs wave_args(const h2o_engine* e)
{
    WaveArgs w;
    w.tab = e->wave_tab; w.clock = e->wave_clock; w.depth = e->wave_depth; w.n = e->n_waves;
    return w;
}

static EnvArgs env_args(const h2o_engine* e)
{
    EnvArgs v;
    v.cond = e->env_cond; v.bodies_per_env = e->bodies_per_env;
    return v;
}

// The water clock advances after every step when something reads it: a wave field or a time-varying grid.
static bool clock_runs(const h2o_engine* e) { return e->n_waves || (e->grid.vals && e->grid.nt > 1); }

static h2o_engine* check(h2o_handle h)
{
    if (!h || h->magic != H2O_MAGIC) {
        fail(H2O_ERR_BAD_HANDLE, "invalid h2o handle");
        return nullptr;
    }
    return h;
}

struct DeviceGuard {
    int old = -1;
    explicit DeviceGuard(int dev)
    {
        cudaGetDevice(&old);
        if (old != dev) cudaSetDevice(dev);
        else old = -1;
    }
    ~DeviceGuard()
    {
        if (old >= 0) cudaSetDevice(old);
    }
};

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---------------------------------------------------------------------------
// tile-kernel configurations
// ---------------------------------------------------------------------------
// T bodies per tile (= threads per CTA), I-deep TMA load ring, O store buffers,
// MB = minimum CTAs per SM promised to the compiler (register budget).
template <int T, int I, int O, int MB, bool CO = false, int BPR = 0> struct Cfg {
    static constexpr int kThreads = T, kIn = I, kOut = O, kMinBlocks = MB;
    static constexpr bool kCopyOnly = CO;  // measurement aid: memory traffic without arithmetic
    static constexpr int kBpr = BPR;       // robot mode specialised for this robot size (0 = run time)
};
#ifndef H2O_MB_DEFAULT
#define H2O_MB_DEFAULT 6
#endif
#ifndef H2O_MB_HEXAPOD
#define H2O_MB_HEXAPOD 4
#endif
template <typename S> struct DefaultCfg;
template <> struct DefaultCfg<float> { using type = Cfg<128, 1, 2, H2O_MB_DEFAULT>; };
template <> struct DefaultCfg<double> { using type = Cfg<64, 1, 2, 6>; };
// With an articulation a tile holds whole robots (and whole 16-byte granules), e.g. 19-body
// hexapods -> multiples of 76 bodies.  Several CTA sizes are compiled and the one whose lanes are
// best used is picked per bodies_per_robot (19: 160 threads carry 152 bodies = 95 %).
// the reference's robot: SILVER2 = Body + 6 x (Coxa, Femur, Tibia) scripted prims (SURVEY.md 8(d) C2)
constexpr int HEXAPOD_BODIES = 19;
template <typename S> struct RobotCfgs;
template <> struct RobotCfgs<float> {
    using A = Cfg<128, 1, 2, 6>;
    using B = Cfg<160, 1, 2, 4>;
    using C = Cfg<256, 1, 2, 3>;
    using Hexapod = Cfg<160, 1, 2, H2O_MB_HEXAPOD, false, HEXAPOD_BODIES>;  // = B with the robot size compiled in
};
template <> struct RobotCfgs<double> {
    using A = Cfg<64, 1, 2, 6>;
    using B = Cfg<96, 1, 2, 4>;
    using C = Cfg<160, 1, 2, 2>;
    using Hexapod = Cfg<160, 1, 2, 2, false, HEXAPOD_BODIES>;  // = C with the robot size compiled in
};

template <typename S, int kLayout, int kParam, bool kRobot, bool kStats, typename C> struct TileLaunch {
    using SM = TileSmem<S, kLayout, kParam, C::kThreads, C::kIn, C::kOut>;
    static auto kernel()
    {
        return &step_tile_kernel<S, kLayout, kParam, kRobot, kStats, C::kThreads, C::kIn, C::kOut, C::kMinBlocks,
                                 C::kCopyOnly, C::kBpr>;
    }
    static size_t smem() { return SM::total(kRobot); }
    static cudaError_t prepare(int* ctas_per_sm)
    {
        cudaError_t e =
            cudaFuncSetAttribute(kernel(), cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem()));
        if (e != cudaSuccess) return e;
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, kernel(), C::kThreads, smem());
    }
};

static long long gcd_ll(long long a, long long b) { return b ? gcd_ll(b, a % b) : a; }

// smallest tile granule: 4 (fp32) or 2 (fp64) bodies keep every stream 16-byte aligned;
// with an articulation a tile must also hold whole robots
static long long tile_unit(size_t esz, int bodies_per_robot)
{
    const long long granule = (long long)(16 / esz);
    if (bodies_per_robot <= 0) return granule;
    return granule / gcd_ll(granule, bodies_per_robot) * bodies_per_robot;
}

// largest tile (bodies) a CTA of `threads` threads can take
static int tile_bodies_for(int threads, size_t esz, int bodies_per_robot)
{
    const long long l = tile_unit(esz, bodies_per_robot);
    if (l > threads) return 0;  // robot does not fit a tile: fused reduction unavailable
    return int(threads / l * l);
}

// ---------------------------------------------------------------------------
// launch overlap of consecutive tile kernels
// ---------------------------------------------------------------------------
// A tile kernel launched with overlap = 1 loads, computes and stores its first tile before it waits for the previous
// grid of its stream (h2o_kernels.cuh, step_tile_kernel).  The host allows that only for two tile launches of the
// library that are adjacent in one stream capture and whose memory accesses do not conflict.  Eager launches always
// wait first: a kernel launched by someone else between two library launches cannot be seen there.

struct Span {  // bytes [lo, hi) of device memory
    uintptr_t lo, hi;
};

struct TileAccess {  // what one tile-kernel launch reads and writes
    Span rd[8];
    Span wr[6];
    int n_rd = 0, n_wr = 0;
};

static void add_span(Span* s, int& n, const void* p, size_t bytes)
{
    if (!p || bytes == 0) return;
    const uintptr_t lo = reinterpret_cast<uintptr_t>(p);
    s[n++] = Span{lo, lo + bytes};
}

static bool spans_meet(const Span* a, int na, const Span* b, int nb)
{
    for (int i = 0; i < na; ++i)
        for (int j = 0; j < nb; ++j)
            if (a[i].lo < b[j].hi && b[j].lo < a[i].hi) return true;
    return false;
}

// The later launch may start before the earlier one has finished: it reads nothing the earlier one writes, writes
// nothing the earlier one writes, and writes nothing the earlier one reads.
static bool accesses_commute(const TileAccess& earlier, const TileAccess& later)
{
    return !spans_meet(earlier.wr, earlier.n_wr, later.rd, later.n_rd) &&
           !spans_meet(earlier.wr, earlier.n_wr, later.wr, later.n_wr) &&
           !spans_meet(later.wr, later.n_wr, earlier.rd, earlier.n_rd);
}

// Every byte a tile launch of `a` (tile_bodies / n_tiles set) may touch, deferred float64 re-evaluation included.
template <typename S, int kLayout, int kParam, bool kRobot>
static TileAccess tile_access(const StepArgs& a)
{
    using TL = TileLayout<S, kLayout, kParam>;
    const size_t rows = size_t(a.n_tiles) * size_t(a.tile_bodies);
    const size_t col = rows * sizeof(S);
    TileAccess t;
    add_span(t.rd, t.n_rd, a.pos, col * TL::E_POS);
    if (TL::E_QUAT) add_span(t.rd, t.n_rd, a.quat, col * TL::E_QUAT);
    add_span(t.rd, t.n_rd, a.lin, col * TL::E_LIN);
    if (TL::E_ANG) add_span(t.rd, t.n_rd, a.ang, col * TL::E_ANG);
    add_span(t.rd, t.n_rd, a.prev, col * TL::E_PREV);
    if (kParam == PARAM_PER_BODY) {
        add_span(t.rd, t.n_rd, a.coeff, col * N_COEFF);
    } else {
        add_span(t.rd, t.n_rd, a.coeff, size_t(a.n_types) * N_COEFF * sizeof(S));
        add_span(t.rd, t.n_rd, a.slot_type, size_t(a.n_slots) * sizeof(int32_t));
    }
    add_span(t.wr, t.n_wr, a.out_force, col * 3);
    add_span(t.wr, t.n_wr, a.out_torque, col * 3);
    add_span(t.wr, t.n_wr, a.prev, col * TL::E_PREV);
    if (kRobot && a.bodies_per_robot > 0)
        add_span(t.wr, t.n_wr, a.out_wrench, rows / size_t(a.bodies_per_robot) * 6 * sizeof(S));
    add_span(t.wr, t.n_wr, a.stats, N_STATS * sizeof(double));
    if (rows > 0) {  // the bitmap words of bodies first_body .. first_body + rows - 1
        const size_t w0 = size_t(a.first_body) >> 5, w1 = (size_t(a.first_body) + rows - 1) >> 5;
        add_span(t.wr, t.n_wr, a.redo_bitmap + w0, (w1 - w0 + 1) * sizeof(uint32_t));
    }
    return t;
}

// The library's last tile launch per stream, kept while that stream is being captured.
struct LastTile {
    unsigned long long capture_id;
    cudaGraphNode_t node;
    TileAccess access;
};
static std::mutex g_last_tile_mu;
static std::unordered_map<cudaStream_t, LastTile> g_last_tile;

// Any other library kernel on the stream: the next tile launch there waits first.
static void forget_last_tile(cudaStream_t s)
{
    std::lock_guard<std::mutex> lk(g_last_tile_mu);
    g_last_tile.erase(s);
}

struct CaptureState {
    bool capturing = false;
    unsigned long long id = 0;
    cudaGraphNode_t only_dep = nullptr;  // the single node the next captured work depends on, or nullptr
};

static CaptureState capture_state(cudaStream_t s)
{
    CaptureState c;
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    const cudaGraphNode_t* deps = nullptr;
    const cudaGraphEdgeData* edges = nullptr;
    size_t n_deps = 0;
    if (cudaStreamGetCaptureInfo_v3(s, &st, &c.id, nullptr, &deps, &edges, &n_deps) != cudaSuccess) {
        cudaGetLastError();  // not an error of the launch: it then simply waits first
        return CaptureState{};
    }
    c.capturing = st == cudaStreamCaptureStatusActive;
    if (c.capturing && n_deps == 1) c.only_dep = deps[0];
    return c;
}

// The overlap decision for a tile launch with access record `acc` after `last` (nullptr = none) in a stream in
// capture state `c`.
static bool may_start_early(const LastTile* last, const CaptureState& c, const TileAccess& acc)
{
    return c.capturing && last && last->capture_id == c.id && c.only_dep && c.only_dep == last->node &&
           accesses_commute(last->access, acc);
}

template <typename S, int kLayout, int kParam, bool kRobot, bool kStats, typename C>
static int launch_tile(h2o_engine* e, StepArgs& a, cudaStream_t stream)
{
    using TLn = TileLaunch<S, kLayout, kParam, kRobot, kStats, C>;
    static int ctas_per_sm[16] = {0};
    int dev = e->device & 15;
    if (ctas_per_sm[dev] == 0) {
        int c = 0;
        CUDA_TRY(TLn::prepare(&c));
        if (c < 1) return fail(H2O_ERR_CUDA, "tile kernel does not fit on an SM (smem %zu)", TLn::smem());
        ctas_per_sm[dev] = c;
    }
    const int tb_max = tile_bodies_for(C::kThreads, sizeof(S), kRobot ? a.bodies_per_robot : 0);
    if (tb_max <= 0)
        return fail(H2O_ERR_BAD_ARGUMENT, "a robot of %d bodies does not fit a %d-thread tile (H2O_ROBOT_CFG?)",
                    a.bodies_per_robot, C::kThreads);
    if (C::kBpr > 0 && (a.bodies_per_robot != C::kBpr ||
                        tb_max != tile_bodies_static(C::kThreads, int(sizeof(S)), C::kBpr > 0 ? C::kBpr : 1)))
        return fail(H2O_ERR_BAD_ARGUMENT, "kernel specialised for %d-body robots launched with %d", C::kBpr,
                    a.bodies_per_robot);
    int cps = ctas_per_sm[dev];
    if (e->max_ctas_per_sm > 0) cps = std::min(cps, e->max_ctas_per_sm);
    const long long slots = (long long)e->sm_count * cps;
    a.tile_bodies = tb_max;
    a.n_tiles = int(std::min<long long>(a.n / tb_max, 0x7fffffff));
    const int grid = int(std::max<long long>(1, std::min<long long>(a.n_tiles, slots)));
    a.overlap = 0;
    if (e->dry_run) {
        e->launches += 1;
        e->last_ctas_per_sm = cps;
        return H2O_OK;
    }
    // Programmatic stream serialisation on every launch: after a tile launch of the library the kernel may start
    // as the previous grid drains (it waits or not as a.overlap says); after any other node it is an ordinary
    // dependency, since the kernel then waits before touching global memory.
    const TileAccess acc = tile_access<S, kLayout, kParam, kRobot>(a);
    std::lock_guard<std::mutex> lk(g_last_tile_mu);
    const CaptureState before = capture_state(stream);
    auto it = g_last_tile.find(stream);
    a.overlap = may_start_early(it == g_last_tile.end() ? nullptr : &it->second, before, acc) ? 1 : 0;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(C::kThreads);
    cfg.dynamicSmemBytes = TLn::smem();
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t err = cudaLaunchKernelEx(&cfg, TLn::kernel(), a);
    const CaptureState after = err == cudaSuccess && before.capturing ? capture_state(stream) : CaptureState{};
    if (after.capturing && after.only_dep) g_last_tile[stream] = LastTile{after.id, after.only_dep, acc};
    else if (it != g_last_tile.end()) g_last_tile.erase(it);
    CUDA_TRY(err);
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    e->last_ctas_per_sm = cps;
    e->last_overlap = a.overlap;
    return H2O_OK;
}

// Wave-slope submersion is in effect: the mode is on and there is a wave field to take the slope of.
static bool slope_on(const h2o_engine* e) { return e->wave_slope && e->n_waves; }
// Fluid-inertia loads are in effect: the mode is on and something accelerates the water (a wave field, or a grid with
// more than one frame).  Otherwise the instantiations without the mode run, so that results stay bit-identical.
static bool inertia_on(const h2o_engine* e) { return e->fluid_inertia && clock_runs(e); }

template <typename S, int kLayout, int kParam, bool kStats>
static int launch_direct(h2o_engine* e, const StepArgs& a, long long body_begin, cudaStream_t stream)
{
    const long long cnt = a.n - body_begin;
    if (cnt <= 0) return H2O_OK;
    const int grid = int((cnt + 255) / 256);
    const WaveArgs wv = wave_args(e);
    const EnvArgs ev = env_args(e);
    const GridArgs gv = e->grid;
    const size_t smem = wave_smem_bytes(wv.n);
    if (e->dry_run) {
        e->launches += 1;
        return H2O_OK;
    }
    forget_last_tile(stream);
    if (inertia_on(e)) {
        if (slope_on(e))
            step_direct_kernel<S, kLayout, kParam, kStats, true, true><<<grid, 256, smem, stream>>>(a, body_begin, wv, ev, gv);
        else
            step_direct_kernel<S, kLayout, kParam, kStats, false, true><<<grid, 256, smem, stream>>>(a, body_begin, wv, ev, gv);
    } else if (slope_on(e)) {
        step_direct_kernel<S, kLayout, kParam, kStats, true><<<grid, 256, smem, stream>>>(a, body_begin, wv, ev, gv);
    } else {
        step_direct_kernel<S, kLayout, kParam, kStats><<<grid, 256, smem, stream>>>(a, body_begin, wv, ev, gv);
    }
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    return H2O_OK;
}

template <typename S, int kLayout>
static int launch_robot_wrench(h2o_engine* e, const StepArgs& a, long long robot_begin, cudaStream_t stream)
{
    const long long n_robots = a.robot_offsets ? a.n_robots_var : a.n / a.bodies_per_robot;
    const long long cnt = n_robots - robot_begin;
    if (cnt <= 0) return H2O_OK;
    const int grid = int((cnt * 32 + 255) / 256);
    if (e->dry_run) {
        e->launches += 1;
        return H2O_OK;
    }
    forget_last_tile(stream);
    robot_wrench_kernel<S, kLayout><<<grid, 256, 0, stream>>>(a, robot_begin);
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    return H2O_OK;
}

template <typename S, int kLayout, int kParam, bool kStats>
static int step_typed2(h2o_engine* e, StepArgs& a, cudaStream_t stream)
{
    using DC = typename DefaultCfg<S>::type;
    const bool robots = a.bodies_per_robot > 0 && a.out_wrench != nullptr;
    const int TB = robots ? tile_bodies_for(RobotCfgs<S>::C::kThreads, sizeof(S), a.bodies_per_robot)
                          : tile_bodies_for(DC::kThreads, sizeof(S), 0);
    // defensive only: every public entry point already rejects tensors that are not 16-byte aligned
    // (check_ptrs / dl_check), so this guards internal callers that slice buffers (h2o_step_host)
    bool ptr_ok = aligned16(a.pos) && aligned16(a.lin) && aligned16(a.prev) && aligned16(a.out_force) &&
                  aligned16(a.out_torque) && (kLayout == LAYOUT_PHYSX || aligned16(a.quat)) &&
                  (kLayout != LAYOUT_SPLIT || aligned16(a.ang)) &&
                  (kParam == PARAM_TABLE || aligned16(a.coeff));
    bool use_tile = false;
    if (e->kernel_choice == H2O_KERNEL_TILE) use_tile = true;
    else if (e->kernel_choice == H2O_KERNEL_AUTO) use_tile = a.n >= (long long)e->sm_count * 256;
    if (TB == 0 || !ptr_ok || a.n < TB) use_tile = false;
    if (a.am_dense || a.surface_eta || e->n_waves || e->env_cond || e->grid.vals || a.warp_compat)
        use_tile = false;  // f3 / f4 modes: direct kernel (+ robot_wrench_kernel)

    long long done_bodies = 0;
    if (use_tile) {
        int rc;
        constexpr bool kTunable = sizeof(S) == 4 && kLayout == LAYOUT_SPLIT && kParam == PARAM_PER_BODY && !kStats;
        bool launched = false;
        if constexpr (kTunable) {
          if (!robots && e->tile_cfg != 0) {
            // tuning variants (h2o_set_tile_config), fp32 / split layout / per-body records only
            launched = true;
            switch (e->tile_cfg) {
#define H2O_CFG(ID, T, I, O, MB) \
    case ID: rc = launch_tile<S, kLayout, kParam, false, kStats, Cfg<T, I, O, MB>>(e, a, stream); break;
                H2O_CFG(1, 256, 2, 2, 2)
                H2O_CFG(2, 256, 1, 2, 3)
                H2O_CFG(3, 128, 2, 2, 5)
                H2O_CFG(4, 128, 1, 2, 6)
                H2O_CFG(5, 128, 1, 2, 7)
                H2O_CFG(6, 128, 1, 2, 8)
                H2O_CFG(7, 64, 1, 2, 12)
                H2O_CFG(8, 64, 2, 2, 12)
                H2O_CFG(9, 96, 1, 2, 9)
#undef H2O_CFG
                case 10: rc = launch_tile<S, kLayout, kParam, false, kStats, Cfg<128, 1, 2, 6, true>>(e, a, stream); break;
                case 11: rc = launch_tile<S, kLayout, kParam, false, kStats, Cfg<256, 2, 2, 2, true>>(e, a, stream); break;
                default: return fail(H2O_ERR_BAD_ARGUMENT, "unknown tile config %d", e->tile_cfg);
            }
          }
        }
        if (!launched) {
            if (!robots) {
                rc = launch_tile<S, kLayout, kParam, false, kStats, DC>(e, a, stream);
            } else {
                using RC = RobotCfgs<S>;
                const int bpr = a.bodies_per_robot;
                const double ua = double(tile_bodies_for(RC::A::kThreads, sizeof(S), bpr)) / RC::A::kThreads;
                const double ub = double(tile_bodies_for(RC::B::kThreads, sizeof(S), bpr)) / RC::B::kThreads;
                const double uc = double(tile_bodies_for(RC::C::kThreads, sizeof(S), bpr)) / RC::C::kThreads;
                int pick = (ua >= ub - 0.03 && ua >= uc - 0.06) ? 0 : (ub >= uc - 0.03 ? 1 : 2);
                if (e->robot_cfg >= 0) pick = e->robot_cfg;
                if (bpr == HEXAPOD_BODIES && e->robot_cfg < 0)
                    rc = launch_tile<S, kLayout, kParam, true, kStats, typename RC::Hexapod>(e, a, stream);
                else if (pick == 0) rc = launch_tile<S, kLayout, kParam, true, kStats, typename RC::A>(e, a, stream);
                else if (pick == 1) rc = launch_tile<S, kLayout, kParam, true, kStats, typename RC::B>(e, a, stream);
                else rc = launch_tile<S, kLayout, kParam, true, kStats, typename RC::C>(e, a, stream);
            }
        }
        if (rc) return rc;
        done_bodies = (long long)a.n_tiles * a.tile_bodies;
        e->last_kernel = H2O_KERNEL_TILE;
    } else {
        e->last_kernel = H2O_KERNEL_DIRECT;
    }
    if (done_bodies < a.n) {
        int rc = launch_direct<S, kLayout, kParam, kStats>(e, a, done_bodies, stream);
        if (rc) return rc;
        if (robots) {
            rc = launch_robot_wrench<S, kLayout>(e, a, done_bodies / a.bodies_per_robot, stream);
            if (rc) return rc;
        }
    }
    if (a.out_wrench && a.robot_offsets) {  // unequal robots: every wrench from the written force / torque arrays
        int rc = launch_robot_wrench<S, kLayout>(e, a, 0, stream);
        if (rc) return rc;
    }
    return H2O_OK;
}

template <typename S>
static int step_typed(h2o_engine* e, int layout, StepArgs& a, cudaStream_t stream)
{
    const bool st = e->stats_on;
#define H2O_DISPATCH(LAY, PAR)                                                      \
    return st ? step_typed2<S, LAY, PAR, true>(e, a, stream) : step_typed2<S, LAY, PAR, false>(e, a, stream)
    if (layout == LAYOUT_SPLIT) {
        if (e->param_mode == PARAM_TABLE) { H2O_DISPATCH(LAYOUT_SPLIT, PARAM_TABLE); }
        else { H2O_DISPATCH(LAYOUT_SPLIT, PARAM_PER_BODY); }
    } else if (layout == LAYOUT_PHYSX) {
        if (e->param_mode == PARAM_TABLE) { H2O_DISPATCH(LAYOUT_PHYSX, PARAM_TABLE); }
        else { H2O_DISPATCH(LAYOUT_PHYSX, PARAM_PER_BODY); }
    } else {
        if (e->param_mode == PARAM_TABLE) { H2O_DISPATCH(LAYOUT_VIEW, PARAM_TABLE); }
        else { H2O_DISPATCH(LAYOUT_VIEW, PARAM_PER_BODY); }
    }
#undef H2O_DISPATCH
}

// With a wave field or a time-varying grid: the clock advances by dt, n times, after the work already in `stream` (counted as a launch).
static int advance_clock(h2o_engine* e, double dt, int n, cudaStream_t stream)
{
    if (e->dry_run) {
        e->launches += 1;
        return H2O_OK;
    }
    forget_last_tile(stream);
    advance_clock_kernel<<<1, 1, 0, stream>>>(e->wave_clock, dt, n);
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    return H2O_OK;
}

// Core step on device pointers (no validation beyond configuration).  tick: advance the water clock after the
// step's kernels (the chunked host pipeline advances it once after all chunks instead).
static int step_device(h2o_engine* e, int layout, const void* pos, const void* quat, const void* lin,
                       const void* ang, double dt, void* f, void* t, void* w, long long n,
                       long long first_body, void* prev, const void* coeff_base, cudaStream_t stream,
                       bool tick = true)
{
    if (e->param_mode < 0) return fail(H2O_ERR_NOT_CONFIGURED, "no parameters set (h2o_set_params_*)");
    if (!(dt > 1e-6)) return H2O_OK;  // hydrodynamics_behavior.py:139
    if (w && e->bodies_per_robot <= 0 && !e->robot_offsets)
        return fail(H2O_ERR_NOT_CONFIGURED, "robot wrench requested but h2o_set_articulation not called");
    if (w && e->robot_offsets && (n != e->n || first_body != 0))
        return fail(H2O_ERR_NOT_CONFIGURED, "unequal robots (h2o_set_articulation_offsets) need whole-batch launches");
    if (w && !e->robot_offsets && (n % e->bodies_per_robot) != 0)
        return fail(H2O_ERR_BAD_SHAPE, "n_bodies %lld is not a multiple of bodies_per_robot %d", n,
                    e->bodies_per_robot);
    StepArgs a;
    memset(&a, 0, sizeof a);
    a.pos = pos; a.quat = quat; a.lin = lin; a.ang = ang;
    a.prev = prev;
    a.coeff = coeff_base;
    a.slot_type = e->slot_type;
    a.out_force = f; a.out_torque = t; a.out_wrench = w;
    a.stats = e->stats_on ? e->stats : nullptr;
    a.n = n;
    a.first_body = first_body;
    a.n_slots = e->n_slots; a.n_types = e->n_types;
    a.bodies_per_robot = e->bodies_per_robot;
    a.quat_wxyz = e->quat_order == H2O_QUAT_WXYZ;
    a.rho = e->rho; a.grav = e->grav; a.inv_dt = 1.0 / dt;
    for (int k = 0; k < 3; ++k) a.current[k] = e->current[k];
    a.surface_z = e->surface_z;
    a.am_dense = e->am_dense; a.am_slot_type = e->am_slot_type; a.am_n_slots = e->am_slots;
    a.robot_offsets = e->robot_offsets; a.n_robots_var = e->n_robots_var;
    a.no_fallback = e->no_fallback;
    a.warp_compat = e->warp_compat;
    a.redo_bitmap = e->redo_bitmap;
    e->last_overlap = 0;
    a.surface_eta = e->surface_eta ? static_cast<const char*>(e->surface_eta) + size_t(first_body) * e->esz : nullptr;
    const int rc = e->dtype == H2O_F32 ? step_typed<float>(e, layout, a, stream) : step_typed<double>(e, layout, a, stream);
    if (rc || !clock_runs(e) || !tick) return rc;
    return advance_clock(e, dt, 1, stream);
}

static const void* coeff_at(h2o_engine* e, long long first_body)
{
    if (e->param_mode == PARAM_PER_BODY)
        return static_cast<const char*>(e->coeff) + size_t(first_body) * N_COEFF * e->esz;
    return e->coeff;
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
extern "C" {

const char* h2o_last_error(void) { return g_last_error.c_str(); }
const char* h2o_version(void) { return "h2o_b200 0.1.0 (sm_100a)"; }

int h2o_device_count(void)
{
    int n = 0;
    cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return -fail(H2O_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(err));
    }
    return n;
}

int h2o_create(h2o_handle* out, int64_t n_bodies, int dtype, int device)
{
    if (!out) return fail(H2O_ERR_BAD_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (n_bodies <= 0) return fail(H2O_ERR_BAD_ARGUMENT, "n_bodies must be positive (got %lld)", (long long)n_bodies);
    if (dtype != H2O_F32 && dtype != H2O_F64) return fail(H2O_ERR_BAD_DTYPE, "dtype must be H2O_F32 or H2O_F64");
    int ndev = 0;
    cudaError_t err = cudaGetDeviceCount(&ndev);
    if (err != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(H2O_ERR_NO_DEVICE, "no CUDA device available (%s); this engine has no CPU path",
                    err == cudaSuccess ? "0 devices" : cudaGetErrorString(err));
    }
    if (device < 0 || device >= ndev) return fail(H2O_ERR_BAD_DEVICE, "device %d out of range [0,%d)", device, ndev);
    DeviceGuard g(device);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(H2O_ERR_BAD_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    h2o_engine* e = new h2o_engine();
    e->device = device;
    e->dtype = dtype;
    e->n = n_bodies;
    e->esz = dtype == H2O_F32 ? 4 : 8;
    e->sm_count = prop.multiProcessorCount;
    if (const char* v = getenv("H2O_MAX_CTAS_PER_SM")) e->max_ctas_per_sm = atoi(v);
    if (const char* v = getenv("H2O_NO_FALLBACK")) e->no_fallback = std::max(0, atoi(v));
    if (const char* v = getenv("H2O_ROBOT_CFG")) e->robot_cfg = std::max(-1, std::min(2, atoi(v)));
    const size_t bitmap_bytes = (size_t(n_bodies) / 32 + 2) * sizeof(uint32_t);
    if (cudaMalloc(&e->prev, size_t(n_bodies) * 6 * e->esz) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&e->stats), N_STATS * sizeof(double)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&e->redo_bitmap), bitmap_bytes) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&e->wave_tab), MAX_WAVE_COMPONENTS * WAVE_STRIDE * sizeof(double)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&e->wave_clock), sizeof(double)) != cudaSuccess ||
        cudaMemset(e->wave_clock, 0, sizeof(double)) != cudaSuccess ||
        cudaMemset(e->redo_bitmap, 0, bitmap_bytes) != cudaSuccess ||
        cudaMemset(e->prev, 0, size_t(n_bodies) * 6 * e->esz) != cudaSuccess ||
        cudaMemset(e->stats, 0, N_STATS * sizeof(double)) != cudaSuccess) {
        const cudaError_t why = cudaGetLastError();
        if (e->prev) cudaFree(e->prev);
        if (e->stats) cudaFree(e->stats);
        if (e->redo_bitmap) cudaFree(e->redo_bitmap);
        if (e->wave_tab) cudaFree(e->wave_tab);
        if (e->wave_clock) cudaFree(e->wave_clock);
        delete e;
        return fail(H2O_ERR_CUDA, "allocating the engine state for %lld bodies failed: %s", (long long)n_bodies,
                    cudaGetErrorString(why));
    }
    *out = e;
    return H2O_OK;
}

int h2o_destroy(h2o_handle h)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    DeviceGuard g(e->device);
    if (e->graph_exec) cudaGraphExecDestroy(e->graph_exec);
    if (e->graph) cudaGraphDestroy(e->graph);
    for (int i = 0; i < 7; ++i) {
        if (e->hp_dev[i]) cudaFree(e->hp_dev[i]);
        if (e->hp_pin[i]) cudaFreeHost(e->hp_pin[i]);
    }
    for (int i = 0; i < HOST_PIPE_STREAMS; ++i)
        if (e->hp_stream[i]) cudaStreamDestroy(e->hp_stream[i]);
    if (e->hp_event) cudaEventDestroy(e->hp_event);
    if (e->capture_stream) cudaStreamDestroy(e->capture_stream);
    if (e->coeff) cudaFree(e->coeff);
    if (e->slot_type) cudaFree(e->slot_type);
    if (e->am_dense) cudaFree(e->am_dense);
    if (e->am_slot_type) cudaFree(e->am_slot_type);
    if (e->robot_offsets) cudaFree(e->robot_offsets);
    if (e->prev) cudaFree(e->prev);
    if (e->stats) cudaFree(e->stats);
    if (e->redo_bitmap) cudaFree(e->redo_bitmap);
    if (e->wave_tab) cudaFree(e->wave_tab);
    if (e->wave_clock) cudaFree(e->wave_clock);
    e->magic = 0;
    delete e;
    return H2O_OK;
}

int h2o_set_globals(h2o_handle h, double water_density, double gravity)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->rho = water_density;
    e->grav = gravity;
    return H2O_OK;
}

int h2o_set_environment(h2o_handle h, const double current_xyz[3], double surface_z)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    for (int k = 0; k < 3; ++k) e->current[k] = current_xyz ? current_xyz[k] : 0.0;
    e->surface_z = surface_z;
    return H2O_OK;
}

int h2o_set_surface_heights(h2o_handle h, const void* eta_dev)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->surface_eta = eta_dev;
    return H2O_OK;
}

int h2o_set_wave_field(h2o_handle h, int n_components, const double* comps, double depth)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    if (n_components == 0) {
        e->n_waves = 0;
        return H2O_OK;
    }
    if (n_components < 0 || n_components > MAX_WAVE_COMPONENTS)
        return fail(H2O_ERR_BAD_ARGUMENT, "n_components %d out of range [0,%d]", n_components, MAX_WAVE_COMPONENTS);
    if (!comps) return fail(H2O_ERR_BAD_ARGUMENT, "comps is NULL");
    if (!(depth > 0.0))  // also refuses NaN and -inf; +inf = deep water
        return fail(H2O_ERR_BAD_ARGUMENT, "depth must be > 0 (+inf = deep water), got %g", depth);
    std::vector<double> tab(size_t(n_components) * WAVE_STRIDE);
    for (int j = 0; j < n_components; ++j) {
        const double* c = comps + 5 * j;
        for (int k = 0; k < 5; ++k)
            if (!std::isfinite(c[k])) return fail(H2O_ERR_BAD_ARGUMENT, "component %d: non-finite value", j);
        if (c[0] < 0.0) return fail(H2O_ERR_BAD_ARGUMENT, "component %d: amplitude %g < 0", j, c[0]);
        if (c[1] == 0.0 && c[2] == 0.0) return fail(H2O_ERR_BAD_ARGUMENT, "component %d: wave vector is zero", j);
        if (!(c[3] > 0.0)) return fail(H2O_ERR_BAD_ARGUMENT, "component %d: omega %g <= 0", j, c[3]);
        wave_table_row(c, depth, tab.data() + size_t(j) * WAVE_STRIDE);
    }
    DeviceGuard g(e->device);
    e->n_waves = 0;  // no field until the upload below succeeds
    CUDA_TRY(cudaMemcpy(e->wave_tab, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice));
    e->n_waves = n_components;
    e->wave_depth = depth;
    return H2O_OK;
}

int h2o_set_wave_slope(h2o_handle h, int enable)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->wave_slope = enable != 0;
    return H2O_OK;
}

int h2o_set_fluid_inertia(h2o_handle h, int enable)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (enable && e->warp_compat)  // checked before the captured rollout is dropped: a refused call leaves it intact
        return fail(H2O_ERR_NOT_CONFIGURED,
                    "fluid-inertia loads follow the Numba semantics: turn Warp compatibility off first");
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->fluid_inertia = enable != 0;
    return H2O_OK;
}

int h2o_wave_time_write(h2o_handle h, double t, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!std::isfinite(t)) return fail(H2O_ERR_BAD_ARGUMENT, "wave time must be finite");
    DeviceGuard g(e->device);
    forget_last_tile(static_cast<cudaStream_t>(stream));
    set_clock_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(e->wave_clock, t);
    CUDA_TRY(cudaGetLastError());
    return H2O_OK;
}

int h2o_wave_time_read(h2o_handle h, double* t, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!t) return fail(H2O_ERR_BAD_ARGUMENT, "t is NULL");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaMemcpyAsync(t, e->wave_clock, sizeof(double), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return H2O_OK;
}

int h2o_wave_sample(h2o_handle h, const void* points, int64_t m, double* out, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (m < 0) return fail(H2O_ERR_BAD_ARGUMENT, "m must be >= 0");
    if (m == 0) return H2O_OK;
    if (!points || !out) return fail(H2O_ERR_BAD_ARGUMENT, "NULL points / out");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int grid = int((m + 255) / 256);
    const size_t smem = (size_t(e->n_waves) * WAVE_STRIDE + 1) * sizeof(double);
    if (e->dtype == H2O_F32)
        wave_sample_kernel<float><<<grid, 256, smem, s>>>(wave_args(e), e->surface_z, static_cast<const float*>(points), m, out);
    else
        wave_sample_kernel<double><<<grid, 256, smem, s>>>(wave_args(e), e->surface_z, static_cast<const double*>(points), m,
                                                           out);
    CUDA_TRY(cudaGetLastError());
    return H2O_OK;
}

int h2o_set_env_conditions(h2o_handle h, int64_t bodies_per_env, const double* cond_dev)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const bool remove = bodies_per_env == 0 || !cond_dev;
    if (!remove) {  // every check before the captured rollout is dropped: a refused call leaves it intact
        if (bodies_per_env < 0) return fail(H2O_ERR_BAD_ARGUMENT, "bodies_per_env must be >= 0");
        if (e->n % bodies_per_env != 0)
            return fail(H2O_ERR_BAD_SHAPE, "bodies_per_env %lld does not divide n_bodies %lld", (long long)bodies_per_env,
                        (long long)e->n);
        if (reinterpret_cast<uintptr_t>(cond_dev) & 7u) return fail(H2O_ERR_ALIGNMENT, "cond is not 8-byte aligned");
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, cond_dev) != cudaSuccess) {
            cudaGetLastError();
            return fail(H2O_ERR_BAD_DEVICE, "cond is not a CUDA pointer");
        }
        if ((attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) || attr.device != e->device)
            return fail(H2O_ERR_BAD_DEVICE, "cond must be device memory on device %d", e->device);
    }
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->env_cond = remove ? nullptr : cond_dev;
    e->bodies_per_env = remove ? 0 : bodies_per_env;
    return H2O_OK;
}

int h2o_reset_envs(h2o_handle h, const uint8_t* env_mask_dev, int restart_waves, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!e->env_cond) return fail(H2O_ERR_NOT_CONFIGURED, "no env conditions set (h2o_set_env_conditions)");
    if (!env_mask_dev) return fail(H2O_ERR_BAD_ARGUMENT, "env_mask is NULL");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int grid = int((e->n + 255) / 256);
    // the borrowed array is the caller's writable tensor; only restart_waves writes to it (column ENV_TAU)
    double* cond = const_cast<double*>(e->env_cond);
    if (e->dtype == H2O_F32)
        reset_envs_kernel<float><<<grid, 256, 0, s>>>(static_cast<float*>(e->prev), e->n, cond, e->bodies_per_env,
                                                      env_mask_dev, restart_waves != 0, e->wave_clock);
    else
        reset_envs_kernel<double><<<grid, 256, 0, s>>>(static_cast<double*>(e->prev), e->n, cond, e->bodies_per_env,
                                                       env_mask_dev, restart_waves != 0, e->wave_clock);
    CUDA_TRY(cudaGetLastError());
    return H2O_OK;
}

int h2o_wave_sample_env(h2o_handle h, const void* points, const int32_t* env_index, int64_t m, double* out,
                        h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!e->env_cond) return fail(H2O_ERR_NOT_CONFIGURED, "no env conditions set (h2o_set_env_conditions)");
    if (m < 0) return fail(H2O_ERR_BAD_ARGUMENT, "m must be >= 0");
    if (m == 0) return H2O_OK;
    if (!points || !env_index || !out) return fail(H2O_ERR_BAD_ARGUMENT, "NULL points / env_index / out");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int grid = int((m + 255) / 256);
    const size_t smem = (size_t(e->n_waves) * WAVE_STRIDE + 1) * sizeof(double);
    const long long n_envs = e->n / e->bodies_per_env;
    if (e->dtype == H2O_F32)
        wave_sample_env_kernel<float><<<grid, 256, smem, s>>>(wave_args(e), env_args(e), n_envs, e->surface_z,
                                                              static_cast<const float*>(points), env_index, m, out);
    else
        wave_sample_env_kernel<double><<<grid, 256, smem, s>>>(wave_args(e), env_args(e), n_envs, e->surface_z,
                                                               static_cast<const double*>(points), env_index, m, out);
    CUDA_TRY(cudaGetLastError());
    return H2O_OK;
}

int h2o_set_current_grid(h2o_handle h, const double* grid_dev, const int64_t dims[4], const double geom[8])
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    GridArgs g{};
    if (grid_dev) {  // every check before the captured rollout is dropped: a refused call leaves it intact
        if (!dims || !geom) return fail(H2O_ERR_BAD_ARGUMENT, "NULL dims / geom");
        int64_t total = 3 * int64_t(sizeof(double));
        for (int k = 0; k < 4; ++k) {
            if (dims[k] < 1) return fail(H2O_ERR_BAD_ARGUMENT, "dims[%d] = %lld < 1", k, (long long)dims[k]);
            if (__builtin_mul_overflow(total, dims[k], &total))
                return fail(H2O_ERR_BAD_ARGUMENT, "grid of %lld x %lld x %lld x %lld x 3 doubles is too large",
                            (long long)dims[0], (long long)dims[1], (long long)dims[2], (long long)dims[3]);
        }
        for (int k = 0; k < 8; ++k)
            if (!std::isfinite(geom[k])) return fail(H2O_ERR_BAD_ARGUMENT, "geom[%d] is not finite", k);
        if (!(geom[3] > 0.0 && geom[4] > 0.0 && geom[5] > 0.0))
            return fail(H2O_ERR_BAD_ARGUMENT, "spacings hx, hy, hz must be > 0");
        if (dims[0] > 1 && !(geom[7] > 0.0)) return fail(H2O_ERR_BAD_ARGUMENT, "frame interval ht must be > 0 when nt > 1");
        if (reinterpret_cast<uintptr_t>(grid_dev) & 7u) return fail(H2O_ERR_ALIGNMENT, "grid is not 8-byte aligned");
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, grid_dev) != cudaSuccess) {
            cudaGetLastError();
            return fail(H2O_ERR_BAD_DEVICE, "grid is not a CUDA pointer");
        }
        if ((attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) || attr.device != e->device)
            return fail(H2O_ERR_BAD_DEVICE, "grid must be device memory on device %d", e->device);
        g.vals = grid_dev;
        g.nt = dims[0]; g.nz = dims[1]; g.ny = dims[2]; g.nx = dims[3];
        g.gx = geom[0]; g.gy = geom[1]; g.gz = geom[2];
        g.hx = geom[3]; g.hy = geom[4]; g.hz = geom[5];
        g.t0 = geom[6]; g.ht = geom[7];
    }
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->grid = g;
    return H2O_OK;
}

int h2o_water_sample(h2o_handle h, const void* points, const int32_t* env_index, int64_t m, double* out,
                     h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (env_index && !e->env_cond) return fail(H2O_ERR_NOT_CONFIGURED, "no env conditions set (h2o_set_env_conditions)");
    if (m < 0) return fail(H2O_ERR_BAD_ARGUMENT, "m must be >= 0");
    if (m == 0) return H2O_OK;
    if (!points || !out) return fail(H2O_ERR_BAD_ARGUMENT, "NULL points / out");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int grid = int((m + 255) / 256);
    const size_t smem = (size_t(e->n_waves) * WAVE_STRIDE + 1) * sizeof(double);
    const long long n_envs = e->env_cond ? e->n / e->bodies_per_env : 0;
    const double* c = e->current;
    if (e->dtype == H2O_F32)
        water_sample_kernel<float><<<grid, 256, smem, s>>>(wave_args(e), env_args(e), e->grid, n_envs, c[0], c[1],
                                                           c[2], e->surface_z, static_cast<const float*>(points),
                                                           env_index, m, out);
    else
        water_sample_kernel<double><<<grid, 256, smem, s>>>(wave_args(e), env_args(e), e->grid, n_envs, c[0], c[1],
                                                            c[2], e->surface_z, static_cast<const double*>(points),
                                                            env_index, m, out);
    CUDA_TRY(cudaGetLastError());
    return H2O_OK;
}

int h2o_water_slope_sample(h2o_handle h, const void* points, const int32_t* env_index, int64_t m, double* out,
                           h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (env_index && !e->env_cond) return fail(H2O_ERR_NOT_CONFIGURED, "no env conditions set (h2o_set_env_conditions)");
    if (m < 0) return fail(H2O_ERR_BAD_ARGUMENT, "m must be >= 0");
    if (m == 0) return H2O_OK;
    if (!points || !out) return fail(H2O_ERR_BAD_ARGUMENT, "NULL points / out");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int grid = int((m + 255) / 256);
    // the slope a step uses: none unless the mode is on and there is a wave field
    WaveArgs wv = wave_args(e);
    if (!slope_on(e)) wv.n = 0;
    const size_t smem = (size_t(wv.n) * WAVE_STRIDE + 1) * sizeof(double);
    const long long n_envs = e->env_cond ? e->n / e->bodies_per_env : 0;
    if (e->dtype == H2O_F32)
        water_slope_sample_kernel<float><<<grid, 256, smem, s>>>(wv, env_args(e), n_envs, e->surface_z,
                                                                 static_cast<const float*>(points), env_index, m, out);
    else
        water_slope_sample_kernel<double><<<grid, 256, smem, s>>>(wv, env_args(e), n_envs, e->surface_z,
                                                                  static_cast<const double*>(points), env_index, m, out);
    CUDA_TRY(cudaGetLastError());
    return H2O_OK;
}

int h2o_fluid_accel_sample(h2o_handle h, const void* points, const int32_t* env_index, int64_t m, double* out,
                           h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (env_index && !e->env_cond) return fail(H2O_ERR_NOT_CONFIGURED, "no env conditions set (h2o_set_env_conditions)");
    if (m < 0) return fail(H2O_ERR_BAD_ARGUMENT, "m must be >= 0");
    if (m == 0) return H2O_OK;
    if (!points || !out) return fail(H2O_ERR_BAD_ARGUMENT, "NULL points / out");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int grid = int((m + 255) / 256);
    // the a_f a step uses: none unless the mode is in effect
    WaveArgs wv = wave_args(e);
    GridArgs gv = e->grid;
    if (!inertia_on(e)) {
        wv.n = 0;
        gv.vals = nullptr;
    }
    const size_t smem = (size_t(wv.n) * WAVE_STRIDE + 1) * sizeof(double);
    const long long n_envs = e->env_cond ? e->n / e->bodies_per_env : 0;
    if (e->dtype == H2O_F32)
        fluid_accel_sample_kernel<float><<<grid, 256, smem, s>>>(wv, env_args(e), gv, n_envs, e->surface_z,
                                                                 static_cast<const float*>(points), env_index, m, out);
    else
        fluid_accel_sample_kernel<double><<<grid, 256, smem, s>>>(wv, env_args(e), gv, n_envs, e->surface_z,
                                                                  static_cast<const double*>(points), env_index, m, out);
    CUDA_TRY(cudaGetLastError());
    return H2O_OK;
}

int h2o_set_part_table(h2o_handle h, int n_types, const double* table_host, int n_slots,
                       const int32_t* slot_type_host)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    if (n_types < 1 || n_types > MAX_TABLE_TYPES)
        return fail(H2O_ERR_BAD_ARGUMENT, "n_types %d out of range [1,%d]", n_types, MAX_TABLE_TYPES);
    if (n_slots < 1 || n_slots > MAX_TABLE_SLOTS)
        return fail(H2O_ERR_BAD_ARGUMENT, "n_slots %d out of range [1,%d]", n_slots, MAX_TABLE_SLOTS);
    if (!table_host || !slot_type_host) return fail(H2O_ERR_BAD_ARGUMENT, "NULL table / slot_type");
    for (int i = 0; i < n_slots; ++i)
        if (slot_type_host[i] < 0 || slot_type_host[i] >= n_types)
            return fail(H2O_ERR_BAD_ARGUMENT, "slot_type[%d] = %d out of range", i, slot_type_host[i]);
    DeviceGuard g(e->device);
    if (e->coeff) { cudaFree(e->coeff); e->coeff = nullptr; }
    if (e->slot_type) { cudaFree(e->slot_type); e->slot_type = nullptr; }
    e->param_mode = -1;  // not configured until the uploads below succeed
    const size_t cnt = size_t(n_types) * N_COEFF;
    CUDA_TRY(cudaMalloc(&e->coeff, cnt * e->esz));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&e->slot_type), n_slots * sizeof(int32_t)));
    if (e->dtype == H2O_F32) {
        std::vector<float> tmp(cnt);
        for (size_t i = 0; i < cnt; ++i) tmp[i] = float(table_host[i]);
        CUDA_TRY(cudaMemcpy(e->coeff, tmp.data(), cnt * sizeof(float), cudaMemcpyHostToDevice));
    } else {
        CUDA_TRY(cudaMemcpy(e->coeff, table_host, cnt * sizeof(double), cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaMemcpy(e->slot_type, slot_type_host, n_slots * sizeof(int32_t), cudaMemcpyHostToDevice));
    e->param_mode = PARAM_TABLE;
    e->n_types = n_types;
    e->n_slots = n_slots;
    e->coeff_rows = n_types;
    return H2O_OK;
}

int h2o_set_added_mass_dense(h2o_handle h, int n_types, const double* matrices_host, int n_slots,
                             const int32_t* slot_type_host)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    DeviceGuard g(e->device);
    if (n_types == 0) {  // back to the wrapper's diagonal
        if (e->am_dense) { cudaFree(e->am_dense); e->am_dense = nullptr; }
        if (e->am_slot_type) { cudaFree(e->am_slot_type); e->am_slot_type = nullptr; }
        e->am_types = e->am_slots = 0;
        return H2O_OK;
    }
    if (n_types < 0 || n_types > MAX_TABLE_TYPES)
        return fail(H2O_ERR_BAD_ARGUMENT, "n_types %d out of range [0,%d]", n_types, MAX_TABLE_TYPES);
    if (!matrices_host) return fail(H2O_ERR_BAD_ARGUMENT, "matrices is NULL");
    const int32_t slot0 = 0;
    if (!slot_type_host) {
        if (n_types != 1) return fail(H2O_ERR_BAD_ARGUMENT, "slot_type is NULL with %d matrices", n_types);
        slot_type_host = &slot0;
        n_slots = 1;
    }
    if (n_slots < 1 || n_slots > MAX_TABLE_SLOTS)
        return fail(H2O_ERR_BAD_ARGUMENT, "n_slots %d out of range [1,%d]", n_slots, MAX_TABLE_SLOTS);
    for (int i = 0; i < n_slots; ++i)
        if (slot_type_host[i] < 0 || slot_type_host[i] >= n_types)
            return fail(H2O_ERR_BAD_ARGUMENT, "slot_type[%d] = %d out of range", i, slot_type_host[i]);
    if (e->am_dense) { cudaFree(e->am_dense); e->am_dense = nullptr; }
    if (e->am_slot_type) { cudaFree(e->am_slot_type); e->am_slot_type = nullptr; }
    e->am_types = e->am_slots = 0;
    const size_t cnt = size_t(n_types) * 36;
    CUDA_TRY(cudaMalloc(&e->am_dense, cnt * e->esz));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&e->am_slot_type), n_slots * sizeof(int32_t)));
    if (e->dtype == H2O_F32) {
        std::vector<float> tmp(cnt);
        for (size_t i = 0; i < cnt; ++i) tmp[i] = float(matrices_host[i]);
        CUDA_TRY(cudaMemcpy(e->am_dense, tmp.data(), cnt * sizeof(float), cudaMemcpyHostToDevice));
    } else {
        CUDA_TRY(cudaMemcpy(e->am_dense, matrices_host, cnt * sizeof(double), cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaMemcpy(e->am_slot_type, slot_type_host, n_slots * sizeof(int32_t), cudaMemcpyHostToDevice));
    e->am_types = n_types;
    e->am_slots = n_slots;
    return H2O_OK;
}

int h2o_set_params_uniform(h2o_handle h, const double c[12], double mass)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!c) return fail(H2O_ERR_BAD_ARGUMENT, "ctor12 is NULL");
    // ctor order (numba_hydrodynamics_wrapper.py:9-10) -> coefficient record order
    const double rec[N_COEFF] = {c[0], c[1], c[2], c[3], c[4], c[5], c[6], c[9], c[10], c[11], mass};
    const int32_t slot0 = 0;
    e->rho = c[7];
    e->grav = c[8];
    return h2o_set_part_table(h, 1, rec, 1, &slot0);
}

int h2o_set_params_per_body(h2o_handle h, const void* coeff, int src_dtype, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    if (!coeff) return fail(H2O_ERR_BAD_ARGUMENT, "coeff is NULL");
    if (src_dtype != H2O_F32 && src_dtype != H2O_F64) return fail(H2O_ERR_BAD_DTYPE, "bad src_dtype");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t cnt = size_t(e->n) * N_COEFF;
    if (e->param_mode != PARAM_PER_BODY) {
        if (e->coeff) { cudaFree(e->coeff); e->coeff = nullptr; }
        e->param_mode = -1;  // not configured until the upload below succeeds
        CUDA_TRY(cudaMalloc(&e->coeff, cnt * e->esz));
    }
    if (src_dtype == e->dtype) {
        CUDA_TRY(cudaMemcpyAsync(e->coeff, coeff, cnt * e->esz, cudaMemcpyDefault, s));
    } else {
        const size_t sesz = src_dtype == H2O_F32 ? 4 : 8;
        void* tmp = nullptr;
        CUDA_TRY(cudaMalloc(&tmp, cnt * sesz));
        cudaError_t err = cudaMemcpyAsync(tmp, coeff, cnt * sesz, cudaMemcpyDefault, s);
        if (err == cudaSuccess) {
            const int grid = int((cnt + 255) / 256);
            if (e->dtype == H2O_F32)
                cast_kernel<float, double><<<grid, 256, 0, s>>>(static_cast<float*>(e->coeff),
                                                                static_cast<const double*>(tmp), (long long)cnt);
            else
                cast_kernel<double, float><<<grid, 256, 0, s>>>(static_cast<double*>(e->coeff),
                                                                static_cast<const float*>(tmp), (long long)cnt);
            err = cudaGetLastError();
        }
        cudaStreamSynchronize(s);
        cudaFree(tmp);
        if (err != cudaSuccess) return fail(H2O_ERR_CUDA, "coefficient conversion failed: %s", cudaGetErrorString(err));
    }
    CUDA_TRY(cudaStreamSynchronize(s));
    e->param_mode = PARAM_PER_BODY;
    e->coeff_rows = e->n;
    e->n_slots = 1;
    e->n_types = 0;
    return H2O_OK;
}

int h2o_set_params_soa(h2o_handle h, const void* const cols[11], int src_dtype, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    if (!cols) return fail(H2O_ERR_BAD_ARGUMENT, "cols is NULL");
    if (src_dtype != H2O_F32 && src_dtype != H2O_F64) return fail(H2O_ERR_BAD_DTYPE, "bad src_dtype");
    DeviceGuard g(e->device);
    SoaCols sc;
    for (int k = 0; k < N_COEFF; ++k) {
        if (!cols[k]) return fail(H2O_ERR_BAD_ARGUMENT, "column %d is NULL", k);
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, cols[k]) != cudaSuccess ||
            (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)) {
            cudaGetLastError();
            return fail(H2O_ERR_BAD_DEVICE, "column %d is not device memory", k);
        }
        if (at.type == cudaMemoryTypeDevice && at.device != e->device)
            return fail(H2O_ERR_BAD_DEVICE, "column %d lives on device %d, handle on %d", k, at.device, e->device);
        sc.col[k] = cols[k];
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t cnt = size_t(e->n) * N_COEFF;
    if (e->param_mode != PARAM_PER_BODY) {
        if (e->coeff) { cudaFree(e->coeff); e->coeff = nullptr; }
        e->param_mode = -1;  // not configured until the upload below succeeds
        CUDA_TRY(cudaMalloc(&e->coeff, cnt * e->esz));
    }
    const int grid = int((e->n + 255) / 256);
    if (e->dtype == H2O_F32) {
        if (src_dtype == H2O_F32) soa_to_records_kernel<float, float><<<grid, 256, 0, s>>>(static_cast<float*>(e->coeff), sc, e->n);
        else soa_to_records_kernel<float, double><<<grid, 256, 0, s>>>(static_cast<float*>(e->coeff), sc, e->n);
    } else {
        if (src_dtype == H2O_F32) soa_to_records_kernel<double, float><<<grid, 256, 0, s>>>(static_cast<double*>(e->coeff), sc, e->n);
        else soa_to_records_kernel<double, double><<<grid, 256, 0, s>>>(static_cast<double*>(e->coeff), sc, e->n);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(s));
    e->param_mode = PARAM_PER_BODY;
    e->coeff_rows = e->n;
    e->n_slots = 1;
    e->n_types = 0;
    return H2O_OK;
}

int h2o_set_articulation(h2o_handle h, int bodies_per_robot)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    if (bodies_per_robot < 0) return fail(H2O_ERR_BAD_ARGUMENT, "bodies_per_robot must be >= 0");
    if (bodies_per_robot > 0 && e->n % bodies_per_robot != 0)
        return fail(H2O_ERR_BAD_SHAPE, "n_bodies %lld is not a multiple of bodies_per_robot %d", (long long)e->n,
                    bodies_per_robot);
    e->bodies_per_robot = bodies_per_robot;
    if (e->robot_offsets) {  // equal runs replace an earlier h2o_set_articulation_offsets
        DeviceGuard g(e->device);
        cudaFree(e->robot_offsets);
        e->robot_offsets = nullptr;
        e->n_robots_var = 0;
    }
    return H2O_OK;
}

int h2o_set_articulation_offsets(h2o_handle h, int64_t n_robots, const int64_t* offsets_host)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    if (n_robots < 1 || !offsets_host) return fail(H2O_ERR_BAD_ARGUMENT, "need n_robots >= 1 and offsets");
    if (offsets_host[0] != 0 || offsets_host[n_robots] != e->n)
        return fail(H2O_ERR_BAD_SHAPE, "offsets must start at 0 and end at n_bodies = %lld", (long long)e->n);
    for (int64_t r = 0; r < n_robots; ++r)
        if (offsets_host[r + 1] <= offsets_host[r])
            return fail(H2O_ERR_BAD_ARGUMENT, "offsets must increase strictly (robot %lld is empty)", (long long)r);
    DeviceGuard g(e->device);
    if (e->robot_offsets) { cudaFree(e->robot_offsets); e->robot_offsets = nullptr; }
    e->n_robots_var = 0;
    std::vector<long long> tmp(offsets_host, offsets_host + n_robots + 1);
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&e->robot_offsets), tmp.size() * sizeof(long long)));
    CUDA_TRY(cudaMemcpy(e->robot_offsets, tmp.data(), tmp.size() * sizeof(long long), cudaMemcpyHostToDevice));
    e->n_robots_var = n_robots;
    e->bodies_per_robot = 0;
    return H2O_OK;
}

int h2o_set_quat_order(h2o_handle h, int order)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    if (order != H2O_QUAT_XYZW && order != H2O_QUAT_WXYZ) return fail(H2O_ERR_BAD_ARGUMENT, "bad quaternion order");
    e->quat_order = order;
    return H2O_OK;
}

int h2o_set_kernel(h2o_handle h, int choice)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    if (choice < H2O_KERNEL_AUTO || choice > H2O_KERNEL_DIRECT) return fail(H2O_ERR_BAD_ARGUMENT, "bad kernel choice");
    e->kernel_choice = choice;
    return H2O_OK;
}

int h2o_set_strict(h2o_handle h, int enable)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->no_fallback = enable ? 0 : 1;
    return H2O_OK;
}

int h2o_set_warp_compat(h2o_handle h, int enable)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (enable && e->fluid_inertia)  // checked before the captured rollout is dropped: a refused call leaves it intact
        return fail(H2O_ERR_NOT_CONFIGURED,
                    "Warp compatibility has no fluid-inertia loads: turn h2o_set_fluid_inertia off first");
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->warp_compat = enable != 0;
    return H2O_OK;
}

int h2o_set_tile_config(h2o_handle h, int cfg)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    if (cfg < 0 || cfg > 11) return fail(H2O_ERR_BAD_ARGUMENT, "tile config must be in [0,11]");
    e->tile_cfg = cfg;
    return H2O_OK;
}

int h2o_enable_stats(h2o_handle h, int enable)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->stats_on = enable != 0;
    return H2O_OK;
}

int h2o_reset(h2o_handle h, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    DeviceGuard g(e->device);
    CUDA_TRY(cudaMemsetAsync(e->prev, 0, size_t(e->n) * 6 * e->esz, static_cast<cudaStream_t>(stream)));
    return H2O_OK;
}

int h2o_set_prev(h2o_handle h, const void* prev_lin, const void* prev_ang, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!prev_lin || !prev_ang) return fail(H2O_ERR_BAD_ARGUMENT, "NULL prev tensor");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int grid = int((e->n + 255) / 256);
    if (e->dtype == H2O_F32)
        pack_prev_kernel<float><<<grid, 256, 0, s>>>(static_cast<float*>(e->prev), static_cast<const float*>(prev_lin),
                                                     static_cast<const float*>(prev_ang), e->n);
    else
        pack_prev_kernel<double><<<grid, 256, 0, s>>>(static_cast<double*>(e->prev),
                                                      static_cast<const double*>(prev_lin),
                                                      static_cast<const double*>(prev_ang), e->n);
    CUDA_TRY(cudaGetLastError());
    return H2O_OK;
}

int h2o_get_prev(h2o_handle h, void* prev_lin, void* prev_ang, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!prev_lin || !prev_ang) return fail(H2O_ERR_BAD_ARGUMENT, "NULL prev tensor");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int grid = int((e->n + 255) / 256);
    if (e->dtype == H2O_F32)
        unpack_prev_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float*>(e->prev), static_cast<float*>(prev_lin),
                                                       static_cast<float*>(prev_ang), e->n);
    else
        unpack_prev_kernel<double><<<grid, 256, 0, s>>>(static_cast<const double*>(e->prev),
                                                        static_cast<double*>(prev_lin), static_cast<double*>(prev_ang),
                                                        e->n);
    CUDA_TRY(cudaGetLastError());
    return H2O_OK;
}

static int check_ptrs(const void* const* ptrs, int cnt)
{
    for (int i = 0; i < cnt; ++i) {
        if (!ptrs[i]) return fail(H2O_ERR_BAD_ARGUMENT, "NULL tensor pointer (argument %d)", i);
        if (!aligned16(ptrs[i])) return fail(H2O_ERR_ALIGNMENT, "tensor pointer %d is not 16-byte aligned", i);
    }
    return H2O_OK;
}

int h2o_step(h2o_handle h, const void* pos, const void* quat, const void* lin_vel, const void* ang_vel, double dt,
             void* out_force, void* out_torque, void* out_robot_wrench, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void* p[6] = {pos, quat, lin_vel, ang_vel, out_force, out_torque};
    if (int rc = check_ptrs(p, 6)) return rc;
    DeviceGuard g(e->device);
    return step_device(e, LAYOUT_SPLIT, pos, quat, lin_vel, ang_vel, dt, out_force, out_torque, out_robot_wrench,
                       e->n, 0, e->prev, coeff_at(e, 0), static_cast<cudaStream_t>(stream));
}

int h2o_step_physx(h2o_handle h, const void* transforms, const void* velocities, double dt, void* out_force,
                   void* out_torque, void* out_robot_wrench, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void* p[4] = {transforms, velocities, out_force, out_torque};
    if (int rc = check_ptrs(p, 4)) return rc;
    DeviceGuard g(e->device);
    return step_device(e, LAYOUT_PHYSX, transforms, nullptr, velocities, nullptr, dt, out_force, out_torque,
                       out_robot_wrench, e->n, 0, e->prev, coeff_at(e, 0), static_cast<cudaStream_t>(stream));
}

int h2o_step_view(h2o_handle h, const void* pos, const void* quat, const void* velocities, double dt,
                  void* out_force, void* out_torque, void* out_robot_wrench, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void* p[5] = {pos, quat, velocities, out_force, out_torque};
    if (int rc = check_ptrs(p, 5)) return rc;
    DeviceGuard g(e->device);
    return step_device(e, LAYOUT_VIEW, pos, quat, velocities, nullptr, dt, out_force, out_torque, out_robot_wrench,
                       e->n, 0, e->prev, coeff_at(e, 0), static_cast<cudaStream_t>(stream));
}

int h2o_bind(h2o_handle h, int layout, const void* pos, const void* quat, const void* lin_vel, const void* ang_vel,
             void* out_force, void* out_torque, void* out_robot_wrench)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (layout != LAYOUT_SPLIT && layout != LAYOUT_PHYSX && layout != LAYOUT_VIEW)
        return fail(H2O_ERR_BAD_ARGUMENT, "bad layout %d", layout);
    if (layout == LAYOUT_SPLIT) {
        const void* p[6] = {pos, quat, lin_vel, ang_vel, out_force, out_torque};
        if (int rc = check_ptrs(p, 6)) return rc;
    } else if (layout == LAYOUT_VIEW) {
        const void* p[5] = {pos, quat, lin_vel, out_force, out_torque};
        if (int rc = check_ptrs(p, 5)) return rc;
    } else {
        const void* p[4] = {pos, lin_vel, out_force, out_torque};
        if (int rc = check_ptrs(p, 4)) return rc;
    }
    DeviceGuard g(e->device);
    // bound tensors must live on the handle's device
    const void* all[7] = {pos, quat, lin_vel, ang_vel, out_force, out_torque, out_robot_wrench};
    for (int i = 0; i < 7; ++i) {
        if (!all[i]) continue;
        cudaPointerAttributes at;
        cudaError_t err = cudaPointerGetAttributes(&at, all[i]);
        if (err != cudaSuccess) {
            cudaGetLastError();
            return fail(H2O_ERR_BAD_DEVICE, "tensor %d: not a CUDA pointer", i);
        }
        if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)
            return fail(H2O_ERR_BAD_DEVICE, "tensor %d is not device memory", i);
        if (at.type == cudaMemoryTypeDevice && at.device != e->device)
            return fail(H2O_ERR_BAD_DEVICE, "tensor %d lives on device %d, handle on %d", i, at.device, e->device);
    }
    e->b_layout = layout;
    e->b_pos = pos; e->b_quat = quat; e->b_lin = lin_vel; e->b_ang = ang_vel;
    e->b_f = out_force; e->b_t = out_torque; e->b_w = out_robot_wrench;
    e->bound = true;
    invalidate_graph(e);
    return H2O_OK;
}

int h2o_unbind(h2o_handle h)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    e->bound = false;
    DeviceGuard g(e->device);
    invalidate_graph(e);
    return H2O_OK;
}

int h2o_step_bound(h2o_handle h, double dt, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!e->bound) return fail(H2O_ERR_NOT_CONFIGURED, "h2o_bind has not been called");
    DeviceGuard g(e->device);
    return step_device(e, e->b_layout, e->b_pos, e->b_quat, e->b_lin, e->b_ang, dt, e->b_f, e->b_t, e->b_w, e->n, 0,
                       e->prev, coeff_at(e, 0), static_cast<cudaStream_t>(stream));
}

static int integrate_device(h2o_engine* e, void* pos, void* quat, void* lin, void* ang, const void* f,
                            const void* t, double dt, double gravity, cudaStream_t s)
{
    if (e->param_mode < 0) return fail(H2O_ERR_NOT_CONFIGURED, "no parameters set (h2o_set_params_*)");
    FreeBodyArgs a;
    memset(&a, 0, sizeof a);
    a.pos = pos; a.quat = quat; a.lin = lin; a.ang = ang; a.force = f; a.torque = t;
    a.coeff = e->coeff; a.slot_type = e->slot_type;
    a.n = e->n; a.n_slots = e->n_slots; a.param_mode = e->param_mode;
    a.quat_wxyz = e->quat_order == H2O_QUAT_WXYZ;
    a.dt = dt; a.gravity = gravity;
    const int grid = int((e->n + 255) / 256);
    if (e->dry_run) {
        e->launches += 1;
        return H2O_OK;
    }
    forget_last_tile(s);
    if (e->dtype == H2O_F32) free_body_kernel<float><<<grid, 256, 0, s>>>(a);
    else free_body_kernel<double><<<grid, 256, 0, s>>>(a);
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    return H2O_OK;
}

int h2o_integrate_free_bodies(h2o_handle h, void* pos, void* quat, void* lin_vel, void* ang_vel, const void* force,
                              const void* torque, double dt, double gravity, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void* p[6] = {pos, quat, lin_vel, ang_vel, force, torque};
    if (int rc = check_ptrs(p, 6)) return rc;
    if (!(dt > 1e-6)) return H2O_OK;
    DeviceGuard g(e->device);
    return integrate_device(e, pos, quat, lin_vel, ang_vel, force, torque, dt, gravity, static_cast<cudaStream_t>(stream));
}

int h2o_set_rollout_mode(h2o_handle h, int free_bodies, double gravity)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    { DeviceGuard gi(e->device); invalidate_graph(e); }
    e->rollout_free_bodies = free_bodies != 0;
    e->rollout_gravity = gravity;
    return H2O_OK;
}

// one rollout step over the bound tensors: fused force step (+ free-body integration)
static int rollout_step(h2o_engine* e, double dt, cudaStream_t s)
{
    int rc = step_device(e, e->b_layout, e->b_pos, e->b_quat, e->b_lin, e->b_ang, dt, e->b_f, e->b_t, e->b_w, e->n, 0,
                         e->prev, coeff_at(e, 0), s);
    if (rc || !e->rollout_free_bodies) return rc;
    if (e->b_layout != LAYOUT_SPLIT)
        return fail(H2O_ERR_NOT_CONFIGURED, "free-body rollouts need the split layout (pos, quat, lin_vel, ang_vel)");
    return integrate_device(e, const_cast<void*>(e->b_pos), const_cast<void*>(e->b_quat), const_cast<void*>(e->b_lin),
                            const_cast<void*>(e->b_ang), e->b_f, e->b_t, dt, e->rollout_gravity, s);
}

int h2o_capture_rollout(h2o_handle h, int n_steps, double dt, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!e->bound) return fail(H2O_ERR_NOT_CONFIGURED, "h2o_bind has not been called");
    if (n_steps < 1) return fail(H2O_ERR_BAD_ARGUMENT, "n_steps must be >= 1");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    invalidate_graph(e);
    // One DRY step first: every per-kernel attribute / occupancy query happens outside capture and the
    // launches of one step are counted, but nothing is launched, so capturing does not advance the
    // carried velocities or (free-body mode) the bound state.  The capture itself runs on an
    // engine-owned stream: the caller's stream may be the legacy default stream, which cannot be captured.
    const int64_t before0 = e->launches;
    e->dry_run = true;
    int rc = rollout_step(e, dt, s);
    e->dry_run = false;
    const int64_t per_step = e->launches - before0;
    e->launches = before0;
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(s));  // order the capture stream after the caller's queued work
    if (!e->capture_stream) CUDA_TRY(cudaStreamCreateWithFlags(&e->capture_stream, cudaStreamNonBlocking));
    s = e->capture_stream;
    CUDA_TRY(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    for (int i = 0; i < n_steps && rc == H2O_OK; ++i) rc = rollout_step(e, dt, s);
    cudaGraph_t graph = nullptr;
    cudaError_t err = cudaStreamEndCapture(s, &graph);
    e->launches = before0;  // captured launches did not execute
    if (rc) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
    }
    if (err != cudaSuccess) return fail(H2O_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(err));
    e->graph = graph;
    CUDA_TRY(cudaGraphInstantiate(&e->graph_exec, e->graph, 0));
    e->graph_steps = n_steps;
    e->graph_launches_per_replay = per_step * n_steps;
    return H2O_OK;
}

int h2o_launch_rollout(h2o_handle h, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!e->graph_exec) return fail(H2O_ERR_NOT_CONFIGURED, "h2o_capture_rollout has not been called");
    DeviceGuard g(e->device);
    CUDA_TRY(cudaGraphLaunch(e->graph_exec, static_cast<cudaStream_t>(stream)));
    e->launches += e->graph_launches_per_replay;
    return H2O_OK;
}

int h2o_rollout_persistent(h2o_handle h, int n_steps, double dt, double gravity, int trace_every, void* trace_out,
                           h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!e->bound) return fail(H2O_ERR_NOT_CONFIGURED, "h2o_bind has not been called");
    if (e->b_layout != LAYOUT_SPLIT)
        return fail(H2O_ERR_NOT_CONFIGURED, "persistent rollouts need the split layout (pos, quat, lin_vel, ang_vel)");
    if (e->param_mode < 0) return fail(H2O_ERR_NOT_CONFIGURED, "no parameters set (h2o_set_params_*)");
    if (n_steps < 1) return fail(H2O_ERR_BAD_ARGUMENT, "n_steps must be >= 1");
    if (trace_every < 0 || (trace_every > 0 && !trace_out))
        return fail(H2O_ERR_BAD_ARGUMENT, "trace_every > 0 needs a trace buffer of (n_steps / trace_every, n_bodies, 9)");
    if (trace_every > n_steps)
        return fail(H2O_ERR_BAD_ARGUMENT, "trace_every (%d) > n_steps (%d): the rollout would write no trace row",
                    trace_every, n_steps);
    if (e->am_dense || e->surface_eta)
        return fail(H2O_ERR_NOT_CONFIGURED,
                    "persistent rollouts keep the wrapper's added-mass diagonal and take no caller height field "
                    "(the built-in wave field works)");
    if (e->warp_compat || e->b_w)
        return fail(H2O_ERR_NOT_CONFIGURED,
                    "persistent rollouts follow the Numba semantics and write no robot wrench: turn Warp "
                    "compatibility off and bind without a robot-wrench output, or use h2o_capture_rollout");
    if (!(dt > 1e-6)) return H2O_OK;  // hydrodynamics_behavior.py:139
    DeviceGuard g(e->device);
    RolloutArgs a;
    memset(&a, 0, sizeof a);
    a.pos = const_cast<void*>(e->b_pos); a.quat = const_cast<void*>(e->b_quat);
    a.lin = const_cast<void*>(e->b_lin); a.ang = const_cast<void*>(e->b_ang);
    a.prev = e->prev;
    a.out_force = e->b_f; a.out_torque = e->b_t;
    a.coeff = e->coeff; a.slot_type = e->slot_type;
    a.trace = trace_every > 0 ? trace_out : nullptr;
    a.stats = e->stats_on ? e->stats : nullptr;
    a.n = e->n;
    a.n_slots = e->n_slots; a.param_mode = e->param_mode;
    a.quat_wxyz = e->quat_order == H2O_QUAT_WXYZ;
    a.n_steps = n_steps; a.trace_every = trace_every;
    a.dt = dt; a.gravity = gravity; a.rho = e->rho; a.grav = e->grav;
    for (int k = 0; k < 3; ++k) a.current[k] = e->current[k];
    a.surface_z = e->surface_z;
    a.no_fallback = e->no_fallback;
    a.waves = wave_args(e);
    a.envs = env_args(e);
    a.grid = e->grid;
    const size_t smem = wave_smem_bytes(e->n_waves);
    // small batches: one warp per CTA so that the warps spread over the SMs (a lone warp per scheduler
    // issues back to back); large batches: ordinary 128-thread CTAs
    const int block = e->n <= (long long)e->sm_count * 4 * 32 ? 32 : 128;
    const int grid = int((e->n + block - 1) / block);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool st = e->stats_on;
    const bool env = e->env_cond != nullptr;
    const bool cg = e->grid.vals != nullptr;
    const bool sl = slope_on(e);
    const bool in = inertia_on(e);
#define H2O_ROLLOUT(S, ST, ENV, CG, SL)              \
    if (st == ST && env == ENV && cg == CG && sl == SL && !in) \
    rollout_persistent_kernel<S, ST, ENV, CG, SL><<<grid, block, smem, s>>>(a)
#define H2O_ROLLOUTS(S, SL) \
    H2O_ROLLOUT(S, true, true, false, SL); H2O_ROLLOUT(S, true, false, false, SL);   \
    H2O_ROLLOUT(S, false, true, false, SL); H2O_ROLLOUT(S, false, false, false, SL); \
    H2O_ROLLOUT(S, true, true, true, SL); H2O_ROLLOUT(S, true, false, true, SL);     \
    H2O_ROLLOUT(S, false, true, true, SL); H2O_ROLLOUT(S, false, false, true, SL)
// the inertia instantiations: only launched with a wave field or a time-varying grid
#define H2O_ROLLOUT_IN(S, ST, ENV, CG, SL)           \
    if (st == ST && env == ENV && cg == CG && sl == SL && in) \
    rollout_persistent_kernel<S, ST, ENV, CG, SL, true><<<grid, block, smem, s>>>(a)
#define H2O_ROLLOUTS_IN(S, SL) \
    H2O_ROLLOUT_IN(S, true, true, false, SL); H2O_ROLLOUT_IN(S, true, false, false, SL);   \
    H2O_ROLLOUT_IN(S, false, true, false, SL); H2O_ROLLOUT_IN(S, false, false, false, SL); \
    H2O_ROLLOUT_IN(S, true, true, true, SL); H2O_ROLLOUT_IN(S, true, false, true, SL);     \
    H2O_ROLLOUT_IN(S, false, true, true, SL); H2O_ROLLOUT_IN(S, false, false, true, SL)
    if (e->dtype == H2O_F32) {
        H2O_ROLLOUTS(float, false);
        H2O_ROLLOUTS(float, true);
        H2O_ROLLOUTS_IN(float, false);
        H2O_ROLLOUTS_IN(float, true);
    } else {
        H2O_ROLLOUTS(double, false);
        H2O_ROLLOUTS(double, true);
        H2O_ROLLOUTS_IN(double, false);
        H2O_ROLLOUTS_IN(double, true);
    }
#undef H2O_ROLLOUTS_IN
#undef H2O_ROLLOUT_IN
#undef H2O_ROLLOUTS
#undef H2O_ROLLOUT
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    e->last_kernel = H2O_KERNEL_DIRECT;
    if (clock_runs(e)) return advance_clock(e, dt, n_steps, s);
    return H2O_OK;
}

int h2o_components(h2o_handle h, const void* pos, const void* quat, const void* lin_vel, const void* ang_vel,
                   const void* lin_acc, const void* ang_acc, void* const out8[8], void* out_sub_ratio,
                   int32_t* out_flags, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (e->param_mode < 0) return fail(H2O_ERR_NOT_CONFIGURED, "no parameters set (h2o_set_params_*)");
    if (!out8) return fail(H2O_ERR_BAD_ARGUMENT, "out8 is NULL");
    const void* p[15] = {pos, quat, lin_vel, ang_vel, lin_acc, ang_acc, out8[0], out8[1], out8[2], out8[3],
                         out8[4], out8[5], out8[6], out8[7], out_sub_ratio};
    for (int i = 0; i < 15; ++i)
        if (!p[i]) return fail(H2O_ERR_BAD_ARGUMENT, "NULL tensor pointer (argument %d)", i);
    DeviceGuard g(e->device);
    ComponentsArgs a;
    memset(&a, 0, sizeof a);
    a.pos = pos; a.quat = quat; a.lin = lin_vel; a.ang = ang_vel; a.lin_acc = lin_acc; a.ang_acc = ang_acc;
    a.coeff = e->coeff;
    a.slot_type = e->slot_type;
    for (int i = 0; i < 8; ++i) a.out[i] = out8[i];
    a.out_ratio = out_sub_ratio;
    a.out_flags = out_flags;
    a.n = e->n;
    a.first_body = 0;
    a.n_slots = e->n_slots; a.n_types = e->n_types;
    a.param_mode = e->param_mode;
    a.quat_wxyz = e->quat_order == H2O_QUAT_WXYZ;
    a.warp_compat = e->warp_compat;
    a.rho = e->rho; a.grav = e->grav;
    for (int k = 0; k < 3; ++k) a.current[k] = e->current[k];
    a.surface_z = e->surface_z;
    const int grid = int((e->n + 255) / 256);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (e->dtype == H2O_F32) components_kernel<float><<<grid, 256, 0, s>>>(a);
    else components_kernel<double><<<grid, 256, 0, s>>>(a);
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    return H2O_OK;
}

// ---- host-buffer pipeline --------------------------------------------------------------
static int hp_init(h2o_engine* e)
{
    if (e->hp_stream[0]) return H2O_OK;
    for (int i = 0; i < HOST_PIPE_STREAMS; ++i) CUDA_TRY(cudaStreamCreateWithFlags(&e->hp_stream[i], cudaStreamNonBlocking));
    return H2O_OK;
}

static bool is_pinned_or_device(const void* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// Device-side alias of a pinned (page-locked, mapped) host buffer, or nullptr if `p` is anything else.
static void* mapped_alias(const void* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    return at.devicePointer;
}

// Host-buffer step.  `in` / `out` follow the layout: split = {pos, quat, lin, ang}, view = {pos, quat, vel6, -},
// physx = {transforms7, -, vel6, -}; out = {force, torque, robot wrench or NULL}.
//
// Pinned host buffers take the ZERO-COPY path: the fused tile kernel is launched straight on them -- its TMA bulk
// loads pull the tiles over PCIe into shared memory and its bulk stores push force / torque back, so transfer
// and arithmetic overlap tile by tile inside one kernel, with no staging buffers, no chunk pipeline and no
// pipeline tail (carried velocities and coefficients stay in HBM).  Pageable buffers are staged through
// engine-owned pinned memory and a chunked H2D -> step -> D2H pipeline on three streams.
static int step_host_impl(h2o_engine* e, int layout, const void* const in[4], void* const out[3], double dt)
{
    static const size_t widths[3][4] = {{3, 4, 3, 3}, {7, 0, 6, 0}, {3, 4, 6, 0}};
    const size_t* per_in = widths[layout];
    const size_t per_out[3] = {3, 3, 6};
    for (int i = 0; i < 4; ++i)
        if (per_in[i] && !in[i]) return fail(H2O_ERR_BAD_ARGUMENT, "NULL host input %d", i);
    if (!out[0] || !out[1]) return fail(H2O_ERR_BAD_ARGUMENT, "NULL host output");
    if (out[2] && e->bodies_per_robot <= 0)
        return fail(H2O_ERR_NOT_CONFIGURED, "robot wrench requested but h2o_set_articulation not called");
    if (e->param_mode < 0) return fail(H2O_ERR_NOT_CONFIGURED, "no parameters set (h2o_set_params_*)");
    if (!(dt > 1e-6)) return H2O_OK;
    DeviceGuard g(e->device);
    if (int rc = hp_init(e)) return rc;
    // No caller stream is passed in: order the engine's streams after everything queued so far on the
    // blocking streams (the legacy default stream synchronises with all of them) -- an event, not a
    // device-wide host synchronisation.
    if (!e->hp_event) CUDA_TRY(cudaEventCreateWithFlags(&e->hp_event, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(e->hp_event, cudaStreamLegacy));
    for (int i = 0; i < HOST_PIPE_STREAMS; ++i) {
        CUDA_TRY(cudaStreamWaitEvent(e->hp_stream[i], e->hp_event, 0));
        forget_last_tile(e->hp_stream[i]);
    }

    // ---- zero-copy path
    {
        void* din[4] = {nullptr, nullptr, nullptr, nullptr};
        void* dout[3] = {nullptr, nullptr, nullptr};
        bool ok = getenv("H2O_HOST_STAGED") == nullptr;
        for (int i = 0; i < 4 && ok; ++i)
            if (per_in[i]) ok = (din[i] = mapped_alias(in[i])) != nullptr && aligned16(din[i]);
        for (int i = 0; i < 3 && ok; ++i)
            if (out[i]) ok = (dout[i] = mapped_alias(out[i])) != nullptr && aligned16(dout[i]);
        if (ok) {
            cudaStream_t s = e->hp_stream[0];
            int rc = step_device(e, layout, din[0], din[1], din[2], din[3], dt, dout[0], dout[1], dout[2], e->n, 0,
                                 e->prev, coeff_at(e, 0), s);
            if (rc) return rc;
            CUDA_TRY(cudaStreamSynchronize(s));
            e->last_host_path = 1;
            return H2O_OK;
        }
    }
    e->last_host_path = 2;

    // ---- staged pipeline.  Pageable host memory goes through engine-owned pinned buffers.
    const void* src[4] = {nullptr, nullptr, nullptr, nullptr};
    void* dst[3];
    bool stage_out[3] = {false, false, false};
    for (int i = 0; i < 4; ++i) {
        if (!per_in[i]) continue;
        const size_t bytes = size_t(e->n) * per_in[i] * e->esz;
        if (e->hp_dev_bytes[i] < bytes) {
            if (e->hp_dev[i]) cudaFree(e->hp_dev[i]);
            e->hp_dev[i] = nullptr; e->hp_dev_bytes[i] = 0;
            CUDA_TRY(cudaMalloc(&e->hp_dev[i], bytes));
            e->hp_dev_bytes[i] = bytes;
        }
        if (is_pinned_or_device(in[i])) src[i] = in[i];
        else {
            if (e->hp_pin_bytes[i] < bytes) {
                if (e->hp_pin[i]) cudaFreeHost(e->hp_pin[i]);
                e->hp_pin[i] = nullptr; e->hp_pin_bytes[i] = 0;
                CUDA_TRY(cudaMallocHost(&e->hp_pin[i], bytes));
                e->hp_pin_bytes[i] = bytes;
            }
            memcpy(e->hp_pin[i], in[i], bytes);
            src[i] = e->hp_pin[i];
        }
    }
    {
        const size_t per_dev_out[3] = {3, 3, 6};
        for (int i = 0; i < 3; ++i) {
            const size_t bytes = size_t(e->n) * per_dev_out[i] * e->esz;
            if (!e->hp_dev[4 + i]) CUDA_TRY(cudaMalloc(&e->hp_dev[4 + i], bytes));
        }
    }
    for (int i = 0; i < 3; ++i) {
        dst[i] = out[i];
        if (!out[i]) continue;
        if (!is_pinned_or_device(out[i])) {
            const size_t bytes = size_t(e->n) * per_out[i] * e->esz / (i == 2 ? std::max(1, e->bodies_per_robot) : 1);
            if (!e->hp_pin[4 + i]) CUDA_TRY(cudaMallocHost(&e->hp_pin[4 + i], bytes));
            dst[i] = e->hp_pin[4 + i];
            stage_out[i] = true;
        }
    }

    // chunking: whole tiles / whole robots per chunk, a few chunks per stream
    const int bpr = (out[2] && e->bodies_per_robot > 0) ? e->bodies_per_robot : 0;
    long long unit = tile_unit(e->esz, bpr);
    while (unit < 256) unit *= 2;  // whole robots and whole 16-byte granules per chunk
    if (e->n_slots > 1) unit = unit / gcd_ll(unit, e->n_slots) * e->n_slots;  // keep slot phase per chunk
    // Chunk plan: the PCIe link is the bottleneck (H2D 52 B + D2H 24 B per body, full duplex), so
    // the H2D engine must never idle and the un-overlapped tail (kernel + D2H of the LAST chunk)
    // must be short: a few large chunks, tapered towards the end.
    int n_chunks = 4;
    if (const char* v = getenv("H2O_HOST_CHUNKS")) n_chunks = std::max(1, std::min(64, atoi(v)));
    std::vector<long long> bounds(1, 0);
    {
        double wsum = 0;
        std::vector<double> wgt(n_chunks);
        for (int k = 0; k < n_chunks; ++k) {
            wgt[k] = (k + 2 >= n_chunks && n_chunks > 2) ? (k + 1 == n_chunks ? 0.45 : 0.8) : 1.0;
            wsum += wgt[k];
        }
        double acc = 0;
        for (int k = 0; k < n_chunks; ++k) {
            acc += wgt[k];
            long long b = (long long)(double(e->n) * acc / wsum);
            b = std::min<long long>(e->n, (b + unit - 1) / unit * unit);
            if (k + 1 == n_chunks) b = e->n;
            if (b > bounds.back()) bounds.push_back(b);
        }
        if (bounds.back() != e->n) bounds.push_back(e->n);
    }

    for (size_t k = 0; k + 1 < bounds.size(); ++k) {
        const long long b0 = bounds[k];
        const long long cnt = bounds[k + 1] - b0;
        cudaStream_t s = e->hp_stream[k % HOST_PIPE_STREAMS];
        const void* dchunk[4] = {nullptr, nullptr, nullptr, nullptr};
        for (int i = 0; i < 4; ++i) {
            if (!per_in[i]) continue;
            const size_t off = size_t(b0) * per_in[i] * e->esz;
            CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(e->hp_dev[i]) + off, static_cast<const char*>(src[i]) + off,
                                     size_t(cnt) * per_in[i] * e->esz, cudaMemcpyDefault, s));
            dchunk[i] = static_cast<char*>(e->hp_dev[i]) + off;
        }
        char* dF = static_cast<char*>(e->hp_dev[4]) + size_t(b0) * 3 * e->esz;
        char* dT = static_cast<char*>(e->hp_dev[5]) + size_t(b0) * 3 * e->esz;
        char* dW = bpr ? static_cast<char*>(e->hp_dev[6]) + size_t(b0 / bpr) * 6 * e->esz : nullptr;
        int rc = step_device(e, layout, dchunk[0], dchunk[1], dchunk[2], dchunk[3], dt, dF, dT, dW, cnt, b0,
                             static_cast<char*>(e->prev) + size_t(b0) * 6 * e->esz, coeff_at(e, b0), s, false);
        if (rc) return rc;
        CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(dst[0]) + size_t(b0) * 3 * e->esz, dF, size_t(cnt) * 3 * e->esz,
                                 cudaMemcpyDefault, s));
        CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(dst[1]) + size_t(b0) * 3 * e->esz, dT, size_t(cnt) * 3 * e->esz,
                                 cudaMemcpyDefault, s));
        if (bpr && dst[2])
            CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(dst[2]) + size_t(b0 / bpr) * 6 * e->esz, dW,
                                     size_t(cnt / bpr) * 6 * e->esz, cudaMemcpyDefault, s));
    }
    for (int i = 0; i < HOST_PIPE_STREAMS; ++i) CUDA_TRY(cudaStreamSynchronize(e->hp_stream[i]));
    if (clock_runs(e)) {  // every chunk has read the clock: one advance for the whole step
        if (int rc = advance_clock(e, dt, 1, e->hp_stream[0])) return rc;
        CUDA_TRY(cudaStreamSynchronize(e->hp_stream[0]));
    }
    for (int i = 0; i < 3; ++i) {
        if (!stage_out[i]) continue;
        const size_t bytes = i == 2 ? size_t(e->n / std::max(1, e->bodies_per_robot)) * 6 * e->esz
                                    : size_t(e->n) * 3 * e->esz;
        memcpy(out[i], dst[i], bytes);
    }
    return H2O_OK;
}

int h2o_step_host(h2o_handle h, const void* pos, const void* quat, const void* lin_vel, const void* ang_vel,
                  double dt, void* out_force, void* out_torque, void* out_robot_wrench)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void* in[4] = {pos, quat, lin_vel, ang_vel};
    void* out[3] = {out_force, out_torque, out_robot_wrench};
    return step_host_impl(e, LAYOUT_SPLIT, in, out, dt);
}

int h2o_step_host_physx(h2o_handle h, const void* transforms, const void* velocities, double dt, void* out_force,
                        void* out_torque, void* out_robot_wrench)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void* in[4] = {transforms, nullptr, velocities, nullptr};
    void* out[3] = {out_force, out_torque, out_robot_wrench};
    return step_host_impl(e, LAYOUT_PHYSX, in, out, dt);
}

int h2o_last_host_path(h2o_handle h)
{
    h2o_engine* e = check(h);
    return e ? e->last_host_path : -1;
}

// ---- statistics / introspection ------------------------------------------------------------
int h2o_stats_device_ptr(h2o_handle h, void** out_ptr)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!out_ptr) return fail(H2O_ERR_BAD_ARGUMENT, "out_ptr is NULL");
    *out_ptr = e->stats;
    return H2O_OK;
}

int h2o_read_stats(h2o_handle h, double out[H2O_N_STATS], int reset, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!out) return fail(H2O_ERR_BAD_ARGUMENT, "out is NULL");
    DeviceGuard g(e->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaMemcpyAsync(out, e->stats, N_STATS * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (reset) CUDA_TRY(cudaMemsetAsync(e->stats, 0, N_STATS * sizeof(double), s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return H2O_OK;
}

int64_t h2o_launch_count(h2o_handle h)
{
    h2o_engine* e = check(h);
    return e ? e->launches : -1;
}
int64_t h2o_n_bodies(h2o_handle h)
{
    h2o_engine* e = check(h);
    return e ? e->n : -1;
}
int h2o_dtype_of(h2o_handle h)
{
    h2o_engine* e = check(h);
    return e ? e->dtype : -1;
}
int h2o_last_ctas_per_sm(h2o_handle h)
{
    h2o_engine* e = check(h);
    return e ? e->last_ctas_per_sm : -1;
}
int h2o_last_kernel(h2o_handle h)
{
    h2o_engine* e = check(h);
    return e ? e->last_kernel : -1;
}
int h2o_prev_device_ptr(h2o_handle h, void** out_ptr)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!out_ptr) return fail(H2O_ERR_BAD_ARGUMENT, "out_ptr is NULL");
    *out_ptr = e->prev;
    return H2O_OK;
}
int h2o_coeff_device_ptr(h2o_handle h, void** out_ptr, int64_t* out_rows)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!out_ptr || !out_rows) return fail(H2O_ERR_BAD_ARGUMENT, "NULL output");
    *out_ptr = e->coeff;
    *out_rows = e->coeff_rows;
    return H2O_OK;
}

// ---- DLPack twins --------------------------------------------------------------------------
static int dl_check(h2o_engine* e, const DLTensor* t, const char* name, int64_t rows, int64_t cols, bool is_int32,
                    const void** out_ptr)
{
    if (!t) return fail(H2O_ERR_BAD_ARGUMENT, "%s: NULL DLTensor", name);
    if (t->device.device_type != kDLCUDA && t->device.device_type != kDLCUDAManaged)
        return fail(H2O_ERR_BAD_DEVICE, "%s: not a CUDA tensor (device_type %d)", name, int(t->device.device_type));
    if (t->device.device_type == kDLCUDA && t->device.device_id != e->device)
        return fail(H2O_ERR_BAD_DEVICE, "%s: on cuda:%d, handle on cuda:%d", name, t->device.device_id, e->device);
    if (is_int32) {
        if (t->dtype.code != kDLInt || t->dtype.bits != 32 || t->dtype.lanes != 1)
            return fail(H2O_ERR_BAD_DTYPE, "%s: expected int32", name);
    } else {
        const int bits = e->dtype == H2O_F32 ? 32 : 64;
        if (t->dtype.code != kDLFloat || t->dtype.bits != bits || t->dtype.lanes != 1)
            return fail(H2O_ERR_BAD_DTYPE, "%s: expected float%d, got code %d bits %d", name, bits, int(t->dtype.code),
                        int(t->dtype.bits));
    }
    const int want_ndim = cols > 0 ? 2 : 1;
    if (t->ndim != want_ndim) return fail(H2O_ERR_BAD_SHAPE, "%s: expected %d-d tensor, got %d-d", name, want_ndim, t->ndim);
    if (t->shape[0] != rows || (cols > 0 && t->shape[1] != cols))
        return fail(H2O_ERR_BAD_SHAPE, "%s: expected shape (%lld%s%lld), got (%lld%s%lld)", name, (long long)rows,
                    cols > 0 ? "," : "", cols > 0 ? (long long)cols : 0LL, (long long)t->shape[0], cols > 0 ? "," : "",
                    cols > 0 ? (long long)t->shape[1] : 0LL);
    if (t->strides) {
        int64_t expect = 1;
        for (int d = t->ndim - 1; d >= 0; --d) {
            if (t->shape[d] != 1 && t->strides[d] != expect)
                return fail(H2O_ERR_NOT_CONTIGUOUS, "%s: not contiguous row-major", name);
            expect *= t->shape[d];
        }
    }
    const void* p = static_cast<const char*>(t->data) + t->byte_offset;
    if (!aligned16(p)) return fail(H2O_ERR_ALIGNMENT, "%s: data pointer is not 16-byte aligned", name);
    *out_ptr = p;
    return H2O_OK;
}

static int dl_wrench(h2o_engine* e, const DLTensor* w, const void** out_ptr)
{
    *out_ptr = nullptr;
    if (!w) return H2O_OK;
    if (e->robot_offsets) return dl_check(e, w, "out_robot_wrench", e->n_robots_var, 6, false, out_ptr);
    if (e->bodies_per_robot <= 0)
        return fail(H2O_ERR_NOT_CONFIGURED, "robot wrench requested but h2o_set_articulation not called");
    return dl_check(e, w, "out_robot_wrench", e->n / e->bodies_per_robot, 6, false, out_ptr);
}

int h2o_step_dl(h2o_handle h, const DLTensor* pos, const DLTensor* quat, const DLTensor* lin_vel,
                const DLTensor* ang_vel, double dt, const DLTensor* out_force, const DLTensor* out_torque,
                const DLTensor* out_robot_wrench, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void *p, *q, *v, *w, *f, *t, *rw;
    int rc;
    if ((rc = dl_check(e, pos, "position", e->n, 3, false, &p))) return rc;
    if ((rc = dl_check(e, quat, "orientation_quat", e->n, 4, false, &q))) return rc;
    if ((rc = dl_check(e, lin_vel, "linear_vel", e->n, 3, false, &v))) return rc;
    if ((rc = dl_check(e, ang_vel, "angular_vel", e->n, 3, false, &w))) return rc;
    if ((rc = dl_check(e, out_force, "out_force", e->n, 3, false, &f))) return rc;
    if ((rc = dl_check(e, out_torque, "out_torque", e->n, 3, false, &t))) return rc;
    if ((rc = dl_wrench(e, out_robot_wrench, &rw))) return rc;
    return h2o_step(h, p, q, v, w, dt, const_cast<void*>(f), const_cast<void*>(t), const_cast<void*>(rw), stream);
}

int h2o_step_physx_dl(h2o_handle h, const DLTensor* transforms, const DLTensor* velocities, double dt,
                      const DLTensor* out_force, const DLTensor* out_torque, const DLTensor* out_robot_wrench,
                      h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void *x, *v, *f, *t, *rw;
    int rc;
    if ((rc = dl_check(e, transforms, "transforms", e->n, 7, false, &x))) return rc;
    if ((rc = dl_check(e, velocities, "velocities", e->n, 6, false, &v))) return rc;
    if ((rc = dl_check(e, out_force, "out_force", e->n, 3, false, &f))) return rc;
    if ((rc = dl_check(e, out_torque, "out_torque", e->n, 3, false, &t))) return rc;
    if ((rc = dl_wrench(e, out_robot_wrench, &rw))) return rc;
    return h2o_step_physx(h, x, v, dt, const_cast<void*>(f), const_cast<void*>(t), const_cast<void*>(rw), stream);
}

int h2o_step_view_dl(h2o_handle h, const DLTensor* pos, const DLTensor* quat, const DLTensor* velocities, double dt,
                     const DLTensor* out_force, const DLTensor* out_torque, const DLTensor* out_robot_wrench,
                     h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void *p, *q, *v, *f, *t, *rw;
    int rc;
    if ((rc = dl_check(e, pos, "position", e->n, 3, false, &p))) return rc;
    if ((rc = dl_check(e, quat, "orientation_quat", e->n, 4, false, &q))) return rc;
    if ((rc = dl_check(e, velocities, "velocities", e->n, 6, false, &v))) return rc;
    if ((rc = dl_check(e, out_force, "out_force", e->n, 3, false, &f))) return rc;
    if ((rc = dl_check(e, out_torque, "out_torque", e->n, 3, false, &t))) return rc;
    if ((rc = dl_wrench(e, out_robot_wrench, &rw))) return rc;
    return h2o_step_view(h, p, q, v, dt, const_cast<void*>(f), const_cast<void*>(t), const_cast<void*>(rw), stream);
}

int h2o_bind_dl(h2o_handle h, int layout, const DLTensor* pos, const DLTensor* quat, const DLTensor* lin_vel,
                const DLTensor* ang_vel, const DLTensor* out_force, const DLTensor* out_torque,
                const DLTensor* out_robot_wrench)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void *p = nullptr, *q = nullptr, *v = nullptr, *w = nullptr, *f, *t, *rw;
    int rc;
    if (layout == LAYOUT_SPLIT) {
        if ((rc = dl_check(e, pos, "position", e->n, 3, false, &p))) return rc;
        if ((rc = dl_check(e, quat, "orientation_quat", e->n, 4, false, &q))) return rc;
        if ((rc = dl_check(e, lin_vel, "linear_vel", e->n, 3, false, &v))) return rc;
        if ((rc = dl_check(e, ang_vel, "angular_vel", e->n, 3, false, &w))) return rc;
    } else if (layout == LAYOUT_PHYSX) {
        if ((rc = dl_check(e, pos, "transforms", e->n, 7, false, &p))) return rc;
        if ((rc = dl_check(e, lin_vel, "velocities", e->n, 6, false, &v))) return rc;
    } else if (layout == LAYOUT_VIEW) {
        if ((rc = dl_check(e, pos, "position", e->n, 3, false, &p))) return rc;
        if ((rc = dl_check(e, quat, "orientation_quat", e->n, 4, false, &q))) return rc;
        if ((rc = dl_check(e, lin_vel, "velocities", e->n, 6, false, &v))) return rc;
    } else {
        return fail(H2O_ERR_BAD_ARGUMENT, "bad layout %d", layout);
    }
    if ((rc = dl_check(e, out_force, "out_force", e->n, 3, false, &f))) return rc;
    if ((rc = dl_check(e, out_torque, "out_torque", e->n, 3, false, &t))) return rc;
    if ((rc = dl_wrench(e, out_robot_wrench, &rw))) return rc;
    return h2o_bind(h, layout, p, q, v, w, const_cast<void*>(f), const_cast<void*>(t), const_cast<void*>(rw));
}

int h2o_components_dl(h2o_handle h, const DLTensor* pos, const DLTensor* quat, const DLTensor* lin_vel,
                      const DLTensor* ang_vel, const DLTensor* lin_acc, const DLTensor* ang_acc,
                      const DLTensor* const out8[8], const DLTensor* out_sub_ratio, const DLTensor* out_flags,
                      h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!out8) return fail(H2O_ERR_BAD_ARGUMENT, "out8 is NULL");
    const void *p, *q, *v, *w, *a, *al, *r, *fl = nullptr;
    const void* o[8];
    int rc;
    if ((rc = dl_check(e, pos, "position", e->n, 3, false, &p))) return rc;
    if ((rc = dl_check(e, quat, "orientation_quat", e->n, 4, false, &q))) return rc;
    if ((rc = dl_check(e, lin_vel, "linear_vel", e->n, 3, false, &v))) return rc;
    if ((rc = dl_check(e, ang_vel, "angular_vel", e->n, 3, false, &w))) return rc;
    if ((rc = dl_check(e, lin_acc, "linear_accel", e->n, 3, false, &a))) return rc;
    if ((rc = dl_check(e, ang_acc, "angular_accel", e->n, 3, false, &al))) return rc;
    static const char* names[8] = {"buoyancy_force", "drag_force", "lift_force", "drag_torque", "added_mass_force",
                                   "added_mass_torque", "center_of_buoyancy", "center_of_pressure"};
    for (int i = 0; i < 8; ++i)
        if ((rc = dl_check(e, out8[i], names[i], e->n, 3, false, &o[i]))) return rc;
    if ((rc = dl_check(e, out_sub_ratio, "sub_ratio", e->n, 0, false, &r))) return rc;
    if (out_flags && (rc = dl_check(e, out_flags, "flags", e->n, 0, true, &fl))) return rc;
    void* oo[8];
    for (int i = 0; i < 8; ++i) oo[i] = const_cast<void*>(o[i]);
    return h2o_components(h, p, q, v, w, a, al, oo, const_cast<void*>(r),
                          static_cast<int32_t*>(const_cast<void*>(fl)), stream);
}

int h2o_set_params_per_body_dl(h2o_handle h, const DLTensor* coeff, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!coeff) return fail(H2O_ERR_BAD_ARGUMENT, "coeff: NULL DLTensor");
    if (coeff->dtype.code != kDLFloat || (coeff->dtype.bits != 32 && coeff->dtype.bits != 64))
        return fail(H2O_ERR_BAD_DTYPE, "coeff: expected float32 or float64");
    if (coeff->ndim != 2 || coeff->shape[0] != e->n || coeff->shape[1] != N_COEFF)
        return fail(H2O_ERR_BAD_SHAPE, "coeff: expected shape (%lld,%d)", (long long)e->n, N_COEFF);
    if (coeff->strides && ((coeff->shape[1] != 1 && coeff->strides[1] != 1) || (coeff->shape[0] != 1 && coeff->strides[0] != N_COEFF)))
        return fail(H2O_ERR_NOT_CONTIGUOUS, "coeff: not contiguous row-major");
    const void* p = static_cast<const char*>(coeff->data) + coeff->byte_offset;
    return h2o_set_params_per_body(h, p, coeff->dtype.bits == 32 ? H2O_F32 : H2O_F64, stream);
}

int h2o_set_prev_dl(h2o_handle h, const DLTensor* prev_lin, const DLTensor* prev_ang, h2o_stream stream)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    const void *a, *b;
    int rc;
    if ((rc = dl_check(e, prev_lin, "prev_lin", e->n, 3, false, &a))) return rc;
    if ((rc = dl_check(e, prev_ang, "prev_ang", e->n, 3, false, &b))) return rc;
    return h2o_set_prev(h, a, b, stream);
}

struct PrevExport {
    DLManagedTensor mt;
    int64_t shape[2];
};
static void prev_export_deleter(DLManagedTensor* self)
{
    if (self) delete static_cast<PrevExport*>(self->manager_ctx);
}

int h2o_export_prev_dl(h2o_handle h, DLManagedTensor** out)
{
    h2o_engine* e = check(h);
    if (!e) return H2O_ERR_BAD_HANDLE;
    if (!out) return fail(H2O_ERR_BAD_ARGUMENT, "out is NULL");
    PrevExport* x = new PrevExport();
    x->shape[0] = e->n;
    x->shape[1] = 6;
    x->mt.dl_tensor.data = e->prev;
    x->mt.dl_tensor.device.device_type = kDLCUDA;
    x->mt.dl_tensor.device.device_id = e->device;
    x->mt.dl_tensor.ndim = 2;
    x->mt.dl_tensor.dtype.code = kDLFloat;
    x->mt.dl_tensor.dtype.bits = e->dtype == H2O_F32 ? 32 : 64;
    x->mt.dl_tensor.dtype.lanes = 1;
    x->mt.dl_tensor.shape = x->shape;
    x->mt.dl_tensor.strides = nullptr;
    x->mt.dl_tensor.byte_offset = 0;
    x->mt.manager_ctx = x;
    x->mt.deleter = prev_export_deleter;
    *out = &x->mt;
    return H2O_OK;
}

// ---------------------------------------------------------------------------
// Diagnostics of the launch overlap for the test suite; not part of the public ABI (include/h2o.h).
// ---------------------------------------------------------------------------
#define H2O_DIAG __attribute__((visibility("default")))

// 1 if the handle's last tile launch was captured to start while the previous grid of its stream drained.
H2O_DIAG int h2o_diag_last_overlap(h2o_handle h)
{
    h2o_engine* e = check(h);
    return e ? e->last_overlap : -1;
}

// The overlap decision of launch_tile, made without a device, for two fp32 split-layout per-body tile launches
// (robot mode when bodies_per_robot > 0) over n bodies each.  ptrs: pos, quat, lin, ang, prev, coeff, force, torque,
// wrench, stats, redo bitmap.  relation: 0 = eager, 1 = same capture and the later launch depends on the earlier one
// alone, 2 = same capture with other dependencies, 3 = another capture.  Returns 1 = start early, 0 = wait first.
H2O_DIAG int h2o_diag_overlap_decision(const void* const earlier[11], int64_t earlier_n, const void* const later[11],
                                       int64_t later_n, int bodies_per_robot, int relation)
{
    auto access = [&](const void* const p[11], int64_t n) {
        StepArgs a;
        memset(&a, 0, sizeof a);
        a.pos = p[0]; a.quat = p[1]; a.lin = p[2]; a.ang = p[3]; a.prev = const_cast<void*>(p[4]); a.coeff = p[5];
        a.out_force = const_cast<void*>(p[6]); a.out_torque = const_cast<void*>(p[7]);
        a.out_wrench = const_cast<void*>(p[8]);
        a.stats = static_cast<double*>(const_cast<void*>(p[9]));
        a.redo_bitmap = static_cast<uint32_t*>(const_cast<void*>(p[10]));
        a.n = n;
        a.bodies_per_robot = bodies_per_robot;
        a.tile_bodies = tile_bodies_for(128, sizeof(float), bodies_per_robot);
        a.n_tiles = a.tile_bodies > 0 ? int(n / a.tile_bodies) : 0;
        return bodies_per_robot > 0 ? tile_access<float, LAYOUT_SPLIT, PARAM_PER_BODY, true>(a)
                                    : tile_access<float, LAYOUT_SPLIT, PARAM_PER_BODY, false>(a);
    };
    const cudaGraphNode_t node = reinterpret_cast<cudaGraphNode_t>(uintptr_t(0x1000));
    const LastTile last{7, node, access(earlier, earlier_n)};
    CaptureState c;
    c.capturing = relation != 0;
    c.id = relation == 3 ? 8 : 7;
    c.only_dep = relation == 1 || relation == 3 ? node : nullptr;
    return may_start_early(&last, c, access(later, later_n)) ? 1 : 0;
}

}  // extern "C"
