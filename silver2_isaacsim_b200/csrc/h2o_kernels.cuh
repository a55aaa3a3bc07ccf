// h2o_kernels.cuh -- sm_100a kernels of the hydrodynamics force engine.
//
// Replaces, for N bodies in one launch, the reference's per-body call stack
//   HydrodynamicsBehavior._apply_behavior   hydrodynamics_behavior.py:176-238
//   -> XHydrodynamicsWrapper.calculate_hydrodynamic_forces
//        numba_hydrodynamics_wrapper.py:34 / warp_hydrodynamics_wrapper.py:79
//   -> solve_hydrodynamics                  numba_hydrodynamics.py:255-314
// (one `dim=1` Warp launch + 6 staging copies + ~30 torch micro-kernels per body).
//
// The kernels share the per-body arithmetic of h2o_model.cuh:
//
//   step_tile_kernel   persistent CTAs; every input array of a tile of bodies is
//                      brought into shared memory by the TMA engine
//                      (cp.async.bulk + mbarrier, multi-stage ring), each thread
//                      computes one body out of shared memory, results go back
//                      through shared memory and TMA bulk stores.  Row-major
//                      (N,3)/(N,4)/(N,6)/(N,7)/(N,11) caller layouts therefore cost
//                      no uncoalesced or partial-sector traffic.  Optional
//                      per-robot wrench summed out of shared memory.
//   step_direct_kernel one thread per body, plain global loads; used for small
//                      batches (latency-bound), tile tails and the f4 generalisations.
//   components_kernel  batched solve_hydrodynamics in the reference's full signature
//                      (eight vectors + sub_ratio), optional Warp-twin compatibility.
//   robot_wrench_kernel  one warp per robot, shuffle reduction (tails, big robots).
//   free_body_kernel   harness stepper for stand-alone rollouts (SURVEY.md 8(f2)).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "h2o_model.cuh"
#include "h2o_waves.cuh"

// study knob (-DH2O_SKIP_ALL=true): the warp-uniform surface-logic skip of the robot-mode kernels in EVERY tile kernel
// (the 80-register default kernel spills on it; used with regime-sorted inputs to bound what an in-tile sort could give)
#ifndef H2O_SKIP_ALL
#define H2O_SKIP_ALL false
#endif

namespace h2o {

enum : int { LAYOUT_SPLIT = 0, LAYOUT_PHYSX = 1, LAYOUT_VIEW = 2 };
enum : int { PARAM_TABLE = 0, PARAM_PER_BODY = 1 };
constexpr int N_COEFF = 11;
constexpr int MAX_TABLE_TYPES = 64;
constexpr int MAX_TABLE_SLOTS = 256;
constexpr int N_STATS = 8;  // sum|F|, max|F|, wet, clamped, nonfinite, still, bodies, re-evaluated in float64

struct StepArgs {
    // LAYOUT_SPLIT: pos (N,3), quat (N,4), lin (N,3), ang (N,3)
    // LAYOUT_PHYSX: pos = transforms (N,7) [p, q], lin = velocities (N,6) [v, w]
    // LAYOUT_VIEW:  pos (N,3), quat (N,4), lin = velocities (N,6) [v, w]  -- what RigidPrimView
    //               hands out (get_world_poses + get_velocities, hydrodynamics_behavior.py:178-179)
    const void* pos;
    const void* quat;
    const void* lin;
    const void* ang;
    void* prev;              // (N,6) previous-step [v, w]; read, then overwritten
    const void* coeff;       // PARAM_PER_BODY: (N,11); PARAM_TABLE: (n_types,11)
    const int32_t* slot_type;  // PARAM_TABLE: (n_slots,) slot -> type
    void* out_force;         // (N,3)
    void* out_torque;        // (N,3)
    void* out_wrench;        // (N / bodies_per_robot, 6) or nullptr
    double* stats;           // N_STATS doubles or nullptr
    long long n;             // bodies
    long long first_body;    // global index of body 0 of this launch (slot lookup)
    int tile_bodies;         // largest tile in bodies (multiple of `unit`, <= threads per CTA)
    int n_tiles;             // number of full tiles handled by the tile kernel (the rest: direct kernel)
    int n_slots, n_types;
    int bodies_per_robot;    // 0 = no articulation
    int quat_wxyz;           // 1: incoming quaternions are wxyz (Isaac core), else xyzw
    double rho, grav, inv_dt;
    double current[3];       // uniform water current (world): the flow-relative velocity is v - current
    double surface_z;        // height of the (flat) water surface; the reference's is z = 0
    // optional dense added mass (SURVEY.md 8(f4)): (am_n_types, 6, 6) row-major in the engine dtype and
    // its own slot -> matrix map; body i uses am_slot_type[(first_body + i) % am_n_slots].  Served by
    // the direct kernel only (the tile kernel keeps the wrapper's diagonal).
    const void* am_dense;
    const int32_t* am_slot_type;
    int am_n_slots;
    // optional non-flat water surface (SURVEY.md 8(f4)): (N,) surface height above surface_z at each body's
    // position, engine dtype, borrowed from the caller.  Direct kernel only.
    const void* surface_eta;
    // optional articulation of UNEQUAL robots: robot r owns bodies [robot_offsets[r], robot_offsets[r+1]);
    // nullptr = equal runs of bodies_per_robot.  Wrenches then come from robot_wrench_kernel.
    const long long* robot_offsets;
    long long n_robots_var;
    uint32_t* redo_bitmap;   // one bit per body of the ENGINE (index first_body + i), all zero between launches:
                             // flagged bodies that found no slot in their CTA's deferred list
    int warp_compat;         // 1: the fused step follows the reference's WARP twin (SURVEY.md Appendix C) instead of the
                             // Numba path: every body through the float64 world-frame formulation, direct kernel only
    int no_fallback;         // study knob H2O_NO_FALLBACK: 1 = keep the fast-path result of flagged bodies,
                             // k = 2^j > 1 = re-evaluate exactly every k-th body instead (cost measurements)
    int overlap;             // tile kernel: 1 = the host proved that this launch touches nothing the previous launch in
                             // the stream writes, and nothing it writes is read there: start before waiting for it
};

// Optional built-in wave field (h2o_set_wave_field): n rows of WAVE_STRIDE doubles, the water depth (+inf = deep)
// and the engine's clock (one double, device).  n == 0 = none.  A parameter of the per-body kernels only (the tile
// kernel, which has no wave code, keeps its StepArgs).
struct WaveArgs {
    const double* tab;
    const double* clock;
    double depth;
    int n;
};

// Optional per-env water conditions (h2o_set_env_conditions): the borrowed (E, ENV_STRIDE) float64 array, read by
// every launch, and the env size; body i (global index) belongs to env i / bodies_per_env.  cond == nullptr = none.
// Like WaveArgs, a parameter of the per-body kernels only.
struct EnvArgs {
    const double* cond;
    long long bodies_per_env;
};

// The optional current grid (h2o_set_current_grid) travels as GridArgs (csrc/h2o_waves.cuh), the third argument of
// this kind, again of the per-body kernels only.

// ---------------------------------------------------------------------------
// PTX wrappers: mbarrier + bulk async copies (TMA engine, SASS UBLKCP)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) {
    }
}
// global -> shared, completion counted on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// shared -> global, tracked by the per-thread bulk async-group
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
                 "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read()
{
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N> __device__ __forceinline__ void bulk_wait_all()
{
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// Programmatic dependent launch (PDL).  griddepcontrol.wait returns once the previous grid of the stream has completed
// and its writes are visible; launch_dependents lets the next grid start once every CTA of this one has executed it (or
// exited).  Invariant of every kernel here: no thread executes launch_dependents before its own wait has returned.  So
// when a grid starts early, only the one grid before it can still be running -- the launch the host checked it against.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait_prerequisites() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2_keep(const void* p)
{
    asm volatile("prefetch.global.L2::evict_last [%0];" ::"l"(p) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------------------
// Per-body input gather (works on shared-memory tiles and on global arrays alike)
// ---------------------------------------------------------------------------
template <typename S> struct BodyPtrs {
    const S* pos;    // SPLIT: 3/body   PHYSX: 7/body
    const S* quat;   // SPLIT: 4/body   PHYSX: unused
    const S* lin;    // SPLIT: 3/body   PHYSX: 6/body
    const S* ang;    // SPLIT: 3/body   PHYSX: unused
    const S* prev;   // 6/body
    const S* coeff;  // 11/record
};

template <typename S> struct Vec2Of;
template <> struct Vec2Of<float> { using type = float2; };
template <> struct Vec2Of<double> { using type = double2; };

template <typename S> struct RawBody {
    S px, py, pz, q0, q1, q2, q3;
    S vx, vy, vz, wx, wy, wz;
    S pvx, pvy, pvz, pwx, pwy, pwz;
};

template <typename S, int kLayout, bool kPrevRow = false>
__device__ __forceinline__ void load_raw(const BodyPtrs<S>& p, long long i, RawBody<S>& r)
{
    using V2 = typename Vec2Of<S>::type;
    if (kLayout == LAYOUT_SPLIT || kLayout == LAYOUT_VIEW) {
        const S* pp = p.pos + 3 * i;
        r.px = pp[0]; r.py = pp[1]; r.pz = pp[2];
        if (sizeof(S) == 4) {
            const float4 q = *reinterpret_cast<const float4*>(p.quat + 4 * i);
            r.q0 = q.x; r.q1 = q.y; r.q2 = q.z; r.q3 = q.w;
        } else {
            const double2 qa = *reinterpret_cast<const double2*>(p.quat + 4 * i);
            const double2 qb = *reinterpret_cast<const double2*>(p.quat + 4 * i + 2);
            r.q0 = qa.x; r.q1 = qa.y; r.q2 = qb.x; r.q3 = qb.y;
        }
        if (kLayout == LAYOUT_SPLIT) {
            const S* pv = p.lin + 3 * i;
            r.vx = pv[0]; r.vy = pv[1]; r.vz = pv[2];
            const S* pw = p.ang + 3 * i;
            r.wx = pw[0]; r.wy = pw[1]; r.wz = pw[2];
        } else {
            const V2* pv = reinterpret_cast<const V2*>(p.lin + 6 * i);
            const V2 a = pv[0], b = pv[1], c = pv[2];
            r.vx = a.x; r.vy = a.y; r.vz = b.x; r.wx = b.y; r.wy = c.x; r.wz = c.y;
        }
    } else {
        const S* pp = p.pos + 7 * i;
        r.px = pp[0]; r.py = pp[1]; r.pz = pp[2];
        r.q0 = pp[3]; r.q1 = pp[4]; r.q2 = pp[5]; r.q3 = pp[6];
        const V2* pv = reinterpret_cast<const V2*>(p.lin + 6 * i);
        const V2 a = pv[0], b = pv[1], c = pv[2];
        r.vx = a.x; r.vy = a.y; r.vz = b.x; r.wx = b.y; r.wy = c.x; r.wz = c.y;
    }
    // kPrevRow: p.prev already points at this body's six previous velocities (a saved copy)
    const V2* pr = reinterpret_cast<const V2*>(kPrevRow ? p.prev : p.prev + 6 * i);
    const V2 a = pr[0], b = pr[1], c = pr[2];
    r.pvx = a.x; r.pvy = a.y; r.pvz = b.x; r.pwx = b.y; r.pwy = c.x; r.pwz = c.y;
}

// Assemble the model input: quaternion order (hydrodynamics_behavior.py:194),
// finite-difference acceleration (hydrodynamics_behavior.py:196-202), coefficients.
// Environment generalisation (SURVEY.md 8(f4)): uniform current and surface height; both zero
// reproduces the reference exactly (x - 0 is exact).
struct Env {
    double cx, cy, cz, surface_z;
};

template <typename S>
__device__ __forceinline__ void make_body_in(const RawBody<S>& r, const S* c, int quat_wxyz, double rho,
                                             double grav, S inv_dt, const Env& env, BodyIn<double, S>& in)
{
    in.pz = double(r.pz) - env.surface_z;
    if (quat_wxyz) {
        in.qx = double(r.q1); in.qy = double(r.q2); in.qz = double(r.q3); in.qw = double(r.q0);
    } else {
        in.qx = double(r.q0); in.qy = double(r.q1); in.qz = double(r.q2); in.qw = double(r.q3);
    }
    // drag, damping and lift see the flow-relative velocity; accelerations are differences of
    // body velocities and do not change under a steady current
    in.vx = r.vx - S(env.cx); in.vy = r.vy - S(env.cy); in.vz = r.vz - S(env.cz);
    in.wx = r.wx; in.wy = r.wy; in.wz = r.wz;
    if (sizeof(S) == 4) {  // fp32 fast path folds 1/dt into the added-mass constants
        in.ax = r.vx - r.pvx; in.ay = r.vy - r.pvy; in.az = r.vz - r.pvz;
        in.bx = r.wx - r.pwx; in.by = r.wy - r.pwy; in.bz = r.wz - r.pwz;
        in.acc_scale = inv_dt;
    } else {
        in.ax = (r.vx - r.pvx) * inv_dt; in.ay = (r.vy - r.pvy) * inv_dt; in.az = (r.vz - r.pvz) * inv_dt;
        in.bx = (r.wx - r.pwx) * inv_dt; in.by = (r.wy - r.pwy) * inv_dt; in.bz = (r.wz - r.pwz) * inv_dt;
        in.acc_scale = S(1);
    }
    in.dimx = c[0]; in.dimy = c[1]; in.dimz = c[2];
    in.c_drag = c[3]; in.c_drag_ang = c[4]; in.k_damp = c[5]; in.k_damp_ang = c[6];
    in.c_am = c[7]; in.c_am_ang = c[8]; in.c_lift = c[9];
    in.rho_h = rho; in.grav_h = grav; in.rho = S(rho);
    in.warp_compat = false;
    in.am_dense = nullptr;
}

// Running statistics kept in registers across a thread's bodies.
struct ThreadStats {
    double sum_f = 0.0, max_f = 0.0;
    unsigned wet = 0, clamped = 0, nonfinite = 0, still = 0, bodies = 0, redone = 0;
};

// fp32 mode, bodies the fast path flags as ill-conditioned (body_wrench_fast: cancelling torque / force
// groups, quaternion far from unit): out-of-line float64 re-evaluation with the world-frame formulation
// (body_terms + net_wrench, the fp64-mode arithmetic), so that fp32 mode meets its bound for EVERY body.
// A few bodies per 10 000: the function re-reads the body's inputs from global memory instead of keeping
// thirty scalars alive across the fast path (the hot path keeps its registers), and is never inlined.
struct ExactStepOut {
    float F[3], T[3];
    float ratio;
    int flags;  // bit 0 clamped, bit 1 still
};
// Core (inlined into its noinline carriers below): the fp64-mode arithmetic on one fp32-stored body.  kSlope: the
// waterline is the tangent plane of slope (sx, sy) (h2o_set_wave_slope).  kInertia: the fluid-acceleration loads for
// a_f = (afx, afy, afz) (h2o_set_fluid_inertia).
template <bool kSlope = false, bool kInertia = false>
__device__ __forceinline__ ExactStepOut exact_eval_f32(const RawBody<float>& r, const float* c, int quat_wxyz, double rho,
                                                        double grav, double inv_dt, double surface_z, float cx, float cy,
                                                        float cz, const float* am_dense, bool warp_compat = false,
                                                        double sx = 0.0, double sy = 0.0, double afx = 0.0,
                                                        double afy = 0.0, double afz = 0.0)
{
    BodyIn<double, double> g;
    g.pz = double(r.pz) - surface_z;
    if (quat_wxyz) { g.qx = r.q1; g.qy = r.q2; g.qz = r.q3; g.qw = r.q0; }
    else { g.qx = r.q0; g.qy = r.q1; g.qz = r.q2; g.qw = r.q3; }
    // flow-relative velocity: the fast path forms it in fp32 (make_body_in), and so does this
    g.vx = double(r.vx - cx); g.vy = double(r.vy - cy); g.vz = double(r.vz - cz);
    g.wx = r.wx; g.wy = r.wy; g.wz = r.wz;
    g.ax = (double(r.vx) - double(r.pvx)) * inv_dt; g.ay = (double(r.vy) - double(r.pvy)) * inv_dt;
    g.az = (double(r.vz) - double(r.pvz)) * inv_dt;
    g.bx = (double(r.wx) - double(r.pwx)) * inv_dt; g.by = (double(r.wy) - double(r.pwy)) * inv_dt;
    g.bz = (double(r.wz) - double(r.pwz)) * inv_dt;
    g.acc_scale = 1.0;
    g.dimx = c[0]; g.dimy = c[1]; g.dimz = c[2];
    g.c_drag = c[3]; g.c_drag_ang = c[4]; g.k_damp = c[5]; g.k_damp_ang = c[6];
    g.c_am = c[7]; g.c_am_ang = c[8]; g.c_lift = c[9];
    g.warp_compat = warp_compat;
    g.rho_h = rho; g.grav_h = grav; g.rho = double(float(rho));  // L constants as the fast path rounds them
    double md[36];
    g.am_dense = nullptr;
    if (am_dense) {
        for (int j = 0; j < 36; ++j) md[j] = double(am_dense[j]);
        g.am_dense = md;
    }
    Terms<double, double> t;
    body_terms<double, double, false, kSlope, kInertia>(g, t, nullptr, sx, sy, afx, afy, afz);
    double F[3], T[3];
    bool clamped;
    net_wrench<double, double, kInertia>(t, double(c[10]), F, T, clamped);
    ExactStepOut o;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        o.F[j] = float(F[j]);
        o.T[j] = float(T[j]);
    }
    o.ratio = float(t.ratio);
    o.flags = (clamped ? 1 : 0) | (t.still ? 2 : 0);
    return o;
}
// Persistent rollout kernel: the body's state lives in registers; handed over by reference (rare path).
__device__ __noinline__ ExactStepOut body_step_exact_f32(const RawBody<float>& r, const float* c, int quat_wxyz, double rho,
                                                         double grav, double inv_dt, double surface_z, float cx, float cy,
                                                         float cz, bool warp_compat = false)
{
    return exact_eval_f32(r, c, quat_wxyz, rho, grav, inv_dt, surface_z, cx, cy, cz, nullptr, warp_compat);
}
// The same with the tangent-plane waterline of slope (sx, sy): its own carrier, so that kernels without slope keep
// their call sites.
__device__ __noinline__ ExactStepOut body_step_exact_f32_slope(const RawBody<float>& r, const float* c, int quat_wxyz,
                                                               double rho, double grav, double inv_dt, double surface_z,
                                                               float cx, float cy, float cz, double sx, double sy,
                                                               bool warp_compat = false)
{
    return exact_eval_f32<true>(r, c, quat_wxyz, rho, grav, inv_dt, surface_z, cx, cy, cz, nullptr, warp_compat, sx, sy);
}
// The same with the fluid-acceleration loads for a_f (and the slope when kSlope): carriers of their own, so that kernels
// without the mode keep their call sites.
template <bool kSlope>
__device__ __noinline__ ExactStepOut body_step_exact_f32_inertia(const RawBody<float>& r, const float* c, int quat_wxyz,
                                                                 double rho, double grav, double inv_dt, double surface_z,
                                                                 float cx, float cy, float cz, double sx, double sy,
                                                                 double afx, double afy, double afz)
{
    return exact_eval_f32<kSlope, true>(r, c, quat_wxyz, rho, grav, inv_dt, surface_z, cx, cy, cz, nullptr, false, sx, sy,
                                        afx, afy, afz);
}
// Step kernels: re-read the flagged body's inputs from global memory (they are L2-resident: the tile was
// streamed in microseconds ago), so the hot path keeps no input alive for this.  Scalars cross the call by
// value (registers), nothing goes through local memory.
template <int kLayout, int kParam, bool kPrevRow>
__device__ __noinline__ ExactStepOut body_step_exact_from_global(
    const float* pos, const float* quat, const float* lin, const float* ang, const float* prev, const float* coeff,
    const int32_t* slot_type, long long i, long long first_body, int n_slots, int quat_wxyz, double rho, double grav,
    double inv_dt, double surface_z, float cx, float cy, float cz, const float* am_dense)
{
    BodyPtrs<float> bp;
    bp.pos = pos; bp.quat = quat; bp.lin = lin; bp.ang = ang; bp.prev = prev; bp.coeff = coeff;
    RawBody<float> r;
    load_raw<float, kLayout, kPrevRow>(bp, i, r);
    const float* c = coeff + N_COEFF * (kParam == PARAM_PER_BODY ? i : (long long)slot_type[(first_body + i) % n_slots]);
    float cl[N_COEFF];
#pragma unroll
    for (int j = 0; j < N_COEFF; ++j) cl[j] = c[j];
    return exact_eval_f32(r, cl, quat_wxyz, rho, grav, inv_dt, surface_z, cx, cy, cz, am_dense);
}
// The same with the tangent-plane waterline of slope (sx, sy) (step_direct_kernel's slope instantiations).
template <int kLayout, int kParam>
__device__ __noinline__ ExactStepOut body_step_exact_from_global_slope(
    const float* pos, const float* quat, const float* lin, const float* ang, const float* prev, const float* coeff,
    const int32_t* slot_type, long long i, long long first_body, int n_slots, int quat_wxyz, double rho, double grav,
    double inv_dt, double surface_z, float cx, float cy, float cz, const float* am_dense, double sx, double sy)
{
    BodyPtrs<float> bp;
    bp.pos = pos; bp.quat = quat; bp.lin = lin; bp.ang = ang; bp.prev = prev; bp.coeff = coeff;
    RawBody<float> r;
    load_raw<float, kLayout, false>(bp, i, r);
    const float* c = coeff + N_COEFF * (kParam == PARAM_PER_BODY ? i : (long long)slot_type[(first_body + i) % n_slots]);
    float cl[N_COEFF];
#pragma unroll
    for (int j = 0; j < N_COEFF; ++j) cl[j] = c[j];
    return exact_eval_f32<true>(r, cl, quat_wxyz, rho, grav, inv_dt, surface_z, cx, cy, cz, am_dense, false, sx, sy);
}
// The same with the fluid-acceleration loads (step_direct_kernel's inertia instantiations).
template <int kLayout, int kParam, bool kSlope>
__device__ __noinline__ ExactStepOut body_step_exact_from_global_inertia(
    const float* pos, const float* quat, const float* lin, const float* ang, const float* prev, const float* coeff,
    const int32_t* slot_type, long long i, long long first_body, int n_slots, int quat_wxyz, double rho, double grav,
    double inv_dt, double surface_z, float cx, float cy, float cz, const float* am_dense, double sx, double sy,
    double afx, double afy, double afz)
{
    BodyPtrs<float> bp;
    bp.pos = pos; bp.quat = quat; bp.lin = lin; bp.ang = ang; bp.prev = prev; bp.coeff = coeff;
    RawBody<float> r;
    load_raw<float, kLayout, false>(bp, i, r);
    const float* c = coeff + N_COEFF * (kParam == PARAM_PER_BODY ? i : (long long)slot_type[(first_body + i) % n_slots]);
    float cl[N_COEFF];
#pragma unroll
    for (int j = 0; j < N_COEFF; ++j) cl[j] = c[j];
    return exact_eval_f32<kSlope, true>(r, cl, quat_wxyz, rho, grav, inv_dt, surface_z, cx, cy, cz, am_dense, false, sx,
                                        sy, afx, afy, afz);
}
// prev_row: nullptr = the body's row of a.prev (still the OLD velocities), else a saved copy of that row.
// surface_z, cx, cy, cz: the waterline and the flow (rounded to float) the fast path saw for this body.
template <int kLayout, int kParam>
__device__ __forceinline__ ExactStepOut redo_exact(const StepArgs& a, long long i, double surface_z, float cx, float cy,
                                                   float cz, const float* prev_row = nullptr)
{
    const float* am = a.am_dense ? reinterpret_cast<const float*>(a.am_dense) + 36 * a.am_slot_type[(a.first_body + i) % a.am_n_slots]
                                 : nullptr;
    if (prev_row)
        return body_step_exact_from_global<kLayout, kParam, true>(
            reinterpret_cast<const float*>(a.pos), reinterpret_cast<const float*>(a.quat),
            reinterpret_cast<const float*>(a.lin), reinterpret_cast<const float*>(a.ang), prev_row,
            reinterpret_cast<const float*>(a.coeff), a.slot_type, i, a.first_body, a.n_slots, a.quat_wxyz, a.rho, a.grav,
            a.inv_dt, surface_z, cx, cy, cz, am);
    return body_step_exact_from_global<kLayout, kParam, false>(
        reinterpret_cast<const float*>(a.pos), reinterpret_cast<const float*>(a.quat), reinterpret_cast<const float*>(a.lin),
        reinterpret_cast<const float*>(a.ang), reinterpret_cast<const float*>(a.prev), reinterpret_cast<const float*>(a.coeff),
        a.slot_type, i, a.first_body, a.n_slots, a.quat_wxyz, a.rho, a.grav, a.inv_dt, surface_z, cx, cy, cz, am);
}
template <int kLayout, int kParam>
__device__ __forceinline__ ExactStepOut redo_exact_slope(const StepArgs& a, long long i, double surface_z, float cx,
                                                         float cy, float cz, double sx, double sy)
{
    const float* am = a.am_dense ? reinterpret_cast<const float*>(a.am_dense) + 36 * a.am_slot_type[(a.first_body + i) % a.am_n_slots]
                                 : nullptr;
    return body_step_exact_from_global_slope<kLayout, kParam>(
        reinterpret_cast<const float*>(a.pos), reinterpret_cast<const float*>(a.quat), reinterpret_cast<const float*>(a.lin),
        reinterpret_cast<const float*>(a.ang), reinterpret_cast<const float*>(a.prev), reinterpret_cast<const float*>(a.coeff),
        a.slot_type, i, a.first_body, a.n_slots, a.quat_wxyz, a.rho, a.grav, a.inv_dt, surface_z, cx, cy, cz, am, sx, sy);
}
template <int kLayout, int kParam, bool kSlope>
__device__ __forceinline__ ExactStepOut redo_exact_inertia(const StepArgs& a, long long i, double surface_z, float cx,
                                                           float cy, float cz, double sx, double sy, const double af[3])
{
    const float* am = a.am_dense ? reinterpret_cast<const float*>(a.am_dense) + 36 * a.am_slot_type[(a.first_body + i) % a.am_n_slots]
                                 : nullptr;
    return body_step_exact_from_global_inertia<kLayout, kParam, kSlope>(
        reinterpret_cast<const float*>(a.pos), reinterpret_cast<const float*>(a.quat), reinterpret_cast<const float*>(a.lin),
        reinterpret_cast<const float*>(a.ang), reinterpret_cast<const float*>(a.prev), reinterpret_cast<const float*>(a.coeff),
        a.slot_type, i, a.first_body, a.n_slots, a.quat_wxyz, a.rho, a.grav, a.inv_dt, surface_z, cx, cy, cz, am, sx, sy,
        af[0], af[1], af[2]);
}

// Deferred re-evaluation at the end of a tile-kernel CTA: one saved body per lane, and the float64 model split
// into four ROLES that four warps evaluate concurrently (a single lane doing all of it under the step
// kernel's register cap takes ~4 us, which is pure tail latency; profiles/r02_fallback_cost.md).  Every role
// instantiates the same body_terms; the compiler keeps only the chains its outputs need.
enum : int { ROLE_DRAG = 0, ROLE_LIFT = 1, ROLE_HYDROSTATIC = 2, ROLE_ADDED_MASS = 3, N_ROLES = 4, ROLE_DOUBLES = 10 };
template <int kRole, int kLayout, int kParam>
__device__ __noinline__ void exact_role_from_global(
    const float* pos, const float* quat, const float* lin, const float* ang, const float* prev_row, const float* coeff,
    const int32_t* slot_type, long long i, long long first_body, int n_slots, int quat_wxyz, double rho, double grav,
    double inv_dt, double surface_z, float cx, float cy, float cz, uint32_t kp_mask, double* out)
{
    BodyPtrs<float> bp;
    bp.pos = pos; bp.quat = quat; bp.lin = lin; bp.ang = ang; bp.prev = prev_row; bp.coeff = coeff;
    RawBody<float> r;
    load_raw<float, kLayout, true>(bp, i, r);
    const float* c = coeff + N_COEFF * (kParam == PARAM_PER_BODY ? i : (long long)slot_type[(first_body + i) % n_slots]);
    BodyIn<double, double> g;
    g.pz = double(r.pz) - surface_z;
    if (quat_wxyz) { g.qx = r.q1; g.qy = r.q2; g.qz = r.q3; g.qw = r.q0; }
    else { g.qx = r.q0; g.qy = r.q1; g.qz = r.q2; g.qw = r.q3; }
    g.vx = double(r.vx - cx); g.vy = double(r.vy - cy); g.vz = double(r.vz - cz);
    g.wx = r.wx; g.wy = r.wy; g.wz = r.wz;
    g.ax = (double(r.vx) - double(r.pvx)) * inv_dt; g.ay = (double(r.vy) - double(r.pvy)) * inv_dt;
    g.az = (double(r.vz) - double(r.pvz)) * inv_dt;
    g.bx = (double(r.wx) - double(r.pwx)) * inv_dt; g.by = (double(r.wy) - double(r.pwy)) * inv_dt;
    g.bz = (double(r.wz) - double(r.pwz)) * inv_dt;
    g.acc_scale = 1.0;
    g.dimx = c[0]; g.dimy = c[1]; g.dimz = c[2];
    g.c_drag = c[3]; g.c_drag_ang = c[4]; g.k_damp = c[5]; g.k_damp_ang = c[6];
    g.c_am = c[7]; g.c_am_ang = c[8]; g.c_lift = c[9];
    g.warp_compat = false;
    g.rho_h = rho; g.grav_h = grav; g.rho = double(float(rho));
    g.am_dense = nullptr;
    Terms<double, double> t;
    body_terms<double, double, false>(g, t, &kp_mask);
    if (kRole == ROLE_DRAG) {
        out[0] = t.fd[0]; out[1] = t.fd[1]; out[2] = t.fd[2];
        out[3] = t.tarm[0]; out[4] = t.tarm[1]; out[5] = t.tarm[2];
        out[6] = t.cop[0]; out[7] = t.cop[1]; out[8] = t.cop[2];
    } else if (kRole == ROLE_LIFT) {
        out[0] = t.fl[0]; out[1] = t.fl[1]; out[2] = t.fl[2];
    } else if (kRole == ROLE_HYDROSTATIC) {
        out[0] = t.td[0]; out[1] = t.td[1]; out[2] = t.td[2];
        out[3] = t.cob[0]; out[4] = t.cob[1]; out[5] = t.cob[2];
        out[6] = t.fbz; out[7] = double(c[10]);
    } else {
        out[0] = t.fam[0]; out[1] = t.fam[1]; out[2] = t.fam[2];
        out[3] = t.tam[0]; out[4] = t.tam[1]; out[5] = t.tam[2];
    }
}
template <int kLayout, int kParam>
__device__ __forceinline__ void redo_role(int role, const StepArgs& a, long long i, double surface_z, const float* prev_row,
                                          uint32_t kp_mask, double* out)
{
#define H2O_ROLE(R)                                                                                                        \
    exact_role_from_global<R, kLayout, kParam>(                                                                            \
        reinterpret_cast<const float*>(a.pos), reinterpret_cast<const float*>(a.quat), reinterpret_cast<const float*>(a.lin), \
        reinterpret_cast<const float*>(a.ang), prev_row, reinterpret_cast<const float*>(a.coeff), a.slot_type, i,         \
        a.first_body, a.n_slots, a.quat_wxyz, a.rho, a.grav, a.inv_dt, surface_z, float(a.current[0]), float(a.current[1]), \
        float(a.current[2]), kp_mask, out)
    if (role == ROLE_DRAG) H2O_ROLE(ROLE_DRAG);
    else if (role == ROLE_LIFT) H2O_ROLE(ROLE_LIFT);
    else if (role == ROLE_HYDROSTATIC) H2O_ROLE(ROLE_HYDROSTATIC);
    else H2O_ROLE(ROLE_ADDED_MASS);
#undef H2O_ROLE
}
// the four partial results of one body -> net wrench + clamp (hydrodynamics_behavior.py:212-226)
__device__ __noinline__ ExactStepOut combine_roles(const double* p)
{
    Terms<double, double> t;
    const double* d = p + ROLE_DRAG * ROLE_DOUBLES;
    const double* l = p + ROLE_LIFT * ROLE_DOUBLES;
    const double* h = p + ROLE_HYDROSTATIC * ROLE_DOUBLES;
    const double* m = p + ROLE_ADDED_MASS * ROLE_DOUBLES;
    for (int k = 0; k < 3; ++k) {
        t.fd[k] = d[k]; t.tarm[k] = d[3 + k]; t.cop[k] = d[6 + k];
        t.fl[k] = l[k];
        t.td[k] = h[k]; t.cob[k] = h[3 + k];
        t.fam[k] = m[k]; t.tam[k] = m[3 + k];
    }
    t.fbz = h[6];
    double F[3], T[3];
    bool clamped;
    net_wrench<double, double>(t, h[7], F, T, clamped);
    ExactStepOut o;
    for (int k = 0; k < 3; ++k) {
        o.F[k] = float(F[k]);
        o.T[k] = float(T[k]);
    }
    o.ratio = 0.f;
    o.flags = clamped ? 1 : 0;
    return o;
}

// fp32 mode: body-frame fast path (returns true when the body must be re-evaluated, see above);
// fp64 mode: the world-frame formulation (exact in dq).  kSlope: the tangent-plane waterline of slope (sx, sy).
// kInertia: the fluid-acceleration loads for a_f = af (h2o_set_fluid_inertia).
template <typename S, bool kWarpSkip = false, bool kSlope = false, bool kInertia = false>
__device__ __forceinline__ bool body_step(const BodyIn<double, S>& in, S mass, S F[3], S T[3], bool& clamped,
                                          bool& still, double& ratio, uint32_t& mask, double sx = 0.0, double sy = 0.0,
                                          const double* af = nullptr)
{
    const double afx = kInertia ? af[0] : 0.0, afy = kInertia ? af[1] : 0.0, afz = kInertia ? af[2] : 0.0;
    if (sizeof(S) == 4) {
        bool suspect;
        body_wrench_fast<double, S, kWarpSkip, kSlope, kInertia>(in, mass, F, T, clamped, ratio, still, suspect, mask,
                                                                 nullptr, sx, sy, afx, afy, afz);
        return suspect;
    } else {
        mask = 0;
        Terms<double, S> t;
        body_terms<double, S, false, kSlope, kInertia>(in, t, nullptr, sx, sy, afx, afy, afz);
        net_wrench<double, S, kInertia>(t, mass, F, T, clamped);
        ratio = t.ratio;
        still = t.still;
        return false;
    }
}

__device__ __forceinline__ void accumulate_stats(ThreadStats& st, double fx, double fy, double fz, double ratio,
                                                 bool clamped, bool still, bool redone)
{
    const double mag = sqrt(fx * fx + fy * fy + fz * fz);
    st.bodies += 1;
    if (mag == mag && mag < 1.7e308) {
        st.sum_f += mag;
        st.max_f = fmax(st.max_f, mag);
    } else {
        st.nonfinite += 1;
    }
    st.wet += (ratio > 0.0) ? 1u : 0u;
    st.clamped += clamped ? 1u : 0u;
    st.still += (ratio > 0.0 && still) ? 1u : 0u;
    st.redone += redone ? 1u : 0u;
}

// One body of a step kernel: fast path + statistics.  Returns true when the body is flagged for the float64
// re-evaluation; kDefer = false does it on the spot (redo_exact), kDefer = true leaves it to the caller.
// `i` = body index inside the launch (a.pos etc. are the launch's base pointers).
// kSlope (direct kernel only, kDefer = false): the tangent-plane waterline of slope (sx, sy), re-evaluation included.
// kInertia (likewise): the fluid-acceleration loads for a_f = af, re-evaluation included.
template <typename S, int kLayout, int kParam, bool kStats, bool kDefer, bool kWarpSkip = false, bool kSlope = false,
          bool kInertia = false>
__device__ __forceinline__ bool step_one_body(const StepArgs& a, long long i, const BodyIn<double, S>& in, S mass,
                                              const Env& env, S F[3], S T[3], ThreadStats& st, uint32_t& mask,
                                              double sx = 0.0, double sy = 0.0, const double* af = nullptr)
{
    bool clamped, still;
    double ratio;
    bool redo = body_step<S, kWarpSkip, kSlope, kInertia>(in, mass, F, T, clamped, still, ratio, mask, sx, sy, af);
    if (sizeof(S) == 4) {
        redo = redo && a.no_fallback != 1;
        if (a.no_fallback > 1) redo = ((a.first_body + i) & (long long)(a.no_fallback - 1)) == 0;  // study knob: every k-th body, k = 2^j
        if (redo && !kDefer) {
            const ExactStepOut o =
                kInertia ? redo_exact_inertia<kLayout, kParam, kSlope>(a, i, env.surface_z, float(env.cx), float(env.cy),
                                                                       float(env.cz), sx, sy, af)
                : kSlope ? redo_exact_slope<kLayout, kParam>(a, i, env.surface_z, float(env.cx), float(env.cy),
                                                           float(env.cz), sx, sy)
                       : redo_exact<kLayout, kParam>(a, i, env.surface_z, float(env.cx), float(env.cy), float(env.cz));
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                F[k] = S(o.F[k]);
                T[k] = S(o.T[k]);
            }
            ratio = double(o.ratio);
            clamped = (o.flags & 1) != 0;
            still = (o.flags & 2) != 0;
        }
    }
    if (kStats) accumulate_stats(st, double(F[0]), double(F[1]), double(F[2]), ratio, clamped, still, redo);
    return redo;
}

__device__ __forceinline__ double warp_sum(double v)
{
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v)
{
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ unsigned warp_sum_u(unsigned v)
{
    return __reduce_add_sync(0xffffffffu, v);
}

// One atomic set per warp at the very end of a (persistent) kernel.
__device__ __forceinline__ void flush_stats(const ThreadStats& st, double* stats)
{
    const double s = warp_sum(st.sum_f);
    const double m = warp_max(st.max_f);
    const unsigned wet = warp_sum_u(st.wet), cl = warp_sum_u(st.clamped), nf = warp_sum_u(st.nonfinite),
                   sl = warp_sum_u(st.still), nb = warp_sum_u(st.bodies), rd = warp_sum_u(st.redone);
    if ((threadIdx.x & 31) == 0 && nb) {
        atomicAdd(&stats[0], s);
        // max of non-negative doubles == max of their bit patterns
        atomicMax(reinterpret_cast<unsigned long long*>(&stats[1]),
                  static_cast<unsigned long long>(__double_as_longlong(m)));
        atomicAdd(&stats[2], double(wet));
        atomicAdd(&stats[3], double(cl));
        atomicAdd(&stats[4], double(nf));
        atomicAdd(&stats[5], double(sl));
        atomicAdd(&stats[6], double(nb));
        atomicAdd(&stats[7], double(rd));
    }
}

// ---------------------------------------------------------------------------
// Shared-memory tile layout
// ---------------------------------------------------------------------------
template <typename S, int kLayout, int kParam> struct TileLayout {
    // elements (of S) per body for each staged stream
    static constexpr int E_POS = (kLayout == LAYOUT_PHYSX) ? 7 : 3;
    static constexpr int E_QUAT = (kLayout == LAYOUT_PHYSX) ? 0 : 4;
    static constexpr int E_LIN = (kLayout == LAYOUT_SPLIT) ? 3 : 6;
    static constexpr int E_ANG = (kLayout == LAYOUT_SPLIT) ? 3 : 0;
    static constexpr int E_PREV = 6;
    static constexpr int E_COEFF = (kParam == PARAM_PER_BODY) ? N_COEFF : 0;
    static constexpr int E_IN = E_POS + E_QUAT + E_LIN + E_ANG + E_PREV + E_COEFF;
    static constexpr int E_OUT = 3 + 3 + 6;  // force, torque, prev
};

// Bodies the fp32 fast path flags are not re-evaluated on the spot (one lane working for microseconds would
// stall its whole CTA at the next barrier, tile after tile): the lane saves the body index and its OLD
// previous velocities (the tile's bulk store is about to overwrite them) and the CTA re-evaluates all its
// saved bodies at the very end, one per lane in parallel, while its last bulk stores drain, then patches
// force / torque (/ robot wrench) with plain stores.  Measured: profiles/r02_fallback_cost.md.
struct RedoEntry {
    long long body;   // index inside the launch
    float prev[6];    // previous [v, w] as they were before this step
    uint32_t mask;    // submerged-keypoint mask of the fast path (the same H compares body_terms would repeat)
    uint32_t pad_;
};
constexpr int REDO_CAP = 24;  // 24 bodies x 4 roles x 10 doubles of scratch fit the smallest input stage

template <typename S, int kLayout, int kParam, int kThreads, int kStagesIn, int kStagesOut>
struct TileSmem {
    using TL = TileLayout<S, kLayout, kParam>;
    static constexpr size_t IN_BYTES = size_t(TL::E_IN) * kThreads * sizeof(S);
    static constexpr size_t OUT_BYTES = size_t(TL::E_OUT) * kThreads * sizeof(S);
    static constexpr size_t TABLE_BYTES =
        (kParam == PARAM_TABLE) ? (size_t(MAX_TABLE_TYPES) * N_COEFF * sizeof(S) + MAX_TABLE_SLOTS) : 0;
    static constexpr size_t ROBOT_BYTES = size_t(kThreads) * 6 * sizeof(S);  // [3][tile] transferred torques + [3][tile] arms
    static constexpr size_t BAR_BYTES = 16 * sizeof(uint64_t);
    static constexpr size_t REDO_BYTES = 16 + size_t(REDO_CAP) * sizeof(RedoEntry);  // count + deferred re-evaluations
    static constexpr size_t OFF_IN = 0;
    static constexpr size_t OFF_OUT = OFF_IN + kStagesIn * IN_BYTES;
    static constexpr size_t OFF_TABLE = OFF_OUT + kStagesOut * OUT_BYTES;
    static constexpr size_t OFF_ROBOT = (OFF_TABLE + TABLE_BYTES + 15) / 16 * 16;
    static constexpr size_t total(bool robots) { return OFF_ROBOT + (robots ? ROBOT_BYTES : 0) + BAR_BYTES + REDO_BYTES; }
};

// ---------------------------------------------------------------------------
// step_tile_kernel
//
// Persistent CTAs; CTA c handles tiles c, c+grid, ...  Per tile:
//   wait(full[stage]) -> every thread pulls its body's 19(+11) scalars from the stage into
//   registers -> barrier A (stage is free again) -> thread 0 immediately re-arms the stage
//   with the TMA loads of the tile kIn iterations ahead -> compute -> results into an output
//   stage -> fence.proxy.async + barrier C -> thread 0 issues the TMA bulk stores.
// Releasing the input stage before the arithmetic means even a single stage overlaps the
// next tile's loads with this tile's compute, which keeps shared memory per CTA small and
// lets many CTAs share an SM (the kernel is issue-bound, so resident warps matter).
// ---------------------------------------------------------------------------
// Bodies per tile when the robot size is a compile-time constant: whole robots AND whole 16-byte
// granules (4 fp32 / 2 fp64 bodies), as many as fit the CTA.  Mirrors tile_bodies_for() on the host.
constexpr int tile_gcd(int a, int b) { return b ? tile_gcd(b, a % b) : a; }
constexpr int tile_bodies_static(int threads, int esz, int bpr)
{
    const int granule = 16 / esz;
    const int unit = granule / tile_gcd(granule, bpr) * bpr;
    return threads / unit * unit;
}

// kBpr > 0 specialises robot mode for one robot size (19 = the SILVER2 hexapod): tile size, robot index
// and the per-robot sums become compile-time (-8 % time on the C4 shard); 0 = any size at run time.
template <typename S, int kLayout, int kParam, bool kRobot, bool kStats, int kThreads, int kStagesIn,
          int kStagesOut, int kMinBlocks, bool kCopyOnly = false, int kBpr = 0>
__global__ void __launch_bounds__(kThreads, kMinBlocks) step_tile_kernel(const __grid_constant__ StepArgs a)
{
    using TL = TileLayout<S, kLayout, kParam>;
    using SM = TileSmem<S, kLayout, kParam, kThreads, kStagesIn, kStagesOut>;
    extern __shared__ __align__(128) unsigned char smem[];

    const int tid = threadIdx.x;
    // bodies per tile: whole robots (<= kThreads) in robot mode, else every lane has a body
    static_assert(kThreads % 4 == 0, "a full tile must keep every bulk copy a 16-byte multiple");
    static_assert(kBpr == 0 || kRobot, "kBpr only applies to robot mode");
    const int TB = kRobot ? (kBpr > 0 ? tile_bodies_static(kThreads, int(sizeof(S)), kBpr > 0 ? kBpr : 1) : a.tile_bodies) : kThreads;
    S* const table = reinterpret_cast<S*>(smem + SM::OFF_TABLE);
    unsigned char* const slot_map = smem + SM::OFF_TABLE + size_t(MAX_TABLE_TYPES) * N_COEFF * sizeof(S);
    S* const robot_acc = reinterpret_cast<S*>(smem + SM::OFF_ROBOT);
    uint64_t* const full_bar =
        reinterpret_cast<uint64_t*>(smem + SM::OFF_ROBOT + (kRobot ? SM::ROBOT_BYTES : 0));
    int* const redo_count = reinterpret_cast<int*>(smem + SM::OFF_ROBOT + (kRobot ? SM::ROBOT_BYTES : 0) + SM::BAR_BYTES);
    RedoEntry* const redo_list = reinterpret_cast<RedoEntry*>(reinterpret_cast<unsigned char*>(redo_count) + 16);

    // per-stream byte sizes of one full tile and offsets inside a stage
    const uint32_t b_pos = uint32_t(TL::E_POS) * TB * sizeof(S);
    const uint32_t b_quat = uint32_t(TL::E_QUAT) * TB * sizeof(S);
    const uint32_t b_lin = uint32_t(TL::E_LIN) * TB * sizeof(S);
    const uint32_t b_ang = uint32_t(TL::E_ANG) * TB * sizeof(S);
    const uint32_t b_prev = uint32_t(TL::E_PREV) * TB * sizeof(S);
    // stage layout is fixed by the largest tile; partial tiles just copy fewer bytes per stream
    const uint32_t o_quat = b_pos, o_lin = o_quat + b_quat, o_ang = o_lin + b_lin, o_prev = o_ang + b_ang,
                   o_coeff = o_prev + b_prev;
    const uint32_t oo_t = 3u * TB * sizeof(S), oo_prev = 2 * oo_t;

    if (tid == 0) {
        for (int s = 0; s < kStagesIn; ++s) mbar_init(&full_bar[s], 1);
        mbar_fence_init();
        fence_proxy_async_smem();
        redo_count[0] = 0;  // deferred entries
        redo_count[1] = 0;  // overflow in the current tile
    }

    // Tile schedule: full tiles dealt round-robin (tile = cta + it*grid).  At any moment the resident
    // CTAs stream one compact window of every array, which is what DRAM pages and the TLB like.
    // Measured alternatives (profiles/r01_sweep_schedules.log): one contiguous share per CTA costs
    // ~10 % of the bandwidth; splitting the ragged last round evenly over all CTAs is ~0.8 us slower.
    // The ragged extra tiles go to the lowest blockIdx values: those CTAs become resident first when this grid
    // starts in the slots of a draining predecessor (overlap mode), so the extra round evens out.
    const int n_it = (a.n_tiles > int(blockIdx.x)) ? (a.n_tiles - int(blockIdx.x) + int(gridDim.x) - 1) / int(gridDim.x) : 0;
    // Overlap mode: the first tile is loaded, computed and stored while the previous grid may still run; the wait
    // (and only then the trigger for the next grid) follows it.  Otherwise wait before the first global access.
    const bool early = a.overlap && n_it > 0;
    if (!early) {
        pdl_wait_prerequisites();
        pdl_launch_dependents();
    }
    const long long round_stride = (long long)gridDim.x * TB;
    const long long first_begin = (long long)blockIdx.x * TB;
    auto tile_start = [&](int it) -> long long { return first_begin + it * round_stride; };
    auto issue_loads = [&](int it, int stage) {
        unsigned char* dst = smem + SM::OFF_IN + size_t(stage) * SM::IN_BYTES;
        const long long b0 = tile_start(it);
        const uint32_t cb = uint32_t(TB) * sizeof(S);  // bytes per body-scalar column
        uint64_t* bar = &full_bar[stage];
        mbar_arrive_expect_tx(bar, cb * TL::E_IN);
        bulk_g2s(dst, reinterpret_cast<const S*>(a.pos) + b0 * TL::E_POS, cb * TL::E_POS, bar);
        if (TL::E_QUAT) bulk_g2s(dst + o_quat, reinterpret_cast<const S*>(a.quat) + b0 * TL::E_QUAT, cb * TL::E_QUAT, bar);
        bulk_g2s(dst + o_lin, reinterpret_cast<const S*>(a.lin) + b0 * TL::E_LIN, cb * TL::E_LIN, bar);
        if (TL::E_ANG) bulk_g2s(dst + o_ang, reinterpret_cast<const S*>(a.ang) + b0 * TL::E_ANG, cb * TL::E_ANG, bar);
        bulk_g2s(dst + o_prev, reinterpret_cast<const S*>(a.prev) + b0 * TL::E_PREV, cb * TL::E_PREV, bar);
        if (TL::E_COEFF)
            bulk_g2s(dst + o_coeff, reinterpret_cast<const S*>(a.coeff) + b0 * TL::E_COEFF, cb * TL::E_COEFF, bar);
    };

    if (tid == 0) {  // prologue: arm every input stage
        for (int j = 0; j < kStagesIn; ++j)
            if (j < n_it) issue_loads(j, j);
    }
    // the part-type table is staged AFTER the first tile's bulk loads are in flight: its global-load
    // latency hides behind theirs (a one-tile-per-CTA launch like C2 is nothing but latencies)
    if (kParam == PARAM_TABLE) {
        const S* g = reinterpret_cast<const S*>(a.coeff);
        for (int i = tid; i < a.n_types * N_COEFF; i += kThreads) table[i] = g[i];
        for (int i = tid; i < a.n_slots; i += kThreads) slot_map[i] = static_cast<unsigned char>(a.slot_type[i]);
    }
    __syncthreads();  // table staged, mbarriers initialised

    ThreadStats st;
    const S inv_dt = S(a.inv_dt);
    const Env env{a.current[0], a.current[1], a.current[2], a.surface_z};
    const int bpr = kBpr > 0 ? kBpr : a.bodies_per_robot;

    long long next_begin = first_begin;
    for (int it = 0; it < n_it; ++it) {
        const int stage = it % kStagesIn;
        const int ostage = it % kStagesOut;
        const int cnt = TB;
        const long long tile_begin = next_begin;
        next_begin += round_stride;
        const bool active = kRobot ? tid < cnt : true;
        const int robots_in_tile = kRobot ? cnt / bpr : 0;
        mbar_wait(&full_bar[stage], (it / kStagesIn) & 1);

        const unsigned char* in = smem + SM::OFF_IN + size_t(stage) * SM::IN_BYTES;
        BodyPtrs<S> bp;
        bp.pos = reinterpret_cast<const S*>(in);
        bp.quat = reinterpret_cast<const S*>(in + o_quat);
        bp.lin = reinterpret_cast<const S*>(in + o_lin);
        bp.ang = reinterpret_cast<const S*>(in + o_ang);
        bp.prev = reinterpret_cast<const S*>(in + o_prev);
        bp.coeff = reinterpret_cast<const S*>(in + o_coeff);

        RawBody<S> r;
        S cl[N_COEFF];
        S* const arm_scratch = robot_acc + 3 * kThreads;  // (p_i - p_base), parked across the arithmetic
        if (active) {
            load_raw<S, kLayout>(bp, tid, r);
            const S* c;
            if (kParam == PARAM_PER_BODY) {
                c = bp.coeff + N_COEFF * tid;
            } else {
                int slot = 0;
                if (a.n_slots > 1) {
                    const int base_mod = int((a.first_body + tile_begin) % a.n_slots);
                    slot = (base_mod + tid) % a.n_slots;
                }
                c = table + N_COEFF * int(slot_map[slot]);
            }
#pragma unroll
            for (int k = 0; k < N_COEFF; ++k) cl[k] = c[k];
            if (kRobot) {
                // arm to the robot's slot-0 body; goes through shared memory instead of living in
                // three registers across the whole model (register budget for 5 CTAs/SM)
                const S* pb = bp.pos + TL::E_POS * ((tid / bpr) * bpr);
                arm_scratch[0 * kThreads + tid] = r.px - pb[0];
                arm_scratch[1 * kThreads + tid] = r.py - pb[1];
                arm_scratch[2 * kThreads + tid] = r.pz - pb[2];
            }
        }
        // the bulk store that last used this output stage must have finished reading it
        if (tid == 0) bulk_wait_read<kStagesOut - 1>();
        __syncthreads();  // (A) input stage consumed, output stage free
        if (tid == 0 && it + kStagesIn < n_it) issue_loads(it + kStagesIn, stage);

        S F[3] = {S(0), S(0), S(0)}, T[3] = {S(0), S(0), S(0)};
        unsigned char* out = smem + SM::OFF_OUT + size_t(ostage) * SM::OUT_BYTES;
        bool overflowed = false;  // flagged, but the CTA's list is full
        if (active) {
            if (kCopyOnly) {
                // measurement aid (tile configs 10/11): same memory traffic, no arithmetic
                F[0] = r.px + cl[0]; F[1] = r.py + cl[3]; F[2] = r.pz + cl[6];
                T[0] = r.q0 + cl[9]; T[1] = r.q1 + r.q2 + r.pvx + r.pvz; T[2] = r.q3 + cl[10] + r.pwy;
            } else {
                BodyIn<double, S> bin;
                make_body_in<S>(r, cl, a.quat_wxyz, a.rho, a.grav, inv_dt, env, bin);
                uint32_t kp_mask;
                // robot mode (fleets: usually every body of a warp is fully submerged) skips the keypoint compares warp-wide;
                // its CTAs run under a 96-register cap, the 80-register default kernel would spill on the branch
                if (step_one_body<S, kLayout, kParam, kStats, true, (kRobot || H2O_SKIP_ALL)>(a, tile_begin + tid, bin, cl[10], env, F, T, st, kp_mask)) {
                    if (sizeof(S) == 4) {
                        const long long bi = tile_begin + tid;
                        const int slot = atomicAdd(redo_count, 1);
                        if (slot < REDO_CAP) {  // prev[bi] in global memory is still the old row: this tile's store comes later
                            const float2* pr = reinterpret_cast<const float2*>(reinterpret_cast<const float*>(a.prev) + 6 * bi);
                            const float2 p0 = pr[0], p1 = pr[1], p2 = pr[2];
                            // keep the body's rows L2-resident until the CTA gets to it (the batch is larger
                            // than the L2: by then they would come from HBM again, ~1 us of the tail)
                            prefetch_l2_keep(reinterpret_cast<const S*>(a.pos) + TL::E_POS * bi);
                            if (TL::E_QUAT) prefetch_l2_keep(reinterpret_cast<const S*>(a.quat) + TL::E_QUAT * bi);
                            prefetch_l2_keep(reinterpret_cast<const S*>(a.lin) + TL::E_LIN * bi);
                            if (TL::E_ANG) prefetch_l2_keep(reinterpret_cast<const S*>(a.ang) + TL::E_ANG * bi);
                            if (TL::E_COEFF) prefetch_l2_keep(reinterpret_cast<const S*>(a.coeff) + TL::E_COEFF * bi);
                            RedoEntry& en = redo_list[slot];
                            en.body = bi;
                            en.mask = kp_mask;
                            en.prev[0] = p0.x; en.prev[1] = p0.y; en.prev[2] = p1.x;
                            en.prev[3] = p1.y; en.prev[4] = p2.x; en.prev[5] = p2.y;
                        } else {  // list full (a workload that flags bodies wholesale): see below
                            overflowed = true;
                        }
                    }
                }
            }

            using V2 = typename Vec2Of<S>::type;
            S* of = reinterpret_cast<S*>(out) + 3 * tid;
            S* ot = reinterpret_cast<S*>(out + oo_t) + 3 * tid;
            of[0] = F[0]; of[1] = F[1]; of[2] = F[2];
            ot[0] = T[0]; ot[1] = T[1]; ot[2] = T[2];
            V2* op = reinterpret_cast<V2*>(reinterpret_cast<S*>(out + oo_prev) + 6 * tid);
            V2 v;
            v.x = r.vx; v.y = r.vy; op[0] = v;
            v.x = r.vz; v.y = r.wx; op[1] = v;
            v.x = r.wy; v.y = r.wz; op[2] = v;
            if (sizeof(S) == 4 && overflowed) {
                // No slot in the deferred list: mark the body in the engine's bitmap and keep its OLD previous
                // velocities in global memory (stage them instead of v), so that the sweep at the end of this
                // CTA can re-evaluate it from global memory alone; it then writes the new row itself.  No call
                // in here: a call inside the tile loop costs the hot path its registers (measured).
                const long long gi = a.first_body + tile_begin + tid;
                atomicOr(a.redo_bitmap + (gi >> 5), 1u << (gi & 31));
                redo_count[1] = 1;
                const V2* pr = reinterpret_cast<const V2*>(reinterpret_cast<const S*>(a.prev) + 6 * (tile_begin + tid));
                op[0] = pr[0]; op[1] = pr[1]; op[2] = pr[2];
            }
        }
        if (kRobot && active) {
            // torque of body i about the robot's slot-0 body: tau_i + (p_i - p_base) x F_i, parked in
            // shared memory ([component][body]) next to the forces already sitting in the output stage
            const S ax = arm_scratch[0 * kThreads + tid], ay = arm_scratch[1 * kThreads + tid],
                    az = arm_scratch[2 * kThreads + tid];
            robot_acc[0 * TB + tid] = T[0] + (ay * F[2] - az * F[1]);
            robot_acc[1 * TB + tid] = T[1] + (az * F[0] - ax * F[2]);
            robot_acc[2 * TB + tid] = T[2] + (ax * F[1] - ay * F[0]);
        }
        fence_proxy_async_smem();
        __syncthreads();  // (C) results (and robot accumulators) complete
        if (tid == 0) {
            const uint32_t cb = uint32_t(cnt) * sizeof(S);
            bulk_s2g(reinterpret_cast<S*>(a.out_force) + tile_begin * 3, out, cb * 3);
            bulk_s2g(reinterpret_cast<S*>(a.out_torque) + tile_begin * 3, out + oo_t, cb * 3);
            bulk_s2g(reinterpret_cast<S*>(a.prev) + tile_begin * 6, out + oo_prev, cb * 6);
            bulk_commit();
        }
        if (kRobot) {
            // Per-robot net wrench: thread (robot, component) sums its robot's bodies straight out of
            // shared memory in body order (deterministic; bank-conflict free for the strides involved).
            // Measured on the C4 shard (profiles/r01_robot_wrench_variants.log): segmented warp-shuffle
            // scan over all lanes + shared-memory atomics 80 us, this 68 us, lane pairs + shuffle 72 us.
            // The scratch is rewritten only after the next tile's barrier (A), which these threads
            // reach after the sum.  (robot_wrench_kernel -- tails, robots larger than a tile -- reduces
            // one robot per warp with shuffles.)  Robots of fewer than 6 bodies have more (robot,
            // component) sums than the tile has threads, hence the stride loop.
            for (int idx = tid; idx < robots_in_tile * 6; idx += kThreads) {
                const int rb = idx / 6, c = idx - 6 * rb;
                const S* src = (c < 3) ? reinterpret_cast<const S*>(out) + 3 * (rb * bpr) + c
                                       : robot_acc + (c - 3) * TB + rb * bpr;
                const int step = (c < 3) ? 3 : 1;
                S sum = S(0);
                if (kBpr > 0) {  // loads first, then the adds in body order
                    S v[kBpr > 0 ? kBpr : 1];
#pragma unroll
                    for (int j = 0; j < kBpr; ++j) v[j] = src[j * step];
#pragma unroll
                    for (int j = 0; j < kBpr; ++j) sum += v[j];
                } else {
#pragma unroll 4
                    for (int j = 0; j < bpr; ++j) sum += src[j * step];
                }
                reinterpret_cast<S*>(a.out_wrench)[(tile_begin / bpr) * 6 + idx] = sum;
            }
        }
        if (early && it == 0) {
            pdl_wait_prerequisites();
            pdl_launch_dependents();
        }
    }
    if (sizeof(S) == 4 && !kCopyOnly) {
        __syncthreads();  // every tile done: the list is complete, every bulk store has been issued
        const int n_redo = redo_count[0] < REDO_CAP ? redo_count[0] : REDO_CAP;
        const bool sweep = redo_count[1] != 0;
        auto patch = [&](long long bi, const ExactStepOut& o) {  // replace a body's fast-path force / torque
            float* of = reinterpret_cast<float*>(a.out_force) + 3 * bi;
            float* ot = reinterpret_cast<float*>(a.out_torque) + 3 * bi;
            if (kRobot) {
                // the per-robot sums were formed from the fast-path values: add the difference
                constexpr int EP = TL::E_POS;
                const float* pos = reinterpret_cast<const float*>(a.pos);
                const long long rb = bi / bpr;
                const float* pb = pos + EP * (rb * bpr);
                const float* pi = pos + EP * bi;
                const float ax = pi[0] - pb[0], ay = pi[1] - pb[1], az = pi[2] - pb[2];
                const float dfx = o.F[0] - of[0], dfy = o.F[1] - of[1], dfz = o.F[2] - of[2];
                float* ow = reinterpret_cast<float*>(a.out_wrench) + rb * 6;
                atomicAdd(ow + 0, dfx); atomicAdd(ow + 1, dfy); atomicAdd(ow + 2, dfz);
                atomicAdd(ow + 3, (o.T[0] - ot[0]) + (ay * dfz - az * dfy));
                atomicAdd(ow + 4, (o.T[1] - ot[1]) + (az * dfx - ax * dfz));
                atomicAdd(ow + 5, (o.T[2] - ot[2]) + (ax * dfy - ay * dfx));
            }
            of[0] = o.F[0]; of[1] = o.F[1]; of[2] = o.F[2];
            ot[0] = o.T[0]; ot[1] = o.T[1]; ot[2] = o.T[2];
        };
        if (n_redo > 0) {  // CTA-uniform
            // scratch = the input stage (no load is in flight any more): [entry][role][ROLE_DOUBLES] doubles
            double* const scratch = reinterpret_cast<double*>(smem + SM::OFF_IN);
            static_assert(size_t(REDO_CAP) * N_ROLES * ROLE_DOUBLES * sizeof(double) <= SM::IN_BYTES || sizeof(S) != 4,
                          "re-evaluation scratch must fit the input stage");
            const int warp = tid >> 5, lane = tid & 31, n_warps = kThreads / 32;
            for (int role = warp; role < N_ROLES; role += n_warps)
                if (lane < n_redo)
                    redo_role<kLayout, kParam>(role, a, redo_list[lane].body, env.surface_z, redo_list[lane].prev,
                                               redo_list[lane].mask, scratch + (lane * N_ROLES + role) * ROLE_DOUBLES);
            __syncthreads();
            ExactStepOut o;
            if (tid < n_redo) o = combine_roles(scratch + tid * N_ROLES * ROLE_DOUBLES);
            if (tid == 0) bulk_wait_all<0>();  // the fast-path values of these bodies have landed ...
            __syncthreads();
            if (tid < n_redo) patch(redo_list[tid].body, o);  // ... and are replaced
        } else {
            // Nothing to patch: the CTA may retire as soon as the bulk stores have READ their shared-memory
            // source (the writes drain on their own; grid completion orders them before the next kernel) --
            // ~0.5 us less tail than waiting for the writes themselves.
            if (tid == 0) {
                if (sweep) bulk_wait_all<0>();
                else bulk_wait_read<0>();
            }
            if (sweep) __syncthreads();
        }
        if (sweep) {
            // The list overflowed in some tile: sweep this CTA's tiles for marked bodies.  Their previous
            // velocities in global memory are still the old ones; after the float64 evaluation the thread
            // writes force, torque and the new row, and clears the mark (the bitmap is all zero again).
            for (int it = 0; it < n_it; ++it) {
                const long long bi = tile_start(it) + tid;
                const long long gi = a.first_body + bi;
                if (tid < TB && ((a.redo_bitmap[gi >> 5] >> (gi & 31)) & 1u)) {
                    const ExactStepOut o = redo_exact<kLayout, kParam>(a, bi, env.surface_z, float(a.current[0]),
                                                                       float(a.current[1]), float(a.current[2]));
                    patch(bi, o);
                    BodyPtrs<float> bp;
                    bp.pos = reinterpret_cast<const float*>(a.pos); bp.quat = reinterpret_cast<const float*>(a.quat);
                    bp.lin = reinterpret_cast<const float*>(a.lin); bp.ang = reinterpret_cast<const float*>(a.ang);
                    bp.prev = reinterpret_cast<const float*>(a.prev); bp.coeff = nullptr;
                    RawBody<float> rr;
                    load_raw<float, kLayout>(bp, bi, rr);
                    float* pv = reinterpret_cast<float*>(a.prev) + 6 * bi;
                    pv[0] = rr.vx; pv[1] = rr.vy; pv[2] = rr.vz; pv[3] = rr.wx; pv[4] = rr.wy; pv[5] = rr.wz;
                    atomicAnd(a.redo_bitmap + (gi >> 5), ~(1u << (gi & 31)));
                }
            }
        }
    } else if (tid == 0) {
        bulk_wait_read<0>();
    }
    if (kStats && a.stats) flush_stats(st, a.stats);
}

// ---------------------------------------------------------------------------
// step_direct_kernel: one thread per body, plain global loads/stores.
// Processes bodies [body_begin, n).  Robot wrench (if requested) is produced by
// robot_wrench_kernel below from the written force/torque arrays.
// Dynamic shared memory: wave_smem_bytes(w.n) (the wave table and the clock value; 0 without waves).
// ---------------------------------------------------------------------------
inline size_t wave_smem_bytes(int n_waves) { return n_waves > 0 ? (size_t(n_waves) * WAVE_STRIDE + 1) * sizeof(double) : 0; }

// Every thread of the CTA: stage the wave table, then the clock value behind it; the caller synchronises.
__device__ __forceinline__ void stage_waves(double* dst, const double* tab, const double* clock, int n_waves)
{
    for (int k = threadIdx.x; k < n_waves * WAVE_STRIDE; k += blockDim.x) dst[k] = tab[k];
    if (threadIdx.x == 0) dst[n_waves * WAVE_STRIDE] = *clock;
}

// kSlope (h2o_set_wave_slope, launched only with a wave field): every body is tested against the tangent plane of the
// wave surface at its position (body_terms / body_wrench_fast), on every path below.
// kInertia (h2o_set_fluid_inertia, launched only with a wave field or a grid with nt > 1, never with Warp
// compatibility): the fluid-acceleration loads for the a_f water_at forms at the body centre, on every path below.
template <typename S, int kLayout, int kParam, bool kStats, bool kSlope = false, bool kInertia = false>
__global__ void __launch_bounds__(256) step_direct_kernel(const __grid_constant__ StepArgs a, long long body_begin,
                                                          const __grid_constant__ WaveArgs wv,
                                                          const __grid_constant__ EnvArgs ev,
                                                          const __grid_constant__ GridArgs gv)
{
    __shared__ S table[(kParam == PARAM_TABLE) ? MAX_TABLE_TYPES * N_COEFF : 1];
    __shared__ unsigned char slot_map[(kParam == PARAM_TABLE) ? MAX_TABLE_SLOTS : 1];
    extern __shared__ double wave_smem[];
    pdl_wait_prerequisites();  // returns at once (plain launch); the trigger lets a following tile launch start early
    pdl_launch_dependents();
    if (wv.n) {
        stage_waves(wave_smem, wv.tab, wv.clock, wv.n);
        __syncthreads();
    }
    if (kParam == PARAM_TABLE) {
        const S* g = reinterpret_cast<const S*>(a.coeff);
        for (int i = threadIdx.x; i < a.n_types * N_COEFF; i += blockDim.x) table[i] = g[i];
        for (int i = threadIdx.x; i < a.n_slots; i += blockDim.x)
            slot_map[i] = static_cast<unsigned char>(a.slot_type[i]);
        __syncthreads();
    }
    ThreadStats st;
    const long long i = body_begin + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.n) {
        BodyPtrs<S> bp;
        bp.pos = reinterpret_cast<const S*>(a.pos);
        bp.quat = reinterpret_cast<const S*>(a.quat);
        bp.lin = reinterpret_cast<const S*>(a.lin);
        bp.ang = reinterpret_cast<const S*>(a.ang);
        bp.prev = reinterpret_cast<const S*>(a.prev);
        bp.coeff = reinterpret_cast<const S*>(a.coeff);
        RawBody<S> r;
        load_raw<S, kLayout>(bp, i, r);
        S cl[N_COEFF];
        if (kParam == PARAM_PER_BODY) {
#pragma unroll
            for (int k = 0; k < N_COEFF; ++k) cl[k] = __ldg(bp.coeff + N_COEFF * i + k);
        } else {
            const S* c = table + N_COEFF * int(slot_map[int((a.first_body + i) % a.n_slots)]);
#pragma unroll
            for (int k = 0; k < N_COEFF; ++k) cl[k] = c[k];
        }
        BodyIn<double, S> bin;
        Env env{a.current[0], a.current[1], a.current[2], a.surface_z};
        double slope[2] = {0.0, 0.0};
        double af[3] = {0.0, 0.0, 0.0};
        if (wv.n || ev.cond || gv.vals) {
            EnvRow row{};
            if (ev.cond) row = env_row(ev.cond, (a.first_body + i) / ev.bodies_per_env);
            // the clock: staged with the wave table, else read directly when only the grid needs it
            const double t = wv.n ? wave_smem[wv.n * WAVE_STRIDE] : (gv.vals ? *wv.clock : 0.0);
            if constexpr (kInertia) {
                const WaterAccel wa = water_at<sizeof(S) == 4, kSlope, true>(
                    a.current, a.surface_z, ev.cond != nullptr, row, wave_smem, wv.n, wv.depth, t, double(r.px),
                    double(r.py), double(r.pz), gv.vals ? &gv : nullptr);
                env = Env{wa.water.cx, wa.water.cy, wa.water.cz, wa.water.surface_z};
                slope[0] = wa.sx;
                slope[1] = wa.sy;
                af[0] = wa.ax; af[1] = wa.ay; af[2] = wa.az;
            } else if constexpr (kSlope) {
                const WaterSlope ws = water_at<sizeof(S) == 4, true>(a.current, a.surface_z, ev.cond != nullptr, row,
                                                                     wave_smem, wv.n, wv.depth, t, double(r.px),
                                                                     double(r.py), double(r.pz), gv.vals ? &gv : nullptr);
                env = Env{ws.water.cx, ws.water.cy, ws.water.cz, ws.water.surface_z};
                slope[0] = ws.sx;
                slope[1] = ws.sy;
            } else {
                const Water w = water_at<sizeof(S) == 4>(a.current, a.surface_z, ev.cond != nullptr, row, wave_smem,
                                                         wv.n, wv.depth, t, double(r.px), double(r.py), double(r.pz),
                                                         gv.vals ? &gv : nullptr);
                env = Env{w.cx, w.cy, w.cz, w.surface_z};
            }
        }
        if (a.surface_eta) env.surface_z += double(reinterpret_cast<const S*>(a.surface_eta)[i]);
        make_body_in<S>(r, cl, a.quat_wxyz, a.rho, a.grav, S(a.inv_dt), env, bin);
        if (a.am_dense)
            bin.am_dense = reinterpret_cast<const S*>(a.am_dense) + 36 * a.am_slot_type[(a.first_body + i) % a.am_n_slots];
        S F[3], T[3];
        uint32_t kp_mask;
        bin.warp_compat = a.warp_compat != 0;  // fp64 mode: body_terms honours it
        if (!kInertia && sizeof(S) == 4 && a.warp_compat) {
            // fp32 mode, Warp-twin semantics: the float64 world-frame formulation for every body (compatibility
            // mode, not a fast path: body_wrench_fast knows only the Numba semantics)
            RawBody<float> rf;
            rf.px = float(r.px); rf.py = float(r.py); rf.pz = float(r.pz);
            rf.q0 = float(r.q0); rf.q1 = float(r.q1); rf.q2 = float(r.q2); rf.q3 = float(r.q3);
            rf.vx = float(r.vx); rf.vy = float(r.vy); rf.vz = float(r.vz);
            rf.wx = float(r.wx); rf.wy = float(r.wy); rf.wz = float(r.wz);
            rf.pvx = float(r.pvx); rf.pvy = float(r.pvy); rf.pvz = float(r.pvz);
            rf.pwx = float(r.pwx); rf.pwy = float(r.pwy); rf.pwz = float(r.pwz);
            float cf[N_COEFF];
#pragma unroll
            for (int k = 0; k < N_COEFF; ++k) cf[k] = float(cl[k]);
            const ExactStepOut o =
                kSlope ? body_step_exact_f32_slope(rf, cf, a.quat_wxyz, a.rho, a.grav, a.inv_dt, env.surface_z,
                                                   float(env.cx), float(env.cy), float(env.cz), slope[0], slope[1], true)
                       : body_step_exact_f32(rf, cf, a.quat_wxyz, a.rho, a.grav, a.inv_dt, env.surface_z,
                                             float(env.cx), float(env.cy), float(env.cz), true);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                F[k] = S(o.F[k]);
                T[k] = S(o.T[k]);
            }
            if (kStats) accumulate_stats(st, double(F[0]), double(F[1]), double(F[2]), double(o.ratio), (o.flags & 1) != 0,
                                         (o.flags & 2) != 0, true);
        } else {
            step_one_body<S, kLayout, kParam, kStats, false, false, kSlope, kInertia>(a, i, bin, cl[10], env, F, T, st,
                                                                                      kp_mask, slope[0], slope[1], af);
        }
        S* of = reinterpret_cast<S*>(a.out_force) + 3 * i;
        S* ot = reinterpret_cast<S*>(a.out_torque) + 3 * i;
        of[0] = F[0]; of[1] = F[1]; of[2] = F[2];
        ot[0] = T[0]; ot[1] = T[1]; ot[2] = T[2];
        using V2 = typename Vec2Of<S>::type;
        V2* op = reinterpret_cast<V2*>(reinterpret_cast<S*>(a.prev) + 6 * i);
        V2 v;
        v.x = r.vx; v.y = r.vy; op[0] = v;
        v.x = r.vz; v.y = r.wx; op[1] = v;
        v.x = r.wy; v.y = r.wz; op[2] = v;
    }
    if (kStats && a.stats) flush_stats(st, a.stats);
}

// Robot wrench from written force/torque arrays for robots [robot_begin, n_robots):
// one warp per robot, lanes stride over its bodies, shuffle reduction.
template <typename S, int kLayout>
__global__ void __launch_bounds__(256) robot_wrench_kernel(const __grid_constant__ StepArgs a, long long robot_begin)
{
    const long long robot = robot_begin + ((long long)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const int lane = threadIdx.x & 31;
    const long long n_robots = a.robot_offsets ? a.n_robots_var : a.n / a.bodies_per_robot;
    if (robot >= n_robots) return;
    constexpr int EP = (kLayout == LAYOUT_PHYSX) ? 7 : 3;
    const S* pos = reinterpret_cast<const S*>(a.pos);
    const S* Fp = reinterpret_cast<const S*>(a.out_force);
    const S* Tp = reinterpret_cast<const S*>(a.out_torque);
    const long long b0 = a.robot_offsets ? a.robot_offsets[robot] : robot * a.bodies_per_robot;
    const long long cnt = a.robot_offsets ? a.robot_offsets[robot + 1] - b0 : a.bodies_per_robot;
    const double bx = double(pos[EP * b0]), by = double(pos[EP * b0 + 1]), bz = double(pos[EP * b0 + 2]);
    double v[6] = {0, 0, 0, 0, 0, 0};
    for (long long j = lane; j < cnt; j += 32) {
        const long long i = b0 + j;
        const double fx = double(Fp[3 * i]), fy = double(Fp[3 * i + 1]), fz = double(Fp[3 * i + 2]);
        const double ax = double(pos[EP * i]) - bx, ay = double(pos[EP * i + 1]) - by,
                     az = double(pos[EP * i + 2]) - bz;
        v[0] += fx; v[1] += fy; v[2] += fz;
        v[3] += double(Tp[3 * i]) + (ay * fz - az * fy);
        v[4] += double(Tp[3 * i + 1]) + (az * fx - ax * fz);
        v[5] += double(Tp[3 * i + 2]) + (ax * fy - ay * fx);
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) v[c] = warp_sum(v[c]);
    if (lane == 0) {
        S* ow = reinterpret_cast<S*>(a.out_wrench) + robot * 6;
#pragma unroll
        for (int c = 0; c < 6; ++c) ow[c] = S(v[c]);
    }
}

// ---------------------------------------------------------------------------
// components_kernel: batched solve_hydrodynamics (numba_hydrodynamics.py:255-314),
// reference output order: buoyancy_force, drag_force, lift_force, drag_torque,
// added_mass_force, added_mass_torque, center_of_buoyancy, center_of_pressure, sub_ratio.
// cob/cop are returned in world coordinates like the reference (zeros when dry).
// ---------------------------------------------------------------------------
struct ComponentsArgs {
    const void *pos, *quat, *lin, *ang, *lin_acc, *ang_acc;
    const void* coeff;
    const int32_t* slot_type;
    void* out[8];     // eight (N,3) arrays
    void* out_ratio;  // (N,)
    int32_t* out_flags;  // (N,) bit0 = "reference raises" (wet, speed <= 1e-6), may be null
    long long n, first_body;
    int n_slots, n_types, param_mode, quat_wxyz;
    int warp_compat;  // reproduce the deviations of the reference's Warp twin (SURVEY.md Appendix C)
    double rho, grav;
    double current[3], surface_z;
};

template <typename S>
__global__ void __launch_bounds__(256) components_kernel(const __grid_constant__ ComponentsArgs a)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const S* c;
    if (a.param_mode == PARAM_PER_BODY) c = reinterpret_cast<const S*>(a.coeff) + N_COEFF * i;
    else c = reinterpret_cast<const S*>(a.coeff) + N_COEFF * a.slot_type[(a.first_body + i) % a.n_slots];
    RawBody<S> r;
    const S* p = reinterpret_cast<const S*>(a.pos) + 3 * i;
    const S* q = reinterpret_cast<const S*>(a.quat) + 4 * i;
    const S* v = reinterpret_cast<const S*>(a.lin) + 3 * i;
    const S* w = reinterpret_cast<const S*>(a.ang) + 3 * i;
    const S* la = reinterpret_cast<const S*>(a.lin_acc) + 3 * i;
    const S* aa = reinterpret_cast<const S*>(a.ang_acc) + 3 * i;
    r.px = p[0]; r.py = p[1]; r.pz = p[2];
    r.q0 = q[0]; r.q1 = q[1]; r.q2 = q[2]; r.q3 = q[3];
    r.vx = v[0]; r.vy = v[1]; r.vz = v[2];
    r.wx = w[0]; r.wy = w[1]; r.wz = w[2];
    r.pvx = r.vx; r.pvy = r.vy; r.pvz = r.vz; r.pwx = r.wx; r.pwy = r.wy; r.pwz = r.wz;
    BodyIn<double, S> in;
    make_body_in<S>(r, c, a.quat_wxyz, a.rho, a.grav, S(0), Env{a.current[0], a.current[1], a.current[2], a.surface_z}, in);
    in.ax = la[0]; in.ay = la[1]; in.az = la[2];
    in.bx = aa[0]; in.by = aa[1]; in.bz = aa[2];
    in.acc_scale = S(1);
    in.warp_compat = a.warp_compat != 0;
    Terms<double, S> t;
    body_terms<double, S, false>(in, t);
    // Numba: a dry body returns zeros everywhere, cob/cop included (numba_hydrodynamics.py:277-279);
    // the Warp twin returns cob = cop = position (warp_hydrodynamics.py:59-61, :290)
    const bool wet = t.ratio > 0.0 || a.warp_compat != 0;
    S* o;
    o = reinterpret_cast<S*>(a.out[0]) + 3 * i; o[0] = S(0); o[1] = S(0); o[2] = S(t.fbz);
    o = reinterpret_cast<S*>(a.out[1]) + 3 * i; o[0] = t.fd[0]; o[1] = t.fd[1]; o[2] = t.fd[2];
    o = reinterpret_cast<S*>(a.out[2]) + 3 * i; o[0] = t.fl[0]; o[1] = t.fl[1]; o[2] = t.fl[2];
    o = reinterpret_cast<S*>(a.out[3]) + 3 * i; o[0] = t.td[0]; o[1] = t.td[1]; o[2] = t.td[2];
    o = reinterpret_cast<S*>(a.out[4]) + 3 * i; o[0] = t.fam[0]; o[1] = t.fam[1]; o[2] = t.fam[2];
    o = reinterpret_cast<S*>(a.out[5]) + 3 * i; o[0] = t.tam[0]; o[1] = t.tam[1]; o[2] = t.tam[2];
    o = reinterpret_cast<S*>(a.out[6]) + 3 * i;
    o[0] = wet ? S(double(r.px) + double(t.cob[0])) : S(0);
    o[1] = wet ? S(double(r.py) + double(t.cob[1])) : S(0);
    o[2] = wet ? S(double(r.pz) + double(t.cob[2])) : S(0);
    o = reinterpret_cast<S*>(a.out[7]) + 3 * i;
    o[0] = wet ? S(double(r.px) + double(t.cop[0])) : S(0);
    o[1] = wet ? S(double(r.py) + double(t.cop[1])) : S(0);
    o[2] = wet ? S(double(r.pz) + double(t.cop[2])) : S(0);
    reinterpret_cast<S*>(a.out_ratio)[i] = S(t.ratio);
    // bit 0: the reference raises / reads an unassigned variable here (A.8; in Warp-compat mode also C4)
    if (a.out_flags) a.out_flags[i] = (t.ratio > 0.0 && (t.still || (a.warp_compat != 0 && t.lift_undefined))) ? 1 : 0;
}

// dtype conversion / packing helpers -----------------------------------------
template <typename D, typename Sx>
__global__ void cast_kernel(D* dst, const Sx* src, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = D(src[i]);
}
// eleven (N,) columns -> (N,11) records (struct-of-arrays parameter upload)
struct SoaCols { const void* col[N_COEFF]; };
template <typename D, typename Sx>
__global__ void soa_to_records_kernel(D* dst, const __grid_constant__ SoaCols cols, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
#pragma unroll
    for (int k = 0; k < N_COEFF; ++k) dst[N_COEFF * i + k] = D(static_cast<const Sx*>(cols.col[k])[i]);
}
// (N,3)+(N,3) <-> (N,6)
template <typename S> __global__ void pack_prev_kernel(S* prev, const S* lin, const S* ang, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        for (int k = 0; k < 3; ++k) {
            prev[6 * i + k] = lin[3 * i + k];
            prev[6 * i + 3 + k] = ang[3 * i + k];
        }
    }
}
template <typename S> __global__ void unpack_prev_kernel(const S* prev, S* lin, S* ang, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        for (int k = 0; k < 3; ++k) {
            lin[3 * i + k] = prev[6 * i + k];
            ang[3 * i + k] = prev[6 * i + 3 + k];
        }
    }
}

// ---------------------------------------------------------------------------
// free_body_kernel (SURVEY.md 8(f2)): stand-alone rigid-body stepper for free boxes, so that
// rollouts (C1 buoy, C5) are self-contained without PhysX.  Semi-implicit Euler: velocities
// first (hydrodynamic wrench + gravity, box inertia m/12 (b^2 + c^2) in the body frame with the
// gyroscopic term), then pose with the new velocities; the quaternion is renormalised.
// Not on the force hot path: arithmetic in double, plain loads/stores, state updated in place.
// ---------------------------------------------------------------------------
struct FreeBodyArgs {
    void *pos, *quat, *lin, *ang;  // (N,3) (N,4) (N,3) (N,3), updated in place
    const void *force, *torque;    // (N,3) world-frame wrench of this step
    const void* coeff;             // records (dims + mass) -- per body or part table
    const int32_t* slot_type;
    long long n;
    int n_slots, param_mode, quat_wxyz;
    double dt, gravity;            // gravity acts along -z
};

// The step itself is free_body_update (h2o_model.cuh), shared with the persistent rollout kernel.
template <typename S> __global__ void __launch_bounds__(256) free_body_kernel(const __grid_constant__ FreeBodyArgs a)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const S* c = reinterpret_cast<const S*>(a.coeff) +
                 N_COEFF * (a.param_mode == PARAM_PER_BODY ? i : (long long)a.slot_type[i % a.n_slots]);
    S* P = reinterpret_cast<S*>(a.pos) + 3 * i;
    S* Q = reinterpret_cast<S*>(a.quat) + 4 * i;
    S* V = reinterpret_cast<S*>(a.lin) + 3 * i;
    S* W = reinterpret_cast<S*>(a.ang) + 3 * i;
    const S* Fp = reinterpret_cast<const S*>(a.force) + 3 * i;
    const S* Tp = reinterpret_cast<const S*>(a.torque) + 3 * i;
    FreeBodyState s;
    s.px = P[0]; s.py = P[1]; s.pz = P[2];
    if (a.quat_wxyz) { s.qw = Q[0]; s.qx = Q[1]; s.qy = Q[2]; s.qz = Q[3]; }
    else { s.qx = Q[0]; s.qy = Q[1]; s.qz = Q[2]; s.qw = Q[3]; }
    s.vx = V[0]; s.vy = V[1]; s.vz = V[2];
    s.wx = W[0]; s.wy = W[1]; s.wz = W[2];
    free_body_update(s, double(Fp[0]), double(Fp[1]), double(Fp[2]), double(Tp[0]), double(Tp[1]), double(Tp[2]),
                     double(c[10]), double(c[0]), double(c[1]), double(c[2]), a.dt, a.gravity);
    P[0] = S(s.px); P[1] = S(s.py); P[2] = S(s.pz);
    V[0] = S(s.vx); V[1] = S(s.vy); V[2] = S(s.vz);
    W[0] = S(s.wx); W[1] = S(s.wy); W[2] = S(s.wz);
    if (a.quat_wxyz) { Q[0] = S(s.qw); Q[1] = S(s.qx); Q[2] = S(s.qy); Q[3] = S(s.qz); }
    else { Q[0] = S(s.qx); Q[1] = S(s.qy); Q[2] = S(s.qz); Q[3] = S(s.qw); }
}

// ---------------------------------------------------------------------------
// rollout_persistent_kernel (SURVEY.md 8(f2), BASELINE configs 1 and 5): K steps of
//   fused force step (hydrodynamics_behavior.py:194-238)  ->  free-body stepper
// for free bodies in ONE launch.  Bodies are independent, so a thread carries its body's pose,
// velocities, previous velocities and coefficient record in registers across all K steps: no launch,
// graph node or global-memory round trip per step.  Every step rounds the state to the storage type
// exactly where the per-step kernels store it, so the rollout equals K x (step kernel + free_body_kernel)
// up to FMA contraction.  Every `trace_every` steps (0 = never) a row [p, v, w] per body goes to `trace`
// (sample-major: (K / trace_every, N, 9)) -- the columns of log_velocity.py:17-20.
// ---------------------------------------------------------------------------
struct RolloutArgs {
    void *pos, *quat, *lin, *ang;  // (N,3) (N,4) (N,3) (N,3) state, updated in place at the end
    void* prev;                    // (N,6) carried velocities, updated in place at the end
    void *out_force, *out_torque;  // (N,3) wrench of the LAST step
    const void* coeff;
    const int32_t* slot_type;
    void* trace;                   // optional (samples, N, 9)
    double* stats;                 // optional statistics over all steps
    long long n;
    int n_slots, param_mode, quat_wxyz;
    int n_steps, trace_every;
    double dt, gravity, rho, grav;
    double current[3], surface_z;
    int no_fallback;
    WaveArgs waves;  // evaluated at each step's position and at t, t + dt, ... from the clock
    EnvArgs envs;    // each body's env row is read once, at kernel start
    GridArgs grid;   // re-evaluated at each step's position and clock value
};

// Dynamic shared memory: wave_smem_bytes(a.waves.n).  kEnv: a.envs.cond is set (a separate instantiation, so that
// the env row held in registers costs nothing without conditions).  kGrid: a.grid.vals is set (likewise: rollouts
// without a grid compile as they did before the grid existed).  kSlope: wave-slope submersion (h2o_set_wave_slope),
// instantiated for rollouts with a wave field only.  kInertia: the fluid-acceleration loads (h2o_set_fluid_inertia),
// launched only with a wave field or a grid with nt > 1.
template <typename S, bool kStats, bool kEnv, bool kGrid, bool kSlope = false, bool kInertia = false>
__global__ void rollout_persistent_kernel(const __grid_constant__ RolloutArgs a)
{
    extern __shared__ double wave_smem[];
    const WaveArgs& wv = a.waves;
    if (wv.n) {
        stage_waves(wave_smem, wv.tab, wv.clock, wv.n);
        __syncthreads();
    }
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    ThreadStats st;
    if (i < a.n) {
        const S* c = reinterpret_cast<const S*>(a.coeff) +
                     N_COEFF * (a.param_mode == PARAM_PER_BODY ? i : (long long)a.slot_type[i % a.n_slots]);
        S cl[N_COEFF];
#pragma unroll
        for (int k = 0; k < N_COEFF; ++k) cl[k] = c[k];
        S* P = reinterpret_cast<S*>(a.pos) + 3 * i;
        S* Q = reinterpret_cast<S*>(a.quat) + 4 * i;
        S* V = reinterpret_cast<S*>(a.lin) + 3 * i;
        S* W = reinterpret_cast<S*>(a.ang) + 3 * i;
        S* PV = reinterpret_cast<S*>(a.prev) + 6 * i;
        RawBody<S> r;
        r.px = P[0]; r.py = P[1]; r.pz = P[2];
        r.q0 = Q[0]; r.q1 = Q[1]; r.q2 = Q[2]; r.q3 = Q[3];
        r.vx = V[0]; r.vy = V[1]; r.vz = V[2];
        r.wx = W[0]; r.wy = W[1]; r.wz = W[2];
        r.pvx = PV[0]; r.pvy = PV[1]; r.pvz = PV[2]; r.pwx = PV[3]; r.pwy = PV[4]; r.pwz = PV[5];
        EnvRow row{};
        if (kEnv) row = env_row(a.envs.cond, i / a.envs.bodies_per_env);
        const S inv_dt = S(1.0 / a.dt);
        S F[3] = {S(0), S(0), S(0)}, T[3] = {S(0), S(0), S(0)};
        double t = wv.n ? wave_smem[wv.n * WAVE_STRIDE] : (kGrid ? *wv.clock : 0.0);
        for (int step = 0; step < a.n_steps; ++step) {
            Env env{a.current[0], a.current[1], a.current[2], a.surface_z};
            double slope[2] = {0.0, 0.0};
            double af[3] = {0.0, 0.0, 0.0};
            if (wv.n || kEnv || kGrid) {
                if constexpr (kInertia) {
                    const WaterAccel wa = water_at<sizeof(S) == 4, kSlope, true>(
                        a.current, a.surface_z, kEnv, row, wave_smem, wv.n, wv.depth, t, double(r.px), double(r.py),
                        double(r.pz), kGrid ? &a.grid : nullptr);
                    env = Env{wa.water.cx, wa.water.cy, wa.water.cz, wa.water.surface_z};
                    slope[0] = wa.sx;
                    slope[1] = wa.sy;
                    af[0] = wa.ax; af[1] = wa.ay; af[2] = wa.az;
                } else if constexpr (kSlope) {
                    const WaterSlope ws = water_at<sizeof(S) == 4, true>(a.current, a.surface_z, kEnv, row, wave_smem,
                                                                         wv.n, wv.depth, t, double(r.px), double(r.py),
                                                                         double(r.pz), kGrid ? &a.grid : nullptr);
                    env = Env{ws.water.cx, ws.water.cy, ws.water.cz, ws.water.surface_z};
                    slope[0] = ws.sx;
                    slope[1] = ws.sy;
                } else {
                    const Water w = water_at<sizeof(S) == 4>(a.current, a.surface_z, kEnv, row, wave_smem,
                                                             wv.n, wv.depth, t, double(r.px), double(r.py), double(r.pz),
                                                             kGrid ? &a.grid : nullptr);
                    env = Env{w.cx, w.cy, w.cz, w.surface_z};
                }
                t += a.dt;  // the same sequence of additions as advance_clock_kernel over single steps
            }
            BodyIn<double, S> bin;
            make_body_in<S>(r, cl, a.quat_wxyz, a.rho, a.grav, inv_dt, env, bin);
            bool clamped, still;
            double ratio;
            uint32_t kp_mask;
            bool redo = body_step<S, false, kSlope, kInertia>(bin, cl[10], F, T, clamped, still, ratio, kp_mask, slope[0],
                                                              slope[1], af);
            if (sizeof(S) == 4) {
                redo = redo && a.no_fallback != 1;
                if (redo) {
                    RawBody<float> rf;
                    rf.px = float(r.px); rf.py = float(r.py); rf.pz = float(r.pz);
                    rf.q0 = float(r.q0); rf.q1 = float(r.q1); rf.q2 = float(r.q2); rf.q3 = float(r.q3);
                    rf.vx = float(r.vx); rf.vy = float(r.vy); rf.vz = float(r.vz);
                    rf.wx = float(r.wx); rf.wy = float(r.wy); rf.wz = float(r.wz);
                    rf.pvx = float(r.pvx); rf.pvy = float(r.pvy); rf.pvz = float(r.pvz);
                    rf.pwx = float(r.pwx); rf.pwy = float(r.pwy); rf.pwz = float(r.pwz);
                    float cf[N_COEFF];
#pragma unroll
                    for (int k = 0; k < N_COEFF; ++k) cf[k] = float(cl[k]);
                    const ExactStepOut o =
                        kInertia ? body_step_exact_f32_inertia<kSlope>(rf, cf, a.quat_wxyz, a.rho, a.grav, 1.0 / a.dt,
                                                                      env.surface_z, float(env.cx), float(env.cy),
                                                                      float(env.cz), slope[0], slope[1], af[0], af[1],
                                                                      af[2])
                        : kSlope ? body_step_exact_f32_slope(rf, cf, a.quat_wxyz, a.rho, a.grav, 1.0 / a.dt, env.surface_z,
                                                           float(env.cx), float(env.cy), float(env.cz), slope[0],
                                                           slope[1])
                               : body_step_exact_f32(rf, cf, a.quat_wxyz, a.rho, a.grav, 1.0 / a.dt, env.surface_z,
                                                     float(env.cx), float(env.cy), float(env.cz));
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        F[k] = S(o.F[k]);
                        T[k] = S(o.T[k]);
                    }
                    ratio = double(o.ratio);
                    clamped = (o.flags & 1) != 0;
                    still = (o.flags & 2) != 0;
                }
            }
            if (kStats) accumulate_stats(st, double(F[0]), double(F[1]), double(F[2]), ratio, clamped, still, redo);
            // v_prev <- v (hydrodynamics_behavior.py:237-238), then the stepper
            r.pvx = r.vx; r.pvy = r.vy; r.pvz = r.vz; r.pwx = r.wx; r.pwy = r.wy; r.pwz = r.wz;
            FreeBodyState s;
            s.px = r.px; s.py = r.py; s.pz = r.pz;
            if (a.quat_wxyz) { s.qw = r.q0; s.qx = r.q1; s.qy = r.q2; s.qz = r.q3; }
            else { s.qx = r.q0; s.qy = r.q1; s.qz = r.q2; s.qw = r.q3; }
            s.vx = r.vx; s.vy = r.vy; s.vz = r.vz;
            s.wx = r.wx; s.wy = r.wy; s.wz = r.wz;
            free_body_update(s, double(F[0]), double(F[1]), double(F[2]), double(T[0]), double(T[1]), double(T[2]),
                             double(cl[10]), double(cl[0]), double(cl[1]), double(cl[2]), a.dt, a.gravity);
            r.px = S(s.px); r.py = S(s.py); r.pz = S(s.pz);
            r.vx = S(s.vx); r.vy = S(s.vy); r.vz = S(s.vz);
            r.wx = S(s.wx); r.wy = S(s.wy); r.wz = S(s.wz);
            if (a.quat_wxyz) { r.q0 = S(s.qw); r.q1 = S(s.qx); r.q2 = S(s.qy); r.q3 = S(s.qz); }
            else { r.q0 = S(s.qx); r.q1 = S(s.qy); r.q2 = S(s.qz); r.q3 = S(s.qw); }
            if (a.trace && a.trace_every > 0 && (step + 1) % a.trace_every == 0) {
                S* tr = reinterpret_cast<S*>(a.trace) + ((long long)((step + 1) / a.trace_every - 1) * a.n + i) * 9;
                tr[0] = r.px; tr[1] = r.py; tr[2] = r.pz;
                tr[3] = r.vx; tr[4] = r.vy; tr[5] = r.vz;
                tr[6] = r.wx; tr[7] = r.wy; tr[8] = r.wz;
            }
        }
        P[0] = r.px; P[1] = r.py; P[2] = r.pz;
        Q[0] = r.q0; Q[1] = r.q1; Q[2] = r.q2; Q[3] = r.q3;
        V[0] = r.vx; V[1] = r.vy; V[2] = r.vz;
        W[0] = r.wx; W[1] = r.wy; W[2] = r.wz;
        PV[0] = r.pvx; PV[1] = r.pvy; PV[2] = r.pvz; PV[3] = r.pwx; PV[4] = r.pwy; PV[5] = r.pwz;
        S* of = reinterpret_cast<S*>(a.out_force) + 3 * i;
        S* ot = reinterpret_cast<S*>(a.out_torque) + 3 * i;
        of[0] = F[0]; of[1] = F[1]; of[2] = F[2];
        ot[0] = T[0]; ot[1] = T[1]; ot[2] = T[2];
    }
    if (kStats && a.stats) flush_stats(st, a.stats);
}

// ---------------------------------------------------------------------------
// Wave clock and sampling (h2o_set_wave_field).  The clock is one double in engine-owned device memory; a step
// evaluates the field at its value and then advance_clock_kernel adds dt to it n times (n = 1 after a step,
// n = K after a K-step persistent rollout), in stream order, so that captured graphs and the host pipeline
// see the same clock as eager steps.
// ---------------------------------------------------------------------------
__global__ void advance_clock_kernel(double* clock, double dt, int n)
{
    double t = *clock;
    for (int k = 0; k < n; ++k) t += dt;
    *clock = t;
}
__global__ void set_clock_kernel(double* clock, double t) { *clock = t; }

// points (m,3) in the engine dtype -> out (m,4) float64 [eta, ux, uy, uz] at the clock's value: the evaluator and
// precision policy of the step kernels.  Dynamic shared memory: (wv.n * WAVE_STRIDE + 1) doubles.
template <typename S>
__global__ void __launch_bounds__(256) wave_sample_kernel(const __grid_constant__ WaveArgs wv, double surface_z,
                                                          const S* points, long long m, double* out)
{
    extern __shared__ double wave_smem[];
    stage_waves(wave_smem, wv.tab, wv.clock, wv.n);
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const S* p = points + 3 * i;
    const WaveSample w = wave_eval<sizeof(S) == 4>(wave_smem, wv.n, wv.depth, double(p[0]), double(p[1]),
                                                   double(p[2]) - surface_z, wave_smem[wv.n * WAVE_STRIDE]);
    double* o = out + 4 * i;
    o[0] = w.eta; o[1] = w.ux; o[2] = w.uy; o[3] = w.uz;
}

// Per-env sampling (h2o_wave_sample_env): point k seen from env env_index[k] -> out row [s eta, s u] (the field
// alone, through water_at); an index outside [0, n_envs) gives a NaN row.  Dynamic shared memory as above.
template <typename S>
__global__ void __launch_bounds__(256) wave_sample_env_kernel(const __grid_constant__ WaveArgs wv,
                                                              const __grid_constant__ EnvArgs ev, long long n_envs,
                                                              double surface_z, const S* points,
                                                              const int32_t* env_index, long long m, double* out)
{
    extern __shared__ double wave_smem[];
    stage_waves(wave_smem, wv.tab, wv.clock, wv.n);
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    double* o = out + 4 * i;
    const long long e = env_index[i];
    if (e < 0 || e >= n_envs) {
        o[0] = o[1] = o[2] = o[3] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    const S* p = points + 3 * i;
    const double zero[3] = {0.0, 0.0, 0.0};
    const Water w = water_at<sizeof(S) == 4>(zero, surface_z, true, env_row(ev.cond, e), wave_smem, wv.n, wv.depth,
                                             wave_smem[wv.n * WAVE_STRIDE], double(p[0]), double(p[1]), double(p[2]));
    o[0] = w.field.eta; o[1] = w.field.ux; o[2] = w.field.uy; o[3] = w.field.uz;
}

// Water sampling (h2o_water_sample): point k -> out row [waterline, flow x, y, z], the full water_at composition a
// step forms at the clock's value (global environment, env row of env_index[k] when env_index is set, grid, waves),
// before a caller height array and the fp32 rounding; an index outside [0, n_envs) gives a NaN row.  Dynamic shared
// memory: (wv.n * WAVE_STRIDE + 1) doubles (the clock is staged even without waves).
template <typename S>
__global__ void __launch_bounds__(256) water_sample_kernel(const __grid_constant__ WaveArgs wv,
                                                           const __grid_constant__ EnvArgs ev,
                                                           const __grid_constant__ GridArgs gv, long long n_envs,
                                                           double cx, double cy, double cz, double surface_z,
                                                           const S* points, const int32_t* env_index, long long m,
                                                           double* out)
{
    extern __shared__ double wave_smem[];
    stage_waves(wave_smem, wv.tab, wv.clock, wv.n);
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    double* o = out + 4 * i;
    EnvRow row{};
    if (env_index) {
        const long long e = env_index[i];
        if (e < 0 || e >= n_envs) {
            o[0] = o[1] = o[2] = o[3] = __longlong_as_double(0x7ff8000000000000ll);
            return;
        }
        row = env_row(ev.cond, e);
    }
    const S* p = points + 3 * i;
    const double current[3] = {cx, cy, cz};
    const Water w = water_at<sizeof(S) == 4>(current, surface_z, env_index != nullptr, row, wave_smem, wv.n, wv.depth,
                                             wave_smem[wv.n * WAVE_STRIDE], double(p[0]), double(p[1]), double(p[2]),
                                             gv.vals ? &gv : nullptr);
    o[0] = w.surface_z; o[1] = w.cx; o[2] = w.cy; o[3] = w.cz;
}

// Slope sampling (h2o_water_slope_sample): point k -> out row [sx, sy], the surface slope a step with
// h2o_set_wave_slope on forms at the clock's value (env row of env_index[k] when env_index is set; the grid and the
// caller height array contribute none); an index outside [0, n_envs) gives a NaN row.  Dynamic shared memory:
// (wv.n * WAVE_STRIDE + 1) doubles.
template <typename S>
__global__ void __launch_bounds__(256) water_slope_sample_kernel(const __grid_constant__ WaveArgs wv,
                                                                 const __grid_constant__ EnvArgs ev, long long n_envs,
                                                                 double surface_z, const S* points,
                                                                 const int32_t* env_index, long long m, double* out)
{
    extern __shared__ double wave_smem[];
    stage_waves(wave_smem, wv.tab, wv.clock, wv.n);
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    double* o = out + 2 * i;
    EnvRow row{};
    if (env_index) {
        const long long e = env_index[i];
        if (e < 0 || e >= n_envs) {
            o[0] = o[1] = __longlong_as_double(0x7ff8000000000000ll);
            return;
        }
        row = env_row(ev.cond, e);
    }
    const S* p = points + 3 * i;
    const double zero[3] = {0.0, 0.0, 0.0};
    const WaterSlope ws = water_at<sizeof(S) == 4, true>(zero, surface_z, env_index != nullptr, row, wave_smem, wv.n,
                                                         wv.depth, wave_smem[wv.n * WAVE_STRIDE], double(p[0]),
                                                         double(p[1]), double(p[2]));
    o[0] = ws.sx; o[1] = ws.sy;
}

// Fluid-acceleration sampling (h2o_fluid_accel_sample): point k -> out row [ax, ay, az], the a_f a step with
// h2o_set_fluid_inertia on forms at the clock's value (env row of env_index[k] when env_index is set; grid, or
// nullptr, and waves); an index outside [0, n_envs) gives a NaN row.  Dynamic shared memory: (wv.n * WAVE_STRIDE + 1)
// doubles.
template <typename S>
__global__ void __launch_bounds__(256) fluid_accel_sample_kernel(const __grid_constant__ WaveArgs wv,
                                                                 const __grid_constant__ EnvArgs ev,
                                                                 const __grid_constant__ GridArgs gv, long long n_envs,
                                                                 double surface_z, const S* points,
                                                                 const int32_t* env_index, long long m, double* out)
{
    extern __shared__ double wave_smem[];
    stage_waves(wave_smem, wv.tab, wv.clock, wv.n);
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    double* o = out + 3 * i;
    EnvRow row{};
    if (env_index) {
        const long long e = env_index[i];
        if (e < 0 || e >= n_envs) {
            o[0] = o[1] = o[2] = __longlong_as_double(0x7ff8000000000000ll);
            return;
        }
        row = env_row(ev.cond, e);
    }
    const S* p = points + 3 * i;
    const double zero[3] = {0.0, 0.0, 0.0};
    const WaterAccel wa = water_at<sizeof(S) == 4, false, true>(zero, surface_z, env_index != nullptr, row, wave_smem,
                                                                wv.n, wv.depth, wave_smem[wv.n * WAVE_STRIDE],
                                                                double(p[0]), double(p[1]), double(p[2]),
                                                                gv.vals ? &gv : nullptr);
    o[0] = wa.ax; o[1] = wa.ay; o[2] = wa.az;
}

// Masked env reset (h2o_reset_envs), one thread per body: the carried [v, omega] of every body of a masked env
// becomes 0; with restart, the env's first body also sets the env's tau to -clock, so that its next step sees its
// sea at env time clock + tau = 0 exactly.
template <typename S>
__global__ void __launch_bounds__(256) reset_envs_kernel(S* prev, long long n, double* cond, long long bodies_per_env,
                                                         const uint8_t* mask, int restart, const double* clock)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long e = i / bodies_per_env;
    if (!mask[e]) return;
#pragma unroll
    for (int k = 0; k < 6; ++k) prev[6 * i + k] = S(0);
    if (restart && i == e * bodies_per_env) cond[ENV_STRIDE * e + ENV_TAU] = -*clock;
}

}  // namespace h2o
