// Host-side instantiation of the fluid-acceleration loads of silver2_isaacsim_b200/csrc/h2o_waves.cuh (the fluid
// acceleration, through water_at) and silver2_isaacsim_b200/csrc/h2o_model.cuh (body_terms / net_wrench and
// body_wrench_fast with the inertia group).
//
// TEST TOOL ONLY: lets the CPU-only tests (tests/test_fluid_inertia.py) run the code the CUDA kernels inline with
// h2o_set_fluid_inertia on against NumPy and tests/inertia_reference.py, without a GPU.  It is not part of the package,
// is not loaded by any product module and is not a fallback path.
#include <cstdint>

#include "../../silver2_isaacsim_b200/csrc/h2o_waves.cuh"

using namespace h2o;

// The fluid acceleration a step forms at points (m,3) and clock t -> out (m,3) [ax, ay, az]; n = 0 for no waves,
// grid == nullptr for no grid (else dims (nt, nz, ny, nx) and geom [gx, gy, gz, hx, hy, hz, t0, ht]); env_index ==
// nullptr applies no env row, else point i is seen from env env_index[i] (rows of cond (n_envs, ENV_STRIDE)), a NaN
// row outside [0, n_envs).
extern "C" __attribute__((visibility("default")))
int emul_accel_sample(int f32, int n, const double* comps, double depth, const double* grid, const int64_t* dims,
                      const double* geom, int64_t m, const double* points, const int32_t* env_index, int64_t n_envs,
                      const double* cond, double t, double surface_z, double* out)
{
    if (n < 0 || n > MAX_WAVE_COMPONENTS) return 1;
    double tab[MAX_WAVE_COMPONENTS * WAVE_STRIDE];
    for (int j = 0; j < n; ++j) wave_table_row(comps + 5 * j, depth, tab + WAVE_STRIDE * j);
    GridArgs g{};
    if (grid) {
        g.vals = grid;
        g.nt = dims[0]; g.nz = dims[1]; g.ny = dims[2]; g.nx = dims[3];
        g.gx = geom[0]; g.gy = geom[1]; g.gz = geom[2];
        g.hx = geom[3]; g.hy = geom[4]; g.hz = geom[5];
        g.t0 = geom[6]; g.ht = geom[7];
    }
    const double zero[3] = {0.0, 0.0, 0.0};
    for (int64_t i = 0; i < m; ++i) {
        const double* p = points + 3 * i;
        double* o = out + 3 * i;
        EnvRow row{};
        if (env_index) {
            const int64_t e = env_index[i];
            if (e < 0 || e >= n_envs) {
                o[0] = o[1] = o[2] = __builtin_nan("");
                continue;
            }
            row = env_row(cond, e);
        }
        const GridArgs* gp = grid ? &g : nullptr;
        const WaterAccel wa =
            f32 ? water_at<true, false, true>(zero, surface_z, env_index != nullptr, row, tab, n, depth, t, p[0], p[1],
                                              p[2], gp)
                : water_at<false, false, true>(zero, surface_z, env_index != nullptr, row, tab, n, depth, t, p[0], p[1],
                                               p[2], gp);
        o[0] = wa.ax; o[1] = wa.ay; o[2] = wa.az;
    }
    return 0;
}

template <typename L> static void fill_in(BodyIn<double, L>& in, int64_t i, const double* pos, const double* quat,
                                          const double* v, const double* w, const double* a, const double* b,
                                          const double* c, double rho, double g)
{
    in.pz = pos[3 * i + 2];
    in.qx = quat[4 * i]; in.qy = quat[4 * i + 1]; in.qz = quat[4 * i + 2]; in.qw = quat[4 * i + 3];
    in.vx = L(v[3 * i]); in.vy = L(v[3 * i + 1]); in.vz = L(v[3 * i + 2]);
    in.wx = L(w[3 * i]); in.wy = L(w[3 * i + 1]); in.wz = L(w[3 * i + 2]);
    in.ax = L(a[3 * i]); in.ay = L(a[3 * i + 1]); in.az = L(a[3 * i + 2]);
    in.bx = L(b[3 * i]); in.by = L(b[3 * i + 1]); in.bz = L(b[3 * i + 2]);
    in.acc_scale = L(1);
    in.dimx = L(c[0]); in.dimy = L(c[1]); in.dimz = L(c[2]);
    in.c_drag = L(c[3]); in.c_drag_ang = L(c[4]); in.k_damp = L(c[5]); in.k_damp_ang = L(c[6]);
    in.c_am = L(c[7]); in.c_am_ang = L(c[8]); in.c_lift = L(c[9]);
    in.rho_h = rho; in.grav_h = g; in.rho = L(rho);
    in.warp_compat = false;
    in.am_dense = nullptr;
}

// One model evaluation per body: pos (n,3) with z measured from the waterline, quat (n,4) xyzw, velocities v, w,
// accelerations a, b (n,3 each), coefficient records (n,11), slope (n,2), fluid acceleration af (n,3); dense: nullptr
// or one row-major 6x6 added-mass matrix per body (n,36).  mode 0: fp64 mode (body_terms + net_wrench); mode 1: fp32
// mode's fused fast path (body_wrench_fast), H = double, L = float, with the float64 world-frame re-evaluation of
// flagged bodies as the step kernels do.  inertia_on / slope_on = 0 run the instantiations without the mode (af /
// slope are then ignored).  Outputs F, T (n,3); comp (n,4) [ratio, flagged, flag_kt, flag_kf] (flag ratios: mode 1).
template <bool kSlope, bool kInertia>
static void run(int mode, int64_t n, const double* pos, const double* quat, const double* v, const double* w,
                const double* a, const double* b, const double* coeff, double rho, double g, const double* slope,
                const double* af, const double* dense, double* F, double* T, double* comp)
{
    for (int64_t i = 0; i < n; ++i) {
        const double sx = kSlope ? slope[2 * i] : 0.0, sy = kSlope ? slope[2 * i + 1] : 0.0;
        const double ax = kInertia ? af[3 * i] : 0.0, ay = kInertia ? af[3 * i + 1] : 0.0,
                     az = kInertia ? af[3 * i + 2] : 0.0;
        const double* c = coeff + 11 * i;
        double* o = comp + 4 * i;
        if (mode == 0) {
            BodyIn<double, double> in;
            fill_in<double>(in, i, pos, quat, v, w, a, b, c, rho, g);
            in.am_dense = dense ? dense + 36 * i : nullptr;
            Terms<double, double> t;
            body_terms<double, double, false, kSlope, kInertia>(in, t, nullptr, sx, sy, ax, ay, az);
            bool clamped;
            net_wrench<double, double, kInertia>(t, c[10], F + 3 * i, T + 3 * i, clamped);
            o[0] = t.ratio; o[1] = 0.0; o[2] = 0.0; o[3] = 0.0;
        } else {
            BodyIn<double, float> in;
            double qf[4];
            for (int k = 0; k < 4; ++k) qf[k] = double(float(quat[4 * i + k]));
            fill_in<float>(in, 0, pos + 3 * i, qf, v + 3 * i, w + 3 * i, a + 3 * i, b + 3 * i, c, rho, g);
            float md[36];
            if (dense) {
                for (int k = 0; k < 36; ++k) md[k] = float(dense[36 * i + k]);
                in.am_dense = md;
            }
            float f[3], tq[3], diag[14];
            bool clamped, still, suspect;
            double ratio;
            uint32_t mask;
            body_wrench_fast<double, float, false, kSlope, kInertia>(in, float(c[10]), f, tq, clamped, ratio, still,
                                                                     suspect, mask, diag, sx, sy, ax, ay, az);
            for (int k = 0; k < 3; ++k) {
                F[3 * i + k] = f[k];
                T[3 * i + k] = tq[k];
            }
            if (suspect) {  // the float64 world-frame re-evaluation, as the step kernels do it
                BodyIn<double, double> ex;
                fill_in<double>(ex, 0, pos + 3 * i, qf, v + 3 * i, w + 3 * i, a + 3 * i, b + 3 * i, c, rho, g);
                ex.vx = in.vx; ex.vy = in.vy; ex.vz = in.vz; ex.wx = in.wx; ex.wy = in.wy; ex.wz = in.wz;
                ex.ax = in.ax; ex.ay = in.ay; ex.az = in.az; ex.bx = in.bx; ex.by = in.by; ex.bz = in.bz;
                ex.dimx = in.dimx; ex.dimy = in.dimy; ex.dimz = in.dimz;
                ex.c_drag = in.c_drag; ex.c_drag_ang = in.c_drag_ang; ex.k_damp = in.k_damp;
                ex.k_damp_ang = in.k_damp_ang; ex.c_am = in.c_am; ex.c_am_ang = in.c_am_ang; ex.c_lift = in.c_lift;
                ex.rho = double(float(rho));
                double mdd[36];
                if (dense) {
                    for (int k = 0; k < 36; ++k) mdd[k] = double(md[k]);
                    ex.am_dense = mdd;
                }
                Terms<double, double> te;
                double fe[3], qe[3];
                body_terms<double, double, false, kSlope, kInertia>(ex, te, nullptr, sx, sy, ax, ay, az);
                net_wrench<double, double, kInertia>(te, double(float(c[10])), fe, qe, clamped);
                for (int k = 0; k < 3; ++k) {
                    F[3 * i + k] = float(fe[k]);
                    T[3 * i + k] = float(qe[k]);
                }
            }
            o[0] = ratio;
            o[1] = suspect ? 1.0 : 0.0;
            o[2] = diag[11];
            o[3] = diag[12];
        }
    }
}

extern "C" __attribute__((visibility("default")))
int emul_inertia_step(int mode, int inertia_on, int slope_on, int64_t n, const double* pos, const double* quat,
                      const double* v, const double* w, const double* a, const double* b, const double* coeff,
                      double rho, double g, const double* slope, const double* af, const double* dense, double* F,
                      double* T, double* comp)
{
    if (mode != 0 && mode != 1) return 1;
#define H2O_RUN(SL, IN) run<SL, IN>(mode, n, pos, quat, v, w, a, b, coeff, rho, g, slope, af, dense, F, T, comp)
    if (slope_on) {
        if (inertia_on) H2O_RUN(true, true);
        else H2O_RUN(true, false);
    } else {
        if (inertia_on) H2O_RUN(false, true);
        else H2O_RUN(false, false);
    }
#undef H2O_RUN
    return 0;
}
