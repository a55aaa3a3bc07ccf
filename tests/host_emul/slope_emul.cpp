// Host-side instantiation of the wave-slope submersion of silver2_isaacsim_b200/csrc/h2o_waves.cuh (the slope
// evaluator, through water_at) and silver2_isaacsim_b200/csrc/h2o_model.cuh (body_terms / body_wrench_fast with the
// tangent-plane waterline).
//
// TEST TOOL ONLY: lets the CPU-only tests (tests/test_wave_slope.py) run the code the CUDA kernels inline with
// h2o_set_wave_slope on against NumPy and tests/slope_reference.py, without a GPU.  It is not part of the package, is
// not loaded by any product module and is not a fallback path.
#include <cstdint>

#include "../../silver2_isaacsim_b200/csrc/h2o_waves.cuh"

using namespace h2o;

// The slope a step forms at points (m,3) and clock t -> out (m,2) [sx, sy]; env_index == nullptr applies no env row,
// else point i is seen from env env_index[i] (rows of cond (n_envs, ENV_STRIDE)), a NaN row outside [0, n_envs).
extern "C" __attribute__((visibility("default")))
int emul_slope_sample(int f32, int n, const double* comps, double depth, int64_t m, const double* points,
                      const int32_t* env_index, int64_t n_envs, const double* cond, double t, double surface_z,
                      double* out)
{
    if (n < 0 || n > MAX_WAVE_COMPONENTS) return 1;
    double tab[MAX_WAVE_COMPONENTS * WAVE_STRIDE];
    for (int j = 0; j < n; ++j) wave_table_row(comps + 5 * j, depth, tab + WAVE_STRIDE * j);
    const double zero[3] = {0.0, 0.0, 0.0};
    for (int64_t i = 0; i < m; ++i) {
        const double* p = points + 3 * i;
        EnvRow row{};
        if (env_index) {
            const int64_t e = env_index[i];
            if (e < 0 || e >= n_envs) {
                out[2 * i] = out[2 * i + 1] = __builtin_nan("");
                continue;
            }
            row = env_row(cond, e);
        }
        const WaterSlope ws =
            f32 ? water_at<true, true>(zero, surface_z, env_index != nullptr, row, tab, n, depth, t, p[0], p[1], p[2])
                : water_at<false, true>(zero, surface_z, env_index != nullptr, row, tab, n, depth, t, p[0], p[1], p[2]);
        out[2 * i] = ws.sx;
        out[2 * i + 1] = ws.sy;
    }
    return 0;
}

// One model evaluation per body: pos (n,3) with z measured from the waterline, quat (n,4) xyzw, velocities v, w,
// accelerations a, b (n,3 each), coefficient records (n,11), slope (n,2).  mode 0: fp64 mode (body_terms + net_wrench);
// mode 1: fp32 mode's fused fast path (body_wrench_fast), H = double, L = float, with the float64 world-frame
// re-evaluation of flagged bodies as the step kernels do.  slope_on = 0 runs the instantiation without slope (the
// slope array is then ignored).  warp_compat: mode 0 only.  Outputs F, T (n,3); comp (n,13) [ratio, cob(3), cop(3),
// fd(3), fbz, mask, flagged] in mode 0 (mode 1: ratio, mask and flagged only, the rest 0).
template <bool kSlope>
static void run(int mode, int warp_compat, int64_t n, const double* pos, const double* quat, const double* v,
                const double* w, const double* a, const double* b, const double* coeff, double rho, double g,
                const double* slope, double* F, double* T, double* comp)
{
    for (int64_t i = 0; i < n; ++i) {
        const double sx = kSlope ? slope[2 * i] : 0.0, sy = kSlope ? slope[2 * i + 1] : 0.0;
        const double* c = coeff + 11 * i;
        double* o = comp + 13 * i;
        for (int k = 0; k < 13; ++k) o[k] = 0.0;
        if (mode == 0) {
            BodyIn<double, double> in;
            in.pz = pos[3 * i + 2];
            in.qx = quat[4 * i]; in.qy = quat[4 * i + 1]; in.qz = quat[4 * i + 2]; in.qw = quat[4 * i + 3];
            in.vx = v[3 * i]; in.vy = v[3 * i + 1]; in.vz = v[3 * i + 2];
            in.wx = w[3 * i]; in.wy = w[3 * i + 1]; in.wz = w[3 * i + 2];
            in.ax = a[3 * i]; in.ay = a[3 * i + 1]; in.az = a[3 * i + 2];
            in.bx = b[3 * i]; in.by = b[3 * i + 1]; in.bz = b[3 * i + 2];
            in.acc_scale = 1.0;
            in.dimx = c[0]; in.dimy = c[1]; in.dimz = c[2];
            in.c_drag = c[3]; in.c_drag_ang = c[4]; in.k_damp = c[5]; in.k_damp_ang = c[6];
            in.c_am = c[7]; in.c_am_ang = c[8]; in.c_lift = c[9];
            in.rho_h = rho; in.grav_h = g; in.rho = rho;
            in.warp_compat = warp_compat != 0;
            in.am_dense = nullptr;
            Terms<double, double> t;
            body_terms<double, double, false, kSlope>(in, t, nullptr, sx, sy);
            bool clamped;
            net_wrench<double, double>(t, c[10], F + 3 * i, T + 3 * i, clamped);
            o[0] = t.ratio;
            for (int k = 0; k < 3; ++k) {
                o[1 + k] = t.cob[k]; o[4 + k] = t.cop[k]; o[7 + k] = t.fd[k];
            }
            o[10] = t.fbz;
            o[11] = double(t.kp_mask);
        } else {
            BodyIn<double, float> in;
            in.pz = pos[3 * i + 2];
            in.qx = double(float(quat[4 * i])); in.qy = double(float(quat[4 * i + 1]));
            in.qz = double(float(quat[4 * i + 2])); in.qw = double(float(quat[4 * i + 3]));
            in.vx = float(v[3 * i]); in.vy = float(v[3 * i + 1]); in.vz = float(v[3 * i + 2]);
            in.wx = float(w[3 * i]); in.wy = float(w[3 * i + 1]); in.wz = float(w[3 * i + 2]);
            in.ax = float(a[3 * i]); in.ay = float(a[3 * i + 1]); in.az = float(a[3 * i + 2]);
            in.bx = float(b[3 * i]); in.by = float(b[3 * i + 1]); in.bz = float(b[3 * i + 2]);
            in.acc_scale = 1.0f;
            in.dimx = float(c[0]); in.dimy = float(c[1]); in.dimz = float(c[2]);
            in.c_drag = float(c[3]); in.c_drag_ang = float(c[4]); in.k_damp = float(c[5]); in.k_damp_ang = float(c[6]);
            in.c_am = float(c[7]); in.c_am_ang = float(c[8]); in.c_lift = float(c[9]);
            in.rho_h = rho; in.grav_h = g; in.rho = float(rho);
            in.warp_compat = false;
            in.am_dense = nullptr;
            float f[3], tq[3];
            bool clamped, still, suspect;
            double ratio;
            uint32_t mask;
            body_wrench_fast<double, float, false, kSlope>(in, float(c[10]), f, tq, clamped, ratio, still, suspect, mask,
                                                           nullptr, sx, sy);
            for (int k = 0; k < 3; ++k) {
                F[3 * i + k] = f[k];
                T[3 * i + k] = tq[k];
            }
            if (suspect) {  // the float64 world-frame re-evaluation, as the step kernels do it
                BodyIn<double, double> ex;
                ex.pz = in.pz; ex.qx = in.qx; ex.qy = in.qy; ex.qz = in.qz; ex.qw = in.qw;
                ex.vx = in.vx; ex.vy = in.vy; ex.vz = in.vz; ex.wx = in.wx; ex.wy = in.wy; ex.wz = in.wz;
                ex.ax = in.ax; ex.ay = in.ay; ex.az = in.az; ex.bx = in.bx; ex.by = in.by; ex.bz = in.bz;
                ex.acc_scale = 1.0;
                ex.dimx = in.dimx; ex.dimy = in.dimy; ex.dimz = in.dimz;
                ex.c_drag = in.c_drag; ex.c_drag_ang = in.c_drag_ang; ex.k_damp = in.k_damp;
                ex.k_damp_ang = in.k_damp_ang; ex.c_am = in.c_am; ex.c_am_ang = in.c_am_ang; ex.c_lift = in.c_lift;
                ex.rho_h = rho; ex.grav_h = g; ex.rho = double(float(rho));
                ex.warp_compat = false;
                ex.am_dense = nullptr;
                Terms<double, double> te;
                double fe[3], qe[3];
                body_terms<double, double, false, kSlope>(ex, te, nullptr, sx, sy);
                net_wrench<double, double>(te, double(float(c[10])), fe, qe, clamped);
                for (int k = 0; k < 3; ++k) {
                    F[3 * i + k] = float(fe[k]);
                    T[3 * i + k] = float(qe[k]);
                }
            }
            o[0] = ratio;
            o[11] = double(mask);
            o[12] = suspect ? 1.0 : 0.0;
        }
    }
}

extern "C" __attribute__((visibility("default")))
int emul_slope_step(int mode, int slope_on, int warp_compat, int64_t n, const double* pos, const double* quat,
                    const double* v, const double* w, const double* a, const double* b, const double* coeff, double rho,
                    double g, const double* slope, double* F, double* T, double* comp)
{
    if (mode != 0 && mode != 1) return 1;
    if (mode == 1 && warp_compat) return 1;
    if (slope_on) run<true>(mode, warp_compat, n, pos, quat, v, w, a, b, coeff, rho, g, slope, F, T, comp);
    else run<false>(mode, warp_compat, n, pos, quat, v, w, a, b, coeff, rho, g, slope, F, T, comp);
    return 0;
}
