// h2o_waves.cuh -- built-in linear (Airy) wave field, evaluated at a point and a clock value.
//
// One evaluator for every caller: the per-body step kernel, the persistent rollout kernel and the
// h2o_wave_sample entry point on the device, tests/host_emul/waves_emul.cpp on the host.  Semantics are
// pinned in include/h2o.h (h2o_set_wave_field): for component j
//   theta_j = kx_j p_x + ky_j p_y - omega_j t + phase_j                      (always float64)
//   eta     = sum a_j cos theta_j
//   u_h     = sum a_j omega_j C_j(z) cos theta_j  k_j / |k_j|,   u_z = sum a_j omega_j S_j(z) sin theta_j
// at z = clamp(p_z - surface_z, -h, 0), with C_j = cosh(k_j (z + h)) / sinh(k_j h),
// S_j = sinh(k_j (z + h)) / sinh(k_j h) (finite depth) or C_j = S_j = exp(k_j z) (deep water).
// The hyperbolic ratios are evaluated as (e^{kz} +- e^{-k(z + 2h)}) / (1 - e^{-2kh}): no overflow at
// any k h, and the denominator comes from the table (computed once on the host with expm1).
// water_at composes the field with the global environment, a per-env conditions row
// (h2o_set_env_conditions) and a current grid (h2o_set_current_grid) into the waterline and flow a body sees.
#pragma once

#include "h2o_model.cuh"

namespace h2o {

constexpr int MAX_WAVE_COMPONENTS = 64;
// one component of the engine's device table (doubles): what the caller gave + constants derived once
enum : int {
    WAVE_KX = 0, WAVE_KY, WAVE_OMEGA, WAVE_PHASE, WAVE_A,
    WAVE_A_OMEGA,  // a * omega
    WAVE_K,        // |k|
    WAVE_KHAT_X, WAVE_KHAT_Y,  // k / |k|
    WAVE_INV_DEN,  // 1 / (1 - e^{-2 k h}); 1 in deep water
    WAVE_STRIDE
};

struct WaveSample {
    double eta, ux, uy, uz;
};
// What a slope instantiation (h2o_set_wave_slope) returns: the field and the surface slope (sx, sy).  The result type
// carries the slope, so that instantiations without it keep their signatures.
struct WaveSlopeSample {
    WaveSample field;
    double sx, sy;
};
// What an acceleration instantiation (h2o_set_fluid_inertia) returns: the field, the slope (zero without kSlope) and
// the time derivative (ax, ay, az) of the orbital velocity.
struct WaveAccelSample {
    WaveSample field;
    double sx, sy;
    double ax, ay, az;
};
template <bool kSlope, bool kAccel = false> struct WaveResult { using type = WaveSample; };
template <> struct WaveResult<true, false> { using type = WaveSlopeSample; };
template <bool kSlope> struct WaveResult<kSlope, true> { using type = WaveAccelSample; };

// theta is formed with separately rounded products and sums, in the order written above, on every
// platform (no FMA contraction), so that it is the same double the NumPy reference forms: at t ~ 1e5 s
// one ulp of theta is ~1e-11 of the amplitude.
H2O_HD double wave_mul(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    volatile double r = a * b;
    return r;
#endif
}
H2O_HD double wave_add(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    volatile double r = a + b;
    return r;
#endif
}

H2O_HD double wave_div(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    volatile double r = a / b;
    return r;
#endif
}

H2O_HD void wave_table_row(const double comp[5], double depth, double row[WAVE_STRIDE])
{
    const double a = comp[0], kx = comp[1], ky = comp[2], omega = comp[3], phase = comp[4];
    const double k = sqrt(kx * kx + ky * ky);
    row[WAVE_KX] = kx; row[WAVE_KY] = ky; row[WAVE_OMEGA] = omega; row[WAVE_PHASE] = phase; row[WAVE_A] = a;
    row[WAVE_A_OMEGA] = a * omega;
    row[WAVE_K] = k;
    row[WAVE_KHAT_X] = kx / k; row[WAVE_KHAT_Y] = ky / k;
    row[WAVE_INV_DEN] = depth < INFINITY ? -1.0 / expm1(-2.0 * k * depth) : 1.0;
}

// kF32: the fp32-mode policy.  The phase stays float64 and is reduced to [-pi, pi] in float64; sine, cosine and
// the depth decay are then evaluated in float (device: MUFU approximations, |error| < 2^-21 on [-pi, pi]), and
// the sums are kept in float64.  The field then stays within 2e-6 of sum a_j (elevation) and of
// sum a_j omega_j (velocity) of the float64 values (tests/test_waves.py).
// kSlope: also the surface gradient sum_j -a_j (kx_j, ky_j) sin theta_j, from the same sine as u_z (float in the fp32
// policy) with float64 sums (WaveSlopeSample).  Without it nothing of the gradient is formed.
// kAccel: also the time derivative of the orbital velocity, sum_j a_j omega_j^2 (C_j sin theta_j khat_j,
// -S_j cos theta_j), from the same sine, cosine and depth decay with float64 sums (WaveAccelSample).
template <bool kF32, bool kSlope = false, bool kAccel = false>
H2O_HD typename WaveResult<kSlope, kAccel>::type wave_eval(const double* tab, int n, double depth, double px,
                                                          double py, double z_rel, double t)
{
    const bool deep = !(depth < INFINITY);
    double z = z_rel < 0.0 ? z_rel : 0.0;
    if (!deep && z < -depth) z = -depth;
    WaveSample s{0.0, 0.0, 0.0, 0.0};
    double gx = 0.0, gy = 0.0;
    double dx = 0.0, dy = 0.0, dz = 0.0;
    for (int j = 0; j < n; ++j) {
        const double* c = tab + WAVE_STRIDE * j;
        const double th = wave_add(wave_add(wave_add(wave_mul(c[WAVE_KX], px), wave_mul(c[WAVE_KY], py)),
                                            -wave_mul(c[WAVE_OMEGA], t)),
                                   c[WAVE_PHASE]);
        const double k = c[WAVE_K];
        double cs, sn, ez, ezb;
        if (kF32) {
            const double r = th - 6.283185307179586 * rint(th * 0.15915494309189535);
            float sf, cf, e0, e1;
#if defined(__CUDA_ARCH__)
            __sincosf(float(r), &sf, &cf);
            e0 = __expf(float(k * z));
            e1 = deep ? 0.0f : __expf(float(-k * (z + 2.0 * depth)));
#else
            sf = sinf(float(r)); cf = cosf(float(r));
            e0 = expf(float(k * z));
            e1 = deep ? 0.0f : expf(float(-k * (z + 2.0 * depth)));
#endif
            cs = cf; sn = sf; ez = e0; ezb = e1;
        } else {
            sn = sin(th); cs = cos(th);
            ez = exp(k * z);
            ezb = deep ? 0.0 : exp(-k * (z + 2.0 * depth));
        }
        const double C = (ez + ezb) * c[WAVE_INV_DEN], S = (ez - ezb) * c[WAVE_INV_DEN];
        const double uh = c[WAVE_A_OMEGA] * C * cs;
        s.eta += c[WAVE_A] * cs;
        s.ux += uh * c[WAVE_KHAT_X];
        s.uy += uh * c[WAVE_KHAT_Y];
        s.uz += c[WAVE_A_OMEGA] * S * sn;
        if constexpr (kSlope) {
            const double as = c[WAVE_A] * sn;
            gx -= as * c[WAVE_KX];
            gy -= as * c[WAVE_KY];
        }
        if constexpr (kAccel) {
            const double aw2 = c[WAVE_A_OMEGA] * c[WAVE_OMEGA];
            const double ah = aw2 * C * sn;
            dx += ah * c[WAVE_KHAT_X];
            dy += ah * c[WAVE_KHAT_Y];
            dz -= aw2 * S * cs;
        }
    }
    if constexpr (kAccel) return WaveAccelSample{s, gx, gy, dx, dy, dz};
    else if constexpr (kSlope) return WaveSlopeSample{s, gx, gy};
    else return s;
}

// ---------------------------------------------------------------------------
// Per-env water conditions (h2o_set_env_conditions): one float64 row per env of bodies_per_env contiguous
// bodies, cond[e] = [cx, cy, cz, dz, s, tau, x0, y0].
// ---------------------------------------------------------------------------
enum : int {
    ENV_CX = 0, ENV_CY, ENV_CZ,  // current added to the global current
    ENV_DZ,                      // water-level offset added to surface_z
    ENV_SCALE,                   // wave scale s
    ENV_TAU,                     // wave time offset (s)
    ENV_X0, ENV_Y0,              // env origin
    ENV_STRIDE
};

struct EnvRow {
    double c[ENV_STRIDE];
};

H2O_HD EnvRow env_row(const double* cond, long long e)
{
    EnvRow r;
    for (int k = 0; k < ENV_STRIDE; ++k) r.c[k] = cond[ENV_STRIDE * e + k];
    return r;
}

// ---------------------------------------------------------------------------
// Current grid (h2o_set_current_grid): a borrowed, C-contiguous float64 array (nt, nz, ny, nx, 3) of velocity
// vectors; node (f, k, j, i) sits at (gx + i hx, gy + j hy, gz + k hz) and at time t0 + f ht.  The kernels read
// it through the read-only path: it is not written during a launch (the caller edits it in stream order only).
// ---------------------------------------------------------------------------
struct GridArgs {
    const double* vals;  // nullptr = no grid
    long long nt, nz, ny, nx;
    double gx, gy, gz, hx, hy, hz, t0, ht;
};

struct GridAxis {
    long long i;  // lower node
    double w;     // weight of the upper node
};

// Coordinate q on an axis of n nodes at o + k h: u = (q - o) / h clamped to [0, n - 1], i = min(floor(u), n - 2),
// w = u - i; a single node gives index 0 and weight 0 (its neighbour is never read).  q must not be NaN.
H2O_HD GridAxis grid_axis(double q, long long n, double o, double h)
{
    if (n == 1) return GridAxis{0, 0.0};
    const double top = double(n - 1);
    double u = wave_div(wave_add(q, -o), h);
    u = u > 0.0 ? (u < top ? u : top) : 0.0;
    long long i = (long long)floor(u);
    if (i > n - 2) i = n - 2;
    return GridAxis{i, wave_add(u, -double(i))};
}

H2O_HD double grid_ld(const double* p)
{
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

// a <- a + w (b - a), component by component, three separately rounded operations
H2O_HD void grid_lerp(double a[3], const double b[3], double w)
{
    for (int c = 0; c < 3; ++c) a[c] = wave_add(a[c], wave_mul(w, wave_add(b[c], -a[c])));
}

// The node at p, interpolated along x (the x-neighbour pair is 6 contiguous doubles), then y, then z.
H2O_HD void grid_x(const double* p, long long nx, double wx, double v[3])
{
    v[0] = grid_ld(p); v[1] = grid_ld(p + 1); v[2] = grid_ld(p + 2);
    if (nx > 1) {
        const double b[3] = {grid_ld(p + 3), grid_ld(p + 4), grid_ld(p + 5)};
        grid_lerp(v, b, wx);
    }
}
H2O_HD void grid_xy(const GridArgs& g, const double* p, double wx, double wy, double v[3])
{
    grid_x(p, g.nx, wx, v);
    if (g.ny > 1) {
        double b[3];
        grid_x(p + 3 * g.nx, g.nx, wx, b);
        grid_lerp(v, b, wy);
    }
}
H2O_HD void grid_xyz(const GridArgs& g, const double* p, double wx, double wy, double wz, double v[3])
{
    grid_xy(g, p, wx, wy, v);
    if (g.nz > 1) {
        double b[3];
        grid_xy(g, p + 3 * g.nx * g.ny, wx, wy, b);
        grid_lerp(v, b, wz);
    }
}

// The grid's velocity at grid-frame coordinates (X, Y, Z) and time T: multilinear, along x, then y, then z, then t,
// held at the boundary outside the lattice and before the first / after the last frame.  Any NaN coordinate gives
// NaN, with no read.
// kDiff: also dv = (G_{f+1} - G_f) / ht, the time derivative of the interpolation (G_f, G_{f+1} the spatial
// interpolations of the two frames it blends), for nt > 1 and T inside [t0, t0 + (nt - 1) ht]; 0 where the grid is
// held and for nt = 1 (h2o_set_fluid_inertia).
template <bool kDiff = false>
H2O_HD void grid_eval(const GridArgs& g, double X, double Y, double Z, double T, double v[3], double* dv = nullptr)
{
    if (X != X || Y != Y || Z != Z || T != T) {  // NaN
        v[0] = v[1] = v[2] = nan("");
        if constexpr (kDiff) dv[0] = dv[1] = dv[2] = nan("");
        return;
    }
    if constexpr (kDiff) dv[0] = dv[1] = dv[2] = 0.0;
    const GridAxis ax = grid_axis(X, g.nx, g.gx, g.hx), ay = grid_axis(Y, g.ny, g.gy, g.hy);
    const GridAxis az = grid_axis(Z, g.nz, g.gz, g.hz), at = grid_axis(T, g.nt, g.t0, g.ht);
    const double* p = g.vals + 3 * (((at.i * g.nz + az.i) * g.ny + ay.i) * g.nx + ax.i);
    grid_xyz(g, p, ax.w, ay.w, az.w, v);
    if (g.nt > 1) {
        double b[3];
        grid_xyz(g, p + 3 * g.nx * g.ny * g.nz, ax.w, ay.w, az.w, b);
        if constexpr (kDiff) {
            const double u = wave_div(wave_add(T, -g.t0), g.ht);  // grid_axis's unclamped coordinate
            if (u >= 0.0 && u <= double(g.nt - 1))
                for (int c = 0; c < 3; ++c) dv[c] = wave_div(wave_add(b[c], -v[c]), g.ht);
        }
        grid_lerp(v, b, at.w);
    }
}

// What a body sees: the waterline (before a caller height array is added), the flow, and the env's field alone
// (s * eta, s * u; zeros without a wave field).
struct Water {
    double surface_z, cx, cy, cz;
    WaveSample field;
};
// water_at's slope instantiation: the same, plus the surface slope (sx, sy) the body is tested against
// (h2o_set_wave_slope): s * the gradient of eta, (0, 0) without a wave field.  The grid, dz and the env's current
// contribute none.
struct WaterSlope {
    Water water;
    double sx, sy;
};
// water_at's acceleration instantiation (h2o_set_fluid_inertia): the same, the slope (zero without kSlope) and the
// fluid acceleration a_f = a_g + s a_w at the body centre (ax, ay, az): a_g the grid's time derivative (grid_eval
// kDiff), a_w the waves' (wave_eval kAccel).  The global and env currents, dz and a caller height array contribute
// none; the convective term (u . grad) u is not formed.
struct WaterAccel {
    Water water;
    double sx, sy;
    double ax, ay, az;
};
template <bool kSlope, bool kAccel = false> struct WaterResult { using type = Water; };
template <> struct WaterResult<true, false> { using type = WaterSlope; };
template <bool kSlope> struct WaterResult<kSlope, true> { using type = WaterAccel; };

// The one composition of the global environment (current, surface_z), the env row (has_row), the current grid
// (grid, or nullptr), the wave table and the clock value t for a body at p, used by every step kernel, the samplers
// and the host emulators.  Every operation with the row or the grid is a separately rounded float64 operation in
// the order include/h2o.h gives:
//   L = surface_z + dz,  X = p_x - x0,  Y = p_y - y0,  Z = p_z - L,  T = t + tau,
//   g = grid_eval(X, Y, Z, T),  field = s * wave_eval(X, Y, Z, T),
//   waterline = L + s eta,  flow = ((current + c) + g) + s u.
// The identity row [0,0,0,0,1,0,0,0] makes each row operation exact, so it reproduces the row-less result bit for
// bit; a grid of zeros does the same for the grid.
// kAccel: also a_f = a_g + s a_w (WaterAccel), every operation separately rounded.
template <bool kF32, bool kSlope = false, bool kAccel = false>
H2O_HD typename WaterResult<kSlope, kAccel>::type water_at(const double current[3], double surface_z, bool has_row,
                                                           const EnvRow& row, const double* tab, int n_waves,
                                                           double depth, double t, double px, double py, double pz,
                                                           const GridArgs* grid = nullptr)
{
    double sx = 0.0, sy = 0.0;
    double ag[3] = {0.0, 0.0, 0.0}, aw[3] = {0.0, 0.0, 0.0};
    Water w{surface_z, current[0], current[1], current[2], {0.0, 0.0, 0.0, 0.0}};
    const double* c = row.c;
    if (has_row) {
        w.surface_z = wave_add(surface_z, c[ENV_DZ]);
        w.cx = wave_add(current[0], c[ENV_CX]);
        w.cy = wave_add(current[1], c[ENV_CY]);
        w.cz = wave_add(current[2], c[ENV_CZ]);
        px = wave_add(px, -c[ENV_X0]);
        py = wave_add(py, -c[ENV_Y0]);
        t = wave_add(t, c[ENV_TAU]);
    }
    const double z_rel = pz - w.surface_z;
    if (grid) {
        double g[3];
        if constexpr (kAccel) grid_eval<true>(*grid, px, py, z_rel, t, g, ag);
        else grid_eval(*grid, px, py, z_rel, t, g);
        w.cx = wave_add(w.cx, g[0]);
        w.cy = wave_add(w.cy, g[1]);
        w.cz = wave_add(w.cz, g[2]);
    }
    if (n_waves) {
        if constexpr (kAccel) {
            const WaveAccelSample wa = wave_eval<kF32, kSlope, true>(tab, n_waves, depth, px, py, z_rel, t);
            w.field = wa.field;
            sx = wa.sx;
            sy = wa.sy;
            aw[0] = wa.ax; aw[1] = wa.ay; aw[2] = wa.az;
        } else if constexpr (kSlope) {
            const WaveSlopeSample ws = wave_eval<kF32, true>(tab, n_waves, depth, px, py, z_rel, t);
            w.field = ws.field;
            sx = ws.sx;
            sy = ws.sy;
        } else {
            w.field = wave_eval<kF32>(tab, n_waves, depth, px, py, z_rel, t);  // the one call site without slope
        }
        if (has_row) {
            const double s = c[ENV_SCALE];
            w.field = WaveSample{wave_mul(s, w.field.eta), wave_mul(s, w.field.ux), wave_mul(s, w.field.uy),
                                 wave_mul(s, w.field.uz)};
            if constexpr (kSlope) {
                sx = wave_mul(s, sx);
                sy = wave_mul(s, sy);
            }
            if constexpr (kAccel)
                for (int k = 0; k < 3; ++k) aw[k] = wave_mul(s, aw[k]);
        }
        w.surface_z = wave_add(w.surface_z, w.field.eta);
        w.cx = wave_add(w.cx, w.field.ux);
        w.cy = wave_add(w.cy, w.field.uy);
        w.cz = wave_add(w.cz, w.field.uz);
    }
    if constexpr (kAccel)
        return WaterAccel{w, sx, sy, wave_add(ag[0], aw[0]), wave_add(ag[1], aw[1]), wave_add(ag[2], aw[2])};
    else if constexpr (kSlope) return WaterSlope{w, sx, sy};
    else return w;
}

}  // namespace h2o
