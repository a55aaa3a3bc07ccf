// h2o_model.cuh -- per-body hydrodynamic force model, structured for a box.
//
// WHAT is computed follows the reference (citations relative to
// /root/reference/src/scripts/physics/):
//   numba_hydrodynamics.py:8-51    quaternion_to_matrix (xyzw, no normalisation)
//   numba_hydrodynamics.py:53-105  analyze_submersion_and_cob
//   numba_hydrodynamics.py:107-143 calculate_pressure_and_area
//   numba_hydrodynamics.py:145-182 calculate_hybrid_drag
//   numba_hydrodynamics.py:184-217 calculate_lift
//   numba_hydrodynamics.py:219-253 calculate_added_mass
//   numba_hydrodynamics.py:255-314 solve_hydrodynamics
//   numba_hydrodynamics_wrapper.py:55-112 box keypoints / faces / added-mass diagonal
//   hydrodynamics_behavior.py:194-238 finite-difference accel, lever arms, clamp
//
// HOW is different: nothing is looped over 27 keypoints / 6 faces / a 6x6 matrix.
// The box structure is used instead:
//   * a keypoint's world height is  p_z + (i*a + j*b) + k*c  with i,j,k in {-1,0,1},
//     a = R20*hx, b = R21*hy, c = R22*hz  -> 13 sums up to sign, 27 compares that
//     build a 27-bit "submerged" mask; centre of buoyancy comes from popcounts.
//   * the six face centres ARE six of those keypoints, so their wet tests are mask bits;
//     face normals are +-columns of R, so only one face per axis can oppose the flow.
//   * lever arms (cob - p, cop - p) are evaluated body-relative: the x,y translation
//     never enters and the reference's world-space cancellation is avoided.
//   * the added-mass matrix is diagonal.
//
// Precision policy: H ("high") carries the waterline (row 2 of R, the 27 tests,
// z_min/z_max, submersion ratio, buoyancy) and the final force/torque sums;
// L ("low") carries everything else.  fp64 mode: H = L = double.  fp32 mode:
// H = double, L = float (storage and traffic stay fp32).
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define H2O_HD __host__ __device__ __forceinline__
#else
#define H2O_HD inline
#endif

namespace h2o {

// ---- small math helpers ---------------------------------------------------
// fp32: MUFU approximation + one Newton step (full fp32 accuracy for normal, positive
// arguments; no IEEE special-case slow path -> no divergent subroutine calls).
// fp64: plain IEEE operations (fp64 mode has twice the time budget per body).
H2O_HD float h2o_abs(float x) { return fabsf(x); }
H2O_HD double h2o_abs(double x) { return fabs(x); }
H2O_HD float h2o_min(float a, float b) { return fminf(a, b); }
H2O_HD double h2o_min(double a, double b) { return fmin(a, b); }
H2O_HD float h2o_max(float a, float b) { return fmaxf(a, b); }
H2O_HD double h2o_max(double a, double b) { return fmax(a, b); }

// Host stand-in for a MUFU approximation: the exact value times (1 + u 2^-22), u in [-1, 1) hashed from the
// argument, so that the CPU precision studies see the error level of rcp.approx / rsqrt.approx (<= 2^-22.x).
#if !defined(__CUDA_ARCH__)
inline float h2o_mufu_noise(float exact, float arg)
{
    uint32_t h;
    memcpy(&h, &arg, 4);
    h ^= h >> 16; h *= 0x7feb352du; h ^= h >> 15; h *= 0x846ca68bu; h ^= h >> 16;
    const float u = float(int32_t(h)) * (1.0f / 2147483648.0f);
    return exact * (1.0f + u * 2.3841858e-7f);
}
#endif

// 1/x, x > 0: MUFU.RCP + one Newton step (full fp32 accuracy for normal, positive arguments; no IEEE
// special-case slow path).  Without the step (-DH2O_NO_NEWTON) the fast path's error doubles and the conditioning
// check would have to flag 2 % of the bodies instead of 0.02 % (tests/harness/flag_study.py).
H2O_HD float h2o_rcp(float x)
{
#if defined(__CUDA_ARCH__)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
#if !defined(H2O_NO_NEWTON)
    r = fmaf(r, fmaf(-x, r, 1.0f), r);
#endif
    return r;
#else
#if defined(H2O_NO_NEWTON)
    return h2o_mufu_noise(1.0f / x, x);
#else
    return 1.0f / x;
#endif
#endif
}
// fp64 on the device: MUFU seed + two Newton steps (full double accuracy for normal, positive arguments)
// instead of the IEEE division / square-root slow paths (~80 instructions each; the float64
// re-evaluation of flagged bodies is latency-critical, see body_wrench_fast).
H2O_HD double h2o_rcp(double x)
{
#if defined(__CUDA_ARCH__)
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return r;
#else
    return 1.0 / x;
#endif
}

// 1/sqrt(x), x > 0: MUFU.RSQ + one Newton step (see h2o_rcp)
H2O_HD float h2o_rsqrt(float x)
{
#if defined(__CUDA_ARCH__)
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
#if !defined(H2O_NO_NEWTON)
    const float t = x * y;
    y = fmaf(0.5f * y, fmaf(-t, y, 1.0f), y);
#endif
    return y;
#else
#if defined(H2O_NO_NEWTON)
    return h2o_mufu_noise(1.0f / sqrtf(x), x);
#else
    return 1.0f / sqrtf(x);
#endif
#endif
}
H2O_HD double h2o_rsqrt(double x)
{
#if defined(__CUDA_ARCH__)
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double hx = 0.5 * x;
    y = fma(y, fma(-hx * y, y, 0.5), y);
    y = fma(y, fma(-hx * y, y, 0.5), y);
    y = fma(y, fma(-hx * y, y, 0.5), y);
    return y;
#else
    return 1.0 / sqrt(x);
#endif
}

// sqrt(x) given r = h2o_rsqrt(x):  x*r with one correction step
H2O_HD float h2o_sqrt_from_rsqrt(float x, float r)
{
    const float s = x * r;
#if !defined(H2O_NO_NEWTON)
    return fmaf(fmaf(-s, s, x), 0.5f * r, s);
#else
    return s;
#endif
}
H2O_HD double h2o_sqrt_from_rsqrt(double x, double r)
{
#if defined(__CUDA_ARCH__)
    const double s = x * r;
    return fma(fma(-s, s, x), 0.5 * r, s);
#else
    (void)r;
    return sqrt(x);
#endif
}

// 1/x for the waterline ratio (H precision).  Device: approximation + two Newton steps.
H2O_HD double h2o_rcp_h(double x)
{
#if defined(__CUDA_ARCH__)
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return r;
#else
    return 1.0 / x;
#endif
}

H2O_HD float h2o_rcp_h(float x) { return 1.0f / x; }

H2O_HD int h2o_popc(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

// mask |= bit  if  t < m      (one compare + one predicated OR on the device)
H2O_HD void h2o_or_if_less(uint32_t& mask, double t, double m, uint32_t bit)
{
#if defined(__CUDA_ARCH__)
    asm("{\n\t.reg .pred p;\n\tsetp.lt.f64 p, %1, %2;\n\t@p or.b32 %0, %0, %3;\n\t}"
        : "+r"(mask)
        : "d"(t), "d"(m), "r"(bit));
#else
    if (t < m) mask |= bit;
#endif
}
H2O_HD void h2o_or_if_less(uint32_t& mask, float t, float m, uint32_t bit)
{
    if (t < m) mask |= bit;
}

// Lift coefficient sin(2*asin(d)) (numba_hydrodynamics.py:197-203), d already clipped.
// kExactTrig follows the reference literally.  Otherwise the identity
// sin(2 asin d) = 2 d sqrt(1 - d^2) is used with 1 - d^2 supplied by the caller from
// a well-conditioned expression (|v_hat x up|^2 - (|up|^2 - 1)), because forming
// 1 - d*d from a rounded d loses all accuracy as |d| -> 1.
template <bool kExactTrig> H2O_HD double lift_coefficient_of(double d, double one_minus_d2)
{
    if (kExactTrig) return sin(2.0 * asin(d));
    const double x = fmax(one_minus_d2, 1e-300);
    return 2.0 * d * h2o_sqrt_from_rsqrt(x, h2o_rsqrt(x));
}
template <bool kExactTrig> H2O_HD float lift_coefficient_of(float d, float one_minus_d2)
{
    if (kExactTrig) return sinf(2.0f * asinf(d));
    const float x = fmaxf(one_minus_d2, 1e-30f);
    return 2.0f * d * h2o_sqrt_from_rsqrt(x, h2o_rsqrt(x));
}

// ---- keypoint bit layout --------------------------------------------------
// bit(i,j,k) = (i+1) + 3*(j+1) + 9*(k+1), i/j/k = sign of the x/y/z offset.
constexpr int kp_bit(int i, int j, int k) { return (i + 1) + 3 * (j + 1) + 9 * (k + 1); }
constexpr uint32_t kp_mask_axis(int axis, int sign)
{
    uint32_t m = 0;
    for (int i = -1; i <= 1; ++i)
        for (int j = -1; j <= 1; ++j)
            for (int k = -1; k <= 1; ++k) {
                const int s = axis == 0 ? i : (axis == 1 ? j : k);
                if (s == sign) m |= 1u << kp_bit(i, j, k);
            }
    return m;
}
constexpr uint32_t KP_ALL = (1u << 27) - 1u;
constexpr uint32_t KP_XP = kp_mask_axis(0, +1), KP_XN = kp_mask_axis(0, -1);
constexpr uint32_t KP_YP = kp_mask_axis(1, +1), KP_YN = kp_mask_axis(1, -1);
constexpr uint32_t KP_ZP = kp_mask_axis(2, +1), KP_ZN = kp_mask_axis(2, -1);

// ---- inputs / outputs -----------------------------------------------------
template <typename H, typename L> struct BodyIn {
    H pz;                 // height of the body origin above the z = 0 waterline
    H qx, qy, qz, qw;     // orientation, xyzw
    L vx, vy, vz;         // linear velocity (world)
    L wx, wy, wz;         // angular velocity (world)
    L ax, ay, az;         // linear acceleration (world) ...
    L bx, by, bz;         // angular acceleration (world) ...
    L acc_scale;          // ... both to be multiplied by this (1, or 1/dt when a,b hold velocity differences;
                          //     only body_wrench_fast honours it, folding it into the added-mass constants)
    // coefficient record (params.py COEFF_FIELDS) + globals
    L dimx, dimy, dimz;
    L c_drag, c_drag_ang, k_damp, k_damp_ang, c_am, c_am_ang, c_lift;
    bool warp_compat;     // body_terms only: the deviations of the reference's Warp twin (SURVEY.md Appendix C, pinned by
                          // tests/golden/reference_warp_golden.npz): accelerations rotated FORWARD into the "body"
                          // frame (warp_hydrodynamics.py:216-217, C1); every rotation is wp.quat_rotate =
                          // R(q) + 2 (|q|^2 - 1) I (C7); centre of buoyancy = mean of the wet keypoints also
                          // for a fully submerged body (:57-58, C9)
    H rho_h, grav_h;      // globals: waterDensity, gravity (H for buoyancy)
    L rho;                // = L(rho_h)
    const L* am_dense;    // optional dense 6x6 added-mass matrix, row-major, body frame (the matrix
                          // calculate_added_mass takes, numba_hydrodynamics.py:220); nullptr = the
                          // wrapper's diagonal built from c_am / c_am_ang (wrapper :101-112)
};

// The body-frame fast path (body_wrench_fast) treats R(q) as orthogonal.  The reference never normalises
// q, so its R is orthogonal only up to dq = |q|^2 - 1.  Quaternions handed out by a simulator are unit to
// fp32 rounding (|dq| <= 2.4e-7); anything further from unit must take body_terms + net_wrench (exact in dq).
constexpr double FAST_PATH_MAX_DQ = 1e-6;
// Conditioning thresholds of body_wrench_fast (see there), chosen with tests/harness/flag_study.py: of 1.4e7
// random wet bodies (C2 / C3 / C4 distributions) no unflagged one comes closer than 0.65x to the fp32-mode
// bound; 2.5e-4 (C3) / 3e-5 (hexapod fleets) of the bodies are flagged.
constexpr double FLAG_KAPPA_T = 0.06, FLAG_KAPPA_F = 0.15;

template <typename H, typename L> struct Terms {
    H ratio;              // submersion ratio (0 => every other field is 0)
    H fbz;                // buoyancy force, +z (numba_hydrodynamics.py:282)
    L fd[3];              // drag force
    L fl[3];              // lift force
    L td[3];              // drag torque
    L fam[3];             // added-mass force
    L tam[3];             // added-mass torque
    L cob[3];             // centre of buoyancy - p   (body-relative lever arm, world axes)
    L cop[3];             // centre of pressure - p
    L tarm[3];            // (cop - p) x drag force, evaluated without cancellation
    L ffk[3];             // Froude-Krylov force rho r V a_f at the centre of buoyancy (kInertia only)
    uint32_t kp_mask;     // 27-bit submerged-keypoint mask (diagnostic)
    bool still;           // wet and speed <= 1e-6: the reference raises here (SURVEY.md A.8)
    bool lift_undefined;  // moving, but the flow is along the body z axis: the Numba path returns zero lift
                          // (numba_hydrodynamics.py:210-211), the Warp twin reads an unassigned lift_dir
                          // (warp_hydrodynamics.py:196-200; SURVEY.md Appendix C4)
};

// ---- waterline: 27 keypoints {-hx,0,hx}x{hy,0,-hy}x{hz,0,-hz} against the plane z = 0
//      (numba_hydrodynamics_wrapper.py:55-73, numba_hydrodynamics.py:271, :59-105), all in H.
// A keypoint's height is p_z + (i a + j b) + k c with a = R20 hx, b = R21 hy, c = R22 hz: 13 sums up to
// sign, 27 strict compares build the submerged mask; z_min / z_max = p_z -+ (|a| + |b| + |c|).
template <typename H> struct Waterline {
    uint32_t mask;   // 27-bit submerged-keypoint mask, bit layout kp_bit()
    H ratio;         // submersion ratio after the 1e-9 cut (numba_hydrodynamics.py:87, :277-279)
    bool partial;    // z_min < 0 < z_max: the centre of buoyancy is the mean of the wet keypoints
    bool warp_needs_keypoints;  // kWarpSkip only: some lane of the warp is cut by the surface (warp-uniform)
};
// kMask = false: the caller already holds the mask (w.mask is left alone); only the ratio is formed
// kWarpSkip (device, robot-mode tile kernels): when NO lane of the warp is cut by the surface -- a fleet walking on
// the sea bed, the reference's main scene (SILVER2 at z = -18.4 m) -- every mask is all-or-nothing and the 27
// compares are skipped for the whole warp.  Exact: ext is the largest keypoint offset bit for bit (same sums, same
// association), rounding is monotone, so fl(pz + ext) < 0 implies t < -pz for every keypoint.  A top keypoint
// exactly ON the surface (z_max == 0) is not wet and takes the compares.
template <typename H, bool kMask = true, bool kWarpSkip = false>
H2O_HD void waterline(H pz, H r20h, H r21h, H r22h, H dxh, H dyh, H dzh, Waterline<H>& w)
{
    const H a = r20h * (dxh * H(0.5));
    const H b = r21h * (dyh * H(0.5));
    const H c = r22h * (dzh * H(0.5));
    const H ext = (h2o_abs(a) + h2o_abs(b)) + h2o_abs(c);  // highest keypoint above p
    const H z_min = pz - ext, z_max = pz + ext;
    bool compare = kMask;
    w.warp_needs_keypoints = true;
#if defined(__CUDA_ARCH__)
    if (kMask && kWarpSkip) {
        const bool cut = !(z_max < H(0)) && !(z_min >= H(0));
        compare = __any_sync(__activemask(), cut);
        w.warp_needs_keypoints = compare;
        if (!compare) w.mask = (z_max < H(0)) ? KP_ALL : 0u;
    }
#endif
    if (compare) {
        const H abp = a + b, abm = a - b;
        const H m = -pz;  // keypoint wet  <=>  fl(t + pz) < 0  <=>  t < -pz  (exact)
        uint32_t mask = 0;
#define H2O_KP(i, j, k, tval)                                                   \
    {                                                                           \
        const H tv = (tval);                                                    \
        h2o_or_if_less(mask, tv, m, 1u << kp_bit(i, j, k));                     \
        h2o_or_if_less(mask, -tv, m, 1u << kp_bit(-(i), -(j), -(k)));           \
    }
        H2O_KP(1, 0, 0, a)
        H2O_KP(0, 1, 0, b)
        H2O_KP(1, 1, 0, abp)
        H2O_KP(1, -1, 0, abm)
        H2O_KP(0, 0, 1, c)
        H2O_KP(1, 0, 1, a + c)
        H2O_KP(1, 0, -1, a - c)
        H2O_KP(0, 1, 1, b + c)
        H2O_KP(0, 1, -1, b - c)
        H2O_KP(1, 1, 1, abp + c)
        H2O_KP(1, 1, -1, abp - c)
        H2O_KP(1, -1, 1, abm + c)
        H2O_KP(1, -1, -1, abm - c)
#undef H2O_KP
        h2o_or_if_less(mask, H(0), m, 1u << kp_bit(0, 0, 0));
        w.mask = mask;
    }
    const bool dry = z_min >= H(0);
    const bool partial = !dry && !(z_max <= H(0));
    H ratio = H(1);
    if (!kWarpSkip || w.warp_needs_keypoints) {  // (no lane cut by the surface: every ratio is 0 or 1)
        const H total_height = z_max - z_min;
        if (partial && !(total_height < H(1e-6))) ratio = h2o_min(H(1), -z_min * h2o_rcp_h(total_height));
    }
    if (dry || !(ratio > H(1e-9))) ratio = H(0);  // numba_hydrodynamics.py:87, :277-279
    w.ratio = ratio;
    w.partial = partial;
}

// Separately rounded products and sums that the compiler neither contracts nor merges with other arithmetic
// (slope_rows: a kernel's remaining code must compile as it does without the slope).
H2O_HD double h2o_mul_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    volatile double r = a * b;
    return r;
#endif
}
H2O_HD double h2o_add_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    volatile double r = a + b;
    return r;
#endif
}
H2O_HD float h2o_mul_rn(float a, float b)
{
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    volatile float r = a * b;
    return r;
#endif
}
H2O_HD float h2o_add_rn(float a, float b)
{
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    volatile float r = a + b;
    return r;
#endif
}

// Wave-slope submersion (h2o_set_wave_slope): the keypoints are tested against the plane through the waterline with
// normal n = (-sx, -sy, 1) instead of the horizontal one.  Keypoint k (body frame) has height
// (p_z - W) + n . (R k) = (p_z - W) + e . k with e = R^T n, i.e. e_c = (R_2c - sx R_0c) - sy R_1c, formed in H;
// waterline() then takes e in place of row 2 of R.  Rows 0 and 1 of R (plus diag_shift on the diagonal: the Warp
// twin's R + 2 dq I) are formed here from q = (x, y, z, w) with the reference's formula, every operation separately
// rounded, so that nothing is shared with the caller's own rotation and the rest of the caller is unchanged.
// n is not normalised: every sign test and the ratio -z_min / (z_max - z_min) are invariant to its length.
// sx = sy = 0 gives e = row 2 (up to the sign of a zero, which no test sees).
template <typename H>
H2O_HD void slope_rows(H sx, H sy, H qx, H qy, H qz, H qw, H diag_shift, H& e0, H& e1, H& e2)
{
    const H x2 = h2o_add_rn(qx, qx), y2 = h2o_add_rn(qy, qy), z2 = h2o_add_rn(qz, qz);
    const H xx = h2o_mul_rn(qx, x2), xy = h2o_mul_rn(qx, y2), xz = h2o_mul_rn(qx, z2);
    const H yy = h2o_mul_rn(qy, y2), yz = h2o_mul_rn(qy, z2), zz = h2o_mul_rn(qz, z2);
    const H wx = h2o_mul_rn(qw, x2), wy = h2o_mul_rn(qw, y2), wz = h2o_mul_rn(qw, z2);
    const H r00 = h2o_add_rn(h2o_add_rn(H(1), -h2o_add_rn(yy, zz)), diag_shift), r01 = h2o_add_rn(xy, -wz),
            r02 = h2o_add_rn(xz, wy);
    const H r10 = h2o_add_rn(xy, wz), r11 = h2o_add_rn(h2o_add_rn(H(1), -h2o_add_rn(xx, zz)), diag_shift),
            r12 = h2o_add_rn(yz, -wx);
    e0 = h2o_add_rn(h2o_add_rn(e0, -h2o_mul_rn(sx, r00)), -h2o_mul_rn(sy, r10));
    e1 = h2o_add_rn(h2o_add_rn(e1, -h2o_mul_rn(sx, r01)), -h2o_mul_rn(sy, r11));
    e2 = h2o_add_rn(h2o_add_rn(e2, -h2o_mul_rn(sx, r02)), -h2o_mul_rn(sy, r12));
}

// One body, branch-free.  kExactTrig: asin/sin as the reference vs 2d*sqrt(1-d^2).
// kSlope: the waterline is the local tangent plane of slope (sx, sy) (slope_rows); everything after the waterline
// uses the real R.
// kInertia: fluid-acceleration loads for the world-frame fluid acceleration (afx, afy, afz) (h2o_set_fluid_inertia):
// the added mass sees a - a_f in place of a, and t.ffk holds the Froude-Krylov force rho r V a_f (net_wrench applies
// it at the centre of buoyancy).
template <typename H, typename L, bool kExactTrig, bool kSlope = false, bool kInertia = false>
H2O_HD void body_terms(const BodyIn<H, L>& in, Terms<H, L>& t, const uint32_t* given_mask = nullptr, H sx = H(0),
                       H sy = H(0), H afx = H(0), H afy = H(0), H afz = H(0))
{
    // ---- rotation (numba_hydrodynamics.py:14-49).  Row 2 in H for the waterline.
    const H hx2 = in.qx + in.qx, hy2 = in.qy + in.qy, hz2 = in.qz + in.qz;
    const H r20h = in.qx * hz2 - in.qw * hy2;
    const H r21h = in.qy * hz2 + in.qw * hx2;
    // |q|^2 - 1: the reference never normalises, so R is orthogonal only up to this.
    const H dqh = ((in.qx * in.qx + in.qy * in.qy) + (in.qz * in.qz + in.qw * in.qw)) - H(1);
    // Warp twin: wp.quat_rotate(q, x) = x (2w^2 - 1) + 2 q_v (q_v.x) + 2w (q_v x x) = (R(q) + 2 dq I) x
    const H diag_shift = in.warp_compat ? (dqh + dqh) : H(0);
    const H r22h = (H(1) - (in.qx * hx2 + in.qy * hy2)) + diag_shift;

    const H dxh = H(in.dimx), dyh = H(in.dimy), dzh = H(in.dimz);
    H e0 = r20h, e1 = r21h, e2 = r22h;  // the waterline rows
    if (kSlope) slope_rows<H>(sx, sy, in.qx, in.qy, in.qz, in.qw, diag_shift, e0, e1, e2);
    Waterline<H> wl;
    if (given_mask) {  // a caller that has run the identical 27 H compares already (body_wrench_fast)
        wl.mask = *given_mask;
        waterline<H, false>(in.pz, e0, e1, e2, dxh, dyh, dzh, wl);
    } else {
        waterline<H>(in.pz, e0, e1, e2, dxh, dyh, dzh, wl);
    }
    const uint32_t mask = wl.mask;
    const H ratio = wl.ratio;
    const bool partial = wl.partial;

    t.kp_mask = mask;
    t.ratio = ratio;
    const L rl = L(ratio);  // 0 for a dry body: every force below is scaled by it

    // ---- full rotation matrix in L
    const L qx = L(in.qx), qy = L(in.qy), qz = L(in.qz), qw = L(in.qw);
    const L x2 = qx + qx, y2 = qy + qy, z2 = qz + qz;
    const L xx = qx * x2, xy = qx * y2, xz = qx * z2;
    const L yy = qy * y2, yz = qy * z2, zz = qz * z2;
    const L wx = qw * x2, wy = qw * y2, wz = qw * z2;
    const L dsh = L(diag_shift);
    const L r00 = (L(1) - (yy + zz)) + dsh, r01 = xy - wz, r02 = xz + wy;
    const L r10 = xy + wz, r11 = (L(1) - (xx + zz)) + dsh, r12 = yz - wx;
    const L r20 = L(r20h), r21 = L(r21h), r22 = L(r22h);
    const L dq = L(dqh);

    const L hx = in.dimx * L(0.5), hy = in.dimy * L(0.5), hz = in.dimz * L(0.5);
    const L ayz = in.dimy * in.dimz, axz = in.dimx * in.dimz, axy = in.dimx * in.dimy;  // face areas
    const L vol = in.dimx * ayz;  // numba_hydrodynamics_wrapper.py:15

    // ---- buoyancy (numba_hydrodynamics.py:282)
    t.fbz = in.rho_h * (ratio * (dxh * dyh * dzh)) * in.grav_h;

    // ---- centre of buoyancy, body-relative: R * (h .* sum(sign)/count)
    const int cnt = h2o_popc(mask);
    const L cinv = ((partial || (in.warp_compat && ratio > H(0))) && cnt > 0) ? h2o_rcp(L(cnt)) : L(0);
    const L csx = L(h2o_popc(mask & KP_XP) - h2o_popc(mask & KP_XN)) * (cinv * hx);
    const L csy = L(h2o_popc(mask & KP_YP) - h2o_popc(mask & KP_YN)) * (cinv * hy);
    const L csz = L(h2o_popc(mask & KP_ZP) - h2o_popc(mask & KP_ZN)) * (cinv * hz);
    const L cobx = r00 * csx + r01 * csy + r02 * csz;
    const L coby = r10 * csx + r11 * csy + r12 * csz;
    const L cobz = r20 * csx + r21 * csy + r22 * csz;

    // ---- flow direction (numba_hydrodynamics.py:285-289)
    const L speed2 = in.vx * in.vx + in.vy * in.vy + in.vz * in.vz;
    const L rs = h2o_rsqrt(h2o_max(speed2, L(1e-30)));
    const L speed = h2o_sqrt_from_rsqrt(speed2, rs);
    const bool moving = speed > L(1e-6);
    const L inv_speed = moving ? rs : L(0);
    const L ux = in.vx * inv_speed, uy = in.vy * inv_speed, uz = in.vz * inv_speed;
    t.still = !moving && (ratio > H(0));

    // ---- projected area + centre of pressure (numba_hydrodynamics.py:113-143).
    // Face normals are +-columns of R; the face opposing the flow on axis j is the one with
    // sign -sgn(d_j), alignment |d_j|, centre = that sign * h_j * R[:,j].  Its wet test is the
    // keypoint bit of the face centre (strict <, in every regime).
    const L d0 = r00 * ux + r10 * uy + r20 * uz;
    const L d1 = r01 * ux + r11 * uy + r21 * uz;
    const L d2 = r02 * ux + r12 * uy + r22 * uz;
    const uint32_t f0 = (d0 < L(0)) ? (1u << kp_bit(1, 0, 0)) : (1u << kp_bit(-1, 0, 0));
    const uint32_t f1 = (d1 < L(0)) ? (1u << kp_bit(0, 1, 0)) : (1u << kp_bit(0, -1, 0));
    const uint32_t f2 = (d2 < L(0)) ? (1u << kp_bit(0, 0, 1)) : (1u << kp_bit(0, 0, -1));
    const L w0 = (mask & f0) ? L(1) : L(0), w1 = (mask & f1) ? L(1) : L(0), w2 = (mask & f2) ? L(1) : L(0);
    // s_j * area = -h_j A_j w_j d_j ;  alignment*area = |d_j| A_j w_j
    const L g0 = w0 * d0, g1 = w1 * d1, g2 = w2 * d2;
    const L area = (h2o_abs(g0) * ayz + h2o_abs(g1) * axz) + h2o_abs(g2) * axy;
    const bool faces = area > L(1e-6);
    const L inv_area = faces ? h2o_rcp(area) : L(0);
    const L ginv = (vol * L(0.5)) * inv_area;  // h_j A_j / area, identical on the three axes
    const L s0 = -(ginv * g0), s1 = -(ginv * g1), s2 = -(ginv * g2);
    const L copx = faces ? (r00 * s0 + r01 * s1 + r02 * s2) : cobx;
    const L copy = faces ? (r10 * s0 + r11 * s1 + r12 * s2) : coby;
    const L copz = faces ? (r20 * s0 + r21 * s1 + r22 * s2) : cobz;

    // ---- hybrid drag (numba_hydrodynamics.py:153-182)
    const L low = L(0.2);
    const L quad = L(0.5) * in.rho * speed2 * in.c_drag * area;  // area = 0 unless moving
    const L kd = in.k_damp * h2o_min(L(1), speed * L(5.0));
    t.fd[0] = (-(quad * ux) - kd * in.vx) * rl;
    t.fd[1] = (-(quad * uy) - kd * in.vy) * rl;
    t.fd[2] = (-(quad * uz) - kd * in.vz) * rl;

    // Lever-arm torque of the drag force, (cop - p) x F_d (hydrodynamics_behavior.py:213).
    // F_d = -psi * v_hat is anti-parallel to the flow and, because h_j * A_j = V/2 on
    // every axis, the face-weighted arm is  cop - p = R s,  s_j = -(V/2A) w_j d_j  with
    // d = R^T v_hat and w_j = [opposing face of axis j is wet].  When every opposing face
    // is wet s is parallel to d and the reference's world-space cross product is pure
    // cancellation (what survives is an artefact of the un-normalised quaternion,
    // R R^T = I - 4 dq [u]x^2, u = vector part, dq = |q|^2 - 1).  Evaluated in the body
    // frame, to first order in dq, nothing cancels:
    //   v_hat x (R s) = R c + 4 dq ( u (u . R c) + (u (u.v_hat) - |u|^2 v_hat) x (R s) ),
    //   c = d x s,  c_x = -(V/2A) d_y d_z (w_z - w_y)  (cyclic).
    // Without face contributions (cop = cob) the plain cross product is used.
    {
        const L psi = faces ? (quad + kd * speed) * rl : L(0);
        const L c0 = -(ginv * d1 * d2 * (w2 - w1));
        const L c1 = -(ginv * d2 * d0 * (w0 - w2));
        const L c2 = -(ginv * d0 * d1 * (w1 - w0));
        const L rcx = r00 * c0 + r01 * c1 + r02 * c2;
        const L rcy = r10 * c0 + r11 * c1 + r12 * c2;
        const L rcz = r20 * c0 + r21 * c1 + r22 * c2;
        const L k4 = L(4) * dq;
        const L udu = qx * ux + qy * uy + qz * uz;
        const L uu = qx * qx + qy * qy + qz * qz;
        const L gx = qx * udu - uu * ux, gy = qy * udu - uu * uy, gz = qz * udu - uu * uz;
        const L urc = qx * rcx + qy * rcy + qz * rcz;
        // plain arm x F_d, kept only when the arm is the centre of buoyancy
        const L nf = faces ? L(0) : L(1);
        const L px = (coby * t.fd[2] - cobz * t.fd[1]) * nf;
        const L py = (cobz * t.fd[0] - cobx * t.fd[2]) * nf;
        const L pz = (cobx * t.fd[1] - coby * t.fd[0]) * nf;
        t.tarm[0] = psi * (rcx + k4 * (qx * urc + (gy * copz - gz * copy))) + px;
        t.tarm[1] = psi * (rcy + k4 * (qy * urc + (gz * copx - gx * copz))) + py;
        t.tarm[2] = psi * (rcz + k4 * (qz * urc + (gx * copy - gy * copx))) + pz;
        if (in.warp_compat) {
            // the factorisation above is for R(q); the Warp twin rotates with R(q) + 2 dq I: plain cross product
            t.tarm[0] = copy * t.fd[2] - copz * t.fd[1];
            t.tarm[1] = copz * t.fd[0] - copx * t.fd[2];
            t.tarm[2] = copx * t.fd[1] - copy * t.fd[0];
        }
    }
    {
        const L as2 = in.wx * in.wx + in.wy * in.wy + in.wz * in.wz;
        const L as = h2o_sqrt_from_rsqrt(as2, h2o_rsqrt(h2o_max(as2, L(1e-30))));
        // -(0.5 rho |w|^2 C V) * w/|w|  ==  -(0.5 rho |w| C V) * w
        const L aq = (as > L(1e-6)) ? L(0.5) * in.rho * as * in.c_drag_ang * vol : L(0);
        const L ka = (aq + in.k_damp_ang * h2o_min(L(1), as * L(5.0))) * rl;
        t.td[0] = -(ka * in.wx);
        t.td[1] = -(ka * in.wy);
        t.td[2] = -(ka * in.wz);
    }
    (void)low;

    // ---- lift (numba_hydrodynamics.py:191-217); up = R[:,2], so -up.v_hat = -d2
    {
        // axis = v_hat x up ; dir = (axis/|axis|) x v_hat
        const L axx = uy * r22 - uz * r12;
        const L axy_ = uz * r02 - ux * r22;
        const L axz_ = ux * r12 - uy * r02;
        const L an2 = axx * axx + axy_ * axy_ + axz_ * axz_;
        const L ra = h2o_rsqrt(h2o_max(an2, L(1e-30)));
        const L an = h2o_sqrt_from_rsqrt(an2, ra);
        const bool ok = !(speed < L(1e-6)) && !(an < L(1e-6));
        t.lift_undefined = !(speed < L(1e-6)) && (an < L(1e-6));
        const L dd = h2o_max(L(-1), h2o_min(L(1), -d2));
        // 1 - d^2 = |v_hat x up|^2 - (|up|^2 - 1),  |up|^2 - 1 = 4 dq (qx^2 + qy^2)
        // (Warp twin: up gains 2 dq e_z, so |up|^2 - 1 gains 2dq (2 r22 - 2dq))
        const L eta = L(4) * dq * (qx * qx + qy * qy) + dsh * ((r22 + r22) - dsh);
        const L cl = lift_coefficient_of<kExactTrig>(dd, an2 - eta);
        const L mag = L(0.5) * in.rho * speed2 * cl * area * in.c_lift;
        const L s = ok ? mag * rl * ra : L(0);
        t.fl[0] = (axy_ * uz - axz_ * uy) * s;
        t.fl[1] = (axz_ * ux - axx * uz) * s;
        t.fl[2] = (axx * uy - axy_ * ux) * s;
    }

    // ---- added mass (numba_hydrodynamics.py:224-253; diagonal of
    //      numba_hydrodynamics_wrapper.py:101-112): -R diag(M) R^T acc * ratio
    {
        const bool fwd = in.warp_compat;  // Numba: R^T a (numba_hydrodynamics.py:229-230); Warp twin: R a
        // kInertia: the fluid-relative acceleration a - a_f
        const L ax = kInertia ? in.ax - L(afx) : in.ax, ay = kInertia ? in.ay - L(afy) : in.ay,
                az = kInertia ? in.az - L(afz) : in.az;
        const L lx = fwd ? r00 * ax + r01 * ay + r02 * az : r00 * ax + r10 * ay + r20 * az;
        const L ly = fwd ? r10 * ax + r11 * ay + r12 * az : r01 * ax + r11 * ay + r21 * az;
        const L lz = fwd ? r20 * ax + r21 * ay + r22 * az : r02 * ax + r12 * ay + r22 * az;
        const L gx = fwd ? r00 * in.bx + r01 * in.by + r02 * in.bz : r00 * in.bx + r10 * in.by + r20 * in.bz;
        const L gy = fwd ? r10 * in.bx + r11 * in.by + r12 * in.bz : r01 * in.bx + r11 * in.by + r21 * in.bz;
        const L gz = fwd ? r20 * in.bx + r21 * in.by + r22 * in.bz : r02 * in.bx + r12 * in.by + r22 * in.bz;
        L fx, fy, fz, tx, ty, tz;
        if (in.am_dense) {  // f6 = -M [a_b; alpha_b]  (numba_hydrodynamics.py:232-243), any 6x6
            const L a6[6] = {lx, ly, lz, gx, gy, gz};
            L f6[6];
            for (int i = 0; i < 6; ++i) {
                L acc = L(0);
                for (int j = 0; j < 6; ++j) acc += in.am_dense[6 * i + j] * a6[j];
                f6[i] = -(acc * rl);
            }
            fx = f6[0]; fy = f6[1]; fz = f6[2];
            tx = f6[3]; ty = f6[4]; tz = f6[5];
        } else {
            const L ml = vol * in.c_am * in.rho * rl;
            fx = -(ml * lx); fy = -(ml * ly); fz = -(ml * lz);
            const L ma = vol * in.c_am_ang * in.rho * rl;
            const L w2s = in.dimx * in.dimx, d2s = in.dimy * in.dimy, h2s = in.dimz * in.dimz;
            tx = -(ma * (d2s + h2s) * gx); ty = -(ma * (w2s + h2s) * gy); tz = -(ma * (w2s + d2s) * gz);
        }
        t.fam[0] = r00 * fx + r01 * fy + r02 * fz;
        t.fam[1] = r10 * fx + r11 * fy + r12 * fz;
        t.fam[2] = r20 * fx + r21 * fy + r22 * fz;
        t.tam[0] = r00 * tx + r01 * ty + r02 * tz;
        t.tam[1] = r10 * tx + r11 * ty + r12 * tz;
        t.tam[2] = r20 * tx + r21 * ty + r22 * tz;
    }

    t.cob[0] = cobx; t.cob[1] = coby; t.cob[2] = cobz;
    t.cop[0] = copx; t.cop[1] = copy; t.cop[2] = copz;
    if (kInertia) {  // Froude-Krylov: rho r V a_f (0 for a dry body)
        const L rv = in.rho * (rl * vol);
        t.ffk[0] = rv * L(afx); t.ffk[1] = rv * L(afy); t.ffk[2] = rv * L(afz);
    }
}

// Net wrench + safety clamp (hydrodynamics_behavior.py:212-226).
// Lever arms are already body-relative, so  (cob - p) x F_b  =  cob_rel x (0,0,fbz).
// Only F_z mixes the H-precision buoyancy with the L terms.
// kInertia: the Froude-Krylov force t.ffk joins the force, and (cob - p) x t.ffk the torque, before the clamp.
template <typename H, typename L, bool kInertia = false>
H2O_HD void net_wrench(const Terms<H, L>& t, L mass, L F[3], L T[3], bool& clamped)
{
    F[0] = (t.fd[0] + t.fl[0]) + t.fam[0];
    F[1] = (t.fd[1] + t.fl[1]) + t.fam[1];
    if (kInertia) {
        F[0] = F[0] + t.ffk[0];
        F[1] = F[1] + t.ffk[1];
        F[2] = L(t.fbz + H(((t.fd[2] + t.fl[2]) + t.fam[2]) + t.ffk[2]));
    } else {
        F[2] = L(t.fbz + H((t.fd[2] + t.fl[2]) + t.fam[2]));
    }

    const L fb = L(t.fbz);
    const L cx = t.cop[0], cy = t.cop[1], cz = t.cop[2];
    T[0] = ((t.cob[1] * fb + t.tarm[0]) + (cy * t.fl[2] - cz * t.fl[1])) + (t.td[0] + t.tam[0]);
    T[1] = ((t.tarm[1] - t.cob[0] * fb) + (cz * t.fl[0] - cx * t.fl[2])) + (t.td[1] + t.tam[1]);
    T[2] = (t.tarm[2] + (cx * t.fl[1] - cy * t.fl[0])) + (t.td[2] + t.tam[2]);
    if (kInertia) {
        T[0] = T[0] + (t.cob[1] * t.ffk[2] - t.cob[2] * t.ffk[1]);
        T[1] = T[1] + (t.cob[2] * t.ffk[0] - t.cob[0] * t.ffk[2]);
        T[2] = T[2] + (t.cob[0] * t.ffk[1] - t.cob[1] * t.ffk[0]);
    }

    // scale = min(1, m*500 / (|F| + 1e-6)); the division only matters when the clamp bites.
    const L max_force = mass * L(500.0);
    const L mag2 = F[0] * F[0] + F[1] * F[1] + F[2] * F[2];
    const L lim = max_force - L(1e-6);
    clamped = !(lim > L(0)) || mag2 > lim * lim;
    if (clamped) {
        const L mag = h2o_sqrt_from_rsqrt(mag2, h2o_rsqrt(h2o_max(mag2, L(1e-30))));
        const L scale = h2o_min(L(1), max_force * h2o_rcp(mag + L(1e-6)));
        clamped = scale < L(1);
        for (int k = 0; k < 3; ++k) {
            F[k] *= scale;
            T[k] *= scale;
        }
    }
}

// ---------------------------------------------------------------------------
// fp32-mode fast path: net wrench only (fused step), torque assembled in the BODY frame.
//
// Same model as body_terms + net_wrench.  In the body frame the box makes most terms trivial:
// the lift axis is v_hat x z_body = (d1, -d0, 0), the lever arms are the face / keypoint
// offsets themselves, the added-inertia tensor is diagonal, and a single rotation takes the
// summed body-frame torque to the world.  It uses R(a x b) = (Ra) x (Rb), exact only for an
// orthogonal R; the reference's R deviates from that by dq = |q|^2 - 1 (~1e-7 for fp32
// quaternions), i.e. by one fp32 rounding of each term -- fine for the fp32 tolerance, not for
// fp64 mode, which keeps the world-frame formulation above.  The one place where dq matters
// even in fp32 (the cancelling cop x F_d, see body_terms) keeps its first-order dq term.
// ---------------------------------------------------------------------------
// kSlope: as body_terms (the tangent-plane waterline of slope (sx, sy)).
// kInertia: as body_terms (fluid acceleration (afx, afy, afz), world frame).  The isotropic diagonal added mass on a_f
// and the Froude-Krylov force join the world-frame force as rho r V (1 + C_a) a_f (rho r V a_f with a dense matrix,
// whose a_f part M [R^T a_f; 0] is formed in the body frame); the Froude-Krylov torque (cob - p) x rho r V R^T a_f is
// formed in the body frame.  Both groups are counted by the conditioning check.
template <typename H, typename L, bool kWarpSkip = false, bool kSlope = false, bool kInertia = false>
H2O_HD void body_wrench_fast(const BodyIn<H, L>& in, L mass, L F[3], L T[3], bool& clamped, H& ratio_out,
                             bool& still, bool& suspect, uint32_t& mask_out, L* diag = nullptr, H sx = H(0),
                             H sy = H(0), H afx = H(0), H afy = H(0), H afz = H(0))
{
    // ---- waterline in H (the same function body_terms calls)
    const H hx2 = in.qx + in.qx, hy2 = in.qy + in.qy, hz2 = in.qz + in.qz;
    const H hxx = in.qx * hx2, hyy = in.qy * hy2, hzz = in.qz * hz2;
    const H hxy = in.qx * hy2, hxz = in.qx * hz2, hyz = in.qy * hz2;
    const H hwx = in.qw * hx2, hwy = in.qw * hy2, hwz = in.qw * hz2;
    const H r20h = hxz - hwy;
    const H r21h = hyz + hwx;
    const H r22h = H(1) - (hxx + hyy);
    const H dqh = ((in.qx * in.qx + in.qy * in.qy) + (in.qz * in.qz + in.qw * in.qw)) - H(1);
    const H dxh = H(in.dimx), dyh = H(in.dimy), dzh = H(in.dimz);
    Waterline<H> wl;
    if (kSlope) {
        H e0 = r20h, e1 = r21h, e2 = r22h;
        slope_rows<H>(sx, sy, in.qx, in.qy, in.qz, in.qw, H(0), e0, e1, e2);
        waterline<H, true, kWarpSkip>(in.pz, e0, e1, e2, dxh, dyh, dzh, wl);
    } else {
        waterline<H, true, kWarpSkip>(in.pz, r20h, r21h, r22h, dxh, dyh, dzh, wl);
    }
    const uint32_t mask = wl.mask;
    const H ratio = wl.ratio;
    const bool partial = wl.partial;
    mask_out = mask;
    ratio_out = ratio;
    const L rl = L(ratio);
    const H fbz = in.rho_h * (ratio * (dxh * dyh * dzh)) * in.grav_h;  // numba_hydrodynamics.py:282

    // ---- rotation matrix in L (row 2 from the H values)
    const L qx = L(in.qx), qy = L(in.qy), qz = L(in.qz), qw = L(in.qw);
    const L x2 = qx + qx, y2 = qy + qy, z2 = qz + qz;
    const L wx = qw * x2, wy = qw * y2, wz = qw * z2;
    const L r00 = (L(1) - qy * y2) - qz * z2, r11 = (L(1) - qx * x2) - qz * z2;
    const L r01 = qx * y2 - wz, r10 = qx * y2 + wz;
    const L r02 = qx * z2 + wy, r12 = qy * z2 - wx;
    const L r20 = L(r20h), r21 = L(r21h), r22 = L(r22h);
    const L k4 = L(4) * L(dqh);

    const L ayz = in.dimy * in.dimz, axz = in.dimx * in.dimz, axy = in.dimx * in.dimy;
    const L vol = in.dimx * ayz;

    // ---- centre of buoyancy in the body frame: h .* sum(sign)/count
    L cinv = L(0), cbx = L(0), cby = L(0), cbz = L(0);
    if (!kWarpSkip || wl.warp_needs_keypoints) {  // no lane cut by the surface: cob = p in every lane
        const int cnt = h2o_popc(mask);
        cinv = (partial && cnt > 0) ? h2o_rcp(L(cnt)) : L(0);
        const L chalf = cinv * L(0.5);
        cbx = L(h2o_popc(mask & KP_XP) - h2o_popc(mask & KP_XN)) * (chalf * in.dimx);
        cby = L(h2o_popc(mask & KP_YP) - h2o_popc(mask & KP_YN)) * (chalf * in.dimy);
        cbz = L(h2o_popc(mask & KP_ZP) - h2o_popc(mask & KP_ZN)) * (chalf * in.dimz);
    }
    // Buoyancy torque (cob - p) x (0,0,fb) needs the horizontal offset of the centre of buoyancy,
    // which vanishes at hydrostatic equilibrium as a difference of O(h) terms: rows 0,1 of R and
    // the weighted sum are carried in H so that the restoring torque of a floating body keeps
    // its relative accuracy (a floating buoy sits exactly in that regime).
    L tbuoy_x = L(0), tbuoy_y = L(0);
    if (!kWarpSkip || wl.warp_needs_keypoints) {  // no lane cut by the surface: cinv = 0 in every lane, the arm is zero
        const H sxh = H(h2o_popc(mask & KP_XP) - h2o_popc(mask & KP_XN)) * (dxh * H(0.5));
        const H syh = H(h2o_popc(mask & KP_YP) - h2o_popc(mask & KP_YN)) * (dyh * H(0.5));
        const H szh = H(h2o_popc(mask & KP_ZP) - h2o_popc(mask & KP_ZN)) * (dzh * H(0.5));
        const H cobx_h = (H(1) - (hyy + hzz)) * sxh + (hxy - hwz) * syh + (hxz + hwy) * szh;
        const H coby_h = (hxy + hwz) * sxh + (H(1) - (hxx + hzz)) * syh + (hyz - hwx) * szh;
        // the cancellation is over once the sums are formed: scale by fb / count in L
        const L scale = cinv * L(fbz);
        tbuoy_x = L(coby_h) * scale;
        tbuoy_y = -(L(cobx_h) * scale);
    }

    // ---- flow direction, world and body (d = R^T v_hat)
    const L speed2 = in.vx * in.vx + in.vy * in.vy + in.vz * in.vz;
    const L rs = h2o_rsqrt(h2o_max(speed2, L(1e-30)));
    const L speed = h2o_sqrt_from_rsqrt(speed2, rs);
    const bool moving = speed > L(1e-6);
    const L inv_speed = moving ? rs : L(0);
    still = !moving && (ratio > H(0));
    // d = R^T v_hat carried in H: when the flow is nearly parallel to a face, d_j is a cancelled sum of O(1)
    // products and the centre of pressure is a RATIO of such alignments; L products of an L-rounded R lose
    // it (1e-5 relative on the drag lever arm for alignments ~1e-3).  All nine H entries of R exist already.
#if defined(H2O_D_IN_L)  // cost experiment only: the round-1 fp32 alignment
    const L ux_ = in.vx * inv_speed, uy_ = in.vy * inv_speed, uz_ = in.vz * inv_speed;
    const L d0 = r00 * ux_ + r10 * uy_ + r20 * uz_;
    const L d1 = r01 * ux_ + r11 * uy_ + r21 * uz_;
    const L d2 = r02 * ux_ + r12 * uy_ + r22 * uz_;
#else
    const H vxh = H(in.vx), vyh = H(in.vy), vzh = H(in.vz);
    const L d0 = L((H(1) - (hyy + hzz)) * vxh + (hxy + hwz) * vyh + r20h * vzh) * inv_speed;
    const L d1 = L((hxy - hwz) * vxh + (H(1) - (hxx + hzz)) * vyh + r21h * vzh) * inv_speed;
    const L d2 = L((hxz + hwy) * vxh + (hyz - hwx) * vyh + r22h * vzh) * inv_speed;
#endif

    // ---- projected area, centre of pressure (body frame) -- see body_terms
    L w0, w1, w2;
    const bool per_face = !kWarpSkip || wl.warp_needs_keypoints;  // warp-uniform
    if (per_face) {
        const uint32_t f0 = (d0 < L(0)) ? (1u << kp_bit(1, 0, 0)) : (1u << kp_bit(-1, 0, 0));
        const uint32_t f1 = (d1 < L(0)) ? (1u << kp_bit(0, 1, 0)) : (1u << kp_bit(0, -1, 0));
        const uint32_t f2 = (d2 < L(0)) ? (1u << kp_bit(0, 0, 1)) : (1u << kp_bit(0, 0, -1));
        w0 = (mask & f0) ? L(1) : L(0); w1 = (mask & f1) ? L(1) : L(0); w2 = (mask & f2) ? L(1) : L(0);
    } else {  // no lane cut by the surface: every face of a body is wet, or none
        w0 = w1 = w2 = mask ? L(1) : L(0);
    }
    const L g0 = w0 * d0, g1 = w1 * d1, g2 = w2 * d2;
    const L area = (h2o_abs(g0) * ayz + h2o_abs(g1) * axz) + h2o_abs(g2) * axy;
    const bool faces = area > L(1e-6);
    const L inv_area = faces ? h2o_rcp(area) : L(0);
    const L ginv = (vol * L(0.5)) * inv_area;
    const L s0 = -(ginv * g0), s1 = -(ginv * g1), s2 = -(ginv * g2);
    const L armx = faces ? s0 : cbx, army = faces ? s1 : cby, armz = faces ? s2 : cbz;  // cop - p

    // ---- drag force (world) and its lever-arm torque (body)
    const L q0 = L(0.5) * in.rho * speed2 * area;
    const L kd = in.k_damp * h2o_min(L(1), speed * L(5.0));
    const L gam = (q0 * in.c_drag * inv_speed + kd) * rl;  // F_d = -gam * v
    const L psi = gam * speed;                              // |F_d| along -v_hat
    // faces: (cop-p) x F_d = psi (c + 4dq (u(u.d) - |u|^2 d) x s), c = d x s factored so that it
    // is exactly zero when every opposing face is wet; otherwise the arm is cob: psi (d x cob)
    const L gd0 = ginv * d0, gd1 = ginv * d1, gd2 = ginv * d2;
    const L udd = qx * d0 + qy * d1 + qz * d2;
    const L uu = qx * qx + qy * qy + qz * qz;
    const L gbx = qx * udd - uu * d0, gby = qy * udd - uu * d1, gbz = qz * udd - uu * d2;
    const L nf = faces ? L(0) : L(1);
    L tdx = k4 * (gby * s2 - gbz * s1), tdy = k4 * (gbz * s0 - gbx * s2), tdz = k4 * (gbx * s1 - gby * s0);
    if (per_face) {  // (otherwise w0 = w1 = w2 and cob = p: both groups are exactly zero)
        tdx = (gd1 * d2) * (w1 - w2) + tdx + nf * (d1 * cbz - d2 * cby);
        tdy = (gd2 * d0) * (w2 - w0) + tdy + nf * (d2 * cbx - d0 * cbz);
        tdz = (gd0 * d1) * (w0 - w1) + tdz + nf * (d0 * cby - d1 * cbx);
    }
    // running sum of the torque groups' magnitudes (conditioning check at the end)
    L mt = h2o_abs(psi) * ((h2o_abs(tdx) + h2o_abs(tdy)) + h2o_abs(tdz));

    // ---- lift in the body frame: axis = d x z = (d1,-d0,0), dir = axis/|axis| x d
    const L an2 = d0 * d0 + d1 * d1;
    const L ra = h2o_rsqrt(h2o_max(an2, L(1e-30)));
    const L an = an2 * ra;
    const bool lift_ok = !(speed < L(1e-6)) && !(an < L(1e-6));
    const L dd = h2o_max(L(-1), h2o_min(L(1), -d2));
    const L omd = h2o_max(an2 - k4 * (qx * qx + qy * qy), L(1e-30));  // 1 - d^2, well conditioned
    const L cl = L(2) * dd * (omd * h2o_rsqrt(omd));
    const L sl = lift_ok ? (q0 * cl * in.c_lift) * (rl * ra) : L(0);
    const L tl = d2 * sl;
    const L flx = -(d0 * tl), fly = -(d1 * tl), flz = an2 * sl;  // body frame

    // ---- added mass: isotropic force in the world frame (R m I R^T = m I), inertia torque in the
    //      body frame; a dense matrix (am_dense) keeps both in the body frame
    const L rv = vol * in.rho * rl * in.acc_scale;
    const L bbx = r00 * in.bx + r10 * in.by + r20 * in.bz;
    const L bby = r01 * in.bx + r11 * in.by + r21 * in.bz;
    const L bbz = r02 * in.bx + r12 * in.by + r22 * in.bz;
    L ml, ffx, ffy, ffz, tbx, tby, tbz;
    L ai0, ai1, ai2;  // added-inertia torque, body frame
    const L cfx = army * flz - armz * fly, cfy = armz * flx - armx * flz, cfz = armx * fly - army * flx;  // arm x F_l
    // kInertia: a_f in the world and body frames, rho r V, and the magnitudes of the groups it forms
    const L afw0 = L(afx), afw1 = L(afy), afw2 = L(afz);
    L afb0 = L(0), afb1 = L(0), afb2 = L(0), ri = L(0), mfi = L(0), mti = L(0);
    if (kInertia) {
        afb0 = r00 * afw0 + r10 * afw1 + r20 * afw2;
        afb1 = r01 * afw0 + r11 * afw1 + r21 * afw2;
        afb2 = r02 * afw0 + r12 * afw1 + r22 * afw2;
        ri = vol * in.rho * rl;
    }
    if (in.am_dense) {
        const L a6[6] = {r00 * in.ax + r10 * in.ay + r20 * in.az, r01 * in.ax + r11 * in.ay + r21 * in.az,
                         r02 * in.ax + r12 * in.ay + r22 * in.az, bbx, bby, bbz};
        const L sc = rl * in.acc_scale;
        L f6[6];
        for (int i = 0; i < 6; ++i) {
            L acc = L(0);
            for (int j = 0; j < 6; ++j) acc += in.am_dense[6 * i + j] * a6[j];
            f6[i] = acc * sc;
            if (kInertia) {  // M [R^T (a - a_f); R^T alpha]: the a_f part, counted by the conditioning check
                const L fa = ((in.am_dense[6 * i] * afb0 + in.am_dense[6 * i + 1] * afb1) + in.am_dense[6 * i + 2] * afb2) * rl;
                f6[i] = f6[i] - fa;
                if (i < 3) mfi += h2o_abs(fa);
                else mti += h2o_abs(fa);
            }
        }
        ml = L(0);
        ffx = flx - f6[0]; ffy = fly - f6[1]; ffz = flz - f6[2];
        ai0 = f6[3]; ai1 = f6[4]; ai2 = f6[5];
    } else {
        ml = rv * in.c_am;
        const L ma = rv * in.c_am_ang;
        const L w2s = in.dimx * in.dimx, d2s = in.dimy * in.dimy, h2s = in.dimz * in.dimz;
        ffx = flx; ffy = fly; ffz = flz;
        // ---- body-frame torque: psi*(...) + arm x F_l + added inertia (buoyancy torque: tbuoy, above)
        ai0 = ma * (d2s + h2s) * bbx; ai1 = ma * (w2s + h2s) * bby; ai2 = ma * (w2s + d2s) * bbz;
    }
    tbx = psi * tdx + (cfx - ai0);
    tby = psi * tdy + (cfy - ai1);
    tbz = psi * tdz + (cfz - ai2);
    mt += ((h2o_abs(cfx) + h2o_abs(cfy)) + h2o_abs(cfz)) + ((h2o_abs(ai0) + h2o_abs(ai1)) + h2o_abs(ai2));
    // kInertia, world-frame force coefficient of a_f: Froude-Krylov, plus the isotropic diagonal added mass
    L kfi = L(0);
    if (kInertia) {
        kfi = in.am_dense ? ri : ri * (L(1) + in.c_am);
        // Froude-Krylov torque, body frame: cob x rho r V R^T a_f
        const L fk0 = ri * afb0, fk1 = ri * afb1, fk2 = ri * afb2;
        const L tf0 = cby * fk2 - cbz * fk1, tf1 = cbz * fk0 - cbx * fk2, tf2 = cbx * fk1 - cby * fk0;
        tbx = tbx + tf0;
        tby = tby + tf1;
        tbz = tbz + tf2;
        mt += ((h2o_abs(tf0) + h2o_abs(tf1)) + h2o_abs(tf2)) + mti;
        mfi += h2o_abs(kfi) * ((h2o_abs(afw0) + h2o_abs(afw1)) + h2o_abs(afw2));
    }

    // ---- angular drag (world): -(0.5 rho |w| C V + k min(1, 5|w|)) ratio * w
    const L as2 = in.wx * in.wx + in.wy * in.wy + in.wz * in.wz;
    const L as = h2o_sqrt_from_rsqrt(as2, h2o_rsqrt(h2o_max(as2, L(1e-30))));
    const L aq = (as > L(1e-6)) ? L(0.5) * in.rho * as * in.c_drag_ang * vol : L(0);
    const L ka = (aq + in.k_damp_ang * h2o_min(L(1), as * L(5.0))) * rl;
    mt += ka * as + (h2o_abs(tbuoy_x) + h2o_abs(tbuoy_y));

    T[0] = ((r00 * tbx + r01 * tby + r02 * tbz) - ka * in.wx) + tbuoy_x;
    T[1] = ((r10 * tbx + r11 * tby + r12 * tbz) - ka * in.wy) + tbuoy_y;
    T[2] = (r20 * tbx + r21 * tby + r22 * tbz) - ka * in.wz;

    F[0] = (r00 * ffx + r01 * ffy + r02 * ffz) - (gam * in.vx + ml * in.ax);
    F[1] = (r10 * ffx + r11 * ffy + r12 * ffz) - (gam * in.vy + ml * in.ay);
    // buoyancy joins in L: its rounding (6e-8 fbz) reaches the bound only where |F| < 0.6 % of fbz, and those
    // bodies are flagged below (|F| < FLAG_KAPPA_F fbz)
    const L fbl = L(fbz);
    if (kInertia) {
        F[0] = F[0] + kfi * afw0;
        F[1] = F[1] + kfi * afw1;
        F[2] = fbl + (((r20 * ffx + r21 * ffy + r22 * ffz) - (gam * in.vz + ml * in.az)) + kfi * afw2);
    } else {
        F[2] = fbl + ((r20 * ffx + r21 * ffy + r22 * ffz) - (gam * in.vz + ml * in.az));
    }

    // ---- conditioning check.  L arithmetic carries ~1e-7 relative error per TERM; the result meets the
    // fp32-mode bound (1e-5 relative per vector, SURVEY.md 8(d)) unless that error is amplified:
    //   (a) the torque groups cancel: |T| << sum of the group magnitudes;
    //   (b) the force groups cancel (buoyancy against drag, mostly);
    //   (c) the quaternion is further from unit than the body-frame formulation tolerates.
    // Such bodies (a few per 100 000) are flagged and the caller re-evaluates them in float64 with the
    // world-frame formulation (body_terms + net_wrench), so fp32 mode stays inside its bound for EVERY body.
    L flag_kt, flag_kf;
    {
        const L t1 = (h2o_abs(T[0]) + h2o_abs(T[1])) + h2o_abs(T[2]);
        const L f1 = (h2o_abs(F[0]) + h2o_abs(F[1])) + h2o_abs(F[2]);
        // (b): buoyancy is the only force group that does not vanish with the velocities, so a cancelled net
        // force means |F| << F_buoyancy.  kInertia: the fluid-acceleration groups do not vanish with the velocities
        // either (and cancel drag exactly in the Morison case): |F| << F_buoyancy + their magnitude
        const L fs = kInertia ? fbl + mfi : fbl;
        flag_kt = t1 / h2o_max(mt, L(1e-30)); flag_kf = f1 / h2o_max(fs, L(1e-30));
#if defined(H2O_NO_FLAGS)  // cost experiment only: no conditioning check (the dq check stays)
        suspect = h2o_abs(dqh) > H(FAST_PATH_MAX_DQ);
#else
        suspect = (t1 < L(FLAG_KAPPA_T) * mt) | (f1 < L(FLAG_KAPPA_F) * fs) | (h2o_abs(dqh) > H(FAST_PATH_MAX_DQ));
#endif
    }

    if (diag) {  // precision study only (tests/harness/precision_study.py): magnitudes of the term groups
        auto mx = [](L a, L b, L c) { return h2o_max(h2o_abs(a), h2o_max(h2o_abs(b), h2o_abs(c))); };
        diag[0] = h2o_abs(psi) * mx(tdx, tdy, tdz);
        diag[1] = mx(cfx, cfy, cfz);
        diag[2] = mx(tbx, tby, tbz);
        diag[3] = ka * mx(in.wx, in.wy, in.wz);
        diag[4] = mx(tbuoy_x, tbuoy_y, L(0));
        diag[5] = mx(T[0], T[1], T[2]);
        diag[6] = mx(ffx, ffy, ffz);
        diag[7] = gam * mx(in.vx, in.vy, in.vz);
        diag[8] = ml * mx(in.ax, in.ay, in.az);
        diag[9] = fbl;
        diag[10] = mx(F[0], F[1], F[2]);
        diag[11] = flag_kt; diag[12] = flag_kf; diag[13] = L(0);
    }

    // ---- safety clamp (hydrodynamics_behavior.py:221-226)
    const L max_force = mass * L(500.0);
    const L mag2 = F[0] * F[0] + F[1] * F[1] + F[2] * F[2];
    const L lim = max_force - L(1e-6);
    clamped = !(lim > L(0)) || mag2 > lim * lim;
    if (clamped) {
        const L mag = h2o_sqrt_from_rsqrt(mag2, h2o_rsqrt(h2o_max(mag2, L(1e-30))));
        const L scale = h2o_min(L(1), max_force * h2o_rcp(mag + L(1e-6)));
        clamped = scale < L(1);
        for (int k = 0; k < 3; ++k) {
            F[k] *= scale;
            T[k] *= scale;
        }
    }
}

// ---- free-body stepper ------------------------------------------------------
// One semi-implicit Euler step of a free box (free_body_kernel, the persistent rollout kernel and the host
// emulator tests/host_emul/free_body_emul.cpp).  State in double, quaternion xyzw; m, dx, dy, dz from the
// coefficient record.  The float64 reference is oracle/free_body.py (integrate).
struct FreeBodyState {
    double px, py, pz, qx, qy, qz, qw, vx, vy, vz, wx, wy, wz;
};
H2O_HD void free_body_update(FreeBodyState& s, double fx, double fy, double fz, double tx, double ty, double tz,
                             double m, double dx, double dy, double dz, double dt, double gravity)
{
    const double qx = s.qx, qy = s.qy, qz = s.qz, qw = s.qw;
    const double im = 1.0 / m;
    // linear: v += dt (F/m + g)
    const double vx = s.vx + dt * fx * im;
    const double vy = s.vy + dt * fy * im;
    const double vz = s.vz + dt * (fz * im - gravity);
    // angular, body frame: I w' = tau_b - w_b x (I w_b)
    const double x2 = qx + qx, y2 = qy + qy, z2 = qz + qz;
    const double r00 = 1 - (qy * y2 + qz * z2), r01 = qx * y2 - qw * z2, r02 = qx * z2 + qw * y2;
    const double r10 = qx * y2 + qw * z2, r11 = 1 - (qx * x2 + qz * z2), r12 = qy * z2 - qw * x2;
    const double r20 = qx * z2 - qw * y2, r21 = qy * z2 + qw * x2, r22 = 1 - (qx * x2 + qy * y2);
    const double Ix = m * (dy * dy + dz * dz) / 12.0, Iy = m * (dx * dx + dz * dz) / 12.0,
                 Iz = m * (dx * dx + dy * dy) / 12.0;
    const double wx = s.wx, wy = s.wy, wz = s.wz;
    const double tbx = r00 * tx + r10 * ty + r20 * tz, tby = r01 * tx + r11 * ty + r21 * tz,
                 tbz = r02 * tx + r12 * ty + r22 * tz;
    double wbx = r00 * wx + r10 * wy + r20 * wz, wby = r01 * wx + r11 * wy + r21 * wz,
           wbz = r02 * wx + r12 * wy + r22 * wz;
    const double gx = wby * (Iz * wbz) - wbz * (Iy * wby), gy = wbz * (Ix * wbx) - wbx * (Iz * wbz),
                 gz = wbx * (Iy * wby) - wby * (Ix * wbx);
    wbx += dt * (tbx - gx) / Ix;
    wby += dt * (tby - gy) / Iy;
    wbz += dt * (tbz - gz) / Iz;
    const double nwx = r00 * wbx + r01 * wby + r02 * wbz, nwy = r10 * wbx + r11 * wby + r12 * wbz,
                 nwz = r20 * wbx + r21 * wby + r22 * wbz;
    // pose with the NEW velocities; q' = q + dt/2 (0,w) * q
    s.px += dt * vx; s.py += dt * vy; s.pz += dt * vz;
    const double h = 0.5 * dt;
    double nqw = qw - h * (nwx * qx + nwy * qy + nwz * qz);
    double nqx = qx + h * (nwx * qw + nwy * qz - nwz * qy);
    double nqy = qy + h * (nwy * qw + nwz * qx - nwx * qz);
    double nqz = qz + h * (nwz * qw + nwx * qy - nwy * qx);
    const double inv = 1.0 / sqrt(nqx * nqx + nqy * nqy + nqz * nqz + nqw * nqw);
    s.qx = nqx * inv; s.qy = nqy * inv; s.qz = nqz * inv; s.qw = nqw * inv;
    s.vx = vx; s.vy = vy; s.vz = vz;
    s.wx = nwx; s.wy = nwy; s.wz = nwz;
}

}  // namespace h2o
