/*
 * h2o.h -- C ABI of the B200-native hydrodynamics force engine (libh2o_b200.so).
 *
 * Drop-in boundary for ONE path of Joagai23/silver2_isaacsim: the per-body, per-step
 * hydrodynamic force/torque evaluation.  Every entry point names the reference
 * interface it replaces (paths relative to /root/reference/src/scripts/physics/).
 *
 * Conventions
 *   - plain C: opaque handle, raw device pointers + sizes (or DLPack DLTensor*, see
 *     h2o_dlpack.h); no C++/torch types cross the boundary.
 *   - every function returns an h2o_status (0 = ok) and never throws;
 *     h2o_last_error() returns a thread-local message for the last failure.
 *   - all tensors are caller-owned, contiguous row-major, dtype == handle dtype,
 *     on the handle's device, 16-byte aligned.  The engine borrows them for the
 *     duration of the call (or until h2o_unbind for bound tensors) and never frees them.
 *     The engine owns only: coefficient records, previous-step velocities, statistics,
 *     captured graphs and pinned staging buffers.
 *   - every launch takes an explicit cudaStream_t (pass torch.cuda.current_stream().cuda_stream);
 *     there are no hidden synchronisations on the step path.
 *   - a handle is not re-entrant: one caller thread at a time
 *     (the reference is called serially from the PhysX step callback,
 *     hydrodynamics_behavior.py:131-141).
 */
#ifndef H2O_H_
#define H2O_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define H2O_API __attribute__((visibility("default")))
#else
#define H2O_API
#endif

typedef struct h2o_engine* h2o_handle;
typedef void* h2o_stream; /* cudaStream_t */

typedef enum {
    H2O_OK = 0,
    H2O_ERR_BAD_HANDLE = 1,
    H2O_ERR_BAD_ARGUMENT = 2,
    H2O_ERR_BAD_SHAPE = 3,
    H2O_ERR_BAD_DTYPE = 4,
    H2O_ERR_BAD_DEVICE = 5,
    H2O_ERR_NOT_CONTIGUOUS = 6,
    H2O_ERR_ALIGNMENT = 7,
    H2O_ERR_NOT_CONFIGURED = 8, /* parameters / bound tensors / rollout missing */
    H2O_ERR_CUDA = 9,
    H2O_ERR_NO_DEVICE = 10
} h2o_status;

typedef enum { H2O_F32 = 0, H2O_F64 = 1 } h2o_dtype;
typedef enum { H2O_QUAT_XYZW = 0, H2O_QUAT_WXYZ = 1 } h2o_quat_order;
typedef enum { H2O_KERNEL_AUTO = 0, H2O_KERNEL_TILE = 1, H2O_KERNEL_DIRECT = 2 } h2o_kernel_choice;

/* Number of scalars in one coefficient record and their order:
 * xDimension, yDimension, zDimension, linearDragCoefficient, angularDragCoefficient,
 * linearDamping, angularDamping, linearAddedMassCoefficient, angularAddedMassCoefficient,
 * liftCoefficient, mass      (names: hydrodynamics_behavior.py:28-46; mass: :172-173) */
#define H2O_N_COEFF 11
/* h2o_stats vector: sum|F|, max|F|, wet bodies, clamped bodies, non-finite forces,
 * wet-and-at-rest bodies (the reference raises there, numba_hydrodynamics.py:118,143),
 * bodies processed, bodies the fp32 fast path handed to the float64 re-evaluation. */
#define H2O_N_STATS 8

H2O_API const char* h2o_last_error(void);
H2O_API const char* h2o_version(void);
/* Number of CUDA devices visible, or a negative h2o_status. */
H2O_API int h2o_device_count(void);

/* ---- construction -------------------------------------------------------------------
 * Replaces XHydrodynamicsWrapper.__init__ (numba_hydrodynamics_wrapper.py:9-32,
 * warp_hydrodynamics_wrapper.py:10-77), batched over n_bodies, and
 * HydrodynamicsBehavior._setup (hydrodynamics_behavior.py:143-174). */
H2O_API int h2o_create(h2o_handle* out, int64_t n_bodies, int dtype, int device);
H2O_API int h2o_destroy(h2o_handle h);

/* waterDensity, gravity (hydrodynamics_behavior.py:30-31; hydrodynamics_config.json "globals") */
H2O_API int h2o_set_globals(h2o_handle h, double water_density, double gravity);

/* Non-flat water surface (SURVEY.md 8(f4)): eta is a DEVICE array (n_bodies,) in the handle's dtype
 * holding the surface elevation above surface_z at each body's position (e.g. a wave field sampled
 * by the caller); the model then sees p_z - surface_z - eta[i] where the reference uses p_z
 * (analyze_submersion_and_cob, numba_hydrodynamics.py:59-105, tests keypoints against z = 0).  The
 * pointer is borrowed and read by every later step until replaced (update the array in place between
 * steps; replacing the pointer drops a rollout captured with h2o_capture_rollout); NULL =
 * flat.  Steps with a height field run on the per-body kernel. */
H2O_API int h2o_set_surface_heights(h2o_handle h, const void* eta_dev);

/* Dense added mass (SURVEY.md 8(f4)).  calculate_added_mass (numba_hydrodynamics.py:219-253) takes
 * ANY 6x6 body-frame matrix M: f6 = -M [R^T a; R^T alpha], F = R f6[0:3] ratio, tau = R f6[3:6] ratio;
 * the wrapper only ever builds a diagonal one (numba_hydrodynamics_wrapper.py:101-112).  This call
 * installs n_types row-major 6x6 matrices (host, float64) and a slot -> matrix map: body i uses
 * matrices[slot_type[i % n_slots]] INSTEAD of the C_a / C_a_omega diagonal of its coefficient record.
 * slot_type may be NULL when n_types == 1.  n_types == 0 restores the diagonal.  Steps with dense
 * matrices run on the per-body kernel (H2O_KERNEL_DIRECT); h2o_components keeps the diagonal. */
H2O_API int h2o_set_added_mass_dense(h2o_handle h, int n_types, const double* matrices, int n_slots,
                                     const int32_t* slot_type);

/* Generalisation the reference's signatures admit but its scenes never use (SURVEY.md 8(f4)):
 * a uniform water current (drag, damping and lift then see v - current) and the height of the flat
 * water surface (the reference's is the plane z = 0).  NULL / 0 = the reference's behaviour. */
H2O_API int h2o_set_environment(h2o_handle h, const double current_xyz[3], double surface_z);

/* Built-in linear (Airy) wave field (SURVEY.md 8(f4)), evaluated on the device at every body's centre on every
 * step.  comps is n_components x 5 host doubles (a, kx, ky, omega, phase), depth the water depth h (+inf = deep
 * water).  For component j, with k_j = |(kx_j, ky_j)|, at body position p and clock value t:
 *   theta_j = kx_j p_x + ky_j p_y - omega_j t + phase_j                        (always float64)
 *   elevation  eta = sum_j a_j cos theta_j: the body's p_z is measured against the waterline surface_z + eta
 *              (+ eta[i] when a height field is also set, h2o_set_surface_heights)
 *   orbital velocity at z = clamp(p_z - surface_z, -h, 0) (measured from the mean level):
 *              u_h = sum_j a_j omega_j C_j(z) cos theta_j (kx_j, ky_j) / k_j,   u_z = sum_j a_j omega_j S_j(z) sin theta_j
 *              finite depth: C_j = cosh(k_j (z + h)) / sinh(k_j h),  S_j = sinh(k_j (z + h)) / sinh(k_j h)
 *              deep water:   C_j = S_j = exp(k_j z)
 * The orbital velocity adds to the uniform current: drag, damping and lift see v - (current + u), formed
 * exactly as the uniform current alone is.  As with the current: accelerations stay differences of BODY
 * velocities, the carried previous velocity stays the body velocity, and no fluid-acceleration
 * (Froude-Krylov inertia) term is added.
 * Precision: fp64 mode evaluates everything in double.  fp32 mode keeps the phase in double and evaluates
 * sine, cosine and the depth decay in float (field within 2e-6 of sum a_j resp. sum a_j omega_j).  eta enters
 * the waterline as a double, like surface_z; current + u is summed in double, rounded once to the handle dtype
 * and subtracted there.
 * Clock: one double in engine-owned device memory.  Every step evaluates the field at the clock's value, then
 * the clock advances by dt in stream order (no host synchronisation; also inside captured rollouts and the host
 * pipeline); a step with dt <= 1e-6 leaves it alone.  h2o_rollout_persistent over K steps uses t, t + dt, ...
 * and leaves the clock bit-identical to K single steps.  The clock starts at 0 and is kept when the field is
 * replaced or removed.
 * At most 64 components; n_components == 0 removes the field.  H2O_ERR_BAD_ARGUMENT for non-finite values,
 * a < 0, omega <= 0, |k| == 0 or depth <= 0 (other than +inf).  The table is copied to engine-owned device
 * memory.  Steps with a wave field run on the per-body kernel; h2o_components ignores the field (as it ignores
 * a height field).  Like every h2o_set_* call this drops a captured rollout. */
H2O_API int h2o_set_wave_field(h2o_handle h, int n_components, const double* comps, double depth);
/* The water clock (read by the wave field and by a time-varying current grid, h2o_set_current_grid),
 * stream-ordered.  The read synchronises the stream.  Neither drops a captured rollout: the graph
 * reads the clock from device memory, so a write between replays moves the field the replay sees. */
H2O_API int h2o_wave_time_write(h2o_handle h, double t, h2o_stream stream);
H2O_API int h2o_wave_time_read(h2o_handle h, double* t, h2o_stream stream);
/* Evaluate the field at the clock's current value with the evaluator and precision policy of the step:
 * points is a DEVICE array (m,3) in the handle dtype (world positions; the velocity depth is measured from
 * surface_z), out a DEVICE array (m,4) float64 of rows [eta, ux, uy, uz] (zeros without a field). */
H2O_API int h2o_wave_sample(h2o_handle h, const void* points, int64_t m, double* out, h2o_stream stream);
/* Wave-slope submersion: enable != 0 tests each body against the wave surface's local tangent plane instead of the
 * horizontal plane through its waterline W (the reference's model at the same level of approximation: its surface is
 * a plane, numba_hydrodynamics.py:59-105).  For a body at env-local (X, Y) and env time T (the theta_j of eta):
 *   sx = s sum_j (-a_j kx_j sin theta_j),   sy = s sum_j (-a_j ky_j sin theta_j)
 * with s the env's wave scale (1 without env conditions).  fp64 mode evaluates it in double; fp32 mode takes the
 * sine in float, as for u_z, and keeps the sums in double.  The slope is (0, 0) with the mode off, without a wave
 * field; the current grid, dz and a caller height array (h2o_set_surface_heights) contribute none.
 * A keypoint's height above the waterline becomes (p_z - W) + e . k, k its body-frame offset and
 *   e_c = (R_2c - sx R_0c) - sy R_1c          (double in both modes, c = x, y, z)
 * with R the rotation the mode uses (R(q), or R(q) + 2 dq I under Warp compatibility).  In the world frame: keypoint w
 * is wet iff w_z - W - sx (w_x - p_x) - sy (w_y - p_y) < 0.  z_min, z_max, the strict wet mask, the submersion ratio
 * and its cuts, the wetted faces (face-centre keypoints) and the centre of buoyancy (the mean of the wet keypoints)
 * are formed from these heights exactly as without slope.  The normal (-sx, -sy, 1) is deliberately not normalised:
 * every sign test and the ratio -z_min / (z_max - z_min) are invariant to its length.  The forces keep the
 * reference's formulas (buoyancy along +z, drag, lift, added mass); no fluid-acceleration term is added.
 * Default 0.  With no wave field the call changes nothing: steps and rollouts are bit-identical to a handle without
 * it.  With a field whose amplitudes are all zero, steps are bit-identical to the mode off; h2o_rollout_persistent
 * runs its own slope instantiation there, whose multiply-add contraction may differ: to rounding.  Every step path
 * that takes a wave field honours the mode (eager, bound, captured, host-buffer, h2o_rollout_persistent);
 * h2o_components ignores it, as it ignores the field.  Like every h2o_set_* call this drops a captured rollout. */
H2O_API int h2o_set_wave_slope(h2o_handle h, int enable);
/* Fluid-acceleration loads: enable != 0 adds the inertia part of Morison's equation, which dominates the wave loads
 * on bodies much smaller than the wavelength.  The fluid acceleration a_f is evaluated at the body centre, at the
 * (X, Y, Z, T) the flow is evaluated at (env-local position, depth below the env's mean level, env time):
 *   waves: a_w = sum_j a_j omega_j^2 (C_j sin theta_j khat_j, -S_j cos theta_j), the time derivative of the orbital
 *          velocity, with its theta_j, C_j, S_j and z clamp (fp32 mode: the same float sine, cosine and decay, double
 *          sums; within 2e-6 of sum a_j omega_j^2)
 *   grid:  a_g = (G_{f+1} - G_f) / ht for nt > 1 and T inside [t0, t0 + (nt - 1) ht], G_f and G_{f+1} the spatial
 *          interpolations of the two frames the interpolation in time blends (separately rounded float64
 *          operations); 0 where the grid is held in time, and for nt == 1
 *   a_f = a_g + s a_w, s the env's wave scale (1 without env conditions), every operation separately rounded.
 * The global and env currents are constant and the caller height array (h2o_set_surface_heights) moves no water:
 * they contribute nothing.  The convective term (u . grad) u is omitted (second order for linear waves), and so is
 * the rotation of the flow (Airy waves are irrotational).
 * With r the submersion ratio, V = dimx dimy dimz and rho = waterDensity, two terms join the net wrench before the
 * safety clamp:
 *   Froude-Krylov  F_FK = rho r V a_f at the centre of buoyancy: the torque gains (cob - p) x F_FK
 *   added mass     its linear part sees a_b - a_f in place of a_b: with the wrapper's diagonal (isotropic C_a rho V)
 *                  this adds C_a rho r V a_f at the body origin (no arm, like the added-mass force itself); with dense
 *                  matrices (h2o_set_added_mass_dense) it is M [R^T (a_b - a_f); R^T alpha_b], so the coupling block
 *                  turns a_f into a torque.  The angular part is unchanged.
 * Dry bodies (r = 0) get nothing.  a_b stays the reference's backward difference of body velocities
 * (hydrodynamics_behavior.py:196-202), half a step behind a_f.  fp32 mode counts both groups in the force and torque
 * conditioning checks, so bodies where they cancel drag or buoyancy are re-evaluated in float64.
 * Default 0.  With the mode off, or with no wave field and no grid with nt > 1, steps and rollouts run the code
 * without the mode and are bit-identical to a handle without it.  Every step path that takes a wave field honours the
 * mode (eager, bound, captured, host-buffer, h2o_rollout_persistent; h2o_reset_envs with restart_waves restarts an
 * env's a_f with its sea); h2o_components ignores it, as it ignores the field.  H2O_ERR_NOT_CONFIGURED when Warp
 * compatibility is on (and h2o_set_warp_compat refuses to turn it on while this mode is on): the Warp twin has no such
 * term.  Like every h2o_set_* call this drops a captured rollout; a refused call leaves it intact. */
H2O_API int h2o_set_fluid_inertia(h2o_handle h, int enable);

/* Per-env water conditions for vectorised scenes (SURVEY.md 8(f4)).  Envs are contiguous, equal runs of bodies:
 * body i (global index) belongs to env e = i / bodies_per_env, and E = n_bodies / bodies_per_env.  cond_dev is a
 * DEVICE array (E, 8) of float64 on the handle's device, 8-byte aligned, one row per env:
 *   cond[e] = [cx, cy, cz, dz, s, tau, x0, y0]
 *   cx, cy, cz  current added to the global current       dz      water-level offset added to surface_z
 *   s           wave scale (multiplies eta and u)         tau     wave time offset (s)
 *   x0, y0      env origin
 * For a body of env e at p with clock value t, every operation a separately rounded float64 operation:
 *   mean level  L_e = surface_z + dz
 *   theta_j   = ((kx_j (p_x - x0) + ky_j (p_y - y0)) - omega_j (t + tau)) + phase_j
 *   velocity depth z = clamp(p_z - L_e, -h, 0)
 *   waterline = L_e + s eta            (+ eta[i] when a height field is also set, h2o_set_surface_heights)
 *   flow      = (current + c_e) + s u  (fp32 mode: summed in double, rounded once to the handle dtype)
 * Without a wave field: waterline L_e, flow current + c_e.  The precision policies of h2o_set_wave_field hold.
 * The identity row [0,0,0,0,1,0,0,0] makes every operation exact: results are bit-identical to a handle without
 * conditions on the same kernel.
 * The array is borrowed, not copied: every later step reads it (a persistent rollout reads each row once at kernel
 * start), so the caller may update it in place between steps or graph replays with no recapture.  It must stay
 * allocated while set.  bodies_per_env == 0 or cond_dev == NULL removes the conditions.  H2O_ERR_BAD_SHAPE when
 * bodies_per_env does not divide n_bodies, H2O_ERR_ALIGNMENT / H2O_ERR_BAD_DEVICE for a misaligned pointer or one
 * not on the handle's device.  Steps with conditions run on the per-body kernel, as with a wave field;
 * h2o_rollout_persistent accepts them; h2o_components ignores them.  Like every h2o_set_* call this drops a
 * captured rollout; a refused call leaves it intact. */
H2O_API int h2o_set_env_conditions(h2o_handle h, int64_t bodies_per_env, const double* cond_dev);
/* Masked reset of the carried state (the per-env _reset, hydrodynamics_behavior.py:240-245), one stream-ordered
 * kernel without host synchronisation: env_mask_dev is a DEVICE array of E bytes; the carried [v, omega] of every
 * body of an env with mask[e] != 0 becomes zero.  restart_waves != 0 also writes cond[e][5] = -clock (read from the
 * device clock) for those envs, in the borrowed array, so that their next step sees their sea at env time exactly 0.
 * Other bodies and rows are left bit-unchanged.  Does not drop a captured rollout.  H2O_ERR_NOT_CONFIGURED without
 * conditions. */
H2O_API int h2o_reset_envs(h2o_handle h, const uint8_t* env_mask_dev, int restart_waves, h2o_stream stream);
/* h2o_wave_sample seen from envs: point k is evaluated for env env_index[k] (DEVICE int32 array (m,)) at the
 * clock's current value, through the step's evaluator.  out rows are [s eta, s ux, s uy, s uz]: the field alone
 * (c_e and dz are not added); zero rows without a wave field; a NaN row for an index outside [0, E).
 * H2O_ERR_NOT_CONFIGURED without conditions. */
H2O_API int h2o_wave_sample_env(h2o_handle h, const void* points, const int32_t* env_index, int64_t m, double* out,
                                h2o_stream stream);

/* Gridded water current (SURVEY.md 8(f4)): a space-time lattice of velocity vectors, such as an ocean-model or ADCP
 * field, a seabed boundary layer or a tidal sequence, interpolated on the device at every body on every step.
 * grid_dev is a C-contiguous DEVICE array of float64 with shape (nt, nz, ny, nx, 3) (dims = [nt, nz, ny, nx]) on the
 * handle's device, 8-byte aligned; geom = [gx, gy, gz, hx, hy, hz, t0, ht] (host).  Node (f, k, j, i) sits at
 * x = gx + i hx, y = gy + j hy, z = gz + k hz and at time t0 + f ht.
 * A body (or sample point) at p with water-clock value t is located, with L = surface_z + dz the env's mean level
 * (dz = 0, x0 = y0 = tau = 0 without env conditions):
 *   X = p_x - x0,  Y = p_y - y0  (env-local, as for waves)
 *   Z = p_z - L                  (from the env's mean level, not from the instantaneous waterline)
 *   T = t + tau                  (env time: h2o_reset_envs(..., restart_waves=1) also restarts an env's frames)
 * On each axis of n nodes, origin o and spacing h, at coordinate q: n == 1 gives index 0 and weight 0 (the axis is
 * constant and no neighbour is read); otherwise u = (q - o) / h clamped to [0, n - 1], i = min(floor(u), n - 2),
 * w = u - i.  Outside the lattice, and before the first or after the last frame, the value is held at the
 * boundary.  Each interpolation is lerp(a, b, w) = a + w (b - a), three separately rounded float64 operations,
 * along x, then y, then z, then t, for each component.  A NaN coordinate gives a NaN value; no input reads outside
 * the array.  The grid value g joins the flow, every addition a separately rounded float64 operation:
 *   flow = ((current + c_e) + g) + s u         (without env conditions: (current + g) + u)
 * fp32 mode sums the flow in double and rounds it once to the handle dtype.  The waterline is unchanged.  So a grid
 * of zeros gives the results of no grid, and a uniform grid of value g with a zero global current gives, bit for
 * bit, the results of no grid and h2o_set_environment(current = g) (h2o_rollout_persistent with a grid runs its own
 * kernel instantiation, whose multiply-add contraction may differ: to rounding there).  Only the model's inputs change, as for waves:
 * accelerations stay differences of body velocities and no fluid-acceleration term is added.
 * The array is borrowed, not copied: every later step reads it, so the caller may edit it in place between steps
 * or graph replays with no recapture (streaming new frames in).  It must stay allocated while set.
 * grid_dev == NULL removes the grid.  H2O_ERR_BAD_ARGUMENT for a dim < 1, a total size that overflows, non-finite
 * geometry, a spacing hx, hy, hz <= 0 or ht <= 0 with nt > 1; H2O_ERR_ALIGNMENT / H2O_ERR_BAD_DEVICE for a
 * misaligned pointer or one not on the handle's device.  Steps with a grid run on the per-body kernel;
 * h2o_rollout_persistent re-evaluates the grid at every step; h2o_components ignores it.  Like every h2o_set_* call
 * this drops a captured rollout; a refused call leaves it intact.
 * Water clock: the clock of h2o_wave_time_write / _read.  It advances by dt after every step (and by K dt after a
 * persistent rollout of K steps) whenever a wave field or a grid with nt > 1 is set. */
H2O_API int h2o_set_current_grid(h2o_handle h, const double* grid_dev, const int64_t dims[4], const double geom[8]);
/* What a step sees at given points and the clock's current value: points is a DEVICE array (m,3) in the handle
 * dtype, out a DEVICE array (m,4) float64 of rows [waterline, flow_x, flow_y, flow_z] -- the full composition of
 * global environment, env row, grid and wave field, before a caller height array (h2o_set_surface_heights) and
 * before the fp32 rounding.  env_index (DEVICE int32 (m,)) applies env env_index[k]'s row to point k; NULL applies
 * none; an index outside [0, E) gives a NaN row.  H2O_ERR_NOT_CONFIGURED for env_index without env conditions. */
H2O_API int h2o_water_sample(h2o_handle h, const void* points, const int32_t* env_index, int64_t m, double* out,
                             h2o_stream stream);
/* The surface slope a step uses at given points and the clock's current value (h2o_set_wave_slope): points as for
 * h2o_water_sample, out a DEVICE array (m,2) float64 of rows [sx, sy]; zero rows with the mode off or without a wave
 * field.  env_index as for h2o_water_sample: a NaN row for an index outside [0, E), H2O_ERR_NOT_CONFIGURED for
 * env_index without env conditions. */
H2O_API int h2o_water_slope_sample(h2o_handle h, const void* points, const int32_t* env_index, int64_t m, double* out,
                                   h2o_stream stream);
/* The fluid acceleration a_f a step uses at given points and the clock's current value (h2o_set_fluid_inertia):
 * points as for h2o_water_sample, out a DEVICE array (m,3) float64 of rows [ax, ay, az]; zero rows with the mode off
 * or with neither a wave field nor a grid with nt > 1.  env_index as for h2o_water_sample: a NaN row for an index
 * outside [0, E), H2O_ERR_NOT_CONFIGURED for env_index without env conditions. */
H2O_API int h2o_fluid_accel_sample(h2o_handle h, const void* points, const int32_t* env_index, int64_t m, double* out,
                                   h2o_stream stream);

/* Same twelve scalars, same order as the reference wrapper ctor
 * (numba_hydrodynamics_wrapper.py:9-10): width, depth, height, linear_drag_coefficient,
 * angular_drag_coefficient, linear_damping, angular_damping, water_density, gravity,
 * linear_mass_coeff, angular_mass_coeff, lift_coefficient; plus the body mass used by the
 * safety clamp (hydrodynamics_behavior.py:172-173, :221-226).  Applies to every body. */
H2O_API int h2o_set_params_uniform(h2o_handle h, const double ctor12[12], double mass);

/* Part-type table (hydrodynamics_config.json "parts"): table is n_types x H2O_N_COEFF host
 * doubles; slot_type[n_slots] maps body slot (global body index mod n_slots) to a type.
 * The table is staged in shared memory by the kernels. */
H2O_API int h2o_set_part_table(h2o_handle h, int n_types, const double* table_host, int n_slots,
                               const int32_t* slot_type_host);

/* Heterogeneous per-body records: coeff is (n_bodies, H2O_N_COEFF), host or device memory,
 * src_dtype H2O_F32/H2O_F64 (converted to the handle dtype on the device). */
H2O_API int h2o_set_params_per_body(h2o_handle h, const void* coeff, int src_dtype, h2o_stream stream);

/* Same, struct-of-arrays: cols[k] is a DEVICE array (n_bodies,) holding coefficient k of every body, in
 * H2O_N_COEFF order (xDimension, yDimension, zDimension, linearDragCoefficient, angularDragCoefficient,
 * linearDamping, angularDamping, linearAddedMassCoefficient, angularAddedMassCoefficient,
 * liftCoefficient -- the per-prim exposed variables of hydrodynamics_behavior.py:32-44 -- and mass, the
 * one _setup reads from the view, :172-174).  Interleaved into the engine's records on the device. */
H2O_API int h2o_set_params_soa(h2o_handle h, const void* const cols[11], int src_dtype, h2o_stream stream);

/* Articulation structure: bodies are grouped in contiguous runs of bodies_per_robot;
 * 0 disables the per-robot wrench. */
H2O_API int h2o_set_articulation(h2o_handle h, int bodies_per_robot);

/* Articulation of UNEQUAL robots (e.g. the reference's main scene: one 19-link SILVER2 plus the Obsea
 * buoy as a robot of its own): robot r owns bodies [offsets[r], offsets[r+1]); offsets is a host array
 * of n_robots + 1 entries, offsets[0] = 0, offsets[n_robots] = n_bodies, strictly increasing.  The
 * out_robot_wrench of the step calls is then (n_robots, 6), each wrench about its robot's first body,
 * reduced from the written force / torque arrays after the force kernel.  h2o_set_articulation
 * replaces it again.  Not available through h2o_step_host. */
H2O_API int h2o_set_articulation_offsets(h2o_handle h, int64_t n_robots, const int64_t* offsets);

/* Isaac core hands quaternions as wxyz and the reference permutes them
 * (hydrodynamics_behavior.py:194); the wrappers themselves take xyzw. */
H2O_API int h2o_set_quat_order(h2o_handle h, int order);
H2O_API int h2o_set_kernel(h2o_handle h, int choice);
/* Follow the reference's WARP twin instead of its Numba path (warp_hydrodynamics.py; SURVEY.md Appendix C;
 * pinned by tests/golden/reference_warp_golden.npz, vectors of the reference's own kernel source): accelerations
 * rotated forward instead of inverse for the added-mass terms (:216-217), every rotation by wp.quat_rotate
 * (= R(q) + 2(|q|^2 - 1) I for an un-normalised quaternion), centre of buoyancy = mean of the wet keypoints also
 * when fully submerged (:57-58), cob = cop = position for a dry body (:59-61, :290).  Applies to h2o_components
 * and to the fused step entry points (the production behaviour script evaluates forces through the Warp wrapper,
 * hydrodynamics_behavior.py:19, :155); the step then runs every body through the float64 formulation on the
 * per-body kernel (a compatibility mode, not a fast path).  Default 0 = the Numba semantics (north star).
 * H2O_ERR_NOT_CONFIGURED for enable != 0 while h2o_set_fluid_inertia is on. */
H2O_API int h2o_set_warp_compat(h2o_handle h, int enable);
/* fp32 mode only.  1 (default): every body meets the fp32-mode bound of the parity criterion (|dF|, |dtau| <=
 * max(1e-5 |.|_inf, 1e-6) against the float64 Numba path): the fused step flags the few bodies per 10 000 whose
 * force / torque groups cancel (or whose quaternion is far from unit) and re-evaluates them in float64 with the
 * world-frame formulation of solve_hydrodynamics (numba_hydrodynamics.py:255-314).  0: flagged bodies keep their
 * fp32 result (about one body per million then misses the bound by up to 3x); saves the re-evaluation tail. */
H2O_API int h2o_set_strict(h2o_handle h, int enable);
/* Tuning knob: tile-kernel variant (threads per CTA / TMA stages); 0 = built-in default. */
H2O_API int h2o_set_tile_config(h2o_handle h, int cfg);
/* Accumulate global statistics inside the step kernel (device-side, no host sync). */
H2O_API int h2o_enable_stats(h2o_handle h, int enable);

/* ---- carried state ------------------------------------------------------------------
 * _last_linear_velocity / _last_angular_velocity (hydrodynamics_behavior.py:196-198,
 * :237-238).  h2o_reset mirrors _reset (:240-245): the next step sees zeros. */
H2O_API int h2o_reset(h2o_handle h, h2o_stream stream);
H2O_API int h2o_set_prev(h2o_handle h, const void* prev_lin, const void* prev_ang, h2o_stream stream);
H2O_API int h2o_get_prev(h2o_handle h, void* prev_lin, void* prev_ang, h2o_stream stream);

/* ---- fused step ---------------------------------------------------------------------
 * Replaces HydrodynamicsBehavior._apply_behavior (hydrodynamics_behavior.py:194-238) for all
 * bodies at once: quaternion reorder, finite-difference acceleration, every force term,
 * body-relative lever arms, net wrench, safety clamp, previous-velocity update.
 *   pos (N,3) quat (N,4) lin_vel (N,3) ang_vel (N,3)  ->  out_force (N,3) out_torque (N,3)
 *   out_robot_wrench: (N / bodies_per_robot, 6) [F, tau about the robot's slot-0 body] or NULL.
 * dt <= 1e-6 is a successful no-op (hydrodynamics_behavior.py:139). */
H2O_API int h2o_step(h2o_handle h, const void* pos, const void* quat, const void* lin_vel,
                     const void* ang_vel, double dt, void* out_force, void* out_torque,
                     void* out_robot_wrench, h2o_stream stream);

/* Same, PhysX tensor-API layout: transforms (N,7) = [p, q], velocities (N,6) = [v, w]
 * (RigidPrimView.get_world_poses / get_velocities, hydrodynamics_behavior.py:178-189). */
H2O_API int h2o_step_physx(h2o_handle h, const void* transforms, const void* velocities, double dt,
                           void* out_force, void* out_torque, void* out_robot_wrench,
                           h2o_stream stream);

/* Same, RigidPrimView layout: pos (N,3), quat (N,4) from get_world_poses and the fused
 * velocities (N,6) = [v, w] from get_velocities (hydrodynamics_behavior.py:178-189) -- no slicing
 * copies on the caller's side. */
H2O_API int h2o_step_view(h2o_handle h, const void* pos, const void* quat, const void* velocities, double dt,
                          void* out_force, void* out_torque, void* out_robot_wrench, h2o_stream stream);

/* Bind the tensors once, then step with a single cheap call (layout: 0 split, 1 physx, 2 view;
 * physx: pass transforms as pos, velocities as lin_vel, quat = ang_vel = NULL;
 * view: pass velocities as lin_vel, ang_vel = NULL). */
H2O_API int h2o_bind(h2o_handle h, int layout, const void* pos, const void* quat, const void* lin_vel,
                     const void* ang_vel, void* out_force, void* out_torque, void* out_robot_wrench);
H2O_API int h2o_unbind(h2o_handle h);
H2O_API int h2o_step_bound(h2o_handle h, double dt, h2o_stream stream);

/* CUDA-graph rollout over the bound tensors: n_steps back-to-back steps captured once,
 * replayed with one launch (the reference captures a single dim=1 kernel,
 * warp_hydrodynamics_wrapper.py:101-120).  Capturing launches nothing: the carried velocities and
 * (free-body mode) the bound state are exactly as before the call.  The graph bakes in the engine's
 * device buffers and constants, so every h2o_set_* / h2o_enable_stats / h2o_bind / h2o_unbind call drops
 * it: h2o_launch_rollout then returns H2O_ERR_NOT_CONFIGURED until the rollout is captured again. */
H2O_API int h2o_capture_rollout(h2o_handle h, int n_steps, double dt, h2o_stream stream);
/* Rollout mode: 0 = static state (force-only rollout), 1 = free bodies: after each step the bound
 * pose / velocity tensors are integrated in place by h2o_integrate_free_bodies (split layout). */
H2O_API int h2o_set_rollout_mode(h2o_handle h, int free_bodies, double gravity);
H2O_API int h2o_launch_rollout(h2o_handle h, h2o_stream stream);

/* Persistent rollout of FREE bodies over the bound tensors (split layout): n_steps x (fused force step ->
 * h2o_integrate_free_bodies) in ONE kernel launch, each thread carrying its body's pose, velocities,
 * previous velocities and coefficients in registers across the steps (bodies are independent:
 * solve_hydrodynamics reads only its own body, numba_hydrodynamics.py:255-314; the behaviour's per-step
 * bookkeeping is hydrodynamics_behavior.py:196-238).  Same result as h2o_capture_rollout in free-body mode
 * (up to FMA contraction) without a launch / graph node per step.  On return of the kernel the bound pose /
 * velocity tensors and the carried velocities hold the final state, out_force / out_torque the last step's
 * wrench.  trace_every > 0: every trace_every-th step a row [p, v, w] (9 scalars, handle dtype) per body
 * goes to trace_out, a device array (n_steps / trace_every, n_bodies, 9) -- the columns of the
 * reference's velocity logger (log_velocity.py:17-20); trace_every > n_steps (no row) is H2O_ERR_BAD_ARGUMENT.
 * The kernel follows the Numba semantics and has no robot-wrench output, so a handle with h2o_set_warp_compat
 * on, or bound with an out_robot_wrench, gets H2O_ERR_NOT_CONFIGURED (h2o_capture_rollout honours both), as
 * does one with dense added mass or a caller height field.  dt <= 1e-6 is a successful no-op. */
H2O_API int h2o_rollout_persistent(h2o_handle h, int n_steps, double dt, double gravity, int trace_every,
                                   void* trace_out, h2o_stream stream);

/* ---- stand-alone free-body stepper (harness; the reference leaves integration to PhysX) ------
 * Semi-implicit Euler for free boxes (mass and dimensions from the coefficient records, box
 * inertia, gravity along -z): velocities first, then pose; all four state tensors updated in place. */
H2O_API int h2o_integrate_free_bodies(h2o_handle h, void* pos, void* quat, void* lin_vel, void* ang_vel,
                                      const void* force, const void* torque, double dt, double gravity,
                                      h2o_stream stream);

/* ---- full-signature components --------------------------------------------------------
 * Replaces XHydrodynamicsWrapper.calculate_hydrodynamic_forces
 * (numba_hydrodynamics_wrapper.py:34-53, warp_hydrodynamics_wrapper.py:79-132) =
 * solve_hydrodynamics (numba_hydrodynamics.py:255-314), batched.  Outputs in the reference's
 * order: buoyancy_force, drag_force, lift_force, drag_torque, added_mass_force,
 * added_mass_torque, center_of_buoyancy, center_of_pressure (each (N,3)), sub_ratio (N,).
 * out_flags (N, int32, may be NULL): bit0 set where the unmodified reference raises TypeError
 * (wet body with speed <= 1e-6); the engine returns cop = cob, area = 0 there. */
H2O_API int h2o_components(h2o_handle h, const void* pos, const void* quat, const void* lin_vel,
                           const void* ang_vel, const void* lin_acc, const void* ang_acc,
                           void* const out8[8], void* out_sub_ratio, int32_t* out_flags,
                           h2o_stream stream);

/* ---- host-buffer path --------------------------------------------------------------------
 * Numba-wrapper style call with HOST arrays (the reference's CPU flavour takes and returns NumPy arrays,
 * numba_hydrodynamics_wrapper.py:34-53).  Synchronous: ordered after the work queued before on the
 * blocking streams (an event on the legacy default stream, no device-wide synchronisation), returns when
 * the results are in the host buffers.
 *   - pinned (page-locked) host buffers, 16-byte aligned: ZERO-COPY.  The fused tile kernel runs directly on
 *     them: its TMA bulk loads pull each tile over PCIe into shared memory, its bulk stores push force /
 *     torque back -- one kernel, transfers overlapped with the arithmetic tile by tile, no staging copy.
 *   - pageable buffers: staged through engine-owned pinned memory, chunked H2D -> step -> D2H pipeline on
 *     three streams.
 * h2o_last_host_path reports which one the last call took (1 zero-copy, 2 staged). */
H2O_API int h2o_step_host(h2o_handle h, const void* pos, const void* quat, const void* lin_vel,
                          const void* ang_vel, double dt, void* out_force, void* out_torque,
                          void* out_robot_wrench);
/* Same with the PhysX tensor-API layout on the host: transforms (N,7) = [p, q], velocities (N,6) = [v, w]
 * (what RigidPrimView.get_world_poses / get_velocities hand out when the simulation runs on the CPU,
 * hydrodynamics_behavior.py:178-189): two input arrays instead of four. */
H2O_API int h2o_step_host_physx(h2o_handle h, const void* transforms, const void* velocities, double dt,
                                void* out_force, void* out_torque, void* out_robot_wrench);
H2O_API int h2o_last_host_path(h2o_handle h);

/* ---- statistics / introspection ----------------------------------------------------------- */
H2O_API int h2o_stats_device_ptr(h2o_handle h, void** out_ptr); /* H2O_N_STATS doubles on device */
H2O_API int h2o_read_stats(h2o_handle h, double out[H2O_N_STATS], int reset, h2o_stream stream);
H2O_API int64_t h2o_launch_count(h2o_handle h); /* kernels launched (or graph nodes replayed) so far */
H2O_API int64_t h2o_n_bodies(h2o_handle h);
H2O_API int h2o_dtype_of(h2o_handle h);
/* Which kernel the last step used: H2O_KERNEL_TILE or H2O_KERNEL_DIRECT. */
H2O_API int h2o_last_kernel(h2o_handle h);
/* Resident CTAs per SM of the last tile-kernel launch (occupancy query result). */
H2O_API int h2o_last_ctas_per_sm(h2o_handle h);
/* Device pointers of engine-owned buffers (zero-copy views for DLPack export on the host side). */
H2O_API int h2o_prev_device_ptr(h2o_handle h, void** out_ptr);  /* (N,6) */
H2O_API int h2o_coeff_device_ptr(h2o_handle h, void** out_ptr, int64_t* out_rows); /* (rows,11) */

#ifdef __cplusplus
}
#endif
#endif /* H2O_H_ */
