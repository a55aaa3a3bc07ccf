// Host-side instantiation of the free-body stepper of silver2_isaacsim_b200/csrc/h2o_model.cuh (free_body_update).
//
// TEST TOOL ONLY: lets the CPU-only tests (tests/test_free_body.py) run the integrator that free_body_kernel and the
// persistent rollout kernel inline against the float64 NumPy reference (oracle/free_body.py), without a GPU.  It is
// not part of the package, is not loaded by any product module and is not a fallback path.
#include <cstdint>

#include "../../silver2_isaacsim_b200/csrc/h2o_model.cuh"

using namespace h2o;

// One step of n boxes, in place: p (n,3), q (n,4) xyzw, v (n,3), w (n,3) from the world-frame wrench F (n,3),
// T (n,3), masses m (n,) and dimensions dims (n,3).
extern "C" __attribute__((visibility("default")))
int emul_free_body_step(int64_t n, double* p, double* q, double* v, double* w, const double* F, const double* T,
                        const double* m, const double* dims, double dt, double gravity)
{
    for (int64_t i = 0; i < n; ++i) {
        FreeBodyState s;
        s.px = p[3 * i]; s.py = p[3 * i + 1]; s.pz = p[3 * i + 2];
        s.qx = q[4 * i]; s.qy = q[4 * i + 1]; s.qz = q[4 * i + 2]; s.qw = q[4 * i + 3];
        s.vx = v[3 * i]; s.vy = v[3 * i + 1]; s.vz = v[3 * i + 2];
        s.wx = w[3 * i]; s.wy = w[3 * i + 1]; s.wz = w[3 * i + 2];
        const double* f = F + 3 * i;
        const double* t = T + 3 * i;
        const double* d = dims + 3 * i;
        free_body_update(s, f[0], f[1], f[2], t[0], t[1], t[2], m[i], d[0], d[1], d[2], dt, gravity);
        p[3 * i] = s.px; p[3 * i + 1] = s.py; p[3 * i + 2] = s.pz;
        q[4 * i] = s.qx; q[4 * i + 1] = s.qy; q[4 * i + 2] = s.qz; q[4 * i + 3] = s.qw;
        v[3 * i] = s.vx; v[3 * i + 1] = s.vy; v[3 * i + 2] = s.vz;
        w[3 * i] = s.wx; w[3 * i + 1] = s.wy; w[3 * i + 2] = s.wz;
    }
    return 0;
}
