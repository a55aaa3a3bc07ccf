// Host-side instantiation of silver2_isaacsim_b200/csrc/h2o_waves.cuh.
//
// TEST TOOL ONLY: lets the CPU-only tests (tests/test_waves.py) run the wave evaluator the CUDA kernels
// inline (same header, same precision policies) against the NumPy reference, without a GPU.  It is not part
// of the package, is not loaded by any product module and is not a fallback path.
#include <cstdint>

#include "../../silver2_isaacsim_b200/csrc/h2o_waves.cuh"

using namespace h2o;

// Wave field at points (m,3) and clock t -> out (m,4) [eta, ux, uy, uz]; comps (n,5) as passed to
// h2o_set_wave_field.  f32 = 1: the fp32-mode policy (host float sin / cos / exp standing in for the MUFU forms).
extern "C" __attribute__((visibility("default")))
int emul_wave_sample(int f32, int n, const double* comps, double depth, int64_t m, const double* points, double t,
                     double surface_z, double* out)
{
    if (n < 0 || n > MAX_WAVE_COMPONENTS) return 1;
    double tab[MAX_WAVE_COMPONENTS * WAVE_STRIDE];
    for (int j = 0; j < n; ++j) wave_table_row(comps + 5 * j, depth, tab + WAVE_STRIDE * j);
    for (int64_t i = 0; i < m; ++i) {
        const double* p = points + 3 * i;
        const WaveSample w = f32 ? wave_eval<true>(tab, n, depth, p[0], p[1], p[2] - surface_z, t)
                                 : wave_eval<false>(tab, n, depth, p[0], p[1], p[2] - surface_z, t);
        out[4 * i] = w.eta; out[4 * i + 1] = w.ux; out[4 * i + 2] = w.uy; out[4 * i + 3] = w.uz;
    }
    return 0;
}
