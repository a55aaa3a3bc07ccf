// Host-side instantiation of the per-env composition of silver2_isaacsim_b200/csrc/h2o_waves.cuh (water_at).
//
// TEST TOOL ONLY: lets the CPU-only tests (tests/test_env_conditions.py) run the code the CUDA kernels inline to
// form each body's waterline and flow from the global environment, an env conditions row, the wave table and the
// clock, against the NumPy reference, without a GPU.  It is not part of the package, is not loaded by any product
// module and is not a fallback path.
#include <cstdint>

#include "../../silver2_isaacsim_b200/csrc/h2o_waves.cuh"

using namespace h2o;


// The wave field seen from envs, through water_at (the composition every step kernel runs): point i of env
// env_index[i] (rows of cond (n_envs, ENV_STRIDE)) -> field (m,4) [s eta, s ux, s uy, s uz], a NaN row for an
// index outside [0, n_envs); water (m,4) [waterline, flow x, y, z] with the global current, or nullptr.
extern "C" __attribute__((visibility("default")))
int emul_wave_sample_env(int f32, int n, const double* comps, double depth, int64_t m, const double* points,
                         const int32_t* env_index, int64_t n_envs, const double* cond, double t, double surface_z,
                         const double* current, double* field, double* water)
{
    if (n < 0 || n > MAX_WAVE_COMPONENTS) return 1;
    double tab[MAX_WAVE_COMPONENTS * WAVE_STRIDE];
    for (int j = 0; j < n; ++j) wave_table_row(comps + 5 * j, depth, tab + WAVE_STRIDE * j);
    for (int64_t i = 0; i < m; ++i) {
        const double* p = points + 3 * i;
        const int64_t e = env_index[i];
        if (e < 0 || e >= n_envs) {
            for (int k = 0; k < 4; ++k) field[4 * i + k] = __builtin_nan("");
            if (water)
                for (int k = 0; k < 4; ++k) water[4 * i + k] = __builtin_nan("");
            continue;
        }
        const EnvRow row = env_row(cond, e);
        const Water w = f32 ? water_at<true>(current, surface_z, true, row, tab, n, depth, t, p[0], p[1], p[2])
                            : water_at<false>(current, surface_z, true, row, tab, n, depth, t, p[0], p[1], p[2]);
        field[4 * i] = w.field.eta; field[4 * i + 1] = w.field.ux; field[4 * i + 2] = w.field.uy;
        field[4 * i + 3] = w.field.uz;
        if (water) {
            water[4 * i] = w.surface_z; water[4 * i + 1] = w.cx; water[4 * i + 2] = w.cy; water[4 * i + 3] = w.cz;
        }
    }
    return 0;
}
