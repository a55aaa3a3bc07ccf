// Host-side instantiation of the current-grid evaluator of silver2_isaacsim_b200/csrc/h2o_waves.cuh (grid_eval) and
// of the composition that uses it (water_at).
//
// TEST TOOL ONLY: lets the CPU-only tests (tests/test_current_grid.py) run the code the CUDA kernels inline against
// the NumPy reference (silver2_isaacsim_b200/currents.py), without a GPU.  It is not part of the package, is not
// loaded by any product module and is not a fallback path.
#include <cstdint>

#include "../../silver2_isaacsim_b200/csrc/h2o_waves.cuh"

using namespace h2o;

static GridArgs grid_of(const int64_t dims[4], const double* vals, const double geom[8])
{
    GridArgs g;
    g.vals = vals;
    g.nt = dims[0]; g.nz = dims[1]; g.ny = dims[2]; g.nx = dims[3];
    g.gx = geom[0]; g.gy = geom[1]; g.gz = geom[2]; g.hx = geom[3]; g.hy = geom[4]; g.hz = geom[5];
    g.t0 = geom[6]; g.ht = geom[7];
    return g;
}

// grid (dims [nt, nz, ny, nx], values (nt, nz, ny, nx, 3), geometry [gx, gy, gz, hx, hy, hz, t0, ht]) at grid-frame
// points (x, y, z, t)[i] -> out (m,3).
extern "C" __attribute__((visibility("default")))
int emul_current_eval(const int64_t* dims, const double* vals, const double* geom, int64_t m, const double* x,
                      const double* y, const double* z, const double* t, double* out)
{
    const GridArgs g = grid_of(dims, vals, geom);
    for (int64_t i = 0; i < m; ++i) grid_eval(g, x[i], y[i], z[i], t[i], out + 3 * i);
    return 0;
}

// water_at at points (m,3) and clock t: the global environment (current, surface_z), the row of env env_index[i]
// of cond (n_envs, ENV_STRIDE) (env_index == nullptr: no row; an index outside [0, n_envs) gives NaN rows), the
// grid (vals == nullptr: none) and n wave components -> field (m,4) [s eta, s u] and water (m,4) [waterline, flow].
extern "C" __attribute__((visibility("default")))
int emul_water(int f32, int n, const double* comps, double depth, const int64_t* dims, const double* vals,
               const double* geom, int64_t m, const double* points, const int32_t* env_index, int64_t n_envs,
               const double* cond, double t, double surface_z, const double* current, double* field, double* water)
{
    if (n < 0 || n > MAX_WAVE_COMPONENTS) return 1;
    double tab[MAX_WAVE_COMPONENTS * WAVE_STRIDE];
    for (int j = 0; j < n; ++j) wave_table_row(comps + 5 * j, depth, tab + WAVE_STRIDE * j);
    GridArgs g{};
    if (vals) g = grid_of(dims, vals, geom);
    for (int64_t i = 0; i < m; ++i) {
        const double* p = points + 3 * i;
        EnvRow row{};
        if (env_index) {
            const int64_t e = env_index[i];
            if (e < 0 || e >= n_envs) {
                for (int k = 0; k < 4; ++k) field[4 * i + k] = water[4 * i + k] = __builtin_nan("");
                continue;
            }
            row = env_row(cond, e);
        }
        const GridArgs* gp = vals ? &g : nullptr;
        const bool has_row = env_index != nullptr;
        const Water w = f32 ? water_at<true>(current, surface_z, has_row, row, tab, n, depth, t, p[0], p[1], p[2], gp)
                            : water_at<false>(current, surface_z, has_row, row, tab, n, depth, t, p[0], p[1], p[2], gp);
        field[4 * i] = w.field.eta; field[4 * i + 1] = w.field.ux; field[4 * i + 2] = w.field.uy;
        field[4 * i + 3] = w.field.uz;
        water[4 * i] = w.surface_z; water[4 * i + 1] = w.cx; water[4 * i + 2] = w.cy; water[4 * i + 3] = w.cz;
    }
    return 0;
}
