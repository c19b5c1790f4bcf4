// emu_power_posterior.cpp -- host versions of the power-posterior launchers of csrc/backend.h (launch_power_posterior,
// launch_temper_weights), for the host-only test double.
//
// Test infrastructure, not a product path: tests/test_power_posterior.py compiles this file together with
// tests/emu/emu_backend.cpp, csrc/engine.cpp and csrc/planner.cpp into a test double of its own.  The two launchers are
// declared weak in backend.h, so the plain test double (tests/emu/Makefile), which does not define them, still loads and
// refuses demcmc_set_temperatures with DEMCMC_EUNSUPPORTED.  Each function honours the contract of the CUDA kernel it
// stands for (k_power_posterior, k_temper_weights); the sums run serially.
#include <math.h>
#include <algorithm>

#include "backend.h"
#include "de_particle.h"

namespace de {
namespace be {

// contract of k_power_posterior: per (local group, slice of PP_ROWS rows) the six partials of de_types.h: PP_OUT
int launch_power_posterior(const double *ll, int64_t row0, int64_t n_rows, int32_t P, int32_t Np, int32_t G_local, const PPDelta &delta, double *part)
{
    const int64_t n_slices = (n_rows + PP_ROWS - 1) / PP_ROWS;
    for (int g = 0; g < G_local; ++g)
        for (int64_t s = 0; s < n_slices; ++s) {
            const int64_t r0 = row0 + s * PP_ROWS, nr = std::min<int64_t>(PP_ROWS, row0 + n_rows - r0);
            auto at = [&](int64_t r, int j) { return ll[(r0 + r) * P + (size_t)g * Np + j]; };
            double sum = 0.0, mx = -INFINITY;
            for (int64_t r = 0; r < nr; ++r) for (int j = 0; j < Np; ++j) { sum += at(r, j); mx = fmax(mx, at(r, j)); }
            const double n = (double)(nr * Np), mean = sum / n, dl = delta.v[g];
            double m2 = 0.0, e1 = 0.0, e2 = 0.0;
            for (int64_t r = 0; r < nr; ++r)
                for (int j = 0; j < Np; ++j) { const double v = at(r, j), x = exp(dl * (v - mx)); m2 += (v - mean) * (v - mean); e1 += x; e2 += x * x; }
            double *o = part + ((size_t)g * n_slices + s) * PP_OUT;
            o[0] = n; o[1] = mean; o[2] = m2; o[3] = mx; o[4] = e1; o[5] = e2;
        }
    return 0;
}

// contract of k_temper_weights
int launch_temper_weights(const ConfigDev &cfg, const double *prior, const double *ll, int64_t n, double *w)
{
    for (int64_t p = 0; p < n; ++p)
        w[p] = prior[p] == -inf() ? -inf() : add(prior[p], tempered_ll(cfg, cfg.group_begin + (int)(p / cfg.Np), ll[p]));
    return 0;
}

} // namespace be
} // namespace de
