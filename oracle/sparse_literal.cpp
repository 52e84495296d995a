// oracle/sparse_literal.cpp — TEST INFRASTRUCTURE ONLY.
//
// A literal restatement of model::SparsifiedGP::_sparsify (src/limbo/model/sparsified_gp.hpp:126-183), the checker of
// limbo_b200/csrc/sparsify.cu.  It shares nothing with the incremental device algorithm: the full distance matrix is
// built once, and every removal recomputes the density of EVERY remaining row by partial-sorting it, then takes the
// first row of strictly smaller density in index order (the reference's sequential tools::par::loop).  Erasing a row
// and column of the matrix is restated as erasing the entry from the list of remaining original indices, which keeps
// their relative order as std::vector::erase does.  Rows are scored on several threads; the argmin stays sequential.
//
// Built with -ffp-contract=off: the distance is sqrt of the sum, from 0 and in order d = 0..D-1, of separately rounded
// squares of differences, as (samples[i] - samples[j]).norm() computes it through oracle/ref_shim/Eigen/Core.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <limits>
#include <thread>
#include <vector>

extern "C" int sparse_literal(long N, int D, const double* X, long max_points, int64_t* keep, int64_t* removed,
    double* removed_density, int nthreads)
{
    if (N < 1 || D < 1 || max_points < D) return -1;
    std::vector<double> dist((size_t)N * N, 0.0);
    for (long i = 0; i < N; ++i)
        for (long j = 0; j < N; ++j) {
            if (i == j) continue;
            double s = 0.0;
            for (int d = 0; d < D; ++d) {
                const double t = X[i * D + d] - X[j * D + d];
                s += t * t;
            }
            dist[(size_t)i * N + j] = std::sqrt(s);
        }
    std::vector<long> live(N);
    for (long i = 0; i < N; ++i) live[i] = i;
    if (nthreads < 1) nthreads = std::max(1u, std::thread::hardware_concurrency());
    std::vector<double> dens(N);
    long t = 0;
    while ((long)live.size() > max_points) {
        const long n = (long)live.size();
        auto score = [&](long i0, long i1) {
            std::vector<double> neighbors;
            for (long i = i0; i < i1; ++i) {
                neighbors.clear();
                for (long j = 0; j < n; ++j)
                    if (j != i) neighbors.push_back(dist[(size_t)live[i] * N + live[j]]);
                std::partial_sort(neighbors.begin(), neighbors.begin() + D, neighbors.end());
                double s = 0.;
                for (int j = 0; j < D; ++j) s += neighbors[j];
                dens[i] = s;
            }
        };
        const long nt = std::min<long>(nthreads, std::max<long>(1, n / 64));
        std::vector<std::thread> pool;
        for (long w = 0; w < nt; ++w) pool.emplace_back(score, n * w / nt, n * (w + 1) / nt);
        for (auto& th : pool) th.join();
        double min_dist = std::numeric_limits<double>::max();
        long denser = -1;
        for (long i = 0; i < n; ++i)
            if (dens[i] < min_dist) {
                min_dist = dens[i];
                denser = i;
            }
        if (denser < 0) return -2;
        if (removed) removed[t] = live[denser];
        if (removed_density) removed_density[t] = min_dist;
        live.erase(live.begin() + denser);
        ++t;
    }
    for (size_t i = 0; i < live.size(); ++i) keep[i] = live[i];
    return 0;
}
