// tests/native/interval_sa_ref.cpp -- TEST INFRASTRUCTURE: CPU reference for interval rank-1 groups.
//
// The same simulated-annealing loop as oracle/cpu_sa_ref.cpp (neal's simulated_annealing_run: xorshift128+, threshold
// 44.36142 / beta, exp(-dE * beta) * 2^64 > rand, eager neighbour updates) with the group term generalised from "squared
// distance to a point" to "squared distance to an interval" (include/qanneal.h, qa_model_set_group_bounds):
//     u = sum_{v in g} a_v s_v + kappa_g,  d(u) = max(lo_g - u, 0, u - hi_g),  E_g = lambda_g * (double)(d*d) * 0.25
//     flip (s, a): u' = u - 2 a s,  dE_g = lambda_g * ((double)(d(u')^2 - d(u)^2) * 0.25)
// Null bounds are the equality groups of the oracle (lambda * (double)(a * (a - s u)) per flip), evaluated exactly as there,
// so this file reproduces the oracle bit for bit on every model the oracle accepts (tests/test_interval_groups_cpu.py).
// Per-read seeding only (neal num_samples = 1 per read).  Built by tests/interval_reference.py with the oracle's flags.
#include <cmath>
#include <cstdint>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

namespace {

inline uint64_t rng_next(uint64_t &s0, uint64_t &s1) {
    uint64_t x = s0;
    const uint64_t y = s1;
    s0 = y;
    x ^= x << 23;
    s1 = x ^ y ^ (x >> 17) ^ (y >> 26);
    return s1 + y;
}

struct Groups {
    int32_t ngroups = 0;
    const int32_t *grp = nullptr;
    const int32_t *coef = nullptr;
    const double *lambda = nullptr;
    const int64_t *kappa = nullptr;
    const int64_t *lo = nullptr;   // null: equality groups
    const int64_t *hi = nullptr;
};

inline int64_t dist(int64_t u, int64_t lo, int64_t hi) { return u < lo ? lo - u : (u > hi ? u - hi : 0); }

inline double group_flip_cost(const Groups &G, int v, int s, const int64_t *M) {
    const int g = G.grp[v];
    if (g < 0) return 0.0;
    const int64_t a = G.coef[v];
    const int64_t u = M[g] + G.kappa[g];
    if (!G.lo) return G.lambda[g] * double(a * (a - int64_t(s) * u));
    const int64_t d0 = dist(u, G.lo[g], G.hi[g]), d1 = dist(u - 2 * a * s, G.lo[g], G.hi[g]);
    return G.lambda[g] * (double(d1 * d1 - d0 * d0) * 0.25);
}

double state_energy(const int8_t *st, int n, const double *h, int64_t m, const int32_t *starts, const int32_t *ends,
                    const double *w, const Groups &G) {
    double e = 0.0;
    for (int v = 0; v < n; ++v) e += st[v] * h[v];
    for (int64_t c = 0; c < m; ++c) e += st[starts[c]] * w[c] * st[ends[c]];
    if (G.ngroups) {
        std::vector<int64_t> M(G.ngroups, 0);
        for (int v = 0; v < n; ++v)
            if (G.grp[v] >= 0) M[G.grp[v]] += int64_t(G.coef[v]) * st[v];
        for (int g = 0; g < G.ngroups; ++g) {
            const int64_t u = M[g] + G.kappa[g];
            const int64_t t = G.lo ? dist(u, G.lo[g], G.hi[g]) : u;
            e += G.lambda[g] * double(t * t) * 0.25;
        }
    }
    return e;
}

}  // namespace

extern "C" {

// states_inout [R][n] +-1, updated in place; energies_out [R]; stats_out [5]: attempts, candidates, draws, accepted,
// neighbour updates.  Returns num_reads or a negative code.
int iref_sample_ising(int32_t n, const double *h, int64_t m, const int32_t *starts, const int32_t *ends, const double *w,
                      int32_t num_reads, int8_t *states_inout, double *energies_out, int32_t num_betas, const double *betas,
                      int32_t sweeps_per_beta, const uint64_t *seeds, int32_t ngroups, const int32_t *grp,
                      const int32_t *coef, const double *lambda, const int64_t *kappa, const int64_t *lo,
                      const int64_t *hi, uint64_t *stats_out) {
    std::vector<int64_t> rowptr(n + 1, 0);
    for (int64_t c = 0; c < m; ++c) {
        if (starts[c] < 0 || ends[c] < 0 || starts[c] >= n || ends[c] >= n || starts[c] == ends[c]) return -2;
        rowptr[starts[c] + 1]++;
        rowptr[ends[c] + 1]++;
    }
    for (int v = 0; v < n; ++v) rowptr[v + 1] += rowptr[v];
    std::vector<int32_t> col(2 * m);
    std::vector<double> val(2 * m);
    {
        std::vector<int64_t> fill(rowptr.begin(), rowptr.end() - 1);
        for (int64_t c = 0; c < m; ++c) {   // neal's push_back order: couplers in order, both endpoints
            col[fill[starts[c]]] = ends[c]; val[fill[starts[c]]++] = w[c];
            col[fill[ends[c]]] = starts[c]; val[fill[ends[c]]++] = w[c];
        }
    }
    Groups G;
    G.ngroups = ngroups; G.grp = grp; G.coef = coef; G.lambda = lambda; G.kappa = kappa; G.lo = lo; G.hi = hi;
    uint64_t tot[5] = {0, 0, 0, 0, 0};
    #pragma omp parallel
    {
        std::vector<double> dE(n);
        std::vector<int64_t> M(ngroups > 0 ? ngroups : 1);
        uint64_t loc[5] = {0, 0, 0, 0, 0};
        #pragma omp for schedule(dynamic, 1)
        for (int r = 0; r < num_reads; ++r) {
            int8_t *st = states_inout + int64_t(r) * n;
            uint64_t s0 = seeds[r] ? seeds[r] : ~uint64_t(0), s1 = 0;
            for (int v = 0; v < n; ++v) {
                double f = h[v];
                for (int64_t e = rowptr[v]; e < rowptr[v + 1]; ++e) f += st[col[e]] * val[e];
                dE[v] = -2 * st[v] * f;
            }
            if (ngroups) {
                for (int g = 0; g < ngroups; ++g) M[g] = 0;
                for (int v = 0; v < n; ++v)
                    if (grp[v] >= 0) M[grp[v]] += int64_t(coef[v]) * st[v];
            }
            for (int b = 0; b < num_betas; ++b) {
                const double beta = betas[b];
                for (int sw = 0; sw < sweeps_per_beta; ++sw) {
                    const double thr = 44.36142 / beta;
                    for (int v = 0; v < n; ++v) {
                        double d = dE[v];
                        if (ngroups) d = d + group_flip_cost(G, v, st[v], M.data());
                        loc[0]++;
                        if (d >= thr) continue;
                        loc[1]++;
                        bool flip = d <= 0.0;
                        if (!flip) {
                            const uint64_t rnd = rng_next(s0, s1);
                            loc[2]++;
                            flip = std::exp(-d * beta) * 18446744073709551616.0 > double(rnd);
                        }
                        if (!flip) continue;
                        loc[3]++;
                        const int mul = 4 * st[v];
                        for (int64_t e = rowptr[v]; e < rowptr[v + 1]; ++e) dE[col[e]] += mul * val[e] * st[col[e]];
                        loc[4] += uint64_t(rowptr[v + 1] - rowptr[v]);
                        if (ngroups && grp[v] >= 0) M[grp[v]] -= 2 * int64_t(coef[v]) * st[v];
                        st[v] = int8_t(-st[v]);
                        dE[v] = -dE[v];
                    }
                }
            }
            energies_out[r] = state_energy(st, n, h, m, starts, ends, w, G);
        }
        #pragma omp critical
        for (int k = 0; k < 5; ++k) tot[k] += loc[k];
    }
    for (int k = 0; k < 5; ++k) stats_out[k] = tot[k];
    return num_reads;
}

int iref_state_energies(int32_t n, const double *h, int64_t m, const int32_t *starts, const int32_t *ends, const double *w,
                        int32_t num_reads, const int8_t *states, double *energies_out, int32_t ngroups, const int32_t *grp,
                        const int32_t *coef, const double *lambda, const int64_t *kappa, const int64_t *lo, const int64_t *hi) {
    Groups G;
    G.ngroups = ngroups; G.grp = grp; G.coef = coef; G.lambda = lambda; G.kappa = kappa; G.lo = lo; G.hi = hi;
    for (int r = 0; r < num_reads; ++r) energies_out[r] = state_energy(states + int64_t(r) * n, n, h, m, starts, ends, w, G);
    return 0;
}

// the group part of the flip cost of variable v in state `st` (what the loop adds to neal's dE[v])
double iref_group_flip_cost(int32_t n, const int8_t *st, int32_t v, int32_t ngroups, const int32_t *grp, const int32_t *coef,
                            const double *lambda, const int64_t *kappa, const int64_t *lo, const int64_t *hi) {
    Groups G;
    G.ngroups = ngroups; G.grp = grp; G.coef = coef; G.lambda = lambda; G.kappa = kappa; G.lo = lo; G.hi = hi;
    std::vector<int64_t> M(ngroups > 0 ? ngroups : 1, 0);
    for (int u = 0; u < n; ++u)
        if (grp[u] >= 0) M[grp[u]] += int64_t(coef[u]) * st[u];
    return group_flip_cost(G, v, st[v], M.data());
}

}  // extern "C"
