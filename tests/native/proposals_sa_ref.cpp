// tests/native/proposals_sa_ref.cpp -- TEST INFRASTRUCTURE: CPU reference for dwave-samplers' sample options.
//
// The simulated-annealing loop of oracle/cpu_sa_ref.cpp (neal's simulated_annealing_run: xorshift128+, threshold
// 44.36142 / beta, eager neighbour updates, neal's push_back adjacency order, get_state_energy) with the two options
// dwave-samplers >= 1.0 added (SURVEY.md Appendix C.8; recalled from its cpu_sa.cpp, not pinned against the package):
//   var_order 1 (randomize_order=True)   attempt k of a sweep visits v = xorshift128+() % n (unsigned 64-bit modulo), drawn
//                                        before anything else; still n attempts per sweep.  0: v = k (neal).
//   proposal 1 (Gibbs)                   skip if dE >= thr (no draw), accept if dE <= -thr (no draw), otherwise draw r and
//                                        accept iff 2^64 > (double)r * (1 + exp(dE * beta)), one rounding per operation.
//                                        0 (Metropolis, neal): skip if dE >= thr, accept if dE <= 0, otherwise accept iff
//                                        exp(-dE * beta) * 2^64 > (double)r.
// `draws` counts every xorshift128+ output consumed, order draws included.  Rank-1 groups as in the oracle (equality
// groups: lambda * (double)(a * (a - s (M + kappa))) per flip) or, with lo / hi, the interval groups of
// tests/native/interval_sa_ref.cpp.  With (var_order, proposal) = (0, 0) this reproduces oracle_sa_sample_ising and
// iref_sample_ising bit for bit (tests/test_proposals_cpu.py).  Seeding as in the oracle: seed_mode 0 per read, 1 one
// stream across reads.  Built by tests/proposals_reference.py with the oracle's flags.
#include <cmath>
#include <cstdint>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

namespace {

inline uint64_t rng_next(uint64_t &s0, uint64_t &s1) {   // neal FASTRAND
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

struct Model {
    int n;
    const double *h;
    std::vector<int64_t> rowptr;
    std::vector<int32_t> col;
    std::vector<double> val;
    Groups G;
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

// one read; counters: attempts, candidates, draws, accepted, neighbour updates
void anneal_one_read(int8_t *st, const Model &Md, const double *betas, int num_betas, int sweeps_per_beta, bool random_order,
                     bool gibbs, uint64_t &s0, uint64_t &s1, double *dE, int64_t *M, uint64_t *cnt) {
    const int n = Md.n;
    const Groups &G = Md.G;
    for (int v = 0; v < n; ++v) {
        double f = Md.h[v];
        for (int64_t e = Md.rowptr[v]; e < Md.rowptr[v + 1]; ++e) f += st[Md.col[e]] * Md.val[e];
        dE[v] = -2 * st[v] * f;
    }
    if (G.ngroups) {
        for (int g = 0; g < G.ngroups; ++g) M[g] = 0;
        for (int v = 0; v < n; ++v)
            if (G.grp[v] >= 0) M[G.grp[v]] += int64_t(G.coef[v]) * st[v];
    }
    for (int b = 0; b < num_betas; ++b) {
        const double beta = betas[b];
        for (int sw = 0; sw < sweeps_per_beta; ++sw) {
            const double thr = 44.36142 / beta;
            for (int k = 0; k < n; ++k) {
                int v = k;
                if (random_order) {
                    v = int(rng_next(s0, s1) % uint64_t(n));
                    cnt[2]++;
                }
                double d = dE[v];
                if (G.ngroups) d = d + group_flip_cost(G, v, st[v], M);
                cnt[0]++;
                if (d >= thr) continue;
                cnt[1]++;
                bool flip = gibbs ? d <= -thr : d <= 0.0;
                if (!flip) {
                    const uint64_t rnd = rng_next(s0, s1);
                    cnt[2]++;
                    flip = gibbs ? 18446744073709551616.0 > double(rnd) * (1.0 + std::exp(d * beta))
                                 : std::exp(-d * beta) * 18446744073709551616.0 > double(rnd);
                }
                if (!flip) continue;
                cnt[3]++;
                const int mul = 4 * st[v];
                for (int64_t e = Md.rowptr[v]; e < Md.rowptr[v + 1]; ++e) dE[Md.col[e]] += mul * Md.val[e] * st[Md.col[e]];
                cnt[4] += uint64_t(Md.rowptr[v + 1] - Md.rowptr[v]);
                if (G.ngroups && G.grp[v] >= 0) M[G.grp[v]] -= 2 * int64_t(G.coef[v]) * st[v];
                st[v] = int8_t(-st[v]);
                dE[v] = -dE[v];
            }
        }
    }
}

}  // namespace

extern "C" {

// states_inout [R][n] +-1, updated in place; energies_out [R]; stats_out [5]: attempts, candidates, draws, accepted,
// neighbour updates.  lo = hi = null: equality groups.  Returns num_reads or a negative code.
int pref_sample_ising(int32_t n, const double *h, int64_t m, const int32_t *starts, const int32_t *ends, const double *w,
                      int32_t num_reads, int8_t *states_inout, double *energies_out, int32_t num_betas, const double *betas,
                      int32_t sweeps_per_beta, const uint64_t *seeds, int32_t seed_mode, int32_t var_order, int32_t proposal,
                      int32_t ngroups, const int32_t *grp, const int32_t *coef, const double *lambda, const int64_t *kappa,
                      const int64_t *lo, const int64_t *hi, uint64_t *stats_out) {
    if (n < 0 || m < 0 || num_reads < 0 || num_betas < 0 || sweeps_per_beta < 0) return -1;
    if ((var_order != 0 && var_order != 1) || (proposal != 0 && proposal != 1) || (seed_mode != 0 && seed_mode != 1)) return -1;
    for (int64_t i = 0; i < int64_t(num_reads) * n; ++i)
        if (states_inout[i] != 1 && states_inout[i] != -1) return -3;
    Model Md;
    Md.n = n;
    Md.h = h;
    Md.rowptr.assign(n + 1, 0);
    for (int64_t c = 0; c < m; ++c) {
        if (starts[c] < 0 || ends[c] < 0 || starts[c] >= n || ends[c] >= n || starts[c] == ends[c]) return -2;
        Md.rowptr[starts[c] + 1]++;
        Md.rowptr[ends[c] + 1]++;
    }
    for (int v = 0; v < n; ++v) Md.rowptr[v + 1] += Md.rowptr[v];
    Md.col.resize(2 * m);
    Md.val.resize(2 * m);
    {
        std::vector<int64_t> fill(Md.rowptr.begin(), Md.rowptr.end() - 1);
        for (int64_t c = 0; c < m; ++c) {   // neal's push_back order: couplers in order, both endpoints
            Md.col[fill[starts[c]]] = ends[c]; Md.val[fill[starts[c]]++] = w[c];
            Md.col[fill[ends[c]]] = starts[c]; Md.val[fill[ends[c]]++] = w[c];
        }
    }
    Md.G.ngroups = ngroups; Md.G.grp = grp; Md.G.coef = coef; Md.G.lambda = lambda; Md.G.kappa = kappa;
    Md.G.lo = lo; Md.G.hi = hi;
    const bool random_order = var_order == 1, gibbs = proposal == 1;
    uint64_t tot[5] = {0, 0, 0, 0, 0};
    if (seed_mode == 1) {   // one xorshift128+ stream across reads (neal num_reads = R)
        uint64_t s0 = seeds[0] ? seeds[0] : ~uint64_t(0), s1 = 0;
        std::vector<double> dE(n);
        std::vector<int64_t> M(ngroups > 0 ? ngroups : 1);
        for (int r = 0; r < num_reads; ++r) {
            int8_t *st = states_inout + int64_t(r) * n;
            anneal_one_read(st, Md, betas, num_betas, sweeps_per_beta, random_order, gibbs, s0, s1, dE.data(), M.data(), tot);
            energies_out[r] = state_energy(st, n, h, m, starts, ends, w, Md.G);
        }
    } else {
        #pragma omp parallel
        {
            std::vector<double> dE(n);
            std::vector<int64_t> M(ngroups > 0 ? ngroups : 1);
            uint64_t loc[5] = {0, 0, 0, 0, 0};
            #pragma omp for schedule(dynamic, 1)
            for (int r = 0; r < num_reads; ++r) {
                int8_t *st = states_inout + int64_t(r) * n;
                uint64_t s0 = seeds[r] ? seeds[r] : ~uint64_t(0), s1 = 0;
                anneal_one_read(st, Md, betas, num_betas, sweeps_per_beta, random_order, gibbs, s0, s1, dE.data(), M.data(),
                                loc);
                energies_out[r] = state_energy(st, n, h, m, starts, ends, w, Md.G);
            }
            #pragma omp critical
            for (int k = 0; k < 5; ++k) tot[k] += loc[k];
        }
    }
    for (int k = 0; k < 5; ++k) stats_out[k] = tot[k];
    return num_reads;
}

}  // extern "C"
