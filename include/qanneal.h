/* qanneal.h -- C ABI of libqanneal.so, the B200 (sm_100a) simulated-annealing sampler.
 *
 * This is the drop-in boundary for the ONE hot path of
 * michal7kw/scRNA_seq_QAnnealing_Clustering: the QUBO/BQM sampling loop its clustering
 * functions hand to a dimod sampler
 *   sampler.sample_qubo(Q, ...)   Python_Functions/BQM_clustering.py:57,75,85,245,263,273
 *                                 Python_Functions/QA_subsampling.py:42,56,65
 *   sampler.sample(bqm, ...)      Python_Functions/BQM_clustering.py:386
 *   sampler.sample_dqm(dqm, ...)  Python_Functions/DQM_clustering.py:45
 *   sampler.sample_cqm(cqm, ...)  Python_Functions/CQM_clustering.py:53,89
 * Offline that sampler is dwave-neal, whose Cython layer binds
 *   int general_simulated_annealing(char* states, double* energies, int num_samples,
 *        vector<double> h, vector<int> coupler_starts, vector<int> coupler_ends,
 *        vector<double> coupler_weights, int sweeps_per_beta, vector<double> beta_schedule,
 *        uint64_t seed, callback interrupt_callback, void* interrupt_function)
 *   (dwave-neal neal/src/cpu_sa.h; dwave-samplers dwave/samplers/sa/src/cpu_sa.h)
 * qa_sa_sample_ising() below is the entry point a maintainer would bind in its place.
 *
 * Conventions
 *  - every function returns int: >= 0 OK, < 0 error code; message via qa_last_error()
 *    (thread-local).  No C++ exception crosses the ABI.
 *  - plain pointers and sizes only.  Data pointers may be HOST pointers or CUDA DEVICE
 *    pointers of the context's device (detected with cudaPointerGetAttributes); model
 *    and scratch memory is owned by the library, every other buffer by the caller.
 *  - calls block until their results are complete.  A qa_ctx is not re-entrant.
 *  - STREAMS: a context launches on its own non-blocking CUDA stream and synchronises it before a call returns, so results
 *    are complete on return for any consumer.  The library does NOT order itself against the caller's streams: a device
 *    buffer handed in (states, seeds, schedules, graph arrays) must be complete -- synchronise the producing stream, or
 *    record an event and wait for it, before the call (bench.py: torch.cuda.synchronize()).
 *  - duplicate couplers (the same pair listed twice) are legal, as for neal; the warp-per-read kernel then issues two
 *    reductions to one address from one instruction, whose relative order the PTX memory model does not define (observed:
 *    lane order).  Vectors derived from a BQM never contain duplicates.
 *  - spins are int8 +1/-1, states are row-major [num_reads][n] and are IN/OUT (initial
 *    states in, final states out), exactly like neal's `states` argument.
 */
#ifndef QANNEAL_H
#define QANNEAL_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QA_OK 0
#define QA_ERR_ARG (-1)      /* bad argument (sizes, null pointers, unknown enum) */
#define QA_ERR_INDEX (-2)    /* coupler index out of range / self loop (neal: runtime_error) */
#define QA_ERR_STATE (-3)    /* initial state not +-1 */
#define QA_ERR_CUDA (-4)     /* CUDA runtime failure (no device, OOM, launch error) */
#define QA_ERR_LIMIT (-5)    /* model exceeds an implementation limit */
#define QA_ERR_INTERRUPTED (-6)

/* seed_mode */
#define QA_SEED_PER_READ 0   /* read r == neal(num_reads=1, seed=seeds[r], initial_states=states[r]) */
#define QA_SEED_STREAM 1     /* one xorshift128+ stream across reads == neal(num_reads=R, seed=seeds[0]) */
/* mode */
#define QA_MODE_REFERENCE 0  /* neal's sequential variable order, bit-exact against the oracle */
#define QA_MODE_THROUGHPUT 1 /* tolerance-parity mode for DENSE models (qa_model_enable_dense): neal's sequential sweep and
                               per-read RNG, local fields of every 8-cell block recomputed by fp64 tensor-core MMAs instead of
                               updated incrementally: same algorithm, different fp64 rounding history -> energies to 1e-12
                               relative, statistical parity.  Models without the dense form run the reference-order kernels
                               (bit-exact) in this mode too */
/* reference-mode kernel selection (both are bit-exact against the oracle) */
#define QA_KERNEL_AUTO 0
#define QA_KERNEL_WARP_PER_READ 1  /* one warp per read: any read count, stream seeding */
#define QA_KERNEL_LOCKSTEP_PUSH 2  /* one warp per 32 reads, read-interleaved fields: many reads (>= ~10^4) */
#define QA_KERNEL_LOCKSTEP_PULL 3  /* retired (round 2): the sparse recompute variant, overtaken by _REPLAY; never selected */
#define QA_KERNEL_REPLAY 4         /* 32 reads per warp, deferred exact neighbour updates replayed at the visit; coupling
                                      slabs TMA-staged per CTA.  Sparse models; falls back to _LOCKSTEP_PUSH otherwise */
#define QA_KERNEL_DENSE 5          /* QA_MODE_THROUGHPUT on a model with the dense k-way form (qa_model_enable_dense):
                                      local fields of 8-cell blocks by fp64 tensor-core MMAs (DMMA) over all cells */

/* var_order / proposal (qa_sa_sample_model_ex, qa_sa_sample_ising_ex): dwave-samplers >= 1.0's sample options
 * randomize_order and proposal_acceptance_criteria, as SURVEY.md Appendix C.8 recalls its cpu_sa.cpp (not pinned against the
 * package).  Per beta thr = 44.36142 / beta; per attempt:
 *   QA_ORDER_SEQUENTIAL      attempt k of a sweep visits variable k (neal)
 *   QA_ORDER_RANDOM          attempt k visits v = r % n (unsigned 64-bit) for r = the read's next xorshift128+ output, drawn
 *                            before anything else; still n attempts per sweep
 *   QA_PROPOSAL_METROPOLIS   skip if dE >= thr; accept if dE <= 0; else draw r, accept iff exp(-dE*beta) * 2^64 > (double)r
 *   QA_PROPOSAL_GIBBS        skip if dE >= thr; accept if dE <= -thr; else draw r, accept iff 2^64 > (double)r * (1 + exp(dE*beta))
 * dE includes the rank-1 group terms.  Every combination is bit-exact against the CPU reference of the tests
 * (tests/native/proposals_sa_ref.cpp, which at the defaults reproduces the oracle bit for bit).
 * Kernels: random order always runs QA_KERNEL_WARP_PER_READ, whatever qa_ctx_set_kernel asked for (the lockstep and replay
 * kernels walk 32 reads through one shared variable order).  Sequential Gibbs runs the kernel the usual rules pick, except
 * that QA_MODE_THROUGHPUT never picks QA_KERNEL_DENSE: with either option the tensor-core kernel is not used. */
#define QA_ORDER_SEQUENTIAL 0
#define QA_ORDER_RANDOM 1
#define QA_PROPOSAL_METROPOLIS 0
#define QA_PROPOSAL_GIBBS 1

#define QA_MAX_GROUPS 64

typedef struct qa_ctx qa_ctx;
typedef struct qa_model qa_model;

/* Counters and device-side phase timings (CUDA events on the context's stream). */
typedef struct qa_stats {
    uint64_t attempts;      /* n * num_sweeps * num_reads */
    uint64_t candidates;    /* attempts with dE <  44.36142/beta  (reached the accept test; Gibbs too) */
    uint64_t draws;         /* xorshift128+ outputs consumed: accept draws (Metropolis 0 < dE < thr, Gibbs -thr < dE < thr)
                               and, with QA_ORDER_RANDOM, one order draw per attempt */
    uint64_t accepted;      /* spin flips performed */
    uint64_t nbr_updates;   /* sum of deg(v) over accepted flips */
    uint64_t active_chunks; /* 32-variable chunks that had >= 1 candidate (0 under QA_ORDER_RANDOM) */
    uint64_t chunks;        /* 32-variable chunks streamed (0 under QA_ORDER_RANDOM) */
    uint64_t near_ties;     /* accept tests decided by < 2^-48 relative margin (Gibbs: |2^64 - r (1 + exp)| <= 2^16) */
    double ms_h2d;          /* host->device copies (0 when inputs are device resident) */
    double ms_build;        /* CSR construction */
    double ms_anneal;       /* annealing kernel(s) */
    double ms_energy;       /* energy (+argmin) kernel(s) */
    double ms_d2h;          /* device->host copies */
    uint32_t anneal_launches;
    uint32_t total_launches; /* kernels of this library launched by the call */
    double ms_total;        /* the whole call on the device: first copy-in event to last copy-out event */
} qa_stats;

const char *qa_last_error(void);
int qa_version(void);
int qa_device_count(void);

/* context = one GPU + one stream + reusable scratch */
int qa_ctx_create(int device_id, qa_ctx **out);
int qa_ctx_destroy(qa_ctx *ctx);
int qa_ctx_synchronize(qa_ctx *ctx);
/* choose the reference-mode annealing kernel (QA_KERNEL_AUTO / _WARP_PER_READ / _LOCKSTEP_PUSH / _REPLAY) */
int qa_ctx_set_kernel(qa_ctx *ctx, int kernel);
/* QA_KERNEL_* the last sampling call of this context actually ran on (after automatic selection / fall-back) */
int qa_ctx_last_kernel(qa_ctx *ctx);
/* number of reads the annealing kernel keeps resident at once (one warp per read) */
int qa_ctx_resident_reads(qa_ctx *ctx);

/* Ising model, neal's vectors: h[n], couplers (starts, ends, weights)[m] in coupler order.
 * Builds the adjacency on the device preserving neal's per-vertex push_back order. */
int qa_model_from_ising(qa_ctx *ctx, int32_t n, const double *h, int64_t m, const int32_t *starts,
                        const int32_t *ends, const double *weights, qa_model **out);
/* Optional lazily-evaluated rank-1 terms  sum_g lambda[g]/4 * (sum_{v: grp[v]==g} coef[v]*s_v + kappa[g])^2
 * (cut+balance, DQM cluster-size and CQM size penalties; SURVEY.md Appendix A). grp[v] = -1: none. */
int qa_model_set_groups(qa_model *model, int32_t ngroups, const int32_t *grp, const int32_t *coef,
                        const double *lambda, const int64_t *kappa);
/* Interval bounds for the groups of qa_model_set_groups (inequality constraints without slack variables).  With
 * u_g = sum_{v: grp[v]==g} coef[v]*s_v + kappa[g] and d(u) = max(lo[g] - u, 0, u - hi[g]), group g contributes
 *     lambda[g] * (double)(d*d) * 0.25
 * and a flip that moves u to u' costs lambda[g] * ((double)(d(u')^2 - d(u)^2) * 0.25): integers exact, one rounding.
 * lo = hi = 0 is the equality term above, bit for bit.  Bounds are clamped to the reachable range
 * [kappa - sum|coef|, kappa + sum|coef|] (INT64_MIN / INT64_MAX: unbounded); lo > hi gives QA_ERR_ARG, a clamped
 * distance d whose square reaches 2^53 QA_ERR_LIMIT.  lo = hi = NULL: equality groups again.  Call after
 * qa_model_set_groups; a later qa_model_set_groups clears the bounds. */
int qa_model_set_group_bounds(qa_model *model, const int64_t *lo, const int64_t *hi);
/* Dense k-way form (BASELINE config 5; the all-pairs same-case term of DQM_clustering.py:36-37 on a dense affinity):
 * variable v = cell*K + case, J[(i,c),(j,c)] = W[i][j] for every case c, J[(i,c),(i,c')] = P.  Derives W (n/K x n/K) and P
 * from the model's adjacency on the device and verifies the structure.  Returns 1 when the model has it -- QA_MODE_THROUGHPUT
 * then anneals it with the tensor-core kernel (neal's sweep order and RNG, fields recomputed per block of 8 cells by
 * mma.sync f64; energies to 1e-12 relative of neal's order) --, 0 when it does not (nothing changes).  K in {1, 2, 4, 8};
 * K = 1 is a general dense Ising model. */
int qa_model_enable_dense(qa_model *model, int32_t cases_per_cell);
/* Replay kernel's coupling slabs, as the last sampling call on the replay kernel built them: the number of blocks that carry
 * a k-way section (one-hot cells of K cases annealed in lockstep; 0: none, or the slabs are not built yet) and their K.
 * QA_REPLAY_KWAY=0 in the environment when the context is created keeps every block in the generic form. */
int64_t qa_model_replay_kway(const qa_model *model, int32_t *k_out);
int qa_model_num_variables(const qa_model *model);
int64_t qa_model_num_couplers(const qa_model *model);
int qa_model_max_degree(const qa_model *model);
/* copy the device-built Ising vectors back (any pointer may be NULL) */
int qa_model_get_ising(const qa_model *model, double *h, int32_t *starts, int32_t *ends, double *weights);
int qa_model_destroy(qa_model *model);

/* Anneal num_reads reads of a resident model.  energies_out[r] is neal's get_state_energy
 * (spin-model energy WITHOUT offset) of the final state.  interrupt may be NULL; it is
 * polled between read waves and a non-zero return stops the run (neal: interrupt_function);
 * the return value is the number of reads completed. */
typedef int (*qa_interrupt_fn)(void *user);
int qa_sa_sample_model(qa_ctx *ctx, qa_model *model, int32_t num_reads, int8_t *states_inout,
                       double *energies_out, int32_t num_betas, const double *beta_schedule,
                       int32_t sweeps_per_beta, const uint64_t *seeds, int32_t seed_mode,
                       int32_t mode, qa_interrupt_fn interrupt, void *interrupt_user,
                       qa_stats *stats_out);

/* qa_sa_sample_model with dwave-samplers' variable order and acceptance rule (QA_ORDER_*, QA_PROPOSAL_*; any other value:
 * QA_ERR_ARG).  (QA_ORDER_SEQUENTIAL, QA_PROPOSAL_METROPOLIS) is qa_sa_sample_model. */
int qa_sa_sample_model_ex(qa_ctx *ctx, qa_model *model, int32_t num_reads, int8_t *states_inout,
                          double *energies_out, int32_t num_betas, const double *beta_schedule,
                          int32_t sweeps_per_beta, const uint64_t *seeds, int32_t seed_mode,
                          int32_t mode, int32_t var_order, int32_t proposal, qa_interrupt_fn interrupt,
                          void *interrupt_user, qa_stats *stats_out);

/* One-shot form mirroring neal's general_simulated_annealing, argument for argument (model built and freed inside):
 * interrupt / interrupt_user are neal's interrupt_callback / interrupt_function (may be NULL); the return value is the number
 * of reads completed. */
int qa_sa_sample_ising(qa_ctx *ctx, int32_t n, const double *h, int64_t m, const int32_t *starts,
                       const int32_t *ends, const double *weights, int32_t num_reads,
                       int8_t *states_inout, double *energies_out, int32_t num_betas,
                       const double *beta_schedule, int32_t sweeps_per_beta, const uint64_t *seeds,
                       int32_t seed_mode, int32_t mode, qa_interrupt_fn interrupt, void *interrupt_user,
                       qa_stats *stats_out);
/* The same for dwave-samplers >= 1.0's general_simulated_annealing, which takes varorder and proposal_acceptance_criteria
 * after the seed and before the interrupt callback (that argument order is recalled, not verified against the package). */
int qa_sa_sample_ising_ex(qa_ctx *ctx, int32_t n, const double *h, int64_t m, const int32_t *starts,
                          const int32_t *ends, const double *weights, int32_t num_reads,
                          int8_t *states_inout, double *energies_out, int32_t num_betas,
                          const double *beta_schedule, int32_t sweeps_per_beta, const uint64_t *seeds,
                          int32_t seed_mode, int32_t mode, int32_t var_order, int32_t proposal,
                          qa_interrupt_fn interrupt, void *interrupt_user, qa_stats *stats_out);

/* Many independent problems in one launch (QA_subsampling.py:24 called per sub-graph).
 * Problem p owns variables [var_offsets[p], var_offsets[p+1]) of h and couplers
 * [coupler_offsets[p], coupler_offsets[p+1]) (indices local to the problem); every problem
 * runs reads_per_problem reads.  states: [num_problems][reads_per_problem][n_p] packed
 * back to back in problem order; energies: [num_problems][reads_per_problem];
 * seeds: [num_problems * reads_per_problem] (per-read seeding only).  Sequential order, Metropolis acceptance. */
int qa_sa_sample_ising_batch(qa_ctx *ctx, int32_t num_problems, const int64_t *var_offsets,
                             const int64_t *coupler_offsets, const double *h, const int32_t *starts,
                             const int32_t *ends, const double *weights, int32_t reads_per_problem,
                             int8_t *states_inout, double *energies_out, int32_t num_betas,
                             const double *beta_schedule, int32_t sweeps_per_beta,
                             const uint64_t *seeds, qa_stats *stats_out);

/* Energies of given states in neal's summation order + warp-shuffle min/argmin
 * (neal get_state_energy, dimod bqm.energies, SampleSet.first). Outputs may be NULL. */
int qa_energy_argmin(qa_ctx *ctx, qa_model *model, int32_t num_reads, const int8_t *states,
                     double *energies_out, double *best_energy, int64_t *best_index,
                     qa_stats *stats_out);

/* ---- model builders on the device --------------------------------------------------------------------------------
 * Graph = n nodes and m_edges weighted edges (eu[e], ev[e], w[e]) in the order networkx yields G.edges (host or device
 * pointers).  Each builder restates one Q-dict construction of the reference on the GPU and leaves a resident model in
 * dimod's to_numpy_vectors order; every floating-point accumulation keeps the reference's order, so h / couplers are
 * bit-identical to the Python builders (models.py).  offset_out: E_binary(x) = E_spin(s) + offset.
 *   qa_build_cut_balance   BQM_clustering.py:29-47   k*cut + gamma*S(S-n), gamma = gamma_factor*W/n; balance term as 1 group
 *   qa_build_subsampling   QA_subsampling.py:26-35   sum (1-w)(x_u x_v - x_u - x_v) + gamma*sum x   (P = 1 in the reference)
 *   qa_build_dqm_onehot    DQM_clustering.py:29-43   one-hot expansion (variable i*K + c), penalty*(sum_c x_ic - 1)^2,
 *                                                    cluster-size term as K groups; intended = 0: set_* semantics as written
 *   qa_build_cqm_penalty   CQM_clustering.py:30-48   objective + A*(one-hot)^2 + B*(N_j - min_size - slack_j)^2 as K groups
 *   qa_build_cqm_interval  same constraint, no slack: objective + A*(one-hot)^2 + B*max(0, min_size - N_j)^2 as K interval
 *                          groups (coef 1, kappa = n - 2*min_size, bounds [0, +inf)); h, couplers and offset are those of
 *                          the first n*K variables of qa_build_cqm_penalty
 */
int qa_build_cut_balance(qa_ctx *ctx, int32_t n, int64_t m_edges, const int32_t *eu, const int32_t *ev, const double *w,
                         double gamma_factor, double k, qa_model **out, double *offset_out, double *gamma_out);
/* qa_build_cut_linear    BQM_clustering.py:210-236 (clustering_bqm_2): k*cut + gamma*sum x, gamma = (W/n)*gamma_factor; sparse */
int qa_build_cut_linear(qa_ctx *ctx, int32_t n, int64_t m_edges, const int32_t *eu, const int32_t *ev, const double *w,
                        double gamma_factor, double k, qa_model **out, double *offset_out, double *gamma_out);
int qa_build_subsampling(qa_ctx *ctx, int32_t n, int64_t m_edges, const int32_t *eu, const int32_t *ev, const double *w,
                         double gamma, double P, qa_model **out, double *offset_out);
int qa_build_dqm_onehot(qa_ctx *ctx, int32_t n, int64_t m_edges, const int32_t *eu, const int32_t *ev, const double *w,
                        int32_t num_cases, double gamma, double penalty, int32_t intended, qa_model **out, double *offset_out);
int qa_build_cqm_penalty(qa_ctx *ctx, int32_t n, int64_t m_edges, const int32_t *eu, const int32_t *ev, const double *w,
                         int32_t num_clusters, int32_t min_size, double onehot_penalty, double size_penalty, qa_model **out,
                         double *offset_out);
int qa_build_cqm_interval(qa_ctx *ctx, int32_t n, int64_t m_edges, const int32_t *eu, const int32_t *ev, const double *w,
                          int32_t num_clusters, int32_t min_size, double onehot_penalty, double size_penalty, qa_model **out,
                          double *offset_out);

/* ---- SNN graph construction on the device (the step before the path: Seurat FindNeighbors as the reference's notebooks use
 * it, R/pbmc3k/Pbmc3k_general_data_preparation.Rmd:47-75, R/benchmarks/Benchmark.Rmd:150-166):
 * exact kNN including self -> shared-neighbour counts s -> w = s/(2k - s) -> prune w < prune -> sequential symmetric degree
 * trim to max_degree (<= 0: no trim).  num_problems independent point sets (points [point_offsets[p], point_offsets[p+1]) of
 * X, row-major [total][dim], host or device) are built in the same launches.  Edges come out with u < v, local indices,
 * sorted by (u, v) per problem -- identical to snn.py's graph.  The edge arrays stay on the device; qa_graph_device_edges
 * hands them to the qa_build_* entry points without a host round trip. ---- */
typedef struct qa_graph qa_graph;
int qa_snn_build(qa_ctx *ctx, int32_t num_problems, const int64_t *point_offsets, int32_t dim, const double *X, int32_t k,
                 double prune, int32_t max_degree, qa_graph **out);
int64_t qa_graph_num_edges(const qa_graph *graph, int32_t problem);   /* problem < 0: all problems */
int qa_graph_num_nodes(const qa_graph *graph, int32_t problem);
int qa_graph_get_edges(const qa_graph *graph, int32_t problem, int32_t *eu, int32_t *ev, double *w);   /* copy out (any may be NULL) */
int qa_graph_device_edges(const qa_graph *graph, int32_t problem, const int32_t **eu, const int32_t **ev, const double **w);
int qa_graph_destroy(qa_graph *graph);

/* ---- recursion driver on the device (the recursive calls of clustering_bqm / clustering_bqm_2 on G.subgraph(S0) and
 * G.subgraph(S1), BQM_clustering.py:113-203, 302-350): all sub-graphs of a recursion level are extracted, built and annealed
 * without a host / networkx round trip. ---- */
/* G.subgraph(part) for every part at once: part[v] in [0, num_parts) or -1 (dropped).  Child p keeps the parent's node order
 * (local index = rank inside the part) and the parent's edge order; edges with ends in different parts are dropped.
 * Graph arrays and part may be host or device pointers.  The result is a qa_graph with num_parts problems. */
int qa_graph_split(qa_ctx *ctx, int32_t n, int64_t m_edges, const int32_t *eu, const int32_t *ev, const double *w,
                   const int32_t *part, int32_t num_parts, qa_graph **out);
/* parent node of every node of child `problem` (problem < 0: all children back to back); host or device destination */
int qa_graph_get_nodes(const qa_graph *graph, int32_t problem, int32_t *node_ids_out);
/* single-problem models (rank-1 groups and their interval bounds included) -> one batched model for qa_sa_sample_model_batch;
 * the inputs stay valid and owned by the caller.  Batched models with groups run on the warp-per-read kernel; problems with
 * and without groups, equality and interval groups, may be mixed in one batch. */
int qa_model_concat(qa_ctx *ctx, int32_t num_models, qa_model *const *models, qa_model **out);
/* qa_sa_sample_ising_batch on a resident batched model.  betas_per_problem = 0: beta_schedules is one schedule [num_betas] for
 * every problem; 1: [num_problems][num_betas], problem p anneals with its own schedule (what separate sampler calls with
 * default beta ranges would do). */
int qa_sa_sample_model_batch(qa_ctx *ctx, qa_model *model, int32_t reads_per_problem, int8_t *states_inout, double *energies_out,
                             int32_t num_betas, const double *beta_schedules, int32_t betas_per_problem, int32_t sweeps_per_beta,
                             const uint64_t *seeds, qa_stats *stats_out);

/* ---- SampleSet post-processing on the device (what the reference does with a SampleSet after the call:
 * energy-sorted iteration and k-th best energies BQM_clustering.py:93-146, the 16 best samples plot_and_save.py:105-126,
 * one-hot decode of DQM / CQM samples plot_and_save.py:46-63).  Pointers may be host or device memory. ---- */
/* order_out[r] = index of the r-th best read: ascending energy, ties in read order (stable); -0.0 and +0.0 tie; every NaN,
 * whatever its sign and payload, comes after +inf, NaNs in read order -- numpy's argsort(energies, kind="stable") */
int qa_sort_reads(qa_ctx *ctx, int32_t num_reads, const double *energies, int32_t *order_out);
/* samples_out[r][0..n) = states[order[r]][0..n) for r < k: only the k best samples leave the device */
int qa_gather_samples(qa_ctx *ctx, int32_t n, int32_t num_reads, const int8_t *states, int32_t k, const int32_t *order,
                      int8_t *samples_out);
/* one-hot decode: variable (cell i, case c) = states[read][i*K + c] (stride >= cells*K bytes per read; on_value = +1 for
 * spins, 1 for binaries).  labels_out[read][cell] = case or -1 when the cell is not one-hot (labels_out may be NULL: only
 * the counts are wanted); violations_out[read] = {cells that are not one-hot, cases with fewer than min_size cells} */
int qa_decode_onehot(qa_ctx *ctx, int32_t cells, int32_t K, int64_t stride, int32_t num_reads, const int8_t *states,
                     int32_t on_value, int32_t min_size, int32_t *labels_out, int32_t *violations_out);

/* Duplicate aggregation (dimod SampleSet.aggregate(): identical samples merged, num_occurrences summed) on the device:
 * rows are hashed (2 x 64 bit), sorted by hash, neighbours compared byte for byte.  first_index_out[u] = the first read of
 * the u-th distinct sample, in order of first occurrence; count_out[u] = its number of occurrences (both sized num_reads,
 * host memory).  Only 8 bytes per read leave the device.  n = 0: one group (0, num_reads), states not read.  Exact unless
 * two distinct rows share the 64-bit first hash and their reads interleave (about num_reads^2 / 2^65 per call): then one
 * sample is reported as two groups. */
int qa_aggregate_reads(qa_ctx *ctx, int32_t n, int32_t num_reads, const int8_t *states, int32_t *num_unique_out,
                       int32_t *first_index_out, int32_t *count_out);

/* Device-resident state matrices for callers without a device allocator of their own (the Python host layer): with
 * return_samples='best_k' the [R][n] state matrix is created, annealed, ranked and reduced to k rows on the device.
 * qa_random_states: +-1 states from a counter-based generator, spin (r, v) = bit (v & 63) of
 * splitmix64-mix(seed, first_read + r, v >> 6) -- a function of the GLOBAL read index, so any sharding gives the same states
 * (schedule.counter_spin_states is the same function in numpy).  states_out: host or device. */
int qa_dev_alloc(qa_ctx *ctx, int64_t bytes, void **out);
int qa_dev_free(qa_ctx *ctx, void *p);
int qa_dev_copy(qa_ctx *ctx, void *dst, const void *src, int64_t bytes);   /* any direction, blocking */
int qa_random_states(qa_ctx *ctx, uint64_t seed, int64_t first_read, int32_t num_reads, int32_t n, int8_t *states_out);

/* Lowest value and its first index (SampleSet.first; the per-rank half of the multi-GPU best-sample gather, SURVEY 8e):
 * warp-shuffle min-reduction in the order of qa_sort_reads, so best_index == order_out[0]: a NaN loses to every number, ties
 * (-0.0 == +0.0) go to the lower index, every value NaN gives (values[0], 0); the value is returned bit for bit.  count = 0:
 * (+inf, -1).  values: host or device pointer. */
int qa_argmin(qa_ctx *ctx, int64_t count, const double *values, double *best_value, int64_t *best_index);
/* The same reduction with its result left on the device: out_device[0] = lowest value, out_device[1] = (double)(index_offset +
 * its first index) -- the 16-byte send buffer of the per-rank all_gather, filled without a host round trip.  count >= 1, so
 * the offset is always added to an index in [0, count). */
int qa_argmin_device(qa_ctx *ctx, int64_t count, const double *values, int64_t index_offset, double *out_device);

/* Test hook, host only (no device needed): the coupling slabs the replay kernel would get for a CSR in host memory
 * (adjacency order).  Returns 1 when the model fits the slab format, 0 when it does not, < 0 on error. */
int qa_debug_pack_slabs(int32_t n, const int32_t *rowptr, const int32_t *col, const double *val, int32_t ngroups,
                        const int32_t *grp, const int32_t *coef, int64_t *nslabs_out, int64_t *bytes_out, int32_t *uniform_out,
                        unsigned char *slabs_out, uint32_t *off_out);

#ifdef __cplusplus
}
#endif
#endif /* QANNEAL_H */
