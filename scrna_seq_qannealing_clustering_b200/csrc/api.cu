// api.cu -- libqanneal.so: context, kernel selection and the sampling entry points of the C ABI (include/qanneal.h).
//
// What it replaces (reference file:line -> upstream algorithm):
//   sampler.sample_qubo / .sample / .sample_dqm / .sample_cqm call sites
//     Python_Functions/BQM_clustering.py:57,75,85,245,263,273,386; QA_subsampling.py:42,56,65;
//     DQM_clustering.py:45; CQM_clustering.py:53,89
//   -> dwave-neal neal/src/cpu_sa.cpp: general_simulated_annealing / simulated_annealing_run /
//      get_flip_energy / get_state_energy / FASTRAND (SURVEY.md rows a8-a11, Appendix C).
// The kernels live in their own translation units (see common.cuh); this file stages caller buffers, picks the kernel, hands
// the launch to it, evaluates the energies and collects the counters.
// Compile: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo (see __graft_entry__.build()).
#include "common.cuh"

using namespace qa;

namespace qa {

thread_local std::string g_err;

namespace {

int check_schedule(int32_t num_betas, const double *betas, int32_t sweeps_per_beta) {
    if (num_betas < 0 || sweeps_per_beta < 0) return fail(QA_ERR_ARG, "negative schedule size");
    if (num_betas > 0 && !betas) return fail(QA_ERR_ARG, "beta_schedule is null");
    return QA_OK;
}

// The annealing kernel of a call.  The rules, in order; the first that applies decides:
//   1. DENSE          QA_MODE_THROUGHPUT on a model with the dense k-way form: one problem, per-read seeds, no interrupt
//                     callback, sequential order and Metropolis acceptance (the tensor-core kernel, tolerance parity; it has
//                     neither dwave-samplers option).  Every other call runs a reference-order kernel:
//                     for sparse models the exact replay kernel is faster than any recompute or graph-coloured update
//                     (DESIGN.md 4.4), and bit-exact results meet the statistical bar trivially.
//   2. WARP_PER_READ  random variable order, whatever kernel was requested: the lockstep and replay kernels walk all 32 reads
//                     of a warp through the same variable, and random order has no order the reads share.
//      WARP_PER_READ  stream seeding (one xorshift128+ stream across reads), and batched models with rank-1 groups
//                     (qa_model_concat): the lockstep and replay kernels keep one copy of lambda / kappa per CTA, the
//                     warp-per-read kernel reads them per problem.
//   3. REPLAY         (deferred exact updates) when requested, or under AUTO from 32 reads per problem and 6144 reads in all
//                     (measured on B200, config 3: 1.26e10 vs 7.5e9 attempts/s for the warp-per-read kernel at 12 500 reads,
//                     4.3e9 vs 5.9e9 at 4096), if the model fits the slab format (build_replay_tables) and an interrupt
//                     callback comes with a single problem: the kernel polls a host-mapped flag whenever a CTA pulls its
//                     next group of reads.
//   4. a requested REPLAY that rule 3 refused (dense rows: the slab format does not apply) runs LOCKSTEP, or
//      WARP_PER_READ with an interrupt callback.
//   5. LOCKSTEP       when requested, or under AUTO from 32 reads per problem and 3.5 tiles of 32 reads per SM, without an
//                     interrupt callback: the lockstep kernel has no stopping point.
//   6. WARP_PER_READ  otherwise: any read count; with an interrupt callback it runs in read waves and polls between them.
// Sequential Gibbs acceptance follows rules 2-6 unchanged: every reference-order kernel has both acceptance rules.
int pick_kernel(qa_ctx *ctx, qa_model *M, int32_t reads_per_problem, int64_t total_reads, int32_t seed_mode, int32_t mode,
                bool interrupt, int32_t var_order, int32_t proposal, int *kernel) {
    const int P = M->num_problems;
    const bool auto_ok = ctx->kernel == QA_KERNEL_AUTO && reads_per_problem >= 32;
    if (mode == QA_MODE_THROUGHPUT && M->dn_ok && P == 1 && !interrupt && seed_mode == QA_SEED_PER_READ &&
        var_order == QA_ORDER_SEQUENTIAL && proposal == QA_PROPOSAL_METROPOLIS) {
        *kernel = QA_KERNEL_DENSE;
        return QA_OK;
    }
    *kernel = QA_KERNEL_WARP_PER_READ;
    if (var_order == QA_ORDER_RANDOM || seed_mode != QA_SEED_PER_READ || (P > 1 && M->ngroups > 0)) return QA_OK;
    if ((ctx->kernel == QA_KERNEL_REPLAY || (auto_ok && total_reads >= 6144)) && (!interrupt || P == 1)) {
        const int rc = build_replay_tables(M);
        if (rc) return rc;
        if (M->rp_ok) {
            *kernel = QA_KERNEL_REPLAY;
            QA_CUDA(cudaMemcpyAsync(M->d_descs, M->descs.data(), P * sizeof(ProblemDesc), cudaMemcpyHostToDevice, ctx->stream));
            return QA_OK;
        }
    }
    if (ctx->kernel == QA_KERNEL_REPLAY) {
        if (!interrupt) *kernel = QA_KERNEL_LOCKSTEP_PUSH;
        return QA_OK;
    }
    if ((ctx->kernel == QA_KERNEL_LOCKSTEP_PUSH || (auto_ok && 2 * total_reads >= (int64_t)ctx->num_sms * 32 * 7)) && !interrupt)
        *kernel = QA_KERNEL_LOCKSTEP_PUSH;
    return QA_OK;
}

// core: anneal all reads of all problems of a model; states/energies already on the device
int run_anneal(qa_ctx *ctx, qa_model *M, int32_t reads_per_problem, int8_t *d_states, double *d_energies,
               int32_t num_betas, const double *d_betas, int32_t sweeps_per_beta, const unsigned long long *d_seeds,
               int32_t seed_mode, int32_t mode, int32_t var_order, int32_t proposal, qa_interrupt_fn interrupt, void *iuser,
               qa_stats *st, int64_t *completed) {
    const int P = M->num_problems;
    const int64_t total_reads = (int64_t)P * reads_per_problem;
    const int32_t rpad = (reads_per_problem + 31) & ~31;
    *completed = 0;
    if (total_reads == 0) return QA_OK;

    // packed transposed spins for the energy kernel
    size_t packed_words = 0;
    for (int p = 0; p < P; ++p) packed_words += (size_t)M->descs[p].nch * rpad;
    int rc = ensure(ctx->packed, std::max<size_t>(packed_words, 1) * sizeof(uint32_t));
    if (rc) return rc;
    {
        size_t off = 0;
        int64_t st_off = 0;
        for (int p = 0; p < P; ++p) {
            ProblemDesc &D = M->descs[p];
            D.reads = reads_per_problem;
            D.rpad = rpad;
            D.read_base = (int64_t)p * reads_per_problem;
            D.states = d_states + st_off;
            D.packedT = (uint32_t *)ctx->packed.p + off;
            D.energies = d_energies + (int64_t)p * reads_per_problem;
            D.betas = ctx->betas_per_problem ? d_betas + (int64_t)p * num_betas : nullptr;
            off += (size_t)D.nch * rpad;
            st_off += (int64_t)reads_per_problem * D.n;
        }
        QA_CUDA(cudaMemcpyAsync(M->d_descs, M->descs.data(), P * sizeof(ProblemDesc), cudaMemcpyHostToDevice, ctx->stream));
    }

    int kernel = 0;
    rc = pick_kernel(ctx, M, reads_per_problem, total_reads, seed_mode, mode, interrupt != nullptr, var_order, proposal, &kernel);
    if (rc) return rc;
    ctx->last_kernel = kernel;
    QA_CUDA(cudaMemsetAsync(ctx->d_stats, 0, (QA_NSTAT + 1 + QA_NDEBUG) * sizeof(unsigned long long), ctx->stream));
    QA_CUDA(cudaMemsetAsync(ctx->d_flag, 0, 2 * sizeof(int), ctx->stream));

    AnnealParams A;
    memset(&A, 0, sizeof(A));
    A.descs = M->d_descs;
    A.num_problems = P;
    A.reads_per_problem = reads_per_problem;
    A.total_reads = total_reads;
    A.betas = d_betas;
    A.num_betas = num_betas;
    A.sweeps_per_beta = sweeps_per_beta;
    A.seeds = d_seeds;
    A.seed_mode = seed_mode;
    A.counter = ctx->d_stats + QA_NSTAT;
    A.stats = ctx->d_stats;
    A.error_flag = ctx->d_flag;

    // the launch itself lives next to each kernel (anneal_*.cu)
    Launch L;
    L.ctx = ctx;
    L.M = M;
    L.A = A;
    L.gk = M->ngroups == 0 ? GK_NONE : M->gbounds ? GK_INTERVAL : M->groups_i32 ? GK_EQ32 : GK_EQ64;
    L.prop = proposal == QA_PROPOSAL_GIBBS ? PROP_GIBBS : PROP_METROPOLIS;
    L.random_order = var_order == QA_ORDER_RANDOM;
    L.interrupt = interrupt;
    L.iuser = iuser;
    L.st = st;
    L.done = 0;
    L.interrupted = false;
    if (kernel == QA_KERNEL_WARP_PER_READ) rc = launch_ref(L);
    else if (kernel == QA_KERNEL_DENSE) rc = launch_dense(L);
    else if (kernel == QA_KERNEL_REPLAY) rc = launch_replay(L);
    else rc = launch_lockstep(L);
    if (rc) return rc;
    const int64_t done = L.done;
    QA_CUDA(cudaEventRecord(ctx->ev[3], ctx->stream));
    if (kernel != QA_KERNEL_DENSE) {   // the dense kernel evaluates the energies itself (one more field pass)
        rc = launch_energy(ctx, M, reads_per_problem);
        if (rc) return rc;
    }
    QA_CUDA(cudaEventRecord(ctx->ev[4], ctx->stream));
    int flag = 0;
    unsigned long long hs[QA_NSTAT + 1 + QA_NDEBUG];
    QA_CUDA(cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(hs, ctx->d_stats, sizeof(hs), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
#ifdef QA_RP_PROFILE
    fprintf(stderr, "[qa profile] cycles summed over warps: setup %llu slab-wait %llu stage-wait %llu prologue %llu batch %llu sequential %llu replay-passes %llu push-passes %llu\n",
            hs[QA_NSTAT + 1], hs[QA_NSTAT + 2], hs[QA_NSTAT + 3], hs[QA_NSTAT + 4], hs[QA_NSTAT + 5], hs[QA_NSTAT + 6], hs[QA_NSTAT + 7], hs[QA_NSTAT + 8]);
#endif
    if (flag == QA_ERR_SMEM_BASE) return fail(QA_ERR_CUDA, "replay kernel: dynamic shared memory does not start where the layout assumed");
    if (flag != 0) return fail(flag, "initial states must be +1/-1");
    if (st) {
        st->candidates += hs[ST_CAND];
        st->draws += hs[ST_DRAWS];
        st->accepted += hs[ST_ACC];
        st->nbr_updates += hs[ST_NBR];
        st->active_chunks += hs[ST_ACTIVE];
        st->chunks += hs[ST_CHUNKS];
        st->near_ties += hs[ST_TIES];
        st->ms_anneal += elapsed(ctx->ev[2], ctx->ev[3]);
        st->ms_energy += elapsed(ctx->ev[3], ctx->ev[4]);
        uint64_t att = 0;
        for (int p = 0; p < P; ++p) att += (uint64_t)M->descs[p].n;
        st->attempts += att * (uint64_t)num_betas * (uint64_t)sweeps_per_beta * (uint64_t)(done / P);
    }
    *completed = done;
    return QA_OK;
}

}  // namespace

// stage caller buffers (host or device), run, and return results
int sample_common(qa_ctx *ctx, qa_model *M, int32_t reads_per_problem, int8_t *states_inout, double *energies_out,
                  int32_t num_betas, const double *beta_schedule, int32_t sweeps_per_beta, const uint64_t *seeds,
                  int32_t seed_mode, int32_t mode, qa_interrupt_fn interrupt, void *iuser, qa_stats *stats_out,
                  int32_t var_order, int32_t proposal) {
    if (!ctx || !M) return fail(QA_ERR_ARG, "null context or model");
    if (var_order != QA_ORDER_SEQUENTIAL && var_order != QA_ORDER_RANDOM) return fail(QA_ERR_ARG, "unknown var_order");
    if (proposal != QA_PROPOSAL_METROPOLIS && proposal != QA_PROPOSAL_GIBBS) return fail(QA_ERR_ARG, "unknown proposal");
    if (M->ctx != ctx) return fail(QA_ERR_ARG, "model belongs to another context");
    if (reads_per_problem < 0) return fail(QA_ERR_ARG, "negative num_reads");
    if (mode != QA_MODE_REFERENCE && mode != QA_MODE_THROUGHPUT) return fail(QA_ERR_ARG, "unknown mode");
    if (seed_mode != QA_SEED_PER_READ && seed_mode != QA_SEED_STREAM) return fail(QA_ERR_ARG, "unknown seed_mode");
    if (seed_mode == QA_SEED_STREAM && M->num_problems != 1) return fail(QA_ERR_ARG, "stream seeding needs a single problem");
    int rc = check_schedule(num_betas, beta_schedule, sweeps_per_beta);
    if (rc) return rc;
    QA_CUDA(cudaSetDevice(ctx->device));
    const int64_t total_reads = (int64_t)M->num_problems * reads_per_problem;
    qa_stats st;
    memset(&st, 0, sizeof(st));
    const uint32_t launches0 = ctx->launches;
    if (total_reads == 0) {
        if (stats_out) *stats_out = st;
        return 0;
    }
    if (!states_inout || !energies_out || !seeds) return fail(QA_ERR_ARG, "null states/energies/seeds");
    const int64_t state_bytes = (int64_t)reads_per_problem * M->n_total;

    QA_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    int8_t *d_states = states_inout;
    const bool st_host = !is_device_ptr(states_inout);
    if (st_host) {
        rc = ensure(ctx->states, (size_t)std::max<int64_t>(state_bytes, 1));
        if (rc) return rc;
        d_states = (int8_t *)ctx->states.p;
        QA_CUDA(cudaMemcpyAsync(d_states, states_inout, (size_t)state_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    double *d_energies = energies_out;
    const bool en_host = !is_device_ptr(energies_out);
    if (en_host) {
        rc = ensure(ctx->energies, (size_t)total_reads * sizeof(double));
        if (rc) return rc;
        d_energies = (double *)ctx->energies.p;
    }
    const int64_t nseeds = seed_mode == QA_SEED_STREAM ? 1 : total_reads;
    const unsigned long long *d_seeds = (const unsigned long long *)seeds;
    if (!is_device_ptr(seeds)) {
        rc = ensure(ctx->seeds, (size_t)nseeds * sizeof(uint64_t));
        if (rc) return rc;
        QA_CUDA(cudaMemcpyAsync(ctx->seeds.p, seeds, (size_t)nseeds * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
        d_seeds = (const unsigned long long *)ctx->seeds.p;
    }
    const double *d_betas = beta_schedule;
    if (num_betas > 0 && !is_device_ptr(beta_schedule)) {
        const size_t nb = (size_t)num_betas * (ctx->betas_per_problem ? (size_t)M->num_problems : 1);
        rc = ensure(ctx->betas, nb * sizeof(double));
        if (rc) return rc;
        QA_CUDA(cudaMemcpyAsync(ctx->betas.p, beta_schedule, nb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        d_betas = (const double *)ctx->betas.p;
    }
    QA_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));

    int64_t completed = 0;
    rc = run_anneal(ctx, M, reads_per_problem, d_states, d_energies, num_betas, d_betas, sweeps_per_beta, d_seeds, seed_mode,
                    mode, var_order, proposal, interrupt, iuser, &st, &completed);
    if (rc) return rc;

    QA_CUDA(cudaEventRecord(ctx->ev[4], ctx->stream));
    if (st_host) QA_CUDA(cudaMemcpyAsync(states_inout, d_states, (size_t)state_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (en_host) QA_CUDA(cudaMemcpyAsync(energies_out, d_energies, (size_t)total_reads * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaEventRecord(ctx->ev[5], ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    st.ms_h2d += elapsed(ctx->ev[0], ctx->ev[1]);
    st.ms_d2h += elapsed(ctx->ev[4], ctx->ev[5]);
    st.ms_total += elapsed(ctx->ev[0], ctx->ev[5]);
    st.total_launches = ctx->launches - launches0;
    if (stats_out) *stats_out = st;
    return (int)std::min<int64_t>(completed / M->num_problems, 0x7fffffff);
}

}  // namespace qa

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char *qa_last_error(void) { return g_err.c_str(); }

int qa_version(void) { return QA_VERSION; }

int qa_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int qa_ctx_create(int device_id, qa_ctx **out) {
    if (!out) return fail(QA_ERR_ARG, "out is null");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(QA_ERR_CUDA, "no CUDA device available: libqanneal has no CPU fallback");
    }
    if (device_id < 0 || device_id >= ndev) return fail(QA_ERR_ARG, "device_id out of range");
    QA_CUDA(cudaSetDevice(device_id));
    qa_ctx *ctx = new qa_ctx();
    ctx->device = device_id;
    cudaDeviceProp prop;
    QA_CUDA(cudaGetDeviceProperties(&prop, device_id));
    ctx->num_sms = prop.multiProcessorCount;
    if (const char *e = getenv("QA_REPLAY_SWITCH_PERMILLE")) ctx->replay_switch_permille = atoi(e);  // development knobs
    if (const char *e = getenv("QA_REPLAY_WARPS")) ctx->replay_warps = atoi(e);
    if (const char *e = getenv("QA_REPLAY_KWAY")) ctx->replay_kway = atoi(e);
    QA_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    for (auto &ev : ctx->ev) QA_CUDA(cudaEventCreate(&ev));
    QA_CUDA(cudaMalloc((void **)&ctx->d_stats, (QA_NSTAT + 1 + QA_NDEBUG) * sizeof(unsigned long long)));
    QA_CUDA(cudaMalloc((void **)&ctx->d_flag, 2 * sizeof(int)));
    QA_CUDA(cudaMalloc((void **)&ctx->d_best_e, sizeof(double)));
    QA_CUDA(cudaMalloc((void **)&ctx->d_best_i, sizeof(long long)));
    QA_CUDA(cudaHostAlloc((void **)&ctx->h_iflag, sizeof(int), cudaHostAllocMapped));
    *ctx->h_iflag = 0;
    QA_CUDA(cudaHostGetDevicePointer((void **)&ctx->d_iflag, ctx->h_iflag, 0));
    *out = ctx;
    return QA_OK;
}

int qa_ctx_destroy(qa_ctx *ctx) {
    if (!ctx) return QA_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    release(ctx->f); release(ctx->spw); release(ctx->fT); release(ctx->sf); release(ctx->states); release(ctx->energies); release(ctx->seeds);
    release(ctx->betas); release(ctx->packed); release(ctx->misc); release(ctx->cubtmp);
    if (ctx->d_stats) cudaFree(ctx->d_stats);
    if (ctx->d_flag) cudaFree(ctx->d_flag);
    if (ctx->d_best_e) cudaFree(ctx->d_best_e);
    if (ctx->d_best_i) cudaFree(ctx->d_best_i);
    if (ctx->h_iflag) cudaFreeHost(ctx->h_iflag);
    for (auto &ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return QA_OK;
}

int qa_ctx_synchronize(qa_ctx *ctx) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    return QA_OK;
}

int qa_ctx_set_kernel(qa_ctx *ctx, int kernel) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    if (kernel != QA_KERNEL_AUTO && kernel != QA_KERNEL_WARP_PER_READ && kernel != QA_KERNEL_LOCKSTEP_PUSH &&
        kernel != QA_KERNEL_REPLAY)
        return fail(QA_ERR_ARG, "kernel must be QA_KERNEL_AUTO, _WARP_PER_READ, _LOCKSTEP_PUSH or _REPLAY");
    ctx->kernel = kernel;
    return QA_OK;
}

int qa_ctx_last_kernel(qa_ctx *ctx) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    return ctx->last_kernel;
}

int qa_ctx_resident_reads(qa_ctx *ctx) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    int reads = 0;
    const int rc = ref_resident_reads(ctx, &reads);
    return rc ? rc : reads;
}

int qa_sa_sample_model_ex(qa_ctx *ctx, qa_model *model, int32_t num_reads, int8_t *states_inout, double *energies_out,
                          int32_t num_betas, const double *beta_schedule, int32_t sweeps_per_beta, const uint64_t *seeds,
                          int32_t seed_mode, int32_t mode, int32_t var_order, int32_t proposal, qa_interrupt_fn interrupt,
                          void *interrupt_user, qa_stats *stats_out) {
    if (model && model->num_problems != 1) return fail(QA_ERR_ARG, "use qa_sa_sample_ising_batch for batched models");
    return sample_common(ctx, model, num_reads, states_inout, energies_out, num_betas, beta_schedule, sweeps_per_beta, seeds,
                         seed_mode, mode, interrupt, interrupt_user, stats_out, var_order, proposal);
}

int qa_sa_sample_model(qa_ctx *ctx, qa_model *model, int32_t num_reads, int8_t *states_inout, double *energies_out,
                       int32_t num_betas, const double *beta_schedule, int32_t sweeps_per_beta, const uint64_t *seeds,
                       int32_t seed_mode, int32_t mode, qa_interrupt_fn interrupt, void *interrupt_user, qa_stats *stats_out) {
    return qa_sa_sample_model_ex(ctx, model, num_reads, states_inout, energies_out, num_betas, beta_schedule, sweeps_per_beta,
                                 seeds, seed_mode, mode, QA_ORDER_SEQUENTIAL, QA_PROPOSAL_METROPOLIS, interrupt, interrupt_user,
                                 stats_out);
}

int qa_sa_sample_ising(qa_ctx *ctx, int32_t n, const double *h, int64_t m, const int32_t *starts, const int32_t *ends,
                       const double *weights, int32_t num_reads, int8_t *states_inout, double *energies_out, int32_t num_betas,
                       const double *beta_schedule, int32_t sweeps_per_beta, const uint64_t *seeds, int32_t seed_mode,
                       int32_t mode, qa_interrupt_fn interrupt, void *interrupt_user, qa_stats *stats_out) {
    return qa_sa_sample_ising_ex(ctx, n, h, m, starts, ends, weights, num_reads, states_inout, energies_out, num_betas,
                                 beta_schedule, sweeps_per_beta, seeds, seed_mode, mode, QA_ORDER_SEQUENTIAL,
                                 QA_PROPOSAL_METROPOLIS, interrupt, interrupt_user, stats_out);
}

int qa_sa_sample_ising_ex(qa_ctx *ctx, int32_t n, const double *h, int64_t m, const int32_t *starts, const int32_t *ends,
                          const double *weights, int32_t num_reads, int8_t *states_inout, double *energies_out,
                          int32_t num_betas, const double *beta_schedule, int32_t sweeps_per_beta, const uint64_t *seeds,
                          int32_t seed_mode, int32_t mode, int32_t var_order, int32_t proposal, qa_interrupt_fn interrupt,
                          void *interrupt_user, qa_stats *stats_out) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    cudaEvent_t b0 = nullptr, b1 = nullptr;
    QA_CUDA(cudaSetDevice(ctx->device));
    QA_CUDA(cudaEventCreate(&b0));
    QA_CUDA(cudaEventCreate(&b1));
    const uint32_t l0 = ctx->launches;
    cudaEventRecord(b0, ctx->stream);
    qa_model *M = nullptr;
    int rc = qa_model_from_ising(ctx, n, h, m, starts, ends, weights, &M);
    cudaEventRecord(b1, ctx->stream);
    if (rc == QA_OK) {
        rc = sample_common(ctx, M, num_reads, states_inout, energies_out, num_betas, beta_schedule, sweeps_per_beta, seeds,
                           seed_mode, mode, interrupt, interrupt_user, stats_out, var_order, proposal);
        if (rc >= 0 && stats_out) {
            cudaEventSynchronize(b1);
            stats_out->ms_build = elapsed(b0, b1);
            stats_out->total_launches = ctx->launches - l0;
        }
    }
    qa_model_destroy(M);
    cudaEventDestroy(b0);
    cudaEventDestroy(b1);
    return rc;
}

int qa_sa_sample_ising_batch(qa_ctx *ctx, int32_t num_problems, const int64_t *var_offsets, const int64_t *coupler_offsets,
                             const double *h, const int32_t *starts, const int32_t *ends, const double *weights,
                             int32_t reads_per_problem, int8_t *states_inout, double *energies_out, int32_t num_betas,
                             const double *beta_schedule, int32_t sweeps_per_beta, const uint64_t *seeds, qa_stats *stats_out) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    if (num_problems < 1 || !var_offsets || !coupler_offsets) return fail(QA_ERR_ARG, "bad batch description");
    for (int p = 0; p < num_problems; ++p)
        if (var_offsets[p + 1] < var_offsets[p] || coupler_offsets[p + 1] < coupler_offsets[p])
            return fail(QA_ERR_ARG, "offsets must be non-decreasing");
    if (var_offsets[0] != 0 || coupler_offsets[0] != 0) return fail(QA_ERR_ARG, "offsets must start at 0");
    QA_CUDA(cudaSetDevice(ctx->device));
    cudaEvent_t b0 = nullptr, b1 = nullptr;
    QA_CUDA(cudaEventCreate(&b0));
    QA_CUDA(cudaEventCreate(&b1));
    const uint32_t l0 = ctx->launches;
    cudaEventRecord(b0, ctx->stream);
    qa_model *M = nullptr;
    int rc = model_create(ctx, num_problems, var_offsets, coupler_offsets, h, starts, ends, weights, &M);
    cudaEventRecord(b1, ctx->stream);
    if (rc == QA_OK) {
        rc = sample_common(ctx, M, reads_per_problem, states_inout, energies_out, num_betas, beta_schedule, sweeps_per_beta,
                           seeds, QA_SEED_PER_READ, QA_MODE_REFERENCE, nullptr, nullptr, stats_out);
        if (rc >= 0 && stats_out) {
            cudaEventSynchronize(b1);
            stats_out->ms_build = elapsed(b0, b1);
            stats_out->total_launches = ctx->launches - l0;
        }
    }
    qa_model_destroy(M);
    cudaEventDestroy(b0);
    cudaEventDestroy(b1);
    return rc;
}

int qa_energy_argmin(qa_ctx *ctx, qa_model *M, int32_t num_reads, const int8_t *states, double *energies_out,
                     double *best_energy, int64_t *best_index, qa_stats *stats_out) {
    if (!ctx || !M) return fail(QA_ERR_ARG, "null context or model");
    if (M->num_problems != 1) return fail(QA_ERR_ARG, "single-problem model required");
    if (num_reads < 0) return fail(QA_ERR_ARG, "negative num_reads");
    qa_stats st;
    memset(&st, 0, sizeof(st));
    if (num_reads == 0) {
        if (best_energy) *best_energy = INFINITY;
        if (best_index) *best_index = -1;
        if (stats_out) *stats_out = st;
        return QA_OK;
    }
    if (!states) return fail(QA_ERR_ARG, "null states");
    QA_CUDA(cudaSetDevice(ctx->device));
    const uint32_t l0 = ctx->launches;
    ProblemDesc &D = M->descs[0];
    const int32_t rpad = (num_reads + 31) & ~31;
    const int64_t state_bytes = (int64_t)num_reads * D.n;
    QA_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    const int8_t *d_states = states;
    if (!is_device_ptr(states)) {
        int rc = ensure(ctx->states, (size_t)std::max<int64_t>(state_bytes, 1));
        if (rc) return rc;
        QA_CUDA(cudaMemcpyAsync(ctx->states.p, states, (size_t)state_bytes, cudaMemcpyHostToDevice, ctx->stream));
        d_states = (const int8_t *)ctx->states.p;
    }
    double *d_energies = energies_out;
    const bool en_host = !energies_out || !is_device_ptr(energies_out);
    if (en_host) {
        int rc = ensure(ctx->energies, (size_t)num_reads * sizeof(double));
        if (rc) return rc;
        d_energies = (double *)ctx->energies.p;
    }
    int rc = ensure(ctx->packed, (size_t)std::max<int64_t>((int64_t)D.nch * rpad, 1) * sizeof(uint32_t));
    if (rc) return rc;
    D.reads = num_reads;
    D.rpad = rpad;
    D.read_base = 0;
    D.states = const_cast<int8_t *>(d_states);
    D.packedT = (uint32_t *)ctx->packed.p;
    D.energies = d_energies;
    QA_CUDA(cudaMemcpyAsync(M->d_descs, &D, sizeof(ProblemDesc), cudaMemcpyHostToDevice, ctx->stream));
    QA_CUDA(cudaMemsetAsync(ctx->d_flag, 0, 2 * sizeof(int), ctx->stream));
    QA_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
    {
        const int64_t threads = (int64_t)num_reads * 32;
        if ((rc = launch_pack_states(ctx, D, threads))) return rc;
        if ((rc = launch_energy(ctx, M, num_reads))) return rc;
        if ((rc = launch_argmin(ctx, d_energies, num_reads))) return rc;
    }
    QA_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    int flag = 0;
    double be = 0;
    long long bi = 0;
    QA_CUDA(cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(&be, ctx->d_best_e, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(&bi, ctx->d_best_i, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    if (energies_out && en_host)
        QA_CUDA(cudaMemcpyAsync(energies_out, d_energies, (size_t)num_reads * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaEventRecord(ctx->ev[3], ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    if (flag != 0) return fail(flag, "states must be +1/-1");
    if (best_energy) *best_energy = be;
    if (best_index) *best_index = bi;
    st.ms_h2d = elapsed(ctx->ev[0], ctx->ev[1]);
    st.ms_energy = elapsed(ctx->ev[1], ctx->ev[2]);
    st.ms_d2h = elapsed(ctx->ev[2], ctx->ev[3]);
    st.total_launches = ctx->launches - l0;
    if (stats_out) *stats_out = st;
    return QA_OK;
}

}  // extern "C"
