// anneal_ref.cu -- k_anneal_ref: one WARP per read, neal's loop in reference order (bit-exact; any read count; stream seeding;
// batched models with rank-1 groups).  Restates neal simulated_annealing_run() (neal/src/cpu_sa.cpp; SURVEY.md rows a8-a11).
//   * the read's local fields f[v] = h_v + sum_j J_vj s_j live in HBM as fp64 and are streamed 32 variables (256 B) at a time
//     with ld.global.cg + prefetch.global.L2 run-ahead; spins are bit-packed.  neal's dE[v] is recovered exactly as -2*s_v*f[v]
//     (scaling by +-2 commutes with rounding), so a flip needs no read of s_j: every neighbour update is one fire-and-forget
//     red.global.add.f64 f[j], -2*s_v*J performed in L2.
//   * the 32 lanes of a chunk decide "candidate" (dE < 44.36142/beta) in parallel; candidates are then resolved in variable
//     order with a warp-uniform xorshift128+ stream, so the sequence of RNG draws, accepts and fp64 roundings is exactly neal's.
//   * persistent grid (multiple of the SM count), reads pulled from an atomic counter; only resident warps own fp64 scratch.
//   * dwave-samplers >= 1.0's sample options (include/qanneal.h): Gibbs acceptance in the chunked loop, and a random-order
//     loop of its own (random_order_sweeps) -- the only kernel that runs random order.
#include "device_common.cuh"

using namespace qa;

namespace {

// ------------------------------------------------------------------------------------------------
// random variable order (dwave-samplers randomize_order=True): per attempt one warp-uniform xorshift128+ draw picks
// v = r % n, then the decision of v as in the chunked loop -- every lane computes it from the same loads and the same RNG
// state, so it is warp-uniform without a shuffle.  There is no chunk register cache: f[v] and the spin word are read from
// the read's scratch at every attempt, and an accepted flip's neighbour reductions are ordered before the next attempt's
// loads by __syncwarp (the next v may be a neighbour just pushed).
// ------------------------------------------------------------------------------------------------
template <GroupKind GROUPS, Proposal PROP>
__device__ void random_order_sweeps(const ProblemDesc &D, const AnnealParams &P, double *__restrict__ f,
                                    uint32_t *__restrict__ spw, unsigned long long &s0, unsigned long long &s1, long long *Mw,
                                    WarpStats &st) {
    const int lane = threadIdx.x & 31;
    const int n = D.n;
    for (int b = 0; b < P.num_betas; ++b) {
        const double beta = (D.betas ? D.betas : P.betas)[b];
        const double thr = 44.36142 / beta;
        for (int sw = 0; sw < P.sweeps_per_beta; ++sw) {
            for (int k = 0; k < n; ++k) {
                const int v = (int)(rng_next(s0, s1) % (unsigned long long)n);   // the order draw comes first
                st.draws++;
                const double fv = __ldcg(f + v);
                const uint32_t wv = __ldcg(spw + (v >> 5));
                const bool up = (wv >> (v & 31)) & 1u;
                double dE = up ? -2.0 * fv : 2.0 * fv;
                int g = -1;
                long long a = 0;
                if (GROUPS != GK_NONE) {
                    g = __ldg(D.grp + v);
                    if (g >= 0) {
                        a = __ldg(D.coef + v);
                        const long long kap = __ldg(D.kappa + g);
                        long long glo = 0, ghi = 0;
                        if (GROUPS == GK_INTERVAL) {
                            glo = __ldg(D.kappa + D.ngroups + g);
                            ghi = __ldg(D.kappa + 2 * D.ngroups + g);
                        }
                        dE = dE + group_flip_cost<GROUPS>(__ldg(D.lambda + g), a, up, Mw[g] + kap, glo, ghi);
                    }
                }
                if (dE >= thr) continue;
                st.cand++;
                bool acc = true;
                if (PROP == PROP_GIBBS ? !(dE <= -thr) : dE > 0.0) {
                    const double rd = __ull2double_rn(rng_next(s0, s1));
                    st.draws++;
                    if (PROP == PROP_GIBBS) {
                        const double q = rd * (1.0 + exp(dE * beta));
                        acc = QA_TWO64 > q;
                        if (fabs(QA_TWO64 - q) <= QA_TWO64 * 3.5527136788005009e-15) st.ties++;
                    } else {
                        const double p = exp(-dE * beta) * QA_TWO64;
                        acc = p > rd;
                        if (fabs(p - rd) <= p * 3.5527136788005009e-15) st.ties++;
                    }
                }
                if (!acc) continue;
                st.acc++;
                const int r0 = __ldg(D.rowptr + v), r1 = __ldg(D.rowptr + v + 1);
                const double cf = up ? -2.0 : 2.0;  // f[j] += -2*s_v*J  <=> dE[j] += 4*s_v*J*s_j
                st.nbr += (unsigned long long)(r1 - r0);
                for (int e = r0 + lane; e < r1; e += 32) red_add_f64(f + __ldg(D.col + e), cf * __ldg(D.val + e));
                __syncwarp();   // every lane has read spw / Mw of this attempt before lane 0 changes them
                if (lane == 0) {
                    __stcg(spw + (v >> 5), wv ^ (1u << (v & 31)));
                    if (GROUPS != GK_NONE) {
                        if (g >= 0) Mw[g] -= 2 * a * (up ? 1 : -1);
                    }
                }
                __syncwarp();   // the reductions and lane 0's stores before the next attempt's loads
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// one read, reference order.  Restates neal simulated_annealing_run() for one `state`.
// ------------------------------------------------------------------------------------------------
// GROUPS: GK_NONE, GK_EQ64 (equality groups of both widths) or GK_INTERVAL; lambda / kappa / bounds are read per problem.
// PROP: the acceptance rule.  RANDOM: random variable order (random_order_sweeps) instead of the chunked sequential loop.
template <GroupKind GROUPS, Proposal PROP, bool RANDOM>
__device__ void anneal_read(const ProblemDesc &D, const AnnealParams &P, int64_t r_local, double *__restrict__ f,
                            uint32_t *__restrict__ spw, unsigned long long &s0, unsigned long long &s1,
                            long long *Mw, WarpStats &st, int *error_flag) {
    const int lane = threadIdx.x & 31;
    const int n = D.n;
    const int nch = D.nch;
    int8_t *state_row = D.states + r_local * (int64_t)n;

    // ---- pack the initial +-1 bytes into spin words (bit = 1 <=> s = +1); padding variables are +1
    for (int cb = 0; cb < nch; cb += 32) {
        uint32_t wg = 0xffffffffu;
        const int cend = min(32, nch - cb);
        for (int k = 0; k < cend; ++k) {
            const int v = (cb + k) * 32 + lane;
            int s = 1;
            if (v < n) {
                s = state_row[v];
                if (s != 1 && s != -1) atomicExch(error_flag, QA_ERR_STATE);
            }
            const uint32_t w = __ballot_sync(FULL_MASK, s > 0);
            if (lane == k) wg = w;
        }
        __stcg(spw + cb + lane, wg);
    }
    __syncwarp();

    // ---- local fields, neal get_flip_energy(): energy = h[v]; for nbr in adjacency order: energy += s_nbr*J
    for (int c = 0; c < nch; ++c) {
        const int v = c * 32 + lane;
        double fv = -INFINITY;  // padding: dE = -2*(+1)*(-inf) = +inf, never a candidate
        if (v < n) {
            fv = D.h[v];
            const int e0 = D.rowptr[v], e1 = D.rowptr[v + 1];
            for (int e = e0; e < e1; ++e) {
                const int j = D.col[e];
                const uint32_t wj = __ldcg(spw + (j >> 5));
                const double J = D.val[e];
                fv += ((wj >> (j & 31)) & 1u) ? J : -J;
            }
        }
        __stcg(f + v, fv);
    }
    if (GROUPS != GK_NONE) {
        for (int g = lane; g < D.ngroups; g += 32) Mw[g] = 0;
        __syncwarp();
        for (int c = 0; c < nch; ++c) {
            const int v = c * 32 + lane;
            const int g = D.grp[v];
            if (g >= 0) {
                const uint32_t wv = __ldcg(spw + c);
                const long long a = D.coef[v];
                atomicAdd(reinterpret_cast<unsigned long long *>(Mw + g),
                          (unsigned long long)(((wv >> lane) & 1u) ? a : -a));
            }
        }
    }
    __syncwarp();

    // ---- the anneal: for beta: for sweep: for var (neal order; random order: random_order_sweeps, and no chunked sweep)
    if (RANDOM) random_order_sweeps<GROUPS, PROP>(D, P, f, spw, s0, s1, Mw, st);
    for (int b = 0; b < (RANDOM ? 0 : P.num_betas); ++b) {
        const double beta = (D.betas ? D.betas : P.betas)[b];
        const double thr = 44.36142 / beta;
        for (int sw = 0; sw < P.sweeps_per_beta; ++sw) {
            uint32_t wg = 0;
            bool gdirty = false;
            for (int c = 0; c < nch; ++c) {
                const int k = c & 31;
                if (k == 0) {
                    wg = __ldcg(spw + c + lane);
                    gdirty = false;
                }
                if ((lane & 15) == 0) {
                    int cp = c + QA_PREFETCH_CHUNKS;
                    if (cp >= nch) cp %= nch;
                    prefetch_l2(f + cp * 32 + lane);
                }
                const int v = c * 32 + lane;
                double fv = __ldcg(f + v);
                uint32_t w = __shfl_sync(FULL_MASK, wg, k);
                int g = -1;
                long long a = 0, kap = 0, glo = 0, ghi = 0;
                double lam = 0.0;
                if (GROUPS != GK_NONE) {
                    g = __ldg(D.grp + v);
                    if (g >= 0) {
                        a = __ldg(D.coef + v);
                        lam = __ldg(D.lambda + g);
                        kap = __ldg(D.kappa + g);
                        if (GROUPS == GK_INTERVAL) {
                            glo = __ldg(D.kappa + D.ngroups + g);
                            ghi = __ldg(D.kappa + 2 * D.ngroups + g);
                        }
                    }
                }
                // neal's delta_energy[v] == -2*s_v*f[v] exactly; plus the lazily evaluated rank-1 cost
                auto flip_cost = [&](uint32_t word) -> double {
                    const bool up = (word >> lane) & 1u;
                    double d = up ? -2.0 * fv : 2.0 * fv;
                    if (GROUPS != GK_NONE) {
                        if (g >= 0) d = d + group_flip_cost<GROUPS>(lam, a, up, Mw[g] + kap, glo, ghi);
                    }
                    return d;
                };
                double dE = flip_cost(w);
                bool cand = !(dE >= thr);  // neal: if (delta_energy[var] >= threshold) continue;
                uint32_t pend = __ballot_sync(FULL_MASK, cand);
                if (pend) {
                    st.active++;
                    const int e0 = __ldg(D.rowptr + v), e1 = __ldg(D.rowptr + v + 1);
                    bool pvalid = false;
                    double p = 0.0;
                    while (pend) {
                        const int l = __ffs(pend) - 1;
                        pend &= pend - 1;
                        st.cand++;
                        const double dEl = __shfl_sync(FULL_MASK, dE, l);
                        bool acc = true;
                        if (PROP == PROP_GIBBS ? !(dEl <= -thr) : dEl > 0.0) {
                            const uint32_t pv = __ballot_sync(FULL_MASK, pvalid);
                            if (!((pv >> l) & 1u)) {
                                // exp(-dE*beta)*2^64 (Gibbs: 1 + exp(dE*beta)) for every lane that may need it (one SIMT pass)
                                if (PROP == PROP_GIBBS) {
                                    if (!pvalid && cand && !(dE <= -thr)) p = 1.0 + exp(dE * beta);
                                } else {
                                    if (!pvalid && cand && dE > 0.0) p = exp(-dE * beta) * QA_TWO64;
                                }
                                pvalid = true;
                            }
                            const unsigned long long rnd = rng_next(s0, s1);
                            st.draws++;
                            const double pl = __shfl_sync(FULL_MASK, p, l);
                            const double rd = __ull2double_rn(rnd);
                            if (PROP == PROP_GIBBS) {
                                const double q = rd * pl;
                                acc = QA_TWO64 > q;  // dwave-samplers Gibbs: 1 / (1 + exp(dE*beta)) > rand / 2^64
                                if (fabs(QA_TWO64 - q) <= QA_TWO64 * 3.5527136788005009e-15) st.ties++;
                            } else {
                                acc = pl > rd;  // neal: exp(-dE*beta) * RANDMAX > rand
                                if (fabs(pl - rd) <= pl * 3.5527136788005009e-15) st.ties++;
                            }
                        }
                        if (acc) {
                            st.acc++;
                            const int r0 = __shfl_sync(FULL_MASK, e0, l);
                            const int r1 = __shfl_sync(FULL_MASK, e1, l);
                            const bool up_l = (w >> l) & 1u;
                            const double cf = up_l ? -2.0 : 2.0;  // f[j] += -2*s_l*J  <=> dE[j] += 4*s_l*J*s_j
                            st.nbr += (unsigned long long)(r1 - r0);
                            uint32_t touched = 0;
                            for (int base = r0; base < r1; base += 32) {
                                const int e = base + lane;
                                const bool valid = e < r1;
                                int j = -1;
                                double d = 0.0;
                                if (valid) {
                                    j = __ldg(D.col + e);
                                    d = cf * __ldg(D.val + e);
                                    red_add_f64(f + j, d);
                                }
                                uint32_t inm = __ballot_sync(FULL_MASK, valid && (j >> 5) == c);
                                while (inm) {  // patch register copies of this chunk, in neighbour order
                                    const int kk = __ffs(inm) - 1;
                                    inm &= inm - 1;
                                    const int tj = __shfl_sync(FULL_MASK, j, kk) & 31;
                                    const double dk = __shfl_sync(FULL_MASK, d, kk);
                                    if (lane == tj) fv += dk;
                                    touched |= 1u << tj;
                                }
                            }
                            w ^= 1u << l;
                            gdirty = true;
                            if (lane == k) wg = w;
                            if (GROUPS != GK_NONE) {
                                const int gl = __shfl_sync(FULL_MASK, g, l);
                                if (gl >= 0) {
                                    const long long al = __shfl_sync(FULL_MASK, a, l);
                                    __syncwarp();
                                    if (lane == 0) Mw[gl] -= 2 * al * (up_l ? 1 : -1);
                                    __syncwarp();
                                    touched |= __ballot_sync(FULL_MASK, g == gl);
                                }
                            }
                            if ((touched >> lane) & 1u) pvalid = false;
                            dE = flip_cost(w);
                            cand = !(dE >= thr);
                            pend = __ballot_sync(FULL_MASK, cand) & ~((2u << l) - 1u);
                        }
                    }
                    __syncwarp();  // order this chunk's reductions before later loads of the same addresses
                }
                if ((k == 31 || c == nch - 1) && gdirty) __stcg(spw + (c & ~31) + lane, wg);
            }
            st.chunks += (unsigned long long)nch;
        }
    }
    __syncwarp();

    // ---- results: +-1 bytes back into the caller's row, packed transposed copy for the energy kernel
    for (int c = 0; c < nch; ++c) {
        const int v = c * 32 + lane;
        const uint32_t w = __ldcg(spw + c);
        if (v < n) state_row[v] = ((w >> lane) & 1u) ? 1 : -1;
    }
    for (int c = lane; c < nch; c += 32) D.packedT[(int64_t)c * D.rpad + r_local] = __ldcg(spw + c);
}

template <GroupKind GROUPS, Proposal PROP, bool RANDOM>
__global__ void __launch_bounds__(QA_TPB_MAX, 4) k_anneal_ref(AnnealParams P) {
    __shared__ long long Msh[GROUPS != GK_NONE ? (QA_TPB_MAX / 32) * QA_MAX_GROUPS : 1];
    __shared__ unsigned long long next_read[QA_TPB_MAX / 32];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int64_t slot = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
    double *f = P.f_scratch + slot * P.f_stride;
    uint32_t *spw = P.spw_scratch + slot * P.spw_stride;
    long long *Mw = GROUPS != GK_NONE ? (Msh + wib * QA_MAX_GROUPS) : Msh;
    WarpStats st = {0, 0, 0, 0, 0, 0, 0};

    if (P.seed_mode == QA_SEED_STREAM) {
        // one xorshift128+ stream across reads (neal num_reads=R): inherently serial, validation only
        if (slot != 0) return;
        unsigned long long s0 = P.seeds[0] ? P.seeds[0] : ~0ull, s1 = 0;
        for (int64_t r = P.read_begin; r < P.read_end; ++r) {
            const int p = (int)(r / P.reads_per_problem);
            const ProblemDesc D = P.descs[p];
            anneal_read<GROUPS, PROP, RANDOM>(D, P, r - D.read_base, f, spw, s0, s1, Mw, st, P.error_flag);
        }
    } else {
        for (;;) {
            if (lane == 0) next_read[wib] = P.read_begin + atomicAdd(P.counter, 1ull);
            __syncwarp();
            const int64_t r = (int64_t)next_read[wib];
            __syncwarp();
            if (r >= P.read_end) break;
            const int p = (int)(r / P.reads_per_problem);
            const ProblemDesc D = P.descs[p];
            const unsigned long long sd = P.seeds[r];
            unsigned long long s0 = sd ? sd : ~0ull, s1 = 0;  // neal: rng_state = {seed ? seed : RANDMAX, 0}
            anneal_read<GROUPS, PROP, RANDOM>(D, P, r - D.read_base, f, spw, s0, s1, Mw, st, P.error_flag);
        }
    }
    if (lane == 0) {
        atomicAdd(P.stats + ST_CAND, st.cand);
        atomicAdd(P.stats + ST_DRAWS, st.draws);
        atomicAdd(P.stats + ST_ACC, st.acc);
        atomicAdd(P.stats + ST_NBR, st.nbr);
        atomicAdd(P.stats + ST_ACTIVE, st.active);
        atomicAdd(P.stats + ST_CHUNKS, st.chunks);
        atomicAdd(P.stats + ST_TIES, st.ties);
    }
}

// EQ32 models run the 64-bit instance: this kernel has no 32-bit one
template <Proposal PROP, bool RANDOM>
void (*ref_instance(GroupKind gk))(AnnealParams) {
    return gk == GK_NONE ? k_anneal_ref<GK_NONE, PROP, RANDOM>
         : gk == GK_INTERVAL ? k_anneal_ref<GK_INTERVAL, PROP, RANDOM> : k_anneal_ref<GK_EQ64, PROP, RANDOM>;
}

void (*ref_kernel(GroupKind gk, Proposal prop, bool random_order))(AnnealParams) {
    if (random_order) return prop == PROP_GIBBS ? ref_instance<PROP_GIBBS, true>(gk) : ref_instance<PROP_METROPOLIS, true>(gk);
    return prop == PROP_GIBBS ? ref_instance<PROP_GIBBS, false>(gk) : ref_instance<PROP_METROPOLIS, false>(gk);
}

}  // namespace

namespace qa {

int ref_resident_reads(qa_ctx *ctx, int *out) {
    int bps = 0;
    QA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_anneal_ref<GK_NONE, PROP_METROPOLIS, false>, QA_TPB_MAX, 0));
    *out = bps * ctx->num_sms * (QA_TPB_MAX / 32);
    return QA_OK;
}

int launch_ref(Launch &L) {
    qa_ctx *ctx = L.ctx;
    AnnealParams &A = L.A;
    const int64_t total_reads = A.total_reads;
    void (*const fn)(AnnealParams) = ref_kernel(L.gk, L.prop, L.random_order);
    const bool stream = A.seed_mode == QA_SEED_STREAM;
    // launch geometry: persistent grid, one warp per resident read
    int wpb = QA_TPB_MAX / 32;
    if (stream) wpb = 1;
    else if (total_reads < (int64_t)ctx->num_sms * wpb) wpb = (int)std::max<int64_t>(1, (total_reads + ctx->num_sms - 1) / ctx->num_sms);
    const int tpb = wpb * 32;
    int bps = 0;
    QA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, fn, tpb, 0));
    if (bps < 1) return fail(QA_ERR_CUDA, "annealing kernel does not fit on an SM");
    int64_t grid = (int64_t)bps * ctx->num_sms;  // multiple of the SM count
    const int64_t need = (total_reads + wpb - 1) / wpb;
    if (need < grid) grid = need;
    if (stream) grid = 1;
    const int64_t slots = grid * wpb;
    const int64_t f_stride = (int64_t)L.M->nch_max * 32;
    const int64_t spw_stride = ((int64_t)L.M->nch_max + 31) & ~31ll;
    int rc = ensure(ctx->f, (size_t)slots * f_stride * sizeof(double));
    if (!rc) rc = ensure(ctx->spw, (size_t)slots * spw_stride * sizeof(uint32_t));
    if (rc) return rc;
    A.f_scratch = (double *)ctx->f.p;
    A.spw_scratch = (uint32_t *)ctx->spw.p;
    A.f_stride = f_stride;
    A.spw_stride = spw_stride;

    // without an interrupt callback the whole job is one launch; with one, read waves of `slots` reads
    const int64_t wave = (L.interrupt && !stream) ? slots : total_reads;
    QA_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    while (L.done < total_reads) {
        A.read_begin = L.done;
        A.read_end = std::min(total_reads, L.done + wave);
        QA_CUDA(cudaMemsetAsync(A.counter, 0, sizeof(unsigned long long), ctx->stream));
        fn<<<(unsigned)grid, tpb, 0, ctx->stream>>>(A);
        QA_CUDA(cudaGetLastError());
        ctx->launches++;
        if (L.st) L.st->anneal_launches++;
        L.done = A.read_end;
        if (L.interrupt && L.done < total_reads) {
            QA_CUDA(cudaStreamSynchronize(ctx->stream));
            if (L.interrupt(L.iuser)) { L.interrupted = true; break; }
        }
    }
    return QA_OK;
}

}  // namespace qa
