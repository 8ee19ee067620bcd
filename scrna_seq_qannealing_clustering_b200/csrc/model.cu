// model.cu -- qa_model: neal's vectors on the device, the adjacency in neal's push_back order (stable radix sort by vertex),
// rank-1 groups.  (neal general_simulated_annealing builds its adjacency lists by appending every coupler to both endpoints in
// coupler order; SURVEY.md row a11.)
#include "common.cuh"

#include <cub/device/device_radix_sort.cuh>

using namespace qa;

#include "adjacency.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// adjacency construction on the device, preserving neal's push_back order (stable sort by vertex)
// ------------------------------------------------------------------------------------------------
__global__ void k_make_entries(int64_t m_total, int32_t num_problems, const int64_t *var_off, const int64_t *cpl_off,
                               const int32_t *starts, const int32_t *ends, uint32_t *keys, uint32_t *vals, int *error_flag) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m_total) return;
    // problem of coupler c (binary search in coupler offsets)
    int lo = 0, hi = num_problems;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (cpl_off[mid] <= c) lo = mid; else hi = mid;
    }
    const int64_t vbase = var_off[lo];
    const int64_t np = var_off[lo + 1] - vbase;
    const int u = starts[c], v = ends[c];
    if (u < 0 || v < 0 || u >= np || v >= np || u == v) {
        atomicExch(error_flag, QA_ERR_INDEX);
        keys[2 * c] = keys[2 * c + 1] = 0;
        vals[2 * c] = (uint32_t)(2 * c);
        vals[2 * c + 1] = (uint32_t)(2 * c + 1);
        return;
    }
    keys[2 * c] = (uint32_t)(vbase + u);      // entry 2c   : row u, neighbour v
    keys[2 * c + 1] = (uint32_t)(vbase + v);  // entry 2c+1 : row v, neighbour u
    vals[2 * c] = (uint32_t)(2 * c);
    vals[2 * c + 1] = (uint32_t)(2 * c + 1);
}

__global__ void k_fill_csr(int64_t entries, const uint32_t *sorted_vals, const int32_t *starts, const int32_t *ends,
                           const double *w, int32_t *col, double *val) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= entries) return;
    const uint32_t e = sorted_vals[i];
    const int64_t c = e >> 1;
    col[i] = (e & 1u) ? starts[c] : ends[c];
    val[i] = w[c];
}


// build CSR (all problems at once) from the device COO already stored in the model
int build_adjacency(qa_model *M) {
    qa_ctx *ctx = M->ctx;
    const int64_t m = M->m_total;
    const int64_t entries = 2 * m;
    const int64_t rows_alloc = M->n_total + 64 + 1;  // padding rows read by the last chunk of the last problem
    if (entries >= (int64_t)0x7fffffff) return fail(QA_ERR_LIMIT, "more than 2^30 couplers: use a structured (group) model");
    if (M->n_total >= (int64_t)0x7fffffff) return fail(QA_ERR_LIMIT, "too many variables");
    QA_CUDA(cudaMalloc((void **)&M->rowptr, rows_alloc * sizeof(int32_t)));
    QA_CUDA(cudaMalloc((void **)&M->col, std::max<int64_t>(entries, 1) * sizeof(int32_t)));
    QA_CUDA(cudaMalloc((void **)&M->val, std::max<int64_t>(entries, 1) * sizeof(double)));
    QA_CUDA(cudaMemsetAsync(ctx->d_flag, 0, 2 * sizeof(int), ctx->stream));
    int64_t *d_off = nullptr;
    const int P = M->num_problems;
    QA_CUDA(cudaMalloc((void **)&d_off, 2 * (P + 1) * sizeof(int64_t)));
    QA_CUDA(cudaMemcpyAsync(d_off, M->var_off.data(), (P + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(d_off + P + 1, M->cpl_off.data(), (P + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    uint32_t *keys = nullptr, *vals = nullptr, *keys2 = nullptr, *vals2 = nullptr;
    int rc = QA_OK;
    if (entries > 0) {
        int rc2 = ensure(ctx->misc, (size_t)entries * 4 * sizeof(uint32_t));
        if (rc2) { cudaFree(d_off); return rc2; }
        keys = (uint32_t *)ctx->misc.p;
        vals = keys + entries;
        keys2 = vals + entries;
        vals2 = keys2 + entries;
        const int tpb = 256;
        k_make_entries<<<(unsigned)((m + tpb - 1) / tpb), tpb, 0, ctx->stream>>>(m, P, d_off, d_off + P + 1, M->starts, M->ends,
                                                                                 keys, vals, ctx->d_flag);
        ctx->launches++;
        int end_bit = 1;
        while (((int64_t)1 << end_bit) < M->n_total + 1 && end_bit < 32) ++end_bit;
        size_t tmp_bytes = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys, keys2, vals, vals2, (int)entries, 0, end_bit, ctx->stream);
        rc2 = ensure(ctx->cubtmp, tmp_bytes);
        if (rc2) { cudaFree(d_off); return rc2; }
        cudaError_t ce = cub::DeviceRadixSort::SortPairs(ctx->cubtmp.p, tmp_bytes, keys, keys2, vals, vals2, (int)entries, 0,
                                                         end_bit, ctx->stream);
        if (ce != cudaSuccess) { cudaFree(d_off); return fail(QA_ERR_CUDA, std::string("radix sort: ") + cudaGetErrorString(ce)); }
        ctx->launches += 4;
        k_fill_csr<<<(unsigned)((entries + tpb - 1) / tpb), tpb, 0, ctx->stream>>>(entries, vals2, M->starts, M->ends, M->w, M->col, M->val);
        ctx->launches++;
    } else {
        int rc2 = ensure(ctx->misc, 256);
        if (rc2) { cudaFree(d_off); return rc2; }
        keys2 = (uint32_t *)ctx->misc.p;
    }
    {
        const int tpb = 256;
        k_rowptr<<<(unsigned)((rows_alloc + tpb - 1) / tpb), tpb, 0, ctx->stream>>>(rows_alloc, entries, keys2, M->rowptr, ctx->d_flag + 1);
        ctx->launches++;
    }
    int flags[2] = {0, 0};
    cudaError_t ce = cudaMemcpyAsync(flags, ctx->d_flag, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_off);
    if (ce != cudaSuccess) return fail(QA_ERR_CUDA, std::string("adjacency build: ") + cudaGetErrorString(ce));
    if (flags[0] != 0) return fail(QA_ERR_INDEX, "coupler index out of range or self-loop");
    M->max_deg = flags[1];
    return rc;
}

}  // namespace

namespace qa {

int finalize_descs(qa_model *M) {
    const int P = M->num_problems;
    M->descs.assign(P, ProblemDesc());
    M->n_max = 0;
    for (int p = 0; p < P; ++p) {
        ProblemDesc &D = M->descs[p];
        const int64_t v0 = M->var_off[p], c0 = M->cpl_off[p];
        D.n = (int32_t)(M->var_off[p + 1] - v0);
        D.nch = (D.n + 31) / 32;
        D.ngroups = 0;
        D.m = M->cpl_off[p + 1] - c0;
        D.rowptr = M->rowptr + v0;
        D.col = M->col;   // rowptr holds global entry positions
        D.val = M->val;
        D.h = M->h + v0;
        D.starts = M->starts + c0;
        D.ends = M->ends + c0;
        D.w = M->w + c0;
        D.grp = nullptr; D.coef = nullptr; D.lambda = nullptr; D.kappa = nullptr;
        D.bw_ptr = nullptr; D.bw_words = nullptr; D.ent_slot = nullptr;
        D.rp_slabs = nullptr; D.rp_off = nullptr; D.rp_nslabs = 0;
        D.betas = nullptr;
        M->n_max = std::max(M->n_max, D.n);
    }
    M->nch_max = (M->n_max + 31) / 32;
    if (!M->d_descs) QA_CUDA(cudaMalloc((void **)&M->d_descs, P * sizeof(ProblemDesc)));
    return QA_OK;
}

int model_create(qa_ctx *ctx, int32_t P, const int64_t *var_off, const int64_t *cpl_off, const double *h,
                 const int32_t *starts, const int32_t *ends, const double *w, qa_model **out) {
    qa_model *M = new qa_model();
    M->ctx = ctx;
    M->num_problems = P;
    M->var_off.assign(var_off, var_off + P + 1);
    M->cpl_off.assign(cpl_off, cpl_off + P + 1);
    M->n_total = var_off[P];
    M->m_total = cpl_off[P];
    int rc = upload(ctx, &M->h, h, (size_t)M->n_total);
    if (!rc) rc = upload(ctx, &M->starts, starts, (size_t)M->m_total);
    if (!rc) rc = upload(ctx, &M->ends, ends, (size_t)M->m_total);
    if (!rc) rc = upload(ctx, &M->w, w, (size_t)M->m_total);
    if (!rc) rc = build_adjacency(M);
    if (!rc) rc = finalize_descs(M);
    if (rc) {
        qa_model_destroy(M);
        return rc;
    }
    *out = M;
    return QA_OK;
}

}  // namespace qa

extern "C" {

int qa_model_from_ising(qa_ctx *ctx, int32_t n, const double *h, int64_t m, const int32_t *starts, const int32_t *ends,
                        const double *weights, qa_model **out) {
    if (!ctx || !out) return fail(QA_ERR_ARG, "null context or out");
    *out = nullptr;
    if (n < 0 || m < 0) return fail(QA_ERR_ARG, "negative size");
    if ((n > 0 && !h) || (m > 0 && (!starts || !ends || !weights))) return fail(QA_ERR_ARG, "null model vector");
    QA_CUDA(cudaSetDevice(ctx->device));
    const int64_t voff[2] = {0, n}, coff[2] = {0, m};
    return model_create(ctx, 1, voff, coff, h, starts, ends, weights, out);
}

int qa_model_set_groups(qa_model *M, int32_t ngroups, const int32_t *grp, const int32_t *coef, const double *lambda,
                        const int64_t *kappa) {
    if (!M) return fail(QA_ERR_ARG, "null model");
    if (M->num_problems != 1) return fail(QA_ERR_ARG, "groups need a single-problem model");
    if (ngroups < 0 || ngroups > QA_MAX_GROUPS) return fail(QA_ERR_LIMIT, "ngroups must be in [0, QA_MAX_GROUPS]");
    qa_ctx *ctx = M->ctx;
    QA_CUDA(cudaSetDevice(ctx->device));
    if (M->grp) { cudaFree(M->grp); M->grp = nullptr; }
    if (M->coef) { cudaFree(M->coef); M->coef = nullptr; }
    if (M->lambda) { cudaFree(M->lambda); M->lambda = nullptr; }
    if (M->kappa) { cudaFree(M->kappa); M->kappa = nullptr; }
    M->gbounds = false;   // new groups are equality groups until bounds are set again
    M->gumin.clear();
    M->gumax.clear();
    M->ngroups = ngroups;
    if (ngroups > 0) M->dn_ok = false;   // the dense form carries no group terms
    if (M->rp_slabs) { cudaFree(M->rp_slabs); M->rp_slabs = nullptr; }   // the slabs carry the group metadata
    if (M->rp_off) { cudaFree(M->rp_off); M->rp_off = nullptr; }
    M->rp_built = false;
    M->rp_ok = false;
    M->descs[0].rp_slabs = nullptr;
    M->descs[0].rp_off = nullptr;
    ProblemDesc &D = M->descs[0];
    D.ngroups = ngroups;
    D.grp = nullptr; D.coef = nullptr; D.lambda = nullptr; D.kappa = nullptr;
    if (ngroups == 0) return QA_OK;
    if (!grp || !coef || !lambda || !kappa) return fail(QA_ERR_ARG, "null group vector");
    const int32_t n = D.n;
    const int64_t npad = (int64_t)D.nch * 32;
    // host-side validation: exact integer arithmetic must stay below 2^53 (and (M+kappa)^2 below 2^62)
    std::vector<int32_t> hg(npad, -1), hc(npad, 0);
    std::vector<int32_t> tg(n), tc(n);
    QA_CUDA(cudaMemcpy(tg.data(), grp, (size_t)n * sizeof(int32_t), cudaMemcpyDefault));
    QA_CUDA(cudaMemcpy(tc.data(), coef, (size_t)n * sizeof(int32_t), cudaMemcpyDefault));
    std::vector<int64_t> hk(ngroups);
    QA_CUDA(cudaMemcpy(hk.data(), kappa, (size_t)ngroups * sizeof(int64_t), cudaMemcpyDefault));
    std::vector<double> sumabs(ngroups, 0.0), maxa(ngroups, 0.0);
    for (int v = 0; v < n; ++v) {
        if (tg[v] >= ngroups) return fail(QA_ERR_ARG, "group index out of range");
        hg[v] = tg[v] < 0 ? -1 : tg[v];
        hc[v] = tc[v];
        if (tg[v] >= 0) {
            sumabs[tg[v]] += std::fabs((double)tc[v]);
            maxa[tg[v]] = std::max(maxa[tg[v]], std::fabs((double)tc[v]));
        }
    }
    M->groups_i32 = true;
    for (int g = 0; g < ngroups; ++g) {
        const double span = sumabs[g] + std::fabs((double)hk[g]);
        if (span >= 2147483648.0 || maxa[g] * (maxa[g] + span) >= 9007199254740992.0)
            return fail(QA_ERR_LIMIT, "group coefficients too large for exact integer evaluation");
        if (maxa[g] * (maxa[g] + span) >= 2147483648.0) M->groups_i32 = false;
    }
    QA_CUDA(cudaMalloc((void **)&M->grp, npad * sizeof(int32_t)));
    QA_CUDA(cudaMalloc((void **)&M->coef, npad * sizeof(int32_t)));
    QA_CUDA(cudaMalloc((void **)&M->lambda, ngroups * sizeof(double)));
    QA_CUDA(cudaMalloc((void **)&M->kappa, 3 * ngroups * sizeof(long long)));   // room for interval bounds behind kappa
    QA_CUDA(cudaMemcpy(M->grp, hg.data(), npad * sizeof(int32_t), cudaMemcpyHostToDevice));
    QA_CUDA(cudaMemcpy(M->coef, hc.data(), npad * sizeof(int32_t), cudaMemcpyHostToDevice));
    QA_CUDA(cudaMemcpy(M->lambda, lambda, ngroups * sizeof(double), cudaMemcpyDefault));
    QA_CUDA(cudaMemcpy(M->kappa, hk.data(), ngroups * sizeof(long long), cudaMemcpyHostToDevice));
    D.grp = M->grp; D.coef = M->coef; D.lambda = M->lambda; D.kappa = M->kappa;
    M->gumin.resize(ngroups);
    M->gumax.resize(ngroups);
    for (int g = 0; g < ngroups; ++g) {   // span < 2^31 above: exact
        M->gumin[g] = hk[g] - (int64_t)sumabs[g];
        M->gumax[g] = hk[g] + (int64_t)sumabs[g];
    }
    return QA_OK;
}

int qa_model_set_group_bounds(qa_model *M, const int64_t *lo, const int64_t *hi) {
    if (!M) return fail(QA_ERR_ARG, "null model");
    if (M->num_problems != 1) return fail(QA_ERR_ARG, "group bounds need a single-problem model");
    if ((lo == nullptr) != (hi == nullptr)) return fail(QA_ERR_ARG, "lo and hi must both be given or both be null");
    qa_ctx *ctx = M->ctx;
    QA_CUDA(cudaSetDevice(ctx->device));
    const int G = M->ngroups;
    if (lo && G == 0) return fail(QA_ERR_ARG, "no groups: call qa_model_set_groups first");
    std::vector<long long> hl(G), hh(G);
    if (lo) {
        QA_CUDA(cudaMemcpy(hl.data(), lo, (size_t)G * sizeof(int64_t), cudaMemcpyDefault));
        QA_CUDA(cudaMemcpy(hh.data(), hi, (size_t)G * sizeof(int64_t), cudaMemcpyDefault));
        for (int g = 0; g < G; ++g) {
            if (hl[g] > hh[g]) return fail(QA_ERR_ARG, "group bound lo > hi");
            // u stays in [umin, umax]: a bound beyond that range never binds, so clamping it leaves d(u) unchanged there
            hl[g] = std::max<long long>(hl[g], M->gumin[g]);
            hh[g] = std::min<long long>(hh[g], M->gumax[g]);
            const __int128 dmax = std::max<__int128>(std::max<__int128>((__int128)hl[g] - M->gumin[g], (__int128)M->gumax[g] - hh[g]), 0);
            if (dmax * dmax >= ((__int128)1 << 53)) return fail(QA_ERR_LIMIT, "group bounds too far from the reachable range for exact integer evaluation");
        }
    }
    if (M->rp_slabs) { cudaFree(M->rp_slabs); M->rp_slabs = nullptr; }
    if (M->rp_off) { cudaFree(M->rp_off); M->rp_off = nullptr; }
    M->rp_built = false;
    M->rp_ok = false;
    ProblemDesc &D = M->descs[0];
    D.rp_slabs = nullptr;
    D.rp_off = nullptr;
    M->gbounds = false;
    if (!lo) return QA_OK;
    QA_CUDA(cudaMemcpy(M->kappa + G, hl.data(), (size_t)G * sizeof(long long), cudaMemcpyHostToDevice));
    QA_CUDA(cudaMemcpy(M->kappa + 2 * G, hh.data(), (size_t)G * sizeof(long long), cudaMemcpyHostToDevice));
    M->gbounds = true;
    return QA_OK;
}

int qa_model_num_variables(const qa_model *M) { return M ? (int)M->n_total : fail(QA_ERR_ARG, "null model"); }
int64_t qa_model_num_couplers(const qa_model *M) { return M ? M->m_total : (int64_t)fail(QA_ERR_ARG, "null model"); }
int qa_model_max_degree(const qa_model *M) { return M ? M->max_deg : fail(QA_ERR_ARG, "null model"); }

int qa_model_get_ising(const qa_model *M, double *h, int32_t *starts, int32_t *ends, double *weights) {
    if (!M) return fail(QA_ERR_ARG, "null model");
    QA_CUDA(cudaSetDevice(M->ctx->device));
    if (h) QA_CUDA(cudaMemcpy(h, M->h, (size_t)M->n_total * sizeof(double), cudaMemcpyDefault));
    if (starts) QA_CUDA(cudaMemcpy(starts, M->starts, (size_t)M->m_total * sizeof(int32_t), cudaMemcpyDefault));
    if (ends) QA_CUDA(cudaMemcpy(ends, M->ends, (size_t)M->m_total * sizeof(int32_t), cudaMemcpyDefault));
    if (weights) QA_CUDA(cudaMemcpy(weights, M->w, (size_t)M->m_total * sizeof(double), cudaMemcpyDefault));
    return QA_OK;
}

int qa_model_destroy(qa_model *M) {
    if (!M) return QA_OK;
    cudaSetDevice(M->ctx->device);
    cudaStreamSynchronize(M->ctx->stream);
    void *ptrs[] = {M->h, M->starts, M->ends, M->w, M->rowptr, M->col, M->val, M->grp, M->coef, M->lambda, M->kappa, M->d_descs,
                    M->bw_ptr, M->bw_words, M->ent_slot, M->rp_slabs, M->rp_off, M->dn_W};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete M;
    return QA_OK;
}

}  // extern "C"
