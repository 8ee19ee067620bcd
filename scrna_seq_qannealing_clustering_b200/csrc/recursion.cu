// recursion.cu -- device side of the recursive bipartition driver (SURVEY.md 8(f) rank 1; reference: the recursion of
// clustering_bqm / clustering_bqm_2, Python_Functions/BQM_clustering.py:113-203, 302-350, which calls itself on
// G.subgraph(S0) and G.subgraph(S1)).
//
//   qa_graph_split            G.subgraph(part) for EVERY part of a node partition at once, on the device: child edge lists in the
//                             parent's edge order with nodes relabelled by their rank inside the part (networkx keeps the
//                             parent's node order), plus the parent node of every child node -- no host / networkx round trip.
//   qa_model_concat           single-problem models (each built by a qa_build_* entry point, rank-1 groups included) -> ONE
//                             batched model, so that all sub-graphs of a recursion level anneal in one launch.
//   qa_sa_sample_model_batch  the batched launch on a resident model, optionally with one beta schedule PER PROBLEM (each
//                             sub-graph gets the default range of its own model, as separate sampler calls would).

#include "common.cuh"

#include <cub/device/device_radix_sort.cuh>

using namespace qa;

namespace {

// key of node v: its part, or num_parts when it is dropped
__global__ void k_split_node_keys(int32_t n, int32_t num_parts, const int32_t *part, uint32_t *keys, uint32_t *vals, int32_t *count,
                                  int *error_flag) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    int p = part[v];
    if (p >= num_parts) { atomicExch(error_flag, QA_ERR_INDEX); p = -1; }
    keys[v] = p < 0 ? (uint32_t)num_parts : (uint32_t)p;
    vals[v] = (uint32_t)v;
    if (p >= 0) atomicAdd(count + p, 1);
}

// sorted position -> local index of the node inside its part
__global__ void k_split_local(int32_t n, int32_t num_parts, const uint32_t *skeys, const uint32_t *svals, const int64_t *node_off,
                              int32_t *local, int32_t *node_ids) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint32_t p = skeys[t];
    const int v = (int)svals[t];
    if (p >= (uint32_t)num_parts) { local[v] = -1; return; }
    local[v] = (int32_t)(t - node_off[p]);   // dropped nodes sort last, so t is also the node's position in node_ids
    node_ids[t] = v;
}

__global__ void k_split_edge_keys(int64_t m, int32_t n, int32_t num_parts, const int32_t *eu, const int32_t *ev, const int32_t *part,
                                  uint32_t *keys, uint32_t *vals, int32_t *count, int *error_flag) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int u = eu[e], v = ev[e];
    uint32_t key = (uint32_t)num_parts;
    if (u < 0 || v < 0 || u >= n || v >= n) atomicExch(error_flag, QA_ERR_INDEX);
    else if (part[u] >= 0 && part[u] < num_parts && part[u] == part[v]) key = (uint32_t)part[u];
    keys[e] = key;
    vals[e] = (uint32_t)e;
    if (key < (uint32_t)num_parts) atomicAdd(count + key, 1);
}

__global__ void k_split_emit(int64_t kept, const uint32_t *svals, const int32_t *eu, const int32_t *ev, const double *w,
                             const int32_t *local, int32_t *ou, int32_t *ov, double *ow) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= kept) return;
    const uint32_t e = svals[t];
    ou[t] = local[eu[e]];
    ov[t] = local[ev[e]];
    ow[t] = w[e];
}

__global__ void k_copy_shift_i32(int64_t count, const int32_t *src, int32_t add, int32_t *dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) dst[i] = src[i] + add;
}

__global__ void k_fill_i32(int64_t count, int32_t value, int32_t *dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) dst[i] = value;
}

int stable_sort_pairs(qa_ctx *ctx, int64_t count, int32_t max_key, uint32_t *keys, uint32_t *keys2, uint32_t *vals, uint32_t *vals2) {
    int end_bit = 1;
    while (((int64_t)1 << end_bit) < (int64_t)max_key + 1 && end_bit < 32) ++end_bit;
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, keys, keys2, vals, vals2, (int)count, 0, end_bit, ctx->stream);
    int rc = ensure(ctx->cubtmp, tmp);
    if (rc) return rc;
    cudaError_t ce = cub::DeviceRadixSort::SortPairs(ctx->cubtmp.p, tmp, keys, keys2, vals, vals2, (int)count, 0, end_bit, ctx->stream);
    if (ce != cudaSuccess) return fail(QA_ERR_CUDA, std::string("radix sort: ") + cudaGetErrorString(ce));
    ctx->launches += 4;
    return QA_OK;
}

}  // namespace

extern "C" {

int qa_graph_split(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w, const int32_t *part,
                   int32_t num_parts, qa_graph **out) {
    if (!ctx || !out) return fail(QA_ERR_ARG, "null argument");
    *out = nullptr;
    if (n < 0 || m < 0 || num_parts < 1) return fail(QA_ERR_ARG, "bad sizes");
    if ((n > 0 && !part) || (m > 0 && (!eu || !ev || !w))) return fail(QA_ERR_ARG, "null graph or partition");
    if (m >= (int64_t)0x7fffffff) return fail(QA_ERR_LIMIT, "too many edges");
    QA_CUDA(cudaSetDevice(ctx->device));
    qa_graph *G = new qa_graph();
    G->ctx = ctx;
    G->num_problems = num_parts;
    G->point_off.assign(num_parts + 1, 0);
    G->edge_off.assign(num_parts + 1, 0);
    SnnScratch sc;
    auto bail = [&](int code) { qa_graph_destroy(G); return code; };
#define SPLIT_CUDA(call)                                                                                              \
    do {                                                                                                              \
        cudaError_t e__ = (call);                                                                                     \
        if (e__ != cudaSuccess) return bail(fail(QA_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__))); \
    } while (0)
    const int tpb = 256;
    auto blocks = [&](int64_t c) { return (unsigned)std::max<int64_t>(1, (c + tpb - 1) / tpb); };
    // inputs on the device
    int32_t *d_part = nullptr, *d_eu = nullptr, *d_ev = nullptr;
    double *d_w = nullptr;
    const int32_t *ppart = part, *peu = eu, *pev = ev;
    const double *pw = w;
    if (n > 0 && !is_device_ptr(part)) {
        SPLIT_CUDA(sc.get(&d_part, (size_t)n));
        SPLIT_CUDA(cudaMemcpyAsync(d_part, part, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        ppart = d_part;
    }
    if (m > 0 && !is_device_ptr(eu)) {
        SPLIT_CUDA(sc.get(&d_eu, (size_t)m));
        SPLIT_CUDA(cudaMemcpyAsync(d_eu, eu, (size_t)m * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        peu = d_eu;
    }
    if (m > 0 && !is_device_ptr(ev)) {
        SPLIT_CUDA(sc.get(&d_ev, (size_t)m));
        SPLIT_CUDA(cudaMemcpyAsync(d_ev, ev, (size_t)m * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        pev = d_ev;
    }
    if (m > 0 && !is_device_ptr(w)) {
        SPLIT_CUDA(sc.get(&d_w, (size_t)m));
        SPLIT_CUDA(cudaMemcpyAsync(d_w, w, (size_t)m * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        pw = d_w;
    }
    const int64_t cnt = std::max<int64_t>(std::max<int64_t>(n, m), 1);
    uint32_t *keys = nullptr, *keys2 = nullptr, *vals = nullptr, *vals2 = nullptr;
    int32_t *ncount = nullptr, *ecount = nullptr, *local = nullptr;
    int64_t *node_off = nullptr;
    SPLIT_CUDA(sc.get(&keys, (size_t)cnt));
    SPLIT_CUDA(sc.get(&keys2, (size_t)cnt));
    SPLIT_CUDA(sc.get(&vals, (size_t)cnt));
    SPLIT_CUDA(sc.get(&vals2, (size_t)cnt));
    SPLIT_CUDA(sc.get(&ncount, (size_t)num_parts));
    SPLIT_CUDA(sc.get(&ecount, (size_t)num_parts));
    SPLIT_CUDA(sc.get(&local, (size_t)std::max(n, 1)));
    SPLIT_CUDA(sc.get(&node_off, (size_t)num_parts + 1));
    SPLIT_CUDA(cudaMemsetAsync(ncount, 0, (size_t)num_parts * sizeof(int32_t), ctx->stream));
    SPLIT_CUDA(cudaMemsetAsync(ecount, 0, (size_t)num_parts * sizeof(int32_t), ctx->stream));
    SPLIT_CUDA(cudaMemsetAsync(ctx->d_flag, 0, 2 * sizeof(int), ctx->stream));
    int rc = QA_OK;
    // nodes: stable sort by part keeps the parent's node order inside every part
    std::vector<int32_t> hn(num_parts, 0), he(num_parts, 0);
    if (n > 0) {
        k_split_node_keys<<<blocks(n), tpb, 0, ctx->stream>>>(n, num_parts, ppart, keys, vals, ncount, ctx->d_flag);
        if ((rc = stable_sort_pairs(ctx, n, num_parts, keys, keys2, vals, vals2))) return bail(rc);
        SPLIT_CUDA(cudaMemcpyAsync(hn.data(), ncount, (size_t)num_parts * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SPLIT_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    for (int p = 0; p < num_parts; ++p) G->point_off[p + 1] = G->point_off[p] + hn[p];
    const int64_t kept_nodes = G->point_off[num_parts];
    SPLIT_CUDA(cudaMemcpyAsync(node_off, G->point_off.data(), ((size_t)num_parts + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    SPLIT_CUDA(cudaMalloc((void **)&G->node_ids, std::max<size_t>((size_t)kept_nodes, 1) * sizeof(int32_t)));
    if (n > 0) {
        k_split_local<<<blocks(n), tpb, 0, ctx->stream>>>(n, num_parts, keys2, vals2, node_off, local, G->node_ids);
        ctx->launches += 2;
    }
    // edges: kept when both ends lie in the same part; stable sort by part keeps the parent's edge order
    if (m > 0) {
        k_split_edge_keys<<<blocks(m), tpb, 0, ctx->stream>>>(m, n, num_parts, peu, pev, ppart, keys, vals, ecount, ctx->d_flag);
        if ((rc = stable_sort_pairs(ctx, m, num_parts, keys, keys2, vals, vals2))) return bail(rc);
        SPLIT_CUDA(cudaMemcpyAsync(he.data(), ecount, (size_t)num_parts * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
    int flag = 0;
    SPLIT_CUDA(cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SPLIT_CUDA(cudaStreamSynchronize(ctx->stream));
    if (flag != 0) return bail(fail(QA_ERR_INDEX, "edge endpoint or part index out of range"));
    for (int p = 0; p < num_parts; ++p) G->edge_off[p + 1] = G->edge_off[p] + he[p];
    const int64_t kept = G->edge_off[num_parts];
    SPLIT_CUDA(cudaMalloc((void **)&G->eu, std::max<size_t>((size_t)kept, 1) * sizeof(int32_t)));
    SPLIT_CUDA(cudaMalloc((void **)&G->ev, std::max<size_t>((size_t)kept, 1) * sizeof(int32_t)));
    SPLIT_CUDA(cudaMalloc((void **)&G->w, std::max<size_t>((size_t)kept, 1) * sizeof(double)));
    if (kept > 0) {
        k_split_emit<<<blocks(kept), tpb, 0, ctx->stream>>>(kept, vals2, peu, pev, pw, local, G->eu, G->ev, G->w);
        ctx->launches += 2;
    }
    SPLIT_CUDA(cudaStreamSynchronize(ctx->stream));
#undef SPLIT_CUDA
    *out = G;
    return QA_OK;
}

int qa_graph_get_nodes(const qa_graph *g, int32_t problem, int32_t *node_ids_out) {
    if (!g || !node_ids_out) return fail(QA_ERR_ARG, "null argument");
    if (!g->node_ids) return fail(QA_ERR_ARG, "this graph was not made by qa_graph_split");
    if (problem >= g->num_problems) return fail(QA_ERR_ARG, "problem index out of range");
    const int64_t b = problem < 0 ? 0 : g->point_off[problem];
    const int64_t e = problem < 0 ? g->point_off[g->num_problems] : g->point_off[problem + 1];
    QA_CUDA(cudaSetDevice(g->ctx->device));
    if (e > b) QA_CUDA(cudaMemcpy(node_ids_out, g->node_ids + b, (size_t)(e - b) * sizeof(int32_t), cudaMemcpyDefault));
    return QA_OK;
}

int qa_model_concat(qa_ctx *ctx, int32_t num_models, qa_model *const *models, qa_model **out) {
    if (!ctx || !models || !out) return fail(QA_ERR_ARG, "null argument");
    *out = nullptr;
    if (num_models < 1) return fail(QA_ERR_ARG, "need at least one model");
    for (int p = 0; p < num_models; ++p) {
        if (!models[p] || models[p]->ctx != ctx) return fail(QA_ERR_ARG, "null model or model of another context");
        if (models[p]->num_problems != 1) return fail(QA_ERR_ARG, "only single-problem models can be concatenated");
    }
    QA_CUDA(cudaSetDevice(ctx->device));
    qa_model *M = new qa_model();
    M->ctx = ctx;
    M->num_problems = num_models;
    M->var_off.assign(num_models + 1, 0);
    M->cpl_off.assign(num_models + 1, 0);
    int64_t gpad = 0, gcount = 0;
    bool bounds = false;   // some input carries interval bounds: every problem with groups gets them (equality: lo = hi = 0)
    for (int p = 0; p < num_models; ++p) {
        bounds = bounds || models[p]->gbounds;
        M->var_off[p + 1] = M->var_off[p] + models[p]->n_total;
        M->cpl_off[p + 1] = M->cpl_off[p] + models[p]->m_total;
        M->max_deg = std::max(M->max_deg, models[p]->max_deg);
        M->ngroups = std::max(M->ngroups, models[p]->ngroups);
        gpad += (int64_t)models[p]->descs[0].nch * 32;   // group-free problems too: see the group copy below
        gcount += std::max(models[p]->ngroups, 0);
    }
    M->n_total = M->var_off[num_models];
    M->m_total = M->cpl_off[num_models];
    auto bail = [&](int code) { qa_model_destroy(M); return code; };
    if (2 * M->m_total >= (int64_t)0x7fffffff || M->n_total >= (int64_t)0x7fffffff) return bail(fail(QA_ERR_LIMIT, "batched model too large"));
#define CAT_CUDA(call)                                                                                                \
    do {                                                                                                              \
        cudaError_t e__ = (call);                                                                                     \
        if (e__ != cudaSuccess) return bail(fail(QA_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__))); \
    } while (0)
    const int64_t entries = 2 * M->m_total;
    const int64_t rows_alloc = M->n_total + 64 + 1;
    const size_t n1 = (size_t)std::max<int64_t>(M->n_total, 1), m1 = (size_t)std::max<int64_t>(M->m_total, 1), e1 = (size_t)std::max<int64_t>(entries, 1);
    CAT_CUDA(cudaMalloc((void **)&M->h, n1 * sizeof(double)));
    CAT_CUDA(cudaMalloc((void **)&M->starts, m1 * sizeof(int32_t)));
    CAT_CUDA(cudaMalloc((void **)&M->ends, m1 * sizeof(int32_t)));
    CAT_CUDA(cudaMalloc((void **)&M->w, m1 * sizeof(double)));
    CAT_CUDA(cudaMalloc((void **)&M->rowptr, (size_t)rows_alloc * sizeof(int32_t)));
    CAT_CUDA(cudaMalloc((void **)&M->col, e1 * sizeof(int32_t)));
    CAT_CUDA(cudaMalloc((void **)&M->val, e1 * sizeof(double)));
    if (M->ngroups > 0) {
        CAT_CUDA(cudaMalloc((void **)&M->grp, (size_t)std::max<int64_t>(gpad, 1) * sizeof(int32_t)));
        CAT_CUDA(cudaMalloc((void **)&M->coef, (size_t)std::max<int64_t>(gpad, 1) * sizeof(int32_t)));
        CAT_CUDA(cudaMalloc((void **)&M->lambda, (size_t)std::max<int64_t>(gcount, 1) * sizeof(double)));
        CAT_CUDA(cudaMalloc((void **)&M->kappa, (size_t)std::max<int64_t>(gcount, 1) * (bounds ? 3 : 1) * sizeof(long long)));
        M->gbounds = bounds;
    }
    const int tpb = 256;
    auto blocks = [&](int64_t c) { return (unsigned)std::max<int64_t>(1, (c + tpb - 1) / tpb); };
    for (int p = 0; p < num_models; ++p) {
        const qa_model *S = models[p];
        const int64_t v0 = M->var_off[p], c0 = M->cpl_off[p];
        const size_t nv = (size_t)S->n_total, nc = (size_t)S->m_total;
        if (nv) CAT_CUDA(cudaMemcpyAsync(M->h + v0, S->h, nv * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        if (nc) {
            CAT_CUDA(cudaMemcpyAsync(M->starts + c0, S->starts, nc * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
            CAT_CUDA(cudaMemcpyAsync(M->ends + c0, S->ends, nc * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
            CAT_CUDA(cudaMemcpyAsync(M->w + c0, S->w, nc * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
            CAT_CUDA(cudaMemcpyAsync(M->col + 2 * c0, S->col, 2 * nc * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
            CAT_CUDA(cudaMemcpyAsync(M->val + 2 * c0, S->val, 2 * nc * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        }
        // row pointers hold global entry positions: this problem's rows start at entry 2 * c0
        if (nv) k_copy_shift_i32<<<blocks((int64_t)nv), tpb, 0, ctx->stream>>>((int64_t)nv, S->rowptr, (int32_t)(2 * c0), M->rowptr + v0);
    }
    k_fill_i32<<<blocks(rows_alloc - M->n_total), tpb, 0, ctx->stream>>>(rows_alloc - M->n_total, (int32_t)entries, M->rowptr + M->n_total);
    ctx->launches += (uint32_t)num_models + 1;
    int rc = finalize_descs(M);
    if (rc) return bail(rc);
    int64_t go = 0, gl = 0;
    for (int p = 0; p < num_models && M->ngroups > 0; ++p) {
        const qa_model *S = models[p];
        const int64_t npad = (int64_t)S->descs[0].nch * 32;
        ProblemDesc &D = M->descs[p];
        if (S->ngroups <= 0) {
            // the group kernels read grp[v] of every problem of the batch: a group-free problem gets grp = -1 everywhere
            // (ngroups stays 0, so lambda / kappa are never read)
            k_fill_i32<<<blocks(npad), tpb, 0, ctx->stream>>>(npad, -1, M->grp + go);
            CAT_CUDA(cudaGetLastError());
            CAT_CUDA(cudaMemsetAsync(M->coef + go, 0, (size_t)npad * sizeof(int32_t), ctx->stream));
            ctx->launches++;
            D.grp = M->grp + go;
            D.coef = M->coef + go;
            go += npad;
            continue;
        }
        CAT_CUDA(cudaMemcpyAsync(M->grp + go, S->grp, (size_t)npad * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        CAT_CUDA(cudaMemcpyAsync(M->coef + go, S->coef, (size_t)npad * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        CAT_CUDA(cudaMemcpyAsync(M->lambda + gl, S->lambda, (size_t)S->ngroups * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        const int64_t gk = bounds ? 3 * gl : gl;   // interval bounds: {kappa, lo, hi} of every problem stay together
        CAT_CUDA(cudaMemcpyAsync(M->kappa + gk, S->kappa, (size_t)S->ngroups * sizeof(long long), cudaMemcpyDeviceToDevice, ctx->stream));
        if (bounds) {
            const size_t gb = 2 * (size_t)S->ngroups * sizeof(long long);
            if (S->gbounds) CAT_CUDA(cudaMemcpyAsync(M->kappa + gk + S->ngroups, S->kappa + S->ngroups, gb, cudaMemcpyDeviceToDevice, ctx->stream));
            else CAT_CUDA(cudaMemsetAsync(M->kappa + gk + S->ngroups, 0, gb, ctx->stream));   // equality groups: lo = hi = 0
        }
        D.ngroups = S->ngroups;
        D.grp = M->grp + go;
        D.coef = M->coef + go;
        D.lambda = M->lambda + gl;
        D.kappa = M->kappa + gk;
        go += npad;
        gl += S->ngroups;
    }
    CAT_CUDA(cudaStreamSynchronize(ctx->stream));
#undef CAT_CUDA
    *out = M;
    return QA_OK;
}

int qa_sa_sample_model_batch(qa_ctx *ctx, qa_model *model, int32_t reads_per_problem, int8_t *states_inout, double *energies_out,
                             int32_t num_betas, const double *beta_schedules, int32_t betas_per_problem, int32_t sweeps_per_beta,
                             const uint64_t *seeds, qa_stats *stats_out) {
    if (!ctx || !model) return fail(QA_ERR_ARG, "null context or model");
    ctx->betas_per_problem = betas_per_problem != 0;
    const int rc = sample_common(ctx, model, reads_per_problem, states_inout, energies_out, num_betas, beta_schedules, sweeps_per_beta,
                                 seeds, QA_SEED_PER_READ, QA_MODE_REFERENCE, nullptr, nullptr, stats_out);
    ctx->betas_per_problem = false;
    return rc;
}

}  // extern "C"
