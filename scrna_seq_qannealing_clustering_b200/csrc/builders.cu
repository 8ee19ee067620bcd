// builders.cu -- qa_build_*: the reference's Q-dict constructions (BQM_clustering.py:36-47, 228-236, DQM_clustering.py:29-43,
// CQM_clustering.py:30-48, QA_subsampling.py:26-35) followed by dimod's from_qubo / change_vartype(SPIN) / to_numpy_vectors, on
// the device, bit-identical to the host builders of models.py.
#include "common.cuh"

#include <cub/device/device_radix_sort.cuh>

using namespace qa;

#include "adjacency.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// model builders on the device (reference: the Python Q-dict loops of BQM_clustering.py:36-47, 228-236,
// DQM_clustering.py:29-43, CQM_clustering.py:30-48, QA_subsampling.py:26-35 followed by dimod's
// from_qubo / change_vartype(SPIN) / to_numpy_vectors).  Every floating-point accumulation keeps the order of the
// Python code: per-vertex sums run sequentially over the vertex's edges in G.edges order, h accumulates Q_ij/4 in
// ascending-neighbour order, so the vectors are bit-identical to models.py (tests/test_gpu_builders.py).
// ------------------------------------------------------------------------------------------------
__global__ void k_graph_entries(int64_t m, int32_t n, const int32_t *eu, const int32_t *ev, uint32_t *keys, uint32_t *vals,
                                int *error_flag) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int u = eu[e], v = ev[e];
    if (u < 0 || v < 0 || u >= n || v >= n || u == v) {
        atomicExch(error_flag, QA_ERR_INDEX);
        keys[2 * e] = keys[2 * e + 1] = 0;
    } else {
        keys[2 * e] = (uint32_t)u;
        keys[2 * e + 1] = (uint32_t)v;
    }
    vals[2 * e] = (uint32_t)(2 * e);
    vals[2 * e + 1] = (uint32_t)(2 * e + 1);
}

// out[v] = base + sum over v's edges, in edge order, of f(w_e):  mode 0: scale*w   1: scale*(1-w)   2: 1 (degree)
// mode 3: weight of the LAST edge touching v (base if isolated)  -- the `set_linear` overwrite of DQM_clustering.py:42-43
__global__ void k_vertex_accumulate(int32_t n, const int32_t *rowptr, const uint32_t *sorted_vals, const double *w, int mode,
                                    double scale, double base, double *out) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    double acc = mode == 3 ? base : 0.0;
    for (int i = rowptr[v]; i < rowptr[v + 1]; ++i) {
        const double we = w[sorted_vals[i] >> 1];
        if (mode == 0) acc += scale * we;
        else if (mode == 1) acc += scale * (1 - we);
        else if (mode == 2) acc += 1.0;
        else acc = we;
    }
    out[v] = (mode == 3) ? acc : acc + base;
}

__global__ void k_seq_sum(int64_t count, const double *x, double scale, double *out) {
    // deterministic left-to-right sum (python / numpy cumsum order); setup only
    if (blockIdx.x || threadIdx.x) return;
    double s = 0.0;
    for (int64_t i = 0; i < count; ++i) s += x[i] * scale;
    *out = s;
}

// QUBO couplers of the k-way models: K copies of every graph edge (same case) + the one-hot pairs of every cell
__global__ void k_kway_couplers(int64_t m, int32_t n, int32_t K, const int32_t *eu, const int32_t *ev, const double *w,
                                double edge_scale, double edge_pre, double edge_shift, double onehot_q, unsigned long long *keys,
                                double *q) {
    const int64_t npairs = (int64_t)K * (K - 1) / 2;
    const int64_t total = m * K + (int64_t)n * npairs;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    int64_t a, b;
    double val;
    if (t < m * K) {
        const int64_t e = t / K;
        const int p = (int)(t % K);
        a = (int64_t)eu[e] * K + p;
        b = (int64_t)ev[e] * K + p;
        val = (edge_pre + edge_scale * w[e]) + edge_shift;  // python: (2g - 2w) - 2g, or -2w - 2g, or -2w
    } else {
        const int64_t u = t - m * K;
        const int64_t i = u / npairs;
        int64_t pr = u % npairs;
        int ca = 0;
        while (pr >= K - 1 - ca) { pr -= K - 1 - ca; ++ca; }
        const int cb = ca + 1 + (int)pr;
        a = i * K + ca;
        b = i * K + cb;
        val = onehot_q;
    }
    const unsigned long long hi = (unsigned long long)max(a, b), lo = (unsigned long long)min(a, b);
    keys[t] = (hi << 32) | lo;
    q[t] = val;
}

__global__ void k_edge_couplers(int64_t m, const int32_t *eu, const int32_t *ev, const double *w, int mode, double scale,
                                unsigned long long *keys, double *q) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const unsigned long long hi = (unsigned long long)max(eu[e], ev[e]), lo = (unsigned long long)min(eu[e], ev[e]);
    keys[e] = (hi << 32) | lo;
    q[e] = mode == 0 ? scale * w[e] : scale * (1 - w[e]);
}

__global__ void k_split_keys(int64_t m, const unsigned long long *keys, const uint32_t *perm, const double *q, int32_t *r,
                             int32_t *c, double *J) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    r[i] = (int32_t)(keys[i] >> 32);
    c[i] = (int32_t)(keys[i] & 0xffffffffu);
    J[i] = q[perm[i]] / 4.0;  // dimod change_vartype(SPIN): J = Q_ij / 4
}

__global__ void k_kway_linear(int32_t n, int32_t K, int32_t nvar, const double *cell_lin, double shift, double *lin) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nvar) return;
    lin[v] = v < n * K ? cell_lin[v / K] + shift : 0.0;
}

// h_v = Q_vv/2 + sum over the row (ascending neighbour = coupler order) of Q_vj/4
__global__ void k_h_from_rows(int32_t n, const double *lin, const int32_t *rowptr, const double *val, double *h) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    double acc = lin[v] / 2.0;
    for (int e = rowptr[v]; e < rowptr[v + 1]; ++e) acc += val[e];
    h[v] = acc;
}

struct GraphDev {
    int32_t n = 0;
    int64_t m = 0;
    int32_t *eu = nullptr, *ev = nullptr;
    double *w = nullptr;
    int32_t *rowptr = nullptr;   // per-vertex edge lists, in G.edges order
    uint32_t *sorted = nullptr;  // entry ids 2e (u side) / 2e+1 (v side)
    void free_all() {
        void *ptrs[] = {eu, ev, w, rowptr, sorted};
        for (void *p : ptrs) if (p) cudaFree(p);
        eu = ev = nullptr; w = nullptr; rowptr = nullptr; sorted = nullptr;
    }
};

int graph_to_device(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w, GraphDev &g) {
    if (n < 0 || m < 0) return fail(QA_ERR_ARG, "negative graph size");
    if (m > 0 && (!eu || !ev || !w)) return fail(QA_ERR_ARG, "null edge list");
    if (2 * m >= (int64_t)0x7fffffff) return fail(QA_ERR_LIMIT, "too many edges");
    g.n = n;
    g.m = m;
    int rc = upload(ctx, &g.eu, eu, (size_t)m);
    if (!rc) rc = upload(ctx, &g.ev, ev, (size_t)m);
    if (!rc) rc = upload(ctx, &g.w, w, (size_t)m);
    if (rc) return rc;
    const int64_t entries = 2 * m;
    QA_CUDA(cudaMalloc((void **)&g.rowptr, (size_t)(n + 2) * sizeof(int32_t)));
    QA_CUDA(cudaMalloc((void **)&g.sorted, (size_t)std::max<int64_t>(entries, 1) * sizeof(uint32_t)));
    QA_CUDA(cudaMemsetAsync(ctx->d_flag, 0, 2 * sizeof(int), ctx->stream));
    rc = ensure(ctx->misc, (size_t)std::max<int64_t>(entries, 1) * 3 * sizeof(uint32_t));
    if (rc) return rc;
    uint32_t *keys = (uint32_t *)ctx->misc.p, *vals = keys + std::max<int64_t>(entries, 1), *keys2 = vals + std::max<int64_t>(entries, 1);
    if (entries > 0) {
        k_graph_entries<<<blocks_for(m), 256, 0, ctx->stream>>>(m, n, g.eu, g.ev, keys, vals, ctx->d_flag);
        int end_bit = 1;
        while (((int64_t)1 << end_bit) < (int64_t)n + 1 && end_bit < 32) ++end_bit;
        size_t tmp = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tmp, keys, keys2, vals, g.sorted, (int)entries, 0, end_bit, ctx->stream);
        rc = ensure(ctx->cubtmp, tmp);
        if (rc) return rc;
        cudaError_t ce = cub::DeviceRadixSort::SortPairs(ctx->cubtmp.p, tmp, keys, keys2, vals, g.sorted, (int)entries, 0, end_bit, ctx->stream);
        if (ce != cudaSuccess) return fail(QA_ERR_CUDA, std::string("radix sort: ") + cudaGetErrorString(ce));
        ctx->launches += 5;
    }
    k_rowptr<<<blocks_for(n + 1), 256, 0, ctx->stream>>>(n + 1, entries, keys2, g.rowptr, ctx->d_flag + 1);
    ctx->launches++;
    int flag = 0;
    QA_CUDA(cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    if (flag) return fail(QA_ERR_INDEX, "edge endpoint out of range or self-loop");
    return QA_OK;
}

int device_seq_sum(qa_ctx *ctx, int64_t count, const double *x, double scale, double *out_host) {
    k_seq_sum<<<1, 32, 0, ctx->stream>>>(count, x, scale, ctx->d_best_e);
    ctx->launches++;
    QA_CUDA(cudaMemcpyAsync(out_host, ctx->d_best_e, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    return QA_OK;
}

// QUBO (lin[nvar], couplers as (hi<<32|lo) keys with values q) -> resident Ising model in dimod's vector order.
// offset_out = sum_i lin_i/2 + sum_c q_c/4 in python's left-to-right order (bqm.qubo_to_ising_vectors).
int lower_qubo(qa_ctx *ctx, int32_t nvar, const double *d_lin, int64_t mq, unsigned long long *d_keys, const double *d_q,
               qa_model **out, double *offset_out) {
    if (mq >= (int64_t)0x3fffffff) return fail(QA_ERR_LIMIT, "too many couplers");
    unsigned long long *keys2 = nullptr;
    uint32_t *perm = nullptr, *perm2 = nullptr;
    int32_t *r = nullptr, *c = nullptr;
    double *J = nullptr;
    const size_t mm = (size_t)std::max<int64_t>(mq, 1);
    int rc = QA_OK;
    auto cleanup = [&]() {
        void *ptrs[] = {keys2, perm, perm2, r, c, J};
        for (void *p : ptrs) if (p) cudaFree(p);
    };
    do {
        if (cudaMalloc((void **)&keys2, mm * 8) != cudaSuccess || cudaMalloc((void **)&perm, mm * 4) != cudaSuccess ||
            cudaMalloc((void **)&perm2, mm * 4) != cudaSuccess || cudaMalloc((void **)&r, mm * 4) != cudaSuccess ||
            cudaMalloc((void **)&c, mm * 4) != cudaSuccess || cudaMalloc((void **)&J, mm * 8) != cudaSuccess) {
            rc = fail(QA_ERR_CUDA, "out of device memory in model builder");
            break;
        }
        if (mq > 0) {
            // identity permutation, then sort by (row = larger index, col = smaller index): dimod to_numpy_vectors order
            std::vector<uint32_t> iota(mq);
            for (int64_t i = 0; i < mq; ++i) iota[i] = (uint32_t)i;
            cudaMemcpyAsync(perm, iota.data(), mq * 4, cudaMemcpyHostToDevice, ctx->stream);
            size_t tmp = 0;
            cub::DeviceRadixSort::SortPairs(nullptr, tmp, d_keys, keys2, perm, perm2, (int)mq, 0, 64, ctx->stream);
            rc = ensure(ctx->cubtmp, tmp);
            if (rc) break;
            cudaError_t ce = cub::DeviceRadixSort::SortPairs(ctx->cubtmp.p, tmp, d_keys, keys2, perm, perm2, (int)mq, 0, 64, ctx->stream);
            if (ce != cudaSuccess) { rc = fail(QA_ERR_CUDA, std::string("radix sort: ") + cudaGetErrorString(ce)); break; }
            k_split_keys<<<blocks_for(mq), 256, 0, ctx->stream>>>(mq, keys2, perm2, d_q, r, c, J);
            cudaStreamSynchronize(ctx->stream);  // iota must outlive the copy
            ctx->launches += 9;
        }
        const int64_t voff[2] = {0, nvar}, coff[2] = {0, mq};
        qa_model *M = nullptr;
        rc = model_create(ctx, 1, voff, coff, d_lin, r, c, J, &M);
        if (rc) break;
        k_h_from_rows<<<blocks_for(nvar), 256, 0, ctx->stream>>>(nvar, d_lin, M->rowptr, M->val, M->h);
        ctx->launches++;
        double s1 = 0.0, s2 = 0.0;
        rc = device_seq_sum(ctx, nvar, d_lin, 0.5, &s1);
        if (!rc) rc = device_seq_sum(ctx, mq, J, 1.0, &s2);
        if (rc) { qa_model_destroy(M); break; }
        *offset_out = (0.0 + s1) + s2;
        *out = M;
    } while (0);
    cleanup();
    return rc;
}

std::vector<int> slack_coefficients_host(int64_t upper) {
    // binary-encoded slack spanning exactly 0..upper (dimod add_linear_inequality_constraint; models.slack_coefficients)
    std::vector<int> c;
    if (upper <= 0) return c;
    int nbits = 0;
    while (((int64_t)2 << nbits) <= upper) ++nbits;  // floor(log2(upper))
    for (int j = 0; j < nbits; ++j) c.push_back(1 << j);
    if (upper - ((int64_t)1 << nbits) >= 0) c.push_back((int)(upper - ((int64_t)1 << nbits) + 1));
    return c;
}

}  // namespace

extern "C" {

int qa_build_cut_balance(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w,
                         double gamma_factor, double k, qa_model **out, double *offset_out, double *gamma_out) {
    if (!ctx || !out || !offset_out) return fail(QA_ERR_ARG, "null argument");
    *out = nullptr;
    QA_CUDA(cudaSetDevice(ctx->device));
    GraphDev g;
    double *lin = nullptr, *q = nullptr;
    unsigned long long *keys = nullptr;
    int rc = graph_to_device(ctx, n, m, eu, ev, w, g);
    do {
        if (rc) break;
        const size_t mm = (size_t)std::max<int64_t>(m, 1);
        if (cudaMalloc((void **)&lin, (size_t)std::max(n, 1) * 8) != cudaSuccess || cudaMalloc((void **)&q, mm * 8) != cudaSuccess ||
            cudaMalloc((void **)&keys, mm * 8) != cudaSuccess) { rc = fail(QA_ERR_CUDA, "out of device memory"); break; }
        // W = G.size(weight) = (sum of weighted degrees) / 2, degrees summed in adjacency (edge) order
        double sumdeg = 0.0;
        k_vertex_accumulate<<<blocks_for(n), 256, 0, ctx->stream>>>(n, g.rowptr, g.sorted, g.w, 0, 1.0, 0.0, lin);
        rc = device_seq_sum(ctx, n, lin, 1.0, &sumdeg);
        if (rc) break;
        const double W = sumdeg / 2;
        const double gamma = gamma_factor * W / n;
        k_vertex_accumulate<<<blocks_for(n), 256, 0, ctx->stream>>>(n, g.rowptr, g.sorted, g.w, 0, k, 0.0, lin);
        k_edge_couplers<<<blocks_for(m), 256, 0, ctx->stream>>>(m, g.eu, g.ev, g.w, 0, k * -2, keys, q);
        ctx->launches += 3;
        double off = 0.0;
        qa_model *M = nullptr;
        rc = lower_qubo(ctx, n, lin, m, keys, q, &M, &off);
        if (rc) break;
        std::vector<int32_t> grp(n, 0), coef(n, 1);
        const double lam = gamma;
        const int64_t kap = 0;
        rc = qa_model_set_groups(M, 1, grp.data(), coef.data(), &lam, &kap);
        if (rc) { qa_model_destroy(M); break; }
        *offset_out = off - gamma * n * n / 4.0;
        if (gamma_out) *gamma_out = gamma;
        *out = M;
    } while (0);
    g.free_all();
    if (lin) cudaFree(lin);
    if (q) cudaFree(q);
    if (keys) cudaFree(keys);
    return rc;
}

// clustering_bqm_2 (BQM_clustering.py:210-236): Q_ii = k*d_i + gamma, Q_uv = -2*k*w on edges, gamma = (W/n)*gamma_factor.  Sparse.
int qa_build_cut_linear(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w,
                        double gamma_factor, double k, qa_model **out, double *offset_out, double *gamma_out) {
    if (!ctx || !out || !offset_out) return fail(QA_ERR_ARG, "null argument");
    *out = nullptr;
    QA_CUDA(cudaSetDevice(ctx->device));
    GraphDev g;
    double *lin = nullptr, *q = nullptr;
    unsigned long long *keys = nullptr;
    int rc = graph_to_device(ctx, n, m, eu, ev, w, g);
    do {
        if (rc) break;
        const size_t mm = (size_t)std::max<int64_t>(m, 1);
        if (cudaMalloc((void **)&lin, (size_t)std::max(n, 1) * 8) != cudaSuccess || cudaMalloc((void **)&q, mm * 8) != cudaSuccess ||
            cudaMalloc((void **)&keys, mm * 8) != cudaSuccess) { rc = fail(QA_ERR_CUDA, "out of device memory"); break; }
        double sumdeg = 0.0;
        k_vertex_accumulate<<<blocks_for(n), 256, 0, ctx->stream>>>(n, g.rowptr, g.sorted, g.w, 0, 1.0, 0.0, lin);
        rc = device_seq_sum(ctx, n, lin, 1.0, &sumdeg);
        if (rc) break;
        const double gamma = (sumdeg / 2 / n) * gamma_factor;          // python: (W / n) * gamma_factor
        k_vertex_accumulate<<<blocks_for(n), 256, 0, ctx->stream>>>(n, g.rowptr, g.sorted, g.w, 0, k, gamma, lin);   // k*d_i + gamma
        k_edge_couplers<<<blocks_for(m), 256, 0, ctx->stream>>>(m, g.eu, g.ev, g.w, 0, k * -2, keys, q);
        ctx->launches += 3;
        rc = lower_qubo(ctx, n, lin, m, keys, q, out, offset_out);
        if (!rc && gamma_out) *gamma_out = gamma;
    } while (0);
    g.free_all();
    if (lin) cudaFree(lin);
    if (q) cudaFree(q);
    if (keys) cudaFree(keys);
    return rc;
}

int qa_build_subsampling(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w, double gamma,
                         double P, qa_model **out, double *offset_out) {
    if (!ctx || !out || !offset_out) return fail(QA_ERR_ARG, "null argument");
    *out = nullptr;
    QA_CUDA(cudaSetDevice(ctx->device));
    GraphDev g;
    double *lin = nullptr, *q = nullptr;
    unsigned long long *keys = nullptr;
    int rc = graph_to_device(ctx, n, m, eu, ev, w, g);
    do {
        if (rc) break;
        const size_t mm = (size_t)std::max<int64_t>(m, 1);
        if (cudaMalloc((void **)&lin, (size_t)std::max(n, 1) * 8) != cudaSuccess || cudaMalloc((void **)&q, mm * 8) != cudaSuccess ||
            cudaMalloc((void **)&keys, mm * 8) != cudaSuccess) { rc = fail(QA_ERR_CUDA, "out of device memory"); break; }
        k_vertex_accumulate<<<blocks_for(n), 256, 0, ctx->stream>>>(n, g.rowptr, g.sorted, g.w, 1, -P, gamma, lin);
        k_edge_couplers<<<blocks_for(m), 256, 0, ctx->stream>>>(m, g.eu, g.ev, g.w, 1, P, keys, q);
        ctx->launches += 2;
        rc = lower_qubo(ctx, n, lin, m, keys, q, out, offset_out);
    } while (0);
    g.free_all();
    if (lin) cudaFree(lin);
    if (q) cudaFree(q);
    if (keys) cudaFree(keys);
    return rc;
}

// shared by the DQM and CQM builders: K copies of the graph + one-hot pairs, then model-specific groups
static int build_kway(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w, int32_t K,
                      int lin_mode, double lin_scale, double lin_base, double lin_shift, double edge_pre, double edge_shift,
                      double A, int32_t extra_vars, qa_model **out, double *off) {
    GraphDev g;
    double *cell = nullptr, *lin = nullptr, *q = nullptr;
    unsigned long long *keys = nullptr;
    int rc = graph_to_device(ctx, n, m, eu, ev, w, g);
    do {
        if (rc) break;
        const int64_t nvar64 = (int64_t)n * K + extra_vars;
        if (nvar64 >= (int64_t)0x7fffffff) { rc = fail(QA_ERR_LIMIT, "too many variables"); break; }
        const int32_t nvar = (int32_t)nvar64;
        const int64_t mq = m * K + (int64_t)n * ((int64_t)K * (K - 1) / 2);
        const size_t mm = (size_t)std::max<int64_t>(mq, 1);
        if (cudaMalloc((void **)&cell, (size_t)std::max(n, 1) * 8) != cudaSuccess ||
            cudaMalloc((void **)&lin, (size_t)std::max(nvar, 1) * 8) != cudaSuccess || cudaMalloc((void **)&q, mm * 8) != cudaSuccess ||
            cudaMalloc((void **)&keys, mm * 8) != cudaSuccess) { rc = fail(QA_ERR_CUDA, "out of device memory"); break; }
        k_vertex_accumulate<<<blocks_for(n), 256, 0, ctx->stream>>>(n, g.rowptr, g.sorted, g.w, lin_mode, lin_scale, lin_base, cell);
        k_kway_linear<<<blocks_for(nvar), 256, 0, ctx->stream>>>(n, K, nvar, cell, lin_shift, lin);
        k_kway_couplers<<<blocks_for(mq), 256, 0, ctx->stream>>>(m, n, K, g.eu, g.ev, g.w, -2.0, edge_pre, edge_shift, 2.0 * A, keys, q);
        ctx->launches += 3;
        rc = lower_qubo(ctx, nvar, lin, mq, keys, q, out, off);
    } while (0);
    g.free_all();
    void *ptrs[] = {cell, lin, q, keys};
    for (void *p : ptrs) if (p) cudaFree(p);
    return rc;
}

// objective + A*(one-hot)^2 + the K cluster-size groups.  slack: B*(N_j - min_size - slack_j)^2 with the binary slack bits
// behind the n*K cell bits; interval: B*max(0, min_size - N_j)^2, no slack bits (u = 2 (N_j - min_size), bounds [0, +inf)).
// The cell part (h, couplers, offset) is the same in both: slack bits only appear in the groups.
static int build_cqm(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w, int32_t K,
                     int32_t min_size, double onehot_penalty, double size_penalty, bool interval, qa_model **out,
                     double *offset_out) {
    if (!ctx || !out || !offset_out) return fail(QA_ERR_ARG, "null argument");
    if (K < 1 || K > QA_MAX_GROUPS) return fail(QA_ERR_LIMIT, "number of clusters must be in [1, QA_MAX_GROUPS]");
    *out = nullptr;
    QA_CUDA(cudaSetDevice(ctx->device));
    const std::vector<int> coeffs = interval ? std::vector<int>() : slack_coefficients_host((int64_t)n - min_size);
    const int nb = (int)coeffs.size();
    double off = 0.0;
    qa_model *M = nullptr;
    // linear = (number of edges at the cell) - A  (CQM_clustering.py:43: coefficient 1 per edge end, not w)
    int rc = build_kway(ctx, n, m, eu, ev, w, K, 2, 0.0, 0.0, -onehot_penalty, 0.0, 0.0, onehot_penalty, K * nb, &M, &off);
    if (rc) return rc;
    const int64_t nx = (int64_t)n * K;
    std::vector<int32_t> grp(nx + (int64_t)K * nb), coef(nx + (int64_t)K * nb);
    for (int64_t v = 0; v < nx; ++v) { grp[v] = (int32_t)(v % K); coef[v] = 1; }
    long long csum = 0;
    for (int c : coeffs) csum += c;
    for (int j = 0; j < K; ++j)
        for (int b = 0; b < nb; ++b) { grp[nx + (int64_t)j * nb + b] = j; coef[nx + (int64_t)j * nb + b] = -coeffs[b]; }
    std::vector<double> lam(K, size_penalty);
    std::vector<int64_t> kap(K, (int64_t)n - csum - 2 * (int64_t)min_size);
    rc = qa_model_set_groups(M, K, grp.data(), coef.data(), lam.data(), kap.data());
    if (!rc && interval) {
        const std::vector<int64_t> lo(K, 0), hi(K, INT64_MAX);
        rc = qa_model_set_group_bounds(M, lo.data(), hi.data());
    }
    if (rc) { qa_model_destroy(M); return rc; }
    *offset_out = off + onehot_penalty * n;
    *out = M;
    return QA_OK;
}

int qa_build_cqm_penalty(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w, int32_t K,
                         int32_t min_size, double onehot_penalty, double size_penalty, qa_model **out, double *offset_out) {
    return build_cqm(ctx, n, m, eu, ev, w, K, min_size, onehot_penalty, size_penalty, false, out, offset_out);
}

int qa_build_cqm_interval(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w, int32_t K,
                          int32_t min_size, double onehot_penalty, double size_penalty, qa_model **out, double *offset_out) {
    return build_cqm(ctx, n, m, eu, ev, w, K, min_size, onehot_penalty, size_penalty, true, out, offset_out);
}

int qa_build_dqm_onehot(qa_ctx *ctx, int32_t n, int64_t m, const int32_t *eu, const int32_t *ev, const double *w, int32_t K,
                        double gamma, double penalty, int32_t intended, qa_model **out, double *offset_out) {
    if (!ctx || !out || !offset_out) return fail(QA_ERR_ARG, "null argument");
    if (K < 1 || K > QA_MAX_GROUPS) return fail(QA_ERR_LIMIT, "number of cases must be in [1, QA_MAX_GROUPS]");
    *out = nullptr;
    QA_CUDA(cudaSetDevice(ctx->device));
    const double base_lin = gamma * (1 - (double)n / K);
    double off = 0.0;
    qa_model *M = nullptr;
    int rc;
    if (!intended)  // as written: last set_linear wins; edges overwrite the all-pairs 2*gamma which stays in the rank-1 group
        rc = build_kway(ctx, n, m, eu, ev, w, K, 3, 0.0, base_lin, -penalty, 0.0, -(2 * gamma), penalty, 0, &M, &off);
    else
        rc = build_kway(ctx, n, m, eu, ev, w, K, 0, 1.0, base_lin, -penalty, 2 * gamma, -(2 * gamma), penalty, 0, &M, &off);
    if (rc) return rc;
    const int64_t nx = (int64_t)n * K;
    std::vector<int32_t> grp(nx), coef(nx, 1);
    for (int64_t v = 0; v < nx; ++v) grp[v] = (int32_t)(v % K);
    std::vector<double> lam(K, gamma);
    std::vector<int64_t> kap(K, (int64_t)n - 1);
    rc = qa_model_set_groups(M, K, grp.data(), coef.data(), lam.data(), kap.data());
    if (rc) { qa_model_destroy(M); return rc; }
    *offset_out = off + penalty * n - gamma * K / 4.0;
    *out = M;
    return QA_OK;
}

}  // extern "C"
