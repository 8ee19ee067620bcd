// anneal_dense.cu -- k_anneal_dense (dense.cuh): dense k-way models on the fp64 tensor cores; structure detection and launch.
#include "device_common.cuh"

using namespace qa;

namespace {

#include "dense.cuh"

}  // namespace

namespace qa {

int launch_dense(Launch &L) {
    qa_ctx *ctx = L.ctx;
    qa_model *M = L.M;
    AnnealParams &A = L.A;
    // dense k-way: one warp = 32 reads, fields of a block of 8 cells by fp64 tensor-core MMAs over all cells (dense.cuh)
    const int K = M->dn.K;
    const int warps = 4;
    const void *fn = K == 1 ? (const void *)k_anneal_dense<1> : K == 2 ? (const void *)k_anneal_dense<2>
                   : K == 4 ? (const void *)k_anneal_dense<4> : (const void *)k_anneal_dense<8>;
    const size_t smem = K == 1 ? dn_smem_bytes<1>(warps) : K == 2 ? dn_smem_bytes<2>(warps)
                      : K == 4 ? dn_smem_bytes<4>(warps) : dn_smem_bytes<8>(warps);
    QA_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int bps = 0;
    QA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessorWithFlags(&bps, fn, warps * 32, smem, cudaOccupancyDefault));
    if (bps < 1) return fail(QA_ERR_CUDA, "dense kernel does not fit on an SM");
    const int64_t total_tiles = (A.reads_per_problem + 31) / 32;
    // every warp pulls 32-read tiles from a counter; no more CTAs than the tiles can fill (warps without a tile leave at once)
    bps = std::min(bps, 2);   // 8 warps per SM beat 12 (measured, see dense.cuh)
    const int64_t grid = std::min<int64_t>((int64_t)bps * ctx->num_sms, (total_tiles + warps - 1) / warps);
    const int64_t stride = (int64_t)M->dn.ngrp * 32 * K;
    const int rc = ensure(ctx->sf, (size_t)grid * warps * stride * sizeof(uint32_t));
    if (rc) return rc;
    A.dn_spins = (uint32_t *)ctx->sf.p;
    A.dn_stride = stride;
    A.total_tiles = total_tiles;
    A.read_begin = 0;
    A.read_end = A.total_reads;
    QA_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    QA_CUDA(cudaMemsetAsync(A.counter, 0, sizeof(unsigned long long), ctx->stream));
    void *args[] = {&A, &M->dn};
    QA_CUDA(cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(warps * 32), args, smem, ctx->stream));
    QA_CUDA(cudaGetLastError());
    ctx->launches++;
    if (L.st) L.st->anneal_launches++;
    L.done = A.total_reads;
    return QA_OK;
}

}  // namespace qa

extern "C" {

// Dense k-way form for k_anneal_dense: W[i][j] = J between (i,c) and (j,c), P = J between two cases of one cell, derived
// from the device CSR and verified: every inter-cell coupler joins equal cases, appears once, and a pair of cells is coupled in
// all K cases with one weight or in none; every cell has all K(K-1)/2 intra-cell couplers once, each equal to P, or no cell
// has any (P = 0).  The kernel anneals exactly that model, so anything else must stay on the reference-order kernels.
// Returns 1 when the model has that structure (QA_MODE_THROUGHPUT then runs the tensor-core kernel), 0 when it does not
// (nothing changes).
int qa_model_enable_dense(qa_model *M, int32_t K) {
    if (!M) return fail(QA_ERR_ARG, "null model");
    if (K != 1 && K != 2 && K != 4 && K != 8) return fail(QA_ERR_ARG, "dense form: cases per cell must be 1, 2, 4 or 8");
    if (M->num_problems != 1 || M->ngroups != 0) return 0;   // batched models and rank-1 group terms are outside the dense form
    const int64_t n = M->n_total;
    if (n == 0 || n % K != 0) return fail(QA_ERR_ARG, "number of variables is not a multiple of the cases per cell");
    qa_ctx *ctx = M->ctx;
    QA_CUDA(cudaSetDevice(ctx->device));
    if (M->dn_W) { cudaFree(M->dn_W); M->dn_W = nullptr; }
    M->dn_ok = false;
    const int32_t ncells = (int32_t)(n / K);
    const int32_t ncp = (ncells + 31) & ~31;
    // P: the first intra-cell coupler of variable 0 (its neighbours 1..K-1 come first in an ascending row; any order works)
    double Pj = 0.0;
    if (K > 1) {
        int32_t rp[2];
        QA_CUDA(cudaMemcpy(rp, M->rowptr, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost));
        const int32_t d0 = rp[1] - rp[0];
        if (d0 > 0) {
            std::vector<int32_t> c0(d0);
            std::vector<double> v0(d0);
            QA_CUDA(cudaMemcpy(c0.data(), M->col + rp[0], (size_t)d0 * sizeof(int32_t), cudaMemcpyDeviceToHost));
            QA_CUDA(cudaMemcpy(v0.data(), M->val + rp[0], (size_t)d0 * sizeof(double), cudaMemcpyDeviceToHost));
            for (int32_t e = 0; e < d0; ++e)
                if (c0[e] < K) { Pj = v0[e]; break; }
        }
    }
    const size_t cells2 = (size_t)ncp * ncp;
    QA_CUDA(cudaMalloc((void **)&M->dn_W, cells2 * sizeof(double)));
    unsigned long long *Wb = reinterpret_cast<unsigned long long *>(M->dn_W);
    unsigned long long *d_counts = nullptr;
    unsigned int *d_seen = nullptr;     // one byte per cell pair (ncp is a multiple of 32: whole words)
    QA_CUDA(cudaMalloc((void **)&d_counts, 3 * sizeof(unsigned long long)));
    cudaError_t ce = cudaMalloc((void **)&d_seen, cells2);
    if (ce != cudaSuccess) {
        cudaFree(d_counts);
        return fail(QA_ERR_CUDA, std::string("dense form: ") + cudaGetErrorString(ce));
    }
    QA_CUDA(cudaMemsetAsync(d_counts, 0, 3 * sizeof(unsigned long long), ctx->stream));
    QA_CUDA(cudaMemsetAsync(d_seen, 0, cells2, ctx->stream));
    QA_CUDA(cudaMemsetAsync(ctx->d_flag, 0, 2 * sizeof(int), ctx->stream));
    const int tpb = 256;
    k_dense_fill<<<(unsigned)((cells2 + tpb - 1) / tpb), tpb, 0, ctx->stream>>>(cells2, Wb);
    for (int pass = 0; pass < 2; ++pass)
        k_dense_scatter<<<(unsigned)((n + tpb - 1) / tpb), tpb, 0, ctx->stream>>>((int32_t)n, K, ncp, M->rowptr, M->col, M->val, Pj, Wb,
                                                                                 d_seen, ctx->d_flag, d_counts, pass);
    k_dense_finish<<<(unsigned)((cells2 + tpb - 1) / tpb), tpb, 0, ctx->stream>>>(cells2, Wb);
    ctx->launches += 4;
    int flag = 0;
    unsigned long long counts[3] = {0, 0, 0};
    ce = cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(counts, d_counts, sizeof(counts), cudaMemcpyDeviceToHost, ctx->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_counts);
    cudaFree(d_seen);
    if (ce != cudaSuccess) return fail(QA_ERR_CUDA, std::string("dense form: ") + cudaGetErrorString(ce));
    const unsigned long long onehot_full = (unsigned long long)n * (unsigned long long)(K - 1);
    if (flag != 0 || counts[0] * (unsigned long long)K != counts[1] || (counts[2] != 0 && counts[2] != onehot_full)) {
        cudaFree(M->dn_W);
        M->dn_W = nullptr;
        return 0;
    }
    M->dn.ncells = ncells;
    M->dn.ncp = ncp;
    M->dn.K = K;
    M->dn.ngrp = ncp / 32;
    M->dn.W = M->dn_W;
    M->dn.P = Pj;
    M->dn_ok = true;
    return 1;
}

}  // extern "C"
