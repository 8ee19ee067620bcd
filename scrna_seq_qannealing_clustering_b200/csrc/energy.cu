// energy.cu -- k_energy: neal get_state_energy() per read in neal's summation order (bit-exact), on the read-transposed packed
// spins the annealing kernels leave behind; k_pack_states brings caller-provided states into that layout.
#include "common.cuh"

using namespace qa;

namespace {

#ifndef QA_EN_BATCH
#define QA_EN_BATCH 16
#endif

// ------------------------------------------------------------------------------------------------
// energies: neal get_state_energy(), one thread per read, reads on lanes (coalesced packedT loads)
// ------------------------------------------------------------------------------------------------
// INTERVAL: the groups carry interval bounds (every problem with groups has them): E_g = lambda * (double)(d*d) * 0.25 with
// d = max(lo - u, 0, u - hi), u = M_g + kappa_g -- the equality term below is the case lo = hi = 0.
template <bool INTERVAL>
__global__ void __launch_bounds__(128) k_energy(const ProblemDesc *descs) {
    const ProblemDesc D = descs[blockIdx.y];
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= D.reads) return;
    const uint32_t *pk = D.packedT + r;
    const int64_t stride = D.rpad;
    double E = 0.0;
    // rank-1 group sums M_g = sum a_v s_v ride along with the linear pass (one pass over the spins for ALL groups)
    long long M[QA_MAX_GROUPS];
    for (int g = 0; g < D.ngroups; ++g) M[g] = 0;
    for (int c = 0; c < D.nch; ++c) {
        const uint32_t w = pk[c * stride];
        const int base = c * 32;
        const int lim = min(32, D.n - base);
        for (int i = 0; i < lim; ++i) {
            const double hv = __ldg(D.h + base + i);
            E += ((w >> i) & 1u) ? hv : -hv;  // state[v]*h[v]
        }
        if (D.ngroups) {
            for (int i = 0; i < lim; ++i) {
                const int g = __ldg(D.grp + base + i);   // uniform
                if (g >= 0) {
                    const long long a = __ldg(D.coef + base + i);
                    M[g] += ((w >> i) & 1u) ? a : -a;
                }
            }
        }
    }
    // couplers in the caller's order: the additions are one dependent chain, the (random-row) spin loads are not -- issue
    // them QA_EN_BATCH couplers at a time.  Measured on config 3 (75 776 reads): 228 ms with batches of 8, 217 ms with 16, 240 ms
    // with 32; keeping the row's word in a register across the couplers that share it (a uniform branch in the add chain) is
    // slower, 261 ms.
    int64_t e = 0;
    for (; e + QA_EN_BATCH <= D.m; e += QA_EN_BATCH) {
        uint32_t bu[QA_EN_BATCH], bv[QA_EN_BATCH];
        double wt[QA_EN_BATCH];
#pragma unroll
        for (int q = 0; q < QA_EN_BATCH; ++q) {
            const int u = __ldg(D.starts + e + q), v = __ldg(D.ends + e + q);
            wt[q] = __ldg(D.w + e + q);
            bu[q] = pk[(int64_t)(u >> 5) * stride] >> (u & 31);
            bv[q] = pk[(int64_t)(v >> 5) * stride] >> (v & 31);
        }
#pragma unroll
        for (int q = 0; q < QA_EN_BATCH; ++q) E += ((bu[q] ^ bv[q]) & 1u) ? -wt[q] : wt[q];  // state[u]*w*state[v]
    }
    for (; e < D.m; ++e) {
        const int u = __ldg(D.starts + e), v = __ldg(D.ends + e);
        const double wt = __ldg(D.w + e);
        const uint32_t bu = (pk[(int64_t)(u >> 5) * stride] >> (u & 31)) & 1u;
        const uint32_t bv = (pk[(int64_t)(v >> 5) * stride] >> (v & 31)) & 1u;
        E += (bu ^ bv) ? -wt : wt;
    }
    for (int g = 0; g < D.ngroups; ++g) {
        const long long t = INTERVAL ? interval_dist(M[g] + D.kappa[g], D.kappa[D.ngroups + g], D.kappa[2 * D.ngroups + g]) : M[g] + D.kappa[g];
        E += D.lambda[g] * (double)(t * t) * 0.25;
    }
    D.energies[r] = E;
}

// pack caller-provided +-1 states into the read-transposed layout (for qa_energy_argmin)
__global__ void k_pack_states(ProblemDesc D, int *error_flag) {
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= D.reads) return;
    const int8_t *row = D.states + r * (int64_t)D.n;
    for (int c = 0; c < D.nch; ++c) {
        const int v = c * 32 + lane;
        int s = 1;
        if (v < D.n) {
            s = row[v];
            if (s != 1 && s != -1) atomicExch(error_flag, QA_ERR_STATE);
        }
        const uint32_t w = __ballot_sync(FULL_MASK, s > 0);
        if (lane == 0) D.packedT[(int64_t)c * D.rpad + r] = w;
    }
}

}  // namespace

namespace qa {

int launch_energy(qa_ctx *ctx, qa_model *M, int32_t reads_per_problem) {
    dim3 g((unsigned)((reads_per_problem + 127) / 128), (unsigned)M->num_problems);
    if (M->gbounds) k_energy<true><<<g, 128, 0, ctx->stream>>>(M->d_descs);
    else k_energy<false><<<g, 128, 0, ctx->stream>>>(M->d_descs);
    QA_CUDA(cudaGetLastError());
    ctx->launches++;
    return QA_OK;
}

int launch_pack_states(qa_ctx *ctx, const ProblemDesc &D, int64_t threads) {
    const int tpb = 256;
    k_pack_states<<<(unsigned)((threads + tpb - 1) / tpb), tpb, 0, ctx->stream>>>(D, ctx->d_flag);
    QA_CUDA(cudaGetLastError());
    ctx->launches++;
    return QA_OK;
}

}  // namespace qa
