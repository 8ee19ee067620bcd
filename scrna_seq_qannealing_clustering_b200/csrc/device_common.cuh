// device_common.cuh -- device helpers shared by the annealing kernels: neal's xorshift128+ step, the accept test with its
// single-precision screen, L2 prefetch / fp64 reduction wrappers, cp.async wrappers, per-lane event counters, group
// parameters in shared memory.
#pragma once

#include "common.cuh"

namespace qa {

__device__ __forceinline__ unsigned long long rng_next(unsigned long long &s0, unsigned long long &s1) {
    // neal FASTRAND (xorshift128+)
    unsigned long long x = s0;
    const unsigned long long y = s1;
    s0 = y;
    x ^= x << 23;
    s1 = x ^ y ^ (x >> 17) ^ (y >> 26);
    return s1 + y;
}

__device__ __forceinline__ void prefetch_l2(const void *p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

__device__ __forceinline__ void red_add_f64(double *addr, double v) {
    // fire-and-forget fp64 reduction performed at L2 (RED.E.ADD.F64); round-to-nearest like the CPU add
    asm volatile("red.global.add.f64 [%0], %1;" ::"l"(addr), "d"(v) : "memory");
}

__device__ __forceinline__ void red_add_f64_if(double *addr, double v, bool pred) {
    // predicated form: no branch / reconvergence point in the neighbour loop
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p red.global.add.f64 [%0], %1;\n\t}" ::"l"(addr), "d"(v), "r"((int)pred)
                 : "memory");
}

struct WarpStats {
    unsigned long long cand, draws, acc, nbr, active, chunks, ties;
};

struct LaneStats {
    unsigned int cand, draws, acc, ties;
    unsigned long long nbr;
};

__device__ __forceinline__ void cp_async4(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// accept test of one variable for every lane (read) of the warp; returns the per-lane accept flag.
// neal: flip iff exp(-dE*beta) * 2^64 > (double)rand.  The fp64 exp, the 64-bit conversion and the fp64 products are the
// longest dependent chain of a step, so the draw is first screened in SINGLE precision on its upper 32 bits:
//   pa = ex2.approx(float(dE) * float(-beta * log2 e)) is within 3e-5 relative of exp(-dE*beta) for -dE*beta in [-44.4, 0]
//        (two roundings of 6e-8 on an exponent of magnitude <= 64 -> 1.2e-5 absolute in the exponent -> 8e-6, + 2 ulp of
//        ex2.approx);
//   rh = float(rand >> 32): rand / 2^32 lies in [rh', rh' + 1) with rh' = floor(rand / 2^32), |rh - rh'| <= 6e-8 rh'.
// rh + 1 < 0.9999 * pa * 2^32  =>  rand < 0.99994 * exp(..) * 2^64: every fp64 evaluation accepts;
// rh     > 1.0001 * pa * 2^32  =>  rand > 1.00006 * exp(..) * 2^64: every fp64 evaluation rejects.
// Only draws inside that band (2e-4 of them, + 2^-32 / p) take the fp64 path -- the result is identical by construction,
// and near ties (|p - r| <= 2^-48 p) can only occur inside the band, where they are still counted.
__device__ __forceinline__ bool ls_accept(double dE, bool cand, double beta, unsigned long long &s0, unsigned long long &s1,
                                          LaneStats &st) {
    bool acc = cand;
    const bool need = cand && dE > 0.0;
    bool exact = false;
    unsigned long long rnd = 0ull;
    if (need) {
        rnd = rng_next(s0, s1);
        st.draws++;
        float pa;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(pa) : "f"(__double2float_rn(dE) * __double2float_rn(beta * -1.4426950408889634)));
        const float rh = __uint2float_rn((unsigned)(rnd >> 32));
        acc = rh + 1.0f < pa * 4294537799.0f;               // 0.9999 * 2^32
        exact = !acc && !(rh > pa * 4295396793.0f);         // 1.0001 * 2^32
    }
    if (__any_sync(FULL_MASK, exact)) {
        if (exact) {
            const double p = exp(-dE * beta) * QA_TWO64;
            double rd;   // volatile: the conversion must stay inside this rare path (the compiler would hoist it)
            asm volatile("cvt.rn.f64.u64 %0, %1;" : "=d"(rd) : "l"(rnd));
            acc = p > rd;
            if (fabs(p - rd) <= p * 3.5527136788005009e-15) st.ties++;
        }
    }
    return acc;
}

// Gibbs (heat-bath) counterpart of ls_accept, dwave-samplers >= 1.0 (SURVEY.md C.8): a candidate (dE < thr) is accepted
// without a draw if dE <= -thr, else iff 2^64 > (double)rand * (1 + exp(dE*beta)).  No single-precision screen: every draw
// takes the fp64 path, so the result is neal's arithmetic by construction.  Near ties: |2^64 - rand (1 + exp)| <= 2^-48 2^64.
__device__ __forceinline__ bool gibbs_accept(double dE, bool cand, double beta, double thr, unsigned long long &s0,
                                             unsigned long long &s1, LaneStats &st) {
    bool acc = cand;
    if (cand && !(dE <= -thr)) {
        const unsigned long long rnd = rng_next(s0, s1);
        st.draws++;
        const double q = __ull2double_rn(rnd) * (1.0 + exp(dE * beta));
        acc = QA_TWO64 > q;
        if (fabs(QA_TWO64 - q) <= QA_TWO64 * 3.5527136788005009e-15) st.ties++;
    }
    return acc;
}

// the accept test of the lockstep and replay kernels for the call's acceptance rule
template <Proposal PROP>
__device__ __forceinline__ bool accept_test(double dE, bool cand, double beta, double thr, unsigned long long &s0,
                                            unsigned long long &s1, LaneStats &st) {
    if (PROP == PROP_GIBBS) return gibbs_accept(dE, cand, beta, thr, s0, s1, st);
    return ls_accept(dE, cand, beta, s0, s1, st);
}

// lambda / kappa of every group into shared memory, kappa_words(GK) words of kappa per group ({kappa, lo, hi} for interval
// groups).  Groups exist only on single-problem models, so the lockstep and replay kernels keep one copy per block.
template <GroupKind GK>
__device__ __forceinline__ void stage_group_params(const ProblemDesc &D0, double *lam_sh, long long *kap_sh) {
    for (int g = threadIdx.x; g < D0.ngroups; g += blockDim.x) {
        lam_sh[g] = D0.lambda[g];
        if (GK == GK_INTERVAL) {
            kap_sh[3 * g] = D0.kappa[g];
            kap_sh[3 * g + 1] = D0.kappa[D0.ngroups + g];
            kap_sh[3 * g + 2] = D0.kappa[2 * D0.ngroups + g];
        } else {
            kap_sh[g] = D0.kappa[g];
        }
    }
}

// warp-reduce the per-lane counters and add them to the launch's totals
__device__ __forceinline__ void flush_lane_stats(const AnnealParams &P, const LaneStats &st) {
    unsigned long long v[5] = {st.cand, st.draws, st.acc, st.ties, st.nbr};
#pragma unroll
    for (int q = 0; q < 5; ++q)
        for (int off = 16; off > 0; off >>= 1) v[q] += __shfl_xor_sync(FULL_MASK, v[q], off);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(P.stats + ST_CAND, v[0]);
        atomicAdd(P.stats + ST_DRAWS, v[1]);
        atomicAdd(P.stats + ST_ACC, v[2]);
        atomicAdd(P.stats + ST_TIES, v[3]);
        atomicAdd(P.stats + ST_NBR, v[4]);
    }
}

}  // namespace qa
