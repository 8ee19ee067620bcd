// dense.cuh -- k_anneal_dense<K>: the dense k-way path (BASELINE.json config 5; SURVEY.md 2.2 K5).
//
// Reference computation: the all-pairs same-case term of DQM_clustering.py:36-37 / BQM_clustering.py:46-47 on a DENSE
// affinity -- every cell interacts with every other cell, so neal's neighbour update after a flip touches n_cells - 1 fields
// and the model's CSR is n_cells^2 * K entries.  The k-way one-hot expansion gives the couplings a Kronecker structure
//     J[(i,c),(j,c')] = [c == c'] * W[i][j]   (i != j)        J[(i,c),(i,c')] = P   (c != c')
// (variable index v = i*K + c), so the inter-cell local fields of ALL reads and cases are one dense contraction
//     F[i][(read, case)] = sum_j W[i][j] * S[j][(read, case)]
// with one n_cells x n_cells matrix W -- the "batched local fields Q.X" of the north star.
//
// Algorithm: neal's sequential sweep and per-read xorshift128+ stream, unchanged.  What changes is WHEN fields are computed:
// nothing is stored per read except the spins (bit-packed).  The sweep walks the cells in blocks of 8; for a block the
// fields of its 8 x K variables are evaluated for the warp's 32 reads by fp64 tensor-core MMAs (mma.sync m8n8k4.f64 = SASS
// DMMA.8x8x4 -- tcgen05 has no f64 kind; on sm_100a every f64 mma shape lowers to 8x8x4) over ALL cells, then the 8 x K
// variables are decided in neal's order with lane = read, flips inside the block being forwarded to the block's later
// cells in shared memory.  Same Markov chain in exact arithmetic; the fp64 summation order differs from neal's incremental
// updates, so this is a tolerance-parity mode (QA_MODE_THROUGHPUT): energies equal the fp64 re-evaluation to 1e-12
// relative, runs coincide with the oracle's until a rounding decides a branch.
//
// Tile shapes: M = 8 cells (rows of W), N = 8 columns per n-tile, 4K n-tiles per warp (32 reads x K cases), K-dim = cells.
//   A fragment  W[i0 + T/4][g*32 + (T%4)*8 + q]          (8 consecutive doubles per thread and 32-cell group: 4 x LDG.128)
//   B fragment  spin of cell g*32 + (T%4)*8 + q in column (T/4)*4K + t, expanded from one bit to +-1.0 in registers
//   C fragment  F[i0 + T/4][column (2*(T%4)+e)*4K + t]
// column a = read_lane*K + case.  Spin words SW[g][a] (bit b = cell g*32 + b) live in global memory (64 KB per warp for
// config 5, L2 resident); a thread's 4K words of a group are contiguous (K x LDG.128).
// Cost: 2 * n_cells flops per attempt, independent of the acceptance rate -- bound by the fp64 tensor pipe.

// (struct DenseDesc -- ncells, ncp, K, ngrp, W, P -- is declared in common.cuh: the model carries one)

__device__ __forceinline__ void dn_dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

template <int K>
struct DnGeom {
    static constexpr int NT = 4 * K;          // n-tiles per warp
    static constexpr int COLS = 32 * K;       // columns per warp
    static constexpr int LD = COLS + 4;       // row stride of the per-warp field block in shared memory (doubles)
};

template <int K>
__host__ __device__ inline size_t dn_smem_bytes(int warps) {
    return (size_t)warps * 8 * DnGeom<K>::LD * sizeof(double);
}

// inter-cell fields of the 8 cells i0..i0+7 for all columns of the warp: C[t][e] (fragment layout above).
// The loads of group g + 1 (8 doubles of W, 4K spin words) are issued before the 128 MMAs of group g: a warp alone on its
// scheduler keeps the fp64 tensor pipe fed.
template <int K>
__device__ __forceinline__ void dn_block_fields(const DenseDesc &Dd, const uint32_t *__restrict__ SW, int i0, int lane,
                                                double (&C)[4 * K][2]) {
    constexpr int NT = DnGeom<K>::NT, COLS = DnGeom<K>::COLS;
    const int r8 = lane >> 2, kap = lane & 3;
    const double2 *ap = reinterpret_cast<const double2 *>(Dd.W + (size_t)(i0 + r8) * Dd.ncp + kap * 8);
    const uint4 *wp = reinterpret_cast<const uint4 *>(SW + r8 * NT);
#pragma unroll
    for (int t = 0; t < NT; ++t) C[t][0] = C[t][1] = 0.0;
    double2 an[4];
    uint4 wn[K];
#pragma unroll
    for (int q = 0; q < 4; ++q) an[q] = __ldg(ap + q);
#pragma unroll
    for (int q = 0; q < K; ++q) wn[q] = __ldcg(wp + q);
    const int ngrp = Dd.ngrp;
#ifdef DN_LOP3
    unsigned sgn;
    asm volatile("mov.u32 %0, 0x80000000;" : "=r"(sgn));   // opaque: kept in a register so that (x & sgn) ^ imm is ONE LOP3
#endif
    for (int g = 0; g < ngrp; ++g) {
        double a[8];
        uint32_t w[NT];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            a[2 * q] = an[q].x;
            a[2 * q + 1] = an[q].y;
        }
#pragma unroll
        for (int q = 0; q < K; ++q) {
            w[4 * q] = wn[q].x >> (kap * 8);
            w[4 * q + 1] = wn[q].y >> (kap * 8);
            w[4 * q + 2] = wn[q].z >> (kap * 8);
            w[4 * q + 3] = wn[q].w >> (kap * 8);
        }
        if (g + 1 < ngrp) {
#pragma unroll
            for (int q = 0; q < 4; ++q) an[q] = __ldg(ap + (size_t)(g + 1) * 16 + q);
#pragma unroll
            for (int q = 0; q < K; ++q) wn[q] = __ldcg(wp + (size_t)(g + 1) * (COLS / 4) + q);
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                // bit -> +-1.0: high word 0xBFF00000 (-1.0) with the sign cleared when the bit is set
#ifdef DN_LOP3
                unsigned hi;
                asm("lop3.b32 %0, %1, %2, %3, 0x6a;" : "=r"(hi) : "r"(w[t] << (31 - q)), "r"(sgn), "r"(0xBFF00000u));   // (a & b) ^ c
#else
                const unsigned hi = ((w[t] << (31 - q)) & 0x80000000u) ^ 0xBFF00000u;
#endif
                dn_dmma(C[t][0], C[t][1], a[q], __hiloint2double((int)hi, 0));
            }
        }
    }
}

template <int K>
__device__ __forceinline__ void dn_store_fields(double *Fb, int lane, const double (&C)[4 * K][2]) {
    constexpr int NT = DnGeom<K>::NT, LD = DnGeom<K>::LD;
    const int r8 = lane >> 2, kap = lane & 3;
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        Fb[r8 * LD + (2 * kap) * NT + t] = C[t][0];
        Fb[r8 * LD + (2 * kap + 1) * NT + t] = C[t][1];
    }
}

// registers are bounded for 3 CTAs per SM (166 instead of 184): measured +19 % at EQUAL occupancy (8 warps per SM: 31.2 against
// 26.2 TFLOP/s on config 5, profiles/r2_ab_dense_variants.log) -- ptxas schedules the operand preparation tighter; 12 warps per
// SM are slower again (27.7), so the host keeps launching 2 CTAs per SM.  (K = 8 holds 64 accumulators: bounded for 2 CTAs.)
#ifndef DN_MIN_CTAS
#define DN_MIN_CTAS 3
#endif
template <int K>
__global__ void __launch_bounds__(128, (K >= 8 ? 2 : DN_MIN_CTAS)) k_anneal_dense(AnnealParams P, DenseDesc Dd) {
    constexpr int COLS = DnGeom<K>::COLS, LD = DnGeom<K>::LD;
    extern __shared__ __align__(16) double dn_smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    double *Fb = dn_smem + (size_t)wib * 8 * LD;
    const ProblemDesc &D = P.descs[0];
    uint32_t *SW = P.dn_spins + ((size_t)blockIdx.x * (blockDim.x >> 5) + wib) * (size_t)P.dn_stride;
    const int n = D.n, ncells = Dd.ncells;
    const double Pj = Dd.P;
    unsigned long long tot[5] = {0, 0, 0, 0, 0};

    for (;;) {
        unsigned long long tile = 0;
        if (lane == 0) tile = atomicAdd(P.counter, 1ull);
        tile = __shfl_sync(FULL_MASK, tile, 0);
        if ((int64_t)tile >= P.total_tiles) break;
        const int64_t r0 = (int64_t)tile * 32;
        const int64_t r = r0 + lane;
        const bool active = r < D.reads;

        // ---- pack: SW[g][rr*K + c] bit b = spin of cell g*32 + b, case c, read r0 + rr (padding cells / reads: +1)
        for (int g = 0; g < Dd.ngrp; ++g) {
            const int cell = g * 32 + lane;
            for (int rr = 0; rr < 32; ++rr) {
                const bool rv = r0 + rr < D.reads;
                const int8_t *row = D.states + (r0 + rr) * (int64_t)n;
#pragma unroll
                for (int c = 0; c < K; ++c) {
                    int s = 1;
                    if (rv && cell < ncells) {
                        s = row[(int64_t)cell * K + c];
                        if (s != 1 && s != -1) atomicExch(P.error_flag, QA_ERR_STATE);
                    }
                    const uint32_t w = __ballot_sync(FULL_MASK, s > 0);
                    if (lane == 0) __stcg(SW + (size_t)g * COLS + rr * K + c, w);
                }
            }
        }
        __syncwarp();

        const unsigned long long sd = active ? P.seeds[D.read_base + r] : 1ull;
        unsigned long long s0 = sd ? sd : ~0ull, s1 = 0;
        LaneStats st = {0, 0, 0, 0, 0};
        double C[4 * K][2];

        for (int b = 0; b < P.num_betas; ++b) {
            const double beta = P.betas[b];
            const double thr = 44.36142 / beta;
            for (int sw = 0; sw < P.sweeps_per_beta; ++sw) {
                for (int i0 = 0; i0 < Dd.ncp; i0 += 8) {
                    if (i0 >= ncells) break;
                    dn_block_fields<K>(Dd, SW, i0, lane, C);
                    dn_store_fields<K>(Fb, lane, C);
                    __syncwarp();
                    // ---- decide the block's 8 x K variables in neal's order, lane = read
                    uint32_t *myw = SW + (size_t)(i0 >> 5) * COLS + lane * K;
                    uint32_t wv[K];
#pragma unroll
                    for (int c = 0; c < K; ++c) wv[c] = __ldcg(myw + c);
                    const int b0 = i0 & 31;
                    bool dirty = false;
                    // the block's own 8 x 8 couplings, two per lane: rows 0-3 in wlo, rows 4-7 in whi, column = lane & 7
                    const double wlo = __ldg(Dd.W + (size_t)(i0 + (lane >> 3)) * Dd.ncp + i0 + (lane & 7));
                    const double whi = __ldg(Dd.W + (size_t)(i0 + 4 + (lane >> 3)) * Dd.ncp + i0 + (lane & 7));
                    for (int m = 0; m < 8; ++m) {
                        const int i = i0 + m;
                        if (i >= ncells) break;
                        double f[K];
                        int s[K];
                        // neighbour updates count neal's way: the CSR degree of the flipped variable (zeros of W are absent)
                        int32_t rp[K + 1];
#pragma unroll
                        for (int c = 0; c <= K; ++c) rp[c] = __ldg(D.rowptr + (size_t)i * K + c);
#pragma unroll
                        for (int c = 0; c < K; ++c) {
                            f[c] = Fb[m * LD + lane * K + c] + __ldg(D.h + (size_t)i * K + c);
                            s[c] = ((wv[c] >> (b0 + m)) & 1u) ? 1 : -1;
                        }
#pragma unroll
                        for (int c = 0; c < K; ++c) {
                            int others = 0;
#pragma unroll
                            for (int c2 = 0; c2 < K; ++c2) others += (c2 != c) ? s[c2] : 0;
                            const double fv = f[c] + Pj * (double)others;
                            const double dE = s[c] > 0 ? -2.0 * fv : 2.0 * fv;
                            const bool cand = active && !(dE >= thr);
                            st.cand += cand;
                            const bool acc = ls_accept(dE, cand, beta, s0, s1, st);
                            if (acc) {
                                st.acc++;
                                st.nbr += (unsigned)(rp[c + 1] - rp[c]);
                                s[c] = -s[c];
                                wv[c] ^= 1u << (b0 + m);
                                dirty = true;
                            }
                            if (m < 7 && __any_sync(FULL_MASK, acc)) {
                                const double d2 = acc ? (s[c] > 0 ? 2.0 : -2.0) : 0.0;   // 2 * s_new
                                for (int m2 = m + 1; m2 < 8; ++m2) {
                                    const double wj = __shfl_sync(FULL_MASK, m2 < 4 ? wlo : whi, (m2 & 3) * 8 + m);
                                    Fb[m2 * LD + lane * K + c] += d2 * wj;
                                }
                            }
                        }
                    }
                    if (dirty) {
#pragma unroll
                        for (int c = 0; c < K; ++c) __stcg(myw + c, wv[c]);
                    }
                    __syncwarp();
                }
            }
        }

        // ---- energy of the final state: E = sum_v s_v * (h_v + (F_v + P * sum_{c' != c} s_ic') / 2), one more field pass
        double E = 0.0;
        for (int i0 = 0; i0 < Dd.ncp; i0 += 8) {
            if (i0 >= ncells) break;
            dn_block_fields<K>(Dd, SW, i0, lane, C);
            dn_store_fields<K>(Fb, lane, C);
            __syncwarp();
            const uint32_t *myw = SW + (size_t)(i0 >> 5) * COLS + lane * K;
            const int b0 = i0 & 31;
            for (int m = 0; m < 8; ++m) {
                const int i = i0 + m;
                if (i >= ncells) break;
                int s[K], S = 0;
#pragma unroll
                for (int c = 0; c < K; ++c) {
                    s[c] = ((__ldcg(myw + c) >> (b0 + m)) & 1u) ? 1 : -1;
                    S += s[c];
                }
#pragma unroll
                for (int c = 0; c < K; ++c) {
                    const double half = 0.5 * (Fb[m * LD + lane * K + c] + Pj * (double)(S - s[c]));
                    const double t = __ldg(D.h + (size_t)i * K + c) + half;
                    E += s[c] > 0 ? t : -t;
                }
            }
            __syncwarp();
        }
        if (active) D.energies[r] = E;

        // ---- unpack the final spins into the caller's rows
        for (int g = 0; g < Dd.ngrp; ++g) {
            const int cell = g * 32 + lane;
            for (int rr = 0; rr < 32; ++rr) {
                if (r0 + rr >= D.reads) break;
                int8_t *row = D.states + (r0 + rr) * (int64_t)n;
#pragma unroll
                for (int c = 0; c < K; ++c) {
                    const uint32_t w = __ldcg(SW + (size_t)g * COLS + rr * K + c);
                    if (cell < ncells) row[(int64_t)cell * K + c] = ((w >> lane) & 1u) ? 1 : -1;
                }
            }
        }
        __syncwarp();
        tot[0] += st.cand;
        tot[1] += st.draws;
        tot[2] += st.acc;
        tot[3] += st.ties;
        tot[4] += st.nbr;
    }
#pragma unroll
    for (int q = 0; q < 5; ++q)
        for (int off = 16; off > 0; off >>= 1) tot[q] += __shfl_xor_sync(FULL_MASK, tot[q], off);
    if (lane == 0) {
        atomicAdd(P.stats + ST_CAND, tot[0]);
        atomicAdd(P.stats + ST_DRAWS, tot[1]);
        atomicAdd(P.stats + ST_ACC, tot[2]);
        atomicAdd(P.stats + ST_TIES, tot[3]);
        atomicAdd(P.stats + ST_NBR, tot[4]);
    }
}

// ---- structure detection: scatter the CSR of a one-hot k-way model into W, verifying the Kronecker form ---------------
// flag bits: 1 = coupler between different cells AND different cases, 2 = case-dependent inter-cell coupling,
//            4 = duplicate inter-cell coupler, 8 = intra-cell couplings differ, 16 = a cell's one-hot couplers are neither all
//            present once nor all absent
// The host then requires (counts[0] = case-0 inter-cell entries, counts[1] = all same-case inter-cell entries, counts[2] =
// intra-cell entries) counts[1] == K * counts[0] -- with no duplicates and every entry of row (i, c) found in row (i, 0), every
// row (i, c) then holds exactly the cells of row (i, 0) -- and counts[2] == 0 or n * (K - 1): all cells complete, or none
// has one-hot couplers (P = 0).
constexpr unsigned long long DN_EMPTY = 0x7ff8dead00000001ull;   // a NaN payload no input produces

__global__ void k_dense_fill(size_t count, unsigned long long *W) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) W[i] = DN_EMPTY;
}

// pass 0: case-0 entries write their cell of W, every same-case inter-cell entry sets bit c of seen[i][j] (a bit already set is
// a duplicate), intra-cell entries are compared with P and must cover the other K - 1 cases exactly once or not at all;
// pass 1: the entries of cases 1..K-1 are compared with W
__global__ void k_dense_scatter(int32_t n, int32_t K, int32_t ncp, const int32_t *rowptr, const int32_t *col, const double *val,
                                double P, unsigned long long *W, unsigned int *seen, int *flag, unsigned long long *counts,
                                int pass) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const int i = v / K, c = v % K;
    unsigned long long n0 = 0, nall = 0;
    unsigned int nintra = 0, cases = 0;
    for (int e = rowptr[v]; e < rowptr[v + 1]; ++e) {
        const int u = col[e];
        const int j = u / K, c2 = u % K;
        const unsigned long long bits = (unsigned long long)__double_as_longlong(val[e]);
        if (i == j) {
            if (pass == 0 && bits != (unsigned long long)__double_as_longlong(P)) atomicOr(flag, 8);
            ++nintra;
            cases |= 1u << c2;
            continue;
        }
        if (c != c2) {
            if (pass == 0) atomicOr(flag, 1);
            continue;
        }
        ++nall;
        const size_t cell = (size_t)i * ncp + j;
        if (pass == 0) {
            // seen: one byte per (i, j), bit c = case c (K <= 8)
            const unsigned int bit = 1u << ((cell & 3) * 8 + c);
            if (atomicOr(seen + (cell >> 2), bit) & bit) atomicOr(flag, 4);
            if (c == 0) {
                ++n0;
                W[cell] = bits;      // two writers only for a duplicate, which is flagged
            }
        } else if (c != 0) {
            if (W[cell] != bits) atomicOr(flag, 2);
        }
    }
    if (pass == 0) {
        if (nintra != 0 && (nintra != (unsigned)(K - 1) || cases != (((1u << K) - 1) & ~(1u << c)))) atomicOr(flag, 16);
        atomicAdd(counts, n0);
        atomicAdd(counts + 1, nall);
        atomicAdd(counts + 2, (unsigned long long)nintra);
    }
}

__global__ void k_dense_finish(size_t count, unsigned long long *W) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count && W[i] == DN_EMPTY) W[i] = 0ull;
}
