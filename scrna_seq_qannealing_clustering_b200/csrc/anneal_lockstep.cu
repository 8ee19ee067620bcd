// anneal_lockstep.cu -- k_anneal_lockstep: 32 reads per warp, neal's EAGER neighbour updates (bit-exact); the kernel for models
// whose rows do not fit the replay kernel's slab format (materialised all-pairs terms, dense rows).
#include "device_common.cuh"

using namespace qa;

namespace {

// ------------------------------------------------------------------------------------------------
// lockstep kernel: one warp = 32 reads of the same problem; the lanes walk the variables together, every lane
// owning one read (its own xorshift128+ state, its own spins, its own decisions).  The CSR row of the current
// variable is shared by the warp, so a neighbour update is ONE coalesced 256-byte reduction for up to 32 reads
// instead of 32 scattered 8-byte ones, and exp()/RNG run on all lanes at once.  A tile runs two kinds of pass:
//   LS_FIELD_SETUP  once: evaluates f[v] = h_v + sum_j J_vj s_j from the bit-packed spins through per-block tables of
//                   distinct spin words (neal's get_flip_energy order) and stores it.
//   LS_PUSH         every sweep: local fields f[v][lane] (fp64, read-interleaved) are kept in HBM and updated by
//                   red.global.add.f64 exactly like the warp-per-read kernel -> bit-exact against the oracle.
// Spins live in the read-transposed packed layout packedT[word][read] the energy kernel consumes.
// ------------------------------------------------------------------------------------------------
constexpr int QA_LS_TPB = 128;   // threads per block of the lockstep kernel
constexpr int QA_LS_WPB = QA_LS_TPB / 32;
constexpr int QA_LS_D = 16;      // variables per staged block
constexpr int QA_LS_CAP = 384;   // CSR entries staged per block (longer blocks fall back to global loads)
constexpr int QA_LS_CAPW = 32;   // distinct spin words per block held in shared memory (aliases the `cur` staging area)
static_assert(QA_LS_CAPW * sizeof(uint32_t) <= QA_LS_D * sizeof(double), "spin-word staging must fit into the field staging area");

// per-warp staging area in shared memory (double buffered by block parity)
struct LsStage {
    double eJ[2][QA_LS_CAP];                    // couplings of the block's CSR entries
    int ej[2][QA_LS_CAP];                       // neighbour indices
    int rowp[QA_LS_D + 1];
    int gm[QA_LS_D];
    int am[QA_LS_D];
    int pad_;
};
struct LsSetupStage {                           // field set-up pass: field evaluation from the spins
    double hb[2][QA_LS_D];                      // h of the block's variables
    unsigned int slotw[2][QA_LS_CAP / 2 + 2];   // per-entry (slot | bit << 8) as 16-bit pairs; slot 255 = own word
    int bw[2][QA_LS_CAPW];                      // distinct spin words referenced by the block
};

struct LsCtx {
    const ProblemDesc &D;
    const AnnealParams &P;
    int64_t r;
    bool active;
    double *fT;
    int *Mcol;
    double *cur;            // smem, per warp [QA_LS_D][32], this lane's column
    LsStage &sg;
    LsSetupStage &sp;
    uint32_t *words;        // smem [QA_LS_CAPW][32], this lane's column; aliases `cur` (never live at the same time)
    const double *lam_sh;
    const long long *kap_sh;
};

// h_v + sum over the CSR row of (+-J) in adjacency order, spin words loaded 8 at a time (loads batched, adds sequential)
__device__ __forceinline__ double ls_field_direct(const ProblemDesc &D, const uint32_t *pk, int64_t rpad, int v, int e0, int e1,
                                                  int own_word, uint32_t w_own) {
    double fv = __ldg(D.h + v);
    for (int e = e0; e < e1; e += 8) {
        int jq[8];
        uint32_t wq[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            jq[q] = __ldg(D.col + min(e + q, e1 - 1));
            const int wj = jq[q] >> 5;
            wq[q] = (wj != own_word) ? pk[(int64_t)wj * rpad] : w_own;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (e + q < e1) {
                const double J = __ldg(D.val + e + q);
                fv += ((wq[q] >> (jq[q] & 31)) & 1u) ? J : -J;
            }
        }
    }
    return fv;
}

enum LsPass { LS_PUSH, LS_FIELD_SETUP };

// LS_PUSH: the whole schedule of push sweeps (bit-exact).  LS_FIELD_SETUP: one pass that only evaluates the local fields
// from the spins and stores them (neal get_flip_energy order), before the push sweeps.
// GROUPS: GK_NONE, GK_EQ64 (equality groups of both widths) or GK_INTERVAL (kap_sh then holds {kappa, lo, hi} per group).
// PROP: the acceptance rule of the push sweeps (the set-up pass decides nothing).
// The loop counters bi / swi are the caller's variables, both 0 on entry: with counters local to this function nvcc orders
// a few instructions of the kernel differently, and the kernel's measured numbers (DESIGN.md 4.2) are for this SASS.
template <LsPass PASS, GroupKind GROUPS, Proposal PROP>
__device__ void ls_sweeps(const LsCtx &c, int &bi, int &swi, unsigned long long &s0, unsigned long long &s1, LaneStats &st) {
    const ProblemDesc &D = c.D;
    const AnnealParams &P = c.P;
    LsStage &sg = c.sg;
    LsSetupStage &sp = c.sp;
    const int lane = threadIdx.x & 31;
    const int n = D.n;
    const int nch = D.nch;
    const int64_t rpad = D.rpad;
    uint32_t *pk = D.packedT + c.r;
    double *fT = c.fT;
    double *cur = c.cur;
    int *Mcol = c.Mcol;
    const bool active = c.active;
    const bool tables = PASS == LS_FIELD_SETUP && D.bw_ptr != nullptr;
    const int nblk = nch * (32 / QA_LS_D);

    // software pipeline over blocks of QA_LS_D variables:
    //   rows (and, for the set-up pass, h / slot bytes / distinct-word list) of block b+1 are copied to shared memory by
    //   cp.async while block b is processed; row pointers and group metadata run two blocks ahead in registers; (push) the
    //   local fields of block b+1 are prefetched into registers and moved to shared memory at the switch.
    auto load_meta = [&](int blk, int &rp, int &gmv, int &amv) {
        const int v = blk * QA_LS_D + lane;
        rp = 0;
        if (lane <= QA_LS_D) rp = __ldg(D.rowptr + v);
        else if (tables && lane <= QA_LS_D + 2) rp = __ldg(D.bw_ptr + blk + (lane - QA_LS_D - 1));
        gmv = -1;
        amv = 0;
        if (GROUPS != GK_NONE) {
            if (lane < QA_LS_D) {
                gmv = __ldg(D.grp + v);
                amv = __ldg(D.coef + v);
            }
        }
    };
    auto stage_rows = [&](int buf, int blk, int rp) {
        const int eb = __shfl_sync(FULL_MASK, rp, 0);
        const int ee = __shfl_sync(FULL_MASK, rp, QA_LS_D);
        const int cnt = ee - eb;
        if (cnt <= QA_LS_CAP) {
            for (int k = lane; k < cnt; k += 32) {
                cp_async4(&sg.ej[buf][k], D.col + eb + k);
                cp_async8(&sg.eJ[buf][k], D.val + eb + k);
            }
            if (PASS == LS_FIELD_SETUP) {
                if (tables) {
                    const int b0 = __shfl_sync(FULL_MASK, rp, QA_LS_D + 1);
                    const int b1 = __shfl_sync(FULL_MASK, rp, QA_LS_D + 2);
                    for (int k = lane; k < b1 - b0; k += 32) cp_async4(&sp.bw[buf][k], D.bw_words + b0 + k);
                    const int a0 = eb & ~1;                       // 16-bit entries staged as aligned 32-bit words
                    const int nw2 = ((ee + 1) & ~1) - a0;
                    for (int k = lane * 2; k < nw2; k += 64) cp_async4(&sp.slotw[buf][k >> 1], D.ent_slot + a0 + k);
                }
            }
        }
        if (PASS == LS_FIELD_SETUP) {
            const int v = blk * QA_LS_D + lane;
            if (lane < QA_LS_D && v < n) cp_async8(&sp.hb[buf][lane], D.h + v);
        }
        cp_async_commit();
    };
    int rp_cur, gm_cur, am_cur, rp_nxt, gm_nxt, am_nxt;
    load_meta(0, rp_cur, gm_cur, am_cur);
    load_meta(nblk > 1 ? 1 : 0, rp_nxt, gm_nxt, am_nxt);
    __syncwarp();
    stage_rows(0, 0, rp_cur);
    double nr[QA_LS_D];
    if (PASS == LS_PUSH) {
#pragma unroll
        for (int i = 0; i < QA_LS_D; ++i) nr[i] = __ldcg(fT + (int64_t)i * 32 + lane);
    }
    int parity = 0;

    const int nbeta = PASS == LS_FIELD_SETUP ? 1 : P.num_betas;
    const int nspb = PASS == LS_FIELD_SETUP ? 1 : P.sweeps_per_beta;
    for (; bi < nbeta; ++bi, swi = 0) {
        const double beta = PASS == LS_FIELD_SETUP ? 1.0 : (D.betas ? D.betas : P.betas)[bi];
        const double thr = 44.36142 / beta;
        for (; swi < nspb; ++swi) {
            uint32_t w = 0;
            bool dirty = false;
            for (int blk = 0; blk < nblk; ++blk) {
                const int v0 = blk * QA_LS_D;
                const int wi = v0 >> 5;
                const int sub = v0 & 31;
                if (sub == 0) {
                    w = pk[(int64_t)wi * rpad];
                    dirty = false;
                }
                int nb = blk + 1;
                if (nb == nblk) nb = 0;
                int nb2 = nb + 1;
                if (nb2 == nblk) nb2 = 0;
                // ---- pipeline: rows of the next block, metadata two blocks ahead, fields of the next block
                __syncwarp();
                stage_rows(parity ^ 1, nb, rp_nxt);
                int rp_nn, gm_nn, am_nn;
                load_meta(nb2, rp_nn, gm_nn, am_nn);
                if (lane <= QA_LS_D) sg.rowp[lane] = rp_cur;
                if (GROUPS != GK_NONE) {
                    if (lane < QA_LS_D) {
                        sg.gm[lane] = gm_cur;
                        sg.am[lane] = am_cur;
                    }
                }
                bool stale = false;
                bool blk_dirty = false;
                if (PASS == LS_PUSH) {
#pragma unroll
                    for (int i = 0; i < QA_LS_D; ++i) cur[i * 32] = nr[i];
#pragma unroll
                    for (int i = 0; i < QA_LS_D; ++i) nr[i] = __ldcg(fT + ((int64_t)nb * QA_LS_D + i) * 32 + lane);
                }
                cp_async_wait<1>();
                __syncwarp();
                const int eb = sg.rowp[0];
                const bool staged = (sg.rowp[QA_LS_D] - eb) <= QA_LS_CAP;
                const int *ej = sg.ej[parity];
                const double *eJ = sg.eJ[parity];
                bool tabled = false;
                const unsigned short *slots = nullptr;
                if (PASS == LS_FIELD_SETUP) {
                    if (tables && staged) {
                        const int nbw = __shfl_sync(FULL_MASK, rp_cur, QA_LS_D + 2) - __shfl_sync(FULL_MASK, rp_cur, QA_LS_D + 1);
                        tabled = !(nbw == 1 && sp.bw[parity][0] < 0);
                        if (tabled) {
                            // this lane's copy of every distinct spin word the block refers to (its own word stays in `w`)
                            for (int s = 0; s < nbw; s += 8) {
                                uint32_t t[8];
#pragma unroll
                                for (int q = 0; q < 8; ++q) t[q] = (s + q < nbw) ? pk[(int64_t)sp.bw[parity][s + q] * rpad] : 0u;
#pragma unroll
                                for (int q = 0; q < 8; ++q)
                                    if (s + q < nbw) c.words[(s + q) * 32] = t[q];
                            }
                            slots = reinterpret_cast<const unsigned short *>(sp.slotw[parity]) + (eb & 1);
                        }
                    }
                }

                for (int i = 0; i < QA_LS_D; ++i) {
                    const int v = v0 + i;
                    if (v >= n) break;  // uniform: padding variables
                    const int e0 = sg.rowp[i], e1 = sg.rowp[i + 1];
                    const bool up = (w >> (sub + i)) & 1u;
                    double fv;
                    if (PASS == LS_PUSH) {
                        fv = cur[i * 32];
                    } else {
                        // evaluate the local field from the spins: h_v + sum_j (+-J) in adjacency order
                        if (tabled) {
                            fv = sp.hb[parity][i];
#pragma unroll 4
                            for (int e = e0; e < e1; ++e) {
                                const int k = e - eb;
                                const unsigned sb = slots[k];             // low byte: slot (255 = own word), high byte: bit
                                const unsigned sl = sb & 255u;
                                const uint32_t wv = (sl == 255u) ? w : c.words[sl * 32];
                                const double J = eJ[k];
                                fv += ((wv >> (sb >> 8)) & 1u) ? J : -J;
                            }
                        } else {
                            fv = ls_field_direct(D, pk, rpad, v, e0, e1, wi, w);
                        }
                        __stcg(fT + (int64_t)v * 32 + lane, fv);
                        continue;
                    }
                    double dE = up ? -2.0 * fv : 2.0 * fv;
                    int g = -1, a = 0;
                    if (GROUPS != GK_NONE) {
                        g = sg.gm[i];
                        if (g >= 0) {
                            a = sg.am[i];
                            const long long *kb = c.kap_sh + kappa_words(GROUPS) * g;
                            dE = dE + group_flip_cost<GROUPS>(c.lam_sh[g], a, up, (long long)Mcol[g * QA_LS_TPB] + kb[0],
                                                              GROUPS == GK_INTERVAL ? kb[1] : 0, GROUPS == GK_INTERVAL ? kb[2] : 0);
                        }
                    }
                    const bool cand = active && !(dE >= thr);
                    if (!__any_sync(FULL_MASK, cand)) continue;
                    if (cand) st.cand++;
                    const bool acc = accept_test<PROP>(dE, cand, beta, thr, s0, s1, st);
                    const unsigned accm = __ballot_sync(FULL_MASK, acc);
                    if (accm == 0) continue;
                    if (acc) {
                        st.acc++;
                        st.nbr += (unsigned long long)(e1 - e0);
                    }
                    const double cf = up ? -2.0 : 2.0;  // f[j] += -2*s_v*J  <=> neal dE[j] += 4*s_v*J*s_j
                    double *fTl = fT + lane;
                    const int nbv0 = nb * QA_LS_D;
                    unsigned hit_next = 0;
                    // neighbours inside the staged block are updated in shared memory only (the block is written back
                    // once, below); all others get one predicated fire-and-forget reduction
                    if (staged) {
#pragma unroll 4
                        for (int k = e0 - eb; k < e1 - eb; ++k) {
                            const int j = ej[k];
                            const double d = cf * eJ[k];
                            const unsigned rel = (unsigned)(j - v0);          // uniform
                            if (rel < (unsigned)QA_LS_D) {
                                if (acc) cur[rel * 32] += d;
                                blk_dirty = true;
                            } else {
                                red_add_f64_if(fTl + (int64_t)j * 32, d, acc);
                                hit_next |= (unsigned)((unsigned)(j - nbv0) < (unsigned)QA_LS_D);
                            }
                        }
                    } else {
                        for (int e = e0; e < e1; ++e) {
                            const int j = __ldg(D.col + e);
                            const double d = cf * __ldg(D.val + e);
                            const unsigned rel = (unsigned)(j - v0);
                            if (rel < (unsigned)QA_LS_D) {
                                if (acc) cur[rel * 32] += d;
                                blk_dirty = true;
                            } else {
                                red_add_f64_if(fTl + (int64_t)j * 32, d, acc);
                                hit_next |= (unsigned)((unsigned)(j - nbv0) < (unsigned)QA_LS_D);
                            }
                        }
                    }
                    stale = stale || (hit_next != 0);  // prefetched registers of the next block are stale
                    if (acc) {
                        w ^= 1u << (sub + i);
                        dirty = true;
                        if (GROUPS != GK_NONE) {
                            if (g >= 0) Mcol[g * QA_LS_TPB] -= 2 * a * (up ? 1 : -1);
                        }
                    }
                }
                if (PASS == LS_PUSH) {
                    if (blk_dirty) {  // uniform: write the staged fields of this block back (coalesced 256 B rows)
#pragma unroll
                        for (int i = 0; i < QA_LS_D; ++i) __stcg(fT + ((int64_t)v0 + i) * 32 + lane, cur[i * 32]);
                    }
                    if (stale) {  // uniform; rare: a flip touched a variable of the prefetched block
#pragma unroll
                        for (int i = 0; i < QA_LS_D; ++i) nr[i] = __ldcg(fT + ((int64_t)nb * QA_LS_D + i) * 32 + lane);
                    }
                }
                if ((sub + QA_LS_D == 32 || blk == nblk - 1) && dirty) pk[(int64_t)wi * rpad] = w;
                rp_cur = rp_nxt; gm_cur = gm_nxt; am_cur = am_nxt;
                rp_nxt = rp_nn; gm_nxt = gm_nn; am_nxt = am_nn;
                parity ^= 1;
            }
        }
    }
    cp_async_wait<0>();
    __syncwarp();
}

template <GroupKind GROUPS, Proposal PROP>
__device__ void lockstep_tile(const LsCtx &c, unsigned long long &s0, unsigned long long &s1, LaneStats &st, int *error_flag) {
    const ProblemDesc &D = c.D;
    const int n = D.n;
    const int nch = D.nch;
    const int64_t rpad = D.rpad;
    const int64_t r = c.r;
    uint32_t *pk = D.packedT + r;  // r < rpad always: padding lanes own a scratch column of packedT

    // ---- pack this read's +-1 bytes (padding lanes and padding variables are +1)
    for (int wi = 0; wi < nch; ++wi) {
        uint32_t w = 0xffffffffu;
        if (c.active) {
            const int8_t *row = D.states + r * (int64_t)n + wi * 32;
            const int lim = min(32, n - wi * 32);
            for (int i = 0; i < lim; ++i) {
                const int s = row[i];
                if (s != 1 && s != -1) atomicExch(error_flag, QA_ERR_STATE);
                if (s < 0) w &= ~(1u << i);
            }
        }
        pk[(int64_t)wi * rpad] = w;
    }
    if (GROUPS != GK_NONE) {
        for (int g = 0; g < D.ngroups; ++g) c.Mcol[g * QA_LS_TPB] = 0;
        for (int wi = 0; wi < nch; ++wi) {
            const uint32_t w = pk[(int64_t)wi * rpad];
            for (int i = 0; i < 32; ++i) {
                const int v = wi * 32 + i;
                const int g = __ldg(D.grp + v);  // uniform
                if (g >= 0) {
                    const int a = __ldg(D.coef + v);
                    c.Mcol[g * QA_LS_TPB] += ((w >> i) & 1u) ? a : -a;
                }
            }
        }
    }
    int setup_bi = 0, setup_swi = 0, bi = 0, swi = 0;
    ls_sweeps<LS_FIELD_SETUP, GK_NONE, PROP>(c, setup_bi, setup_swi, s0, s1, st);  // local fields from the current spins
    ls_sweeps<LS_PUSH, GROUPS, PROP>(c, bi, swi, s0, s1, st);

    // ---- final spins back to the caller's +-1 rows
    if (c.active) {
        for (int wi = 0; wi < nch; ++wi) {
            const uint32_t w = pk[(int64_t)wi * rpad];
            int8_t *row = D.states + r * (int64_t)n + wi * 32;
            const int lim = min(32, n - wi * 32);
            for (int i = 0; i < lim; ++i) row[i] = ((w >> i) & 1u) ? 1 : -1;
        }
    }
}

__host__ __device__ inline size_t ls_smem_bytes(int max_groups, GroupKind gk) {
    size_t b = sizeof(double) * QA_LS_D * QA_LS_TPB;   // cur (push sweeps) / spin words (field set-up pass)
    b += (sizeof(LsStage) + sizeof(LsSetupStage)) * QA_LS_WPB;
    b += (sizeof(double) + kappa_words(gk) * sizeof(long long)) * (size_t)max_groups;
    b += sizeof(int) * (size_t)max_groups * QA_LS_TPB;
    return b;
}

template <GroupKind GROUPS, Proposal PROP>
__global__ void __launch_bounds__(QA_LS_TPB, 3) k_anneal_lockstep(AnnealParams P) {
    extern __shared__ __align__(16) unsigned char ls_smem[];
    // layout: [cur: D x TPB doubles, aliased by the spin words] [LsStage x warps] [LsSetupStage x warps] [lambda] [kappa] [M]
    // (interval groups: [kappa] is {kappa, lo, hi} per group)
    unsigned char *sp = ls_smem;
    double *cur_all = reinterpret_cast<double *>(sp);
    sp += sizeof(double) * QA_LS_D * QA_LS_TPB;
    LsStage *stages = reinterpret_cast<LsStage *>(sp);
    sp += sizeof(LsStage) * QA_LS_WPB;
    LsSetupStage *setup_stages = reinterpret_cast<LsSetupStage *>(sp);
    sp += sizeof(LsSetupStage) * QA_LS_WPB;
    uint32_t *words_all = reinterpret_cast<uint32_t *>(cur_all);
    double *lam_sh = reinterpret_cast<double *>(sp);
    sp += sizeof(double) * P.max_groups;
    long long *kap_sh = reinterpret_cast<long long *>(sp);
    sp += kappa_words(GROUPS) * sizeof(long long) * P.max_groups;
    int *M_all = reinterpret_cast<int *>(sp);
    __shared__ unsigned long long next_tile[QA_LS_WPB];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int64_t slot = (int64_t)blockIdx.x * QA_LS_WPB + wib;
    double *fT = P.fT_scratch ? P.fT_scratch + slot * P.fT_stride : nullptr;
    if (GROUPS != GK_NONE) stage_group_params<GROUPS>(P.descs[0], lam_sh, kap_sh);
    __syncthreads();
    LaneStats st = {0, 0, 0, 0, 0};
    for (;;) {
        if (lane == 0) next_tile[wib] = atomicAdd(P.counter, 1ull);
        __syncwarp();
        const int64_t tile = (int64_t)next_tile[wib];
        __syncwarp();
        if (tile >= P.total_tiles) break;
        const int p = (int)(tile / P.tiles_per_problem);
        const int64_t tip = tile % P.tiles_per_problem;
        const ProblemDesc D = P.descs[p];
        const int64_t r = tip * 32 + lane;
        const bool active = r < D.reads;
        const unsigned long long sd = active ? P.seeds[D.read_base + r] : 1ull;
        unsigned long long s0 = sd ? sd : ~0ull, s1 = 0;
        const LsCtx c = {D, P, r, active, fT, M_all + threadIdx.x, cur_all + wib * (QA_LS_D * 32) + lane, stages[wib],
                         setup_stages[wib], words_all + wib * (QA_LS_CAPW * 32) + lane, lam_sh, kap_sh};
        lockstep_tile<GROUPS, PROP>(c, s0, s1, st, P.error_flag);
    }
    flush_lane_stats(P, st);
}

// Block word tables for the field set-up pass: per block of QA_LS_D variables the distinct spin words (32 variables each)
// its CSR rows refer to, and per CSR entry the slot of its word in that list.  Built once per model on the host from the
// device-built CSR (a setup step, O(entries)); blocks that exceed the shared-memory capacities get a -1 sentinel.
int build_word_tables(qa_model *M) {
    if (M->tables_built) return QA_OK;
    qa_ctx *ctx = M->ctx;
    const int64_t entries = 2 * M->m_total;
    const int64_t rows_alloc = M->n_total + 64 + 1;
    std::vector<int32_t> rowptr(rows_alloc), col(std::max<int64_t>(entries, 1));
    QA_CUDA(cudaMemcpy(rowptr.data(), M->rowptr, rows_alloc * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (entries) QA_CUDA(cudaMemcpy(col.data(), M->col, entries * sizeof(int32_t), cudaMemcpyDeviceToHost));
    std::vector<int32_t> bw_ptr, bw_words;
    std::vector<unsigned short> slot(std::max<int64_t>(entries, 1) + 8, 255);
    std::vector<int64_t> blk_base(M->num_problems + 1, 0);
    bw_ptr.push_back(0);
    std::vector<int32_t> stamp, slot_of;
    for (int p = 0; p < M->num_problems; ++p) {
        const int64_t v_off = M->var_off[p];
        const int n = (int)(M->var_off[p + 1] - v_off);
        const int nch = (n + 31) / 32;
        const int nblk = nch * (32 / QA_LS_D);
        blk_base[p] = (int64_t)bw_ptr.size() - 1;
        stamp.assign(nch, -1);
        slot_of.assign(nch, 0);
        for (int b = 0; b < nblk; ++b) {
            const int v0 = b * QA_LS_D;
            const int64_t eb = rowptr[v_off + std::min(v0, n)];
            const int64_t ee = rowptr[v_off + std::min(v0 + QA_LS_D, n)];
            const size_t first = bw_words.size();
            const int own = v0 >> 5;
            bool ok = (ee - eb) <= QA_LS_CAP;
            for (int64_t e = eb; e < ee && ok; ++e) {
                const int wj = col[e] >> 5;
                const unsigned short bit = (unsigned short)((col[e] & 31) << 8);
                if (wj == own) { slot[e] = 255 | bit; continue; }
                if (stamp[wj] != b) {
                    if (bw_words.size() - first >= (size_t)QA_LS_CAPW) { ok = false; break; }
                    stamp[wj] = b;
                    slot_of[wj] = (int32_t)(bw_words.size() - first);
                    bw_words.push_back(wj);
                }
                slot[e] = (unsigned short)slot_of[wj] | bit;
            }
            if (!ok) {
                bw_words.resize(first);
                bw_words.push_back(-1);  // sentinel: block not tabled, kernel falls back to direct loads
                for (int w = 0; w < nch; ++w) if (stamp[w] == b) stamp[w] = -1;
            }
            bw_ptr.push_back((int32_t)bw_words.size());
        }
        // one extra pointer per problem so that the two-ahead metadata loads of the last block stay in range
    }
    blk_base[M->num_problems] = (int64_t)bw_ptr.size() - 1;
    for (int k = 0; k < 4; ++k) bw_ptr.push_back((int32_t)bw_words.size());
    if (bw_words.empty()) bw_words.push_back(-1);
    QA_CUDA(cudaMalloc((void **)&M->bw_ptr, bw_ptr.size() * sizeof(int32_t)));
    QA_CUDA(cudaMalloc((void **)&M->bw_words, bw_words.size() * sizeof(int32_t)));
    QA_CUDA(cudaMalloc((void **)&M->ent_slot, slot.size() * sizeof(unsigned short)));
    QA_CUDA(cudaMemcpyAsync(M->bw_ptr, bw_ptr.data(), bw_ptr.size() * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(M->bw_words, bw_words.data(), bw_words.size() * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(M->ent_slot, slot.data(), slot.size() * sizeof(unsigned short), cudaMemcpyHostToDevice, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int p = 0; p < M->num_problems; ++p) {
        M->descs[p].bw_ptr = M->bw_ptr + blk_base[p];
        M->descs[p].bw_words = M->bw_words;
        M->descs[p].ent_slot = M->ent_slot;
    }
    M->tables_built = true;
    return QA_OK;
}

}  // namespace

namespace qa {

int launch_lockstep(Launch &L) {
    qa_ctx *ctx = L.ctx;
    qa_model *M = L.M;
    AnnealParams &A = L.A;
    // lockstep: one warp = 32 reads of one problem
    const int tpp = (A.reads_per_problem + 31) / 32;
    const int64_t total_tiles = (int64_t)A.num_problems * tpp;
    const size_t smem = ls_smem_bytes(std::max(M->ngroups, 1), L.gk);
    // EQ32 models run the 64-bit instance: this kernel has no 32-bit one
    const void *fn = L.prop == PROP_GIBBS
                         ? (L.gk == GK_NONE ? (const void *)k_anneal_lockstep<GK_NONE, PROP_GIBBS>
                            : L.gk == GK_INTERVAL ? (const void *)k_anneal_lockstep<GK_INTERVAL, PROP_GIBBS>
                                                  : (const void *)k_anneal_lockstep<GK_EQ64, PROP_GIBBS>)
                         : (L.gk == GK_NONE ? (const void *)k_anneal_lockstep<GK_NONE, PROP_METROPOLIS>
                            : L.gk == GK_INTERVAL ? (const void *)k_anneal_lockstep<GK_INTERVAL, PROP_METROPOLIS>
                                                  : (const void *)k_anneal_lockstep<GK_EQ64, PROP_METROPOLIS>);
    QA_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int bps = 0;
    QA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessorWithFlags(&bps, fn, QA_LS_TPB, smem, cudaOccupancyDefault));
    if (bps < 1) return fail(QA_ERR_CUDA, "lockstep kernel does not fit on an SM");
    const int wpb = QA_LS_TPB / 32;
    int64_t grid = (int64_t)bps * ctx->num_sms;
    const int64_t need = (total_tiles + wpb - 1) / wpb;
    // spread few tiles over all SMs: prefer more blocks with idle warps to fewer full blocks
    if (need < grid) grid = std::min<int64_t>(grid, std::max<int64_t>(need, std::min<int64_t>(total_tiles, (int64_t)ctx->num_sms)));
    const int64_t fT_stride = (int64_t)M->nch_max * 32 * 32;
    {
        // read-interleaved local fields for the resident tiles
        size_t free_b = 0, total_b = 0;
        QA_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const size_t per_slot = (size_t)fT_stride * sizeof(double);
        const size_t budget = (size_t)((double)(free_b + ctx->fT.bytes) * 0.85);
        int64_t max_slots = (int64_t)(budget / per_slot);
        if (max_slots < wpb) return fail(QA_ERR_CUDA, "not enough device memory for one block of local fields");
        if (grid * wpb > max_slots) grid = max_slots / wpb;
        const int rc = ensure(ctx->fT, (size_t)grid * wpb * per_slot);
        if (rc) return rc;
        A.fT_scratch = (double *)ctx->fT.p;
    }
    const int rc = build_word_tables(M);  // the field set-up pass runs on these
    if (rc) return rc;
    QA_CUDA(cudaMemcpyAsync(M->d_descs, M->descs.data(), A.num_problems * sizeof(ProblemDesc), cudaMemcpyHostToDevice, ctx->stream));
    A.fT_stride = fT_stride;
    A.tiles_per_problem = tpp;
    A.total_tiles = total_tiles;
    A.max_groups = std::max(M->ngroups, 1);
    A.read_begin = 0;
    A.read_end = A.total_reads;
    QA_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    QA_CUDA(cudaMemsetAsync(A.counter, 0, sizeof(unsigned long long), ctx->stream));
    void *args[] = {&A};
    QA_CUDA(cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(QA_LS_TPB), args, smem, ctx->stream));
    QA_CUDA(cudaGetLastError());
    ctx->launches++;
    if (L.st) L.st->anneal_launches++;
    L.done = A.total_reads;
    return QA_OK;
}

}  // namespace qa
