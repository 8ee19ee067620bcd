// anneal_replay.cu -- k_anneal_replay (replay.cuh): the headline kernel; its host-side slab packer and launch.
#include "device_common.cuh"

using namespace qa;

namespace {

#include "replay.cuh"

}  // namespace

namespace qa {

// Coupling slabs of the replay kernel (replay.cuh): per block one contiguous {RpHdr, RpEntry[]} record.  Consecutive variables are packed greedily into blocks of at most RP_D variables inside
// ONE 16-variable half-word, RP_MAXBW foreign half-words and RP_CAP entry slots.  A row's entries are in REPLAY order --
// neighbours u > v ascending, then u < v ascending (stable, so duplicate couplers keep their adjacency order) -- split
// into the PRE part (u > v, then u < v0: known when the block starts; padded to rounds of 4 with
// zero-coupling entries) and the SEQ part (v0 <= u < v: decided inside the block).  The slab holds the pre parts of all
// rows, then the seq parts of all rows.  Built once per model on the host from the device-built CSR (a setup step,
// O(entries)).  Models whose blocks would hold fewer than 4 variables on average (dense rows, or sparse rows scattered over
// many half-words) leave rp_ok false and run on the other kernels.
//
// K-way section.  One-hot k-way models (models.cqm_model, dqm_model: variable v = cell * K + case) have cells of K aligned
// consecutive variables whose rows share one neighbour-cell list.  A cell CONFORMS when every row (i, p) has exactly the
// other K - 1 cases of its own cell as intra-cell neighbours, each once, and otherwise only neighbours (j, p) of its own case,
// each cell j once, with the same set of cells j and bitwise the same J_ij in all K rows.  Then row (i, p)'s pre part is
//     (i, p') for p' > p  |  (j, p) for j > i ascending  |  (j, p) for j < v0 / K ascending
// and the last two lists are the same for all K rows.  A block of whole conforming cells gets, behind its seq region, a
// section with one RpEntry per (cell, neighbour cell) in that order (J, slot, j*K << RP_J_SHIFT, and in bits 0-4 the shift of
// case K - 1; case p shifts 2 (K - 1 - p) more), counted against RP_CAP.  The batch phase then runs the K rows of a cell in
// lockstep (replay.cuh: rp_kway_batch): one entry and one slot word per neighbour cell for K independent fp64 chains.  The
// generic entries stay complete, so every other pass, and the intra-cell part of the batch phase, reads them as before.
// rowptr / col / val of one problem (rows local); fills conf[cell] and returns the number of variables in conforming cells.
static int64_t kway_conforming(int n, const int32_t *rowptr, const int32_t *col, const double *val, int K, std::vector<char> &conf) {
    const int ncell = n / K;
    conf.assign(ncell, 0);
    int64_t nvar = 0;
    std::vector<std::pair<int32_t, double>> first, cur;
    for (int i = 0; i < ncell; ++i) {
        const int b = i * K;
        bool ok = true;
        for (int p = 0; p < K && ok; ++p) {
            const int v = b + p;
            uint32_t intra = 0u;
            cur.clear();
            for (int64_t e = rowptr[v]; e < rowptr[v + 1] && ok; ++e) {
                const int j = col[e];
                if (j >= b && j < b + K) {
                    const uint32_t bit = 1u << (j - b);
                    ok = j != v && (intra & bit) == 0u;
                    intra |= bit;
                } else {
                    ok = j % K == p;
                    cur.push_back({j / K, val[e]});
                }
            }
            ok = ok && intra == (((1u << K) - 1u) & ~(1u << p));
            if (!ok) break;
            std::sort(cur.begin(), cur.end(), [](const std::pair<int32_t, double> &a, const std::pair<int32_t, double> &c) {
                return a.first < c.first;
            });
            for (size_t k = 1; k < cur.size() && ok; ++k) ok = cur[k].first != cur[k - 1].first;
            if (p == 0) {
                first = cur;
            } else {
                ok = ok && cur.size() == first.size();
                for (size_t k = 0; k < cur.size() && ok; ++k)
                    ok = cur[k].first == first[k].first && memcmp(&cur[k].second, &first[k].second, sizeof(double)) == 0;
            }
        }
        if (ok) {
            conf[i] = 1;
            nvar += K;
        }
    }
    return nvar;
}

// Pure host part of the slab construction (no CUDA calls: the CPU test-suite drives it through qa_debug_pack_slabs).
// rowptr holds global entry positions per global row (problem p's rows start at var_off[p]), col local neighbour indices.
bool pack_replay_slabs(int P, const int64_t *var_off, const int32_t *rowptr, const int32_t *col, const double *val, int ngroups,
                       const std::vector<int32_t> &hg, const std::vector<int32_t> &hc, int slots, RpPacked &out, bool kway) {
    const int RP_MAXBW = slots - 1;   // foreign half-words per block
    std::vector<uint32_t> &off = out.off;
    std::vector<unsigned char> &slabs = out.slabs;
    out.blk_base.assign(P, 0);
    out.nslabs.assign(P, 0);
    off.clear();
    slabs.clear();
    out.uniform = true;
    out.adj_sorted = true;
    out.kway_k = 0;
    out.kway_blocks = 0;
    struct Nb { int32_t j; double J; };
    struct Row { std::vector<Nb> later, early, seq; };   // u > v | u < v0 | v0 <= u < v
    std::vector<int32_t> stamp, slot_of;
    std::vector<Row> rows(RP_D);
    std::vector<size_t> hdr_pos;
    std::vector<int32_t> row_words;
    std::vector<char> conf, conf_k;
    for (int p = 0; p < P; ++p) {
        const int64_t v_off = var_off[p];
        const int n = (int)(var_off[p + 1] - v_off);
        if (n == 0 || n > RP_MAX_VARS) return false;   // the entry word holds a 20-bit neighbour index
        // the cell size under which the most variables conform (ties: the larger K, more independent chains)
        int K = 0;
        conf.clear();
        if (kway) {
            int64_t best = 0;
            for (int k : {2, 4, 8, 16}) {
                const int64_t c = kway_conforming(n, rowptr + v_off, col, val, k, conf_k);
                if (c > 0 && c >= best) {
                    best = c;
                    K = k;
                    conf.swap(conf_k);
                }
            }
        }
        const int nhw = (n + 15) / 16;
        const int npad = nhw * 16;
        out.blk_base[p] = (int64_t)off.size();
        hdr_pos.clear();
        stamp.assign(nhw, -1);
        slot_of.assign(nhw, 0);
        int b = 0;   // block (slab) index inside the problem; doubles as the stamp of the half-word -> slot map
        for (int v0 = 0; v0 < npad; ++b) {
            const int own = v0 >> 4;
            const int vmax = std::min(v0 + RP_D, (own + 1) * 16);   // never across a half-word
            RpHdr H;
            memset(&H, 0, sizeof(H));
            for (int i = 0; i < RP_D; ++i) H.ga[i] = 255;
            int nbw = 0, nv = 0;
            size_t slots_pre = 0, slots_seq = 0;
            for (int v = v0; v < vmax; ++v) {
                Row &R = rows[nv];
                R.later.clear();
                R.early.clear();
                R.seq.clear();
                if (v < n) {
                    for (int64_t e = rowptr[v_off + v]; e < rowptr[v_off + v + 1]; ++e) {
                        const Nb nb{col[e], val[e]};
                        if (nb.j > v) R.later.push_back(nb);
                        else if (nb.j < v0) R.early.push_back(nb);
                        else R.seq.push_back(nb);
                        if (e > rowptr[v_off + v] && col[e] < col[e - 1]) out.adj_sorted = false;
                    }
                }
                auto by_index = [](const Nb &a, const Nb &b2) { return a.j < b2.j; };
                std::stable_sort(R.later.begin(), R.later.end(), by_index);
                std::stable_sort(R.early.begin(), R.early.end(), by_index);
                std::stable_sort(R.seq.begin(), R.seq.end(), by_index);
                const size_t npre = R.later.size() + R.early.size();
                const size_t deg = npre + R.seq.size();
                if (R.seq.size() > 255 || deg > 0xffff) return false;
                // does the row still fit into this block?  (entry slots, and the foreign half-words it would add)
                row_words.clear();
                for (int part = 0; part < 2; ++part)
                    for (const Nb &nb : (part == 0 ? R.later : R.early)) {
                        const int wj = nb.j >> 4;
                        if (wj != own && stamp[wj] != b && std::find(row_words.begin(), row_words.end(), wj) == row_words.end())
                            row_words.push_back(wj);
                    }
                const size_t pre_slots = (npre + 3) / 4 * 4;
                const bool fits = slots_pre + slots_seq + pre_slots + R.seq.size() <= (size_t)RP_CAP &&
                                  nbw + (int)row_words.size() <= RP_MAXBW && pre_slots / 4 <= 255;
                if (!fits) {
                    if (nv == 0) return false;   // a single row exceeds the format: dense model
                    break;
                }
                for (int wj : row_words) {
                    stamp[wj] = b;
                    slot_of[wj] = nbw + 1;
                    H.bw[nbw++] = wj;
                }
                const int i = nv++;
                if (v < n && ngroups > 0 && hg[v] >= 0) {
                    if (hc[v] >= (1 << 23) || hc[v] <= -(1 << 23)) return false;  // coefficient does not fit the packed form
                    H.ga[i] = (int32_t)((uint32_t)hg[v] | ((uint32_t)hc[v] << 8));
                }
                H.rowa[i] = (uint32_t)(pre_slots / 4) | ((uint32_t)R.seq.size() << 8) | ((uint32_t)deg << 16);
                H.rowb[i] = (uint32_t)R.later.size() | ((uint32_t)npre << 16);
                slots_pre += pre_slots;
                slots_seq += R.seq.size();
            }
            // the block is closed: lay out the pre region (rows in order, padded), then the seq region
            std::vector<RpEntry> E;
            E.reserve(slots_pre + slots_seq);
            auto emit = [&](const Nb &nb) {
                const int wj = nb.j >> 4;
                RpEntry en;
                en.J = nb.J;
                en.zero = 0u;
                en.B = (uint32_t)(30 - 2 * (nb.j & 15)) | ((uint32_t)(wj == own ? 0 : slot_of[wj]) << 7) | ((uint32_t)nb.j << RP_J_SHIFT);
                E.push_back(en);
            };
            for (int i = 0; i < nv; ++i) {
                for (const Nb &nb : rows[i].later) emit(nb);
                for (const Nb &nb : rows[i].early) emit(nb);
                while (E.size() % 4) {
                    RpEntry en;
                    en.J = 0.0;          // fma(0, sigma, f) == f
                    en.zero = 0u;
                    en.B = 30u | ((uint32_t)(v0 + i) << RP_J_SHIFT);   // slot 0
                    E.push_back(en);
                }
            }
            H.seq_off = (int32_t)E.size();
            for (int i = 0; i < nv; ++i)
                for (const Nb &nb : rows[i].seq) emit(nb);
            // k-way section: whole conforming cells only
            bool kw = K > 0 && v0 % K == 0 && nv % K == 0 && v0 + nv <= n;
            for (int c = v0 / K; kw && c < (v0 + nv) / K; ++c) kw = conf[c] != 0;
            if (kw) {
                const size_t gen = E.size();
                const int c0 = v0 / K;
                for (int c = c0; c < (v0 + nv) / K; ++c) {
                    const Row &R = rows[(c - c0) * K];   // case 0: its later / early lists hold the neighbour cells in order
                    for (int part = 0; part < 2; ++part)
                        for (const Nb &nb : (part == 0 ? R.later : R.early)) {
                            if (nb.j >= c * K && nb.j < (c + 1) * K) continue;   // intra-cell
                            const int wj = nb.j >> 4;
                            RpEntry en;
                            en.J = nb.J;
                            en.zero = 0u;
                            en.B = (uint32_t)(30 - 2 * ((nb.j + K - 1) & 15)) | ((uint32_t)(wj == own ? 0 : slot_of[wj]) << 7) |
                                   ((uint32_t)nb.j << RP_J_SHIFT);
                            E.push_back(en);
                        }
                }
                if (E.size() <= (size_t)RP_CAP) {
                    H.kway = (int32_t)((uint32_t)gen | ((uint32_t)K << 16));
                    out.kway_blocks++;
                } else {
                    E.resize(gen);   // the section does not fit the stage: generic block
                }
            }
            H.nent = (int32_t)E.size();
            H.nbw = nbw;
            H.v0 = v0;
            H.nv = nv;
            out.uniform = out.uniform && nv == RP_D;
            if (slabs.size() / 16 > 0xfffffff0ull) return false;
            off.push_back((uint32_t)(slabs.size() / 16));
            hdr_pos.push_back(slabs.size());
            const unsigned char *hp = reinterpret_cast<const unsigned char *>(&H);
            slabs.insert(slabs.end(), hp, hp + sizeof(H));
            const unsigned char *ep = reinterpret_cast<const unsigned char *>(E.data());
            slabs.insert(slabs.end(), ep, ep + E.size() * sizeof(RpEntry));
            v0 += nv;
        }
        out.nslabs[p] = b;
        if (K > 0) out.kway_k = K;
        if ((int64_t)b * 4 > (int64_t)npad) return false;   // fewer than 4 variables per block on average: replaying does not pay
        // every slab also carries the half-word list of the next block (cyclic), staged while this block decides, and the slot
        // that holds the PREVIOUS block's half-word (the one word that staging cannot have up to date)
        for (size_t k = 0; k < hdr_pos.size(); ++k) {
            RpHdr *cur = reinterpret_cast<RpHdr *>(slabs.data() + hdr_pos[k]);
            const RpHdr *nxt = reinterpret_cast<const RpHdr *>(slabs.data() + hdr_pos[(k + 1) % hdr_pos.size()]);
            cur->nbw_next = nxt->nbw;
            memcpy(cur->bw_next, nxt->bw, sizeof(cur->bw_next));
            cur->prev_slot = 0;
            if (k > 0) {
                const RpHdr *prv = reinterpret_cast<const RpHdr *>(slabs.data() + hdr_pos[k - 1]);
                const int phw = prv->v0 >> 4;
                if (phw != (cur->v0 >> 4))
                    for (int s = 0; s < cur->nbw; ++s)
                        if (cur->bw[s] == phw) cur->prev_slot = s + 1;
            }
        }
    }
    off.push_back((uint32_t)(slabs.size() / 16));
    return !slabs.empty();
}

int build_replay_tables(qa_model *M) {
    if (M->rp_built) return QA_OK;
    qa_ctx *ctx = M->ctx;
    M->rp_built = true;
    M->rp_ok = false;
    const int64_t entries = 2 * M->m_total;
    const int64_t rows_alloc = M->n_total + 64 + 1;
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    std::vector<int32_t> rowptr(rows_alloc), col(std::max<int64_t>(entries, 1));
    std::vector<double> val(std::max<int64_t>(entries, 1));
    QA_CUDA(cudaMemcpy(rowptr.data(), M->rowptr, rows_alloc * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (entries) {
        QA_CUDA(cudaMemcpy(col.data(), M->col, entries * sizeof(int32_t), cudaMemcpyDeviceToHost));
        QA_CUDA(cudaMemcpy(val.data(), M->val, entries * sizeof(double), cudaMemcpyDeviceToHost));
    }
    std::vector<int32_t> hg, hc;
    if (M->ngroups > 0) {
        const int64_t npad = (int64_t)M->descs[0].nch * 32;
        hg.resize(npad);
        hc.resize(npad);
        QA_CUDA(cudaMemcpy(hg.data(), M->grp, npad * sizeof(int32_t), cudaMemcpyDeviceToHost));
        QA_CUDA(cudaMemcpy(hc.data(), M->coef, npad * sizeof(int32_t), cudaMemcpyDeviceToHost));
    }
    RpPacked pk;
    // 32 half-word slots per warp when the blocks fit (4 KB per warp), else 64 (scattered neighbourhoods)
    const bool kw = ctx->replay_kway != 0;
    M->rp_slots = 32;
    if (!pack_replay_slabs(M->num_problems, M->var_off.data(), rowptr.data(), col.data(), val.data(), M->ngroups, hg, hc, 32, pk, kw)) {
        M->rp_slots = 64;
        if (!pack_replay_slabs(M->num_problems, M->var_off.data(), rowptr.data(), col.data(), val.data(), M->ngroups, hg, hc, 64, pk, kw))
            return QA_OK;   // the model does not fit the slab format: rp_ok stays false
    }
    M->rp_kway_k = pk.kway_blocks > 0 ? pk.kway_k : 0;
    M->rp_kway_blocks = pk.kway_blocks;
    const std::vector<uint32_t> &off = pk.off;
    const std::vector<unsigned char> &slabs = pk.slabs;
    const std::vector<int64_t> &blk_base = pk.blk_base;
    const std::vector<int32_t> &nslabs = pk.nslabs;
    const bool uniform = pk.uniform;
    M->rp_adj_sorted = pk.adj_sorted;
    QA_CUDA(cudaMalloc((void **)&M->rp_slabs, slabs.size()));
    QA_CUDA(cudaMalloc((void **)&M->rp_off, off.size() * sizeof(uint32_t)));
    QA_CUDA(cudaMemcpyAsync(M->rp_slabs, slabs.data(), slabs.size(), cudaMemcpyHostToDevice, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(M->rp_off, off.data(), off.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int p = 0; p < M->num_problems; ++p) {
        M->descs[p].rp_slabs = M->rp_slabs;
        M->descs[p].rp_off = M->rp_off + blk_base[p];
        M->descs[p].rp_nslabs = nslabs[p];
    }
    M->rp_ok = true;
    M->rp_uniform = uniform;
    return QA_OK;
}

// the instance for the acceptance rule, the model's group kind and slot count; models with k-way blocks run the one with the
// k-way batch phase.  The Gibbs instances live in their own translation unit (anneal_replay_gibbs.cu): this one's module
// holds exactly the Metropolis instances, and the two compile in parallel.
static const void *replay_kernel(const qa_model *M, GroupKind gk, Proposal prop) {
    return prop == PROP_GIBBS ? replay_gibbs_kernel(M, gk) : replay_instance<PROP_METROPOLIS>(M, gk);
}

int launch_replay(Launch &L) {
    qa_ctx *ctx = L.ctx;
    qa_model *M = L.M;
    AnnealParams &A = L.A;
    const int P = A.num_problems;
    // replay: one CTA = `nw` consecutive 32-read tiles of one problem, coupling slabs shared through a TMA ring
    const int tpp = (A.reads_per_problem + 31) / 32;
    const int mg = std::max(M->ngroups, 1);
    int nw = ctx->replay_warps;
    if (nw < 1 || nw > RP_MAX_WARPS) {
        nw = 1;
        while (nw < RP_MAX_WARPS && nw < tpp) nw *= 2;
        while (nw > 1 && rp_smem_bytes(nw, mg, ctx->rp_smem_base, M->rp_slots, L.gk) > (size_t)(226 * 1024 / RP_MIN_CTAS - 1024)) nw /= 2;   // RP_MIN_CTAS CTAs per SM
        // less than one full wave of 8-warp CTAs: 4-warp CTAs (3 per SM) balance the SMs better -- measured on config 3
        // (profiles/r2_probe_strong_scaling_read_counts.log): 50 000 reads 7.4e10 against 6.8e10 with 8 warps, 25 000 and 12 500
        // reads within 1 % of the best choice; 1- and 2-warp CTAs are residency-limited by the slab ring's shared memory
        if ((int64_t)P * tpp < (int64_t)RP_MIN_CTAS * ctx->num_sms * RP_MAX_WARPS && nw > 4) nw = 4;
        // very few tiles: prefer narrower CTAs on every SM to wide CTAs on some of them
        while (nw > 1 && (int64_t)P * ((tpp + nw - 1) / nw) < (int64_t)ctx->num_sms) nw /= 2;
    }
    const int64_t gpp = (tpp + nw - 1) / nw;
    const int64_t total_items = (int64_t)P * gpp;
    size_t smem = rp_smem_bytes(nw, mg, ctx->rp_smem_base, M->rp_slots, L.gk);
    const void *fn = replay_kernel(M, L.gk, L.prop);
    QA_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int bps = 0;
    QA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessorWithFlags(&bps, fn, nw * 32, smem, cudaOccupancyDefault));
    if (bps < 1) return fail(QA_ERR_CUDA, "replay kernel does not fit on an SM");
    int64_t grid = std::min<int64_t>((int64_t)bps * ctx->num_sms, total_items);
    const int64_t fT_stride = (int64_t)M->nch_max * 32 * 32;
    const int64_t sf_stride = (int64_t)M->nch_max * 2 * 32;
    {
        size_t free_b = 0, total_b = 0;
        QA_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const size_t per_slot = (size_t)fT_stride * sizeof(double) + (size_t)sf_stride * sizeof(uint32_t);
        const size_t budget = (size_t)((double)(free_b + ctx->fT.bytes + ctx->sf.bytes) * 0.9);
        const int64_t max_slots = (int64_t)(budget / per_slot);
        if (max_slots < nw) return fail(QA_ERR_CUDA, "not enough device memory for one CTA of local fields");
        if (grid * nw > max_slots) grid = max_slots / nw;
        int rc = ensure(ctx->fT, (size_t)grid * nw * fT_stride * sizeof(double) + 4096);   // + the look-ahead rows of the last slot
        if (!rc) rc = ensure(ctx->sf, (size_t)grid * nw * sf_stride * sizeof(uint32_t));
        if (rc) return rc;
    }
    A.fT_scratch = (double *)ctx->fT.p;
    A.fT_stride = fT_stride;
    A.sf_scratch = ctx->sf.p;
    A.sf_stride = sf_stride;
    A.tiles_per_problem = tpp;
    A.groups_per_problem = gpp;
    A.total_items = total_items;
    A.max_groups = mg;
    A.switch_permille = ctx->replay_switch_permille;
    A.rp_slab_init = M->rp_adj_sorted ? 1 : 0;
    A.read_begin = 0;
    A.read_end = A.total_reads;
    if (L.interrupt) {
        *ctx->h_iflag = 0;
        A.interrupt_flag = ctx->d_iflag;
    }
    QA_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    QA_CUDA(cudaMemsetAsync(A.counter, 0, sizeof(unsigned long long), ctx->stream));
    void *args[] = {&A};
    QA_CUDA(cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(nw * 32), args, smem, ctx->stream));
    QA_CUDA(cudaGetLastError());
    ctx->launches++;
    {   // the kernel leaves at once if dynamic shared memory does not start where the layout assumed: relaunch with the real base
        int fl[2] = {0, 0};
        QA_CUDA(cudaMemcpyAsync(fl, ctx->d_flag, sizeof(fl), cudaMemcpyDeviceToHost, ctx->stream));
        if (!ctx->rp_base_checked) {   // first launch of this context only (costs a synchronisation)
            QA_CUDA(cudaStreamSynchronize(ctx->stream));
            if (fl[0] == QA_ERR_SMEM_BASE) {
                ctx->rp_smem_base = (unsigned)fl[1];
                smem = rp_smem_bytes(nw, mg, ctx->rp_smem_base, M->rp_slots, L.gk);
                QA_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                QA_CUDA(cudaMemsetAsync(ctx->d_flag, 0, 2 * sizeof(int), ctx->stream));
                QA_CUDA(cudaMemsetAsync(A.counter, 0, sizeof(unsigned long long), ctx->stream));
                QA_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
                QA_CUDA(cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(nw * 32), args, smem, ctx->stream));
                QA_CUDA(cudaGetLastError());
                ctx->launches++;
            }
            ctx->rp_base_checked = true;
        }
    }
    if (L.st) L.st->anneal_launches++;
    L.done = A.total_reads;
    if (L.interrupt) {   // poll the callback while the launch runs; CTAs stop pulling work once the flag is up
        QA_CUDA(cudaEventRecord(ctx->ev[3], ctx->stream));
        for (;;) {
            const cudaError_t q = cudaEventQuery(ctx->ev[3]);
            if (q == cudaSuccess) break;
            if (q != cudaErrorNotReady) return fail(QA_ERR_CUDA, std::string("replay kernel: ") + cudaGetErrorString(q));
            if (!L.interrupted && L.interrupt(L.iuser)) {
                *reinterpret_cast<volatile int *>(ctx->h_iflag) = 1;
                L.interrupted = true;
            }
            struct timespec ts = {0, 200000};
            nanosleep(&ts, nullptr);
        }
        if (L.interrupted) {   // groups are handed out in read order: the first `pulled` groups are complete
            unsigned long long pulled = 0;
            QA_CUDA(cudaMemcpyAsync(&pulled, A.counter, sizeof(pulled), cudaMemcpyDeviceToHost, ctx->stream));
            QA_CUDA(cudaStreamSynchronize(ctx->stream));
            L.done = std::min<int64_t>(A.total_reads, (int64_t)std::min<unsigned long long>(pulled, (unsigned long long)total_items) * nw * 32);
        }
    }
    return QA_OK;
}

}  // namespace qa
