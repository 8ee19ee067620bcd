// replay.cuh -- k_anneal_replay: bit-exact reference-order annealing with DEFERRED neighbour updates.
// Included by qanneal.cu (needs ProblemDesc, AnnealParams, LaneStats, ls_accept, red_add_f64_if).
//
// neal (cpu_sa.cpp simulated_annealing_run, SURVEY.md row a8) pushes every accepted flip of u into the flip energies of
// all neighbours j at once.  On a GPU with 32 reads per warp that is a random 8-byte read-modify-write per (flip, neighbour)
// on a field matrix far larger than L2; measured on B200 (tools/ubench_update.cu) the memory system tops out at
// 1.5-2.8e10 attempts/s for every acceptance rate >= 5 % -- the lockstep push kernel already sits at that ceiling.
//
// This kernel keeps the SAME arithmetic but changes when it happens.  Per read it stores
//     f[v]  the local field h_v + sum_j J_vj s_j as of the LAST VISIT of v      (fp64, read-interleaved f[v][lane])
//     D[v]  "spin is down", F[v] "v flipped at its last visit"   (bit-packed per 16 variables: one word per half-word and
//           lane, bit 2i+1 = D, bit 2i = F of variable 16*hw + i)
// Between two visits of v every neighbour u is visited exactly once, so the updates neal would have pushed into f[v] are
//     + 2 s_u J_uv   for the flagged neighbours u > v (flipped later in the previous sweep), ascending u, then
//     + 2 s_u J_uv   for the flagged neighbours u < v (flipped earlier in this sweep),       ascending u
// -- the same fp64 additions in the same order (s_u is the spin after the flip; a neighbour cannot flip twice in that
// window).  Replaying them at the visit gives bit-identical fields, decisions, RNG draws and final states, but the memory
// traffic becomes sequential and fully coalesced: 8 B of field per attempt (+8 B when it changed) plus the {S|F} words of
// the neighbour cells, instead of 16 B x 4 (sector granularity) per (flip, neighbour).
// When flips become rare the cost balance inverts (a replay touches every neighbour of every variable, a push only the
// neighbours of accepted flips), so once the CTA-wide acceptance of a sweep drops below P.switch_permille the tile runs one
// catch-up pass (pending u > v updates only) and finishes the schedule pushing, as neal does.  Both forms are exact, so
// the hand-over point does not influence the result.
// The derivation does not depend on the acceptance rule, so it holds for dwave-samplers' Gibbs rule (PROP_GIBBS) as well: each
// variable is still visited once per sweep, so a neighbour still cannot flip twice between two visits; a field of +-0 is still
// unobservable, because Gibbs compares dE with +-thr (never with the sign of zero) and exp(+-0) = 1; and the hand-over reads
// acceptance counts only.
//
// Blocks.  The host packs consecutive variables greedily into blocks (at most RP_D = 16 variables inside ONE 16-variable
// half-word, RP_MAXBW foreign half-words, RP_CAP entry slots) and builds one contiguous slab {RpHdr, RpEntry[]} per block.
// A row's entries are split where the data dependence is:
//     pre part   neighbours u > v (ascending) then neighbours u < v0 (ascending): everything that is known when the block
//                starts -- padded to rounds of 4 entries (padding: flag mask 0)
//     seq part   neighbours v0 <= u < v (ascending): decided inside this block, read from the REGISTER that holds the
//                block's own {S|F} word
// so a block runs in two phases: a BATCH phase that streams the pre parts of all rows (no dependence on this block's
// decisions: table loads run one round ahead, 6 instructions per entry: LDS.128 entry, LOP3 slot address, LDS word, SHF,
// LOP3, DFMA -- see rp_add_entry) and leaves the partial sums in shared memory, and a SEQUENTIAL
// phase (seq entries + neal's Metropolis decision per variable).  The foreign half-words of block b+1 are copied into the
// warp's slot region by cp.async while block b is in its sequential phase (which does not read the slots); the only word
// that can be stale in that copy -- block b's own -- is patched from the register when block b+1 starts.
//
// All warps of a CTA walk the blocks together; slabs are brought into a 4-stage shared-memory ring with cp.async.bulk
// (TMA 1-D) completing on mbarriers, and released by one mbarrier arrive per warp -- no __syncthreads in the sweep.  There
// is no fixed producer: whichever warp first gets within RP_DIST blocks of a slab that has not been requested yet claims it
// (one shared-memory CAS) and issues the copy.
#pragma once

constexpr int RP_D = 16;                      // variables per block, at most (= one half-word of spins)
constexpr int RP_SLOTS = 64;                  // half-word slots per warp, at most: slot 0 = the block's own half-word.  Two kernel
                                              // instances: 32 slots (4 KB per warp; local graphs such as config 3) and 64 slots
                                              // (8 KB; scattered neighbourhoods such as the 1000-cell sub-problems of config 4)
#ifndef RP_CAP
#define RP_CAP 448     // entry slots per slab (pre parts in rounds of 4, then the seq parts)
#endif
#ifndef RP_STAGES
#define RP_STAGES 4   // ring stages: stage = g % RP_STAGES, phase = (g / RP_STAGES) & 1 for the running block counter g
#endif
#ifndef RP_LA
#define RP_LA 4     // local fields are loaded this many rows ahead of their use in the batch phase
#endif
#ifndef RP_PF_DIST
#define RP_PF_DIST 32   // L2 run-ahead of the field rows, in variables
#endif
#ifndef RP_DIST
#define RP_DIST 2     // slabs are requested this many blocks ahead of the first warp that will need them (< RP_STAGES)
#endif
static_assert(RP_DIST < RP_STAGES, "the ring must hold the block in use and the requested ones");
// Development build (-DQA_RP_PROFILE): clock64() cycles summed per warp into the QA_NDEBUG counters behind the read counter,
// printed by the host after every sampling call.  Slots: 0 set-up pass, 1 slab wait, 2 stage wait, 3 prologue (block start
// to batch phase, waits excluded), 4 batch phase, 5 sequential phase, 6 replay passes, 7 catch-up and push passes.
#ifdef QA_RP_PROFILE
#define RP_CLK(t) const long long t = clock64()
#define RP_PROF(k, d) (c.prof[k] += (d))
#else
#define RP_CLK(t)
#define RP_PROF(k, d)
#endif
constexpr int RP_PS_BYTES = RP_D * 32 * 8;       // per warp: partial sums [row][lane] (push phase: the block's fields)
__host__ __device__ constexpr int rp_sf_bytes(int slots) { return slots * 32 * 4; }   // per warp: [slot][lane] words, aligned to its size
__host__ __device__ constexpr uint32_t rp_slot_mask(int slots) { return (uint32_t)(slots - 1) << 7; }
#ifndef RP_MAX_WARPS
#define RP_MAX_WARPS 8    // warps per CTA (upper bound; the host picks a power of two)
#endif
#ifndef RP_MIN_CTAS
#define RP_MIN_CTAS 2     // resident CTAs per SM the register allocation is bounded for
#endif

struct alignas(16) RpHdr {
    int32_t nent;               // entry slots in this slab (pre region incl. padding, seq region, k-way section)
    int32_t nbw;                // distinct neighbour half-words other than the block's own
    int32_t v0;                 // first variable of the block
    int32_t nv;                 // variables in the block (1 .. RP_D; v0 .. v0+nv-1 lie in one 16-variable half-word)
    int32_t prev_slot;          // slot holding the PREVIOUS block's half-word (0: not referenced / same half-word / first block)
    int32_t seq_off;            // entry slot where the seq region starts (multiple of 4)
    int32_t nbw_next;           // the half-word list of the NEXT block (cyclic): staged while this block decides
    int32_t kway;               // k-way section (anneal_replay.cu): entry slot where it starts (bits 0-15) | K << 16; 0: none
    uint32_t rowa[RP_D];        // pre rounds (bits 0-7) | seq entries (8-15) | degree (16-31)
    uint32_t rowb[RP_D];        // later entries u > v (0-15) | pre entries without padding (16-31)
    int32_t ga[RP_D];           // group (low byte, 255: none) | coefficient << 8
    int32_t bw[RP_SLOTS];       // neighbour half-word indices, slot s+1 holds half-word bw[s]
    int32_t bw_next[RP_SLOTS];
};
static_assert(sizeof(RpHdr) % 16 == 0, "slab header layout");
constexpr uint32_t RP_H_NBW = offsetof(RpHdr, nbw), RP_H_V0 = offsetof(RpHdr, v0), RP_H_NV = offsetof(RpHdr, nv),
                   RP_H_PREV = offsetof(RpHdr, prev_slot), RP_H_SEQ = offsetof(RpHdr, seq_off), RP_H_KW = offsetof(RpHdr, kway),
                   RP_H_ROWA = offsetof(RpHdr, rowa), RP_H_ROWB = offsetof(RpHdr, rowb), RP_H_GA = offsetof(RpHdr, ga),
                   RP_H_BW = offsetof(RpHdr, bw), RP_H_NBWN = offsetof(RpHdr, nbw_next), RP_H_BWN = offsetof(RpHdr, bw_next);
struct __align__(16) RpEntry {
    double J;      // the coupling (0.0 for padding entries: fma(0, sigma, f) == f)
    uint32_t zero; // low word of sigma: the entry's LDS.128 delivers the register pair {0, B} the DFMA multiplies by
    uint32_t B;    // bits 0-4: 30 - 2 * (j & 15) (left shift that brings the neighbour's D bit to bit 31, its F bit to bit 30);
                   // bits 7-12: slot; bits 13-31: neighbour j (local variable index, < 2^19)
};
constexpr int RP_MAX_VARS = 1 << 19;
constexpr int RP_J_SHIFT = 13;
constexpr int RP_STAGE_BYTES = (int)sizeof(RpHdr) + (RP_CAP + 8) * (int)sizeof(RpEntry);   // + two rounds of read-ahead slack
static_assert(RP_STAGE_BYTES % 16 == 0, "stage alignment");

// ---- mbarrier / TMA 1-D primitives -----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// shared-memory accesses by explicit address (volatile: kept in program order among themselves and after the barrier waits)
__device__ __forceinline__ int4 lds_v4(uint32_t a) {
    int4 r;
    asm volatile("ld.volatile.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(a));
    return r;
}
__device__ __forceinline__ uint32_t lds_vu32(uint32_t a) {
    uint32_t r;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(r) : "r"(a));
    return r;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t r;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(a));
    return r;
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t x) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(x) : "memory");
}
__device__ __forceinline__ double lds_f64(uint32_t a) {
    double r;
    asm volatile("ld.volatile.shared.f64 %0, [%1];" : "=d"(r) : "r"(a));
    return r;
}
__device__ __forceinline__ void sts_f64(uint32_t a, double v) {
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory");
}
// 16-byte asynchronous copy global (L2) -> shared (LDGSTS.BYPASS): no register staging, completion by cp.async.wait_all
__device__ __forceinline__ void rp_cp_async16(uint32_t dst_s, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_s), "l"(src) : "memory");
}
__device__ __forceinline__ void rp_cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// One replay entry: f += (neighbour up ? +2J : -2J) on the lanes whose copy of the neighbour's word has the F bit set.
// One shift brings the neighbour's (D, F) bit pair to bits (31, 30); those two bits ARE the high word of a double sigma:
// sign = D, exponent field 0x400 or 0 -> sigma = +-2.0 (flagged) or +-0.0 (not flagged).  fma(J, sigma, f) has an exact
// product and ONE rounding: bit-identical to neal's  f += 4 s J s_j / (-2 s)  addition of +-2J, and the exact identity for
// an unflagged neighbour (a zero field may change its sign, which no decision can observe: dE = -+2f is compared with
// >= thr and <= 0 only).  SHF, LOP3, DFMA -- the DFMA chain is the only serial dependence of a replay.
__device__ __forceinline__ void rp_add_entry(double &f, const int4 &q, uint32_t w) {
    const uint32_t x = w << ((uint32_t)q.w & 31u);
    f = fma(__hiloint2double(q.y, q.x), __hiloint2double((int)(x & 0xC0000000u), q.z), f);   // q.z == 0
}

// Batch phase of a block with a k-way section (anneal_replay.cu): whole cells of K one-hot cases whose rows share one
// neighbour-cell list.  The rows of a cell run in lockstep in chunks of KR = min(K, 8) rows (two chunks per cell for K = 16),
// one accumulator per row: first each row's intra-cell later cases (its first entries in the generic pre region, read against
// the register W, which holds the block's own half-word), then the section's neighbour cells: per neighbour cell one entry and
// one slot word, loaded a step ahead, and per row SHF, LOP3, DFMA into its own chain.  Row p of a chunk adds the same terms in
// the same order as its generic pre part, with no padding entries: the partial sums are bit-identical.  The fields of the next
// chunk are copied (cp.async) into its partial-sum rows while this one runs; those of the first rows come from the block
// look-ahead fq.  Returns the chg mask (partial sum != field), as the generic batch phase does.
template <int KR, int SLOTS>
__device__ __forceinline__ uint32_t rp_kway_batch(uint32_t hdr, uint32_t ent, uint32_t kw, int nv, const double *fB,
                                                  const double (&fq)[RP_LA], uint32_t W, uint32_t sfb, uint32_t psb) {
    const int K = (int)(kw >> 16);
    uint32_t sec = ent + (kw & 0xffffu) * 16u;   // the current cell's neighbour-cell entries
    uint32_t a = ent;                            // the current row's generic pre part
    uint32_t chg = 0u;
    const uint32_t lane = threadIdx.x & 31u;
    // the warp's copy of row r (256 B): lanes 16 h .. 16 h + 15 copy 16 B each of row r + h
    const uint32_t cp_dst = psb - 8u * lane + (lane >> 4) * 256u + (lane & 15u) * 16u;
    const double *const cp_src = fB - lane + (lane >> 4) * 32 + (lane & 15u) * 2;
    double acc[KR];
#pragma unroll
    for (int k = 0; k < KR; ++k) acc[k] = k < RP_LA ? fq[k] : __ldcg(fB + k * 32);
#pragma unroll
    for (int k = 0; k < KR; ++k) sts_f64(psb + (uint32_t)k * 256u, acc[k]);   // the fields, for the chg test
#pragma unroll 1
    for (int r0 = 0; r0 < nv; r0 += KR) {
        if (r0 > 0) {   // this chunk's fields, copied into its partial-sum rows while the previous chunk ran
            rp_cp_async_wait_all();
            __syncwarp();
#pragma unroll
            for (int k = 0; k < KR; ++k) acc[k] = lds_f64(psb + (uint32_t)(r0 + k) * 256u);
        }
        if (r0 + KR < nv) {   // the next chunk's fields -> its partial-sum rows (no register staging)
#pragma unroll
            for (int k = 0; k < KR; k += 2) rp_cp_async16(cp_dst + (uint32_t)(r0 + KR + k) * 256u, cp_src + (r0 + KR + k) * 32);
        }
        // intra-cell later cases: row k of the chunk has xs + KR - 1 - k of them (xs = 8 for the first chunk of a 16-way cell)
        const int xs = K - KR - r0 % K;
        uint32_t ar[KR];
#pragma unroll
        for (int k = 0; k < KR; ++k) {
            ar[k] = a;
            a += (lds_u32(hdr + RP_H_ROWA + 4u * (uint32_t)(r0 + k)) & 255u) * 64u;
        }
#pragma unroll 1
        for (int m = 0; m < xs; ++m) {
#pragma unroll
            for (int k = 0; k < KR; ++k) rp_add_entry(acc[k], lds_v4(ar[k] + 16u * (uint32_t)m), W);
        }
#pragma unroll
        for (int m = 0; m < KR - 1; ++m) {
#pragma unroll
            for (int k = 0; k < KR - 1 - m; ++k) rp_add_entry(acc[k], lds_v4(ar[k] + 16u * (uint32_t)(xs + m)), W);
        }
        // neighbour cells: j > i ascending, then j < v0 / K ascending; the count is the pre part of the cell's last case
        const int cl = r0 - r0 % K + K - 1;
        const int nn = (int)(lds_u32(hdr + RP_H_ROWB + 4u * (uint32_t)cl) >> 16);
        const uint32_t xsh = 2u * (uint32_t)xs;
        auto step = [&](const int4 &q, uint32_t w) {
            const uint32_t x = (w << ((uint32_t)q.w & 31u)) << xsh;   // case KR - 1 of the chunk at bits (31, 30)
            const double J = __hiloint2double(q.y, q.x);
#pragma unroll
            for (int k = 0; k < KR; ++k)
                acc[k] = fma(J, __hiloint2double((int)((x << (2 * (KR - 1 - k))) & 0xC0000000u), q.z), acc[k]);   // q.z == 0
        };
        uint32_t e = sec;
        int4 qa = lds_v4(e);
        uint32_t wa = lds_vu32(((uint32_t)qa.w & rp_slot_mask(SLOTS)) | sfb);
        int t = 0;
#pragma unroll 1
        for (; t + 2 <= nn; t += 2) {   // reads up to two entries past the section: inside the stage's read-ahead slack
            const int4 qb = lds_v4(e + 16u);
            const uint32_t wb = lds_vu32(((uint32_t)qb.w & rp_slot_mask(SLOTS)) | sfb);
            step(qa, wa);
            qa = lds_v4(e + 32u);
            wa = lds_vu32(((uint32_t)qa.w & rp_slot_mask(SLOTS)) | sfb);
            step(qb, wb);
            e += 32u;
        }
        if (t < nn) step(qa, wa);
        if ((r0 + KR) % K == 0) sec += (uint32_t)nn * 16u;   // the cell is complete
#pragma unroll
        for (int k = 0; k < KR; ++k) {
            const uint32_t pa = psb + (uint32_t)(r0 + k) * 256u;
            if (acc[k] != lds_f64(pa)) chg |= 1u << (r0 + k);
            sts_f64(pa, acc[k]);
        }
    }
    return chg;
}

struct RpCtx {
    // ring (CTA-shared)
    uint32_t full_s, empty_s, stage_s;   // shared addresses: full[0], empty[0] (8 B apart), stage 0
    unsigned *issued;                    // shared: running index of the next slab to request
    const unsigned char *slabs;          // global slab storage
    const uint32_t *off;                 // [nblk + 1] slab offsets of this problem, in 16-byte units
    uint32_t gb;                         // running index of the next block this warp consumes
    // per lane
    double *fT;                          // f[v][lane], this lane's column
    uint32_t *SF;                        // {S | F << 16}[half-word][lane], this lane's column
    uint32_t sfb_s;                      // shared address of this lane's column in the warp's slot region (4 KB aligned + 4 * lane)
    uint32_t psb_s;                      // shared address of this lane's column in the warp's partial-sum region
    int *Mcol;
    int mstride;
    const double *lam;
    const long long *kap;
    const double *h;                     // linear biases of the current problem (field set-up pass)
    unsigned long long s0, s1;
    LaneStats st;
    bool active;
    int n, nblk, npad;
#ifdef QA_RP_PROFILE
    long long prof[QA_NDEBUG];
#endif
};

// lane 0 of any warp: request every slab up to running index `tgt` that nobody has requested yet and whose ring stage is
// free.  `blk` is the block the calling warp is about to consume (running index c.gb); slabs follow the cyclic block order
// of the passes.  NON-BLOCKING: a stage still in use by a slower warp ends the attempt (a warp that blocked here would couple
// the fastest warp of the CTA to the slowest one: measured -8 % with one block of slack less); the request is retried by
// whoever comes next, and by any warp that finds its own slab missing (rp_pass).
__device__ __forceinline__ void rp_request(RpCtx &c, uint32_t tgt, int blk) {
    unsigned cur = *reinterpret_cast<volatile unsigned *>(c.issued);
    while ((int)(tgt - cur) >= 0) {
        const uint32_t st = cur % RP_STAGES, ph = (cur / RP_STAGES) & 1u;
        if (!mbar_try_wait(c.empty_s + 8u * st, ph ^ 1u)) return;   // not every warp has released the previous use of that stage
        const unsigned old = atomicCAS(c.issued, cur, cur + 1u);
        if (old == cur) {
            int b = blk + (int)(cur - c.gb);
            while (b >= c.nblk) b -= c.nblk;
            const uint32_t o0 = __ldg(c.off + b), o1 = __ldg(c.off + b + 1);
            const uint32_t bytes = (o1 - o0) * 16u;
            mbar_expect_tx(c.full_s + 8u * st, bytes);
            tma_load_1d(c.stage_s + st * (uint32_t)RP_STAGE_BYTES, c.slabs + (size_t)o0 * 16u, bytes, c.full_s + 8u * st);
            cur = cur + 1u;
        } else {
            cur = old;
        }
    }
}

// the warp's rows of the foreign half-words listed at shared address `list_s` -> slots 1 .. nb (asynchronous).  A slot is one
// 128-byte row [lane] in shared memory exactly as in global memory, so the warp copies four rows per instruction (8 lanes x
// 16 bytes each); every lane later reads only its own column.
__device__ __forceinline__ void rp_stage_issue(const RpCtx &c, uint32_t list_s, int nb) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t dst = c.sfb_s - 4u * lane + 128u + (lane >> 3) * 128u + (lane & 7u) * 16u;
    const uint32_t *src = c.SF - lane + (lane & 7u) * 4u;
    __syncwarp();   // every lane has finished reading the slots of the previous block
    for (int s0 = 0; s0 < nb; s0 += 4) {
        const int s = s0 + (int)(lane >> 3);
        if (s < nb) {
            const uint32_t w = lds_u32(list_s + 4u * (uint32_t)s);
            rp_cp_async16(dst + (uint32_t)s0 * 128u, src + (int64_t)w * 32);
        }
    }
}
// wait for the staged rows (own copies), make them visible to the other lanes
__device__ __forceinline__ void rp_stage_wait() {
    rp_cp_async_wait_all();
    __syncwarp();
}

// group term of a decision: M_g + kappa_g and the bounds from shared memory
template <GroupKind GROUPS>
__device__ __forceinline__ double rp_group_flip_cost(const RpCtx &c, int g, int ca, bool up) {
    if (GROUPS == GK_EQ32) {   // kappa's low 32-bit word, added in 32-bit arithmetic (the host checked the ranges)
        const int m = c.Mcol[g * c.mstride] + reinterpret_cast<const int *>(c.kap)[2 * g];
        return group_flip_cost<GK_EQ32>(c.lam[g], ca, up, m, 0, 0);
    }
    if (GROUPS == GK_EQ64) {
        // group_flip_cost's form, written out: with M_g + kappa_g formed before the product, nvcc allocates the registers
        // of the k-way instances (which spill) differently
        const long long t = (long long)ca * ((long long)ca - (up ? 1 : -1) * ((long long)c.Mcol[g * c.mstride] + c.kap[g]));
        return c.lam[g] * (double)t;
    }
    const long long *kb = c.kap + 3 * g;
    return group_flip_cost<GK_INTERVAL>(c.lam[g], ca, up, (long long)c.Mcol[g * c.mstride] + kb[0], kb[1], kb[2]);
}

// One pass over all blocks.  MODE 0: replay sweep.  MODE 1: catch-up (pending later-neighbour updates only, no decisions).
// MODE 2: push sweep (neal's eager form).  MODE 3: field set-up f[v] = h_v + sum_j J_vj s_j in neal's get_flip_energy order,
// for models whose adjacency lists are ascending (then adjacency order = pre entries u < v0, seq entries, later entries).
// GROUPS: the group term (GK_INTERVAL: c.kap holds {kappa, lo, hi} per group).  KWAY: the slabs carry k-way sections
// (rp_kway_batch); false compiles the replay sweep without the section test, so models without k-way blocks run exactly the
// generic kernel.  PROP: the acceptance rule of the decisions (modes 0 and 2).
template <int MODE, GroupKind GROUPS, int SLOTS, bool KWAY = false, Proposal PROP = PROP_METROPOLIS>
__device__ void rp_pass(RpCtx &c, double beta, bool has_next_pass) {
    const int lane = threadIdx.x & 31;
    const double thr = 44.36142 / beta;
    const int n = c.n, nblk = c.nblk;
    double *const fT = c.fT;
    uint32_t *const SF = c.SF;
    const uint32_t sfb = c.sfb_s, psb = c.psb_s;
    const bool active = c.active;
    uint32_t W = 0u, W0 = 0u, Wprev = 0u;   // the block's own half-word: bit 2i+1 = D (spin down), bit 2i = F (flipped)

    double fq[RP_LA];   // fields of the next RP_LA rows of the batch phase
#pragma unroll
    for (int k = 0; k < RP_LA; ++k) fq[k] = 0.0;
    if (MODE <= 1) {    // rows 0 .. RP_LA-1 of block 0 (every problem has at least one full half-word of padded variables)
#pragma unroll
        for (int k = 0; k < RP_LA; ++k) fq[k] = __ldcg(fT + k * 32);
    }

    const uint32_t g_last = c.gb + (uint32_t)nblk - 1u;   // running index of the last block of this pass
    for (int blk = 0; blk < nblk; ++blk) {
        RP_CLK(t_top);
        const uint32_t stage = c.gb % RP_STAGES, phase = (c.gb / RP_STAGES) & 1u;
        if (lane == 0) {
            uint32_t tgt = c.gb + (uint32_t)RP_DIST;
            if (!has_next_pass && (int)(tgt - g_last) > 0) tgt = g_last;
            rp_request(c, tgt, blk);
        }
        __syncwarp();
        RP_CLK(t_sw);
        while (!mbar_try_wait(c.full_s + 8u * stage, phase)) {   // usually there; else make sure somebody has asked for it
            if (lane == 0) rp_request(c, c.gb, blk);
        }
#ifdef QA_RP_PROFILE
        long long t_wait = clock64() - t_sw;
        RP_PROF(1, t_wait);
#endif
        const uint32_t hdr = c.stage_s + stage * (uint32_t)RP_STAGE_BYTES;   // shared address of the slab
        const uint32_t ent = hdr + (uint32_t)sizeof(RpHdr);
        const int v0 = (int)lds_u32(hdr + RP_H_V0);
        const int nv = (int)lds_u32(hdr + RP_H_NV);
        const int hw = v0 >> 4;
        const int sub = v0 & 15;
        double *const fB = fT + (int64_t)v0 * 32;
        const int ilim = min(nv, n - v0);   // uniform: padding variables are not visited
        if (sub == 0) {
            W = __ldcg(SF + (int64_t)hw * 32);
            W0 = W;
        }
        {   // L2 run-ahead of the field rows RP_PF_DIST variables on: 16 rows x 256 B = 128 sectors, one per lane and instruction
            int pv = (v0 & ~(RP_D - 1)) + RP_PF_DIST;   // a 16-row group ahead (wraps into the next sweep)
            if (pv >= c.npad) pv -= c.npad;
            const char *pa = reinterpret_cast<const char *>(fT - lane + (int64_t)pv * 32) + lane * 32;
#pragma unroll
            for (int k = 0; k < 4; ++k) asm volatile("prefetch.global.L2 [%0];" ::"l"(pa + k * 1024));
        }
        if (MODE != 2) {
            // the foreign half-words were requested while the previous block decided; the first block of a pass asks now
            if (blk == 0) rp_stage_issue(c, hdr + RP_H_BW, (int)lds_u32(hdr + RP_H_NBW));
            RP_CLK(t_gw);
            rp_stage_wait();
#ifdef QA_RP_PROFILE
            RP_PROF(2, clock64() - t_gw);
            t_wait += clock64() - t_gw;
#endif
            const uint32_t ps = lds_u32(hdr + RP_H_PREV);
            if (blk != 0 && ps != 0u) sts_u32(sfb + ps * 128u, Wprev);   // the one word that copy could not have up to date
            sts_u32(sfb, W);
        }

        if (MODE == 0) {
            // ---- batch phase: pre parts of all rows; table entries are loaded one round ahead of their use (two buffers, rounds
            // in pairs: no register rotation); rows in groups of RP_LA so that the field look-ahead needs no rotation either
            RP_CLK(t_batch);
            RP_PROF(3, t_batch - t_top - t_wait);
            uint32_t a = ent;
            uint32_t chg = 0u;
            const uint32_t kw = KWAY ? lds_u32(hdr + RP_H_KW) : 0u;
            if (KWAY && kw != 0u) {
                const int K = (int)(kw >> 16);
                chg = K == 2 ? rp_kway_batch<2, SLOTS>(hdr, ent, kw, nv, fB, fq, W, sfb, psb)
                    : K == 4 ? rp_kway_batch<4, SLOTS>(hdr, ent, kw, nv, fB, fq, W, sfb, psb)
                             : rp_kway_batch<8, SLOTS>(hdr, ent, kw, nv, fB, fq, W, sfb, psb);
            } else {
#pragma unroll 1
                for (int i0 = 0; i0 < nv; i0 += RP_LA) {
#pragma unroll
                    for (int kk = 0; kk < RP_LA; ++kk) {
                        const int i = i0 + kk;
                        if (i < nv) {
                            double p = fq[kk];
                            if (i + RP_LA < nv) fq[kk] = __ldcg(fB + (i + RP_LA) * 32);
                            const double f0 = p;
                            const int nr = (int)(lds_u32(hdr + RP_H_ROWA + 4u * (uint32_t)i) & 255u);
                            int4 qa[4], qb[4];
                            uint32_t w[4];
#pragma unroll
                            for (int k = 0; k < 4; ++k) qa[k] = lds_v4(a + 16u * k);
                            int r = 0;
#pragma unroll 1
                            for (; r + 2 <= nr; r += 2) {
#pragma unroll
                                for (int k = 0; k < 4; ++k) qb[k] = lds_v4(a + 64u + 16u * k);
#pragma unroll
                                for (int k = 0; k < 4; ++k) w[k] = lds_vu32(((uint32_t)qa[k].w & rp_slot_mask(SLOTS)) | sfb);
#pragma unroll
                                for (int k = 0; k < 4; ++k) rp_add_entry(p, qa[k], w[k]);
#pragma unroll
                                for (int k = 0; k < 4; ++k) qa[k] = lds_v4(a + 128u + 16u * k);
#pragma unroll
                                for (int k = 0; k < 4; ++k) w[k] = lds_vu32(((uint32_t)qb[k].w & rp_slot_mask(SLOTS)) | sfb);
#pragma unroll
                                for (int k = 0; k < 4; ++k) rp_add_entry(p, qb[k], w[k]);
                                a += 128u;
                            }
                            if (r < nr) {
#pragma unroll
                                for (int k = 0; k < 4; ++k) w[k] = lds_vu32(((uint32_t)qa[k].w & rp_slot_mask(SLOTS)) | sfb);
#pragma unroll
                                for (int k = 0; k < 4; ++k) rp_add_entry(p, qa[k], w[k]);
                                a += 64u;
                            }
                            sts_f64(psb + (uint32_t)i * 256u, p);
                            if (p != f0) chg |= 1u << i;
                        }
                    }
                }
            }
            // the batch phase is the last reader of the slots: request the next block's half-words now, load its first fields
            if (blk + 1 < nblk) {
                rp_stage_issue(c, hdr + RP_H_BWN, (int)lds_u32(hdr + RP_H_NBWN));
                const double *fN = fB + nv * 32;
#pragma unroll
                for (int k = 0; k < RP_LA; ++k) fq[k] = __ldcg(fN + k * 32);
            }

            RP_CLK(t_seq);
            RP_PROF(4, t_seq - t_batch);
            // ---- sequential phase: in-block earlier neighbours from the register, then neal's decision
            uint32_t as = ent + lds_u32(hdr + RP_H_SEQ) * 16u;
#pragma unroll 1
            for (int i = 0; i < ilim; ++i) {
                const uint32_t ra = lds_u32(hdr + RP_H_ROWA + 4u * (uint32_t)i);
                const double pv = lds_f64(psb + (uint32_t)i * 256u);
                double fv = pv;
                const uint32_t ae = as + ((ra >> 8) & 255u) * 16u;
                for (; as + 16u < ae; as += 32u) {
                    const int4 qa = lds_v4(as), qb = lds_v4(as + 16u);
                    rp_add_entry(fv, qa, W);
                    rp_add_entry(fv, qb, W);
                }
                if (as < ae) {
                    const int4 qa = lds_v4(as);
                    rp_add_entry(fv, qa, W);
                    as += 16u;
                }
                if (((chg >> i) & 1u) != 0u || fv != pv) __stcg(fB + i * 32, fv);
                const uint32_t fb = 1u << (2 * (sub + i)), db = fb << 1;
                const bool up = (W & db) == 0u;
                double dE = up ? -2.0 * fv : 2.0 * fv;
                int g = 255, ca = 0;
                if (GROUPS != GK_NONE) {
                    const int ga = (int)lds_u32(hdr + RP_H_GA + 4u * (uint32_t)i);
                    g = ga & 255;
                    if (g != 255) {
                        ca = ga >> 8;
                        dE = dE + rp_group_flip_cost<GROUPS>(c, g, ca, up);
                    }
                }
                const bool cand = active && !(dE >= thr);
                bool acc = false;
                if (__any_sync(FULL_MASK, cand)) {
                    if (cand) c.st.cand++;
                    acc = accept_test<PROP>(dE, cand, beta, thr, c.s0, c.s1, c.st);
                }
                // F[v] := accepted (also when nothing was accepted: the flag of the previous visit must be cleared)
                W = acc ? ((W | fb) ^ db) : (W & ~fb);
                if (acc) {
                    c.st.acc++;
                    c.st.nbr += (unsigned long long)(ra >> 16);
                    if (GROUPS != GK_NONE) {
                        if (g != 255) c.Mcol[g * c.mstride] -= 2 * ca * (up ? 1 : -1);
                    }
                }
            }
            RP_PROF(5, clock64() - t_seq);
        } else if (MODE == 1) {
            // ---- catch-up: the pending later-neighbour updates (a prefix of every pre part), no decisions
            uint32_t a = ent;
#pragma unroll 1
            for (int i0 = 0; i0 < nv; i0 += RP_LA) {
#pragma unroll
                for (int kk = 0; kk < RP_LA; ++kk) {
                    const int i = i0 + kk;
                    if (i < nv) {
                        double p = fq[kk];
                        if (i + RP_LA < nv) fq[kk] = __ldcg(fB + (i + RP_LA) * 32);
                        const double f0 = p;
                        const uint32_t nr = lds_u32(hdr + RP_H_ROWA + 4u * (uint32_t)i) & 255u;
                        const uint32_t nl = lds_u32(hdr + RP_H_ROWB + 4u * (uint32_t)i) & 0xffffu;
                        for (uint32_t k = 0; k < nl; ++k) {
                            const int4 q = lds_v4(a + 16u * k);
                            rp_add_entry(p, q, lds_vu32(((uint32_t)q.w & rp_slot_mask(SLOTS)) | sfb));
                        }
                        a += nr * 64u;
                        if (p != f0) __stcg(fB + i * 32, p);
                    }
                }
            }
            if (blk + 1 < nblk) {
                rp_stage_issue(c, hdr + RP_H_BWN, (int)lds_u32(hdr + RP_H_NBWN));
                const double *fN = fB + nv * 32;
#pragma unroll
                for (int k = 0; k < RP_LA; ++k) fq[k] = __ldcg(fN + k * 32);
            }
        } else if (MODE == 3) {
            // ---- set-up: h_v, then the earlier neighbours (pre entries u < v0, seq entries), then the later ones, ascending:
            // neal's get_flip_energy order for ascending adjacency lists, one rounding per term.
            uint32_t a = ent;
            uint32_t as = ent + lds_u32(hdr + RP_H_SEQ) * 16u;
#pragma unroll 1
            for (int i = 0; i < nv; ++i) {
                const uint32_t ra = lds_u32(hdr + RP_H_ROWA + 4u * (uint32_t)i);
                const uint32_t rb = lds_u32(hdr + RP_H_ROWB + 4u * (uint32_t)i);
                const uint32_t nl = rb & 0xffffu, np = rb >> 16, ns = (ra >> 8) & 255u;
                if (i < ilim) {
                    double fv = __ldg(c.h + v0 + i);
                    auto add1 = [&](uint32_t ad) {
                        const int4 q = lds_v4(ad);
                        const uint32_t w = lds_vu32(((uint32_t)q.w & rp_slot_mask(SLOTS)) | sfb);
                        const uint32_t x = w << ((uint32_t)q.w & 31u);
                        fv = fv + __hiloint2double(q.y ^ (int)(x & 0x80000000u), q.x);   // down: -J
                    };
                    for (uint32_t k = nl; k < np; ++k) add1(a + 16u * k);
                    for (uint32_t k = 0; k < ns; ++k) add1(as + 16u * k);
                    for (uint32_t k = 0; k < nl; ++k) add1(a + 16u * k);
                    __stcg(fB + i * 32, fv);
                }
                a += (ra & 255u) * 64u;
                as += ns * 16u;
            }
            if (blk + 1 < nblk) rp_stage_issue(c, hdr + RP_H_BWN, (int)lds_u32(hdr + RP_H_NBWN));
        } else {
            // ---- push sweep: the block's fields staged in shared memory, neal's eager neighbour updates
            {
                double t[RP_D];
#pragma unroll
                for (int i = 0; i < RP_D; ++i)
                    if (i < nv) t[i] = __ldcg(fB + i * 32);
#pragma unroll
                for (int i = 0; i < RP_D; ++i)
                    if (i < nv) sts_f64(psb + (uint32_t)i * 256u, t[i]);
            }
            bool blk_dirty = false;
            uint32_t a = ent;
            uint32_t as = ent + lds_u32(hdr + RP_H_SEQ) * 16u;
#pragma unroll 1
            for (int i = 0; i < ilim; ++i) {
                const uint32_t ra = lds_u32(hdr + RP_H_ROWA + 4u * (uint32_t)i);
                const uint32_t a_row = a, as_row = as;
                a += (ra & 255u) * 64u;
                as += ((ra >> 8) & 255u) * 16u;
                const double fv = lds_f64(psb + (uint32_t)i * 256u);
                const uint32_t db = 2u << (2 * (sub + i));
                const bool up = (W & db) == 0u;
                double dE = up ? -2.0 * fv : 2.0 * fv;
                int g = 255, ca = 0;
                if (GROUPS != GK_NONE) {
                    const int ga = (int)lds_u32(hdr + RP_H_GA + 4u * (uint32_t)i);
                    g = ga & 255;
                    if (g != 255) {
                        ca = ga >> 8;
                        dE = dE + rp_group_flip_cost<GROUPS>(c, g, ca, up);
                    }
                }
                const bool cand = active && !(dE >= thr);
                bool acc = false;
                if (__any_sync(FULL_MASK, cand)) {
                    if (cand) c.st.cand++;
                    acc = accept_test<PROP>(dE, cand, beta, thr, c.s0, c.s1, c.st);
                }
                if (__ballot_sync(FULL_MASK, acc) == 0u) continue;
                const int sgn = up ? (int)0x80000000u : 0;   // f[j] += -2 s_v J
                const uint32_t np = lds_u32(hdr + RP_H_ROWB + 4u * (uint32_t)i) >> 16;
#pragma unroll
                for (int part = 0; part < 2; ++part) {
                    const uint32_t ab = part == 0 ? a_row : as_row;
                    const uint32_t cnt = part == 0 ? np : ((ra >> 8) & 255u);
#pragma unroll 4
                    for (uint32_t k = 0; k < cnt; ++k) {
                        const int4 q = lds_v4(ab + 16u * k);
                        const int j = (int)((uint32_t)q.w >> RP_J_SHIFT);
                        const double d = __hiloint2double(q.y ^ sgn, q.x) * 2.0;   // exact
                        if ((uint32_t)(j - v0) < (uint32_t)nv) {   // uniform: neighbour staged in this block
                            const uint32_t cad = psb + ((uint32_t)(j - v0) << 8);
                            if (acc) sts_f64(cad, lds_f64(cad) + d);
                            blk_dirty = true;
                        } else {
                            red_add_f64_if(fT + (int64_t)j * 32, d, acc);
                        }
                    }
                }
                if (acc) {
                    W ^= db;
                    c.st.acc++;
                    c.st.nbr += (unsigned long long)(ra >> 16);
                    if (GROUPS != GK_NONE) {
                        if (g != 255) c.Mcol[g * c.mstride] -= 2 * ca * (up ? 1 : -1);
                    }
                }
            }
            if (blk_dirty) {  // uniform: write the staged fields back (coalesced 256 B rows)
#pragma unroll
                for (int i = 0; i < RP_D; ++i)
                    if (i < nv) __stcg(fB + i * 32, lds_f64(psb + (uint32_t)i * 256u));
            }
        }
        if ((MODE == 0 || MODE == 2) && sub + nv == RP_D) {
            if (W != W0) __stcg(SF + (int64_t)hw * 32, W);
        }
        Wprev = W;
        // release the stage: one arrive per warp
        __syncwarp();
        if (lane == 0) mbar_arrive(c.empty_s + 8u * stage);
        ++c.gb;
    }
}

// The set-up pass as a real call with the context passed BY VALUE: its registers do not add to the pressure of the sweep
// loops.
template <int SLOTS>
__device__ __noinline__ uint32_t rp_setup_pass(RpCtx c) {
    rp_pass<3, GK_NONE, SLOTS>(c, 1.0, true);
    return c.gb;
}

// local field of v in neal's get_flip_energy order (adjacency order), spins from the {S|F} scratch; loads batched by 8
__device__ __forceinline__ double rp_field_direct(const ProblemDesc &D, const uint32_t *SF, int v, int e0, int e1) {
    double fv = __ldg(D.h + v);
    for (int e = e0; e < e1; e += 8) {
        int jq[8];
        uint32_t wq[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            jq[q] = __ldg(D.col + min(e + q, e1 - 1));
            wq[q] = __ldcg(SF + (int64_t)(jq[q] >> 4) * 32);
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (e + q < e1) {
                const double J = __ldg(D.val + e + q);
                fv += ((wq[q] >> (2 * (jq[q] & 15) + 1)) & 1u) ? -J : J;
            }
        }
    }
    return fv;
}

// Shared-memory layout: [slab stages][mbarriers][CTA scratch][lambda][kappa][group counters] then, aligned to rp_sf_bytes(SLOTS) in
// the shared window (so that a slot address is formed by OR), one slot region per warp, then one partial-sum region per warp.
// `smem_base` is the shared-window offset of the dynamic allocation (1 KB on sm_100: the system-reserved bytes); the kernel
// verifies the assumption.
__host__ __device__ inline size_t rp_fixed_bytes(int nw, int max_groups, GroupKind gk) {
    size_t b = (size_t)RP_STAGES * RP_STAGE_BYTES + 8 * (2 * RP_STAGES) + 32;
    b += (sizeof(double) + kappa_words(gk) * sizeof(long long)) * (size_t)max_groups;
    b += sizeof(int) * (size_t)max_groups * nw * 32;
    return b;
}
__host__ __device__ inline size_t rp_smem_bytes(int nw, int max_groups, unsigned smem_base, int slots, GroupKind gk) {
    const size_t fixed = rp_fixed_bytes(nw, max_groups, gk);
    const size_t sf = (size_t)rp_sf_bytes(slots);
    const size_t pad = (sf - (smem_base + fixed) % sf) % sf;
    return fixed + pad + (size_t)nw * (sf + RP_PS_BYTES);
}

template <GroupKind GROUPS, Proposal PROP, int SLOTS, bool KWAY>
__global__ void __launch_bounds__(RP_MAX_WARPS * 32, RP_MIN_CTAS) k_anneal_replay(AnnealParams P) {
    constexpr uint32_t RP_SF_BYTES = (uint32_t)rp_sf_bytes(SLOTS);
    extern __shared__ __align__(16) unsigned char rp_raw[];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int NW = blockDim.x >> 5;
    uint32_t raw_s;   // opaque to the compiler: it would otherwise re-derive the window address (S2R + LEA) inside the hot loops
    asm volatile("mov.u32 %0, %1;" : "=r"(raw_s) : "r"((uint32_t)__cvta_generic_to_shared(rp_raw)));
    const uint32_t fixed = (uint32_t)rp_fixed_bytes(NW, P.max_groups, GROUPS);
    const uint32_t base_s = (raw_s + fixed + (uint32_t)RP_SF_BYTES - 1u) & ~((uint32_t)RP_SF_BYTES - 1u);    // warp regions
    {
        uint32_t dyn;
        asm volatile("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
        if (base_s - raw_s + (uint32_t)NW * (RP_SF_BYTES + RP_PS_BYTES) > dyn) {   // uniform: report the real base and leave
            if (threadIdx.x == 0) {
                P.error_flag[1] = (int)raw_s;
                atomicExch(P.error_flag, QA_ERR_SMEM_BASE);
            }
            return;
        }
    }
    unsigned char *tail = rp_raw + (size_t)RP_STAGES * RP_STAGE_BYTES;
    const uint32_t bars_s = raw_s + (uint32_t)RP_STAGES * RP_STAGE_BYTES;
    unsigned *issued_sh = reinterpret_cast<unsigned *>(tail + 8 * (2 * RP_STAGES));
    long long *item_sh = reinterpret_cast<long long *>(tail + 8 * (2 * RP_STAGES) + 8);
    unsigned *acc_sh = reinterpret_cast<unsigned *>(tail + 8 * (2 * RP_STAGES) + 16);   // [2]
    double *lam_sh = reinterpret_cast<double *>(tail + 8 * (2 * RP_STAGES) + 32);
    long long *kap_sh = reinterpret_cast<long long *>(lam_sh + P.max_groups);
    int *M_all = reinterpret_cast<int *>(kap_sh + kappa_words(GROUPS) * P.max_groups);

    if (threadIdx.x == 0) {
        for (int s = 0; s < RP_STAGES; ++s) {
            mbar_init(bars_s + 8u * s, 1);                     // full: the requester's arrive.expect_tx
            mbar_init(bars_s + 8u * (RP_STAGES + s), NW);      // empty: one arrive per warp
        }
        *issued_sh = 0u;
        acc_sh[0] = 0u;
        acc_sh[1] = 0u;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (GROUPS != GK_NONE) stage_group_params<GROUPS>(P.descs[0], lam_sh, kap_sh);
    __syncthreads();

    RpCtx c;
    c.full_s = bars_s;
    c.empty_s = bars_s + 8u * RP_STAGES;
    c.stage_s = raw_s;
    c.issued = issued_sh;
    c.gb = 0u;
    c.sfb_s = base_s + (uint32_t)wib * RP_SF_BYTES + (uint32_t)lane * 4u;
    c.psb_s = base_s + (uint32_t)NW * RP_SF_BYTES + (uint32_t)wib * RP_PS_BYTES + (uint32_t)lane * 8u;
    c.Mcol = M_all + threadIdx.x;
    c.mstride = (int)blockDim.x;
    c.lam = lam_sh;
    c.kap = kap_sh;
    c.st = {0, 0, 0, 0, 0};
#ifdef QA_RP_PROFILE
    for (int k = 0; k < QA_NDEBUG; ++k) c.prof[k] = 0;
#endif
    const int64_t slot = (int64_t)blockIdx.x * NW + wib;
    c.fT = P.fT_scratch + slot * P.fT_stride + lane;
    c.SF = reinterpret_cast<uint32_t *>(P.sf_scratch) + slot * P.sf_stride + lane;
    int acc_par = 0;

    bool first_item = true;   // neal polls its interrupt callback BETWEEN reads: every CTA completes the first group it takes
    for (;;) {
        if (threadIdx.x == 0) {
            // host-mapped flag raised by the caller's interrupt callback: stop pulling work (without counting the pull)
            if (P.interrupt_flag != nullptr && !first_item && *reinterpret_cast<const volatile int *>(P.interrupt_flag) != 0)
                *item_sh = (long long)P.total_items;
            else
                *item_sh = (long long)atomicAdd(P.counter, 1ull);
        }
        first_item = false;
        __syncthreads();
        const int64_t item = *item_sh;
        __syncthreads();
        if (item >= P.total_items) break;
        const int p = (int)(item / P.groups_per_problem);
        const int64_t q = item % P.groups_per_problem;
        const ProblemDesc D = P.descs[p];
        const int64_t tile = q * NW + wib;
        const int64_t r = tile * 32 + lane;
        const bool active = r < D.reads;
        const long long cta_reads = min((long long)NW * 32, (long long)D.reads - (long long)q * NW * 32);
        c.active = active;
        c.n = D.n;
        c.nblk = D.rp_nslabs;
        c.npad = D.nch * 32;
        c.slabs = D.rp_slabs;
        c.h = D.h;
        c.off = D.rp_off;
        const long long total_sweeps = (long long)P.num_betas * P.sweeps_per_beta;
        if (lane == 0 && total_sweeps > 0) rp_request(c, c.gb + (uint32_t)RP_DIST, 0);   // overlaps with the set-up below

        const unsigned long long sd = active ? P.seeds[D.read_base + r] : 1ull;
        c.s0 = sd ? sd : ~0ull;
        c.s1 = 0;
        const int n = D.n, nhw = D.nch * 2;
        // ---- pack this read's +-1 bytes into D bits (padding lanes and padding variables are +1: D = 0), clear the flags
        {
            const int8_t *row0 = D.states + r * (int64_t)n;
            const bool vec = active && ((reinterpret_cast<uintptr_t>(row0) & 15u) == 0u);
            for (int hw = 0; hw < nhw; ++hw) {
                uint32_t w = 0u;
                if (active) {
                    const int8_t *row = row0 + hw * 16;
                    const int lim = min(16, n - hw * 16);
                    if (vec && lim == 16) {
                        const int4 t = *reinterpret_cast<const int4 *>(row);
                        const uint32_t tw[4] = {(uint32_t)t.x, (uint32_t)t.y, (uint32_t)t.z, (uint32_t)t.w};
                        bool bad = false;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const uint32_t neg = (tw[k] >> 7) & 0x01010101u;          // sign bit of every byte
                            bad = bad || tw[k] != 0x01010101u + neg * 0xfeu;          // every byte 0x01 or 0xff
                            w |= (((neg << 1) | (neg >> 5) | (neg >> 11) | (neg >> 17)) & 0xaau) << (8 * k);
                        }
                        if (bad) atomicExch(P.error_flag, QA_ERR_STATE);
                    } else {
                        for (int i = 0; i < lim; ++i) {
                            const int s = row[i];
                            if (s != 1 && s != -1) atomicExch(P.error_flag, QA_ERR_STATE);
                            if (s < 0) w |= 2u << (2 * i);
                        }
                    }
                }
                __stcg(c.SF + (int64_t)hw * 32, w);
            }
        }
        if (GROUPS != GK_NONE) {
            for (int g = 0; g < D.ngroups; ++g) c.Mcol[g * c.mstride] = 0;
            for (int hw = 0; hw < nhw; ++hw) {
                const uint32_t w = __ldcg(c.SF + (int64_t)hw * 32);
                for (int i = 0; i < 16; ++i) {
                    const int v = hw * 16 + i;
                    const int g = __ldg(D.grp + v);  // uniform
                    if (g >= 0) {
                        const int a = __ldg(D.coef + v);
                        c.Mcol[g * c.mstride] += ((w >> (2 * i + 1)) & 1u) ? -a : a;
                    }
                }
            }
        }
        // ---- local fields in neal's get_flip_energy order: through the slab ring when the adjacency lists are ascending,
        // else row by row from the CSR
        RP_CLK(t_setup);
        if (P.rp_slab_init) {
            if (total_sweeps > 0) c.gb = rp_setup_pass<SLOTS>(c);
        } else {
            int e0 = __ldg(D.rowptr);
            for (int v = 0; v < n; ++v) {
                const int e1 = __ldg(D.rowptr + v + 1);
                __stcg(c.fT + (int64_t)v * 32, rp_field_direct(D, c.SF, v, e0, e1));
                e0 = e1;
            }
        }
        RP_PROF(0, clock64() - t_setup);
        // ---- the schedule: replay sweeps while flips are frequent, then one catch-up pass and push sweeps
        bool push = false;
        long long done = 0;
        for (int bi = 0; bi < P.num_betas; ++bi) {
            const double beta = (D.betas ? D.betas : P.betas)[bi];
            for (int swi = 0; swi < P.sweeps_per_beta; ++swi) {
                ++done;
                const bool more = done < total_sweeps;
#ifdef QA_RP_PROFILE
                if (blockIdx.x == 0 && threadIdx.x == 0)
                    printf("[qa sweep] %lld beta %.4g mode %s clock %lld\n", done, beta, push ? "push" : "replay", clock64());
#endif
                RP_CLK(t_pass);
                if (push) {
                    rp_pass<2, GROUPS, SLOTS, false, PROP>(c, beta, more);
                    RP_PROF(7, clock64() - t_pass);
                } else {
                    const unsigned acc0 = c.st.acc;
                    rp_pass<0, GROUPS, SLOTS, KWAY, PROP>(c, beta, more);
                    RP_PROF(6, clock64() - t_pass);
                    if (more) {  // CTA-uniform hand-over decision
                        unsigned wacc = c.st.acc - acc0;
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) wacc += __shfl_xor_sync(FULL_MASK, wacc, o);
                        if (lane == 0) atomicAdd(acc_sh + acc_par, wacc);
                        __syncthreads();
                        const unsigned long long tot = acc_sh[acc_par];
                        if (threadIdx.x == 0) acc_sh[acc_par ^ 1] = 0u;
                        acc_par ^= 1;
                        if (tot * 1000ull < (unsigned long long)P.switch_permille * (unsigned long long)n * (unsigned long long)cta_reads) {
                            RP_CLK(t_cu);
                            rp_pass<1, GK_NONE, SLOTS>(c, beta, true);
                            RP_PROF(7, clock64() - t_cu);
                            push = true;
                        }
                    }
                }
            }
        }
        // ---- final spins: packed transposed layout for the energy kernel (bit = 1: spin up), +-1 bytes for the caller
        if (active) {
            int8_t *row0 = D.states + r * (int64_t)n;
            const bool vec = (reinterpret_cast<uintptr_t>(row0) & 15u) == 0u;
            uint32_t up32 = 0u;
            for (int hw = 0; hw < nhw; ++hw) {
                const uint32_t w = __ldcg(c.SF + (int64_t)hw * 32);
                uint32_t x = (w >> 1) & 0x55555555u;           // the 16 D bits, compressed to the low half
                x = (x | (x >> 1)) & 0x33333333u;
                x = (x | (x >> 2)) & 0x0f0f0f0fu;
                x = (x | (x >> 4)) & 0x00ff00ffu;
                x = (x | (x >> 8)) & 0x0000ffffu;
                const uint32_t up16 = ~x & 0xffffu;
                if (hw & 1) D.packedT[(int64_t)(hw >> 1) * D.rpad + r] = up32 | (up16 << 16);
                else up32 = up16;
                int8_t *row = row0 + hw * 16;
                const int lim = min(16, n - hw * 16);
                if (vec && lim == 16) {
                    uint32_t o[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t t = (w >> (8 * k)) & 0xaau;
                        const uint32_t sp = ((t >> 1) | (t << 5) | (t << 11) | (t << 17)) & 0x01010101u;   // down flag per byte
                        o[k] = 0x01010101u + sp * 0xfeu;
                    }
                    *reinterpret_cast<int4 *>(row) = make_int4((int)o[0], (int)o[1], (int)o[2], (int)o[3]);
                } else {
                    for (int i = 0; i < lim; ++i) row[i] = ((w >> (2 * i + 1)) & 1u) ? -1 : 1;
                }
            }
        }
    }
    flush_lane_stats(P, c.st);
#ifdef QA_RP_PROFILE
    if (lane == 0)
        for (int k = 0; k < QA_NDEBUG; ++k) atomicAdd(P.stats + QA_NSTAT + 1 + k, (unsigned long long)c.prof[k]);
#endif
}

// the kernel instance for the acceptance rule, group kind, slot count and k-way form of a model
template <Proposal PROP, int SLOTS, bool KWAY>
static const void *replay_instance(GroupKind gk) {
    switch (gk) {
    case GK_NONE: return (const void *)k_anneal_replay<GK_NONE, PROP, SLOTS, KWAY>;
    case GK_EQ32: return (const void *)k_anneal_replay<GK_EQ32, PROP, SLOTS, KWAY>;
    case GK_EQ64: return (const void *)k_anneal_replay<GK_EQ64, PROP, SLOTS, KWAY>;
    default: return (const void *)k_anneal_replay<GK_INTERVAL, PROP, SLOTS, KWAY>;
    }
}

template <Proposal PROP>
static const void *replay_instance(const qa_model *M, GroupKind gk) {
    const bool kway = M->rp_kway_blocks > 0;
    if (M->rp_slots == 32) return kway ? replay_instance<PROP, 32, true>(gk) : replay_instance<PROP, 32, false>(gk);
    return kway ? replay_instance<PROP, 64, true>(gk) : replay_instance<PROP, 64, false>(gk);
}
