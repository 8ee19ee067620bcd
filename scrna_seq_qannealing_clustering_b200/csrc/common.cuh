// common.cuh -- declarations shared by the translation units of libqanneal.so (internal; the public C ABI is include/qanneal.h).
//
//   api.cu              context, kernel selection (run_anneal), sample entry points
//   model.cu            adjacency construction, qa_model, rank-1 groups
//   anneal_ref.cu       k_anneal_ref       one warp per read
//   anneal_lockstep.cu  k_anneal_lockstep  32 reads per warp, eager updates
//   anneal_replay.cu    k_anneal_replay    32 reads per warp, deferred exact updates (replay.cuh), slab packer
//   anneal_replay_gibbs.cu                 its Gibbs-acceptance instances
//   anneal_dense.cu     k_anneal_dense     dense k-way models on the fp64 tensor cores (dense.cuh)
//   energy.cu           k_energy, k_pack_states
//   builders.cu         qa_build_*          model builders on the device
//   postprocess.cu      sort / aggregate / gather / decode / argmin / random states
//   snn.cu              qa_snn_build        SNN graph construction
//   recursion.cu        qa_graph_split, qa_model_concat, qa_sa_sample_model_batch
#pragma once

#include "../../include/qanneal.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <string>
#include <vector>

#define QA_VERSION 200
#define FULL_MASK 0xffffffffu

namespace qa {

extern thread_local std::string g_err;   // api.cu

inline int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

#define QA_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(QA_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));         \
    } while (0)

// ------------------------------------------------------------------------------------------------
// device-side problem description (one per independent problem; a plain model is a batch of one)
// ------------------------------------------------------------------------------------------------
struct ProblemDesc {
    int32_t n;        // variables
    int32_t nch;      // 32-variable chunks = ceil(n/32)
    int32_t ngroups;  // rank-1 groups (0: none)
    int32_t reads;    // reads of this problem
    int32_t rpad;     // reads padded to a multiple of 32 (stride of packedT)
    int32_t pad_;
    int64_t m;        // couplers
    int64_t read_base;  // index of this problem's read 0 in the global read numbering
    const int32_t *rowptr;  // [nch*32 + 1] entries valid (padding rows are empty)
    const int32_t *col;     // CSR neighbour, local variable index
    const double *val;      // CSR coupling
    const double *h;        // [n]
    const int32_t *starts;  // COO in caller order (energy summation order)
    const int32_t *ends;
    const double *w;
    const int32_t *grp;     // [nch*32] or null
    const int32_t *coef;    // [nch*32]
    const double *lambda;   // [ngroups]
    const long long *kappa; // [ngroups]; interval groups (qa_model_set_group_bounds): [3][ngroups] = kappa, lo, hi
    int8_t *states;         // [reads][n]
    uint32_t *packedT;      // [nch][rpad] final spins, bit i of word (c, r) = spin of variable 32c+i (1: +1)
    double *energies;       // [reads]
    // block word tables of the lockstep kernel's field set-up pass (null until built): for every block of 16 variables the
    // distinct spin words its CSR rows refer to, and per CSR entry the index of its word in that list (255 = the block's own word)
    const int32_t *bw_ptr;      // [nblk + 1], this problem's first block at index 0 (values are global offsets)
    const int32_t *bw_words;    // global array
    const unsigned short *ent_slot; // indexed like col: slot | (bit << 8)
    // coupling slabs of the replay kernel (null until built): one {RpHdr, RpEntry[]} per block of 16 variables
    const unsigned char *rp_slabs;  // global slab storage
    const uint32_t *rp_off;         // [rp_nslabs + 1] slab offsets of this problem in 16-byte units
    int32_t rp_nslabs;              // blocks (slabs) of this problem
    int32_t pad2_;
    const double *betas;            // this problem's own beta schedule [num_betas], or null: the launch's shared schedule
};

struct AnnealParams {
    const ProblemDesc *descs;
    int32_t num_problems;
    int32_t reads_per_problem;   // uniform (batch) ; == total reads for a single model
    int64_t total_reads;
    const double *betas;
    int32_t num_betas;
    int32_t sweeps_per_beta;
    const unsigned long long *seeds;
    int32_t seed_mode;
    double *f_scratch;           // [slots][f_stride]
    uint32_t *spw_scratch;       // [slots][spw_stride]
    int64_t f_stride;
    int64_t spw_stride;
    unsigned long long *counter; // next read to hand out
    unsigned long long *stats;   // QA_NSTAT counters
    int *error_flag;
    int64_t read_begin;          // wave support: global read range [read_begin, read_end)
    int64_t read_end;
    // lockstep kernels (one warp = 32 reads of one problem)
    double *fT_scratch;          // [slots][fT_stride]  read-interleaved local fields f[v][lane]
    int64_t fT_stride;           // n_pad_max * 32
    int32_t tiles_per_problem;
    int32_t max_groups;          // stride of the per-thread group counters in shared memory
    int64_t total_tiles;
    // replay kernel (one CTA = `warps` consecutive 32-read tiles of one problem)
    void *sf_scratch;            // [slots][sf_stride] {S | F << 16} half-word words, read-interleaved (uint32)
    int64_t sf_stride;           // nch_max * 2 * 32
    int64_t groups_per_problem;  // ceil(tiles_per_problem / warps per CTA)
    int64_t total_items;         // num_problems * groups_per_problem
    int32_t switch_permille;     // replay -> push hand-over: CTA-wide acceptance of a sweep below this many per mille
    int32_t rp_slab_init;        // adjacency lists ascending: the field set-up pass runs through the slab ring
    const int *interrupt_flag;   // host-mapped flag (or null): CTAs stop pulling work once it is non-zero
    // dense k-way kernel (dense.cuh)
    uint32_t *dn_spins;          // [slots][dn_stride] bit-packed spins, one slot per resident warp
    int64_t dn_stride;           // (ncp / 32) * 32 * K words
};

enum { ST_CAND = 0, ST_DRAWS, ST_ACC, ST_NBR, ST_ACTIVE, ST_CHUNKS, ST_TIES, QA_NSTAT };
constexpr int QA_NDEBUG = 8;   // development counters behind the read counter (QA_RP_PROFILE builds print them)

constexpr int QA_TPB_MAX = 256;
// measured on B200 (config 3): lockstep wins from ~3.5 tiles of 32 reads per SM, warp-per-read below that
constexpr int QA_PREFETCH_CHUNKS = 16;  // run-ahead distance of the L2 prefetch, in 256-byte chunks
constexpr double QA_TWO64 = 18446744073709551616.0;

struct DenseDesc {
    int32_t ncells;      // cells
    int32_t ncp;         // cells padded to a multiple of 32 (padding rows / columns of W are zero)
    int32_t K;           // cases per cell; variable v = cell*K + case
    int32_t ngrp;        // ncp / 32
    const double *W;     // [ncp][ncp] same-case coupling between cells, zero diagonal
    double P;            // coupling between two cases of one cell
};

constexpr int QA_ERR_SMEM_BASE = -100;   // internal: the replay kernel's dynamic shared memory does not start where the host assumed

struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
};

}  // namespace qa

struct qa_ctx {
    int device = 0;
    int num_sms = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    qa::DevBuf f, spw, fT, sf, states, energies, seeds, betas, packed, misc, cubtmp;
    int kernel = 0;  // QA_KERNEL_*
    int replay_switch_permille = 20;  // replay -> push hand-over threshold (QA_REPLAY_SWITCH_PERMILLE overrides)
    int replay_warps = 0;             // warps per CTA of the replay kernel (0: automatic; QA_REPLAY_WARPS overrides)
    int replay_kway = 1;              // k-way sections in the replay slabs (QA_REPLAY_KWAY=0: generic blocks only)
    int last_kernel = 0;              // QA_KERNEL_* the last sampling call ran on
    unsigned rp_smem_base = 1024;     // shared-window offset of dynamic shared memory (verified by the replay kernel)
    bool rp_base_checked = false;
    bool betas_per_problem = false;   // transient: the running call carries one beta schedule per problem ([P][num_betas])
    int *h_iflag = nullptr, *d_iflag = nullptr;  // host-mapped interrupt flag polled by the replay kernel
    unsigned long long *d_stats = nullptr;  // QA_NSTAT counters + 1 read counter
    int *d_flag = nullptr;
    double *d_best_e = nullptr;
    long long *d_best_i = nullptr;
    uint32_t launches = 0;
};

struct qa_model {
    qa_ctx *ctx = nullptr;
    int32_t num_problems = 1;
    int64_t n_total = 0;   // sum of n_p
    int64_t m_total = 0;
    int32_t n_max = 0, nch_max = 0;
    int32_t max_deg = 0;
    int32_t ngroups = 0;
    std::vector<int64_t> var_off, cpl_off;  // host copies [P+1]
    // device arrays (owned)
    double *h = nullptr;
    int32_t *starts = nullptr, *ends = nullptr;
    double *w = nullptr;
    int32_t *rowptr = nullptr, *col = nullptr;
    double *val = nullptr;
    int32_t *grp = nullptr, *coef = nullptr;
    double *lambda = nullptr;
    long long *kappa = nullptr;
    bool gbounds = false;  // the groups carry interval bounds: kappa[ngroups .. 3 ngroups) = lo, hi (clamped to the reachable range)
    std::vector<int64_t> gumin, gumax;         // host: reachable range kappa -+ sum |a| of every group (single-problem models)
    qa::ProblemDesc *d_descs = nullptr;
    std::vector<qa::ProblemDesc> descs;  // host mirror (pointers are device pointers)
    // block word tables of the lockstep kernel's field set-up pass (built on first use)
    int32_t *bw_ptr = nullptr, *bw_words = nullptr;
    unsigned short *ent_slot = nullptr;
    bool tables_built = false;
    // coupling slabs of the replay kernel (built on first use; rp_ok = the model fits the slab format)
    unsigned char *rp_slabs = nullptr;
    uint32_t *rp_off = nullptr;
    bool rp_built = false, rp_ok = false;
    bool rp_uniform = false;   // every block holds exactly RP_D variables
    int rp_slots = 32;         // half-word slots per warp the slabs were packed for (32 or 64)
    bool rp_adj_sorted = false; // adjacency lists ascending: field set-up through the slab ring
    int32_t rp_kway_k = 0;      // cell size of the k-way blocks (0: none)
    int64_t rp_kway_blocks = 0; // slabs with a k-way section
    bool groups_i32 = false;   // every group term a*(a - s*(M+kappa)) fits 32-bit integers
    // dense k-way form (dense.cuh): W and P derived from the CSR by qa_model_enable_dense
    double *dn_W = nullptr;
    bool dn_ok = false;
    qa::DenseDesc dn = {};
};

struct qa_graph {
    qa_ctx *ctx = nullptr;
    int32_t num_problems = 0;
    std::vector<int64_t> point_off, edge_off;   // host copies [P + 1]
    int32_t *eu = nullptr, *ev = nullptr;       // device, local indices, sorted by (problem, u, v)
    double *w = nullptr;
    int32_t *node_ids = nullptr;                // qa_graph_split: parent node of every local node, or null
};

namespace qa {

inline int ensure(DevBuf &b, size_t bytes) {
    if (bytes <= b.bytes && b.p) return QA_OK;
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
    if (bytes == 0) bytes = 256;
    QA_CUDA(cudaMalloc(&b.p, bytes));
    b.bytes = bytes;
    return QA_OK;
}

inline void release(DevBuf &b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
}

inline bool is_device_ptr(const void *p) {
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

inline float elapsed(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

template <typename T>
inline int upload(qa_ctx *ctx, T **dst, const T *src, size_t count) {
    *dst = nullptr;
    QA_CUDA(cudaMalloc((void **)dst, std::max<size_t>(count, 1) * sizeof(T)));
    if (count)
        QA_CUDA(cudaMemcpyAsync(*dst, src, count * sizeof(T), cudaMemcpyDefault, ctx->stream));
    return QA_OK;
}

// Interval rank-1 group term (qa_model_set_group_bounds).  u = sum_g a_v s_v + kappa, d(u) = max(lo - u, 0, u - hi),
// E = lambda * (double)(d*d) * 0.25.  Flipping a variable with spin s and coefficient a moves u to u - 2 a s; the change of the
// term is an exact integer difference, scaled by 0.25 (exact) and rounded once by the product with lambda.  For lo = hi = 0,
// d(u')^2 - d(u)^2 = 4 a (a - s u): bitwise the equality groups' lambda * (double)(a * (a - s u)).  The host keeps every
// d^2 below 2^53.
__host__ __device__ __forceinline__ long long interval_dist(long long u, long long lo, long long hi) {
    return u < lo ? lo - u : (u > hi ? u - hi : 0ll);
}
__host__ __device__ __forceinline__ double interval_flip_cost(double lam, long long a, bool up, long long u, long long lo,
                                                              long long hi) {
    const long long d0 = interval_dist(u, lo, hi);
    const long long d1 = interval_dist(up ? u - 2 * a : u + 2 * a, lo, hi);
    return lam * ((double)(d1 * d1 - d0 * d0) * 0.25);
}

// Kind of a model's rank-1 group term, decided once per launch (run_anneal) and the GROUPS template argument of every
// annealing kernel.  EQ32: equality groups whose terms the host proved to fit 32-bit integers (qa_model::groups_i32).
enum GroupKind { GK_NONE = 0, GK_EQ32 = 1, GK_EQ64 = 2, GK_INTERVAL = 3 };

// Acceptance rule of a sampling call (QA_PROPOSAL_*), the PROP template argument of every annealing kernel but the dense one
enum Proposal { PROP_METROPOLIS = QA_PROPOSAL_METROPOLIS, PROP_GIBBS = QA_PROPOSAL_GIBBS };

// 64-bit words of kappa staged per group in shared memory: {kappa, lo, hi} for interval groups, kappa otherwise
__host__ __device__ constexpr int kappa_words(GroupKind gk) { return gk == GK_INTERVAL ? 3 : 1; }

// Change of the group term when a variable with coefficient a and spin up / down flips, u = M_g + kappa_g.  Equality groups:
// lambda * (double)(a * (a - s u)), in 32-bit integers for GK_EQ32 (u then holds a 32-bit sum).  lo / hi are read for
// interval groups only.
template <GroupKind GK>
__host__ __device__ __forceinline__ double group_flip_cost(double lam, long long a, bool up, long long u, long long lo,
                                                           long long hi) {
    if (GK == GK_INTERVAL) return interval_flip_cost(lam, a, up, u, lo, hi);
    if (GK == GK_EQ32) {
        const int m = (int)u;
        const int t = (int)a * ((int)a - (up ? m : -m));
        return lam * (double)t;
    }
    const long long t = a * (a - (up ? 1 : -1) * u);
    return lam * (double)t;
}

inline unsigned blocks_for(int64_t count, int tpb = 256) { return (unsigned)std::max<int64_t>(1, (count + tpb - 1) / tpb); }

// device scratch of one build, freed on every path
struct SnnScratch {
    std::vector<void *> ptrs;
    ~SnnScratch() { for (void *p : ptrs) if (p) cudaFree(p); }
    template <typename T> cudaError_t get(T **p, size_t count) {
        cudaError_t e = cudaMalloc((void **)p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) ptrs.push_back(*p);
        return e;
    }
};

// ---- host functions that cross translation units -----------------------------------------------------------------------
// model.cu
int finalize_descs(qa_model *M);
int model_create(qa_ctx *ctx, int32_t P, const int64_t *var_off, const int64_t *cpl_off, const double *h, const int32_t *starts,
                 const int32_t *ends, const double *w, qa_model **out);
// api.cu
int sample_common(qa_ctx *ctx, qa_model *M, int32_t reads_per_problem, int8_t *states_inout, double *energies_out,
                  int32_t num_betas, const double *beta_schedule, int32_t sweeps_per_beta, const uint64_t *seeds,
                  int32_t seed_mode, int32_t mode, qa_interrupt_fn interrupt, void *iuser, qa_stats *stats_out,
                  int32_t var_order = QA_ORDER_SEQUENTIAL, int32_t proposal = QA_PROPOSAL_METROPOLIS);

// one annealing launch: what run_anneal (api.cu) hands to the kernel's own translation unit
struct Launch {
    qa_ctx *ctx;
    qa_model *M;
    AnnealParams A;        // also the launch's shape: reads_per_problem, total_reads, seed_mode
    GroupKind gk;
    Proposal prop;         // acceptance rule
    bool random_order;     // QA_ORDER_RANDOM (warp-per-read kernel only)
    qa_interrupt_fn interrupt;
    void *iuser;
    qa_stats *st;
    int64_t done;          // out: reads completed
    bool interrupted;      // out
};
int launch_ref(Launch &L);        // anneal_ref.cu
int ref_resident_reads(qa_ctx *ctx, int *out);
int launch_lockstep(Launch &L);   // anneal_lockstep.cu
int launch_replay(Launch &L);     // anneal_replay.cu
const void *replay_gibbs_kernel(const qa_model *M, GroupKind gk);   // anneal_replay_gibbs.cu
int build_replay_tables(qa_model *M);
int launch_dense(Launch &L);      // anneal_dense.cu
int launch_energy(qa_ctx *ctx, qa_model *M, int32_t reads_per_problem);            // energy.cu: k_energy on the packed spins
int launch_pack_states(qa_ctx *ctx, const ProblemDesc &D, int64_t threads);         //            caller states -> packedT
int launch_argmin(qa_ctx *ctx, const double *d_values, int64_t count);              // postprocess.cu: -> ctx->d_best_e / d_best_i

// coupling slabs of the replay kernel, host part (anneal_replay.cu; also behind the CPU test hook qa_debug_pack_slabs)
struct RpPacked {
    std::vector<uint32_t> off;          // slab offsets in 16-byte units, one terminator
    std::vector<unsigned char> slabs;
    std::vector<int64_t> blk_base;      // first slab of every problem in `off`
    std::vector<int32_t> nslabs;
    bool uniform = true;                // every block holds exactly RP_D variables
    bool adj_sorted = true;             // every adjacency list is ascending (dimod's vector order): slab order serves the set-up
    int32_t kway_k = 0;                 // cell size of the k-way sections (anneal_replay.cu), 0: none
    int64_t kway_blocks = 0;            // blocks that carry a k-way section
};
// kway = false: no k-way sections (every block in the generic form)
bool pack_replay_slabs(int P, const int64_t *var_off, const int32_t *rowptr, const int32_t *col, const double *val, int ngroups,
                       const std::vector<int32_t> &hg, const std::vector<int32_t> &hc, int slots, RpPacked &out, bool kway = true);

}  // namespace qa
