// postprocess.cu -- SampleSet post-processing on the device (SURVEY.md 8f-2).  
//
// What the reference does with a SampleSet after the sampler call (all on the host, one sample at a time):
//   response.data(fields=['sample','energy','num_occurrences'])  -- energy-sorted iteration       BQM_clustering.py:93,281,397
//   response.record.energy[0] / [3]                              -- k-th best energy              BQM_clustering.py:133-146
//   sampleset.samples()[:16]                                      -- the 16 best samples           plot_and_save.py:105-126
//   sample[(i, c)] / 'v_i,c' == 1 -> label                        -- one-hot decode of DQM / CQM   plot_and_save.py:46-63
// With 10^5 reads of 10^5 variables the int8 state matrix is 13 GB: ordering, picking and decoding on the device means only
// the k best samples (and the labels) cross PCIe.
#include "common.cuh"

#include <cub/device/device_radix_sort.cuh>

using namespace qa;

namespace {

// (x, i) comes before (e, j) in the order of qa_sort_reads: a NaN after every number, equal values (-0.0 == +0.0) and two
// NaNs by index
__device__ __forceinline__ bool argmin_before(double x, long long i, double e, long long j) {
    const bool xn = x != x, en = e != e;
    if (xn != en) return en;
    return xn ? i < j : (x < e || (x == e && i < j));
}

// warp-shuffle min / argmin in the order of the sort (-> SampleSet.first).  A thread without values holds (NaN, INT64_MAX),
// which every value passes, so for count >= 1 the result is a value of the input and its index; all NaN: (values[0], 0).
__global__ void __launch_bounds__(1024) k_argmin(const double *energies, int64_t count, double *best_e, long long *best_i) {
    __shared__ double se[32];
    __shared__ long long si[32];
    const double none = __longlong_as_double(0x7ff8000000000000ll);
    double e = none;
    long long idx = 0x7fffffffffffffffll;
    for (int64_t i = threadIdx.x; i < count; i += blockDim.x) {
        const double x = energies[i];
        if (argmin_before(x, i, e, idx)) { e = x; idx = i; }
    }
    for (int off = 16; off > 0; off >>= 1) {
        const double oe = __shfl_xor_sync(FULL_MASK, e, off);
        const long long oi = __shfl_xor_sync(FULL_MASK, idx, off);
        if (argmin_before(oe, oi, e, idx)) { e = oe; idx = oi; }
    }
    if ((threadIdx.x & 31) == 0) { se[threadIdx.x >> 5] = e; si[threadIdx.x >> 5] = idx; }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int nw = (blockDim.x + 31) >> 5;
        e = threadIdx.x < nw ? se[threadIdx.x] : none;
        idx = threadIdx.x < nw ? si[threadIdx.x] : 0x7fffffffffffffffll;
        for (int off = 16; off > 0; off >>= 1) {
            const double oe = __shfl_xor_sync(FULL_MASK, e, off);
            const long long oi = __shfl_xor_sync(FULL_MASK, idx, off);
            if (argmin_before(oe, oi, e, idx)) { e = oe; idx = oi; }
        }
        if (threadIdx.x == 0) { *best_e = e; *best_i = idx; }
    }
}

// order-preserving map double -> uint64 (ascending): x + 0.0 turns -0.0 into +0.0, so the two tie; every NaN, whatever its
// sign and payload, gets the largest key and so sorts after +inf (in read order: the radix sort is stable)
__global__ void k_energy_keys(int32_t count, const double *e, unsigned long long *keys, int32_t *idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    idx[i] = i;
    if (!e) return;   // index ramp only
    const double x = e[i];
    unsigned long long b = (unsigned long long)__double_as_longlong(x + 0.0);
    b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
    keys[i] = x != x ? ~0ull : b;
}

// samples_out[r] = states[order[r]] for r < k  (one block per output row, coalesced 16-byte copies when aligned)
__global__ void k_gather_rows(int32_t n, const int8_t *states, const int32_t *order, int8_t *out) {
    const int8_t *src = states + (int64_t)order[blockIdx.x] * n;
    int8_t *dst = out + (int64_t)blockIdx.x * n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}

// one thread per (read, cell): label = the single case whose bit is set, -1 if the cell is not one-hot
__global__ void k_decode_onehot(int32_t cells, int32_t K, int64_t stride, int32_t reads, const int8_t *states, int32_t on_value,
                                int32_t *labels, int32_t *sizes, int32_t *violations) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)reads * cells) return;
    const int32_t r = (int32_t)(t / cells), c = (int32_t)(t % cells);
    const int8_t *row = states + (int64_t)r * stride + (int64_t)c * K;
    int cnt = 0, lab = -1;
    for (int k = 0; k < K; ++k)
        if (row[k] == on_value) { ++cnt; lab = k; }
    if (cnt != 1) {
        lab = -1;
        atomicAdd(violations + 2 * r, 1);
    } else {
        atomicAdd(sizes + (int64_t)r * K + lab, 1);
    }
    if (labels) labels[t] = lab;
}

__global__ void k_count_small_clusters(int32_t reads, int32_t K, int32_t min_size, const int32_t *sizes, int32_t *violations) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= reads) return;
    int bad = 0;
    for (int k = 0; k < K; ++k) bad += sizes[(int64_t)r * K + k] < min_size;
    violations[2 * r + 1] = bad;
}

// counter-based initial states: spin (r, v) = bit (v & 63) of splitmix64(seed, global read r, word v >> 6); 1 -> -1.
// Depends only on (seed, global read index, variable): identical for any sharding of the reads over GPUs, and restated in
// numpy by schedule.counter_spin_states for the host path.
__host__ __device__ inline unsigned long long qa_mix64(unsigned long long seed, unsigned long long r, unsigned long long w) {
    unsigned long long z = (seed + 1ull) * 0xD1342543DE82EF95ull + r * 0x9E3779B97F4A7C15ull + w * 0xC2B2AE3D27D4EB4Full;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__global__ void k_random_states(unsigned long long seed, int64_t first_read, int32_t reads, int32_t n, int8_t *states) {
    const int64_t words = ((int64_t)n + 63) / 64;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)reads * words) return;
    const int64_t r = t / words, w = t % words;
    const unsigned long long bits = qa_mix64(seed, (unsigned long long)(first_read + r), (unsigned long long)w);
    int8_t *row = states + r * (int64_t)n + w * 64;
    const int lim = (int)min((int64_t)64, (int64_t)n - w * 64);
    for (int i = 0; i < lim; ++i) row[i] = ((bits >> i) & 1ull) ? -1 : 1;
}

// 2 x 64-bit hash of every row (one block per read): duplicate detection for SampleSet.aggregate()
__global__ void k_hash_rows(int32_t n, const int8_t *states, unsigned long long *h1, unsigned long long *h2) {
    const int8_t *row = states + (int64_t)blockIdx.x * n;
    unsigned long long a = 0x9E3779B97F4A7C15ull, b = 0xC2B2AE3D27D4EB4Full;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const unsigned long long x = (unsigned long long)(unsigned char)row[i] + 1ull;
        a += qa_mix64(x, (unsigned long long)i, 1ull);          // order-independent sum of position-keyed mixes
        b ^= qa_mix64(x, (unsigned long long)i, 2ull) * 0x9E3779B97F4A7C15ull;
    }
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b ^= __shfl_xor_sync(0xffffffffu, b, o);
    }
    __shared__ unsigned long long sa[32], sb[32];
    if ((threadIdx.x & 31) == 0) { sa[threadIdx.x >> 5] = a; sb[threadIdx.x >> 5] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { a += sa[w]; b ^= sb[w]; }
        h1[blockIdx.x] = a;
        h2[blockIdx.x] = b;
    }
}

// sorted position p (reads ordered by h1, ties in read order): head[p] = 1 when read idx[p] differs from read idx[p-1]
// (both hashes, then the full rows: one block per position)
__global__ void k_mark_heads(int32_t n, const int8_t *states, const unsigned long long *h1s, const int32_t *idx,
                             const unsigned long long *h2, int32_t *head) {
    const int p = blockIdx.x;
    if (p == 0) { if (threadIdx.x == 0) head[0] = 1; return; }
    const int a = idx[p], b = idx[p - 1];
    __shared__ int differ;
    if (threadIdx.x == 0) differ = (h1s[p] != h1s[p - 1] || h2[a] != h2[b]) ? 1 : 0;
    __syncthreads();
    if (!differ) {
        const int8_t *ra = states + (int64_t)a * n, *rb = states + (int64_t)b * n;
        int d = 0;
        for (int i = threadIdx.x; i < n; i += blockDim.x) d |= ra[i] != rb[i];
        if (d) atomicOr(&differ, 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) head[p] = differ;
}

// stage `bytes` of a caller buffer (host or device) on the device; returns the device pointer to use
__global__ void k_argmin_pack(const double *best_e, const long long *best_i, long long offset, double *out) {
    out[0] = *best_e;
    out[1] = (double)(*best_i + offset);   // k_argmin of count >= 1 values gives an index in [0, count); read indices are < 2^53: exact
}

int stage_in(qa_ctx *ctx, DevBuf &buf, const void *p, size_t bytes, const void **dev) {
    if (is_device_ptr(p)) { *dev = p; return QA_OK; }
    int rc = ensure(buf, bytes);
    if (rc) return rc;
    QA_CUDA(cudaMemcpyAsync(buf.p, p, bytes, cudaMemcpyHostToDevice, ctx->stream));
    *dev = buf.p;
    return QA_OK;
}

}  // namespace

namespace qa {

int launch_argmin(qa_ctx *ctx, const double *d_values, int64_t count) {
    k_argmin<<<1, 1024, 0, ctx->stream>>>(d_values, count, ctx->d_best_e, ctx->d_best_i);
    QA_CUDA(cudaGetLastError());
    ctx->launches++;
    return QA_OK;
}

}  // namespace qa

extern "C" {

int qa_sort_reads(qa_ctx *ctx, int32_t num_reads, const double *energies, int32_t *order_out) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    if (num_reads < 0) return fail(QA_ERR_ARG, "negative num_reads");
    if (num_reads == 0) return QA_OK;
    if (!energies || !order_out) return fail(QA_ERR_ARG, "null energies / order");
    QA_CUDA(cudaSetDevice(ctx->device));
    const void *d_e = nullptr;
    int rc = stage_in(ctx, ctx->energies, energies, (size_t)num_reads * sizeof(double), &d_e);
    if (rc) return rc;
    // scratch: keys, keys2 (u64), idx, idx2 (i32)
    const size_t kb = (size_t)num_reads * sizeof(unsigned long long), ib = (size_t)num_reads * sizeof(int32_t);
    rc = ensure(ctx->misc, 2 * kb + 2 * ib + 64);
    if (rc) return rc;
    unsigned long long *keys = (unsigned long long *)ctx->misc.p, *keys2 = keys + num_reads;
    int32_t *idx = (int32_t *)(keys2 + num_reads), *idx2 = idx + num_reads;
    k_energy_keys<<<(num_reads + 255) / 256, 256, 0, ctx->stream>>>(num_reads, (const double *)d_e, keys, idx);
    ctx->launches++;
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, keys, keys2, idx, idx2, num_reads, 0, 64, ctx->stream);
    rc = ensure(ctx->cubtmp, tmp);
    if (rc) return rc;
    cudaError_t ce = cub::DeviceRadixSort::SortPairs(ctx->cubtmp.p, tmp, keys, keys2, idx, idx2, num_reads, 0, 64, ctx->stream);
    if (ce != cudaSuccess) return fail(QA_ERR_CUDA, std::string("radix sort: ") + cudaGetErrorString(ce));
    ctx->launches += 8;
    QA_CUDA(cudaMemcpyAsync(order_out, idx2, ib, cudaMemcpyDefault, ctx->stream));   // radix sort is stable: ties keep read order
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    return QA_OK;
}

int qa_gather_samples(qa_ctx *ctx, int32_t n, int32_t num_reads, const int8_t *states, int32_t k, const int32_t *order,
                      int8_t *samples_out) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    if (n < 0 || num_reads < 0 || k < 0) return fail(QA_ERR_ARG, "negative size");
    if (k == 0 || n == 0) return QA_OK;
    if (!states || !order || !samples_out) return fail(QA_ERR_ARG, "null states / order / samples_out");
    QA_CUDA(cudaSetDevice(ctx->device));
    std::vector<int32_t> ho(k);
    QA_CUDA(cudaMemcpy(ho.data(), order, (size_t)k * sizeof(int32_t), cudaMemcpyDefault));
    for (int32_t r : ho)
        if (r < 0 || r >= num_reads) return fail(QA_ERR_INDEX, "order entry out of range");
    if (!is_device_ptr(states)) {   // host matrix: nothing to gain from the device, copy the rows directly
        for (int32_t r = 0; r < k; ++r)
            QA_CUDA(cudaMemcpy(samples_out + (int64_t)r * n, states + (int64_t)ho[r] * n, (size_t)n, cudaMemcpyDefault));
        return QA_OK;
    }
    int rc = ensure(ctx->seeds, (size_t)k * sizeof(int32_t));
    if (rc) return rc;
    QA_CUDA(cudaMemcpyAsync(ctx->seeds.p, ho.data(), (size_t)k * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    int8_t *d_out = samples_out;
    const bool out_host = !is_device_ptr(samples_out);
    if (out_host) {
        rc = ensure(ctx->packed, (size_t)k * n);
        if (rc) return rc;
        d_out = (int8_t *)ctx->packed.p;
    }
    k_gather_rows<<<k, 256, 0, ctx->stream>>>(n, states, (const int32_t *)ctx->seeds.p, d_out);
    QA_CUDA(cudaGetLastError());
    ctx->launches++;
    if (out_host) QA_CUDA(cudaMemcpyAsync(samples_out, d_out, (size_t)k * n, cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    return QA_OK;
}

int qa_decode_onehot(qa_ctx *ctx, int32_t cells, int32_t K, int64_t stride, int32_t num_reads, const int8_t *states,
                     int32_t on_value, int32_t min_size, int32_t *labels_out, int32_t *violations_out) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    if (cells < 0 || K < 1 || num_reads < 0 || stride < (int64_t)cells * K) return fail(QA_ERR_ARG, "bad one-hot geometry");
    if (num_reads == 0 || cells == 0) return QA_OK;
    if (!states || !violations_out) return fail(QA_ERR_ARG, "null states / violations");   // labels_out may be NULL: counts only
    QA_CUDA(cudaSetDevice(ctx->device));
    const void *d_states = nullptr;
    int rc = stage_in(ctx, ctx->states, states, (size_t)num_reads * stride, &d_states);
    if (rc) return rc;
    const size_t lb = labels_out ? (size_t)num_reads * cells * sizeof(int32_t) : 0, sb = (size_t)num_reads * K * sizeof(int32_t),
                 vb = (size_t)num_reads * 2 * sizeof(int32_t);
    rc = ensure(ctx->misc, lb + sb + vb + 64);
    if (rc) return rc;
    int32_t *d_lab = (int32_t *)ctx->misc.p, *d_sizes = d_lab + lb / sizeof(int32_t), *d_viol = d_sizes + (size_t)num_reads * K;
    QA_CUDA(cudaMemsetAsync(d_sizes, 0, sb + vb, ctx->stream));
    const int64_t total = (int64_t)num_reads * cells;
    k_decode_onehot<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(cells, K, stride, num_reads, (const int8_t *)d_states,
                                                                               on_value, labels_out ? d_lab : nullptr, d_sizes, d_viol);
    k_count_small_clusters<<<(num_reads + 255) / 256, 256, 0, ctx->stream>>>(num_reads, K, min_size, d_sizes, d_viol);
    QA_CUDA(cudaGetLastError());
    ctx->launches += 2;
    if (labels_out) QA_CUDA(cudaMemcpyAsync(labels_out, d_lab, lb, cudaMemcpyDefault, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(violations_out, d_viol, vb, cudaMemcpyDefault, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    return QA_OK;
}

int qa_dev_alloc(qa_ctx *ctx, int64_t bytes, void **out) {
    if (!ctx || !out || bytes < 0) return fail(QA_ERR_ARG, "bad arguments");
    *out = nullptr;
    QA_CUDA(cudaSetDevice(ctx->device));
    QA_CUDA(cudaMalloc(out, (size_t)std::max<int64_t>(bytes, 1)));
    return QA_OK;
}

int qa_dev_free(qa_ctx *ctx, void *p) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    if (!p) return QA_OK;
    QA_CUDA(cudaSetDevice(ctx->device));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    QA_CUDA(cudaFree(p));
    return QA_OK;
}

int qa_dev_copy(qa_ctx *ctx, void *dst, const void *src, int64_t bytes) {
    if (!ctx || bytes < 0) return fail(QA_ERR_ARG, "bad arguments");
    if (bytes == 0) return QA_OK;
    if (!dst || !src) return fail(QA_ERR_ARG, "null pointer");
    QA_CUDA(cudaSetDevice(ctx->device));
    QA_CUDA(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDefault, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    return QA_OK;
}

int qa_random_states(qa_ctx *ctx, uint64_t seed, int64_t first_read, int32_t num_reads, int32_t n, int8_t *states_out) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    if (num_reads < 0 || n < 0 || first_read < 0) return fail(QA_ERR_ARG, "negative size");
    if (num_reads == 0 || n == 0) return QA_OK;
    if (!states_out) return fail(QA_ERR_ARG, "null states_out");
    QA_CUDA(cudaSetDevice(ctx->device));
    const int64_t bytes = (int64_t)num_reads * n;
    int8_t *d_out = states_out;
    const bool out_host = !is_device_ptr(states_out);
    if (out_host) {
        int rc = ensure(ctx->states, (size_t)bytes);
        if (rc) return rc;
        d_out = (int8_t *)ctx->states.p;
    }
    const int64_t threads = (int64_t)num_reads * (((int64_t)n + 63) / 64);
    k_random_states<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->stream>>>((unsigned long long)seed, first_read, num_reads, n, d_out);
    QA_CUDA(cudaGetLastError());
    ctx->launches++;
    if (out_host) QA_CUDA(cudaMemcpyAsync(states_out, d_out, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    return QA_OK;
}

int qa_aggregate_reads(qa_ctx *ctx, int32_t n, int32_t num_reads, const int8_t *states, int32_t *num_unique_out,
                       int32_t *first_index_out, int32_t *count_out) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    if (n < 0 || num_reads < 0) return fail(QA_ERR_ARG, "negative size");
    if (!num_unique_out) return fail(QA_ERR_ARG, "null num_unique_out");
    *num_unique_out = 0;
    if (num_reads == 0) return QA_OK;
    if (!first_index_out || !count_out) return fail(QA_ERR_ARG, "null outputs");
    if (n == 0) {   // every read is the empty sample: one group, nothing to read
        first_index_out[0] = 0;
        count_out[0] = num_reads;
        *num_unique_out = 1;
        return QA_OK;
    }
    if (!states) return fail(QA_ERR_ARG, "null states");
    QA_CUDA(cudaSetDevice(ctx->device));
    const void *d_states = nullptr;
    int rc = stage_in(ctx, ctx->states, states, (size_t)num_reads * n, &d_states);
    if (rc) return rc;
    const size_t R = (size_t)num_reads;
    // scratch: h1, h1s, h2 (u64), idx, idxs, head (i32)
    rc = ensure(ctx->misc, 3 * R * sizeof(unsigned long long) + 3 * R * sizeof(int32_t) + 64);
    if (rc) return rc;
    unsigned long long *h1 = (unsigned long long *)ctx->misc.p, *h1s = h1 + R, *h2 = h1s + R;
    int32_t *idx = (int32_t *)(h2 + R), *idxs = idx + R, *head = idxs + R;
    k_hash_rows<<<num_reads, 128, 0, ctx->stream>>>(n, (const int8_t *)d_states, h1, h2);
    k_energy_keys<<<(num_reads + 255) / 256, 256, 0, ctx->stream>>>(num_reads, nullptr, nullptr, idx);   // idx = 0 .. R-1
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, h1, h1s, idx, idxs, num_reads, 0, 64, ctx->stream);
    rc = ensure(ctx->cubtmp, tmp);
    if (rc) return rc;
    cudaError_t ce = cub::DeviceRadixSort::SortPairs(ctx->cubtmp.p, tmp, h1, h1s, idx, idxs, num_reads, 0, 64, ctx->stream);
    if (ce != cudaSuccess) return fail(QA_ERR_CUDA, std::string("radix sort: ") + cudaGetErrorString(ce));
    k_mark_heads<<<num_reads, 128, 0, ctx->stream>>>(n, (const int8_t *)d_states, h1s, idxs, h2, head);
    QA_CUDA(cudaGetLastError());
    ctx->launches += 11;
    // the group structure is tiny next to the state matrix: finish on the host (R x 8 bytes leave the device)
    std::vector<int32_t> hidx(R), hhead(R);
    QA_CUDA(cudaMemcpyAsync(hidx.data(), idxs, R * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(hhead.data(), head, R * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    // groups are runs of the h1-sorted order (stable: inside a run reads ascend), split where k_mark_heads found a different
    // row.  Exact unless two distinct rows share the 64-bit h1 and their reads interleave (A, B, A in read order): then A's
    // reads form two groups.  No merge pass for that: the chance of an h1 collision is about R^2 / 2^65 per call.
    std::vector<std::pair<int32_t, int32_t>> groups;   // (first read index, count)
    for (size_t p = 0; p < R; ++p) {
        if (hhead[p]) groups.emplace_back(hidx[p], 1);
        else groups.back().second++;
    }
    std::sort(groups.begin(), groups.end());          // dimod.SampleSet.aggregate keeps the order of first occurrence
    for (size_t u = 0; u < groups.size(); ++u) {
        first_index_out[u] = groups[u].first;
        count_out[u] = groups[u].second;
    }
    *num_unique_out = (int32_t)groups.size();
    return QA_OK;
}

int qa_argmin(qa_ctx *ctx, int64_t count, const double *values, double *best_value, int64_t *best_index) {
    if (!ctx) return fail(QA_ERR_ARG, "null context");
    if (count < 0) return fail(QA_ERR_ARG, "negative count");
    if (count == 0) {
        if (best_value) *best_value = INFINITY;
        if (best_index) *best_index = -1;
        return QA_OK;
    }
    if (!values) return fail(QA_ERR_ARG, "null values");
    QA_CUDA(cudaSetDevice(ctx->device));
    const void *d_v = nullptr;
    int rc = stage_in(ctx, ctx->energies, values, (size_t)count * sizeof(double), &d_v);
    if (rc) return rc;
    k_argmin<<<1, 1024, 0, ctx->stream>>>((const double *)d_v, count, ctx->d_best_e, ctx->d_best_i);
    QA_CUDA(cudaGetLastError());
    ctx->launches++;
    double be = 0;
    long long bi = 0;
    QA_CUDA(cudaMemcpyAsync(&be, ctx->d_best_e, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaMemcpyAsync(&bi, ctx->d_best_i, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    if (best_value) *best_value = be;
    if (best_index) *best_index = bi;
    return QA_OK;
}

// SURVEY 2.2 K6 / N1: the per-rank half of the multi-GPU best-sample exchange writes (best energy, GLOBAL read index) straight
// into the device buffer the caller hands to its all_gather (16 bytes per rank) -- no host round trip between the reduction
// and the collective.
int qa_argmin_device(qa_ctx *ctx, int64_t count, const double *values, int64_t index_offset, double *out_device) {
    if (!ctx || !out_device) return fail(QA_ERR_ARG, "null argument");
    if (count < 1 || !values) return fail(QA_ERR_ARG, "need at least one value");
    if (!is_device_ptr(out_device)) return fail(QA_ERR_ARG, "out_device must be device memory (the collective's send buffer)");
    QA_CUDA(cudaSetDevice(ctx->device));
    const void *d_v = nullptr;
    int rc = stage_in(ctx, ctx->energies, values, (size_t)count * sizeof(double), &d_v);
    if (rc) return rc;
    k_argmin<<<1, 1024, 0, ctx->stream>>>((const double *)d_v, count, ctx->d_best_e, ctx->d_best_i);
    k_argmin_pack<<<1, 1, 0, ctx->stream>>>(ctx->d_best_e, ctx->d_best_i, index_offset, out_device);
    QA_CUDA(cudaGetLastError());
    ctx->launches += 2;
    QA_CUDA(cudaStreamSynchronize(ctx->stream));
    return QA_OK;
}

int64_t qa_model_replay_kway(const qa_model *M, int32_t *k_out) {
    if (!M) return fail(QA_ERR_ARG, "null model");
    const bool on = M->rp_ok && M->rp_kway_blocks > 0;
    if (k_out) *k_out = on ? M->rp_kway_k : 0;
    return on ? M->rp_kway_blocks : 0;
}

/* Test hook, host only (no device needed): pack the replay kernel's coupling slabs for one problem whose CSR (adjacency order,
 * rowptr[n + 1], col, val) is in host memory.  Returns 1 when the model fits the slab format (0: it does not, negative: error);
 * on success *nslabs_out / *bytes_out / *uniform_out are set and, when the buffers are given (bytes_out reports the size to
 * allocate), slabs_out receives the serialized slabs and off_out[nslabs + 1] their offsets in 16-byte units. */
int qa_debug_pack_slabs(int32_t n, const int32_t *rowptr, const int32_t *col, const double *val, int32_t ngroups,
                        const int32_t *grp, const int32_t *coef, int64_t *nslabs_out, int64_t *bytes_out, int32_t *uniform_out,
                        unsigned char *slabs_out, uint32_t *off_out) {
    if (n < 1 || !rowptr || !nslabs_out || !bytes_out || !uniform_out) return fail(QA_ERR_ARG, "bad arguments");
    const int64_t npad = ((int64_t)n + 31) / 32 * 32;   // covers the packer's 16-variable padding
    std::vector<int32_t> rp(npad + 1);
    for (int64_t v = 0; v <= npad; ++v) rp[v] = rowptr[std::min<int64_t>(v, n)];
    std::vector<int32_t> hg, hc;
    if (ngroups > 0) {
        if (!grp || !coef) return fail(QA_ERR_ARG, "null group vectors");
        hg.assign(npad, -1);
        hc.assign(npad, 0);
        for (int32_t v = 0; v < n; ++v) { hg[v] = grp[v]; hc[v] = coef[v]; }
    }
    const int64_t var_off[2] = {0, n};
    RpPacked pk;
    const char *kw_env = getenv("QA_REPLAY_KWAY");   // as qa_ctx_create reads it
    const bool kw = !(kw_env && atoi(kw_env) == 0);
    if (!pack_replay_slabs(1, var_off, rp.data(), col, val, ngroups, hg, hc, 32, pk, kw) &&
        !pack_replay_slabs(1, var_off, rp.data(), col, val, ngroups, hg, hc, 64, pk, kw)) return 0;
    *nslabs_out = pk.nslabs[0];
    *bytes_out = (int64_t)pk.slabs.size();
    *uniform_out = pk.uniform ? 1 : 0;
    if (slabs_out) memcpy(slabs_out, pk.slabs.data(), pk.slabs.size());
    if (off_out) memcpy(off_out, pk.off.data(), pk.off.size() * sizeof(uint32_t));
    return 1;
}

}  // extern "C"
