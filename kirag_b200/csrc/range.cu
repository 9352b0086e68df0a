// range.cu — range search (faiss IndexFlatIP::range_search): every row whose canonical score is above a radius.
//
// The entries of a query come from one of two sources:
//   CandSource   the candidate buffer of ONE bf16 filter scan with the fixed threshold radius - eps(q) - <q, c>,
//                rescored in fp32 (filter path: a superset of the answer by the eps bound, exact after rescoring)
//   DenseSource  the dense fp32 scores of the exact scan (exact path)
// and leave through the same steps:
//   range_count_kernel     per-query number of entries with score > radius (NaN fails the test)
//   range_collect_kernel   appends them, packed as 64-bit sort items (common.cuh: pack_item), to the query's segment
//                          of a flat item array; positions inside a segment are reserved with atomics, so the
//                          segment is unordered until it is sorted below
//   range_emit_kernel      segments of at most kRangeRun items: one CTA sorts the segment in shared memory (bitonic)
//                          and writes D / I (row + id_offset) at the query's offset of the result
//   longer segments        range_sort_runs_kernel sorts runs of kRangeRun items in place, range_merge_kernel merges
//                          neighbouring runs by rank (own position + binary-search rank in the sibling run, the way
//                          exchange.cu merges shard lists) until one run is left, range_write_kernel writes D / I
// The keys are distinct (rows are), so the result does not depend on the order in which entries were appended.
#include "common.cuh"

namespace kirag {

constexpr int kRangeThreads = 256;
constexpr int kRangeSortThreads = 512;

struct CandSource {
    const Cand* cand;
    int64_t cap;      // candidate slots per query
    const float* scores;
    int64_t m;        // rescored scores per query (>= every complete buffer's count)
    const int* cnt;
    __device__ __forceinline__ int64_t count(int64_t q) const {
        const int c = cnt[q];
        return c > cap ? 0 : c;  // an overflowed buffer is incomplete: that query is answered by another pass
    }
    __device__ __forceinline__ bool get(int64_t q, int64_t j, float* s, int32_t* row) const {
        const int32_t id = cand[q * cap + j].id;
        if (id < 0) return false;
        *s = scores[q * m + j];
        *row = id;
        return true;
    }
};

struct DenseSource {
    const float* scores;
    int64_t ld, n;
    __device__ __forceinline__ int64_t count(int64_t) const { return n; }
    __device__ __forceinline__ bool get(int64_t q, int64_t j, float* s, int32_t* row) const {
        *s = scores[q * ld + j];
        *row = (int32_t)j;
        return true;
    }
};

__global__ void range_threshold_kernel(const int* __restrict__ qmap, const float* __restrict__ qnorm,
                                       const float* __restrict__ qerr, const float* __restrict__ qcdot, float radius,
                                       float eps_a, float eps_b, int64_t nb, int64_t nb_pad, float* __restrict__ tau,
                                       int* __restrict__ cnt) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb_pad) return;
    if (i >= nb) { tau[i] = INFINITY; return; }
    const int64_t q = qmap ? qmap[i] : i;
    // the shadow holds x - c: its scores are lower than the true ones by <q, c>
    float t = radius - (eps_a * qnorm[q] + eps_b * qerr[q]) - qcdot[q];
    if (!(t == t)) t = -INFINITY;  // non-finite query norms: keep everything, rescoring decides
    tau[i] = t;
    cnt[i] = 0;
}

// grid (slices, queries): the block's strided share of query blockIdx.y's entries
template <class Src>
__device__ __forceinline__ int block_hits(const Src& src, int64_t q, float radius, int* s_part) {
    const int64_t n = src.count(q);
    int c = 0;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        float s;
        int32_t row;
        if (src.get(q, j, &s, &row) && s > radius) ++c;
    }
    c = __reduce_add_sync(0xffffffffu, c);
    if (threadIdx.x == 0) *s_part = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(s_part, c);
    __syncthreads();
    return *s_part;
}

template <class Src>
__global__ void __launch_bounds__(kRangeThreads) range_count_kernel(Src src, float radius, int* __restrict__ counts) {
    __shared__ int s_part;
    const int64_t q = blockIdx.y;
    const int part = block_hits(src, q, radius, &s_part);
    if (threadIdx.x == 0 && part) atomicAdd(counts + q, part);
}

template <class Src>
__global__ void __launch_bounds__(kRangeThreads) range_collect_kernel(Src src, float radius,
                                                                      unsigned long long* __restrict__ cursor,
                                                                      uint64_t* __restrict__ items) {
    __shared__ int s_part;
    __shared__ unsigned long long s_base;
    __shared__ int s_pos;
    const int64_t q = blockIdx.y;
    const int part = block_hits(src, q, radius, &s_part);
    if (part == 0) return;
    if (threadIdx.x == 0) {
        s_base = atomicAdd(cursor + q, (unsigned long long)part);
        s_pos = 0;
    }
    __syncthreads();
    const int64_t n = src.count(q);
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        float s;
        int32_t row;
        if (src.get(q, j, &s, &row) && s > radius) items[s_base + atomicAdd(&s_pos, 1)] = pack_item(s, row);
    }
}

// loads len (<= kRangeRun) items into shared memory and sorts them descending
__device__ __forceinline__ void load_and_sort(uint64_t* sm, const uint64_t* src, int len) {
    int P = 32;
    while (P < len) P <<= 1;
    for (int i = threadIdx.x; i < P; i += blockDim.x) sm[i] = (i < len) ? src[i] : 0ull;  // key 0 (NaN) sorts last
    __syncthreads();
    bitonic_sort_desc(sm, P);
}

__device__ __forceinline__ void write_result(uint64_t it, int64_t id_offset, float* D, int64_t* I) {
    *D = key_score(item_key(it));
    *I = (int64_t)item_id(it) + id_offset;
}

// grid nq: the segments of at most kRangeRun items
__global__ void __launch_bounds__(kRangeSortThreads) range_emit_kernel(const uint64_t* __restrict__ items,
                                                                       const int64_t* __restrict__ src_off,
                                                                       const int64_t* __restrict__ lims, int64_t id_offset,
                                                                       float* __restrict__ D, int64_t* __restrict__ I) {
    extern __shared__ uint64_t sm[];
    const int64_t q = blockIdx.x;
    const int64_t lo = lims[q], len = lims[q + 1] - lo;
    if (len == 0 || len > kRangeRun) return;
    load_and_sort(sm, items + src_off[q], (int)len);
    for (int j = threadIdx.x; j < (int)len; j += blockDim.x) write_result(sm[j], id_offset, D + lo + j, I + lo + j);
}

// grid (runs of the longest segment, long segments): run blockIdx.x of segment blockIdx.y, sorted in place
__global__ void __launch_bounds__(kRangeSortThreads) range_sort_runs_kernel(uint64_t* __restrict__ items,
                                                                            const int64_t* __restrict__ seg_src,
                                                                            const int64_t* __restrict__ seg_len) {
    extern __shared__ uint64_t sm[];
    const int64_t s = blockIdx.y, r0 = (int64_t)blockIdx.x * kRangeRun, len = seg_len[s];
    if (r0 >= len) return;
    const int n = (int)((len - r0 < kRangeRun) ? (len - r0) : kRangeRun);
    uint64_t* p = items + seg_src[s] + r0;
    load_and_sort(sm, p, n);
    for (int j = threadIdx.x; j < n; j += blockDim.x) p[j] = sm[j];
}

// segment of flat element t: the last s with seg_e0[s] <= t
__device__ __forceinline__ int find_segment(const int64_t* seg_e0, int n_seg, int64_t t) {
    int a = 0, b = n_seg - 1;
    while (a < b) {
        const int m = (a + b + 1) >> 1;
        if (seg_e0[m] <= t) a = m; else b = m - 1;
    }
    return a;
}

// One merge pass over every element of the long segments: sorted runs of w items, pairs (2i, 2i+1) become one run
// of 2w.  An element's new position = its position in its own run + the number of sibling elements ahead of it.
__global__ void range_merge_kernel(const uint64_t* __restrict__ src, uint64_t* __restrict__ dst,
                                   const int64_t* __restrict__ seg_src, const int64_t* __restrict__ seg_len,
                                   const int64_t* __restrict__ seg_e0, int n_seg, int64_t total, int64_t w) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int s = find_segment(seg_e0, n_seg, t);
    const int64_t e = t - seg_e0[s], len = seg_len[s];
    const uint64_t* seg = src + seg_src[s];
    const int64_t run = e / w, rs = run * w;
    int64_t sib_lo, sib_hi, out0;
    if (run & 1) {
        sib_lo = rs - w; sib_hi = rs; out0 = sib_lo;
    } else {
        sib_lo = rs + w; sib_hi = (rs + 2 * w < len) ? rs + 2 * w : len; out0 = rs;
        if (sib_hi < sib_lo) sib_hi = sib_lo;
    }
    const uint64_t v = seg[e];
    int64_t a = sib_lo, b = sib_hi;  // first sibling item below v (runs are descending, keys distinct)
    while (a < b) {
        const int64_t m = (a + b) >> 1;
        if (seg[m] > v) a = m + 1; else b = m;
    }
    dst[seg_src[s] + out0 + (e - rs) + (a - sib_lo)] = v;
}

__global__ void range_write_kernel(const uint64_t* __restrict__ items, const int64_t* __restrict__ seg_src,
                                   const int64_t* __restrict__ seg_dst, const int64_t* __restrict__ seg_e0, int n_seg,
                                   int64_t total, int64_t id_offset, float* __restrict__ D, int64_t* __restrict__ I) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int s = find_segment(seg_e0, n_seg, t);
    const int64_t e = t - seg_e0[s];
    write_result(items[seg_src[s] + e], id_offset, D + seg_dst[s] + e, I + seg_dst[s] + e);
}

// ------------------------------------------------------------------ hosts ----
int launch_range_threshold(const int* qmap, const float* qnorm, const float* qerr, const float* qcdot, float radius,
                           float eps_a, float eps_b, int64_t nb, int64_t nb_pad, float* tau, int* cnt, cudaStream_t st) {
    if (nb_pad <= 0) return 0;
    range_threshold_kernel<<<(unsigned)((nb_pad + 255) / 256), 256, 0, st>>>(qmap, qnorm, qerr, qcdot, radius, eps_a,
                                                                            eps_b, nb, nb_pad, tau, cnt);
    KIRAG_LAUNCH_OK("range_threshold_kernel");
    return 0;
}

// slices per query: about 16 items per thread, at most 4096 blocks per query
static dim3 range_grid(int64_t longest, int64_t nq) {
    int64_t x = (longest + 16 * kRangeThreads - 1) / (16 * kRangeThreads);
    if (x < 1) x = 1;
    if (x > 4096) x = 4096;
    return dim3((unsigned)x, (unsigned)nq);
}

template <class Src>
static int range_count(const Src& src, int64_t longest, int64_t nq, float radius, int* counts, cudaStream_t st) {
    KIRAG_CHECK(nq <= 65535, "range_count: %lld queries in one launch", (long long)nq);
    KIRAG_CUDA_OK(cudaMemsetAsync(counts, 0, (size_t)nq * sizeof(int), st));
    range_count_kernel<Src><<<range_grid(longest, nq), kRangeThreads, 0, st>>>(src, radius, counts);
    KIRAG_LAUNCH_OK("range_count_kernel");
    return 0;
}

template <class Src>
static int range_collect(const Src& src, int64_t longest, int64_t nq, float radius, unsigned long long* cursor,
                         uint64_t* items, cudaStream_t st) {
    KIRAG_CHECK(nq <= 65535, "range_collect: %lld queries in one launch", (long long)nq);
    range_collect_kernel<Src><<<range_grid(longest, nq), kRangeThreads, 0, st>>>(src, radius, cursor, items);
    KIRAG_LAUNCH_OK("range_collect_kernel");
    return 0;
}

int launch_range_count_cand(const Cand* cand, int cap, const float* rescored, int m, const int* cnt, int64_t nq,
                            float radius, int* counts, cudaStream_t st) {
    if (nq <= 0) return 0;
    return range_count(CandSource{cand, cap, rescored, m, cnt}, m, nq, radius, counts, st);
}

int launch_range_collect_cand(const Cand* cand, int cap, const float* rescored, int m, const int* cnt, int64_t nq,
                              float radius, unsigned long long* cursor, uint64_t* items, cudaStream_t st) {
    if (nq <= 0) return 0;
    return range_collect(CandSource{cand, cap, rescored, m, cnt}, m, nq, radius, cursor, items, st);
}

int launch_range_count_dense(const float* scores, int64_t ld, int64_t n, int nq, float radius, int* counts,
                             cudaStream_t st) {
    if (nq <= 0) return 0;
    return range_count(DenseSource{scores, ld, n}, n, nq, radius, counts, st);
}

int launch_range_collect_dense(const float* scores, int64_t ld, int64_t n, int nq, float radius,
                               unsigned long long* cursor, uint64_t* items, cudaStream_t st) {
    if (nq <= 0) return 0;
    return range_collect(DenseSource{scores, ld, n}, n, nq, radius, cursor, items, st);
}

int launch_range_emit(uint64_t* items, uint64_t* items2, int64_t nq, const int64_t* src_off, const int64_t* lims,
                      int n_seg, int64_t longest, int64_t total_long, const int64_t* tab, int64_t id_offset, float* D,
                      int64_t* I, cudaStream_t st) {
    if (nq <= 0) return 0;
    const size_t smem = (size_t)kRangeRun * sizeof(uint64_t);
    if (ensure_dynamic_smem(range_emit_kernel, smem) || ensure_dynamic_smem(range_sort_runs_kernel, smem)) return 1;
    range_emit_kernel<<<(unsigned)nq, kRangeSortThreads, smem, st>>>(items, src_off, lims, id_offset, D, I);
    KIRAG_LAUNCH_OK("range_emit_kernel");
    if (n_seg == 0) return 0;
    KIRAG_CHECK(n_seg <= 65535, "range_emit: %d long segments in one call", n_seg);
    const int64_t* d_src = tab;
    const int64_t* d_dst = tab + n_seg;
    const int64_t* d_len = tab + 2 * n_seg;
    const int64_t* d_e0 = tab + 3 * n_seg;
    const int64_t runs = (longest + kRangeRun - 1) / kRangeRun;
    KIRAG_CHECK(runs < 0x7fffffffLL, "range_emit: segment of %lld items is too long", (long long)longest);
    range_sort_runs_kernel<<<dim3((unsigned)runs, (unsigned)n_seg), kRangeSortThreads, smem, st>>>(items, d_src, d_len);
    KIRAG_LAUNCH_OK("range_sort_runs_kernel");
    const unsigned blocks = (unsigned)((total_long + 255) / 256);
    uint64_t* cur = items;
    uint64_t* nxt = items2;
    for (int64_t w = kRangeRun; w < longest; w *= 2) {
        range_merge_kernel<<<blocks, 256, 0, st>>>(cur, nxt, d_src, d_len, d_e0, n_seg, total_long, w);
        KIRAG_LAUNCH_OK("range_merge_kernel");
        uint64_t* t = cur; cur = nxt; nxt = t;
    }
    range_write_kernel<<<blocks, 256, 0, st>>>(cur, d_src, d_dst, d_e0, n_seg, total_long, id_offset, D, I);
    KIRAG_LAUNCH_OK("range_write_kernel");
    return 0;
}

}  // namespace kirag
