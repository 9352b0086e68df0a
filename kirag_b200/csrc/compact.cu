// compact.cu — row removal (kirag_index_remove_ids / kirag_index_remove_range): the removal bitmap over the old rows,
// the kept count of every 128-row group, and the gather of the kept rows of a source range into a dense staging buffer
// (api.cu plans the pieces and writes them back through the ordinary add path).  On an index with an id table the
// bitmap is built from the table (selection by external id) and the table is compacted like the rows.
#include "common.cuh"

#include <cub/device/device_radix_sort.cuh>

namespace kirag {

// bit r of bits = old row r is removed.  Ids outside [0, n_rows) and repeated ids are harmless.
__global__ void mark_ids_kernel(const int64_t* __restrict__ ids, int64_t n_ids, int64_t n_rows, uint32_t* bits) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_ids; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = ids[i];
        if (r >= 0 && r < n_rows) atomicOr(bits + (r >> 5), 1u << (r & 31));
    }
}

// rows [lo, hi) removed (0 <= lo < hi <= n_rows); one thread per word, the only writer of that word
__global__ void mark_range_kernel(int64_t lo, int64_t hi, uint32_t* bits) {
    const int64_t w = (lo >> 5) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t a = w * 32 > lo ? w * 32 : lo;
    const int64_t b = w * 32 + 32 < hi ? w * 32 + 32 : hi;
    if (a >= b) return;
    const int n = (int)(b - a), s = (int)(a - w * 32);
    bits[w] |= (n == 32 ? 0xffffffffu : ((1u << n) - 1u)) << s;
}

// kept[g] = rows of group g (128 rows, the last one shorter) that are not removed
__global__ void kept_counts_kernel(const uint32_t* __restrict__ bits, int64_t n_rows, int64_t n_groups, int* kept) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    const int64_t rows = n_rows - g * 128 < 128 ? n_rows - g * 128 : 128;
    const uint4 w = *reinterpret_cast<const uint4*>(bits + g * 4);
    kept[g] = (int)rows - (__popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w));
}

static int launch_kept_counts(const uint32_t* bits, int64_t n_rows, int* kept, cudaStream_t st) {
    const int64_t n_groups = (n_rows + 127) / 128;
    kept_counts_kernel<<<(unsigned)((n_groups + 255) / 256), 256, 0, st>>>(bits, n_rows, n_groups, kept);
    KIRAG_LAUNCH_OK("kept_counts_kernel");
    return 0;
}

int launch_removal_counts(const int64_t* ids, int64_t n_ids, int64_t lo, int64_t hi, int64_t n_rows, uint32_t* bits,
                          int* kept, cudaStream_t st) {
    const int64_t n_groups = (n_rows + 127) / 128;
    KIRAG_CUDA_OK(cudaMemsetAsync(bits, 0, (size_t)n_groups * 16, st));
    if (ids) {
        if (n_ids > 0) {
            const int64_t blocks = (n_ids + 255) / 256;
            mark_ids_kernel<<<(unsigned)(blocks < 65536 ? blocks : 65536), 256, 0, st>>>(ids, n_ids, n_rows, bits);
            KIRAG_LAUNCH_OK("mark_ids_kernel");
        }
    } else if (lo < hi) {
        const int64_t words = ((hi - 1) >> 5) - (lo >> 5) + 1;
        mark_range_kernel<<<(unsigned)((words + 255) / 256), 256, 0, st>>>(lo, hi, bits);
        KIRAG_LAUNCH_OK("mark_range_kernel");
    }
    return launch_kept_counts(bits, n_rows, kept, st);
}

// ---- selection by external id (index with an id table) ----------------------------------------------------------
// One warp per 32 rows: lane l tests row 32 w + l and the warp's ballot is bit word w, written by lane 0 alone (no
// atomics).  A range selection is one compare per row; a batch (sel sorted ascending) one binary search per row.
__global__ void __launch_bounds__(256) mark_by_id_kernel(const int64_t* __restrict__ table, int64_t n_rows,
                                                         const int64_t* __restrict__ sel, int64_t n_sel, int64_t lo,
                                                         int64_t hi, uint32_t* __restrict__ bits) {
    const int lane = threadIdx.x & 31;
    const int64_t n_words = (n_rows + 31) >> 5;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_words; w += warps) {
        const int64_t r = (w << 5) + lane;
        bool hit = false;
        if (r < n_rows) {
            const int64_t id = table[r];
            if (sel) {
                int64_t a = 0, b = n_sel;  // first entry >= id
                while (a < b) {
                    const int64_t m = (a + b) >> 1;
                    if (sel[m] < id) a = m + 1; else b = m;
                }
                hit = a < n_sel && sel[a] == id;
            } else {
                hit = lo <= id && id < hi;
            }
        }
        const uint32_t word = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) bits[w] = word;
    }
}

int launch_removal_counts_by_id(const int64_t* table, int64_t n_rows, const int64_t* sel, int64_t n_sel, int64_t lo,
                                int64_t hi, uint32_t* bits, int* kept, cudaStream_t st) {
    const int64_t n_groups = (n_rows + 127) / 128;
    // the words past the last row (up to the group's four) stay zero
    KIRAG_CUDA_OK(cudaMemsetAsync(bits, 0, (size_t)n_groups * 16, st));
    const int64_t blocks = ((n_rows + 31) / 32 + 7) / 8;  // 8 warps per block
    mark_by_id_kernel<<<(unsigned)(blocks < 65536 ? blocks : 65536), 256, 0, st>>>(table, n_rows, sel, n_sel, lo, hi,
                                                                                  bits);
    KIRAG_LAUNCH_OK("mark_by_id_kernel");
    return launch_kept_counts(bits, n_rows, kept, st);
}

size_t sort_ids_temp_bytes(int64_t n) {
    size_t bytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, bytes, static_cast<const int64_t*>(nullptr), static_cast<int64_t*>(nullptr),
                                   (int)n);
    return bytes;
}

int launch_sort_ids(const int64_t* in, int64_t* out, int64_t n, void* temp, size_t temp_bytes, cudaStream_t st) {
    KIRAG_CHECK(n >= 0 && n <= 0x7fffffffLL, "sort_ids: %lld ids in one selection (at most 2^31 - 1)", (long long)n);
    if (n == 0) return 0;
    KIRAG_CUDA_OK(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, in, out, (int)n, 0, 64, st));
    count_launch();
    return 0;
}

// new row number of the kept old row i (bit clear): kept rows of the groups before + kept rows before i in its group
__device__ __forceinline__ int64_t kept_rank(const uint32_t* bits, const int64_t* group_base, int64_t i, uint32_t w) {
    const int64_t g = i >> 7;
    int removed_before = __popc(w & ((1u << (i & 31)) - 1u));
    for (int64_t v = g * 4; v < (i >> 5); ++v) removed_before += __popc(bits[v]);
    return group_base[g] + (i - g * 128) - removed_before;
}

__global__ void compact_ids_kernel(const int64_t* __restrict__ table, const uint32_t* __restrict__ bits,
                                   const int64_t* __restrict__ group_base, int64_t i0, int64_t n_rows, int64_t j0,
                                   int64_t* __restrict__ out) {
    for (int64_t i = i0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows;
         i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t w = bits[i >> 5];
        if ((w >> (i & 31)) & 1u) continue;
        out[kept_rank(bits, group_base, i, w) - j0] = table[i];
    }
}

int launch_compact_ids(const int64_t* table, const uint32_t* bits, const int64_t* group_base, int64_t i0, int64_t n_rows,
                       int64_t j0, int64_t* out, cudaStream_t st) {
    if (i0 >= n_rows) return 0;
    const int64_t blocks = (n_rows - i0 + 255) / 256;
    compact_ids_kernel<<<(unsigned)(blocks < 65536 ? blocks : 65536), 256, 0, st>>>(table, bits, group_base, i0, n_rows,
                                                                                   j0, out);
    KIRAG_LAUNCH_OK("compact_ids_kernel");
    return 0;
}

// One warp per old row i of [i0, i1): a kept row whose new number (group_base[i / 128] + kept rows before it in its
// group) falls in [j0, j1) is copied from its shard's master (stripe arithmetic; G = 1: the index's own master) to row
// (new - j0) of out.  Every load of a row is issued before its stores; the copy is bandwidth-bound and has no arithmetic.
constexpr int kGatherBatch = 8;  // 16-byte loads in flight per lane
template <bool VEC4>
__global__ void __launch_bounds__(256) gather_kept_kernel(const __grid_constant__ ShardMasters masters, int G, int d,
                                                          const uint32_t* __restrict__ bits,
                                                          const int64_t* __restrict__ group_base, int64_t i0, int64_t i1,
                                                          int64_t j0, int64_t j1, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = i0 + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); i < i1; i += warps) {
        const uint32_t w = bits[i >> 5];
        if ((w >> (i & 31)) & 1u) continue;
        const int64_t dst = kept_rank(bits, group_base, i, w);
        if (dst < j0 || dst >= j1) continue;
        const float* src = masters.p[stripe_shard(i, G)] + stripe_local(i, G) * d;
        float* o = out + (dst - j0) * d;
        if (VEC4) {
            for (int c0 = lane * 4; c0 < d; c0 += kGatherBatch * 128) {
                float4 v[kGatherBatch];
#pragma unroll
                for (int u = 0; u < kGatherBatch; ++u)
                    if (c0 + u * 128 < d) v[u] = __ldcs(reinterpret_cast<const float4*>(src + c0 + u * 128));
#pragma unroll
                for (int u = 0; u < kGatherBatch; ++u)
                    if (c0 + u * 128 < d) *reinterpret_cast<float4*>(o + c0 + u * 128) = v[u];
            }
        } else {
            for (int c0 = lane; c0 < d; c0 += kGatherBatch * 32) {
                float v[kGatherBatch];
#pragma unroll
                for (int u = 0; u < kGatherBatch; ++u)
                    if (c0 + u * 32 < d) v[u] = __ldcs(src + c0 + u * 32);
#pragma unroll
                for (int u = 0; u < kGatherBatch; ++u)
                    if (c0 + u * 32 < d) o[c0 + u * 32] = v[u];
            }
        }
    }
}

int launch_gather_kept(const ShardMasters& masters, int G, int d, const uint32_t* bits, const int64_t* group_base,
                       int64_t i0, int64_t i1, int64_t j0, int64_t j1, float* out, int num_sms, cudaStream_t st) {
    if (i1 <= i0 || j1 <= j0) return 0;
    const int64_t want = (i1 - i0 + 7) / 8;  // 8 warps per block
    const int64_t cap = (int64_t)num_sms * 16;
    const unsigned blocks = (unsigned)(want < cap ? want : cap);
    bool vec4 = (d % 4) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    for (int s = 0; s < G; ++s) vec4 = vec4 && (reinterpret_cast<uintptr_t>(masters.p[s]) & 15) == 0;
    if (vec4)
        gather_kept_kernel<true><<<blocks, 256, 0, st>>>(masters, G, d, bits, group_base, i0, i1, j0, j1, out);
    else
        gather_kept_kernel<false><<<blocks, 256, 0, st>>>(masters, G, d, bits, group_base, i0, i1, j0, j1, out);
    KIRAG_LAUNCH_OK("gather_kept_kernel");
    return 0;
}

}  // namespace kirag
