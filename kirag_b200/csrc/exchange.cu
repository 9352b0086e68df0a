// exchange.cu — fused peer-memory exchange + merge of the row-sharded search.
//
// No counterpart in the reference (its FAISS search is single-process CPU,
// /root/reference/retriever/index.py:47).  After the per-shard search every rank holds the exact
// top-k of ITS rows for every query; the global answer is the top-k of the union.  Instead of an
// NCCL all-gather followed by a merge kernel, ONE kernel per rank does both over NVLink peer
// memory (buffers mapped with CUDA IPC, one process per GPU):
//   push   : CTA b stores the result rows of its query range [q_lo, q_hi) into slot `rank` of
//            EVERY rank's exchange buffer (plain coalesced stores; remote ones travel over NVLink),
//            then publishes flag[rank][b] = epoch in every rank's buffer (release, system scope);
//   wait   : CTA b polls its OWN flags[g][b] (acquire, system scope) until all G ranks have
//            delivered that query range — there is no grid-wide or GPU-wide barrier, a query
//            range is merged as soon as its G pieces are there;
//   merge  : the G lists are sorted by (score desc, id asc) and hold distinct ids, so two lists are
//            merged by ranking: position in the own list + binary-search rank in the other one.
//            A pairwise tree (log2 G rounds, truncated to k after every round) merges the G lists
//            of a query; four queries are in flight per CTA.  No sort.
// Buffers are double-buffered by epoch parity: a rank can be at most one call ahead of its peers
// (it cannot finish call e before every peer has STARTED call e, i.e. finished call e-1), so
// data of call e+1 never lands in a slot that call e-1 is still reading.
// Every CTA pushes before it waits and the grid is small enough to be co-resident, so the wait
// cannot deadlock; it is bounded anyway (~20 s) so that a dead peer is an error, not a hang: the kernel
// then writes the offending rank into a mapped host word and returns (no trap: the context stays usable),
// and the next call on the exchange object fails with that message.
#include "common.cuh"
#include "../../include/kirag_b200.h"

#include <cstdio>
#include <cstring>
#include <new>

namespace kirag {

constexpr int kMaxRanks = 16;
constexpr int kExchangeMaxBlocks = 296;  // flags per (parity, source rank); 2 CTAs per SM on 148 SMs

struct ExchangeArgs {
    uint8_t* peer[kMaxRanks];  // exchange buffer of every rank as mapped in THIS process (peer[rank] = own)
    int rank, G;
    int64_t nq;
    int k;
    const int* words;    // device: [0..1] OR of the carried flags by epoch parity, [2] the epoch of THIS call (advanced on
                         // the device by exchange_tick_kernel, so that a captured CUDA graph can be replayed)
    size_t slot_bytes;   // capacity of one (parity, source rank) slot
    size_t flags_off;    // byte offset of the flag region
    size_t ids_off;      // byte offset of the id block inside a slot for this call (after nq*k scores)
                         // NB: the field `flags_off` above is the barrier-flag region of the whole buffer; the
                         // per-query certificate flags live at `qflags_off` inside every slot
    const float* D_loc;
    const int64_t* I_loc;
    float* D_out;
    int64_t* I_out;
    int vec16;     // rows can be copied with 16-byte accesses (k % 4 == 0, aligned bases)
    int n_groups;  // thread groups per CTA in the merge phase (1, 2 or 4), one query each at a time
    int tree;      // 1: pairwise merge tree (needs two list buffers in shared memory), 0: rank-everything merge
    const int* flags_loc;  // optional: this rank's per-query certificate flags (device), carried along with the rows
    size_t qflags_off;     // byte offset of the per-query flag block inside a slot (fixed per exchange object)
    int* any_flag;         // device: OR over all ranks and queries of the carried flags (identical on every rank)
    int* timeout_word;     // mapped pinned host word: set to 1 + source rank if a peer never delivered
};

__device__ __forceinline__ uint8_t* slot_ptr(const ExchangeArgs& a, int parity, int dst, int src) {
    return a.peer[dst] + ((size_t)parity * a.G + src) * a.slot_bytes;
}
__device__ __forceinline__ int* flag_ptr(const ExchangeArgs& a, int parity, int dst, int src, int block) {
    return reinterpret_cast<int*>(a.peer[dst] + a.flags_off) + ((size_t)parity * kMaxRanks + src) * kExchangeMaxBlocks + block;
}
__device__ __forceinline__ void st_release_sys(int* p, int v) {
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_sys(const int* p) {
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

constexpr int kExchangeThreads = 512;

// Advances the epoch ON THE DEVICE (one thread) and clears the flag word of the new parity.  The epoch only has to
// differ from the values two calls back; it is advanced in unsigned arithmetic so that a long-running server wraps
// around instead of overflowing; 0 is the "never written" flag value and is skipped keeping the parity sequence
// (... 0xffffffff odd, 2 even).  Keeping the epoch on the device (instead of passing it as a kernel argument) is
// what makes an exchange replayable from a CUDA graph.
__global__ void exchange_tick_kernel(int* words) {
    unsigned e = (unsigned)words[2] + 1u;
    if (e == 0u) e = 2u;
    words[2] = (int)e;
    words[e & 1u] = 0;
}

__global__ void __launch_bounds__(kExchangeThreads, 2) exchange_merge_kernel(const ExchangeArgs a) {
    extern __shared__ uint64_t xsmem[];
    const int G = a.G, k = a.k;
    const int L = G * k;
    __shared__ int n_valid_all[4][2 * kMaxRanks];
    const int b = blockIdx.x, NB = gridDim.x;
    const int64_t q_lo = a.nq * b / NB, q_hi = a.nq * (b + 1) / NB;
    const int64_t e_lo = q_lo * k, e_hi = q_hi * k;
    // epoch of this call: written by the tick kernel launched right before this one on the same stream
    const int epoch = __ldcg(a.words + 2);
    const int parity = (int)((unsigned)epoch & 1u);

    // ------------------------------------------------------------------ push ----
    // peers are visited in a rank-rotated order so that the G ranks do not all hit the same
    // destination at the same time; 16-byte stores when the rows allow it
    for (int p = 0; p < G; ++p) {
        const int dst = (a.rank + p) % G;
        uint8_t* slot = slot_ptr(a, parity, dst, a.rank);
        float* sd = reinterpret_cast<float*>(slot);
        int64_t* si = reinterpret_cast<int64_t*>(slot + a.ids_off);
        if (a.vec16) {
            const float4* srcd = reinterpret_cast<const float4*>(a.D_loc + e_lo);
            float4* dstd = reinterpret_cast<float4*>(sd + e_lo);
            const int64_t nd = (e_hi - e_lo) >> 2;
            for (int64_t i = threadIdx.x; i < nd; i += blockDim.x) dstd[i] = srcd[i];
            const longlong2* srci = reinterpret_cast<const longlong2*>(a.I_loc + e_lo);
            longlong2* dsti = reinterpret_cast<longlong2*>(si + e_lo);
            const int64_t ni = (e_hi - e_lo) >> 1;
            for (int64_t i = threadIdx.x; i < ni; i += blockDim.x) dsti[i] = srci[i];
        } else {
            for (int64_t i = e_lo + threadIdx.x; i < e_hi; i += blockDim.x) {
                sd[i] = a.D_loc[i];
                si[i] = a.I_loc[i];
            }
        }
        if (a.flags_loc) {
            int* sf = reinterpret_cast<int*>(slot + a.qflags_off);
            for (int64_t qq = q_lo + threadIdx.x; qq < q_hi; qq += blockDim.x) sf[qq] = a.flags_loc[qq];
        }
    }
    __syncthreads();
    if (threadIdx.x < G) {
        // the barrier above ordered every thread's stores before this fence (cumulativity)
        __threadfence_system();
        st_release_sys(flag_ptr(a, parity, threadIdx.x, a.rank, b), epoch);
    }
    // ------------------------------------------------------------------ wait ----
    __shared__ int s_timed_out;
    if (threadIdx.x == 0) s_timed_out = 0;
    __syncthreads();
    if (threadIdx.x < G) {
        const int* f = flag_ptr(a, parity, a.rank, threadIdx.x, b);
        if (ld_acquire_sys(f) != epoch) {
            const long long t0 = clock64();
            while (ld_acquire_sys(f) != epoch) {
                __nanosleep(64);
                if (clock64() - t0 > 40000000000LL) {
                    // a peer never delivered (~20 s): report through the mapped host word and leave the kernel;
                    // the context stays usable and the host turns the word into an error status
                    printf("kirag exchange: rank %d block %d timed out waiting for rank %d (epoch %d, flag %d)\n",
                           a.rank, b, (int)threadIdx.x, epoch, ld_acquire_sys(f));
                    *reinterpret_cast<volatile int*>(a.timeout_word) = 1 + (int)threadIdx.x;
                    __threadfence_system();
                    s_timed_out = 1;
                    break;
                }
            }
        }
        __threadfence_system();
    }
    __syncthreads();
    if (s_timed_out) return;
    if (a.flags_loc) {
        // OR of every rank's certificate flags for this CTA's queries: the same value on every rank, so all
        // ranks take the same decision about re-answering without a host collective
        int mine = 0;
        for (int64_t qq = q_lo + threadIdx.x; qq < q_hi; qq += blockDim.x)
            for (int g = 0; g < G; ++g)
                mine |= __ldcg(reinterpret_cast<const int*>(slot_ptr(a, parity, a.rank, g) + a.qflags_off) + qq);
        if (__any_sync(0xffffffffu, mine != 0) && (threadIdx.x & 31) == 0) atomicOr(a.any_flag + parity, 1);
    }
    // ----------------------------------------------------------------- merge ----
    // The CTA splits into n_groups thread groups; each merges one query at a time in its own slice of
    // shared memory and synchronises with a named barrier of its own.
    const int n_groups = a.n_groups;
    const int gthreads = kExchangeThreads / n_groups;
    const int grp = threadIdx.x / gthreads;
    const int gt = threadIdx.x - grp * gthreads;
    int* n_valid = n_valid_all[grp];
    if (a.tree) {
        // pairwise merge tree (common.cuh::merge_tree): O(G k log k) steps per query instead of O(G^2 k log k)
        int64_t* ids_buf = reinterpret_cast<int64_t*>(xsmem) + (size_t)grp * 2 * L;                               // [2][L]
        uint32_t* keys_buf = reinterpret_cast<uint32_t*>(reinterpret_cast<int64_t*>(xsmem) + (size_t)n_groups * 2 * L) +
                             (size_t)grp * 2 * L;                                                                    // [2][L]
        int* const nv[2] = {n_valid, n_valid + kMaxRanks};
        for (int64_t q = q_lo + grp; q < q_hi; q += n_groups) {
            if (gt < G) nv[0][gt] = 0;
            group_barrier(1 + grp, gthreads);
            for (int i = gt; i < L; i += gthreads) {
                const int g = i / k, j = i - g * k;
                const uint8_t* slot = slot_ptr(a, parity, a.rank, g);
                const int64_t id = __ldcg(reinterpret_cast<const int64_t*>(slot + a.ids_off) + q * k + j);
                uint32_t key = 0u;
                if (id >= 0) key = score_key(__ldcg(reinterpret_cast<const float*>(slot) + q * k + j));
                keys_buf[i] = key;
                ids_buf[i] = id;
                if (key != 0u) atomicAdd(&nv[0][g], 1);  // valid items form a prefix of each list
            }
            group_barrier(1 + grp, gthreads);
            const int cur = merge_tree(keys_buf, ids_buf, nv, G, k, gt, gthreads, 1 + grp);
            const int total = nv[cur][0];
            for (int j = gt; j < k; j += gthreads) {
                const bool ok = j < total;
                a.D_out[q * k + j] = ok ? key_score(keys_buf[(size_t)cur * L + j]) : -FLT_MAX;
                a.I_out[q * k + j] = ok ? ids_buf[(size_t)cur * L + j] : -1;
            }
            group_barrier(1 + grp, gthreads);
        }
        return;
    }
    // rank-everything merge (lists too long for two shared-memory buffers): an item's global rank is the sum
    // of its binary-search ranks in the other lists
    int64_t* ids = reinterpret_cast<int64_t*>(xsmem) + (size_t)grp * L;                        // [L]
    uint32_t* keys = reinterpret_cast<uint32_t*>(reinterpret_cast<int64_t*>(xsmem) + (size_t)n_groups * L) + (size_t)grp * L;  // [L]
    for (int64_t q = q_lo + grp; q < q_hi; q += n_groups) {
        if (gt < G) n_valid[gt] = 0;
        group_barrier(1 + grp, gthreads);
        for (int i = gt; i < L; i += gthreads) {
            const int g = i / k, j = i - g * k;
            const uint8_t* slot = slot_ptr(a, parity, a.rank, g);
            const int64_t id = __ldcg(reinterpret_cast<const int64_t*>(slot + a.ids_off) + q * k + j);
            uint32_t key = 0u;
            if (id >= 0) key = score_key(__ldcg(reinterpret_cast<const float*>(slot) + q * k + j));
            const bool ok = key != 0u;
            keys[i] = key;
            ids[i] = ok ? id : INT64_MAX;
            if (ok) atomicAdd(&n_valid[g], 1);  // valid items form a prefix of each list
        }
        group_barrier(1 + grp, gthreads);
        int total = 0;
        for (int g = 0; g < G; ++g) total += n_valid[g];
        for (int i = gt; i < L; i += gthreads) {
            const int g = i / k, j = i - g * k;
            if (j >= n_valid[g]) continue;
            const uint32_t key = keys[i];
            const int64_t id = ids[i];
            int r = j;  // items of its own list that precede it
            for (int h = 0; h < G; ++h)
                if (h != g) r += count_before(keys + h * k, ids + h * k, n_valid[h], key, id);
            if (r < k) {
                a.D_out[q * k + r] = key_score(key);
                a.I_out[q * k + r] = id;
            }
        }
        for (int j = total + gt; j < k; j += gthreads) {  // fewer than k results in total
            a.D_out[q * k + j] = -FLT_MAX;
            a.I_out[q * k + j] = -1;
        }
        group_barrier(1 + grp, gthreads);
    }
}

}  // namespace kirag

using namespace kirag;

struct kirag_exchange {
    int device = 0;
    int rank = 0;
    int world = 1;
    int64_t max_nq = 0;
    int max_k = 0;
    size_t slot_bytes = 0;
    size_t flags_off = 0;
    size_t total_bytes = 0;
    uint8_t* own = nullptr;
    uint8_t* peer[kMaxRanks] = {nullptr};
    bool opened[kMaxRanks] = {false};  // mapped with cudaIpcOpenMemHandle (to be closed)
    bool connected = false;
    size_t qflags_off = 0;       // per-query certificate flags inside a slot
    int64_t qflags_cap = 0;      // queries the flag block of a slot can hold
    int* any_dev = nullptr;      // [0..1] OR of the carried flags by parity, [2] epoch (device-side source of truth)
    int* any_host = nullptr;     // pinned + mapped: [0..2] copy of any_dev after every exchange; [3]: time-out word
    cudaStream_t stream = nullptr;  // stream of the previous exchange (epoch double-buffering is only safe if a rank's
    bool stream_set = false;        // exchanges execute in call order: another stream first waits for last_ev)
    cudaEvent_t last_ev = nullptr;  // recorded behind every exchange
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

namespace {
struct DeviceGuardLite {
    int prev = -1;
    explicit DeviceGuardLite(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev); else prev = -1;
    }
    ~DeviceGuardLite() { if (prev >= 0) cudaSetDevice(prev); }
};
}  // namespace

extern "C" {

int kirag_exchange_create(int device, int rank, int world, int64_t max_nq, int max_k, kirag_exchange_t** out) {
    KIRAG_CHECK(out != nullptr, "exchange_create: null out pointer");
    *out = nullptr;
    KIRAG_CHECK(world >= 1 && world <= kMaxRanks, "exchange_create: world size %d not in [1, %d]", world, kMaxRanks);
    KIRAG_CHECK(rank >= 0 && rank < world, "exchange_create: rank %d not in [0, %d)", rank, world);
    KIRAG_CHECK(max_nq > 0 && max_k > 0, "exchange_create: max_nq and max_k must be positive");
    KIRAG_CHECK((int64_t)world * max_k <= 8192, "exchange_create: world*max_k=%lld exceeds 8192",
                (long long)world * max_k);
    int prev = -1;
    cudaGetDevice(&prev);
    KIRAG_CUDA_OK(cudaSetDevice(device));
    kirag_exchange* x = new (std::nothrow) kirag_exchange();
    KIRAG_CHECK(x != nullptr, "exchange_create: out of host memory");
    x->device = device;
    x->rank = rank;
    x->world = world;
    x->max_nq = max_nq;
    x->max_k = max_k;
    x->qflags_off = align_up((size_t)max_nq * max_k * 4, 16) + align_up((size_t)max_nq * max_k * 8, 16);
    x->qflags_cap = max_nq;
    x->slot_bytes = x->qflags_off + align_up((size_t)x->qflags_cap * 4, 16);
    x->flags_off = align_up(2 * (size_t)world * x->slot_bytes, 256);
    x->total_bytes = x->flags_off + 2 * (size_t)kMaxRanks * kExchangeMaxBlocks * sizeof(int);
    cudaError_t e = cudaMalloc((void**)&x->own, x->total_bytes);
    if (e != cudaSuccess) {
        set_error("exchange_create: cudaMalloc(%zu) failed: %s", x->total_bytes, cudaGetErrorString(e));
        delete x;
        if (prev >= 0) cudaSetDevice(prev);
        return 1;
    }
    e = cudaMemset(x->own, 0, x->total_bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        set_error("exchange_create: clearing the buffer failed: %s", cudaGetErrorString(e));
        cudaFree(x->own);
        delete x;
        if (prev >= 0) cudaSetDevice(prev);
        return 1;
    }
    if (cudaMalloc((void**)&x->any_dev, 4 * sizeof(int)) != cudaSuccess ||
        cudaMemset(x->any_dev, 0, 4 * sizeof(int)) != cudaSuccess ||
        cudaHostAlloc((void**)&x->any_host, 4 * sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
        set_error("exchange_create: allocating the flag words failed: %s", cudaGetErrorString(cudaGetLastError()));
        if (x->any_dev) cudaFree(x->any_dev);
        cudaFree(x->own);
        delete x;
        if (prev >= 0) cudaSetDevice(prev);
        return 1;
    }
    x->any_host[0] = x->any_host[1] = x->any_host[2] = x->any_host[3] = 0;
    x->peer[rank] = x->own;
    if (world == 1) x->connected = true;
    if (prev >= 0) cudaSetDevice(prev);
    *out = x;
    return 0;
}

int kirag_exchange_destroy(kirag_exchange_t* x) {
    if (!x) return 0;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(x->device);
    cudaDeviceSynchronize();
    for (int g = 0; g < x->world; ++g)
        if (x->opened[g] && x->peer[g]) cudaIpcCloseMemHandle(x->peer[g]);
    if (x->own) cudaFree(x->own);
    if (x->any_dev) cudaFree(x->any_dev);
    if (x->any_host) cudaFreeHost(x->any_host);
    if (x->last_ev) cudaEventDestroy(x->last_ev);
    delete x;
    if (prev >= 0) cudaSetDevice(prev);
    return 0;
}

int kirag_exchange_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }

int kirag_exchange_export(kirag_exchange_t* x, void* handle_out) {
    KIRAG_CHECK(x && handle_out, "exchange_export: null argument");
    DeviceGuardLite guard(x->device);
    cudaIpcMemHandle_t h;
    KIRAG_CUDA_OK(cudaIpcGetMemHandle(&h, x->own));
    memcpy(handle_out, &h, sizeof(h));
    return 0;
}

int kirag_exchange_connect(kirag_exchange_t* x, const void* handles_all) {
    KIRAG_CHECK(x && handles_all, "exchange_connect: null argument");
    KIRAG_CHECK(!x->connected || x->world == 1, "exchange_connect: already connected");
    DeviceGuardLite guard(x->device);
    const uint8_t* hp = static_cast<const uint8_t*>(handles_all);
    for (int g = 0; g < x->world; ++g) {
        if (g == x->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, hp + (size_t)g * sizeof(h), sizeof(h));
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            set_error("exchange_connect: cudaIpcOpenMemHandle for rank %d failed: %s", g, cudaGetErrorString(e));
            cudaGetLastError();
            return 1;
        }
        x->peer[g] = static_cast<uint8_t*>(p);
        x->opened[g] = true;
    }
    x->connected = true;
    return 0;
}

int kirag_exchange_connect_ptrs(kirag_exchange_t* x, void* const* peer_buffers) {
    KIRAG_CHECK(x && peer_buffers, "exchange_connect_ptrs: null argument");
    for (int g = 0; g < x->world; ++g) {
        if (g == x->rank) continue;
        KIRAG_CHECK(peer_buffers[g] != nullptr, "exchange_connect_ptrs: null buffer for rank %d", g);
        // a buffer on another device must be peer-accessible from this rank's device (same device: always fine)
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, peer_buffers[g]) == cudaSuccess && attr.type == cudaMemoryTypeDevice &&
            attr.device != x->device) {
            int can = 0;
            KIRAG_CUDA_OK(cudaDeviceCanAccessPeer(&can, x->device, attr.device));
            KIRAG_CHECK(can, "exchange_connect_ptrs: device %d cannot access rank %d's buffer on device %d", x->device, g,
                        attr.device);
            DeviceGuardLite guard(x->device);
            cudaError_t e = cudaDeviceEnablePeerAccess(attr.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                set_error("exchange_connect_ptrs: cudaDeviceEnablePeerAccess(%d) failed: %s", attr.device, cudaGetErrorString(e));
                return 1;
            }
            cudaGetLastError();
        } else {
            cudaGetLastError();
        }
        x->peer[g] = static_cast<uint8_t*>(peer_buffers[g]);
    }
    x->connected = true;
    return 0;
}

void* kirag_exchange_buffer(kirag_exchange_t* x) { return x ? x->own : nullptr; }

static int exchange_merge_impl(kirag_exchange_t* x, const float* D_loc, const int64_t* I_loc, const int* flags_loc,
                               int64_t nq, int k, float* D_out, int64_t* I_out, void* stream) {
    KIRAG_CHECK(x != nullptr, "exchange_merge: null exchange");
    KIRAG_CHECK(x->connected, "exchange_merge: peers are not connected (call kirag_exchange_connect first)");
    KIRAG_CHECK(k > 0 && k <= x->max_k, "exchange_merge: k=%d not in [1, %d]", k, x->max_k);
    KIRAG_CHECK(nq >= 0 && nq * (int64_t)k <= x->max_nq * (int64_t)x->max_k,
                "exchange_merge: nq*k=%lld exceeds the capacity %lld", (long long)(nq * k),
                (long long)(x->max_nq * x->max_k));
    if (nq == 0) return 0;
    KIRAG_CHECK(D_loc && I_loc && D_out && I_out, "exchange_merge: null buffer");
    KIRAG_CHECK(!flags_loc || nq <= x->qflags_cap, "exchange_merge: nq=%lld exceeds the flag capacity %lld", (long long)nq,
                (long long)x->qflags_cap);
    // Epoch double-buffering assumes that this rank's exchanges EXECUTE in call order.  Calls on one stream are
    // ordered by the stream; a call on another stream first waits for the event recorded behind the previous
    // exchange.  A call that is being captured into a CUDA graph can neither wait for outside work nor be waited
    // for: whoever replays the graph orders the replays against this rank's other exchanges (ShardedFlatIP
    // synchronises the replay stream at the end of every search).
    KIRAG_CHECK(x->any_host[3] == 0, "exchange_merge: an earlier exchange timed out waiting for rank %d (a peer died or "
                "skipped a call); this exchange object is no longer usable", x->any_host[3] - 1);
    cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing((cudaStream_t)stream, &capturing);
    if (capturing == cudaStreamCaptureStatusNone) {
        if (!x->last_ev) KIRAG_CUDA_OK(cudaEventCreateWithFlags(&x->last_ev, cudaEventDisableTiming));
        if (x->stream_set && x->stream != (cudaStream_t)stream)
            KIRAG_CUDA_OK(cudaStreamWaitEvent((cudaStream_t)stream, x->last_ev, 0));
        x->stream = (cudaStream_t)stream;
        x->stream_set = true;
    }
    DeviceGuardLite guard(x->device);
    ExchangeArgs a{};
    for (int g = 0; g < x->world; ++g) a.peer[g] = x->peer[g];
    a.rank = x->rank;
    a.G = x->world;
    a.nq = nq;
    a.k = k;
    a.words = x->any_dev;
    a.slot_bytes = x->slot_bytes;
    a.flags_off = x->flags_off;
    a.ids_off = align_up((size_t)nq * k * 4, 16);
    a.D_loc = D_loc;
    a.I_loc = I_loc;
    a.D_out = D_out;
    a.I_out = I_out;
    // the grid must be the same on every rank (flags are per block): derived from nq only
    int blocks = (int)(nq < kExchangeMaxBlocks ? nq : kExchangeMaxBlocks);
    const size_t list_bytes = (size_t)x->world * k * 12;
    a.tree = (2 * list_bytes <= 96 * 1024) ? 1 : 0;  // two buffers of G*k (key, id) pairs per merge group
    const size_t per_query = a.tree ? 2 * list_bytes : list_bytes;
    int n_groups = 4;
    while (n_groups > 1 && per_query * n_groups > 96 * 1024) n_groups >>= 1;
    a.n_groups = n_groups;
    a.vec16 = (k % 4 == 0) && ((reinterpret_cast<uintptr_t>(D_loc) & 15) == 0) &&
              ((reinterpret_cast<uintptr_t>(I_loc) & 15) == 0) && ((a.ids_off & 15) == 0);
    const size_t smem = per_query * n_groups;
    if (smem > 48 * 1024 && ensure_dynamic_smem(exchange_merge_kernel, 96 * 1024)) return 1;
    a.flags_loc = flags_loc;
    a.qflags_off = x->qflags_off;
    a.any_flag = x->any_dev;
    a.timeout_word = x->any_host + 3;  // mapped pinned memory: same address on the device under UVA
    exchange_tick_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(x->any_dev);
    KIRAG_LAUNCH_OK("exchange_tick_kernel");
    exchange_merge_kernel<<<blocks, kExchangeThreads, smem, (cudaStream_t)stream>>>(a);
    KIRAG_LAUNCH_OK("exchange_merge_kernel");
    // both flag words and the epoch they belong to: the host picks the word of the LAST executed exchange, also
    // after a graph replay that it did not enqueue itself
    KIRAG_CUDA_OK(cudaMemcpyAsync(x->any_host, x->any_dev, 3 * sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    if (capturing == cudaStreamCaptureStatusNone) KIRAG_CUDA_OK(cudaEventRecord(x->last_ev, (cudaStream_t)stream));
    return 0;
}

int kirag_exchange_merge_topk(kirag_exchange_t* x, const float* D_loc, const int64_t* I_loc, int64_t nq, int k,
                              float* D_out, int64_t* I_out, void* stream) {
    return exchange_merge_impl(x, D_loc, I_loc, nullptr, nq, k, D_out, I_out, stream);
}

int kirag_exchange_merge_topk_flags(kirag_exchange_t* x, const float* D_loc, const int64_t* I_loc, const int* flags_loc,
                                    int64_t nq, int k, float* D_out, int64_t* I_out, void* stream) {
    KIRAG_CHECK(flags_loc != nullptr, "exchange_merge_flags: null flags");
    return exchange_merge_impl(x, D_loc, I_loc, flags_loc, nq, k, D_out, I_out, stream);
}

int kirag_exchange_last_any_flag(kirag_exchange_t* x) {
    if (!x) return -1;
    if (x->any_host[3] != 0) {
        set_error("exchange: timed out waiting for rank %d", x->any_host[3] - 1);
        return -2;
    }
    return x->any_host[(unsigned)x->any_host[2] & 1u];
}

}  // extern "C"
