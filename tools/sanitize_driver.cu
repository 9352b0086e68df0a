// sanitize_driver.cu — a torch-free driver that runs every kernel family of libkirag_b200.so on small shapes, so that
// compute-sanitizer (memcheck / racecheck / synccheck / initcheck) can watch them without paying for a Python start-up
// under the tool.  Built and run by tools/sanitize.sh on the GPU box; every case checks its result against a host
// computation, so a "passed" under the sanitizer is also a correctness pass.
//
//   ./sanitize_driver [case]     case = scan | search | pool | exchange | topk | host_rescore | host_exact | multi_merge |
//                                       remove_compact | id_map | all (default)
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

#include "../include/kirag_b200.h"

#define CK(x)                                                                         \
    do {                                                                              \
        if ((x) != 0) {                                                               \
            fprintf(stderr, "FAILED %s (%s:%d): %s\n", #x, __FILE__, __LINE__, kirag_last_error()); \
            exit(2);                                                                  \
        }                                                                             \
    } while (0)
#define CU(x)                                                                         \
    do {                                                                              \
        cudaError_t e_ = (x);                                                         \
        if (e_ != cudaSuccess) {                                                      \
            fprintf(stderr, "CUDA FAILED %s: %s\n", #x, cudaGetErrorString(e_));      \
            exit(2);                                                                  \
        }                                                                             \
    } while (0)

static std::vector<float> unit_rows(std::mt19937& rng, int n, int d) {
    std::normal_distribution<float> g(0.f, 1.f);
    std::vector<float> x((size_t)n * d);
    for (int r = 0; r < n; ++r) {
        double s = 0;
        for (int c = 0; c < d; ++c) { x[(size_t)r * d + c] = g(rng); s += (double)x[(size_t)r * d + c] * x[(size_t)r * d + c]; }
        const float inv = (float)(1.0 / std::sqrt(s));
        for (int c = 0; c < d; ++c) x[(size_t)r * d + c] *= inv;
    }
    return x;
}

static void host_topk(const std::vector<float>& xb, int n, const std::vector<float>& xq, int nq, int d, int k,
                      std::vector<int64_t>* I) {
    I->assign((size_t)nq * k, -1);
    std::vector<std::pair<double, int>> s((size_t)n);
    for (int q = 0; q < nq; ++q) {
        for (int r = 0; r < n; ++r) {
            double a = 0;
            for (int c = 0; c < d; ++c) a += (double)xq[(size_t)q * d + c] * xb[(size_t)r * d + c];
            s[(size_t)r] = {-a, r};
        }
        std::partial_sort(s.begin(), s.begin() + std::min(k, n), s.end());
        for (int j = 0; j < std::min(k, n); ++j) (*I)[(size_t)q * k + j] = s[(size_t)j].second;
    }
}

// every tcgen05 scan variant through the dense-score test hook (KIRAG_DEBUG_BQ selects the kernel)
static void case_scan() {
    std::mt19937 rng(1);
    const int n = 1500, d = 128;
    auto xb = unit_rows(rng, n, d);
    kirag_index_t* h = nullptr;
    CK(kirag_index_create(d, KIRAG_METRIC_INNER_PRODUCT, 0, &h));
    CK(kirag_index_add(h, xb.data(), n, 0, nullptr));
    const struct { const char* bq; int nq; } variants[] = {{"64r", 40}, {"64s", 40}, {"128r", 100}, {"128s", 100}, {"256s", 300}};
    for (const auto& v : variants) {
        setenv("KIRAG_DEBUG_BQ", v.bq, 1);
        auto xq = unit_rows(rng, v.nq, d);
        std::vector<float> got((size_t)n * v.nq);
        CK(kirag_index_debug_scores(h, xq.data(), v.nq, got.data()));
        double worst = 0;
        for (int r = 0; r < n; r += 7)
            for (int q = 0; q < v.nq; q += 3) {
                double a = 0;
                for (int c = 0; c < d; ++c) a += (double)xq[(size_t)q * d + c] * xb[(size_t)r * d + c];
                worst = std::max(worst, std::fabs(a - got[(size_t)r * v.nq + q]));
            }
        printf("scan variant KIRAG_DEBUG_BQ=%s nq=%d: max |bf16 score - fp64| = %.2e %s\n", v.bq, v.nq, worst,
               worst < 1e-2 ? "ok" : "BAD");
        if (!(worst < 1e-2)) exit(3);
    }
    unsetenv("KIRAG_DEBUG_BQ");
    CK(kirag_index_destroy(h));
}

// full searches: every level kernel, compaction, rescoring, final / fused tail, exact scan, async + finish
static void case_search() {
    std::mt19937 rng(2);
    const int n = 40000, d = 128, k = 10;
    auto xb = unit_rows(rng, n, d);
    kirag_index_t* h = nullptr;
    CK(kirag_index_create(d, KIRAG_METRIC_INNER_PRODUCT, 0, &h));
    CK(kirag_index_add(h, xb.data(), n / 2, 0, nullptr));
    CK(kirag_index_add(h, xb.data() + (size_t)(n / 2) * d, n - n / 2, 0, nullptr));
    for (int nq : {2, 40, 100, 200}) {
        auto xq = unit_rows(rng, nq, d);
        std::vector<float> D((size_t)nq * k), De((size_t)nq * k);
        std::vector<int64_t> I((size_t)nq * k), Ie((size_t)nq * k), Ih;
        kirag_search_stats_t st;
        CK(kirag_index_search_ex(h, xq.data(), nq, k, D.data(), I.data(), 0, 0, KIRAG_PATH_AUTO, &st, nullptr));
        CK(kirag_index_search_ex(h, xq.data(), nq, k, De.data(), Ie.data(), 0, 0, KIRAG_PATH_EXACT, nullptr, nullptr));
        host_topk(xb, n, xq, nq, d, k, &Ih);
        int diff = 0, diff_host = 0;
        for (size_t i = 0; i < I.size(); ++i) { diff += I[i] != Ie[i] || D[i] != De[i]; diff_host += I[i] != Ih[i]; }
        printf("search nq=%d: levels=%d fast=%lld launches=%lld, AUTO vs EXACT differences %d, vs host fp64 %d %s\n", nq,
               st.levels, (long long)st.n_fast, (long long)st.kernel_launches, diff, diff_host,
               diff == 0 && diff_host <= 2 ? "ok" : "BAD");
        if (diff != 0 || diff_host > 2) exit(3);
    }
    // device pointers, asynchronous half + finish
    const int nq = 6;
    auto xq = unit_rows(rng, nq, d);
    float *qd, *Dd;
    int64_t* Id;
    CU(cudaMalloc(&qd, (size_t)nq * d * 4));
    CU(cudaMalloc(&Dd, (size_t)nq * k * 4));
    CU(cudaMalloc(&Id, (size_t)nq * k * 8));
    CU(cudaMemcpy(qd, xq.data(), (size_t)nq * d * 4, cudaMemcpyHostToDevice));
    cudaStream_t st;
    CU(cudaStreamCreate(&st));
    CK(kirag_index_search_async(h, qd, nq, k, Dd, Id, 0, st));
    int64_t changed = -1;
    CK(kirag_index_search_finish(h, nullptr, &changed));
    std::vector<int64_t> I((size_t)nq * k), Ih;
    CU(cudaMemcpy(I.data(), Id, I.size() * 8, cudaMemcpyDeviceToHost));
    host_topk(xb, n, xq, nq, d, k, &Ih);
    int diff = 0;
    for (size_t i = 0; i < I.size(); ++i) diff += I[i] != Ih[i];
    printf("search_async + finish: changed=%lld, differences vs host %d %s\n", (long long)changed, diff, diff <= 1 ? "ok" : "BAD");
    if (diff > 1) exit(3);
    CU(cudaFree(qd)); CU(cudaFree(Dd)); CU(cudaFree(Id));
    CU(cudaStreamDestroy(st));
    CK(kirag_index_destroy(h));
}

// pooling epilogue: cluster / DSMEM kernel forward (mean + cls) and backward
static void case_pool() {
    std::mt19937 rng(3);
    std::normal_distribution<float> g(0.f, 1.f);
    const int B = 5, S = 37, H = 256;
    std::vector<float> hid((size_t)B * S * H);
    for (auto& v : hid) v = g(rng);
    std::vector<int64_t> mask((size_t)B * S, 0);
    const int lens[B] = {37, 1, 17, 8, 30};
    for (int b = 0; b < B; ++b)
        for (int s = 0; s < lens[b]; ++s) mask[(size_t)b * S + s] = 1;
    float *dh, *dout, *dnorm, *dgo, *dgh;
    int64_t* dm;
    CU(cudaMalloc(&dh, hid.size() * 4));
    CU(cudaMalloc(&dm, mask.size() * 8));
    CU(cudaMalloc(&dout, (size_t)B * H * 4));
    CU(cudaMalloc(&dnorm, (size_t)B * 4));
    CU(cudaMalloc(&dgo, (size_t)B * H * 4));
    CU(cudaMalloc(&dgh, hid.size() * 4));
    CU(cudaMemcpy(dh, hid.data(), hid.size() * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dm, mask.data(), mask.size() * 8, cudaMemcpyHostToDevice));
    for (int mode : {KIRAG_POOL_MEAN, KIRAG_POOL_CLS}) {
        CK(kirag_pool_normalize_fwd_saved(dh, dm, dout, dnorm, B, S, H, (int64_t)S * H, H, S, KIRAG_DTYPE_F32, KIRAG_MASK_I64, mode,
                                          1, 0, nullptr));
        std::vector<float> out((size_t)B * H);
        CU(cudaMemcpy(out.data(), dout, out.size() * 4, cudaMemcpyDeviceToHost));
        double worst = 0;
        for (int b = 0; b < B; ++b) {
            std::vector<double> p((size_t)H, 0.0);
            if (mode == KIRAG_POOL_MEAN) {
                for (int s = 0; s < lens[b]; ++s)
                    for (int c = 0; c < H; ++c) p[(size_t)c] += hid[((size_t)b * S + s) * H + c];
                for (auto& v : p) v /= lens[b];
            } else {
                for (int c = 0; c < H; ++c) p[(size_t)c] = hid[((size_t)b * S) * H + c];
            }
            double nn = 0;
            for (double v : p) nn += v * v;
            nn = std::max(std::sqrt(nn), 1e-12);
            for (int c = 0; c < H; ++c) worst = std::max(worst, std::fabs(p[(size_t)c] / nn - out[(size_t)b * H + c]));
        }
        CU(cudaMemcpy(dgo, dout, (size_t)B * H * 4, cudaMemcpyDeviceToDevice));
        CK(kirag_pool_normalize_backward(dgo, dout, dnorm, dm, dgh, B, S, H, S, KIRAG_DTYPE_F32, KIRAG_MASK_I64, mode, 1, 0, nullptr));
        CU(cudaDeviceSynchronize());
        printf("pool mode %d: max |out - fp64| = %.2e %s\n", mode, worst, worst < 1e-5 ? "ok" : "BAD");
        if (!(worst < 1e-5)) exit(3);
    }
    CU(cudaFree(dh)); CU(cudaFree(dm)); CU(cudaFree(dout)); CU(cudaFree(dnorm)); CU(cudaFree(dgo)); CU(cudaFree(dgh));
}

// peer exchange + merge: G ranks in this process, one stream each (the kernels spin on each other's flags)
static void case_exchange() {
    const int G = 4, nq = 9, k = 20;
    kirag_exchange_t* x[G];
    void* bufs[G];
    for (int g = 0; g < G; ++g) { CK(kirag_exchange_create(0, g, G, 16, 32, &x[g])); bufs[g] = kirag_exchange_buffer(x[g]); }
    for (int g = 0; g < G; ++g) CK(kirag_exchange_connect_ptrs(x[g], bufs));
    std::mt19937 rng(4);
    std::vector<std::vector<float>> D(G, std::vector<float>((size_t)nq * k));
    std::vector<std::vector<int64_t>> I(G, std::vector<int64_t>((size_t)nq * k));
    for (int g = 0; g < G; ++g)
        for (int q = 0; q < nq; ++q) {
            std::vector<std::pair<float, int64_t>> items;
            for (int j = 0; j < k; ++j) items.push_back({-(float)(rng() % 13) * 0.5f, (int64_t)g * 100000 + (int64_t)(rng() % 90000)});
            std::sort(items.begin(), items.end());
            for (int j = 0; j < k; ++j) { D[g][(size_t)q * k + j] = -items[(size_t)j].first; I[g][(size_t)q * k + j] = items[(size_t)j].second; }
        }
    float *dD[G], *oD[G];
    int64_t *dI[G], *oI[G];
    int* dF[G];
    cudaStream_t st[G];
    for (int round = 0; round < 3; ++round) {
        for (int g = 0; g < G; ++g) {
            if (round == 0) {
                CU(cudaMalloc(&dD[g], (size_t)nq * k * 4)); CU(cudaMalloc(&oD[g], (size_t)nq * k * 4));
                CU(cudaMalloc(&dI[g], (size_t)nq * k * 8)); CU(cudaMalloc(&oI[g], (size_t)nq * k * 8));
                CU(cudaMalloc(&dF[g], (size_t)nq * 4));
                CU(cudaStreamCreate(&st[g]));
                CU(cudaMemcpy(dD[g], D[g].data(), (size_t)nq * k * 4, cudaMemcpyHostToDevice));
                CU(cudaMemcpy(dI[g], I[g].data(), (size_t)nq * k * 8, cudaMemcpyHostToDevice));
            }
            std::vector<int> f((size_t)nq, 0);
            if (round == 1 && g == 2) f[3] = 1;
            CU(cudaMemcpy(dF[g], f.data(), (size_t)nq * 4, cudaMemcpyHostToDevice));
        }
        CU(cudaDeviceSynchronize());
        for (int g = 0; g < G; ++g)
            CK(kirag_exchange_merge_topk_flags(x[g], dD[g], dI[g], dF[g], nq, k, oD[g], oI[g], st[g]));
        CU(cudaDeviceSynchronize());
        // host merge
        int bad = 0;
        for (int q = 0; q < nq; ++q) {
            std::vector<std::pair<float, int64_t>> all;
            for (int g = 0; g < G; ++g)
                for (int j = 0; j < k; ++j) all.push_back({-D[g][(size_t)q * k + j], I[g][(size_t)q * k + j]});
            std::sort(all.begin(), all.end());
            for (int g = 0; g < G; ++g) {
                std::vector<int64_t> got((size_t)k);
                CU(cudaMemcpy(got.data(), oI[g] + (size_t)q * k, (size_t)k * 8, cudaMemcpyDeviceToHost));
                for (int j = 0; j < k; ++j) bad += got[(size_t)j] != all[(size_t)j].second;
            }
        }
        int any_ok = 1;
        for (int g = 0; g < G; ++g) any_ok &= kirag_exchange_last_any_flag(x[g]) == (round == 1 ? 1 : 0);
        printf("exchange round %d (G=%d): id mismatches %d, flag word %s\n", round, G, bad, any_ok ? "ok" : "BAD");
        if (bad || !any_ok) exit(3);
    }
    for (int g = 0; g < G; ++g) {
        CU(cudaFree(dD[g])); CU(cudaFree(oD[g])); CU(cudaFree(dI[g])); CU(cudaFree(oI[g])); CU(cudaFree(dF[g]));
        CU(cudaStreamDestroy(st[g]));
        CK(kirag_exchange_destroy(x[g]));
    }
}

static void case_topk() {
    std::mt19937 rng(5);
    const int nt = 3000, d = 64, nq = 7, k = 20;
    auto t = unit_rows(rng, nt, d);
    auto q = unit_rows(rng, nq, d);
    std::vector<float> D((size_t)nq * k);
    std::vector<int64_t> I((size_t)nq * k), Ih;
    for (int rep = 0; rep < 2; ++rep) CK(kirag_topk_ip(q.data(), nq, t.data(), nt, d, k, D.data(), I.data(), 0, 0, nullptr));
    host_topk(t, nt, q, nq, d, k, &Ih);
    int diff = 0;
    for (size_t i = 0; i < I.size(); ++i) diff += I[i] != Ih[i];
    printf("topk_ip (scratch index reused): differences vs host %d %s\n", diff, diff <= 1 ? "ok" : "BAD");
    if (diff > 1) exit(3);
    CK(kirag_topk_ip_release());
}

// host-resident master (KIRAG_INDEX_HOST_MASTER): 140k rows x 128, more than one 64-MB staging piece
static kirag_index_t* host_master_index(const std::vector<float>& xb, int n, int d) {
    kirag_index_t* h = nullptr;
    CK(kirag_index_create_ex(d, KIRAG_METRIC_INNER_PRODUCT, 0, KIRAG_INDEX_HOST_MASTER, &h));
    CK(kirag_index_add(h, xb.data(), n, 0, nullptr));
    int64_t dev_b = 0, host_b = 0;
    CK(kirag_index_storage_bytes(h, &dev_b, &host_b));
    if (host_b < (int64_t)n * d * 4 || dev_b >= (int64_t)n * d * 4) {
        printf("host master storage: device %lld B, host %lld B BAD\n", (long long)dev_b, (long long)host_b);
        exit(3);
    }
    return h;
}

// the rescoring gather from pinned host rows: three-launch tail of the filter path, every batch size
static void case_host_rescore() {
    std::mt19937 rng(6);
    const int n = 140000, d = 128, k = 10;
    auto xb = unit_rows(rng, n, d);
    kirag_index_t* h = host_master_index(xb, n, d);
    for (int nq : {1, 40, 200}) {
        auto xq = unit_rows(rng, nq, d);
        std::vector<float> D((size_t)nq * k);
        std::vector<int64_t> I((size_t)nq * k), Ih;
        kirag_search_stats_t st;
        CK(kirag_index_search_ex(h, xq.data(), nq, k, D.data(), I.data(), 0, 0, KIRAG_PATH_AUTO, &st, nullptr));
        host_topk(xb, n, xq, nq, d, k, &Ih);
        int diff = 0;
        double worst = 0;
        for (int q = 0; q < nq; ++q)
            for (int j = 0; j < k; ++j) {
                const size_t i = (size_t)q * k + j;
                diff += I[i] != Ih[i];
                double a = 0;
                for (int c = 0; c < d; ++c) a += (double)xq[(size_t)q * d + c] * xb[(size_t)I[i] * d + c];
                worst = std::max(worst, std::fabs(a - D[i]));
            }
        printf("host-master search nq=%d: fast=%lld, ids vs host fp64 %d, max |score - fp64| = %.2e %s\n", nq,
               (long long)st.n_fast, diff, worst, diff <= 2 && worst < 1e-5 ? "ok" : "BAD");
        if (diff > 2 || !(worst < 1e-5)) exit(3);
    }
    CK(kirag_index_destroy(h));
}

// the exact fp32 scan of a host master, staged through HBM in pieces (two pieces here)
static void case_host_exact() {
    std::mt19937 rng(7);
    const int n = 140000, d = 128, k = 10, nq = 20;
    auto xb = unit_rows(rng, n, d);
    kirag_index_t* h = host_master_index(xb, n, d);
    auto xq = unit_rows(rng, nq, d);
    std::vector<float> D((size_t)nq * k);
    std::vector<int64_t> I((size_t)nq * k), Ih;
    CK(kirag_index_search_ex(h, xq.data(), nq, k, D.data(), I.data(), 0, 0, KIRAG_PATH_EXACT, nullptr, nullptr));
    host_topk(xb, n, xq, nq, d, k, &Ih);
    int diff = 0;
    double worst = 0;
    for (int q = 0; q < nq; ++q)
        for (int j = 0; j < k; ++j) {
            const size_t i = (size_t)q * k + j;
            diff += I[i] != Ih[i];
            double a = 0;
            for (int c = 0; c < d; ++c) a += (double)xq[(size_t)q * d + c] * xb[(size_t)I[i] * d + c];
            worst = std::max(worst, std::fabs(a - D[i]));
        }
    printf("host-master staged exact scan nq=%d: ids vs host fp64 %d, max |score - fp64| = %.2e %s\n", nq, diff, worst,
           diff <= 1 && worst < 1e-5 ? "ok" : "BAD");
    if (diff > 1 || !(worst < 1e-5)) exit(3);
    CK(kirag_index_destroy(h));
}

// multi-device index with three shards on device 0: the top-k merge (shared-memory and workspace variants), ids remapped
// from the 128-row stripes, and the range merge; checked against the host answer and against a single-device index
static void case_multi_merge() {
    std::mt19937 rng(8);
    const int n = 5000, d = 64, nq = 6;
    auto xb = unit_rows(rng, n, d);
    auto xq = unit_rows(rng, nq, d);
    const int devs[3] = {0, 0, 0};
    kirag_index_t* m = nullptr;
    kirag_index_t* s = nullptr;
    CK(kirag_index_create_multi(d, KIRAG_METRIC_INNER_PRODUCT, devs, 3, 0, &m));
    CK(kirag_index_create(d, KIRAG_METRIC_INNER_PRODUCT, 0, &s));
    CK(kirag_index_add(m, xb.data(), 1000, 0, nullptr));
    CK(kirag_index_add(m, xb.data() + (size_t)1000 * d, n - 1000, 0, nullptr));
    CK(kirag_index_add(s, xb.data(), n, 0, nullptr));
    for (int k : {10, 2048}) {  // 2048: G*k too large for shared memory, the merge runs in its global workspace
        std::vector<float> D((size_t)nq * k), Ds((size_t)nq * k);
        std::vector<int64_t> I((size_t)nq * k), Is((size_t)nq * k), Ih;
        CK(kirag_index_search_ex(m, xq.data(), nq, k, D.data(), I.data(), 0, 7, KIRAG_PATH_AUTO, nullptr, nullptr));
        CK(kirag_index_search_ex(s, xq.data(), nq, k, Ds.data(), Is.data(), 0, 7, KIRAG_PATH_AUTO, nullptr, nullptr));
        host_topk(xb, n, xq, nq, d, std::min(k, 10), &Ih);
        int diff = 0, differ = 0;
        for (int q = 0; q < nq; ++q)
            for (int j = 0; j < std::min(k, 10); ++j) diff += I[(size_t)q * k + j] - 7 != Ih[(size_t)q * std::min(k, 10) + j];
        for (size_t i = 0; i < I.size(); ++i) differ += I[i] != Is[i] || memcmp(&D[i], &Ds[i], 4) != 0;
        printf("multi merge k=%d: ids vs host fp64 %d, entries differing from one device %d %s\n", k, diff, differ,
               diff <= 1 && differ == 0 ? "ok" : "BAD");
        if (diff > 1 || differ) exit(3);
    }
    std::vector<int64_t> lims(nq + 1), lims_s(nq + 1);
    CK(kirag_index_range_search(m, xq.data(), nq, 0.2f, 0, 3, KIRAG_PATH_AUTO, lims.data(), nullptr, nullptr));
    std::vector<float> D((size_t)lims[nq]);
    std::vector<int64_t> I((size_t)lims[nq]);
    CK(kirag_index_range_fetch(m, D.data(), I.data(), 0, nullptr));
    CK(kirag_index_range_search(s, xq.data(), nq, 0.2f, 0, 3, KIRAG_PATH_AUTO, lims_s.data(), nullptr, nullptr));
    std::vector<float> Ds((size_t)lims_s[nq]);
    std::vector<int64_t> Is((size_t)lims_s[nq]);
    CK(kirag_index_range_fetch(s, Ds.data(), Is.data(), 0, nullptr));
    const bool same = lims == lims_s && I == Is && memcmp(D.data(), Ds.data(), D.size() * 4) == 0;
    printf("multi range merge: %lld entries, equal to one device: %s\n", (long long)lims[nq], same ? "ok" : "BAD");
    if (!same || lims[nq] == 0) exit(3);
    CK(kirag_index_destroy(m));
    CK(kirag_index_destroy(s));
}

// row removal on small shapes: the removal bitmap (ids with duplicates and ids outside the index, and a range), the kept
// counts and the gather kernel, on a single-device index (d = 100: the scalar gather; d = 64: the 16-byte gather) and
// on three shards of one GPU; the rows left are checked against the host's compaction
static void case_remove_compact() {
    std::mt19937 rng(9);
    for (int d : {100, 64}) {
        for (int G : {1, 3}) {
            const int n = 3000;
            auto xb = unit_rows(rng, n, d);
            kirag_index_t* h = nullptr;
            const int devs[3] = {0, 0, 0};
            if (G == 1) CK(kirag_index_create(d, KIRAG_METRIC_INNER_PRODUCT, 0, &h));
            else CK(kirag_index_create_multi(d, KIRAG_METRIC_INNER_PRODUCT, devs, G, 0, &h));
            CK(kirag_index_add(h, xb.data(), n, 0, nullptr));
            std::vector<char> keep(n, 1);
            std::vector<int64_t> ids = {5, 5, -2, n, 129, 2999, 1000};
            for (int i = 1500; i < 1800; i += 3) ids.push_back(i);
            for (int64_t i : ids)
                if (i >= 0 && i < n) keep[(size_t)i] = 0;
            int64_t removed = -1, want = 0;
            for (char c : keep) want += !c;
            CK(kirag_index_remove_ids(h, ids.data(), (int64_t)ids.size(), &removed, nullptr));
            std::vector<float> rows;
            for (int i = 0; i < n; ++i)
                if (keep[(size_t)i]) rows.insert(rows.end(), xb.begin() + (size_t)i * d, xb.begin() + (size_t)(i + 1) * d);
            // then a range, in the new ids
            const int64_t lo = 200, hi = 700;
            int64_t removed_r = -1;
            CK(kirag_index_remove_range(h, lo, hi, &removed_r, nullptr));
            rows.erase(rows.begin() + lo * d, rows.begin() + hi * d);
            const int64_t nt = kirag_index_ntotal(h);
            std::vector<float> got((size_t)nt * d);
            CK(kirag_index_reconstruct(h, 0, nt, got.data(), 0, nullptr));
            const bool ok = removed == want && removed_r == hi - lo && nt == (int64_t)(rows.size() / d) &&
                            memcmp(got.data(), rows.data(), rows.size() * 4) == 0;
            printf("remove compact d=%d G=%d: %lld + %lld rows removed, %lld left %s\n", d, G, (long long)removed,
                   (long long)removed_r, (long long)nt, ok ? "ok" : "BAD");
            if (!ok) exit(3);
            CK(kirag_index_destroy(h));
        }
    }
}

// id map (KIRAG_INDEX_ID_MAP) on small shapes, single-device and three shards of one GPU: add with ids (negative and
// repeated ids), a search whose ids must be the ids of the host's top-k rows (d = 64: the filter path and the fused tail
// or final kernel; the multi-device merge), then a batch removal by id (the device sort and the binary-search marking)
// and a range removal by id value, each checked against the host's restatement of the table
static void case_id_map() {
    std::mt19937 rng(10);
    const int n = 3000, d = 64, nq = 4, k = 10;
    for (int G : {1, 3}) {
        auto xb = unit_rows(rng, n, d);
        auto xq = unit_rows(rng, nq, d);
        std::vector<int64_t> ids((size_t)n);
        for (int i = 0; i < n; ++i) ids[(size_t)i] = ((int64_t)(i * 7919 % n) - 1000) * 1000003;
        for (int i = 0; i < 40; ++i) ids[(size_t)(2000 + i)] = ids[(size_t)i];  // repeated ids
        kirag_index_t* h = nullptr;
        const int devs[3] = {0, 0, 0};
        if (G == 1) CK(kirag_index_create_ex(d, KIRAG_METRIC_INNER_PRODUCT, 0, KIRAG_INDEX_ID_MAP, &h));
        else CK(kirag_index_create_multi(d, KIRAG_METRIC_INNER_PRODUCT, devs, G, KIRAG_INDEX_ID_MAP, &h));
        CK(kirag_index_add_with_ids(h, xb.data(), ids.data(), n, 0, nullptr));
        std::vector<float> D((size_t)nq * k);
        std::vector<int64_t> I((size_t)nq * k), Ih;
        CK(kirag_index_search(h, xq.data(), nq, k, D.data(), I.data(), 0, 0, nullptr));
        host_topk(xb, n, xq, nq, d, k, &Ih);
        bool ok = true;
        for (size_t j = 0; j < I.size(); ++j) ok = ok && I[j] == ids[(size_t)Ih[j]];
        // batch by id (with an absent id and a repeat), then a range of id values
        std::vector<int64_t> sel = {ids[5], ids[5], ids[77], 123456789, ids[2999]};
        for (int i = 1500; i < 1800; i += 3) sel.push_back(ids[(size_t)i]);
        std::vector<int64_t> keep_ids;
        for (int64_t v : ids)
            if (std::find(sel.begin(), sel.end(), v) == sel.end()) keep_ids.push_back(v);
        int64_t removed = -1;
        CK(kirag_index_remove_ids(h, sel.data(), (int64_t)sel.size(), &removed, nullptr));
        ok = ok && removed == n - (int64_t)keep_ids.size();
        const int64_t lo = -300LL * 1000003, hi = 200LL * 1000003;
        std::vector<int64_t> left;
        for (int64_t v : keep_ids)
            if (v < lo || v >= hi) left.push_back(v);
        int64_t removed_r = -1;
        CK(kirag_index_remove_range(h, lo, hi, &removed_r, nullptr));
        const int64_t nt = kirag_index_ntotal(h);
        std::vector<int64_t> table((size_t)nt);
        CK(kirag_index_id_map(h, 0, nt, table.data(), 0, nullptr));
        ok = ok && removed_r == (int64_t)(keep_ids.size() - left.size()) && table == left;
        printf("id map G=%d: search mapped, %lld + %lld rows removed by id, %lld left %s\n", G, (long long)removed,
               (long long)removed_r, (long long)nt, ok ? "ok" : "BAD");
        if (!ok) exit(3);
        CK(kirag_index_destroy(h));
    }
}

int main(int argc, char** argv) {
    const std::string which = argc > 1 ? argv[1] : "all";
    if (which == "scan" || which == "all") case_scan();
    if (which == "search" || which == "all") case_search();
    if (which == "pool" || which == "all") case_pool();
    if (which == "exchange" || which == "all") case_exchange();
    if (which == "topk" || which == "all") case_topk();
    if (which == "host_rescore" || which == "all") case_host_rescore();
    if (which == "host_exact" || which == "all") case_host_exact();
    if (which == "multi_merge" || which == "all") case_multi_merge();
    if (which == "remove_compact" || which == "all") case_remove_compact();
    if (which == "id_map" || which == "all") case_id_map();
    CU(cudaDeviceSynchronize());
    printf("sanitize_driver %s: passed\n", which.c_str());
    return 0;
}
