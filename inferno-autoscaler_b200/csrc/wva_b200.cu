// wva_b200.cu — C-ABI (include/wva_b200.h) over the sm_100a kernels.
//
// One ctx = one CUDA device + one stream.  All entry points launch kernels; there is no host
// implementation of any arithmetic in this file (and no fallback when CUDA is unavailable).
#include "wva_kernels.cuh"

#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace wva;

namespace {

std::string g_create_error;

// dynamic shared memory of k_greedy_solve / k_greedy_solve_ranked: 11264 heap entries of 20 bytes,
// or the rank bitmap of 1.7 M states
constexpr int kGreedySmem = 220 * 1024;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes < 256 ? 256 : bytes;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        cudaError_t e = cudaMallocHost(&p, bytes < 4096 ? 4096 : bytes);
        if (e == cudaSuccess) cap = bytes < 4096 ? 4096 : bytes;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

}  // namespace

// NCCL, resolved at run time: the library has no link-time dependency on it (a box without NCCL can
// still run single-GPU), and inside a process that already loaded a libnccl.so.2 (PyTorch's bundled
// one) the same copy is used.  Only the handful of entry points the path needs; their C ABI has been
// stable across NCCL 2.x.
namespace {
typedef struct ncclComm* nccl_comm_t;
struct nccl_unique_id { char internal[128]; };
struct NcclApi {
    void* handle = nullptr;
    int (*GetUniqueId)(nccl_unique_id*) = nullptr;
    int (*CommInitRank)(nccl_comm_t*, int, nccl_unique_id, int) = nullptr;
    int (*CommInitAll)(nccl_comm_t*, int, const int*) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string err;
    bool ok = false;
};
NcclApi g_nccl;
std::once_flag g_nccl_once;
const NcclApi& nccl_api() {
    std::call_once(g_nccl_once, [] {
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) { g_nccl.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (g_nccl.handle) break; }
        if (!g_nccl.handle) { g_nccl.err = std::string("dlopen(libnccl.so.2): ") + (dlerror() ? dlerror() : "not found"); return; }
        auto sym = [&](const char* n) { void* p = dlsym(g_nccl.handle, n); if (!p) g_nccl.err = std::string("missing NCCL symbol ") + n; return p; };
        g_nccl.GetUniqueId = (int (*)(nccl_unique_id*))sym("ncclGetUniqueId");
        g_nccl.CommInitRank = (int (*)(nccl_comm_t*, int, nccl_unique_id, int))sym("ncclCommInitRank");
        g_nccl.CommInitAll = (int (*)(nccl_comm_t*, int, const int*))sym("ncclCommInitAll");
        g_nccl.CommDestroy = (int (*)(nccl_comm_t))sym("ncclCommDestroy");
        g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t))sym("ncclAllGather");
        g_nccl.GroupStart = (int (*)())sym("ncclGroupStart");
        g_nccl.GroupEnd = (int (*)())sym("ncclGroupEnd");
        g_nccl.GetErrorString = (const char* (*)(int))sym("ncclGetErrorString");
        g_nccl.ok = g_nccl.err.empty();
    });
    return g_nccl;
}
constexpr int kNcclChar = 0;   // ncclInt8 / ncclChar
}  // namespace

// One helper thread per context: runs the candidate sweep's host side while the calling thread
// drives the pair sizing (both have stream synchronisations in the middle).
struct SweepWorker {
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::function<void()> job;
    bool has = false, done = false, quit = false;
    void start() {
        th = std::thread([this] {
            std::unique_lock<std::mutex> lk(m);
            for (;;) {
                cv.wait(lk, [this] { return has || quit; });
                if (quit) return;
                std::function<void()> j = std::move(job);
                has = false;
                lk.unlock();
                j();
                lk.lock();
                done = true;
                cv.notify_all();
            }
        });
    }
    void submit(std::function<void()> j) {
        { std::lock_guard<std::mutex> lk(m); job = std::move(j); has = true; done = false; }
        cv.notify_all();
    }
    void wait() { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [this] { return done; }); }
    void stop() {
        if (!th.joinable()) return;
        { std::lock_guard<std::mutex> lk(m); quit = true; }
        cv.notify_all();
        th.join();
    }
};

struct wva_ctx {
    int device = 0;
    SweepWorker worker;
    // wva_analyze: the calling thread does not enter its first stream synchronisation before the sweep thread
    // has issued its kernel (a thread blocked in a synchronisation call can hold up the other's launches)
    std::atomic<bool> sweep_launched{true};
    // host-side plan of the per-pair service-rate tables of k_pairs_warp: an upper bound of every pair's
    // N from the uploaded image (pair_batch_size without the validity tests), offsets for the shard
    std::vector<long long> hostN;
    bool plan_valid = false;
    long long plan_total = 0, plan_maxN = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t gstream = nullptr;      // the candidate sweep has its own stream so it can overlap the pair sizing
    cudaStream_t gstream2 = nullptr;     // k_scan_lean runs beside k_scan_cert and the exact-chain kernels
    cudaEvent_t evPrep = nullptr, evLean = nullptr;
    cudaEvent_t evg0 = nullptr, evg1 = nullptr, evJoin = nullptr, evFork = nullptr;
    std::mutex errMutex;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr;
    std::string err;
    std::atomic<int64_t> launches{0};
    int64_t phase_usec[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};

    // system image: arrays are laid out with spare rows (Scap servers, Mcap models) so that the incremental
    // updates of pkg/core/system.go:99-171 touch only the rows that change (wva_system_update_*)
    int Scap = 0, Mcap = 0;
    size_t off_srv[15] = {0}, off_perf[8] = {0}, off_cap = 0;
    int64_t last_h2d_bytes = 0;
    std::vector<int32_t> h_srv_model, h_srv_out, h_srv_mb, h_pmb, h_pat;    // host copies that size the pair tables (hostN)
    std::vector<float> h_srv_arr;
    bool have_system = false;
    DevSystem dsys{};
    DevBuf arena;
    PinnedBuf staging;
    int S = 0, A = 0, M = 0, T = 0;
    int s0 = 0, ns = 0;

    // pair results (full S*A extent; a rank fills its shard rows)
    DevBuf pairBuf; DevAllocs pairs{}; unsigned char* feasible = nullptr;
    bool pairs_valid = false; bool pairs_complete = false;
    DevBuf pairN, pairOrder, pairHist, slowList, slowCount, stepCounter, scratch, scratchOff, pairTabs, pairTabOff, pairPbuf;
    int pairs_warp_max = 1 << 22;
    int pairs_pstore = 0;
    int pairs_smem = 1;
    int certified = 1;
    int grid_rows = 1;
    int grid_scan = 1;          // certified sweeps: 1 = the scan kernels k_scan_prep / k_scan_cert / k_scan_lean (default), 0 = the round-1 kernels
    int pairs_debug = 0;
    DevBuf pairDbg;

    // solution
    DevBuf chosenBuf; DevAllocs chosen{}; int* chosen_acc = nullptr; bool solved = false;
    DevBuf totals;
    DevBuf greedyBuf;
    bool greedy_attr = false;
    int grid_list_warp = 1;     // deferred sweep chains: one warp per chain when the list is short
    int grid_fused = 1;         // scan mode: no host round trip between the sweep kernels and the exact chains when the list is long
    int greedy_ranked = 2;      // 2: static-order scan, 1: ranked queue, 0: always the heap kernel
    int greedy_path = 0;        // last limited solve: 1 heap, 2 ranked queue, 3 static-order scan
    uint64_t greedy_stats[4] = {0, 0, 0, 0};
    unsigned long long* greedy_stats_dev = nullptr;

    // grid
    DevBuf keys, bestDev, cube, status, counters, gridSlow, gridSlowCount, faultList, faultCount;
    DevBuf heavyList, heavyCost, heavyOrder, heavyHist, pairTab, blockSlot, listSlot, gscratch, rowInfo, rateTab;
    int grid_tail_cap = -1; int last_heavy = 0, last_slow = 0, last_heavy_slice = 0;
    int last_fused = 0;         // the last sweep slice did not stop at the host between its kernels
    int heavy_hint = 0;         // deferred chains of the last slice swept (survives across calls: reconciles repeat)
    cudaEvent_t evh0 = nullptr, evh1 = nullptr;
    // solve / totals phases: own event pairs, read lazily (a call that returns nothing to the host does not
    // wait for the device; wva_phase_time_usec does)
    cudaEvent_t evS0 = nullptr, evS1 = nullptr, evT0 = nullptr, evT1 = nullptr;
    mutable bool pendS = false, pendT = false;
    int grid_r = 0, grid_b = 0; bool grid_valid = false;
    uint64_t grid_counters[3] = {0, 0, 0};
    // per-(server, accelerator) sweep winners (wva_grid_set_pair_winners): full S*A extent like the pair records,
    // a rank fills its shard rows; valid/complete as pairs_valid/pairs_complete
    int grid_pair_winners = 0;
    DevBuf gridPairBuf, gridPairKeys; DevAllocs gridPairs{}; unsigned char* gridFeasible = nullptr;
    bool gpairs_valid = false, gpairs_complete = false;
    DevBuf sizeStatus, sizeList, sizeCount;   // wva_grid_pairs_size
    // wva_analyze_scenarios: records of n_scen scenarios (full S*A extent each, a rank fills its shard rows), their
    // unlimited solutions and totals; separate from everything above, which the call leaves untouched
    DevBuf scenRates, scenRecBuf, scenChosenBuf, scenTotals, scenGather, scenList, scenCount, scenCfg, scenRate, scenMetrics, scenStatus;
    DevAllocs scenPairs{}, scenChosen{}; unsigned char* scenFeasible = nullptr; int* scenChosenAcc = nullptr;
    int scen_n = 0; bool scen_valid = false;

    // multi-rank exchange (wva_comm_init / wva_group_create)
    nccl_comm_t comm = nullptr; int comm_rank = 0, comm_size = 1; bool comm_owned = false;
    DevBuf commTotals, commChunk, commGather;

    // misc io buffers for the low-level API
    DevBuf ioA, ioB, ioC, ioD, ioE, ioF, ioG;
};

namespace {

int fail(wva_ctx* c, int code, const std::string& msg) {
    if (c) { std::lock_guard<std::mutex> g(c->errMutex); c->err = msg; } else g_create_error = msg;
    return code;
}
#define CK(expr)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return fail(ctx, WVA_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));       \
    } while (0)
#define LAUNCH_CHECK()                                                                             \
    do {                                                                                           \
        ctx->launches++;                                                                           \
        cudaError_t _e = cudaGetLastError();                                                       \
        if (_e != cudaSuccess) return fail(ctx, WVA_ECUDA, std::string("kernel launch: ") + cudaGetErrorString(_e)); \
    } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct PhaseTimer {
    wva_ctx* c; int phase; cudaStream_t st; cudaEvent_t e0, e1;
    PhaseTimer(wva_ctx* c_, int p) : c(c_), phase(p), st(c_->stream), e0(c_->ev0), e1(c_->ev1) { cudaEventRecord(e0, st); }
    PhaseTimer(wva_ctx* c_, int p, cudaStream_t s, cudaEvent_t a, cudaEvent_t b) : c(c_), phase(p), st(s), e0(a), e1(b) { cudaEventRecord(e0, st); }
    // call after the stream has been synchronised (or will be by the event sync below)
    void stop() {
        cudaEventRecord(e1, st);
        cudaEventSynchronize(e1);
        float ms = 0.0f;
        cudaEventElapsedTime(&ms, e0, e1);
        c->phase_usec[phase] = (int64_t)(ms * 1000.0f + 0.5f);
    }
};

// carve a DevAllocs of n records out of one buffer
cudaError_t carve_allocs(DevBuf& buf, size_t n, DevAllocs& a, unsigned char** feasible, int** chosen_acc) {
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    size_t o_rep = take(n * 8), o_bat = take(n * 8), o_acc = take(n * 4), o_cost = take(n * 4), o_val = take(n * 4),
           o_itl = take(n * 4), o_ttft = take(n * 4), o_rho = take(n * 4), o_arr = take(n * 4), o_fe = take(n),
           o_ch = chosen_acc ? take(n * 4) : 0;
    cudaError_t e = buf.ensure(off);
    if (e != cudaSuccess) return e;
    char* b = buf.as<char>();
    a.num_replicas = (long long*)(b + o_rep); a.batch_size = (long long*)(b + o_bat); a.acc = (int*)(b + o_acc);
    a.cost = (float*)(b + o_cost); a.value = (float*)(b + o_val); a.itl = (float*)(b + o_itl);
    a.ttft = (float*)(b + o_ttft); a.rho = (float*)(b + o_rho); a.max_arrv = (float*)(b + o_arr);
    if (feasible) *feasible = (unsigned char*)(b + o_fe);
    if (chosen_acc) *chosen_acc = (int*)(b + o_ch);
    return cudaSuccess;
}

cudaError_t download_allocs(wva_ctx* ctx, const DevAllocs& d, size_t first, size_t n, wva_alloc_soa* h, size_t hfirst) {
    cudaError_t e;
#define DL(field, dfield, T)                                                                                         \
    if (h->field) {                                                                                                  \
        e = cudaMemcpyAsync(h->field + hfirst, d.dfield + first, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream); \
        if (e != cudaSuccess) return e;                                                                              \
    }
    DL(acc, acc, int32_t) DL(num_replicas, num_replicas, int64_t) DL(batch_size, batch_size, int64_t)
    DL(cost, cost, float) DL(value, value, float) DL(itl, itl, float) DL(ttft, ttft, float) DL(rho, rho, float)
    DL(max_arrv_rate_per_replica, max_arrv, float)
#undef DL
    return cudaSuccess;
}

// rows [first, first + n) of each of `blocks` consecutive blocks of `pitch` records, into the same places of h
cudaError_t download_allocs_blocks(wva_ctx* ctx, const DevAllocs& d, size_t first, size_t n, size_t pitch, size_t blocks, wva_alloc_soa* h) {
    cudaError_t e;
#define DL(field, dfield, T)                                                                                              \
    if (h->field) {                                                                                                       \
        e = cudaMemcpy2DAsync(h->field + first, pitch * sizeof(T), d.dfield + first, pitch * sizeof(T), n * sizeof(T), blocks, \
                              cudaMemcpyDeviceToHost, ctx->stream);                                                       \
        if (e != cudaSuccess) return e;                                                                                   \
    }
    DL(acc, acc, int32_t) DL(num_replicas, num_replicas, int64_t) DL(batch_size, batch_size, int64_t)
    DL(cost, cost, float) DL(value, value, float) DL(itl, itl, float) DL(ttft, ttft, float) DL(rho, rho, float)
    DL(max_arrv_rate_per_replica, max_arrv, float)
#undef DL
    return cudaSuccess;
}

// limited mode with a communicator: every rank packs the candidate records of its shard into one chunk,
// ONE ncclAllGather moves all chunks, the other ranks' rows are scattered into place.
int comm_gather_pairs(wva_ctx* ctx, const DevAllocs& recs, unsigned char* feasible, bool& complete) {
    const NcclApi& nc = nccl_api();
    if (!nc.ok) return fail(ctx, WVA_ECUDA, "NCCL unavailable: " + nc.err);
    const int A = ctx->A, G = ctx->comm_size;
    const size_t capServers = ((size_t)ctx->S + G - 1) / G;
    if ((size_t)ctx->ns > capServers)
        return fail(ctx, WVA_EINVAL, "shard larger than ceil(S / ranks): use wva_comm_shard for the limited-capacity exchange");
    const size_t cap = (capServers ? capServers : 1) * A;
    const size_t chunkBytes = pair_chunk_bytes(cap);
    CK(ctx->commChunk.ensure(chunkBytes));
    CK(ctx->commGather.ensure(chunkBytes * G));
    const int nPairs = ctx->ns * A;
    k_pairs_pack<<<(nPairs + 255) / 256 + 1, 256, 0, ctx->stream>>>(recs, feasible, ctx->s0 * A, nPairs, cap, ctx->commChunk.as<unsigned char>());
    LAUNCH_CHECK();
    int nrc = nc.AllGather(ctx->commChunk.p, ctx->commGather.p, chunkBytes, kNcclChar, ctx->comm, ctx->stream);
    if (nrc != 0) return fail(ctx, WVA_ECUDA, std::string("ncclAllGather(pairs): ") + nc.GetErrorString(nrc));
    dim3 grid((unsigned)((cap + 255) / 256 < 1024 ? (cap + 255) / 256 : 1024), (unsigned)G);
    k_pairs_unpack<<<grid, 256, 0, ctx->stream>>>(ctx->commGather.as<unsigned char>(), chunkBytes, cap, ctx->comm_rank, (size_t)ctx->S * A,
                                                   recs, feasible);
    LAUNCH_CHECK();
    complete = true;
    return WVA_OK;
}

}  // namespace

extern "C" {

int wva_abi_version(void) { return WVA_ABI_VERSION; }

const char* wva_last_error(const wva_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int wva_ctx_create(int device, wva_ctx** out) {
    wva_ctx* ctx = nullptr;
    if (!out) return fail(nullptr, WVA_EINVAL, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, WVA_ECUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0"));
    if (device < 0 || device >= n) return fail(nullptr, WVA_EINVAL, "device index out of range");
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, WVA_ECUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(nullptr, WVA_ECUDA, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, WVA_ECUDA, "device is not sm_100 class; this library carries sm_100a code only");
    ctx = new wva_ctx;
    ctx->device = device;
    int prioLo = 0, prioHi = 0;                       // numerically lower = more urgent
    cudaDeviceGetStreamPriorityRange(&prioLo, &prioHi);
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->evk0)) != cudaSuccess || (e = cudaEventCreate(&ctx->evk1)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->evh0)) != cudaSuccess || (e = cudaEventCreate(&ctx->evh1)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->evS0)) != cudaSuccess || (e = cudaEventCreate(&ctx->evS1)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->evT0)) != cudaSuccess || (e = cudaEventCreate(&ctx->evT1)) != cudaSuccess ||
        // the sweep's stream outranks the one of its cube-writing half (k_scan_lean): when the exact-chain kernel and
        // k_scan_lean become runnable together, the few blocks of the former are placed first (see grid_run)
        (e = cudaStreamCreateWithPriority(&ctx->gstream, cudaStreamNonBlocking, prioHi)) != cudaSuccess ||
        (e = cudaStreamCreateWithPriority(&ctx->gstream2, cudaStreamNonBlocking, prioLo)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&ctx->evPrep, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&ctx->evLean, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->evg0)) != cudaSuccess || (e = cudaEventCreate(&ctx->evg1)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&ctx->evJoin, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&ctx->evFork, cudaEventDisableTiming)) != cudaSuccess) {
        std::string msg = std::string("stream/event create: ") + cudaGetErrorString(e);
        delete ctx;
        return fail(nullptr, WVA_ECUDA, msg);
    }
    // The pair kernel and the sweep run side by side on two streams.  They ask for different amounts of shared
    // memory; with the default (per-kernel) L1/shared split an SM has to drain before it can take blocks of the
    // other kernel, and the two were observed to run one after the other every other step.  One split for all.
    {
        const void* kernels[] = {(const void*)k_grid, (const void*)k_grid_rows, (const void*)k_grid_wrow, (const void*)k_grid_list,
                                 (const void*)k_grid_list_warp, (const void*)k_pairs_warp, (const void*)k_pairs, (const void*)k_grid_claim,
                                 (const void*)k_grid_best_init, (const void*)k_scan_prep, (const void*)k_scan_cert<2>, (const void*)k_scan_cert<3>, (const void*)k_scan_lean};
        if (!std::getenv("WVA_NO_CARVEOUT"))
            for (const void* k : kernels) cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaGetLastError();
    }
    *out = ctx;
    return WVA_OK;
}

void wva_ctx_destroy(wva_ctx* ctx) {
    if (!ctx) return;
    ctx->worker.stop();
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->comm && ctx->comm_owned && nccl_api().ok) nccl_api().CommDestroy(ctx->comm);
    ctx->comm = nullptr;
    DevBuf* bufs[] = {&ctx->arena, &ctx->pairBuf, &ctx->pairN, &ctx->pairOrder, &ctx->pairHist, &ctx->slowList,
                      &ctx->slowCount, &ctx->stepCounter, &ctx->scratch, &ctx->scratchOff, &ctx->pairTabs, &ctx->pairTabOff, &ctx->pairPbuf, &ctx->chosenBuf, &ctx->totals,
                      &ctx->greedyBuf, &ctx->keys, &ctx->bestDev, &ctx->cube, &ctx->status, &ctx->counters,
                      &ctx->gridSlow, &ctx->gridSlowCount, &ctx->faultList, &ctx->faultCount, &ctx->heavyList, &ctx->heavyCost,
                      &ctx->heavyOrder, &ctx->heavyHist, &ctx->pairTab, &ctx->blockSlot, &ctx->listSlot, &ctx->gscratch, &ctx->rowInfo, &ctx->rateTab, &ctx->ioA, &ctx->ioB,
                      &ctx->ioC, &ctx->ioD, &ctx->ioE, &ctx->ioF, &ctx->ioG, &ctx->commTotals, &ctx->commChunk, &ctx->commGather,
                      &ctx->sizeStatus, &ctx->sizeList, &ctx->sizeCount, &ctx->scenRates, &ctx->scenRecBuf, &ctx->scenChosenBuf,
                      &ctx->scenTotals, &ctx->scenGather, &ctx->scenList, &ctx->scenCount, &ctx->scenCfg, &ctx->scenRate,
                      &ctx->scenMetrics, &ctx->scenStatus};
    for (DevBuf* b : bufs) b->release();
    ctx->staging.release();
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    cudaEventDestroy(ctx->evk0);
    cudaEventDestroy(ctx->evk1);
    cudaEventDestroy(ctx->evh0);
    cudaEventDestroy(ctx->evh1);
    cudaEventDestroy(ctx->evS0); cudaEventDestroy(ctx->evS1); cudaEventDestroy(ctx->evT0); cudaEventDestroy(ctx->evT1);
    cudaEventDestroy(ctx->evg0);
    cudaEventDestroy(ctx->evg1);
    cudaEventDestroy(ctx->evJoin);
    cudaEventDestroy(ctx->evFork);
    cudaEventDestroy(ctx->evPrep); cudaEventDestroy(ctx->evLean);
    cudaStreamDestroy(ctx->gstream2);
    cudaStreamDestroy(ctx->gstream);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

void* wva_stream(const wva_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int64_t wva_launch_count(const wva_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }
static void resolve_lazy_timers(const wva_ctx* ctx) {
    wva_ctx* c = const_cast<wva_ctx*>(ctx);
    float ms = 0.0f;
    if (c->pendS && cudaEventSynchronize(c->evS1) == cudaSuccess && cudaEventElapsedTime(&ms, c->evS0, c->evS1) == cudaSuccess)
        c->phase_usec[WVA_PHASE_SOLVE] = (int64_t)(ms * 1000.0f + 0.5f);
    if (c->pendT && cudaEventSynchronize(c->evT1) == cudaSuccess && cudaEventElapsedTime(&ms, c->evT0, c->evT1) == cudaSuccess)
        c->phase_usec[WVA_PHASE_TOTALS] = (int64_t)(ms * 1000.0f + 0.5f);
    c->pendS = c->pendT = false;
}
int64_t wva_phase_time_usec(const wva_ctx* ctx, int phase) {
    if (!ctx || phase < 0 || phase >= 9) return 0;
    resolve_lazy_timers(ctx);
    return ctx->phase_usec[phase];
}
int64_t wva_solution_time_usec(const wva_ctx* ctx) { return wva_phase_time_usec(ctx, WVA_PHASE_SOLVE); }

// N of CreateAllocation (allocation.go:77-87) per pair of servers [s0, s1), or an upper bound where the device
// finds the pair unusable (it then needs no table at all): sizes the tables of the warp-per-pair kernel
// without a device round trip
static void host_plan_rows(wva_ctx* ctx, int s0, int s1) {
    const int A = ctx->A;
    for (int s = s0; s < s1; ++s) {
        const int m = ctx->h_srv_model[(size_t)s];
        const long long outTok = ctx->h_srv_out[(size_t)s];
        for (int a = 0; a < A; ++a) ctx->hostN[(size_t)s * A + a] = 0;
        if (ctx->h_srv_arr[(size_t)s] == 0.0f || outTok == 0) continue;
        for (int a = 0; a < A; ++a) {
            long long n;
            if (ctx->h_srv_mb[(size_t)s] > 0) n = ctx->h_srv_mb[(size_t)s];
            else if (m < 0) n = 0;
            else {
                const size_t pi = (size_t)m * A + a;
                const long long prod = (long long)((unsigned long long)(long long)ctx->h_pmb[pi] * (unsigned long long)(long long)ctx->h_pat[pi]);
                n = (outTok == -1) ? (long long)(0ull - (unsigned long long)prod) : prod / outTok;
                if (n < 1) n = 1;
            }
            ctx->hostN[(size_t)s * A + a] = n;
        }
    }
}

// ---------------------------------------------------------------------------------------------
int wva_system_upload(wva_ctx* ctx, const wva_system_soa* h) {
    if (!ctx || !h) return fail(ctx, WVA_EINVAL, "null argument");
    CK(cudaSetDevice(ctx->device));
    const int S = h->n_servers, A = h->n_accels, M = h->n_models, T = h->n_types;
    if (S < 0 || A <= 0 || M < 0 || T <= 0) return fail(ctx, WVA_EINVAL, "bad dimensions");
    if ((size_t)S * (size_t)A > 0x7fffffffULL) return fail(ctx, WVA_EINVAL, "S*A exceeds 2^31-1");
    // validation of the index arrays (cheap, host side; no arithmetic of the path happens here)
    for (int a = 0; a < A; ++a)
        if (h->acc_type[a] < 0 || h->acc_type[a] >= T) return fail(ctx, WVA_EINVAL, "acc_type out of range");
    for (int s = 0; s < S; ++s) {
        if (h->srv_model[s] >= M) return fail(ctx, WVA_EINVAL, "srv_model out of range");
        if (h->srv_cur_acc[s] < WVA_ACC_UNKNOWN || h->srv_cur_acc[s] >= A) return fail(ctx, WVA_EINVAL, "srv_cur_acc out of range");
        if (h->srv_priority[s] < 1 || h->srv_priority[s] > 100)
            return fail(ctx, WVA_EINVAL, "srv_priority must be in [1,100] (Server.Priority(), serviceclass.go:28-37)");
    }
    PhaseTimer timer(ctx, WVA_PHASE_UPLOAD);
    struct Item { const void* src; size_t bytes; size_t off; };
    std::vector<Item> items;
    size_t off = 0;
    // spare rows for wva_system_update_servers / _models: 1/16 more, at least 64
    const int Scap = S + (S / 16 > 64 ? S / 16 : 64), Mcap = M + (M / 16 > 64 ? M / 16 : 64);
    auto add = [&](const void* src, size_t n, size_t cap, size_t elem) { items.push_back({src, n * elem, off}); size_t o = off; off = align_up(off + cap * elem, 256); return o; };
    const size_t MA = (size_t)M * A, MAcap = (size_t)Mcap * A;
    size_t o_acc_cost = add(h->acc_cost, A, A, 4), o_acc_mult = add(h->acc_multiplicity, A, A, 4), o_acc_type = add(h->acc_type, A, A, 4);
    size_t o_cap = add(h->type_capacity, (size_t)T, (size_t)T, 8);
    size_t o_pa = add(h->perf_alpha, MA, MAcap, 4), o_pb = add(h->perf_beta, MA, MAcap, 4), o_pg = add(h->perf_gamma, MA, MAcap, 4), o_pd = add(h->perf_delta, MA, MAcap, 4);
    size_t o_pmb = add(h->perf_max_batch, MA, MAcap, 4), o_pat = add(h->perf_at_tokens, MA, MAcap, 4), o_pac = add(h->perf_acc_count, MA, MAcap, 4), o_pv = add(h->perf_valid, MA, MAcap, 1);
    const size_t Sz = (size_t)S, Sc = (size_t)Scap;
    size_t o_sm = add(h->srv_model, Sz, Sc, 4), o_sar = add(h->srv_arrival_rpm, Sz, Sc, 4), o_sin = add(h->srv_in_tokens, Sz, Sc, 4),
           o_sout = add(h->srv_out_tokens, Sz, Sc, 4), o_stt = add(h->srv_slo_ttft, Sz, Sc, 4), o_sit = add(h->srv_slo_itl, Sz, Sc, 4),
           o_stp = add(h->srv_slo_tps, Sz, Sc, 4), o_stv = add(h->srv_target_valid, Sz, Sc, 1), o_spr = add(h->srv_priority, Sz, Sc, 4),
           o_smr = add(h->srv_min_replicas, Sz, Sc, 4), o_smb = add(h->srv_max_batch, Sz, Sc, 4), o_ska = add(h->srv_keep_acc, Sz, Sc, 1),
           o_sca = add(h->srv_cur_acc, Sz, Sc, 4), o_scr = add(h->srv_cur_replicas, Sz, Sc, 4), o_scc = add(h->srv_cur_cost, Sz, Sc, 4);
    const size_t total = off;
    ctx->Scap = Scap; ctx->Mcap = Mcap; ctx->off_cap = o_cap;
    {
        const size_t os_[15] = {o_sm, o_sar, o_sin, o_sout, o_stt, o_sit, o_stp, o_stv, o_spr, o_smr, o_smb, o_ska, o_sca, o_scr, o_scc};
        const size_t op_[8] = {o_pa, o_pb, o_pg, o_pd, o_pmb, o_pat, o_pac, o_pv};
        for (int i = 0; i < 15; ++i) ctx->off_srv[i] = os_[i];
        for (int i = 0; i < 8; ++i) ctx->off_perf[i] = op_[i];
    }
    ctx->last_h2d_bytes = (int64_t)total;
    CK(ctx->arena.ensure(total));
    CK(ctx->staging.ensure(total));
    char* st = (char*)ctx->staging.p;
    for (const Item& it : items) if (it.bytes) std::memcpy(st + it.off, it.src, it.bytes);
    CK(cudaMemcpyAsync(ctx->arena.p, st, total, cudaMemcpyHostToDevice, ctx->stream));
    char* d = ctx->arena.as<char>();
    DevSystem& ds = ctx->dsys;
    ds.S = S; ds.A = A; ds.M = M; ds.T = T; ds.cert = ctx->certified;
    ds.acc_cost = (const float*)(d + o_acc_cost); ds.acc_multiplicity = (const int*)(d + o_acc_mult); ds.acc_type = (const int*)(d + o_acc_type);
    ds.type_capacity = (const long long*)(d + o_cap);
    ds.perf_alpha = (const float*)(d + o_pa); ds.perf_beta = (const float*)(d + o_pb); ds.perf_gamma = (const float*)(d + o_pg); ds.perf_delta = (const float*)(d + o_pd);
    ds.perf_max_batch = (const int*)(d + o_pmb); ds.perf_at_tokens = (const int*)(d + o_pat); ds.perf_acc_count = (const int*)(d + o_pac); ds.perf_valid = (const unsigned char*)(d + o_pv);
    ds.srv_model = (const int*)(d + o_sm); ds.srv_arrival_rpm = (const float*)(d + o_sar); ds.srv_in_tokens = (const int*)(d + o_sin); ds.srv_out_tokens = (const int*)(d + o_sout);
    ds.srv_slo_ttft = (const float*)(d + o_stt); ds.srv_slo_itl = (const float*)(d + o_sit); ds.srv_slo_tps = (const float*)(d + o_stp); ds.srv_target_valid = (const unsigned char*)(d + o_stv);
    ds.srv_priority = (const int*)(d + o_spr); ds.srv_min_replicas = (const int*)(d + o_smr); ds.srv_max_batch = (const int*)(d + o_smb); ds.srv_keep_acc = (const unsigned char*)(d + o_ska);
    ds.srv_cur_acc = (const int*)(d + o_sca); ds.srv_cur_replicas = (const int*)(d + o_scr); ds.srv_cur_cost = (const float*)(d + o_scc);
    ctx->S = S; ctx->A = A; ctx->M = M; ctx->T = T;
    ctx->s0 = 0; ctx->ns = S;
    // host copies of what sizes the pair tables
    ctx->h_srv_model.assign(h->srv_model, h->srv_model + S); ctx->h_srv_out.assign(h->srv_out_tokens, h->srv_out_tokens + S);
    ctx->h_srv_mb.assign(h->srv_max_batch, h->srv_max_batch + S); ctx->h_srv_arr.assign(h->srv_arrival_rpm, h->srv_arrival_rpm + S);
    ctx->h_pmb.assign(h->perf_max_batch, h->perf_max_batch + MA); ctx->h_pat.assign(h->perf_at_tokens, h->perf_at_tokens + MA);
    ctx->hostN.assign((size_t)S * A, 0);
    host_plan_rows(ctx, 0, S);
    ctx->plan_valid = false;
    ctx->have_system = true;
    ctx->pairs_valid = ctx->pairs_complete = ctx->solved = ctx->grid_valid = ctx->gpairs_valid = ctx->gpairs_complete = ctx->scen_valid = false;
    timer.stop();
    return WVA_OK;
}

int wva_set_shard(wva_ctx* ctx, int32_t first, int32_t count) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    if (first < 0 || count < 0 || first + count > ctx->S) return fail(ctx, WVA_EINVAL, "shard out of range");
    ctx->s0 = first; ctx->ns = count;
    ctx->plan_valid = false;
    ctx->pairs_valid = ctx->pairs_complete = ctx->solved = ctx->grid_valid = ctx->gpairs_valid = ctx->gpairs_complete = ctx->scen_valid = false;
    return WVA_OK;
}

// ---------------------------------------------------------------------------------------------
int wva_analyze_pairs(wva_ctx* ctx, wva_alloc_soa* out, uint8_t* feasible) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    CK(cudaSetDevice(ctx->device));
    const int A = ctx->A;
    const size_t nAll = (size_t)ctx->S * A;
    const int nPairs = ctx->ns * A;
    CK(carve_allocs(ctx->pairBuf, nAll ? nAll : 1, ctx->pairs, &ctx->feasible, nullptr));
    CK(ctx->slowList.ensure((size_t)(nPairs ? nPairs : 1) * 4));
    CK(ctx->slowCount.ensure(4));
    CK(ctx->stepCounter.ensure(32));
    CK(ctx->pairN.ensure((size_t)(nPairs ? nPairs : 1) * 8));
    PhaseTimer timer(ctx, WVA_PHASE_PAIRS);
    CK(cudaMemsetAsync(ctx->slowCount.p, 0, 4, ctx->stream));
    CK(cudaMemsetAsync(ctx->stepCounter.p, 0, 32, ctx->stream));
    int slow = 0;
    if (nPairs > 0) {
        if (nPairs <= ctx->pairs_warp_max) {
            // latency-oriented variant: one warp per pair, per-pair {rate, reciprocal} tables in HBM; the table
            // plan comes from the host copy of N (made at upload) and is kept while image and shard stay
            if (!ctx->plan_valid) {
                std::vector<long long> offs((size_t)nPairs);
                long long total = 0, maxN = 0;
                const long long budget = (2LL << 30) / 16;          // at most 2 GB of tables
                const long long* nHost = ctx->hostN.data() + (size_t)ctx->s0 * A;
                for (int i = 0; i < nPairs; ++i) { const long long N = nHost[(size_t)i]; if (N > maxN && N <= (1LL << 26)) maxN = N; }
                // a pair whose table fits the warp's shared-memory slice (<= 3072 entries) needs no table in HBM at all: only
                // larger ones draw on the budget (round 1 reserved HBM for every pair; at 800 000 pairs per rank -- BASELINE
                // config 5 -- that blew the budget and sent most pairs to the materialised path)
                const long long inSmem = ctx->pairs_smem ? (maxN < 3072 ? maxN : 3072) : 0;
                for (int i = 0; i < nPairs; ++i) {
                    long long N = nHost[(size_t)i];
                    if (N <= 0 || N <= inSmem) { offs[(size_t)i] = 0; continue; }   // no queueing work, or table in shared memory: offset unused
                    if (N > (1LL << 26) || total + N > budget) { offs[(size_t)i] = -1; continue; }
                    offs[(size_t)i] = total; total += N;
                }
                CK(ctx->pairTabs.ensure((size_t)(total ? total : 1) * 16));
                CK(ctx->pairTabOff.ensure((size_t)nPairs * 8));
                CK(cudaMemcpyAsync(ctx->pairTabOff.p, offs.data(), (size_t)nPairs * 8, cudaMemcpyHostToDevice, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));               // offs is a local
                ctx->plan_total = total; ctx->plan_maxN = maxN; ctx->plan_valid = true;
            }
            const long long maxN = ctx->plan_maxN;
            const int warpsPerBlock = WVA_PAIRS_WARP_THREADS / 32;
            // shared-memory tables: up to 3072 entries (48 KB) per warp, 4 warps per block
            int smemEntries = ctx->pairs_smem ? (int)(maxN < 3072 ? maxN : 3072) : 0;
            const size_t smemBytes = (size_t)smemEntries * 16 * warpsPerBlock;
            if (smemBytes > 48 * 1024)
                CK(cudaFuncSetAttribute(k_pairs_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemBytes));
            // chain-value buffers (pass 2 reads p[n] back instead of re-running the recurrence): one
            // [K+1][32] block per pair while that stays under 4 GB
            const long long strideK = 11 * maxN + 1;
            double* pbuf = nullptr;
            if (ctx->pairs_pstore && maxN > 0 && (double)nPairs * (double)strideK * 256.0 <= 4.0 * (1u << 30)) {
                CK(ctx->pairPbuf.ensure((size_t)nPairs * (size_t)strideK * 256));
                pbuf = ctx->pairPbuf.as<double>();
            }
            if (ctx->pairs_debug) CK(ctx->pairDbg.ensure((size_t)nPairs * 16));
            k_pairs_warp<<<(nPairs + warpsPerBlock - 1) / warpsPerBlock, WVA_PAIRS_WARP_THREADS, smemBytes, ctx->stream>>>(
                ctx->dsys, ctx->s0, nPairs, ctx->pairTabOff.as<long long>(), ctx->pairTabs.as<double2>(), ctx->pairs, ctx->feasible,
                ctx->slowList.as<int>(), ctx->slowCount.as<int>(), ctx->stepCounter.as<unsigned long long>(), smemEntries, pbuf, strideK,
                ctx->pairs_debug ? ctx->pairDbg.as<unsigned long long>() : nullptr);
            LAUNCH_CHECK();
        } else {
        k_pair_batch<<<(nPairs + 255) / 256, 256, 0, ctx->stream>>>(ctx->dsys, ctx->s0, nPairs, ctx->pairN.as<long long>());
        LAUNCH_CHECK();
        const int* order = nullptr;
        if (nPairs > 1024) {
            // order pairs by chain length (bucket = bit length of N, heaviest first) so that the lanes
            // of a warp run chains of similar length
            CK(ctx->pairOrder.ensure((size_t)nPairs * 4));
            CK(ctx->pairHist.ensure(2 * 65 * 4));
            CK(cudaMemsetAsync(ctx->pairHist.p, 0, 2 * 65 * 4, ctx->stream));
            int* hist = ctx->pairHist.as<int>();
            k_pair_bucket_hist<<<(nPairs + 255) / 256, 256, 0, ctx->stream>>>(ctx->pairN.as<long long>(), nPairs, hist);
            LAUNCH_CHECK();
            int hh[65];
            CK(cudaMemcpyAsync(hh, hist, 65 * 4, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            int cur[65]; int run = 0;
            for (int b = 64; b >= 0; --b) { cur[b] = run; run += hh[b]; }
            CK(cudaMemcpyAsync(hist + 65, cur, 65 * 4, cudaMemcpyHostToDevice, ctx->stream));
            k_pair_bucket_scatter<<<(nPairs + 255) / 256, 256, 0, ctx->stream>>>(ctx->pairN.as<long long>(), nPairs, hist + 65,
                                                                                   ctx->pairOrder.as<int>());
            LAUNCH_CHECK();
            order = ctx->pairOrder.as<int>();
        }
        k_pairs<<<(nPairs + 127) / 128, 128, 0, ctx->stream>>>(ctx->dsys, ctx->s0, nPairs, order, ctx->pairs, ctx->feasible,
                                                              ctx->slowList.as<int>(), ctx->slowCount.as<int>(),
                                                              ctx->stepCounter.as<unsigned long long>());
        LAUNCH_CHECK();
        }
        CK(cudaMemcpyAsync(&slow, ctx->slowCount.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
        static const bool noSpin = std::getenv("WVA_NO_SPIN") != nullptr;
        while (!noSpin && !ctx->sweep_launched.load(std::memory_order_acquire)) std::this_thread::yield();
        CK(cudaStreamSynchronize(ctx->stream));
    }
    if (slow > 0) {
        // pairs whose chain hit an overflow-rescale branch: re-run with p[] materialised in HBM
        std::vector<int> list((size_t)slow);
        CK(cudaMemcpy(list.data(), ctx->slowList.p, (size_t)slow * 4, cudaMemcpyDeviceToHost));
        std::vector<long long> nAllPairs((size_t)nPairs);
        k_pair_batch<<<(nPairs + 255) / 256, 256, 0, ctx->stream>>>(ctx->dsys, ctx->s0, nPairs, ctx->pairN.as<long long>());
        LAUNCH_CHECK();
        CK(cudaMemcpyAsync(nAllPairs.data(), ctx->pairN.p, (size_t)nPairs * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        std::vector<long long> offs((size_t)slow);
        long long total = 0;
        for (int i = 0; i < slow; ++i) {
            long long N = nAllPairs[(size_t)list[(size_t)i]];
            if (N > (1LL << 32)) return fail(ctx, WVA_EINVAL, "pair needs the materialised path with an unreasonably large batch size");
            offs[(size_t)i] = total;
            total += 11 * N + 1;
        }
        size_t freeB = 0, totB = 0;
        CK(cudaMemGetInfo(&freeB, &totB));
        if ((size_t)total * 8 > freeB / 2) return fail(ctx, WVA_ECUDA, "not enough device memory for the materialised chain path");
        CK(ctx->scratch.ensure((size_t)total * 8));
        CK(ctx->scratchOff.ensure((size_t)slow * 8));
        CK(cudaMemcpyAsync(ctx->scratchOff.p, offs.data(), (size_t)slow * 8, cudaMemcpyHostToDevice, ctx->stream));
        k_pairs_literal<<<(slow + 63) / 64, 64, 0, ctx->stream>>>(ctx->dsys, ctx->s0, ctx->slowList.as<int>(), slow,
                                                                 ctx->scratch.as<double>(), ctx->scratchOff.as<long long>(),
                                                                 ctx->pairs, ctx->feasible, ctx->stepCounter.as<unsigned long long>());
        LAUNCH_CHECK();
        CK(cudaStreamSynchronize(ctx->stream));
    }
    timer.stop();
    ctx->pairs_valid = true;
    ctx->pairs_complete = (ctx->s0 == 0 && ctx->ns == ctx->S);
    ctx->solved = false;
    if (nPairs > 0 && (out || feasible)) {
        const size_t first = (size_t)ctx->s0 * A;
        if (out) CK(download_allocs(ctx, ctx->pairs, first, (size_t)nPairs, out, first));
        if (feasible) CK(cudaMemcpyAsync(feasible + first, ctx->feasible + first, (size_t)nPairs, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return WVA_OK;
}

// device addresses of the pair results (for the host-side NCCL all-gather of limited mode)
int wva_pairs_device(wva_ctx* ctx, wva_alloc_soa* dev, uint8_t** feasible) {
    if (!ctx || !dev) return WVA_EINVAL;
    if (!ctx->pairs_valid) return fail(ctx, WVA_ESTATE, "analyze_pairs has not run");
    dev->acc = ctx->pairs.acc; dev->num_replicas = (int64_t*)ctx->pairs.num_replicas; dev->batch_size = (int64_t*)ctx->pairs.batch_size;
    dev->cost = ctx->pairs.cost; dev->value = ctx->pairs.value; dev->itl = ctx->pairs.itl; dev->ttft = ctx->pairs.ttft;
    dev->rho = ctx->pairs.rho; dev->max_arrv_rate_per_replica = ctx->pairs.max_arrv;
    if (feasible) *feasible = ctx->feasible;
    return WVA_OK;
}
// the host gathered every rank's rows into the device arrays: all S*A records are now valid
int wva_pairs_commit(wva_ctx* ctx) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->pairs_valid) return fail(ctx, WVA_ESTATE, "analyze_pairs has not run");
    CK(cudaSetDevice(ctx->device));
    CK(cudaDeviceSynchronize());       // the caller's collectives may have run on any stream
    ctx->pairs_complete = true;
    return WVA_OK;
}
int wva_set_certified_tails(wva_ctx* ctx, int32_t on) {
    if (!ctx) return WVA_EINVAL;
    ctx->certified = (on & 1) ? 1 : 0;
    // bit 1: always one thread per candidate; bit 2: always one thread per row; bit 3: always one warp per row
    ctx->grid_rows = (on & 2) ? 0 : ((on & 4) ? 2 : ((on & 8) ? 3 : 1));
    // bits 1-3 select one of the round-1 kernels explicitly (and switch the scan kernel off); bit 4 (16): round-1
    // automatic choice (k_grid / k_grid_rows by shard size); bit 5 (32): scan kernel tuned for 3 blocks per SM
    ctx->grid_scan = ((on & (2 | 4 | 8 | 16)) || !(on & 1)) ? 0 : ((on & 32) ? 2 : 1);     // bit 5: k_scan_cert tuned for 2 blocks per SM
    ctx->dsys.cert = ctx->certified;
    return WVA_OK;
}
int wva_pairs_set_pstore(wva_ctx* ctx, int32_t on) {
    if (!ctx) return WVA_EINVAL;
    ctx->pairs_pstore = (on & 1) ? 1 : 0;
    ctx->pairs_smem = (on & 2) ? 0 : 1;        // bit 1: keep the tables in HBM instead of shared memory (tuning/debug)
    ctx->pairs_debug = (on & 4) ? 1 : 0;       // bit 2: record per-pair cycles / rounds (wva_pair_debug)
    return WVA_OK;
}
int wva_pairs_set_warp_max(wva_ctx* ctx, int32_t max_pairs) {
    if (!ctx || max_pairs < 0) return WVA_EINVAL;
    ctx->pairs_warp_max = max_pairs;
    return WVA_OK;
}
int wva_pair_steps(wva_ctx* ctx, uint64_t* steps) {
    if (!ctx || !steps) return WVA_EINVAL;
    if (!ctx->stepCounter.p) { *steps = 0; return WVA_OK; }
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpy(steps, ctx->stepCounter.p, 8, cudaMemcpyDeviceToHost));
    return WVA_OK;
}
int wva_pair_debug(wva_ctx* ctx, uint64_t* out /* 2 per pair of the shard: cycles, (rounds<<32)|rounds with evaluations */, int32_t n_pairs) {
    if (!ctx || !out) return WVA_EINVAL;
    if (!ctx->pairDbg.p || (size_t)n_pairs * 16 > ctx->pairDbg.cap) return fail(ctx, WVA_ESTATE, "no debug record");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpy(out, ctx->pairDbg.p, (size_t)n_pairs * 16, cudaMemcpyDeviceToHost));
    return WVA_OK;
}
// instrumentation of the warp-per-pair kernel: {chain steps, sum of bisection rounds, max rounds, trailing-Analyze misses}
int wva_pair_counters(wva_ctx* ctx, uint64_t out[4]) {
    if (!ctx || !out) return WVA_EINVAL;
    if (!ctx->stepCounter.p) { out[0] = out[1] = out[2] = out[3] = 0; return WVA_OK; }
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpy(out, ctx->stepCounter.p, 32, cudaMemcpyDeviceToHost));
    return WVA_OK;
}

// ---------------------------------------------------------------------------------------------
static int grid_run(wva_ctx* ctx, int r_max, int b_max, bool want_cube, bool want_status, bool fork_join = true) {
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    if (r_max < 1 || r_max > WVA_GRID_MAX_R || b_max < 1 || b_max > WVA_GRID_MAX_B || ctx->A > WVA_GRID_MAX_A)
        return fail(ctx, WVA_EINVAL, "grid extents out of range (A<=256, r_max<=1024, b_max<=8192)");
    CK(cudaSetDevice(ctx->device));
    ctx->gpairs_valid = ctx->gpairs_complete = false;
    const int ns = ctx->ns, A = ctx->A;
    const size_t nPairs = (size_t)ns * A;
    const size_t perPair = (size_t)r_max * (size_t)b_max;
    const size_t nCand = nPairs * perPair;
    CK(ctx->keys.ensure((size_t)(ns ? ns : 1) * 8));
    CK(ctx->bestDev.ensure((size_t)(ns ? ns : 1) * sizeof(wva_grid_best)));
    CK(ctx->counters.ensure(3 * 8));
    CK(ctx->gridSlowCount.ensure(8));                 // [0] literal-path count, [1] deferred count
    CK(ctx->heavyHist.ensure(2 * 256 * 4));
    if (want_cube) {
        if (nCand * sizeof(wva_metrics) > ctx->cube.cap) {
            size_t freeB = 0, totB = 0;
            CK(cudaMemGetInfo(&freeB, &totB));
            if (nCand * sizeof(wva_metrics) > freeB - (freeB >> 3)) return fail(ctx, WVA_ECUDA, "metric cube does not fit in device memory");
        }
        CK(ctx->cube.ensure(nCand * sizeof(wva_metrics)));
    }
    if (want_status) CK(ctx->status.ensure(nCand ? nCand : 1));

    // The sweep runs over slices of servers so that the published service-rate tables (16 B per
    // pair and batch size) stay within ~1 GB.
    int srvPerSlice = ns;
    {
        const size_t tabPerServer = (size_t)A * b_max * sizeof(double2);
        size_t maxSrv = ((size_t)1 << 30) / (tabPerServer ? tabPerServer : 1);
        if (maxSrv < 1) maxSrv = 1;
        if ((size_t)srvPerSlice > maxSrv) srvPerSlice = (int)maxSrv;
        if (srvPerSlice < 1) srvPerSlice = 1;
    }
    const size_t slicePairsMax = (size_t)srvPerSlice * A;
    CK(ctx->pairTab.ensure(slicePairsMax * (size_t)b_max * sizeof(double2)));

    GridParams gp;
    gp.r_max = r_max; gp.b_max = b_max;
    int n_rchunks = 1;
    if (slicePairsMax > 0 && slicePairsMax < 2368) {
        n_rchunks = (int)((2368 + slicePairsMax - 1) / slicePairsMax);
        if (n_rchunks > r_max) n_rchunks = r_max;
    }
    gp.r_chunk = (r_max + n_rchunks - 1) / n_rchunks;
    gp.n_rchunks = (r_max + gp.r_chunk - 1) / gp.r_chunk;
    gp.s0 = ctx->s0; gp.ns = ns;
    gp.cube = want_cube ? ctx->cube.as<wva_metrics>() : nullptr;
    gp.status = want_status ? ctx->status.as<unsigned char>() : nullptr;
    gp.keys = ctx->keys.as<unsigned long long>();
    gp.counters = ctx->counters.as<unsigned long long>();
    gp.pair_keys = nullptr; gp.pair_rec = DevAllocs{}; gp.pair_feasible = nullptr;
    if (ctx->grid_pair_winners) {
        const size_t nAll = (size_t)ctx->S * A;
        CK(carve_allocs(ctx->gridPairBuf, nAll ? nAll : 1, ctx->gridPairs, &ctx->gridFeasible, nullptr));
        CK(ctx->gridPairKeys.ensure((nPairs ? nPairs : 1) * 8));
        gp.pair_keys = ctx->gridPairKeys.as<unsigned long long>(); gp.pair_rec = ctx->gridPairs; gp.pair_feasible = ctx->gridFeasible;
    }
    gp.pair_tab = ctx->pairTab.as<double2>();
    // with certified tails almost no chain runs a long exact tail any more: finishing the few that do
    // inside the sweep kernel is cheaper than a second kernel + host round trip (cap < 0 = automatic)
    gp.tail_cap = ctx->grid_tail_cap >= 0 ? ctx->grid_tail_cap : (ctx->certified ? 0 : 192);

    gp.slow_count = ctx->gridSlowCount.as<int>();
    gp.heavy_count = ctx->gridSlowCount.as<int>() + 1;

    const size_t sliceCandMax = slicePairsMax * perPair;
    // deferred-chain list: at most one entry per candidate of a slice, capped at 16M entries (the
    // sweep kernel finishes a chain itself when the list is full)
    size_t heavy_cap_sz = sliceCandMax < (size_t)(16u << 20) ? sliceCandMax : (size_t)(16u << 20);
    if (heavy_cap_sz < 1) heavy_cap_sz = 1;
    const int heavy_cap = (int)heavy_cap_sz;
    CK(ctx->heavyList.ensure(heavy_cap_sz * 8));
    CK(ctx->heavyCost.ensure(heavy_cap_sz * 4));
    CK(ctx->heavyOrder.ensure(heavy_cap_sz * 4));
    gp.heavy_list = ctx->heavyList.as<unsigned long long>(); gp.heavy_cost = ctx->heavyCost.as<float>();
    gp.heavy_cap = heavy_cap;
    int slow_cap = 1 << 16;
    CK(ctx->gridSlow.ensure((size_t)slow_cap * 8));

    // certified tails on: one thread per (server, accelerator, replicas) row with a shared ramp (k_grid_rows);
    // off: one thread per candidate (k_grid)
    // (the row kernel needs >= 32 K rows to fill the machine: each thread walks its row's batch sizes serially)
    // Shards with few rows split every pair over n_bseg blocks of b_seg batch sizes (>= 32 each) so that
    // about 64 K threads exist; below 16 K threads the per-candidate kernel is used.
    gp.n_bseg = 1; gp.b_seg = b_max;
    {
        const size_t rows = slicePairsMax * (size_t)r_max;
        if (rows > 0 && rows < 65536) {
            int want = (int)((65536 + rows - 1) / rows);
            const int maxSeg = b_max / 32 > 0 ? b_max / 32 : 1;
            if (want > maxSeg) want = maxSeg;
            gp.b_seg = (b_max + want - 1) / want;
            gp.n_bseg = (b_max + gp.b_seg - 1) / gp.b_seg;
        }
    }
    // (measured on config 2, 8 192 rows x 8 segments: row kernel 0.47 ms + 0.45 ms for the 356 candidates whose
    // certificate is ambiguous -- the exact chain of one b = 512 candidate is 11 264 dependent steps -- against
    // 0.55 ms for the per-candidate kernel, which finishes such chains inline while other warps work; so
    // segmentation is used only when asked for)
    const bool scanMode = ctx->certified && ctx->grid_scan != 0;
    const bool rowsMode = !scanMode && ctx->certified && ctx->grid_rows && ctx->grid_rows != 3 &&
                          (ctx->grid_rows == 2 || slicePairsMax * (size_t)r_max >= 32768);
    if (!(rowsMode && ctx->grid_rows == 2)) { gp.n_bseg = 1; gp.b_seg = b_max; }
    // one warp per row (k_grid_wrow), 8 rows per block: only when asked for.  Measured on config 2 (8 192 rows):
    // 0.33 ms for the rows + 0.38 ms for the 356 candidates whose certificate is ambiguous (k_grid_list_warp;
    // the phase lasts as long as its slowest exact chain) against 0.67 ms for k_grid on the same box, which
    // runs those chains inline while other warps work.
    const bool wrowMode = !scanMode && ctx->certified && !rowsMode && ctx->grid_rows == 3 &&
                          (size_t)b_max * 20 + 16 + (size_t)(WVA_GRID_THREADS / 32) * (WVA_WX_CP + 1 + 1024) * 8 <= 200 * 1024;
    if (wrowMode) {
        gp.r_chunk = WVA_GRID_THREADS / 32;
        gp.n_rchunks = (r_max + gp.r_chunk - 1) / gp.r_chunk;
    }
    if (scanMode) {
        // one warp per row, 8 warps per block: a pair's rows are split over blocks only while the shard has fewer
        // than ~4 blocks per SM of them (each block rebuilds the pair's 10 KB table)
        int chunks = 1;
        if (slicePairsMax > 0 && slicePairsMax < 592) chunks = (int)((592 + slicePairsMax - 1) / slicePairsMax);
        const int maxChunks = (r_max + WVA_SCAN_WARPS - 1) / WVA_SCAN_WARPS;
        if (chunks > maxChunks) chunks = maxChunks;
        const int minChunks = (r_max + WVA_SCAN_MAXROWS - 1) / WVA_SCAN_MAXROWS;     // a block holds the exact-stop records of <= 64 rows
        if (chunks < minChunks) chunks = minChunks;
        gp.r_chunk = (r_max + chunks - 1) / chunks;
        gp.r_chunk = (gp.r_chunk + WVA_SCAN_WARPS - 1) / WVA_SCAN_WARPS * WVA_SCAN_WARPS;
        gp.n_rchunks = (r_max + gp.r_chunk - 1) / gp.r_chunk;
    }
    const size_t smem = (size_t)b_max * 20;
    if (smem > 48 * 1024) {
        CK(cudaFuncSetAttribute(k_grid, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(cudaFuncSetAttribute(k_grid_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(cudaFuncSetAttribute(k_scan_prep, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(cudaFuncSetAttribute(k_scan_cert<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(cudaFuncSetAttribute(k_scan_cert<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    CK(cudaFuncSetAttribute(k_grid_list_own, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    // k_grid_wrow: the table, then per warp the checkpoints and the quotient buffer of warp_exact
    const size_t smemW = align_up(smem, 16) + (size_t)(WVA_GRID_THREADS / 32) * (WVA_WX_CP + 1 + 1024) * 8;
    if (smemW > 48 * 1024) CK(cudaFuncSetAttribute(k_grid_wrow, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemW));
    if (slicePairsMax * (size_t)gp.n_rchunks > 0x7fffffffULL) return fail(ctx, WVA_EINVAL, "too many grid blocks");
    {
        const size_t perPairBlocks = (size_t)(gp.n_rchunks > gp.n_bseg ? gp.n_rchunks : gp.n_bseg);
        CK(ctx->blockSlot.ensure((slicePairsMax * perPairBlocks * (scanMode ? 2 : 1) + 1) * sizeof(GridSlot)));
        if (scanMode) CK(ctx->rowInfo.ensure((slicePairsMax * (size_t)r_max + 1) * sizeof(ScanRow)));
        if (scanMode) CK(ctx->rateTab.ensure((slicePairsMax * (size_t)b_max + 1) * sizeof(float2)));
    }
    gp.row_info = scanMode ? ctx->rowInfo.as<ScanRow>() : nullptr;
    gp.rate_tab = scanMode ? ctx->rateTab.as<float2>() : nullptr;
    gp.block_slot = ctx->blockSlot.as<GridSlot>();
    const long long stride = 11LL * b_max + 1;

    // order the sweep after whatever the main stream has queued (the system upload), run it on its own stream
    if (fork_join) {
        CK(cudaEventRecord(ctx->evFork, ctx->stream));
        CK(cudaStreamWaitEvent(ctx->gstream, ctx->evFork, 0));
    }
    PhaseTimer timer(ctx, WVA_PHASE_GRID, ctx->gstream, ctx->evg0, ctx->evg1);
    ctx->phase_usec[WVA_PHASE_GRID_KERNEL] = 0; ctx->phase_usec[WVA_PHASE_GRID_HEAVY] = 0;
    ctx->last_heavy = 0; ctx->last_slow = 0; ctx->last_heavy_slice = 0;
    CK(cudaMemsetAsync(ctx->keys.p, 0xff, (size_t)(ns ? ns : 1) * 8, ctx->gstream));
    CK(cudaMemsetAsync(ctx->counters.p, 0, 3 * 8, ctx->gstream));
    if (ns > 0) {
        k_grid_best_init<<<(ns + 255) / 256, 256, 0, ctx->gstream>>>(ns, ctx->bestDev.as<wva_grid_best>(), gp, A);
        LAUNCH_CHECK();
    }
    for (int sBeg = 0; sBeg < ns; sBeg += srvPerSlice) {
        const int sCnt = (ns - sBeg) < srvPerSlice ? (ns - sBeg) : srvPerSlice;
        const size_t slicePairs = (size_t)sCnt * A;
        const size_t nBlocks = rowsMode ? slicePairs * (size_t)gp.n_bseg : slicePairs * (size_t)gp.n_rchunks;
        gp.pair_base = sBeg * A;
        int counts[2] = {0, 0};
        int slow = 0, heavy = 0;
        bool leanPending = false;
        // Long deferred lists (as seen in the previous call / slice): the sweep does not stop at the host between its kernels.
        // The exact-chain kernel reads the list length from device memory and owns a few SMs (k_grid_list_own), k_scan_lean
        // gets the others.  The list's slots are sized from the previous length; a list that outgrows them redoes the slice
        // the stop-and-go way (keys only ever decrease towards the true minimum: safe).
        bool fused = scanMode && ctx->grid_fused && ctx->heavy_hint > 4096;
        for (int attempt = 0; attempt < 3; ++attempt) {
            gp.slow_list = ctx->gridSlow.as<unsigned long long>(); gp.slow_cap = slow_cap;
            CK(cudaMemsetAsync(ctx->gridSlowCount.p, 0, 8, ctx->gstream));
            CK(cudaEventRecord(ctx->evk0, ctx->gstream));
            if (fused) {
                size_t fusedCap = 2 * (size_t)ctx->heavy_hint + 65536;
                if (fusedCap > (size_t)heavy_cap) fusedCap = (size_t)heavy_cap;
                CK(ctx->listSlot.ensure((fusedCap + (size_t)slow_cap + 1) * sizeof(GridSlot)));
                gp.list_slot = ctx->listSlot.as<GridSlot>();
                k_scan_prep<<<(unsigned)nBlocks, WVA_SCAN_MAXROWS, smem, ctx->gstream>>>(ctx->dsys, gp);
                LAUNCH_CHECK();
                if (ctx->grid_scan == 2) k_scan_cert<2><<<(unsigned)nBlocks, WVA_SCAN_WARPS * 32, smem, ctx->gstream>>>(ctx->dsys, gp);
                else k_scan_cert<3><<<(unsigned)nBlocks, WVA_SCAN_WARPS * 32, smem, ctx->gstream>>>(ctx->dsys, gp);
                LAUNCH_CHECK();
                ctx->sweep_launched.store(true, std::memory_order_release);
                CK(cudaEventRecord(ctx->evk1, ctx->gstream));
                CK(cudaEventRecord(ctx->evh0, ctx->gstream));
                int* hist = ctx->heavyHist.as<int>();
                CK(cudaMemsetAsync(hist, 0, 256 * 4, ctx->gstream));
                k_heavy_hist_dev<<<296, 256, 0, ctx->gstream>>>(gp.heavy_cost, gp.heavy_count, (int)fusedCap, hist);
                LAUNCH_CHECK();
                k_heavy_prefix<<<1, 256, 0, ctx->gstream>>>(hist);
                LAUNCH_CHECK();
                k_heavy_scatter_dev<<<296, 256, 0, ctx->gstream>>>(gp.heavy_cost, gp.heavy_count, (int)fusedCap, hist, ctx->heavyOrder.as<int>());
                LAUNCH_CHECK();
                // both halves become runnable here; this stream has the higher priority, so the chain kernel's blocks are placed first
                CK(cudaEventRecord(ctx->evPrep, ctx->gstream));
                CK(cudaStreamWaitEvent(ctx->gstream2, ctx->evPrep, 0));
                int nOwn = (ctx->heavy_hint + 511) / 512;
                nOwn = nOwn < 8 ? 8 : (nOwn > 32 ? 32 : nOwn);
                k_grid_list_own<<<nOwn, 512, 200 * 1024, ctx->gstream>>>(ctx->dsys, gp, gp.heavy_list, ctx->heavyOrder.as<int>(), gp.heavy_count, (int)fusedCap);
                LAUNCH_CHECK();
                CK(cudaEventRecord(ctx->evh1, ctx->gstream));
                k_scan_lean<<<(unsigned)nBlocks, WVA_SCAN_WARPS * 32, 46 * 1024, ctx->gstream2>>>(ctx->dsys, gp);
                LAUNCH_CHECK();
                CK(cudaEventRecord(ctx->evLean, ctx->gstream2));
                leanPending = true;
                CK(cudaMemcpyAsync(counts, ctx->gridSlowCount.p, 8, cudaMemcpyDeviceToHost, ctx->gstream));
                CK(cudaStreamSynchronize(ctx->gstream));
                float kms = 0.0f, hms = 0.0f;
                CK(cudaEventElapsedTime(&kms, ctx->evk0, ctx->evk1));
                CK(cudaEventElapsedTime(&hms, ctx->evh0, ctx->evh1));
                ctx->phase_usec[WVA_PHASE_GRID_KERNEL] += (int64_t)(kms * 1000.0f + 0.5f);
                ctx->phase_usec[WVA_PHASE_GRID_HEAVY] += (int64_t)(hms * 1000.0f + 0.5f);
                slow = counts[0];
                if ((size_t)counts[1] > fusedCap) {                    // the list outgrew its slots: once more, stop-and-go
                    ctx->heavy_hint = 0; fused = false;
                    CK(cudaStreamWaitEvent(ctx->gstream, ctx->evLean, 0));
                    continue;
                }
                heavy = counts[1];
                if (slow <= slow_cap) break;
                slow_cap = slow;
                CK(ctx->gridSlow.ensure((size_t)slow_cap * 8));
                CK(cudaStreamWaitEvent(ctx->gstream, ctx->evLean, 0));
                continue;
            }
            if (scanMode) {
                // exact stop of every row, then the two halves of the sweep (before / after the stop)
                k_scan_prep<<<(unsigned)nBlocks, WVA_SCAN_MAXROWS, smem, ctx->gstream>>>(ctx->dsys, gp);
                LAUNCH_CHECK();
                // k_scan_cert first (it owns the register file: 128 registers x 512 threads per SM), then k_scan_lean on a second
                // stream BESIDE the exact-chain kernels that follow on this one: those are a few hundred latency-bound warps,
                // k_scan_lean is bound by the cube's HBM write.  (k_scan_lean asks for 46 KB of shared memory it does not use so
                // that at most 4 of its blocks sit on an SM and a block of the exact-chain kernel still finds registers there.)
                if (ctx->grid_scan == 2) k_scan_cert<2><<<(unsigned)nBlocks, WVA_SCAN_WARPS * 32, smem, ctx->gstream>>>(ctx->dsys, gp);
                else k_scan_cert<3><<<(unsigned)nBlocks, WVA_SCAN_WARPS * 32, smem, ctx->gstream>>>(ctx->dsys, gp);
                LAUNCH_CHECK();
                CK(cudaEventRecord(ctx->evPrep, ctx->gstream));
                CK(cudaStreamWaitEvent(ctx->gstream2, ctx->evPrep, 0));
                k_scan_lean<<<(unsigned)nBlocks, WVA_SCAN_WARPS * 32, 46 * 1024, ctx->gstream2>>>(ctx->dsys, gp);
                CK(cudaEventRecord(ctx->evLean, ctx->gstream2));
                leanPending = true;
            }
            else if (rowsMode) k_grid_rows<<<(unsigned)nBlocks, WVA_ROWS_THREADS, smem, ctx->gstream>>>(ctx->dsys, gp);
            else if (wrowMode) k_grid_wrow<<<(unsigned)nBlocks, WVA_GRID_THREADS, smemW, ctx->gstream>>>(ctx->dsys, gp);
            else k_grid<<<(unsigned)nBlocks, WVA_GRID_THREADS, smem, ctx->gstream>>>(ctx->dsys, gp);
            LAUNCH_CHECK();
            ctx->sweep_launched.store(true, std::memory_order_release);
            CK(cudaEventRecord(ctx->evk1, ctx->gstream));
            CK(cudaMemcpyAsync(counts, ctx->gridSlowCount.p, 8, cudaMemcpyDeviceToHost, ctx->gstream));
            CK(cudaStreamSynchronize(ctx->gstream));
            slow = counts[0]; heavy = counts[1] < heavy_cap ? counts[1] : heavy_cap;
            {
                float kms = 0.0f;
                CK(cudaEventElapsedTime(&kms, ctx->evk0, ctx->evk1));
                ctx->phase_usec[WVA_PHASE_GRID_KERNEL] += (int64_t)(kms * 1000.0f + 0.5f);
            }
            CK(ctx->listSlot.ensure(((size_t)heavy + (size_t)(slow > slow_cap ? slow : slow_cap) + 1) * sizeof(GridSlot)));
            gp.list_slot = ctx->listSlot.as<GridSlot>();
            if (heavy > 0) {
                // long chains: order by estimated length (longest first), one thread per chain
                int* hist = ctx->heavyHist.as<int>();
                CK(cudaEventRecord(ctx->evh0, ctx->gstream));
                const int* order = nullptr;
                if (heavy >= 4096) {     // a short list fits in one wave: ordering it buys nothing.  Longer ones: the lanes of a warp
                                         // should hold chains of similar length (the warp lasts as long as its longest chain, and
                                         // solve_uni enters a block run only when every lane can): measured -13 % on the phase
                                         // at config 4 (127 k chains), -3 % at config 3 (13 k)
                    CK(cudaMemsetAsync(hist, 0, 256 * 4, ctx->gstream));
                    k_heavy_hist<<<(heavy + 255) / 256, 256, 0, ctx->gstream>>>(gp.heavy_cost, heavy, hist);
                    LAUNCH_CHECK();
                    k_heavy_prefix<<<1, 256, 0, ctx->gstream>>>(hist);
                    LAUNCH_CHECK();
                    k_heavy_scatter<<<(heavy + 255) / 256, 256, 0, ctx->gstream>>>(gp.heavy_cost, heavy, hist, ctx->heavyOrder.as<int>());
                    LAUNCH_CHECK();
                    order = ctx->heavyOrder.as<int>();
                }
                // few chains: the phase lasts as long as ONE exact chain -- one warp per chain (cooperative pass 2);
                // many: one thread per chain, ordered by length
                const size_t smemLW = (size_t)WVA_LISTW_WARPS * (2 * (size_t)b_max + WVA_WX_CP + 1 + 1024) * 8;
                if (heavy <= 4096 && smemLW <= 200 * 1024 && ctx->grid_list_warp) {
                    if (smemLW > 48 * 1024)
                        CK(cudaFuncSetAttribute(k_grid_list_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemLW));
                    k_grid_list_warp<<<(heavy + WVA_LISTW_WARPS - 1) / WVA_LISTW_WARPS, WVA_LISTW_WARPS * 32, smemLW, ctx->gstream>>>(
                        ctx->dsys, gp, gp.heavy_list, heavy, 0);
                } else {
                    k_grid_list<<<(heavy + 127) / 128, 128, 0, ctx->gstream>>>(ctx->dsys, gp, gp.heavy_list, order, heavy, nullptr, 0, 0);
                }
                LAUNCH_CHECK();
                CK(cudaEventRecord(ctx->evh1, ctx->gstream));
                CK(cudaMemcpyAsync(counts, ctx->gridSlowCount.p, 4, cudaMemcpyDeviceToHost, ctx->gstream));
                CK(cudaStreamSynchronize(ctx->gstream));
                slow = counts[0];
                float hms = 0.0f;
                CK(cudaEventElapsedTime(&hms, ctx->evh0, ctx->evh1));
                ctx->phase_usec[WVA_PHASE_GRID_HEAVY] += (int64_t)(hms * 1000.0f + 0.5f);
            }
            if (slow <= slow_cap) break;
            slow_cap = slow;                          // rare: more literal-path candidates than the list holds
            CK(ctx->gridSlow.ensure((size_t)slow_cap * 8));
            // keys only ever decrease towards the true minimum: redoing the slice is safe (the work
            // counters then count the slice twice)
        }
        ctx->last_heavy += heavy; ctx->last_slow += slow; ctx->last_heavy_slice = heavy; ctx->heavy_hint = heavy; ctx->last_fused = fused ? 1 : 0;
        int listSlots = heavy;
        if (slow > 0) {
            size_t freeB = 0, totB = 0;
            CK(cudaMemGetInfo(&freeB, &totB));
            // process the literal list in pieces that fit in memory
            size_t per = (size_t)stride * 8;
            size_t maxItems = (freeB / 2) / per;
            if (maxItems == 0) return fail(ctx, WVA_ECUDA, "not enough device memory for the materialised chain path");
            if (maxItems > (size_t)slow) maxItems = (size_t)slow;
            CK(ctx->gscratch.ensure(maxItems * per));
            for (size_t done = 0; done < (size_t)slow; done += maxItems) {
                int n = (int)(((size_t)slow - done) < maxItems ? ((size_t)slow - done) : maxItems);
                k_grid_list<<<(n + 127) / 128, 128, 0, ctx->gstream>>>(ctx->dsys, gp, ctx->gridSlow.as<unsigned long long>() + done, nullptr,
                                                                   n, ctx->gscratch.as<double>(), stride, heavy + (int)done);
                LAUNCH_CHECK();
            }
            listSlots += slow;
        }
        if (leanPending) CK(cudaStreamWaitEvent(ctx->gstream, ctx->evLean, 0));     // join k_scan_lean
        // winners of the slice: the slot that carries a server's minimum key writes its record
        if (nBlocks > 0) {
            const size_t nSlots = scanMode ? 2 * nBlocks : nBlocks;       // k_scan_cert and k_scan_lean each publish one slot per block
            k_grid_claim<<<(unsigned)((nSlots + 255) / 256), 256, 0, ctx->gstream>>>(ctx->dsys, gp, gp.block_slot, (int)nSlots, ctx->bestDev.as<wva_grid_best>());
            LAUNCH_CHECK();
        }
        if (listSlots > 0) {
            k_grid_claim<<<(listSlots + 255) / 256, 256, 0, ctx->gstream>>>(ctx->dsys, gp, gp.list_slot, listSlots, ctx->bestDev.as<wva_grid_best>());
            LAUNCH_CHECK();
        }
    }
    CK(cudaMemcpyAsync(ctx->grid_counters, ctx->counters.p, 3 * 8, cudaMemcpyDeviceToHost, ctx->gstream));
    CK(cudaStreamSynchronize(ctx->gstream));
    timer.stop();
    // later work on the main stream sees the sweep's results
    if (fork_join) {
        CK(cudaEventRecord(ctx->evJoin, ctx->gstream));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->evJoin, 0));
    }
    ctx->grid_r = r_max; ctx->grid_b = b_max; ctx->grid_valid = true;
    ctx->gpairs_valid = ctx->grid_pair_winners != 0;
    ctx->gpairs_complete = ctx->gpairs_valid && ctx->s0 == 0 && ctx->ns == ctx->S;
    return WVA_OK;
}

int wva_analyze_grid_device(wva_ctx* ctx, int32_t r_max, int32_t b_max, int32_t want_cube) {
    if (!ctx) return WVA_EINVAL;
    return grid_run(ctx, r_max, b_max, want_cube != 0, want_cube != 0);
}

int wva_grid_fetch(wva_ctx* ctx, wva_grid_best* best) {
    if (!ctx || !best) return WVA_EINVAL;
    if (!ctx->grid_valid) return fail(ctx, WVA_ESTATE, "no grid sweep has run");
    CK(cudaSetDevice(ctx->device));
    if (ctx->ns > 0) {
        CK(cudaMemcpyAsync(best, ctx->bestDev.p, (size_t)ctx->ns * sizeof(wva_grid_best), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return WVA_OK;
}

// Analyze, both halves at once: Server.Calculate for every pair (main stream) and the candidate
// sweep (its own stream, driven by a helper host thread) are independent and overlap on the device.
// Results stay in HBM; fetch them with wva_pairs_fetch / wva_grid_fetch.
int wva_analyze(wva_ctx* ctx, int32_t r_max, int32_t b_max, int32_t want_cube) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    CK(cudaSetDevice(ctx->device));
    // fork: the sweep starts after what the main stream holds now (the upload), not after the pair kernels
    CK(cudaEventRecord(ctx->evFork, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->gstream, ctx->evFork, 0));
    int rcGrid = WVA_OK;
    const int dev = ctx->device;
    if (!ctx->worker.th.joinable()) ctx->worker.start();
    static const bool timeline = std::getenv("WVA_TIMELINE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = now();
    double tg0 = 0, tg1 = 0;
    ctx->sweep_launched.store(false, std::memory_order_release);
    ctx->worker.submit([&] {
        tg0 = now(); cudaSetDevice(dev);
        rcGrid = grid_run(ctx, r_max, b_max, want_cube != 0, want_cube != 0, false);
        ctx->sweep_launched.store(true, std::memory_order_release);      // also on the error paths
        tg1 = now();
    });
    // The sweep's first kernels go to the device BEFORE the pair kernel.  k_pairs_warp takes every register of every SM
    // (4 blocks x 128 threads x 128 registers) for 3-4 waves: launched first, it kept the sweep waiting until its last wave
    // (analyze = pairs + sweep, 5.7 ms at config 3); launched behind k_scan_prep / k_scan_cert it shares the SMs with them
    // from the start (4.2 ms).  Costs the calling thread the ~30 us the sweep thread needs to get there.
    static const bool pairsFirst = std::getenv("WVA_PAIRS_FIRST") != nullptr;
    while (!pairsFirst && !ctx->sweep_launched.load(std::memory_order_acquire)) std::this_thread::yield();
    const double t1 = now();
    int rcPairs = wva_analyze_pairs(ctx, nullptr, nullptr);
    const double t2 = now();
    ctx->worker.wait();
    const double t3 = now();
    if (timeline)
        fprintf(stderr, "analyze: submit %.0f us, pairs call %.0f us, wait for sweep %.0f us | sweep thread started at +%.0f, ran %.0f us\n",
                t1 - t0, t2 - t1, t3 - t2, tg0 - t0, tg1 - tg0);
    // join: later work on the main stream sees the sweep's results
    CK(cudaEventRecord(ctx->evJoin, ctx->gstream));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->evJoin, 0));
    return rcPairs != WVA_OK ? rcPairs : rcGrid;
}

int wva_pairs_fetch(wva_ctx* ctx, wva_alloc_soa* out, uint8_t* feasible) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->pairs_valid) return fail(ctx, WVA_ESTATE, "analyze_pairs has not run (or a limited solve consumed its records)");
    CK(cudaSetDevice(ctx->device));
    const size_t nPairs = (size_t)ctx->ns * ctx->A, first = (size_t)ctx->s0 * ctx->A;
    if (nPairs > 0) {
        if (out) CK(download_allocs(ctx, ctx->pairs, first, nPairs, out, first));
        if (feasible) CK(cudaMemcpyAsync(feasible + first, ctx->feasible + first, nPairs, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return WVA_OK;
}

int wva_analyze_grid(wva_ctx* ctx, int32_t r_max, int32_t b_max, wva_grid_best* best, wva_metrics* cube, uint8_t* status) {
    if (!ctx) return WVA_EINVAL;
    int rc = grid_run(ctx, r_max, b_max, cube != nullptr, status != nullptr);
    if (rc != WVA_OK) return rc;
    const size_t nCand = (size_t)ctx->ns * ctx->A * (size_t)r_max * (size_t)b_max;
    if (best && ctx->ns > 0) CK(cudaMemcpyAsync(best, ctx->bestDev.p, (size_t)ctx->ns * sizeof(wva_grid_best), cudaMemcpyDeviceToHost, ctx->stream));
    if (cube && nCand) CK(cudaMemcpyAsync(cube, ctx->cube.p, nCand * sizeof(wva_metrics), cudaMemcpyDeviceToHost, ctx->stream));
    if (status && nCand) CK(cudaMemcpyAsync(status, ctx->status.p, nCand, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return WVA_OK;
}

int wva_grid_set_tail_cap(wva_ctx* ctx, int32_t tail_cap) {
    if (!ctx) return WVA_EINVAL;
    ctx->grid_tail_cap = tail_cap;
    return WVA_OK;
}
int wva_grid_set_fused(wva_ctx* ctx, int32_t on) {
    if (!ctx) return WVA_EINVAL;
    ctx->grid_fused = on ? 1 : 0;
    return WVA_OK;
}
int wva_grid_last_fused(const wva_ctx* ctx) { return ctx ? ctx->last_fused : WVA_EINVAL; }
int wva_grid_set_pair_winners(wva_ctx* ctx, int32_t on) {
    if (!ctx) return WVA_EINVAL;
    ctx->grid_pair_winners = on ? 1 : 0;
    return WVA_OK;
}
int wva_grid_pairs_fetch(wva_ctx* ctx, wva_alloc_soa* out, uint8_t* feasible) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->gpairs_valid) return fail(ctx, WVA_ESTATE, "no valid sweep winners per pair (wva_grid_set_pair_winners off, no sweep since, or consumed by a limited solve)");
    CK(cudaSetDevice(ctx->device));
    const size_t nPairs = (size_t)ctx->ns * ctx->A, first = (size_t)ctx->s0 * ctx->A;
    if (nPairs > 0) {
        if (out) CK(download_allocs(ctx, ctx->gridPairs, first, nPairs, out, first));
        if (feasible) CK(cudaMemcpyAsync(feasible + first, ctx->gridFeasible + first, nPairs, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return WVA_OK;
}
int wva_grid_list_sizes(const wva_ctx* ctx, int32_t* deferred, int32_t* literal) {
    if (!ctx) return WVA_EINVAL;
    if (deferred) *deferred = ctx->last_heavy;
    if (literal) *literal = ctx->last_slow;
    return WVA_OK;
}
int wva_grid_deferred_fetch(wva_ctx* ctx, uint64_t* ids, int32_t cap, int32_t* n) {
    if (!ctx || !n || cap < 0 || (cap > 0 && !ids)) return WVA_EINVAL;
    if (!ctx->grid_valid) return fail(ctx, WVA_ESTATE, "no grid sweep has run");
    *n = ctx->last_heavy_slice;
    const int k = ctx->last_heavy_slice < cap ? ctx->last_heavy_slice : cap;
    if (k > 0) {
        CK(cudaSetDevice(ctx->device));
        CK(cudaMemcpy(ids, ctx->heavyList.p, (size_t)k * 8, cudaMemcpyDeviceToHost));
    }
    return WVA_OK;
}
int wva_grid_counters(const wva_ctx* ctx, uint64_t* steps_executed, uint64_t* steps_algorithmic, uint64_t* candidates_ok) {
    if (!ctx) return WVA_EINVAL;
    if (steps_executed) *steps_executed = ctx->grid_counters[0];
    if (steps_algorithmic) *steps_algorithmic = ctx->grid_counters[1];
    if (candidates_ok) *candidates_ok = ctx->grid_counters[2];
    return WVA_OK;
}

// ---------------------------------------------------------------------------------------------
}  // extern "C"

// Solver.Solve over one candidate record set (S*A records + feasible flags): the pair records of
// wva_analyze_pairs (wva_solve) or the sweep's per-pair winners (wva_solve_grid).  `valid` / `complete` are the
// set's state flags: a limited solve gathers missing rows (communicator attached) and consumes the set.
static int solve_records(wva_ctx* ctx, const wva_optimizer_spec* spec, int32_t* chosen_acc, wva_alloc_soa* chosen,
                         const DevAllocs& recs, unsigned char* feasible, bool& valid, bool& complete, const char* incomplete_msg) {
    CK(cudaSetDevice(ctx->device));
    const int S = ctx->S, A = ctx->A, T = ctx->T;
    CK(carve_allocs(ctx->chosenBuf, (size_t)(S ? S : 1), ctx->chosen, nullptr, &ctx->chosen_acc));
    PhaseTimer timer(ctx, WVA_PHASE_SOLVE, ctx->stream, ctx->evS0, ctx->evS1);
    ctx->pendS = false;
    int first = 0, count = S;
    if (spec->unlimited) {
        first = ctx->s0; count = ctx->ns;          // separable: a rank solves its own servers
        if (count > 0) {
            k_solve_unlimited<<<(count + 127) / 128, 128, 0, ctx->stream>>>(ctx->dsys, first, count, recs, feasible,
                                                                          ctx->chosen_acc, ctx->chosen, 0, 0);
            LAUNCH_CHECK();
        }
    } else {
        if (!complete && ctx->comm) {
            int rc = comm_gather_pairs(ctx, recs, feasible, complete);
            if (rc != WVA_OK) return rc;
        }
        if (!complete) return fail(ctx, WVA_ESTATE, incomplete_msg);
        // carve greedy buffers
        if (T > 256) return fail(ctx, WVA_EINVAL, "the device greedy solver holds at most 256 accelerator types");
        if ((unsigned long long)(S ? S : 1) * (unsigned long long)A >= (1ull << 31))
            return fail(ctx, WVA_EINVAL, "servers x accelerators must stay below 2^31 for the greedy solver");
        size_t off = 0;
        auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
        const size_t nS = (size_t)(S ? S : 1);
        const size_t nSA = nS * A;
        size_t o_order = take(nSA * 4), o_cand = take(nSA * sizeof(GreedyCand)), o_upr = take(nSA * 8), o_rep = take(nSA * 8), o_ct = take(nSA * 4),
               o_n = take(nS * 4), o_gs = take(104 * 4), o_gi = take(nS * 4), o_un = take(nS * 4), o_ha = take(nS * 8),
               o_hb = take(nS * 8), o_hs = take(nS * 4), o_tk = take(nS * sizeof(GreedyTicket)), o_li = take(nS * 4),
               o_nan = take(8), o_stats = take(32), o_key = take(nS * 4);
        // ranked queue: states sorted by their fixed key (see k_greedy_solve_ranked)
        size_t n2 = GREEDY_TILE;
        while (n2 < nSA) n2 <<= 1;
        // static-order scan (wva_greedy_scan.cuh): the default; shared memory holds one bit per server
        const size_t doneBytes = align_up((nS + 31) / 32 * 4, 16);
        const bool scannable = nSA < (1u << 24) && A <= 32 && doneBytes + 4096 <= (size_t)kGreedySmem && ctx->greedy_ranked >= 2;
        const bool rankable = !scannable && nSA < (1u << 24) && greedy_bitmap_bytes(nSA, nullptr, nullptr, nullptr) + 4096 <= (size_t)kGreedySmem &&
                              ctx->greedy_ranked >= 1;
        size_t o_ka = 0, o_kb = 0, o_ks = 0, o_pos = 0, o_sn = 0, o_rec = 0, o_np = 0, o_ge = 0, o_gb = 0, o_top = 0, o_succ = 0;
        if (rankable || scannable) {
            o_ka = take(n2 * 8); o_kb = take(n2 * 4); o_ks = take(n2 * 4); o_pos = take(nSA * 4); o_sn = take(nSA * 4);
            o_rec = take(n2 * 16); o_np = take(n2 * 8); o_ge = take(n2 * 4); o_gb = take(n2 * 4); o_top = take((n2 + 1) * 4); o_succ = take(nS * 4);
        }
        CK(ctx->greedyBuf.ensure(off));
        char* b = ctx->greedyBuf.as<char>();
        GreedyBufs g;
        g.order = (int*)(b + o_order); g.cand = (GreedyCand*)(b + o_cand); g.upr = (long long*)(b + o_upr); g.rep = (long long*)(b + o_rep);
        g.ctype = (int*)(b + o_ct); g.nCand = (int*)(b + o_n); g.groupStart = (int*)(b + o_gs); g.groupItems = (int*)(b + o_gi);
        g.unalloc = (int*)(b + o_un); g.heapA = (unsigned long long*)(b + o_ha); g.heapB = (unsigned long long*)(b + o_hb);
        g.heapSlot = (unsigned*)(b + o_hs); g.tickets = (GreedyTicket*)(b + o_tk); g.liveIdx = (int*)(b + o_li);
        g.nanFlag = (int*)(b + o_nan);
        g.stats = (unsigned long long*)(b + o_stats);
        g.smemBytes = kGreedySmem;
        GreedyRank gr{};
        GreedyScan gsc{};
        if (rankable || scannable) {
            gr.ka = (unsigned long long*)(b + o_ka); gr.kb = (unsigned*)(b + o_kb); gr.kslot = (unsigned*)(b + o_ks);
            gr.posOf = (unsigned*)(b + o_pos); gr.snext = (int*)(b + o_sn); gr.rec = (int4*)(b + o_rec); gr.nextPos = (int2*)(b + o_np);
            gr.gend = (int*)(b + o_ge); gr.gbeg = (int*)(b + o_gb); gr.top = (int*)(b + o_top); gr.succ = (int*)(b + o_succ); gr.n2 = (unsigned)n2;
            // the scan path lays its arrays over the ranked queue's
            gsc.ka = gr.ka; gsc.kb = gr.kb; gsc.kslot = gr.kslot; gsc.posOf = gr.posOf; gsc.runHead = (unsigned char*)(b + o_sn);
            gsc.ev = gr.rec; gsc.push = gr.nextPos; gsc.gbeg = gr.gbeg; gsc.stackTop = gr.top; gsc.stackBuf = gr.gend;
            gsc.nEv = g.nanFlag; gsc.n2 = (unsigned)n2;
        }
        if (!ctx->greedy_attr) {
            CK(cudaFuncSetAttribute(k_greedy_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, kGreedySmem));
            CK(cudaFuncSetAttribute(k_greedy_solve_ranked, cudaFuncAttributeMaxDynamicSharedMemorySize, kGreedySmem));
            CK(cudaFuncSetAttribute(k_greedy_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, kGreedySmem));
            ctx->greedy_attr = true;
        }
        int* chosenKey = (int*)(b + o_key);
        CK(cudaMemsetAsync(g.groupStart, 0, 104 * 4, ctx->stream));
        CK(cudaMemsetAsync(g.nanFlag, 0, 8, ctx->stream));
        CK(cudaMemsetAsync(g.stats, 0, 32, ctx->stream));
        CK(cudaMemsetAsync(chosenKey, 0xff, nS * 4, ctx->stream));
        if (S > 0) {
            k_greedy_prepare<<<(S + 127) / 128, 128, 0, ctx->stream>>>(ctx->dsys, recs, feasible, g);
            LAUNCH_CHECK();
            k_greedy_bucket_count<<<(S + 255) / 256, 256, 0, ctx->stream>>>(ctx->dsys, g);
            LAUNCH_CHECK();
            if (rankable || scannable) {
                const unsigned nb = (unsigned)((n2 + 255) / 256), nt = (unsigned)(n2 / GREEDY_TILE);
                if (scannable) k_greedy_scan_keys<<<nb, 256, 0, ctx->stream>>>(ctx->dsys, g, gsc);
                else k_greedy_states<<<nb, 256, 0, ctx->stream>>>(ctx->dsys, g, gr);
                LAUNCH_CHECK();
                k_greedy_bitonic_tile<<<nt, 512, 0, ctx->stream>>>(gr, 2u, (unsigned)GREEDY_TILE);
                LAUNCH_CHECK();
                for (size_t k = 2 * (size_t)GREEDY_TILE; k <= n2; k <<= 1) {
                    for (size_t j = k >> 1; j >= (size_t)GREEDY_TILE; j >>= 1) {
                        k_greedy_bitonic_step<<<(unsigned)((n2 / 2 + 255) / 256), 256, 0, ctx->stream>>>(gr, (unsigned)k, (unsigned)j);
                        LAUNCH_CHECK();
                    }
                    k_greedy_bitonic_tile<<<nt, 512, 0, ctx->stream>>>(gr, (unsigned)k, (unsigned)k);
                    LAUNCH_CHECK();
                }
                CK(cudaMemsetAsync(gr.gend, 0, n2 * 4, ctx->stream));
                CK(cudaMemsetAsync(gr.top, 0, (n2 + 1) * 4, ctx->stream));
                k_greedy_index<<<nb, 256, 0, ctx->stream>>>(gr);
                LAUNCH_CHECK();
                if (scannable) {
                    CK(cudaMemsetAsync(gsc.gbeg, 0xff, n2 * 4, ctx->stream));
                    k_greedy_scan_groups<<<nb, 256, 0, ctx->stream>>>(ctx->dsys, gsc);
                    LAUNCH_CHECK();
                    k_greedy_scan_records<<<nb, 256, 0, ctx->stream>>>(ctx->dsys, g, gsc);
                    LAUNCH_CHECK();
                } else {
                    k_greedy_tie_groups<<<nb, 256, 0, ctx->stream>>>(gr);
                    LAUNCH_CHECK();
                    k_greedy_records<<<nb, 256, 0, ctx->stream>>>(ctx->dsys, g, gr);
                    LAUNCH_CHECK();
                    k_greedy_tie_init<<<nb, 256, 0, ctx->stream>>>(ctx->dsys, g, gr);
                    LAUNCH_CHECK();
                }
            }
            ctx->greedy_path = scannable ? 3 : rankable ? 2 : 1;
            if (ctx->greedy_path == 3) {
                // shared memory: one bit per server (stopped or not), plus the ticket pool of the round-robin policies
                size_t smem = doneBytes;
                const bool tickets = spec->saturation_policy == WVA_POLICY_ROUND_ROBIN || spec->saturation_policy == WVA_POLICY_PRIORITY_ROUND_ROBIN;
                if (tickets) smem = std::min((size_t)kGreedySmem, smem + nS * (sizeof(GreedyTicket) + 4));
                g.smemBytes = (int)smem;
                k_greedy_scan<<<1, 32, smem, ctx->stream>>>(ctx->dsys, recs, g, gsc, chosenKey, spec->delayed_best_effort ? 1 : 0,
                                                           spec->saturation_policy);
            }
            else if (ctx->greedy_path == 2) {
                // shared memory: the rank bitmap, plus the ticket pool when a round-robin policy can
                // use it; whatever is not asked for stays L1 for the record loads
                size_t smem = align_up(greedy_bitmap_bytes(nSA, nullptr, nullptr, nullptr), 16);
                const bool tickets = spec->saturation_policy == WVA_POLICY_ROUND_ROBIN || spec->saturation_policy == WVA_POLICY_PRIORITY_ROUND_ROBIN;
                if (tickets) smem = std::min((size_t)kGreedySmem, smem + nS * (sizeof(GreedyTicket) + 4));
                g.smemBytes = (int)smem;
                k_greedy_solve_ranked<<<1, 32, smem, ctx->stream>>>(ctx->dsys, recs, g, gr, chosenKey,
                                                                   spec->delayed_best_effort ? 1 : 0, spec->saturation_policy);
            }
            else
                k_greedy_solve<<<1, 32, kGreedySmem, ctx->stream>>>(ctx->dsys, recs, g, chosenKey, spec->delayed_best_effort ? 1 : 0,
                                                                   spec->saturation_policy);
            LAUNCH_CHECK();
            ctx->greedy_stats_dev = g.stats;
            k_greedy_collect<<<(S + 127) / 128, 128, 0, ctx->stream>>>(ctx->dsys, recs, g.order, chosenKey, ctx->chosen_acc, ctx->chosen);
            LAUNCH_CHECK();
        }
        // best-effort scaling mutated the candidate records in place (greedy.go:208-212): the
        // device copy no longer equals what the analysis produced
        valid = false;
    }
    if (spec->unlimited && !chosen_acc && !chosen) {
        // nothing goes back to the host: leave the work queued (later calls use the same stream) and read the
        // phase time when somebody asks for it
        CK(cudaEventRecord(ctx->evS1, ctx->stream));
        ctx->pendS = true;
        ctx->solved = true;
        return WVA_OK;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    timer.stop();
    ctx->solved = true;
    if (!spec->unlimited && S > 0 && ctx->greedy_stats_dev)
        CK(cudaMemcpy(ctx->greedy_stats, ctx->greedy_stats_dev, 32, cudaMemcpyDeviceToHost));
    if (count > 0) {
        if (chosen_acc) CK(cudaMemcpyAsync(chosen_acc + first, ctx->chosen_acc + first, (size_t)count * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (chosen) CK(download_allocs(ctx, ctx->chosen, (size_t)first, (size_t)count, chosen, (size_t)first));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return WVA_OK;
}

extern "C" {

int wva_solve(wva_ctx* ctx, const wva_optimizer_spec* spec, int32_t* chosen_acc, wva_alloc_soa* chosen) {
    if (!ctx || !spec) return fail(ctx, WVA_EINVAL, "null argument");
    if (!ctx->pairs_valid) return fail(ctx, WVA_ESTATE, "wva_solve needs wva_analyze_pairs first");
    return solve_records(ctx, spec, chosen_acc, chosen, ctx->pairs, ctx->feasible, ctx->pairs_valid, ctx->pairs_complete,
                         "limited-capacity solve needs the candidates of every server (wva_comm_init, or gather them and wva_pairs_commit)");
}

int wva_solve_grid(wva_ctx* ctx, const wva_optimizer_spec* spec, int32_t* chosen_acc, wva_alloc_soa* chosen) {
    if (!ctx || !spec) return fail(ctx, WVA_EINVAL, "null argument");
    if (!ctx->gpairs_valid)
        return fail(ctx, WVA_ESTATE, "wva_solve_grid needs a sweep with wva_grid_set_pair_winners on (records are invalidated by an image "
                                     "change or a sweep with the option off, and consumed by a limited solve)");
    return solve_records(ctx, spec, chosen_acc, chosen, ctx->gridPairs, ctx->gridFeasible, ctx->gpairs_valid, ctx->gpairs_complete,
                         "limited-capacity solve needs the sweep winners of every server (wva_comm_init)");
}

int wva_solve_set_ranked(wva_ctx* ctx, int32_t on) {
    if (!ctx) return WVA_EINVAL;
    ctx->greedy_ranked = on < 0 ? 0 : (on > 2 ? 2 : on);
    return WVA_OK;
}
int wva_solve_greedy_path(const wva_ctx* ctx) { return ctx ? ctx->greedy_path : WVA_EINVAL; }
int wva_solve_stats(wva_ctx* ctx, uint64_t out[4]) {
    if (!ctx || !out) return WVA_EINVAL;
    for (int i = 0; i < 4; ++i) out[i] = ctx->greedy_stats[i];
    return WVA_OK;
}

int wva_allocate_by_type(wva_ctx* ctx, int64_t* count, float* cost) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->solved) return fail(ctx, WVA_ESTATE, "wva_allocate_by_type needs wva_solve first");
    CK(cudaSetDevice(ctx->device));
    const int T = ctx->T;
    CK(ctx->totals.ensure((size_t)T * 12));
    PhaseTimer timer(ctx, WVA_PHASE_TOTALS, ctx->stream, ctx->evT0, ctx->evT1);
    ctx->pendT = false;
    long long* dcount = ctx->totals.as<long long>();
    float* dcost = (float*)(ctx->totals.as<char>() + (size_t)T * 8);
    k_totals<<<T, 1024, 0, ctx->stream>>>(ctx->dsys, ctx->s0, ctx->ns, ctx->chosen_acc, ctx->chosen, dcount, dcost, 0);
    LAUNCH_CHECK();
    if (ctx->comm) {
        // the one exchange step of the path: all-gather of the {count, cost} partials, summed in rank order
        const NcclApi& nc = nccl_api();
        CK(ctx->commTotals.ensure((size_t)ctx->comm_size * T * 12));
        int nrc = nc.AllGather(ctx->totals.p, ctx->commTotals.p, (size_t)T * 12, kNcclChar, ctx->comm, ctx->stream);
        if (nrc != 0) return fail(ctx, WVA_ECUDA, std::string("ncclAllGather(totals): ") + nc.GetErrorString(nrc));
        k_totals_merge<<<(T + 63) / 64, 64, 0, ctx->stream>>>(T, ctx->comm_size, ctx->commTotals.as<unsigned char>(), dcount, dcost);
        LAUNCH_CHECK();
    }
    if (!count && !cost) {            // totals stay on the device (wva_type_totals_device): no wait
        CK(cudaEventRecord(ctx->evT1, ctx->stream));
        ctx->pendT = true;
        return WVA_OK;
    }
    timer.stop();
    if (count) CK(cudaMemcpyAsync(count, dcount, (size_t)T * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (cost) CK(cudaMemcpyAsync(cost, dcost, (size_t)T * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return WVA_OK;
}

int wva_type_totals_device(wva_ctx* ctx, void** dev_ptr, size_t* bytes) {
    if (!ctx || !dev_ptr) return WVA_EINVAL;
    if (!ctx->totals.p) return fail(ctx, WVA_ESTATE, "wva_allocate_by_type has not run");
    *dev_ptr = ctx->totals.p;
    if (bytes) *bytes = (size_t)ctx->T * 12;
    return WVA_OK;
}

int wva_type_totals_merge(wva_ctx* ctx, const void* gathered_dev, int32_t n_ranks) {
    if (!ctx || !gathered_dev || n_ranks < 1) return fail(ctx, WVA_EINVAL, "null argument");
    if (!ctx->totals.p) return fail(ctx, WVA_ESTATE, "wva_allocate_by_type has not run");
    CK(cudaSetDevice(ctx->device));
    const int T = ctx->T;
    k_totals_merge<<<(T + 63) / 64, 64, 0, ctx->stream>>>(T, n_ranks, (const unsigned char*)gathered_dev, ctx->totals.as<long long>(),
                                                         (float*)(ctx->totals.as<char>() + (size_t)T * 8));
    LAUNCH_CHECK();
    return WVA_OK;
}

// ---------------------------------------------------------------------------------------------
// low-level analyzer API
static int queue_scratch(wva_ctx* ctx, const wva_queue_config* cfg, const std::vector<int>& list, DevBuf& offBuf) {
    std::vector<long long> offs(list.size());
    long long total = 0;
    for (size_t i = 0; i < list.size(); ++i) {
        const wva_queue_config& c = cfg[list[i]];
        offs[i] = total;
        total += (long long)c.max_batch_size + (long long)c.max_queue_size + 1;
    }
    size_t freeB = 0, totB = 0;
    CK(cudaMemGetInfo(&freeB, &totB));
    if ((size_t)total * 8 > freeB / 2) return fail(ctx, WVA_ECUDA, "not enough device memory for the materialised chain path");
    CK(ctx->scratch.ensure((size_t)total * 8));
    CK(offBuf.ensure(list.size() * 8));
    CK(cudaMemcpyAsync(offBuf.p, offs.data(), list.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    return WVA_OK;
}

int wva_queue_analyze(wva_ctx* ctx, int32_t n, const wva_queue_config* cfg, const float* rate, wva_metrics* metrics, uint8_t* status) {
    if (!ctx || n < 0 || !cfg || !rate || !metrics || !status) return fail(ctx, WVA_EINVAL, "null argument");
    if (n == 0) return WVA_OK;
    CK(cudaSetDevice(ctx->device));
    CK(ctx->ioA.ensure((size_t)n * sizeof(wva_queue_config)));
    CK(ctx->ioB.ensure((size_t)n * 4));
    CK(ctx->ioC.ensure((size_t)n * sizeof(wva_metrics)));
    CK(ctx->ioD.ensure((size_t)n));
    CK(ctx->faultList.ensure((size_t)n * 4));
    CK(ctx->faultCount.ensure(4));
    CK(cudaMemcpyAsync(ctx->ioA.p, cfg, (size_t)n * sizeof(wva_queue_config), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->ioB.p, rate, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->faultCount.p, 0, 4, ctx->stream));
    k_queue_analyze<<<(n + 127) / 128, 128, 0, ctx->stream>>>(n, ctx->ioA.as<wva_queue_config>(), ctx->ioB.as<float>(),
                                                             ctx->ioC.as<wva_metrics>(), ctx->ioD.as<unsigned char>(), nullptr,
                                                             nullptr, nullptr, ctx->faultList.as<int>(), ctx->faultCount.as<int>());
    LAUNCH_CHECK();
    int nf = 0;
    CK(cudaMemcpyAsync(&nf, ctx->faultCount.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (nf > 0) {
        std::vector<int> list((size_t)nf);
        CK(cudaMemcpy(list.data(), ctx->faultList.p, (size_t)nf * 4, cudaMemcpyDeviceToHost));
        int rc = queue_scratch(ctx, cfg, list, ctx->scratchOff);
        if (rc != WVA_OK) return rc;
        CK(ctx->ioG.ensure((size_t)nf * 4));
        CK(cudaMemcpyAsync(ctx->ioG.p, list.data(), (size_t)nf * 4, cudaMemcpyHostToDevice, ctx->stream));
        k_queue_analyze<<<(nf + 127) / 128, 128, 0, ctx->stream>>>(nf, ctx->ioA.as<wva_queue_config>(), ctx->ioB.as<float>(),
                                                                  ctx->ioC.as<wva_metrics>(), ctx->ioD.as<unsigned char>(),
                                                                  ctx->scratch.as<double>(), ctx->scratchOff.as<long long>(),
                                                                  ctx->ioG.as<int>(), ctx->faultList.as<int>(), ctx->faultCount.as<int>());
        LAUNCH_CHECK();
    }
    CK(cudaMemcpyAsync(metrics, ctx->ioC.p, (size_t)n * sizeof(wva_metrics), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(status, ctx->ioD.p, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return WVA_OK;
}

int wva_queue_size(wva_ctx* ctx, int32_t n, const wva_queue_config* cfg, const float* target, float* rates, wva_metrics* metrics,
                   float* achieved, uint8_t* status) {
    if (!ctx || n < 0 || !cfg || !target || !rates || !metrics || !achieved || !status) return fail(ctx, WVA_EINVAL, "null argument");
    if (n == 0) return WVA_OK;
    CK(cudaSetDevice(ctx->device));
    CK(ctx->ioA.ensure((size_t)n * sizeof(wva_queue_config)));
    CK(ctx->ioB.ensure((size_t)n * 12));
    CK(ctx->ioC.ensure((size_t)n * sizeof(wva_metrics)));
    CK(ctx->ioD.ensure((size_t)n));
    CK(ctx->ioE.ensure((size_t)n * 12));
    CK(ctx->ioF.ensure((size_t)n * 12));
    CK(ctx->faultList.ensure((size_t)n * 4));
    CK(ctx->faultCount.ensure(4));
    CK(cudaMemcpyAsync(ctx->ioA.p, cfg, (size_t)n * sizeof(wva_queue_config), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->ioB.p, target, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->faultCount.p, 0, 4, ctx->stream));
    k_queue_size<<<(n + 127) / 128, 128, 0, ctx->stream>>>(n, ctx->ioA.as<wva_queue_config>(), ctx->ioB.as<float>(), ctx->ioE.as<float>(),
                                                          ctx->ioC.as<wva_metrics>(), ctx->ioF.as<float>(), ctx->ioD.as<unsigned char>(),
                                                          nullptr, nullptr, nullptr, ctx->faultList.as<int>(), ctx->faultCount.as<int>());
    LAUNCH_CHECK();
    int nf = 0;
    CK(cudaMemcpyAsync(&nf, ctx->faultCount.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (nf > 0) {
        std::vector<int> list((size_t)nf);
        CK(cudaMemcpy(list.data(), ctx->faultList.p, (size_t)nf * 4, cudaMemcpyDeviceToHost));
        int rc = queue_scratch(ctx, cfg, list, ctx->scratchOff);
        if (rc != WVA_OK) return rc;
        CK(ctx->ioG.ensure((size_t)nf * 4));
        CK(cudaMemcpyAsync(ctx->ioG.p, list.data(), (size_t)nf * 4, cudaMemcpyHostToDevice, ctx->stream));
        k_queue_size<<<(nf + 127) / 128, 128, 0, ctx->stream>>>(nf, ctx->ioA.as<wva_queue_config>(), ctx->ioB.as<float>(), ctx->ioE.as<float>(),
                                                               ctx->ioC.as<wva_metrics>(), ctx->ioF.as<float>(), ctx->ioD.as<unsigned char>(),
                                                               ctx->scratch.as<double>(), ctx->scratchOff.as<long long>(), ctx->ioG.as<int>(),
                                                               ctx->faultList.as<int>(), ctx->faultCount.as<int>());
        LAUNCH_CHECK();
    }
    CK(cudaMemcpyAsync(rates, ctx->ioE.p, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(achieved, ctx->ioF.p, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(metrics, ctx->ioC.p, (size_t)n * sizeof(wva_metrics), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(status, ctx->ioD.p, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return WVA_OK;
}

// QueueAnalyzer.Size for every sweep record of the shard (kernels: wva_kernels.cuh, k_grid_size_*).  The warp path
// (shards up to wva_pairs_set_warp_max pairs) lists what it cannot finish; the listed records, or all of them on the
// thread path, are sized by k_queue_size, including its materialised-p[] re-run.
int wva_grid_pairs_size(wva_ctx* ctx, uint8_t* status) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->gpairs_valid)
        return fail(ctx, WVA_ESTATE, "no valid sweep winners per pair to size (wva_grid_set_pair_winners off, no sweep since, or consumed by a limited solve)");
    CK(cudaSetDevice(ctx->device));
    const int A = ctx->A, nPairs = ctx->ns * A;
    const int firstPair = ctx->s0 * A;
    CK(ctx->sizeStatus.ensure((size_t)(nPairs ? nPairs : 1)));
    CK(ctx->sizeList.ensure((size_t)(nPairs ? nPairs : 1) * 4));
    CK(ctx->sizeCount.ensure(4));
    PhaseTimer timer(ctx, WVA_PHASE_GRID_SIZE);
    if (nPairs > 0) {
        int* list = ctx->sizeList.as<int>();
        unsigned char* st = ctx->sizeStatus.as<unsigned char>();
        CK(cudaMemsetAsync(ctx->sizeCount.p, 0, 4, ctx->stream));
        if (nPairs <= ctx->pairs_warp_max) {
            // a record's b is at most the sweep's b_max: the table fits the warp's slice of up to 3072 entries (48 KB)
            // unless b_max is larger; records above the slice are listed
            const int smemEntries = ctx->grid_b < 3072 ? ctx->grid_b : 3072;
            const int warpsPerBlock = WVA_PAIRS_WARP_THREADS / 32;
            const size_t smemBytes = (size_t)smemEntries * 16 * warpsPerBlock;
            if (smemBytes > 48 * 1024)
                CK(cudaFuncSetAttribute(k_grid_size_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemBytes));
            k_grid_size_warp<<<(nPairs + warpsPerBlock - 1) / warpsPerBlock, WVA_PAIRS_WARP_THREADS, smemBytes, ctx->stream>>>(
                ctx->dsys, ctx->s0, nPairs, ctx->gridPairs, ctx->gridFeasible, st, list, ctx->sizeCount.as<int>(), smemEntries);
        } else {
            k_grid_size_list<<<(nPairs + 255) / 256, 256, 0, ctx->stream>>>(firstPair, nPairs, ctx->gridFeasible, st, list,
                                                                           ctx->sizeCount.as<int>());
        }
        LAUNCH_CHECK();
        int n = 0;
        CK(cudaMemcpyAsync(&n, ctx->sizeCount.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (n > 0) {
            CK(ctx->ioA.ensure((size_t)n * sizeof(wva_queue_config)));
            CK(ctx->ioB.ensure((size_t)n * 12));
            CK(ctx->ioC.ensure((size_t)n * sizeof(wva_metrics)));
            CK(ctx->ioD.ensure((size_t)n));
            CK(ctx->ioE.ensure((size_t)n * 12));
            CK(ctx->ioF.ensure((size_t)n * 12));
            CK(ctx->faultList.ensure((size_t)n * 4));
            CK(ctx->faultCount.ensure(4));
            wva_queue_config* cfg = ctx->ioA.as<wva_queue_config>();
            k_grid_size_gather<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->dsys, ctx->s0, list, n, ctx->gridPairs, cfg, ctx->ioB.as<float>());
            LAUNCH_CHECK();
            CK(cudaMemsetAsync(ctx->faultCount.p, 0, 4, ctx->stream));
            k_queue_size<<<(n + 127) / 128, 128, 0, ctx->stream>>>(n, cfg, ctx->ioB.as<float>(), ctx->ioE.as<float>(), ctx->ioC.as<wva_metrics>(),
                                                                  ctx->ioF.as<float>(), ctx->ioD.as<unsigned char>(), nullptr, nullptr, nullptr,
                                                                  ctx->faultList.as<int>(), ctx->faultCount.as<int>());
            LAUNCH_CHECK();
            int nf = 0;
            CK(cudaMemcpyAsync(&nf, ctx->faultCount.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            if (nf > 0) {
                // overflow-rescale chains: the same records again with p[] materialised in HBM (as wva_queue_size)
                std::vector<int> flist((size_t)nf);
                std::vector<wva_queue_config> hcfg((size_t)n);
                CK(cudaMemcpy(flist.data(), ctx->faultList.p, (size_t)nf * 4, cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(hcfg.data(), cfg, (size_t)n * sizeof(wva_queue_config), cudaMemcpyDeviceToHost));
                int rc = queue_scratch(ctx, hcfg.data(), flist, ctx->scratchOff);
                if (rc != WVA_OK) return rc;
                CK(ctx->ioG.ensure((size_t)nf * 4));
                CK(cudaMemcpyAsync(ctx->ioG.p, flist.data(), (size_t)nf * 4, cudaMemcpyHostToDevice, ctx->stream));
                k_queue_size<<<(nf + 127) / 128, 128, 0, ctx->stream>>>(nf, cfg, ctx->ioB.as<float>(), ctx->ioE.as<float>(), ctx->ioC.as<wva_metrics>(),
                                                                       ctx->ioF.as<float>(), ctx->ioD.as<unsigned char>(), ctx->scratch.as<double>(),
                                                                       ctx->scratchOff.as<long long>(), ctx->ioG.as<int>(),
                                                                       ctx->faultList.as<int>(), ctx->faultCount.as<int>());
                LAUNCH_CHECK();
            }
            k_grid_size_scatter<<<(n + 127) / 128, 128, 0, ctx->stream>>>(firstPair, list, n, ctx->ioC.as<wva_metrics>(),
                                                                         ctx->ioD.as<unsigned char>(), ctx->gridPairs, st);
            LAUNCH_CHECK();
        }
        if (status) CK(cudaMemcpyAsync(status + firstPair, st, (size_t)nPairs, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    timer.stop();
    return WVA_OK;
}

}  // extern "C"

// k_queue_size / k_queue_analyze listed rows in faultList (overflow-rescale chains): run them again with p[] materialised
// in HBM, as wva_queue_size does.  `cfg` holds the n device rows the kernel read; relaunch(nf) issues the re-run over
// the nf rows listed in ctx->ioG with the scratch offsets in ctx->scratchOff.
template <class Relaunch>
static int queue_fault_rerun(wva_ctx* ctx, const wva_queue_config* cfg, size_t n, Relaunch relaunch) {
    int nf = 0;
    CK(cudaMemcpyAsync(&nf, ctx->faultCount.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (nf == 0) return WVA_OK;
    std::vector<int> flist((size_t)nf);
    std::vector<wva_queue_config> hcfg(n);
    CK(cudaMemcpy(flist.data(), ctx->faultList.p, (size_t)nf * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(hcfg.data(), cfg, n * sizeof(wva_queue_config), cudaMemcpyDeviceToHost));
    int rc = queue_scratch(ctx, hcfg.data(), flist, ctx->scratchOff);
    if (rc != WVA_OK) return rc;
    CK(ctx->ioG.ensure((size_t)nf * 4));
    CK(cudaMemcpyAsync(ctx->ioG.p, flist.data(), (size_t)nf * 4, cudaMemcpyHostToDevice, ctx->stream));
    relaunch(nf);
    LAUNCH_CHECK();
    return WVA_OK;
}

// wva_analyze_scenarios' thread path for n pairs (`list`, or every shard pair when list is null): one Size per pair
// (k_queue_size), one Analyze per (pair, scenario) (k_queue_analyze), the records composed by k_scen_scatter
static int scen_thread_path(wva_ctx* ctx, const int* list, int n, int L, const float* rates) {
    const size_t rows = (size_t)n * L;
    if (rows > 0x7fffffffULL) return fail(ctx, WVA_EINVAL, "pairs x scenarios on the thread path exceed 2^31-1 rows");
    const int nr = (int)rows;
    CK(ctx->ioA.ensure((size_t)n * sizeof(wva_queue_config)));
    CK(ctx->ioB.ensure((size_t)n * 12));
    CK(ctx->ioC.ensure((size_t)n * sizeof(wva_metrics)));
    CK(ctx->ioD.ensure((size_t)n));
    CK(ctx->ioE.ensure((size_t)n * 12));
    CK(ctx->ioF.ensure((size_t)n * 12));
    CK(ctx->scenCfg.ensure(rows * sizeof(wva_queue_config)));
    CK(ctx->scenRate.ensure(rows * 4));
    CK(ctx->scenMetrics.ensure(rows * sizeof(wva_metrics)));
    CK(ctx->scenStatus.ensure(rows));
    CK(ctx->faultList.ensure(rows * 4));
    CK(ctx->faultCount.ensure(4));
    wva_queue_config* cfg = ctx->ioA.as<wva_queue_config>();
    float* target = ctx->ioB.as<float>();
    wva_metrics* qm = ctx->ioC.as<wva_metrics>();
    unsigned char* qs = ctx->ioD.as<unsigned char>();
    wva_queue_config* rcfg = ctx->scenCfg.as<wva_queue_config>();
    float* rrate = ctx->scenRate.as<float>();
    wva_metrics* am = ctx->scenMetrics.as<wva_metrics>();
    unsigned char* as = ctx->scenStatus.as<unsigned char>();
    k_scen_gather<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->dsys, ctx->s0, list, n, L, rates, cfg, target);
    LAUNCH_CHECK();
    CK(cudaMemsetAsync(ctx->faultCount.p, 0, 4, ctx->stream));
    k_queue_size<<<(n + 127) / 128, 128, 0, ctx->stream>>>(n, cfg, target, ctx->ioE.as<float>(), qm, ctx->ioF.as<float>(), qs, nullptr,
                                                          nullptr, nullptr, ctx->faultList.as<int>(), ctx->faultCount.as<int>());
    LAUNCH_CHECK();
    int rc = queue_fault_rerun(ctx, cfg, (size_t)n, [&](int nf) {
        k_queue_size<<<(nf + 127) / 128, 128, 0, ctx->stream>>>(nf, cfg, target, ctx->ioE.as<float>(), qm, ctx->ioF.as<float>(), qs,
                                                               ctx->scratch.as<double>(), ctx->scratchOff.as<long long>(),
                                                               ctx->ioG.as<int>(), ctx->faultList.as<int>(), ctx->faultCount.as<int>());
    });
    if (rc != WVA_OK) return rc;
    const unsigned rowBlocks = (unsigned)((rows + 255) / 256);
    k_scen_rows<<<rowBlocks, 256, 0, ctx->stream>>>(ctx->dsys, ctx->s0, list, n, L, rates, cfg, qm, qs, rcfg, rrate);
    LAUNCH_CHECK();
    CK(cudaMemsetAsync(ctx->faultCount.p, 0, 4, ctx->stream));
    k_queue_analyze<<<(nr + 127) / 128, 128, 0, ctx->stream>>>(nr, rcfg, rrate, am, as, nullptr, nullptr, nullptr, ctx->faultList.as<int>(),
                                                              ctx->faultCount.as<int>());
    LAUNCH_CHECK();
    rc = queue_fault_rerun(ctx, rcfg, rows, [&](int nf) {
        k_queue_analyze<<<(nf + 127) / 128, 128, 0, ctx->stream>>>(nf, rcfg, rrate, am, as, ctx->scratch.as<double>(),
                                                                  ctx->scratchOff.as<long long>(), ctx->ioG.as<int>(),
                                                                  ctx->faultList.as<int>(), ctx->faultCount.as<int>());
    });
    if (rc != WVA_OK) return rc;
    k_scen_scatter<<<rowBlocks, 256, 0, ctx->stream>>>(ctx->dsys, ctx->s0, list, n, L, rates, cfg, qm, qs, am, as, ctx->scenPairs,
                                                      ctx->scenFeasible);
    LAUNCH_CHECK();
    return WVA_OK;
}

extern "C" {

// What-if Server.Calculate -> SolveUnlimited -> AllocateByType over n_scen load scenarios (kernels: wva_kernels.cuh,
// k_scen_*).  Shards up to wva_pairs_set_warp_max pairs take one warp per pair (listing what it cannot finish), larger
// ones the thread path.  Everything else of the context is left as it was.
int wva_analyze_scenarios(wva_ctx* ctx, int32_t n_scen, const float* arrival_rpm, int32_t* chosen_acc, wva_alloc_soa* chosen,
                          int64_t* type_count, float* type_cost) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    if (n_scen < 1 || n_scen > WVA_MAX_SCENARIOS) return fail(ctx, WVA_EINVAL, "n_scen must be in [1, 1024]");
    if (!arrival_rpm) return fail(ctx, WVA_EINVAL, "arrival_rpm is NULL");
    const int S = ctx->S, A = ctx->A, T = ctx->T, L = n_scen;
    for (size_t i = 0; i < (size_t)L * S; ++i)
        if (!std::isfinite(arrival_rpm[i])) return fail(ctx, WVA_EINVAL, "scenario arrival rates must be finite");
    CK(cudaSetDevice(ctx->device));
    ctx->scen_valid = false;
    const size_t SA = (size_t)S * A;
    const int nPairs = ctx->ns * A;
    CK(ctx->scenRates.ensure((size_t)L * (S ? S : 1) * 4));
    CK(carve_allocs(ctx->scenRecBuf, (size_t)L * (SA ? SA : 1), ctx->scenPairs, &ctx->scenFeasible, nullptr));
    CK(carve_allocs(ctx->scenChosenBuf, (size_t)L * (S ? S : 1), ctx->scenChosen, nullptr, &ctx->scenChosenAcc));
    CK(ctx->scenTotals.ensure((size_t)L * T * 12));
    CK(ctx->scenList.ensure((size_t)(nPairs ? nPairs : 1) * 4));
    CK(ctx->scenCount.ensure(4));
    PhaseTimer timer(ctx, WVA_PHASE_SCENARIOS);
    float* rates = ctx->scenRates.as<float>();
    if (S > 0) CK(cudaMemcpyAsync(rates, arrival_rpm, (size_t)L * S * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (nPairs > 0) {
        int n = nPairs;
        const int* list = nullptr;
        if (nPairs <= ctx->pairs_warp_max) {
            // the warp's table slice: the shard's largest N (host copy of the image), at most 3072 entries (48 KB);
            // larger pairs are listed
            long long maxN = 0;
            for (int s = ctx->s0; s < ctx->s0 + ctx->ns; ++s) {
                const long long outTok = ctx->h_srv_out[(size_t)s];
                const int m = ctx->h_srv_model[(size_t)s];
                if (outTok <= 0 || m < 0) continue;
                for (int a = 0; a < A; ++a) {
                    long long N = ctx->h_srv_mb[(size_t)s];
                    if (N <= 0) {
                        const size_t pi = (size_t)m * A + a;
                        N = (long long)ctx->h_pmb[pi] * (long long)ctx->h_pat[pi] / outTok;
                    }
                    if (N > maxN) maxN = N;
                }
            }
            const int smemEntries = (int)(maxN < 3072 ? (maxN < 1 ? 1 : maxN) : 3072);
            const int warpsPerBlock = WVA_PAIRS_WARP_THREADS / 32;
            const size_t smemBytes = (size_t)smemEntries * 16 * warpsPerBlock;
            if (smemBytes > 48 * 1024)
                CK(cudaFuncSetAttribute(k_scen_pairs_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemBytes));
            CK(cudaMemsetAsync(ctx->scenCount.p, 0, 4, ctx->stream));
            k_scen_pairs_warp<<<(nPairs + warpsPerBlock - 1) / warpsPerBlock, WVA_PAIRS_WARP_THREADS, smemBytes, ctx->stream>>>(
                ctx->dsys, ctx->s0, nPairs, L, rates, ctx->scenPairs, ctx->scenFeasible, ctx->scenList.as<int>(), ctx->scenCount.as<int>(),
                smemEntries);
            LAUNCH_CHECK();
            CK(cudaMemcpyAsync(&n, ctx->scenCount.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            list = ctx->scenList.as<int>();
        }
        if (n > 0) {
            int rc = scen_thread_path(ctx, list, n, L, rates);
            if (rc != WVA_OK) return rc;
        }
        // SolveUnlimited of every scenario over the shard's servers
        k_solve_unlimited<<<dim3((unsigned)((ctx->ns + 127) / 128), (unsigned)L), 128, 0, ctx->stream>>>(
            ctx->dsys, ctx->s0, ctx->ns, ctx->scenPairs, ctx->scenFeasible, ctx->scenChosenAcc, ctx->scenChosen, SA, (size_t)S);
        LAUNCH_CHECK();
    }
    // AllocateByType of every scenario: partials {count[L*T]; cost[L*T]}, with a communicator ONE all-gather and the
    // rank-order sum of k_totals_merge over L*T entries
    long long* dcount = ctx->scenTotals.as<long long>();
    float* dcost = (float*)(ctx->scenTotals.as<char>() + (size_t)L * T * 8);
    k_totals<<<dim3((unsigned)T, (unsigned)L), 1024, 0, ctx->stream>>>(ctx->dsys, ctx->s0, ctx->ns, ctx->scenChosenAcc, ctx->scenChosen,
                                                                      dcount, dcost, (size_t)S);
    LAUNCH_CHECK();
    if (ctx->comm) {
        const NcclApi& nc = nccl_api();
        CK(ctx->scenGather.ensure((size_t)ctx->comm_size * L * T * 12));
        int nrc = nc.AllGather(ctx->scenTotals.p, ctx->scenGather.p, (size_t)L * T * 12, kNcclChar, ctx->comm, ctx->stream);
        if (nrc != 0) return fail(ctx, WVA_ECUDA, std::string("ncclAllGather(scenario totals): ") + nc.GetErrorString(nrc));
        k_totals_merge<<<(L * T + 63) / 64, 64, 0, ctx->stream>>>(L * T, ctx->comm_size, ctx->scenGather.as<unsigned char>(), dcount, dcost);
        LAUNCH_CHECK();
    }
    CK(cudaStreamSynchronize(ctx->stream));
    timer.stop();
    ctx->scen_n = L;
    ctx->scen_valid = true;
    if (ctx->ns > 0) {
        const size_t first = (size_t)ctx->s0, cnt = (size_t)ctx->ns;
        if (chosen_acc)
            CK(cudaMemcpy2DAsync(chosen_acc + first, (size_t)S * 4, ctx->scenChosenAcc + first, (size_t)S * 4, cnt * 4, (size_t)L,
                                 cudaMemcpyDeviceToHost, ctx->stream));
        if (chosen) CK(download_allocs_blocks(ctx, ctx->scenChosen, first, cnt, (size_t)S, (size_t)L, chosen));
    }
    if (type_count) CK(cudaMemcpyAsync(type_count, dcount, (size_t)L * T * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (type_cost) CK(cudaMemcpyAsync(type_cost, dcost, (size_t)L * T * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return WVA_OK;
}

int wva_scenario_pairs_fetch(wva_ctx* ctx, int32_t scen, wva_alloc_soa* out, uint8_t* feasible) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->scen_valid)
        return fail(ctx, WVA_ESTATE, "no scenario records (wva_analyze_scenarios has not run since the last image upload, update or shard change)");
    if (scen < 0 || scen >= ctx->scen_n) return fail(ctx, WVA_EINVAL, "scenario index out of range");
    CK(cudaSetDevice(ctx->device));
    const size_t SA = (size_t)ctx->S * ctx->A, first = (size_t)ctx->s0 * ctx->A, n = (size_t)ctx->ns * ctx->A;
    const size_t off = (size_t)scen * SA;
    if (n > 0) {
        if (out) CK(download_allocs(ctx, ctx->scenPairs, off + first, n, out, first));
        if (feasible) CK(cudaMemcpyAsync(feasible + first, ctx->scenFeasible + off + first, n, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return WVA_OK;
}

// ---------------------------------------------------------------------------------------------
// Device self-test of the hoisted division: compares div_hoisted(a, b, rcp_refined(b)) with a / b
// on n operand pairs produced on the device from a counter-based generator; returns the number of
// mismatching results (bitwise, NaNs compared by class).  Used by tests/test_div_gpu.py.
}  // extern "C"

namespace wva {
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
    x += 0x9e3779b97f4a7c15ULL;
    x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ULL;
    x = (x ^ (x >> 27)) * 0x94d049bb133111ebULL;
    return x ^ (x >> 31);
}
__global__ void k_div_selftest(unsigned long long seed, unsigned long long n, int mode, unsigned long long* mismatches) {
    unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long bad = 0;
    for (; i < n; i += stride) {
        unsigned long long ra = splitmix64(seed + 2 * i), rb = splitmix64(seed + 2 * i + 1);
        double a = 1.0, b = 1.0;
        if (mode >= 3) {
        } else if (mode == 0) {                 // chain-like operands: positive, any exponent; divisor a float32 value
            a = __longlong_as_double((long long)(ra & 0x7fffffffffffffffULL));
            float bf = __uint_as_float((unsigned)(rb & 0x7fffffffu));
            b = (double)bf;
        } else if (mode == 1) {          // arbitrary doubles (all exponents, both signs)
            a = __longlong_as_double((long long)ra);
            b = __longlong_as_double((long long)rb);
        } else {                         // moderate exponents: the common case of the chain
            a = __longlong_as_double((long long)((ra & 0x800fffffffffffffULL) | ((0x3ffULL - 40 + (ra >> 52) % 80) << 52)));
            b = __longlong_as_double((long long)((rb & 0x000fffffffffffffULL) | ((0x3ffULL - 20 + (rb >> 52) % 40) << 52)));
        }
        if (mode >= 3) {                  // float32: div_hoisted_f32 against the plain operator
            float af, bf;
            if (mode == 3) {              // exponents 2^-67 .. 2^66: the fast window [2^-60, 2^60] and both of its edges, both signs
                af = __uint_as_float((unsigned)(ra & 0x807fffffu) | ((unsigned)(60u + (ra >> 40) % 134u) << 23));
                bf = __uint_as_float((unsigned)(rb & 0x807fffffu) | ((unsigned)(60u + (rb >> 40) % 134u) << 23));
            } else {                      // any bit patterns: zeros, subnormals, Inf, NaN, extreme exponents
                af = __uint_as_float((unsigned)ra); bf = __uint_as_float((unsigned)rb);
            }
            const float reff = af / bf;
            const float gotf = div_hoisted_f32(af, bf, rcp_refined_f32(bf), f32_div_window(bf));
            const bool samef = (__float_as_uint(reff) == __float_as_uint(gotf)) || (reff != reff && gotf != gotf);
            if (!samef) ++bad;
            continue;
        }
        double ref = a / b;
        double got = divisor_in_window(b) ? div_hoisted(a, b, rcp_refined(b)) : a / b;
        bool same = (__double_as_longlong(ref) == __double_as_longlong(got)) || (ref != ref && got != got);
        if (!same) ++bad;
    }
    if (bad) atomicAdd(mismatches, bad);
}
}  // namespace wva

extern "C" int wva_selftest_division(wva_ctx* ctx, uint64_t seed, uint64_t n, int mode, uint64_t* mismatches) {
    if (!ctx || !mismatches) return WVA_EINVAL;
    CK(cudaSetDevice(ctx->device));
    CK(ctx->counters.ensure(3 * 8));
    CK(cudaMemsetAsync(ctx->counters.p, 0, 8, ctx->stream));
    wva::k_div_selftest<<<148 * 8, 256, 0, ctx->stream>>>(seed, n, mode, ctx->counters.as<unsigned long long>());
    LAUNCH_CHECK();
    CK(cudaMemcpyAsync(mismatches, ctx->counters.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return WVA_OK;
}

// ---------------------------------------------------------------------------------------------
// multi-GPU: communicator per ctx (one process per GPU) and device groups (one process, several GPUs)
// ---------------------------------------------------------------------------------------------
extern "C" {

int wva_comm_unique_id(void* id_out) {
    if (!id_out) return fail(nullptr, WVA_EINVAL, "id_out is NULL");
    const NcclApi& nc = nccl_api();
    if (!nc.ok) return fail(nullptr, WVA_ECUDA, "NCCL unavailable: " + nc.err);
    nccl_unique_id id;
    int rc = nc.GetUniqueId(&id);
    if (rc != 0) return fail(nullptr, WVA_ECUDA, std::string("ncclGetUniqueId: ") + nc.GetErrorString(rc));
    std::memcpy(id_out, &id, WVA_COMM_ID_BYTES);
    return WVA_OK;
}

int wva_comm_init(wva_ctx* ctx, const void* id, int32_t rank, int32_t n_ranks) {
    if (!ctx || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(ctx, WVA_EINVAL, "bad communicator arguments");
    if (ctx->comm) return fail(ctx, WVA_ESTATE, "a communicator is already attached");
    const NcclApi& nc = nccl_api();
    if (!nc.ok) return fail(ctx, WVA_ECUDA, "NCCL unavailable: " + nc.err);
    CK(cudaSetDevice(ctx->device));
    nccl_unique_id uid;
    std::memcpy(&uid, id, WVA_COMM_ID_BYTES);
    nccl_comm_t comm = nullptr;
    int rc = nc.CommInitRank(&comm, n_ranks, uid, rank);
    if (rc != 0) return fail(ctx, WVA_ECUDA, std::string("ncclCommInitRank: ") + nc.GetErrorString(rc));
    ctx->comm = comm; ctx->comm_rank = rank; ctx->comm_size = n_ranks; ctx->comm_owned = true;
    return WVA_OK;
}

int wva_comm_destroy(wva_ctx* ctx) {
    if (!ctx) return WVA_EINVAL;
    if (ctx->comm) {
        CK(cudaSetDevice(ctx->device));
        CK(cudaStreamSynchronize(ctx->stream));
        if (ctx->comm_owned && nccl_api().ok) nccl_api().CommDestroy(ctx->comm);
    }
    ctx->comm = nullptr; ctx->comm_rank = 0; ctx->comm_size = 1; ctx->comm_owned = false;
    return WVA_OK;
}

int wva_comm_info(const wva_ctx* ctx, int32_t* rank, int32_t* n_ranks) {
    if (!ctx) return WVA_EINVAL;
    if (rank) *rank = ctx->comm ? ctx->comm_rank : 0;
    if (n_ranks) *n_ranks = ctx->comm ? ctx->comm_size : 1;
    return WVA_OK;
}

int wva_comm_shard(wva_ctx* ctx) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    const long long S = ctx->S, g = ctx->comm ? ctx->comm_rank : 0, G = ctx->comm ? ctx->comm_size : 1;
    const int first = (int)(S * g / G), last = (int)(S * (g + 1) / G);
    return wva_set_shard(ctx, first, last - first);
}

}  // extern "C"

struct wva_group {
    std::vector<wva_ctx*> ctxs;
    std::string err;
    int S = 0, A = 0;
    // run f(i, ctx) on one host thread per device, return the first failure
    template <class F> int each(F f) {
        const int n = (int)ctxs.size();
        std::vector<int> rc((size_t)n, WVA_OK);
        if (n == 1) rc[0] = f(0, ctxs[0]);
        else {
            std::vector<std::thread> th;
            for (int i = 0; i < n; ++i) th.emplace_back([&, i] { rc[(size_t)i] = f(i, ctxs[(size_t)i]); });
            for (auto& t : th) t.join();
        }
        for (int i = 0; i < n; ++i)
            if (rc[(size_t)i] != WVA_OK) { err = "device " + std::to_string(ctxs[(size_t)i]->device) + ": " + wva_last_error(ctxs[(size_t)i]); return rc[(size_t)i]; }
        return WVA_OK;
    }
};

extern "C" {

int wva_group_create(const int32_t* device_ids, int32_t n_devices, wva_group** out) {
    if (!out) return fail(nullptr, WVA_EINVAL, "out is NULL");
    *out = nullptr;
    if (!device_ids || n_devices < 1 || n_devices > 64) return fail(nullptr, WVA_EINVAL, "bad device list");
    const NcclApi& nc = nccl_api();
    if (n_devices > 1 && !nc.ok) return fail(nullptr, WVA_ECUDA, "NCCL unavailable: " + nc.err);
    wva_group* g = new wva_group;
    for (int i = 0; i < n_devices; ++i) {
        wva_ctx* c = nullptr;
        int rc = wva_ctx_create(device_ids[i], &c);
        if (rc != WVA_OK) { wva_group_destroy(g); return rc; }
        g->ctxs.push_back(c);
    }
    if (nc.ok) {
        std::vector<nccl_comm_t> comms((size_t)n_devices, nullptr);
        std::vector<int> devs(device_ids, device_ids + n_devices);
        int rc = nc.CommInitAll(comms.data(), n_devices, devs.data());
        if (rc != 0) {
            std::string msg = std::string("ncclCommInitAll: ") + nc.GetErrorString(rc);
            wva_group_destroy(g);
            return fail(nullptr, WVA_ECUDA, msg);
        }
        for (int i = 0; i < n_devices; ++i) {
            wva_ctx* c = g->ctxs[(size_t)i];
            c->comm = comms[(size_t)i]; c->comm_rank = i; c->comm_size = n_devices; c->comm_owned = true;
        }
    }
    *out = g;
    return WVA_OK;
}

void wva_group_destroy(wva_group* g) {
    if (!g) return;
    for (wva_ctx* c : g->ctxs) wva_ctx_destroy(c);
    delete g;
}

int32_t wva_group_size(const wva_group* g) { return g ? (int32_t)g->ctxs.size() : 0; }
wva_ctx* wva_group_ctx(wva_group* g, int32_t i) { return (g && i >= 0 && (size_t)i < g->ctxs.size()) ? g->ctxs[(size_t)i] : nullptr; }
const char* wva_group_last_error(const wva_group* g) { return g ? g->err.c_str() : g_create_error.c_str(); }

int wva_group_upload(wva_group* g, const wva_system_soa* host) {
    if (!g || !host) return WVA_EINVAL;
    int rc = g->each([&](int, wva_ctx* c) {
        int r = wva_system_upload(c, host);
        return r != WVA_OK ? r : wva_comm_shard(c);
    });
    if (rc == WVA_OK) { g->S = host->n_servers; g->A = host->n_accels; }
    return rc;
}

int wva_group_analyze(wva_group* g, int32_t r_max, int32_t b_max, int32_t want_cube) {
    if (!g) return WVA_EINVAL;
    return g->each([&](int, wva_ctx* c) {
        return r_max > 0 ? wva_analyze(c, r_max, b_max, want_cube) : wva_analyze_pairs(c, nullptr, nullptr);
    });
}

int wva_group_pairs_fetch(wva_group* g, wva_alloc_soa* out, uint8_t* feasible) {
    if (!g) return WVA_EINVAL;
    return g->each([&](int, wva_ctx* c) { return wva_pairs_fetch(c, out, feasible); });   // each ctx writes its own rows
}

int wva_group_grid_fetch(wva_group* g, wva_grid_best* best) {
    if (!g || !best) return WVA_EINVAL;
    return g->each([&](int, wva_ctx* c) { return wva_grid_fetch(c, best + c->s0); });
}

int wva_group_solve(wva_group* g, const wva_optimizer_spec* spec, int32_t* chosen_acc, wva_alloc_soa* chosen) {
    if (!g || !spec) return WVA_EINVAL;
    // unlimited: every device solves and returns its own servers; limited: the gathered, replicated greedy
    // yields the same assignment everywhere -- device 0 returns it
    return g->each([&](int i, wva_ctx* c) {
        const bool mine = spec->unlimited || i == 0;
        return wva_solve(c, spec, mine ? chosen_acc : nullptr, mine ? chosen : nullptr);
    });
}

int wva_group_grid_pairs_fetch(wva_group* g, wva_alloc_soa* out, uint8_t* feasible) {
    if (!g) return WVA_EINVAL;
    return g->each([&](int, wva_ctx* c) { return wva_grid_pairs_fetch(c, out, feasible); });   // each ctx writes its own rows
}
int wva_group_grid_pairs_size(wva_group* g, uint8_t* status) {
    if (!g) return WVA_EINVAL;
    return g->each([&](int, wva_ctx* c) { return wva_grid_pairs_size(c, status); });            // each ctx sizes its own rows
}

int wva_group_analyze_scenarios(wva_group* g, int32_t n_scen, const float* arrival_rpm, int32_t* chosen_acc, wva_alloc_soa* chosen,
                                int64_t* type_count, float* type_cost) {
    if (!g) return WVA_EINVAL;
    // each ctx writes its own rows of chosen; the totals are global on every device -- device 0 returns them
    return g->each([&](int i, wva_ctx* c) {
        return wva_analyze_scenarios(c, n_scen, arrival_rpm, chosen_acc, chosen, i == 0 ? type_count : nullptr, i == 0 ? type_cost : nullptr);
    });
}
int wva_group_scenario_pairs_fetch(wva_group* g, int32_t scen, wva_alloc_soa* out, uint8_t* feasible) {
    if (!g) return WVA_EINVAL;
    return g->each([&](int, wva_ctx* c) { return wva_scenario_pairs_fetch(c, scen, out, feasible); });   // each ctx writes its own rows
}

int wva_group_solve_grid(wva_group* g, const wva_optimizer_spec* spec, int32_t* chosen_acc, wva_alloc_soa* chosen) {
    if (!g || !spec) return WVA_EINVAL;
    return g->each([&](int i, wva_ctx* c) {
        const bool mine = spec->unlimited || i == 0;
        return wva_solve_grid(c, spec, mine ? chosen_acc : nullptr, mine ? chosen : nullptr);
    });
}

int wva_group_allocate_by_type(wva_group* g, int64_t* count, float* cost) {
    if (!g) return WVA_EINVAL;
    return g->each([&](int i, wva_ctx* c) { return wva_allocate_by_type(c, i == 0 ? count : nullptr, i == 0 ? cost : nullptr); });
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// cgo-callable forms: every array its own argument (no pointer-to-pointer crosses the boundary)
// ---------------------------------------------------------------------------------------------
extern "C" {

int wva_system_upload_arrays(wva_ctx* ctx, int32_t n_servers, int32_t n_accels, int32_t n_models, int32_t n_types,
        const float* acc_cost, const int32_t* acc_multiplicity, const int32_t* acc_type, const int64_t* type_capacity,
        const float* perf_alpha, const float* perf_beta, const float* perf_gamma, const float* perf_delta,
        const int32_t* perf_max_batch, const int32_t* perf_at_tokens, const int32_t* perf_acc_count, const uint8_t* perf_valid,
        const int32_t* srv_model, const float* srv_arrival_rpm, const int32_t* srv_in_tokens, const int32_t* srv_out_tokens,
        const float* srv_slo_ttft, const float* srv_slo_itl, const float* srv_slo_tps, const uint8_t* srv_target_valid,
        const int32_t* srv_priority, const int32_t* srv_min_replicas, const int32_t* srv_max_batch, const uint8_t* srv_keep_acc,
        const int32_t* srv_cur_acc, const int32_t* srv_cur_replicas, const float* srv_cur_cost) {
    wva_system_soa h;
    h.n_servers = n_servers; h.n_accels = n_accels; h.n_models = n_models; h.n_types = n_types;
    h.acc_cost = acc_cost; h.acc_multiplicity = acc_multiplicity; h.acc_type = acc_type; h.type_capacity = type_capacity;
    h.perf_alpha = perf_alpha; h.perf_beta = perf_beta; h.perf_gamma = perf_gamma; h.perf_delta = perf_delta;
    h.perf_max_batch = perf_max_batch; h.perf_at_tokens = perf_at_tokens; h.perf_acc_count = perf_acc_count; h.perf_valid = perf_valid;
    h.srv_model = srv_model; h.srv_arrival_rpm = srv_arrival_rpm; h.srv_in_tokens = srv_in_tokens; h.srv_out_tokens = srv_out_tokens;
    h.srv_slo_ttft = srv_slo_ttft; h.srv_slo_itl = srv_slo_itl; h.srv_slo_tps = srv_slo_tps; h.srv_target_valid = srv_target_valid;
    h.srv_priority = srv_priority; h.srv_min_replicas = srv_min_replicas; h.srv_max_batch = srv_max_batch; h.srv_keep_acc = srv_keep_acc;
    h.srv_cur_acc = srv_cur_acc; h.srv_cur_replicas = srv_cur_replicas; h.srv_cur_cost = srv_cur_cost;
    return wva_system_upload(ctx, &h);
}

static wva_alloc_soa make_alloc_soa(int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value, float* itl,
                                    float* ttft, float* rho, float* max_arrv) {
    wva_alloc_soa o;
    o.acc = acc; o.num_replicas = num_replicas; o.batch_size = batch_size; o.cost = cost; o.value = value; o.itl = itl;
    o.ttft = ttft; o.rho = rho; o.max_arrv_rate_per_replica = max_arrv;
    return o;
}

int wva_analyze_pairs_arrays(wva_ctx* ctx, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica, uint8_t* feasible) {
    wva_alloc_soa o = make_alloc_soa(acc, num_replicas, batch_size, cost, value, itl, ttft, rho, max_arrv_rate_per_replica);
    return wva_analyze_pairs(ctx, &o, feasible);
}

int wva_pairs_fetch_arrays(wva_ctx* ctx, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica, uint8_t* feasible) {
    wva_alloc_soa o = make_alloc_soa(acc, num_replicas, batch_size, cost, value, itl, ttft, rho, max_arrv_rate_per_replica);
    return wva_pairs_fetch(ctx, &o, feasible);
}

int wva_solve_arrays(wva_ctx* ctx, int32_t unlimited, int32_t delayed_best_effort, int32_t saturation_policy,
        int32_t* chosen_acc, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica) {
    wva_optimizer_spec spec;
    spec.unlimited = unlimited; spec.delayed_best_effort = delayed_best_effort; spec.saturation_policy = saturation_policy;
    wva_alloc_soa o = make_alloc_soa(acc, num_replicas, batch_size, cost, value, itl, ttft, rho, max_arrv_rate_per_replica);
    return wva_solve(ctx, &spec, chosen_acc, &o);
}

int wva_grid_pairs_fetch_arrays(wva_ctx* ctx, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica, uint8_t* feasible) {
    wva_alloc_soa o = make_alloc_soa(acc, num_replicas, batch_size, cost, value, itl, ttft, rho, max_arrv_rate_per_replica);
    return wva_grid_pairs_fetch(ctx, &o, feasible);
}

int wva_solve_grid_arrays(wva_ctx* ctx, int32_t unlimited, int32_t delayed_best_effort, int32_t saturation_policy,
        int32_t* chosen_acc, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica) {
    wva_optimizer_spec spec;
    spec.unlimited = unlimited; spec.delayed_best_effort = delayed_best_effort; spec.saturation_policy = saturation_policy;
    wva_alloc_soa o = make_alloc_soa(acc, num_replicas, batch_size, cost, value, itl, ttft, rho, max_arrv_rate_per_replica);
    return wva_solve_grid(ctx, &spec, chosen_acc, &o);
}

int wva_analyze_scenarios_arrays(wva_ctx* ctx, int32_t n_scen, const float* arrival_rpm, int32_t* chosen_acc, int32_t* acc,
        int64_t* num_replicas, int64_t* batch_size, float* cost, float* value, float* itl, float* ttft, float* rho,
        float* max_arrv_rate_per_replica, int64_t* type_count, float* type_cost) {
    wva_alloc_soa o = make_alloc_soa(acc, num_replicas, batch_size, cost, value, itl, ttft, rho, max_arrv_rate_per_replica);
    return wva_analyze_scenarios(ctx, n_scen, arrival_rpm, chosen_acc, &o, type_count, type_cost);
}

int wva_scenario_pairs_fetch_arrays(wva_ctx* ctx, int32_t scen, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost,
        float* value, float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica, uint8_t* feasible) {
    wva_alloc_soa o = make_alloc_soa(acc, num_replicas, batch_size, cost, value, itl, ttft, rho, max_arrv_rate_per_replica);
    return wva_scenario_pairs_fetch(ctx, scen, &o, feasible);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// incremental updates of the resident image (pkg/core/system.go:99-171)
// ---------------------------------------------------------------------------------------------
namespace {
void invalidate_after_update(wva_ctx* ctx) {
    ctx->s0 = 0; ctx->ns = ctx->S;
    ctx->dsys.S = ctx->S; ctx->dsys.M = ctx->M;
    ctx->plan_valid = false;
    ctx->pairs_valid = ctx->pairs_complete = ctx->solved = ctx->grid_valid = ctx->gpairs_valid = ctx->gpairs_complete = ctx->scen_valid = false;
}
}  // namespace

extern "C" {

int64_t wva_upload_bytes(const wva_ctx* ctx) { return ctx ? ctx->last_h2d_bytes : 0; }

int wva_system_dims(const wva_ctx* ctx, int32_t* n_servers, int32_t* n_accels, int32_t* n_models, int32_t* n_types) {
    if (!ctx) return WVA_EINVAL;
    if (n_servers) *n_servers = ctx->S;
    if (n_accels) *n_accels = ctx->A;
    if (n_models) *n_models = ctx->M;
    if (n_types) *n_types = ctx->T;
    return WVA_OK;
}

int wva_system_update_servers(wva_ctx* ctx, int32_t first, int32_t count, const wva_system_soa* r) {
    if (!ctx || !r || count < 0 || first < 0) return fail(ctx, WVA_EINVAL, "bad argument");
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    if (r->n_servers != count) return fail(ctx, WVA_EINVAL, "rows->n_servers must equal count");
    if (first > ctx->S) return fail(ctx, WVA_EINVAL, "rows must be contiguous with the image (first <= S)");
    if ((long long)first + count > ctx->Scap) return fail(ctx, WVA_ECAPACITY, "no spare server rows left: upload the image again");
    if (((size_t)first + (size_t)count) * (size_t)ctx->A > 0x7fffffffULL) return fail(ctx, WVA_EINVAL, "S*A exceeds 2^31-1");
    for (int i = 0; i < count; ++i) {
        if (r->srv_model[i] >= ctx->M) return fail(ctx, WVA_EINVAL, "srv_model out of range");
        if (r->srv_cur_acc[i] < WVA_ACC_UNKNOWN || r->srv_cur_acc[i] >= ctx->A) return fail(ctx, WVA_EINVAL, "srv_cur_acc out of range");
        if (r->srv_priority[i] < 1 || r->srv_priority[i] > 100) return fail(ctx, WVA_EINVAL, "srv_priority must be in [1,100]");
    }
    if (count == 0) { ctx->last_h2d_bytes = 0; return WVA_OK; }
    CK(cudaSetDevice(ctx->device));
    PhaseTimer timer(ctx, WVA_PHASE_UPLOAD);
    const void* src[15] = {r->srv_model, r->srv_arrival_rpm, r->srv_in_tokens, r->srv_out_tokens, r->srv_slo_ttft, r->srv_slo_itl, r->srv_slo_tps,
                           r->srv_target_valid, r->srv_priority, r->srv_min_replicas, r->srv_max_batch, r->srv_keep_acc, r->srv_cur_acc,
                           r->srv_cur_replicas, r->srv_cur_cost};
    const size_t elem[15] = {4, 4, 4, 4, 4, 4, 4, 1, 4, 4, 4, 1, 4, 4, 4};
    // one pinned staging block, one async copy per array (the touched rows only)
    size_t need = 0;
    for (int k = 0; k < 15; ++k) need += align_up((size_t)count * elem[k], 16);
    CK(cudaStreamSynchronize(ctx->stream));                      // the staging buffer may still feed an earlier copy
    CK(ctx->staging.ensure(need));
    char* st = (char*)ctx->staging.p;
    char* d = ctx->arena.as<char>();
    size_t so = 0; int64_t moved = 0;
    for (int k = 0; k < 15; ++k) {
        const size_t bytes = (size_t)count * elem[k];
        std::memcpy(st + so, src[k], bytes);
        CK(cudaMemcpyAsync(d + ctx->off_srv[k] + (size_t)first * elem[k], st + so, bytes, cudaMemcpyHostToDevice, ctx->stream));
        so += align_up(bytes, 16); moved += (int64_t)bytes;
    }
    const int newS = first + count > ctx->S ? first + count : ctx->S;
    ctx->h_srv_model.resize((size_t)newS); ctx->h_srv_out.resize((size_t)newS); ctx->h_srv_mb.resize((size_t)newS); ctx->h_srv_arr.resize((size_t)newS);
    for (int i = 0; i < count; ++i) {
        ctx->h_srv_model[(size_t)first + i] = r->srv_model[i]; ctx->h_srv_out[(size_t)first + i] = r->srv_out_tokens[i];
        ctx->h_srv_mb[(size_t)first + i] = r->srv_max_batch[i]; ctx->h_srv_arr[(size_t)first + i] = r->srv_arrival_rpm[i];
    }
    ctx->S = newS;
    ctx->hostN.resize((size_t)newS * ctx->A, 0);
    host_plan_rows(ctx, first, first + count);
    ctx->last_h2d_bytes = moved;
    invalidate_after_update(ctx);
    timer.stop();
    return WVA_OK;
}

int wva_system_update_models(wva_ctx* ctx, int32_t first, int32_t count, const wva_system_soa* r) {
    if (!ctx || !r || count < 0 || first < 0) return fail(ctx, WVA_EINVAL, "bad argument");
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    if (r->n_models != count) return fail(ctx, WVA_EINVAL, "rows->n_models must equal count");
    if (first > ctx->M) return fail(ctx, WVA_EINVAL, "rows must be contiguous with the image (first <= M)");
    if ((long long)first + count > ctx->Mcap) return fail(ctx, WVA_ECAPACITY, "no spare model rows left: upload the image again");
    if (count == 0) { ctx->last_h2d_bytes = 0; return WVA_OK; }
    CK(cudaSetDevice(ctx->device));
    PhaseTimer timer(ctx, WVA_PHASE_UPLOAD);
    const int A = ctx->A;
    const void* src[8] = {r->perf_alpha, r->perf_beta, r->perf_gamma, r->perf_delta, r->perf_max_batch, r->perf_at_tokens, r->perf_acc_count, r->perf_valid};
    const size_t elem[8] = {4, 4, 4, 4, 4, 4, 4, 1};
    const size_t n = (size_t)count * A;
    size_t need = 0;
    for (int k = 0; k < 8; ++k) need += align_up(n * elem[k], 16);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(ctx->staging.ensure(need));
    char* st = (char*)ctx->staging.p;
    char* d = ctx->arena.as<char>();
    size_t so = 0; int64_t moved = 0;
    for (int k = 0; k < 8; ++k) {
        const size_t bytes = n * elem[k];
        std::memcpy(st + so, src[k], bytes);
        CK(cudaMemcpyAsync(d + ctx->off_perf[k] + (size_t)first * A * elem[k], st + so, bytes, cudaMemcpyHostToDevice, ctx->stream));
        so += align_up(bytes, 16); moved += (int64_t)bytes;
    }
    const int newM = first + count > ctx->M ? first + count : ctx->M;
    ctx->h_pmb.resize((size_t)newM * A, 0); ctx->h_pat.resize((size_t)newM * A, 0);
    for (size_t i = 0; i < n; ++i) { ctx->h_pmb[(size_t)first * A + i] = r->perf_max_batch[i]; ctx->h_pat[(size_t)first * A + i] = r->perf_at_tokens[i]; }
    ctx->M = newM;
    // servers of the touched models get a new table plan
    for (int s = 0; s < ctx->S; ++s) { const int m = ctx->h_srv_model[(size_t)s]; if (m >= first && m < first + count) host_plan_rows(ctx, s, s + 1); }
    ctx->last_h2d_bytes = moved;
    invalidate_after_update(ctx);
    timer.stop();
    return WVA_OK;
}

int wva_system_remove_server(wva_ctx* ctx, int32_t index) {
    if (!ctx) return WVA_EINVAL;
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    if (index < 0 || index >= ctx->S) return fail(ctx, WVA_EINVAL, "server index out of range");
    CK(cudaSetDevice(ctx->device));
    const int last = ctx->S - 1, A = ctx->A;
    if (index != last) {
        k_server_move<<<1, 32, 0, ctx->stream>>>(ctx->dsys, last, index);
        LAUNCH_CHECK();
        ctx->h_srv_model[(size_t)index] = ctx->h_srv_model[(size_t)last]; ctx->h_srv_out[(size_t)index] = ctx->h_srv_out[(size_t)last];
        ctx->h_srv_mb[(size_t)index] = ctx->h_srv_mb[(size_t)last]; ctx->h_srv_arr[(size_t)index] = ctx->h_srv_arr[(size_t)last];
        for (int a = 0; a < A; ++a) ctx->hostN[(size_t)index * A + a] = ctx->hostN[(size_t)last * A + a];
    }
    ctx->S = last;
    ctx->h_srv_model.resize((size_t)last); ctx->h_srv_out.resize((size_t)last); ctx->h_srv_mb.resize((size_t)last); ctx->h_srv_arr.resize((size_t)last);
    ctx->hostN.resize((size_t)last * A);
    ctx->last_h2d_bytes = 0;
    invalidate_after_update(ctx);
    return WVA_OK;
}

int wva_system_set_capacity(wva_ctx* ctx, const int64_t* type_capacity) {
    if (!ctx || !type_capacity) return fail(ctx, WVA_EINVAL, "null argument");
    if (!ctx->have_system) return fail(ctx, WVA_ESTATE, "no system uploaded");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    const size_t bytes = (size_t)ctx->T * 8;
    CK(ctx->staging.ensure(bytes));
    std::memcpy(ctx->staging.p, type_capacity, bytes);
    CK(cudaMemcpyAsync(ctx->arena.as<char>() + ctx->off_cap, ctx->staging.p, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ctx->last_h2d_bytes = (int64_t)bytes;
    ctx->solved = false;                                     // the candidates (pairs) do not depend on capacities
    return WVA_OK;
}

}  // extern "C"

extern "C" int wva_model_solve(wva_ctx* ctx, int64_t K, const float* serv_rate, int32_t n_rates, int32_t n_calls,
                               const float* lambda, const float* mu, float* out, double* p_out) {
    if (!ctx || !serv_rate || !lambda || !mu || !out || K < 0 || n_rates < 1 || n_calls < 0) return fail(ctx, WVA_EINVAL, "bad argument");
    if (K > (1LL << 28)) return fail(ctx, WVA_EINVAL, "K too large for the materialised model");
    if (n_calls == 0) return WVA_OK;
    CK(cudaSetDevice(ctx->device));
    CK(ctx->ioA.ensure((size_t)n_rates * 4));
    CK(ctx->ioB.ensure((size_t)n_calls * 8));
    CK(ctx->ioC.ensure((size_t)n_calls * 36));
    CK(ctx->scratch.ensure((size_t)(K + 1) * 8));
    CK(ctx->faultCount.ensure(4));
    CK(cudaMemcpyAsync(ctx->ioA.p, serv_rate, (size_t)n_rates * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->ioB.p, lambda, (size_t)n_calls * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->ioB.as<char>() + (size_t)n_calls * 4, mu, (size_t)n_calls * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->faultCount.p, 0, 4, ctx->stream));
    k_model_solve<<<1, 32, 0, ctx->stream>>>((long long)K, ctx->ioA.as<float>(), n_rates, n_calls, ctx->ioB.as<float>(),
                                            ctx->ioB.as<float>() + n_calls, ctx->scratch.as<double>(), ctx->ioC.as<float>(), ctx->faultCount.as<int>());
    LAUNCH_CHECK();
    int fault = 0;
    CK(cudaMemcpyAsync(out, ctx->ioC.p, (size_t)n_calls * 36, cudaMemcpyDeviceToHost, ctx->stream));
    if (p_out) CK(cudaMemcpyAsync(p_out, ctx->scratch.p, (size_t)(K + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&fault, ctx->faultCount.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (fault) return fail(ctx, WVA_ENONFINITE, "the reference does not terminate on this input (service rate <= 0 or NaN inside mm1modelstatedependent.go:84-89)");
    return WVA_OK;
}
