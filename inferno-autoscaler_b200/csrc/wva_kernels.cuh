// wva_kernels.cuh — sm_100a kernels of the Analyze -> Optimize path.
//
//   k_pairs          one thread per (server, accelerator): core.CreateAllocation + penalty
//   k_grid           candidate sweep: one thread per (server, accel, replicas, batch) candidate,
//                    service-rate tables staged in shared memory, warp-shuffle + block argmin
//   k_grid_list      deferred long chains / materialised-p[] chains, one thread per candidate
//   k_grid_claim     per-server (and, when asked for, per-pair) winners from the published (key, metrics) slots
//   k_grid_size_*    QueueAnalyzer.Size of the sweep's per-pair records (wva_grid_pairs_size)
//   k_solve_unlimited / k_greedy_*   the assignment step
//   k_scen_*         Server.Calculate under many load scenarios, one Size per pair (wva_analyze_scenarios)
//   k_totals         System.AllocateByType partial sums (input of the one NCCL allreduce)
//   k_queue_analyze / k_queue_size   the pkg/analyzer public API, batched
#pragma once

#include "wva_device.cuh"

namespace wva {

// Device copy of wva_system_soa (device pointers).
struct DevSystem {
    int S, A, M, T;
    int cert;      // tuning: certified closed-form tails on (1) / off (0); results identical either way
    const float* acc_cost; const int* acc_multiplicity; const int* acc_type;
    const long long* type_capacity;
    const float *perf_alpha, *perf_beta, *perf_gamma, *perf_delta;
    const int *perf_max_batch, *perf_at_tokens, *perf_acc_count; const unsigned char* perf_valid;
    const int* srv_model; const float* srv_arrival_rpm; const int *srv_in_tokens, *srv_out_tokens;
    const float *srv_slo_ttft, *srv_slo_itl, *srv_slo_tps; const unsigned char* srv_target_valid;
    const int *srv_priority, *srv_min_replicas, *srv_max_batch; const unsigned char* srv_keep_acc;
    const int *srv_cur_acc, *srv_cur_replicas; const float* srv_cur_cost;
};

struct DevAllocs {   // wva_alloc_soa with device pointers
    int* acc; long long* num_replicas; long long* batch_size;
    float *cost, *value, *itl, *ttft, *rho, *max_arrv;
};

__device__ __forceinline__ void store_alloc(const DevAllocs& o, size_t i, const AllocRec& a) {
    o.acc[i] = a.acc; o.num_replicas[i] = a.numReplicas; o.batch_size[i] = a.batchSize;
    o.cost[i] = a.cost; o.value[i] = a.value; o.itl[i] = a.itl; o.ttft[i] = a.ttft; o.rho[i] = a.rho;
    o.max_arrv[i] = a.maxArrv;
}
__device__ __forceinline__ AllocRec load_alloc(const DevAllocs& o, size_t i) {
    AllocRec a;
    a.acc = o.acc[i]; a.numReplicas = o.num_replicas[i]; a.batchSize = o.batch_size[i];
    a.cost = o.cost[i]; a.value = o.value[i]; a.itl = o.itl[i]; a.ttft = o.ttft[i]; a.rho = o.rho[i];
    a.maxArrv = o.max_arrv[i];
    return a;
}

__device__ __forceinline__ long long num_instances(const DevSystem& sys, int m, int a) {   // model.go:45-54
    int c = sys.perf_acc_count[(size_t)m * sys.A + a];
    return c <= 0 ? 1 : c;
}
// the nil-returning lookups of CreateAllocation, allocation.go:41-70
__device__ __forceinline__ bool pair_lookups_ok(const DevSystem& sys, int s, int a) {
    if (sys.srv_arrival_rpm[s] < 0.0f || sys.srv_in_tokens[s] < 0 || sys.srv_out_tokens[s] < 0) return false;
    int m = sys.srv_model[s];
    if (m < 0 || m >= sys.M) return false;
    if (!sys.perf_valid[(size_t)m * sys.A + a]) return false;
    if (!sys.srv_target_valid[s]) return false;
    return true;
}
// Server.GetCandidateAccelerators, server.go:70-82
__device__ __forceinline__ bool is_candidate_accel(const DevSystem& sys, int s, int a) {
    if (sys.srv_keep_acc[s]) {
        int cur = sys.srv_cur_acc[s];
        if (cur != WVA_ACC_NONE) return cur == a;
    }
    return true;
}

// zeroLoadAllocation, allocation.go:259-288
__device__ AllocRec zero_load_allocation(const DevSystem& sys, int s, int a) {
    AllocRec out = empty_alloc();
    long long numReplicas = sys.srv_min_replicas[s];
    if (numReplicas == 0) return out;
    int m = sys.srv_model[s];
    size_t pi = (size_t)m * sys.A + a;
    long long maxBatch = sys.perf_max_batch[pi];
    if (sys.srv_max_batch[s] > 0) maxBatch = sys.srv_max_batch[s];
    long long total = go_muli(num_instances(sys, m, a), numReplicas);
    float cost = sys.acc_cost[a] * (float)total;
    float alpha = sys.perf_alpha[pi], beta = sys.perf_beta[pi], gamma = sys.perf_gamma[pi], delta = sys.perf_delta[pi];
    float decode = alpha + beta;
    float bb = beta * (float)maxBatch;
    float maxDecode = alpha + bb;
    float prefill = gamma + delta;
    float maxServ = prefill + maxDecode;
    out.acc = a; out.numReplicas = numReplicas; out.batchSize = maxBatch;
    out.cost = cost; out.itl = decode; out.ttft = prefill; out.rho = 0.0f;
    out.maxArrv = (float)maxBatch / maxServ;
    out.value = cost;
    return out;
}

// N of CreateAllocation (allocation.go:77-87); 0 when the pair never reaches the queue analyzer.
__device__ __forceinline__ long long pair_batch_size(const DevSystem& sys, int s, int a) {
    if (!pair_lookups_ok(sys, s, a) || !is_candidate_accel(sys, s, a)) return 0;
    if (sys.srv_arrival_rpm[s] == 0.0f || sys.srv_out_tokens[s] == 0) return 0;
    if (sys.srv_max_batch[s] > 0) return sys.srv_max_batch[s];
    size_t pi = (size_t)sys.srv_model[s] * sys.A + a;
    long long n = go_divi(go_muli(sys.perf_max_batch[pi], sys.perf_at_tokens[pi]), sys.srv_out_tokens[s]);
    return n > 1 ? n : 1;
}

// core.CreateAllocation, allocation.go:27-163.  Returns false for nil.  `fault` is set when the
// streaming solver met an overflow-rescale case and no scratch was supplied (caller re-runs the
// pair in the literal kernel).
__device__ bool create_allocation(const DevSystem& sys, int s, int a, double* scratch, AllocRec& out, int& fault,
                                  unsigned long long& steps) {
    fault = 0;
    if (!pair_lookups_ok(sys, s, a)) return false;
    const float arrival = sys.srv_arrival_rpm[s];
    const long long inTok = sys.srv_in_tokens[s], outTok = sys.srv_out_tokens[s];
    if (arrival == 0.0f || outTok == 0) { out = zero_load_allocation(sys, s, a); return true; }
    const int m = sys.srv_model[s];
    const size_t pi = (size_t)m * sys.A + a;
    const long long K = outTok;
    long long N;
    if (sys.srv_max_batch[s] > 0) N = sys.srv_max_batch[s];
    else { N = go_divi(go_muli(sys.perf_max_batch[pi], sys.perf_at_tokens[pi]), K); if (N < 1) N = 1; }
    const long long maxQueue = go_muli(N, WVA_MAX_QUEUE_TO_BATCH_RATIO);
    if (!config_ok(N, maxQueue, inTok, K)) return false;
    ServiceParms sp; sp.alpha = sys.perf_alpha[pi]; sp.beta = sys.perf_beta[pi];
    sp.gamma = sys.perf_gamma[pi]; sp.delta = sys.perf_delta[pi];
    Analyzer qa;
    qa.build(sp, N, maxQueue, inTok, K, scratch);
    qa.cert = sys.cert != 0;
    const float tTTFT = sys.srv_slo_ttft[s], tITL = sys.srv_slo_itl[s], tTPS = sys.srv_slo_tps[s];
    float rates[3], achieved[3];
    wva_metrics metrics;
    bool ok = size_queue(qa, tTTFT, tITL, tTPS, rates, metrics, achieved);
    if (qa.fault) { fault = qa.fault; steps += qa.steps; return false; }
    if (!ok) { steps += qa.steps; return false; }
    const float rateStar = metrics.throughput;
    float totalRate;
    if (tTPS == 0.0f) totalRate = arrival / 60.0f;
    else totalRate = tTPS / (float)K;
    long long numReplicas = go_f64_to_int(ceil((double)totalRate / (double)rateStar));
    if (numReplicas < (long long)sys.srv_min_replicas[s]) numReplicas = sys.srv_min_replicas[s];
    const long long totalNumInstances = go_muli(num_instances(sys, m, a), numReplicas);
    const float cost = sys.acc_cost[a] * (float)totalNumInstances;
    const float rate = totalRate / (float)numReplicas;
    int st = qa.analyze(rate, metrics);
    steps += qa.steps;
    if (qa.fault) { fault = qa.fault; return false; }
    if (st != WVA_CAND_OK) return false;
    out.acc = a; out.numReplicas = numReplicas; out.batchSize = N;
    out.cost = cost; out.itl = metrics.avg_token_time;
    out.ttft = metrics.avg_wait_time + metrics.avg_prefill_time;
    out.rho = metrics.rho; out.maxArrv = rateStar / 1000.0f;
    out.value = cost;
    return true;
}

// Server.Calculate for one pair: candidate filter + CreateAllocation + transition penalty (server.go:55-67)
__device__ bool calculate_pair(const DevSystem& sys, int s, int a, double* scratch, AllocRec& out, int& fault,
                               unsigned long long& steps) {
    fault = 0;
    if (!is_candidate_accel(sys, s, a)) return false;
    if (!create_allocation(sys, s, a, scratch, out, fault, steps)) return false;
    out.value = transition_penalty(sys.srv_cur_acc[s], sys.srv_cur_replicas[s], sys.srv_cur_cost[s], out.acc,
                                   out.numReplicas, out.cost);
    return true;
}

// ---------------------------------------------------------------------------------------
// k_pairs: one thread per pair.  `order` (optional) permutes pair ids so that a warp holds pairs
// of similar chain length (sorted by N on the device beforehand) — lanes then finish together.
// Literal variant: `list` holds the pair ids that need the materialised path, scratch_off their
// p[] offsets.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_pairs(DevSystem sys, int s0, int nPairs, const int* __restrict__ order, DevAllocs out, unsigned char* feasible,
        int* slow_list, int* slow_count, unsigned long long* step_counter) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long steps = 0;
    if (t < nPairs) {
        int pid = order ? order[t] : t;           // pair id relative to shard: (s - s0) * A + a
        int s = s0 + pid / sys.A, a = pid % sys.A;
        AllocRec rec = empty_alloc();
        int fault = 0;
        bool ok = calculate_pair(sys, s, a, nullptr, rec, fault, steps);
        size_t gi = (size_t)s * sys.A + a;
        if (fault == 1) {
            int k = atomicAdd(slow_count, 1);
            slow_list[k] = pid;                   // capacity = nPairs
            ok = false;
        }
        if (!ok) rec = empty_alloc();
        store_alloc(out, gi, rec);
        feasible[gi] = ok ? 1 : 0;
    }
    // warp-reduce the step counter
    for (int o = 16; o > 0; o >>= 1) steps += __shfl_down_sync(0xffffffffu, steps, o);
    if ((threadIdx.x & 31) == 0 && steps) atomicAdd(step_counter, steps);
}

__global__ void __launch_bounds__(64)
k_pairs_literal(DevSystem sys, int s0, const int* __restrict__ list, int nList, double* scratch,
                const long long* __restrict__ scratch_off, DevAllocs out, unsigned char* feasible,
                unsigned long long* step_counter) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nList) return;
    int pid = list[t];
    int s = s0 + pid / sys.A, a = pid % sys.A;
    AllocRec rec = empty_alloc();
    int fault = 0;
    unsigned long long steps = 0;
    bool ok = calculate_pair(sys, s, a, scratch + scratch_off[t], rec, fault, steps);
    if (!ok) rec = empty_alloc();
    size_t gi = (size_t)s * sys.A + a;
    store_alloc(out, gi, rec);
    feasible[gi] = ok ? 1 : 0;
    atomicAdd(step_counter, steps);
}

// ---------------------------------------------------------------------------------------
// k_pairs_warp: one WARP per (server, accelerator) pair — the latency-oriented variant used when
// there are fewer pairs than the GPU has warps.  core.CreateAllocation is a chain of ~25-205
// dependent Solves (two bisections, then two Analyzes); a single thread runs them one after the
// other.  Here:
//   * the pair's {service rate, refined reciprocal} table is built once by the 32 lanes into global
//     memory (N x 16 B), so every chain step, ramp included, is DMUL + DMUL + 2 DFMA;
//   * the TTFT and ITL bisections of QueueAnalyzer.Size run concurrently on the two half-warps
//     (they only share the model through the stale-rho validity test, which is vacuous for
//     K = 11N >= 11 and lambda >= 0: SURVEY Appendix D.3);
//   * each bisection is evaluated speculatively: the interval endpoints are known float32 values, so
//     the midpoints of the next 4 levels of the bisection tree (15 nodes) are known too; 15 lanes
//     evaluate them at once and the warp then walks the tree with the reference's own comparisons.
//     The sequence of midpoints, iteration count (<= 100) and early exits are exactly those of
//     analyzer.BinarySearch (utils.go:26-70); evaluations off the realised path are discarded;
//   * the two trailing Analyzes (queueanalyzer.go:237-241, allocation.go:148) run side by side: the
//     second one's rate depends on the first one's throughput, which equals lambda*1000 exactly
//     whenever float32(p[K]) < 2^-25 — it is evaluated under that guess and re-done if wrong.
// Lanes call solve_uni together (idle lanes pass active = false), so the passes stay converged.
// ---------------------------------------------------------------------------------------

// x of node `node` (1-based heap index; children 2j = "xMax = x", 2j+1 = "xMin = x") of the
// bisection tree over [lo, hi]
__device__ __forceinline__ float bisect_node_x(float lo, float hi, int node) {
    const int depth = 31 - __clz(node);
    float x = 0.5f * (lo + hi);
    for (int l = depth - 1; l >= 0; --l) {
        if ((node >> l) & 1) lo = x; else hi = x;
        x = 0.5f * (lo + hi);
    }
    return x;
}

struct WarpPair {
    ServFormula sv; ProvTableF pv;
    double* pstore;                 // this lane's column of the warp's chain-value buffer, or nullptr
    bool cert;
    int N, K; long long inTok, outTok; bool tame;
    float rateMin, rateMax;
};

// one evaluation per lane (EvalTTFT / EvalITL / Analyze share the Solve); returns false when the
// lane's chain needs the materialised path.  certOnly: a speculative evaluation — if the certified tail
// cannot decide, report `uncertain` instead of running the long exact tail (the caller re-evaluates the
// node exactly only if the bisection actually walks through it).
__device__ __forceinline__ bool warp_solve(const WarpPair& wp, bool active, float x, SolveStats& st, unsigned long long& steps,
                                           bool& valid, bool certOnly, bool& uncertain) {
    int rc = solve_uni(wp.pv, wp.N, wp.K, x, wp.tame, st, steps, active, wp.pstore, wp.cert, certOnly);
    valid = true; uncertain = false;
    if (!active) return true;
    if (x < 0.0f) { valid = false; return true; }                       // queuemodel.go:31 (stale rho is in [0,1] < K)
    if (rc == WVA_SOLVE_UNCERTAIN) { uncertain = true; return true; }
    if (rc == WVA_SOLVE_CAREFUL) rc = solve_stream(wp.sv, (long long)wp.N, (long long)wp.K, x, wp.tame, st, steps);
    return rc == WVA_SOLVE_OK;
}
__device__ __forceinline__ float eval_y(const WarpPair& wp, int kind, const SolveStats& st) {
    float effConc = effective_concurrency(st.avgServTime, wp.sv.sp, wp.inTok, wp.outTok, wp.N);
    if (kind == 0) return st.avgWaitTime + prefill_time(wp.sv.sp, wp.inTok, effConc);   // EvalTTFT :270-279
    return decode_time(wp.sv.sp, effConc);                                              // EvalITL  :283-290
}
// QueueAnalyzer.Analyze's metrics from a Solve (queueanalyzer.go:152-173)
__device__ __forceinline__ void metrics_from(const WarpPair& wp, const SolveStats& st, wva_metrics& m) {
    float effConc = effective_concurrency(st.avgServTime, wp.sv.sp, wp.inTok, wp.outTok, wp.N);
    float rho = st.avgNumInServers / (float)wp.N;
    rho = go_minf(go_maxf(rho, 0.0f), 1.0f);
    m.throughput = st.throughput * 1000.0f;
    m.avg_resp_time = st.avgRespTime;
    m.avg_wait_time = st.avgWaitTime;
    m.avg_num_in_serv = st.avgNumInServers;
    m.avg_prefill_time = prefill_time(wp.sv.sp, wp.inTok, effConc);
    m.avg_token_time = decode_time(wp.sv.sp, effConc);
    m.max_rate = wp.rateMax;
    m.rho = rho;
}
__device__ __forceinline__ SolveStats shfl_stats(const SolveStats& s, int src) {
    SolveStats o;
    o.rho = __shfl_sync(0xffffffffu, s.rho, src);
    o.avgNumInServers = __shfl_sync(0xffffffffu, s.avgNumInServers, src);
    o.avgNumInSystem = __shfl_sync(0xffffffffu, s.avgNumInSystem, src);
    o.throughput = __shfl_sync(0xffffffffu, s.throughput, src);
    o.avgRespTime = __shfl_sync(0xffffffffu, s.avgRespTime, src);
    o.avgServTime = __shfl_sync(0xffffffffu, s.avgServTime, src);
    o.avgWaitTime = __shfl_sync(0xffffffffu, s.avgWaitTime, src);
    return o;
}

#define WVA_PAIRS_WARP_THREADS 128
// Shared part of the warp-per-pair kernels: one (server, accelerator) pair on one warp, every lane running the scalar
// part redundantly (uniform control flow).  BuildModel (queueanalyzer.go:99-131, the {rate, refined reciprocal} table
// built cooperatively), the two speculative half-warp bisections of QueueAnalyzer.Size and its trailing
// Analyze(requestRate) (:185-241) are common to all instantiations:
//   PAIR_ALLOC (k_pairs_warp): core.CreateAllocation -- N from the image, replicas, and the second Analyze
//                  (allocation.go:148) speculated beside the trailing one; `rec` is the allocation, `ok` = non-nil;
//   PAIR_SIZE  (k_grid_size_warp): Size alone at N = `batch`, MaxQueueSize 10 N; ok: rec.maxArrv = Throughput / 1000,
//                  !ok: Size returned an error.  The caller has checked that the pair holds a sweep record;
//   PAIR_SCEN  (k_scen_pairs_warp): Size alone at CreateAllocation's N (allocation.go:77-87); ok: *pmOut holds the
//                  pair's model, its table left in the warp's shared-memory slice, and Size's rateStar, for the caller's
//                  per-scenario Analyze calls.  The caller has run the rate-independent checks (candidate, lookups) and
//                  made sure the server has output tokens and some positive scenario rate.
// toSlow: the pair needs the thread path (no table budget / larger than the shared-memory slice, a bad service-rate
// table, or a chain that needs the materialised p[]).
enum PairMode { PAIR_ALLOC, PAIR_SIZE, PAIR_SCEN };
struct PairModel { WarpPair wp; float rateStar; };
template <int kMode>
__device__ __forceinline__ void warp_pair_size(const DevSystem& sys, const int s, const int a, const int pid, const int lane,
                                               const long long batch, const long long* __restrict__ tabOff, double2* tabs,
                                               unsigned char* smem, const int smemEntriesPerWarp, double* pbuf,
                                               const long long pbufStrideK, unsigned long long* step_counter, AllocRec& rec, bool& ok,
                                               bool& toSlow, unsigned long long& steps, int& activeRounds, int& totalRounds,
                                               int& pendEvals, long long& solveCycles, PairModel* pmOut = nullptr) {
    constexpr bool kAlloc = kMode == PAIR_ALLOC, kScen = kMode == PAIR_SCEN;
    do {
        if (kAlloc && (!is_candidate_accel(sys, s, a) || !pair_lookups_ok(sys, s, a))) break;
        const float arrival = sys.srv_arrival_rpm[s];
        const long long inTok = sys.srv_in_tokens[s], outTok = sys.srv_out_tokens[s];
        if (kAlloc && (arrival == 0.0f || outTok == 0)) { rec = zero_load_allocation(sys, s, a); ok = true; break; }
        const int m = sys.srv_model[s];
        const size_t pi = (size_t)m * sys.A + a;
        const long long Kt = outTok;
        long long N = batch;
        if (kAlloc || kScen) {
            if (sys.srv_max_batch[s] > 0) N = sys.srv_max_batch[s];
            else { N = go_divi(go_muli(sys.perf_max_batch[pi], sys.perf_at_tokens[pi]), Kt); if (N < 1) N = 1; }
        }
        const long long maxQueue = go_muli(N, WVA_MAX_QUEUE_TO_BATCH_RATIO);
        if (!config_ok(N, maxQueue, inTok, Kt)) break;
        // no table budget / (sizing) larger than the shared-memory slice: a thread kernel handles the pair
        if (kAlloc ? (tabOff[pid] < 0 || N > (1LL << 26)) : N > smemEntriesPerWarp) { toSlow = true; break; }
        WarpPair wp;
        ServiceParms sp; sp.alpha = sys.perf_alpha[pi]; sp.beta = sys.perf_beta[pi];
        sp.gamma = sys.perf_gamma[pi]; sp.delta = sys.perf_delta[pi];
        wp.sv.init(sp, inTok, Kt);
        wp.N = (int)N; wp.K = (int)(maxQueue + N); wp.inTok = inTok; wp.outTok = Kt;
        wp.tame = tame_parms(sp, inTok, Kt);
        wp.cert = sys.cert != 0;
        // the table lives in shared memory when it fits (29-cycle loads in the ramp), else in HBM
        double2* tab = (!kAlloc || wp.N <= smemEntriesPerWarp)
                           ? reinterpret_cast<double2*>(smem) + (size_t)(threadIdx.x >> 5) * smemEntriesPerWarp
                           : tabs + tabOff[pid];
        wp.pstore = (pbuf && (long long)wp.K + 1 <= pbufStrideK) ? pbuf + (size_t)pid * (size_t)pbufStrideK * 32 + lane : nullptr;
        // BuildModel (queueanalyzer.go:99-131): the table, cooperatively
        bool bad = false;
        for (int i = lane; i < wp.N; i += 32) {
            float r = wp.sv.rate(i + 1);
            if (!(r > 0.0f) || !(r < CUDART_INF_F)) bad = true;
            double d = (double)r;
            tab[i] = make_double2(d, rcp_refined(d));
        }
        __syncwarp();
        if (__any_sync(0xffffffffu, bad)) { toSlow = true; break; }
        wp.pv.tab = tab; wp.pv.sf = &wp.sv;
        {
            float lambdaMin = wp.sv.rate(1) * WVA_EPSILON;
            float lambdaMax = wp.sv.rate(wp.N) * (1.0f - WVA_EPSILON);
            wp.rateMin = lambdaMin * 1000.0f; wp.rateMax = lambdaMax * 1000.0f;
        }
        const float tTTFT = sys.srv_slo_ttft[s], tITL = sys.srv_slo_itl[s], tTPS = sys.srv_slo_tps[s];
        // ---- QueueAnalyzer.Size (queueanalyzer.go:185-255) ------------------------------------
        if (tITL < 0.0f || tTTFT < 0.0f || tTPS < 0.0f) break;
        const float lambdaMin = wp.rateMin / 1000.0f, lambdaMax = wp.rateMax / 1000.0f;
        const int half = lane >> 4, hl = lane & 15, base = lane & 16;
        const float target = half == 0 ? tTTFT : tITL;
        const bool searching = target > 0.0f;          // this half-warp's bisection is requested
        float lo = lambdaMin, hi = lambdaMax;
        float xStar = lambdaMax;                       // lambdaStar when the target is disabled
        int ind = 0, iters = 0;
        bool done = !searching, failed = false, inc = false;
        if (searching && lambdaMin > lambdaMax) { failed = true; done = true; }     // utils.go:29-31
        SolveStats st; st.rho = st.avgNumInServers = st.avgNumInSystem = st.throughput = st.avgRespTime = st.avgServTime = st.avgWaitTime = 0.0f;
        float lastX = -1.0f;                           // this lane's most recent evaluation point
        float ylo = 0.0f, yhi = 0.0f;                  // eval(lo), eval(hi): always known after the first round,
                                                       // so a midpoint that rounds onto an endpoint costs nothing
        bool first = true;
        int rounds = 0;
        while (__any_sync(0xffffffffu, !done)) {
            ++rounds;
            // --- choose this lane's evaluation point ---
            int node = 0; bool act = false; float x = 0.0f;
            if (!done) {
                if (first) {
                    if (hl == 0) { act = true; x = lo; }
                    else if (hl == 1) { act = true; x = hi; }
                    else if (hl <= 8) { node = hl - 1; act = true; x = bisect_node_x(lo, hi, node); }
                } else if (hl >= 1) { node = hl; act = true; x = bisect_node_x(lo, hi, node); }
                // never evaluate beyond the reference's iteration budget
                if (node > 0 && (31 - __clz(node)) >= WVA_BISECT_MAXIT - iters) act = false;
                // a midpoint equal to an endpoint of its own interval has a known value.  Endpoints of
                // deeper nodes are midpoints of shallower ones, so it is enough to test against the
                // node's own [lo', hi']: recompute them along the path.
                if (node > 0 && act) {
                    float l2 = lo, h2 = hi, xm = 0.5f * (lo + hi);
                    for (int l = (31 - __clz(node)) - 1; l >= 0; --l) { if ((node >> l) & 1) l2 = xm; else h2 = xm; xm = 0.5f * (l2 + h2); }
                    if (xm == l2 || xm == h2) act = false;      // resolved from the memo while walking
                }
            }
            bool valid, unc;
            if (__any_sync(0xffffffffu, act)) ++activeRounds;
            ++totalRounds;
            // tree nodes are speculative (certOnly); the two boundary evaluations are needed for sure
            const long long tw0 = clock64();
            bool solved = warp_solve(wp, act, x, st, steps, valid, node > 0, unc);
            solveCycles += clock64() - tw0;
            if (act && !unc) lastX = x;
            if (__any_sync(0xffffffffu, act && !solved)) { toSlow = true; break; }
            float y = act && valid && !unc ? eval_y(wp, half, st) : 0.0f;
            // --- walk the realised path (uniform inside each half-warp) ---
            if (first) {
                const float yb0 = __shfl_sync(0xffffffffu, y, base + 0), yb1 = __shfl_sync(0xffffffffu, y, base + 1);
                const bool v0 = __shfl_sync(0xffffffffu, (int)valid, base + 0), v1 = __shfl_sync(0xffffffffu, (int)valid, base + 1);
                if (!done) {
                    if (!v0) { failed = true; done = true; }
                    else if (within_tolerance(yb0, target, WVA_BISECT_TOL)) { xStar = lo; ind = 0; done = true; }
                    else if (!v1) { failed = true; done = true; }
                    else if (within_tolerance(yb1, target, WVA_BISECT_TOL)) { xStar = hi; ind = 0; done = true; }
                    else {
                        inc = yb0 < yb1;
                        ylo = yb0; yhi = yb1;
                        if ((inc && target < yb0) || (!inc && target > yb0)) { xStar = lo; ind = -1; done = true; }
                        else if ((inc && target > yb1) || (!inc && target < yb1)) { xStar = hi; ind = +1; done = true; }
                    }
                }
            }
            {
                const int levels = first ? 3 : 4;
                int cur = 1, lvl = 0;
                bool slowExit = false;
                for (;;) {
                    bool pend = false;                 // this half-warp walked into a node whose speculative evaluation was uncertain
                    for (int l = 0; l < levels; ++l) {
                        const int src = base + (first ? cur + 1 : cur);
                        float ys = __shfl_sync(0xffffffffu, y, src);
                        bool vs = __shfl_sync(0xffffffffu, (int)valid, src);
                        const bool us = __shfl_sync(0xffffffffu, (int)unc, src);
                        if (!done && !pend && l == lvl) {
                            if (iters == WVA_BISECT_MAXIT) { done = true; }
                            else {
                                const float xs = 0.5f * (lo + hi);
                                bool known = true;
                                if (xs == lo) { ys = ylo; vs = true; } else if (xs == hi) { ys = yhi; vs = true; }
                                else if (us) known = false;
                                if (!known) pend = true;           // needs the exact chain: evaluated below, then the walk resumes here
                                else {
                                    ++iters; ++lvl;
                                    if (!vs) { failed = true; done = true; }
                                    else {
                                        xStar = xs;
                                        if (within_tolerance(ys, target, WVA_BISECT_TOL)) done = true;
                                        else if ((inc && target < ys) || (!inc && target > ys)) { hi = xs; yhi = ys; cur = 2 * cur; }
                                        else { lo = xs; ylo = ys; cur = 2 * cur + 1; }
                                        if (!done && iters == WVA_BISECT_MAXIT) done = true;
                                    }
                                }
                            }
                        }
                    }
                    if (!__any_sync(0xffffffffu, pend)) break;
                    // exact evaluation of the pending node(s): the lane that owns node `cur` of a pending half-warp
                    const bool mine = pend && (hl == (first ? cur + 1 : cur));
                    bool v2, u2;
                    ++activeRounds; ++pendEvals;
                    bool solved2 = warp_solve(wp, mine, x, st, steps, v2, false, u2);
                    if (__any_sync(0xffffffffu, mine && !solved2)) { slowExit = true; break; }
                    if (mine) { valid = v2; unc = false; lastX = x; y = v2 ? eval_y(wp, half, st) : 0.0f; }
                }
                if (slowExit) { toSlow = true; break; }
            }
            first = false;
        }
        if (kAlloc && lane == 0) { atomicAdd(step_counter + 1, (unsigned long long)rounds); atomicMax(step_counter + 2, (unsigned long long)rounds); }
        if (toSlow) break;
        // results of the two bisections
        const bool failT = __shfl_sync(0xffffffffu, (int)failed, 0), failI = __shfl_sync(0xffffffffu, (int)failed, 16);
        const int indT = __shfl_sync(0xffffffffu, ind, 0), indI = __shfl_sync(0xffffffffu, ind, 16);
        const float lTTFT = __shfl_sync(0xffffffffu, xStar, 0), lITL = __shfl_sync(0xffffffffu, xStar, 16);
        if ((tTTFT > 0.0f && (failT || indT < 0))) break;                  // :205-214
        if ((tITL > 0.0f && (failI || indI < 0))) break;                   // :218-228
        float lTPS = lambdaMax;
        if (tTPS > 0.0f) lTPS = lambdaMax * (1.0f - WVA_STABILITY_SAFETY);
        const float lambda = go_minf(go_minf(lTTFT, lITL), lTPS);
        const float requestRate = lambda * 1000.0f;
        // ---- Analyze(requestRate) (:237-241) and, kAlloc, Analyze(totalRate/replicas) (allocation.go:148) ----
        if (requestRate <= 0.0f || requestRate > wp.rateMax) break;        // :135-143 -> Size fails -> nil
        const float x1 = requestRate / 1000.0f;
        float totalRate = 0.0f, rate2Guess = 0.0f;
        int minRep = 0;
        bool rate2GuessOk = false;
        if (kAlloc) {
            if (tTPS == 0.0f) totalRate = arrival / 60.0f;
            else totalRate = tTPS / (float)Kt;
            minRep = sys.srv_min_replicas[s];
            // guess: throughput == x1 (blocking probability below float32 resolution)
            const float rateStarGuess = x1 * 1000.0f;
            long long repGuess = go_f64_to_int(ceil((double)totalRate / (double)rateStarGuess));
            if (repGuess < (long long)minRep) repGuess = minRep;
            rate2Guess = totalRate / (float)repGuess;
            rate2GuessOk = !(rate2Guess <= 0.0f) && !(rate2Guess > wp.rateMax);
        }
        // reuse an evaluation already made at exactly x1 if some lane has one
        const unsigned have = __ballot_sync(0xffffffffu, lastX == x1);
        SolveStats st1, st2;
        bool valid1 = true, valid2 = true, solved = true;
        {
            const bool needX1 = (have == 0u);
            const bool actA = (lane == 0) && needX1, actB = kAlloc && (lane == 1) && rate2GuessOk;
            SolveStats stl = st;
            bool v;
            bool uu;
            solved = warp_solve(wp, actA || actB, lane == 0 ? x1 : rate2Guess / 1000.0f, stl, steps, v, false, uu);
            if (__any_sync(0xffffffffu, (actA || actB) && !solved)) { toSlow = true; break; }
            if (needX1) { st1 = shfl_stats(stl, 0); valid1 = __shfl_sync(0xffffffffu, (int)v, 0); }
            else { st1 = shfl_stats(st, __ffs(have) - 1); valid1 = true; }
            st2 = shfl_stats(stl, 1); valid2 = __shfl_sync(0xffffffffu, (int)v, 1);
        }
        if (!valid1) break;
        wva_metrics m1; metrics_from(wp, st1, m1);
        const float rateStar = m1.throughput;
        if (kScen) { pmOut->wp = wp; pmOut->wp.pv.sf = &pmOut->wp.sv; pmOut->rateStar = rateStar; ok = true; break; }
        if (!kAlloc) { rec.maxArrv = rateStar / 1000.0f; ok = true; break; }    // Size's metrics.Throughput / 1000
        long long numReplicas = go_f64_to_int(ceil((double)totalRate / (double)rateStar));
        if (numReplicas < (long long)minRep) numReplicas = minRep;
        const long long totalNumInstances = go_muli(num_instances(sys, m, a), numReplicas);
        const float cost = sys.acc_cost[a] * (float)totalNumInstances;
        const float rate2 = totalRate / (float)numReplicas;
        if (rate2 <= 0.0f || rate2 > wp.rateMax) break;                    // Analyze error -> nil
        if (lane == 0) atomicAdd(step_counter + 3, (unsigned long long)((have == 0u ? 1 : 0) + ((rate2GuessOk && rate2 == rate2Guess) ? 0 : 100)));
        if (!(rate2GuessOk && rate2 == rate2Guess)) {
            // the guess missed: evaluate the real second rate
            SolveStats stl = st; bool v;
            bool uu;
            solved = warp_solve(wp, lane == 0, rate2 / 1000.0f, stl, steps, v, false, uu);
            if (__any_sync(0xffffffffu, lane == 0 && !solved)) { toSlow = true; break; }
            st2 = shfl_stats(stl, 0); valid2 = __shfl_sync(0xffffffffu, (int)v, 0);
        }
        if (!valid2) break;
        wva_metrics m2; metrics_from(wp, st2, m2);
        rec.acc = a; rec.numReplicas = numReplicas; rec.batchSize = N;
        rec.cost = cost; rec.itl = m2.avg_token_time;
        rec.ttft = m2.avg_wait_time + m2.avg_prefill_time;
        rec.rho = m2.rho; rec.maxArrv = rateStar / 1000.0f;
        rec.value = cost;
        ok = true;
    } while (false);
}

__global__ void __launch_bounds__(WVA_PAIRS_WARP_THREADS)
k_pairs_warp(DevSystem sys, int s0, int nPairs, const long long* __restrict__ tabOff, double2* tabs, DevAllocs out,
             unsigned char* feasible, int* slow_list, int* slow_count, unsigned long long* step_counter,
             int smemEntriesPerWarp, double* pbuf, long long pbufStrideK, unsigned long long* dbg) {
    extern __shared__ __align__(16) unsigned char pairs_smem[];
    const long long tStart = clock64();
    int activeRounds = 0, totalRounds = 0, pendEvals = 0;
    long long solveCycles = 0;
    const int pid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;      // warp-uniform
    const int lane = threadIdx.x & 31;
    if (pid >= nPairs) return;
    const int s = s0 + pid / sys.A, a = pid % sys.A;
    const size_t gi = (size_t)s * sys.A + a;
    unsigned long long steps = 0;
    AllocRec rec = empty_alloc();
    bool ok = false;          // CreateAllocation != nil
    bool toSlow = false;      // needs the materialised path (whole pair re-done by k_pairs_literal)

    warp_pair_size<PAIR_ALLOC>(sys, s, a, pid, lane, 0, tabOff, tabs, pairs_smem, smemEntriesPerWarp, pbuf, pbufStrideK, step_counter,
                               rec, ok, toSlow, steps, activeRounds, totalRounds, pendEvals, solveCycles);

    if (ok) rec.value = transition_penalty(sys.srv_cur_acc[s], sys.srv_cur_replicas[s], sys.srv_cur_cost[s], rec.acc,
                                           rec.numReplicas, rec.cost);
    const unsigned long long tEnd = clock64();
    for (int o = 16; o > 0; o >>= 1) steps += __shfl_down_sync(0xffffffffu, steps, o);
    if (dbg && lane == 0) {
        // word 0: cycles (36 bits) | exact re-evaluations of uncertain nodes (8 bits) << 36 | chain steps / 1024 (20 bits) << 44
        unsigned long long ks = (unsigned long long)solveCycles >> 10; if (ks > 0xfffffull) ks = 0xfffffull;
        dbg[2 * pid] = ((tEnd - tStart) & 0xfffffffffull) | ((unsigned long long)(pendEvals & 0xff) << 36) | (ks << 44);
        dbg[2 * pid + 1] = ((unsigned long long)totalRounds << 32) | (unsigned)activeRounds;
    }
    if (lane == 0) {
        if (toSlow) { ok = false; slow_list[atomicAdd(slow_count, 1)] = pid; }
        if (!ok) rec = empty_alloc();
        store_alloc(out, gi, rec);
        feasible[gi] = ok ? 1 : 0;
        if (steps) atomicAdd(step_counter, steps);
    }
}

// ---------------------------------------------------------------------------------------
// wva_grid_pairs_size: QueueAnalyzer.Size for every sweep record of the shard at the record's own batch size b
// (CreateAllocation's Size, allocation.go:81-131, with N = b, MaxQueueSize = 10 b).  status[pid] (shard-local pair):
// 0 no record, 1 sized (max_arrv_rate_per_replica = Throughput / 1000), 2 Size returned an error (record unchanged).
// k_grid_size_warp (one warp per pair) lists the records it cannot finish; k_grid_size_list lists every record when
// the thread path is chosen.  Listed records go through k_grid_size_gather -> k_queue_size -> k_grid_size_scatter.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(WVA_PAIRS_WARP_THREADS)
k_grid_size_warp(DevSystem sys, int s0, int nPairs, DevAllocs recs, const unsigned char* __restrict__ feasible,
                 unsigned char* __restrict__ status, int* list, int* list_count, int smemEntriesPerWarp) {
    extern __shared__ __align__(16) unsigned char size_smem[];
    const int pid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;      // warp-uniform
    const int lane = threadIdx.x & 31;
    if (pid >= nPairs) return;
    const int s = s0 + pid / sys.A, a = pid % sys.A;
    const size_t gi = (size_t)s * sys.A + a;
    if (!feasible[gi]) { if (lane == 0) status[pid] = 0; return; }
    unsigned long long steps = 0;
    int activeRounds = 0, totalRounds = 0, pendEvals = 0;
    long long solveCycles = 0;
    AllocRec rec = empty_alloc();
    bool ok = false, toSlow = false;
    warp_pair_size<PAIR_SIZE>(sys, s, a, pid, lane, recs.batch_size[gi], nullptr, nullptr, size_smem, smemEntriesPerWarp, nullptr, 0,
                              nullptr, rec, ok, toSlow, steps, activeRounds, totalRounds, pendEvals, solveCycles);
    if (lane == 0) {
        if (toSlow) list[atomicAdd(list_count, 1)] = pid;
        else {
            if (ok) recs.max_arrv[gi] = rec.maxArrv;
            status[pid] = ok ? 1 : 2;
        }
    }
}

__global__ void k_grid_size_list(int firstPair, int nPairs, const unsigned char* __restrict__ feasible, unsigned char* __restrict__ status,
                                 int* list, int* list_count) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nPairs) return;
    status[t] = 0;
    if (feasible[(size_t)firstPair + t]) list[atomicAdd(list_count, 1)] = t;
}

// k_queue_size inputs of the listed records: {b, 10 b, alpha, beta, gamma, delta, in, out} and {TTFT, ITL, TPS}
__global__ void k_grid_size_gather(DevSystem sys, int s0, const int* __restrict__ list, int n, DevAllocs recs,
                                   wva_queue_config* __restrict__ cfg, float* __restrict__ target) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int pid = list[t];
    const int s = s0 + pid / sys.A, a = pid % sys.A;
    const size_t gi = (size_t)s * sys.A + a, pi = (size_t)sys.srv_model[s] * sys.A + a;
    const long long b = recs.batch_size[gi];
    wva_queue_config c;
    c.max_batch_size = (int)b; c.max_queue_size = (int)go_muli(b, WVA_MAX_QUEUE_TO_BATCH_RATIO);
    c.alpha = sys.perf_alpha[pi]; c.beta = sys.perf_beta[pi]; c.gamma = sys.perf_gamma[pi]; c.delta = sys.perf_delta[pi];
    c.avg_input_tokens = sys.srv_in_tokens[s]; c.avg_output_tokens = sys.srv_out_tokens[s];
    cfg[t] = c;
    target[3 * t] = sys.srv_slo_ttft[s]; target[3 * t + 1] = sys.srv_slo_itl[s]; target[3 * t + 2] = sys.srv_slo_tps[s];
}

__global__ void k_grid_size_scatter(int firstPair, const int* __restrict__ list, int n, const wva_metrics* __restrict__ metrics,
                                    const unsigned char* __restrict__ qstatus, DevAllocs recs, unsigned char* __restrict__ status) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int pid = list[t];
    if (qstatus[t] == 0) recs.max_arrv[(size_t)firstPair + pid] = metrics[t].throughput / 1000.0f;
    status[pid] = qstatus[t] == 0 ? 1 : 2;
}

// ---------------------------------------------------------------------------------------
// wva_analyze_scenarios: Server.Calculate of every shard pair under L load scenarios, scenario l replacing each server's
// arrival rate by rates[l*S + s].  Every input of QueueAnalyzer.Size is independent of the arrival rate
// (allocation.go:77-131), so a pair runs Size once; per scenario only the nil / zero-load branches (:50, :73-75), the
// replica count, the cost and the trailing Analyze(totalRate / replicas) (:133-160) remain.  The records of scenario l
// are the S*A records at offset l*S*A of one record set.
//   k_scen_pairs_warp   one warp per pair: Size through warp_pair_size<PAIR_SCEN>, then the scenarios 32 at a time,
//                       lane = scenario, one warp_solve for all lanes; pairs it cannot finish are listed;
//   k_scen_gather -> k_queue_size -> k_scen_rows -> k_queue_analyze -> k_scen_scatter
//                       the listed pairs (every pair on the thread path): Size and the per-scenario Analyze through the
//                       batched analyzer kernels (materialised-p[] re-runs included), records composed by the scatter.
// ---------------------------------------------------------------------------------------

// the nil checks of Server.Calculate + CreateAllocation that do not read the arrival rate (server.go:70-82,
// allocation.go:41-70 without :50)
__device__ __forceinline__ bool scen_pair_usable(const DevSystem& sys, int s, int a) {
    if (!is_candidate_accel(sys, s, a)) return false;
    if (sys.srv_in_tokens[s] < 0 || sys.srv_out_tokens[s] < 0) return false;
    const int m = sys.srv_model[s];
    if (m < 0 || m >= sys.M) return false;
    if (!sys.perf_valid[(size_t)m * sys.A + a]) return false;
    return sys.srv_target_valid[s] != 0;
}

// does server s see a positive rate in any scenario (else its pairs need no Size)
__device__ __forceinline__ bool scen_any_positive(const float* __restrict__ rates, int L, int S, int s, int from, int step) {
    bool any = false;
    for (int l = from; l < L; l += step) any |= rates[(size_t)l * S + s] > 0.0f;
    return any;
}

// N of CreateAllocation (allocation.go:77-87)
__device__ __forceinline__ long long scen_batch(const DevSystem& sys, int s, int a) {
    if (sys.srv_max_batch[s] > 0) return sys.srv_max_batch[s];
    const size_t pi = (size_t)sys.srv_model[s] * sys.A + a;
    const long long N = go_divi(go_muli(sys.perf_max_batch[pi], sys.perf_at_tokens[pi]), (long long)sys.srv_out_tokens[s]);
    return N < 1 ? 1 : N;
}

#define WVA_SCEN_NIL  0    // CreateAllocation returns nil
#define WVA_SCEN_ZERO 1    // zeroLoadAllocation: `rec` is the allocation
#define WVA_SCEN_RATE 2    // Analyze(rate2) decides; numReplicas and cost are set
// One scenario of a usable pair up to its trailing Analyze (allocation.go:50, :73-75, :133-147).  sized / rateStar:
// the pair's Size succeeded with metrics.Throughput rateStar.
__device__ __forceinline__ int scen_step(const DevSystem& sys, int s, int a, float r, bool sized, float rateStar,
                                         long long& numReplicas, float& cost, float& rate2, AllocRec& rec) {
    if (r < 0.0f) return WVA_SCEN_NIL;
    const long long Kt = sys.srv_out_tokens[s];
    if (r == 0.0f || Kt == 0) { rec = zero_load_allocation(sys, s, a); return WVA_SCEN_ZERO; }
    if (!sized) return WVA_SCEN_NIL;
    const float tTPS = sys.srv_slo_tps[s];
    float totalRate;
    if (tTPS == 0.0f) totalRate = r / 60.0f;
    else totalRate = tTPS / (float)Kt;
    numReplicas = go_f64_to_int(ceil((double)totalRate / (double)rateStar));
    if (numReplicas < (long long)sys.srv_min_replicas[s]) numReplicas = sys.srv_min_replicas[s];
    cost = sys.acc_cost[a] * (float)go_muli(num_instances(sys, sys.srv_model[s], a), numReplicas);
    rate2 = totalRate / (float)numReplicas;
    return WVA_SCEN_RATE;
}

// the allocation once Analyze(rate2) returned m2 (allocation.go:150-160)
__device__ __forceinline__ AllocRec scen_alloc(int a, long long N, long long numReplicas, float cost, float rateStar,
                                               const wva_metrics& m2) {
    AllocRec rec;
    rec.acc = a; rec.numReplicas = numReplicas; rec.batchSize = N;
    rec.cost = cost; rec.itl = m2.avg_token_time;
    rec.ttft = m2.avg_wait_time + m2.avg_prefill_time;
    rec.rho = m2.rho; rec.maxArrv = rateStar / 1000.0f;
    rec.value = cost;
    return rec;
}

// record i of the scenario set: the allocation with its transition penalty (server.go:62-64), or nil
__device__ __forceinline__ void scen_store(const DevSystem& sys, int s, const DevAllocs& recs, unsigned char* feasible, size_t i,
                                           bool ok, AllocRec rec) {
    if (ok) rec.value = transition_penalty(sys.srv_cur_acc[s], sys.srv_cur_replicas[s], sys.srv_cur_cost[s], rec.acc,
                                           rec.numReplicas, rec.cost);
    else rec = empty_alloc();
    store_alloc(recs, i, rec);
    feasible[i] = ok ? 1 : 0;
}

__global__ void __launch_bounds__(WVA_PAIRS_WARP_THREADS)
k_scen_pairs_warp(DevSystem sys, int s0, int nPairs, int L, const float* __restrict__ rates, DevAllocs recs,
                  unsigned char* __restrict__ feasible, int* list, int* list_count, int smemEntriesPerWarp) {
    extern __shared__ __align__(16) unsigned char scen_smem[];
    const int pid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;      // warp-uniform
    const int lane = threadIdx.x & 31;
    if (pid >= nPairs) return;
    const int S = sys.S;
    const int s = s0 + pid / sys.A, a = pid % sys.A;
    const size_t gi = (size_t)s * sys.A + a, SA = (size_t)S * sys.A;
    const bool usable = scen_pair_usable(sys, s, a);
    const bool anyPos = __any_sync(0xffffffffu, scen_any_positive(rates, L, S, s, lane, 32));
    PairModel pm;
    pm.rateStar = 0.0f;
    bool sized = false, toSlow = false;
    unsigned long long steps = 0;
    if (usable && anyPos && sys.srv_out_tokens[s] != 0) {
        int activeRounds = 0, totalRounds = 0, pendEvals = 0;
        long long solveCycles = 0;
        AllocRec rec = empty_alloc();
        warp_pair_size<PAIR_SCEN>(sys, s, a, pid, lane, 0, nullptr, nullptr, scen_smem, smemEntriesPerWarp, nullptr, 0, nullptr,
                                  rec, sized, toSlow, steps, activeRounds, totalRounds, pendEvals, solveCycles, &pm);
    }
    for (int base = 0; base < L && !toSlow; base += 32) {
        const int l = base + lane;
        const bool active = l < L;
        AllocRec rec = empty_alloc();
        long long reps = 0;
        float cost = 0.0f, rate2 = 0.0f;
        const int kind = (active && usable) ? scen_step(sys, s, a, rates[(size_t)l * S + s], sized, pm.rateStar, reps, cost, rate2, rec)
                                            : WVA_SCEN_NIL;
        bool ok = kind == WVA_SCEN_ZERO;
        // Analyze's range checks (queueanalyzer.go:135-143), as k_pairs_warp
        const bool need = kind == WVA_SCEN_RATE && !(rate2 <= 0.0f || rate2 > pm.wp.rateMax);
        // lanes with the same rate2 share one evaluation: every positive scenario of a TPS-target server has the same
        const unsigned long long key = need ? (unsigned long long)__float_as_uint(rate2) : (0x100000000ull | (unsigned)lane);
        const int leader = __ffs(__match_any_sync(0xffffffffu, key)) - 1;
        const bool eval = need && leader == lane;
        if (__any_sync(0xffffffffu, eval)) {
            SolveStats st;
            st.rho = st.avgNumInServers = st.avgNumInSystem = st.throughput = st.avgRespTime = st.avgServTime = st.avgWaitTime = 0.0f;
            bool v = false, uu;
            const bool solved = warp_solve(pm.wp, eval, rate2 / 1000.0f, st, steps, v, false, uu);
            if (__any_sync(0xffffffffu, eval && !solved)) { toSlow = true; break; }
            st = shfl_stats(st, leader);
            v = __shfl_sync(0xffffffffu, (int)v, leader);
            if (need && v) {
                wva_metrics m2; metrics_from(pm.wp, st, m2);
                rec = scen_alloc(a, pm.wp.N, reps, cost, pm.rateStar, m2);
                ok = true;
            }
        }
        if (active) scen_store(sys, s, recs, feasible, (size_t)l * SA + gi, ok, rec);
    }
    if (toSlow && lane == 0) list[atomicAdd(list_count, 1)] = pid;
}

// k_queue_size inputs of the listed pairs (list == nullptr: every shard pair): CreateAllocation's configuration
// {N, 10 N, alpha, beta, gamma, delta, in, out} and the server's {TTFT, ITL, TPS}.  A pair that needs no Size (not
// usable, no output tokens, no positive scenario rate) gets N = 0: k_queue_size then fails its configuration check
// without running anything.
__global__ void k_scen_gather(DevSystem sys, int s0, const int* __restrict__ list, int n, int L, const float* __restrict__ rates,
                              wva_queue_config* __restrict__ cfg, float* __restrict__ target) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int pid = list ? list[t] : t;
    const int s = s0 + pid / sys.A, a = pid % sys.A;
    wva_queue_config c;
    c.max_batch_size = 0; c.max_queue_size = 0;
    c.alpha = c.beta = c.gamma = c.delta = 0.0f;
    c.avg_input_tokens = sys.srv_in_tokens[s]; c.avg_output_tokens = sys.srv_out_tokens[s];
    if (scen_pair_usable(sys, s, a) && sys.srv_out_tokens[s] != 0 && scen_any_positive(rates, L, sys.S, s, 0, 1)) {
        const size_t pi = (size_t)sys.srv_model[s] * sys.A + a;
        const long long N = scen_batch(sys, s, a);
        c.max_batch_size = (int)N; c.max_queue_size = (int)go_muli(N, WVA_MAX_QUEUE_TO_BATCH_RATIO);
        c.alpha = sys.perf_alpha[pi]; c.beta = sys.perf_beta[pi]; c.gamma = sys.perf_gamma[pi]; c.delta = sys.perf_delta[pi];
    }
    cfg[t] = c;
    target[3 * t] = sys.srv_slo_ttft[s]; target[3 * t + 1] = sys.srv_slo_itl[s]; target[3 * t + 2] = sys.srv_slo_tps[s];
}

// k_queue_analyze inputs, one row per (listed pair t, scenario l) at t*L + l: the pair's configuration and rate2 where
// the scenario reaches the trailing Analyze, else N = 0 (configuration check fails, nothing runs)
__global__ void k_scen_rows(DevSystem sys, int s0, const int* __restrict__ list, int n, int L, const float* __restrict__ rates,
                            const wva_queue_config* __restrict__ cfg, const wva_metrics* __restrict__ qmetrics,
                            const unsigned char* __restrict__ qstatus, wva_queue_config* __restrict__ rcfg, float* __restrict__ rrate) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)n * L) return;
    const int t = (int)(idx / L), l = (int)(idx % L);
    const int pid = list ? list[t] : t;
    const int s = s0 + pid / sys.A, a = pid % sys.A;
    AllocRec rec;
    long long reps = 0;
    float cost = 0.0f, rate2 = 0.0f;
    const int kind = scen_pair_usable(sys, s, a)
                         ? scen_step(sys, s, a, rates[(size_t)l * sys.S + s], qstatus[t] == 0, qmetrics[t].throughput, reps, cost, rate2, rec)
                         : WVA_SCEN_NIL;
    wva_queue_config c = cfg[t];
    if (kind != WVA_SCEN_RATE) c.max_batch_size = 0;
    rcfg[idx] = c;
    rrate[idx] = kind == WVA_SCEN_RATE ? rate2 : 0.0f;
}

// the records of the listed pairs from their Size (qmetrics / qstatus per pair) and Analyze rows (ametrics / astatus)
__global__ void k_scen_scatter(DevSystem sys, int s0, const int* __restrict__ list, int n, int L, const float* __restrict__ rates,
                               const wva_queue_config* __restrict__ cfg, const wva_metrics* __restrict__ qmetrics,
                               const unsigned char* __restrict__ qstatus, const wva_metrics* __restrict__ ametrics,
                               const unsigned char* __restrict__ astatus, DevAllocs recs, unsigned char* __restrict__ feasible) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)n * L) return;
    const int t = (int)(idx / L), l = (int)(idx % L);
    const int pid = list ? list[t] : t;
    const int s = s0 + pid / sys.A, a = pid % sys.A;
    AllocRec rec = empty_alloc();
    long long reps = 0;
    float cost = 0.0f, rate2 = 0.0f;
    const float rateStar = qmetrics[t].throughput;
    const int kind = scen_pair_usable(sys, s, a)
                         ? scen_step(sys, s, a, rates[(size_t)l * sys.S + s], qstatus[t] == 0, rateStar, reps, cost, rate2, rec)
                         : WVA_SCEN_NIL;
    bool ok = kind == WVA_SCEN_ZERO;
    if (kind == WVA_SCEN_RATE && astatus[idx] == WVA_CAND_OK) {
        rec = scen_alloc(a, cfg[t].max_batch_size, reps, cost, rateStar, ametrics[idx]);
        ok = true;
    }
    scen_store(sys, s, recs, feasible, (size_t)l * sys.S * sys.A + (size_t)s * sys.A + a, ok, rec);
}

// N per pair (0 = no queueing work) — used to order pairs by chain length and to size scratch.
__global__ void k_pair_batch(DevSystem sys, int s0, int nPairs, long long* __restrict__ nOut) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nPairs) return;
    nOut[t] = pair_batch_size(sys, s0 + t / sys.A, t % sys.A);
}
// bucket = position of the highest set bit of N (0 for N == 0): 0..63
__global__ void k_pair_bucket_hist(const long long* __restrict__ nIn, int nPairs, int* __restrict__ hist) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nPairs) return;
    long long n = nIn[t];
    int b = n <= 0 ? 0 : (64 - __clzll(n));
    atomicAdd(&hist[b], 1);
}
// scatter pair ids into descending-bucket order (heaviest first); order within a bucket is free
__global__ void k_pair_bucket_scatter(const long long* __restrict__ nIn, int nPairs, int* __restrict__ cursor,
                                      int* __restrict__ order) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nPairs) return;
    long long n = nIn[t];
    int b = n <= 0 ? 0 : (64 - __clzll(n));
    int pos = atomicAdd(&cursor[b], 1);
    order[pos] = t;
}

// ---------------------------------------------------------------------------------------
// Candidate sweep
// ---------------------------------------------------------------------------------------

// best candidate of a block / a list thread: key + the metrics a wva_grid_best needs
struct GridSlot { unsigned long long key; float cost, itl, ttft, rho; int sl; int pad; };
struct ScanRow;

struct GridParams {
    int r_max, b_max;
    int r_chunk, n_rchunks;          // replicas per block / blocks per pair
    int b_seg, n_bseg;               // row kernel: batch sizes per block / blocks per pair
    int s0, ns;                      // shard
    int pair_base;                   // (server, accelerator) pairs of the shard that precede the slice being swept
    wva_metrics* cube;               // [ns*A*r_max*b_max] or nullptr
    unsigned char* status;           // same extent or nullptr
    unsigned long long* keys;        // [ns] per-server argmin key (initialised to ~0)
    unsigned long long* counters;    // [0] steps executed, [1] algorithmic steps, [2] candidates analysed ok
    unsigned long long* slow_list; int* slow_count; int slow_cap;   // candidate ids (relative to shard) needing the literal path
    double2* pair_tab;               // [ns*A][b_max] {rate, refined reciprocal}: written by k_grid, read by the list kernel
    struct GridSlot* block_slot;     // [blocks of k_grid] best candidate of each block with its metrics
    struct GridSlot* list_slot;      // [heavy_cap + slow_cap] one per list-kernel thread
    int tail_cap;                    // tail steps a candidate may take inside k_grid before it is deferred
    unsigned long long* heavy_list; float* heavy_cost; int* heavy_count; int heavy_cap;   // deferred (long) chains
    ScanRow* row_info;               // [slice pairs * r_max] k_scan_prep -> k_scan_cert / k_scan_lean
    float2* rate_tab;                // [slice pairs * b_max] {RateRange.Max, RateTargetTPS} of batch size b (k_scan_prep)
    // per-(server, accelerator) winners (wva_grid_set_pair_winners); pair_keys == nullptr: off
    unsigned long long* pair_keys;   // [ns*A] per-pair argmin key (initialised to ~0), shard-local pair index
    DevAllocs pair_rec;              // [S*A] records written by k_grid_claim (rows of the shard)
    unsigned char* pair_feasible;    // [S*A]
};

// order-preserving map float -> uint32 (ascending), -0 canonicalised by the caller
__device__ __forceinline__ unsigned sortable_f32(float v) {
    unsigned b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float unsortable_f32(unsigned k) {
    unsigned b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
    return __uint_as_float(b);
}
// key = (value, accelerator, replicas, batch) lexicographic
__device__ __forceinline__ unsigned long long make_key(float value, int a, int r, int b) {
    return ((unsigned long long)sortable_f32(value) << 32) | ((unsigned long long)a << 24) |
           ((unsigned long long)(r - 1) << 14) | (unsigned long long)(b - 1);
}
#define WVA_KEY_NONE 0xffffffffffffffffULL
#define WVA_GRID_MAX_A 256
#define WVA_GRID_MAX_R 1024
#define WVA_GRID_MAX_B 8192

// Per-server constants of the sweep, computed once per block
struct GridServer {
    float totalRate;                 // allocation.go:134-139
    float sloTTFT, sloITL, sloTPS;
    long long inTok, outTok;
    int minReplicas;
    int curAcc, curRep; float curCost;
    float accCost; long long numInst;
    ServiceParms sp;
    bool cert;
};

// QueueAnalyzer.Analyze (queueanalyzer.go:134-174) on a fresh analyzer with MaxBatchSize b,
// MaxQueueSize 10 b, service rates from the shared-memory table.  A fresh model has p[0] = 0 so
// the validity test (queuemodel.go:30-31) sees rho = 1: valid iff 1 < K and lambda >= 0.
__device__ __forceinline__ int analyze_table(const ServTable& tb, const GridServer& gs, int b, float rate, bool tame,
                                             int tailCap, wva_metrics& m, float& rateTPS, unsigned long long& steps,
                                             float& deferCost) {
    const int K = b * WVA_MAX_QUEUE_TO_BATCH_RATIO + b;
    const float lambdaMax = tb.rateF[b - 1] * (1.0f - WVA_EPSILON);
    const float rateMax = lambdaMax * 1000.0f;
    const float lamMaxBack = rateMax / 1000.0f;
    rateTPS = (lamMaxBack * (1.0f - WVA_STABILITY_SAFETY)) * 1000.0f;    // TargetRate.RateTargetTPS, :231-234,:246
    if (rate <= 0.0f) return WVA_CAND_ERR_RATE_LE0;
    if (rate > rateMax) return WVA_CAND_ERR_RATE_MAX;
    const float lambda = rate / 1000.0f;
    if ((1.0f >= (float)K) || (lambda < 0.0f)) return WVA_CAND_ERR_MODEL;
    SolveStats st;
    ProvTable pv; pv.rateD = tb.rateD; pv.rcp = tb.rcp; pv.rateF_ = tb.rateF;
    int rc = solve_fast(pv, b, K, lambda, tame, tailCap, st, steps, deferCost, gs.cert);
    if (rc == WVA_SOLVE_DEFER) return -2;                                 // long chain: heavy kernel
    if (rc == WVA_SOLVE_CAREFUL) rc = solve_stream_table(tb, b, K, lambda, tame, st, steps);
    if (rc != WVA_SOLVE_OK) return -1;                                    // literal path
    float effConc = effective_concurrency(st.avgServTime, gs.sp, gs.inTok, gs.outTok, b);
    float rho = st.avgNumInServers / (float)b;
    rho = go_minf(go_maxf(rho, 0.0f), 1.0f);
    m.throughput = st.throughput * 1000.0f;
    m.avg_resp_time = st.avgRespTime;
    m.avg_wait_time = st.avgWaitTime;
    m.avg_num_in_serv = st.avgNumInServers;
    m.avg_prefill_time = prefill_time(gs.sp, gs.inTok, effConc);
    m.avg_token_time = decode_time(gs.sp, effConc);
    m.max_rate = rateMax;
    m.rho = rho;
    return WVA_CAND_OK;
}

// SLO / replica constraints of a candidate and its key (WVA_KEY_NONE when infeasible)
__device__ __forceinline__ unsigned long long candidate_key(const GridServer& gs, int a, int r, int b, float rate,
                                                            float rateTPS, const wva_metrics& m, bool& feasible) {
    const float ttft = m.avg_wait_time + m.avg_prefill_time;
    const float itl = m.avg_token_time;
    feasible = (!(gs.sloTTFT > 0.0f) || ttft <= gs.sloTTFT) && (!(gs.sloITL > 0.0f) || itl <= gs.sloITL) &&
               (!(gs.sloTPS > 0.0f) || rate <= rateTPS) && (r >= gs.minReplicas);
    if (!feasible) return WVA_KEY_NONE;
    const float cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
    float value = transition_penalty(gs.curAcc, gs.curRep, gs.curCost, a, (long long)r, cost);
    value = value + 0.0f;
    if (value != value) return WVA_KEY_NONE;
    return make_key(value, a, r, b);
}

__device__ __forceinline__ void load_grid_server(const DevSystem& sys, int s, int a, GridServer& gs) {
    const int m = sys.srv_model[s];
    const size_t pi = (size_t)m * sys.A + a;
    gs.sp.alpha = sys.perf_alpha[pi]; gs.sp.beta = sys.perf_beta[pi];
    gs.sp.gamma = sys.perf_gamma[pi]; gs.sp.delta = sys.perf_delta[pi];
    gs.inTok = sys.srv_in_tokens[s]; gs.outTok = sys.srv_out_tokens[s];
    gs.sloTTFT = sys.srv_slo_ttft[s]; gs.sloITL = sys.srv_slo_itl[s]; gs.sloTPS = sys.srv_slo_tps[s];
    gs.totalRate = (gs.sloTPS == 0.0f) ? sys.srv_arrival_rpm[s] / 60.0f : gs.sloTPS / (float)gs.outTok;
    gs.minReplicas = sys.srv_min_replicas[s];
    gs.curAcc = sys.srv_cur_acc[s]; gs.curRep = sys.srv_cur_replicas[s]; gs.curCost = sys.srv_cur_cost[s];
    gs.accCost = sys.acc_cost[a];
    gs.numInst = num_instances(sys, m, a);
    gs.cert = sys.cert != 0;
}

// Block = one (server, accelerator) pair x one chunk of replica counts.  The pair's service-rate
// table (float, double and refined reciprocal, 20 B per batch size) is built once into shared
// memory; warps then pull (replicas, 32 consecutive batch sizes) work items from a shared counter:
// lanes of a warp share lambda and differ only by batch size, so their trip counts are close.
// Chains whose tail outlasts gp.tail_cap are deferred to k_grid_list.
#define WVA_GRID_THREADS 256
__global__ void __launch_bounds__(WVA_GRID_THREADS, 3)
k_grid(DevSystem sys, GridParams gp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* rateD = reinterpret_cast<double*>(smem_raw);
    double* rcp = rateD + gp.b_max;
    float* rateF = reinterpret_cast<float*>(rcp + gp.b_max);
    __shared__ int sh_item, sh_nGood;
    __shared__ unsigned long long sh_key;
    __shared__ unsigned long long sh_cnt[3];

    const int pairSlice = blockIdx.x / gp.n_rchunks;       // pair index inside the slice
    const int pairLocal = gp.pair_base + pairSlice;        // (s - s0) * A + a
    const int rchunk = blockIdx.x % gp.n_rchunks;
    const int sl = pairLocal / sys.A, a = pairLocal % sys.A;
    const int s = gp.s0 + sl;
    const int r_lo = rchunk * gp.r_chunk + 1;
    const int r_hi = min(gp.r_max, r_lo + gp.r_chunk - 1);
    const int B = gp.b_max;
    const int lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        sh_item = 0; sh_nGood = B; sh_key = WVA_KEY_NONE; sh_cnt[0] = sh_cnt[1] = sh_cnt[2] = 0;
        gp.block_slot[blockIdx.x].key = WVA_KEY_NONE;
    }

    const bool pairOk = pair_lookups_ok(sys, s, a) && is_candidate_accel(sys, s, a);
    GridServer gs;
    int blockStatus = WVA_CAND_OK;
    if (!pairOk) blockStatus = WVA_CAND_ERR_PAIR;
    else {
        load_grid_server(sys, s, a, gs);
        if (gs.inTok < 0 || gs.outTok < 1 || gs.sloTTFT < 0.0f || gs.sloITL < 0.0f || gs.sloTPS < 0.0f)
            blockStatus = WVA_CAND_ERR_CONFIG;
    }
    const size_t candBase = ((size_t)pairLocal * gp.r_max) * (size_t)B;
    if (blockStatus != WVA_CAND_OK) {
        // whole block shares one error status; zero metrics
        if (gp.status || gp.cube) {
            const size_t n = (size_t)(r_hi - r_lo + 1) * B;
            const size_t off = candBase + (size_t)(r_lo - 1) * B;
            for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
                if (gp.status) gp.status[off + i] = (unsigned char)blockStatus;
                if (gp.cube) { float4 z = make_float4(0, 0, 0, 0); float4* c = reinterpret_cast<float4*>(&gp.cube[off + i]); c[0] = z; c[1] = z; }
            }
        }
        return;
    }
    __syncthreads();

    // ---- stage the service-rate table (and publish it for the deferred-chain kernel) ------------
    ServFormula sf; sf.init(gs.sp, gs.inTok, gs.outTok);
    double2* gtab = (rchunk == 0) ? gp.pair_tab + (size_t)pairSlice * B : nullptr;
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
        float r = sf.rate(i + 1);
        rateF[i] = r;
        double d = (double)r;
        double y = rcp_refined(d);
        rateD[i] = d;
        rcp[i] = y;
        if (gtab) gtab[i] = make_double2(d, y);
        if (!(r > 0.0f) || !(r < CUDART_INF_F)) atomicMin(&sh_nGood, i);
    }
    const bool tame = tame_parms(gs.sp, gs.inTok, gs.outTok);
    __syncthreads();
    ServTable tb; tb.rateF = rateF; tb.rateD = rateD; tb.rcp = rcp;
    const int nGood = sh_nGood;

    // ---- sweep ------------------------------------------------------------------------------
    const int bChunks = (B + 31) / 32;
    const int nItems = (r_hi - r_lo + 1) * bChunks;
    unsigned long long bestKey = WVA_KEY_NONE;
    float bestItl = 0.0f, bestTtft = 0.0f, bestRho = 0.0f;
    unsigned long long steps = 0, algSteps = 0, okCount = 0;
    for (;;) {
        int item;
        if (lane == 0) item = atomicAdd(&sh_item, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= nItems) break;
        // heaviest items first: large batch sizes have the longest ramps
        const int bc = bChunks - 1 - (item % bChunks);
        const int r = r_lo + item / bChunks;
        const int b = bc * 32 + lane + 1;
        if (b > B) continue;
        const size_t ci = candBase + (size_t)(r - 1) * B + (size_t)(b - 1);
        const float rate = gs.totalRate / (float)r;
        wva_metrics m;
        m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
        m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
        float rateTPS = 0.0f;
        int st;
        bool feasible = false;
        float deferCost = 0.0f;
        bool deferred = false;
        if (b > nGood) st = -1;
        else {
            // one call site: the second trip (cap 0) only happens when the deferred list is full
            // short chains (K <= 1024) never leave this kernel: deferral only pays for long tails
            for (int cap = (11 * b <= 1024) ? 0 : gp.tail_cap;; cap = 0) {
                st = analyze_table(tb, gs, b, rate, tame, cap, m, rateTPS, steps, deferCost);
                if (st != -2) break;
                int k = atomicAdd(gp.heavy_count, 1);
                if (k < gp.heavy_cap) { gp.heavy_list[k] = (unsigned long long)ci; gp.heavy_cost[k] = deferCost; deferred = true; break; }
            }
        }
        if (deferred) continue;      // long chain: k_grid_list groups chains of similar length
        if (st == -1) {
            // literal path: queue the candidate, outputs come from k_grid_list
            int k = atomicAdd(gp.slow_count, 1);
            if (k < gp.slow_cap) gp.slow_list[k] = (unsigned long long)ci;
            continue;
        }
        if (st == WVA_CAND_OK) {
            okCount++;
            algSteps += 2ULL * (unsigned long long)(11 * b + 1);
            unsigned long long key = candidate_key(gs, a, r, b, rate, rateTPS, m, feasible);
            if (key < bestKey) {
                bestKey = key; bestItl = m.avg_token_time; bestTtft = m.avg_wait_time + m.avg_prefill_time; bestRho = m.rho;
            }
        } else {
            m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
            m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
        }
        if (gp.cube) {
            float4* c = reinterpret_cast<float4*>(&gp.cube[ci]);
            c[0] = make_float4(m.throughput, m.avg_resp_time, m.avg_wait_time, m.avg_num_in_serv);
            c[1] = make_float4(m.avg_prefill_time, m.avg_token_time, m.max_rate, m.rho);
        }
        if (gp.status) gp.status[ci] = (unsigned char)(st | (feasible ? WVA_CAND_FEASIBLE : 0));
    }

    // ---- warp-shuffle then block argmin; the owner of the block minimum publishes its metrics ----
    unsigned long long warpKey = bestKey;
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long other = __shfl_down_sync(0xffffffffu, warpKey, o);
        if (other < warpKey) warpKey = other;
        steps += __shfl_down_sync(0xffffffffu, steps, o);
        algSteps += __shfl_down_sync(0xffffffffu, algSteps, o);
        okCount += __shfl_down_sync(0xffffffffu, okCount, o);
    }
    if (lane == 0) {
        if (warpKey != WVA_KEY_NONE) atomicMin(&sh_key, warpKey);
        atomicAdd(&sh_cnt[0], steps); atomicAdd(&sh_cnt[1], algSteps); atomicAdd(&sh_cnt[2], okCount);
    }
    __syncthreads();
    const unsigned long long blockKey = sh_key;
    if (blockKey != WVA_KEY_NONE && bestKey == blockKey) {          // keys are unique per candidate: one owner
        GridSlot sl_; sl_.key = blockKey; sl_.itl = bestItl; sl_.ttft = bestTtft; sl_.rho = bestRho; sl_.sl = sl; sl_.pad = 0;
        const int r = (int)((blockKey >> 14) & 0x3ff) + 1;
        sl_.cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
        gp.block_slot[blockIdx.x] = sl_;
        atomicMin(&gp.keys[sl], blockKey);
        if (gp.pair_keys) atomicMin(&gp.pair_keys[gp.pair_base + (int)(blockIdx.x / (unsigned)gp.n_rchunks)], blockKey);   // a block covers one pair (index re-derived: no register live across the sweep)
    }
    if (threadIdx.x == 0) {
        atomicAdd(&gp.counters[0], sh_cnt[0]); atomicAdd(&gp.counters[1], sh_cnt[1]); atomicAdd(&gp.counters[2], sh_cnt[2]);
    }
}

// ---------------------------------------------------------------------------------------
// k_grid_rows: the sweep with ONE THREAD PER ROW (server, accelerator, replicas).
//
// All candidates of a row share lambda = totalRate / r, and the chain of batch size b uses
// servRate[min(n, b-1)]: its first b steps are the first b steps of the chain of every larger batch
// size.  So a row needs ONE ramp p[1..B]; candidate b is evaluated at the moment the ramp reaches state b,
// from (p[b], sum_{i<=b} p[i], sum_{i<=b} i p[i]) and the certified closed-form tail (cert_eval) — O(1) per
// candidate instead of O(b) + tail.  When the ramp itself dies out (p[n] below 2^-68 of every aggregate
// with all later ratios <= 0.998), the remaining candidates of the row share the frozen sums.
// A candidate whose certificate fails (ambiguous float32 rounding, ill-conditioned closed form, value
// window left) is appended to the deferred list and evaluated by the exact chain in k_grid_list.
// Lanes of a warp hold consecutive r of the same pair: they step n together, so the shared-memory
// table reads are broadcasts.
// Small shards have too few rows to fill the machine: a pair is then split over n_bseg blocks, block
// `seg` evaluating the batch sizes (seg*b_seg, (seg+1)*b_seg] of every row after running the ramp up
// to seg*b_seg without evaluating anything (the ramp is a few instructions per step, a candidate a
// few hundred).
// ---------------------------------------------------------------------------------------
#define WVA_ROWS_THREADS 32
__global__ void __launch_bounds__(WVA_ROWS_THREADS, 16)
k_grid_rows(DevSystem sys, GridParams gp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* rateD = reinterpret_cast<double*>(smem_raw);
    double* rcp = rateD + gp.b_max;
    float* rateF = reinterpret_cast<float*>(rcp + gp.b_max);
    __shared__ int sh_nGood;
    __shared__ unsigned long long sh_key;
    __shared__ unsigned long long sh_cnt[3];

    const int pairSlice = blockIdx.x / gp.n_bseg, seg = blockIdx.x % gp.n_bseg;
    const int pairLocal = gp.pair_base + pairSlice;
    const int sl = pairLocal / sys.A, a = pairLocal % sys.A;
    const int s = gp.s0 + sl;
    const int B = gp.b_max, R = gp.r_max;
    const int b0 = seg * gp.b_seg;                                   // this block: states b0+1 .. b1
    const int b1 = (b0 + gp.b_seg < B) ? b0 + gp.b_seg : B;
    const int lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        sh_nGood = b1; sh_key = WVA_KEY_NONE; sh_cnt[0] = sh_cnt[1] = sh_cnt[2] = 0;
        gp.block_slot[blockIdx.x].key = WVA_KEY_NONE;
    }
    const bool pairOk = pair_lookups_ok(sys, s, a) && is_candidate_accel(sys, s, a);
    GridServer gs;
    int blockStatus = WVA_CAND_OK;
    if (!pairOk) blockStatus = WVA_CAND_ERR_PAIR;
    else {
        load_grid_server(sys, s, a, gs);
        if (gs.inTok < 0 || gs.outTok < 1 || gs.sloTTFT < 0.0f || gs.sloITL < 0.0f || gs.sloTPS < 0.0f)
            blockStatus = WVA_CAND_ERR_CONFIG;
    }
    const size_t candBase = ((size_t)pairLocal * R) * (size_t)B;
    if (blockStatus != WVA_CAND_OK) {
        if (gp.status || gp.cube) {
            const int w = b1 - b0;
            const size_t n = (size_t)R * w;
            for (size_t j = threadIdx.x; j < n; j += blockDim.x) {
                const size_t i = (j / w) * (size_t)B + (size_t)b0 + (j % w);
                if (gp.status) gp.status[candBase + i] = (unsigned char)blockStatus;
                if (gp.cube) { float4 z = make_float4(0, 0, 0, 0); float4* c = reinterpret_cast<float4*>(&gp.cube[candBase + i]); c[0] = z; c[1] = z; }
            }
        }
        return;
    }
    __syncthreads();
    ServFormula sf; sf.init(gs.sp, gs.inTok, gs.outTok);
    double2* gtab = gp.pair_tab + (size_t)pairSlice * B;
    for (int i = threadIdx.x; i < b1; i += blockDim.x) {
        float r = sf.rate(i + 1);
        rateF[i] = r;
        double d = (double)r;
        double y = rcp_refined(d);
        rateD[i] = d; rcp[i] = y;
        if (i >= b0) gtab[i] = make_double2(d, y);                  // each block publishes its own part
        if (!(r > 0.0f) || !(r < CUDART_INF_F)) atomicMin(&sh_nGood, i);
    }
    const bool tame = tame_parms(gs.sp, gs.inTok, gs.outTok);
    __syncthreads();
    const int nGood = sh_nGood;

    unsigned long long bestKey = WVA_KEY_NONE;
    float bestItl = 0.0f, bestTtft = 0.0f, bestRho = 0.0f;
    unsigned long long steps = 0, algSteps = 0, okCount = 0;

    for (int r = threadIdx.x + 1; r <= R; r += blockDim.x) {
        const float rate = gs.totalRate / (float)r;
        const float lambda = rate / 1000.0f;
        double lam = (double)lambda;
        const bool lamOk = (lam >= 0x1p-100 && lam <= 0x1p20);
        lam = pin(lam);
        const float cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
        float value = transition_penalty(gs.curAcc, gs.curRep, gs.curCost, a, (long long)r, cost);
        value = value + 0.0f;
        // shared ramp state
        double p = 1.0, sum = 1.0, uN = 0.0, dn = 0.0;
        double exInSys = 0.0, exSumP = 0.0;     // exact normalised sums of a stopped row
        unsigned thrHi = 0u, hmin = 0x3ff00000u;
        bool stopped = false;        // ramp died out: sums frozen
        bool broken = !lamOk;        // chain left the value window (or bad table entry): rest of the row goes to the exact kernels
        const size_t rowBase = candBase + (size_t)(r - 1) * B;
        for (int n = 0; n < b1; ++n) {
            const int b = n + 1;
            // ---- one step of the shared ramp: state b ----
            if (!stopped && !broken) {
                if (b > nGood) broken = true;
                else {
                    const double t = p * lam;
                    const double pn = div_core(t, rateD[n], rcp[n]);
                    const unsigned hq = (unsigned)__double2hiint(pn);
                    if (hq - WVA_WIN_LO >= WVA_WIN_SPAN) broken = true;
                    else {
                        sum += pn; dn += 1.0; uN += dn * pn; p = pn;
                        ++steps;
                        if (n == 0 && pn >= 0x1p-400)      // 2^-68 min(1,p1) / K_max: the neglected mass is < 2^-58 of every aggregate
                            thrHi = (unsigned)__double2hiint((0x1p-68 * fmin(1.0, pn)) / (double)(11 * B));
                        hmin = hq < hmin ? hq : hmin;
                        if (hq < thrHi && tame && lambda <= 0.998f * rateF[n] && sum <= 0x1p400) {
                            // The chain has died out (solve_stream's truncation rule with a 2^10 stricter threshold):
                            // every candidate b >= this state sees the SAME normalised prefix, exactly.  Run the
                            // reference's second pass once for the row (mm1modelstatedependent.go:49-55 up to here).
                            stopped = true;
                            const double S = sum;
                            if ((int)(hmin >> 20) - (int)((unsigned)__double2hiint(S) >> 20) < -1000) broken = true;
                            else {
                                const double yS = rcp_refined(S);
                                double q = div_core(1.0, S, yS), pp = 1.0, di = 0.0;
                                exSumP = q; exInSys = 0.0;
                                for (int i = 1; i <= b; ++i) {
                                    pp = div_core(pp * lam, rateD[i - 1], rcp[i - 1]);
                                    q = div_core(pp, S, yS);
                                    di += 1.0;
                                    exInSys += di * q;
                                    exSumP += q;
                                }
                                steps += (unsigned long long)b;
                            }
                        }
                    }
                }
            }
            // ---- candidate (r, b) ----
            if (n < b0) continue;                                    // another block's batch sizes
            const size_t ci = rowBase + (size_t)n;
            const int K = 11 * b;
            const float lambdaMax = rateF[n] * (1.0f - WVA_EPSILON);
            const float rateMax = lambdaMax * 1000.0f;
            int st;
            bool feasible = false;
            wva_metrics m;
            m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
            m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
            if (b > nGood) {                                   // bad table entry: literal path decides
                int k = atomicAdd(gp.slow_count, 1);
                if (k < gp.slow_cap) gp.slow_list[k] = (unsigned long long)ci;
                continue;
            }
            if (rate <= 0.0f) st = WVA_CAND_ERR_RATE_LE0;
            else if (rate > rateMax) st = WVA_CAND_ERR_RATE_MAX;
            else if (lambda < 0.0f) st = WVA_CAND_ERR_MODEL;
            else {
                SolveStats so;
                bool certified = false;
                if (!broken) {
                    if (stopped) {
                        // exact: avgNumInServers is captured at i == b (mm1modelstatedependent.go:52-54) from sums that no
                        // longer change; float32(p[K]) < 2^-58 so throughput == lambda
                        const double inServ = exInSys + (1.0 - exSumP) * (double)b;
                        finish_stats(so, lambda, inServ, exInSys, 0.0f);
                        certified = true;
                    } else {
                        CertIn c; c.pN = p; c.sumRamp = sum; c.uN = uN; c.lam = lam; c.sTail = rateD[n]; c.N = b; c.K = K; c.lambda = lambda;
                        certified = cert_eval(c, so);
                    }
                }
                if (!certified) {
                    // exact chain in k_grid_list; when that list is full, right here
                    int k = atomicAdd(gp.heavy_count, 1);
                    if (k < gp.heavy_cap) { gp.heavy_list[k] = (unsigned long long)ci; gp.heavy_cost[k] = (float)K; continue; }
                    ServTable tb; tb.rateF = rateF; tb.rateD = rateD; tb.rcp = rcp;
                    float rt, dc;
                    int st2 = analyze_table(tb, gs, b, rate, tame, 0, m, rt, steps, dc);
                    if (st2 < 0) { int k2 = atomicAdd(gp.slow_count, 1); if (k2 < gp.slow_cap) gp.slow_list[k2] = (unsigned long long)ci; continue; }
                    so.avgServTime = 0.0f;      // metrics already final in m
                    st = st2;
                    goto have_metrics;
                }
                st = WVA_CAND_OK;
                {
                    const float effConc = effective_concurrency(so.avgServTime, gs.sp, gs.inTok, gs.outTok, b);
                    float rho = so.avgNumInServers / (float)b;
                    rho = go_minf(go_maxf(rho, 0.0f), 1.0f);
                    m.throughput = so.throughput * 1000.0f;
                    m.avg_resp_time = so.avgRespTime;
                    m.avg_wait_time = so.avgWaitTime;
                    m.avg_num_in_serv = so.avgNumInServers;
                    m.avg_prefill_time = prefill_time(gs.sp, gs.inTok, effConc);
                    m.avg_token_time = decode_time(gs.sp, effConc);
                    m.max_rate = rateMax;
                    m.rho = rho;
                }
            have_metrics:
                if (st != WVA_CAND_OK) {
                    m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
                    m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
                    goto write_out;
                }
                okCount++;
                algSteps += 2ULL * (unsigned long long)(K + 1);
                const float lamMaxBack = rateMax / 1000.0f;
                const float rateTPS = (lamMaxBack * (1.0f - WVA_STABILITY_SAFETY)) * 1000.0f;
                const float ttft = m.avg_wait_time + m.avg_prefill_time;
                const float itl = m.avg_token_time;
                feasible = (!(gs.sloTTFT > 0.0f) || ttft <= gs.sloTTFT) && (!(gs.sloITL > 0.0f) || itl <= gs.sloITL) &&
                           (!(gs.sloTPS > 0.0f) || rate <= rateTPS) && (r >= gs.minReplicas);
                if (feasible && value == value) {              // a NaN value is never selected
                    const unsigned long long key = make_key(value, a, r, b);
                    if (key < bestKey) { bestKey = key; bestItl = itl; bestTtft = ttft; bestRho = m.rho; }
                }
            }
        write_out:
            if (gp.cube) {
                float4* c = reinterpret_cast<float4*>(&gp.cube[ci]);
                c[0] = make_float4(m.throughput, m.avg_resp_time, m.avg_wait_time, m.avg_num_in_serv);
                c[1] = make_float4(m.avg_prefill_time, m.avg_token_time, m.max_rate, m.rho);
            }
            if (gp.status) gp.status[ci] = (unsigned char)(st | (feasible ? WVA_CAND_FEASIBLE : 0));
        }
    }
    // ---- block argmin + counters ------------------------------------------------------------------
    unsigned long long warpKey = bestKey;
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long other = __shfl_down_sync(0xffffffffu, warpKey, o);
        if (other < warpKey) warpKey = other;
        steps += __shfl_down_sync(0xffffffffu, steps, o);
        algSteps += __shfl_down_sync(0xffffffffu, algSteps, o);
        okCount += __shfl_down_sync(0xffffffffu, okCount, o);
    }
    if (lane == 0) {
        if (warpKey != WVA_KEY_NONE) atomicMin(&sh_key, warpKey);
        atomicAdd(&sh_cnt[0], steps); atomicAdd(&sh_cnt[1], algSteps); atomicAdd(&sh_cnt[2], okCount);
    }
    __syncthreads();
    const unsigned long long blockKey = sh_key;
    if (blockKey != WVA_KEY_NONE && bestKey == blockKey) {
        GridSlot sl_; sl_.key = blockKey; sl_.itl = bestItl; sl_.ttft = bestTtft; sl_.rho = bestRho; sl_.sl = sl; sl_.pad = 0;
        const int r = (int)((blockKey >> 14) & 0x3ff) + 1;
        sl_.cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
        gp.block_slot[blockIdx.x] = sl_;
        atomicMin(&gp.keys[sl], blockKey);
        if (gp.pair_keys) atomicMin(&gp.pair_keys[gp.pair_base + (int)(blockIdx.x / (unsigned)gp.n_bseg)], blockKey);   // a block covers one pair (index re-derived: no register live across the sweep)
    }
    if (threadIdx.x == 0) {
        atomicAdd(&gp.counters[0], sh_cnt[0]); atomicAdd(&gp.counters[1], sh_cnt[1]); atomicAdd(&gp.counters[2], sh_cnt[2]);
    }
}

// ---------------------------------------------------------------------------------------
// k_grid_wrow: the sweep with ONE WARP PER ROW (server, accelerator, replicas) -- shards too small for
// one thread per row.  As in k_grid_rows the row's candidates share one ramp; here all 32 lanes run
// it in lockstep (same values in every lane) and lane l keeps the state (p[b], sum, sum i p[i]) of
// its own batch size b = 32 c + l + 1; after every 32 steps the lanes evaluate their 32 candidates
// together (certified closed-form tail, or the row's frozen exact sums once the ramp has died out).
// Against one thread per candidate (k_grid) a row costs one ramp of B steps instead of one per
// 32-candidate item (B/32 ramps of growing length).  A candidate whose certificate fails needs the
// exact chain (2 x 11 b dependent steps); such candidates cluster -- the aggregates of one row
// converge as b grows, so if the limit sits on a float32 rounding boundary every large b of that row
// is ambiguous -- hence they are not run where they are found (one warp would run them one after the
// other) but deferred to the list kernels, which spread them over the whole GPU (k_grid_list_warp:
// one warp per chain).  Should that list be full, a block-local list is evaluated by the block's
// warps afterwards.
// Block = (pair, chunk of replica counts); warps pull rows from a shared counter.
// ---------------------------------------------------------------------------------------
#define WVA_WROW_LIST 2048
__global__ void __launch_bounds__(WVA_GRID_THREADS, 2)
k_grid_wrow(DevSystem sys, GridParams gp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* rateD = reinterpret_cast<double*>(smem_raw);
    double* rcp = rateD + gp.b_max;
    float* rateF = reinterpret_cast<float*>(rcp + gp.b_max);
    __shared__ int sh_item, sh_nGood;
    __shared__ int sh_hcount, sh_hnext;
    __shared__ int sh_heavy[WVA_WROW_LIST];            // (r - r_lo) * B + (b - 1) of the candidates that need the exact chain
    __shared__ unsigned long long sh_key;
    __shared__ unsigned long long sh_cnt[3];

    const int pairSlice = blockIdx.x / gp.n_rchunks;
    const int pairLocal = gp.pair_base + pairSlice;
    const int rchunk = blockIdx.x % gp.n_rchunks;
    const int sl = pairLocal / sys.A, a = pairLocal % sys.A;
    const int s = gp.s0 + sl;
    const int r_lo = rchunk * gp.r_chunk + 1;
    const int r_hi = min(gp.r_max, r_lo + gp.r_chunk - 1);
    const int B = gp.b_max;
    const int lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        sh_item = 0; sh_nGood = B; sh_key = WVA_KEY_NONE; sh_cnt[0] = sh_cnt[1] = sh_cnt[2] = 0;
        sh_hcount = 0; sh_hnext = 0;
        gp.block_slot[blockIdx.x].key = WVA_KEY_NONE;
    }
    const bool pairOk = pair_lookups_ok(sys, s, a) && is_candidate_accel(sys, s, a);
    GridServer gs;
    int blockStatus = WVA_CAND_OK;
    if (!pairOk) blockStatus = WVA_CAND_ERR_PAIR;
    else {
        load_grid_server(sys, s, a, gs);
        if (gs.inTok < 0 || gs.outTok < 1 || gs.sloTTFT < 0.0f || gs.sloITL < 0.0f || gs.sloTPS < 0.0f)
            blockStatus = WVA_CAND_ERR_CONFIG;
    }
    const size_t candBase = ((size_t)pairLocal * gp.r_max) * (size_t)B;
    if (blockStatus != WVA_CAND_OK) {
        if (gp.status || gp.cube) {
            const size_t n = (size_t)(r_hi - r_lo + 1) * B;
            const size_t off = candBase + (size_t)(r_lo - 1) * B;
            for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
                if (gp.status) gp.status[off + i] = (unsigned char)blockStatus;
                if (gp.cube) { float4 z = make_float4(0, 0, 0, 0); float4* c = reinterpret_cast<float4*>(&gp.cube[off + i]); c[0] = z; c[1] = z; }
            }
        }
        return;
    }
    __syncthreads();
    ServFormula sf; sf.init(gs.sp, gs.inTok, gs.outTok);
    double2* gtab = (rchunk == 0) ? gp.pair_tab + (size_t)pairSlice * B : nullptr;
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
        float r = sf.rate(i + 1);
        rateF[i] = r;
        double d = (double)r;
        double y = rcp_refined(d);
        rateD[i] = d; rcp[i] = y;
        if (gtab) gtab[i] = make_double2(d, y);
        if (!(r > 0.0f) || !(r < CUDART_INF_F)) atomicMin(&sh_nGood, i);
    }
    const bool tame = tame_parms(gs.sp, gs.inTok, gs.outTok);
    __syncthreads();
    ServTable tb; tb.rateF = rateF; tb.rateD = rateD; tb.rcp = rcp;
    const int nGood = sh_nGood;

    const int nRows = r_hi - r_lo + 1;
    unsigned long long bestKey = WVA_KEY_NONE;
    float bestItl = 0.0f, bestTtft = 0.0f, bestRho = 0.0f;
    unsigned long long steps = 0, algSteps = 0, okCount = 0;
    for (;;) {
        int item;
        if (lane == 0) item = atomicAdd(&sh_item, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= nRows) break;
        const int r = r_lo + item;
        const float rate = gs.totalRate / (float)r;
        const float lambda = rate / 1000.0f;
        double lam = (double)lambda;
        const bool lamOk = (lam >= 0x1p-100 && lam <= 0x1p20);
        lam = pin(lam);
        const float cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
        float value = transition_penalty(gs.curAcc, gs.curRep, gs.curCost, a, (long long)r, cost);
        value = value + 0.0f;
        // shared ramp state (identical in all lanes)
        double p = 1.0, sum = 1.0, uN = 0.0, dn = 0.0;
        double exInSys = 0.0, exSumP = 0.0;     // exact normalised sums of a stopped row
        unsigned thrHi = 0u, hmin = 0x3ff00000u;
        bool stopped = false;        // ramp died out: sums frozen
        bool broken = !lamOk;        // chain left the value window (or bad table entry)
        const size_t rowBase = candBase + (size_t)(r - 1) * B;
        for (int n0 = 0; n0 < B; n0 += 32) {
            // ---- 32 steps of the shared ramp; lane l keeps the state after step n0 + l ----
            double cP = 1.0, cSum = 1.0, cUN = 0.0;
            bool cStopped = false, cBroken = true;
            const int nEnd = (n0 + 32 < B) ? n0 + 32 : B;
            for (int n = n0; n < nEnd; ++n) {
                // four steps at once while nothing special can happen in them (see ramp_run): all quotients
                // inside the division window and none below the die-out threshold
                if (!stopped && !broken && n > 0 && n + 4 <= nEnd && n + 4 <= nGood) {
                    const double p1 = div_core(p * lam, rateD[n], rcp[n]);
                    const double p2 = div_core(p1 * lam, rateD[n + 1], rcp[n + 1]);
                    const double p3 = div_core(p2 * lam, rateD[n + 2], rcp[n + 2]);
                    const double p4 = div_core(p3 * lam, rateD[n + 3], rcp[n + 3]);
                    const unsigned h1 = (unsigned)__double2hiint(p1), h2 = (unsigned)__double2hiint(p2);
                    const unsigned h3 = (unsigned)__double2hiint(p3), h4 = (unsigned)__double2hiint(p4);
                    const unsigned wmax = max(max(h1 - WVA_WIN_LO, h2 - WVA_WIN_LO), max(h3 - WVA_WIN_LO, h4 - WVA_WIN_LO));
                    const unsigned hm = min(min(h1, h2), min(h3, h4));
                    if (wmax < WVA_WIN_SPAN && !(hm < thrHi && tame)) {
                        const double s1 = sum + p1, s2 = s1 + p2, s3 = s2 + p3, s4 = s3 + p4;
                        const double d1 = dn + 1.0, d2 = d1 + 1.0, d3 = d2 + 1.0, d4 = d3 + 1.0;
                        const double u1 = uN + d1 * p1, u2 = u1 + d2 * p2, u3 = u2 + d3 * p3, u4 = u3 + d4 * p4;
                        const int k = lane - (n - n0);
                        if ((unsigned)k < 4u) {
                            cP = k == 0 ? p1 : (k == 1 ? p2 : (k == 2 ? p3 : p4));
                            cSum = k == 0 ? s1 : (k == 1 ? s2 : (k == 2 ? s3 : s4));
                            cUN = k == 0 ? u1 : (k == 1 ? u2 : (k == 2 ? u3 : u4));
                            cStopped = false; cBroken = false;
                        }
                        p = p4; sum = s4; dn = d4; uN = u4;
                        hmin = hm < hmin ? hm : hmin;
                        if (lane == 0) steps += 4;
                        n += 3;
                        continue;
                    }
                }
                const int b = n + 1;
                if (!stopped && !broken) {
                    if (b > nGood) broken = true;
                    else {
                        const double t = p * lam;
                        const double pn = div_core(t, rateD[n], rcp[n]);
                        const unsigned hq = (unsigned)__double2hiint(pn);
                        if (hq - WVA_WIN_LO >= WVA_WIN_SPAN) broken = true;
                        else {
                            sum += pn; dn += 1.0; uN += dn * pn; p = pn;
                            if (lane == 0) ++steps;
                            if (n == 0 && pn >= 0x1p-400)
                                thrHi = (unsigned)__double2hiint((0x1p-68 * fmin(1.0, pn)) / (double)(11 * B));
                            hmin = hq < hmin ? hq : hmin;
                            if (hq < thrHi && tame && lambda <= 0.998f * rateF[n] && sum <= 0x1p400) {
                                // the chain has died out: one exact second pass for the rest of the row (see k_grid_rows)
                                stopped = true;
                                const double S = sum;
                                if ((int)(hmin >> 20) - (int)((unsigned)__double2hiint(S) >> 20) < -1000) broken = true;
                                else {
                                    const double yS = rcp_refined(S);
                                    double q = div_core(1.0, S, yS), pp = 1.0, di = 0.0;
                                    exSumP = q; exInSys = 0.0;
                                    for (int i = 1; i <= b; ++i) {
                                        pp = div_core(pp * lam, rateD[i - 1], rcp[i - 1]);
                                        q = div_core(pp, S, yS);
                                        di += 1.0;
                                        exInSys += di * q;
                                        exSumP += q;
                                    }
                                    if (lane == 0) steps += (unsigned long long)b;
                                }
                            }
                        }
                    }
                }
                if (n - n0 == lane) { cP = p; cSum = sum; cUN = uN; cStopped = stopped; cBroken = broken; }
            }
            // ---- the 32 candidates (r, n0 + lane + 1) ----
            const int n = n0 + lane;
            if (n >= B) continue;
            const int b = n + 1;
            const size_t ci = rowBase + (size_t)n;
            const int K = 11 * b;
            const float lambdaMax = rateF[n] * (1.0f - WVA_EPSILON);
            const float rateMax = lambdaMax * 1000.0f;
            int st;
            bool feasible = false;
            wva_metrics m;
            m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
            m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
            if (b > nGood) {                                   // bad table entry: literal path decides
                int k = atomicAdd(gp.slow_count, 1);
                if (k < gp.slow_cap) gp.slow_list[k] = (unsigned long long)ci;
                continue;
            }
            if (rate <= 0.0f) st = WVA_CAND_ERR_RATE_LE0;
            else if (rate > rateMax) st = WVA_CAND_ERR_RATE_MAX;
            else if (lambda < 0.0f) st = WVA_CAND_ERR_MODEL;
            else {
                SolveStats so;
                bool certified = false;
                if (!cBroken) {
                    if (cStopped) {
                        const double inServ = exInSys + (1.0 - exSumP) * (double)b;
                        finish_stats(so, lambda, inServ, exInSys, 0.0f);
                        certified = true;
                    } else {
                        CertIn c; c.pN = cP; c.sumRamp = cSum; c.uN = cUN; c.lam = lam; c.sTail = rateD[n]; c.N = b; c.K = K; c.lambda = lambda;
                        certified = cert_eval(c, so);
                    }
                }
                if (!certified) {
                    // the exact chain: later, by all warps of the block (inline only when the list is full)
                    // the exact chain: in the deferred-chain kernel (one warp per chain, all SMs); only when that
                    // list is full, in this block's own list below
                    {
                        int k = atomicAdd(gp.heavy_count, 1);
                        if (k < gp.heavy_cap) { gp.heavy_list[k] = (unsigned long long)ci; gp.heavy_cost[k] = (float)K; continue; }
                    }
                    const int hk = atomicAdd(&sh_hcount, 1);
                    if (hk < WVA_WROW_LIST) { sh_heavy[hk] = (r - r_lo) * B + n; continue; }
                    float rt, dc;
                    int st2 = analyze_table(tb, gs, b, rate, tame, 0, m, rt, steps, dc);
                    if (st2 < 0) { int k2 = atomicAdd(gp.slow_count, 1); if (k2 < gp.slow_cap) gp.slow_list[k2] = (unsigned long long)ci; continue; }
                    so.avgServTime = 0.0f;      // metrics already final in m
                    st = st2;
                    goto have_metrics;
                }
                st = WVA_CAND_OK;
                {
                    const float effConc = effective_concurrency(so.avgServTime, gs.sp, gs.inTok, gs.outTok, b);
                    float rho = so.avgNumInServers / (float)b;
                    rho = go_minf(go_maxf(rho, 0.0f), 1.0f);
                    m.throughput = so.throughput * 1000.0f;
                    m.avg_resp_time = so.avgRespTime;
                    m.avg_wait_time = so.avgWaitTime;
                    m.avg_num_in_serv = so.avgNumInServers;
                    m.avg_prefill_time = prefill_time(gs.sp, gs.inTok, effConc);
                    m.avg_token_time = decode_time(gs.sp, effConc);
                    m.max_rate = rateMax;
                    m.rho = rho;
                }
            have_metrics:
                if (st != WVA_CAND_OK) {
                    m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
                    m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
                    goto write_out;
                }
                okCount++;
                algSteps += 2ULL * (unsigned long long)(K + 1);
                const float lamMaxBack = rateMax / 1000.0f;
                const float rateTPS = (lamMaxBack * (1.0f - WVA_STABILITY_SAFETY)) * 1000.0f;
                const float ttft = m.avg_wait_time + m.avg_prefill_time;
                const float itl = m.avg_token_time;
                feasible = (!(gs.sloTTFT > 0.0f) || ttft <= gs.sloTTFT) && (!(gs.sloITL > 0.0f) || itl <= gs.sloITL) &&
                           (!(gs.sloTPS > 0.0f) || rate <= rateTPS) && (r >= gs.minReplicas);
                if (feasible && value == value) {              // a NaN value is never selected
                    const unsigned long long key = make_key(value, a, r, b);
                    if (key < bestKey) { bestKey = key; bestItl = itl; bestTtft = ttft; bestRho = m.rho; }
                }
            }
        write_out:
            if (gp.cube) {
                float4* c = reinterpret_cast<float4*>(&gp.cube[ci]);
                c[0] = make_float4(m.throughput, m.avg_resp_time, m.avg_wait_time, m.avg_num_in_serv);
                c[1] = make_float4(m.avg_prefill_time, m.avg_token_time, m.max_rate, m.rho);
            }
            if (gp.status) gp.status[ci] = (unsigned char)(st | (feasible ? WVA_CAND_FEASIBLE : 0));
        }
    }

    // ---- the block's uncertified candidates: exact chains, one per WARP (warp_exact) --------------
    __syncthreads();
    {
        const int nHeavy = sh_hcount < WVA_WROW_LIST ? sh_hcount : WVA_WROW_LIST;
        double* wx = reinterpret_cast<double*>(smem_raw + (((size_t)B * 20 + 15) & ~(size_t)15)) +
                     (size_t)(threadIdx.x >> 5) * (WVA_WX_CP + 1 + 1024);
        for (;;) {
            int idx;
            if (lane == 0) idx = atomicAdd(&sh_hnext, 1);
            idx = __shfl_sync(0xffffffffu, idx, 0);
            if (idx >= nHeavy) break;
            const int code = sh_heavy[idx];
            const int r = r_lo + code / B, n = code % B, b = n + 1;
            const size_t ci = candBase + (size_t)(r - 1) * B + (size_t)n;
            const float rate = gs.totalRate / (float)r;
            const float lambda = rate / 1000.0f;
            wva_metrics m;
            m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
            m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
            float rateTPS = 0.0f, dc = 0.0f;
            bool feasible = false;
            int st = WVA_CAND_OK;
            SolveStats so;
            unsigned long long wsteps = 0;
            if (warp_exact(tb, b, 11 * b, lambda, wx, wx + WVA_WX_CP + 1, lane, so, wsteps)) {
                // same epilogue as analyze_table
                const float rateMax = (rateF[n] * (1.0f - WVA_EPSILON)) * 1000.0f;
                const float lamMaxBack = rateMax / 1000.0f;
                rateTPS = (lamMaxBack * (1.0f - WVA_STABILITY_SAFETY)) * 1000.0f;
                const float effConc = effective_concurrency(so.avgServTime, gs.sp, gs.inTok, gs.outTok, b);
                float rho = so.avgNumInServers / (float)b;
                rho = go_minf(go_maxf(rho, 0.0f), 1.0f);
                m.throughput = so.throughput * 1000.0f;
                m.avg_resp_time = so.avgRespTime;
                m.avg_wait_time = so.avgWaitTime;
                m.avg_num_in_serv = so.avgNumInServers;
                m.avg_prefill_time = prefill_time(gs.sp, gs.inTok, effConc);
                m.avg_token_time = decode_time(gs.sp, effConc);
                m.max_rate = rateMax;
                m.rho = rho;
                steps += wsteps;
            } else if (lane == 0) {
                st = analyze_table(tb, gs, b, rate, tame, 0, m, rateTPS, steps, dc);     // per-thread solver, all cases
            }
            __syncwarp();
            if (lane != 0) continue;
            if (st < 0) { int k2 = atomicAdd(gp.slow_count, 1); if (k2 < gp.slow_cap) gp.slow_list[k2] = (unsigned long long)ci; continue; }
            if (st == WVA_CAND_OK) {
                okCount++;
                algSteps += 2ULL * (unsigned long long)(11 * b + 1);
                const unsigned long long key = candidate_key(gs, a, r, b, rate, rateTPS, m, feasible);
                if (key < bestKey) {
                    bestKey = key; bestItl = m.avg_token_time; bestTtft = m.avg_wait_time + m.avg_prefill_time; bestRho = m.rho;
                }
            } else {
                m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
                m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
            }
            if (gp.cube) {
                float4* c = reinterpret_cast<float4*>(&gp.cube[ci]);
                c[0] = make_float4(m.throughput, m.avg_resp_time, m.avg_wait_time, m.avg_num_in_serv);
                c[1] = make_float4(m.avg_prefill_time, m.avg_token_time, m.max_rate, m.rho);
            }
            if (gp.status) gp.status[ci] = (unsigned char)(st | (feasible ? WVA_CAND_FEASIBLE : 0));
        }
    }

    // ---- warp-shuffle then block argmin; the owner of the block minimum publishes its metrics ----
    unsigned long long warpKey = bestKey;
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long other = __shfl_down_sync(0xffffffffu, warpKey, o);
        if (other < warpKey) warpKey = other;
        steps += __shfl_down_sync(0xffffffffu, steps, o);
        algSteps += __shfl_down_sync(0xffffffffu, algSteps, o);
        okCount += __shfl_down_sync(0xffffffffu, okCount, o);
    }
    if (lane == 0) {
        if (warpKey != WVA_KEY_NONE) atomicMin(&sh_key, warpKey);
        atomicAdd(&sh_cnt[0], steps); atomicAdd(&sh_cnt[1], algSteps); atomicAdd(&sh_cnt[2], okCount);
    }
    __syncthreads();
    const unsigned long long blockKey = sh_key;
    if (blockKey != WVA_KEY_NONE && bestKey == blockKey) {
        GridSlot sl_; sl_.key = blockKey; sl_.itl = bestItl; sl_.ttft = bestTtft; sl_.rho = bestRho; sl_.sl = sl; sl_.pad = 0;
        const int r = (int)((blockKey >> 14) & 0x3ff) + 1;
        sl_.cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
        gp.block_slot[blockIdx.x] = sl_;
        atomicMin(&gp.keys[sl], blockKey);
        if (gp.pair_keys) atomicMin(&gp.pair_keys[gp.pair_base + (int)(blockIdx.x / (unsigned)gp.n_rchunks)], blockKey);   // a block covers one pair (index re-derived: no register live across the sweep)
    }
    if (threadIdx.x == 0) {
        atomicAdd(&gp.counters[0], sh_cnt[0]); atomicAdd(&gp.counters[1], sh_cnt[1]); atomicAdd(&gp.counters[2], sh_cnt[2]);
    }
}

// Candidate evaluated through the formula-based analyzer.  Same arithmetic as analyze_table, hence
// the same bits.  tab: the pair's published {rate, reciprocal} table (unified-loop streaming solver)
// or nullptr; scratch: p[] for the literal path or nullptr.
__device__ int analyze_candidate(const DevSystem& sys, int s, int a, int r, int b, const double2* tab, double* scratch,
                                 GridServer& gs, wva_metrics& m, float& rate, float& rateTPS, int& fault,
                                 unsigned long long& steps) {
    load_grid_server(sys, s, a, gs);
    Analyzer qa;
    qa.build(gs.sp, b, (long long)b * WVA_MAX_QUEUE_TO_BATCH_RATIO, gs.inTok, gs.outTok, scratch);
    qa.tab = tab; qa.uni = true; qa.cert = sys.cert != 0;
    const float lamMaxBack = qa.rateMax / 1000.0f;
    rateTPS = (lamMaxBack * (1.0f - WVA_STABILITY_SAFETY)) * 1000.0f;
    rate = gs.totalRate / (float)r;
    int st = qa.analyze(rate, m);
    fault = qa.fault;
    steps += qa.steps;
    return st;
}

// Candidates from a list, one thread each.
//   scratch == nullptr : the deferred long chains (streaming, unified-loop solver on the published
//                        tables); `order` sorts them by estimated length so that the lanes of a warp
//                        finish together; a chain that needs the materialised path is appended to
//                        the literal list.
//   scratch != nullptr : the literal list (p[] materialised, `stride` doubles per thread).
// Each thread publishes key + metrics in gp.list_slot[slot_base + t] for k_grid_claim.
// one candidate of a list: evaluate, publish key + metrics in gp.list_slot[slot] for k_grid_claim
__device__ __forceinline__ void grid_list_item(const DevSystem& sys, const GridParams& gp, const size_t ci, const int slotIdx, double* scratchRow,
                                               unsigned long long& steps, unsigned long long& alg, unsigned long long& okc) {
    const int B = gp.b_max;
    const int b = (int)(ci % B) + 1;
    const int r = (int)((ci / B) % gp.r_max) + 1;
    const int pairLocal = (int)(ci / ((size_t)B * gp.r_max));
    const int sl = pairLocal / sys.A, a = pairLocal % sys.A, s = gp.s0 + sl;
    GridServer gs; wva_metrics m; float rate, rateTPS; int fault = 0;
    GridSlot slot; slot.key = WVA_KEY_NONE; slot.cost = slot.itl = slot.ttft = slot.rho = 0.0f; slot.sl = sl; slot.pad = 0;
    int st = analyze_candidate(sys, s, a, r, b, scratchRow ? nullptr : gp.pair_tab + (size_t)(pairLocal - gp.pair_base) * B,
                               scratchRow, gs, m, rate, rateTPS, fault, steps);
    if (fault == 1) {
        int k = atomicAdd(gp.slow_count, 1);
        if (k < gp.slow_cap) gp.slow_list[k] = (unsigned long long)ci;
    } else {
        bool feasible = false;
        if (st == WVA_CAND_OK) {
            unsigned long long key = candidate_key(gs, a, r, b, rate, rateTPS, m, feasible);
            if (key != WVA_KEY_NONE) {
                slot.key = key; slot.itl = m.avg_token_time; slot.ttft = m.avg_wait_time + m.avg_prefill_time;
                slot.rho = m.rho; slot.cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
                if (key < gp.keys[sl]) atomicMin(&gp.keys[sl], key);
                if (gp.pair_keys) {          // pair index from (sl, a), live here anyway
                    unsigned long long* pk = gp.pair_keys + (sl * sys.A + a);
                    if (key < *pk) atomicMin(pk, key);
                }
            }
            alg += 2ULL * (unsigned long long)(11 * b + 1);
            okc += 1;
        } else {
            m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
            m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
        }
        if (gp.cube) {
            float4* c = reinterpret_cast<float4*>(&gp.cube[ci]);
            c[0] = make_float4(m.throughput, m.avg_resp_time, m.avg_wait_time, m.avg_num_in_serv);
            c[1] = make_float4(m.avg_prefill_time, m.avg_token_time, m.max_rate, m.rho);
        }
        if (gp.status) gp.status[ci] = (unsigned char)(st | (feasible ? WVA_CAND_FEASIBLE : 0));
    }
    gp.list_slot[slotIdx] = slot;
}

__device__ __forceinline__ void grid_list_counters(const GridParams& gp, unsigned long long steps, unsigned long long alg, unsigned long long okc) {
    for (int o = 16; o > 0; o >>= 1) {
        steps += __shfl_down_sync(0xffffffffu, steps, o);
        alg += __shfl_down_sync(0xffffffffu, alg, o);
        okc += __shfl_down_sync(0xffffffffu, okc, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (steps) atomicAdd(&gp.counters[0], steps);
        if (alg) atomicAdd(&gp.counters[1], alg);
        if (okc) atomicAdd(&gp.counters[2], okc);
    }
}

__global__ void __launch_bounds__(128)
k_grid_list(DevSystem sys, GridParams gp, const unsigned long long* __restrict__ list, const int* __restrict__ order,
            int nList, double* scratch, long long stride, int slot_base) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long steps = 0, alg = 0, okc = 0;
    if (t < nList)
        grid_list_item(sys, gp, (size_t)list[order ? order[t] : t], slot_base + t, scratch ? scratch + (size_t)t * stride : nullptr, steps, alg, okc);
    grid_list_counters(gp, steps, alg, okc);
}

// The deferred long chains again, for the sweep that does not stop at the host between its kernels: the number of
// chains is read from device memory (*count, clamped to cap), the grid is a handful of 512-thread blocks that ask for
// 200 KB of shared memory they do not use -- so each block has an SM to itself and the cube-writing kernel that
// runs beside it (k_scan_lean, issue-bound) cannot slow the 4 dependent-chain warps per scheduler down -- and the
// threads stride over the list (ordered longest first).
__global__ void __launch_bounds__(512, 1)
k_grid_list_own(DevSystem sys, GridParams gp, const unsigned long long* __restrict__ list, const int* __restrict__ order,
                const int* __restrict__ count, int cap) {
    const int n = min(*count, cap);
    const int G = gridDim.x * blockDim.x;
    unsigned long long steps = 0, alg = 0, okc = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += G)
        grid_list_item(sys, gp, (size_t)list[order[i]], i, nullptr, steps, alg, okc);
    grid_list_counters(gp, steps, alg, okc);
}

// Deferred candidates, one WARP each (warp_exact): for short lists, where the latency of a single
// exact chain -- not throughput -- sets the duration of the phase.  The warp copies the first b
// entries of the pair's published table into its shared-memory slice, runs the cooperative exact
// chain and lane 0 publishes like k_grid_list; chains outside warp_exact's scope fall back to the
// per-thread analyzer on lane 0.  Dynamic shared memory: per warp 2 b_max + WVA_WX_CP + 1 + 1024 doubles.
#define WVA_LISTW_WARPS 4
__global__ void __launch_bounds__(WVA_LISTW_WARPS * 32)
k_grid_list_warp(DevSystem sys, GridParams gp, const unsigned long long* __restrict__ list, int nList, int slot_base) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int B = gp.b_max;
    double* rateD = reinterpret_cast<double*>(smem_raw) + (size_t)w * (2 * (size_t)B + WVA_WX_CP + 1 + 1024);
    double* rcp = rateD + B;
    double* cp = rcp + B;
    double* qbuf = cp + WVA_WX_CP + 1;
    unsigned long long steps = 0, alg = 0, okc = 0;
    for (int t = blockIdx.x * WVA_LISTW_WARPS + w; t < nList; t += gridDim.x * WVA_LISTW_WARPS) {
        const size_t ci = (size_t)list[t];
        const int b = (int)(ci % B) + 1;
        const int r = (int)((ci / B) % gp.r_max) + 1;
        const int pairLocal = (int)(ci / ((size_t)B * gp.r_max));
        const int sl = pairLocal / sys.A, a = pairLocal % sys.A, s = gp.s0 + sl;
        const double2* tab = gp.pair_tab + (size_t)(pairLocal - gp.pair_base) * B;
        __syncwarp();
        for (int i = lane; i < b; i += 32) { const double2 v = tab[i]; rateD[i] = v.x; rcp[i] = v.y; }
        __syncwarp();
        GridServer gs; wva_metrics m; float rate, rateTPS; int fault = 0;
        m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
        m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
        GridSlot slot; slot.key = WVA_KEY_NONE; slot.cost = slot.itl = slot.ttft = slot.rho = 0.0f; slot.sl = sl; slot.pad = 0;
        load_grid_server(sys, s, a, gs);
        rate = gs.totalRate / (float)r;
        const float lambda = rate / 1000.0f;
        const float rateMax = ((float)rateD[b - 1] * (1.0f - WVA_EPSILON)) * 1000.0f;
        int st;
        ServTable tb; tb.rateF = nullptr; tb.rateD = rateD; tb.rcp = rcp;
        SolveStats so;
        unsigned long long wsteps = 0;
        const bool inScope = rate > 0.0f && !(rate > rateMax) && !(lambda < 0.0f);
#ifdef WVA_DEBUG_CAREFUL
        const long long tdbg0 = clock64();
        const bool wxok = inScope && warp_exact(tb, b, 11 * b, lambda, cp, qbuf, lane, so, wsteps);
        const long long tdbg1 = clock64();
        if (lane == 0) printf("listwarp b=%d lambda=%g rho=%g ok=%d cycles=%lld\n", b, (double)lambda, (double)lambda / rateD[b - 1], (int)wxok, tdbg1 - tdbg0);
        if (wxok) {
#else
        if (inScope && warp_exact(tb, b, 11 * b, lambda, cp, qbuf, lane, so, wsteps)) {
#endif
            const float lamMaxBack = rateMax / 1000.0f;
            rateTPS = (lamMaxBack * (1.0f - WVA_STABILITY_SAFETY)) * 1000.0f;
            const float effConc = effective_concurrency(so.avgServTime, gs.sp, gs.inTok, gs.outTok, b);
            float rho = so.avgNumInServers / (float)b;
            rho = go_minf(go_maxf(rho, 0.0f), 1.0f);
            m.throughput = so.throughput * 1000.0f;
            m.avg_resp_time = so.avgRespTime;
            m.avg_wait_time = so.avgWaitTime;
            m.avg_num_in_serv = so.avgNumInServers;
            m.avg_prefill_time = prefill_time(gs.sp, gs.inTok, effConc);
            m.avg_token_time = decode_time(gs.sp, effConc);
            m.max_rate = rateMax;
            m.rho = rho;
            st = WVA_CAND_OK;
            if (lane == 0) steps += wsteps;
        } else if (lane == 0) {
#ifdef WVA_DEBUG_CAREFUL
            const long long tf0 = clock64();
#endif
            st = analyze_candidate(sys, s, a, r, b, tab, nullptr, gs, m, rate, rateTPS, fault, steps);
#ifdef WVA_DEBUG_CAREFUL
            printf("listwarp fallback b=%d cycles=%lld\n", b, clock64() - tf0);
#endif
        }
        __syncwarp();
        if (lane != 0) continue;
        if (fault == 1) {
            int k = atomicAdd(gp.slow_count, 1);
            if (k < gp.slow_cap) gp.slow_list[k] = (unsigned long long)ci;
        } else {
            bool feasible = false;
            if (st == WVA_CAND_OK) {
                unsigned long long key = candidate_key(gs, a, r, b, rate, rateTPS, m, feasible);
                if (key != WVA_KEY_NONE) {
                    slot.key = key; slot.itl = m.avg_token_time; slot.ttft = m.avg_wait_time + m.avg_prefill_time;
                    slot.rho = m.rho; slot.cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
                    if (key < gp.keys[sl]) atomicMin(&gp.keys[sl], key);
                    if (gp.pair_keys) {          // pair index from (sl, a), live here anyway
                        unsigned long long* pk = gp.pair_keys + (sl * sys.A + a);
                        if (key < *pk) atomicMin(pk, key);
                    }
                }
                alg += 2ULL * (unsigned long long)(11 * b + 1);
                okc += 1;
            } else {
                m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
                m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
            }
            if (gp.cube) {
                float4* c = reinterpret_cast<float4*>(&gp.cube[ci]);
                c[0] = make_float4(m.throughput, m.avg_resp_time, m.avg_wait_time, m.avg_num_in_serv);
                c[1] = make_float4(m.avg_prefill_time, m.avg_token_time, m.max_rate, m.rho);
            }
            if (gp.status) gp.status[ci] = (unsigned char)(st | (feasible ? WVA_CAND_FEASIBLE : 0));
        }
        gp.list_slot[slot_base + t] = slot;
    }
    if (lane == 0) {
        if (steps) atomicAdd(&gp.counters[0], steps);
        if (alg) atomicAdd(&gp.counters[1], alg);
        if (okc) atomicAdd(&gp.counters[2], okc);
    }
}

// ---- ordering of the deferred chains by estimated length (256 buckets, longest first) --------
__device__ __forceinline__ int heavy_bucket(float cost) {
    int k = (int)(__float_as_uint(cost < 1.0f ? 1.0f : cost) >> 19) - (127 << 4);    // 16 buckets per octave
    k = k < 0 ? 0 : (k > 255 ? 255 : k);
    return 255 - k;
}
__global__ void k_heavy_hist(const float* __restrict__ cost, int n, int* __restrict__ hist) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) atomicAdd(&hist[heavy_bucket(cost[t])], 1);
}
__global__ void k_heavy_prefix(int* hist /*[256] -> exclusive prefix in place*/) {
    __shared__ int sh[256];
    int t = threadIdx.x;
    sh[t] = hist[t];
    __syncthreads();
    if (t == 0) { int run = 0; for (int i = 0; i < 256; ++i) { int c = sh[i]; sh[i] = run; run += c; } }
    __syncthreads();
    hist[t] = sh[t];
}
__global__ void k_heavy_scatter(const float* __restrict__ cost, int n, int* __restrict__ cursor, int* __restrict__ order) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) order[atomicAdd(&cursor[heavy_bucket(cost[t])], 1)] = t;
}
// ordering kernels with the list length in device memory
__global__ void k_heavy_hist_dev(const float* __restrict__ cost, const int* __restrict__ count, int cap, int* __restrict__ hist) {
    const int n = min(*count, cap);
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) atomicAdd(&hist[heavy_bucket(cost[t])], 1);
}
__global__ void k_heavy_scatter_dev(const float* __restrict__ cost, const int* __restrict__ count, int cap, int* __restrict__ cursor, int* __restrict__ order) {
    const int n = min(*count, cap);
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) order[atomicAdd(&cursor[heavy_bucket(cost[t])], 1)] = t;
}


// Per-server winners: keys[] holds the minimum key of every server; the slot that carries that key
// (exactly one: keys are unique per candidate) writes the wva_grid_best record.  No re-evaluation.
// With per-pair winners on, the pair keys and records of the shard are reset here too (empty record, infeasible).
__global__ void k_grid_best_init(int ns, wva_grid_best* __restrict__ best, GridParams gp, int A) {
    int sl = blockIdx.x * blockDim.x + threadIdx.x;
    if (sl >= ns) return;
    wva_grid_best out;
    out.acc = -1; out.replicas = 0; out.batch = 0; out.cost = out.value = out.itl = out.ttft = out.rho = 0.0f;
    best[sl] = out;
    if (gp.pair_keys) {
        for (int a = 0; a < A; ++a) {
            const size_t pl = (size_t)sl * A + a, gi = (size_t)gp.s0 * A + pl;
            gp.pair_keys[pl] = WVA_KEY_NONE;
            store_alloc(gp.pair_rec, gi, empty_alloc());
            gp.pair_feasible[gi] = 0;
        }
    }
}
// A slot that carries its server's minimum key writes the wva_grid_best record; with per-pair winners on, a slot that
// carries its pair's minimum key also writes that pair's candidate record (a server's winner is its best pair's winner).
__global__ void k_grid_claim(DevSystem sys, GridParams gp, const GridSlot* __restrict__ slots, int nSlots, wva_grid_best* __restrict__ best) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nSlots) return;
    const GridSlot sl_ = slots[t];
    if (sl_.key == WVA_KEY_NONE) return;
    const int a = (int)((sl_.key >> 24) & 0xff), r = (int)((sl_.key >> 14) & 0x3ff) + 1, b = (int)(sl_.key & 0x3fff) + 1;
    const float value = unsortable_f32((unsigned)(sl_.key >> 32));
    if (gp.pair_keys) {
        const size_t pl = (size_t)sl_.sl * sys.A + a;
        if (gp.pair_keys[pl] == sl_.key) {
            // the per-replica rate the candidate was analysed at: scan_row_ctx's lambda (load_grid_server's totalRate)
            const int s = gp.s0 + sl_.sl;
            const float sloTPS = sys.srv_slo_tps[s];
            const float totalRate = (sloTPS == 0.0f) ? sys.srv_arrival_rpm[s] / 60.0f : sloTPS / (float)(long long)sys.srv_out_tokens[s];
            AllocRec rec;
            rec.acc = a; rec.numReplicas = r; rec.batchSize = b;
            rec.cost = sl_.cost; rec.value = value; rec.itl = sl_.itl; rec.ttft = sl_.ttft; rec.rho = sl_.rho;
            rec.maxArrv = (totalRate / (float)r) / 1000.0f;
            const size_t gi = (size_t)gp.s0 * sys.A + pl;
            store_alloc(gp.pair_rec, gi, rec);
            gp.pair_feasible[gi] = 1;
        }
    }
    if (gp.keys[sl_.sl] != sl_.key) return;
    wva_grid_best out;
    out.acc = a; out.replicas = r; out.batch = b;
    out.cost = sl_.cost;
    out.value = value;
    out.itl = sl_.itl; out.ttft = sl_.ttft; out.rho = sl_.rho;
    best[sl_.sl] = out;
}

// ---------------------------------------------------------------------------------------
// pkg/analyzer batched public API
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_queue_analyze(int n, const wva_queue_config* __restrict__ cfg, const float* __restrict__ rate,
                wva_metrics* __restrict__ metrics, unsigned char* __restrict__ status, double* scratch,
                const long long* __restrict__ scratch_off, const int* __restrict__ list, int* fault_list, int* fault_count) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int i = list ? list[t] : t;
    wva_queue_config c = cfg[i];
    wva_metrics m;
    m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
    m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
    int st;
    if (!config_ok(c.max_batch_size, c.max_queue_size, c.avg_input_tokens, c.avg_output_tokens)) st = WVA_CAND_ERR_CONFIG;
    else {
        ServiceParms sp; sp.alpha = c.alpha; sp.beta = c.beta; sp.gamma = c.gamma; sp.delta = c.delta;
        Analyzer qa;
        qa.build(sp, c.max_batch_size, c.max_queue_size, c.avg_input_tokens, c.avg_output_tokens,
                 scratch ? scratch + scratch_off[t] : nullptr);
        st = qa.analyze(rate[i], m);
        if (qa.fault == 1) { fault_list[atomicAdd(fault_count, 1)] = i; return; }
        if (st != WVA_CAND_OK) {
            m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
            m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
        }
    }
    metrics[i] = m;
    status[i] = (unsigned char)st;
}

__global__ void __launch_bounds__(128)
k_queue_size(int n, const wva_queue_config* __restrict__ cfg, const float* __restrict__ target,
             float* __restrict__ rates, wva_metrics* __restrict__ metrics, float* __restrict__ achieved,
             unsigned char* __restrict__ status, double* scratch, const long long* __restrict__ scratch_off,
             const int* __restrict__ list, int* fault_list, int* fault_count) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int i = list ? list[t] : t;
    wva_queue_config c = cfg[i];
    wva_metrics m;
    m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
    m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
    float rt[3] = {0.0f, 0.0f, 0.0f}, ach[3] = {0.0f, 0.0f, 0.0f};
    bool ok = false;
    if (config_ok(c.max_batch_size, c.max_queue_size, c.avg_input_tokens, c.avg_output_tokens)) {
        ServiceParms sp; sp.alpha = c.alpha; sp.beta = c.beta; sp.gamma = c.gamma; sp.delta = c.delta;
        Analyzer qa;
        qa.build(sp, c.max_batch_size, c.max_queue_size, c.avg_input_tokens, c.avg_output_tokens,
                 scratch ? scratch + scratch_off[t] : nullptr);
        ok = size_queue(qa, target[3 * i], target[3 * i + 1], target[3 * i + 2], rt, m, ach);
        if (qa.fault == 1) { fault_list[atomicAdd(fault_count, 1)] = i; return; }
        if (!ok) {
            m.throughput = m.avg_resp_time = m.avg_wait_time = m.avg_num_in_serv = 0.0f;
            m.avg_prefill_time = m.avg_token_time = m.max_rate = m.rho = 0.0f;
            rt[0] = rt[1] = rt[2] = ach[0] = ach[1] = ach[2] = 0.0f;
        }
    }
    metrics[i] = m;
    for (int k = 0; k < 3; ++k) { rates[3 * i + k] = rt[k]; achieved[3 * i + k] = ach[k]; }
    status[i] = ok ? 0 : 1;
}

// ---------------------------------------------------------------------------------------
// Optimize
// ---------------------------------------------------------------------------------------

__device__ __forceinline__ DevAllocs allocs_at(const DevAllocs& o, size_t off) {
    DevAllocs r;
    r.acc = o.acc + off; r.num_replicas = o.num_replicas + off; r.batch_size = o.batch_size + off;
    r.cost = o.cost + off; r.value = o.value + off; r.itl = o.itl + off; r.ttft = o.ttft + off; r.rho = o.rho + off;
    r.max_arrv = o.max_arrv + off;
    return r;
}

// SolveUnlimited, solver.go:63-79: per server argmin of value with strict '<' from MaxFloat32,
// candidates visited in ascending accelerator index (canonical order for Go's random map order).
// blockIdx.y selects a record set (wva_analyze_scenarios: one per scenario) at pairStride records / flags, and its
// solution at chosenStride; a single set runs with gridDim.y = 1.
__global__ void k_solve_unlimited(DevSystem sys, int s0, int ns, DevAllocs pairs, const unsigned char* __restrict__ feasible,
                                  int* __restrict__ chosen_acc, DevAllocs chosen, size_t pairStride, size_t chosenStride) {
    int sl = blockIdx.x * blockDim.x + threadIdx.x;
    if (sl >= ns) return;
    if (blockIdx.y) {
        pairs = allocs_at(pairs, blockIdx.y * pairStride); feasible += blockIdx.y * pairStride;
        chosen = allocs_at(chosen, blockIdx.y * chosenStride); chosen_acc += blockIdx.y * chosenStride;
    }
    int s = s0 + sl;
    float minVal = 3.40282346638528859811704183484516925e+38f;
    int minKey = -1;
    for (int a = 0; a < sys.A; ++a) {
        size_t i = (size_t)s * sys.A + a;
        if (!feasible[i]) continue;
        float v = pairs.value[i];
        if (v < minVal) { minVal = v; minKey = a; }
    }
    chosen_acc[s] = minKey;
    store_alloc(chosen, (size_t)s, minKey >= 0 ? load_alloc(pairs, (size_t)s * sys.A + minKey) : empty_alloc());
}

// System.AllocateByType (system.go:271-300) over servers [s0, s0+ns): one block per accelerator
// type.  The float32 cost sum keeps a fixed order (ascending server index): the block stages 1024
// servers' contributions in shared memory in parallel, then warp 0 adds them in order (a server
// of another type contributes +0, which leaves a float32 sum that started at +0 unchanged).
// The int64 unit counts wrap and are associative: plain tree reduction.
// totals = { long long count[T]; float cost[T] }.  blockIdx.y selects a solution (wva_analyze_scenarios: one per
// scenario) at chosenStride servers, whose totals go to count / cost + blockIdx.y * T.
__global__ void __launch_bounds__(1024) k_totals(DevSystem sys, int s0, int ns, const int* __restrict__ chosen_acc, DevAllocs chosen,
                                                 long long* __restrict__ count, float* __restrict__ cost, size_t chosenStride) {
    __shared__ float vals[1024];
    __shared__ long long part[32];
    const int t = blockIdx.x;
    if (blockIdx.y) {
        chosen = allocs_at(chosen, blockIdx.y * chosenStride); chosen_acc += blockIdx.y * chosenStride;
        count += (size_t)blockIdx.y * sys.T; cost += (size_t)blockIdx.y * sys.T;
    }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    long long c = 0; float k = 0.0f;
    for (int base = 0; base < ns; base += 1024) {
        const int s = s0 + base + tid;
        float v = 0.0f;
        if (base + tid < ns && chosen_acc[s] >= 0) {
            const int gi = chosen.acc[s];
            const int m = sys.srv_model[s];
            if (gi >= 0 && m >= 0 && sys.acc_type[gi] == t) {
                c += go_muli(go_muli(chosen.num_replicas[s], num_instances(sys, m, gi)), (long long)sys.acc_multiplicity[gi]);
                v = chosen.cost[s];
            }
        }
        vals[tid] = v;
        __syncthreads();
        if (warp == 0) {
            const int cnt = min(1024, ns - base);
            for (int b = 0; b < cnt; b += 32) {
                const float mine = vals[b + lane];
#pragma unroll
                for (int j = 0; j < 32; ++j) k = k + __shfl_sync(0xffffffffu, mine, j);
            }
        }
        __syncthreads();
    }
    for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
    if (lane == 0) part[warp] = c;
    __syncthreads();
    if (tid == 0) {
        long long tot = 0;
        for (int w = 0; w < 32; ++w) tot += part[w];
        count[t] = tot; cost[t] = k;
    }
}

// Sum the per-rank partial totals of a sharded run in rank order (deterministic, unlike a ring or
// tree all-reduce): gathered = n_ranks blocks of { long long count[T]; float cost[T] }.
__global__ void k_totals_merge(int T, int n_ranks, const unsigned char* __restrict__ gathered, long long* __restrict__ count,
                               float* __restrict__ cost) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    long long c = 0; float k = 0.0f;
    for (int r = 0; r < n_ranks; ++r) {
        const unsigned char* blk = gathered + (size_t)r * T * 12;
        c += reinterpret_cast<const long long*>(blk)[t];
        k = k + reinterpret_cast<const float*>(blk + (size_t)T * 8)[t];
    }
    count[t] = c; cost[t] = k;
}

// pkg/analyzer's bare model: a sequence of MM1ModelStateDependent.Solve(lambda, mu) calls on ONE model instance
// NewMM1ModelStateDependent(K, servRate) (mm1modelstatedependent.go:15-116 through QueueModel.Solve, queuemodel.go:27-37).
// The model keeps p[] between calls -- the validity test reads the PREVIOUS call's p[0] -- and the getters keep the last
// valid statistics.  Literal algorithm with p[] in global memory, one thread (this is the low-level API, not the path).
struct ArrayServ { const float* r; __device__ __forceinline__ float rate(long long n) const { return r[n - 1]; } };
__global__ void k_model_solve(long long K, const float* __restrict__ serv, int nRates, int nCalls, const float* __restrict__ lambda,
                              const float* __restrict__ mu, double* __restrict__ p, float* __restrict__ out, int* __restrict__ fault) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    for (long long i = 0; i <= K; ++i) p[i] = 0.0;
    float st[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};      // isValid, rho, resp, wait, serv, inSystem, queueLen, inServers, throughput
    ArrayServ sv; sv.r = serv;
    unsigned long long steps = 0;
    for (int c = 0; c < nCalls; ++c) {
        const float lam = lambda[c], m = mu[c];
        const float rho = 1.0f - (float)p[0];                              // ComputeRho on the stale p[0]
        st[1] = rho;
        if ((rho < 0.0f) || (rho >= (float)K) || (lam < 0.0f) || (m <= 0.0f)) st[0] = 0.0f;
        else {
            SolveStats so;
            if (solve_literal(p, sv, (long long)nRates, K, lam, so, steps)) { *fault = 1; st[0] = 0.0f; }
            else {
                st[0] = 1.0f; st[1] = so.rho; st[2] = so.avgRespTime; st[3] = so.avgWaitTime; st[4] = so.avgServTime;
                st[5] = so.avgNumInSystem; st[6] = so.throughput * so.avgWaitTime; st[7] = so.avgNumInServers; st[8] = so.throughput;
            }
        }
        for (int k = 0; k < 9; ++k) out[9 * c + k] = st[k];
    }
}

// RemoveServer (system.go:165-171) on the resident image: the last server's row moves into the freed slot.
__global__ void k_server_move(DevSystem sys, int from, int to) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
#define MV(field, T) const_cast<T*>(sys.field)[to] = sys.field[from];
    MV(srv_model, int) MV(srv_arrival_rpm, float) MV(srv_in_tokens, int) MV(srv_out_tokens, int) MV(srv_slo_ttft, float)
    MV(srv_slo_itl, float) MV(srv_slo_tps, float) MV(srv_target_valid, unsigned char) MV(srv_priority, int) MV(srv_min_replicas, int)
    MV(srv_max_batch, int) MV(srv_keep_acc, unsigned char) MV(srv_cur_acc, int) MV(srv_cur_replicas, int) MV(srv_cur_cost, float)
#undef MV
}

// ---- multi-rank exchange of the candidate records (limited mode) -----------------------------
// One chunk per rank: {int first_pair, n_pairs, pad, pad} then SoA sections of `cap` records each
// (replicas i64, batch i64, accelerator i32, 6 x f32, feasible u8 = 45 B per record).
struct PairChunk {
    long long* rep; long long* bat; int* acc; float* f[6]; unsigned char* fe; int* hdr;
};
__host__ __device__ __forceinline__ size_t pair_chunk_bytes(size_t cap) { return (16 + cap * 45 + 15) / 16 * 16; }
__device__ __forceinline__ PairChunk pair_chunk_at(unsigned char* base, size_t cap) {
    PairChunk c;
    c.hdr = reinterpret_cast<int*>(base);
    unsigned char* q = base + 16;
    c.rep = reinterpret_cast<long long*>(q); q += cap * 8;
    c.bat = reinterpret_cast<long long*>(q); q += cap * 8;
    c.acc = reinterpret_cast<int*>(q); q += cap * 4;
    for (int k = 0; k < 6; ++k) { c.f[k] = reinterpret_cast<float*>(q); q += cap * 4; }
    c.fe = q;
    return c;
}
__global__ void k_pairs_pack(DevAllocs pairs, const unsigned char* __restrict__ feasible, int firstPair, int nPairs, size_t cap,
                             unsigned char* __restrict__ chunk) {
    PairChunk c = pair_chunk_at(chunk, cap);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) { c.hdr[0] = firstPair; c.hdr[1] = nPairs; c.hdr[2] = 0; c.hdr[3] = 0; }
    if (i >= nPairs) return;
    const size_t g = (size_t)firstPair + i;
    c.rep[i] = pairs.num_replicas[g]; c.bat[i] = pairs.batch_size[g]; c.acc[i] = pairs.acc[g];
    c.f[0][i] = pairs.cost[g]; c.f[1][i] = pairs.value[g]; c.f[2][i] = pairs.itl[g];
    c.f[3][i] = pairs.ttft[g]; c.f[4][i] = pairs.rho[g]; c.f[5][i] = pairs.max_arrv[g];
    c.fe[i] = feasible[g];
}
// grid.y = source rank; rows of the calling rank itself are skipped (they are already in place)
__global__ void k_pairs_unpack(unsigned char* __restrict__ gathered, size_t chunkBytes, size_t cap, int myRank, size_t nPairsAll,
                               DevAllocs pairs, unsigned char* __restrict__ feasible) {
    const int r = blockIdx.y;
    if (r == myRank) return;
    PairChunk c = pair_chunk_at(gathered + (size_t)r * chunkBytes, cap);
    const int first = c.hdr[0], n = c.hdr[1];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const size_t g = (size_t)first + i;
        if (g >= nPairsAll) return;
        pairs.num_replicas[g] = c.rep[i]; pairs.batch_size[g] = c.bat[i]; pairs.acc[g] = c.acc[i];
        pairs.cost[g] = c.f[0][i]; pairs.value[g] = c.f[1][i]; pairs.itl[g] = c.f[2][i];
        pairs.ttft[g] = c.f[3][i]; pairs.rho[g] = c.f[4][i]; pairs.max_arrv[g] = c.f[5][i];
        feasible[g] = c.fe[i];
    }
}

// ---- greedy ------------------------------------------------------------------------------

// cmp.Compare for float32: NaN lowest, -0 == +0
__device__ __forceinline__ int go_cmpf(float x, float y) {
    bool xn = x != x, yn = y != y;
    if (xn) return yn ? 0 : -1;
    if (yn) return 1;
    if (x < y) return -1;
    if (x > y) return 1;
    return 0;
}

struct GreedyTicket {      // allocateEqually's serverAllocationTicket (greedy.go:226-236)
    long long upr;         // units one replica takes
    long long cur;         // replicas the candidate wants
    long long got;         // replicas handed out
    int slot;              // s*A + position in the server's candidate order (-1: none)
    int type;
};

// what the sequential pass reads of one candidate: one 16-byte load; a server's candidates are
// contiguous (one 128-byte line for 8 accelerators)
struct __align__(16) GreedyCand {
    long long count;       // units the candidate takes: replicas x instances x multiplicity
    float val;
    int tf;                // type | GREEDY_LAST (server's last candidate) | GREEDY_SKIP (no accelerator)
};
constexpr int GREEDY_LAST = 1 << 16, GREEDY_SKIP = 1 << 17;

struct GreedyBufs {
    // per server, candidates in greedy order (ascending value, stable on accelerator index)
    int* order;            // [S*A] candidate key (accelerator index)
    GreedyCand* cand;      // [S*A]
    long long* upr;        // [S*A] units per replica (instances x multiplicity)
    long long* rep;        // [S*A] replicas
    int* ctype;            // [S*A] accelerator type, -1 when the candidate has no accelerator
    int* nCand;            // [S]
    int* groupStart;       // [102] population / start offset of each priority (1..100)
    int* groupItems;       // [S]
    int* unalloc;          // [S]
    unsigned long long* heapA;   // [S] heap storage used when a group does not fit shared memory
    unsigned long long* heapB;   // [S]
    unsigned* heapSlot;          // [S]
    GreedyTicket* tickets;       // [S] ditto for allocateEqually
    int* liveIdx;                // [S]
    int* nanFlag;          // [2]
    unsigned long long* stats;   // [4] instrumentation: queue pops, failed placements, cycles in the queue loop, cycles in bestEffort
    int smemBytes;         // dynamic shared memory handed to k_greedy_solve
};

// per server: sort candidate keys by value (greedy.go:57-63) and lay the fields the sequential
// pass reads out in that order, so that one pop costs one dependent load
__global__ void k_greedy_prepare(DevSystem sys, DevAllocs pairs, const unsigned char* __restrict__ feasible, GreedyBufs g) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= sys.S) return;
    const size_t base = (size_t)s * sys.A;
    int* ord = g.order + base;
    int n = 0;
    for (int a = 0; a < sys.A; ++a) {
        size_t i = base + a;
        if (!feasible[i]) continue;
        float v = pairs.value[i];
        int j = n++;
        // stable insertion sort by cmp.Compare(value)
        while (j > 0 && go_cmpf(pairs.value[base + ord[j - 1]], v) > 0) { ord[j] = ord[j - 1]; --j; }
        ord[j] = a;
    }
    g.nCand[s] = n;
    const int m = sys.srv_model[s];
    for (int k = 0; k < n; ++k) {
        size_t ai = base + ord[k];
        float v = pairs.value[ai];
        int gi = pairs.acc[ai];
        long long upr = 0; int t = -1;
        if (m >= 0 && gi >= 0) { upr = go_muli(num_instances(sys, m, gi), (long long)sys.acc_multiplicity[gi]); t = sys.acc_type[gi]; }
        const long long reps = pairs.num_replicas[ai];
        g.upr[base + k] = upr;
        g.rep[base + k] = reps;
        g.ctype[base + k] = t;
        GreedyCand cd;
        cd.count = go_muli(reps, upr);
        cd.val = v;
        cd.tf = (t < 0 ? GREEDY_SKIP : t) | (k == n - 1 ? GREEDY_LAST : 0);
        g.cand[base + k] = cd;
    }
}

// monotone map float32 -> uint32 for cmp.Compare on non-NaN values (-0 and +0 coincide)
__device__ __forceinline__ unsigned f32_sortable(float f) {
    if (f != f) return 0u;                       // cmp.Compare: NaN sorts before every number
    f = f + 0.0f;
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// orderFunc, greedy.go:76-85, as a pair of ascending 64-bit keys: priority ascending, delta
// descending, current value descending, and -- refining ties into a strict order -- the recency
// stamp descending: an entry re-inserted by slices.BinarySearchFunc lands before every equal
// entry (largest stamp first); the initial stable sort keeps equal entries in ascending server
// index (stamp = -index).
__device__ __forceinline__ void greedy_keys(int priority, float delta, float value, int stamp,
                                            unsigned long long& ka, unsigned long long& kb) {
    ka = ((unsigned long long)(unsigned)priority << 32) | (unsigned)~f32_sortable(delta);
    // orderFunc looks at the values only when the deltas compare == (greedy.go:78-80): two NaN deltas are "equal" whatever
    // the values are
    kb = ((unsigned long long)(delta != delta ? 0u : (unsigned)~f32_sortable(value)) << 32) | (unsigned)~((unsigned)stamp + 0x80000000u);
}

// 4-ary min-heap on (a, b), structure of arrays so that shared memory is used to the byte
struct GreedyHeap {
    unsigned long long* a; unsigned long long* b; unsigned* slot; int n;
    // place (va,vb,vs) at or below position i
    __device__ __forceinline__ void siftDown(int i, unsigned long long va, unsigned long long vb, unsigned vs) {
        for (;;) {
            const int l = 4 * i + 1;
            if (l >= n) break;
            int c = l;
            unsigned long long ca = a[l], cb = b[l];
            if (l + 3 < n) {
                const unsigned long long a1 = a[l + 1], b1 = b[l + 1], a2 = a[l + 2], b2 = b[l + 2], a3 = a[l + 3], b3 = b[l + 3];
                if (a1 < ca || (a1 == ca && b1 < cb)) { c = l + 1; ca = a1; cb = b1; }
                if (a2 < ca || (a2 == ca && b2 < cb)) { c = l + 2; ca = a2; cb = b2; }
                if (a3 < ca || (a3 == ca && b3 < cb)) { c = l + 3; ca = a3; cb = b3; }
            } else {
                for (int k = l + 1; k < n; ++k) {
                    const unsigned long long ak = a[k], bk = b[k];
                    if (ak < ca || (ak == ca && bk < cb)) { c = k; ca = ak; cb = bk; }
                }
            }
            if (!(ca < va || (ca == va && cb < vb))) break;
            a[i] = ca; b[i] = cb; slot[i] = slot[c];
            i = c;
        }
        a[i] = va; b[i] = vb; slot[i] = vs;
    }
    __device__ __forceinline__ void popRoot() {
        --n;
        if (n > 0) siftDown(0, a[n], b[n], slot[n]);
    }
};

// pull a candidate record's line into L1 ahead of its use (no destination register: never waited on)
__device__ __forceinline__ void greedy_touch(const GreedyCand* p) {
    asm volatile("prefetch.global.L1 [%0];" :: "l"(p));
}

struct GreedyCtx {
    DevSystem sys; DevAllocs pairs; GreedyBufs g; int* chosen;
    long long* avail;          // [T] shared memory
    long long* usum;           // [T] shared memory scratch (allocateEqually)
    unsigned char* pool;       // dynamic shared memory
    int lane;
};

// allocate, greedy.go:107-166, over the servers in items[0..n); returns the number of unallocated
// entries written to g.unalloc.  The warp builds the queue; lane 0 runs the sequential pass.
__device__ int greedy_allocate(GreedyCtx& c, const int* items, int n) {
    const int A = c.sys.A;
    GreedyHeap h;
    if ((size_t)n * 20 <= (size_t)c.g.smemBytes) {
        h.a = reinterpret_cast<unsigned long long*>(c.pool);
        h.b = h.a + n;
        h.slot = reinterpret_cast<unsigned*>(h.b + n);
    } else { h.a = c.g.heapA; h.b = c.g.heapB; h.slot = c.g.heapSlot; }
    int hn = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        int i = i0 + c.lane;
        int s = i < n ? items[i] : -1;
        int nc = s >= 0 ? c.g.nCand[s] : 0;
        unsigned m = __ballot_sync(0xffffffffu, nc > 0);
        if (nc > 0) {
            size_t base = (size_t)s * A;
            float v0 = c.g.cand[base].val;
            float d = nc > 1 ? c.g.cand[base + 1].val - v0 : 3.40282346638528859811704183484516925e+38f;
            int pos = hn + __popc(m & ((1u << c.lane) - 1u));
            greedy_keys(c.sys.srv_priority[s], d, v0, -s, h.a[pos], h.b[pos]);
            h.slot[pos] = (unsigned)base;
        }
        hn += __popc(m);
    }
    __syncwarp();
    int nUn = 0;
    if (c.lane == 0) {
        h.n = hn;
        for (int i = (hn - 2) / 4; i >= 0 && hn > 1; --i) h.siftDown(i, h.a[i], h.b[i], h.slot[i]);
        int stampCounter = 1;
        while (h.n > 0) {
            const unsigned slot = h.slot[0];
            const int4 raw = *reinterpret_cast<const int4*>(c.g.cand + slot);
            // the next roots come from the top two levels: start their loads now
            {
                const int lim = h.n < 21 ? h.n : 21;
                for (int q = 1; q < lim; ++q) greedy_touch(c.g.cand + h.slot[q]);
            }
            const int tf = raw.w;
            const int s = (int)(slot / (unsigned)A);
            if (tf & GREEDY_SKIP) { h.popRoot(); continue; }             // no model / GetAccelerator("") == nil
            const int t = tf & 0xffff;
            const long long count = (long long)(((unsigned long long)(unsigned)raw.y << 32) | (unsigned)raw.x);
            if (c.avail[t] >= count) {
                c.avail[t] -= count;
                c.chosen[s] = (int)slot;
                h.popRoot();
                continue;
            }
            if (tf & GREEDY_LAST) { c.g.unalloc[nUn++] = s; h.popRoot(); continue; }
            const GreedyCand nx = c.g.cand[slot + 1];
            const float d = (nx.tf & GREEDY_LAST) ? 3.40282346638528859811704183484516925e+38f : c.g.cand[slot + 2].val - nx.val;
            unsigned long long ka, kb;
            greedy_keys((int)(h.a[0] >> 32), d, nx.val, stampCounter++, ka, kb);
            h.siftDown(0, ka, kb, slot + 1);
        }
    }
    nUn = __shfl_sync(0xffffffffu, nUn, 0);
    __syncwarp();
    return nUn;
}

// scale the chosen candidate to `got` of its `cur` replicas (greedy.go:208-212, :305-311)
__device__ __forceinline__ void greedy_scale(GreedyCtx& c, int s, int slot, long long got, long long cur) {
    const int key = c.g.order[slot];
    const size_t ai = (size_t)s * c.sys.A + key;
    const float factor = (float)got / (float)cur;
    c.pairs.cost[ai] = c.pairs.cost[ai] * factor;
    c.pairs.value[ai] = c.pairs.value[ai] * factor;
    c.pairs.num_replicas[ai] = got;
    c.chosen[s] = slot;
}

// allocateMaximally, greedy.go:194-223, 32 servers of the list at a time: lane l owns server l and a cursor over its
// candidates.  Inside this function `available` only shrinks (a server takes maxReplicas * upr <= available), so a
// candidate without room for one replica now never gets it later and the cursor only moves forward.  The lanes that found
// a candidate are then served in list order; after each one the lanes waiting on the same accelerator type look again
// (same candidate first).  The records of the 32 winners are scaled together at the end (greedy.go:208-212).
__device__ void greedy_allocate_maximally(GreedyCtx& c, const int* list, int n) {
    const unsigned FULL = 0xffffffffu;
    const int A = c.sys.A;
    for (int i0 = 0; i0 < n; i0 += 32) {
        int s = 0, nc = 0;
        if (i0 + c.lane < n) {
            s = list[i0 + c.lane];
            if (c.sys.srv_model[s] >= 0) nc = c.g.nCand[s];
        }
        const size_t slot0 = (size_t)s * A;
        int k = 0, t = -1;
        long long upr = 0, cur = 0;
        // first candidate from k on with room for at least one replica
        auto look = [&]() -> bool {
            for (; k < nc; ++k) {
                t = c.g.ctype[slot0 + k]; upr = c.g.upr[slot0 + k];
                if (t >= 0 && upr > 0) {
                    cur = c.g.rep[slot0 + k];
                    long long maxRep = go_divi(c.avail[t], upr);
                    if (cur < maxRep) maxRep = cur;
                    if (maxRep > 0) return true;
                }
            }
            return false;
        };
        bool has = look();
        long long got = 0, gotCur = 0; int gotSlot = -1;
        for (;;) {
            const unsigned m = __ballot_sync(FULL, has);
            if (!m) break;
            const int f = __ffs(m) - 1;
            if (c.lane == f) {
                long long maxRep = go_divi(c.avail[t], upr);
                if (cur < maxRep) maxRep = cur;
                got = maxRep; gotCur = cur; gotSlot = (int)slot0 + k;
                c.avail[t] -= go_muli(maxRep, upr);
                has = false;
            }
            __syncwarp();
            const int tF = __shfl_sync(FULL, t, f);
            if (has && t == tF) has = look();
        }
        if (gotSlot >= 0) greedy_scale(c, s, gotSlot, got, gotCur);
        __syncwarp();
    }
}

// allocateEqually, greedy.go:239-316
__device__ void greedy_allocate_equally(GreedyCtx& c, const int* list, int n) {
    const int A = c.sys.A;
    GreedyTicket* tk; int* liveIdx;
    if ((size_t)n * (sizeof(GreedyTicket) + 4) <= (size_t)c.g.smemBytes) {
        tk = reinterpret_cast<GreedyTicket*>(c.pool);
        liveIdx = reinterpret_cast<int*>(tk + n);
    } else { tk = c.g.tickets; liveIdx = c.g.liveIdx; }
    // round 1: every present ticket picks the first candidate with room for one replica, then takes its first replica.
    // 32 tickets at a time, as in greedy_allocate_maximally: lane l owns ticket l and a forward-only cursor (`available`
    // only shrinks here), the lanes that found a candidate are served in list order, and after a ticket took its replica
    // the lanes waiting on the same type look again.
    const unsigned FULL = 0xffffffffu;
    int live = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + c.lane;
        int s = 0, nc = 0;
        if (i < n) {
            s = list[i];
            if (c.sys.srv_model[s] >= 0) nc = c.g.nCand[s];
        }
        const size_t slot0 = (size_t)s * A;
        GreedyTicket me; me.upr = 0; me.cur = 0; me.slot = -1; me.got = 0; me.type = -1;
        int k = 0, t = -1;
        long long upr = 0;
        auto look = [&]() -> bool {
            for (; k < nc; ++k) {
                t = c.g.ctype[slot0 + k]; upr = c.g.upr[slot0 + k];
                if (t >= 0 && upr > 0 && c.avail[t] >= upr) return true;
            }
            return false;
        };
        bool has = look();
        bool isLive = false;
        for (;;) {
            const unsigned m = __ballot_sync(FULL, has);
            if (!m) break;
            const int f = __ffs(m) - 1;
            if (c.lane == f) {
                me.slot = (int)slot0 + k; me.upr = upr; me.type = t; me.cur = c.g.rep[slot0 + k];
                // allocatable = min(available/upr, cur) > 0, with upr > 0
                if (me.cur > 0) { me.got = 1; c.avail[t] -= upr; isLive = true; }
                has = false;
            }
            __syncwarp();
            const int tF = __shfl_sync(FULL, t, f);
            if (has && t == tF) has = look();
        }
        const unsigned ml = __ballot_sync(FULL, isLive);
        if (isLive) liveIdx[live + __popc(ml & ((1u << c.lane) - 1u))] = i;
        live += __popc(ml);
        if (i < n) tk[i] = me;
        __syncwarp();
    }
    // later rounds: one replica per live ticket per round, in list order.  A round in which every
    // live ticket is served takes sum(upr) per type, so k = min over types of avail / sum such rounds
    // can be applied at once (same result as running them: nobody drops out before round k+1).
    if (c.lane == 0) {
        const int T = c.sys.T;
        while (live > 0) {
            int w = 0;
            for (int j = 0; j < live; ++j) {
                const int i = liveIdx[j];
                GreedyTicket& me = tk[i];
                if (c.avail[me.type] >= me.upr && me.cur > 0) {
                    me.got++;
                    c.avail[me.type] -= me.upr;
                    liveIdx[w++] = i;
                }
            }
            live = w;
            if (live == 0) break;
            for (int t = 0; t < T; ++t) c.usum[t] = 0;
            for (int j = 0; j < live; ++j) { const GreedyTicket& me = tk[liveIdx[j]]; c.usum[me.type] += me.upr; }
            long long k = 0x7fffffffffffffffLL;
            for (int t = 0; t < T; ++t) if (c.usum[t] > 0) { const long long kt = c.avail[t] / c.usum[t]; if (kt < k) k = kt; }
            if (k > 0 && k < 0x7fffffffffffffffLL) {
                for (int t = 0; t < T; ++t) if (c.usum[t] > 0) c.avail[t] -= k * c.usum[t];
                for (int j = 0; j < live; ++j) tk[liveIdx[j]].got += k;
            }
        }
    }
    __syncwarp();
    for (int i = c.lane; i < n; i += 32) {
        const GreedyTicket me = tk[i];
        if (me.got > 0) greedy_scale(c, list[i], me.slot, me.got, me.cur);
    }
    __syncwarp();
}

// bestEffort, greedy.go:169-190 (list is grouped by priority already)
__device__ void greedy_best_effort(GreedyCtx& c, const int* list, int n, int policy) {
    if (policy == WVA_POLICY_PRIORITY_EXHAUSTIVE) greedy_allocate_maximally(c, list, n);
    else if (policy == WVA_POLICY_ROUND_ROBIN) greedy_allocate_equally(c, list, n);
    else if (policy == WVA_POLICY_PRIORITY_ROUND_ROBIN) {
        int i = 0;
        while (i < n) {                                              // makePriorityGroups, :321-341
            int j = i + 1;
            int pr = c.sys.srv_priority[list[i]];
            while (j < n && c.sys.srv_priority[list[j]] == pr) ++j;
            greedy_allocate_equally(c, list + i, j - i);
            i = j;
        }
    }
}

// Bucket servers by priority (counting sort).  Priorities come from Server.Priority() and are in
// [1,100] (serviceclass.go:28-37, server.go:92-97); wva_system_upload rejects anything else.
__global__ void k_greedy_bucket_count(DevSystem sys, GreedyBufs g) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= sys.S) return;
    atomicAdd(&g.groupStart[sys.srv_priority[s]], 1);
}

// SolveGreedy, greedy.go:35-104: the sequential assignment, one warp.  Every step depends on the
// capacities left by the previous one, so lane 0 walks a priority queue held in shared memory
// (two 64-bit keys + a slot per entry; see greedy_keys); the other lanes help where the reference
// scans a server's candidates or builds lists.  Servers are bucketed by priority first.
__global__ void __launch_bounds__(32) k_greedy_solve(DevSystem sys, DevAllocs pairs, GreedyBufs g, int* chosen,
                                                       int delayedBestEffort, int policy) {
    extern __shared__ __align__(16) unsigned char greedy_pool[];
    __shared__ long long avail[256];
    __shared__ long long usum[256];
    __shared__ int cursor[104];
    if (blockIdx.x != 0) return;
    const int lane = threadIdx.x;
    GreedyCtx c; c.sys = sys; c.pairs = pairs; c.g = g; c.chosen = chosen; c.avail = avail; c.usum = usum; c.pool = greedy_pool; c.lane = lane;
    for (int t = lane; t < sys.T; t += 32) avail[t] = sys.type_capacity[t];
    // groupStart[p] holds the population of priority p (1..100): exclusive prefix sum, then a
    // stable scatter in ascending server index
    if (lane == 0) {
        int run = 0;
        for (int p = 0; p <= 101; ++p) { int cnt = g.groupStart[p]; g.groupStart[p] = run; cursor[p] = run; run += cnt; }
    }
    __syncwarp();
    for (int s0 = 0; s0 < sys.S; s0 += 32) {
        const int s = s0 + lane;
        const int p = s < sys.S ? sys.srv_priority[s] : 101;
        const unsigned peers = __match_any_sync(0xffffffffu, p);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        if (s < sys.S) g.groupItems[cursor[p] + rank] = s;
        __syncwarp();
        if (rank == 0) cursor[p] += __popc(peers);
        __syncwarp();
    }
    __threadfence_block();
    if (delayedBestEffort) {
        // one allocate() over everything (the comparator orders by priority first), then one bestEffort
        int nUn = greedy_allocate(c, g.groupItems, sys.S);
        greedy_best_effort(c, g.unalloc, nUn, policy);
    } else {
        for (int p = 1; p <= 100; ++p) {                              // makePriorityGroups(entries), :96-103
            int lo = g.groupStart[p], hi = g.groupStart[p + 1];
            if (hi <= lo) continue;
            int nUn = greedy_allocate(c, g.groupItems + lo, hi - lo);
            greedy_best_effort(c, g.unalloc, nUn, policy);
        }
    }
}

// ---- greedy, ranked-queue path -----------------------------------------------------------------
// Every entry the reference's sorted slice can ever hold is one of the S*A states (server, position
// in its candidate order), and the key of a state -- priority, delta to the next candidate, value
// -- is fixed once the candidates are sized.  Sorting the states once (bitonic network, all SMs)
// turns the comparator into an integer rank; the queue becomes a bitmap over ranks in shared
// memory (64-ary, 4 levels) and a pop is four find-first-set steps plus one 16-byte record load.
// Only the recency tie-break of greedy_keys is dynamic.  States with one key (a "tie group", e.g.
// zero-load servers on the same accelerator) sort next to each other; among them the reference
// pops the most recently inserted first, the initial entries in ascending server index last.
// That is a stack: a tie group hands its rank range out from the top end downwards, so the entry
// inserted last always holds the smallest occupied rank of the group, and the record stored at a
// rank of a tie group is written when the entry is inserted.

struct GreedyRank {
    unsigned long long* ka;    // [N2] sort key: priority << 32 | ~sortable(delta)
    unsigned* kb;              // [N2]           ~sortable(value)
    unsigned* kslot;           // [N2] payload: state s*A+k, 0xffffffff for padding
    unsigned* posOf;           // [S*A] rank of a state (initial entries of a tie group: the rank handed out)
    int* snext;                // [S*A] where the server's next state goes: -1 none, >= 0 its rank, <= -2: tie group starting at -2-x
    int4* rec;                 // [N2] per rank: { count lo, count hi, tf | priority << 18 | GREEDY_TIE, state }
    int2* nextPos;             // [N2] per rank: { snext of the state stored there, end of the rank's tie group or 0 }
    int* gend;                 // [N2] per rank: end of its tie group, 0 outside tie groups
    int* gbeg;                 // [N2] per rank: start of its tie group (valid where gend != 0)
    int* top;                  // [N2+1] per tie group (indexed by its end): entries currently queued
    int* succ;                 // [S] log of the states placed by the queue loop
    unsigned n2;               // padded length (power of two)
};
constexpr int GREEDY_TIE = 1 << 25;

constexpr int GREEDY_TILE = 2048;

__global__ void k_greedy_states(DevSystem sys, GreedyBufs g, GreedyRank r) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= r.n2) return;
    unsigned long long a = ~0ull; unsigned b = ~0u, slot = ~0u;
    if (i < (unsigned)sys.S * (unsigned)sys.A) {
        const int s = (int)(i / (unsigned)sys.A), k = (int)(i - (unsigned)s * (unsigned)sys.A);
        const int n = g.nCand[s];
        if (k < n) {
            const float v = g.cand[i].val;
            const float d = k + 1 < n ? g.cand[i + 1].val - v : 3.40282346638528859811704183484516925e+38f;
            a = ((unsigned long long)(unsigned)sys.srv_priority[s] << 32) | (unsigned)~f32_sortable(d);
            b = d != d ? 0u : ~f32_sortable(v);           // NaN deltas compare equal without looking at the values (greedy.go:78-80)
            slot = i;
        }
    }
    r.ka[i] = a; r.kb[i] = b; r.kslot[i] = slot;
}

// (key, state) order: equal keys are laid out in ascending state = ascending server index
__device__ __forceinline__ bool greedy_rank_less(unsigned long long a1, unsigned b1, unsigned s1, unsigned long long a2, unsigned b2, unsigned s2) {
    return a1 < a2 || (a1 == a2 && (b1 < b2 || (b1 == b2 && s1 < s2)));
}

// bitonic stages with partner distance < GREEDY_TILE, in shared memory: for k = kLo..kHi (doubling)
// the steps j = min(k/2, TILE/2) .. 1
__global__ void __launch_bounds__(512) k_greedy_bitonic_tile(GreedyRank r, unsigned kLo, unsigned kHi) {
    __shared__ unsigned long long sa[GREEDY_TILE];
    __shared__ unsigned sb[GREEDY_TILE];
    __shared__ unsigned ss[GREEDY_TILE];
    const unsigned base = blockIdx.x * GREEDY_TILE;
    for (unsigned i = threadIdx.x; i < GREEDY_TILE; i += 512) { sa[i] = r.ka[base + i]; sb[i] = r.kb[base + i]; ss[i] = r.kslot[base + i]; }
    __syncthreads();
    for (unsigned k = kLo; k <= kHi; k <<= 1) {
        unsigned j0 = k >> 1; if (j0 > GREEDY_TILE / 2) j0 = GREEDY_TILE / 2;
        for (unsigned j = j0; j > 0; j >>= 1) {
            for (unsigned idx = threadIdx.x; idx < GREEDY_TILE / 2; idx += 512) {
                const unsigned i = 2 * (idx & ~(j - 1)) + (idx & (j - 1));
                const unsigned p = i + j;
                const bool asc = ((base + i) & k) == 0;
                const unsigned long long a1 = sa[i], a2 = sa[p]; const unsigned b1 = sb[i], b2 = sb[p], s1 = ss[i], s2 = ss[p];
                if (greedy_rank_less(a2, b2, s2, a1, b1, s1) == asc && s1 != s2) {
                    sa[i] = a2; sa[p] = a1; sb[i] = b2; sb[p] = b1; ss[i] = s2; ss[p] = s1;
                }
            }
            __syncthreads();
        }
    }
    for (unsigned i = threadIdx.x; i < GREEDY_TILE; i += 512) { r.ka[base + i] = sa[i]; r.kb[base + i] = sb[i]; r.kslot[base + i] = ss[i]; }
}

// one bitonic step (k, j) with j >= GREEDY_TILE, in global memory
__global__ void k_greedy_bitonic_step(GreedyRank r, unsigned k, unsigned j) {
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= r.n2 / 2) return;
    const unsigned i = 2 * (idx & ~(j - 1)) + (idx & (j - 1));
    const unsigned p = i + j;
    const bool asc = (i & k) == 0;
    const unsigned long long a1 = r.ka[i], a2 = r.ka[p]; const unsigned b1 = r.kb[i], b2 = r.kb[p], s1 = r.kslot[i], s2 = r.kslot[p];
    if (greedy_rank_less(a2, b2, s2, a1, b1, s1) == asc && s1 != s2) {
        r.ka[i] = a2; r.ka[p] = a1; r.kb[i] = b2; r.kb[p] = b1; r.kslot[i] = s2; r.kslot[p] = s1;
    }
}

// rank of every state
__global__ void k_greedy_index(GreedyRank r) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= r.n2) return;
    const unsigned slot = r.kslot[i];
    if (slot != ~0u) r.posOf[slot] = i;
}

// last rank of a tie group (two or more states with one key), else false; g0/g1 = its range
__device__ __forceinline__ bool greedy_tie_tail(const GreedyRank& r, unsigned i, unsigned& g0, unsigned& g1) {
    if (i == 0 || i >= r.n2 || r.kslot[i] == ~0u) return false;
    const unsigned long long a = r.ka[i]; const unsigned b = r.kb[i];
    if (i + 1 < r.n2 && r.kslot[i + 1] != ~0u && r.ka[i + 1] == a && r.kb[i + 1] == b) return false;
    if (!(r.ka[i - 1] == a && r.kb[i - 1] == b)) return false;
    unsigned j = i - 1;
    while (j > 0 && r.ka[j - 1] == a && r.kb[j - 1] == b) --j;
    g0 = j; g1 = i + 1;
    return true;
}

// gend[] of every member of a tie group (gend is zeroed before)
__global__ void k_greedy_tie_groups(GreedyRank r) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned g0, g1;
    if (!greedy_tie_tail(r, i, g0, g1)) return;
    for (unsigned q = g0; q < g1; ++q) { r.gend[q] = (int)g1; r.gbeg[q] = (int)g0; }
}

__device__ __forceinline__ int4 greedy_make_rec(const GreedyCand& cd, int priority, int tie, unsigned slot) {
    int4 v;
    v.x = (int)(unsigned)((unsigned long long)cd.count & 0xffffffffull);
    v.y = (int)(unsigned)((unsigned long long)cd.count >> 32);
    v.z = cd.tf | (priority << 18) | tie;
    v.w = (int)slot;
    return v;
}

// per state: where the following state of the server goes; per rank: the state sorted there
__global__ void k_greedy_records(DevSystem sys, GreedyBufs g, GreedyRank r) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= r.n2) return;
    const unsigned slot = r.kslot[i];
    if (slot == ~0u) return;
    const GreedyCand cd = g.cand[slot];
    int nx = -1;
    if (!(cd.tf & GREEDY_LAST)) {
        const unsigned q = r.posOf[slot + 1];
        nx = r.gend[q] ? -2 - r.gbeg[q] : (int)q;
    }
    r.snext[slot] = nx;
    r.rec[i] = greedy_make_rec(cd, (int)(r.ka[i] >> 32), r.gend[i] ? GREEDY_TIE : 0, slot);
    r.nextPos[i] = make_int2(nx, r.gend[i]);
}

// the initial entries (first candidates) of a tie group take its top ranks in ascending server index
__global__ void k_greedy_tie_init(DevSystem sys, GreedyBufs g, GreedyRank r) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned g0, g1;
    if (!greedy_tie_tail(r, i, g0, g1)) return;
    const unsigned A = (unsigned)sys.A;
    int cnt = 0;
    for (unsigned q = g0; q < g1; ++q) if (r.kslot[q] % A == 0) ++cnt;
    const int pr = (int)(r.ka[i] >> 32);
    int idx = 0;
    for (unsigned q = g0; q < g1; ++q) {
        const unsigned slot = r.kslot[q];
        if (slot % A != 0) continue;
        const unsigned pos = g1 - (unsigned)cnt + (unsigned)idx++;
        r.posOf[slot] = pos;
        r.rec[pos] = greedy_make_rec(g.cand[slot], pr, GREEDY_TIE, slot);
        r.nextPos[pos] = make_int2(r.snext[slot], (int)g1);
    }
    r.top[g1] = cnt;
}

// 64-ary bitmap over ranks, four levels (up to 2^24 ranks)
struct GreedyBitmap {
    unsigned long long* l0; unsigned long long* l1; unsigned long long* l2; unsigned long long* l3;
    __device__ __forceinline__ int findMin() const {          // -1 when empty
        const unsigned long long w3 = l3[0];
        if (!w3) return -1;
        int i = __ffsll((long long)w3) - 1;
        i = i * 64 + __ffsll((long long)l2[i]) - 1;
        i = i * 64 + __ffsll((long long)l1[i]) - 1;
        i = i * 64 + __ffsll((long long)l0[i]) - 1;
        return i;
    }
    // smallest set rank > p, -1 when there is none
    __device__ __forceinline__ int nextAfter(int p) const {
        int w = p >> 6;
        unsigned long long bits = (p & 63) == 63 ? 0ull : (l0[w] & (~0ull << ((p & 63) + 1)));
        if (bits) return w * 64 + __ffsll((long long)bits) - 1;
        int i1 = w >> 6;
        bits = (w & 63) == 63 ? 0ull : (l1[i1] & (~0ull << ((w & 63) + 1)));
        if (!bits) {
            int i2 = i1 >> 6;
            bits = (i1 & 63) == 63 ? 0ull : (l2[i2] & (~0ull << ((i1 & 63) + 1)));
            if (!bits) {
                bits = (i2 & 63) == 63 ? 0ull : (l3[0] & (~0ull << ((i2 & 63) + 1)));
                if (!bits) return -1;
                i2 = __ffsll((long long)bits) - 1;
                bits = l2[i2];
            }
            i1 = i2 * 64 + __ffsll((long long)bits) - 1;
            bits = l1[i1];
        }
        w = i1 * 64 + __ffsll((long long)bits) - 1;
        return w * 64 + __ffsll((long long)l0[w]) - 1;
    }
    __device__ __forceinline__ void set(int p) {
        const unsigned long long w = l0[p >> 6];
        l0[p >> 6] = w | (1ull << (p & 63));
        if (w) return;                                   // the upper levels already know this word
        l1[p >> 12] |= 1ull << ((p >> 6) & 63);
        l2[p >> 18] |= 1ull << ((p >> 12) & 63);
        l3[0] |= 1ull << ((p >> 18) & 63);
    }
    __device__ __forceinline__ void clear(int p) {
        unsigned long long w = l0[p >> 6] & ~(1ull << (p & 63));
        l0[p >> 6] = w;
        if (w) return;
        w = l1[p >> 12] & ~(1ull << ((p >> 6) & 63));
        l1[p >> 12] = w;
        if (w) return;
        w = l2[p >> 18] & ~(1ull << ((p >> 12) & 63));
        l2[p >> 18] = w;
        if (w) return;
        l3[0] &= ~(1ull << ((p >> 18) & 63));
    }
};

__host__ __device__ inline size_t greedy_bitmap_bytes(size_t nStates, size_t* w0, size_t* w1, size_t* w2) {
    const size_t a = (nStates + 63) / 64, b = (a + 63) / 64, c = (b + 63) / 64;
    if (w0) *w0 = a; if (w1) *w1 = b; if (w2) *w2 = c;
    return (a + b + c + 1) * 8;
}

// SolveGreedy on the ranked queue.  With the priority in the top key bits one queue serves all
// priority groups: the group boundary (greedy.go:96-103) is where the popped priority changes.
__global__ void __launch_bounds__(32) k_greedy_solve_ranked(DevSystem sys, DevAllocs pairs, GreedyBufs g, GreedyRank r, int* chosen,
                                                              int delayedBestEffort, int policy) {
    extern __shared__ __align__(16) unsigned char greedy_pool[];
    __shared__ long long avail[256];
    __shared__ long long usum[256];
    if (blockIdx.x != 0) return;
    const int lane = threadIdx.x;
    const int A = sys.A;
    size_t w0, w1, w2;
    const size_t bmBytes = greedy_bitmap_bytes((size_t)sys.S * A, &w0, &w1, &w2);
    GreedyBitmap bm;
    bm.l0 = reinterpret_cast<unsigned long long*>(greedy_pool);
    bm.l1 = bm.l0 + w0; bm.l2 = bm.l1 + w1; bm.l3 = bm.l2 + w2;
    GreedyCtx c; c.sys = sys; c.pairs = pairs; c.g = g; c.chosen = chosen; c.avail = avail; c.usum = usum; c.lane = lane;
    c.pool = greedy_pool + ((bmBytes + 15) & ~(size_t)15);
    c.g.smemBytes = g.smemBytes - (int)((bmBytes + 15) & ~(size_t)15);
    for (int t = lane; t < sys.T; t += 32) avail[t] = sys.type_capacity[t];
    for (size_t i = lane; i < w0 + w1 + w2 + 1; i += 32) bm.l0[i] = 0;
    __syncwarp();
    // every server with a candidate starts at its first one (greedy.go:45-73)
    for (int s = lane; s < sys.S; s += 32)
        if (g.nCand[s] > 0) {
            const unsigned p = r.posOf[(size_t)s * A];
            atomicOr(&bm.l0[p >> 6], 1ull << (p & 63));
        }
    __syncwarp();
    for (size_t i = lane; i < w0; i += 32) if (bm.l0[i]) atomicOr(&bm.l1[i >> 6], 1ull << (i & 63));
    __syncwarp();
    for (size_t i = lane; i < w1; i += 32) if (bm.l1[i]) atomicOr(&bm.l2[i >> 6], 1ull << (i & 63));
    __syncwarp();
    for (size_t i = lane; i < w2; i += 32) if (bm.l2[i]) atomicOr(&bm.l3[0], 1ull << (i & 63));
    __syncwarp();

    int curPr = -1;
    unsigned long long nPops = 0, nFails = 0, cycQueue = 0, cycBest = 0;
    int nSucc = 0;                       // placements are logged (r.succ) and scattered to chosen[] at the end
    // lane 0 keeps the bitmap word that holds the minimum in a register (cw, cb): a pop is one
    // find-first-set unless the word runs empty, and the record of the following set bit is loaded
    // one iteration ahead.  A server whose placement fails moves to its next candidate; when that
    // state ranks before everything queued (the usual case: the reference re-inserts it at the
    // head of the slice) it is simply evaluated next, reading the server's contiguous candidate
    // records, without going through the queue.
    int cw = -1; unsigned long long cb = 0;
    int pfPos = -1; int2 pfNx = make_int2(0, 0); int4 pfRec = make_int4(0, 0, 0, 0);
    for (;;) {
        int nUn = 0, more = 0, nextPr = -1;
        const long long t0 = clock64();
        if (lane == 0) {
            for (;;) {
                if (cb == 0) {
                    const int m0 = bm.findMin();
                    if (m0 < 0) break;
                    cw = m0 >> 6; cb = bm.l0[cw];
                }
                const int p = cw * 64 + __ffsll((long long)cb) - 1;
                int4 rec; int2 nx;
                if (p == pfPos) { rec = pfRec; nx = pfNx; }
                else { rec = r.rec[p]; nx = r.nextPos[p]; }
                const unsigned long long rest = cb & (cb - 1);            // without p
                if (rest) {
                    pfPos = cw * 64 + __ffsll((long long)rest) - 1;
                    pfRec = r.rec[pfPos]; pfNx = r.nextPos[pfPos];
                } else pfPos = -1;
                int tf = rec.z;
                const int pr = (tf >> 18) & 0x7f;
                if (!delayedBestEffort && pr != curPr) {
                    if (curPr < 0) curPr = pr;
                    else { more = 1; nextPr = pr; break; }
                }
                ++nPops;
                // take p out; m = what the queue holds next (-1: nothing)
                cb = rest;
                bm.l0[cw] = rest;
                int m;
                if (rest) m = pfPos;
                else {
                    bm.clear(p);                                          // propagate the empty word upwards
                    m = bm.findMin();
                    if (m >= 0) { cw = m >> 6; cb = bm.l0[cw]; }
                }
                if (nx.y) r.top[nx.y] = nx.y - p - 1;                     // tie group: p was its lowest occupied rank
                int state = rec.w, np = nx.x;
                // a failed placement walks through the server's following candidates: start pulling their lines in now
                // (one line holds a server's 8 candidate records; fire and forget)
                if (!(tf & GREEDY_LAST)) {
                    asm volatile("prefetch.global.L1 [%0];" :: "l"(g.cand + state + 1));
                    asm volatile("prefetch.global.L1 [%0];" :: "l"(r.snext + state + 1));
                }
                long long count = (long long)(((unsigned long long)(unsigned)rec.y << 32) | (unsigned)rec.x);
                for (;;) {
                    if (tf & GREEDY_SKIP) break;                          // no model / GetAccelerator("") == nil
                    const int t = tf & 0xffff;
                    if (avail[t] >= count) {
                        avail[t] -= count;
                        r.succ[nSucc++] = state;
                        break;
                    }
                    ++nFails;
                    if (np == -1) { g.unalloc[nUn++] = state; break; }    // state for now, server below
                    // does the next state go to the head of the queue?  A tie group hands out the rank
                    // below its lowest occupied one, so it does as soon as the queue starts inside or
                    // after the group.
                    const bool front = m < 0 || (np >= 0 ? np < m : m >= -2 - np);
                    ++state;
                    if (front) {
                        const int4 cd = *reinterpret_cast<const int4*>(g.cand + state);
                        np = r.snext[state];
                        count = (long long)(((unsigned long long)(unsigned)cd.y << 32) | (unsigned)cd.x);
                        tf = cd.w;
                        continue;
                    }
                    int q = np;
                    if (np < -1) {
                        const int g1 = r.gend[-2 - np];
                        const int depth = r.top[g1];
                        r.top[g1] = depth + 1;
                        q = g1 - 1 - depth;
                        r.rec[q] = greedy_make_rec(g.cand[state], pr, GREEDY_TIE, (unsigned)state);
                        r.nextPos[q] = make_int2(r.snext[state], g1);
                    }
                    bm.set(q);                                            // q > m: the cached word stays the minimum's
                    if ((q >> 6) == cw) cb |= 1ull << (q & 63);
                    break;
                }
            }
        }
        nUn = __shfl_sync(0xffffffffu, nUn, 0);
        more = __shfl_sync(0xffffffffu, more, 0);
        nextPr = __shfl_sync(0xffffffffu, nextPr, 0);
        __syncwarp();
        for (int i = lane; i < nUn; i += 32) g.unalloc[i] = (int)((unsigned)g.unalloc[i] / (unsigned)A);
        __syncwarp();
        const long long t1 = clock64();
        if (!delayedBestEffort || !more) greedy_best_effort(c, g.unalloc, nUn, policy);
        cycQueue += (unsigned long long)(t1 - t0);
        cycBest += (unsigned long long)(clock64() - t1);
        if (!more) break;
        curPr = nextPr;
    }
    nSucc = __shfl_sync(0xffffffffu, nSucc, 0);
    __syncwarp();
    for (int i = lane; i < nSucc; i += 32) { const int state = r.succ[i]; chosen[(unsigned)state / (unsigned)A] = state; }
    if (lane == 0) { g.stats[0] = nPops; g.stats[1] = nFails; g.stats[2] = cycQueue; g.stats[3] = cycBest; }
}

// copy the chosen candidates out (after best-effort scaling)
__global__ void k_greedy_collect(DevSystem sys, DevAllocs pairs, const int* __restrict__ order, const int* __restrict__ chosen_key, int* __restrict__ chosen_acc,
                                 DevAllocs chosen) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= sys.S) return;
    const int slot = chosen_key[s];              // s*A + position in the greedy order, or -1
    const int key = slot >= 0 ? order[slot] : -1;
    chosen_acc[s] = key;
    store_alloc(chosen, (size_t)s, key >= 0 ? load_alloc(pairs, (size_t)s * sys.A + key) : empty_alloc());
}

}  // namespace wva

#include "wva_grid_scan.cuh"
#include "wva_greedy_scan.cuh"
