/*
 * wva_b200.h — C-ABI of the B200-native Analyze -> Optimize hot path of the
 * Workload-Variant-Autoscaler (llm-d-incubation/inferno-autoscaler).
 *
 * The reference is pure Go (CGO_ENABLED=0, Dockerfile:25) and has no FFI for this
 * path.  This header is the boundary a cgo shim binds (see INTEGRATION.md and go/):
 * every entry point names the reference Go function(s) it replaces, file:line
 * relative to the reference tree.
 *
 * Conventions
 *   - plain C99 POD, no callbacks, no retained caller pointers: every call copies
 *     what it needs before returning (cgo pointer rules).
 *   - return 0 (WVA_OK) or a negative WVA_E* code; never aborts, never prints.
 *     wva_last_error(ctx) gives a human readable message for the last failure.
 *   - one in-flight call per ctx (the reference path is non re-entrant too: it goes
 *     through package globals core.TheSystem / analyzer.Model, pkg/core/system.go:12,
 *     pkg/analyzer/utils.go:73).
 *   - strings (accelerator, type, model, class, server names) are interned to dense
 *     indices by the host side; the native side sees integers only.
 *   - there is NO CPU fallback: every compute entry point launches sm_100a kernels
 *     and fails with WVA_ECUDA when no device is usable.
 *
 * Arithmetic contract: float32/float64 typing, operation order and rounding points
 * are those of the reference (pkg/analyzer, pkg/core/allocation.go); results are
 * bit-identical to the Go implementation for finite inputs.
 */
#ifndef WVA_B200_H
#define WVA_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WVA_ABI_VERSION 1

/* ---- status codes ------------------------------------------------------- */
#define WVA_OK          0
#define WVA_EINVAL     -1   /* bad argument / inconsistent sizes                    */
#define WVA_ECUDA      -2   /* CUDA runtime failure (no device, OOM, launch error) */
#define WVA_ESTATE     -3   /* call order violated (e.g. solve before analyze)     */
#define WVA_ENOSOLUTION -4  /* "no feasible allocations found" (internal/optimizer/optimizer.go:38-40) */
#define WVA_ENONFINITE -5   /* an input on which the reference itself does not terminate (wva_model_solve) */

/* ---- tunables (package vars of the reference; part of the parity contract) */
#define WVA_MAX_QUEUE_TO_BATCH_RATIO 10      /* pkg/config/defaults.go:18 */
#define WVA_ACCEL_PENALTY_FACTOR     0.1f    /* pkg/config/defaults.go:21 */
#define WVA_EPSILON                  0.001f  /* pkg/analyzer/queueanalyzer.go:8  */
#define WVA_STABILITY_SAFETY         0.1f    /* pkg/analyzer/queueanalyzer.go:11 */
#define WVA_BISECT_TOL               1e-6f   /* pkg/analyzer/utils.go:8 */
#define WVA_BISECT_MAXIT             100     /* pkg/analyzer/utils.go:9 */
#define WVA_DEFAULT_PRIORITY         100     /* pkg/config/defaults.go:27-33 */

/* ---- saturation policies: pkg/config/config.go:4-41 ---------------------- */
#define WVA_POLICY_NONE                 0
#define WVA_POLICY_PRIORITY_EXHAUSTIVE  1
#define WVA_POLICY_PRIORITY_ROUND_ROBIN 2
#define WVA_POLICY_ROUND_ROBIN          3

/* ---- special accelerator indices ---------------------------------------- */
#define WVA_ACC_NONE    (-1)  /* the empty accelerator name ""                     */
#define WVA_ACC_UNKNOWN (-2)  /* a non-empty name that is not in the accelerator map */

/*
 * System image, structure of arrays (host pointers; the library copies).
 * Source of truth for the fields: pkg/config/types.go:29-37 (AcceleratorSpec),
 * :64-84 (ModelAcceleratorPerfData), :92-104 (ServiceClassSpec/ModelTarget),
 * :112-139 (ServerSpec/AllocationData/ServerLoadSpec), :52-61 (capacity).
 * The per-server SLO/priority arrays are the (class, model) lookups of
 * pkg/core/allocation.go:64-70 and pkg/core/server.go:92-97 resolved by the host.
 */
typedef struct wva_system_soa {
    int32_t n_servers;   /* S */
    int32_t n_accels;    /* A */
    int32_t n_models;    /* M */
    int32_t n_types;     /* T */

    /* accelerators [A] */
    const float*   acc_cost;          /* AcceleratorSpec.Cost                       */
    const int32_t* acc_multiplicity;  /* AcceleratorSpec.Multiplicity               */
    const int32_t* acc_type;          /* dense index of AcceleratorSpec.Type, [0,T) */

    /* accelerator types [T] */
    const int64_t* type_capacity;     /* System.capacity[type]; a type absent from the map is 0 */

    /* model x accelerator perf table [M*A], row-major by model */
    const float*   perf_alpha;        /* DecodeParms.Alpha   */
    const float*   perf_beta;         /* DecodeParms.Beta    */
    const float*   perf_gamma;        /* PrefillParms.Gamma  */
    const float*   perf_delta;        /* PrefillParms.Delta  */
    const int32_t* perf_max_batch;    /* MaxBatchSize        */
    const int32_t* perf_at_tokens;    /* AtTokens            */
    const int32_t* perf_acc_count;    /* AccCount (<=0 means 1, pkg/core/model.go:45-54) */
    const uint8_t* perf_valid;        /* model.PerfData(acc) != nil */

    /* servers [S] */
    const int32_t* srv_model;         /* dense model index, -1 = model not in system  */
    const float*   srv_arrival_rpm;   /* ServerLoadSpec.ArrivalRate (req/min)         */
    const int32_t* srv_in_tokens;     /* AvgInTokens                                  */
    const int32_t* srv_out_tokens;    /* AvgOutTokens                                 */
    const float*   srv_slo_ttft;      /* Target.TTFT                                  */
    const float*   srv_slo_itl;       /* Target.ITL                                   */
    const float*   srv_slo_tps;       /* Target.TPS                                   */
    const uint8_t* srv_target_valid;  /* service class exists AND has a target for the model */
    const int32_t* srv_priority;      /* Server.Priority(): class priority or 100     */
    const int32_t* srv_min_replicas;  /* ServerSpec.MinNumReplicas                    */
    const int32_t* srv_max_batch;     /* ServerSpec.MaxBatchSize override, 0 = none   */
    const uint8_t* srv_keep_acc;      /* ServerSpec.KeepAccelerator                   */
    const int32_t* srv_cur_acc;       /* CurrentAlloc.Accelerator: index, WVA_ACC_NONE, WVA_ACC_UNKNOWN */
    const int32_t* srv_cur_replicas;  /* CurrentAlloc.NumReplicas                     */
    const float*   srv_cur_cost;      /* CurrentAlloc.Cost                            */
} wva_system_soa;

/*
 * Allocation records, structure of arrays (caller-allocated, length n).
 * Mirrors core.Allocation (pkg/core/allocation.go:13-24).
 */
typedef struct wva_alloc_soa {
    int32_t* acc;           /* Allocation.accelerator as index; WVA_ACC_NONE for the zero-replica zero-load record */
    int64_t* num_replicas;  /* Go int */
    int64_t* batch_size;    /* Go int */
    float*   cost;
    float*   value;
    float*   itl;
    float*   ttft;
    float*   rho;
    float*   max_arrv_rate_per_replica;  /* req/msec */
} wva_alloc_soa;

/* analyzer.AnalysisMetrics, pkg/analyzer/queueanalyzer.go:61-71 (same field order) */
typedef struct wva_metrics {
    float throughput;       /* req/sec */
    float avg_resp_time;    /* msec */
    float avg_wait_time;    /* msec */
    float avg_num_in_serv;
    float avg_prefill_time; /* msec */
    float avg_token_time;   /* msec */
    float max_rate;         /* req/sec */
    float rho;
} wva_metrics;

/* candidate status byte of the grid sweep */
#define WVA_CAND_OK          0  /* Analyze succeeded                                            */
#define WVA_CAND_FEASIBLE    1  /* bit 0 set: Analyze succeeded AND all SLO/replica constraints hold */
#define WVA_CAND_ERR_PAIR    2  /* pair lookups fail (allocation.go:41-70) or not a candidate accelerator (server.go:70-82) */
#define WVA_CAND_ERR_CONFIG  4  /* NewQueueAnalyzer rejects (queueanalyzer.go:337-352)          */
#define WVA_CAND_ERR_RATE_LE0 6 /* Analyze: rate <= 0 (queueanalyzer.go:135-137)                */
#define WVA_CAND_ERR_RATE_MAX 8 /* Analyze: rate > RateRange.Max (:140-143)                     */
#define WVA_CAND_ERR_MODEL   10 /* Analyze: model invalid (:147-150)                            */

/* per-server winner of the grid sweep */
typedef struct wva_grid_best {
    int32_t acc;        /* accelerator index, -1 when no candidate is feasible */
    int32_t replicas;
    int32_t batch;
    float   cost;       /* acc.Cost * float32(numInstances * replicas)         */
    float   value;      /* TransitionPenalty(current -> candidate)             */
    float   itl;
    float   ttft;
    float   rho;
} wva_grid_best;

typedef struct wva_optimizer_spec {   /* pkg/config/types.go:151-155 */
    int32_t unlimited;
    int32_t delayed_best_effort;
    int32_t saturation_policy;        /* WVA_POLICY_*; SaturatedAllocationPolicyEnum(string) done by host */
} wva_optimizer_spec;

typedef struct wva_ctx wva_ctx;

/* ---- lifecycle ----------------------------------------------------------- */

/* Create a context bound to one CUDA device (one process per GPU).  The only slow
 * call (CUDA context creation); the Go side makes it once per process. */
int  wva_ctx_create(int device, wva_ctx** out);
void wva_ctx_destroy(wva_ctx* ctx);
const char* wva_last_error(const wva_ctx* ctx);   /* ctx may be NULL: returns the create error */
int  wva_abi_version(void);

/* Replaces core.NewSystem + System.SetFromSpec (pkg/core/system.go:67-90) and the
 * manager.NewManager side effect core.TheSystem = system (pkg/manager/manager.go:13-19).
 * Uploads the image to HBM; invalidates previous analysis. */
int wva_system_upload(wva_ctx* ctx, const wva_system_soa* host);

/* Incremental updates of the RESIDENT image (System.AddServerFromSpec / RemoveServer / SetCountFromSpec /
 * Model.AddPerfDataFromSpec, pkg/core/system.go:99-171, model.go:45-54): only the touched rows cross PCIe.
 * wva_system_upload lays the arrays out with spare rows (1/16 more, at least 64); an update that would
 * outgrow them fails with WVA_ECAPACITY and the caller uploads the whole image again.  Every update
 * invalidates previous analysis results and resets the shard to "everything".
 *   wva_system_update_servers: overwrite server rows [first, first+count) from rows->srv_* (arrays of
 *       `count` entries; rows->n_servers == count); first + count may extend the image (first <= S);
 *   wva_system_update_models:  overwrite the perf rows of models [first, first+count) from rows->perf_*
 *       (count * A entries; rows->n_models == count); may extend M the same way;
 *   wva_system_remove_server:  the last server's row moves into `index` (device-side), S shrinks by one --
 *       the host keeps its name -> index map in step;
 *   wva_system_set_capacity:   the T capacity counters.
 * wva_upload_bytes: bytes the last upload / update call moved host -> device. */
#define WVA_ECAPACITY  -6   /* the resident image has no spare row left: upload again */
int wva_system_update_servers(wva_ctx* ctx, int32_t first, int32_t count, const wva_system_soa* rows);
int wva_system_update_models(wva_ctx* ctx, int32_t first, int32_t count, const wva_system_soa* rows);
int wva_system_remove_server(wva_ctx* ctx, int32_t index);
int wva_system_set_capacity(wva_ctx* ctx, const int64_t* type_capacity);
int64_t wva_upload_bytes(const wva_ctx* ctx);
int wva_system_dims(const wva_ctx* ctx, int32_t* n_servers, int32_t* n_accels, int32_t* n_models, int32_t* n_types);

/* cgo-callable forms.  cgo forbids passing a Go pointer to memory that itself holds Go pointers
 * ("cgo argument has Go pointer to unpinned Go pointer"): a Go-allocated wva_system_soa / wva_alloc_soa
 * whose fields point at Go slices cannot be passed as-is.  These variants take every array as its own
 * argument -- each is a pointer to pointer-free memory, which cgo allows without pinning -- and are
 * otherwise identical to wva_system_upload / wva_analyze_pairs / wva_pairs_fetch / wva_solve.  (The struct
 * forms remain for C, C++ and ctypes callers, and for Go callers that pin with runtime.Pinner.) */
int wva_system_upload_arrays(wva_ctx* ctx, int32_t n_servers, int32_t n_accels, int32_t n_models, int32_t n_types,
        const float* acc_cost, const int32_t* acc_multiplicity, const int32_t* acc_type, const int64_t* type_capacity,
        const float* perf_alpha, const float* perf_beta, const float* perf_gamma, const float* perf_delta,
        const int32_t* perf_max_batch, const int32_t* perf_at_tokens, const int32_t* perf_acc_count, const uint8_t* perf_valid,
        const int32_t* srv_model, const float* srv_arrival_rpm, const int32_t* srv_in_tokens, const int32_t* srv_out_tokens,
        const float* srv_slo_ttft, const float* srv_slo_itl, const float* srv_slo_tps, const uint8_t* srv_target_valid,
        const int32_t* srv_priority, const int32_t* srv_min_replicas, const int32_t* srv_max_batch, const uint8_t* srv_keep_acc,
        const int32_t* srv_cur_acc, const int32_t* srv_cur_replicas, const float* srv_cur_cost);
int wva_analyze_pairs_arrays(wva_ctx* ctx, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica, uint8_t* feasible);
int wva_pairs_fetch_arrays(wva_ctx* ctx, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica, uint8_t* feasible);
int wva_solve_arrays(wva_ctx* ctx, int32_t unlimited, int32_t delayed_best_effort, int32_t saturation_policy,
        int32_t* chosen_acc, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica);
/* ... and of wva_grid_pairs_fetch / wva_solve_grid (sweep winners per pair, below) */
int wva_grid_pairs_fetch_arrays(wva_ctx* ctx, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica, uint8_t* feasible);
int wva_solve_grid_arrays(wva_ctx* ctx, int32_t unlimited, int32_t delayed_best_effort, int32_t saturation_policy,
        int32_t* chosen_acc, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost, float* value,
        float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica);
/* ... and of wva_analyze_scenarios / wva_scenario_pairs_fetch (load scenarios, below) */
int wva_analyze_scenarios_arrays(wva_ctx* ctx, int32_t n_scen, const float* arrival_rpm, int32_t* chosen_acc, int32_t* acc,
        int64_t* num_replicas, int64_t* batch_size, float* cost, float* value, float* itl, float* ttft, float* rho,
        float* max_arrv_rate_per_replica, int64_t* type_count, float* type_cost);
int wva_scenario_pairs_fetch_arrays(wva_ctx* ctx, int32_t scen, int32_t* acc, int64_t* num_replicas, int64_t* batch_size, float* cost,
        float* value, float* itl, float* ttft, float* rho, float* max_arrv_rate_per_replica, uint8_t* feasible);

/* Multi-GPU sharding (SURVEY 8e): this rank owns servers [first, first+count) of the
 * uploaded image; analysis kernels touch only those; solve/allocate_by_type produce the
 * rank's partial results.  Default shard = everything. */
int wva_set_shard(wva_ctx* ctx, int32_t first_server, int32_t count);

/* ---- Analyze ------------------------------------------------------------- */

/* Replaces Server.Calculate for all servers (pkg/core/server.go:55-67), i.e. one
 * core.CreateAllocation (pkg/core/allocation.go:27-163) per (server, accelerator)
 * followed by value = curAllocation.TransitionPenalty(alloc) (:291-300).
 * out has S*A records (server-major); feasible[s*A+a] = 1 when CreateAllocation
 * returned non-nil and the accelerator is a candidate for the server.  Results stay
 * resident on the device for wva_solve.  out / feasible may be NULL (device only). */
int wva_analyze_pairs(wva_ctx* ctx, wva_alloc_soa* out, uint8_t* feasible);

/* Candidate sweep (north_star): for every (server, accelerator, replicas r in 1..r_max,
 * batch b in 1..b_max) evaluate
 *     analyzer.NewQueueAnalyzer({MaxBatchSize b, MaxQueueSize 10 b}, {in, out})  (queueanalyzer.go:87-131)
 *     .Analyze(totalRate / float32(r))                                            (queueanalyzer.go:134-174)
 * with totalRate as in allocation.go:134-139, test the SLOs, and reduce per server to the
 * feasible candidate of minimum (value, accelerator, replicas, batch), value being the
 * transition penalty of cost = acc.Cost * float32(numInstances * r).
 *   best    [S]                 per-server winner (may be NULL)
 *   cube    [S*A*r_max*b_max]   full metrics, index ((s*A+a)*r_max+(r-1))*b_max+(b-1)  (may be NULL)
 *   status  [S*A*r_max*b_max]   WVA_CAND_* per candidate                                (may be NULL)
 * cube/status are HOST pointers; use wva_analyze_grid_device to keep them in HBM. */
int wva_analyze_grid(wva_ctx* ctx, int32_t r_max, int32_t b_max,
                     wva_grid_best* best, wva_metrics* cube, uint8_t* status);

/* Same sweep, results left in HBM (cube only materialised when want_cube != 0).
 * wva_grid_fetch copies the per-server winners to the host. */
int wva_analyze_grid_device(wva_ctx* ctx, int32_t r_max, int32_t b_max, int32_t want_cube);
int wva_grid_fetch(wva_ctx* ctx, wva_grid_best* best);

/* Both halves of Analyze in one call: wva_analyze_pairs and wva_analyze_grid_device are independent
 * and are run concurrently (the sweep on its own stream).  Results stay in HBM:
 * wva_pairs_fetch / wva_grid_fetch copy them out, wva_solve consumes the pair records in place. */
int wva_analyze(wva_ctx* ctx, int32_t r_max, int32_t b_max, int32_t want_cube);
int wva_pairs_fetch(wva_ctx* ctx, wva_alloc_soa* out, uint8_t* feasible);

/* Sweep winners per (server, accelerator) pair, as solver input.  With wva_grid_set_pair_winners(ctx, 1)
 * (default 0) every sweep (wva_analyze_grid, wva_analyze_grid_device, wva_analyze, wva_group_analyze) also
 * leaves S*A candidate records in HBM, laid out like the pair records of wva_analyze_pairs (a rank fills its
 * shard rows).  The record of pair (s, a) is the sweep's feasible candidate of that pair with the smallest
 * (value, replicas, batch) -- the per-server winner of wva_grid_best is the best of its pairs' records:
 *     acc = a, num_replicas = r, batch_size = b,
 *     cost  = acc.Cost * float32(numInstances * r), value = the transition penalty (as wva_grid_best),
 *     itl, ttft, rho of the candidate (as wva_grid_best),
 *     max_arrv_rate_per_replica = (totalRate / float32(r)) / 1000: the per-replica rate, req/msec, the candidate
 *         was analysed at.  The sweep runs no QueueAnalyzer.Size, so this is NOT the SLO-bound rate that
 *         CreateAllocation records there (allocation.go:141-160); the greedy does not read the field.
 * feasible[s*A+a] = 0 (record empty, acc = WVA_ACC_NONE) when the pair has no feasible candidate: no load, not
 * a candidate accelerator, or no (r, b) in the sweep's extents meets the SLOs.
 * The records are invalidated by any image upload / update / shard change and by a sweep with the option off;
 * a limited-capacity wva_solve_grid consumes them (best-effort scaling writes them in place).  They are
 * independent of the pair records of wva_analyze_pairs.
 *   wva_grid_pairs_fetch: copy the shard's records out (rows of other shards untouched), like wva_pairs_fetch;
 *   wva_solve_grid: wva_solve (same unlimited argmin, same greedy paths, policies and delayed best-effort,
 *       pkg/solver/solver.go:32-79, greedy.go:35-341) over the sweep records instead of the pair records.
 *       It writes the same solution, so wva_allocate_by_type and wva_solution_time_usec work after it.  With a
 *       communicator attached a limited solve all-gathers the records like wva_solve; without one it needs
 *       the whole image as its shard.  WVA_ESTATE when no valid sweep records exist. */
int wva_grid_set_pair_winners(wva_ctx* ctx, int32_t on);
int wva_grid_pairs_fetch(wva_ctx* ctx, wva_alloc_soa* out, uint8_t* feasible);
int wva_solve_grid(wva_ctx* ctx, const wva_optimizer_spec* spec, int32_t* chosen_acc, wva_alloc_soa* chosen);

/* QueueAnalyzer.Size for every sweep record of the shard, at the record's own batch size.  For each pair (s, a) of
 * the shard with a valid record of batch size b, what CreateAllocation computes at allocation.go:81-131 with N = b:
 *     analyzer.NewQueueAnalyzer({MaxBatchSize b, MaxQueueSize 10 b, alpha beta gamma delta of (model, a)}, {in, out})
 *     .Size({TTFT, ITL, TPS of the server})                                           (queueanalyzer.go:185-255)
 * When Size succeeds, the record's max_arrv_rate_per_replica becomes float32(metrics.Throughput / 1000) (req/msec, as
 * allocation.go:131, :160), so that MaxRPM / Saturated (allocation.go:233, :254) and the analyzer response see the
 * SLO-bound rate; no other field changes.
 *   status[s*A+a] (host, may be NULL; rows of other shards untouched): 0 = no record, 1 = sized, 2 = Size returned an
 *       error and the record keeps the rate it was analysed at (e.g. a per-replica rate below Size's lambdaMin leaves
 *       the bisection no bracket, utils.go:26-70).  The record stays solver input: the greedy does not read the field.
 * WVA_ESTATE when no valid sweep records exist (as wva_grid_pairs_fetch).  Sized records stay valid:
 * wva_grid_pairs_fetch and wva_solve_grid (every mode; a limited solve still consumes them) carry the sized rate; with
 * a communicator attached each rank sizes its shard rows and the limited solve's all-gather moves the sized rates.
 * Shards up to wva_pairs_set_warp_max pairs take one warp per pair, larger ones one thread per record; same results.
 * Timed under WVA_PHASE_GRID_SIZE.  Nothing changes unless this is called. */
int wva_grid_pairs_size(wva_ctx* ctx, uint8_t* status /* [S*A] host, may be NULL */);

/* What-if Analyze -> unlimited Optimize -> AllocateByType over n_scen load scenarios.  Scenario l replaces every
 * server's ServerLoadSpec.ArrivalRate by arrival_rpm[l*S + s]; nothing else of the image changes.
 *   Pair records: pair (s, a) of scenario l gets exactly what wva_analyze_pairs gives when the image's arrival rate of
 *       s is arrival_rpm[l*S + s]: Server.Calculate's candidate filter, CreateAllocation and the transition penalty
 *       (server.go:55-67, allocation.go:27-163, :291-300).  A negative rate gives nil (allocation.go:50), 0 gives
 *       zeroLoadAllocation (:73-75).  Every input of QueueAnalyzer.Size is independent of the rate, so each pair runs
 *       Size once and one trailing Analyze(totalRate / replicas) per scenario; a TPS-target server's positive
 *       scenarios all share one (allocation.go:135-139).
 *   chosen_acc[l*S + s], chosen[l*S + s] (host, may be NULL): SolveUnlimited of scenario l (solver.go:63-79), the
 *       argmin of value with strict '<' from MaxFloat32 in ascending accelerator index, as wva_solve unlimited.
 *   type_count[l*T + t], type_cost[l*T + t] (host, may be NULL): System.AllocateByType of scenario l
 *       (system.go:271-300), summed in the fixed float32 order of wva_allocate_by_type.
 * Limited-capacity (greedy) solves per scenario are not offered.
 * The call leaves the image, the pair records, the sweep records, the solution and the totals as they were: a later
 * wva_solve, wva_solve_grid or wva_allocate_by_type behaves as if it had not run.  Its records (L*S*A of 45 bytes,
 * full S*A extent per scenario) stay valid for wva_scenario_pairs_fetch until the next wva_analyze_scenarios, image
 * upload, image update or shard change; after those the fetch returns WVA_ESTATE.
 * Errors: WVA_ESTATE without an uploaded image; WVA_EINVAL for n_scen outside [1, WVA_MAX_SCENARIOS] or a NaN / Inf
 * rate; WVA_ECUDA when the record buffer cannot be allocated.
 * With a communicator attached each rank fills its shard rows (records and chosen); the per-scenario partial totals
 * {count[L*T]; cost[L*T]} move in ONE ncclAllGather and are summed in rank order (k_totals_merge over L*T entries), so
 * every rank returns the global totals.  Shards up to wva_pairs_set_warp_max pairs take one warp per pair, larger
 * ones one thread per pair and per (pair, scenario); same results.  The number of kernel launches does not grow with
 * n_scen.  Timed under WVA_PHASE_SCENARIOS. */
#define WVA_MAX_SCENARIOS 1024
int wva_analyze_scenarios(wva_ctx* ctx, int32_t n_scen, const float* arrival_rpm /* [n_scen*S] host */,
                          int32_t* chosen_acc /* [n_scen*S] or NULL */, wva_alloc_soa* chosen /* n_scen*S or NULL */,
                          int64_t* type_count /* [n_scen*T] or NULL */, float* type_cost /* [n_scen*T] or NULL */);
/* scenario scen's S*A records of the shard (rows of other shards untouched), like wva_pairs_fetch */
int wva_scenario_pairs_fetch(wva_ctx* ctx, int32_t scen, wva_alloc_soa* out /* S*A */, uint8_t* feasible /* S*A */);

/* Device addresses of the S*A candidate records of wva_analyze_pairs (dev->... are DEVICE pointers,
 * server-major, same extents as the host variant).  Multi-GPU limited-capacity mode: each rank
 * fills its shard rows, the host all-gathers the rows over NCCL in place, then calls
 * wva_pairs_commit so that wva_solve may run the (sequential, replicated) greedy assignment. */
int wva_pairs_device(wva_ctx* ctx, wva_alloc_soa* dev, uint8_t** feasible);
/* Ordering contract: wva_pairs_commit waits for ALL work previously issued to the device by this
 * process (cudaDeviceSynchronize), so the caller's collectives may run on any stream.  (With
 * wva_comm_init the library gathers the rows itself and none of this is needed.) */
int wva_pairs_commit(wva_ctx* ctx);
/* Tuning: certified closed-form tails (DESIGN.md section 4 (iii)) on/off and the sweep kernel.  Chains that
 * would run a long constant-rate tail are first evaluated from the ramp plus the geometric closed form and
 * accepted only when every float32 rounding of the result is unambiguous within a proven error bound;
 * otherwise the exact chain runs.  Results are identical in every mode.
 *   on = 1 (default): one WARP per (server, accelerator, replicas) row, lanes = 32 consecutive batch sizes:
 *           k_scan_prep finds every row's exact stop, k_scan_cert evaluates the batch sizes before it (ramp
 *           by warp scans + certificate), k_scan_lean the ones after it (frozen exact sums);  on = 33: same with
 *           k_scan_cert's register allocation for 2 instead of 3 blocks per SM;
 *   on = 0: no certificate, exact chains only (one thread per candidate);
 *   on = 17: round-1 automatic choice: one thread per row (shared sequential ramp) for shards with >= 32 K rows,
 *           one thread per candidate below;  on = 3 / 5 / 9: always one thread per candidate / one thread per
 *           row / one warp per row with a lockstep ramp (tuning, A-B). */
int wva_set_certified_tails(wva_ctx* ctx, int32_t on);
/* Tuning: shards with at most max_pairs (server, accelerator) pairs use the warp-per-pair kernel
 * (speculative bisection, lowest latency); larger shards use one thread per pair (highest
 * throughput).  Results do not depend on it.  Default 2^22 (measured: the warp kernel is ~30x faster than thread-per-pair even at 8 000 pairs
 * because its lanes stay converged); 0 = always thread-per-pair. */
int wva_pairs_set_warp_max(wva_ctx* ctx, int32_t max_pairs);
/* Tuning (warp-per-pair kernel): keep the chain values of pass 1 in HBM and read them back in pass 2
 * instead of re-running the recurrence.  Same results; off by default (measured slower on B200: the
 * loads expose L2 latency that the recomputation does not have). */
int wva_pairs_set_pstore(wva_ctx* ctx, int32_t on);
/* Chain-state updates executed by the last wva_analyze_pairs (instrumentation). */
int wva_pair_steps(wva_ctx* ctx, uint64_t* steps);
/* warp-per-pair kernel counters: {chain steps, sum of bisection rounds over pairs, max rounds of a pair,
 * trailing-Analyze evaluations that the cache / guess did not cover (+100 per missed guess)}. */
int wva_pair_counters(wva_ctx* ctx, uint64_t out[4]);
/* With wva_pairs_set_pstore(ctx, 4) set before wva_analyze_pairs: per pair of the shard two words
 * (profiling aid): [0] = SM cycles (bits 0-35) | exact re-evaluations of uncertain speculative nodes
 * (bits 36-43) | chain steps / 1024 (bits 44-63); [1] = (rounds << 32) | rounds-with-evaluations. */
int wva_pair_debug(wva_ctx* ctx, uint64_t* out, int32_t n_pairs);

/* ---- Optimize ------------------------------------------------------------ */

/* Replaces solver.Solver.Solve (pkg/solver/solver.go:32-60): SolveUnlimited (:63-79) or
 * SolveGreedy (pkg/solver/greedy.go:35-341) over the candidates of the last
 * wva_analyze_pairs.  chosen_acc[s] = key of the chosen candidate in allAllocations
 * (accelerator index) or -1 when the server received no allocation; chosen = a copy of
 * the chosen core.Allocation (after best-effort scaling, greedy.go:208-212, :302-311).
 * Canonical tie-break: ascending accelerator index, ascending server index. */
int wva_solve(wva_ctx* ctx, const wva_optimizer_spec* spec,
              int32_t* chosen_acc, wva_alloc_soa* chosen);

/* Tuning (limited-capacity solve): 2 (default) = static-order scan -- the (server, candidate) pairs are sorted
 * once by the running maximum of their keys and `allocate` is one linear pass of a warp over that order
 * (csrc/wva_greedy_scan.cuh); 1 = round 1's ranked queue (states sorted once, the sequential pass on a rank bitmap
 * in shared memory); 0 = always the heap kernel.  The library itself falls back (2 -> 1 -> 0) when a path's shared
 * memory does not fit (2: one bit per server; 1: one bit per state, ~1.7 M states) or there are more than 32
 * accelerators (2).  Same results on every path.  wva_solve_greedy_path reports what the last limited solve ran:
 * 1 heap, 2 ranked queue, 3 static-order scan, 0 none yet. */
int wva_solve_set_ranked(wva_ctx* ctx, int32_t on);
int wva_solve_greedy_path(const wva_ctx* ctx);
/* Instrumentation of the last limited solve.  Ranked queue: {queue pops, placements that did not fit,
 * SM cycles in the queue loop, SM cycles in bestEffort}; static-order scan: {events, batches | runs popped
 * from shared-group stacks << 32, SM cycles in the pass, SM cycles in bestEffort}. */
int wva_solve_stats(wva_ctx* ctx, uint64_t out[4]);

/* Replaces System.AllocateByType (pkg/core/system.go:271-300): per accelerator type
 * count += replicas*numInstances*multiplicity, cost += alloc.cost over this rank's shard.
 * The sums are left in a device buffer (wva_type_totals_device) so the host can run the
 * exchange step of the path on it; this call returns the LOCAL totals.  With count == cost == NULL
 * nothing is copied back and the call does not wait for the device (same for wva_solve in unlimited
 * mode with chosen_acc == chosen == NULL): later calls are ordered on the context's stream. */
int wva_allocate_by_type(wva_ctx* ctx, int64_t* count, float* cost);

/* Device address of the {int64 count[T]; then float cost[T]} totals written by the last
 * wva_allocate_by_type: count at ptr, cost at ptr + 8*T bytes.  The device sum uses a
 * fixed order (ascending server index) — Go sums in random map order (system.go:273,297). */
int wva_type_totals_device(wva_ctx* ctx, void** dev_ptr, size_t* bytes);

/* Sharded runs with a HOST-driven collective (no wva_comm_init): every rank all-gathers its 12*T-byte
 * totals block (ONE collective); this call then sums the n_ranks gathered blocks (device memory,
 * rank-major) in rank order into the totals buffer -- one launch, and unlike a ring/tree all-reduce the
 * float32 cost sums come out the same on every rank and every run.
 * Ordering contract: the merge kernel is enqueued on wva_stream(ctx); the caller's collective must
 * have been enqueued on that same stream (or have completed) before this call. */
int wva_type_totals_merge(wva_ctx* ctx, const void* gathered_dev, int32_t n_ranks);

/* optimizer.SolutionTimeMsec (pkg/solver/optimizer.go:30-34): device+host time of the
 * last wva_solve in microseconds. */
int64_t wva_solution_time_usec(const wva_ctx* ctx);

/* ---- multi-GPU inside the library ------------------------------------------ *
 * SURVEY 8(b)/(e): servers shard over the GPUs of one box, accelerator / perf / type tables are
 * replicated, Analyze needs no communication, and Optimize has ONE exchange step whose site in the
 * reference is System.AllocateByType (pkg/core/system.go:271-300).  NCCL is resolved at run time
 * (dlopen of libnccl.so.2), so the library still loads on a box without it; the calls below then
 * fail with WVA_ECUDA.
 *
 * (1) one process per GPU (torchrun, MPI, N Go processes): rank 0 obtains an id, the host
 *     distributes its 128 bytes by any means, every rank attaches its ctx.  With a communicator
 *     attached:
 *       - wva_comm_shard gives the rank its contiguous server range [floor(S*g/G), floor(S*(g+1)/G));
 *       - wva_allocate_by_type all-gathers the 12*T-byte {count, cost} partials (ONE ncclAllGather on
 *         the ctx stream) and sums them in rank order: every rank returns the GLOBAL totals, bit-equal
 *         on every rank and every run;
 *       - wva_solve in limited mode first all-gathers the candidate records of all ranks' shards
 *         (packed, ONE ncclAllGather of 45 B per (server, accelerator)), then runs the identical
 *         sequential greedy on every rank;
 *       - unlimited wva_solve stays local (separable), chosen_acc / chosen are filled for the shard. */
#define WVA_COMM_ID_BYTES 128
int wva_comm_unique_id(void* id_out /* WVA_COMM_ID_BYTES */);
int wva_comm_init(wva_ctx* ctx, const void* id, int32_t rank, int32_t n_ranks);
int wva_comm_destroy(wva_ctx* ctx);
int wva_comm_info(const wva_ctx* ctx, int32_t* rank, int32_t* n_ranks);   /* 0 / 1 without a communicator */
int wva_comm_shard(wva_ctx* ctx);

/* (2) ONE process driving several GPUs -- the shape of the reference's caller, a single reconcile
 *     goroutine (internal/controller/variantautoscaling_controller.go:143-166).  A group owns one ctx
 *     per device and an ncclCommInitAll communicator; every call fans out to one host thread per
 *     device and joins.  Host outputs have the full extent (S servers / S*A pairs) and are assembled
 *     from the shards; totals are global. */
typedef struct wva_group wva_group;
int  wva_group_create(const int32_t* device_ids, int32_t n_devices, wva_group** out);
void wva_group_destroy(wva_group* g);
int32_t wva_group_size(const wva_group* g);
wva_ctx* wva_group_ctx(wva_group* g, int32_t i);          /* per-device ctx (tuning, instrumentation) */
const char* wva_group_last_error(const wva_group* g);
int wva_group_upload(wva_group* g, const wva_system_soa* host);      /* replicate the image, shard the servers */
int wva_group_analyze(wva_group* g, int32_t r_max, int32_t b_max, int32_t want_cube);   /* r_max = 0: pairs only */
int wva_group_pairs_fetch(wva_group* g, wva_alloc_soa* out, uint8_t* feasible);
int wva_group_grid_fetch(wva_group* g, wva_grid_best* best /* [S] */);
int wva_group_solve(wva_group* g, const wva_optimizer_spec* spec, int32_t* chosen_acc, wva_alloc_soa* chosen);
/* the sweep-record forms (wva_grid_set_pair_winners on every device's ctx: wva_group_ctx) */
int wva_group_grid_pairs_fetch(wva_group* g, wva_alloc_soa* out, uint8_t* feasible);
int wva_group_solve_grid(wva_group* g, const wva_optimizer_spec* spec, int32_t* chosen_acc, wva_alloc_soa* chosen);
int wva_group_grid_pairs_size(wva_group* g, uint8_t* status /* [S*A] */);
/* load scenarios: every device fills its shard rows of chosen_acc / chosen / the records; totals are global */
int wva_group_analyze_scenarios(wva_group* g, int32_t n_scen, const float* arrival_rpm, int32_t* chosen_acc, wva_alloc_soa* chosen,
                                int64_t* type_count, float* type_cost);
int wva_group_scenario_pairs_fetch(wva_group* g, int32_t scen, wva_alloc_soa* out, uint8_t* feasible);
int wva_group_allocate_by_type(wva_group* g, int64_t* count, float* cost);

/* ---- low-level analyzer API (pkg/analyzer public surface) ------------------ */

typedef struct wva_queue_config {  /* analyzer.Configuration + RequestSize */
    int32_t max_batch_size;
    int32_t max_queue_size;
    float   alpha, beta, gamma, delta;
    int32_t avg_input_tokens;
    int32_t avg_output_tokens;
} wva_queue_config;

/* n independent QueueAnalyzer.Analyze calls (fresh analyzer each), one thread per
 * request: metrics[i], status[i] (WVA_CAND_OK or WVA_CAND_ERR_*). */
int wva_queue_analyze(wva_ctx* ctx, int32_t n, const wva_queue_config* cfg,
                      const float* rate, wva_metrics* metrics, uint8_t* status);

/* n independent QueueAnalyzer.Size calls (queueanalyzer.go:185-255).  target = TTFT, ITL,
 * TPS triples; rates = RateTargetTTFT/ITL/TPS triples; achieved = TTFT/ITL/TPS triples.
 * status[i]: 0 ok, 1 = error (target below bounded region / invalid). */
int wva_queue_size(wva_ctx* ctx, int32_t n, const wva_queue_config* cfg,
                   const float* target /*3n*/, float* rates /*3n*/, wva_metrics* metrics,
                   float* achieved /*3n*/, uint8_t* status);

/* The bare queueing model of pkg/analyzer: n_calls consecutive MM1ModelStateDependent.Solve(lambda[i], mu[i]) calls on ONE
 * model NewMM1ModelStateDependent(K, serv_rate[0..n_rates)) (mm1modelstatedependent.go:15-116, queuemodel.go:27-37).  The
 * model keeps its state between calls (the validity test reads the previous call's p[0]; invalid calls leave the
 * statistics of the last valid one).  out[9*i .. 9*i+8] = {isValid, rho, avgRespTime, avgWaitTime, avgServTime,
 * avgNumInSystem, avgQueueLength, avgNumInServers, throughput} after call i; p_out (may be NULL): the K+1 state
 * probabilities after the last call. */
int wva_model_solve(wva_ctx* ctx, int64_t K, const float* serv_rate, int32_t n_rates, int32_t n_calls,
                    const float* lambda, const float* mu, float* out, double* p_out);

/* ---- instrumentation ----------------------------------------------------- */

/* Kernel launches issued by this ctx since creation (for bench.py's gpu_launches). */
int64_t wva_launch_count(const wva_ctx* ctx);
/* Device time (CUDA events on the ctx stream) of the last call of each phase, usec. */
int64_t wva_phase_time_usec(const wva_ctx* ctx, int phase);
#define WVA_PHASE_UPLOAD 0
#define WVA_PHASE_PAIRS  1
#define WVA_PHASE_GRID   2
#define WVA_PHASE_SOLVE  3
#define WVA_PHASE_TOTALS 4
#define WVA_PHASE_GRID_KERNEL 5   /* the sweep kernel alone (events right around its launch) */
#define WVA_PHASE_GRID_HEAVY  6   /* ordering + processing of the deferred long chains */
#define WVA_PHASE_GRID_SIZE   7   /* wva_grid_pairs_size */
#define WVA_PHASE_SCENARIOS   8   /* wva_analyze_scenarios (downloads excluded) */
/* The cudaStream_t every call of this ctx is enqueued on (so a host can record its own events
 * on it or order other work after it). */
void* wva_stream(const wva_ctx* ctx);
/* Sweep tuning: candidates whose chain tail needs more than tail_cap steps are deferred from the
 * per-pair sweep kernel to a second kernel that groups chains of similar length (0 = never defer,
 * negative = automatic: 0 when certified tails are on, 192 otherwise).  Results do not depend on it.  wva_grid_list_sizes: how many candidates the last sweep deferred /
 * sent to the materialised-p[] path. */
int wva_grid_set_tail_cap(wva_ctx* ctx, int32_t tail_cap);
int wva_grid_list_sizes(const wva_ctx* ctx, int32_t* deferred, int32_t* literal);
/* Tuning (sweep): when the previous sweep deferred more than 4096 candidates to the exact-chain kernels, the next one
 * launches all its kernels without stopping at the host in between (the chain kernel reads the list length from device
 * memory and runs on SMs of its own beside the cube-writing half).  on = 1 (default) / 0 = always stop and go.  Same
 * results either way.  wva_grid_last_fused: 1 when the last sweep slice ran that way. */
int wva_grid_set_fused(wva_ctx* ctx, int32_t on);
int wva_grid_last_fused(const wva_ctx* ctx);
/* Candidate ids (cube indices relative to the shard) the last sweep slice handed to the exact-chain
 * kernel because their certificate was ambiguous or their tail outlasted tail_cap (at most cap are
 * copied; *n = how many there were).  Test/diagnostic aid: parity tests re-evaluate exactly these. */
int wva_grid_deferred_fetch(wva_ctx* ctx, uint64_t* ids, int32_t cap, int32_t* n);
/* Work counters of the last grid sweep: chain steps actually executed and the
 * algorithmic chain steps (sum over analysable candidates of 2*(11b+1)). */
int wva_grid_counters(const wva_ctx* ctx, uint64_t* steps_executed, uint64_t* steps_algorithmic,
                      uint64_t* candidates_ok);

/* Device self-test of the hoisted-reciprocal double division used by the chain kernels: n operand
 * pairs from a counter-based generator (mode 0: positive a of any exponent / float32-valued b;
 * 1: arbitrary doubles; 2: moderate exponents; 3: float32 operands inside the fast window of the hoisted float32
 * division; 4: arbitrary float32 bit patterns) are divided both ways; *mismatches counts results that differ
 * bitwise from the plain IEEE operator. */
int wva_selftest_division(wva_ctx* ctx, uint64_t seed, uint64_t n, int mode, uint64_t* mismatches);

#ifdef __cplusplus
}
#endif
#endif /* WVA_B200_H */
