// Package native is the cgo binding of the B200 library (include/wva_b200.h).
//
// WRITTEN WITHOUT A GO TOOLCHAIN: the build image of this repository has no `go`, so this file has
// never been compiled.  It is the binding a maintainer drops into the reference tree (module
// github.com/llm-d-incubation/workload-variant-autoscaler) next to the replacement packages in
// go/pkg; build with CGO_ENABLED=1 (the reference Dockerfile:25 sets 0) and
//   CGO_CFLAGS=-I<repo>/include  CGO_LDFLAGS="-L<repo>/inferno-autoscaler_b200 -lwva_b200"
//
// cgo pointer rules (cmd/cgo "Passing pointers"):
//   (1) the library retains no Go pointer after a call returns (wva_b200.h "Conventions": it copies);
//   (2) a Go pointer passed to C must not point at memory that itself holds Go pointers.  The struct forms
//       wva_system_upload / wva_analyze_pairs / wva_solve take a struct OF pointers: a Go-allocated
//       C.wva_system_soa whose fields point at Go slices violates (2) and panics under the default
//       GODEBUG=cgocheck=1 ("cgo argument has Go pointer to unpinned Go pointer").  This binding therefore
//       calls the *_arrays forms of the header, where every slice is its own argument (a pointer to
//       pointer-free memory needs no pinning).  The only struct-of-pointers call is Group.Upload, which builds
//       the struct in C memory and pins every slice with runtime.Pinner for the duration of the call.
package native

/*
#cgo LDFLAGS: -lwva_b200
#include <stdlib.h>
#include "wva_b200.h"
*/
import "C"

import (
	"fmt"
	"runtime"
	"sync"
	"unsafe"
)

// SystemImage is the structure-of-arrays form of config.SystemSpec (wva_system_soa).
type SystemImage struct {
	S, A, M, T int

	AccCost         []float32
	AccMultiplicity []int32
	AccType         []int32
	TypeCapacity    []int64

	PerfAlpha, PerfBeta, PerfGamma, PerfDelta []float32
	PerfMaxBatch, PerfAtTokens, PerfAccCount  []int32
	PerfValid                                 []uint8

	SrvModel                         []int32
	SrvArrivalRPM                    []float32
	SrvInTokens, SrvOutTokens        []int32
	SrvSloTTFT, SrvSloITL, SrvSloTPS []float32
	SrvTargetValid                   []uint8
	SrvPriority, SrvMinReplicas      []int32
	SrvMaxBatch                      []int32
	SrvKeepAcc                       []uint8
	SrvCurAcc, SrvCurReplicas        []int32
	SrvCurCost                       []float32
}

// Allocs mirrors wva_alloc_soa (one record per index).
type Allocs struct {
	Acc                                   []int32
	NumReplicas, BatchSize                []int64
	Cost, Value, ITL, TTFT, Rho, MaxArrv []float32
}

func newAllocs(n int) *Allocs {
	return &Allocs{Acc: make([]int32, n), NumReplicas: make([]int64, n), BatchSize: make([]int64, n),
		Cost: make([]float32, n), Value: make([]float32, n), ITL: make([]float32, n), TTFT: make([]float32, n),
		Rho: make([]float32, n), MaxArrv: make([]float32, n)}
}

// Context wraps wva_ctx: one per process (creation builds the CUDA context), one call at a time —
// the same constraint the reference has through its package globals (pkg/core/system.go:12).
type Context struct {
	mu  sync.Mutex
	ctx *C.wva_ctx
}

var (
	defaultOnce sync.Once
	defaultCtx  *Context
	defaultErr  error
)

// Default returns the process-wide context on CUDA device 0 (WVA_B200_DEVICE overrides in the shim).
func Default() (*Context, error) {
	defaultOnce.Do(func() { defaultCtx, defaultErr = NewContext(0) })
	return defaultCtx, defaultErr
}

func NewContext(device int) (*Context, error) {
	var c *C.wva_ctx
	if rc := C.wva_ctx_create(C.int(device), &c); rc != C.WVA_OK {
		return nil, fmt.Errorf("wva_ctx_create: %d: %s", int(rc), C.GoString(C.wva_last_error(nil)))
	}
	ctx := &Context{ctx: c}
	runtime.SetFinalizer(ctx, func(x *Context) { C.wva_ctx_destroy(x.ctx) })
	return ctx, nil
}

func (c *Context) err(rc C.int, what string) error {
	if rc == C.WVA_OK {
		return nil
	}
	return fmt.Errorf("%s: %d: %s", what, int(rc), C.GoString(C.wva_last_error(c.ctx)))
}

func f32p(s []float32) *C.float { if len(s) == 0 { return nil }; return (*C.float)(unsafe.Pointer(&s[0])) }
func i32p(s []int32) *C.int32_t { if len(s) == 0 { return nil }; return (*C.int32_t)(unsafe.Pointer(&s[0])) }
func i64p(s []int64) *C.int64_t { if len(s) == 0 { return nil }; return (*C.int64_t)(unsafe.Pointer(&s[0])) }
func u8p(s []uint8) *C.uint8_t  { if len(s) == 0 { return nil }; return (*C.uint8_t)(unsafe.Pointer(&s[0])) }

// Upload replaces core.NewSystem + System.SetFromSpec on the native side (wva_system_upload).
func (c *Context) Upload(img *SystemImage) error {
	c.mu.Lock()
	defer c.mu.Unlock()
	rc := C.wva_system_upload_arrays(c.ctx, C.int32_t(img.S), C.int32_t(img.A), C.int32_t(img.M), C.int32_t(img.T),
		f32p(img.AccCost), i32p(img.AccMultiplicity), i32p(img.AccType), i64p(img.TypeCapacity),
		f32p(img.PerfAlpha), f32p(img.PerfBeta), f32p(img.PerfGamma), f32p(img.PerfDelta),
		i32p(img.PerfMaxBatch), i32p(img.PerfAtTokens), i32p(img.PerfAccCount), u8p(img.PerfValid),
		i32p(img.SrvModel), f32p(img.SrvArrivalRPM), i32p(img.SrvInTokens), i32p(img.SrvOutTokens),
		f32p(img.SrvSloTTFT), f32p(img.SrvSloITL), f32p(img.SrvSloTPS), u8p(img.SrvTargetValid),
		i32p(img.SrvPriority), i32p(img.SrvMinReplicas), i32p(img.SrvMaxBatch), u8p(img.SrvKeepAcc),
		i32p(img.SrvCurAcc), i32p(img.SrvCurReplicas), f32p(img.SrvCurCost))
	return c.err(rc, "wva_system_upload_arrays")
}

// AnalyzePairs replaces Server.Calculate for all servers: S*A records + feasible flags.
func (c *Context) AnalyzePairs(s, a int) (*Allocs, []uint8, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	n := s * a
	if n == 0 {
		return newAllocs(0), nil, nil
	}
	out, fe := newAllocs(n), make([]uint8, n)
	rc := C.wva_analyze_pairs_arrays(c.ctx, i32p(out.Acc), i64p(out.NumReplicas), i64p(out.BatchSize), f32p(out.Cost), f32p(out.Value),
		f32p(out.ITL), f32p(out.TTFT), f32p(out.Rho), f32p(out.MaxArrv), u8p(fe))
	if err := c.err(rc, "wva_analyze_pairs_arrays"); err != nil {
		return nil, nil, err
	}
	return out, fe, nil
}

// Solve replaces solver.Solver.Solve: chosen candidate key per server (-1 = none) and a copy of it.
func (c *Context) Solve(s int, unlimited, delayedBestEffort bool, policy int) ([]int32, *Allocs, int64, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	b := func(v bool) C.int32_t { if v { return 1 }; return 0 }
	if s == 0 {
		return nil, newAllocs(0), 0, nil
	}
	key, out := make([]int32, s), newAllocs(s)
	rc := C.wva_solve_arrays(c.ctx, b(unlimited), b(delayedBestEffort), C.int32_t(policy), i32p(key),
		i32p(out.Acc), i64p(out.NumReplicas), i64p(out.BatchSize), f32p(out.Cost), f32p(out.Value),
		f32p(out.ITL), f32p(out.TTFT), f32p(out.Rho), f32p(out.MaxArrv))
	if err := c.err(rc, "wva_solve_arrays"); err != nil {
		return nil, nil, 0, err
	}
	return key, out, int64(C.wva_solution_time_usec(c.ctx)), nil
}

// AllocateByType replaces System.AllocateByType (per accelerator type totals of this process' shard).
func (c *Context) AllocateByType(t int) ([]int64, []float32, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	count, cost := make([]int64, t), make([]float32, t)
	if t == 0 {
		return count, cost, nil
	}
	return count, cost, c.err(C.wva_allocate_by_type(c.ctx, i64p(count), f32p(cost)), "wva_allocate_by_type")
}

// Analyze runs Server.Calculate for every pair of the shard and the candidate sweep side by side
// (wva_analyze); results stay on the device for Solve / PairsFetch / GridFetch.
func (c *Context) Analyze(rMax, bMax int) error {
	c.mu.Lock()
	defer c.mu.Unlock()
	return c.err(C.wva_analyze(c.ctx, C.int32_t(rMax), C.int32_t(bMax), 0), "wva_analyze")
}

// Tuning knobs (results never depend on them; see include/wva_b200.h).  SolvePath: 2 = static-order scan (default),
// 1 = ranked queue, 0 = heap.  SweepFused: false = the sweep always stops at the host between its kernels.
func (c *Context) SetSolvePath(path int) error {
	c.mu.Lock()
	defer c.mu.Unlock()
	return c.err(C.wva_solve_set_ranked(c.ctx, C.int32_t(path)), "wva_solve_set_ranked")
}

func (c *Context) SetSweepFused(on bool) error {
	c.mu.Lock()
	defer c.mu.Unlock()
	v := C.int32_t(0)
	if on {
		v = 1
	}
	return c.err(C.wva_grid_set_fused(c.ctx, v), "wva_grid_set_fused")
}

// SetSweepPairWinners: every later sweep (Analyze, AnalyzeGrid) also keeps its best candidate of each
// (server, accelerator) pair on the device, for GridPairsFetch / SolveGrid.
func (c *Context) SetSweepPairWinners(on bool) error {
	c.mu.Lock()
	defer c.mu.Unlock()
	v := C.int32_t(0)
	if on {
		v = 1
	}
	return c.err(C.wva_grid_set_pair_winners(c.ctx, v), "wva_grid_set_pair_winners")
}

// GridPairsFetch copies the sweep's per-pair winners of the shard out: S*A records + feasible flags.
func (c *Context) GridPairsFetch(s, a int) (*Allocs, []uint8, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	n := s * a
	if n == 0 {
		return newAllocs(0), nil, nil
	}
	out, fe := newAllocs(n), make([]uint8, n)
	rc := C.wva_grid_pairs_fetch_arrays(c.ctx, i32p(out.Acc), i64p(out.NumReplicas), i64p(out.BatchSize), f32p(out.Cost), f32p(out.Value),
		f32p(out.ITL), f32p(out.TTFT), f32p(out.Rho), f32p(out.MaxArrv), u8p(fe))
	if err := c.err(rc, "wva_grid_pairs_fetch_arrays"); err != nil {
		return nil, nil, err
	}
	return out, fe, nil
}

// GridPairsSize runs QueueAnalyzer.Size on the device for every sweep record of the shard at the record's own
// batch size; a sized record's MaxArrv becomes the SLO-bound rate per replica.  Status per pair of the S*A
// extent: 0 no record, 1 sized, 2 Size failed (record unchanged); rows of other shards stay 0.
func (c *Context) GridPairsSize(s, a int) ([]uint8, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	n := s * a
	if n == 0 {
		return nil, nil
	}
	st := make([]uint8, n)
	if err := c.err(C.wva_grid_pairs_size(c.ctx, u8p(st)), "wva_grid_pairs_size"); err != nil {
		return nil, err
	}
	return st, nil
}

// AnalyzeScenarios evaluates what Analyze -> unlimited Solve -> AllocateByType would give for every row of
// arrivalRPM (nScen rows of s rates, row-major; each row replaces every server's arrival rate), one Size per pair.
// Returns chosen[l*s+i] (-1 = none), the chosen records, and count / cost [l*t+j]; the resident image and results
// are left untouched.
func (c *Context) AnalyzeScenarios(s, t int, arrivalRPM []float32) ([]int32, *Allocs, []int64, []float32, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	if s == 0 || len(arrivalRPM)%s != 0 {
		return nil, nil, nil, nil, fmt.Errorf("AnalyzeScenarios: %d rates is not a whole number of %d-server rows", len(arrivalRPM), s)
	}
	l := len(arrivalRPM) / s
	key, out := make([]int32, l*s), newAllocs(l*s)
	count, cost := make([]int64, l*t), make([]float32, l*t)
	rc := C.wva_analyze_scenarios_arrays(c.ctx, C.int32_t(l), f32p(arrivalRPM), i32p(key),
		i32p(out.Acc), i64p(out.NumReplicas), i64p(out.BatchSize), f32p(out.Cost), f32p(out.Value),
		f32p(out.ITL), f32p(out.TTFT), f32p(out.Rho), f32p(out.MaxArrv), i64p(count), f32p(cost))
	if err := c.err(rc, "wva_analyze_scenarios_arrays"); err != nil {
		return nil, nil, nil, nil, err
	}
	return key, out, count, cost, nil
}

// ScenarioPairsFetch copies scenario scen's S*A pair records of the last AnalyzeScenarios.
func (c *Context) ScenarioPairsFetch(scen, s, a int) (*Allocs, []uint8, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	n := s * a
	if n == 0 {
		return newAllocs(0), nil, nil
	}
	out, fe := newAllocs(n), make([]uint8, n)
	rc := C.wva_scenario_pairs_fetch_arrays(c.ctx, C.int32_t(scen), i32p(out.Acc), i64p(out.NumReplicas), i64p(out.BatchSize),
		f32p(out.Cost), f32p(out.Value), f32p(out.ITL), f32p(out.TTFT), f32p(out.Rho), f32p(out.MaxArrv), u8p(fe))
	if err := c.err(rc, "wva_scenario_pairs_fetch_arrays"); err != nil {
		return nil, nil, err
	}
	return out, fe, nil
}

// SolveGrid is Solve over the sweep's per-pair winners instead of the pair records.
func (c *Context) SolveGrid(s int, unlimited, delayedBestEffort bool, policy int) ([]int32, *Allocs, int64, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	b := func(v bool) C.int32_t { if v { return 1 }; return 0 }
	if s == 0 {
		return nil, newAllocs(0), 0, nil
	}
	key, out := make([]int32, s), newAllocs(s)
	rc := C.wva_solve_grid_arrays(c.ctx, b(unlimited), b(delayedBestEffort), C.int32_t(policy), i32p(key),
		i32p(out.Acc), i64p(out.NumReplicas), i64p(out.BatchSize), f32p(out.Cost), f32p(out.Value),
		f32p(out.ITL), f32p(out.TTFT), f32p(out.Rho), f32p(out.MaxArrv))
	if err := c.err(rc, "wva_solve_grid_arrays"); err != nil {
		return nil, nil, 0, err
	}
	return key, out, int64(C.wva_solution_time_usec(c.ctx)), nil
}

// SetShard restricts the following calls to servers [first, first+count) (one process per GPU).
func (c *Context) SetShard(first, count int) error {
	c.mu.Lock()
	defer c.mu.Unlock()
	return c.err(C.wva_set_shard(c.ctx, C.int32_t(first), C.int32_t(count)), "wva_set_shard")
}

// CommUniqueID / CommInit / CommShard: one process per GPU.  Rank 0 makes the 128-byte id, the caller
// distributes it (any transport), every rank attaches; from then on AllocateByType returns GLOBAL totals
// (the library runs the NCCL all-gather and the rank-order sum) and a limited Solve gathers the candidate
// rows itself.
func CommUniqueID() ([]byte, error) {
	id := make([]byte, C.WVA_COMM_ID_BYTES)
	if rc := C.wva_comm_unique_id(unsafe.Pointer(&id[0])); rc != C.WVA_OK {
		return nil, fmt.Errorf("wva_comm_unique_id: %d: %s", int(rc), C.GoString(C.wva_last_error(nil)))
	}
	return id, nil
}

func (c *Context) CommInit(id []byte, rank, nRanks int) error {
	c.mu.Lock()
	defer c.mu.Unlock()
	if len(id) != C.WVA_COMM_ID_BYTES {
		return fmt.Errorf("communicator id must have %d bytes", int(C.WVA_COMM_ID_BYTES))
	}
	return c.err(C.wva_comm_init(c.ctx, unsafe.Pointer(&id[0]), C.int32_t(rank), C.int32_t(nRanks)), "wva_comm_init")
}

func (c *Context) CommShard() error {
	c.mu.Lock()
	defer c.mu.Unlock()
	return c.err(C.wva_comm_shard(c.ctx), "wva_comm_shard")
}

// TypeTotalsMerge sums the per-rank totals blocks that the host all-gathered (device memory,
// rank-major, 12*T bytes each) in rank order into this context's totals buffer: the exchange step of
// a sharded reconcile.  The collective itself belongs to the caller (NCCL / MPI binding of its choice).
func (c *Context) TypeTotalsMerge(gatheredDev unsafe.Pointer, nRanks int) error {
	c.mu.Lock()
	defer c.mu.Unlock()
	return c.err(C.wva_type_totals_merge(c.ctx, gatheredDev, C.int32_t(nRanks)), "wva_type_totals_merge")
}

// GridBest is wva_grid_best.
type GridBest struct {
	Acc, Replicas, Batch       int32
	Cost, Value, ITL, TTFT, Rho float32
}

// AnalyzeGrid runs the (server x accelerator x replicas x batch) candidate sweep; one winner per server.
func (c *Context) AnalyzeGrid(s, rMax, bMax int) ([]GridBest, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	best := make([]GridBest, s)
	if s == 0 {
		return best, nil
	}
	rc := C.wva_analyze_grid(c.ctx, C.int32_t(rMax), C.int32_t(bMax), (*C.wva_grid_best)(unsafe.Pointer(&best[0])), nil, nil)
	return best, c.err(rc, "wva_analyze_grid")
}

// QueueConfig is wva_queue_config; Metrics is wva_metrics (analyzer.AnalysisMetrics).
type QueueConfig struct {
	MaxBatchSize, MaxQueueSize int32
	Alpha, Beta, Gamma, Delta  float32
	AvgInputTokens, AvgOutputTokens int32
}
type Metrics struct {
	Throughput, AvgRespTime, AvgWaitTime, AvgNumInServ, AvgPrefillTime, AvgTokenTime, MaxRate, Rho float32
}

// QueueAnalyze: n independent QueueAnalyzer.Analyze calls.
func (c *Context) QueueAnalyze(cfg []QueueConfig, rate []float32) ([]Metrics, []uint8, error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	n := len(cfg)
	m, st := make([]Metrics, n), make([]uint8, n)
	if n == 0 {
		return m, st, nil
	}
	rc := C.wva_queue_analyze(c.ctx, C.int32_t(n), (*C.wva_queue_config)(unsafe.Pointer(&cfg[0])), f32p(rate),
		(*C.wva_metrics)(unsafe.Pointer(&m[0])), u8p(st))
	return m, st, c.err(rc, "wva_queue_analyze")
}

// ModelSolve: a sequence of MM1ModelStateDependent.Solve(lambda[i], mu[i]) calls on one model
// NewMM1ModelStateDependent(K, servRate); out has 9 floats per call {isValid, rho, avgRespTime, avgWaitTime,
// avgServTime, avgNumInSystem, avgQueueLength, avgNumInServers, throughput}; p = probabilities after the last call.
func (c *Context) ModelSolve(K int, servRate, lambda, mu []float32) (out []float32, p []float64, err error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	n := len(lambda)
	out, p = make([]float32, 9*n), make([]float64, K+1)
	if n == 0 || len(servRate) == 0 || len(mu) != n {
		return out, p, fmt.Errorf("bad ModelSolve arguments")
	}
	rc := C.wva_model_solve(c.ctx, C.int64_t(K), f32p(servRate), C.int32_t(len(servRate)), C.int32_t(n), f32p(lambda), f32p(mu),
		f32p(out), (*C.double)(unsafe.Pointer(&p[0])))
	return out, p, c.err(rc, "wva_model_solve")
}

// QueueSize: n independent QueueAnalyzer.Size calls; target/rates/achieved are (TTFT, ITL, TPS) triples.
func (c *Context) QueueSize(cfg []QueueConfig, target []float32) (rates []float32, m []Metrics, achieved []float32, status []uint8, err error) {
	c.mu.Lock()
	defer c.mu.Unlock()
	n := len(cfg)
	rates, achieved, m, status = make([]float32, 3*n), make([]float32, 3*n), make([]Metrics, n), make([]uint8, n)
	if n == 0 {
		return
	}
	rc := C.wva_queue_size(c.ctx, C.int32_t(n), (*C.wva_queue_config)(unsafe.Pointer(&cfg[0])), f32p(target), f32p(rates),
		(*C.wva_metrics)(unsafe.Pointer(&m[0])), f32p(achieved), u8p(status))
	err = c.err(rc, "wva_queue_size")
	return
}

// Group wraps wva_group: ONE process (the single reconcile goroutine of
// internal/controller/variantautoscaling_controller.go:143-166) driving every GPU of the box.  Servers are
// sharded over the devices by the library; outputs have the full extent; totals are global.
type Group struct {
	mu sync.Mutex
	g  *C.wva_group
	n  int
}

func NewGroup(devices []int32) (*Group, error) {
	if len(devices) == 0 {
		return nil, fmt.Errorf("no devices")
	}
	var g *C.wva_group
	if rc := C.wva_group_create(i32p(devices), C.int32_t(len(devices)), &g); rc != C.WVA_OK {
		return nil, fmt.Errorf("wva_group_create: %d: %s", int(rc), C.GoString(C.wva_last_error(nil)))
	}
	grp := &Group{g: g, n: len(devices)}
	runtime.SetFinalizer(grp, func(x *Group) { C.wva_group_destroy(x.g) })
	return grp, nil
}

func (g *Group) err(rc C.int, what string) error {
	if rc == C.WVA_OK {
		return nil
	}
	return fmt.Errorf("%s: %d: %s", what, int(rc), C.GoString(C.wva_group_last_error(g.g)))
}

// Upload replicates the image on every device and shards the servers.  wva_group_upload takes the struct
// form, so the slices are pinned for the duration of the call (runtime.Pinner, Go >= 1.21; the reference
// is on go1.23, go.mod:7) -- the one place this binding builds a C struct of Go pointers.
func (g *Group) Upload(img *SystemImage) error {
	g.mu.Lock()
	defer g.mu.Unlock()
	var pin runtime.Pinner
	defer pin.Unpin()
	pf := func(s []float32) *C.float { if len(s) == 0 { return nil }; pin.Pin(&s[0]); return (*C.float)(unsafe.Pointer(&s[0])) }
	pi := func(s []int32) *C.int32_t { if len(s) == 0 { return nil }; pin.Pin(&s[0]); return (*C.int32_t)(unsafe.Pointer(&s[0])) }
	pl := func(s []int64) *C.int64_t { if len(s) == 0 { return nil }; pin.Pin(&s[0]); return (*C.int64_t)(unsafe.Pointer(&s[0])) }
	pu := func(s []uint8) *C.uint8_t { if len(s) == 0 { return nil }; pin.Pin(&s[0]); return (*C.uint8_t)(unsafe.Pointer(&s[0])) }
	h := (*C.wva_system_soa)(C.calloc(1, C.size_t(unsafe.Sizeof(C.wva_system_soa{}))))   // C memory: may hold pinned Go pointers
	defer C.free(unsafe.Pointer(h))
	h.n_servers, h.n_accels, h.n_models, h.n_types = C.int32_t(img.S), C.int32_t(img.A), C.int32_t(img.M), C.int32_t(img.T)
	h.acc_cost, h.acc_multiplicity, h.acc_type, h.type_capacity = pf(img.AccCost), pi(img.AccMultiplicity), pi(img.AccType), pl(img.TypeCapacity)
	h.perf_alpha, h.perf_beta, h.perf_gamma, h.perf_delta = pf(img.PerfAlpha), pf(img.PerfBeta), pf(img.PerfGamma), pf(img.PerfDelta)
	h.perf_max_batch, h.perf_at_tokens, h.perf_acc_count, h.perf_valid = pi(img.PerfMaxBatch), pi(img.PerfAtTokens), pi(img.PerfAccCount), pu(img.PerfValid)
	h.srv_model, h.srv_arrival_rpm, h.srv_in_tokens, h.srv_out_tokens = pi(img.SrvModel), pf(img.SrvArrivalRPM), pi(img.SrvInTokens), pi(img.SrvOutTokens)
	h.srv_slo_ttft, h.srv_slo_itl, h.srv_slo_tps, h.srv_target_valid = pf(img.SrvSloTTFT), pf(img.SrvSloITL), pf(img.SrvSloTPS), pu(img.SrvTargetValid)
	h.srv_priority, h.srv_min_replicas, h.srv_max_batch, h.srv_keep_acc = pi(img.SrvPriority), pi(img.SrvMinReplicas), pi(img.SrvMaxBatch), pu(img.SrvKeepAcc)
	h.srv_cur_acc, h.srv_cur_replicas, h.srv_cur_cost = pi(img.SrvCurAcc), pi(img.SrvCurReplicas), pf(img.SrvCurCost)
	return g.err(C.wva_group_upload(g.g, h), "wva_group_upload")
}

// Analyze: Server.Calculate for every pair (and the candidate sweep when rMax > 0) on all devices.
func (g *Group) Analyze(rMax, bMax int) error {
	g.mu.Lock()
	defer g.mu.Unlock()
	return g.err(C.wva_group_analyze(g.g, C.int32_t(rMax), C.int32_t(bMax), 0), "wva_group_analyze")
}

// GridPairsSize: Context.GridPairsSize on every device (each sizes its shard), status of the full S*A extent.
func (g *Group) GridPairsSize(s, a int) ([]uint8, error) {
	g.mu.Lock()
	defer g.mu.Unlock()
	n := s * a
	if n == 0 {
		return nil, nil
	}
	st := make([]uint8, n)
	if err := g.err(C.wva_group_grid_pairs_size(g.g, u8p(st)), "wva_group_grid_pairs_size"); err != nil {
		return nil, err
	}
	return st, nil
}

// AllocateByType: global per-type totals (NCCL all-gather of the partials inside the library).
func (g *Group) AllocateByType(t int) ([]int64, []float32, error) {
	g.mu.Lock()
	defer g.mu.Unlock()
	count, cost := make([]int64, t), make([]float32, t)
	if t == 0 {
		return count, cost, nil
	}
	return count, cost, g.err(C.wva_group_allocate_by_type(g.g, i64p(count), f32p(cost)), "wva_group_allocate_by_type")
}
