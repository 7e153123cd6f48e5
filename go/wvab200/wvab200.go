// Package wvab200 binds libwva_b200.so (include/wva_b200.h) into WVA's controller.
//
// NOT COMPILED IN THIS REPO'S CI: the build image has no Go toolchain.  It is the binding a
// WVA maintainer would add (see INTEGRATION.md); the same C ABI is exercised by the Python
// ctypes harness in tests/.
//
// It replaces, behind the existing adapter types,
//   - modelanalyzer.ModelAnalyzer.AnalyzeModel   (internal/modelanalyzer/analyzer.go:25-34)  -> ModelAnalyzer
//   - optimizer.VariantAutoscalingsEngine.Optimize (internal/optimizer/optimizer.go:30-54)   -> VariantAutoscalingsEngine
// i.e. Server.Calculate + Manager.Optimize + System.GenerateSolution of pkg/core, pkg/manager; plus
//   - Engine.Upload / UpdateLoad / Resolve: the streaming reconcile (fleet resident on the GPU, only the load
//     columns travel per tick: wva_upload / wva_update_load / wva_resolve)
//   - Engine.ResolveScenarios: Resolve under many arrival-rate scenarios in one call (wva_resolve_scenarios)
//   - Engine.Summarize: System.AllocateByType + Solver.Solve's allocation diffs (wva_summarize).
//   - Engine.MM1K: analyzer.MM1KModel (closed form) for arrays of (K, lambda, mu) (wva_mm1k_solve).
// tests/c_abi/solve_smoke.c drives the same entry points from compiled C.
package wvab200

/*
#cgo CFLAGS: -I${SRCDIR}/../../include
#cgo LDFLAGS: -L${SRCDIR}/../../workload_variant_autoscaler_b200 -lwva_b200 -lcudart
#include <stdlib.h>
#include "wva_b200.h"
*/
import "C"

import (
	"context"
	"fmt"
	"runtime"
	"sync"
	"unsafe"

	llmdOptv1alpha1 "github.com/llm-d-incubation/workload-variant-autoscaler/api/v1alpha1"
	interfaces "github.com/llm-d-incubation/workload-variant-autoscaler/internal/interfaces"
	"github.com/llm-d-incubation/workload-variant-autoscaler/internal/utils"
	"github.com/llm-d-incubation/workload-variant-autoscaler/pkg/config"
)

const (
	accNone    = -1 // accelerator name ""
	accUnknown = -2 // a name that is not in the accelerator table
	accAbsent  = -3 // no allocation at all ("none" in core.CreateAllocationDiff)
)

// Engine owns one wva_handle (one GPU). One solve at a time, like the reference L1.
type Engine struct {
	mu   sync.Mutex
	h    *C.wva_handle
	last *fleet // the fleet of the most recent Solve / Upload (names for Summarize)
}

func NewEngine(device int) (*Engine, error) {
	var h *C.wva_handle
	if rc := C.wva_create(&h, C.int(device)); rc != C.WVA_OK {
		return nil, fmt.Errorf("wva_create: %s", C.GoString(C.wva_strerror(rc)))
	}
	e := &Engine{h: h}
	runtime.SetFinalizer(e, func(e *Engine) { e.Close() })
	return e, nil
}

func (e *Engine) Close() {
	e.mu.Lock()
	defer e.mu.Unlock()
	if e.h != nil {
		C.wva_destroy(e.h)
		e.h = nil
	}
}

// fleet is the flat SoA image of config.SystemSpec (System.SetFromSpec's joins, done with maps here).
type fleet struct {
	accNames, serverNames, typeNames                           []string
	accCost                                                    []float32
	accMult, accType, typeCap                                  []int32
	perfPresent                                                []uint8
	alpha, beta, gamma, delta                                  []float32
	accCount, maxBatch, atTokens                               []int32
	srvModel, srvPrio, srvMinRep, srvMaxBatch, inTok, outTok   []int32
	srvHasTarget, srvKeep                                      []uint8
	sloITL, sloTTFT, sloTPS, arrival, curCost                  []float32
	curAcc, curRep                                             []int32
	unlimited, delayedBestEffort                               bool
	saturationPolicy                                           int
	loads                                                      []config.ServerLoadSpec // per packed server
}

func pack(spec *config.SystemSpec) *fleet {
	f := &fleet{}
	accIdx, typeIdx, modelIdx := map[string]int{}, map[string]int{}, map[string]int{}
	// AddAcceleratorFromSpec replaces an accelerator whose name repeats (pkg/core/system.go:99-101): the LAST
	// spec wins, at the position of the first (same rule as Fleet.from_spec in the Python packer)
	lastAcc := map[string]config.AcceleratorSpec{}
	for _, a := range spec.Accelerators.Spec {
		if _, dup := accIdx[a.Name]; !dup {
			accIdx[a.Name] = len(f.accNames)
			f.accNames = append(f.accNames, a.Name)
		}
		lastAcc[a.Name] = a
	}
	for _, name := range f.accNames {
		a := lastAcc[name]
		if _, ok := typeIdx[a.Type]; !ok {
			typeIdx[a.Type] = len(typeIdx)
		}
		f.accCost = append(f.accCost, a.Cost)
		f.accMult = append(f.accMult, int32(a.Multiplicity))
		f.accType = append(f.accType, int32(typeIdx[a.Type]))
	}
	for _, c := range spec.Capacity.Count { // a capacity entry may name a type no accelerator has
		if _, ok := typeIdx[c.Type]; !ok {
			typeIdx[c.Type] = len(typeIdx)
		}
	}
	f.typeNames = make([]string, len(typeIdx))
	for name, t := range typeIdx {
		f.typeNames[t] = name
	}
	f.typeCap = make([]int32, len(typeIdx))
	for _, c := range spec.Capacity.Count {
		if t, ok := typeIdx[c.Type]; ok {
			f.typeCap[t] = int32(c.Count)
		}
	}
	for _, pd := range spec.Models.PerfData {
		if _, ok := modelIdx[pd.Name]; !ok {
			modelIdx[pd.Name] = len(modelIdx)
		}
	}
	A, M := len(f.accNames), len(modelIdx)
	n := M * A
	f.perfPresent = make([]uint8, n)
	f.alpha, f.beta, f.gamma, f.delta = make([]float32, n), make([]float32, n), make([]float32, n), make([]float32, n)
	f.accCount, f.maxBatch, f.atTokens = make([]int32, n), make([]int32, n), make([]int32, n)
	for _, pd := range spec.Models.PerfData {
		a, ok := accIdx[pd.Acc]
		if !ok {
			continue
		}
		k := modelIdx[pd.Name]*A + a
		f.perfPresent[k] = 1
		f.alpha[k], f.beta[k] = pd.DecodeParms.Alpha, pd.DecodeParms.Beta
		f.gamma[k], f.delta[k] = pd.PrefillParms.Gamma, pd.PrefillParms.Delta
		f.accCount[k], f.maxBatch[k], f.atTokens[k] = int32(pd.AccCount), int32(pd.MaxBatchSize), int32(pd.AtTokens)
	}
	type class struct {
		prio    int
		targets map[string]config.ModelTarget
	}
	classes := map[string]class{}
	for _, sc := range spec.ServiceClasses.Spec {
		p := sc.Priority
		if p < config.DefaultHighPriority || p > config.DefaultLowPriority {
			p = config.DefaultServiceClassPriority
		}
		c := class{prio: p, targets: map[string]config.ModelTarget{}}
		for _, mt := range sc.ModelTargets {
			c.targets[mt.Model] = mt
		}
		classes[sc.Name] = c
	}
	// s.servers[v.Name] = ... (pkg/core/system.go:151-153): a repeated server name replaces the earlier spec
	lastSrv := map[string]config.ServerSpec{}
	for _, sv := range spec.Servers.Spec {
		if _, dup := lastSrv[sv.Name]; !dup {
			f.serverNames = append(f.serverNames, sv.Name)
		}
		lastSrv[sv.Name] = sv
	}
	for _, name := range f.serverNames {
		sv := lastSrv[name]
		f.loads = append(f.loads, sv.CurrentAlloc.Load)
		m, ok := modelIdx[sv.Model]
		if !ok {
			m = -1
		}
		f.srvModel = append(f.srvModel, int32(m))
		cls := sv.Class
		if cls == "" {
			cls = config.DefaultServiceClassName
		}
		prio, has := config.DefaultServiceClassPriority, uint8(0)
		var t config.ModelTarget
		if c, ok := classes[cls]; ok {
			prio = c.prio
			if mt, ok := c.targets[sv.Model]; ok {
				t, has = mt, 1
			}
		}
		f.srvPrio = append(f.srvPrio, int32(prio))
		f.srvHasTarget = append(f.srvHasTarget, has)
		f.sloITL, f.sloTTFT, f.sloTPS = append(f.sloITL, t.SLO_ITL), append(f.sloTTFT, t.SLO_TTFT), append(f.sloTPS, t.SLO_TPS)
		keep := uint8(0)
		if sv.KeepAccelerator {
			keep = 1
		}
		f.srvKeep = append(f.srvKeep, keep)
		f.srvMinRep = append(f.srvMinRep, int32(sv.MinNumReplicas))
		f.srvMaxBatch = append(f.srvMaxBatch, int32(sv.MaxBatchSize))
		ld := sv.CurrentAlloc.Load
		f.arrival = append(f.arrival, ld.ArrivalRate)
		f.inTok, f.outTok = append(f.inTok, int32(ld.AvgInTokens)), append(f.outTok, int32(ld.AvgOutTokens))
		ca := int32(accNone)
		if name := sv.CurrentAlloc.Accelerator; name != "" {
			if a, ok := accIdx[name]; ok {
				ca = int32(a)
			} else {
				ca = accUnknown
			}
		}
		f.curAcc = append(f.curAcc, ca)
		f.curRep = append(f.curRep, int32(sv.CurrentAlloc.NumReplicas))
		f.curCost = append(f.curCost, sv.CurrentAlloc.Cost)
	}
	f.unlimited = spec.Optimizer.Spec.Unlimited
	f.delayedBestEffort = spec.Optimizer.Spec.DelayedBestEffort
	f.saturationPolicy = int(config.SaturatedAllocationPolicyEnum(spec.Optimizer.Spec.SaturationPolicy))
	return f
}

func f32p(s []float32) *C.float {
	if len(s) == 0 {
		return nil
	}
	return (*C.float)(unsafe.Pointer(&s[0]))
}
func i32p(s []int32) *C.int32_t {
	if len(s) == 0 {
		return nil
	}
	return (*C.int32_t)(unsafe.Pointer(&s[0]))
}
func u8p(s []uint8) *C.uint8_t {
	if len(s) == 0 {
		return nil
	}
	return (*C.uint8_t)(unsafe.Pointer(&s[0]))
}

// cFleet fills the C image of a packed fleet.  The struct holds Go pointers: they are pinned on `pin` for the
// duration of the call that uses it (cgo rule; the library never retains them, include/wva_b200.h).
func cFleet(f *fleet, pin *runtime.Pinner) C.wva_fleet {
	var cf C.wva_fleet
	S := len(f.serverNames)
	cf.n_acc, cf.n_types = C.int32_t(len(f.accNames)), C.int32_t(len(f.typeCap))
	cf.n_models, cf.n_servers = C.int32_t(len(f.perfPresent)/max(len(f.accNames), 1)), C.int32_t(S)
	cf.acc_cost, cf.acc_multiplicity, cf.acc_type, cf.type_capacity = f32p(f.accCost), i32p(f.accMult), i32p(f.accType), i32p(f.typeCap)
	cf.perf_present, cf.perf_alpha, cf.perf_beta, cf.perf_gamma, cf.perf_delta = u8p(f.perfPresent), f32p(f.alpha), f32p(f.beta), f32p(f.gamma), f32p(f.delta)
	cf.perf_acc_count, cf.perf_max_batch, cf.perf_at_tokens = i32p(f.accCount), i32p(f.maxBatch), i32p(f.atTokens)
	cf.srv_model, cf.srv_priority, cf.srv_has_target = i32p(f.srvModel), i32p(f.srvPrio), u8p(f.srvHasTarget)
	cf.srv_slo_itl, cf.srv_slo_ttft, cf.srv_slo_tps = f32p(f.sloITL), f32p(f.sloTTFT), f32p(f.sloTPS)
	cf.srv_keep_acc, cf.srv_min_replicas, cf.srv_max_batch = u8p(f.srvKeep), i32p(f.srvMinRep), i32p(f.srvMaxBatch)
	cf.srv_arrival_rpm, cf.srv_in_tokens, cf.srv_out_tokens = f32p(f.arrival), i32p(f.inTok), i32p(f.outTok)
	cf.srv_cur_acc, cf.srv_cur_replicas, cf.srv_cur_cost = i32p(f.curAcc), i32p(f.curRep), f32p(f.curCost)
	for _, p := range []unsafe.Pointer{unsafe.Pointer(cf.acc_cost), unsafe.Pointer(cf.acc_multiplicity), unsafe.Pointer(cf.acc_type),
		unsafe.Pointer(cf.type_capacity), unsafe.Pointer(cf.perf_present), unsafe.Pointer(cf.perf_alpha), unsafe.Pointer(cf.perf_beta),
		unsafe.Pointer(cf.perf_gamma), unsafe.Pointer(cf.perf_delta), unsafe.Pointer(cf.perf_acc_count), unsafe.Pointer(cf.perf_max_batch),
		unsafe.Pointer(cf.perf_at_tokens), unsafe.Pointer(cf.srv_model), unsafe.Pointer(cf.srv_priority), unsafe.Pointer(cf.srv_has_target),
		unsafe.Pointer(cf.srv_slo_itl), unsafe.Pointer(cf.srv_slo_ttft), unsafe.Pointer(cf.srv_slo_tps), unsafe.Pointer(cf.srv_keep_acc),
		unsafe.Pointer(cf.srv_min_replicas), unsafe.Pointer(cf.srv_max_batch), unsafe.Pointer(cf.srv_arrival_rpm), unsafe.Pointer(cf.srv_in_tokens),
		unsafe.Pointer(cf.srv_out_tokens), unsafe.Pointer(cf.srv_cur_acc), unsafe.Pointer(cf.srv_cur_replicas), unsafe.Pointer(cf.srv_cur_cost)} {
		if p != nil {
			pin.Pin(p)
		}
	}
	if f.unlimited {
		cf.unlimited = 1
	}
	if f.delayedBestEffort {
		cf.delayed_best_effort = 1
	}
	cf.saturation_policy = C.int32_t(f.saturationPolicy)
	C.wva_tunables_default(&cf.tun)
	cf.tun.max_queue_to_batch_ratio = C.int32_t(config.MaxQueueToBatchRatio)
	cf.tun.accel_penalty_factor = C.float(config.AccelPenaltyFactor)
	return cf
}

// allocs is the host SoA of core.Allocation records the library writes (wva_allocs).
type allocs struct {
	feasible                                []uint8
	acc, replicas, batch                    []int32
	cost, value, itl, ttft, rho, maxRate    []float32
}

func newAllocs(n int, pin *runtime.Pinner) (*allocs, C.wva_allocs) {
	a := &allocs{feasible: make([]uint8, n), acc: make([]int32, n), replicas: make([]int32, n), batch: make([]int32, n),
		cost: make([]float32, n), value: make([]float32, n), itl: make([]float32, n), ttft: make([]float32, n),
		rho: make([]float32, n), maxRate: make([]float32, n)}
	var c C.wva_allocs
	c.feasible, c.acc, c.replicas, c.batch = u8p(a.feasible), i32p(a.acc), i32p(a.replicas), i32p(a.batch)
	c.cost, c.value, c.itl, c.ttft, c.rho, c.max_rate = f32p(a.cost), f32p(a.value), f32p(a.itl), f32p(a.ttft), f32p(a.rho), f32p(a.maxRate)
	for _, p := range []unsafe.Pointer{unsafe.Pointer(c.feasible), unsafe.Pointer(c.acc), unsafe.Pointer(c.replicas), unsafe.Pointer(c.batch),
		unsafe.Pointer(c.cost), unsafe.Pointer(c.value), unsafe.Pointer(c.itl), unsafe.Pointer(c.ttft), unsafe.Pointer(c.rho),
		unsafe.Pointer(c.max_rate)} {
		if p != nil {
			pin.Pin(p)
		}
	}
	return a, c
}

// slice views records lo .. hi-1 (one scenario's block of a wva_resolve_scenarios result).
func (a *allocs) slice(lo, hi int) *allocs {
	return &allocs{feasible: a.feasible[lo:hi], acc: a.acc[lo:hi], replicas: a.replicas[lo:hi], batch: a.batch[lo:hi],
		cost: a.cost[lo:hi], value: a.value[lo:hi], itl: a.itl[lo:hi], ttft: a.ttft[lo:hi], rho: a.rho[lo:hi],
		maxRate: a.maxRate[lo:hi]}
}

func (e *Engine) fail(what string, rc C.int) error {
	return fmt.Errorf("%s: %s: %s", what, C.GoString(C.wva_strerror(rc)), C.GoString(C.wva_last_error(e.h)))
}

// solution = System.GenerateSolution (pkg/core/system.go:303-319) over the winner records.
func (f *fleet) solution(win *allocs) *config.AllocationSolution {
	sol := &config.AllocationSolution{Spec: map[string]config.AllocationData{}}
	for s := range f.serverNames {
		if win.feasible[s] == 0 {
			continue
		}
		name := ""
		if win.acc[s] >= 0 {
			name = f.accNames[win.acc[s]]
		}
		sol.Spec[f.serverNames[s]] = config.AllocationData{
			Accelerator: name, NumReplicas: int(win.replicas[s]), MaxBatch: int(win.batch[s]), Cost: win.cost[s],
			ITLAverage: win.itl[s], TTFTAverage: win.ttft[s], Load: f.loads[s],
		}
	}
	return sol
}

// Solve = SetFromSpec + Server.Calculate for every server + Manager.Optimize + GenerateSolution.
func (e *Engine) Solve(spec *config.SystemSpec) (*config.AllocationSolution, error) {
	f := pack(spec)
	var pin runtime.Pinner
	defer pin.Unpin()
	cf := cFleet(f, &pin)
	win, cwin := newAllocs(len(f.serverNames), &pin)
	e.mu.Lock()
	defer e.mu.Unlock()
	if rc := C.wva_solve(e.h, &cf, nil, &cwin); rc != C.WVA_OK {
		return nil, e.fail("wva_solve", rc)
	}
	e.last = f
	return f.solution(win), nil
}

// CandidateAllocation is one entry of Server.AllAllocations() as the library computed it (core.Allocation's
// fields are private to pkg/core; AllocationFromData covers the subset the CR status needs).
type CandidateAllocation struct {
	Data                  config.AllocationData // accelerator, numReplicas, maxBatch, cost, itl, ttft
	Value, Rho            float32
	MaxArrvRatePerReplica float32 // req/msec
}

// Analyze = Server.Calculate for every server (pkg/core/server.go:55-67): per server name, the candidate
// allocation per accelerator name (nil candidates are absent, as in the reference's map).
func (e *Engine) Analyze(spec *config.SystemSpec) (map[string]map[string]CandidateAllocation, error) {
	f := pack(spec)
	var pin runtime.Pinner
	defer pin.Unpin()
	cf := cFleet(f, &pin)
	A := len(f.accNames)
	cand, ccand := newAllocs(len(f.serverNames)*A, &pin)
	e.mu.Lock()
	defer e.mu.Unlock()
	if rc := C.wva_analyze(e.h, &cf, &ccand); rc != C.WVA_OK {
		return nil, e.fail("wva_analyze", rc)
	}
	out := map[string]map[string]CandidateAllocation{}
	for s, srv := range f.serverNames {
		m := map[string]CandidateAllocation{}
		for a := 0; a < A; a++ {
			k := s*A + a
			if cand.feasible[k] == 0 {
				continue
			}
			name := ""
			if cand.acc[k] >= 0 {
				name = f.accNames[cand.acc[k]]
			}
			m[name] = CandidateAllocation{
				Data: config.AllocationData{Accelerator: name, NumReplicas: int(cand.replicas[k]), MaxBatch: int(cand.batch[k]),
					Cost: cand.cost[k], ITLAverage: cand.itl[k], TTFTAverage: cand.ttft[k], Load: f.loads[s]},
				Value: cand.value[k], Rho: cand.rho[k], MaxArrvRatePerReplica: cand.maxRate[k],
			}
		}
		out[srv] = m
	}
	return out, nil
}

// ---- streaming reconcile: the fleet stays resident on the GPU, only the load columns move per tick ----------

// Resident is the handle-side image of the last Upload (names for reading results back).
type Resident struct {
	f *fleet
}

// Upload packs the spec once and makes it resident (wva_upload).
func (e *Engine) Upload(spec *config.SystemSpec) (*Resident, error) {
	f := pack(spec)
	var pin runtime.Pinner
	defer pin.Unpin()
	cf := cFleet(f, &pin)
	e.mu.Lock()
	defer e.mu.Unlock()
	if rc := C.wva_upload(e.h, &cf); rc != C.WVA_OK {
		return nil, e.fail("wva_upload", rc)
	}
	e.last = f
	return &Resident{f: f}, nil
}

// UpdateLoad replaces the load of the named servers (collector output: internal/collector/collector.go:158-260)
// and ships the three load columns (wva_update_load: 12 B per server).
func (e *Engine) UpdateLoad(r *Resident, loads map[string]config.ServerLoadSpec) error {
	f := r.f
	for s, name := range f.serverNames {
		if ld, ok := loads[name]; ok {
			f.loads[s] = ld
			f.arrival[s], f.inTok[s], f.outTok[s] = ld.ArrivalRate, int32(ld.AvgInTokens), int32(ld.AvgOutTokens)
		}
	}
	var pin runtime.Pinner
	defer pin.Unpin()
	pa, pi, po := f32p(f.arrival), i32p(f.inTok), i32p(f.outTok)
	for _, p := range []unsafe.Pointer{unsafe.Pointer(pa), unsafe.Pointer(pi), unsafe.Pointer(po)} {
		if p != nil {
			pin.Pin(p)
		}
	}
	e.mu.Lock()
	defer e.mu.Unlock()
	if rc := C.wva_update_load(e.h, pa, pi, po); rc != C.WVA_OK {
		return e.fail("wva_update_load", rc)
	}
	return nil
}

// Resolve = Manager.Optimize + GenerateSolution on the resident fleet (wva_resolve).
func (e *Engine) Resolve(r *Resident) (*config.AllocationSolution, error) {
	var pin runtime.Pinner
	defer pin.Unpin()
	win, cwin := newAllocs(len(r.f.serverNames), &pin)
	e.mu.Lock()
	defer e.mu.Unlock()
	if rc := C.wva_resolve(e.h, nil, &cwin); rc != C.WVA_OK {
		return nil, e.fail("wva_resolve", rc)
	}
	return r.f.solution(win), nil
}

// ResolveScenarios is Resolve under len(loads) arrival-rate scenarios in one call (wva_resolve_scenarios): forecast
// peaks, load percentiles, "what at 2x traffic".  loads[l] maps server names to scenario l's ArrivalRate (req/min);
// a server missing from it keeps its resident rate.  Solution l equals UpdateLoad(arrival rates of loads[l]) +
// Resolve, but the resident fleet keeps its own load, and Summarize has nothing to report until the next solve.
func (e *Engine) ResolveScenarios(r *Resident, loads []map[string]float32) ([]*config.AllocationSolution, error) {
	f := r.f
	L, S := len(loads), len(f.serverNames)
	if L == 0 {
		return nil, nil
	}
	rows := make([]float32, L*S)
	for l, ld := range loads {
		row := rows[l*S : (l+1)*S]
		copy(row, f.arrival)
		for s, name := range f.serverNames {
			if v, ok := ld[name]; ok {
				row[s] = v
			}
		}
	}
	var pin runtime.Pinner
	defer pin.Unpin()
	pr := f32p(rows)
	pin.Pin(unsafe.Pointer(pr))
	win, cwin := newAllocs(L*S, &pin)
	e.mu.Lock()
	defer e.mu.Unlock()
	if rc := C.wva_resolve_scenarios(e.h, C.int32_t(L), pr, nil, &cwin); rc != C.WVA_OK {
		return nil, e.fail("wva_resolve_scenarios", rc)
	}
	out := make([]*config.AllocationSolution, L)
	for l := range out {
		sol := f.solution(win.slice(l*S, (l+1)*S))
		for s, name := range f.serverNames { // the solution reports the load it was sized for
			if d, ok := sol.Spec[name]; ok {
				d.Load.ArrivalRate = rows[l*S+s]
				sol.Spec[name] = d
			}
		}
		out[l] = sol
	}
	return out, nil
}

// ---- System.AllocateByType + Solver.Solve's diffs ---------------------------------------------------------

// TypeTotal mirrors core.AllocationByType (pkg/core/system.go:60-65).
type TypeTotal struct {
	Count, Limit int
	Cost         float32
}

// MM1KStats mirrors the statistics of analyzer.MM1KModel after Solve (pkg/analyzer/queuemodel.go:10-19).
type MM1KStats struct {
	IsValid                                                                                     bool
	Rho, AvgNumInSystem, Throughput, AvgRespTime, AvgServTime, AvgWaitTime, AvgQueueLength float32
}

// MM1K evaluates analyzer.MM1KModel (closed form, pkg/analyzer/mm1kmodel.go) for n (K, lambda, mu) triples
// on the device (wva_mm1k_solve).
func (e *Engine) MM1K(K []int32, lambda, mu []float32) ([]MM1KStats, error) {
	n := len(K)
	if len(lambda) != n || len(mu) != n {
		return nil, fmt.Errorf("wva_mm1k_solve: K, lambda, mu must have one length")
	}
	if n == 0 {
		return nil, nil
	}
	valid := make([]uint8, n)
	cols := make([][]float32, 7)
	for i := range cols {
		cols[i] = make([]float32, n)
	}
	var pin runtime.Pinner
	defer pin.Unpin()
	var out C.wva_mm1k_out
	out.is_valid = u8p(valid)
	out.rho, out.avg_num_in_system, out.throughput, out.avg_resp_time = f32p(cols[0]), f32p(cols[1]), f32p(cols[2]), f32p(cols[3])
	out.avg_serv_time, out.avg_wait_time, out.avg_queue_length = f32p(cols[4]), f32p(cols[5]), f32p(cols[6])
	pin.Pin(unsafe.Pointer(out.is_valid))
	for _, p := range []*C.float{out.rho, out.avg_num_in_system, out.throughput, out.avg_resp_time, out.avg_serv_time,
		out.avg_wait_time, out.avg_queue_length} {
		pin.Pin(unsafe.Pointer(p))
	}
	e.mu.Lock()
	defer e.mu.Unlock()
	if rc := C.wva_mm1k_solve(e.h, C.int32_t(n), i32p(K), f32p(lambda), f32p(mu), &out); rc != C.WVA_OK {
		return nil, e.fail("wva_mm1k_solve", rc)
	}
	res := make([]MM1KStats, n)
	for i := range res {
		res[i] = MM1KStats{valid[i] != 0, cols[0][i], cols[1][i], cols[2][i], cols[3][i], cols[4][i], cols[5][i], cols[6][i]}
	}
	return res, nil
}

// Diff mirrors core.AllocationDiff (pkg/core/allocation.go:344-350); accelerator "none" = no allocation.
type Diff struct {
	OldAccelerator, NewAccelerator string
	OldNumReplicas, NewNumReplicas int
	CostDiff                       float32
}

// Summarize reads both for the most recent Solve / Resolve on this engine (wva_summarize).
func (e *Engine) Summarize() (map[string]TypeTotal, map[string]Diff, error) {
	f := e.last
	if f == nil {
		return nil, nil, fmt.Errorf("wva_summarize: no solution yet")
	}
	typeNames := f.typeNames
	T, S := len(f.typeCap), len(f.serverNames)
	present, count, limit, cost := make([]uint8, T), make([]int64, T), make([]int32, T), make([]float32, T)
	oa, na, or, nr, dc := make([]int32, S), make([]int32, S), make([]int32, S), make([]int32, S), make([]float32, S)
	var pin runtime.Pinner
	defer pin.Unpin()
	var cs C.wva_summary
	cs.type_present, cs.type_limit, cs.type_cost = u8p(present), i32p(limit), f32p(cost)
	if T > 0 {
		cs.type_count = (*C.int64_t)(unsafe.Pointer(&count[0]))
	}
	cs.diff_old_acc, cs.diff_new_acc, cs.diff_old_replicas, cs.diff_new_replicas, cs.diff_cost = i32p(oa), i32p(na), i32p(or), i32p(nr), f32p(dc)
	for _, p := range []unsafe.Pointer{unsafe.Pointer(cs.type_present), unsafe.Pointer(cs.type_count), unsafe.Pointer(cs.type_limit),
		unsafe.Pointer(cs.type_cost), unsafe.Pointer(cs.diff_old_acc), unsafe.Pointer(cs.diff_new_acc), unsafe.Pointer(cs.diff_old_replicas),
		unsafe.Pointer(cs.diff_new_replicas), unsafe.Pointer(cs.diff_cost)} {
		if p != nil {
			pin.Pin(p)
		}
	}
	e.mu.Lock()
	defer e.mu.Unlock()
	if rc := C.wva_summarize(e.h, &cs); rc != C.WVA_OK {
		return nil, nil, e.fail("wva_summarize", rc)
	}
	name := func(a int32) string {
		switch {
		case a >= 0:
			return f.accNames[a]
		case a == accAbsent:
			return "none"
		default:
			return "" // accNone; an unknown current accelerator keeps the name it had in the spec
		}
	}
	byType := map[string]TypeTotal{}
	for t := 0; t < T; t++ {
		if present[t] != 0 {
			byType[typeNames[t]] = TypeTotal{Count: int(count[t]), Limit: int(limit[t]), Cost: cost[t]}
		}
	}
	diffs := map[string]Diff{}
	for s, srv := range f.serverNames {
		diffs[srv] = Diff{OldAccelerator: name(oa[s]), NewAccelerator: name(na[s]), OldNumReplicas: int(or[s]),
			NewNumReplicas: int(nr[s]), CostDiff: dc[s]}
	}
	return byType, diffs, nil
}

// ---- drop-ins for the controller's two adapter types -------------------------------------------------------

// ModelAnalyzer is the drop-in for internal/modelanalyzer.ModelAnalyzer (analyzer.go:12-34): the controller
// calls AnalyzeModel once per server in a loop (variantautoscaling_controller.go:148-156); the first call
// analyses the WHOLE fleet in one device call and the rest read the cached table.
type ModelAnalyzer struct {
	engine *Engine
	spec   *config.SystemSpec
	once   sync.Once
	table  map[string]map[string]CandidateAllocation
	err    error
}

func NewModelAnalyzer(engine *Engine, spec *config.SystemSpec) *ModelAnalyzer {
	return &ModelAnalyzer{engine: engine, spec: spec}
}

// ModelAcceleratorAllocation carries what interfaces.ModelAcceleratorAllocation carries (types.go:12-18); the
// embedded *inferno.Allocation of the original is replaced by its exported data, because core.Allocation cannot
// be built outside pkg/core with rho / maxArrvRatePerReplica set.
type ModelAcceleratorAllocation struct {
	Allocation         CandidateAllocation
	RequiredPrefillQPS float64
	RequiredDecodeQPS  float64
	Reason             string
}

// AnalyzeModel mirrors analyzer.go:25-34 + CreateModelAnalyzeResponseFromAllocations (utils.go:9-24): an unknown
// server yields an empty response, never an error.
func (ma *ModelAnalyzer) AnalyzeModel(ctx context.Context, va llmdOptv1alpha1.VariantAutoscaling) (map[string]*ModelAcceleratorAllocation, error) {
	ma.once.Do(func() { ma.table, ma.err = ma.engine.Analyze(ma.spec) })
	if ma.err != nil {
		return nil, ma.err
	}
	out := map[string]*ModelAcceleratorAllocation{}
	for acc, c := range ma.table[utils.FullName(va.Name, va.Namespace)] {
		qps := float64(c.MaxArrvRatePerReplica * 1000) // float32 product first, as alloc.MaxArrvRatePerReplica() * 1000
		out[acc] = &ModelAcceleratorAllocation{Allocation: c, RequiredPrefillQPS: qps, RequiredDecodeQPS: qps, Reason: "markovian analysis"}
	}
	return out, nil
}

// VariantAutoscalingsEngine is the drop-in for internal/optimizer.VariantAutoscalingsEngine
// (same method set: interfaces.VariantAutoscalingsEngine, internal/interfaces/interfaces.go:10-17).
type VariantAutoscalingsEngine struct {
	engine *Engine
	spec   *config.SystemSpec
}

func NewVariantAutoscalingsEngine(engine *Engine, spec *config.SystemSpec) *VariantAutoscalingsEngine {
	return &VariantAutoscalingsEngine{engine: engine, spec: spec}
}

// Optimize mirrors internal/optimizer/optimizer.go:30-54 (the analysis argument is ignored there too).
func (v *VariantAutoscalingsEngine) Optimize(ctx context.Context, vaList llmdOptv1alpha1.VariantAutoscalingList,
	_ map[string]*interfaces.ModelAnalyzeResponse) (map[string]llmdOptv1alpha1.OptimizedAlloc, error) {
	sol, err := v.engine.Solve(v.spec)
	if err != nil {
		return nil, err
	}
	if len(sol.Spec) == 0 {
		return nil, fmt.Errorf("no feasible allocations found for all variants: ")
	}
	out := make(map[string]llmdOptv1alpha1.OptimizedAlloc)
	for _, va := range vaList.Items {
		if oa, err := utils.CreateOptimizedAlloc(va.Name, va.Namespace, sol); err == nil {
			out[va.Name] = *oa
		}
	}
	return out, nil
}
