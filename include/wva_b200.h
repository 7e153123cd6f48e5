/*
 * wva_b200.h — C ABI of the B200-native WVA optimizer hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b): the seam between WVA's L2
 * adapters (internal/modelanalyzer, internal/optimizer) and the L1 "inferno"
 * optimizer library (pkg/analyzer, pkg/core, pkg/solver, pkg/manager).  The Go
 * side packs a `config.SystemSpec` (pkg/config/types.go:11-21) into the flat
 * SoA `wva_fleet` below, makes ONE call, and reads back what
 * `System.GenerateSolution()` (pkg/core/system.go:303-319) would have produced.
 *
 * Plain C: pointers + sizes only.  All arrays are caller-owned HOST memory; the
 * library never retains a caller pointer after a call returns (cgo rule).  One
 * call at a time per handle (the reference L1 is non-reentrant as well:
 * pkg/core/system.go:10-13, pkg/analyzer/utils.go:73).
 *
 * Error model (pkg/core/allocation.go:42-70,111-130,150-153): an infeasible
 * candidate is DATA (`feasible == 0`, the reference's `nil *Allocation`), never
 * an error code.  Negative return values are hard errors only (bad arguments,
 * CUDA failure, missing device).
 *
 * Arithmetic contract: results are bit-identical to the reference Go code built
 * for amd64 at GOAMD64=v1 (IEEE binary32/binary64, round-to-nearest-even, no FMA
 * contraction) — integers exactly, float32 outputs bit-for-bit.
 */
#ifndef WVA_B200_H
#define WVA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WVA_ABI_VERSION 2

/* ---- return codes ------------------------------------------------------- */
#define WVA_OK 0
#define WVA_ERR_BAD_ARG (-1)     /* NULL pointer, negative size, id out of range   */
#define WVA_ERR_NO_DEVICE (-2)   /* no CUDA device / requested ordinal missing      */
#define WVA_ERR_CUDA (-3)        /* a CUDA runtime call failed (see wva_last_error) */
#define WVA_ERR_NOMEM (-4)       /* host or device allocation failed                */
#define WVA_ERR_STATE (-5)       /* call sequence error (e.g. resolve before upload)*/
#define WVA_ERR_UNSUPPORTED (-6) /* input outside the supported numeric domain      */

/* ---- sentinels ---------------------------------------------------------- */
#define WVA_ACC_NONE (-1)    /* accelerator name "" (pkg/core/allocation.go:264)    */
#define WVA_ACC_UNKNOWN (-2) /* a name that is not in the accelerator table         */
#define WVA_ACC_ABSENT (-3)  /* no allocation at all: CreateAllocationDiff's "none"  */

/* saturation policies: pkg/config/config.go:4-41 */
#define WVA_SAT_NONE 0
#define WVA_SAT_PRIORITY_EXHAUSTIVE 1
#define WVA_SAT_PRIORITY_ROUND_ROBIN 2
#define WVA_SAT_ROUND_ROBIN 3

typedef struct wva_handle wva_handle;

/*
 * Tunables that are package-level variables in the reference
 * (pkg/config/defaults.go:18,21).  wva_tunables_default() fills the reference values.
 */
typedef struct wva_tunables {
    int32_t max_queue_to_batch_ratio; /* config.MaxQueueToBatchRatio = 10          */
    float accel_penalty_factor;       /* config.AccelPenaltyFactor   = 0.1         */
} wva_tunables;

/*
 * The fleet: flat SoA image of config.SystemSpec after the joins that
 * System.SetFromSpec (pkg/core/system.go:82-194) performs with Go maps.
 *
 *   A accelerators   — config.AcceleratorSpec   (pkg/config/types.go:29-37)
 *   T accelerator types + capacity — config.AcceleratorCount (types.go:52-56)
 *   M models; perf data per (model, accelerator), row-major [M*A]
 *                    — config.ModelAcceleratorPerfData (types.go:64-72)
 *   S servers        — config.ServerSpec (types.go:112-121) joined with its
 *                      service class / model target (types.go:92-105)
 */
typedef struct wva_fleet {
    /* accelerators [A] */
    int32_t n_acc;
    const float *acc_cost;           /* AcceleratorSpec.Cost (cents/hr)                 */
    const int32_t *acc_multiplicity; /* AcceleratorSpec.Multiplicity                    */
    const int32_t *acc_type;         /* type id in [0, n_types)                         */

    /* accelerator types [T]; only read in limited (greedy) mode */
    int32_t n_types;
    const int32_t *type_capacity; /* CapacityData count; types absent in Go map = 0  */

    /* per (model, accelerator) [M*A], index m*A + a */
    int32_t n_models;
    const uint8_t *perf_present;   /* 1 iff model.PerfData(acc) != nil                */
    const float *perf_alpha;       /* DecodeParms.Alpha                               */
    const float *perf_beta;        /* DecodeParms.Beta                                */
    const float *perf_gamma;       /* PrefillParms.Gamma                              */
    const float *perf_delta;       /* PrefillParms.Delta                              */
    const int32_t *perf_acc_count; /* AccCount (<=0 -> 1, pkg/core/model.go:52-55)    */
    const int32_t *perf_max_batch; /* MaxBatchSize                                    */
    const int32_t *perf_at_tokens; /* AtTokens                                        */

    /* servers [S] */
    int32_t n_servers;
    const int32_t *srv_model;       /* model id, or -1 if the model name is unknown   */
    const int32_t *srv_priority;    /* service class priority (server.go:92-97)       */
    const uint8_t *srv_has_target;  /* service class exists AND has a target for model*/
    const float *srv_slo_itl;       /* Target.ITL  (msec)                             */
    const float *srv_slo_ttft;      /* Target.TTFT (msec)                             */
    const float *srv_slo_tps;       /* Target.TPS  (tokens/sec)                       */
    const uint8_t *srv_keep_acc;    /* ServerSpec.KeepAccelerator                     */
    const int32_t *srv_min_replicas;/* ServerSpec.MinNumReplicas                      */
    const int32_t *srv_max_batch;   /* ServerSpec.MaxBatchSize override (0 = none)    */
    const float *srv_arrival_rpm;   /* ServerLoadSpec.ArrivalRate (req/min)           */
    const int32_t *srv_in_tokens;   /* ServerLoadSpec.AvgInTokens                     */
    const int32_t *srv_out_tokens;  /* ServerLoadSpec.AvgOutTokens                    */
    const int32_t *srv_cur_acc;     /* CurrentAlloc.Accelerator: id, NONE or UNKNOWN  */
    const int32_t *srv_cur_replicas;/* CurrentAlloc.NumReplicas                       */
    const float *srv_cur_cost;      /* CurrentAlloc.Cost                              */

    /* optimizer spec (pkg/config/types.go:151-155) */
    uint8_t unlimited;
    uint8_t delayed_best_effort;
    int32_t saturation_policy; /* WVA_SAT_* */

    wva_tunables tun;
} wva_fleet;

/*
 * One candidate allocation per (server, accelerator): the fields of
 * core.Allocation (pkg/core/allocation.go:13-24).  Arrays have S*A entries
 * (index s*A + a) for candidate tables, S entries for per-server winners.
 * Any pointer may be NULL (that column is not written).
 */
typedef struct wva_allocs {
    uint8_t *feasible;  /* 0 = nil allocation                                        */
    int32_t *acc;       /* accelerator id; WVA_ACC_NONE for the zero-replica case    */
    int32_t *replicas;  /* numReplicas                                               */
    int32_t *batch;     /* batchSize                                                 */
    float *cost;        /* cost                                                      */
    float *value;       /* value (transition penalty, pkg/core/server.go:60-63)      */
    float *itl;         /* expected inter-token latency (msec)                       */
    float *ttft;        /* expected queueing + prefill time (msec)                   */
    float *rho;         /* utilisation                                               */
    float *max_rate;    /* maxArrvRatePerReplica (req/msec)                          */
} wva_allocs;

/*
 * Candidate grid (the build's generalisation, SURVEY.md §8d): every
 * (server, accelerator, batch, replica) cell is one QueueAnalyzer.Analyze
 * (pkg/analyzer/queueanalyzer.go:134-174) at rate totalRate(server)/replicas
 * with MaxBatchSize = batch, followed by the SLO feasibility test, the cost and
 * the transition penalty.  Cell index = ((s*A + a)*B + bi)*R + ri.
 */
typedef struct wva_grid {
    int32_t n_batch;
    const int32_t *batch; /* [B] batch sizes, each >= 1                           */
    int32_t n_replicas;
    const int32_t *replicas; /* [R] replica counts, each >= 1                     */
} wva_grid;

/* Optional per-cell table (any pointer may be NULL). flags bit0 = Analyze ok,
 * bit1 = SLO-feasible (implies bit0). */
typedef struct wva_cells {
    uint8_t *flags;
    float *ttft;       /* AvgWaitTime + AvgPrefillTime                             */
    float *itl;        /* AvgTokenTime                                             */
    float *rho;        /* Rho                                                      */
    float *throughput; /* Throughput (req/sec)                                     */
} wva_cells;

/* Latency sweep (BASELINE config 3): for each (server, accelerator) pair,
 * Analyze at n_rates rates linearly spaced in [RateRange.Min, RateRange.Max*0.999].
 * Output index = (s*A + a)*n_rates + i. valid = 0 where the pair has no model or
 * Analyze returned an error.  Points whose chain leaves the streaming solve's numeric
 * window (including those the reference rescales) are re-run on the stored-vector
 * fallback; WVA_ERR_UNSUPPORTED only where the reference's rescale would not
 * terminate or more than 2^22 points need the fallback. */
typedef struct wva_sweep_out {
    uint8_t *valid;
    float *rate;       /* req/sec                                                  */
    float *ttft;
    float *itl;
    float *throughput;
    float *rho;
} wva_sweep_out;

/* ---- lifecycle ---------------------------------------------------------- */

/* Reference values of the package-level tunables. */
void wva_tunables_default(wva_tunables *t);

/* Create an engine bound to CUDA device `device` (ordinal). Fails with
 * WVA_ERR_NO_DEVICE when there is no such GPU: there is no CPU fallback. */
int wva_create(wva_handle **out, int device);
void wva_destroy(wva_handle *h);

const char *wva_strerror(int code);
/* Text of the last hard error on this handle ("" if none). */
const char *wva_last_error(const wva_handle *h);
int wva_abi_version(void);

/* ---- the hot path -------------------------------------------------------- */

/*
 * Server.Calculate for every server (pkg/core/server.go:55-67): one
 * CreateAllocation (pkg/core/allocation.go:27-163) per candidate accelerator and
 * value = TransitionPenalty(current, candidate) (allocation.go:291-300).
 * Replaces ModelAnalyzer.AnalyzeModel (internal/modelanalyzer/analyzer.go:25-34)
 * called in a loop at internal/controller/variantautoscaling_controller.go:149-156.
 * `candidates` has S*A entries.
 */
int wva_analyze(wva_handle *h, const wva_fleet *fleet, wva_allocs *candidates);

/*
 * Analyze + Solver.Solve (pkg/solver/solver.go:32-59): SolveUnlimited
 * (solver.go:63-79) when fleet->unlimited, else SolveGreedy
 * (pkg/solver/greedy.go:35-104) over the device-computed candidates.  Replaces
 * VariantAutoscalingsEngine.Optimize (internal/optimizer/optimizer.go:30-54) =
 * Manager.Optimize (pkg/manager/manager.go:21-27) + System.GenerateSolution
 * (pkg/core/system.go:303-319).  `winners` has S entries; `candidates` (S*A) may
 * be NULL.  Ties on value are resolved to the lowest accelerator id (the
 * reference resolves them by Go map iteration order, i.e. randomly).
 */
int wva_solve(wva_handle *h, const wva_fleet *fleet, wva_allocs *candidates,
              wva_allocs *winners);

/*
 * Full candidate grid + per-server min-value SLO-feasible cell.
 * Winner order: value, then cost, then replicas, then batch, then accelerator id
 * (all ascending).  `cells` may be NULL.
 */
int wva_grid_solve(wva_handle *h, const wva_fleet *fleet, const wva_grid *grid,
                   wva_cells *cells, wva_allocs *winners);

/*
 * Solver.SolveGreedy + the best-effort saturation policies (pkg/solver/greedy.go:35-341) over a candidate
 * table the caller already holds: `candidates` (S*A, value = transition penalty as wva_analyze returns it) is
 * read, and modified where the reference scales best-effort allocations; `winners` (S) is written.  Host only
 * (no handle, no device work).  The multi-GPU limited mode shards candidate generation over the ranks,
 * all-gathers the candidate tables and calls this on every rank (SURVEY.md 8e): the greedy pass is one
 * sequential walk over a shared capacity map and does not shard.
 */
int wva_solve_greedy(const wva_fleet *fleet, wva_allocs *candidates, wva_allocs *winners);

/* Latency sweep of QueueAnalyzer.Analyze over n_rates rates per (server, acc). */
int wva_sweep(wva_handle *h, const wva_fleet *fleet, int32_t n_rates, wva_sweep_out *out);

/*
 * What Manager.Optimize / Solver.Solve leave behind besides the per-server solution
 * (pkg/manager/manager.go:21-27): the per-accelerator-type totals of System.AllocateByType
 * (pkg/core/system.go:271-300) and the per-server orchestration differences of
 * CreateAllocationDiff (pkg/core/allocation.go:353-380, collected by pkg/solver/solver.go:51-58).
 * Any pointer may be NULL (that column is not written).
 *
 *   type_*  [T]: present = the type has an entry in the reference's allocationByType map (some
 *                server was allocated an accelerator of that type); count = sum of
 *                numReplicas * numInstances(model, acc) * multiplicity(acc); limit = capacity of the
 *                type (0 when the capacity map has no entry); cost = sum of the allocations' cost.
 *                The reference accumulates the float32 cost in Go map order (random); here the order
 *                is ascending server index.
 *   diff_*  [S]: old = CurrentAlloc of the server spec (always present: core/server.go:49), new = the
 *                solution's allocation, accelerator WVA_ACC_ABSENT / 0 replicas / cost 0 when the
 *                server got none ("none" in the reference); cost = newCost - oldCost.
 */
typedef struct wva_summary {
    uint8_t *type_present;
    int64_t *type_count;
    int32_t *type_limit;
    float *type_cost;
    int32_t *diff_old_acc;
    int32_t *diff_new_acc;
    int32_t *diff_old_replicas;
    int32_t *diff_new_replicas;
    float *diff_cost;
} wva_summary;

/* Summary of the most recent wva_solve / wva_resolve / wva_grid_solve on this handle (the winners
 * stay resident until the next call).  WVA_ERR_STATE when there is none. */
int wva_summarize(wva_handle *h, wva_summary *out);

/* ---- MM1KModel (closed form) --------------------------------------------- */

/*
 * MM1KModel.Solve for n independent (K, lambda, mu) triples: pkg/analyzer/mm1kmodel.go:19-92 over
 * QueueModel.Solve (queuemodel.go:27-37).  The reference keeps this model next to the state-dependent one but
 * does not call it on the production path; it is here so that every model of pkg/analyzer has a device function.
 * One thread per triple, p[] is streamed (never stored).  math.Pow is restated from the Go standard library's
 * binary-powering algorithm (integer exponents only occur) so that host oracle and device agree bit for bit; it is
 * not pinned against the Go binary (no Go toolchain here), see DESIGN.md.
 * Columns have n entries (host pointers, any may be NULL); entries of an invalid triple are 0 except rho.
 * K < 0 is WVA_ERR_BAD_ARG (NewMM1KModel returns nil), K > 2^20 WVA_ERR_UNSUPPORTED.
 */
typedef struct wva_mm1k_out {
    uint8_t *is_valid;
    float *rho;
    float *avg_num_in_system;
    float *throughput;
    float *avg_resp_time;
    float *avg_serv_time;
    float *avg_wait_time;
    float *avg_queue_length;
    double *sum_p; /* sum of the state probabilities as the reference accumulates it */
} wva_mm1k_out;
int wva_mm1k_solve(wva_handle *h, int32_t n, const int32_t *K, const float *lambda, const float *mu,
                   wva_mm1k_out *out);

/* ---- streaming reconcile (BASELINE config 5) ---------------------------- */

/* Make `fleet` resident on the device (copies everything; caller memory is not
 * retained). Subsequent wva_update_load / wva_resolve calls reuse it. */
int wva_upload(wva_handle *h, const wva_fleet *fleet);
/* Replace the load columns of the resident fleet (any pointer may be NULL =
 * keep). Arrays have S entries. */
int wva_update_load(wva_handle *h, const float *arrival_rpm, const int32_t *in_tokens,
                    const int32_t *out_tokens);
/* wva_solve on the resident fleet. */
int wva_resolve(wva_handle *h, wva_allocs *candidates, wva_allocs *winners);
/* The reconcile of wva_resolve, repeated for n_scen arrival-rate columns of the resident fleet
 * (forecast peaks, load percentiles, "what at 2x traffic").
 *   arrival_rpm [n_scen * S]  row l = ServerLoadSpec.ArrivalRate of every server in scenario l (req/min)
 *   candidates  [n_scen * S * A], index (l*S + s)*A + a; may be NULL
 *   winners     [n_scen * S],     index l*S + s
 * Scenario l's records are bit-identical to wva_update_load(arrival_rpm = row l) + wva_resolve, in unlimited and
 * limited mode, and the call fails with the code wva_resolve would return for some scenario.  Only the arrival rate
 * varies: QueueAnalyzer.Size never reads it, so each candidate is sized once and only CreateAllocation's per-load
 * steps and final Analyze run per scenario.  The resident fleet (its load columns included) is not changed, but the
 * most recent solution is cleared as by wva_update_load; wva_last_kernel_ms / wva_last_device_ms cover this call.
 * WVA_ERR_BAD_ARG for n_scen < 1 or a NULL arrival_rpm / winners; WVA_ERR_UNSUPPORTED for n_scen > 65535 or
 * n_scen * S * A > 2^31 - 1 (the kernels' index range). */
int wva_resolve_scenarios(wva_handle *h, int32_t n_scen, const float *arrival_rpm, wva_allocs *candidates,
                          wva_allocs *winners);

/* ---- device-resident variants (used by the multi-GPU driver and bench) --- */

/*
 * As wva_grid_solve / wva_resolve on the resident fleet, but `winners` columns are
 * DEVICE pointers (e.g. torch tensors) and nothing is copied to the host; the
 * work is enqueued on the handle's stream and the call returns without
 * synchronising.  wva_stream() exposes that cudaStream_t so that the caller can
 * order an NCCL all-gather of the winner records after it.
 */
int wva_grid_solve_device(wva_handle *h, const wva_grid *grid, wva_allocs *winners_dev);
int wva_resolve_device(wva_handle *h, wva_allocs *winners_dev);
void *wva_stream(wva_handle *h);
int wva_synchronize(wva_handle *h);

/* Number of kernel launches issued by this handle since creation. */
int64_t wva_launch_count(const wva_handle *h);
/* Device time (ms, CUDA events on the handle's stream) of the dominant kernel in
 * the most recent call, and of the whole call's device work. */
float wva_last_kernel_ms(const wva_handle *h);
float wva_last_device_ms(const wva_handle *h);

/* --- multi-GPU: all-gather of the per-rank winner block over peer memory --------------------
 * One process per GPU on one node.  Replaces the collective the reference does not have (its optimizer
 * is single-process; SURVEY.md 8e): each rank writes its block straight into every peer's gathered
 * buffer over NVLink and waits for the peers' blocks, in ONE kernel on the handle's stream.
 *   wva_xchg_create   allocate this rank's gathered buffer, return its 64-byte CUDA IPC handle
 *   wva_xchg_open     register the IPC handle of rank `peer_rank` (exchange the handles with any
 *                     host-side transport, e.g. torch.distributed all_gather_object); call for every rank
 *   wva_xchg_publish  enqueue the exchange of `src_block` (device memory, block_bytes); *gathered is the
 *                     device address of this step's [world][*slot_stride] byte buffer, valid once the
 *                     stream has passed the call (double-buffered by step parity)
 *   wva_xchg_error    after a synchronize: 1 if a peer never arrived (the kernel gives up after ~2 s)
 */
int wva_xchg_create(wva_handle *h, int world, int rank, size_t block_bytes, void *ipc_handle_out);
int wva_xchg_open(wva_handle *h, int peer_rank, const void *ipc_handle);
int wva_xchg_publish(wva_handle *h, const void *src_block, void **gathered, size_t *slot_stride);
int wva_xchg_error(wva_handle *h);
int wva_xchg_destroy(wva_handle *h);

#ifdef __cplusplus
}
#endif
#endif /* WVA_B200_H */
