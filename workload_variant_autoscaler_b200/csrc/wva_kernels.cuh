// wva_kernels.cuh — sm_100a kernels of the WVA optimizer hot path.
//
//   build_pair_tables   servRate[n] (+ double-word reciprocal) per (server, accelerator)
//   grid_* kernels K2   one Analyze per (server, acc, batch, replica) cell: row sharing, length-class
//                       sort, persistent warps pulling 32-cell items, fused feasibility + batch-rank minimum
//   grid_fallback       stored-vector re-run of the rare cells the streaming solve bails on
//   grid_finalize  K3   per-server argmin over partials (warp shuffle -> smem -> record)
//   sz2_* kernels  K1   (wva_size.cuh) CreateAllocation per (server, acc) candidate as rounds of sorted solve
//                       batches with speculative bisection trees
//   size_fallback       stored-vector re-run of candidates that bailed
//   trivial_kernel      nil / zero-load candidates (per scenario for wva_resolve_scenarios)
//   unlimited_kernel    Server.Calculate value + SolveUnlimited argmin per server (and scenario)
//   sweep_kernel        Analyze over a rate sweep per (server, acc)
//   sweep_fallback      stored-vector re-run of sweep points that bailed
#pragma once
#include "wva_device.cuh"

namespace wva {

// Device image of wva_fleet (all pointers are device pointers).
struct DevFleet {
    int A, T, M, S;
    const float* acc_cost;
    const int* acc_mult;
    const int* acc_type;
    const int* type_capacity;
    const uint8_t* perf_present;
    const float *perf_alpha, *perf_beta, *perf_gamma, *perf_delta;
    const int *perf_acc_count, *perf_max_batch, *perf_at_tokens;
    const int *srv_model, *srv_priority;
    const uint8_t* srv_has_target;
    const float *srv_slo_itl, *srv_slo_ttft, *srv_slo_tps;
    const uint8_t* srv_keep_acc;
    const int *srv_min_replicas, *srv_max_batch;
    const float* srv_arrival_rpm;
    const int *srv_in_tokens, *srv_out_tokens;
    const int *srv_cur_acc, *srv_cur_replicas;
    const float* srv_cur_cost;
    int ratio;      // config.MaxQueueToBatchRatio
    float penalty;  // config.AccelPenaltyFactor
};

// One candidate allocation (core.Allocation, pkg/core/allocation.go:13-24).
struct Cand {
    float value, cost;
    int replicas, batch, acc;
    float itl, ttft, rho, max_rate;
    int feasible;
};
__device__ __forceinline__ Cand cand_nil() {
    Cand c;
    c.value = 0.f; c.cost = 0.f; c.replicas = 0; c.batch = 0; c.acc = -1;
    c.itl = 0.f; c.ttft = 0.f; c.rho = 0.f; c.max_rate = 0.f; c.feasible = 0;
    return c;
}
// Grid winner order: value, cost, replicas, batch, accelerator id (ascending).
__device__ __forceinline__ bool cand_better(const Cand& x, const Cand& y) {
    if (!x.feasible) return false;
    if (!y.feasible) return true;
    if (x.value != y.value) return x.value < y.value;
    if (x.cost != y.cost) return x.cost < y.cost;
    if (x.replicas != y.replicas) return x.replicas < y.replicas;
    if (x.batch != y.batch) return x.batch < y.batch;
    return x.acc < y.acc;
}
__device__ __forceinline__ Cand cand_shfl_down(const Cand& c, int d) {
    Cand o;
    o.value = __shfl_down_sync(0xffffffffu, c.value, d);
    o.cost = __shfl_down_sync(0xffffffffu, c.cost, d);
    o.replicas = __shfl_down_sync(0xffffffffu, c.replicas, d);
    o.batch = __shfl_down_sync(0xffffffffu, c.batch, d);
    o.acc = __shfl_down_sync(0xffffffffu, c.acc, d);
    o.itl = __shfl_down_sync(0xffffffffu, c.itl, d);
    o.ttft = __shfl_down_sync(0xffffffffu, c.ttft, d);
    o.rho = __shfl_down_sync(0xffffffffu, c.rho, d);
    o.max_rate = __shfl_down_sync(0xffffffffu, c.max_rate, d);
    o.feasible = __shfl_down_sync(0xffffffffu, c.feasible, d);
    return o;
}
__device__ __forceinline__ Cand cand_warp_min(Cand c) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        Cand o = cand_shfl_down(c, d);
        if (cand_better(o, c)) c = o;
    }
    return c;
}

// SoA columns of wva_allocs on the device.
struct AllocCols {
    uint8_t* feasible;
    int *acc, *replicas, *batch;
    float *cost, *value, *itl, *ttft, *rho, *max_rate;
};
__device__ __forceinline__ void store_cand(const AllocCols& o, size_t i, const Cand& c) {
    if (o.feasible) o.feasible[i] = (uint8_t)c.feasible;
    if (o.acc) o.acc[i] = c.acc;
    if (o.replicas) o.replicas[i] = c.replicas;
    if (o.batch) o.batch[i] = c.batch;
    if (o.cost) o.cost[i] = c.cost;
    if (o.value) o.value[i] = c.value;
    if (o.itl) o.itl[i] = c.itl;
    if (o.ttft) o.ttft[i] = c.ttft;
    if (o.rho) o.rho[i] = c.rho;
    if (o.max_rate) o.max_rate[i] = c.max_rate;
}
__device__ __forceinline__ Cand load_cand(const AllocCols& o, size_t i) {
    Cand c;
    c.feasible = o.feasible[i]; c.acc = o.acc[i]; c.replicas = o.replicas[i]; c.batch = o.batch[i];
    c.cost = o.cost[i]; c.value = o.value[i]; c.itl = o.itl[i]; c.ttft = o.ttft[i]; c.rho = o.rho[i];
    c.max_rate = o.max_rate[i];
    return c;
}

// ---------------------------------------------------------------------------
// Gates of CreateAllocation (allocation.go:42-75) + candidate rule (server.go:70-82).
// bit0: the pair can be analysed under load; bit1: zero-load candidate; 0: nil.
// ---------------------------------------------------------------------------
enum { PAIR_LOAD = 1, PAIR_ZERO = 2 };

__device__ __forceinline__ int pair_class(const DevFleet& f, int s, int a, bool honour_keep) {
    if (honour_keep && f.srv_keep_acc[s] && f.srv_cur_acc[s] != -1 && f.srv_cur_acc[s] != a) return 0;
    if (f.srv_arrival_rpm[s] < 0.0f || f.srv_in_tokens[s] < 0 || f.srv_out_tokens[s] < 0) return 0;
    const int m = f.srv_model[s];
    if (m < 0 || m >= f.M) return 0;
    if (!f.perf_present[m * f.A + a]) return 0;
    if (!f.srv_has_target[s]) return 0;
    if (f.srv_arrival_rpm[s] == 0.0f || f.srv_out_tokens[s] == 0) return PAIR_ZERO;
    return PAIR_LOAD;
}
__device__ __forceinline__ int num_instances(const DevFleet& f, int m, int a) {  // model.go:50-57
    const int c = f.perf_acc_count[m * f.A + a];
    return c <= 0 ? 1 : c;
}
__device__ __forceinline__ QParams qparams_of(const DevFleet& f, int s, int a) {
    const int k = f.srv_model[s] * f.A + a;
    QParams q;
    q.alpha = f.perf_alpha[k]; q.beta = f.perf_beta[k]; q.gamma = f.perf_gamma[k]; q.delta = f.perf_delta[k];
    q.in_tok = f.srv_in_tokens[s]; q.out_tok = f.srv_out_tokens[s];
    return q;
}
__device__ __forceinline__ float total_rate_of(const DevFleet& f, int s) {  // allocation.go:134-139
    if (f.srv_slo_tps[s] == 0.0f) return __fdiv_rn(f.srv_arrival_rpm[s], 60.0f);
    return __fdiv_rn(f.srv_slo_tps[s], (float)f.srv_out_tokens[s]);
}
__device__ __forceinline__ float penalty_of(const DevFleet& f, int s, const Cand& c) {
    return transition_penalty(f.penalty, f.srv_cur_acc[s], f.srv_cur_replicas[s], f.srv_cur_cost[s], c.acc,
                              c.replicas, c.cost);
}
// zeroLoadAllocation: allocation.go:259-288 (value = cost; caller applies the penalty)
__device__ __forceinline__ Cand zero_load_alloc(const DevFleet& f, int s, int a) {
    Cand c = cand_nil();
    c.feasible = 1;
    const long long nrep = f.srv_min_replicas[s];
    if (nrep == 0) return c;  // accelerator "", all zero
    const int m = f.srv_model[s], k = m * f.A + a;
    int max_batch = f.perf_max_batch[k];
    if (f.srv_max_batch[s] > 0) max_batch = f.srv_max_batch[s];
    const long long total = (long long)num_instances(f, m, a) * nrep;
    c.acc = a;
    c.replicas = (int)nrep;
    c.batch = max_batch;
    c.cost = __fmul_rn(f.acc_cost[a], (float)total);
    c.value = c.cost;
    c.itl = __fadd_rn(f.perf_alpha[k], f.perf_beta[k]);
    const float max_decode = __fadd_rn(f.perf_alpha[k], __fmul_rn(f.perf_beta[k], (float)max_batch));
    c.ttft = __fadd_rn(f.perf_gamma[k], f.perf_delta[k]);
    c.max_rate = __fdiv_rn((float)max_batch, __fadd_rn(c.ttft, max_decode));
    return c;
}

// ---------------------------------------------------------------------------
// Shared head tables: entry n (0-based) of table t = {servRate[n], yh, yl} as doubles + {min(servRate[n..]),
// max(servRate[0..n])} as floats (32 B, two 16 B loads per head step), plus a float column
// ls[n] = sum_{i<n} log2(servRate[i]) used only to ESTIMATE chain lengths for scheduling.
// ---------------------------------------------------------------------------
// Per (table, batch index) constants shared by the 64 replica levels of a pair:
// x = RateRange.Max (req/s) for N = batch, y = log2 servRate[N-1], z = ls[N-1], w = log2 servRate[0].
// Per (server, replica index): x = rate (req/s), y = lambda (req/ms), z = log2 lambda.
__global__ void __launch_bounds__(128) build_pair_tables(DevFleet f, const int* __restrict__ tab_pair,
                                                         const long long* __restrict__ tab_off,
                                                         const int* __restrict__ tab_len, int n_tab,
                                                         double* __restrict__ tab, float* __restrict__ ls,
                                                         const int* __restrict__ batch, int B,
                                                         float4* __restrict__ pb) {
    __shared__ double wsum[4];
    __shared__ double carry_s;
    const int t = blockIdx.x;
    if (t >= n_tab) return;
    const int pair = tab_pair[t];
    const int s = pair / f.A, a = pair % f.A;
    const QParams q = qparams_of(f, s, a);
    double* out = tab + 4 * tab_off[t];
    const int len = tab_len[t];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* l = ls ? ls + tab_off[t] + t : nullptr;  // len + 1 entries per table
    // forward sweep in tiles of 128: entries + exclusive prefix sum of log2(servRate)
    if (threadIdx.x == 0) carry_s = 0.0;
    __syncthreads();
    for (int base = 0; base < len; base += blockDim.x) {
        const int n = base + threadIdx.x;
        double lg = 0.0;
        if (n < len) {
            const float srf = serv_rate(q, n + 1);
            const double sr = (double)srf;
            const Recip r = make_recip(sr);
            out[4 * n + 0] = sr;
            out[4 * n + 1] = r.yh;
            out[4 * n + 2] = r.yl;
            lg = (double)log2f(srf);
        }
        double inc = lg;  // inclusive warp scan
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double o = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += o;
        }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        double off = carry_s;
        for (int w = 0; w < warp; ++w) off += wsum[w];
        if (l && n < len) l[n] = (float)(off + inc - lg);
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry_s = off + inc;
        __syncthreads();
    }
    if (l && threadIdx.x == 0) l[len] = (float)carry_s;
    // column 4 = {float suffix minimum, float prefix maximum} of servRate (exact: the rates are float32).
    // A NaN rate poisons the suffix minimum to 0 (early exit disabled) and the prefix maximum to +inf.
    __shared__ float wmin[4];
    __shared__ float carry_m;
    if (threadIdx.x == 0) carry_m = 3.402823466e38f;
    __syncthreads();
    for (int base = 0; base < len; base += blockDim.x) {  // backward: suffix minimum
        const int n = len - 1 - (base + threadIdx.x);     // thread 0 takes the last entry
        float v = n >= 0 ? (float)out[4 * n] : 3.402823466e38f;
        if (!(v == v)) v = 0.0f;
        float m = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const float o = __shfl_up_sync(0xffffffffu, m, d);
            if (lane >= d) m = fminf(m, o);
        }
        if (lane == 31) wmin[warp] = m;
        __syncthreads();
        float pre = carry_m;
        for (int w = 0; w < warp; ++w) pre = fminf(pre, wmin[w]);
        m = fminf(m, pre);
        if (n >= 0) ((float*)(out + 4 * n + 3))[0] = m;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry_m = m;
        __syncthreads();
    }
    if (threadIdx.x == 0) carry_m = 0.0f;
    __syncthreads();
    for (int base = 0; base < len; base += blockDim.x) {  // forward: prefix maximum
        const int n = base + threadIdx.x;
        float v = n < len ? (float)out[4 * n] : 0.0f;
        if (!(v == v)) v = 3.402823466e38f;
        float m = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const float o = __shfl_up_sync(0xffffffffu, m, d);
            if (lane >= d) m = fmaxf(m, o);
        }
        if (lane == 31) wmin[warp] = m;
        __syncthreads();
        float pre = carry_m;
        for (int w = 0; w < warp; ++w) pre = fmaxf(pre, wmin[w]);
        m = fmaxf(m, pre);
        if (n < len) ((float*)(out + 4 * n + 3))[1] = m;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry_m = m;
        __syncthreads();
    }
    if (pb) {
        const float l2s0 = log2f((float)out[0]);
        for (int bi = threadIdx.x; bi < B; bi += blockDim.x) {
            const int b = batch[bi];
            const float sN = (float)out[4 * (b - 1)];
            pb[(size_t)t * B + bi] = make_float4(rate_max_of(sN), log2f(sN), l[b - 1], l2s0);
        }
    }
}


// ---------------------------------------------------------------------------
// K2: candidate grid.
//
//   grid_rows        per (pair, replica level): the chain every large-enough batch size shares
//                    (solve_row); also the (server, replica) rate block and the batch-rank reset
//   grid_sort_local  per chunk of 8192 cells: gates + Analyze's rate checks; cells that share their
//                    row's chain are finished inline; the others get a log-domain length estimate,
//                    an 8-bit class and a local counting sort -> warp items; the last CTA plans
//                    grid_kernel's queues (grid_items_plan)
//   grid_items_scatter  items ordered globally, longest class first
//   grid_kernel      persistent CTA per SM; warps pull items (32 cells of nearly equal chain length)
//                    from a long and a short queue: streaming solve, metrics, SLO feasibility,
//                    per-cell columns, atomicMin of the smallest feasible batch rank per
//                    (server, accelerator, replica)
//   grid_fallback   stored-vector re-run of the rare cells the streaming solve bails on
//   grid_finalize   per-server argmin (warp shuffle -> shared memory -> winner record)
//
// For a fixed (server, accelerator, replica level) the transition penalty and the cost do
// not depend on the batch size, so the winner among batch sizes is the smallest feasible
// one; the per-server winner is then the best of the A*R survivors under the order
// value, cost, replicas, batch, accelerator.
// ---------------------------------------------------------------------------
struct CellCols {
    uint8_t* flags;  // bit0: Analyze ok, bit1: SLO-feasible
    float *ttft, *itl, *rho, *throughput;
};
constexpr int kSortChunk = 8192;   // cells per CTA in the local counting sort
constexpr int kSortThreads = 512;
constexpr int kGridStash = 24;     // chain states kept in shared memory between the two passes (per lane)
constexpr int kClasses = 256;      // 8-bit length classes; class 255 = not analysable
struct GridArgs {
    DevFleet f;
    const int* batch;        // [B]
    const int* batch_rank;   // [B] rank of batch[bi] in ascending (batch, bi) order
    const int* rank_to_bi;   // [B] inverse of batch_rank
    const int* replicas;     // [R]
    int B, R;
    const double* tab;       // shared head tables
    const float* ls;         // prefix log2 sums (estimate only)
    const long long* pair_tab_off;  // [S*A] entry offset of the pair's table (-1: none)
    const int* pair_tab_idx;        // [S*A] table index (for the ls / pb columns)
    const float4* pb;               // [n_tab * B] per (table, batch): rmax, log2 sN, ls[N-1], log2 s0
    float4* rt;               // [S * R] per (server, replica): rate, lambda, log2 lambda
    double* row_acc;                // [S*A*R] shared-chain results per (server, accelerator, replica)
    double* row_sump;
    int* row_j;                     // last state of the shared chain (INT_MAX: no sharing)
    uint8_t* row_res;               // 1: grid_rows resolved the row's shared cells into best_rank (§3.2b)
    int row_resolve;                // 0: row resolution off (WVA_GRID_ROWRES=0)
    int Bmax;                       // table length
    long long n_cells;
    unsigned* order;         // [n_cells] cell ids, sorted by length class inside each chunk of kSortChunk cells
    unsigned long long* items;         // warp work items (start | count << 32 | class << 40), unsorted
    unsigned long long* items_sorted;  // the same, longest class first
    unsigned* item_count;    // [0] number of items, [1..256] items per class, [257..512] class cursors
    int* best_rank;          // [S*A*R] smallest feasible batch rank (INT_MAX: none)
    CellCols cells;          // internal per-cell columns (ttft, itl, rho always present)
    float4* pair_rec;        // [S*A][3] per pair: {alpha, beta, gamma, delta}, {in_tok, out_tok (int bits), slo_ttft, slo_itl},
                             // {min_replicas, tps flag (int bits), 0, 0} -- one 48-byte record instead of ten scattered loads
    uint4* recs;             // [items][32] per sorted cell: {cell, lambda bits, table entry offset, batch size | class << 23 | pad << 31}
    int want_cells;          // 0: the caller did not ask for the cell table -> cells that share their row's chain store
                             // nothing (grid_finalize recomputes the few winners among them); 1: every cell is stored
    int* fb_count;           // cells that need the stored-vector fallback
    long long* fb_cells;
    int fb_cap;
    int long_per_sm;         // grid_kernel: long items per sub-partition 0 (< 0: chosen per launch by grid_items_plan)
    int n_ctas;              // CTAs of grid_kernel (= SMs)
    int long_share;          // ... and how many other warps of that sub-partition may pull short items meanwhile
    int long_cls;            // items of class <= long_cls are "long" ...
    unsigned long_cap;       // ... up to this many (long_per_sm x CTAs)
    unsigned* dbg_cycles;    // diagnostics: per order index, SM cycles spent in grid_kernel (or NULL)
    size_t dbg_n;            // cells; dbg_cycles[dbg_n + idx] holds the warp timeline (start ns, SM, end ns)
};

__device__ __forceinline__ void decode_cell(const GridArgs& g, long long cell, int& s, int& a, int& bi, int& ri) {
    unsigned t = (unsigned)cell;  // n_cells < 2^32 (checked on the host): 32-bit divisions
    const unsigned R = (unsigned)g.R, B = (unsigned)g.B, A = (unsigned)g.f.A;
    unsigned q = t / R;
    ri = (int)(t - q * R);
    t = q;
    q = t / B;
    bi = (int)(t - q * B);
    t = q;
    q = t / A;
    a = (int)(t - q * A);
    s = (int)q;
}

// Estimated number of chain states before exact early termination (scheduling only; any
// value is correct, a good one makes the 32 lanes of a warp finish together).
__device__ __forceinline__ float estimate_len(const double* /*tab*/, const float* ls, int N, int K, float /*lambda*/,
                                              float l2lam, float l2s0, float l2sN, float lsNm1) {
    const float thr = -78.0f + fminf(0.0f, l2lam - l2s0);
    const float d = l2sN - l2lam;                     // tail decay per state (> 0 when analysable)
    const float L0 = (float)(N - 1) * l2lam - lsNm1;  // log2 p[N-1]
    float est;
    if (L0 >= thr || N == 1) {
        est = (float)(N - 1) + (L0 - thr) / fmaxf(d, 1e-9f) + 2.0f;
    } else {
        // the chain dies inside the head.  log2 p[j] = j*l2lam - ls[j] rises from 0 to the mode and
        // falls afterwards, and thr < 0, so {j : log2 p[j] < thr} is an upper set: one binary search
        int lo = 1, hi = N - 1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if ((float)mid * l2lam - ls[mid] < thr) hi = mid; else lo = mid + 1;
        }
        est = (float)lo + 2.0f;
    }
    return fminf(fmaxf(est, 2.0f), (float)K);
}
__device__ __forceinline__ int length_class(float est) {  // 0 = longest ... 254 = shortest
    const int c = (int)(log2f(est) * 12.0f);  // ~6 % wide classes
    return 254 - min(max(c, 0), 254);
}

// Warp-aggregated shared-memory counter: returns this lane's slot among the lanes that
// increment the same counter (one atomic per distinct counter per warp).
__device__ __forceinline__ unsigned agg_inc(unsigned* counters, int key) {
    const unsigned peers = __match_any_sync(__activemask(), key);
    const int leader = __ffs(peers) - 1;
    const int lane = threadIdx.x & 31;
    unsigned base = 0;
    if (lane == leader) base = atomicAdd(&counters[key], (unsigned)__popc(peers));
    base = __shfl_sync(peers, base, leader);
    return base + __popc(peers & ((1u << lane) - 1u));
}

// SLO feasibility of an analysed cell (the build's grid semantics, SURVEY.md §8d).  The per-server
// targets and the stability limit of the (pair, batch) are row constants; rate/1000 is the cell's lambda.
struct FeasRow {
    float slo_ttft, slo_itl, lim;  // lim = RateRange.Max/1000 * (1 - 0.1): Size's stability margin (queueanalyzer.go:231-234)
    int min_replicas;
    bool tps;
};
__device__ __forceinline__ float feas_lim(float rmax) { return __fmul_rn(__fdiv_rn(rmax, 1000.0f), __fsub_rn(1.0f, 0.1f)); }
__device__ __forceinline__ FeasRow feas_row(const DevFleet& f, int s, float rmax) {
    FeasRow fr;
    fr.slo_ttft = f.srv_slo_ttft[s];
    fr.slo_itl = f.srv_slo_itl[s];
    fr.min_replicas = f.srv_min_replicas[s];
    fr.tps = f.srv_slo_tps[s] > 0.0f;
    fr.lim = feas_lim(rmax);
    return fr;
}
__device__ __forceinline__ bool cell_feasible(const FeasRow& fr, int r, float lambda, const Metrics& m) {
    bool feas = (fr.slo_ttft == 0.0f || m.ttft <= fr.slo_ttft) && (fr.slo_itl == 0.0f || m.avg_token_time <= fr.slo_itl) &&
                (r >= fr.min_replicas);
    if (fr.tps) feas = feas && (lambda <= fr.lim);
    return feas;
}
// Analyze's rate checks for a cell of a pair that has a table (queueanalyzer.go:135-143): a positive rate inside the
// stability range of the batch size (rmax = RateRange.Max), and a queue of at least two states (K = b + b * ratio).
__device__ __forceinline__ bool cell_analysable(float rate, float rmax, int K) {
    return !(rate <= 0.0f) && !(rate > rmax) && K >= 2;
}
// The cell's chain is its row's shared chain (§3.2a): the row has one (jl != INT_MAX) and the batch size is past it.
__device__ __forceinline__ bool cell_shared(int jl, int b, int K) {
    return jl != INT_MAX && b >= jl + 2 && K < (1 << 23);
}
__device__ __forceinline__ void store_cell(const GridArgs& g, long long cell, int ok, int feas, const Metrics& m) {
    g.cells.flags[cell] = (uint8_t)(ok | (feas << 1));
    g.cells.ttft[cell] = m.ttft;
    g.cells.itl[cell] = m.avg_token_time;
    g.cells.rho[cell] = m.rho;
    if (g.cells.throughput) g.cells.throughput[cell] = m.throughput;
}

// A cell that shares its row's chain (grid_sort_local): stats_from_row + metrics_from with everything that does
// not depend on the batch size hoisted — per pair (PairConst: the operands of EffectiveConcurrency, PrefillTime,
// DecodeTime), per (pair, replica level) (resp = avgNumInSystem / throughput, 1 - sumP).  Same operations in the
// same order on the same operands as the unhoisted functions, hence the same bits.
struct PairConst {
    float gamma, d_in, alpha, beta, ec_base, ec_den;
    int in_zero;
};
__device__ __forceinline__ PairConst pair_const(const QParams& q) {
    PairConst pc;
    const float tokens = (float)(q.out_tok - 1);                    // queueanalyzer.go:296-302
    pc.gamma = q.gamma;
    pc.alpha = q.alpha;
    pc.beta = q.beta;
    pc.d_in = __fmul_rn(q.delta, (float)q.in_tok);                  // delta * inTokens (:258, :300)
    pc.ec_base = __fadd_rn(q.gamma, __fmul_rn(q.alpha, tokens));
    pc.ec_den = __fadd_rn(pc.d_in, __fmul_rn(q.beta, tokens));
    pc.in_zero = q.in_tok == 0;
    return pc;
}
// resp: (float)acc / throughput with throughput = lambda * (1 - 0) = lambda
__device__ __forceinline__ float row_resp_time(double acc, float lambda) {
    return __fdiv_rn((float)acc, __fmul_rn(lambda, __fsub_rn(1.0f, 0.0f)));
}
__device__ __forceinline__ Metrics shared_cell_metrics(const PairConst& pc, double acc, double one_m_sump, float resp,
                                                       float lambda, int N) {
    const double in_serv = __dadd_rn(acc, __dmul_rn(one_m_sump, (double)N));  // mm1modelstatedependent.go:53
    const float in_serv_f = (float)in_serv;
    const float thr = __fmul_rn(lambda, __fsub_rn(1.0f, 0.0f));
    const float serv = __fdiv_rn(in_serv_f, thr);
    float w = __fsub_rn(resp, serv);
    if (w < 0.0f) w = 0.0f;
    const float fN = (float)N;
    const float eff = go_minf(go_maxf(__fdiv_rn(__fsub_rn(serv, pc.ec_base), pc.ec_den), 0.0f), fN);
    Metrics m;
    m.avg_prefill_time = pc.in_zero ? 0.0f : __fadd_rn(pc.gamma, __fmul_rn(pc.d_in, eff));
    m.avg_token_time = __fadd_rn(pc.alpha, __fmul_rn(pc.beta, eff));
    m.rho = go_minf(go_maxf(__fdiv_rn(in_serv_f, fN), 0.0f), 1.0f);
    m.throughput = __fmul_rn(thr, 1000.0f);
    m.avg_wait_time = w;
    m.ttft = __fadd_rn(w, m.avg_prefill_time);
    return m;
}

// The same evaluation when (float)avgNumInServers does not depend on the batch size.  avgNumInServers =
// acc + (1 - sumP) * N in float64, and 1 - sumP is a few ulps of 1 at most (the chain died before state N), so
// for all N <= Nmax the float64 value stays inside the float32 rounding interval of acc unless acc sits within
// ~1e-13 relative of an interval edge.  row_invariant() proves it for a (pair, replica level) with an exact bound:
// lo_b, hi_b = the float32 rounding boundaries around acc (exact in float64); |in_serv - acc| <= |m| N (1 + 2^-52)
// + acc 2^-53, and both distances are exact differences (Sterbenz), so d > 2 RN(|m| Nmax) + acc 2^-50 implies
// lo_b < in_serv < hi_b, i.e. (float)in_serv == (float)acc for every batch size of the grid.  Then the service
// time, the waiting time and the unclamped effective concurrency are constants of the row and a cell costs a
// min, two multiply-adds and the SLO comparisons.  Rows that fail the test take shared_cell_metrics.
struct RowInv {
    float f0, w0, effu;  // (float)avgNumInServers, waiting time, max(effective concurrency, 0) before the clamp at N
};
__device__ __forceinline__ bool row_invariant(const PairConst& pc, double acc, double one_m_sump, float resp, float lambda,
                                              int Nmax, RowInv& ri) {
    const float f0 = (float)acc;
    if (!(f0 > 1e-30f && f0 < 1e30f)) return false;
    const float up = __uint_as_float(__float_as_uint(f0) + 1u), dn = __uint_as_float(__float_as_uint(f0) - 1u);
    const double hi_b = 0.5 * ((double)f0 + (double)up), lo_b = 0.5 * ((double)dn + (double)f0);
    const double d = fmin(hi_b - acc, acc - lo_b);
    const double tb = __dmul_rn(fabs(one_m_sump), (double)Nmax);
    if (!(d > __dadd_rn(__dmul_rn(2.0, tb), __dmul_rn(acc, 0x1p-50)))) return false;
    const float thr = __fmul_rn(lambda, __fsub_rn(1.0f, 0.0f));
    const float serv = __fdiv_rn(f0, thr);
    float w = __fsub_rn(resp, serv);
    if (w < 0.0f) w = 0.0f;
    ri.f0 = f0;
    ri.w0 = w;
    ri.effu = go_maxf(__fdiv_rn(__fsub_rn(serv, pc.ec_base), pc.ec_den), 0.0f);
    return true;
}
__device__ __forceinline__ Metrics shared_cell_metrics_inv(const PairConst& pc, const RowInv& ri, float lambda, int N,
                                                           bool want_rho) {
    const float fN = (float)N;
    const float eff = go_minf(ri.effu, fN);
    Metrics m;
    m.avg_prefill_time = pc.in_zero ? 0.0f : __fadd_rn(pc.gamma, __fmul_rn(pc.d_in, eff));
    m.avg_token_time = __fadd_rn(pc.alpha, __fmul_rn(pc.beta, eff));
    m.rho = want_rho ? go_minf(go_maxf(__fdiv_rn(ri.f0, fN), 0.0f), 1.0f) : 0.0f;
    m.throughput = __fmul_rn(__fmul_rn(lambda, __fsub_rn(1.0f, 0.0f)), 1000.0f);
    m.avg_wait_time = ri.w0;
    m.ttft = __fadd_rn(ri.w0, m.avg_prefill_time);
    return m;
}

// Row resolution (DESIGN §3.2b).  On an invariant row a shared cell depends on its batch size N only through
// eff = min(effu, N), which does not decrease as N grows.  With the operands below finite, beta >= 0 and d_in >= 0 (or
// no input tokens), itl = RN(alpha + RN(beta eff)) and ttft = RN(w0 + RN(gamma + RN(d_in eff))) do not decrease either
// (RN is monotone), so the SLO part of cell_feasible holds for a prefix of the batch sizes.  Everything else a shared
// cell's feasibility depends on is a function of the batch size alone (row_gate).  Hence the smallest feasible shared
// rank of the row is the first rank that passes row_gate if the SLO test holds there, and there is none otherwise.
__device__ __forceinline__ bool row_monotone(const PairConst& pc, const RowInv& ri) {
    const bool prefill = pc.in_zero || (isfinite(pc.d_in) && pc.d_in >= 0.0f);
    return isfinite(pc.alpha) && isfinite(pc.beta) && pc.beta >= 0.0f && isfinite(pc.gamma) && prefill &&
           isfinite(ri.w0) && isfinite(ri.effu);
}
// The conditions under which a cell of the row is analysed as a shared cell, plus the TPS stability limit of its
// feasibility: the parts that depend on the batch size and not on the chain.
__device__ __forceinline__ bool row_gate(float rate, float lambda, bool tps, float rmax, int jl, int b, int K) {
    return cell_analysable(rate, rmax, K) && cell_shared(jl, b, K) && (!tps || lambda <= feas_lim(rmax));
}

// One CTA per (server, accelerator) pair, one lane per replica level: the chain every large-enough
// batch size shares.  The pair's table is staged in shared memory first (coalesced), so the serial
// chains read it at shared-memory latency instead of waiting for L2 on every step.
constexpr int kRowsSmemEntries = 1536;  // 48 KB of 32-byte entries; longer tables are read from global

// The smallest feasible batch rank among the shared cells of a row that row_monotone admits (INT_MAX: none), t = the
// pair's table index.  A row whose cells all fail row_gate scans every rank, so the loads go four ranks at a time.
__device__ __forceinline__ int resolve_row(const GridArgs& g, int t, float rate, float lambda, FeasRow fr, int rep,
                                           const PairConst& pc, const RowInv& inv, int jl) {
    const int B = g.B;
    int lo = 0, hi = B;  // first rank with a batch size past the shared chain (ranks ascend with the batch size)
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (g.batch[g.rank_to_bi[mid]] >= jl + 2) hi = mid; else lo = mid + 1;
    }
    const float* rmax = (const float*)(g.pb + (size_t)t * B);  // component x of the (table, batch) constants
    for (int r0 = lo; r0 < B; r0 += 4) {
        int bi[4], b[4];
        float rm[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) bi[u] = g.rank_to_bi[min(r0 + u, B - 1)];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            b[u] = g.batch[bi[u]];
            rm[u] = rmax[4 * bi[u]];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int K = b[u] + b[u] * g.f.ratio;
            if (r0 + u < B && row_gate(rate, lambda, fr.tps, rm[u], jl, b[u], K)) {
                fr.lim = feas_lim(rm[u]);
                const Metrics m = shared_cell_metrics_inv(pc, inv, lambda, b[u], false);
                return cell_feasible(fr, rep, lambda, m) ? r0 + u : INT_MAX;
            }
        }
    }
    return INT_MAX;
}

__global__ void __launch_bounds__(128) grid_rows(GridArgs g) {
    extern __shared__ double rows_tab[];
    const DevFleet& f = g.f;
    const int sa = blockIdx.x;
    const int s = sa / f.A;
    const long long toff = g.pair_tab_off[sa];
    const double* tab = toff >= 0 ? g.tab + 4 * toff : nullptr;
    const bool staged = toff >= 0 && g.Bmax <= kRowsSmemEntries;
    if (staged) {
        // all of a thread's loads first, then its stores: one L2 round trip instead of one per iteration
        const double2* src = (const double2*)tab;
        double2* dst = (double2*)rows_tab;
        const int n16 = 2 * g.Bmax;
        for (int i0 = threadIdx.x; i0 < n16; i0 += 8 * blockDim.x) {
            double2 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * blockDim.x;
                if (i < n16) v[u] = src[i];
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * blockDim.x;
                if (i < n16) dst[i] = v[u];
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // the pair's constants as one record (grid_kernel reads it once per item)
        const int a = sa - s * f.A;
        const int m = f.srv_model[s];
        float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m >= 0 && m < f.M) {
            const int k = m * f.A + a;
            r0 = make_float4(f.perf_alpha[k], f.perf_beta[k], f.perf_gamma[k], f.perf_delta[k]);
        }
        g.pair_rec[3 * sa + 0] = r0;
        g.pair_rec[3 * sa + 1] = make_float4(__int_as_float(f.srv_in_tokens[s]), __int_as_float(f.srv_out_tokens[s]),
                                             f.srv_slo_ttft[s], f.srv_slo_itl[s]);
        g.pair_rec[3 * sa + 2] = make_float4(__int_as_float(f.srv_min_replicas[s]),
                                             __int_as_float(f.srv_slo_tps[s] > 0.0f ? 1 : 0), 0.f, 0.f);
    }
    float l2s0 = 0.f, ls_end = 0.f;
    if (toff >= 0) {
        l2s0 = log2f((float)tab[0]);
        ls_end = (g.ls + toff + g.pair_tab_idx[sa])[g.Bmax - 1];
    }
    // row resolution (§3.2b) only when the caller does not want the cell table: grid_sort_local then never visits the
    // shared cells of a resolved row
    const bool resolve = toff >= 0 && g.row_resolve && !g.want_cells;
    PairConst pc{};
    FeasRow fr{};
    if (resolve) {
        pc = pair_const(qparams_of(f, s, sa - s * f.A));
        fr = feas_row(f, s, 0.0f);
    }
    for (int ri = threadIdx.x; ri < g.R; ri += blockDim.x) {
        const size_t row = (size_t)sa * g.R + ri;
        int j = INT_MAX;
        double acc = 0.0, sump = 0.0;
        // per-replica rate, lambda and log2(lambda) of the server (rate = total / replicas, lambda = rate / 1000): every pair CTA
        // derives its own copy, the CTA of accelerator 0 publishes it for the later kernels; the
        // (pair, replica) slot of the batch-rank minimum is reset here too (or set to the resolved row's minimum)
        const float rate = __fdiv_rn(total_rate_of(f, s), (float)g.replicas[ri]);
        const float lambda = __fdiv_rn(rate, 1000.0f);
        const float4 rt = make_float4(rate, lambda, log2f(lambda), 0.0f);
        if (sa == s * f.A) g.rt[s * g.R + ri] = rt;
        if (toff >= 0 && rt.x > 0.0f) {
            // skip rows whose chain is (by the log-domain estimate) still far from negligible at the end of
            // the table: they cannot be shared and would only burn Bmax steps to find that out
            const float thr = -78.0f + fminf(0.0f, rt.z - l2s0);
            const float Lend = (float)(g.Bmax - 1) * rt.z - ls_end;
            int jl = 0;
            if (Lend < thr + 8.0f) {
                const bool ok = staged ? solve_row(rows_tab, g.Bmax, rt.y, acc, sump, jl) : solve_row(tab, g.Bmax, rt.y, acc, sump, jl);
                if (ok) j = jl;
            }
        }
        int best = INT_MAX;
        uint8_t res = 0;
        if (resolve && j != INT_MAX) {
            RowInv inv;
            if (row_invariant(pc, acc, __dsub_rn(1.0, sump), row_resp_time(acc, lambda), lambda, g.Bmax, inv) &&
                row_monotone(pc, inv)) {
                res = 1;
                best = resolve_row(g, g.pair_tab_idx[sa], rt.x, lambda, fr, g.replicas[ri], pc, inv, j);
            }
        }
        g.best_rank[row] = best;
        g.row_res[row] = res;
        g.row_j[row] = j;
        g.row_acc[row] = acc;
        g.row_sump[row] = sump;
    }
}

// Counter increment for lanes whose equal keys sit in CONTIGUOUS lane ranges (along a row the
// length class is monotone in the replica level, so equal classes are adjacent): one atomic per
// run instead of one per lane, found with a shuffle and a ballot.  Returns the lane's slot.
__device__ __forceinline__ unsigned seg_inc(unsigned* counters, int key) {
    const unsigned act = __activemask();
    const int lane = threadIdx.x & 31;
    const int prev = __shfl_up_sync(act, key, 1);
    const bool prev_active = lane > 0 && ((act >> (lane - 1)) & 1u);
    const unsigned heads = __ballot_sync(act, !prev_active || prev != key);
    const unsigned upto = (lane == 31) ? 0xffffffffu : ((2u << lane) - 1u);
    const int seg_start = 31 - __clz(heads & upto);
    const unsigned above = heads & ~upto;
    const int seg_end = above ? (__ffs(above) - 1) : 32;  // exclusive; inactive lanes start a new run too
    const unsigned seg_mask = (seg_end == 32 ? 0xffffffffu : ((1u << seg_end) - 1u)) & ~((1u << seg_start) - 1u) & act;
    unsigned base = 0;
    if (lane == seg_start) base = atomicAdd(&counters[key], (unsigned)__popc(seg_mask));
    base = __shfl_sync(act, base, seg_start);
    return base + __popc(seg_mask & ((1u << lane) - 1u));
}

// Estimate + LOCAL counting sort, one CTA per chunk of kSortChunk consecutive cells (cells of
// one or two (server, accelerator) pairs): length classes are computed into shared memory,
// histogrammed, scanned and scattered without leaving the CTA.  Each run of 32 sorted cells
// becomes one warp work item tagged with its (longest) class; grid_sort_items then orders the
// items globally, so the launch is longest-first while a pair's cells stay adjacent.
__device__ __forceinline__ void grid_items_plan(const GridArgs& g);
__global__ void __launch_bounds__(kSortThreads, 2) grid_sort_local(GridArgs g) {
    __shared__ __align__(16) uint8_t keys[kSortChunk];
    __shared__ uint8_t sorted_keys[kSortChunk];
    __shared__ unsigned hist[kClasses];
    __shared__ unsigned cursor[kClasses];
    __shared__ unsigned item_base;
    const DevFleet& f = g.f;
    if (threadIdx.x < kClasses) hist[threadIdx.x] = 0;
    // every key starts as class 255 (not analysable, or finished here): the walk stores only the other classes
    static_assert(kSortChunk == 16 * kSortThreads, "one 16-byte store per thread fills the keys");
    reinterpret_cast<uint4*>(keys)[threadIdx.x] = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    __syncthreads();
    const long long base = (long long)blockIdx.x * kSortChunk;
    const int n_here = (int)min((long long)kSortChunk, g.n_cells - base);
    // walk the chunk row by row (a row = the R replica levels of one (server, accelerator, batch)):
    // the row's constants are decoded once per warp, lanes take the replica levels
    {
        const unsigned R = (unsigned)g.R, B = (unsigned)g.B, A = (unsigned)f.A;
        const unsigned row0 = (unsigned)(base / R), row1 = (unsigned)((base + n_here - 1) / R);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        // feasible shared cells lower best_rank[(pair, replica level)]: a lane meets the same replica
        // levels row after row, so it keeps the running minimum of its first two levels in registers
        // and issues one atomic per pair instead of one per cell
        unsigned cur_sa = 0xffffffffu;
        int best0 = INT_MAX, best1 = INT_MAX;
        auto flush_best = [&]() {
            if (best0 != INT_MAX) atomicMin(&g.best_rank[(size_t)cur_sa * R + lane], best0);
            if (best1 != INT_MAX) atomicMin(&g.best_rank[(size_t)cur_sa * R + lane + 32], best1);
            best0 = best1 = INT_MAX;
        };
        // pair-level constants are re-read only when the walk crosses into the next pair; so are the
        // lane's own row constants (its first two replica levels: rate, lambda, the row's shared chain)
        // what a lane knows about the shared cells of its row: evaluated per cell (general or invariant form), or
        // already resolved into best_rank by grid_rows (§3.2b)
        enum : uint8_t { kRowCells = 0, kRowInv = 1, kRowResolved = 2 };
        struct LaneRow {
            float4 rt;
            // shared-chain results of the row.  kRowCells: a = sum(i p[i]), b = 1 - sumP, r = resp (avgNumInSystem /
            // throughput).  kRowInv (row_invariant holds): the three floats of RowInv ride in the same registers
            // (a = {f0, w0}, r = effu), so the hot loop carries no more state than before.  kRowResolved: unused.
            double a, b;
            float r;
            int jl, rep;
            uint8_t kind;
        };
        LaneRow c0{}, c1{};
        unsigned sa = (row0 + warp) / B;
        int bi = (int)(row0 + warp - sa * B);
        int s = 0, t = 0;
        long long toff = -1;
        PairConst pc{};
        FeasRow fr{};
        auto load_lane = [&](unsigned ri, LaneRow& c) {
            if (ri >= R || toff < 0) return;
            const size_t rowid = (size_t)sa * R + ri;
            c.rt = g.rt[(unsigned)s * R + ri];
            c.jl = g.row_j[rowid];
            c.kind = g.row_res[rowid] ? kRowResolved : kRowCells;
            if (c.kind == kRowResolved) return;
            c.a = g.row_acc[rowid];
            c.b = __dsub_rn(1.0, g.row_sump[rowid]);
            c.r = row_resp_time(c.a, c.rt.y);
            c.rep = g.replicas[ri];
            RowInv inv;
            if (c.jl != INT_MAX && row_invariant(pc, c.a, c.b, c.r, c.rt.y, g.Bmax, inv)) {
                c.kind = kRowInv;
                c.a = __hiloint2double(__float_as_int(inv.w0), __float_as_int(inv.f0));
                c.r = inv.effu;
            }
        };
        for (unsigned row = row0 + warp; row <= row1; row += kSortThreads / 32, bi += kSortThreads / 32) {
            while (bi >= (int)B) {
                bi -= (int)B;
                ++sa;
            }
            if (sa != cur_sa) {
                flush_best();
                cur_sa = sa;
                s = (int)(sa / A);
                toff = g.pair_tab_off[sa];
                if (toff >= 0) {
                    t = g.pair_tab_idx[sa];
                    pc = pair_const(qparams_of(f, s, (int)(sa - (unsigned)s * A)));
                }
                fr = feas_row(f, s, 0.0f);
                load_lane(lane, c0);
                load_lane(lane + 32, c1);
            }
            const int b = g.batch[bi];
            const int K = b + b * f.ratio;
            // a cell that is key 255 without any work: outside the chunk, no table, or one that would share the chain
            // of a resolved row (then it is either shared and already in best_rank, or not analysable)
            auto idle = [&](unsigned ri, const LaneRow& c) {
                const long long cell = (long long)row * R + ri;
                return ri >= R || cell < base || cell >= base + n_here || toff < 0 ||
                       (c.kind == kRowResolved && cell_shared(c.jl, b, K));
            };
            if (R <= 64 && __all_sync(0xffffffffu, idle(lane, c0) && idle(lane + 32, c1))) continue;
            float4 pb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (toff >= 0) pb = g.pb[(size_t)t * g.B + bi];
            if (fr.tps) fr.lim = feas_lim(pb.x);
            const int rank = g.batch_rank[bi];
            // one cell: (row, ri) with the lane's cached row constants
            auto do_cell = [&](unsigned ri, const LaneRow& c, int slot) {
                if (idle(ri, c)) return;
                int key = 255;
                if (cell_analysable(c.rt.x, pb.x, K)) {  // Analyze: queueanalyzer.go:135-143
                    if (cell_shared(c.jl, b, K)) {
                        // the whole solve is shared with the row: only the N-dependent tail is per cell
                        const long long cell = (long long)row * R + ri;
                        Metrics m;
                        if (c.kind == kRowInv) {
                            RowInv inv;
                            inv.f0 = __int_as_float(__double2loint(c.a));
                            inv.w0 = __int_as_float(__double2hiint(c.a));
                            inv.effu = c.r;
                            m = shared_cell_metrics_inv(pc, inv, c.rt.y, b, g.want_cells != 0);
                        } else {
                            m = shared_cell_metrics(pc, c.a, c.b, c.r, c.rt.y, b);
                        }
                        const bool feas = cell_feasible(fr, c.rep, c.rt.y, m);
                        if (g.want_cells) store_cell(g, cell, 1, feas ? 1 : 0, m);
                        if (feas) {
                            if (slot == 0) best0 = min(best0, rank);
                            else if (slot == 1) best1 = min(best1, rank);
                            else atomicMin(&g.best_rank[(size_t)sa * R + ri], rank);
                        }
                    } else {
                        key = length_class(estimate_len(g.tab + 4 * toff, g.ls + toff + t, b, K, c.rt.y, c.rt.z, pb.w, pb.y, pb.z));
                    }
                }
                if (key != 255) {  // class 255 (finished here / not analysable) needs no slot and keeps its key
                    keys[(long long)row * R + ri - base] = (uint8_t)key;
                    seg_inc(hist, key);
                }
                // (the cell table, when requested, is cleared by the host before the launch: cells that are never
                // analysed read back as 0 without a store per cell here)
            };
            if ((unsigned)lane < R) do_cell(lane, c0, 0);
            if ((unsigned)lane + 32 < R) do_cell(lane + 32, c1, 1);
            for (unsigned ri = lane + 64; ri < R; ri += 32) {
                LaneRow c;
                load_lane(ri, c);
                do_cell(ri, c, 2);
            }
        }
        flush_best();
    }
    __syncthreads();
    if (threadIdx.x < 32) {  // exclusive scan of the 256 class counts by one warp
        unsigned run = 0;
        for (int c0 = 0; c0 < kClasses; c0 += 32) {
            const unsigned v = hist[c0 + threadIdx.x];
            unsigned inc = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned o = __shfl_up_sync(0xffffffffu, inc, d);
                if ((int)threadIdx.x >= d) inc += o;
            }
            cursor[c0 + threadIdx.x] = run + inc - v;
            run += __shfl_sync(0xffffffffu, inc, 31);
        }
    }
    __syncthreads();
    const int n_active = (int)cursor[255];  // class 255 (not analysable) sorts last
    for (int k = threadIdx.x; k < n_here; k += kSortThreads) {
        const int key = keys[k];
        if (key == 255) continue;
        const unsigned pos = seg_inc(cursor, key);
        g.order[base + pos] = (unsigned)(base + k);
        sorted_keys[pos] = (uint8_t)key;
    }
    const int n_items = (n_active + 31) >> 5;
    if (threadIdx.x == 0) item_base = n_items ? atomicAdd(g.item_count, (unsigned)n_items) : 0u;
    __syncthreads();
    for (int w = threadIdx.x; w < n_items; w += kSortThreads) {
        const unsigned start = (unsigned)(base + 32 * w);
        const unsigned cnt = (unsigned)min(32, n_active - 32 * w);
        const int cls = sorted_keys[32 * w];
        g.items[item_base + w] = (unsigned long long)start | ((unsigned long long)cnt << 32) |
                                 ((unsigned long long)cls << 40);
        agg_inc(g.item_count + 1, cls);  // global items-per-class histogram (warp-aggregated)
    }
    // the last CTA to get here turns the global histogram into class cursors and plans grid_kernel's queues
    // (one launch less than a separate single-CTA kernel)
    __shared__ bool last_cta;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last_cta = atomicAdd(g.item_count + 2 * kClasses + 6, 1u) == gridDim.x - 1;
    __syncthreads();
    if (last_cta) {
        __threadfence();
        grid_items_plan(g);
    }
}

// Global order of the warp items by class (longest first): class cursors from the global
// histogram, then a multi-CTA scatter with warp-aggregated atomics.
// grid_kernel's CTA shape (the kernel is further down; grid_items_plan plans its queues)
#ifndef WVA_GK_WARPS
#define WVA_GK_WARPS 16
#endif
constexpr int kGkWarps = WVA_GK_WARPS;    // 4 per sub-partition; 128 registers per thread keep the two FP64 chains of pass 2 apart
constexpr int kGkThreads = kGkWarps * 32;
constexpr int kGkTabWin = 32;  // table entries staged per warp (solve_shared_t STAGED)
constexpr int kGkLong = -1;    // long-item warps per CTA: automatic     // long-item warps per SM (sub-partition 0)
// Model of grid_kernel's launch time, calibrated on BASELINE config 2 with seeds 42..49 (tools/seed_times.py
// prints the plan next to the measured time): class c holds chains of 2^((254-c)/12) states;
//   item_us  what an item costs the short queue: ~0.099 us per state (two passes, ~96 cycles per state
//            and pass next to three other warps of the sub-partition, stalls included) + 7 us fixed;
//   long_us  an item that has its sub-partition to itself: 0.0564 us per state + 4 us.
__device__ __forceinline__ float class_len(int c) { return exp2f((float)(254 - c) * (1.0f / 12.0f)); }
__device__ __forceinline__ float item_us(int c) { return 0.0987f * class_len(c) + 7.0f; }
__device__ __forceinline__ float long_us(int c) { return 0.0564f * class_len(c) + 4.0f; }
// Runs in ONE CTA of at least kClasses threads (the last CTA of grid_sort_local to finish); threads beyond
// kClasses only take part in the barriers.
__device__ __forceinline__ void grid_items_plan(const GridArgs& g) {
    __shared__ unsigned cnt[kClasses + 1];  // exclusive prefix of the class counts (cnt[kClasses] = all items)
    __shared__ float wrk[kClasses + 1];     // exclusive prefix of the classes' work (warp-microseconds)
    __shared__ unsigned s_cnt[kClasses];
    __shared__ float s_wrk[kClasses];
    const int c = threadIdx.x;
    const bool on = c < kClasses;
    const unsigned mine = on ? __ldcg(g.item_count + 1 + c) : 0u;  // other CTAs' atomics: read at L2
    if (on) {
        s_cnt[c] = mine;
        s_wrk[c] = c < 255 ? (float)mine * item_us(c) : 0.0f;
    }
    __syncthreads();
    for (int d = 1; d < kClasses; d <<= 1) {  // inclusive Hillis-Steele scans
        const unsigned a = (on && c >= d) ? s_cnt[c - d] : 0u;
        const float w = (on && c >= d) ? s_wrk[c - d] : 0.0f;
        __syncthreads();
        if (on) {
            s_cnt[c] += a;
            s_wrk[c] += w;
        }
        __syncthreads();
    }
    if (on) {
        cnt[c + 1] = s_cnt[c];
        wrk[c + 1] = s_wrk[c];
        g.item_count[1 + kClasses + c] = s_cnt[c] - mine;  // class cursors for grid_items_scatter
    }
    if (c == 0) {
        cnt[0] = 0;
        wrk[0] = 0.0f;
    }
    __syncthreads();
    // grid_kernel's queues: the long queue is the head of the sorted list, the short queue the rest.
    // How many long items share a sub-partition (L) is chosen per launch from a two-term model of the
    // launch time, max(longest item at L per sub-partition, short-queue work / worker warps): more per
    // sub-partition slows the long chains (x1.15 alone, x1.31, x1.58, x2.0 measured for L = 1..4) but
    // takes fewer sub-partitions away from the short queue.  Thread l evaluates L = l + 1.
    __shared__ float t_of[kGkWarps / 4];
    const int long_cls = g.long_cls < 0 ? -1 : (g.long_cls > 254 ? 254 : g.long_cls);
    const unsigned n_long_all = long_cls >= 0 ? cnt[long_cls + 1] : 0u;
    if (c < kGkWarps / 4) {
        const float slow[4] = {1.155f, 1.31f, 1.585f, 2.0f};
        const int l = c + 1;
        const unsigned nl = min(n_long_all, (unsigned)(l * g.n_ctas));
        const unsigned ctas = (nl + l - 1) / l;
        // work of the nl longest items: whole classes below the class that holds item nl, part of that one
        int lo = 0, hi = kClasses;  // first class k with cnt[k + 1] >= nl
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (cnt[mid + 1] >= nl) hi = mid; else lo = mid + 1;
        }
        const int k = lo < kClasses ? lo : kClasses - 1;
        const float long_work = wrk[k] + (float)(nl - cnt[k]) * item_us(k);
        int c_max = 0;
        while (c_max < kClasses - 1 && cnt[c_max + 1] == 0) ++c_max;  // longest class present
        const float workers = (float)(kGkWarps * g.n_ctas) - (float)(kGkWarps / 4) * (float)ctas;
        const float t_short = (wrk[kClasses] - long_work) / fmaxf(workers, 1.0f);
        const float t_long = nl ? slow[c] * long_us(c_max) : 0.0f;
        t_of[c] = fmaxf(t_short, t_long);
        g.item_count[2 * kClasses + 8 + 2 * c] = __float_as_uint(t_short);  // diagnostics (wva_dbg_read_plan)
        g.item_count[2 * kClasses + 9 + 2 * c] = __float_as_uint(t_long);
    }
    __syncthreads();
    if (c == 0) {
        int L = g.long_per_sm;
        if (L < 0) {
            L = 1;
            for (int l = 2; l <= kGkWarps / 4; ++l)
                if (t_of[l - 1] < t_of[L - 1]) L = l;
        }
        const unsigned n_long = min(n_long_all, (unsigned)(L * g.n_ctas));
        g.item_count[2 * kClasses + 1] = n_long;
        g.item_count[2 * kClasses + 2] = 0;
        g.item_count[2 * kClasses + 3] = n_long;
        g.item_count[2 * kClasses + 4] = (unsigned)L;
    }
}
// Warp per item: the item takes its place in the global order (class cursors, longest class first) and its
// cells become 16-byte records in that order — cell id, lambda, the pair's table offset and the batch size —
// so that grid_kernel fetches an item's operands with ONE coalesced load instead of a chain of dependent ones
// (queue slot -> item -> order -> batch / replica / pair lists -> rate block).  A partial item (the last of a sort
// chunk) is padded with copies of its first cell, flagged, so that the whole warp takes part in the staged loads.
__global__ void __launch_bounds__(256) grid_items_scatter(GridArgs g) {
    const DevFleet& f = g.f;
    const unsigned n = *g.item_count;
    const unsigned lane = threadIdx.x & 31;
    const unsigned warps = (gridDim.x * blockDim.x) >> 5;
    for (unsigned i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
        const unsigned long long it = g.items[i];
        unsigned pos = 0;
        if (lane == 0) {
            pos = atomicAdd(g.item_count + 1 + kClasses + (unsigned)((it >> 40) & 0xff), 1u);
            g.items_sorted[pos] = it;
        }
        pos = __shfl_sync(0xffffffffu, pos, 0);
        const bool valid = lane < (unsigned)((it >> 32) & 0xff);
        const unsigned cell = g.order[(unsigned)it + (valid ? lane : 0u)];
        int s, a, bi, ri;
        decode_cell(g, (long long)cell, s, a, bi, ri);
        const float lambda = g.rt[s * g.R + ri].y;
        const unsigned toff = (unsigned)g.pair_tab_off[s * f.A + a];
        const unsigned b = (unsigned)g.batch[bi];
        // w: batch size (bits 0..22) | the item's length class (bits 23..30) | pad flag (bit 31)
        g.recs[(size_t)pos * 32 + lane] = make_uint4(cell, __float_as_uint(lambda), toff,
                                                     b | ((unsigned)((it >> 40) & 0xff) << 23) | (valid ? 0u : 0x80000000u));
    }
}

// ---------------------------------------------------------------------------
// grid_kernel — persistent, one CTA of kGkWarps warps per SM, warps pull items (32 cells of similar
// chain length) from two queues over the globally sorted item list:
//   * the LONG queue = the first n_long items (the longest chains, at most kGkLong per SM).  Their
//     latency bounds the launch: a 2816-state chain is 5632 dependent steps of >= 48 cycles, and
//     under equal sharing of a saturated FP64 pipe it would run 2-3x slower.  Warp w issues on SM
//     sub-partition w % 4 (tools/subpart_bench.cu), so the long items are pulled only by kGkLong
//     warps of sub-partition 0 and the other warps of that sub-partition stay parked until this
//     CTA's long warps are done: the long chains get a pipe to themselves;
//   * the SHORT queue = everything else, longest first, pulled by all other warps (and by the
//     sub-partition-0 warps once the CTA's long work is finished).
// ---------------------------------------------------------------------------
constexpr int kQLongN = 2 * kClasses + 1, kQLongCtr = kQLongN + 1, kQShortCtr = kQLongN + 2;  // in item_count[]

// Per-warp shared memory of grid_kernel (doubles): the pass-1 stash, the staged table window (+ the lanes' tail
// entries) and the pair record of the current item.
constexpr int kGkStashD = kGridStash * 32;              // [state][lane]
constexpr int kGkTbufD = kStagedTbufD;                  // staged table window + the lanes' tail entries
constexpr int kGkPairD = 8;                             // 48-byte pair record (padded to 64)
constexpr int kGkWarpD = kGkStashD + kGkTbufD + kGkPairD;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// One item: 32 records (one per lane) already in shared memory.  The solver gets everything it reads from the
// table in one batch of loads (solve_shared_t STAGED); the pair's constants travel into shared memory by
// cp.async meanwhile and are read back after the solve, so no operand of the epilogue is held in registers
// across the solver call and none is fetched by a dependent load afterwards.
__device__ __forceinline__ void item_run(const GridArgs& g, unsigned w, const uint4 rec, unsigned lane, double* warp_smem) {
    const DevFleet& f = g.f;
    double* stash_warp = warp_smem;
    double* tbuf_warp = warp_smem + kGkStashD;
    float4* pair_buf = reinterpret_cast<float4*>(warp_smem + kGkStashD + kGkTbufD);
    const unsigned idx = w * 32 + lane;
    const long long t_start = g.dbg_cycles ? clock64() : 0;
    unsigned long long t_start_ns = 0;
    if (g.dbg_cycles) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_start_ns));
    const unsigned cell = rec.x;
    const float lambda = __uint_as_float(rec.y);
    const double* tab = g.tab + 4 * (size_t)rec.z;
    const int N = (int)(rec.w & 0x7fffffu);
    const bool valid = (rec.w >> 31) == 0;
    const int K = N + N * f.ratio;
    const unsigned pair = cell / ((unsigned)g.B * (unsigned)g.R);
    // one pair per item is the rule (an item is cut from one sort chunk); then lanes 0..2 fetch its record
    const bool one_pair = __all_sync(0xffffffffu, pair == __shfl_sync(0xffffffffu, pair, 0));
    __syncwarp();  // the previous item's readers of pair_buf are done
    if (one_pair && lane < 3) cp_async16(pair_buf + lane, g.pair_rec + 3 * (size_t)pair + lane);
    cp_async_commit();
    ModelStats st;
    WVA_PROF_T(10);
    const int rc = solve_shared_t<kGridStash, 10, true>(tab, N, K, lambda, st, stash_warp + lane, tbuf_warp);
    WVA_PROF_T(11);
    cp_async_wait<0>();
    __syncwarp();
    if (valid) {
        if (rc != kSolveOk) {
            const int k = atomicAdd(g.fb_count, 1);
            if (k < g.fb_cap) g.fb_cells[k] = (long long)cell;
        } else {
            const float4 r0 = one_pair ? pair_buf[0] : g.pair_rec[3 * (size_t)pair + 0];
            const float4 r1 = one_pair ? pair_buf[1] : g.pair_rec[3 * (size_t)pair + 1];
            const float4 r2 = one_pair ? pair_buf[2] : g.pair_rec[3 * (size_t)pair + 2];
            QParams q;
            q.alpha = r0.x; q.beta = r0.y; q.gamma = r0.z; q.delta = r0.w;
            q.in_tok = __float_as_int(r1.x); q.out_tok = __float_as_int(r1.y);
            FeasRow fr;
            fr.slo_ttft = r1.z;
            fr.slo_itl = r1.w;
            fr.min_replicas = __float_as_int(r2.x);
            fr.tps = __float_as_int(r2.y) != 0;
            fr.lim = feas_lim(rate_max_of(st.tail_rate));  // RateRange.Max of (pair, N) from servRate[N-1]
            int s, a, bi, ri;
            decode_cell(g, (long long)cell, s, a, bi, ri);
            const Metrics m = metrics_from(q, N, st);
            const bool feas = cell_feasible(fr, g.replicas[ri], lambda, m);
            store_cell(g, (long long)cell, 1, feas ? 1 : 0, m);
            if (feas) atomicMin(&g.best_rank[(size_t)pair * g.R + ri], g.batch_rank[bi]);
            if (g.dbg_cycles) {
                g.dbg_cycles[idx] = (unsigned)(clock64() - t_start);
                if (lane < 3) {  // timeline: [0] start ns, [1] SM id, [2] end ns (low 32 bits of %globaltimer)
                    unsigned long long t_end;
                    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_end));
                    unsigned smid;
                    asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
                    g.dbg_cycles[g.dbg_n + idx] = lane == 0 ? (unsigned)t_start_ns : lane == 1 ? smid : (unsigned)t_end;
                }
            }
        }
    }
    __syncwarp();
    WVA_PROF_T(14);
}

__global__ void __launch_bounds__(kGkThreads, 1) grid_kernel(GridArgs g) {
    extern __shared__ __align__(16) double grid_smem[];
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* warp_smem = grid_smem + (size_t)warp * kGkWarpD;
    const unsigned n_items = g.item_count[0], n_long = g.item_count[kQLongN];
    const bool sub0 = (warp & 3) == 0;
    // the long items are spread over as few CTAs as possible (long_per_sm per CTA): the other CTAs keep all
    // four sub-partitions for the short queue
    const int per = (int)g.item_count[kQLongN + 3];  // long items per sub-partition, chosen by grid_items_plan
    const int long_ctas = per > 0 ? (int)((n_long + per - 1) / per) : 0;
    const int my_long = (int)blockIdx.x < long_ctas ? per : 0;
    const bool long_warp = sub0 && (int)(warp >> 2) < my_long;
    // sub-partition 0: long_per_sm warps pull the long queue, long_share more may pull short items next
    // to them, the rest wait on named barrier 1 (blocked in hardware: no issue slots) until the long warps
    // of this CTA have drained the long queue
    const int n_parked = my_long > 0 ? kGkWarps / 4 - my_long - g.long_share : 0;
    const int bar_threads = 32 * (my_long + (n_parked > 0 ? n_parked : 0));
    if (long_warp && n_long) {
        for (;;) {
            unsigned w = 0;
            if (lane == 0) w = atomicAdd(g.item_count + kQLongCtr, 1u);
            w = __shfl_sync(0xffffffffu, w, 0);
            if (w >= n_long) break;
            const uint4 rec = g.recs[(size_t)w * 32 + lane];
            item_run(g, w, rec, lane, warp_smem);
        }
        if (n_parked > 0) asm volatile("bar.arrive 1, %0;" ::"r"(bar_threads) : "memory");
    } else if (sub0 && my_long > 0 && !long_warp && (int)(warp >> 2) >= my_long + g.long_share) {
        asm volatile("bar.sync 1, %0;" ::"r"(bar_threads) : "memory");
    }
    // short queue: the list is longest-first and every warp takes the next item when it is free (LPT).  Reserving
    // items ahead of time (records prefetched two deep with cp.async) was measured and dropped: it hands a warp
    // two of the longest items back to back (the launch doubled), and restricted to the short classes it bought
    // nothing (0.219 vs 0.207 ms) — the four warps of a sub-partition already overlap each other's item boundaries.
    for (;;) {
        unsigned w = 0;
        if (lane == 0) w = atomicAdd(g.item_count + kQShortCtr, 1u);
        w = __shfl_sync(0xffffffffu, w, 0);
        if (w >= n_items) break;
        const uint4 rec = g.recs[(size_t)w * 32 + lane];
        item_run(g, w, rec, lane, warp_smem);
    }
}

// Stored-vector re-run of bailed cells. One thread per slot; slot k handles cells
// k, k + n_slots, ...  scratch per slot: (Kmax + 1) doubles then Nmax floats.
__global__ void grid_fallback(GridArgs g, double* scratch, size_t slot_doubles, int Kmax, int* fb_status) {
    const DevFleet& f = g.f;
    const int n_slots = gridDim.x * blockDim.x;
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    int n = *g.fb_count;
    if (n > g.fb_cap) n = g.fb_cap;
    double* p = scratch + (size_t)slot * slot_doubles;
    float* sr = (float*)(p + Kmax + 1);  // servRate copy lives behind the p[0..Kmax] vector
    for (int k = slot; k < n; k += n_slots) {
        const long long cell = g.fb_cells[k];
        int s, a, bi, ri;
        decode_cell(g, cell, s, a, bi, ri);
        const int b = g.batch[bi], r = g.replicas[ri];
        const double* tab = g.tab + 4 * g.pair_tab_off[s * f.A + a];
        for (int i = 0; i < b; ++i) sr[i] = (float)tab[4 * i];
        const float rmax = rate_max_of(sr[b - 1]);
        const float rate = __fdiv_rn(total_rate_of(f, s), (float)r);
        ModelStats st;
        const int rc = solve_stored(p, sr, b, b + b * f.ratio, __fdiv_rn(rate, 1000.0f), st);
        if (rc != 0) {
            atomicExch(fb_status, rc);
            continue;
        }
        const QParams q = qparams_of(f, s, a);
        const Metrics m = metrics_from(q, b, st);
        const bool feas = cell_feasible(feas_row(f, s, rmax), r, __fdiv_rn(rate, 1000.0f), m);
        store_cell(g, cell, 1, feas ? 1 : 0, m);
        if (feas) atomicMin(&g.best_rank[((size_t)s * f.A + a) * g.R + ri], g.batch_rank[bi]);
    }
}

// K3: per-server argmin.  One CTA per server: one candidate per (accelerator, replica
// level) = its smallest feasible batch size; warp-shuffle reduction, cross-warp reduction
// staged through shared memory.  The order (value, cost, replicas, batch, accelerator) does not involve the
// latency metrics, so only the keys are reduced; the winner's itl / ttft / rho are fetched once at the end:
// from the cell columns, or — for a cell that shares its row's chain and was not stored (want_cells == 0) —
// by the same stats_from_row + metrics_from evaluation grid_sort_local ran for it.
struct GridKey {
    float value, cost;
    int replicas, batch, acc, bi, ri, feasible;  // bi < 0: zero-load allocation of accelerator ri
};
__device__ __forceinline__ bool key_better(const GridKey& x, const GridKey& y) {
    if (!x.feasible) return false;
    if (!y.feasible) return true;
    if (x.value != y.value) return x.value < y.value;
    if (x.cost != y.cost) return x.cost < y.cost;
    if (x.replicas != y.replicas) return x.replicas < y.replicas;
    if (x.batch != y.batch) return x.batch < y.batch;
    return x.acc < y.acc;
}
__device__ __forceinline__ GridKey key_warp_min(GridKey c) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        GridKey o;
        o.value = __shfl_down_sync(0xffffffffu, c.value, d);
        o.cost = __shfl_down_sync(0xffffffffu, c.cost, d);
        o.replicas = __shfl_down_sync(0xffffffffu, c.replicas, d);
        o.batch = __shfl_down_sync(0xffffffffu, c.batch, d);
        o.acc = __shfl_down_sync(0xffffffffu, c.acc, d);
        o.bi = __shfl_down_sync(0xffffffffu, c.bi, d);
        o.ri = __shfl_down_sync(0xffffffffu, c.ri, d);
        o.feasible = __shfl_down_sync(0xffffffffu, c.feasible, d);
        if (key_better(o, c)) c = o;
    }
    return c;
}
__global__ void __launch_bounds__(256) grid_finalize(GridArgs g, AllocCols winners) {
    const DevFleet& f = g.f;
    const int s = blockIdx.x;
    GridKey best{};
    best.acc = -1;
    for (int k = threadIdx.x; k < f.A * g.R; k += blockDim.x) {
        const int a = k / g.R, ri = k % g.R;
        const int rank = g.best_rank[((size_t)s * f.A + a) * g.R + ri];
        if (rank == INT_MAX) continue;
        const int bi = g.rank_to_bi[rank];
        const int r = g.replicas[ri];
        Cand c = cand_nil();
        const long long total = (long long)num_instances(f, f.srv_model[s], a) * (long long)r;
        c.acc = a;
        c.replicas = r;
        c.cost = __fmul_rn(f.acc_cost[a], (float)total);
        GridKey key;
        key.value = penalty_of(f, s, c);
        key.cost = c.cost;
        key.replicas = r;
        key.batch = g.batch[bi];
        key.acc = a;
        key.bi = bi;
        key.ri = ri;
        key.feasible = 1;
        if (key_better(key, best)) best = key;
    }
    // zero-traffic servers: the reference's zeroLoadAllocation per candidate accelerator
    for (int a = threadIdx.x; a < f.A; a += blockDim.x) {
        if (pair_class(f, s, a, true) == PAIR_ZERO) {
            Cand c = zero_load_alloc(f, s, a);
            GridKey key;
            key.value = penalty_of(f, s, c);
            key.cost = c.cost;
            key.replicas = c.replicas;
            key.batch = c.batch;
            key.acc = c.acc;
            key.bi = -1;
            key.ri = a;
            key.feasible = 1;
            if (key_better(key, best)) best = key;
        }
    }
    best = key_warp_min(best);
    __shared__ GridKey sm[8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) sm[warp] = best;
    __syncthreads();
    if (warp == 0) {
        GridKey k = sm[0];
        if (lane > 0 && lane < (int)(blockDim.x >> 5)) k = sm[lane];
        if (lane >= (int)(blockDim.x >> 5)) k.feasible = 0;
        k = key_warp_min(k);
        if (lane == 0) {
            Cand c = cand_nil();
            if (k.feasible && k.bi < 0) {
                c = zero_load_alloc(f, s, k.ri);
                c.value = penalty_of(f, s, c);
            } else if (k.feasible) {
                const int a = k.acc, ri = k.ri, b = k.batch;
                c.feasible = 1;
                c.acc = a;
                c.replicas = k.replicas;
                c.batch = b;
                c.cost = k.cost;
                c.value = k.value;
                const size_t row = ((size_t)s * f.A + a) * g.R + ri;
                const long long cell = ((long long)row / g.R * g.B + k.bi) * g.R + ri;
                const int jl = g.row_j[row];
                const int K = b + b * f.ratio;
                if (!g.want_cells && cell_shared(jl, b, K)) {
                    // the cell shares its row's chain and was not stored: the evaluation grid_sort_local (or, for a
                    // resolved row, grid_rows) ran for it, again
                    const float lambda = g.rt[s * g.R + ri].y;
                    ModelStats st;
                    stats_from_row(g.row_acc[row], g.row_sump[row], b, lambda, st);
                    const Metrics m = metrics_from(qparams_of(f, s, a), b, st);
                    c.itl = m.avg_token_time;
                    c.ttft = m.ttft;
                    c.rho = m.rho;
                } else {
                    c.itl = g.cells.itl[cell];
                    c.ttft = g.cells.ttft[cell];
                    c.rho = g.cells.rho[cell];
                }
                c.max_rate = __fdiv_rn(rate_max_of((float)g.tab[4 * (g.pair_tab_off[s * f.A + a] + b - 1)]), 1000.0f);
            }
            store_cand(winners, s, c);
        }
    }
}

// ---------------------------------------------------------------------------
// K1: size candidates (CreateAllocation).
// ---------------------------------------------------------------------------

// Solver policies: a solver evaluates Model.Solve(lambda, 1) and reports bail-outs.
struct StoredSolver {  // stored-vector fallback
    double* p;
    const float* sr;
    int N, K;
    int bail;
    __device__ __forceinline__ int solve(float lambda, ModelStats& st) {
        const int rc = solve_stored(p, sr, N, K, lambda, st);
        if (rc != 0) bail = rc;
        return rc;
    }
};

// EvalTTFT / EvalITL (queueanalyzer.go:270-290) + BinarySearch (utils.go:26-70).
// which = 0: TTFT, 1: ITL.  Returns 0 ok (xstar, ind), 2 eval error / bail.
template <class Solver>
__device__ int eval_target(Solver& sv, const QParams& q, int which, float x, float& y) {
    ModelStats st;
    if (sv.solve(x, st) != 0) return 2;
    const float eff = effective_concurrency(q, st.avg_serv_time, sv.N);
    if (which == 0)
        y = __fadd_rn(st.avg_wait_time, prefill_time(q, eff));
    else
        y = decode_time(q, eff);
    return 0;
}
template <class Solver>
__device__ int binary_search(Solver& sv, const QParams& q, int which, float xmin, float xmax, float ytarget,
                             float& xstar, int& ind) {
    xstar = 0.0f;
    ind = 0;
    if (xmin > xmax) return 1;
    float y0, y1;
    if (eval_target(sv, q, which, xmin, y0)) return 2;
    if (within_tolerance(y0, ytarget, 1e-6f)) { xstar = xmin; return 0; }
    if (eval_target(sv, q, which, xmax, y1)) return 2;
    if (within_tolerance(y1, ytarget, 1e-6f)) { xstar = xmax; return 0; }
    const bool increasing = y0 < y1;
    if ((increasing && ytarget < y0) || (!increasing && ytarget > y0)) { xstar = xmin; ind = -1; return 0; }
    if ((increasing && ytarget > y1) || (!increasing && ytarget < y1)) { xstar = xmax; ind = 1; return 0; }
    float xs = 0.0f, ys = 0.0f;
    for (int it = 0; it < 100; ++it) {
        xs = __fmul_rn(0.5f, __fadd_rn(xmin, xmax));
        if (eval_target(sv, q, which, xs, ys)) return 2;
        if (within_tolerance(ys, ytarget, 1e-6f)) break;
        const float pmin = xmin, pmax = xmax;
        if ((increasing && ytarget < ys) || (!increasing && ytarget > ys))
            xmax = xs;
        else
            xmin = xs;
        // Fixed point: the iteration is a deterministic function of (xmin, xmax), so once an
        // iteration leaves both bounds unchanged (the float32 interval has collapsed) the
        // reference's remaining iterations repeat the same solve and return the same xStar.
        if (xmin == pmin && xmax == pmax) break;
    }
    xstar = xs;
    return 0;
}

// Analyze (queueanalyzer.go:134-174) -> 0 ok.
template <class Solver>
__device__ int analyze(Solver& sv, const QParams& q, float rmax, float rate, Metrics& m) {
    if (rate <= 0.0f) return 1;
    if (rate > rmax) return 2;
    ModelStats st;
    if (sv.solve(__fdiv_rn(rate, 1000.0f), st) != 0) return 3;
    m = metrics_from(q, sv.N, st);
    return 0;
}

// CreateAllocation under load (allocation.go:77-163); value = cost.
// s1 / sN = servRate[0] / servRate[N-1] (float32).
template <class Solver>
__device__ Cand create_allocation(const DevFleet& f, int s, int a, Solver& sv, float s1, float sN) {
    Cand out = cand_nil();
    if (sv.K < 2) return out;  // a model with K <= 1 is never valid (queuemodel.go:31, stale rho = 1)
    const QParams q = qparams_of(f, s, a);
    const float rmin = rate_min_of(s1), rmax = rate_max_of(sN);
    const float slo_ttft = f.srv_slo_ttft[s], slo_itl = f.srv_slo_itl[s], slo_tps = f.srv_slo_tps[s];
    if (slo_itl < 0.0f || slo_ttft < 0.0f || slo_tps < 0.0f) return out;  // TargetPerf.check :322-329
    const float lambda_min = __fdiv_rn(rmin, 1000.0f), lambda_max = __fdiv_rn(rmax, 1000.0f);
    int ind = 0;
    float l_ttft = lambda_max, l_itl = lambda_max, l_tps = lambda_max;
    if (slo_ttft > 0.0f) {  // queueanalyzer.go:205-215
        const int err = binary_search(sv, q, 0, lambda_min, lambda_max, slo_ttft, l_ttft, ind);
        if (ind < 0 || err != 0) return out;
    }
    if (slo_itl > 0.0f) {  // :218-228
        const int err = binary_search(sv, q, 1, lambda_min, lambda_max, slo_itl, l_itl, ind);
        if (ind < 0 || err != 0) return out;
    }
    if (slo_tps > 0.0f) l_tps = __fmul_rn(lambda_max, __fsub_rn(1.0f, 0.1f));  // :231-234
    const float lambda = go_minf(go_minf(l_ttft, l_itl), l_tps);
    Metrics m;
    if (analyze(sv, q, rmax, __fmul_rn(lambda, 1000.0f), m) != 0) return out;  // :237-241
    const float rate_star = m.throughput;

    const float total_rate = total_rate_of(f, s);  // allocation.go:134-141
    long long nrep = go_f64_to_int(ceil(__ddiv_rn((double)total_rate, (double)rate_star)));
    const long long min_rep = f.srv_min_replicas[s];
    if (nrep < min_rep) nrep = min_rep;
    const long long total = (long long)num_instances(f, f.srv_model[s], a) * nrep;  // :144-145
    const float cost = __fmul_rn(f.acc_cost[a], (float)total);
    const float rate = __fdiv_rn(total_rate, (float)nrep);  // :148-153
    if (analyze(sv, q, rmax, rate, m) != 0) return out;
    out.feasible = 1;
    out.acc = a;
    out.replicas = (int)nrep;
    out.batch = sv.N;
    out.cost = cost;
    out.value = cost;
    out.itl = m.avg_token_time;
    out.ttft = m.ttft;
    out.rho = m.rho;
    out.max_rate = __fdiv_rn(rate_star, 1000.0f);
    return out;
}

struct SizeArgs {
    DevFleet f;
    const int* cand_pair;  // [n_cand] pair ids sorted by descending N
    const int* cand_N;     // [n_cand]
    int n_cand;
    AllocCols cand;        // [n_scen*S*A]
    int* fb_count;
    int* fb_list;          // entries j * n_scen + l: candidate j bailed under scenario l
    int fb_cap;
    const float* scen_rpm;  // [n_scen*S] arrival columns of wva_resolve_scenarios; NULL = the fleet's own
    int n_scen;             // 1 without scenarios
};

// Stored-vector re-run of bailed candidates (slot k handles list entries k, k+n_slots, ..).
__global__ void size_fallback(SizeArgs g, double* scratch, size_t slot_doubles, int Kmax, int* fb_status) {
    DevFleet f = g.f;
    const int n_slots = gridDim.x * blockDim.x;
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    int n = *g.fb_count;
    if (n > g.fb_cap) n = g.fb_cap;
    double* p = scratch + (size_t)slot * slot_doubles;
    float* sr = (float*)(p + Kmax + 1);
    for (int k = slot; k < n; k += n_slots) {
        const int e = g.fb_list[k];
        const int j = e / g.n_scen, l = e - j * g.n_scen;
        if (g.scen_rpm) f.srv_arrival_rpm = g.scen_rpm + (size_t)l * f.S;
        const int pair = g.cand_pair[j];
        const int s = pair / f.A, a = pair % f.A;
        StoredSolver sv;
        sv.N = g.cand_N[j];
        sv.K = sv.N + sv.N * f.ratio;
        sv.p = p;
        sv.sr = sr;
        sv.bail = 0;
        const QParams q = qparams_of(f, s, a);
        for (int i = 0; i < sv.N; ++i) sr[i] = serv_rate(q, i + 1);
        for (int i = 0; i <= sv.K; ++i) p[i] = 0.0;
        Cand c = create_allocation(f, s, a, sv, sr[0], sr[sv.N - 1]);
        if (sv.bail) {
            atomicExch(fb_status, sv.bail);
            c = cand_nil();
        }
        store_cand(g.cand, (size_t)l * f.S * f.A + pair, c);
    }
}

// ---------------------------------------------------------------------------
// K1 (size candidates as rounds of sorted solve batches) lives in wva_size.cuh; the sort workspace and the
// item ordering kernels it shares with nothing else stay here next to the grid's.
// ---------------------------------------------------------------------------
struct SortWs {
    unsigned* order;
    unsigned long long* items;
    unsigned long long* items_sorted;
    unsigned* item_count;  // [0] items, [1..256] per class, [257..512] cursors
};
enum { PH_SEARCH = 0, PH_WAIT_STAR = 1, PH_WAIT_FINAL = 2, PH_DONE = 3, PH_NIL = 4, PH_BAIL = 5 };
__global__ void __launch_bounds__(256) ws_items_scan(SortWs ws) {
    __shared__ unsigned tot[kClasses];
    tot[threadIdx.x] = ws.item_count[1 + threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned acc = 0;
        for (int c = 0; c < kClasses; ++c) {
            ws.item_count[1 + kClasses + c] = acc;
            acc += tot[c];
        }
    }
}
__global__ void __launch_bounds__(256) ws_items_scatter(SortWs ws) {
    const unsigned n = *ws.item_count;
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long it = ws.items[i];
    ws.items_sorted[agg_inc(ws.item_count + 1 + kClasses, (int)((it >> 40) & 0xff))] = it;
}


// nil and zero-load candidates (everything the size kernel does not own).  blockIdx.y = scenario l of
// wva_resolve_scenarios: row l of scen_rpm replaces the fleet's arrival column and the records go to block l.
__global__ void trivial_kernel(DevFleet f, AllocCols cand, const float* scen_rpm) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= f.S * f.A) return;
    if (scen_rpm) f.srv_arrival_rpm = scen_rpm + (size_t)blockIdx.y * f.S;
    const int s = pair / f.A, a = pair % f.A;
    const int cls = pair_class(f, s, a, true);
    if (cls == PAIR_LOAD) return;
    Cand c = cand_nil();
    if (cls == PAIR_ZERO) c = zero_load_alloc(f, s, a);
    store_cand(cand, (size_t)blockIdx.y * f.S * f.A + pair, c);
}

// Server.Calculate's value (server.go:60-63) + SolveUnlimited (solver.go:63-79):
// one thread per server; strict '<' from MaxFloat32, lowest accelerator id wins ties.  blockIdx.y = scenario
// (candidate block y, winner block y); nothing here reads the arrival rate.
__global__ void unlimited_kernel(DevFleet f, AllocCols cand, AllocCols winners) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= f.S) return;
    float min_val = 3.40282346638528859811704183484516925440e+38f;
    Cand best = cand_nil();
    const size_t scen = blockIdx.y;
    for (int a = 0; a < f.A; ++a) {
        const size_t i = (scen * f.S + s) * f.A + a;
        if (!cand.feasible[i]) continue;
        Cand c = load_cand(cand, i);
        c.value = penalty_of(f, s, c);
        cand.value[i] = c.value;
        if (c.value < min_val) {
            min_val = c.value;
            best = c;
        }
    }
    store_cand(winners, scen * f.S + s, best);
}

// ---------------------------------------------------------------------------
// What Manager.Optimize / Solver.Solve leave behind next to the solution: System.AllocateByType
// (pkg/core/system.go:271-300) and CreateAllocationDiff per server (pkg/core/allocation.go:353-380,
// pkg/solver/solver.go:51-58).  One CTA: the diffs are element-wise; the per-type totals add float32
// costs in ascending server index (the reference's own order is Go map order), so thread t owns type t
// and walks the servers in order, chunk by chunk through shared memory (coalesced loads, serial adds).
// ---------------------------------------------------------------------------
struct SummaryOut {
    uint8_t* type_present;
    long long* type_count;
    int* type_limit;
    float* type_cost;
    int *diff_old_acc, *diff_new_acc, *diff_old_replicas, *diff_new_replicas;
    float* diff_cost;
};
constexpr int kSumChunk = 1024;
constexpr int kSumMaxTypes = 1024;  // 256 threads x 4 owned types
__global__ void __launch_bounds__(256) summary_kernel(DevFleet f, AllocCols win, SummaryOut o) {
    __shared__ int s_type[kSumChunk];
    __shared__ long long s_units[kSumChunk];
    __shared__ float s_cost[kSumChunk];
    // one accumulator set per owned type (thread t owns types t, t + 256, ...: at most 4 in registers)
    constexpr int kOwn = 4;
    long long cnt[kOwn];
    float cost[kOwn];
    int present[kOwn];
#pragma unroll
    for (int k = 0; k < kOwn; ++k) { cnt[k] = 0; cost[k] = 0.0f; present[k] = 0; }
    for (int base = 0; base < f.S; base += kSumChunk) {
        const int n = min(kSumChunk, f.S - base);
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const int s = base + i;
            const int feas = win.feasible[s], acc = win.acc[s], rep = win.replicas[s];
            const float c = win.cost[s];
            int type = -1;
            long long units = 0;
            const int m = f.srv_model[s];
            if (feas && acc >= 0 && acc < f.A && m >= 0 && m < f.M) {  // system.go:276-284
                const int t = f.acc_type[acc];
                if (t >= 0 && t < f.T) {
                    type = t;
                    const long long inst = f.perf_present[m * f.A + acc] ? num_instances(f, m, acc) : 0;
                    units = (long long)rep * inst * (long long)f.acc_mult[acc];  // :296
                }
            }
            s_type[i] = type;
            s_units[i] = units;
            s_cost[i] = c;
            // CreateAllocationDiff(current, solution)
            if (o.diff_old_acc) o.diff_old_acc[s] = f.srv_cur_acc[s];
            if (o.diff_old_replicas) o.diff_old_replicas[s] = f.srv_cur_replicas[s];
            if (o.diff_new_acc) o.diff_new_acc[s] = feas ? acc : -3;
            if (o.diff_new_replicas) o.diff_new_replicas[s] = feas ? rep : 0;
            if (o.diff_cost) o.diff_cost[s] = __fsub_rn(feas ? c : 0.0f, f.srv_cur_cost[s]);
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kOwn; ++k) {
            const int t = threadIdx.x + k * blockDim.x;
            if (t < f.T) {
                for (int i = 0; i < n; ++i)
                    if (s_type[i] == t) {
                        present[k] = 1;
                        cnt[k] += s_units[i];
                        cost[k] = __fadd_rn(cost[k], s_cost[i]);  // :297, float32
                    }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int k = 0; k < kOwn; ++k) {
        const int t = threadIdx.x + k * blockDim.x;
        if (t < f.T) {
            if (o.type_present) o.type_present[t] = (uint8_t)present[k];
            if (o.type_count) o.type_count[t] = cnt[k];
            if (o.type_limit) o.type_limit[t] = f.type_capacity[t];
            if (o.type_cost) o.type_cost[t] = cost[k];
        }
    }
}

// ---------------------------------------------------------------------------
// MM1KModel (closed form): pkg/analyzer/mm1kmodel.go:19-92 over QueueModel.Solve (queuemodel.go:27-37).  One
// thread per (K, lambda, mu) triple; the probabilities are streamed in the reference's order (sumP and the
// sum(i p[i]) accumulate over i = 0..K), never stored.
// ---------------------------------------------------------------------------
struct Mm1kArgs {
    int n;
    const int* K;
    const float* lambda;
    const float* mu;
    uint8_t* is_valid;
    float *rho, *avg_num_in_system, *throughput, *avg_resp_time, *avg_serv_time, *avg_wait_time, *avg_queue_length;
    double* sum_p;
};
__global__ void __launch_bounds__(128) mm1k_kernel(Mm1kArgs g) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= g.n) return;
    const int K = g.K[q];
    const float lambda = g.lambda[q], mu = g.mu[q];
    const float rho = (lambda == mu) ? 1.0f : __fdiv_rn(lambda, mu);  // ComputeRho: mm1kmodel.go:38-44
    // QueueModel.Solve validity: queuemodel.go:31 with GetRhoMax = K (mm1kmodel.go:46-48)
    const bool valid = !((rho < 0.0f) || (rho >= (float)K) || (lambda < 0.0f) || (mu <= 0.0f));
    float nsys = 0.f, thr = 0.f, resp = 0.f, serv = 0.f, wait = 0.f, qlen = 0.f;
    double sum_p = 0.0;
    if (valid) {
        const double r = (double)rho;
        // computeProbabilities: mm1kmodel.go:51-72
        const double p0 = (rho == 1.0f) ? __ddiv_rn(1.0, (double)(K + 1))
                                        : __ddiv_rn(__dsub_rn(1.0, r), __dsub_rn(1.0, go_pow_uint(r, (long long)K + 1)));
        double temp = 0.0, pK = 0.0;
        for (int i = 0; i <= K; ++i) {
            const double pi = __dmul_rn(p0, go_pow_uint(r, (long long)i));
            sum_p = __dadd_rn(sum_p, pi);
            temp = __dadd_rn(temp, __dmul_rn((double)i, pi));  // computeStatistics: :75-92
            pK = pi;
        }
        nsys = (float)temp;
        thr = __fmul_rn(lambda, __fsub_rn(1.0f, (float)pK));
        resp = __fdiv_rn(nsys, thr);
        serv = __fdiv_rn(1.0f, mu);
        wait = __fsub_rn(resp, serv);
        if (wait < 0.0f) wait = 0.0f;
        qlen = __fmul_rn(thr, wait);
    }
    g.is_valid[q] = valid ? 1 : 0;
    g.rho[q] = rho;
    g.avg_num_in_system[q] = nsys;
    g.throughput[q] = thr;
    g.avg_resp_time[q] = resp;
    g.avg_serv_time[q] = serv;
    g.avg_wait_time[q] = wait;
    g.avg_queue_length[q] = qlen;
    g.sum_p[q] = sum_p;
}

// ---------------------------------------------------------------------------
// Latency sweep: warp = 32 consecutive rates of one (server, acc) pair.
// ---------------------------------------------------------------------------
struct SweepArgs {
    DevFleet f;
    const int* pair_list;  // pairs sorted by descending N
    const int* pair_N;     // N per entry of pair_list
    const long long* tab_off;  // shared-table entry offset per entry of pair_list
    const double* tab;
    int n_pairs, n_rates, n_chunks;
    unsigned* counter;
    uint8_t* valid;
    float *rate, *ttft, *itl, *throughput, *rho;
    int* fb_count;         // sweep points that need the stored-vector fallback
    long long* fb_points;  // their point indices e * n_rates + i (entry of pair_list, rate index), up to fb_cap
    int fb_cap;
};

__global__ void __launch_bounds__(256) sweep_kernel(SweepArgs g) {
    const DevFleet& f = g.f;
    const int lane = threadIdx.x & 31;
    const unsigned n_items = (unsigned)g.n_pairs * g.n_chunks;
    for (;;) {
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(g.counter, 1u);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int e = item / g.n_chunks, chunk = item % g.n_chunks;
        const int pair = g.pair_list[e];
        const int s = pair / f.A, a = pair % f.A;
        const int N = g.pair_N[e], K = N + N * f.ratio;
        const double* tab = g.tab + 4 * g.tab_off[e];
        Recip tail;
        tail.b = tab[4 * (N - 1)];
        tail.yh = tab[4 * (N - 1) + 1];
        tail.yl = tab[4 * (N - 1) + 2];
        const float rmin = rate_min_of((float)tab[0]), rmax = rate_max_of((float)tail.b);
        const int i = chunk * 32 + lane;
        if (i < g.n_rates) {
        const float hi = __fmul_rn(rmax, 0.999f);
        const float span = __fsub_rn(hi, rmin);
        const float frac = g.n_rates > 1 ? __fdiv_rn((float)i, (float)(g.n_rates - 1)) : 0.0f;
        const float rate = __fadd_rn(rmin, __fmul_rn(span, frac));
        const size_t o = (size_t)pair * g.n_rates + i;
        g.rate[o] = rate;
        uint8_t ok = 0;
        Metrics m;
        m.ttft = m.avg_token_time = m.rho = m.throughput = 0.0f;
        if (!(rate <= 0.0f) && !(rate > rmax) && K >= 2) {
            ModelStats st;
            const QParams q = qparams_of(f, s, a);
            if (solve_shared(tab, N, K, __fdiv_rn(rate, 1000.0f), st) == kSolveOk) {
                m = metrics_from(q, N, st);
                ok = 1;
            } else {
                const int k = atomicAdd(g.fb_count, 1);
                if (k < g.fb_cap) g.fb_points[k] = (long long)e * g.n_rates + i;
            }
        }
        g.valid[o] = ok;
        g.ttft[o] = m.ttft;
        g.itl[o] = m.avg_token_time;
        g.throughput[o] = m.throughput;
        g.rho[o] = m.rho;
        }
    }
}

// Stored-vector re-run of the sweep points sweep_kernel bailed on (p or the sum left the streaming solve's window,
// e.g. a chain the reference rescales).  Slots as in grid_fallback; the rate is recomputed exactly as sweep_kernel
// computed it.
__global__ void sweep_fallback(SweepArgs g, double* scratch, size_t slot_doubles, int Kmax, int* fb_status) {
    const DevFleet& f = g.f;
    const int n_slots = gridDim.x * blockDim.x;
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    int n = *g.fb_count;
    if (n > g.fb_cap) n = g.fb_cap;
    double* p = scratch + (size_t)slot * slot_doubles;
    float* sr = (float*)(p + Kmax + 1);
    for (int k = slot; k < n; k += n_slots) {
        const long long pt = g.fb_points[k];
        const int e = (int)(pt / g.n_rates), i = (int)(pt % g.n_rates);
        const int pair = g.pair_list[e];
        const int s = pair / f.A, a = pair % f.A;
        const int N = g.pair_N[e], K = N + N * f.ratio;
        const double* tab = g.tab + 4 * g.tab_off[e];
        for (int j = 0; j < N; ++j) sr[j] = (float)tab[4 * j];
        const float rmin = rate_min_of(sr[0]), rmax = rate_max_of(sr[N - 1]);
        const float hi = __fmul_rn(rmax, 0.999f);
        const float span = __fsub_rn(hi, rmin);
        const float frac = g.n_rates > 1 ? __fdiv_rn((float)i, (float)(g.n_rates - 1)) : 0.0f;
        const float rate = __fadd_rn(rmin, __fmul_rn(span, frac));
        ModelStats st;
        const int rc = solve_stored(p, sr, N, K, __fdiv_rn(rate, 1000.0f), st);
        if (rc != 0) {
            atomicExch(fb_status, rc);
            continue;
        }
        const Metrics m = metrics_from(qparams_of(f, s, a), N, st);
        const size_t o = (size_t)pair * g.n_rates + i;
        g.valid[o] = 1;
        g.ttft[o] = m.ttft;
        g.itl[o] = m.avg_token_time;
        g.throughput[o] = m.throughput;
        g.rho[o] = m.rho;
    }
}

}  // namespace wva
