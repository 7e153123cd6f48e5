// wva_size.cuh — K1, the reference's decision path: CreateAllocation (pkg/core/allocation.go:27-163) for every
// (server, accelerator) candidate as ROUNDS of sorted solve batches with SPECULATIVE bisection.
//
// The reference runs, per candidate, two sequential bisections (pkg/analyzer/utils.go:26-70) of <= 102 model
// solves each, then two Analyze calls.  The solves of one bisection depend on each other only through ONE
// comparison per iteration, and the next midpoint can only be one of two values; so a round evaluates the whole
// binary tree of midpoints the next D iterations can reach (2^D - 1 solves: node 1 = mid(lo, hi), node 2v / 2v + 1 =
// the midpoints after "target below" / "target above" at node v), and the state machine then walks the tree with
// the reference's comparisons, tolerance test and iteration count.  Every lambda is produced by the reference's own
// float32 expression 0.5 * (xmin + xmax) on the reference's own bounds, so the D iterations a round resolves are
// the reference's iterations, bit for bit; the evaluations off the taken path are discarded.  D iterations per
// round instead of one: ~36 rounds become ~36 / D + 3.
//
// Why this is also the fix for the memory traffic: every candidate owns a service-rate table (its token profile is
// its own), and with one request per candidate per round each lane of a solve warp streamed a different table
// (530 MB of DRAM reads per round on 100 k candidates, FP64 pipe at 16 %).  The 2 x (2^D - 1) requests of a
// candidate share ONE table; they are emitted into consecutive slots and, once the interval has narrowed, fall
// into the same length class, so the sort keeps them adjacent and a solve warp reads a few tables instead of 32.
//
// Rounds are enqueued without host synchronisation (grids sized for the worst case, every kernel leaves at once
// when its work list is empty); the host looks at the request counter once per group of rounds.
#pragma once
#include "wva_kernels.cuh"

namespace wva {

constexpr int kSzMaxDepth = 5;  // midpoint tree depth: at most 31 evaluations per search per round

enum { SZ2_START = 0, SZ2_WAIT_FIRST = 1, SZ2_WAIT_ITER = 2, SZ2_DONE = 3, SZ2_OFF = 4 };

struct Sz2Args {
    DevFleet f;
    const int* cand_pair;  // [n] pair ids, descending N
    const int* cand_N;     // [n]
    int n_cand;
    int depth;             // D
    const double* tab;     // shared-format tables, one per candidate
    const long long* tab_off;  // [n]
    const float* ls;
    // search state, index 2*j + which (0: TTFT, 1: ITL)
    float *xmin, *xmax, *xs;
    uint8_t *sst, *inc, *iter;
    int8_t* ind;
    int* slot;             // [2n] first request slot of the search this round
    // candidate state
    uint8_t* phase;
    float *rmax, *l2s0, *l2sN, *lsN, *rate_star, *cost;
    long long* nrep;
    int* aslot;            // [n] request slot of the candidate's Analyze this round
    // requests of the current round
    unsigned* req_id;      // 4*j + kind (0 TTFT eval, 1 ITL eval, 2 Analyze(lambda*), 3 Analyze(final))
    int* req_scen;         // scenario of a kind-3 request emitted by sz2_expand
    float* req_lam;
    uint8_t* req_key;
    float4* req_out;       // kinds 0/1: x = y; kinds 2/3: throughput, ttft, itl, rho
    uint8_t* req_bail;
    unsigned* n_req;       // device counter of this round
    unsigned* n_live;      // device counter: candidates that are not finished yet (host stop test)
    SortWs ws;
    AllocCols cand;
    int* fb_count;
    int* fb_list;
    int fb_cap;
    unsigned* dbg;         // diagnostics (WVA_SIZE_DBG_ROUND): per slot {SM cycles, N, lambda bits, warp}, or NULL
    const float* scen_rpm;  // wva_resolve_scenarios: [n_scen*S] arrival columns (sz2_expand / sz2_consume)
    int n_scen;
};

__device__ __forceinline__ float sz_mid(float lo, float hi) { return __fmul_rn(0.5f, __fadd_rn(lo, hi)); }  // utils.go:55

// Midpoint of heap node v (1-based) of the tree over (lo, hi): follow v's path bits below its leading one.
__device__ __forceinline__ float sz_node_value(int v, float lo, float hi) {
    const int depth = 31 - __clz(v);
    for (int b = depth - 1; b >= 0; --b) {
        const float x = sz_mid(lo, hi);
        if ((v >> b) & 1) lo = x; else hi = x;
    }
    return sz_mid(lo, hi);
}

__global__ void __launch_bounds__(256) sz2_init(Sz2Args g) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= g.n_cand) return;
    const DevFleet& f = g.f;
    const int pair = g.cand_pair[j], s = pair / f.A;
    const int N = g.cand_N[j], K = N + N * f.ratio;
    const double* tab = g.tab + 4 * g.tab_off[j];
    const float s1 = (float)tab[0], sN = (float)tab[4 * (N - 1)];
    const float rmin = rate_min_of(s1), rmax = rate_max_of(sN);
    g.rmax[j] = rmax;
    g.l2s0[j] = log2f(s1);
    g.l2sN[j] = log2f(sN);
    g.lsN[j] = (g.ls + g.tab_off[j] + j)[N - 1];
    const float slo_ttft = f.srv_slo_ttft[s], slo_itl = f.srv_slo_itl[s], slo_tps = f.srv_slo_tps[s];
    uint8_t ph = PH_SEARCH;
    // K <= 1: the model is never valid (queuemodel.go:31); negative targets: TargetPerf.check :322-329
    if (K < 2 || slo_itl < 0.0f || slo_ttft < 0.0f || slo_tps < 0.0f) ph = PH_NIL;
    g.phase[j] = ph;
    const float lmin = __fdiv_rn(rmin, 1000.0f), lmax = __fdiv_rn(rmax, 1000.0f);
    for (int w = 0; w < 2; ++w) {
        const float target = w == 0 ? slo_ttft : slo_itl;
        g.xmin[2 * j + w] = lmin;
        g.xmax[2 * j + w] = lmax;
        g.xs[2 * j + w] = lmax;  // lambdaStar when the target is disabled (queueanalyzer.go:205,218)
        g.sst[2 * j + w] = target > 0.0f ? SZ2_START : SZ2_OFF;
        g.ind[2 * j + w] = 0;
        g.iter[2 * j + w] = 0;
        g.slot[2 * j + w] = -1;
    }
    g.aslot[j] = -1;
    if (ph == PH_NIL) store_cand(g.cand, pair, cand_nil());
}

// Advance every candidate: consume last round's results (walking the midpoint trees with the reference's
// comparisons), then emit this round's requests into consecutive slots.
// STAR (wva_resolve_scenarios): stop after Analyze(lambda*) with rateStar in rate_star[j] and phase PH_DONE; nil and
// bailed candidates only leave their phase behind (no record, no fallback entry): sz2_expand handles them per scenario.
template <bool STAR>
__global__ void __launch_bounds__(256) sz2_advance(Sz2Args g) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const DevFleet& f = g.f;
    const int D = g.depth, M = (1 << D) - 1;
    const int lane = threadIdx.x & 31;
    int ph = PH_DONE;
    int pair = 0, s = 0, a = 0;
    float rmax = 0.0f;
    if (j < g.n_cand) {
        ph = g.phase[j];
        pair = g.cand_pair[j];
        s = pair / f.A;
        a = pair % f.A;
        rmax = g.rmax[j];
    }
    const bool live_in = ph < PH_DONE;
    // what this thread will emit: per search a tree (optionally preceded by the two end points), or one Analyze
    int emit_n[2] = {0, 0};
    bool emit_ends[2] = {false, false};
    float emit_lo[2] = {0.f, 0.f}, emit_hi[2] = {0.f, 0.f};
    int an_kind = -1;
    float an_lambda = 0.0f;
    if (live_in) {
        if (ph == PH_SEARCH) {
            bool all_done = true, nil = false, bail = false;
            for (int w = 0; w < 2 && !bail && !nil; ++w) {
                const int k = 2 * j + w;
                int st = g.sst[k];
                if (st == SZ2_DONE || st == SZ2_OFF) continue;
                const float target = w == 0 ? f.srv_slo_ttft[s] : f.srv_slo_itl[s];
                float lo = g.xmin[k], hi = g.xmax[k];
                bool searching = true;
                if (st == SZ2_START) {  // utils.go:29-31
                    if (lo > hi) { nil = true; break; }
                    emit_ends[w] = true;
                    st = SZ2_WAIT_FIRST;
                } else {
                    int base = g.slot[k];
                    bool inc = g.inc[k] != 0;
                    if (st == SZ2_WAIT_FIRST) {  // utils.go:36-51: the two boundary evaluations
                        if (g.req_bail[base]) { bail = true; break; }
                        const float y0 = g.req_out[base].x;
                        if (within_tolerance(y0, target, 1e-6f)) { g.xs[k] = lo; searching = false; }
                        else {
                            if (g.req_bail[base + 1]) { bail = true; break; }
                            const float y1 = g.req_out[base + 1].x;
                            if (within_tolerance(y1, target, 1e-6f)) { g.xs[k] = hi; searching = false; }
                            else {
                                inc = y0 < y1;
                                g.inc[k] = inc;
                                if ((inc && target < y0) || (!inc && target > y0)) { g.xs[k] = lo; g.ind[k] = -1; searching = false; }
                                else if ((inc && target > y1) || (!inc && target < y1)) { g.xs[k] = hi; g.ind[k] = 1; searching = false; }
                            }
                        }
                        base += 2;
                        st = SZ2_WAIT_ITER;
                    }
                    if (searching) {  // utils.go:54-68, D iterations: walk the tree of midpoints evaluated last round
                        int it = g.iter[k];
                        int v = 1;
                        for (int level = 0; level < D; ++level) {
                            const float xs = sz_mid(lo, hi);
                            if (g.req_bail[base + v - 1]) { bail = true; break; }
                            const float y = g.req_out[base + v - 1].x;
                            g.xs[k] = xs;
                            if (within_tolerance(y, target, 1e-6f)) { searching = false; break; }
                            const float pmin = lo, pmax = hi;
                            if ((inc && target < y) || (!inc && target > y)) { hi = xs; v = 2 * v; }
                            else { lo = xs; v = 2 * v + 1; }
                            ++it;
                            // fixed point of the float32 interval: the remaining iterations repeat this solve
                            if ((lo == pmin && hi == pmax) || it >= 100) { searching = false; break; }
                        }
                        if (bail) break;
                        g.iter[k] = (uint8_t)it;
                        g.xmin[k] = lo;
                        g.xmax[k] = hi;
                    }
                    if (!searching) st = SZ2_DONE;
                }
                g.sst[k] = (uint8_t)st;
                if (st == SZ2_DONE) {
                    if (g.ind[k] < 0) { nil = true; break; }  // "target is below the bounded region"
                } else {
                    emit_n[w] = M + (emit_ends[w] ? 2 : 0);
                    emit_lo[w] = lo;
                    emit_hi[w] = hi;
                    all_done = false;
                }
            }
            if (bail) ph = PH_BAIL;
            else if (nil) ph = PH_NIL;
            else if (all_done) {
                // queueanalyzer.go:231-241: lambda = min(lambdaStarTTFT, lambdaStarITL, lambdaStarTPS)
                const float lmax = __fdiv_rn(rmax, 1000.0f);
                float l_tps = lmax;
                if (f.srv_slo_tps[s] > 0.0f) l_tps = __fmul_rn(lmax, __fsub_rn(1.0f, 0.1f));
                const float lambda = go_minf(go_minf(g.xs[2 * j], g.xs[2 * j + 1]), l_tps);
                const float rate = __fmul_rn(lambda, 1000.0f);
                if (rate <= 0.0f || rate > rmax) ph = PH_NIL;  // Analyze: :135-143
                else { an_kind = 2; an_lambda = __fdiv_rn(rate, 1000.0f); ph = PH_WAIT_STAR; }
            }
            if (ph != PH_SEARCH) emit_n[0] = emit_n[1] = 0;
        } else if (ph == PH_WAIT_STAR) {
            const int slot = g.aslot[j];
            if (g.req_bail[slot]) ph = PH_BAIL;
            else if (STAR) {
                g.rate_star[j] = g.req_out[slot].x;  // metrics.Throughput
                ph = PH_DONE;
            } else {
                const float rate_star = g.req_out[slot].x;  // metrics.Throughput
                const float total_rate = total_rate_of(f, s);  // allocation.go:134-141
                long long nrep = go_f64_to_int(ceil(__ddiv_rn((double)total_rate, (double)rate_star)));
                const long long min_rep = f.srv_min_replicas[s];
                if (nrep < min_rep) nrep = min_rep;
                const long long total = (long long)num_instances(f, f.srv_model[s], a) * nrep;
                g.rate_star[j] = rate_star;
                g.nrep[j] = nrep;
                g.cost[j] = __fmul_rn(f.acc_cost[a], (float)total);
                const float rate = __fdiv_rn(total_rate, (float)nrep);  // :148-153
                if (rate <= 0.0f || rate > rmax) ph = PH_NIL;
                else { an_kind = 3; an_lambda = __fdiv_rn(rate, 1000.0f); ph = PH_WAIT_FINAL; }
            }
        } else {  // PH_WAIT_FINAL
            const int slot = g.aslot[j];
            if (g.req_bail[slot]) ph = PH_BAIL;
            else {
                const float4 m = g.req_out[slot];
                Cand c = cand_nil();
                c.feasible = 1;
                c.acc = a;
                c.replicas = (int)g.nrep[j];
                c.batch = g.cand_N[j];
                c.cost = g.cost[j];
                c.value = c.cost;
                c.itl = m.z;
                c.ttft = m.y;
                c.rho = m.w;
                c.max_rate = __fdiv_rn(g.rate_star[j], 1000.0f);
                store_cand(g.cand, pair, c);
                ph = PH_DONE;
            }
        }
        if (!STAR) {
            if (ph == PH_NIL) store_cand(g.cand, pair, cand_nil());
            if (ph == PH_BAIL) {
                const int k = atomicAdd(g.fb_count, 1);
                if (k < g.fb_cap) g.fb_list[k] = j;
                store_cand(g.cand, pair, cand_nil());
            }
        }
        g.phase[j] = (uint8_t)ph;
    }
    // ---- consecutive request slots per thread: warp scan of the counts, one atomic per warp ----
    const int mine = emit_n[0] + emit_n[1] + (an_kind >= 0 ? 1 : 0);
    int incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    const int warp_total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned warp_base = 0;
    if (lane == 31 && warp_total > 0) warp_base = atomicAdd(g.n_req, (unsigned)warp_total);
    warp_base = __shfl_sync(0xffffffffu, warp_base, 31);
    const unsigned live_now = __ballot_sync(0xffffffffu, ph < PH_DONE);
    if (lane == 0 && live_now) atomicAdd(g.n_live, (unsigned)__popc(live_now));
    if (mine == 0) return;
    unsigned slot = warp_base + (unsigned)(incl - mine);
    const int N = g.cand_N[j], K = N + N * f.ratio;
    const long long off = g.tab_off[j];
    const float l2s0 = g.l2s0[j], l2sN = g.l2sN[j], lsN = g.lsN[j];
    auto put = [&](int kind, float lambda) {
        g.req_id[slot] = (unsigned)j * 4u + (unsigned)kind;
        g.req_lam[slot] = lambda;
        g.req_key[slot] = (uint8_t)length_class(estimate_len(g.tab + 4 * off, g.ls + off + j, N, K, lambda, log2f(lambda),
                                                             l2s0, l2sN, lsN));
        ++slot;
    };
    for (int w = 0; w < 2; ++w) {
        if (emit_n[w] == 0) continue;
        g.slot[2 * j + w] = (int)slot;
        if (emit_ends[w]) {
            put(w, emit_lo[w]);
            put(w, emit_hi[w]);
        }
        for (int v = 1; v <= M; ++v) put(w, sz_node_value(v, emit_lo[w], emit_hi[w]));
    }
    if (an_kind >= 0) {
        g.aslot[j] = (int)slot;
        put(an_kind, an_lambda);
    }
}

// Local counting sort of this round's requests by length class (keys precomputed by sz2_advance); stable inside a
// warp's 32 requests, so the requests of one candidate (consecutive slots) stay adjacent within their class.
__global__ void __launch_bounds__(kSortThreads) sz2_sort_local(Sz2Args g) {
    __shared__ uint8_t keys[kSortChunk];
    __shared__ uint8_t sorted_keys[kSortChunk];
    __shared__ unsigned hist[kClasses];
    __shared__ unsigned cursor[kClasses];
    __shared__ unsigned item_base;
    const unsigned n_req = *g.n_req;
    const unsigned base = blockIdx.x * kSortChunk;
    if (base >= n_req) return;
    if (threadIdx.x < kClasses) hist[threadIdx.x] = 0;
    __syncthreads();
    const int n_here = (int)min((unsigned)kSortChunk, n_req - base);
    for (int k = threadIdx.x; k < n_here; k += kSortThreads) {
        const int key = g.req_key[base + k];
        keys[k] = (uint8_t)key;
        agg_inc(hist, key);
    }
    __syncthreads();
    if (threadIdx.x < 32) {
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
    // one warp pass at a time in request order (warp w takes requests 32 w .. 32 w + 31 of each stripe): a
    // candidate's requests keep their relative order inside a class
    for (int k0 = 0; k0 < n_here; k0 += kSortThreads) {
        const int k = k0 + threadIdx.x;
        if (k < n_here) {
            const int key = keys[k];
            const unsigned pos = agg_inc(cursor, key);
            g.ws.order[base + pos] = base + k;
            sorted_keys[pos] = (uint8_t)key;
        }
    }
    const int n_items = (n_here + 31) >> 5;
    if (threadIdx.x == 0) item_base = atomicAdd(g.ws.item_count, (unsigned)n_items);
    __syncthreads();
    for (int w = threadIdx.x; w < n_items; w += kSortThreads) {
        const unsigned cnt = (unsigned)min(32, n_here - 32 * w);
        const int cls = sorted_keys[32 * w];
        g.ws.items[item_base + w] = (unsigned long long)(base + 32 * w) | ((unsigned long long)cnt << 32) |
                                    ((unsigned long long)cls << 40);
        agg_inc(g.ws.item_count + 1, cls);
    }
}

// One request per lane, 32 requests of similar chain length per warp.
template <int REV>
__global__ void __launch_bounds__(256, 4) sz2_solve(Sz2Args g) {
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned w = idx >> 5, lane = idx & 31;
    if (w >= *g.ws.item_count) return;
    const unsigned long long item = g.ws.items_sorted[w];
    if (lane >= (unsigned)((item >> 32) & 0xff)) return;
    const unsigned slot = g.ws.order[(unsigned)item + lane];
    const unsigned id = g.req_id[slot];
    const int j = (int)(id >> 2), kind = (int)(id & 3);
    const DevFleet& f = g.f;
    const int pair = g.cand_pair[j];
    const int N = g.cand_N[j], K = N + N * f.ratio;
    const float lambda = g.req_lam[slot];
    ModelStats st;
    const long long t0 = g.dbg ? clock64() : 0;
    const int rc = solve_private<REV>(g.tab + 4 * g.tab_off[j], N, K, lambda, st);
    if (g.dbg) {
        g.dbg[4 * slot] = (unsigned)(clock64() - t0);
        g.dbg[4 * slot + 1] = (unsigned)N | ((unsigned)kind << 16);
        g.dbg[4 * slot + 2] = __float_as_uint(lambda);
        g.dbg[4 * slot + 3] = w;
    }
    g.req_bail[slot] = rc != kSolveOk;
    if (rc != kSolveOk) return;
    const QParams q = qparams_of(f, pair / f.A, pair % f.A);
    float4 out;
    if (kind <= 1) {  // EvalTTFT / EvalITL: queueanalyzer.go:270-290
        const float eff = effective_concurrency(q, st.avg_serv_time, N);
        out.x = kind == 0 ? __fadd_rn(st.avg_wait_time, prefill_time(q, eff)) : decode_time(q, eff);
        out.y = out.z = out.w = 0.0f;
    } else {  // Analyze: :152-172
        const Metrics m = metrics_from(q, N, st);
        out = make_float4(m.throughput, m.ttft, m.avg_token_time, m.rho);
    }
    g.req_out[slot] = out;
}

// ---------------------------------------------------------------------------
// wva_resolve_scenarios (DESIGN §3.8): after a STAR run of the rounds, rateStar (or nil / bail) per candidate does not
// depend on the arrival rate; only CreateAllocation's per-load steps and its final Analyze do.  sz2_expand applies the
// steps per (candidate, scenario) and emits one kind-3 request per survivor, sz2_sort_local / ws_items_* / sz2_solve
// run that round unchanged, and sz2_consume writes the records into the scenario's block.
// ---------------------------------------------------------------------------
struct LoadStep {
    long long nrep;
    float cost, rate;
};
// allocation.go:134-153 with the arrival column of f (the expressions of sz2_advance's PH_WAIT_STAR)
__device__ __forceinline__ LoadStep load_step(const DevFleet& f, int s, int a, float rate_star) {
    LoadStep r;
    const float total_rate = total_rate_of(f, s);
    r.nrep = go_f64_to_int(ceil(__ddiv_rn((double)total_rate, (double)rate_star)));
    const long long min_rep = f.srv_min_replicas[s];
    if (r.nrep < min_rep) r.nrep = min_rep;
    const long long total = (long long)num_instances(f, f.srv_model[s], a) * r.nrep;
    r.cost = __fmul_rn(f.acc_cost[a], (float)total);
    r.rate = __fdiv_rn(total_rate, (float)r.nrep);
    return r;
}

// One thread per (candidate j, scenario l), t = j * n_scen + l: a candidate's requests take consecutive slots.
__global__ void __launch_bounds__(256) sz2_expand(Sz2Args g) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int L = g.n_scen;
    int j = 0, l = 0;
    bool emit = false;
    float lambda = 0.0f;
    if (t < (long long)g.n_cand * L) {
        j = (int)(t / L);
        l = (int)(t - (long long)j * L);
        DevFleet f = g.f;
        f.srv_arrival_rpm = g.scen_rpm + (size_t)l * f.S;
        const int pair = g.cand_pair[j], s = pair / f.A, a = pair % f.A;
        if (pair_class(f, s, a, true) == PAIR_LOAD) {  // otherwise trivial_kernel owns the record
            const int ph = g.phase[j];
            if (ph == PH_DONE) {
                const LoadStep st = load_step(f, s, a, g.rate_star[j]);
                if (!(st.rate <= 0.0f || st.rate > g.rmax[j])) {  // Analyze: queueanalyzer.go:135-143
                    emit = true;
                    lambda = __fdiv_rn(st.rate, 1000.0f);
                }
            } else if (ph == PH_BAIL) {
                const int k = atomicAdd(g.fb_count, 1);
                if (k < g.fb_cap) g.fb_list[k] = (int)t;
            }
            if (!emit) store_cand(g.cand, (size_t)l * f.S * f.A + pair, cand_nil());
        }
    }
    const int mine = emit ? 1 : 0;
    int incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    const int warp_total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned warp_base = 0;
    if (lane == 31 && warp_total > 0) warp_base = atomicAdd(g.n_req, (unsigned)warp_total);
    warp_base = __shfl_sync(0xffffffffu, warp_base, 31);
    if (!emit) return;
    const unsigned slot = warp_base + (unsigned)(incl - mine);
    const int N = g.cand_N[j], K = N + N * g.f.ratio;
    const long long off = g.tab_off[j];
    g.req_id[slot] = (unsigned)j * 4u + 3u;
    g.req_scen[slot] = l;
    g.req_lam[slot] = lambda;
    g.req_key[slot] = (uint8_t)length_class(estimate_len(g.tab + 4 * off, g.ls + off + j, N, K, lambda, log2f(lambda),
                                                         g.l2s0[j], g.l2sN[j], g.lsN[j]));
}

// One thread per request of sz2_expand's round: the record of PH_WAIT_FINAL, or a stored-vector fallback entry.
__global__ void __launch_bounds__(256) sz2_consume(Sz2Args g) {
    const unsigned slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= *g.n_req) return;
    const int j = (int)(g.req_id[slot] >> 2), l = g.req_scen[slot];
    DevFleet f = g.f;
    f.srv_arrival_rpm = g.scen_rpm + (size_t)l * f.S;
    const int pair = g.cand_pair[j], s = pair / f.A, a = pair % f.A;
    const size_t out = (size_t)l * f.S * f.A + pair;
    if (g.req_bail[slot]) {
        const int k = atomicAdd(g.fb_count, 1);
        if (k < g.fb_cap) g.fb_list[k] = j * g.n_scen + l;
        store_cand(g.cand, out, cand_nil());
        return;
    }
    const LoadStep st = load_step(f, s, a, g.rate_star[j]);
    const float4 m = g.req_out[slot];
    Cand c = cand_nil();
    c.feasible = 1;
    c.acc = a;
    c.replicas = (int)st.nrep;
    c.batch = g.cand_N[j];
    c.cost = st.cost;
    c.value = c.cost;
    c.itl = m.z;
    c.ttft = m.y;
    c.rho = m.w;
    c.max_rate = __fdiv_rn(g.rate_star[j], 1000.0f);
    store_cand(g.cand, out, c);
}

// ---------------------------------------------------------------------------
// Small fleets (BASELINE configs[0]: one VariantAutoscaling = one candidate): ONE warp per candidate runs the whole
// CreateAllocation in one launch — the same speculative midpoint trees, but evaluated by the warp's lanes (round one:
// the two end points + 15 midpoints = 4 iterations; later rounds: 31 midpoints = 5 iterations) and walked in
// registers with warp shuffles.  No rounds, no sort, no host round trip: a reconcile of a handful of variants is
// three launches (trivial, this, unlimited argmin) instead of sixty.  Same lambdas, same solves, same comparisons
// as the round-based path and the reference.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float sz_eval(const QParams& q, int which, const double* tab, int N, int K, float x, int& bail) {
    ModelStats st;
    if (solve_shared(tab, N, K, x, st) != kSolveOk) { bail = 1; return 0.0f; }
    const float eff = effective_concurrency(q, st.avg_serv_time, N);  // queueanalyzer.go:270-290
    return which == 0 ? __fadd_rn(st.avg_wait_time, prefill_time(q, eff)) : decode_time(q, eff);
}
__global__ void __launch_bounds__(128) size_warp_kernel(SizeArgs g, const double* __restrict__ tabs,
                                                        const long long* __restrict__ tab_off) {
    const int j = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (j >= g.n_cand) return;
    const DevFleet& f = g.f;
    const int pair = g.cand_pair[j], s = pair / f.A, a = pair % f.A;
    const int N = g.cand_N[j], K = N + N * f.ratio;
    const double* tab = tabs + 4 * tab_off[j];
    const QParams q = qparams_of(f, s, a);
    const float rmin = rate_min_of((float)tab[0]), rmax = rate_max_of((float)tab[4 * (N - 1)]);
    const float slo_ttft = f.srv_slo_ttft[s], slo_itl = f.srv_slo_itl[s], slo_tps = f.srv_slo_tps[s];
    bool nil = K < 2 || slo_itl < 0.0f || slo_ttft < 0.0f || slo_tps < 0.0f;  // queuemodel.go:31, TargetPerf.check
    bool bail = false;
    const float lmin = __fdiv_rn(rmin, 1000.0f), lmax = __fdiv_rn(rmax, 1000.0f);
    float xstar[2] = {lmax, lmax};  // lambdaStar when a target is disabled (queueanalyzer.go:205,218)
    for (int w = 0; w < 2 && !nil && !bail; ++w) {
        const float target = w == 0 ? slo_ttft : slo_itl;
        if (!(target > 0.0f)) continue;
        float lo = lmin, hi = lmax;
        if (lo > hi) { nil = true; break; }  // utils.go:29-31
        bool first = true, searching = true, inc = false;
        int it = 0, ind = 0;
        float xs = 0.0f;
        while (searching && !bail) {
            // this lane's evaluation point: round one = {xmin, xmax, nodes 1..15}, later rounds = nodes 1..31
            const int D = first ? 4 : 5;
            const int v_mine = first ? lane - 1 : lane + 1;
            const bool has = first ? lane < 17 : lane < 31;
            float x = lo;
            if (first && lane == 1) x = hi;
            if (has && !(first && lane < 2)) x = sz_node_value(v_mine, lo, hi);
            float y = 0.0f;
            int b = 0;
            if (has) y = sz_eval(q, w, tab, N, K, x, b);
            __syncwarp();
            if (first) {  // utils.go:36-51: the two boundary evaluations
                const float y0 = __shfl_sync(0xffffffffu, y, 0), y1 = __shfl_sync(0xffffffffu, y, 1);
                const int b0 = __shfl_sync(0xffffffffu, b, 0), b1 = __shfl_sync(0xffffffffu, b, 1);
                if (b0) { bail = true; break; }
                if (within_tolerance(y0, target, 1e-6f)) { xs = lo; searching = false; }
                else {
                    if (b1) { bail = true; break; }
                    if (within_tolerance(y1, target, 1e-6f)) { xs = hi; searching = false; }
                    else {
                        inc = y0 < y1;
                        if ((inc && target < y0) || (!inc && target > y0)) { xs = lo; ind = -1; searching = false; }
                        else if ((inc && target > y1) || (!inc && target < y1)) { xs = hi; ind = 1; searching = false; }
                    }
                }
            }
            if (searching) {  // utils.go:54-68, D iterations over the evaluated tree
                int v = 1;
                for (int level = 0; level < D; ++level) {
                    const int src = first ? v + 1 : v - 1;  // the lane that evaluated node v
                    const float yv = __shfl_sync(0xffffffffu, y, src);
                    const int bv = __shfl_sync(0xffffffffu, b, src);
                    xs = sz_mid(lo, hi);
                    if (bv) { bail = true; break; }
                    if (within_tolerance(yv, target, 1e-6f)) { searching = false; break; }
                    const float pmin = lo, pmax = hi;
                    if ((inc && target < yv) || (!inc && target > yv)) { hi = xs; v = 2 * v; }
                    else { lo = xs; v = 2 * v + 1; }
                    ++it;
                    if ((lo == pmin && hi == pmax) || it >= 100) { searching = false; break; }
                }
            }
            first = false;
        }
        xstar[w] = xs;
        if (ind < 0) nil = true;  // "target is below the bounded region"
    }
    Cand out = cand_nil();
    if (!nil && !bail) {
        // queueanalyzer.go:231-241, allocation.go:134-163 — every lane computes the same values
        float l_tps = lmax;
        if (slo_tps > 0.0f) l_tps = __fmul_rn(lmax, __fsub_rn(1.0f, 0.1f));
        const float lambda = go_minf(go_minf(xstar[0], xstar[1]), l_tps);
        const float rate0 = __fmul_rn(lambda, 1000.0f);
        ModelStats st;
        if (rate0 <= 0.0f || rate0 > rmax) nil = true;
        else if (solve_shared(tab, N, K, __fdiv_rn(rate0, 1000.0f), st) != kSolveOk) bail = true;
        else {
            const float rate_star = metrics_from(q, N, st).throughput;
            const float total_rate = total_rate_of(f, s);
            long long nrep = go_f64_to_int(ceil(__ddiv_rn((double)total_rate, (double)rate_star)));
            const long long min_rep = f.srv_min_replicas[s];
            if (nrep < min_rep) nrep = min_rep;
            const long long total = (long long)num_instances(f, f.srv_model[s], a) * nrep;
            const float cost = __fmul_rn(f.acc_cost[a], (float)total);
            const float rate = __fdiv_rn(total_rate, (float)nrep);
            if (rate <= 0.0f || rate > rmax) nil = true;
            else if (solve_shared(tab, N, K, __fdiv_rn(rate, 1000.0f), st) != kSolveOk) bail = true;
            else {
                const Metrics m = metrics_from(q, N, st);
                out.feasible = 1;
                out.acc = a;
                out.replicas = (int)nrep;
                out.batch = N;
                out.cost = cost;
                out.value = cost;
                out.itl = m.avg_token_time;
                out.ttft = m.ttft;
                out.rho = m.rho;
                out.max_rate = __fdiv_rn(rate_star, 1000.0f);
            }
        }
    }
    if (lane == 0) {
        if (bail) {
            const int k = atomicAdd(g.fb_count, 1);
            if (k < g.fb_cap) g.fb_list[k] = j;
            out = cand_nil();
        }
        store_cand(g.cand, pair, out);
    }
}

// Per-round reset of the device counters (one tiny kernel instead of two memsets; part of the captured round).
__global__ void sz2_round_reset(Sz2Args g) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        *g.n_req = 0;
        *g.n_live = 0;
    }
    if (i < 2 * kClasses + 1) g.ws.item_count[i] = 0;
}

}  // namespace wva
