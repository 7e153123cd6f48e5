// wva_b200.cu — host engine + C ABI (include/wva_b200.h) over the sm_100a kernels.
//
// Host-side mirror of pkg/core.System / pkg/manager.Manager for the hot path: the fleet
// is packed once into a single device arena (one H2D copy), derived work lists
// (candidates ordered by queue size, shared service-rate tables) are cached on the
// handle, every call enqueues its kernels on the handle's stream and ends with one D2H
// copy of the result block.  There is no CPU compute fallback: without a CUDA device
// wva_create fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/wva_b200.h"
#include "wva_kernels.cuh"
#include "wva_size.cuh"

using namespace wva;

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};
struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Host copy of the fleet columns (the caller's pointers are never retained).
struct HostFleet {
    int A = 0, T = 0, M = 0, S = 0;
    std::vector<float> acc_cost;
    std::vector<int32_t> acc_mult, acc_type, type_capacity;
    std::vector<uint8_t> perf_present;
    std::vector<float> perf_alpha, perf_beta, perf_gamma, perf_delta;
    std::vector<int32_t> perf_acc_count, perf_max_batch, perf_at_tokens;
    std::vector<int32_t> srv_model, srv_priority;
    std::vector<uint8_t> srv_has_target;
    std::vector<float> srv_slo_itl, srv_slo_ttft, srv_slo_tps;
    std::vector<uint8_t> srv_keep_acc;
    std::vector<int32_t> srv_min_replicas, srv_max_batch;
    std::vector<float> srv_arrival_rpm;
    std::vector<int32_t> srv_in_tokens, srv_out_tokens, srv_cur_acc, srv_cur_replicas;
    std::vector<float> srv_cur_cost;
    bool unlimited = true, delayed_best_effort = false;
    int saturation_policy = 0;
    wva_tunables tun{10, 0.1f};

    // the gates of pair_class that do not read the arrival rate
    bool rate_free_gates(int s, int a, bool honour_keep) const {
        if (honour_keep && srv_keep_acc[s] && srv_cur_acc[s] != WVA_ACC_NONE && srv_cur_acc[s] != a) return false;
        if (srv_in_tokens[s] < 0 || srv_out_tokens[s] < 0) return false;
        const int m = srv_model[s];
        if (m < 0 || m >= M) return false;
        if (!perf_present[(size_t)m * A + a]) return false;
        return srv_has_target[s] != 0;
    }
    // gates of CreateAllocation + candidate rule (mirrors pair_class on the device)
    int pair_class(int s, int a, bool honour_keep) const {
        if (srv_arrival_rpm[s] < 0.0f || !rate_free_gates(s, a, honour_keep)) return 0;
        if (srv_arrival_rpm[s] == 0.0f || srv_out_tokens[s] == 0) return PAIR_ZERO;
        return PAIR_LOAD;
    }
    // batch size of a candidate: pkg/core/allocation.go:77-87
    int pair_batch(int s, int a) const {
        if (srv_max_batch[s] > 0) return srv_max_batch[s];
        const size_t k = (size_t)srv_model[s] * A + a;
        const long long t = (long long)perf_max_batch[k] * (long long)perf_at_tokens[k] / srv_out_tokens[s];
        return (int)std::max<long long>(t, 1);
    }
};

struct Column {
    size_t off, bytes;
};

}  // namespace

struct wva_handle {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr, ev_d0 = nullptr, ev_d1 = nullptr;
    std::string err;
    int64_t launches = 0;
    float last_kernel_ms = 0.f, last_device_ms = 0.f;

    // resident fleet
    bool resident = false;
    HostFleet hf;
    DevBuf arena;
    PinBuf stage;
    DevFleet df{};
    Column col_rate{}, col_in{}, col_out{};
    uint64_t epoch_tokens = 0;  // bumped when service-rate tables become stale

    // size path caches
    uint64_t size_epoch = ~0ull;
    std::vector<int> cand_pair, cand_N;
    int size_Nmax = 0;
    DevBuf d_cand_pair, d_cand_N;
    DevBuf d_sz_tab, d_sz_ls, d_sz_off, d_sz_state, d_sz_req, d_sz_sort;
    PinBuf sz_pin;
    // wva_resolve_scenarios: its own candidate list and tables (the list can differ from the size path's), cached
    // while the token statistics and the set of servers loaded in some scenario stay the same
    uint64_t scen_epoch = ~0ull;
    std::vector<uint8_t> scen_loaded;
    std::vector<int> scen_pair, scen_N;
    int scen_Nmax = 0;
    DevBuf d_scen_pair, d_scen_N, d_scen_tab, d_scen_ls, d_scen_off, d_scen_rpm;

    // grid path caches
    uint64_t grid_epoch = ~0ull;
    std::vector<int> grid_batch, grid_replicas;
    int grid_Bmax = 0, grid_n_tab = 0;
    DevBuf d_grid_lists, d_pair_tab, d_tab_pair, d_tab_off, d_tab_len, d_tab, d_ls, d_sort, d_best, d_pb, d_rows;
    // shared
    DevBuf d_cand_block, d_win_block, d_ctrl, d_fb_list, d_scratch, d_cells, d_sweep, d_dbg;
    // peer exchange of the winner block (multi-GPU, one process per GPU on one node)
    struct Xchg {
        int world = 0, rank = 0;
        size_t block_bytes = 0, slot_stride = 0;   // one gathered buffer = world * slot_stride bytes
        char* local = nullptr;                     // [2 parities][world slots] + flags, cudaMalloc'ed here
        size_t local_bytes = 0, flags_off = 0;
        std::vector<char*> peer;                   // base pointers of every rank's buffer (peer[rank] == local)
        char** d_peer = nullptr;
        unsigned long long epoch = 0;
        int* d_err = nullptr;
    } xchg;
    // the most recent solution (for wva_summarize): 0 none, 1 winner block on the device, 2 host copy (greedy)
    int last_kind = 0;
    std::vector<int32_t> last_acc, last_replicas;
    std::vector<float> last_cost;
    std::vector<uint8_t> last_feasible;
    DevBuf d_summary;
    bool dbg_cycles = false;
    const unsigned* dbg_plan = nullptr;
    size_t dbg_n = 0;
    const int* dbg_row_j = nullptr;  // row_j / row_res of the last grid solve (wva_dbg_read_rows)
    const uint8_t* dbg_row_res = nullptr;
    size_t dbg_rows_n = 0;
    int dbg_fb_count = 0;  // solves of the last call that took the stored-vector fallback (wva_dbg_fallback_count)
    PinBuf out_stage;

    int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
        err = what;
        if (e != cudaSuccess) {
            err += ": ";
            err += cudaGetErrorString(e);
        }
        return code;
    }
};

#define CK(call)                                                              \
    do {                                                                      \
        cudaError_t _e = (call);                                              \
        if (_e != cudaSuccess) return h->fail(WVA_ERR_CUDA, #call, _e);       \
    } while (0)

namespace {


// control block on the device: a handful of ints
enum { CTRL_COUNTER = 0, CTRL_FB_COUNT = 1, CTRL_FB_STATUS = 2, CTRL_INTS = 8 };

// ---- SoA result blocks -------------------------------------------------------
struct Block {
    size_t off_feasible, off_acc, off_replicas, off_batch, off_cost, off_value, off_itl, off_ttft, off_rho, off_rate;
    size_t bytes;
    size_t n;
};
Block block_layout(size_t n) {
    Block b;
    size_t o = 0;
    b.n = n;
    b.off_feasible = o; o = align_up(o + n, 16);
    b.off_acc = o; o = align_up(o + 4 * n, 16);
    b.off_replicas = o; o = align_up(o + 4 * n, 16);
    b.off_batch = o; o = align_up(o + 4 * n, 16);
    b.off_cost = o; o = align_up(o + 4 * n, 16);
    b.off_value = o; o = align_up(o + 4 * n, 16);
    b.off_itl = o; o = align_up(o + 4 * n, 16);
    b.off_ttft = o; o = align_up(o + 4 * n, 16);
    b.off_rho = o; o = align_up(o + 4 * n, 16);
    b.off_rate = o; o = align_up(o + 4 * n, 16);
    b.bytes = o;
    return b;
}
AllocCols block_cols(void* base, const Block& b) {
    char* p = (char*)base;
    AllocCols c;
    c.feasible = (uint8_t*)(p + b.off_feasible);
    c.acc = (int*)(p + b.off_acc);
    c.replicas = (int*)(p + b.off_replicas);
    c.batch = (int*)(p + b.off_batch);
    c.cost = (float*)(p + b.off_cost);
    c.value = (float*)(p + b.off_value);
    c.itl = (float*)(p + b.off_itl);
    c.ttft = (float*)(p + b.off_ttft);
    c.rho = (float*)(p + b.off_rho);
    c.max_rate = (float*)(p + b.off_rate);
    return c;
}
void scatter_block(const void* host_block, const Block& b, const wva_allocs* out) {
    if (!out) return;
    const char* p = (const char*)host_block;
    const size_t n = b.n;
    if (out->feasible) memcpy(out->feasible, p + b.off_feasible, n);
    if (out->acc) memcpy(out->acc, p + b.off_acc, 4 * n);
    if (out->replicas) memcpy(out->replicas, p + b.off_replicas, 4 * n);
    if (out->batch) memcpy(out->batch, p + b.off_batch, 4 * n);
    if (out->cost) memcpy(out->cost, p + b.off_cost, 4 * n);
    if (out->value) memcpy(out->value, p + b.off_value, 4 * n);
    if (out->itl) memcpy(out->itl, p + b.off_itl, 4 * n);
    if (out->ttft) memcpy(out->ttft, p + b.off_ttft, 4 * n);
    if (out->rho) memcpy(out->rho, p + b.off_rho, 4 * n);
    if (out->max_rate) memcpy(out->max_rate, p + b.off_rate, 4 * n);
}
AllocCols cols_from_abi(const wva_allocs* a) {
    AllocCols c{};
    if (!a) return c;
    c.feasible = a->feasible; c.acc = a->acc; c.replicas = a->replicas; c.batch = a->batch;
    c.cost = a->cost; c.value = a->value; c.itl = a->itl; c.ttft = a->ttft; c.rho = a->rho;
    c.max_rate = a->max_rate;
    return c;
}

// ---- fleet validation + upload ----------------------------------------------
// nullptr when the fleet is well formed, else what is wrong with it
const char* fleet_problem(const wva_fleet* f) {
    if (!f) return "fleet is NULL";
    if (f->n_acc < 0 || f->n_types < 0 || f->n_models < 0 || f->n_servers < 0) return "negative size in fleet";
    const bool need_a = f->n_acc > 0, need_t = f->n_types > 0, need_ma = f->n_models > 0 && f->n_acc > 0,
               need_s = f->n_servers > 0;
    if (need_a && (!f->acc_cost || !f->acc_multiplicity || !f->acc_type)) return "NULL accelerator column";
    if (need_t && !f->type_capacity) return "NULL capacity column";
    if (need_ma && (!f->perf_present || !f->perf_alpha || !f->perf_beta || !f->perf_gamma || !f->perf_delta ||
                    !f->perf_acc_count || !f->perf_max_batch || !f->perf_at_tokens))
        return "NULL perf column";
    if (need_s && (!f->srv_model || !f->srv_priority || !f->srv_has_target || !f->srv_slo_itl || !f->srv_slo_ttft ||
                   !f->srv_slo_tps || !f->srv_keep_acc || !f->srv_min_replicas || !f->srv_max_batch ||
                   !f->srv_arrival_rpm || !f->srv_in_tokens || !f->srv_out_tokens || !f->srv_cur_acc ||
                   !f->srv_cur_replicas || !f->srv_cur_cost))
        return "NULL server column";
    for (int a = 0; a < f->n_acc; ++a)
        if (f->n_types > 0 && (f->acc_type[a] < 0 || f->acc_type[a] >= f->n_types)) return "accelerator type id out of range";
    if (f->tun.max_queue_to_batch_ratio < 0) return "negative queue ratio";
    return nullptr;
}
int validate_fleet(wva_handle* h, const wva_fleet* f) {
    if (const char* what = fleet_problem(f)) return h->fail(WVA_ERR_BAD_ARG, what);
    return WVA_OK;
}

template <class T>
void copy_col(std::vector<T>& dst, const T* src, size_t n) {
    dst.assign(src, src + n);
}

template <class T>
Column place(std::vector<std::pair<Column, const void*>>& plan, size_t& off, const std::vector<T>& v) {
    Column c{off, v.size() * sizeof(T)};
    plan.push_back({c, v.data()});
    off = align_up(off + std::max<size_t>(c.bytes, 1));
    return c;
}

// Host copy of every column (the caller's pointers are never retained).
void fill_host_fleet(HostFleet& hf, const wva_fleet* f) {
    const size_t A = f->n_acc, T = f->n_types, M = f->n_models, S = f->n_servers;
    hf.A = (int)A; hf.T = (int)T; hf.M = (int)M; hf.S = (int)S;
    copy_col(hf.acc_cost, f->acc_cost, A);
    copy_col(hf.acc_mult, f->acc_multiplicity, A);
    copy_col(hf.acc_type, f->acc_type, A);
    copy_col(hf.type_capacity, f->type_capacity, T);
    copy_col(hf.perf_present, f->perf_present, M * A);
    copy_col(hf.perf_alpha, f->perf_alpha, M * A);
    copy_col(hf.perf_beta, f->perf_beta, M * A);
    copy_col(hf.perf_gamma, f->perf_gamma, M * A);
    copy_col(hf.perf_delta, f->perf_delta, M * A);
    copy_col(hf.perf_acc_count, f->perf_acc_count, M * A);
    copy_col(hf.perf_max_batch, f->perf_max_batch, M * A);
    copy_col(hf.perf_at_tokens, f->perf_at_tokens, M * A);
    copy_col(hf.srv_model, f->srv_model, S);
    copy_col(hf.srv_priority, f->srv_priority, S);
    copy_col(hf.srv_has_target, f->srv_has_target, S);
    copy_col(hf.srv_slo_itl, f->srv_slo_itl, S);
    copy_col(hf.srv_slo_ttft, f->srv_slo_ttft, S);
    copy_col(hf.srv_slo_tps, f->srv_slo_tps, S);
    copy_col(hf.srv_keep_acc, f->srv_keep_acc, S);
    copy_col(hf.srv_min_replicas, f->srv_min_replicas, S);
    copy_col(hf.srv_max_batch, f->srv_max_batch, S);
    copy_col(hf.srv_arrival_rpm, f->srv_arrival_rpm, S);
    copy_col(hf.srv_in_tokens, f->srv_in_tokens, S);
    copy_col(hf.srv_out_tokens, f->srv_out_tokens, S);
    copy_col(hf.srv_cur_acc, f->srv_cur_acc, S);
    copy_col(hf.srv_cur_replicas, f->srv_cur_replicas, S);
    copy_col(hf.srv_cur_cost, f->srv_cur_cost, S);
    hf.unlimited = f->unlimited != 0;
    hf.delayed_best_effort = f->delayed_best_effort != 0;
    hf.saturation_policy = f->saturation_policy;
    hf.tun = f->tun;
}

int upload_fleet(wva_handle* h, const wva_fleet* f) {
    int rc = validate_fleet(h, f);
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));  // the pinned stage may still feed an earlier async copy
    HostFleet& hf = h->hf;
    fill_host_fleet(hf, f);

    // one arena, one H2D copy; the three load columns are adjacent so that
    // wva_update_load moves a single contiguous range
    std::vector<std::pair<Column, const void*>> plan;
    size_t off = 0;
    Column c_rate = place(plan, off, hf.srv_arrival_rpm);
    Column c_in = place(plan, off, hf.srv_in_tokens);
    Column c_out = place(plan, off, hf.srv_out_tokens);
    Column c_acc_cost = place(plan, off, hf.acc_cost);
    Column c_acc_mult = place(plan, off, hf.acc_mult);
    Column c_acc_type = place(plan, off, hf.acc_type);
    Column c_cap = place(plan, off, hf.type_capacity);
    Column c_pp = place(plan, off, hf.perf_present);
    Column c_pa = place(plan, off, hf.perf_alpha);
    Column c_pb = place(plan, off, hf.perf_beta);
    Column c_pg = place(plan, off, hf.perf_gamma);
    Column c_pd = place(plan, off, hf.perf_delta);
    Column c_pc = place(plan, off, hf.perf_acc_count);
    Column c_pm = place(plan, off, hf.perf_max_batch);
    Column c_pt = place(plan, off, hf.perf_at_tokens);
    Column c_sm = place(plan, off, hf.srv_model);
    Column c_sp = place(plan, off, hf.srv_priority);
    Column c_st = place(plan, off, hf.srv_has_target);
    Column c_si = place(plan, off, hf.srv_slo_itl);
    Column c_sf = place(plan, off, hf.srv_slo_ttft);
    Column c_ss = place(plan, off, hf.srv_slo_tps);
    Column c_sk = place(plan, off, hf.srv_keep_acc);
    Column c_sn = place(plan, off, hf.srv_min_replicas);
    Column c_sb = place(plan, off, hf.srv_max_batch);
    Column c_ca = place(plan, off, hf.srv_cur_acc);
    Column c_cr = place(plan, off, hf.srv_cur_replicas);
    Column c_cc = place(plan, off, hf.srv_cur_cost);
    const size_t total = off;
    CK(h->arena.ensure(total));
    CK(h->stage.ensure(total));
    for (auto& pr : plan)
        if (pr.first.bytes) memcpy((char*)h->stage.p + pr.first.off, pr.second, pr.first.bytes);
    CK(cudaMemcpyAsync(h->arena.p, h->stage.p, total, cudaMemcpyHostToDevice, h->stream));

    char* d = (char*)h->arena.p;
    DevFleet& df = h->df;
    df.A = hf.A; df.T = hf.T; df.M = hf.M; df.S = hf.S;
    df.acc_cost = (const float*)(d + c_acc_cost.off);
    df.acc_mult = (const int*)(d + c_acc_mult.off);
    df.acc_type = (const int*)(d + c_acc_type.off);
    df.type_capacity = (const int*)(d + c_cap.off);
    df.perf_present = (const uint8_t*)(d + c_pp.off);
    df.perf_alpha = (const float*)(d + c_pa.off);
    df.perf_beta = (const float*)(d + c_pb.off);
    df.perf_gamma = (const float*)(d + c_pg.off);
    df.perf_delta = (const float*)(d + c_pd.off);
    df.perf_acc_count = (const int*)(d + c_pc.off);
    df.perf_max_batch = (const int*)(d + c_pm.off);
    df.perf_at_tokens = (const int*)(d + c_pt.off);
    df.srv_model = (const int*)(d + c_sm.off);
    df.srv_priority = (const int*)(d + c_sp.off);
    df.srv_has_target = (const uint8_t*)(d + c_st.off);
    df.srv_slo_itl = (const float*)(d + c_si.off);
    df.srv_slo_ttft = (const float*)(d + c_sf.off);
    df.srv_slo_tps = (const float*)(d + c_ss.off);
    df.srv_keep_acc = (const uint8_t*)(d + c_sk.off);
    df.srv_min_replicas = (const int*)(d + c_sn.off);
    df.srv_max_batch = (const int*)(d + c_sb.off);
    df.srv_arrival_rpm = (const float*)(d + c_rate.off);
    df.srv_in_tokens = (const int*)(d + c_in.off);
    df.srv_out_tokens = (const int*)(d + c_out.off);
    df.srv_cur_acc = (const int*)(d + c_ca.off);
    df.srv_cur_replicas = (const int*)(d + c_cr.off);
    df.srv_cur_cost = (const float*)(d + c_cc.off);
    df.ratio = hf.tun.max_queue_to_batch_ratio;
    df.penalty = hf.tun.accel_penalty_factor;
    h->col_rate = c_rate; h->col_in = c_in; h->col_out = c_out;
    h->resident = true;
    h->epoch_tokens++;
    h->last_kind = 0;
    return WVA_OK;
}

int ensure_ctrl(wva_handle* h) {
    CK(h->d_ctrl.ensure(CTRL_INTS * sizeof(int)));
    CK(cudaMemsetAsync(h->d_ctrl.p, 0, CTRL_INTS * sizeof(int), h->stream));
    return WVA_OK;
}

// Scratch for the stored-vector fallback kernels: a fixed number of slots.
constexpr int kFbBlocks = 2, kFbThreads = 64, kFbSlots = kFbBlocks * kFbThreads;
int ensure_scratch(wva_handle* h, int Nmax, int ratio, size_t* slot_doubles, int* Kmax) {
    *Kmax = Nmax + Nmax * ratio;
    *slot_doubles = (size_t)*Kmax + 1 + ((size_t)Nmax + 1) / 2 + 1;
    CK(h->d_scratch.ensure(*slot_doubles * sizeof(double) * kFbSlots));
    return WVA_OK;
}

// ---- size path (K1) ---------------------------------------------------------
// Keep a candidate list (pair ids sorted by descending N; Ns indexed by pair id) on the host and the device, and build
// one shared-format service-rate table per candidate (N entries).
int upload_size_list(wva_handle* h, const std::vector<int>& pairs, const std::vector<int>& Ns, std::vector<int>& cand_pair,
                     std::vector<int>& cand_N, int& Nmax, DevBuf& d_pair, DevBuf& d_N, DevBuf& d_off, DevBuf& d_tab,
                     DevBuf& d_ls) {
    const int n = (int)pairs.size();
    cand_pair = pairs;
    cand_N.resize(n);
    for (int j = 0; j < n; ++j) cand_N[j] = Ns[pairs[j]];
    Nmax = n ? cand_N[0] : 1;
    if (n) {
        CK(d_pair.ensure(sizeof(int) * n));
        CK(d_N.ensure(sizeof(int) * n));
        CK(cudaMemcpyAsync(d_pair.p, cand_pair.data(), sizeof(int) * n, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(d_N.p, cand_N.data(), sizeof(int) * n, cudaMemcpyHostToDevice, h->stream));
        // one shared-format service-rate table per candidate (N entries), cached until the token
        // statistics or the fleet change
        std::vector<long long> off(n + 1, 0);
        for (int j = 0; j < n; ++j) off[j + 1] = off[j] + cand_N[j];
        CK(d_off.ensure(sizeof(long long) * (n + 1)));
        CK(d_tab.ensure(sizeof(double) * 4 * (size_t)off[n] + 1024));
        CK(d_ls.ensure(sizeof(float) * ((size_t)off[n] + n + 1)));
        CK(cudaMemcpyAsync(d_off.p, off.data(), sizeof(long long) * (n + 1), cudaMemcpyHostToDevice, h->stream));
        build_pair_tables<<<n, 128, 0, h->stream>>>(h->df, (const int*)d_pair.p, (const long long*)d_off.p,
                                                    (const int*)d_N.p, n, (double*)d_tab.p, (float*)d_ls.p, nullptr, 0,
                                                    nullptr);
        h->launches++;
        CK(cudaGetLastError());
    }
    return WVA_OK;
}

int prepare_size(wva_handle* h) {
    if (h->size_epoch == h->epoch_tokens) return WVA_OK;
    const HostFleet& hf = h->hf;
    const int A = hf.A, S = hf.S;
    std::vector<int> pairs;
    std::vector<int> Ns((size_t)S * A, 0);
    for (int s = 0; s < S; ++s)
        for (int a = 0; a < A; ++a)
            if (hf.pair_class(s, a, true) == PAIR_LOAD) {
                const int N = hf.pair_batch(s, a);
                if (N > (1 << 20)) return h->fail(WVA_ERR_UNSUPPORTED, "batch size above 2^20");
                Ns[(size_t)s * A + a] = N;
                pairs.push_back(s * A + a);
            }
    std::stable_sort(pairs.begin(), pairs.end(), [&](int x, int y) { return Ns[x] > Ns[y]; });
    int rc = upload_size_list(h, pairs, Ns, h->cand_pair, h->cand_N, h->size_Nmax, h->d_cand_pair, h->d_cand_N,
                              h->d_sz_off, h->d_sz_tab, h->d_sz_ls);
    if (rc) return rc;
    h->size_epoch = h->epoch_tokens;
    return WVA_OK;
}

// Round-based K1 with speculative bisection trees: see the comment at the top of wva_size.cuh.
int size_depth_for(int n) {
    int d = n <= 2048 ? 5 : (n <= 8192 ? 4 : (n <= 40000 ? 3 : 2));
    if (const char* e = getenv("WVA_SIZE_DEPTH")) d = atoi(e);
    return std::min(std::max(d, 1), kSzMaxDepth);
}
// `star` (wva_resolve_scenarios): the rounds stop at rateStar (sz2_advance<true>), the request block holds at least
// min_cap slots, and *star receives the rounds' arguments for the scenario round that follows.
int run_size_rounds(wva_handle* h, const SizeArgs& sa, int n, const double* tab, const long long* tab_off,
                    const float* ls, Sz2Args* star = nullptr, size_t min_cap = 0) {
    const int D = size_depth_for(n);
    int size_rev = 1;  // solver returns to the block vote after a per-step excursion (0 = stays on the per-step path)
    if (const char* e = getenv("WVA_SIZE_REV")) size_rev = atoi(e);
    // blocks of sz2_solve per SM (register limit: 4).  Fewer co-resident warps = a larger share of the sub-partition's
    // FP64 pipe for each, i.e. a shorter critical path for the rounds that are as long as their longest chains;
    // unused dynamic shared memory is what limits the residency.
    int solve_bpsm = 4;
    if (const char* e = getenv("WVA_SIZE_BLOCKS_PER_SM")) solve_bpsm = std::min(std::max(atoi(e), 1), 4);
    size_t solve_pad = 0;
    if (solve_bpsm < 4) {
        solve_pad = (size_t)(227 * 1024) / (size_t)solve_bpsm - 2048;
        solve_pad = solve_pad / 1024 * 1024;
        CK(cudaFuncSetAttribute(sz2_solve<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_pad));
        CK(cudaFuncSetAttribute(sz2_solve<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)solve_pad));
    }
    int dbg_round = -1;  // diagnostics: record per-request SM cycles of this round's sz2_solve (wva_dbg_read_size)
    if (const char* e = getenv("WVA_SIZE_DBG_ROUND")) dbg_round = atoi(e);
    const size_t per_cand = 2 * ((size_t)(1 << D) - 1 + 2);  // two searches: a tree each, plus the two end points
    const size_t cap = std::max(per_cand * (size_t)n, min_cap);  // requests per round, worst case
    const size_t n2 = 2 * (size_t)n;
    // state block
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes, 16); return at; };
    const size_t o_xmin = take(4 * n2), o_xmax = take(4 * n2), o_xs = take(4 * n2);
    const size_t o_sst = take(n2), o_inc = take(n2), o_iter = take(n2), o_ind = take(n2), o_slot = take(4 * n2);
    const size_t o_phase = take(n), o_rmax = take(4 * (size_t)n), o_l2s0 = take(4 * (size_t)n), o_l2sN = take(4 * (size_t)n),
                 o_lsN = take(4 * (size_t)n), o_rstar = take(4 * (size_t)n), o_cost = take(4 * (size_t)n),
                 o_nrep = take(8 * (size_t)n), o_aslot = take(4 * (size_t)n);
    CK(h->d_sz_state.ensure(o));
    char* sp = (char*)h->d_sz_state.p;
    // request block
    o = 0;
    const size_t r_id = take(4 * cap), r_lam = take(4 * cap), r_key = take(cap), r_out = take(16 * cap), r_bail = take(cap),
                 r_cnt = take(16);
    const size_t r_scen = star ? take(4 * cap) : 0;
    CK(h->d_sz_req.ensure(o));
    char* rp = (char*)h->d_sz_req.p;
    // sort workspace
    const size_t chunks = (cap + kSortChunk - 1) / kSortChunk;
    const size_t max_items = (cap + 31) / 32 + chunks;
    o = 0;
    const size_t w_order = take(4 * cap), w_items = take(8 * max_items), w_sorted = take(8 * max_items),
                 w_cnt = take(4 * (2 * kClasses + 8));
    CK(h->d_sz_sort.ensure(o));
    char* wp = (char*)h->d_sz_sort.p;
    CK(h->sz_pin.ensure(64));

    Sz2Args g{};
    g.f = sa.f;
    g.cand_pair = sa.cand_pair;
    g.cand_N = sa.cand_N;
    g.n_cand = n;
    g.depth = D;
    g.tab = tab;
    g.tab_off = tab_off;
    g.ls = ls;
    g.xmin = (float*)(sp + o_xmin); g.xmax = (float*)(sp + o_xmax); g.xs = (float*)(sp + o_xs);
    g.sst = (uint8_t*)(sp + o_sst); g.inc = (uint8_t*)(sp + o_inc); g.iter = (uint8_t*)(sp + o_iter);
    g.ind = (int8_t*)(sp + o_ind); g.slot = (int*)(sp + o_slot);
    g.phase = (uint8_t*)(sp + o_phase);
    g.rmax = (float*)(sp + o_rmax); g.l2s0 = (float*)(sp + o_l2s0); g.l2sN = (float*)(sp + o_l2sN); g.lsN = (float*)(sp + o_lsN);
    g.rate_star = (float*)(sp + o_rstar); g.cost = (float*)(sp + o_cost);
    g.nrep = (long long*)(sp + o_nrep);
    g.aslot = (int*)(sp + o_aslot);
    g.req_id = (unsigned*)(rp + r_id); g.req_lam = (float*)(rp + r_lam); g.req_key = (uint8_t*)(rp + r_key);
    g.req_out = (float4*)(rp + r_out); g.req_bail = (uint8_t*)(rp + r_bail);
    g.n_req = (unsigned*)(rp + r_cnt); g.n_live = g.n_req + 1;
    g.req_scen = star ? (int*)(rp + r_scen) : nullptr;
    g.ws.order = (unsigned*)(wp + w_order); g.ws.items = (unsigned long long*)(wp + w_items);
    g.ws.items_sorted = (unsigned long long*)(wp + w_sorted); g.ws.item_count = (unsigned*)(wp + w_cnt);
    g.cand = sa.cand;
    g.fb_count = sa.fb_count; g.fb_list = sa.fb_list; g.fb_cap = sa.fb_cap;
    g.scen_rpm = sa.scen_rpm; g.n_scen = sa.n_scen;

    const unsigned nb = (unsigned)((n + 255) / 256);
    const unsigned cks = (unsigned)chunks, items_blocks = (unsigned)((max_items + 255) / 256),
                   solve_blocks = (unsigned)((max_items * 32 + 255) / 256);
    sz2_init<<<nb, 256, 0, h->stream>>>(g);
    h->launches++;
    unsigned* pin = (unsigned*)h->sz_pin.p;
    // Rounds are enqueued in groups without looking at the device: every kernel of a round leaves at once when the
    // round has no requests, so over-launching costs microseconds while a host round trip per round costs more.
    // A search needs 1 + ceil(100 / D) rounds at most, then two Analyze rounds and the final consume.
    const int max_rounds = 1 + (100 + D - 1) / D + 4;
    const int group = 4;
    for (int round = 0; round < max_rounds; round += group) {
        for (int r = 0; r < group; ++r) {
            sz2_round_reset<<<3, 256, 0, h->stream>>>(g);
            if (star) sz2_advance<true><<<nb, 256, 0, h->stream>>>(g);
            else sz2_advance<false><<<nb, 256, 0, h->stream>>>(g);
            sz2_sort_local<<<cks, kSortThreads, 0, h->stream>>>(g);
            ws_items_scan<<<1, 256, 0, h->stream>>>(g.ws);
            ws_items_scatter<<<items_blocks, 256, 0, h->stream>>>(g.ws);
            g.dbg = nullptr;
            if (dbg_round == round + r) {
                CK(h->d_dbg.ensure(16 * cap));
                CK(cudaMemsetAsync(h->d_dbg.p, 0, 16 * cap, h->stream));
                g.dbg = (unsigned*)h->d_dbg.p;
                h->dbg_n = cap;
            }
            if (size_rev) sz2_solve<1><<<solve_blocks, 256, solve_pad, h->stream>>>(g);
            else sz2_solve<0><<<solve_blocks, 256, solve_pad, h->stream>>>(g);
            h->launches += 6;
        }
        // candidates still unfinished after the group's last advance decide whether another group is needed
        CK(cudaMemcpyAsync(pin, g.n_live, sizeof(unsigned), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (*pin == 0) break;
    }
    CK(cudaGetLastError());
    if (star) {
        g.dbg = nullptr;
        *star = g;
    }
    return WVA_OK;
}

// Enqueue analyze (+ unlimited solve). cand/winner columns are device pointers.
int enqueue_size(wva_handle* h, const AllocCols& cand, const AllocCols* winners) {
    int rc = prepare_size(h);
    if (rc) return rc;
    rc = ensure_ctrl(h);
    if (rc) return rc;
    const HostFleet& hf = h->hf;
    const int n_pairs = hf.S * hf.A;
    const int n = (int)h->cand_pair.size();
    if (n_pairs > 0) {
        trivial_kernel<<<(n_pairs + 255) / 256, 256, 0, h->stream>>>(h->df, cand, nullptr);
        h->launches++;
    }
    SizeArgs g{};
    g.f = h->df;
    g.cand_pair = (const int*)h->d_cand_pair.p;
    g.cand_N = (const int*)h->d_cand_N.p;
    g.n_cand = n;
    g.cand = cand;
    g.fb_count = (int*)h->d_ctrl.p + CTRL_FB_COUNT;
    CK(h->d_fb_list.ensure(sizeof(int) * std::max(n, 1)));
    g.fb_list = (int*)h->d_fb_list.p;
    g.fb_cap = std::max(n, 1);
    g.n_scen = 1;
    CK(cudaEventRecord(h->ev_k0, h->stream));
    int small_max = 1024;  // up to here a warp per candidate beats rounds (the GPU is mostly empty either way)
    if (const char* e = getenv("WVA_SIZE_SMALL_MAX")) small_max = atoi(e);
    if (n > 0 && n <= small_max) {
        size_warp_kernel<<<(unsigned)((n + 3) / 4), 128, 0, h->stream>>>(g, (const double*)h->d_sz_tab.p,
                                                                          (const long long*)h->d_sz_off.p);
        h->launches++;
    } else if (n > 0) {
        rc = run_size_rounds(h, g, n, (const double*)h->d_sz_tab.p, (const long long*)h->d_sz_off.p,
                             (const float*)h->d_sz_ls.p);
        if (rc) return rc;
    }
    CK(cudaEventRecord(h->ev_k1, h->stream));
    if (n > 0) {
        size_t slot_doubles;
        int Kmax;
        rc = ensure_scratch(h, h->size_Nmax, hf.tun.max_queue_to_batch_ratio, &slot_doubles, &Kmax);
        if (rc) return rc;
        size_fallback<<<kFbBlocks, kFbThreads, 0, h->stream>>>(g, (double*)h->d_scratch.p, slot_doubles, Kmax,
                                                               (int*)h->d_ctrl.p + CTRL_FB_STATUS);
        h->launches++;
    }
    if (winners && hf.S > 0) {
        unlimited_kernel<<<(hf.S + 127) / 128, 128, 0, h->stream>>>(h->df, cand, *winners);
        h->launches++;
    }
    CK(cudaGetLastError());
    return WVA_OK;
}

int finish_timing(wva_handle* h) {
    CK(cudaEventRecord(h->ev_d1, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    cudaEventElapsedTime(&h->last_kernel_ms, h->ev_k0, h->ev_k1);
    cudaEventElapsedTime(&h->last_device_ms, h->ev_d0, h->ev_d1);
    return WVA_OK;
}

int check_fallback_status(wva_handle* h, const int* ctrl_host, long long cap) {
    h->dbg_fb_count = ctrl_host[CTRL_FB_COUNT];  // before the cap test: a count above it is reported as well
    if (ctrl_host[CTRL_FB_STATUS] != 0)
        return h->fail(WVA_ERR_UNSUPPORTED, "input outside the supported numeric domain (rescale loop does not terminate)");
    if ((long long)ctrl_host[CTRL_FB_COUNT] > cap)
        return h->fail(WVA_ERR_UNSUPPORTED, "too many cells need the stored-vector fallback");
    return WVA_OK;
}

// resident analyze/solve with host outputs
int run_size_host(wva_handle* h, wva_allocs* candidates, wva_allocs* winners) {
    if (!h->resident) return h->fail(WVA_ERR_STATE, "no resident fleet (call wva_upload first)");
    const HostFleet& hf = h->hf;
    const size_t n_pairs = (size_t)hf.S * hf.A;
    const Block bc = block_layout(n_pairs), bw = block_layout(hf.S);
    CK(h->d_cand_block.ensure(bc.bytes + 16));
    CK(h->d_win_block.ensure(bw.bytes + 16));
    const AllocCols dc = block_cols(h->d_cand_block.p, bc), dw = block_cols(h->d_win_block.p, bw);
    CK(cudaEventRecord(h->ev_d0, h->stream));
    int rc = enqueue_size(h, dc, winners ? &dw : nullptr);
    if (rc) return rc;
    const size_t stage_bytes = align_up(bc.bytes) + align_up(bw.bytes) + 256;
    CK(h->out_stage.ensure(stage_bytes));
    char* hs = (char*)h->out_stage.p;
    if (candidates && bc.bytes) CK(cudaMemcpyAsync(hs, h->d_cand_block.p, bc.bytes, cudaMemcpyDeviceToHost, h->stream));
    if (winners && bw.bytes)
        CK(cudaMemcpyAsync(hs + align_up(bc.bytes), h->d_win_block.p, bw.bytes, cudaMemcpyDeviceToHost, h->stream));
    int* ctrl_host = (int*)(hs + align_up(bc.bytes) + align_up(bw.bytes));
    CK(cudaMemcpyAsync(ctrl_host, h->d_ctrl.p, CTRL_INTS * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    rc = finish_timing(h);
    if (rc) return rc;
    rc = check_fallback_status(h, ctrl_host, (long long)h->cand_pair.size() + 1);
    if (rc) return rc;
    scatter_block(hs, bc, candidates);
    scatter_block(hs + align_up(bc.bytes), bw, winners);
    return WVA_OK;
}

// ---- grid path (K2 + K3) ----------------------------------------------------
int validate_grid(wva_handle* h, const wva_grid* g) {
    if (!g) return h->fail(WVA_ERR_BAD_ARG, "grid is NULL");
    if (g->n_batch < 0 || g->n_replicas < 0) return h->fail(WVA_ERR_BAD_ARG, "negative grid size");
    if ((g->n_batch > 0 && !g->batch) || (g->n_replicas > 0 && !g->replicas))
        return h->fail(WVA_ERR_BAD_ARG, "NULL grid column");
    for (int i = 0; i < g->n_batch; ++i)
        if (g->batch[i] < 1 || g->batch[i] > (1 << 20)) return h->fail(WVA_ERR_BAD_ARG, "batch size out of range");
    for (int i = 0; i < g->n_replicas; ++i)
        if (g->replicas[i] < 1) return h->fail(WVA_ERR_BAD_ARG, "replica count out of range");
    return WVA_OK;
}

struct GridPlan {
    GridArgs args;
    size_t n_cells;
    int n_blocks;
    int Bmax;
};

// Per-cell columns kept on the device for every grid solve: flags + ttft/itl/rho (+ throughput
// when the caller asked for the cell table).
int ensure_cells(wva_handle* h, GridPlan& plan, bool want_cells, bool want_throughput) {
    const size_t nc = std::max<size_t>(plan.n_cells, 1);
    const size_t bytes = align_up(nc) + 4 * align_up(4 * nc);
    CK(h->d_cells.ensure(bytes));
    char* p = (char*)h->d_cells.p;
    plan.args.cells.flags = (uint8_t*)p;
    plan.args.cells.ttft = (float*)(p + align_up(nc));
    plan.args.cells.itl = (float*)(p + align_up(nc) + align_up(4 * nc));
    plan.args.cells.rho = (float*)(p + align_up(nc) + 2 * align_up(4 * nc));
    plan.args.cells.throughput = want_throughput ? (float*)(p + align_up(nc) + 3 * align_up(4 * nc)) : nullptr;
    plan.args.want_cells = want_cells ? 1 : 0;
    return WVA_OK;
}

int prepare_grid(wva_handle* h, const wva_grid* grid, GridPlan* plan) {
    const HostFleet& hf = h->hf;
    const int A = hf.A, S = hf.S, B = grid->n_batch, R = grid->n_replicas;
    const bool same_grid = h->grid_epoch == h->epoch_tokens && (int)h->grid_batch.size() == B &&
                           (int)h->grid_replicas.size() == R &&
                           std::equal(h->grid_batch.begin(), h->grid_batch.end(), grid->batch) &&
                           std::equal(h->grid_replicas.begin(), h->grid_replicas.end(), grid->replicas);
    const int n_pairs = S * A;
    int Bmax = 1;
    for (int i = 0; i < B; ++i) Bmax = std::max(Bmax, grid->batch[i]);
    // device lists: batch[B], batch_rank[B], rank_to_bi[B], replicas[R]
    CK(h->d_grid_lists.ensure(sizeof(int) * (size_t)(3 * B + R + 1)));
    CK(h->d_pair_tab.ensure((sizeof(long long) + sizeof(int)) * std::max(n_pairs, 1)));
    long long* d_pair_off = (long long*)h->d_pair_tab.p;
    int* d_pair_idx = (int*)(d_pair_off + std::max(n_pairs, 1));
    if (!same_grid) {
        // pageable sources: cudaMemcpyAsync has consumed them by the time it returns
        std::vector<int> lists(3 * B + R + 1), tab_pair, tab_len, pair_idx(std::max(n_pairs, 1), -1);
        std::vector<long long> pair_tab(std::max(n_pairs, 1), -1), tab_off;
        h->grid_batch.assign(grid->batch, grid->batch + B);
        h->grid_replicas.assign(grid->replicas, grid->replicas + R);
        std::vector<int> order(B);
        std::iota(order.begin(), order.end(), 0);
        std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return grid->batch[x] < grid->batch[y]; });
        for (int i = 0; i < B; ++i) {
            lists[i] = grid->batch[i];
            lists[B + order[i]] = i;      // batch_rank[bi]
            lists[2 * B + i] = order[i];  // rank_to_bi[rank]
        }
        for (int i = 0; i < R; ++i) lists[3 * B + i] = grid->replicas[i];
        if (3 * B + R > 0)
            CK(cudaMemcpyAsync(h->d_grid_lists.p, lists.data(), sizeof(int) * (size_t)(3 * B + R), cudaMemcpyHostToDevice,
                               h->stream));
        // shared service-rate tables for every pair that carries load
        long long off = 0;
        for (int s = 0; s < S; ++s)
            for (int a = 0; a < A; ++a)
                if (hf.pair_class(s, a, true) == PAIR_LOAD && hf.srv_out_tokens[s] >= 1) {
                    pair_tab[(size_t)s * A + a] = off;
                    pair_idx[(size_t)s * A + a] = (int)tab_pair.size();
                    tab_pair.push_back(s * A + a);
                    tab_off.push_back(off);
                    tab_len.push_back(Bmax);
                    off += Bmax;
                }
        if (off > 0xffffffffll) return h->fail(WVA_ERR_UNSUPPORTED, "grid tables above 2^32 entries");
        const int n_tab = (int)tab_pair.size();
        CK(cudaMemcpyAsync(d_pair_off, pair_tab.data(), sizeof(long long) * std::max(n_pairs, 1), cudaMemcpyHostToDevice,
                           h->stream));
        CK(cudaMemcpyAsync(d_pair_idx, pair_idx.data(), sizeof(int) * std::max(n_pairs, 1), cudaMemcpyHostToDevice,
                           h->stream));
        if (n_tab) {
            CK(h->d_tab_pair.ensure(sizeof(int) * n_tab));
            CK(h->d_tab_off.ensure(sizeof(long long) * n_tab));
            CK(h->d_tab_len.ensure(sizeof(int) * n_tab));
            CK(h->d_tab.ensure(sizeof(double) * 4 * (size_t)off));
            CK(h->d_ls.ensure(sizeof(float) * ((size_t)off + n_tab)));
            CK(cudaMemcpyAsync(h->d_tab_pair.p, tab_pair.data(), sizeof(int) * n_tab, cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(h->d_tab_off.p, tab_off.data(), sizeof(long long) * n_tab, cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(h->d_tab_len.p, tab_len.data(), sizeof(int) * n_tab, cudaMemcpyHostToDevice, h->stream));
        }
        h->grid_n_tab = n_tab;
        h->grid_Bmax = Bmax;
        h->grid_epoch = h->epoch_tokens;
    }
    // the tables are rebuilt on every call (only the host-side work lists are cached):
    // they are part of the evaluation, not an input
    // [tables x batch] constants, then the [server x replica] rate block grid_rows fills (always allocated)
    CK(h->d_pb.ensure(sizeof(float4) * ((size_t)h->grid_n_tab * std::max(B, 1) + (size_t)S * std::max(R, 1) + 1)));
    if (h->grid_n_tab) {
        float4* d_pb = (float4*)h->d_pb.p;
        build_pair_tables<<<h->grid_n_tab, 128, 0, h->stream>>>(h->df, (const int*)h->d_tab_pair.p,
                                                                (const long long*)h->d_tab_off.p,
                                                                (const int*)h->d_tab_len.p, h->grid_n_tab,
                                                                (double*)h->d_tab.p, (float*)h->d_ls.p,
                                                                (const int*)h->d_grid_lists.p, B, d_pb);
        h->launches += 1;
        CK(cudaGetLastError());
    }
    GridArgs& g = plan->args;
    g = GridArgs{};
    g.f = h->df;
    g.batch = (const int*)h->d_grid_lists.p;
    g.batch_rank = g.batch + B;
    g.rank_to_bi = g.batch + 2 * B;
    g.replicas = g.batch + 3 * B;
    g.B = B;
    g.R = R;
    g.tab = (const double*)h->d_tab.p;
    g.ls = (const float*)h->d_ls.p;
    g.pair_tab_off = d_pair_off;
    g.pair_tab_idx = d_pair_idx;
    g.pb = (const float4*)h->d_pb.p;
    g.rt = (float4*)h->d_pb.p + (size_t)h->grid_n_tab * std::max(B, 1);
    const unsigned long long n_cells = (unsigned long long)S * A * B * R;
    if (n_cells > 0xfffffff0ull) return h->fail(WVA_ERR_UNSUPPORTED, "grid too large for one call (>= 2^32 cells)");
    g.n_cells = (long long)n_cells;
    plan->n_cells = (size_t)n_cells;
    plan->n_blocks = (int)((n_cells + kSortChunk - 1) / kSortChunk);
    const size_t nc = std::max<size_t>(plan->n_cells, 1);
    // sort workspace: order u32 [n_cells] | items u64 | items_sorted u64 | item counter
    const size_t max_items = (nc + 31) / 32 + (size_t)std::max(plan->n_blocks, 1);
    // ... | per-cell records in global item order (32 x 16 bytes per item)
    const size_t ws = align_up(4 * nc) + 2 * align_up(8 * max_items) + align_up(4 * (2 * kClasses + 32)) +
                      align_up(512 * max_items);
    CK(h->d_sort.ensure(ws));
    char* w = (char*)h->d_sort.p;
    g.order = (unsigned*)w;
    g.items = (unsigned long long*)(w + align_up(4 * nc));
    g.items_sorted = (unsigned long long*)(w + align_up(4 * nc) + align_up(8 * max_items));
    g.item_count = (unsigned*)(w + align_up(4 * nc) + 2 * align_up(8 * max_items));
    g.recs = (uint4*)(w + align_up(4 * nc) + 2 * align_up(8 * max_items) + align_up(4 * (2 * kClasses + 32)));
    h->dbg_plan = g.item_count + 2 * kClasses + 1;
    const size_t n_best = std::max<size_t>((size_t)S * A * R, 1);
    CK(h->d_best.ensure(sizeof(int) * n_best));
    g.best_rank = (int*)h->d_best.p;
    const size_t n_pairs_alloc = std::max<size_t>((size_t)S * A, 1);
    const size_t rows_bytes = align_up((2 * sizeof(double) + sizeof(int)) * n_best + 64);
    CK(h->d_rows.ensure(rows_bytes + align_up(48 * n_pairs_alloc) + n_best));
    g.row_acc = (double*)h->d_rows.p;
    g.row_sump = g.row_acc + n_best;
    g.row_j = (int*)(g.row_sump + n_best);
    g.pair_rec = (float4*)((char*)h->d_rows.p + rows_bytes);
    g.row_res = (uint8_t*)h->d_rows.p + rows_bytes + align_up(48 * n_pairs_alloc);
    h->dbg_row_j = g.row_j;
    h->dbg_row_res = g.row_res;
    h->dbg_rows_n = (size_t)S * A * R;
    // row resolution (DESIGN §3.2b); WVA_GRID_ROWRES=0 keeps the per-cell evaluation of every shared cell
    g.row_resolve = 1;
    if (const char* e = getenv("WVA_GRID_ROWRES")) g.row_resolve = atoi(e) != 0;
    g.Bmax = h->grid_Bmax;
    g.fb_count = (int*)h->d_ctrl.p + CTRL_FB_COUNT;
    g.fb_cap = (int)std::min<size_t>(nc, (size_t)1 << 22);
    CK(h->d_fb_list.ensure(sizeof(long long) * g.fb_cap));
    g.fb_cells = (long long*)h->d_fb_list.p;
    {
        // grid_kernel's long queue: items of at least ~min_len states, at most long_per_sm per SM
        int long_per_sm = kGkLong, min_len = 1024;
        if (const char* e = getenv("WVA_GRID_LONG")) long_per_sm = std::min(std::max(atoi(e), -1), kGkWarps / 4);
        if (const char* e = getenv("WVA_GRID_LONG_MINLEN")) min_len = std::max(atoi(e), 2);
        g.long_per_sm = long_per_sm;
        g.long_share = 0;
        if (const char* e = getenv("WVA_GRID_SHARE")) g.long_share = std::max(atoi(e), 0);
        g.long_cls = 254 - std::min(std::max((int)(log2f((float)min_len) * 12.0f), 0), 254);
        g.long_cap = (unsigned)(std::max(long_per_sm, 0) * h->sm_count);
        g.n_ctas = h->sm_count;
    }
    if (h->dbg_cycles) {
        CK(h->d_dbg.ensure(sizeof(unsigned) * nc * 2));
        CK(cudaMemsetAsync(h->d_dbg.p, 0, sizeof(unsigned) * nc * 2, h->stream));
        g.dbg_cycles = (unsigned*)h->d_dbg.p;
        g.dbg_n = nc;
        h->dbg_n = nc;
    }
    plan->Bmax = Bmax;
    return WVA_OK;
}

int enqueue_grid(wva_handle* h, GridPlan& plan, const AllocCols& winners) {
    GridArgs& g = plan.args;
    const HostFleet& hf = h->hf;
    size_t slot_doubles;
    int Kmax;
    int rc = ensure_scratch(h, plan.Bmax, hf.tun.max_queue_to_batch_ratio, &slot_doubles, &Kmax);
    if (rc) return rc;
    const size_t n_best = (size_t)hf.S * hf.A * g.R;
    if (plan.n_cells == 0) CK(cudaEventRecord(h->ev_k0, h->stream));
    if (plan.n_cells > 0) {
        CK(cudaMemsetAsync(g.item_count, 0, sizeof(unsigned) * (2 * kClasses + 32), h->stream));
        {
            const int rows_threads = g.R >= 128 ? 128 : (g.R > 32 ? 64 : 32);
            const size_t rows_smem = g.Bmax <= kRowsSmemEntries ? (size_t)g.Bmax * 32 : 0;
            grid_rows<<<(unsigned)(hf.S * hf.A), rows_threads, rows_smem, h->stream>>>(g);
        }
        h->launches++;
        grid_sort_local<<<plan.n_blocks, kSortThreads, 0, h->stream>>>(g);
        // one warp per item; the item count lives on the device, so launch for the worst case
        const size_t max_items = (plan.n_cells + 31) / 32 + (size_t)plan.n_blocks;
        (void)max_items;
        grid_items_scatter<<<(unsigned)(16 * h->sm_count), 256, 0, h->stream>>>(g);  // warp per item (grid-stride)
        h->launches++;
        CK(cudaEventRecord(h->ev_k0, h->stream));  // wva_last_kernel_ms = the dominant kernel alone
        const size_t smem = (size_t)kGkWarps * kGkWarpD * sizeof(double);
        grid_kernel<<<(unsigned)h->sm_count, kGkThreads, smem, h->stream>>>(g);
        h->launches += 2;
    }
    CK(cudaEventRecord(h->ev_k1, h->stream));
    if (plan.n_cells > 0) {
        grid_fallback<<<kFbBlocks, kFbThreads, 0, h->stream>>>(g, (double*)h->d_scratch.p, slot_doubles, Kmax,
                                                               (int*)h->d_ctrl.p + CTRL_FB_STATUS);
        h->launches++;
    }
    if (hf.S > 0) {
        grid_finalize<<<hf.S, 256, 0, h->stream>>>(g, winners);
        h->launches++;
    }
    CK(cudaGetLastError());
    return WVA_OK;
}


// ---- limited mode: SolveGreedy on the host over device-computed candidates --------------
// pkg/solver/greedy.go:35-341.  The candidate generation (the expensive part) ran on the
// device; the greedy pass is inherently sequential over a shared capacity map (SURVEY.md
// §8e), so it stays on the host.  Sorts are stable (the reference's pdqsort is not): ties
// resolve by server id / accelerator id.
struct HostCand {
    uint8_t feasible;
    int acc, replicas, batch;
    float cost, value, itl, ttft, rho, max_rate;
};

struct GreedyEntry {  // greedy.go:16-22
    int server, priority, cur = 0;
    std::vector<int> accs;  // candidate accelerator ids ordered by value
    float delta = 0.f;
};

inline int cmp_f32(float a, float b) {  // cmp.Compare: NaN sorts first
    const bool an = a != a, bn = b != b;
    if (an || bn) return an && bn ? 0 : (an ? -1 : 1);
    return a < b ? -1 : (a > b ? 1 : 0);
}

class GreedySolver {
  public:
    GreedySolver(const HostFleet& f, std::vector<HostCand>& cand, std::vector<HostCand>& win)
        : f_(f), cand_(cand), win_(win), avail_(f.type_capacity.begin(), f.type_capacity.end()) {}

    void run() {
        const int S = f_.S, A = f_.A;
        std::vector<GreedyEntry> pool;
        pool.reserve(S);
        for (int s = 0; s < S; ++s) {
            win_[s] = HostCand{};
            win_[s].acc = WVA_ACC_NONE;
            GreedyEntry e;
            e.server = s;
            e.priority = f_.srv_priority[s];
            for (int a = 0; a < A; ++a)
                if (at(s, a).feasible) e.accs.push_back(a);
            if (e.accs.empty()) continue;
            std::stable_sort(e.accs.begin(), e.accs.end(),
                             [&](int x, int y) { return cmp_f32(at(s, x).value, at(s, y).value) < 0; });
            e.delta = e.accs.size() > 1 ? at(s, e.accs[1]).value - at(s, e.accs[0]).value : FLT_MAX;
            pool.push_back(std::move(e));
        }
        std::vector<GreedyEntry*> entries;
        for (auto& e : pool) entries.push_back(&e);
        std::stable_sort(entries.begin(), entries.end(),
                         [&](GreedyEntry* x, GreedyEntry* y) { return order(*x, *y) < 0; });
        if (f_.delayed_best_effort) {
            std::vector<GreedyEntry*> un = allocate(entries);
            best_effort(un);
        } else {
            size_t i = 0;
            while (i < entries.size()) {  // makePriorityGroups :321-341
                size_t j = i + 1;
                while (j < entries.size() && entries[j]->priority == entries[i]->priority) ++j;
                std::vector<GreedyEntry*> group(entries.begin() + i, entries.begin() + j);
                std::vector<GreedyEntry*> un = allocate(group);
                best_effort(un);
                i = j;
            }
        }
    }

  private:
    HostCand& at(int s, int a) { return cand_[(size_t)s * f_.A + a]; }
    HostCand& cur(const GreedyEntry& e) { return at(e.server, e.accs[e.cur]); }
    int units(int s, int a) const {
        const int c = f_.perf_acc_count[(size_t)f_.srv_model[s] * f_.A + a];
        return (c <= 0 ? 1 : c) * f_.acc_mult[a];
    }
    int order(GreedyEntry& a, GreedyEntry& b) {  // greedy.go:76-85
        if (a.priority != b.priority) return a.priority < b.priority ? -1 : 1;
        if (a.delta == b.delta) return cmp_f32(cur(b).value, cur(a).value);
        return cmp_f32(b.delta, a.delta);
    }
    std::vector<GreedyEntry*> allocate(std::vector<GreedyEntry*> q) {  // greedy.go:107-166
        std::vector<GreedyEntry*> un;
        size_t head = 0;
        while (head < q.size()) {
            GreedyEntry* top = q[head++];
            if (top->accs.empty()) continue;
            HostCand& al = cur(*top);
            const int g = al.acc;
            if (g < 0 || g >= f_.A) continue;  // accelerator "" (zero-replica allocation)
            const int t = f_.acc_type[g];
            const int count = al.replicas * units(top->server, g);
            if (avail_[t] >= count) {
                avail_[t] -= count;
                win_[top->server] = al;
                continue;
            }
            top->cur++;
            if (top->cur + 1 < (int)top->accs.size()) {
                top->delta = at(top->server, top->accs[top->cur + 1]).value - cur(*top).value;
            } else if (top->cur == (int)top->accs.size()) {
                un.push_back(top);
                continue;
            } else {
                top->delta = FLT_MAX;
            }
            // slices.BinarySearchFunc: leftmost position whose element does not order before top
            auto it = std::partition_point(q.begin() + head, q.end(), [&](GreedyEntry* e) { return order(*e, *top) < 0; });
            q.insert(it, top);
        }
        return un;
    }
    void scale_to(HostCand& al, int replicas) {  // greedy.go:206-211
        const float factor = (float)replicas / (float)al.replicas;
        al.cost *= factor;
        al.value *= factor;
        al.replicas = replicas;
    }
    void allocate_maximally(const std::vector<GreedyEntry*>& es) {  // greedy.go:194-223
        for (GreedyEntry* e : es)
            for (int a : e->accs) {
                HostCand& al = at(e->server, a);
                if (al.acc < 0 || al.acc >= f_.A) continue;
                const int upr = units(e->server, al.acc);
                if (upr <= 0) continue;
                const int t = f_.acc_type[al.acc];
                const int mx = std::min(avail_[t] / upr, al.replicas);
                if (mx > 0) {
                    scale_to(al, mx);
                    win_[e->server] = al;
                    avail_[t] -= mx * upr;
                    break;
                }
            }
    }
    void allocate_equally(const std::vector<GreedyEntry*>& es) {  // greedy.go:239-316
        struct Ticket {
            bool present = true, active = false, allocated = false;
            int type = 0, upr = 0, n = 0;
            HostCand* fin = nullptr;
        };
        std::vector<Ticket> tk(es.size());
        size_t live = es.size();
        while (live > 0) {
            for (size_t k = 0; k < es.size(); ++k) {
                Ticket& t = tk[k];
                if (!t.present) continue;
                if (!t.active) {
                    for (int a : es[k]->accs) {
                        HostCand& al = at(es[k]->server, a);
                        if (al.acc < 0 || al.acc >= f_.A) continue;
                        const int upr = units(es[k]->server, al.acc);
                        if (upr > 0 && avail_[f_.acc_type[al.acc]] >= upr) {
                            t.active = true;
                            t.type = f_.acc_type[al.acc];
                            t.upr = upr;
                            t.fin = &al;
                            break;
                        }
                    }
                    if (!t.active) {
                        t.present = false;
                        --live;
                        continue;
                    }
                }
                if (std::min(avail_[t.type] / t.upr, t.fin->replicas) > 0) {
                    t.n++;
                    avail_[t.type] -= t.upr;
                    t.allocated = true;
                } else {
                    t.present = false;
                    --live;
                }
            }
        }
        for (size_t k = 0; k < es.size(); ++k)
            if (tk[k].allocated) {
                scale_to(*tk[k].fin, tk[k].n);
                win_[es[k]->server] = *tk[k].fin;
            }
    }
    void best_effort(const std::vector<GreedyEntry*>& un) {  // greedy.go:169-190
        switch (f_.saturation_policy) {
        case WVA_SAT_PRIORITY_EXHAUSTIVE: allocate_maximally(un); break;
        case WVA_SAT_PRIORITY_ROUND_ROBIN: {
            size_t i = 0;
            while (i < un.size()) {
                size_t j = i + 1;
                while (j < un.size() && un[j]->priority == un[i]->priority) ++j;
                allocate_equally(std::vector<GreedyEntry*>(un.begin() + i, un.begin() + j));
                i = j;
            }
            break;
        }
        case WVA_SAT_ROUND_ROBIN: allocate_equally(un); break;
        default: break;
        }
    }
    const HostFleet& f_;
    std::vector<HostCand>& cand_;
    std::vector<HostCand>& win_;
    std::vector<int> avail_;
};

void block_to_cands(const void* host_block, const Block& b, std::vector<HostCand>& out) {
    const char* p = (const char*)host_block;
    out.resize(b.n);
    for (size_t i = 0; i < b.n; ++i) {
        HostCand& c = out[i];
        c.feasible = ((const uint8_t*)(p + b.off_feasible))[i];
        c.acc = ((const int*)(p + b.off_acc))[i];
        c.replicas = ((const int*)(p + b.off_replicas))[i];
        c.batch = ((const int*)(p + b.off_batch))[i];
        c.cost = ((const float*)(p + b.off_cost))[i];
        c.value = ((const float*)(p + b.off_value))[i];
        c.itl = ((const float*)(p + b.off_itl))[i];
        c.ttft = ((const float*)(p + b.off_ttft))[i];
        c.rho = ((const float*)(p + b.off_rho))[i];
        c.max_rate = ((const float*)(p + b.off_rate))[i];
    }
}
// writes v into records at .. at + v.size() - 1 of out
void cands_to_abi(const std::vector<HostCand>& v, wva_allocs* out, size_t at = 0) {
    if (!out) return;
    for (size_t k = 0; k < v.size(); ++k) {
        const HostCand& c = v[k];
        const size_t i = at + k;
        if (out->feasible) out->feasible[i] = c.feasible;
        if (out->acc) out->acc[i] = c.acc;
        if (out->replicas) out->replicas[i] = c.replicas;
        if (out->batch) out->batch[i] = c.batch;
        if (out->cost) out->cost[i] = c.cost;
        if (out->value) out->value[i] = c.value;
        if (out->itl) out->itl[i] = c.itl;
        if (out->ttft) out->ttft[i] = c.ttft;
        if (out->rho) out->rho[i] = c.rho;
        if (out->max_rate) out->max_rate[i] = c.max_rate;
    }
}

bool abi_to_cands(const wva_allocs* in, size_t n, std::vector<HostCand>& out) {
    if (!in || (n && (!in->feasible || !in->acc || !in->replicas || !in->cost || !in->value))) return false;
    out.resize(n);
    for (size_t i = 0; i < n; ++i) {
        HostCand& c = out[i];
        c.feasible = in->feasible[i];
        c.acc = in->acc[i];
        c.replicas = in->replicas[i];
        c.batch = in->batch ? in->batch[i] : 0;
        c.cost = in->cost[i];
        c.value = in->value[i];
        c.itl = in->itl ? in->itl[i] : 0.0f;
        c.ttft = in->ttft ? in->ttft[i] : 0.0f;
        c.rho = in->rho ? in->rho[i] : 0.0f;
        c.max_rate = in->max_rate ? in->max_rate[i] : 0.0f;
    }
    return true;
}

// resident analyze + greedy solve with host outputs
int run_greedy_host(wva_handle* h, wva_allocs* candidates, wva_allocs* winners) {
    const HostFleet& hf = h->hf;
    for (int a = 0; a < hf.A; ++a)
        if (hf.T <= 0 || hf.acc_type[a] < 0 || hf.acc_type[a] >= hf.T)
            return h->fail(WVA_ERR_BAD_ARG, "limited mode needs a type id and a capacity for every accelerator");
    const size_t n_pairs = (size_t)hf.S * hf.A;
    const Block bc = block_layout(n_pairs), bw = block_layout(hf.S);
    CK(h->d_cand_block.ensure(bc.bytes + 16));
    CK(h->d_win_block.ensure(bw.bytes + 16));
    const AllocCols dc = block_cols(h->d_cand_block.p, bc), dw = block_cols(h->d_win_block.p, bw);
    CK(cudaEventRecord(h->ev_d0, h->stream));
    int rc = enqueue_size(h, dc, &dw);  // the unlimited kernel also assigns value = transition penalty
    if (rc) return rc;
    const size_t stage_bytes = align_up(bc.bytes) + 256;
    CK(h->out_stage.ensure(stage_bytes));
    char* hs = (char*)h->out_stage.p;
    if (bc.bytes) CK(cudaMemcpyAsync(hs, h->d_cand_block.p, bc.bytes, cudaMemcpyDeviceToHost, h->stream));
    int* ctrl_host = (int*)(hs + align_up(bc.bytes));
    CK(cudaMemcpyAsync(ctrl_host, h->d_ctrl.p, CTRL_INTS * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    rc = finish_timing(h);
    if (rc) return rc;
    rc = check_fallback_status(h, ctrl_host, (long long)h->cand_pair.size() + 1);
    if (rc) return rc;
    std::vector<HostCand> cand, win((size_t)hf.S);
    block_to_cands(hs, bc, cand);
    GreedySolver(hf, cand, win).run();
    cands_to_abi(cand, candidates);
    cands_to_abi(win, winners);
    h->last_feasible.resize(hf.S); h->last_acc.resize(hf.S); h->last_replicas.resize(hf.S); h->last_cost.resize(hf.S);
    for (int s = 0; s < hf.S; ++s) {
        h->last_feasible[s] = win[s].feasible;
        h->last_acc[s] = win[s].acc;
        h->last_replicas[s] = win[s].replicas;
        h->last_cost[s] = win[s].cost;
    }
    h->last_kind = 2;
    return WVA_OK;
}

// ---- scenarios (wva_resolve_scenarios, DESIGN §3.8) --------------------------------------------------------------
// Candidate list: every pair that passes the gates of CreateAllocation that do not read the arrival rate, has
// out_tokens > 0, and carries load (a rate neither == 0 nor < 0, NaN included) in at least one scenario.  That is the
// union over the scenarios of the lists prepare_size would build.
int prepare_scenarios(wva_handle* h, int L, const float* rpm) {
    const HostFleet& hf = h->hf;
    const int A = hf.A, S = hf.S;
    // the list is a function of the token epoch and of which servers carry load in some scenario
    std::vector<uint8_t> loaded(S, 0);
    for (int s = 0; s < S; ++s)
        for (int l = 0; l < L && !loaded[s]; ++l) {
            const float r = rpm[(size_t)l * S + s];
            loaded[s] = !(r == 0.0f) && !(r < 0.0f);
        }
    if (h->scen_epoch == h->epoch_tokens && loaded == h->scen_loaded) return WVA_OK;
    std::vector<int> pairs;
    std::vector<int> Ns((size_t)S * A, 0);
    for (int s = 0; s < S; ++s) {
        if (hf.srv_out_tokens[s] <= 0 || !loaded[s]) continue;
        for (int a = 0; a < A; ++a)
            if (hf.rate_free_gates(s, a, true)) {
                const int N = hf.pair_batch(s, a);
                if (N > (1 << 20)) return h->fail(WVA_ERR_UNSUPPORTED, "batch size above 2^20");
                Ns[(size_t)s * A + a] = N;
                pairs.push_back(s * A + a);
            }
    }
    std::stable_sort(pairs.begin(), pairs.end(), [&](int x, int y) { return Ns[x] > Ns[y]; });
    int rc = upload_size_list(h, pairs, Ns, h->scen_pair, h->scen_N, h->scen_Nmax, h->d_scen_pair, h->d_scen_N,
                              h->d_scen_off, h->d_scen_tab, h->d_scen_ls);
    if (rc) return rc;
    h->scen_loaded = loaded;
    h->scen_epoch = h->epoch_tokens;
    return WVA_OK;
}

// Size once (the rounds up to Analyze(lambda*)), then one round of final Analyze requests over (candidate, scenario),
// then the per-scenario trivial / fallback / unlimited kernels.  The resident fleet is not modified.
int run_scenarios(wva_handle* h, int L, const float* rpm, wva_allocs* candidates, wva_allocs* winners) {
    const HostFleet& hf = h->hf;
    if (!hf.unlimited)
        for (int a = 0; a < hf.A; ++a)
            if (hf.T <= 0 || hf.acc_type[a] < 0 || hf.acc_type[a] >= hf.T)
                return h->fail(WVA_ERR_BAD_ARG, "limited mode needs a type id and a capacity for every accelerator");
    int rc = prepare_scenarios(h, L, rpm);
    if (rc) return rc;
    rc = ensure_ctrl(h);
    if (rc) return rc;
    const size_t S = hf.S, A = hf.A;
    const int n = (int)h->scen_pair.size();
    const size_t n_req = (size_t)n * L;
    const Block bc = block_layout((size_t)L * S * A), bw = block_layout((size_t)L * S);
    CK(h->d_cand_block.ensure(bc.bytes + 16));
    CK(h->d_win_block.ensure(bw.bytes + 16));
    CK(h->d_scen_rpm.ensure(sizeof(float) * (size_t)L * S + 16));
    const AllocCols dc = block_cols(h->d_cand_block.p, bc), dw = block_cols(h->d_win_block.p, bw);
    const float* d_rpm = (const float*)h->d_scen_rpm.p;
    CK(cudaEventRecord(h->ev_d0, h->stream));
    if (S) CK(cudaMemcpyAsync(h->d_scen_rpm.p, rpm, sizeof(float) * (size_t)L * S, cudaMemcpyHostToDevice, h->stream));
    if (S * A > 0) {
        trivial_kernel<<<dim3((unsigned)((S * A + 255) / 256), (unsigned)L), 256, 0, h->stream>>>(h->df, dc, d_rpm);
        h->launches++;
    }
    SizeArgs g{};
    g.f = h->df;
    g.cand_pair = (const int*)h->d_scen_pair.p;
    g.cand_N = (const int*)h->d_scen_N.p;
    g.n_cand = n;
    g.cand = dc;
    g.fb_count = (int*)h->d_ctrl.p + CTRL_FB_COUNT;
    CK(h->d_fb_list.ensure(sizeof(int) * std::max<size_t>(n_req, 1)));
    g.fb_list = (int*)h->d_fb_list.p;
    g.fb_cap = (int)std::max<size_t>(n_req, 1);  // one entry per (candidate, scenario) at most
    g.scen_rpm = d_rpm;
    g.n_scen = L;
    CK(cudaEventRecord(h->ev_k0, h->stream));
    if (n > 0) {
        SizeArgs rounds = g;
        rounds.cand = AllocCols{};  // in STAR mode the rounds write no record
        Sz2Args z;
        rc = run_size_rounds(h, rounds, n, (const double*)h->d_scen_tab.p, (const long long*)h->d_scen_off.p,
                             (const float*)h->d_scen_ls.p, &z, n_req);
        if (rc) return rc;
        z.cand = dc;
        int size_rev = 1;
        if (const char* e = getenv("WVA_SIZE_REV")) size_rev = atoi(e);
        const size_t chunks = (n_req + kSortChunk - 1) / kSortChunk, max_items = (n_req + 31) / 32 + chunks;
        const unsigned nb = (unsigned)((n_req + 255) / 256);
        sz2_round_reset<<<3, 256, 0, h->stream>>>(z);
        sz2_expand<<<nb, 256, 0, h->stream>>>(z);
        sz2_sort_local<<<(unsigned)chunks, kSortThreads, 0, h->stream>>>(z);
        ws_items_scan<<<1, 256, 0, h->stream>>>(z.ws);
        ws_items_scatter<<<(unsigned)((max_items + 255) / 256), 256, 0, h->stream>>>(z.ws);
        const unsigned solve_blocks = (unsigned)((max_items * 32 + 255) / 256);
        if (size_rev) sz2_solve<1><<<solve_blocks, 256, 0, h->stream>>>(z);
        else sz2_solve<0><<<solve_blocks, 256, 0, h->stream>>>(z);
        sz2_consume<<<nb, 256, 0, h->stream>>>(z);
        h->launches += 7;
    }
    CK(cudaEventRecord(h->ev_k1, h->stream));
    if (n > 0) {
        size_t slot_doubles;
        int Kmax;
        rc = ensure_scratch(h, h->scen_Nmax, hf.tun.max_queue_to_batch_ratio, &slot_doubles, &Kmax);
        if (rc) return rc;
        size_fallback<<<kFbBlocks, kFbThreads, 0, h->stream>>>(g, (double*)h->d_scratch.p, slot_doubles, Kmax,
                                                               (int*)h->d_ctrl.p + CTRL_FB_STATUS);
        h->launches++;
    }
    if (S > 0) {  // also assigns value = transition penalty, which the greedy pass reads
        unlimited_kernel<<<dim3((unsigned)((S + 127) / 128), (unsigned)L), 128, 0, h->stream>>>(h->df, dc, dw);
        h->launches++;
    }
    CK(cudaGetLastError());
    const bool want_cand = candidates || !hf.unlimited, want_win = hf.unlimited;
    CK(h->out_stage.ensure(align_up(bc.bytes) + align_up(bw.bytes) + 256));
    char* hs = (char*)h->out_stage.p;
    if (want_cand && bc.bytes) CK(cudaMemcpyAsync(hs, h->d_cand_block.p, bc.bytes, cudaMemcpyDeviceToHost, h->stream));
    if (want_win && bw.bytes)
        CK(cudaMemcpyAsync(hs + align_up(bc.bytes), h->d_win_block.p, bw.bytes, cudaMemcpyDeviceToHost, h->stream));
    int* ctrl_host = (int*)(hs + align_up(bc.bytes) + align_up(bw.bytes));
    CK(cudaMemcpyAsync(ctrl_host, h->d_ctrl.p, CTRL_INTS * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    rc = finish_timing(h);
    if (rc) return rc;
    rc = check_fallback_status(h, ctrl_host, (long long)n_req + 1);
    if (rc) return rc;
    if (hf.unlimited) {
        scatter_block(hs, bc, candidates);
        scatter_block(hs + align_up(bc.bytes), bw, winners);
        return WVA_OK;
    }
    // limited mode: SolveGreedy once per scenario (it never reads the arrival rate)
    std::vector<HostCand> all, cand, win(S);
    block_to_cands(hs, bc, all);
    for (int l = 0; l < L; ++l) {
        cand.assign(all.begin() + (size_t)l * S * A, all.begin() + (size_t)(l + 1) * S * A);
        GreedySolver(hf, cand, win).run();
        cands_to_abi(cand, candidates, (size_t)l * S * A);
        cands_to_abi(win, winners, (size_t)l * S);
    }
    return WVA_OK;
}

}  // namespace

// =============================================================================
// C ABI
// =============================================================================
extern "C" {

void wva_tunables_default(wva_tunables* t) {
    if (!t) return;
    t->max_queue_to_batch_ratio = 10;  // pkg/config/defaults.go:18
    t->accel_penalty_factor = 0.1f;    // pkg/config/defaults.go:21
}

int wva_abi_version(void) { return WVA_ABI_VERSION; }

const char* wva_strerror(int code) {
    switch (code) {
    case WVA_OK: return "ok";
    case WVA_ERR_BAD_ARG: return "bad argument";
    case WVA_ERR_NO_DEVICE: return "no CUDA device";
    case WVA_ERR_CUDA: return "CUDA runtime error";
    case WVA_ERR_NOMEM: return "out of memory";
    case WVA_ERR_STATE: return "call sequence error";
    case WVA_ERR_UNSUPPORTED: return "input outside the supported domain";
    default: return "unknown error";
    }
}

const char* wva_last_error(const wva_handle* h) { return h ? h->err.c_str() : ""; }

int wva_create(wva_handle** out, int device) {
    if (!out) return WVA_ERR_BAD_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return WVA_ERR_NO_DEVICE;
    if (cudaSetDevice(device) != cudaSuccess) return WVA_ERR_NO_DEVICE;
    wva_handle* h = new (std::nothrow) wva_handle();
    if (!h) return WVA_ERR_NOMEM;
    h->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) h->sm_count = prop.multiProcessorCount;
    cudaFuncSetAttribute(grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)((size_t)kGkWarps * kGkWarpD * sizeof(double)));
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&h->ev_k0) != cudaSuccess || cudaEventCreate(&h->ev_k1) != cudaSuccess ||
        cudaEventCreate(&h->ev_d0) != cudaSuccess || cudaEventCreate(&h->ev_d1) != cudaSuccess) {
        delete h;
        return WVA_ERR_CUDA;
    }
    *out = h;
    return WVA_OK;
}

void wva_destroy(wva_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    DevBuf* bufs[] = {&h->arena, &h->d_cand_pair, &h->d_cand_N, &h->d_sz_tab, &h->d_sz_ls, &h->d_sz_off, &h->d_sz_state, &h->d_sz_req, &h->d_sz_sort, &h->d_grid_lists,
                      &h->d_pair_tab, &h->d_tab_pair, &h->d_tab_off, &h->d_tab_len, &h->d_tab, &h->d_ls, &h->d_sort, &h->d_best, &h->d_pb, &h->d_rows,
                      &h->d_cand_block, &h->d_win_block, &h->d_ctrl, &h->d_fb_list, &h->d_scratch,
                      &h->d_cells, &h->d_sweep, &h->d_summary, &h->d_dbg};
    for (DevBuf* b : bufs) b->release();
    h->stage.release();
    h->out_stage.release();
    h->sz_pin.release();
    if (h->ev_k0) cudaEventDestroy(h->ev_k0);
    if (h->ev_k1) cudaEventDestroy(h->ev_k1);
    if (h->ev_d0) cudaEventDestroy(h->ev_d0);
    if (h->ev_d1) cudaEventDestroy(h->ev_d1);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

// ---------------------------------------------------------------------------
// Winner-block all-gather over peer memory (NVLink / NVSwitch), fused into ONE kernel per step:
// CTA d copies this rank's block into rank d's gathered buffer (slot = this rank) with plain peer
// stores, publishes the step's epoch in rank d's flag word for this rank (release, system scope),
// then waits until rank d's block has arrived HERE.  When the kernel retires every slot of the
// local gathered buffer holds this step's blocks.  Two buffer parities: a fast rank may already
// publish step e+1 while a slow one still reads step e.  The payload is 40 B per server, so the
// exchange is latency: two NVLink hops instead of a library collective's launch + protocol.
// ---------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) xchg_publish(const char* __restrict__ src, size_t bytes, char* const* __restrict__ peers,
                                                    int world, int rank, size_t slot_stride, size_t flags_off,
                                                    unsigned long long epoch, int* err) {
    const int d = blockIdx.x;
    const size_t parity_off = (size_t)(epoch & 1ull) * (size_t)world * slot_stride;
    char* dst = peers[d] + parity_off + (size_t)rank * slot_stride;
    const size_t n16 = bytes / 16;
    for (size_t i = threadIdx.x; i < n16; i += blockDim.x) ((int4*)dst)[i] = ((const int4*)src)[i];
    for (size_t i = 16 * n16 + threadIdx.x; i < bytes; i += blockDim.x) dst[i] = src[i];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        // my flag word in rank d's memory: flags[src rank]
        volatile unsigned long long* theirs = (volatile unsigned long long*)(peers[d] + flags_off) + rank;
        *theirs = epoch;
        __threadfence_system();
        // wait for rank d's block of this epoch in MY memory
        volatile unsigned long long* mine = (volatile unsigned long long*)(peers[rank] + flags_off) + d;
        const long long t0 = clock64();
        while (*mine < epoch) {
            if (clock64() - t0 > (4ll << 30)) {  // ~2 s: a peer is gone; report instead of hanging the GPU
                *err = 1;
                break;
            }
            __nanosleep(200);
        }
        __threadfence_system();
    }
}
}  // namespace

extern "C" {
int wva_xchg_create(wva_handle* h, int world, int rank, size_t block_bytes, void* ipc_handle_out /* 64 bytes */) {
    if (!h || world < 1 || rank < 0 || rank >= world || !ipc_handle_out) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    auto& x = h->xchg;
    x.world = world;
    x.rank = rank;
    x.block_bytes = block_bytes;
    x.slot_stride = (block_bytes + 255) / 256 * 256;
    x.flags_off = 2 * (size_t)world * x.slot_stride;
    x.local_bytes = x.flags_off + 8 * (size_t)world + 256;
    CK(cudaMalloc((void**)&x.local, x.local_bytes));  // its own allocation: IPC exports whole allocations
    CK(cudaMemset(x.local, 0, x.local_bytes));
    CK(cudaMalloc((void**)&x.d_peer, sizeof(char*) * world));
    CK(cudaMalloc((void**)&x.d_err, sizeof(int)));
    CK(cudaMemset(x.d_err, 0, sizeof(int)));
    x.peer.assign(world, nullptr);
    x.peer[rank] = x.local;
    x.epoch = 0;
    cudaIpcMemHandle_t hd;
    CK(cudaIpcGetMemHandle(&hd, x.local));
    static_assert(sizeof(hd) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(ipc_handle_out, &hd, sizeof(hd));
    return WVA_OK;
}
int wva_xchg_open(wva_handle* h, int peer_rank, const void* ipc_handle) {
    if (!h || !ipc_handle || peer_rank < 0 || peer_rank >= h->xchg.world) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    auto& x = h->xchg;
    if (peer_rank != x.rank) {
        cudaIpcMemHandle_t hd;
        memcpy(&hd, ipc_handle, sizeof(hd));
        void* p = nullptr;
        CK(cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
        x.peer[peer_rank] = (char*)p;
    }
    bool all = true;
    for (char* p : x.peer) all = all && p != nullptr;
    if (all) CK(cudaMemcpy(x.d_peer, x.peer.data(), sizeof(char*) * x.world, cudaMemcpyHostToDevice));
    return WVA_OK;
}
// Enqueue the exchange of `src_block` (device memory, block_bytes) on the handle's stream; returns the
// device address of the gathered buffer of this step ([world][slot_stride] bytes) in *gathered.
int wva_xchg_publish(wva_handle* h, const void* src_block, void** gathered, size_t* slot_stride) {
    if (!h || !src_block || h->xchg.world < 1 || !h->xchg.d_peer) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    auto& x = h->xchg;
    for (char* p : x.peer)
        if (!p) return h->fail(WVA_ERR_STATE, "wva_xchg_publish: not every peer buffer is open");
    ++x.epoch;
    xchg_publish<<<x.world, 256, 0, h->stream>>>((const char*)src_block, x.block_bytes, x.d_peer, x.world, x.rank, x.slot_stride,
                                                 x.flags_off, x.epoch, x.d_err);
    h->launches++;
    if (gathered) *gathered = x.local + (size_t)(x.epoch & 1ull) * (size_t)x.world * x.slot_stride;
    if (slot_stride) *slot_stride = x.slot_stride;
    CK(cudaGetLastError());
    return WVA_OK;
}
int wva_xchg_error(wva_handle* h) {  // after a synchronize: 1 = a peer never arrived
    if (!h || !h->xchg.d_err) return 0;
    int e = 0;
    cudaMemcpy(&e, h->xchg.d_err, sizeof(int), cudaMemcpyDeviceToHost);
    return e;
}
int wva_xchg_destroy(wva_handle* h) {
    if (!h) return WVA_ERR_BAD_ARG;
    auto& x = h->xchg;
    cudaSetDevice(h->device);
    for (int r = 0; r < (int)x.peer.size(); ++r)
        if (r != x.rank && x.peer[r]) cudaIpcCloseMemHandle(x.peer[r]);
    if (x.local) cudaFree(x.local);
    if (x.d_peer) cudaFree(x.d_peer);
    if (x.d_err) cudaFree(x.d_err);
    x = wva_handle::Xchg();
    return WVA_OK;
}
}  // extern "C"

void* wva_stream(wva_handle* h) { return h ? (void*)h->stream : nullptr; }

int wva_synchronize(wva_handle* h) {
    if (!h) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return WVA_OK;
}

int64_t wva_launch_count(const wva_handle* h) { return h ? h->launches : 0; }
float wva_last_kernel_ms(const wva_handle* h) { return h ? h->last_kernel_ms : 0.f; }
float wva_last_device_ms(const wva_handle* h) { return h ? h->last_device_ms : 0.f; }

int wva_upload(wva_handle* h, const wva_fleet* fleet) {
    if (!h) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    int rc = upload_fleet(h, fleet);
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));
    return WVA_OK;
}

int wva_update_load(wva_handle* h, const float* arrival_rpm, const int32_t* in_tokens, const int32_t* out_tokens) {
    if (!h) return WVA_ERR_BAD_ARG;
    if (!h->resident) return h->fail(WVA_ERR_STATE, "no resident fleet (call wva_upload first)");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));  // the pinned stage may still feed an earlier async copy
    HostFleet& hf = h->hf;
    const size_t S = hf.S;
    bool tokens_changed = false, class_changed = false;
    if (arrival_rpm) {
        for (size_t s = 0; s < S && !class_changed; ++s)
            class_changed = ((arrival_rpm[s] == 0.0f) != (hf.srv_arrival_rpm[s] == 0.0f)) ||
                            ((arrival_rpm[s] < 0.0f) != (hf.srv_arrival_rpm[s] < 0.0f));
        hf.srv_arrival_rpm.assign(arrival_rpm, arrival_rpm + S);
        memcpy((char*)h->stage.p + h->col_rate.off, arrival_rpm, 4 * S);
    }
    if (in_tokens) {
        tokens_changed = tokens_changed || !std::equal(in_tokens, in_tokens + S, hf.srv_in_tokens.begin());
        hf.srv_in_tokens.assign(in_tokens, in_tokens + S);
        memcpy((char*)h->stage.p + h->col_in.off, in_tokens, 4 * S);
    }
    if (out_tokens) {
        tokens_changed = tokens_changed || !std::equal(out_tokens, out_tokens + S, hf.srv_out_tokens.begin());
        hf.srv_out_tokens.assign(out_tokens, out_tokens + S);
        memcpy((char*)h->stage.p + h->col_out.off, out_tokens, 4 * S);
    }
    // the three load columns are adjacent in the arena: one copy
    const size_t lo = h->col_rate.off, hi = h->col_out.off + h->col_out.bytes;
    if (S) CK(cudaMemcpyAsync((char*)h->arena.p + lo, (char*)h->stage.p + lo, hi - lo, cudaMemcpyHostToDevice, h->stream));
    if (tokens_changed || class_changed) h->epoch_tokens++;
    h->last_kind = 0;
    return WVA_OK;
}

int wva_analyze(wva_handle* h, const wva_fleet* fleet, wva_allocs* candidates) {
    if (!h || !candidates) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    int rc = upload_fleet(h, fleet);
    if (rc) return rc;
    // Server.Calculate also assigns value = transition penalty: run the unlimited
    // kernel into a scratch winner block so that candidate values are final
    wva_allocs dummy{};
    return run_size_host(h, candidates, &dummy);
}

// SolveGreedy + best-effort policies over a candidate table the caller already holds (host only, no device work):
// the multi-GPU limited mode all-gathers the per-shard candidate tables and runs this redundantly on every rank.
int wva_solve_greedy(const wva_fleet* fleet, wva_allocs* candidates, wva_allocs* winners) {
    if (fleet_problem(fleet) || !winners) return WVA_ERR_BAD_ARG;
    HostFleet hf;
    fill_host_fleet(hf, fleet);
    for (int a = 0; a < hf.A; ++a)
        if (hf.T <= 0 || hf.acc_type[a] < 0 || hf.acc_type[a] >= hf.T) return WVA_ERR_BAD_ARG;
    std::vector<HostCand> cand, win((size_t)hf.S);
    if (!abi_to_cands(candidates, (size_t)hf.S * hf.A, cand)) return WVA_ERR_BAD_ARG;
    GreedySolver(hf, cand, win).run();
    cands_to_abi(cand, candidates);
    cands_to_abi(win, winners);
    return WVA_OK;
}

int wva_resolve(wva_handle* h, wva_allocs* candidates, wva_allocs* winners) {
    if (!h || !winners) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    if (!h->resident) return h->fail(WVA_ERR_STATE, "no resident fleet (call wva_upload first)");
    if (!h->hf.unlimited) return run_greedy_host(h, candidates, winners);
    const int rc = run_size_host(h, candidates, winners);
    if (rc == WVA_OK) h->last_kind = 1;
    return rc;
}

int wva_resolve_scenarios(wva_handle* h, int32_t n_scen, const float* arrival_rpm, wva_allocs* candidates,
                          wva_allocs* winners) {
    if (!h || n_scen < 1 || !arrival_rpm || !winners) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    if (!h->resident) return h->fail(WVA_ERR_STATE, "no resident fleet (call wva_upload first)");
    h->last_kind = 0;  // like wva_update_load: the scenarios are not a solution of the resident fleet
    if (n_scen > 65535 || (long long)n_scen * h->hf.S * h->hf.A > 0x7fffffffll)
        return h->fail(WVA_ERR_UNSUPPORTED, "n_scen above 65535 or n_scen * S * A above 2^31 - 1");
    return run_scenarios(h, n_scen, arrival_rpm, candidates, winners);
}

int wva_solve(wva_handle* h, const wva_fleet* fleet, wva_allocs* candidates, wva_allocs* winners) {
    if (!h || !winners) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    int rc = upload_fleet(h, fleet);
    if (rc) return rc;
    return wva_resolve(h, candidates, winners);
}

int wva_resolve_device(wva_handle* h, wva_allocs* winners_dev) {
    if (!h || !winners_dev) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    if (!h->resident) return h->fail(WVA_ERR_STATE, "no resident fleet (call wva_upload first)");
    if (!h->hf.unlimited) return h->fail(WVA_ERR_UNSUPPORTED, "limited (greedy) mode has host outputs only: use wva_resolve");
    const HostFleet& hf = h->hf;
    const Block bc = block_layout((size_t)hf.S * hf.A);
    CK(h->d_cand_block.ensure(bc.bytes + 16));
    const AllocCols dc = block_cols(h->d_cand_block.p, bc);
    const AllocCols dw = cols_from_abi(winners_dev);
    CK(cudaEventRecord(h->ev_d0, h->stream));
    int rc = enqueue_size(h, dc, &dw);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev_d1, h->stream));
    return WVA_OK;
}

int wva_grid_solve_device(wva_handle* h, const wva_grid* grid, wva_allocs* winners_dev) {
    if (!h || !winners_dev) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    if (!h->resident) return h->fail(WVA_ERR_STATE, "no resident fleet (call wva_upload first)");
    int rc = validate_grid(h, grid);
    if (rc) return rc;
    rc = ensure_ctrl(h);
    if (rc) return rc;
    GridPlan plan;
    rc = prepare_grid(h, grid, &plan);
    if (rc) return rc;
    rc = ensure_cells(h, plan, false, false);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev_d0, h->stream));
    rc = enqueue_grid(h, plan, cols_from_abi(winners_dev));
    if (rc) return rc;
    CK(cudaEventRecord(h->ev_d1, h->stream));
    return WVA_OK;
}

int wva_grid_solve(wva_handle* h, const wva_fleet* fleet, const wva_grid* grid, wva_cells* cells, wva_allocs* winners) {
    if (!h || !winners) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    int rc = validate_grid(h, grid);
    if (rc) return rc;
    rc = upload_fleet(h, fleet);
    if (rc) return rc;
    rc = ensure_ctrl(h);
    if (rc) return rc;
    GridPlan plan;
    rc = prepare_grid(h, grid, &plan);
    if (rc) return rc;
    const HostFleet& hf = h->hf;
    const Block bw = block_layout(hf.S);
    CK(h->d_win_block.ensure(bw.bytes + 16));
    const AllocCols dw = block_cols(h->d_win_block.p, bw);
    // per-cell columns live on the device for every solve; they travel to the host only on request
    const size_t nc = plan.n_cells;
    const bool want_cells = cells && (cells->flags || cells->ttft || cells->itl || cells->rho || cells->throughput);
    rc = ensure_cells(h, plan, want_cells, want_cells && cells->throughput);
    if (rc) return rc;
    if (want_cells && nc)  // cells that are never analysed must read back as 0
        CK(cudaMemsetAsync(h->d_cells.p, 0, align_up(nc) + 4 * align_up(4 * nc), h->stream));
    CK(cudaEventRecord(h->ev_d0, h->stream));
    rc = enqueue_grid(h, plan, dw);
    if (rc) return rc;
    const size_t stage_bytes = align_up(bw.bytes) + 256;
    CK(h->out_stage.ensure(stage_bytes));
    char* hs = (char*)h->out_stage.p;
    if (bw.bytes) CK(cudaMemcpyAsync(hs, h->d_win_block.p, bw.bytes, cudaMemcpyDeviceToHost, h->stream));
    int* ctrl_host = (int*)(hs + align_up(bw.bytes));
    CK(cudaMemcpyAsync(ctrl_host, h->d_ctrl.p, CTRL_INTS * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (want_cells && nc) {
        const char* p = (const char*)h->d_cells.p;
        if (cells->flags) CK(cudaMemcpyAsync(cells->flags, p, nc, cudaMemcpyDeviceToHost, h->stream));
        if (cells->ttft) CK(cudaMemcpyAsync(cells->ttft, p + align_up(nc), 4 * nc, cudaMemcpyDeviceToHost, h->stream));
        if (cells->itl)
            CK(cudaMemcpyAsync(cells->itl, p + align_up(nc) + align_up(4 * nc), 4 * nc, cudaMemcpyDeviceToHost, h->stream));
        if (cells->rho)
            CK(cudaMemcpyAsync(cells->rho, p + align_up(nc) + 2 * align_up(4 * nc), 4 * nc, cudaMemcpyDeviceToHost, h->stream));
        if (cells->throughput)
            CK(cudaMemcpyAsync(cells->throughput, p + align_up(nc) + 3 * align_up(4 * nc), 4 * nc, cudaMemcpyDeviceToHost,
                               h->stream));
    }
    rc = finish_timing(h);
    if (rc) return rc;
    rc = check_fallback_status(h, ctrl_host, plan.args.fb_cap);
    if (rc) return rc;
    scatter_block(hs, bw, winners);
    h->last_kind = 1;
    return WVA_OK;
}

// System.AllocateByType + CreateAllocationDiff over the most recent solution (include/wva_b200.h).
int wva_summarize(wva_handle* h, wva_summary* out) {
    if (!h || !out) return WVA_ERR_BAD_ARG;
    CK(cudaSetDevice(h->device));
    if (!h->resident || h->last_kind == 0) return h->fail(WVA_ERR_STATE, "no solution to summarise (solve first)");
    const HostFleet& hf = h->hf;
    const size_t S = hf.S, T = hf.T;
    if (h->last_kind == 2) {  // greedy winners live on the host: same loops as the kernel
        for (size_t t = 0; t < T; ++t) {
            if (out->type_present) out->type_present[t] = 0;
            if (out->type_count) out->type_count[t] = 0;
            if (out->type_limit) out->type_limit[t] = hf.type_capacity[t];
            if (out->type_cost) out->type_cost[t] = 0.0f;
        }
        std::vector<float> cost(T, 0.0f);
        std::vector<int64_t> cnt(T, 0);
        for (size_t s = 0; s < S; ++s) {
            const int feas = h->last_feasible[s], acc = h->last_acc[s], rep = h->last_replicas[s];
            const float c = h->last_cost[s];
            const int m = hf.srv_model[s];
            if (feas && acc >= 0 && acc < hf.A && m >= 0 && m < hf.M) {
                const int t = hf.acc_type[acc];
                if (t >= 0 && t < hf.T) {
                    int inst = 0;
                    if (hf.perf_present[(size_t)m * hf.A + acc]) {
                        inst = hf.perf_acc_count[(size_t)m * hf.A + acc];
                        if (inst <= 0) inst = 1;
                    }
                    cnt[t] += (int64_t)rep * inst * (int64_t)hf.acc_mult[acc];
                    cost[t] = cost[t] + c;
                    if (out->type_present) out->type_present[t] = 1;
                }
            }
            if (out->diff_old_acc) out->diff_old_acc[s] = hf.srv_cur_acc[s];
            if (out->diff_old_replicas) out->diff_old_replicas[s] = hf.srv_cur_replicas[s];
            if (out->diff_new_acc) out->diff_new_acc[s] = feas ? acc : WVA_ACC_ABSENT;
            if (out->diff_new_replicas) out->diff_new_replicas[s] = feas ? rep : 0;
            if (out->diff_cost) out->diff_cost[s] = (feas ? c : 0.0f) - hf.srv_cur_cost[s];
        }
        for (size_t t = 0; t < T; ++t) {
            if (out->type_count) out->type_count[t] = cnt[t];
            if (out->type_cost) out->type_cost[t] = cost[t];
        }
        return WVA_OK;
    }
    if (T > (size_t)kSumMaxTypes) return h->fail(WVA_ERR_UNSUPPORTED, "more accelerator types than summary_kernel owns");
    // device winner block of the last solve
    const Block bw = block_layout(S);
    const AllocCols dw = block_cols(h->d_win_block.p, bw);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + std::max<size_t>(bytes, 1), 16); return at; };
    const size_t o_cnt = take(8 * T), o_pres = take(T), o_lim = take(4 * T), o_cost = take(4 * T);
    const size_t o_oa = take(4 * S), o_na = take(4 * S), o_or = take(4 * S), o_nr = take(4 * S), o_dc = take(4 * S);
    CK(h->d_summary.ensure(o));
    CK(h->out_stage.ensure(o));
    char* d = (char*)h->d_summary.p;
    SummaryOut so;
    so.type_count = (long long*)(d + o_cnt);
    so.type_present = (uint8_t*)(d + o_pres);
    so.type_limit = (int*)(d + o_lim);
    so.type_cost = (float*)(d + o_cost);
    so.diff_old_acc = (int*)(d + o_oa);
    so.diff_new_acc = (int*)(d + o_na);
    so.diff_old_replicas = (int*)(d + o_or);
    so.diff_new_replicas = (int*)(d + o_nr);
    so.diff_cost = (float*)(d + o_dc);
    summary_kernel<<<1, 256, 0, h->stream>>>(h->df, dw, so);
    h->launches++;
    CK(cudaGetLastError());
    char* hs = (char*)h->out_stage.p;
    CK(cudaMemcpyAsync(hs, d, o, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (out->type_count) memcpy(out->type_count, hs + o_cnt, 8 * T);
    if (out->type_present) memcpy(out->type_present, hs + o_pres, T);
    if (out->type_limit) memcpy(out->type_limit, hs + o_lim, 4 * T);
    if (out->type_cost) memcpy(out->type_cost, hs + o_cost, 4 * T);
    if (out->diff_old_acc) memcpy(out->diff_old_acc, hs + o_oa, 4 * S);
    if (out->diff_new_acc) memcpy(out->diff_new_acc, hs + o_na, 4 * S);
    if (out->diff_old_replicas) memcpy(out->diff_old_replicas, hs + o_or, 4 * S);
    if (out->diff_new_replicas) memcpy(out->diff_new_replicas, hs + o_nr, 4 * S);
    if (out->diff_cost) memcpy(out->diff_cost, hs + o_dc, 4 * S);
    return WVA_OK;
}

// MM1KModel.Solve for n triples (include/wva_b200.h).
int wva_mm1k_solve(wva_handle* h, int32_t n, const int32_t* K, const float* lambda, const float* mu, wva_mm1k_out* out) {
    if (!h || !out || n < 0 || (n > 0 && (!K || !lambda || !mu))) return WVA_ERR_BAD_ARG;
    if (n == 0) return WVA_OK;
    for (int i = 0; i < n; ++i)
        if (K[i] < 0) return h->fail(WVA_ERR_BAD_ARG, "MM1K: negative K");  // NewMM1KModel returns nil (mm1kmodel.go:20-22)
    for (int i = 0; i < n; ++i)  // one thread walks the K + 1 states of a triple: bound the launch
        if (K[i] > (1 << 20)) return h->fail(WVA_ERR_UNSUPPORTED, "MM1K: K above 2^20");
    CK(cudaSetDevice(h->device));
    const size_t N = (size_t)n;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes, 16); return at; };
    const size_t i_K = take(4 * N), i_lam = take(4 * N), i_mu = take(4 * N);
    const size_t in_bytes = o;
    const size_t o_sum = take(8 * N), o_valid = take(N), o_rho = take(4 * N), o_nsys = take(4 * N), o_thr = take(4 * N),
                 o_resp = take(4 * N), o_serv = take(4 * N), o_wait = take(4 * N), o_qlen = take(4 * N);
    CK(h->d_summary.ensure(o));
    CK(h->out_stage.ensure(o));
    char* d = (char*)h->d_summary.p;
    char* hs = (char*)h->out_stage.p;
    memcpy(hs + i_K, K, 4 * N);
    memcpy(hs + i_lam, lambda, 4 * N);
    memcpy(hs + i_mu, mu, 4 * N);
    CK(cudaMemcpyAsync(d, hs, in_bytes, cudaMemcpyHostToDevice, h->stream));
    Mm1kArgs g;
    g.n = n;
    g.K = (const int*)(d + i_K);
    g.lambda = (const float*)(d + i_lam);
    g.mu = (const float*)(d + i_mu);
    g.sum_p = (double*)(d + o_sum);
    g.is_valid = (uint8_t*)(d + o_valid);
    g.rho = (float*)(d + o_rho);
    g.avg_num_in_system = (float*)(d + o_nsys);
    g.throughput = (float*)(d + o_thr);
    g.avg_resp_time = (float*)(d + o_resp);
    g.avg_serv_time = (float*)(d + o_serv);
    g.avg_wait_time = (float*)(d + o_wait);
    g.avg_queue_length = (float*)(d + o_qlen);
    mm1k_kernel<<<(unsigned)((N + 127) / 128), 128, 0, h->stream>>>(g);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(hs + in_bytes, d + in_bytes, o - in_bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (out->sum_p) memcpy(out->sum_p, hs + o_sum, 8 * N);
    if (out->is_valid) memcpy(out->is_valid, hs + o_valid, N);
    if (out->rho) memcpy(out->rho, hs + o_rho, 4 * N);
    if (out->avg_num_in_system) memcpy(out->avg_num_in_system, hs + o_nsys, 4 * N);
    if (out->throughput) memcpy(out->throughput, hs + o_thr, 4 * N);
    if (out->avg_resp_time) memcpy(out->avg_resp_time, hs + o_resp, 4 * N);
    if (out->avg_serv_time) memcpy(out->avg_serv_time, hs + o_serv, 4 * N);
    if (out->avg_wait_time) memcpy(out->avg_wait_time, hs + o_wait, 4 * N);
    if (out->avg_queue_length) memcpy(out->avg_queue_length, hs + o_qlen, 4 * N);
    return WVA_OK;
}

int wva_sweep(wva_handle* h, const wva_fleet* fleet, int32_t n_rates, wva_sweep_out* out) {
    if (!h || !out || n_rates < 1) return WVA_ERR_BAD_ARG;
    if (!out->valid || !out->rate || !out->ttft || !out->itl || !out->throughput || !out->rho)
        return h->fail(WVA_ERR_BAD_ARG, "NULL sweep output column");
    CK(cudaSetDevice(h->device));
    int rc = upload_fleet(h, fleet);
    if (rc) return rc;
    rc = ensure_ctrl(h);
    if (rc) return rc;
    const HostFleet& hf = h->hf;
    const int A = hf.A, S = hf.S;
    // every (server, acc) with a profile, ignoring keepAccelerator; sorted by descending N
    std::vector<int> pairs, Ns((size_t)S * A, 0);
    for (int s = 0; s < S; ++s)
        for (int a = 0; a < A; ++a) {
            const int m = hf.srv_model[s];
            if (hf.srv_in_tokens[s] < 0 || hf.srv_out_tokens[s] < 1 || m < 0 || m >= hf.M ||
                !hf.perf_present[(size_t)m * A + a])
                continue;
            const int N = hf.pair_batch(s, a);
            if (N > (1 << 20)) return h->fail(WVA_ERR_UNSUPPORTED, "batch size above 2^20");
            Ns[(size_t)s * A + a] = N;
            pairs.push_back(s * A + a);
        }
    std::stable_sort(pairs.begin(), pairs.end(), [&](int x, int y) { return Ns[x] > Ns[y]; });
    const int n = (int)pairs.size();
    std::vector<int> lens(n);
    std::vector<long long> offs(n);
    long long off = 0;
    for (int e = 0; e < n; ++e) {
        lens[e] = Ns[pairs[e]];
        offs[e] = off;
        off += lens[e];
    }
    const size_t n_out = (size_t)S * A * n_rates;
    const size_t out_bytes = align_up(n_out) + 5 * align_up(4 * n_out);
    CK(h->d_sweep.ensure(std::max<size_t>(out_bytes, 256)));
    char* p = (char*)h->d_sweep.p;
    CK(cudaMemsetAsync(p, 0, std::max<size_t>(out_bytes, 256), h->stream));
    CK(cudaEventRecord(h->ev_d0, h->stream));
    CK(cudaEventRecord(h->ev_k0, h->stream));
    long long fb_cap = 0;
    if (n) {
        CK(h->d_tab_pair.ensure(sizeof(int) * n));
        CK(h->d_tab_off.ensure(sizeof(long long) * n));
        CK(h->d_tab_len.ensure(sizeof(int) * n));
        CK(h->d_tab.ensure(sizeof(double) * 4 * (size_t)off));
        CK(cudaMemcpyAsync(h->d_tab_pair.p, pairs.data(), sizeof(int) * n, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_tab_off.p, offs.data(), sizeof(long long) * n, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_tab_len.p, lens.data(), sizeof(int) * n, cudaMemcpyHostToDevice, h->stream));
        h->grid_epoch = ~0ull;  // the shared-table buffers now hold sweep tables
        build_pair_tables<<<n, 128, 0, h->stream>>>(h->df, (const int*)h->d_tab_pair.p, (const long long*)h->d_tab_off.p,
                                                    (const int*)h->d_tab_len.p, n, (double*)h->d_tab.p, nullptr,
                                                    nullptr, 0, nullptr);
        h->launches++;
        SweepArgs g{};
        g.f = h->df;
        g.pair_list = (const int*)h->d_tab_pair.p;
        g.pair_N = (const int*)h->d_tab_len.p;
        g.tab_off = (const long long*)h->d_tab_off.p;
        g.tab = (const double*)h->d_tab.p;
        g.n_pairs = n;
        g.n_rates = n_rates;
        g.n_chunks = (n_rates + 31) / 32;
        g.counter = (unsigned*)h->d_ctrl.p + CTRL_COUNTER;
        g.valid = (uint8_t*)p;
        g.rate = (float*)(p + align_up(n_out));
        g.ttft = (float*)(p + align_up(n_out) + align_up(4 * n_out));
        g.itl = (float*)(p + align_up(n_out) + 2 * align_up(4 * n_out));
        g.throughput = (float*)(p + align_up(n_out) + 3 * align_up(4 * n_out));
        g.rho = (float*)(p + align_up(n_out) + 4 * align_up(4 * n_out));
        g.fb_count = (int*)h->d_ctrl.p + CTRL_FB_COUNT;
        fb_cap = (long long)std::min<size_t>((size_t)n * n_rates, (size_t)1 << 22);
        g.fb_cap = (int)fb_cap;
        CK(h->d_fb_list.ensure(sizeof(long long) * g.fb_cap));
        g.fb_points = (long long*)h->d_fb_list.p;
        // The fallback's scratch is sized for the longest chain before the launch, as the grid and size paths do:
        // 128 slots of (K + 1) doubles, about 12 GB at N = 2^20 with the default queue ratio, kept by the handle.
        size_t slot_doubles;
        int Kmax;
        rc = ensure_scratch(h, lens[0], hf.tun.max_queue_to_batch_ratio, &slot_doubles, &Kmax);  // lens: descending
        if (rc) return rc;
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sweep_kernel, 256, 0));
        per_sm = std::max(1, std::min(per_sm, 8));
        const unsigned items = (unsigned)n * g.n_chunks;
        unsigned blocks = std::min<unsigned>((unsigned)(h->sm_count * per_sm), (items + 7) / 8);
        CK(cudaEventRecord(h->ev_k0, h->stream));
        sweep_kernel<<<blocks, 256, 0, h->stream>>>(g);
        CK(cudaEventRecord(h->ev_k1, h->stream));
        sweep_fallback<<<kFbBlocks, kFbThreads, 0, h->stream>>>(g, (double*)h->d_scratch.p, slot_doubles, Kmax,
                                                                (int*)h->d_ctrl.p + CTRL_FB_STATUS);
        h->launches += 2;
        CK(cudaGetLastError());
    } else {
        CK(cudaEventRecord(h->ev_k1, h->stream));
    }
    CK(h->out_stage.ensure(256));
    int* ctrl_host = (int*)h->out_stage.p;
    CK(cudaMemcpyAsync(ctrl_host, h->d_ctrl.p, CTRL_INTS * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (n_out) {
        CK(cudaMemcpyAsync(out->valid, p, n_out, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(out->rate, p + align_up(n_out), 4 * n_out, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(out->ttft, p + align_up(n_out) + align_up(4 * n_out), 4 * n_out, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(out->itl, p + align_up(n_out) + 2 * align_up(4 * n_out), 4 * n_out, cudaMemcpyDeviceToHost,
                           h->stream));
        CK(cudaMemcpyAsync(out->throughput, p + align_up(n_out) + 3 * align_up(4 * n_out), 4 * n_out,
                           cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(out->rho, p + align_up(n_out) + 4 * align_up(4 * n_out), 4 * n_out, cudaMemcpyDeviceToHost,
                           h->stream));
    }
    rc = finish_timing(h);
    if (rc) return rc;
    return check_fallback_status(h, ctrl_host, fb_cap);
}

// ---- self-check of the exact-division primitive (not part of the public ABI) ------------------
// Compares div_recip (Markstein correction around a double-word reciprocal) with div.rn.f64 on
// pseudo-random operands drawn from the solver's exponent windows, including adversarial
// divisors next to powers of two and float32-valued divisors.  Returns the mismatch count.
__global__ void div_selfcheck_kernel(unsigned long long seed, int iters, unsigned long long* mismatches) {
    unsigned long long x = seed ^ (0x9E3779B97F4A7C15ull * (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x + 1));
    auto next = [&]() {  // xorshift64*
        x ^= x >> 12; x ^= x << 25; x ^= x >> 27;
        return x * 0x2545F4914F6CDD1Dull;
    };
    unsigned long long bad = 0;
    for (int it = 0; it < iters; ++it) {
        const unsigned long long r0 = next(), r1 = next(), r2 = next();
        // divisor: mantissa random / float32-valued / all-ones / one-above-power-of-two; exponent in [-60, 60]
        unsigned long long mb = r0 & 0x000FFFFFFFFFFFFFull;
        switch (r2 & 3) {
        case 0: mb &= 0x000FFFFFE0000000ull; break;                 // float32-valued (24-bit significand)
        case 1: mb = 0x000FFFFFFFFFFFFFull - (r0 & 0xff); break;    // just below a power of two
        case 2: mb = r0 & 0xff; break;                              // just above a power of two
        default: break;
        }
        const long long eb = (long long)((r2 >> 8) % 121) - 60;
        const double b = __longlong_as_double((long long)(((unsigned long long)(1023 + eb) << 52) | mb));
        // dividend: random mantissa (sometimes all ones), exponent in [-340, 940] (p * lambda)
        unsigned long long ma = r1 & 0x000FFFFFFFFFFFFFull;
        if (((r2 >> 20) & 7) == 0) ma = 0x000FFFFFFFFFFFFFull - (r1 & 0xf);
        const long long ea = (long long)((r2 >> 24) % 1281) - 340;
        const double a = __longlong_as_double((long long)(((unsigned long long)(1023 + ea) << 52) | ma));
        const Recip rc = make_recip(b);
        const double q = div_recip(a, rc), want = __ddiv_rn(a, b);
        if (__double_as_longlong(q) != __double_as_longlong(want)) ++bad;
        // the cheaper low word used for the normalising sum (zl = RN(e * zh))
        Recip z = rc;
        z.yl = __dmul_rn(__fma_rn(-b, rc.yh, 1.0), rc.yh);
        const double q2 = div_recip(a, z);
        if (__double_as_longlong(q2) != __double_as_longlong(want)) ++bad;
        // the tail step with the pre-multiplied low word (step_recip): p in [2^-280, 2^880), float32 lambda in
        // [2^-60, 2^60]
        {
            const unsigned long long r3 = next();
            const long long ep = (long long)(r3 % 1160) - 280;
            const double pp = __longlong_as_double((long long)(((unsigned long long)(1023 + ep) << 52) | ma));
            const long long el = (long long)((r3 >> 12) % 121) - 60;
            const double lam = __longlong_as_double(
                (long long)(((unsigned long long)(1023 + el) << 52) | ((r3 >> 20) & 0x000FFFFFE0000000ull)));
            const double got = step_recip(pp, lam, __dmul_rn(lam, rc.yl), rc);
            const double want3 = __ddiv_rn(__dmul_rn(pp, lam), b);
            if (__double_as_longlong(got) != __double_as_longlong(want3)) ++bad;
        }
        // the division by the normalising sum: sum in [1, 2^900), p in [max(2^-280, sum * 2^-960), sum]
        {
            const unsigned long long r4 = next(), r5 = next();
            const long long es = (long long)(r4 % 900);
            const double S = __longlong_as_double((long long)(((unsigned long long)(1023 + es) << 52) | (r5 & 0x000FFFFFFFFFFFFFull)));
            const long long lo = es - 959 > -280 ? es - 959 : -280;
            const long long epp = lo + (long long)((r4 >> 16) % (unsigned long long)(es - lo + 1));
            const double pp = __longlong_as_double((long long)(((unsigned long long)(1023 + epp) << 52) | mb));
            Recip zz;
            zz.b = S;
            zz.yh = __ddiv_rn(1.0, S);
            zz.yl = __dmul_rn(__fma_rn(-S, zz.yh, 1.0), zz.yh);
            const double got = div_recip(pp, zz), want4 = __ddiv_rn(pp, S);
            if (__double_as_longlong(got) != __double_as_longlong(want4)) ++bad;
        }
    }
    if (bad) atomicAdd(mismatches, bad);
}

// ---- diagnostics (not part of the public ABI) ------------------------------------------
// Per-cell SM cycles of the last grid solve, in launch order, followed by the cell ids.
// Runs blocks*256*iters*2 random divisions; returns the number of results that differ from div.rn.f64.
long long wva_dbg_div_selfcheck(wva_handle* h, unsigned long long seed, int blocks, int iters) {
    if (!h) return -1;
    cudaSetDevice(h->device);
    unsigned long long* d = nullptr;
    if (cudaMalloc(&d, sizeof(unsigned long long)) != cudaSuccess) return -1;
    cudaMemsetAsync(d, 0, sizeof(unsigned long long), h->stream);
    div_selfcheck_kernel<<<blocks, 256, 0, h->stream>>>(seed, iters, d);
    unsigned long long out = ~0ull;
    cudaMemcpyAsync(&out, d, sizeof(out), cudaMemcpyDeviceToHost, h->stream);
    cudaStreamSynchronize(h->stream);
    cudaFree(d);
    return (long long)out;
}

#ifdef WVA_PROF
int wva_dbg_prof(long long* out, int reset) {
    if (reset) { long long z[16] = {0}; return (int)cudaMemcpyToSymbol(wva::wva_prof, z, sizeof(z)); }
    return (int)cudaMemcpyFromSymbol(out, wva::wva_prof, sizeof(long long) * 16);
}
#endif
int wva_dbg_read_plan(wva_handle* h, unsigned* out32) {  // grid_items_plan's queue plan: item_count[2*kClasses+1 ..+31]
    if (!h || !h->d_sort.p || !h->dbg_plan) return -1;
    return (int)cudaMemcpy(out32, h->dbg_plan, sizeof(unsigned) * 31, cudaMemcpyDeviceToHost);
}
int wva_dbg_enable_cycles(wva_handle* h, int on) {
    if (!h) return WVA_ERR_BAD_ARG;
    h->dbg_cycles = on != 0;
    return WVA_OK;
}
int wva_dbg_szcnt(unsigned long long* out24, int reset) {
#ifdef WVA_SZCNT
    if (reset) { unsigned long long z[24] = {0}; return (int)cudaMemcpyToSymbol(wva::wva_szcnt, z, sizeof(z)); }
    return (int)cudaMemcpyFromSymbol(out24, wva::wva_szcnt, sizeof(unsigned long long) * 24);
#else
    (void)out24; (void)reset;
    return -1;
#endif
}
long long wva_dbg_read_size(wva_handle* h, unsigned* out4, long long cap) {  // rows of {cycles, N | kind << 16, lambda bits, warp}
    if (!h || !h->d_dbg.p) return 0;
    const long long n = std::min<long long>((long long)h->dbg_n, cap);
    cudaMemcpy(out4, h->d_dbg.p, 16 * n, cudaMemcpyDeviceToHost);
    return n;
}
// Per (server, accelerator, replica level) of the last grid solve: the shared chain's last state (INT_MAX: none) and
// whether grid_rows resolved the row (§3.2b).  Returns the number of rows copied.
long long wva_dbg_read_rows(wva_handle* h, int* row_j, uint8_t* row_res, long long cap) {
    if (!h || !h->dbg_row_j) return 0;
    const long long n = std::min<long long>((long long)h->dbg_rows_n, cap);
    cudaMemcpy(row_j, h->dbg_row_j, sizeof(int) * n, cudaMemcpyDeviceToHost);
    cudaMemcpy(row_res, h->dbg_row_res, n, cudaMemcpyDeviceToHost);
    return n;
}
// Number of cells (grid), candidates (analyze / solve / resolve) or sweep points of the last call that left the
// streaming solve's exponent windows and were re-run on the stored-vector fallback (-1 without a handle).
int wva_dbg_fallback_count(wva_handle* h) { return h ? h->dbg_fb_count : -1; }
long long wva_dbg_read_cycles(wva_handle* h, unsigned* cycles, unsigned* cells, long long cap) {
    if (!h || !h->d_dbg.p) return 0;
    const long long n = std::min<long long>((long long)h->dbg_n, cap);
    cudaMemcpy(cycles, h->d_dbg.p, sizeof(unsigned) * n, cudaMemcpyDeviceToHost);
    cudaMemcpy(cells, (unsigned*)h->d_dbg.p + h->dbg_n, sizeof(unsigned) * n, cudaMemcpyDeviceToHost);
    return n;
}

}  // extern "C"
