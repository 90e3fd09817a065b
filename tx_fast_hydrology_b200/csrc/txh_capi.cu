// txh_capi.cu -- the C ABI declared in include/txh.h.
// Handles own the topology, the schedule and their device copies; all member-batched
// state lives in caller-owned device buffers.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/txh.h"
#include "txh_kernels.cuh"
#include "txh_topology.hpp"

using namespace txh;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what)
{
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? TXH_E_NODEVICE : TXH_E_CUDA;
}
#define CU(call)                                                   \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call);      \
    } while (0)

template <class T>
int upload(T** dptr, const std::vector<T>& v)
{
    const size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(T);
    CU(cudaMalloc((void**)dptr, bytes));
    if (!v.empty()) CU(cudaMemcpy(*dptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return TXH_OK;
}

// Grow-only device buffer of a handle: reallocated when `count` elements do not fit, once the handle's stream has
// drained (a queued launch may still read the old one); new memory is filled with the byte `fill` unless it is < 0.
template <class T>
int grow(T** buf, size_t* cap, size_t count, cudaStream_t st, int fill = -1)
{
    if (count <= *cap) return TXH_OK;
    if (*buf) { CU(cudaStreamSynchronize(st)); CU(cudaFree(*buf)); *buf = nullptr; *cap = 0; }
    CU(cudaMalloc((void**)buf, count * sizeof(T)));
    *cap = count;
    if (fill >= 0) CU(cudaMemsetAsync(*buf, fill, count * sizeof(T), st));
    return TXH_OK;
}

// Development aid (TXH_TRACE_FILE, TXH_LANE_TRACE): when the environment variable `env` names a file, `launch` runs
// with a zeroed device timeline of `words` counters in `trace`, which is then written to that file behind the header
// `hd` and `extra_bytes` of `extra` (synchronous).  Otherwise `launch` runs with trace == nullptr.
template <class Launch>
int traced_launch(const char* env, unsigned long long*& trace, size_t words, const long long (&hd)[4], const void* extra,
                  size_t extra_bytes, cudaStream_t st, Launch&& launch)
{
    const char* file = getenv(env);
    trace = nullptr;
    if (!file || !*file) { CU(launch()); return TXH_OK; }
    CU(cudaMalloc((void**)&trace, words * sizeof(unsigned long long)));
    CU(cudaMemsetAsync(trace, 0, words * sizeof(unsigned long long), st));
    CU(launch());
    std::vector<unsigned long long> h(words);
    CU(cudaMemcpyAsync(h.data(), trace, words * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaFree(trace));
    if (FILE* fp = fopen(file, "wb")) {
        fwrite(hd, sizeof(hd), 1, fp);
        if (extra_bytes) fwrite(extra, 1, extra_bytes, fp);
        fwrite(h.data(), sizeof(unsigned long long), h.size(), fp);
        fclose(fp);
    }
    return TXH_OK;
}

}  // namespace

struct txh_net {
    Topology topo;
    Schedule sched;
    std::vector<double> coef_host;      // [n][4] schedule order, then cumA [n], then linkA [n_link]
    bool have_coef = false, coef_dirty = false;
    // device side
    bool dev_ready = false;
    int num_sms = 0;
    unsigned long long watchdog_ns = 10000000000ull;
    TaskDesc* d_tasks = nullptr;
    int32_t *d_notify = nullptr, *d_init_ready = nullptr, *d_up_off = nullptr, *d_up_pos = nullptr, *d_lvl_pos = nullptr,
            *d_reach_of_pos = nullptr, *d_pos_of_reach = nullptr;
    uint32_t *d_hdr = nullptr, *d_inw = nullptr;
    uint8_t* d_outlet = nullptr;
    int32_t* d_inner = nullptr; int64_t n_inner = 0;   // schedule positions that have upstream reaches
    int4* d_inner_rec = nullptr;        // the same rows as {row, first three upstream rows | -1}; w == -2: more in the lists
    double* d_coef = nullptr;           // same layout as coef_host
    double* d_qtmp = nullptr;           // [n] schedule-order scratch for txh_route_step
    int32_t* d_pending = nullptr; size_t pairs_cap = 0;
    unsigned long long* d_queue = nullptr; size_t queue_cap = 0;
    double* d_side = nullptr; size_t side_cap = 0;   // side buffer [n_side][ld]
    unsigned long long* d_qctl = nullptr;     // [0] head, [1] tail, [2] completed, [4] status word
    int32_t* d_status = nullptr;
    StepInterp* d_steps = nullptr; size_t steps_cap = 0;
    StepInterp* d_unit_step = nullptr;
    int32_t* d_rec_slot = nullptr;
    int32_t* d_rec_pos = nullptr; size_t rec_pos_cap = 0;   // positions of the recorded reaches (txh_run_assimilating_rec)
    int32_t* d_tmp_idx = nullptr; size_t tmp_idx_cap = 0;
    int32_t* h_status = nullptr;        // pinned mirror of d_status (word 0) and the solver info (word 1)
    std::vector<int64_t> obs_cached;    // gauge list whose positions are resident in d_obs
    int32_t* d_obs = nullptr; size_t obs_cap = 0;
    int32_t* d_gauge_of_pos = nullptr;  // [n] gauge index of each schedule position, or -1
    // ensemble update applied by the next window launch while it loads its tasks (txh_run_assimilating, txh_window.cu)
    int32_t* d_gfix_off = nullptr;      // [window tasks + 1] gauge terms per task, for the gauges in obs_cached
    int2* d_gfix = nullptr; size_t gfix_cap = 0; bool gfix_ok = false;
    // window-mode kernel
    WTaskDesc* d_wtasks = nullptr;
    uint32_t *d_whdr = nullptr, *d_winw = nullptr;
    int32_t* d_wprod = nullptr;
    double* d_ring = nullptr; size_t ring_cap = 0; int ring_ld = 0;
    int route_kernel = 0;               // 0 auto (lane for small ensembles, else window), 1 dataflow, 2 window, 3 lane
    // lane kernel (txh_lane.cu): one schedule per member tile, built on first use
    struct LaneDev {
        LaneSchedule sched;
        bool built = false, ok = false, on_dev = false;
        LaneRegionDesc* d_regions = nullptr;
        int4* d_meta = nullptr;
        int32_t* d_xbeg = nullptr;
        uint16_t* d_child = nullptr;
    };
    LaneStep* d_lsteps = nullptr; size_t lsteps_cap = 0;
    LaneStep* d_unit_lstep = nullptr;
    LaneDev lane[5];                    // member tiles 1, 2, 4, 8, 16
    int lane_max_members = 4;           // ensembles up to this size may take the lane kernel (row state in registers)
    int lane_cap_rows = 0;              // rows per region; 0 = from the size of the network and the SM count
    int lane_ctas = 1;                  // regions (CTAs) per SM the schedule is sized for (measured: 1 is best, DESIGN.md)
    double* d_lring = nullptr; size_t lring_cap = 0;
    double* d_stage = nullptr; size_t stage_cap = 0;   // reach-order staging of txh_pack_host / txh_unpack_host
    double* stats_rowsum = nullptr;     // txh_set_stats_output: row sums of the final outflows of every txh_route_run
    double stats_scale = 1.0;
    double* T_hist = nullptr;           // txh_set_transform_history: update k of a run_assimilating call solves into
    int64_t T_hist_cap = 0;             // T_hist + k*M*M (capacity in doubles)
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> route_events;   // txh_run_assimilating(time_every > 0)
};

struct txh_forcing {
    txh_net* net;
    int64_t R, M;
    std::vector<double> times;
    double* d_times = nullptr;          // [R] the same on the device
    double* d_F = nullptr;              // [R][n] schedule order
    double* d_W = nullptr;              // [R][M] or nullptr
    // txh_forcing_update_async: the table arrives in row chunks on a copy stream of its own; a routing call waits
    // (on its stream) for the chunks its steps read
    cudaStream_t copy_stream = nullptr;
    double* d_stage = nullptr;          // [R][n] reach order, private to the handle
    cudaEvent_t reuse_ev = nullptr;
    std::vector<cudaEvent_t> chunk_ev;
    std::vector<int64_t> chunk_begin;   // first row of each chunk
    size_t waited = 0;                  // chunks the routing stream has been made to wait for
};

namespace {

int ensure_device(txh_net* net)
{
    if (net->dev_ready) return TXH_OK;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(TXH_E_NODEVICE, "no CUDA device visible: libtxh has no CPU fallback");
    }
    int dev = 0;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&net->num_sms, cudaDevAttrMultiProcessorCount, dev));
    const Schedule& s = net->sched;
    int rc;
    if ((rc = upload(&net->d_tasks, s.tasks))) return rc;
    if ((rc = upload(&net->d_notify, s.notify))) return rc;
    if ((rc = upload(&net->d_init_ready, s.init_ready))) return rc;
    if ((rc = upload(&net->d_hdr, s.hdr))) return rc;
    if ((rc = upload(&net->d_inw, s.inw))) return rc;
    if ((rc = upload(&net->d_up_off, s.up_off))) return rc;
    if ((rc = upload(&net->d_up_pos, s.up_pos))) return rc;
    {
        std::vector<int32_t> inner;                            // rows with upstream reaches (inflow_gain_kernel)
        for (int64_t k = 0; k < net->topo.n; ++k) if (s.up_off[k + 1] > s.up_off[k]) inner.push_back((int32_t)k);
        net->n_inner = (int64_t)inner.size();
        if ((rc = upload(&net->d_inner, inner))) return rc;
        std::vector<int4> rec(inner.size());
        for (size_t e = 0; e < inner.size(); ++e) {
            const int32_t k = inner[e], u0 = s.up_off[k], cnt = s.up_off[k + 1] - u0;
            // the sum keeps the order of the lists (first upstream reach first), like nutils.py:84-85 does per visit
            rec[e] = make_int4(k, s.up_pos[u0], cnt > 1 ? s.up_pos[u0 + 1] : -1, cnt > 3 ? -2 : (cnt > 2 ? s.up_pos[u0 + 2] : -1));
        }
        if ((rc = upload(&net->d_inner_rec, rec))) return rc;
    }
    if ((rc = upload(&net->d_lvl_pos, s.lvl_pos))) return rc;
    if ((rc = upload(&net->d_reach_of_pos, s.reach_of_pos))) return rc;
    if ((rc = upload(&net->d_pos_of_reach, s.pos_of_reach))) return rc;
    if ((rc = upload(&net->d_outlet, s.is_outlet_pos))) return rc;
    if ((rc = upload(&net->d_wtasks, s.wtasks))) return rc;
    if ((rc = upload(&net->d_whdr, s.whdr))) return rc;
    if ((rc = upload(&net->d_winw, s.winw))) return rc;
    if ((rc = upload(&net->d_wprod, s.wprod))) return rc;
    if (const char* k = getenv("TXH_ROUTE_KERNEL")) {
        if (!strcmp(k, "dataflow")) net->route_kernel = 1;
        else if (!strcmp(k, "window")) net->route_kernel = 2;
        else if (!strcmp(k, "lane")) net->route_kernel = 3;
    }
    if (const char* k = getenv("TXH_LANE_MAX_M")) net->lane_max_members = std::max(0, std::min(16, atoi(k)));
    if (const char* k = getenv("TXH_LANE_CAP")) net->lane_cap_rows = std::max(0, atoi(k));
    if (const char* k = getenv("TXH_LANE_CTAS")) net->lane_ctas = std::max(1, std::min(8, atoi(k)));
    CU(cudaMalloc((void**)&net->d_coef, sizeof(double) * (6 * net->topo.n + net->sched.link_last.size() + 1)));
    CU(cudaMalloc((void**)&net->d_qtmp, sizeof(double) * net->topo.n));
    CU(cudaMalloc((void**)&net->d_qctl, 64));
    net->d_status = reinterpret_cast<int32_t*>(net->d_qctl + 4);
    CU(cudaMemset(net->d_qctl, 0, 64));
    CU(cudaMalloc((void**)&net->d_rec_slot, sizeof(int32_t) * net->topo.n));
    CU(cudaMallocHost((void**)&net->h_status, 2 * sizeof(int32_t)));
    net->h_status[0] = net->h_status[1] = 0;
    const StepInterp unit{0, 0, 1.0, 0.0};
    CU(cudaMalloc((void**)&net->d_unit_step, sizeof(StepInterp)));
    CU(cudaMemcpy(net->d_unit_step, &unit, sizeof(unit), cudaMemcpyHostToDevice));
    if (const char* w = getenv("TXH_WATCHDOG_MS")) {
        const long ms = atol(w);
        if (ms > 0) net->watchdog_ns = (unsigned long long)ms * 1000000ull;
    }
    net->dev_ready = true;
    return TXH_OK;
}

int ensure_coef(txh_net* net, cudaStream_t st)
{
    if (!net->have_coef) return fail(TXH_E_STATE, "coefficients not set: call txh_compute_coeffs or txh_set_coeffs first");
    if (net->coef_dirty) {
        // synchronous on purpose: coef_host may be rewritten by the caller right after
        CU(cudaMemcpyAsync(net->d_coef, net->coef_host.data(), sizeof(double) * net->coef_host.size(),
                           cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));
        net->coef_dirty = false;
    }
    return TXH_OK;
}

// Synchronise `st` and report what the device recorded since the last report: a watchdog bail-out (status word)
// or a failed factorisation (info word).  Both words are cleared once reported, so the handle is usable again
// after the caller has re-uploaded a sane state; the rings of the persistent kernels are re-armed with them
// (an abandoned launch leaves cells behind).
int report_status(txh_net* net, cudaStream_t st)
{
    CU(cudaMemcpyAsync(net->h_status, net->d_status, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const int32_t status = net->h_status[0], info = net->h_status[1];
    if (status == 0 && info == 0) return TXH_OK;
    CU(cudaMemsetAsync(net->d_status, 0, 2 * sizeof(int32_t), st));
    if (status != 0) {
        if (net->d_ring) CU(cudaMemsetAsync(net->d_ring, 0xff, net->ring_cap * sizeof(double), st));
        if (net->d_lring) CU(cudaMemsetAsync(net->d_lring, 0xff, net->lring_cap * sizeof(double), st));
        CU(cudaMemsetAsync(net->d_qctl, 0, 32, st));                    // queue cursors, tickets
        CU(cudaMemsetAsync(net->d_qctl + 5, 0, 24, st));                // done counters, lane ticket
        CU(cudaStreamSynchronize(st));
        return fail(TXH_E_WATCHDOG, "a routing launch bailed out on its dataflow watchdog (a wait for another task "
                                    "exceeded TXH_WATCHDOG_MS; the state arrays of that call are undefined)");
    }
    CU(cudaStreamSynchronize(st));
    if (info > 0)
        return fail(TXH_E_INVALID, "an ensemble innovation covariance was not positive definite (Cholesky pivot " +
                                   std::to_string(info) + ")");
    return fail(TXH_E_INVALID, "a Kalman innovation covariance P[s][:,s] + R was singular (Gauss-Jordan pivot " +
                               std::to_string(-info) + ")");
}

int check_M(int64_t M)
{
    if (M < 1 || M > (int64_t(1) << 24)) return fail(TXH_E_INVALID, "member count out of range");
    return TXH_OK;
}

struct StepPlan {                   // forcing interpolation resolved by the init kernel (times == nullptr: unit step)
    const double* times = nullptr;
    int64_t R = 0, t0_ns = 0, dt_ns = 0;
    int method = 1;
};

// Outflows of the rows with a slot (slot == nullptr: off) recorded after every `every`-th step of a call; `base` steps
// of the call came before this routing call (the step that ends its step s is base + s + 1).
struct Recording {
    const int32_t* slot = nullptr;
    double* out = nullptr;
    int every = 1, count = 0;
    int64_t base = 0;
};

// An ensemble update still owed to the state (txh_run_assimilating): the first window launch of a routing call applies
// it while it loads its tasks, and a recording launch also writes the update's recorded rows (rec_prior, rec_post).
struct OwedUpdate {
    const double* T; const double* W; const double* qs; int64_t M;
    double* rec_prior; double* rec_post; const double* rec_mean;
};

// the forcing interpolation fields of the InitArgs of a launch's steps [s0, s0 + ns)
InitArgs step_init(const txh_net* net, const StepPlan& plan, int64_t s0, int64_t ns)
{
    InitArgs ia{};
    ia.times = plan.times; ia.steps_out = net->d_steps; ia.t0_ns = plan.t0_ns; ia.dt_ns = plan.dt_ns;
    ia.step_base = s0; ia.R = (int32_t)plan.R; ia.nsteps = (int32_t)ns; ia.method = plan.method;
    return ia;
}

// common launcher for the persistent dataflow kernel
int run_dataflow(txh_net* net, double* O, double* I, int64_t M, const double* F, const double* W, int wm_ld,
                 const StepPlan& plan, int64_t nsteps, const Recording& rec, cudaStream_t st)
{
    const Schedule& s = net->sched;
    const int ld = (int)txh_row_stride(M);
    const int nmb = (ld + kMemberBlock - 1) / kMemberBlock;
    const size_t pairs = (size_t)s.tasks.size() * nmb;
    if (pairs >= (size_t(1) << 31)) return fail(TXH_E_INVALID, "too many (task, member block) pairs");
    // the ready queue never wraps: one slot per (pair, step); long runs go out in several launches
    const int64_t max_entries = int64_t(1) << 25;
    const int64_t steps_per_launch = std::max<int64_t>(1, std::min<int64_t>(nsteps, max_entries / (int64_t)pairs));
    int rc;
    if ((rc = grow(&net->d_pending, &net->pairs_cap, pairs, st)) ||
        (rc = grow(&net->d_side, &net->side_cap, (size_t)std::max(1, s.n_side) * ld, st)) ||   // [n_side][ld]
        (rc = grow(&net->d_queue, &net->queue_cap, pairs * (size_t)steps_per_launch, st)))
        return rc;
    if (plan.times && (rc = grow(&net->d_steps, &net->steps_cap, (size_t)steps_per_launch, st))) return rc;
    const StepInterp* d_steps = plan.times ? net->d_steps : net->d_unit_step;
    for (int64_t s0 = 0; s0 < nsteps; s0 += steps_per_launch) {
        const int64_t ns = std::min<int64_t>(steps_per_launch, nsteps - s0);
        InitArgs ia = step_init(net, plan, s0, ns);
        ia.tasks = net->d_tasks; ia.init_ready = net->d_init_ready; ia.pending = net->d_pending;
        ia.queue = net->d_queue; ia.q_head = net->d_qctl;
        ia.n_tasks = (int32_t)s.tasks.size(); ia.n_mblocks = nmb; ia.n_init = (int32_t)s.init_ready.size();
        ia.queue_entries = (long long)pairs * ns;
        CU(launch_dataflow_init(ia, st));
        RouteArgs a{};
        a.tasks = net->d_tasks; a.notify = net->d_notify; a.hdr = net->d_hdr; a.inw = net->d_inw;
        a.coef = net->d_coef; a.cumA = net->d_coef + 4 * net->topo.n; a.linkA = net->d_coef + 5 * net->topo.n;
        a.O = O; a.I = I; a.Side = net->d_side; a.F = F; a.steps = d_steps; a.Wmul = W;
        a.rec_slot = rec.slot; a.rec_out = rec.out; a.rec_step_base = rec.base + s0;
        a.pending = ia.pending; a.queue = net->d_queue; a.q_head = net->d_qctl;
        a.status = net->d_status; a.watchdog_ns = net->watchdog_ns;
        a.total = (long long)pairs * ns;
        a.n = net->topo.n; a.n_tasks = ia.n_tasks; a.n_mblocks = nmb; a.nsteps = (int32_t)ns;
        a.slots = std::max(1, s.slots_used); a.ld = ld; a.M = (int32_t)M;
        a.wm_ld = wm_ld; a.rec_every = std::max(1, rec.every); a.rec_count = rec.count;
        // per-warp shared memory: [scratch slots][staging][row ring].  Staging of a walking task:
        // [coef][f0][f1][hdr][words]; of a LINK task: [A_last per segment][records]; 16-byte aligned parts.
        auto up16 = [](int x) { return (x + 15) & ~15; };
        const int L = std::max(1, s.max_len);
        a.max_words = std::min(1024, std::max(16, s.max_words));
        a.max_words_link = std::min(2048, std::max(16, s.max_link_words));
        a.off_coef = a.slots * 32 * (int)sizeof(double2);
        a.off_f0 = a.off_coef + 4 * L * (int)sizeof(double);
        a.off_f1 = a.off_f0 + up16(L * (int)sizeof(double));
        a.off_hdr = a.off_f1 + up16(L * (int)sizeof(double));
        a.off_inw = a.off_hdr + up16(L * (int)sizeof(uint32_t));
        const int end_walk = a.off_inw + up16(a.max_words * (int)sizeof(uint32_t));
        a.off_inw_link = a.off_coef + up16(std::max(1, s.max_link_len) * (int)sizeof(double));
        const int end_link = a.off_inw_link + up16(a.max_words_link * (int)sizeof(uint32_t));
        a.off_ring = std::max(end_walk, end_link);
        a.smem_per_warp = a.off_ring + kRingBytes;
        // the per-task timeline of this launch
        const long long hd[4] = {(long long)pairs, (long long)ns, (long long)s.tasks.size(), (long long)nmb};
        if ((rc = traced_launch("TXH_TRACE_FILE", a.trace, (size_t)a.total * 4, hd, nullptr, 0, st,
                                [&] { return launch_route_dataflow(a, net->num_sms, st); })))
            return rc;
    }
    return TXH_OK;
}

// Per-warp shared-memory layout of route_window_kernel.  A launch that applies an ensemble update keeps the 64 x 64
// transform in shared memory and runs shorter input rings (txh_window.cu: kInRingUpd, kSegRingUpd) to keep its warps:
// at the headline shape 16 x 12,432 B + 33,168 B of the 232,448 B a CTA may have.
void window_smem_layout(const Schedule& s, bool upd, WinArgs& a)
{
    auto up16 = [](int x) { return (x + 15) & ~15; };
    const int rc = std::max(1, s.w_max_len), slots = std::max(1, s.slots_used);
    // `seg_ring` rows for the input stream of a segment ([scratch | ring]), `in_ring` for a pocket's
    const int in_ring = upd ? 2 : 4, seg_ring = upd ? 6 : 8;
    a.off_scr = rc * 512;
    a.off_in = a.off_scr + slots * 512;
    a.off_rec = a.off_in + std::max(in_ring, seg_ring - slots) * 512;
    a.off_cum = a.off_rec + rc * 48;
    a.off_cumc = a.off_cum + up16(rc * 8);
    a.off_words = a.off_cumc + up16(rc * 8);
    a.off_list = a.off_words + up16(std::max(1, s.w_max_words) * 4);
    a.off_mbar = a.off_list + up16(std::max(1, s.w_max_words) * 4);
    a.smem_per_warp = a.off_mbar + 16;                        // + the warp's mbarrier (bulk staging of the state rows)
    const char* bulk = getenv("TXH_WINDOW_BULK");
    if (bulk && atoi(bulk) == 0) a.off_mbar = 0;
}

// Whether route_window_kernel takes the schedule at M members (ok), and the warps per CTA of a launch without (wpc) and
// with (wpc_upd) an ensemble update to apply.  The kernel declines when a CTA would hold fewer than two warps (rows of
// a task x 1 KB per warp), when the schedule has rows it would own, and when ring slots need offsets beyond 32 bits.
// Allocates and launches nothing.
struct WindowFit {
    bool ok;
    int wpc, wpc_upd;
};
WindowFit window_fit(const txh_net* net, int64_t M)
{
    const Schedule& s = net->sched;
    const int steps_bytes = 16 * 24;                          // StepInterp records of one launch (<= 16 steps), once per CTA
    const int smem_max = 227 * 1024;
    int warps_cap = 16;
    if (const char* k = getenv("TXH_WINDOW_WARPS")) warps_cap = std::max(1, std::min(16, atoi(k)));
    WinArgs a{};
    window_smem_layout(s, true, a);
    const int wpc_upd = std::min(warps_cap, (smem_max - steps_bytes - 64 * 64 * (int)sizeof(double) - 16) / a.smem_per_warp);
    window_smem_layout(s, false, a);
    const int wpc = std::min(warps_cap, (smem_max - 1024 - steps_bytes) / a.smem_per_warp);
    const bool ok = wpc >= 2 && s.w_n_own == 0 &&
                    (size_t)std::max(1, s.n_wslots) * txh_row_stride(M) * sizeof(double) < (size_t(1) << 32);
    return {ok, wpc, wpc_upd};
}

// The window-resident kernel (txh_window.cu): state in shared memory for all steps of a launch; its first launch
// applies `upd`.  Returns 1 when the kernel declines the schedule (window_fit) or cannot apply `upd`; the caller falls
// back to the dataflow kernel.
int run_window(txh_net* net, double* O, double* I, int64_t M, const double* F, const double* W, int wm_ld,
               const StepPlan& plan, int64_t nsteps, const Recording& rec, double* rowsum, double rowsum_scale,
               const OwedUpdate* upd, cudaStream_t st)
{
    const Schedule& s = net->sched;
    const int ld = (int)txh_row_stride(M);
    const int nmb = (ld + kMemberBlock - 1) / kMemberBlock;
    const size_t pairs = (size_t)s.wtasks.size() * nmb;
    if (pairs >= (size_t(1) << 31)) return fail(TXH_E_INVALID, "too many (task, member block) pairs");
    const WindowFit fit = window_fit(net, M);
    if (!fit.ok || (upd && (nmb != 1 || upd->M != M || fit.wpc_upd < 2))) return 1;
    // ring[step][slot][ld]: one launch covers 16 steps, up to 64 while the ring stays below 64 MiB (few members):
    // a launch costs the critical path of one step before its pipeline is full, so longer launches amortise it
    const size_t slot_row = (size_t)std::max(1, s.n_wslots) * ld;
    const int64_t spl_max = std::min<int64_t>(64, std::max<int64_t>(16, (int64_t)((size_t(64) << 20) / (slot_row * sizeof(double)))));
    int64_t spl = std::min<int64_t>(spl_max, nsteps);
    while (spl > 1 && slot_row * spl * sizeof(double) > (size_t(1) << 30)) --spl;
    // every cell starts EMPTY (all bits set); consumers put EMPTY back, so a finished launch leaves the whole
    // ring EMPTY again whatever row stride the next launch lays over it
    int rc;
    if ((rc = grow(&net->d_ring, &net->ring_cap, slot_row * spl, st, 0xff))) return rc;
    net->ring_ld = ld;
    if (plan.times && (rc = grow(&net->d_steps, &net->steps_cap, (size_t)spl, st))) return rc;
    const StepInterp* d_steps = plan.times ? net->d_steps : net->d_unit_step;
    WinArgs a{};
    for (int64_t s0 = 0; s0 < nsteps; s0 += spl) {
        const int64_t ns = std::min<int64_t>(spl, nsteps - s0);
        // up to 16 steps every warp resolves the forcing interpolation itself (no init launch: the kernel re-arms
        // its own ticket); longer launches read the records an init kernel leaves in global memory
        const bool own_steps = ns <= 16;
        if (!own_steps) CU(launch_window_init(step_init(net, plan, s0, ns), net->d_qctl + 3, st));
        a.times = plan.times; a.t0_ns = plan.t0_ns; a.dt_ns = plan.dt_ns; a.step_base = s0; a.R = (int32_t)plan.R;
        a.method = plan.method; a.done = net->d_qctl + 5;
        a.tasks = net->d_wtasks; a.hdr = net->d_whdr; a.inw = net->d_winw; a.prod = net->d_wprod;
        a.coef = net->d_coef; a.cumA = net->d_coef + 4 * net->topo.n;
        a.cumC = net->d_coef + 5 * net->topo.n + s.link_last.size();
        a.O = O; a.I = I; a.ring = net->d_ring; a.ticket = net->d_qctl + 3;
        a.F = F; a.steps = (own_steps && plan.times) ? nullptr : d_steps; a.Wmul = W; a.status = net->d_status; a.watchdog_ns = net->watchdog_ns;
        a.n = net->topo.n; a.n_tasks = (int32_t)s.wtasks.size(); a.n_mblocks = nmb; a.nsteps = (int32_t)ns;
        a.n_slots = std::max(1, s.n_wslots); a.ld = ld; a.M = (int32_t)M; a.wm_ld = wm_ld;
        // the row sums ride on the last step of the call when one warp covers all members of a row
        a.rowsum = (rowsum && nmb == 1 && s0 + ns == nsteps) ? rowsum : nullptr;
        a.rowsum_scale = rowsum_scale;
        a.upT = nullptr;
        if (s0 == 0 && upd) {
            // the ensemble update owed to the state is applied by this launch while it loads its tasks
            a.upT = upd->T; a.upW = upd->W; a.upQs = upd->qs;
            a.gfix_off = net->d_gfix_off; a.gfix = net->d_gfix;
            if (rec.slot) { a.rec_prior = upd->rec_prior; a.rec_post = upd->rec_post; a.rec_mean = upd->rec_mean; }
            window_smem_layout(s, true, a);
            a.off_T = fit.wpc_upd * a.smem_per_warp;
        } else window_smem_layout(s, false, a);
        a.off_steps = a.upT ? a.off_T + 64 * 64 * (int)sizeof(double) + 16 : fit.wpc * a.smem_per_warp;
        a.rec_slot = rec.slot; a.rec_out = rec.out; a.rec_step_base = rec.base + s0;
        a.rec_every = std::max(1, rec.every); a.rec_count = rec.count;
        a.nap_min = 32; a.nap_max = 256;
        if (const char* k = getenv("TXH_WINDOW_NAP")) { int lo = 32, hi = 256; if (sscanf(k, "%d,%d", &lo, &hi) >= 1) { a.nap_min = std::max(0, lo); a.nap_max = std::max(a.nap_min, hi); } }
        // the per-task timeline of this launch
        const long long hd[4] = {(long long)pairs, (long long)ns, (long long)s.wtasks.size(), -(long long)nmb};
        if ((rc = traced_launch("TXH_TRACE_FILE", a.trace, pairs * (size_t)(4 + ns), hd, nullptr, 0, st,
                                [&] { return launch_route_window(a, a.upT ? fit.wpc_upd : fit.wpc, net->num_sms, st); })))
            return rc;
    }
    return TXH_OK;
}

// ---- lane kernel (txh_lane.cu): lanes = reaches, for deterministic runs and small ensembles --------------
constexpr size_t kLaneSmemBudget = 200 * 1024;

int lane_tile_index(int64_t M) { return M <= 1 ? 0 : M <= 2 ? 1 : M <= 4 ? 2 : M <= 8 ? 3 : 4; }

// host side only: the schedule for member tile index `ti` (built once per handle).  Without an explicit cap the
// rows per region follow from the size of the network: one region per SM while that keeps a region within two
// passes of a CTA's threads (all regions are then resident at once and run as one pipeline).
txh_net::LaneDev* lane_schedule(txh_net* net, int ti, int num_sms)
{
    txh_net::LaneDev& L = net->lane[ti];
    if (!L.built) {
        std::string err;
        int side_min = 32;
        if (const char* k = getenv("TXH_LANE_SIDE_MIN")) side_min = atoi(k);
        if (net->lane_cap_rows > 0) {
            L.ok = L.sched.build(net->topo, net->sched.pos_of_reach, 1 << ti, net->lane_cap_rows, kLaneSmemBudget, side_min, err);
        } else {
            // lane_ctas regions per SM, all resident at once while the network is small enough.  Measured on B200
            // (profiles/r02_lane_sweeps.jsonl): the SM's issue rate is set by warps x their dependent-instruction
            // chains, not by the size of a barrier domain, so one large region per SM (fewest streams and hops) wins.
            const int ctas = std::max(1, net->lane_ctas);
            const int cap_max = std::max(64, 1024 / ctas - 48);            // threads of a CTA = rows + stream mirrors
            const int64_t slots = (int64_t)num_sms * ctas;
            const int64_t per = (net->topo.n + slots - 1) / slots;
            int cap = (int)std::min<int64_t>(cap_max, std::max<int64_t>(std::min(320, cap_max), per + per / 50));
            for (;;) {
                L.ok = L.sched.build(net->topo, net->sched.pos_of_reach, 1 << ti, cap, kLaneSmemBudget, side_min, err);
                if (!L.ok || (int64_t)L.sched.regions.size() <= slots || cap >= cap_max) break;
                cap = std::min(cap_max, cap + std::max(4, cap / 12));
            }
        }
        L.built = true;
        if (!L.ok) g_err = err;
    }
    return &L;
}

// Returns 1 when the lane schedule cannot be built for this network (the caller falls back).
int run_lane(txh_net* net, double* O, double* I, int64_t M, const double* F, const double* W, int wm_ld,
             const StepPlan& plan, int64_t nsteps, const Recording& rec, cudaStream_t st)
{
    const int ti = lane_tile_index(M), mt = 1 << ti;
    if (M > 16) return 1;
    txh_net::LaneDev* L = lane_schedule(net, ti, net->num_sms);
    if (!L->ok) return 1;
    const LaneSchedule& s = L->sched;
    int rc;
    if (!L->on_dev) {
        std::vector<int4> meta(s.row_reach.size());
        for (size_t i = 0; i < meta.size(); ++i) {
            const int32_t j = s.row_reach[i];
            meta[i] = make_int4(j >= 0 ? net->sched.pos_of_reach[j] : -1, s.row_off[i] | (s.row_nx[i] << 16), s.row_c01[i],
                                s.row_slot[i]);
        }
        if ((rc = upload(&L->d_regions, s.regions))) return rc;
        if ((rc = upload(&L->d_meta, meta))) return rc;
        if ((rc = upload(&L->d_xbeg, s.row_xbeg))) return rc;
        if ((rc = upload(&L->d_child, s.child))) return rc;
        L->on_dev = true;
    }
    if (!net->d_unit_lstep) {
        const LaneStep unit{1.0, 0.0, 0, 0, 0, 0};
        CU(cudaMalloc((void**)&net->d_unit_lstep, sizeof(LaneStep)));
        CU(cudaMemcpy(net->d_unit_lstep, &unit, sizeof(unit), cudaMemcpyHostToDevice));
    }
    const int ld = (int)txh_row_stride(M);
    // streams ring[slot][member][step]: one launch covers as many steps as fit 128 MiB
    const size_t streams = (size_t)std::max(1, s.n_slots) * (size_t)M;
    int64_t spl = std::min<int64_t>(nsteps, 4096);
    if (const char* k = getenv("TXH_LANE_SPL")) { const long v = atol(k); if (v > 0) spl = std::min<int64_t>(spl, v); }
    while (spl > 16 && streams * (size_t)((spl + 15) & ~int64_t(15)) * sizeof(double) > (size_t(128) << 20)) spl = (spl + 1) / 2;
    const size_t ring_need = streams * (size_t)((spl + 15) & ~int64_t(15));
    if ((rc = grow(&net->d_lring, &net->lring_cap, ring_need, st, 0xff))) return rc;   // every cell starts EMPTY
    if (plan.times) {
        if ((rc = grow(&net->d_lsteps, &net->lsteps_cap, (size_t)spl, st))) return rc;
    } else if (nsteps != 1) {
        return fail(TXH_E_INVALID, "internal: a launch without a forcing table covers one step");
    }
    const LaneStep* d_steps = plan.times ? net->d_lsteps : net->d_unit_lstep;
    // shared memory: the largest region (every CTA lays its region out itself, LaneSchedule::region_bytes)
    LaneArgs a{};
    size_t smem = (s.max_bytes + 31) & ~size_t(15);
    if (smem > 227 * 1024) return 1;
    // the per-step interpolation records ride in shared memory too when they fit
    if (plan.times && smem + 32 * (size_t)spl <= 200 * 1024) { a.off_steps = (int32_t)smem; smem += 32 * (size_t)spl; }
    a.lag = 24;                                            // (measured: 24 / 32 / 48 steps -> C2 2.47 / 2.53 / 2.69 ms, C4 5.72 / 5.81 / 6.16 ms)
    if (const char* k = getenv("TXH_LANE_LAG")) a.lag = std::max(24, std::min(4096, atoi(k)));
    a.vote_every = 64;
    if (const char* k = getenv("TXH_LANE_VOTE_EVERY")) { const int v = atoi(k); if (v > 0 && (v & (v - 1)) == 0) a.vote_every = v; }
    const int tv = s.max_virt > 0 ? std::min(128, (s.max_virt + 31) / 32 * 32) : 0;
    const int tr = (s.max_real + 31) / 32 * 32;                            // one row per thread
    if (tr + tv > 1024) return 1;
    a.TR = tr;
    const int threads = tr + tv;
    // every CTA of the grid must be resident (a region waits for regions claimed before it): ask the runtime how many
    // CTAs of this shape fit an SM
    int per_sm = 1;
    CU(lane_occupancy(mt, F != nullptr, W != nullptr, threads, smem, &per_sm));
    if (per_sm < 1) return 1;
    const int grid = (int)std::min<int64_t>((int64_t)net->num_sms * per_sm, (int64_t)s.regions.size());
    for (int64_t s0 = 0; s0 < nsteps; s0 += spl) {
        const int64_t ns = std::min<int64_t>(spl, nsteps - s0);
        if (plan.times) CU(launch_lane_init(step_init(net, plan, s0, ns), net->d_lsteps, net->d_qctl + 6, st));
        a.regions = L->d_regions; a.meta = L->d_meta; a.xbeg = L->d_xbeg; a.child = L->d_child;
        a.coef = net->d_coef; a.O = O; a.I = I; a.F = F; a.steps = d_steps; a.Wmul = W;
        a.ring = net->d_lring; a.ticket = net->d_qctl + 6; a.done = net->d_qctl + 7;
        a.status = net->d_status; a.watchdog_ns = net->watchdog_ns;
        a.rec_slot = rec.slot; a.rec_out = rec.out; a.rec_step_base = rec.base + s0;
        a.rec_every = std::max(1, rec.every); a.rec_count = rec.count;
        a.n = net->topo.n; a.n_regions = (int32_t)s.regions.size(); a.nsteps = (int32_t)ns;
        a.splp = (int32_t)((ns + 15) & ~int64_t(15)); a.ld = ld; a.M = (int32_t)M; a.wm_ld = wm_ld;
        a.R = plan.times ? (int32_t)plan.R : 1;
        // the region timeline of this launch, behind the region descriptors
        const long long hd[4] = {(long long)s.regions.size(), (long long)ns, (long long)threads, (long long)grid};
        if ((rc = traced_launch("TXH_LANE_TRACE", a.trace, 8 * s.regions.size(), hd, s.regions.data(),
                                s.regions.size() * sizeof(LaneRegionDesc), st,
                                [&] { return launch_route_lane(a, mt, threads, smem, grid, st); })))
            return rc;
    }
    return TXH_OK;
}

// Lane kernel or window kernel?  Forced by TXH_ROUTE_KERNEL, else the lane kernel for small ensembles when the launch
// is long enough to amortise its pipeline fill.  Measured on B200 (DESIGN.md section 4.2): an iteration of the lane
// kernel costs ~1 us and a launch runs nsteps + fill iterations, fill = sum over the deepest chain of regions of
// (internal depth + lag); the window kernel costs ~(40 + n/1000) us per launch of at most 64 steps plus
// ~(4 + 4e-5 n) us per step (n = 100k: 138 + 8.1 us; n = 1,000: 4.5 us per step).
bool lane_wanted(txh_net* net, int64_t M, int64_t nsteps)
{
    if (net->route_kernel == 3) return M <= 16;
    if (net->route_kernel != 0 || M > net->lane_max_members) return false;
    txh_net::LaneDev* L = lane_schedule(net, lane_tile_index(M), net->num_sms);
    if (!L->ok) return false;
    const LaneSchedule& s = L->sched;
    int hmax = 0; double extra = 0.0;
    for (const LaneRegionDesc& r : s.regions) { hmax = std::max(hmax, r.height); extra += r.n_extra; }
    extra /= std::max<size_t>(1, s.regions.size());
    const double n = (double)net->topo.n;
    const double t_lane = (double)nsteps + (hmax + 1) * (extra + 32.0);
    const double t_win = std::ceil((double)nsteps / 64.0) * (40.0 + 1e-3 * n) + (double)nsteps * (4.0 + 4e-5 * n);
    return t_lane <= t_win;
}

// routing entry: the lane kernel for small ensembles, else the window kernel (or what the environment says); the
// dataflow kernel where the window kernel declines the schedule.  rowsum (nullptr: off) receives rowsum_scale * the
// member sums of the final outflows.  upd (nullptr: none) is applied by the first window launch; a routing call that
// cannot apply it fails.
int run_routing(txh_net* net, double* O, double* I, int64_t M, const double* F, const double* W, int wm_ld,
                const StepPlan& plan, int64_t nsteps, cudaStream_t st, const Recording& rec = Recording(),
                double* rowsum = nullptr, double rowsum_scale = 1.0, const OwedUpdate* upd = nullptr)
{
    const int ld = (int)txh_row_stride(M);
    int rc = 1;                                           // 1: the kernel declined, the next one routes
    bool sums_done = false;                               // by the window kernel, on its last step
    if (!upd && lane_wanted(net, M, nsteps)) rc = run_lane(net, O, I, M, F, W, wm_ld, plan, nsteps, rec, st);
    if (rc == 1 && net->route_kernel != 1) {
        rc = run_window(net, O, I, M, F, W, wm_ld, plan, nsteps, rec, rowsum, rowsum_scale, upd, st);
        sums_done = rc == TXH_OK && ld <= kMemberBlock;
    }
    if (rc == 1 && upd) return fail(TXH_E_STATE, "the routing launch did not take the pending ensemble update");
    if (rc == 1) rc = run_dataflow(net, O, I, M, F, W, wm_ld, plan, nsteps, rec, st);
    if (rc == TXH_OK && rowsum && !sums_done)
        CU(launch_enkf_stats(O, ld, (int)M, net->topo.n, rowsum_scale, nullptr, rowsum, nullptr, st));
    return rc;
}

}  // namespace

// error reporting for the host-only translation units (txh_geojson.cpp)
int txh_set_error_(int code, const char* msg) { return fail(code, msg ? msg : ""); }

extern "C" {

const char* txh_last_error(void) { return g_err.c_str(); }
int txh_version(void) { return 100; }
int txh_device_count(void)
{
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) { cudaGetLastError(); return 0; }
    return c;
}
int64_t txh_launch_count(void) { return launch_count(); }
int64_t txh_row_stride(int64_t M) { return (M + 1) & ~int64_t(1); }

int txh_create(int64_t n, const int64_t* endnodes, const int32_t* sp, txh_net** out)
{
    if (!endnodes || !out) return fail(TXH_E_INVALID, "null argument");
    txh_net* net = new (std::nothrow) txh_net();
    if (!net) return fail(TXH_E_INVALID, "out of memory");
    std::string err;
    if (!net->topo.build(n, endnodes, err)) { delete net; return fail(TXH_E_TOPOLOGY, err); }
    SchedParams p;
    if (sp) { p.long_path_min = sp[0]; p.spine_cap = sp[1]; p.pocket_cap = sp[2]; p.max_slots = sp[3]; p.link_cap = sp[4]; }
    if (const char* lw = getenv("TXH_LEN_WEIGHT")) p.len_weight = atoi(lw);
    if (const char* sc = getenv("TXH_SIDE_CAP")) p.side_cap = std::max(1, atoi(sc));
    if (const char* pc = getenv("TXH_POCKET_CAP")) p.pocket_cap = std::max(4, std::min(16, atoi(pc)));
    if (!net->sched.build(net->topo, p, err)) { delete net; return fail(TXH_E_INVALID, err); }
    *out = net;
    return TXH_OK;
}

void txh_destroy(txh_net* net)
{
    if (!net) return;
    if (net->dev_ready) {
        cudaFree(net->d_tasks); cudaFree(net->d_notify); cudaFree(net->d_init_ready); cudaFree(net->d_hdr); cudaFree(net->d_inw);
        for (auto& ev : net->route_events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
        cudaFree(net->d_up_off); cudaFree(net->d_up_pos); cudaFree(net->d_lvl_pos); cudaFree(net->d_inner); cudaFree(net->d_inner_rec);
        cudaFree(net->d_reach_of_pos); cudaFree(net->d_pos_of_reach); cudaFree(net->d_outlet);
        cudaFree(net->d_coef); cudaFree(net->d_qtmp); cudaFree(net->d_qctl); cudaFree(net->d_rec_slot);
        cudaFree(net->d_unit_step);
        if (net->d_rec_pos) cudaFree(net->d_rec_pos);
        if (net->d_pending) cudaFree(net->d_pending);
        if (net->d_queue) cudaFree(net->d_queue);
        if (net->d_side) cudaFree(net->d_side);
        if (net->d_steps) cudaFree(net->d_steps);
        if (net->d_tmp_idx) cudaFree(net->d_tmp_idx);
        if (net->d_obs) cudaFree(net->d_obs);
        if (net->d_gauge_of_pos) cudaFree(net->d_gauge_of_pos);
        cudaFree(net->d_gfix_off); cudaFree(net->d_gfix);
        cudaFree(net->d_wtasks); cudaFree(net->d_whdr); cudaFree(net->d_winw); cudaFree(net->d_wprod);
        if (net->d_ring) cudaFree(net->d_ring);
        if (net->d_lring) cudaFree(net->d_lring);
        for (auto& L : net->lane) { cudaFree(L.d_regions); cudaFree(L.d_meta); cudaFree(L.d_xbeg); cudaFree(L.d_child); }
        if (net->d_lsteps) cudaFree(net->d_lsteps);
        if (net->d_unit_lstep) cudaFree(net->d_unit_lstep);
        if (net->d_stage) cudaFree(net->d_stage);
        if (net->h_status) cudaFreeHost(net->h_status);
    }
    delete net;
}

int64_t txh_n(const txh_net* net) { return net ? net->topo.n : 0; }

static void widen(const std::vector<int32_t>& v, int64_t* out) { for (size_t i = 0; i < v.size(); ++i) out[i] = v[i]; }

int txh_get_indegree(const txh_net* net, int64_t* out)
{
    if (!net || !out) return fail(TXH_E_INVALID, "null argument");
    widen(net->topo.indeg, out); return TXH_OK;
}
int txh_get_headwaters(const txh_net* net, int64_t* heads, int64_t* count)
{
    if (!net || !heads || !count) return fail(TXH_E_INVALID, "null argument");
    widen(net->topo.heads, heads); *count = (int64_t)net->topo.heads.size(); return TXH_OK;
}
int txh_get_levels(const txh_net* net, int64_t* level, int64_t* nlevels)
{
    if (!net || !nlevels) return fail(TXH_E_INVALID, "null argument");
    if (level) widen(net->topo.level, level);
    *nlevels = net->topo.nlevels; return TXH_OK;
}
int txh_get_level_order(const txh_net* net, int64_t* order, int64_t* offsets)
{
    if (!net || !order || !offsets) return fail(TXH_E_INVALID, "null argument");
    widen(net->topo.topo, order); widen(net->topo.level_off, offsets); return TXH_OK;
}
int txh_get_chains(const txh_net* net, int64_t* cid, int64_t* cpos, int64_t* clen, int64_t* nchains)
{
    if (!net || !cid || !cpos || !clen || !nchains) return fail(TXH_E_INVALID, "null argument");
    widen(net->topo.chain_id, cid); widen(net->topo.chain_pos, cpos); widen(net->topo.chain_len, clen);
    *nchains = (int64_t)net->topo.chain_len.size(); return TXH_OK;
}
int txh_get_paths(const txh_net* net, int64_t* pid, int64_t* ppos)
{
    if (!net || !pid || !ppos) return fail(TXH_E_INVALID, "null argument");
    widen(net->topo.path_id, pid); widen(net->topo.path_pos, ppos); return TXH_OK;
}
int txh_get_visit_order(const txh_net* net, int64_t* order)
{
    if (!net || !order) return fail(TXH_E_INVALID, "null argument");
    widen(net->topo.visit, order); return TXH_OK;
}
int txh_get_schedule_info(const txh_net* net, int64_t info[10])
{
    if (!net || !info) return fail(TXH_E_INVALID, "null argument");
    const Schedule& s = net->sched;
    info[0] = (int64_t)s.tasks.size(); info[1] = s.n_spine; info[2] = s.n_pocket;
    info[3] = (int64_t)s.inw.size(); info[4] = (int64_t)s.notify.size(); info[5] = s.slots_used;
    info[6] = s.row_fallbacks; info[7] = s.cp_tasks; info[8] = s.cp_cost; info[9] = net->topo.nlevels;
    return TXH_OK;
}
int txh_get_schedule(const txh_net* net, int64_t* pos_of_reach, int32_t* task_desc, int32_t* notify,
                     uint32_t* hdr, uint32_t* inw)
{
    if (!net) return fail(TXH_E_INVALID, "null argument");
    const Schedule& s = net->sched;
    if (pos_of_reach) widen(s.pos_of_reach, pos_of_reach);
    if (task_desc) std::memcpy(task_desc, s.tasks.data(), s.tasks.size() * sizeof(TaskDesc));
    if (notify) std::memcpy(notify, s.notify.data(), s.notify.size() * sizeof(int32_t));
    if (hdr) std::memcpy(hdr, s.hdr.data(), s.hdr.size() * sizeof(uint32_t));
    if (inw) std::memcpy(inw, s.inw.data(), s.inw.size() * sizeof(uint32_t));
    return TXH_OK;
}

int txh_get_window_info(const txh_net* net, int64_t info[8])
{
    if (!net || !info) return fail(TXH_E_INVALID, "null argument");
    const Schedule& s = net->sched;
    info[0] = (int64_t)s.wtasks.size(); info[1] = s.n_wslots; info[2] = s.w_max_len; info[3] = s.w_max_words;
    info[4] = s.w_max_prod; info[5] = (int64_t)s.winw.size(); info[6] = (int64_t)s.wprod.size(); info[7] = s.w_cp_tasks;
    return TXH_OK;
}
int txh_get_window_schedule(const txh_net* net, int32_t* wtask_desc, uint32_t* whdr, uint32_t* winw, int32_t* wprod)
{
    if (!net) return fail(TXH_E_INVALID, "null argument");
    const Schedule& s = net->sched;
    if (wtask_desc) std::memcpy(wtask_desc, s.wtasks.data(), s.wtasks.size() * sizeof(WTaskDesc));
    if (whdr) std::memcpy(whdr, s.whdr.data(), s.whdr.size() * sizeof(uint32_t));
    if (winw) std::memcpy(winw, s.winw.data(), s.winw.size() * sizeof(uint32_t));
    if (wprod) std::memcpy(wprod, s.wprod.data(), s.wprod.size() * sizeof(int32_t));
    return TXH_OK;
}

int txh_get_lane_info(txh_net* net, int64_t M, int64_t cap_rows, int64_t info[8])
{
    if (!net || !info || M < 1 || M > 16) return fail(TXH_E_INVALID, "bad argument");
    if (cap_rows > 0) {
        if (net->lane_cap_rows != (int)cap_rows) for (auto& L : net->lane) if (!L.on_dev) L.built = false;
        net->lane_cap_rows = (int)cap_rows;
    }
    txh_net::LaneDev* L = lane_schedule(net, lane_tile_index(M), net->num_sms > 0 ? net->num_sms : 148);
    if (!L->ok) return fail(TXH_E_INVALID, g_err);
    const LaneSchedule& s = L->sched;
    info[0] = (int64_t)s.regions.size(); info[1] = (int64_t)s.row_reach.size(); info[2] = (int64_t)s.child.size();
    info[3] = s.n_slots; info[4] = s.max_real; info[5] = s.max_virt; info[6] = s.max_extra; info[7] = s.mt;
    return TXH_OK;
}
int txh_get_lane_schedule(txh_net* net, int64_t M, int32_t* regions, int32_t* rows, int32_t* child)
{
    if (!net || M < 1 || M > 16) return fail(TXH_E_INVALID, "bad argument");
    txh_net::LaneDev* L = lane_schedule(net, lane_tile_index(M), net->num_sms > 0 ? net->num_sms : 148);
    if (!L->ok) return fail(TXH_E_INVALID, g_err);
    const LaneSchedule& s = L->sched;
    if (regions) std::memcpy(regions, s.regions.data(), s.regions.size() * sizeof(LaneRegionDesc));
    if (rows)
        for (size_t i = 0; i < s.row_reach.size(); ++i) {
            rows[6 * i] = s.row_reach[i]; rows[6 * i + 1] = s.row_off[i]; rows[6 * i + 2] = s.row_c01[i];
            rows[6 * i + 3] = s.row_nx[i]; rows[6 * i + 4] = s.row_xbeg[i]; rows[6 * i + 5] = s.row_slot[i];
        }
    if (child) for (size_t i = 0; i < s.child.size(); ++i) child[i] = s.child[i];
    return TXH_OK;
}

int txh_set_coeffs(txh_net* net, const double* al, const double* be, const double* ch, const double* ga)
{
    if (!net || !al || !be || !ch || !ga) return fail(TXH_E_INVALID, "null argument");
    const int64_t n = net->topo.n;
    const Schedule& sc = net->sched;
    net->coef_host.resize(6 * n + sc.link_last.size());
    double* cum = net->coef_host.data() + 4 * n;
    for (int64_t k = 0; k < n; ++k) {
        const int32_t j = sc.reach_of_pos[k];
        net->coef_host[4 * k] = al[j]; net->coef_host[4 * k + 1] = be[j];
        net->coef_host[4 * k + 2] = ch[j]; net->coef_host[4 * k + 3] = ga[j];
        // prefix product of alpha along the segment (rows whose header carries the continue bit)
        cum[k] = (k > 0 && (sc.hdr[k] & HDR_ACC)) ? cum[k - 1] * al[j] : al[j];
    }
    for (size_t e = 0; e < sc.link_last.size(); ++e) net->coef_host[5 * n + e] = cum[sc.link_last[e]];
    // window kernel: p_k' = P0_k + C_k o_in along a segment, C_k = beta_k A_{k-1} + chi_k A_k, A_{-1} = 1
    double* cumc = net->coef_host.data() + 5 * n + sc.link_last.size();
    for (int64_t k = 0; k < n; ++k) {
        const int32_t j = sc.reach_of_pos[k];
        const double aprev = (k > 0 && (sc.hdr[k] & HDR_ACC)) ? cum[k - 1] : 1.0;
        cumc[k] = be[j] * aprev + ch[j] * cum[k];
    }
    net->have_coef = true; net->coef_dirty = true;
    return TXH_OK;
}

int txh_compute_coeffs(txh_net* net, const double* K, const double* X, double dt, double* al, double* be,
                       double* ch, double* ga)
{
    if (!net || !K || !X) return fail(TXH_E_INVALID, "null argument");
    const int64_t n = net->topo.n;
    std::vector<double> a(n), b(n), c(n), g(n);
    for (int64_t j = 0; j < n; ++j) {
        // muskingum.py:332-347, same operation order
        const double k = K[j], x = X[j];
        a[j] = (dt - 2 * k * x) / (2 * k * (1 - x) + dt);
        b[j] = (dt + 2 * k * x) / (2 * k * (1 - x) + dt);
        c[j] = (2 * k * (1 - x) - dt) / (2 * k * (1 - x) + dt);
        g[j] = dt / (k * (1 - x) + dt / 2);
    }
    if (al) std::memcpy(al, a.data(), n * sizeof(double));
    if (be) std::memcpy(be, b.data(), n * sizeof(double));
    if (ch) std::memcpy(ch, c.data(), n * sizeof(double));
    if (ga) std::memcpy(ga, g.data(), n * sizeof(double));
    return txh_set_coeffs(net, a.data(), b.data(), c.data(), g.data());
}

int txh_pack_host(txh_net* net, const double* src, int64_t M, int layout, double* dst, void* stream)
{
    if (!net || !src || !dst) return fail(TXH_E_INVALID, "null argument");
    int rc;
    if ((rc = check_M(M)) || (rc = ensure_device(net))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = net->topo.n;
    if ((rc = grow(&net->d_stage, &net->stage_cap, (size_t)n * M, st))) return rc;
    double* tmp = net->d_stage;
    CU(cudaMemcpyAsync(tmp, src, sizeof(double) * n * M, cudaMemcpyHostToDevice, st));
    CU(launch_pack(net->d_reach_of_pos, tmp, dst, n, (int)M, (int)txh_row_stride(M), layout, st));
    return TXH_OK;
}

int txh_unpack_host(txh_net* net, const double* src, int64_t M, int layout, double* dst, void* stream)
{
    if (!net || !src || !dst) return fail(TXH_E_INVALID, "null argument");
    int rc;
    if ((rc = check_M(M)) || (rc = ensure_device(net))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = net->topo.n;
    if ((rc = grow(&net->d_stage, &net->stage_cap, (size_t)n * M, st))) return rc;
    double* tmp = net->d_stage;
    CU(launch_unpack(net->d_reach_of_pos, src, tmp, n, (int)M, (int)txh_row_stride(M), layout, st));
    CU(cudaMemcpyAsync(dst, tmp, sizeof(double) * n * M, cudaMemcpyDeviceToHost, st));
    return report_status(net, st);
}

int txh_pack_dev(txh_net* net, const double* src, int64_t M, double* dst, void* stream)
{
    if (!net || !src || !dst) return fail(TXH_E_INVALID, "null argument");
    int rc;
    if ((rc = check_M(M)) || (rc = ensure_device(net))) return rc;
    CU(launch_pack(net->d_reach_of_pos, src, dst, net->topo.n, (int)M, (int)txh_row_stride(M), 0, (cudaStream_t)stream));
    return TXH_OK;
}

int txh_unpack_dev(txh_net* net, const double* src, int64_t M, double* dst, void* stream)
{
    if (!net || !src || !dst) return fail(TXH_E_INVALID, "null argument");
    int rc;
    if ((rc = check_M(M)) || (rc = ensure_device(net))) return rc;
    CU(launch_unpack(net->d_reach_of_pos, src, dst, net->topo.n, (int)M, (int)txh_row_stride(M), 0, (cudaStream_t)stream));
    return TXH_OK;
}

int txh_gather_rows(txh_net* net, const double* X, int64_t M, const int64_t* idx, int64_t count, double* out,
                    void* stream)
{
    if (!net || !X || !idx || !out || count < 0) return fail(TXH_E_INVALID, "bad argument");
    int rc;
    if ((rc = check_M(M)) || (rc = ensure_device(net))) return rc;
    if (count == 0) return TXH_OK;
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<int32_t> pos(count);
    for (int64_t k = 0; k < count; ++k) {
        if (idx[k] < 0 || idx[k] >= net->topo.n) return fail(TXH_E_INVALID, "reach index out of range");
        pos[k] = net->sched.pos_of_reach[idx[k]];
    }
    if ((rc = grow(&net->d_tmp_idx, &net->tmp_idx_cap, (size_t)count, st))) return rc;
    CU(cudaMemcpyAsync(net->d_tmp_idx, pos.data(), sizeof(int32_t) * count, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));      // `pos` is a stack-lifetime buffer
    CU(launch_gather_rows(net->d_tmp_idx, count, X, (int)txh_row_stride(M), (int)M, out, st));
    return TXH_OK;
}

int txh_init_inflows(txh_net* net, const double* O, double* I, int64_t M, void* stream)
{
    if (!net || !O || !I) return fail(TXH_E_INVALID, "null argument");
    int rc;
    if ((rc = check_M(M)) || (rc = ensure_device(net))) return rc;
    CU(launch_init_inflows(net->d_up_off, net->d_up_pos, net->d_outlet, O, I, net->topo.n,
                           (int)txh_row_stride(M), (int)M, (cudaStream_t)stream));
    return TXH_OK;
}

int txh_forcing_create(txh_net* net, int64_t R, const double* times, const double* table, int64_t M,
                       const double* mul, void* stream, txh_forcing** out)
{
    if (!net || !times || !table || !out || R < 1) return fail(TXH_E_INVALID, "bad argument");
    int rc;
    if ((rc = ensure_device(net))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    for (int64_t r = 1; r < R; ++r)
        if (!(times[r] >= times[r - 1])) return fail(TXH_E_INVALID, "forcing times must be sorted ascending");
    const int64_t n = net->topo.n;
    txh_forcing* f = new (std::nothrow) txh_forcing();
    if (!f) return fail(TXH_E_INVALID, "out of memory");
    f->net = net; f->R = R; f->M = mul ? M : 0;
    f->times.assign(times, times + R);
    // one H2D copy of the table as given (pinned or pageable) into the handle's staging buffer, columns
    // permuted into schedule order on the device
    if ((rc = grow(&net->d_stage, &net->stage_cap, (size_t)R * n, st))) { delete f; return rc; }
    double* tmp = net->d_stage;
    cudaError_t e = cudaMalloc((void**)&f->d_F, sizeof(double) * R * n);
    if (e == cudaSuccess) e = cudaMalloc((void**)&f->d_times, sizeof(double) * R);
    if (e == cudaSuccess) e = cudaMemcpyAsync(f->d_times, f->times.data(), sizeof(double) * R, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(tmp, table, sizeof(double) * R * n, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = launch_permute_rows(net->d_reach_of_pos, tmp, f->d_F, n, R, st);
    if (e == cudaSuccess && mul) {
        if (M < 1) { cudaFree(f->d_F); cudaFree(f->d_times); delete f; return fail(TXH_E_INVALID, "member multipliers need M >= 1"); }
        e = cudaMalloc((void**)&f->d_W, sizeof(double) * R * M);
        if (e == cudaSuccess) e = cudaMemcpyAsync(f->d_W, mul, sizeof(double) * R * M, cudaMemcpyHostToDevice, st);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { cudaFree(f->d_F); cudaFree(f->d_W); cudaFree(f->d_times); delete f; return cuda_fail(e, "forcing upload"); }
    *out = f;
    return TXH_OK;
}

int txh_forcing_update(txh_forcing* f, const double* times, const double* table, const double* mul, void* stream)
{
    if (!f || !times || !table) return fail(TXH_E_INVALID, "null argument");
    if ((mul != nullptr) != (f->d_W != nullptr)) return fail(TXH_E_INVALID, "member multipliers must stay present / absent");
    txh_net* net = f->net;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = net->topo.n, R = f->R;
    for (int64_t r = 1; r < R; ++r)
        if (!(times[r] >= times[r - 1])) return fail(TXH_E_INVALID, "forcing times must be sorted ascending");
    int rc;
    if ((rc = txh_forcing_wait(f))) return rc;
    if ((rc = grow(&net->d_stage, &net->stage_cap, (size_t)R * n, st))) return rc;
    double* tmp = net->d_stage;
    f->times.assign(times, times + R);
    CU(cudaMemcpyAsync(f->d_times, f->times.data(), sizeof(double) * R, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(tmp, table, sizeof(double) * R * n, cudaMemcpyHostToDevice, st));
    CU(launch_permute_rows(net->d_reach_of_pos, tmp, f->d_F, n, R, st));
    if (mul) CU(cudaMemcpyAsync(f->d_W, mul, sizeof(double) * R * f->M, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));          // `times` and pageable sources may be reused by the caller
    return TXH_OK;
}

int txh_forcing_update_async(txh_forcing* f, const double* times, const double* table, const double* mul, void* stream)
{
    if (!f || !times || !table) return fail(TXH_E_INVALID, "null argument");
    if ((mul != nullptr) != (f->d_W != nullptr)) return fail(TXH_E_INVALID, "member multipliers must stay present / absent");
    txh_net* net = f->net;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = net->topo.n, R = f->R;
    for (int64_t r = 1; r < R; ++r)
        if (!(times[r] >= times[r - 1])) return fail(TXH_E_INVALID, "forcing times must be sorted ascending");
    if (!f->copy_stream) {
        CU(cudaStreamCreateWithFlags(&f->copy_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&f->reuse_ev, cudaEventDisableTiming));
        CU(cudaMalloc((void**)&f->d_stage, sizeof(double) * R * n));
        // a first chunk small enough that routing starts at once, then ~16 MiB pieces
        const int64_t rows_per = std::max<int64_t>(1, (int64_t)((size_t(16) << 20) / (sizeof(double) * n)));
        for (int64_t r = 0; r < R; r += (r == 0 ? std::min<int64_t>(2, rows_per) : rows_per)) f->chunk_begin.push_back(r);
        f->chunk_ev.resize(f->chunk_begin.size());
        for (cudaEvent_t& e : f->chunk_ev) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    f->times.assign(times, times + R);
    CU(cudaMemcpyAsync(f->d_times, f->times.data(), sizeof(double) * R, cudaMemcpyHostToDevice, st));
    if (mul) CU(cudaMemcpyAsync(f->d_W, mul, sizeof(double) * R * f->M, cudaMemcpyHostToDevice, st));
    // the table may still be read by launches already queued on `st`
    CU(cudaEventRecord(f->reuse_ev, st));
    CU(cudaStreamWaitEvent(f->copy_stream, f->reuse_ev, 0));
    for (size_t c = 0; c < f->chunk_begin.size(); ++c) {
        const int64_t r0 = f->chunk_begin[c], r1 = c + 1 < f->chunk_begin.size() ? f->chunk_begin[c + 1] : R;
        CU(cudaMemcpyAsync(f->d_stage + r0 * n, table + r0 * n, sizeof(double) * (r1 - r0) * n, cudaMemcpyHostToDevice,
                           f->copy_stream));
        CU(launch_permute_rows(net->d_reach_of_pos, f->d_stage + r0 * n, f->d_F + r0 * n, n, r1 - r0, f->copy_stream));
        CU(cudaEventRecord(f->chunk_ev[c], f->copy_stream));
    }
    f->waited = 0;
    return TXH_OK;
}

int txh_forcing_wait(txh_forcing* f)
{
    if (!f) return fail(TXH_E_INVALID, "null argument");
    if (f->copy_stream) CU(cudaStreamSynchronize(f->copy_stream));
    f->waited = f->chunk_ev.size();
    return TXH_OK;
}

void txh_forcing_destroy(txh_forcing* f)
{
    if (!f) return;
    if (f->copy_stream) {
        cudaStreamSynchronize(f->copy_stream);
        for (cudaEvent_t e : f->chunk_ev) cudaEventDestroy(e);
        cudaEventDestroy(f->reuse_ev);
        cudaStreamDestroy(f->copy_stream);
        cudaFree(f->d_stage);
    }
    cudaFree(f->d_F);
    if (f->d_times) cudaFree(f->d_times);
    if (f->d_W) cudaFree(f->d_W);
    delete f;
}

}  // extern "C"

namespace {
// Recording slot of every schedule position (-1: not recorded) -> net->d_rec_slot, once per call.  A reach listed twice
// keeps its last slot (txh_route_run's rule; txh_run_assimilating_rec refuses duplicates before it gets here).
int upload_rec_slots(txh_net* net, const int64_t* rec_reach, int64_t rec_count, cudaStream_t st)
{
    std::vector<int32_t> slot(net->topo.n, -1);
    for (int64_t k = 0; k < rec_count; ++k) {
        if (rec_reach[k] < 0 || rec_reach[k] >= net->topo.n) return fail(TXH_E_INVALID, "recorded reach out of range");
        slot[net->sched.pos_of_reach[rec_reach[k]]] = (int32_t)k;
    }
    CU(cudaMemcpyAsync(net->d_rec_slot, slot.data(), sizeof(int32_t) * net->topo.n, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    return TXH_OK;
}

// txh_route_run once the arguments are checked and the recording slots are on the device
int route_run_impl(txh_net* net, double* O, double* I, int64_t M, const txh_forcing* fo, int64_t t0_ns, int64_t dt_ns,
                   int64_t nsteps, int method, const Recording& rec, double* rowsum, double rowsum_scale,
                   const OwedUpdate* upd, cudaStream_t st)
{
    if (nsteps == 0) return TXH_OK;
    StepPlan plan;
    if (fo) { plan.times = fo->d_times; plan.R = fo->R; plan.t0_ns = t0_ns; plan.dt_ns = dt_ns; plan.method = method; }
    if (fo && fo->waited < fo->chunk_ev.size()) {
        // a table still arriving (txh_forcing_update_async): wait for the row chunks these steps interpolate in
        txh_forcing* fw = const_cast<txh_forcing*>(fo);
        const double x_end = (double)(t0_ns + nsteps * dt_ns);
        const int64_t need = std::min<int64_t>(fo->R - 1, std::lower_bound(fo->times.begin(), fo->times.end(), x_end) - fo->times.begin());
        while (fw->waited < fw->chunk_ev.size() && fw->chunk_begin[fw->waited] <= need) {
            CU(cudaStreamWaitEvent(st, fw->chunk_ev[fw->waited], 0));
            ++fw->waited;
        }
    }
    return run_routing(net, O, I, M, fo ? fo->d_F : nullptr, fo ? fo->d_W : nullptr, fo ? (int)fo->M : 0,
                       plan, nsteps, st, rec, rowsum, rowsum_scale, upd);
}
}  // namespace

extern "C" {

int txh_route_run(txh_net* net, double* O, double* I, int64_t M, const txh_forcing* fo, int64_t t0_ns,
                  int64_t dt_ns, int64_t nsteps, int method, const int64_t* rec_reach, int64_t rec_count,
                  int64_t rec_every, double* rec_out, void* stream)
{
    if (!net || !O || !I) return fail(TXH_E_INVALID, "null argument");
    if (nsteps < 0 || nsteps > (1 << 24)) return fail(TXH_E_INVALID, "nsteps out of range");
    if (fo && fo->net != net) return fail(TXH_E_INVALID, "forcing belongs to another network");
    if (fo && fo->d_W && fo->M != M) return fail(TXH_E_INVALID, "forcing member multipliers do not match M");
    if (rec_count > 0 && (!rec_reach || !rec_out || rec_every < 1)) return fail(TXH_E_INVALID, "bad recording arguments");
    int rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = check_M(M)) || (rc = ensure_device(net)) || (rc = ensure_coef(net, st))) return rc;
    if (nsteps == 0) return TXH_OK;
    if (rec_count > 0 && (rc = upload_rec_slots(net, rec_reach, rec_count, st))) return rc;
    const Recording rec{rec_count > 0 ? net->d_rec_slot : nullptr, rec_out, (int)rec_every, (int)rec_count, 0};
    return route_run_impl(net, O, I, M, fo, t0_ns, dt_ns, nsteps, method, rec, net->stats_rowsum, net->stats_scale,
                          nullptr, st);
}

int txh_route_step(txh_net* net, double* O, double* I, int64_t M, const double* q, void* stream)
{
    if (!net || !O || !I) return fail(TXH_E_INVALID, "null argument");
    int rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = check_M(M)) || (rc = ensure_device(net)) || (rc = ensure_coef(net, st))) return rc;
    if (q) CU(launch_permute_vec(net->d_reach_of_pos, q, net->d_qtmp, net->topo.n, st));
    return run_routing(net, O, I, M, q ? net->d_qtmp : nullptr, nullptr, 0, StepPlan(), 1, st);
}

int txh_route_step_levels(txh_net* net, double* O, double* I, int64_t M, const double* q, void* stream)
{
    if (!net || !O || !I) return fail(TXH_E_INVALID, "null argument");
    int rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = check_M(M)) || (rc = ensure_device(net)) || (rc = ensure_coef(net, st))) return rc;
    if (q) CU(launch_permute_vec(net->d_reach_of_pos, q, net->d_qtmp, net->topo.n, st));
    const Schedule& s = net->sched;
    for (int32_t l = 0; l + 1 < (int32_t)s.lvl_off.size(); ++l) {
        LevelArgs a{};
        a.lvl_pos = net->d_lvl_pos + s.lvl_off[l]; a.count = s.lvl_off[l + 1] - s.lvl_off[l];
        a.up_off = net->d_up_off; a.up_pos = net->d_up_pos; a.coef = net->d_coef;
        a.q = q ? net->d_qtmp : nullptr; a.O = O; a.I = I; a.ld = (int)txh_row_stride(M); a.M = (int)M;
        CU(launch_route_level(a, st));
    }
    return TXH_OK;
}

int txh_route_apply(txh_net* net, double* X, double* Iscr, int64_t M, void* stream)
{
    if (!net || !X || !Iscr) return fail(TXH_E_INVALID, "null argument");
    int rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = check_M(M)) || (rc = ensure_device(net)) || (rc = ensure_coef(net, st))) return rc;
    // nutils.py:148-154: i_prev = init_inflows(o_prev) (self-loop included), then _ax
    CU(launch_init_inflows(net->d_up_off, net->d_up_pos, net->d_outlet, X, Iscr, net->topo.n,
                           (int)txh_row_stride(M), (int)M, st));
    return run_routing(net, X, Iscr, M, nullptr, nullptr, 0, StepPlan(), 1, st);
}

int txh_apply_gain(txh_net* net, const double* G, double* O, double* I, int64_t M, void* stream)
{
    if (!net || !G || !O || !I) return fail(TXH_E_INVALID, "null argument");
    int rc;
    if ((rc = check_M(M)) || (rc = ensure_device(net))) return rc;
    CU(launch_apply_gain(net->d_up_off, net->d_up_pos, G, O, I, net->topo.n, (int)txh_row_stride(M), (int)M,
                         (cudaStream_t)stream));
    return TXH_OK;
}

int txh_check(txh_net* net, void* stream)
{
    if (!net) return fail(TXH_E_INVALID, "null argument");
    if (!net->dev_ready) return TXH_OK;
    // the status word (watchdog) and the solver info word travel only here: launches stay back to back
    return report_status(net, (cudaStream_t)stream);
}

}  // extern "C"

// ---- assimilation ---------------------------------------------------------------------------
namespace {
int obs_positions(txh_net* net, const int64_t* obs, int64_t m, cudaStream_t st, int32_t** d_pos)
{
    if ((int64_t)net->obs_cached.size() == m && std::equal(obs, obs + m, net->obs_cached.begin())) {
        *d_pos = net->d_obs;                              // same gauges as last time: already resident
        return TXH_OK;
    }
    std::vector<int32_t> pos(m);
    for (int64_t k = 0; k < m; ++k) {
        if (obs[k] < 0 || obs[k] >= net->topo.n) return fail(TXH_E_INVALID, "gauge reach index out of range");
        if (k > 0 && obs[k] <= obs[k - 1]) return fail(TXH_E_INVALID, "gauge reach indices must be strictly ascending");
        pos[k] = net->sched.pos_of_reach[obs[k]];
    }
    int rc;
    if ((rc = grow(&net->d_obs, &net->obs_cap, (size_t)m, st))) return rc;
    std::vector<int32_t> gop(net->topo.n, -1);
    for (int64_t k = 0; k < m; ++k) gop[pos[k]] = (int32_t)k;
    if (!net->d_gauge_of_pos) CU(cudaMalloc((void**)&net->d_gauge_of_pos, sizeof(int32_t) * net->topo.n));
    CU(cudaMemcpyAsync(net->d_obs, pos.data(), sizeof(int32_t) * m, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(net->d_gauge_of_pos, gop.data(), sizeof(int32_t) * net->topo.n, cudaMemcpyHostToDevice, st));
    // gauge terms of the update per window task (route_window_kernel applies the update while it loads a task): the
    // gauged row itself (kind 0) and the row it drains into (kind 1: its inflow takes the gain of the gauged row,
    // nutils.py:127-134; the up lists hold no self-loops)
    const Schedule& s = net->sched;
    const size_t ntask = s.wtasks.size();
    std::vector<int32_t> task_of_pos(net->topo.n, -1), down(net->topo.n, -1);
    for (size_t k = 0; k < ntask; ++k)
        for (int32_t r = 0; r < s.wtasks[k].len; ++r) task_of_pos[s.wtasks[k].begin + r] = (int32_t)k;
    for (int64_t k = 0; k < net->topo.n; ++k)
        for (int32_t u = s.up_off[k]; u < s.up_off[k + 1]; ++u) down[s.up_pos[u]] = (int32_t)k;
    std::vector<std::vector<int2>> per_task(ntask);
    bool fix_ok = ntask > 0;
    for (int64_t g = 0; g < m && fix_ok; ++g) {
        const int32_t k = pos[g], d = down[k];
        if (task_of_pos[k] < 0 || (d >= 0 && task_of_pos[d] < 0)) { fix_ok = false; break; }
        per_task[task_of_pos[k]].push_back(make_int2(k - s.wtasks[task_of_pos[k]].begin, (int)g));
        if (d >= 0) per_task[task_of_pos[d]].push_back(make_int2((d - s.wtasks[task_of_pos[d]].begin) | (1 << 16), (int)g));
    }
    std::vector<int32_t> goff(ntask + 1, 0);
    std::vector<int2> gfix;
    if (fix_ok)
        for (size_t k = 0; k < ntask; ++k) { gfix.insert(gfix.end(), per_task[k].begin(), per_task[k].end()); goff[k + 1] = (int32_t)gfix.size(); }
    if (!net->d_gfix_off) CU(cudaMalloc((void**)&net->d_gfix_off, sizeof(int32_t) * (ntask + 1)));
    if ((rc = grow(&net->d_gfix, &net->gfix_cap, std::max<size_t>(gfix.size(), 16), st))) return rc;
    net->gfix_ok = fix_ok;
    CU(cudaMemcpyAsync(net->d_gfix_off, goff.data(), sizeof(int32_t) * (ntask + 1), cudaMemcpyHostToDevice, st));
    if (!gfix.empty()) CU(cudaMemcpyAsync(net->d_gfix, gfix.data(), sizeof(int2) * gfix.size(), cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    net->obs_cached.assign(obs, obs + m);
    *d_pos = net->d_obs;
    return TXH_OK;
}
int* info_word(txh_net* net) { return net->d_status + 1; }
}  // namespace

extern "C" {

int txh_set_stats_output(txh_net* net, double* rowsum, double scale)
{
    if (!net) return fail(TXH_E_INVALID, "null argument");
    net->stats_rowsum = rowsum; net->stats_scale = scale;
    return TXH_OK;
}

int txh_enkf_stats(txh_net* net, const double* O, int64_t Mloc, const int64_t* obs, int64_t m, double scale,
                   double* rowsum, double* HX, void* stream)
{
    if (!net || !O || !obs || !HX || m < 1) return fail(TXH_E_INVALID, "bad argument");
    int rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = check_M(Mloc)) || (rc = ensure_device(net))) return rc;
    int32_t* d_pos = nullptr;
    if ((rc = obs_positions(net, obs, m, st, &d_pos))) return rc;
    const int ld = (int)txh_row_stride(Mloc);
    if (rowsum) CU(launch_enkf_stats(O, ld, (int)Mloc, net->topo.n, scale, net->d_gauge_of_pos, rowsum, HX, st));
    else CU(launch_gather_rows(d_pos, m, O, ld, (int)Mloc, HX, st));       // the sums came with the routing launch
    return TXH_OK;
}

int64_t txh_enkf_work_size(int64_t m, int64_t Mtot)
{
    const int64_t direct = m * m + 2 * m * Mtot + m;
    const int64_t nsplit = Mtot <= 128 ? 8 : 1;
    const int64_t woodbury = 4 * m * Mtot + nsplit * 2 * Mtot * Mtot + Mtot * Mtot;
    return std::max(direct, woodbury);
}

}  // extern "C"

namespace {
// txh_enkf_solve; with O_gather the gauge rows HX are gathered from the state (unsharded ensemble, ld = row stride of
// Mtot members) inside the first kernel instead of by a launch of their own
int enkf_solve_impl(txh_net* net, int64_t m, int64_t Mtot, double* HX, const double* O_gather, const double* Zp,
                    const double* mean, const int64_t* obs, const double* qs, const double* R, const double* Dinv,
                    int dinv_kind, double* work, double* W, double* T, void* stream)
{
    if (!net || !HX || !Zp || !mean || !obs || !qs || !R || !work || !W || !T || m < 1 || Mtot < 2)
        return fail(TXH_E_INVALID, "bad argument");
    if (dinv_kind < 0 || dinv_kind > 2 || (dinv_kind != 0 && !Dinv)) return fail(TXH_E_INVALID, "bad D^-1 argument");
    int rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = ensure_device(net))) return rc;
    int32_t* d_pos = nullptr;
    if ((rc = obs_positions(net, obs, m, st, &d_pos))) return rc;
    if (dinv_kind != 0 && Mtot < m) {
        // ensemble-space form (txh_da.cu): the Mtot x Mtot system replaces the m x m one and T is its solution
        const int Mt = (int)Mtot, nsplit = Mtot <= 128 ? 8 : 1;
        static const bool fused_ok = [] { const char* k = getenv("TXH_ENKF_FUSED"); return !(k && atoi(k) == 0); }();
        if (fused_ok && dinv_kind == 1 && Mt <= 64) {
            // one cluster launch: gather, split-K product, reduction, Cholesky solve and W (txh_da.cu)
            CU(launch_enkf_small_system(HX, O_gather, (int)txh_row_stride(Mtot), Zp, mean, d_pos, Dinv, (int)m, Mt,
                                        (double)(Mtot - 1), T, W, info_word(net), st));
            return TXH_OK;
        }
        double* Bc = work;                                  // [m][2Mt] = [HA | dz]
        double* Y = Bc + 2 * m * Mtot;                      // [m][2Mt] = D^-1 Bc
        double* Cp = Y + 2 * m * Mtot;                      // [nsplit][Mt][2Mt] split-K partials of HA^T Y
        CU(launch_innovation_cat(HX, O_gather, (int)txh_row_stride(Mtot), Zp, mean, d_pos, dinv_kind == 1 ? Dinv : nullptr,
                                 (int)m, Mt, Bc, Y, st));
        if (dinv_kind == 2)
            CU(launch_dgemm(0, 0, (int)m, 2 * Mt, (int)m, 1.0, Dinv, (int)m, Bc, 2 * Mt, 0.0, Y, 2 * Mt, st));
        CU(launch_dgemm_splitk(1, 0, Mt, 2 * Mt, (int)m, Bc, 2 * Mt, Y, 2 * Mt, Cp, 2 * Mt, nsplit,
                               (long long)Mt * 2 * Mt, st));
        if (Mt <= 128) {
            CU(launch_chol_solve_small(Cp, nsplit, (long long)Mt * 2 * Mt, Mt, (double)(Mtot - 1), T, info_word(net), st));
        } else {
            double* Cf = Cp + (size_t)nsplit * 2 * Mt * Mt;  // blocked Cholesky: (C0 + (Mt-1) I) Z = C1, Z in place in T
            CU(launch_woodbury_assemble(Cp, nsplit, (long long)Mt * 2 * Mt, Mt, (double)(Mtot - 1), Cf, T, st));
            CU(launch_spd_solve(Cf, T, Mt, Mt, info_word(net), st));
        }
        // W = Y_dz - Y_HA Z
        CU(launch_dgemm_ex(0, 0, (int)m, Mt, Mt, -1.0, Y, 2 * Mt, T, Mt, 1.0, Y + Mt, 2 * Mt, W, Mt, st));
    } else {
        if (O_gather) CU(launch_gather_rows(d_pos, m, O_gather, (int)txh_row_stride(Mtot), (int)Mtot, HX, st));
        double* S = work;
        double* HA = S + m * m;
        double* mean_obs = HA + m * Mtot;
        CU(launch_gather_rows(d_pos, m, mean, 1, 1, mean_obs, st));
        CU(launch_innovation(HX, Zp, mean_obs, (int)m, (int)Mtot, HA, W, st));                    // W <- dz
        CU(launch_dgemm(0, 1, (int)m, (int)m, (int)Mtot, 1.0, HA, (int)Mtot, HA, (int)Mtot, 0.0, S, (int)m, st));
        CU(launch_innov_cov_finish(S, qs, R, (int)m, 1.0 / (double)(Mtot - 1), st));
        CU(launch_spd_solve(S, W, (int)m, (int)Mtot, info_word(net), st));                        // W <- S^-1 dz
        CU(launch_dgemm(1, 0, (int)Mtot, (int)Mtot, (int)m, 1.0 / (double)(Mtot - 1), HA, (int)Mtot, W, (int)Mtot, 0.0,
                        T, (int)Mtot, st));
    }
    // asynchronous: a failed factorisation leaves a non-zero info word that txh_check reports
    return TXH_OK;
}
}  // namespace

extern "C" {

int txh_enkf_solve(txh_net* net, int64_t m, int64_t Mtot, const double* HX, const double* Zp, const double* mean,
                   const int64_t* obs, const double* qs, const double* R, const double* Dinv, int dinv_kind,
                   double* work, double* W, double* T, void* stream)
{
    return enkf_solve_impl(net, m, Mtot, const_cast<double*>(HX), nullptr, Zp, mean, obs, qs, R, Dinv, dinv_kind, work, W, T,
                           stream);
}

int txh_enkf_apply(txh_net* net, double* O, double* I, int64_t Mloc, const double* Xall, int64_t ldx,
                   int64_t x_block_stride, int64_t Mtot, int64_t col0, const double* mean, const double* T, const int64_t* obs, int64_t m, const double* qs,
                   const double* W, double* G, void* stream)
{
    if (!net || !O || !I || !mean || !T || !obs || !qs || !W || !G) return fail(TXH_E_INVALID, "null argument");
    if (col0 < 0 || col0 + Mloc > Mtot) return fail(TXH_E_INVALID, "shard columns out of range");
    int rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = check_M(Mloc)) || (rc = ensure_device(net))) return rc;
    int32_t* d_pos = nullptr;
    if ((rc = obs_positions(net, obs, m, st, &d_pos))) return rc;
    const int ld = (int)txh_row_stride(Mloc);
    if (!Xall) { if (Mtot != Mloc) return fail(TXH_E_INVALID, "gathered ensemble missing"); Xall = O; ldx = ld; x_block_stride = 0; }
    if (x_block_stride != 0 && (Mtot % Mloc != 0 || ldx < Mloc)) return fail(TXH_E_INVALID, "bad gathered-ensemble layout");
    const int Mb = x_block_stride != 0 ? (int)Mloc : (int)Mtot;
    // O += gain and G = gain (tensor cores), gauge rows, then I += sum of the upstream gains.  The in-place
    // update of O is row-local; when the ensemble being transformed IS O and a row spans several 64-column
    // groups, a later group would read members an earlier one has already updated: then O is updated from G
    // afterwards instead.
    const bool fuse_o = Xall != O || ld <= 64;
    CU(launch_enkf_update(Xall, (int)ldx, (int)Mtot, mean, T + col0, (int)Mtot, (int)Mloc, fuse_o ? O : nullptr, G, ld,
                          net->topo.n, net->d_gauge_of_pos, qs, W, (int)col0, net->num_sms, Mb, (long long)x_block_stride,
                          st));
    if (fuse_o) CU(launch_inflow_gain(net->d_inner, net->n_inner, net->d_up_off, net->d_up_pos, G, I, ld, st));
    else CU(launch_apply_gain(net->d_up_off, net->d_up_pos, G, O, I, net->topo.n, ld, (int)Mloc, st));
    return TXH_OK;
}

int txh_enkf_apply_peers(txh_net* net, const double* O_in, double* O_out, double* I, int64_t Mloc,
                         const double* const* shard_ptrs, int64_t world, int64_t Mtot, int64_t col0, const double* mean,
                         const double* T, const int64_t* obs, int64_t m, const double* qs, const double* W, double* G,
                         void* stream)
{
    if (!net || !O_in || !O_out || !I || !shard_ptrs || !mean || !T || !obs || !qs || !W || !G)
        return fail(TXH_E_INVALID, "null argument");
    if (world < 1 || world > kMaxPeers || Mtot != Mloc * world) return fail(TXH_E_INVALID, "bad shard layout");
    if (col0 < 0 || col0 + Mloc > Mtot) return fail(TXH_E_INVALID, "shard columns out of range");
    if (O_in == O_out) return fail(TXH_E_INVALID, "the posterior needs a buffer of its own: peers may still read O_in");
    int rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = check_M(Mloc)) || (rc = ensure_device(net))) return rc;
    int32_t* d_pos = nullptr;
    if ((rc = obs_positions(net, obs, m, st, &d_pos))) return rc;
    const int ld = (int)txh_row_stride(Mloc);
    PeerBlocks pb{};
    pb.count = (int)world;
    for (int64_t b = 0; b < world; ++b) {
        if (!shard_ptrs[b]) return fail(TXH_E_INVALID, "null shard pointer");
        pb.p[b] = shard_ptrs[b];
    }
    CU(launch_enkf_update(O_in, ld, (int)Mtot, mean, T + col0, (int)Mtot, (int)Mloc, const_cast<double*>(O_in), G, ld,
                          net->topo.n, net->d_gauge_of_pos, qs, W, (int)col0, net->num_sms, (int)Mloc, 0, st, &pb, O_out));
    CU(launch_inflow_gain(net->d_inner, net->n_inner, net->d_up_off, net->d_up_pos, G, I, ld, st));
    return TXH_OK;
}

int txh_run_assimilating(txh_net* net, double* O, double* I, int64_t M, const txh_forcing* fo, int64_t t0_ns,
                         int64_t dt_ns, int64_t nsteps, int64_t every, int method, const int64_t* obs, int64_t m,
                         const double* Zp, const double* qs, const double* R, const double* Dinv, int dinv_kind,
                         double* rowsum, double* HX, double* work, double* W, double* T, double* G, int64_t time_every,
                         void* obs_ready_event, void* stream)
{
    return txh_run_assimilating_rec(net, O, I, M, fo, t0_ns, dt_ns, nsteps, every, method, obs, m, Zp, qs, R, Dinv, dinv_kind,
                                    rowsum, HX, work, W, T, G, time_every, obs_ready_event, nullptr, 0, 1, nullptr, nullptr,
                                    stream);
}

int txh_run_assimilating_rec(txh_net* net, double* O, double* I, int64_t M, const txh_forcing* fo, int64_t t0_ns,
                             int64_t dt_ns, int64_t nsteps, int64_t every, int method, const int64_t* obs, int64_t m,
                             const double* Zp, const double* qs, const double* R, const double* Dinv, int dinv_kind,
                             double* rowsum, double* HX, double* work, double* W, double* T, double* G, int64_t time_every,
                             void* obs_ready_event, const int64_t* rec_reach, int64_t rec_count, int64_t rec_every,
                             double* rec_out, double* prior_out, void* stream)
{
    if (!net || !O || !I || !obs || !Zp || !qs || !R || !rowsum || !HX || !work || !W || !T || !G || every < 1 || m < 1)
        return fail(TXH_E_INVALID, "bad argument");
    if (rec_count < 0 || rec_every < 1 || (rec_count > 0 && (!rec_reach || !rec_out)))
        return fail(TXH_E_INVALID, "bad recording arguments");
    if (net->T_hist && (nsteps / every) * M * M > net->T_hist_cap)
        return fail(TXH_E_INVALID, "the transform history holds fewer than nsteps / every transforms of M x M");
    // segments: nwin windows of `every` steps, each followed by an update, then the remaining steps
    const int64_t nwin = nsteps / every, nseg = nwin + (nsteps > nwin * every ? 1 : 0);
    auto seg_steps = [&](int64_t k) { return k < nwin ? every : nsteps - nwin * every; };
    // the checks txh_route_run makes of every routing call
    if (nwin > 0 && every > (1 << 24)) return fail(TXH_E_INVALID, "nsteps out of range");
    if (fo && fo->net != net) return fail(TXH_E_INVALID, "forcing belongs to another network");
    if (fo && fo->d_W && fo->M != M) return fail(TXH_E_INVALID, "forcing member multipliers do not match M");
    int rc;
    if ((rc = check_M(M))) return rc;
    const bool rec = rec_count > 0;
    if (rec) {
        std::vector<char> seen(net->topo.n, 0);
        for (int64_t k = 0; k < rec_count; ++k) {
            if (rec_reach[k] < 0 || rec_reach[k] >= net->topo.n) return fail(TXH_E_INVALID, "recorded reach out of range");
            if (seen[rec_reach[k]]++) return fail(TXH_E_INVALID, "recorded reach listed twice");
        }
    }
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = ensure_device(net)) || (rc = ensure_coef(net, st))) return rc;
    if (rec) {
        // the slots and positions of the recorded reaches once per call
        if ((rc = upload_rec_slots(net, rec_reach, rec_count, st)) ||
            (rc = grow(&net->d_rec_pos, &net->rec_pos_cap, (size_t)rec_count, st)))
            return rc;
        std::vector<int32_t> pos(rec_count);
        for (int64_t k = 0; k < rec_count; ++k) pos[k] = net->sched.pos_of_reach[rec_reach[k]];
        CU(cudaMemcpyAsync(net->d_rec_pos, pos.data(), sizeof(int32_t) * rec_count, cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));
    }
    const int ld = (int)txh_row_stride(M);
    // where update k's transform goes and where its consumers read it
    auto T_of = [&](int64_t k) -> double* { return net->T_hist ? net->T_hist + (size_t)k * M * M : T; };
    // where update k's recorded rows go: the forecast to prior_out[k], the posterior -- what the state holds after step
    // (k+1) every -- to that step's rec_out slot (the routing launch recorded the forecast there)
    auto rec_prior_of = [&](int64_t k) -> double* {
        return rec && prior_out ? prior_out + (size_t)k * rec_count * M : nullptr;
    };
    auto rec_post_of = [&](int64_t k) -> double* {
        const int64_t s_end = (k + 1) * every;
        return rec && s_end % rec_every == 0 ? rec_out + (size_t)(s_end / rec_every - 1) * rec_count * M : nullptr;
    };
    // Right after a routing launch the forecast inflows are exactly the sums of the upstream forecast outflows
    // (nutils.py:84-85), so i + N gain = N (o + gain): the gains are never stored.  When the window kernel routes the
    // next segment, it applies the update itself while it loads its tasks (p is linear in the state rows, txh_window.cu):
    // the posterior state only goes to memory after the last window; otherwise the transform kernel updates O in place
    // and the posterior inflows are rebuilt from the posterior outflows.
    static const bool fuse_load_ok = [] { const char* k = getenv("TXH_ENKF_FUSE_LOAD"); return !(k && atoi(k) == 0); }();
    const WindowFit fit = window_fit(net, M);
    const bool fuse_load = fuse_load_ok && ld <= kMemberBlock && (net->route_kernel == 0 || net->route_kernel == 2) &&
                           !lane_wanted(net, M, every) && fit.ok && fit.wpc_upd >= 2;
    // update k applied by the stand-alone kernels: its rows recorded first, while O still holds the forecast
    auto apply_update = [&](int64_t k) -> int {
        double *prior = rec_prior_of(k), *post = rec_post_of(k);
        if (prior || post)
            CU(launch_enkf_record(O, ld, (int)M, rowsum, T_of(k), net->d_gauge_of_pos, qs, W, net->d_rec_pos, (int)rec_count,
                                  prior, post, st));
        if (ld > kMemberBlock) return txh_enkf_apply(net, O, I, M, nullptr, 0, 0, M, 0, rowsum, T_of(k), obs, m, qs, W, G, stream);
        CU(launch_enkf_update(O, ld, (int)M, rowsum, T_of(k), (int)M, (int)M, O, nullptr, ld, net->topo.n, net->d_gauge_of_pos,
                              qs, W, 0, net->num_sms, (int)M, 0, st));
        CU(launch_inflow_rebuild(net->d_inner_rec, net->n_inner, net->d_up_off, net->d_up_pos, O, I, ld, st));
        return TXH_OK;
    };
    OwedUpdate owed{};                                     // the update the next routing launch applies, if handed over
    bool handed_over = false;
    int64_t t = t0_ns;
    for (int64_t k = 0; k < nseg; ++k) {
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        const bool timed = k < nwin && time_every > 0 && k % time_every == 0 && net->route_events.size() < 4096;
        if (timed) { CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1)); CU(cudaEventRecord(e0, st)); }
        const Recording rk = rec ? Recording{net->d_rec_slot, rec_out, (int)rec_every, (int)rec_count, k * every} : Recording();
        // the row sums of the forecast ride on the last step of every window (the mean of the update)
        rc = route_run_impl(net, O, I, M, fo, t, dt_ns, seg_steps(k), method, rk, k < nwin ? rowsum : nullptr,
                            1.0 / (double)M, handed_over ? &owed : nullptr, st);
        if (timed) { CU(cudaEventRecord(e1, st)); net->route_events.emplace_back(e0, e1); }
        if (rc != TXH_OK) return rc;
        if (k == nwin) break;                              // the remaining steps: no update follows
        t += every * dt_ns;
        // observations still on their way (copied on another stream): the first update waits for them, the first
        // window does not
        if (k == 0 && obs_ready_event) CU(cudaStreamWaitEvent(st, (cudaEvent_t)obs_ready_event, 0));
        if ((rc = enkf_solve_impl(net, m, M, HX, O, Zp + (size_t)k * m * M, rowsum, obs, qs, R, Dinv, dinv_kind, work, W,
                                  T_of(k), stream)))
            return rc;
        // the update rides on the next routing launch when that is a window launch with room for it (and every gauge
        // term falls in a window task); otherwise, and after the last segment, the stand-alone kernels apply it now
        handed_over = fuse_load && k + 1 < nseg && net->gfix_ok && !lane_wanted(net, M, seg_steps(k + 1));
        if (handed_over) owed = OwedUpdate{T_of(k), W, qs, M, rec_prior_of(k), rec_post_of(k), rowsum};
        else if ((rc = apply_update(k))) return rc;
    }
    return TXH_OK;
}

int txh_set_transform_history(txh_net* net, double* T_hist, int64_t capacity)
{
    if (!net) return fail(TXH_E_INVALID, "null argument");
    if (T_hist && capacity < 0) return fail(TXH_E_INVALID, "negative transform history capacity");
    net->T_hist = T_hist; net->T_hist_cap = T_hist ? capacity : 0;
    return TXH_OK;
}

int64_t txh_enks_work_size(int64_t M, int64_t nupd) { return M < 1 || nupd < 0 ? 0 : 6 * nupd * M * M; }

int txh_enks_smooth(int64_t M, int64_t nupd, int64_t every, const double* T_hist, int64_t nslots, int64_t rec_count,
                    int64_t rec_every, int64_t lag, const double* rec, double* out, double* work, void* stream)
{
    if (M < 2 || M > 4096) return fail(TXH_E_INVALID, "member count out of range [2, 4096]");
    if (nupd < 0 || nupd > (int64_t(1) << 30) || every < 1) return fail(TXH_E_INVALID, "bad update count or cadence");
    if (nslots < 0 || rec_count < 0 || rec_every < 1) return fail(TXH_E_INVALID, "bad recording shape");
    if (lag < 0) return fail(TXH_E_INVALID, "negative smoother lag");
    if (!T_hist || !rec || !out || !work) return fail(TXH_E_INVALID, "null buffer");
    const uintptr_t bytes = (uintptr_t)(nslots * rec_count * M) * sizeof(double);
    const uintptr_t r0 = (uintptr_t)rec, o0 = (uintptr_t)out;
    if (bytes > 0 && r0 < o0 + bytes && o0 < r0 + bytes)
        return fail(TXH_E_INVALID, "out overlaps rec: the smoothed hydrographs need a buffer of their own");
    if (txh_device_count() == 0) return fail(TXH_E_NODEVICE, "no CUDA device visible: libtxh has no CPU fallback");
    CU(launch_enks_smooth((int)M, (int)nupd, every, T_hist, nslots, rec_count, rec_every, lag, rec, out, work,
                          (cudaStream_t)stream));
    return TXH_OK;
}

int txh_get_route_timings(txh_net* net, double* ms_out, int64_t capacity, int64_t* count)
{
    if (!net || !count || (capacity > 0 && !ms_out)) return fail(TXH_E_INVALID, "null argument");
    *count = (int64_t)net->route_events.size();
    for (int64_t i = 0; i < *count && i < capacity; ++i) {
        float ms = 0.f;
        CU(cudaEventSynchronize(net->route_events[i].second));
        CU(cudaEventElapsedTime(&ms, net->route_events[i].first, net->route_events[i].second));
        ms_out[i] = ms;
    }
    if (capacity >= *count) {                                  // read out: the events are done with
        for (auto& ev : net->route_events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
        net->route_events.clear();
    }
    return TXH_OK;
}

int txh_dgemm(int transA, int transB, int64_t M, int64_t N, int64_t K, double alpha, const double* A, int64_t lda,
              const double* B, int64_t ldb, double beta, double* C, int64_t ldc, void* stream)
{
    // K = 0: A and B are never read (C = beta C), so empty operands may come without an address
    if ((K > 0 && (!A || !B)) || !C || M < 0 || N < 0 || K < 0) return fail(TXH_E_INVALID, "bad argument");
    if (txh_device_count() == 0) return fail(TXH_E_NODEVICE, "no CUDA device visible: libtxh has no CPU fallback");
    CU(launch_dgemm(transA, transB, (int)M, (int)N, (int)K, alpha, A, (int)lda, B, (int)ldb, beta, C, (int)ldc,
                    (cudaStream_t)stream));
    return TXH_OK;
}

int txh_spd_solve(int64_t m, int64_t k, double* S, double* B, void* stream)
{
    if (!S || !B || m < 1 || k < 1) return fail(TXH_E_INVALID, "bad argument");
    if (txh_device_count() == 0) return fail(TXH_E_NODEVICE, "no CUDA device visible: libtxh has no CPU fallback");
    cudaStream_t st = (cudaStream_t)stream;
    int* d_info = nullptr;
    CU(cudaMalloc((void**)&d_info, sizeof(int)));
    CU(cudaMemsetAsync(d_info, 0, sizeof(int), st));
    CU(launch_spd_solve(S, B, (int)m, (int)k, d_info, st));
    int info = 0;
    CU(cudaMemcpyAsync(&info, d_info, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    cudaFree(d_info);
    if (info != 0) return fail(TXH_E_INVALID, "matrix is not positive definite");
    return TXH_OK;
}

int txh_inverse(int64_t m, double* A, double* work, void* stream)
{
    if (!A || !work || m < 1) return fail(TXH_E_INVALID, "bad argument");
    if (txh_device_count() == 0) return fail(TXH_E_NODEVICE, "no CUDA device visible: libtxh has no CPU fallback");
    cudaStream_t st = (cudaStream_t)stream;
    int* d_info = nullptr;
    CU(cudaMalloc((void**)&d_info, sizeof(int)));
    CU(cudaMemsetAsync(d_info, 0, sizeof(int), st));
    CU(launch_inverse(A, work, (int)m, d_info, st));
    int info = 0;
    CU(cudaMemcpyAsync(&info, d_info, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    cudaFree(d_info);
    if (info != 0) return fail(TXH_E_INVALID, "matrix is singular");
    return TXH_OK;
}

static inline int64_t up4(int64_t x) { return (x + 3) & ~int64_t(3); }

int64_t txh_kf_work_size(const txh_net* net, int64_t m)
{
    if (!net || m < 1) return 0;
    const int64_t n = net->topo.n, ld = txh_row_stride(n);
    return 2 * n * ld + up4(n * n) + 2 * up4(n * m) + 2 * up4(m * m) + up4(2 * n) + up4(m) + 16;
}

int txh_kf_filter(txh_net* net, const double* P_in, double* P_out, double* P_prior, const double* Q, const double* R,
                  const int64_t* obs, int64_t m, const double* z, double* O, double* I, double* K, double* gain,
                  double* dz, double* work, void* stream)
{
    if (!net || !P_in || !P_out || !Q || !R || !obs || !z || !O || !I || !K || !gain || !dz || !work || m < 1)
        return fail(TXH_E_INVALID, "bad argument");
    int rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = net->topo.n;
    if ((rc = check_M(n)) || (rc = ensure_device(net)) || (rc = ensure_coef(net, st))) return rc;
    if (m > n) return fail(TXH_E_INVALID, "more gauges than reaches");
    int32_t* d_pos = nullptr;
    if ((rc = obs_positions(net, obs, m, st, &d_pos))) return rc;
    const int ld = (int)txh_row_stride(n), ld1 = (int)txh_row_stride(1);
    double* X = work;
    double* X2 = X + n * ld;
    double* Pm = P_prior ? P_prior : X2 + n * ld;
    double* Ps = X2 + n * ld + up4(n * n);
    double* Prow = Ps + up4(n * m);
    double* S = Prow + up4(n * m);
    double* Sw = S + up4(m * m);
    double* Gp = Sw + up4(m * m);
    double* zd = Gp + up4(2 * n);
    CU(cudaMemcpyAsync(zd, z, sizeof(double) * m, cudaMemcpyHostToDevice, st));
    // P- = A (A P)^T + Q, nutils.py:194-214 (X2 doubles as the inflow scratch of the first pass and vice versa)
    CU(launch_pack(net->d_reach_of_pos, P_in, X, n, (int)n, ld, 0, st));
    CU(launch_init_inflows(net->d_up_off, net->d_up_pos, net->d_outlet, X, X2, n, ld, (int)n, st));
    if ((rc = run_routing(net, X, X2, n, nullptr, nullptr, 0, StepPlan(), 1, st))) return rc;
    CU(launch_kf_repack_transposed(net->d_reach_of_pos, net->d_pos_of_reach, X, X2, (int)n, ld, st));
    CU(launch_init_inflows(net->d_up_off, net->d_up_pos, net->d_outlet, X2, X, n, ld, (int)n, st));
    if ((rc = run_routing(net, X2, X, n, nullptr, nullptr, 0, StepPlan(), 1, st))) return rc;
    CU(launch_kf_prior_finish(net->d_reach_of_pos, net->d_pos_of_reach, net->d_gauge_of_pos, X2, ld, Q, R, (int)n, (int)m,
                              Pm, Ps, Prow, S, st));
    // K = P-[:, s] inv(P-[s][:, s] + R)   (da.py:119)
    CU(launch_inverse(S, Sw, (int)m, info_word(net), st));
    CU(launch_dgemm(0, 0, (int)n, (int)m, (int)m, 1.0, Ps, (int)m, S, (int)m, 0.0, K, (int)m, st));
    // dz = z - o[s], gain = K dz (da.py:112, 121), P+ = P- - K P-[s] (da.py:122)
    CU(launch_kf_gain(net->d_reach_of_pos, d_pos, zd, O, ld1, K, (int)n, (int)m, dz, gain, Gp, st));
    CU(launch_dgemm_ex(0, 0, (int)n, (int)n, (int)m, -1.0, K, (int)m, Prow, (int)n, 1.0, Pm, (int)n, P_out, (int)n, st));
    // da.py:124-126
    CU(launch_apply_gain(net->d_up_off, net->d_up_pos, Gp, O, I, n, ld1, 1, st));
    return TXH_OK;
}

}  // extern "C"

// ---- batched dense Kalman filters of a generation of sub-models ---------------------------------------------------
struct txh_kfb {
    txh_net* net = nullptr;                    // the UNION network of the sub-models (reach order: block after block)
    std::vector<KfbBlock> blocks;
    int64_t n_u = 0, m_tot = 0, pp = 0, nm = 0, mm = 0;
    int max_n = 0, max_m = 0, ld = 0;
    KfbBlock* d_blocks = nullptr;
    int32_t *d_blk_of_reach = nullptr, *d_gl_of_reach = nullptr, *d_obs_reach = nullptr;
    double *d_P = nullptr, *d_Pprev = nullptr, *d_Q = nullptr, *d_R = nullptr, *d_Pm = nullptr, *d_Ps = nullptr, *d_Prow = nullptr,
           *d_S = nullptr, *d_K = nullptr, *d_z = nullptr, *d_dz = nullptr, *d_gain = nullptr, *d_Gp = nullptr, *d_X = nullptr,
           *d_X2 = nullptr;
};

extern "C" {

// kfb_inverse_kernel holds a block's m x m system and four m-vectors in 200 KB of shared memory
int64_t txh_kfb_max_gauges(void)
{
    int64_t m = 0;
    while ((size_t)4 * (m + 1) + (size_t)(m + 1) * (m + 1) <= 200 * 1024 / sizeof(double)) ++m;
    return m;
}

int txh_kfb_create(txh_net* net, int64_t nblocks, const int64_t* n_k, const int64_t* m_k, const int64_t* obs_local, txh_kfb** out)
{
    if (!net || !n_k || !m_k || !obs_local || !out || nblocks < 1) return fail(TXH_E_INVALID, "bad argument");
    int rc;
    if ((rc = ensure_device(net))) return rc;
    txh_kfb* b = new (std::nothrow) txh_kfb();
    if (!b) return fail(TXH_E_INVALID, "out of memory");
    b->net = net;
    std::vector<int32_t> blk_of_reach, gl_of_reach, obs_reach;
    int64_t row0 = 0, g0 = 0;
    for (int64_t k = 0; k < nblocks; ++k) {
        if (n_k[k] < 1 || m_k[k] < 1 || m_k[k] > n_k[k]) { delete b; return fail(TXH_E_INVALID, "bad block size"); }
        KfbBlock blk{};
        blk.n = (int32_t)n_k[k]; blk.m = (int32_t)m_k[k]; blk.row0 = (int32_t)row0; blk.g_off = (int32_t)g0; blk.active = 1;
        blk.p_off = b->pp; blk.nm_off = b->nm; blk.mm_off = b->mm;
        b->pp += n_k[k] * n_k[k]; b->nm += n_k[k] * m_k[k]; b->mm += m_k[k] * m_k[k];
        b->max_n = std::max(b->max_n, blk.n); b->max_m = std::max(b->max_m, blk.m);
        std::vector<int32_t> gl(n_k[k], -1);
        for (int64_t g = 0; g < m_k[k]; ++g) {
            const int64_t j = obs_local[g0 + g];
            if (j < 0 || j >= n_k[k] || (g > 0 && j <= obs_local[g0 + g - 1])) {
                delete b; return fail(TXH_E_INVALID, "gauge indices of a block must be strictly ascending local reaches");
            }
            gl[j] = (int32_t)g;
            obs_reach.push_back((int32_t)(row0 + j));
        }
        for (int64_t i = 0; i < n_k[k]; ++i) blk_of_reach.push_back((int32_t)k);
        gl_of_reach.insert(gl_of_reach.end(), gl.begin(), gl.end());
        b->blocks.push_back(blk);
        row0 += n_k[k]; g0 += m_k[k];
    }
    if (row0 != net->topo.n) { delete b; return fail(TXH_E_INVALID, "block sizes do not add up to the union network"); }
    if (b->max_m > txh_kfb_max_gauges()) {
        delete b; return fail(TXH_E_INVALID, "a block has too many gauges for the batched inverse");
    }
    b->n_u = row0; b->m_tot = g0;
    b->ld = (int)txh_row_stride(b->max_n);
    if ((rc = upload(&b->d_blocks, b->blocks)) || (rc = upload(&b->d_blk_of_reach, blk_of_reach)) ||
        (rc = upload(&b->d_gl_of_reach, gl_of_reach)) || (rc = upload(&b->d_obs_reach, obs_reach))) { delete b; return rc; }
    auto dalloc = [](double** p, size_t count) { return cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(double)); };
    cudaError_t e = cudaSuccess;
    for (auto pr : {std::make_pair(&b->d_P, (size_t)b->pp), std::make_pair(&b->d_Pprev, (size_t)b->pp), std::make_pair(&b->d_Q, (size_t)b->pp),
                    std::make_pair(&b->d_Pm, (size_t)b->pp), std::make_pair(&b->d_R, (size_t)b->mm), std::make_pair(&b->d_S, (size_t)b->mm),
                    std::make_pair(&b->d_Ps, (size_t)b->nm), std::make_pair(&b->d_Prow, (size_t)b->nm), std::make_pair(&b->d_K, (size_t)b->nm),
                    std::make_pair(&b->d_z, (size_t)b->m_tot), std::make_pair(&b->d_dz, (size_t)b->m_tot),
                    std::make_pair(&b->d_gain, (size_t)b->n_u), std::make_pair(&b->d_Gp, (size_t)b->n_u * 2),
                    std::make_pair(&b->d_X, (size_t)b->n_u * b->ld), std::make_pair(&b->d_X2, (size_t)b->n_u * b->ld)})
        if (e == cudaSuccess) e = dalloc(pr.first, pr.second);
    if (e != cudaSuccess) { txh_kfb_destroy(b); return cuda_fail(e, "batched filter buffers"); }
    *out = b;
    return TXH_OK;
}

void txh_kfb_destroy(txh_kfb* b)
{
    if (!b) return;
    cudaFree(b->d_blocks); cudaFree(b->d_blk_of_reach); cudaFree(b->d_gl_of_reach); cudaFree(b->d_obs_reach);
    for (double* p : {b->d_P, b->d_Pprev, b->d_Q, b->d_R, b->d_Pm, b->d_Ps, b->d_Prow, b->d_S, b->d_K, b->d_z, b->d_dz, b->d_gain,
                      b->d_Gp, b->d_X, b->d_X2})
        cudaFree(p);
    delete b;
}

// which: 0 P (posterior), 1 Q, 2 R, 3 P of the previous update, 4 K, 5 dz, 6 gain
static int kfb_locate(txh_kfb* b, int64_t block, int which, double** ptr, size_t* count)
{
    if (!b || block < 0 || block >= (int64_t)b->blocks.size()) return fail(TXH_E_INVALID, "bad block");
    const KfbBlock& k = b->blocks[block];
    switch (which) {
        case 0: *ptr = b->d_P + k.p_off; *count = (size_t)k.n * k.n; break;
        case 1: *ptr = b->d_Q + k.p_off; *count = (size_t)k.n * k.n; break;
        case 2: *ptr = b->d_R + k.mm_off; *count = (size_t)k.m * k.m; break;
        case 3: *ptr = b->d_Pprev + k.p_off; *count = (size_t)k.n * k.n; break;
        case 4: *ptr = b->d_K + k.nm_off; *count = (size_t)k.n * k.m; break;
        case 5: *ptr = b->d_dz + k.g_off; *count = (size_t)k.m; break;
        case 6: *ptr = b->d_gain + k.row0; *count = (size_t)k.n; break;
        default: return fail(TXH_E_INVALID, "bad matrix selector");
    }
    return TXH_OK;
}

int txh_kfb_set(txh_kfb* b, int64_t block, int which, const double* host, void* stream)
{
    double* p; size_t c; int rc;
    if (!host) return fail(TXH_E_INVALID, "null argument");
    if ((rc = kfb_locate(b, block, which, &p, &c))) return rc;
    if (which > 2) return fail(TXH_E_INVALID, "only P, Q and R can be set");
    CU(cudaMemcpyAsync(p, host, c * sizeof(double), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return TXH_OK;
}

int txh_kfb_get(txh_kfb* b, int64_t block, int which, double* host, void* stream)
{
    double* p; size_t c; int rc;
    if (!host) return fail(TXH_E_INVALID, "null argument");
    if ((rc = kfb_locate(b, block, which, &p, &c))) return rc;
    CU(cudaMemcpyAsync(host, p, c * sizeof(double), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return TXH_OK;
}

int txh_kfb_filter(txh_kfb* b, const uint8_t* active, const double* z_host, double* O, double* I, void* stream)
{
    if (!b || !active || !z_host || !O || !I) return fail(TXH_E_INVALID, "null argument");
    txh_net* net = b->net;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = ensure_device(net)) || (rc = ensure_coef(net, st))) return rc;
    bool any = false, changed = false;
    for (size_t k = 0; k < b->blocks.size(); ++k) {
        const int32_t a = active[k] ? 1 : 0;
        changed |= a != b->blocks[k].active;
        b->blocks[k].active = a;
        any |= a != 0;
    }
    if (!any) return TXH_OK;
    if (changed) {
        CU(cudaMemcpyAsync(b->d_blocks, b->blocks.data(), b->blocks.size() * sizeof(KfbBlock), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));
    }
    CU(cudaMemcpyAsync(b->d_z, z_host, sizeof(double) * b->m_tot, cudaMemcpyHostToDevice, st));
    // P before this update, for the blocks it updates; a block that is not due keeps the P before its last one
    for (const KfbBlock& k : b->blocks)
        if (k.active)
            CU(cudaMemcpyAsync(b->d_Pprev + k.p_off, b->d_P + k.p_off, sizeof(double) * k.n * k.n,
                               cudaMemcpyDeviceToDevice, st));
    const int n_u = (int)b->n_u, ld = b->ld, M = b->max_n;
    // P- = A (A P)^T + Q for every block at once: the blocks' columns are the members of two routing launches
    CU(launch_kfb_pack(b->d_blocks, b->d_blk_of_reach, net->d_pos_of_reach, b->d_P, b->d_X, n_u, ld, st));
    CU(launch_init_inflows(net->d_up_off, net->d_up_pos, net->d_outlet, b->d_X, b->d_X2, n_u, ld, M, st));
    if ((rc = run_routing(net, b->d_X, b->d_X2, M, nullptr, nullptr, 0, StepPlan(), 1, st))) return rc;
    CU(launch_kfb_transpose(b->d_blocks, b->d_blk_of_reach, net->d_pos_of_reach, b->d_X, b->d_X2, n_u, ld, st));
    CU(launch_init_inflows(net->d_up_off, net->d_up_pos, net->d_outlet, b->d_X2, b->d_X, n_u, ld, M, st));
    if ((rc = run_routing(net, b->d_X2, b->d_X, M, nullptr, nullptr, 0, StepPlan(), 1, st))) return rc;
    CU(launch_kfb_update(b->d_blocks, (int)b->blocks.size(), b->max_m, b->d_blk_of_reach, net->d_pos_of_reach, b->d_gl_of_reach,
                         b->d_obs_reach, b->d_X2, n_u, ld, b->d_Q, b->d_R, b->d_z, O, (int)txh_row_stride(1), b->d_Pm, b->d_Ps,
                         b->d_Prow, b->d_S, b->d_K, b->d_dz, b->d_gain, b->d_Gp, b->d_P, info_word(net), st));
    // da.py:124-126 on the union state (inactive blocks have a zero gain)
    CU(launch_apply_gain(net->d_up_off, net->d_up_pos, b->d_Gp, O, I, n_u, (int)txh_row_stride(1), 1, st));
    return TXH_OK;
}

}  // extern "C"
