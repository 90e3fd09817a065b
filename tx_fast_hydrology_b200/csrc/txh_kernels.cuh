// txh_kernels.cuh -- device-side argument blocks and launcher prototypes (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include <vector>

#include "txh_topology.hpp"

namespace txh {

// The one owner of a device allocation: capacity() elements of T, move-only, freed on destruction.  It converts to
// its pointer, so launch arguments read as they would from a raw one.  An allocation, copy or fill that fails leaves
// it empty (nullptr, capacity 0).  An empty buffer makes no CUDA call, not even when it is destroyed.
template <class T>
class DevBuf {
public:
    DevBuf() = default;
    DevBuf(DevBuf&& o) noexcept : p_(o.p_), cap_(o.cap_) { o.p_ = nullptr; o.cap_ = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept
    {
        if (this != &o) { reset(); p_ = o.p_; cap_ = o.cap_; o.p_ = nullptr; o.cap_ = 0; }
        return *this;
    }
    ~DevBuf() { reset(); }
    operator T*() const { return p_; }
    T* get() const { return p_; }
    size_t capacity() const { return cap_; }
    void reset()
    {
        if (p_) cudaFree(p_);
        p_ = nullptr; cap_ = 0;
    }
    // `count` elements of new, uninitialised memory in place of the old
    cudaError_t alloc(size_t count)
    {
        reset();
        const cudaError_t e = cudaMalloc((void**)&p_, count * sizeof(T));
        if (e != cudaSuccess) { p_ = nullptr; return e; }
        cap_ = count;
        return cudaSuccess;
    }
    // a synchronous copy of `v` (one element when `v` is empty)
    cudaError_t upload(const std::vector<T>& v)
    {
        cudaError_t e = alloc(std::max<size_t>(v.size(), 1));
        if (e == cudaSuccess && !v.empty()) e = cudaMemcpy(p_, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) reset();
        return e;
    }
    // Grow-only: reallocated when `count` elements do not fit, once `st` has drained (a queued launch may still read
    // the old memory); new memory is filled with the byte `fill` unless it is < 0.
    cudaError_t grow(size_t count, cudaStream_t st, int fill = -1)
    {
        if (count <= cap_) return cudaSuccess;
        cudaError_t e = p_ ? cudaStreamSynchronize(st) : cudaSuccess;
        if (e != cudaSuccess) return e;
        e = alloc(count);
        if (e == cudaSuccess && fill >= 0) e = cudaMemsetAsync(p_, fill, count * sizeof(T), st);
        if (e != cudaSuccess) reset();
        return e;
    }

private:
    T* p_ = nullptr;
    size_t cap_ = 0;
};

// Interpolation of the forcing table for one step, resolved on the host exactly as
// nutils.py:21-34 does (searchsorted-left, clamped ends): q = w0*F[r0] + w1*F[r1].
struct StepInterp {
    int32_t r0, r1;
    double w0, w1;
};

// nutils.py:21-34: np.searchsorted(xp, x) (side='left'), clamped ends, linear weights or the nearer row
__device__ __forceinline__ StepInterp interp_step(const double* __restrict__ times, int R, double x, int method)
{
    int lo = 0, hi = R;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (times[mid] < x) lo = mid + 1; else hi = mid;
    }
    StepInterp si;
    if (lo == 0) { si.r0 = 0; si.r1 = 0; si.w0 = 1.0; si.w1 = 0.0; }
    else if (lo >= R) { si.r0 = R - 1; si.r1 = R - 1; si.w0 = 1.0; si.w1 = 0.0; }
    else {
        const double dx_0 = __dsub_rn(x, times[lo - 1]), dx_1 = __dsub_rn(times[lo], x);
        if (method == 1) {
            const double frac = __ddiv_rn(dx_0, __dadd_rn(dx_0, dx_1));
            si.r0 = lo - 1; si.r1 = lo; si.w0 = __dsub_rn(1.0, frac); si.w1 = frac;
        } else {
            const int r = fabs(dx_0) <= fabs(dx_1) ? lo - 1 : lo;
            si.r0 = r; si.r1 = r; si.w0 = 1.0; si.w1 = 0.0;
        }
    }
    return si;
}

// The same record for route_lane_kernel, 32 bytes (two 128-bit loads); bit 31 of r1 is set when the bracket
// (r0, r1) differs from the previous step's, bit 30 when it moved on by exactly one row.
struct LaneStep {
    double w0, w1;
    int32_t r0, r1;
    int32_t pad0, pad1;
};

constexpr int kWarpsPerCta = 4;
constexpr int kMemberBlock = 64;          // members per warp: one double2 per lane
constexpr int kRingBytes = 2 * 12 * 512;  // per-warp row ring: 2 arrays x 12 rows x 512 B (see txh_route.cu)
// every byte of an EMPTY cell of the window and lane kernels' hand-over rings (txh_device.cuh): the fill of a new ring
constexpr int kEmptyByte = 0xff;

// launch bookkeeping of the launchers (txh_launch_count) and their grid sizes
void count_launch();
inline unsigned nblk(long long work, int threads) { return (unsigned)((work + threads - 1) / threads); }

struct RouteArgs {
    const TaskDesc* tasks;
    const int32_t* notify;
    const uint32_t* hdr;
    const uint32_t* inw;
    const double* coef;                   // [n][4] = alpha, beta, chi, gamma (schedule order)
    const double* cumA;                   // [n] prefix product of alpha from the first reach of the segment
    const double* linkA;                  // [link entries] cumA at the last reach of each segment
    double* O;
    double* I;
    double* Side;                         // [n_side][ld] outflows of the pocket roots, in PRE order (scratch)
    const double* F;                      // [R][n] schedule order, or nullptr
    const StepInterp* steps;              // [nsteps]
    const double* Wmul;                   // [R][wm_ld] member multipliers, or nullptr
    const int32_t* rec_slot;              // [n] recording slot of each position or -1; nullptr = off
    double* rec_out;                      // [nrec_steps][rec_count][M]
    long long rec_step_base;              // steps of the call before this launch
    // dataflow runtime state (one entry per (task, member block) pair)
    int32_t* pending;                     // outstanding dependencies of the pair's next step
    unsigned long long* queue;            // ready queue: (step << 32) | (pair + 1), 0 = not yet pushed
    unsigned long long* q_head;           // pop cursor; q_head[1] = push cursor
    int32_t* status;
    unsigned long long watchdog_ns;
    long long total;                      // pairs * nsteps = entries ever pushed
    int64_t n;
    int32_t n_tasks, n_mblocks, nsteps, slots;
    int32_t ld, M, wm_ld, rec_every, rec_count;
    // per-warp shared-memory area (bytes): [scratch slots][coef][f0][f1][hdr][inw][row ring]
    int32_t smem_per_warp, off_coef, off_f0, off_f1, off_hdr, off_inw, off_ring, max_words;
    int32_t off_inw_link, max_words_link; // LINK layout: A_last at off_coef, records at off_inw_link
    unsigned long long* trace;            // optional [total][4] timeline, nullptr = off
};

struct InitArgs {
    const TaskDesc* tasks;
    const int32_t* init_ready;
    int32_t* pending;
    unsigned long long* queue;
    unsigned long long* q_head;
    int32_t n_tasks, n_mblocks, n_init;
    long long queue_entries;              // slots of the ready queue to clear (pairs * steps of this launch)
    // forcing interpolation of this launch's steps, resolved on the device (nullptr times = skip)
    const double* times;                  // [R] float64 ns since epoch
    StepInterp* steps_out;                // [nsteps]
    long long t0_ns, dt_ns, step_base;
    int32_t R, nsteps, method;
};

// route_window_kernel (txh_window.cu)
struct WinArgs {
    const WTaskDesc* tasks;
    const uint32_t* hdr;                  // window headers per position
    const uint32_t* inw;
    const int32_t* prod;
    const double* coef;                   // [n][4]
    const double* cumA;                   // [n] prefix product of alpha along the segment
    const double* cumC;                   // [n] beta_k A_{k-1} + chi_k A_k (see route_window_kernel)
    double* O;
    double* I;
    double* ring;                         // [nsteps][n_slots][ld] rows handed between tasks; EMPTY (all bits set) when idle
    unsigned long long* ticket;           // zero at launch; the last warp to leave the kernel zeroes it again
    unsigned long long* done;             // warps that have left the kernel
    const double* F;                      // [R][n] schedule order, or nullptr
    const StepInterp* steps;              // [nsteps] interpolation records, or nullptr: every warp resolves them itself
    const double* times;                  // ... from the forcing times [R] (steps == nullptr)
    long long t0_ns, dt_ns, step_base;    // step s of the launch ends at t0_ns + (step_base + s + 1) * dt_ns
    int32_t R, method;
    const double* Wmul;                   // [R][wm_ld] or nullptr
    int32_t* status;
    unsigned long long watchdog_ns;
    int64_t n;
    int32_t n_tasks, n_mblocks, nsteps, n_slots, ld, M, wm_ld;
    // per-warp shared memory (bytes): [p rows][scratch slots][input ring][row records][cumA][cumC][words][slot list][mbarrier]
    int32_t smem_per_warp, off_scr, off_in, off_rec, off_cum, off_cumc, off_words, off_list;
    int32_t off_steps;                    // CTA-wide (behind the per-warp areas and T): interpolation records of the launch's steps
    int32_t off_mbar;                     // > 0: per-warp mbarrier for the bulk (TMA) staging of the state rows
    unsigned long long* trace;            // optional [pairs][4 + nsteps] timeline (claim, loaded, end, kind|smid, publish per step)
    double* rowsum;                       // optional [n]: scale * sum over the members of the final outflows (n_mblocks == 1)
    double rowsum_scale;
    // optional: the ensemble update that is still owed to the state (txh_run_assimilating), applied while a task is
    // loaded -- p+ = p + (p - mean(p)) T + gauge terms, see route_window_kernel (n_mblocks == 1)
    const double* upT;                    // [M][M] ensemble transform, nullptr = no update pending
    int32_t off_T;                        // CTA-wide shared-memory copy of T (32 KB, behind the per-warp areas)
    int32_t nap_min, nap_max;             // back-off (ns) of a warp polling for a row another task has not published yet
    const double* upW;                    // [gauges][M]
    const double* upQs;                   // [gauges]
    const int32_t* gfix_off;              // [n_tasks + 1] gauge terms per task
    const int2* gfix;                     // {row in task | kind << 16 (0: the row's own gauge, chi; 1: an upstream gauge, beta), gauge}
    // optional recording (REC variant): the outflow of every recorded row after every rec_every-th step of the call
    const int32_t* rec_slot;              // [n] recording slot of each position or -1; nullptr = off
    double* rec_out;                      // [steps recorded][rec_count][M]
    long long rec_step_base;              // steps of the call before this launch
    int32_t rec_every, rec_count;
    // UPD + REC: the recorded rows of the update this launch applies, [rec_count][M] each (nullptr = not wanted):
    // the forecast (rec_prior) and the posterior o + (o - mean) T + qs W (rec_post); rec_mean = the forecast's row means
    double* rec_prior;
    double* rec_post;
    const double* rec_mean;
};

// route_lane_kernel (txh_lane.cu): lanes = reaches, time-skewed regions, state in shared memory
struct LaneArgs {
    const LaneRegionDesc* regions;        // ticket order
    const int4* meta;                     // per row: {position (-1: virtual), skew offset | further children << 16,
                                          //           first two children c0 | c1 << 16, slot}
    const int32_t* xbeg;                  // per row: first further child (relative to the region's child_off)
    const uint16_t* child;
    const double* coef;                   // [n][4]
    double* O;
    double* I;
    const double* F;                      // [R][n] schedule order, or nullptr
    const LaneStep* steps;                // [nsteps] interpolation records of this launch
    const double* Wmul;                   // [R][wm_ld] or nullptr
    double* ring;                         // [n_slots][M][splp] streams between regions; EMPTY (all bits set) when idle
    unsigned long long* ticket;           // zero at launch; the last CTA to leave zeroes it again
    unsigned long long* done;
    int32_t* status;
    unsigned long long watchdog_ns;
    const int32_t* rec_slot;              // [n] recording slot of each position or -1; nullptr = off
    double* rec_out;                      // [steps recorded][rec_count][M]
    long long rec_step_base;              // steps of the call before this launch
    int64_t n;
    int32_t n_regions, nsteps, splp, ld, M, wm_ld, R, rec_every, rec_count;
    int32_t TR;                           // threads [0, TR) own real rows, the rest the virtual rows
    int32_t off_steps;                    // > 0: the per-step records are staged in shared memory at this offset
    int32_t vote_every;                   // power of two: iterations between barrier votes on abandoning the launch
    int32_t lag;                          // steps a producer region is ahead before its consumer starts / resumes
    unsigned long long* trace;            // optional [n_regions][8]: claim, loaded, last lag wait over, end (ns), iterations,
                                          // SM, slow-path polls, -- ; nullptr = off
};

struct LevelArgs {
    const int32_t* lvl_pos;               // positions of this level
    int32_t count;
    const int32_t* up_off;
    const int32_t* up_pos;
    const double* coef;
    const double* q;                      // [n] schedule order or nullptr
    double* O;
    double* I;
    int32_t ld, M;
};

cudaError_t launch_dataflow_init(const InitArgs& a, cudaStream_t st);
cudaError_t launch_route_dataflow(const RouteArgs& a, int num_sms, cudaStream_t st);
cudaError_t launch_route_level(const LevelArgs& a, cudaStream_t st);
cudaError_t launch_window_init(const InitArgs& a, unsigned long long* ticket, cudaStream_t st);
cudaError_t launch_route_window(const WinArgs& a, int warps_per_cta, int num_sms, cudaStream_t st);
cudaError_t launch_route_lane(const LaneArgs& a, int mt, int threads, size_t smem, int grid, cudaStream_t st);
cudaError_t lane_occupancy(int mt, bool f, bool w, int threads, size_t smem, int* per_sm);
cudaError_t launch_lane_init(const InitArgs& a, LaneStep* out, unsigned long long* ticket, cudaStream_t st);
cudaError_t launch_init_inflows(const int32_t* up_off, const int32_t* up_pos, const uint8_t* is_outlet,
                                const double* O, double* I, int64_t n, int ld, int M, cudaStream_t st);
cudaError_t launch_apply_gain(const int32_t* up_off, const int32_t* up_pos, const double* G, double* O,
                              double* I, int64_t n, int ld, int M, cudaStream_t st);
// dst[pos][m] = src[reach_of_pos[pos]][m]   (src [n][M] dense, dst [n][ld])
cudaError_t launch_pack(const int32_t* reach_of_pos, const double* src, double* dst, int64_t n, int M,
                        int ld, int src_member_major, cudaStream_t st);
cudaError_t launch_unpack(const int32_t* reach_of_pos, const double* src, double* dst, int64_t n, int M,
                          int ld, int dst_member_major, cudaStream_t st);
cudaError_t launch_gather_rows(const int32_t* pos, int64_t count, const double* X, int ld, int M,
                               double* out, cudaStream_t st);
cudaError_t launch_permute_rows(const int32_t* reach_of_pos, const double* src, double* dst, int64_t n, int64_t R,
                                cudaStream_t st);
// vector permute: dst[pos] = src[reach_of_pos[pos]]
cudaError_t launch_permute_vec(const int32_t* reach_of_pos, const double* src, double* dst, int64_t n,
                               cudaStream_t st);

int64_t launch_count();

// ---- assimilation (txh_da.cu) --------------------------------------------------------------------
cudaError_t launch_dgemm(int transA, int transB, int M, int N, int K, double alpha, const double* A, int lda,
                         const double* B, int ldb, double beta, double* C, int ldc, cudaStream_t st);
cudaError_t launch_dgemm_splitk(int transA, int transB, int M, int N, int K, const double* A, int lda, const double* B,
                                int ldb, double* Cpart, int ldc, int nsplit, long long pstride, cudaStream_t st);
// A gauge whose observation row holds a NaN is missing at that update (txh_da.cu: gauge_row_missing).  The solve
// leaves it out with a diagonal D; with a dense one it writes this value to the info word instead, which txh_check
// reports.  It lies outside the pivots the other solves write there (1..m Cholesky, -1..-m Gauss-Jordan).
constexpr int kInfoMissingObs = -0x7fffffff - 1;
// O != nullptr: HX is gathered from the gauge rows of O on the way (and written out)
cudaError_t launch_innovation_cat(double* HX, const double* O, int ldo, const double* Zp, const double* mean,
                                  const int32_t* obs_pos, const double* dinv_diag, int m, int Mt, double* Bc, double* Y,
                                  int* info, cudaStream_t st);
cudaError_t launch_chol_solve_small(const double* Cpart, int nsplit, long long pstride, int Mt, double shift, double* Z,
                                    int* info, cudaStream_t st);
cudaError_t launch_enkf_small_system(double* HX, const double* O, int ldo, const double* Zp, const double* mean,
                                     const int32_t* obs_pos, const double* dinv_diag, int m, int Mt, double shift,
                                     double* T, double* W, int* info, cudaStream_t st);
cudaError_t launch_dgemm_ex(int transA, int transB, int M, int N, int K, double alpha, const double* A, int lda,
                            const double* B, int ldb, double beta, const double* Cin, int ldcin, double* C, int ldc,
                            cudaStream_t st);
cudaError_t launch_woodbury_assemble(const double* Cpart, int nsplit, long long pstride, int Mt, double shift, double* Cf,
                                     double* C1, cudaStream_t st);
cudaError_t launch_enkf_stats(const double* X, int ld, int M, int64_t n, double scale, const int32_t* gauge_of_pos,
                              double* rowsum, double* HX, cudaStream_t st);
// diag_R: R (and D) diagonal, a missing gauge gets zero rows of HA and dz; otherwise it is reported through *info
cudaError_t launch_innovation(const double* HX, const double* Zp, const double* mean_obs, int m, int M, bool diag_R,
                              double* HA, double* dz, int* info, cudaStream_t st);
cudaError_t launch_innov_cov_finish(double* S, const double* qs, const double* R, int m, double scale, cudaStream_t st);
cudaError_t launch_spd_solve(double* S, double* B, int m, int k, int* info, cudaStream_t st);
cudaError_t launch_inverse(double* A, double* W, int m, int* info, cudaStream_t st);
// State matrices of the shards of a member-sharded ensemble, read in place (peer GPUs mapped over NVLink)
constexpr int kMaxPeers = 16;
struct PeerBlocks {
    const double* p[kMaxPeers];
    int count;
};
cudaError_t launch_enkf_update(const double* Xall, int ldx, int Mtot, const double* mean, const double* T, int ldt,
                               int Mloc, double* O, double* G, int ld, int64_t n, const int32_t* gauge_of_pos,
                               const double* qs, const double* W, int col0, int num_sms, int Mb, long long blk_stride,
                               cudaStream_t st, const PeerBlocks* peers = nullptr, double* Oout = nullptr);
cudaError_t launch_inflow_rebuild(const int4* rec, int64_t n_inner, const int32_t* up_off, const int32_t* up_pos,
                                  const double* O, double* I, int ld, cudaStream_t st);
// prior_out[k][:] = O[rec_pos[k]][:] (forecast), post_out[k][:] = the same row after the update of (T, W) (da.py:124-126);
// either may be nullptr.  Launched between the ensemble-space system and the next routing launch (PDL chain).
cudaError_t launch_enkf_record(const double* O, int ld, int M, const double* mean, const double* T,
                               const int32_t* gauge_of_pos, const double* qs, const double* W, const int32_t* rec_pos,
                               int rec_count, double* prior_out, double* post_out, cudaStream_t st);
// The square-root (kind 1, ETKF, Mt <= 64) or relaxed (kind 0, rtpp > 0) form of a solved (T, W), in place; an ETKF
// eigensolve that does not converge writes kInfoEtkfNoConvergence to *info
constexpr int kInfoEtkfNoConvergence = -0x7fffffff;
cudaError_t launch_enkf_transform_post(double* T, double* W, int Mt, int m, int kind, double rtpp, int* info,
                                       cudaStream_t st);
// txh_enks_smooth (arguments checked by the caller): cumulative transforms, then one pass over rec
cudaError_t launch_enks_smooth(int M, int nupd, long long every, const double* T_hist, long long nslots, long long rec_count,
                               long long rec_every, long long lag, const double* rec, double* out, double* work,
                               cudaStream_t st);
cudaError_t launch_inflow_gain(const int32_t* inner, int64_t n_inner, const int32_t* up_off, const int32_t* up_pos,
                               const double* G, double* I, int ld, cudaStream_t st);

// ---- batched dense filters of a generation of sub-models (txh_kf.cu) ------------------------------
struct KfbBlock {
    int32_t n, m;             // reaches / gauges of the sub-model
    int32_t row0;             // first reach of the block in the union network
    int32_t g_off;            // first gauge of the block in the concatenated gauge arrays
    int32_t active;           // 0: this filter is not due, leave its block alone
    int32_t pad_;
    long long p_off;          // offsets (doubles) of the block in the packed [n][n], [n][m] / [m][n], [m][m] buffers
    long long nm_off, mm_off;
};
cudaError_t launch_kfb_pack(const KfbBlock* blocks, const int32_t* blk_of_reach, const int32_t* pos_of_reach, const double* P,
                            double* X, int n_u, int ld, cudaStream_t st);
cudaError_t launch_kfb_transpose(const KfbBlock* blocks, const int32_t* blk_of_reach, const int32_t* pos_of_reach,
                                 const double* X, double* X2, int n_u, int ld, cudaStream_t st);
cudaError_t launch_kfb_update(const KfbBlock* blocks, int nblocks, int max_m, const int32_t* blk_of_reach,
                              const int32_t* pos_of_reach, const int32_t* gl_of_reach, const int32_t* obs_reach,
                              const double* X2, int n_u, int ld, const double* Q, const double* R, const double* z,
                              const double* O, int ldo, double* Pm, double* Ps, double* Prow, double* S, double* K, double* dz,
                              double* gain, double* Gp, double* P, int* info, cudaStream_t st);

// ---- dense per-sub-basin filter glue (txh_kf.cu) ---------------------------------------------------
cudaError_t launch_kf_repack_transposed(const int32_t* reach_of_pos, const int32_t* pos_of_reach, const double* X,
                                        double* X2, int n, int ld, cudaStream_t st);
cudaError_t launch_kf_prior_finish(const int32_t* reach_of_pos, const int32_t* pos_of_reach, const int32_t* gauge_of_pos,
                                   const double* X2, int ld, const double* Q, const double* R, int n, int m, double* Pm,
                                   double* Ps, double* Prow, double* S, cudaStream_t st);
cudaError_t launch_kf_gain(const int32_t* reach_of_pos, const int32_t* obs_pos, const double* z, const double* O, int ldo,
                           const double* K, int n, int m, double* dz, double* gain, double* Gp, cudaStream_t st);

}  // namespace txh
