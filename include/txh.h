/*
 * txh.h -- C ABI of libtxh, the B200 (sm_100a) routing + assimilation hot path
 * that replaces the numba/scipy kernels of future-water/tx-fast-hydrology.
 *
 * The reference has no FFI layer; its boundary is a handful of free functions
 * imported by name from tx_fast_hydrology/nutils.py plus the attribute protocol of
 * the `Muskingum` object (SURVEY.md section 8b).  Each entry point below names the
 * reference interface it replaces (file:line relative to the reference root).
 * The ctypes binding a maintainer would add is shown in INTEGRATION.md and is what
 * tx_fast_hydrology_b200/_lib.py does.
 *
 * Conventions
 *   - every function returns 0 on success, a negative TXH_E_* code on failure;
 *     txh_last_error() returns the message of the calling thread's last failure.
 *   - no exceptions cross the boundary; plain pointers and sizes only.
 *   - `host` pointers are ordinary process memory; `dev` pointers are CUDA device
 *     memory owned by the caller (e.g. torch tensors' data_ptr()).
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Launches
 *     are asynchronous unless stated; a handle is not thread-safe, distinct handles are.
 *   - member-batched state is stored in "schedule order": a row per reach, rows
 *     permuted into task order (see DESIGN.md), `ld` doubles per row with the
 *     ensemble members contiguous: X[pos * ld + member].  txh_row_stride(M) gives
 *     ld; txh_pack_* / txh_unpack_* convert from and to the reference's reach order.
 */
#ifndef TXH_H
#define TXH_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TXH_OK             0
#define TXH_E_INVALID     -1   /* bad argument */
#define TXH_E_TOPOLOGY    -2   /* cycle / out-of-range endnodes */
#define TXH_E_CUDA        -3   /* CUDA runtime error */
#define TXH_E_NODEVICE    -4   /* no CUDA device: the product path has no CPU fallback */
#define TXH_E_WATCHDOG    -5   /* a dataflow wait exceeded its bound (kernel bailed out) */
#define TXH_E_STATE       -6   /* call order (e.g. coefficients not set) */

typedef struct txh_net txh_net;           /* topology + schedule + device descriptors */
typedef struct txh_forcing txh_forcing;   /* lateral-inflow table resident in HBM */

const char* txh_last_error(void);
int txh_version(void);
/* number of visible CUDA devices (0 on a CPU-only box; never fails) */
int txh_device_count(void);

/* ---- topology pass ---------------------------------------------------------------
 * Replaces Muskingum.compute_indegree (muskingum.py:322-330), the per-step headwater
 * mask (muskingum.py:444) and the implicit ordering of the walk in nutils.py:72-88.
 * Host-only, exact integers; works without a GPU.  `endnodes[j]` is the downstream
 * reach of j, an outlet is endnodes[j] == j (muskingum.py:897-902); startnodes is
 * arange(n) as the reference kernels assume (nutils.py:73-83).
 * sched_params = {long_path_min, spine_cap, pocket_cap, max_slots, link_cap}, NULL = defaults. */
int txh_create(int64_t n, const int64_t* endnodes, const int32_t* sched_params, txh_net** out);
void txh_destroy(txh_net* net);
int64_t txh_n(const txh_net* net);
int txh_get_indegree(const txh_net* net, int64_t* indegree /*[n]*/);
int txh_get_headwaters(const txh_net* net, int64_t* heads /*[n]*/, int64_t* count);
int txh_get_levels(const txh_net* net, int64_t* level /*[n]*/, int64_t* nlevels);
int txh_get_level_order(const txh_net* net, int64_t* order /*[n]*/, int64_t* offsets /*[nlevels+1]*/);
int txh_get_chains(const txh_net* net, int64_t* chain_id /*[n]*/, int64_t* chain_pos /*[n]*/,
                   int64_t* chain_len /*[n] (first nchains used)*/, int64_t* nchains);
int txh_get_paths(const txh_net* net, int64_t* path_id /*[n]*/, int64_t* path_pos /*[n]*/);
int txh_get_visit_order(const txh_net* net, int64_t* order /*[n]*/);      /* nutils.py:72-88 */
/* schedule introspection (tests, tuning).  info = {n_tasks, n_spine_segments, n_pocket_tasks,
 * n_input_words, n_notify, slots_used, row_fallbacks, cp_tasks, cp_cost, nlevels}.
 * task_desc rows are 12 int32: begin, len, in_off, nfy_off, n_same, n_next, need0, need, kind, pad x3 */
int txh_get_schedule_info(const txh_net* net, int64_t info[10]);
int txh_get_schedule(const txh_net* net, int64_t* pos_of_reach /*[n]*/, int32_t* task_desc /*[n_tasks*12]*/,
                     int32_t* notify, uint32_t* hdr /*[n]*/, uint32_t* inw);

/* window-mode schedule (route_window_kernel): info = {n_tasks, n_slots, max_len, max_words, max_producers,
 * n_input_words, n_producer_entries, cp_tasks}; task rows are 12 int32: begin, len, kind, in_off, n_words,
 * prod_off, n_prod, out_slot, n_in, pad x3 */
int txh_get_window_info(const txh_net* net, int64_t info[8]);
int txh_get_window_schedule(const txh_net* net, int32_t* wtask_desc, uint32_t* whdr /*[n]*/, uint32_t* winw,
                            int32_t* wprod);

/* lane schedule (route_lane_kernel, ensembles of up to 16 members: lanes are reaches, regions of the network run
 * time-skewed in shared memory).  Host only.  cap_rows > 0 overrides the rows per region for schedules not yet
 * in use.  info = {n_regions, n_row_entries, n_child_entries, n_slots, max_real, max_virt, max_extra, member_tile};
 * regions rows are 8 int32: row_off, n_real, n_virt, child_off, n_child, n_extra, height, pad; rows are 6 int32
 * per entry: reach (-1: virtual row), skew offset, the first two children c0 | c1 << 16 (region-local rows; a
 * missing child is the region's zero row, n_real + n_virt), number of further children, their first entry in
 * `child` (relative to the region's child_off), slot (real: stream published, virtual: stream mirrored; -1
 * none); child: region-local rows.
 * Replaces the implicit ordering of the reference's headwater walk (nutils.py:72-88) for M <= 16. */
int txh_get_lane_info(txh_net* net, int64_t M, int64_t cap_rows, int64_t info[8]);
int txh_get_lane_schedule(txh_net* net, int64_t M, int32_t* regions, int32_t* rows, int32_t* child);

/* NHD flowline GeoJSON -> network arrays in ONE native pass over the file: replaces the per-feature Python loops of
 * load_nhd_geojson (muskingum.py:877-917).  comid[i], shape_length[i] ("Shape_Length") and endnodes[i] = index of the
 * feature whose COMID equals feature i's toCOMID, or i itself when there is none (outlet = self-loop,
 * muskingum.py:897-902).  Geometry is skipped.  Host only.  Call with capacity = 0 to get `count`, then with arrays of
 * that size. */
int txh_scan_nhd_geojson(const char* path, int64_t capacity, int64_t* comid /*[capacity]*/, int64_t* endnodes,
                         double* shape_length, int64_t* count);

/* ---- coefficients ----------------------------------------------------------------
 * txh_compute_coeffs replaces Muskingum.compute_muskingum_coeffs (muskingum.py:332-360):
 * host arithmetic in the reference's operation order; results returned in reach order
 * and installed on the handle.  txh_set_coeffs installs user-mutated arrays
 * (Muskingum.set_transmissive_boundary, muskingum.py:567-571). */
int txh_compute_coeffs(txh_net* net, const double* K, const double* X, double dt,
                       double* alpha, double* beta, double* chi, double* gamma /* host [n], may be NULL */);
int txh_set_coeffs(txh_net* net, const double* alpha, const double* beta, const double* chi,
                   const double* gamma /* host [n] */);

/* ---- layout ------------------------------------------------------------------------ */
int64_t txh_row_stride(int64_t M);                       /* doubles per row for M members */
/* host reach-order -> device schedule-order.  layout 0: src[reach*M + m]; 1: src[m*n + reach] */
int txh_pack_host(txh_net* net, const double* src_host, int64_t M, int layout, double* dst_dev, void* stream);
int txh_unpack_host(txh_net* net, const double* src_dev, int64_t M, int layout, double* dst_host, void* stream);
/* device reach-order [n][M] <-> device schedule-order */
int txh_pack_dev(txh_net* net, const double* src_dev, int64_t M, double* dst_dev, void* stream);
int txh_unpack_dev(txh_net* net, const double* src_dev, int64_t M, double* dst_dev, void* stream);
/* gather rows of the listed reaches: out[k*M + m] = X[pos(reach_idx[k])*ld + m]  (device out) */
int txh_gather_rows(txh_net* net, const double* X_dev, int64_t M, const int64_t* reach_idx_host,
                    int64_t count, double* out_dev, void* stream);

/* ---- state initialisation ------------------------------------------------------------
 * Muskingum.init_states (muskingum.py:410-419) and numba_init_inflows (nutils.py:136-141):
 * I[j] = sum of upstream O, PLUS the reach's own O at self-loop outlets (no guard there). */
int txh_init_inflows(txh_net* net, const double* O_dev, double* I_dev, int64_t M, void* stream);

/* ---- forcing table -------------------------------------------------------------------
 * The (T x n) lateral-inflow table `simulate` interpolates every step
 * (muskingum.py:526-531 -> nutils.interpolate_sample, nutils.py:5-39), uploaded once.
 * times: float64 ns since epoch (index.astype(int).astype(float)); table: host [R][n] in
 * reach order (pinned memory makes the upload asynchronous; the call returns after it completed).
 * member_mul (optional, host [R][M]): member m sees table[r][j]*member_mul[r][m]. */
int txh_forcing_create(txh_net* net, int64_t R, const double* times, const double* table_host,
                       int64_t M, const double* member_mul_host, void* stream, txh_forcing** out);
/* new values for an existing table of the same shape (a new forecast cycle): no allocation, one H2D copy */
int txh_forcing_update(txh_forcing* f, const double* times, const double* table_host, const double* member_mul_host,
                       void* stream);
/* The same without waiting for the copy: the table (PINNED host memory, untouched until txh_forcing_wait or the
 * end of the run that reads it) arrives in row chunks on a copy stream owned by the handle, and every later
 * txh_route_run / txh_run_assimilating makes its stream wait only for the chunks its steps interpolate in -- the
 * upload overlaps the routing of the earlier hours. */
int txh_forcing_update_async(txh_forcing* f, const double* times, const double* table_host,
                             const double* member_mul_host, void* stream);
int txh_forcing_wait(txh_forcing* f);
void txh_forcing_destroy(txh_forcing* f);

/* ---- routing ---------------------------------------------------------------------------
 * txh_route_run: `nsteps` timesteps of _ax_bu (nutils.py:64-89) as called from the simulate
 * loop (muskingum.py:527-533), forcing interpolated at t0 + (s+1)*dt for step s exactly as
 * nutils.py:21-34 does (searchsorted-left, clamped ends, linear; times are integer ns as
 * Timestamp.value is, muskingum.py:528-530).  One persistent dataflow
 * kernel; O/I are updated in place ([n rows][ld], schedule order).
 *   method: 1 linear, 0 nearest.   forcing == NULL: zero lateral inflow.
 *   rec_*: optional recording of the outflow of `rec_count` reaches after every
 *   `rec_every`-th step into rec_out_dev[(step/rec_every)][k][M] (device). */
int txh_route_run(txh_net* net, double* O_dev, double* I_dev, int64_t M,
                  const txh_forcing* forcing, int64_t t0_ns, int64_t dt_ns, int64_t nsteps, int method,
                  const int64_t* rec_reach_host, int64_t rec_count, int64_t rec_every,
                  double* rec_out_dev, void* stream);
/* one step with an explicit lateral-inflow vector (Muskingum.step, muskingum.py:467-483):
 * q_dev is [n] in REACH order on the device (shared by all members), or NULL. */
int txh_route_step(txh_net* net, double* O_dev, double* I_dev, int64_t M, const double* q_dev, void* stream);
/* the same step evaluated level by level (one launch per topological level); the
 * level-scheduled triangular solve kept as a second, independent device path. */
int txh_route_step_levels(txh_net* net, double* O_dev, double* I_dev, int64_t M, const double* q_dev, void* stream);
/* X <- A.X for every column: numba_init_inflows + _ax (nutils.py:143-169, `_ap_par`);
 * I_scratch_dev is a caller buffer of the same shape as X. */
int txh_route_apply(txh_net* net, double* X_dev, double* I_scratch_dev, int64_t M, void* stream);
/* _apply_gain (nutils.py:116-134) + the in-place update of da.py:124-126:
 * O += G ; I[j] += sum_{u->j, u!=j} G[u]   (G in schedule order, same shape) */
int txh_apply_gain(txh_net* net, const double* G_dev, double* O_dev, double* I_dev, int64_t M, void* stream);

/* ---- assimilation ------------------------------------------------------------------------
 * Ensemble form of KalmanFilter.filter (da.py:91-136) with P := sample covariance of the forecast
 * ensemble + diagonal Q (the reference has no ensemble filter; SURVEY.md section 8c):
 *   dz = Zp - O[s]                       (da.py:112, per member, Zp = perturbed observations)
 *   S  = HA HA^T/(Mtot-1) + Q[s,s] + R   (da.py:117-119: P[s][:,s] + R_cov)
 *   W  = S^-1 dz ;  T = HA^T W/(Mtot-1)
 *   gain = A T + Q[:,s] W                (da.py:119-121: K dz with K = P[:,s] S^-1)
 *   O += gain ; I += N gain              (da.py:124-126: _apply_gain)
 * A = O - mean are the anomalies, HA their gauge rows.  Three phases so that a member-sharded run
 * can combine the statistics between them (all-reduce of the row sums, all-gather of HX / X):
 *   txh_enkf_stats : local row sums at every reach + this shard's gauge rows (one pass over the state)
 *   txh_enkf_solve : innovation covariance (FP64 tensor cores), Cholesky solve, transform
 *   txh_enkf_apply : gain = A T on the FP64 tensor cores + gauge-row term, then the in-place update
 * obs_reach: gauged reach indices ascending (da.py:33-44); all matrices row-major on the device. */
int txh_enkf_stats(txh_net* net, const double* O_dev, int64_t Mloc, const int64_t* obs_reach_host, int64_t m,
                   double scale /* rowsum = scale * sum; 1/Mtot gives the mean of an unsharded ensemble */,
                   double* rowsum_dev /*[n] schedule order*/, double* HX_dev /*[m][Mloc]*/, void* stream);
/* Every later routing call on the handle also leaves rowsum[pos] = scale * (sum over the members of the final
 * outflow of the reach at schedule position pos) in rowsum_dev [n] -- the first half of txh_enkf_stats, fused
 * into the last step of the launch.  NULL switches it off.  txh_enkf_stats with rowsum_dev == NULL then only
 * gathers the gauge rows. */
int txh_set_stats_output(txh_net* net, double* rowsum_dev, double scale);
/* doubles of workspace txh_enkf_solve needs */
int64_t txh_enkf_work_size(int64_t m, int64_t Mtot);
/* Dinv (optional): the inverse of D = R + diag(qs), which is constant between updates -- dinv_kind 1: its
 * diagonal [m] (R diagonal), 2: dense [m][m], 0: not supplied.  When it is supplied and Mtot < m the m x m
 * solve collapses to an Mtot x Mtot one in ensemble space (Sherman-Morrison-Woodbury; txh_da.cu). */
int txh_enkf_solve(txh_net* net, int64_t m, int64_t Mtot, const double* HX_dev /*[m][Mtot]*/,
                   const double* Zp_dev /*[m][Mtot]*/, const double* mean_dev /*[n] schedule order*/,
                   const int64_t* obs_reach_host, const double* qs_dev /*[m] diag(Q) at the gauges*/,
                   const double* R_dev /*[m][m]*/, const double* Dinv_dev, int dinv_kind,
                   double* work_dev /* txh_enkf_work_size(m, Mtot) doubles */,
                   double* W_dev /*[m][Mtot] out*/, double* T_dev /*[Mtot][Mtot] out*/, void* stream);
int txh_enkf_apply(txh_net* net, double* O_dev, double* I_dev, int64_t Mloc, const double* Xall_dev /* [n][ldx] gathered
                   ensemble in schedule order, or NULL to use O_dev (Mtot == Mloc) */, int64_t ldx,
                   int64_t x_block_stride /* 0: one [n][ldx] matrix; else Xall is Mtot/Mloc blocks of [n][ldx], this
                   many doubles apart, block b = the state rows of shard b (an all-gather of O_dev) */, int64_t Mtot,
                   int64_t col0 /* first global member of this shard */, const double* mean_dev, const double* T_dev,
                   const int64_t* obs_reach_host, int64_t m, const double* qs_dev, const double* W_dev,
                   double* G_dev /* scratch, same shape as O_dev */, void* stream);

/* txh_enkf_apply for a member-sharded ensemble whose shards are read IN PLACE: shard_ptrs[b] (host array of `world`
 * device pointers) is the state matrix [n][row_stride(Mloc)] of shard b -- this GPU's own (== O_in for b = rank) or a
 * peer GPU's buffer mapped into this process (CUDA IPC / symmetric memory over NVLink).  The transform kernel loads
 * the peers' rows tile by tile while it multiplies (no all-gather in front of it) and writes the posterior of this
 * shard to O_out, a different buffer than O_in: peers may still be reading O_in.  The caller orders the launches
 * across GPUs (every shard's forecast complete before any transform starts, e.g. by the all-reduce of the row sums)
 * and alternates the two buffers.  nutils.py:157-169 shards the same loop over columns with prange. */
int txh_enkf_apply_peers(txh_net* net, const double* O_in_dev, double* O_out_dev, double* I_dev, int64_t Mloc,
                         const double* const* shard_ptrs_host, int64_t world, int64_t Mtot, int64_t col0,
                         const double* mean_dev, const double* T_dev, const int64_t* obs_reach_host, int64_t m,
                         const double* qs_dev, const double* W_dev, double* G_dev, void* stream);

/* The whole assimilating run of an unsharded ensemble in one call: `every` routing steps per launch (the row
 * sums ride on its last step), then one ensemble update with Zp_dev[k] ([m][M], the k-th update's per-member
 * observations), nsteps / every times, then the remaining steps -- the loop of simulate + a filter callback
 * gated to every `every`-th step (muskingum.py:527-536, da.py:56-61), with the host out of it.
 * time_every > 0: every time_every-th routing launch is bracketed by CUDA events on `stream` (kept over
 * calls, at most 4096); txh_get_route_timings synchronises them, returns their durations (ms) and, when
 * `capacity` covers them all, releases them (capacity 0: just count). */
int txh_run_assimilating(txh_net* net, double* O_dev, double* I_dev, int64_t M, const txh_forcing* forcing,
                         int64_t t0_ns, int64_t dt_ns, int64_t nsteps, int64_t every, int method,
                         const int64_t* obs_reach_host, int64_t m, const double* Zp_dev /*[nsteps/every][m][M]*/,
                         const double* qs_dev, const double* R_dev, const double* Dinv_dev, int dinv_kind,
                         double* rowsum_dev /*[n]*/, double* HX_dev /*[m][M]*/, double* work_dev, double* W_dev,
                         double* T_dev, double* G_dev, int64_t time_every,
                         void* obs_ready_event /* cudaEvent_t or NULL: Zp_dev is complete once it has fired (an upload
                         on another stream); only the first update waits for it */, void* stream);
/* txh_run_assimilating, also recording ensemble hydrographs at `rec_count` reaches (reference order, distinct):
 *   rec_out_dev[s / rec_every - 1][k][M] after every step s (1-based over the call) with s % rec_every == 0 holds
 *   what the state holds after that step: the forecast, or the posterior (o + gain) at an update step;
 *   prior_out_dev (NULL: not wanted) [nsteps / every][k][M] holds the forecast the j-th update started from.
 * rec_count == 0 is txh_run_assimilating.  TXH_E_INVALID before any device work for a reach out of range or listed
 * twice, rec_every < 1, or rec_count > 0 without rec_reach_host / rec_out_dev. */
int txh_run_assimilating_rec(txh_net* net, double* O_dev, double* I_dev, int64_t M, const txh_forcing* forcing,
                             int64_t t0_ns, int64_t dt_ns, int64_t nsteps, int64_t every, int method,
                             const int64_t* obs_reach_host, int64_t m, const double* Zp_dev, const double* qs_dev,
                             const double* R_dev, const double* Dinv_dev, int dinv_kind, double* rowsum_dev,
                             double* HX_dev, double* work_dev, double* W_dev, double* T_dev, double* G_dev,
                             int64_t time_every, void* obs_ready_event, const int64_t* rec_reach_host, int64_t rec_count,
                             int64_t rec_every, double* rec_out_dev, double* prior_out_dev, void* stream);
int txh_get_route_timings(txh_net* net, double* ms_out, int64_t capacity, int64_t* count);
/* While set, update k (0-based) of every txh_run_assimilating(_rec) call on the handle solves its ensemble transform
 * into T_hist_dev + k*M*M ([M][M] row-major) instead of into T_dev, and every consumer of that update reads it there:
 * the transforms of a call survive it (txh_enks_smooth).  A call whose (nsteps / every) * M * M exceeds
 * capacity_doubles fails with TXH_E_INVALID before any device work.  NULL switches it off. */
int txh_set_transform_history(txh_net* net, double* T_hist_dev, int64_t capacity_doubles);

/* ---- ensemble Kalman smoother of recorded hydrographs ----------------------------------------------------------------
 * Fixed-lag EnKS of the slots txh_run_assimilating_rec recorded, from the transforms it kept (txh_set_transform_history):
 * update u (0-based) happened after step (u+1)*every with transform T_u = T_hist_dev + u*M*M; slot j of rec_dev
 * ([nslots][rec_count][M]) holds the ensemble X_j after step s_j = (j+1)*rec_every.  Every update with
 * s_j < (u+1)*every <= s_j + lag is applied to the slot, in increasing u:
 *     X_j <- X_j + (X_j - mean over the members of X_j) T_u
 * which is the EnKS gain A_j HA^T S^-1 dz/(M-1) of the update's innovation solve (the Q[:,s] W term of the filter gain
 * is not: model noise added at the update is uncorrelated with earlier states).  Result in out_dev, the same shape as
 * rec_dev and a buffer of its own (rec_dev is left alone).  lag = 0 or a slot no later update reaches: a copy.
 * TXH_E_INVALID before any device work for M < 2, nupd < 0, every, rec_every < 1, lag < 0, a null buffer or out
 * overlapping rec; TXH_E_NODEVICE without a device.  Asynchronous. */
int64_t txh_enks_work_size(int64_t M, int64_t nupd);           /* doubles of work_dev */
int txh_enks_smooth(int64_t M, int64_t nupd, int64_t every, const double* T_hist_dev, int64_t nslots, int64_t rec_count,
                    int64_t rec_every, int64_t lag, const double* rec_dev, double* out_dev, double* work_dev, void* stream);

/* Dense products of KalmanFilter.filter for small n (da.py:115-122): C = alpha op(A) op(B) + beta C,
 * row-major FP64 on the tensor cores (mma.sync m8n8k4 = DMMA).  With K = 0, A and B are not read and may be null. */
int txh_dgemm(int transA, int transB, int64_t M, int64_t N, int64_t K, double alpha, const double* A_dev,
              int64_t lda, const double* B_dev, int64_t ldb, double beta, double* C_dev, int64_t ldc, void* stream);
/* In-place Cholesky solve S X = B for SPD S [m][m] (destroyed), B [m][k] -> X.  Synchronous;
 * returns TXH_E_INVALID if S is not positive definite. */
int txh_spd_solve(int64_t m, int64_t k, double* S_dev, double* B_dev, void* stream);
/* A <- inv(A) by Gauss-Jordan with partial pivoting (np.linalg.inv, da.py:119); work [m][m]. Synchronous. */
int txh_inverse(int64_t m, double* A_dev, double* work_dev, void* stream);

/* ---- dense Kalman filter of a single-member model: KalmanFilter.filter, da.py:91-136 ------------
 * One update as a chain of launches with no host round trip (the measurement vector is the only host input):
 *   P- = A P A^T + Q  (_aqat_par, nutils.py:194-214: the columns of P ride as members of two routing
 *   launches), K = P-[:, s] inv(P-[s][:, s] + R), gain = K (z - o[s]), P+ = P- - K P-[s], then
 *   o += gain and i += sum of upstream gains (_apply_gain, nutils.py:116-134) in place on the state rows.
 * P_in [n][n] (posterior of the previous update), P_out [n][n] (may alias P_in), P_prior nullable [n][n],
 * Q [n][n], R [m][m] in ascending gauge order (da.py:36-44), all device, row-major, reach order.
 * obs_host [m] ascending reach indices, z_host [m].  O, I: state rows of the model (M = 1).
 * K [n][m], gain [n] (reach order), dz [m]: device outputs.  work: txh_kf_work_size(net, m) doubles.
 * Asynchronous; a singular innovation covariance is reported by txh_check. */
int64_t txh_kf_work_size(const txh_net* net, int64_t m);
int txh_kf_filter(txh_net* net, const double* P_in, double* P_out, double* P_prior, const double* Q_dev,
                  const double* R_dev, const int64_t* obs_host, int64_t m, const double* z_host, double* O,
                  double* I, double* K_dev, double* gain_dev, double* dz_dev, double* work_dev, void* stream);

/* ---- batched dense Kalman filters: ONE chain of launches for the filters of a whole generation of sub-models --------
 * app/app.py:130-141 binds one KalmanFilter per sub-model of a split network and da.py:91-136 fires for each of them
 * after every step.  The sub-models are disjoint forests: `union_net` is the network of all their reaches, block after
 * block (block k: reaches [sum n_0..n_{k-1}, + n_k), local downstream links shifted accordingly).  The columns of every
 * covariance block ride as members of the SAME two routing launches (_aqat_par, nutils.py:194-214), the m_k x m_k
 * inverses run one CTA per block, and the gains correct the union state in place (_apply_gain, nutils.py:116-134).
 * obs_local: the gauge reaches of every block, LOCAL indices, ascending per block, concatenated (da.py:36-44 order).
 * which (txh_kfb_set / _get): 0 P (posterior), 1 Q, 2 R -- settable -- 3 P before the last update, 4 K [n][m], 5 dz [m],
 * 6 gain [n]; matrices row-major in the block's local reach / gauge order.
 * txh_kfb_filter: active[k] = 0 leaves block k alone (its filter is not due, da.py:49-61); z_host: the measurement
 * vectors of all blocks concatenated; O, I: state rows of the UNION model (M = 1).  Asynchronous after its copies.
 * A block that is not due keeps P, P before its last update, K, dz and gain.
 * txh_kfb_max_gauges: the most gauges a block may have (its inverse runs in shared memory); txh_kfb_create refuses more. */
typedef struct txh_kfb txh_kfb;
int64_t txh_kfb_max_gauges(void);
int txh_kfb_create(txh_net* union_net, int64_t nblocks, const int64_t* n_k, const int64_t* m_k, const int64_t* obs_local,
                   txh_kfb** out);
void txh_kfb_destroy(txh_kfb* b);
int txh_kfb_set(txh_kfb* b, int64_t block, int which, const double* host, void* stream);
int txh_kfb_get(txh_kfb* b, int64_t block, int which, double* host, void* stream);
int txh_kfb_filter(txh_kfb* b, const uint8_t* active_host, const double* z_host, double* O_dev, double* I_dev, void* stream);

/* Synchronise `stream` and report a poisoned launch (TXH_E_WATCHDOG), an innovation covariance that was
 * not positive definite in an earlier txh_enkf_solve (TXH_E_INVALID), or a CUDA fault. */
int txh_check(txh_net* net, void* stream);

/* kernel-launch counter (bench.py's gpu_launches claim) */
int64_t txh_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* TXH_H */
