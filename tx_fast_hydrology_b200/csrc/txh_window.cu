// txh_window.cu -- window-resident routing kernel for sm_100a.
//
// route_window_kernel evaluates `nsteps` timesteps of the Muskingum update (tx_fast_hydrology/nutils.py:64-89,
// as called from muskingum.py:527-533) in ONE launch with the network state resident in shared memory:
// the network is cut into tasks of a few rows each (pockets = bundled side subtrees, segments = pieces of
// the long paths; txh_topology.cpp), a warp claims a task, loads its rows of O and I once, runs EVERY
// step of the launch on them in shared memory, and writes them back once.  HBM/L2 traffic per launch is
// one read and one write of the state plus the single rows tasks hand to each other, instead of a read
// and a write per step.
//
// Tasks exchange rows through a slot ring in global memory, ring[step][slot][ld]: a pocket publishes the
// outflow of its root, a segment the outflow of its last reach, per step.  A per-task progress word
// (steps published, release/acquire) orders them; tasks are claimed in a topological order, so a task
// only ever waits for tasks claimed before it, which are running or done -- every CTA is resident.
// Along a long path the step is the affine recurrence o_k = alpha_k (o_{k-1} + side_k) + r_k, so a
// segment first evaluates it with nothing entering (PRE), then needs ONE fused multiply-add per hop,
// out = A_last * o_in + B_last, before handing on -- consecutive steps ripple down the path as a
// systolic wavefront -- and fixes its interior rows up afterwards (FIX).
// Ensemble members are the SIMD axis: a lane owns two adjacent member columns (128-bit accesses).
//
// Update variant (template parameter UPD; txh_run_assimilating): the launch also applies the ensemble Kalman update the
// state still owes -- p is linear in the state rows and the update acts on the member axis, so each task transforms its
// freshly loaded p rows with the 64 x 64 matrix T on the FP64 tensor cores (transform_p_rows) and the posterior state
// never goes through global memory.  Such a launch may start while the kernel that computes T still runs
// (programmatic dependent launch): it loads its first tasks and waits for T only then (stage_T).
//
// Recording variant (template parameter REC; txh_route_run / txh_run_assimilating_rec with rec_*): after every step of
// the call that is a multiple of rec_every the outflow of each recorded row goes to rec_out[step / rec_every - 1][k][M].
// A row's slot k rides in the spare word of its per-row record.  A pocket row has its outflow in registers every step;
// a segment's interior rows never form theirs before the last step of a launch (only p0 is kept, the FIX loop folds
// C_k o_in into it), so PRE stores B_k into the row's rec_out cell and the same lane adds A_k o_in in the FIX loop.
#include <cstdlib>

#include "txh_kernels.cuh"

namespace txh {

void count_launch();

namespace {

__device__ __forceinline__ int ld_relaxed_s32(const int* p)
{
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ double2 ld_row(const double* p) { return __ldcg(reinterpret_cast<const double2*>(p)); }
__device__ __forceinline__ void st_row(double* p, double2 v) { __stcg(reinterpret_cast<double2*>(p), v); }
__device__ __forceinline__ void cp_async4(unsigned sa, const void* g)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sa), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async16(unsigned sa, const void* g)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ double2 lds_row(unsigned sa)
{
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(sa));
    return v;
}
__device__ __forceinline__ void sts_row(unsigned sa, double2 v)
{
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(sa), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ double lds_f64(unsigned sa)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(sa));
    return v;
}
__device__ __forceinline__ void sts_f64(unsigned sa, double v)
{
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(sa), "d"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(unsigned sa)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(sa));
    return v;
}
__device__ __forceinline__ void sts_u32(unsigned sa, uint32_t v)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(sa), "r"(v) : "memory");
}

// ---- TMA bulk copies (cp.async.bulk, 1-D) + mbarrier: the rows of a task are contiguous in global memory, and with
// 64 doubles per row (one member block) their shared-memory image is contiguous too, so ONE elected lane moves all
// outflow rows of a task with one instruction (and its inflow rows with another) instead of every lane issuing a
// 16-byte cp.async per row.
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned mbar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned mbar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned phase)
{
    unsigned ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(mbar), "r"(phase) : "memory");
    } while (!ok);
}

// Programmatic dependent launch: a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start
// once every CTA of the kernel before it in the stream has executed launch_dependents (or exited); what that kernel
// wrote is only visible after wait.
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

constexpr int kInRing = 4;                 // pockets: rows of other tasks in flight per warp (cp.async ring)
constexpr int kSegRing = 8;                // segments: the ring also takes the (unused) scratch slots
constexpr int kInRingUpd = 2;              // the update variant gives two ring rows per warp to the CTA's copy of T (16 warps
constexpr int kSegRingUpd = 6;             // fit instead of 14; measured: the ring depth does not matter, 3 / 7 rows at 15
                                           // warps ran as fast as 2 / 6); the per-warp layout of the launch is sized accordingly
constexpr int kStepsStaged = 16;            // interpolation records of a launch kept in shared memory
constexpr int kWinThreads = 512;           // one CTA per SM, up to 16 warps
constexpr uint32_t kIdMask = 0x3fffffffu;

// Hand-over protocol: a ring cell that has not been written holds the EMPTY pattern (all bits set -- a NaN no
// arithmetic produces).  The producer just stores its row; the consumer polls the 16 bytes of its own two
// member columns until neither is EMPTY, and puts EMPTY back (every cell has exactly one reader), so the
// ring is clean again when the launch ends.  No flags, no fences: a lane only ever depends on the cell the
// same lane of the producer wrote.
__device__ __forceinline__ bool cell_full(double2 v)
{
    return __double_as_longlong(v.x) != -1ll && __double_as_longlong(v.y) != -1ll;
}
__device__ __forceinline__ double2 ld_cell_relaxed(const double* p)
{
    double2 v;
    asm volatile("ld.relaxed.gpu.global.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double2 empty_cell()
{
    return make_double2(__longlong_as_double(-1ll), __longlong_as_double(-1ll));
}

// Polls `cell` (this lane's 16 bytes of a ring row) until it is full; `v` is what an earlier read saw.
// Returns false when the launch is being abandoned (watchdog / poisoned handle).  (Moving the polling loop into a
// function of its own to shrink the dozen walks that inline it costs 40 us per launch: the call spills the walk's
// registers.)
__device__ __forceinline__ bool wait_cell(const WinArgs& a, const double* cell, bool active, double2& v, int lane)
{
    bool ok = !active || cell_full(v);
    if (__all_sync(0xffffffffu, ok)) return true;
    unsigned spins = 0, nap = (unsigned)a.nap_min;
    unsigned long long t0 = 0;
    for (;;) {
        if (!ok) { v = ld_cell_relaxed(cell); ok = cell_full(v); }
        if (__all_sync(0xffffffffu, ok)) return true;
        if ((++spins & 15u) == 0) {
            if (ld_relaxed_s32(a.status) != 0) return false;
            const unsigned long long now = globaltimer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > a.watchdog_ns) { if (lane == 0) atomicExch(a.status, 1); return false; }
        }
        if (nap) __nanosleep(nap);
        if (nap < (unsigned)a.nap_max) nap <<= 1;
    }
}

// Rows handed over by other tasks, consumed in a fixed order every step: a continuous stream (step, index)
// prefetched D rows ahead through a shared-memory ring, across step boundaries.  One cp.async group per row.
// A prefetch that came too early sees EMPTY and the consumer falls back to polling the cell itself.
// The list holds byte offsets of the slots inside one step of the ring.
struct InStream {
    int in_flight;             // rows issued and not yet consumed
    int pi, ci;                // index of the next row to issue / consume within its step
    int psteps;                // steps left to issue (including the current one)
    unsigned slot_i, slot_c;   // byte offsets of the ring cells of the next issue / next consume
    char* pbase;               // this lane's columns of the ring step being issued / consumed
    char* cbase;
    bool dead;                 // the launch is being abandoned: stop waiting
};

template <int D>
__device__ __forceinline__ void stream_issue(InStream& st, const WinArgs& a, unsigned ring_sa, unsigned list_sa, int nL,
                                             size_t step_bytes, bool active)
{
    if (active) cp_async16(ring_sa + st.slot_i, st.pbase + lds_u32(list_sa + 4u * st.pi));
    cp_async_commit();
    st.slot_i = st.slot_i + 512u == D * 512u ? 0u : st.slot_i + 512u;
    ++st.in_flight;
    if (++st.pi == nL) { st.pi = 0; --st.psteps; st.pbase += step_bytes; }
}

template <int D>
__device__ __forceinline__ double2 stream_next(InStream& st, const WinArgs& a, unsigned ring_sa, unsigned list_sa, int nL,
                                               size_t step_bytes, bool active, int lane)
{
    if (st.in_flight >= D) cp_async_wait_group<D - 1>();                // the oldest of D rows in flight
    else cp_async_wait_all();
    double2 v = lds_row(ring_sa + st.slot_c);
    double* cell = reinterpret_cast<double*>(st.cbase + lds_u32(list_sa + 4u * st.ci));
    if (!st.dead && !wait_cell(a, cell, active, v, lane)) st.dead = true;
    if (active) st_row(cell, empty_cell());
    st.slot_c = st.slot_c + 512u == D * 512u ? 0u : st.slot_c + 512u;
    --st.in_flight;
    if (++st.ci == nL) { st.ci = 0; st.cbase += step_bytes; }
    if (st.psteps > 0) stream_issue<D>(st, a, ring_sa, list_sa, nL, step_bytes, active);
    return v;
}

// scale * (sum of this row over the members of the warp's block), lane 0 stores it (last step of a launch)
__device__ __forceinline__ void emit_rowsum(const WinArgs& a, int pos, int col, double2 on, int lane)
{
    double v = (col < a.M ? on.x : 0.0) + (col + 1 < a.M ? on.y : 0.0);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) a.rowsum[pos] = v * a.rowsum_scale;
}

// this lane's columns (< M) of a recorded row: rj = index of the recorded step, rs = the row's slot
__device__ __forceinline__ double* rec_cell(const WinArgs& a, int rj, int rs, int col)
{
    return a.rec_out + ((size_t)rj * a.rec_count + rs) * a.M + col;
}
__device__ __forceinline__ void rec_store(const WinArgs& a, int rj, int rs, int col, double2 v)
{
    double* d = rec_cell(a, rj, rs, col);
    if (col < a.M) d[0] = v.x;
    if (col + 1 < a.M) d[1] = v.y;
}

// Per-row record in shared memory (48 bytes): everything a row update needs besides its state row, read with
// three 128-bit loads one row ahead of the arithmetic.
//   +0 header word   +4 recording slot (REC)   +8 alpha   +16 beta   +24 chi   +32 gamma*F[r0]   +40 gamma*F[r1]
constexpr unsigned kRec = 48u;
struct RowIn {
    uint32_t h;
    double al, be, ch, g0, g1;
    double2 p;
};
__device__ __forceinline__ RowIn load_rowin(unsigned rec_sa, unsigned p_sa)
{
    RowIn x;
    x.h = lds_u32(rec_sa);
    x.al = lds_f64(rec_sa + 8u);
    const double2 bc = lds_row(rec_sa + 16u), g = lds_row(rec_sa + 32u);
    x.be = bc.x; x.ch = bc.y; x.g0 = g.x; x.g1 = g.y;
    x.p = lds_row(p_sa);
    return x;
}

struct FCtx {
    double w0, w1;
    double2 wm0, wm1;
};

// gamma*q of this lane's two members; the staged rows already carry gamma
template <bool HAS_F, bool HAS_W>
__device__ __forceinline__ double2 forcing_q(const FCtx& c, double g0, double g1)
{
    double2 q = make_double2(0.0, 0.0);
    if (HAS_F) {
        if (HAS_W) { q.x = c.wm0.x * g0 + c.wm1.x * g1; q.y = c.wm0.y * g0 + c.wm1.y * g1; }
        else { q.x = c.w0 * g0 + c.w1 * g1; q.y = q.x; }
    }
    return q;
}

// per-task context
struct Tk {
    unsigned sP, sScr, sIn, sRec, sCum, sCumC, sWords, sList;
    int len, n_in, nL, col, lane, begin, ld;
    unsigned ldb;              // bytes of a ring row (ld doubles; a ring step stays below 4 GiB, see window_fit)
    bool active;
    double* Ig;
    double* Og;
    size_t step_bytes;
};

// recording slot of row r of the task (-1: not recorded), staged at task load
__device__ __forceinline__ int rec_slot_of(const Tk& tk, int r) { return (int)lds_u32(tk.sRec + kRec * r + 4u); }

// p + gamma*q of this lane's two members, accumulated with fused multiply-adds (one operation less per member than
// forming q first)
template <bool HAS_F, bool HAS_W>
__device__ __forceinline__ double2 forcing_add(const FCtx& c, double g0, double g1, double2 p)
{
    if (HAS_F) {
        if (HAS_W) {
            p.x = fma(c.wm1.x, g1, fma(c.wm0.x, g0, p.x));
            p.y = fma(c.wm1.y, g1, fma(c.wm0.y, g0, p.y));
        } else {
            const double q = c.w0 * g0 + c.w1 * g1;
            p.x += q; p.y += q;
        }
    }
    return p;
}

// One step of a pocket: depth-first walk, o' = alpha*inflow + (p + gamma q), p' = beta*inflow + chi*o'.
// Two thirds of the rows (C3) are leaves or chain rows: no input word, no push, at most a scratch row to park in.  One
// test of the header skips the input loop for them, and the scratch store is predicated (profiles/r05_pocket_row_sass.txt:
// 40 instructions per such row, 52 / 60 when the record was read one row ahead into registers of its own).  The record
// of the next row is read into the registers each field of this row frees after its last use, so the loop edge moves
// only the header instead of the whole record; the arithmetic of the row covers the latency of the loads.  (Unrolling
// the walk by two rows instead was 8 % slower: the kernel is sensitive to its code size.)  Past the last row the loads
// read the next area of the warp's shared memory and are not used.
template <bool LAST, bool HAS_F, bool HAS_W, int IR, bool REC>
__device__ __forceinline__ void pocket_step(const WinArgs& a, const Tk& tk, InStream& ist, const FCtx& fc, char* ringS,
                                            int rj)
{
    unsigned aRec = tk.sRec, aP = tk.sP, aW = tk.sWords;
    double* ig = tk.Ig;
    double* og = tk.Og;
    double2 acc = make_double2(0.0, 0.0);
    RowIn x = load_rowin(aRec, aP);
    for (int r = 0; r < tk.len; ++r) {
        const uint32_t h = x.h;
        const uint32_t park = h & 0x3eu;                         // (scratch row + 1) << 1 the outflow is parked in, 0: none
        double2 inflow = (h & HDR_ACC) ? acc : make_double2(0.0, 0.0);
        // the next row, whose record the loads below read (an opaque add: the old addresses die here)
        asm("add.u32 %0, %0, %1;" : "+r"(aRec) : "n"(kRec));
        asm("add.u32 %0, %0, 512;" : "+r"(aP));
        if (h & ~0x3fu) {                                        // input words and / or a push
            for (uint32_t k = (h >> 6) & 0x1ffffffu; k > 0; --k) {
                const uint32_t w = lds_u32(aW);
                aW += 4u;
                const double2 v = (w & WIN_SLOT) ? stream_next<IR>(ist, a, tk.sIn, tk.sList, tk.nL, tk.step_bytes, tk.active, tk.lane)
                                                 : lds_row(tk.sScr + (w << 9));
                inflow.x += v.x; inflow.y += v.y;
            }
        }
        const bool push = (h & HDR_PUSH) != 0u;
        x.h = lds_u32(aRec);
        const double2 pq = forcing_add<HAS_F, HAS_W>(fc, x.g0, x.g1, x.p);
        {
            const double2 g = lds_row(aRec + 32u);
            x.g0 = g.x; x.g1 = g.y;
            x.p = lds_row(aP);
        }
        double2 on;
        on.x = fma(x.al, inflow.x, pq.x);
        on.y = fma(x.al, inflow.y, pq.y);
        x.al = lds_f64(aRec + 8u);
        if (!LAST) {
            double2 pn;
            pn.x = x.be * inflow.x + x.ch * on.x;
            pn.y = x.be * inflow.y + x.ch * on.y;
            const double2 bc = lds_row(aRec + 16u);
            x.be = bc.x; x.ch = bc.y;
            sts_row(aP - 512u, pn);
        } else {
            const double2 bc = lds_row(aRec + 16u);
            x.be = bc.x; x.ch = bc.y;
            if (tk.active) { st_row(ig, inflow); st_row(og, on); }
            if (a.rowsum) emit_rowsum(a, tk.begin + r, tk.col, on, tk.lane);
        }
        if (REC && rj >= 0) {
            const int rs = rec_slot_of(tk, r);
            if (rs >= 0) rec_store(a, rj, rs, tk.col, on);
        }
        if (push) {                                              // published: the slot word follows the inputs
            const uint32_t slot = lds_u32(aW);
            aW += 4u;
            if (tk.active) st_row(reinterpret_cast<double*>(ringS + slot * tk.ldb), on);
        }
        if (park) sts_row(tk.sScr - 512u + (park << 8), on);
        acc = on;
        ig += tk.ld; og += tk.ld;
    }
}

// One step of a segment.  PRE: side_k = pocket roots joining reach k; B_k = the recurrence with nothing entering
// the segment; what the NEXT step needs of this one is affine in the flow o_in entering the segment:
//   p_k' = beta_k i_k + chi_k o_k = P0_k + C_k o_in,   P0_k = beta_k (side_k + B_{k-1}) + chi_k B_k,
//   C_k = beta_k A_{k-1} + chi_k A_k  (A = prefix product of alpha, A_{-1} = 1; precomputed).
// Hop: out = A_last * o_in + B_last, handed on before anything else.  In the last step (side_k, B_k) are
// parked in the global I / O rows for the final fix-up o_k = B_k + A_k o_in, i_k = o_{k-1} + side_k.
template <bool LAST, bool HAS_F, bool HAS_W, int SR, bool REC>
__device__ __forceinline__ void segment_step(const WinArgs& a, const Tk& tk, InStream& ist, const FCtx& fc, char* ringS,
                                             int out_slot, unsigned long long* trs, int rj)
{
    unsigned aRec = tk.sRec, aP = tk.sP;
    double* ig = tk.Ig;
    double* og = tk.Og;
    double2 B = make_double2(0.0, 0.0);
    RowIn nx = load_rowin(aRec, aP);
    for (int r = 0; r < tk.len; ++r) {
        const RowIn x = nx;
        if (r + 1 < tk.len) nx = load_rowin(aRec + kRec, aP + 512u);
        const uint32_t h = x.h;
        double2 inflow = (h & HDR_ACC) ? B : make_double2(0.0, 0.0);   // side_k + B_{k-1}
        double2 side = make_double2(0.0, 0.0);
        for (uint32_t k = (h >> 6) & 0x1fffu; k > 0; --k) {
            const double2 v = stream_next<SR>(ist, a, tk.sScr, tk.sList, tk.nL, tk.step_bytes, tk.active, tk.lane);
            side.x += v.x; side.y += v.y;
        }
        inflow.x += side.x; inflow.y += side.y;
        const double2 q = forcing_q<HAS_F, HAS_W>(fc, x.g0, x.g1);
        B.x = x.al * inflow.x + (x.p.x + q.x);
        B.y = x.al * inflow.y + (x.p.y + q.y);
        if (!LAST) {
            double2 p0;
            p0.x = x.be * inflow.x + x.ch * B.x;
            p0.y = x.be * inflow.y + x.ch * B.y;
            sts_row(aP, p0);
            if (REC && rj >= 0) {                                   // B_k; the FIX loop adds A_k o_in
                const int rs = rec_slot_of(tk, r);
                if (rs >= 0) rec_store(a, rj, rs, tk.col, B);
            }
        } else {
            if (tk.active) { st_row(ig, side); st_row(og, B); }
            ig += tk.ld; og += tk.ld;
        }
        aRec += kRec; aP += 512u;
    }
    // hop
    double2 oin = make_double2(0.0, 0.0);
    for (int k = 0; k < tk.n_in; ++k) {
        double* cell = reinterpret_cast<double*>(ringS + (size_t)(lds_u32(tk.sWords + 4u * k) & kIdMask) * tk.ld * sizeof(double));
        double2 v = tk.active ? ld_cell_relaxed(cell) : make_double2(0.0, 0.0);
        if (!ist.dead && !wait_cell(a, cell, tk.active, v, tk.lane)) ist.dead = true;
        if (tk.active) st_row(cell, empty_cell());
        oin.x += v.x; oin.y += v.y;
    }
    const double Al = lds_f64(tk.sCum + 8u * (tk.len - 1));
    double2 out;
    out.x = Al * oin.x + B.x;
    out.y = Al * oin.y + B.y;
    if (tk.active && out_slot >= 0) st_row(reinterpret_cast<double*>(ringS + (size_t)out_slot * tk.ld * sizeof(double)), out);
    if (trs && tk.lane == 0) *trs = globaltimer_ns();
    if (!LAST) {
        // FIX, folded into the next state: p_k' = P0_k + C_k o_in
        unsigned aQ = tk.sP, aC = tk.sCumC;
        for (int r = 0; r < tk.len; ++r) {
            const double C = lds_f64(aC);
            double2 p0 = lds_row(aQ);
            p0.x = C * oin.x + p0.x;
            p0.y = C * oin.y + p0.y;
            sts_row(aQ, p0);
            if (REC && rj >= 0) {
                // o_k = B_k + A_k o_in (B_k parked in the row's cell by PRE); the last row's is `out`
                const int rs = rec_slot_of(tk, r);
                if (rs >= 0) {
                    double2 o = out;
                    if (r + 1 < tk.len) {
                        const double A = lds_f64(tk.sCum + 8u * r);
                        const double* d = rec_cell(a, rj, rs, tk.col);
                        const double b0 = tk.col < a.M ? d[0] : 0.0, b1 = tk.col + 1 < a.M ? d[1] : 0.0;
                        o.x = A * oin.x + b0;
                        o.y = A * oin.y + b1;
                    }
                    rec_store(a, rj, rs, tk.col, o);
                }
            }
            aQ += 512u; aC += 8u;
        }
    } else {
        // final FIX (each lane re-reads its own cells of the parked rows)
        double2 op = oin;
        ig = tk.Ig; og = tk.Og;
        for (int r = 0; r < tk.len; ++r) {
            double2 side = make_double2(0.0, 0.0), Bk = side;
            if (tk.active) { side = ld_row(ig); Bk = ld_row(og); }
            double2 on = out;
            if (r + 1 < tk.len) {
                const double A = lds_f64(tk.sCum + 8u * r);
                on.x = A * oin.x + Bk.x;
                on.y = A * oin.y + Bk.y;
            }
            double2 it;
            it.x = op.x + side.x;
            it.y = op.y + side.y;
            if (tk.active) { st_row(og, on); st_row(ig, it); }
            if (a.rowsum) emit_rowsum(a, tk.begin + r, tk.col, on, tk.lane);
            if (REC && rj >= 0) {
                const int rs = rec_slot_of(tk, r);
                if (rs >= 0) rec_store(a, rj, rs, tk.col, on);
            }
            op = on;
            ig += tk.ld; og += tk.ld;
        }
    }
}

// D(8x8) += A(8x4) * B(4x8), FP64 tensor cores.  lane = 4g + t: a = A[g][t], b = B[t][g], c0 = C[g][2t], c1 = C[g][2t+1]
__device__ __forceinline__ void dmma8x8x4(double& c0, double& c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// The ensemble update owed to the state, applied to the freshly loaded p rows of a task (da.py:112-126 in ensemble
// form, see txh_da.cu).  The update acts on the member axis, o+ = o + (o - mean(o)) T (+ qs W on gauged rows), and
// after a routing step i = sum of the upstream o, so i+ = sum of the upstream o+ = i + (i - mean(i)) T (+ the gauge
// terms of the upstream rows); p = beta i + chi o is linear in both with per-row scalars, hence
//     p+ = p + (p - mean(p)) T + chi qs_g W_g [row gauged] + beta sum over gauged upstream rows of qs_u W_u
// and the posterior state never makes the trip through HBM: the next window starts from the prior rows the last one
// wrote.  8-row tiles on the FP64 tensor cores; lane (g, t) owns row g, members 8j + 2t, 8j + 2t + 1 of a tile (the
// k index of a fragment is permuted accordingly, as in enkf_update64_kernel).  T lives in shared memory, once per
// CTA, zero-padded to 64 x 64 and swizzled: element (k, c) at k*64 + (((c >> 3) ^ ((k >> 1) & 3)) << 3) + (c & 7), so
// the four rows k0, k0+2, k0+4, k0+6 a B fragment touches fall into different banks without padding.
__device__ __forceinline__ unsigned t_swz(int k, int c) { return (unsigned)(k * 64 + ((((c >> 3) ^ ((k >> 1) & 3)) << 3) | (c & 7))) * 8u; }

__device__ __noinline__ void transform_p_rows(const WinArgs& a, unsigned sb, unsigned sT, int len, int lane)
{
    const int g = lane >> 2, t = lane & 3, M = a.M;
    const double invM = 1.0 / (double)M;
    for (int r0 = 0; r0 < len; r0 += 8) {
        const bool ok = r0 + g < len;
        const unsigned ra = sb + (unsigned)(ok ? r0 + g : r0) * 512u + t * 16u;
        // row mean: the four lanes of a row hold 16 members each
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const double2 v = lds_row(ra + j * 64u);
            const int k = 8 * j + 2 * t;
            s += (k < M ? v.x : 0.0) + (k + 1 < M ? v.y : 0.0);
        }
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        const double mu = s * invM;
        // 8 independent accumulator chains (one per column tile); the k loop is a real loop, so the 8 tensor-core
        // operations of a k step stay next to each other (fully unrolled, ptxas schedules one chain after the other
        // and a warp then issues one DMMA per two latencies instead of one per pipe slot)
        double acc[8][2];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j][0] = acc[j][1] = 0.0;
#pragma unroll 2
        for (int ks = 0; ks < 16; ++ks) {
            const int k = 8 * (ks >> 1) + 2 * t + (ks & 1);
            const double pv = lds_f64(ra - t * 16u + (unsigned)k * 8u);
            const double av = (ok && k < M) ? pv - mu : 0.0;
            double b[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) b[j] = lds_f64(sT + t_swz(k, 8 * j + g));
#pragma unroll
            for (int j = 0; j < 8; ++j) dmma8x8x4(acc[j][0], acc[j][1], av, b[j]);
        }
        if (ok) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                double2 v = lds_row(ra + j * 64u);
                v.x += acc[j][0]; v.y += acc[j][1];
                sts_row(ra + j * 64u, v);
            }
        }
    }
}

// UPD + REC: the forecast and the posterior of the task's recorded rows for the update this launch applies (the posterior
// of the fused loop never reaches HBM otherwise).  Runs at task load, T staged, before the task writes any row of O: the
// forecast row is still in O.  A lane loads its two members and forms o + sum_j (o_j - mean) T[j][c] + qs_g W_g[c] (own
// gauge) with the other members shuffled in: one memory latency per row, not one per member.
__device__ __noinline__ void record_posterior(const WinArgs& a, unsigned sRec, unsigned sT, int task, int begin, int len,
                                              int lane)
{
    const int M = a.M, c0 = 2 * lane, c1 = c0 + 1;
    for (int r = 0; r < len; ++r) {
        const int rs = (int)lds_u32(sRec + kRec * r + 4u);
        if (rs < 0) continue;
        const double* o = a.O + (size_t)(begin + r) * a.ld;
        const double mu = __ldcg(a.rec_mean + begin + r);
        // this lane's two members of the row in one load; member j comes from lane j / 2 by a shuffle
        const double2 ov = c0 < a.ld ? ld_row(o + c0) : make_double2(0.0, 0.0);
        double g0 = 0.0, g1 = 0.0;
#pragma unroll 4
        for (int j = 0; j < M; j += 2) {
            const double oa = __shfl_sync(0xffffffffu, ov.x, j >> 1) - mu, ob = __shfl_sync(0xffffffffu, ov.y, j >> 1) - mu;
            g0 = fma(oa, lds_f64(sT + t_swz(j, c0 & 63)), g0);
            g1 = fma(oa, lds_f64(sT + t_swz(j, c1 & 63)), g1);
            if (j + 1 < M) {
                g0 = fma(ob, lds_f64(sT + t_swz(j + 1, c0 & 63)), g0);
                g1 = fma(ob, lds_f64(sT + t_swz(j + 1, c1 & 63)), g1);
            }
        }
        for (int e = __ldg(a.gfix_off + task), e1 = __ldg(a.gfix_off + task + 1); e < e1; ++e) {
            const int2 x = __ldg(a.gfix + e);
            if ((x.x >> 16) != 0 || (x.x & 0xffff) != r) continue;      // the row's own gauge only
            const double q = __ldg(a.upQs + x.y);
            const double* wr = a.upW + (size_t)x.y * M;
            if (c0 < M) g0 += q * __ldg(wr + c0);
            if (c1 < M) g1 += q * __ldg(wr + c1);
        }
        const size_t at = (size_t)rs * M;
        if (c0 < M) {
            if (a.rec_prior) a.rec_prior[at + c0] = ov.x;
            if (a.rec_post) a.rec_post[at + c0] = ov.x + g0;
        }
        if (c1 < M) {
            if (a.rec_prior) a.rec_prior[at + c1] = ov.y;
            if (a.rec_post) a.rec_post[at + c1] = ov.y + g1;
        }
    }
}

// Shared-memory state of a task: ONE row per reach, p = beta*i + chi*o, the part of the next update that
// depends on the old state (o' = alpha*inflow + (gamma*q + p)); the outflows and inflows themselves only
// exist in registers, and are written to global memory in the last step of the launch.
template <bool HAS_F, bool HAS_W, bool UPD, bool REC>
__global__ void __launch_bounds__(kWinThreads, 1)
route_window_kernel(const WinArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_all[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const unsigned sb = (unsigned)__cvta_generic_to_shared(smem_all + (size_t)warp * a.smem_per_warp);
    const unsigned sSteps = (unsigned)__cvta_generic_to_shared(smem_all) + (unsigned)a.off_steps;   // one copy per CTA
    constexpr int IR = UPD ? kInRingUpd : kInRing, SR = UPD ? kSegRingUpd : kSegRing;
    const int nmb = a.n_mblocks, ld = a.ld;
    const long long total = (long long)a.n_tasks * nmb;
    Tk tk;
    tk.sP = sb + lane * 16u; tk.sScr = sb + a.off_scr + lane * 16u; tk.sIn = sb + a.off_in + lane * 16u;
    tk.sRec = sb + a.off_rec; tk.sCum = sb + a.off_cum; tk.sCumC = sb + a.off_cumc;
    tk.sWords = sb + a.off_words; tk.sList = sb + a.off_list;
    tk.lane = lane; tk.ld = ld; tk.ldb = (unsigned)ld * (unsigned)sizeof(double);
    tk.step_bytes = (size_t)a.n_slots * ld * sizeof(double);
    // bulk staging of the state rows (see the helpers above): one mbarrier per warp
    const bool bulk = a.off_mbar > 0 && ld == kMemberBlock;
    const unsigned sMbar = sb + a.off_mbar;
    unsigned mphase = 0;
    if (bulk) {
        if (lane == 0) mbar_init(sMbar, 1);
        __syncwarp();
    }
    // The ensemble transform of the update this launch applies while it loads its tasks: one copy per CTA, behind the
    // per-warp areas.  The launch may have started before the kernel that computes T has finished (programmatic
    // dependent launch): every warp loads its first task, which needs nothing of that kernel, THEN waits for it, stages
    // its share of T and waits for the other warps' shares (a counter in shared memory; a warp without a task stages
    // its share before it leaves).
    const unsigned sT = (unsigned)__cvta_generic_to_shared(smem_all) + (unsigned)a.off_T;
    const unsigned sTcount = sT + 64u * 64u * 8u;
    bool t_ready = !UPD;
    if (UPD && threadIdx.x == 0) sts_u32(sTcount, 0u);
    // the launch's interpolation records (24 B each), once per CTA when they fit (<= kStepsStaged): copied, or -- no
    // init kernel -- resolved here, one step per lane (nothing of this depends on the kernel in front of the launch)
    if (HAS_F && a.nsteps <= kStepsStaged && warp == 0) {
        if (a.steps != nullptr) {
            for (int i = lane; i < 6 * a.nsteps; i += 32) sts_u32(sSteps + 4u * i, __ldg(reinterpret_cast<const uint32_t*>(a.steps) + i));
        } else if (lane < a.nsteps) {
            const StepInterp si = interp_step(a.times, a.R, (double)(a.t0_ns + (a.step_base + lane + 1) * a.dt_ns), a.method);
            sts_u32(sSteps + 24u * lane, (uint32_t)si.r0); sts_u32(sSteps + 24u * lane + 4u, (uint32_t)si.r1);
            sts_f64(sSteps + 24u * lane + 8u, si.w0); sts_f64(sSteps + 24u * lane + 16u, si.w1);
        }
    }
    __syncthreads();
    griddep_launch_dependents();
    auto stage_T = [&]() {
        griddep_wait();
        const int nw = blockDim.x >> 5;
        for (int e = warp * 32 + lane; e < 64 * 64; e += nw * 32) {
            const int k = e >> 6, c = e & 63;
            sts_f64(sT + t_swz(k, c), (k < a.M && c < a.M) ? __ldcg(a.upT + (size_t)k * a.M + c) : 0.0);
        }
        __threadfence_block();
        __syncwarp();
        if (lane == 0) atomicAdd(reinterpret_cast<unsigned*>(smem_all + a.off_T + 64 * 64 * 8), 1u);
        while (lds_u32(sTcount) < (unsigned)nw) __nanosleep(64);
        __threadfence_block();
        t_ready = true;
    };

    for (;;) {
        long long t = 0;
        if (lane == 0) t = (long long)atomicAdd(a.ticket, 1ull);
        t = __shfl_sync(0xffffffffu, t, 0);
        if (t >= total || ld_relaxed_s32(a.status) != 0) {      // (status: a launch on this handle was poisoned)
            if (!t_ready) stage_T();                             // the other warps of the CTA wait for this share
            break;
        }
        const int task = (int)(t / nmb);
        const int mb = (int)(t - (long long)task * nmb);
        const WTaskDesc td = a.tasks[task];
        unsigned long long* tr = a.trace ? a.trace + (size_t)t * (4 + a.nsteps) : nullptr;
        if (tr && lane == 0) tr[0] = globaltimer_ns();
        const int len = td.len;
        const int col = mb * kMemberBlock + lane * 2;
        const bool active = col < ld;
        const int ccol = active ? col : 0;
        tk.len = len; tk.n_in = td.n_in; tk.col = col; tk.active = active; tk.begin = td.begin;
        tk.Og = a.O + (size_t)td.begin * ld + ccol;
        tk.Ig = a.I + (size_t)td.begin * ld + ccol;

        // ---- load the task: input stream, step records, per-row records; rows of I and O -> p ----
        for (int i = lane; i < td.n_words; i += 32) cp_async4(tk.sWords + 4u * i, a.inw + td.in_off + i);
        // the launch's interpolation records: in shared memory when they fit (<= kStepsStaged), else read in place
        const bool steps_staged = a.nsteps <= kStepsStaged;
        auto step_rows = [&](int s) -> int2 {
            if (steps_staged) return make_int2((int)lds_u32(sSteps + 24u * s), (int)lds_u32(sSteps + 24u * s + 4u));
            return make_int2(__ldg(&a.steps[s].r0), __ldg(&a.steps[s].r1));
        };
        auto step_weights = [&](int s) -> double2 {
            if (steps_staged) return make_double2(lds_f64(sSteps + 24u * s + 8u), lds_f64(sSteps + 24u * s + 16u));
            return make_double2(__ldg(&a.steps[s].w0), __ldg(&a.steps[s].w1));
        };
        // rows of O straight into their p slots, rows of I (SR at a time) into the [scratch | ring] area: every
        // load of the task is in flight before the first is waited for
        if (bulk) {
            // the rows were last touched by this warp's ordinary stores: order them before the async proxy's writes
            __syncwarp();
            if (lane == 0) {
                fence_proxy_async();
                const unsigned bo = 512u * (unsigned)len, bi = 512u * (unsigned)(len < SR ? len : SR);
                mbar_expect_tx(sMbar, bo + bi);
                bulk_g2s(sb, a.O + (size_t)td.begin * ld, bo, sMbar);
                bulk_g2s(sb + a.off_scr, a.I + (size_t)td.begin * ld, bi, sMbar);
            }
        } else if (active) {
            for (int r = 0; r < len; ++r) {
                cp_async16(tk.sP + 512u * r, tk.Og + (size_t)r * ld);
                if (r < SR) cp_async16(tk.sScr + 512u * r, tk.Ig + (size_t)r * ld);
            }
        }
        cp_async_commit();
        for (int i = lane; i < len; i += 32) {
            const double2 ab = *reinterpret_cast<const double2*>(a.coef + 4 * (size_t)(td.begin + i));
            const double2 cg = *reinterpret_cast<const double2*>(a.coef + 4 * (size_t)(td.begin + i) + 2);
            const unsigned rec = tk.sRec + kRec * i;
            sts_u32(rec, a.hdr[td.begin + i]);
            if (REC) sts_u32(rec + 4u, (uint32_t)__ldg(a.rec_slot + td.begin + i));
            sts_f64(rec + 8u, ab.x);
            sts_row(rec + 16u, make_double2(ab.y, cg.x));
            sts_row(rec + 32u, make_double2(0.0, 0.0));
            sts_f64(tk.sCum + 8u * i, a.cumA[td.begin + i]);
            sts_f64(tk.sCumC + 8u * i, a.cumC[td.begin + i]);
        }
        for (int r0 = 0; r0 < len; r0 += SR) {
            if (r0 > 0) {
                if (bulk) {
                    __syncwarp();                               // the previous chunk has been read by every lane
                    if (lane == 0) {
                        fence_proxy_async();
                        const unsigned bi = 512u * (unsigned)(len - r0 < SR ? len - r0 : SR);
                        mbar_expect_tx(sMbar, bi);
                        bulk_g2s(sb + a.off_scr, a.I + (size_t)(td.begin + r0) * ld, bi, sMbar);
                    }
                } else if (active) {
                    for (int r = r0; r < len && r < r0 + SR; ++r) cp_async16(tk.sScr + 512u * (r - r0), tk.Ig + (size_t)r * ld);
                }
                cp_async_commit();
            }
            cp_async_wait_all();
            if (bulk) { mbar_wait(sMbar, mphase); mphase ^= 1u; }
            __syncwarp();
            for (int r = r0; r < len && r < r0 + SR; ++r) {
                const double2 bc = lds_row(tk.sRec + kRec * r + 16u);
                double2 p = make_double2(0.0, 0.0);
                if (active) {
                    const double2 oo = lds_row(tk.sP + 512u * r), io = lds_row(tk.sScr + 512u * (r - r0));
                    p.x = bc.x * io.x + bc.y * oo.x;
                    p.y = bc.x * io.y + bc.y * oo.y;
                }
                sts_row(tk.sP + 512u * r, p);
            }
        }
        if (UPD) {
            // the update of the last window is still owed to these rows (see transform_p_rows)
            __syncwarp();
            if (!t_ready) stage_T();
            transform_p_rows(a, sb, sT, len, lane);
            __syncwarp();
            for (int e = __ldg(a.gfix_off + task), e1 = __ldg(a.gfix_off + task + 1); e < e1; ++e) {
                const int2 x = __ldg(a.gfix + e);
                const int rl = x.x & 0xffff;
                const double2 bc = lds_row(tk.sRec + kRec * rl + 16u);
                const double q = ((x.x >> 16) ? bc.x : bc.y) * __ldg(a.upQs + x.y);
                if (active) {
                    const double* wr = a.upW + (size_t)x.y * a.M;
                    double2 pv = lds_row(tk.sP + 512u * rl);
                    if (col < a.M) pv.x += q * __ldg(wr + col);
                    if (col + 1 < a.M) pv.y += q * __ldg(wr + col + 1);
                    sts_row(tk.sP + 512u * rl, pv);
                }
            }
            __syncwarp();
            if (REC && (a.rec_prior || a.rec_post)) record_posterior(a, tk.sRec, sT, task, td.begin, len, lane);
        }
        // rows of other tasks consumed through the input ring, in consumption order: byte offsets of their slots
        int nL = 0;
        for (int base = 0; base < td.n_words; base += 32) {
            const int i = base + lane;
            const uint32_t w = i < td.n_words ? lds_u32(tk.sWords + 4u * i) : 0u;
            const bool is = (w & WIN_SLOT) != 0u && i >= td.n_in;
            const unsigned m = __ballot_sync(0xffffffffu, is);
            if (is) sts_u32(tk.sList + 4u * (nL + __popc(m & ((1u << lane) - 1u))), (w & kIdMask) * (unsigned)(ld * sizeof(double)));
            nL += __popc(m);
        }
        __syncwarp();
        tk.nL = nL;
        int cur_r0 = -1, cur_r1 = -1;
        if (tr && lane == 0) tr[1] = globaltimer_ns();
        // per-step forcing weights of this lane's two members: (w0*mul[r0][m], w1*mul[r1][m]), muskingum.py:528-531
        auto load_fctx = [&](int s) -> FCtx {
            FCtx c;
            c.w0 = c.w1 = 0.0; c.wm0 = c.wm1 = make_double2(0.0, 0.0);
            if (HAS_F) {
                const int2 rr = step_rows(s);
                const int r0 = rr.x, r1 = rr.y;
                const double2 ww = step_weights(s);
                c.w0 = ww.x; c.w1 = ww.y;
                if (HAS_W) {
                    const int c0 = min(col, a.wm_ld - 1), c1 = min(col + 1, a.wm_ld - 1);
                    const double* m0 = a.Wmul + (size_t)r0 * a.wm_ld;
                    const double* m1 = a.Wmul + (size_t)r1 * a.wm_ld;
                    c.wm0 = make_double2(c.w0 * __ldg(m0 + c0), c.w0 * __ldg(m0 + c1));
                    c.wm1 = make_double2(c.w1 * __ldg(m1 + c0), c.w1 * __ldg(m1 + c1));
                }
            }
            return c;
        };
        FCtx fc_next = load_fctx(0);
        const bool seg = td.kind == WTASK_SEG;
        const unsigned ring_sa = seg ? tk.sScr : tk.sIn;
        InStream ist;
        ist.in_flight = 0; ist.pi = ist.ci = 0; ist.slot_i = ist.slot_c = 0u; ist.dead = false;
        ist.psteps = nL > 0 ? a.nsteps : 0;
        ist.pbase = reinterpret_cast<char*>(a.ring + ccol);
        ist.cbase = ist.pbase;
        for (int j = 0; j < (seg ? SR : IR) && ist.psteps > 0; ++j) {
            if (seg) stream_issue<SR>(ist, a, ring_sa, tk.sList, nL, tk.step_bytes, active);
            else stream_issue<IR>(ist, a, ring_sa, tk.sList, nL, tk.step_bytes, active);
        }

        for (int s = 0; s < a.nsteps; ++s) {
            const bool last = s + 1 == a.nsteps;                   // outflows and inflows go to global memory
            char* ringS = reinterpret_cast<char*>(a.ring + ccol) + (size_t)s * tk.step_bytes;
            const FCtx fc = fc_next;
            int rj = -1;                                          // index of this step in rec_out, if it is recorded
            if (REC) {
                const long long gs = a.rec_step_base + s + 1;
                if (gs % a.rec_every == 0) rj = (int)(gs / a.rec_every - 1);
            }
            if (HAS_F) {
                const int2 rr = step_rows(s);
                const int r0 = rr.x, r1 = rr.y;
                if (r0 != cur_r0 || r1 != cur_r1) {              // a new bracket of the forcing table
                    const double* F0 = a.F + (size_t)r0 * a.n + td.begin;
                    const double* F1 = a.F + (size_t)r1 * a.n + td.begin;
                    __syncwarp();
                    // the rows are stored multiplied by gamma: o' = alpha*inflow + (p + c0*(gamma f0) + c1*(gamma f1))
                    for (int i = lane; i < len; i += 32) {
                        const double ga = a.coef[4 * (size_t)(td.begin + i) + 3];
                        sts_row(tk.sRec + kRec * i + 32u, make_double2(ga * __ldg(F0 + i), ga * __ldg(F1 + i)));
                    }
                    __syncwarp();
                    cur_r0 = r0; cur_r1 = r1;
                }
                if (!last) fc_next = load_fctx(s + 1);           // in flight during this step
            }
            if (!seg) {
                if (last) pocket_step<true, HAS_F, HAS_W, IR, REC>(a, tk, ist, fc, ringS, rj);
                else pocket_step<false, HAS_F, HAS_W, IR, REC>(a, tk, ist, fc, ringS, rj);
                if (tr && lane == 0) tr[4 + s] = globaltimer_ns();
            } else {
                unsigned long long* trs = tr ? tr + 4 + s : nullptr;
                if (last) segment_step<true, HAS_F, HAS_W, SR, REC>(a, tk, ist, fc, ringS, td.out_slot, trs, rj);
                else segment_step<false, HAS_F, HAS_W, SR, REC>(a, tk, ist, fc, ringS, td.out_slot, trs, rj);
            }
            if (ist.dead) break;
        }
        cp_async_wait_all();
        if (tr && lane == 0) {
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            tr[2] = globaltimer_ns();
            tr[3] = ((unsigned long long)smid << 8) | (unsigned)td.kind;
        }
        __syncwarp();
    }
    // the last warp to leave re-arms the ticket for the next launch on this handle
    if (lane == 0) {
        __threadfence();
        if (atomicAdd(a.done, 1ull) + 1ull == (unsigned long long)gridDim.x * (blockDim.x >> 5)) {
            *a.done = 0ull;
            *a.ticket = 0ull;
        }
    }
}

// ticket and the forcing interpolation of the launch's steps (see dataflow_init_kernel)
__global__ void __launch_bounds__(256) window_init_kernel(const InitArgs a, unsigned long long* ticket)
{
    const long long gid0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    if (gid0 == 0) *ticket = 0ull;
    if (a.times) {
        for (long long s = gid0; s < a.nsteps; s += stride) {
            const StepInterp si = interp_step(a.times, a.R, (double)(a.t0_ns + (a.step_base + s + 1) * a.dt_ns), a.method);
            a.steps_out[s] = si;
        }
    }
}

template <bool REC>
auto pick_window_kernel(bool f, bool w, bool u) -> void (*)(const WinArgs)
{
    if (!f) return u ? route_window_kernel<false, false, true, REC> : route_window_kernel<false, false, false, REC>;
    if (!w) return u ? route_window_kernel<true, false, true, REC> : route_window_kernel<true, false, false, REC>;
    return u ? route_window_kernel<true, true, true, REC> : route_window_kernel<true, true, false, REC>;
}

}  // namespace

cudaError_t launch_window_init(const InitArgs& a, unsigned long long* ticket, cudaStream_t st)
{
    window_init_kernel<<<1, 256, 0, st>>>(a, ticket);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_route_window(const WinArgs& a, int warps_per_cta, int num_sms, cudaStream_t st)
{
    const size_t smem = (size_t)a.off_steps + 16 * 24;          // [per-warp areas][T + counter (update variant)][step records]
    (void)warps_per_cta;
    static const bool pdl = [] { const char* k = getenv("TXH_PDL"); return !(k && atoi(k) == 0); }();
    const bool f = a.F != nullptr, w = a.Wmul != nullptr;
    const bool u = a.upT != nullptr;
    void (*kern)(const WinArgs) = a.rec_slot ? pick_window_kernel<true>(f, w, u) : pick_window_kernel<false>(f, w, u);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const long long pairs = (long long)a.n_tasks * a.n_mblocks;
    long long want = (pairs + warps_per_cta - 1) / warps_per_cta;
    const unsigned grid = (unsigned)(want < num_sms ? (want < 1 ? 1 : want) : num_sms);   // one resident CTA per SM
    (void)want;
    if (u) {
        // the launch that applies an update may overlap the tail of the kernel that computes it (see stage_T)
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(warps_per_cta * 32); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute attr{};
        attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr.val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
        cfg.attrs = &attr; cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, kern, a);
        count_launch();
        return e != cudaSuccess ? e : cudaGetLastError();
    }
    kern<<<grid, warps_per_cta * 32, smem, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

}  // namespace txh
