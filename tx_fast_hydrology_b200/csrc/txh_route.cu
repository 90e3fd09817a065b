// txh_route.cu -- routing kernels for sm_100a.
//
// The per-timestep Muskingum update  o = alpha*i_next + beta*i_prev + chi*o_prev + gamma*q,
// i_next[down] += o  (tx_fast_hydrology/nutils.py:64-89) is a sparse unit-lower-triangular
// solve per step.  route_dataflow_kernel evaluates `nsteps` of them in ONE persistent
// launch: the network is cut into tasks (pure-chain spine segments and bundled side
// subtrees, txh_topology.cpp); warps claim (step, task, member-block) tickets in a
// topological, critical-path-first order and synchronise point-to-point through
// per-task step counters in global memory -- no grid-wide barrier, so consecutive
// timesteps overlap along the network (time skewing) while every dependency of the
// reference's walk is honoured.  Ensemble members are the SIMD axis: a lane owns two
// adjacent member columns (one 128-bit access per row), so a thread only ever
// reads values of its own columns and intra-task hand-offs need no synchronisation.
#include "txh_device.cuh"

#include <atomic>

namespace txh {

static std::atomic<int64_t> g_launches{0};
int64_t launch_count() { return g_launches.load(); }
void count_launch() { g_launches++; }

namespace {

constexpr int kRing = 12;     // rows in flight per warp and state array (cp.async ring in shared memory)
constexpr int kRingPre = 6;   // PRE tasks stream four arrays (I, O, two side rows): 4 x 6 == 2 x 12 slots

__device__ __forceinline__ void fence_acq_rel() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }

// Per-warp shared-memory staging of one task's per-reach metadata: filled once per task by
// asynchronous global->shared copies (LDGSTS), read back as broadcast LDS in the reach loop,
// so no reach pays an L2 round trip for its coefficients, header, forcing or input words.
struct Stage {
    unsigned coef;           // shared-window byte addresses: [len][4] doubles
    unsigned f0, f1;         // [len] doubles
    unsigned hdr;            // [len] words
    unsigned inw;            // the task's input words, when they fit
    const uint32_t* inw_g;   // ... else read from global memory
    __device__ __forceinline__ double al(int i) const { return lds_f64(coef + 32u * i); }
    __device__ __forceinline__ double be(int i) const { return lds_f64(coef + 32u * i + 8u); }
    __device__ __forceinline__ double ch(int i) const { return lds_f64(coef + 32u * i + 16u); }
    __device__ __forceinline__ double ga(int i) const { return lds_f64(coef + 32u * i + 24u); }
    __device__ __forceinline__ uint32_t h(int i) const { return lds_u32(hdr + 4u * i); }
    __device__ __forceinline__ uint32_t word(int t) const { return inw_g ? __ldg(inw_g + t) : lds_u32(inw + 4u * t); }
};

struct StepCtx {
    double w0, w1;
    double2 wm0, wm1;
};

template <bool HAS_F, bool HAS_W>
__device__ __forceinline__ double2 forcing_q(const StepCtx& c, const Stage& st, int i)
{
    double2 q = make_double2(0.0, 0.0);
    if (HAS_F) {
        const double f0 = lds_f64(st.f0 + 8u * i), f1 = lds_f64(st.f1 + 8u * i);
        if (HAS_W) { q.x = c.wm0.x * f0 + c.wm1.x * f1; q.y = c.wm0.y * f0 + c.wm1.y * f1; }
        else { q.x = c.w0 * f0 + c.w1 * f1; q.y = q.x; }
    }
    return q;
}

template <bool REC>
__device__ __forceinline__ void record(const RouteArgs& a, int k, int s, int col, double2 on)
{
    if (REC) {
        const int rs = a.rec_slot[k];
        const long long gs = a.rec_step_base + s + 1;
        if (rs >= 0 && (gs % a.rec_every) == 0 && col < a.M) {
            double* dst = a.rec_out + ((size_t)(gs / a.rec_every - 1) * a.rec_count + rs) * a.M + col;
            dst[0] = on.x;
            if (col + 1 < a.M) dst[1] = on.y;
        }
    }
}

// Row streaming.  A task's I / O rows are contiguous (schedule order), so the warp keeps the next
// kRing rows of both arrays in flight with asynchronous global->shared copies; every lane copies and
// later reads back only its own 16-byte cell (its two member columns), so completion is tracked
// per thread with cp.async groups: one group per row, committed even when empty.
// ring cell address: ring + ((arr * D + slot) * 32 + lane) * 16, `ring` already includes the lane term.

// POCKET: a bundle of side subtrees evaluated depth-first by one warp.  Intermediate
// outflows travel through the accumulator or this lane's scratch column.
template <bool HAS_F, bool HAS_W, bool REC>
__device__ __forceinline__ void run_pocket(const RouteArgs& a, const TaskDesc& td, const Stage& st, int s, int col,
                                           bool active, double2* scratch, const StepCtx& sc, unsigned ring)
{
    const int ld = a.ld, len = td.len;
    const int ccol = active ? col : 0;
    double* Ob = a.O + ccol;
    double* Or = Ob + (size_t)td.begin * ld;
    double* Ir = a.I + ccol + (size_t)td.begin * ld;
    const unsigned ringO = ring + kRing * 512u;
#pragma unroll
    for (int j = 0; j < kRing; ++j) {
        if (active && j < len) { cp_async16(ring + j * 512u, Ir + (size_t)j * ld); cp_async16(ringO + j * 512u, Or + (size_t)j * ld); }
        cp_async_commit();
    }
    cp_async_wait_group<kRing>();                       // this thread's share of the staged metadata ...
    __syncwarp();                                       // ... and every other lane's
    int wi = 0, sl = 0;
    double2 acc = make_double2(0.0, 0.0);
    for (int i = 0; i < len; ++i) {
        cp_async_wait_group<kRing - 1>();               // row i has landed
        const double2 io = lds_row(ring + sl * 512u), oo = lds_row(ringO + sl * 512u);
        if (active && i + kRing < len) {
            cp_async16(ring + sl * 512u, Ir + (size_t)(i + kRing) * ld);
            cp_async16(ringO + sl * 512u, Or + (size_t)(i + kRing) * ld);
        }
        cp_async_commit();
        sl = sl + 1 == kRing ? 0 : sl + 1;
        const uint32_t h = st.h(i);
        const double al = st.al(i), be = st.be(i), ch = st.ch(i), ga = st.ga(i);
        double2 inflow = (h & HDR_ACC) ? acc : make_double2(0.0, 0.0);
        const int nin = (int)((h >> 6) & 0x1ffffffu);
        for (int t = 0; t < nin; ++t) {
            const uint32_t w = st.word(wi++);
            double2 v;
            if (w & INW_ROW) v = active ? ld_row(Ob + (size_t)(w & ~INW_ROW) * ld) : make_double2(0.0, 0.0);
            else v = scratch[w * 32];
            inflow.x += v.x; inflow.y += v.y;
        }
        const double2 q = forcing_q<HAS_F, HAS_W>(sc, st, i);
        double2 on;
        on.x = al * inflow.x + (be * io.x + ch * oo.x + ga * q.x);
        on.y = al * inflow.y + (be * io.y + ch * oo.y + ga * q.y);
        if (active) { st_row(Ir + (size_t)i * ld, inflow); st_row(Or + (size_t)i * ld, on); }
        if (h & HDR_PUSH) {                             // pocket root: hand the outflow to the spine's side slab
            const uint32_t sidx = st.word(wi++);
            if (active) st_row(a.Side + (size_t)sidx * ld + ccol, on);
        }
        const uint32_t slot = (h >> 1) & 31u;
        if (slot) scratch[(slot - 1) * 32] = on;
        acc = on;
        record<REC>(a, td.begin + i, s, col, on);
    }
    cp_async_wait_all();
}

// PRE: one spine segment -- sums the side inflow pushed by the pocket roots (a contiguous slab
// of the side buffer, consumed in order), folds the old state and the forcing into
// r = beta*i_prev + chi*o_prev + gamma*q, and runs the segment's recurrence with no flow entering
// it:  B_k = alpha_k (B_{k-1} + side_k) + r_k.  (side_k, B_k) are parked in the segment's own I / O
// rows.  State rows and the first two side rows of every reach travel through the ring.
template <bool HAS_F, bool HAS_W>
__device__ __forceinline__ void run_pre(const RouteArgs& a, const TaskDesc& td, const Stage& st, int col, bool active,
                                        const StepCtx& sc, unsigned ring)
{
    const int ld = a.ld, len = td.len;
    const int ccol = active ? col : 0;
    double* Or = a.O + ccol + (size_t)td.begin * ld;
    double* Ir = a.I + ccol + (size_t)td.begin * ld;
    const double* Sr = a.Side + ccol + (size_t)td.side_off * ld;
    const unsigned ringO = ring + kRingPre * 512u, ringG = ring + 2 * kRingPre * 512u, ringH = ring + 3 * kRingPre * 512u;
    cp_async_wait_all();                                // the side-row counts come from the staged headers
    __syncwarp();
    int cq = 0;                                         // side-row cursor of the prefetcher
#pragma unroll
    for (int j = 0; j < kRingPre; ++j) {
        if (j < len) {
            const int nin = (int)((st.h(j) >> 6) & 0x1fffu);
            if (active) {
                cp_async16(ring + j * 512u, Ir + (size_t)j * ld); cp_async16(ringO + j * 512u, Or + (size_t)j * ld);
                if (nin > 0) cp_async16(ringG + j * 512u, Sr + (size_t)cq * ld);
                if (nin > 1) cp_async16(ringH + j * 512u, Sr + (size_t)(cq + 1) * ld);
            }
            cq += nin;
        }
        cp_async_commit();
    }
    int ci = 0, sl = 0;
    double2 B = make_double2(0.0, 0.0);
    for (int i = 0; i < len; ++i) {
        cp_async_wait_group<kRingPre - 1>();
        const uint32_t h = st.h(i);
        const int nin = (int)((h >> 6) & 0x1fffu);
        const double2 io = lds_row(ring + sl * 512u), oo = lds_row(ringO + sl * 512u);
        double2 side = nin > 0 ? lds_row(ringG + sl * 512u) : make_double2(0.0, 0.0);
        if (nin > 1) { const double2 v = lds_row(ringH + sl * 512u); side.x += v.x; side.y += v.y; }
        const int ip = i + kRingPre;
        if (ip < len) {
            const int np = (int)((st.h(ip) >> 6) & 0x1fffu);
            if (active) {
                cp_async16(ring + sl * 512u, Ir + (size_t)ip * ld); cp_async16(ringO + sl * 512u, Or + (size_t)ip * ld);
                if (np > 0) cp_async16(ringG + sl * 512u, Sr + (size_t)cq * ld);
                if (np > 1) cp_async16(ringH + sl * 512u, Sr + (size_t)(cq + 1) * ld);
            }
            cq += np;
        }
        cp_async_commit();
        sl = sl + 1 == kRingPre ? 0 : sl + 1;
        for (int t = 2; t < nin; ++t) {
            if (active) {
                const double2 v = ld_row(Sr + (size_t)(ci + t) * ld);
                side.x += v.x; side.y += v.y;
            }
        }
        ci += nin;
        const double al = st.al(i), be = st.be(i), ch = st.ch(i), ga = st.ga(i);
        const double2 q = forcing_q<HAS_F, HAS_W>(sc, st, i);
        double2 inflow = side;
        if (h & HDR_ACC) { inflow.x += B.x; inflow.y += B.y; }
        B.x = al * inflow.x + (be * io.x + ch * oo.x + ga * q.x);
        B.y = al * inflow.y + (be * io.y + ch * oo.y + ga * q.y);
        if (active) { st_row(Ir + (size_t)i * ld, side); st_row(Or + (size_t)i * ld, B); }
    }
    cp_async_wait_all();
}

// LINK: one long path.  Walks its segments in order; the flow entering a segment is the previous
// segment's outflow plus the outlets of the long tributaries joining there, and the segment's
// outflow is  out = A_last * o_in + B_last  (B_last parked by PRE in the segment's last O row,
// A_last staged from linkA).  Writes the final outflow of every segment's last reach.
template <bool REC>
__device__ __forceinline__ void run_link(const RouteArgs& a, const TaskDesc& td, const Stage& st, int s, int col,
                                         bool active, unsigned ring)
{
    const int ld = a.ld, len = td.len;
    const int ccol = active ? col : 0;
    double* Ob = a.O + ccol;
    const unsigned ringG = ring + kRing * 512u;
    cp_async_wait_all();                                // records and A_last come from the staging area
    __syncwarp();
    int wq = 0;
#pragma unroll
    for (int j = 0; j < kRing; ++j) {
        if (j < len) {
            const uint32_t last = st.word(wq) & ~INW_ROW;
            const int nl = (int)st.word(wq + 1);
            if (active) {
                cp_async16(ring + j * 512u, Ob + (size_t)last * ld);
                if (nl > 0) cp_async16(ringG + j * 512u, Ob + (size_t)(st.word(wq + 2) & ~INW_ROW) * ld);
            }
            wq += 2 + nl;
        }
        cp_async_commit();
    }
    int wi = 0, sl = 0;
    double2 o = make_double2(0.0, 0.0);
    for (int j = 0; j < len; ++j) {
        cp_async_wait_group<kRing - 1>();
        const uint32_t last = st.word(wi) & ~INW_ROW;
        const int nl = (int)st.word(wi + 1);
        const double2 B = lds_row(ring + sl * 512u);
        double2 oin = o;
        if (nl > 0) { const double2 v = lds_row(ringG + sl * 512u); oin.x += v.x; oin.y += v.y; }
        for (int t = 1; t < nl; ++t) {
            if (active) {
                const double2 v = ld_row(Ob + (size_t)(st.word(wi + 2 + t) & ~INW_ROW) * ld);
                oin.x += v.x; oin.y += v.y;
            }
        }
        wi += 2 + nl;
        if (j + kRing < len) {
            const uint32_t lastp = st.word(wq) & ~INW_ROW;
            const int np = (int)st.word(wq + 1);
            if (active) {
                cp_async16(ring + sl * 512u, Ob + (size_t)lastp * ld);
                if (np > 0) cp_async16(ringG + sl * 512u, Ob + (size_t)(st.word(wq + 2) & ~INW_ROW) * ld);
            }
            wq += 2 + np;
        }
        cp_async_commit();
        sl = sl + 1 == kRing ? 0 : sl + 1;
        const double A = lds_f64(st.f0 + 8u * j);
        o.x = A * oin.x + B.x;
        o.y = A * oin.y + B.y;
        if (active) st_row(Ob + (size_t)last * ld, o);
        record<REC>(a, (int)last, s, col, o);
    }
    cp_async_wait_all();
}

// FIX: one spine segment, every reach independent:  o_k = B_k + A_k * o_in,  i_k = o_{k-1} + side_k,
// with o_in the flow entering the segment (rows listed in the task's stream) and A_k the prefix
// product of alpha from the segment's first reach (staged from cumA).  The last row already holds
// its final outflow (LINK).
template <bool REC>
__device__ __forceinline__ void run_fix(const RouteArgs& a, const TaskDesc& td, const Stage& st, int s, int col,
                                        bool active, unsigned ring)
{
    const int ld = a.ld, len = td.len;
    const int ccol = active ? col : 0;
    double* Ob = a.O + ccol;
    double* Or = Ob + (size_t)td.begin * ld;
    double* Ir = a.I + ccol + (size_t)td.begin * ld;
    const unsigned ringO = ring + kRing * 512u;
#pragma unroll
    for (int j = 0; j < kRing; ++j) {
        if (active && j < len) { cp_async16(ring + j * 512u, Ir + (size_t)j * ld); cp_async16(ringO + j * 512u, Or + (size_t)j * ld); }
        cp_async_commit();
    }
    cp_async_wait_group<kRing>();
    __syncwarp();
    double2 oin = make_double2(0.0, 0.0);
    for (int t = 0; t < td.n_words; ++t) {
        if (active) {
            const double2 v = ld_row(Ob + (size_t)(st.word(t) & ~INW_ROW) * ld);
            oin.x += v.x; oin.y += v.y;
        }
    }
    int sl = 0;
    double2 op = oin;
    for (int i = 0; i < len; ++i) {
        cp_async_wait_group<kRing - 1>();
        const double2 side = lds_row(ring + sl * 512u), B = lds_row(ringO + sl * 512u);
        if (active && i + kRing < len) {
            cp_async16(ring + sl * 512u, Ir + (size_t)(i + kRing) * ld);
            cp_async16(ringO + sl * 512u, Or + (size_t)(i + kRing) * ld);
        }
        cp_async_commit();
        sl = sl + 1 == kRing ? 0 : sl + 1;
        double2 it, on = B;
        it.x = op.x + side.x;
        it.y = op.y + side.y;
        if (i + 1 < len) {
            const double A = lds_f64(st.f0 + 8u * i);
            on.x = A * oin.x + B.x;
            on.y = A * oin.y + B.y;
            if (active) st_row(Or + (size_t)i * ld, on);
            record<REC>(a, td.begin + i, s, col, on);
        }
        if (active) st_row(Ir + (size_t)i * ld, it);
        op = on;
    }
    cp_async_wait_all();
}

// Prepares the dataflow runtime for one launch: the ready queue cleared and seeded with every task that
// has no same-step producer, the dependency counters, and the forcing interpolation of every step of the
// launch -- nutils.py:21-34 evaluated in float64 exactly as the reference does (searchsorted-left,
// clamped ends; x = float(next_timestep.value), muskingum.py:528-530).  Queue entry = (step << 32) | (pair + 1).
__global__ void __launch_bounds__(256) dataflow_init_kernel(const InitArgs a)
{
    const long long gid0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long pairs = (long long)a.n_tasks * a.n_mblocks;
    const long long seeded = (long long)a.n_init * a.n_mblocks;
    for (long long gid = gid0; gid < a.queue_entries; gid += stride) {
        unsigned long long e = 0ull;
        if (gid < seeded) {
            const int t = a.init_ready[gid / a.n_mblocks];
            e = (unsigned long long)(t * a.n_mblocks + gid % a.n_mblocks) + 1ull;
        }
        a.queue[gid] = e;
    }
    for (long long gid = gid0; gid < pairs; gid += stride) a.pending[gid] = a.tasks[gid / a.n_mblocks].need0;
    if (a.times) {
        for (long long s = gid0; s < a.nsteps; s += stride) {
            const double x = (double)(a.t0_ns + (a.step_base + s + 1) * a.dt_ns);
            int lo = 0, hi = a.R;                                   // np.searchsorted(xp, x), side='left'
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (a.times[mid] < x) lo = mid + 1; else hi = mid;
            }
            StepInterp si;
            if (lo == 0) { si.r0 = 0; si.r1 = 0; si.w0 = 1.0; si.w1 = 0.0; }
            else if (lo >= a.R) { si.r0 = a.R - 1; si.r1 = a.R - 1; si.w0 = 1.0; si.w1 = 0.0; }
            else {
                const double dx_0 = __dsub_rn(x, a.times[lo - 1]), dx_1 = __dsub_rn(a.times[lo], x);
                if (a.method == 1) {
                    const double frac = __ddiv_rn(dx_0, __dadd_rn(dx_0, dx_1));
                    si.r0 = lo - 1; si.r1 = lo; si.w0 = __dsub_rn(1.0, frac); si.w1 = frac;
                } else {
                    const int r = fabs(dx_0) <= fabs(dx_1) ? lo - 1 : lo;
                    si.r0 = r; si.r1 = r; si.w0 = 1.0; si.w1 = 0.0;
                }
            }
            a.steps_out[s] = si;
        }
    }
    if (gid0 == 0) {
        a.q_head[0] = 0ull;
        a.q_head[1] = (unsigned long long)seeded;
        a.q_head[2] = 0ull;     // completed tasks
    }
}

template <bool HAS_F, bool HAS_W, bool REC>
__global__ void __launch_bounds__(kWarpsPerCta * 32, 3)
route_dataflow_kernel(const RouteArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_all[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    unsigned char* wbase = smem_all + (size_t)warp * a.smem_per_warp;
    double2* scratch = reinterpret_cast<double2*>(wbase) + lane;            // this lane's column of every slot
    const unsigned sbase = (unsigned)__cvta_generic_to_shared(wbase);
    const int nmb = a.n_mblocks;
    unsigned long long* q_tail = a.q_head + 1;
    unsigned long long* n_done = a.q_head + 2;
    const long long pairs = (long long)a.n_tasks * nmb;

    if (ld_relaxed_s32(a.status) != 0) return;          // a previous launch on this handle was poisoned

    long long next_entry = 0;                       // task made ready by this warp: run it without queueing
    for (;;) {
        unsigned long long t_pop = 0;
        if (a.trace && lane == 0) t_pop = globaltimer_ns();
        long long entry = next_entry;
        next_entry = 0;
        if (entry == 0) {
            // ---- pop: claim a queue position, wait until its producer has published it ----
            if (lane == 0) {
                const unsigned long long idx = atomicAdd(a.q_head, 1ull);
                entry = -1;
                if ((long long)idx < a.total) {
                    const unsigned long long* slot = a.queue + idx;
                    unsigned spins = 0, nap = 64;
                    unsigned long long t0 = 0;
                    for (;;) {
                        unsigned long long v;
                        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(slot) : "memory");
                        if (v != 0ull) { entry = (long long)v; break; }
                        if ((++spins & 15u) == 0) {
                            unsigned long long fin;
                            asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(fin) : "l"(n_done) : "memory");
                            if ((long long)fin >= a.total) break;           // everything ran (inline continuations skip the queue)
                            if (ld_relaxed_s32(a.status) != 0) break;
                            const unsigned long long now = globaltimer_ns();
                            if (t0 == 0) t0 = now;
                            else if (now - t0 > a.watchdog_ns) { atomicExch(a.status, 1); break; }
                        }
                        __nanosleep(nap);
                        if (nap < 1024u) nap <<= 1;
                    }
                    if (entry > 0) fence_acq_rel();                          // acquire: the producers' rows are visible
                }
            }
            entry = __shfl_sync(0xffffffffu, entry, 0);
            if (entry <= 0) break;
        }
        const int pair = (int)((unsigned long long)entry & 0xffffffffull) - 1;
        const int s = (int)((unsigned long long)entry >> 32);
        const int task = pair / nmb;
        const int mb = pair - task * nmb;
        const TaskDesc td = a.tasks[task];
        unsigned long long t_begin = 0;
        if (a.trace && lane == 0) t_begin = globaltimer_ns();

        // ---- stage the task's metadata in shared memory (asynchronous copies) ----------------
        StepInterp si;
        si.r0 = si.r1 = 0; si.w0 = si.w1 = 0.0;
        Stage st;
        const bool walks = td.kind == TASK_POCKET || td.kind == TASK_PRE;     // evaluates the Muskingum update itself
        const bool link = td.kind == TASK_LINK;
        // LINK tasks lay the staging area out differently: [A_last per segment][records]
        const int off_f0 = link ? a.off_coef : a.off_f0;
        const int off_inw = link ? a.off_inw_link : a.off_inw;
        const int cap_words = link ? a.max_words_link : a.max_words;
        st.coef = sbase + a.off_coef; st.f0 = sbase + off_f0; st.f1 = sbase + a.off_f1;
        st.hdr = sbase + a.off_hdr; st.inw = sbase + off_inw; st.inw_g = nullptr;
        {
            if (td.n_words <= cap_words)
                for (int i = lane; i < td.n_words; i += 32) cp_async4(wbase + off_inw + 4 * i, a.inw + td.in_off + i);
            else
                st.inw_g = a.inw + td.in_off;
            if (walks) {
                const double* gc = a.coef + 4 * (size_t)td.begin;
                for (int i = lane; i < 2 * td.len; i += 32) cp_async16(wbase + a.off_coef + 16 * i, gc + 2 * i);
                for (int i = lane; i < td.len; i += 32) cp_async4(wbase + a.off_hdr + 4 * i, a.hdr + td.begin + i);
                if (HAS_F) {
                    si = a.steps[s];
                    const double* F0 = a.F + (size_t)si.r0 * a.n + td.begin;
                    const double* F1 = a.F + (size_t)si.r1 * a.n + td.begin;
                    for (int i = lane; i < td.len; i += 32) {
                        cp_async8(wbase + a.off_f0 + 8 * i, F0 + i);
                        cp_async8(wbase + a.off_f1 + 8 * i, F1 + i);
                    }
                }
            } else {
                // prefix products of alpha: per reach of the segment (FIX) / per segment of the path (LINK)
                const double* ga = (link ? a.linkA : a.cumA) + td.begin;
                for (int i = lane; i < td.len; i += 32) cp_async8(wbase + off_f0 + 8 * i, ga + i);
            }
        }
        const int col = mb * kMemberBlock + lane * 2;
        const bool active = col < a.ld;
        StepCtx sc;
        sc.w0 = si.w0; sc.w1 = si.w1; sc.wm0 = sc.wm1 = make_double2(0.0, 0.0);
        if (HAS_F && HAS_W && walks) {
            // member m sees  (w0*mul[r0][m])*F[r0] + (w1*mul[r1][m])*F[r1]
            const int c0 = min(col, a.wm_ld - 1), c1 = min(col + 1, a.wm_ld - 1);
            const double* m0 = a.Wmul + (size_t)si.r0 * a.wm_ld;
            const double* m1 = a.Wmul + (size_t)si.r1 * a.wm_ld;
            sc.wm0 = make_double2(si.w0 * __ldg(m0 + c0), si.w0 * __ldg(m0 + c1));
            sc.wm1 = make_double2(si.w1 * __ldg(m1 + c0), si.w1 * __ldg(m1 + c1));
        }
        cp_async_commit();                              // group 0 of this task: the staged metadata
        const unsigned ring = sbase + a.off_ring + lane * 16u;
        if (td.kind == TASK_POCKET) run_pocket<HAS_F, HAS_W, REC>(a, td, st, s, col, active, scratch, sc, ring);
        else if (td.kind == TASK_PRE) run_pre<HAS_F, HAS_W>(a, td, st, col, active, sc, ring);
        else if (td.kind == TASK_LINK) run_link<REC>(a, td, st, s, col, active, ring);
        else run_fix<REC>(a, td, st, s, col, active, ring);

        // ---- completion: re-arm, then notify dependants with release atomics -----------------
        unsigned long long t_comp = 0;
        if (a.trace && lane == 0) t_comp = globaltimer_ns();
        const bool more = s + 1 < a.nsteps;
        if (more && lane == 0) a.pending[pair] = td.need;   // nobody can signal step s+1 before the notifications below
        __syncwarp();                                        // every lane's rows + the re-arm precede the releases
        const int nn = td.n_same + (more ? td.n_next : 0);
        for (int d0 = 0; d0 < nn; d0 += 32) {
            const int d = d0 + lane;
            int tgt = -1;
            bool ready = false;
            if (d < nn) {
                tgt = a.notify[td.nfy_off + d] * nmb + mb;
                int old;
                // release: this task's rows precede the signal; acquire: a lane that completes the
                // dependant's count has the other contributors' rows ordered before the hand-off
                asm volatile("atom.acq_rel.gpu.global.add.s32 %0, [%1], -1;" : "=r"(old) : "l"(a.pending + tgt) : "memory");
                ready = old == 1;
            }
            const unsigned mask = __ballot_sync(0xffffffffu, ready);
            if (mask != 0u) {
                // entry of the dependant: same-step targets run step s, next-step targets step s + 1
                const long long e = ((long long)(d < td.n_same ? s : s + 1) << 32) | (long long)(unsigned)(tgt + 1);
                if (next_entry == 0) {
                    // keep one ready dependant for this warp (a LINK if there is one): no queue round trip
                    const bool is_chain = ready && a.tasks[tgt / nmb].kind == TASK_LINK;
                    const unsigned cm = __ballot_sync(0xffffffffu, is_chain);
                    const int keep = __ffs(cm ? cm : mask) - 1;
                    next_entry = __shfl_sync(0xffffffffu, e, keep);
                    if (lane == keep) ready = false;
                }
                const unsigned pm = __ballot_sync(0xffffffffu, ready);      // lanes that still have to queue theirs
                if (pm != 0u) {
                    unsigned long long base = 0;
                    const int leader = __ffs(pm) - 1;
                    if (lane == leader) base = atomicAdd(q_tail, (unsigned long long)__popc(pm));
                    base = __shfl_sync(0xffffffffu, base, leader);
                    if (ready) {
                        const unsigned long long idx = base + __popc(pm & ((1u << lane) - 1u));
                        asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(a.queue + idx), "l"(e) : "memory");
                    }
                }
            }
        }
        if (lane == 0) {
            atomicAdd(n_done, 1ull);
            if (a.trace) {
                const unsigned sm = smid();
                unsigned long long* tr = a.trace + 4 * ((size_t)s * pairs + pair);
                tr[0] = t_pop; tr[1] = t_begin; tr[2] = t_comp;
                tr[3] = (globaltimer_ns() << 16) | ((unsigned long long)(sm & 0xffu) << 8) | (unsigned)td.kind;
            }
        }
        __syncwarp();
    }
}

// One topological level of one step (independent second device path).
__global__ void __launch_bounds__(256) route_level_kernel(const LevelArgs a)
{
    const int half = (a.ld + 1) / 2;                          // double2 columns per row
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)a.count * half) return;
    const int r = (int)(gid / half);
    const int col = (int)(gid - (long long)r * half) * 2;
    const int k = a.lvl_pos[r];
    double2 inflow = make_double2(0.0, 0.0);
    for (int u = a.up_off[k]; u < a.up_off[k + 1]; ++u) {
        const double2 v = ld_row(a.O + (size_t)a.up_pos[u] * a.ld + col);
        inflow.x += v.x; inflow.y += v.y;
    }
    const double al = a.coef[4 * (size_t)k], be = a.coef[4 * (size_t)k + 1], ch = a.coef[4 * (size_t)k + 2],
                 ga = a.coef[4 * (size_t)k + 3];
    double* Orow = a.O + (size_t)k * a.ld + col;
    double* Irow = a.I + (size_t)k * a.ld + col;
    const double2 io = ld_row(Irow), oo = ld_row(Orow);
    const double q = a.q ? a.q[k] : 0.0;
    double2 on;
    on.x = al * inflow.x + (be * io.x + ch * oo.x + ga * q);
    on.y = al * inflow.y + (be * io.y + ch * oo.y + ga * q);
    st_row(Irow, inflow);
    st_row(Orow, on);
}

__global__ void __launch_bounds__(256)
init_inflows_kernel(const int32_t* up_off, const int32_t* up_pos, const uint8_t* is_outlet,
                    const double* O, double* I, long long n, int ld)
{
    const int half = (ld + 1) / 2;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n * half) return;
    const long long k = gid / half;
    const int col = (int)(gid - k * half) * 2;
    double2 s = make_double2(0.0, 0.0);
    for (int u = up_off[k]; u < up_off[k + 1]; ++u) {
        const double2 v = *reinterpret_cast<const double2*>(O + (size_t)up_pos[u] * ld + col);
        s.x += v.x; s.y += v.y;
    }
    if (is_outlet[k]) {      // muskingum.py:417 / nutils.py:136-141: no self-loop guard
        const double2 v = *reinterpret_cast<const double2*>(O + (size_t)k * ld + col);
        s.x += v.x; s.y += v.y;
    }
    *reinterpret_cast<double2*>(I + (size_t)k * ld + col) = s;
}

__global__ void __launch_bounds__(256)
apply_gain_kernel(const int32_t* up_off, const int32_t* up_pos, const double* G, double* O, double* I,
                  long long n, int ld)
{
    const int half = (ld + 1) / 2;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n * half) return;
    const long long k = gid / half;
    const int col = (int)(gid - k * half) * 2;
    double2 s = make_double2(0.0, 0.0);
    for (int u = up_off[k]; u < up_off[k + 1]; ++u) {
        const double2 v = *reinterpret_cast<const double2*>(G + (size_t)up_pos[u] * ld + col);
        s.x += v.x; s.y += v.y;
    }
    const double2 g = *reinterpret_cast<const double2*>(G + (size_t)k * ld + col);
    double2* op = reinterpret_cast<double2*>(O + (size_t)k * ld + col);
    double2* ip = reinterpret_cast<double2*>(I + (size_t)k * ld + col);
    double2 o = *op, i = *ip;
    o.x += g.x; o.y += g.y;
    i.x += s.x; i.y += s.y;
    *op = o; *ip = i;
}

__global__ void __launch_bounds__(256)
pack_kernel(const int32_t* reach_of_pos, const double* src, double* dst, long long n, int M, int ld,
            int src_member_major)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n * ld) return;
    const long long k = gid / ld;
    const int m = (int)(gid - k * ld);
    double v = 0.0;
    if (m < M) {
        const long long j = reach_of_pos[k];
        v = src_member_major ? src[(size_t)m * n + j] : src[(size_t)j * M + m];
    }
    dst[gid] = v;
}

__global__ void __launch_bounds__(256)
unpack_kernel(const int32_t* reach_of_pos, const double* src, double* dst, long long n, int M, int ld,
              int dst_member_major)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n * M) return;
    const long long k = gid / M;
    const int m = (int)(gid - k * M);
    const long long j = reach_of_pos[k];
    const double v = src[(size_t)k * ld + m];
    if (dst_member_major) dst[(size_t)m * n + j] = v; else dst[(size_t)j * M + m] = v;
}

__global__ void __launch_bounds__(256)
gather_rows_kernel(const int32_t* pos, long long count, const double* X, int ld, int M, double* out)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= count * M) return;
    const long long k = gid / M;
    const int m = (int)(gid - k * M);
    out[gid] = X[(size_t)pos[k] * ld + m];
}

// dst[r][k] = src[r][reach_of_pos[k]] for a row-major [R][n] table
__global__ void __launch_bounds__(256)
permute_rows_kernel(const int32_t* reach_of_pos, const double* src, double* dst, long long n, long long R)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n * R) return;
    const long long r = gid / n, k = gid - r * n;
    dst[gid] = src[r * n + reach_of_pos[k]];
}

__global__ void __launch_bounds__(256)
permute_vec_kernel(const int32_t* reach_of_pos, const double* src, double* dst, long long n)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid < n) dst[gid] = src[reach_of_pos[gid]];
}

}  // namespace

cudaError_t launch_dataflow_init(const InitArgs& a, cudaStream_t st)
{
    long long work = (long long)a.n_tasks * a.n_mblocks;
    if (a.queue_entries > work) work = a.queue_entries;
    unsigned blocks = nblk(work, 256);
    if (blocks > 1184u) blocks = 1184u;                       // grid-stride beyond 8 CTAs per SM
    dataflow_init_kernel<<<blocks, 256, 0, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_route_dataflow(const RouteArgs& a, int num_sms, cudaStream_t st)
{
    const size_t smem = (size_t)kWarpsPerCta * a.smem_per_warp;
    void (*kern)(const RouteArgs) = nullptr;
    const bool f = a.F != nullptr, w = a.Wmul != nullptr, r = a.rec_slot != nullptr;
    if (!f) kern = r ? route_dataflow_kernel<false, false, true> : route_dataflow_kernel<false, false, false>;
    else if (!w) kern = r ? route_dataflow_kernel<true, false, true> : route_dataflow_kernel<true, false, false>;
    else kern = r ? route_dataflow_kernel<true, true, true> : route_dataflow_kernel<true, true, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kWarpsPerCta * 32, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    const long long pairs = (long long)a.n_tasks * a.n_mblocks;
    long long want = (pairs + kWarpsPerCta - 1) / kWarpsPerCta;       // one step's worth of warps is plenty
    long long cap = (long long)num_sms * occ;
    const unsigned grid = (unsigned)(want < cap ? (want < 1 ? 1 : want) : cap);
    kern<<<grid, kWarpsPerCta * 32, smem, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_route_level(const LevelArgs& a, cudaStream_t st)
{
    const int half = (a.ld + 1) / 2;
    route_level_kernel<<<nblk((long long)a.count * half, 256), 256, 0, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_init_inflows(const int32_t* up_off, const int32_t* up_pos, const uint8_t* is_outlet,
                                const double* O, double* I, int64_t n, int ld, int M, cudaStream_t st)
{
    (void)M;
    init_inflows_kernel<<<nblk(n * ((ld + 1) / 2), 256), 256, 0, st>>>(up_off, up_pos, is_outlet, O, I, n, ld);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_apply_gain(const int32_t* up_off, const int32_t* up_pos, const double* G, double* O,
                              double* I, int64_t n, int ld, int M, cudaStream_t st)
{
    (void)M;
    apply_gain_kernel<<<nblk(n * ((ld + 1) / 2), 256), 256, 0, st>>>(up_off, up_pos, G, O, I, n, ld);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_pack(const int32_t* reach_of_pos, const double* src, double* dst, int64_t n, int M,
                        int ld, int src_member_major, cudaStream_t st)
{
    pack_kernel<<<nblk(n * ld, 256), 256, 0, st>>>(reach_of_pos, src, dst, n, M, ld, src_member_major);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_unpack(const int32_t* reach_of_pos, const double* src, double* dst, int64_t n, int M,
                          int ld, int dst_member_major, cudaStream_t st)
{
    unpack_kernel<<<nblk(n * M, 256), 256, 0, st>>>(reach_of_pos, src, dst, n, M, ld, dst_member_major);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_gather_rows(const int32_t* pos, int64_t count, const double* X, int ld, int M,
                               double* out, cudaStream_t st)
{
    gather_rows_kernel<<<nblk(count * M, 256), 256, 0, st>>>(pos, count, X, ld, M, out);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_permute_rows(const int32_t* reach_of_pos, const double* src, double* dst, int64_t n, int64_t R,
                                cudaStream_t st)
{
    permute_rows_kernel<<<nblk(n * R, 256), 256, 0, st>>>(reach_of_pos, src, dst, n, R);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_permute_vec(const int32_t* reach_of_pos, const double* src, double* dst, int64_t n,
                               cudaStream_t st)
{
    permute_vec_kernel<<<nblk(n, 256), 256, 0, st>>>(reach_of_pos, src, dst, n);
    count_launch();
    return cudaGetLastError();
}

}  // namespace txh
