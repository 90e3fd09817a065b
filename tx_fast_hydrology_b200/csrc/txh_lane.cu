// txh_lane.cu -- reach-parallel, time-skewed routing kernel for small ensembles (sm_100a).
//
// route_lane_kernel evaluates `nsteps` timesteps of the Muskingum update (tx_fast_hydrology/nutils.py:64-89,
// as called from muskingum.py:456 and the simulate loop muskingum.py:527-533) with LANES = REACHES.  It is the
// path for deterministic runs and small ensembles (M <= 16), where the member-per-lane window kernel
// (txh_window.cu) leaves 31 of 32 lanes idle.
//
// The network is cut into regions (LaneSchedule, txh_topology.cpp); a CTA claims a region and keeps its
// state in shared memory for every step of the launch.  Row j of a region evaluates timestep s in iteration
// k = s + off[j]; off decreases by one along every edge, so what a row needs from its upstream rows in
// iteration k was written in iteration k - 1: one __syncthreads per iteration, every row busy on its own
// timestep (time skewing: the 1,000-level dependency chain of a step costs nothing once the pipeline is
// full).  Per row and step:
//     inflow = sum of the upstream outflows               (shared-memory gathers, fixed child order)
//     o' = alpha*inflow + (p + gamma*q),   p' = beta*inflow + chi*o'      (p = beta*i + chi*o of the old state)
// Outflows crossing regions travel through streams ring[slot][member][step] in global memory: an unwritten
// cell holds EMPTY (all bits set); the consumer mirrors a stream as a virtual row, stays `lag` steps behind its
// producer so that its cp.async prefetches (two 8-step batches ahead) find data -- whenever it catches up it falls
// back by `lag` steps again -- and puts EMPTY back into every cell it has consumed.  Regions are claimed in a
// topological order, so a region only waits for regions that are running or done (every CTA is resident).
// The forcing is interpolated per step exactly as nutils.py:21-34 does; its bracket rows live in shared
// memory and the next row is prefetched (cp.async) one bracket ahead.
#include <algorithm>
#include <type_traits>

#include "txh_device.cuh"

namespace txh {

namespace {

__device__ __forceinline__ void bar_sync() { asm volatile("bar.sync 0;" ::: "memory"); }
__device__ __forceinline__ int bar_or(int pred)
{
    int r;
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.s32 q, %1, 0;\n\tbar.red.or.pred p, 0, q;\n\tselp.s32 %0, 1, 0, p;\n\t}"
                 : "=r"(r) : "r"(pred) : "memory");
    return r;
}

// Streams are read in batches of kBatch steps (64 bytes), prefetched TWO batches ahead with cp.async into a
// four-batch window in shared memory.  Producer and consumer regions advance at the same rate, so a consumer
// that started right behind its producer would find every prefetch EMPTY and pay a trip to L2 per step; it
// therefore waits once, before its first step, until the producer is `lag` steps ahead (or done), and every
// later prefetch lands on cells that are already written.
constexpr int kBatch = 8;
constexpr int kExtCells = 4 * kBatch;      // shared-memory window of a stream

// A new forcing bracket for a row: (pr0, pr1) -> (r0, r1).  f0, f1 are the rows of the old bracket at this reach,
// fn the row after them, requested when the old bracket was entered (a plain load whose register is not touched
// until now, a dozen iterations later: the latency is hidden without any wait); anything else (irregular tables,
// jumps of the nearest-row method) is read in place.
__device__ __forceinline__ void rotate_bracket(double& f0, double& f1, double& fn, const double* __restrict__ Fcol, int64_t n,
                                               int R, int pr0, int pr1, int r0, int r1)
{
    const int pn = min(max(pr0, pr1) + 1, R - 1);
    const double n0 = r0 == pr0 ? f0 : r0 == pr1 ? f1 : r0 == pn ? fn : __ldg(Fcol + (size_t)r0 * n);
    const double n1 = r1 == pr0 ? f0 : r1 == pr1 ? f1 : r1 == pn ? fn : __ldg(Fcol + (size_t)r1 * n);
    f0 = n0; f1 = n1;
    const int nn = min(max(r0, r1) + 1, R - 1);
    fn = nn == r0 ? n0 : nn == r1 ? n1 : __ldg(Fcol + (size_t)nn * n);
}

// One row (reach) per thread; everything a row needs every step -- coefficients, the forcing bracket, p = beta*i +
// chi*o of up to four members -- lives in REGISTERS for the whole launch.  Shared memory carries only what rows
// exchange: the outflows of this and the previous iteration (gathered by the downstream rows), the windows of the
// incoming streams, and the lists of children beyond the first two.  (A first version kept 64-byte row records in
// shared memory: their 128-bit loads at a 64-byte stride cost four times the ideal wavefronts and made the kernel
// shared-memory-bandwidth bound at ~5,000 cycles per iteration; profiles/r02_lane_kernel_history.md.)
template <int MT, bool HAS_F, bool HAS_W>
__global__ void __launch_bounds__(1024, 1)
route_lane_kernel(const LaneArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_all[];
    __shared__ int sRegion;
    constexpr bool PREG = MT <= 4;                              // p in registers (else in shared memory)
    constexpr int MR = PREG ? MT : 1;
    const unsigned sbase = (unsigned)__cvta_generic_to_shared(smem_all);
    const int tid = threadIdx.x;
    const int TR = a.TR, TV = (int)blockDim.x - a.TR;
    const int nsteps = a.nsteps, M = a.M, ld = a.ld;
    const size_t splp = (size_t)a.splp;
    bool abandon = false;                                      // watchdog / poisoned handle: decided by a barrier vote
    int first_region = -1;

    for (;;) {
        if (tid == 0) {
            const long long t = (long long)atomicAdd(a.ticket, 1ull);
            sRegion = (t < a.n_regions && ld_relaxed_s32(a.status) == 0) ? (int)t : -1;
        }
        __syncthreads();
        const int reg = sRegion;
        if (reg < 0) break;
        if (first_region < 0) first_region = reg;              // the step records are staged once per CTA
        const LaneRegionDesc rd = a.regions[reg];
        const int nr = rd.n_real, nv = rd.n_virt;
        unsigned long long* tr = a.trace ? a.trace + 8 * (size_t)reg : nullptr;    // development aid: region timeline
        if (tr && tid == 0) tr[0] = globaltimer_ns();
        // shared-memory layout of this region (LaneSchedule::region_bytes)
        const int rv = nr + nv + 1;                            // rows of an outflow buffer: real, virtual, ZERO
        const unsigned sOb = sbase;                            // [2][MT][rv] outflows of this / the previous iteration
        const unsigned sExt = sOb + 16u * MT * rv;             // [nv][MT][32] stream windows
        const unsigned sMetaV = sExt + 256u * MT * nv;         // [nv] records of the virtual rows
        const unsigned sChild = sMetaV + 16u * nv;             // children beyond the first two
        const unsigned sP = sChild + (((unsigned)(2 * rd.n_child)) + 15u & ~15u);   // [MT][nr] (MT > 4 only)
        const unsigned sFn = sP + (PREG ? 0u : ((8u * MT * (unsigned)nr + 15u) & ~15u));   // [nr] forcing row after the bracket
        const unsigned sSteps = sbase + a.off_steps;           // [nsteps] per-step records (when they fit)
        // ---- this thread's row ----------------------------------------------------------------------------
        const bool has_row = tid < nr;
        int off = 0, nx = 0, slot = -1, pos = 0, rec = -1;
        unsigned c0a = 0, c1a = 0, xa0 = 0;
        double al = 0.0, be = 0.0, ch = 0.0, ga = 0.0, f0 = 0.0, f1 = 0.0, fn = 0.0;
        double p[MR];
#pragma unroll
        for (int m = 0; m < MR; ++m) p[m] = 0.0;
        if (has_row) {
            const int4 mt = a.meta[rd.row_off + tid];
            pos = mt.x; off = mt.y & 0xffff; nx = (int)((unsigned)mt.y >> 16); slot = mt.w;
            c0a = 8u * ((unsigned)mt.z & 0xffffu); c1a = 8u * ((unsigned)mt.z >> 16);
            if (nx > 0) xa0 = sChild + 2u * (unsigned)a.xbeg[rd.row_off + tid];
            const double2 ab = *reinterpret_cast<const double2*>(a.coef + 4 * (size_t)pos);
            const double2 cg = *reinterpret_cast<const double2*>(a.coef + 4 * (size_t)pos + 2);
            al = ab.x; be = ab.y; ch = cg.x; ga = cg.y;
            if (HAS_F) {
                const int r0s = __ldg(&a.steps[0].r0), r1s = __ldg(&a.steps[0].r1) & 0x3fffffff;
                f0 = __ldg(a.F + (size_t)r0s * a.n + pos);
                f1 = __ldg(a.F + (size_t)r1s * a.n + pos);
                fn = __ldg(a.F + (size_t)min(max(r0s, r1s) + 1, a.R - 1) * a.n + pos);
                sts_f64(sFn + 8u * (unsigned)tid, fn);
            }
            if (a.rec_slot) rec = a.rec_slot[pos];
            const double* og = a.O + (size_t)pos * ld;
            const double* ig = a.I + (size_t)pos * ld;
#pragma unroll
            for (int m = 0; m < MT; ++m) {
                double pm = 0.0;
                if (m < M) pm = be * __ldcg(ig + m) + ch * __ldcg(og + m);
                if (PREG) p[m < MR ? m : 0] = pm;
                else sts_f64(sP + 8u * ((unsigned)m * nr + tid), pm);
            }
        }
        {
            const int4* gm = a.meta + rd.row_off + nr;
            for (int i = tid; i < nv; i += blockDim.x) sts_i4(sMetaV + 16u * i, gm[i]);
            const uint16_t* gc = a.child + rd.child_off;
            for (int i = tid; i < rd.n_child; i += blockDim.x) sts_u16(sChild + 2u * i, gc[i]);
            // the ZERO row of both buffers: what a missing child reads
            for (int i = tid; i < 2 * MT; i += blockDim.x) sts_f64(sOb + 8u * ((unsigned)i * rv + (nr + nv)), 0.0);
            if (HAS_F && a.off_steps > 0 && reg == first_region) {
                const int4* gs = reinterpret_cast<const int4*>(a.steps);
                for (int i = tid; i < 2 * nsteps; i += blockDim.x) sts_i4(sSteps + 16u * i, gs[i]);
            }
        }
        if (tid >= TR) {
            // the first two batches of every incoming stream (most likely still EMPTY: fetched again after the lag wait)
            for (int v = tid - TR; v < nv; v += TV) {
                const int vslot = a.meta[rd.row_off + nr + v].w;
                for (int m = 0; m < M; ++m) {
                    const unsigned ex = sExt + 256u * ((unsigned)v * MT + m);
                    const double* g = a.ring + ((size_t)vslot * M + m) * splp;
#pragma unroll
                    for (int q = 0; q < kBatch; ++q) cp_async16(ex + 16u * q, g + 2 * q);
                }
            }
            cp_async_commit();
        }
        __syncthreads();

        const int niter = nsteps + rd.n_extra - 1;
        const unsigned ra = 8u * (unsigned)tid;                 // this row's cell in an outflow buffer
        if (tr && tid == 0) { tr[1] = globaltimer_ns(); tr[4] = (unsigned long long)niter; tr[6] = 0ull; tr[7] = 0ull; }
        int dead = 0;
        int kreq = -16;                                         // iteration of this row's last forcing request
        // Two loops, one per role -- the threads that own rows and the threads that mirror incoming streams -- meeting at
        // the same barrier once per iteration (bar.sync / bar.red count arrivals, not program counters): each loop keeps
        // only its own state live, which matters at 64 registers per thread.  Every vote_every-th barrier also votes on
        // abandoning the launch.
        if (tid < TR) {
        // (two instances: the per-step records in shared memory -- the usual case -- or read in place; a run-time choice
        // inside the loop keeps both address computations and both loads alive in every iteration)
        auto real_loop = [&](auto steps_in_smem) {
        constexpr bool SM = decltype(steps_in_smem)::value;
        // (chunks of vote_every iterations: a plain barrier inside, the voting one at the end of a chunk; the two outflow
        // buffers swap by XOR with the difference of their addresses)
        unsigned obc = sOb, obp = sOb + 8u * (unsigned)(MT * rv);
        const unsigned obx = obc ^ obp;
        for (int k0 = 0; k0 < niter && !abandon; k0 += a.vote_every) {
        const int k1 = min(k0 + a.vote_every, niter);
        for (int k = k0; k < k1; ++k, obc ^= obx, obp ^= obx) {
            // the forcing row after a row's bracket waits in shared memory, requested with cp.async when the bracket was
            // entered: one (possibly empty) group per iteration and thread, so everything requested nine or more
            // iterations ago has landed after this wait.  (Kept in a register and requested with a plain load, the
            // value blocked the whole warp: a few lanes change bracket in EVERY iteration, their load is still in flight
            // when the next lanes read the register, and the iteration paid a global-memory latency, ~0.9 us.)
            if (HAS_F) cp_async_wait_group<8>();
            const int s = k - off;
            if (has_row && (unsigned)s < (unsigned)nsteps) {
                double w0 = 0.0, w1 = 0.0;
                int fr0 = 0, fr1 = 0;
                if (HAS_F) {
                    int r1f;
                    if (SM) {
                        const double2 ww = lds_row(sSteps + 32u * s);
                        const int4 rr = lds_i4(sSteps + 32u * s + 16u);
                        w0 = ww.x; w1 = ww.y; fr0 = rr.x; r1f = rr.y;
                    } else {
                        const LaneStep* st = a.steps + s;
                        const double2 ww = *reinterpret_cast<const double2*>(&st->w0);
                        const int2 rr = *reinterpret_cast<const int2*>(&st->r0);
                        w0 = ww.x; w1 = ww.y; fr0 = rr.x; r1f = rr.y;
                    }
                    fr1 = r1f & 0x3fffffff;
                    if (r1f < 0) {                               // the bracket differs from the previous step's
                        if (k - kreq < 9) cp_async_wait_all();    // requested too recently for the wait above (dense tables)
                        if (r1f & 0x40000000) {
                            // the usual case, marked by lane_init_kernel: the bracket moved on by one row -- shift, and
                            // request the row after it
                            f0 = f1; f1 = lds_f64(sFn + ra);
                            const int nn = min(fr1 + 1, a.R - 1);
                            if (nn != fr1) { cp_async8(sFn + ra, a.F + (size_t)nn * a.n + pos); kreq = k; }
                        } else {
                            int pr0, pr1;
                            if (SM) { const int4 pp = lds_i4(sSteps + 32u * (s - 1) + 16u); pr0 = pp.x; pr1 = pp.y; }
                            else { pr0 = __ldg(&a.steps[s - 1].r0); pr1 = __ldg(&a.steps[s - 1].r1); }
                            fn = lds_f64(sFn + ra);
                            rotate_bracket(f0, f1, fn, a.F + pos, a.n, a.R, pr0, pr1 & 0x3fffffff, fr0, fr1);
                            sts_f64(sFn + ra, fn);
                        }
                    }
                }
                double q = 0.0;
                if (HAS_F && !HAS_W) q = ga * (w0 * f0 + w1 * f1);
                const bool last = s + 1 == nsteps;
#pragma unroll
                for (int m = 0; m < MT; ++m) {
                    const unsigned mo = 8u * (unsigned)(m * rv);
                    double infl = lds_f64(obp + mo + c0a) + lds_f64(obp + mo + c1a);
                    if (nx > 0) {                               // confluences of more than two reaches (rows sorted last)
                        unsigned xa = xa0;
                        for (int c = 0; c < nx; ++c, xa += 2u) infl += lds_f64(obp + mo + 8u * lds_u16(xa));
                    }
                    double qm = q;
                    if (HAS_W) {
                        const int mc = min(m, a.wm_ld - 1);
                        qm = ga * (w0 * __ldg(a.Wmul + (size_t)fr0 * a.wm_ld + mc) * f0 +
                                   w1 * __ldg(a.Wmul + (size_t)fr1 * a.wm_ld + mc) * f1);
                    }
                    double pm;
                    if (PREG) pm = p[m < MR ? m : 0];
                    else pm = lds_f64(sP + 8u * ((unsigned)m * nr + tid));
                    const double o = al * infl + (pm + qm);
                    pm = be * infl + ch * o;
                    if (PREG) p[m < MR ? m : 0] = pm;
                    else sts_f64(sP + 8u * ((unsigned)m * nr + tid), pm);
                    sts_f64(obc + mo + ra, o);
                    if ((slot >= 0 || last) && (MT == 1 || m < M)) {
                        if (slot >= 0) __stcg(a.ring + ((size_t)slot * M + m) * splp + s, o);
                        if (last) {
                            __stcg(a.O + (size_t)pos * ld + m, o);
                            __stcg(a.I + (size_t)pos * ld + m, infl);
                        }
                    }
                    if (rec >= 0 && (MT == 1 || m < M)) {
                        const long long gs = a.rec_step_base + s + 1;
                        if (gs % a.rec_every == 0)
                            a.rec_out[((size_t)(gs / a.rec_every - 1) * a.rec_count + rec) * M + m] = o;
                    }
                }
            }
            if (HAS_F) cp_async_commit();
            if (k + 1 < k1) bar_sync();
        }
        if (bar_or(dead)) abandon = true;
        }
        };
        if (a.off_steps > 0) real_loop(std::true_type{}); else real_loop(std::false_type{});
        } else {
        unsigned obc = sOb;
        const unsigned obx = 8u * (unsigned)(MT * rv);
        for (int k0 = 0; k0 < niter && !abandon; k0 += a.vote_every) {
        const int k1 = min(k0 + a.vote_every, niter);
        for (int k = k0; k < k1; ++k, obc = (obc == sOb ? sOb + obx : sOb)) {
            {
                for (int v = tid - TR; v < nv; v += TV) {
                    const int4 mt = lds_i4(sMetaV + 16u * v);
                    const int sv = k - (mt.y & 0xffff);
                    if ((unsigned)sv >= (unsigned)nsteps) continue;
                    const double* g0 = a.ring + (size_t)mt.w * M * splp;
                    const unsigned ex0 = sExt + 256u * ((unsigned)v * MT);
                    // Wait until the producer is `lag` steps ahead of step `from` (or has finished), then fetch the
                    // batch of `from` and the two after it.  Used before the first step and whenever the consumer has
                    // caught up with its producer: consumers then advance in bursts at full speed instead of paying a
                    // trip to L2 per step at the producer's heels (which would compound along a chain of regions).
                    // The wait polls the stream of member `mp`, at a cell that member has not consumed yet (cells this
                    // thread has consumed hold EMPTY again and would never fill).
                    auto lag_and_fetch = [&](int from, int mp) {
                        const int need = min(nsteps, from + a.lag) - 1;
                        unsigned spins = 0;
                        unsigned long long t0 = 0;
                        while (!dead && is_empty(ld_relaxed_f64(g0 + (size_t)mp * splp + need))) {
                            if ((++spins & 15u) == 0) {
                                if (ld_relaxed_s32(a.status) != 0) { dead = 1; break; }
                                const unsigned long long now = globaltimer_ns();
                                if (t0 == 0) t0 = now;
                                else if (now - t0 > a.watchdog_ns) { atomicExch(a.status, 1); dead = 1; break; }
                            }
                            __nanosleep(200);
                        }
                        cp_async_wait_all();                                 // older prefetches must not land on top of this
                        const int b0 = from & ~(kBatch - 1);
                        for (int m = 0; m < M; ++m)
#pragma unroll
                            for (int q = 0; q < 3 * kBatch / 2; ++q) {
                                const int c = b0 + 2 * q;
                                if (c < (int)splp) cp_async16(ex0 + 256u * m + 8u * (c & (kExtCells - 1)), g0 + (size_t)m * splp + c);
                            }
                        cp_async_commit();
                        cp_async_wait_all();
                    };
                    if (sv == 0) {
                        lag_and_fetch(0, M - 1);                             // producers write their members in ascending order
                        if (tr) atomicMax(tr + 2, globaltimer_ns());           // last first-step lag wait of the region over
                    } else if ((sv & (kBatch - 1)) == 0) {
                        cp_async_wait_all();                                 // batches sv/8 and sv/8 + 1 are in the window
                        if (sv + 2 * kBatch < nsteps) {
                            for (int m = 0; m < M; ++m) {
                                const unsigned ex = ex0 + 256u * m + 8u * ((sv + 2 * kBatch) & (kExtCells - 1));
                                const double* g = g0 + (size_t)m * splp + sv + 2 * kBatch;
#pragma unroll
                                for (int q = 0; q < kBatch / 2; ++q) cp_async16(ex + 16u * q, g + 2 * q);
                            }
                        }
                        cp_async_commit();
                    }
                    for (int m = 0; m < M; ++m) {
                        double* cell = a.ring + ((size_t)mt.w * M + m) * splp + sv;
                        const unsigned ea = ex0 + 256u * m + 8u * (sv & (kExtCells - 1));
                        double val = lds_f64(ea);
                        if (is_empty(val)) {
                            // caught up with the producer: fall back by `lag` steps, then continue from the window
                            if (tr) atomicAdd(tr + 6, 1ull);
                            lag_and_fetch(sv, m);
                            val = lds_f64(ea);
                            unsigned spins = 0, nap = 32;
                            unsigned long long t0 = 0;
                            while (is_empty(val)) {                          // (stores to different cells may land out of order)
                                val = ld_relaxed_f64(cell);
                                if (!is_empty(val)) break;
                                if ((++spins & 15u) == 0) {
                                    if (dead || ld_relaxed_s32(a.status) != 0) { dead = 1; val = 0.0; break; }
                                    const unsigned long long now = globaltimer_ns();
                                    if (t0 == 0) t0 = now;
                                    else if (now - t0 > a.watchdog_ns) { atomicExch(a.status, 1); dead = 1; val = 0.0; break; }
                                }
                                __nanosleep(nap);
                                if (nap < 256u) nap <<= 1;
                            }
                        }
                        __stcg(cell, empty_f64());
                        sts_f64(obc + 8u * ((unsigned)m * rv + nr + v), val);
                    }
                }
            }
            if (k + 1 < k1) bar_sync();
        }
        if (bar_or(dead)) abandon = true;
        }
        }
        cp_async_wait_all();
        if (tr && tid == 0) {
            const unsigned sm = smid();
            tr[3] = globaltimer_ns(); tr[5] = sm;
        }
        if (abandon) break;
    }
    // the last CTA to leave re-arms the ticket for the next launch on this handle
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(a.done, 1ull) + 1ull == (unsigned long long)gridDim.x) {
            *a.done = 0ull;
            *a.ticket = 0ull;
        }
    }
}

// forcing interpolation of the launch's steps (nutils.py:21-34); bit 31 of r1: the bracket changed, bit 30: by one row
__global__ void __launch_bounds__(256) lane_init_kernel(const InitArgs a, LaneStep* out, unsigned long long* ticket)
{
    const long long gid0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    if (gid0 == 0) *ticket = 0ull;
    for (long long s = gid0; s < a.nsteps; s += stride) {
        const StepInterp si = interp_step(a.times, a.R, (double)(a.t0_ns + (a.step_base + s + 1) * a.dt_ns), a.method);
        bool changed = false, regular = false;
        if (s > 0) {
            const StepInterp sp = interp_step(a.times, a.R, (double)(a.t0_ns + (a.step_base + s) * a.dt_ns), a.method);
            changed = sp.r0 != si.r0 || sp.r1 != si.r1;
            // regular: the new bracket is (old r1, the row the kernel prefetched after the old bracket)
            regular = changed && si.r0 == sp.r1 && si.r1 == min(max(sp.r0, sp.r1) + 1, a.R - 1) && si.r1 != si.r0;
        }
        LaneStep ls;
        ls.w0 = si.w0; ls.w1 = si.w1; ls.r0 = si.r0;
        ls.r1 = si.r1 | (changed ? (int)0x80000000 : 0) | (regular ? 0x40000000 : 0); ls.pad0 = ls.pad1 = 0;
        out[s] = ls;
    }
}

template <int MT>
cudaError_t launch_mt(const LaneArgs& a, int threads, size_t smem, int grid, cudaStream_t st)
{
    void (*kern)(const LaneArgs) = nullptr;
    const bool f = a.F != nullptr, w = a.Wmul != nullptr;
    if (!f) kern = route_lane_kernel<MT, false, false>;
    else if (!w) kern = route_lane_kernel<MT, true, false>;
    else kern = route_lane_kernel<MT, true, true>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, threads, smem, st>>>(a);
    count_launch();
    return cudaGetLastError();
}



template <int MT>
cudaError_t occupancy_mt(bool f, bool w, int threads, size_t smem, int* per_sm)
{
    void (*kern)(const LaneArgs) = nullptr;
    if (!f) kern = route_lane_kernel<MT, false, false>;
    else if (!w) kern = route_lane_kernel<MT, true, false>;
    else kern = route_lane_kernel<MT, true, true>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, kern, threads, smem);
}

}  // namespace

cudaError_t lane_occupancy(int mt, bool f, bool w, int threads, size_t smem, int* per_sm)
{
    switch (mt) {
        case 1: return occupancy_mt<1>(f, w, threads, smem, per_sm);
        case 2: return occupancy_mt<2>(f, w, threads, smem, per_sm);
        case 4: return occupancy_mt<4>(f, w, threads, smem, per_sm);
        case 8: return occupancy_mt<8>(f, w, threads, smem, per_sm);
        case 16: return occupancy_mt<16>(f, w, threads, smem, per_sm);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_lane_init(const InitArgs& a, LaneStep* out, unsigned long long* ticket, cudaStream_t st)
{
    const int blocks = (int)std::min<long long>(64, (a.nsteps + 255) / 256);
    lane_init_kernel<<<blocks < 1 ? 1 : blocks, 256, 0, st>>>(a, out, ticket);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_route_lane(const LaneArgs& a, int mt, int threads, size_t smem, int grid, cudaStream_t st)
{
    switch (mt) {
        case 1: return launch_mt<1>(a, threads, smem, grid, st);
        case 2: return launch_mt<2>(a, threads, smem, grid, st);
        case 4: return launch_mt<4>(a, threads, smem, grid, st);
        case 8: return launch_mt<8>(a, threads, smem, grid, st);
        case 16: return launch_mt<16>(a, threads, smem, grid, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace txh
