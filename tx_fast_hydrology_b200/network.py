"""`RiverNetwork`: Python owner of a `txh_net` handle (topology + schedule +
device descriptors) and thin typed wrappers over the routing entry points.

Device state is held in torch CUDA tensors (torch is the allocator / stream
plumbing); only raw pointers cross into libtxh.
"""
import ctypes

import numpy as np

from . import _lib as L


def _cuda_ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _check_f64_cuda(t, name):
    import torch
    if not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
        raise ValueError(f"`{name}` must be a contiguous float64 CUDA tensor")


_raw_stream = None


def _stream_ptr():
    """The current torch stream as a cudaStream_t (the raw getter: `current_stream()` builds a Python
    Stream object on every call, 15 us -- more than a launch)."""
    global _raw_stream
    import torch
    if _raw_stream is None:
        _raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", False)
    if _raw_stream:
        return ctypes.c_void_p(_raw_stream(torch.cuda.current_device()))
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class Forcing:
    """Lateral-inflow table resident in HBM (`txh_forcing`)."""

    def __init__(self, net, times_ns, table, member_mul=None):
        """`table` [R][n] and `member_mul` [R][M]: numpy arrays or (pinned) CPU torch tensors, float64."""
        lib = L.load()
        self.net = net
        times = L.as_f64(np.asarray(times_ns).astype(np.float64))
        tptr, tshape, self._keep_t = self._host_ptr(table)
        R, n = tshape
        if n != net.n or times.size != R:
            raise ValueError("forcing table must be [len(times)][n]")
        M, mp = 0, None
        self.h2d_bytes = R * n * 8
        if member_mul is not None:
            mp, mshape, self._keep_m = self._host_ptr(member_mul)
            if mshape[0] != R:
                raise ValueError("member multipliers must be [len(times)][M]")
            M = mshape[1]
            self.h2d_bytes += R * M * 8
        h = ctypes.c_void_p()
        L.check(lib.txh_forcing_create(net.handle, R, L.ptr_f64(times), tptr, M, mp, _stream_ptr(), ctypes.byref(h)))
        self.handle = h
        self.R = R
        self.M = M

    @staticmethod
    def _host_ptr(a):
        if hasattr(a, "data_ptr"):                      # CPU torch tensor (possibly pinned)
            assert a.dtype.is_floating_point and a.element_size() == 8 and a.is_contiguous() and not a.is_cuda
            return ctypes.c_void_p(a.data_ptr()), tuple(a.shape), a
        a = L.as_f64(a)
        return ctypes.c_void_p(a.ctypes.data), a.shape, a

    def update(self, times_ns, table, member_mul=None, overlap=False):
        """New values for the resident table (same shape): one host->device copy, no allocation.
        `overlap` (pinned CPU torch tensors only): return at once; the table arrives in row chunks on a copy
        stream and later routing calls wait only for the rows their steps read -- do not touch the buffers
        until the run that uses them has finished (or call `wait()`)."""
        times = L.as_f64(np.asarray(times_ns).astype(np.float64))
        tptr, tshape, keep_t = self._host_ptr(table)
        if tshape != (self.R, self.net.n) or times.size != self.R:
            raise ValueError("forcing update must keep the table shape")
        mp, keep_m = None, None
        if member_mul is not None:
            mp, mshape, keep_m = self._host_ptr(member_mul)
            if mshape != (self.R, self.M):
                raise ValueError("member multipliers must keep their shape")
        pinned = all(hasattr(x, "is_pinned") and x.is_pinned() for x in (table, member_mul) if x is not None)
        if overlap and pinned:
            self._keep_t, self._keep_m = keep_t, keep_m
            L.check(L.load().txh_forcing_update_async(self.handle, L.ptr_f64(times), tptr, mp, _stream_ptr()))
        else:
            L.check(L.load().txh_forcing_update(self.handle, L.ptr_f64(times), tptr, mp, _stream_ptr()))

    def wait(self):
        """Block until an overlapped `update` has landed."""
        L.check(L.load().txh_forcing_wait(self.handle))

    def close(self):
        if getattr(self, "handle", None):
            L.load().txh_forcing_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RiverNetwork:
    def __init__(self, endnodes, sched_params=None):
        lib = L.load()
        self._lib = lib
        end = L.as_i64(endnodes)
        self.n = int(end.size)
        sp = None
        if sched_params is not None:
            sp = list(sched_params) + [8] * (5 - len(sched_params))
            sp = (ctypes.c_int32 * 5)(*[int(x) for x in sp])
        h = ctypes.c_void_p()
        L.check(lib.txh_create(self.n, L.ptr_i64(end), sp, ctypes.byref(h)))
        self.handle = h
        self.endnodes = end

    def close(self):
        if getattr(self, "handle", None):
            self._lib.txh_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- topology (host, exact integers) -------------------------------------------------
    def indegree(self):
        out = np.empty(self.n, dtype=np.int64)
        L.check(self._lib.txh_get_indegree(self.handle, L.ptr_i64(out)))
        return out

    def headwaters(self):
        out = np.empty(self.n, dtype=np.int64)
        cnt = ctypes.c_int64()
        L.check(self._lib.txh_get_headwaters(self.handle, L.ptr_i64(out), ctypes.byref(cnt)))
        return out[:cnt.value].copy()

    def levels(self):
        out = np.empty(self.n, dtype=np.int64)
        nl = ctypes.c_int64()
        L.check(self._lib.txh_get_levels(self.handle, L.ptr_i64(out), ctypes.byref(nl)))
        return out, int(nl.value)

    def level_order(self):
        _, nl = self.levels()
        order = np.empty(self.n, dtype=np.int64)
        off = np.empty(nl + 1, dtype=np.int64)
        L.check(self._lib.txh_get_level_order(self.handle, L.ptr_i64(order), L.ptr_i64(off)))
        return order, off

    def chains(self):
        cid = np.empty(self.n, dtype=np.int64); cpos = np.empty(self.n, dtype=np.int64)
        clen = np.empty(self.n, dtype=np.int64); nc = ctypes.c_int64()
        L.check(self._lib.txh_get_chains(self.handle, L.ptr_i64(cid), L.ptr_i64(cpos), L.ptr_i64(clen),
                                         ctypes.byref(nc)))
        return cid, cpos, clen[:nc.value].copy()

    def paths(self):
        pid = np.empty(self.n, dtype=np.int64); ppos = np.empty(self.n, dtype=np.int64)
        L.check(self._lib.txh_get_paths(self.handle, L.ptr_i64(pid), L.ptr_i64(ppos)))
        return pid, ppos

    def visit_order(self):
        out = np.empty(self.n, dtype=np.int64)
        L.check(self._lib.txh_get_visit_order(self.handle, L.ptr_i64(out)))
        return out

    def schedule_info(self):
        info = np.zeros(10, dtype=np.int64)
        L.check(self._lib.txh_get_schedule_info(self.handle, L.ptr_i64(info)))
        keys = ["n_tasks", "n_spine", "n_pocket", "n_input_words", "n_notify", "slots_used",
                "row_fallbacks", "cp_tasks", "cp_cost", "nlevels"]
        return dict(zip(keys, (int(x) for x in info)))

    def schedule(self):
        info = self.schedule_info()
        pos = np.empty(self.n, dtype=np.int64)
        tasks = np.empty((info["n_tasks"], 12), dtype=np.int32)
        deps = np.empty(max(1, info["n_notify"]), dtype=np.int32)
        hdr = np.empty(self.n, dtype=np.uint32)
        inw = np.empty(max(1, info["n_input_words"]), dtype=np.uint32)
        L.check(self._lib.txh_get_schedule(
            self.handle, L.ptr_i64(pos), tasks.ctypes.data_as(L.p_i32), deps.ctypes.data_as(L.p_i32),
            hdr.ctypes.data_as(L.p_u32), inw.ctypes.data_as(L.p_u32)))
        return {"pos_of_reach": pos, "tasks": tasks, "notify": deps[:info["n_notify"]], "hdr": hdr,
                "inw": inw[:info["n_input_words"]]}

    def window_schedule(self):
        info = np.zeros(8, dtype=np.int64)
        L.check(self._lib.txh_get_window_info(self.handle, L.ptr_i64(info)))
        keys = ["n_tasks", "n_slots", "max_len", "max_words", "max_prod", "n_words", "n_prod", "cp_tasks"]
        d = dict(zip(keys, (int(x) for x in info)))
        tasks = np.empty((d["n_tasks"], 12), dtype=np.int32)
        hdr = np.empty(self.n, dtype=np.uint32)
        inw = np.empty(max(1, d["n_words"]), dtype=np.uint32)
        prod = np.empty(max(1, d["n_prod"]), dtype=np.int32)
        L.check(self._lib.txh_get_window_schedule(
            self.handle, tasks.ctypes.data_as(L.p_i32), hdr.ctypes.data_as(L.p_u32), inw.ctypes.data_as(L.p_u32),
            prod.ctypes.data_as(L.p_i32)))
        d.update(tasks=tasks, hdr=hdr, inw=inw[:d["n_words"]], prod=prod[:d["n_prod"]])
        return d

    def lane_schedule(self, M=1, cap_rows=0):
        """The reach-parallel schedule route_lane_kernel runs for ensembles of M <= 16 members (host only)."""
        info = np.zeros(8, dtype=np.int64)
        L.check(self._lib.txh_get_lane_info(self.handle, int(M), int(cap_rows), L.ptr_i64(info)))
        keys = ["n_regions", "n_rows", "n_child", "n_slots", "max_real", "max_virt", "max_extra", "member_tile"]
        d = dict(zip(keys, (int(x) for x in info)))
        regions = np.empty((d["n_regions"], 8), dtype=np.int32)
        rows = np.empty((max(1, d["n_rows"]), 6), dtype=np.int32)
        child = np.empty(max(1, d["n_child"]), dtype=np.int32)
        L.check(self._lib.txh_get_lane_schedule(self.handle, int(M), regions.ctypes.data_as(L.p_i32),
                                                rows.ctypes.data_as(L.p_i32), child.ctypes.data_as(L.p_i32)))
        d.update(regions=regions, rows=rows[:d["n_rows"]], child=child[:d["n_child"]])
        return d

    # ---- coefficients ---------------------------------------------------------------------
    def compute_coeffs(self, K, X, dt):
        K = L.as_f64(K); X = L.as_f64(X)
        out = [np.empty(self.n) for _ in range(4)]
        L.check(self._lib.txh_compute_coeffs(self.handle, L.ptr_f64(K), L.ptr_f64(X), float(dt),
                                             *[L.ptr_f64(o) for o in out]))
        return tuple(out)

    def set_coeffs(self, alpha, beta, chi, gamma):
        arrs = [L.as_f64(a) for a in (alpha, beta, chi, gamma)]
        L.check(self._lib.txh_set_coeffs(self.handle, *[L.ptr_f64(a) for a in arrs]))

    # ---- device state ---------------------------------------------------------------------
    @staticmethod
    def row_stride(M):
        return int(L.load().txh_row_stride(int(M)))

    def alloc_state(self, M, device="cuda"):
        import torch
        return torch.zeros((self.n, self.row_stride(M)), dtype=torch.float64, device=device)

    def pack_host(self, src, M, dst, member_major=False):
        """Host array (numpy, or a pinned CPU torch tensor) in reach order -> device schedule order."""
        ptr, shape, keep = Forcing._host_ptr(src)
        if int(np.prod(shape)) != self.n * int(M):
            raise ValueError(f"pack_host: source must hold {self.n} x {M} doubles, got shape {tuple(shape)}")
        if tuple(dst.shape) != (self.n, self.row_stride(M)) or not dst.is_contiguous():
            raise ValueError("pack_host: destination must be a contiguous alloc_state(M) tensor")
        L.check(self._lib.txh_pack_host(self.handle, ctypes.cast(ptr, L.p_f64), int(M), int(member_major),
                                        _cuda_ptr(dst), _stream_ptr()))
        del keep

    def unpack_host(self, src, M, member_major=False, out=None):
        """Device schedule order -> host reach order; `out` may be a pinned CPU torch tensor."""
        if out is None:
            out = np.empty((M, self.n) if member_major else (self.n, M), dtype=np.float64)
            optr = L.ptr_f64(out)
        else:
            # a caller buffer crosses the C ABI as a raw pointer: settle size, type and layout here
            if hasattr(out, "data_ptr"):
                ok = (out.numel() == self.n * int(M) and out.element_size() == 8 and out.dtype.is_floating_point
                      and out.is_contiguous() and not out.is_cuda)
                optr = ctypes.cast(ctypes.c_void_p(out.data_ptr()), L.p_f64)
            else:
                ok = (isinstance(out, np.ndarray) and out.size == self.n * int(M) and out.dtype == np.float64
                      and out.flags.c_contiguous)
                optr = L.ptr_f64(out) if ok else None
            if not ok:
                raise ValueError(f"unpack_host: `out` must be a contiguous float64 host buffer of {self.n} x {M} values")
        if tuple(src.shape) != (self.n, self.row_stride(M)) or not src.is_contiguous():
            raise ValueError("unpack_host: source must be a contiguous alloc_state(M) tensor")
        L.check(self._lib.txh_unpack_host(self.handle, _cuda_ptr(src), int(M), int(member_major), optr,
                                          _stream_ptr()))
        return out

    def pack_dev(self, src, M, dst):
        L.check(self._lib.txh_pack_dev(self.handle, _cuda_ptr(src), int(M), _cuda_ptr(dst), _stream_ptr()))

    def unpack_dev(self, src, M, dst):
        L.check(self._lib.txh_unpack_dev(self.handle, _cuda_ptr(src), int(M), _cuda_ptr(dst), _stream_ptr()))

    def gather_rows(self, X, M, reach_idx, out):
        idx = L.as_i64(reach_idx)
        L.check(self._lib.txh_gather_rows(self.handle, _cuda_ptr(X), int(M), L.ptr_i64(idx), idx.size,
                                          _cuda_ptr(out), _stream_ptr()))

    def init_inflows(self, O, I, M):
        L.check(self._lib.txh_init_inflows(self.handle, _cuda_ptr(O), _cuda_ptr(I), int(M), _stream_ptr()))

    # ---- routing ----------------------------------------------------------------------------
    def route_run(self, O, I, M, forcing, t0_ns, dt_ns, nsteps, method=1, rec_reach=None, rec_every=1,
                  rec_out=None):
        """`method`: 1 linear, 0 nearest row (nutils.interpolate_sample)."""
        if isinstance(method, bool) or method not in (0, 1):
            raise ValueError(f"`method` must be 0 (nearest) or 1 (linear), got {method!r}")
        fh = forcing.handle if forcing is not None else None
        if rec_reach is not None:
            rr = L.as_i64(rec_reach)
            rp, rc, ro = L.ptr_i64(rr), rr.size, _cuda_ptr(rec_out)
        else:
            rp, rc, ro = L.p_i64(), 0, None
        L.check(self._lib.txh_route_run(self.handle, _cuda_ptr(O), _cuda_ptr(I), int(M), fh, int(t0_ns),
                                        int(dt_ns), int(nsteps), int(method), rp, rc, int(rec_every), ro,
                                        _stream_ptr()))

    def run_assimilating(self, O, I, M, forcing, t0_ns, dt_ns, nsteps, every, obs_reach, Zp, qs, R, Dinv, dinv_kind,
                         rowsum, HX, work, W, T, G, method=1, time_every=0, obs_ready=None, rec_reach=None, rec_every=1,
                         rec_out=None, prior_out=None):
        """`txh_run_assimilating`: routing windows + ensemble updates of an unsharded ensemble, host out of the loop.
        With `rec_reach`: `txh_run_assimilating_rec`, hydrographs into `rec_out` (and the priors into `prior_out`)."""
        idx = L.as_i64(obs_reach)
        args = (self.handle, _cuda_ptr(O), _cuda_ptr(I), int(M), forcing.handle if forcing is not None else None,
                int(t0_ns), int(dt_ns), int(nsteps), int(every), int(method), L.ptr_i64(idx), idx.size, _cuda_ptr(Zp),
                _cuda_ptr(qs), _cuda_ptr(R), _cuda_ptr(Dinv) if Dinv is not None else None, int(dinv_kind),
                _cuda_ptr(rowsum), _cuda_ptr(HX), _cuda_ptr(work), _cuda_ptr(W), _cuda_ptr(T), _cuda_ptr(G),
                int(time_every), ctypes.c_void_p(obs_ready.cuda_event) if obs_ready is not None else None)
        if rec_reach is None:
            L.check(self._lib.txh_run_assimilating(*args, _stream_ptr()))
            return
        rr = L.as_i64(rec_reach)
        L.check(self._lib.txh_run_assimilating_rec(*args, L.ptr_i64(rr), rr.size, int(rec_every), _cuda_ptr(rec_out),
                                                   _cuda_ptr(prior_out) if prior_out is not None else None,
                                                   _stream_ptr()))

    def set_transform_history(self, T_hist=None):
        """While set, update k of every `run_assimilating` call solves its ensemble transform into `T_hist[k]`
        ([>= updates][M][M] float64 contiguous CUDA tensor) instead of into `T`; None switches it off."""
        if T_hist is not None:
            _check_f64_cuda(T_hist, "T_hist")
            if T_hist.dim() != 3 or T_hist.shape[1] != T_hist.shape[2]:
                raise ValueError(f"set_transform_history: `T_hist` must be [updates][M][M], got {tuple(T_hist.shape)}")
        self._T_hist_keep = T_hist
        L.check(self._lib.txh_set_transform_history(self.handle, _cuda_ptr(T_hist) if T_hist is not None else None,
                                                    T_hist.numel() if T_hist is not None else 0))

    ENKF_METHODS = ("stochastic", "etkf")

    def set_enkf_transform(self, method="stochastic", rtpp=0.0):
        """`txh_set_enkf_transform`: the form of the ensemble update every later `enkf_solve` and `run_assimilating`
        on the handle solves -- "stochastic" (perturbed observations, the default) or "etkf" (square root, needs
        identical observation columns, at most 64 members in all) -- and the relaxation to prior perturbations
        `rtpp` in [0, 1)."""
        if method not in self.ENKF_METHODS:
            raise ValueError(f"set_enkf_transform: `method` must be one of {self.ENKF_METHODS}, got {method!r}")
        L.check(self._lib.txh_set_enkf_transform(self.handle, self.ENKF_METHODS.index(method), float(rtpp)))

    @staticmethod
    def enks_work_size(M, nupd):
        return int(L.load().txh_enks_work_size(int(M), int(nupd)))

    def enks_smooth(self, M, nupd, every, T_hist, rec, rec_every, lag, out, work=None):
        """`txh_enks_smooth`: the fixed-lag ensemble Kalman smoother of recorded hydrographs `rec`
        ([slots][k][M], slot j after step (j+1)*rec_every) from the transforms `T_hist[:nupd]` of updates after every
        `every`-th step; `lag` in steps.  Writes `out` (same shape as `rec`, a buffer of its own) and returns it."""
        for name, t in (("T_hist", T_hist), ("rec", rec), ("out", out)):
            _check_f64_cuda(t, name)
        M, nupd = int(M), int(nupd)
        if T_hist.dim() != 3 or T_hist.shape[0] < nupd or tuple(T_hist.shape[1:]) != (M, M):
            raise ValueError(f"enks_smooth: `T_hist` must be [>= {nupd}][{M}][{M}], got {tuple(T_hist.shape)}")
        if rec.dim() != 3 or rec.shape[2] != M or tuple(out.shape) != tuple(rec.shape):
            raise ValueError(f"enks_smooth: `rec` and `out` must both be [slots][k][{M}], got {tuple(rec.shape)} and "
                             f"{tuple(out.shape)}")
        if work is None:
            import torch
            work = torch.empty(max(1, self.enks_work_size(M, nupd)), dtype=torch.float64, device=rec.device)
        elif work.numel() < self.enks_work_size(M, nupd):
            raise ValueError("enks_smooth: `work` is smaller than enks_work_size(M, nupd)")
        L.check(self._lib.txh_enks_smooth(M, nupd, int(every), _cuda_ptr(T_hist), rec.shape[0], rec.shape[1],
                                          int(rec_every), int(lag), _cuda_ptr(rec), _cuda_ptr(out), _cuda_ptr(work),
                                          _stream_ptr()))
        return out

    def route_timings(self):
        """Durations (ms) of the routing launches `run_assimilating(time_every=...)` bracketed; synchronises."""
        cnt = np.zeros(1, dtype=np.int64)
        L.check(self._lib.txh_get_route_timings(self.handle, L.p_f64(), 0, L.ptr_i64(cnt)))
        out = np.zeros(max(1, int(cnt[0])))
        L.check(self._lib.txh_get_route_timings(self.handle, L.ptr_f64(out), int(cnt[0]), L.ptr_i64(cnt)))
        return out[:int(cnt[0])]

    def route_step(self, O, I, M, q_dev=None, levels=False):
        fn = self._lib.txh_route_step_levels if levels else self._lib.txh_route_step
        L.check(fn(self.handle, _cuda_ptr(O), _cuda_ptr(I), int(M),
                   _cuda_ptr(q_dev) if q_dev is not None else None, _stream_ptr()))

    def route_apply(self, X, Iscr, M):
        L.check(self._lib.txh_route_apply(self.handle, _cuda_ptr(X), _cuda_ptr(Iscr), int(M), _stream_ptr()))

    def apply_gain(self, G, O, I, M):
        L.check(self._lib.txh_apply_gain(self.handle, _cuda_ptr(G), _cuda_ptr(O), _cuda_ptr(I), int(M),
                                         _stream_ptr()))

    # ---- assimilation ----------------------------------------------------------------------
    def set_stats_output(self, rowsum=None, scale=1.0):
        """Routing calls also leave scale * (member sum of the final outflows) in `rowsum` [n]; None = off."""
        self._stats_keep = rowsum
        L.check(self._lib.txh_set_stats_output(self.handle, _cuda_ptr(rowsum) if rowsum is not None else None,
                                               float(scale)))

    def enkf_stats(self, O, Mloc, obs_reach, rowsum, HX, scale=1.0):
        """`rowsum` None: the sums came with the routing launch (set_stats_output); only gather the gauge rows."""
        idx = L.as_i64(obs_reach)
        L.check(self._lib.txh_enkf_stats(self.handle, _cuda_ptr(O), int(Mloc), L.ptr_i64(idx), idx.size,
                                         float(scale), _cuda_ptr(rowsum) if rowsum is not None else None,
                                         _cuda_ptr(HX), _stream_ptr()))

    def kf_work_size(self, m):
        return int(self._lib.txh_kf_work_size(self.handle, int(m)))

    def kf_filter(self, P_in, P_out, P_prior, Q, R, obs_reach, z, O, I, K, gain, dz, work):
        """KalmanFilter.filter (da.py:91-136) as one chain of launches; `z` is the host measurement vector."""
        idx = L.as_i64(obs_reach)
        zz = L.as_f64(z)
        L.check(self._lib.txh_kf_filter(self.handle, _cuda_ptr(P_in), _cuda_ptr(P_out),
                                        _cuda_ptr(P_prior) if P_prior is not None else None, _cuda_ptr(Q),
                                        _cuda_ptr(R), L.ptr_i64(idx), idx.size, L.ptr_f64(zz), _cuda_ptr(O),
                                        _cuda_ptr(I), _cuda_ptr(K), _cuda_ptr(gain), _cuda_ptr(dz), _cuda_ptr(work),
                                        _stream_ptr()))

    @staticmethod
    def enkf_work_size(m, Mtot):
        return int(L.load().txh_enkf_work_size(int(m), int(Mtot)))

    def enkf_solve(self, m, Mtot, HX, Zp, mean, obs_reach, qs, R, work, W, T, Dinv=None, dinv_kind=0):
        idx = L.as_i64(obs_reach)
        L.check(self._lib.txh_enkf_solve(self.handle, int(m), int(Mtot), _cuda_ptr(HX), _cuda_ptr(Zp),
                                         _cuda_ptr(mean), L.ptr_i64(idx), _cuda_ptr(qs), _cuda_ptr(R),
                                         _cuda_ptr(Dinv) if Dinv is not None else None, int(dinv_kind),
                                         _cuda_ptr(work), _cuda_ptr(W), _cuda_ptr(T), _stream_ptr()))

    def enkf_apply(self, O, I, Mloc, Xall, ldx, Mtot, col0, mean, T, obs_reach, qs, W, G, x_block_stride=0):
        """`x_block_stride` != 0: Xall is the all-gather of the shards' state rows, [world][n][ldx]."""
        idx = L.as_i64(obs_reach)
        L.check(self._lib.txh_enkf_apply(self.handle, _cuda_ptr(O), _cuda_ptr(I), int(Mloc),
                                         _cuda_ptr(Xall) if Xall is not None else None, int(ldx),
                                         int(x_block_stride), int(Mtot),
                                         int(col0), _cuda_ptr(mean), _cuda_ptr(T), L.ptr_i64(idx), idx.size,
                                         _cuda_ptr(qs), _cuda_ptr(W), _cuda_ptr(G), _stream_ptr()))

    def enkf_apply_peers(self, O_in, O_out, I, Mloc, shard_ptrs, Mtot, col0, mean, T, obs_reach, qs, W, G):
        """`txh_enkf_apply_peers`: the shards' state matrices (`shard_ptrs`: device addresses, one per rank, peers
        mapped over NVLink) are read in place; the posterior of this shard goes to `O_out`."""
        idx = L.as_i64(obs_reach)
        arr = (ctypes.c_void_p * len(shard_ptrs))(*[int(p) for p in shard_ptrs])
        L.check(self._lib.txh_enkf_apply_peers(self.handle, _cuda_ptr(O_in), _cuda_ptr(O_out), _cuda_ptr(I), int(Mloc),
                                               arr, len(shard_ptrs), int(Mtot), int(col0), _cuda_ptr(mean), _cuda_ptr(T),
                                               L.ptr_i64(idx), idx.size, _cuda_ptr(qs), _cuda_ptr(W), _cuda_ptr(G),
                                               _stream_ptr()))

    def check(self):
        L.check(self._lib.txh_check(self.handle, _stream_ptr() if self._has_cuda() else None))

    @staticmethod
    def _has_cuda():
        try:
            import torch
            return torch.cuda.is_available()
        except Exception:
            return False


def _check_matrix(name, t, rows=None, cols=None, contiguous=False):
    """Raw device pointers cross the C ABI below: a matrix must be a 2-D float64 CUDA tensor of the expected shape
    whose rows are contiguous (row-major with a leading dimension); `contiguous` also rules out a leading dimension
    wider than a row."""
    import torch
    if not isinstance(t, torch.Tensor) or t.dim() != 2:
        raise ValueError(f'`{name}` must be a 2-D tensor')
    if (rows is not None and t.shape[0] != rows) or (cols is not None and t.shape[1] != cols):
        raise ValueError(f'`{name}` must be ({rows}, {cols}), got {tuple(t.shape)}')
    if t.numel() and ((t.shape[1] > 1 and t.stride(1) != 1) or (t.shape[0] > 1 and t.stride(0) < t.shape[1])):
        raise ValueError(f'`{name}` must be row-major with contiguous rows, got strides {t.stride()}')
    if contiguous and not t.is_contiguous():
        raise ValueError(f'`{name}` must be contiguous')
    if t.dtype != torch.float64:
        raise ValueError(f'`{name}` must be float64, got {t.dtype}')
    if not t.is_cuda:
        raise ValueError(f'`{name}` must be a CUDA tensor')


def dgemm(A, B, C, transA=False, transB=False, alpha=1.0, beta=0.0):
    """C = alpha op(A) op(B) + beta C on the FP64 tensor cores (row-major CUDA tensors, float64; a row slice such as
    X[:, :k] is fine, a transposed view is not: pass the transpose flag instead)."""
    _check_matrix('C', C)
    M, N = C.shape
    _check_matrix('A', A)
    K = A.shape[0] if transA else A.shape[1]
    _check_matrix('A', A, *((K, M) if transA else (M, K)))
    _check_matrix('B', B, *((N, K) if transB else (K, N)))
    lib = L.load()
    L.check(lib.txh_dgemm(int(transA), int(transB), M, N, K, float(alpha), _cuda_ptr(A), A.stride(0),
                          _cuda_ptr(B), B.stride(0), float(beta), _cuda_ptr(C), C.stride(0), _stream_ptr()))
    return C


def spd_solve(S, B):
    """In place: B <- S^-1 B for SPD S (S is overwritten by its Cholesky factor)."""
    _check_matrix('S', S, contiguous=True)
    m = S.shape[0]
    _check_matrix('S', S, m, m, contiguous=True)
    _check_matrix('B', B, m, None, contiguous=True)
    L.check(L.load().txh_spd_solve(m, B.shape[1], _cuda_ptr(S), _cuda_ptr(B), _stream_ptr()))
    return B


def inverse(A):
    """In place: A <- inv(A), Gauss-Jordan with partial pivoting."""
    import torch
    _check_matrix('A', A, contiguous=True)
    m = A.shape[0]
    _check_matrix('A', A, m, m, contiguous=True)
    work = torch.empty_like(A)
    L.check(L.load().txh_inverse(m, _cuda_ptr(A), _cuda_ptr(work), _stream_ptr()))
    return A
