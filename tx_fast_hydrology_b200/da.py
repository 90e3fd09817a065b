"""Data-assimilation callbacks on the GPU.

`KalmanFilter` is the drop-in for the reference's dense-covariance filter
(tx_fast_hydrology/da.py:14-136): same constructor, same hooks
(`__on_simulation_start__`, `__on_step_end__`), same `filter()` algebra, same
gauge ordering (columns and R permuted to ascending reach index, da.py:36-44),
same in-place gain application -- with the covariance propagation
`_aqat_par` (nutils.py:194-214) running as two member-batched routing launches
(the columns of P are the members) and the dense products on the FP64 tensor
cores.  It is meant for the reference's use case, per-sub-basin models of
10^2..10^3 reaches.

`EnsembleKalmanFilter` is the ensemble form of the same update for networks whose
n x n covariance cannot exist (n ~ 10^5): P is the sample covariance of the
member-batched forecast plus a diagonal Q (SURVEY.md section 8c).  Members may be
sharded over ranks; the statistics are then combined with torch.distributed
collectives (NCCL over NVLink) between the three device phases.
"""
import copy
import datetime as _dt
import logging

import numpy as np
import pandas as pd

from .callbacks import BaseCallback
from .network import dgemm, inverse
from .sharding import combine_statistics
from .nutils import interpolate_sample

logger = logging.getLogger(__name__)


def _gauge_setup(model, measurements):
    """da.py:27-44: asserts, gauge -> reach index map, ascending-index permutation."""
    assert isinstance(measurements.index, pd.DatetimeIndex)
    assert (measurements.index.tz == _dt.timezone.utc)
    reach_index_map = pd.Series(np.arange(len(model.reach_ids)), index=model.reach_ids)
    reach_indices = reach_index_map.reindex(measurements.columns).values
    assert not np.isnan(reach_indices.astype(float)).any()
    reach_indices = reach_indices.astype(int)
    permutations = np.argsort(reach_indices)
    if not (permutations == np.arange(len(reach_indices))).all():
        logger.warning('Measurement indices not sorted. Permuting columns...')
    return reach_indices[permutations], permutations


class _MeasurementTable:
    """`measurements` is a live attribute in the reference: the service loop reassigns it on every forecast
    cycle (app/app.py:75-80) and `interpolate_input` / `latest_timestamp` read it on every call (da.py:63-81).
    The drop-in keeps float64 copies of the index and the values for the device path, rebuilt on assignment.
    A frame whose columns are the filter's gauges in another order is re-ordered by label (the reference would
    silently pair gauges with the wrong reaches); another column set is an error."""

    @property
    def measurements(self):
        return self._measurements

    @measurements.setter
    def measurements(self, frame):
        assert isinstance(frame.index, pd.DatetimeIndex)
        assert (frame.index.tz == _dt.timezone.utc)
        known = getattr(self, '_measurements', None)
        if known is not None:
            if frame.shape[1] != known.shape[1] or set(frame.columns) != set(known.columns):
                raise ValueError('new measurements must carry the same gauge columns as the filter was built with')
            if list(frame.columns) != list(known.columns):
                frame = frame[known.columns]
        self._measurements = frame
        self._meas_times = frame.index.astype(int).astype(float).values
        self._meas_values = np.ascontiguousarray(frame.values, dtype=np.float64)


class KalmanFilter(_MeasurementTable, BaseCallback):
    def __init__(self, model, measurements, Q_cov, R_cov, P_t_init):
        import torch
        self.model = model
        self.Q_cov = Q_cov
        self.reach_ids = model.reach_ids
        self.gage_reach_ids = measurements.columns
        self.datetime = copy.deepcopy(model.datetime)
        self.num_measurements = measurements.shape[1]
        if model.members != 1:
            raise ValueError('the dense KalmanFilter needs a single-member model')
        self.reach_indices, perm = _gauge_setup(model, measurements)
        s = np.zeros(model.n, dtype=bool)
        s[self.reach_indices] = True
        self.s = s
        self.measurements = measurements.iloc[:, perm]
        n, m = model.n, self.num_measurements
        R_full = np.asarray(R_cov, dtype=np.float64)
        if R_full.shape != (m, m):
            raise ValueError(f'`R_cov` must be ({m}, {m}), got {R_full.shape}')
        self.R_cov = R_full[perm, :][:, perm]
        self.reach_indices = np.ascontiguousarray(self.reach_indices, dtype=np.int64)
        # The reference adds Q_cov with numpy broadcasting (da.py:115-116), so a scalar or a row vector works
        # there; the device chain reads dense n x n / m x m matrices through raw pointers, so the shapes are
        # settled here, before anything crosses the C ABI.
        try:
            Q_full = np.ascontiguousarray(np.broadcast_to(np.asarray(Q_cov, dtype=np.float64), (n, n)))
        except ValueError:
            raise ValueError(f'`Q_cov` must broadcast to ({n}, {n}), got {np.shape(Q_cov)}')
        P_full = np.ascontiguousarray(P_t_init, dtype=np.float64)
        if P_full.shape != (n, n):
            raise ValueError(f'`P_t_init` must be ({n}, {n}), got {P_full.shape}')
        # device-resident matrices
        self._torch = torch
        dev = 'cuda'
        self._P = torch.as_tensor(P_full, device=dev).clone()
        self._Q = torch.as_tensor(Q_full, device=dev)
        self._R = torch.as_tensor(np.ascontiguousarray(self.R_cov), device=dev)
        self._idx = torch.as_tensor(self.reach_indices, device=dev)
        self._P_prev = self._P
        self._K_d = self._dz_d = self._gain_d = None
        self._work = None
        self.saved_states = {}
        self.save_state()

    # numpy views of the device matrices, as the reference exposes them
    @property
    def P_t_next(self):
        return self._P.cpu().numpy()

    @P_t_next.setter
    def P_t_next(self, value):
        value = np.ascontiguousarray(value, dtype=np.float64)
        if value.shape != (self.model.n, self.model.n):
            raise ValueError(f'`P_t_next` must be ({self.model.n}, {self.model.n}), got {value.shape}')
        self._P = self._torch.as_tensor(value, device='cuda').clone()

    @property
    def P_t_prev(self):
        return self._P_prev.cpu().numpy()

    def __on_simulation_start__(self):
        if self.model.datetime > self.latest_timestamp:
            return None
        return self.filter()

    def __on_step_end__(self):
        if self.model.datetime > self.latest_timestamp:
            return None
        return self.filter()

    @property
    def latest_measurement(self):
        return self.measurements.iloc[-1, :].values

    @property
    def latest_timestamp(self):
        return self.measurements.index[-1]

    def interpolate_input(self, datetime, method='linear'):
        if method not in ('linear', 'nearest'):
            raise ValueError
        return interpolate_sample(float(datetime.value), self._meas_times, self._meas_values,
                                  method=1 if method == 'linear' else 0)

    def save_state(self):
        self.saved_states['datetime'] = self.datetime
        self.saved_states['P_t_next'] = self._P.clone()

    def load_state(self):
        self.datetime = self.saved_states['datetime']
        self._P = self.saved_states['P_t_next']

    def _aqat(self, P):
        """nutils.py:194-214 (`_aqat_par`): A (A P)^T, the columns of P routed as members."""
        torch = self._torch
        net, n = self.model.network, self.model.n
        self.model._sync_coeffs()
        X = net.alloc_state(n)
        scr = net.alloc_state(n)
        out = torch.empty((n, n), dtype=torch.float64, device='cuda')
        net.pack_dev(P.contiguous(), n, X)
        net.route_apply(X, scr, n)
        net.unpack_dev(X, n, out)
        net.pack_dev(out.t().contiguous(), n, X)
        net.route_apply(X, scr, n)
        net.unpack_dev(X, n, out)
        return out

    # K, dz, gain of the last update stay on the device until somebody looks at them
    K = property(lambda self: None if self._K_d is None else self._K_d.cpu().numpy())
    dz = property(lambda self: None if self._dz_d is None else self._dz_d.cpu().numpy())
    gain = property(lambda self: None if self._gain_d is None else self._gain_d.cpu().numpy())

    def _device_filter(self, Z, keep_prior=False):
        """One `txh_kf_filter` chain: covariance propagation, gain, covariance update and the in-place
        state correction (da.py:112-126), no host round trip besides the measurement vector."""
        torch = self._torch
        mdl = self.model
        n, m = mdl.n, self.num_measurements
        mdl._ensure_device()
        mdl._sync_coeffs()
        net, d = mdl.network, mdl._dev
        if self._work is None:
            self._work = torch.empty(net.kf_work_size(m), dtype=torch.float64, device='cuda')
        f64 = dict(dtype=torch.float64, device='cuda')
        P_prev = self._P if self._P.is_contiguous() else self._P.contiguous()
        P_next = torch.empty((n, n), **f64)
        P_prior = torch.empty((n, n), **f64) if keep_prior else None
        K = torch.empty((n, m), **f64)
        gain = torch.empty(n, **f64)
        dz = torch.empty(m, **f64)
        net.kf_filter(P_prev, P_next, P_prior, self._Q, self._R, self.reach_indices, Z, d['O'], d['I'], K, gain, dz,
                      self._work)
        mdl._device_advanced()
        self._P, self._P_prev = P_next, P_prev
        self._K_d, self._gain_d, self._dz_d = K, gain, dz
        return P_prior

    def filter(self):
        """da.py:91-136 on the device; the model state is corrected in place in HBM."""
        mdl = self.model
        Z = self.interpolate_input(mdl.datetime)
        self._device_filter(Z)
        self.datetime = mdl.datetime


class KalmanSmoother(KalmanFilter):
    """Rauch-Tung-Striebel smoother callback (tx_fast_hydrology/da.py:139-264): the forward pass is the dense
    filter with every prior / posterior covariance kept ON THE DEVICE, the backward pass
    J = (P_p[t+1]^-1 A P_f[t])^T,  x_s[t] = x_f[t] + J (x_s[t+1] - x_p[t+1]),  P_s[t] = P_f[t] + J (P_s[t+1] - P_p[t+1])
    runs at simulation end with the operator product as a member-batched routing launch and the dense
    products on the FP64 tensor cores.  Kept quirks: measurements are looked up at the exact model time
    (da.py:190), states are rebound rather than updated in place (da.py:205-206), the covariance recursion has
    no trailing J^T (da.py:257)."""

    def __init__(self, model, measurements, Q_cov, R_cov, P_t_init):
        super().__init__(model, measurements, Q_cov, R_cov, P_t_init)
        self.N = len(measurements) - 1
        t = model.datetime
        self.datetimes = [t]
        self.P_f = {t: self._P.clone()}
        self.P_p = {t: self._P.clone()}
        self.i_hat_f = {t: model.i_t_next.copy()}
        self.o_hat_f = {t: model.o_t_next.copy()}
        self.i_hat_p = {t: model.i_t_next.copy()}
        self.o_hat_p = {t: model.o_t_next.copy()}
        self.i_hat_s = None
        self.o_hat_s = None
        self.P_s = None

    def __on_simulation_end__(self):
        return self.smooth()

    def _ap(self, P):
        """nutils.py:157-169 (`_ap_par`): A P, the columns of P routed as members."""
        torch = self._torch
        net, n = self.model.network, self.model.n
        self.model._sync_coeffs()
        X = net.alloc_state(n)
        scr = net.alloc_state(n)
        out = torch.empty((n, n), dtype=torch.float64, device='cuda')
        net.pack_dev(P.contiguous(), n, X)
        net.route_apply(X, scr, n)
        net.unpack_dev(X, n, out)
        return out

    def filter(self):
        """da.py:170-219."""
        mdl = self.model
        t = mdl.datetime
        i_prior = mdl._peek_state('i_t_next')
        o_prior = mdl._peek_state('o_t_next')
        Z = self.measurements.loc[t].values                                  # exact time, no interpolation
        P_prior = self._device_filter(Z, keep_prior=True)
        i_next = mdl._peek_state('i_t_next')                                 # fresh arrays (da.py:203-206)
        o_next = mdl._peek_state('o_t_next')
        self.i_hat_f[t] = i_next; self.i_hat_p[t] = i_prior
        self.o_hat_f[t] = o_next; self.o_hat_p[t] = o_prior
        self.P_p[t] = P_prior; self.P_f[t] = self._P
        self.datetimes.append(t)
        self.datetime = t

    def smooth(self):
        """da.py:221-264, backward pass on the device."""
        torch = self._torch
        n = self.model.n
        ts = self.datetimes
        N = len(ts) - 1
        last = self.datetime
        P_s = {last: self.P_f[last]}
        dev = dict(dtype=torch.float64, device='cuda')
        x_s = torch.as_tensor(np.stack([self.i_hat_f[last], self.o_hat_f[last]], axis=1), **dev).contiguous()
        i_hat_s, o_hat_s = {last: self.i_hat_f[last]}, {last: self.o_hat_f[last]}
        for k in reversed(range(N)):
            t, tp1 = ts[k], ts[k + 1]
            A_Pf = self._ap(self.P_f[t])
            J = torch.empty((n, n), **dev)
            dgemm(A_Pf, inverse(self.P_p[tp1].clone()), J, transA=True, transB=True)     # (P_p^-1 A P_f)^T
            x_f = torch.as_tensor(np.stack([self.i_hat_f[t], self.o_hat_f[t]], axis=1), **dev).contiguous()
            x_p = torch.as_tensor(np.stack([self.i_hat_p[tp1], self.o_hat_p[tp1]], axis=1), **dev).contiguous()
            x_new = x_f.clone()
            dgemm(J, (x_s - x_p).contiguous(), x_new, alpha=1.0, beta=1.0)
            P = self.P_f[t].clone()
            dgemm(J, (P_s[tp1] - self.P_p[tp1]).contiguous(), P, alpha=1.0, beta=1.0)
            x_s = x_new
            xs_host = x_new.cpu().numpy()
            i_hat_s[t] = xs_host[:, 0].copy(); o_hat_s[t] = xs_host[:, 1].copy()
            P_s[t] = P
        self.i_hat_s = pd.DataFrame.from_dict(i_hat_s, orient='index')
        self.i_hat_s.columns = self.model.reach_ids
        self.o_hat_s = pd.DataFrame.from_dict(o_hat_s, orient='index')
        self.o_hat_s.columns = self.model.reach_ids
        self.P_s = P_s


class EnsembleKalmanFilter(_MeasurementTable, BaseCallback):
    """Ensemble Kalman update of a member-batched `Muskingum(members=M)`.

    measurements : DataFrame [times x gauges], columns are reach ids (as for KalmanFilter)
    Q_diag       : scalar or [n] diagonal of the model-noise covariance
    R_cov        : [m][m] observation-noise covariance
    obs_noise    : optional [len(measurements)][m][M_total] perturbations added to the interpolated
                   measurements per member (supplied as data so CPU and GPU consume identical numbers);
                   zeros if omitted (deterministic ensemble update)
    every        : pd.Timedelta cadence (e.g. hourly); None = every step as the reference (da.py:56-61)
    group        : torch.distributed process group when members are sharded over ranks (this rank
                   holds columns [rank*M, (rank+1)*M) of the global ensemble); None = the default group
                   if torch.distributed is initialised; False = never sharded (independent ensembles)
    """

    def __init__(self, model, measurements, Q_diag, R_cov, obs_noise=None, every=None, group=None):
        import torch
        self._torch = torch
        self.model = model
        self.reach_indices, perm = _gauge_setup(model, measurements)
        self.measurements = measurements.iloc[:, perm]
        self.num_measurements = m = self.measurements.shape[1]
        if np.shape(R_cov) != (m, m):
            raise ValueError(f'`R_cov` must be ({m}, {m}), got {np.shape(R_cov)}')
        self.reach_indices = np.ascontiguousarray(self.reach_indices, dtype=np.int64)
        self.every = every
        self.group = group
        self.rank, self.world = 0, 1
        if group is False:                     # this rank's ensemble is whole (e.g. one independent basin per rank)
            self.group = group = None
        elif group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.rank = torch.distributed.get_rank(group)
            self.world = torch.distributed.get_world_size(group)
        self.M = model.members
        self.Mtot = self.M * self.world
        if self.Mtot < 2:
            # the sample covariance divides by Mtot - 1: refused here, before any device work, rather than by the
            # first solve, after the assimilation loop has already routed a window
            raise ValueError(f'an ensemble Kalman filter needs at least 2 members in all, got {self.Mtot} '
                             f'({self.M} per rank x {self.world} ranks)')
        Rp =np.asarray(R_cov, dtype=np.float64)[perm, :][:, perm]
        q = np.broadcast_to(np.asarray(Q_diag, dtype=np.float64), (model.n,))
        self._R = torch.as_tensor(np.ascontiguousarray(Rp), device='cuda')
        self._qs = torch.as_tensor(np.ascontiguousarray(q[self.reach_indices]), device='cuda')
        self._noise = None
        if obs_noise is not None:
            noise = np.asarray(obs_noise, dtype=np.float64)[:, perm, :]
            assert noise.shape == (len(self.measurements), m, self.Mtot)
            self._noise = noise
        n, Mt = model.n, self.Mtot
        f64 = dict(dtype=torch.float64, device='cuda')
        self._rowsum = torch.empty(n, **f64)
        self._HX = torch.empty((m, self.M), **f64)
        self._HXall = torch.empty((m, Mt), **f64) if self.world > 1 else self._HX
        self._work = torch.empty(model.network.enkf_work_size(m, Mt), **f64)
        # D = R + diag(Q[s,s]) never changes: its inverse (diagonal or dense) lets the update solve in
        # ensemble space when the ensemble is smaller than the gauge network
        D = Rp + np.diag(q[self.reach_indices])
        if np.count_nonzero(D - np.diag(np.diagonal(D))) == 0:
            self._Dinv, self._dinv_kind = torch.as_tensor(1.0 / np.diagonal(D), device='cuda').contiguous(), 1
        else:
            self._Dinv, self._dinv_kind = inverse(torch.as_tensor(np.ascontiguousarray(D), device='cuda').clone()), 2
        self._W = torch.empty((m, Mt), **f64)
        self._T = torch.empty((Mt, Mt), **f64)
        self._G = model.network.alloc_state(self.M)
        self._Xall = None
        self.n_updates = 0
        self.datetime = copy.deepcopy(model.datetime)
        # member-sharded ensembles: "peers" = the transform reads the other shards' state rows where they live
        # (symmetric memory over NVLink, two buffers alternating), "allgather" = NCCL all-gather first
        self.update_path = None
        self._sym = None
        if self.world > 1:
            self.update_path = 'allgather'
            import os
            if os.environ.get('TXH_MEMBER_UPDATE', 'peers') == 'peers':
                self._setup_peers()

    def _setup_peers(self):
        """Two symmetric-memory state buffers per rank (torch.distributed._symmetric_memory): every rank can load
        from every other rank's buffers inside a kernel.  The model's outflow state moves into the first one.
        Collective; any failure leaves the all-gather path in place."""
        torch = self._torch
        mdl = self.model
        try:
            import torch.distributed._symmetric_memory as symm
            dist = torch.distributed
            grp = self.group if self.group is not None else dist.group.WORLD
            mdl._ensure_device()
            O = mdl._dev['O']
            bufs = []
            for _ in range(2):
                t = symm.empty(tuple(O.shape), dtype=torch.float64, device=O.device)
                hdl = symm.rendezvous(t, grp)
                ptrs = [int(p) for p in hdl.buffer_ptrs]
                if len(ptrs) != self.world or ptrs[self.rank] != t.data_ptr():
                    raise RuntimeError('unexpected symmetric-memory layout')
                bufs.append((t, ptrs, hdl))
            ok = torch.ones(1, device=O.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
            if float(ok.item()) != 1.0:
                raise RuntimeError('a peer could not set up symmetric memory')
            bufs[0][0].copy_(O)
            mdl._dev['O'] = bufs[0][0]
            self._sym, self._cur = bufs, 0
            self.update_path = 'peers'
        except Exception as e:                    # noqa: BLE001 -- optional fast path: report and carry on
            logger.warning('member-sharded update falls back to all-gather: %s', e)
            self._sym = None

    def release_peers(self):
        """Collective.  A member-sharded filter on the peer-read path owns buffers other ranks load from inside
        their kernels: before it goes away every rank must have finished its last update.  Synchronises the
        device, meets the other ranks at a barrier, and moves the state back into an ordinary tensor."""
        if self._sym is None:
            return
        torch = self._torch
        torch.cuda.synchronize()
        torch.distributed.barrier(group=self.group)
        mdl = self.model
        if mdl._dev is not None:
            mdl._dev['O'] = mdl._dev['O'].clone()
        self._sym = None
        self.update_path = 'allgather'

    @property
    def latest_timestamp(self):
        return self.measurements.index[-1]

    def _due(self):
        t = self.model.datetime
        if t > self.latest_timestamp:
            return False
        if self.every is not None and (t.value % int(self.every.value)) != 0:
            return False
        return True

    def __on_simulation_start__(self):
        return self.filter() if self._due() else None

    def __on_step_end__(self):
        return self.filter() if self._due() else None

    def perturbed_observations(self, datetime):
        """[m][Mtot] per-member observations at `datetime` (interpolated measurements + supplied noise)."""
        x = float(datetime.value)
        Z = interpolate_sample(x, self._meas_times, self._meas_values)
        Zp = np.repeat(Z[:, None], self.Mtot, axis=1)
        if self._noise is not None:
            flat = self._noise.reshape(self._noise.shape[0], -1)
            Zp = Zp + interpolate_sample(x, self._meas_times, flat).reshape(Z.size, self.Mtot)
        return np.ascontiguousarray(Zp)

    def stats_scale(self):
        return 1.0 / self.Mtot if self.world == 1 else 1.0

    def filter(self, Zp_dev=None, stats_fresh=False):
        """One ensemble update on the device.  `Zp_dev` ([m][Mtot] CUDA tensor) overrides the
        interpolated observations (used by the fast path that pre-stages them).  `stats_fresh`: the row
        sums of the forecast are already in `self._rowsum` (written by the routing launch)."""
        torch = self._torch
        mdl = self.model
        net = mdl.network
        O, I = mdl.device_state
        if self._sym is not None and O is not self._sym[self._cur][0]:
            # the state was rebound to another tensor: bring it back into the shared buffer BEFORE the all-reduce
            # below, which orders it ahead of every peer's transform
            self._sym[self._cur][0].copy_(O)
            mdl._dev['O'] = O = self._sym[self._cur][0]
        M, Mt, m = self.M, self.Mtot, self.num_measurements
        if Zp_dev is None:
            Zp_dev = torch.as_tensor(self.perturbed_observations(mdl.datetime), device='cuda')
        dist = torch.distributed
        # one pass over the state: row sums (already the mean when the ensemble is not sharded) + gauge rows
        net.enkf_stats(O, M, self.reach_indices, None if stats_fresh else self._rowsum, self._HX,
                       scale=self.stats_scale())
        Xall, ldx, xstride, gather = None, 0, 0, None
        mean = self._rowsum
        if self.world > 1 and self._sym is not None:
            # The all-reduce of the row sums doubles as the cross-GPU barrier: once it has completed on this
            # rank, every rank's forecast (written before its contribution, in stream order) is final, and every
            # rank has left the previous update, i.e. nobody reads the buffer this update is about to overwrite.
            cur, nxt = self._sym[self._cur], self._sym[self._cur ^ 1]
            mean, self._HXall = combine_statistics(self._rowsum, self._HX, Mt, group=self.group)
            net.enkf_solve(m, Mt, self._HXall, Zp_dev, mean, self.reach_indices, self._qs, self._R, self._work,
                           self._W, self._T, self._Dinv, self._dinv_kind)
            net.enkf_apply_peers(cur[0], nxt[0], I, M, cur[1], Mt, self.rank * M, mean, self._T, self.reach_indices,
                                 self._qs, self._W, self._G)
            mdl._dev['O'] = nxt[0]
            self._cur ^= 1
            mdl._device_advanced()
            self.n_updates += 1
            self.datetime = mdl.datetime
            return
        if self.world > 1:
            # ensemble mean over all shards (all-reduce) + every shard's gauge rows (all-gather); the state rows
            # of every shard follow on the collective stream while the small system is solved
            mean, self._HXall = combine_statistics(self._rowsum, self._HX, Mt, group=self.group)
            ld = net.row_stride(M)
            if self._Xall is None:
                self._Xall = torch.empty((self.world, mdl.n, ld), dtype=torch.float64, device='cuda')
            gather = dist.all_gather_into_tensor(self._Xall, O, group=self.group, async_op=True)
            Xall, ldx, xstride = self._Xall, ld, mdl.n * ld
        net.enkf_solve(m, Mt, self._HXall, Zp_dev, mean, self.reach_indices, self._qs, self._R, self._work,
                       self._W, self._T, self._Dinv, self._dinv_kind)
        if gather is not None:
            gather.wait()
        net.enkf_apply(O, I, M, Xall, ldx, Mt, self.rank * M, mean, self._T, self.reach_indices, self._qs,
                       self._W, self._G, x_block_stride=xstride)
        mdl._device_advanced()
        self.n_updates += 1
        self.datetime = mdl.datetime


class BatchedKalmanFilters:
    """The dense `KalmanFilter`s of several INDEPENDENT sub-models advanced in lockstep (the reference's operating
    mode, app/app.py:130-141: one filter per sub-model of a split network, `filter()` after every step,
    da.py:49-61).  The sub-models are disjoint forests, so their union is one network: one routing launch steps
    them all, and ONE chain of launches (`txh_kfb_filter`) runs every filter -- the columns of all covariance
    blocks ride as members of the same two routing launches (`_aqat_par`, nutils.py:194-214), the m x m inverses
    run one CTA per block -- instead of a 14-launch chain per sub-model.

    `models`: Muskingum objects whose only callback is a `KalmanFilter` under the key it was bound with, all at
    the same `datetime` with the same `timedelta`.  `run(inputs)` does for each of them what
    `simulate_iter(inputs[name])` + the filter's hooks do, and leaves models and filters in the state the
    per-model path leaves them in."""

    def __init__(self, models):
        import torch
        from . import _lib as L
        from .muskingum import Muskingum
        self._torch, self._L = torch, L
        self.models = list(models)
        self.filters = []
        for mdl in self.models:
            kfs = list(mdl.callbacks.values())
            if len(kfs) != 1 or type(kfs[0]) is not KalmanFilter or mdl.members != 1:
                raise ValueError('every model needs exactly one KalmanFilter callback and a single member')
            self.filters.append(kfs[0])
        t0, dt = self.models[0].datetime, self.models[0].timedelta
        if any(m.datetime != t0 or m.timedelta != dt for m in self.models):
            raise ValueError('models must share datetime and timedelta')
        sizes = [m.n for m in self.models]
        self.row0 = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        d = {'name': 'union', 'datetime': t0, 'timedelta': dt,
             'reach_ids': [f'{k}:{r}' for k, m in enumerate(self.models) for r in m.reach_ids],
             'startnodes': np.arange(self.row0[-1], dtype=np.int64),
             'endnodes': np.concatenate([m.endnodes + self.row0[k] for k, m in enumerate(self.models)]).astype(np.int64),
             'K': np.concatenate([m.K for m in self.models]), 'X': np.concatenate([m.X for m in self.models]),
             'o_t': np.concatenate([m._peek_state('o_t_next') for m in self.models])}
        self.union = u = Muskingum(d, load_optional=False)
        for name in ('alpha', 'beta', 'chi', 'gamma'):                 # user-mutated coefficients travel too
            setattr(u, name, np.concatenate([getattr(m, name) for m in self.models]))
        u.init_states(o_t_next=d['o_t'], i_t_next=np.concatenate([m._peek_state('i_t_next') for m in self.models]))
        u.o_t_prev = np.concatenate([m._peek_state('o_t_prev') for m in self.models])
        u.i_t_prev = np.concatenate([m._peek_state('i_t_prev') for m in self.models])
        lib = L.load()
        n_k = L.as_i64(sizes)
        m_k = L.as_i64([kf.num_measurements for kf in self.filters])
        obs = L.as_i64(np.concatenate([kf.reach_indices for kf in self.filters]))
        self.g0 = np.concatenate([[0], np.cumsum(m_k)]).astype(np.int64)
        import ctypes
        h = ctypes.c_void_p()
        L.check(lib.txh_kfb_create(u.network.handle, len(self.models), L.ptr_i64(n_k), L.ptr_i64(m_k), L.ptr_i64(obs),
                                   ctypes.byref(h)))
        self.handle = h
        self._lib = lib
        for k, kf in enumerate(self.filters):
            for which, t in ((0, kf._P), (1, kf._Q), (2, kf._R)):
                a = L.as_f64(t.cpu().numpy())
                L.check(lib.txh_kfb_set(h, k, which, L.ptr_f64(a), None))
        self.n_updates = 0
        self._ran = np.zeros(len(self.filters), dtype=bool)     # the filters that have updated at least once

    def close(self):
        if getattr(self, 'handle', None):
            self._lib.txh_kfb_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _get(self, k, which, shape):
        out = np.empty(shape, dtype=np.float64)
        self._L.check(self._lib.txh_kfb_get(self.handle, k, which, self._L.ptr_f64(out), None))
        return out

    def filter(self):
        """`KalmanFilter.filter` (da.py:91-136) of every filter that is due at the union model's time."""
        import ctypes
        u = self.union
        active = np.array([u.datetime <= kf.latest_timestamp for kf in self.filters], dtype=np.uint8)
        if not active.any():
            return
        z = np.concatenate([kf.interpolate_input(u.datetime) if a else np.zeros(kf.num_measurements)
                            for kf, a in zip(self.filters, active)])
        u._ensure_device()
        u._sync_coeffs()
        d = u._dev
        from .network import _cuda_ptr, _stream_ptr
        self._L.check(self._lib.txh_kfb_filter(self.handle, active.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)),
                                               self._L.ptr_f64(self._L.as_f64(z)), _cuda_ptr(d['O']), _cuda_ptr(d['I']),
                                               _stream_ptr()))
        u._device_advanced()
        self._ran |= active.astype(bool)
        for kf, a in zip(self.filters, active):
            if a:
                kf.datetime = u.datetime
        self.n_updates += 1

    def run(self, inputs):
        """`inputs`: {model name: forcing DataFrame} with one common index.  Returns {name: (values [steps+1][n], times)}:
        the rows AsyncSimulation records -- row 0 is the state after the simulation-start hooks."""
        from .nutils import interpolate_sample
        u = self.union
        frames = [inputs[m.name][m.reach_ids] for m in self.models]
        index = frames[0].index
        if any(not f.index.equals(index) for f in frames):
            raise ValueError('the forcing frames of a batched generation must share one index')
        times = index.astype(int).astype(float).values
        table = np.ascontiguousarray(np.concatenate([f.values for f in frames], axis=1), dtype=np.float64)
        end_time = index.max()
        torch = self._torch
        nsteps = 0 if not end_time > u.datetime else int(-((u.datetime - end_time) // u.timedelta))
        # the hydrographs are recorded on the device (one unpack launch per step, no host round trip in the loop)
        rec = torch.empty((nsteps + 1, u.n, 1), dtype=torch.float64, device='cuda')

        def record(row):
            u._ensure_device()
            u.network.unpack_dev(u._dev['O'], 1, rec[row])

        self.filter()                                              # __on_simulation_start__ of every filter
        record(0)
        stamps, k = [u.datetime], 0
        while u.datetime < end_time:
            p = interpolate_sample(float((u.datetime + u.timedelta).value), times, table)
            u.step_iter(p)
            self.filter()                                          # __on_step_end__
            k += 1
            record(k)
            stamps.append(u.datetime)
        self._write_back()
        values = rec[:k + 1, :, 0].cpu().numpy()
        return {m.name: (values[:, self.row0[i]:self.row0[i + 1]], list(stamps)) for i, m in enumerate(self.models)}

    def _write_back(self):
        """Sub-models and their filters end up where the per-model path would have left them."""
        torch = self._torch
        u = self.union
        u.network.check()
        state = {key: u._peek_state(key) for key in ('o_t_next', 'i_t_next', 'o_t_prev', 'i_t_prev')}
        for k, (m, kf) in enumerate(zip(self.models, self.filters)):
            sl = slice(self.row0[k], self.row0[k + 1])
            m.init_states(o_t_next=state['o_t_next'][sl], i_t_next=state['i_t_next'][sl])
            m.o_t_prev = np.array(state['o_t_prev'][sl]); m.i_t_prev = np.array(state['i_t_prev'][sl])
            m.datetime = u.datetime
            n, mm = m.n, kf.num_measurements
            kf._P = torch.as_tensor(self._get(k, 0, (n, n)), device='cuda')
            if self._ran[k]:                     # P before, K, dz and gain of its last update, as the per-model path
                kf._P_prev = torch.as_tensor(self._get(k, 3, (n, n)), device='cuda')
                kf._K_d = torch.as_tensor(self._get(k, 4, (n, mm)), device='cuda')
                kf._dz_d = torch.as_tensor(self._get(k, 5, (mm,)), device='cuda')
                kf._gain_d = torch.as_tensor(self._get(k, 6, (n,)), device='cuda')
