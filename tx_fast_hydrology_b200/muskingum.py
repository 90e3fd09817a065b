"""`Muskingum`: drop-in for the reference's model object (tx_fast_hydrology/muskingum.py:20-606)
whose routing runs on the GPU.

Same constructor, attributes, `step` / `simulate` entry points, callback firing
order and state save/load behaviour as the reference; the numba call at
muskingum.py:456 (`_ax_bu`) is replaced by `txh_route_step` and the Python loop of
`simulate_iter` (muskingum.py:527-533) gains a device-resident fast path, `run()`,
that keeps Python out of the per-step loop.

State lives in HBM in the library's schedule order.  `o_t_next`, `i_t_next`,
`o_t_prev`, `i_t_prev` are numpy views of it, materialised on access; once
looked at they may have been mutated in place (KalmanFilter does, da.py:125-126),
so the host copy is pushed back before the next launch.  Reference quirks kept
on purpose (SURVEY.md appendix A): self-loop inflow in `init_states` (A.3),
`dt = timedelta.seconds` (A.4), the variable-timestep behaviour of `step` (A.5),
`load_state` aliasing (A.12), the never-raised ValueError in `simulate` (A.13).

Extension: `members=M` batches M ensemble members; state arrays are then (n, M).
"""
import copy as _copy
import datetime as _dt
import json
import logging
import os
import uuid

import numpy as np
import pandas as pd

from .callbacks import BaseCallback
from .network import Forcing, RiverNetwork

DEFAULT_START_TIME = pd.to_datetime(0., utc=True)
DEFAULT_TIMEDELTA = pd.to_timedelta(3600, unit='s')

_REQUIRED = ('name', 'datetime', 'timedelta', 'reach_ids', 'startnodes', 'endnodes', 'K', 'X', 'o_t')
_OPTIONAL = ('paths', 'dx')


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("tx_fast_hydrology_b200 needs a CUDA device: there is no CPU fallback")
    return torch


class Muskingum:
    def __init__(self, data, load_optional=True, create_state_space=False, sparse=False,
                 members=1, sched_params=None):
        self.sparse = sparse
        self.callbacks = {}
        self.saved_states = {}
        self.sinks = []
        self.sources = []
        self.members = int(members)
        self._sched_params = sched_params
        if isinstance(data, dict):
            self.load_model(data, load_optional=load_optional)
        elif isinstance(data, str):
            self.load_model_file(data, load_optional=load_optional)
        else:
            raise TypeError('`data` must be a file path or dictionary.')
        self.logger = logging.getLogger(self.name)
        n = self.n
        # dense A/B of muskingum.py:163-168 are out of scope (O(n^2), unused by the hot path)
        self.A = None
        self.B = None
        if create_state_space:
            raise NotImplementedError('dense state-space matrices are not built by the GPU drop-in')
        self._coef = {}
        self._coef_dirty = True
        self.alpha = np.zeros(n, dtype=np.float64)
        self.beta = np.zeros(n, dtype=np.float64)
        self.chi = np.zeros(n, dtype=np.float64)
        self.gamma = np.zeros(n, dtype=np.float64)
        self._dev = None                 # device tensors, created on first use
        self._dev_valid = False
        self._host_ref = {}
        shape = (n,) if self.members == 1 else (n, self.members)
        o0 = np.asarray(self._o_t_initial, dtype=np.float64)
        if o0.shape != shape:
            o0 = np.broadcast_to(o0.reshape(n, -1), (n, self.members)).reshape(shape)
        # materialised numpy views of the state; "dirty" = may differ from the device copy
        self._host = {'o_t_next': np.array(o0, dtype=np.float64), 'i_t_next': np.zeros(shape),
                      'o_t_prev': np.zeros(shape), 'i_t_prev': np.zeros(shape)}
        self._host_dirty = True
        self.init_states(o_t_next=self._host['o_t_next'])
        self._host['o_t_prev'] = self._host['o_t_next'].copy()
        self._host['i_t_prev'] = self._host['i_t_next'].copy()
        self.compute_muskingum_coeffs()
        self.save_state()

    # ------------------------------------------------------------------ metadata
    @property
    def info(self):
        return {'name': self.name, 'datetime': self.datetime, 'timedelta': self.timedelta,
                'reach_ids': self.reach_ids, 'startnodes': self.startnodes, 'endnodes': self.endnodes,
                'K': self.K, 'X': self.X, 'o_t': self.o_t_next, 'dx': self.dx, 'paths': self.paths}

    @property
    def name(self):
        return self._name

    @name.setter
    def name(self, new_name):
        if not isinstance(new_name, str):
            new_name = str(new_name)
        self._name = new_name

    @property
    def datetime(self):
        return self._datetime

    @datetime.setter
    def datetime(self, new_datetime):
        if not isinstance(new_datetime, pd.Timestamp):
            raise TypeError('New datetime must be of type `pd.Timestamp`')
        if new_datetime.tz != _dt.timezone.utc:
            raise ValueError('New datetime must be UTC.')
        self._datetime = new_datetime

    @property
    def timedelta(self):
        return self._timedelta

    @timedelta.setter
    def timedelta(self, new_timedelta):
        if not isinstance(new_timedelta, pd.Timedelta):
            raise TypeError('New timedelta must be of type `pd.Timedelta`')
        self._timedelta = new_timedelta

    @property
    def dt(self):
        return float(self.timedelta.seconds)          # muskingum.py:247-250 (seconds component)

    # ------------------------------------------------------------------ state views
    def _materialise(self):
        if not self._host:
            net, M, d = self.network, self.members, self._dev
            net.check()
            shape = (self.n,) if M == 1 else (self.n, M)
            self._host = {
                'o_t_next': net.unpack_host(d['O'], M).reshape(shape),
                'i_t_next': net.unpack_host(d['I'], M).reshape(shape),
                'o_t_prev': net.unpack_host(d['Op'], M).reshape(shape),
                'i_t_prev': net.unpack_host(d['Ip'], M).reshape(shape),
            }
            # what the device holds: an array handed out and still equal to this at the next launch is not
            # uploaded again (callbacks that only READ the state cost no PCIe traffic)
            self._host_ref = {k: v.copy() for k, v in self._host.items()}
        # a caller holding these arrays may write into them (da.py:125-126 does)
        self._host_dirty = True
        return self._host

    def _state_get(self, key):
        return self._materialise()[key]

    def _peek_state(self, key):
        """A private copy of a state array that leaves the device copy authoritative."""
        dirty = self._host_dirty
        v = np.array(self._materialise()[key])
        self._host_dirty = dirty
        return v

    def _state_set(self, key, value):
        h = self._materialise()
        h[key] = value
        self._host_ref.pop(key, None)
        self._host_dirty = True

    o_t_next = property(lambda self: self._state_get('o_t_next'),
                        lambda self, v: self._state_set('o_t_next', v))
    i_t_next = property(lambda self: self._state_get('i_t_next'),
                        lambda self, v: self._state_set('i_t_next', v))
    o_t_prev = property(lambda self: self._state_get('o_t_prev'),
                        lambda self, v: self._state_set('o_t_prev', v))
    i_t_prev = property(lambda self: self._state_get('i_t_prev'),
                        lambda self, v: self._state_set('i_t_prev', v))

    @property
    def o_t(self):
        return self.o_t_next

    @o_t.setter
    def o_t(self, new_o_t):
        try:
            new_o_t = np.asarray(new_o_t, dtype=np.float64)
        except Exception:
            raise TypeError('New `o_t` must be convertible to float64 np.ndarray')
        self.o_t_next = new_o_t

    # ------------------------------------------------------------------ loading
    def load_model(self, obj, load_optional=True):
        defaults = {'name': str(uuid.uuid4()), 'datetime': DEFAULT_START_TIME,
                    'timedelta': DEFAULT_TIMEDELTA, 'dx': None, 'paths': []}
        if not set(_REQUIRED).issubset(obj.keys()):
            raise ValueError(f'Model field must contain fields {set(_REQUIRED)}')
        for key, dtype in (('startnodes', np.int64), ('endnodes', np.int64), ('K', np.float64),
                           ('X', np.float64), ('o_t', np.float64)):
            v = obj[key]
            if not isinstance(v, np.ndarray) or v.dtype != dtype:
                raise TypeError('Typing of input arrays is incorrect.')
        n = obj['startnodes'].size
        if not (obj['endnodes'].size == obj['K'].size == obj['X'].size == n) or obj['o_t'].shape[0] != n:
            raise ValueError('Arrays are not the same length')
        fields = _REQUIRED + (_OPTIONAL if load_optional else ())
        for field in fields:
            value = obj.setdefault(field, defaults[field]) if field in defaults else obj[field]
            if field == 'o_t':
                self.__dict__['_o_t_initial'] = value
            else:
                setattr(self, field, value)
        if not load_optional:
            self.dx, self.paths = None, []
        self.n = n
        if not (self.startnodes == np.arange(n)).all():
            # the reference silently mis-indexes in this case (nutils.py:73-83, SURVEY.md A.1)
            raise ValueError('`startnodes` must equal arange(n)')
        self.network = RiverNetwork(self.endnodes, self._sched_params)
        self.indegree = self.compute_indegree(self.startnodes, self.endnodes)

    def load_model_file(self, file_path, load_optional=True):
        self.load_model(load_model_file(file_path, load_optional=load_optional))

    def dump_model_file(self, file_path, dump_optional=True):
        return dump_model_file(self.info, file_path, dump_optional=dump_optional)

    @classmethod
    def from_model_file(cls, file_path, load_optional=True, **kwargs):
        return cls(load_model_file(file_path, load_optional=load_optional), **kwargs)

    def compute_indegree(self, startnodes, endnodes):
        """muskingum.py:322-330, from the exact-integer topology pass."""
        return self.network.indegree()

    # ------------------------------------------------------------------ coefficients
    def compute_alpha(self, K, X, dt):
        return (dt - 2 * K * X) / (2 * K * (1 - X) + dt)

    def compute_beta(self, K, X, dt):
        return (dt + 2 * K * X) / (2 * K * (1 - X) + dt)

    def compute_chi(self, K, X, dt):
        return (2 * K * (1 - X) - dt) / (2 * K * (1 - X) + dt)

    def compute_gamma(self, K, X, dt):
        return dt / (K * (1 - X) + dt / 2)

    def compute_muskingum_coeffs(self, K=None, X=None, dt=None):
        self.logger.info('Computing Muskingum coefficients...')
        K = self.K if K is None else K
        X = self.X if X is None else X
        dt = self.dt if dt is None else dt
        a, b, c, g = self.network.compute_coeffs(K, X, dt)     # muskingum.py:332-360 on the handle
        self.alpha, self.beta, self.chi, self.gamma = a, b, c, g
        self._coef_dirty = False                               # the handle already holds exactly these

    def set_transmissive_boundary(self, index):
        """muskingum.py:567-571 (which writes the four arrays in place)."""
        for name, value in (('alpha', 1.), ('beta', 0.), ('chi', 0.), ('gamma', 0.)):
            arr = np.array(self._coef[name])
            arr[index] = value
            setattr(self, name, arr)

    # alpha / beta / chi / gamma: the arrays the kernels read live on the device, so a change has to be seen.  The
    # attributes hand out READ-ONLY arrays and assignment installs a copy: `model.alpha = new_array` (or
    # compute_muskingum_coeffs / set_transmissive_boundary) is how coefficients change; an in-place write from outside
    # raises numpy's "assignment destination is read-only" instead of being silently missed.  (Comparing four arrays
    # of n doubles before every launch, the alternative, cost 4.5 ms per call at CONUS scale.)
    def _coef_get(name):
        return lambda self: self._coef[name]

    def _coef_set(name):
        def setter(self, value):
            arr = np.array(value, dtype=np.float64).reshape(-1)
            if arr.size != self.n:
                raise ValueError(f'`{name}` must hold {self.n} values, got {arr.size}')
            arr.flags.writeable = False
            self._coef[name] = arr
            self._coef_dirty = True
        return setter

    alpha = property(_coef_get('alpha'), _coef_set('alpha'))
    beta = property(_coef_get('beta'), _coef_set('beta'))
    chi = property(_coef_get('chi'), _coef_set('chi'))
    gamma = property(_coef_get('gamma'), _coef_set('gamma'))
    del _coef_get, _coef_set

    def _sync_coeffs(self):
        """Re-install the coefficients on the handle after a change (see the properties above)."""
        if self._coef_dirty:
            self.network.set_coeffs(self.alpha, self.beta, self.chi, self.gamma)
            self._coef_dirty = False

    # ------------------------------------------------------------------ device plumbing
    def _ensure_device(self):
        torch = _torch()
        net, M = self.network, self.members
        if self._dev is None:
            self._dev = {k: net.alloc_state(M) for k in ('O', 'I', 'Op', 'Ip')}
            self._dev_valid = False
        if self._host and (self._host_dirty or not self._dev_valid):
            h, d = self._host, self._dev
            ref = self._host_ref if self._dev_valid else {}
            for hk, dk in (('o_t_next', 'O'), ('i_t_next', 'I'), ('o_t_prev', 'Op'), ('i_t_prev', 'Ip')):
                v = np.asarray(h[hk], dtype=np.float64)
                if v.size != self.n * M:
                    raise ValueError(f'`{hk}` must hold {self.n} x {M} values, got shape {np.shape(h[hk])}')
                if hk in ref and ref[hk].shape == v.shape and np.array_equal(ref[hk], v):
                    continue                                   # untouched since it was downloaded
                net.pack_host(v.reshape(self.n, M), M, d[dk])
                ref[hk] = v.copy()
            self._host_ref = ref
        self._dev_valid = True
        self._host_dirty = False
        return torch

    def _device_advanced(self):
        self._host = {}
        self._host_ref = {}
        self._host_dirty = False

    def init_states(self, o_t_next=None, i_t_next=None):
        """muskingum.py:410-419: i = scatter-add of o over endnodes (self-loops included)."""
        h = self._materialise()
        full = (self.n,) if self.members == 1 else (self.n, self.members)
        o = np.zeros(full) if o_t_next is None else np.array(
            np.broadcast_to(np.asarray(o_t_next, dtype=np.float64).reshape(self.n, -1),
                            (self.n, self.members)).reshape(full))
        h['o_t_next'] = o
        if i_t_next is None:
            i = np.zeros(full)
            np.add.at(i, self.endnodes, o[self.startnodes])
            h['i_t_next'] = i
        else:
            h['i_t_next'] = np.array(np.asarray(i_t_next, dtype=np.float64).reshape(full))
        for k in ('o_t_prev', 'i_t_prev'):
            if k not in h or np.shape(h[k]) != full:
                h[k] = np.zeros(full)
        self._host_ref = {}
        self._host_dirty = True

    # ------------------------------------------------------------------ stepping
    def step_iter(self, p_t_next, timedelta=None):
        """muskingum.py:435-465 with the numba call replaced by one device launch."""
        if timedelta is None:
            timedelta = self.timedelta
            dt = self.dt
        else:
            dt = float(timedelta.seconds)
        if dt != self.dt:
            self.logger.warning('Timestep has changed. Recomputing Muskingum coefficients.')
            self.compute_muskingum_coeffs(dt=dt)
        for _, callback in self.callbacks.items():
            callback.__on_step_start__()
        torch = self._ensure_device()
        self._sync_coeffs()
        d, net, M = self._dev, self.network, self.members
        d['Op'].copy_(d['O'])
        d['Ip'].copy_(d['I'])
        q_host = np.ascontiguousarray(p_t_next, dtype=np.float64)
        if q_host.shape != (self.n,):
            raise ValueError(f'`p_t_next` must be a vector of {self.n} lateral inflows, got shape {q_host.shape}')
        q = torch.from_numpy(q_host).cuda()
        net.route_step(d['O'], d['I'], M, q)
        self._device_advanced()
        self.datetime += timedelta
        for _, callback in self.callbacks.items():
            callback.__on_step_end__()
        self.logger.debug('Stepped to time %s', self.datetime)

    def step(self, p_t_next, timedelta=None):
        return self.step_iter(p_t_next, timedelta=timedelta)

    def simulate_iter(self, dataframe, start_time=None, end_time=None, o_t_init=None, **kwargs):
        """muskingum.py:499-536: generator yielding `self` after every step."""
        assert isinstance(dataframe.index, pd.DatetimeIndex)
        assert (dataframe.index.tz == _dt.timezone.utc)
        cols = pd.Index(dataframe.columns)
        assert cols.get_indexer(pd.Index(self.reach_ids)).min() >= 0
        if end_time is None:
            end_time = dataframe.index.max()
        elif not isinstance(end_time, pd.Timestamp):
            raise TypeError('`end_time` must be of type `pd.Timestamp`')
        if start_time is not None:
            self.datetime = start_time          # (the reference builds, but never raises, a ValueError here)
        if o_t_init is not None:
            self.init_states(o_t_next=o_t_init)
        for _, callback in self.callbacks.items():
            callback.__on_simulation_start__()
        if getattr(self, '_capture_start', False):
            # AsyncSimulation's first output row is the state AFTER the simulation-start hooks: the reference stores a
            # reference to o_t_next there and a filter bound to the model corrects that array in place
            # (simulation.py:126-127, da.py:124-126)
            self._start_outflow = self._peek_state('o_t_next')
        dataframe = dataframe[self.reach_ids]
        times = dataframe.index.astype(int).astype(float).values
        table = np.ascontiguousarray(dataframe.values, dtype=np.float64)
        from .nutils import interpolate_sample
        while self.datetime < end_time:
            next_timestep = self.datetime + self.timedelta
            p_t_next = interpolate_sample(float(next_timestep.value), times, table)
            self.step_iter(p_t_next, **kwargs)
            yield self
        for _, callback in self.callbacks.items():
            callback.__on_simulation_end__()

    def simulate(self, dataframe, start_time=None, end_time=None, o_t_init=None, **kwargs):
        return self.simulate_iter(dataframe, start_time=start_time, end_time=end_time,
                                  o_t_init=o_t_init, **kwargs)

    # ------------------------------------------------------------------ device-resident fast path
    def make_forcing(self, dataframe=None, times_ns=None, table=None, member_mul=None):
        """Upload a forcing table once.  Either a DataFrame (as `simulate` takes) or raw arrays."""
        if dataframe is not None:
            dataframe = dataframe[self.reach_ids]
            times_ns = dataframe.index.astype(int).values
            table = dataframe.values
        return Forcing(self.network, times_ns, table, member_mul)

    def run(self, forcing, nsteps, record_reaches=None, record_every=1, method='linear'):
        """`nsteps` steps of the simulate loop (muskingum.py:527-533) in ONE persistent kernel
        launch: forcing interpolated on the device at t + dt, state updated in HBM, Python out
        of the loop.  Fires no per-step callbacks (bind-free fast path); returns the recorded
        outflows [nsteps // record_every][len(record_reaches)][members] as a CUDA tensor, or None.
        `o_t_prev` / `i_t_prev` afterwards hold the state before the last step only if nsteps == 1.
        `method`: 'linear' or 'nearest' (the row interpolation of nutils.interpolate_sample)."""
        if method not in ('linear', 'nearest'):
            raise ValueError(f"`method` must be 'linear' or 'nearest', got {method!r}")
        torch = self._ensure_device()
        self._sync_coeffs()
        d, net, M = self._dev, self.network, self.members
        rec = None
        if record_reaches is not None:
            rec = torch.zeros((nsteps // record_every, len(record_reaches), M), dtype=torch.float64,
                              device='cuda')
        step_ns = int(self.timedelta.value)
        if step_ns != int(round(self.dt * 1e9)):
            raise ValueError('run() needs a whole-second timestep below one day')
        if nsteps == 1:
            d['Op'].copy_(d['O']); d['Ip'].copy_(d['I'])
        net.route_run(d['O'], d['I'], M, forcing, int(self.datetime.value), step_ns, int(nsteps),
                      method=1 if method == 'linear' else 0, rec_reach=record_reaches,
                      rec_every=record_every, rec_out=rec)
        self._device_advanced()
        self.datetime = self.datetime + nsteps * self.timedelta
        return rec

    def _record_reaches(self, record_reaches, record_every, nsteps):
        """Checked reach list (reference order) of a recording run, as int64 numpy."""
        if isinstance(record_every, bool) or int(record_every) != record_every or record_every < 1:
            raise ValueError(f'`record_every` must be a positive integer, got {record_every!r}')
        idx = np.asarray(record_reaches.cpu() if hasattr(record_reaches, 'cpu') else record_reaches)
        if idx.ndim != 1 or idx.size == 0 or not np.issubdtype(idx.dtype, np.integer):
            raise ValueError('`record_reaches` must be a non-empty 1-D list of integer reach indices')
        idx = idx.astype(np.int64)
        n = len(self.reach_ids)
        if idx.min() < 0 or idx.max() >= n:
            raise ValueError(f'`record_reaches` out of range [0, {n})')
        if np.unique(idx).size != idx.size:
            raise ValueError('`record_reaches` lists a reach twice')
        if nsteps // int(record_every) < 1:
            raise ValueError(f'`record_every` = {record_every} records nothing in {nsteps} steps')
        return idx

    def run_assimilating(self, forcing, nsteps, enkf, every, observations, timers=None, observations_ready=None,
                         record_reaches=None, record_every=1, record_prior=False, smooth_lag=None):
        """Device-resident run with periodic ensemble assimilation: `every` routing steps in one
        persistent launch, then one `EnsembleKalmanFilter` update with `observations[k]` ([m][Mtot]
        CUDA tensor of per-member observations for the k-th update), repeated; nothing returns to
        the host in between.  Mirrors simulate + a KalmanFilter callback gated to every `every`-th
        step (the reference filters every step, da.py:56-61; SURVEY.md section 8c iv).
        `timers`: optional list; every 8th routing launch is bracketed by CUDA events -- the unsharded path
        keeps them in the library (`network.route_timings()` returns their durations), the sharded one appends
        (start, end) torch event pairs.
        `observations_ready`: optional `torch.cuda.Event` recorded after an upload of `observations` on another
        stream; the first update waits for it (the first routing window does not).
        `record_reaches` (reach indices, reference order): also record the ensemble hydrographs there and return
        `rec`, a CUDA tensor [nsteps // record_every][k][members]: after every `record_every`-th step what a simulate
        loop with the filter bound sees in `o_t_next` -- the forecast, or the posterior at an update step.  With
        `record_prior`, returns (rec, prior), prior [nsteps // every][k][members] the forecast each update started from.
        A member-sharded filter records this rank's members.  Without `record_reaches`, returns None.
        The Python loop (observations as a list, or a member-sharded filter) records every step of a window into a
        scratch buffer and copies the wanted steps out, and each of its routing calls uploads the slot map again and
        synchronises: correct, with per-window host work on a path that already has it; the in-library loop does this
        once per call.
        `smooth_lag` (steps, needs `record_reaches`): also return the hydrographs of the fixed-lag ensemble Kalman
        smoother, `smoothed` shaped like `rec`, as (rec, smoothed) or (rec, prior, smoothed): slot j (after step
        s = (j+1) record_every) conditioned on every update of the call after s up to s + smooth_lag, from the
        transforms the updates solved (txh_enks_smooth; DESIGN.md §4.4).  `rec` keeps the filtered hydrographs.  A
        lag of at least `nsteps` gives the fixed-interval smoother.  Not for a member-sharded filter."""
        if smooth_lag is not None:
            if isinstance(smooth_lag, bool) or not isinstance(smooth_lag, (int, np.integer)) or smooth_lag < 0:
                raise ValueError(f'`smooth_lag` must be a non-negative integer number of steps, got {smooth_lag!r}')
            if record_reaches is None:
                raise ValueError('`smooth_lag` smooths recorded hydrographs: it needs `record_reaches`')
            if getattr(enkf, 'world', 1) > 1:
                raise ValueError('`smooth_lag` is not available for a member-sharded filter (smoothing one rank\'s '
                                 'members needs every rank\'s)')
        ridx = None if record_reaches is None else self._record_reaches(record_reaches, record_every, nsteps)
        torch = self._ensure_device()
        self._sync_coeffs()
        d, net, M = self._dev, self.network, self.members
        step_ns = int(self.timedelta.value)
        t = int(self.datetime.value)
        nwin = nsteps // every
        rec = prior = None
        if ridx is not None:
            record_every = int(record_every)
            rec = torch.zeros((nsteps // record_every, ridx.size, M), dtype=torch.float64, device='cuda')
            if record_prior:
                prior = torch.zeros((nwin, ridx.size, M), dtype=torch.float64, device='cuda')
        # smoothing: update k's transform kept in T_hist[k]
        T_hist = None if smooth_lag is None else torch.empty((max(nwin, 1), M, M), dtype=torch.float64, device='cuda')

        def result():
            if rec is None:
                return None
            out = (rec, prior) if record_prior else (rec,)
            if T_hist is not None:
                out += (net.enks_smooth(M, nwin, every, T_hist, rec, record_every, smooth_lag, torch.empty_like(rec)),)
            return out if len(out) > 1 else rec
        if torch.is_tensor(observations) or isinstance(observations, np.ndarray):
            want = (enkf.num_measurements, enkf.Mtot)
            if observations.ndim != 3 or observations.shape[0] < nwin or tuple(observations.shape[1:]) != want:
                raise ValueError(f'`observations` must be [>= {nwin}][{want[0]}][{want[1]}], got {tuple(observations.shape)}')
        if (enkf.world == 1 and torch.is_tensor(observations) and observations.is_cuda and observations.is_contiguous()
                and observations.shape[0] >= nwin and observations.dtype == torch.float64):
            # one call: the loop below, in the library (txh_run_assimilating)
            if T_hist is not None:
                net.set_transform_history(T_hist)
            try:
                net.run_assimilating(d['O'], d['I'], M, forcing, t, step_ns, nsteps, every, enkf.reach_indices,
                                     observations, enkf._qs, enkf._R, enkf._Dinv, enkf._dinv_kind, enkf._rowsum,
                                     enkf._HX, enkf._work, enkf._W, enkf._T, enkf._G,
                                     time_every=8 if timers is not None else 0, obs_ready=observations_ready,
                                     rec_reach=ridx, rec_every=record_every, rec_out=rec, prior_out=prior)
            finally:
                if T_hist is not None:
                    net.set_transform_history(None)
            if T_hist is not None and nwin:
                enkf._T.copy_(T_hist[nwin - 1])             # the filter's last transform, as without smoothing
            enkf.n_updates += nwin
            self._datetime = pd.Timestamp(t + nsteps * step_ns, tz='UTC')
            enkf.datetime = self._datetime
            self._device_advanced()
            return result()
        if observations_ready is not None:
            torch.cuda.current_stream().wait_event(observations_ready)
        # recording: every step of a window into `win`, the steps that are multiples of record_every copied out of it
        win = None if rec is None else torch.empty((every, ridx.size, M), dtype=torch.float64, device='cuda')

        def route(nst, s0):
            if rec is None:
                net.route_run(d['O'], d['I'], M, forcing, t, step_ns, nst)
                return
            net.route_run(d['O'], d['I'], M, forcing, t, step_ns, nst, rec_reach=ridx, rec_every=1, rec_out=win)
            first = (s0 // record_every + 1) * record_every         # first recorded step of the window (1-based)
            steps = torch.arange(first, s0 + nst + 1, record_every, device='cuda')
            if steps.numel():
                rec.index_copy_(0, steps // record_every - 1, win.index_select(0, steps - s0 - 1))

        # the ensemble row sums ride on the last step of every routing launch
        net.set_stats_output(enkf._rowsum, enkf.stats_scale())
        for k in range(nwin):
            timed = timers is not None and k % 8 == 0      # events cost a few microseconds: sample every 8th launch
            if timed:
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
            route(every, k * every)
            if timed:
                e1.record()
                timers.append((e0, e1))
            t += every * step_ns
            self._datetime = pd.Timestamp(t, tz='UTC')
            if prior is not None:
                net.gather_rows(d['O'], M, ridx, prior[k])
            enkf.filter(observations[k], stats_fresh=True)
            if T_hist is not None:
                T_hist[k].copy_(enkf._T)
            s_end = (k + 1) * every
            if rec is not None and s_end % record_every == 0:
                # the posterior; a filter on the peer-read path has swapped the state buffer
                net.gather_rows(d['O'], M, ridx, rec[s_end // record_every - 1])
        net.set_stats_output(None)
        rest = nsteps - nwin * every
        if rest:
            route(rest, nwin * every)
            t += rest * step_ns
        self._datetime = pd.Timestamp(t, tz='UTC')
        self._device_advanced()
        return result()

    def upload_state(self, o_t_next, i_t_next=None):
        """`init_states` (muskingum.py:410-419) without the host round trip: `o_t_next` ([n][members],
        numpy or a pinned CPU torch tensor) goes straight to HBM and the inflows are the device
        scatter-add of the outflows over `endnodes` (self-loops included) unless given."""
        self._ensure_device()
        d, net, M = self._dev, self.network, self.members
        net.pack_host(o_t_next, M, d['O'])
        if i_t_next is None:
            net.init_inflows(d['O'], d['I'], M)
        else:
            net.pack_host(i_t_next, M, d['I'])
        self._device_advanced()

    def download_state(self, out_o=None, out_i=None):
        """(o_t_next, i_t_next) in reach order; `out_*` may be pinned CPU torch tensors [n][members]."""
        self._ensure_device()
        d, net, M = self._dev, self.network, self.members
        o = net.unpack_host(d['O'], M, out=out_o)
        i = net.unpack_host(d['I'], M, out=out_i) if out_i is not None else None
        return o, i

    @property
    def device_state(self):
        """(O, I) CUDA tensors [n][row_stride(members)] in schedule order (see DESIGN.md)."""
        self._ensure_device()
        return self._dev['O'], self._dev['I']

    # ------------------------------------------------------------------ checkpointing
    def save_state(self):
        """muskingum.py:573-580: snapshot (copies) + callback fan-out."""
        self.logger.info(f'Saving state for model {self.name} at time {self.datetime}...')
        self.saved_states['datetime'] = self.datetime
        self.saved_states['i_t_next'] = self._peek_state('i_t_next')
        self.saved_states['o_t_next'] = self._peek_state('o_t_next')
        for _, callback in self.callbacks.items():
            callback.__on_save_state__()

    def load_state(self):
        """muskingum.py:582-588: restore by reference (aliasing kept, SURVEY.md A.12)."""
        self.datetime = self.saved_states['datetime']
        self.i_t_next = self.saved_states['i_t_next']
        self.o_t_next = self.saved_states['o_t_next']
        self.logger.info(f'Loading state for model {self.name} at time {self.datetime}...')
        for _, callback in self.callbacks.items():
            callback.__on_load_state__()

    def bind_callback(self, callback, key='callback'):
        assert isinstance(callback, BaseCallback)
        self.callbacks[key] = callback

    def unbind_callback(self, key):
        return self.callbacks.pop(key)

    def copy(self):
        """Independent model with the same parameters, state (current and previous step), saved state and
        clock -- what `copy.deepcopy` gives on the reference object, minus the callbacks, sinks and sources,
        which hold references to other objects and are left unbound."""
        d = {k: _copy.deepcopy(v) for k, v in self.info.items()}
        d['o_t'] = np.array(self._peek_state('o_t_next'))
        new = type(self)(d, members=self.members, sched_params=self._sched_params)
        new.init_states(o_t_next=self._peek_state('o_t_next'), i_t_next=self._peek_state('i_t_next'))
        new.o_t_prev = self._peek_state('o_t_prev')
        new.i_t_prev = self._peek_state('i_t_prev')
        new.alpha, new.beta, new.chi, new.gamma = self.alpha, self.beta, self.chi, self.gamma
        new.saved_states = {k: (np.array(v) if isinstance(v, np.ndarray) else v) for k, v in self.saved_states.items()}
        return new

    @classmethod
    def from_nhd_geojson(cls, file_path, load_paths=True, **kwargs):
        """muskingum.py:877-917 as the reference exposes it (a classmethod around the loader)."""
        return cls(load_nhd_geojson(file_path, load_paths=load_paths), **kwargs)


    def split(self, indices, name=None, create_state_space=False):
        """Cut the network at the reaches `indices` (muskingum.py:607-714): every weakly connected piece of
        the cut forest becomes its own model (named "0", "1", ... in component order), wired by one-way
        `Connection`s.  The downstream model loses the cut reach's contribution to its inflow state, so the
        collection stepped with `AsyncSimulation` reproduces the un-split run.  Returns a `ModelCollection`."""
        from scipy.sparse import coo_matrix, csgraph
        if create_state_space:
            raise NotImplementedError('dense state-space matrices are not built by the GPU drop-in')
        if self.members != 1:
            raise ValueError('split() needs a single-member model')
        n = self.n
        end = self.endnodes.copy()
        cut = np.asarray(indices, dtype=np.int64).reshape(-1)
        if cut.size and (cut.min() < 0 or cut.max() >= n):
            raise ValueError('split index out of range')
        cut_down = end[cut].copy()                       # the reach each cut reach used to drain into
        end[cut] = cut                                   # cut reaches become outlets
        adj = coo_matrix((np.ones(n, dtype=np.int8), (end, np.arange(n))), shape=(n, n))
        n_comp, labels = csgraph.connected_components(adj)
        o_next, i_next = self.o_t_next, self.i_t_next
        o_prev, i_prev = self.o_t_prev, self.i_t_prev
        models, local_index = [], np.empty(n, dtype=np.int64)
        for comp in range(n_comp):
            sel = np.flatnonzero(labels == comp)
            local_index[sel] = np.arange(sel.size)
            d = {'name': str(comp), 'datetime': self.datetime, 'timedelta': self.timedelta,
                 'reach_ids': [self.reach_ids[j] for j in sel],
                 'startnodes': np.arange(sel.size, dtype=np.int64), 'endnodes': local_index[end[sel]].astype(np.int64),
                 'K': self.K[sel].copy(), 'X': self.X[sel].copy(), 'o_t': np.array(o_next[sel], dtype=np.float64),
                 'dx': None if self.dx is None else np.asarray(self.dx)[sel],
                 'paths': [self.paths[j] for j in sel] if len(self.paths) == n else []}
            sub = type(self)(d, sched_params=self._sched_params)
            sub.alpha, sub.beta, sub.chi, sub.gamma = self.alpha[sel], self.beta[sel], self.chi[sel], self.gamma[sel]
            sub.init_states(o_t_next=o_next[sel], i_t_next=i_next[sel])
            sub.o_t_prev = np.array(o_prev[sel]); sub.i_t_prev = np.array(i_prev[sel])
            models.append(sub)
        for u, dwn in zip(cut, cut_down):
            if dwn == u:
                continue                                  # cutting at an outlet separates nothing
            up_model, dn_model = models[labels[u]], models[labels[dwn]]
            ui, di = int(local_index[u]), int(local_index[dwn])
            i_dn = dn_model.i_t_next
            i_dn[di] -= up_model.o_t_next[ui]             # muskingum.py:690
            dn_model.i_t_next = i_dn
            connection = Connection(up_model, dn_model, ui, di)
            up_model.sinks.append(connection)
            dn_model.sources.append(connection)
        for sub in models:
            sub.save_state()
        return ModelCollection(models, name=name)


class Connection:
    """One-way link between two sub-models (muskingum.py:716-726): reach `upstream_index` of
    `upstream_model` drains into reach `downstream_index` of `downstream_model`."""

    def __init__(self, upstream_model, downstream_model, upstream_index, downstream_index, name=None):
        self.upstream_model = upstream_model
        self.downstream_model = downstream_model
        self.upstream_index = upstream_index
        self.downstream_index = downstream_index
        self.name = str(uuid.uuid4()) if name is None else name


class ModelCollection:
    """A forest of sub-models (muskingum.py:728-836)."""

    def __init__(self, models, name=None):
        self.models = {model.name: model for model in models}
        self.name = str(uuid.uuid4()) if name is None else name

    @property
    def info(self):
        return {}

    def _common(self, attr, what):
        values = set(getattr(model, attr) for model in self.models.values())
        if len(values) != 1:
            raise ValueError(f'Models must all have the same {what}')
        return values.pop()

    @property
    def datetime(self):
        return pd.to_datetime(self._common('datetime', 'datetime'))

    @property
    def timedelta(self):
        return pd.to_timedelta(self._common('timedelta', 'timedelta'))

    def load_states(self):
        for model in self.models.values():
            model.load_state()

    def save_states(self):
        for model in self.models.values():
            model.save_state()

    def set_datetime(self, timestamp):
        for model in self.models.values():
            model.datetime = timestamp

    def init_states(self, streamflow):
        for model in self.models.values():
            model.init_states(o_t_next=np.asarray(streamflow[model.reach_ids], dtype=np.float64))

    def connections(self):
        seen = {}
        for model in self.models.values():
            for c in list(model.sinks) + list(model.sources):
                seen.setdefault(c.name, c)
        return seen

    def dump_model_collection(self, file_path, model_file_paths={}, dump_optional=True):
        connections = {name: {'upstream_model': c.upstream_model.name, 'downstream_model': c.downstream_model.name,
                              'upstream_index': int(c.upstream_index), 'downstream_index': int(c.downstream_index)}
                       for name, c in self.connections().items()}
        keys = _REQUIRED + (_OPTIONAL if dump_optional else ())
        models = {name: {'model': {k: model.info[k] for k in keys},
                         'sinks': [c.name for c in model.sinks], 'sources': [c.name for c in model.sources]}
                  for name, model in self.models.items()}
        with open(file_path, 'w') as f:
            json.dump({'models': models, 'connections': connections}, f, cls=_Encoder)

    @classmethod
    def from_file(cls, file_path, load_optional=True, **kwargs):
        return cls(load_model_collection(file_path, load_optional=load_optional), **kwargs)


def _decode_model(obj, load_optional=True):
    for key, dtype in (('startnodes', np.int64), ('endnodes', np.int64), ('K', np.float64),
                       ('X', np.float64), ('o_t', np.float64), ('dx', np.float64)):
        if obj.get(key) is not None:
            obj[key] = np.asarray(obj[key], dtype=dtype)
    if 'datetime' in obj:
        obj['datetime'] = pd.Timestamp(obj['datetime'])
    if 'timedelta' in obj:
        obj['timedelta'] = pd.Timedelta(obj['timedelta'])
    if not load_optional:
        obj.pop('dx', None)
        obj.pop('paths', None)
    return obj


def load_model_collection(file_path, load_optional=True):
    """Collection JSON -> list of wired models (muskingum.py:920-944)."""
    with open(file_path) as f:
        info = json.load(f)
    models = {}
    for _, model_info in info['models'].items():
        model = Muskingum(_decode_model(model_info['model'], load_optional), load_optional=load_optional)
        models[model.name] = model
    for name, c in info['connections'].items():
        connection = Connection(models[c['upstream_model']], models[c['downstream_model']],
                                c['upstream_index'], c['downstream_index'], name=name)
        connection.upstream_model.sinks.append(connection)
        connection.downstream_model.sources.append(connection)
    return list(models.values())


# ---------------------------------------------------------------------- JSON I/O
class _Encoder(json.JSONEncoder):
    def default(self, obj):
        if isinstance(obj, np.ndarray):
            return obj.tolist()
        if isinstance(obj, (pd.Timestamp, pd.Timedelta)):
            return obj.isoformat()
        return json.JSONEncoder.default(self, obj)


def load_model_file(file_path, load_optional=True):
    """Model JSON -> the dict `Muskingum` takes (reference: muskingum.py:839-862, io.py)."""
    with open(file_path) as f:
        obj = json.load(f)
    for key, dtype in (('startnodes', np.int64), ('endnodes', np.int64), ('K', np.float64),
                       ('X', np.float64), ('o_t', np.float64), ('dx', np.float64)):
        if obj.get(key) is not None:
            obj[key] = np.asarray(obj[key], dtype=dtype)
    if 'datetime' in obj:
        obj['datetime'] = pd.Timestamp(obj['datetime'])
    if 'timedelta' in obj:
        obj['timedelta'] = pd.Timedelta(obj['timedelta'])
    if not load_optional:
        obj.pop('dx', None)
        obj.pop('paths', None)
    return obj


def load_nhd_geojson(file_path, load_paths=True):
    """NHD flowline GeoJSON -> the dict `Muskingum` takes (muskingum.py:877-917): reach = feature, COMID /
    toCOMID give the downstream link (a missing toCOMID makes the reach an outlet, i.e. a self-loop), defaults
    K = 3600 s, X = 0.29, o_t = 1e-3.

    The attributes come from ONE native pass over the file (`txh_scan_nhd_geojson`, csrc/txh_geojson.cpp): no
    per-feature Python loop, no Python objects for the geometry, the id -> index join a sort + binary search --
    CONUS-size files do not spend their time here.  `load_paths=True` (the reference's behaviour) additionally
    json-loads the file for the `paths` polylines, which only plotting uses; pass False for large files."""
    import ctypes
    from . import _lib as L
    lib = L.load()
    cnt = ctypes.c_int64()
    path = os.fsencode(file_path)
    L.check(lib.txh_scan_nhd_geojson(path, 0, None, None, None, ctypes.byref(cnt)))
    n = int(cnt.value)
    comid = np.empty(n, dtype=np.int64); endnodes = np.empty(n, dtype=np.int64); dx = np.empty(n, dtype=np.float64)
    L.check(lib.txh_scan_nhd_geojson(path, n, L.ptr_i64(comid), L.ptr_i64(endnodes), L.ptr_f64(dx), ctypes.byref(cnt)))
    paths = []
    if load_paths:
        with open(file_path) as f:
            paths = [np.asarray(ft['geometry']['paths']) for ft in json.load(f)['features']]
    return {
        'name': str(uuid.uuid4()), 'datetime': DEFAULT_START_TIME, 'timedelta': DEFAULT_TIMEDELTA,
        'reach_ids': comid.astype(str).tolist(), 'startnodes': np.arange(n, dtype=np.int64), 'endnodes': endnodes,
        'K': 3600 * np.ones(n, dtype=np.float64), 'X': 0.29 * np.ones(n, dtype=np.float64),
        'o_t': 1e-3 * np.ones(n, dtype=np.float64), 'dx': dx, 'paths': paths,
    }


def dump_model_file(obj, file_path, dump_optional=True):
    keys = _REQUIRED + (_OPTIONAL if dump_optional else ())
    with open(file_path, 'w') as f:
        json.dump({k: obj[k] for k in keys if k in obj}, f, cls=_Encoder)
