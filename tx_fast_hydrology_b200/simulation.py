"""Orchestration of a forest of sub-models and the `CheckPoint` callback
(tx_fast_hydrology/simulation.py).

`AsyncSimulation` (simulation.py:94-166) runs the sub-models of a `ModelCollection` in dependency order:
a sub-model starts once every sub-model draining into it has finished its whole run, and the hydrograph of
the upstream exit reach enters the downstream entry reach as extra lateral inflow,
(alpha*i_next + beta*i_prev)/gamma -- which reproduces the un-split update exactly.  A sub-model without
callbacks runs its whole span in device-resident launches with the trajectory recorded on the GPU
(`Muskingum.run`); one with callbacks (a Kalman filter per sub-basin, as app.py:130-141 binds them) steps
through `simulate_iter` so that every hook fires as in the reference.

`CheckPoint` (simulation.py:169-211) saves the model state once when `model.datetime >= checkpoint_time`
and fans save/load out to sibling callbacks."""
import asyncio
import datetime
import logging

import numpy as np
import pandas as pd

from .callbacks import BaseCallback

logger = logging.getLogger(__name__)


class Simulation:
    def __init__(self, model_collection, inputs):
        self.model_collection = model_collection
        self.models = model_collection.models
        self.inputs = self.load_inputs(inputs)
        self.outputs = {}

    def load_inputs(self, inputs):
        return {name: inputs[model.reach_ids].copy() for name, model in self.models.items()}

    def simulate(self):
        raise NotImplementedError

    @property
    def datetime(self):
        return self.model_collection.datetime

    def load_states(self):
        self.model_collection.load_states()

    def save_states(self):
        self.model_collection.save_states()

    def init_states(self, streamflow):
        self.model_collection.init_states(streamflow)

    def set_datetime(self, timestamp):
        self.model_collection.set_datetime(timestamp)


class AsyncSimulation(Simulation):
    async def simulate(self):
        """Awaitable like the reference's (simulation.py:98-108); `run()` is the plain-call form."""
        return self.run()

    batch_filters = True      # sub-models that are ready together and carry only a KalmanFilter run as one batch

    def run(self):
        pending = {name: len(model.sources) for name, model in self.models.items()}
        ready = [name for name, k in pending.items() if k == 0]
        done = 0

        def finished(name, outputs):
            nonlocal done
            model = self.models[name]
            self.outputs[name] = outputs
            done += 1
            for connection in model.sinks:
                down = connection.downstream_model
                if down.name == name:
                    continue
                self._accumulate(outputs, model, connection)
                pending[down.name] -= 1
                if pending[down.name] == 0:
                    ready.append(down.name)

        while ready:
            batch = self._batchable(ready) if self.batch_filters else []
            if len(batch) >= 2:
                for name in batch:
                    ready.remove(name)
                for name, outputs in self._simulate_batch(batch).items():
                    finished(name, outputs)
                continue
            name = ready.pop(0)
            finished(name, self._simulate(self.models[name], self.inputs[name]))
        if done != len(self.models):
            raise ValueError('sub-model connections contain a cycle')
        return self.outputs

    def _batchable(self, names):
        """The ready sub-models whose filters can run as ONE chain of launches (da.BatchedKalmanFilters): a single
        plain KalmanFilter callback with no more gauges than a batched block takes, one member, a whole-second step,
        the same clock and forcing index."""
        from . import _lib
        from .da import KalmanFilter
        max_gauges = _lib.load().txh_kfb_max_gauges()
        out = []
        for name in names:
            m = self.models[name]
            cbs = list(m.callbacks.values())
            if len(cbs) != 1 or type(cbs[0]) is not KalmanFilter or m.members != 1:
                continue
            if cbs[0].num_measurements > max_gauges:
                continue
            if m.timedelta.value != int(round(m.dt * 1e9)):
                continue
            if out:
                first = self.models[out[0]]
                if (m.datetime != first.datetime or m.timedelta != first.timedelta or
                        not self.inputs[name].index.equals(self.inputs[out[0]].index)):
                    continue
            out.append(name)
        return out

    def _simulate_batch(self, names):
        """One generation of independent sub-models with a Kalman filter each, stepped in lockstep on their union."""
        from .da import BatchedKalmanFilters
        models = [self.models[name] for name in names]
        bkf = BatchedKalmanFilters(models)
        try:
            res = bkf.run({name: self.inputs[name] for name in names})
        finally:
            bkf.close()
        outputs = {}
        for name in names:
            values, times = res[name]
            outputs[name] = pd.DataFrame(values, index=pd.to_datetime(times, utc=True), columns=self.inputs[name].columns)
        return outputs

    def _simulate(self, model, inputs):
        """Whole run of one sub-model; rows = start time + every step, columns = reach ids."""
        logger.debug(f'Started job for sub-watershed {model.name}')
        start, dt = model.datetime, model.timedelta
        first = model._peek_state('o_t_next')
        end_time = inputs.index.max()
        nsteps = 0 if not end_time > start else int(-((start - end_time) // dt))      # steps while datetime < end
        whole = dt.value == int(round(model.dt * 1e9))
        if model.callbacks or nsteps == 0 or not whole:
            rows, times = [first], [start]
            model._capture_start = True
            try:
                for state in model.simulate_iter(inputs):
                    rows.append(state._peek_state('o_t_next')); times.append(state.datetime)
            finally:
                model._capture_start = False
            # row 0 aliases o_t_next in the reference, so it shows what the simulation-start hooks (a Kalman filter's
            # first update) did to the state (simulation.py:126-127)
            rows[0] = getattr(model, '_start_outflow', first)
            values = np.stack(rows)
        else:
            assert isinstance(inputs.index, pd.DatetimeIndex) and str(inputs.index.tz) == 'UTC'
            forcing = model.make_forcing(dataframe=inputs)
            rec = model.run(forcing, nsteps, record_reaches=np.arange(model.n), record_every=1)
            model.network.check()
            values = np.concatenate([first[None, :], rec.cpu().numpy()[:, :, 0]], axis=0)
            times = [start + k * dt for k in range(nsteps + 1)]
            forcing.close()
        outputs = pd.DataFrame(values, index=pd.to_datetime(times, utc=True), columns=inputs.columns)
        return outputs

    def _accumulate(self, outputs, upstream_model, connection):
        """simulation.py:137-166: the exit hydrograph becomes lateral inflow of the entry reach."""
        down = connection.downstream_model
        inputs = self.inputs[down.name]
        o = outputs[upstream_model.reach_ids[connection.upstream_index]].values
        i_t_prev, i_t_next = o[:-1], o[1:]
        k = connection.downstream_index
        inputs.loc[:, down.reach_ids[k]] += (down.alpha[k] * i_t_next / down.gamma[k]
                                             + down.beta[k] * i_t_prev / down.gamma[k])


class CheckPoint(BaseCallback):
    def __init__(self, model, checkpoint_time=None, timedelta=None):
        self.model = model
        if checkpoint_time is None:
            if timedelta is None:
                raise ValueError('Either `checkpoint_time` or `timedelta` must not be `None`.')
            checkpoint_time = model.datetime + datetime.timedelta(seconds=timedelta)
        self.checkpoint_time = checkpoint_time
        self.timedelta = timedelta
        self.model_saved = False

    def __on_simulation_start__(self):
        if self.timedelta is None:
            return None
        self.set_checkpoint(self.model.datetime + datetime.timedelta(seconds=self.timedelta))

    def __on_step_end__(self):
        if (self.model.datetime >= self.checkpoint_time) and (not self.model_saved):
            self.model.save_state()
            self.model_saved = True

    def __on_save_state__(self):
        for _, callback in self.model.callbacks.items():
            if hasattr(callback, 'save_state'):
                callback.save_state()

    def __on_load_state__(self):
        for _, callback in self.model.callbacks.items():
            if hasattr(callback, 'load_state'):
                callback.load_state()

    def set_checkpoint(self, checkpoint_time):
        logger.info(f'Setting checkpoint time to {checkpoint_time}')
        self.checkpoint_time = checkpoint_time
        self.model_saved = False
