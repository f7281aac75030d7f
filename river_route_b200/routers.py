"""
Host side of the routers: the same classes, constructor arguments, config keys, lifecycle, hooks and
errors as river_route.Muskingum / RapidMuskingum / UnitMuskingum, with ``_router`` -- the seam named in
SURVEY.md 8b (river_route/routers/TransformMuskingum.py:150-152, Muskingum.py:262-290) -- marshalling
arrays to librr_b200.so instead of calling the numba loops.  Everything here is plain Python host code
(config, parquet / netCDF I/O, time bookkeeping); no arithmetic of the routing path runs on the CPU.
"""
from __future__ import annotations

import dataclasses
import datetime
import json
import logging
import os
import sys
from typing import Any, Callable, Iterator

import numpy as np
import pandas as pd

from .plan import MODE_MUSKINGUM, MODE_RAPID, MODE_UNIT, STAT_EXCEED, Plan, downstream_index, parse_statistics
from .runoff import runoff_to_qlateral
from .uhkernels import UnitHydrograph

__all__ = ['Configs', 'Muskingum', 'RapidMuskingum', 'UnitMuskingum', 'PROGRESS']

PROGRESS = 25  # custom log level of the reference (river_route/logging.py:3-4)
logging.addLevelName(PROGRESS, 'PROGRESS')

_CHOICES = {
    'grid_accumulation_type': ('incremental', 'cumulative'),
    'runoff_processing_mode': ('sequential', 'ensemble'),
    'log_level': ('DEBUG', 'INFO', 'PROGRESS', 'WARNING', 'ERROR', 'CRITICAL'),
}
_PATHS = ('params_file', 'discharge_dir', 'channel_state_init_file', 'channel_state_final_file', 'grid_weights_file',
          'uh_kernel_file', 'uh_state_init_file', 'uh_state_final_file')
_PATH_LISTS = ('discharge_files', 'qlateral_files', 'grid_runoff_files')
_INPUT_PATHS = ('params_file', 'channel_state_init_file', 'grid_weights_file', 'uh_kernel_file', 'uh_state_init_file')
_INPUT_LISTS = ('qlateral_files', 'grid_runoff_files')
_OUTPUT_FILES = ('channel_state_final_file', 'uh_state_final_file')


@dataclasses.dataclass
class Configs:
    """
    The configuration surface of the reference (river_route/routers/Config.py:31-65, examples/config.yaml):
    same keys, defaults, path normalisation (:112-130), discharge_dir resolution (:146-164), existence checks
    (:132-183) and value checks (:87-93).
    """
    params_file: Any = None
    discharge_dir: Any = None
    discharge_files: Any = dataclasses.field(default_factory=list)
    channel_state_init_file: Any = None
    channel_state_final_file: Any = None
    dt_routing: int = 0
    dt_total: int = 0
    dt_discharge: int = 0
    dt_runoff: int = 0
    start_datetime: str = '1970-01-01'
    qlateral_files: Any = dataclasses.field(default_factory=list)
    grid_runoff_files: Any = dataclasses.field(default_factory=list)
    grid_weights_file: Any = None
    grid_accumulation_type: str = 'incremental'
    runoff_processing_mode: str = 'sequential'
    uh_kernel_file: Any = None
    uh_state_init_file: Any = None
    uh_state_final_file: Any = None
    log: bool = True
    progress_bar: bool = True
    log_level: str = 'PROGRESS'
    log_stream: str = 'stdout'
    log_format: str = '%(levelname)s - %(asctime)s - %(message)s'
    var_river_id: str = 'river_id'
    var_discharge: str = 'Q'
    var_grid_runoff: str = 'ro'
    var_x: str = 'x'
    var_y: str = 'y'
    var_t: str = 'time'

    def __setattr__(self, name, value):
        allowed = _CHOICES.get(name)
        if allowed is not None and value not in allowed:
            raise ValueError(f'{name} must be one of {sorted(allowed)}, got {value!r}')
        object.__setattr__(self, name, value)

    def __post_init__(self):
        self.progress_bar = bool(self.log) and bool(self.progress_bar)
        for key in _PATH_LISTS:                       # a single path means a one-element list
            val = getattr(self, key)
            if isinstance(val, (str, os.PathLike)) and val:
                setattr(self, key, [str(val)])
            elif val is None:
                setattr(self, key, [])
        for key in _PATHS:
            if getattr(self, key):
                setattr(self, key, os.path.abspath(getattr(self, key)))
        for key in _PATH_LISTS:
            setattr(self, key, [os.path.abspath(p) for p in getattr(self, key)])
        # where the discharge goes: a directory (names derived from the inputs) or explicit files
        if self.discharge_dir:
            if self.discharge_files:
                raise ValueError('Provide discharge_dir or discharge_files, not both')
            inputs = self.qlateral_files or self.grid_runoff_files
            names = [f'discharge_{os.path.basename(f)}' for f in inputs] or ['discharge.nc']
            self.discharge_files = [os.path.join(self.discharge_dir, nm) for nm in names]
        elif not self.discharge_files:
            raise ValueError('Provide discharge_dir (or discharge_files for explicit output paths)')
        for key in _INPUT_PATHS:
            val = getattr(self, key)
            if val and not os.path.exists(val):
                raise FileNotFoundError(f'{key} not found: {val}')
        for key in _INPUT_LISTS:
            for path in getattr(self, key):
                if not os.path.exists(path):
                    raise FileNotFoundError(f'{key}: {path} not found')
        outputs = [getattr(self, k) for k in _OUTPUT_FILES if getattr(self, k)] + list(self.discharge_files)
        for path in outputs:
            if not os.path.exists(os.path.dirname(path)):
                raise NotADirectoryError(f'Output directory not found for specified output path: {path}')
        if self.discharge_dir and not os.path.isdir(self.discharge_dir):
            raise NotADirectoryError(f'Output directory not found: {self.discharge_dir}')
        if self.params_file in (None, '', []):
            raise ValueError('Missing required config: params_file')


def _read_config_file(path) -> dict:
    text = str(path)
    if text.endswith('.json'):
        with open(path) as f:
            return json.load(f)
    if text.endswith(('.yml', '.yaml')):
        import yaml
        with open(path) as f:
            return yaml.load(f, Loader=yaml.FullLoader)
    raise RuntimeError('Unrecognized simulation config file type. Must be .json or .yaml')


class Muskingum:
    """
    Muskingum channel routing without lateral inflow (river_route/routers/Muskingum.py).  The solve
    (I - c1 A) Q(t+1) = c2 A Q(t) + c3 Q(t) runs on the GPU (RR_MODE_MUSKINGUM of include/rr_b200.h).
    """
    _ROUTER_REQUIRED_CONFIGS = ('channel_state_init_file', 'dt_routing', 'dt_total')
    _network_time_signature = None

    def __init__(self, configs=None, **kwargs):
        raw = _read_config_file(configs) if configs not in (None, '') and not isinstance(configs, Configs) else {}
        if isinstance(configs, Configs):
            raw = dataclasses.asdict(configs)
            if raw.get('discharge_dir'):
                raw['discharge_files'] = []      # derived from discharge_dir by Configs itself; passing both is an error
        # _shard: a river_route_b200.distributed.Shard -- this process routes only the drainage basins packed to its rank
        # (one process per GPU under torchrun; see distributed.py).  Not a config key.
        self._shard = kwargs.pop('_shard', None)
        raw.update(kwargs)
        raw.pop('_router', None)
        self.cfg = configs if isinstance(configs, Configs) and not kwargs else Configs(**raw)
        self.logger = logging.getLogger(f'river_route_b200.{id(self):x}')
        self.logger.disabled = not self.cfg.log
        self.logger.setLevel(PROGRESS if self.cfg.log_level == 'PROGRESS' else self.cfg.log_level)
        handler = logging.StreamHandler(sys.stdout) if self.cfg.log_stream == 'stdout' \
            else logging.FileHandler(self.cfg.log_stream)
        handler.setFormatter(logging.Formatter(self.cfg.log_format))
        self.logger.addHandler(handler)
        self._writer: Callable | None = None
        self.plan: Plan | None = None

    def __repr__(self):
        return f'{type(self).__name__}(params_file={self.cfg.params_file!r})'

    # ---------------- validation ----------------
    def _validate_configs(self):
        for key in self._ROUTER_REQUIRED_CONFIGS:
            if not getattr(self.cfg, key, None):
                raise ValueError(f'{key} is required for {type(self).__name__}')
        self._validate_router_configs()

    def _validate_router_configs(self):
        if len(self.cfg.discharge_files) != 1:
            raise ValueError('Muskingum requires exactly one entry in discharge_files')

    # ---------------- state ----------------
    def _read_initial_state(self):
        if hasattr(self, 'channel_state'):
            return
        if not self.cfg.channel_state_init_file:
            self.logger.warning('channel_state_init_file not provided. Defaulting to zero initial conditions')
            self.channel_state = np.zeros(self.n, dtype=np.float64)
            return
        self.channel_state = self._mine(pd.read_parquet(self.cfg.channel_state_init_file).values.flatten()
                                        .astype(np.float64, copy=False))

    def _write_final_state(self):
        if self.cfg.channel_state_final_file:
            state = self._gathered(self.channel_state)
            if state is not None:
                pd.DataFrame({'Q': state}).to_parquet(self.cfg.channel_state_final_file)

    # ---------------- basin sharding (river_route_b200.distributed) ----------------
    def _mine(self, full, axis=-1):
        """This rank's river segments of an array over all segments of the params file."""
        return full if self._shard is None else self._shard.take(full, axis=axis)

    def _gathered(self, local):
        """Per-segment vector or (T, segments) array of this rank -> params-file order on rank 0, None elsewhere."""
        if self._shard is None:
            return local
        return self._shard.gather_vector(local) if local.ndim == 1 else self._shard.gather_columns(local)

    # ---------------- network ----------------
    def _set_network_dependent_vectors(self):
        """params parquet -> ids, k, x and the device plan (replaces Muskingum.py:141-169 + tools.adjacency_matrix)."""
        df = pd.read_parquet(self.cfg.params_file, columns=[self.cfg.var_river_id, 'k', 'x', 'downstream_river_id'])
        self.river_ids = df[self.cfg.var_river_id].to_numpy(dtype=np.int64, copy=False)
        self.k = df['k'].to_numpy(dtype=np.float64, copy=False)
        self.x = df['x'].to_numpy(dtype=np.float64, copy=False)
        # duplicate ids, unknown downstream ids and topological order raise the reference's ValueErrors
        down = downstream_index(self.river_ids, df['downstream_river_id'].to_numpy(dtype=np.int64, copy=False))
        self.river_ids_all = self.river_ids            # what the output files list: every segment of the params file
        device = -1
        if self._shard is not None:
            # whole drainage basins only, original relative order kept: confluences sum in the reference's order
            idx, down = self._shard.split(down)
            self.river_ids, self.k, self.x = self.river_ids[idx], np.ascontiguousarray(self.k[idx]), np.ascontiguousarray(self.x[idx])
            device = self._shard.device_index
            if self._output_river_ids is not None:
                raise ValueError('set_output_rivers is not available in basin-sharded runs')
        self.n = int(self.river_ids.shape[0])
        if self.plan is None or not np.array_equal(down, getattr(self, 'down', None)):
            # a new plan has no coefficients yet: forget the cached time signature so that the next file sets them
            # (the reference keeps c1..c3 and its CSC arrays on self, so a second route() just works there)
            self.plan = Plan(down, device=device)
            self._network_time_signature = None
            self._detach_transform()
        self.down = down
        self.logger.log(PROGRESS, f'Network: {self.n} river segments')

    @property
    def A(self):
        """scipy CSC adjacency matrix A[downstream, upstream] = 1, built on demand (river_route/tools.py:75-109)."""
        import scipy.sparse
        has = self.down >= 0
        return scipy.sparse.csc_matrix((np.ones(int(has.sum())), (self.down[has], np.flatnonzero(has))),
                                       shape=(self.n, self.n))

    def _muskingum_coefficients(self, dt_routing):
        """c1, c2, c3 with the reference's exact expressions and check (Muskingum.py:172-185)."""
        dt_div_k = dt_routing / self.k
        denominator = dt_div_k + (2 * (1 - self.x))
        _2x = 2 * self.x
        self.c1 = (dt_div_k - _2x) / denominator
        self.c2 = (dt_div_k + _2x) / denominator
        self.c3 = ((2 * (1 - self.x)) - dt_div_k) / denominator
        if not np.allclose(self.c1 + self.c2 + self.c3, 1):
            self.logger.warning('Muskingum coefficients do not sum to 1')
            raise ValueError('Muskingum coefficients do not sum to 1, check routing parameters and time step')

    def _set_muskingum_coefficients(self, dt_routing):
        self._muskingum_coefficients(dt_routing)
        self.plan.set_coefficients(self.c1, self.c2, self.c3, None)

    # ---------------- lifecycle ----------------
    def route(self):
        self.logger.log(PROGRESS, 'Beginning routing')
        t1 = datetime.datetime.now()
        self._validate_configs()
        self._set_network_dependent_vectors()
        self._apply_output_subset()
        self._read_initial_state()
        self._hook_before_route()
        self._execute_routing()
        self._write_final_state()
        self._hook_after_route()
        self.logger.log(PROGRESS, f'Routing completed in {(datetime.datetime.now() - t1).total_seconds()} seconds')
        return self

    def _execute_routing(self):
        self.dt_routing = self.cfg.dt_routing
        self.dt_total = self.cfg.dt_total
        self.dt_discharge = self.cfg.dt_discharge or self.dt_routing
        if not (self.dt_total >= self.dt_discharge >= self.dt_routing):
            raise ValueError('Need dt_total >= dt_discharge >= dt_routing')
        if self.dt_total % self.dt_discharge != 0:
            raise ValueError('dt_total must be an integer multiple of dt_discharge')
        if self.dt_discharge % self.dt_routing != 0:
            raise ValueError('dt_discharge must be an integer multiple of dt_routing')
        num_output_steps = int(self.dt_total / self.dt_discharge)
        num_routing_per_output = int(self.dt_discharge / self.dt_routing)
        self._set_muskingum_coefficients(self.dt_routing)
        dates = pd.date_range(start=self.cfg.start_datetime, periods=num_output_steps,
                              freq=pd.to_timedelta(self.dt_discharge, unit='s')).to_numpy()
        if _is_stock(self, '_router', Muskingum):
            # the writer receives float32 (Muskingum.py:259): cast on the device, copy back half the bytes
            q32 = np.empty((num_output_steps, self._n_out), dtype=np.float32)
            self._route_channel(q32, num_routing_per_output)
        else:
            q32 = self._host_subset(self._router(num_output_steps, num_routing_per_output)).astype(np.float32, copy=False)
        self._write(dates, q32, self.cfg.discharge_files[0])

    def _route_channel(self, discharge_array, num_routing_per_output):
        if not np.any(self.channel_state):
            self.logger.warning(
                'Initial channel state is all zeros. Muskingum routing without lateral inflow requires a '
                'non-zero initial state to produce meaningful results. Provide channel_state_init_file.')
        q_t = self.channel_state.astype(np.float64, copy=True)
        self.plan.route_host(MODE_MUSKINGUM, q_t, None, discharge_array, num_routing_per_output)
        self.channel_state = q_t
        return discharge_array

    def _router(self, num_output_steps, num_routing_per_output):
        """The seam of Muskingum.py:262-290: returns the fp64 (num_output_steps, n) discharge array."""
        return self._full_width(lambda: self._route_channel(
            np.zeros((num_output_steps, self.n), dtype=np.float64), num_routing_per_output))

    def _full_width(self, call):
        """Run ``call`` with the device output subset switched off: the reference seams return all segments."""
        idx = getattr(self, '_output_idx', None)
        if idx is None:
            return call()
        self.plan.set_output_subset(None)
        try:
            return call()
        finally:
            self.plan.set_output_subset(idx)

    def _host_subset(self, q_array):
        idx = getattr(self, '_output_idx', None)
        return q_array if idx is None else q_array[:, idx]

    def _hook_before_route(self):
        return

    def _hook_after_route(self):
        return

    def _detach_transform(self):
        return

    # ---------------- output ----------------
    _output_river_ids = None

    def set_output_rivers(self, river_ids=None):
        """
        Extension: hand the writer only these river segments (ids of the params file, any order) -- what the
        reference's "save a subset of the routed flows" writer does on the host
        (docs/tutorial/advanced.md:147-170), done on the device so that only those columns cross PCIe.  The writer
        then receives a ``(time, len(river_ids))`` array and the default netCDF writer stores those ids.
        """
        self._output_river_ids = None if river_ids is None else np.asarray(river_ids, dtype=np.int64)
        return self

    def _apply_output_subset(self):
        """Resolve the requested ids against the params file (after the network is known) -> plan subset."""
        if self._output_river_ids is None:
            self.plan.set_output_subset(None)
            self._output_idx = None
            return
        sorter = np.argsort(self.river_ids, kind='stable')
        where = np.searchsorted(self.river_ids, self._output_river_ids, sorter=sorter)
        found = sorter[np.minimum(where, self.n - 1)]
        missing = self._output_river_ids[self.river_ids[found] != self._output_river_ids]
        if missing.size:
            raise ValueError(f'set_output_rivers: ids not in the params file: {np.unique(missing)[:10].tolist()}')
        self._output_idx = found.astype(np.int32)
        self.plan.set_output_subset(self._output_idx)

    @property
    def _n_out(self):
        return self.n if getattr(self, '_output_idx', None) is None else int(self._output_idx.shape[0])

    def set_write_discharges(self, func):
        """Inject a writer ``func(dates, q_array, q_file, routed_file='')`` (Muskingum.py:308-317)."""
        self._writer = func
        return self

    def _write(self, dates, q_array, q_file, routed_file=''):
        q_array = self._gathered(q_array)              # sharded runs: all segments, params-file order, on rank 0
        if q_array is not None:
            (self._writer or self._write_discharges)(dates, q_array, q_file, routed_file)

    def _write_discharges(self, dates, q_array, q_file, routed_file=''):
        """The reference's netCDF layout (Muskingum.py:337-351): time f8, river id i4, Q f4 (time, river_id)."""
        with self._open_discharge_file(dates, q_array.shape[1], q_file, routed_file) as out:
            out.write_rows(0, q_array)

    def _open_discharge_file(self, dates, n_cols, q_file, routed_file='', statistics=None, horizon='steps'):
        """The same file, opened for writing row slabs as they come back from the GPU (streamed runs)."""
        ids = getattr(self, 'river_ids_all', self.river_ids) if getattr(self, '_output_idx', None) is None \
            else self.river_ids[self._output_idx]
        return _DischargeFile(q_file, dates, ids, n_cols, self.cfg.var_river_id, self.cfg.var_discharge, routed_file,
                              statistics, horizon)


class TransformMuskingum(Muskingum):
    """Routers driven by lateral inflow files (river_route/routers/TransformMuskingum.py)."""
    _ROUTER_REQUIRED_CONFIGS = ()
    _as_volumes = False
    _mode = MODE_RAPID
    _ensemble_stats = None

    def set_ensemble_statistics(self, path, statistics=('mean', 'std', 'min', 'max', 'p25', 'p50', 'p75'),
                                thresholds=None, horizon='steps'):
        """
        Extension: in ``runoff_processing_mode='ensemble'`` with ``qlateral_files``, write per-time-step statistics
        across the members to ONE netCDF at ``path`` instead of one discharge file per member.  The statistics are
        computed on the device, so only they cross PCIe.  The file has the discharge files' time / river-id layout
        (after the ``dt_discharge`` resample, honouring ``set_output_rivers``) and one float32 variable
        ``<var_discharge>_<stat>`` per statistic (e.g. ``Q_mean``, ``Q_p25``; percentiles carry a ``percentile``
        attribute).  ``statistics``: ``'mean'``, ``'std'`` (ddof=0), ``'min'``, ``'max'``, ``'p0'`` .. ``'p100'``; each
        equals numpy's over the members' fp64 discharge, cast to float32.  The final channel state is the member mean,
        as without statistics.  ``path=None`` switches back to member files.

        Flood warnings: ``thresholds`` is a table (a parquet path or a DataFrame) with a river-id column
        (``cfg.var_river_id``) and one column of per-river flows per label, e.g. return periods ``rp2`` .. ``rp100``.
        ``'exceed_<label>'`` is then the fraction of members whose discharge is strictly above the river's threshold,
        ``np.mean(x > thr, axis=0)``, written as ``<var_discharge>_exceed_<label>`` (units ``1``, attribute
        ``threshold``).  Rivers missing from the table get NaN thresholds, which are never exceeded (0); table rivers
        outside the network are ignored; duplicate ids, or no id of the network in the table, raise ``ValueError``.

        ``horizon``: ``'steps'`` writes the per-step variables; ``'peaks'`` writes, per statistic, its maximum over the
        whole forecast horizon, ``<var_discharge>_<stat>_peak(river_id)`` (float32 of the fp64 peak), and the time of
        its first occurrence, ``<var_discharge>_<stat>_peak_time(river_id)`` (seconds since the first output time),
        and no per-step variables: no per-step rows are copied back from the device; ``'both'`` writes both.  The peak
        time is the first argmax of the fp64 statistic, so it can differ from the argmax of the float32 per-step
        variable where two fp64 values round to the same float32.
        """
        if horizon not in ('steps', 'peaks', 'both'):
            raise ValueError(f"horizon must be 'steps', 'peaks' or 'both', got {horizon!r}")
        if path is None:
            self._ensemble_stats = None
            return self
        table, labels = None, ()
        if thresholds is not None:
            table = thresholds if isinstance(thresholds, pd.DataFrame) else pd.read_parquet(thresholds)
            if self.cfg.var_river_id not in table.columns:
                raise ValueError(f'thresholds table needs a {self.cfg.var_river_id!r} column')
            labels = tuple(str(c) for c in table.columns if c != self.cfg.var_river_id)
        self._ensemble_stats = (str(path), parse_statistics(statistics, labels), table, horizon)
        return self

    def _threshold_rows(self, table, labels):
        """The thresholds table's columns ``labels`` on the params-file river order: {label: (n,) float64}, NaN for
        rivers the table does not list."""
        rid = self.cfg.var_river_id
        ids = table[rid].to_numpy(dtype=np.int64)
        if np.unique(ids).shape[0] != ids.shape[0]:
            raise ValueError('thresholds table lists a river id more than once')
        pos = pd.Index(ids).get_indexer(self.river_ids)
        hit = pos >= 0
        if not hit.any():
            raise ValueError(f'no river id of the thresholds table is in the network ({rid!r})')
        cols = {str(c): c for c in table.columns if c != rid}
        rows = {}
        for label in labels:
            col = table[cols[label]].to_numpy(dtype=np.float64)
            rows[label] = np.full(self.n, np.nan)
            rows[label][hit] = col[pos[hit]]
        return rows

    def _qlateral_generator(self) -> Iterator[tuple]:
        """Yields (dates, (T, n) fp64 lateral array, input file, output file) per input file (:30-51)."""
        if self.cfg.qlateral_files:
            for lateral_file, discharge_file in zip(self.cfg.qlateral_files, self.cfg.discharge_files):
                dates, array = _read_qlateral(lateral_file)
                yield dates, array, lateral_file, discharge_file
        elif self.cfg.grid_runoff_files and self.cfg.grid_weights_file:
            for runoff_file, discharge_file in zip(self.cfg.grid_runoff_files, self.cfg.discharge_files):
                ds = runoff_to_qlateral(runoff_file, grid_weights_file=self.cfg.grid_weights_file,
                                        var_runoff=self.cfg.var_grid_runoff, var_x=self.cfg.var_x, var_y=self.cfg.var_y,
                                        var_t=self.cfg.var_t, var_river_id=self.cfg.var_river_id,
                                        cumulative=self.cfg.grid_accumulation_type == 'cumulative',
                                        as_volumes=self._as_volumes)
                yield (ds['time'].values.astype('datetime64[s]'), ds['qlateral'].values.astype(np.float64, copy=False),
                       runoff_file, discharge_file)

    def _validate_router_configs(self):
        qlateral = self.cfg.qlateral_files
        grids = self.cfg.grid_runoff_files and self.cfg.grid_weights_file
        if qlateral and grids:
            raise ValueError('Provide qlateral_files or grid_runoff_files with grid_weights_file, not both')
        if not qlateral and not grids:
            raise ValueError('Provide qlateral_files or grid_runoff_files with grid_weights_file')
        if len(self.cfg.discharge_files) != len(qlateral) + len(self.cfg.grid_runoff_files or []):
            raise ValueError('Number of resolved discharge output files must match number of input files')
        if self._ensemble_stats is not None:
            self._validate_ensemble_statistics()

    def _validate_ensemble_statistics(self):
        cfg = self.cfg
        if cfg.runoff_processing_mode != 'ensemble':
            raise ValueError("set_ensemble_statistics needs runoff_processing_mode='ensemble'")
        if self._mode == MODE_UNIT:
            raise ValueError('set_ensemble_statistics is not available for UnitMuskingum')
        if not cfg.qlateral_files:
            raise ValueError('set_ensemble_statistics needs qlateral_files (grid_runoff_files ensembles are not supported)')
        if self._writer is not None:
            raise ValueError('set_ensemble_statistics writes its own file: it cannot be combined with set_write_discharges')
        if self._shard is not None and self._shard.world > 1:
            raise ValueError('set_ensemble_statistics is not available in basin-sharded runs')
        if len(cfg.qlateral_files) > 64:
            raise ValueError(f'set_ensemble_statistics supports at most 64 members, got {len(cfg.qlateral_files)}')

    def _set_network_and_time_dependent_vectors(self, dates):
        """Time bookkeeping of TransformMuskingum.py:66-106; the device coefficients are refreshed only when the
        (dt_total, dt_runoff, dt_discharge, dt_routing) signature changes, as the reference caches them."""
        self.dt_runoff = self.cfg.dt_runoff or int((dates[1] - dates[0]).astype('timedelta64[s]').astype(int))
        self.dt_discharge = self.cfg.dt_discharge or self.dt_runoff
        self.dt_total = self.cfg.dt_total or self.dt_runoff * dates.shape[0]
        if not self.cfg.dt_routing:
            self.logger.warning('dt_routing was not provided or is Null/False, defaulting to dt_runoff')
        self.dt_routing = self.cfg.dt_routing or self.dt_runoff
        signature = (self.dt_total, self.dt_runoff, self.dt_discharge, self.dt_routing)
        if self._network_time_signature == signature:
            return
        for big, small, msg in ((self.dt_total, self.dt_runoff, 'dt_total must be >= dt_runoff'),
                                (self.dt_total, self.dt_discharge, 'dt_total must be >= dt_discharge'),
                                (self.dt_discharge, self.dt_runoff, 'dt_discharge must be >= dt_runoff'),
                                (self.dt_runoff, self.dt_routing, 'dt_runoff must be >= dt_routing')):
            if big < small:
                raise ValueError(msg)
        for big, small, msg in ((self.dt_total, self.dt_runoff, 'dt_total must be an integer multiple of dt_runoff'),
                                (self.dt_total, self.dt_discharge, 'dt_total must be an integer multiple of dt_discharge'),
                                (self.dt_discharge, self.dt_runoff, 'dt_discharge must be an integer multiple of dt_runoff'),
                                (self.dt_runoff, self.dt_routing, 'dt_runoff must be an integer multiple of dt_routing')):
            if big % small != 0:
                raise ValueError(msg)
        self.num_runoff_steps = int(self.dt_total / self.dt_runoff)
        self.num_runoff_steps_per_discharge = int(self.dt_discharge / self.dt_runoff)
        self.num_routing_steps_per_runoff = int(self.dt_runoff / self.dt_routing)
        self._set_muskingum_coefficients(self.dt_routing)
        self._network_time_signature = signature

    def _set_muskingum_coefficients(self, dt_routing):
        self._muskingum_coefficients(dt_routing)
        self.c4 = self.c1 + self.c2                                         # TransformMuskingum.py:104
        self.plan.set_coefficients(self.c1, self.c2, self.c3, self.c4 / self.dt_runoff)   # RapidMuskingum.py:25

    def _execute_routing(self):
        """
        The per-file loop of TransformMuskingum.py:108-148.  With the stock ``_router`` the tail of the loop
        (``dt_discharge`` resample :128-139 and the float32 cast :146) runs on the device, so only float32 output
        rows cross PCIe; with the stock generator and grid inputs the weight table (and unit hydrograph) also run
        there and the lateral inflows never leave the GPU.  A subclass that overrides ``_router`` or
        ``_qlateral_generator`` gets the reference's sequence on fp64 host arrays instead.
        """
        self._ensemble_member_states = []
        if self._ensemble_stats is not None:
            return self._execute_ensemble_statistics()
        device_tail = _is_stock(self, '_router', TransformMuskingum)
        if (device_tail and self.cfg.qlateral_files and _is_stock(self, '_qlateral_generator', TransformMuskingum)
                and _is_stock(self, '_route_lateral', TransformMuskingum, UnitMuskingum)):
            return self._execute_routing_streamed()
        fused_grid = (device_tail and not self.cfg.qlateral_files and self.cfg.grid_runoff_files
                      and self.cfg.grid_weights_file and _is_stock(self, '_qlateral_generator', TransformMuskingum))
        files = self._gathered_runoff_generator() if fused_grid else self._qlateral_generator()
        if self.cfg.progress_bar:
            from tqdm import tqdm
            files = tqdm(files, total=len(self.cfg.qlateral_files or self.cfg.grid_runoff_files), desc='Files Routed')
        for dates, data, runoff_file, discharge_file, *kind in files:
            self.logger.info(f'Routing qlateral: {runoff_file}')
            self._set_network_and_time_dependent_vectors(dates)
            k = self.num_runoff_steps_per_discharge if self.dt_discharge > self.dt_runoff else 1
            if kind != ['runoff']:
                data = self._mine(data, axis=1)         # lateral inflows of this rank's segments
            if device_tail:
                q32 = np.empty((self.num_runoff_steps // k, self._n_out), dtype=np.float32)
                q_t = self._route_runoff(data, q32, k) if kind == ['runoff'] else self._route_lateral(data, q32, k)
            else:
                q_t, q_array = self._router(data)
                if k > 1:                                                    # :128-139
                    q_array = q_array.reshape((int(self.dt_total / self.dt_discharge),
                                               int(self.dt_discharge / self.dt_runoff), self.n)).mean(axis=1)
                q32 = self._host_subset(q_array).astype(np.float32, copy=False)
            if self.cfg.runoff_processing_mode == 'sequential':
                self.channel_state = q_t
            else:                                                            # every member starts from the same state
                self._ensemble_member_states.append(q_t.copy())
            if k > 1:
                dates = dates[::self.num_runoff_steps_per_discharge]
            self._write(dates, q32, discharge_file, runoff_file)
        if self.cfg.runoff_processing_mode == 'ensemble':
            self.channel_state = np.array(self._ensemble_member_states).mean(axis=0)   # :145-146

    # ---------------- qlateral files, streamed: file slab -> pinned buffer -> GPU -> pinned buffer -> file slab --------
    def _execute_routing_streamed(self):
        """
        The per-file loop of TransformMuskingum.py:108-148 for ``qlateral_files`` without ever holding a (T, n) array of
        a file on the host: row slabs are read into page-locked buffers in the dtype they are stored in (a float32
        variable crosses PCIe as float32 and is upcast on the device -- the same bits as ``astype(float64)``, :36),
        routed with the channel state chained on the way, and the float32 rows the writer gets (:146) land in page-locked
        buffers and are written slab by slab.  A reader and a writer thread keep the next and the previous slab moving
        while the GPU works on the current one.  An injected writer (``set_write_discharges``) still receives one whole
        array per file, as its protocol says.
        """
        from concurrent.futures import ThreadPoolExecutor
        pairs = list(zip(self.cfg.qlateral_files, self.cfg.discharge_files))
        if (self.cfg.runoff_processing_mode == 'ensemble' and len(pairs) > 1 and self._mode != MODE_UNIT
                and self._writer is None and (self._shard is None or self._shard.world == 1)
                and _is_stock(self, '_route_rows', TransformMuskingum)):
            return self._execute_ensemble_batched(pairs)
        if self.cfg.progress_bar:
            from tqdm import tqdm
            pairs = tqdm(pairs, total=len(pairs), desc='Files Routed')
        with ThreadPoolExecutor(max_workers=2) as pool:
            for lateral_file, discharge_file in pairs:
                self.logger.info(f'Routing qlateral: {lateral_file}')
                with _LateralFile(lateral_file) as src:
                    dates = src.dates
                    self._set_network_and_time_dependent_vectors(dates)
                    n_all = int(getattr(self, 'river_ids_all', self.river_ids).shape[0])
                    self._check_lateral_shape(src.shape, n_all)
                    q_t = self._route_file_in_slabs(src, dates, lateral_file, discharge_file, pool)
                if self.cfg.runoff_processing_mode == 'sequential':
                    self.channel_state = q_t
                else:                                                        # every member starts from the same state
                    self._ensemble_member_states.append(q_t.copy())
        if self.cfg.runoff_processing_mode == 'ensemble':
            self.channel_state = np.array(self._ensemble_member_states).mean(axis=0)   # :145-146

    def _execute_ensemble_batched(self, pairs):
        """
        ``runoff_processing_mode='ensemble'`` (TransformMuskingum.py:121-126, :145-146) with the members batched: every
        file is one member, all members start from the same channel state, and the members of a time slab are routed by
        ONE device call (``rr_route_ensemble_host``: one wavefront launch per chunk covers all of them).  Members are
        taken in groups that fit the page-locked slab budget; each member's float32 rows go to its own discharge file;
        the final channel state is the mean of the members' final states in member (= file) order.  The reference
        routes the members one after the other (or in separate processes, docs/references/parallelism.md:77-112).
        """
        from concurrent.futures import ThreadPoolExecutor
        n, M = self.n, len(pairs)
        states = np.empty((M, n), dtype=np.float64)
        budget = float(os.environ.get('RR_ROUTER_SLAB_BYTES', 2 << 30))
        q0 = self.channel_state.astype(np.float64, copy=True)
        done, mean = 0, None
        with ThreadPoolExecutor(max_workers=4) as pool:
            while done < M:
                srcs = [_LateralFile(pairs[done][0])]
                try:
                    dates = srcs[0].dates
                    self._set_network_and_time_dependent_vectors(dates)
                    T = self.num_runoff_steps
                    k = self.num_runoff_steps_per_discharge if self.dt_discharge > self.dt_runoff else 1
                    unit = int(np.lcm(16, k))
                    G = int(max(1, min(M - done, 64, budget // max(1, unit * n * srcs[0].dtype.itemsize))))
                    dtype = self._open_members([p[0] for p in pairs[done:done + G]], srcs)
                    slab = self._slab_rows(T, k, G * n * dtype.itemsize)
                    starts = list(range(0, T, slab))
                    lat = [[self._pinned(('elat', b, m), (slab, n), dtype) for m in range(G)] for b in range(2)]
                    out = [[self._pinned(('eout', b, m), (slab // k, n), np.float32) for m in range(G)] for b in range(2)]
                    files = [self._open_discharge_file(srcs[m].dates[::k] if k > 1 else srcs[m].dates, n, pairs[done + m][1],
                                                       pairs[done + m][0]) for m in range(G)]
                    q_members = q0
                    try:
                        def read(s_):
                            t0, t1 = starts[s_], min(T, starts[s_] + slab)
                            list(pool.map(lambda m: srcs[m].read(t0, t1, lat[s_ % 2][m]), range(G)))
                            return t1 - t0

                        def route(s_, rows):
                            nonlocal mean, q_members
                            out_s = [a[:rows // k] for a in out[s_ % 2]]
                            group_states = states[done:done + G]
                            mean = self.plan.route_ensemble_host(self._mode, q_members, [a[:rows] for a in lat[s_ % 2]], out_s,
                                                                 self.num_routing_steps_per_runoff, resample=k, q_final=group_states)
                            q_members = np.ascontiguousarray(group_states)
                            return out_s

                        def write(s_, out_s):
                            for f, o in zip(files, out_s):
                                f.write_rows(starts[s_] // k, o)
                        self._slab_loop(pool, len(starts), read, route, write)
                    finally:
                        for f in files:
                            f.close()
                finally:
                    for src in srcs:
                        src.close()
                done += G
        self._ensemble_member_states = list(states)
        # one group: the device mean (member order, then / M) is the answer; several groups: numpy over all members
        self.channel_state = mean if G == M else np.array(self._ensemble_member_states).mean(axis=0)   # :145-146

    def _execute_ensemble_statistics(self):
        """
        ``set_ensemble_statistics``: every qlateral file is one member, all start from the same channel state, and each
        time slab of ALL members is routed and reduced by one ``Plan.route_ensemble_stats_host`` call (statistics need
        every member of a time step in the same call, so the work is ordered time slab first).  Slab rows come from
        RR_ROUTER_SLAB_BYTES over all members; reads and writes run on the thread pool around the device call.
        """
        from concurrent.futures import ThreadPoolExecutor
        path, parsed, table, horizon = self._ensemble_stats
        cfg = self.cfg
        M = len(cfg.qlateral_files)
        names = [p[0] for p in parsed]
        n, S = self.n, len(parsed)
        steps, want_peaks = horizon != 'peaks', horizon != 'steps'
        used = list(dict.fromkeys(p[0][7:] for p in parsed if p[1] == STAT_EXCEED))   # labels, in order of first use
        mean = None
        if used:
            self.plan.set_thresholds(self._threshold_rows(table, used))
        srcs = [_LateralFile(cfg.qlateral_files[0])]
        try:
            dates = srcs[0].dates
            self._set_network_and_time_dependent_vectors(dates)
            T = self.num_runoff_steps
            k = self.num_runoff_steps_per_discharge if self.dt_discharge > self.dt_runoff else 1
            dtype = self._open_members(cfg.qlateral_files, srcs)
            if os.environ.get('RR_ROUTER_SLAB_ROWS'):
                rows = int(os.environ['RR_ROUTER_SLAB_ROWS'])
            else:
                rows = int(float(os.environ.get('RR_ROUTER_SLAB_BYTES', 2 << 30)) // max(1, M * n * dtype.itemsize))
            unit = int(np.lcm(16, k)) if rows >= np.lcm(16, k) else k      # at least one dt_discharge interval
            slab = min(T, max(unit, rows // unit * unit))
            starts = list(range(0, T, slab))
            lat = [[self._pinned(('elat', b, m), (slab, n), dtype) for m in range(M)] for b in range(2)]
            out = [[self._pinned(('estat', b, s), (slab // k, self._n_out), np.float32) for s in range(S)] for b in range(2)] \
                if steps else None
            if want_peaks:
                # per-call peaks, merged over the slabs on the host with the same strict '>' (the earliest row wins)
                call_peak = (np.empty((S, self._n_out)), np.empty((S, self._n_out), dtype=np.int32))
                peak, peak_row = np.full((S, self._n_out), -np.inf), np.zeros((S, self._n_out), dtype=np.int64)
            states = np.empty((M, n), dtype=np.float64)
            q_members = self.channel_state.astype(np.float64, copy=True)
            out_file = self._open_discharge_file(dates[::k] if k > 1 else dates, self._n_out, path,
                                                 ', '.join(str(f) for f in cfg.qlateral_files), statistics=parsed,
                                                 horizon=horizon)
            with out_file, ThreadPoolExecutor(max_workers=4) as pool:
                def read(s_):
                    t0, t1 = starts[s_], min(T, starts[s_] + slab)
                    list(pool.map(lambda m: srcs[m].read(t0, t1, lat[s_ % 2][m]), range(M)))
                    return t1 - t0

                def route(s_, rows):
                    nonlocal mean, q_members
                    out_s = [a[:rows // k] for a in out[s_ % 2]] if steps else None
                    # later slabs start from the members' own states (q_members is states once the first slab is done)
                    lat_s = [a[:rows] for a in lat[s_ % 2]]
                    if want_peaks:
                        mean = self.plan.route_ensemble_stats_host(self._mode, q_members, lat_s, names, out_s,
                                                                   self.num_routing_steps_per_runoff, resample=k,
                                                                   q_final=states, peaks=call_peak)
                        better = call_peak[0] > peak
                        np.copyto(peak, call_peak[0], where=better)
                        np.copyto(peak_row, call_peak[1] + starts[s_] // k, where=better)
                    else:
                        mean = self.plan.route_ensemble_stats_host(self._mode, q_members, lat_s, names, out_s,
                                                                   self.num_routing_steps_per_runoff, resample=k,
                                                                   q_final=states)
                    q_members = states
                    return out_s

                def write(s_, outs):
                    for i, o in enumerate(outs):
                        out_file.write_rows(starts[s_] // k, o, i)
                self._slab_loop(pool, len(starts), read, route, write if steps else None)
                if want_peaks:
                    out_file.write_peaks(peak, peak_row)
        finally:
            for src in srcs:
                src.close()
        self._ensemble_member_states = list(states)
        self.channel_state = mean                      # member-order mean, then / M (TransformMuskingum.py:145-146)

    @staticmethod
    def _slab_loop(pool, n, read, route, write=None, inline=False):
        """Slabs 0 .. n-1 with read-ahead and write-behind on ``pool``: ``read(s)`` of slab s+1 runs while slab s is
        routed by ``route(s, read(s))`` on the calling thread, and ``write(s, route(s, ...))`` of slab s while slab s+1 is
        routed (``inline``: on the calling thread -- collectives of a sharded run; ``write=None``: nothing to write).
        Slab s uses the buffers of s % 2: it is routed only after the write of slab s-2 has finished."""
        nxt = pool.submit(read, 0)
        pending = [None, None]
        for s in range(n):
            got = nxt.result()
            if s + 1 < n:
                nxt = pool.submit(read, s + 1)
            if pending[s % 2] is not None:
                pending[s % 2].result()                # this output buffer has been written
            routed = route(s, got)
            if write is not None and inline:
                write(s, routed)
            elif write is not None:
                pending[s % 2] = pool.submit(write, s, routed)
        for f in pending:
            if f is not None:
                f.result()

    def _open_members(self, lateral_files, srcs):
        """Open the qlateral files of ensemble members not yet in ``srcs`` (the caller closes them) and check every member
        against the first: shape (num_runoff_steps, n), the same number of time steps and time step.  Returns the
        members' common dtype, float64 when they differ."""
        for lat_file in lateral_files[len(srcs):]:
            srcs.append(_LateralFile(lat_file))
        dates = srcs[0].dates
        for src, lat_file in zip(srcs, lateral_files):
            self.logger.info(f'Routing qlateral: {lat_file}')
            self._check_lateral_shape(src.shape, self.n)
            if src.dates.shape != dates.shape or (len(dates) > 1 and src.dates[1] - src.dates[0] != dates[1] - dates[0]):
                raise ValueError('ensemble members must have the same number of time steps and time step')
        return srcs[0].dtype if all(s_.dtype == srcs[0].dtype for s_ in srcs) else np.dtype(np.float64)

    def _slab_rows(self, T, k, row_bytes):
        """Rows per slab: about RR_ROUTER_SLAB_BYTES (2 GiB) of lateral inflows, whole 16-row groups of the device
        pipeline and whole dt_discharge intervals."""
        if os.environ.get('RR_ROUTER_SLAB_ROWS'):
            rows = int(os.environ['RR_ROUTER_SLAB_ROWS'])
        else:
            rows = int(float(os.environ.get('RR_ROUTER_SLAB_BYTES', 2 << 30)) // max(row_bytes, 1))
        unit = int(np.lcm(16, k))
        rows = max(unit, rows // unit * unit)
        return T if rows >= T else rows

    def _pinned(self, key, shape, dtype):
        """Page-locked scratch array, kept (and grown) across slabs and files: pinning costs ~0.3 s per GB."""
        from ._lib import pinned_empty
        pool = self.__dict__.setdefault('_pinned_pool', {})
        need = int(np.prod(shape)) * np.dtype(dtype).itemsize
        buf = pool.get(key)
        if buf is None or buf.nbytes < need:
            buf = pool[key] = pinned_empty((max(need, 1),), np.uint8)
        return buf[:need].view(dtype).reshape(shape)

    def _route_file_in_slabs(self, src, dates, lateral_file, discharge_file, pool):
        T, n = self.num_runoff_steps, self.n
        k = self.num_runoff_steps_per_discharge if self.dt_discharge > self.dt_runoff else 1
        dates_out = dates[::k] if k > 1 else dates
        slab = self._slab_rows(T, k, src.shape[1] * src.dtype.itemsize)
        starts = list(range(0, T, slab))
        sharded = self._shard is not None and self._shard.world > 1
        lat_bufs = [self._pinned(('lat', b), (slab, n), src.dtype) for b in range(2)]
        out_bufs = [self._pinned(('out', b), (slab // k, self._n_out), np.float32) for b in range(2)]
        wide = np.empty((slab, src.shape[1]), dtype=src.dtype) if sharded else None   # full rows before this rank's columns are taken

        def read(s):
            t0, t1 = starts[s], min(T, starts[s] + slab)
            if sharded:
                src.read(t0, t1, wide)
                np.take(wide[:t1 - t0], self._shard.idx, axis=1, out=lat_bufs[s % 2][:t1 - t0])
                return lat_bufs[s % 2][:t1 - t0]
            return src.read(t0, t1, lat_bufs[s % 2])

        whole = None                                   # an injected writer gets the file's whole array
        out_file = None
        if self._writer is not None:
            whole = np.empty((T // k, self._n_out), dtype=np.float32)
        elif not sharded or self._shard.is_root:
            n_cols = self._n_out if not sharded else int(self.river_ids_all.shape[0])
            out_file = self._open_discharge_file(dates_out, n_cols, discharge_file, lateral_file)

        def write(s, rows):
            r0 = starts[s] // k
            if whole is not None:
                whole[r0:r0 + rows.shape[0]] = rows
                return
            rows = self._gathered(rows)                # sharded: all segments in params-file order on rank 0
            if out_file is not None:
                out_file.write_rows(r0, rows)

        q_t = self.channel_state.astype(np.float64, copy=True)

        def route(s, lat):
            out = out_bufs[s % 2][:lat.shape[0] // k]
            self._route_rows(lat, out, k, q_t, s == 0, s == len(starts) - 1)
            return out
        try:
            # collectives of a sharded run stay on the calling thread (one communicator, ordered calls)
            self._slab_loop(pool, len(starts), read, route, write, inline=sharded)
        finally:
            if out_file is not None:
                out_file.close()
        if whole is not None:
            self._write(dates_out, whole, discharge_file, lateral_file)
        return q_t

    def _route_rows(self, qlateral, out, resample, q_t, first=True, last=True):
        """One slab of a file's lateral inflows -> ``out``; the channel state ``q_t`` is read and updated in place
        (``first`` / ``last``: the slab opens / closes the file)."""
        self.plan.route_host(self._mode, q_t, qlateral, out, self.num_routing_steps_per_runoff, resample=resample)

    def _check_lateral_shape(self, shape, width):
        if tuple(shape) != (self.num_runoff_steps, width):
            raise ValueError(f'qlateral shape {tuple(shape)} does not match (num_runoff_steps, n) = '
                             f'{(self.num_runoff_steps, width)}')

    def _route_lateral(self, qlateral, out, resample=1):
        """Lateral inflows (T, n) on the host -> ``out`` (fp64 or float32, resampled); returns the final state."""
        self._check_lateral_shape(qlateral.shape, self.n)
        q_t = self.channel_state.astype(np.float64, copy=True)
        self.plan.route_host(self._mode, q_t, qlateral, out, self.num_routing_steps_per_runoff, resample=resample)
        return q_t

    def _route_runoff(self, runoff_raw, out, resample=1):
        """Gathered grid runoff (T, n_points) -> ``out`` in one device residency; returns the final state."""
        self._check_lateral_shape(runoff_raw.shape, self._transform.n_points)
        q_t = self.channel_state.astype(np.float64, copy=True)
        self.plan.runoff_route_host(self._transform, self._mode, q_t, runoff_raw, out,
                                    self.num_routing_steps_per_runoff,
                                    cumulative=self.cfg.grid_accumulation_type == 'cumulative',
                                    as_volumes=self._as_volumes, resample=resample)
        return q_t

    _transform = None
    _transform_key = None
    _weight_table = None

    def _ensure_transform(self, factor, flat_shape=None):
        """Weight table netCDF -> device-resident CSR over the params-file river order (runoff.py:255-295), with the
        unit conversion factor folded into the weights before duplicates are summed, as the reference does (:292-293).
        ``flat_shape`` = (ny, nx): column indices become flat cell ids ``y * nx + x`` (entry order unchanged, so the
        sums are too) and the SpMM reads the whole grid -- the pointwise gather of runoff.py:270-279 then happens on
        the device instead of in numpy."""
        from .runoff import build_weight_csr, read_weight_table
        from .transforms import Transform
        key = (factor, flat_shape)
        if self._transform is not None and key == self._transform_key:
            return
        if self._weight_table is None:
            self._weight_table = read_weight_table(self.cfg.grid_weights_file, self.cfg.var_river_id)
        tb = self._weight_table
        indptr, indices, data, cx, cy, rivers, area = build_weight_csr(
            tb['river_id'], tb['x_index'], tb['y_index'], tb['proportion'], tb['area_sqm'], factor)
        # the reference assumes this order (runoff.py:265) and would silently route the wrong catchments otherwise
        if rivers.shape[0] != self.river_ids_all.shape[0] or \
                not np.array_equal(np.asarray(rivers).astype(np.int64), self.river_ids_all):
            raise ValueError('grid_weights_file must list the river segments of params_file in the same order')
        if self._shard is not None:                     # this rank's rows of the weight matrix; every cell column stays
            indptr, indices, data = _csr_rows(indptr, indices, data, self._shard.idx)
            area = self._mine(np.asarray(area))
        n_points = len(cx)
        if flat_shape is not None:
            ny, nx = flat_shape
            if cx.max(initial=0) >= nx or cy.max(initial=0) >= ny:
                raise ValueError('weight table refers to grid cells outside the runoff grid')
            indices = (cy[indices] * nx + cx[indices]).astype(np.int32)
            n_points = ny * nx
        self._detach_transform()
        self._transform = Transform(indptr, indices, data, n_points, area=area)
        self._transform_key = key
        self._cells = (cx, cy)
        self._attach_unit_hydrograph()

    def _count_weight_cells(self):
        """Number of distinct grid cells the weight table touches."""
        from .runoff import read_weight_table
        if self._weight_table is None:
            self._weight_table = read_weight_table(self.cfg.grid_weights_file, self.cfg.var_river_id)
        if not hasattr(self, '_n_weight_cells'):
            tb = self._weight_table
            x, y = np.asarray(tb['x_index']).astype(np.int64), np.asarray(tb['y_index']).astype(np.int64)
            self._n_weight_cells = len(pd.unique(x * (int(y.max(initial=0)) + 1) + y))
        return self._n_weight_cells

    def _attach_unit_hydrograph(self):
        return

    def _detach_transform(self):
        if self._transform is not None:
            self._transform.close()
            self._transform = None

    def _gathered_runoff_generator(self) -> Iterator[tuple]:
        """Yields (dates, gathered runoff (T, n_points) in the file's dtype, input file, output file) per grid file:
        the pointwise ``isel`` of runoff.py:267-280; everything after it happens on the device."""
        from .runoff import _conversion_factor, gather_grid_runoff, grid_layout, grid_runoff_unit
        names = dict(var_runoff=self.cfg.var_grid_runoff, var_x=self.cfg.var_x, var_y=self.cfg.var_y, var_t=self.cfg.var_t)
        for runoff_file, discharge_file in zip(self.cfg.grid_runoff_files, self.cfg.discharge_files):
            factor = _conversion_factor(grid_runoff_unit(runoff_file, self.cfg.var_grid_runoff))
            # catchments covering a good part of a (time, y, x) grid: ship the grid as it is and let the SpMM index
            # it (numpy's pointwise gather of a million cells per time step costs more than routing them)
            dims, ny, nx = grid_layout(runoff_file, **names)
            flat = dims == (self.cfg.var_t, self.cfg.var_y, self.cfg.var_x) and 4 * self._count_weight_cells() >= ny * nx
            self._ensure_transform(factor, (ny, nx) if flat else None)
            cx, cy = self._cells
            dates, raw = gather_grid_runoff(runoff_file, cx, cy, flat=flat, **names)
            if len(dates) > 2 and not np.all(np.diff(dates) == dates[1] - dates[0]):
                # irregular time axis: the reference resamples the lateral inflows on the host (runoff.py:316-329)
                ds = runoff_to_qlateral(runoff_file, grid_weights_file=self.cfg.grid_weights_file,
                                        var_runoff=self.cfg.var_grid_runoff, var_x=self.cfg.var_x, var_y=self.cfg.var_y,
                                        var_t=self.cfg.var_t, var_river_id=self.cfg.var_river_id,
                                        cumulative=self.cfg.grid_accumulation_type == 'cumulative',
                                        as_volumes=self._as_volumes)
                yield (ds['time'].values.astype('datetime64[s]'), ds['qlateral'].values.astype(np.float64, copy=False),
                       runoff_file, discharge_file, 'lateral')
                continue
            yield dates, raw, runoff_file, discharge_file, 'runoff'

    def _router(self, qlateral):
        """The seam of TransformMuskingum.py:150-152: (final state, fp64 (T, n) discharge array)."""
        discharge_array = np.zeros((self.num_runoff_steps, self.n), dtype=np.float64)
        q_t = self._full_width(lambda: self._route_lateral(qlateral, discharge_array))
        return q_t, discharge_array


def _csr_rows(indptr, indices, data, rows):
    """Rows ``rows`` (ascending) of a CSR matrix, entry order within a row unchanged."""
    counts = np.diff(indptr)[rows]
    new_ptr = np.zeros(rows.shape[0] + 1, dtype=np.int32)
    np.cumsum(counts, out=new_ptr[1:])
    pos = np.arange(int(new_ptr[-1]), dtype=np.int64) - np.repeat(new_ptr[:-1].astype(np.int64), counts) \
        + np.repeat(indptr[rows].astype(np.int64), counts)
    return new_ptr, np.ascontiguousarray(indices[pos]), np.ascontiguousarray(data[pos])


def _is_stock(obj, name, *owners) -> bool:
    """True when ``obj.<name>`` is still the implementation of one of ``owners`` (not overridden by a subclass or
    patched on the instance): only then may the host-visible fp64 intermediate be skipped."""
    if name in vars(obj):
        return False
    impl = getattr(type(obj), name, None)
    return any(impl is vars(o).get(name) for o in owners)


class RapidMuskingum(TransformMuskingum):
    """Muskingum routing with direct lateral inflow volumes (river_route/routers/RapidMuskingum.py)."""
    _as_volumes = True
    _mode = MODE_RAPID


class UnitMuskingum(TransformMuskingum):
    """Muskingum routing with unit-hydrograph lateral inflow (river_route/routers/UnitMuskingum.py): runoff depths
    are convolved with the UH kernel on the GPU, headwaters pass the convolved inflow through, inner reaches are
    routed; the headwater / inner split lives inside the device plan."""
    _ROUTER_REQUIRED_CONFIGS = ('uh_kernel_file',)
    _as_volumes = False
    _mode = MODE_UNIT
    _uh: UnitHydrograph | None = None

    def _hook_before_route(self):
        if self._uh is None:
            self._uh = UnitHydrograph(self.cfg.uh_kernel_file)
            if self.cfg.uh_state_init_file:
                self._uh.set_state(self.cfg.uh_state_init_file)
            if self._shard is not None:                 # this rank's basins of the (n_kernel_steps, n_basins) arrays
                self._uh.kernel = self._mine(self._uh.kernel, axis=1)
                self._uh.state = self._mine(self._uh.state, axis=1)
        if not hasattr(self, 'hw_idx'):
            incoming = np.bincount(self.down[self.down >= 0], minlength=self.n)
            self.hw_idx = np.where(incoming == 0)[0]
            self.inner_idx = np.where(incoming != 0)[0]
            self.logger.info(f'Headwater split: {len(self.hw_idx)} headwater, {len(self.inner_idx)} inner '
                             f'({len(self.hw_idx) / self.n * 100:.0f}% excluded from solve)')

    def _set_muskingum_coefficients(self, dt_routing):
        self._muskingum_coefficients(dt_routing)
        self.c4 = self.c1 + self.c2
        self.plan.set_coefficients(self.c1, self.c2, self.c3, None)

    def _route_lateral(self, qlateral, out, resample=1):
        self._check_lateral_shape(qlateral.shape, self.n)
        self._sync_uh_state()                       # a device-resident carry-over (grid files routed earlier) comes home
        convolved = self._uh.convolve(qlateral)     # UnitMuskingum.py:75
        if self._transform is not None and self._transform.n_ks:
            self._attach_unit_hydrograph()
        return super()._route_lateral(convolved, out, resample)

    def _route_rows(self, qlateral, out, resample, q_t, first=True, last=True):
        self._sync_uh_state()
        convolved = self._uh.convolve(qlateral)     # UnitMuskingum.py:75; the carry-over state chains the slabs
        if self._transform is not None and self._transform.n_ks:
            self._attach_unit_hydrograph()
        # Inside a file q_ch and q_full are two vectors (q_full = q_ch + lateral, _numba_kernels.py:165); they become
        # one only where the reference recombines them, at the end of a file (UnitMuskingum.py:94-98).  Slabs of one file
        # therefore chain the kernel-level pair (q_t is q_ch), and only the last slab recombines.
        if first:
            self._q_full = q_t.copy()               # :78-79  q_ch = q_full = channel_state
        self.plan.route_host(self._mode, q_t, convolved, out, self.num_routing_steps_per_runoff, q_full=self._q_full,
                             resample=resample)
        if last:
            q_t[self.inner_idx] = self._q_full[self.inner_idx]
            q_t[self.hw_idx] = convolved[-1][self.hw_idx]

    def _attach_unit_hydrograph(self):
        # the carry-over state moves to the device and stays there between files (UnitHydrograph.py:100-105)
        self._transform.set_unit_hydrograph(self._uh.kernel, self._uh.state)

    def _detach_transform(self):
        self._sync_uh_state()
        super()._detach_transform()

    def _sync_uh_state(self):
        if self._transform is not None and self._transform.n_ks and self._uh is not None:
            self._uh.state = self._transform.uh_state()

    def _write_final_state(self):
        self._sync_uh_state()
        super()._write_final_state()
        if self.cfg.uh_state_final_file and self._uh is not None:
            state = self._gathered(self._uh.state)
            if state is not None:
                pd.DataFrame(state.T).to_parquet(self.cfg.uh_state_final_file)   # UnitHydrograph.write_state layout


class _DischargeFile:
    """Discharge netCDF with the reference's layout (Muskingum.py:337-351), written in row slabs."""

    def __init__(self, path, dates, river_ids, n_cols, var_river_id, var_discharge, routed_file='', statistics=None,
                 horizon='steps'):
        """``statistics`` (``[(name, kind, q)]`` of ``plan.parse_statistics``): one variable ``<var_discharge>_<name>``
        per ensemble statistic instead of the one discharge variable.  ``horizon`` ('steps' / 'peaks' / 'both', see
        ``set_ensemble_statistics``): per-step variables, horizon-peak variables (``write_peaks``) or both."""
        from . import ncio
        self.ds = ncio.open_nc(path, 'w')
        ds = self.ds
        ds.createDimension('time', len(dates))
        ds.createDimension(var_river_id, n_cols)
        ds.runoff_file = str(routed_file)
        tv = ds.createVariable('time', 'f8', ('time',))
        tv.units = f'seconds since {pd.Timestamp(dates[0]).strftime("%Y-%m-%d %H:%M:%S")}'
        tv[:] = (dates - dates[0]).astype('timedelta64[s]').astype(np.int64)
        iv = ds.createVariable(var_river_id, 'i4', (var_river_id,))
        iv[:] = np.asarray(river_ids).astype(np.int32)
        self.vars, self.peak_vars = [], []
        self.dates = dates
        for name, kind, q in statistics or [(None, None, None)]:
            if horizon != 'peaks':
                qv = ds.createVariable(var_discharge if name is None else f'{var_discharge}_{name}', 'f4', ('time', var_river_id))
                self._describe(qv, name, kind, q)
                self.vars.append(qv)
            if horizon != 'steps':
                pv = ds.createVariable(f'{var_discharge}_{name}_peak', 'f4', (var_river_id,))
                self._describe(pv, name, kind, q)
                pv.long_name = f'Peak over the forecast horizon of the {pv.long_name[0].lower()}{pv.long_name[1:]}'
                tv_ = ds.createVariable(f'{var_discharge}_{name}_peak_time', 'f8', (var_river_id,))
                tv_.long_name = f'Time of the first occurrence of the peak of {var_discharge}_{name}'
                tv_.units = tv.units
                self.peak_vars.append((pv, tv_))
        self.qv = self.vars[0] if self.vars else None

    @staticmethod
    def _describe(v, name, kind, q):
        if kind == STAT_EXCEED:
            v.long_name = f'Fraction of ensemble members above the {name[7:]} threshold'
            v.units = '1'
            v.threshold = name[7:]
            return
        v.long_name = 'Discharge at catchment outlet' if name is None else f'Ensemble {name} of the discharge at catchment outlet'
        v.standard_name = 'discharge'
        v.aggregation_method = 'mean'
        v.units = 'm3 s-1'
        if kind == 4:
            v.percentile = q

    def write_rows(self, t0, rows, var=0):
        self.vars[var][t0:t0 + rows.shape[0], :] = rows

    def write_peaks(self, values, rows):
        """values (S, n_cols) fp64 and rows (S, n_cols) output-row indices: the peak variables of every statistic."""
        seconds = (self.dates - self.dates[0]).astype('timedelta64[s]').astype(np.float64)
        for (pv, tv_), v, r in zip(self.peak_vars, values, rows):
            pv[:] = v.astype(np.float32)
            tv_[:] = seconds[r]

    def close(self):
        if self.ds is not None:
            self.ds.close()
            self.ds = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class _LateralFile:
    """qlateral netCDF -- variable ``qlateral(time, river_id)``, docs/references/io-file-schema.md:52-55 -- opened for
    reading row slabs straight into (pinned) buffers, in the dtype it is stored in when that is float32 / float64."""

    def __init__(self, path):
        from . import ncio
        self.ds = ncio.open_nc(path, mmap=True)
        tv = self.ds.variables['time']
        self.dates = ncio.decode_time(ncio.read_array(tv), ncio.attrs_of(tv).get('units', ''))
        self.var = self.ds.variables['qlateral']
        self.time_major = tuple(self.var.dimensions)[0] == 'time'
        shape = tuple(int(x) for x in self.var.shape)
        self.shape = shape if self.time_major else shape[::-1]
        kind = np.dtype(self.var.dtype if hasattr(self.var, 'dtype') else self.var.data.dtype)
        self.dtype = np.dtype(np.float32) if (kind.kind == 'f' and kind.itemsize == 4) else np.dtype(np.float64)
        self._whole = None

    def read(self, t0, t1, out):
        """rows [t0, t1) -> out[:t1 - t0] (masked entries become NaN like the reference's xarray read)."""
        raw = getattr(self.var, 'data', None)
        if self.time_major and isinstance(raw, np.ndarray) and \
                not any(k in getattr(self.var, '_attributes', {}) for k in ('missing_value', '_FillValue', 'scale_factor', 'add_offset')):
            # classic file through scipy, plain values: one byte-swapping copy straight from the memory map
            np.copyto(out[:t1 - t0], raw[t0:t1], casting='unsafe')
            return out[:t1 - t0]
        if self.time_major:
            a = self.var[t0:t1]
        else:
            if self._whole is None:
                self._whole = np.asarray(self.var[:]).T
            a = self._whole[t0:t1]
        if isinstance(a, np.ma.MaskedArray):
            a = a.filled(np.nan)
        out[:t1 - t0] = a
        return out[:t1 - t0]

    def close(self):
        self._whole = self.var = None
        if self.ds is not None:
            try:
                self.ds.close()
            except Exception:
                pass
            self.ds = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def _read_qlateral(path):
    """qlateral netCDF: variable ``qlateral(time, river_id)`` (docs/references/io-file-schema.md:52-55)."""
    from . import ncio
    with ncio.open_nc(path) as ds:
        tv = ds.variables['time']
        dates = ncio.decode_time(ncio.read_array(tv), ncio.attrs_of(tv).get('units', ''))
        var = ds.variables['qlateral']
        array = ncio.read_array(var)
        if tuple(var.dimensions)[0] != 'time':
            array = array.T
    return dates, array.astype(np.float64, copy=False)
