"""
Host-side handle of the wavefront plan (``rr_plan`` in include/rr_b200.h) and the topology helpers.

The plan plays the role of the reference's cached sparse arrays
(``Muskingum._set_network_dependent_vectors`` / ``_set_muskingum_coefficients``,
river_route/routers/Muskingum.py:141-193): it is built once per network and reused for every file.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import lib, check

MODE_MUSKINGUM, MODE_RAPID, MODE_UNIT = 0, 1, 2
_STAT_KINDS = {'mean': 0, 'std': 1, 'min': 2, 'max': 3}   # RR_STAT_*; 'pQ' is RR_STAT_PERCENTILE (4) with q = Q
STAT_EXCEED = 5   # RR_STAT_EXCEED: 'exceed_<label>', q = the label's threshold row


def downstream_index(river_ids, downstream_ids) -> np.ndarray:
    """
    int32 index of each reach's downstream reach (-1 for outlets) with the reference's checks and
    error messages: duplicate ids (routers/Muskingum.py:153-154), downstream ids that are not river
    ids (Muskingum.py:161-166, river_route/tools.py:101-102) and topological order (tools.py:103-104).
    """
    river_ids = np.ascontiguousarray(river_ids, dtype=np.int64)
    downstream_ids = np.ascontiguousarray(downstream_ids, dtype=np.int64)
    if river_ids.ndim != 1 or river_ids.shape != downstream_ids.shape:
        raise ValueError('river_ids and downstream_ids must be 1D arrays of the same length')
    down = np.empty(river_ids.shape[0], dtype=np.int32)
    bad = C.c_int64(0)
    rc = lib.rr_downstream_index(river_ids.shape[0], _lib.as_i64p(river_ids), _lib.as_i64p(downstream_ids),
                                 _lib.as_i32p(down), C.byref(bad))
    if rc == 2 and bad.value > 0:
        # Muskingum.py:161-166 runs before adjacency_matrix and lists every positive unknown id
        unknown = np.setdiff1d(downstream_ids[downstream_ids > 0], river_ids)
        raise ValueError(f'params_file has downstream IDs not in river_id column: {unknown[:10].tolist()}')
    check(rc)
    return down


def label_basins(down: np.ndarray, n_parts: int = 0):
    """
    Drainage-basin label of every reach (basins numbered by ascending outlet index) and, when
    ``n_parts`` > 0, the LPT bin-packing of basins over that many GPUs by reach count.
    Returns (basin, n_basins, part-or-None).
    """
    down = np.ascontiguousarray(down, dtype=np.int32)
    basin = np.empty(down.shape[0], dtype=np.int32)
    nb = C.c_int64(0)
    part = np.empty(down.shape[0], dtype=np.int32) if n_parts > 0 else None
    check(lib.rr_label_basins(down.shape[0], _lib.as_i32p(down), _lib.as_i32p(basin), C.byref(nb), int(n_parts),
                              _lib.as_i32p(part) if part is not None else None))
    return basin, int(nb.value), part


def parse_statistics(names, thresholds=()) -> list:
    """
    Ensemble statistic names -> ``[(name, kind, q)]``: ``'mean'``, ``'std'`` (population, ddof=0), ``'min'``, ``'max'``
    and percentiles ``'p0'`` .. ``'p100'`` (integer q, numpy's default 'linear' method).  With threshold labels
    (``thresholds``, in threshold-row order, e.g. ``('rp2', 'rp10')``), ``'exceed_<label>'`` is the fraction of members
    strictly above that threshold, ``np.mean(x > thr, axis=0)``, and resolves to ``(name, 5, row of the label)``.  At
    most 16, no duplicates; anything else raises ``ValueError``.
    """
    labels = list(thresholds)
    if len(set(labels)) != len(labels):
        raise ValueError(f'duplicate threshold labels in {labels}')
    if isinstance(names, str):
        names = [names]
    names = list(names)
    if not 1 <= len(names) <= _lib.MAX_STATS:
        raise ValueError(f'between 1 and {_lib.MAX_STATS} ensemble statistics, got {len(names)}')
    out = []
    for name in names:
        if not isinstance(name, str):
            raise ValueError(f'ensemble statistic names are strings, got {name!r}')
        if name in _STAT_KINDS:
            out.append((name, _STAT_KINDS[name], 0))
        elif name[:1] == 'p' and name[1:].isdigit() and str(int(name[1:])) == name[1:] and int(name[1:]) <= 100:
            out.append((name, 4, int(name[1:])))
        elif name.startswith('exceed_') and name[7:] in labels:
            out.append((name, STAT_EXCEED, labels.index(name[7:])))
        else:
            hint = f", or 'exceed_<label>' with a label of {labels}" if labels else ''
            raise ValueError(f"unknown ensemble statistic {name!r}: use 'mean', 'std', 'min', 'max' or 'p0' .. 'p100'{hint}")
    if len({o[0] for o in out}) != len(out):
        raise ValueError(f'duplicate ensemble statistics in {names}')
    return out


def _stats_spec(names, thresholds=()):
    spec = _lib.StatsSpec()
    parsed = parse_statistics(names, thresholds)
    spec.n_stats = len(parsed)
    for s, (_, kind, q) in enumerate(parsed):
        spec.kind[s], spec.q[s] = kind, q
    return spec


def ensemble_stats_dev(stats, n_members: int, x_ptr: int, member_stride: int, ld: int, rows: int, n_out: int,
                       out_ptrs, ldo: int, out_f32: bool, subset_ptr: int = 0, stream: int = 0, *, thresholds=(),
                       thr_ptr: int = 0, ldt: int = 0, peak_ptrs=None, ldk: int = 0, row0: int = 0) -> None:
    """The statistics kernel alone on device pointers (``rr_ensemble_stats_dev``): member m, row t, reach i is
    ``x[m * member_stride + t * ld + i]``; ``out_ptrs[s]`` is (rows, ldo) float32 / float64 of statistic ``stats[s]``;
    column c shows reach ``subset[c]`` (int32 device array) or reach c.  Asynchronous on ``stream``.

    Keyword-only (``rr_ensemble_stats_dev_ex``): ``'exceed_<label>'`` names resolve against ``thresholds`` (labels in
    row order) and read the fp64 device array ``thr_ptr`` [rows][ldt] at reach ``subset[c]``; ``peak_ptrs = (peak,
    peak_row)`` are device (S, ldk) float64 / int32 running peaks, updated where a row's value is strictly greater, with
    rows numbered from ``row0`` (start peak at -inf).  ``out_ptrs`` may be ``None`` when ``peak_ptrs`` is given."""
    spec = _stats_spec(stats, thresholds)
    if out_ptrs is not None and len(out_ptrs) != spec.n_stats:
        raise ValueError('one output array per statistic')
    arr = C.c_void_p * spec.n_stats
    outs = arr(*out_ptrs) if out_ptrs is not None else None
    if not (thr_ptr or peak_ptrs is not None or out_ptrs is None):
        check(lib.rr_ensemble_stats_dev(C.byref(spec), int(n_members), C.c_void_p(x_ptr), int(member_stride), int(ld),
                                        int(rows), int(n_out), C.c_void_p(subset_ptr or None), outs, int(ldo),
                                        int(bool(out_f32)), C.c_void_p(stream or None)))
        return
    peak, peak_row = peak_ptrs if peak_ptrs is not None else (0, 0)
    check(lib.rr_ensemble_stats_dev_ex(C.byref(spec), int(n_members), C.c_void_p(x_ptr), int(member_stride), int(ld),
                                       int(rows), int(n_out), C.c_void_p(subset_ptr or None), C.c_void_p(thr_ptr or None),
                                       int(ldt), outs, int(ldo), int(bool(out_f32)), C.c_void_p(peak or None),
                                       C.c_void_p(peak_row or None), int(ldk), int(row0), C.c_void_p(stream or None)))


def down_from_csc(indptr, indices, n: int) -> np.ndarray:
    """
    Recover the downstream-index vector from the CSC arrays the reference passes to its kernels
    (A[downstream, upstream] = 1, one entry per non-outlet column; tools.py:108-109).
    """
    indptr = np.asarray(indptr)
    indices = np.asarray(indices)
    if indptr.shape[0] != n + 1:
        raise ValueError('csc_indptr has the wrong length for this state vector')
    counts = np.diff(indptr)
    if counts.size and counts.max() > 1:
        raise ValueError('a river segment has more than one downstream segment; not a valid routing network')
    down = np.full(n, -1, dtype=np.int32)
    has = counts == 1
    down[has] = indices[indptr[:-1][has]]
    return down


class Plan:
    """Owns an ``rr_plan``.  ``down`` is the int32 downstream-index vector (-1 = outlet)."""

    RENUMBER = {'auto': 0, 'never': 1, 'always': 2}

    def __init__(self, down, time_tile: int = 0, tile_stride: int = 0, device: int = -1, threads_per_cta: int = 0,
                 raw_budget_bytes: int = 0, renumber: str = 'auto', staging: str = 'auto'):
        down = np.ascontiguousarray(down, dtype=np.int32)
        self.n = int(down.shape[0])
        self.down = down
        opts = _lib.PlanOpts(int(time_tile), int(tile_stride), int(device), int(threads_per_cta), int(raw_budget_bytes),
                             self.RENUMBER[renumber], {'auto': 0, 'registers': 1, 'registers-tiled': 2, 'tma': 3, 'out-reach-major': 4, 'lateral-grouped': 5, 'direct': 6, 'direct-nohw': 7}[staging])
        handle = C.c_void_p()
        check(lib.rr_plan_create(self.n, _lib.as_i32p(down), C.byref(opts), C.byref(handle)))
        self._h = handle
        self._coeff_key = None
        self.n_out = self.n                     # columns the host streaming calls copy back (see set_output_subset)
        self.threshold_labels = ()              # labels of the rows set by set_thresholds

    def close(self):
        if getattr(self, '_h', None):
            lib.rr_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def info(self) -> dict:
        inf = _lib.PlanInfo()
        check(lib.rr_plan_get_info(self._h, C.byref(inf)))
        return {k: getattr(inf, k) for k, _ in inf._fields_}

    def set_coefficients(self, c1, c2, c3, c4_dt=None):
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (c1, c2, c3)]
        c4 = None if c4_dt is None else np.ascontiguousarray(c4_dt, dtype=np.float64)
        for a in arrs + ([c4] if c4 is not None else []):
            if a.shape != (self.n,):
                raise ValueError('coefficient vectors must have one value per river segment')
        check(lib.rr_plan_set_coefficients(self._h, *[_lib.as_f64p(a) for a in arrs],
                                           _lib.as_f64p(c4) if c4 is not None else None))

    def set_output_subset(self, indices=None):
        """
        Copy back only these river segments (params-file indices, any order) from the host streaming calls -- the
        device-side form of the reference's subset-writer pattern (docs/tutorial/advanced.md:147-170).  ``None``
        or an empty list restores the full output.  The whole network is still routed.
        """
        idx = np.zeros(0, dtype=np.int32) if indices is None else np.ascontiguousarray(indices, dtype=np.int32)
        if idx.ndim != 1:
            raise ValueError('indices must be a 1D list of river segment indices')
        check(lib.rr_plan_set_output_subset(self._h, idx.shape[0], _lib.as_i32p(idx) if idx.shape[0] else None))
        self.n_out = int(idx.shape[0]) or self.n

    def set_thresholds(self, thresholds=None):
        """
        Per-river thresholds for the ``'exceed_<label>'`` ensemble statistics: an ordered mapping from label to a float
        (n,) array in params-file order (e.g. return-period flows; NaN: never exceeded).  The labels are kept in
        ``threshold_labels``; ``None`` or an empty mapping clears them.
        """
        items = list((thresholds or {}).items())
        labels = tuple(k for k, _ in items)
        if not all(isinstance(k, str) and k for k in labels) or len(set(labels)) != len(labels):
            raise ValueError(f'threshold labels must be distinct non-empty strings, got {list(labels)}')
        rows = np.empty((len(items), self.n), dtype=np.float64)
        for r, (label, a) in enumerate(items):
            a = np.asarray(a)
            if a.shape != (self.n,) or a.dtype.kind != 'f':
                raise ValueError(f'threshold {label!r} must be a float ({self.n},) array, got {a.dtype} {a.shape}')
            rows[r] = a
        check(lib.rr_plan_set_thresholds(self._h, len(items), _lib.as_f64p(rows) if items else None, self.n))
        self.threshold_labels = labels

    # ---- host arrays (numpy) : H2D / route / D2H streamed inside the library ----
    def route_host(self, mode: int, q_state: np.ndarray, lateral, out: np.ndarray, substeps: int, q_full=None,
                   resample: int = 1):
        """
        One reference kernel call on host arrays.  ``q_state`` (n,) is updated in place with the final state,
        ``out`` is overwritten.  ``lateral`` is (T, n) or None for MODE_MUSKINGUM.

        ``out`` is (T, n) float64 -- the reference kernel's contract -- or, for the router-level tail done on the
        device, (T / resample, n) float64 or float32: ``resample`` consecutive rows are averaged
        (TransformMuskingum.py:128-139) and a float32 ``out`` receives ``astype(np.float32)`` of that (:146).
        """
        if q_state.dtype != np.float64 or not q_state.flags.c_contiguous or q_state.shape != (self.n,):
            raise ValueError('q_state must be a contiguous float64 vector with one value per river segment')
        if out.dtype not in (np.float64, np.float32) or out.ndim != 2 or out.shape[1] != self.n_out:
            raise ValueError('discharge array must be float64 (or float32) with shape (T, n) '
                             '(n = size of the output subset when one is set)')
        resample = int(resample)
        if resample < 1:
            raise ValueError('resample must be a positive integer')
        T = out.shape[0] * resample
        ldo = _lib.rows_ld(out)
        p_lat, ldl, lat_f32 = None, self.n, False
        if mode != MODE_MUSKINGUM:
            if lateral.ndim != 2 or lateral.shape[1] != self.n or lateral.shape[0] != T:
                raise ValueError(f'lateral inflow shape {lateral.shape} does not match (T, n) = {(T, self.n)}')
            if lateral.dtype == np.float32 and (self.n == 1 or lateral.strides[1] == 4):
                lat_f32 = True       # crosses PCIe as stored, upcast (exactly) on the device: rr_route_host_typed
            elif lateral.dtype != np.float64 or (self.n > 1 and lateral.strides[1] != 8):
                # the reference's grid path hands over an F-ordered transposed view (runoff.py:298)
                lateral = np.ascontiguousarray(lateral, dtype=np.float64)
            ldl = _lib.rows_ld(lateral)
            p_lat = lateral.ctypes.data_as(_lib.c_f64p)
        p_qf = None
        if q_full is not None:
            if q_full.dtype != np.float64 or not q_full.flags.c_contiguous or q_full.shape != (self.n,):
                raise ValueError('q_full must be a contiguous float64 vector with one value per river segment')
            p_qf = _lib.as_f64p(q_full)
        if lat_f32:
            check(lib.rr_route_host_typed(self._h, int(mode), _lib.as_f64p(q_state), p_qf, C.cast(p_lat, C.c_void_p), 1, ldl,
                                          out.ctypes.data_as(C.c_void_p), ldo, T, int(substeps),
                                          int(out.dtype == np.float32), resample))
        elif out.dtype == np.float64 and resample == 1 and self.n_out == self.n:
            check(lib.rr_route_host(self._h, int(mode), _lib.as_f64p(q_state), p_qf, p_lat, ldl, _lib.as_f64p(out),
                                    ldo, T, int(substeps)))
        else:
            check(lib.rr_route_host_ex(self._h, int(mode), _lib.as_f64p(q_state), p_qf, p_lat, ldl,
                                       out.ctypes.data_as(C.c_void_p), ldo, T, int(substeps),
                                       int(out.dtype == np.float32), resample))

    def runoff_route_host(self, transform, mode: int, q_state: np.ndarray, runoff: np.ndarray, out: np.ndarray,
                          substeps: int, cumulative: bool = False, force_positive: bool = False,
                          as_volumes: bool = False, resample: int = 1):
        """
        Gathered grid runoff (T, n_points), float32 or float64, -> discharge in one device residency
        (``rr_runoff_route_host``): weight table [-> unit hydrograph] -> route -> resample / float32.
        ``transform`` is a :class:`river_route_b200.transforms.Transform` built for this plan's river order.
        """
        if q_state.dtype != np.float64 or not q_state.flags.c_contiguous or q_state.shape != (self.n,):
            raise ValueError('q_state must be a contiguous float64 vector with one value per river segment')
        if out.dtype not in (np.float64, np.float32) or out.ndim != 2 or out.shape[1] != self.n_out:
            raise ValueError('discharge array must be float64 (or float32) with shape (T, n) '
                             '(n = size of the output subset when one is set)')
        if transform.n_rivers != self.n:
            raise ValueError('weight table rows do not match the number of river segments')
        resample = int(resample)
        if resample < 1:
            raise ValueError('resample must be a positive integer')
        T = out.shape[0] * resample
        if runoff.dtype not in (np.float32, np.float64):
            runoff = runoff.astype(np.float64)
        if runoff.ndim != 2 or runoff.shape != (T, transform.n_points):
            raise ValueError(f'runoff shape {runoff.shape} does not match (T, n_points) = {(T, transform.n_points)}')
        if transform.n_points > 1 and runoff.strides[1] != runoff.itemsize:
            runoff = np.ascontiguousarray(runoff)
        check(lib.rr_runoff_route_host(self._h, transform._h, int(mode), _lib.as_f64p(q_state),
                                       runoff.ctypes.data_as(C.c_void_p), int(runoff.dtype == np.float32),
                                       _lib.rows_ld(runoff), T, int(cumulative), int(force_positive), int(as_volumes),
                                       out.ctypes.data_as(C.c_void_p), _lib.rows_ld(out), int(substeps),
                                       int(out.dtype == np.float32), resample))

    # ---- device pointers (torch tensors used purely as device buffers) ----
    def route_dev(self, mode: int, q_state_ptr: int, lateral_ptr: int, ldl: int, out_ptr: int, ldo: int, T: int,
                  substeps: int, stream: int = 0, q_full_ptr: int = 0):
        check(lib.rr_route_dev(self._h, int(mode), C.c_void_p(q_state_ptr), C.c_void_p(q_full_ptr or None),
                               C.c_void_p(lateral_ptr or None), int(ldl), C.c_void_p(out_ptr), int(ldo), int(T),
                               int(substeps), C.c_void_p(stream or None)))

    def route_ensemble_dev(self, mode: int, q_init_ptr: int, lateral_ptrs, ldl: int, out_ptrs, ldo: int,
                           q_final_ptrs, T: int, substeps: int, stream: int = 0):
        m = len(out_ptrs)
        arr = C.c_void_p * m
        lat = arr(*lateral_ptrs) if lateral_ptrs else None
        check(lib.rr_route_ensemble_dev(self._h, int(mode), C.c_void_p(q_init_ptr), m, lat, int(ldl), arr(*out_ptrs),
                                        int(ldo), arr(*q_final_ptrs), int(T), int(substeps),
                                        C.c_void_p(stream or None)))

    def route_ensemble_host(self, mode: int, q_init: np.ndarray, laterals, outs, substeps: int, resample: int = 1,
                            q_final: np.ndarray | None = None):
        """
        ``len(outs)`` ensemble members from host arrays (pinned for full PCIe rate) in one call: every member starts
        from ``q_init`` (n,) (TransformMuskingum.py:121-126) -- or, for a later time slab of the same members, from its
        own row of ``q_init`` (members, n) --, the members of each time chunk share one launch, and the
        returned vector is the mean of the members' final states in member order (:145-146).  ``laterals[m]`` is
        (T, n) float64 or float32 (all members the same dtype; None for MODE_MUSKINGUM), ``outs[m]`` (T / resample, n)
        float64 or float32 (all the same dtype); ``q_final`` (members, n), if given, receives the members' states.
        """
        M = len(outs)
        if M < 1 or (mode != MODE_MUSKINGUM and len(laterals) != M):
            raise ValueError('one lateral array and one discharge array per member')
        if q_init.dtype != np.float64 or not q_init.flags.c_contiguous or q_init.shape not in ((self.n,), (M, self.n)):
            raise ValueError('q_init must be a contiguous float64 (n,) vector or (members, n) array')
        ld_init = self.n if q_init.ndim == 2 else 0
        resample = int(resample)
        T = outs[0].shape[0] * resample
        odt = outs[0].dtype
        for o in outs:
            if o.dtype != odt or odt not in (np.float64, np.float32) or o.shape != (T // resample, self.n) or \
                    _lib.rows_ld(o) != _lib.rows_ld(outs[0]):
                raise ValueError('discharge arrays must share dtype (float64 / float32), shape (T, n) and row stride')
        arr = C.c_void_p * M
        p_lat, ldl, lat_f32 = None, self.n, 0
        if mode != MODE_MUSKINGUM:
            ldt = laterals[0].dtype
            lat_f32 = int(ldt == np.float32)
            for a in laterals:
                if a.dtype != ldt or ldt not in (np.float64, np.float32) or a.shape != (T, self.n) or \
                        _lib.rows_ld(a) != _lib.rows_ld(laterals[0]):
                    raise ValueError('lateral arrays must share dtype (float64 / float32), shape (T, n) and row stride')
            ldl = _lib.rows_ld(laterals[0])
            p_lat = arr(*[a.ctypes.data for a in laterals])
        q_mean = np.empty(self.n, dtype=np.float64)
        if q_final is not None and (q_final.dtype != np.float64 or q_final.shape != (M, self.n) or not q_final.flags.c_contiguous):
            raise ValueError('q_final must be a contiguous float64 (members, n) array')
        check(lib.rr_route_ensemble_host(self._h, int(mode), _lib.as_f64p(q_init), ld_init, M, p_lat, lat_f32, ldl,
                                         arr(*[o.ctypes.data for o in outs]), _lib.rows_ld(outs[0]), int(odt == np.float32),
                                         _lib.as_f64p(q_final) if q_final is not None else None, self.n,
                                         _lib.as_f64p(q_mean), T, int(substeps), resample))
        return q_mean

    def route_ensemble_stats_host(self, mode: int, q_init: np.ndarray, laterals, stats, outs, substeps: int,
                                  resample: int = 1, q_final: np.ndarray | None = None, peaks=None):
        """
        As ``route_ensemble_host`` -- same members, inputs, state chaining, ``q_final`` and returned member-mean state --
        but the members' discharge stays on the device: per time chunk it is averaged over ``resample`` rows and reduced
        to the statistics named in ``stats`` (see ``parse_statistics``; ``'exceed_<label>'`` against the labels of
        ``set_thresholds``), and only those cross PCIe.  ``outs[s]`` is (T / resample, n_out) float32 or float64 (all
        the same dtype) for statistic ``stats[s]``; n_out follows the output subset (``set_output_subset``).  Every
        statistic equals numpy on the stacked fp64 member outputs bit for bit (``np.mean`` / ``np.std`` / ``np.min`` /
        ``np.max`` / ``np.percentile`` over axis 0; exceedance ``np.mean(x > thr, axis=0)``).

        ``peaks = (values, rows)``, (S, n_out) float64 and int32 arrays, receives each statistic's maximum over this
        call's output rows and the first row where it occurs (``rows.max(axis=0)`` / ``rows.argmax(axis=0)`` of the fp64
        statistic rows), kept on the device for the whole call.  ``outs`` may then be ``None``: no per-step rows are
        kept or copied back, and T comes from the lateral arrays.
        """
        spec = _stats_spec(stats, self.threshold_labels)
        M = len(laterals) if laterals is not None else 0
        if mode == MODE_MUSKINGUM:
            raise ValueError('ensemble statistics need lateral inflows (RapidMuskingum members)')
        if not 1 <= M <= 64:
            raise ValueError('ensemble statistics need 1 to 64 members')
        if outs is None and peaks is None:
            raise ValueError('give per-step arrays (outs), peaks or both')
        if outs is not None and len(outs) != spec.n_stats:
            raise ValueError('one output array per statistic')
        if q_init.dtype != np.float64 or not q_init.flags.c_contiguous or q_init.shape not in ((self.n,), (M, self.n)):
            raise ValueError('q_init must be a contiguous float64 (n,) vector or (members, n) array')
        ld_init = self.n if q_init.ndim == 2 else 0
        resample = int(resample)
        n_out = self.n_out
        T = outs[0].shape[0] * resample if outs is not None else laterals[0].shape[0]
        if outs is not None:
            odt = outs[0].dtype
            for o in outs:
                if o.dtype != odt or odt not in (np.float64, np.float32) or o.shape != (T // resample, n_out) or \
                        _lib.rows_ld(o) != _lib.rows_ld(outs[0]):
                    raise ValueError('statistic arrays must share dtype (float64 / float32), shape (T / resample, n_out) and row stride')
        ldt = laterals[0].dtype
        for a in laterals:
            if a.dtype != ldt or ldt not in (np.float64, np.float32) or a.shape != (T, self.n) or \
                    _lib.rows_ld(a) != _lib.rows_ld(laterals[0]):
                raise ValueError('lateral arrays must share dtype (float64 / float32), shape (T, n) and row stride')
        if q_final is not None and (q_final.dtype != np.float64 or q_final.shape != (M, self.n) or not q_final.flags.c_contiguous):
            raise ValueError('q_final must be a contiguous float64 (members, n) array')
        if peaks is not None:
            pv, pr = peaks
            if pv.dtype != np.float64 or pr.dtype != np.int32 or pv.shape != (spec.n_stats, n_out) or \
                    pr.shape != pv.shape or not (pv.flags.c_contiguous and pr.flags.c_contiguous):
                raise ValueError('peaks must be contiguous (S, n_out) float64 values and int32 rows')
        q_mean = np.empty(self.n, dtype=np.float64)
        arr_m, arr_s = C.c_void_p * M, C.c_void_p * spec.n_stats
        check(lib.rr_route_ensemble_stats_host_ex(
            self._h, int(mode), _lib.as_f64p(q_init), ld_init, M, arr_m(*[a.ctypes.data for a in laterals]),
            int(ldt == np.float32), _lib.rows_ld(laterals[0]), C.byref(spec),
            arr_s(*[o.ctypes.data for o in outs]) if outs is not None else None,
            _lib.rows_ld(outs[0]) if outs is not None else 0, int(outs is not None and odt == np.float32),
            _lib.as_f64p(q_final) if q_final is not None else None, self.n, _lib.as_f64p(q_mean), T, int(substeps), resample,
            _lib.as_f64p(pv) if peaks is not None else None, _lib.as_i32p(pr) if peaks is not None else None,
            n_out if peaks is not None else 0))
        return q_mean

    def tile_rows(self, T: int, substeps: int = 1) -> int:
        """Output rows per work item the library picks for a call of T rows (its per-call cost model)."""
        return int(lib.rr_plan_tile_rows(self._h, int(T), int(substeps)))

    def read_profile(self):
        """Cycle counters of -DRR_PROFILE builds: ticket/decode, constants+waits, item body, publish (summed over warps)."""
        out = (C.c_uint64 * 8)()
        check(lib.rr_plan_read_profile(self._h, out))
        return list(out)

    # ---- introspection (tests, DESIGN.md numbers) ----
    def arrays(self) -> dict:
        inf = self.info
        ptrs = [_lib.c_i32p(), _lib.c_i32p(), _lib.c_u8p()] + [_lib.c_i32p() for _ in range(7)]
        check(lib.rr_plan_get_arrays(self._h, *[C.byref(p) for p in ptrs]))
        n, e, nb, nd = inf['n_work'], inf['n_edges'], inf['n_blocks'], inf['n_dep_edges']   # working slots (see 'perm')
        sizes = [n + 1, e, n, e, n, nb, nb + 1, nd, inf['n_export'], n if inf['renumbered'] else 0]
        names = ['up_ptr', 'up_idx', 'skew', 'slot_src', 'export_id', 'blk_level', 'dep_ptr', 'dep_idx', 'exp_span',
                 'perm']
        out = {}
        for name, p, sz in zip(names, ptrs, sizes):
            out[name] = np.ctypeslib.as_array(p, shape=(sz,)).copy() if sz > 0 else np.zeros(0, dtype=np.int32)
        # downstream slot in the WORKING order (== self.down unless the plan is renumbered).  A renumbered plan pads
        # every level to whole blocks: perm[slot] is the user index of the slot, -1 for padding
        if inf['renumbered']:
            perm = out['perm']
            real = perm >= 0
            inv = np.empty(self.n, dtype=np.int64)
            inv[perm[real]] = np.flatnonzero(real)
            d = self.down[perm[real]]
            down_w = np.full(n, -1, dtype=np.int32)
            down_w[real] = np.where(d >= 0, inv[np.where(d >= 0, d, 0)], -1)
            out['down'] = down_w
            out['inv'] = inv
        else:
            out['perm'] = None
            out['down'] = self.down
        return out

    def schedule(self, n_tiles: int, tile_stride: int):
        """Ticket order as (block, tile) pairs -- the kernel decodes tickets with the same table."""
        nb = self.info['n_blocks']
        blocks = np.empty(nb * n_tiles, dtype=np.int32)
        tiles = np.empty(nb * n_tiles, dtype=np.int32)
        n_items = C.c_int64(0)
        check(lib.rr_plan_schedule(self._h, int(n_tiles), int(tile_stride), C.byref(n_items), _lib.as_i32p(blocks),
                                   _lib.as_i32p(tiles)))
        assert n_items.value == nb * n_tiles
        return blocks, tiles


def launch_count(reset: bool = False) -> int:
    """Kernel launches issued by the library on this thread (bench.py's gpu_launches)."""
    return int(lib.rr_launch_count(1 if reset else 0))


def timing_enable(on: bool = True) -> None:
    """Record CUDA events around every kernel this library launches (read with ``timing_read``)."""
    lib.rr_timing_enable(1 if on else 0)


def timing_read(reset: bool = True) -> dict:
    """Accumulated device time (ms) and launch counts per kernel class since the last reset."""
    ms = (C.c_double * 4)()
    cnt = (C.c_int64 * 4)()
    lib.rr_timing_read(ms, cnt, 1 if reset else 0)
    names = ('route', 'permute_to_working', 'permute_to_user', 'other')
    return {n: {'ms': ms[i], 'launches': cnt[i]} for i, n in enumerate(names)}
