"""B200-native drop-in for the reference's HDDStream (clustering/hddstream.py:29-549).

Same constructor, same entry point `online_microcluster_maintenance(input_dataset, daystamp, reset_param)`,
same attributes read by app.run (`pcore_MC`, `outlier_MC`, `final_clusters`, `last_data_timestamp`, ...).
All clustering arithmetic runs in hand-written sm_100a CUDA kernels behind the C ABI of
include/chronoclust_b200.h; this class only derives the scalar parameters with Python's own float
semantics (exactly where the reference derives them), moves arrays across the boundary and wraps the
exported state in Microcluster / FinalCluster objects.  There is no CPU fallback.
"""
import ctypes as C
import logging
import sys

import numpy as np

from . import _hostio, _lib, cellstats
from .scaling import cofactor_vector
from .objects import FinalCluster, Microcluster


_NP_DTYPES = {np.dtype(np.float64): _lib.DTYPE_F64, np.dtype(np.float32): _lib.DTYPE_F32}


def _input_rows(x, device):
    """How input_dataset goes to ccb_ingest_ex: (pointer, CCB_DTYPE_*, on_device, ld, rows), `rows` being the array or
    tensor the pointer points into (the caller's own where possible; keep it alive until the call returns).

    float32 / float64 rows with unit column stride and a row stride >= D go in without a copy, with ld = the row stride:
    numpy arrays and CPU tensors as host input, CUDA tensors on the handle's `device` as device input (a CUDA tensor on
    another device raises ValueError).  Everything else is made float64 and C-contiguous on the host, as numpy does."""
    torch = sys.modules.get("torch")  # a caller that passes a tensor has imported torch
    if torch is not None and isinstance(x, torch.Tensor):
        x = x.detach()
        if x.is_cuda:
            if x.device.index != device:
                raise ValueError(f"input_dataset is on {x.device}, this HDDStream runs on cuda:{device}")
            code = {torch.float64: _lib.DTYPE_F64, torch.float32: _lib.DTYPE_F32}.get(x.dtype)
            if code is not None and x.dim() == 2 and x.shape[0] > 0 and x.stride(1) == 1:
                ld = x.stride(0) if x.shape[0] > 1 else x.shape[1]  # (the stride of a single row means nothing)
                if ld >= x.shape[1]:
                    return x.data_ptr(), code, True, ld, x
        x = x.cpu().numpy()
    if isinstance(x, np.ndarray) and x.ndim == 2 and x.shape[0] > 0 and x.flags.aligned:
        code, isz = _NP_DTYPES.get(x.dtype), x.dtype.itemsize  # (a byte-swapped dtype is not among the keys)
        ld = x.strides[0] // isz if x.shape[0] > 1 else x.shape[1]  # (the stride of a single row means nothing)
        if code is not None and x.strides[1] == isz and x.strides[0] % isz == 0 and ld >= x.shape[1]:
            return x.ctypes.data, code, False, ld, x
    x = np.ascontiguousarray(x, dtype=np.float64)
    return x.ctypes.data, _lib.DTYPE_F64, False, (x.shape[1] if x.ndim == 2 else 0), x


def column_map(columns, width):
    """`columns` as int32 indices into rows `width` wide (HDDStream.online_microcluster_maintenance(columns=)).  ValueError
    for rows wider than 64 columns, an empty list, more than 64 entries, or an entry that is not an integer, lies outside
    [0, width) or repeats an earlier one."""
    if width > 64:
        raise ValueError(f"rows of {width} columns: at most 64 are supported")
    try:
        entries = list(columns)
    except TypeError:
        raise ValueError("columns must be a sequence of column indices") from None
    if not 1 <= len(entries) <= 64:
        raise ValueError(f"columns holds {len(entries)} entries; 1 to 64 are supported")
    out = []
    for c in entries:
        if isinstance(c, (bool, np.bool_)) or not isinstance(c, (int, np.integer)):
            raise ValueError(f"column {c!r} is not an integer")
        if not 0 <= int(c) < width:
            raise ValueError(f"column {int(c)} outside [0, {width})")
        if int(c) in out:
            raise ValueError(f"column {int(c)} appears twice")
        out.append(int(c))
    return np.array(out, np.int32)


class _PointsView(object):
    """Per-timepoint cell -> MC assignment; builds Microcluster.points dicts on demand.  The input arrays or tensors are
    BORROWED, not copied (the reference copies every row into a Python list, microcluster.py:149): a caller that
    overwrites its array or tensor in place after the call changes what `points` hands out.  float32 rows are handed out
    widened to float64, and the rows of a CUDA tensor are gathered on its device and brought back as float64 -- the same
    values the float64 path hands out.  Rows ingested with a column map hand out their clustering columns only, in map
    order; rows ingested with arcsinh cofactors hand out the transformed values (the host's ccbio_arcsinh_host, the
    device's bits)."""

    def __init__(self):
        self.segments = []  # [(X, assign_uid, scaler, column map, cofactors)] since the last reset (hddstream.py:208-213)
        self._index = None

    def reset(self):
        self.segments = []
        self._index = None

    def add(self, X, assign, scaler=None, cols=None, cof=None):
        """scaler = (scale_, min_): X holds RAW rows that were scaled on the device; the coordinates handed out are
        X * scale_ + min_ of the requested rows (numpy's elementwise arithmetic = the device's two roundings).
        cols: int32 column map into the rows of X (the coordinates are X[:, cols]), or None.  cof: float64 arcsinh
        cofactors by column of X (applied before the scaler), or None."""
        self.segments.append((X, assign, scaler, cols, cof))
        self._index = None

    def _build(self):
        idx = {}
        for si, (_, assign, _sc, _cols, _cof) in enumerate(self.segments):
            order = np.argsort(assign, kind="stable")
            sa = assign[order]
            cuts = np.flatnonzero(np.diff(sa)) + 1
            starts = np.concatenate(([0], cuts))
            ends = np.concatenate((cuts, [len(sa)]))
            for s, e in zip(starts, ends):
                if e > s:
                    idx.setdefault(int(sa[s]), []).append((si, order[s:e]))
        self._index = idx

    def rows_of(self, uid):
        """[(segment index, ascending row indices)] of the cells absorbed by MC `uid`."""
        if self._index is None:
            self._build()
        return self._index.get(int(uid), [])

    def points_of(self, uid):
        out = {}
        for si, rows in self.rows_of(uid):
            X, _, sc, cols, cof = self.segments[si]
            if isinstance(X, np.ndarray):
                sel = X[rows] if cols is None else X[np.ix_(rows, cols)]
            else:  # a CUDA tensor
                import torch

                sel = X[torch.from_numpy(rows).to(X.device)]
                if cols is not None:
                    sel = sel[:, torch.from_numpy(cols.astype(np.int64)).to(X.device)]
                sel = sel.cpu().numpy()
            if cof is not None:  # (widened, then transformed, before the scaler arithmetic)
                sel = _hostio.arcsinh_host(sel, cof if cols is None else cof[cols])
            else:
                sel = sel.astype(np.float64, copy=False)
            if sc is not None:
                sel = sel * sc[0]
                sel = sel + sc[1]
            vals = sel.tolist()
            for r, v in zip(rows.tolist(), vals):
                out[r] = v
        return out


class HDDStream(object):
    # CUDA ordinal an unpickled instance comes back on (pickle cannot pass constructor arguments): app.run(device=n,
    # restore_program=True) sets it before loading program_images/hddstream
    restore_device = 0

    def __init__(self, config, logger, device=0, chunk=0, bsv_bmin=0, bsv_iters=0, bsv_stream=0, off_csr_min_m=0):
        """config: dict with beta, delta, epsilon, lambda, k, mu, pi, omicron, upsilon (hddstream.py:30-67)."""
        self.config = config
        self.pi = None
        self.mu = None
        self.epsilon = float(self.config['epsilon'])
        self.epsilon_squared = self.epsilon ** 2
        self.upsilon = float(self.config['upsilon']) * self.epsilon
        self.delta = self.calculate_pref_dim_variance_threshold()
        self.delta_squared = self.delta ** 2
        self.beta = float(self.config['beta'])
        self.k = float(self.config['k'])
        self.lambbda = float(self.config['lambda'])
        self.omicron = None

        self.final_clusters = []
        self.last_data_timestamp = 0
        self.dataset_dimensionality = 0
        self.logger = logger if logger is not None else logging.getLogger("chronoclust_b200")
        self.dataset_size = 0

        # engine knobs (never affect results): chunk caps the block length of the ordered engine, bsv_* shape its blocks
        # and rounds, off_csr_min_m moves the switch between the two formulations of the offline cluster growth
        self._device, self._chunk = device, chunk
        self._bsv = (bsv_bmin, bsv_iters, bsv_stream, off_csr_min_m)
        self._h = None
        self._handle_dim = 0  # D of the handle
        self._views = _PointsView()
        self._lists = [None, None]  # cached Microcluster lists (pcore, outlier)
        self.last_assignment = None  # uid of the MC every row of the last call went to
        self.last_stage = None
        self.last_cluster_label = None  # cluster index of every pcore MC (list order) after the offline phase
        self._last_device_input = None  # (rows, assignments) of the last CUDA-tensor ingest, read by cluster_statistics
        self._stats_width = None  # columns of the rows of the last ingest, when they are not dataset_dimensionality

    # ------------------------------------------------------------------------------------------
    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                _lib.lib().ccb_destroy(h)
            except Exception:
                pass

    def __getstate__(self):
        """Same tuple layout as the reference (hddstream.py:69-73), lists as real objects."""
        return (self.pi, self.mu, self.epsilon, self.epsilon_squared, self.upsilon, self.delta, self.delta_squared,
                self.beta, self.k, self.lambbda, self.omicron, self.pcore_MC, self.outlier_MC,
                self.last_data_timestamp, self.dataset_dimensionality, self.dataset_size,
                self.pcore_MC_last_id, self.outlier_MC_last_id, self.config)

    def __setstate__(self, state):
        (self.pi, self.mu, self.epsilon, self.epsilon_squared, self.upsilon, self.delta, self.delta_squared,
         self.beta, self.k, self.lambbda, self.omicron, pcore, outlier, self.last_data_timestamp,
         self.dataset_dimensionality, self.dataset_size) = state[:16]
        pl, ol = (state[16], state[17]) if len(state) > 17 else (None, None)
        self.config = state[18] if len(state) > 18 else None
        self.final_clusters = []
        self.logger = logging.getLogger("chronoclust_b200")
        self._device = type(self).restore_device
        self._chunk = 0
        self._bsv = (0, 0, 0, 0)
        self._h = None
        self._handle_dim = 0
        self._views = _PointsView()
        self._lists = [None, None]
        self.last_assignment = self.last_stage = self.last_cluster_label = None
        self._last_device_input = self._stats_width = None
        if self.dataset_dimensionality:
            self._ensure_handle(self.dataset_dimensionality)
            self._import(0, pcore)
            self._import(1, outlier)
            if pl is None:  # the reference forgets its counters when pickling; recover the smallest safe ones
                pl = 1 + max([int(list(m.id)[0]) for m in pcore] + [-1])
                ol = 1 + max([int(m.prev_outlier_id) for m in list(pcore) + list(outlier)] + [-1])
            _lib.check(_lib.lib().ccb_set_counters(self._h, int(pl), int(ol)), self._h)

    def set_logger(self, logger):
        self.logger = logger

    def set_config(self, config):
        self.config = config

    # ------------------------------------------------------------------------------------------
    def calculate_pref_dim_variance_threshold(self):
        variance_threshold = float(self.config['delta'])
        if variance_threshold > 1 or variance_threshold < 0:
            sys.exit("Given delta ({}) is out of range. Must be within 0-1.".format(variance_threshold))
        return variance_threshold

    def calculate_density_threshold(self):
        return float(self.config['mu']) * self.dataset_size

    def _set_dataset_dependent_parameters(self, input_dataset, dataset_dim=None):
        # hddstream.py:89-128: omicron from the PREVIOUS dataset size, then mu from the current one
        if dataset_dim is None:
            dataset_dim = input_dataset.shape[1]
        self.dataset_dimensionality = dataset_dim
        config_pi = float(self.config['pi'])
        self.pi = dataset_dim if config_pi <= 0 else round(config_pi)
        self.omicron = self.config['omicron'] * self.dataset_size
        self.dataset_size = input_dataset.shape[0]
        self.mu = self.calculate_density_threshold()

    def _ensure_handle(self, D):
        if self._h is not None:
            return
        L = _lib.lib()
        prm = _lib.Params(D=D, device=self._device, eps2=self.epsilon_squared, upsilon_eps=self.upsilon,
                          upsilon_eps2=self.upsilon ** 2, delta=self.delta, delta2=self.delta_squared, beta=self.beta,
                          k=self.k, chunk=self._chunk, bsv_bmin=self._bsv[0], bsv_iters=self._bsv[1],
                          bsv_stream=self._bsv[2], off_csr_min_m=self._bsv[3])
        h = C.c_void_p()
        rc = L.ccb_create(C.byref(prm), C.byref(h))
        if rc != 0:
            _lib.check(rc, None)
        self._h, self._handle_dim = h, D
        try:
            _lib.check(L.ccb_set_dnrm2(h, _lib.scipy_dnrm2_pointer()), h)
        except ImportError:
            pass  # the built-in restatement of OpenBLAS' x87 dnrm2 settles borderline pairs instead

    # ------------------------------------------------------------------------------------------
    def online_microcluster_maintenance(self, input_dataset, input_dataset_daystamp, reset_param=True,
                                        run_offline=True, scaler=None, columns=None, cofactors=None):
        """input_dataset: [N, D] cells -- a numpy array, a CPU tensor or a CUDA tensor on this instance's device.  float32 and
        float64 rows with unit column stride go in without a copy (row-strided views included); float32 rows are widened
        to float64 on the device, which is exact, so results are those of the float64 path on the widened rows.  Other
        inputs are made float64 on the host first.  For a CUDA tensor the call waits for the work queued on the current
        torch stream of its device; last_assignment / last_stage come back to the host either way.

        scaler (extension, SURVEY 8f-3): a fitted sklearn MinMaxScaler (or a (scale_, min_) pair) -- input_dataset then
        holds RAW rows and the min-max transform x * scale_ + min_ runs on the device behind the host -> device copy
        (ccb_ingest_ex) instead of as a host pass; results are those of scaling on the host first, bit for bit.

        columns (extension): a sequence of D distinct column indices into input_dataset's W <= 64 columns -- the engine then
        clusters input_dataset[:, columns] (dataset_dimensionality = D) and gives bit for bit what the float64 path gives on
        those gathered rows; the gather runs on the device, the rows go in without a copy as above, and the scaler's vectors
        have D entries.  `points` hands out the gathered coordinates, and cluster_statistics reports all W columns.
        ValueError before any device work for a bad entry (see column_map) or a D that differs from the handle's.

        cofactors (extension): the arcsinh transform of cytometry intensities, run on the device as the rows are staged --
        a number for every column, or one per column of input_dataset (W entries with `columns`, by input column); a
        column with cofactor c > 0 is clustered as asinh(x / c) (scaling.arcsinh: widened first, one IEEE division, then
        csrc/asinh.h, the same bits on host and device), one with c = 0 stays linear.  The order is: widen, gather,
        asinh, scaler, so the scaler belongs to the transformed values.  Results are those of the float64 path on
        scaling.arcsinh(input_dataset, cofactors) (then gathered), bit for bit; `points` and cluster_statistics report
        transformed columns in transformed space.  ValueError before any device work for a bad cofactor (see
        scaling.cofactor_vector)."""
        xp, dtype, on_device, ld, X = _input_rows(input_dataset, self._device)
        if X.ndim != 2:
            raise ValueError("input_dataset must be 2-D")
        cols = None if columns is None else column_map(columns, X.shape[1])
        D = X.shape[1] if cols is None else len(cols)
        if cols is not None and self._h is not None and D != self._handle_dim:
            raise ValueError(f"{D} columns given; this HDDStream clusters {self._handle_dim} markers")
        cof = None if cofactors is None else cofactor_vector(cofactors, X.shape[1])
        sc = mn = None
        if scaler is not None:
            sc, mn = (scaler.scale_, scaler.min_) if hasattr(scaler, "scale_") else scaler
            sc = np.ascontiguousarray(sc, np.float64)
            mn = np.ascontiguousarray(mn, np.float64)
            if sc.shape != (D,) or mn.shape != (D,):
                raise ValueError("scaler vectors must have one entry per marker")
        if reset_param:
            self._set_dataset_dependent_parameters(X, D)
        self._ensure_handle(D)
        L, h, logger = _lib.lib(), self._h, self.logger
        logger.info(f"Setting up online phase for timepoint {input_dataset_daystamp} with following params:\n"
                    f"Pcore density threshold factor(beta) = {self.beta}\n"
                    f"Decay rate(lambda) = {self.lambbda}\n"
                    f"Radius threshold(epsilon) = {self.epsilon}\n"
                    f"Max projected dimensionality(pi) = {self.pi}\n"
                    f"Density threshold(mu) = {self.mu} = {self.mu}\n"
                    f"Variance threshold(delta) = {self.delta}\n"
                    f"K = {self.k}\n"
                    f"PreDeCon epsilon(upsilon) = {self.upsilon}\n"
                    f"Outlier deletion point(omicron) = {self.omicron}\n")
        decay = (self.last_data_timestamp - input_dataset_daystamp) != 0
        factor = 1.0
        if decay:
            logger.info("Decaying and downgrading microclusters")
            interval = input_dataset_daystamp - self.last_data_timestamp
            factor = 2 ** (-self.lambbda * interval)  # hddstream.py:283, Python float power
            # a NEW view per timepoint (hddstream.py:208-213 clears the points): Microcluster copies kept by the trackers
            # stay bound to the view -- cells and assignment -- of the timepoint they were made in
            self._views = _PointsView()
        _lib.check(L.ccb_begin_timepoint(h, float(self.mu), float(self.omicron), int(self.pi), int(decay),
                                         float(factor)), h)
        N = X.shape[0]
        logger.info("Starting online microcluster maintenance for timepoint {}".format(input_dataset_daystamp))
        self._last_device_input = self._stats_width = None
        if on_device:
            assign, stage = self._ingest_tensor(X, xp, dtype, ld, sc, mn, cols, cof)
        else:
            assign = np.empty(N, np.int32)
            stage = np.empty(N, np.uint8)
            _lib.check(L.ccb_ingest_tx(h, xp, dtype, 0, N, ld, X.shape[1], _lib.ptr(cols), _lib.ptr(cof), _lib.ptr(sc),
                                       _lib.ptr(mn), _lib.ptr(assign), _lib.ptr(stage)), h)
        if cols is not None:
            self._stats_width = X.shape[1]
        self._views.add(X, assign, None if sc is None else (sc, mn), cols, cof)
        self.last_assignment, self.last_stage = assign, stage
        self._lists = [None, None]
        logger.info("Finish online microcluster maintenance for timepoint {}".format(input_dataset_daystamp))
        cnt = self.counts()
        logger.info("Online maintenance yield {} pcores and {} outlier".format(cnt[0], cnt[1]))
        self.last_data_timestamp = input_dataset_daystamp
        if run_offline:
            self.offline_clustering(input_dataset_daystamp)

    def _ingest_tensor(self, X, xp, dtype, ld, sc, mn, cols=None, cof=None):
        """ccb_ingest_tx on the rows of a CUDA tensor X: the handle's stream first waits for the work queued on the current
        torch stream (whatever produced X), and the per-cell results come back to the host behind the engine."""
        import torch

        N = X.shape[0]
        mine = torch.cuda.ExternalStream(self.stream_ptr, device=X.device)
        cur = torch.cuda.current_stream(X.device)
        assign_d = torch.empty(N, dtype=torch.int32, device=X.device)
        stage_d = torch.empty(N, dtype=torch.uint8, device=X.device)
        mine.wait_stream(cur)  # (after the allocations: earlier users of that memory on `cur` are done first)
        _lib.check(_lib.lib().ccb_ingest_tx(self._h, xp, dtype, 1, N, ld, X.shape[1], _lib.ptr(cols), _lib.ptr(cof),
                                            _lib.ptr(sc), _lib.ptr(mn), assign_d.data_ptr(), stage_d.data_ptr()), self._h)
        # the copies, and the release of the temporaries, are ordered on `cur` behind everything the handle queued
        cur.wait_stream(mine)
        self._last_device_input = (X, assign_d)  # the handle reads both again in cluster_statistics
        return assign_d.cpu().numpy(), stage_d.cpu().numpy()

    def offline_clustering(self, dataset_daystamp):
        L, h = _lib.lib(), self._h
        nc = C.c_int64(0)
        _lib.check(L.ccb_offline(h, C.byref(nc)), h)
        sizes = (C.c_int64 * 3)()
        _lib.check(L.ccb_cluster_sizes(h, C.byref(sizes)), h)
        ncl, nmem, M = int(sizes[0]), int(sizes[1]), int(sizes[2])
        D = self.dataset_dimensionality
        off, mem = np.zeros(ncl + 1, np.int64), np.zeros(nmem, np.int64)
        w = np.zeros(ncl, np.float64)
        cf1, cf2, cen, pref = (np.zeros((ncl, D), np.float64) for _ in range(4))
        label = np.full(M, -1, np.int32)
        _lib.check(L.ccb_export_clusters(h, _lib.ptr(off), _lib.ptr(mem), _lib.ptr(w), _lib.ptr(cf1), _lib.ptr(cf2),
                                         _lib.ptr(cen), _lib.ptr(pref), _lib.ptr(label)), h)
        self.final_clusters = [
            FinalCluster(mem[off[c]:off[c + 1]], cf1[c].copy(), cf2[c].copy(), float(w[c]), cen[c].copy(), pref[c].copy())
            for c in range(ncl)]
        self.last_cluster_label = label
        self.logger.info('Finish offline clustering for dataset with timepoint: {}'.format(dataset_daystamp))
        self.logger.info("Offline clustering yield {} clusters.".format(len(self.final_clusters)))

    # ------------------------------------------------------------------------------------------
    def counts(self):
        out = (C.c_int64 * 4)()
        _lib.check(_lib.lib().ccb_counts(self._h, C.byref(out)), self._h)
        return [int(v) for v in out]

    def stats(self):
        st = _lib.Stats()
        _lib.check(_lib.lib().ccb_get_stats(self._h, C.byref(st)), self._h)
        return st.as_dict()

    def reset(self):
        """Forgets all microclusters and counters (a new run with the same parameters and device)."""
        if self._h is not None:
            _lib.check(_lib.lib().ccb_reset(self._h), self._h)
        self._views = _PointsView()
        self._lists = [None, None]
        self.final_clusters = []
        self.last_data_timestamp = 0
        self.dataset_size = 0
        self.last_assignment = self.last_stage = self.last_cluster_label = None
        self._last_device_input = self._stats_width = None

    @property
    def stream_ptr(self):
        return _lib.lib().ccb_stream(self._h)

    def ingest_device(self, x_ptr, N, ld, daystamp, assign_ptr, stage_ptr=None, run_offline=True):
        """online_microcluster_maintenance for a dataset already resident on the handle's device
        (raw device pointers; per-row results stay on the device).  Used by bench.py for `value`."""
        L, h = _lib.lib(), self._h
        shape = type("S", (), {"shape": (N, self.dataset_dimensionality)})
        self._set_dataset_dependent_parameters(shape)
        decay = (self.last_data_timestamp - daystamp) != 0
        factor = 2 ** (-self.lambbda * (daystamp - self.last_data_timestamp)) if decay else 1.0
        _lib.check(L.ccb_begin_timepoint(h, float(self.mu), float(self.omicron), int(self.pi), int(decay),
                                         float(factor)), h)
        _lib.check(L.ccb_ingest_device(h, x_ptr, N, ld, assign_ptr, stage_ptr), h)
        self._stats_width = None
        self._lists = [None, None]
        self.last_data_timestamp = daystamp
        if run_offline:
            self.offline_clustering(daystamp)

    def enable_timing(self, on=True):
        _lib.check(_lib.lib().ccb_enable_timing(self._h, int(on)), self._h)

    def timing(self, reset=False):
        """{category: (gpu milliseconds, bracketed launch groups)} measured with CUDA events."""
        ms, n = (C.c_double * 16)(), (C.c_int64 * 16)()
        _lib.check(_lib.lib().ccb_get_timing(self._h, C.byref(ms), C.byref(n), int(reset)), self._h)
        return {c: (float(ms[i]), int(n[i])) for i, c in enumerate(_lib.CATEGORIES)}

    @property
    def pcore_MC_last_id(self):
        return self.counts()[2] if self._h else 0

    @property
    def outlier_MC_last_id(self):
        return self.counts()[3] if self._h else 0

    def export_arrays(self, which):
        """(ids, uids, w, cf1, cf2, cen, pref) of a list, in list order."""
        D = self.dataset_dimensionality
        n = self.counts()[which] if self._h else 0
        ids, uids, w = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.float64)
        arrs = [np.zeros((n, D), np.float64) for _ in range(4)]
        if n:
            _lib.check(_lib.lib().ccb_export_list(self._h, which, _lib.ptr(ids), _lib.ptr(uids), _lib.ptr(w),
                                                  *[_lib.ptr(a) for a in arrs]), self._h)
        return (ids, uids, w) + tuple(arrs)

    def _objects(self, which):
        if self._lists[which] is None:
            ids, uids, w, cf1, cf2, cen, pref = self.export_arrays(which)
            out = []
            for i in range(len(ids)):
                mid = [int(ids[i])] if which == 0 else {int(ids[i])}
                out.append(Microcluster(cf1=cf1[i].copy(), cf2=cf2[i].copy(), id=mid, cumulative_weight=float(w[i]),
                                        preferred_dimension_vector=pref[i].copy(), cluster_centroids=cen[i].copy(),
                                        prev_outlier_id=int(uids[i]), points_source=self._views.points_of))
            self._lists[which] = out
        return self._lists[which]

    @property
    def pcore_MC(self):
        return self._objects(0) if self._h else []

    @property
    def outlier_MC(self):
        return self._objects(1) if self._h else []

    def _import(self, which, mcs):
        D = self.dataset_dimensionality
        n = len(mcs)
        ids = np.array([int(list(m.id)[0]) for m in mcs], np.int64)
        uids = np.array([int(m.prev_outlier_id) for m in mcs], np.int64)
        w = np.array([float(m.cumulative_weight) for m in mcs], np.float64)
        f = lambda attr: np.ascontiguousarray(
            np.array([np.asarray(getattr(m, attr), np.float64) for m in mcs], np.float64).reshape(n, D))
        cf1, cf2, cen, pref = f("CF1"), f("CF2"), f("cluster_centroids"), f("preferred_dimension_vector")
        _lib.check(_lib.lib().ccb_import_list(self._h, which, n, _lib.ptr(ids), _lib.ptr(uids), _lib.ptr(w),
                                              _lib.ptr(cf1), _lib.ptr(cf2), _lib.ptr(cen), _lib.ptr(pref)), self._h)
        self._lists[which] = None

    def import_arrays(self, which, ids, uids, w, cf1, cf2, cen, pref):
        c = lambda a, t: np.ascontiguousarray(a, dtype=t)
        _lib.check(_lib.lib().ccb_import_list(
            self._h, which, len(ids), _lib.ptr(c(ids, np.int64)), _lib.ptr(c(uids, np.int64)), _lib.ptr(c(w, np.float64)),
            _lib.ptr(c(cf1, np.float64)), _lib.ptr(c(cf2, np.float64)), _lib.ptr(c(cen, np.float64)),
            _lib.ptr(c(pref, np.float64))), self._h)
        self._lists[which] = None

    def offline_intermediates(self):
        """White-box view of the last offline phase: core flags, N(p), WN(p) as byte matrices, w_p."""
        L, h = _lib.lib(), self._h
        sizes = (C.c_int64 * 3)()
        _lib.check(L.ccb_cluster_sizes(h, C.byref(sizes)), h)
        M, D = int(sizes[2]), self.dataset_dimensionality
        core, nbr, wn = np.zeros(M, np.uint8), np.zeros((M, M), np.uint8), np.zeros((M, M), np.uint8)
        w = np.zeros((M, D), np.float64)
        _lib.check(L.ccb_export_offline(h, _lib.ptr(core), _lib.ptr(nbr), _lib.ptr(wn), _lib.ptr(w)), h)
        return core, nbr, wn, w

    def cluster_labels_for_points(self):
        """Vectorised per-row cluster index (-1 = unclustered) of the last call, from the device
        assignment array: row -> MC uid -> pcore list position -> cluster index."""
        ids, uids, *_ = self.export_arrays(0)
        lab = self.last_cluster_label if self.last_cluster_label is not None else np.full(len(ids), -1, np.int32)
        lut = {int(u): int(l) for u, l in zip(uids, lab)}
        a = self.last_assignment
        uniq, inv = np.unique(a, return_inverse=True)
        m = np.array([lut.get(int(u), -1) for u in uniq], np.int32)
        return m[inv]

    def cluster_statistics(self, quantiles=(), groups=None):
        """Per-cluster statistics of the cells of the last online_microcluster_maintenance call, computed on the GPU:
        GroupStats(count, mean, median, quantiles) (chronoclust_b200.cellstats) with one row per cluster -- row c is
        final_clusters[c] -- and a last row for the cells in no cluster.  The values are the cells as the engine read
        them, widened to float64 and, with a scaler, brought back to the input scale ((x - min_) / scale_, as
        cluster_points_D{t}.csv holds them); median and quantiles are numpy's bit for bit (see group_statistics).
        After an ingest with `columns`, the statistics cover every one of the W columns of input_dataset (arrays [.., W]):
        a clustering column as just described (under a scaler: inverse_transform(transform(x))), every other column as
        the raw value widened to float64.  After an ingest with `cofactors`, every column with a cofactor is reported in
        transformed space (asinh(x / c), then as just described).

        groups: optional integer array over the pcore list (pcore_MC order, -1 = no group) replacing the clusters of the
        offline phase; the result then has max(groups) + 2 rows.  ValueError without an offline result or `groups`;
        CCBError when no cells have been ingested since the handle's last timepoint start, reset or restore."""
        if groups is None:
            if self.last_cluster_label is None:
                raise ValueError("no offline result: run the offline phase or pass groups")
            groups, G = self.last_cluster_label, len(self.final_clusters)
        else:
            groups = np.asarray(groups)
            if groups.ndim != 1 or groups.dtype.kind not in "iu":
                raise ValueError("groups must be a 1-D integer array over the pcore list")
            if len(groups) and int(groups.min()) < -1:
                raise ValueError("groups must be >= -1")
            G = int(groups.max()) + 1 if len(groups) else 0
        if self._h is None:
            raise _lib.CCBError("no cells have been ingested")
        return cellstats.cluster_statistics(self._h, self._stats_width or self.dataset_dimensionality, groups, G, quantiles)
