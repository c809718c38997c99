"""chronoclust_b200.app.run -- drop-in for chronoclust.app.run (reference app.py:32-226).

Same keyword parameters and the same output files: result.csv, cluster_points_D{t}.csv, parameters.csv,
logs/Chronoclust.log, program_images/{hddstream, tracking_by_lineage, tracking_by_historical_association}.  What happens
between the input files and those outputs is organised for a GPU in the middle:

  inputs    every CSV is parsed ONCE, all files concurrently on a thread pool (pandas' C parser releases the GIL; it is the
            reference's own parser, so the cells are the reference's doubles).  The reference parses each file twice
            (Scaler.__init__, then the timepoint loop; scaler.py:27-36, app.py:170).
  scaling   the joint min-max fit streams the parsed arrays through MinMaxScaler.partial_fit; the transform runs on the
            device behind the host -> device copy (ccb_ingest_scaled; SURVEY 8f-3), bit-identical to sklearn's.
  hot path  HDDStream.online_microcluster_maintenance -> CUDA (online + offline phase).
  tracking  lineage / historical association on the host (north_star), the association and gating scans on the device
            (ccb_assoc_nearest[2]; SURVEY 8f-1, 8f-4).
  outputs   result.csv rows are formatted as the reference formats them; the per-cell table is assembled from the device's
            row -> microcluster assignment (no per-cell Python objects) and written by the native multi-threaded writer
            (csrc/hostio.c, byte-identical to DataFrame.to_csv) on a background thread while the next timepoint runs
            (SURVEY 8f-2).
"""
import csv
import logging
import os
import pickle
import threading
from concurrent.futures import ThreadPoolExecutor
from decimal import ROUND_HALF_UP, Decimal

import numpy as np
import pandas as pd

from . import _hostio, cellstats
from .hddstream import HDDStream
from .objects import Cluster
from .scaling import Scaler, cofactor_vector
from .tracking import TrackByHistoricalAssociation, TrackByLineage

STATE_FILES = ("hddstream", "tracking_by_historical_association", "tracking_by_lineage")
PARAM_NAMES = ("beta", "delta", "epsilon", "lambda", "k", "mu", "pi", "omicron", "upsilon")
# a gating argmin of the device is accepted when the runner-up is further away than this (relative); closer calls are
# re-evaluated with the reference's own Python expression (see ccb_assoc_nearest2 in include/chronoclust_b200.h)
GATE_GUARD = 1e-9


# ---- inputs ---------------------------------------------------------------------------------------------------------------
class _Timepoints(object):
    """The input files, parsed once each and concurrently; `cells(t)` blocks until file t is there."""

    def __init__(self, files):
        self.files = list(files)
        workers = max(1, min(len(self.files), os.cpu_count() or 1))
        self._pool = ThreadPoolExecutor(max_workers=workers, thread_name_prefix="ccb-read")
        self._jobs = [self._pool.submit(self._parse, f) for f in self.files]

    @staticmethod
    def _parse(path):
        frame = pd.read_csv(path, header=0, sep=',')
        return [str(c) for c in frame.columns], frame.to_numpy()

    def attributes(self):
        """Marker names = the header line of the first file (app.py:490-492)."""
        return self._jobs[0].result()[0]

    def cells(self, t):
        return self._jobs[t].result()[1]

    def release(self, t):
        self._jobs[t] = None

    def close(self):
        self._pool.shutdown(wait=False)


def _fit_joint_scaler(timepoints, wanted, cols=None, cofactors=None):
    """MinMaxScaler over all timepoints jointly (scaler.py:27-36), fed one parsed array at a time -- on the clustering
    columns `cols` only when given (the fit is column-wise: the vectors are those of a fit on files holding only them),
    and on their arcsinh-transformed values with `cofactors` (by file column; what the engine then scales)."""
    scaler = Scaler()
    for t in wanted:
        cells = timepoints.cells(t)
        cells = cells if cols is None else cells[:, cols]
        if cofactors is not None:
            cells = _hostio.arcsinh_host(np.asarray(cells, np.float64), cofactors if cols is None else cofactors[cols])
        scaler.scaler.partial_fit(cells)
    return scaler


def clustering_columns(attributes, clustering_markers):
    """Column indices of `clustering_markers` (names from the first file's header, in the order given), or None for every
    column.  ValueError for an unknown or repeated name, or an empty list."""
    if clustering_markers is None:
        return None
    names = [str(m) for m in clustering_markers]
    if not names:
        raise ValueError("clustering_markers is empty")
    unknown = [m for m in names if m not in attributes]
    if unknown:
        raise ValueError(f"clustering_markers not in the header of the first file: {unknown}")
    if len(set(names)) != len(names):
        raise ValueError(f"clustering_markers repeats a name: {names}")
    return [attributes.index(m) for m in names]


def arcsinh_cofactors_by_column(attributes, cols, arcsinh_cofactors):
    """app.run(arcsinh_cofactors=) as one float64 cofactor per column of the files (0: linear), or None.  A number applies
    to every clustering marker (the columns `cols`, or every column); a dict {marker name: cofactor} to the columns it
    names, clustering or not.  ValueError for an unknown name or a cofactor that is not 0 or positive and finite."""
    if arcsinh_cofactors is None:
        return None
    W = len(attributes)
    if isinstance(arcsinh_cofactors, dict):
        unknown = [m for m in arcsinh_cofactors if str(m) not in attributes]
        if unknown:
            raise ValueError(f"arcsinh_cofactors names markers not in the header of the first file: {unknown}")
        named = {attributes.index(str(m)): c for m, c in arcsinh_cofactors.items()}
        try:
            return cofactor_vector([named.get(c, 0.0) for c in range(W)], W)
        except ValueError as exc:
            raise ValueError(f"arcsinh_cofactors: {exc}") from None
    try:
        value = cofactor_vector(arcsinh_cofactors, 1)[0]
    except ValueError as exc:
        raise ValueError(f"arcsinh_cofactors must be a number or a dict of marker names to numbers: {exc}") from None
    out = np.zeros(W, np.float64)
    out[slice(None) if cols is None else cols] = value
    return out


# ---- outputs --------------------------------------------------------------------------------------------------------------
class _PointsWriter(object):
    """cluster_points_D{t}.csv on a background thread; at most one file in flight so that memory stays bounded."""

    def __init__(self):
        self._thread = None
        self._error = None

    def _job(self, path, header, raw, scaler, cols, cofactors, label_idx, labels):
        try:
            _hostio.write_points_csv(path, header, points_values(raw, scaler, cols, cofactors), label_idx, labels)
        except BaseException as exc:  # surfaced by the next submit / by close
            self._error = exc

    def wait(self):
        if self._thread is not None:
            self._thread.join()
            self._thread = None
        if self._error is not None:
            err, self._error = self._error, None
            raise err

    def submit(self, *args):
        self.wait()
        self._thread = threading.Thread(target=self._job, args=args, name="ccb-write")
        self._thread.start()

    close = wait


def output_headers(attributes, markers, gating):
    """Header rows of result.csv (centroid columns: the clustering `markers`), cluster_points_D{t}.csv and
    cluster_statistics.csv (every column of the files, `attributes`)."""
    result = ['timepoint', 'cumulative_size', 'pcore_ids', 'pref_dimensions'] + markers + \
             ['tracking_by_lineage', 'tracking_by_association'] + (['predicted_label'] if gating else [])
    stats = ['timepoint', 'tracking_by_lineage', 'cell_count'] + [f'median_{a}' for a in attributes] + \
            [f'mean_{a}' for a in attributes]
    return result, ['id', 'cluster_id'] + attributes, stats


def points_values(raw, scaler, cols=None, cofactors=None):
    """The values of cluster_points_D{t}.csv for the parsed cells `raw`: a column with an arcsinh cofactor (`cofactors`, by
    column; 0 = none) holds x = asinh(raw / c) (scaling.arcsinh), every other column x = the parsed value; then, with a
    scaler, the clustering columns (`cols`, or every column) hold inverse_transform(transform(x)), what the reference
    writes (app.py:175, 299-301)."""
    if cofactors is not None:
        raw = _hostio.arcsinh_host(raw, cofactors)
    if scaler is None:
        return raw
    if cols is None:
        return scaler.reverse_scaling(scaler.scale_data(raw))
    values = np.array(raw, np.float64)
    values[:, cols] = scaler.reverse_scaling(scaler.scale_data(raw[:, cols]))
    return values


def _pcore_labels(hddstream, clusters):
    """Lineage label of every pcore MC -- its index into `labels`, in pcore list order, 0 = 'None' -- and the MCs' uids:
    the one mapping behind both the per-cell table and cluster_statistics.csv.  A label shared by several clusters is
    one entry of `labels`."""
    labels = ["None"]
    index_of = {}
    label_of_pcore = {}
    for cluster in clusters:
        idx = index_of.setdefault(str(cluster.id), len(labels))
        if idx == len(labels):
            labels.append(str(cluster.id))
        for pid in cluster.pcore_ids:
            label_of_pcore[int(pid)] = idx
    ids, uids = hddstream.export_arrays(0)[:2]
    return np.array([label_of_pcore.get(pid, 0) for pid in ids.tolist()], np.int32), uids, labels


def _cell_labels(hddstream, clusters):
    """Per input row the index of its lineage label (app.py:263-360 without the per-cell objects): row -> uid of the MC that
    absorbed it (device array) -> pcore id -> the cluster holding that pcore id; everything else is 'None'."""
    label_idx, uids, labels = _pcore_labels(hddstream, clusters)
    assign = hddstream.last_assignment
    lut = np.zeros(int(max(int(assign.max(initial=0)), int(uids.max(initial=0)))) + 1, np.int32)
    for uid, idx in zip(uids.tolist(), label_idx.tolist()):
        lut[uid] = idx
    return lut[assign], labels


def _statistics_rows(timepoint, hddstream, clusters):
    """cluster_statistics.csv rows of a timepoint: per lineage label the cells the per-cell table gives that label, their
    count and per-marker medians and means, computed on the device; then the 'None' row."""
    label_idx, _, labels = _pcore_labels(hddstream, clusters)
    return cellstats.statistics_rows(timepoint, labels, hddstream.cluster_statistics(groups=label_idx - 1))


def _result_rows(timepoint, clusters, scaler, gate_labels):
    """One result.csv row per cluster, formatted like app.py:229-260."""
    rows = []
    for n, cluster in enumerate(clusters):
        centre = np.asarray(cluster.centroid, np.float64)
        if scaler is not None:
            centre = scaler.reverse_scaling([centre])[0]
        row = [timepoint, cluster.cumulative_weight, cluster.get_pcore_ids_as_str(),
               cluster.get_preferred_dimensions_as_str()]
        row.extend(np.round(centre, 5).tolist())
        row.append(cluster.id)
        row.append(cluster.get_historical_associates_as_str())
        if gate_labels is not None:
            row.append(gate_labels[n])
        rows.append(row)
    return rows


# ---- gating (SURVEY 8f-4) --------------------------------------------------------------------------------------------------
def _read_gates(path, attributes):
    """{day: {centroid tuple: population name}} in file order (app.py:136-145)."""
    gates = {}
    if path is None:
        return gates
    frame = pd.read_csv(path)
    for _, gate in frame.iterrows():
        gates.setdefault(int(gate['Day']), {})[tuple(gate[attributes].values)] = gate['PopName']
    return gates


def transform_gates(gates, cofactors):
    """The gating centroids of _read_gates (in the files' units) in the space the engine clusters: every marker with
    cofactor c != 0 (`cofactors`, one per clustering marker) as asinh(x / c) (scaling.arcsinh)."""
    out = {}
    for day, by_centroid in gates.items():
        cen = np.array([list(c) for c in by_centroid.keys()], np.float64).reshape(len(by_centroid), len(cofactors))
        cen = _hostio.arcsinh_host(cen, cofactors)
        out[day] = {tuple(row): name for row, name in zip(cen.tolist(), by_centroid.values())}
    return out


def find_closest_gating(gating_dict, cluster, scaler):
    """The reference's scan for ONE cluster (app.py:497-512), its expression unchanged: the tie-break authority."""
    best, best_label = None, None
    for centroid, label in gating_dict.items():
        point = scaler.scale_data([centroid])[0].tolist() if scaler else centroid
        d = cluster.get_projected_dist_to_point(np.array(point))
        if best is None or d < best:
            best, best_label = d, label
    return best_label


def closest_gates(gating_dict, clusters, scaler, k, device=0):
    """The gating label of every cluster of a timepoint: one (clusters x gates) scan on the device.  A cluster whose two
    nearest gates are closer together than GATE_GUARD (relative) is re-evaluated with find_closest_gating."""
    if not clusters:
        return []
    names = list(gating_dict.values())
    gates = np.array([list(c) for c in gating_dict.keys()], np.float64)
    if scaler is not None:
        gates = np.asarray(scaler.scale_data(gates), np.float64)
    D = gates.shape[1]
    cen = np.ascontiguousarray([np.asarray(c.centroid, np.float64) for c in clusters]).reshape(len(clusters), D)
    pref = np.ascontiguousarray([np.asarray(c.preferred_dimensions, np.float64) for c in clusters]).reshape(len(clusters), D)
    scan = _device_gate_scan(cen, pref, gates, float(k), device)
    out = []
    for n, cluster in enumerate(clusters):
        sure = scan is not None and (scan[2][n] - scan[1][n]) > GATE_GUARD * max(scan[2][n], 1e-300)
        out.append(names[int(scan[0][n])] if sure else find_closest_gating(gating_dict, cluster, scaler))
    return out


def _device_gate_scan(cen, pref, gates, k, device):
    """(best, dist, dist2) from ccb_assoc_nearest2, or None when the preference vectors are not {1, k}-valued or no CUDA
    device can be reached (the caller then uses the reference expression for every cluster)."""
    if not np.isin(pref, (1.0, k)).all():
        return None
    try:
        import torch

        if not torch.cuda.is_available():
            return None
    except ImportError:
        return None
    from . import _lib

    Q, D = cen.shape
    mask = np.zeros(Q, np.uint64)
    if k != 1.0:
        mask = ((pref == k) * (np.uint64(1) << np.arange(D, dtype=np.uint64))).sum(axis=1).astype(np.uint64)
    dev = torch.device("cuda", device)
    tc = torch.from_numpy(np.ascontiguousarray(cen)).to(dev)
    tg = torch.from_numpy(np.ascontiguousarray(gates)).to(dev)
    tm = torch.from_numpy(mask.view(np.int64)).to(dev)
    best = torch.empty(Q, dtype=torch.int32, device=dev)
    d1 = torch.empty(Q, dtype=torch.float64, device=dev)
    d2 = torch.empty(Q, dtype=torch.float64, device=dev)
    _lib.check(_lib.lib().ccb_assoc_nearest2(device, None, tc.data_ptr(), tm.data_ptr(), Q, tg.data_ptr(), len(gates), D, k,
                                             best.data_ptr(), d1.data_ptr(), d2.data_ptr()))
    torch.cuda.synchronize(dev)
    return best.cpu().numpy(), d1.cpu().numpy(), d2.cpu().numpy()


# ---- program state (app.py:402-465) ------------------------------------------------------------------------------------------
def save_program_state(hddstream, output_dir, tracker_by_association, tracker_by_lineage):
    folder = os.path.join(output_dir, "program_images")
    os.makedirs(folder, exist_ok=True)
    for name, obj in zip(STATE_FILES, (hddstream, tracker_by_association, tracker_by_lineage)):
        with open(os.path.join(folder, name), "wb") as f:
            pickle.dump(obj, f)


def restore_program_state(program_state_dir, device=0):
    HDDStream.restore_device = device
    state = []
    for name in STATE_FILES:
        with open(os.path.join(program_state_dir, name), "rb") as f:
            state.append(pickle.load(f))
    return tuple(state)


def setup_logger(log_dir):
    os.makedirs(log_dir, exist_ok=True)
    logging.basicConfig(filename=os.path.join(log_dir, "Chronoclust.log"),
                        format='%(asctime)s [%(levelname)-8s] %(message)s')
    logger = logging.getLogger()  # the root logger, as in the reference (app.py:468-479)
    logger.setLevel(logging.INFO)
    return logger


# ---- entry point ------------------------------------------------------------------------------------------------------------
def run(data, output_directory, gating_centroid_file=None, normalise_data=True, restore_program=False,
        param_beta=0.8, param_delta=0.0, param_epsilon=0.03, param_lambda=0, param_k=1,
        param_mu=0.001, param_pi=0, param_omicron=0.0, param_upsilon=1, device=0, cluster_statistics=False,
        clustering_markers=None, arcsinh_cofactors=None):
    """Run ChronoClust on a list of per-timepoint CSV files (in time order).  See the reference's app.run for the meaning of
    every parameter.  Additions: `device` (CUDA ordinal); `cluster_statistics` -- also write cluster_statistics.csv, per
    timepoint and lineage label the number of cells and their per-marker medians and means (the cells and values of
    cluster_points_D{t}.csv), computed on the device, then the same for the cells in no cluster ('None');
    `clustering_markers` -- names of the markers to cluster on, from the first file's header, in the order given (default:
    every column).  The scaler is fitted on them, the gating file is read on them and result.csv's centroid columns are
    them; cluster_points_D{t}.csv and cluster_statistics.csv still cover every column of the files, the others holding
    the parsed values.  An unknown or repeated name raises ValueError before any clustering.
    `arcsinh_cofactors` -- cluster asinh(x / c) of cytometry intensities (scaling.arcsinh; typically c = 5 for mass and
    around 150 for flow cytometry): a number applies to every clustering marker, a dict {marker name: cofactor} to the
    markers it names, clustering or not (the others stay linear; 0 also means linear).  The transform runs on the device
    as the cells are staged, the scaler is fitted on the transformed values, and the gating file keeps the files' units
    (its centroids are transformed when read).  result.csv, cluster_points_D{t}.csv and cluster_statistics.csv then
    hold transformed columns in transformed space; the cofactors are logged.  An unknown name or a cofactor that is not
    0 or positive and finite raises ValueError before any clustering."""
    logger = setup_logger(os.path.join(output_directory, "logs"))
    logger.info("ChronoClust (B200 hot path) starts on cuda:%d with %d timepoint file(s)", device, len(data))
    values = (param_beta, param_delta, param_epsilon, param_lambda, param_k, param_mu, param_pi, param_omicron,
              param_upsilon)
    config = dict(zip(PARAM_NAMES, values))

    state_dir = os.path.join(output_directory, "program_images")
    resumed = restore_program and os.path.isdir(state_dir)
    if resumed:
        logger.info("Resuming from the program state in %s", state_dir)
        hddstream, by_association, by_lineage = restore_program_state(state_dir, device)
        hddstream.set_logger(logger)
        hddstream.set_config(config)
    else:
        if restore_program:
            logger.warning("No program_images under %s: starting from scratch", output_directory)
        hddstream = HDDStream(config, logger, device=device)
        by_association, by_lineage = TrackByHistoricalAssociation(), TrackByLineage()
    by_association.device = device

    timepoints = _Timepoints(data)
    writer = _PointsWriter()
    try:
        attributes = timepoints.attributes()
        cols = clustering_columns(attributes, clustering_markers)
        markers = attributes if cols is None else [attributes[c] for c in cols]
        cofactors = arcsinh_cofactors_by_column(attributes, cols, arcsinh_cofactors)
        gates = _read_gates(gating_centroid_file, markers)
        if cofactors is not None:
            logger.info("arcsinh cofactors (0: linear): %s",
                        ", ".join(f"{a}={c!r}" for a, c in zip(attributes, cofactors.tolist())))
            gates = transform_gates(gates, cofactors if cols is None else cofactors[cols])
        header, points_header, stats_header = output_headers(attributes, markers, gating_centroid_file)
        result_path = os.path.join(output_directory, "result.csv")
        with open(result_path, 'w') as f:
            csv.writer(f).writerow(header)
        stats_path = os.path.join(output_directory, "cluster_statistics.csv")
        if cluster_statistics:
            with open(stats_path, 'w') as f:
                csv.writer(f).writerow(stats_header)

        scaler = None
        if normalise_data:
            logger.info("Fitting the joint min-max scaler over all timepoints")
            scaler = _fit_joint_scaler(timepoints, range(len(data)), cols, cofactors)

        for timepoint in range(len(data)):
            if resumed and hddstream.last_data_timestamp >= timepoint:
                timepoints.release(timepoint)
                continue
            raw = np.ascontiguousarray(timepoints.cells(timepoint), dtype=np.float64)
            logger.info("Timepoint %d: %d cells x %d markers", timepoint, raw.shape[0], raw.shape[1])

            # ---- the hot path: online + offline clustering on the GPU (the min-max transform rides along on the device)
            hddstream.online_microcluster_maintenance(raw, timepoint, scaler=scaler.scaler if scaler else None,
                                                      columns=cols, cofactors=cofactors)

            pcore_by_id = {mc.id[0]: mc for mc in hddstream.pcore_MC}
            for found in hddstream.final_clusters:
                size = Decimal(str(found.cumulative_weight)).quantize(Decimal('1.1'), rounding=ROUND_HALF_UP)
                cluster = Cluster(list(found.id), found.cluster_centroids, size, found.preferred_dimension_vector)
                cluster.add_pcore_objects(pcore_by_id)
                by_lineage.add_new_child_cluster(cluster)
            by_lineage.calculate_ids()
            by_association.set_current_clusters(by_lineage.child_clusters)
            by_association.track_cluster_history()

            clusters = by_association.current_clusters
            gates_now = gates.get(timepoint)
            gate_labels = closest_gates(gates_now, clusters, scaler, hddstream.k, device) if gates_now else None
            with open(result_path, 'a') as f:
                csv.writer(f).writerows(_result_rows(timepoint, clusters, scaler, gate_labels))

            if cluster_statistics:
                with open(stats_path, 'a') as f:
                    csv.writer(f).writerows(_statistics_rows(timepoint, hddstream, by_lineage.child_clusters))
            label_idx, labels = _cell_labels(hddstream, by_lineage.child_clusters)
            writer.submit(os.path.join(output_directory, f"cluster_points_D{timepoint}.csv"),
                          points_header, raw, scaler, cols, cofactors, label_idx, labels)
            timepoints.release(timepoint)

            by_lineage.transfer_child_to_parent()
            by_association.transfer_current_to_previous()
            save_program_state(hddstream, output_directory, by_association, by_lineage)
            logger.info("Timepoint %d done: %d clusters", timepoint, len(clusters))
        writer.close()
    finally:
        timepoints.close()
        try:
            writer.close()
        except Exception:
            logger.exception("writing the per-cell table failed")
            raise

    with open(os.path.join(output_directory, "parameters.csv"), 'w') as f:
        w = csv.DictWriter(f, config.keys())
        w.writeheader()
        w.writerow(config)
    logger.info("ChronoClust finished")
