"""Joint min-max normalisation of all timepoints (host component; north_star keeps scaling on the host).

Drop-in for the reference's `Scaler` (scaling/scaler.py:11-53): same constructor and method names, and the same
sklearn `MinMaxScaler` underneath, so the scaled fp64 values that feed the bit-exact path are identical.  Differences
in HOW it gets there:

* the fit streams the timepoint files one at a time through `partial_fit` (running column minima / maxima are exact, so
  the fitted `scale_` / `min_` equal those of one fit over the concatenation, bit for bit) instead of holding every cell
  of every timepoint in one Python list;
* `device_vectors()` hands the fitted `(scale_, min_)` to `HDDStream.online_microcluster_maintenance(..., scaler=)`, which
  applies the transform on the device behind the host -> device copy (`ccb_ingest_ex`, SURVEY 8f-3);
* `fit_columns_on_device` computes a file's column minima / maxima with `ccb_colminmax_ex` (np.nanmin / np.nanmax
  semantics, float32 or float64) for callers whose data already lives on the GPU.
"""
import numpy as np
import pandas as pd
from sklearn.preprocessing import MinMaxScaler


def _read_cells(path):
    return pd.read_csv(path, header=0, sep=',').to_numpy()


class Scaler(object):
    def __init__(self, data_files=None):
        self.scaler = MinMaxScaler()
        self.input_data = []
        self.files = list(data_files) if data_files is not None else []
        for path in self.files:
            self.scaler.partial_fit(_read_cells(path))

    # ---- reference API ---------------------------------------------------------------------------------------------
    def fit_scaler(self, data):
        """Refit on an in-memory array (scaler.py:38-41); the array is remembered as the reference does."""
        self.scaler = MinMaxScaler().fit(data)
        self.set_input_data(data)

    def scale_data(self, data):
        return self.scaler.transform(data)

    def reverse_scaling(self, data):
        return self.scaler.inverse_transform(data)

    def set_input_data(self, data):
        self.input_data = data

    def get_input_data(self):
        """The cells the scaler was set up with.  After a file-streamed fit they are re-read on demand."""
        if len(self.input_data) == 0 and self.files:
            self.input_data = np.concatenate([_read_cells(p) for p in self.files], axis=0)
        return self.input_data

    # ---- device side (SURVEY 8f-3) -----------------------------------------------------------------------------------
    def device_vectors(self):
        """(scale_, min_) as contiguous fp64 vectors for the scaled ingest: x * scale_ + min_, two roundings."""
        return (np.ascontiguousarray(self.scaler.scale_, np.float64), np.ascontiguousarray(self.scaler.min_, np.float64))

    @staticmethod
    def fit_columns_on_device(x_dev, device=0):
        """Column minima / maxima of a CUDA tensor [N, D] (float32 or float64, rows with unit column stride and any row
        stride) ignoring NaN -- the reductions of MinMaxScaler.partial_fit -- through ccb_colminmax_ex, after the work
        queued on the current stream.  float32 values are widened to float64 first (exact).  Returns two fp64 numpy
        vectors."""
        import torch

        from . import _lib

        code = {torch.float64: _lib.DTYPE_F64, torch.float32: _lib.DTYPE_F32}.get(x_dev.dtype)
        if code is None or x_dev.dim() != 2:
            raise ValueError("fit_columns_on_device takes a 2-D float32 or float64 CUDA tensor")
        if x_dev.stride(1) != 1:
            x_dev = x_dev.contiguous()
        n, d = x_dev.shape
        ld = x_dev.stride(0) if n > 1 else d
        mn = torch.empty(d, dtype=torch.float64, device=x_dev.device)
        mx = torch.empty(d, dtype=torch.float64, device=x_dev.device)
        stream = torch.cuda.current_stream(x_dev.device)
        _lib.check(_lib.lib().ccb_colminmax_ex(device, stream.cuda_stream, x_dev.data_ptr(), code, n, ld, d,
                                               mn.data_ptr(), mx.data_ptr()))
        stream.synchronize()
        return mn.cpu().numpy(), mx.cpu().numpy()
