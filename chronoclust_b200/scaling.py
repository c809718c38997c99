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

It also holds the arcsinh transform of cytometry intensities (`arcsinh`, `cofactor_vector`): the values
`HDDStream.online_microcluster_maintenance(cofactors=)` clusters, computed on the host or on the device with one
definition that gives the same bits on both (csrc/asinh.h).
"""
import numbers
import sys

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


# ---- arcsinh transform of cytometry intensities ---------------------------------------------------------------------------
def cofactor_vector(cofactors, width):
    """The arcsinh cofactors of rows `width` wide as a float64 vector: a scalar applies to every column, a sequence gives
    one cofactor per column.  0 leaves a column linear; any other cofactor must be positive and finite.  ValueError for a
    sequence of another length, an entry that is not a real number, or one that is negative, NaN or infinite."""
    if isinstance(cofactors, (numbers.Real, np.floating, np.integer)) and not isinstance(cofactors, (bool, np.bool_)):
        entries = [cofactors] * width
    else:
        try:
            entries = list(cofactors)
        except TypeError:
            raise ValueError("cofactors must be a number or a sequence of numbers") from None
        if len(entries) != width:
            raise ValueError(f"{len(entries)} cofactors for {width} columns")
    for c in entries:
        if isinstance(c, (bool, np.bool_)) or not isinstance(c, (numbers.Real, np.floating, np.integer)):
            raise ValueError(f"cofactor {c!r} is not a number")
        if not 0.0 <= float(c) < float("inf"):
            raise ValueError(f"cofactor {c!r}: a cofactor is 0 (linear) or positive and finite")
    return np.array(entries, np.float64).reshape(width)


def arcsinh(x, cofactors):
    """asinh(x / c) per column of the 2-D float32 / float64 rows `x`, as the engine computes it: every value is widened to
    float64 first (exact), divided by its column's cofactor c (one IEEE division) and transformed with csrc/asinh.h's
    restatement of fdlibm's asinh; columns with c == 0 are only widened.  Returns float64 rows [N, D]: a CUDA tensor for a
    CUDA tensor (ccb_arcsinh, after the work queued on the current stream; asynchronous like any torch operation), a numpy
    array otherwise (the multithreaded host library).  Both give the same bits.

    `cofactors`: see cofactor_vector.  Note that np.arcsinh(x32 / 5) is not this function: for float32 input numpy divides
    and transforms in float32, and even in float64 numpy's arcsinh and the C library's differ from this one (and from
    each other) in the last bits."""
    torch = sys.modules.get("torch")
    if torch is not None and isinstance(x, torch.Tensor) and x.is_cuda:
        from . import _lib

        code = {torch.float64: _lib.DTYPE_F64, torch.float32: _lib.DTYPE_F32}.get(x.dtype)
        if code is None:
            x, code = x.to(torch.float64), _lib.DTYPE_F64
        if x.dim() != 2:
            raise ValueError("arcsinh takes 2-D rows")
        cof = cofactor_vector(cofactors, x.shape[1])
        if x.shape[1] > 1 and x.stride(1) != 1 or x.shape[0] > 1 and x.stride(0) < x.shape[1]:
            x = x.contiguous()
        n, d = x.shape
        out = torch.empty((n, d), dtype=torch.float64, device=x.device)
        if n:
            ld = x.stride(0) if n > 1 else d
            stream = torch.cuda.current_stream(x.device)
            _lib.check(_lib.lib().ccb_arcsinh(x.device.index, stream.cuda_stream, x.data_ptr(), code, n, ld, d,
                                              cof.ctypes.data, out.data_ptr()))
        return out
    if torch is not None and isinstance(x, torch.Tensor):
        x = x.detach().numpy()
    x = np.asarray(x)
    if x.ndim != 2:
        raise ValueError("arcsinh takes 2-D rows")
    from . import _hostio

    return _hostio.arcsinh_host(x, cofactor_vector(cofactors, x.shape[1]))
