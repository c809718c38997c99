"""ctypes binding of chronoclust_b200/csrc/hostio.c (host-side writer of the per-cell output table, SURVEY 8f-2, and the
host side of the arcsinh transform)."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libccb_hostio.so")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            from . import build

            build.build_hostio()
        L = C.CDLL(SO_PATH)
        L.ccbio_write_points_csv.restype = C.c_int
        L.ccbio_write_points_csv.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int64,
                                             C.c_void_p, C.c_char_p, C.c_void_p, C.c_int32]
        L.ccbio_arcsinh_host.restype = C.c_int
        L.ccbio_arcsinh_host.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                         C.c_int32]
        L.ccbio_repr.restype = C.c_int
        L.ccbio_repr.argtypes = [C.c_double, C.c_char_p]
        _LIB = L
    return _LIB


def csv_field(text):
    """A string as csv.QUOTE_MINIMAL (pandas' default) writes it."""
    text = str(text)
    if any(c in text for c in ',"\r\n'):
        return '"' + text.replace('"', '""') + '"'
    return text


def write_points_csv(path, header_names, values, label_idx, labels, id0=0, threads=0):
    """id,label,values... rows exactly as pandas.DataFrame({'id':..,'cluster_id':..,<markers>}).to_csv(index=False)
    writes them (float64 columns: repr(float); NaN: empty field), formatted on every host core.

    values: [n, D] float64 (any row stride, unit column stride); label_idx: [n] int32 into `labels` (list of str)."""
    values = np.asarray(values, np.float64)
    if values.ndim != 2 or (values.shape[1] > 1 and values.strides[1] != 8):
        values = np.ascontiguousarray(values, np.float64)
    if values.strides[0] % 8:
        values = np.ascontiguousarray(values, np.float64)
    label_idx = np.ascontiguousarray(label_idx, np.int32)
    n, d = values.shape
    if label_idx.shape != (n,):
        raise ValueError("one label index per row")
    fields = [csv_field(s).encode() for s in labels]
    pool = b"".join(fields)
    off = np.zeros(len(fields) + 1, np.int64)
    np.cumsum([len(f) for f in fields], out=off[1:])
    header = (",".join(csv_field(h) for h in header_names) + "\n").encode()
    rc = lib().ccbio_write_points_csv(os.fsencode(path), header, n, d, values.ctypes.data, values.strides[0] // 8 if n else d,
                                      id0, label_idx.ctypes.data, pool, off.ctypes.data, threads)
    if rc != 0:
        raise OSError(rc, os.strerror(rc), str(path))


def arcsinh_host(x, cofactor, threads=0):
    """ccbio_arcsinh_host: [n, d] float64 rows of the float32 / float64 rows `x` (numpy, unit column stride, any row stride),
    every column with cofactor[c] != 0 as ccb_asinh(x / cofactor[c]) -- the device's values bit for bit.  `cofactor`:
    float64 [d], already checked (scaling.cofactor_vector)."""
    x = np.asarray(x)
    if x.dtype not in (np.float32, np.float64):
        x = x.astype(np.float64)
    if x.ndim != 2:
        raise ValueError("arcsinh takes 2-D rows")
    isz = x.itemsize
    if (x.shape[1] > 1 and x.strides[1] != isz) or (x.shape[0] > 1 and (x.strides[0] % isz or
                                                                         x.strides[0] < x.shape[1] * isz)):
        x = np.ascontiguousarray(x)
    n, d = x.shape
    ld = x.strides[0] // isz if n > 1 else d
    cof = np.ascontiguousarray(cofactor, np.float64)
    if cof.shape != (d,):
        raise ValueError(f"{cof.size} cofactors for {d} columns")
    out = np.empty((n, d), np.float64)
    rc = lib().ccbio_arcsinh_host(x.ctypes.data, 1 if x.dtype == np.float32 else 0, n, ld, d, cof.ctypes.data,
                                  out.ctypes.data, threads)
    if rc != 0:
        raise OSError(rc, os.strerror(rc))
    return out
