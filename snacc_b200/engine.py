"""ctypes binding of libsnacc_b200.so -- the only way the package computes compressed sizes.

There is deliberately no CPU fallback: if the CUDA library is missing or no GPU is visible the
calls raise (north_star: "no CPU fallback").
"""
import ctypes
import os

import numpy as np

from . import _build

CODEC_IDS = {"lz4": 0, "gzip": 1, "zlib": 2, "bzip2": 3}
GETSIZEOF_BIAS = 33       # sys.getsizeof(b"") on 64-bit CPython 3 (reference pairwise_ncd.py:90)

_STATUS = {-1: "CUDA error", -2: "bad argument", -3: "empty sequence", -4: "codec not supported on the GPU path",
           -5: "nothing uploaded", -6: "stream too large"}

_lib = None


class SnaccGpuError(RuntimeError):
    pass


def load_library():
    """Load libsnacc_b200.so; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_build.LIB_PATH):
        raise SnaccGpuError(f"{_build.LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU fallback)")
    lib = ctypes.CDLL(_build.LIB_PATH)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    lib.snacc_version.restype = ctypes.c_int
    lib.snacc_last_error.restype = ctypes.c_char_p
    lib.snacc_last_error.argtypes = [vp]
    lib.snacc_ctx_create.argtypes = [ctypes.c_int, ctypes.POINTER(vp)]
    lib.snacc_ctx_destroy.argtypes = [vp]
    lib.snacc_ctx_destroy.restype = None
    lib.snacc_upload.argtypes = [vp, vp, vp, i32, vp, i64, ctypes.c_int]
    lib.snacc_upload_device.argtypes = [vp, vp, vp, i32, vp, i64, ctypes.c_int]
    lib.snacc_download_sequence.argtypes = [vp, i32, vp]
    lib.snacc_single_sizes.argtypes = [vp, ctypes.c_int, vp, i64, vp]
    lib.snacc_pair_sizes.argtypes = [vp, ctypes.c_int, vp, vp, i64, vp]
    lib.snacc_tile_sizes.argtypes = [vp, ctypes.c_int, i32, i32, i32, i32, vp]
    lib.snacc_ncd.argtypes = [vp, vp, vp, i32, ctypes.c_int, i32, vp]
    lib.snacc_upgma.argtypes = [vp, vp, i32, ctypes.c_int, vp]
    lib.snacc_last_kernel_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i64)]
    lib.snacc_set_option.argtypes = [vp, ctypes.c_char_p, i64]
    lib.snacc_get_stat.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(ctypes.c_double)]
    lib.snacc_prefix_record_bytes.restype = i64
    lib.snacc_prefix_record_bytes.argtypes = [vp, ctypes.c_int]
    lib.snacc_export_prefix.argtypes = [vp, ctypes.c_int, vp, i64, vp]
    lib.snacc_import_prefix.argtypes = [vp, ctypes.c_int, vp, i64, vp]
    lib.snacc_csv_write.restype = ctypes.c_int
    lib.snacc_csv_write.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_char_p), vp, i64, vp, ctypes.c_int]
    lib.snacc_fasta_parse.restype = i64
    lib.snacc_fasta_parse.argtypes = [vp, ctypes.c_uint64, vp, ctypes.POINTER(ctypes.c_uint64), vp, i64]
    _lib = lib
    return lib


class Engine:
    """One GPU context: upload a corpus once, then ask for single / pair / tile sizes."""

    def __init__(self, device=0):
        self._lib = load_library()
        h = ctypes.c_void_p()
        rc = self._lib.snacc_ctx_create(int(device), ctypes.byref(h))
        if rc != 0 or not h:
            raise SnaccGpuError(f"snacc_ctx_create(device={device}) failed: {_STATUS.get(rc, rc)} "
                                "(a CUDA device is required; there is no CPU fallback)")
        self._h = h
        self.device = int(device)
        self.n_seqs = 0
        self.lengths = None

    def close(self):
        if getattr(self, "_h", None):
            self._lib.snacc_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc):
        if rc != 0:
            msg = self._lib.snacc_last_error(self._h).decode(errors="replace")
            if rc == -3:
                raise ValueError(msg or "No sequence extracted.")
            if rc == -4:
                raise KeyError(msg or "codec not supported on the GPU path")
            raise SnaccGpuError(f"{_STATUS.get(rc, rc)}: {msg}")

    # ---- corpus ----
    def upload(self, data, seq_offsets, rec_offsets=None, reverse_complement=False):
        """data: uint8 array (all sequences concatenated); seq_offsets: n+1 offsets; rec_offsets: FASTA
        record offsets (needed for per-record reverse complement)."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        so = np.ascontiguousarray(seq_offsets, dtype=np.uint64)
        ro = None if rec_offsets is None else np.ascontiguousarray(rec_offsets, dtype=np.uint64)
        self._check(self._lib.snacc_upload(self._h, data.ctypes.data, so.ctypes.data, so.size - 1,
                                           None if ro is None else ro.ctypes.data,
                                           0 if ro is None else ro.size - 1, int(bool(reverse_complement))))
        self.n_seqs = so.size - 1
        self.lengths = np.diff(so.astype(np.int64))

    def upload_device(self, device_ptr, seq_offsets, rec_offsets=None, reverse_complement=False):
        """Same as upload() but the bytes already sit on this context's device (e.g. after an NCCL
        broadcast into a torch tensor: pass tensor.data_ptr())."""
        so = np.ascontiguousarray(seq_offsets, dtype=np.uint64)
        ro = None if rec_offsets is None else np.ascontiguousarray(rec_offsets, dtype=np.uint64)
        self._check(self._lib.snacc_upload_device(self._h, ctypes.c_void_p(int(device_ptr)), so.ctypes.data,
                                                  so.size - 1, None if ro is None else ro.ctypes.data,
                                                  0 if ro is None else ro.size - 1, int(bool(reverse_complement))))
        self.n_seqs = so.size - 1
        self.lengths = np.diff(so.astype(np.int64))

    def upload_sequences(self, seqs, reverse_complement=False, records=None):
        """seqs: list of bytes/uint8 arrays.  records: optional list (per sequence) of record lengths."""
        arrs = [np.frombuffer(s, dtype=np.uint8) if isinstance(s, (bytes, bytearray)) else np.asarray(s, dtype=np.uint8)
                for s in seqs]
        so = np.zeros(len(arrs) + 1, dtype=np.uint64)
        so[1:] = np.cumsum([a.size for a in arrs])
        data = np.concatenate(arrs) if arrs else np.zeros(0, np.uint8)
        ro = None
        if records is None and reverse_complement:
            records = [[a.size] for a in arrs]          # one record per sequence
        if records is not None:
            flat = [l for rl in records for l in rl]
            ro = np.zeros(len(flat) + 1, dtype=np.uint64)
            ro[1:] = np.cumsum(flat)
        self.upload(data, so, ro, reverse_complement)

    def download_sequence(self, i):
        out = np.zeros(int(self.lengths[i]), dtype=np.uint8)
        self._check(self._lib.snacc_download_sequence(self._h, int(i), out.ctypes.data))
        return out

    # ---- sizes (raw compressed lengths, no +33) ----
    def single_sizes(self, algorithm, idx=None):
        idx = np.arange(self.n_seqs, dtype=np.int32) if idx is None else np.ascontiguousarray(idx, dtype=np.int32)
        out = np.zeros(idx.size, dtype=np.int64)
        self._check(self._lib.snacc_single_sizes(self._h, _codec(algorithm), idx.ctypes.data, idx.size, out.ctypes.data))
        return out

    def pair_sizes(self, algorithm, xs, ys):
        xs = np.ascontiguousarray(xs, dtype=np.int32)
        ys = np.ascontiguousarray(ys, dtype=np.int32)
        if xs.shape != ys.shape:
            raise ValueError("xs and ys differ in shape")
        out = np.zeros(xs.size, dtype=np.int64)
        self._check(self._lib.snacc_pair_sizes(self._h, _codec(algorithm), xs.ctypes.data, ys.ctypes.data, xs.size,
                                               out.ctypes.data))
        return out.reshape(xs.shape)

    def tile_sizes(self, algorithm, row0, n_rows, col0, n_cols, out=None):
        """rows [row0, row0+n_rows) x cols [col0, col0+n_cols) of the ordered-pair matrix; ``out``: a C-contiguous
        int64 (n_rows, n_cols) array to fill in place (e.g. a slice of a pinned buffer), else a new array"""
        if out is None:
            out = np.empty((n_rows, n_cols), dtype=np.int64)
        elif out.dtype != np.int64 or out.shape != (n_rows, n_cols) or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous int64 array of shape (n_rows, n_cols)")
        self._check(self._lib.snacc_tile_sizes(self._h, _codec(algorithm), row0, n_rows, col0, n_cols, out.ctypes.data))
        return out

    # ---- multi-GPU: per-sequence prefix state (see include/snacc_b200.h) ----
    def prefix_record_bytes(self, algorithm):
        return int(self._lib.snacc_prefix_record_bytes(self._h, _codec(algorithm)))

    def export_prefix(self, algorithm, seqs):
        seqs = np.ascontiguousarray(seqs, dtype=np.int32)
        out = np.zeros((seqs.size, self.prefix_record_bytes(algorithm)), dtype=np.uint8)
        self._check(self._lib.snacc_export_prefix(self._h, _codec(algorithm), seqs.ctypes.data, seqs.size, out.ctypes.data))
        return out

    def import_prefix(self, algorithm, seqs, records):
        seqs = np.ascontiguousarray(seqs, dtype=np.int32)
        records = np.ascontiguousarray(records, dtype=np.uint8)
        if records.size != seqs.size * self.prefix_record_bytes(algorithm):
            raise ValueError("prefix records do not match the sequence list")
        self._check(self._lib.snacc_import_prefix(self._h, _codec(algorithm), seqs.ctypes.data, seqs.size, records.ctypes.data))

    def ncd(self, C, S, formula=0, bias=GETSIZEOF_BIAS, out=None):
        C = np.ascontiguousarray(C, dtype=np.int64)
        S = np.ascontiguousarray(S, dtype=np.int64)
        n = C.size
        if out is None:
            D = np.empty((n, n), dtype=np.float64)
        elif out.dtype != np.float64 or out.shape != (n, n) or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous float64 (n, n) array")
        else:
            D = out
        self._check(self._lib.snacc_ncd(self._h, C.ctypes.data, S.ctypes.data, n, int(formula), int(bias), D.ctypes.data))
        return D

    def upgma(self, D, metrify=True):
        """scipy's linkage matrix ((n-1) x 4) of average-linkage clustering of the distance matrix D, computed on the
        device; ``metrify`` first symmetrises D and zeroes its diagonal (reference misc.py:20-25).  Raises ValueError
        where scipy does: a non-finite entry, and with ``metrify`` off an asymmetric matrix or a non-zero diagonal."""
        D = np.ascontiguousarray(D, dtype=np.float64)
        n = D.shape[0] if D.ndim else 0
        if D.ndim != 2 or D.shape[1] != n or n < 2:
            raise ValueError("D must be a square matrix with at least two rows")
        Z = np.zeros((n - 1, 4), dtype=np.float64)
        rc = self._lib.snacc_upgma(self._h, D.ctypes.data, n, int(bool(metrify)), Z.ctypes.data)
        if rc == -2:                                   # input the reference rejects
            raise ValueError(self._lib.snacc_last_error(self._h).decode(errors="replace"))
        self._check(rc)
        return Z

    # ---- instrumentation ----
    def last_kernel_ms(self):
        ms = ctypes.c_double(0)
        n = ctypes.c_int64(0)
        self._lib.snacc_last_kernel_ms(self._h, ctypes.byref(ms), ctypes.byref(n))
        return ms.value, n.value

    def stat(self, name):
        v = ctypes.c_double(0)
        self._check(self._lib.snacc_get_stat(self._h, name.encode(), ctypes.byref(v)))
        return v.value

    def set_option(self, name, value):
        self._check(self._lib.snacc_set_option(self._h, name.encode(), int(value)))


def _codec(algorithm):
    if algorithm not in CODEC_IDS:
        raise KeyError(f"compression '{algorithm}' is not supported on the GPU path (supported: lz4, gzip, zlib, bzip2)")
    return CODEC_IDS[algorithm]
