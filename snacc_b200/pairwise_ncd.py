"""Host-side mirror of the reference's ``snacc/pairwise_ncd.py`` for the GPU path.

Same names, argument meaning and error behaviour as the reference:
  extract_sequences   pairwise_ncd.py:15-39
  compressed_size     pairwise_ncd.py:42-90   (returns ``(sequences, len(compressed) + 33)``)
  compute_distance    pairwise_ncd.py:93-111
plus the batch entry point the new CLI calls instead of the thread-pool fan-out of cli.py:104-136:
  ncd_matrix(files, algorithm, reverse_complement=False, fast_mode=False, gpus=None)
All compressed sizes come from libsnacc_b200.so (CUDA, sm_100a).  There is no CPU fallback: without
the library or a GPU these functions raise.
"""
import threading
from pathlib import Path

import numpy as np

from . import fasta
from .engine import CODEC_IDS, GETSIZEOF_BIAS, Engine

_EXT = {"lzma": ".lzma", "gzip": ".gz", "bzip2": ".bz2", "zlib": ".ZLIB", "lz4": ".lz4"}
_lock = threading.Lock()
_engine = None


def _shared_engine():
    global _engine
    with _lock:
        if _engine is None:
            _engine = Engine(0)
        return _engine


def _complement_table():
    pairs = {"A": "T", "C": "G", "G": "C", "T": "A", "M": "K", "R": "Y", "W": "W", "S": "S", "Y": "R", "K": "M",
             "V": "B", "H": "D", "D": "H", "B": "V", "X": "X", "N": "N", "U": "A"}
    t = bytearray(range(256))
    for k, v in pairs.items():
        t[ord(k)] = ord(v)
        t[ord(k.lower())] = ord(v.lower())
    return bytes(t)


_COMPLEMENT = _complement_table()


def extract_sequences(sequences, reverse_complement=False):
    """Concatenated record sequences of a FASTA file (or of a tuple of two files) as ``str``."""
    if type(sequences) == tuple:
        return (extract_sequences(sequences[0], reverse_complement=reverse_complement)
                + extract_sequences(sequences[1], reverse_complement=reverse_complement))
    data, recs = fasta.read_fasta(Path(sequences).absolute())
    if data.size == 0:
        raise ValueError(f"No sequence extracted. Ensure that file {Path(sequences).absolute()} contains a proper "
                         "FASTA definition line (i.e. a line that starts with '>sequence_name').")
    if not reverse_complement:
        return data.tobytes().decode("latin-1")
    out, pos = [], 0
    raw = data.tobytes()
    for r in recs:
        out.append(raw[pos:pos + r].translate(_COMPLEMENT)[::-1])
        pos += r
    return b"".join(out).decode("latin-1")


def compressed_size(sequences, algorithm, reverse_complement=False, save_directory=None, BWT=False, bwte_inputs={}):
    """Compressed size of one file or of the concatenation of a tuple of two files.

    Drop-in for the reference function: returns ``(sequences, size)`` with ``size`` including the +33 of
    ``sys.getsizeof``.  Routed through a batch of one on the GPU; thread-safe."""
    ext = _EXT[algorithm]            # KeyError for an unknown algorithm, like the reference
    if algorithm not in CODEC_IDS:
        raise KeyError(f"compression '{algorithm}' is not supported on the GPU path (supported: lz4, gzip, zlib, bzip2)")
    if save_directory:
        raise NotImplementedError("save_directory is not supported on the GPU path: only sizes are produced, "
                                  f"no {ext} stream is materialised")
    files = list(sequences) if type(sequences) == tuple else [sequences]
    data, so, ro = fasta.load_corpus(files)
    eng = _shared_engine()
    with _lock:
        eng.upload(data, so, ro, reverse_complement)
        if len(files) == 2:
            size = int(eng.pair_sizes(algorithm, [0], [1])[0])
        else:
            size = int(eng.single_sizes(algorithm, [0])[0])
    return (sequences, size + GETSIZEOF_BIAS)


def compute_distance(x, y, cxy, cyx):
    """NCD of two files from their four compressed sizes (reference formula, float64)."""
    lo, hi = (y, x) if x > y else (x, y)
    return min((cxy - lo) / hi, (cyx - lo) / hi)


def ncd_matrix(files, algorithm, reverse_complement=False, fast_mode=False, gpus=None, engine=None,
               rows_per_call=None):
    """All-pairs sizes and distances for ``files`` (already de-duplicated and ordered by the caller).

    Returns ``(labels, C, S, D)``: ``C[i] = len(compress(x_i))``, ``S[i, j] = len(compress(x_i + x_j))`` (raw
    lengths, no +33), ``D`` the float64 NCD matrix with the reference formula (both orders, +33 bias) or,
    with ``fast_mode``, the one-order formula on the upper triangle mirrored.

    Multi-GPU: inside a ``torch.distributed`` process group (one process per GPU, e.g. under ``torchrun``) every
    rank parses and uploads its band of the files, the corpus is all-gathered over NVLink, every rank computes its
    columns of S and all ranks return the full result.  From a plain process, ``gpus=N`` (N > 1) launches N such
    ranks (``sharding.run_multi_gpu``) and returns rank 0's result; ``gpus`` in (None, 1) uses this process's GPU."""
    from . import sharding
    if algorithm not in CODEC_IDS:
        raise KeyError(f"compression '{algorithm}' is not supported on the GPU path (supported: lz4, gzip, zlib, bzip2)")
    files = [Path(f) for f in files]
    if gpus is not None and int(gpus) > 1 and sharding._dist() is None and engine is None:
        return sharding.run_multi_gpu(files, algorithm, reverse_complement, fast_mode, int(gpus))
    return sharding.all_pairs(files, algorithm, reverse_complement, fast_mode, engine=engine,
                              rows_per_call=rows_per_call)
