"""gzip / zlib sizes when the deflate state of a call is split into memory-bounded bands of y sequences.

Every size is compared with the unbanded call on the same context and with Python's zlib (raw deflate at level 9 / 6,
memLevel 8: gzip = raw + 18, zlib = raw + 6).  `deflate_band_bytes` caps the y-side state of one band so that small
corpora go through many bands; results must not change."""
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle.make_golden import synth_vector
from snacc_b200 import synth
from snacc_b200.engine import Engine, SnaccGpuError

pytestmark = pytest.mark.gpu

LEVEL = {"gzip": (9, 18), "zlib": (6, 6)}
BAND_BYTES = 5_000_000          # one to three y of the tile corpus per band (its largest y needs ~2.5 MB at level 6)


def zlib_size(data, algo):
    level, wrapper = LEVEL[algo]
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, zlib.Z_DEFAULT_STRATEGY)
    return len(c.compress(bytes(data)) + c.flush()) + wrapper


def zlib_sizes(items, algo):
    with ThreadPoolExecutor() as ex:                       # zlib releases the GIL
        return np.array(list(ex.map(lambda d: zlib_size(d, algo), items)), dtype=np.int64)


@pytest.fixture(scope="module")
def corpus():
    g = synth.phylogeny(2, 140_000, seed=21)               # >= 128 KiB: parallel parse alone, canonical stream
    g.append(synth.mutate(np.random.default_rng(22), g[0]))
    g.append(synth_vector("dna", 30_000, 23))              # shorter than DFL_CANON_MIN (36 864)
    g.append(synth_vector("dna", 5_000, 24))               # shorter than DFL_XTAIL (40 960): whole x index
    g.append(synth_vector("nrun", 60_000, 25))             # non-ACGT bytes
    g.append(synth_vector("bytes", 50_000, 26))            # random bytes: no canonical stream, serial parse of y
    return [np.asarray(s, dtype=np.uint8) for s in g]


@pytest.fixture(scope="module")
def reference(corpus):
    """zlib sizes of every single and every ordered pair, per codec"""
    n = len(corpus)
    out = {}
    for algo in LEVEL:
        C = zlib_sizes(corpus, algo)
        S = zlib_sizes([np.concatenate([corpus[a], corpus[b]]) for a in range(n) for b in range(n)], algo).reshape(n, n)
        out[algo] = (C, S)
    return out


def banded(engine, value):
    engine.set_option("deflate_band_bytes", value)
    engine.set_option("invalidate_caches", 1)


@pytest.mark.parametrize("algo", ["gzip", "zlib"])
def test_forced_bands_tiles(engine, corpus, reference, algo):
    n = len(corpus)
    engine.upload_sequences(corpus)
    try:
        banded(engine, 0)
        S0 = engine.tile_sizes(algo, 0, n, 0, n)
        assert engine.stat("deflate_bands") == 1
        banded(engine, BAND_BYTES)
        S1 = engine.tile_sizes(algo, 0, n, 0, n)
        bands = engine.stat("deflate_bands")
        assert bands > 1
        # each sequence is fully prepared at most twice: once for its record, once as the y of its band
        assert engine.stat("deflate_prepared_seqs") <= 2 * n
        assert np.array_equal(S1, S0)
        assert np.array_equal(S1, reference[algo][1])
        # a second tile on the banded context: the records stay, only the y bands are prepared again
        S2 = engine.tile_sizes(algo, 0, n, 2, 3)
        assert np.array_equal(S2, reference[algo][1][:, 2:5])
        assert engine.stat("deflate_prepared_seqs") == 3
    finally:
        banded(engine, 0)


@pytest.mark.parametrize("algo", ["gzip", "zlib"])
def test_forced_bands_job_lists(engine, corpus, reference, algo):
    """unsorted, repeated y and x == y jobs come back in job order"""
    n = len(corpus)
    rng = np.random.default_rng(31)
    xs = rng.integers(0, n, size=40).astype(np.int32)
    ys = rng.permutation(np.repeat(np.arange(n), 7))[:40].astype(np.int32)
    xs[:n] = ys[:n]                                        # x == y
    ref = reference[algo][1][xs, ys]
    engine.upload_sequences(corpus)
    try:
        banded(engine, 0)
        got0 = engine.pair_sizes(algo, xs, ys)
        banded(engine, BAND_BYTES)
        got1 = engine.pair_sizes(algo, xs, ys)
        assert engine.stat("deflate_bands") > 1
        assert np.array_equal(got0, ref) and np.array_equal(got1, ref)
        # the fast-mode shape: upper triangle only
        tx, ty = np.triu_indices(n, 1)
        assert np.array_equal(engine.pair_sizes(algo, tx, ty), reference[algo][1][tx, ty])
        # whole x indexes (deflate_tail_index 0): the planner counts the larger x side and its sort scratch
        engine.set_option("deflate_tail_index", 0)
        banded(engine, BAND_BYTES)
        assert np.array_equal(engine.pair_sizes(algo, xs, ys), ref)
        assert engine.stat("deflate_bands") > 1
    finally:
        engine.set_option("deflate_tail_index", 1)
        banded(engine, 0)


@pytest.mark.parametrize("algo", ["gzip", "zlib"])
def test_forced_bands_singles_and_records(engine, corpus, reference, algo):
    n = len(corpus)
    idx = np.arange(n, dtype=np.int32)
    engine.upload_sequences(corpus)
    try:
        banded(engine, 0)
        C0 = engine.single_sizes(algo)
        R0 = engine.export_prefix(algo, idx)
        banded(engine, BAND_BYTES)
        C1 = engine.single_sizes(algo)
        assert engine.stat("deflate_bands") > 1
        R1 = engine.export_prefix(algo, idx)
        assert np.array_equal(C0, reference[algo][0]) and np.array_equal(C1, C0)
        assert np.array_equal(R1, R0)
    finally:
        banded(engine, 0)


@pytest.mark.parametrize("algo", ["gzip", "zlib"])
def test_default_plan_one_band(engine, corpus, reference, algo):
    """without the option a small corpus fits: one band, every sequence prepared once, and the state stays resident"""
    n = len(corpus)
    engine.upload_sequences(corpus)
    banded(engine, 0)
    assert np.array_equal(engine.single_sizes(algo), reference[algo][0])
    assert engine.stat("deflate_bands") == 1 and engine.stat("deflate_prepared_seqs") == n
    assert np.array_equal(engine.tile_sizes(algo, 0, n, 0, n), reference[algo][1])
    assert engine.stat("deflate_bands") == 1 and engine.stat("deflate_prepared_seqs") == 0


@pytest.mark.parametrize("algo", ["gzip", "zlib"])
def test_rank_state_bytes(algo):
    """one context standing in for a rank: the sequences it does not own arrive only as imported records.  Its deflate
    state is the x side of all sequences plus the y side of its own columns: with 3 of 8 as y at most half of what
    the same context needs with all 8 as y.  Fresh contexts, so that no other test's buffers count."""
    g = synth.phylogeny(8, 400_000, seed=41)
    n = len(g)
    theirs = np.array([0, 2, 4, 6, 7], dtype=np.int32)
    mine = np.array([1, 3, 5], dtype=np.int32)
    xs, ys = np.repeat(np.arange(n), mine.size).astype(np.int32), np.tile(mine, n)
    with Engine(0) as other:                               # "another rank" parses its sequences
        other.upload_sequences(g)
        other.single_sizes(algo, theirs)
        recs = other.export_prefix(algo, theirs)
    with Engine(0) as rank:
        rank.upload_sequences(g)
        rank.import_prefix(algo, theirs, recs)
        S_mine = rank.pair_sizes(algo, xs, ys)
        part = rank.stat("deflate_state_bytes")
        assert rank.stat("deflate_bands") == 1
    with Engine(0) as whole:
        whole.upload_sequences(g)
        ax, ay = np.repeat(np.arange(n), n).astype(np.int32), np.tile(np.arange(n), n).astype(np.int32)
        S_all = whole.pair_sizes(algo, ax, ay).reshape(n, n)
        full = whole.stat("deflate_state_bytes")
    assert 0 < part <= full / 2, (part, full)
    assert np.array_equal(S_mine, S_all[xs, ys])
    assert np.array_equal(S_mine, zlib_sizes([np.concatenate([g[a], g[b]]) for a, b in zip(xs, ys)], algo))


@pytest.mark.parametrize("algo", ["gzip", "zlib"])
def test_budget_below_one_y_is_refused(engine, corpus, reference, algo):
    n = len(corpus)
    engine.upload_sequences(corpus)
    try:
        banded(engine, 1000)
        with pytest.raises(SnaccGpuError) as e:
            engine.pair_sizes(algo, np.arange(n), np.arange(n))
        assert "stream too large" in str(e.value) and "bytes are free" in str(e.value)
    finally:
        banded(engine, 0)
    assert np.array_equal(engine.pair_sizes(algo, np.arange(n), np.arange(n)), np.diag(reference[algo][1]))
