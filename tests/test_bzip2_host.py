"""CPU: the product's bzip2 size functions (snacc_b200/csrc/bzip2.cuh: RLE1, block cut, x-prefix / junction
decomposition of a pair, MTF + RLE2, Huffman table choice, bit count), compiled for the host by tests/host_emu_bzip2.cu
with a plain host rotation sort as the BWT, against len(bz2.compress(...)) -- the reference's own call
(pairwise_ncd.py:76).  Also pins the numpy reference BWT of tests/test_bzip2_kernels_gpu.py to that host sort, and
checks that its crafted Fibonacci last columns reach the 17-bit code-length cap."""
import bz2
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from snacc_b200 import _build

HERE = os.path.dirname(os.path.abspath(__file__))
MAXB = 100000 * 9 - 19            # nblockMAX of level 9


@pytest.fixture(scope="module")
def bz(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("bzemu") / "libhost_emu_bzip2.so")
    subprocess.check_call([_build._nvcc(), "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                           "-Xcompiler", "-fPIC", "-shared", "-o", so, os.path.join(HERE, "host_emu_bzip2.cu")])
    e = ctypes.CDLL(so)
    e.emu_bz2_single.restype = ctypes.c_int64
    e.emu_bz2_single.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_void_p]
    e.emu_bz2_pair.restype = ctypes.c_int64
    e.emu_bz2_pair.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_void_p]
    e.emu_bz2_block_lengths.restype = ctypes.c_int64
    e.emu_bz2_block_lengths.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_int64]
    e.emu_bz2_code_lengths.restype = None
    e.emu_bz2_code_lengths.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]
    e.emu_bz2_bwt.restype = None
    e.emu_bz2_bwt.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_void_p]
    e.emu_bz2_rescaled_builds.restype = ctypes.c_int32
    e.emu_bz2_rescaled_builds.argtypes = [ctypes.c_char_p, ctypes.c_uint32]
    return e


def single(bz, s):
    return bz.emu_bz2_single(s, len(s), None)


def pair(bz, x, y):
    nb = ctypes.c_int64(0)
    return bz.emu_bz2_pair(x, len(x), y, len(y), ctypes.byref(nb)), nb.value


def no_runs(n, seed):
    """n bytes with no two neighbours equal: RLE1 leaves them as they are"""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 255, n, dtype=np.int64)
    return (np.cumsum(a + 1) % 256).astype(np.uint8).tobytes()


def dna(n, seed, alphabet=b"ACGT"):
    rng = np.random.default_rng(seed)
    return np.frombuffer(alphabet, np.uint8)[rng.integers(0, len(alphabet), n)].tobytes()


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 255, 256, 257, 258, 259, 260, 9999, 10000, 10001])
def test_short_lengths(bz, n):
    for s in (no_runs(n, n), b"A" * n, dna(n, n)):
        assert single(bz, s) == len(bz2.compress(s))


@pytest.mark.parametrize("n", [MAXB - 5, MAXB - 1, MAXB, MAXB + 1, MAXB + 5, 2 * MAXB - 1, 2 * MAXB + 1])
def test_block_cut_lengths(bz, n):
    s = no_runs(n, n)
    out = np.zeros(4, np.uint32)
    nb = bz.emu_bz2_block_lengths(s, n, out.ctypes.data, 4)
    # no runs: RLE1 bytes = input bytes; a block closes once it holds nblockMAX bytes and more input follows
    assert nb == (n - 1) // MAXB + 1
    assert single(bz, s) == len(bz2.compress(s))


@pytest.mark.parametrize("run", [4, 5, 255, 256, 1000])
def test_run_straddling_a_cut(bz, run):
    # the run starts just before the cut, so its emission decides where the block closes
    for before in (MAXB - 3, MAXB - 1, MAXB):
        s = no_runs(before, run + before)
        s = s + bytes([s[-1] ^ 0x55]) * run + no_runs(5000, 7)
        assert single(bz, s) == len(bz2.compress(s)), before


def test_three_blocks(bz):
    s = dna(2 * MAXB + 200000, 3, b"ACGTN")
    assert single(bz, s) == len(bz2.compress(s))


@pytest.mark.parametrize("kind", ["acgt", "iupac", "lower", "protein", "all256", "runs"])
def test_alphabets(bz, kind):
    rng = random.Random(kind)
    alph = {"acgt": b"ACGT", "iupac": b"ACGTNRYKMSWBDHV", "lower": b"ACGTacgtn", "protein": b"ACDEFGHIKLMNPQRSTVWYX",
            "all256": bytes(range(256)), "runs": b"AN"}[kind]
    for n in (50, 3000, 40000):
        if kind == "runs":
            s = b"".join(bytes([rng.choice(alph)]) * rng.choice([1, 3, 4, 5, 40, 300]) for _ in range(n // 40))
        else:
            s = bytes(rng.choice(alph) for _ in range(n))
        assert single(bz, s) == len(bz2.compress(s))


def code_lengths(bz, freq, max_len):
    freq = np.ascontiguousarray(freq, np.int32)
    out = np.zeros(freq.size, np.uint8)
    bz.emu_bz2_code_lengths(freq.ctypes.data, freq.size, max_len, out.ctypes.data)
    return out


def test_code_length_rescale(bz):
    # Fibonacci frequencies give a Huffman code 1, 2, ..., 24 bits long; the 17-bit cap makes the build rescale the
    # weights (1 + (w >> 8) / 2) until every code fits, and the lengths still satisfy Kraft's equality
    fib = [1, 1]
    while len(fib) < 25:
        fib.append(fib[-1] + fib[-2])
    free = code_lengths(bz, fib, 64)
    assert free.max() == 24
    capped = code_lengths(bz, fib, 17)
    assert capped.max() <= 17
    assert sum(2.0 ** -int(l) for l in capped) == 1.0


def test_geometric_bytes(bz):
    rng = np.random.default_rng(5)
    for p in (0.5, 0.6, 0.7):
        s = np.minimum(rng.geometric(p, 400000) - 1, 255).astype(np.uint8).tobytes()
        assert single(bz, s) == len(bz2.compress(s))


@pytest.mark.parametrize("n_mtf", [199, 200, 201, 599, 600, 601, 1199, 1200, 1201, 2399, 2400, 2401])
def test_table_count_thresholds(bz, n_mtf):
    # random bytes with no neighbours equal: nMTF is close to the length (the BWT brings a few equal bytes together, so
    # zero runs shorten it a little), so a few lengths around each threshold put nMTF on both sides of it
    for n in range(n_mtf - 3, n_mtf + 6):
        s = no_runs(n, n)
        assert single(bz, s) == len(bz2.compress(s))


@pytest.mark.parametrize("period", [1, 2, 3, 258])
def test_periodic_blocks(bz, period):
    unit = no_runs(period, period) if period > 1 else b"A"
    for n in (1000, 50000, MAXB + 7):
        s = (unit * (n // period + 1))[:n]
        assert single(bz, s) == len(bz2.compress(s)), n


@pytest.mark.parametrize("tail,head", [(3, 1), (2, 2), (1, 3), (254, 1), (255, 1), (255, 0), (250, 6), (100, 900)])
def test_pair_runs_merge_at_the_junction(bz, tail, head):
    x = dna(3000, tail) + b"T" * tail
    y = b"T" * head + b"G" + dna(3000, head)
    got, _ = pair(bz, x, y)
    assert got == len(bz2.compress(x + y))


@pytest.mark.parametrize("nx", [1000, MAXB - 2, MAXB, MAXB + 3, MAXB + 70000])
def test_pair_decomposition_around_one_block(bz, nx):
    x = no_runs(nx, nx)
    for y in (dna(20000, 1), bytes([x[-1]]) * 300 + dna(100, 2), bytes([x[-1]]) * 4):
        got, _ = pair(bz, x, y)
        assert got == len(bz2.compress(x + y))


def test_pair_decomposition_multi_block(bz):
    x, y = dna(MAXB + 123456, 9, b"ACGTN"), dna(MAXB + 54321, 10)
    got, nblocks = pair(bz, x, y)
    assert nblocks >= 3
    assert got == len(bz2.compress(x + y))


def test_fuzz_planted_repeats(bz):
    rng = random.Random(2024)
    for _ in range(150):
        alph = rng.choice([b"ACGT", b"ACGTN", b"AC", bytes(range(256)), b"ACDEFGHIKLMNPQRSTVWY"])
        parts = []
        for _ in range(rng.randint(1, 6)):
            r = rng.random()
            if r < 0.5 or not parts:
                parts.append(bytes(rng.choice(alph) for _ in range(rng.randint(1, 2000))))
            elif r < 0.8:
                src = b"".join(parts)
                a = rng.randrange(len(src))
                parts.append(src[a:a + rng.randint(1, 3000)])
            else:
                parts.append(bytes([rng.choice(alph)]) * rng.randint(1, 600))
        s = b"".join(parts)
        cut = rng.randint(1, len(s) - 1) if len(s) > 1 else 0
        if cut:
            got, _ = pair(bz, s[:cut], s[cut:])
            assert got == len(bz2.compress(s)), (len(s), cut)
        assert single(bz, s) == len(bz2.compress(s))


def test_reference_bwt_equals_the_emulator(bz):
    # the numpy BWT that tests/test_bzip2_kernels_gpu.py holds the device kernels to, pinned byte for byte to the
    # emulator's on every block those tests use
    from test_bzip2_kernels_gpu import family_cases, parallel_map, ref_bwt

    def emu_bwt(t):
        out = ctypes.create_string_buffer(len(t))
        bz.emu_bz2_bwt(t, len(t), out)
        return out.raw

    cases = family_cases()
    bad = [f"{fam} n={n}" for (fam, n, _), a, b in zip(cases, parallel_map(lambda c: ref_bwt(c[2]), cases),
                                                        parallel_map(lambda c: emu_bwt(c[2]), cases)) if a != b]
    assert not bad, bad


def test_fibonacci_mtf_columns_reach_the_code_length_cap(bz):
    # the crafted last columns that tests/test_bzip2_kernels_gpu.py gives the bit-count kernel for the 17-bit rescale:
    # some of their 4 x 6 table builds go past 17 bits and rescale, and not all of them, so the tables' lengths differ
    from test_bzip2_kernels_gpu import crafted_last_columns
    cols = crafted_last_columns()
    for name in ("fibonacci_mtf_25", "fibonacci_mtf_27"):
        L = cols[name]
        assert 0 < bz.emu_bz2_rescaled_builds(L, len(L)) < 4 * 6, name
    # a witness that the count is not positive for any column: random bytes never reach the cap
    assert bz.emu_bz2_rescaled_builds(cols["nmtf2400"], 2400) == 0
