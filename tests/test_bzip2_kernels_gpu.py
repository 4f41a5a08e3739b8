"""GPU: the bzip2 device kernels (snacc_b200/csrc/bzip2.cuh) one by one, and the device driver end to end on inputs
where a prefix-doubling BWT and the block planner go wrong.

- The BWT of both sort regimes (bz_bwt_smem_kernel, bz_bwt_global_kernel), launched directly through
  tests/gpu_bzip2_kernels.cu, against `ref_bwt` below: numpy prefix doubling, pinned to the emulator's BWT by
  tests/test_bzip2_host.py on the CPU.  Periodic, self-repeating and near-repeating blocks up to nblockMAX + 4 bytes
  run the late doubling rounds, the h >= n exit and the full 20-bit rank keys, which random DNA never does.
- bz_bits_kernel on those last columns and on crafted ones against the serial bit count of the host emulation, and
  against libbz2 itself for run-free blocks.
- The engine against len(bz2.compress(...)) on every job of repetitive genomes, duplicated genomes, junctions behind a
  multi-block x, the shared-memory routing boundary, batches of more than 65 536 blocks or 192 MiB, and its caches
  across calls and uploads.
"""
import bz2
import ctypes
import os
import subprocess
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
MAXB = 100000 * 9 - 19                  # nblockMAX of level 9: the cut makes blocks of at most MAXB + 4 bytes
SMEM_MAX_N = 24576                      # BZ_SMEM_MAX_N: larger blocks sort in global memory
BATCH_BLOCKS = 1 << 16                  # BZ_BATCH_BLOCKS
BATCH_BYTES = 192 << 20                 # BZ_BATCH_BYTES

LENGTHS = [1, 2, 3, 4, 5, 7, 8, 9, 1023, 1024, 1025, SMEM_MAX_N - 1, SMEM_MAX_N, SMEM_MAX_N + 1,
           65535, 65536, 65537, 262144, MAXB - 1, MAXB, MAXB + 4]
PERIODS = [1, 2, 3, 5, 255, 256, 4096, "n/3"]


# ---- reference BWT ---------------------------------------------------------------------------------------------------
def ref_bwt(t):
    """last column of the sorted cyclic rotations of t: prefix doubling, np.lexsort on (rank[i], rank[i + h]) and dense
    re-ranking, until every rank is distinct or h >= n (what is still tied then is equal rotations)"""
    a = np.frombuffer(bytes(t), np.uint8)
    n = a.size
    idx = np.arange(n, dtype=np.int64)
    rank = a.astype(np.int64)
    h = 1
    while True:
        second = rank[(idx + h) % n]
        sa = np.lexsort((second, rank))
        r1, r2 = rank[sa], second[sa]
        head = np.ones(n, bool)
        head[1:] = (r1[1:] != r1[:-1]) | (r2[1:] != r2[:-1])
        rank = np.empty(n, np.int64)
        rank[sa] = np.cumsum(head) - 1
        if rank[sa[-1]] == n - 1 or h >= n:
            break
        h *= 2
    return a[(sa - 1) % n].tobytes()


# ---- input families --------------------------------------------------------------------------------------------------
def _rng(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


def _acgt(n, rng):
    return np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes()


def rle1_run(b, T):
    """the RLE1 emissions of a run of T bytes b: chunks of 255 as b b b b 251, the rest as itself (1-3) or b b b b c-4"""
    out = bytes([b]) * 4 + b"\xfb"
    r = T % 255
    return out * (T // 255) + (bytes([b]) * r if r < 4 else bytes([b]) * 4 + bytes([r - 4]))


def _fibonacci_word(n):
    a, b = b"a", b"ab"
    while len(b) < n:
        a, b = b, b + a
    return b[:n]


def _thue_morse(n):
    i = np.arange(n, dtype=np.uint64)
    c = np.zeros(n, np.uint8)
    while i.any():
        c ^= (i & np.uint64(1)).astype(np.uint8)
        i >>= np.uint64(1)
    return (c + ord("a")).tobytes()


def family_block(fam, n):
    """n bytes of one family (seeded by family and length)"""
    rng = _rng(fam, n)
    if fam == "acgt":
        return _acgt(n, rng)
    if fam == "all256":
        a = rng.integers(0, 256, n).astype(np.uint8)
        if n >= 256:
            a[rng.choice(n, 256, replace=False)] = rng.permutation(256)
        return a.tobytes()
    if fam == "binary":
        return rng.integers(0, 2, n).astype(np.uint8).tobytes()
    if fam.startswith("period"):
        p = fam[len("period"):]
        p = max(1, n // 3) if p == "n/3" else int(p)
        unit = rng.integers(0, 256, p).astype(np.uint8).tobytes()
        return (unit * (n // p + 1))[:n]
    if fam in ("xx", "xx1"):
        x = _acgt((n + 1) // 2, rng)
        s = bytearray((x * 2)[:n])
        if fam == "xx1" and n >= 2:
            m = len(x) + len(x) // 2
            m = min(m, n - 1)
            s[m] = (s[m] + 1) % 256                     # one byte changed in the middle of the second copy
        return bytes(s)
    if fam == "fibonacci":
        return _fibonacci_word(n)
    if fam == "thue_morse":
        return _thue_morse(n)
    if fam == "nrun":
        return (b"NNNN\xfb" * (n // 5 + 1))[:n]        # RLE1 of a long N run
    if fam == "acgt_gaps":
        s = _acgt(n, rng)
        return (s[:n // 3] + rle1_run(ord("N"), 10000) + s[n // 3:2 * n // 3] + rle1_run(ord("N"), 100000) +
                s[2 * n // 3:])[:n]
    raise ValueError(fam)


FAMILIES = (["acgt", "all256", "binary"] + [f"period{p}" for p in PERIODS] +
            ["xx", "xx1", "fibonacci", "thue_morse", "nrun", "acgt_gaps"])


def family_cases():
    """(family, n, block) for every family and length; a period as long as the block is not periodic and is left out"""
    out = []
    for fam in FAMILIES:
        for n in LENGTHS:
            if fam.startswith("period") and fam != "period1" and fam != "periodn/3" and int(fam[6:]) >= n:
                continue
            out.append((fam, n, family_block(fam, n)))
    return out


def parallel_map(f, items):
    """f over items on all host threads (numpy's sorts and libbz2 release the GIL)"""
    with ThreadPoolExecutor(os.cpu_count()) as ex:
        return list(ex.map(f, items))


# ---- GPU part --------------------------------------------------------------------------------------------------------
def _build_lib(tmp_path_factory, src, name):
    from snacc_b200 import _build
    so = str(tmp_path_factory.mktemp(name) / f"lib{name}.so")
    subprocess.check_call([_build._nvcc(), "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                           "-Xcompiler", "-fPIC", "-shared", "-o", so, os.path.join(HERE, src)])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def kbz(tmp_path_factory):
    k = _build_lib(tmp_path_factory, "gpu_bzip2_kernels.cu", "gpu_bzip2_kernels")
    k.kbz_bwt.restype = ctypes.c_int
    k.kbz_bwt.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]
    k.kbz_bits.restype = ctypes.c_int
    k.kbz_bits.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p]
    return k


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    e = _build_lib(tmp_path_factory, "host_emu_bzip2.cu", "host_emu_bzip2_k")
    e.emu_bz2_block_bits.restype = ctypes.c_int64
    e.emu_bz2_block_bits.argtypes = [ctypes.c_char_p, ctypes.c_uint32]
    e.emu_bz2_block_lengths.restype = ctypes.c_int64
    e.emu_bz2_block_lengths.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_int64]
    return e


def kernel_bwt(kbz, blocks, regime):
    lens = np.array([len(b) for b in blocks], np.uint32)
    out = ctypes.create_string_buffer(int(lens.sum()))
    rc = kbz.kbz_bwt(b"".join(blocks), lens.ctypes.data, len(blocks), regime, out)
    assert rc == 0, f"kbz_bwt: error {rc}"
    raw, res, o = out.raw, [], 0
    for n in lens:
        res.append(raw[o:o + int(n)])
        o += int(n)
    return res


def kernel_bits(kbz, Ls):
    lens = np.array([len(b) for b in Ls], np.uint32)
    bits = np.zeros(len(Ls), np.int64)
    rc = kbz.kbz_bits(b"".join(Ls), lens.ctypes.data, len(Ls), bits.ctypes.data)
    assert rc == 0, f"kbz_bits: error {rc}"
    return bits


def emu_bits(emu, Ls):
    return np.array(parallel_map(lambda L: emu.emu_bz2_block_bits(L, len(L)), Ls), np.int64)


def stream_bytes(bits):
    return (32 + 48 + 32 + bits + 7) // 8


@pytest.fixture(scope="module")
def cases():
    """every family block with its reference last column"""
    c = family_cases()
    refs = parallel_map(lambda fnb: ref_bwt(fnb[2]), c)
    return [(f, n, b, L) for (f, n, b), L in zip(c, refs)]


def _bwt_mismatches(cases, got):
    bad = []
    for (fam, n, _, want), L in zip(cases, got):
        if L != want:
            a, b = np.frombuffer(L, np.uint8), np.frombuffer(want, np.uint8)
            i = int(np.flatnonzero(a != b)[0])
            bad.append(f"{fam} n={n}: first difference at {i} (kernel {a[i]}, reference {b[i]})")
    return bad


@pytest.mark.gpu
@pytest.mark.parametrize("regime", [0, 1], ids=["smem", "global"])
def test_bwt_kernel_equals_reference(kbz, cases, regime):
    # blocks up to BZ_SMEM_MAX_N bytes go through both kernels
    sel = [c for c in cases if regime == 1 or c[1] <= SMEM_MAX_N]
    got = kernel_bwt(kbz, [c[2] for c in sel], regime)
    bad = _bwt_mismatches(sel, got)
    assert not bad, f"{len(bad)} of {len(sel)} blocks differ:\n" + "\n".join(bad[:40])


@pytest.mark.gpu
def test_bits_kernel_on_reference_bwts(kbz, emu, cases):
    Ls = [c[3] for c in cases]
    got, want = kernel_bits(kbz, Ls), emu_bits(emu, Ls)
    bad = [f"{c[0]} n={c[1]}: {g} != {w}" for c, g, w in zip(cases, got, want) if g != w]
    assert not bad, "\n".join(bad[:40])


def _run_free(b):
    """no 4 equal bytes in a row: RLE1 leaves the bytes as they are"""
    a = np.frombuffer(b, np.uint8)
    return a.size < 4 or not np.any((a[3:] == a[:-3]) & (a[2:-1] == a[:-3]) & (a[1:-2] == a[:-3]))


@pytest.mark.gpu
def test_bits_kernel_on_run_free_blocks_equals_libbz2(kbz, cases):
    # a run-free block of at most nblockMAX bytes is its own RLE1 image and one block: bz2.compress sees exactly it
    sel = [c for c in cases if c[1] <= MAXB and _run_free(c[2])]
    assert len(sel) > 50
    got = stream_bytes(kernel_bits(kbz, [c[3] for c in sel]))
    want = np.array(parallel_map(lambda c: len(bz2.compress(c[2])), sel), np.int64)
    bad = [f"{c[0]} n={c[1]}: {g} != {w}" for c, g, w in zip(sel, got, want) if g != w]
    assert not bad, "\n".join(bad[:40])


def _no_runs(n, rng, alphabet=256):
    """n symbols, no two neighbours equal"""
    a = rng.integers(1, alphabet, n)
    return (np.cumsum(a) % alphabet).astype(np.uint8).tobytes()


def _mtf_decode(indices, nsym):
    """the bytes whose MTF positions are `indices` (initial list 0 .. nsym-1)"""
    yy = list(range(nsym))
    out = bytearray(len(indices))
    for i, j in enumerate(indices):
        b = yy.pop(j)
        yy.insert(0, b)
        out[i] = b
    return bytes(out)


def _fibonacci_positions(K):
    """MTF positions 1..K, position k repeated fib(k + 1) times (1, 2, 3, 5, ...)"""
    fib = [1, 2]
    while len(fib) < K:
        fib.append(fib[-1] + fib[-2])
    return np.repeat(np.arange(1, K + 1), fib)


def crafted_last_columns():
    rng = np.random.default_rng(77)
    cols = {}
    for n in range(1, 6):
        cols[f"short{n}_acgt"] = _acgt(n, rng)
        cols[f"short{n}_same"] = b"\x07" * n
        cols[f"short{n}_256"] = rng.integers(0, 256, n).astype(np.uint8).tobytes()
    cols["one_run_maxb+4"] = b"\x00" * (MAXB + 4)                  # RLE2 of a huge zero run
    cols["one_run_then_other"] = b"A" * (MAXB + 3) + b"C"
    a = rng.integers(0, 256, 20000).astype(np.uint8)
    a[:256] = rng.permutation(256)
    cols["all256"] = rng.permutation(a).tobytes()                 # alphaSize 258
    cols["all256_long"] = rng.integers(0, 256, MAXB).astype(np.uint8).tobytes()
    for p in (0.05, 0.3, 0.5, 0.7, 0.95):
        cols[f"geometric{p}"] = np.minimum(rng.geometric(p, 300000) - 1, 255).astype(np.uint8).tobytes()
    for t in (200, 600, 1200, 2400):
        for n in range(t - 3, t + 3):                             # nMTF is n or n + 1 here
            cols[f"nmtf{n}"] = _no_runs(n, rng)
    # MTF positions 1..K with Fibonacci frequencies in random order.  The six tables share the symbols, which flattens
    # each table's counts; with K = 25 and 27 some code-length builds still go past 17 bits and rescale, and others do
    # not (tests/test_bzip2_host.py checks both).  In runs of one position per group of 50 instead, every table
    # specialises: no build rescales, and the selectors carry the cost.
    for K in (25, 27):
        cols[f"fibonacci_mtf_{K}"] = _mtf_decode(rng.permutation(_fibonacci_positions(K)).tolist(), K + 1)
    groups = np.sort(_fibonacci_positions(24))
    groups = groups[: groups.size // 50 * 50].reshape(-1, 50)
    cols["fibonacci_mtf_grouped"] = _mtf_decode(groups[rng.permutation(len(groups))].ravel().tolist(), 25)
    return cols


@pytest.mark.gpu
def test_bits_kernel_on_crafted_last_columns(kbz, emu):
    cols = crafted_last_columns()
    names, Ls = list(cols), list(cols.values())
    got, want = kernel_bits(kbz, Ls), emu_bits(emu, Ls)
    bad = [f"{k}: {g} != {w}" for k, g, w in zip(names, got, want) if g != w]
    assert not bad, "\n".join(bad)


# ---- the engine end to end -------------------------------------------------------------------------------------------
def ref_sizes(xs, ys, seqs):
    """len(bz2.compress(x [+ y])) on all host threads"""
    return np.array(parallel_map(lambda k: len(bz2.compress(seqs[xs[k]] + (seqs[ys[k]] if ys[k] >= 0 else b""))),
                                 range(len(xs))), np.int64)


def all_pairs(n):
    return [a.astype(np.int32).ravel() for a in np.divmod(np.arange(n * n), n)]


def check_all(engine, seqs, xs=None, ys=None):
    """every single and the listed ordered pairs (all of them by default) against libbz2"""
    n = len(seqs)
    if xs is None:
        xs, ys = all_pairs(n)
    engine.upload_sequences(seqs)
    got_c = engine.single_sizes("bzip2")
    got_s = engine.pair_sizes("bzip2", xs, ys)
    blocks, smem = engine.stat("bzip2_blocks"), engine.stat("bzip2_smem_blocks")
    want_c = ref_sizes(list(range(n)), [-1] * n, seqs)
    want_s = ref_sizes(list(xs), list(ys), seqs)
    bad = np.flatnonzero(got_s != want_s)
    assert np.array_equal(got_c, want_c), np.flatnonzero(got_c != want_c)
    assert bad.size == 0, [(int(xs[k]), int(ys[k]), int(got_s[k]), int(want_s[k])) for k in bad[:20]]
    return blocks, smem


def _mutate_one(s, pos):
    a = bytearray(s)
    a[pos] = {65: 67, 67: 71, 71: 84, 84: 65}.get(a[pos], 65)
    return bytes(a)


def _no_runs_acgt(n, rng, first=None, avoid_last=None):
    """n ACGT bytes with no two neighbours equal (RLE1 leaves them as they are); `first`: its first byte; `avoid_last`:
    a byte its last one must not be"""
    acgt = np.frombuffer(b"ACGT", np.uint8)
    steps = rng.integers(1, 4, n)
    steps[0] = rng.integers(0, 4) if first is None else int(np.flatnonzero(acgt == first)[0])
    a = acgt[np.cumsum(steps) % 4]
    if avoid_last is not None and n >= 2 and a[-1] == avoid_last:
        a[-1] = next(c for c in acgt if c != avoid_last and c != a[-2])
    return a.tobytes()


@pytest.mark.gpu
def test_repetitive_genomes(engine):
    rng = np.random.default_rng(31)
    unit37, unit3k = _acgt(37, rng), _acgt(3000, rng)
    s = _acgt(400000, rng)
    seqs = [
        (unit37 * (500000 // 37 + 1))[:500000],
        (unit3k * (2500000 // 3000 + 1))[:2500000],
        (b"AC" * 600001)[:1200001],
        (b"ACG" * 400000)[:1100000],
        s[:100000] + b"N" * 10**4 + s[100000:200000] + b"N" * 10**5 + s[200000:] + b"N" * 10**6 + _acgt(50000, rng),
        b"N" * 10**6 + _acgt(3000, rng),
        b"A" * 3000000,
    ]
    blocks, smem = check_all(engine, seqs)
    assert smem < blocks


@pytest.mark.gpu
def test_duplicated_genomes(engine):
    # the pair x.x is a block holding x twice (every long rotation ties with its copy); x.x' with one substitution in
    # x' holds two copies with a common prefix of up to |x| / 2 that do not tie.  2 * 449 990 bytes fit one block,
    # 2 * 449 991 do not.
    rng = np.random.default_rng(32)
    seqs = []
    for n in (12000, 100000, 449990, 449991, 1200000):
        x = _acgt(n, rng)
        seqs += [x, _mutate_one(x, n // 2)]
    xs, ys = [], []
    for k in range(0, len(seqs), 2):
        for a in (k, k + 1):
            for b in (k, k + 1):
                xs.append(a)
                ys.append(b)
    check_all(engine, seqs, np.array(xs, np.int32), np.array(ys, np.int32))


def _junction_corpus():
    """x's of RLE1 length around one and two blocks ending in runs of one byte; y's starting with the same byte"""
    rng = np.random.default_rng(33)
    b = ord("T")
    xs = []
    for target in (MAXB - 3, MAXB + 2, 2 * MAXB + 5):
        for tail in (1, 3, 4, 254, 255, 256, 1000):
            body = _no_runs_acgt(target - len(rle1_run(b, tail)), rng, avoid_last=b)
            xs.append(body + bytes([b]) * tail)
    # RLE1 length exactly MAXB and MAXB + 1 with a one-byte final emission: x's last block alone is that emission
    for target in (MAXB, MAXB + 1):
        for tail in (1, 4):
            xs.append(_no_runs_acgt(target - len(rle1_run(b, tail)), rng, avoid_last=b) + bytes([b]) * tail)
    ys = [_no_runs_acgt(20000, rng, first=ord("G"))]
    for head in (1, 4, 300):
        ys.append(bytes([b]) * head + _no_runs_acgt(20000, rng, first=ord("G")))
    ys.append(bytes([b]) * 5000)                                   # y is one run
    return xs, ys


@pytest.mark.gpu
def test_junction_behind_a_multi_block_x(engine):
    xs_, ys_ = _junction_corpus()
    seqs = xs_ + ys_
    nx = len(xs_)
    jx = np.repeat(np.arange(nx), len(ys_)).astype(np.int32)
    jy = np.tile(np.arange(nx, len(seqs)), nx).astype(np.int32)
    engine.upload_sequences(seqs)
    want_c = ref_sizes(list(range(len(seqs))), [-1] * len(seqs), seqs)
    want_s = ref_sizes(list(jx), list(jy), seqs)
    try:
        for smem in (1, 0):
            for prefix in (1, 0):
                engine.set_option("bzip2_smem", smem)
                engine.set_option("bzip2_prefix", prefix)
                got_c = engine.single_sizes("bzip2")
                got_s = engine.pair_sizes("bzip2", jx, jy)
                bad = np.flatnonzero(got_s != want_s)
                assert np.array_equal(got_c, want_c), (smem, prefix, np.flatnonzero(got_c != want_c))
                assert bad.size == 0, (smem, prefix, [(int(jx[k]), int(jy[k])) for k in bad[:20]])
                if prefix:
                    assert engine.stat("bzip2_prefix_blocks") > 0
    finally:
        engine.set_option("bzip2_smem", 1)
        engine.set_option("bzip2_prefix", 1)


@pytest.mark.gpu
def test_shared_memory_routing_boundary(engine):
    # run-free sequences that start with A and end with C: RLE1 length = input length, also across a junction
    rng = np.random.default_rng(34)

    def seq(n):
        s = _no_runs_acgt(n - 1, rng, first=ord("A"), avoid_last=ord("C"))
        return s + b"C"
    seqs = [seq(SMEM_MAX_N), seq(SMEM_MAX_N + 1), seq(SMEM_MAX_N // 2), seq(SMEM_MAX_N // 2), seq(SMEM_MAX_N // 2 + 1)]
    lens = np.array([len(s) for s in seqs])
    n = len(seqs)
    xs, ys = all_pairs(n)
    engine.upload_sequences(seqs)
    got_c = engine.single_sizes("bzip2")
    assert engine.stat("bzip2_blocks") == n
    assert engine.stat("bzip2_smem_blocks") == int((lens <= SMEM_MAX_N).sum())
    got_s = engine.pair_sizes("bzip2", xs, ys)
    assert engine.stat("bzip2_blocks") == n * n
    assert engine.stat("bzip2_smem_blocks") == int((lens[xs] + lens[ys] <= SMEM_MAX_N).sum())
    assert np.array_equal(got_c, ref_sizes(list(range(n)), [-1] * n, seqs))
    assert np.array_equal(got_s, ref_sizes(list(xs), list(ys), seqs))


@pytest.mark.gpu
def test_more_than_65536_blocks_in_one_call(engine):
    rng = np.random.default_rng(35)
    seqs = [_acgt(int(rng.integers(1000, 3001)), rng) for _ in range(260)]
    n = len(seqs)
    xs, ys = all_pairs(n)
    engine.upload_sequences(seqs)
    got = engine.pair_sizes("bzip2", xs, ys)
    assert engine.stat("bzip2_blocks") > BATCH_BLOCKS
    pick = np.union1d(rng.choice(n * n, 5000, replace=False), np.arange(n) * (n + 1))
    assert np.array_equal(got[pick], ref_sizes(list(xs[pick]), list(ys[pick]), seqs))


def emu_block_lengths(emu, s):
    """RLE1 lengths of the blocks the cut makes of s alone"""
    out = np.zeros(16, np.uint32)
    nb = emu.emu_bz2_block_lengths(s, len(s), out.ctypes.data, out.size)
    assert 0 < nb <= out.size
    return out[:nb].tolist()


def plan_batches(xs, ys, seqs, emu):
    """The blocks of a pair call, in bz_run's order and cut into its batches on the host: for each job, x's closed
    blocks the first time x appears (bzip2_prefix 1, nothing cached), then the rest of the job's blocks.  The closed
    blocks of x are its blocks alone but the last; the job's blocks are those of x.y after them.  Returns
    (batch index of every closed block of each x, batch indices of each job's own blocks, blocks, closed blocks used)."""
    alone = parallel_map(lambda s: emu_block_lengths(emu, s), seqs)
    closed = [b[:-1] for b in alone]
    joined = parallel_map(lambda k: emu_block_lengths(emu, seqs[xs[k]] + seqs[ys[k]]), range(len(xs)))
    batch, nblk, nbytes = 0, 0, 0

    def place(w):
        nonlocal batch, nblk, nbytes
        if nblk == BATCH_BLOCKS or nbytes + w > BATCH_BYTES:
            batch, nblk, nbytes = batch + 1, 0, 0
        nblk += 1
        nbytes += (w + 15) & ~15
        return batch

    closed_batch, job_batches, blocks, used = {}, [], 0, 0
    for k, (x, y) in enumerate(zip(xs, ys)):
        x = int(x)
        if closed[x] and x not in closed_batch:
            closed_batch[x] = [place(w) for w in closed[x]]
        used += len(closed[x])
        assert joined[k][:len(closed[x])] == closed[x]           # x's closed blocks close the same way in x.y
        job_batches.append([place(w) for w in joined[k][len(closed[x]):]])
        blocks += len(job_batches[-1])
    blocks += sum(len(v) for v in closed_batch.values())
    return closed_batch, job_batches, blocks, used


@pytest.mark.gpu
def test_more_than_192_mib_of_blocks_in_one_call(engine, emu):
    # Ten 2.5 Mbp sequences, each two closed blocks and an open tail; one pair call on a fresh upload, so the call
    # itself computes every x's closed blocks.  Jobs go y by y: the first ten jobs compute the closed blocks of all ten
    # x in the first batch, and the jobs of the last y, which add those bits to theirs, finish in a later batch.
    rng = np.random.default_rng(36)
    root = _acgt(2_500_000, rng)
    seqs = []
    for _ in range(10):
        a = np.frombuffer(root, np.uint8).copy()
        k = rng.random(a.size) < 0.01
        a[k] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(k.sum()))]
        seqs.append(a.tobytes())
    n = len(seqs)
    ys, xs = [a.astype(np.int32).ravel() for a in np.divmod(np.arange(n * n), n)]
    closed_batch, job_batches, blocks, used = plan_batches(xs, ys, seqs, emu)
    assert sorted(closed_batch) == list(range(n)) and all(b == [0, 0] for b in closed_batch.values())
    assert max(job_batches[-1]) > 0
    engine.upload_sequences(seqs)
    got = engine.pair_sizes("bzip2", xs, ys)
    assert engine.stat("bzip2_blocks") == blocks
    computed = sum(len(b) for b in closed_batch.values())
    assert engine.stat("bzip2_prefix_blocks") == used - computed      # computed in this call and reused n - 1 times
    assert np.array_equal(got, ref_sizes(list(xs), list(ys), seqs))
    assert np.array_equal(engine.single_sizes("bzip2"), ref_sizes(list(range(n)), [-1] * n, seqs))


@pytest.mark.gpu
def test_caches_across_calls_and_uploads(engine):
    rng = np.random.default_rng(37)
    lens = [1_300_000, 2_000_000, 950_000, 40_000, 7_000, 25_000]

    def corpus():
        return [_acgt(k - 600, rng) + b"T" * 600 for k in lens]
    n = len(lens)
    xs, ys = all_pairs(n)
    first = np.isin(xs, [0, 2, 4])
    seqs = corpus()
    engine.upload_sequences(seqs)
    c = engine.single_sizes("bzip2")
    s1 = engine.pair_sizes("bzip2", xs[first], ys[first])
    s2 = engine.pair_sizes("bzip2", xs[~first], ys[~first])
    assert engine.stat("bzip2_prefix_blocks") > 0                  # x's closed blocks from the singles call
    assert np.array_equal(c, ref_sizes(list(range(n)), [-1] * n, seqs))
    assert np.array_equal(s1, ref_sizes(list(xs[first]), list(ys[first]), seqs))
    assert np.array_equal(s2, ref_sizes(list(xs[~first]), list(ys[~first]), seqs))
    # another corpus of the same shape keeps the device buffers and must forget every cached bit count
    seqs = corpus()
    engine.upload_sequences(seqs)
    want = ref_sizes(list(xs), list(ys), seqs)
    assert np.array_equal(engine.pair_sizes("bzip2", xs, ys), want)
    engine.set_option("invalidate_caches", 1)
    assert np.array_equal(engine.pair_sizes("bzip2", xs, ys), want)
