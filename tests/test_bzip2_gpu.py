"""GPU: bzip2 sizes on the device (snacc_b200/csrc/bzip2.cuh) against the reference's own call, len(bz2.compress(...))
(pairwise_ncd.py:76), and against the sizes the unmodified reference produced on the committed fixtures."""
import bz2
import json
import os
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
MAXB = 100000 * 9 - 19


def ref_sizes(xs, ys, seqs):
    """len(bz2.compress(x [+ y])) on all host threads (bz2 releases the GIL)"""
    def one(k):
        x, y = xs[k], ys[k]
        return len(bz2.compress(seqs[x] + (seqs[y] if y >= 0 else b"")))
    with ThreadPoolExecutor(os.cpu_count()) as ex:
        return np.array(list(ex.map(one, range(len(xs)))), dtype=np.int64)


def dna(n, rng, alphabet=b"ACGT"):
    return np.frombuffer(alphabet, np.uint8)[rng.integers(0, len(alphabet), n)].tobytes()


def mutate(s, rate, rng):
    a = np.frombuffer(s, np.uint8).copy()
    k = rng.random(a.size) < rate
    a[k] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(k.sum()))]
    return a.tobytes()


@pytest.fixture(scope="module")
def gold(golden_dir):
    return json.load(open(os.path.join(golden_dir, "reference_sizes_lzma_bzip2.json")))


@pytest.mark.parametrize("rc", [False, True])
def test_fixtures_match_reference_sizes(golden_dir, gold, rc):
    from snacc_b200.pairwise_ncd import ncd_matrix
    want = gold["cases"]["bzip2_rc" if rc else "bzip2"]
    files = [Path(golden_dir) / "fasta" / f for f in gold["files"]]
    labels, C, S, D = ncd_matrix(files, "bzip2", reverse_complement=rc)
    assert (C + gold["bias"]).tolist() == want["C"]
    assert (S + gold["bias"]).tolist() == want["S"]
    assert np.array_equal(D, np.array(want["D"]))


def test_engine_ncd_and_shim(golden_dir, gold, engine):
    from snacc_b200 import fasta
    from snacc_b200.pairwise_ncd import compressed_size
    want = gold["cases"]["bzip2"]
    files = [Path(golden_dir) / "fasta" / f for f in gold["files"]]
    data, so, ro = fasta.load_corpus(files)
    engine.upload(data, so, ro)
    n = len(files)
    C = engine.single_sizes("bzip2")
    xs, ys = np.divmod(np.arange(n * n), n)
    S = engine.pair_sizes("bzip2", xs, ys).reshape(n, n)
    assert np.array_equal(engine.ncd(C, S), np.array(want["D"]))
    assert compressed_size(files[0], "bzip2") == (files[0], want["C"][0])
    assert compressed_size((files[0], files[1]), "bzip2") == ((files[0], files[1]), want["S"][0][1])


def golden_csv(golden_dir, gold, path):
    """the CSV the CLI writes for the golden bzip2 distances, rows in the CLI's file order"""
    from snacc_b200 import cli as gcli
    files = [Path(golden_dir) / "fasta" / f for f in gold["files"]]
    order = gcli.collect_files([str(f) for f in files])
    perm = [[str(f) for f in files].index(str(o)) for o in order]
    D = np.array(gold["cases"]["bzip2"]["D"])[np.ix_(perm, perm)]
    gcli.write_distance_csv(order, D, path)
    return files


def test_cli_csv_matches_the_golden_distances(golden_dir, gold, tmp_path, monkeypatch):
    from click.testing import CliRunner
    from snacc_b200 import cli as gcli
    want = tmp_path / "want.csv"
    files = golden_csv(golden_dir, gold, want)
    out = tmp_path / "dist.csv"
    monkeypatch.chdir(tmp_path)
    r = CliRunner().invoke(gcli.cli, [str(f) for f in files] + ["-o", str(out), "-c", "bzip2", "--no-show-progress"])
    assert r.exit_code == 0, r.output
    assert out.read_text() == want.read_text()


def _check_corpus(engine, seqs, xs, ys, **opts):
    engine.upload_sequences(seqs)
    for k, v in opts.items():
        engine.set_option(k, v)
    try:
        got_c = engine.single_sizes("bzip2")
        got_s = engine.pair_sizes("bzip2", xs, ys)
    finally:
        engine.set_option("bzip2_smem", 1)
        engine.set_option("bzip2_prefix", 1)
    n = len(seqs)
    assert np.array_equal(got_c, ref_sizes(list(range(n)), [-1] * n, seqs))
    assert np.array_equal(got_s, ref_sizes(list(xs), list(ys), seqs))
    return got_c, got_s


def test_boundaries_and_alphabets(engine):
    rng = np.random.default_rng(11)
    seqs = [b"A", b"AC", b"AAAA", b"T" * 255, b"T" * 256, b"G" * 1000 + b"A", dna(24576, rng), dna(24570, rng),
            dna(30000, rng, b"ACGTNRYKM"), dna(5000, rng, b"acgtnACGT"), dna(8000, rng, b"ACDEFGHIKLMNPQRSTVWYX"),
            bytes(range(256)) * 40, b"N" * 3000 + dna(3000, rng) + b"N" * 700, dna(MAXB - 3, rng),
            dna(MAXB + 40000, rng, b"ACGTN")]
    n = len(seqs)
    xs = rng.integers(0, n, 120).astype(np.int32)
    ys = rng.integers(0, n, 120).astype(np.int32)
    _check_corpus(engine, seqs, xs, ys)


def test_switches_give_identical_sizes(engine):
    rng = np.random.default_rng(12)
    base = dna(MAXB + 300000, rng)
    seqs = [mutate(base, 0.01, rng) for _ in range(3)] + [dna(5000, rng), dna(20000, rng), dna(50000, rng)]
    n = len(seqs)
    xs, ys = [a.astype(np.int32).ravel() for a in np.divmod(np.arange(n * n), n)]
    c1, s1 = _check_corpus(engine, seqs, xs, ys)
    assert engine.stat("bzip2_prefix_blocks") > 0
    smem_on = engine.stat("bzip2_smem_blocks")
    assert smem_on > 0
    c2, s2 = _check_corpus(engine, seqs, xs, ys, bzip2_smem=0, bzip2_prefix=0)
    assert engine.stat("bzip2_smem_blocks") == 0 and engine.stat("bzip2_prefix_blocks") == 0
    assert np.array_equal(c1, c2) and np.array_equal(s1, s2)


def test_c3_sample_all_blocks_in_shared_memory(engine):
    rng = np.random.default_rng(13)
    root = dna(10700, rng)
    seqs = [mutate(root, 0.05, rng) for _ in range(64)]
    engine.upload_sequences(seqs)
    xs = rng.integers(0, 64, 3000).astype(np.int32)
    ys = rng.integers(0, 64, 3000).astype(np.int32)
    got = engine.pair_sizes("bzip2", xs, ys)
    assert engine.stat("bzip2_smem_blocks") == engine.stat("bzip2_blocks") == 3000
    pick = rng.choice(3000, 300, replace=False)
    assert np.array_equal(got[pick], ref_sizes(list(xs[pick]), list(ys[pick]), seqs))


def test_multi_block_pairs(engine):
    rng = np.random.default_rng(14)
    root = dna(2_500_000, rng)
    seqs = [mutate(root, 0.02, rng) for _ in range(6)]
    n = len(seqs)
    xs, ys = [a.astype(np.int32).ravel() for a in np.divmod(np.arange(n * n), n)]
    _check_corpus(engine, seqs, xs, ys)
    assert engine.stat("bzip2_prefix_blocks") > 0


@pytest.mark.parametrize("fast", [False, True])
def test_c1_shape_cli(tmp_path, monkeypatch, fast):
    from click.testing import CliRunner
    from snacc_b200 import cli as gcli
    from snacc_b200.sharding import ncd_host
    rng = np.random.default_rng(15)
    root = dna(4_450_000, rng)
    seqs = [mutate(root, 0.03, rng) for _ in range(8)]
    files = []
    for i, s in enumerate(seqs):
        f = tmp_path / f"g{i}.fasta"
        f.write_bytes(b">g%d\n" % i + b"\n".join(s[k:k + 80] for k in range(0, len(s), 80)) + b"\n")
        files.append(f)
    n = len(seqs)
    C = ref_sizes(list(range(n)), [-1] * n, seqs)
    xs, ys = np.divmod(np.arange(n * n), n)
    S = ref_sizes(list(xs), list(ys), seqs).reshape(n, n)
    if fast:
        # --fast-mode computes x.y for i <= j only and mirrors it: the lower triangle never sees the order y.x
        iu = np.triu_indices(n, 1)
        S[(iu[1], iu[0])] = S[iu]
    D = ncd_host(C, S, fast_mode=fast)
    out = tmp_path / "dist.csv"
    monkeypatch.chdir(tmp_path)
    args = [str(f) for f in files] + ["-o", str(out), "-c", "bzip2", "--no-show-progress"]
    r = CliRunner().invoke(gcli.cli, args + (["--fast-mode", "True"] if fast else []))
    assert r.exit_code == 0, r.output
    want = tmp_path / "want.csv"
    gcli.write_distance_csv(files, D, want)
    assert out.read_text() == want.read_text()


def test_two_rank_cli_over_nccl(golden_dir, gold, tmp_path):
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    want = tmp_path / "want.csv"
    files = golden_csv(golden_dir, gold, want)
    root = str(Path(__file__).resolve().parents[1])
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = tmp_path / "dist.csv"
    cmd = [sys.executable, "-m", "snacc_b200.cli", "--gpus", "2"] + [str(f) for f in files] + \
        ["-o", str(out), "-c", "bzip2", "--no-show-progress"]
    r = subprocess.run(cmd, cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert out.read_text() == want.read_text()
