"""GPU (-m gpu): the CUDA path, called through the C ABI (ctypes Engine), against the oracle and the
golden fixtures written by the unmodified reference.  Integer sizes must be identical; NCD bit-exact."""
import json
import os
from pathlib import Path

import numpy as np
import pytest

from oracle import lib as olib
from oracle import snacc_oracle
from oracle.fasta_shim import COMPLEMENT_TABLE
from oracle.make_golden import VECTOR_KINDS, synth_vector

pytestmark = pytest.mark.gpu

ALGOS = ["lz4", "gzip", "zlib"]


def _ref_len(data, algo):
    return olib.ref_compressed_len(data, algo)


@pytest.fixture(scope="module")
def ref_sizes(golden_dir):
    return json.load(open(os.path.join(golden_dir, "reference_sizes.json")))


@pytest.mark.parametrize("case", ["lz4", "lz4_rc", "gzip", "gzip_rc"])
def test_fixture_matrix_equals_reference_golden(engine, golden_dir, ref_sizes, case):
    """all singles + all ordered pairs of the committed FASTA fixtures == what the reference's own
    compressed_size returned (incl. multi-record reverse complement done on the device)"""
    from snacc_b200.pairwise_ncd import ncd_matrix
    algo, rc = case.split("_")[0], case.endswith("_rc")
    files = [Path(golden_dir) / "fasta" / f for f in ref_sizes["files"]]
    labels, C, S, D = ncd_matrix(files, algo, reverse_complement=rc, engine=engine)
    want = ref_sizes["cases"][case]
    assert (C + 33).tolist() == want["C"]
    assert (S + 33).tolist() == want["S"]
    assert np.array_equal(D, np.array(want["D"]))
    assert np.array_equal(engine.ncd(C, S), np.array(want["D"]))


@pytest.mark.parametrize("algo", ["lz4", "gzip"])
def test_fast_mode_computes_the_upper_triangle_only(engine, golden_dir, ref_sizes, algo):
    """--fast-mode True (README flag; SURVEY.md 8a divergence ledger): S(i, j) for i <= j only, mirrored, NCD from that one
    order -- the sizes it does compute are the reference's"""
    from snacc_b200.pairwise_ncd import ncd_matrix
    from snacc_b200.sharding import ncd_host
    files = [Path(golden_dir) / "fasta" / f for f in ref_sizes["files"]]
    n = len(files)
    labels, C, S, D = ncd_matrix(files, algo, fast_mode=True, engine=engine)
    want = ref_sizes["cases"][algo]
    Sref = np.array(want["S"]) - 33
    iu = np.triu_indices(n, 1)
    Sref[(iu[1], iu[0])] = Sref[iu]
    assert (C + 33).tolist() == want["C"]
    assert np.array_equal(S, Sref)
    assert np.array_equal(D, ncd_host(C, Sref, fast_mode=True))


@pytest.mark.parametrize("case", ["lz4", "gzip_rc"])
def test_cli_csv_is_byte_identical_to_reference_cli(golden_dir, tmp_path, case, monkeypatch):
    from click.testing import CliRunner
    from snacc_b200 import cli as gcli
    algo, rc = case.split("_")[0], case.endswith("_rc")
    d = Path(golden_dir) / "fasta"
    files = [str(f) for f in sorted(d.iterdir()) if not f.name.startswith("big")]
    out = tmp_path / "dist.csv"
    monkeypatch.chdir(tmp_path)
    args = files + ["-o", str(out), "-c", algo, "--no-show-progress"] + (["--reverse-compliment", "True"] if rc else [])
    r = CliRunner().invoke(gcli.cli, args)
    assert r.exit_code == 0, r.output
    got = out.read_text().replace(str(d.absolute()) + "/", "")
    assert got == (Path(golden_dir) / f"reference_cli_{case}.csv").read_text()
    assert (tmp_path / "dist.md").exists()


def test_single_job_shim_matches_reference_signature(golden_dir, ref_sizes):
    import snacc_b200
    f = Path(golden_dir) / "fasta" / "g1.fasta"
    g = Path(golden_dir) / "fasta" / "multi.fa"
    i, j = ref_sizes["files"].index("g1.fasta"), ref_sizes["files"].index("multi.fa")
    assert snacc_b200.compressed_size(f, "lz4") == (f, ref_sizes["cases"]["lz4"]["C"][i])
    assert snacc_b200.compressed_size((f, g), "lz4", reverse_complement=True) == ((f, g), ref_sizes["cases"]["lz4_rc"]["S"][i][j])


@pytest.mark.parametrize("algo", ALGOS)
def test_regime_boundaries_and_alphabets(engine, algo):
    """lengths straddling every regime boundary x adversarial alphabets, singles and random pairs"""
    rng = np.random.default_rng(5)
    sizes = [1, 2, 3, 5, 12, 13, 300, 11000, 40000, 65274, 65535, 65536, 65537, 70000, 131072, 140000]
    seqs = [synth_vector(kind, n, 17 * k + n) for k, kind in enumerate(VECTOR_KINDS) for n in sizes
            if not (algo == "gzip" and n > 70000 and kind in ("run", "period", "low", "nrun"))]
    engine.upload_sequences(seqs)
    C = engine.single_sizes(algo)
    ref = np.array([_ref_len(s, algo) for s in seqs])
    assert np.array_equal(C, ref), np.nonzero(C != ref)[0][:10]
    m = 400 if algo == "lz4" else 150
    xs, ys = rng.integers(0, len(seqs), m), rng.integers(0, len(seqs), m)
    S = engine.pair_sizes(algo, xs, ys)
    refp = np.array([_ref_len(np.concatenate([seqs[a], seqs[b]]), algo) for a, b in zip(xs, ys)])
    bad = np.nonzero(S != refp)[0]
    assert bad.size == 0, [(int(xs[b]), int(ys[b]), seqs[xs[b]].size, seqs[ys[b]].size, int(S[b]), int(refp[b])) for b in bad[:5]]


def test_on_device_reverse_complement(engine):
    rng = np.random.default_rng(2)
    alpha = np.frombuffer(b"ACGTacgtNnRYKMSWBDHVUu-*", dtype=np.uint8)
    seqs, recs = [], []
    for i in range(5):
        rl = [int(v) for v in rng.integers(0, 400, size=int(rng.integers(1, 5)))]
        rl[0] += 1
        seqs.append(rng.choice(alpha, size=sum(rl)))
        recs.append(rl)
    engine.upload_sequences(seqs, reverse_complement=True, records=recs)
    for i, (s, rl) in enumerate(zip(seqs, recs)):
        raw, parts, pos = s.tobytes(), [], 0
        for r in rl:
            parts.append(raw[pos:pos + r].translate(COMPLEMENT_TABLE)[::-1])
            pos += r
        assert engine.download_sequence(i).tobytes() == b"".join(parts)


def test_empty_sequence_is_value_error(engine):
    with pytest.raises(ValueError):
        engine.upload_sequences([b"ACGT", b""])


def test_unsupported_codec_is_key_error(engine):
    engine.upload_sequences([b"ACGTACGTACGT"])
    with pytest.raises(KeyError):
        engine.single_sizes("lzma")


@pytest.mark.parametrize("algo", ALGOS)
def test_small_stream_config_sample(engine, algo):
    """c3 shape: dengue-sized (~11 kbp) genomes, random sample of pair jobs + all singles"""
    from snacc_b200 import synth
    g = synth.phylogeny(64, 10700, seed=3)
    engine.upload_sequences(g)
    C = engine.single_sizes(algo)
    assert np.array_equal(C, np.array([_ref_len(s, algo) for s in g]))
    rng = np.random.default_rng(3)
    m = 3000 if algo == "lz4" else 300
    xs, ys = rng.integers(0, 64, m), rng.integers(0, 64, m)
    S = engine.pair_sizes(algo, xs, ys)
    chk = rng.choice(m, size=min(m, 300), replace=False)
    for k in chk:
        assert S[k] == _ref_len(np.concatenate([g[xs[k]], g[ys[k]]]), algo)


def test_full_size_genomes_lz4(engine):
    """c4 shape at full length (5 Mbp): tile of ordered pairs vs the real liblz4, plus the size-independent
    properties: prefix-checkpoint path == from-scratch path (single of a concatenated upload) and
    determinism under a different number of streams in flight."""
    from snacc_b200 import synth
    g = synth.phylogeny(6, 5_000_000, seed=4, n_indels=2)
    engine.upload_sequences(g)
    C = engine.single_sizes("lz4")
    assert np.array_equal(C, np.array([olib.ref_lz4f_size(s) for s in g]))
    S = engine.tile_sizes("lz4", 0, 3, 0, 6)
    ref = np.array([[olib.ref_lz4f_size(np.concatenate([g[i], g[j]])) for j in range(6)] for i in range(3)])
    assert np.array_equal(S, ref)
    engine.set_option("streams_in_flight", 8)
    engine.set_option("invalidate_caches", 1)
    assert np.array_equal(engine.tile_sizes("lz4", 0, 3, 0, 6), ref)
    engine.set_option("streams_in_flight", 0)
    # concatenation uploaded as ONE sequence takes the no-checkpoint route through the same kernel
    engine.upload_sequences([np.concatenate([g[0], g[1]])])
    assert engine.single_sizes("lz4")[0] == ref[0, 1]
    D = engine.ncd(C[:3], S[:, :3])
    assert np.array_equal(D, snacc_oracle.ncd_from_sizes(C[:3], S[:, :3]))


def test_packed_and_bytewise_lz4_paths_agree(engine):
    """the 2-bit tile kernels and the byte-wise kernels are two independent implementations of the same
    frame size; mixed corpus (a sequence with N falls back to the byte-wise path inside the same call)"""
    from snacc_b200 import synth
    g = synth.phylogeny(12, 150000, seed=9) + [synth_vector("nrun", 90000, 5)]
    engine.upload_sequences(g)
    n = len(g)
    S = engine.tile_sizes("lz4", 0, n, 0, n)
    assert engine.stat("packed_jobs") == 144 and engine.stat("bytewise_jobs") == n * n - 144
    engine.set_option("lz4_packed", 0)
    try:
        S2 = engine.tile_sizes("lz4", 0, n, 0, n)
    finally:
        engine.set_option("lz4_packed", 1)
    assert np.array_equal(S, S2)
    chk = np.random.default_rng(1).integers(0, n, size=(40, 2))
    for i, j in chk:
        assert S[i, j] == olib.ref_lz4f_size(np.concatenate([g[i], g[j]]))


def test_megabase_genomes_gzip(engine):
    """c2 shape (scaled to 1.2 Mbp so that zlib finishes in seconds): all singles, a tile of pairs, warm caches"""
    from snacc_b200 import synth
    g = synth.phylogeny(4, 1_200_000, seed=6, n_indels=2)
    engine.upload_sequences(g)
    C = engine.single_sizes("gzip")
    assert np.array_equal(C, np.array([_ref_len(s, "gzip") for s in g]))
    S = engine.tile_sizes("gzip", 0, 2, 0, 4)
    ref = np.array([[_ref_len(np.concatenate([g[i], g[j]]), "gzip") for j in range(4)] for i in range(2)])
    assert np.array_equal(S, ref)
    assert np.array_equal(engine.tile_sizes("gzip", 0, 2, 0, 4), ref)          # checkpoints and tables reused
    engine.set_option("invalidate_caches", 1)
    assert np.array_equal(engine.tile_sizes("gzip", 0, 2, 0, 4), ref)          # and rebuilt
    assert engine.stat("deflate_serial_jobs") == 0                             # every pair stream used the canonical stream of y
    engine.set_option("deflate_canonical", 0)                                  # the full serial parse gives the same sizes
    try:
        assert np.array_equal(engine.tile_sizes("gzip", 0, 2, 0, 4), ref)
    finally:
        engine.set_option("deflate_canonical", 1)
    engine.set_option("deflate_junction", 2)                                   # general junction walk instead of the smem kernel
    try:
        assert np.array_equal(engine.tile_sizes("gzip", 0, 2, 0, 4), ref)
    finally:
        engine.set_option("deflate_junction", 3)
    engine.set_option("deflate_index6", 0)                                     # match tables from the 3-byte chain walk only
    engine.set_option("invalidate_caches", 1)
    try:
        assert np.array_equal(engine.tile_sizes("gzip", 0, 2, 0, 4), ref)
        assert np.array_equal(engine.single_sizes("gzip"), C)
    finally:
        engine.set_option("deflate_index6", 1)
        engine.set_option("invalidate_caches", 1)
    Sz = engine.tile_sizes("zlib", 1, 2, 0, 3)
    refz = np.array([[_ref_len(np.concatenate([g[i], g[j]]), "zlib") for j in range(3)] for i in (1, 2)])
    assert np.array_equal(Sz, refz)
    assert np.array_equal(engine.single_sizes("zlib"), np.array([_ref_len(s, "zlib") for s in g]))


def test_full_size_genomes_gzip(engine):
    """c5 shape: 5 Mbp genomes, gzip level 9 -- every shortcut of the deflate path at full size (≈ 50 blocks per stream,
    ≈ 35 of them taken from the canonical symbol stream, several window slides inside the junction) against zlib 1.3
    run on all host cores; and the same sizes with the shortcuts switched off"""
    from snacc_b200 import synth
    g = synth.phylogeny(3, 5_000_000, seed=5)
    n = len(g)
    engine.upload_sequences(g)
    C = engine.single_sizes("gzip")
    S = engine.tile_sizes("gzip", 0, n, 0, n)
    assert engine.stat("deflate_serial_jobs") == 0
    corpus = np.concatenate(g)
    so = np.zeros(n + 1, dtype=np.uint64)
    so[1:] = np.cumsum([x.size for x in g])
    xs = np.concatenate([np.repeat(np.arange(n, dtype=np.int32), n), np.arange(n, dtype=np.int32)])
    ys = np.concatenate([np.tile(np.arange(n, dtype=np.int32), n), np.full(n, -1, dtype=np.int32)])      # y < 0: x alone
    threads = len(os.sched_getaffinity(0))
    sizes = olib.ref_batch_sizes(corpus, so, xs, ys, "gzip", threads)
    ref = sizes[:n * n].reshape(n, n)
    assert np.array_equal(S, ref)
    assert np.array_equal(C, sizes[n * n:])
    for opt in ("deflate_canonical", "deflate_index6"):
        engine.set_option(opt, 0)
        engine.set_option("invalidate_caches", 1)
        try:
            assert np.array_equal(engine.tile_sizes("gzip", 0, 2, 0, n), ref[:2])
        finally:
            engine.set_option(opt, 1)
    engine.set_option("invalidate_caches", 1)


@pytest.mark.parametrize("algo", ALGOS)
def test_repetitive_inputs(engine, algo):
    """single-base runs of 40-60 k, a 37-base tandem repeat, a 3 kbp unit repeated, N runs: one hash bucket holds almost
    every position (radix sort, head/tail packs, chain limits, nice_length stops, LZ4 matches of tens of kilobases)"""
    rng = np.random.default_rng(3)

    def dna(n):
        return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)]

    unit, u2 = dna(37), dna(3000)
    seqs = [np.concatenate([np.full(40000, 65, np.uint8), dna(20000)]),
            np.concatenate([dna(5000), np.full(60000, 65, np.uint8), dna(30000)]),
            np.tile(unit, 2000), np.tile(unit, 2500), np.tile(u2, 20),
            np.concatenate([np.tile(u2, 15), dna(40000)]),
            np.concatenate([np.full(3000, 78, np.uint8), dna(60000), np.full(200, 78, np.uint8), dna(20000)])]
    n = len(seqs)
    engine.upload_sequences(seqs)
    C = engine.single_sizes(algo)
    S = engine.tile_sizes(algo, 0, n, 0, n)
    assert np.array_equal(C, np.array([_ref_len(s, algo) for s in seqs]))
    ref = np.array([[_ref_len(np.concatenate([a, b]), algo) for b in seqs] for a in seqs])
    assert np.array_equal(S, ref)


def test_lz4_stale_table_slots(engine):
    """A/T-only stretches of 66 k - 300 k bases between ACGT stretches: slots of k-mers with C/G age far beyond the
    131072 positions the 17-bit slot encoding can tell apart; the rolling sweep must have retired them"""
    from snacc_b200 import synth
    seqs = []
    for seed in range(3):
        x, y = synth.stale_slot_stream(seed)
        seqs += [x, y]
    engine.upload_sequences(seqs)
    n = len(seqs)
    S = engine.tile_sizes("lz4", 0, n, 0, n)
    assert engine.stat("packed_jobs") == n * n
    ref = np.array([[olib.ref_lz4f_size(np.concatenate([a, b])) for b in seqs] for a in seqs])
    assert np.array_equal(S, ref)


# ---- the parity contract of BASELINE.md section 3 / SURVEY.md 8d at the named shapes --------------------------------------
def _ref_jobs(seqs, xs, ys, algo):
    """real liblz4 / zlib on all host cores: jobs (xs[k], ys[k]); ys[k] < 0 = xs[k] alone"""
    corpus = np.concatenate(seqs)
    so = np.zeros(len(seqs) + 1, dtype=np.uint64)
    so[1:] = np.cumsum([s.size for s in seqs])
    return olib.ref_batch_sizes(corpus, so, np.asarray(xs, np.int32), np.asarray(ys, np.int32), algo,
                                len(os.sched_getaffinity(0)))


def _write_fasta_records(path, records, width=70):
    with open(path, "wb") as fh:
        for k, seq in enumerate(records):
            fh.write(b">contig_%d some description\n" % k)
            full = seq.size // width
            body = np.empty((full, width + 1), dtype=np.uint8)
            body[:, :width] = seq[:full * width].reshape(full, width)
            body[:, width] = 10
            body.tofile(fh)
            if seq.size > full * width:
                fh.write(seq[full * width:].tobytes() + b"\n")


@pytest.fixture(scope="module")
def mystery_genomes(tmp_path_factory):
    """stand-ins for the reference's missing test_dataset/mysteryGenome_1..8.fasta (SURVEY.md 0.7): 8 related genomes of
    ~4.45 Mbp (the Demo notebook's sizes); two of the files hold several records (per-record reverse complement)"""
    from snacc_b200 import synth
    d = tmp_path_factory.mktemp("mystery")
    g = synth.phylogeny(8, 4_450_000, seed=1, n_indels=3)
    files, recs = [], []
    for i, seq in enumerate(g):
        cuts = [0, seq.size] if i not in (2, 5) else [0, 1_000_003, 1_000_003, 3_200_000, seq.size]   # incl. an empty record
        parts = [seq[a:b] for a, b in zip(cuts[:-1], cuts[1:])]
        p = d / f"mysteryGenome_{i + 1}.fasta"
        _write_fasta_records(p, parts)
        files.append(p)
        recs.append(parts)
    return d, files, recs


@pytest.mark.parametrize("case", ["c1_lz4", "c2_gzip_rc"])
def test_config_c1_c2_cli_csv_at_the_named_shape(mystery_genomes, tmp_path, monkeypatch, case):
    """BASELINE.json configs[0] / configs[1]: mysteryGenome_1..8 (8 x ~4.45 Mbp) through the CLI, `-c lz4` and `-c gzip
    --reverse-compliment True`: CSV byte-identical to the reference route (cli.py:104-142 restated: real liblz4 / zlib
    sizes -> compute_distance -> pandas pivot -> to_csv), all 8 + 64 sizes equal"""
    from click.testing import CliRunner
    from snacc_b200 import cli as gcli
    from snacc_b200.pairwise_ncd import ncd_matrix
    d, files, recs = mystery_genomes
    algo, rc = ("lz4", False) if case == "c1_lz4" else ("gzip", True)
    seqs = []
    for parts in recs:
        if rc:
            parts = [np.frombuffer(p.tobytes().translate(COMPLEMENT_TABLE)[::-1], dtype=np.uint8) for p in parts]
        seqs.append(np.concatenate(parts))
    n = len(seqs)
    xs = np.concatenate([np.repeat(np.arange(n), n), np.arange(n)])
    ys = np.concatenate([np.tile(np.arange(n), n), np.full(n, -1)])
    ref = _ref_jobs(seqs, xs, ys, algo)
    Sref, Cref = ref[:n * n].reshape(n, n), ref[n * n:]
    out = tmp_path / "dist.csv"
    monkeypatch.chdir(tmp_path)
    args = [str(d), "-o", str(out), "-c", algo, "--no-show-progress"] + (["--reverse-compliment", "True"] if rc else [])
    r = CliRunner().invoke(gcli.cli, args)
    assert r.exit_code == 0, r.output
    want = tmp_path / "want.csv"
    order = snacc_oracle.sorted_files([d])
    assert [p.name for p in order] == [f"mysteryGenome_{i}.fasta" for i in range(1, 9)]
    snacc_oracle.write_csv(order, snacc_oracle.ncd_from_sizes(Cref, Sref), want)
    assert out.read_bytes() == want.read_bytes()
    log = (tmp_path / "dist.md").read_text()
    assert f"* Compression method: {algo}" in log and f"* Reverse complement: {rc}" in log
    assert all(f"* {p}" in log for p in order)
    labels, C, S, D = ncd_matrix(order, algo, reverse_complement=rc)
    assert np.array_equal(C, Cref) and np.array_equal(S, Sref)


def test_config_c3_sample_of_ten_thousand_jobs(engine):
    """c3 shape (BASELINE.json configs[2]): dengue-sized genomes, single-block LZ4 regime, rectangle mode; >= 10^4 of the
    pair jobs and all singles against the real liblz4 (SURVEY.md 8d)"""
    from snacc_b200 import synth
    g = synth.phylogeny(160, 10700, seed=3)
    n = len(g)
    engine.upload_sequences(g)
    C = engine.single_sizes("lz4")
    S = engine.tile_sizes("lz4", 0, n, 0, n)
    assert engine.stat("packed_jobs") == n * n
    rng = np.random.default_rng(3)
    k = rng.choice(n * n, size=12000, replace=False)
    xs, ys = k // n, k % n
    ref = _ref_jobs(g, np.concatenate([xs, np.arange(n)]), np.concatenate([ys, np.full(n, -1)]), "lz4")
    assert np.array_equal(S[xs, ys], ref[:k.size])
    assert np.array_equal(C, ref[k.size:])


def test_config_c4_sample_of_256_jobs(engine):
    """c4 shape: 5 Mbp genomes, linked LZ4 regime; >= 256 sampled ordered pair jobs + all singles against the real liblz4"""
    from snacc_b200 import synth
    g = synth.phylogeny(20, 5_000_000, seed=4, n_indels=2)
    n = len(g)
    engine.upload_sequences(g)
    C = engine.single_sizes("lz4")
    S = engine.tile_sizes("lz4", 0, n, 0, n)
    assert engine.stat("packed_jobs") == n * n and engine.stat("bytewise_jobs") == 0
    rng = np.random.default_rng(4)
    k = rng.choice(n * n, size=300, replace=False)
    xs, ys = k // n, k % n
    ref = _ref_jobs(g, np.concatenate([xs, np.arange(n)]), np.concatenate([ys, np.full(n, -1)]), "lz4")
    assert np.array_equal(S[xs, ys], ref[:k.size])
    assert np.array_equal(C, ref[k.size:])


def test_config_c5_sample_of_64_gzip_jobs(engine):
    """c5 shape: 5 Mbp genomes, gzip level 9, both orders; >= 64 sampled ordered pair jobs + singles against zlib 1.3"""
    from snacc_b200 import synth
    g = synth.phylogeny(10, 5_000_000, seed=5)
    n = len(g)
    engine.upload_sequences(g)
    C = engine.single_sizes("gzip")
    S = engine.tile_sizes("gzip", 0, n, 0, n)
    assert engine.stat("deflate_serial_jobs") == 0
    rng = np.random.default_rng(5)
    k = rng.choice(n * n, size=66, replace=False)
    xs, ys = k // n, k % n
    ref = _ref_jobs(g, np.concatenate([xs, np.arange(4)]), np.concatenate([ys, np.full(4, -1)]), "gzip")
    assert np.array_equal(S[xs, ys], ref[:k.size])
    assert np.array_equal(C[:4], ref[k.size:])
    assert np.array_equal(S, S.T) is False or n == 1          # both orders are really computed (asymmetric sizes)


# ---- the product's multi-GPU path on hardware (needs 2 GPUs) ------------------------------------------------------------
def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("launcher", ["torchrun", "gpus_flag"])
def test_two_rank_cli_over_nccl(golden_dir, tmp_path, launcher):
    """`python -m torch.distributed.run --nproc-per-node 2 -m snacc_b200.cli ...` and `snacc --gpus 2`: every rank parses
    its band of the files, NCCL all-gather of the corpus, column bands, one writer; CSV byte-identical to the reference
    CLI's, for the reference semantics and for --fast-mode"""
    import subprocess
    import sys
    if _n_gpus() < 2:
        pytest.skip("needs two GPUs")
    d = Path(golden_dir) / "fasta"
    files = [str(f) for f in sorted(d.iterdir()) if not f.name.startswith("big")]
    root = str(Path(__file__).resolve().parents[1])
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    for fast in (False, True):
        out = tmp_path / f"dist_{launcher}_{int(fast)}.csv"
        tail = files + ["-o", str(out), "-c", "lz4", "--no-show-progress"] + (["--fast-mode", "True"] if fast else [])
        if launcher == "torchrun":
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--standalone",
                   "--local-addr", "127.0.0.1", "-m", "snacc_b200.cli"] + tail
        else:
            cmd = [sys.executable, "-m", "snacc_b200.cli", "--gpus", "2"] + tail
        r = subprocess.run(cmd, cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        got = out.read_text().replace(str(d.absolute()) + "/", "")
        if not fast:
            assert got == (Path(golden_dir) / "reference_cli_lz4.csv").read_text()
        else:
            from snacc_b200.pairwise_ncd import ncd_matrix
            from snacc_b200 import cli as gcli
            labels, C, S, D = ncd_matrix([Path(f) for f in files], "lz4", fast_mode=True)
            want = tmp_path / "want_fast.csv"
            gcli.write_distance_csv([Path(f) for f in files], D, want)
            assert out.read_text() == want.read_text()
        assert (tmp_path / (out.stem + ".md")).exists()


def test_two_rank_matrix_at_scale_over_nccl(tmp_path):
    """2 ranks, 12 x 1.5 Mbp genomes: sharded corpus load + NCCL all-gather + column bands == the single-GPU result,
    lz4 and gzip"""
    import subprocess
    import sys
    if _n_gpus() < 2:
        pytest.skip("needs two GPUs")
    from snacc_b200 import synth
    from snacc_b200.pairwise_ncd import ncd_matrix
    g = synth.phylogeny(12, 1_500_000, seed=8)
    files = []
    for i, s in enumerate(g):
        p = tmp_path / f"g{i:02d}.fa"
        _write_fasta_records(p, [s])
        files.append(p)
    for algo in ("lz4", "gzip"):
        _, C1, S1, D1 = ncd_matrix(files, algo, reverse_complement=True)
        _, C2, S2, D2 = ncd_matrix(files, algo, reverse_complement=True, gpus=2)
        assert np.array_equal(C1, C2) and np.array_equal(S1, S2) and np.array_equal(D1, D2)


@pytest.mark.parametrize("algo", ["gzip", "zlib"])
def test_deflate_prefix_records_exchange(engine, algo):
    """what the multi-GPU path does for the deflate codecs, on one GPU: sequences prepared 'elsewhere' enter only as
    imported prefix records (checkpoint + size); pair streams x.y with such an x, and the singles, equal zlib's"""
    from snacc_b200 import synth
    g = synth.phylogeny(6, 400_000, seed=11) + [synth_vector("dna", 70000, 3), synth_vector("dna", 200, 4)]
    n = len(g)
    engine.upload_sequences(g)
    assert engine.prefix_record_bytes(algo) > 0 and engine.prefix_record_bytes("lz4") == 0
    theirs = np.array([0, 2, 4, 6, 7], dtype=np.int32)            # "prepared by another rank"
    mine = np.array([1, 3, 5], dtype=np.int32)
    engine.single_sizes(algo, theirs)
    recs = engine.export_prefix(algo, theirs)
    engine.set_option("invalidate_caches", 1)
    engine.import_prefix(algo, theirs, recs)
    C = engine.single_sizes(algo)                                  # theirs: from the records; mine: parsed here
    assert np.array_equal(C, np.array([_ref_len(s, algo) for s in g]))
    xs, ys = np.repeat(np.arange(n), mine.size), np.tile(mine, n)  # all x against my y
    S = engine.pair_sizes(algo, xs, ys)
    ref = np.array([_ref_len(np.concatenate([g[a], g[b]]), algo) for a, b in zip(xs, ys)])
    assert np.array_equal(S, ref)
    # the same with the whole 3-byte index for the x-only sequences (default: their last 40 KiB only), and then a
    # sequence that was x-only becomes a y (its index is rebuilt whole)
    try:
        engine.set_option("invalidate_caches", 1)
        engine.set_option("deflate_tail_index", 0)
        engine.import_prefix(algo, theirs, recs)
        assert np.array_equal(engine.pair_sizes(algo, xs, ys), ref)
    finally:
        engine.set_option("deflate_tail_index", 1)
    engine.set_option("invalidate_caches", 1)
    engine.import_prefix(algo, theirs, recs)
    assert np.array_equal(engine.pair_sizes(algo, xs, ys), ref)
    xs2, ys2 = np.arange(n), np.full(n, 0)                        # sequence 0 (x-only so far) as y
    ref2 = np.array([_ref_len(np.concatenate([g[a], g[0]]), algo) for a in xs2])
    assert np.array_equal(engine.pair_sizes(algo, xs2, ys2), ref2)
    assert np.array_equal(engine.pair_sizes(algo, xs, ys), ref)
    engine.set_option("invalidate_caches", 1)


@pytest.mark.parametrize("algo", ["gzip", "zlib"])
def test_deflate_sequence_alone_in_parallel_chunks(engine, algo):
    """the sequence-alone products (size, checkpoint, canonical stream) from the chunked path (dfl_chunk_*_kernel +
    dfl_alone_kernel) and from the serial kernel are the same bytes: sizes == zlib, prefix records identical, and pair
    streams built on either equal zlib's; periodic inputs that the chunked path gives up still come out right"""
    from snacc_b200 import synth
    g = synth.phylogeny(5, 700_000, seed=12) + [synth_vector("dna", 140_000, 3), synth_vector("dna", 90_000, 4),
                                                np.tile(synth_vector("dna", 517, 5), 600), synth_vector("run", 300_000, 6)]
    n = len(g)
    engine.upload_sequences(g)
    allseq = np.arange(n, dtype=np.int32)
    ref_c = np.array([_ref_len(s, algo) for s in g])
    out = {}
    try:
        for mode in (1, 0):
            engine.set_option("invalidate_caches", 1)
            engine.set_option("deflate_parallel_prep", mode)
            C = engine.single_sizes(algo)
            assert np.array_equal(C, ref_c), (mode, np.flatnonzero(C != ref_c).tolist())
            stood = engine.stat("deflate_parallel_prep_seqs")
            assert (stood >= 6) if mode else (stood == 0), (mode, stood)
            xs, ys = np.repeat(allseq, 3), np.tile(np.array([0, 5, 7], dtype=np.int32), n)
            out[mode] = (engine.export_prefix(algo, allseq).copy(), engine.pair_sizes(algo, xs, ys))
    finally:
        engine.set_option("deflate_parallel_prep", 1)
        engine.set_option("invalidate_caches", 1)
    assert np.array_equal(out[0][0], out[1][0])
    assert np.array_equal(out[0][1], out[1][1])
    ref = np.array([_ref_len(np.concatenate([g[a], g[b]]), algo) for a, b in zip(xs, ys)])
    assert np.array_equal(out[1][1], ref)


def _sprinkle(seq, rate, seed, alt=b"NNNNRYKMSWacgtn", runs=3):
    """what real assemblies contain: a fraction `rate` of the bases replaced by N / IUPAC / lower-case bytes, a few N runs"""
    rng = np.random.default_rng(seed)
    s = np.array(seq, dtype=np.uint8, copy=True)
    m = rng.random(s.size) < rate
    s[m] = np.frombuffer(alt, dtype=np.uint8)[rng.integers(0, len(alt), int(m.sum()))]
    for _ in range(runs):
        a = int(rng.integers(0, max(1, s.size - 1)))
        s[a:a + int(rng.integers(1, 400))] = ord("N")
    return s


def test_lz4_sequences_with_sparse_non_alphabet_bytes_stay_on_the_tile_kernels(engine):
    """VERDICT r1 'cliff': an N / IUPAC code / soft-masked base no longer sends a genome to the byte-wise kernel.  Flagged
    bases are crossed with byte-exact steps (pk_step_exact), candidates whose window holds one get a forced mismatch, k-mers
    with such bytes live in the overflow table: sizes equal liblz4's for every pair, and the jobs stay 'packed'"""
    from snacc_b200 import synth
    g = synth.phylogeny(8, 150000, seed=9)
    seqs = [_sprinkle(s, r, 40 + i) for i, (s, r) in enumerate(zip(g, [1e-4, 1e-4, 1e-3, 0, 3e-3, 1e-5, 0, 1e-4]))]
    seqs[1][-2:] = ord("N"); seqs[2][:3] = ord("n"); seqs[4][65530:65541] = ord("N"); seqs[5][131071] = ord("R")
    seqs += [_sprinkle(synth.phylogeny(1, 30000, seed=3)[0], 1e-3, 77),       # flagged and shorter than a block
             synth_vector("nrun", 90000, 5)]                                  # 10 % N: too dense, byte-wise
    n = len(seqs)
    engine.upload_sequences(seqs)
    C = engine.single_sizes("lz4")
    assert np.array_equal(C, np.array([olib.ref_lz4f_size(s) for s in seqs]))
    S = engine.tile_sizes("lz4", 0, n, 0, n)
    ref = _ref_jobs(seqs, np.repeat(np.arange(n), n), np.tile(np.arange(n), n), "lz4").reshape(n, n)
    assert np.array_equal(S, ref), np.argwhere(S != ref)[:10].tolist()
    # only the jobs touching the dense sequence (and the single-block pair of the short one with itself) are byte-wise
    assert engine.stat("bytewise_jobs") <= 2 * n + 1 and engine.stat("packed_jobs") >= (n - 1) * (n - 1) - 1
    engine.set_option("lz4_packed", 0)
    try:
        assert np.array_equal(engine.tile_sizes("lz4", 0, n, 0, n), ref)
    finally:
        engine.set_option("lz4_packed", 1)


def test_lz4_full_size_genomes_with_flagged_bases(engine):
    """c4 shape with 1e-4 of the bases outside the alphabet: every job on the tile kernels, sizes == liblz4"""
    from snacc_b200 import synth
    g = [_sprinkle(s, 1e-4, 60 + i, runs=6) for i, s in enumerate(synth.phylogeny(5, 5_000_000, seed=4, n_indels=2))]
    n = len(g)
    engine.upload_sequences(g)
    C = engine.single_sizes("lz4")
    S = engine.tile_sizes("lz4", 0, n, 0, n)
    assert engine.stat("packed_jobs") == n * n and engine.stat("bytewise_jobs") == 0
    ref = _ref_jobs(g, np.concatenate([np.repeat(np.arange(n), n), np.arange(n)]),
                    np.concatenate([np.tile(np.arange(n), n), np.full(n, -1)]), "lz4")
    assert np.array_equal(S, ref[:n * n].reshape(n, n))
    assert np.array_equal(C, ref[n * n:])


@pytest.mark.parametrize("flagged", [False, True])
def test_lz4_tile_segments(engine, flagged):
    """Tiles of the linked pair kernel cut into segments that different CTAs continue (PkSegStore, option lz4_segments):
    sizes == liblz4 for every pair, with mixed lengths (different numbers of ring states per tile), with and without
    flagged bases (their overflow tables then persist per stream)"""
    from snacc_b200 import synth
    g = synth.phylogeny(7, 600000, seed=21) + synth.phylogeny(4, 331000, seed=22)
    if flagged:
        g = [_sprinkle(s, 1e-4, 90 + i) for i, s in enumerate(g)]
    n = len(g)
    engine.upload_sequences(g)
    engine.single_sizes("lz4")
    ref = _ref_jobs(g, np.repeat(np.arange(n), n), np.tile(np.arange(n), n), "lz4").reshape(n, n)
    try:
        for k in (3, 2, 8):
            engine.set_option("lz4_segments", k)
            S = engine.tile_sizes("lz4", 0, n, 0, n)
            assert np.array_equal(S, ref), (k, np.argwhere(S != ref)[:10].tolist())
            assert engine.stat("lz4_segments") == min(k, 4)       # 331 kbp = 8 ring states: at most 4 segments
            assert engine.stat("packed_jobs") == n * n
    finally:
        engine.set_option("lz4_segments", 0)


@pytest.mark.parametrize("n", [2, 3, 8, 97, 600])
def test_metrify_and_upgma_on_the_device_equal_scipy(engine, n):
    """SURVEY.md 8f rank 4: metrify (misc.py:20-25) + UPGMA (distmatrix_to_tree.py:9-15) on the device: scipy's linkage
    matrix bit for bit (ids, heights and leaf counts) and the reference's Newick string byte for byte"""
    from oracle import tree_oracle
    from snacc_b200 import distmatrix_to_tree as d2t
    rng = np.random.default_rng(n)
    pts = rng.random((n, 6))
    D = np.sqrt(((pts[:, None, :] - pts[None, :, :]) ** 2).sum(-1)) * (1 + 0.05 * rng.random((n, n)))   # asymmetric, NCD-like
    np.fill_diagonal(D, 0.9 + 0.1 * rng.random(n))                                                    # non-zero diagonal
    Zref = tree_oracle.hierarchical(tree_oracle.metrify(D))
    Z = d2t.linkage_from_distances(D, engine=engine)
    assert np.array_equal(Z, Zref)
    assert np.array_equal(d2t.hierarchical(tree_oracle.metrify(D), engine=engine), Z)
    names = [f"genome_{i}.fasta" for i in range(n)]
    assert d2t.newick_from_linkage(Z, names) == tree_oracle.newick(Zref, names)


def test_tree_from_the_cli_csv(engine, golden_dir, tmp_path):
    """distmatrix_to_tree.main on the CSV the CLI writes (the on-disk contract, cli.py:138-142 -> misc.py:15-17)"""
    from oracle import tree_oracle
    from snacc_b200 import distmatrix_to_tree as d2t
    from snacc_b200.misc import read_dist_values_names
    csv = Path(golden_dir) / "reference_cli_lz4.csv"
    out = tmp_path / "tree.nwk"
    d2t.main(str(csv), None, str(out))
    names, D = read_dist_values_names(str(csv))
    assert out.read_text() == tree_oracle.newick(tree_oracle.hierarchical(tree_oracle.metrify(D)), names)
