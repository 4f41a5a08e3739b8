"""bzip2 sizes on the device: pairs/s at the c3 shape (many short sequences, every pair job one block sorted in shared
memory) and at a c4-like sample (few 5 Mbp sequences, 900 kB blocks sorted in global memory), the device time of each
stage, parity against len(bz2.compress(...)) on a sample of the jobs, and the libbz2 rate on all host cores over a
sample of the same jobs.  Prints one JSON line; exits non-zero on a parity mismatch.

    python tools/bench_bzip2.py [--c3-n 1000] [--c4-n 16] [--steps 3] [--warmup 1]
"""
import argparse
import bz2
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from snacc_b200.engine import Engine  # noqa: E402

STAGES = ("bzip2_rle_gather_ms", "bzip2_bwt_small_ms", "bzip2_bwt_large_ms", "bzip2_bits_ms")


def phylogeny(n, length, rate, seed):
    """n sequences that differ from one random root by point substitutions at `rate`"""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    root = acgt[rng.integers(0, 4, length)]
    out = []
    for _ in range(n):
        a = root.copy()
        k = rng.random(length) < rate
        a[k] = acgt[rng.integers(0, 4, int(k.sum()))]
        out.append(a.tobytes())
    return out


def cpu_sizes(seqs, xs, ys, threads):
    def one(k):
        return len(bz2.compress(seqs[xs[k]] + (seqs[ys[k]] if ys[k] >= 0 else b"")))
    with ThreadPoolExecutor(threads) as ex:
        return np.array(list(ex.map(one, range(len(xs)))), dtype=np.int64)


def run_shape(eng, name, seqs, steps, warmup, cpu_jobs, parity_jobs, rng):
    n = len(seqs)
    eng.upload_sequences(seqs)
    res = {"shape": name, "n_seqs": n, "seq_len": len(seqs[0]), "pair_jobs": n * n, "single_jobs": n}
    times, stages, S = [], [], None
    for step in range(warmup + steps):
        eng.set_option("invalidate_caches", 1)
        st = dict.fromkeys(STAGES, 0.0)
        t0 = time.perf_counter()
        C = eng.single_sizes("bzip2")
        for k in STAGES:
            st[k] += eng.stat(k)
        S = eng.tile_sizes("bzip2", 0, n, 0, n)
        dt = time.perf_counter() - t0
        for k in STAGES:
            st[k] += eng.stat(k)
        if step >= warmup:
            times.append(dt)
            stages.append(st)
    res["step_s"] = [round(t, 4) for t in times]
    res["pairs_per_s"] = round(n * n / float(np.median(times)), 1)
    res["stage_ms_median_step"] = {k: round(float(np.median([s[k] for s in stages])), 2) for k in STAGES}
    res["blocks_last_call"] = eng.stat("bzip2_blocks")
    res["smem_blocks_last_call"] = eng.stat("bzip2_smem_blocks")
    # parity: a sample of pairs and every single against the reference call
    k = rng.choice(n * n, min(parity_jobs, n * n), replace=False)
    xs, ys = (k // n).astype(np.int32), (k % n).astype(np.int32)
    threads = os.cpu_count()
    want = cpu_sizes(seqs, xs, ys, threads)
    want_c = cpu_sizes(seqs, np.arange(n), np.full(n, -1), threads)
    res["parity_jobs"] = int(k.size + n)
    res["parity_ok"] = bool(np.array_equal(S.ravel()[k], want) and np.array_equal(C, want_c))
    # libbz2 on all host cores over a sample of the same pair jobs
    k = rng.choice(n * n, min(cpu_jobs, n * n), replace=False)
    t0 = time.perf_counter()
    cpu_sizes(seqs, (k // n).astype(np.int32), (k % n).astype(np.int32), threads)
    cpu_rate = k.size / (time.perf_counter() - t0)
    res["cpu_libbz2_pairs_per_s"] = round(cpu_rate, 1)
    res["cpu_threads"] = threads
    res["speedup_vs_cpu"] = round(res["pairs_per_s"] / cpu_rate, 2)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c3-n", type=int, default=1000)
    ap.add_argument("--c3-len", type=int, default=10700)
    ap.add_argument("--c4-n", type=int, default=16)
    ap.add_argument("--c4-len", type=int, default=5_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    rng = np.random.default_rng(a.seed)
    out = {"bench": "bzip2"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        out["gpu"], out["power_limit"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the numbers are still reported, without the card
        out["gpu"] = f"unknown ({e})"
    with Engine(0) as eng:
        out["c3"] = run_shape(eng, "c3", phylogeny(a.c3_n, a.c3_len, 0.02, a.seed), a.steps, a.warmup,
                              cpu_jobs=4000, parity_jobs=500, rng=rng)
        out["c4"] = run_shape(eng, "c4-like", phylogeny(a.c4_n, a.c4_len, 0.01, a.seed + 1), a.steps, a.warmup,
                              cpu_jobs=2 * os.cpu_count(), parity_jobs=24, rng=rng)
    ok = out["c3"]["parity_ok"] and out["c4"]["parity_ok"]
    out["parity_ok"] = ok
    print(json.dumps(out))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
