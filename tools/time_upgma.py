"""Time the tree step on the device (``snacc_upgma``: metrify + UPGMA) on seeded NCD-like matrices, and check each result
against scipy's linkage bit for bit.

    python tools/time_upgma.py [n ...]          (default: 1000 4000 10000)

Each call is timed on the host clock; ``snacc_upgma`` synchronises its stream before it returns, so the time is the
whole call: the upload of the n x n matrix, the kernels, the download of Z and the host sort.  One warm-up call per
size, then the median and minimum of three.  The matrices are NCD values of integer sizes in a narrow range, so they
have many ties, as real NCD matrices of similar genomes do.  The card's name and power limit are printed with the
table, since a time means little without them.
"""
import subprocess
import sys
import time

import numpy as np
import scipy.cluster.hierarchy
import scipy.spatial.distance

sys.path.insert(0, ".")
from snacc_b200.engine import Engine  # noqa: E402


def ncd_like(n, seed, bias=33):
    """the reference's NCD (pairwise_ncd.py:93-111) of sizes C in [10 000, 10 100) and S = max(C_i, C_j) + 200 .. 259"""
    rng = np.random.default_rng(seed)
    C = rng.integers(10_000, 10_100, n) + bias
    S = np.maximum(C[:, None], C[None, :]) + rng.integers(200, 260, (n, n))
    lo = np.minimum(C[:, None], C[None, :]).astype(np.float64)
    hi = np.maximum(C[:, None], C[None, :]).astype(np.float64)
    return np.minimum((S - lo) / hi, (S.T - lo) / hi)


def scipy_tree(D):
    """the reference's tree step: metrify (misc.py:20-25), then linkage(squareform(D_sym), "average")"""
    D_sym = 0.5 * (D + D.T)
    np.fill_diagonal(D_sym, 0.0)
    return scipy.cluster.hierarchy.linkage(scipy.spatial.distance.squareform(D_sym), method="average")


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"unknown ({e})"


def main():
    sizes = [int(a) for a in sys.argv[1:]] or [1000, 4000, 10000]
    print(f"card: {card()}")
    print("| n | call ms (median of 3) | call ms (min) | scipy linkage ms | Z == scipy (rows that differ) |")
    print("|---|---|---|---|---|")
    with Engine(0) as eng:
        for n in sizes:
            D = ncd_like(n, seed=n)
            eng.upgma(D)                                               # warm-up
            times = []
            for _ in range(3):
                t = time.perf_counter()
                Z = eng.upgma(D)
                times.append((time.perf_counter() - t) * 1e3)
            t = time.perf_counter()
            Zref = scipy_tree(D)
            t_ref = (time.perf_counter() - t) * 1e3
            differ = int((Z != Zref).any(axis=1).sum())
            print(f"| {n} | {np.median(times):.1f} | {min(times):.1f} | {t_ref:.1f} | {differ == 0} ({differ}) |", flush=True)


if __name__ == "__main__":
    main()
