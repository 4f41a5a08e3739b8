"""gzip / zlib NCD matrices whose deflate state does not fit in device memory at once, on one GPU.

Runs what `ncd_matrix` runs on one GPU once the corpus is uploaded -- `sharding.sizes_matrix` (C(i) of every sequence,
then every ordered pair) and the float64 NCD epilogue (`Engine.ncd`) -- on seeded synthetic genomes generated on the
device (uploaded device to device instead of parsed from 20 GB of FASTA).  The shapes:

  gzip, 4 096 x 5 Mbp   ~250 GB of deflate state if every sequence were prepared at once
  zlib, 2 048 x 5 Mbp   (the c5 corpus of bench.py) ~191 GB likewise

For each: bands, peak deflate state bytes and full preparations of every library call, wall time, pairs/s, and
parity of a seeded sample of 64 pair jobs and 16 singles against zlib (Python's module, on all host cores).  The card's name, power limit and
free / total memory are read in the same run.

    python tools/deflate_beyond_memory.py --out profiles/r04_deflate_beyond_memory_n1.json [--shape gzip:4096 ...]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

GENOME_LEN = 5_000_000
LEVEL = {"gzip": (9, 18), "zlib": (6, 6)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,memory.total,memory.free", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, total, free = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "memory_total": total, "memory_free": free}


def zlib_size(data, algo):
    level, wrapper = LEVEL[algo]
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, zlib.Z_DEFAULT_STRATEGY)
    return len(c.compress(data) + c.flush()) + wrapper


def run_shape(algo, n, seed, n_pairs, n_singles):
    import torch
    from snacc_b200 import sharding, synth
    from snacc_b200.engine import Engine
    dev = torch.device("cuda", 0)
    t0 = time.perf_counter()
    genomes = synth.phylogeny_torch(n, GENOME_LEN, seed, dev)
    lengths = np.array([g.numel() for g in genomes], dtype=np.int64)
    so = np.zeros(n + 1, dtype=np.uint64)
    so[1:] = np.cumsum(lengths)
    corpus = torch.cat(genomes)
    del genomes
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    rep = {"codec": algo, "n": n, "genome_len": GENOME_LEN, "corpus_bytes": int(so[-1]), "seed": seed,
           "generate_s": round(gen_s, 1)}
    with Engine(0) as eng:
        eng.upload_device(corpus.data_ptr(), so)
        del corpus
        torch.cuda.empty_cache()
        free, total = torch.cuda.mem_get_info(0)
        rep["device_free_before"], rep["device_total"] = int(free), int(total)
        # the deflate statistics of every library call sizes_matrix makes (the instance's methods, wrapped)
        rep["calls"] = []
        for name in ("single_sizes", "tile_sizes", "pair_sizes"):
            def wrapped(*a, _f=getattr(eng, name), _name=name, **k):
                t = time.perf_counter()
                r = _f(*a, **k)
                rep["calls"].append({"call": _name, "s": round(time.perf_counter() - t, 2),
                                     **{s: int(eng.stat("deflate_" + s)) for s in
                                        ("bands", "state_bytes", "prepared_seqs", "serial_jobs")}})
                return r
            setattr(eng, name, wrapped)
        t0 = time.perf_counter()
        C, S = sharding.sizes_matrix(eng, algo)
        t2 = time.perf_counter()
        D = eng.ncd(C, S)
        t3 = time.perf_counter()
        rep["sizes_matrix_s"] = round(t2 - t0, 2)
        rep["ncd_s"] = round(t3 - t2, 2)
        rep["wall_s"] = round(t3 - t0, 2)
        rep["pairs_per_s"] = round(n * n / (t3 - t0), 1)
        rep["finite"] = bool(np.isfinite(D).all())
        # parity on a seeded sample against zlib on all host cores
        rng = np.random.default_rng(seed + 1)
        jobs = rng.integers(0, n, size=(n_pairs, 2))
        singles = rng.choice(n, size=n_singles, replace=False)
        need = sorted(set(jobs.ravel().tolist()) | set(singles.tolist()))
        host = {i: eng.download_sequence(i).tobytes() for i in need}
    t4 = time.perf_counter()
    with ThreadPoolExecutor(os.cpu_count()) as ex:             # zlib releases the GIL
        ref_p = list(ex.map(lambda j: zlib_size(host[j[0]] + host[j[1]], algo), jobs.tolist()))
        ref_s = list(ex.map(lambda i: zlib_size(host[i], algo), singles.tolist()))
    rep["parity"] = {"pair_jobs": n_pairs, "singles": n_singles, "host_cores": os.cpu_count(),
                     "host_s": round(time.perf_counter() - t4, 1),
                     "pairs_equal": bool(np.array_equal(S[jobs[:, 0], jobs[:, 1]], np.array(ref_p))),
                     "singles_equal": bool(np.array_equal(C[singles], np.array(ref_s)))}
    return rep


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON report path")
    ap.add_argument("--shape", action="append", default=[], help="codec:n_genomes (default: gzip:4096 and zlib:2048)")
    ap.add_argument("--seed", type=int, default=5)
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--singles", type=int, default=16)
    args = ap.parse_args()
    shapes = [(s.split(":")[0], int(s.split(":")[1])) for s in args.shape] or [("gzip", 4096), ("zlib", 2048)]
    for algo, _ in shapes:
        if algo not in LEVEL:
            ap.error(f"codec {algo!r}: gzip or zlib")
    report = {"card": card(), "runs": []}
    for algo, n in shapes:
        report["runs"].append(run_shape(algo, n, args.seed, args.pairs, args.singles))
        print(json.dumps(report["runs"][-1]), flush=True)
    report["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(report, f, indent=1)
    ok = all(r["parity"]["pairs_equal"] and r["parity"]["singles_equal"] and r["finite"] for r in report["runs"])
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
