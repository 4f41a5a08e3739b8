"""``snacc`` command line for the GPU path; flag-compatible with the reference ``snacc/cli.py:16-78``.

File discovery (cli.py:89-102), the DataFrame pivot + CSV (cli.py:138-142) and the markdown run log
(cli.py:147-160) keep the reference behaviour; the thread-pool fan-out over N singles and N*N ordered
pairs (cli.py:104-136) is replaced by one batch call into libsnacc_b200.so.

Also accepted, because the reference README documents them (README.md:57-58): ``--reverse-compliment
BOOL`` and ``--fast-mode BOOL``.  ``--fast-mode True`` computes only the upper triangle (one order) and
uses (C(xy) - min) / max; the reference code defines no semantics for it.
"""
import sys
from datetime import datetime
from pathlib import Path

import os

import click
import numpy as np

from . import __version__
from .pairwise_ncd import ncd_matrix

SUFFIXES = [".fasta", ".fna", ".fa", ".faa", ".fsa"]


def collect_files(sequences, fasta=(), directories=()):
    """cli.py:89-102: positional files + -f files + suffix-filtered contents of positional / -d
    directories; de-duplicated; sorted by str(absolute path)."""
    sequences = [Path(s) for s in sequences]
    files = [p for p in sequences if p.is_file()]
    files.extend(Path(f) for f in fasta)
    sequences.extend(Path(d) for d in directories)
    for directory in [p for p in sequences if p.is_dir()]:
        for f in directory.iterdir():
            if f.suffix.lower() in SUFFIXES:
                files.append(f)
    return sorted(set(files), key=lambda x: str(x.absolute()))


def write_distance_csv(files, D, output):
    """The CSV of cli.py:138-142 -- long table -> pivot(index='file', columns='file2') -> to_csv with Path labels --
    written directly: rows and columns in the order pandas sorts the Path labels, header cell ``file``, labels quoted
    the way csv.QUOTE_MINIMAL does, floats as their shortest round-trip repr.  Byte-identical to the pandas route
    (tests/test_host_logic.py compares the two) without building a DataFrame of N^2 Python objects: 4 M rows at c5."""
    import csv
    import io
    n = len(files)
    files = [Path(f) for f in files]
    if len(set(files)) != n:
        raise ValueError("Index contains duplicate entries, cannot reshape")      # what DataFrame.pivot raises
    order = sorted(range(n), key=lambda i: files[i])
    D = np.asarray(D, dtype=np.float64)
    cell = io.StringIO()
    quote = csv.writer(cell, lineterminator="")

    def label(pth):
        cell.seek(0); cell.truncate(0)
        quote.writerow([str(pth)])
        return cell.getvalue()

    labels = [label(f) for f in files]
    header = ",".join(["file"] + [labels[j] for j in order])
    if _write_csv_native(output, header, labels, D, order):
        return
    with open(output, "w", newline="") as f:
        f.write(header + "\n")
        for i in order:
            row = D[i, order]
            vals = [("" if v != v else repr(v)) for v in row.tolist()]                  # NaN -> empty cell, like to_csv
            f.write(labels[i] + "," + ",".join(vals) + "\n")


def _write_csv_native(output, header, labels, D, order):
    """snacc_csv_write of libsnacc_b200.so (a host function of the C ABI, all host threads): the same bytes as the loop
    above, 10^8 cells (c3) in seconds instead of most of a minute.  False when the library is not built -- formatting is
    host work either way."""
    import ctypes
    from .engine import SnaccGpuError, load_library
    try:
        lib = load_library()
        fn = lib.snacc_csv_write
    except (SnaccGpuError, OSError, AttributeError):
        return False
    n = len(labels)
    Dc = np.ascontiguousarray(D, dtype=np.float64)
    arr = (ctypes.c_char_p * max(n, 1))(*[s.encode("utf-8") for s in labels])
    od = np.ascontiguousarray(order, dtype=np.int32)
    rc = fn(os.fsencode(str(output)), header.encode("utf-8"), arr, Dc.ctypes.data, n, od.ctypes.data, 0)
    if rc != 0:
        raise OSError(f"snacc_csv_write failed for {output}")
    return True


def _parse_bool(ctx, param, value):
    if value is None:
        return None
    v = str(value).strip().lower()
    if v in ("true", "1", "yes", "y", "t"):
        return True
    if v in ("false", "0", "no", "n", "f"):
        return False
    raise click.BadParameter(f"expected True or False, got {value!r}")


@click.command(context_settings=dict(help_option_names=["-h", "--help"]))
@click.argument("sequences", type=click.Path(exists=True, resolve_path=True), nargs=-1)
@click.option("-f", "--fasta", type=click.Path(dir_okay=False, exists=True, resolve_path=True), multiple=True,
              hidden=True, help="FASTA file containing sequence to compare.")
@click.option("-d", "--directory", "directories",
              type=click.Path(dir_okay=True, file_okay=False, exists=True, resolve_path=True), multiple=True,
              help="Directory containing FASTA files to compare.")
@click.option("-n", "--num-threads", "numThreads", type=int, default=None,
              help="Accepted for compatibility; the GPU engine does not use host threads for compression.")
@click.option("-o", "--output", type=click.Path(dir_okay=False, exists=False),
              help="The location for the output CSV file.", prompt="Output CSV path")
@click.option("-s", "--save-compression", "saveCompression",
              type=click.Path(dir_okay=True, file_okay=False, resolve_path=True), default=None,
              help="Not supported on the GPU path (only sizes are produced).")
@click.option("-c", "--compression", default="lzma", type=click.Choice(["lzma", "gzip", "bzip2", "zlib", "lz4"]),
              help="The compression algorithm to use. The GPU path supports lz4, gzip, zlib and bzip2.")
@click.option("--show-progress/--no-show-progress", "showProgress", default=True,
              help="Accepted for compatibility.")
@click.option("-r", "--reverse_complement", is_flag=True, default=False,
              help="Whether to use the reverse complement of the sequence.")
@click.option("--reverse-compliment", "reverse_compliment", default=None, callback=_parse_bool,
              help="README spelling of -r: True or False.")
@click.option("--fast-mode", "fast_mode", default=None, callback=_parse_bool,
              help="True: one concatenation order only (upper triangle), NCD = (C(xy) - min) / max.")
@click.option("--gpus", "gpus", type=int, default=None,
              help="Number of GPUs of this box to use (one process per GPU is launched). Default: the GPUs of the "
                   "torchrun process group this command runs in, else one.")
@click.option("--log/--no-log", "log", default=True, help="Whether to save a log.")
def cli(sequences, fasta, directories, numThreads, compression, showProgress, saveCompression, output,
        reverse_complement, reverse_compliment, fast_mode, gpus, log):
    start_time = datetime.now()
    if fasta:
        click.secho("Warning: the -f flag is deprecated. Please pass files and paths directly.", fg="yellow")
    if saveCompression:
        raise click.UsageError("-s/--save-compression is not supported on the GPU path: compressed streams are "
                               "never materialised, only their sizes are computed")
    if compression not in ("lz4", "gzip", "zlib", "bzip2"):
        raise click.UsageError(f"-c {compression} is not supported on the GPU path (supported: lz4, gzip, zlib, "
                               "bzip2); there is no CPU fallback" + (" -- lzma is the reference's default (cli.py:52), "
                                                                     "so pass -c lz4, -c gzip, -c zlib or -c bzip2 "
                                                                     "explicitly"
                                                             if compression == "lzma" else ""))
    if reverse_compliment is not None:
        reverse_complement = reverse_compliment
    output = Path(output)
    files = collect_files(sequences, fasta, directories)
    if not files:
        raise click.UsageError("no FASTA files found")

    from . import sharding
    sharding.init_distributed()           # under torchrun: join the group, bind to GPU LOCAL_RANK (no-op otherwise)
    try:
        rank0 = sharding.is_rank0()
        n = len(files)
        n_pairs = n * (n + 1) // 2 if fast_mode else n * n
        if rank0:
            click.secho(f"Compressing {n} files and {n_pairs} {'unordered' if fast_mode else 'ordered'} pairs on "
                        "the GPU...", fg="green")
        bar = None
        if showProgress and rank0:
            from tqdm import tqdm
            bar = tqdm(total=n + n_pairs, unit="job")        # the reference shows one bar per fan-out (cli.py:172-174)
        t0 = datetime.now()
        labels, C, S, D = ncd_matrix(files, compression, reverse_complement=reverse_complement,
                                     fast_mode=bool(fast_mode), gpus=gpus)
        compute_s = (datetime.now() - t0).total_seconds()
        if bar is not None:
            bar.update(n + n_pairs)
            bar.close()
        if rank0:
            t1 = datetime.now()
            write_distance_csv(files, D, output)
            csv_s = (datetime.now() - t1).total_seconds()
            if log:
                world = sharding._dist().get_world_size() if sharding._dist() else (gpus or 1)
                with open(output.stem + ".md", "w") as f:
                    print(log_template.format(time=datetime.now(), duration=datetime.now() - start_time,
                                              method=compression, rev_comp=reverse_complement,
                                              output_path=output.absolute(),
                                              py_version=str(sys.version.replace("\n", "")),
                                              snacc_version=__version__, jobs=n + n_pairs, pairs=n * (n + 1) // 2,
                                              compute_s=compute_s, csv_s=csv_s, gpus=world,
                                              pairs_per_s=(n * (n + 1) // 2) / max(compute_s, 1e-9)), file=f)
                    for _f in [str(_file.absolute()) for _file in files]:
                        print("*", _f, file=f)
    finally:
        sharding.shutdown_distributed()


log_template = '''# `snacc` Analysis
## Run Information
* Analysis time: {time}
* Analysis duration: {duration}
* Compression method: {method}
* Reverse complement: {rev_comp}
* Output filepath: {output_path}
* Compressor jobs: {jobs} ({pairs} unordered pairs) in {compute_s:.3f} s on the GPU path ({gpus} GPU(s), {pairs_per_s:.1f} pairs/s, FASTA parsing and upload included); CSV written in {csv_s:.3f} s

## Version Information
* Python: {py_version}
* snacc (b200): {snacc_version}

## Analyzed Files
'''


if __name__ == "__main__":
    cli()
