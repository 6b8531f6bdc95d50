"""Read a config-5-shaped counts table (1e6 samples x 200 annotations) with the host reader and with the GPU reader
(gatb_parse_counts), plain and gzipped, and run gat-compare on two such tables both ways.

    python tools/counts_table_bench.py [--samples 1000000] [--rows 200] [--out result.json]

The GPU reader's time is split into file read (+ gzip decompression on the host), upload, the parse kernels (CUDA
events around every launch, gatb_profile) and the batched statistics.  The results of the two readers are compared
(statistics with ==, the sample matrices exactly) and the JSON records the GPU's name and power limit.  The tables
are written to a temporary directory, which is removed at the end."""
import argparse
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STATS = ["expected", "stddev", "lower95", "upper95", "fold", "pvalue"]


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                      text=True, timeout=30)
        info["power_limit"] = out.strip()
    except (OSError, subprocess.SubprocessError):
        info["power_limit"] = "unknown"
    return info


def write_table(ctx, path, rows, samples, seed):
    """a table as run() writes it: the text of every column from gatb_format_counts"""
    import torch
    rng = np.random.default_rng(seed)
    m = torch.from_numpy(rng.poisson(20000, size=(samples, rows)).astype(np.int32)).to("cuda")
    text, off = ctx.format_counts(device_ptr=m.data_ptr(), n_samples=samples, n_cols=rows)
    obs = rng.integers(15000, 25000, size=rows)
    with open(path, "wb") as f:
        f.write(b"track\tannotation\tobserved\tcounts\n")
        for a in range(rows):
            f.write(b"merged\tanno%03d\t%d\t" % (a, obs[a]))
            f.write(text[int(off[a]):int(off[a + 1])].tobytes())
            f.write(b"\n")
    return os.path.getsize(path)


def same_results(a, b):
    if len(a) != len(b):
        return False
    for x, y in zip(a, b):
        if (x.track, x.annotation, x.observed) != (y.track, y.annotation, y.observed):
            return False
        if any(getattr(x, k) != getattr(y, k) for k in STATS):
            return False
    return True


def device_phases(ctx, path):
    """the steps of Engine.readCountsTable + the statistics of fromCounts, each timed to a synchronise"""
    import torch
    from gat_b200 import engine as Engine
    dev = torch.device("cuda", ctx.device)
    t = {}
    t0 = time.perf_counter()
    with (gzip.open(path, "rb") if path.endswith(".gz") else open(path, "rb")) as f:
        raw = f.read()
    t["read_s"] = time.perf_counter() - t0
    n_head = len(Engine.COUNTS_HEADER)
    body = np.frombuffer(raw, dtype=np.uint8, offset=n_head)
    n_lines = raw.count(b"\n", n_head)
    t0 = time.perf_counter()
    text = torch.from_numpy(body.copy()).to(dev)
    torch.cuda.synchronize(dev)
    t["upload_s"] = time.perf_counter() - t0
    ctx.profile(True)
    ctx.profile_read()
    t0 = time.perf_counter()
    table = ctx.parse_counts(text.data_ptr(), body.size, n_lines)
    counts = torch.empty((table["n_samples"], table["n_rows"]), dtype=torch.int32, device=dev)
    ctx.parse_counts(text.data_ptr(), body.size, n_lines, counts_ptr=counts.data_ptr())
    t["parse_calls_s"] = time.perf_counter() - t0
    t["parse_kernels_ms"] = ctx.profile_read()["other"][0]
    ctx.profile(False)
    t0 = time.perf_counter()
    ctx.column_stats(None, np.zeros(table["n_rows"]), device_ptr=counts.data_ptr(), n_samples=table["n_samples"],
                     n_cols=table["n_rows"], is_float=0)
    t["statistics_s"] = time.perf_counter() - t0
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=1000000)
    ap.add_argument("--rows", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import gat_b200
    from gat_b200 import compare, engine as Engine
    ctx = Engine.getContext()
    res = dict(gpu_info(), samples=args.samples, rows=args.rows)
    tmp = tempfile.mkdtemp(prefix="gatb_counts_")
    try:
        plain = os.path.join(tmp, "c1.tsv")
        res["bytes"] = write_table(ctx, plain, args.rows, args.samples, 1)
        with open(plain, "rb") as fi, gzip.open(plain + ".gz", "wb", compresslevel=1) as fo:
            shutil.copyfileobj(fi, fo, 64 << 20)
        res["bytes_gz"] = os.path.getsize(plain + ".gz")
        second = os.path.join(tmp, "c2.tsv")
        write_table(ctx, second, args.rows, args.samples, 2)
        gat_b200.fromCounts(plain)                            # warm-up: context, kernels, pools
        torch.cuda.synchronize()
        for name, path in (("tsv", plain), ("tsv_gz", plain + ".gz")):
            leg = {}
            t0 = time.perf_counter()
            dev = gat_b200.fromCounts(path)
            leg["device_fromCounts_s"] = time.perf_counter() - t0
            leg["device_phases"] = device_phases(ctx, path)
            t0 = time.perf_counter()
            host = gat_b200._fromCountsHost(path)
            leg["host_fromCounts_s"] = time.perf_counter() - t0
            leg["identical_statistics"] = same_results(dev, host)
            leg["identical_samples"] = bool(np.array_equal(
                dev[0]._lazy[0].host(), np.stack([r._source for r in host], axis=1).astype(np.uint32)))
            del dev, host
            res[name] = leg
        # gat-compare on two tables, both readers (the host leg with the GPU reader switched off)
        outs, reader = {}, Engine.readCountsTable
        for name, fn in (("device", reader), ("host", lambda f: None)):
            Engine.readCountsTable = fn
            out = os.path.join(tmp, "compare_%s.tsv" % name)
            t0 = time.perf_counter()
            compare.main(["gat-compare", plain, second, "--stdout=" + out])
            res["compare_%s_s" % name] = time.perf_counter() - t0
            outs[name] = open(out, "rb").read()
        Engine.readCountsTable = reader
        res["compare_identical_output"] = outs["device"] == outs["host"]
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res, sort_keys=True)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1, sort_keys=True) + "\n")


if __name__ == "__main__":
    main()
