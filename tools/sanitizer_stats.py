"""Small run of the TMA-streamed column statistics and of the placement kernels, for compute-sanitizer (memcheck /
racecheck / synccheck): shapes that use the bulk-copy path, the partial last chunk and several select passes.

    compute-sanitizer --tool racecheck python tools/sanitizer_stats.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))

import numpy as np  # noqa: E402

from gat_b200 import device  # noqa: E402
import helpers  # noqa: E402

ctx = device.Context(0)
rng = np.random.default_rng(3)
for l, A in ((3001, 1000), (5000, 125), (777, 9)):
    counts = rng.integers(0, 70000, size=(l, A)).astype(np.uint32)
    obs = counts[0].astype(np.float64)
    got = ctx.column_stats(counts, obs, pseudo_count=1.0)
    assert np.array_equal(got["expected"], counts.sum(axis=0, dtype=np.uint64) / l)
    srt = np.sort(counts, axis=0)
    off = int(0.05 * l)
    assert np.array_equal(got["lower95"], srt[min(off, l - 1)].astype(np.float64))
pr = helpers.random_problem(rng, n_contigs=3, n_iso=3, nseg=120, n_annot=5)
smp = device.Sampler(ctx, pr["unit_contig"], pr["n_contigs"], True, pr["unit_segments"], pr["unit_workspace"])
annos = device.Annotations(ctx, pr["annotations"], key_ws_nseg=pr["cws_nseg"])
res, info = smp.run(annos, ["nucleotide-overlap", "segment-overlap"], seed=5, track=0, sample_begin=0, n_samples=64)
smp.close()
annos.close()
ctx.close()
print("ok")
