"""Placement units that take the first checkpoint's less common paths: placements that start in a few buckets of
the counting sort's plan (a workspace of two small, distant pieces: the keys are too clustered for the counting
sort and go to the bitonic sort), a few crowded buckets next to sparse ones, a dense unit whose buckets hold several
keys, and a unit with one dominant segment, whose placements far outnumber its segments.  Each unit runs once with
its estimated buffer and once with 64 slots, where the buffer fills up and is merged early, before the first
checkpoint.  Every sample must equal the oracle bit for bit, on the GPU and on the emulated kernels."""
import os
import sys

import numpy as np
import pytest

from tests import helpers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))


def _segments_in(rng, pieces, n, lmin, lmax):
    """n segments of lmin .. lmax bases, each starting inside one of the workspace pieces (then normalized)"""
    out = []
    for _ in range(n):
        s, e = pieces[int(rng.integers(0, len(pieces)))]
        start = int(rng.integers(s, e))
        out.append((start, start + int(rng.integers(lmin, lmax + 1))))
    return helpers.normalize(np.array(sorted(out), dtype=np.uint32))


def _units(rng):
    units = []
    # two small pieces 50 Mb apart: the plan's buckets span the gap, every placement lands in the first or
    # the last bucket
    ws = np.array([[1000, 6000], [50000000, 50005000]], dtype=np.uint32)
    units.append((_segments_in(rng, ws, 300, 10, 40), ws))
    # the same with a third piece in between: two crowded buckets next to sparse ones
    ws = np.array([[0, 3000], [2000000, 2600000], [9000000, 9002000]], dtype=np.uint32)
    units.append((_segments_in(rng, ws, 400, 20, 200), ws))
    # one evenly used piece, many segments: several keys per bucket
    ws = np.array([[0, 3000000]], dtype=np.uint32)
    units.append((_segments_in(rng, ws, 700, 50, 3000), ws))
    # one dominant segment: the short ones are drawn over and over, far more placements than segments
    ws = np.array([[0, 4000000]], dtype=np.uint32)
    segs = _segments_in(rng, np.array([[0, 300000]], dtype=np.uint32), 60, 100, 400)
    units.append((np.concatenate([segs, np.array([[1000000, 1090000]], dtype=np.uint32)]), ws))
    return units


def _check(ctx, oracle, monkeypatch, n_samples):
    from gat_b200 import device
    rng = np.random.default_rng(41)
    for u, (segs, ws) in enumerate(_units(rng)):
        for cap_max in (None, "64"):        # 64 slots: the buffer fills up before the first checkpoint
            if cap_max:
                monkeypatch.setenv("GATB_PLACE_CAP_MAX", cap_max)
            smp = device.Sampler(ctx, [0], 1, False, [segs], [ws])
            monkeypatch.delenv("GATB_PLACE_CAP_MAX", raising=False)
            placed, status = smp.place(seed=77 + u, track=1, sample_begin=5, n_samples=n_samples)
            smp.close()
            assert not (status & device.UNIT_OVERFLOW).any()
            for s in range(n_samples):
                exp, _ = oracle.sampler_annotator_philox(segs, ws, 77 + u, 1, 0, 5 + s, cap=1 << 16)
                assert np.array_equal(placed[s][0], exp), (u, cap_max, s, placed[s][0][:4], exp[:4])


@pytest.mark.gpu
def test_clustered_units_match_oracle(ctx, oracle, monkeypatch):
    _check(ctx, oracle, monkeypatch, 16)


def test_clustered_units_match_oracle_emulated(oracle, monkeypatch):
    import emu_context
    ctx = emu_context.context()
    try:
        _check(ctx, oracle, monkeypatch, 4)
    finally:
        ctx.close()
