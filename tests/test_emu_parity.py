"""CPU parity of the kernels' own code: the GPU parity tests of tests/test_gpu_parity.py, test_gpu_prep.py and
test_gpu_round2.py, run on a machine WITHOUT a GPU against the SIMT-emulated build of the library's .cu sources
(tests/emu: every CUDA thread a fiber, warp collectives and __syncthreads as rendezvous, the CUDA runtime as plain
host memory).  Same test bodies, same C ABI, same oracle -- only the library handle differs.

This is test infrastructure: nothing under gat_b200/ builds or loads the emulated library, and gat_b200._lib.load()
refuses it (test_engine_refuses_the_emulated_build).  What it buys: the placement / counting / preparation /
statistics kernels are checked bit for bit against the oracle on every CPU run of the suite, and a kernel whose
lanes disagree about a warp collective fails here as a reported deadlock instead of hanging a GPU.
"""
import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))


@pytest.fixture(scope="module")
def emu_lib():
    import emu_context
    return emu_context.library()


@pytest.fixture(scope="module")
def emu_ctx(emu_lib):
    import emu_context
    c = emu_context.context()
    yield c
    c.close()


# (module, test function, extra keyword arguments besides ctx / oracle)
CASES = [
    ("test_gpu_parity", "test_place_single_units_match_oracle", {}),
    ("test_gpu_parity", "test_place_problem_matches_oracle", {"n_iso": 0}),
    ("test_gpu_parity", "test_place_problem_matches_oracle", {"n_iso": 3}),
    ("test_gpu_parity", "test_count_lists_match_oracle", {}),
    ("test_gpu_parity", "test_run_matches_oracle", {"n_iso": 0}),
    ("test_gpu_parity", "test_run_matches_oracle", {"n_iso": 3}),
    ("test_gpu_parity", "test_column_stats_match_oracle", {}),
    ("test_gpu_parity", "test_column_stats_float_and_reference", {}),
    ("test_gpu_parity", "test_invalid_inputs_fail_loudly", {}),
    ("test_gpu_parity", "test_sampler_segments_matches_oracle", {}),
    ("test_gpu_parity", "test_sampler_shift_matches_oracle", {}),
    ("test_gpu_parity", "test_count_filter_edge_geometries", {}),
    ("test_gpu_parity", "test_overlap_pieces_counter_matches_intersect", {}),
    ("test_gpu_prep", "test_lists_from_rows_normalize_and_merge", {}),
    ("test_gpu_prep", "test_lists_restrict_collapse_select", {}),
    ("test_gpu_prep", "test_invalid_rows_fail_loudly", {}),
    ("test_gpu_round2", "test_skewed_unit_grows_its_buffer", {}),
    ("test_gpu_round2", "test_overflow_growth_is_exercised", {}),
    ("test_gpu_round2", "test_streamed_column_stats_exact_and_layout_independent", {}),
    ("test_gpu_round2", "test_column_stats_do_not_depend_on_the_kernel_that_computes_them", {}),
    ("test_gpu_parity", "test_async_annotations_same_counts_and_deferred_errors", {}),
    ("test_gpu_parity", "test_count_index_geometries_match_oracle", {}),
    ("test_gpu_properties", "test_isochore_config_matches_oracle", {}),
]


@pytest.mark.parametrize("module,name,extra", CASES, ids=["%s%s" % (c[1], "".join("-%s%s" % kv for kv in c[2].items())) for c in CASES])
def test_gpu_test_body_on_the_emulated_kernels(emu_ctx, oracle, monkeypatch, tmp_path, module, name, extra):
    fn = getattr(importlib.import_module("tests." + module), name)
    kwargs = dict(extra)
    wanted = fn.__code__.co_varnames[:fn.__code__.co_argcount]
    for arg, value in (("ctx", emu_ctx), ("oracle", oracle), ("monkeypatch", monkeypatch), ("tmp_path", tmp_path)):
        if arg in wanted:
            kwargs[arg] = value
    fn(**kwargs)


def test_engine_refuses_the_emulated_build(emu_lib, monkeypatch):
    """the engine's loader must not accept the emulated build, whatever GATB_LIB says"""
    import build_emu
    from gat_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", build_emu.LIB)
    with pytest.raises(ImportError):
        _lib.load()
