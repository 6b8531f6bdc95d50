"""CPU run of the counts-table reader and device gat-compare test bodies of tests/test_gpu_counts_table.py on the
SIMT-emulated build of the kernels (tests/emu, as tests/test_emu_parity.py does): the parse kernels of count.cu and
gatb_compare_stats_device are checked on every CPU run of the suite, at small sizes."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))


@pytest.fixture(scope="module")
def emu_ctx():
    import emu_context
    c = emu_context.context()
    yield c
    c.close()


@pytest.mark.parametrize("name", ["test_parse_grammar_edges", "test_parse_tile_edges", "test_parse_random_tables",
                                  "test_compare_stats_device_equals_host"])
def test_counts_table_body_on_the_emulated_kernels(emu_ctx, name):
    from tests import test_gpu_counts_table as T
    getattr(T, name)(emu_ctx)
