"""The host-only workspace sizes of the rebuild's tail (dmm_topk_workspace_bytes, dmm_topk_pruned_workspace_bytes,
dmm_build_adj_workspace_bytes) against the geometry tests/test_rebuild_tail_kernels_gpu.py builds its cases from; these
run without a GPU."""
import pytest

from diffmm_b200 import _lib
from test_rebuild_tail_kernels_gpu import SEG_COLS, SEGMENT_CASES, _seg

EDGES = [0, 1, 4097, 12345678]


def _align256(x):
    return (x + 255) // 256 * 256


@pytest.mark.parametrize("S,n_cols", SEGMENT_CASES)
def test_segment_workspace_is_S_times_the_edges(S, n_cols):
    lib = _lib.load()
    assert _seg(n_cols)[0] == S
    for E in EDGES:
        assert lib.dmm_topk_workspace_bytes(n_cols, E) == S * E * 4


@pytest.mark.parametrize("n_cols", [1, 224, 8191, SEG_COLS])
def test_rows_of_one_segment_need_no_workspace(n_cols):
    assert _lib.load().dmm_topk_workspace_bytes(n_cols, 1000) == 0
    assert _lib.load().dmm_topk_workspace_bytes(SEG_COLS + 1, 1000) == 2 * 1000 * 4


@pytest.mark.parametrize("n_rows", [0, 1, 63, 64, 65, 1000])
@pytest.mark.parametrize("n_cols", [224, 3200, 70001, 524288, 524289])
def test_pruned_workspace_layout(n_rows, n_cols):
    """[count at 0 | deferred-row list at 256 | one chunk-list slot per edge | segment workspace], 256-byte aligned."""
    lib = _lib.load()
    for E in EDGES:
        want = 256 + _align256(4 * max(n_rows, 1)) + _align256(4 * max(E, 1)) + lib.dmm_topk_workspace_bytes(n_cols, E)
        assert lib.dmm_topk_pruned_workspace_bytes(n_rows, n_cols, E) == want


@pytest.mark.parametrize("U,I", [(1, 1), (300, 255), (60000, 100000), (10 ** 6, (1 << 20) + 3)])
@pytest.mark.parametrize("E", [0, 1, 1000, 4_700_000, 6_000_000, 12_800_000, (1 << 31) - 1])
def test_adj_workspace_covers_the_sort_scratch(U, I, E):
    """Beyond the carved arrays (three E-entry int32 lists, item counts, item offsets, d^-1/2), the radix sort gets at
    least the two extra E x 4-byte arrays CUB allocates for separate input and output buffers."""
    e4 = _align256(4 * max(E, 1))
    fixed = 3 * e4 + _align256(4 * (I + 1)) + _align256(8 * (I + 1)) + _align256(8 * (U + I))
    assert _lib.load().dmm_build_adj_workspace_bytes(U, I, E) - fixed >= 8 * E
