"""CPU-only: the launch plans of the tcgen05 contraction (dmm_gemm_plan, which makes no CUDA call) over a sweep of shapes
at 148 SMs.  Every (tile cell x epilogue kind) pair and every ring depth of the TMA epilogue that the sweep reaches must
appear in the case table of tests/test_gemm_kernels_gpu.py, each case's written plan must be the query's answer (a cost
model change that moves a case off its cell fails here), and no reachable plan may leave the operand ring without room."""
import ctypes as C
import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gemm_kernels_gpu import CASES, KIND_CODE, NUM_SMS, SPLITK_CASES  # noqa: E402

# M enters the plan only through ceil(M / 128) and ceil(M / 256), constant on every block (128 j, 128 (j + 1)]: the ends
# of the blocks stand for all M from 1 to 20,000
MS = sorted({1, 20000} | {128 * j for j in range(1, 157)} | {128 * j + 1 for j in range(157)})
NS = sorted(set(range(1, 301)) | {1024, 7050, 18357, 80000, 500000} | set(range(19000, 25601, 16)) | {25600})
KS_SPLIT = [1, 64, 512, 1024, 1040, 1536, 2048, 2560, 3072, 3584, 4096, 4160, 4608, 7050, 18357, 70000]


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as g
    g.build()
    from diffmm_b200 import _lib
    _lib.load()
    return _lib


def flag_sets(L):
    """One flag combination per distinct input of the plan: the TMA epilogue's ring depends on an fp32 residual and a
    bf16 output, the register epilogues only on their kind."""
    f32, hi = L.GEMM_OUT_F32, L.GEMM_OUT_HI
    tma = [f32, hi, f32 | hi, L.GEMM_RESIDUAL | f32, L.GEMM_RESIDUAL | hi, L.GEMM_RESIDUAL | f32 | hi]
    reg = [L.GEMM_RES_HI | hi, L.GEMM_RES_HI | f32]
    x3 = [L.GEMM_A_LO | L.GEMM_B_LO | f32, hi | L.GEMM_OUT_LO, L.GEMM_RES_HI | L.GEMM_RES_LO | hi | L.GEMM_OUT_LO]
    return tma + reg + x3


def query(L, M, N, K, flags):
    pl = L.GemmLaunchPlan()
    rc = L.load().dmm_gemm_plan(NUM_SMS, M, N, K, flags, C.byref(pl))
    return rc, pl


@pytest.fixture(scope="module")
def sweep(L):
    cells, stages, bad = set(), set(), []
    for flags in flag_sets(L):
        for M in MS:
            for N in NS:
                rc, pl = query(L, M, N, 64, flags)
                if rc != 0:
                    bad.append((M, N, flags, L.last_error()))
                    continue
                cells.add((pl.bn, pl.ctas, pl.split, pl.epilogue))
                if pl.epilogue == L.GEMM_EPI_TMA:
                    stages.add((pl.bn, pl.ctas, pl.stages))
    return cells, stages, bad


def test_no_reachable_plan_lacks_room_for_the_operand_ring(sweep):
    assert sweep[2] == []


def test_every_reachable_cell_and_kind_has_a_case(sweep):
    cells, _, _ = sweep
    table = {(c.plan[0], c.plan[1], c.plan[2], KIND_CODE[c.kind]) for c in CASES}
    assert cells - table == set()
    assert len(cells) == 27


def test_every_reachable_tma_ring_depth_has_a_case(sweep):
    _, stages, _ = sweep
    table = {(c.plan[0], c.plan[1], c.plan[3]) for c in CASES if c.kind == "tma"}
    assert {s for _, _, s in stages} - {s for _, _, s in table} == set()
    assert 2 in {s for _, _, s in table}


@pytest.mark.parametrize("c", CASES, ids=[c.id for c in CASES])
def test_case_table_plans_are_the_query_answers(L, c):
    rc, pl = query(L, c.M, c.N, c.K, c.flags)
    assert rc == 0, L.last_error()
    assert (pl.bn, pl.ctas, pl.split, pl.stages, pl.nbuf, pl.epilogue, pl.ksplit) == c.plan + (KIND_CODE[c.kind], 1)
    assert pl.sub_bn * pl.split == pl.bn
    assert pl.grid % pl.ctas == 0 and 0 < pl.grid <= NUM_SMS


def test_every_reachable_split_k_factor_has_a_case(L):
    flags = L.GEMM_SPLITK | L.GEMM_OUT_F32 | L.GEMM_OUT_HI | L.GEMM_OUT_LO
    reached = set()
    for M in MS[::4] + [1, 257]:
        for N in NS[::4] + [129, 520, 1024]:
            for K in KS_SPLIT:
                rc, pl = query(L, M, N, K, flags)
                assert rc == 0
                reached.add(pl.ksplit)
                if pl.ksplit > 1:
                    assert (pl.bn, pl.ctas, pl.split, pl.epilogue) == (256, 2, 1, L.GEMM_EPI_TMA)
    assert reached - {ks for _, _, _, ks in SPLITK_CASES} == set()
    for M, N, K, ks in SPLITK_CASES:
        assert query(L, M, N, K, flags)[1].ksplit == ks, (M, N, K)


def test_plan_rejects_bad_arguments(L):
    assert query(L, 0, 64, 64, L.GEMM_OUT_F32)[0] == -1
    assert query(L, 64, 64, 1 << 31, L.GEMM_OUT_F32)[0] == -1
    assert query(L, 64, 64, 64, 1 << 9)[0] == -1
    pl = L.GemmLaunchPlan()
    assert L.load().dmm_gemm_plan(0, 64, 64, 64, L.GEMM_OUT_F32, C.byref(pl)) == -1
