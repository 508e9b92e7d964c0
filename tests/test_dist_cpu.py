"""world_size-2 gloo tests (CPU) of the multi-GPU host logic: row blocks, the edge all-gather that
follows the user-sharded rebuild, and the X-block all-gather of the row-partitioned propagation.
The per-rank compute is stood in by the numpy oracle (the CUDA kernels need a GPU)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as td
import torch.multiprocessing as mp

from diffmm_b200 import dist as ddist
from oracle import diffmm_oracle as O


def test_row_blocks_cover_and_balance():
    for n, w in [(10, 1), (10, 3), (19445, 8), (5, 8)]:
        b = ddist.row_blocks(n, w)
        assert b[0][0] == 0 and b[-1][1] == n and all(x[1] == y[0] for x, y in zip(b, b[1:]))
        assert max(e - s for s, e in b) - min(e - s for s, e in b) <= 1
    ptr = torch.tensor([0, 100, 100, 101, 102, 103, 104, 105, 106])
    b = ddist.row_blocks(8, 2, ptr)
    assert b == [(0, 1), (1, 8)] or b[0][1] <= 2            # the heavy first row gets its own block


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, U, I, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    td.init_process_group("gloo", rank=rank, world_size=world)
    try:
        rng = np.random.default_rng(0)                       # same data on every rank
        scores = rng.standard_normal((U, I)).astype(np.float32)
        deg = rng.integers(0, 9, U)
        indptr = np.zeros(U + 1, dtype=np.int64)
        np.cumsum(deg, out=indptr[1:])
        r0, r1 = ddist.shard_rows(U, world, rank)
        items = torch.full((int(indptr[-1]),), -1, dtype=torch.int32)
        local = O.topk_edges(scores[r0:r1], deg[r0:r1])      # stand-in for denoise chain + dmm_topk_edges
        items[indptr[r0]:indptr[r1]] = torch.from_numpy(np.concatenate(local).astype(np.int32))
        full = ddist.allgather_edges_multi({"m": items}, torch.from_numpy(indptr), U)["m"]
        want = np.concatenate(O.topk_edges(scores, deg)).astype(np.int32)
        ok_edges = bool((full.numpy() == want).all())

        # row-partitioned propagation: local SpMM on the local row block after an all-gather of X blocks
        users = np.repeat(np.arange(U), deg)
        adj = O.normalized_adj_csr(users, want, U, I)
        N = U + I
        x = rng.standard_normal((N, 8)).astype(np.float32)
        blocks = ddist.row_blocks(N, world)
        a, b = blocks[rank]
        xg = ddist.allgather_rows(torch.from_numpy(x[a:b].copy()), blocks)
        y_local = O.spmm_csr(*adj, xg.numpy())[a:b]
        yg = ddist.allgather_rows(torch.from_numpy(y_local.copy()), blocks)
        ok_spmm = bool(np.allclose(yg.numpy(), O.spmm_csr(*adj, x), rtol=1e-6, atol=1e-6))
        ret[rank] = (ok_edges, ok_spmm)
    finally:
        td.destroy_process_group()


@pytest.mark.parametrize("world", [2])
def test_sharded_edge_gather_and_propagation_gloo(world):
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), 101, 37, ret), nprocs=world, join=True)
    assert dict(ret) == {r: (True, True) for r in range(world)}


# ---------------------------------------------------------------------------------------------- partitioned propagation
def _fake_spmm(adj, x, *, alpha=1.0, beta=0.0, z=None, out=None, row0=0, row1=None):
    """CPU stand-in of ops.spmm (the CUDA kernel needs a GPU): same row-block contract, numpy oracle arithmetic."""
    row1 = adj.n_nodes if row1 is None else row1
    if out is None:
        out = torch.empty((adj.n_nodes, x.shape[1]), dtype=torch.float32)
    y = O.spmm_csr(adj.ptr.numpy(), adj.idx.numpy(), adj.val.numpy(), x.detach().numpy())
    out[row0:row1] = torch.from_numpy(y[row0:row1])
    return out


def _prop_loss(spmm_fn, adj, e0, w):
    """Three propagation layers with a nonlinearity in between and a scalar loss (the shape of Main.py:315-330)."""
    e, acc = e0, 0.0
    for _ in range(3):
        e = torch.tanh(spmm_fn(adj, e))
        acc = acc + e
    return (acc * w).sum()


def _prop_worker(rank, world, port, U, I, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    td.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from diffmm_b200 import autograd as ag, ops
        ops.spmm = _fake_spmm
        rng = np.random.default_rng(5)
        deg = rng.integers(0, 7, U)
        users = np.repeat(np.arange(U), deg)
        items = np.concatenate([np.sort(rng.choice(I, k, replace=False)) for k in deg]).astype(np.int32)
        ptr, idx, val = O.normalized_adj_csr(users, items, U, I)
        adj = ops.CsrAdj(torch.from_numpy(ptr), torch.from_numpy(idx), torch.from_numpy(val), U, I)
        N = U + I
        x = torch.from_numpy(rng.standard_normal((N, 8)).astype(np.float32))
        w = torch.from_numpy(rng.standard_normal((N, 8)).astype(np.float32))
        e_single = x.clone().requires_grad_(True)
        ag.set_partition(None)
        l1 = _prop_loss(ag.spmm, adj, e_single, w)
        l1.backward()
        part = ddist.PropPartition(U, I, td.group.WORLD)
        assert sum(b - a for a, b in part.row_ranges()) <= N and part.world == world
        ag.set_partition(part)
        e_part = x.clone().requires_grad_(True)
        l2 = _prop_loss(ag.spmm, adj, e_part, w)
        l2.backward()
        ag.set_partition(None)
        ret[rank] = (bool(torch.allclose(l1, l2, rtol=1e-6)), bool(torch.allclose(e_single.grad, e_part.grad, rtol=1e-5, atol=1e-6)),
                     [tuple(r) for r in part.row_ranges()])
    finally:
        td.destroy_process_group()


@pytest.mark.parametrize("U,I", [(40, 24), (41, 23)])      # evenly divisible and with leftover rows on both sides
def test_partitioned_propagation_values_and_gradients_gloo(U, I):
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_prop_worker, args=(world, _free_port(), U, I, ret), nprocs=world, join=True)
    got = dict(ret)
    assert all(got[r][0] and got[r][1] for r in range(world)), got
    covered = sorted(set(x for r in range(world) for a, b in got[r][2] for x in range(a, b)))
    assert covered == list(range(U + I))
