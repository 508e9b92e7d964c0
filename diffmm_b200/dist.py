"""Multi-GPU plumbing: one process per GPU, torch.distributed (NCCL over NVLink on the B200 box,
gloo in the CPU tests).  The path shards in two places (SURVEY.md §8e):

  * rebuild (denoise chain + top-k): users are independent -> contiguous user blocks per rank, Denoise
    weights replicated, NO data-path collective; one all-gather of the emitted edge lists at the end
    (offsets are the train-CSR indptr, known a priori because k_u = deg(u));
  * propagation: rows of the symmetric adjacency and of X are block-partitioned, one all-gather of the
    X blocks per SpMM layer, local SpMM on the local row block (dmm_spmm_csr row0/row1).

The reference has no distributed code at all (single process, single device).
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
import torch.distributed as td


def world_size(group=None) -> int:
    return td.get_world_size(group) if td.is_available() and td.is_initialized() else 1


def rank(group=None) -> int:
    return td.get_rank(group) if td.is_available() and td.is_initialized() else 0


def row_blocks(n_rows: int, world: int, weights: Optional[torch.Tensor] = None) -> List[Tuple[int, int]]:
    """Contiguous row blocks, one per rank.  With ``weights`` (e.g. CSR indptr, i.e. cumulative nnz) the cut
    points balance the cumulative weight instead of the row count; blocks stay contiguous and cover [0, n)."""
    if weights is None:
        cuts = [(n_rows * r) // world for r in range(world + 1)]
    else:
        cum = weights.detach().to("cpu", torch.float64)
        # cum has n_rows + 1 entries (indptr); add the row index so that zero-degree rows still cost something
        cost = cum + torch.arange(n_rows + 1, dtype=torch.float64)
        total = float(cost[-1])
        targets = torch.tensor([total * r / world for r in range(1, world)], dtype=torch.float64)
        inner = torch.searchsorted(cost, targets).clamp_(0, n_rows).tolist() if world > 1 else []
        cuts = [0] + [int(c) for c in inner] + [n_rows]
        for i in range(1, len(cuts)):
            cuts[i] = max(cuts[i], cuts[i - 1])
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def shard_rows(n_rows: int, world: int, rk: int, indptr: Optional[torch.Tensor] = None) -> Tuple[int, int]:
    """User block of rank ``rk`` for the rebuild.  Rows cost the same GEMM work regardless of degree, so the
    split is by row count (indptr is accepted for API symmetry and ignored)."""
    return row_blocks(n_rows, world)[rk]


class EdgeGatherPlan:
    """Host-side layout of the edge all-gather that follows the user-sharded rebuild, computed once per dataset
    (the offsets are the train-CSR indptr at the block boundaries, so no device sync is needed per call)."""

    def __init__(self, indptr: torch.Tensor, n_users: int, world: int):
        self.blocks = row_blocks(n_users, world)
        ptr_cpu = indptr.detach().to("cpu")
        self.offs = [(int(ptr_cpu[a]), int(ptr_cpu[b])) for a, b in self.blocks]
        self.seg = max(1, max(e - s for s, e in self.offs))
        self.world = world


def allgather_edges_multi(items: dict, indptr: torch.Tensor, n_users: int, group=None,
                          plan: Optional[EdgeGatherPlan] = None) -> dict:
    """Every rank filled items[m][indptr[r0]:indptr[r1]) of each modality m for its user block; returns the complete
    edge lists on every rank.  The edge lists of ALL modalities go in ONE collective: every rank packs its segment of
    each list into one padded send buffer [M, seg] (padding is never read back), one all_gather_into_tensor, and one
    index_select per modality compacts the [world, M, seg] result into the CSR-ordered list (the index is precomputed
    per plan).  3 + M launches per rebuild instead of M x (zero fill + copy + collective + world slice copies)."""
    world, rk = world_size(group), rank(group)
    if world == 1:
        return dict(items)
    if plan is None or plan.world != world:
        plan = EdgeGatherPlan(indptr, n_users, world)
    offs, seg = plan.offs, plan.seg
    names = list(items)
    M = len(names)
    first = items[names[0]]
    dev, dt = first.device, first.dtype
    s, e = offs[rk]
    send = torch.empty((M, seg), dtype=dt, device=dev)
    for k, m in enumerate(names):
        send[k, : e - s].copy_(items[m][s:e])
    recv = torch.empty((world, M, seg), dtype=dt, device=dev)
    td.all_gather_into_tensor(recv.view(-1), send.view(-1), group=group)
    key = ("_unpack_index", M)
    cache = getattr(plan, "_unpack_cache", None)
    if cache is None:
        cache = plan._unpack_cache = {}
    src = cache.get(key)
    if src is None or src[0].device != dev:
        src = []
        for k in range(M):
            src.append(torch.cat([torch.arange((r * M + k) * seg, (r * M + k) * seg + (b - a), dtype=torch.int64)
                                  for r, (a, b) in enumerate(offs)]).to(dev))
        cache[key] = src
    flat = recv.view(-1)
    return {m: flat.index_select(0, src[k]) for k, m in enumerate(names)}


def allgather_rows(x_local: torch.Tensor, blocks: List[Tuple[int, int]], group=None) -> torch.Tensor:
    """All-gather of row-partitioned X blocks (N x D) before a row-partitioned SpMM layer."""
    world, rk = world_size(group), rank(group)
    if world == 1:
        return x_local
    D = x_local.shape[1]
    seg = max(1, max(b - a for a, b in blocks))
    send = torch.zeros((seg, D), dtype=x_local.dtype, device=x_local.device)
    a, b = blocks[rk]
    send[: b - a] = x_local
    recv = torch.empty((seg * world, D), dtype=x_local.dtype, device=x_local.device)
    td.all_gather_into_tensor(recv, send, group=group)
    return torch.cat([recv[r * seg: r * seg + (b - a)] for r, (a, b) in enumerate(blocks)], 0)


# ------------------------------------------------------------------------------------------------------------------
# Row-partitioned propagation (north_star: "embedding tables are row-partitioned for propagation, with NCCL all-gather
# over NVLink per GCN layer"; reference call sites Model.py:90,93,105,111,114,123,130 and Main.py:319).
# ------------------------------------------------------------------------------------------------------------------
class PropPartition:
    """Row partition of the N = U + I node rows of the symmetric normalised adjacency for one process group.

    Rank r owns the user rows [r su, (r + 1) su) and the item rows U + [r si, (r + 1) si), su = U // W, si = I // W:
    user rows carry ~deg(u) entries and item rows ~E / I, so cutting BOTH ranges evenly balances the ranks (a single
    contiguous cut of [users; items] would give the item-row ranks three times the entries of the user-row ranks at the
    ifashion shape).  The < W leftover rows of either range are computed by every rank (no communication).  Y keeps the
    natural [users; items] layout: the two evenly divided regions are all-gathered IN PLACE (equal counts, no padding,
    no unpack copies)."""

    def __init__(self, n_users: int, n_items: int, group=None):
        self.group = group
        self.world = world_size(group)
        self.rank = rank(group)
        self.n_users, self.n_items = int(n_users), int(n_items)
        self.su = self.n_users // self.world
        self.si = self.n_items // self.world

    @property
    def n_nodes(self):
        return self.n_users + self.n_items

    def row_ranges(self):
        """[(row0, row1)] this rank computes: its user block, its item block, and the replicated leftovers."""
        U, W, r, su, si = self.n_users, self.world, self.rank, self.su, self.si
        out = []
        if su > 0:
            out.append((r * su, (r + 1) * su))
        if W * su < U:
            out.append((W * su, U))
        if si > 0:
            out.append((U + r * si, U + (r + 1) * si))
        if U + W * si < self.n_nodes:
            out.append((U + W * si, self.n_nodes))
        return out

    def product_(self, spmm_rows, y: torch.Tensor) -> torch.Tensor:
        """Runs ``spmm_rows(row0, row1)`` (writes y[row0:row1]) over this rank's blocks and all-gathers y in place.  On
        CUDA the all-gather of the user region is issued on a side stream as soon as the user blocks are written, so
        it travels over NVLink while the item blocks are still being computed."""
        if self.world == 1 or not y.is_cuda:
            for r0, r1 in self.row_ranges():
                spmm_rows(r0, r1)
            return self.gather_(y)
        U, W, r, su, si = self.n_users, self.world, self.rank, self.su, self.si
        main = torch.cuda.current_stream(y.device)
        if getattr(self, "_comm_stream", None) is None:
            self._comm_stream = torch.cuda.Stream(device=y.device)
        comm = self._comm_stream
        ranges = self.row_ranges()
        user_ranges = [(a, b) for a, b in ranges if b <= U]
        item_ranges = [(a, b) for a, b in ranges if a >= U]
        for a, b in user_ranges:
            spmm_rows(a, b)
        if su > 0:
            comm.wait_stream(main)
            with torch.cuda.stream(comm):
                td.all_gather_into_tensor(y[: W * su], y[r * su:(r + 1) * su], group=self.group)
        for a, b in item_ranges:
            spmm_rows(a, b)
        if si > 0:
            td.all_gather_into_tensor(y[U: U + W * si], y[U + r * si: U + (r + 1) * si], group=self.group)
        main.wait_stream(comm)
        y.record_stream(comm)
        return y

    def gather_(self, y: torch.Tensor) -> torch.Tensor:
        """In-place all-gather of the evenly divided user and item regions of y [N, D] (every rank has written its own
        blocks and the leftovers): afterwards every rank holds the whole y."""
        if self.world == 1:
            return y
        U, W, r, su, si = self.n_users, self.world, self.rank, self.su, self.si
        if su > 0:
            td.all_gather_into_tensor(y[: W * su], y[r * su:(r + 1) * su], group=self.group)
        if si > 0:
            td.all_gather_into_tensor(y[U: U + W * si], y[U + r * si: U + (r + 1) * si], group=self.group)
        return y
