"""Tensor-level wrappers over the C ABI (include/diffmm_b200.h).

Every function takes CUDA torch tensors (memory + stream plumbing only), validates layout, and
calls exactly one C-ABI entry point on the current stream.  No arithmetic happens in PyTorch here.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import GemmEpilogue


def pad_to(n: int, m: int) -> int:
    return (n + m - 1) // m * m


def _p(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


_call_device = 0       # device of the tensors of the C-ABI call being assembled (set by _ctx, read by _stream)


def _stream():
    # raw handle of torch's current stream ON THE TENSORS' DEVICE (torch.cuda.current_stream() builds a Python Stream
    # object: ~15 us).  Every wrapper evaluates _ctx(tensor) before _stream() (argument order of _lib.call).
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(_call_device))


def _ctx(t: torch.Tensor):
    """Context of the tensor's device.  Kernels are launched on the CURRENT device, so the tensor must live there:
    the library never switches devices behind the caller's back (run under ``torch.cuda.device(t.device)``)."""
    global _call_device
    if not t.is_cuda:
        raise _lib.DiffMMError("diffmm_b200 operators need CUDA tensors (there is no CPU fallback)")
    cur = torch.cuda.current_device()
    idx = t.device.index if t.device.index is not None else cur
    if idx != cur:
        raise _lib.DiffMMError(f"tensor on cuda:{idx} but the current device is cuda:{cur}: call under "
                               f"torch.cuda.device({idx}) (Coach does this for base.gpu)")
    _call_device = idx
    return _lib.ctx(idx)


def _row_major(t: torch.Tensor, name: str) -> int:
    """Returns the leading dimension (elements) of a 2-D row-major (possibly padded) tensor."""
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError(f"{name}: expected a 2-D tensor with unit inner stride, got shape {tuple(t.shape)} strides {t.stride()}")
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


def _f32_vector(t, n: int, name: str):
    """Checks that t is a contiguous 1-D fp32 tensor of exactly n elements: the kernels read it through a raw pointer."""
    if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or t.dim() != 1 or not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous 1-D float32 tensor, got "
                         f"{getattr(t, 'dtype', type(t).__name__)} {tuple(getattr(t, 'shape', ()))}")
    if t.numel() != n:
        raise ValueError(f"{name}: expected {n} elements, got {t.numel()}")


def _f32_matrix(t, name: str):
    """Checks that t is a 2-D fp32 tensor with unit inner stride and returns its leading dimension."""
    if not isinstance(t, torch.Tensor) or t.dtype != torch.float32:
        raise ValueError(f"{name}: expected a float32 tensor, got {getattr(t, 'dtype', type(t).__name__)}")
    return _row_major(t, name)


def _time_emb_weights(emb_w, emb_b) -> int:
    """The d x d time-embedding Linear (weight row-major and dense, as the kernels index it): returns d."""
    if not isinstance(emb_w, torch.Tensor) or emb_w.dtype != torch.float32 or emb_w.dim() != 2 \
            or emb_w.shape[0] != emb_w.shape[1] or not emb_w.is_contiguous():
        raise ValueError(f"emb_w: expected a contiguous square float32 matrix, got "
                         f"{getattr(emb_w, 'dtype', type(emb_w).__name__)} {tuple(getattr(emb_w, 'shape', ()))}")
    d = emb_w.shape[0]
    _f32_vector(emb_b, d, "emb_b")
    return d


# ----------------------------------------------------------------------------------------- packing
def pack_bf16(src: torch.Tensor, ld_dst: Optional[int] = None, transpose: bool = False, split: bool = True):
    """fp32 [R, C] -> (hi, lo) bf16 [R, ld] (or [C, ld] transposed); lo is None when split=False."""
    assert src.dtype == torch.float32
    ld_src = _row_major(src, "src")
    R, Cc = src.shape
    out_rows, inner = (Cc, R) if transpose else (R, Cc)
    ld = pad_to(inner, 64) if ld_dst is None else ld_dst
    hi = torch.empty((out_rows, ld), dtype=torch.bfloat16, device=src.device)
    lo = torch.empty_like(hi) if split else None
    _lib.call("dmm_pack_bf16", _ctx(src), _p(src), R, Cc, ld_src, _p(hi), _p(lo), ld, int(transpose), _stream())
    return hi, lo


def pack_bf16_pair(src: torch.Tensor, split: bool = True):
    """fp32 [R, C] -> ((hi, lo) [R, pad64(C)], (hi, lo) [C, pad64(R)]): both orientations from one read of src."""
    assert src.dtype == torch.float32
    ld_src = _row_major(src, "src")
    R, Cc = src.shape
    ld_n, ld_t = pad_to(Cc, 64), pad_to(R, 64)
    bf = dict(dtype=torch.bfloat16, device=src.device)
    n_hi, t_hi = torch.empty((R, ld_n), **bf), torch.empty((Cc, ld_t), **bf)
    n_lo, t_lo = (torch.empty_like(n_hi), torch.empty_like(t_hi)) if split else (None, None)
    _lib.call("dmm_pack_bf16_pair", _ctx(src), _p(src), R, Cc, ld_src, _p(n_hi), _p(n_lo), ld_n, _p(t_hi), _p(t_lo), ld_t,
              _stream())
    return (n_hi, n_lo), (t_hi, t_lo)


def pack_bf16_into(src: torch.Tensor, hi: torch.Tensor, lo: Optional[torch.Tensor], transpose: bool = False):
    ld_src = _row_major(src, "src")
    ld = _row_major(hi, "hi")
    R, Cc = src.shape
    _lib.call("dmm_pack_bf16", _ctx(src), _p(src), R, Cc, ld_src, _p(hi), _p(lo), ld, int(transpose), _stream())


def csr_rows_to_dense(indptr, indices, n_rows, n_cols, *, row_ids=None, row0=0, x_f32=None, a_bf16=None):
    """Binary CSR rows -> dense fp32 tile and/or bf16 operand tile (zero filled to n_cols)."""
    assert indptr.dtype == torch.int64 and indices.dtype == torch.int32
    ld_x = _row_major(x_f32, "x_f32") if x_f32 is not None else 0
    ld_a = _row_major(a_bf16, "a_bf16") if a_bf16 is not None else 0
    _lib.call("dmm_csr_rows_to_dense", _ctx(indptr), _p(indptr), _p(indices), _p(row_ids), int(row0), int(n_rows),
              int(n_cols), _p(x_f32), ld_x, _p(a_bf16), ld_a, _stream())


def time_embedding(emb_w, emb_b, n_rows, *, t=None, t_all=0, a_hi=None, a_lo=None, col0=0, temb_f32=None):
    d = _time_emb_weights(emb_w, emb_b)
    ld_a = _row_major(a_hi, "a_hi") if a_hi is not None else 0
    _lib.call("dmm_time_embedding", _ctx(emb_w), _p(t), int(t_all), int(n_rows), int(d), _p(emb_w), _p(emb_b),
              _p(a_hi), _p(a_lo), ld_a, int(col0), _p(temb_f32), _stream())


def time_bias(emb_w, emb_b, weight, col0, bias, t0, n_t=1, out=None):
    """bias_eff[i] = bias + weight[:, col0:col0+d] @ temb(t0 + i), i < n_t (fp32 [n_t, H]); weight is the fp32
    [H, K] Linear weight."""
    d = _time_emb_weights(emb_w, emb_b)
    ld_w = _f32_matrix(weight, "weight")
    H = weight.shape[0]
    if not 0 <= col0 <= weight.shape[1] - d:
        raise ValueError(f"weight: columns col0 .. col0 + d = {col0} .. {col0 + d} outside its {weight.shape[1]} columns")
    if bias is not None:
        _f32_vector(bias, H, "bias")
    if out is None:
        out = torch.empty((n_t, H), dtype=torch.float32, device=weight.device)
    assert out.is_contiguous() and out.numel() >= n_t * H
    _lib.call("dmm_time_bias", _ctx(weight), int(t0), int(n_t), int(d), _p(emb_w), _p(emb_b), _p(weight),
              ld_w, int(col0), _p(bias), H, _p(out), _stream())
    return out


_GATHER_SPLIT = os.environ.get("DIFFMM_GATHER_SPLIT", "1") != "0"


def csr_gather_act(indptr, indices, n_rows, n_cols, wt_hi, wt_lo, bias, act, n_out, h_hi, h_lo, *, row_ids=None, row0=0,
                   z_f32=None, order=None, vals=None):
    """h = act(bias + sum of the rows of W^T selected by each binary CSR row) -> bf16 hi (+ lo); z_f32 (optional)
    receives the sums without bias.  order (int32 permutation of the rows): scheduling order, e.g. longest rows first.
    vals (fp32, indexed like indices): entry values of non-binary sparse rows (csr_qsample_values)."""
    assert indptr.dtype == torch.int64 and indices.dtype == torch.int32
    assert order is None or (order.dtype == torch.int32 and order.numel() == n_rows)
    assert vals is None or (vals.dtype == torch.float32 and vals.numel() == indices.numel())
    counters = getattr(order, "_dmm_counters", None) if order is not None else None
    if counters is not None and n_out <= 1024 and _GATHER_SPLIT:
        # rows divided by length inside one launch (order / counters from rows_long_first): bit-identical results
        max_long = indices.numel() // (order._dmm_threshold + 1)
        _lib.call("dmm_csr_gather_act_split", _ctx(indptr), _p(indptr), _p(indices), _p(vals), _p(row_ids), _p(order),
                  _p(counters), int(max_long), int(row0), int(n_rows), int(n_cols), _p(wt_hi), _p(wt_lo),
                  _row_major(wt_hi, "wt_hi"), _p(bias), int(act), int(n_out), _p(h_hi), _p(h_lo), _row_major(h_hi, "h_hi"),
                  _p(z_f32), _row_major(z_f32, "z_f32") if z_f32 is not None else 0, _stream())
        return
    _lib.call("dmm_csr_gather_act", _ctx(indptr), _p(indptr), _p(indices), _p(vals), _p(row_ids), _p(order), int(row0), int(n_rows),
              int(n_cols),
              _p(wt_hi), _p(wt_lo), _row_major(wt_hi, "wt_hi"), _p(bias), int(act), int(n_out), _p(h_hi), _p(h_lo),
              _row_major(h_hi, "h_hi"), _p(z_f32), _row_major(z_f32, "z_f32") if z_f32 is not None else 0, _stream())


def csr_qsample_values(indptr, indices, n_rows, n_cols, noise, coef_a, coef_b, vals, *, row_ids=None, row0=0):
    """vals[e] = coef_a + coef_b * noise[r, indices[e]] / max(||noise[r]||, 1e-12) for the entries of the selected binary
    rows: the default-noise q_sample (Model.py:324-341) keeps a binary row's sparsity pattern."""
    assert noise.dtype == torch.float32 and vals.dtype == torch.float32 and vals.numel() == indices.numel()
    _lib.call("dmm_csr_qsample_values", _ctx(indptr), _p(indptr), _p(indices), _p(row_ids), int(row0), int(n_rows), int(n_cols),
              _p(noise), _row_major(noise, "noise"), float(coef_a), float(coef_b), _p(vals), _stream())
    return vals


def csr_qsample_values_rng(indptr, indices, n_rows, n_cols, seed, coef_a, coef_b, vals, *, row_ids=None, row0=0,
                           full_rows=False):
    """csr_qsample_values with the N(0, 1) rows generated inside the kernel (Philox keyed by the device int64 `seed`).
    full_rows=False draws only the support normals and one chi-square variate for the rest of the squared norm (the
    same joint distribution of the outputs, O(k) per row)."""
    assert seed.dtype == torch.int64 and seed.is_cuda and vals.dtype == torch.float32 and vals.numel() == indices.numel()
    _lib.call("dmm_csr_qsample_values_rng", _ctx(indptr), _p(indptr), _p(indices), _p(row_ids), int(row0), int(n_rows),
              int(n_cols), _p(seed), float(coef_a), float(coef_b), _p(vals), int(bool(full_rows)), _stream())
    return vals


def rows_long_first(indptr, row0, n_rows, threshold=32):
    """int32 permutation of the block's rows with the rows of more than `threshold` entries in front (scheduling order
    of csr_gather_act; arbitrary among equals)."""
    order = torch.empty(n_rows, dtype=torch.int32, device=indptr.device)
    counters = torch.empty(2, dtype=torch.int32, device=indptr.device)
    _lib.call("dmm_rows_long_first", _ctx(indptr), _p(indptr), int(row0), int(n_rows), int(threshold), _p(order), _p(counters),
              _stream())
    # counters[0] = number of long rows (device scalar): csr_gather_act divides the launch by it
    order._dmm_counters, order._dmm_threshold = counters, int(threshold)
    return order


def gemv_f32(w, K, x, out=None):
    """y = w[:, :K] @ x (fp32)."""
    ld_w = _f32_matrix(w, "w")
    n_rows = w.shape[0]
    if not 0 < K <= w.shape[1]:
        raise ValueError(f"K = {K} outside 1..{w.shape[1]} (the columns of w)")
    _f32_vector(x, K, "x")
    if out is None:
        out = torch.empty(n_rows, dtype=torch.float32, device=w.device)
    _f32_vector(out, n_rows, "out")
    _lib.call("dmm_gemv_f32", _ctx(w), _p(w), ld_w, int(n_rows), int(K), _p(x), _p(out), _stream())
    return out


def bias_act_pack(z, bias, act, h_hi, h_lo=None):
    """h = act(z + bias) -> bf16 hi (+ lo)."""
    ld_z = _f32_matrix(z, "z")
    n_rows, n_cols = z.shape
    if bias is not None:
        _f32_vector(bias, n_cols, "bias")
    _lib.call("dmm_bias_act_pack", _ctx(z), _p(z), ld_z, _p(bias), int(n_rows), int(n_cols), int(act), _p(h_hi),
              _p(h_lo), _row_major(h_hi, "h_hi"), _stream())


def csr_axpy_bf16(indptr, indices, n_rows, n_cols, beta, x_hi, x_lo, *, row_ids=None, row0=0):
    """x[r, c] += beta at the CSR positions (x as bf16 hi (+ lo))."""
    _lib.call("dmm_csr_axpy_bf16", _ctx(indptr), _p(indptr), _p(indices), _p(row_ids), int(row0), int(n_rows), int(n_cols),
              float(beta), _p(x_hi), _p(x_lo), _row_major(x_hi, "x_hi"), _stream())


def q_sample(x0, noise, coef_a, coef_b, mode, *, x_t=None, a_hi=None, a_lo=None):
    """x_t = a[r] x0 + b[r] noise (mode 0) or the default sign(x0)*normalize(noise) (mode 1)."""
    n_rows, n_cols = x0.shape
    _lib.call("dmm_q_sample", _ctx(x0), _p(x0), _row_major(x0, "x0"), _p(noise), _row_major(noise, "noise"),
              _p(coef_a), _p(coef_b), n_rows, n_cols, int(mode), _p(x_t),
              _row_major(x_t, "x_t") if x_t is not None else 0, _p(a_hi), _p(a_lo),
              _row_major(a_hi, "a_hi") if a_hi is not None else 0, _stream())


# ----------------------------------------------------------------------------------------- GEMM
def _epilogue(bias, act, alpha, beta, residual, out_f32, out_hi, out_lo, res_hi=None, res_lo=None, res_pre_act=False,
              post_bias=None, post_act=0, cmax=None):
    ep = GemmEpilogue()
    ep.cmax = cmax.data_ptr() if cmax is not None else None
    ep.ld_cmax = _row_major(cmax, "cmax") if cmax is not None else 0
    ep.res_pre_act = int(bool(res_pre_act))
    ep.post_act = int(post_act)
    ep.post_bias = post_bias.data_ptr() if post_bias is not None else None
    ep.res_hi = res_hi.data_ptr() if res_hi is not None else None
    ep.res_lo = res_lo.data_ptr() if res_lo is not None else None
    ep.ld_res16 = _row_major(res_hi, "res_hi") if res_hi is not None else 0
    ep.bias = bias.data_ptr() if bias is not None else None
    ep.act = int(act)
    ep.alpha = float(alpha)
    ep.beta = float(beta)
    ep.residual = residual.data_ptr() if residual is not None else None
    ep.ld_res = _row_major(residual, "residual") if residual is not None else 0
    ep.out_f32 = out_f32.data_ptr() if out_f32 is not None else None
    ep.ld_out = _row_major(out_f32, "out_f32") if out_f32 is not None else 0
    ep.out_hi = out_hi.data_ptr() if out_hi is not None else None
    ep.out_lo = out_lo.data_ptr() if out_lo is not None else None
    ep.ld_out16 = _row_major(out_hi, "out_hi") if out_hi is not None else 0
    return ep


def gemm_bf16_tn(a_hi, a_lo, b_hi, b_lo, M, N, K, *, bias=None, act=0, alpha=1.0, beta=0.0, residual=None,
                 out_f32=None, out_hi=None, out_lo=None, res_hi=None, res_lo=None, res_pre_act=False,
                 post_bias=None, post_act=0, cmax=None):
    """C[M,N] = epi(A[M,K] . B[N,K]^T) on tcgen05; lo operands add the split-bf16 correction passes.
    cmax (fp32 [M, >= ceil(N/32)]): per-row maxima of the 32-column chunks of the result (top-k pruning side array).
    The residual of the epilogue (alpha * v + beta * R) is fp32 (`residual`) or bf16 hi(+lo) (`res_hi/res_lo`);
    with res_pre_act it is a partial sum of the same contraction and enters before the activation.
    post_bias / post_act: the bf16 output gets post_act(v + post_bias) while out_f32 keeps v."""
    ep = _epilogue(bias, act, alpha, beta, residual, out_f32, out_hi, out_lo, res_hi, res_lo, res_pre_act, post_bias,
                   post_act, cmax)
    _lib.call("dmm_gemm_bf16_tn", _ctx(a_hi), _p(a_hi), _p(a_lo), _row_major(a_hi, "a_hi"), _p(b_hi), _p(b_lo),
              _row_major(b_hi, "b_hi"), int(M), int(N), int(K), C.byref(ep), _stream())


def gemm_bf16_tn_splitk(a_hi, b_hi, M, N, K, *, out_f32=None, out_hi=None, out_lo=None):
    """C = A . B^T (single-pass bf16, no epilogue terms) with the k blocks of every tile divided over several work items
    when the output has few tiles and K is long (dmm_gemm_bf16_tn_splitk); plain contraction otherwise."""
    ctx = _ctx(a_hi)
    ws_bytes = int(_lib.load().dmm_gemm_splitk_workspace_bytes(ctx, int(M), int(N), int(K)))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=a_hi.device) if ws_bytes > 0 else None
    _lib.call("dmm_gemm_bf16_tn_splitk", ctx, _p(a_hi), _row_major(a_hi, "a_hi"), _p(b_hi), _row_major(b_hi, "b_hi"), int(M),
              int(N), int(K), _p(out_f32), _row_major(out_f32, "out_f32") if out_f32 is not None else 0, _p(out_hi), _p(out_lo),
              _row_major(out_hi, "out_hi") if out_hi is not None else 0, _p(ws), ws_bytes, _stream())


def gemm_f32_tn(a, b, M, N, K, *, bias=None, act=0, alpha=1.0, beta=0.0, residual=None, out_f32=None,
                out_hi=None, out_lo=None, res_pre_act=False, post_bias=None, post_act=0):
    ep = _epilogue(bias, act, alpha, beta, residual, out_f32, out_hi, out_lo, None, None, res_pre_act, post_bias, post_act)
    _lib.call("dmm_gemm_f32_tn", _ctx(a), _p(a), _row_major(a, "a"), _p(b), _row_major(b, "b"), int(M), int(N), int(K),
              C.byref(ep), _stream())


# ----------------------------------------------------------------------------------------- top-k
def topk_edges(scores, n_cols, out_ptr, row_base, out_users, out_items, status=None, order=None):
    """Emits, for each row r, the (out_ptr[r+1]-out_ptr[r]) largest columns (ascending) at out_ptr[r].
    order (int32 permutation of the rows): scheduling order, e.g. largest k first.  Rows wider than 8192 columns use
    the column-segment pass + merge (a temporary list of segments x emitted entries, bounded by out_items.numel())."""
    assert scores.dtype == torch.float32 and out_ptr.dtype == torch.int64 and out_items.dtype == torch.int32
    n_rows = scores.shape[0]
    assert out_ptr.numel() >= n_rows + 1
    n_edges = int(out_items.numel())
    ws_bytes = int(_lib.load().dmm_topk_workspace_bytes(int(n_cols), n_edges))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=scores.device) if ws_bytes > 0 else None
    _lib.call("dmm_topk_edges", _ctx(scores), _p(scores), _row_major(scores, "scores"), n_rows, int(n_cols), _p(out_ptr),
              int(row_base), _p(out_users), _p(out_items), _p(status), _p(order), _p(ws), ws_bytes, n_edges, _stream())


def cmax_buffer(n_rows: int, n_cols: int, device) -> torch.Tensor:
    """fp32 [n_rows, pad4(ceil(n_cols / 32))] side array for gemm_bf16_tn(cmax=...) / topk_edges_pruned."""
    return torch.empty((n_rows, pad_to((n_cols + 31) // 32, 4)), dtype=torch.float32, device=device)


def topk_edges_pruned(scores, n_cols, cmax, out_ptr, row_base, out_users, out_items, status=None, order=None):
    """topk_edges for scores whose producer also wrote the per-chunk maxima `cmax` (gemm_bf16_tn(cmax=...)): reads only
    the chunks that can hold a row's k largest scores.  Same output, bit for bit."""
    assert scores.dtype == torch.float32 and cmax.dtype == torch.float32 and out_ptr.dtype == torch.int64
    assert out_items.dtype == torch.int32
    n_rows = scores.shape[0]
    assert out_ptr.numel() >= n_rows + 1 and cmax.shape[0] >= n_rows
    n_edges = int(out_items.numel())
    ws_bytes = int(_lib.load().dmm_topk_pruned_workspace_bytes(n_rows, int(n_cols), n_edges))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=scores.device)
    _lib.call("dmm_topk_edges_pruned", _ctx(scores), _p(scores), _row_major(scores, "scores"), n_rows, int(n_cols), _p(cmax),
              _row_major(cmax, "cmax"), _p(out_ptr), int(row_base), _p(out_users), _p(out_items), _p(status), _p(order),
              _p(ws), ws_bytes, n_edges, _stream())


# ----------------------------------------------------------------------------------------- adjacency
@dataclass
class CsrAdj:
    """Normalised bipartite adjacency D^-1/2 ([[0,R],[R^T,0]] + I) D^-1/2 in CSR over N = U + I nodes."""
    ptr: torch.Tensor      # int64 [N+1]
    idx: torch.Tensor      # int32 [2E+N], ascending inside each row
    val: torch.Tensor      # fp32  [2E+N]
    n_users: int
    n_items: int
    plan: Optional[torch.Tensor] = None        # long-row plan of the SpMM (dmm_spmm_plan), built on first use
    workspace: Optional[torch.Tensor] = None   # partial rows of the planned chunks
    separable: bool = False                    # val[r, c] = d_r^-1/2 d_c^-1/2 with d_r = entries of row r (D^-1/2 (A + I) D^-1/2)

    @property
    def n_nodes(self):
        return self.n_users + self.n_items

    @property
    def nnz(self):
        return self.idx.numel()

    def to_torch_coo(self):
        """Torch sparse COO view (int64 indices) for callers that still use torch.sparse.mm."""
        counts = (self.ptr[1:] - self.ptr[:-1])
        rows = torch.repeat_interleave(torch.arange(self.n_nodes, device=self.ptr.device), counts)
        return torch.sparse_coo_tensor(torch.stack([rows, self.idx.long()]), self.val, (self.n_nodes, self.n_nodes))


def build_norm_adj(row_ptr: torch.Tensor, items: torch.Tensor, n_users: int, n_items: int,
                   status: Optional[torch.Tensor] = None) -> CsrAdj:
    """status (optional int32 [1] on the device): bit 1 is OR-ed in when an item id is out of range."""
    assert row_ptr.dtype == torch.int64 and items.dtype == torch.int32
    E = int(items.numel())
    N = n_users + n_items
    dev = row_ptr.device
    lib = _lib.load()
    ws_bytes = int(lib.dmm_build_adj_workspace_bytes(n_users, n_items, E))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    ptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
    idx = torch.empty(2 * E + N, dtype=torch.int32, device=dev)
    val = torch.empty(2 * E + N, dtype=torch.float32, device=dev)
    _lib.call("dmm_build_norm_adj_csr", _ctx(row_ptr), _p(row_ptr), _p(items), n_users, n_items, E, _p(ptr), _p(idx),
              _p(val), _p(ws), ws_bytes, _p(status), _stream())
    return CsrAdj(ptr, idx, val, n_users, n_items, separable=True)


# ----------------------------------------------------------------------------------------- SpMM
def _ensure_plan(adj: CsrAdj, device):
    if adj.plan is None:
        lib = _lib.load()
        nnz = int(adj.nnz)
        adj.plan = torch.empty(int(lib.dmm_spmm_plan_bytes(adj.n_nodes, nnz)), dtype=torch.uint8, device=device)
        adj.workspace = torch.empty(int(lib.dmm_spmm_workspace_bytes(nnz, 64)), dtype=torch.uint8, device=device)
        _lib.call("dmm_spmm_plan", _ctx(adj.ptr), _p(adj.ptr), adj.n_nodes, nnz, _p(adj.plan), adj.plan.numel(), _stream())


def spmm_table_bf16(adj: CsrAdj, x: torch.Tensor, x2: Optional[torch.Tensor] = None, table: Optional[torch.Tensor] = None):
    """Gather table of spmm_norm_bf16: T = bf16(d^-1/2 [x ; x2]) [N, 64] (the concatenation is never materialised)."""
    assert adj.separable, "the bf16 propagation needs val = d_r^-1/2 d_c^-1/2 (build_norm_adj / normalizeAdj adjacencies)"
    n_first = x.shape[0]
    assert x.dtype == torch.float32 and x.shape[1] == 64 and n_first + (x2.shape[0] if x2 is not None else 0) == adj.n_nodes
    assert x2 is None or (x2.dtype == torch.float32 and x2.shape[1] == 64)
    _ensure_plan(adj, x.device)
    if table is None:
        table = torch.empty((adj.n_nodes, 64), dtype=torch.bfloat16, device=x.device)
    _lib.call("dmm_spmm_table_bf16", _ctx(x), _p(x), _row_major(x, "x"), n_first, _p(x2),
              _row_major(x2, "x2") if x2 is not None else 0, adj.n_nodes, _p(adj.plan), int(adj.nnz), _p(table), _stream())
    return table


def spmm_norm_bf16(adj: CsrAdj, x: Optional[torch.Tensor] = None, *, x2=None, table=None, alpha=1.0, beta=0.0, z=None, out=None,
                   row0=0, row1=None):
    """out[row0:row1] = alpha * A[row0:row1] . [x ; x2] (+ beta * z[row0:row1]) in the single-pass bf16 precision of the
    propagation: the gathered operand is rounded to bf16 once (T = bf16(d^-1/2 X), built here unless `table` is given),
    sums, row scaling and output are fp32.  Separable adjacencies only (CsrAdj.separable)."""
    if table is None:
        table = spmm_table_bf16(adj, x, x2)
    else:
        _ensure_plan(adj, table.device)
    assert table.dtype == torch.bfloat16 and table.shape == (adj.n_nodes, 64) and table.is_contiguous()
    if out is None:
        out = torch.empty((adj.n_nodes, 64), dtype=torch.float32, device=table.device)
    row1 = adj.n_nodes if row1 is None else row1
    _lib.call("dmm_spmm_norm_bf16", _ctx(table), _p(adj.idx), int(row0), int(row1), adj.n_nodes, _p(table), float(alpha),
              float(beta), _p(z), _row_major(z, "z") if z is not None else 0, _p(out), _row_major(out, "out"), _p(adj.plan),
              int(adj.nnz), _p(adj.workspace), adj.workspace.numel(), _stream())
    return out


# (fp32 gather table: every adjacency)
def spmm(adj: CsrAdj, x: torch.Tensor, *, alpha=1.0, beta=0.0, z=None, out=None, row0=0, row1=None):
    """out[row0:row1] = alpha * A[row0:row1] . x (+ beta * z[row0:row1]); rows outside the block untouched."""
    assert x.dtype == torch.float32 and x.shape[0] == adj.n_nodes
    D = x.shape[1]
    if out is None:
        out = torch.empty((adj.n_nodes, D), dtype=torch.float32, device=x.device)
    row1 = adj.n_nodes if row1 is None else row1
    nnz = int(adj.nnz)
    if D == 64:
        _ensure_plan(adj, x.device)
    plan, ws = (adj.plan, adj.workspace) if D == 64 else (None, None)
    _lib.call("dmm_spmm_csr", _ctx(x), _p(adj.ptr), _p(adj.idx), _p(adj.val), int(row0), int(row1), _p(x),
              _row_major(x, "x"), D, float(alpha), float(beta), _p(z), _row_major(z, "z") if z is not None else 0,
              _p(out), _row_major(out, "out"), _p(plan), nnz, _p(ws), ws.numel() if ws is not None else 0, _stream())
    return out


def spmm_replan(adj: CsrAdj):
    """Rebuilds the long-row plan of ``adj`` in place after its arrays were overwritten (same buffers: captured
    CUDA graphs keep pointing at them)."""
    if adj.plan is not None:
        _lib.call("dmm_spmm_plan", _ctx(adj.ptr), _p(adj.ptr), adj.n_nodes, int(adj.nnz), _p(adj.plan), adj.plan.numel(),
                  _stream())


def sign_noise_(e: torch.Tensor, rnd: torch.Tensor, noise_degree: float):
    """In place e += sign(e) * normalize_rows(rnd) * noise_degree (Main.py:320-321)."""
    _lib.call("dmm_sign_noise_", _ctx(e), _p(e), _row_major(e, "e"), _p(rnd), _row_major(rnd, "rnd"), e.shape[0],
              e.shape[1], float(noise_degree), _stream())
    return e


# ----------------------------------------------------------------------------------------- gcn_MM glue
def rownorm_fwd(x: torch.Tensor, eps: float = 1e-12):
    """F.normalize(x) per row (Model.py:89-93): returns (y, inv); inv < 0 flags a row clamped at eps."""
    assert x.dtype == torch.float32 and x.dim() == 2
    y = torch.empty((x.shape[0], x.shape[1]), dtype=torch.float32, device=x.device)
    inv = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
    _lib.call("dmm_rownorm_fwd", _ctx(x), _p(x), _row_major(x, "x"), x.shape[0], x.shape[1], float(eps), _p(y), y.shape[1], _p(inv),
              _stream())
    return y, inv


def rownorm_bwd(y: torch.Tensor, inv: torch.Tensor, g: torch.Tensor):
    gx = torch.empty_like(y)
    _lib.call("dmm_rownorm_bwd", _ctx(y), _p(y), _row_major(y, "y"), _p(inv), _p(g), _row_major(g, "g"), y.shape[0], y.shape[1],
              _p(gx), gx.shape[1], _stream())
    return gx


def _ptr_array(tensors):
    return (C.c_void_p * len(tensors))(*[t.data_ptr() if t is not None else None for t in tensors])


def _dense(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_contiguous() or t.dtype != torch.float32:
        raise _lib.DiffMMError(f"{name}: dense contiguous fp32 tensor expected")
    return t


def modal_mix_fwd(y: torch.Tensor, zs, w: torch.Tensor, lam: float):
    """sum_m w[m] (y + lam zs[m]) (Model.py:116-119,125-127); w: device fp32 [M]."""
    y = _dense(y, "y")
    zs = [_dense(z, "z") for z in zs]
    out = torch.empty_like(y)
    arr = _ptr_array(zs)
    _lib.call("dmm_modal_mix_fwd", _ctx(y), _p(y), arr, _p(w), len(zs), float(lam), y.numel(), _p(out), _stream())
    return out


def modal_mix_bwd(g: torch.Tensor, y: torch.Tensor, zs, w: torch.Tensor, lam: float, need_gz=True):
    """Returns (gy, [gz_m], gw [M]) of modal_mix_fwd; gw from per-CTA partial sums added in a fixed order."""
    g = _dense(g, "g")
    M = len(zs)
    gy = torch.empty_like(y)
    gzs = [torch.empty_like(y) if need_gz else None for _ in range(M)]
    rows = (y.numel() // 4 + 255) // 256
    partial = torch.empty((rows, M), dtype=torch.float32, device=y.device)
    az, agz = _ptr_array(zs), _ptr_array(gzs)
    _lib.call("dmm_modal_mix_bwd", _ctx(y), _p(g), _p(y), az, _p(w), M, float(lam), y.numel(), _p(gy), agz, _p(partial), _stream())
    return gy, gzs, partial.sum(0)


# ----------------------------------------------------------------------------------------- losses
def bpr_fwd_bwd(u_emb, i_emb, users, pos, neg, grad_scale=1.0, want_grad=True):
    B, D = users.numel(), u_emb.shape[1]
    dev = u_emb.device
    row_loss = torch.empty(B, dtype=torch.float32, device=dev)
    loss = torch.empty((), dtype=torch.float32, device=dev)
    g = [torch.empty((B, D), dtype=torch.float32, device=dev) for _ in range(3)] if want_grad else [None] * 3
    _lib.call("dmm_bpr_fwd_bwd", _ctx(u_emb), _p(u_emb), _row_major(u_emb, "u_emb"), _p(i_emb), _row_major(i_emb, "i_emb"),
              _p(users), _p(pos), _p(neg), B, D, float(grad_scale), _p(row_loss), _p(loss), _p(g[0]), _p(g[1]), _p(g[2]),
              _stream())
    return loss, g


def infonce_fwd(v1, v2, idx, temperature):
    B, D = idx.numel(), v1.shape[1]
    dev = v1.device
    ws = torch.empty(int(_lib.load().dmm_infonce_workspace_floats(B, D, 0)), dtype=torch.float32, device=dev)
    row_loss = torch.empty(B, dtype=torch.float32, device=dev)
    loss = torch.empty((), dtype=torch.float32, device=dev)
    lse = torch.empty(B, dtype=torch.float32, device=dev)
    inv1 = torch.empty(B, dtype=torch.float32, device=dev)
    inv2 = torch.empty(B, dtype=torch.float32, device=dev)
    _lib.call("dmm_infonce_fwd", _ctx(v1), _p(v1), _row_major(v1, "v1"), _p(v2), _row_major(v2, "v2"), _p(idx), B, D,
              float(temperature), _p(ws), _p(row_loss), _p(loss), _p(lse), _p(inv1), _p(inv2), _stream())
    return loss, (lse, inv1, inv2)


def infonce_bwd(v1, v2, idx, temperature, saved, grad_scale=1.0):
    B, D = idx.numel(), v1.shape[1]
    dev = v1.device
    lse, inv1, inv2 = saved
    ws = torch.empty(int(_lib.load().dmm_infonce_workspace_floats(B, D, 1)), dtype=torch.float32, device=dev)
    g1 = torch.empty((B, D), dtype=torch.float32, device=dev)
    g2 = torch.empty((B, D), dtype=torch.float32, device=dev)
    _lib.call("dmm_infonce_bwd", _ctx(v1), _p(v1), _row_major(v1, "v1"), _p(v2), _row_major(v2, "v2"), _p(idx), B, D,
              float(temperature), _p(lse), _p(inv1), _p(inv2), float(grad_scale), _p(ws), _p(g1), _p(g2), _stream())
    return g1, g2


def scatter_add_rows(src, idx, dst):
    _lib.call("dmm_scatter_add_rows", _ctx(src), _p(src), _row_major(src, "src"), _p(idx), idx.numel(), src.shape[1],
              _p(dst), _row_major(dst, "dst"), _stream())
    return dst


# ----------------------------------------------------------------------------------------- evaluation
def eval_mask_scores(indptr, indices, row_ids, scores, n_cols, fill=-1e8):
    """scores[r, train items of user row_ids[r]] = fill (Main.py:410 without dense mask rows)."""
    assert row_ids.dtype == torch.int64 and scores.dtype == torch.float32
    _lib.call("dmm_eval_mask_scores", _ctx(scores), _p(indptr), _p(indices), _p(row_ids), int(row_ids.numel()), int(n_cols),
              _p(scores), _row_major(scores, "scores"), float(fill), _stream())


def eval_metrics(scores, top_items, K, row_ids, test_ptr, test_items, inv_log2, max_dcg, out):
    """out[r] = (recall, ndcg, precision) of user row_ids[r] in float64 (Main.py:422-448)."""
    assert out.dtype == torch.float64 and inv_log2.dtype == torch.float64 and max_dcg.dtype == torch.float64
    assert top_items.dtype == torch.int32 and test_items.dtype == torch.int32 and test_ptr.dtype == torch.int64
    _lib.call("dmm_eval_metrics", _ctx(scores), _p(scores), _row_major(scores, "scores"), int(row_ids.numel()), _p(top_items),
              int(K), _p(row_ids), _p(test_ptr), _p(test_items), _p(inv_log2), _p(max_dcg), _p(out), _stream())
    return out


def eval_mask_scores_cmax(indptr, indices, row_ids, scores, n_cols, cmax, fill=-1e8):
    """eval_mask_scores, then the chunk maxima cmax (gemm_bf16_tn(cmax=...)) of every chunk it wrote are recomputed, so
    topk_edges_pruned stays exact on the masked scores."""
    assert row_ids.dtype == torch.int64 and scores.dtype == torch.float32 and cmax.dtype == torch.float32
    _lib.call("dmm_eval_mask_scores_cmax", _ctx(scores), _p(indptr), _p(indices), _p(row_ids), int(row_ids.numel()),
              int(n_cols), _p(scores), _row_major(scores, "scores"), float(fill), _p(cmax), _row_major(cmax, "cmax"), _stream())


def topn_rank(scores, sel, N, items, out_scores):
    """Row r's N selected columns sel[r, :N] (topk_edges with k = N) in rank order (score desc, column asc):
    items int32 [rows, >= N] (-1 where the score is -inf), out_scores fp32 [rows, >= N]."""
    assert scores.dtype == torch.float32 and sel.dtype == torch.int32 and items.dtype == torch.int32
    assert out_scores.dtype == torch.float32
    n_rows = sel.shape[0]
    assert scores.shape[0] >= n_rows and items.shape[0] >= n_rows and out_scores.shape[0] >= n_rows
    _lib.call("dmm_topn_rank", _ctx(scores), _p(scores), _row_major(scores, "scores"), n_rows, _p(sel), _row_major(sel, "sel"),
              int(N), _p(items), _row_major(items, "items"), _p(out_scores), _row_major(out_scores, "out_scores"), _stream())


def score_pairs(user, item, u_idx, i_idx, x3, out):
    """out[p] = score(user[u_idx[p]], item[i_idx[p]]) (fp32 rows; split-bf16 terms, bf16x3 when x3, else bf16); NaN for
    an index out of range."""
    assert user.dtype == torch.float32 and item.dtype == torch.float32 and out.dtype == torch.float32
    assert u_idx.dtype == torch.int64 and i_idx.dtype == torch.int32 and u_idx.numel() == i_idx.numel() <= out.numel()
    assert u_idx.is_contiguous() and i_idx.is_contiguous() and out.is_contiguous()
    _lib.call("dmm_score_pairs", _ctx(user), _p(user), _row_major(user, "user"), user.shape[0], _p(item),
              _row_major(item, "item"), item.shape[0], user.shape[1], _p(u_idx), _p(i_idx), u_idx.numel(), int(bool(x3)),
              _p(out), _stream())
    return out


def rank_candidates(user, item, cand, N, x3, items, out_scores):
    """Row r's candidates cand[r] (int32, -1 = empty) scored for user[r], deduplicated and ranked (score desc, item asc):
    the first N into items int32 [rows, >= N] / out_scores fp32 [rows, >= N], (-1, -inf) past the distinct candidates."""
    assert user.dtype == torch.float32 and item.dtype == torch.float32 and cand.dtype == torch.int32
    assert items.dtype == torch.int32 and out_scores.dtype == torch.float32
    n_rows = cand.shape[0]
    assert user.shape[0] >= n_rows and items.shape[0] >= n_rows and out_scores.shape[0] >= n_rows
    _lib.call("dmm_rank_candidates", _ctx(user), _p(user), _row_major(user, "user"), _p(item), _row_major(item, "item"),
              item.shape[0], user.shape[1], _p(cand), _row_major(cand, "cand"), n_rows, cand.shape[1], int(N), int(bool(x3)),
              _p(items), _row_major(items, "items"), _p(out_scores), _row_major(out_scores, "out_scores"), _stream())


def eval_metrics_cutoffs(ranked, N, cutoffs, row_ids, test_ptr, test_items, inv_log2, max_dcg, out):
    """out[r, j] = (recall, ndcg, precision) at cutoffs[j] (host ints, strictly increasing, <= N) of user row_ids[r]'s
    ranked list ranked[r, :N] in float64 (Main.py:422-448 per prefix)."""
    assert out.dtype == torch.float64 and inv_log2.dtype == torch.float64 and max_dcg.dtype == torch.float64
    assert ranked.dtype == torch.int32 and test_items.dtype == torch.int32 and test_ptr.dtype == torch.int64
    assert row_ids.dtype == torch.int64 and out.is_contiguous() and out.numel() >= row_ids.numel() * len(cutoffs) * 3
    cut = (C.c_int32 * len(cutoffs))(*[int(c) for c in cutoffs])
    _lib.call("dmm_eval_metrics_cutoffs", _ctx(ranked), _p(ranked), _row_major(ranked, "ranked"), int(row_ids.numel()), int(N),
              cut, len(cutoffs), _p(row_ids), _p(test_ptr), _p(test_items), _p(inv_log2), _p(max_dcg), _p(out), _stream())
    return out


# ----------------------------------------------------------------------------------------- fused training step
def train_prep(x0, noise, t, tab_a, tab_b, emb_w, emb_b, a_hi, a_lo, x0_hi, te_raw):
    """x_t = tab_a[t] x0 + tab_b[t] noise and the time-embedding columns as the bf16 operand a_hi (+ a_lo); x0 as a bf16
    operand (optional); te_raw = raw [cos, sin] time features (optional)."""
    B, I = x0.shape
    _lib.call("dmm_train_prep", _ctx(x0), _p(x0), _row_major(x0, "x0"), _p(noise), _row_major(noise, "noise"), _p(t), _p(tab_a),
              _p(tab_b), B, I, int(emb_w.shape[0]), _p(emb_w), _p(emb_b), _p(a_hi), _p(a_lo), _row_major(a_hi, "a_hi"),
              _p(x0_hi), _row_major(x0_hi, "x0_hi") if x0_hi is not None else 0, _p(te_raw), _stream())


def gate_fwd(p, gate_w, gate_b, sig, g_hi, g_lo):
    assert gate_w.shape == (64, 64) and gate_w.is_contiguous() and sig.is_contiguous()
    _lib.call("dmm_gate_fwd", _ctx(p), _p(p), _row_major(p, "p"), p.shape[0], _p(gate_w), _p(gate_b), _p(sig), _p(g_hi), _p(g_lo),
              _row_major(g_hi, "g_hi"), _stream())


def gate_bwd_pre(dg, p, sig, dpre):
    _lib.call("dmm_gate_bwd_pre", _ctx(p), _p(dg), _row_major(dg, "dg"), _p(p), _row_major(p, "p"), _p(sig), p.shape[0], _p(dpre),
              _stream())


def diff_loss_fwd(diff, umd, x0f, ui, t, w_tab, sim_weight, loss, mse, um, stats):
    B, I = diff.shape
    _lib.call("dmm_diff_loss_fwd", _ctx(diff), _p(diff), _row_major(diff, "diff"), B, I, _p(umd), _row_major(umd, "umd"), _p(x0f),
              _row_major(x0f, "x0f"), _p(ui), _row_major(ui, "ui"), _p(t), _p(w_tab), float(sim_weight), _p(loss), _p(mse), _p(um),
              _p(stats), _stream())


def diff_loss_bwd(g_loss, um, ui, stats, t, w_tab, sim_weight, n_cols, cm, dumc_hi, dumc_lo, d_ui):
    B = um.shape[0]
    _lib.call("dmm_diff_loss_bwd", _ctx(um), _p(g_loss), _p(um), _p(ui), _row_major(ui, "ui"), _p(stats), _p(t), _p(w_tab),
              float(sim_weight), B, int(n_cols), _p(cm), _p(dumc_hi), _p(dumc_lo), _row_major(dumc_hi, "dumc_hi"), _p(d_ui),
              _stream())


def hidden_bwd(dh, h_f32, h_hi, h_lo, cm, H, dz, dz_hi, dz_lo, dzt_hi, dzt_lo, hct_hi, hct_lo):
    """dz = cm dh (1 - h^2) (fp32 and operand), dz^T and (cm h)^T; cm None: no row scale (dz = dh (1 - h^2), h^T)."""
    B = dh.shape[0]
    _lib.call("dmm_hidden_bwd", _ctx(dh), _p(dh), _row_major(dh, "dh"), _p(h_f32),
              _row_major(h_f32, "h_f32") if h_f32 is not None else 0, _p(h_hi), _p(h_lo),
              _row_major(h_hi, "h_hi") if h_hi is not None else 0, _p(cm), B,
              int(H), _p(dz), _row_major(dz, "dz"), _p(dz_hi), _p(dz_lo), _row_major(dz_hi, "dz_hi"), _p(dzt_hi), _p(dzt_lo),
              _p(hct_hi), _p(hct_lo), _row_major(dzt_hi, "dzt_hi"), _stream())


def transpose_bf16(src_hi, src_lo, rows, cols, dst_hi, dst_lo):
    _lib.call("dmm_transpose_bf16", _ctx(src_hi), _p(src_hi), _p(src_lo), _row_major(src_hi, "src_hi"), int(rows), int(cols),
              _p(dst_hi), _p(dst_lo), _row_major(dst_hi, "dst_hi"), _stream())


def colsum(src, row_scale=None):
    """out[c] = sum_r row_scale[r] * src[r, c] (fp32; rows added in order)."""
    R, Cc = src.shape
    out = torch.empty(Cc, dtype=torch.float32, device=src.device)
    _lib.call("dmm_colsum", _ctx(src), _p(src), _row_major(src, "src"), R, Cc, _p(row_scale), _p(out), _stream())
    return out


def atb_small(x, y):
    """x^T y for skinny fp32 matrices x [R, m], y [R, n] (m, n <= 64)."""
    R, m = x.shape
    n = y.shape[1]
    ws = torch.empty(int(_lib.load().dmm_atb_small_workspace_floats(m, n)), dtype=torch.float32, device=x.device)
    out = torch.empty((m, n), dtype=torch.float32, device=x.device)
    _lib.call("dmm_atb_small", _ctx(x), _p(x), _row_major(x, "x"), m, _p(y), _row_major(y, "y"), n, R, _p(ws), _p(out), _stream())
    return out


# ----------------------------------------------------------------------------------------- fused BPR + InfoNCE
def _loss_structs(tables, problems, bpr):
    """problems: [(i1, i2, idx, row_offset, temperature, weight)] over `tables`; bpr: (i_table, item_offset, users, pos, neg)."""
    P = len(problems)
    arr = (_lib.NceProblem * P)()
    for k, (i1, i2, idx, off, temp, weight) in enumerate(problems):
        a, b = tables[i1], tables[i2]
        arr[k].v1, arr[k].ld1 = a.data_ptr(), _row_major(a, "view")
        arr[k].v2, arr[k].ld2 = b.data_ptr(), _row_major(b, "view")
        arr[k].idx, arr[k].row_offset = idx.data_ptr(), int(off)
        arr[k].temperature, arr[k].weight = float(temp), float(weight)
    it, item_off, users, pos, neg = bpr
    bp = _lib.BprProblem()
    bp.emb, bp.ld_emb, bp.item_offset = tables[it].data_ptr(), _row_major(tables[it], "emb"), int(item_off)
    bp.users, bp.pos, bp.neg = users.data_ptr(), pos.data_ptr(), neg.data_ptr()
    return arr, bp


def bpr_infonce_fwd(tables, problems, bpr, B):
    """Every loss of a joint step in three launches.  Returns (losses [P + 2]: InfoNCE means, BPR, weighted contrastive
    total; saved = (lse [P, B], inv [P, 2, B]))."""
    P = len(problems)
    dev = tables[0].device
    arr, bp = _loss_structs(tables, problems, bpr)
    ws = torch.empty(int(_lib.load().dmm_bpr_infonce_workspace_floats(B, P, 0)), dtype=torch.float32, device=dev)
    losses = torch.empty(P + 2, dtype=torch.float32, device=dev)
    lse = torch.empty((P, B), dtype=torch.float32, device=dev)
    inv = torch.empty((P, 2, B), dtype=torch.float32, device=dev)
    _lib.call("dmm_bpr_infonce_fwd", _ctx(tables[0]), arr, P, C.byref(bp), int(B), _p(ws), _p(losses), _p(lse), _p(inv), _stream())
    return losses, (lse, inv)


def bpr_infonce_bwd(tables, problems, bpr, B, saved, g_cl, g_bpr, grad_tables):
    """Scatter-adds d(g_bpr BPR + g_cl total) into grad_tables (one zeroed fp32 [N, 64] tensor or None per table)."""
    P = len(problems)
    dev = tables[0].device
    arr, bp = _loss_structs(tables, problems, bpr)
    lse, inv = saved
    ws = torch.empty(int(_lib.load().dmm_bpr_infonce_workspace_floats(B, P, 1)), dtype=torch.float32, device=dev)
    ptrs = (C.c_void_p * (2 * P + 1))()
    lds = (C.c_int64 * (2 * P + 1))()
    slots = [(i1, i2) for (i1, i2, *_rest) in problems]
    for k, (i1, i2) in enumerate(slots):
        for s, it in enumerate((i1, i2)):
            g = grad_tables[it]
            ptrs[2 * k + s] = g.data_ptr() if g is not None else None
            lds[2 * k + s] = _row_major(g, "grad") if g is not None else 0
    gb = grad_tables[bpr[0]]
    ptrs[2 * P] = gb.data_ptr() if gb is not None else None
    lds[2 * P] = _row_major(gb, "grad") if gb is not None else 0
    _lib.call("dmm_bpr_infonce_bwd", _ctx(tables[0]), arr, P, C.byref(bp), int(B), _p(lse), _p(inv), _p(g_cl), _p(g_bpr), _p(ws),
              ptrs, lds, _stream())
