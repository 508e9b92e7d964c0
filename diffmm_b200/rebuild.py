"""Reverse-diffusion chain + per-user top-k graph rebuild, entirely on device.

Replaces, for the rebuild phase of Coach.trainEpoch (reference Main.py:195-253):
  GaussianDiffusion.generate_view / p_mean_variance (Model.py:300-322,357-378) — S x (cat, 2 cuBLAS
  SGEMMs, tanh, axpby), the Python double loop of per-user torch.topk + int(tensor) syncs
  (Main.py:224-230), and the scipy adjacency build + H2D (Main.py:113-116, DataHandler.py:53-93).

Per user block the data flow is
  [dense x_start / sampling_step > 0 only: rows -> bf16 operand tile   dmm_pack_bf16 / dmm_q_sample]
  b1'[i] = b1 + W1[:, I:] temb(i), all i at once                       dmm_time_bias
  for i = S-1..0:
                   h = tanh(x_t W1[:, :I]^T + b1')   (bf16 hi/lo)      dmm_gemm_bf16_tn  (tcgen05)
                     (first step, binary CSR rows: gather-sum of W1^T  dmm_csr_gather_act)
                   x_t = c1[i] (h W2^T + b2) + c2[i] x_t  (bf16 operand in place; fp32 scores at i = 0)
                     (first step: c2 x0 added at the CSR positions     dmm_csr_axpy_bf16)
                   (deeper denoise_dim: h = tanh(h W_k^T + b_k) for each hidden-to-hidden layer in between, dmm_gemm_bf16_tn)
  top-k_u (k_u = deg(u)) -> item ids at the train-CSR offsets          dmm_topk_edges
and once per modality
  edges -> normalised CSR adjacency                                    dmm_build_norm_adj_csr
Users are independent, so blocks can be any size (results do not depend on it) and shard across
ranks with no data-path collective except the final edge all-gather (dist.py).
"""
from __future__ import annotations

import contextlib
import os
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import ops, rng
from .autograd import check_precision, packed_weight, packed_weight_pair


class ChainWorkspace:
    """Device buffers of one user block, reused across steps, modalities and blocks.  ``hidden`` is the width of a
    one-hidden-layer Denoise or the tuple of hidden widths of a deeper one (hidden_widths): the two hidden operand
    buffers are sized by the widest layer, the fp32 state and the time bias by the first (= last) hidden width."""

    def __init__(self, rows: int, n_items: int, hidden, d_emb: int, split: bool, device):
        widths = _widths(hidden)
        self.rows, self.n_items, self.widths, self.d_emb, self.split = rows, n_items, widths, d_emb, split
        self.hidden = widths[0]
        self.ld_a = ops.pad_to(n_items, 64)
        self.ld_x = ops.pad_to(n_items, 32)
        self.ld_h = ops.pad_to(max(widths), 64)
        bf = dict(dtype=torch.bfloat16, device=device)
        self.device = device
        self._a = None            # bf16 operand copy of x_t [rows, ld_a] (+ lo): only the dense-input / full-chain paths
        self.h_hi = torch.empty((rows, self.ld_h), **bf)
        self.h_lo = torch.empty((rows, self.ld_h), **bf) if split else None
        self._h2 = None           # second hidden operand (the hidden-space chain ping-pongs: a step reads h_t, writes h_{t-1};
                                  # so do the hidden-to-hidden layers of a deeper Denoise)
        self.x = torch.empty((rows, self.ld_x), dtype=torch.float32, device=device)
        self.z = None             # fp32 hidden pre-activation state [rows, pad4(hidden)] of the hidden-space chain
        self.bias_eff = None      # [S, hidden] fp32, sized on first use
        self.partial = None       # fp32 partial sums of a K-chunked GEMM1 (scale-out widths only)
        self._cmax = None         # fp32 [rows, pad4(ceil(I / 32))] chunk maxima of the scores (top-k pruning side array)

    def operand(self):
        if self._a is None:
            bf = dict(dtype=torch.bfloat16, device=self.device)
            self._a = (torch.empty((self.rows, self.ld_a), **bf),
                       torch.empty((self.rows, self.ld_a), **bf) if self.split else None)
        return self._a

    def hidden2(self):
        if self._h2 is None:
            bf = dict(dtype=torch.bfloat16, device=self.device)
            self._h2 = (torch.empty((self.rows, self.ld_h), **bf),
                        torch.empty((self.rows, self.ld_h), **bf) if self.split else None)
        return self._h2

    def state(self):
        if self.z is None:
            self.z = torch.empty((self.rows, ops.pad_to(self.hidden, 4)), dtype=torch.float32, device=self.device)
        return self.z

    def chunk_max(self):
        if self._cmax is None:
            self._cmax = ops.cmax_buffer(self.rows, self.n_items, self.device)
        return self._cmax

    def fits(self, rows, n_items, hidden, d_emb, split):
        return (rows <= self.rows and n_items == self.n_items and _widths(hidden) == self.widths and d_emb == self.d_emb
                and split == self.split)


def _widths(hidden) -> Tuple[int, ...]:
    return (int(hidden),) if isinstance(hidden, (int, np.integer)) else tuple(int(w) for w in hidden)


def hidden_widths(den) -> Tuple[int, ...]:
    """Widths of the 2L - 1 hidden activations of a Denoise with denoise_dim = [d_1, ..., d_L], in forward order:
    d_L, d_{L-1}, ..., d_1, ..., d_{L-1}, d_L (Model.py:160-162).  (d_L,) for the shipped one-entry configs."""
    return tuple(int(layer.weight.shape[0]) for layer in list(den.in_layers) + list(den.out_layers)[:-1])


def _layers(den):
    """(first, inner, last) Linear layers of a Denoise: in_layers[0] ([x_t, temb] -> d_L), the 2L - 2 hidden-to-hidden
    layers in forward order (tanh after each, like after the first) and out_layers[-1] (d_L -> items, no activation)."""
    layers = list(den.in_layers) + list(den.out_layers)
    return layers[0], layers[1:-1], layers[-1]


def _inner_operands(inner, split):
    """(W_k hi, lo), b_k, out width, in width of every hidden-to-hidden layer (packed operands are cached per version)."""
    return [(packed_weight(layer.weight, False, split), layer.bias.detach(), layer.weight.shape[0], layer.weight.shape[1])
            for layer in inner]


def _inner_layers(inner_ops, M, h_hi, h_lo, g_hi, g_lo):
    """h <- tanh(h W_k^T + b_k) through the hidden-to-hidden layers (one contraction with a bias + tanh epilogue each),
    ping-ponging between the two operand buffers.  Returns (current, other) with the last activation current."""
    for (w_hi, w_lo), b, n_out, k in inner_ops:
        ops.gemm_bf16_tn(h_hi, h_lo, w_hi, w_lo, M, n_out, k, bias=b, act=1, out_hi=g_hi, out_lo=g_lo)
        h_hi, h_lo, g_hi, g_lo = g_hi, g_lo, h_hi, h_lo
    return h_hi, h_lo, g_hi, g_lo


def chain_mode() -> str:
    """'hidden' (default) or 'full' (DIFFMM_CHAIN=full): see denoise_chain."""
    m = os.environ.get("DIFFMM_CHAIN", "hidden")
    if m not in ("hidden", "full"):
        raise ValueError(f"DIFFMM_CHAIN must be 'hidden' or 'full', got {m!r}")
    return m


def _hidden_operators(den, W1, W2, b2, I, split):
    """P = W1[:, :I] W2 (H x H) and q = W1[:, :I] b2 (H) of the hidden-space chain, cached per weight version and
    precision.  P is one tensor-pipe contraction over the items (three-pass split-bf16, i.e. fp32-faithful, in
    bf16x3 mode; single pass in bf16 mode, where it is then rounded to bf16 like every other operand); q is an
    fp32 matrix-vector product on the master weights."""
    key = (W1._version, W2._version, b2._version, W1.data_ptr(), W2.data_ptr(), split)
    ent = getattr(den, "_dmm_hidden_ops", None)
    if ent is None or ent[0] != key:
        H = W1.shape[0]
        packed_weight_pair(W1, split)                            # both orientations of each weight from one read:
        packed_weight_pair(W2, split)                            # W1 / W1^T (operand, gather table), W2 / W2^T
        w1_hi, w1_lo = packed_weight(W1, False, split)           # [H, pad(I + d)], K-major over items
        w2t_hi, w2t_lo = packed_weight(W2, True, split)          # W2^T [H, pad(I)],  K-major over items
        if split:
            P = torch.empty((H, ops.pad_to(H, 4)), dtype=torch.float32, device=W1.device)[:, :H]
            ops.gemm_bf16_tn(w1_hi, w1_lo, w2t_hi, w2t_lo, H, H, I, out_f32=P)
            p_hi, p_lo = ops.pack_bf16(P, split=True)
        else:
            # single-pass mode: the contraction's epilogue rounds P to the bf16 operand directly (same round-to-nearest
            # as dmm_pack_bf16 on the fp32 result, one launch and one 4 MB round trip fewer)
            ld = ops.pad_to(H, 64)
            p_hi = torch.zeros((H, ld), dtype=torch.bfloat16, device=W1.device) if ld != H else \
                torch.empty((H, ld), dtype=torch.bfloat16, device=W1.device)
            # 16 pair tiles at H = 1024 and a long K: split-K keeps every SM busy (42 -> ~20 us at I = 7050, 2.2 -> 0.6 ms at 500k)
            ops.gemm_bf16_tn_splitk(w1_hi, w2t_hi, H, H, I, out_hi=p_hi[:, :H])
            p_lo = None
        q = ops.gemv_f32(W1.detach(), I, b2.detach())
        ent = (key, p_hi, p_lo, q)
        den._dmm_hidden_ops = ent
    return ent[1], (ent[2] if split else None), ent[3]


def denoise_chain(diff, den, *, x_dense: Optional[torch.Tensor] = None,
                  csr: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, row_ids: Optional[torch.Tensor] = None,
                  row0: int = 0, n_rows: Optional[int] = None, sampling_step: int = 0,
                  precision: Optional[str] = None, ws: Optional[ChainWorkspace] = None,
                  noise: Optional[torch.Tensor] = None, mode: Optional[str] = None,
                  order: Optional[torch.Tensor] = None, want_cmax: bool = False) -> torch.Tensor:
    """generate_view (Model.py:300-322) for a block of users given as dense rows or CSR rows.
    Returns the fp32 [n_rows, I] scores (a view of the workspace: consume before the next call).
    want_cmax: the last contraction also writes the per-row maxima of the 32-column chunks of the scores into
    ``ws.chunk_max()[:n_rows]`` (the pruning side array of ops.topk_edges_pruned).

    mode 'hidden' (default).  Between two tanh's the reverse chain is affine: with z_t = x_t W1x^T (W1x = the item
    columns of W1), h_t = tanh(z_t + b1'(t)), pred_t = h_t W2^T + b2 and x_{t-1} = c1 pred_t + c2 x_t
    (Model.py:212-215,375),
        z_{t-1} = x_{t-1} W1x^T = c1 (h_t P^T + q) + c2 z_t,      P = W1x W2  (H x H),  q = W1x b2,
    so the state of the chain is the H-dimensional z (fp32), every intermediate step is ONE [rows, H] x [H, H]
    contraction instead of two [rows, I] x [I, H] ones, and only the last step needs item space:
        scores = x_0 = c1_0 (h_0 W2^T + b2)      (c2_0 = 0: alpha_bar_prev(0) = 1, Model.py:262-268).
    Same function of the inputs, S - 1 item-space contraction pairs fewer.  P and q are rebuilt (inside the
    timed region of bench.py) whenever the weights change.  z_S comes from the CSR gather (x_S = x0) or from one
    dense first-layer contraction (dense x_start or sampling_step > 0).
    mode 'full' (DIFFMM_CHAIN=full) runs the literal chain: 2 item-space contractions per step.

    A deeper Denoise (denoise_dim = [d_1, ..., d_L]) has the 2L - 2 hidden-to-hidden layers between its first layer
    in_layers[0] (W1 above) and its last layer out_layers[-1] (W2 above).  Both chains run them as one contraction with
    a bias + tanh epilogue each, between producing h (the first activation) and reading it (the last one); the hidden
    space of the algebra above is the d_L wide one at both ends, so P = W1x W2 stays d_L x d_L."""
    first, inner, last = _layers(den)
    W1, b1, W2, b2 = first.weight, first.bias, last.weight, last.bias
    H, K1 = W1.shape
    I = W2.shape[0]
    d = den.time_emb_dim
    assert K1 == I + d
    widths = hidden_widths(den)
    precision = check_precision(precision or den.precision)
    split = precision == "bf16x3"
    dev = W1.device
    if x_dense is not None:
        n_rows = x_dense.shape[0]
        assert x_dense.shape[1] == I
    assert n_rows is not None and n_rows > 0
    if ws is None or not ws.fits(n_rows, I, widths, d, split):
        ws = ChainWorkspace(n_rows, I, widths, d, split, dev)
    M = n_rows
    S = diff.steps
    mode = mode or chain_mode()
    c2_last = float(np.float32(diff._h_coef2[0]))
    if mode == "full" or c2_last != 0.0 or S < 2:
        return _denoise_chain_full(diff, den, ws, M, x_dense=x_dense, csr=csr, row_ids=row_ids, row0=row0,
                                   sampling_step=sampling_step, split=split, noise=noise, order=order, want_cmax=want_cmax)

    h_hi, h_lo, x = ws.h_hi[:M], (ws.h_lo[:M] if split else None), ws.x[:M]
    xv = x[:, :I]
    z = ws.state()[:M, :H]
    emb_w, emb_b = den.emb_layer.weight.detach(), den.emb_layer.bias.detach()
    W1d, b1d, b2d = W1.detach(), b1.detach(), b2.detach()
    if ws.bias_eff is None or ws.bias_eff.shape[0] != S:
        ws.bias_eff = torch.empty((S, H), dtype=torch.float32, device=dev)
    ops.time_bias(emb_w, emb_b, W1d, I, b1d, 0, S, out=ws.bias_eff)          # b1 + W1[:, I:] temb(i), every step
    p_hi, p_lo, q = _hidden_operators(den, W1, W2, b2, I, split)
    w1_hi, w1_lo = packed_weight(W1, False, split)
    w2_hi, w2_lo = packed_weight(W2, False, split)

    # z_S = x_S W1x^T and h_{S-1} = tanh(z_S + b1'(S-1))
    if csr is not None:
        # binary CSR rows: the first layer is a gather-sum over W1^T (x0 is never densified).  A q_sample'd start
        # (sampling_step > 0, default noise) keeps the rows' sparsity pattern -- sign(x0) zeroes the noise wherever x0
        # is zero (Model.py:337) -- so only the entry values change (dmm_csr_qsample_values) and the gather is weighted.
        vals = None
        if sampling_step > 0:
            vals = _qsample_values(diff, csr, row_ids, row0, M, I, sampling_step, noise, dev)
        w1t_hi, w1t_lo = packed_weight(W1, True, split)                    # W1^T [I + d, pad(H)]: gathered by item id
        ops.csr_gather_act(csr[0], csr[1], M, I, w1t_hi, w1t_lo, ws.bias_eff[S - 1], 1, H, h_hi, h_lo,
                           row_ids=row_ids, row0=row0, z_f32=z, order=order, vals=vals)
    else:
        a_hi, a_lo = ws.operand()
        a_hi = a_hi[:M]
        a_lo = a_lo[:M] if split else None
        _fill_operand(diff, ws, M, I, a_hi, a_lo, x_dense, csr, row_ids, row0, sampling_step, split, noise, dev)
        ops.gemm_bf16_tn(a_hi, a_lo, w1_hi, w1_lo, M, H, I, out_f32=z)
        ops.bias_act_pack(z, ws.bias_eff[S - 1], 1, h_hi, h_lo)
    g_hi, g_lo = ws.hidden2()
    g_hi, g_lo = g_hi[:M], (g_lo[:M] if split else None)
    inner_ops = _inner_operands(inner, split)
    for i in range(S - 1, 0, -1):
        c1 = float(np.float32(diff._h_coef1[i]))          # fp64 table -> .float() (Model.py:352)
        c2 = float(np.float32(diff._h_coef2[i]))
        h_hi, h_lo, g_hi, g_lo = _inner_layers(inner_ops, M, h_hi, h_lo, g_hi, g_lo)
        # z_i = c1 (h_i P^T + q) + c2 z_{i+1} (fp32 state, in place) and, in the same epilogue,
        # h_{i-1} = tanh(z_i + b1'(i-1)) into the OTHER operand buffer (other CTAs still read h_i)
        # (the last intermediate step only needs h_0: its z is never read again, so it is not written: 80 MB less at baby)
        ops.gemm_bf16_tn(h_hi, h_lo, p_hi, p_lo, M, H, H, bias=q, alpha=c1, beta=c2, residual=z, out_f32=z if i > 1 else None,
                         out_hi=g_hi, out_lo=g_lo, post_bias=ws.bias_eff[i - 1], post_act=1)
        h_hi, h_lo, g_hi, g_lo = g_hi, g_lo, h_hi, h_lo
    c1 = float(np.float32(diff._h_coef1[0]))
    h_hi, h_lo, g_hi, g_lo = _inner_layers(inner_ops, M, h_hi, h_lo, g_hi, g_lo)
    ops.gemm_bf16_tn(h_hi, h_lo, w2_hi, w2_lo, M, I, H, bias=b2d, alpha=c1, out_f32=xv,
                     cmax=ws.chunk_max()[:M] if want_cmax else None)
    return xv


NOISE_BLOCK_BYTES = 64 << 20     # randn sub-block of the sparse q_sample: written and re-read while still L2 resident


def _qsample_values(diff, csr, row_ids, row0, M, I, sampling_step, noise, dev):
    """Entry values of x_t = q_sample(x0, sampling_step - 1) for the binary CSR rows [row0, row0 + M) (fp32, indexed like
    csr[1]; entries of other rows are left untouched).  Device RNG (default): dmm_csr_qsample_values_rng generates the
    rows in the kernel.  DIFFMM_CPU_RNG=1 / DIFFMM_QSAMPLE_RNG=torch: the randn draw is torch's (Model.py:337), made in row
    sub-blocks of NOISE_BLOCK_BYTES that stay L2 resident between the generator's write and the kernel's read."""
    indptr, indices = csr
    vals = torch.empty(indices.numel(), dtype=torch.float32, device=dev)
    t = sampling_step - 1
    ca = float(np.float32(diff._h_sqrt_ac[t]))            # fp64 table -> .float() (Model.py:352), host copies: no sync
    cb = float(np.float32(diff._h_sqrt_1mac[t]))
    if noise is not None:
        ops.csr_qsample_values(indptr, indices, M, I, noise, ca, cb, vals, row_ids=row_ids, row0=row0)
        return vals
    mode = os.environ.get("DIFFMM_QSAMPLE_RNG", "chi2")
    if mode not in ("chi2", "philox", "torch"):
        raise ValueError(f"DIFFMM_QSAMPLE_RNG must be chi2, philox or torch, got {mode!r}")
    if not rng.cpu_rng() and mode != "torch":
        # default: the noise is generated inside the kernel (Philox keyed by one draw of torch's device generator:
        # reproducible under torch.manual_seed, no host sync) and never written to HBM.  'chi2' draws the support normals
        # and one chi-square variate for the rest of the row's squared norm (same joint distribution of the outputs, O(k)
        # per row); 'philox' generates all I normals of every row
        seed = torch.randint(0, 2 ** 62, (1,), dtype=torch.int64, device=dev)
        ops.csr_qsample_values_rng(indptr, indices, M, I, seed, ca, cb, vals, row_ids=row_ids, row0=row0,
                                   full_rows=mode == "philox")
        return vals
    sub = max(1, min(M, NOISE_BLOCK_BYTES // (4 * I)))
    buf = torch.empty((sub, ops.pad_to(I, 4)), dtype=torch.float32, device=dev)
    for s0 in range(0, M, sub):
        n = min(sub, M - s0)
        if rng.cpu_rng():
            buf[:n, :I].copy_(torch.randn((n, I), dtype=torch.float32))
        else:
            buf[:n].normal_()             # device generator like randn_like; rows padded to 16 bytes (pad columns unused)
        ops.csr_qsample_values(indptr, indices, n, I, buf[:n, :I], ca, cb, vals,
                               row_ids=row_ids[s0:s0 + n] if row_ids is not None else None, row0=row0 + s0)
    return vals


def _fill_operand(diff, ws, M, I, a_hi, a_lo, x_dense, csr, row_ids, row0, sampling_step, split, noise, dev):
    """x_S as the bf16 operand of the first layer: binary rows (sampling_step == 0) or q_sample'd rows."""
    if sampling_step == 0:
        if csr is not None:
            ops.csr_rows_to_dense(csr[0], csr[1], M, I, row_ids=row_ids, row0=row0, a_bf16=a_hi)
            if split:
                a_lo[:, :I].zero_()           # 0/1 rows are exact in bf16
        else:
            xd = x_dense if (x_dense.stride(1) == 1 and x_dense.dtype == torch.float32) else x_dense.float().contiguous()
            ops.pack_bf16_into(xd, a_hi, a_lo)
    else:
        if csr is not None:
            x0 = torch.empty((M, ws.ld_x), dtype=torch.float32, device=dev)
            ops.csr_rows_to_dense(csr[0], csr[1], M, I, row_ids=row_ids, row0=row0, x_f32=x0)
            x0 = x0[:, :I]
        else:
            x0 = x_dense if x_dense.stride(1) == 1 else x_dense.contiguous()
        if noise is None:
            noise = rng.randn_like(x0)                                       # Model.py:337 draw
        ta, tb = diff._tables_f32(dev)
        t = sampling_step - 1
        ca = ta[t].expand(M).contiguous()
        cb = tb[t].expand(M).contiguous()
        ops.q_sample(x0, noise, ca, cb, 1, a_hi=a_hi, a_lo=a_lo)


def _denoise_chain_full(diff, den, ws, M, *, x_dense, csr, row_ids, row0, sampling_step, split, noise, order=None,
                        want_cmax=False):
    """The literal chain: S x (first layer + tanh, [hidden-to-hidden layers + tanh,] last layer + posterior mean) in item
    space."""
    first, inner, last = _layers(den)
    W1, b1, W2, b2 = first.weight, first.bias, last.weight, last.bias
    H = W1.shape[0]
    I = W2.shape[0]
    dev = W1.device
    a_hi, a_lo = ws.operand()
    a_hi, h_hi, x = a_hi[:M], ws.h_hi[:M], ws.x[:M]
    a_lo = a_lo[:M] if split else None
    h_lo = ws.h_lo[:M] if split else None
    xv = x[:, :I]
    inner_ops = _inner_operands(inner, split)
    if inner_ops:
        g_hi, g_lo = ws.hidden2()
        g_hi, g_lo = g_hi[:M], (g_lo[:M] if split else None)

    S = diff.steps
    # Binary CSR rows at the head of the chain (sampling_step == 0): the first layer of the first reverse step
    # is a gather-sum over W1^T and x0 is never densified (dmm_csr_gather_act / dmm_csr_axpy_bf16).
    sparse_first = sampling_step == 0 and csr is not None and S >= 2
    if not sparse_first:
        _fill_operand(diff, ws, M, I, a_hi, a_lo, x_dense, csr, row_ids, row0, sampling_step, split, noise, dev)

    w1_hi, w1_lo = packed_weight(W1, False, split)
    w2_hi, w2_lo = packed_weight(W2, False, split)
    if sparse_first:
        w1t_hi, w1t_lo = packed_weight(W1, True, split)            # W1^T [I + d, pad(H)]: gathered by item id
    emb_w, emb_b = den.emb_layer.weight.detach(), den.emb_layer.bias.detach()
    W1d, b1d, b2d = W1.detach(), b1.detach(), b2.detach()
    ax_hi = a_hi[:, :I]
    ax_lo = a_lo[:, :I] if split else None
    # every row of a step shares the timestep (Model.py:319): the time-embedding columns of
    # cat([x_t, temb]) (Model.py:203) fold into the bias, b1 + W1[:, I:] temb(i), in fp32 (all steps at once)
    if ws.bias_eff is None or ws.bias_eff.shape[0] != S:
        ws.bias_eff = torch.empty((S, H), dtype=torch.float32, device=dev)
    ops.time_bias(emb_w, emb_b, W1d, I, b1d, 0, S, out=ws.bias_eff)
    for i in range(S - 1, -1, -1):
        bias1 = ws.bias_eff[i]
        first_sparse = sparse_first and i == S - 1
        if first_sparse:
            ops.csr_gather_act(csr[0], csr[1], M, I, w1t_hi, w1t_lo, bias1, 1, H, h_hi, h_lo,
                               row_ids=row_ids, row0=row0, order=order)
        else:
            _gemm1(ws, a_hi, a_lo, w1_hi, w1_lo, M, H, I, bias1, h_hi, h_lo)
        if inner_ops:
            h_hi, h_lo, g_hi, g_lo = _inner_layers(inner_ops, M, h_hi, h_lo, g_hi, g_lo)
        c1 = float(np.float32(diff._h_coef1[i]))          # fp64 table -> .float() (Model.py:352)
        c2 = float(np.float32(diff._h_coef2[i]))
        # x_t lives only as the bf16 operand (hi, and lo in bf16x3 mode: hi + lo carries 16 mantissa bits):
        # the posterior mean c1 * pred + c2 * x_t reads it as the residual and overwrites it in place, so
        # an intermediate step moves 2 (4) bytes per element each way instead of 4 + 4 + 2.  The last step
        # (c2 == 0 for beta_fixed schedules) writes the fp32 scores the top-k consumes.
        use_res = c2 != 0.0 and not first_sparse
        if i == 0:
            ops.gemm_bf16_tn(h_hi, h_lo, w2_hi, w2_lo, M, I, H, bias=b2d, alpha=c1, beta=c2,
                             res_hi=ax_hi if use_res else None, res_lo=ax_lo if use_res else None, out_f32=xv,
                             cmax=ws.chunk_max()[:M] if want_cmax else None)
        else:
            ops.gemm_bf16_tn(h_hi, h_lo, w2_hi, w2_lo, M, I, H, bias=b2d, alpha=c1, beta=c2,
                             res_hi=ax_hi if use_res else None, res_lo=ax_lo if use_res else None,
                             out_hi=ax_hi, out_lo=ax_lo)
            if first_sparse and c2 != 0.0:
                ops.csr_axpy_bf16(csr[0], csr[1], M, I, c2, ax_hi, ax_lo, row_ids=row_ids, row0=row0)
    return xv


K_CHUNK = 8192          # columns of W1 per launch once W1 outgrows the L2 (128 k-blocks of 64)
L2_WEIGHT_BYTES = 48 << 20


def _gemm1(ws, a_hi, a_lo, w1_hi, w1_lo, M, H, K, bias, h_hi, h_lo):
    """h = tanh(x_t W1[:, :K]^T + bias).  At scale-out widths (K = 500k items) W1 is ~1 GB and the persistent CTAs
    walk 7813 k-blocks; with narrow single-CTA tiles they drifted apart until nothing was shared through the L2
    (measured: 35 GB of DRAM reads for 5 GB of operands, 461 TFLOP/s).  The tile cost model now picks the CTA-pair
    kernel there (829 TFLOP/s in one launch).  DIFFMM_K_CHUNK=1 instead issues the contraction in K chunks of 8192
    columns, each launch re-aligning the CTAs, with the partial sums in an fp32 buffer
    (dmm_gemm_epilogue.res_pre_act) and bias + tanh in the last chunk: measured equal, kept as an option."""
    if H * K * 2 <= L2_WEIGHT_BYTES or K <= 2 * K_CHUNK or os.environ.get("DIFFMM_K_CHUNK", "0") != "1":
        ops.gemm_bf16_tn(a_hi, a_lo, w1_hi, w1_lo, M, H, K, bias=bias, act=1, out_hi=h_hi, out_lo=h_lo)
        return
    ld = ops.pad_to(H, 4)
    if ws.partial is None or ws.partial.shape[0] < M or ws.partial.shape[1] != ld:
        ws.partial = torch.empty((ws.rows, ld), dtype=torch.float32, device=a_hi.device)
    part = ws.partial[:M, :H]
    k0 = 0
    while k0 < K:
        kc = min(K_CHUNK, K - k0)
        last = k0 + kc >= K
        sl = slice(k0, k0 + kc)
        al = a_lo[:, sl] if a_lo is not None else None
        wl = w1_lo[:, sl] if w1_lo is not None else None
        res = part if k0 > 0 else None
        if last:
            ops.gemm_bf16_tn(a_hi[:, sl], al, w1_hi[:, sl], wl, M, H, kc, bias=bias, act=1, beta=1.0, residual=res,
                             res_pre_act=True, out_hi=h_hi, out_lo=h_lo)
        else:
            ops.gemm_bf16_tn(a_hi[:, sl], al, w1_hi[:, sl], wl, M, H, kc, beta=1.0, residual=res, out_f32=part)
        k0 += kc


def default_block_rows(n_users: int, n_items: int, hidden, split: bool, budget_bytes: int = 12 << 30) -> int:
    """Largest user block whose workspace stays under ``budget_bytes`` (multiple of 128 rows).  ``hidden``: a width or
    the tuple of hidden widths (the hidden operands are sized by the widest)."""
    per_row = ops.pad_to(n_items + 16, 64) * 2 * (2 if split else 1) + ops.pad_to(n_items, 32) * 4 \
        + ops.pad_to(max(_widths(hidden)), 64) * 2 * (2 if split else 1)
    rows = max(128, (budget_bytes // per_row) // 128 * 128)
    return int(min(n_users, rows))


_ORDER_CACHE: dict = {}


def longest_rows_first(indptr: torch.Tensor, row0: int, n_rows: int) -> torch.Tensor:
    """Scheduling order of dmm_csr_gather_act for the user block [row0, row0 + n_rows): users with more than 32
    interactions first (int32 permutation).  A user with hundreds of interactions is a chain of dozens of dependent
    gather rounds; scheduled last it IS the tail of the launch (measured: a third of the kernel), scheduled first it
    overlaps everything else.  One small kernel (dmm_rows_long_first), no host sync; cached per indptr tensor (same
    object, same version)."""
    key = (id(indptr), indptr._version, indptr.data_ptr(), row0, n_rows)
    ent = _ORDER_CACHE.get("last")
    if ent is not None and ent[0] == key:
        return ent[1]
    order = ops.rows_long_first(indptr, row0, n_rows, 32)
    _ORDER_CACHE["last"] = (key, order, indptr)        # the tensor is kept alive so that id() stays unique
    return order


_SIDE_STREAMS: Dict[Tuple[int, int], list] = {}


def _side_streams(dev: torch.device, n: int, staggered: bool = False):
    """n side streams of the device.  staggered: falling priorities (stream 0 highest), so the pipeline on stream 0 gets
    the SMs first and finishes first while the later ones fill its gaps -- its tail (collective, adjacency build) then
    overlaps the pipelines still running."""
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), n, staggered)
    if key not in _SIDE_STREAMS:
        if staggered:
            _SIDE_STREAMS[key] = [torch.cuda.Stream(device=dev, priority=-(n - 1 - i)) for i in range(n)]
        else:
            _SIDE_STREAMS[key] = [torch.cuda.Stream(device=dev) for _ in range(n)]
    return _SIDE_STREAMS[key]


def rebuild_edges(diff, denoise_models: Dict[str, torch.nn.Module], indptr: torch.Tensor, indices: torch.Tensor,
                  n_users: int, n_items: int, sampling_step: int = 0, precision: Optional[str] = None,
                  row_range: Optional[Tuple[int, int]] = None, block_rows: Optional[int] = None,
                  out_items: Optional[Dict[str, torch.Tensor]] = None, per_modality=None,
                  per_modality_out: Optional[dict] = None, status: Optional[torch.Tensor] = None,
                  staggered: bool = False) -> Dict[str, torch.Tensor]:
    """Top-k item ids per modality for users in ``row_range`` (default all), written at the train-CSR
    offsets (k_u = deg(u), Main.py:215-216,226).  Returns {modality: int32 [E]} (only this range filled).

    The modalities are independent (own Denoise weights, own output), so each one runs as its own pipeline
    (operand packs, chain, top-k and the optional ``per_modality(items)`` follow-up, e.g. the adjacency build) on a
    side CUDA stream forked from / joined to the caller's stream: the latency-bound small kernels and the HBM-bound
    top-k of one modality fill the gaps of the tensor-bound contractions of the other.  DIFFMM_STREAMS=1 keeps
    everything on the caller's stream.  status (optional int32 [1] device tensor): error bits of the top-k (bit 0:
    a user with more interactions than items) are OR-ed in; check it at the caller's next host sync."""
    r0, r1 = row_range if row_range is not None else (0, n_users)
    any_den = next(iter(denoise_models.values()))
    precision = check_precision(precision or any_den.precision)
    split = precision == "bf16x3"
    if block_rows is None:
        block_rows = default_block_rows(r1 - r0, n_items, max(max(hidden_widths(d)) for d in denoise_models.values()), split)
        env = os.environ.get("DIFFMM_BLOCK_ROWS")
        if env:
            block_rows = max(128, min(block_rows, int(env)))
    E = int(indices.numel())
    dev = indptr.device
    prune = os.environ.get("DIFFMM_TOPK_PRUNE", "1") != "0"
    if out_items is None:
        out_items = {m: torch.empty(max(E, 1), dtype=torch.int32, device=dev)[:E] for m in denoise_models}
    mods = list(denoise_models.items())
    orders = {b0: longest_rows_first(indptr, b0, min(b0 + block_rows, r1) - b0) for b0 in range(r0, r1, block_rows)}
    n_streams = min(int(os.environ.get("DIFFMM_STREAMS", "2")), len(mods))
    streams = []
    staggered = staggered or os.environ.get("DIFFMM_STAGGER_ALL") == "1"      # experiment switch: priorities without a tail
    if n_streams > 1 and dev.type == "cuda" and not torch.cuda.is_current_stream_capturing():
        streams = _side_streams(dev, n_streams, staggered)
        main = torch.cuda.current_stream(dev)
        fork = torch.cuda.Event()
        fork.record(main)
        for st in streams:
            st.wait_event(fork)
    with torch.no_grad():
        for mi, (m, den) in enumerate(mods):
            st = streams[mi % len(streams)] if streams else None
            with (torch.cuda.stream(st) if st is not None else contextlib.nullcontext()):
                ws = None
                widths = hidden_widths(den)
                for b0 in range(r0, r1, block_rows):
                    b1 = min(b0 + block_rows, r1)
                    if ws is None or not ws.fits(b1 - b0, n_items, widths, den.time_emb_dim, split):
                        ws = ChainWorkspace(b1 - b0, n_items, widths, den.time_emb_dim, split, dev)
                    scores = denoise_chain(diff, den, csr=(indptr, indices), row0=b0, n_rows=b1 - b0,
                                           sampling_step=sampling_step, precision=precision, ws=ws, order=orders.get(b0),
                                           want_cmax=prune)
                    if prune:      # the contraction left the chunk maxima: the top-k reads only the chunks that matter
                        ops.topk_edges_pruned(scores, n_items, ws.chunk_max()[:b1 - b0], indptr[b0:], b0, None, out_items[m],
                                              status=status, order=orders.get(b0))
                    else:
                        ops.topk_edges(scores, n_items, indptr[b0:], b0, None, out_items[m], status=status,
                                       order=orders.get(b0))
                if per_modality is not None:
                    per_modality_out[m] = per_modality(out_items[m])
    for st in streams:
        main.wait_stream(st)
    return out_items


def rebuild_modal_adj(diff, denoise_models: Dict[str, torch.nn.Module], indptr: torch.Tensor, indices: torch.Tensor,
                      n_users: int, n_items: int, sampling_step: int = 0, precision: Optional[str] = None,
                      block_rows: Optional[int] = None, group=None, plan=None,
                      status: Optional[torch.Tensor] = None) -> Dict[str, ops.CsrAdj]:
    """The whole rebuild phase (Main.py:195-253): {modality: normalised CSR adjacency}.
    With a torch.distributed ``group`` of more than one rank, users are row-sharded and the edge lists
    all-gathered (dist.py); every rank then builds the same adjacency.
    status (optional int32 [1] device tensor, zeroed by the caller): device-side error bits (bit 0: k_u > items in the
    top-k, bit 1: item id out of range in the adjacency build); the caller reads it at its next host sync."""
    from . import dist as ddist
    sharded = group is not None and ddist.world_size(group) > 1
    if not sharded:
        adjs: Dict[str, ops.CsrAdj] = {}
        rebuild_edges(diff, denoise_models, indptr, indices, n_users, n_items, sampling_step, precision,
                      block_rows=block_rows,
                      per_modality=lambda v: ops.build_norm_adj(indptr, v, n_users, n_items, status=status),
                      per_modality_out=adjs, status=status)
        return {m: adjs[m] for m in denoise_models}
    row_range = ddist.shard_rows(n_users, ddist.world_size(group), ddist.rank(group), indptr)
    return rebuild_sharded(diff, denoise_models, indptr, indices, n_users, n_items, sampling_step, precision, row_range,
                           group=group, plan=plan, block_rows=block_rows, status=status)


def rebuild_sharded(diff, denoise_models, indptr, indices, n_users, n_items, sampling_step, precision, row_range, *,
                    group=None, plan=None, block_rows=None, status=None, full_items: Optional[dict] = None,
                    local_hook=None):
    """User-sharded rebuild of one rank: chain + top-k on ``row_range``, the edge lists of all ranks, the whole-graph
    adjacencies.  Default: equal-priority modality pipelines, join, ONE all-gather for all modalities, then the builds on
    the side streams.  DIFFMM_STAGGER=1 (experiment, measured SLOWER: 1.458 vs 1.412 ms per step at 2 GPUs): the pipelines
    run on side streams of falling priority and each one continues into its own all-gather and adjacency build, so that
    the first modality's exchange would overlap the chains still running (collectives in modality order on every rank).
    local_hook(items_m) (optional) runs inside every modality's pipeline once its local edge list is complete (e.g. a copy
    of the rank's slice to pinned host memory that overlaps the exchange)."""
    from . import dist as ddist
    if os.environ.get("DIFFMM_STAGGER", "0") != "1" or len(denoise_models) < 2:
        items = rebuild_edges(diff, denoise_models, indptr, indices, n_users, n_items, sampling_step, precision,
                              row_range=row_range, block_rows=block_rows, status=status, per_modality=local_hook,
                              per_modality_out={} if local_hook is not None else None)
        return gather_and_build(items, indptr, n_users, n_items, group, plan, full_items=full_items, status=status)
    if plan is None or plan.world != ddist.world_size(group):
        plan = ddist.EdgeGatherPlan(indptr, n_users, ddist.world_size(group))

    def tail(local_items):
        if local_hook is not None:
            local_hook(local_items)
        full = ddist.allgather_edges(local_items, indptr, n_users, group, plan)
        return ops.build_norm_adj(indptr, full, n_users, n_items, status=status), full

    res: dict = {}
    rebuild_edges(diff, denoise_models, indptr, indices, n_users, n_items, sampling_step, precision, row_range=row_range,
                  block_rows=block_rows, status=status, per_modality=tail, per_modality_out=res, staggered=True)
    if full_items is not None:
        full_items.update({m: r[1] for m, r in res.items()})
    return {m: res[m][0] for m in denoise_models}


def gather_and_build(items: Dict[str, torch.Tensor], indptr: torch.Tensor, n_users: int, n_items: int, group=None,
                     plan=None, full_items: Optional[dict] = None,
                     status: Optional[torch.Tensor] = None) -> Dict[str, ops.CsrAdj]:
    """Sharded tail of the rebuild: the edge lists are all-gathered on the caller's stream, one collective per modality
    in program order (a collective issued from inside a modality pipeline makes every rank wait for the slowest rank's
    pipeline in the middle of its own: measured 4 % slower at 8 GPUs), then the whole-graph adjacencies are built
    concurrently on the side streams."""
    from . import dist as ddist
    full = ddist.allgather_edges_multi(items, indptr, n_users, group, plan)      # every modality in ONE collective
    if full_items is not None:
        full_items.update(full)
    dev = indptr.device
    n_streams = min(int(os.environ.get("DIFFMM_STREAMS", "2")), len(full))
    if n_streams <= 1 or dev.type != "cuda" or torch.cuda.is_current_stream_capturing():
        return {m: ops.build_norm_adj(indptr, v, n_users, n_items, status=status) for m, v in full.items()}
    streams = _side_streams(dev, n_streams)
    main = torch.cuda.current_stream(dev)
    fork = torch.cuda.Event()
    fork.record(main)
    adjs = {}
    for i, (m, v) in enumerate(full.items()):
        st = streams[i % len(streams)]
        if i < len(streams):
            st.wait_event(fork)
        with torch.cuda.stream(st):
            adjs[m] = ops.build_norm_adj(indptr, v, n_users, n_items, status=status)
    for st in streams:
        main.wait_stream(st)
    return adjs
