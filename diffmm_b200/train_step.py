"""Fused Denoise training step: GaussianDiffusion.training_losses (reference Model.py:385-428) with Denoise.forward
(Model.py:183-220) inlined, forward AND backward scheduled by hand on the C-ABI kernels.

Per modality and batch the reference's autograd graph (q_sample, cat, gate, two Linear layers, mse, two skinny
products, cosine similarity) becomes twelve tensor-pipe contractions (dmm_gemm_bf16_tn) and ten small kernels
(csrc/train.cu) -- about 25 launches instead of the ~215 of the per-op path:

  forward   dmm_train_prep       x_t = a_t x0 + b_t noise and the time-embedding columns, straight into the bf16 operand
            G1  P    = x_t F                          [B, 64]   (Model.py:205)
            dmm_gate_fwd         G = P sigmoid(P Wg^T + bg)              (:206-207)
            G2  x_t' = x_t + G F^T                    in place on the operand (:208)
            G3  h    = tanh([x_t', temb] W1^T + b1)   bf16 operand       (:210-213)
            G4  diff = h W2^T + b2 - x0               fp32 + bf16 operand (:215, :407)
            G5  umd  = diff F ;  G6  [x0 F | x0 E]    (um = umd + x0 F, ui = x0 E: :416-417)
            dmm_diff_loss_fwd    w_t mse + sim_weight (1 - cos(um, ui)) per row, float64 (:407-425)
  backward  dmm_diff_loss_bwd    cm = g w 2 / I,  dumc = (dL/dum) / cm
            G7  d_out' = diff + dumc F^T   (dL/dout = cm d_out'; the row scale cm is applied where it is cheap)
            dmm_colsum -> db2 ;  dmm_pack_bf16(transpose) -> d_out'^T
            G9  dh' = d_out' W2 ;  dmm_hidden_bwd -> dz = cm dh' (1 - h^2), dz^T, (cm h)^T ;  dmm_colsum -> db1
            G8  dW2 = d_out'^T (cm h) ;  dmm_transpose_bf16 -> a^T ;  G10 dW1 = dz^T [x_t', temb]
            G11 dxa = dz W1 ;  G12 dG = dxa F ;  dmm_gate_bwd_pre, dmm_atb_small, dmm_colsum -> gate / emb_layer grads

A deeper denoise_dim adds, per hidden-to-hidden layer, one forward contraction (bias + tanh epilogue) and in the
backward dh = dz W_k, dmm_hidden_bwd without a row scale, dW_k = dz^T h and dmm_colsum (DenoiseLossFn).

The gradient w.r.t. the item embeddings (through ui and the reg term) is NOT produced here: the reference zeroes it
before any optimiser step uses it (Main.py:375; SURVEY App. D.6).  Callers that need it keep the per-op path
(GaussianDiffusion.training_losses falls back when i_embs requires grad)."""
from __future__ import annotations

import os
import weakref

import torch

from . import ops
from .autograd import packed_weight, packed_weight_pair

_FEAT_CACHE: dict = {}


def clear_caches() -> None:
    """Drops the cached feature / item-embedding operand copies (graph capture: they must be rebuilt inside the step)."""
    _FEAT_CACHE.clear()


def enabled() -> bool:
    return os.environ.get("DIFFMM_FUSED_TRAIN", "1") != "0"


def _rows4(t: torch.Tensor) -> torch.Tensor:
    """fp32 row-major view with a 16-byte aligned leading dimension (GEMM residual / TMA requirement)."""
    if t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= t.shape[1] and t.stride(0) % 4 == 0 and t.data_ptr() % 16 == 0:
        return t
    buf = torch.empty((t.shape[0], ops.pad_to(t.shape[1], 4)), dtype=torch.float32, device=t.device)
    buf[:, :t.shape[1]].copy_(t)
    return buf[:, :t.shape[1]]


def feature_operands(feat: torch.Tensor, i_embs: torch.Tensor, split: bool):
    """bf16 operand copies of the modality features F [I, 64] and the item embeddings E [I, 64]:
    F as [I, 64] (K = 64 contractions) and [F^T; E^T] as [128, pad64(I)] (K = I contractions).  Cached per tensor
    object and version: both are constant during a diffusion-training phase."""
    key = (id(feat), id(i_embs), split)
    ent = _FEAT_CACHE.get(key)
    ver = (feat._version, i_embs._version, feat.data_ptr(), i_embs.data_ptr())
    if ent is None or ent[0]() is not feat or ent[1]() is not i_embs or ent[2] != ver:
        if len(_FEAT_CACHE) > 16:
            _FEAT_CACHE.clear()
        f = feat.detach()
        f = f if (f.stride(1) == 1 and f.stride(0) >= f.shape[1]) else f.contiguous()
        e = i_embs.detach()
        e = e if (e.stride(1) == 1 and e.stride(0) >= e.shape[1]) else e.contiguous()
        f_hi, f_lo = ops.pack_bf16(f, split=split)                                   # [I, 64]
        ft_hi, ft_lo = ops.pack_bf16(f, transpose=True, split=split)                 # [64, pad64(I)]
        et_hi, et_lo = ops.pack_bf16(e, transpose=True, split=split)
        fte_hi = torch.cat([ft_hi, et_hi], 0)
        fte_lo = torch.cat([ft_lo, et_lo], 0) if split else None
        ent = (weakref.ref(feat), weakref.ref(i_embs), ver, (f_hi, f_lo, fte_hi, fte_lo))
        _FEAT_CACHE[key] = ent
    return ent[3]


class DenoiseLossFn(torch.autograd.Function):
    """loss_core[b] = w_t mse_b + sim_weight (1 - cos(um_b, ui_b)) (float64 [B]) for one modality and batch; gradients for
    every Denoise parameter.  ``layers`` is the flat list w_0, b_0, ..., w_{2L-1}, b_{2L-1} of the Denoise's Linear
    layers in forward order (in_layers then out_layers; every one a Parameter autograd sees): the first maps
    [x_t', temb] to the hidden space, the 2L - 2 inner ones map hidden to hidden (tanh after each), the last maps back
    to the items.

    Where the per-row scale cm (dL/dout = cm d_out') enters: exactly once, at the top.  The last layer's gradients take
    it through (cm h)^T and the scaled column sum; dz of the top hidden activation is cm dh' (1 - h^2).  Every layer
    below works on that true gradient, so its hidden_bwd runs without a row scale (cm NULL: dz = dh (1 - h^2), h^T)."""

    @staticmethod
    def forward(ctx, x0, t, noise, feat, i_embs, emb_w, emb_b, gate_w, gate_b, tabs, sim_weight, precision, *layers):
        split = precision == "bf16x3"
        dev = x0.device
        B, I = x0.shape
        weights, biases = layers[0::2], layers[1::2]
        assert len(weights) >= 2 and len(biases) == len(weights)
        w1, b1, w2, b2 = weights[0], biases[0], weights[-1], biases[-1]
        H, K1 = w1.shape
        d = emb_w.shape[0]
        assert K1 == I + d and w2.shape == (I, H) and feat.shape == (I, 64)
        tab_a, tab_b, w_tab = tabs
        x0 = _rows4(x0.detach())
        noise = noise.detach()
        noise = noise if (noise.stride(1) == 1 and noise.stride(0) >= I) else noise.contiguous()
        t = t.to(dev, torch.int64).contiguous()
        f_hi, f_lo, fte_hi, fte_lo = feature_operands(feat, i_embs, split)
        bf = dict(dtype=torch.bfloat16, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        Kp = ops.pad_to(I + d, 64)
        a_hi = torch.empty((B, Kp), **bf)
        # the lo part of x_t is kept in single-pass mode too, but only as the RESIDUAL of the gate add (x_t' = x_t + G F^T
        # is then rounded to bf16 once, like the per-op path's fp32 sum); it is an operand only in bf16x3 mode
        a_lo = torch.empty((B, Kp), **bf)
        x0_hi = torch.empty((B, ops.pad_to(I, 64)), **bf)
        te_raw = torch.empty((B, d), **f32)
        ops.train_prep(x0, noise, t, tab_a, tab_b, emb_w.detach(), emb_b.detach(), a_hi, a_lo, x0_hi, te_raw)
        # [x0 F | x0 E]: x0 is binary, exact in bf16
        xfe = torch.empty((B, 128), **f32)
        ops.gemm_bf16_tn(x0_hi, None, fte_hi, fte_lo, B, 128, I, out_f32=xfe)
        x0f, ui = xfe[:, :64], xfe[:, 64:]
        # gate: P = x_t F, G = P sigmoid(P Wg^T + bg), x_t' = x_t + G F^T (in place on the operand)
        P = torch.empty((B, 64), **f32)
        a_lo_op = a_lo if split else None
        ops.gemm_bf16_tn(a_hi, a_lo_op, fte_hi[:64], fte_lo[:64] if split else None, B, 64, I, out_f32=P)
        sig = torch.empty((B, 64), **f32)
        g_hi = torch.empty((B, 64), **bf)
        g_lo = torch.empty((B, 64), **bf) if split else None
        ops.gate_fwd(P, gate_w.detach(), gate_b.detach(), sig, g_hi, g_lo)
        ops.gemm_bf16_tn(g_hi, g_lo, f_hi, f_lo, B, I, 64, alpha=1.0, beta=1.0, res_hi=a_hi[:, :I], res_lo=a_lo[:, :I],
                         out_hi=a_hi[:, :I], out_lo=a_lo[:, :I] if split else None)
        # h = tanh([x_t', temb] W1^T + b1), then h <- tanh(h W_k^T + b_k) through the inner layers: every activation is
        # kept as the bf16 operand (next contraction, h^T of the weight gradient) and in fp32 (tanh' of saturated units
        # needs h beyond bf16; 4 MB each at B = 1024, width 1024)
        acts = []
        h_prev, h_prev_lo, k = a_hi, a_lo_op, I + d
        for w, b in zip(weights[:-1], biases[:-1]):
            n = w.shape[0]
            assert w.shape[1] == k
            (w_hi, w_lo), _ = packed_weight_pair(w, split)
            Hp = ops.pad_to(n, 64)
            h_hi = torch.empty((B, Hp), **bf)
            h_lo = torch.empty((B, Hp), **bf) if split else None
            h_f32 = torch.empty((B, ops.pad_to(n, 4)), **f32)[:, :n]
            ops.gemm_bf16_tn(h_prev, h_prev_lo, w_hi, w_lo, B, n, k, bias=b.detach(), act=1, out_f32=h_f32,
                             out_hi=h_hi[:, :n], out_lo=h_lo[:, :n] if split else None)
            acts.append((h_f32, h_hi, h_lo))
            h_prev, h_prev_lo, k = h_hi, h_lo, n
        # diff = h W2^T + b2 - x0
        (w2_hi, w2_lo), _ = packed_weight_pair(w2, split)
        diff = torch.empty((B, ops.pad_to(I, 4)), **f32)[:, :I]
        d_hi = torch.empty((B, ops.pad_to(I, 64)), **bf)
        d_lo = torch.empty((B, ops.pad_to(I, 64)), **bf) if split else None
        ops.gemm_bf16_tn(h_prev, h_prev_lo, w2_hi, w2_lo, B, I, H, bias=b2.detach(), alpha=1.0, beta=-1.0, residual=x0,
                         out_f32=diff, out_hi=d_hi[:, :I], out_lo=d_lo[:, :I] if split else None)
        umd = torch.empty((B, 64), **f32)
        ops.gemm_bf16_tn(d_hi, d_lo, fte_hi[:64], fte_lo[:64] if split else None, B, 64, I, out_f32=umd)
        loss = torch.empty(B, dtype=torch.float64, device=dev)
        mse = torch.empty(B, **f32)
        um = torch.empty((B, 64), **f32)
        stats = torch.empty((B, 3), **f32)
        ops.diff_loss_fwd(diff, umd, x0f, ui, t, w_tab, float(sim_weight), loss, mse, um, stats)
        ctx.split, ctx.sim_weight, ctx.dims = split, float(sim_weight), (B, I, H, d)
        ctx.tabs = tabs
        ctx.feat_ops = (f_hi, f_lo, fte_hi, fte_lo)
        ctx.bufs = (a_hi, a_lo_op, acts, d_hi, d_lo, diff)
        ctx.save_for_backward(t, P, sig, um, ui, stats, te_raw, *weights)
        ctx.mse = mse
        return loss

    @staticmethod
    def backward(ctx, g_loss):
        t, P, sig, um, ui, stats, te_raw, *weights = ctx.saved_tensors
        w1, w2 = weights[0], weights[-1]
        split = ctx.split
        B, I, H, d = ctx.dims
        f_hi, f_lo, fte_hi, fte_lo = ctx.feat_ops
        a_hi, a_lo, acts, d_hi, d_lo, diff = ctx.bufs
        _, _, w_tab = ctx.tabs
        dev = t.device
        bf = dict(dtype=torch.bfloat16, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        Bp = ops.pad_to(B, 64)

        def hidden_grad_bufs(n):
            """dz (fp32, operand), dz^T and the transposed activation of a hidden activation of width n."""
            Np = ops.pad_to(n, 64)
            dz = torch.empty((B, ops.pad_to(n, 4)), **f32)[:, :n]
            hi = (torch.empty((B, Np), **bf), torch.empty((n, Bp), **bf), torch.empty((n, Bp), **bf))
            lo = (torch.empty((B, Np), **bf), torch.empty((n, Bp), **bf), torch.empty((n, Bp), **bf)) if split \
                else (None, None, None)
            return dz, hi, lo

        g_loss = g_loss.to(torch.float64).contiguous()
        cm = torch.empty(B, **f32)
        dumc_hi = torch.empty((B, 64), **bf)
        dumc_lo = torch.empty((B, 64), **bf) if split else None
        ops.diff_loss_bwd(g_loss, um, ui, stats, t, w_tab, ctx.sim_weight, I, cm, dumc_hi, dumc_lo, None)
        # d_out' = diff + dumc F^T, in place (fp32 and operand copies); dL/dout = cm d_out'
        ops.gemm_bf16_tn(dumc_hi, dumc_lo, f_hi, f_lo, B, I, 64, alpha=1.0, beta=1.0, residual=diff, out_f32=diff,
                         out_hi=d_hi[:, :I], out_lo=d_lo[:, :I] if split else None)
        db2 = ops.colsum(diff, cm)
        dT_hi, dT_lo = ops.pack_bf16(diff, transpose=True, split=split)                    # [I, pad64(B)]
        w2t_hi, w2t_lo = packed_weight(w2, True, split)                                   # W2^T [H, pad64(I)]
        dh = torch.empty((B, ops.pad_to(H, 4)), **f32)[:, :H]
        ops.gemm_bf16_tn(d_hi, d_lo, w2t_hi, w2t_lo, B, H, I, out_f32=dh)
        # top hidden activation: the row scale cm enters here, once
        dz, (dz_hi, dzt_hi, hct_hi), (dz_lo, dzt_lo, hct_lo) = hidden_grad_bufs(H)
        ops.hidden_bwd(dh, acts[-1][0], None, None, cm, H, dz, dz_hi, dz_lo, dzt_hi, dzt_lo, hct_hi, hct_lo)
        dW2 = torch.empty((I, ops.pad_to(H, 4)), **f32)[:, :H]
        ops.gemm_bf16_tn(dT_hi, dT_lo, hct_hi, hct_lo, I, H, B, out_f32=dW2)
        grads = [(dW2.contiguous() if dW2.stride(0) != H else dW2, db2)]
        # inner layers, top down: layer j maps activation j - 1 (width k) to activation j (width n, whose dz is at hand)
        for j in range(len(weights) - 2, 0, -1):
            w = weights[j]
            n, k = w.shape
            wt_hi, wt_lo = packed_weight(w, True, split)                                  # W_j^T [k, pad64(n)]
            dh = torch.empty((B, ops.pad_to(k, 4)), **f32)[:, :k]
            ops.gemm_bf16_tn(dz_hi, dz_lo, wt_hi, wt_lo, B, k, n, out_f32=dh)
            dzp, (dzp_hi, dzpt_hi, ht_hi), (dzp_lo, dzpt_lo, ht_lo) = hidden_grad_bufs(k)
            ops.hidden_bwd(dh, acts[j - 1][0], None, None, None, k, dzp, dzp_hi, dzp_lo, dzpt_hi, dzpt_lo, ht_hi, ht_lo)
            dW = torch.empty((n, ops.pad_to(k, 4)), **f32)[:, :k]
            ops.gemm_bf16_tn(dzt_hi, dzt_lo, ht_hi, ht_lo, n, k, B, out_f32=dW)
            grads.append((dW.contiguous() if dW.stride(0) != k else dW, ops.colsum(dz, None)))
            dz, dz_hi, dz_lo, dzt_hi, dzt_lo = dzp, dzp_hi, dzp_lo, dzpt_hi, dzpt_lo
        db1 = ops.colsum(dz, None)
        aT_hi = torch.empty((I + d, Bp), **bf)
        aT_lo = torch.empty((I + d, Bp), **bf) if split else None
        ops.transpose_bf16(a_hi, a_lo, B, I + d, aT_hi, aT_lo)
        dW1 = torch.empty((H, ops.pad_to(I + d, 4)), **f32)[:, :I + d]
        ops.gemm_bf16_tn(dzt_hi, dzt_lo, aT_hi, aT_lo, H, I + d, B, out_f32=dW1)
        grads.append((dW1.contiguous() if dW1.stride(0) != I + d else dW1, db1))
        w1t_hi, w1t_lo = packed_weight(w1, True, split)                                   # W1^T [I + d, pad64(H)]
        dxa = torch.empty((B, ops.pad_to(I + d, 4)), **f32)[:, :I + d]
        dxa_hi = torch.empty((B, ops.pad_to(I + d, 64)), **bf)
        dxa_lo = torch.empty((B, ops.pad_to(I + d, 64)), **bf) if split else None
        ops.gemm_bf16_tn(dz_hi, dz_lo, w1t_hi, w1t_lo, B, I + d, H, out_f32=dxa, out_hi=dxa_hi[:, :I + d],
                         out_lo=dxa_lo[:, :I + d] if split else None)
        dG = torch.empty((B, 64), **f32)
        ops.gemm_bf16_tn(dxa_hi, dxa_lo, fte_hi[:64], fte_lo[:64] if split else None, B, 64, I, out_f32=dG)
        dpre = torch.empty((B, 64), **f32)
        ops.gate_bwd_pre(dG, P, sig, dpre)
        dWg = ops.atb_small(dpre, P)
        dbg = ops.colsum(dpre, None)
        dtemb = dxa[:, I:I + d]
        dWe = ops.atb_small(dtemb, te_raw)
        dbe = ops.colsum(dtemb, None)
        ctx.bufs = None
        layer_grads = [g for pair in reversed(grads) for g in pair]
        # x0, t, noise, feat, i_embs, emb_w, emb_b, gate_w, gate_b, tabs, sim_weight, precision, *layers
        return (None, None, None, None, None, dWe, dbe, dWg, dbg, None, None, None, *layer_grads)


def denoise_loss(diff, den, x_start, timesteps, noise, modal_feat, i_embs):
    """Fused training_losses core for one modality: (B,) float64 = w_t mse + sim_weight sim (the reg term is added by
    the caller)."""
    tabs = diff._train_tables(x_start.device)
    layers = [p for layer in list(den.in_layers) + list(den.out_layers) for p in (layer.weight, layer.bias)]
    return DenoiseLossFn.apply(x_start, timesteps, noise, modal_feat, i_embs, den.emb_layer.weight, den.emb_layer.bias,
                               den.gate_layer.weight, den.gate_layer.bias, tabs, diff.config.hyper.sim_weight, den.precision,
                               *layers)
