"""Model / Denoise / GaussianDiffusion with the reference's call surface (reference Model.py:15-428),
running on the sm_100a kernels of libdiffmm_b200.so.

Same class names, constructor arguments, parameter names (state-dict compatible), method names
and return conventions as the reference, so ``Main.py -c conf/*.toml`` binds to these symbols
unchanged.  What runs underneath:
  * Model.gcn_MM           -> CSR SpMM kernel (dmm_spmm_csr), A.[u;i] computed once (it is computed M
                              times identically at Model.py:110-114,122-123)
  * Denoise.forward        -> tcgen05 GEMMs with fused bias/tanh epilogues (dmm_gemm_bf16_tn)
  * GaussianDiffusion.generate_view (p_sample loop) -> fused chain: CSR/dense rows -> bf16 operand,
                              [time-embedding columns], GEMM1+tanh, GEMM2+posterior-mean epilogue
  * forward_cal_xt (q_sample) -> dmm_q_sample
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch
import torch.nn.functional as F
from torch import Tensor, nn

from . import ops, rng
from .autograd import (check_precision, linear_tn, modal_mix, packed_weight, row_normalize, spmm, spmm_axpy,
                       spmm_cat)
from .Utils.Utils import *  # noqa: F401,F403  (the reference star-imports its losses here, Model.py:7)
from .Utils.Utils import l2_reg_loss

init = nn.init.xavier_uniform_


def _as_csr(adj) -> ops.CsrAdj:
    """Accepts a CsrAdj or a torch sparse tensor produced by DataHandler.makeTorchAdj (which carries
    its CSR twin as ``_dmm_csr``); any other torch sparse tensor is converted once and cached."""
    if isinstance(adj, ops.CsrAdj):
        return adj
    csr = getattr(adj, "_dmm_csr", None)
    if csr is None:
        from .DataHandler import csr_from_torch_sparse
        csr = csr_from_torch_sparse(adj)
        try:
            adj._dmm_csr = csr
        except Exception:  # pragma: no cover
            pass
    return csr


@dataclass
class GCNOutput:
    u_final_embs: Tensor
    i_final_embs: Tensor
    u_image_embs: Tensor
    i_image_embs: Tensor
    u_text_embs: Tensor
    i_text_embs: Tensor
    u_audio_embs: Optional[Tensor] = None
    i_audio_embs: Optional[Tensor] = None
    # not in the reference: the un-split [N, 64] node tables (final, then one per modality) for the fused loss call
    final_embs: Optional[Tensor] = None
    base_product: Optional[Tensor] = None      # A . [u_embs ; i_embs]: also layer 0 of the cross-layer CL (Main.py:319)
    modal_embs: Optional[list] = None


class Model(nn.Module):
    """Reference Model.py:15-134."""

    def __init__(self, config, image_embedding, text_embedding, audio_embedding=None):
        super().__init__()
        self.config = config
        self.device = torch.device(f"cuda:{self.config.base.gpu}" if torch.cuda.is_available() else "cpu")
        self.u_embs = nn.Parameter(init(torch.empty(self.config.data.user_num, self.config.base.latdim)))
        self.i_embs = nn.Parameter(init(torch.empty(self.config.data.item_num, self.config.base.latdim)))

        self.image_layer = nn.Linear(self.config.data.image_feat_dim, self.config.base.latdim)
        self.text_layer = nn.Linear(self.config.data.text_feat_dim, self.config.base.latdim)
        if audio_embedding is not None:
            self.audio_layer = nn.Linear(self.config.data.audio_feat_dim, self.config.base.latdim)

        self.image_embedding = image_embedding
        self.text_embedding = text_embedding
        self.audio_embedding = audio_embedding

        if audio_embedding is not None:
            self.modal_weight = nn.Parameter(torch.tensor([0.3333, 0.3333, 0.3333]))
        else:
            self.modal_weight = nn.Parameter(torch.tensor([0.5, 0.5]))
        self.softmax = nn.Softmax(dim=-1)
        self.leakyrelu = nn.LeakyReLU(0.2)

    # ---- accessors (Model.py:41-58) ------------------------------------------------------------
    def getItemEmbs(self):
        return self.i_embs

    def getUserEmbs(self):
        return self.u_embs

    def _project(self, layer: nn.Linear, feats: Tensor) -> Tensor:
        # the feature matrices are constants of the model: their packed operand copies are cached
        return linear_tn(feats, layer.weight, layer.bias, 0, getattr(self.config.base, "precision", "bf16"),
                         const_input=not feats.requires_grad)

    def getImageFeats(self) -> Tensor:
        return self._project(self.image_layer, self.image_embedding)

    def getTextFeats(self) -> Tensor:
        return self._project(self.text_layer, self.text_embedding)

    def getAudioFeats(self) -> Optional[Tensor]:
        if self.audio_embedding is None:
            return None
        return self._project(self.audio_layer, self.audio_embedding)

    # ---- propagation (Model.py:60-134) ---------------------------------------------------------
    def gcn_MM(self, adj, image_adj, text_adj, audio_adj=None) -> GCNOutput:
        user = self.config.data.user_num
        A = _as_csr(adj)
        weight = self.softmax(self.modal_weight)
        lam = self.config.hyper.modal_adj_weight

        feats = [self.getImageFeats(), self.getTextFeats()]
        madj = [_as_csr(image_adj), _as_csr(text_adj)]
        if self.audio_embedding is not None:
            feats.append(self.getAudioFeats())
            madj.append(_as_csr(audio_adj))

        prec = getattr(self.config.base, "precision", "bf16")
        # the element-wise glue between the products runs as fused launches (csrc/prop.cu: F.normalize, the modality mix,
        # the residual tail in the SpMM epilogue) on the GPU; DIFFMM_FUSED_PROP=0 keeps the per-op ATen expressions
        fused = self.u_embs.is_cuda and self.u_embs.shape[1] == 64 and os.environ.get("DIFFMM_FUSED_PROP", "1") != "0"
        norm = row_normalize if fused else F.normalize
        zs = [spmm_cat(a, self.u_embs, norm(f), prec) for a, f in zip(madj, feats)]            # :89-93,104-105
        y = spmm_cat(A, self.u_embs, self.i_embs, prec)           # :110-114,122-123 (identical products, once)
        if fused:
            modal_embs = modal_mix(weight, lam, y, zs)             # :116-119,125-127
            # :129-131 — ``final_embs = modal_embs`` aliases, so both in-place adds hit the same tensor:
            # final = (m0 + A m0) + residual_weight * (m0 + A m0) = (1 + residual_weight) (A m0 + m0)
            final_embs = spmm_axpy(A, modal_embs, 1.0 + self.config.hyper.residual_weight, prec)
        else:
            modal_embs = None
            for m, z in enumerate(zs):
                aware = y + lam * z
                modal_embs = weight[m] * aware if modal_embs is None else modal_embs + weight[m] * aware
            t = modal_embs + spmm(A, modal_embs, prec)
            final_embs = t + self.config.hyper.residual_weight * t

        out = GCNOutput(final_embs[:user], final_embs[user:], zs[0][:user], zs[0][user:], zs[1][:user], zs[1][user:])
        if self.audio_embedding is not None:
            out.u_audio_embs, out.i_audio_embs = zs[2][:user], zs[2][user:]
        out.final_embs, out.modal_embs = final_embs, zs
        out.base_product = y
        return out


class Denoise(nn.Module):
    """Reference Model.py:136-220 (time-embedding MLP [I+d] -> H -> I with tanh, optional modality gate)."""

    def __init__(self, in_dims: list, out_dims: list, config, dropout=0.5):
        super().__init__()
        self.device = torch.device(f"cuda:{config.base.gpu}" if torch.cuda.is_available() else "cpu")
        self.in_dims = in_dims
        self.out_dims = out_dims
        self.time_emb_dim = config.base.d_emb_size
        self.precision = check_precision(getattr(config.base, "precision", "bf16"))

        self.emb_layer = nn.Linear(self.time_emb_dim, self.time_emb_dim)
        in_dims_temp = [self.in_dims[0] + self.time_emb_dim] + list(self.in_dims[1:])
        out_dims_temp = list(self.out_dims)
        self.in_layers = nn.ModuleList([nn.Linear(a, b) for a, b in zip(in_dims_temp[:-1], in_dims_temp[1:])])
        self.out_layers = nn.ModuleList([nn.Linear(a, b) for a, b in zip(out_dims_temp[:-1], out_dims_temp[1:])])
        self.drop = nn.Dropout(dropout)           # constructed, never applied (Model.py:164)
        self.init_weights()
        self.modal_emb_dim = config.base.latdim
        self.gate_layer = nn.Linear(self.modal_emb_dim, self.modal_emb_dim)   # default init (after init_weights)

    def init_weights(self):
        for layer in list(self.in_layers) + list(self.out_layers) + [self.emb_layer]:
            nn.init.xavier_normal_(layer.weight)
            if layer.bias is not None:
                nn.init.normal_(layer.bias, mean=0.0, std=0.001)

    def time_embedding(self, timesteps: Tensor) -> Tensor:
        """Model.py:196-202 (differentiable w.r.t. emb_layer)."""
        half = self.time_emb_dim // 2
        freqs = torch.exp(-math.log(10000) * torch.arange(0, half, dtype=torch.float32, device=timesteps.device) / half)
        temp = timesteps.unsqueeze(-1).float() * freqs.unsqueeze(0)
        time_emb = torch.cat([torch.cos(temp), torch.sin(temp)], dim=-1)
        if self.time_emb_dim % 2:
            time_emb = torch.cat([time_emb, torch.zeros_like(time_emb[:, :1])], dim=-1)
        return F.linear(time_emb, self.emb_layer.weight, self.emb_layer.bias)   # 10x10: not a kernel

    def forward(self, x_t: Tensor, timesteps: Tensor, modal_feat: Optional[Tensor] = None) -> Tensor:
        prec = self.precision
        time_emb = self.time_embedding(timesteps)
        if modal_feat is not None:
            proj = linear_tn(x_t, modal_feat.t(), None, 0, prec)                           # :205  x_t F
            gate = torch.sigmoid(F.linear(proj, self.gate_layer.weight, self.gate_layer.bias))   # :206 (64x64)
            x_t = x_t + linear_tn(proj * gate, modal_feat, None, 0, prec)                  # :207-208  G F^T
        h = torch.cat([x_t, time_emb], dim=-1)                                             # :210
        for layer in self.in_layers:
            h = linear_tn(h, layer.weight, layer.bias, 1, prec)                            # :211-213
        for i, layer in enumerate(self.out_layers):
            last = i == len(self.out_layers) - 1
            h = linear_tn(h, layer.weight, layer.bias, 0 if last else 1, prec)             # :214-218
        return h


class GaussianDiffusion(nn.Module):
    """Reference Model.py:222-428."""

    def __init__(self, config, beta_fixed=True):
        super().__init__()
        self.config = config
        self.device = torch.device(f"cuda:{config.base.gpu}" if torch.cuda.is_available() else "cpu")
        self.noise_scale = config.hyper.noise_scale
        self.noise_min = config.hyper.noise_min
        self.noise_max = config.hyper.noise_max
        self.steps = config.hyper.steps
        if self.noise_scale != 0:
            self.betas = torch.tensor(self.get_betas(), dtype=torch.float64, device=self.device)
            if beta_fixed:
                self.betas[0] = 0.0001
            self.calculate_for_diffusion()

    def get_betas(self):
        """Model.py:239-250."""
        start = self.noise_scale * self.noise_min
        end = self.noise_scale * self.noise_max
        variance = np.linspace(start, end, self.steps, dtype=np.float64)
        alpha_bar = 1 - variance
        betas = [1 - alpha_bar[0]]
        for i in range(1, self.steps):
            betas.append(min(1 - alpha_bar[i] / alpha_bar[i - 1], 0.999))
        return np.array(betas)

    def calculate_for_diffusion(self):
        """Model.py:252-275 — fp64 tables; host copies are kept for the kernels' scalar arguments."""
        alphas = 1.0 - self.betas
        dev = self.betas.device
        self.alphas_cumprod = torch.cumprod(alphas, dim=0)
        self.alphas_cumprod_prev = torch.cat([torch.tensor([1.0], device=dev), self.alphas_cumprod[:-1]])
        self.alphas_cumprod_next = torch.cat([self.alphas_cumprod[1:], torch.tensor([0.0], device=dev)])
        self.sqrt_alphas_cumprod = torch.sqrt(self.alphas_cumprod)
        self.sqrt_one_minus_alphas_cumprod = torch.sqrt(1.0 - self.alphas_cumprod)
        self.log_one_minus_alphas_cumprod = torch.log(1.0 - self.alphas_cumprod)
        self.sqrt_reciprocal_alphas_cumprod = torch.sqrt(1.0 / self.alphas_cumprod)
        self.sqrt_reciprocalm1_alphas_cumprod = torch.sqrt(1.0 / self.alphas_cumprod - 1)
        self.posterior_variance = self.betas * (1.0 - self.alphas_cumprod_prev) / (1.0 - self.alphas_cumprod)
        self.posterior_log_variance_clipped = torch.log(
            torch.cat([self.posterior_variance[1].unsqueeze(0), self.posterior_variance[1:]]))
        self.posterior_mean_coef1 = self.betas * torch.sqrt(self.alphas_cumprod_prev) / (1.0 - self.alphas_cumprod)
        self.posterior_mean_coef2 = (1.0 - self.alphas_cumprod_prev) * torch.sqrt(alphas) / (1.0 - self.alphas_cumprod)
        self._h_coef1 = self.posterior_mean_coef1.cpu().numpy()
        self._h_coef2 = self.posterior_mean_coef2.cpu().numpy()
        self._h_sqrt_ac = self.sqrt_alphas_cumprod.cpu().numpy()
        self._h_sqrt_1mac = self.sqrt_one_minus_alphas_cumprod.cpu().numpy()
        self._coef_tables_f32 = None

    def _train_tables(self, device):
        """Device tables of the fused training step: sqrt(abar), sqrt(1 - abar) as fp32 (Model.py:352 casts) and the
        float64 loss weight w_t = SNR(max(t - 1, 0)) - SNR(t), w_0 = 1 (Model.py:380-383,410-412)."""
        ent = getattr(self, "_train_tabs", None)
        if ent is None or ent[0].device != device:
            ta, tb = self._tables_f32(device)
            ac = self.alphas_cumprod.to(device)
            snr = ac / (1 - ac + 1e-8)
            idx = torch.arange(self.steps, device=device)
            w = snr[torch.clamp(idx - 1, min=0)] - snr[idx]
            w = torch.where(idx == 0, 1.0, w).to(torch.float64).contiguous()
            ent = (ta.contiguous(), tb.contiguous(), w)
            self._train_tabs = ent
        return ent

    def _tables_f32(self, device):
        if self._coef_tables_f32 is None or self._coef_tables_f32[0].device != device:
            self._coef_tables_f32 = (self.sqrt_alphas_cumprod.float().to(device),
                                     self.sqrt_one_minus_alphas_cumprod.float().to(device))
        return self._coef_tables_f32

    # ---- q_sample (Model.py:324-355) -----------------------------------------------------------
    def _extract_into_tensor(self, var: Tensor, timesteps: Tensor, broadcast_shape):
        res = var.to(timesteps.device)[timesteps].float()
        while len(res.shape) < len(broadcast_shape):
            res = res.unsqueeze(-1)
        return res.expand(broadcast_shape)

    def forward_cal_xt(self, x_0: Tensor, timesteps: Tensor, noise: Optional[Tensor] = None):
        """x_t = sqrt(abar_t) x_0 + sqrt(1 - abar_t) noise; default noise sign(x_0) * normalize(randn)."""
        mode = 0
        if noise is None:
            noise = rng.randn_like(x_0)        # same draw as Model.py:337
            mode = 1
        ta, tb = self._tables_f32(x_0.device)
        timesteps = timesteps.to(x_0.device)
        x_t = torch.empty((x_0.shape[0], ops.pad_to(x_0.shape[1], 4)), dtype=torch.float32, device=x_0.device)[:, :x_0.shape[1]]
        ops.q_sample(_rows2(x_0), _rows2(noise), ta[timesteps].contiguous(), tb[timesteps].contiguous(), mode, x_t=x_t)
        return x_t

    q_sample = forward_cal_xt       # spelling used by BASELINE.json's north_star

    # ---- p_sample (Model.py:300-322, 357-378) ---------------------------------------------------
    def p_mean_variance(self, denoise: Denoise, x_t: Tensor, timesteps: Tensor, noise: Optional[Tensor] = None):
        predicted_x0 = denoise.forward(x_t, timesteps)
        model_log_variance = self._extract_into_tensor(self.posterior_log_variance_clipped, timesteps, x_t.shape)
        model_mean = (self._extract_into_tensor(self.posterior_mean_coef1, timesteps, x_t.shape) * predicted_x0
                      + self._extract_into_tensor(self.posterior_mean_coef2, timesteps, x_t.shape) * x_t)
        return model_mean, model_log_variance

    def generate_view(self, model: Denoise, x_start: Tensor, sampling_step: int):
        """Deterministic reverse loop i = S-1..0 on the fused inference chain (no autograd tape)."""
        from .rebuild import denoise_chain
        with torch.no_grad():
            return denoise_chain(self, model, x_dense=x_start, sampling_step=sampling_step)

    p_sample = generate_view

    def SNR(self, t: Tensor) -> Tensor:
        """Model.py:380-383 (fp64)."""
        ac = self.alphas_cumprod.to(t.device)
        return ac[t] / (1 - ac[t] + 1e-8)

    # ---- training loss (Model.py:385-428) -------------------------------------------------------
    def training_losses(self, model: Denoise, x_start: Tensor, i_embs: Tensor, modal_feat: Tensor,
                        timesteps: Optional[Tensor] = None, noise: Optional[Tensor] = None):
        """Returns the (B,) fp64 per-row loss.  ``timesteps`` / ``noise`` may be injected (parity tests);
        by default they are drawn exactly like the reference: randint on the CPU generator then moved
        (Model.py:397), randn_like on the device generator (:400)."""
        batch_size = x_start.size(0)
        if timesteps is None:
            timesteps = torch.randint(0, self.steps, (batch_size,)).long()
        timesteps = timesteps.to(x_start.device)
        if noise is None:
            noise = rng.randn_like(x_start)
        from . import train_step
        if (train_step.enabled() and x_start.is_cuda
                and modal_feat is not None and modal_feat.shape[1] == 64 and not modal_feat.requires_grad
                and not i_embs.requires_grad and not x_start.requires_grad):
            # the hot configuration (Main.py:153-170 with the dead item-embedding gradient dropped): forward and backward
            # of the whole loss scheduled by hand on the kernels (train_step.py), for any denoise_dim depth
            core = train_step.denoise_loss(self, model, x_start, timesteps, noise, modal_feat, i_embs)
            reg_loss = l2_reg_loss(self.config.train.reg, [i_embs], self.device)
            return core + reg_loss * self.config.train.reg
        x_t = self.forward_cal_xt(x_start, timesteps, noise)
        model_output = model.forward(x_t, timesteps, modal_feat=modal_feat)

        reconstruction_loss = F.mse_loss(model_output, x_start, reduction="none").mean(dim=-1)
        timesteps_minus1 = torch.clamp(timesteps - 1, min=0)
        weight = self.SNR(timesteps_minus1) - self.SNR(timesteps)
        weight = torch.where(timesteps == 0, 1.0, weight)      # scalar branch: no host tensor (CUDA-graph capturable)
        reconstruction_loss = weight * reconstruction_loss

        prec = model.precision
        user_modal_embs = linear_tn(model_output, modal_feat.t(), None, 0, prec)           # :416
        user_id_embs = linear_tn(x_start, i_embs.t(), None, 0, prec)                       # :417
        sim_loss = 1 - F.cosine_similarity(user_modal_embs, user_id_embs, dim=-1)

        reg_loss = l2_reg_loss(self.config.train.reg, [i_embs], self.device).expand(batch_size)
        return reconstruction_loss + sim_loss * self.config.hyper.sim_weight + reg_loss * self.config.train.reg


def _rows2(t: Tensor) -> Tensor:
    if t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= t.shape[1]:
        return t
    return t.contiguous()
