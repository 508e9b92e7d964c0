"""Trainer with the reference's CLI, ``Coach`` method names, phases, RNG order and log lines
(reference Main.py:18-487), driving the B200 kernels:

  phase 1 (Main.py:145-192)  diffusion training       — Denoise fwd/bwd on tcgen05 GEMMs
  phase 2 (Main.py:195-253)  modality graph rebuild   — rebuild.rebuild_modal_adj (no host sync per edge)
  phase 3 (Main.py:292-377)  joint training           — CSR SpMM + fused BPR / InfoNCE kernels
  eval    (Main.py:390-448)  scores + masked top-20 on device, the reference's metric arithmetic on host

Usage: ``python -m diffmm_b200.Main -c conf/tiktok.toml`` (or put diffmm_b200/dropin first on sys.path and
run the reference's own Main.py unchanged: it then binds to these Model/DataHandler/Utils symbols).
"""
from __future__ import annotations

import argparse
import ast
import os
import random
import time

import numpy as np
import torch
import torch.nn.functional as F
from torch import Tensor
from torch.optim.adam import Adam
from torch.optim.lr_scheduler import CosineAnnealingLR

from . import ops, recommend, rng
from .autograd import joint_losses, linear_tn, spmm, spmm_cat
from .Conf import Config, load_config
from .DataHandler import DataHandler
from .optim import FusedStepAdam
from .Model import Denoise, GaussianDiffusion, Model, _as_csr
from .rebuild import rebuild_modal_adj
from .Utils.Log import Log
from .Utils.Utils import InfoNCE, bpr_loss, l2_reg_loss

main_log = None      # module global like the reference (Main.py:471)
config = None


class _NullLog:
    def info(self, *_a, **_k):
        pass


def _log():
    return main_log if main_log is not None else _NullLog()


class Coach:
    def __init__(self, handler: DataHandler, config: Config, group=None):
        self.handler = handler
        self.config = config
        self.group = group
        self.device = torch.device(f"cuda:{self.config.base.gpu}" if torch.cuda.is_available() else "cpu")
        if self.device.type == "cuda":
            torch.cuda.set_device(self.device)      # the kernels launch on the current device (base.gpu), like torch's own
        self.phase_seconds = {}
        # multi-GPU (one process per GPU, `group` = the torch.distributed group): the rebuild is user-sharded
        # (rebuild_modal_adj) and every propagation product is row-partitioned with one all-gather per layer
        from . import autograd as _ag
        from . import dist as ddist
        if group is not None and ddist.world_size(group) > 1:
            _ag.set_partition(ddist.PropPartition(self.config.data.user_num, self.config.data.item_num, group))
        else:
            _ag.set_partition(None)
        _log().info(f"USER: {self.config.data.user_num}, ITEM: {self.config.data.item_num}")
        _log().info(f"NUM OF INTERACTIONS: {len(self.handler.trainData)}")

    @property
    def has_audio(self):
        return getattr(self.handler, "has_audio", self.config.data.name == "tiktok")

    def makePrint(self, name, epoch, results: dict):
        result_str = f"Epoch {epoch}/{self.config.train.epoch}, {name}: "
        for metric in results:
            result_str += f"{metric}={results[metric]:.5f}, "
        return result_str[:-2] + "  "

    def save_max(self, new: list, old: list) -> list:
        return [i if i > j else j for i, j in zip(new, old)]

    def run(self):
        self.prepareModel()
        _log().info("Model Initialized ✅")
        recallMax, ndcgMax, precisionMax = 0, 0, 0
        his_max = [0, 0, 0]
        bestEpoch = 0
        self.history = []
        _log().info("Start training 🚀")
        try:
            for epoch in range(0, self.config.train.epoch):
                tstFlag = (epoch % self.config.train.tstEpoch == 0)
                result = self.trainEpoch()
                if self.config.train.use_lr_scheduler:
                    self.model_scheduler.step()
                    self.image_scheduler.step()
                    self.text_scheduler.step()
                    if self.has_audio:
                        self.audio_scheduler.step()
                _log().info(self.makePrint("⏩ Train", epoch, result))
                rec = dict(epoch=epoch, train=result)
                if tstFlag:
                    result = self.testEpoch()
                    rec["test"] = result
                    his_max = self.save_max([result["Recall"], result["NDCG"], result["Precision"]], his_max)
                    if result["Recall"] > recallMax:
                        recallMax, ndcgMax, precisionMax = result["Recall"], result["NDCG"], result["Precision"]
                        bestEpoch = epoch
                    _log().info(self.makePrint("🧪 Test", epoch, result))
                self.history.append(rec)
                _log().info(f"💡 Current best: Epoch: {bestEpoch}, Recall: {recallMax:.5f}({his_max[0]:.5f}), NDCG: {ndcgMax:.5f}({his_max[1]:.5f}), Precision: {precisionMax:.5f}({his_max[2]:.5f})")
            _log().info(f"Best epoch: {bestEpoch}, Recall: {recallMax:.5f}({his_max[0]:.5f}), NDCG: {ndcgMax:.5f}({his_max[1]:.5f}), Precision: {precisionMax:.5f}({his_max[2]:.5f})")
        except KeyboardInterrupt:
            _log().info("🈲 Training interrupted by user!")

    def prepareModel(self):
        """Main.py:85-110 — same construction order (parameter init consumes the torch RNG)."""
        h = self.handler
        if self.has_audio:
            self.model = Model(self.config, h.image_feats.detach(), h.text_feats.detach(), h.audio_feats.detach()).cuda(self.device)
        else:
            self.model = Model(self.config, h.image_feats.detach(), h.text_feats.detach()).cuda(self.device)
        # graph replay needs the optimiser state (step counter) on the device: capturable Adam, same update rule.
        # Graph mode: Adam with the one-launch update of csrc/optim.cu (optim.FusedStepAdam: torch's optimiser object, state
        # and scheduler interplay; the step is ONE pass over p / g / m / v evaluating the operation sequence of torch's
        # capturable foreach implementation -- bit-identical, tests/test_optim_gpu.py).  DIFFMM_ADAM=foreach: torch's foreach
        # implementation (fourteen passes); DIFFMM_ADAM=torch_fused: torch's own fused kernel (not validated against the
        # parity runs)
        adam_impl = os.environ.get("DIFFMM_ADAM", "dmm")
        if adam_impl not in ("dmm", "foreach", "torch_fused"):
            raise ValueError(f"DIFFMM_ADAM must be dmm, foreach or torch_fused, got {adam_impl!r}")

        def graph_adam(params):
            lr = torch.tensor(float(self.config.train.lr), device=self.device)
            if adam_impl == "dmm":
                return FusedStepAdam(params, lr=lr, weight_decay=0, capturable=True)
            return Adam(params, lr=lr, weight_decay=0, capturable=True, fused=True if adam_impl == "torch_fused" else None)

        def eager_adam(params):
            # eager mode (python-float lr, host-side step counters): the one-launch step reproduces torch's non-capturable
            # foreach sequence bit for bit as well
            if adam_impl == "dmm":
                return FusedStepAdam(params, lr=self.config.train.lr, weight_decay=0)
            return Adam(params, lr=self.config.train.lr, weight_decay=0, fused=True if adam_impl == "torch_fused" else None)
        if self._use_graph():
            # device-resident step counter and learning rate: one captured graph serves every epoch (the scheduler
            # updates a tensor lr in place)
            self.opt = graph_adam(self.model.parameters())
        else:
            self.opt = eager_adam(self.model.parameters())
        self.model_scheduler = CosineAnnealingLR(self.opt, T_max=self.config.train.epoch, eta_min=1e-4)
        self.diffusion_model = GaussianDiffusion(self.config).cuda(self.device)

        out_dims = ast.literal_eval(self.config.base.denoise_dim) + [self.config.data.item_num]
        in_dims = out_dims[::-1]
        def denoise_adam(params):
            # graph mode: phase 1 is replayed from a CUDA graph as well (device-resident step counter and lr)
            if self._use_graph():
                return graph_adam(params)
            return eager_adam(params)

        self.image_denoise_model = Denoise(in_dims, out_dims, self.config).cuda(self.device)
        self.image_denoise_opt = denoise_adam(self.image_denoise_model.parameters())
        self.image_scheduler = CosineAnnealingLR(self.image_denoise_opt, T_max=self.config.train.epoch, eta_min=1e-4)
        self.text_denoise_model = Denoise(in_dims, out_dims, self.config).cuda(self.device)
        self.text_denoise_opt = denoise_adam(self.text_denoise_model.parameters())
        self.text_scheduler = CosineAnnealingLR(self.text_denoise_opt, T_max=self.config.train.epoch, eta_min=1e-4)
        if self.has_audio:
            self.audio_denoise_model = Denoise(in_dims, out_dims, self.config).cuda(self.device)
            self.audio_denoise_opt = denoise_adam(self.audio_denoise_model.parameters())
            self.audio_scheduler = CosineAnnealingLR(self.audio_denoise_opt, T_max=self.config.train.epoch, eta_min=1e-4)

    def makeTorchAdj(self, u_list, i_list, edge_list):
        """Main.py:113-116 (kept for callers that still build edge lists on the host)."""
        from scipy.sparse import coo_matrix
        mat = coo_matrix((edge_list, (u_list, i_list)), shape=(self.config.data.user_num, self.config.data.item_num), dtype=np.float32)
        return DataHandler.makeTorchAdj(mat, self.config.data.user_num, self.config.data.item_num, self.device)

    # ------------------------------------------------------------------------------------------
    def _denoise_dict(self):
        d = {"image": self.image_denoise_model, "text": self.text_denoise_model}
        if self.has_audio:
            d["audio"] = self.audio_denoise_model
        return d

    def _use_graph(self) -> bool:
        """Phases 1 and 3 from CUDA graphs: the default (``base.cuda_graph``; DIFFMM_CUDA_GRAPH=0 / 1 overrides); never
        with the CPU-RNG parity mode, whose noise draws happen on the host, nor across ranks."""
        env = os.environ.get("DIFFMM_CUDA_GRAPH", "")
        want = bool(getattr(self.config.base, "cuda_graph", True)) if env not in ("0", "1") else env == "1"
        from . import dist as ddist
        multi = self.group is not None and ddist.world_size(self.group) > 1     # collectives stay outside graph capture
        return want and torch.cuda.is_available() and not rng.cpu_rng() and not multi

    def _tick(self, name, t0):
        torch.cuda.synchronize()
        self.phase_seconds[name] = self.phase_seconds.get(name, 0.0) + (time.perf_counter() - t0)

    def trainDiffusion(self):
        """Phase 1 (Main.py:145-192).  Same arithmetic as the reference's loop, which reads every loss with .item()
        (a host sync per modality and batch), normalises the summed loss by the python float total and keeps running
        python-float sums: here those scalars stay on the device in float64 (IEEE-identical adds and divides, the fp32
        divisor is the fp32 rounding of the float64 total exactly like torch's scalar division), read once per epoch."""
        if self._use_graph():
            return self._trainDiffusionGraph()
        zero = torch.zeros((), dtype=torch.float64, device=self.device)
        image_diff_loss, text_diff_loss, audio_diff_loss = zero.clone(), zero.clone(), zero.clone()
        # Model parameters do not move during phase 1, so the projected features the reference recomputes every batch
        # (Main.py:149-151,166) are computed once; the item embeddings enter detached: their gradient from this phase is
        # zeroed before any optimiser step could use it (Main.py:375), and dropping it selects the fused step
        i_embs = self.model.getItemEmbs().detach()
        with torch.no_grad():
            image_feats = self.model.getImageFeats().detach()
            text_feats = self.model.getTextFeats().detach()
            audio_feats = self.model.getAudioFeats().detach() if self.has_audio else None
        for i, batch_data in enumerate(self.handler.diffusionLoader):
            batch_u_items = batch_data[0]

            batch_image_loss = self.diffusion_model.training_losses(self.image_denoise_model, batch_u_items, i_embs, image_feats)
            loss_image = batch_image_loss.mean()
            image_diff_loss = image_diff_loss + loss_image.detach().double()
            batch_text_loss = self.diffusion_model.training_losses(self.text_denoise_model, batch_u_items, i_embs, text_feats)
            loss_text = batch_text_loss.mean()
            text_diff_loss = text_diff_loss + loss_text.detach().double()

            self.image_denoise_opt.zero_grad()
            self.text_denoise_opt.zero_grad()
            if self.has_audio:
                self.audio_denoise_opt.zero_grad()
                batch_audio_loss = self.diffusion_model.training_losses(self.audio_denoise_model, batch_u_items, i_embs, audio_feats)
                loss_audio = batch_audio_loss.mean()
                audio_diff_loss = audio_diff_loss + loss_audio.detach().double()
                total_loss = loss_image.detach().double() + loss_text.detach().double() + loss_audio.detach().double()
                batch_diff_loss = (loss_image + loss_text + loss_audio) / total_loss.to(loss_image.dtype)
                image_diff_loss = image_diff_loss / total_loss
                text_diff_loss = text_diff_loss / total_loss
                audio_diff_loss = audio_diff_loss / total_loss
            else:
                total_loss = loss_image.detach().double() + loss_text.detach().double()
                batch_diff_loss = (loss_image + loss_text) / total_loss.to(loss_image.dtype)
                image_diff_loss = image_diff_loss / total_loss
                text_diff_loss = text_diff_loss / total_loss
            batch_diff_loss.backward()
            self.image_denoise_opt.step()
            self.text_denoise_opt.step()
            if self.has_audio:
                self.audio_denoise_opt.step()
        return image_diff_loss.item(), text_diff_loss.item(), audio_diff_loss.item()

    def _diffusion_step(self, batch_u_items, ts, acc):
        """One batch of phase 1 with the timesteps given (drawn on the host in the reference's order): the M per-row
        losses, their normalised sum, backward, M Adam steps; acc[k] <- (acc[k] + loss_k) / total in place (float64),
        the running sums of Main.py:155-182.  No host sync, no host tensor: capturable."""
        i_embs = self.model.getItemEmbs().detach()       # dead gradient dropped (Main.py:375): selects the fused step
        dens = [self.image_denoise_model, self.text_denoise_model]
        opts = [self.image_denoise_opt, self.text_denoise_opt]
        with torch.no_grad():
            feats = [self.model.getImageFeats().detach(), self.model.getTextFeats().detach()]
            if self.has_audio:
                feats.append(self.model.getAudioFeats().detach())
        if self.has_audio:
            dens.append(self.audio_denoise_model)
            opts.append(self.audio_denoise_opt)
        losses = [self.diffusion_model.training_losses(d, batch_u_items, i_embs, f, timesteps=t).mean()
                  for d, f, t in zip(dens, feats, ts)]
        for o in opts:
            o.zero_grad()
        # the item embeddings also receive a (never used: Main.py:375 zeroes it first) gradient here; dropping the old
        # one keeps a captured backward from accumulating into a tensor that lives outside the graph's memory pool
        self.model.zero_grad(set_to_none=True)
        total = losses[0].detach().double()
        for l in losses[1:]:
            total = total + l.detach().double()
        summed = losses[0]
        for l in losses[1:]:
            summed = summed + l
        batch_diff_loss = summed / total.to(summed.dtype)
        for k, l in enumerate(losses):
            acc[k] = (acc[k] + l.detach().double()) / total
        batch_diff_loss.backward()
        for o in opts:
            o.step()

    def _trainDiffusionGraph(self):
        """Phase 1 replayed from ONE CUDA graph (captured in the first epoch after two eager warm-up batches): the
        batch rows and the host-drawn timesteps are copied into static buffers; the last, smaller batch runs eagerly.
        The device noise comes from torch's graph-safe Philox offsets."""
        from . import autograd as _ag
        B = self.config.train.batch
        M = 3 if self.has_audio else 2
        S = self.diffusion_model.steps
        I = self.config.data.item_num
        if not hasattr(self, "_diff_acc"):
            self._diff_acc = torch.zeros(3, dtype=torch.float64, device=self.device)
            self._diff_rows = torch.zeros((B, ops.pad_to(I, 4)), dtype=torch.float32, device=self.device)[:, :I]
            self._diff_ts = [torch.zeros(B, dtype=torch.int64, device=self.device) for _ in range(M)]
            self._diff_graph = None
            self._diff_warm = 0
        acc = self._diff_acc
        acc.zero_()
        from . import train_step as _ts
        stale = False           # a replay moved the weights without bumping their version counters
        for batch_data in self.handler.diffusionLoader:
            rows = batch_data[0]
            n = rows.shape[0]
            ts = [torch.randint(0, S, (n,)).long() for _ in range(M)]          # Model.py:397 draws, image / text / audio
            if n != B:
                if stale:       # the eager tail batch must not see operand copies made before the last replayed update
                    _ag._PACK_CACHE.clear()
                    _ts.clear_caches()
                    stale = False
                self._diffusion_step(rows, [t.to(self.device) for t in ts], acc)
                continue
            self._diff_rows.copy_(rows)
            for dst, src in zip(self._diff_ts, ts):
                dst.copy_(src, non_blocking=True)
            if self._diff_graph is None and self._diff_warm < 2:
                side = torch.cuda.Stream(device=self.device)
                side.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(side):
                    self._diffusion_step(self._diff_rows, self._diff_ts, acc)
                torch.cuda.current_stream(self.device).wait_stream(side)
                self._diff_warm += 1
                continue
            if self._diff_graph is None:
                _ag._PACK_CACHE.clear()          # packed weights must be (re)built inside the captured step
                from . import train_step as _ts
                _ts.clear_caches()               # ... and so must the feature / item-embedding operand copies
                torch.cuda.synchronize(self.device)
                self._diff_graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._diff_graph):
                    self._diffusion_step(self._diff_rows, self._diff_ts, acc)
            self._diff_graph.replay()
            stale = True
        # a replay updates the weights without bumping their version counters: drop everything derived from them
        _ag._PACK_CACHE.clear()
        _ts.clear_caches()
        for den in self._denoise_dict().values():
            den._dmm_hidden_ops = None
        out = acc.tolist()
        return out[0], out[1], out[2]

    def rebuildGraphs(self):
        """Phase 2 (Main.py:195-253) on device.  The shuffled loader of the reference only permutes users,
        which cannot change the adjacency; its RNG draws are replayed so later phases see the same stream."""
        h = self.handler
        it = iter(h.diffusionLoader.index_batches())
        next(it, None)                                   # base-seed + sampler-seed + randperm draws
        if not hasattr(self, "_rebuild_status"):
            self._rebuild_status = torch.zeros(1, dtype=torch.int32, device=self.device)
        adjs = rebuild_modal_adj(self.diffusion_model, self._denoise_dict(), h.train_indptr, h.train_indices,
                                 self.config.data.user_num, self.config.data.item_num,
                                 self.config.hyper.sampling_step, getattr(self.config.base, "precision", "bf16"),
                                 group=self.group, status=self._rebuild_status)
        self.image_adj, self.text_adj = adjs["image"], adjs["text"]
        if self.has_audio:
            self.audio_adj = adjs["audio"]

    def _check_rebuild_status(self):
        """Device-side error bits of the rebuild (top-k asked for more entries than items; item id out of range in the
        adjacency build), read once per epoch: a corrupt modality graph must not train silently."""
        st = getattr(self, "_rebuild_status", None)
        if st is not None:
            bits = int(st.item())
            if bits:
                st.zero_()
                raise RuntimeError(f"graph rebuild flagged device-side errors (status bits {bits:#x}: "
                                   f"1 = a user has more train interactions than there are items, 2 = item id out of range)")

    def _joint_step(self, users, pos_items, neg_items, biadj):
        """One batch of phase 3 (Main.py:297-377): losses, backward, Adam step.  Returns the four detached loss
        scalars (rec, reg, cl, total) as device tensors."""
        cfg = self.config
        U = cfg.data.user_num
        if self.has_audio:
            gcn_output = self.model.gcn_MM(self.handler.torchBiAdj, self.image_adj, self.text_adj, self.audio_adj)
        else:
            gcn_output = self.model.gcn_MM(self.handler.torchBiAdj, self.image_adj, self.text_adj)
        final_user_embs, final_item_embs = gcn_output.u_final_embs, gcn_output.i_final_embs

        fused = os.environ.get("DIFFMM_FUSED_LOSS", "1") != "0" and cfg.base.latdim == 64
        if not fused:
            rec_loss = bpr_loss(final_user_embs[users], final_item_embs[pos_items], final_item_embs[neg_items])
        reg_loss = l2_reg_loss(cfg.train.reg, [self.model.u_embs, self.model.i_embs], self.device)

        # cross-layer CL (Main.py:315-330)
        all_embs = []
        all_embs_cl = None
        joint_embs = None
        for k in range(3):
            if k == 0:
                # A . [u ; i] is the very product gcn_MM computed on the same operands (Model.py:110-114): taken from there
                # when the adjacency is the same object, else computed from the two blocks (no concatenation pass)
                same = gcn_output.base_product is not None and _as_csr(self.handler.torchBiAdj) is biadj
                joint_embs = gcn_output.base_product if same else spmm_cat(biadj, self.model.u_embs, self.model.i_embs, cfg.base.precision)
            else:
                joint_embs = spmm(biadj, joint_embs, cfg.base.precision)
            random_noise = rng.rand_like(joint_embs)
            joint_embs = _SignNoise.apply(joint_embs, random_noise, cfg.hyper.noise_degree)
            all_embs.append(joint_embs)
            if k == 0:
                all_embs_cl = joint_embs
        final_embs = torch.mean(torch.stack(all_embs), dim=0)
        T, R = cfg.hyper.modal_cl_temp, cfg.hyper.modal_cl_rate
        n_mod = 3 if self.has_audio else 2
        if fused:
            # every loss term of the step in ONE call (dmm_bpr_infonce_fwd / _bwd): tables = [final, z_image, z_text(,
            # z_audio), cross-layer mean, cross-layer first]; 'u' terms index user rows, 'i' terms item rows (+U)
            tables = [gcn_output.final_embs, *gcn_output.modal_embs, final_embs, all_embs_cl]
            i_mean, i_first = 1 + n_mod, 2 + n_mod
            Tc, Rc = cfg.hyper.cross_cl_temp, cfg.hyper.cross_cl_rate
            problems = [(i_mean, i_first, "u", Tc, Rc), (i_mean, i_first, "i", Tc, Rc)]
            if cfg.base.cl_method == 1:      # pairwise between modalities (Main.py:345-350,360-362)
                for a, b in [(0, 1)] + ([(0, 2), (1, 2)] if self.has_audio else []):
                    problems += [(1 + a, 1 + b, "u", T, R), (1 + a, 1 + b, "i", T, R)]
            else:                            # main view as the anchor (Main.py:351-356,363-367)
                for m in range(n_mod):
                    problems += [(0, 1 + m, "u", T, R), (0, 1 + m, "i", T, R)]
            rec_loss, cl_loss = joint_losses(problems, 0, U, users, pos_items, neg_items, tables)
        else:
            cl1_user_embs, cl1_item_embs = final_embs[:U], final_embs[U:]
            cl2_user_embs, cl2_item_embs = all_embs_cl[:U], all_embs_cl[U:]
            cl_loss = (InfoNCE(cl1_user_embs, cl2_user_embs, users, cfg.hyper.cross_cl_temp)
                       + InfoNCE(cl1_item_embs, cl2_item_embs, pos_items, cfg.hyper.cross_cl_temp)) * cfg.hyper.cross_cl_rate
            views = [(gcn_output.u_image_embs, gcn_output.i_image_embs), (gcn_output.u_text_embs, gcn_output.i_text_embs)]
            if self.has_audio:
                views.append((gcn_output.u_audio_embs, gcn_output.i_audio_embs))
            if cfg.base.cl_method == 1:      # pairwise between modalities (Main.py:345-350,360-362)
                pairs = [(0, 1)] + ([(0, 2), (1, 2)] if self.has_audio else [])
                for a, b in pairs:
                    cl_loss = cl_loss + (InfoNCE(views[a][0], views[b][0], users, T) + InfoNCE(views[a][1], views[b][1], pos_items, T)) * R
            else:                            # main view as the anchor (Main.py:351-356,363-367)
                for vu, vi in views:
                    cl_loss = cl_loss + (InfoNCE(final_user_embs, vu, users, T) + InfoNCE(final_item_embs, vi, pos_items, T)) * R

        batch_joint_loss = rec_loss + reg_loss + cl_loss
        self.opt.zero_grad()
        batch_joint_loss.backward()
        self.opt.step()
        return rec_loss.detach(), reg_loss.detach(), cl_loss.detach(), batch_joint_loss.detach()

    def _bind_static_adjacencies(self):
        """Graph mode: the rebuilt modality adjacencies of this epoch are copied into persistent buffers (their sizes
        are fixed: nnz = 2E + N) and the SpMM plans rebuilt in place, so the graph captured in the first epoch stays valid."""
        if not hasattr(self, "_static_adj"):
            self._static_adj = {}
        for name in ("image_adj", "text_adj", "audio_adj"):
            new = getattr(self, name, None)
            if new is None:
                continue
            st = self._static_adj.get(name)
            if st is None:
                self._static_adj[name] = new          # the first epoch's arrays become the persistent ones
            elif st is not new:
                st.ptr.copy_(new.ptr)
                st.idx.copy_(new.idx)
                st.val.copy_(new.val)
                ops.spmm_replan(st)
                setattr(self, name, st)

    def trainJoint(self):
        """Phase 3 (Main.py:292-377).  The running sums stay on the device in float64 (the exact value of the
        reference's python-float sums of fp32 .item()s, Main.py:311-312,370,373) and are read once per epoch: no
        host sync inside the loop.  With ``_use_graph()`` the full-size batches replay ONE CUDA graph captured in the
        first epoch (persistent adjacency buffers, device-resident Adam step and learning rate); the batch indices
        are copied into static buffers, the last, smaller batch runs eagerly."""
        from . import autograd as _ag
        cfg = self.config
        B = cfg.train.batch
        use_graph = self._use_graph()
        if use_graph:
            self._bind_static_adjacencies()
            if not hasattr(self, "_joint_acc"):
                self._joint_acc = torch.zeros(4, dtype=torch.float64, device=self.device)
                self._joint_static = [torch.empty(B, dtype=torch.int64, device=self.device) for _ in range(3)]
                self._joint_graph = None
                self._joint_warm = 0
            acc = self._joint_acc
            acc.zero_()
            static = self._joint_static
        else:
            acc = torch.zeros(4, dtype=torch.float64, device=self.device)      # rec, reg, cl, total
        biadj = _as_csr(self.handler.torchBiAdj)
        for i, batch_data in enumerate(self.handler.trainLoader):
            users, pos_items, neg_items = batch_data
            users = users.long().cuda(self.device)
            pos_items = pos_items.long().cuda(self.device)
            neg_items = neg_items.long().cuda(self.device)
            if not use_graph or users.numel() != B:
                if use_graph and getattr(self, "_joint_stale", False):
                    _ag._PACK_CACHE.clear()      # eager tail batch after replays: operand copies are one update stale
                    self._joint_stale = False
                acc += torch.stack(self._joint_step(users, pos_items, neg_items, biadj)).double()
                continue
            for dst, src in zip(static, (users, pos_items, neg_items)):
                dst.copy_(src)
            if self._joint_graph is None and self._joint_warm < 2:
                # eager warm-up on a side stream (allocator, SpMM plans, lazy initialisation) before the capture
                side = torch.cuda.Stream(device=self.device)
                side.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(side):
                    acc += torch.stack(self._joint_step(*static, biadj)).double()
                torch.cuda.current_stream(self.device).wait_stream(side)
                self._joint_warm += 1
                continue
            if self._joint_graph is None:
                _ag._PACK_CACHE.clear()          # packed weights must be (re)built inside the captured step
                torch.cuda.synchronize(self.device)
                self._joint_graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._joint_graph):
                    acc += torch.stack(self._joint_step(*static, biadj)).double()
            self._joint_graph.replay()
            self._joint_stale = True
        out = acc.tolist()
        self._check_rebuild_status()             # rides on the sync above: no extra round trip per epoch
        if use_graph:
            _ag._PACK_CACHE.clear()              # packs written by the replays are one optimiser step stale
        return out[3], out[0], out[1], out[2]

    def trainEpoch(self):
        t0 = time.perf_counter()
        self.handler.trainData.negSampling()
        self.phase_seconds["neg_sampling"] = self.phase_seconds.get("neg_sampling", 0.0) + (time.perf_counter() - t0)
        train_steps = len(self.handler.trainData) // self.config.train.batch
        diffusion_steps = len(self.handler.diffusionData) // self.config.train.batch

        _log().info("Diffusion model training")
        t0 = time.perf_counter()
        image_diff_loss, text_diff_loss, audio_diff_loss = self.trainDiffusion()
        self._tick("diffusion_train", t0)

        _log().info("Re-build multimodal UI matrix")
        t0 = time.perf_counter()
        self.rebuildGraphs()
        self._tick("rebuild", t0)

        _log().info("Joint training 🤝")
        t0 = time.perf_counter()
        ep_loss, ep_rec_loss, ep_reg_loss, ep_cl_loss = self.trainJoint()
        self._tick("joint_train", t0)

        result = dict()
        result["Loss"] = ep_loss / train_steps
        result["BPR Loss"] = ep_rec_loss / train_steps
        result["reg loss"] = ep_reg_loss / train_steps
        result["CL loss"] = ep_cl_loss / train_steps
        result["image loss"] = image_diff_loss / diffusion_steps
        result["text loss"] = text_diff_loss / diffusion_steps
        if self.has_audio:
            result["audio loss"] = audio_diff_loss / diffusion_steps
        return result

    def testEpoch(self):
        """Main.py:390-448 on the device: scores on the tensor pipe (fp32-faithful bf16x3), train mask written from the
        train CSR (dmm_eval_mask_scores), top-K (dmm_topk_edges with k = K), ranking + Recall / NDCG / Precision per user in
        float64 (dmm_eval_metrics) -- no host round trip per batch; ONE device->host copy of the per-user metrics at the
        end, summed on the host in the reference's order (per test_batch, then across batches) so the totals carry its
        float64 rounding.  top-K > 32 keeps the host path (testEpochHost)."""
        K = int(self.config.base.topk)
        if K > 32 or self.device.type != "cuda":
            return self.testEpochHost()
        t0 = time.perf_counter()
        testData = self.handler.testData
        iter(self.handler.testLoader)        # the reference's loop draws one DataLoader base seed here (RNG parity)
        I = self.config.data.item_num
        ev = getattr(self, "_eval_cache", None)
        if ev is None or ev["K"] != K:
            users = np.asarray(testData.test_users, dtype=np.int64)
            U = self.config.data.user_num
            tptr = np.zeros(U + 1, dtype=np.int64)
            for u in users:
                tptr[u + 1] = len(testData.test_user_its[u])
            np.cumsum(tptr, out=tptr)
            titems = np.fromiter((it for u in np.sort(users) for it in testData.test_user_its[u]), dtype=np.int32,
                                 count=int(tptr[-1]))
            if Coach._MAX_DCG is None or len(Coach._MAX_DCG) != K + 1:
                Coach._MAX_DCG = [np.sum([np.reciprocal(np.log2(loc + 2)) for loc in range(t)]) for t in range(K + 1)]
            inv = np.array([np.reciprocal(np.log2(p + 2)) for p in range(K)], dtype=np.float64)
            dev = self.device
            ev = dict(K=K, users=torch.from_numpy(users).to(dev), n=len(users), test_ptr=torch.from_numpy(tptr).to(dev),
                      test_items=torch.from_numpy(titems).to(dev), inv_log2=torch.from_numpy(inv).to(dev),
                      max_dcg=torch.tensor([float(v) for v in Coach._MAX_DCG], dtype=torch.float64, device=dev),
                      out=torch.empty((len(users), 3), dtype=torch.float64, device=dev))
            self._eval_cache = ev
        n = ev["n"]
        chunk = int(max(256, min(8192, (1 << 30) // (4 * max(I, 1)))))
        with torch.no_grad():
            if self.has_audio:
                gcn_output = self.model.gcn_MM(self.handler.torchBiAdj, self.image_adj, self.text_adj, self.audio_adj)
            else:
                gcn_output = self.model.gcn_MM(self.handler.torchBiAdj, self.image_adj, self.text_adj)
            user_embs, item_embs = gcn_output.u_final_embs, gcn_output.i_final_embs
            h = self.handler
            for s in range(0, n, chunk):
                usr = ev["users"][s:s + chunk]
                b = usr.numel()
                scores = linear_tn(user_embs[usr], item_embs, None, 0, "bf16x3")            # Main.py:410 U_b I^T
                ops.eval_mask_scores(h.train_indptr, h.train_indices, usr, scores, I, -1e8)   # * (1 - mask) - mask * 1e8
                if ev.get("kptr") is None or ev["kptr"].numel() < b + 1:
                    ev["kptr"] = torch.arange(chunk + 1, dtype=torch.int64, device=self.device) * K
                top = torch.empty(b * K, dtype=torch.int32, device=self.device)
                ops.topk_edges(scores, I, ev["kptr"], 0, None, top)                          # Main.py:411
                ops.eval_metrics(scores, top, K, usr, ev["test_ptr"], ev["test_items"], ev["inv_log2"], ev["max_dcg"],
                                 ev["out"][s:s + b])
        vals = ev["out"].cpu().numpy()       # the one host sync of the evaluation
        epRecall = epNdcg = epPrecision = 0
        tb = int(self.config.train.test_batch)
        for s in range(0, n, tb):            # the reference's association: per-batch sums, then the sum of those
            r = g = p = 0
            for a, b_, c in vals[s:s + tb].tolist():
                r += a
                g += b_
                p += c
            epRecall += r
            epNdcg += g
            epPrecision += p
        self._tick("eval", t0)
        return {"Recall": epRecall / n, "NDCG": epNdcg / n, "Precision": epPrecision / n}

    def testEpochHost(self):
        """Main.py:390-420 with the train mask applied from the device CSR, torch.topk and the host metric arithmetic
        (calcRes); the checker of testEpoch and the path for top-K > 32."""
        t0 = time.perf_counter()
        testData = self.handler.testData
        iter(self.handler.testLoader)        # the reference's loop draws one DataLoader base seed here (RNG parity)
        epRecall = epNdcg = epPrecision = 0
        with torch.no_grad():
            if self.has_audio:
                gcn_output = self.model.gcn_MM(self.handler.torchBiAdj, self.image_adj, self.text_adj, self.audio_adj)
            else:
                gcn_output = self.model.gcn_MM(self.handler.torchBiAdj, self.image_adj, self.text_adj)
            user_embs, item_embs = gcn_output.u_final_embs, gcn_output.i_final_embs
            users_all = torch.from_numpy(np.asarray(testData.test_users)).long()
            tb = self.config.train.test_batch
            I = self.config.data.item_num
            for s in range(0, len(users_all), tb):
                usr = users_all[s:s + tb].cuda(self.device)
                trainMask = self.handler.diffusionData.rows(usr)
                predict = linear_tn(user_embs[usr], item_embs, None, 0, "bf16x3")[:, :I] * (1 - trainMask) - trainMask * 1e8
                _, top_idxs = torch.topk(predict, self.config.base.topk)
                recall, ndcg, precision = self.calcRes(top_idxs.cpu().numpy(), testData.test_user_its, usr.cpu())
                epRecall += recall
                epNdcg += ndcg
                epPrecision += precision
        n = len(testData)
        self._tick("eval", t0)
        return {"Recall": epRecall / n, "NDCG": epNdcg / n, "Precision": epPrecision / n}

    def _final_embs(self):
        """(user, item) final embeddings of gcn_MM, as testEpoch computes them for its scores."""
        with torch.no_grad():
            if self.has_audio:
                out = self.model.gcn_MM(self.handler.torchBiAdj, self.image_adj, self.text_adj, self.audio_adj)
            else:
                out = self.model.gcn_MM(self.handler.torchBiAdj, self.image_adj, self.text_adj)
        return out.u_final_embs, out.i_final_embs

    def recommend(self, users, n, exclude_train=True):
        """The n best items of each user in ``users`` (host ints), in rank order: (items int64 [len(users), n], scores fp32
        [len(users), n]) on the device, score descending then item id ascending, the evaluation's bf16x3 scores.  With
        exclude_train the user's train items are never recommended (a list with fewer than n items left ends in item -1,
        score -inf).  Draws no random numbers and changes no parameter."""
        U, I = self.config.data.user_num, self.config.data.item_num
        n = recommend.check_n(n, I)
        rid = np.asarray(users.numpy() if isinstance(users, Tensor) else users)
        if rid.ndim != 1 or (rid.size and (rid.dtype.kind not in "iu" or rid.min() < 0 or rid.max() >= U)):
            raise ValueError(f"users must be a 1-D sequence of user ids in 0..{U - 1}")
        rid = rid.astype(np.int64)
        h = self.handler
        user_embs, item_embs = self._final_embs()
        with torch.no_grad():
            u = user_embs[recommend.to_device(rid, self.device)]
            return recommend.score_topn(u, item_embs, n, exclude=(h.train_indptr, h.train_indices, rid) if exclude_train
                                        else None, precision="bf16x3")

    def evaluate(self, cutoffs=(10, 20, 50)):
        """Recall / NDCG / Precision at every cutoff over testEpoch's test users from ONE ranked list per user: the train
        items are masked with the reference's -1e8 (Main.py:410), the lists are ranked on the device and scored at every
        cutoff in float64 with calcRes' arithmetic (Main.py:422-448), and the per-user values are summed on the host in the
        reference's association (per test_batch, then across batches).  evaluate((K,)) returns exactly testEpoch()'s
        floats under the keys "Recall@K", "NDCG@K", "Precision@K".  Unlike testEpoch it does not touch the test DataLoader:
        it draws no random numbers and changes no parameter, so it can run between epochs of a seeded run."""
        I = self.config.data.item_num
        cuts = recommend.check_cutoffs(cutoffs, I)
        N = cuts[-1]
        testData = self.handler.testData
        users = np.asarray(testData.test_users, dtype=np.int64)
        n = len(users)
        dev = self.device
        tptr, titems = recommend.heldout_csr(users, testData.test_user_its, self.config.data.user_num)
        inv, max_dcg = recommend.metric_tables(N)
        h = self.handler
        user_embs, item_embs = self._final_embs()
        with torch.no_grad():
            usr = recommend.to_device(users, dev)
            ranked, _ = recommend._topn(user_embs[usr], item_embs, N, (h.train_indptr, h.train_indices, usr), -1e8, "bf16x3")
            out = torch.empty((n, len(cuts), 3), dtype=torch.float64, device=dev)
            ops.eval_metrics_cutoffs(ranked, N, cuts, usr, recommend.to_device(tptr, dev), recommend.to_device(titems, dev),
                                     recommend.to_device(inv, dev), recommend.to_device(max_dcg, dev), out)
        vals = out.cpu().numpy()             # the one host sync of the evaluation
        tb = int(self.config.train.test_batch)
        res = {}
        for j, c in enumerate(cuts):
            tot = [0, 0, 0]
            for s in range(0, n, tb):        # the reference's association: per-batch sums, then the sum of those
                part = [0, 0, 0]
                for row in vals[s:s + tb, j].tolist():
                    for m in range(3):
                        part[m] += row[m]
                for m in range(3):
                    tot[m] += part[m]
            res[f"Recall@{c}"], res[f"NDCG@{c}"], res[f"Precision@{c}"] = (t / n for t in tot)
        return res

    def score(self, users, items):
        """The bf16x3 scores of the pairs (users[p], items[p]) (fp32 [P] on the device; users / items: equal-length 1-D
        integer arrays, host data or CUDA tensors).  Same terms as ``evaluate``'s scores, summed in another order
        (recommend.score_pairs).  Draws no random numbers and changes no parameter."""
        user_embs, item_embs = self._final_embs()
        with torch.no_grad():
            return recommend.score_pairs(user_embs, item_embs, users, items, precision="bf16x3")

    def rank_candidates(self, users, candidates, n):
        """Row b of ``candidates`` (int [len(users), C], -1 = empty slot) ranked for user users[b] (host ints): (items
        int64, scores fp32) [len(users), n] on the device, score descending then item id ascending, bf16x3 scores as
        ``score`` gives them.  Train items are not excluded: the caller chose the candidates."""
        U = self.config.data.user_num
        rid = np.asarray(users.numpy() if isinstance(users, Tensor) else users)
        if rid.ndim != 1 or (rid.size and (rid.dtype.kind not in "iu" or rid.min() < 0 or rid.max() >= U)):
            raise ValueError(f"users must be a 1-D sequence of user ids in 0..{U - 1}")
        user_embs, item_embs = self._final_embs()
        with torch.no_grad():
            u = user_embs[recommend.to_device(rid.astype(np.int64), self.device)]
            return recommend.rank_candidates(u, item_embs, candidates, n, precision="bf16x3")

    def evaluate_sampled(self, n_neg=100, cutoffs=(1, 5, 10), seed=0):
        """HR@K and NDCG@K of the sampled-negative protocol over testEpoch's test users: every (user, held-out item)
        instance ranks its item against n_neg negatives drawn uniformly without replacement from the items in neither
        the user's train nor its test items (recommend.sampled_candidates with np.random.default_rng(seed)).  The rows are
        ranked on the device with bf16x3 scores (recommend.rank_candidates); a tie between the held-out item and a
        negative goes to the smaller item id (the library's total order).  With one test item per row,
        dmm_eval_metrics_cutoffs' Recall@K is HR@K and its NDCG@K is 1 / log2(p + 2) at position p < K.  Returns
        {"HR@K": ..., "NDCG@K": ...} per cutoff (1 <= K <= min(1024, 1 + n_neg)), each the mean over instances summed on
        the host in float64 in instance order.  Draws no random numbers from a global generator, does not touch the test
        DataLoader and changes no parameter."""
        cuts = recommend.check_cutoffs(cutoffs, 1 + recommend.check_n_neg(n_neg))
        N = cuts[-1]
        h = self.handler
        testData = h.testData
        users = np.asarray(testData.test_users, dtype=np.int64)
        train_csr = (h.train_indptr.cpu().numpy(), h.train_indices.cpu().numpy())
        inst_users, cand = recommend.sampled_candidates(users, testData.test_user_its, train_csr,
                                                        self.config.data.item_num, n_neg, seed)
        T = inst_users.size
        if T == 0:
            raise ValueError("the test set holds no held-out items")
        dev = self.device
        inv, max_dcg = recommend.metric_tables(N)
        user_embs, item_embs = self._final_embs()
        with torch.no_grad(), torch.cuda.device(dev):
            u = user_embs[recommend.to_device(inst_users, dev)]
            ranked, _ = recommend._rank_candidates(u, item_embs, recommend.to_device(cand, dev), N, "bf16x3")
            rows = torch.arange(T, dtype=torch.int64, device=dev)
            out = torch.empty((T, len(cuts), 3), dtype=torch.float64, device=dev)
            ops.eval_metrics_cutoffs(ranked, N, cuts, rows, torch.arange(T + 1, dtype=torch.int64, device=dev),
                                     recommend.to_device(np.ascontiguousarray(cand[:, 0]), dev),
                                     recommend.to_device(inv, dev), recommend.to_device(max_dcg, dev), out)
        vals = out.cpu().numpy()             # the one host sync of the evaluation
        res = {}
        for j, c in enumerate(cuts):
            hr = ndcg = 0.0
            for r_, g_ in vals[:, j, :2].tolist():
                hr += r_
                ndcg += g_
            res[f"HR@{c}"], res[f"NDCG@{c}"] = hr / T, ndcg / T
        return res

    _MAX_DCG = None

    def calcRes(self, top_idxs: np.ndarray, test_u_its: list, users: Tensor):
        """Main.py:422-448 vectorised over the batch with the same float64 arithmetic in the same order
        (per-user hit sums follow the order of the user's test items, the batch totals are added user by user)."""
        assert top_idxs.shape[0] == len(users)
        topk = self.config.base.topk
        if Coach._MAX_DCG is None or len(Coach._MAX_DCG) != topk + 1:
            Coach._MAX_DCG = [np.sum([np.reciprocal(np.log2(loc + 2)) for loc in range(t)]) for t in range(topk + 1)]
        users = users.tolist() if hasattr(users, "tolist") else list(users)
        B = len(users)
        tst_num = np.fromiter((len(test_u_its[u]) for u in users), dtype=np.int64, count=B)
        seg = np.repeat(np.arange(B), tst_num)
        items = np.fromiter((it for u in users for it in test_u_its[u]), dtype=np.int64, count=int(tst_num.sum()))
        eq = top_idxs[seg].astype(np.int64) == items[:, None]                  # [pairs, topk]
        hit = eq.any(axis=1)
        pos = eq.argmax(axis=1)                                                # list.index: first occurrence
        gain = np.where(hit, np.reciprocal(np.log2(pos + 2.0)), 0.0)
        recall_hits = np.bincount(seg, weights=hit.astype(np.float64), minlength=B)
        dcg = np.bincount(seg, weights=gain, minlength=B)                      # accumulates in item order
        max_dcg = np.array([Coach._MAX_DCG[min(int(t), topk)] for t in tst_num])
        allRecall = allNdcg = allPrecision = 0
        for r, n_, p in zip((recall_hits / tst_num).tolist(), (dcg / max_dcg).tolist(), (recall_hits / topk).tolist()):
            allRecall += r
            allNdcg += n_
            allPrecision += p
        return allRecall, allNdcg, allPrecision


class _SignNoise(torch.autograd.Function):
    """e + sign(e) * normalize(rnd) * noise_degree (Main.py:320-321); d/de = identity (sign has zero grad)."""

    @staticmethod
    def forward(ctx, e, rnd, noise_degree):
        out = e.detach().clone()
        ops.sign_noise_(out, rnd, float(noise_degree))
        return out

    @staticmethod
    def backward(ctx, g):
        return g, None, None


def seed_it(seed):
    """Main.py:450-456."""
    random.seed(seed)
    os.environ["PYTHONSEED"] = str(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    torch.cuda.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)


def main(argv=None):
    global main_log, config
    parser = argparse.ArgumentParser(description="Model Configs")
    parser.add_argument("--config", "-c", default="conf/test.toml", type=str, help="config file path")
    args = parser.parse_args(argv)
    try:
        config = load_config(args.config)
        print(f"Load configuration ({config.data.name}) file successfully👌")
    except Exception as e:
        print(f"Error loading configuration file: {e}")
        raise SystemExit(1)
    seed_it(config.base.seed)
    main_log = Log("main", config.data.name)
    main_log.info("Start")
    main_log.info("Configuration Details:")
    for section, options in config.__dict__.items():
        main_log.info(f"{section}: {options}")
    data_handler = DataHandler(config)
    main_log.info("Load Data")
    data_handler.LoadData()
    coach = Coach(data_handler, config)
    coach.run()
    return coach


if __name__ == "__main__":
    main()
