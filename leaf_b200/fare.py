"""The LEAF / TextFARE training iteration on the engine: the body of train_one_epoch_text_only's batch loop
(/root/reference/utils_AT.py:291-366) - frozen anchor, LEAF attack, forward + backward of the B winners, gradient
accumulation, clipping, AdamW with the reference's two parameter groups (/root/reference/train_AT_text_only.py:326-341)
and, under torch.distributed, the data-parallel gradient all-reduce the reference delegates to DDP.

What is native: everything that touches the tower (K1-K4), the AdamW update (one launch over the flat parameter
buffer), the gradient-norm reduction. What stays torch: the two-line loss expression and the NCCL all-reduce call.
The scheduler, the data loader, logging and checkpointing are the caller's, unchanged (SURVEY.md 8: out of scope).
"""
from __future__ import annotations

import ctypes
import math
import os
import weakref

import torch
import torch.distributed as dist

from ._native import BACKWARD_HOOK, check
from .attack import V_DEFAULT, attack_text_leaf
from .engine import _ptr, _stream
from .eval_attacks import attack_text_charmer_inference
from .tower import LeafTextTower


class FareTrainer:
    """One object per process (GPU). Hyper-parameters carry the reference's names (params_AT.py, scripts/train_leaf_*.sh):
    lr, wd, beta1, beta2, eps, accum_freq, grad_clip_norm, rho, k_adv, constrain, normalize_fare, use_charmer."""

    def __init__(self, tower: LeafTextTower, frozen: LeafTextTower, V=V_DEFAULT, rho: int = 50, k_adv: int = 1, lr: float = 1e-5,
                 wd: float = 1e-4, beta1: float = 0.9, beta2: float = 0.98, eps: float = 1e-6, accum_freq: int = 1,
                 grad_clip_norm: float = None, constrain=False, normalize_fare: bool = False, use_charmer: bool = False,
                 group=None, overlap_allreduce: bool = True, backward_sm_budget: int = None):
        self.tower, self.frozen, self.V = tower, frozen, list(V)
        self.rho, self.k_adv, self.constrain = rho, k_adv, constrain
        self.lr, self.wd, self.beta1, self.beta2, self.eps = lr, wd, beta1, beta2, eps
        self.accum_freq, self.grad_clip_norm = accum_freq, grad_clip_norm
        self.normalize_fare, self.use_charmer, self.group = normalize_fare, use_charmer, group
        tower.trainable()
        tower.attach_grads()
        tower.zero_grad()
        self.exp_avg = torch.zeros_like(tower.flat_params)
        self.exp_avg_sq = torch.zeros_like(tower.flat_params)
        self._norm = torch.zeros(1, dtype=torch.float32, device=tower.flat_params.device)
        self.opt_step = 0            # optimizer steps taken
        self.micro = 0               # micro-batches seen
        # ---- data-parallel gradient exchange overlapped with the backward (what DDP's bucketed all-reduce does for the
        #      reference, train_AT_text_only.py:310-317): leaf_backward calls back after every layer; the callback records an
        #      event and queues an all-reduce of that layer's slice of the flat gradient buffer behind it on a side stream ----
        self._distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self.overlap_allreduce = bool(overlap_allreduce) and self._distributed
        self._works, self._reduced = [], False
        # SMs the backward's persistent GEMM grids may take while the exchange runs beside them (None: all of them)
        self.backward_sm_budget = int(os.environ.get("LEAF_BACKWARD_SM_BUDGET", "0")) if backward_sm_budget is None else int(backward_sm_budget)
        if self.overlap_allreduce:
            self._side = torch.cuda.Stream(device=tower.flat_params.device)
            self._layer_ranges, self._rest_ranges = self._gradient_ranges()
            self._hook_armed = False
            me = weakref.ref(self)

            def thunk(layer, user):                           # a no-op once this trainer is gone (the engine may outlive it)
                tr = me()
                if tr is not None:
                    tr._on_backward_layer(layer, user)

            eng = tower.leaf_engine
            eng._backward_hook = BACKWARD_HOOK(thunk)         # the ctypes thunk lives as long as the engine that calls it
            check(eng._lib.leaf_set_backward_hook(eng._h, ctypes.cast(eng._backward_hook, ctypes.c_void_p), None))

    def _gradient_ranges(self):
        """Contiguous [lo, hi) element ranges of the flat gradient buffer: one list per layer holding that layer's weight
        MATRICES (adjacent in the buffer: the stable sort of LeafTextTower keeps the state dict's layer order inside the
        weight-decay group), and the rest (every 1-D parameter, the embeddings, the projection) reduced at the end."""
        t = self.tower
        span = lambda k: (t._slices[k][0], t._slices[k][0] + (t._slices[k][1] + 3) // 4 * 4)
        per_layer, taken = [], []
        for l in range(t.leaf_engine.layers):
            ks = [k for k in t._slices if k.startswith(f"transformer.resblocks.{l}.") and len(t._slices[k][2]) >= 2]
            per_layer.append(self._merge([span(k) for k in ks]))
            taken += ks
        rest = self._merge([span(k) for k in t._slices if k not in taken])
        return per_layer, rest

    @staticmethod
    def _merge(spans):
        out = []
        for lo, hi in sorted(spans):
            if out and out[-1][1] == lo:
                out[-1][1] = hi
            else:
                out.append([lo, hi])
        return [tuple(x) for x in out]

    def _on_backward_layer(self, layer, _user):
        if not self._hook_armed:
            return
        ranges = self._rest_ranges if layer == -1 else self._layer_ranges[layer] if layer < len(self._layer_ranges) else []
        if not ranges:
            return
        g = self.tower.flat_grads
        ev = torch.cuda.Event()
        ev.record()                                           # after this layer's gradients on the backward's stream
        self._side.wait_event(ev)
        with torch.cuda.stream(self._side):
            for lo, hi in ranges:
                self._works.append(dist.all_reduce(g[lo:hi], op=dist.ReduceOp.AVG, group=self.group, async_op=True))
        if layer == -1:
            self._reduced = True

    # ---- pieces (public so that a caller can keep its own loop and swap single stages) -------------------------------
    @torch.no_grad()
    def anchors(self, texts):
        """utils_AT.py:296."""
        return self.frozen.encode_text(self.frozen.tokenizer(texts), normalize=self.normalize_fare)

    @torch.no_grad()
    def attack(self, texts, anchors):
        """utils_AT.py:297-309."""
        dev = self.tower.flat_params.device
        if self.use_charmer:
            return [attack_text_charmer_inference(self.tower, None, t, anchors[j], dev, objective="l2", n=self.rho, k=self.k_adv,
                                                  constrain=self.constrain, V=self.V)[0] for j, t in enumerate(texts)]
        return attack_text_leaf(self.tower, None, texts, anchors, dev, objective="l2", n=self.rho, k=self.k_adv, V=self.V,
                                constrain=self.constrain)[1]

    def lr_at(self, step: int) -> float:
        """Hook for the caller's scheduler (utils_AT.py:287-288); constant by default."""
        return self.lr

    def _exchange(self):
        """Data-parallel average of the accumulated gradients: wait for the slices exchanged while the backward ran, or one
        blocking all-reduce of the flat buffer."""
        if not self._distributed:
            return
        if self._reduced:                                     # already exchanged slice by slice while the backward ran
            for w in self._works:
                w.wait()                                      # stream-level: the next kernels queue behind the collectives
            self._works, self._reduced = [], False
        else:
            dist.all_reduce(self.tower.flat_grads, op=dist.ReduceOp.AVG, group=self.group)

    def _clip_scale(self, grad_scale: float = 1.0) -> float:
        """torch.nn.utils.clip_grad_norm_(norm_type=2): the factor min(1, max_norm / (total_norm + 1e-6))."""
        eng, g = self.tower.leaf_engine, self.tower.flat_grads
        eng.set_deterministic(torch.are_deterministic_algorithms_enabled())
        self._norm.zero_()
        check(eng._lib.leaf_sumsq(eng._h, _ptr(g), g.numel(), _ptr(self._norm), _stream()))
        total = math.sqrt(float(self._norm.item())) * grad_scale
        return min(1.0, self.grad_clip_norm / (total + 1e-6))

    def optimizer_step(self, grad_scale: float = 1.0):
        """utils_AT.py:338-362 with scaler = None: all-reduce (DDP's job in the reference), clip, AdamW, zero_grad; then the
        engine re-casts its bf16 operand copies from the updated fp32 parameters."""
        t = self.tower
        g, eng = t.flat_grads, t.leaf_engine
        self._exchange()
        scale = grad_scale
        if self.grad_clip_norm is not None:                       # the clip is folded into AdamW's gradient scale
            scale *= self._clip_scale(grad_scale)
        self.opt_step += 1
        f = ctypes.c_float
        check(eng._lib.leaf_adamw(eng._h, _ptr(t.flat_params), _ptr(g), _ptr(self.exp_avg), _ptr(self.exp_avg_sq), g.numel(),
                                  t.n_nodecay, f(self.lr_at(self.opt_step)), f(self.beta1), f(self.beta2), f(self.eps), f(self.wd),
                                  self.opt_step, f(scale), _stream()))
        t.zero_grad()
        t.refresh()

    # ---- the iteration ---------------------------------------------------------------------------------------------------
    def step(self, texts):
        """One micro-batch of utils_AT.py:291-366. Returns (loss_FARE_text as a 0-d tensor, adversarial texts)."""
        t = self.tower
        anchors = self.anchors(texts)
        adv_texts = self.attack(texts, anchors.clone())
        tok, lens = t.tokenizer(adv_texts, with_lengths=True)                              # :312 (lengths ride on the status read)
        feats = t.encode_text(tok, normalize=self.normalize_fare, host_lengths=lens)       # :317-319 (train mode == eval: no dropout)
        loss = torch.nn.functional.mse_loss(anchors, feats, reduction="none").sum(dim=-1).mean()      # :321-322
        last = (self.micro + 1) % self.accum_freq == 0
        # The reference clips the ACCUMULATED gradients after every micro-batch (:356-357), and its DDP wrapper averages them
        # in every backward; without clipping, one exchange during the last micro-batch's backward gives the same sums.
        clip_now = self.grad_clip_norm is not None and not last
        budget = self.overlap_allreduce and (last or clip_now) and self.backward_sm_budget > 0
        if self.overlap_allreduce:
            self._hook_armed = last or clip_now
        if budget:
            check(t.leaf_engine._lib.leaf_set_sm_budget(t.leaf_engine._h, self.backward_sm_budget))
        (loss / self.accum_freq).backward()                                                # :329-337
        if budget:
            check(t.leaf_engine._lib.leaf_set_sm_budget(t.leaf_engine._h, 0))
        if self.overlap_allreduce:
            self._hook_armed = False
        self.micro += 1
        if last:
            self.optimizer_step()
        elif clip_now:
            self._exchange()                                  # averaging identical accumulated values again changes nothing
            s = self._clip_scale()
            if s < 1.0:
                eng, g = t.leaf_engine, t.flat_grads
                check(eng._lib.leaf_scale(eng._h, _ptr(g), g.numel(), ctypes.c_float(s), _stream()))
        return loss.detach(), adv_texts
